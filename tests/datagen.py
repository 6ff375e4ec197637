"""Deterministic test inputs (seeded), thin ctypes helpers shared by the tests, and the stored
results of the unmodified reference (tests/golden/reference*, written by
scripts/record_reference_golden.py from a reference build in oracle/_ref)."""
import ctypes as C
import functools
import hashlib
import json
import os

import numpy as np

vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@functools.lru_cache(None)
def golden():
    """The reference's results: small values and per-group digests (reference.json)."""
    with open(os.path.join(GOLDEN, "reference.json")) as f:
        return json.load(f)


@functools.lru_cache(None)
def golden_arrays(name):
    """Frames and chunks the reference wrote (reference_<name>.npz)."""
    with np.load(os.path.join(GOLDEN, f"reference_{name}.npz")) as z:
        return {k: z[k] for k in z.files}


class Transcript:
    """What one library returned over a series of cases, kept as one digest per group of cases.
    The reference's transcript is stored; the oracle's or the emulator's must equal it group by group."""

    def __init__(self):
        self.hashes, self.h = {}, None

    def group(self, *key):
        self.h = self.hashes["/".join(map(str, key))] = hashlib.blake2b(digest_size=8)

    def add(self, *vals):
        for v in vals:
            self.h.update(v.tobytes() if isinstance(v, np.ndarray) else int(v).to_bytes(8, "little", signed=True))

    def digests(self):
        return {k: h.hexdigest() for k, h in self.hashes.items()}


def check_transcript(key, t):
    want, got = golden()["transcripts"][key], t.digests()
    assert sorted(got) == sorted(want), (key, "cases differ from the recorded ones")
    bad = [k for k in want if got[k] != want[k]]
    assert not bad, f"{key}: differs from the reference in groups {bad[:8]}"


class Api:
    """The entry points the transcripts call, bound to the reference's names or to the oracle's."""

    def __init__(self, lib, reference):
        self.lib, self.reference = lib, reference
        p = "" if reference else "orc_"
        self.lz4_compress = getattr(lib, "LZ4_compress_fast" if reference else "orc_lz4_compress_fast")
        self.lz4_decompress = getattr(lib, "LZ4_decompress_safe" if reference else "orc_lz4_decompress_safe")
        self.blosclz_compress = getattr(lib, p + "blosclz_compress")
        self.blosclz_decompress = getattr(lib, p + "blosclz_decompress")
        self.getitem = getattr(lib, "blosc_getitem" if reference else "orc_getitem")
        self.ctx = ("blosc_" if reference else "orc_") + "compress_ctx", ("blosc_" if reference else "orc_") + "decompress_ctx"

    def compress(self, *args, **kw):
        return compress(self.lib, self.ctx[0], *args, **kw)

    def decompress(self, *args, **kw):
        return decompress(self.lib, self.ctx[1], *args, **kw)

    def filter(self, op, ts, n, src, dst):
        """op: shuffle, unshuffle, bitshuffle or bitunshuffle"""
        if not self.reference:
            return getattr(self.lib, "orc_" + op)(sz(ts), sz(n), ptr(src), ptr(dst))
        args = [sz(ts), sz(n), ptr(src), ptr(dst)]
        if op.startswith("bit"):
            args.append(ptr(np.zeros(n + 64, np.uint8)))
        return getattr(self.lib, "blosc_internal_" + op)(*args)


def ptr(a):
    return a.ctypes.data_as(vp)


def bench_words(nbytes, rshift=19, start=0):
    """bench/bench.c:141-170 synthetic buffer: int32 w[i] = ((i<<26)^(i<<18)^(i<<11)^(i<<3)^i) & mask."""
    i = np.arange(start, start + (nbytes + 3) // 4, dtype=np.uint32)
    w = ((i << np.uint32(26)) ^ (i << np.uint32(18)) ^ (i << np.uint32(11)) ^ (i << np.uint32(3)) ^ i)
    if rshift < 32:
        w &= np.uint32((1 << rshift) - 1)
    return w.view(np.uint8)[:nbytes].copy()


def gen(kind, n, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "rand":
        return rng.integers(0, 256, n, dtype=np.uint8)
    if kind == "bench":
        return bench_words(n)
    if kind == "zeros":
        return np.zeros(n, np.uint8)
    if kind == "lowent":
        return rng.integers(0, 4, n, dtype=np.uint8)
    if kind == "text":
        words = [bytes(rng.integers(97, 123, rng.integers(2, 9), dtype=np.uint8)) for _ in range(200)]
        out = b" ".join(words[j] for j in rng.integers(0, 200, n // 4 + 8))
        return np.frombuffer(out[:n], np.uint8).copy()
    if kind == "ramp":
        return (np.arange(n) // 7 % 251).astype(np.uint8)
    if kind == "i32":
        return np.arange(n // 4 + 1, dtype=np.int32).view(np.uint8)[:n].copy()
    if kind == "f32":
        return np.linspace(0, 100, n // 4 + 1, dtype=np.float32).view(np.uint8)[:n].copy()
    if kind == "mixed":          # compressible runs interleaved with noise: raw and compressed splits in one chunk
        a = np.zeros(n, np.uint8)
        noise = rng.integers(0, 256, n, dtype=np.uint8)
        seg = max(n // 16, 1)
        for k in range(0, n, seg):
            if (k // seg) % 2:
                a[k:k + seg] = noise[k:k + seg]
            else:
                a[k:k + seg] = (np.arange(min(seg, n - k)) // 3 % 200).astype(np.uint8)
        return a
    raise ValueError(kind)


def compress(lib, fn, clevel, shuf, ts, src, destsize, comp, bs=0, nt=1, fill=0xAA):
    dest = np.full(destsize + 64, fill, np.uint8)
    r = getattr(lib, fn)(ci(clevel), ci(shuf), sz(ts), sz(len(src)), ptr(src), ptr(dest), sz(destsize), comp.encode(), sz(bs), ci(nt))
    return r, dest


def decompress(lib, fn, chunk, destsize, nt=1):
    dest = np.zeros(destsize + 64, np.uint8)
    r = getattr(lib, fn)(ptr(chunk), ptr(dest), sz(destsize), ci(nt))
    return r, dest
