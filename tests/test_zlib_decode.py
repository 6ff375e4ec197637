"""zlib chunks (SURVEY.md section 8, row f4): decode-only GPU inflate.

The algorithm lives in a third-party library of the reference (zlib 1.3.1, vendored under
internal-complibs/ and absent from this repository), so parity is pinned on (1) the reference's
own golden chunks compat/blosc-*-zlib*.cdata, (2) streams produced and judged by the system's
zlib (Python's `zlib` module = the same upstream library): every level / strategy / window size,
stored, fixed and dynamic blocks, and damaged streams must get zlib's accept/reject verdict, and
(3) chunks the reference's own zlib path wrote, stored in tests/golden/reference_zlib.npz (inputs
kept small enough to store).  CPU: the device code inside the SIMT emulator.  GPU: through the C ABI."""
import ctypes as C
import glob
import os
import zlib

import numpy as np
import pytest

from datagen import bench_words, ci, compress, decompress, gen, golden_arrays, ptr, sz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _streams():
    """(name, original bytes, zlib stream) covering all DEFLATE block types."""
    rng = np.random.default_rng(5)
    datas = {
        "bench": bench_words(200000).tobytes(),
        "text": gen("text", 70000, 1).tobytes(),
        "rand": gen("rand", 40000, 2).tobytes(),               # stored blocks
        "zeros": bytes(100000),                                 # long matches, distance 1
        "i32": gen("i32", 131072).tobytes(),
        "tiny": b"a",
        "empty": b"",
        "mixed": gen("mixed", 150000, 3).tobytes(),
    }
    out = []
    for name, d in datas.items():
        for level in (1, 5, 9):
            out.append((f"{name}-l{level}", d, zlib.compress(d, level)))
        for strategy, tag in ((zlib.Z_FIXED, "fixed"), (zlib.Z_HUFFMAN_ONLY, "huff"), (zlib.Z_RLE, "rle")):
            co = zlib.compressobj(6, zlib.DEFLATED, 15, 8, strategy)
            out.append((f"{name}-{tag}", d, co.compress(d) + co.flush()))
        co = zlib.compressobj(6, zlib.DEFLATED, 9)              # 512-byte window
        out.append((f"{name}-w9", d, co.compress(d) + co.flush()))
        co = zlib.compressobj(0)                                # stored only
        out.append((f"{name}-l0", d, co.compress(d) + co.flush()))
        co = zlib.compressobj(6)                                # several blocks incl. an empty stored one (sync flush)
        half = len(d) // 2
        out.append((f"{name}-sync", d, co.compress(d[:half]) + co.flush(zlib.Z_SYNC_FLUSH) + co.compress(d[half:]) + co.flush()))
    return out


def _zlib_verdict(stream, cap):
    """What uncompress() does with `cap` bytes of room: decoded bytes or None."""
    try:
        do = zlib.decompressobj()
        got = do.decompress(stream, cap + 1)
        if not do.eof or len(got) > cap:
            return None
        return got
    except zlib.error:
        return None


def test_inflate_matches_zlib_emu(emu):
    emu.emu_zlib_decode.restype = C.c_int
    for name, d, st in _streams():
        src = np.frombuffer(st, np.uint8).copy()
        for cap in (len(d), len(d) + 7, max(len(d) - 1, 0)):
            out = np.full(cap + 16, 0x77, np.uint8)
            r = emu.emu_zlib_decode(ptr(src), ci(len(src)), ptr(out), ci(cap))
            want = _zlib_verdict(st, cap)
            if want is None:
                assert r == -1, (name, cap, r)
            else:
                assert r == len(want) and bytes(out[:r]) == want and (out[cap:] == 0x77).all(), (name, cap, r)
        # trailing bytes after the stream are ignored by uncompress()
        ext = np.concatenate([src, np.arange(5, dtype=np.uint8)])
        out = np.zeros(len(d) + 16, np.uint8)
        assert emu.emu_zlib_decode(ptr(ext), ci(len(ext)), ptr(out), ci(len(d))) == len(d)


def test_inflate_rejects_what_zlib_rejects_emu(emu):
    emu.emu_zlib_decode.restype = C.c_int
    rng = np.random.default_rng(9)
    nbad = ngood = 0
    for name, d, st in _streams():
        if len(d) > 80000 or len(st) < 8:
            continue
        for trial in range(25):
            c = bytearray(st)
            kind = trial % 5
            if kind == 0:
                c = c[:rng.integers(1, len(c))]                                  # truncated
            elif kind == 1:
                c[rng.integers(0, min(len(c), 12))] ^= 1 << rng.integers(0, 8)   # header / first block header
            elif kind == 2:
                c[-rng.integers(1, 5)] ^= 0x10                                   # Adler-32
            else:
                for pos in rng.integers(0, len(c), kind - 2):
                    c[pos] = rng.integers(0, 256)
            c = bytes(c)
            src = np.frombuffer(c, np.uint8).copy()
            out = np.full(len(d) + 16, 0x77, np.uint8)
            r = emu.emu_zlib_decode(ptr(src), ci(len(src)), ptr(out), ci(len(d)))
            want = _zlib_verdict(c, len(d))
            if want is None:
                assert r == -1, (name, trial, r)
                nbad += 1
            else:
                assert r == len(want) and bytes(out[:r]) == want, (name, trial, r)
                ngood += 1
            assert (out[len(d):] == 0x77).all()
    assert nbad > 300 and ngood > 5


def _compat_zlib_files():
    return sorted(f for f in glob.glob(os.path.join(ROOT, "tests", "golden", "compat", "*.cdata")) if "zlib" in f)


def test_compat_zlib_goldens_emu(emu):
    """The reference's own zlib golden chunks (blosc 1.3.0 ... 1.14.0) decode to int32 data[i] = i."""
    want = np.arange(1000000, dtype=np.int32).view(np.uint8)
    files = _compat_zlib_files()
    assert len(files) == 5
    for f in files[:2]:                                        # the emulator is slow: two files here, all five on the GPU
        chunk = np.fromfile(f, np.uint8)
        out = np.zeros(4000000 + 64, np.uint8)
        assert emu.blosc_decompress_ctx(ptr(chunk), ptr(out), sz(4000000), ci(1)) == 4000000, f
        assert (out[:4000000] == want).all()
        item = np.zeros(4096, np.uint8)
        assert emu.blosc_getitem(ptr(chunk), ci(250000), ci(1024), ptr(item)) == 4096
        assert (item == want[1000000:1004096]).all()
        bad = chunk.copy(); bad[len(bad) // 2] ^= 0x55
        assert emu.blosc_decompress_ctx(ptr(bad), ptr(out), sz(4000000), ci(1)) == -1
    assert emu.blosc_compress_ctx(ci(5), ci(1), sz(4), sz(1000), ptr(want), ptr(out), sz(2000), b"zlib", sz(0), ci(1)) == -5   # decode only


CHUNKS = [(kind, n, ts, shuf, clevel) for kind, n in (("bench", 6000), ("text", 3001), ("mixed", 6000), ("rand", 1000))
          for ts, shuf, clevel in ((4, 1, 5), (8, 2, 1), (1, 0, 9), (3, 1, 6))]


def _chunk_key(kind, n, ts, shuf, clevel):
    return f"chunk-{kind}-{n}-{ts}-{shuf}-{clevel}"


def _reference_chunks():
    stored = golden_arrays("zlib")
    assert len(stored) == len(CHUNKS)
    return [(kind, n, ts, shuf, clevel, gen(kind, n, 4), stored[_chunk_key(kind, n, ts, shuf, clevel)])
            for kind, n, ts, shuf, clevel in CHUNKS]


def test_zlib_chunks_from_the_reference_emu(emu):
    """Chunks written by the reference's own zlib path (built with its vendored zlib 1.3.1): the
    reference's framing (splits, raw splits, leftover block) around zlib streams."""
    for kind, n, ts, shuf, clevel, src, chunk in _reference_chunks():
        r, out = decompress(emu, "blosc_decompress_ctx", chunk, n)
        assert r == n and (out[:n] == src).all() and (out[n:] == 0).all(), (kind, ts, shuf, clevel)


@pytest.mark.gpu
def test_compat_zlib_goldens_gpu(pkg, cuda):
    want = np.arange(1000000, dtype=np.int32).view(np.uint8)
    files = _compat_zlib_files()
    assert len(files) == 5
    for f in files:
        chunk = np.fromfile(f, np.uint8)
        out = np.zeros(4000000 + 64, np.uint8)
        assert pkg.decompress_ctx(chunk, out, 4000000) == 4000000, f
        assert (out[:4000000] == want).all() and (out[4000000:] == 0).all()
        bad = chunk.copy(); bad[len(bad) // 3] ^= 0x55
        assert pkg.decompress_ctx(bad, out, 4000000) == -1


@pytest.mark.gpu
def test_zlib_chunks_from_the_reference_gpu(pkg, ref, cuda):
    """Chunks written by the reference's own zlib path: several typesizes / filters / levels, bench.c data,
    text, compressible runs mixed with noise, and noise.  Where oracle/_ref was built, also 2 MiB of bench.c
    data, text and 1 MiB of mixed data, written by the reference on the spot."""
    if ref is not None:
        for kind, n in (("bench", 2 << 20), ("text", 300001), ("mixed", 1 << 20)):
            src = gen(kind, n, 4)
            for ts, shuf, clevel in ((4, 1, 5), (8, 2, 1), (1, 0, 9), (3, 1, 6)):
                cb, chunk = compress(ref, "blosc_compress_ctx", clevel, shuf, ts, src, n + 16, "zlib")
                assert cb > 0
                out = np.zeros(n + 64, np.uint8)
                assert pkg.decompress_ctx(chunk, out, n) == n
                assert (out[:n] == src).all() and (out[n:] == 0).all(), (kind, ts, shuf, clevel)
    for kind, n, ts, shuf, clevel, src, chunk in _reference_chunks():
        out = np.zeros(n + 64, np.uint8)
        assert pkg.decompress_ctx(chunk, out, n) == n
        assert (out[:n] == src).all() and (out[n:] == 0).all()


def reference_golden(ref, orc):
    arrays = {}
    for kind, n, ts, shuf, clevel in CHUNKS:
        src = gen(kind, n, 4)
        cb, chunk = compress(ref, "blosc_compress_ctx", clevel, shuf, ts, src, n + 16, "zlib")
        assert cb > 0 and decompress(ref, "blosc_decompress_ctx", chunk, n)[0] == n
        arrays[_chunk_key(kind, n, ts, shuf, clevel)] = chunk[:cb].copy()
    return arrays
