"""zstd chunks (SURVEY.md section 8, row f4): decode-only GPU zstd frame decoder.

The algorithm lives in a third-party library of the reference (zstd 1.5.6, vendored under
internal-complibs/ and absent from this repository), so parity is pinned on (1) the reference's
own golden chunks compat/blosc-*-zstd*.cdata and (2) frames written and judged by that very
library: all levels, raw / RLE / compressed blocks, Huffman and FSE table modes, multi-block
frames with treeless literals and repeat-mode / RLE sequence tables (test_stored_frames_cover_the_block_modes
checks they are there), checksums; damaged frames must get ZSTD_decompress()'s accept/reject verdict.
The frames and chunks the reference wrote are stored in tests/golden/reference_zstd.npz (inputs kept
small enough to store), its verdicts in tests/golden/reference.json.
CPU: the device code inside the SIMT emulator."""
import ctypes as C
import glob
import hashlib
import os

import numpy as np
import pytest

from datagen import Transcript, bench_words, check_transcript, ci, compress, decompress, gen, golden, golden_arrays, ptr, sz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _zstd(ref):
    ref.ZSTD_compress.restype = C.c_size_t
    ref.ZSTD_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int]
    ref.ZSTD_decompress.restype = C.c_size_t
    ref.ZSTD_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    ref.ZSTD_isError.restype = C.c_uint
    ref.ZSTD_isError.argtypes = [C.c_size_t]
    ref.ZSTD_compressBound.restype = C.c_size_t
    ref.ZSTD_compressBound.argtypes = [C.c_size_t]
    ref.ZSTD_createCCtx.restype = C.c_void_p
    ref.ZSTD_CCtx_setParameter.restype = C.c_size_t
    ref.ZSTD_CCtx_setParameter.argtypes = [C.c_void_p, C.c_int, C.c_int]
    ref.ZSTD_compress2.restype = C.c_size_t
    ref.ZSTD_compress2.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    ref.ZSTD_freeCCtx.argtypes = [C.c_void_p]
    return ref


LEVELS = (1, 3, 5, 9, 15, 19, 22, -5)


def _tiled_noisy():
    """300 kB of a repeated text with one byte in 100 replaced: several compressed blocks whose literals reuse
    the previous block's Huffman table (treeless literals) and whose sequences repeat the previous tables"""
    rng = np.random.default_rng(3)
    t = np.tile(gen("text", 3000, 1), 100)
    t[rng.integers(0, len(t), 3000)] = rng.integers(97, 123, 3000)
    return t


def _sparse():
    """zeros with a random byte every 97 positions: blocks whose offsets are one code (an RLE offset table)"""
    z = np.zeros(200000, np.uint8)
    z[::97] = np.random.default_rng(1).integers(1, 256, len(z[::97]))
    return z


def _datas():
    """name -> (input, the levels its frames are written at); the larger inputs only at levels that give the
    block modes they are there for"""
    d = {
        "bench": bench_words(1000),
        "plane": (bench_words(12000 * 4).view(np.uint32) >> 8).astype(np.uint8),    # a shuffled byte-plane
        "text": gen("text", 3000, 1),
        "rand": gen("rand", 1000, 2),
        "zeros": np.zeros(300000, np.uint8),
        "i32": gen("i32", 3000),
        "mixed": gen("mixed", 3000, 3),
        "lowent": gen("lowent", 3000, 4),
        "tiny": np.frombuffer(b"abcabcabcabcabcabcabcabcabcabcabc", np.uint8).copy(),
        "one": np.frombuffer(b"x", np.uint8).copy(),
        "empty": np.zeros(0, np.uint8),
    }
    out = {k: (v, LEVELS) for k, v in d.items()}
    out["tiled_noisy"] = (_tiled_noisy(), (9, 19))
    out["sparse"] = (_sparse(), (1, 3))
    return out


def _write_frames(ref):
    """What the reference's zstd writes for each input: every level, and one frame with a checksum, without the
    content size and with a small window."""
    out = {}
    for name, (d, levels) in _datas().items():
        n = len(d)
        for level in levels:
            buf = np.zeros(int(ref.ZSTD_compressBound(n)) + 16, np.uint8)
            r = ref.ZSTD_compress(ptr(buf), len(buf), ptr(d), n, level)
            assert not ref.ZSTD_isError(r)
            out[f"{name}-l{level}"] = buf[:r].copy()
        cctx = ref.ZSTD_createCCtx()
        for prm, val in ((100, 3), (201, 1), (200, 0), (101, 12)):   # compressionLevel, checksumFlag, contentSizeFlag, windowLog
            assert not ref.ZSTD_isError(ref.ZSTD_CCtx_setParameter(cctx, prm, val))
        buf = np.zeros(int(ref.ZSTD_compressBound(n)) + 16, np.uint8)
        r = ref.ZSTD_compress2(cctx, ptr(buf), len(buf), ptr(d), n)
        assert not ref.ZSTD_isError(r)
        out[f"{name}-cksum"] = buf[:r].copy()
        ref.ZSTD_freeCCtx(cctx)
    return out


def _frames():
    stored, datas = golden_arrays("zstd"), _datas()
    names = sorted(k for k in stored if not k.startswith("chunk"))
    assert len(names) == sum(len(levels) + 1 for _, levels in datas.values())
    return [(k, datas[k.split("-", 1)[0]][0], stored[k]) for k in names]


def _block_modes(frame):
    """What the blocks of one zstd frame use (RFC 8878 sections 3.1.1.1 - 3.1.1.3.2): counts of blocks, compressed
    blocks, treeless literal sections, sequence sections with a repeat-mode table and with an RLE offset table."""
    b = bytes(frame)
    assert b[:4] == bytes.fromhex("28b52ffd")
    fhd = b[4]
    single, did, fcs = (fhd >> 5) & 1, fhd & 3, fhd >> 6
    p = 5 + (0 if single else 1) + (0, 1, 2, 4)[did] + ((1 if single else 0), 2, 4, 8)[fcs]
    c = dict(blocks=0, compressed=0, treeless=0, repeat=0, rle_offsets=0)
    last = 0
    while not last:
        h = int.from_bytes(b[p:p + 3], "little")
        p += 3
        last, btype, size = h & 1, (h >> 1) & 3, h >> 3
        c["blocks"] += 1
        if btype == 2:
            c["compressed"] += 1
            q, lt, sf = p, b[p] & 3, (b[p] >> 2) & 3
            if lt < 2:                                          # raw or RLE literals
                hs, regen = ((1, b[q] >> 3) if sf in (0, 2) else (2, (b[q] >> 4) + (b[q + 1] << 4)) if sf == 1 else
                             (3, (b[q] >> 4) + (b[q + 1] << 4) + (b[q + 2] << 12)))
                q += hs + (regen if lt == 0 else 1)
            else:                                               # Huffman-coded, with (2) or without (3) a tree
                hs, bits = ((3, 10), (3, 10), (4, 14), (5, 18))[sf]
                q += hs + ((int.from_bytes(b[q:q + hs], "little") >> (4 + bits)) & ((1 << bits) - 1))
                c["treeless"] += lt == 3
            n0 = b[q]
            if n0:
                q += 1 if n0 < 128 else 2 if n0 < 255 else 3
                ll, of, ml = b[q] >> 6, (b[q] >> 4) & 3, (b[q] >> 2) & 3
                c["repeat"] += 3 in (ll, of, ml)
                c["rle_offsets"] += of == 1
        p += 1 if btype == 1 else size
    return c


def test_stored_frames_cover_the_block_modes():
    """the stored frames keep the decoder paths they were chosen for: multi-block frames, treeless literals,
    repeat-mode and RLE sequence tables"""
    total = {}
    for _, _, fr in _frames():
        for k, v in _block_modes(fr).items():
            total[k] = total.get(k, 0) + v
    assert total["compressed"] >= 150 and total["treeless"] >= 10 and total["repeat"] >= 4 and total["rle_offsets"] >= 10, total


def _digest(a):
    return hashlib.blake2b(a.tobytes(), digest_size=8).hexdigest()


def _ref_verdict(ref, frame, cap):
    """ZSTD_decompress() with `cap` bytes of room: the decoded bytes, or None when it refuses."""
    out = np.zeros(cap + 16, np.uint8)
    r = ref.ZSTD_decompress(ptr(out), cap, ptr(frame), len(frame))
    return None if ref.ZSTD_isError(r) else out[:r]


def _frame_verdicts(decode):
    """decode(frame, cap) -> the decoded bytes or None, for every stored frame and three room sizes"""
    t = Transcript()
    for name, d, fr in _frames():
        t.group(name)
        for cap in (len(d), len(d) + 9, max(len(d) - 1, 0)):
            got = decode(fr, cap)
            t.add(-1) if got is None else t.add(len(got), got)
    return t


def test_zstd_frames_emu(emu):
    emu.emu_zstd_decode.restype = C.c_int

    def decode(fr, cap):
        out = np.full(cap + 16, 0x77, np.uint8)
        r = emu.emu_zstd_decode(ptr(fr), ci(len(fr)), ptr(out), ci(cap))
        assert (out[cap:] == 0x77).all() and r >= -1
        return None if r == -1 else out[:r]
    check_transcript("zstd_frames", _frame_verdicts(decode))


def _damaged():
    """(name, original, damaged frame): truncations, bit flips in the header, trailing bytes, random bytes"""
    rng = np.random.default_rng(21)
    for name, d, fr in _frames():
        if len(d) > 310000 or len(fr) < 12 or not any(t in name for t in ("l3", "l19", "cksum")):
            continue
        for trial in range(20):
            c = fr.copy()
            kind = trial % 5
            if kind == 0:
                c = c[:rng.integers(1, len(c))]
            elif kind == 1:
                c[rng.integers(0, min(len(c), 16))] ^= 1 << rng.integers(0, 8)
            elif kind == 2:
                c = np.concatenate([c, rng.integers(0, 256, 3, dtype=np.uint8)])
            else:
                for pos in rng.integers(0, len(c), kind - 2):
                    c[pos] = rng.integers(0, 256)
            yield name, trial, kind, d, c


def test_zstd_rejects_what_zstd_rejects_emu(emu):
    emu.emu_zstd_decode.restype = C.c_int
    nbad = ngood = nstrict = 0
    verdicts = golden()["zstd_damaged_verdicts"]
    cases = list(_damaged())
    assert len(cases) == len(verdicts)
    for (name, trial, kind, d, c), (want_n, want_digest) in zip(cases, verdicts):
        out = np.full(len(d) + 16, 0x77, np.uint8)
        r = emu.emu_zstd_decode(ptr(c), ci(len(c)), ptr(out), ci(len(d)))
        if want_n < 0:
            assert r == -1, (name, trial, kind, r)
            nbad += 1
        elif r == -1:
            # zstd's table-driven Huffman fast loops do not verify that a damaged literal stream is
            # used up exactly (they then emit garbage); this decoder does, and refuses such frames
            assert emu.emu_zstd_fail_line() > 0
            nstrict += 1
        else:
            assert r == want_n and _digest(out[:r]) == want_digest, (name, trial, kind, r)
            ngood += 1
        assert (out[len(d):] == 0x77).all()
    assert nbad > 200 and nstrict <= nbad // 20, (nbad, ngood, nstrict)


def _compat_zstd_files():
    return sorted(f for f in glob.glob(os.path.join(ROOT, "tests", "golden", "compat", "*.cdata")) if "zstd" in f)


COMPAT_DIVS = (2, 3, 5)
CHUNKS = [(kind, n, ts, shuf, clevel) for kind, n in (("bench", 6000), ("text", 3001), ("mixed", 6000), ("rand", 1000))
          for ts, shuf, clevel in ((4, 1, 5), (8, 2, 1), (1, 0, 9), (3, 1, 6))]
ARANGE = np.arange(1000000, dtype=np.int32).view(np.uint8)


def _chunk_key(kind, n, ts, shuf, clevel):
    return f"chunk-{kind}-{n}-{ts}-{shuf}-{clevel}"


def _damaged_compat():
    for f in _compat_zstd_files():
        chunk = np.fromfile(f, np.uint8)
        for div in COMPAT_DIVS:                                 # no checksum in these frames: damage may go unnoticed
            bad = chunk.copy(); bad[len(bad) // div] ^= 0x55
            yield f"{os.path.basename(f)}/{div}", bad


def _check_damaged_compat(decode, divs):
    """decode(chunk, out) -> return value; against the reference's stored verdict on the same damaged chunk"""
    want = golden()["zstd_compat_damaged"]
    for key, bad in _damaged_compat():
        if int(key.rsplit("/", 1)[1]) not in divs:
            continue
        out = np.zeros(4000000 + 64, np.uint8)
        r = decode(bad, out)
        r_ref, ref_digest = want[key]
        if r_ref < 0:
            assert r == -1, key
        elif r >= 0:
            assert r == r_ref and _digest(out[:r]) == ref_digest, key


def test_compat_zstd_goldens_and_reference_chunks_emu(emu):
    files = _compat_zstd_files()
    assert len(files) == 3
    for f in files:
        chunk = np.fromfile(f, np.uint8)
        out = np.zeros(4000000 + 64, np.uint8)
        assert emu.blosc_decompress_ctx(ptr(chunk), ptr(out), sz(4000000), ci(1)) == 4000000, f
        assert (out[:4000000] == ARANGE).all()
    _check_damaged_compat(lambda bad, out: emu.blosc_decompress_ctx(ptr(bad), ptr(out), sz(4000000), ci(1)), (2, 3))
    stored = golden_arrays("zstd")
    for kind, n, ts, shuf, clevel in CHUNKS:
        src, chunk = gen(kind, n, 4), stored[_chunk_key(kind, n, ts, shuf, clevel)]
        r, out = decompress(emu, "blosc_decompress_ctx", chunk, n)
        assert r == n and (out[:n] == src).all() and (out[n:] == 0).all(), (kind, ts, shuf, clevel)
    # getitem decodes only the blocks it needs (one zstd frame per block)
    chunk = stored["chunk-arange"]
    emu.blosc_getitem.restype = C.c_int
    for start, nitems in ((0, 10), (65000, 3000), (999000, 1000), (131071, 2)):
        item = np.full(nitems * 4 + 8, 0x33, np.uint8)
        assert emu.blosc_getitem(ptr(chunk), ci(start), ci(nitems), ptr(item)) == nitems * 4
        assert (item[:nitems * 4] == ARANGE[start * 4:(start + nitems) * 4]).all() and (item[nitems * 4:] == 0x33).all()
    out = np.zeros(2000 + 64, np.uint8)
    assert emu.blosc_compress_ctx(ci(5), ci(1), sz(4), sz(1000), ptr(ARANGE), ptr(out), sz(2000), b"zstd", sz(0), ci(1)) == -5   # decode only


@pytest.mark.gpu
def test_compat_zstd_goldens_gpu(pkg, cuda):
    files = _compat_zstd_files()
    assert len(files) == 3
    for f in files:
        chunk = np.fromfile(f, np.uint8)
        out = np.zeros(4000000 + 64, np.uint8)
        assert pkg.decompress_ctx(chunk, out, 4000000) == 4000000, f
        assert (out[:4000000] == ARANGE).all() and (out[4000000:] == 0).all()
    # zstd frames carry no checksum here: damage may go unnoticed, in which case both decoders must produce the same bytes
    _check_damaged_compat(lambda bad, out: pkg.decompress_ctx(bad, out, 4000000), COMPAT_DIVS)


LARGE = (("bench", 4 << 20), ("text", 300001), ("mixed", 1 << 20))       # up to 16 blocks of realistic data


@pytest.mark.gpu
def test_zstd_chunks_from_the_reference_gpu(pkg, ref, cuda):
    """the stored chunks; where oracle/_ref was built, also chunks of several MiB the reference writes on the spot"""
    if ref is not None:
        _zstd(ref)
        for kind, n in LARGE:
            src = gen(kind, n, 4)
            for ts, shuf, clevel in ((4, 1, 5), (8, 2, 1), (1, 0, 9), (3, 1, 6)):
                cb, chunk = compress(ref, "blosc_compress_ctx", clevel, shuf, ts, src, n + 16, "zstd")
                assert cb > 0
                out = np.zeros(n + 64, np.uint8)
                assert pkg.decompress_ctx(chunk, out, n) == n
                assert (out[:n] == src).all() and (out[n:] == 0).all(), (kind, ts, shuf, clevel)
    stored = golden_arrays("zstd")
    for kind, n, ts, shuf, clevel in CHUNKS:
        src, chunk = gen(kind, n, 4), stored[_chunk_key(kind, n, ts, shuf, clevel)]
        out = np.zeros(n + 64, np.uint8)
        assert pkg.decompress_ctx(chunk, out, n) == n
        assert (out[:n] == src).all() and (out[n:] == 0).all()
    out = np.zeros(len(ARANGE) + 64, np.uint8)
    assert pkg.decompress_ctx(stored["chunk-arange"], out, len(ARANGE)) == len(ARANGE) and (out[:len(ARANGE)] == ARANGE).all()


def reference_golden(ref, orc):
    ref = _zstd(ref)
    arrays = _write_frames(ref)
    for kind, n, ts, shuf, clevel in CHUNKS:
        src = gen(kind, n, 4)
        cb, chunk = compress(ref, "blosc_compress_ctx", clevel, shuf, ts, src, n + 16, "zstd")
        assert cb > 0 and decompress(ref, "blosc_decompress_ctx", chunk, n)[0] == n
        arrays[_chunk_key(kind, n, ts, shuf, clevel)] = chunk[:cb].copy()
    cb, chunk = compress(ref, "blosc_compress_ctx", 5, 1, 4, ARANGE, len(ARANGE) + 16, "zstd")
    arrays["chunk-arange"] = chunk[:cb].copy()
    return arrays


def reference_verdicts(ref, orc):
    """Run after the frames are stored: the reference's verdicts on them and on damaged copies."""
    ref = _zstd(ref)
    t = _frame_verdicts(lambda fr, cap: _ref_verdict(ref, fr, cap))
    damaged = []
    for name, trial, kind, d, c in _damaged():
        got = _ref_verdict(ref, c, len(d))
        damaged.append([-1, ""] if got is None else [len(got), _digest(got)])
    compat = {}
    for key, bad in _damaged_compat():
        r, out = decompress(ref, "blosc_decompress_ctx", bad, 4000000)
        compat[key] = [r, _digest(out[:max(r, 0)])]
    return {"transcripts": {"zstd_frames": t.digests()}, "zstd_damaged_verdicts": damaged, "zstd_compat_damaged": compat}
