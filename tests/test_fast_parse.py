"""The segment-parallel LZ4 parse (BLOSC_B200_PARSE=fast, csrc/dev_lz4fast.cuh).

Its chunks are not the reference's bytes, so parity is what north_star asks of a compressor: the
oracle (whose decoder is pinned to the reference's by test_oracle_vs_ref.py and test_hostile_input.py)
and, where oracle/_ref was built, the UNMODIFIED reference itself decode every chunk to the original bytes, the chunk header / bstarts / split prefixes are
well-formed, nothing is written past the returned size, and the ratio on the bench.c planes is
not worse than the reference's own (BASELINE.md: 7.11 / 13.16 / 36.70 / 26.32 at typesize 2/4/8/16).
The reference's own sizes and chunk headers are stored in tests/golden/reference.json.
CPU: the device code runs in the SIMT emulator.  GPU: through the C ABI of libblosc_b200.so."""
import os

import numpy as np
import pytest

from datagen import compress, decompress, gen, golden

KINDS = ("bench", "rand", "zeros", "lowent", "text", "ramp", "i32", "f32", "mixed")


@pytest.fixture()
def fast_env():
    old = os.environ.get("BLOSC_B200_PARSE")
    os.environ["BLOSC_B200_PARSE"] = "fast"
    yield
    if old is None:
        os.environ.pop("BLOSC_B200_PARSE", None)
    else:
        os.environ["BLOSC_B200_PARSE"] = old


def _decoders(orc, ref):
    return [(orc, "orc_decompress_ctx")] + ([(ref, "blosc_decompress_ctx")] if ref else [])


def _check(chunk, r, n, src, decoders):
    assert r > 0
    assert (chunk[r:] == 0xAA).all(), "wrote past the returned size"
    assert int.from_bytes(bytes(chunk[4:8]), "little") == n and int.from_bytes(bytes(chunk[12:16]), "little") == r
    for lib, fn in decoders:
        dn, out = decompress(lib, fn, chunk, n)
        assert dn == n and (out[:n] == src).all(), fn


@pytest.mark.parametrize("kind", KINDS)
def test_emu_fast_chunks_decode_with_the_reference(emu, ref, orc, fast_env, kind):
    for n in (1 << 20, 300001, 65536 + 77, 4096 + 5, 1000, 200, 13):
        src = gen(kind, n, seed=n & 7)
        for ts, shuf, clevel in ((4, 1, 5), (1, 0, 5), (8, 1, 9), (2, 2, 1), (16, 1, 5), (3, 1, 5)):
            r, chunk = compress(emu, "blosc_compress_ctx", clevel, shuf, ts, src, n + 16, "lz4")
            _check(chunk, r, n, src, _decoders(orc, ref) + [(emu, "blosc_decompress_ctx")])


def test_emu_fast_odd_shapes(emu, ref, orc, fast_env):
    """unaligned sources, forced block sizes (unsplit streams longer than a group of 32 segments), tiny destsize"""
    base = gen("bench", (1 << 20) + 64)
    for off in (1, 2, 3):
        src = base[off:off + 500001].copy()
        r, chunk = compress(emu, "blosc_compress_ctx", 5, 0, 1, src, len(src) + 16, "lz4")
        _check(chunk, r, len(src), src, _decoders(orc, ref))
    src = gen("i32", 1 << 20)
    for bs in (4096, 100000, 1 << 19):
        r, chunk = compress(emu, "blosc_compress_ctx", 5, 1, 32, src, len(src) + 16, "lz4", bs)   # typesize 32: never split
        _check(chunk, r, len(src), src, _decoders(orc, ref))
    # a destination that is too small for the compressed chunk: 0, as blosc_compress (test_maxout.c)
    src = gen("rand", 100000)
    r, _ = compress(emu, "blosc_compress_ctx", 5, 1, 4, src, 100000 + 15, "lz4")
    assert r == 0
    src = gen("bench", 1 << 20)
    full, _ = compress(emu, "blosc_compress_ctx", 5, 1, 4, src, len(src) + 16, "lz4")
    r, chunk = compress(emu, "blosc_compress_ctx", 5, 1, 4, src, full, "lz4")
    assert r in (0, full)
    r, _ = compress(emu, "blosc_compress_ctx", 5, 1, 4, src, full - 1, "lz4")
    assert r == 0


RATIO_TS = (2, 4, 8, 16)


def test_emu_fast_ratio_on_bench_planes(emu, fast_env):
    """not worse than the reference's own ratio on the data BASELINE.json is quoted on"""
    n = 4 << 20
    src = gen("bench", n)
    for ts, want in zip(RATIO_TS, golden()["fast_parse_ratio_cbytes"]):
        got, _ = compress(emu, "blosc_compress_ctx", 5, 1, ts, src, n + 16, "lz4")
        assert 0 < got <= want * 1.02, (ts, got, want)


def test_emu_fast_is_opt_in(emu, orc):
    """without the variable the chunk is the reference's, byte for byte"""
    os.environ.pop("BLOSC_B200_PARSE", None)
    src = gen("bench", 1 << 20)
    w, want = compress(orc, "orc_compress_ctx", 5, 1, 4, src, len(src) + 16, "lz4")
    g, got = compress(emu, "blosc_compress_ctx", 5, 1, 4, src, len(src) + 16, "lz4")
    assert g == w and (got[:g] == want[:w]).all()


LZ4HC_EMU = [(kind, n, ts, shuf, clevel) for kind in ("bench", "f32", "i32", "lowent", "zeros", "mixed", "rand", "text")
             for n in (1 << 20, 300001, 5000) for ts, shuf, clevel in ((4, 1, 5), (8, 1, 9), (1, 0, 1), (2, 2, 3))]
LZ4HC_GPU = [(kind, n, ts, shuf, clevel) for kind in ("bench", "f32", "zeros", "mixed", "rand")
             for n in (4 << 20, 300001) for ts, shuf, clevel in ((4, 1, 5), (8, 1, 9), (2, 2, 3))]


def _lz4hc_key(kind, n, ts, shuf, clevel):
    return f"{kind}/{n}/{ts}/{shuf}/{clevel}"


def _check_lz4hc(lib, decoders, kind, src, ts, shuf, clevel, gpu=None):
    n = len(src)
    want_n, want = golden()["lz4hc_chunks"][_lz4hc_key(kind, n, ts, shuf, clevel)]   # size and first 12 bytes
    want = bytes.fromhex(want)
    if gpu is None:
        r, chunk = compress(lib, "blosc_compress_ctx", clevel, shuf, ts, src, n + 16, "lz4hc")
    else:
        r, chunk = gpu
    assert r > 0 and (chunk[r:] == 0xAA).all()
    for dlib, fn in decoders:
        dn, out = decompress(dlib, fn, chunk, n)
        assert dn == n and (out[:n] == src).all(), fn
    memcpyed = lambda c: bool(c[2] & 0x2)
    if not memcpyed(chunk) and not memcpyed(want):
        # same header as the reference's lz4hc chunk: format version, LZ4 format id + flags, typesize, nbytes, blocksize
        assert bytes(chunk[:12]) == want, (bytes(chunk[:12]).hex(), want.hex())
    return r, want_n


def test_emu_lz4hc_chunks(emu, ref, orc):
    """SURVEY.md section 8 row f4: blosc_compress_ctx(..., "lz4hc", ...) (blosc.c:422-433).  The chunks are LZ4-format
    (LZ4HC and LZ4 share it, blosc.h:96) from the hash-chain parser run with LZ4HC's search effort; the reference decodes
    them, the header is the reference's, and the size stays within 1.6x of LZ4_compress_HC's on compressible data."""
    os.environ.pop("BLOSC_B200_PARSE", None)
    for kind, n, ts, shuf, clevel in LZ4HC_EMU:
        src = gen(kind, n)
        got, want = _check_lz4hc(emu, _decoders(orc, ref), kind, src, ts, shuf, clevel)
        if kind in ("bench", "i32", "lowent", "zeros", "mixed") and n >= 300001 and want < n // 2:
            assert got <= 1.6 * want, (kind, n, ts, shuf, clevel, got, want)


# ---------------------------------------------------------------- GPU
def _gpu_compress(pkg, clevel, shuf, ts, src, destsize, comp, bs=0):
    dest = np.full(destsize + 64, 0xAA, np.uint8)
    r = pkg.compress_ctx(clevel, shuf, ts, len(src), src, dest, destsize, comp, bs, 4)
    return r, dest


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_gpu_fast_chunks_decode_with_the_oracle(pkg, orc, cuda, fast_env, kind):
    ref_path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "libblosc_ref.so")
    decoders = [(orc, "orc_decompress_ctx")]
    if os.path.exists(ref_path):
        import ctypes as C
        lib = C.CDLL(ref_path)
        lib.blosc_decompress_ctx.restype = C.c_int
        decoders.append((lib, "blosc_decompress_ctx"))
    for n in (4 << 20, 1000000, 300001, 65536 + 77, 4096 + 5, 1000, 200):
        src = gen(kind, n, seed=n & 7)
        for ts, shuf, clevel in ((4, 1, 5), (1, 0, 5), (8, 1, 9), (2, 2, 1), (16, 1, 5), (3, 1, 5), (2, 1, 5)):
            r, chunk = _gpu_compress(pkg, clevel, shuf, ts, src, n + 16, "lz4")
            _check(chunk, r, n, src, decoders)
            out = np.zeros(n + 64, np.uint8)
            assert pkg.decompress_ctx(chunk, out, n) == n and (out[:n] == src).all()


@pytest.mark.gpu
def test_gpu_lz4hc_chunks(pkg, emu, orc, ref, cuda):
    os.environ.pop("BLOSC_B200_PARSE", None)
    for kind, n, ts, shuf, clevel in LZ4HC_GPU:
        src = gen(kind, n)
        g = _gpu_compress(pkg, clevel, shuf, ts, src, n + 16, "lz4hc")
        _check_lz4hc(None, _decoders(orc, ref), kind, src, ts, shuf, clevel, gpu=g)
        w, want = compress(emu, "blosc_compress_ctx", clevel, shuf, ts, src, n + 16, "lz4hc")
        assert g[0] == w and (g[1][:w] == want[:w]).all()          # deterministic: GPU == emulator
        out = np.zeros(n + 64, np.uint8)
        assert pkg.decompress_ctx(g[1], out, n) == n and (out[:n] == src).all()


@pytest.mark.gpu
def test_gpu_fast_equals_emulator(pkg, emu, cuda, fast_env):
    """the parse is deterministic: the GPU writes what the emulator writes"""
    for kind, n, ts, shuf in (("bench", 4 << 20, 4, 1), ("f32", 1000000, 8, 1), ("mixed", 1 << 20, 2, 2), ("text", 300001, 1, 0)):
        src = gen(kind, n)
        w, want = compress(emu, "blosc_compress_ctx", 5, shuf, ts, src, n + 16, "lz4")
        g, got = _gpu_compress(pkg, 5, shuf, ts, src, n + 16, "lz4")
        assert g == w and (got[:g] == want[:w]).all(), (kind, n)


@pytest.mark.gpu
def test_gpu_fast_full_size_ratio_and_round_trip(pkg, cuda, fast_env):
    """BASELINE.json configs[1] and the typesize sweep of configs[4], device resident, 256 MiB"""
    torch = cuda
    n = 256 << 20
    d_src = torch.from_numpy(gen("bench", n)).cuda()
    d_chunk = torch.zeros(n + 16, dtype=torch.uint8, device="cuda")
    d_out = torch.zeros(n, dtype=torch.uint8, device="cuda")
    for ts, ref_cbytes in ((2, 37749776), (4, 20401680), (8, 7313680), (16, 10199056)):
        cb = pkg.compress_ctx(5, 1, ts, n, d_src, d_chunk, n + 16, "lz4")
        assert 0 < cb <= ref_cbytes * 1.02, (ts, cb, ref_cbytes)
        d_out.zero_()
        assert pkg.decompress_ctx(d_chunk, d_out, n) == n
        assert torch.equal(d_out, d_src)


def test_emu_frames_with_fast_parse_and_lz4hc(emu, ref, orc, fast_env):
    """frames (several chunks in flight, each with its own chain index and segment records) written with the fast parse
    and with "lz4hc": every chunk of the frame decodes on its own (oracle, and the reference where built), the frame
    round-trips"""
    import ctypes as C
    sz, ci, ll = C.c_size_t, C.c_int, C.c_longlong
    emu.blosc_b200_frame_bound.restype = sz; emu.blosc_b200_frame_bound.argtypes = [sz, sz, sz]
    emu.blosc_b200_frame_compress.restype = ll
    emu.blosc_b200_frame_compress.argtypes = [ci, ci, sz, sz, C.c_void_p, C.c_void_p, sz, C.c_char_p, sz, sz, ci]
    emu.blosc_b200_frame_decompress.restype = ll; emu.blosc_b200_frame_decompress.argtypes = [C.c_void_p, sz, C.c_void_p, sz, ci]
    emu.blosc_b200_frame_chunk.restype = ll; emu.blosc_b200_frame_chunk.argtypes = [C.c_void_p, sz, sz, C.POINTER(sz)]
    n, cs = 1000003, 1 << 18
    for kind, comp, ts, shuf in (("bench", "lz4", 4, 1), ("mixed", "lz4hc", 8, 1), ("f32", "lz4", 2, 2)):
        src = gen(kind, n)
        bound = emu.blosc_b200_frame_bound(n, ts, cs)
        frame = np.full(bound + 64, 0xAA, np.uint8)
        fb = emu.blosc_b200_frame_compress(5, shuf, ts, n, src.ctypes.data, frame.ctypes.data, bound, comp.encode(), 0, cs, 4)
        assert fb > 0 and (frame[fb:] == 0xAA).all()
        ccs = cs - (cs % ts if ts > 1 else 0)
        for i in range((n + ccs - 1) // ccs):
            cb = sz(0)
            off = emu.blosc_b200_frame_chunk(frame.ctypes.data, fb, i, C.byref(cb))
            piece = src[i * ccs:(i + 1) * ccs]
            for dlib, fn in _decoders(orc, ref):
                dn, out = decompress(dlib, fn, frame[off:off + cb.value].copy(), len(piece))
                assert dn == len(piece) and (out[:len(piece)] == piece).all(), (kind, i, fn)
        back = np.zeros(n + 64, np.uint8)
        assert emu.blosc_b200_frame_decompress(frame.ctypes.data, fb, back.ctypes.data, n, 1) == n and (back[:n] == src).all()


def _synth(rng, n):
    """runs, noise, short periods, copies from far back, staircases, low-entropy bytes -- in random order and lengths"""
    out = np.zeros(n, np.uint8)
    p = 0
    while p < n:
        k, L = int(rng.integers(0, 6)), int(min(rng.integers(1, 5000), n - p))
        if k == 0:
            out[p:p + L] = rng.integers(0, 256)
        elif k == 1:
            out[p:p + L] = rng.integers(0, 256, L)
        elif k == 2:
            out[p:p + L] = np.resize(rng.integers(0, 256, int(rng.integers(1, 300)), dtype=np.uint8), L)
        elif k == 3 and p > 10:
            off = int(rng.integers(1, min(p, 70000)))
            for i in range(L):
                out[p + i] = out[p + i - off]
        elif k == 4:
            out[p:p + L] = (np.arange(L) // int(rng.integers(1, 9))) % 251
        else:
            out[p:p + L] = rng.integers(0, 4, L)
        p += L
    return out


def test_emu_fast_parse_fuzz(emu, ref, orc, fast_env):
    """differential fuzz (a longer run of the same generator, 8 800 cases, found nothing): random structure, sizes,
    typesizes, filters, levels, forced block sizes, "lz4" and "lz4hc" -- the oracle (and the reference where built)
    must decode every chunk"""
    rng = np.random.default_rng(7)
    for _ in range(160):
        n = int(rng.choice([13, 100, 1000, 4097, 70001, 200003]))
        src = _synth(rng, n)
        ts, shuf, cl = int(rng.choice([1, 2, 3, 4, 8, 16, 32])), int(rng.integers(0, 3)), int(rng.integers(1, 10))
        comp, bs = str(rng.choice(["lz4", "lz4hc"])), int(rng.choice([0, 0, 0, 4096, 100000]))
        r, chunk = compress(emu, "blosc_compress_ctx", cl, shuf, ts, src, n + 16, comp, bs)
        assert r > 0 and (chunk[r:] == 0xAA).all(), (n, ts, shuf, cl, comp, bs)
        for dlib, fn in _decoders(orc, ref):
            dn, out = decompress(dlib, fn, chunk, n)
            assert dn == n and (out[:n] == src).all(), (n, ts, shuf, cl, comp, bs, fn)


def reference_golden(ref, orc):
    src = gen("bench", 4 << 20)
    ratio = [compress(ref, "blosc_compress_ctx", 5, 1, ts, src, len(src) + 16, "lz4")[0] for ts in RATIO_TS]
    hc = {}
    for kind, n, ts, shuf, clevel in sorted(set(LZ4HC_EMU + LZ4HC_GPU)):
        r, chunk = compress(ref, "blosc_compress_ctx", clevel, shuf, ts, gen(kind, n), n + 16, "lz4hc")
        hc[_lz4hc_key(kind, n, ts, shuf, clevel)] = [r, bytes(chunk[:12]).hex()]
    return {"fast_parse_ratio_cbytes": ratio, "lz4hc_chunks": hc}
