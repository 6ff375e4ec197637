"""CPU tests of the PRODUCT's device code: the kernels of c-blosc_b200/csrc/dev_*.cuh compiled
with g++ and run in the lock-step SIMT emulator (tests/emu), and the product's host code
(blosc_b200.c) linked against that emulated backend.  Everything is compared with the oracle,
bit for bit.  (The real CUDA build is exercised by the -m gpu tests.)"""
import numpy as np
import pytest

from datagen import ci, compress, decompress, gen, ptr, sz

KINDS = ["bench", "rand", "zeros", "lowent", "text", "i32", "mixed"]


@pytest.mark.parametrize("kind", KINDS)
def test_lz4_warp_codec(emu, orc, kind):
    for n in [0, 1, 12, 13, 16, 33, 67, 255, 1000, 5000, 65546, 65547, 100000]:
        src = gen(kind, n, seed=n)
        for accel, cap in ((5, n), (1, n), (9, n // 2), (5, n + n // 255 + 16), (5, 70)):
            a = np.zeros(cap + 64, np.uint8); b = np.zeros(cap + 64, np.uint8)
            ra = orc.orc_lz4_compress_fast(ptr(src), ptr(a), ci(n), ci(cap), ci(accel))
            rb = emu.emu_lz4_encode(ptr(src), ci(n), ptr(b), ci(cap), ci(accel))
            assert ra == rb, (kind, n, accel, cap, ra, rb)
            if ra > 0:
                assert (a[:ra] == b[:ra]).all() and (b[ra:] == 0).all()
                for c2 in (n, n + 3, max(n - 1, 0)):
                    o1 = np.zeros(n + 8, np.uint8); o2 = np.zeros(n + 8, np.uint8)
                    d1 = orc.orc_lz4_decompress_safe(ptr(a), ptr(o1), ci(ra), ci(c2))
                    d2 = emu.emu_lz4_decode(ptr(a), ci(ra), ptr(o2), ci(c2))
                    assert (d1 < 0) == (d2 < 0) and (d1 < 0 or d1 == d2)
                    if c2 == n:
                        assert d2 == n and (o2[:n] == src).all() and (o2[n:] == 0).all()


@pytest.mark.parametrize("kind", KINDS)
def test_blosclz_warp_codec(emu, orc, kind):
    for n in [0, 15, 16, 17, 33, 67, 128, 255, 1000, 5000, 16500, 70000]:
        src = gen(kind, n, seed=n)
        for clevel, split, cap in ((5, 1, n), (5, 0, n), (1, 1, n), (2, 0, n), (9, 1, n), (5, 1, n // 2), (5, 1, 66), (5, 1, 65)):
            a = np.zeros(cap + 64, np.uint8); b = np.zeros(cap + 64, np.uint8)
            ra = orc.orc_blosclz_compress(ci(clevel), ptr(src), ci(n), ptr(a), ci(cap), ci(split))
            rb = emu.emu_blz_encode(ci(clevel), ptr(src), ci(n), ptr(b), ci(cap), ci(split))
            assert ra == rb, (kind, n, clevel, split, cap, ra, rb)
            if ra > 0:
                assert (a[:ra] == b[:ra]).all()
                o2 = np.zeros(n + 8, np.uint8)
                assert emu.emu_blz_decode(ptr(a), ci(ra), ptr(o2), ci(n)) == n
                assert (o2[:n] == src).all() and (o2[n:] == 0).all()


def test_decoders_reject_garbage(emu, orc):
    """Corrupted streams: same accept/reject verdict as the oracle, no out-of-bounds write."""
    rng = np.random.default_rng(3)
    src = gen("text", 20000)
    a = np.zeros(20064, np.uint8)
    ra = orc.orc_lz4_compress_fast(ptr(src), ptr(a), ci(20000), ci(20000), ci(1))
    b = np.zeros(20064, np.uint8)
    rb = orc.orc_blosclz_compress(ci(5), ptr(src), ci(20000), ptr(b), ci(20000), ci(1))
    for _ in range(150):
        for buf, n, fo, fe in ((a, ra, "orc_lz4_decompress_safe", "emu_lz4_decode"), (a, ra, "orc_lz4_decompress_safe", "emu_lz4_decode_pair"),
                               (b, rb, "orc_blosclz_decompress", "emu_blz_decode")):
            c = buf[:n].copy()
            pos = rng.integers(0, n, 4)
            c[pos] = rng.integers(0, 256, 4, dtype=np.uint8)
            o1 = np.zeros(20016, np.uint8); o2 = np.zeros(20016, np.uint8)
            if fo.startswith("orc_lz4"):
                d1 = getattr(orc, fo)(ptr(c), ptr(o1), ci(n), ci(20000)); d2 = getattr(emu, fe)(ptr(c), ci(n), ptr(o2), ci(20000))
            else:
                d1 = getattr(orc, fo)(ptr(c), ci(n), ptr(o1), ci(20000)); d2 = getattr(emu, fe)(ptr(c), ci(n), ptr(o2), ci(20000))
            assert (d1 <= 0) == (d2 <= 0) or d1 == d2, (fo, d1, d2)
            if d1 > 0 and d1 == d2:
                assert (o1[:d1] == o2[:d1]).all()
            assert (o2[20000:] == 0).all()


@pytest.mark.parametrize("dev", [0, 1])
def test_filter_kernels(emu, orc, dev):
    """dev=1 makes the emulated backend treat caller pointers as device pointers (no staging copy),
    so misaligned user buffers reach the kernels directly."""
    emu.emu_set_all_device(dev)
    try:
        for ts in [1, 2, 3, 4, 5, 8, 16, 17]:
            for n in [0, 1, 7, 8, 64, 500, 1792, 8000, 8192, 32768, 100000, 131072, 131072 + 24]:
                base = gen("rand", n + 3, seed=ts)
                for off in ((0, 1) if dev else (0,)):
                    src = base[off:off + n]
                    for mode, fn in enumerate(["orc_shuffle", "orc_unshuffle", "orc_bitshuffle", "orc_bitunshuffle"]):
                        if mode >= 2 and n < ts:
                            continue
                        a = np.zeros(n + 1, np.uint8); b = np.zeros(n + 1, np.uint8)
                        getattr(orc, fn)(sz(ts), sz(n), ptr(src), ptr(a))
                        assert emu.blosc_b200_filter(ci(mode), sz(ts), sz(n), ptr(src), ptr(b)) == 0
                        assert (a == b).all(), (fn, ts, n, dev, off)
    finally:
        emu.emu_set_all_device(0)


@pytest.mark.parametrize("kind", ["bench", "i32", "mixed", "rand"])
def test_library_against_oracle(emu, orc, kind):
    """Host framing + every kernel: chunks identical to the oracle's, decode, getitem."""
    for dev in (0, 1):
        emu.emu_set_all_device(dev)
        try:
            for n in ([0, 1, 100, 128, 129, 1000, 4096, 32768, 100000, 300000] if dev == 0 else [129, 4096, 100000]):
                src = gen(kind, n, seed=n)
                for comp in ("lz4", "blosclz"):
                    for ts, shuf, clevel, bs in ((4, 1, 5, 0), (8, 2, 5, 0), (1, 0, 5, 0), (2, 1, 9, 0), (16, 1, 1, 0), (7, 1, 5, 0), (17, 2, 5, 0),
                                                 (4, 2, 5, 4096), (4, 1, 0, 0), (256, 1, 5, 0), (3, 2, 9, 100)):
                        ra, a = compress(orc, "orc_compress_ctx", clevel, shuf, ts, src, n + 16, comp, bs)
                        rb, b = compress(emu, "blosc_compress_ctx", clevel, shuf, ts, src, n + 16, comp, bs)
                        assert ra == rb, (kind, n, comp, ts, shuf, clevel, bs, ra, rb)
                        if ra <= 0:
                            continue
                        assert (a[:ra] == b[:ra]).all() and (b[ra:] == 0xAA).all()
                        d2, o2 = decompress(emu, "blosc_decompress_ctx", a, n)
                        assert d2 == n and (o2[:n] == src).all()
                        if 0 < n <= 100000:
                            nit = n // int(a[3])
                            for st, cnt in ((0, nit), (nit // 3, nit // 2), (nit - 1, 1), (0, 0)):
                                g1 = np.zeros(n + 8, np.uint8); g2 = np.zeros(n + 8, np.uint8)
                                r1 = orc.orc_getitem(ptr(a), ci(st), ci(cnt), ptr(g1))
                                r2 = emu.blosc_getitem(ptr(a), ci(st), ci(cnt), ptr(g2))
                                assert r1 == r2 and (g1 == g2).all()
        finally:
            emu.emu_set_all_device(0)


def test_library_error_codes(emu):
    src = gen("rand", 100000)
    n = len(src)
    assert compress(emu, "blosc_compress_ctx", 5, 1, 4, src, n + 15, "lz4")[0] == 0
    assert compress(emu, "blosc_compress_ctx", 5, 1, 4, src, n + 16, "lz4")[0] == n + 16
    assert compress(emu, "blosc_compress_ctx", 5, 1, 4, src, 15, "lz4")[0] == 0
    assert compress(emu, "blosc_compress_ctx", 11, 1, 4, src, n + 16, "lz4")[0] == -10
    assert compress(emu, "blosc_compress_ctx", 5, 4, 4, src, n + 16, "lz4")[0] == -10
    assert compress(emu, "blosc_compress_ctx", 5, 1, 0, src, n + 16, "lz4")[0] == -10
    assert compress(emu, "blosc_compress_ctx", 5, 1, 4, src, n + 16, "zstd")[0] == -5
    big = gen("rand", 300000)      # > 1 block, so the reference would take the pool path and validate nthreads
    assert compress(emu, "blosc_compress_ctx", 5, 0, 1, big, len(big) + 16, "lz4", 0, 0)[0] == -1
    assert compress(emu, "blosc_compress_ctx", 5, 0, 1, big, len(big) + 16, "lz4", 0, 257)[0] == -1
    assert compress(emu, "blosc_compress_ctx", 5, 1, 4, src, n + 16, "lz4", 0, 0)[0] == n + 16   # single block: serial path, no check
    cb, chunk = compress(emu, "blosc_compress_ctx", 5, 1, 4, gen("bench", n), n + 16, "lz4")
    c = chunk.copy(); c[0] = 3
    assert decompress(emu, "blosc_decompress_ctx", c, n)[0] == -1
    c = chunk.copy(); c[1] = 2
    assert decompress(emu, "blosc_decompress_ctx", c, n)[0] == -9
    c = chunk.copy(); c[2] = (c[2] & 0x1f) | (2 << 5)          # snappy: not built, as in the stock reference
    assert decompress(emu, "blosc_decompress_ctx", c, n)[0] == -5
    assert decompress(emu, "blosc_decompress_ctx", chunk, n - 1)[0] == -1
    c = chunk.copy(); c[20:24] = 0xff
    assert decompress(emu, "blosc_decompress_ctx", c, n)[0] == -1


def test_lz4_decoder_paths_are_all_exercised(emu, orc):
    """The batch-parallel, single-sequence and general decode paths must all run (and agree with
    the source) on shuffled bench.c data -- guards against a fast path silently never being taken."""
    import ctypes as C
    counters = (C.c_longlong * 4)()
    src = gen("bench", 1 << 20)
    cb, chunk = compress(orc, "orc_compress_ctx", 5, 1, 4, src, len(src) + 16, "lz4")
    emu.emu_lz4d_counters(counters)
    before = list(counters)
    dn, out = decompress(emu, "blosc_decompress_ctx", chunk, len(src))
    emu.emu_lz4d_counters(counters)
    batch, fast, general, dense = (counters[i] - before[i] for i in range(4))
    assert dn == len(src) and (out[:dn] == src).all()
    assert dense > 10000 and batch > 100 and fast > 0 and general > 0, (batch, fast, general, dense)


def test_pageable_host_staging(emu, orc):
    """Host buffers that are not page-locked go through the pinned bounce slices filled by the copy
    thread pool (blosc_b200.c h2d_any / d2h_any): multi-slice pipeline in both directions."""
    emu.emu_set_all_pinned(0)
    try:
        n = (20 << 20) + 4321                     # > 2 bounce slices each way
        src = gen("bench", n)
        cb, chunk = compress(emu, "blosc_compress_ctx", 5, 1, 4, src, n + 16, "lz4")
        assert cb > 0
        dn, out = decompress(emu, "blosc_decompress_ctx", chunk, n)
        assert dn == n and (out[:n] == src).all()
        rnd = gen("rand", 12 << 20)               # MEMCPYED fallback: the compressed side is large too
        cb, chunk = compress(emu, "blosc_compress_ctx", 5, 1, 4, rnd, len(rnd) + 16, "blosclz")
        assert cb == len(rnd) + 16
        dn, out = decompress(emu, "blosc_decompress_ctx", chunk, len(rnd))
        assert dn == len(rnd) and (out[:dn] == rnd).all()
    finally:
        emu.emu_set_all_pinned(1)


def test_lz4_dense_path_on_corrupted_chains(emu, orc):
    """The dense decoder path (32 literal-free sequences per step) on a byte-plane of shuffled
    bench.c data: same accept/reject verdict and same bytes as the oracle when single bytes of the
    stream are damaged (offsets reaching before the block, overlapping sources, broken tokens)."""
    import ctypes as C
    rng = np.random.default_rng(11)
    words = gen("bench", 1 << 19).view(np.uint32)
    n = len(words)
    best = (0, None, None)
    for b in range(3):                                         # the chain-heavy byte-plane of the shuffle
        pl = ((words >> (8 * b)) & 0xff).astype(np.uint8)
        buf = np.zeros(n + 64, np.uint8)
        r = orc.orc_lz4_compress_fast(ptr(pl), ptr(buf), ci(n), ci(n), ci(5))
        if r > best[0]:
            best = (r, pl, buf)
    ra, plane, a = best
    assert 0 < ra < n // 2
    counters = (C.c_longlong * 4)()
    emu.emu_lz4d_counters(counters)
    dense0 = counters[3]
    o = np.zeros(n + 8, np.uint8)
    assert emu.emu_lz4_decode(ptr(a), ci(ra), ptr(o), ci(n)) == n and (o[:n] == plane).all()
    emu.emu_lz4d_counters(counters)
    assert counters[3] - dense0 > 5000
    for trial in range(120):
        c = a[:ra].copy()
        for pos in rng.integers(0, ra, 1 + trial % 3):
            kind = trial % 4
            c[pos] = (0, 0xF0, 0x0F, int(rng.integers(0, 256)))[kind]
        o1 = np.zeros(n + 8, np.uint8)
        d1 = orc.orc_lz4_decompress_safe(ptr(c), ptr(o1), ci(ra), ci(n))
        for decode in (emu.emu_lz4_decode, emu.emu_lz4_decode_pair):
            o2 = np.zeros(n + 8, np.uint8)
            d2 = decode(ptr(c), ci(ra), ptr(o2), ci(n))
            assert (d1 < 0) == (d2 < 0), (trial, decode.__name__, d1, d2)
            if d1 >= 0:
                assert d1 == d2 and (o1[:d1] == o2[:d1]).all() and (o2[n:] == 0).all(), (trial, decode.__name__)


def test_lz4_decode_unaligned_destination(emu, orc):
    """The decoder stages output in its shared-memory ring and flushes it with 16-byte stores:
    destinations at every phase of a 16-byte line, nothing written outside [dst, dst+n)."""
    import ctypes as C
    for kind, n in (("bench", 70001), ("text", 30011), ("i32", 9000), ("zeros", 5000)):
        src = gen(kind, n, seed=3) if kind != "bench" else (gen("bench", 4 * n).view(np.uint32)[:n] >> 8).astype(np.uint8)
        a = np.zeros(n + 64, np.uint8)
        ra = orc.orc_lz4_compress_fast(ptr(src), ptr(a), ci(n), ci(n + 64), ci(1))
        assert ra > 0
        for shift in (1, 4, 7, 8, 13, 15):
            buf = np.full(n + 64, 0x5A, np.uint8)
            dst = C.c_void_p(buf.ctypes.data + shift)
            assert emu.emu_lz4_decode(ptr(a), ci(ra), dst, ci(n)) == n
            assert (buf[shift:shift + n] == src).all() and (buf[:shift] == 0x5A).all() and (buf[shift + n:] == 0x5A).all()


def test_lz4_packed_table_is_bit_exact(emu, orc, monkeypatch):
    """The 17-bit packed hash table used when several chunks are in flight (frames): same bytes as
    the plain table and the oracle, at stream level and through the library."""
    emu.emu_set_lz4_pack(1)
    try:
        for kind in KINDS:
            for n in (65547, 70001, 131072):
                src = gen(kind, n, seed=n) if kind != "bench" else (gen("bench", 4 * n).view(np.uint32)[:n] >> 8).astype(np.uint8)
                for accel, cap in ((5, n), (1, n), (9, n // 2), (5, n + n // 255 + 16)):
                    a = np.zeros(cap + 64, np.uint8); b = np.zeros(cap + 64, np.uint8)
                    ra = orc.orc_lz4_compress_fast(ptr(src), ptr(a), ci(n), ci(cap), ci(accel))
                    rb = emu.emu_lz4_encode(ptr(src), ci(n), ptr(b), ci(cap), ci(accel))
                    assert ra == rb and (ra <= 0 or (a[:ra] == b[:ra]).all()), (kind, n, accel, cap, ra, rb)
    finally:
        emu.emu_set_lz4_pack(0)
    monkeypatch.setenv("BLOSC_B200_LZ4_PACK", "1")
    for kind, n, ts in (("bench", 2 << 20, 4), ("mixed", 1 << 20, 2), ("text", (1 << 20) + 4096, 8)):
        src = gen(kind, n, 3)
        r1, c1 = compress(emu, "blosc_compress_ctx", 5, 1, ts, src, n + 16, "lz4")
        r2, c2 = compress(orc, "orc_compress_ctx", 5, 1, ts, src, n + 16, "lz4")
        assert r1 == r2 and (c1[:r1] == c2[:r2]).all(), (kind, n, ts)


def test_lz4_pair_decoder_equals_single_warp_decoder(emu, orc):
    """lz4_pair_parse + lz4_pair_copier (parser warp + copier warp per stream) against lz4_decode_warp and the oracle: same bytes on valid
    streams of every kind and size, same accept / reject verdict (and same bytes when accepted) on damaged ones."""
    emu.emu_lz4_decode_pair.restype = ci
    rng = np.random.default_rng(5)
    for kind in ("bench", "text", "zeros", "lowent", "mixed", "rand", "i32", "f32"):
        for n in (13, 200, 4097, 70001, 300000):
            src = gen(kind, n, seed=n & 3)
            a = np.zeros(n + n // 255 + 64, np.uint8)
            ra = orc.orc_lz4_compress_fast(ptr(src), ptr(a), ci(n), ci(len(a)), ci(1 + (n & 7)))
            assert ra > 0
            o1, o2 = np.full(n + 8, 0x55, np.uint8), np.full(n + 8, 0x55, np.uint8)
            assert emu.emu_lz4_decode_pair(ptr(a), ci(ra), ptr(o2), ci(n)) == n and (o2[:n] == src).all() and (o2[n:] == 0x55).all()
            # wrong capacity, truncated input
            assert emu.emu_lz4_decode_pair(ptr(a), ci(ra), ptr(o2), ci(n - 1)) == emu.emu_lz4_decode(ptr(a), ci(ra), ptr(o1), ci(n - 1))
            assert emu.emu_lz4_decode_pair(ptr(a), ci(ra - 1), ptr(o2), ci(n)) == emu.emu_lz4_decode(ptr(a), ci(ra - 1), ptr(o1), ci(n))
            for trial in range(12):
                c = a[:ra].copy()
                for pos in rng.integers(0, ra, 1 + trial % 3):
                    c[pos] = (0, 0xF0, 0x0F, int(rng.integers(0, 256)))[trial % 4]
                o1[:] = 0x55; o2[:] = 0x55
                d1 = emu.emu_lz4_decode(ptr(c), ci(ra), ptr(o1), ci(n))
                d2 = emu.emu_lz4_decode_pair(ptr(c), ci(ra), ptr(o2), ci(n))
                assert d1 == d2, (kind, n, trial, d1, d2)
                if d1 >= 0:
                    assert (o1[:n] == o2[:n]).all()
                assert (o2[n:] == 0x55).all()


def test_chunks_decode_with_one_warp_per_stream_too(emu, orc):
    """the single-warp LZ4 decoder stays available (BLOSC_B200_LZ4D_PAIR=0 in the product)"""
    emu.emu_set_lz4d_pair(0)
    try:
        for kind, n, ts, shuf in (("bench", 1 << 20, 4, 1), ("mixed", 300001, 8, 2), ("text", 70001, 1, 0)):
            src = gen(kind, n)
            cb, chunk = compress(orc, "orc_compress_ctx", 5, shuf, ts, src, n + 16, "lz4")
            dn, out = decompress(emu, "blosc_decompress_ctx", chunk, n)
            assert dn == n and (out[:n] == src).all()
    finally:
        emu.emu_set_lz4d_pair(1)


def test_blosclz_dense_path_on_corrupted_chains(emu, orc):
    """The dense BloscLZ decoder path (up to 32 two-byte match tokens per step) on the byte-planes of shuffled bench.c
    data: the oracle's bytes on the valid streams, and the oracle's accept / reject verdict (and bytes, when accepted) when
    single bytes of the stream are damaged -- distances reaching before the block, overlapping sources, far-distance and
    length-extension markers appearing in the middle of a chain."""
    rng = np.random.default_rng(17)
    words = gen("bench", 1 << 19).view(np.uint32)
    n = len(words)
    for b in range(3):
        plane = ((words >> (8 * b)) & 0xff).astype(np.uint8)
        a = np.zeros(n + 64, np.uint8)
        ra = orc.orc_blosclz_compress(ci(5), ptr(plane), ci(n), ptr(a), ci(n), ci(1))
        if ra <= 0:
            continue
        o = np.zeros(n + 8, np.uint8)
        assert emu.emu_blz_decode(ptr(a), ci(ra), ptr(o), ci(n)) == n and (o[:n] == plane).all() and (o[n:] == 0).all()
        for trial in range(60):
            c = a[:ra].copy()
            for pos in rng.integers(1, ra, 1 + trial % 3):
                c[pos] = (0, 0xFF, 0xE0 | int(rng.integers(0, 32)), 0x3F, int(rng.integers(0, 256)))[trial % 5]
            o1 = np.zeros(n + 16, np.uint8); o2 = np.zeros(n + 16, np.uint8)
            d1 = orc.orc_blosclz_decompress(ptr(c), ci(ra), ptr(o1), ci(n))
            d2 = emu.emu_blz_decode(ptr(c), ci(ra), ptr(o2), ci(n))
            assert (d1 <= 0) == (d2 <= 0) or d1 == d2, (b, trial, d1, d2)
            if d1 > 0 and d1 == d2:
                assert (o1[:d1] == o2[:d1]).all(), (b, trial)
            assert (o2[n:] == 0).all()
