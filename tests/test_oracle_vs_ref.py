"""Pins the oracle (oracle/blosc_oracle.c, our plain-C restatement) to the UNMODIFIED reference:
filters, both codecs (bytes of the compressed streams included) and the whole ctx API must agree
byte for byte.  The reference's results for every case below are stored as digests in
tests/golden/reference.json; the oracle runs the same cases and must produce the same digests."""
import numpy as np
import pytest

from datagen import Api, Transcript, check_transcript, ci, gen, golden, ptr

KINDS = ["rand", "bench", "zeros", "lowent", "text", "ramp", "i32", "f32", "mixed"]
CTX_KINDS = ["bench", "rand", "i32", "text", "mixed"]


def filters(api):
    t = Transcript()
    for ts in [1, 2, 3, 4, 5, 7, 8, 12, 16, 17, 32, 33, 255]:
        t.group(ts)
        for n in [0, 1, 7, 8, 64, 192, 500, 1000, 1792, 8000, 8192, 100000, 131072]:
            src = gen("rand", n, seed=ts + n)
            for op in ("shuffle", "unshuffle") + (("bitshuffle", "bitunshuffle") if n >= ts else ()):
                a = np.zeros(n + 1, np.uint8)
                api.filter(op, ts, n, src, a)
                t.add(a)
    return t


def lz4_streams(api, kind):
    t = Transcript()
    for n in [0, 1, 5, 12, 13, 15, 16, 33, 64, 67, 128, 255, 1000, 4096, 65535, 65546, 65547, 70000, 131072, 200001]:
        t.group(n)
        src = gen(kind, n, seed=n)
        for accel in (1, 5, 9):
            for cap in sorted({n, max(n - 1, 0), n // 2, n + n // 255 + 16, 70}):
                a = np.zeros(cap + 64, np.uint8)
                ra = api.lz4_compress(ptr(src), ptr(a), ci(n), ci(cap), ci(accel))
                t.add(ra, a[:max(ra, 0)])
                if ra > 0:
                    for c2 in (n, n + 3, max(n - 1, 0)):
                        o = np.zeros(n + 8, np.uint8)
                        d = api.lz4_decompress(ptr(a), ptr(o), ci(ra), ci(c2))
                        t.add(max(d, -1))                   # a rejection is any negative value
                        if c2 == n:
                            assert d == n and (o[:n] == src).all(), (kind, n, accel, cap)
    return t


def blosclz_streams(api, kind):
    t = Transcript()
    for n in [0, 1, 15, 16, 17, 33, 64, 66, 67, 128, 255, 1000, 4096, 16500, 65536, 70000, 131072, 200001]:
        t.group(n)
        src = gen(kind, n, seed=n)
        for clevel in (1, 2, 5, 9):
            for split in (0, 1):
                for cap in sorted({n, max(n - 1, 0), n // 2, 66, 65}):
                    a = np.zeros(cap + 64, np.uint8)
                    ra = api.blosclz_compress(ci(clevel), ptr(src), ci(n), ptr(a), ci(cap), ci(split))
                    t.add(ra, a[:max(ra, 0)])
                    if ra > 0:
                        o = np.zeros(n + 8, np.uint8)
                        d = api.blosclz_decompress(ptr(a), ci(ra), ptr(o), ci(n))
                        assert d == n and (o[:n] == src).all(), (kind, n, clevel, split, cap)
                        t.add(d)
    return t


def ctx_api(api, kind):
    t = Transcript()
    for n in [0, 1, 100, 127, 128, 129, 1000, 4096, 32768, 65536, 100000, 641091, (1 << 20) + 12345]:
        src = gen(kind, n, seed=n)
        for comp in ("lz4", "blosclz"):
            t.group(n, comp)
            for ts in ([1, 2, 3, 4, 8, 16, 17, 256] if n <= 100000 else [4, 8]):
                for shuf in (0, 1, 2):
                    for clevel in ([0, 1, 5, 9] if n <= 100000 else [5]):
                        for bs in ([0, 100, 4096] if n <= 100000 else [0]):
                            for destsize in sorted({n + 16, n + 15, max(16, n // 2), 15}):
                                r, a = api.compress(clevel, shuf, ts, src, destsize, comp, bs)
                                t.add(r)
                                if r <= 0:
                                    continue
                                t.add(a[:r])
                                d, o = api.decompress(a, n)
                                assert d == n and (o[:n] == src).all(), (kind, n, comp, ts, shuf, clevel, bs, destsize)
                                if 0 < n <= 4096:
                                    nit = n // int(a[3])
                                    for st, cnt in ((0, nit), (nit // 3, nit // 2), (nit - 1, 1)):
                                        g = np.zeros(n + 8, np.uint8)
                                        t.add(api.getitem(ptr(a), ci(st), ci(cnt), ptr(g)), g)
    return t


def test_filters(orc):
    check_transcript("filters", filters(Api(orc, False)))


@pytest.mark.parametrize("kind", KINDS)
def test_lz4_streams(orc, kind):
    check_transcript(f"lz4_streams/{kind}", lz4_streams(Api(orc, False), kind))


@pytest.mark.parametrize("kind", KINDS)
def test_blosclz_streams(orc, kind):
    check_transcript(f"blosclz_streams/{kind}", blosclz_streams(Api(orc, False), kind))


@pytest.mark.parametrize("kind", CTX_KINDS)
def test_ctx_api(orc, kind):
    """blosc_compress_ctx / blosc_decompress_ctx / blosc_getitem: same return codes, same chunk bytes."""
    check_transcript(f"ctx_api/{kind}", ctx_api(Api(orc, False), kind))


def reference_multithread_cbytes(ref):
    from datagen import compress
    src = gen("bench", 8 << 20)
    return [compress(ref, "blosc_compress_ctx", 5, 1, 4, src, len(src) + 16, "lz4", 0, nt)[0] for nt in (1, 4)]


def test_reference_multithread_same_cbytes(orc):
    """SURVEY 9.5: ctx compress with nthreads>1 gives the same cbytes (block order may differ) -- the reference's
    sizes with 1 and 4 threads are stored, and the oracle's single answer is that size."""
    from datagen import compress
    r1, r4 = golden()["multithread_cbytes"]
    assert r1 == r4
    src = gen("bench", 8 << 20)
    assert compress(orc, "orc_compress_ctx", 5, 1, 4, src, len(src) + 16, "lz4")[0] == r1


def reference_golden(ref, orc):
    api = Api(ref, True)
    tr = {"filters": filters(api).digests()}
    for k in KINDS:
        tr[f"lz4_streams/{k}"] = lz4_streams(api, k).digests()
        tr[f"blosclz_streams/{k}"] = blosclz_streams(api, k).digests()
    for k in CTX_KINDS:
        tr[f"ctx_api/{k}"] = ctx_api(api, k).digests()
    return {"transcripts": tr, "multithread_cbytes": reference_multithread_cbytes(ref)}
