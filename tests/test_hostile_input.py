"""Damaged / hostile input: the accept-reject verdict (and the bytes, when accepted) must be the
reference's.  CPU: the reference's verdicts (stored in tests/golden/reference.json) vs oracle vs the
product's device code in the SIMT emulator.  GPU: the CUDA library vs the oracle (ADVICE r1:
negative header nbytes, LZ4 offset 0, the 9-literal rule of the batch path, frame slots)."""
import ctypes as C

import numpy as np
import pytest

from datagen import Transcript, check_transcript, ci, compress, gen, golden, ptr, sz


def _lz4_mutants(orc, rng, count):
    """Reference-valid LZ4 streams with a few bytes changed; offsets forced to 0 in a third of them."""
    out = []
    for kind, n in (("bench", 6000), ("text", 20000), ("lowent", 9000), ("i32", 5000)):
        src = gen(kind, n, seed=n)
        cap = n + n // 255 + 32
        a = np.zeros(cap + 64, np.uint8)
        ra = orc.orc_lz4_compress_fast(ptr(src), ptr(a), ci(n), ci(cap), ci(1))
        assert ra > 0
        for k in range(count):
            c = a[:ra].copy()
            if k % 3 == 0:                               # zero a 16-bit field somewhere: very often an offset
                p = int(rng.integers(1, ra - 2))
                c[p] = 0; c[p + 1] = 0
            else:
                pos = rng.integers(0, ra, 1 + k % 4)
                c[pos] = rng.integers(0, 256, len(pos), dtype=np.uint8)
            out.append((c, n))
    return out


def _lz4_verdicts(orc, decode):
    """decode(c, n, out) -> return value; one group per mutant: the verdict and, when accepted, the bytes."""
    rng = np.random.default_rng(11)
    t, accepted = Transcript(), 0
    for i, (c, n) in enumerate(_lz4_mutants(orc, rng, 120)):
        t.group(i)
        o = np.zeros(n + 16, np.uint8)
        d = decode(c, n, o)
        t.add(max(d, -1))                                # a rejection is any negative value
        if d >= 0:
            t.add(o[:d])
            accepted += 1
    return t, accepted


def test_lz4_decode_verdicts_match_reference(orc, emu):
    t, accepted = _lz4_verdicts(orc, lambda c, n, o: orc.orc_lz4_decompress_safe(ptr(c), ptr(o), ci(len(c)), ci(n)))
    check_transcript("lz4_mutant_verdicts", t)
    assert accepted > 10
    outs = []

    def emu_decode(c, n, o):
        d = emu.emu_lz4_decode(ptr(c), ci(len(c)), ptr(o), ci(n))
        outs.append((o, n))
        return d
    check_transcript("lz4_mutant_verdicts", _lz4_verdicts(orc, emu_decode)[0])
    assert all((o[n:] == 0).all() for o, n in outs)


OFFSET_ZERO = bytes([0x1f, 0x41, 0x00, 0x00, 0x01]) + bytes([0x50]) + b"ABCDE"


def test_lz4_offset_zero_decodes_to_zeros(orc, emu):
    """token 0x1f: 1 literal, match length 15+1+4 = 20, offset 0; then the mandatory last literals."""
    c = np.frombuffer(OFFSET_ZERO, np.uint8).copy()
    n = 1 + 20 + 5
    want_n, want = golden()["lz4_offset_zero"]
    assert want_n == n and bytes.fromhex(want) == b"A" + bytes(20) + b"ABCDE"       # what the reference does
    o = np.full(n + 8, 0xEE, np.uint8)
    assert orc.orc_lz4_decompress_safe(ptr(c), ptr(o), ci(len(c)), ci(n)) == n
    assert bytes(o[:n]) == b"A" + bytes(20) + b"ABCDE"
    for decode in (emu.emu_lz4_decode, emu.emu_lz4_decode_pair):
        o = np.full(n + 8, 0xEE, np.uint8)
        assert decode(ptr(c), ci(len(c)), ptr(o), ci(n)) == n
        assert bytes(o[:n]) == b"A" + bytes(20) + b"ABCDE"


def _hostile_headers(src):
    """(chunk, destsize) pairs built from a valid chunk of `src`."""
    import struct
    n = len(src)
    cases = []
    for nbytes, flags, cbytes in ((-5, 0x02 | 0x20, 11), (-5, 0x20, 64), (-1, 0x02, 15), (-128, 0x01 | 0x20, 16),
                                  (-(1 << 31), 0x02, -(1 << 31) + 16), (-5, 0x02, 0), (n, 0x02, n + 15), (n, 0x22, n + 17)):
        h = bytes([2, 1, flags & 0xff, 4]) + struct.pack("<iii", nbytes, 4096, cbytes)
        cases.append((np.frombuffer(h + bytes(src[:256]), np.uint8).copy(), 1 << 16))
    return cases


def test_hostile_header_cpu(orc, emu):
    src = gen("i32", 8192)
    want = golden()["hostile_header_returns"]
    assert len(want) == len(_hostile_headers(src))
    for (c, destsize), r0 in zip(_hostile_headers(src), want):
        o1 = np.zeros(destsize, np.uint8); o2 = np.zeros(destsize, np.uint8)
        r1 = orc.orc_decompress_ctx(ptr(c), ptr(o1), sz(destsize), ci(1))
        r2 = emu.blosc_decompress_ctx(ptr(c), ptr(o2), sz(destsize), ci(1))
        assert r0 == r1 == r2, (bytes(c[:16]).hex(), r0, r1, r2)
        assert not o2.any()


@pytest.mark.gpu
def test_hostile_header_gpu(pkg, cuda, orc):
    src = gen("i32", 8192)
    for c, destsize in _hostile_headers(src):
        o1 = np.zeros(destsize, np.uint8)
        r1 = orc.orc_decompress_ctx(ptr(c), ptr(o1), sz(destsize), ci(1))
        o2 = np.zeros(destsize, np.uint8)
        assert pkg.decompress_ctx(c, o2, destsize) == r1
        d_c = cuda.from_numpy(c).cuda(); d_o = cuda.zeros(destsize, dtype=cuda.uint8, device="cuda")
        assert pkg.decompress_ctx(d_c, d_o, destsize) == r1
        assert not o2.any() and not bool(d_o.any())


@pytest.mark.gpu
def test_lz4_verdicts_gpu(pkg, cuda, orc):
    """Mutated LZ4 streams wrapped into single-block unsplit chunks: the CUDA decoder against the oracle."""
    import struct
    rng = np.random.default_rng(5)
    for c, n in _lz4_mutants(orc, rng, 40):
        o1 = np.zeros(n + 16, np.uint8)
        d1 = orc.orc_lz4_decompress_safe(ptr(c), ptr(o1), ci(len(c)), ci(n))
        cb = 16 + 4 + 4 + len(c)
        chunk = bytes([2, 1, 0x10 | 0x20, 1]) + struct.pack("<iii", n, n, cb) + struct.pack("<ii", 20, len(c)) + bytes(c)
        ch = np.frombuffer(chunk, np.uint8).copy()
        r0 = orc.orc_decompress_ctx(ptr(ch), ptr(np.zeros(n, np.uint8)), sz(n), ci(1))
        o2 = np.zeros(n, np.uint8)
        r = pkg.decompress_ctx(ch, o2, n)
        assert r == r0, (r, r0, d1)
        if d1 == n:
            assert r == n and (o2 == o1[:n]).all()
        else:
            assert r < 0


def test_frame_slot_validation(emu):
    """A chunk header inside a frame that claims more bytes than its slot is refused (ADVICE r1)."""
    emu.blosc_b200_frame_compress.restype = C.c_longlong
    emu.blosc_b200_frame_decompress.restype = C.c_longlong
    emu.blosc_b200_frame_bound.restype = C.c_size_t
    n, chunk = 300000, 100000
    src = gen("i32", n)
    bound = emu.blosc_b200_frame_bound(sz(n), sz(4), sz(chunk))
    fr = np.zeros(bound, np.uint8)
    fb = emu.blosc_b200_frame_compress(ci(5), ci(1), sz(4), sz(n), ptr(src), ptr(fr), sz(bound), b"lz4", sz(0), sz(chunk), ci(1))
    assert fb > 0
    out = np.zeros(n, np.uint8)
    assert emu.blosc_b200_frame_decompress(ptr(fr), sz(fb), ptr(out), sz(n), ci(1)) == n and (out == src).all()
    off1 = int(np.frombuffer(fr[32 + 8:32 + 16].tobytes(), "<u8")[0])
    bad = fr.copy()
    bad[off1 + 12:off1 + 16] = np.frombuffer(np.int32(1 << 30).tobytes(), np.uint8)     # cbytes far beyond the slot
    assert emu.blosc_b200_frame_decompress(ptr(bad), sz(fb), ptr(out), sz(n), ci(1)) == -1
    bad = fr.copy()
    bad[off1 + 4:off1 + 8] = np.frombuffer(np.int32(chunk - 4).tobytes(), np.uint8)      # nbytes != the chunk's share
    assert emu.blosc_b200_frame_decompress(ptr(bad), sz(fb), ptr(out), sz(n), ci(1)) == -1


def reference_golden(ref, orc):
    t = _lz4_verdicts(orc, lambda c, n, o: ref.LZ4_decompress_safe(ptr(c), ptr(o), ci(len(c)), ci(n)))[0]
    c = np.frombuffer(OFFSET_ZERO, np.uint8).copy()
    o = np.zeros(26 + 8, np.uint8)
    d = ref.LZ4_decompress_safe(ptr(c), ptr(o), ci(len(c)), ci(26))
    src = gen("i32", 8192)
    headers = [ref.blosc_decompress_ctx(ptr(h), ptr(np.zeros(ds, np.uint8)), sz(ds), ci(1)) for h, ds in _hostile_headers(src)]
    return {"transcripts": {"lz4_mutant_verdicts": t.digests()},
            "lz4_offset_zero": [d, bytes(o[:max(d, 0)]).hex()], "hostile_header_returns": headers}
