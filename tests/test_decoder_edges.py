"""LZ4 and BloscLZ decoders on streams built to sit on their thresholds.

Encoders hit the values where the decoders change behaviour (which tier runs, whether a match source is read from the
16 KiB shared-memory ring or from global memory, which end-of-block rule applies) only by chance.  The streams here
are written sequence by sequence from (literals, match length, offset) lists, at, one below and one above each such
value, and their expected output is computed by a plain byte-at-a-time copy.  CPU: the oracle, both LZ4 schedules
(one warp per stream, parser/copier pair) and the BloscLZ decoder in the SIMT emulator.  GPU: the same streams wrapped
into chunks and decoded by decode_kernel<LZ4>, decode_kernel<BLOSCLZ> and decode_pair_kernel.

Ring-read limits.  Every tier reads a match byte from the ring when its offset is at most a bound.  A ring slot holds
output position p until position p + 16384 is written; the lanes of a warp may run in any order between two warp
synchronisations (the SIMT emulator runs them one after another, alternately forward and backward), so a source byte
s is safe in a step only if s + 16384 is not an output byte of that step (or the copy order provably writes it later
from the same lane).  With the step's first output byte at op and its largest output W, the first source byte is
op - off and its alias op - off + 16384 falls inside the step once off >= 16384 - (W - 1).  The largest safe offset is
therefore 16384 - W for each tier:

  tier     W (largest step output)                             safe limit   shipped bound
  dense    24 short x 18 + LZ4D_DENSE_LONG (8) long x 273 = 2616   13768        13696 (16384-2624-64)
  batch    11 sequences whose tokens start in 32 input bytes: 208  16176        16000 (16384-320-64)
  single   the match (<= 18 bytes) after <= 9 literals read in one  16366        16320 (16384-64)
           instruction: only match bytes alias, W = 18
  general  how 1: mlen <= 2048                                     14336        14272 (16384-2048-64)
  lone     273 (one long match)                                    16111        15872 (16384-512)

The lone tier is only reached when the dense step rejects its lane 0, i.e. with off < ml + 8 <= 281, so its bound
never decides anything.  Each family below puts streams exactly at the limit and one byte past it (the latter read
from global memory with the shipped bounds).

Cut rules that only need a source to lie before the step's first output byte (LZ4 dense `off < incl + 8`, BloscLZ
dense `dist < incl + 8`) are correct down to `off < incl`: the 8 bytes of slack cover bytes the word-wise copy reads
past the source and never uses.  The streams here put offsets at incl - 1, incl, incl + 7 and incl + 8.
"""
import ctypes as C
import struct

import numpy as np
import pytest

from datagen import Transcript, check_transcript, ci, ptr, sz

S = 81920                      # every family stream decodes to S bytes: one split of the GPU test chunks
RING = 16384


# ---------------------------------------------------------------------------------------------------------------------
# stream builders and the byte-at-a-time reference

def _varlen(v):
    out = bytearray()
    while v >= 255:
        out.append(255)
        v -= 255
    out.append(v)
    return out


def _lits(lit, rng):
    return bytes(lit) if not isinstance(lit, (int, np.integer)) else rng.integers(0, 256, int(lit), dtype=np.uint8).tobytes()


def _copy(out, off, n):
    """n bytes from `off` back, one at a time (offset 0 decodes to zeros, as LZ4_decompress_safe does)"""
    if off == 0 or off > len(out):
        out += bytes(n)
        return
    for _ in range(n):
        out.append(out[-off])


def lz4_layout(seqs, tail, rng, size=None):
    """An LZ4 block from `seqs` = [(literals, match_len, offset)] (literals: a count of random bytes, or bytes) and a
    final run of `tail` literals; with `size`, the final run is size - (bytes before it) long instead, at least `tail`.
    Returns (stream, expected output, [(input pos, output pos of the match) of every sequence])."""
    st, out, where = bytearray(), bytearray(), []
    for lit, ml, off in seqs:
        lb = _lits(lit, rng)
        lp = len(lb)
        where.append((len(st), len(out) + lp))
        mn = ml - 4
        st.append((min(lp, 15) << 4) | min(mn, 15))
        if lp >= 15:
            st += _varlen(lp - 15)
        st += lb
        out += lb
        st += struct.pack("<H", off)
        if mn >= 15:
            st += _varlen(mn - 15)
        _copy(out, off, ml)
    if size is not None:
        assert size - len(out) >= tail, (size, len(out), tail)
        tail = size - len(out)
    lb = _lits(tail, rng)
    where.append((len(st), len(out)))
    st.append(min(len(lb), 15) << 4)
    if len(lb) >= 15:
        st += _varlen(len(lb) - 15)
    st += lb
    out += lb
    return np.frombuffer(bytes(st), np.uint8).copy(), np.frombuffer(bytes(out), np.uint8).copy(), where


def lz4_stream(seqs, tail, rng, size=None):
    """(stream, expected output): see lz4_layout"""
    return lz4_layout(seqs, tail, rng, size)[:2]


def blosclz_stream(items, rng, size=None, final_match=None):
    """A BloscLZ stream from `items`: an int n is a literal run (one control byte per <= 32 literals, blosclz.c:758-776),
    (length, distance) a match: lengths 3..8 in the control byte, >= 9 with 255-extension bytes, distances up to 8191
    near, 8192 .. 65535 + 8192 far (blosclz.c:699-727).  With `size` a final literal run pads the output to size bytes.
    `final_match` = (length, far distance) ends the stream on a match token, which the decoder does not copy
    (blosclz.c:736; a near one would leave its distance byte last, which is refused).  Returns (stream, expected output)."""
    st, out = bytearray(), bytearray()
    items = list(items)
    if size is not None:
        n = size - sum(it if isinstance(it, int) else it[0] for it in items)
        assert n >= 0
        if n:
            items.append(n)
    assert isinstance(items[0], int) and isinstance(items[-1], int)        # a match that ends the stream is not copied
    for it in items:
        if isinstance(it, int):
            lb = _lits(it, rng)
            for k in range(0, len(lb), 32):
                run = lb[k:k + 32]
                st.append((len(run) - 1) | (0x20 if not st else 0))
                st += run
                out += run
            continue
        st += _blz_match(*it)
        _copy(out, it[1], it[0])
    if final_match is not None:
        st += _blz_match(*final_match)
    return np.frombuffer(bytes(st), np.uint8).copy(), np.frombuffer(bytes(out), np.uint8).copy()


def _blz_match(length, dist):
    far = dist > 8191
    d = dist - 8192 if far else dist - 1
    assert 3 <= length and 0 <= d <= 65535 and (far or d != 8191)
    code = 7 if length >= 9 else length - 2
    b = bytearray([(code << 5) | (31 if far else d >> 8)])
    if code == 7:
        b += _varlen(length - 9)
    b += bytes([255, d >> 8, d & 255]) if far else bytes([d & 255])
    return b


# ---------------------------------------------------------------------------------------------------------------------
# LZ4 case families.  Each returns [(name, seqs, tail, checks)] where checks are (sequence index, offset) of matches whose
# first source byte must differ from the byte 16384 later, so that a ring read past the safe limit gives wrong output.

def _prelude(rng, until=17000):
    """literal runs with short matches: general-tier steps that fill the output sources are read from"""
    seqs = []
    while sum(l + m for l, m, _ in seqs) < until:
        seqs.append((1000, 4, int(rng.integers(100, 900))))
    return seqs


def _aligner(rng, nwarm=24):
    """Long literal-free matches (dense steps of 8), then one whose length byte is 255: the dense step stops in front of
    it, the dense attempt on it fails and sets dense_skip = 1, and the general path takes it.  The next sequence is
    therefore parsed with the dense path skipped once."""
    seqs = [(0, int(rng.integers(19, 60)), int(rng.integers(2300, 12000))) for _ in range(nwarm)]
    return seqs + [(0, 19 + 255 + int(rng.integers(0, 40)), int(rng.integers(2300, 12000)))]


def _filler(rng):
    """one sequence for the single-sequence tier (offset < 320 keeps it out of the batch): consumes the skipped dense
    attempt, so that the next sequence starts a dense attempt"""
    return (2, 6, int(rng.integers(40, 320)))


def _far(rng, n):
    return [int(rng.integers(3000, 12000)) for _ in range(n)]


def fam_dense_chains():
    """Dense chains with 0..9 long (0x0F, one length byte) matches per 32 sequences: the LZ4D_DENSE_LONG = 8 cut, the
    0x0F,..,255 stop, and offsets around the dense ring bound 13696 and the derived limit 13768."""
    rng = np.random.default_rng(101)
    out = []
    for nlong in range(10):
        seqs = _prelude(rng)
        for rep in range(6):
            lanes = []
            longs = set(rng.choice(32, nlong, replace=False).tolist())
            for i in range(32):
                off = int(rng.choice([13695, 13696, 13697, 13767, 13768, 13769] + _far(rng, 6)))
                lanes.append((0, int(rng.integers(19, 274)) if i in longs else int(rng.integers(4, 19)), off))
            if rep == 3:
                lanes[int(rng.integers(1, 31))] = (0, 19 + 255 + 3, 5000)          # the 0x0F,..,255 stop
            seqs += lanes
        out.append((f"chains{nlong}", seqs, 5000, []))
    return out


DENSE_LIMIT = RING - (24 * 18 + 8 * 273)          # 13768


def fam_dense_ring():
    """Dense steps of the largest output (8 long matches of 273 bytes, 24 short ones of 18: 2616 bytes) whose lane 0 is
    a long match at offsets around the shipped bound 13696, 13760 and the derived limit 13768: its first source byte
    op - off shares a ring slot with the step's last output byte, written by lane 31 before lane 0's long match is
    copied, once off >= 16384 - 2615.  A ninth long match (LZ4D_DENSE_LONG 9) makes the step 2871 bytes, which the
    shipped bound no longer covers."""
    rng = np.random.default_rng(102)
    out = []
    for e in (13695, 13696, 13697, 13759, 13760, 13761, DENSE_LIMIT - 1, DENSE_LIMIT, DENSE_LIMIT + 1):
        for nlong in (8, 9):
            seqs = _prelude(rng) + _aligner(rng) + [_filler(rng)]
            lanes = [(0, 273, e)] + [(0, 273, o) for o in _far(rng, nlong - 1)] + [(0, 18, o) for o in _far(rng, 32 - nlong)]
            k = len(seqs)
            seqs += lanes + [(0, 18, o) for o in _far(rng, 40)]
            out.append((f"ring{e}_long{nlong}", seqs, 3000, [(k, e)]))
    return out


def fam_dense_cut():
    """The self-overlap cut `off < incl + 8` of the dense step: lane j's offset at incl_j - 1 (source overlaps the
    step's own output), incl_j, incl_j + 7 and incl_j + 8; steps of 3, 4 and 5 chained sequences (LZ4D_DENSE_MIN)."""
    rng = np.random.default_rng(103)
    out = []
    for d in (-1, 0, 7, 8):
        for j in (1, 4, 13, 31):
            seqs = _prelude(rng) + _aligner(rng) + [_filler(rng)]
            mls = [int(rng.integers(4, 19)) for _ in range(32)]
            offs = _far(rng, 32)
            offs[j] = sum(mls[:j + 1]) + d
            seqs += [(0, m, o) for m, o in zip(mls, offs)] + [(0, 18, o) for o in _far(rng, 32)]
            out.append((f"cut{d}_lane{j}", seqs, 3000, []))
    for cnt in (3, 4, 5):
        seqs = _prelude(rng)
        for _ in range(30):
            seqs += [(0, int(rng.integers(4, 19)), o) for o in _far(rng, cnt)] + [(12, 4, int(rng.integers(3000, 9000)))]
        out.append((f"run{cnt}", seqs, 3000, []))
    return out


def fam_lone():
    """Lone long matches with small periods (off < ml + 8: the dense step rejects lane 0): offsets 1..33, ml + 7 and
    ml + 8 (the latter a one-lane dense step)."""
    rng = np.random.default_rng(104)
    seqs = _prelude(rng)
    for ml in (19, 20, 31, 32, 33, 64, 100, 272, 273):
        for off in sorted({1, 2, 3, 4, 7, 8, 31, 32, 33, ml - 1, ml, ml + 1, ml + 7, ml + 8}):
            seqs += [(0, ml, off), (0, ml, off)]
    return [("lone", seqs, 4000, [])]


BATCH_LIMIT = RING - 208                          # 16176


def _batch_max(rng, e):
    """the largest batch step (208 bytes): nine 3-byte sequences, one with 1 literal, one with 9; lane 0's offset e"""
    seqs = [(0, 18, e)] + [(0, 18, o) for o in _far(rng, 8)] + [(1, 18, int(rng.integers(3000, 12000))),
                                                              (9, 18, int(rng.integers(3000, 12000)))]
    return seqs


def fam_batch():
    """Batch steps: 9 and 10 literals per sequence (the 12-byte window holds the offset of 9 at most), offsets 319,
    320, 321 (LZ4D_BATCH_OUT), match nibbles 14 and 15, and the largest step (208 bytes) with lane 0 at offsets
    around the shipped bound 16000 and the derived limit 16176 right after the aligner, so that the batch starts on it."""
    rng = np.random.default_rng(105)
    out = []
    seqs = _prelude(rng)
    for _ in range(120):
        lit = int(rng.choice([0, 1, 8, 9, 10, 11]))
        seqs.append((lit, int(rng.choice([4, 17, 18, 19])), int(rng.choice([319, 320, 321, 4095, 4096, 12345]))))
    out.append(("lits9_10", seqs, 3000, []))
    for e in (15999, 16000, 16001, BATCH_LIMIT - 1, BATCH_LIMIT, BATCH_LIMIT + 1):
        seqs, checks = _prelude(rng, 20000), []
        for _ in range(6):
            seqs += _aligner(rng, 17)
            checks.append((len(seqs), e))
            seqs += _batch_max(rng, e)
        out.append((f"ring{e}", seqs, 3000, checks))
    return out


SINGLE_LIMIT = RING - 18                          # 16366


def fam_single():
    """The single-sequence tier near the end of the block, where the batch path's op + 320 <= oend - 12 no longer
    holds: offsets around 16320 (shipped bound) and the derived limit 16366, 0..9 literals, off = total - 1 / total
    (self-overlap: general path)."""
    rng = np.random.default_rng(106)
    out = []
    for e in (16319, 16320, 16321, SINGLE_LIMIT - 1, SINGLE_LIMIT, SINGLE_LIMIT + 1):
        for lit in (0, 5, 9):
            seqs = _prelude(rng, 20000)
            tailseqs, checks = [], []
            for k in range(10):
                checks.append((len(seqs) + k, e))
                tailseqs.append((lit, 18, e))
            tailseqs += [(lit, 17, lit + 16), (lit, 17, lit + 17)]
            out.append((f"off{e}_lit{lit}", _fit(seqs + tailseqs, 12), 12, checks))
    return out


GENERAL_LIMIT = RING - 2048                       # 14336


def fam_general():
    """General-tier matches of 2047, 2048 (how 1 or 2), 2049 and 70000 bytes (how 3: global copy, ring_lo reset), at
    offsets around the shipped bound 14272 and the derived limit 14336 and at small periods; each followed by near
    matches whose sources lie in the span the ring did not mirror."""
    rng = np.random.default_rng(107)
    out = []
    for e in (14271, 14272, 14273, GENERAL_LIMIT - 1, GENERAL_LIMIT, GENERAL_LIMIT + 1):
        seqs, checks = _prelude(rng, 20000), []
        for lit in (0, 3, 40):
            checks.append((len(seqs), e))
            seqs += [(lit, 2048, e), (lit, 2047, e), (lit, 2049, e)]
            seqs += [(0, int(rng.integers(4, 19)), int(rng.integers(20, 2000))) for _ in range(40)]
        out.append((f"off{e}", seqs, 3000, checks))
    for off in (1, 3, 31, 32, 33, 2047, 2048):
        seqs = _prelude(rng, 2500) + [(5, 2048, off), (0, 2049, off)]
        seqs += [(0, int(rng.integers(4, 19)), int(rng.integers(20, 2000))) for _ in range(64)]
        out.append((f"period{off}", seqs, 3000, []))
    seqs = _prelude(rng, 3000) + [(7, 70000, 2500)] + [(0, int(rng.integers(4, 19)), int(rng.integers(20, 3000))) for _ in range(80)]
    out.append(("long70000", seqs, 1000, []))
    return out


def fam_literals():
    """Literal runs of 16320, 16321 and 20000 bytes (> 16320 moves ring_lo), then matches reaching back into them."""
    rng = np.random.default_rng(108)
    out = []
    for n in (16319, 16320, 16321, 20000):
        seqs = [(n, 4, 16000)]
        for off in (16319, 16320, 16321, 16000, 3000, 400):
            seqs += [(0, 18, off), (2, 9, off + 3), (0, 100, off)]
        seqs += [(0, int(rng.integers(4, 19)), int(rng.integers(16000, 16384))) for _ in range(64)]
        out.append((f"lits{n}", seqs, 3000, []))
    return out


def fam_offset_zero():
    """offset == 0 (decodes to zeros, resets ring_lo) followed by near matches into and across the zeros"""
    rng = np.random.default_rng(109)
    seqs = _prelude(rng, 5000)
    for ml in (4, 18, 19, 300, 2049):
        seqs += [(3, ml, 0)] + [(0, int(rng.integers(4, 19)), int(rng.integers(1, ml + 40))) for _ in range(40)]
        seqs += [(0, 18, int(o)) for o in rng.integers(320, 2000, 40)]
    return [("zero", seqs, 3000, [])]


def fam_offset_max():
    """offset 65535 (and 65534) in every tier"""
    rng = np.random.default_rng(110)
    seqs = _prelude(rng, 66000)
    for _ in range(2):
        seqs += [(0, int(rng.integers(4, 19)), 65535) for _ in range(40)]
        seqs += [(0, 273, 65535)] * 9 + [(2, 10, 65534), (0, 18, 65533), (12, 30, 65535), (0, 2049, 65535)]
    return [("off65535", seqs, 1000, [])]


def _fit(seqs, tail, size=S, idx=0):
    """grow the literal run of seqs[idx] so that the stream decodes to `size` with exactly `tail` final literals"""
    body = sum((l if isinstance(l, int) else len(l)) + m for l, m, _ in seqs)
    l0, m0, o0 = seqs[idx]
    assert size - tail - body >= 0
    return seqs[:idx] + [(l0 + size - tail - body, m0, o0)] + seqs[idx + 1:]


def fam_margins():
    """The last sequences exactly on the end-of-block rules (a match starting at oend - 12, a match ending at
    oend - 5) and the tier entry margins one byte either side: dense op + 2624 <= oend - 12 and ip + 112 <= iend, batch
    op + 320 <= oend - 12 and ip + 49 <= iend, single ip + 20 <= iend."""
    rng = np.random.default_rng(111)
    out = []
    base = lambda: [(1000, 4, 700)] + _prelude(rng, 16000)                      # noqa: E731
    # a 7-byte match then 5 final literals: the match starts at oend - 12; a 40-byte one ends at oend - 5
    out.append(("mflimit", _fit(base() + [(3, 7, 5000)], 5), 5, []))
    out.append(("lastlits", _fit(base() + [(3, 40, 5000)], 5), 5, []))
    # dense, output: the attempt at the chain's first sequence sees S - op = 2636 + d
    for d in (-1, 0, 1):
        chain = [(0, 18, o) for o in _far(rng, 128)]
        out.append((f"dense_out{d}", _fit(base() + _aligner(rng) + [_filler(rng)] + chain, 2636 + d - 128 * 18), 2636 + d - 128 * 18, []))
    # dense, input: 26 long matches (104 bytes) and a final token with t literals: iend - ip = 105 + t
    for t in (6, 7, 8):
        chain = [(0, 273, o) for o in _far(rng, 26)]
        out.append((f"dense_in{105 + t}", _fit(base() + _aligner(rng) + [_filler(rng)] + chain, t), t, []))
    # batch, output: S - op = 332 + d at the sequence after the aligner
    for d in (-1, 0, 1):
        chain = [(0, 18, o) for o in _far(rng, 12)]
        out.append((f"batch_out{d}", _fit(base() + _aligner(rng) + chain, 332 + d - 12 * 18), 332 + d - 12 * 18, []))
    # batch, input: k 3-byte sequences and m long ones: iend - ip = 3k + 4m + 1 + 5
    for k, m in ((2, 9), (1, 10), (4, 8)):
        chain = [(0, 18, o) for o in _far(rng, k)] + [(0, 273, o) for o in _far(rng, m)]
        out.append((f"batch_in{3 * k + 4 * m + 6}", _fit(base() + _aligner(rng) + chain, 5), 5, []))
    # single, input: a 9-literal sequence then t final literals: iend - ip = 3 + 9 + 1 + t
    for t in (6, 7, 8):
        out.append((f"single_in{13 + t}", _fit(base() + [(9, 18, 4000)], t), t, []))
    return out


FAMILIES = {"dense_chains": (fam_dense_chains, 3), "dense_ring": (fam_dense_ring, 3), "dense_cut": (fam_dense_cut, 3),
            "lone": (fam_lone, 3), "batch": (fam_batch, 0), "single": (fam_single, 1), "general": (fam_general, 2),
            "literals": (fam_literals, 2), "offset_zero": (fam_offset_zero, 2), "offset_max": (fam_offset_max, 3),
            "margins": (fam_margins, 2)}
# the counter of emu_lz4d_counters each family's tier advances: 0 batch, 1 single, 2 general, 3 dense (and lone)

# numeric thresholds each family must put values at, one below and one above: (family, values used, threshold)
THRESHOLDS = [("dense_ring", "offset", 13696), ("dense_ring", "offset", 13760), ("dense_ring", "offset", DENSE_LIMIT),
              ("dense_chains", "offset", 13696), ("batch", "offset", 320), ("batch", "offset", 16000),
              ("batch", "offset", BATCH_LIMIT), ("batch", "literals", 9), ("batch", "match", 18),
              ("single", "offset", 16320), ("single", "offset", SINGLE_LIMIT), ("general", "offset", 14272),
              ("general", "offset", GENERAL_LIMIT), ("general", "match", 2048), ("literals", "literals", 16320),
              ("literals", "offset", 16320), ("lone", "offset", 32), ("offset_max", "offset", 65534)]


def _seq_lit(l):
    return l if isinstance(l, int) else len(l)


def lz4_family(name):
    """[(case name, stream, expected)] of one family, all decoding to S bytes"""
    cases = []
    for i, (case, seqs, tail, checks) in enumerate(FAMILIES[name][0]()):
        rng = np.random.default_rng(1000 + i)
        for _ in range(16):                      # literal bytes redrawn until every checked alias differs
            st, exp, where = lz4_layout(seqs, tail, rng, S)
            if all(where[k][1] - e + RING >= S or exp[where[k][1] - e] != exp[where[k][1] - e + RING] for k, e in checks):
                break
        else:
            raise AssertionError(case)
        assert len(exp) == S, (case, len(exp))
        cases.append((f"{name}/{case}", st, exp))
    return cases


# ---------------------------------------------------------------------------------------------------------------------
# BloscLZ

def blz_families():
    """[(case name, stream, expected)]: dense runs of exactly 3 and 4 tokens (LZ4D_DENSE_MIN's BloscLZ twin), the
    dist = incl + 7 / incl + 8 cut (and incl - 1, incl), near / far distances 8190, 8191, 8192, 73726, 73727, length
    extensions 263..266, literal runs of 1..32, the dense margin op + 256 <= maxout, and a final match token."""
    rng = np.random.default_rng(201)
    cases = []
    pad = [1] * 33                               # 33 one-literal runs: the dense back-off has run out after them

    def near():
        return (int(rng.integers(3, 9)), int(rng.integers(300, 2000)))

    for cnt in (3, 4, 5, 32, 33):
        items = [2000]
        for _ in range(40):
            items += pad + [near() for _ in range(cnt)]
        cases.append((f"run{cnt}", items))
    for d in (-1, 0, 7, 8):
        items = [2000]
        for j in (1, 3, 4, 9, 31):
            toks = [near() for _ in range(32)]
            toks[j] = (toks[j][0], sum(t[0] for t in toks[:j + 1]) + d)
            items += pad + toks
        cases.append((f"cut{d}", items))
    items = [32] * 2400
    for dist in (8190, 8191, 8192, 8193, 65535 + 8191, 73726, 73727):
        items += [(int(rng.integers(3, 9)), dist), (int(rng.integers(9, 300)), dist), 5]
    cases.append(("distances", items))
    items = [3000]
    for n in (262, 263, 264, 265, 266, 519, 520, 9, 8, 3):
        items += [(n, int(rng.integers(1, 2000))), int(rng.integers(1, 33))]
    items += [n for n in range(1, 33)]
    cases.append(("extensions", items))
    out = []
    for name, items in cases:
        st, exp = blosclz_stream(items, rng, S)
        out.append((f"blosclz/{name}", st, exp, S))
    for t in (243, 244, 245):                    # dense margin: op + 256 <= maxout at the run of 4
        body = [S - t - 12 - 33] + pad + [(3, 500)] * 4
        st, exp = blosclz_stream(body + [t], rng)
        out.append((f"blosclz/margin{t}", st, exp, S))
    for r in (16, 17, 18):                       # dense margin: ip + 66 <= length at a run of 8 (49 + r bytes left)
        st, exp = blosclz_stream([S - 33 - 24 - 32 - r] + pad + [(3, 500)] * 8 + [32, r], rng)
        out.append((f"blosclz/margin_in{49 + r}", st, exp, S + 4096))
    st, exp = blosclz_stream([S - 4000] + [(8, 3000)] * 100 + [3200], rng, final_match=(9, 8192 + 100))
    out.append(("blosclz/final_match", st, exp, S + 9))      # the final match must fit, uncopied as it is
    return out


# ---------------------------------------------------------------------------------------------------------------------
# near misses: valid streams with exactly one rule broken by exactly one byte

def lz4_near_misses():
    """[(name, stream, cap)]: each stream decodes to S bytes where it is valid (cap S + 1 / S - 1 where the capacity
    is the rule broken)"""
    rng = np.random.default_rng(301)
    pre = [(1000, 4, 700)] + _prelude(rng, 16000)
    out = []

    def add(name, seqs, tail, cap_delta=0, cut=0, idx=0):
        st, exp = lz4_stream(_fit(seqs, tail, idx=idx), tail, rng)
        assert len(exp) == S
        out.append((name, st[:len(st) - cut] if cut else st, S + cap_delta))

    add("match_at_oend-12", pre + [(3, 7, 5000)], 5)
    add("match_at_oend-11", pre + [(3, 6, 5000)], 5)          # the last match starts one byte late
    add("match_end_oend-5", pre + [(3, 40, 5000)], 5)
    add("match_end_oend-4", pre + [(3, 40, 5000)], 4)         # only 4 final literals
    add("lits_to_iend", pre + [(3, 40, 5000)], 20)
    add("lits_past_iend", pre + [(3, 40, 5000)], 20, cut=1)   # the final run is one byte longer than the input
    add("lits15_past_iend", pre + [(3, 40, 5000)], 15, cut=1)  # ... with its length byte at iend - 15
    add("lits300_past_iend", pre + [(3, 40, 5000)], 300, cut=1)
    add("offset_to_start", [(100, 18, 100)] + pre, 50, idx=1)
    add("offset_before_start", [(100, 18, 101)] + pre, 50, idx=1)   # the source starts one byte before the block
    add("offset_before_start_batch", [(2000, 4, 100)] + [(0, 18, o) for o in (900, 1000, 1100)] + [(0, 18, 2059)] + pre,
        600, idx=5)
    add("offset_before_start_dense", [(3000, 4, 100)] + [(0, 18, 2000)] * 8 + [(0, 18, 3149)] + [(0, 18, 2000)] * 40 + pre,
        3000, idx=50)
    for t, ml in ((3, 19 + 255 + 10), (2, 19 + 510 + 10)):   # the last match length byte at iend - 5 / iend - 4
        add(f"mlen_byte_iend-{t + 2}", pre + [(0, ml, 5000)], t, cap_delta=8)
    for cap in (-1, 1):
        add(f"cap{cap:+d}", pre + [(0, 18, 3000)] * 64, 40, cap_delta=cap)
        add(f"cap{cap:+d}_offset0", pre + [(3, 30, 0)], 40, cap_delta=cap)
    return out


def blz_near_misses():
    """[(name, stream, maxout)], S bytes where valid"""
    rng = np.random.default_rng(302)
    out = []
    for dist, name in ((3000, "ref_at_start"), (3001, "ref_before_start"), (73727, "far_before_start")):
        st, exp = blosclz_stream([3000, (8, dist)], rng, S)
        out.append((name, st, S))
    st, exp = blosclz_stream([S - 3009, (9, 1000), 3000], rng, final_match=(9, 8192 + 500))
    for d in (0, -1):                                         # op + len of the (uncopied) final match one past maxout
        out.append((f"final_match_maxout{d:+d}", st, S + 9 + d))
    st, exp = blosclz_stream([S - 60, (40, 1000), 20], rng)
    out.append(("match_past_maxout", st, S - 21))
    out.append(("lits_past_maxout", st, S - 1))
    out.append(("lits_past_end", st[:-1], S))
    st, exp = blosclz_stream([3000, (300, 1000)], rng, S)
    out.append(("ext_cut", st[:3000 // 32 + 1 + 3000 + 2], S))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU

@pytest.fixture(scope="module")
def lz4_cases():
    return {name: lz4_family(name) for name in FAMILIES}


@pytest.fixture(scope="module")
def blz_cases():
    return blz_families()


def _lz4_decoders(emu):
    emu.emu_lz4_decode_pair.restype = C.c_int
    return (("inline", emu.emu_lz4_decode), ("pair", emu.emu_lz4_decode_pair))


def test_builders_agree_with_oracle(orc):
    """the stream builders' byte-at-a-time output against the oracle (pinned to the reference's decoders)"""
    rng = np.random.default_rng(1)
    for seqs, tail in (([(20, 4, 7), (0, 19, 1), (15, 18, 20), (300, 300, 255), (0, 4000, 600), (9, 70000, 1)], 5),
                       ([(0, 4, 0)] * 3 + [(1, 18, 0), (40, 2048, 17)], 40), ([(16320, 5, 16320), (0, 19 + 255, 3)], 300)):
        st, exp = lz4_stream(seqs, tail, rng)
        o = np.zeros(len(exp) + 64, np.uint8)
        assert orc.orc_lz4_decompress_safe(ptr(st), ptr(o), ci(len(st)), ci(len(exp))) == len(exp)
        assert (o[:len(exp)] == exp).all()
    for items, fm in (([9000, (3, 5), (8, 1), (9, 2), (264, 3), 32, 33, (8, 8191), (4, 8192), 1], None),
                      ([80000, (7, 73727), (266, 73726), (9, 8192), (10, 8191), 1], (4, 9000))):
        st, exp = blosclz_stream(items, rng, final_match=fm)
        o = np.zeros(len(exp) + 64, np.uint8)
        cap = len(exp) + (fm[0] if fm else 0)                  # the final match must fit, uncopied as it is
        assert orc.orc_blosclz_decompress(ptr(st), ci(len(st)), ptr(o), ci(cap)) == len(exp)
        assert (o[:len(exp)] == exp).all()


def test_families_cover_thresholds():
    """both sides of every threshold appear in the generated sequences"""
    for fam, what, t in THRESHOLDS:
        vals = set()
        for _, seqs, _, _ in FAMILIES[fam][0]():
            for l, m, o in seqs:
                vals.add({"offset": o, "match": m, "literals": _seq_lit(l)}[what])
        assert {t - 1, t, t + 1} <= vals, (fam, what, t)


@pytest.mark.parametrize("family", list(FAMILIES))
def test_lz4_family(emu, orc, lz4_cases, family):
    """oracle, single-warp and pair decoders: the model's bytes and return value, nothing written at or past cap;
    the tier the family aims at runs; each stream once more into a destination at 16-byte phase 7"""
    counters = (C.c_longlong * 4)()
    emu.emu_lz4d_counters(counters)
    before = list(counters)
    for case, st, exp in lz4_cases[family]:
        n = len(exp)
        o = np.zeros(n + 64, np.uint8)
        assert orc.orc_lz4_decompress_safe(ptr(st), ptr(o), ci(len(st)), ci(n)) == n, case
        assert (o[:n] == exp).all(), case
        for dname, decode in _lz4_decoders(emu):
            o = np.full(n + 64, 0xA5, np.uint8)
            r = decode(ptr(st), ci(len(st)), ptr(o), ci(n))
            bad = np.flatnonzero(o[:n] != exp)
            assert r == n and not len(bad), (case, dname, r, bad[:8])
            assert (o[n:] == 0xA5).all(), (case, dname)
        buf = np.full(n + 96, 0xA5, np.uint8)
        shift = (7 - buf.ctypes.data) % 16
        r = emu.emu_lz4_decode(ptr(st), ci(len(st)), C.c_void_p(buf.ctypes.data + shift), ci(n))
        assert r == n and (buf[shift:shift + n] == exp).all(), case
        assert (buf[:shift] == 0xA5).all() and (buf[shift + n:] == 0xA5).all(), case
    emu.emu_lz4d_counters(counters)
    delta = [counters[i] - before[i] for i in range(4)]
    assert delta[FAMILIES[family][1]] > 0, (family, delta)


def test_blosclz_families(emu, orc, blz_cases):
    """oracle and the BloscLZ decoder: the model's bytes and return value, nothing written past them"""
    for case, st, exp, cap in blz_cases:
        n = len(exp)
        o = np.zeros(cap + 64, np.uint8)
        assert orc.orc_blosclz_decompress(ptr(st), ci(len(st)), ptr(o), ci(cap)) == n, case
        assert (o[:n] == exp).all(), case
        o = np.full(cap + 64, 0xA5, np.uint8)
        r = emu.emu_blz_decode(ptr(st), ci(len(st)), ptr(o), ci(cap))
        bad = np.flatnonzero(o[:n] != exp)
        assert r == n and not len(bad), (case, r, bad[:8])
        assert (o[n:] == 0xA5).all(), case


def _near_miss_transcript(lz4, blz):
    """lz4(stream, cap, out) / blz(stream, maxout, out) -> return value; one group per near miss"""
    t = Transcript()
    for name, st, cap in lz4_near_misses():
        t.group("lz4", name)
        o = np.zeros(cap + 64, np.uint8)
        d = lz4(st, cap, o)
        t.add(max(d, -1))
        if d >= 0:
            t.add(o[:d])
    for name, st, cap in blz_near_misses():
        t.group("blosclz", name)
        o = np.zeros(cap + 64, np.uint8)
        d = blz(st, cap, o)
        t.add(max(d, 0))
        if d > 0:
            t.add(o[:d])
    return t


def test_near_misses_match_reference(orc, emu):
    """one rule broken by one byte: the reference's verdict (and bytes) in the oracle and in both LZ4 schedules and the
    BloscLZ decoder, nothing written past cap"""
    accepted = []

    def blz(lib):
        def f(st, cap, o):
            d = lib(ptr(st), ci(len(st)), ptr(o), ci(cap))
            assert (o[cap:] == 0).all()
            return d
        return f
    check_transcript("decoder_edge_verdicts", _near_miss_transcript(
        lambda st, cap, o: orc.orc_lz4_decompress_safe(ptr(st), ptr(o), ci(len(st)), ci(cap)), blz(orc.orc_blosclz_decompress)))
    for _, decode in _lz4_decoders(emu):
        def lz4(st, cap, o, decode=decode):
            d = decode(ptr(st), ci(len(st)), ptr(o), ci(cap))
            assert (o[cap:] == 0).all()
            accepted.append(d >= 0)
            return d
        check_transcript("decoder_edge_verdicts", _near_miss_transcript(lz4, blz(emu.emu_blz_decode)))
    assert 4 < sum(accepted) < len(accepted) - 4


def reference_golden(ref, orc):
    t = _near_miss_transcript(lambda st, cap, o: ref.LZ4_decompress_safe(ptr(st), ptr(o), ci(len(st)), ci(cap)),
                              lambda st, cap, o: ref.blosclz_decompress(ptr(st), ci(len(st)), ptr(o), ci(cap)))
    return {"transcripts": {"decoder_edge_verdicts": t.digests()}}


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the same streams in hand-made chunks (header, bstarts, a size prefix per split: blosc.c:760-784)

def make_chunk(streams, typesize, flags, blocksize, nbytes):
    """streams in block order, `typesize` splits per full block unless flags has 0x10 (then one), one for the leftover"""
    nsplits = 1 if flags & 0x10 else typesize
    nfull, left = divmod(nbytes, blocksize)
    nblocks = nfull + (1 if left else 0)
    assert len(streams) == nfull * nsplits + (1 if left else 0)
    pos = 16 + 4 * nblocks
    bstarts, body, k = [], [], 0
    for b in range(nblocks):
        bstarts.append(pos)
        for _ in range(nsplits if b < nfull else 1):
            st = streams[k]
            k += 1
            body += [struct.pack("<i", len(st)), st.tobytes()]
            pos += 4 + len(st)
    head = bytes([2, 1, flags, typesize]) + struct.pack("<iii", nbytes, blocksize, pos)
    return np.frombuffer(head + struct.pack(f"<{nblocks}i", *bstarts) + b"".join(body), np.uint8).copy()


def _gpu_decode(cuda, pkg, orc, chunk, nbytes):
    """(oracle code, GPU code, GPU output equals the oracle's)"""
    want = np.zeros(nbytes + 64, np.uint8)
    r0 = orc.orc_decompress_ctx(ptr(chunk), ptr(want), sz(nbytes), ci(1))
    d_c = cuda.from_numpy(chunk).cuda()
    d_o = cuda.full((nbytes + 4096,), 0xA5, dtype=cuda.uint8, device="cuda")
    r = pkg.decompress_ctx(d_c, d_o, nbytes)
    got = d_o.cpu().numpy()
    assert (got[nbytes:] == 0xA5).all(), "written past destsize"
    return r0, r, r0 < 0 or (got[:nbytes] == want[:nbytes]).all()


def _all_lz4():
    return [c for name in FAMILIES for c in lz4_family(name)]


@pytest.mark.gpu
def test_single_warp_decoder_gpu(pkg, cuda, orc):
    """one-split chunks (flags 0x10), typesize 1, one stream per block: decode_kernel<LZ4> and <BLOSCLZ>"""
    for fmt, streams in ((1, [st for _, st, _ in _all_lz4()]), (0, [st for _, st, exp, cap in blz_families() if len(exp) == cap == S])):
        chunk = make_chunk(streams, 1, 0x10 | fmt << 5, S, S * len(streams))
        r0, r, same = _gpu_decode(cuda, pkg, orc, chunk, S * len(streams))
        assert r0 == r == S * len(streams) and same, (fmt, r0, r)


def _pair_streams():
    cases = _all_lz4()
    nstreams = 148 * 12 + 7                                   # > SMs x PAIR_CTAS_PER_SM: every CTA decodes several
    return [cases[k % len(cases)][1] for k in range(nstreams // 4 * 4)] + [cases[0][1]]


@pytest.mark.gpu
def test_pair_decoder_gpu(pkg, cuda, orc):
    """four-split chunks (typesize 4, no shuffle, LZ4) with more streams than the pair kernel has CTAs, plus a
    leftover block: every CTA runs several streams back to back through its parser / copier queue"""
    streams = _pair_streams()
    nbytes = S * len(streams)
    chunk = make_chunk(streams, 4, 1 << 5, 4 * S, nbytes)
    r0, r, same = _gpu_decode(cuda, pkg, orc, chunk, nbytes)
    assert r0 == r == nbytes and same, (r0, r)


@pytest.mark.gpu
def test_near_miss_splits_gpu(pkg, cuda, orc):
    """a chunk of good splits with one near miss: the oracle's return code, for both LZ4 schedules and BloscLZ"""
    good = [st for _, st, _ in _all_lz4()[:12]]
    for k, (name, st, _) in enumerate(lz4_near_misses()):
        for ts, flags in ((4, 1 << 5), (1, 0x10 | 1 << 5)):
            ss = list(good)
            ss[k % 12] = st
            chunk = make_chunk(ss, ts, flags, S * ts, S * 12)
            r0, r, same = _gpu_decode(cuda, pkg, orc, chunk, S * 12)
            assert r == r0 and same, (name, ts, r0, r)
    good = [c[1] for c in blz_families()[:6]]
    for k, (name, st, _) in enumerate(blz_near_misses()):
        ss = list(good)
        ss[k % 6] = st
        chunk = make_chunk(ss, 1, 0x10, S, S * 6)
        r0, r, same = _gpu_decode(cuda, pkg, orc, chunk, S * 6)
        assert r == r0 and same, (name, r0, r)
