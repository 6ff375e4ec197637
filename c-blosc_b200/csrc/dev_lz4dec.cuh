/*
 * dev_lz4dec.cuh -- LZ4 block decoder, sm_100a: LZ4_decompress_safe semantics (lz4.c:2022-2445).
 *
 * lz4d_parse walks the tokens in four tiers: a dense path for chains of literal-free sequences (one 3-byte sequence
 * per lane, long matches with one extra length byte taken inline: up to 32 sequences per step, every lane copying its
 * own match), a batch path (every lane speculatively parses the sequence that would start at its input byte; the chain
 * of real starts is resolved with one ballot or a short shuffle walk and up to 11 sequences are copied 32 output bytes
 * per instruction), a single-sequence fast path, and the general path with warp-wide literal and period-replicating
 * match copies.  A per-warp shared-memory ring mirrors the last 16 KiB of output so match sources -- a few KiB back in
 * >99% of the sequences of shuffled data -- do not wait behind the global stores that produced them.
 *
 * Every tier ends by handing its step (destination, source and length of every sequence) to a sink, and every step is
 * copied by the tier's copy routine (lz4d_copy_*).  Two sinks give two schedules of the same decoder:
 *
 *   Lz4dInline  lz4_decode_warp, one warp per stream: the step is copied at once, its values still in registers.
 *   Lz4dQueue   lz4_pair_parse + lz4_pair_copier, two warps per stream.  On the hard byte-plane of shuffled data one
 *               warp is a chain of ~150 k dependent instructions, yet parsing step k+1 needs nothing from the copies
 *               of step k -- only the byte counts, which the parse itself produces.  So the parser warp writes each
 *               step as a descriptor into a queue of LZ4P_Q slots in shared memory, and the copier warp, which owns
 *               the output and the ring, takes them in order.  Hand-over with named barriers (bar.sync / bar.arrive,
 *               64 threads): FULL(s) parser -> copier, EMPTY(s) back.
 *
 * Both return the same verdict and write the same bytes for every accepted stream (tests run both).
 */
#pragma once
#include "dev_lz4.cuh"

#ifdef SIMT_EMU
static long long g_dbg_lz4d_batch_seqs = 0, g_dbg_lz4d_fast_seqs = 0, g_dbg_lz4d_general_seqs = 0, g_dbg_lz4d_dense_seqs = 0;
#define LZ4D_DBG(x) do { if (lane == 0) (x)++; } while (0)
#define LZ4D_DBGN(x, n) do { if (lane == 0) (x) += (n); } while (0)
#else
#define LZ4D_DBG(x) do {} while (0)
#define LZ4D_DBGN(x, n) do {} while (0)
#endif
#define LZ4D_RING 16384                      /* bytes of recent output mirrored in shared memory, per warp */
#define LZ4D_RMASK (LZ4D_RING - 1)
#define LZ4D_BATCH_OUT 320                   /* a batch writes < 320 bytes (11 sequences x <= 27) */
#define LZ4D_BATCH_SMASK 24                  /* word of the batch table where its 10 start-bit words begin */
#define LZ4D_DENSE_LONG 8                    /* long matches (one extra length byte) a dense step takes inline */
#define LZ4D_DENSE_OUT 2624                  /* a dense step writes <= 24 x 18 + 8 x 273 bytes */
#define LZ4D_DENSE_MIN 4                     /* fewer chained 3-byte sequences than this: the 11-wide batch path is as good */
#define LZ4D_SCRATCH 256                     /* per-warp shared scratch after the ring: sequence table + start-bit words */
#define LZ4D_SMEM (LZ4D_RING + LZ4D_SCRATCH)

/* ---- copy routines, one per tier.  Every output byte also goes into the ring. ---- */

/* Dense step: lanes [0, cnt) hold one literal-free sequence each (kind 1: short match, 2: long match, marked in
 * longm); every source lies before the step's first output byte.  Every lane copies its own short match, 4 source
 * bytes per step: from the ring (two aligned words + funnel shift) or, for far offsets, from the output in global
 * memory.  The warp copies the long ones. */
DEV void lz4d_copy_dense(u8* out, smem_addr_t ring, int dst, int off, int ml, int kind, bool from_ring, int cnt, unsigned longm) {
  const int lane = lane_id();
  const int match = dst - off;
  const int mls = (lane < cnt && kind == 1) ? ml : 0;
  const int mlmax = __ballot_sync(FULLMASK, mls > 16) ? 18 : (__ballot_sync(FULLMASK, mls > 8) ? 16 : 8);
  u8* o = out + dst;
#pragma unroll 1
  for (int k = 0; k < mlmax; k += 4) {
    if (k < mls) {
      u32 v;
      if (from_ring) {
        const u32 m = (u32)(match + k);
        v = __funnelshift_r(smem_ld_u32(ring, m & (LZ4D_RMASK & ~3u)), smem_ld_u32(ring, (m + 4u) & (LZ4D_RMASK & ~3u)), (m & 3u) * 8u);
      } else v = ld_u32(out + match + k);       /* may read a few bytes past the source: they are not used */
      const int nb = mls - k;
      const u32 r = (u32)(dst + k);
      o[k] = (u8)v; smem_st_u8(ring, r & LZ4D_RMASK, v);
      if (nb > 1) { o[k + 1] = (u8)(v >> 8); smem_st_u8(ring, (r + 1u) & LZ4D_RMASK, v >> 8); }
      if (nb > 2) { o[k + 2] = (u8)(v >> 16); smem_st_u8(ring, (r + 2u) & LZ4D_RMASK, v >> 16); }
      if (nb > 3) { o[k + 3] = (u8)(v >> 24); smem_st_u8(ring, (r + 3u) & LZ4D_RMASK, v >> 24); }
    }
  }
  for (unsigned tm = longm; tm; tm &= tm - 1u) {
    const int t = __ffs((int)tm) - 1;
    const int td = __shfl_sync(FULLMASK, dst, t), tmt = __shfl_sync(FULLMASK, match, t), tl = __shfl_sync(FULLMASK, ml, t);
    const bool tring = __shfl_sync(FULLMASK, (int)from_ring, t) != 0;
    for (int k = lane; k < tl; k += 32) {
      const u32 v = tring ? smem_ld_u8(ring, (u32)(tmt + k) & LZ4D_RMASK) : (u32)out[tmt + k];
      out[td + k] = (u8)v;
      smem_st_u8(ring, (u32)(td + k) & LZ4D_RMASK, v);
    }
  }
}

/* One long match at op whose source may overlap its own output (small offsets): period copy by the warp.  The sources
 * all lie before op, so no lane waits for another. */
DEV void lz4d_copy_lone(u8* out, smem_addr_t ring, int op, int len, int off, bool from_ring) {
  const int match = op - off;
  for (int k = lane_id(); k < len; k += 32) {
    const int src = match + (off >= len ? k : k % off);
    const u32 v = from_ring ? smem_ld_u8(ring, (u32)src & LZ4D_RMASK) : (u32)out[src];
    out[op + k] = (u8)v;
    smem_st_u8(ring, (u32)(op + k) & LZ4D_RMASK, v);
  }
}

/* Batch step: `total` bytes at op from up to 11 sequences.  tbl[2i] = opre | lit << 9 | lane << 13 (the sequence's
 * output position in the step, its literal count, its token's input position relative to ip), tbl[2i+1] = offset;
 * bit y of the start-bit words at tbl + LZ4D_BATCH_SMASK marks output byte y where a sequence begins.  One output byte
 * per lane and instruction. */
DEV void lz4d_copy_batch(const u8* in, u8* out, smem_addr_t ring, const u32* tbl, int ip, int op, int total, int ring_lo) {
  const int lane = lane_id();
  const u32* smask = tbl + LZ4D_BATCH_SMASK;
  int kbase = 0;
  for (int r = 0; r * 32 < total; r++) {
    const u32 w = smask[r];
    const int y = r * 32 + lane;
    if (y < total) {
      const int k = kbase + __popc(w & ((2u << lane) - 1u)) - 1;
      const u32 e0 = tbl[2 * k], offk = tbl[2 * k + 1];
      const int opre = (int)(e0 & 511u), litk = (int)((e0 >> 9) & 15u), lanek = (int)(e0 >> 13);
      const int j = y - opre;
      u32 v;
      if (j < litk) v = in[ip + lanek + 1 + j];
      else {
        const int src = op + opre + litk - (int)offk + (j - litk);
        const int m0 = op + opre + litk - (int)offk;
        if ((int)offk <= LZ4D_RING - LZ4D_BATCH_OUT - 64 && m0 >= ring_lo) v = smem_ld_u8(ring, (u32)src & LZ4D_RMASK);
        else v = out[src];
      }
      out[op + y] = (u8)v;
      smem_st_u8(ring, (u32)(op + y) & LZ4D_RMASK, v);
    }
    kbase += __popc(w);
  }
}

/* Single-sequence step: lit literals at in + ip + 1, then a match of total - lit bytes whose source lies strictly
 * before its own output; one lane per output byte. */
DEV void lz4d_copy_single(const u8* in, u8* out, smem_addr_t ring, int ip, int op, int lit, int total, int off, bool use_ring) {
  const int lane = lane_id();
  const int match = op + lit - off;
  if (lane < total) {
    u32 v;
    if (lane < lit) v = in[ip + 1 + lane];
    else if (use_ring) v = smem_ld_u8(ring, (u32)(match + lane - lit) & LZ4D_RMASK);
    else v = out[match + lane - lit];
    out[op + lane] = (u8)v;
    smem_st_u8(ring, (u32)(op + lane) & LZ4D_RMASK, v);
  }
}

/* General step: len literals from lits to op, then (mlen > 0) a match of mlen bytes at offset off.  how: 0 zero fill
 * (offset 0), 1 period copy from the ring, 2 period copy from global memory, 3 long match (not mirrored in the ring). */
DEV void lz4d_copy_general(const u8* lits, u8* out, smem_addr_t ring, int op, int len, int mlen, int off, int how) {
  const int lane = lane_id();
  for (int k = lane; k < len; k += 32) {
    const u32 v = lits[k];
    out[op + k] = (u8)v;
    smem_st_u8(ring, (u32)(op + k) & LZ4D_RMASK, v);
  }
  if (mlen == 0) return;
  op += len;
  const int match = op - off;
  __syncwarp();                                             /* earlier output must be visible to all lanes */
  if (how == 0) {
    /* not a valid stream, but LZ4_decompress_safe accepts it: every copy routine first clears the destination word
     * ("silence msan warning when offset==0", lz4.c:2386-2390; LZ4_memcpy_using_offset_base) and then replicates
     * it, so the match decodes to zeros */
    for (int k = lane; k < mlen; k += 32) out[op + k] = 0;
  } else if (how <= 2) {
    /* sources lie before op; inside the ring they are not overwritten by this copy.  Far sources are read from global
     * memory, but the output still goes into the ring so that it stays a mirror of the last 16 KiB */
    for (int k0 = 0; k0 < mlen; k0 += 32) {
      const int k = k0 + lane;
      if (k < mlen) {
        const int src = match + (off >= mlen ? k : k % off);
        const u32 v = how == 1 ? smem_ld_u8(ring, (u32)src & LZ4D_RMASK) : (u32)out[src];
        out[op + k] = (u8)v;
        smem_st_u8(ring, (u32)(op + k) & LZ4D_RMASK, v);
      }
    }
  } else warp_copy_match(out, op, match, mlen);
}

/* read_variable_length (lz4.c:1979-2020): adds the length bytes at ip to len; false once ip passes ilimit or len
 * passes oend (the same verdict as the reference's later output checks, without int overflow on hostile input) */
DEV bool lz4d_varlen(const u8* in, int& ip, int& len, int ilimit, int oend) {
  u32 sb;
  do {
    sb = in[ip++];
    len += (int)sb;
    if (ip > ilimit || len > oend) return false;
  } while (sb == 255);
  return true;
}

/* ---- the parser: LZ4_decompress_safe for one stream (lz4.c:2451-2456; safe-loop rules :2234-2436), every step handed
 * to `sink`.  Returns the number of bytes the stream decodes to, or -1.  offset == 0 decodes to zeros, as in the
 * reference.  A rejected stream may leave any prefix of its steps written; nothing is written at or past cap. ---- */
template <class Sink>
DEV int lz4d_parse(const u8* __restrict__ in, const int csize, const int cap, Sink& sink) {
  const int iend = csize, oend = cap;
  const int lane = lane_id();
  const StreamBase ib = make_stream_base(in);
  if (cap == 0) return (csize == 1 && in[0] == 0) ? 0 : -1;   /* lz4.c:2062-2066 */
  if (csize == 0) return -1;
  sink.start();
  int ip = 0, op = 0, result = -1;           /* -1 until the last literals are reached */
  int ring_lo = 0;                           /* positions [max(ring_lo, op-RING), op) are valid in the ring */
  int dense_skip = 0, dense_back = 0;
  for (;;) {
    /* ---- dense path: a run of literal-free sequences, one per lane ----
     * The byte-planes of shuffled data decode to long chains of 3-byte sequences (token with
     * 0 literals and a 4..18 byte match, 16-bit offset).  If the sequence at ip is of that form the
     * next one starts at ip+3, so lane l parses the 3 bytes at ip+3l and the leading run of lanes
     * that all see this form are real sequences.  A prefix sum of the match lengths gives every
     * lane its output position; sequences whose source lies entirely before the batch's first
     * output byte are independent, and every lane copies its own match. */
    if (dense_skip > 0) dense_skip--;
    else if (ip + 112 <= iend && op + LZ4D_DENSE_OUT <= oend - LZ4_MFLIMIT) {
      u32 b0, b1, b2;
      ldp_win12(ib, ip + 3 * lane, b0, b1, b2);               /* bytes ip+3l .. ip+3l+11 (touches < ip+109) */
      lz4d_prefetch(in, ip + 256 + 128 * lane, lane < 2 ? iend : 0);
      /* Segments: lanes [c, e) see 3-byte sequences at byte shift s; the sequence that ends a
       * segment is very often a longer literal-free match with one extra length byte (token 0x0F,
       * offset, len): lane e takes it and the next segment starts one byte later (shift s+1). */
      int kind = 0, ml = 0, off = 0, c = 0, sft = 0;
      u32 w = b0;
      for (;;) {
        const u32 tok = w & 0xffu;
        const unsigned okm = __ballot_sync(FULLMASK, lane >= c && (tok >> 4) == 0u && (tok & 15u) != 15u);
        const unsigned stop = ~okm & ~((1u << c) - 1u);        /* first lane >= c that is not such a sequence */
        const int e = stop ? __ffs((int)stop) - 1 : 32;
        if (lane >= c && lane < e) { kind = 1; ml = (int)(tok & 15u) + 4; off = (int)((w >> 8) & 0xffffu); }
        c = e;
        if (e >= 32 || sft == LZ4D_DENSE_LONG) break;
        const u32 tw = __shfl_sync(FULLMASK, w, e);
        if ((tw & 0xffu) != 0x0fu || (tw >> 24) == 255u) break;
        if (lane == e) { kind = 2; ml = 19 + (int)(tw >> 24); off = (int)((tw >> 8) & 0xffffu); }
        c = e + 1; sft++;
        if (c >= 32) break;
        w = sft < 4 ? __funnelshift_r(b0, b1, 8u * (u32)sft) : (sft == 4 ? b1 : (sft < 8 ? __funnelshift_r(b1, b2, 8u * (u32)(sft - 4)) : b2));
      }
      int cnt = c;                                             /* lanes [0, cnt) hold one sequence each */
      int incl = ml;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(FULLMASK, incl, d);
        if (lane >= d) incl += t;
      }
      const int dst = op + incl - ml, match = dst - off;
      /* first sequence that reads its own batch's output (or is invalid: off == 0, match < 0) ends the run;
       * 8 bytes of slack because the word-wise copy reads up to 7 bytes past the end of its source */
      const unsigned bad = __ballot_sync(FULLMASK, lane < cnt && (off < incl + 8 || match < 0));
      if (bad) cnt = __ffs((int)bad) - 1;
      const unsigned longm = __ballot_sync(FULLMASK, lane < cnt && kind == 2);
      if (cnt >= LZ4D_DENSE_MIN || longm) {
        const int total = __shfl_sync(FULLMASK, incl, cnt - 1);
        const bool from_ring = off <= LZ4D_RING - LZ4D_DENSE_OUT - 64 && match >= ring_lo;
        sink.dense(dst, off, ml, kind, from_ring, cnt, longm);
        ip += 3 * cnt + __popc(longm); op += total;
        LZ4D_DBGN(g_dbg_lz4d_dense_seqs, cnt);
        dense_back = 0;
        continue;
      }
      /* a lone long match whose source overlaps its own output (small offsets): period copy by the warp */
      {
        const u32 tw = __shfl_sync(FULLMASK, b0, 0);
        const int tlen = 19 + (int)(tw >> 24), toff = (int)((tw >> 8) & 0xffffu), tmatch = op - toff;
        if ((tw & 0xffu) == 0x0fu && (tw >> 24) != 255u && toff != 0 && tmatch >= 0 && op + tlen <= oend - LZ4_MFLIMIT) {
          sink.lone(op, tlen, toff, toff <= LZ4D_RING - 512 && tmatch >= ring_lo);
          ip += 4; op += tlen;
          LZ4D_DBG(g_dbg_lz4d_dense_seqs);
          dense_back = 0;
          continue;
        }
      }
      dense_back = dense_back < 8 ? dense_back + 1 : 8;   /* not that kind of data right here: back off */
      dense_skip = dense_back;
    }
    /* ---- batch path: up to 11 short sequences per round ----
     * Lane l speculates that a sequence starts at input byte ip+l and parses it from its own
     * 12-byte window.  Sequences whose offset reaches back past everything this batch can write
     * (>= LZ4D_BATCH_OUT) cannot depend on each other, so once the chain of real starts is known
     * (one ballot when every sequence is the 3-byte literal-free form, a shuffle walk otherwise)
     * all their output bytes are produced 32 per instruction. */
    if (ip + 49 <= iend && op + LZ4D_BATCH_OUT <= oend - LZ4_MFLIMIT) {   /* a 9-literal sequence of lane 31 ends at ip+41 <= iend-8 (lz4.c:2289) */
      u32 b0, b1, b2;
      ldp_win12(ib, ip + lane, b0, b1, b2);
      const u32 token = b0 & 0xffu;
      const int lit = (int)(token >> 4), mln = (int)(token & 15u);
      const int ob = 1 + lit;                                  /* window byte of the 16-bit offset (valid for lit <= 9: token, literals and offset fit the 12-byte window) */
      const u32 ow = ob < 4 ? __funnelshift_r(b0, b1, 8u * ob) : (ob < 8 ? __funnelshift_r(b1, b2, 8u * (ob - 4)) : b2 >> (8u * ((ob - 8) & 3)));
      const int off = (int)(ow & 0xffffu);
      const int L = 3 + lit, O = lit + mln + 4;
      const bool good = lit <= 9 && mln != 15 && off >= LZ4D_BATCH_OUT;
      int nseq = 0, consumed = 0, total = 0, my_rank = -1, my_opre = 0;
      const unsigned g3 = __ballot_sync(FULLMASK, good && lit == 0);
      if ((g3 & 0x49249249u) == 0x49249249u) {                 /* starts at lanes 0,3,...,30 */
        const bool real = (lane % 3) == 0;
        const int v = real ? O : 0;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const int t = __shfl_up_sync(FULLMASK, incl, d);
          if (lane >= d) incl += t;
        }
        if (real) { my_rank = lane / 3; my_opre = incl - v; }
        nseq = 11; consumed = 33;
        total = __shfl_sync(FULLMASK, incl, 31);
      } else {
        const u32 packed = (good ? 1u : 0u) | ((u32)L << 1) | ((u32)O << 5);
        int cur = 0;
        while (cur < 32) {
          const u32 pk = __shfl_sync(FULLMASK, packed, cur);
          if (!(pk & 1u)) break;
          if (lane == cur) { my_rank = nseq; my_opre = total; }
          total += (int)((pk >> 5) & 31u);
          cur += (int)((pk >> 1) & 15u);
          nseq++;
        }
        consumed = cur;
      }
      if (nseq > 0) {
        const int match = op + my_opre + lit - off;            /* meaningful on real lanes */
        if (__ballot_sync(FULLMASK, my_rank >= 0 && match < 0)) break;   /* lz4.c:2356 */
        u32* tbl = sink.batch_table();                         /* 11 x {info, off}, start-bit words at LZ4D_BATCH_SMASK */
        u32* smask = tbl + LZ4D_BATCH_SMASK;
        if (lane < 10) smask[lane] = 0;
        __syncwarp();
        if (my_rank >= 0) {
          tbl[2 * my_rank] = (u32)my_opre | ((u32)lit << 9) | ((u32)lane << 13);
          tbl[2 * my_rank + 1] = (u32)off;
          atomicOr(&smask[my_opre >> 5], 1u << (my_opre & 31));
        }
        sink.batch(tbl, ip, op, total, ring_lo);
        ip += consumed; op += total;
        LZ4D_DBGN(g_dbg_lz4d_batch_seqs, nseq);
        continue;
      }
    }
    /* ---- single-sequence fast path: short sequence, source strictly before its own output ---- */
    if (ip + 20 <= iend) {
      u32 b0, b1, b2;
      ldp_win12(ib, ip, b0, b1, b2);
      const u32 token = b0 & 0xffu;
      const int lit = (int)(token >> 4), mln = (int)(token & 15u);
      if (lit <= 9 && mln != 15) {
        const int ml = mln + 4, total = lit + ml;
        const int ob = 1 + lit;
        const u32 ow = ob < 4 ? __funnelshift_r(b0, b1, 8u * ob) : (ob < 8 ? __funnelshift_r(b1, b2, 8u * (ob - 4)) : b2 >> (8u * (ob - 8)));
        const int off = (int)(ow & 0xffffu);
        const int match = op + lit - off;
        if (off >= total && op + total <= oend - LZ4_MFLIMIT) { /* no self-overlap; far from the end of the block */
          if (match < 0) break;                                /* lz4.c:2356 (off == 0 cannot get here: off >= total >= 4) */
          sink.single(ip, op, lit, total, off, off <= LZ4D_RING - 64 && match >= ring_lo);
          ip += 3 + lit; op += total;
          LZ4D_DBG(g_dbg_lz4d_fast_seqs);
          continue;
        }
      }
    }
    /* ---- general path: one sequence, literals and match in one step ---- */
    LZ4D_DBG(g_dbg_lz4d_general_seqs);
    const u32 token = in[ip++];
    int len = (int)(token >> 4);
    if (len == 15 && (ip >= iend - 15 || !lz4d_varlen(in, ip, len, iend - 15, oend))) break;   /* read_variable_length(ip, iend-15, 1) */
    int cpy = op + len;
    const bool last = cpy > oend - LZ4_MFLIMIT || ip + len > iend - (2 + 1 + LZ4_LASTLITERALS);   /* lz4.c:2289-2331 */
    if (last && (ip + len != iend || cpy > oend)) break;
    if (len > LZ4D_RING - 64) ring_lo = cpy - (LZ4D_RING - 64) > ring_lo ? cpy - (LZ4D_RING - 64) : ring_lo;
    if (last) {                                               /* the last sequence: literals only */
      sink.general(ip, op, len, 0, 0, 0);
      result = cpy;
      break;
    }
    const int lsrc = ip, lop = op;
    ip += len; op = cpy;
    const int off = (int)in[ip] | ((int)in[ip + 1] << 8);
    ip += 2;
    const int match = op - off;
    int mlen = (int)(token & 15u);
    if (mlen == 15 && !lz4d_varlen(in, ip, mlen, iend - LZ4_LASTLITERALS + 1, oend)) break;   /* read_variable_length(ip, iend-4, 0) */
    mlen += 4;
    if (match < 0) break;                                     /* lz4.c:2356 */
    cpy = op + mlen;
    if (cpy > oend - LZ4_LASTLITERALS) break;                 /* lz4.c:2423 */
    int how;
    if (off == 0) { how = 0; ring_lo = cpy; }                 /* decodes to zeros, which the ring does not mirror */
    else if (mlen <= 2048) how = off <= LZ4D_RING - 2048 - 64 && match >= ring_lo ? 1 : 2;
    else { how = 3; ring_lo = cpy; }                          /* global sources; the ring no longer mirrors this span */
    sink.general(lsrc, lop, len, mlen, off, how);
    op = cpy;
  }
  return sink.finish(result);
}

/* ---- one warp per stream: every step is copied at once.  `scratch` is the warp's LZ4D_SMEM bytes of shared memory:
 * the ring, then the batch table. ---- */
struct Lz4dInline {
  const u8* in;
  u8* out;
  u8* scratch;
  smem_addr_t ring;
  DEV void start() {}
  DEV void dense(int dst, int off, int ml, int kind, bool from_ring, int cnt, unsigned longm) {
    lz4d_copy_dense(out, ring, dst, off, ml, kind, from_ring, cnt, longm);
    __syncwarp();
  }
  DEV void lone(int op, int len, int off, bool from_ring) {
    lz4d_copy_lone(out, ring, op, len, off, from_ring);
    __syncwarp();
  }
  DEV u32* batch_table() { return (u32*)(scratch + LZ4D_RING); }
  DEV void batch(const u32* tbl, int ip, int op, int total, int ring_lo) {
    __syncwarp();
    lz4d_copy_batch(in, out, ring, tbl, ip, op, total, ring_lo);
    __syncwarp();
  }
  DEV void single(int ip, int op, int lit, int total, int off, bool use_ring) {
    lz4d_copy_single(in, out, ring, ip, op, lit, total, off, use_ring);
    __syncwarp();
  }
  DEV void general(int lsrc, int op, int len, int mlen, int off, int how) {
    lz4d_copy_general(in + lsrc, out, ring, op, len, mlen, off, how);
    __syncwarp();
  }
  DEV int finish(int result) { return result; }
};

DEV int lz4_decode_warp(const u8* __restrict__ in, const int csize, u8* out, const int cap, u8* scratch) {
  Lz4dInline sink{in, out, scratch, smem_addr(scratch)};
  return lz4d_parse(in, csize, cap, sink);
}

/* ---- two warps per stream: the parser queues every step for the copier ---- */
#define LZ4P_Q 4                               /* descriptor slots */
#define LZ4P_BAR_FULL(s) (1 + (s))
#define LZ4P_BAR_EMPTY(s) (1 + LZ4P_Q + (s))
enum { LZ4P_END = 0, LZ4P_DENSE = 1, LZ4P_LONE = 2, LZ4P_BATCH = 3, LZ4P_SINGLE = 4, LZ4P_GENERAL = 5, LZ4P_START = 6, LZ4P_QUIT = 7 };

struct Lz4pSlot {
  u32 type;
  u32 p[7];                                    /* scalars of the step */
  u32 w[64];                                   /* DENSE: two words per lane; BATCH: the batch table */
};
#define LZ4P_SMEM (LZ4D_RING + LZ4P_Q * (int)sizeof(Lz4pSlot))

struct Lz4dQueue {
  const u8* in;
  u8* out;
  Lz4pSlot* slots;
  int k;                                       /* descriptors of this stream so far */
  /* the slot of descriptor k, once the copier is done with descriptor k - Q */
  DEV Lz4pSlot* acquire() {
    const int s = k & (LZ4P_Q - 1);
    if (k >= LZ4P_Q) bar_sync(LZ4P_BAR_EMPTY(s), 64);
    return &slots[s];
  }
  DEV void publish() {
    __syncwarp();
    __threadfence_block();
    bar_arrive(LZ4P_BAR_FULL(k & (LZ4P_Q - 1)), 64);
    k++;
  }
  DEV void start() {
    Lz4pSlot* q = acquire();
    if (lane_id() == 0) {
      q->type = LZ4P_START;
      q->p[0] = (u32)(u64)(uintptr_t)in; q->p[1] = (u32)((u64)(uintptr_t)in >> 32);
      q->p[2] = (u32)(u64)(uintptr_t)out; q->p[3] = (u32)((u64)(uintptr_t)out >> 32);
    }
    publish();
  }
  /* p0 = cnt, p1 = longm; lane l: w[2l] = dst, w[2l+1] = off | ml << 16 | kind << 28 | from_ring << 31 */
  DEV void dense(int dst, int off, int ml, int kind, bool from_ring, int cnt, unsigned longm) {
    Lz4pSlot* q = acquire();
    const int lane = lane_id();
    q->w[2 * lane] = (u32)dst;
    q->w[2 * lane + 1] = (u32)off | ((u32)ml << 16) | ((u32)kind << 28) | (from_ring ? 0x80000000u : 0u);
    if (lane == 0) { q->type = LZ4P_DENSE; q->p[0] = (u32)cnt; q->p[1] = longm; }
    publish();
  }
  DEV void lone(int op, int len, int off, bool from_ring) {
    Lz4pSlot* q = acquire();
    if (lane_id() == 0) { q->type = LZ4P_LONE; q->p[0] = (u32)op; q->p[1] = (u32)len; q->p[2] = (u32)off; q->p[3] = from_ring; }
    publish();
  }
  DEV u32* batch_table() { return acquire()->w; }
  DEV void batch(const u32*, int ip, int op, int total, int ring_lo) {
    Lz4pSlot* q = &slots[k & (LZ4P_Q - 1)];
    if (lane_id() == 0) { q->type = LZ4P_BATCH; q->p[0] = (u32)ip; q->p[1] = (u32)op; q->p[2] = (u32)total; q->p[3] = (u32)ring_lo; }
    publish();
  }
  DEV void single(int ip, int op, int lit, int total, int off, bool use_ring) {
    Lz4pSlot* q = acquire();
    if (lane_id() == 0) {
      q->type = LZ4P_SINGLE; q->p[0] = (u32)ip; q->p[1] = (u32)op; q->p[2] = (u32)lit; q->p[3] = (u32)total; q->p[4] = (u32)off;
      q->p[5] = use_ring;
    }
    publish();
  }
  DEV void general(int lsrc, int op, int len, int mlen, int off, int how) {
    Lz4pSlot* q = acquire();
    if (lane_id() == 0) {
      q->type = LZ4P_GENERAL; q->p[0] = (u32)lsrc; q->p[1] = (u32)op; q->p[2] = (u32)len; q->p[3] = (u32)mlen;
      q->p[4] = (u32)off; q->p[5] = (u32)how;
    }
    publish();
  }
  /* END, then wait until the copier is done with every descriptor: the EMPTY arrivals of the last ones have no acquire
   * that consumes them, and taking them leaves both warps with every barrier idle for the next stream */
  DEV int finish(int result) {
    Lz4pSlot* q = acquire();
    if (lane_id() == 0) q->type = LZ4P_END;
    publish();
    for (int j = k > LZ4P_Q ? k - LZ4P_Q : 0; j < k; j++) bar_sync(LZ4P_BAR_EMPTY(j & (LZ4P_Q - 1)), 64);
    __syncwarp();
    return result;
  }
};

/* Parser warp: the stream's verdict as lz4_decode_warp's; the copier has finished with the stream when this returns. */
DEV int lz4_pair_parse(const u8* __restrict__ in, const int csize, u8* out, const int cap, Lz4pSlot* slots) {
  Lz4dQueue sink{in, out, slots, 0};
  return lz4d_parse(in, csize, cap, sink);
}

/* Copier warp: takes the descriptors in order and runs the tier's copy routine on each, until QUIT. */
DEV void lz4_pair_copier(u8* ring_ptr, Lz4pSlot* slots) {
  const int lane = lane_id();
  const smem_addr_t ring = smem_addr(ring_ptr);
  const u8* in = nullptr;
  u8* out = nullptr;
  int k = 0;
  for (;;) {
    const int s = k & (LZ4P_Q - 1);
    bar_sync(LZ4P_BAR_FULL(s), 64);
    const Lz4pSlot* q = &slots[s];
    const u32 type = *(const volatile u32*)&q->type;
    if (type == LZ4P_QUIT) return;
    const u32 p0 = *(const volatile u32*)&q->p[0], p1 = *(const volatile u32*)&q->p[1], p2 = *(const volatile u32*)&q->p[2],
              p3 = *(const volatile u32*)&q->p[3], p4 = *(const volatile u32*)&q->p[4], p5 = *(const volatile u32*)&q->p[5];
    if (type == LZ4P_START) {
      in = (const u8*)(((u64)p1 << 32) | p0);
      out = (u8*)(((u64)p3 << 32) | p2);
    } else if (type == LZ4P_DENSE) {
      const u32 wd = *(const volatile u32*)&q->w[2 * lane], wx = *(const volatile u32*)&q->w[2 * lane + 1];
      lz4d_copy_dense(out, ring, (int)wd, (int)(wx & 0xffffu), (int)((wx >> 16) & 0xfffu), (int)((wx >> 28) & 3u), (wx >> 31) != 0u,
                      (int)p0, p1);
    } else if (type == LZ4P_LONE) {
      lz4d_copy_lone(out, ring, (int)p0, (int)p1, (int)p2, p3 != 0u);
    } else if (type == LZ4P_BATCH) {
      lz4d_copy_batch(in, out, ring, q->w, (int)p0, (int)p1, (int)p2, (int)p3);
    } else if (type == LZ4P_SINGLE) {
      lz4d_copy_single(in, out, ring, (int)p0, (int)p1, (int)p2, (int)p3, (int)p4, p5 != 0u);
    } else if (type == LZ4P_GENERAL) {
      lz4d_copy_general(in + p0, out, ring, (int)p1, (int)p2, (int)p3, (int)p4, (int)p5);
    }
    __syncwarp();
    bar_arrive(LZ4P_BAR_EMPTY(s), 64);
    k = type == LZ4P_END ? 0 : k + 1;
  }
}

/* tell the copier that there are no more streams */
DEV void lz4_pair_quit(Lz4pSlot* slots) {
  if (lane_id() == 0) slots[0].type = LZ4P_QUIT;
  __syncwarp();
  __threadfence_block();
  bar_arrive(LZ4P_BAR_FULL(0), 64);
}

/* A CTA of two warps that decodes streams as parser / copier pairs: warp 1 runs the copier for the life of the CTA and
 * gets nullptr when it is done; warp 0 gets the slots to hand to lz4_pair_parse, then lz4_pair_quit. */
DEV Lz4pSlot* lz4_pair_setup(u8* smem) {
  Lz4pSlot* slots = (Lz4pSlot*)(smem + LZ4D_RING);
  if ((threadIdx.x >> 5) == 1) { lz4_pair_copier(smem, slots); return nullptr; }
  return slots;
}
