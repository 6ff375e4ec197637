/*
 * dev_lz4.cuh -- LZ4 block encoder, one warp per stream, sm_100a (the decoder is dev_lz4dec.cuh).
 *
 * Bit-exact replay of LZ4_compress_fast's greedy parse
 * (reference: internal-complibs/lz4-1.10.0/lz4.c:930-1338, called from
 * blosc/blosc.c:413-420 with acceleration = 10 - clevel and maxout = neblock, i.e.
 * limitedOutput).  The sequential "probe, skip, probe" search loop (lz4.c:1043-1101)
 * is evaluated 32 probes at a time: lane l computes the position the l-th probe
 * WOULD visit (closed form of the skip schedule), hashes it, and resolves the hash
 * table state it would observe -- the table as left by earlier rounds, overridden by
 * the nearest lower lane with the same hash (__match_any_sync).  The first hitting
 * lane wins, and only probes up to and including it are committed to the table, so
 * the table evolves exactly as in the serial code and the output is byte-identical.
 */
#pragma once
#include "dev_common.cuh"

#define LZ4_MFLIMIT 12
#define LZ4_LASTLITERALS 5
#define LZ4_TABLE_BYTES 16384          /* lz4.h:163,696  LZ4_MEMORY_USAGE 14 */
#define LZ4_TAB17_BYTES (8192 + 512)    /* packed variant of the 4096-entry table: u16 + 1 bit per entry */
#define LZ4_TAB17_MINLEN 65547         /* shorter streams use the 8192-entry byU16 table (lz4.c:710,1389), which cannot shrink */
#define LZ4_TAB17_MAXLEN 131072

template <bool U16>
DEV u32 lz4_hash_at(const u8* __restrict__ s, int pos) {       /* lz4.c:777-806 */
  if (U16) return (ld_u32(s + pos) * 2654435761u) >> (32 - 13);
  const u64 seq = (u64)ld_u32(s + pos) | ((u64)s[pos + 4] << 32);   /* low 5 bytes are all hash5 uses */
  return (u32)(((seq << 24) * 889523592379ull) >> (64 - 12));
}

#define LZ4_SCALAR_PROBES 4     /* probes done one at a time before the 32-wide rounds (must be <= 64) */

/* Offset from the search start of the it-th probe of the skip schedule
 * (lz4.c:1043-1053): steps are 1, then accel + (k >> 6) for k = 0,1,2,... */
DEV long long lz4_probe_offset(int it, int accel) {
  if (it == 0) return 0;
  const long long m = it - 1;
  const long long c = m >> 6;
  return 1 + m * accel + 32 * c * (c - 1) + c * (m - 64 * c);
}

/* Position-based window loads: the stream base is split once into an aligned word pointer
 * (s32) and a byte phase (sal); a window at byte position p then costs one 64-bit address
 * computation (IMAD.WIDE) instead of one per word. */
struct StreamBase {
  const u8* s;
  const u32* s32;
  int sal;
  const uint4* s128;     /* the same stream seen as aligned 16-byte granules */
  int sal16;
};
DEV StreamBase make_stream_base(const u8* s) {
  StreamBase b;
  b.s = s;
  b.s32 = (const u32*)((uintptr_t)s & ~(uintptr_t)3);
  b.sal = (int)((uintptr_t)s & 3u);
  b.s128 = (const uint4*)((uintptr_t)s & ~(uintptr_t)15);
  b.sal16 = (int)((uintptr_t)s & 15u);
  return b;
}
/* 12 bytes at position p as three little-endian words.  GPU: four aligned read-only word loads
 * + funnel shifts; touches the aligned words around [p, p+12), i.e. at most byte p+15 --
 * callers guarantee p+16 <= end of the stream (the emulator build reads exactly 12 bytes). */
DEV void ldp_win12(const StreamBase& sb, int p, u32& b0, u32& b1, u32& b2) {
#ifdef SIMT_EMU
  memcpy(&b0, sb.s + p, 4); memcpy(&b1, sb.s + p + 4, 4); memcpy(&b2, sb.s + p + 8, 4);
#else
  const int q = p + sb.sal;
  const u32* w = sb.s32 + (q >> 2);
  const u32 sh = (u32)(q & 3) * 8u;
  const u32 w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2), w3 = __ldg(w + 3);
  b0 = __funnelshift_r(w0, w1, sh); b1 = __funnelshift_r(w1, w2, sh); b2 = __funnelshift_r(w2, w3, sh);
#endif
}
/* The same in two steps, for loads that are requested long before their bytes are needed:
 * ldp_raw12 only issues the aligned word loads, ldp_take12 aligns them (first use of the data). */
DEV void ldp_raw12(const StreamBase& sb, int p, u32& r0, u32& r1, u32& r2, u32& r3) {
#ifdef SIMT_EMU
  memcpy(&r0, sb.s + p, 4); memcpy(&r1, sb.s + p + 4, 4); memcpy(&r2, sb.s + p + 8, 4); r3 = 0;
#else
  const u32* w = sb.s32 + ((p + sb.sal) >> 2);
  r0 = __ldg(w); r1 = __ldg(w + 1); r2 = __ldg(w + 2); r3 = __ldg(w + 3);
#endif
}
DEV void ldp_take12(const StreamBase& sb, int p, u32 r0, u32 r1, u32 r2, u32 r3, u32& b0, u32& b1, u32& b2) {
#ifdef SIMT_EMU
  (void)sb; (void)p; (void)r3; b0 = r0; b1 = r1; b2 = r2;
#else
  const u32 sh = (u32)((p + sb.sal) & 3) * 8u;
  b0 = __funnelshift_r(r0, r1, sh); b1 = __funnelshift_r(r1, r2, sh); b2 = __funnelshift_r(r2, r3, sh);
#endif
}
/* 8 bytes at position p; touches at most byte p+11 */
DEV void ldp_win8(const StreamBase& sb, int p, u32& b0, u32& b1) {
#ifdef SIMT_EMU
  memcpy(&b0, sb.s + p, 4); memcpy(&b1, sb.s + p + 4, 4);
#else
  const int q = p + sb.sal;
  const u32* w = sb.s32 + (q >> 2);
  const u32 sh = (u32)(q & 3) * 8u;
  const u32 w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
  b0 = __funnelshift_r(w0, w1, sh); b1 = __funnelshift_r(w1, w2, sh);
#endif
}

/* 17 bytes at position p (four words + the byte p+16) in two steps, as ldp_raw12 / ldp_take12:
 * ldp_raw20 issues five aligned word loads (touches at most byte p+19), ldp_take17 aligns them. */
DEV void ldp_raw20(const StreamBase& sb, int p, u32 (&r)[5]) {
#ifdef SIMT_EMU
  memcpy(&r[0], sb.s + p, 16); r[4] = sb.s[p + 16];
#else
  const u32* w = sb.s32 + ((p + sb.sal) >> 2);
  r[0] = __ldg(w); r[1] = __ldg(w + 1); r[2] = __ldg(w + 2); r[3] = __ldg(w + 3); r[4] = __ldg(w + 4);
#endif
}
DEV void ldp_take17(const StreamBase& sb, int p, const u32 (&r)[5], u32& a0, u32& a1, u32& a2, u32& a3, u32& a4b) {
#ifdef SIMT_EMU
  (void)sb; (void)p; a0 = r[0]; a1 = r[1]; a2 = r[2]; a3 = r[3]; a4b = r[4] & 0xffu;
#else
  const u32 sh = (u32)((p + sb.sal) & 3) * 8u;
  a0 = __funnelshift_r(r[0], r[1], sh); a1 = __funnelshift_r(r[1], r[2], sh);
  a2 = __funnelshift_r(r[2], r[3], sh); a3 = __funnelshift_r(r[3], r[4], sh);
  a4b = (r[4] >> sh) & 0xffu;
#endif
}
/* The same 17 bytes for a GATHER (every lane its own, unrelated position): two aligned 128-bit
 * loads instead of five 32-bit ones -- a warp-wide gather costs one L1 tag cycle per distinct line
 * and instruction, so the instruction count is what matters -- and a two-level select network that
 * brings the five words that hold the bytes into place.  Touches [p & ~15, +32). */
DEV void ldp_gather17(const StreamBase& sb, int p, u32& c0, u32& c1, u32& c2, u32& c3, u32& c4b) {
#ifdef SIMT_EMU
  memcpy(&c0, sb.s + p, 4); memcpy(&c1, sb.s + p + 4, 4); memcpy(&c2, sb.s + p + 8, 4); memcpy(&c3, sb.s + p + 12, 4);
  c4b = sb.s[p + 16];
#else
  const int q = p + sb.sal16;
  const uint4* w = sb.s128 + (q >> 4);
  const uint4 v0 = __ldg(w), v1 = __ldg(w + 1);
  const bool k1 = (q & 4) != 0, k2 = (q & 8) != 0;
  const u32 sh = (u32)(q & 3) * 8u;
  const u32 t0 = k1 ? v0.y : v0.x, t1 = k1 ? v0.z : v0.y, t2 = k1 ? v0.w : v0.z, t3 = k1 ? v1.x : v0.w;
  const u32 t4 = k1 ? v1.y : v1.x, t5 = k1 ? v1.z : v1.y, t6 = k1 ? v1.w : v1.z;
  const u32 u0 = k2 ? t2 : t0, u1 = k2 ? t3 : t1, u2 = k2 ? t4 : t2, u3 = k2 ? t5 : t3, u4 = k2 ? t6 : t4;
  c0 = __funnelshift_r(u0, u1, sh); c1 = __funnelshift_r(u1, u2, sh);
  c2 = __funnelshift_r(u2, u3, sh); c3 = __funnelshift_r(u3, u4, sh);
  c4b = (u4 >> sh) & 0xffu;
#endif
}

/* L1 prefetch of the line holding byte p of a stream of `end` bytes (no-op past the end) */
DEV void lz4d_prefetch(const u8* base, int p, int end) {
#ifndef SIMT_EMU
  if (p < end) asm volatile("prefetch.global.L1 [%0];" :: "l"(base + p));
#else
  (void)base; (void)p; (void)end;
#endif
}

/* 4 bytes at position p; touches at most byte p+7 */
DEV u32 ldp_win4(const StreamBase& sb, int p) {
#ifdef SIMT_EMU
  u32 b0; memcpy(&b0, sb.s + p, 4); return b0;
#else
  const int q = p + sb.sal;
  const u32* w = sb.s32 + (q >> 2);
  return __funnelshift_r(__ldg(w), __ldg(w + 1), (u32)(q & 3) * 8u);
#endif
}

template <bool U16>
DEV u32 lz4_hash_seq(u32 lo, u32 b4) {                        /* lz4.c:777-806 on bytes already in registers */
  if (U16) return (lo * 2654435761u) >> (32 - 13);
  const u64 seq = (u64)lo | ((u64)(b4 & 0xffu) << 32);
  return (u32)(((seq << 24) * 889523592379ull) >> (64 - 12));
}

/* LZ4_count continuation for matches that outgrow the scalar compares: first round 4 bytes per
 * lane (128 bytes, two loads per lane), only then the 512-bytes-per-round loop.  p > q, `n` =
 * stream length, limit = matchlimit. */
DEV int lz4_count_tail(const StreamBase& sb, const u8* __restrict__ s, int p, int q, int limit, int n) {
  if (p + 136 <= n) {                                           /* p + 128 <= limit and the loads stay inside the stream */
    const int lane = lane_id();
    const u32 x = ldp_win4(sb, p + 4 * lane) ^ ldp_win4(sb, q + 4 * lane);
    const unsigned full = __ballot_sync(FULLMASK, x == 0u);
    if (full != FULLMASK) {
      const int fl = __ffs((int)~full) - 1;
      return fl * 4 + eq_bytes32(__shfl_sync(FULLMASK, x, fl));
    }
    return 128 + warp_count_match(s, p + 128, q + 128, limit);
  }
  return warp_count_match(s, p, q, limit);
}

/* ---- team mode: one CTA of four warps per stream ------------------------------------------------
 * A lone warp spends ~6 cycles per instruction on its dependent chain (ALU latency 4, one issue
 * per 2 cycles and pipe), so on a hard byte-plane the serial LZ4 loop is bound by the NUMBER of
 * instructions one warp has to issue per sequence, not by memory.  In team mode the stream's warp
 * ("walker") keeps only what is inherently serial -- which position the parse lands on next, the
 * table stores, the output -- and three helper warps ("preparers") do the rest ahead of it:
 * for every position of a 32-position tile a preparer computes hash, table lookup, candidate
 * gather, 17-byte compare and packs the verdict {hit, match length, offset} into a shared-memory
 * ring; the walker reads the verdict of the position it lands on with one 8-byte shared load.
 * A verdict can be stale: the preparer of tile t starts when the walker has finished tile t-3, so
 * it cannot have seen the table stores of tiles t-2 .. t.  The walker keeps the hashes of exactly
 * those stores in a 32-entry register ring (one per lane) and tests "is the hash of this position
 * among them" with one compare + ballot; such a position (rare) is resolved by the scalar code.
 * The parse, the table and the output stay byte-identical to LZ4_compress_fast.
 * Hand-offs use named barriers (bar.sync / bar.arrive, 64 threads each): GO(i) walker -> preparer i
 * "tile may be prepared", FULL(i) preparer i -> walker "tile is in the ring"; preparer i owns the
 * tiles i, i+3, i+6, ... of a session.  Waiting warps are descheduled by the barrier hardware. */
#ifdef SIMT_EMU
static long long g_dbg_lz4t_sessions = 0, g_dbg_lz4t_seqs = 0, g_dbg_lz4t_stale = 0, g_dbg_lz4t_x[6];
#define LZ4T_DBG(x) do { if (lane_id() == 0) (x)++; } while (0)
#else
#define LZ4T_DBG(x) do {} while (0)
#endif
#define LZ4T_RING 256                      /* positions in the verdict ring = 8 tiles */
#define LZ4T_BAR_FULL(i) (1 + (i))
#define LZ4T_BAR_GO(i) (4 + (i))
#define LZ4T_QUIT 1
#define LZ4T_END 0xffffffffu               /* verdict of a tile too close to the end of the stream to be prepared */
#define LZ4T_LONG 13                       /* match-length field: 13 = "13 or more bytes after the first four" */
struct Lz4Team {
  uint2 vd[LZ4T_RING];                     /* .x verdict: bit 0 hit, bits 2..5 length field, bits 8..23 offset; .y hash */
  const u8* s;                             /* current stream */
  int n;
  int base;                                /* position of ring entry 0 in this session */
  int gen;                                 /* session number: a preparer restarts at its first tile when it changes */
  int cmd;                                 /* LZ4T_QUIT ends the preparers */
  int u16;                                 /* table flavour of the current stream */
};
#define LZ4T_SMEM_BYTES ((int)sizeof(Lz4Team))

DEV int lz4t_ld_i32(const int* p) { return *(const volatile int*)p; }

template <bool U16>
DEV void lz4_team_prepare_tile(Lz4Team* tm, const void* tabmem, const u8* s, int n, int w0) {
  const int lane = lane_id();
  const int p = w0 + lane;
  const int e = (w0 - lz4t_ld_i32(&tm->base) + lane) & (LZ4T_RING - 1);
  if (w0 + 31 + 24 > n) { tm->vd[e] = make_uint2(LZ4T_END, 0u); return; }     /* loads below reach byte p+19 (+3) */
  const StreamBase sb = make_stream_base(s);
  u32 r[5], a0, a1, a2, a3, a4, c0, c1, c2, c3, c4;
  ldp_raw20(sb, p, r);
  ldp_take17(sb, p, r, a0, a1, a2, a3, a4);
  const u32 h = lz4_hash_seq<U16>(a0, a1);
  /* racing with the walker's stores is fine: whatever this read misses is in the walker's ring */
  const int snap = U16 ? (int)((const volatile u16*)tabmem)[h] : (int)((const volatile u32*)tabmem)[h];
  u32 vx = 0;
  if (snap < p) {                                      /* always true for entries the serial code could see here */
    ldp_gather17(sb, snap, c0, c1, c2, c3, c4);
    const u32 x1 = a1 ^ c1, x2 = a2 ^ c2, x3 = a3 ^ c3;
    u32 m;
    if (x1) m = (u32)(__ffs((int)x1) - 1) >> 3;
    else if (x2) m = 4u + ((u32)(__ffs((int)x2) - 1) >> 3);
    else if (x3) m = 8u + ((u32)(__ffs((int)x3) - 1) >> 3);
    else m = a4 != c4 ? 12u : (u32)LZ4T_LONG;
    const bool hit = (U16 || snap + 65535 >= p) && c0 == a0;
    vx = (hit ? 1u : 0u) | (m << 2) | ((u32)((p - snap) & 0xffff) << 8);
  }
  tm->vd[e] = make_uint2(vx, h);
}

/* body of preparer warp i (0..2); returns when the walker posts LZ4T_QUIT */
DEV void lz4_team_preparer(Lz4Team* tm, const void* tabmem, int i) {
  int gen_seen = -1, tile = i;
  for (;;) {
    bar_sync(LZ4T_BAR_GO(i), 64);
    if (lz4t_ld_i32(&tm->cmd) == LZ4T_QUIT) return;
    const int gen = lz4t_ld_i32(&tm->gen);
    if (gen != gen_seen) { gen_seen = gen; tile = i; }
    const u8* s = *(const u8* const volatile*)&tm->s;
    const int n = lz4t_ld_i32(&tm->n), w0 = lz4t_ld_i32(&tm->base) + 32 * tile;
    if (lz4t_ld_i32(&tm->u16)) lz4_team_prepare_tile<true>(tm, tabmem, s, n, w0);
    else lz4_team_prepare_tile<false>(tm, tabmem, s, n, w0);
    tile += 3;
    __threadfence_block();
    bar_arrive(LZ4T_BAR_FULL(i), 64);
  }
}

/* Returns the compressed size, or 0 when the stream does not fit in `cap`
 * (LZ4_compress_fast's limitedOutput failure).  Uniform across the warp.
 * `tabmem` is LZ4_TABLE_BYTES of shared memory private to this warp.
 *
 * Hot-path shape (driven by the ncu source view: ~250 dependent warp instructions per sequence
 * on the hard byte-plane in v1, 72 now): everything uniform across the warp is computed
 * redundantly by all lanes; table stores in the scalar sections are done by lane 0 between
 * __syncwarp()s.  The first four probes of every search are scalar and work on 12-byte register
 * windows (one round of aligned loads each); the "test next position" probe that follows every
 * match is an inner loop on a lane-cached window (see below); a sequence with < 15 literals and a
 * short match is written by ONE predicated store (lane 0 = token, lanes 1..lit = literals, the
 * next two = offset).  The 32-wide probe rounds only run when the scalar probes miss. */
/* PACK (only with the 12-bit byU32 table, streams of at most 128 KiB): positions are 17 bits wide, so
 * the table is kept as 4096 x u16 plus one bit per entry -- 8.5 KiB instead of 16 KiB, i.e. twice as
 * many streams per SM.  It costs a few instructions per probe; measured with 4 chunks in flight it wins
 * at typesize 2 and 8 and loses at typesize 4, so the host only uses it on request (BLOSC_B200_LZ4_PACK=1). */
template <bool U16, bool PACK = false, bool TEAM = false>
DEV int lz4_encode_warp(const u8* __restrict__ s, const int n, u8* __restrict__ d, const int cap,
                        const int accel, void* tabmem, int* need_out, Lz4Team* tm = nullptr) {
  const int lane = lane_id();
  const StreamBase sb = make_stream_base(s);
  u16* tab16 = (u16*)tabmem;
  u32* tab32 = (u32*)tabmem;
  u32* tabhi = (u32*)((u8*)tabmem + 8192);                   /* PACK: bit 16 of the 4096 entries */
#define LZ4_TGET(h) (U16 ? (int)tab16[h] : PACK ? ((int)tab16[h] | (int)(((tabhi[(h) >> 5] >> ((h) & 31u)) & 1u) << 16)) : (int)tab32[h])
#define LZ4_TPUT(h, v) do { if (U16) tab16[h] = (u16)(v); else if (PACK) { tab16[h] = (u16)(v); const u32 m_ = 1u << ((h) & 31u); \
                            if ((v) & 0x10000) atomicOr(&tabhi[(h) >> 5], m_); else atomicAnd(&tabhi[(h) >> 5], ~m_); } \
                            else tab32[h] = (u32)(v); } while (0)

  for (int i = lane; i < (PACK ? LZ4_TAB17_BYTES : LZ4_TABLE_BYTES) / 4; i += 32) tab32[i] = 0;   /* LZ4_initStream, lz4.c:1384 */
  __syncwarp();

  const bool limited = (long long)cap < (long long)n + n / 255 + 16;   /* lz4.c:1388,1395 */
  const int olimit = cap;
  const int mfl1 = n - LZ4_MFLIMIT + 1;       /* mflimitPlusOne */
  const int matchlimit = n - LZ4_LASTLITERALS;
  int ip = 1, anchor = 0, op = 0;
  int need = 0;                               /* max left-hand side of the limitedOutput checks = smallest capacity that passes */
#define LZ4_LIMIT(v) do { const int v_ = (v); if (v_ > need) need = v_; if (limited && v_ > olimit) return 0; } while (0)
  /* first byte (lz4.c:1005-1010): table[hash(0)] = 0, which the zeroed table already says */

  /* Lane-cached window for the literal-free chains that dominate shuffled data: lane l keeps the
   * 12 bytes at position w0+l and their hash, so the "fill table at ip-2 / test ip" step
   * (lz4.c:1236-1294) fetches both hashes and the bytes to compare with shuffles instead of
   * reloading and re-hashing; a refill costs one round of loads per 2-3 sequences.  The 3-byte
   * sequences such a chain produces (token, offset) are parked one per lane and written together. */
  int w0 = -(1 << 30);
  u32 wq0 = 0, wq1 = 0, wq2 = 0, wh = 0;
  int pb = -(1 << 30);                       /* base of the window requested ahead of time */
  u32 pq0 = 0, pq1 = 0, pq2 = 0, pq3 = 0;    /* its raw aligned words */
  int nrec = 0, recop = 0;
  u32 rec = 0;
#define LZ4_FLUSH_CHECKED() do { if (nrec) { LZ4_LIMIT(op + (1 + LZ4_LASTLITERALS)); } LZ4_FLUSH(); } while (0)
#define LZ4_FLUSH() do { if (lane < nrec) { d[recop] = (u8)rec; d[recop + 1] = (u8)(rec >> 8); d[recop + 2] = (u8)(rec >> 16); \
                                             if ((rec & 15u) == 15u) d[recop + 3] = (u8)(rec >> 24); } nrec = 0; } while (0)

  if (n >= LZ4_MFLIMIT + 1) {                 /* lz4.c:1002 */
    bool post = false;                        /* true: a match just ended at ip (== anchor) */
    for (;;) {
      int match = 0, lit = 0, back = 0;
      u32 ipn = 0, cn = 0;                    /* bytes [ip+4, ip+8) and [match+4, match+8) of the hit */
      bool have_next = false, hit = false, imm = false, have_mc = false;
      int mc_carry = 0;

      bool scalar_post = post;
      if (TEAM && post && ip + 64 <= n) {
        /* ---- chained "test next position" (lz4.c:1236-1294) with the verdicts prepared by the helper
         * warps (see "team mode" above) ---- */
        scalar_post = false;
        bool finished = false, reanchor = false;
        if (nrec >= 24) LZ4_FLUSH_CHECKED();
        LZ4T_DBG(g_dbg_lz4t_sessions);
        const int base = ip - 2;
        if (lane == 0) {
          tm->s = s; tm->n = n; tm->u16 = U16 ? 1 : 0; tm->base = base;
          tm->gen = lz4t_ld_i32(&tm->gen) + 1;
        }
        __syncwarp();
        __threadfence_block();
        bar_arrive(LZ4T_BAR_GO(0), 64); bar_arrive(LZ4T_BAR_GO(1), 64); bar_arrive(LZ4T_BAR_GO(2), 64);
        u32 out = 7u;                         /* preparers that were told to go and whose tile has not been taken yet */
        int t = 0, li = 2;                    /* current tile of the session and position inside it: ip == base + 32 t + li */
        u32 ring_h = 0xffffffffu;             /* lane l: hash of the (l mod 32)-th most recent table store, or invalid */
        int ring_n = 0, rs_lo = 0, rs_1 = 0, rs_2 = 0;   /* stores so far; ring_n when tile t-2 / t-1 / t began */
        bool ovf = false;                     /* more than 32 stores inside the window: every verdict counts as stale */
        bar_sync(LZ4T_BAR_FULL(0), 64); out &= ~1u;
        const smem_addr_t vda = smem_addr(tm->vd);
        for (;;) {
          const u32 e = (u32)(32 * t + li);
          u32 pk, h;
          smem_ld_u32x2(vda, (e & (LZ4T_RING - 1)) << 3, pk, h);
          const u32 h2 = smem_ld_u32(vda, (((e - 2u) & (LZ4T_RING - 1)) << 3) + 4u);
          LZ4_TPUT(h2, ip - 2);                                            /* every lane the same word: no hand-off between lanes */
          if (ring_n - rs_lo >= 32) ovf = true;
          if (lane == (ring_n & 31)) ring_h = h2;
          ring_n++;
          const unsigned stale = __ballot_sync(FULLMASK, ring_h == h);
          if (stale || ovf || pk == LZ4T_END) { LZ4T_DBG(g_dbg_lz4t_stale); scalar_post = true; break; }      /* the plain probe below looks this one up itself */
          LZ4_TPUT(h, ip);                                                 /* lz4.c:1291: ip goes into the table, hit or not */
          if (ring_n - rs_lo >= 32) ovf = true;
          if (lane == (ring_n & 31)) ring_h = h;
          ring_n++;
          if (!(pk & 1u)) { LZ4T_DBG(g_dbg_lz4t_x[0]); ip++; break; }                                 /* lz4.c:1298; on to the search below */
          const int off = (int)(pk >> 8);
          int mc = (int)((pk >> 2) & 15u);
          if (mc == LZ4T_LONG) {
            LZ4T_DBG(g_dbg_lz4t_x[1]);
            mc = LZ4T_LONG + lz4_count_tail(sb, s, ip + 4 + LZ4T_LONG, ip - off + 4 + LZ4T_LONG, matchlimit, n);   /* ip+64 <= n: far from matchlimit */
            if (mc >= 15 + 255) {                                          /* very long match: general emission below */
              hit = true; imm = true; match = ip - off;
              have_mc = true; mc_carry = mc;
              LZ4T_DBG(g_dbg_lz4t_x[2]);
              break;
            }
          }
          /* lz4.c:1187-1226 with 0 literals: token, offset and -- from 19 bytes on -- one length byte.
           * Both limitedOutput checks of such a sequence ask for (op after it) + 6 <= olimit; op only
           * grows inside a chain, so the check is made once per parked batch, before anything is
           * written (LZ4_FLUSH_CHECKED) */
          const bool ext = mc >= 15;
          LZ4T_DBG(g_dbg_lz4t_seqs);
          if (lane == nrec) { rec = (ext ? 15u | ((u32)(mc - 15) << 24) : (u32)mc) | ((u32)off << 8); recop = op; }
          nrec++;
          op += ext ? 4 : 3;
          ip += mc + 4;
          li += mc + 4;
          anchor = ip;
          if (ip + 64 > n) {                                               /* a match ended close to the end of the stream */
            if (ip >= mfl1) finished = true;                               /* lz4.c:1230-1233 */
            else scalar_post = true;                                       /* the plain probe below takes over */
            break;
          }
          if (li >= 128) { LZ4T_DBG(g_dbg_lz4t_x[3]); reanchor = true; break; }                       /* jumped past everything that is being prepared */
          while (li >= 32) {                                               /* on to the next tile */
            __threadfence_block();
            bar_arrive(LZ4T_BAR_GO(t % 3), 64); out |= 1u << (t % 3);      /* its preparer may start tile t+3 */
            t++; li -= 32;
            rs_lo = rs_1; rs_1 = rs_2; rs_2 = ring_n;                      /* the window is now the stores of tiles t-2 .. t */
            {
              const int k = ring_n - 1 - ((ring_n - 1 - lane) & 31);       /* index of the store this lane holds */
              if (ring_n == 0 || k < rs_lo) ring_h = 0xffffffffu;
              ovf = ring_n - rs_lo > 32;
            }
            bar_sync(LZ4T_BAR_FULL(t % 3), 64); out &= ~(1u << (t % 3));
            if (nrec >= 24) LZ4_FLUSH_CHECKED();
          }
        }
        /* leave the session: take the tiles that are still being prepared, so that every preparer is
         * parked at its GO barrier again */
        for (int i = 0; i < 3; i++)
          if (out & (1u << i)) bar_sync(LZ4T_BAR_FULL(i), 64);
        if (finished) break;
        if (reanchor) continue;
      }
      if (!TEAM && post && ip + 64 <= n) {
        scalar_post = false;
        /* ---- chained "test next position" on the lane-cached window: stays in this loop for as
         * long as every match is immediately followed by another one ---- */
        bool room = true;
        for (;;) {
          if (ip - 2 < w0 || ip > w0 + 31) {
            if (nrec >= 24) LZ4_FLUSH_CHECKED();                             /* a window serves at most 8 sequences */
            /* The window that follows (base w0+30: the first ip past this window is >= w0+32) was
             * requested at the previous refill, so its bytes are here by now; only a long match
             * that jumps over it pays for a blocking load. */
            if (ip - 2 >= pb && ip <= pb + 31) { w0 = pb; ldp_take12(sb, w0 + lane, pq0, pq1, pq2, pq3, wq0, wq1, wq2); }
            else { w0 = ip - 2; ldp_win12(sb, w0 + lane, wq0, wq1, wq2); }   /* reaches byte w0+46 < ip+64 <= n */
            wh = lz4_hash_seq<U16>(wq0, wq1);
            pb = w0 + 30;
            if (pb + 31 + 16 <= n) ldp_raw12(sb, pb + lane, pq0, pq1, pq2, pq3);   /* not waited for */
            else pb = -(1 << 30);
            lz4d_prefetch(s, w0 + 192, lane == 0 ? n : 0);                   /* the line a few refills ahead */
          }
          const int li = ip - w0;                                            /* 2 .. 31 */
          const u32 h2 = __shfl_sync(FULLMASK, wh, li - 2);
          const u32 h = __shfl_sync(FULLMASK, wh, li);
          const u32 seq = __shfl_sync(FULLMASK, wq0, li);
          const u32 n4 = __shfl_sync(FULLMASK, wq1, li);                     /* bytes ip+4 .. ip+7 */
          const u32 n8 = __shfl_sync(FULLMASK, wq2, li);                     /* bytes ip+8 .. ip+11 */
          if (lane == 0) LZ4_TPUT(h2, ip - 2);
          __syncwarp();
          const int cand = LZ4_TGET(h);
          __syncwarp();                    /* every lane has read the old entry before lane 0 overwrites it */
          if (lane == 0) LZ4_TPUT(h, ip);
          u32 c0, c1, c2;
          ldp_win12(sb, cand, c0, c1, c2);   /* cand is a position < ip whatever the table holds: safe even when it is too far back */
          if (!((U16 || cand + 65535 >= ip) && c0 == seq)) { ip++; break; }  /* lz4.c:1298; on to the search below */
          int mc;
          const u32 x1 = n4 ^ c1, x2 = n8 ^ c2;
          if (x1 | x2) {
            const u32 xx = x1 ? x1 : x2;
            mc = ((__ffs((int)xx) - 1) >> 3) + (x1 ? 0 : 4);
          } else {                                                           /* >= 12 bytes: next 8 from memory */
            u32 p3, p4, q3, q4;
            ldp_win8(sb, ip + 12, p3, p4);
            ldp_win8(sb, cand + 12, q3, q4);
            const u32 x3 = p3 ^ q3, x4 = p4 ^ q4;
            if (x3) mc = 8 + eq_bytes32(x3);
            else if (x4) mc = 12 + eq_bytes32(x4);
            else mc = 16 + lz4_count_tail(sb, s, ip + 20, cand + 20, matchlimit, n);   /* ip+64 <= n: far from matchlimit */
          }
          if (mc >= 15 + 255) {                                              /* very long match: general emission below */
            hit = true; imm = true; match = cand;
            have_mc = true; mc_carry = mc;
            break;
          }
          /* lz4.c:1187-1226 with 0 literals: token, offset and -- from 19 bytes on -- one length byte.
           * Both limitedOutput checks of such a sequence ask for (op after it) + 6 <= olimit; op only
           * grows inside a chain, so the check is made once per parked batch, before anything is
           * written (LZ4_FLUSH_CHECKED) */
          const bool ext = mc >= 15;
          const int off = ip - cand;
          if (lane == nrec) { rec = (ext ? 15u | ((u32)(mc - 15) << 24) : (u32)mc) | ((u32)off << 8); recop = op; }
          nrec++;
          op += ext ? 4 : 3;
          ip += mc + 4;
          anchor = ip;
          if (ip + 64 > n) { room = false; break; }
        }
        if (!room) {                                                         /* a match ended close to the end of the stream */
          if (ip >= mfl1) break;                                             /* lz4.c:1230-1233 */
          continue;                                                          /* post stays true: the plain probe below takes over */
        }
      }
      if (scalar_post) {
        /* ---- fill table at ip-2, test position ip (lz4.c:1236-1294); no literals on a hit ---- */
        u32 b0, b1, b2 = 0;
        const bool wide = ip + 14 <= n;
        if (wide) ldp_win12(sb, ip - 2, b0, b1, b2);
        else { b0 = ld_u32(s + ip - 2); b1 = ld_u32(s + ip + 2); }
        const u32 seq = __funnelshift_r(b0, b1, 16);                       /* bytes ip .. ip+3 */
        const u32 h2 = lz4_hash_seq<U16>(b0, b1);                          /* 5th byte of ip-2 is s[ip+2] */
        const u32 h = lz4_hash_seq<U16>(seq, b1 >> 16);                    /* 5th byte of ip is s[ip+4] */
        if (lane == 0) LZ4_TPUT(h2, ip - 2);
        __syncwarp();
        const int cand = LZ4_TGET(h);
        __syncwarp();                      /* every lane has read the old entry before lane 0 overwrites it */
        if (lane == 0) LZ4_TPUT(h, ip);
        if (U16 || cand + 65535 >= ip) {
          u32 c0, c1;
          ldp_win8(sb, cand, c0, c1);
          if (c0 == seq) {
            hit = true; imm = true; match = cand;
            ipn = __funnelshift_r(b1, b2, 16); cn = c1; have_next = wide;
          }
        }
        if (!hit) ip++;                                                    /* lz4.c:1298 */
      }

      if (!hit) {
        /* ---- find a match (lz4.c:1043-1101): two scalar probes, then 32-wide rounds ---- */
        bool ended = false;
        for (int it = 0; it < LZ4_SCALAR_PROBES; it++) {
          const int pos = ip + (it ? 1 + (it - 1) * accel : 0);            /* probe offsets 0, 1, 1+accel, 1+2*accel (lz4.c:1043-1053) */
          if (ip + 1 + it * accel > mfl1) { ended = true; break; }         /* `goto _last_literals` (lz4.c:1055) */
          u32 b0, b1 = 0, b2 = 0;
          const bool wide = pos + 16 <= n;
          if (wide) ldp_win12(sb, pos, b0, b1, b2);
          else { b0 = ld_u32(s + pos); b1 = (u32)s[pos + 4]; }
          const u32 h = lz4_hash_seq<U16>(b0, b1);
          __syncwarp();                    /* table writes of the previous step are visible */
          const int cand = LZ4_TGET(h);
          __syncwarp();
          if (lane == 0) LZ4_TPUT(h, pos);
          if (U16 || cand + 65535 >= pos) {
            u32 c0, c1;
            ldp_win8(sb, cand, c0, c1);
            if (c0 == b0) {
              hit = true; ip = pos; match = cand;
              ipn = b1; cn = c1; have_next = wide;
              break;
            }
          }
        }
        if (!hit && !ended) {
          __syncwarp();
          for (int base_it = LZ4_SCALAR_PROBES;; base_it += 32) {
            const int itl = base_it + lane;
            const bool valid = ip + lz4_probe_offset(itl + 1, accel) <= mfl1;
            const int pos = valid ? ip + (int)lz4_probe_offset(itl, accel) : 0;
            u32 h = 0x80000000u | (u32)lane, seq = 0;
            if (valid) { seq = ld_u32(s + pos); h = lz4_hash_at<U16>(s, pos); }
            const unsigned vmask = __ballot_sync(FULLMASK, valid);
            const unsigned peers = __match_any_sync(FULLMASK, h);
            const unsigned lower = peers & ((1u << lane) - 1u);
            int cand = 0;
            bool lhit = false;
            if (valid) {
              cand = lower ? ip + (int)lz4_probe_offset(base_it + (31 - __clz((int)lower)), accel) : LZ4_TGET(h);
              if (U16 || cand + 65535 >= pos) lhit = ld_u32(s + cand) == seq;   /* lz4.c:1090-1101 */
            }
            const unsigned found = __ballot_sync(FULLMASK, lhit);
            const int nvalid = __popc(vmask);                       /* valid lanes form a prefix */
            const int f = found ? __ffs((int)found) - 1 : 32;
            const int last = f < nvalid - 1 ? f : nvalid - 1;       /* last probe committed to the table */
            __syncwarp();                                           /* all lookups done before any commit */
            if (valid && lane <= last) {
              const unsigned le = last >= 31 ? FULLMASK : ((1u << (last + 1)) - 1u);
              if ((((peers & le) >> lane) >> 1) == 0) LZ4_TPUT(h, pos);  /* highest committed lane per hash wins */
            }
            __syncwarp();
            if (found) {
              ip = __shfl_sync(FULLMASK, pos, f);
              match = __shfl_sync(FULLMASK, cand, f);
              hit = true;
              break;
            }
            if (nvalid < 32) break;                                  /* ran into the end: last literals */
          }
        }
        if (!hit) break;                                             /* -> last literals */

        /* ---- catch up (lz4.c:1107-1109) ---- */
        if (ip > anchor && match > 0 && s[ip - 1] == s[match - 1]) {
          for (;;) {
            const int a = ip - 1 - back - lane, b = match - 1 - back - lane;
            const bool ok = a >= anchor && b >= 0 && s[a] == s[b];
            const unsigned m = __ballot_sync(FULLMASK, ok);
            const int step = m == FULLMASK ? 32 : __ffs((int)~m) - 1;
            back += step;
            if (step < 32) break;
          }
        }
        lit = ip - back - anchor;
      }

      /* ---- match length (lz4.c:1182-1184): LZ4_count(start+4, ...) = catch-up bytes + forward bytes.
       * Most matches of shuffled data are 8..20 bytes long: compare that much with scalar
       * (warp-uniform) loads first and only then fall into the 512-bytes-per-round warp loop. ---- */
      int mc;
      if (have_mc) mc = mc_carry;                                    /* already counted by the chained probe */
      else {
        const int room = matchlimit - (ip + 4);                      /* >= 3 because ip < mflimitPlusOne */
        if (have_next) {
          const u32 x = ipn ^ cn;
          if (x) mc = eq_bytes32(x);
          else if (room > 20) {
            u32 p0, p1, p2, q0, q1, q2;                              /* bytes [ip+8, ip+20) vs [match+8, match+20) */
            ldp_win12(sb, ip + 8, p0, p1, p2);                        /* ip+8+16 <= n because room > 20 */
            ldp_win12(sb, match + 8, q0, q1, q2);
            const u32 x0 = p0 ^ q0, x1 = p1 ^ q1, x2 = p2 ^ q2;
            if (x0) mc = 4 + eq_bytes32(x0);
            else if (x1) mc = 8 + eq_bytes32(x1);
            else if (x2) mc = 12 + eq_bytes32(x2);
            else mc = 16 + lz4_count_tail(sb, s, ip + 20, match + 20, matchlimit, n);
          } else mc = 4 + (room > 4 ? warp_count_match(s, ip + 8, match + 8, matchlimit) : 0);
          if (mc > room) mc = room;
        } else mc = warp_count_match(s, ip + 4, match + 4, matchlimit);
      }
      const int off = ip - match;
      ip += mc + 4;
      mc += back;

      /* ---- emit (lz4.c:1112-1226) ---- */
      LZ4_FLUSH_CHECKED();
      const int token = op++;
      if (!imm) LZ4_LIMIT(op + lit + (2 + 1 + LZ4_LASTLITERALS) + lit / 255);
      if (lit < 15 && mc < 15) {
        LZ4_LIMIT(op + lit + 2 + (1 + LZ4_LASTLITERALS));
        u32 v;
        if (lane == 0) v = ((u32)lit << 4) | (u32)mc;
        else if (lane <= lit) v = s[anchor + lane - 1];
        else v = lane == lit + 1 ? (u32)off : (u32)off >> 8;
        if (lane <= lit + 2) d[token + lane] = (u8)v;
        op += lit + 2;
      } else {
        u32 tokval;
        if (lit >= 15) {
          const int len = lit - 15, nff = len / 255;
          tokval = 15u << 4;
          warp_fill_bytes(d + op, nff, 255);
          if (lane == 0) d[op + nff] = (u8)(len - nff * 255);
          op += nff + 1;
        } else tokval = (u32)lit << 4;
        warp_copy_bytes(d + op, s + anchor, lit);
        op += lit;
        if (lane == 0) { d[op] = (u8)off; d[op + 1] = (u8)(off >> 8); }
        op += 2;
        LZ4_LIMIT(op + (1 + LZ4_LASTLITERALS) + (mc + 240) / 255);
        if (mc >= 15) {
          tokval += 15;
          const int rest = mc - 15, nff = rest / 255;
          warp_fill_bytes(d + op, nff, 255);
          if (lane == 0) d[op + nff] = (u8)(rest - nff * 255);
          op += nff + 1;
        } else tokval += (u32)mc;
        if (lane == 0) d[token] = (u8)tokval;
      }

      anchor = ip;
      if (ip >= mfl1) break;                                         /* lz4.c:1230-1233 */
      post = true;
    }
  }

  /* ---- last literals (lz4.c:1302-1329) ---- */
  LZ4_FLUSH_CHECKED();
  const int lastRun = n - anchor;
  LZ4_LIMIT(op + lastRun + 1 + (lastRun + 255 - 15) / 255);
  if (lastRun >= 15) {
    const int acc = lastRun - 15, nff = acc / 255;
    if (lane == 0) d[op] = (u8)(15u << 4);
    op++;
    warp_fill_bytes(d + op, nff, 255);
    if (lane == 0) d[op + nff] = (u8)(acc - nff * 255);
    op += nff + 1;
  } else {
    if (lane == 0) d[op] = (u8)(lastRun << 4);
    op++;
  }
  warp_copy_bytes(d + op, s + anchor, lastRun);
  op += lastRun;
  *need_out = need;
  return op;
#undef LZ4_FLUSH_CHECKED
#undef LZ4_FLUSH
#undef LZ4_LIMIT
#undef LZ4_TGET
#undef LZ4_TPUT
}
