/*
 * dev_chunk.cuh -- chunk-level kernels: the GPU replacement of c-blosc's block
 * scheduler (reference blosc/blosc.c:803-918 serial_blosc/parallel_blosc/do_job and
 * :1706-1887 t_blosc) and of the per-block pipeline blosc_c / blosc_d (:591-800).
 *
 *   encode_kernel   one warp per LZ stream (= one split of one Blosc block): codec into a
 *                   worst-case slot (capacity neblock, as t_blosc's tmp2, :1810-1811)
 *   scan_kernel     exclusive scan of the per-block compressed sizes -> bstarts, total
 *                   cbytes and the "does it fit in destsize" verdict (:1843-1856)
 *   compact_kernel  writes the 16-byte header, bstarts[] and the int32-prefixed split
 *                   payloads at their final offsets (:1148-1247, :715, :1860)
 *   decode_kernel   one warp per LZ stream: bounds-checked walk of the size prefixes
 *                   (:761-770), raw-split copy or codec (:773-783)
 */
#pragma once
#include "b2_args.h"
#include "dev_blosclz.cuh"
#include "dev_common.cuh"
#include "dev_inflate.cuh"
#include "dev_lz4.cuh"
#include "dev_lz4dec.cuh"
#include "dev_lz4fast.cuh"
#include "dev_zstd.cuh"



/* Dynamic scheduling (the GPU counterpart of t_blosc's shared block counter, blosc.c:1769-1776):
 * every warp pulls the next job number from a global counter until none is left.  Jobs are
 * numbered longest-first as far as that is knowable without looking at the data: the unsplit
 * leftover block first, then split-major (split s of every block before split s+1), so that
 * the byte-planes that turn out to be hard start in the first wave and the cheap ones fill in
 * behind them.  Returns the stream index, or -1 when the queue is empty.  Every warp of a launch
 * draws exactly one ticket past the end, so a launch consumes nstreams + (warps launched) tickets. */
DEV int next_stream(int* queue, unsigned base, const StreamMap& m) {
  int job = 0;
  if (lane_id() == 0) job = (int)((unsigned)atomicAdd(queue, 1) - base);
  job = __shfl_sync(FULLMASK, job, 0);
  if (job >= m.nstreams) return -1;
  const int nfs = m.nfull * m.nsplits;
  if (m.leftover) {
    if (job == 0) return nfs;
    job--;
  }
  const int s = job / m.nfull, b = job - s * m.nfull;
  return b * m.nsplits + s;
}

/* stream index -> (block, offset inside the uncompressed buffer, length) */
DEV void stream_locate(const StreamMap& m, int idx, int* block, long long* off, int* len, int* split) {
  const int nfs = m.nfull * m.nsplits;
  if (idx < nfs) {
    const int b = idx / m.nsplits, s = idx - b * m.nsplits;
    const int neblock = m.blocksize / m.nsplits;
    *block = m.first_block + b;
    *off = (long long)(m.first_block + b) * m.blocksize + (long long)s * neblock;
    *len = neblock;
    *split = s;
  } else {
    *block = m.first_block + m.nfull;
    *off = (long long)(m.first_block + m.nfull) * m.blocksize;
    *len = m.leftover;
    *split = 0;
  }
}


/* L2 loads for words written by other SMs during this launch */
DEV int ld_cg_i32(const int* p) {
#ifdef SIMT_EMU
  return *p;
#else
  return __ldcg(p);
#endif
}

/* End of a launch that counts finished streams: a warp that finished `mine` of them adds them to *done; true for the
 * warp whose addition completes all nstreams (its loads after this see every other warp's writes). */
DEV bool finished_launch(int* done, int mine, int nstreams) {
  if (mine == 0) return false;
  __threadfence();
  int last = 0;
  if (lane_id() == 0) last = atomicAdd(done, mine) + mine == nstreams;
  last = __shfl_sync(FULLMASK, last, 0);
  if (!last) return false;
  __threadfence();
  return true;
}

/* The block scan of t_blosc's ordered copy-out (blosc.c:1843-1856) by ONE warp: exclusive scan of the
 * per-block compressed sizes -> bstarts, total cbytes and the "does it fit" verdict.  Run by the warp
 * that finishes the last stream of an encode launch, so compression needs no separate scan launch
 * (a 1-CTA launch queues behind the encoders of every other chunk in flight). */
DEV void warp_scan_blocks(const ScanArgs& a) {
  const int lane = lane_id();
  const int nblocks = a.nfull + (a.has_leftover ? 1 : 0);
  const int per = (nblocks + 31) / 32;
  const int b0 = lane * per < nblocks ? lane * per : nblocks, b1 = b0 + per < nblocks ? b0 + per : nblocks;
  long long sum = 0;
  for (int b = b0; b < b1; b++) {
    if (b < a.nfull) for (int s = 0; s < a.nsplits; s++) sum += 4 + (long long)ld_cg_i32(&a.csizes[(long long)b * a.nsplits + s]);
    else sum += 4 + (long long)ld_cg_i32(&a.csizes[(long long)a.nfull * a.nsplits]);
  }
  long long incl = sum;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const long long t = __shfl_up_sync(FULLMASK, incl, d);
    if (lane >= d) incl += t;
  }
  long long pos = 16 + 4ll * nblocks + (incl - sum);
  int bad = 0;
  for (int b = b0; b < b1; b++) {
    a.bstarts[b] = (int)(pos > 0x7fffffffll ? 0x7fffffffll : pos);
    const int ns = b < a.nfull ? a.nsplits : 1;
    const int neblock = b < a.nfull ? a.blocksize / a.nsplits : a.leftover;
    for (int s = 0; s < ns; s++) {
      const long long idx = b < a.nfull ? (long long)b * a.nsplits + s : (long long)a.nfull * a.nsplits;
      const int c = ld_cg_i32(&a.csizes[idx]);
      if (a.serial) {
        /* serial_blosc hands each codec call maxout = min(neblock, room left in dest) (blosc.c:646-651):
         * a clamped call only succeeds if the stream would have fitted that smaller budget, and a
         * raw split needs the full neblock (blosc.c:705-711) */
        const long long room = a.destsize - (pos + 4);
        if (room < neblock && !(room > 0 && c < neblock && ld_cg_i32(&a.needs[idx]) <= room)) bad = 1;
      }
      pos += 4 + (long long)c;
    }
  }
  const unsigned anybad = __ballot_sync(FULLMASK, bad);
  const long long total = 16 + 4ll * nblocks + __shfl_sync(FULLMASK, incl, 31);
  if (lane == 0) {
    a.result[B2_R_CBYTES] = (int)(total > 0x7fffffffll ? 0x7fffffffll : total);
    a.result[B2_R_FITS] = (total <= a.destsize && anybad == 0u) ? 1 : 0;       /* blosc.c:1848 / :836-839 give up */
  }
}

__global__ void encode_kernel(EncodeArgs a) {
#ifdef SIMT_EMU
  u8* smem = simt::g_dynsmem;
#else
  extern __shared__ __align__(16) u8 smem[];
#endif
  const int warp = (int)(threadIdx.x >> 5);
  void* tab = smem + (size_t)warp * a.table_bytes;
  int mine = 0;
  for (;;) {
    const int idx = next_stream(a.queue, a.queue_base, a.map);
    if (idx < 0) break;
    int block, len, split;
    long long off;
    stream_locate(a.map, idx, &block, &off, &len, &split);
    const u8* in = a.in + off;
    u8* out = a.slots + off;
    int c, need = 0;
    if (a.codec == B2_CODEC_LZ4) {
      if (a.table_bytes == LZ4_TAB17_BYTES) c = lz4_encode_warp<false, true>(in, len, out, len, a.accel, tab, &need);   /* host guarantees the length range */
      else if (len < 65536 + LZ4_MFLIMIT - 1) c = lz4_encode_warp<true>(in, len, out, len, a.accel, tab, &need);   /* lz4.c:710,1389 */
      else c = lz4_encode_warp<false>(in, len, out, len, a.accel, tab, &need);
    } else {
      c = blz_encode_warp(a.clevel, in, len, out, len, a.split_flag, tab, a.table_bytes, &need);
    }
    if (c <= 0 || c >= len) c = len;           /* blosc.c:705-714: incompressible split is stored raw */
    if (lane_id() == 0) { a.csizes[idx] = c; a.needs[idx] = need; }
    mine++;
    __syncwarp();
  }
  /* whoever completes the stream count does the block scan and puts the counters back to zero */
  if (!finished_launch(a.done, mine, a.map.nstreams)) return;
  if (a.fold_scan) warp_scan_blocks(a.scan);
  __syncwarp();
  if (lane_id() == 0) *a.done = 0;       /* (the ticket counter is never reset: warps that got no stream may still be polling it) */
}


/* LZ4 in team mode (dev_lz4.cuh): one CTA of four warps per stream -- a walker that owns the parse,
 * the table and the output, and three preparers that work ahead of it.  Shared memory: the stream's
 * hash table, then the Lz4Team block.  The walker warp alone draws tickets, counts finished streams
 * and runs the block scan, exactly as a warp of encode_kernel does. */
#define TEAM_WARPS 4
#define TEAM_CTAS_PER_SM 8
#define TEAM_SMEM_BYTES (LZ4_TABLE_BYTES + ((LZ4T_SMEM_BYTES + 15) & ~15))
__global__ void __launch_bounds__(TEAM_WARPS * 32, TEAM_CTAS_PER_SM) encode_team_kernel(EncodeArgs a) {
#ifdef SIMT_EMU
  u8* smem = simt::g_dynsmem;
#else
  extern __shared__ __align__(16) u8 smem[];
#endif
  void* tab = smem;
  Lz4Team* tm = (Lz4Team*)(smem + LZ4_TABLE_BYTES);
  const int warp = (int)(threadIdx.x >> 5);
  /* CTAs land on the SMs round-robin, so the CTAs of one SM differ in blockIdx / num_sms: rotating the
   * walker role with it puts the (busy) walkers of co-resident teams on different sub-partitions */
  const int walker = (int)((blockIdx.x / (unsigned)(a.num_sms > 0 ? a.num_sms : 1)) & 3u);
  if (threadIdx.x == 0) { tm->cmd = 0; tm->gen = 0; }
  __syncthreads();
  if (warp != walker) { lz4_team_preparer(tm, tab, (warp - walker - 1) & 3); return; }
  int mine = 0;
  for (;;) {
    const int idx = next_stream(a.queue, a.queue_base, a.map);
    if (idx < 0) break;
    int block, len, split;
    long long off;
    stream_locate(a.map, idx, &block, &off, &len, &split);
    const u8* in = a.in + off;
    u8* out = a.slots + off;
    int c, need = 0;
    if (len < 65536 + LZ4_MFLIMIT - 1) c = lz4_encode_warp<true, false, true>(in, len, out, len, a.accel, tab, &need, tm);   /* lz4.c:710,1389 */
    else c = lz4_encode_warp<false, false, true>(in, len, out, len, a.accel, tab, &need, tm);
    if (c <= 0 || c >= len) c = len;           /* blosc.c:705-714: incompressible split is stored raw */
    if (lane_id() == 0) { a.csizes[idx] = c; a.needs[idx] = need; }
    mine++;
    __syncwarp();
  }
  if (lane_id() == 0) *(volatile int*)&tm->cmd = LZ4T_QUIT;
  __syncwarp();
  __threadfence_block();
  bar_arrive(LZ4T_BAR_GO(0), 64); bar_arrive(LZ4T_BAR_GO(1), 64); bar_arrive(LZ4T_BAR_GO(2), 64);
  if (!finished_launch(a.done, mine, a.map.nstreams)) return;
  if (a.fold_scan) warp_scan_blocks(a.scan);
  __syncwarp();
  if (lane_id() == 0) *a.done = 0;
}


/* ---- segment-parallel LZ4 (dev_lz4fast.cuh): index_kernel, parse_kernel ---- */
#define INDEX_WARPS 4
/* one warp per stream, FAST_TAB_BYTES of shared memory each */
__global__ void __launch_bounds__(INDEX_WARPS * 32) index_kernel(FastArgs a) {
#ifdef SIMT_EMU
  u8* smem = simt::g_dynsmem;
#else
  extern __shared__ __align__(16) u8 smem[];
#endif
  const int warp = (int)(threadIdx.x >> 5);
  u32* tab = (u32*)(smem + (size_t)warp * FAST_TAB_BYTES);
  for (int idx = (int)blockIdx.x * INDEX_WARPS + warp; idx < a.map.nstreams; idx += (int)gridDim.x * INDEX_WARPS) {
    int block, len, split;
    long long off;
    stream_locate(a.map, idx, &block, &off, &len, &split);
    lz4f_index_warp(a.in + off, len, a.prev + off, tab, (u32)a.hash_mask);
    __syncwarp();
  }
}

/* One CTA per window of a stream (at most B2_FAST_WIN_MAX bytes): the window's bytes are staged in shared memory, then every THREAD parses one segment of FAST_SEG bytes.
 * Candidate compares -- the random accesses of LZ matching -- hit shared memory; only the chain links (prev[]) and
 * candidates in front of the window come from L2. */
__global__ void __launch_bounds__(B2_FAST_WIN_MAX / FAST_SEG, 3) parse_kernel(FastArgs a) {
#ifdef SIMT_EMU
  u8* smem = simt::g_dynsmem;
#else
  extern __shared__ __align__(16) u8 smem[];
#endif
  u32* sdata = (u32*)smem;
  int* sjob = (int*)(smem + a.win_bytes + 48);
  const int tid = (int)threadIdx.x, lane = lane_id();
  const int nfs = a.map.nfull * a.map.nsplits;
  const int njobs = nfs * a.groups_full + a.groups_left;
  const int spw = a.win_bytes / FAST_SEG;         /* segments per window (the CTA has a.threads <= spw threads) */
  for (;;) {
    if (tid == 0) { sjob[0] = (int)((unsigned)atomicAdd(a.queue, 1) - a.queue_base); sjob[1] = 0; }
    __syncthreads();
    const int job = sjob[0];
    if (job >= njobs) break;
    int idx, g, K;
    if (job < a.groups_left) { idx = nfs; g = job; K = a.segs_left; }
    else {
      /* split-major, as next_stream: the byte-planes that turn out to be hard start first */
      const int j = job - a.groups_left;
      const int per_split = a.map.nfull * a.groups_full;
      const int s = j / per_split, r = j - s * per_split;
      const int b = r / a.groups_full;
      g = r - b * a.groups_full;
      idx = b * a.map.nsplits + s; K = a.segs_full;
    }
    int block, len, split;
    long long off;
    stream_locate(a.map, idx, &block, &off, &len, &split);
    FastSeg* segs = a.segs + (long long)idx * a.segs_full;
    FastView v = fast_view(a.in + off, len);
    const int wa = g * a.win_bytes, wb = wa + a.win_bytes < len ? wa + a.win_bytes : len;
    /* stage the 16-byte granules that overlap the window (they lie inside the buffer's allocation: device
     * allocations start and end on coarser boundaries than that) */
    int i_lo = (wa + v.sal) >> 2;
    i_lo -= (int)(((uintptr_t)(v.w + i_lo) & 15u) >> 2);
    const int i_hi = i_lo + ((((wb + v.sal + 3) >> 2) - i_lo + 3) & ~3);
#ifdef SIMT_EMU
    for (int i = i_lo + tid; i < i_hi; i += (int)blockDim.x) sdata[i - i_lo] = (i >= 0 && i < v.nwords) ? v.w[i] : 0u;
#else
    {
      const uint4* g4 = (const uint4*)(v.w + i_lo);
      uint4* s4 = (uint4*)sdata;
      const int n4 = (i_hi - i_lo) >> 2;
#pragma unroll 4
      for (int i = tid; i < n4; i += (int)blockDim.x) s4[i] = __ldg(g4 + i);
    }
#endif
    __syncthreads();
    v.sm = sdata; v.sm_lo = i_lo; v.sm_hi = i_hi;
    v.lo_pos = wa; v.bias = v.sal - 4 * i_lo;      /* position p is byte p + sal - 4 i_lo of the staged words */
    /* the threads draw the window's segments from a counter: a thread whose segment was cheap takes another one
     * instead of waiting at the barrier for the slowest (the CTA may have fewer threads than the window has segments) */
    for (;;) {
      const int t = atomicAdd(&sjob[1], 1);
      const int k = g * spw + t;
      if (t >= spw || k >= K) break;
      const int sa = k * FAST_SEG, sb = sa + FAST_SEG < len ? sa + FAST_SEG : len;
      lz4f_parse_lane(v, len, a.prev + off, sa, sb, a.slots + off + sa, &segs[k], a.depth, a.accel, a.lazy);
    }
    __syncthreads();                               /* shared memory may be reused */
  }
}

/* One warp per stream: scan of its segment records (pending literals, continued matches, output offsets, compressed
 * size); the warp that finishes the last stream runs the block scan, exactly as in encode_kernel. */
#define FSCAN_WARPS 4
__global__ void __launch_bounds__(FSCAN_WARPS * 32) fscan_kernel(FastArgs a) {
  const int lane = lane_id();
  const int nfs = a.map.nfull * a.map.nsplits;
  int mine = 0;
  for (int idx = (int)blockIdx.x * FSCAN_WARPS + (int)(threadIdx.x >> 5); idx < a.map.nstreams; idx += (int)gridDim.x * FSCAN_WARPS) {
    int block, len, split;
    long long off;
    stream_locate(a.map, idx, &block, &off, &len, &split);
    int ptail = 0;
    int c = lz4f_stream_scan(a.segs + (long long)idx * a.segs_full, idx < nfs ? a.segs_full : a.segs_left, len, &ptail);
    if (c >= len) c = len;                         /* blosc.c:705-714: incompressible split is stored raw */
    if (lane == 0) { a.csizes[idx] = c; a.needs[idx] = c; a.ptail[idx] = ptail; }
    mine++;
    __syncwarp();
  }
  if (!finished_launch(a.done, mine, a.map.nstreams)) return;
  if (a.fold_scan) warp_scan_blocks(a.scan);
  __syncwarp();
  if (lane == 0) *a.done = 0;
}


#define SCAN_THREADS 1024
__global__ void __launch_bounds__(SCAN_THREADS) scan_kernel(ScanArgs a) {
  __shared__ long long part[SCAN_THREADS];
  const int tid = (int)threadIdx.x;
  const int nblocks = a.nfull + (a.has_leftover ? 1 : 0);
  const int per = (nblocks + SCAN_THREADS - 1) / SCAN_THREADS;
  const int b0 = tid * per, b1 = b0 + per < nblocks ? b0 + per : nblocks;
  long long sum = 0;
  for (int b = b0; b < b1; b++) {
    if (b < a.nfull) for (int s = 0; s < a.nsplits; s++) sum += 4 + (long long)a.csizes[(long long)b * a.nsplits + s];
    else sum += 4 + (long long)a.csizes[(long long)a.nfull * a.nsplits];
  }
  part[tid] = sum;
  __syncthreads();
  /* Hillis-Steele inclusive scan over the 1024 partials */
  for (int d = 1; d < SCAN_THREADS; d <<= 1) {
    const long long v = tid >= d ? part[tid - d] : 0;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  long long pos = 16 + 4ll * nblocks + (tid ? part[tid - 1] : 0);
  int bad = 0;
  for (int b = b0; b < b1; b++) {
    a.bstarts[b] = (int)(pos > 0x7fffffffll ? 0x7fffffffll : pos);
    const int ns = b < a.nfull ? a.nsplits : 1;
    const int neblock = b < a.nfull ? a.blocksize / a.nsplits : a.leftover;
    for (int s = 0; s < ns; s++) {
      const long long idx = b < a.nfull ? (long long)b * a.nsplits + s : (long long)a.nfull * a.nsplits;
      const int c = a.csizes[idx];
      if (a.serial) {
        /* serial_blosc hands each codec call maxout = min(neblock, room left in dest) (blosc.c:646-651):
         * a clamped call only succeeds if the stream would have fitted that smaller budget, and a
         * raw split needs the full neblock (blosc.c:705-711) */
        const long long room = a.destsize - (pos + 4);
        if (room < neblock && !(room > 0 && c < neblock && a.needs[idx] <= room)) bad = 1;
      }
      pos += 4 + (long long)c;
    }
  }
  if (bad) atomicOr(&a.result[2], 1);
  __syncthreads();
  if (tid == SCAN_THREADS - 1) {
    const long long total = 16 + 4ll * nblocks + part[SCAN_THREADS - 1];
    a.result[0] = (int)(total > 0x7fffffffll ? 0x7fffffffll : total);
    a.result[1] = (total <= a.destsize && a.result[2] == 0) ? 1 : 0;   /* blosc.c:1848 / :836-839 give up */
    a.result[2] = 0;
  }
}

/* CTA-cooperative copy, any alignment; vectorised when src/dst are mutually aligned */
DEV void cta_copy_bytes(u8* __restrict__ dst, const u8* __restrict__ src, int n) {
  const int tid = (int)threadIdx.x, nt = (int)blockDim.x;
  if ((((uintptr_t)dst ^ (uintptr_t)src) & 15u) == 0 && n >= 64) {
    int head = (int)((16u - ((uintptr_t)dst & 15u)) & 15u);
    if (head > n) head = n;
    for (int i = tid; i < head; i += nt) dst[i] = src[i];
    const int nv = (n - head) >> 4;
    const uint4* s4 = (const uint4*)(src + head);
    uint4* d4 = (uint4*)(dst + head);
    for (int i = tid; i < nv; i += nt) d4[i] = s4[i];
    for (int i = head + (nv << 4) + tid; i < n; i += nt) dst[i] = src[i];
  } else {
    for (int i = tid; i < n; i += nt) dst[i] = src[i];
  }
}


#define COMPACT_THREADS 256
__global__ void __launch_bounds__(COMPACT_THREADS) compact_kernel(CompactArgs a) {
  if (a.result[1] == 0) return;                 /* does not fit: host falls back to a MEMCPYED chunk */
  const int tid = (int)threadIdx.x;
  if (blockIdx.x == 0 && tid == 0) {            /* blosc.c:1154-1215 + :1275 */
    st_u32_bytes(a.dest, a.hdr0);
    st_u32_bytes(a.dest + 4, (u32)a.nbytes32);
    st_u32_bytes(a.dest + 8, (u32)a.map.blocksize);
    st_u32_bytes(a.dest + 12, (u32)a.result[0]);
  }
  for (int b = (int)blockIdx.x; b < a.nblocks; b += (int)gridDim.x) {
    int pos = a.bstarts[b];
    if (tid == 0) st_u32_bytes(a.dest + 16 + 4ll * b, (u32)pos);     /* blosc.c:816,1847 */
    const int ns = b < a.map.nfull ? a.map.nsplits : 1;
    for (int s = 0; s < ns; s++) {
      const int idx = b < a.map.nfull ? b * a.map.nsplits + s : a.map.nfull * a.map.nsplits;
      int blk, len, sp;
      long long off;
      stream_locate(a.map, idx, &blk, &off, &len, &sp);
      const int c = a.csizes[idx];
      if (tid == 0) st_u32_bytes(a.dest + pos, (u32)c);               /* blosc.c:715 */
      if (a.segs && c != len)
        lz4f_stitch_cta(a.dest + pos + 4, c, a.in + off, len, a.slots + off, a.segs + (long long)idx * a.segs_full,
                        b < a.map.nfull ? a.segs_full : a.segs_left, a.ptail[idx]);
      else cta_copy_bytes(a.dest + pos + 4, (c == len ? a.in : a.slots) + off, c);
      pos += 4 + c;
    }
  }
}


/* byte-wise: the size prefixes may sit in the last bytes of a caller-owned device chunk, and the
 * word-pair form of ld_u32 would touch up to 3 bytes past cbytes */
DEV int ld_i32(const u8* p) { return (int)((u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16) | ((u32)p[3] << 24)); }

/* Walk the size prefixes of a block up to one of its splits (blosc.c:760-771, :784): *so = the offset of the split's
 * payload in the chunk, *cs = its compressed size.  Returns 0 or B2_ERR_BOUNDS. */
DEV int locate_split(const DecodeArgs& a, int block, int split, int* so_out, int* cs_out) {
  int so = ld_i32(a.chunk + 16 + 4ll * block);
  int cs = 0;
  for (int s = 0; s <= split; s++) {
    if (so < 0 || so > a.cbytes - 4) return B2_ERR_BOUNDS;
    cs = ld_i32(a.chunk + so);
    so += 4;
    if (cs < 0 || cs > a.cbytes - so) return B2_ERR_BOUNDS;
    if (s < split) so += cs;
  }
  *so_out = so;
  *cs_out = cs;
  return 0;
}

#define DECODE_WARPS 4
/* dynamic shared memory: DECODE_WARPS * LZ4D_SMEM bytes (per-warp ring of recent output) */
/* One instantiation per codec: the bit-serial inflate must not cost the LZ decoders registers,
 * stack or instruction-cache footprint. */
template <int CODEC>
__global__ void __launch_bounds__(DECODE_WARPS * 32) decode_kernel(DecodeArgs a) {
#ifdef SIMT_EMU
  u8* smem = simt::g_dynsmem;
#else
  extern __shared__ __align__(16) u8 smem[];
#endif
  const int warp = (int)(threadIdx.x >> 5);
  int mine = 0;
  for (;;) {
    const int idx = next_stream(a.queue, a.queue_base, a.map);
    if (idx < 0) break;
    int block, len, split;
    long long off;
    stream_locate(a.map, idx, &block, &off, &len, &split);
    int so = 0, cs = 0;
    int err = locate_split(a, block, split, &so, &cs);
    if (!err) {
      u8* out = a.out + (off - a.out_shift);
      const u8* src = a.chunk + so;
      if (cs == len) warp_copy_bytes(out, src, len);                    /* stored raw, blosc.c:773-776 */
      else {
        int n;
        if (CODEC == B2_CODEC_LZ4) n = lz4_decode_warp(src, cs, out, len, smem + (size_t)warp * LZ4D_SMEM);
        else if (CODEC == B2_CODEC_ZLIB) n = zlib_decode_warp(src, cs, out, len, smem + (size_t)warp * LZ4D_SMEM);
        else if (CODEC == B2_CODEC_ZSTD) n = zstd_decode_warp(src, cs, out, len, smem + (size_t)warp * LZ4D_SMEM);
        else n = blz_decode_warp(src, cs, out, len);
        if (n != len) err = B2_ERR_CODEC;                               /* blosc.c:778-782 */
      }
    }
    if (err && lane_id() == 0) atomicMin(a.status, err);
    mine++;
    __syncwarp();
  }
  if (!finished_launch(a.done, mine, a.map.nstreams)) return;
  if (lane_id() == 0) { *a.status_out = ld_cg_i32(a.status); *a.status = 0; *a.done = 0; }
}


/* LZ4 chunks: one CTA of two warps per stream -- a parser that walks the tokens and a copier that owns the output
 * (dev_lz4dec.cuh).  The parser warp alone draws tickets, checks the size prefixes, counts finished streams and
 * publishes the verdict, exactly as a warp of decode_kernel does. */
#define PAIR_CTAS_PER_SM 12
__global__ void __launch_bounds__(64) decode_pair_kernel(DecodeArgs a) {
#ifdef SIMT_EMU
  u8* smem = simt::g_dynsmem;
#else
  extern __shared__ __align__(16) u8 smem[];
#endif
  Lz4pSlot* slots = lz4_pair_setup(smem);
  if (!slots) return;
  int mine = 0;
  for (;;) {
    const int idx = next_stream(a.queue, a.queue_base, a.map);
    if (idx < 0) break;
    int block, len, split;
    long long off;
    stream_locate(a.map, idx, &block, &off, &len, &split);
    int so = 0, cs = 0;
    int err = locate_split(a, block, split, &so, &cs);
    if (!err) {
      u8* out = a.out + (off - a.out_shift);
      const u8* src = a.chunk + so;
      if (cs == len) warp_copy_bytes(out, src, len);                    /* stored raw, blosc.c:773-776 */
      else if (lz4_pair_parse(src, cs, out, len, slots) != len) err = B2_ERR_CODEC;   /* blosc.c:778-782 */
    }
    if (err && lane_id() == 0) atomicMin(a.status, err);
    mine++;
    __syncwarp();
  }
  lz4_pair_quit(slots);
  if (!finished_launch(a.done, mine, a.map.nstreams)) return;
  if (lane_id() == 0) { *a.status_out = ld_cg_i32(a.status); *a.status = 0; *a.done = 0; }
}
