/*
 * backend_emu.cpp -- TEST INFRASTRUCTURE ONLY.
 *
 * Implements c-blosc_b200/csrc/b2_backend.h on plain host memory by running the very
 * same device kernels (dev_*.cuh) inside the lock-step SIMT emulator.  Linking the
 * product's host code (blosc_b200.c) against this file gives a CPU-runnable build of
 * the whole library for the `-m "not gpu"` tests.  It is never shipped or loaded by
 * the product: the product's .so links backend_cuda.cu instead.
 */
#include "simt_emu.h"

#include <new>

#include "../../c-blosc_b200/csrc/b2_backend.h"
#include "../../c-blosc_b200/csrc/dev_chunk.cuh"
#include "../../c-blosc_b200/csrc/dev_filters.cuh"

struct b2_stream_s { int dummy; };
static int g_all_device = 0;
static long long g_launches = 0;
static int g_last_need = 0;
static int g_blz_pack = 1;
static int g_lz4_pack = 0;

extern "C" {

void emu_set_all_device(int on) { g_all_device = on; }
unsigned long long emu_collectives(void) { return simt::g_collectives; }
int emu_last_need(void) { return g_last_need; }
void emu_set_blz_pack(int on) { g_blz_pack = on; }
void emu_set_lz4_pack(int on) { g_lz4_pack = on; }
void emu_lz4d_counters(long long* c) { c[0] = g_dbg_lz4d_batch_seqs; c[1] = g_dbg_lz4d_fast_seqs; c[2] = g_dbg_lz4d_general_seqs; c[3] = g_dbg_lz4d_dense_seqs; }

int b2_backend_init(void) { return 0; }
int b2_get_device(void) { return 0; }
int b2_set_device(int) { return 0; }
int b2_device_prepare(void) { return 0; }
int b2_stream_create(b2_stream_t* s) { *s = new b2_stream_s; return 0; }
void b2_stream_destroy(b2_stream_t s) { delete s; }
int b2_stream_sync(b2_stream_t) { return 0; }
int b2_dev_alloc(void** p, size_t n) { *p = malloc(n ? n : 1); return *p ? 0 : -1; }
void b2_dev_free(void* p) { free(p); }
int b2_pinned_alloc(void** p, size_t n) { *p = malloc(n ? n : 1); return *p ? 0 : -1; }
void b2_pinned_free(void* p) { free(p); }
int b2_ptr_is_device(const void*) { return g_all_device; }
static int g_all_pinned = 1;
void emu_set_all_pinned(int on) { g_all_pinned = on; }
int b2_ptr_is_pinned(const void*) { return g_all_pinned; }
struct b2_event_s { int dummy; };
int b2_event_create(b2_event_t* e) { *e = new b2_event_s; return 0; }
void b2_event_destroy(b2_event_t e) { delete e; }
int b2_event_record(b2_event_t, b2_stream_t) { return 0; }
int b2_event_sync(b2_event_t) { return 0; }
int b2_copy_h2d(void* d, const void* h, size_t n, b2_stream_t) { memcpy(d, h, n); return 0; }
int b2_copy_d2h(void* h, const void* d, size_t n, b2_stream_t) { memcpy(h, d, n); return 0; }
int b2_copy_d2d(void* d, const void* s, size_t n, b2_stream_t) { memmove(d, s, n); return 0; }
int b2_memset_dev(void* d, int v, size_t n, b2_stream_t) { memset(d, v, n); return 0; }
void b2_prof_enable(int) {}
void b2_prof_reset(void) {}
int b2_prof_get(int, double* ms, long long* n) { if (ms) *ms = 0; if (n) *n = 0; return 0; }
long long b2_launch_count(void) { return g_launches; }

int b2_launch_filter(const FilterArgs* a, b2_stream_t) {
  const bool bit = a->mode >= FILT_BITSHUFFLE;
  const long long nblocks = (a->nbytes + a->blocksize - 1) / a->blocksize;
  const long long ipb = (a->blocksize / a->typesize + FILT_TILE - 1) / FILT_TILE + 1;
  long long ctas = (nblocks * ipb + FILT_WARPS - 1) / FILT_WARPS;
  if (ctas > 7) ctas = 7;          /* small odd grid: exercises the grid-stride loop */
  if (ctas < 1) ctas = 1;
  g_launches++;
  FilterArgs args = *a;
  simt::launch(simt::Dim3((unsigned)ctas), simt::Dim3(FILT_WARPS * 32), bit ? FILT_WARPS * 16 * FILT_TILE : 0,
               [&] { if (args.typesize == 4) filter_kernel<4>(args); else filter_kernel<0>(args); });
  return 0;
}

static int g_lz4_team = 1;
void emu_set_lz4_team(int on) { g_lz4_team = on; }
void emu_lz4t_counters(long long* c) { c[0] = g_dbg_lz4t_sessions; c[1] = g_dbg_lz4t_seqs; c[2] = g_dbg_lz4t_stale; for (int i = 0; i < 4; i++) c[3 + i] = g_dbg_lz4t_x[i]; }

int b2_launch_encode(const EncodeArgs* a, b2_stream_t) {
  if (g_lz4_team && a->codec == B2_CODEC_LZ4 && a->table_bytes == LZ4_TABLE_BYTES) {
    int ctas = a->map.nstreams;
    if (ctas > 3) ctas = 3;          /* few CTAs: every team goes through several streams */
    if (ctas <= 0) return 0;
    g_launches++;
    EncodeArgs args = *a;
    args.num_sms = 2;
    args.queue_base = *a->queue_base_host;
    *a->queue_base_host += (unsigned)a->map.nstreams + (unsigned)ctas;
    simt::launch(simt::Dim3((unsigned)ctas), simt::Dim3(TEAM_WARPS * 32), TEAM_SMEM_BYTES, [&] { encode_team_kernel(args); });
    return 0;
  }
  int wpc = 65536 / a->table_bytes;
  if (wpc > 4) wpc = 4;
  if (wpc < 1) wpc = 1;
  const int ctas = (a->map.nstreams + wpc - 1) / wpc;
  if (ctas <= 0) return 0;
  g_launches++;
  EncodeArgs args = *a;
  args.queue_base = *a->queue_base_host;
  *a->queue_base_host += (unsigned)a->map.nstreams + (unsigned)ctas * (unsigned)wpc;
  simt::launch(simt::Dim3((unsigned)ctas), simt::Dim3(wpc * 32), (size_t)wpc * a->table_bytes, [&] { encode_kernel(args); });
  return 0;
}

int b2_launch_fast(const FastArgs* a, b2_stream_t) {
  if (a->map.nstreams <= 0) return 0;
  g_launches += 3;
  FastArgs args = *a;
  simt::launch(simt::Dim3(2), simt::Dim3(INDEX_WARPS * 32), INDEX_WARPS * FAST_TAB_BYTES, [&] { index_kernel(args); });
  const long long njobs = (long long)a->map.nfull * a->map.nsplits * a->groups_full + a->groups_left;
  long long ctas = njobs < 3 ? njobs : 3;
  args.queue_base = *a->queue_base_host;
  *a->queue_base_host += (unsigned)njobs + (unsigned)ctas;
  simt::launch(simt::Dim3((unsigned)ctas), simt::Dim3(a->threads), (size_t)a->win_bytes + 64, [&] { parse_kernel(args); });
  simt::launch(simt::Dim3(2), simt::Dim3(FSCAN_WARPS * 32), 0, [&] { fscan_kernel(args); });
  return 0;
}

int b2_launch_scan(const ScanArgs* a, b2_stream_t) {
  g_launches++;
  ScanArgs args = *a;
  simt::launch(simt::Dim3(1), simt::Dim3(SCAN_THREADS), 0, [&] { scan_kernel(args); });
  return 0;
}

int b2_launch_compact(const CompactArgs* a, b2_stream_t) {
  int ctas = a->nblocks;
  if (ctas > 5) ctas = 5;
  if (ctas <= 0) return 0;
  g_launches++;
  CompactArgs args = *a;
  simt::launch(simt::Dim3((unsigned)ctas), simt::Dim3(COMPACT_THREADS), 0, [&] { compact_kernel(args); });
  return 0;
}

static int g_lz4d_pair = 1;
void emu_set_lz4d_pair(int on) { g_lz4d_pair = on; }

int b2_launch_decode(const DecodeArgs* a, b2_stream_t) {
  if (g_lz4d_pair && a->codec == B2_CODEC_LZ4) {
    int ctas = a->map.nstreams < 3 ? a->map.nstreams : 3;      /* few CTAs: every pair goes through several streams */
    if (ctas <= 0) return 0;
    g_launches++;
    DecodeArgs args = *a;
    args.queue_base = *a->queue_base_host;
    *a->queue_base_host += (unsigned)a->map.nstreams + (unsigned)ctas;
    simt::launch(simt::Dim3((unsigned)ctas), simt::Dim3(64), LZ4P_SMEM, [&] { decode_pair_kernel(args); });
    return 0;
  }
  const int wpc = DECODE_WARPS;
  const int ctas = (a->map.nstreams + wpc - 1) / wpc;
  if (ctas <= 0) return 0;
  g_launches++;
  DecodeArgs args = *a;
  args.queue_base = *a->queue_base_host;
  *a->queue_base_host += (unsigned)a->map.nstreams + (unsigned)ctas * (unsigned)wpc;
  simt::launch(simt::Dim3((unsigned)ctas), simt::Dim3(wpc * 32), (size_t)wpc * LZ4D_SMEM, [&] {
    if (args.codec == B2_CODEC_LZ4) decode_kernel<B2_CODEC_LZ4>(args);
    else if (args.codec == B2_CODEC_ZLIB) decode_kernel<B2_CODEC_ZLIB>(args);
    else if (args.codec == B2_CODEC_ZSTD) decode_kernel<B2_CODEC_ZSTD>(args);
    else decode_kernel<B2_CODEC_BLOSCLZ>(args);
  });
  return 0;
}

/* ---- single-stream entry points for codec unit tests (one warp) ---- */
int emu_lz4_encode(const unsigned char* src, int n, unsigned char* dst, int cap, int accel) {
  int result = 0;
  simt::launch(simt::Dim3(1), simt::Dim3(32), LZ4_TABLE_BYTES, [&] {
    int need = 0;
    int r;
    if (g_lz4_pack && n >= LZ4_TAB17_MINLEN && n <= LZ4_TAB17_MAXLEN) r = lz4_encode_warp<false, true>(src, n, dst, cap, accel, simt::g_dynsmem, &need);
    else r = n < 65536 + LZ4_MFLIMIT - 1 ? lz4_encode_warp<true>(src, n, dst, cap, accel, simt::g_dynsmem, &need)
                                        : lz4_encode_warp<false>(src, n, dst, cap, accel, simt::g_dynsmem, &need);
    if ((threadIdx.x & 31) == 3) g_last_need = need;
    if ((threadIdx.x & 31) == 7) result = r;
  });
  return result;
}
/* the same stream through a whole team (walker + three preparers) */
int emu_lz4_encode_team(const unsigned char* src, int n, unsigned char* dst, int cap, int accel, int walker) {
  int result = 0;
  simt::launch(simt::Dim3(1), simt::Dim3(TEAM_WARPS * 32), TEAM_SMEM_BYTES, [&] {
    unsigned char* smem = simt::g_dynsmem;
    Lz4Team* tm = (Lz4Team*)(smem + LZ4_TABLE_BYTES);
    const int warp = (int)(threadIdx.x >> 5);
    if (threadIdx.x == 0) { tm->cmd = 0; tm->gen = 0; }
    __syncthreads();
    if (warp != walker) { lz4_team_preparer(tm, smem, (warp - walker - 1) & 3); return; }
    int need = 0;
    int r = n < 65536 + LZ4_MFLIMIT - 1 ? lz4_encode_warp<true, false, true>(src, n, dst, cap, accel, smem, &need, tm)
                                        : lz4_encode_warp<false, false, true>(src, n, dst, cap, accel, smem, &need, tm);
    if ((threadIdx.x & 31) == 0) *(volatile int*)&tm->cmd = LZ4T_QUIT;
    __syncwarp();
    bar_arrive(LZ4T_BAR_GO(0), 64); bar_arrive(LZ4T_BAR_GO(1), 64); bar_arrive(LZ4T_BAR_GO(2), 64);
    if ((threadIdx.x & 31) == 3) g_last_need = need;
    if ((threadIdx.x & 31) == 7) result = r;
  });
  return result;
}
int emu_lz4_decode(const unsigned char* src, int csize, unsigned char* dst, int cap) {
  int result = 0;
  simt::launch(simt::Dim3(1), simt::Dim3(32), LZ4D_SMEM, [&] {
    int r = lz4_decode_warp(src, csize, dst, cap, simt::g_dynsmem);
    if ((threadIdx.x & 31) == 13) result = r;
  });
  return result;
}
/* the same stream through a parser / copier pair */
int emu_lz4_decode_pair(const unsigned char* src, int csize, unsigned char* dst, int cap) {
  int result = 0;
  simt::launch(simt::Dim3(1), simt::Dim3(64), LZ4P_SMEM, [&] {
    Lz4pSlot* slots = lz4_pair_setup(simt::g_dynsmem);
    if (!slots) return;
    int r = lz4_pair_parse(src, csize, dst, cap, slots);
    lz4_pair_quit(slots);
    if ((threadIdx.x & 31) == 13) result = r;
  });
  return result;
}
int emu_blz_encode(int clevel, const unsigned char* src, int n, unsigned char* dst, int maxout, int split) {
  int result = 0;
  simt::launch(simt::Dim3(1), simt::Dim3(32), 65536, [&] {
    int need = 0;
    int r = blz_encode_warp(clevel, src, n, dst, maxout, split, simt::g_dynsmem, (n <= BLZ_TAB17_MAXLEN && g_blz_pack) ? BLZ_TAB17_BYTES : 65536, &need);
    if ((threadIdx.x & 31) == 3) g_last_need = need;
    if ((threadIdx.x & 31) == 31) result = r;
  });
  return result;
}
int emu_blz_decode(const unsigned char* src, int csize, unsigned char* dst, int cap) {
  int result = 0;
  simt::launch(simt::Dim3(1), simt::Dim3(32), 0, [&] {
    int r = blz_decode_warp(src, csize, dst, cap);
    if ((threadIdx.x & 31) == 0) result = r;
  });
  return result;
}

int emu_zlib_decode(const unsigned char* src, int csize, unsigned char* dst, int cap) {
  int result = 0;
  simt::launch(simt::Dim3(1), simt::Dim3(32), INF_SMEM_BYTES, [&] {
    int r = zlib_decode_warp(src, csize, dst, cap, simt::g_dynsmem);
    if ((threadIdx.x & 31) == 17) result = r;
  });
  return result;
}

int emu_zstd_fail_line(void) { return g_zs_fail_line; }
int emu_zstd_decode(const unsigned char* src, int csize, unsigned char* dst, int cap) {
  int result = 0;
  simt::launch(simt::Dim3(1), simt::Dim3(32), ZS_SMEM_BYTES, [&] {
    int r = zstd_decode_warp(src, csize, dst, cap, simt::g_dynsmem);
    if ((threadIdx.x & 31) == 9) result = r;
  });
  return result;
}

}  // extern "C"
