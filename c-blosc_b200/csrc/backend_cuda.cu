/*
 * backend_cuda.cu -- CUDA (sm_100a) implementation of b2_backend.h: kernel launches,
 * device memory, streams, per-kernel event timing.  Compiled with
 *   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo
 * Grid sizing: the codec kernels launch one warp per LZ stream and let the hardware
 * scheduler keep all 148 SMs busy (12 LZ4 warps / 3 BloscLZ warps resident per SM, the
 * limit being the shared-memory hash tables); the bandwidth-bound filter kernel runs a
 * grid-stride loop over 148 x 8 CTAs.
 */
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include "b2_backend.h"
#include "dev_chunk.cuh"
#include "dev_filters.cuh"

struct b2_stream_s {
  cudaStream_t s;
};

#define B2_MAX_DEVICES 64
static int g_sms[B2_MAX_DEVICES];     /* SM count per device, filled by b2_device_prepare */
static int g_prof_on = 0;
static double g_prof_ms[B2_K_COUNT];
static long long g_prof_n[B2_K_COUNT];
static long long g_launches = 0;

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      fprintf(stderr, "blosc_b200: CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
      return -1;                                                                              \
    }                                                                                         \
  } while (0)

static int num_sms(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return 148; }
  return (dev >= 0 && dev < B2_MAX_DEVICES && g_sms[dev] > 0) ? g_sms[dev] : 148;
}

/* per-device one-time setup (SM count; opt-in to > 48 KiB dynamic shared memory) */
extern "C" int b2_device_prepare(void) {
  int dev = 0, n = 0;
  CK(cudaGetDevice(&dev));
  if (dev >= 0 && dev < B2_MAX_DEVICES && g_sms[dev] == 0) {
    CK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    g_sms[dev] = n;
  }
  /* (no cudaFuncAttributePreferredSharedMemoryCarveout: measured, the codec kernels are faster with the driver's
   * default split -- fewer resident CTAs but more L1 -- than with the largest shared-memory carve-out) */
  CK(cudaFuncSetAttribute(encode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
  CK(cudaFuncSetAttribute(encode_team_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TEAM_SMEM_BYTES));
  CK(cudaFuncSetAttribute(decode_kernel<B2_CODEC_LZ4>, cudaFuncAttributeMaxDynamicSharedMemorySize, DECODE_WARPS * LZ4D_SMEM));
  CK(cudaFuncSetAttribute(decode_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ4P_SMEM));
  CK(cudaFuncSetAttribute(decode_kernel<B2_CODEC_BLOSCLZ>, cudaFuncAttributeMaxDynamicSharedMemorySize, DECODE_WARPS * LZ4D_SMEM));
  CK(cudaFuncSetAttribute(decode_kernel<B2_CODEC_ZLIB>, cudaFuncAttributeMaxDynamicSharedMemorySize, DECODE_WARPS * LZ4D_SMEM));
  CK(cudaFuncSetAttribute(decode_kernel<B2_CODEC_ZSTD>, cudaFuncAttributeMaxDynamicSharedMemorySize, DECODE_WARPS * LZ4D_SMEM));
  CK(cudaFuncSetAttribute(index_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, INDEX_WARPS * FAST_TAB_BYTES));
  CK(cudaFuncSetAttribute(parse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, B2_FAST_WIN_MAX + 64));
  CK(cudaFuncSetAttribute(filter_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, FILT_WARPS * 16 * FILT_TILE));
  CK(cudaFuncSetAttribute(filter_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, FILT_WARPS * 16 * FILT_TILE));
  CK(cudaFuncSetAttribute(filter_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, FILT_WARPS * 16 * FILT_TILE));
  CK(cudaFuncSetAttribute(filter_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, FILT_WARPS * 16 * FILT_TILE));
  return 0;
}

extern "C" int b2_backend_init(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) { cudaGetLastError(); return -1; }
  return b2_device_prepare();
}

extern "C" int b2_get_device(void) { int d = 0; if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); return 0; } return d; }
extern "C" int b2_set_device(int dev) { CK(cudaSetDevice(dev)); return 0; }

extern "C" int b2_stream_create(b2_stream_t* s) {
  b2_stream_s* st = new b2_stream_s;
  /* a blocking stream: like cudaMemcpy, a call is ordered after whatever the caller has already queued on
   * the legacy default stream (where e.g. PyTorch produces the buffers it hands in) */
  if (cudaStreamCreateWithFlags(&st->s, cudaStreamDefault) != cudaSuccess) { delete st; return -1; }
  *s = st;
  return 0;
}
extern "C" void b2_stream_destroy(b2_stream_t s) { if (s) { cudaStreamDestroy(s->s); delete s; } }
extern "C" int b2_stream_sync(b2_stream_t s) { CK(cudaStreamSynchronize(s ? s->s : 0)); return 0; }

extern "C" int b2_dev_alloc(void** p, size_t n) { CK(cudaMalloc(p, n)); return 0; }
extern "C" void b2_dev_free(void* p) { cudaFree(p); }
extern "C" int b2_pinned_alloc(void** p, size_t n) { CK(cudaMallocHost(p, n)); return 0; }
extern "C" void b2_pinned_free(void* p) { cudaFreeHost(p); }

extern "C" int b2_ptr_is_device(const void* p) {
  cudaPointerAttributes a;
  if (p == NULL) return 0;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return 0; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

extern "C" int b2_ptr_is_pinned(const void* p) {
  cudaPointerAttributes a;
  if (p == NULL) return 0;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return 0; }
  return a.type == cudaMemoryTypeHost;
}

struct b2_event_s { cudaEvent_t e; };
extern "C" int b2_event_create(b2_event_t* e) {
  b2_event_s* ev = new b2_event_s;
  if (cudaEventCreateWithFlags(&ev->e, cudaEventDisableTiming) != cudaSuccess) { delete ev; return -1; }
  *e = ev;
  return 0;
}
extern "C" void b2_event_destroy(b2_event_t e) { if (e) { cudaEventDestroy(e->e); delete e; } }
extern "C" int b2_event_record(b2_event_t e, b2_stream_t s) { CK(cudaEventRecord(e->e, s->s)); return 0; }
extern "C" int b2_event_sync(b2_event_t e) { CK(cudaEventSynchronize(e->e)); return 0; }

extern "C" int b2_copy_h2d(void* d, const void* h, size_t n, b2_stream_t s) { CK(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, s->s)); return 0; }
extern "C" int b2_copy_d2h(void* h, const void* d, size_t n, b2_stream_t s) { CK(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, s->s)); return 0; }
extern "C" int b2_copy_d2d(void* d, const void* s_, size_t n, b2_stream_t s) { CK(cudaMemcpyAsync(d, s_, n, cudaMemcpyDeviceToDevice, s->s)); return 0; }
extern "C" int b2_memset_dev(void* d, int v, size_t n, b2_stream_t s) { CK(cudaMemsetAsync(d, v, n, s->s)); return 0; }

/* ---- profiling: CUDA events recorded on the launching stream around every kernel;
 * nothing synchronises until the numbers are read (b2_prof_get), so profiling can stay
 * on inside a timed region. ---- */
#include <mutex>
#include <vector>
struct PendingEv { cudaEvent_t e0, e1; int kind; };
static std::vector<PendingEv> g_pending;
static std::mutex g_prof_mu;

struct ProfScope {
  cudaEvent_t e0, e1;
  int kind;
  cudaStream_t s;
  bool on;
  ProfScope(int k, cudaStream_t st) : kind(k), s(st), on(g_prof_on != 0) {
    if (on) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, s); }
  }
  ~ProfScope() {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_launches++;
    if (on) { cudaEventRecord(e1, s); g_pending.push_back({e0, e1, kind}); }
  }
};

static void prof_resolve() {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (auto& p : g_pending) {
    float ms = 0;
    cudaEventSynchronize(p.e1);
    cudaEventElapsedTime(&ms, p.e0, p.e1);
    g_prof_ms[p.kind] += ms; g_prof_n[p.kind]++;
    cudaEventDestroy(p.e0); cudaEventDestroy(p.e1);
  }
  g_pending.clear();
}

extern "C" void b2_prof_enable(int on) { g_prof_on = on; }
extern "C" void b2_prof_reset(void) { prof_resolve(); for (int i = 0; i < B2_K_COUNT; i++) { g_prof_ms[i] = 0; g_prof_n[i] = 0; } }
extern "C" int b2_prof_get(int kind, double* ms, long long* n) {
  if (kind < 0 || kind >= B2_K_COUNT) return -1;
  prof_resolve();
  if (ms) *ms = g_prof_ms[kind];
  if (n) *n = g_prof_n[kind];
  return 0;
}
extern "C" long long b2_launch_count(void) { return g_launches; }

extern "C" int b2_launch_filter(const FilterArgs* a, b2_stream_t s) {
  const bool bit = a->mode >= FILT_BITSHUFFLE;
  const bool inverse = a->mode == FILT_UNSHUFFLE || a->mode == FILT_BITUNSHUFFLE;
  const long long nblocks = (a->nbytes + a->blocksize - 1) / a->blocksize;
  const long long ipb = (a->blocksize / a->typesize + FILT_TILE - 1) / FILT_TILE + 1;
  long long ctas = (nblocks * ipb + FILT_WARPS - 1) / FILT_WARPS;
  /* one kernel instantiation per common typesize; the grid is exactly what is resident (a grid-stride loop with a
   * partial second wave ends with most SMs idle) */
  void (*kern)(FilterArgs) = a->typesize == 2 ? filter_kernel<2> : a->typesize == 4 ? filter_kernel<4> : a->typesize == 8 ? filter_kernel<8> : filter_kernel<0>;
  const size_t smem = bit ? FILT_WARPS * 16 * FILT_TILE : 0;
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, FILT_WARPS * 32, smem) != cudaSuccess || per_sm < 1) { cudaGetLastError(); per_sm = 4; }
  const long long cap = (long long)num_sms() * per_sm;
  if (ctas > cap) ctas = cap;
  if (ctas < 1) ctas = 1;
  ProfScope ps(inverse ? B2_K_UNFILTER : B2_K_FILTER, s->s);
  kern<<<(unsigned)ctas, FILT_WARPS * 32, smem, s->s>>>(*a);
  CK(cudaGetLastError());
  return 0;
}

/* LZ4 with the plain 16 KiB table can run in team mode (one CTA of four warps per stream).  It shortens the
 * critical path of a hard stream but keeps fewer streams in flight, so it pays when most streams of a block are
 * cheap and one is hard -- measured on the bench.c planes: +20 % at typesize 4 (one hard byte-plane of four),
 * -50 % at typesize 2 (both planes hard), -25 % at typesize 8 / 16.  Default: blocks of four splits when the
 * chunk has the device to itself (a frame keeps several chunks in flight: streams per SM win there);
 * BLOSC_B200_LZ4_TEAM=0 / 1 forces it off / on. */
static int team_wanted(const EncodeArgs* a) {
  static int env = -2;
  if (env == -2) { const char* e = getenv("BLOSC_B200_LZ4_TEAM"); env = (e && *e) ? (atoi(e) != 0) : -1; }
  if (a->codec != B2_CODEC_LZ4 || a->table_bytes != LZ4_TABLE_BYTES) return 0;
  return env >= 0 ? env : (a->map.nsplits == 4 && !a->many);
}

extern "C" int b2_launch_encode(const EncodeArgs* a, b2_stream_t s) {
  if (team_wanted(a)) {
    int ctas = a->map.nstreams;
    const int cap = num_sms() * TEAM_CTAS_PER_SM;
    if (ctas > cap) ctas = cap;
    if (ctas <= 0) return 0;
    ProfScope ps(B2_K_ENCODE, s->s);
    EncodeArgs args = *a;
    args.num_sms = num_sms();
    args.queue_base = *a->queue_base_host;
    *a->queue_base_host += (unsigned)a->map.nstreams + (unsigned)ctas;      /* one ticket-drawing warp per CTA */
    encode_team_kernel<<<ctas, TEAM_WARPS * 32, TEAM_SMEM_BYTES, s->s>>>(args);
    CK(cudaGetLastError());
    return 0;
  }
  int wpc = 65536 / a->table_bytes;           /* 64 KiB of tables per CTA -> 3 CTAs per SM */
  if (wpc > 4) wpc = 4;
  if (wpc < 1) wpc = 1;
  const int ctas = (a->map.nstreams + wpc - 1) / wpc;
  if (ctas <= 0) return 0;
  ProfScope ps(B2_K_ENCODE, s->s);
  EncodeArgs args = *a;
  args.queue_base = *a->queue_base_host;
  *a->queue_base_host += (unsigned)a->map.nstreams + (unsigned)ctas * (unsigned)wpc;
  encode_kernel<<<ctas, wpc * 32, (size_t)wpc * a->table_bytes, s->s>>>(args);
  CK(cudaGetLastError());
  return 0;
}

/* segment-parallel LZ4: the hash-chain index of every stream, then one lane per segment */
extern "C" int b2_launch_fast(const FastArgs* a, b2_stream_t s) {
  if (a->map.nstreams <= 0) return 0;
  {
    int ctas = (a->map.nstreams + INDEX_WARPS - 1) / INDEX_WARPS;
    ProfScope ps(B2_K_INDEX, s->s);
    index_kernel<<<ctas, INDEX_WARPS * 32, INDEX_WARPS * FAST_TAB_BYTES, s->s>>>(*a);
    CK(cudaGetLastError());
  }
  {
    const long long njobs = (long long)a->map.nfull * a->map.nsplits * a->groups_full + a->groups_left;
    const int threads = a->threads;
    const size_t smem = (size_t)a->win_bytes + 64;
    int per_sm = (int)((size_t)220 * 1024 / (smem + 1024));
    if (per_sm * threads > 2048) per_sm = 2048 / threads;
    if (per_sm < 1) per_sm = 1;
    long long ctas = njobs;
    const long long cap = (long long)num_sms() * per_sm;
    if (ctas > cap) ctas = cap;
    ProfScope ps(B2_K_PARSE, s->s);
    FastArgs args = *a;
    args.queue_base = *a->queue_base_host;
    *a->queue_base_host += (unsigned)njobs + (unsigned)ctas;      /* one ticket-drawing thread per CTA */
    parse_kernel<<<(unsigned)ctas, threads, smem, s->s>>>(args);
    CK(cudaGetLastError());
  }
  {
    const int ctas = (a->map.nstreams + FSCAN_WARPS - 1) / FSCAN_WARPS;
    ProfScope ps(B2_K_SCAN, s->s);
    fscan_kernel<<<ctas, FSCAN_WARPS * 32, 0, s->s>>>(*a);
    CK(cudaGetLastError());
  }
  return 0;
}

extern "C" int b2_launch_scan(const ScanArgs* a, b2_stream_t s) {
  ProfScope ps(B2_K_SCAN, s->s);
  scan_kernel<<<1, SCAN_THREADS, 0, s->s>>>(*a);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int b2_launch_compact(const CompactArgs* a, b2_stream_t s) {
  int ctas = a->nblocks;
  if (ctas > num_sms() * 8) ctas = num_sms() * 8;
  if (ctas <= 0) return 0;
  ProfScope ps(B2_K_COMPACT, s->s);
  compact_kernel<<<ctas, COMPACT_THREADS, 0, s->s>>>(*a);
  CK(cudaGetLastError());
  return 0;
}

/* LZ4 streams can be decoded by a parser / copier pair of warps per stream (dev_lz4dec.cuh).  Like the encoder's
 * team mode it shortens the critical path of a hard stream and costs throughput where every stream is hard (a
 * descriptor per sequence on the general path): measured on the bench.c planes 0.75 -> 0.53 ms at typesize 4
 * (fast-parse chunks 0.86 -> 0.56, lz4hc 2.03 -> 1.21), but 1.04 -> 1.22 ms at typesize 2 and 0.95 -> 1.07 at typesize 8.
 * Default: blocks of four splits when the call has the device to itself; BLOSC_B200_LZ4D_PAIR=0 / 1 forces it. */
static int pair_wanted(const DecodeArgs* a) {
  static int env = -2;
  if (env == -2) { const char* e = getenv("BLOSC_B200_LZ4D_PAIR"); env = (e && *e) ? (atoi(e) != 0) : -1; }
  if (a->codec != B2_CODEC_LZ4) return 0;
  return env >= 0 ? env : (a->map.nsplits == 4 && !a->many);
}

extern "C" int b2_launch_decode(const DecodeArgs* a, b2_stream_t s) {
  if (pair_wanted(a)) {
    int ctas = a->map.nstreams;
    const int cap = num_sms() * PAIR_CTAS_PER_SM;
    if (ctas > cap) ctas = cap;
    if (ctas <= 0) return 0;
    ProfScope ps(B2_K_DECODE, s->s);
    DecodeArgs args = *a;
    args.queue_base = *a->queue_base_host;
    *a->queue_base_host += (unsigned)a->map.nstreams + (unsigned)ctas;      /* one ticket-drawing warp per CTA */
    decode_pair_kernel<<<ctas, 64, LZ4P_SMEM, s->s>>>(args);
    CK(cudaGetLastError());
    return 0;
  }
  const int wpc = DECODE_WARPS;
  const int ctas = (a->map.nstreams + wpc - 1) / wpc;
  if (ctas <= 0) return 0;
  ProfScope ps(B2_K_DECODE, s->s);
  const size_t sm = (size_t)wpc * LZ4D_SMEM;
  DecodeArgs args = *a;
  args.queue_base = *a->queue_base_host;
  *a->queue_base_host += (unsigned)a->map.nstreams + (unsigned)ctas * (unsigned)wpc;
  if (a->codec == B2_CODEC_LZ4) decode_kernel<B2_CODEC_LZ4><<<ctas, wpc * 32, sm, s->s>>>(args);
  else if (a->codec == B2_CODEC_ZLIB) decode_kernel<B2_CODEC_ZLIB><<<ctas, wpc * 32, sm, s->s>>>(args);
  else if (a->codec == B2_CODEC_ZSTD) decode_kernel<B2_CODEC_ZSTD><<<ctas, wpc * 32, sm, s->s>>>(args);
  else decode_kernel<B2_CODEC_BLOSCLZ><<<ctas, wpc * 32, sm, s->s>>>(args);
  CK(cudaGetLastError());
  return 0;
}
