// bathgpu.cu -- C-ABI layer of libbathgpu.so (see include/bathgpu.h).
// Context, device memory, profile images, block upload/packing, stage launchers.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <math.h>
#include <thread>
#include <vector>
#include <string>
#include <algorithm>
#include <mutex>
#include <memory>

#include "../../include/bathgpu.h"
#include "fs_parser.cuh"
#include "fs_parser_v3.cuh"
#include "fs_backward.cuh"
#include "fs_domain.cuh"
#include "orf_domain.cuh"
#include "orf_filters.cuh"
#include "orf_finder.cuh"
#include "bias_filter.cuh"
#include "microbench.cuh"
#include "launch.h"
#include <chrono>

using namespace bathgpu;

namespace {

// Device memory comes from the device's stream-ordered pool (cudaMallocAsync): a buffer that has to grow hands its old block back to
// the pool and takes a larger one without the device-wide synchronisation of cudaFree / cudaMalloc -- with several contexts per GPU
// those stalled every context's stage calls whenever one of them outgrew a workspace (3 s of 1.2 s x 8 contexts on the config-4 search
// leg, profiles/r02d_search_alloc_trace.md).  The pool keeps what is freed (release threshold = no limit, set in bathgpu_create),
// so the blocks a context lets go are what the next one's growth is served from.
static thread_local cudaStream_t tl_alloc_stream = nullptr;      // the stream of the context the calling thread is working for
struct DevBuf {
  void  *p = nullptr;
  size_t cap = 0;
  DevBuf() = default;
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  ~DevBuf() { release(); }          // bathgpu_destroy selects the context's device before the context goes away
  int reserve(size_t bytes) { return bytes <= cap ? BATHGPU_OK : reserve_exact(bytes + bytes / 2 + 256); }
  int reserve_exact(size_t bytes) {
    if (bytes <= cap) return BATHGPU_OK;
    static const bool trace = getenv("BATHGPU_TRACE") != nullptr;      // tuning aid: slow (re)allocations on stderr
    const auto t0 = std::chrono::steady_clock::now();
    const size_t old = cap;
    cudaStream_t st = tl_alloc_stream;
    if (p) cudaFreeAsync(p, st);
    p = nullptr; cap = 0;
    const size_t want = (bytes + 511) & ~(size_t)511;
    if (cudaMallocAsync(&p, want, st) != cudaSuccess) { cudaGetLastError(); p = nullptr; return BATHGPU_EMEM; }
    // the block is used from the context's other streams as well (chunked uploads): make the allocation complete before anyone sees it
    if (cudaStreamSynchronize(st) != cudaSuccess) { cudaGetLastError(); return BATHGPU_EMEM; }
    cap = want;
    if (trace) {
      const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      if (ms >= 1.0) fprintf(stderr, "[bathgpu] device buffer %zu -> %zu bytes: %.2f ms\n", old, want, ms);
    }
    return BATHGPU_OK;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct FsProfileImage {
  int   which = 0, M = 0, nrows = 0, J = 0, mpad = 0, scan_steps = 5;
  DevBuf emis;     // [nrows][mpad]
  DevBuf emis_bck, cellb3;   // the 3-codon Backward parser's table copy and constants (fs_backward.cuh, Bck3Consts)
  DevBuf cellbmw;  // the same for the multi-warp Backward kernel (fs_backward_mw.cuh)
  DevBuf emis_fwd; // [nrows][mpad] the Forward parsers' copy: match->match odds folded in as well (fs_parser.cuh, FwdConsts)
  DevBuf cellc;    // forward lane constants
  DevBuf cellmw;   // the same for the multi-warp Forward kernel (J >= 16: 8 nodes per lane, J/8 warps per window)
  int    mw_scan_steps = 5;
  DevBuf cellb;    // backward lane constants
  DevBuf cellf5;   // 5-codon full-matrix Forward lane constants (fs_domain.cuh)
  DevBuf amino;    // [20][mpad] amino-acid odds, unfolded, permuted (null2)
  DevBuf oaflags;  // [mpad] transition-allowed bits per node (optimal accuracy masks)
  DevBuf oapass;   // [5][32] D pass-through flags of the optimal-accuracy scan
  DevBuf tfvraw;   // [8][M+1] transition odds as given (traceback)
  DevBuf zinv;     // [mpad] 1/Z(k) by node, k-1 (un-folds the stored match cells when a Forward matrix is handed out)
  bool  loaded = false;
};

// bathgpu_load_fs_profile_set: n profile images of one codon length in one device block, beside the context's own profile
struct FsProfileSet {
  int n = 0;
  std::vector<int> J, scan_steps, mw_scan_steps;     // per profile: what picks the kernel (bathgpu_fs_set_scores groups by it)
  std::vector<FsSetProfile> table;                   // device pointers into arena; tEM / tEL are set per call
  DevBuf arena, dtable, dwins, dwprof, dsc, dst, dcounter;
};

}  // namespace

struct TargetSlot {          // one resident target: packed DNA + codon classes + survivor residues (e.g. one strand of one chunk of the target)
  DevBuf  dna_bytes, dna4, residues, cls;
  int64_t block_n = 0, nres = 0;
  bool    bytes_valid = false;      // dna_bytes holds the block (a host-packed upload fills dna4 only; the byte form is made when something asks for it)
};
constexpr int kMaxSlots = 1 << 16;

struct bathgpu_ctx {
  int           device = 0;
  cudaDeviceProp prop{};
  cudaStream_t  stream = nullptr, copy_stream = nullptr, stream2 = nullptr;
  cudaStream_t  bulk_stream = nullptr;                // low priority: the throughput-bound translation + MSV pass (see BulkScope)
  cudaEvent_t   chunk_ev[16] = {};
  cudaEvent_t   ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t   sync_ev = nullptr;                    // blocking-sync event: a host thread waiting for its stream sleeps instead of spinning
  std::string   err;
  FsProfileImage fs3, fs5;
  FsProfileSet  set3, set5;
  std::vector<std::unique_ptr<TargetSlot>> slot;      // grows on demand (bathgpu_select_slot)
  int           cur = 0;
  TargetSlot   &S() { return *slot[cur]; }
  TargetSlot   &slot_at(int i) { while ((int)slot.size() <= i) slot.emplace_back(new TargetSlot()); return *slot[i]; }
  DevBuf        wins, fwdsc, status, counter;
  int           nstaged = 0;
  DevBuf        scratch;
  DevBuf        fxmx, bxmx, lsf, lsb, xoff, dmocc, dbtot, detot, bcksc;
  int64_t       xrows = 0;          // rows held in fxmx/bxmx by the last bck_decode chunk
  // ORF-stage filters
  bool          flt_loaded = false;
  bathgpu_filter_params flt{};
  int           flt_W = 0, flt_P = 0;
  DevBuf        f_rbv, f_rwv, f_twv, f_ddsum, f_nrb, orfs, fsc, fst, fwins, fnw;
  DevBuf        b_items, b_tables, b_out;      // bias filter
  DevBuf        o_tiles, o_cnt, o_base, o_blocks, o_first, o_tjb, o_null, o_meta, o_hits, o_counters;
  long long     o_nhits = 0, o_nres = 0;
  cudaEvent_t   o_ev[6] = {};                      // boundaries of the kernel groups of the last bathgpu_orfs_msv_screen call
  float         o_ms[5] = {};                      // classes, count pass, emit pass, MSV, screen
  long long     o_scored = 0, o_norf = 0;          // residues and ORFs the MSV kernel scored
  // domain stage workspace (last chunk stays resident for bathgpu_fs_fetch_domain_matrices)
  DevBuf        envs, dpp, doa, dfx, dppx, doax, dlsf, dfw, dbk, doasc, dnull2, dstat, dtoff, dtlen, dsteps, ddcell, dmxout;
  std::vector<long long> dom_xoff;
  std::vector<int>       dom_L;
  float         last_ms = 0.f;
  int           last_launches = 0;
};

static int fail(bathgpu_ctx *ctx, int code, const char *fmt, ...)
{
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

#define CUDA_TRY(ctx, call)                                                                      \
  do { cudaError_t e_ = (call);                                                                  \
       if (e_ != cudaSuccess) { cudaGetLastError();                                              \
         return fail(ctx, BATHGPU_ECUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); } } while (0)

// every stage call starts here: the context's device becomes current and its stream the one device buffers are (re)allocated on
static cudaError_t enter(bathgpu_ctx *ctx)
{
  tl_alloc_stream = ctx->stream;
  return cudaSetDevice(ctx->device);
}

// The per-envelope matrices (posterior / optimal-accuracy cells of fs_domain.cuh and orf_domain.cuh, the Forward matrix of the
// multi-domain branch) are the context's one large workspace.  It is taken at its full budget the first time it is needed and the
// stage calls cut their batches to fit it, so it never has to grow in the middle of a search whatever the profile length
// (growing a 0.4 GB block to 0.8 GB costs ~0.1 s of driver time; 30 of those fell into the third profile of the config-4 search).
// BATHGPU_MATRIX_MB overrides the budget (default 2048).
static size_t matrix_budget()
{
  static const size_t b = [] { const char *e = getenv("BATHGPU_MATRIX_MB"); const long long v = e ? atoll(e) : 0; return (size_t)(v > 0 ? v : 2048) << 20; }();
  return b;
}
static int reserve_matrices(bathgpu_ctx *ctx, size_t pp_bytes, size_t oa_bytes)
{
  const size_t b = matrix_budget();
  if (ctx->dpp.reserve_exact(std::max(pp_bytes, b / 10 * 7 + (1u << 20))) != BATHGPU_OK) return BATHGPU_EMEM;
  if (oa_bytes && ctx->doa.reserve_exact(std::max(oa_bytes, b / 10 * 3 + (1u << 20))) != BATHGPU_OK) return BATHGPU_EMEM;
  return BATHGPU_OK;
}

// A stage call ends by waiting for its stream.  cudaStreamSynchronize spins on a core, and a search drives 12-24 contexts, one host
// thread each, beside a host pool as wide as the machine.  BATHGPU_BLOCKING_SYNC=1 makes the waiting threads sleep on a blocking-sync
// event, =2 polls and yields the core in between.  Measured on a 16-core B200 box (3 profiles x 1 Gbp): sleeping 4.19-4.38 Gbp/s against
// 4.42-4.66 spinning, and the one-call Forward path from host buffers 15.8 against 15.2 ms; poll + yield equal to spinning within the
// run-to-run spread (4.45-4.62).  With sleeping waits the search uses 5.1 core-seconds in 0.66 s: the host is half idle, so the waits are
// not what limits it, and spinning stays the default.
static const int g_sync_mode = [] { const char *e = getenv("BATHGPU_BLOCKING_SYNC"); return e ? atoi(e) : 0; }();   // 0 spin, 1 sleep, 2 poll + yield
static inline cudaError_t wait_stream(bathgpu_ctx *ctx)
{
  if (g_sync_mode == 2) {                                    // give the core to a runnable pool worker between polls
    for (;;) {
      const cudaError_t q = cudaStreamQuery(ctx->stream);
      if (q != cudaErrorNotReady) return q;
      std::this_thread::yield();
    }
  }
  if (g_sync_mode != 1 || !ctx->sync_ev) return cudaStreamSynchronize(ctx->stream);
  const cudaError_t e = cudaEventRecord(ctx->sync_ev, ctx->stream);
  return e != cudaSuccess ? e : cudaEventSynchronize(ctx->sync_ev);
}

// For the length of a call, the context's work goes to its low-priority stream (every entry point starts and ends with the
// context's streams idle, so nothing has to be ordered between the two).
struct BulkScope {
  bathgpu_ctx *ctx; cudaStream_t saved;
  explicit BulkScope(bathgpu_ctx *c) : ctx(c), saved(c->stream) { if (c->bulk_stream) c->stream = c->bulk_stream; }
  ~BulkScope() { ctx->stream = saved; }
};

// ---------------------------------------------------------------------------------------------
extern "C" int bathgpu_create(int device, bathgpu_ctx **ret_ctx)
{
  if (!ret_ctx) return BATHGPU_EINVAL;
  *ret_ctx = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return BATHGPU_ENODEVICE; }
  if (device < 0 || device >= ndev) return BATHGPU_EINVAL;
  bathgpu_ctx *ctx = new bathgpu_ctx();
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaGetDeviceProperties(&ctx->prop, device) != cudaSuccess) {
    cudaGetLastError(); delete ctx; return BATHGPU_ENODEVICE;
  }
  if (ctx->prop.major < 10) { delete ctx; return BATHGPU_ENODEVICE; }   // sm_100a code only
  // Several contexts share a device (a search drives 12-24).  Most stage calls are chains of small latency-bound kernels; the
  // translation + MSV pass fills the device for milliseconds.  The context's own stream gets the highest priority and that pass a
  // lowest-priority one, so another context's small kernels are placed as blocks drain instead of queueing behind the pass
  // (BATHGPU_PRIORITIES=0: one priority).  Measured: no difference beyond the run-to-run spread on one B200 (4.37-4.59 against
  // 4.08-4.69 Gbp/s); kept because it costs nothing and bounds the worst case.
  int prio_lo = 0, prio_hi = 0;
  {
    const char *e = getenv("BATHGPU_PRIORITIES");
    if (!(e && atoi(e) == 0) && cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi) != cudaSuccess) { cudaGetLastError(); prio_lo = prio_hi = 0; }
  }
  if (cudaStreamCreateWithPriority(&ctx->stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
      (prio_lo != prio_hi && cudaStreamCreateWithPriority(&ctx->bulk_stream, cudaStreamNonBlocking, prio_lo) != cudaSuccess) ||
      cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
      cudaEventCreateWithFlags(&ctx->sync_ev, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess) {
    cudaGetLastError(); delete ctx; return BATHGPU_ECUDA;
  }
  {                                // the pool never hands memory back to the driver on its own: what one stage frees the next one reuses
    cudaMemPool_t pool;
    unsigned long long keep = ~0ULL;
    if (cudaDeviceGetDefaultMemPool(&pool, device) != cudaSuccess || cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep) != cudaSuccess) {
      cudaGetLastError(); bathgpu_destroy(ctx); return BATHGPU_ECUDA;
    }
  }
  tl_alloc_stream = ctx->stream;
  ctx->slot_at(1);                 // slots 0 and 1 exist from the start
  *ret_ctx = ctx;
  return BATHGPU_OK;
}

extern "C" void bathgpu_destroy(bathgpu_ctx *ctx)
{
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  // every device buffer of the context (profile images, target slots, stage workspaces) is a DevBuf and frees itself with the context
  cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
  if (ctx->sync_ev) cudaEventDestroy(ctx->sync_ev);
  for (auto &e : ctx->o_ev) if (e) cudaEventDestroy(e);
  if (ctx->bulk_stream) cudaStreamDestroy(ctx->bulk_stream);
  cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) { cudaStreamDestroy(ctx->copy_stream); cudaStreamDestroy(ctx->stream2); for (auto &e : ctx->chunk_ev) if (e) cudaEventDestroy(e); }
  delete ctx;
}

extern "C" const char *bathgpu_last_error(const bathgpu_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }

extern "C" int bathgpu_device_info(const bathgpu_ctx *ctx, int *sm_count, int *clock_khz, size_t *total_mem)
{
  if (!ctx) return BATHGPU_EINVAL;
  if (sm_count)  *sm_count  = ctx->prop.multiProcessorCount;
  if (clock_khz) { int khz = 0; cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device); *clock_khz = khz; }
  if (total_mem) *total_mem = ctx->prop.totalGlobalMem;
  return BATHGPU_OK;
}

extern "C" int bathgpu_last_stage_timing(const bathgpu_ctx *ctx, float *ms, int *launches)
{
  if (!ctx) return BATHGPU_EINVAL;
  if (ms) *ms = ctx->last_ms;
  if (launches) *launches = ctx->last_launches;
  return BATHGPU_OK;
}

// Page-locking memory costs about a millisecond per megabyte, so freed buffers are kept (up to 8 GiB in all) and handed out again.
namespace {
struct PinnedCache {
  std::mutex mu;
  std::vector<std::pair<void *, size_t>> idle;      // free buffers
  std::vector<std::pair<void *, size_t>> live;      // handed out: their sizes
  size_t idle_bytes = 0;
  ~PinnedCache() { for (auto &b : idle) cudaFreeHost(b.first); }
};
PinnedCache g_pinned;
}

extern "C" void *bathgpu_host_alloc(size_t bytes)
{
  // sizes are rounded up to a power of two (64 KiB at least), so that a buffer given back is the size the next request asks for:
  // page-locking blocks every other thread's CUDA calls while it runs, and a search whose staging buffers missed the cache by a few
  // bytes stalled all its device contexts for 30-100 ms at a time
  size_t want = (size_t)64 << 10;
  while (want < bytes) want <<= 1;
  bytes = want;
  std::lock_guard<std::mutex> lock(g_pinned.mu);
  int best = -1;
  for (int i = 0; i < (int)g_pinned.idle.size(); ++i)
    if (g_pinned.idle[i].second >= bytes && (best < 0 || g_pinned.idle[i].second < g_pinned.idle[best].second)) best = i;
  if (best >= 0 && g_pinned.idle[best].second <= 4 * bytes) {
    auto b = g_pinned.idle[best];
    g_pinned.idle.erase(g_pinned.idle.begin() + best);
    g_pinned.idle_bytes -= b.second;
    g_pinned.live.push_back(b);
    return b.first;
  }
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  g_pinned.live.push_back({ p, bytes });
  return p;
}

extern "C" void bathgpu_host_free(void *p)
{
  if (!p) return;
  std::lock_guard<std::mutex> lock(g_pinned.mu);
  for (size_t i = 0; i < g_pinned.live.size(); ++i)
    if (g_pinned.live[i].first == p) {
      auto b = g_pinned.live[i];
      g_pinned.live.erase(g_pinned.live.begin() + i);
      if (g_pinned.idle_bytes + b.second <= ((size_t)8 << 30)) { g_pinned.idle.push_back(b); g_pinned.idle_bytes += b.second; }
      else cudaFreeHost(p);
      return;
    }
  cudaFreeHost(p);
}

// 16-bit lane operations per second (add and max each counted, two halves per register) the device sustains: bench.py's denominator
// for the MSV and Viterbi filters
extern "C" int bathgpu_measure_int16_peak(bathgpu_ctx *ctx, double *tera_ops)
{
  if (!ctx || !tera_ops) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_measure_int16_peak");
  CUDA_TRY(ctx, enter(ctx));
  if (ctx->scratch.reserve(1 << 20) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  const int blocks = ctx->prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  const double ops = (double)blocks * threads * (double)iters * 8.0 * 16.0 * 4.0;
  float best = 1e30f;
  for (int rep = 0; rep < 6; ++rep) {
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    int16x2_probe_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->scratch.as<unsigned>(), iters, 0x00030001u, 0x00050002u);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
    float ms = 0.f;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (rep >= 2 && ms < best) best = ms;
  }
  *tera_ops = ops / (best * 1e-3) / 1e12;
  return BATHGPU_OK;
}

extern "C" int bathgpu_measure_fp32_peak(bathgpu_ctx *ctx, double *tflops, double *sm_mhz_effective)
{
  if (!ctx || !tflops) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_measure_fp32_peak");
  CUDA_TRY(ctx, enter(ctx));
  if (ctx->scratch.reserve(1 << 20) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  const int blocks = ctx->prop.multiProcessorCount * 8, threads = 256, iters = 4096;
  const double flop = (double)blocks * threads * (double)iters * 8.0 * 16.0 * 2.0;
  float best = 1e30f;
  for (int rep = 0; rep < 6; ++rep) {     // first reps warm the clocks up
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    fp32_fma_probe_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->scratch.as<float>(), iters, 0.999f, 1e-3f);
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
    float ms = 0.f;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    if (rep >= 2 && ms < best) best = ms;
  }
  *tflops = flop / (best * 1e-3) / 1e12;
  if (sm_mhz_effective)   // clock at which 128 lanes x 2 flop x SMs would give this rate
    *sm_mhz_effective = *tflops * 1e12 / (2.0 * 128.0 * ctx->prop.multiProcessorCount) / 1e6;
  return BATHGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// profile images
static const int kSupportedJ[] = { 1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 16, 24, 32 };   // 16, 24, 32: part of the state spills (launch.h)

static int choose_J(int M)
{
  static const int bump = [] { const char *e = getenv("BATHGPU_J_BUMP"); return e ? atoi(e) : 0; }();   // tuning: odd node counts rounded up to even
  for (int J : kSupportedJ) if (32 * J >= M) return (bump && J >= 3 && J <= 7 && (J & 1)) ? J + 1 : J;
  return 0;
}

static inline int perm_index(int kk, int J)   // position of node k=kk+1 inside a table row
{
  const int VEC = (J % 4 == 0) ? 4 : ((J % 2 == 0) ? 2 : 1);
  int lane = kk / J, j = kk % J;
  return (j / VEC) * (32 * VEC) + lane * VEC + (j % VEC);
}

namespace {
enum { tBM = 0, tMM, tIM, tDM, tMD, tMI, tII, tDD };

// What every device image of a profile is folded with (all in double, rounded once):
//   s(k) = tBM(k-1): entry odds of node k.  The kernels carry V(k)/s(k), so s(k) must be positive
//          (true for every local-mode profile: occ(k) > 0, src/modelconfig.c:90-97).
//   Z(k) = 1 + tMD(k) * sum_{k'>k} prod_{m=k+1}^{k'-1} tDD(m): E(i) = sum_k M(i,k) Z(k).
struct Fold {
  int M = 0, J = 0, mpad = 0, ld = 0;
  const float *tfv = nullptr;
  std::vector<double> sK, zK;
  // per-node transition odds, source-node indexed; zero beyond M
  double T(int t, int k) const { return (k >= 0 && k <= M) ? (double)tfv[(size_t)t * ld + k] : 0.0; }
};
}  // namespace

// The argument checks of bathgpu_load_fs_profile and the folding constants of one profile.  f.J is set once the arguments passed.
static int fold_profile(bathgpu_ctx *ctx, int which, int M, int nrows, const float *rfv, const float *tfv, Fold &f)
{
  if (!ctx || !rfv || !tfv || M < 1) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_load_fs_profile");
  if (which != 3 && which != 5)     return fail(ctx, BATHGPU_EINVAL, "codon_lengths must be 3 or 5");
  const int want_rows = (which == 3 ? 338 : 1367) + BATHGPU_KP;
  if (nrows != want_rows)           return fail(ctx, BATHGPU_EINVAL, "nrows %d != %d for %d codon lengths", nrows, want_rows, which);
  const int J = choose_J(M);
  if (J == 0) return fail(ctx, BATHGPU_EINVAL, "model length %d exceeds the single-warp kernels' limit (%d)", M, 32 * 32);
  f.M = M; f.J = J; f.mpad = 32 * J; f.ld = M + 1; f.tfv = tfv;
  const int mpad = f.mpad;
  auto T = [&](int t, int k) -> double { return f.T(t, k); };
  std::vector<double> &sK = f.sK, &zK = f.zK;
  std::vector<double> Tsum(mpad + 2, 0.0);
  sK.assign(mpad + 2, 1.0); zK.assign(mpad + 2, 0.0);
  for (int k = 1; k <= M; ++k) {
    sK[k] = T(tBM, k - 1);
    if (!(sK[k] > 0.0) || !std::isfinite(sK[k]))
      return fail(ctx, BATHGPU_EINVAL, "node %d has entry odds %g: only local-mode profiles are supported", k, sK[k]);
  }
  for (int k = M - 1; k >= 1; --k) Tsum[k] = 1.0 + T(tDD, k + 1) * Tsum[k + 1];
  for (int k = 1; k <= M; ++k) zK[k] = 1.0 + T(tMD, k) * Tsum[k];
  return BATHGPU_OK;
}

// emission table, permuted [c][J/VEC][lane][VEC], scaled by s(k) Z(k)
static void emission_table(const Fold &f, int nrows, const float *rfv, std::vector<float> &emis)
{
  const int M = f.M, J = f.J, mpad = f.mpad, ld = f.ld;
  emis.assign((size_t)nrows * mpad, 0.0f);
  for (int c = 0; c < nrows; ++c)
    for (int k = 1; k <= M; ++k)
      emis[(size_t)c * mpad + perm_index(k - 1, J)] = (float)((double)rfv[(size_t)c * ld + k] * f.sK[k] * f.zK[k]);
}

// The Forward parsers' table copy ef, lane constants cc, the multi-warp kernel's constants mw (3 codon lengths, J >= 16; else empty)
// and the D->D scan steps they need
static void forward3_tables(const Fold &f, int which, int nrows, const float *rfv, std::vector<float> &ef, std::vector<float> &cc,
                            std::vector<float> &mw, int &scan_steps, int &mw_scan_steps)
{
  const int M = f.M, J = f.J, mpad = f.mpad, ld = f.ld;
  const std::vector<double> &sK = f.sK, &zK = f.zK;
  auto T = [&](int t, int k) -> double { return f.T(t, k); };
  {
    cc.assign((size_t)(FC_COUNT * J + FL_COUNT) * 32, 0.0f);
    auto C = [&](int which_c, int j, int lane) -> float & { return cc[(size_t)(which_c * J + j) * 32 + lane]; };
    // Scaled forms of the Forward parsers (fs_parser.cuh, FwdConsts): the table copy they read carries mm(k) too, and the
    // delete and insert chains are divided by g(k) and hi(k) so that the match value enters every chain with coefficient 1.
    // Divisors that vanish take tiny stand-ins: node M has no way out (mm := 1, its flow is never read); a node no delete or
    // insert path leaves (no shipped model has one before node M) leaves a relative trace of 1e-20 or less.
    auto mmK = [&](int k) -> double {
      if (k >= M) return 1.0;
      const double v = T(tMM, k) / (zK[k] * sK[k + 1]);
      return v > 0.0 ? v : 1.0e-12;
    };
    auto mdK = [&](int k) -> double { return std::max(T(tMD, k) / (zK[k] * mmK(k)), 1.0e-20); };
    auto gK  = [&](int k) -> double { return (k >= 2 && k <= M) ? mdK(k - 1) : 1.0; };
    // node 1 has no delete state (D(i,1) = 0): its dd and dm are 0, which also cancels whatever lane 0 is handed as inflow
    auto ddS = [&](int k) -> double { return (k >= 2 && k < M) ? gK(k) * T(tDD, k) / mdK(k) : 0.0; };
    std::vector<double> bfull(32, 1.0), bscaled(32, 1.0);
    ef.assign((size_t)nrows * mpad, 0.0f);
    for (int c = 0; c < nrows; ++c)
      for (int k = 1; k <= M; ++k)
        ef[(size_t)c * mpad + perm_index(k - 1, J)] = (float)((double)rfv[(size_t)c * ld + k] * sK[k] * zK[k] * mmK(k));
    for (int lane = 0; lane < 32; ++lane) {
      double pp = 1.0, ps = 1.0;
      for (int j = 0; j < J; ++j) {
        int k = lane * J + j + 1;
        if (k <= M) {
          double sn = sK[k + 1];      // s(k+1); 1.0 at k = M where every outgoing transition is 0
          C(FC_MM, j, lane) = (float)(1.0 / mmK(k));                                                         // qm
          C(FC_DM, j, lane) = (k >= 2) ? (float)(gK(k) * T(tDM, k) / sn) : 0.0f;
          C(FC_MD, j, lane) = (float)(T(tMD, k) / zK[k]);          // not read by the kernels any more; kept for the layout
          C(FC_DD, j, lane) = (float)ddS(k);
          C(FC_MI, j, lane) = (float)std::max(T(tMI, k) * T(tIM, k) / (zK[k] * sn * mmK(k)), 1.0e-20);      // hi
          C(FC_II, j, lane) = (float)T(tII, k);
        }
        pp *= T(tDD, k);
        ps *= ddS(k);
      }
      bfull[lane] = pp; bscaled[lane] = ps;
    }
    std::vector<double> b(bfull), bs(bscaled);
    scan_steps = 5;
    for (int s = 0; s < 5; ++s) {
      int d = 1 << s;
      std::vector<double> nb(b), nbs(bs);
      double biggest = 0.0;
      for (int lane = 0; lane < 32; ++lane) {
        cc[(size_t)(FC_COUNT * J + FL_B0 + s) * 32 + lane] = (lane >= d) ? (float)bs[lane] : 0.0f;
        if (lane >= d) { biggest = std::max(biggest, b[lane]); nb[lane] = b[lane] * b[lane - d]; nbs[lane] = bs[lane] * bs[lane - d]; }
      }
      bs.swap(nbs);
      // step s carries D in from 2^s lanes away with these multipliers: below 1e-9 everywhere it (and every later step) changes
      // nothing at float resolution -- the cut-off the reference's own D->D passes apply (fwdback_fs.c:415-453)
      if (biggest < 1.0e-9 && scan_steps == 5) scan_steps = std::max(s, 2);
      b.swap(nb);
    }
    if (which == 3 && J >= 16) {
      // multi-warp Forward kernel (fs_parser_mw.cuh): JW nodes per lane, NW = J/JW warps, virtual lane v = 32 w + lane owns nodes
      // JW v + 1 .. JW v + JW
      const int JW = kMwNodesPerLane, NW = J / JW, VL = 32 * NW;
      mw.assign((size_t)(5 * JW + 6) * VL + NW, 0.0f);
      std::vector<double> lp(VL, 1.0), lpfull(VL, 1.0);
      for (int v = 0; v < VL; ++v)
        for (int j = 0; j < JW; ++j) {
          const int k = v * JW + j + 1;
          if (k <= M) {
            const double sn = sK[k + 1];
            mw[(size_t)(0 * JW + j) * VL + v] = (float)(1.0 / mmK(k));
            mw[(size_t)(1 * JW + j) * VL + v] = (k >= 2) ? (float)(gK(k) * T(tDM, k) / sn) : 0.0f;
            mw[(size_t)(2 * JW + j) * VL + v] = (float)ddS(k);
            mw[(size_t)(3 * JW + j) * VL + v] = (float)std::max(T(tMI, k) * T(tIM, k) / (zK[k] * sn * mmK(k)), 1.0e-20);
            mw[(size_t)(4 * JW + j) * VL + v] = (float)T(tII, k);
          }
          lp[v] *= ddS(k); lpfull[v] *= T(tDD, k);
        }
      mw_scan_steps = 3;
      for (int w = 0; w < NW; ++w) {
        std::vector<double> bsw(lp.begin() + 32 * w, lp.begin() + 32 * w + 32), bw(lpfull.begin() + 32 * w, lpfull.begin() + 32 * w + 32);
        double q = 1.0;
        for (int lane = 0; lane < 32; ++lane) { mw[(size_t)(5 * JW + 5) * VL + 32 * w + lane] = (float)q; q *= lp[32 * w + lane]; }
        mw[(size_t)(5 * JW + 6) * VL + w] = (float)q;                     // PW(w): the whole warp's product
        int need = 5;
        for (int s2 = 0; s2 < 5; ++s2) {
          const int d = 1 << s2;
          std::vector<double> nbs(bsw), nb(bw);
          double biggest = 0.0;
          for (int lane = 0; lane < 32; ++lane) {
            mw[(size_t)(5 * JW + s2) * VL + 32 * w + lane] = (lane >= d) ? (float)bsw[lane] : 0.0f;
            if (lane >= d) { biggest = std::max(biggest, bw[lane]); nbs[lane] = bsw[lane] * bsw[lane - d]; nb[lane] = bw[lane] * bw[lane - d]; }
          }
          bsw.swap(nbs); bw.swap(nb);
          if (biggest < 1.0e-9 && need == 5) need = std::max(s2, 3);
        }
        mw_scan_steps = std::max(mw_scan_steps, need);
      }
      if (getenv("BATHGPU_FULL_SCAN")) mw_scan_steps = 5;
    } else mw.clear();
    if (getenv("BATHGPU_FULL_SCAN")) scan_steps = 5;
  }
}

// the full-matrix 5-codon Forward lane constants (fs_domain.cuh, Fwd5Const)
static void fs5_forward_consts(const Fold &f, std::vector<float> &cc)
{
  const int M = f.M, J = f.J;
  const std::vector<double> &sK = f.sK, &zK = f.zK;
  auto T = [&](int t, int k) -> double { return f.T(t, k); };
  cc.assign((size_t)(F5_COUNT * J + 5) * 32, 0.0f);
  auto C = [&](int which_c, int j, int lane) -> float & { return cc[(size_t)(which_c * J + j) * 32 + lane]; };
  std::vector<double> bfull(32, 1.0);
  for (int lane = 0; lane < 32; ++lane) {
    double pp = 1.0;
    for (int j = 0; j < J; ++j) {
      int k = lane * J + j + 1;
      if (k <= M) {
        double sn = sK[k + 1];
        C(F5_MM, j, lane) = (float)(T(tMM, k) / (zK[k] * sn));
        C(F5_IM, j, lane) = (float)(T(tIM, k) / sn);
        C(F5_DM, j, lane) = (float)(T(tDM, k) / sn);
        C(F5_MD, j, lane) = (float)(T(tMD, k) / zK[k]);
        C(F5_DD, j, lane) = (float)T(tDD, k);
        C(F5_MI, j, lane) = (float)(T(tMI, k) / zK[k]);
        C(F5_II, j, lane) = (float)T(tII, k);
      }
      pp *= T(tDD, k);
    }
    bfull[lane] = pp;
  }
  std::vector<double> b(bfull);
  for (int s = 0; s < 5; ++s) {
    int d = 1 << s;
    std::vector<double> nb(b);
    for (int lane = 0; lane < 32; ++lane) {
      cc[(size_t)(F5_COUNT * J + s) * 32 + lane] = (lane >= d) ? (float)b[lane] : 0.0f;
      if (lane >= d) nb[lane] = b[lane] * b[lane - d];
    }
    b.swap(nb);
  }
}

extern "C" int bathgpu_load_fs_profile(bathgpu_ctx *ctx, int which, int M, int nrows, const float *rfv, const float *tfv)
{
  Fold f;
  const int fst = fold_profile(ctx, which, M, nrows, rfv, tfv, f);
  if (fst != BATHGPU_OK) {
    if (f.J) (which == 3 ? ctx->fs3 : ctx->fs5).loaded = false;      // a profile refused past the argument checks leaves no image behind
    return fst;
  }
  CUDA_TRY(ctx, enter(ctx));

  FsProfileImage &im = (which == 3) ? ctx->fs3 : ctx->fs5;
  im.loaded = false;
  const int J = f.J;
  im.which = which; im.M = M; im.nrows = nrows; im.J = J; im.mpad = f.mpad;
  const int mpad = im.mpad, ld = M + 1;
  auto T = [&](int t, int k) -> double { return f.T(t, k); };
  const std::vector<double> &sK = f.sK, &zK = f.zK;
  std::vector<float> emis;
  emission_table(f, nrows, rfv, emis);

  // ---- forward constants
  {
    std::vector<float> ef, cc, mw;
    forward3_tables(f, which, nrows, rfv, ef, cc, mw, im.scan_steps, im.mw_scan_steps);
    if (im.emis_fwd.reserve(ef.size() * sizeof(float)) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
    CUDA_TRY(ctx, cudaMemcpyAsync(im.emis_fwd.p, ef.data(), ef.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
    if (!mw.empty()) {
      if (im.cellmw.reserve(mw.size() * sizeof(float)) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
      CUDA_TRY(ctx, cudaMemcpyAsync(im.cellmw.p, mw.data(), mw.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
      CUDA_TRY(ctx, wait_stream(ctx));
    } else im.cellmw.release();
    if (im.cellc.reserve(cc.size() * sizeof(float)) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
    CUDA_TRY(ctx, cudaMemcpyAsync(im.cellc.p, cc.data(), cc.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
  }

  // ---- backward constants (fs_backward.cuh)
  {
    std::vector<float> cc((size_t)(BC_COUNT * J + BL_COUNT) * 32, 0.0f);
    auto C = [&](int which_c, int j, int lane) -> float & { return cc[(size_t)(which_c * J + j) * 32 + lane]; };
    std::vector<double> bfull(32, 1.0);
    for (int lane = 0; lane < 32; ++lane) {
      double pp = 1.0;
      for (int j = 0; j < J; ++j) {
        int k = lane * J + j + 1;
        if (k <= M) {
          double sn = sK[k + 1];      // entry odds of node k+1 (1.0 at k = M, where every transition out is 0)
          C(BC_VMM, j, lane) = (float)(T(tMM, k) / (sn * zK[k]));
          C(BC_VIM, j, lane) = (float)(T(tIM, k) / sn);
          C(BC_VDM, j, lane) = (float)(T(tDM, k) / sn);
          C(BC_DD,  j, lane) = (float)T(tDD, k);
          C(BC_MD,  j, lane) = (float)(T(tMD, k) / zK[k]);
          C(BC_MI,  j, lane) = (float)(T(tMI, k) / zK[k]);
          C(BC_II,  j, lane) = (float)T(tII, k);
        }
        pp *= T(tDD, k);
      }
      bfull[lane] = pp;
    }
    std::vector<double> b(bfull);
    for (int s = 0; s < 5; ++s) {
      int d = 1 << s;
      std::vector<double> nb(b);
      for (int lane = 0; lane < 32; ++lane) {
        cc[(size_t)(BC_COUNT * J + BL_B0 + s) * 32 + lane] = (lane + d <= 31) ? (float)b[lane] : 0.0f;
        if (lane + d <= 31) nb[lane] = b[lane] * b[lane + d];
      }
      b.swap(nb);
    }
    if (im.cellb.reserve(cc.size() * sizeof(float)) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
    CUDA_TRY(ctx, cudaMemcpyAsync(im.cellb.p, cc.data(), cc.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
  }

  // ---- the 3-codon Backward parser's scaled constants and table copy (fs_backward.cuh, Bck3Consts)
  {
    auto vmmE = [&](int k) -> double {               // match->match odds as the flow into node k+1 sees them; stand-ins where they vanish
      if (k < 1 || k >= M) return 1.0;
      const double v = T(tMM, k) / (sK[k + 1] * zK[k]);
      return v > 0.0 ? v : 1.0e-12;
    };
    auto rE = [&](int k) -> double { return (k >= 1 && k < M) ? std::max(T(tDM, k) / sK[k + 1] / vmmE(k), 1.0e-20) : 1.0; };
    auto uE = [&](int k) -> double { return (k >= 1 && k < M) ? std::max(T(tIM, k) / sK[k + 1] / vmmE(k), 1.0e-20) : 1.0; };
    auto dd3 = [&](int k) -> double { return (k >= 1 && k < M) ? rE(k + 1) * T(tDD, k) / rE(k) : 0.0; };
    std::vector<float> eb((size_t)nrows * mpad, 0.0f);
    for (int c = 0; c < nrows; ++c)
      for (int k = 1; k <= M; ++k)
        eb[(size_t)c * mpad + perm_index(k - 1, J)] = (float)((double)rfv[(size_t)c * ld + k] * sK[k] * zK[k] * vmmE(k - 1));
    std::vector<float> cc((size_t)(B3_COUNT * J + 5) * 32, 0.0f);
    auto C = [&](int which_c, int j, int lane) -> float & { return cc[(size_t)(which_c * J + j) * 32 + lane]; };
    std::vector<double> b(32, 1.0);
    for (int lane = 0; lane < 32; ++lane) {
      double pp = 1.0;
      for (int j = 0; j < J; ++j) {
        int k = lane * J + j + 1;
        if (k <= M) {
          C(B3_QB, j, lane) = (float)(1.0 / vmmE(k - 1));
          C(B3_DD, j, lane) = (float)dd3(k);
          C(B3_MD, j, lane) = (k < M) ? (float)(rE(k + 1) * T(tMD, k) / zK[k]) : 0.0f;
          C(B3_MI, j, lane) = (float)(uE(k) * T(tMI, k) / zK[k]);
          C(B3_II, j, lane) = (float)T(tII, k);
        }
        pp *= dd3(k);
      }
      b[lane] = pp;
    }
    for (int s = 0; s < 5; ++s) {
      int d = 1 << s;
      std::vector<double> nb(b);
      for (int lane = 0; lane < 32; ++lane) {
        cc[(size_t)(B3_COUNT * J + s) * 32 + lane] = (lane + d <= 31) ? (float)b[lane] : 0.0f;
        if (lane + d <= 31) nb[lane] = b[lane] * b[lane + d];
      }
      b.swap(nb);
    }
    if (which == 3 && J >= 16) {
      // multi-warp Backward kernel (fs_backward_mw.cuh): virtual lane v = 32 w + lane owns nodes JW v + 1 .. JW v + JW
      const int JW = kMwNodesPerLane, NW = J / JW, VL = 32 * NW;
      std::vector<float> mw((size_t)(5 * JW + 6) * VL + 2 * NW, 0.0f);
      std::vector<double> lp(VL, 1.0);
      for (int v = 0; v < VL; ++v)
        for (int j = 0; j < JW; ++j) {
          const int k = v * JW + j + 1;
          if (k <= M) {
            mw[(size_t)(0 * JW + j) * VL + v] = (float)(1.0 / vmmE(k - 1));
            mw[(size_t)(1 * JW + j) * VL + v] = (float)dd3(k);
            mw[(size_t)(2 * JW + j) * VL + v] = (k < M) ? (float)(rE(k + 1) * T(tMD, k) / zK[k]) : 0.0f;
            mw[(size_t)(3 * JW + j) * VL + v] = (float)(uE(k) * T(tMI, k) / zK[k]);
            mw[(size_t)(4 * JW + j) * VL + v] = (float)T(tII, k);
          }
          lp[v] *= (k <= M) ? dd3(k) : 0.0;
        }
      for (int w = 0; w < NW; ++w) {
        std::vector<double> bw(lp.begin() + 32 * w, lp.begin() + 32 * w + 32);
        for (int s2 = 0; s2 < 5; ++s2) {
          const int d = 1 << s2;
          std::vector<double> nb(bw);
          for (int lane = 0; lane < 32; ++lane) {
            mw[(size_t)(5 * JW + s2) * VL + 32 * w + lane] = (lane + d <= 31) ? (float)bw[lane] : 0.0f;
            if (lane + d <= 31) nb[lane] = bw[lane] * bw[lane + d];
          }
          bw.swap(nb);
        }
        const int k_a = 32 * w * JW + 1, k_b = 32 * (w + 1) * JW;          // first and last node of the warp
        auto ddk = [&](int k) -> double { return (k >= 1 && k <= M) ? dd3(k) : 0.0; };
        for (int lane = 0; lane < 31; ++lane) {                            // QU: from the first node of lane + 1 to the warp's last node but one
          double qq = 1.0;
          for (int k = (32 * w + lane + 1) * JW + 1; k <= k_b - 1; ++k) qq *= ddk(k);
          mw[(size_t)(5 * JW + 5) * VL + 32 * w + lane] = (float)qq;
        }
        double pw = 1.0;
        for (int k = k_a; k <= k_b - 1; ++k) pw *= ddk(k);
        mw[(size_t)(5 * JW + 6) * VL + w] = (float)pw;
        mw[(size_t)(5 * JW + 6) * VL + NW + w] = (float)ddk(k_b);
      }
      if (im.cellbmw.reserve(mw.size() * sizeof(float)) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
      CUDA_TRY(ctx, cudaMemcpyAsync(im.cellbmw.p, mw.data(), mw.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
      CUDA_TRY(ctx, wait_stream(ctx));
    } else im.cellbmw.release();
    if (im.cellb3.reserve(cc.size() * sizeof(float)) != BATHGPU_OK || im.emis_bck.reserve(eb.size() * sizeof(float)) != BATHGPU_OK)
      return fail(ctx, BATHGPU_EMEM, "device allocation failed");
    CUDA_TRY(ctx, cudaMemcpyAsync(im.cellb3.p, cc.data(), cc.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(im.emis_bck.p, eb.data(), eb.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
  }

  // ---- full-matrix Forward constants, null2 amino rows, optimal-accuracy masks, raw transitions (fs_domain.cuh)
  {
    std::vector<float> cc;
    fs5_forward_consts(f, cc);
    const int amino0 = nrows - BATHGPU_KP;
    std::vector<float> am((size_t)20 * mpad, 0.0f);
    for (int x = 0; x < 20; ++x)
      for (int k = 1; k <= M; ++k) am[(size_t)x * mpad + perm_index(k - 1, J)] = rfv[(size_t)(amino0 + x) * ld + k];
    std::vector<uint32_t> fl(mpad, 0u);
    std::vector<int> lane_pass(32, 1);
    for (int k = 1; k <= M; ++k) {
      uint32_t f = 0;
      if (T(tBM, k - 1) > 0.0) f |= OF_BM;
      if (T(tMM, k - 1) > 0.0) f |= OF_MM;
      if (T(tIM, k - 1) > 0.0) f |= OF_IM;
      if (T(tDM, k - 1) > 0.0) f |= OF_DM;
      if (T(tMD, k - 1) > 0.0) f |= OF_MD;
      if (T(tDD, k - 1) > 0.0) f |= OF_DD;
      if (T(tMI, k) > 0.0)     f |= OF_MI;
      if (T(tII, k) > 0.0)     f |= OF_II;
      fl[k - 1] = f;             // indexed by lane*J + j, NOT permuted
      if (!(f & OF_DD)) lane_pass[(k - 1) / J] = 0;
    }
    // nodes beyond M never pass anything on; they are forced to -inf in the kernel
    std::vector<float> pass((size_t)5 * 32, 0.0f);
    {
      std::vector<int> cur(lane_pass);
      for (int s = 0; s < 5; ++s) {
        int d = 1 << s;
        std::vector<int> nx(cur);
        for (int lane = 0; lane < 32; ++lane) {
          pass[(size_t)s * 32 + lane] = (lane >= d && cur[lane]) ? 1.0f : 0.0f;
          if (lane >= d) nx[lane] = cur[lane] && cur[lane - d];
        }
        cur.swap(nx);
      }
    }
    if (im.cellf5.reserve(cc.size() * 4) != BATHGPU_OK || im.amino.reserve(am.size() * 4) != BATHGPU_OK ||
        im.oaflags.reserve(fl.size() * 4) != BATHGPU_OK || im.oapass.reserve(pass.size() * 4) != BATHGPU_OK ||
        im.tfvraw.reserve((size_t)8 * ld * 4) != BATHGPU_OK || im.zinv.reserve((size_t)mpad * 4) != BATHGPU_OK)
      return fail(ctx, BATHGPU_EMEM, "device allocation failed");
    std::vector<float> zi(mpad, 0.0f);
    for (int k = 1; k <= M; ++k) zi[k - 1] = (float)(1.0 / zK[k]);
    CUDA_TRY(ctx, cudaMemcpyAsync(im.zinv.p, zi.data(), zi.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(im.cellf5.p, cc.data(), cc.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(im.amino.p, am.data(), am.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(im.oaflags.p, fl.data(), fl.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(im.oapass.p, pass.data(), pass.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(im.tfvraw.p, tfv, (size_t)8 * ld * 4, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
  }

  if (im.emis.reserve(emis.size() * sizeof(float)) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  CUDA_TRY(ctx, cudaMemcpyAsync(im.emis.p, emis.data(), emis.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  im.loaded = true;
  // CUDA loads kernels lazily: touch the ones this profile will use now, not inside the first stage call
#define X(S) preload_fwd_##S(J); preload_bck_##S(J); preload_fs5_##S(J); preload_orf_##S(J);
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return BATHGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// block upload: ESL_DSQ bytes -> 4-bit packed words, one guard word in front, 24 behind
__global__ void pack_dna4_kernel(const uint8_t *__restrict__ dsq, long long n, uint32_t *__restrict__ out, long long nwords)
{
  long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nwords) return;
  uint32_t word = 0;
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    long long p = w * 8 + b - 8;          // 0-based nt index
    uint32_t  code = 15u;
    if (p >= 0 && p < n) { code = dsq[p + 1]; if (code > 15u) code = 15u; }
    word |= code << (4 * b);
  }
  out[w] = word;
}

__global__ void pack_dna4_range_kernel(const uint8_t *__restrict__ dsq, long long n, uint32_t *__restrict__ out, long long wlo, long long whi)
{
  const long long w = wlo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= whi) return;
  uint32_t word = 0;
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const long long p = w * 8 + b - 8;
    uint32_t code = 15u;
    if (p >= 0 && p < n) { code = dsq[p + 1]; if (code > 15u) code = 15u; }
    word |= code << (4 * b);
  }
  out[w] = word;
}

extern "C" int bathgpu_select_slot(bathgpu_ctx *ctx, int slot)
{
  if (!ctx || slot < 0 || slot >= kMaxSlots) return fail(ctx, BATHGPU_EINVAL, "slot must be in 0..%d", kMaxSlots - 1);
  ctx->slot_at(slot);
  ctx->cur = slot;
  return BATHGPU_OK;
}

extern "C" int bathgpu_upload_block(bathgpu_ctx *ctx, const uint8_t *dsq, int64_t n)
{
  if (!ctx || !dsq || n < 1) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_upload_block");
  CUDA_TRY(ctx, enter(ctx));
  const long long nwords = (n + 8 + 7) / 8 + 24;     // kernels prefetch up to ~100 nt past a window
  if (ctx->S().dna_bytes.reserve((size_t)n + 2) != BATHGPU_OK || ctx->S().dna4.reserve((size_t)nwords * 4) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for a %lld-nt block", (long long)n);
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->S().dna_bytes.p, dsq, (size_t)n + 2, cudaMemcpyHostToDevice, ctx->stream));
  const int threads = 256;
  const long long blocks = (nwords + threads - 1) / threads;
  pack_dna4_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(ctx->S().dna_bytes.as<uint8_t>(), n, ctx->S().dna4.as<uint32_t>(), nwords);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, wait_stream(ctx));
  ctx->S().block_n = n; ctx->S().bytes_valid = true;
  return BATHGPU_OK;
}

extern "C" int bathgpu_upload_block_segments(bathgpu_ctx *ctx, const uint8_t *const *seg, const int64_t *seg_n, int nseg)
{
  if (!ctx || !seg || !seg_n || nseg < 1) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_upload_block_segments");
  long long n = 0;
  for (int g = 0; g < nseg; ++g) {
    if (!seg[g] || seg_n[g] < 1) return fail(ctx, BATHGPU_EINVAL, "segment %d is empty", g);
    n += seg_n[g];
  }
  CUDA_TRY(ctx, enter(ctx));
  TargetSlot &S = ctx->S();
  const long long nwords = (n + 8 + 7) / 8 + 24;
  if (S.dna_bytes.reserve((size_t)n + 2) != BATHGPU_OK || S.dna4.reserve((size_t)nwords * 4) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for a %lld-nt block", n);
  uint8_t *d = S.dna_bytes.as<uint8_t>();
  CUDA_TRY(ctx, cudaMemsetAsync(d, 255, 1, ctx->stream));
  CUDA_TRY(ctx, cudaMemsetAsync(d + n + 1, 255, 1, ctx->stream));
  long long off = 0;
  for (int g = 0; g < nseg; ++g) {
    CUDA_TRY(ctx, cudaMemcpyAsync(d + 1 + off, seg[g], (size_t)seg_n[g], cudaMemcpyHostToDevice, ctx->stream));
    off += seg_n[g];
  }
  pack_dna4_kernel<<<(unsigned)((nwords + 255) / 256), 256, 0, ctx->stream>>>(d, n, S.dna4.as<uint32_t>(), nwords);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, wait_stream(ctx));
  S.block_n = n; S.nres = 0; S.bytes_valid = true;
  return BATHGPU_OK;
}

// ---- host-packed blocks: two nucleotides per byte (nucleotide 2j+1 of dsq in the low nibble of byte j, 2j+2 in the high one, codes
// above 15 stored as 15 = N), which is the device's own packed layout from word 1 on -- the block crosses the link at half the bytes
// and needs no packing pass.
extern "C" int64_t bathgpu_packed4_bytes(int64_t n) { return n < 0 ? 0 : (n + 1) / 2; }

extern "C" int bathgpu_pack_dna4(const uint8_t *dsq, int64_t n, uint8_t *packed)
{
  if (!dsq || !packed || n < 1) return BATHGPU_EINVAL;
  const uint8_t *d = dsq + 1;
  const int64_t full = n / 2;
  for (int64_t j = 0; j < full; ++j) {
    const uint8_t lo = d[2 * j] > 15 ? 15 : d[2 * j], hi = d[2 * j + 1] > 15 ? 15 : d[2 * j + 1];
    packed[j] = (uint8_t)(lo | (hi << 4));
  }
  if (n & 1) packed[full] = (uint8_t)((d[n - 1] > 15 ? 15 : d[n - 1]) | 0xF0);
  return BATHGPU_OK;
}

// guard word in front, the nibbles behind nucleotide n and the 24 guard words behind the data
__global__ void dna4_guards_kernel(uint32_t *__restrict__ out, long long n)
{
  const long long wl = (n + 7) / 8;                       // word of the last nucleotide
  const int t = threadIdx.x;
  if (t == 0) out[0] = 0xFFFFFFFFu;
  else if (t == 1) { const int k = (int)(n - 8 * (wl - 1)); if (k < 8) out[wl] |= 0xFFFFFFFFu << (4 * k); }
  else if (t < 26) out[wl + t - 1] = 0xFFFFFFFFu;
}

// A host-packed chunk lands in device memory by DMA and is read by the Forward kernel from there; the byte path's packing kernel left
// its output in L2 instead (a 100 Mbp block is 50 MB packed, L2 holds 126 MB), and the Forward kernel's first touch of a window is
// latency-bound: 15.67 against 15.19 ms per 100 Mbp.  One prefetch per 128-byte line behind each chunk's copy puts the packed words in L2.
__global__ void l2_prefetch_kernel(const uint8_t *__restrict__ p, long long nbytes)
{
  const long long line = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (line * 128 < nbytes) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + line * 128));
}

// the byte form of a packed block (ORF finder, reverse complement read bytes): bytes[1 + p] = nibble p, sentinels at both ends
__global__ void unpack_dna4_kernel(const uint32_t *__restrict__ dna4, long long n, uint8_t *__restrict__ bytes)
{
  const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // packed word w + 1 holds nucleotides 8w .. 8w+7
  if (8 * w >= n) return;
  const uint32_t word = dna4[w + 1];
#pragma unroll
  for (int b = 0; b < 8; ++b) if (8 * w + b < n) bytes[1 + 8 * w + b] = (uint8_t)((word >> (4 * b)) & 15u);
  if (w == 0) { bytes[0] = 255; bytes[n + 1] = 255; }
}

extern "C" int bathgpu_upload_block_packed4(bathgpu_ctx *ctx, const uint8_t *packed, int64_t n)
{
  if (!ctx || !packed || n < 1) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_upload_block_packed4");
  CUDA_TRY(ctx, enter(ctx));
  const long long nwords = (n + 8 + 7) / 8 + 24;
  TargetSlot &S = ctx->S();
  if (S.dna_bytes.reserve((size_t)n + 2) != BATHGPU_OK || S.dna4.reserve((size_t)nwords * 4) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for a %lld-nt block", (long long)n);
  CUDA_TRY(ctx, cudaMemcpyAsync(S.dna4.as<uint8_t>() + 4, packed, (size_t)((n + 1) / 2), cudaMemcpyHostToDevice, ctx->stream));
  dna4_guards_kernel<<<1, 32, 0, ctx->stream>>>(S.dna4.as<uint32_t>(), n);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, wait_stream(ctx));
  S.block_n = n; S.nres = 0; S.bytes_valid = false;
  return BATHGPU_OK;
}

// dst[1 + p] = complement of src[n - p] (Easel's DNA alphabet: A C G T - R Y M K S W H B V D N * ~)
__global__ void revcomp_kernel(const uint8_t *__restrict__ src, long long n, uint8_t *__restrict__ dst)
{
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const uint8_t comp[18] = { 3, 2, 1, 0, 4, 6, 5, 8, 7, 9, 10, 14, 13, 12, 11, 15, 16, 17 };
  const uint8_t c = src[n - p];
  dst[1 + p] = (c < 18) ? comp[c] : c;
  if (p == 0) { dst[0] = 255; dst[n + 1] = 255; }
}

// The reverse complement of the sequence resident in slot src becomes the resident sequence of slot dst, without a second
// trip over the host link (bathsearch reverse-complements each block on the host, src/bathsearch.c:1087-1096).
extern "C" int bathgpu_revcomp_slot(bathgpu_ctx *ctx, int src, int dst)
{
  if (!ctx || src < 0 || src >= kMaxSlots || dst < 0 || dst >= kMaxSlots || src == dst) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_revcomp_slot");
  ctx->slot_at(std::max(src, dst));
  TargetSlot &A = *ctx->slot[src], &B = *ctx->slot[dst];
  if (A.block_n == 0) return fail(ctx, BATHGPU_EINVAL, "no block uploaded in slot %d", src);
  CUDA_TRY(ctx, enter(ctx));
  const long long n = A.block_n;
  const long long nwords = (n + 8 + 7) / 8 + 24;
  if (B.dna_bytes.reserve((size_t)n + 2) != BATHGPU_OK || B.dna4.reserve((size_t)nwords * 4) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for a %lld-nt block", n);
  if (!A.bytes_valid) {                                     // host-packed upload: the byte form is made now
    unpack_dna4_kernel<<<(unsigned)(((n + 7) / 8 + 255) / 256), 256, 0, ctx->stream>>>(A.dna4.as<uint32_t>(), n, A.dna_bytes.as<uint8_t>());
    A.bytes_valid = true;
  }
  revcomp_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(A.dna_bytes.as<uint8_t>(), n, B.dna_bytes.as<uint8_t>());
  pack_dna4_kernel<<<(unsigned)((nwords + 255) / 256), 256, 0, ctx->stream>>>(B.dna_bytes.as<uint8_t>(), n, B.dna4.as<uint32_t>(), nwords);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, wait_stream(ctx));
  B.block_n = n; B.nres = 0; B.bytes_valid = true;
  return BATHGPU_OK;
}


static cudaError_t dispatch_fwd(bool xmx, int J, const FsParserArgs &a, int sms, cudaStream_t s);

// Upload a block and score its windows in one call, with the upload hidden behind the kernel: the block crosses the link in
// chunks on a second stream, and the windows that end inside the part already resident are scored while the rest is in flight
// (per block the reference uploads nothing and calls p7_ForwardParser_Frameshift_3Codons window by window, src/p7_pipeline.c:1450).
static int fs_fwd_block_impl(bathgpu_ctx *ctx, const uint8_t *dsq, const uint8_t *packed, int64_t n, const bathgpu_window *wins, int nwin,
                             const float xfE[2], float *fwdsc, int32_t *status)
{
  if (!ctx || (!dsq && !packed) || n < 1 || !wins || nwin < 1 || !xfE || !fwdsc || !status) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_fwd_block");
  if (!ctx->fs3.loaded) return fail(ctx, BATHGPU_EINVAL, "3-codon profile not loaded");
  for (int w = 0; w < nwin; ++w)
    if (wins[w].L < 3 || wins[w].start < 1 || wins[w].start + wins[w].L - 1 > n)
      return fail(ctx, BATHGPU_EINVAL, "window %d (start %lld, L %d) is outside the block (n=%lld) or shorter than 3", w, (long long)wins[w].start, wins[w].L, (long long)n);
  CUDA_TRY(ctx, enter(ctx));
  if (!ctx->copy_stream) {
    CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    CUDA_TRY(ctx, cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
    for (auto &e : ctx->chunk_ev) CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  TargetSlot &S = ctx->S();
  const long long nwords = (n + 8 + 7) / 8 + 24;
  if (S.dna_bytes.reserve((size_t)n + 2) != BATHGPU_OK || S.dna4.reserve((size_t)nwords * 4) != BATHGPU_OK ||
      ctx->wins.reserve((size_t)nwin * sizeof(WindowDesc)) != BATHGPU_OK || ctx->fwdsc.reserve((size_t)nwin * 4) != BATHGPU_OK ||
      ctx->status.reserve((size_t)nwin * 4) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  S.block_n = n; S.nres = 0; S.bytes_valid = (packed == nullptr);
  // windows in order of their last nucleotide ; callers that tile a block are already in order
  static_assert(sizeof(WindowDesc) == sizeof(bathgpu_window), "descriptor layouts must agree");
  bool in_order = true;
  for (int w = 1; w < nwin && in_order; ++w) in_order = wins[w - 1].start + wins[w - 1].L <= wins[w].start + wins[w].L;
  std::vector<int> order;
  std::vector<WindowDesc> sorted;
  std::vector<float> sc;
  std::vector<int> st;
  if (!in_order) {
    order.resize((size_t)nwin); sorted.resize((size_t)nwin); sc.resize((size_t)nwin); st.resize((size_t)nwin);
    for (int w = 0; w < nwin; ++w) order[w] = w;
    std::sort(order.begin(), order.end(), [&](int x, int y) { return wins[x].start + wins[x].L < wins[y].start + wins[y].L; });
    for (int w = 0; w < nwin; ++w) memcpy(&sorted[w], &wins[order[w]], sizeof(WindowDesc));
  }
  const WindowDesc *hw = in_order ? reinterpret_cast<const WindowDesc *>(wins) : sorted.data();
  // Chunks grow fourfold: scoring a chunk takes several times longer than moving it, so every later chunk arrives while the
  // one before it is being scored, and the first one is small enough that the device starts almost at once.
  long long cuts[8]; int K = 0;
  {
    long long first = n / 85, p = 0;
    // the first launch should fill the device: one resident wave of windows (16 warps per SM) has to end inside the first chunk
    const int wave = ctx->prop.multiProcessorCount * 16;
    if (nwin > wave) first = std::min<long long>(std::max<long long>(first, hw[wave].start + hw[wave].L), std::max<long long>(first, n / 8));
    if (n < (4 << 20)) first = n;
    for (long long sz = std::max<long long>(first, 1 << 20); p < n && K < 7; sz *= 4) { p = std::min<long long>(n, (p + sz + 7) & ~7LL); cuts[K++] = p; }
    cuts[K - 1] = n;
  }
  cudaEvent_t *pack_ev = ctx->chunk_ev, *join_ev = ctx->chunk_ev + 8;
  for (int c = 0; c < K; ++c) {
    const long long p0 = c ? cuts[c - 1] : 0, p1 = cuts[c];                       // 0-based nucleotides [p0, p1); dsq[1 + p] is nucleotide p
    if (packed) {
      // host-packed: bytes p0/2 .. (p1+1)/2 land in the packed words themselves (cuts are multiples of 8 except the last)
      CUDA_TRY(ctx, cudaMemcpyAsync(S.dna4.as<uint8_t>() + 4 + p0 / 2, packed + p0 / 2, (size_t)((p1 + 1) / 2 - p0 / 2), cudaMemcpyHostToDevice, ctx->copy_stream));
      {
        const long long b0 = (4 + p0 / 2) & ~127LL, b1 = 4 + (p1 + 1) / 2, lines = (b1 - b0 + 127) / 128;
        l2_prefetch_kernel<<<(unsigned)((lines + 255) / 256), 256, 0, ctx->copy_stream>>>(S.dna4.as<uint8_t>() + b0, b1 - b0);
      }
      if (p1 >= n) dna4_guards_kernel<<<1, 32, 0, ctx->copy_stream>>>(S.dna4.as<uint32_t>(), n);
      else if (c == 0) dna4_guards_kernel<<<1, 1, 0, ctx->copy_stream>>>(S.dna4.as<uint32_t>(), n);     // the front guard word (thread 0 only)
    } else {
      CUDA_TRY(ctx, cudaMemcpyAsync(S.dna_bytes.as<uint8_t>() + 1 + p0, dsq + 1 + p0, (size_t)(p1 - p0), cudaMemcpyHostToDevice, ctx->copy_stream));
      // packed word w holds nucleotides 8w-8 .. 8w-1: this chunk completes words p0/8+1 .. p1/8 (and the tail guard at the end)
      const long long wlo = (c == 0) ? 0 : p0 / 8 + 1, whi = (p1 >= n) ? nwords : p1 / 8 + 1;
      if (whi > wlo)
        pack_dna4_range_kernel<<<(unsigned)((whi - wlo + 255) / 256), 256, 0, ctx->copy_stream>>>(S.dna_bytes.as<uint8_t>(), n, S.dna4.as<uint32_t>(), wlo, whi);
    }
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(pack_ev[c], ctx->copy_stream));
  }
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->wins.p, hw, (size_t)nwin * sizeof(WindowDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, 64, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  // launches alternate between two streams, so the tail of one launch (its last windows finishing on a thinning set of SMs)
  // is filled by the head of the next
  const FsProfileImage &im = ctx->fs3;
  int w0 = 0, launches = 0;
  for (int c = 0; c < K; ++c) {
    const long long ready_nt = (c == K - 1) ? n : 8 * (cuts[c] / 8);               // nucleotides whose packed words are complete
    int w1 = w0;
    while (w1 < nwin && hw[w1].start + hw[w1].L - 1 <= ready_nt) ++w1;
    if (c == K - 1) w1 = nwin;
    if (w1 == w0) continue;
    cudaStream_t s = (launches & 1) ? ctx->stream2 : ctx->stream;
    if (launches == 1) CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev0, 0));    // descriptors and counters are set on the first stream
    CUDA_TRY(ctx, cudaStreamWaitEvent(s, pack_ev[c], 0));
    FsParserArgs a{};
    a.emis = im.emis_fwd.as<float>(); a.cellc = im.cellc.as<float>(); a.dna4 = S.dna4.as<uint32_t>();
    a.wins = ctx->wins.as<WindowDesc>() + w0; a.nwin = w1 - w0; a.mpad = im.mpad; a.tEM = xfE[0]; a.tEL = xfE[1];
    a.fwdsc = ctx->fwdsc.as<float>() + w0; a.status = ctx->status.as<int>() + w0; a.xmx = nullptr; a.xoff = nullptr;
    a.counter = ctx->counter.as<int>() + launches; a.scan_steps = im.scan_steps; a.cellmw = im.cellmw.as<float>(); a.mw_scan_steps = im.mw_scan_steps;
    CUDA_TRY(ctx, dispatch_fwd(false, im.J, a, ctx->prop.multiProcessorCount, s));
    ++launches;
    w0 = w1;
  }
  if (launches > 1) {
    CUDA_TRY(ctx, cudaEventRecord(join_ev[0], ctx->stream2));
    CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, join_ev[0], 0));
  }
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(in_order ? fwdsc : sc.data(), ctx->fwdsc.p, (size_t)nwin * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(in_order ? status : st.data(), ctx->status.p, (size_t)nwin * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
  if (!in_order) for (int w = 0; w < nwin; ++w) { fwdsc[order[w]] = sc[w]; status[order[w]] = st[w]; }
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
  ctx->last_launches = launches;
  ctx->nstaged = 0;
  return BATHGPU_OK;
}

extern "C" int bathgpu_fs_fwd_block(bathgpu_ctx *ctx, const uint8_t *dsq, int64_t n, const bathgpu_window *wins, int nwin,
                                    const float xfE[2], float *fwdsc, int32_t *status)
{
  if (!dsq) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_fwd_block");
  return fs_fwd_block_impl(ctx, dsq, nullptr, n, wins, nwin, xfE, fwdsc, status);
}

extern "C" int bathgpu_fs_fwd_block_packed4(bathgpu_ctx *ctx, const uint8_t *packed, int64_t n, const bathgpu_window *wins, int nwin,
                                            const float xfE[2], float *fwdsc, int32_t *status)
{
  if (!packed) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_fwd_block_packed4");
  return fs_fwd_block_impl(ctx, nullptr, packed, n, wins, nwin, xfE, fwdsc, status);
}

// ---------------------------------------------------------------------------------------------
// Forward parser stage
// BATHGPU_FWD=3|4 forces a kernel generation for A/B runs (3: the row-pair schedule; 4: row pairs on packed FP32, fs_parser_v4.cuh).  Unset: per node count, what measured faster on B200 (profiles/r02_forward_v3_v4.md): the packed
// kernel at 10 nodes per lane (256 < M <= 320: +21 % at M = 279), the scalar row-pair kernel elsewhere (equal at 6 and 12, the packed one
// spills at 7-8 and loses a third at 16: 628 vs 907 GCUPS at M = 409).
static int fwd_version(int J)
{
  static const int forced = [] { const char *e = getenv("BATHGPU_FWD"); int x = e ? atoi(e) : 0; return (x == 3 || x == 4) ? x : 0; }();
  if (forced) return forced;
  return (J == 10) ? 4 : 3;
}

// one launch entry per kernel family and node-count set (launch.h; kernels_tu.cu)
static cudaError_t dispatch_fwd(bool xmx, int J, const FsParserArgs &a, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
  const int v = fwd_version(J);
#define X(S) if (launch_fs3_forward_##S(J, xmx, v, a, sms, s, &e)) return e;
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return cudaErrorInvalidValue;
}

static int check_windows(bathgpu_ctx *ctx, const bathgpu_window *wins, int n)
{
  for (int w = 0; w < n; ++w) {
    if (wins[w].L < 3 || wins[w].start < 1 || wins[w].start + wins[w].L - 1 > ctx->S().block_n)
      return fail(ctx, BATHGPU_EINVAL, "window %d (start %lld, L %d) is outside the uploaded block (n=%lld) or shorter than 3",
                  w, (long long)wins[w].start, wins[w].L, (long long)ctx->S().block_n);
  }
  return BATHGPU_OK;
}

extern "C" int bathgpu_stage_windows(bathgpu_ctx *ctx, const bathgpu_window *wins, int n)
{
  if (!ctx || !wins || n < 1) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_stage_windows");
  if (ctx->S().block_n == 0)      return fail(ctx, BATHGPU_EINVAL, "no block uploaded");
  int st = check_windows(ctx, wins, n);
  if (st != BATHGPU_OK) return st;
  CUDA_TRY(ctx, enter(ctx));
  static_assert(sizeof(WindowDesc) == sizeof(bathgpu_window), "descriptor layouts must agree");
  if (ctx->wins.reserve((size_t)n * sizeof(WindowDesc)) != BATHGPU_OK || ctx->fwdsc.reserve((size_t)n * 4) != BATHGPU_OK ||
      ctx->status.reserve((size_t)n * 4) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->wins.p, wins, (size_t)n * sizeof(WindowDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  ctx->nstaged = n;
  return BATHGPU_OK;
}

extern "C" int bathgpu_fs_fwd_staged(bathgpu_ctx *ctx, const float xfE[2])
{
  if (!ctx || !xfE)          return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_fwd_staged");
  if (!ctx->fs3.loaded)      return fail(ctx, BATHGPU_EINVAL, "3-codon profile not loaded");
  if (ctx->nstaged < 1)      return fail(ctx, BATHGPU_EINVAL, "no windows staged");
  CUDA_TRY(ctx, enter(ctx));
  const FsProfileImage &im = ctx->fs3;
  FsParserArgs a{};
  a.emis = im.emis_fwd.as<float>(); a.cellc = im.cellc.as<float>(); a.dna4 = ctx->S().dna4.as<uint32_t>();
  a.wins = ctx->wins.as<WindowDesc>(); a.nwin = ctx->nstaged; a.mpad = im.mpad;
  a.tEM = xfE[0]; a.tEL = xfE[1];
  a.fwdsc = ctx->fwdsc.as<float>(); a.status = ctx->status.as<int>();
  a.xmx = nullptr; a.xoff = nullptr; a.counter = ctx->counter.as<int>(); a.scan_steps = im.scan_steps; a.cellmw = im.cellmw.as<float>(); a.mw_scan_steps = im.mw_scan_steps;

  CUDA_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, 4, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  CUDA_TRY(ctx, dispatch_fwd(false, im.J, a, ctx->prop.multiProcessorCount, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
  ctx->last_launches = 1;
  return BATHGPU_OK;
}

extern "C" int bathgpu_fetch_scores(bathgpu_ctx *ctx, float *fwdsc, int32_t *status, int n)
{
  if (!ctx || n < 1 || n > ctx->nstaged) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fetch_scores");
  CUDA_TRY(ctx, enter(ctx));
  if (fwdsc)  CUDA_TRY(ctx, cudaMemcpyAsync(fwdsc,  ctx->fwdsc.p,  (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (status) CUDA_TRY(ctx, cudaMemcpyAsync(status, ctx->status.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  return BATHGPU_OK;
}

extern "C" int bathgpu_fs_fwd_windows(bathgpu_ctx *ctx, const bathgpu_window *wins, int n, const float xfE[2],
                                      float *fwdsc, int32_t *status)
{
  int st;
  if (!fwdsc || !status) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_fwd_windows");
  if ((st = bathgpu_stage_windows(ctx, wins, n)) != BATHGPU_OK) return st;
  if ((st = bathgpu_fs_fwd_staged(ctx, xfE))     != BATHGPU_OK) return st;
  return bathgpu_fetch_scores(ctx, fwdsc, status, n);
}

// ---------------------------------------------------------------------------------------------
static cudaError_t dispatch_bck(int J, const FsBackwardArgs &a, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
#define X(S) if (launch_fs3_backward_##S(J, a, sms, s, &e)) return e;
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return cudaErrorInvalidValue;
}

// a10 + a11 for one chunk of windows whose descriptors are already in ctx->wins
// x_off0 / fx_out / bx_out: when given, the X rows of both parsers are returned (rows of this chunk start at x_off0)
// and the decoding kernel is skipped (xf5_loop == nullptr)
static int bck_decode_chunk(bathgpu_ctx *ctx, const bathgpu_window *wins, int n, const float xfE[2], const float xf5_loop[3],
                            const int64_t *out_offset, float *mocc, float *btot, float *etot,
                            float *fwdsc, float *bcksc, int32_t *status,
                            int64_t x_off0 = 0, float *fx_out = nullptr, float *bx_out = nullptr)
{
  const bool decode = (xf5_loop != nullptr);
  const FsProfileImage &im = ctx->fs3;
  std::vector<long long> xoff(n + 1, 0);
  for (int w = 0; w < n; ++w) xoff[w + 1] = xoff[w] + wins[w].L + 1;
  const size_t rows = (size_t)xoff[n];

  if (ctx->wins.reserve((size_t)n * sizeof(WindowDesc)) != BATHGPU_OK || ctx->fwdsc.reserve((size_t)n * 4) != BATHGPU_OK ||
      ctx->bcksc.reserve((size_t)n * 4) != BATHGPU_OK || ctx->status.reserve((size_t)n * 4) != BATHGPU_OK ||
      ctx->counter.reserve(64) != BATHGPU_OK || ctx->xoff.reserve((size_t)(n + 1) * 8) != BATHGPU_OK ||
      ctx->fxmx.reserve(rows * 24) != BATHGPU_OK || ctx->bxmx.reserve(rows * 24) != BATHGPU_OK ||
      ctx->lsf.reserve((rows + 2 * (size_t)n) * 4) != BATHGPU_OK || ctx->lsb.reserve((rows + 2 * (size_t)n) * 4) != BATHGPU_OK ||
      ctx->dmocc.reserve(rows * 4) != BATHGPU_OK || ctx->dbtot.reserve(rows * 4) != BATHGPU_OK || ctx->detot.reserve(rows * 4) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for %d windows (%zu rows)", n, rows);
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->wins.p, wins, (size_t)n * sizeof(WindowDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->xoff.p, xoff.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  ctx->nstaged = n;
  ctx->xrows = (int64_t)rows;

  const int sms = ctx->prop.multiProcessorCount;
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));

  FsParserArgs fa{};
  fa.emis = im.emis_fwd.as<float>(); fa.cellc = im.cellc.as<float>(); fa.dna4 = ctx->S().dna4.as<uint32_t>();
  fa.wins = ctx->wins.as<WindowDesc>(); fa.nwin = n; fa.mpad = im.mpad; fa.tEM = xfE[0]; fa.tEL = xfE[1];
  fa.fwdsc = ctx->fwdsc.as<float>(); fa.status = ctx->status.as<int>();
  fa.xmx = ctx->fxmx.as<float>(); fa.xoff = ctx->xoff.as<long long>(); fa.counter = ctx->counter.as<int>(); fa.scan_steps = im.scan_steps; fa.cellmw = im.cellmw.as<float>(); fa.mw_scan_steps = im.mw_scan_steps;
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, 4, ctx->stream));
  CUDA_TRY(ctx, dispatch_fwd(true, im.J, fa, sms, ctx->stream));

  FsBackwardArgs ba{};
  ba.emis = im.emis_bck.as<float>(); ba.cellb = im.cellb3.as<float>(); ba.cellbmw = im.cellbmw.as<float>(); ba.dna4 = fa.dna4; ba.wins = fa.wins; ba.nwin = n; ba.mpad = im.mpad;
  ba.tEM = xfE[0]; ba.tEL = xfE[1]; ba.fxmx = ctx->fxmx.as<float>(); ba.bxmx = ctx->bxmx.as<float>(); ba.xoff = fa.xoff;
  ba.bcksc = ctx->bcksc.as<float>(); ba.status = fa.status; ba.counter = fa.counter;
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, 4, ctx->stream));
  CUDA_TRY(ctx, dispatch_bck(im.J, ba, sms, ctx->stream));

  std::vector<float> hm, hb, he;
  if (decode) {
    DomainDecodeArgs da{};
    da.fxmx = ba.fxmx; da.bxmx = ba.bxmx; da.xoff = fa.xoff; da.wins = fa.wins; da.nwin = n;
    da.tNL = xf5_loop[0]; da.tJL = xf5_loop[1]; da.tCL = xf5_loop[2];
    da.lsf = ctx->lsf.as<float>(); da.lsb = ctx->lsb.as<float>();
    da.mocc = ctx->dmocc.as<float>(); da.btot = ctx->dbtot.as<float>(); da.etot = ctx->detot.as<float>();
    da.ooff = fa.xoff; da.status = fa.status;
    fs_domain_decoding_kernel<<<(n + 3) / 4, 128, 0, ctx->stream>>>(da);
    CUDA_TRY(ctx, cudaGetLastError());
  }
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));

  if (decode) {
    hm.resize(rows); hb.resize(rows); he.resize(rows);
    CUDA_TRY(ctx, cudaMemcpyAsync(hm.data(), ctx->dmocc.p, rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(hb.data(), ctx->dbtot.p, rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(he.data(), ctx->detot.p, rows * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (fx_out) CUDA_TRY(ctx, cudaMemcpyAsync(fx_out + (size_t)x_off0 * 6, ctx->fxmx.p, rows * 24, cudaMemcpyDeviceToHost, ctx->stream));
  if (bx_out) CUDA_TRY(ctx, cudaMemcpyAsync(bx_out + (size_t)x_off0 * 6, ctx->bxmx.p, rows * 24, cudaMemcpyDeviceToHost, ctx->stream));
  if (fwdsc) CUDA_TRY(ctx, cudaMemcpyAsync(fwdsc, ctx->fwdsc.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (bcksc) CUDA_TRY(ctx, cudaMemcpyAsync(bcksc, ctx->bcksc.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(status, ctx->status.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  float ms = 0.f;
  CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  ctx->last_ms += ms;
  ctx->last_launches += decode ? 3 : 2;
  if (decode)
    for (int w = 0; w < n; ++w) {
      const size_t len = (size_t)wins[w].L + 1;
      memcpy(mocc + out_offset[w], hm.data() + xoff[w], len * 4);
      memcpy(btot + out_offset[w], hb.data() + xoff[w], len * 4);
      memcpy(etot + out_offset[w], he.data() + xoff[w], len * 4);
    }
  return BATHGPU_OK;
}

extern "C" int bathgpu_fs_bck_decode(bathgpu_ctx *ctx, const bathgpu_window *wins, int n, const float xfE[2],
                                     const float xf5_loop[3], const int64_t *out_offset,
                                     float *mocc, float *btot, float *etot, float *fwdsc, float *bcksc, int32_t *status)
{
  if (!ctx || !wins || n < 1 || !xfE || !xf5_loop || !out_offset || !mocc || !btot || !etot || !status)
    return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_bck_decode");
  if (!ctx->fs3.loaded)  return fail(ctx, BATHGPU_EINVAL, "3-codon profile not loaded");
  if (ctx->S().block_n == 0) return fail(ctx, BATHGPU_EINVAL, "no block uploaded");
  int st = check_windows(ctx, wins, n);
  if (st != BATHGPU_OK) return st;
  for (int w = 0; w < n; ++w)
    if (wins[w].L < 5) return fail(ctx, BATHGPU_EINVAL, "window %d: the Backward parser needs L >= 5 (fwdback_fs.c:600)", w);
  CUDA_TRY(ctx, enter(ctx));
  ctx->last_ms = 0.f; ctx->last_launches = 0;
  // chunks bounded by X-row memory: 68 B per row of scratch
  const size_t max_rows = (size_t)16 << 20;
  int w0 = 0;
  while (w0 < n) {
    size_t rows = 0;
    int w1 = w0;
    while (w1 < n && (w1 == w0 || rows + wins[w1].L + 1 <= max_rows)) { rows += wins[w1].L + 1; ++w1; }
    st = bck_decode_chunk(ctx, wins + w0, w1 - w0, xfE, xf5_loop, out_offset + w0, mocc, btot, etot,
                          fwdsc ? fwdsc + w0 : nullptr, bcksc ? bcksc + w0 : nullptr, status + w0);
    if (st != BATHGPU_OK) return st;
    w0 = w1;
  }
  return BATHGPU_OK;
}

// a10 alone: Forward (keeping X rows) + Backward parsers over windows; X rows of both come back to the host, which
// runs p7_DomainDecoding_Frameshift itself (it needs a length-model value that depends on the previous window's
// envelopes, src/p7_domaindef.c:320-325, :1018 -- an O(L) scalar pass the reference also does per window).
extern "C" int bathgpu_fs_fwd_bck_xrows(bathgpu_ctx *ctx, const bathgpu_window *wins, int n, const float xfE[2],
                                        float *fwd_xrows, float *bck_xrows, float *fwdsc, float *bcksc, int32_t *status)
{
  if (!ctx || !wins || n < 1 || !xfE || !fwd_xrows || !bck_xrows || !status)
    return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_fwd_bck_xrows");
  if (!ctx->fs3.loaded)  return fail(ctx, BATHGPU_EINVAL, "3-codon profile not loaded");
  if (ctx->S().block_n == 0) return fail(ctx, BATHGPU_EINVAL, "no block uploaded");
  int st = check_windows(ctx, wins, n);
  if (st != BATHGPU_OK) return st;
  for (int w = 0; w < n; ++w)
    if (wins[w].L < 5) return fail(ctx, BATHGPU_EINVAL, "window %d: the Backward parser needs L >= 5 (fwdback_fs.c:600)", w);
  CUDA_TRY(ctx, enter(ctx));
  ctx->last_ms = 0.f; ctx->last_launches = 0;
  const size_t max_rows = (size_t)16 << 20;
  int w0 = 0;
  int64_t x0 = 0;
  while (w0 < n) {
    size_t rows = 0;
    int w1 = w0;
    while (w1 < n && (w1 == w0 || rows + wins[w1].L + 1 <= max_rows)) { rows += wins[w1].L + 1; ++w1; }
    st = bck_decode_chunk(ctx, wins + w0, w1 - w0, xfE, nullptr, nullptr, nullptr, nullptr, nullptr,
                          fwdsc ? fwdsc + w0 : nullptr, bcksc ? bcksc + w0 : nullptr, status + w0, x0, fwd_xrows, bck_xrows);
    if (st != BATHGPU_OK) return st;
    x0 += (int64_t)rows;
    w0 = w1;
  }
  return BATHGPU_OK;
}

extern "C" int bathgpu_fs_fetch_xrows(bathgpu_ctx *ctx, int which, float *out, int64_t nrows)
{
  if (!ctx || !out || nrows < 1 || nrows > ctx->xrows || (which != 0 && which != 1))
    return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_fetch_xrows");
  CUDA_TRY(ctx, enter(ctx));
  const DevBuf &b = which ? ctx->bxmx : ctx->fxmx;
  CUDA_TRY(ctx, cudaMemcpyAsync(out, b.p, (size_t)nrows * 24, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  return BATHGPU_OK;
}

static cudaError_t dispatch_domains(int J, const DomainArgs &a, const TraceArgs &t, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
#define X(S) if (launch_fs5_domains_##S(J, a, t, sms, s, &e)) return e;
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return cudaErrorInvalidValue;
}

// p7_trace_fs_Reverse (src/p7_trace.c:2527-2568): pull N/C/J residues back by one, then reverse.
static void finish_trace(TraceStep *tr, int n)
{
  for (int z = 0; z + 1 < n; ++z) {
    if (tr[z].st == tr[z + 1].st && (tr[z].st == TS_N || tr[z].st == TS_C || tr[z].st == TS_J)) {
      if (tr[z].i == 0 && tr[z + 1].i > 0) {
        tr[z].i = tr[z + 1].i;   tr[z + 1].i = 0;
        tr[z].pp = tr[z + 1].pp; tr[z + 1].pp = 0.0f;
      }
    }
  }
  std::reverse(tr, tr + n);
}

static int domains_chunk(bathgpu_ctx *ctx, const bathgpu_envelope *envs, int n, const float xfE5[2],
                         bathgpu_domain_result *results, bathgpu_trace_step *traces, int64_t max_steps, int64_t &steps_used)
{
  const FsProfileImage &im = ctx->fs5;
  const int M = im.M, mpad = im.mpad;
  std::vector<long long> xoff(n + 1, 0), toff(n + 1, 0);
  for (int e = 0; e < n; ++e) { xoff[e + 1] = xoff[e] + envs[e].L + 1; toff[e + 1] = toff[e] + envs[e].L + M + 8; }
  const size_t rows = (size_t)xoff[n];
  static_assert(sizeof(EnvelopeDesc) == sizeof(bathgpu_envelope), "descriptor layouts must agree");
  static_assert(sizeof(TraceStep) == sizeof(bathgpu_trace_step), "trace step layouts must agree");

  if (ctx->envs.reserve((size_t)n * sizeof(EnvelopeDesc)) != BATHGPU_OK || ctx->xoff.reserve((size_t)(n + 1) * 8) != BATHGPU_OK ||
      ctx->dtoff.reserve((size_t)(n + 1) * 8) != BATHGPU_OK || ctx->dtlen.reserve((size_t)n * 4) != BATHGPU_OK ||
      reserve_matrices(ctx, (rows + 1) * kPPCells * mpad * 4, rows * kOACells * mpad * 4) != BATHGPU_OK ||        /* + 1: the optimal-accuracy sweep prefetches one row ahead */
      ctx->dfx.reserve(rows * 24) != BATHGPU_OK || ctx->dppx.reserve(rows * 24) != BATHGPU_OK || ctx->doax.reserve(rows * 24) != BATHGPU_OK ||
      ctx->dlsf.reserve(rows * 4) != BATHGPU_OK || ctx->dfw.reserve((size_t)n * 4) != BATHGPU_OK || ctx->dbk.reserve((size_t)n * 4) != BATHGPU_OK ||
      ctx->doasc.reserve((size_t)n * 4) != BATHGPU_OK || ctx->dnull2.reserve((size_t)n * 29 * 4) != BATHGPU_OK ||
      ctx->dstat.reserve((size_t)n * 4) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK ||
      ctx->dsteps.reserve((size_t)toff[n] * sizeof(TraceStep)) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for %d envelopes (%zu rows, M=%d)", n, rows, M);
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->envs.p, envs, (size_t)n * sizeof(EnvelopeDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->xoff.p, xoff.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->dtoff.p, toff.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));

  DomainArgs a{};
  a.emis = im.emis.as<float>(); a.amino = im.amino.as<float>(); a.cellf = im.cellf5.as<float>(); a.cellb = im.cellb.as<float>();
  a.oapass = im.oapass.as<float>(); a.oaflags = im.oaflags.as<uint32_t>(); a.dna4 = ctx->S().dna4.as<uint32_t>();
  a.envs = ctx->envs.as<EnvelopeDesc>(); a.nenv = n; a.M = M; a.mpad = mpad; a.tEM = xfE5[0]; a.tEL = xfE5[1];
  a.xoff = ctx->xoff.as<long long>(); a.pp = ctx->dpp.as<float>(); a.oa = ctx->doa.as<float>(); a.fx = ctx->dfx.as<float>();
  a.ppx = ctx->dppx.as<float>(); a.oax = ctx->doax.as<float>(); a.lsf = ctx->dlsf.as<float>();
  a.fwdsc = ctx->dfw.as<float>(); a.bcksc = ctx->dbk.as<float>(); a.oasc = ctx->doasc.as<float>();
  a.null2 = ctx->dnull2.as<float>(); a.status = ctx->dstat.as<int>(); a.counter = ctx->counter.as<int>();
  TraceArgs t{};
  t.steps = ctx->dsteps.as<TraceStep>(); t.toff = ctx->dtoff.as<long long>(); t.tlen = ctx->dtlen.as<int>();
  t.tfv = im.tfvraw.as<float>(); t.J = im.J;

  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  CUDA_TRY(ctx, dispatch_domains(im.J, a, t, ctx->prop.multiProcessorCount, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));

  std::vector<float> fw(n), bk(n), oa(n), n2((size_t)n * 29);
  std::vector<int> st(n), tl(n);
  std::vector<TraceStep> steps((size_t)toff[n]);
  CUDA_TRY(ctx, cudaMemcpyAsync(fw.data(), ctx->dfw.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(bk.data(), ctx->dbk.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(oa.data(), ctx->doasc.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(n2.data(), ctx->dnull2.p, (size_t)n * 29 * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(st.data(), ctx->dstat.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(tl.data(), ctx->dtlen.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(steps.data(), ctx->dsteps.p, steps.size() * sizeof(TraceStep), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  float ms = 0.f;
  CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  ctx->last_ms += ms;
  ctx->last_launches += 4;
  ctx->dom_xoff = xoff;
  ctx->dom_L.assign(n, 0);
  for (int e = 0; e < n; ++e) ctx->dom_L[e] = envs[e].L;

  for (int e = 0; e < n; ++e) {
    bathgpu_domain_result &r = results[e];
    r.envsc = fw[e]; r.bcksc = bk[e]; r.oasc = oa[e]; r.status = st[e];
    memcpy(r.null2, &n2[(size_t)e * 29], 29 * 4);
    r.trace_offset = (int32_t)steps_used; r.trace_len = 0;
    if (st[e] == 0 && tl[e] > 0) {
      if (steps_used + tl[e] > max_steps)
        return fail(ctx, BATHGPU_EINVAL, "trace buffer too small: %lld steps needed so far, %lld given", (long long)(steps_used + tl[e]), (long long)max_steps);
      TraceStep *tr = &steps[(size_t)toff[e]];
      finish_trace(tr, tl[e]);
      memcpy(traces + steps_used, tr, (size_t)tl[e] * sizeof(TraceStep));
      r.trace_len = tl[e];
      steps_used += tl[e];
    }
  }
  return BATHGPU_OK;
}

extern "C" int bathgpu_fs_domains(bathgpu_ctx *ctx, const bathgpu_envelope *envs, int n, const float xfE5[2],
                                  bathgpu_domain_result *results, bathgpu_trace_step *traces, int64_t max_steps)
{
  if (!ctx || !envs || n < 1 || !xfE5 || !results || !traces || max_steps < 1)
    return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_domains");
  if (!ctx->fs5.loaded)  return fail(ctx, BATHGPU_EINVAL, "5-codon profile not loaded");
  if (ctx->S().block_n == 0) return fail(ctx, BATHGPU_EINVAL, "no block uploaded");
  for (int e = 0; e < n; ++e)
    if (envs[e].L < 6 || envs[e].start < 1 || envs[e].start + envs[e].L - 1 > ctx->S().block_n)
      return fail(ctx, BATHGPU_EINVAL, "envelope %d (start %lld, L %d) is outside the uploaded block (n=%lld) or shorter than 6",
                  e, (long long)envs[e].start, envs[e].L, (long long)ctx->S().block_n);
  CUDA_TRY(ctx, enter(ctx));
  ctx->last_ms = 0.f; ctx->last_launches = 0;
  // chunks bounded by matrix memory: (7 + 3) * mpad * 4 B per row
  const size_t row_bytes = (size_t)(kPPCells + kOACells) * ctx->fs5.mpad * 4;
  const size_t max_rows = std::max<size_t>(matrix_budget() / row_bytes - 1, 4096);
  int64_t steps_used = 0;
  int e0 = 0;
  while (e0 < n) {
    size_t rows = 0;
    int e1 = e0;
    while (e1 < n && (e1 == e0 || rows + envs[e1].L + 1 <= max_rows)) { rows += envs[e1].L + 1; ++e1; }
    int st = domains_chunk(ctx, envs + e0, e1 - e0, xfE5, results + e0, traces, max_steps, steps_used);
    if (st != BATHGPU_OK) return st;
    e0 = e1;
  }
  return BATHGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// Forward matrices for the stochastic traceback (a16)
static cudaError_t dispatch_forward_matrix(int J, const DomainArgs &a, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
#define X(S) if (launch_fs5_forward_matrix_##S(J, a, sms, s, &e)) return e;
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return cudaErrorInvalidValue;
}

// Stored Forward cells -> the reference's cell order and values: out[(row * (M+1) + k) * 8 + {D, I, M_C0..M_C5}]
// (src/impl_sse/impl_sse.h:296-314, un-striped); match cells are stored times Z(k) (fs_domain.cuh) and divided back here.
__global__ void fs5_export_forward_kernel(const float *__restrict__ pp, const float *__restrict__ dcell, const float *__restrict__ zinv,
                                          int J, int M, int mpad, long long rows, float *__restrict__ out)
{
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * (M + 1)) return;
  const long long row = t / (M + 1);
  const int k = (int)(t - row * (M + 1));
  float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
  if (k > 0) {
    const int VEC = (J % 4 == 0) ? 4 : ((J % 2 == 0) ? 2 : 1);
    const int kk = k - 1, lane = kk / J, j = kk % J;
    const int p = (j / VEC) * (32 * VEC) + lane * VEC + (j % VEC);
    const float *r = pp + (size_t)row * kPPCells * mpad + p;
    const float zi = zinv[kk];
    lo.x = dcell[(size_t)row * mpad + p];
    lo.y = r[(size_t)PP_I * mpad];
    lo.z = r[(size_t)PP_C0 * mpad] * zi;
    lo.w = r[(size_t)(PP_C0 + 1) * mpad] * zi;
    hi.x = r[(size_t)(PP_C0 + 2) * mpad] * zi;
    hi.y = r[(size_t)(PP_C0 + 3) * mpad] * zi;
    hi.z = r[(size_t)(PP_C0 + 4) * mpad] * zi;
    hi.w = r[(size_t)(PP_C0 + 5) * mpad] * zi;
  }
  float4 *o = reinterpret_cast<float4 *>(out + (size_t)t * 8);
  o[0] = lo; o[1] = hi;
}

extern "C" int bathgpu_fs_forward_matrices(bathgpu_ctx *ctx, const bathgpu_envelope *regs, int n, const float xfE5[2],
                                           float *mx, float *xrows, int64_t max_rows, float *fwdsc, int32_t *status)
{
  if (!ctx || !regs || n < 1 || !xfE5 || (!mx) != (!xrows) || !fwdsc || !status) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_forward_matrices");
  const bool scores_only = !mx;          // p7_ForwardParser_Frameshift_5Codons: the score, nothing handed back
  if (!ctx->fs5.loaded)      return fail(ctx, BATHGPU_EINVAL, "5-codon profile not loaded");
  if (ctx->S().block_n == 0) return fail(ctx, BATHGPU_EINVAL, "no block uploaded");
  int64_t total = 0;
  for (int e = 0; e < n; ++e) {
    if (regs[e].L < 6 || regs[e].start < 1 || regs[e].start + regs[e].L - 1 > ctx->S().block_n)
      return fail(ctx, BATHGPU_EINVAL, "region %d (start %lld, L %d) is outside the uploaded block (n=%lld) or shorter than 6",
                  e, (long long)regs[e].start, regs[e].L, (long long)ctx->S().block_n);
    total += regs[e].L + 1;
  }
  if (!scores_only && total > max_rows) return fail(ctx, BATHGPU_EINVAL, "matrix buffer too small: %lld rows needed, %lld given", (long long)total, (long long)max_rows);
  CUDA_TRY(ctx, enter(ctx));
  const FsProfileImage &im = ctx->fs5;
  const int M = im.M, mpad = im.mpad;
  ctx->last_ms = 0.f; ctx->last_launches = 0;
  // chunks bounded by device memory: 8 stored cells + 8 exported per node and row
  const size_t row_bytes = (size_t)(kPPCells + 1) * mpad * 4 + (size_t)(M + 1) * 32 + 32;
  const size_t cap_rows = std::max<size_t>(std::min<size_t>(((size_t)4 << 30) / row_bytes, matrix_budget() / 10 * 7 / ((size_t)kPPCells * mpad * 4)), 8192);
  int e0 = 0;
  int64_t row0 = 0;
  while (e0 < n) {
    int e1 = e0;
    size_t rows = 0;
    while (e1 < n && (e1 == e0 || rows + regs[e1].L + 1 <= cap_rows)) { rows += regs[e1].L + 1; ++e1; }
    const int m = e1 - e0;
    std::vector<long long> xoff(m + 1, 0);
    for (int e = 0; e < m; ++e) xoff[e + 1] = xoff[e] + regs[e0 + e].L + 1;
    if (ctx->envs.reserve((size_t)m * sizeof(EnvelopeDesc)) != BATHGPU_OK || ctx->xoff.reserve((size_t)(m + 1) * 8) != BATHGPU_OK ||
        reserve_matrices(ctx, rows * kPPCells * mpad * 4, 0) != BATHGPU_OK || ctx->ddcell.reserve(rows * mpad * 4) != BATHGPU_OK ||
        ctx->dmxout.reserve(scores_only ? 32 : rows * (size_t)(M + 1) * 32) != BATHGPU_OK || ctx->dfx.reserve(rows * 24) != BATHGPU_OK ||
        ctx->dlsf.reserve(rows * 4) != BATHGPU_OK || ctx->dfw.reserve((size_t)m * 4) != BATHGPU_OK ||
        ctx->dstat.reserve((size_t)m * 4) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK)
      return fail(ctx, BATHGPU_EMEM, "device allocation failed for %d regions (%zu rows, M=%d)", m, rows, M);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->envs.p, regs + e0, (size_t)m * sizeof(EnvelopeDesc), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->xoff.p, xoff.data(), (size_t)(m + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    DomainArgs a{};
    a.emis = im.emis.as<float>(); a.cellf = im.cellf5.as<float>(); a.dna4 = ctx->S().dna4.as<uint32_t>();
    a.envs = ctx->envs.as<EnvelopeDesc>(); a.nenv = m; a.M = M; a.mpad = mpad; a.tEM = xfE5[0]; a.tEL = xfE5[1];
    a.xoff = ctx->xoff.as<long long>(); a.pp = ctx->dpp.as<float>(); a.dcell = ctx->ddcell.as<float>(); a.fx = ctx->dfx.as<float>();
    a.lsf = ctx->dlsf.as<float>(); a.fwdsc = ctx->dfw.as<float>(); a.status = ctx->dstat.as<int>(); a.counter = ctx->counter.as<int>();
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    CUDA_TRY(ctx, dispatch_forward_matrix(im.J, a, ctx->prop.multiProcessorCount, ctx->stream));
    const long long cells = (long long)rows * (M + 1);
    if (!scores_only) {
      fs5_export_forward_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, ctx->stream>>>(ctx->dpp.as<float>(), ctx->ddcell.as<float>(), im.zinv.as<float>(),
                                                                                          im.J, M, mpad, (long long)rows, ctx->dmxout.as<float>());
      CUDA_TRY(ctx, cudaGetLastError());
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    if (!scores_only) {
      CUDA_TRY(ctx, cudaMemcpyAsync(mx + (size_t)row0 * (M + 1) * 8, ctx->dmxout.p, (size_t)cells * 32, cudaMemcpyDeviceToHost, ctx->stream));
      CUDA_TRY(ctx, cudaMemcpyAsync(xrows + (size_t)row0 * 6, ctx->dfx.p, rows * 24, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CUDA_TRY(ctx, cudaMemcpyAsync(fwdsc + e0, ctx->dfw.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(status + e0, ctx->dstat.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
    float ms = 0.f;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->last_ms += ms; ctx->last_launches += scores_only ? 1 : 2;
    row0 += (int64_t)rows;
    e0 = e1;
  }
  ctx->dom_L.clear(); ctx->dom_xoff.clear();           // the posterior matrices of the last bathgpu_fs_domains call are gone
  return BATHGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// Profile sets: the frameshift Forward parsers over windows that each name their profile (the calibration of many models at once)
extern "C" int bathgpu_load_fs_profile_set(bathgpu_ctx *ctx, int which, int n, const int *M, const int *nrows,
                                           const float *const *rfv, const float *const *tfv)
{
  if (!ctx || n < 1 || !M || !nrows || !rfv || !tfv) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_load_fs_profile_set");
  if (which != 3 && which != 5) return fail(ctx, BATHGPU_EINVAL, "codon_lengths must be 3 or 5");
  FsProfileSet &ps = (which == 3) ? ctx->set3 : ctx->set5;
  ps.n = 0;
  // every table starts on a 256-byte boundary of the block (the kernels read them with 16-byte vector loads)
  std::vector<float> host;
  std::vector<size_t> off_emis(n), off_cc(n), off_mw(n);
  ps.J.assign(n, 0); ps.scan_steps.assign(n, 5); ps.mw_scan_steps.assign(n, 5);
  std::vector<float> tab, cc, mw;
  auto append = [&](const std::vector<float> &v) -> size_t {
    const size_t at = (host.size() + 63) & ~(size_t)63;
    host.resize(at + v.size(), 0.0f);
    std::copy(v.begin(), v.end(), host.begin() + at);
    return at;
  };
  for (int p = 0; p < n; ++p) {
    Fold f;
    const int st = fold_profile(ctx, which, M[p], nrows[p], rfv[p], tfv[p], f);
    if (st != BATHGPU_OK) return fail(ctx, st, "profile %d of the set: %s", p, std::string(ctx->err).c_str());
    if (which == 3) forward3_tables(f, 3, nrows[p], rfv[p], tab, cc, mw, ps.scan_steps[p], ps.mw_scan_steps[p]);
    else { emission_table(f, nrows[p], rfv[p], tab); fs5_forward_consts(f, cc); mw.clear(); }
    ps.J[p] = f.J;
    off_emis[p] = append(tab);
    off_cc[p] = append(cc);
    off_mw[p] = mw.empty() ? (size_t)-1 : append(mw);
  }
  CUDA_TRY(ctx, enter(ctx));
  if (ps.arena.reserve(host.size() * sizeof(float)) != BATHGPU_OK || ps.dtable.reserve((size_t)n * sizeof(FsSetProfile)) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for a set of %d profiles (%zu bytes)", n, host.size() * sizeof(float));
  CUDA_TRY(ctx, cudaMemcpyAsync(ps.arena.p, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  const float *base = ps.arena.as<float>();
  ps.table.assign(n, FsSetProfile{});
  for (int p = 0; p < n; ++p) {
    ps.table[p].emis = base + off_emis[p];
    ps.table[p].cellc = base + off_cc[p];
    ps.table[p].cellmw = (off_mw[p] == (size_t)-1) ? nullptr : base + off_mw[p];
  }
  ps.n = n;
#define X(S) preload_fwd_##S(ps.J[0]); preload_fs5_##S(ps.J[0]);
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return BATHGPU_OK;
}

static cudaError_t dispatch_fwd_set(int J, const FsParserArgs &a, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
  const int v = fwd_version(J);
#define X(S) if (launch_fs3_forward_set_##S(J, v, a, sms, s, &e)) return e;
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return cudaErrorInvalidValue;
}

static cudaError_t dispatch_fs5_set(int J, const DomainArgs &a, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
#define X(S) if (launch_fs5_forward_set_##S(J, a, sms, s, &e)) return e;
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return cudaErrorInvalidValue;
}

extern "C" int bathgpu_fs_set_scores(bathgpu_ctx *ctx, int which, const bathgpu_set_window *wins, int n, const float *xfE,
                                     float *fwdsc, int32_t *status)
{
  if (!ctx || !wins || n < 1 || !xfE || !fwdsc || !status) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_set_scores");
  if (which != 3 && which != 5) return fail(ctx, BATHGPU_EINVAL, "codon_lengths must be 3 or 5");
  FsProfileSet &ps = (which == 3) ? ctx->set3 : ctx->set5;
  if (ps.n < 1)              return fail(ctx, BATHGPU_EINVAL, "no %d-codon profile set loaded", which);
  if (ctx->S().block_n == 0) return fail(ctx, BATHGPU_EINVAL, "no block uploaded");
  const int minL = (which == 3) ? 3 : 6;
  for (int w = 0; w < n; ++w) {
    if (wins[w].profile < 0 || wins[w].profile >= ps.n)
      return fail(ctx, BATHGPU_EINVAL, "window %d names profile %d of a set of %d", w, wins[w].profile, ps.n);
    if (wins[w].L < minL || wins[w].start < 1 || wins[w].start + wins[w].L - 1 > ctx->S().block_n)
      return fail(ctx, BATHGPU_EINVAL, "window %d (start %lld, L %d) is outside the uploaded block (n=%lld) or shorter than %d",
                  w, (long long)wins[w].start, wins[w].L, (long long)ctx->S().block_n, minL);
  }
  CUDA_TRY(ctx, enter(ctx));
  // one launch per kernel the single-profile dispatch would pick: node count per lane J and, on the 3-codon side, the D->D scan
  // steps the kernel is instantiated for; windows of one profile stay together and in call order
  auto key = [&](int p) -> long long { return which == 3 ? ((long long)ps.J[p] * 8 + ps.scan_steps[p]) * 8 + ps.mw_scan_steps[p] : ps.J[p]; };
  std::vector<int> order(n);
  for (int w = 0; w < n; ++w) order[w] = w;
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
    const int px = wins[x].profile, py = wins[y].profile;
    const long long kx = key(px), ky = key(py);
    return kx != ky ? kx < ky : px < py;
  });
  static_assert(sizeof(WindowDesc) == sizeof(EnvelopeDesc), "descriptor layouts must agree");
  std::vector<WindowDesc> hw(n);
  std::vector<int> hp(n), grp;
  for (int z = 0; z < n; ++z) {
    const bathgpu_set_window &sw = wins[order[z]];
    hw[z].start = sw.start; hw[z].L = sw.L; hw[z].pmove = sw.pmove; hw[z].ploop = sw.ploop;
    hp[z] = sw.profile;
    if (z == 0 || key(hp[z]) != key(hp[z - 1])) grp.push_back(z);
  }
  const int ng = (int)grp.size();
  grp.push_back(n);
  std::vector<FsSetProfile> table(ps.table);
  for (int p = 0; p < ps.n; ++p) { table[p].tEM = xfE[2 * p]; table[p].tEL = xfE[2 * p + 1]; }
  if (ps.dwins.reserve((size_t)n * sizeof(WindowDesc)) != BATHGPU_OK || ps.dwprof.reserve((size_t)n * 4) != BATHGPU_OK ||
      ps.dsc.reserve((size_t)n * 4) != BATHGPU_OK || ps.dst.reserve((size_t)n * 4) != BATHGPU_OK ||
      ps.dcounter.reserve((size_t)ng * 4) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  CUDA_TRY(ctx, cudaMemcpyAsync(ps.dwins.p, hw.data(), (size_t)n * sizeof(WindowDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ps.dwprof.p, hp.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ps.dtable.p, table.data(), (size_t)ps.n * sizeof(FsSetProfile), cudaMemcpyHostToDevice, ctx->stream));
  if (which == 5) {
    // The 5-codon kernel writes every row of its matrix (rows nobody reads here): windows take turns in a ring of scratch matrices
    // as large as the matrix budget allows; two windows that share a slot at the same time only overwrite each other's unread rows.
    int maxL = 0, maxJ = 0;
    for (int z = 0; z < n; ++z) { maxL = std::max(maxL, hw[z].L); maxJ = std::max(maxJ, ps.J[hp[z]]); }
    const size_t rows_per = (size_t)maxL + 1, mpad = (size_t)32 * maxJ;
    const size_t slots = std::max<size_t>(1, std::min<size_t>((size_t)n, matrix_budget() / 10 * 7 / (rows_per * kPPCells * mpad * 4)));
    const size_t rows = slots * rows_per;
    std::vector<long long> xo(n);
    for (int z = 0; z < n; ++z) xo[z] = (long long)((size_t)z % slots * rows_per);
    if (ctx->xoff.reserve((size_t)n * 8) != BATHGPU_OK || reserve_matrices(ctx, rows * kPPCells * mpad * 4, 0) != BATHGPU_OK ||
        ctx->ddcell.reserve(rows * mpad * 4) != BATHGPU_OK || ctx->dfx.reserve(rows * 24) != BATHGPU_OK || ctx->dlsf.reserve(rows * 4) != BATHGPU_OK)
      return fail(ctx, BATHGPU_EMEM, "device allocation failed");
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->xoff.p, xo.data(), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
  }
  CUDA_TRY(ctx, cudaMemsetAsync(ps.dcounter.p, 0, (size_t)ng * 4, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  const int sms = ctx->prop.multiProcessorCount;
  for (int g = 0; g < ng; ++g) {
    const int b = grp[g], e = grp[g + 1], p0 = hp[b], J = ps.J[p0];
    if (which == 3) {
      FsParserArgs a{};
      a.dna4 = ctx->S().dna4.as<uint32_t>(); a.wins = ps.dwins.as<WindowDesc>() + b; a.nwin = e - b; a.mpad = 32 * J;
      a.fwdsc = ps.dsc.as<float>() + b; a.status = ps.dst.as<int>() + b; a.counter = ps.dcounter.as<int>() + g;
      a.scan_steps = ps.scan_steps[p0]; a.mw_scan_steps = ps.mw_scan_steps[p0]; a.cellmw = table[p0].cellmw;
      a.set = ps.dtable.as<FsSetProfile>(); a.wprof = ps.dwprof.as<int>() + b;
      CUDA_TRY(ctx, dispatch_fwd_set(J, a, sms, ctx->stream));
    } else {
      DomainArgs a{};
      a.dna4 = ctx->S().dna4.as<uint32_t>(); a.envs = ps.dwins.as<EnvelopeDesc>() + b; a.nenv = e - b; a.mpad = 32 * J;
      a.fwdsc = ps.dsc.as<float>() + b; a.status = ps.dst.as<int>() + b; a.counter = ps.dcounter.as<int>() + g;
      a.set = ps.dtable.as<FsSetProfile>(); a.wprof = ps.dwprof.as<int>() + b;
      a.xoff = ctx->xoff.as<long long>() + b; a.pp = ctx->dpp.as<float>(); a.dcell = ctx->ddcell.as<float>(); a.fx = ctx->dfx.as<float>();
      a.lsf = ctx->dlsf.as<float>();
      CUDA_TRY(ctx, dispatch_fs5_set(J, a, sms, ctx->stream));
    }
  }
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  std::vector<float> sc(n);
  std::vector<int> st(n);
  CUDA_TRY(ctx, cudaMemcpyAsync(sc.data(), ps.dsc.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(st.data(), ps.dst.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  for (int z = 0; z < n; ++z) { fwdsc[order[z]] = sc[z]; status[order[z]] = st[z]; }
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
  ctx->last_launches = ng;
  if (which == 5) { ctx->dom_L.clear(); ctx->dom_xoff.clear(); }        // the posterior matrices of the last bathgpu_fs_domains call are gone
  return BATHGPU_OK;
}

// Test/diagnostic access to the matrices of envelope e of the LAST chunk of the last bathgpu_fs_domains call,
// un-permuted: pp [(L+1)][(M+1)][8] in the reference's cell order {D,I,C0..C5} (impl_sse.h:296-314; D = 0),
// oa [(L+1)][(M+1)][3] {M,D,I}, ppx / oax [(L+1)][6].
extern "C" int bathgpu_fs_fetch_domain_matrices(bathgpu_ctx *ctx, int e, float *pp, float *oa, float *ppx, float *oax)
{
  if (!ctx || e < 0 || e >= (int)ctx->dom_L.size()) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fs_fetch_domain_matrices");
  CUDA_TRY(ctx, enter(ctx));
  const FsProfileImage &im = ctx->fs5;
  const int M = im.M, mpad = im.mpad, J = im.J, L = ctx->dom_L[e];
  const size_t r0 = (size_t)ctx->dom_xoff[e], nr = (size_t)L + 1;
  std::vector<float> hp(nr * kPPCells * mpad), ho(nr * kOACells * mpad);
  CUDA_TRY(ctx, cudaMemcpy(hp.data(), ctx->dpp.as<float>() + r0 * kPPCells * mpad, hp.size() * 4, cudaMemcpyDeviceToHost));
  CUDA_TRY(ctx, cudaMemcpy(ho.data(), ctx->doa.as<float>() + r0 * kOACells * mpad, ho.size() * 4, cudaMemcpyDeviceToHost));
  if (ppx) CUDA_TRY(ctx, cudaMemcpy(ppx, ctx->dppx.as<float>() + r0 * 6, nr * 24, cudaMemcpyDeviceToHost));
  if (oax) CUDA_TRY(ctx, cudaMemcpy(oax, ctx->doax.as<float>() + r0 * 6, nr * 24, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < nr; ++i)
    for (int k = 0; k <= M; ++k) {
      float *pc = pp ? pp + (i * (M + 1) + k) * 8 : nullptr;
      float *oc = oa ? oa + (i * (M + 1) + k) * 3 : nullptr;
      if (k == 0) {
        if (pc) for (int c = 0; c < 8; ++c) pc[c] = 0.f;
        if (oc) for (int c = 0; c < 3; ++c) oc[c] = -INFINITY;
        continue;
      }
      const int p = perm_index(k - 1, J);
      if (pc) {
        pc[0] = 0.f;
        pc[1] = hp[(i * kPPCells + PP_I) * mpad + p];
        for (int c = 0; c < 6; ++c) pc[2 + c] = hp[(i * kPPCells + PP_C0 + c) * mpad + p];
      }
      if (oc) {
        oc[0] = ho[(i * kOACells + OA_M) * mpad + p];
        oc[1] = ho[(i * kOACells + OA_D) * mpad + p];
        oc[2] = ho[(i * kOACells + OA_I) * mpad + p];
      }
    }
  return BATHGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// ORF-stage integer filters
extern "C" int bathgpu_load_filter_profile(bathgpu_ctx *ctx, const bathgpu_filter_params *prm,
                                           const uint8_t *rbv, const int16_t *rwv, const int16_t *twv)
{
  if (!ctx || !prm || !rbv || !rwv || !twv || prm->M < 1) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_load_filter_profile");
  const int M = prm->M, ld = M + 1;
  if (M > 1024) return fail(ctx, BATHGPU_EINVAL, "model length %d exceeds the single-warp kernels' limit (1024)", M);
  if (prm->cpu_lanes_u8 < 1 || prm->cpu_lanes_i16 < 1) return fail(ctx, BATHGPU_EINVAL, "cpu lane counts must be positive");
  CUDA_TRY(ctx, enter(ctx));
  ctx->flt_loaded = false;
  ctx->flt = *prm;
  int W = (M + 127) / 128, P = (M + 63) / 64;
  if (W == 5) W = 6; else if (W == 7) W = 8;             // instantiated widths (launch.h)
  if (P > 6) P = (P <= 8) ? 8 : (P <= 12) ? 12 : 16;
  ctx->flt_W = W; ctx->flt_P = P;
  const int nb = 128 * W, nw = 64 * P;                 // nodes per padded row
  std::vector<uint8_t> hb((size_t)29 * nb, 255);
  std::vector<int16_t> hw((size_t)29 * nw, -32768), ht((size_t)8 * nw, -32768), hn((size_t)29 * nw, -255);
  for (int x = 0; x < 29; ++x)
    for (int k = 1; k <= M; ++k) {
      hb[(size_t)x * nb + (k - 1)] = rbv[(size_t)x * ld + k];
      hw[(size_t)x * nw + (k - 1)] = rwv[(size_t)x * ld + k];
      hn[(size_t)x * nw + (k - 1)] = (int16_t)(-(int)rbv[(size_t)x * ld + k]);
    }
  for (int t = 0; t < 8; ++t)
    for (int k = 1; k <= M; ++k) {
      // BM,MM,IM,DM act on the way INTO node k: source node k-1; the others are taken at node k itself
      const int src = (t < 4) ? k - 1 : k;
      ht[(size_t)t * nw + (k - 1)] = twv[(size_t)t * ld + src];
    }
  // lane constants of the D->D closure scan (orf_filters.cuh): nodes per lane = 2P
  std::vector<int> dds((size_t)6 * 32, 0);
  {
    const int n = 2 * P;
    auto tDD = [&](int k) -> long long { return (k >= 1 && k <= M) ? (long long)twv[(size_t)7 * ld + k] : -32768LL; };
    std::vector<long long> T0(32, 0);
    for (int lane = 0; lane < 32; ++lane) {
      const int first = lane * n + 1;                  // first node of the lane
      long long t = (lane > 0) ? tDD(first - 1) : 0;
      for (int j = 0; j + 1 < n; ++j) t += tDD(first + j);
      T0[lane] = t;
      dds[(size_t)5 * 32 + lane] = (lane > 0) ? (int)tDD(first - 1) : 0;
    }
    std::vector<long long> cur(T0);
    for (int s = 0; s < 5; ++s) {
      const int d = 1 << s;
      std::vector<long long> nx(cur);
      for (int lane = 0; lane < 32; ++lane) {
        dds[(size_t)s * 32 + lane] = (int)std::max(cur[lane], -(1LL << 28));
        if (lane >= d) nx[lane] = cur[lane] + cur[lane - d];
      }
      cur.swap(nx);
    }
  }
  if (ctx->f_rbv.reserve(hb.size()) != BATHGPU_OK || ctx->f_rwv.reserve(hw.size() * 2) != BATHGPU_OK ||
      ctx->f_twv.reserve(ht.size() * 2) != BATHGPU_OK || ctx->f_ddsum.reserve(dds.size() * 4) != BATHGPU_OK || ctx->f_nrb.reserve(hn.size() * 2) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->f_rbv.p, hb.data(), hb.size(), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->f_rwv.p, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->f_nrb.p, hn.data(), hn.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->f_twv.p, ht.data(), ht.size() * 2, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->f_ddsum.p, dds.data(), dds.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  ctx->flt_loaded = true;
  preload_msv_filter(W, P); preload_vit_filter_lo(P); preload_vit_filter_hi(P);
  return BATHGPU_OK;
}

extern "C" int bathgpu_upload_orfs(bathgpu_ctx *ctx, const uint8_t *residues, int64_t n)
{
  if (!ctx || !residues || n < 1) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_upload_orfs");
  CUDA_TRY(ctx, enter(ctx));
  if (ctx->S().residues.reserve((size_t)n + 64) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->S().residues.p, residues, (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  ctx->S().nres = n;
  return BATHGPU_OK;
}

static int stage_orfs(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, int max_wins)
{
  if (!ctx->flt_loaded) return fail(ctx, BATHGPU_EINVAL, "filter profile not loaded");
  if (ctx->S().nres == 0)   return fail(ctx, BATHGPU_EINVAL, "no ORF residues uploaded");
  for (int o = 0; o < n; ++o)
    if (orfs[o].L < 1 || orfs[o].offset < 0 || orfs[o].offset + orfs[o].L > ctx->S().nres)
      return fail(ctx, BATHGPU_EINVAL, "ORF %d (offset %lld, L %d) is outside the uploaded residues (n=%lld)",
                  o, (long long)orfs[o].offset, orfs[o].L, (long long)ctx->S().nres);
  static_assert(sizeof(OrfDesc) == sizeof(bathgpu_orf), "descriptor layouts must agree");
  static_assert(sizeof(WindowRec) == sizeof(bathgpu_orf_window), "window layouts must agree");
  if (ctx->orfs.reserve((size_t)n * sizeof(OrfDesc)) != BATHGPU_OK || ctx->fsc.reserve((size_t)n * 4) != BATHGPU_OK ||
      ctx->fst.reserve((size_t)n * 4) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK || ctx->fnw.reserve(64) != BATHGPU_OK ||
      ctx->fwins.reserve((size_t)std::max(max_wins, 1) * sizeof(WindowRec)) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->orfs.p, orfs, (size_t)n * sizeof(OrfDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, 4, ctx->stream));
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->fnw.p, 0, 4, ctx->stream));
  return BATHGPU_OK;
}

static FilterArgs filter_args(bathgpu_ctx *ctx, int n, int max_wins)
{
  FilterArgs a{};
  const bathgpu_filter_params &p = ctx->flt;
  a.residues = ctx->S().residues.as<uint8_t>(); a.res_stride = 1; a.orfs = ctx->orfs.as<OrfDesc>(); a.norf = n; a.M = p.M;
  a.rbv = ctx->f_rbv.as<uint32_t>(); a.nrb = ctx->f_nrb.as<uint32_t>(); a.rbv_bytes = ctx->f_rbv.as<uint8_t>(); a.rowwords_b = 32 * ctx->flt_W;
  a.tbm_b = p.tbm_b; a.tec_b = p.tec_b; a.base_b = p.base_b; a.bias_b = p.bias_b; a.scale_b = p.scale_b;
  a.rwv = ctx->f_rwv.as<uint32_t>(); a.twv = ctx->f_twv.as<uint32_t>(); a.ddsum = ctx->f_ddsum.as<int>(); a.rowwords_w = 32 * ctx->flt_P;
  a.base_w = p.base_w; a.ddbound_w = p.ddbound_w; a.xw_E_move = p.xw_E_move; a.xw_E_loop = p.xw_E_loop; a.scale_w = p.scale_w;
  a.lanes_u8 = p.cpu_lanes_u8; a.lanes_i16 = p.cpu_lanes_i16;
  a.sc = ctx->fsc.as<float>(); a.status = ctx->fst.as<int>(); a.wins = ctx->fwins.as<WindowRec>(); a.nwins = ctx->fnw.as<int>();
  a.max_wins = max_wins; a.counter = ctx->counter.as<int>();
  return a;
}

static cudaError_t dispatch_msv(int mode, int W, const FilterArgs &a, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
  return launch_msv_filter(W, a.rowwords_w / 32, mode, a, sms, s, &e) ? e : cudaErrorInvalidValue;
}

static cudaError_t dispatch_vit(int P, const FilterArgs &a, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
  return (launch_vit_filter_lo(P, a, sms, s, &e) || launch_vit_filter_hi(P, a, sms, s, &e)) ? e : cudaErrorInvalidValue;
}

static int fetch_windows(bathgpu_ctx *ctx, bathgpu_orf_window *wins, int max_wins, int *nwins)
{
  int nw = 0;
  CUDA_TRY(ctx, cudaMemcpyAsync(&nw, ctx->fnw.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  if (nw > max_wins) return fail(ctx, BATHGPU_EINVAL, "window buffer too small: %d windows found, room for %d", nw, max_wins);
  if (nw > 0) {
    CUDA_TRY(ctx, cudaMemcpyAsync(wins, ctx->fwins.p, (size_t)nw * sizeof(WindowRec), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
    // the reference appends windows ORF by ORF in target order (src/p7_pipeline.c:1669-1680)
    std::sort(wins, wins + nw, [](const bathgpu_orf_window &x, const bathgpu_orf_window &y) {
      return x.orf != y.orf ? x.orf < y.orf : x.n < y.n; });
  }
  *nwins = nw;
  return BATHGPU_OK;
}

static int finish_filter(bathgpu_ctx *ctx, int n, float *sc, int32_t *status, int launches)
{
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  if (sc)     CUDA_TRY(ctx, cudaMemcpyAsync(sc, ctx->fsc.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (status) CUDA_TRY(ctx, cudaMemcpyAsync(status, ctx->fst.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
  ctx->last_launches = launches;
  return BATHGPU_OK;
}

extern "C" int bathgpu_msv_orfs(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, float *sc, int32_t *status)
{
  if (!ctx || !orfs || n < 1 || !sc || !status) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_msv_orfs");
  CUDA_TRY(ctx, enter(ctx));
  int st = stage_orfs(ctx, orfs, n, 0);
  if (st != BATHGPU_OK) return st;
  FilterArgs a = filter_args(ctx, n, 0);
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  CUDA_TRY(ctx, dispatch_msv(0, ctx->flt_W, a, ctx->prop.multiProcessorCount, ctx->stream));
  return finish_filter(ctx, n, sc, status, 1);
}

extern "C" int bathgpu_ssv_windows(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, bathgpu_orf_window *wins, int max_wins, int *nwins)
{
  if (!ctx || !orfs || n < 1 || !wins || max_wins < 1 || !nwins) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_ssv_windows");
  CUDA_TRY(ctx, enter(ctx));
  int st = stage_orfs(ctx, orfs, n, max_wins);
  if (st != BATHGPU_OK) return st;
  FilterArgs a = filter_args(ctx, n, max_wins);
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  CUDA_TRY(ctx, dispatch_msv(1, ctx->flt_W, a, ctx->prop.multiProcessorCount, ctx->stream));
  if ((st = finish_filter(ctx, n, nullptr, nullptr, 1)) != BATHGPU_OK) return st;
  return fetch_windows(ctx, wins, max_wins, nwins);
}

extern "C" int bathgpu_vit_orfs(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, float *sc, int32_t *status,
                                bathgpu_orf_window *wins, int max_wins, int *nwins)
{
  if (!ctx || !orfs || n < 1 || !sc || !status) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_vit_orfs");
  bool any = false;
  for (int o = 0; o < n; ++o) any = any || (orfs[o].flags & 1);
  if (any && (!wins || max_wins < 1 || !nwins)) return fail(ctx, BATHGPU_EINVAL, "window output buffers are required when any ORF asks for windows");
  CUDA_TRY(ctx, enter(ctx));
  int st = stage_orfs(ctx, orfs, n, any ? max_wins : 0);
  if (st != BATHGPU_OK) return st;
  FilterArgs a = filter_args(ctx, n, any ? max_wins : 0);
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  CUDA_TRY(ctx, dispatch_vit(ctx->flt_P, a, ctx->prop.multiProcessorCount, ctx->stream));
  if ((st = finish_filter(ctx, n, sc, status, 1)) != BATHGPU_OK) return st;
  if (nwins) *nwins = 0;
  if (any) return fetch_windows(ctx, wins, max_wins, nwins);
  return BATHGPU_OK;
}

extern "C" int bathgpu_fwd_orfs(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, float nj, const float xfE[2], float *fwdsc, int32_t *status)
{
  if (!ctx || !orfs || n < 1 || !xfE || !fwdsc || !status) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_fwd_orfs");
  if (!ctx->fs3.loaded) return fail(ctx, BATHGPU_EINVAL, "3-codon profile not loaded");
  if (ctx->S().nres == 0)   return fail(ctx, BATHGPU_EINVAL, "no ORF residues uploaded");
  for (int o = 0; o < n; ++o)
    if (orfs[o].L < 1 || orfs[o].offset < 0 || orfs[o].offset + orfs[o].L > ctx->S().nres)
      return fail(ctx, BATHGPU_EINVAL, "ORF %d is outside the uploaded residues", o);
  CUDA_TRY(ctx, enter(ctx));
  if (ctx->orfs.reserve((size_t)n * sizeof(OrfDesc)) != BATHGPU_OK || ctx->fsc.reserve((size_t)n * 4) != BATHGPU_OK ||
      ctx->fst.reserve((size_t)n * 4) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->orfs.p, orfs, (size_t)n * sizeof(OrfDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, 4, ctx->stream));
  const FsProfileImage &im = ctx->fs3;
  OrfFwdArgs a{};
  a.emis = im.emis_fwd.as<float>(); a.cellc = im.cellc.as<float>(); a.residues = ctx->S().residues.as<uint8_t>();
  a.orfs = ctx->orfs.p; a.orf_stride = (int)sizeof(OrfDesc); a.norf = n; a.mpad = im.mpad; a.nj = nj;
  a.tEM = xfE[0]; a.tEL = xfE[1]; a.fwdsc = ctx->fsc.as<float>(); a.status = ctx->fst.as<int>(); a.counter = ctx->counter.as<int>();
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  const int sms = ctx->prop.multiProcessorCount;
  cudaError_t e = cudaErrorInvalidValue;
  bool found = false;
#define X(S) if (!found) found = launch_orf_forward_parser_##S(im.J, a, sms, ctx->stream, &e);
  BATHGPU_FOR_EACH_SET(X)
#undef X
  if (!found) e = cudaErrorInvalidValue;
  CUDA_TRY(ctx, e);
  return finish_filter(ctx, n, fwdsc, status, 1);
}

// ---------------------------------------------------------------------------------------------
// Standard-translation branch: protein Forward/Backward over ORFs and the per-envelope domain stage (orf_domain.cuh)
static cudaError_t dispatch_orf_domains(int J, bool full, const OrfDomainArgs &a, const TraceArgs &t, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
#define X(S) if (launch_orf_domains_##S(J, full, a, t, sms, s, &e)) return e;
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return cudaErrorInvalidValue;
}

static const FsProfileImage *orf_image(bathgpu_ctx *ctx) { return ctx->fs3.loaded ? &ctx->fs3 : (ctx->fs5.loaded ? &ctx->fs5 : nullptr); }

// One chunk of ORFs / envelopes.  full == false: X rows of both parsers to the host; full == true: results + traces.
static int orf_chunk(bathgpu_ctx *ctx, const EnvelopeDesc *envs, int n, const float xfE[2], bool full,
                     float *fwd_xrows, float *bck_xrows, float *fwdsc, float *bcksc, int32_t *status, int64_t x_off0,
                     bathgpu_domain_result *results, bathgpu_trace_step *traces, int64_t max_steps, int64_t *steps_used)
{
  const FsProfileImage &im = *orf_image(ctx);
  const int M = im.M, mpad = im.mpad;
  std::vector<long long> xoff(n + 1, 0), toff(n + 1, 0);
  for (int e = 0; e < n; ++e) { xoff[e + 1] = xoff[e] + envs[e].L + 1; toff[e + 1] = toff[e] + envs[e].L + M + 8; }
  const size_t rows = (size_t)xoff[n];
  if (ctx->envs.reserve((size_t)n * sizeof(EnvelopeDesc)) != BATHGPU_OK || ctx->xoff.reserve((size_t)(n + 1) * 8) != BATHGPU_OK ||
      ctx->dfx.reserve(rows * 24) != BATHGPU_OK || ctx->bxmx.reserve(rows * 24) != BATHGPU_OK || ctx->dlsf.reserve(rows * 4) != BATHGPU_OK ||
      ctx->dfw.reserve((size_t)n * 4) != BATHGPU_OK || ctx->dbk.reserve((size_t)n * 4) != BATHGPU_OK ||
      ctx->dstat.reserve((size_t)n * 4) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for %d ORFs (%zu rows)", n, rows);
  if (full && (ctx->dtoff.reserve((size_t)(n + 1) * 8) != BATHGPU_OK || ctx->dtlen.reserve((size_t)n * 4) != BATHGPU_OK ||
               reserve_matrices(ctx, rows * kPPCellsP * mpad * 4, rows * kOACells * mpad * 4) != BATHGPU_OK ||
               ctx->dppx.reserve(rows * 24) != BATHGPU_OK || ctx->doax.reserve(rows * 24) != BATHGPU_OK ||
               ctx->doasc.reserve((size_t)n * 4) != BATHGPU_OK || ctx->dnull2.reserve((size_t)n * 29 * 4) != BATHGPU_OK ||
               ctx->dsteps.reserve((size_t)toff[n] * sizeof(TraceStep)) != BATHGPU_OK))
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for %d envelopes (%zu rows, M=%d)", n, rows, M);
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->envs.p, envs, (size_t)n * sizeof(EnvelopeDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->xoff.p, xoff.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  if (full) CUDA_TRY(ctx, cudaMemcpyAsync(ctx->dtoff.p, toff.data(), (size_t)(n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));

  OrfDomainArgs a{};
  a.emis = im.emis.as<float>(); a.amino0 = im.nrows - BATHGPU_KP; a.amino = im.amino.as<float>();
  a.cellf = im.cellf5.as<float>(); a.cellb = im.cellb.as<float>(); a.oapass = im.oapass.as<float>(); a.oaflags = im.oaflags.as<uint32_t>();
  a.residues = ctx->S().residues.as<uint8_t>(); a.envs = ctx->envs.as<EnvelopeDesc>(); a.nenv = n; a.M = M; a.mpad = mpad;
  a.tEM = xfE[0]; a.tEL = xfE[1]; a.xoff = ctx->xoff.as<long long>();
  a.pp = ctx->dpp.as<float>(); a.oa = ctx->doa.as<float>(); a.fx = ctx->dfx.as<float>(); a.bx = ctx->bxmx.as<float>();
  a.ppx = ctx->dppx.as<float>(); a.oax = ctx->doax.as<float>(); a.lsf = ctx->dlsf.as<float>();
  a.fwdsc = ctx->dfw.as<float>(); a.bcksc = ctx->dbk.as<float>(); a.oasc = ctx->doasc.as<float>();
  a.null2 = ctx->dnull2.as<float>(); a.status = ctx->dstat.as<int>(); a.counter = ctx->counter.as<int>();
  a.lanes_f32 = ctx->flt_loaded ? std::max(1, ctx->flt.cpu_lanes_u8 / 4) : 4;
  TraceArgs t{};
  t.steps = ctx->dsteps.as<TraceStep>(); t.toff = ctx->dtoff.as<long long>(); t.tlen = ctx->dtlen.as<int>();
  t.tfv = im.tfvraw.as<float>(); t.J = im.J;

  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  CUDA_TRY(ctx, dispatch_orf_domains(im.J, full, a, t, ctx->prop.multiProcessorCount, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));

  std::vector<float> fw(n), bk(n);
  std::vector<int> st(n);
  CUDA_TRY(ctx, cudaMemcpyAsync(fw.data(), ctx->dfw.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(bk.data(), ctx->dbk.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(st.data(), ctx->dstat.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  if (!full) {
    CUDA_TRY(ctx, cudaMemcpyAsync(fwd_xrows + (size_t)x_off0 * 6, ctx->dfx.p, rows * 24, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(bck_xrows + (size_t)x_off0 * 6, ctx->bxmx.p, rows * 24, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
    float ms = 0.f;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->last_ms += ms; ctx->last_launches += 2;
    for (int e = 0; e < n; ++e) { if (fwdsc) fwdsc[e] = fw[e]; if (bcksc) bcksc[e] = bk[e]; status[e] = st[e]; }
    return BATHGPU_OK;
  }
  std::vector<float> oa(n), n2((size_t)n * 29);
  std::vector<int> tl(n);
  std::vector<TraceStep> steps((size_t)toff[n]);
  CUDA_TRY(ctx, cudaMemcpyAsync(oa.data(), ctx->doasc.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(n2.data(), ctx->dnull2.p, (size_t)n * 29 * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(tl.data(), ctx->dtlen.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(steps.data(), ctx->dsteps.p, steps.size() * sizeof(TraceStep), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  float ms = 0.f;
  CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
  ctx->last_ms += ms; ctx->last_launches += 4;
  ctx->dom_xoff = xoff;
  ctx->dom_L.assign(n, 0);
  for (int e = 0; e < n; ++e) ctx->dom_L[e] = envs[e].L;
  for (int e = 0; e < n; ++e) {
    bathgpu_domain_result &r = results[e];
    r.envsc = fw[e]; r.bcksc = bk[e]; r.oasc = oa[e]; r.status = st[e];
    memcpy(r.null2, &n2[(size_t)e * 29], 29 * 4);
    r.trace_offset = (int32_t)*steps_used; r.trace_len = 0;
    if (st[e] == 0 && tl[e] > 0) {
      if (*steps_used + tl[e] > max_steps)
        return fail(ctx, BATHGPU_EINVAL, "trace buffer too small: %lld steps needed so far, %lld given", (long long)(*steps_used + tl[e]), (long long)max_steps);
      TraceStep *tr = &steps[(size_t)toff[e]];
      finish_trace(tr, tl[e]);
      memcpy(traces + *steps_used, tr, (size_t)tl[e] * sizeof(TraceStep));
      r.trace_len = tl[e];
      *steps_used += tl[e];
    }
  }
  return BATHGPU_OK;
}

extern "C" int bathgpu_orf_fwd_bck_xrows(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, float nj, const float xfE[2],
                                         float *fwd_xrows, float *bck_xrows, float *fwdsc, float *bcksc, int32_t *status)
{
  if (!ctx || !orfs || n < 1 || !xfE || !fwd_xrows || !bck_xrows || !status)
    return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_orf_fwd_bck_xrows");
  if (!orf_image(ctx))    return fail(ctx, BATHGPU_EINVAL, "no frameshift profile loaded (its amino-acid rows are the protein profile)");
  if (ctx->S().nres == 0) return fail(ctx, BATHGPU_EINVAL, "no ORF residues uploaded");
  std::vector<EnvelopeDesc> ed((size_t)n);
  for (int o = 0; o < n; ++o) {
    if (orfs[o].L < 1 || orfs[o].offset < 0 || orfs[o].offset + orfs[o].L > ctx->S().nres)
      return fail(ctx, BATHGPU_EINVAL, "ORF %d is outside the uploaded residues", o);
    ed[o].start = orfs[o].offset; ed[o].L = orfs[o].L;
    ed[o].pmove = (2.0f + nj) / ((float)orfs[o].L + 2.0f + nj);      // p7_oprofile_ReconfigRestLength (p7_oprofile.c:1312-1313)
    ed[o].ploop = 1.0f - ed[o].pmove;
  }
  CUDA_TRY(ctx, enter(ctx));
  ctx->last_ms = 0.f; ctx->last_launches = 0;
  const size_t max_rows = (size_t)16 << 20;
  int o0 = 0;
  int64_t x0 = 0;
  while (o0 < n) {
    size_t rows = 0;
    int o1 = o0;
    while (o1 < n && (o1 == o0 || rows + ed[o1].L + 1 <= max_rows)) { rows += ed[o1].L + 1; ++o1; }
    int st = orf_chunk(ctx, ed.data() + o0, o1 - o0, xfE, false, fwd_xrows, bck_xrows, fwdsc ? fwdsc + o0 : nullptr,
                       bcksc ? bcksc + o0 : nullptr, status + o0, x0, nullptr, nullptr, 0, nullptr);
    if (st != BATHGPU_OK) return st;
    x0 += (int64_t)rows;
    o0 = o1;
  }
  return BATHGPU_OK;
}

extern "C" int bathgpu_orf_domains(bathgpu_ctx *ctx, const bathgpu_envelope *envs, int n, const float xfE[2],
                                   bathgpu_domain_result *results, bathgpu_trace_step *traces, int64_t max_steps)
{
  if (!ctx || !envs || n < 1 || !xfE || !results || !traces || max_steps < 1)
    return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_orf_domains");
  if (!orf_image(ctx))    return fail(ctx, BATHGPU_EINVAL, "no frameshift profile loaded (its amino-acid rows are the protein profile)");
  if (ctx->S().nres == 0) return fail(ctx, BATHGPU_EINVAL, "no ORF residues uploaded");
  for (int e = 0; e < n; ++e)
    if (envs[e].L < 1 || envs[e].start < 0 || envs[e].start + envs[e].L > ctx->S().nres)
      return fail(ctx, BATHGPU_EINVAL, "envelope %d (offset %lld, L %d) is outside the uploaded residues (n=%lld)",
                  e, (long long)envs[e].start, envs[e].L, (long long)ctx->S().nres);
  CUDA_TRY(ctx, enter(ctx));
  ctx->last_ms = 0.f; ctx->last_launches = 0;
  const size_t row_bytes = (size_t)kOACells * orf_image(ctx)->mpad * 4 / 3 * 10;      // the optimal-accuracy cells have 3/10 of the workspace
  const size_t max_rows = std::max<size_t>(matrix_budget() / row_bytes - 1, 4096);
  int64_t steps_used = 0;
  int e0 = 0;
  while (e0 < n) {
    size_t rows = 0;
    int e1 = e0;
    while (e1 < n && (e1 == e0 || rows + envs[e1].L + 1 <= max_rows)) { rows += envs[e1].L + 1; ++e1; }
    int st = orf_chunk(ctx, reinterpret_cast<const EnvelopeDesc *>(envs) + e0, e1 - e0, xfE, true, nullptr, nullptr, nullptr, nullptr, nullptr, 0,
                       results + e0, traces, max_steps, &steps_used);
    if (st != BATHGPU_OK) return st;
    e0 = e1;
  }
  return BATHGPU_OK;
}

// ---- f2, multi-domain regions of the standard branch: p7_Forward over a region of an ORF with the whole matrix handed back
static cudaError_t dispatch_orf_forward_matrix(int J, const OrfDomainArgs &a, int sms, cudaStream_t s)
{
  cudaError_t e = cudaErrorInvalidValue;
#define X(S) if (launch_orf_forward_matrix_##S(J, a, sms, s, &e)) return e;
  BATHGPU_FOR_EACH_SET(X)
#undef X
  return cudaErrorInvalidValue;
}

// stored cells -> out[(row (M+1) + k) 4 + {M, D, I, 0}] (P7_OMX cell order p7X_M, p7X_D, p7X_I; src/impl_sse/impl_sse.h:296-314,
// un-striped); match cells are stored times Z(k) and divided back here
__global__ void orf_export_forward_kernel(const float *__restrict__ pp, const float *__restrict__ dcell, const float *__restrict__ zinv,
                                          int J, int M, int mpad, long long rows, float *__restrict__ out)
{
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * (M + 1)) return;
  const long long row = t / (M + 1);
  const int k = (int)(t - row * (M + 1));
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (k > 0) {
    const int VEC = (J % 4 == 0) ? 4 : ((J % 2 == 0) ? 2 : 1);
    const int kk = k - 1, lane = kk / J, j = kk % J;
    const int p = (j / VEC) * (32 * VEC) + lane * VEC + (j % VEC);
    const float *r = pp + (size_t)row * kPPCellsP * mpad + p;
    c.x = r[(size_t)PPP_M * mpad] * zinv[kk];
    c.y = dcell[(size_t)row * mpad + p];
    c.z = r[(size_t)PPP_I * mpad];
  }
  reinterpret_cast<float4 *>(out)[t] = c;
}

extern "C" int bathgpu_orf_forward_matrices(bathgpu_ctx *ctx, const bathgpu_envelope *regs, int n, const float xfE[2],
                                            float *mx, float *xrows, int64_t max_rows, float *fwdsc, int32_t *status)
{
  if (!ctx || !regs || n < 1 || !xfE || !mx || !xrows || !fwdsc || !status) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_orf_forward_matrices");
  if (!orf_image(ctx))    return fail(ctx, BATHGPU_EINVAL, "no frameshift profile loaded (its amino-acid rows are the protein profile)");
  if (ctx->S().nres == 0) return fail(ctx, BATHGPU_EINVAL, "no ORF residues uploaded");
  int64_t total = 0;
  for (int e = 0; e < n; ++e) {
    if (regs[e].L < 1 || regs[e].start < 0 || regs[e].start + regs[e].L > ctx->S().nres)
      return fail(ctx, BATHGPU_EINVAL, "region %d (offset %lld, L %d) is outside the uploaded residues (n=%lld)", e, (long long)regs[e].start, regs[e].L,
                  (long long)ctx->S().nres);
    total += regs[e].L + 1;
  }
  if (total > max_rows) return fail(ctx, BATHGPU_EINVAL, "matrix buffer too small: %lld rows needed, %lld given", (long long)total, (long long)max_rows);
  CUDA_TRY(ctx, enter(ctx));
  const FsProfileImage &im = *orf_image(ctx);
  const int M = im.M, mpad = im.mpad;
  ctx->last_ms = 0.f; ctx->last_launches = 0;
  const size_t cap_rows = std::max<size_t>(matrix_budget() / 10 * 7 / ((size_t)kPPCellsP * mpad * 4) / 2, 8192);
  int e0 = 0;
  int64_t row0 = 0;
  while (e0 < n) {
    int e1 = e0;
    size_t rows = 0;
    while (e1 < n && (e1 == e0 || rows + regs[e1].L + 1 <= cap_rows)) { rows += regs[e1].L + 1; ++e1; }
    const int m = e1 - e0;
    std::vector<long long> xoff(m + 1, 0);
    for (int e = 0; e < m; ++e) xoff[e + 1] = xoff[e] + regs[e0 + e].L + 1;
    if (ctx->envs.reserve((size_t)m * sizeof(EnvelopeDesc)) != BATHGPU_OK || ctx->xoff.reserve((size_t)(m + 1) * 8) != BATHGPU_OK ||
        reserve_matrices(ctx, rows * kPPCellsP * mpad * 4, 0) != BATHGPU_OK || ctx->ddcell.reserve(rows * mpad * 4) != BATHGPU_OK ||
        ctx->dmxout.reserve(rows * (size_t)(M + 1) * 16) != BATHGPU_OK || ctx->dfx.reserve(rows * 24) != BATHGPU_OK ||
        ctx->dlsf.reserve(rows * 4) != BATHGPU_OK || ctx->dfw.reserve((size_t)m * 4) != BATHGPU_OK || ctx->doasc.reserve((size_t)m * 4) != BATHGPU_OK ||
        ctx->dstat.reserve((size_t)m * 4) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK)
      return fail(ctx, BATHGPU_EMEM, "device allocation failed for %d regions (%zu rows, M=%d)", m, rows, M);
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->envs.p, regs + e0, (size_t)m * sizeof(EnvelopeDesc), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(ctx->xoff.p, xoff.data(), (size_t)(m + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    OrfDomainArgs a{};
    a.emis = im.emis.as<float>(); a.amino0 = im.nrows - BATHGPU_KP; a.cellf = im.cellf5.as<float>();
    a.residues = ctx->S().residues.as<uint8_t>(); a.envs = ctx->envs.as<EnvelopeDesc>(); a.nenv = m; a.M = M; a.mpad = mpad;
    a.tEM = xfE[0]; a.tEL = xfE[1]; a.xoff = ctx->xoff.as<long long>();
    a.pp = ctx->dpp.as<float>(); a.dcell = ctx->ddcell.as<float>(); a.fx = ctx->dfx.as<float>(); a.lsf = ctx->dlsf.as<float>();
    a.fwdsc = ctx->dfw.as<float>(); a.oasc = ctx->doasc.as<float>(); a.status = ctx->dstat.as<int>(); a.counter = ctx->counter.as<int>();
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    CUDA_TRY(ctx, dispatch_orf_forward_matrix(im.J, a, ctx->prop.multiProcessorCount, ctx->stream));
    const long long cells = (long long)rows * (M + 1);
    orf_export_forward_kernel<<<(unsigned)((cells + 255) / 256), 256, 0, ctx->stream>>>(ctx->dpp.as<float>(), ctx->ddcell.as<float>(), im.zinv.as<float>(),
                                                                                        im.J, M, mpad, (long long)rows, ctx->dmxout.as<float>());
    CUDA_TRY(ctx, cudaGetLastError());
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(mx + (size_t)row0 * (M + 1) * 4, ctx->dmxout.p, (size_t)cells * 16, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(xrows + (size_t)row0 * 6, ctx->dfx.p, rows * 24, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(fwdsc + e0, ctx->dfw.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(status + e0, ctx->dstat.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, wait_stream(ctx));
    float ms = 0.f;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->last_ms += ms; ctx->last_launches += 2;
    row0 += (int64_t)rows;
    e0 = e1;
  }
  return BATHGPU_OK;
}

// Test/diagnostic: matrices of envelope e of the last chunk of the last bathgpu_orf_domains call, un-permuted, in the
// reference's cell order {M,D,I}: pp and oa [(L+1)][(M+1)][3], ppx / oax [(L+1)][6].
extern "C" int bathgpu_orf_fetch_domain_matrices(bathgpu_ctx *ctx, int e, float *pp, float *oa, float *ppx, float *oax)
{
  if (!ctx || e < 0 || e >= (int)ctx->dom_L.size() || !orf_image(ctx)) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_orf_fetch_domain_matrices");
  CUDA_TRY(ctx, enter(ctx));
  const FsProfileImage &im = *orf_image(ctx);
  const int M = im.M, mpad = im.mpad, J = im.J, L = ctx->dom_L[e];
  const size_t r0 = (size_t)ctx->dom_xoff[e], nr = (size_t)L + 1;
  std::vector<float> hp(nr * kPPCellsP * mpad), ho(nr * kOACells * mpad);
  CUDA_TRY(ctx, cudaMemcpy(hp.data(), ctx->dpp.as<float>() + r0 * kPPCellsP * mpad, hp.size() * 4, cudaMemcpyDeviceToHost));
  CUDA_TRY(ctx, cudaMemcpy(ho.data(), ctx->doa.as<float>() + r0 * kOACells * mpad, ho.size() * 4, cudaMemcpyDeviceToHost));
  if (ppx) CUDA_TRY(ctx, cudaMemcpy(ppx, ctx->dppx.as<float>() + r0 * 6, nr * 24, cudaMemcpyDeviceToHost));
  if (oax) CUDA_TRY(ctx, cudaMemcpy(oax, ctx->doax.as<float>() + r0 * 6, nr * 24, cudaMemcpyDeviceToHost));
  for (size_t i = 0; i < nr; ++i)
    for (int k = 0; k <= M; ++k) {
      float *pc = pp ? pp + (i * (M + 1) + k) * 3 : nullptr;
      float *oc = oa ? oa + (i * (M + 1) + k) * 3 : nullptr;
      if (k == 0) {
        if (pc) for (int c = 0; c < 3; ++c) pc[c] = 0.f;
        if (oc) for (int c = 0; c < 3; ++c) oc[c] = -INFINITY;
        continue;
      }
      const int p = perm_index(k - 1, J);
      if (pc) { pc[0] = hp[(i * kPPCellsP + PPP_M) * mpad + p]; pc[1] = 0.f; pc[2] = hp[(i * kPPCellsP + PPP_I) * mpad + p]; }
      if (oc) { oc[0] = ho[(i * kOACells + OA_M) * mpad + p]; oc[1] = ho[(i * kOACells + OA_D) * mpad + p]; oc[2] = ho[(i * kOACells + OA_I) * mpad + p]; }
    }
  return BATHGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// a5: the bias-composition filter over ORFs or over the three frames of DNA windows (bias_filter.cuh)
extern "C" int bathgpu_bias_forward(bathgpu_ctx *ctx, int kind, const bathgpu_bias_item *items, int n, const float *tables, int ntab,
                                    float t10, float t11, const uint8_t gcode[64], float *out)
{
  if (!ctx || (kind != 0 && kind != 1) || !items || n < 1 || !tables || ntab < 1 || !out || (kind == 1 && !gcode))
    return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_bias_forward");
  TargetSlot &S = ctx->S();
  static_assert(sizeof(BiasItem) == sizeof(bathgpu_bias_item), "item layouts must agree");
  for (int i = 0; i < n; ++i) {
    const bathgpu_bias_item &d = items[i];
    if (d.table < 0 || d.table >= ntab || d.L < 0) return fail(ctx, BATHGPU_EINVAL, "bias item %d: table %d of %d, L %d", i, d.table, ntab, d.L);
    if (kind == 0 ? (d.start < 0 || d.start + d.L > S.nres) : (d.start < 1 || d.start + d.L - 1 > S.block_n))
      return fail(ctx, BATHGPU_EINVAL, "bias item %d (start %lld, L %d) is outside the resident %s", i, (long long)d.start, d.L, kind == 0 ? "residues" : "sequence");
  }
  CUDA_TRY(ctx, enter(ctx));
  const int per = (kind == 1) ? 3 : 1;
  if (ctx->b_items.reserve((size_t)n * sizeof(BiasItem)) != BATHGPU_OK || ctx->b_tables.reserve((size_t)ntab * 58 * 4) != BATHGPU_OK ||
      ctx->b_out.reserve((size_t)n * per * 4) != BATHGPU_OK) return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->b_items.p, items, (size_t)n * sizeof(BiasItem), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->b_tables.p, tables, (size_t)ntab * 58 * 4, cudaMemcpyHostToDevice, ctx->stream));
  BiasArgs a{};
  a.items = ctx->b_items.as<BiasItem>(); a.n = n; a.kind = kind; a.tables = ctx->b_tables.as<float>(); a.t10 = t10; a.t11 = t11;
  a.residues = S.residues.as<uint8_t>(); a.dna4 = S.dna4.as<uint32_t>(); a.out = ctx->b_out.as<float>();
  if (gcode) memcpy(a.gcode, gcode, 64);
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  const long long nthreads = (long long)n * per * 32;           // a warp per item
  bias_forward_kernel<<<(unsigned)((nthreads + 127) / 128), 128, 0, ctx->stream>>>(a);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->b_out.p, (size_t)n * per * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
  ctx->last_launches = 1;
  return BATHGPU_OK;
}

// ---------------------------------------------------------------------------------------------
// f1: ORFs of every block of the resident strand found on the device, MSV over all of them, F1 screen (orf_finder.cuh)
extern "C" int bathgpu_orfs_msv_screen(bathgpu_ctx *ctx, const bathgpu_block *blocks, int nblocks, int complement, const uint8_t gcode[64],
                                       int min_len, const uint8_t *tjb_of, const float *null_of, int max_len, double min_bits,
                                       int64_t *norfs_per_block, int64_t *nhits, int64_t *nres)
{
  if (!ctx || !blocks || nblocks < 1 || !gcode || min_len < 1 || !tjb_of || !null_of || max_len < 1 || !nhits || !nres)
    return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_orfs_msv_screen");
  if (!ctx->flt_loaded)      return fail(ctx, BATHGPU_EINVAL, "filter profile not loaded");
  TargetSlot &S = ctx->S();
  if (S.block_n == 0)        return fail(ctx, BATHGPU_EINVAL, "no block uploaded");
  BulkScope bulk(ctx);
  static_assert(sizeof(BlockDesc) == sizeof(bathgpu_block), "block layouts must agree");
  static_assert(sizeof(OrfHit) == sizeof(bathgpu_orf_hit), "hit layouts must agree");
  std::vector<int> tile_block, tile_p0;
  std::vector<long long> first_tile((size_t)nblocks + 1, 0);
  for (int b = 0; b < nblocks; ++b) {
    if (blocks[b].n < 0 || blocks[b].goff < 0 || blocks[b].goff + blocks[b].n > S.block_n)
      return fail(ctx, BATHGPU_EINVAL, "block %d (offset %lld, n %d) is outside the uploaded sequence (n=%lld)", b, (long long)blocks[b].goff, blocks[b].n, (long long)S.block_n);
    first_tile[b] = (long long)tile_block.size();
    if (blocks[b].n >= 3)
      for (int p0 = 1; p0 <= blocks[b].n + 1; p0 += kOrfTile) { tile_block.push_back(b); tile_p0.push_back(p0); }
  }
  first_tile[nblocks] = (long long)tile_block.size();
  // the residues of every ORF of every block fit in sum of the block lengths (three frames of n/3 codons each); blocks overlap by
  // their context, so this can exceed the sequence length
  long long sum_block_n = 0;
  for (int b = 0; b < nblocks; ++b) sum_block_n += blocks[b].n;
  const int ntiles = (int)tile_block.size();
  *nhits = 0; *nres = 0;
  ctx->o_nhits = 0; ctx->o_nres = 0; S.nres = 0;
  if (norfs_per_block) for (int b = 0; b < nblocks; ++b) norfs_per_block[b] = 0;
  if (ntiles == 0) return BATHGPU_OK;
  CUDA_TRY(ctx, enter(ctx));
  const long long n = S.block_n;
  if (S.cls.reserve((size_t)n + 64) != BATHGPU_OK || ctx->o_tiles.reserve((size_t)ntiles * 8) != BATHGPU_OK || ctx->o_cnt.reserve((size_t)ntiles * 4) != BATHGPU_OK ||
      ctx->o_base.reserve((size_t)ntiles * 8) != BATHGPU_OK || ctx->o_blocks.reserve((size_t)nblocks * sizeof(BlockDesc)) != BATHGPU_OK ||
      ctx->o_first.reserve((size_t)nblocks * 8) != BATHGPU_OK || ctx->o_tjb.reserve((size_t)max_len + 1) != BATHGPU_OK ||
      ctx->o_null.reserve(((size_t)max_len + 1) * 4) != BATHGPU_OK || ctx->o_counters.reserve(64) != BATHGPU_OK || ctx->counter.reserve(64) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed");
  int *d_tile_block = ctx->o_tiles.as<int>(), *d_tile_p0 = ctx->o_tiles.as<int>() + ntiles;
  CUDA_TRY(ctx, cudaMemcpyAsync(d_tile_block, tile_block.data(), (size_t)ntiles * 4, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(d_tile_p0, tile_p0.data(), (size_t)ntiles * 4, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->o_blocks.p, blocks, (size_t)nblocks * sizeof(BlockDesc), cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->o_tjb.p, tjb_of, (size_t)max_len + 1, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->o_null.p, null_of, ((size_t)max_len + 1) * 4, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
  if (!ctx->o_ev[0]) for (auto &e : ctx->o_ev) CUDA_TRY(ctx, cudaEventCreate(&e));
  for (float &m : ctx->o_ms) m = 0.f;
  ctx->o_scored = 0; ctx->o_norf = 0;
  GeneticCode gc;
  memcpy(gc.aa, gcode, 64);
  CUDA_TRY(ctx, cudaEventRecord(ctx->o_ev[0], ctx->stream));
  {
    const long long nthreads = (n + 7) / 8;
    codon_class_kernel<<<(unsigned)((nthreads + 255) / 256), 256, 0, ctx->stream>>>(S.dna4.as<uint32_t>(), n, gc, S.cls.as<uint8_t>());
  }
  CUDA_TRY(ctx, cudaEventRecord(ctx->o_ev[1], ctx->stream));
  OrfScanArgs sa{};
  sa.cls = S.cls.as<uint8_t>(); sa.blocks = ctx->o_blocks.as<BlockDesc>(); sa.tile_block = d_tile_block; sa.tile_p0 = d_tile_p0;
  sa.ntiles = ntiles; sa.min_len = min_len; sa.complement = complement; sa.tile_cnt = ctx->o_cnt.as<int>();
  orf_scan_kernel<false><<<ntiles, kOrfTileThreads, 0, ctx->stream>>>(sa);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaEventRecord(ctx->o_ev[2], ctx->stream));
  std::vector<int> cnt((size_t)ntiles);
  CUDA_TRY(ctx, cudaMemcpyAsync(cnt.data(), ctx->o_cnt.p, (size_t)ntiles * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  std::vector<long long> base((size_t)ntiles + 1, 0), bfirst((size_t)nblocks, 0);
  for (int t = 0; t < ntiles; ++t) base[t + 1] = base[t] + cnt[t];
  for (int b = 0; b < nblocks; ++b) {
    bfirst[b] = base[first_tile[b]];
    if (norfs_per_block) norfs_per_block[b] = base[first_tile[b + 1]] - base[first_tile[b]];
  }
  const long long N = base[ntiles];
  if (N == 0) return BATHGPU_OK;
  if (N > 0x7fffffffLL) return fail(ctx, BATHGPU_EINVAL, "%lld ORFs in one call: split the sequence", N);
  if (ctx->orfs.reserve((size_t)N * sizeof(OrfDesc)) != BATHGPU_OK || ctx->o_meta.reserve((size_t)N * sizeof(OrfMeta)) != BATHGPU_OK ||
      ctx->fsc.reserve((size_t)N * 4) != BATHGPU_OK || ctx->fst.reserve((size_t)N * 4) != BATHGPU_OK ||
      ctx->o_hits.reserve((size_t)N * sizeof(OrfHit)) != BATHGPU_OK || S.residues.reserve((size_t)sum_block_n / 3 * 3 + 64) != BATHGPU_OK)
    return fail(ctx, BATHGPU_EMEM, "device allocation failed for %lld ORFs", N);
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->o_base.p, base.data(), (size_t)ntiles * 8, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->o_first.p, bfirst.data(), (size_t)nblocks * 8, cudaMemcpyHostToDevice, ctx->stream));
  sa.tile_base = ctx->o_base.as<long long>(); sa.block_first = ctx->o_first.as<long long>(); sa.tjb_of = ctx->o_tjb.as<uint8_t>();
  sa.max_len = max_len; sa.descs = ctx->orfs.as<OrfDesc>(); sa.meta = ctx->o_meta.as<OrfMeta>();
  sa.scored = ctx->o_counters.as<unsigned long long>() + 2;
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->o_counters.p, 0, 32, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->o_ev[5], ctx->stream));
  orf_scan_kernel<true><<<ntiles, kOrfTileThreads, 0, ctx->stream>>>(sa);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaEventRecord(ctx->o_ev[3], ctx->stream));
  // MSV over every ORF, residues read from the codon classes with stride 3
  CUDA_TRY(ctx, cudaMemsetAsync(ctx->counter.p, 0, 4, ctx->stream));
  FilterArgs fa = filter_args(ctx, (int)N, 0);
  fa.residues = S.cls.as<uint8_t>(); fa.res_stride = 3;
  CUDA_TRY(ctx, dispatch_msv(0, ctx->flt_W, fa, ctx->prop.multiProcessorCount, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->o_ev[4], ctx->stream));
  OrfScreenArgs ra{};
  ra.cls = S.cls.as<uint8_t>(); ra.descs = ctx->orfs.as<OrfDesc>(); ra.meta = ctx->o_meta.as<OrfMeta>(); ra.usc = ctx->fsc.as<float>();
  ra.status = ctx->fst.as<int>(); ra.norf = N; ra.null_of = ctx->o_null.as<float>(); ra.max_len = max_len; ra.min_bits = min_bits;
  ra.hits = ctx->o_hits.as<OrfHit>(); ra.residues = S.residues.as<uint8_t>(); ra.counters = ctx->o_counters.as<unsigned long long>();
  orf_screen_kernel<<<(unsigned)((N + 255) / 256), 256, 0, ctx->stream>>>(ra);
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
  unsigned long long hc[3] = { 0, 0, 0 };
  CUDA_TRY(ctx, cudaMemcpyAsync(hc, ctx->o_counters.p, 24, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->last_ms, ctx->ev0, ctx->ev1));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->o_ms[0], ctx->o_ev[0], ctx->o_ev[1]));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->o_ms[1], ctx->o_ev[1], ctx->o_ev[2]));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->o_ms[2], ctx->o_ev[5], ctx->o_ev[3]));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->o_ms[3], ctx->o_ev[3], ctx->o_ev[4]));
  CUDA_TRY(ctx, cudaEventElapsedTime(&ctx->o_ms[4], ctx->o_ev[4], ctx->ev1));
  ctx->o_scored = (long long)hc[2]; ctx->o_norf = N;
  ctx->last_launches = 5;
  ctx->o_nhits = (long long)hc[0]; ctx->o_nres = (long long)hc[1];
  S.nres = (int64_t)hc[1];
  *nhits = (int64_t)hc[0]; *nres = (int64_t)hc[1];
  return BATHGPU_OK;
}

extern "C" int bathgpu_orfs_stage_breakdown(bathgpu_ctx *ctx, float ms[5], int64_t *norfs, int64_t *residues_scored)
{
  if (!ctx || !ms) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_orfs_stage_breakdown");
  for (int z = 0; z < 5; ++z) ms[z] = ctx->o_ms[z];
  if (norfs) *norfs = ctx->o_norf;
  if (residues_scored) *residues_scored = ctx->o_scored;
  return BATHGPU_OK;
}

extern "C" int bathgpu_orfs_fetch(bathgpu_ctx *ctx, bathgpu_orf_hit *hits, uint8_t *residues)
{
  if (!ctx || (ctx->o_nhits > 0 && (!hits || !residues))) return fail(ctx, BATHGPU_EINVAL, "bad arguments to bathgpu_orfs_fetch");
  if (ctx->o_nhits == 0) return BATHGPU_OK;
  CUDA_TRY(ctx, enter(ctx));
  CUDA_TRY(ctx, cudaMemcpyAsync(hits, ctx->o_hits.p, (size_t)ctx->o_nhits * sizeof(OrfHit), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(residues, ctx->S().residues.p, (size_t)ctx->o_nres, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, wait_stream(ctx));
  std::sort(hits, hits + ctx->o_nhits, [](const bathgpu_orf_hit &x, const bathgpu_orf_hit &y) {
    return x.block != y.block ? x.block < y.block : x.index < y.index; });
  return BATHGPU_OK;
}
