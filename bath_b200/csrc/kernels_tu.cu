// kernels_tu.cu -- template instantiations of one kernel family for one set of node counts (see launch.h).
// Compiled once per -DBATHGPU_FAMILY=<n> -DBATHGPU_SET=<n> combination by bath_b200/build.py.
#include <algorithm>
#include <cstdlib>
#include "launch.h"
#include "fs_parser.cuh"
#include "fs_parser_v3.cuh"
#include "fs_parser_v4.cuh"
#include "fs_parser_mw.cuh"
#include "fs_backward.cuh"
#include "fs_backward_mw.cuh"
#include "fs_domain.cuh"
#include "orf_domain.cuh"
#include "orf_filters.cuh"

#define FAM_FWD 1
#define FAM_BCK 2
#define FAM_FS5 3
#define FAM_ORF 4
#define FAM_FILT_MSV 5
#define FAM_FILT_VIT_LO 6
#define FAM_FILT_VIT_HI 7

#if   BATHGPU_SET == 0
#define SETNAME a
#define JLIST(X) X(1) X(2) X(3) X(4) X(5)
#elif BATHGPU_SET == 1
#define SETNAME b
#define JLIST(X) X(6) X(7) X(8)
#elif BATHGPU_SET == 2
#define SETNAME c
#define JLIST(X) X(10) X(12)
#elif BATHGPU_SET == 3
#define SETNAME d
#define JLIST(X) X(16)
#elif BATHGPU_SET == 4
#define SETNAME e
#define JLIST(X) X(24)
#elif BATHGPU_SET == 5
#define SETNAME f
#define JLIST(X) X(32)
#endif
#define CAT2(a, b) a##b
#define CAT(a, b) CAT2(a, b)

namespace bathgpu {

template <class K> static void touch(K kernel) { cudaFuncAttributes fa; cudaFuncGetAttributes(&fa, kernel); }

template <class K> static int grid_for(K kernel, int threads, size_t smem, int n, int sms)
{
  int nb = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem);
  return std::max(1, std::min(n, sms * std::max(nb, 1)));
}

#if BATHGPU_FAMILY == FAM_FWD
// resident one-warp blocks per SM of the row-pair Forward kernel: what fits, capped at the measured optimum for this J
// (BATHGPU_V3_RESIDENT in fs_parser_v3.cuh; BATHGPU_FWD_WARPS overrides it for tuning runs)
template <class K> static int fwd_grid(K kernel, int J, int n, int sms)
{
  static const int env_cap = [] { const char *e = getenv("BATHGPU_FWD_WARPS"); return e ? atoi(e) : 0; }();
  int nb = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, 32, 0);
  const int cap = env_cap > 0 ? env_cap : BATHGPU_V3_RESIDENT(J);
  return std::max(1, std::min(n, sms * std::max(1, std::min(nb, cap))));
}

// models past the one-warp kernels' register budget (J >= 16): J/8 warps per window (fs_parser_mw.cuh); BATHGPU_FWD_MW=0 keeps the
// one-warp kernel for comparison
template <int NW, int JW, bool XMX, bool SET = false> static cudaError_t run_fwd_mw(const FsParserArgs &a, int sms, cudaStream_t s)
{
  if (a.mw_scan_steps <= 3) fs3_forward_parser_kernel_mw<NW, JW, XMX, 3, SET><<<grid_for(fs3_forward_parser_kernel_mw<NW, JW, XMX, 3, SET>, 32 * NW, 0, a.nwin, sms), 32 * NW, 0, s>>>(a);
  else                      fs3_forward_parser_kernel_mw<NW, JW, XMX, 5, SET><<<grid_for(fs3_forward_parser_kernel_mw<NW, JW, XMX, 5, SET>, 32 * NW, 0, a.nwin, sms), 32 * NW, 0, s>>>(a);
  return cudaGetLastError();
}

// SET: the windows of a profile set (FsParserArgs::set); a.cellmw non-null when the set's profiles have multi-warp images
template <int J, bool XMX, bool SET = false> static cudaError_t run_fwd(int version, const FsParserArgs &a, int sms, cudaStream_t s)
{
  if constexpr (J >= 16) {
    // BATHGPU_FWD_MW: 0 never, 1 (default) from 24 nodes per lane up -- at 16 the one-warp kernel is still ahead (800 vs 620 GCUPS
    // at M = 409) --, 2 from 16 up
    static const int mw_mode = [] { const char *e = getenv("BATHGPU_FWD_MW"); return e ? atoi(e) : 1; }();
    if (version >= 3 && a.cellmw && (mw_mode >= 2 || (mw_mode == 1 && J >= 24))) return run_fwd_mw<J / kMwNodesPerLane, kMwNodesPerLane, XMX, SET>(a, sms, s);
  }
  if (version >= 4) {                 // packed-FP32 row pairs (fs_parser_v4.cuh)
    if (a.scan_steps <= 2)      fs3_forward_parser_kernel_v4<J, XMX, 2, SET><<<fwd_grid(fs3_forward_parser_kernel_v4<J, XMX, 2, SET>, J, a.nwin, sms), 32, 0, s>>>(a);
    else if (a.scan_steps == 3) fs3_forward_parser_kernel_v4<J, XMX, 3, SET><<<fwd_grid(fs3_forward_parser_kernel_v4<J, XMX, 3, SET>, J, a.nwin, sms), 32, 0, s>>>(a);
    else                        fs3_forward_parser_kernel_v4<J, XMX, 5, SET><<<fwd_grid(fs3_forward_parser_kernel_v4<J, XMX, 5, SET>, J, a.nwin, sms), 32, 0, s>>>(a);
  }
  else {                              // scalar row pairs (fs_parser_v3.cuh); the first-generation one-row kernel is gone
    if (a.scan_steps <= 2)      fs3_forward_parser_kernel_v3<J, XMX, 2, SET><<<fwd_grid(fs3_forward_parser_kernel_v3<J, XMX, 2, SET>, J, a.nwin, sms), 32, 0, s>>>(a);
    else if (a.scan_steps == 3) fs3_forward_parser_kernel_v3<J, XMX, 3, SET><<<fwd_grid(fs3_forward_parser_kernel_v3<J, XMX, 3, SET>, J, a.nwin, sms), 32, 0, s>>>(a);
    else                        fs3_forward_parser_kernel_v3<J, XMX, 5, SET><<<fwd_grid(fs3_forward_parser_kernel_v3<J, XMX, 5, SET>, J, a.nwin, sms), 32, 0, s>>>(a);
  }
  return cudaGetLastError();
}
// the Forward parser over the windows of a profile set: the kernel run_fwd picks for the set's J, scan steps and version
bool CAT(launch_fs3_forward_set_, SETNAME)(int J, int version, const FsParserArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: *err = run_fwd<J_, false, true>(version, a, sms, s); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
bool CAT(launch_fs3_forward_, SETNAME)(int J, bool xmx, int version, const FsParserArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: *err = xmx ? run_fwd<J_, true>(version, a, sms, s) : run_fwd<J_, false>(version, a, sms, s); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
void CAT(preload_fwd_, SETNAME)(int J)
{
  switch (J) {
#define X(J_) case J_: touch(fs3_forward_parser_kernel_v3<J_, false, 2>); touch(fs3_forward_parser_kernel_v3<J_, true, 2>); touch(fs3_forward_parser_kernel_v3<J_, false, 3>); \
                       touch(fs3_forward_parser_kernel_v3<J_, true, 3>); touch(fs3_forward_parser_kernel_v3<J_, false, 5>); touch(fs3_forward_parser_kernel_v3<J_, true, 5>); \
                       if (J_ == 10) { touch(fs3_forward_parser_kernel_v4<J_, false, 2>); touch(fs3_forward_parser_kernel_v4<J_, true, 2>); touch(fs3_forward_parser_kernel_v4<J_, false, 3>); \
                                       touch(fs3_forward_parser_kernel_v4<J_, true, 3>); touch(fs3_forward_parser_kernel_v4<J_, false, 5>); touch(fs3_forward_parser_kernel_v4<J_, true, 5>); } \
                       break;
  JLIST(X)
#undef X
  default: break;
  }
}
#endif

#if BATHGPU_FAMILY == FAM_BCK
// models past the one-warp kernel's register budget: J/8 warps per window (fs_backward_mw.cuh), from 16 nodes per lane up (M > 384:
// 434 -> 475 GCUPS at M = 409, 289 -> 363 at M = 624, 202 -> 391 at M = 903).  BATHGPU_BCK_MW=0 keeps the one-warp kernel
template <int J> static cudaError_t run_bck(const FsBackwardArgs &a, int sms, cudaStream_t s)
{
  if constexpr (J >= 16) {
    static const int mw_mode = [] { const char *e = getenv("BATHGPU_BCK_MW"); return e ? atoi(e) : 1; }();
    if (a.cellbmw && mw_mode >= 1) {
      constexpr int NW = J / kMwNodesPerLane;
      fs3_backward_parser_kernel_mw<NW, kMwNodesPerLane><<<grid_for(fs3_backward_parser_kernel_mw<NW, kMwNodesPerLane>, 32 * NW, 0, a.nwin, sms), 32 * NW, 0, s>>>(a);
      return cudaGetLastError();
    }
  }
  fs3_backward_parser_kernel<J><<<grid_for(fs3_backward_parser_kernel<J>, BckTune<J>::kThreads, 0, a.nwin, sms), BckTune<J>::kThreads, 0, s>>>(a);
  return cudaGetLastError();
}
bool CAT(launch_fs3_backward_, SETNAME)(int J, const FsBackwardArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: *err = run_bck<J_>(a, sms, s); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
void CAT(preload_bck_, SETNAME)(int J)
{
  switch (J) {
#define X(J_) case J_: touch(fs3_backward_parser_kernel<J_>); if constexpr (J_ >= 16) touch(fs3_backward_parser_kernel_mw<J_ / kMwNodesPerLane, kMwNodesPerLane>); break;
  JLIST(X)
#undef X
  default: break;
  }
}
#endif

#if BATHGPU_FAMILY == FAM_FS5
template <int J> static cudaError_t run_fs5(const DomainArgs &a, const TraceArgs &t, int sms, cudaStream_t s)
{
  cudaError_t e;
  if ((e = cudaMemsetAsync(a.counter, 0, 4, s)) != cudaSuccess) return e;
  fs5_forward_kernel<J><<<grid_for(fs5_forward_kernel<J>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);
  if ((e = cudaMemsetAsync(a.counter, 0, 4, s)) != cudaSuccess) return e;
  fs5_backward_decode_kernel<J><<<grid_for(fs5_backward_decode_kernel<J>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);
  if ((e = cudaMemsetAsync(a.counter, 0, 4, s)) != cudaSuccess) return e;
  fs5_optacc_kernel<J><<<grid_for(fs5_optacc_kernel<J>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);
  fs5_oatrace_kernel<<<(a.nenv + 3) / 4, 128, 0, s>>>(a, t);
  return cudaGetLastError();
}
bool CAT(launch_fs5_domains_, SETNAME)(int J, const DomainArgs &a, const TraceArgs &t, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: *err = run_fs5<J_>(a, t, sms, s); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
// Forward alone, D cells kept: the matrix the stochastic traceback samples from (p7_Forward_Frameshift before
// region_trace_ensemble_frameshift, src/p7_domaindef.c:411-414)
bool CAT(launch_fs5_forward_matrix_, SETNAME)(int J, const DomainArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: if ((*err = cudaMemsetAsync(a.counter, 0, 4, s)) != cudaSuccess) return true;                               \
                       fs5_forward_kernel<J_, true><<<grid_for(fs5_forward_kernel<J_, true>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);   \
                       *err = cudaGetLastError(); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
// the scores of p7_ForwardParser_Frameshift_5Codons over the envelopes of a profile set (launch_fs5_forward_matrix's kernel)
bool CAT(launch_fs5_forward_set_, SETNAME)(int J, const DomainArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: fs5_forward_kernel<J_, true, true><<<grid_for(fs5_forward_kernel<J_, true, true>, 32, 0, a.nenv, sms), 32, 0, s>>>(a); \
                       *err = cudaGetLastError(); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
void CAT(preload_fs5_, SETNAME)(int J)
{
  switch (J) {
#define X(J_) case J_: touch(fs5_forward_kernel<J_>); touch(fs5_backward_decode_kernel<J_>); touch(fs5_optacc_kernel<J_>); touch(fs5_oatrace_kernel); break;
  JLIST(X)
#undef X
  default: break;
  }
}
#endif

#if BATHGPU_FAMILY == FAM_ORF
template <int J> static cudaError_t run_orf(bool full, const OrfDomainArgs &a, const TraceArgs &t, int sms, cudaStream_t s)
{
  cudaError_t e;
  if ((e = cudaMemsetAsync(a.counter, 0, 4, s)) != cudaSuccess) return e;
  if (!full) {
    orf_forward_kernel<J, false><<<grid_for(orf_forward_kernel<J, false>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);
    if ((e = cudaMemsetAsync(a.counter, 0, 4, s)) != cudaSuccess) return e;
    orf_backward_kernel<J, false><<<grid_for(orf_backward_kernel<J, false>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);
    return cudaGetLastError();
  }
  orf_forward_kernel<J, true><<<grid_for(orf_forward_kernel<J, true>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);
  if ((e = cudaMemsetAsync(a.counter, 0, 4, s)) != cudaSuccess) return e;
  orf_backward_kernel<J, true><<<grid_for(orf_backward_kernel<J, true>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);
  if ((e = cudaMemsetAsync(a.counter, 0, 4, s)) != cudaSuccess) return e;
  orf_optacc_kernel<J><<<grid_for(orf_optacc_kernel<J>, 32, 0, a.nenv, sms), 32, 0, s>>>(a);
  orf_oatrace_kernel<<<(a.nenv + 3) / 4, 128, 0, s>>>(a, t);
  return cudaGetLastError();
}
// the Forward matrix alone, D cells kept (multi-domain regions of the standard branch: the stochastic traceback reads it)
bool CAT(launch_orf_forward_matrix_, SETNAME)(int J, const OrfDomainArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: *err = cudaMemsetAsync(a.counter, 0, 4, s); if (*err != cudaSuccess) return true; \
                       orf_forward_kernel<J_, true, true><<<grid_for(orf_forward_kernel<J_, true, true>, 32, 0, a.nenv, sms), 32, 0, s>>>(a); *err = cudaGetLastError(); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
bool CAT(launch_orf_domains_, SETNAME)(int J, bool full, const OrfDomainArgs &a, const TraceArgs &t, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: *err = run_orf<J_>(full, a, t, sms, s); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
bool CAT(launch_orf_forward_parser_, SETNAME)(int J, const OrfFwdArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (J) {
#define X(J_) case J_: orf_forward_parser_kernel<J_><<<grid_for(orf_forward_parser_kernel<J_>, 32, 0, a.norf, sms), 32, 0, s>>>(a); \
                       *err = cudaGetLastError(); return true;
  JLIST(X)
#undef X
  default: return false;
  }
}
void CAT(preload_orf_, SETNAME)(int J)
{
  switch (J) {
#define X(J_) case J_: touch(orf_forward_kernel<J_, false>); touch(orf_forward_kernel<J_, true>); touch(orf_backward_kernel<J_, false>); \
                       touch(orf_backward_kernel<J_, true>); touch(orf_optacc_kernel<J_>); touch(orf_oatrace_kernel); touch(orf_forward_parser_kernel<J_>); break;
  JLIST(X)
#undef X
  default: break;
  }
}
#endif

#if BATHGPU_FAMILY == FAM_FILT_MSV
template <int W, int MODE> static cudaError_t run_msv(const FilterArgs &a, int sms, cudaStream_t s)
{
  const size_t smem = (size_t)29 * 32 * W * 4;
  msv_filter_kernel<W, MODE><<<grid_for(msv_filter_kernel<W, MODE>, 128, smem, (a.norf + 3) / 4, sms), 128, smem, s>>>(a);
  return cudaGetLastError();
}
template <int P> static cudaError_t run_msv16(const FilterArgs &a, int sms, cudaStream_t s)
{
  const size_t smem = (size_t)29 * 32 * P * 4;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(msv16_filter_kernel<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  msv16_filter_kernel<P><<<grid_for(msv16_filter_kernel<P>, 128, smem, (a.norf + 3) / 4, sms), 128, smem, s>>>(a);
  return cudaGetLastError();
}
// mode 0: MSV scores (16-bit lanes, P words per lane); mode 1: SSV windows (byte lanes, W words per lane)
bool launch_msv_filter(int W, int P, int mode, const FilterArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  if (mode == 0) {
    switch (P) {
#define X(P_) case P_: *err = run_msv16<P_>(a, sms, s); return true;
    X(1) X(2) X(3) X(4) X(5) X(6) X(8) X(12) X(16)
#undef X
    default: return false;
    }
  }
  switch (W) {
#define X(W_) case W_: *err = run_msv<W_, 1>(a, sms, s); return true;
  X(1) X(2) X(3) X(4) X(6) X(8)
#undef X
  default: return false;
  }
}
void preload_msv_filter(int W, int P)
{
  switch (W) {
#define X(W_) case W_: touch(msv_filter_kernel<W_, 1>); break;
  X(1) X(2) X(3) X(4) X(6) X(8)
#undef X
  default: break;
  }
  switch (P) {
#define X(P_) case P_: touch(msv16_filter_kernel<P_>); break;
  X(1) X(2) X(3) X(4) X(5) X(6) X(8) X(12) X(16)
#undef X
  default: break;
  }
}
#endif

#if BATHGPU_FAMILY == FAM_FILT_VIT_LO || BATHGPU_FAMILY == FAM_FILT_VIT_HI
template <int P> static cudaError_t run_vit(const FilterArgs &a, int sms, cudaStream_t s)
{
  const size_t smem = (size_t)(29 + 8) * 32 * P * 4;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(vit_filter_kernel<P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  vit_filter_kernel<P><<<grid_for(vit_filter_kernel<P>, 128, smem, (a.norf + 3) / 4, sms), 128, smem, s>>>(a);
  return cudaGetLastError();
}
#if BATHGPU_FAMILY == FAM_FILT_VIT_LO
bool launch_vit_filter_lo(int P, const FilterArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (P) {
#define X(P_) case P_: *err = run_vit<P_>(a, sms, s); return true;
  X(1) X(2) X(3) X(4) X(5) X(6)
#undef X
  default: return false;
  }
}
void preload_vit_filter_lo(int P)
{
  switch (P) {
#define X(P_) case P_: touch(vit_filter_kernel<P_>); break;
  X(1) X(2) X(3) X(4) X(5) X(6)
#undef X
  default: break;
  }
}
#else
bool launch_vit_filter_hi(int P, const FilterArgs &a, int sms, cudaStream_t s, cudaError_t *err)
{
  switch (P) {
#define X(P_) case P_: *err = run_vit<P_>(a, sms, s); return true;
  X(8) X(12) X(16)
#undef X
  default: return false;
  }
}
void preload_vit_filter_hi(int P)
{
  switch (P) {
#define X(P_) case P_: touch(vit_filter_kernel<P_>); break;
  X(8) X(12) X(16)
#undef X
  default: break;
  }
}
#endif
#endif

}  // namespace bathgpu
