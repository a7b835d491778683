// launch.h -- the kernel families behind bathgpu.cu, one launch entry per family and node-count set.
// kernels_tu.cu is compiled once per (family, set) so that the template instantiations build in parallel
// (bath_b200/build.py); bathgpu.cu only sees these plain functions.  Each returns false when the requested
// template parameter is not in its set.
#pragma once
#include <cuda_runtime.h>

namespace bathgpu {

struct FsParserArgs;
struct FsBackwardArgs;
struct DomainArgs;
struct TraceArgs;
struct OrfDomainArgs;
struct OrfFwdArgs;
struct FilterArgs;

// J (nodes per lane) sets: a = 1..5, b = 6..8, c = 10,12, d = 16, e = 24, f = 32 (the last three spill part of the
// per-node state to local memory: they exist so that models up to M = 1024 run at all, at reduced speed)
#define BATHGPU_FOR_EACH_SET(X) X(a) X(b) X(c) X(d) X(e) X(f)

#define BATHGPU_DECLARE_SET(S)                                                                                                       \
  bool launch_fs3_forward_##S(int J, bool xmx, int version, const FsParserArgs &a, int sms, cudaStream_t s, cudaError_t *err);       \
  bool launch_fs3_backward_##S(int J, const FsBackwardArgs &a, int sms, cudaStream_t s, cudaError_t *err);                           \
  bool launch_fs5_domains_##S(int J, const DomainArgs &a, const TraceArgs &t, int sms, cudaStream_t s, cudaError_t *err);            \
  bool launch_fs5_forward_matrix_##S(int J, const DomainArgs &a, int sms, cudaStream_t s, cudaError_t *err);                         \
  bool launch_orf_domains_##S(int J, bool full, const OrfDomainArgs &a, const TraceArgs &t, int sms, cudaStream_t s, cudaError_t *err); \
  bool launch_orf_forward_matrix_##S(int J, const OrfDomainArgs &a, int sms, cudaStream_t s, cudaError_t *err);                            \
  bool launch_orf_forward_parser_##S(int J, const OrfFwdArgs &a, int sms, cudaStream_t s, cudaError_t *err);                        \
  bool launch_fs3_forward_set_##S(int J, int version, const FsParserArgs &a, int sms, cudaStream_t s, cudaError_t *err);            \
  bool launch_fs5_forward_set_##S(int J, const DomainArgs &a, int sms, cudaStream_t s, cudaError_t *err);                            \
  void preload_fwd_##S(int J); void preload_bck_##S(int J); void preload_fs5_##S(int J); void preload_orf_##S(int J);
BATHGPU_FOR_EACH_SET(BATHGPU_DECLARE_SET)
#undef BATHGPU_DECLARE_SET

// nodes per lane of the multi-warp Forward kernel for long models (fs_parser_mw.cuh); the constant image built by bathgpu.cu and the
// kernel instantiations must agree.  4 nodes per lane (twice the warps per window) was measured at half the speed: 235 vs 458 GCUPS
// at M = 903.
constexpr int kMwNodesPerLane = 8;

// integer filters: W words (4 nodes each) per lane for MSV/SSV, P words (2 nodes each) per lane for Viterbi
bool launch_msv_filter(int W, int P, int mode, const FilterArgs &a, int sms, cudaStream_t s, cudaError_t *err);
bool launch_vit_filter_lo(int P, const FilterArgs &a, int sms, cudaStream_t s, cudaError_t *err);      // P = 1..6
bool launch_vit_filter_hi(int P, const FilterArgs &a, int sms, cudaStream_t s, cudaError_t *err);      // P = 8, 12, 16
// Touch the kernels a profile of this size will use, so that the driver loads their code when the profile is loaded and not
// inside the first stage call (CUDA loads kernels lazily).
void preload_msv_filter(int W, int P); void preload_vit_filter_lo(int P); void preload_vit_filter_hi(int P);

}  // namespace bathgpu
