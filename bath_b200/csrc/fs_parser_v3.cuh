// fs_parser_v3.cuh -- frameshift Forward parser, row-pair schedule.
//
// Same recurrence, carried quantities and tables as fs_parser.cuh (read its header first).  What changes is
// the schedule: DP rows i and i+1 depend only on rows <= i-1 (the quasi-codon look-back starts two rows
// back: W(i+1) was finished by row i-1), so the two rows are computed in ONE basic block and the compiler
// interleaves their instruction streams.  The per-row cost of this kernel is latency, not issue slots: each
// row has two serial shuffle chains (the E sum and the D->D scan, ~140 cycles each); pairing rows overlaps
// the chains of two rows inside one warp, which is worth more than the warps the extra registers cost.
// The rescale test (xE > 1e4, fwdback_fs.c:472-496) is taken once per pair: if row i rescales, row i+1's
// freshly computed values are scaled with everything else (they are linear in the state they were computed
// from), then row i+1 is tested on its scaled xE exactly as the reference would see it.
#pragma once
#include "fs_parser.cuh"

// The E sums of a row pair reduced in one butterfly (pair_allsum: 6 shuffles for 10).  Measured on B200 per node count
// (scripts/j_sweep.py, 16 384 windows of 1200 nt): +2.2 % at J = 3 (M = 78), +3.4 % at J = 4 (M = 116-121), +2.9 % at J = 5 (M = 131-152),
// +4.5 % at J = 2, +1.4 % at J = 8; -1.5 % at J = 6, where the pair sits at the 128-register cap, 0 at J = 7 and 16.
#ifndef BATHGPU_V3_JOINT_E
#define BATHGPU_V3_JOINT_E(J) (((J) >= 2 && (J) <= 5) || (J) == 8)
#endif

namespace bathgpu {

struct RowOut { float xE, xN, xJ, xC, xB, scale; };

// Row i without the rescale test and without the X-row store.
// HEAD: the row may be one of the first rows of the window (pad rows i < 0, rows 0..2 where N is held at 1); only the first
// 32 rows of a window run the instantiation that tests for it.
template <int J, int VEC, int PH, int NS, bool HEAD>
__device__ __forceinline__ void fwd_row_compute(int i, int lane, FwdState<J> &S, const FwdConsts<J> &K,
                                                const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t cw,
                                                float ploop, float pmove, float tEL, float tEM, RowOut &R)
{
  constexpr int P0 = PH, P1 = (PH + 3) & 3, P2 = (PH + 2) & 3, P3 = (PH + 1) & 3;
  float e2[J], e3[J], e4[J], m[J];
  load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw & 511u) * rowbytes), e2);
  load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)((cw >> 9) & 511u) * rowbytes), e3);
  load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw >> 18) * rowbytes), e4);

  float es0 = 0.f, es1 = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    float t = S.W[P2][j] * e4[j];              // W[P0] was finished last (by row i-2): its term closes the chain (+1-3 %)
    t = fmaf(S.W[P1][j], e3[j], t);
    t = fmaf(S.W[P0][j], e2[j], t);
    m[j] = t;
    if (j == 0) es0 = t * K.qm[0]; else if (j == 1) es1 = t * K.qm[1]; else if (j & 1) es1 = fmaf(t, K.qm[j], es1); else es0 = fmaf(t, K.qm[j], es0);
  }
  float xE = warp_allsum(J > 1 ? es0 + es1 : es0);

  float A = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j) A = (j == 0) ? m[0] : fmaf(A, K.dd[j], m[j]);   // scaled delete chain: the match term needs no multiply
#pragma unroll
  for (int s = 0; s < NS; ++s) {                 // NS < 5: the products of D->D odds over 2^NS lanes are below 1e-9 for this profile
    float up = __shfl_up_sync(0xffffffffu, A, 1 << s);
    A = fmaf(K.bs[s], up, A);
  }
  float d = __shfl_up_sync(0xffffffffu, A, 1);      // lane 0 reads its own A: node 1 has no delete state, its dd and dm are 0 (bathgpu.cu)

  float xN = S.xN[P3] * ploop;
  if constexpr (HEAD) xN = (i < 3) ? ((i >= 0) ? 1.0f : 0.0f) : xN;
  float xJ = fmaf(S.xJ[P3], ploop, xE * tEL);
  float xC = fmaf(S.xC[P3], ploop, xE * tEM);
  float xB = fmaf(xJ, pmove, xN * pmove);

  float o[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    float t = fmaf(S.I[P0][j], K.hi[j], m[j]);
    o[j] = fmaf(d, K.dm[j], t);
    if (j + 1 < J) d = fmaf(d, K.dd[j], m[j]);
    S.I[P1][j] = fmaf(S.I[P0][j], K.ii[j], m[j]);
  }
  float oprev = __shfl_up_sync(0xffffffffu, o[J - 1], 1);
  if (lane == 0) oprev = 0.f;                       // a select: a 0/1 lane constant in an FMA costs a register the J = 6 kernel lacks
  S.W[P2][0] = xB + oprev;
#pragma unroll
  for (int j = 1; j < J; ++j) S.W[P2][j] = xB + o[j - 1];
  S.xN[P0] = xN; S.xJ[P0] = xJ; S.xC[P0] = xC;
  R.xE = xE; R.xN = xN; R.xJ = xJ; R.xC = xC; R.xB = xB; R.scale = 1.0f;
}

// The row in two halves, for the joint E reduction of a row pair (fwd_row_pair): the first half ends with the lane's partial E sum
// and the delete chain's inflow, the second starts from the reduced E.
template <int J> struct RowMid { float m[J]; float es, d; };

template <int J, int VEC, int PH, int NS>
__device__ __forceinline__ void fwd_row_front(const FwdState<J> &S, const FwdConsts<J> &K, const char *__restrict__ emis_lane, unsigned rowbytes,
                                              uint32_t cw, RowMid<J> &X)
{
  constexpr int P0 = PH, P1 = (PH + 3) & 3, P2 = (PH + 2) & 3;
  float e2[J], e3[J], e4[J];
  load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw & 511u) * rowbytes), e2);
  load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)((cw >> 9) & 511u) * rowbytes), e3);
  load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw >> 18) * rowbytes), e4);
  float es0 = 0.f, es1 = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    float t = S.W[P2][j] * e4[j];
    t = fmaf(S.W[P1][j], e3[j], t);
    t = fmaf(S.W[P0][j], e2[j], t);
    X.m[j] = t;
    if (j == 0) es0 = t * K.qm[0]; else if (j == 1) es1 = t * K.qm[1]; else if (j & 1) es1 = fmaf(t, K.qm[j], es1); else es0 = fmaf(t, K.qm[j], es0);
  }
  X.es = (J > 1) ? es0 + es1 : es0;
  float A = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j) A = (j == 0) ? X.m[0] : fmaf(A, K.dd[j], X.m[j]);
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    float up = __shfl_up_sync(0xffffffffu, A, 1 << s);
    A = fmaf(K.bs[s], up, A);
  }
  X.d = __shfl_up_sync(0xffffffffu, A, 1);
}

template <int J, int PH, bool HEAD>
__device__ __forceinline__ void fwd_row_back(int i, int lane, FwdState<J> &S, const FwdConsts<J> &K, const RowMid<J> &X, float xE,
                                             float ploop, float pmove, float tEL, float tEM, RowOut &R)
{
  constexpr int P0 = PH, P1 = (PH + 3) & 3, P2 = (PH + 2) & 3, P3 = (PH + 1) & 3;
  float d = X.d;
  float xN = S.xN[P3] * ploop;
  if constexpr (HEAD) xN = (i < 3) ? ((i >= 0) ? 1.0f : 0.0f) : xN;
  float xJ = fmaf(S.xJ[P3], ploop, xE * tEL);
  float xC = fmaf(S.xC[P3], ploop, xE * tEM);
  float xB = fmaf(xJ, pmove, xN * pmove);
  float o[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    float t = fmaf(S.I[P0][j], K.hi[j], X.m[j]);
    o[j] = fmaf(d, K.dm[j], t);
    if (j + 1 < J) d = fmaf(d, K.dd[j], X.m[j]);
    S.I[P1][j] = fmaf(S.I[P0][j], K.ii[j], X.m[j]);
  }
  float oprev = __shfl_up_sync(0xffffffffu, o[J - 1], 1);
  if (lane == 0) oprev = 0.f;
  S.W[P2][0] = xB + oprev;
#pragma unroll
  for (int j = 1; j < J; ++j) S.W[P2][j] = xB + o[j - 1];
  S.xN[P0] = xN; S.xJ[P0] = xJ; S.xC[P0] = xC;
  R.xE = xE; R.xN = xN; R.xJ = xJ; R.xC = xC; R.xB = xB; R.scale = 1.0f;
}

template <int J>
__device__ __forceinline__ void scale_state(FwdState<J> &S, float sf)
{
#pragma unroll
  for (int r = 0; r < 4; ++r) {
#pragma unroll
    for (int j = 0; j < J; ++j) { S.W[r][j] *= sf; S.I[r][j] *= sf; }
    S.xN[r] *= sf; S.xJ[r] *= sf; S.xC[r] *= sf;
  }
}

template <bool XMX>
__device__ __forceinline__ void store_xrow(int i, int lane, const RowOut &R, float *__restrict__ xrow)
{
  if constexpr (XMX) {
    if (lane == 0 && i >= 0) {
      float2 *x2 = reinterpret_cast<float2 *>(xrow + (size_t)i * 6);
      x2[0] = make_float2(R.xE, R.xN);
      x2[1] = make_float2(R.xJ, R.xB);
      x2[2] = make_float2(R.xC, R.scale);
    }
  }
}

// Rows i (phase PH) and i+1 (phase PH+1) in one block, then the rescale logic for both in order.
template <int J, int VEC, int PH, bool XMX, int NS, bool HEAD>
__device__ __forceinline__ void fwd_row_pair(int i, int lane, FwdState<J> &S, const FwdConsts<J> &K,
                                             const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t cwA, uint32_t cwB,
                                             float ploop, float pmove, float tEL, float tEM,
                                             float &totscale, float *__restrict__ xrow)
{
  RowOut A, B;
  if constexpr (BATHGPU_V3_JOINT_E(J)) {
    RowMid<J> XA, XB;
    fwd_row_front<J, VEC, PH, NS>(S, K, emis_lane, rowbytes, cwA, XA);
    fwd_row_front<J, VEC, PH + 1, NS>(S, K, emis_lane, rowbytes, cwB, XB);
    float xEA, xEB;
    pair_allsum(lane, XA.es, XB.es, xEA, xEB);
    fwd_row_back<J, PH, HEAD>(i, lane, S, K, XA, xEA, ploop, pmove, tEL, tEM, A);
    fwd_row_back<J, PH + 1, HEAD>(i + 1, lane, S, K, XB, xEB, ploop, pmove, tEL, tEM, B);
  } else {
    fwd_row_compute<J, VEC, PH, NS, HEAD>(i, lane, S, K, emis_lane, rowbytes, cwA, ploop, pmove, tEL, tEM, A);
    fwd_row_compute<J, VEC, PH + 1, NS, HEAD>(i + 1, lane, S, K, emis_lane, rowbytes, cwB, ploop, pmove, tEL, tEM, B);
  }
  if (__builtin_expect(A.xE > 1.0e4f || B.xE > 1.0e4f, 0)) {          // rare, warp-uniform
    if (A.xE > 1.0e4f) {
      const float sf = 1.0f / A.xE;
      scale_state<J>(S, sf);                     // includes what row i+1 has just written
      A.scale = A.xE; A.xN *= sf; A.xJ *= sf; A.xC *= sf; A.xB *= sf;
      B.xE *= sf; B.xN *= sf; B.xJ *= sf; B.xC *= sf; B.xB *= sf;
      totscale += logf(A.xE);
      A.xE = 1.0f;
    }
    if (B.xE > 1.0e4f) {
      const float sf = 1.0f / B.xE;
      scale_state<J>(S, sf);
      B.scale = B.xE; B.xN *= sf; B.xJ *= sf; B.xC *= sf; B.xB *= sf;
      totscale += logf(B.xE);
      B.xE = 1.0f;
    }
  }
  store_xrow<XMX>(i, lane, A, xrow);
  store_xrow<XMX>(i + 1, lane, B, xrow);
}

#ifndef BATHGPU_V3_WARPS
// resident warps per SM the kernel is compiled for (register budget 65536/(32 n)); measured on B200 per J
// (J = 6: a budget of 13 makes ptxas settle on 128 registers without spilling, 16 resident warps: +2.7 % over 152 registers / 12 warps;
//  J = 5, 8, 10 pushed the same way spill and lose 15-20 %)
#define BATHGPU_V3_WARPS(J) ((J) <= 2 ? 20 : (J) == 3 ? 18 : (J) == 4 ? 16 : (J) == 5 ? 14 : (J) == 6 ? 13 : (J) == 7 ? 10 : (J) == 8 ? 9 : 8)
#endif

#ifndef BATHGPU_V3_RESIDENT
// resident warps per SM the launch aims for (the grid is sized to it; kernels_tu.cu): no cap until measured otherwise
#define BATHGPU_V3_RESIDENT(J) 64
#endif

// SET: the windows of a profile set (FsParserArgs::set), constants and table re-read whenever a warp's next window has another profile
template <int J, bool XMX, int NS = 5, bool SET = false>
__global__ void __launch_bounds__(32, BATHGPU_V3_WARPS(J)) fs3_forward_parser_kernel_v3(FsParserArgs a)
{
  constexpr int VEC = VecOf<J>::V;
  const int lane = threadIdx.x & 31;

  FwdConsts<J> K;
  const char    *emis_lane = nullptr;
  float          tEM = a.tEM, tEL = a.tEL;
  int            cur = -1;
  if constexpr (!SET) {
    load_fwd_consts<J>(a.cellc, lane, K);
    emis_lane = reinterpret_cast<const char *>(a.emis + lane * VEC);
  }
  const unsigned rowbytes  = (unsigned)a.mpad * 4u;

  for (;;) {
    int w = 0;
    if (lane == 0) w = atomicAdd(a.counter, 1);
    w = __shfl_sync(0xffffffffu, w, 0);
    if (w >= a.nwin) break;
    if constexpr (SET) {
      const int p = a.wprof[w];
      if (p != cur) {
        cur = p;
        const FsSetProfile sp = a.set[p];
        load_fwd_consts<J>(sp.cellc, lane, K);
        emis_lane = reinterpret_cast<const char *>(sp.emis + lane * VEC);
        tEM = sp.tEM; tEL = sp.tEL;
      }
    }

    const WindowDesc wd = a.wins[w];
    const int   L     = wd.L;
    const float pmove = wd.pmove, ploop = wd.ploop;
    float *xrow = nullptr;
    if constexpr (XMX) xrow = a.xmx + (size_t)a.xoff[w] * 6;

    FwdState<J> S;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int j = 0; j < J; ++j) { S.W[r][j] = 0.f; S.I[r][j] = 0.f; }
      S.xN[r] = 0.f; S.xJ[r] = 0.f; S.xC[r] = 0.f;
    }
    float totscale = 0.f;

    const int nq  = (L + 4) >> 2;
    const int pad = 4 * nq - (L + 1);
    long long nib = (wd.start - 1) + (long long)(lane - pad - 3) - 1 + 8;
    uint32_t lo = __ldg(a.dna4 + (nib >> 3)), hi = __ldg(a.dna4 + (nib >> 3) + 1);
    int i = -pad;

    // 32 rows per chunk: lane l prepares the codon word of row i + l; the first chunk runs the HEAD instantiation
#define BATHGPU_V3_CHUNK(HEAD_)                                                                                                   \
    {                                                                                                                             \
      const uint32_t cwl = codon_word(lo, hi, (int)(nib & 7) * 4, i + lane, L);                                                   \
      nib += 32;                                                                                                                  \
      if (q0 + 8 < nq) { lo = __ldg(a.dna4 + (nib >> 3)); hi = __ldg(a.dna4 + (nib >> 3) + 1); }                                  \
      const int qn = min(8, nq - q0);                                                                                             \
      for (int qq = 0; qq < qn; ++qq) {                                                                                           \
        const uint32_t c0 = __shfl_sync(0xffffffffu, cwl, qq * 4 + 0);                                                            \
        const uint32_t c1 = __shfl_sync(0xffffffffu, cwl, qq * 4 + 1);                                                            \
        const uint32_t c2 = __shfl_sync(0xffffffffu, cwl, qq * 4 + 2);                                                            \
        const uint32_t c3 = __shfl_sync(0xffffffffu, cwl, qq * 4 + 3);                                                            \
        fwd_row_pair<J, VEC, 0, XMX, NS, HEAD_>(i, lane, S, K, emis_lane, rowbytes, c0, c1, ploop, pmove, tEL, tEM, totscale, xrow); i += 2; \
        fwd_row_pair<J, VEC, 2, XMX, NS, HEAD_>(i, lane, S, K, emis_lane, rowbytes, c2, c3, ploop, pmove, tEL, tEM, totscale, xrow); i += 2; \
      }                                                                                                                           \
    }
    int q0 = 0;
    BATHGPU_V3_CHUNK(true)
    for (q0 = 8; q0 < nq; q0 += 8) BATHGPU_V3_CHUNK(false)
#undef BATHGPU_V3_CHUNK

    {
      float tot = S.xC[3] + S.xC[2] * ploop + S.xC[1] * ploop;
      int   st  = 0;
      float sc;
      if (isnan(tot) || isinf(tot))  { st = 16; sc = tot; }
      else if (L > 2 && tot == 0.0f) { st = 16; sc = -INFINITY; }
      else sc = totscale + logf(tot * pmove);
      if (lane == 0) { a.fwdsc[w] = sc; a.status[w] = st; }
    }
  }
}

}  // namespace bathgpu
