// fs_parser_mw.cuh -- frameshift Forward parser for LONG models (384 < M <= 1024): several warps per window.
//
// The one-warp kernels keep a window's whole row state in one warp's registers; beyond 12 nodes per lane ptxas moves part of it to
// local memory and the kernel falls from 1.0-1.3 TCUPS to 0.23 at M = 903.  Here a window belongs to a block of NW = 2..4 warps and
// every lane owns JW = 8 nodes (the best-running register footprint of fs_parser_v3.cuh), node k = 8 (32 w + lane) + j + 1.  The
// recurrence, the folded table, the scaled chains and the row-pair schedule are those of fs_parser_v3.cuh; what is new is the two
// places where a DP row couples the warps:
//   * E(i) is the sum of the warps' partial sums, and the delete chain's carry into warp w is the chain value at the end of warp
//     w-1: X(w) = A31(w) + PW(w) X(w-1), with A31 the warp's own scan result (zero carry-in) and PW the product of the D->D odds
//     over the warp's 256 nodes -- a profile constant; lane l then takes X(w-1) Q(l) on top of its local inflow, Q(l) = the same
//     product over the lanes in front of it.  One barrier per row pair (both rows' values go through shared memory together);
//   * the flow out of a warp's last node is the entry value of the next warp's first node: a second barrier per pair.
// Each exchange slot is written before a barrier, read after it and rewritten only after the next barrier (racecheck: 0 hazards).
// The specials (N, J, C, B) are computed redundantly by every warp from the same E, so the rescale decision is block-uniform.
// The emission table is the one-warp kernels' (J = 8 NW nodes per lane, [J/4][32][4] floats per row): virtual lane v = 32 w + lane
// reads the two float4 of chunks 2 (v % (J/8)) .. +1 of real lane v / (J/8), 128 contiguous bytes per 8 lanes.
#pragma once
#include "fs_parser_v3.cuh"

namespace bathgpu {

// lane-constant image of the multi-warp kernel: [5 JW + 6][32 NW] floats (qm, dm, dd, hi, ii per node; 5 scan multipliers; Q), then PW[NW]

template <int NW> struct MwShared {
  float A[2][NW], E[2][NW], W[2][NW];
  int   win;
};

// first half of a row: emissions, match values, the warp's E partial and its delete-chain scan with zero carry-in
// the three table rows of one DP row, this lane's 8 nodes.  The table of a long model (1.1-1.5 MB) lives in L2 and 42 % of the
// stall samples of the first version waited for these loads, so they are issued one row pair ahead: the next pair's rows travel
// while this pair sits at its barriers.
template <int JW> struct MwRows { float e2[JW], e3[JW], e4[JW]; };
template <int JW>
__device__ __forceinline__ void mw_load_rows(const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t cw, MwRows<JW> &R)
{
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw & 511u) * rowbytes), R.e2);
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)((cw >> 9) & 511u) * rowbytes), R.e3);
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw >> 18) * rowbytes), R.e4);
}

template <int JW, int PH, int NS>
__device__ __forceinline__ void mw_row_front(const FwdState<JW> &S, const FwdConsts<JW> &K, const MwRows<JW> &T,
                                             float (&m)[JW], float &epart, float &A, float &dloc)
{
  constexpr int P0 = PH, P1 = (PH + 3) & 3, P2 = (PH + 2) & 3;
  const float (&e2)[JW] = T.e2, (&e3)[JW] = T.e3, (&e4)[JW] = T.e4;
  float es0 = 0.f, es1 = 0.f;
#pragma unroll
  for (int j = 0; j < JW; ++j) {
    float t = S.W[P2][j] * e4[j];
    t = fmaf(S.W[P1][j], e3[j], t);
    t = fmaf(S.W[P0][j], e2[j], t);
    m[j] = t;
    if (j == 0) es0 = t * K.qm[0]; else if (j == 1) es1 = t * K.qm[1]; else if (j & 1) es1 = fmaf(t, K.qm[j], es1); else es0 = fmaf(t, K.qm[j], es0);
  }
  epart = warp_allsum(es0 + es1);
  A = m[0];
#pragma unroll
  for (int j = 1; j < JW; ++j) A = fmaf(A, K.dd[j], m[j]);
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    float up = __shfl_up_sync(0xffffffffu, A, 1 << s);
    A = fmaf(K.bs[s], up, A);
  }
  dloc = __shfl_up_sync(0xffffffffu, A, 1);
}

// Also measured and dropped: both rows' E shares reduced in one butterfly (upper half-warp row i+1, lower row i: 5 shuffles for 10)
// together with a 2-step scan: 452 vs 458 GCUPS at M = 903, 468 vs 519 at M = 624.
// Requesting the next pair's six table rows towards L1 with prefetch instructions instead of loading them early was measured first and
// LOSES 6-11 % (404 vs 429 GCUPS at M = 903): off.
#ifndef BATHGPU_MW_PREFETCH
#define BATHGPU_MW_PREFETCH 0
#endif
__device__ __forceinline__ void mw_prefetch_rows(const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t cw)
{
  const char *p2 = emis_lane + (size_t)(cw & 511u) * rowbytes, *p3 = emis_lane + (size_t)((cw >> 9) & 511u) * rowbytes,
             *p4 = emis_lane + (size_t)(cw >> 18) * rowbytes;
  asm volatile("prefetch.global.L1 [%0];" :: "l"(p2));  asm volatile("prefetch.global.L1 [%0];" :: "l"(p2 + 512));
  asm volatile("prefetch.global.L1 [%0];" :: "l"(p3));  asm volatile("prefetch.global.L1 [%0];" :: "l"(p3 + 512));
  asm volatile("prefetch.global.L1 [%0];" :: "l"(p4));  asm volatile("prefetch.global.L1 [%0];" :: "l"(p4 + 512));
}

// second half: specials from the block-wide E, the chains replayed from the true inflow, the outflow into row i+2
template <int JW, int PH, bool HEAD>
__device__ __forceinline__ void mw_row_back(int i, int lane, FwdState<JW> &S, const FwdConsts<JW> &K, const float (&m)[JW], float xE, float d,
                                            float ploop, float pmove, float tEL, float tEM, RowOut &R, float &wnext)
{
  constexpr int P0 = PH, P1 = (PH + 3) & 3, P2 = (PH + 2) & 3, P3 = (PH + 1) & 3;
  float xN = S.xN[P3] * ploop;
  if constexpr (HEAD) xN = (i < 3) ? ((i >= 0) ? 1.0f : 0.0f) : xN;
  float xJ = fmaf(S.xJ[P3], ploop, xE * tEL);
  float xC = fmaf(S.xC[P3], ploop, xE * tEM);
  float xB = fmaf(xJ, pmove, xN * pmove);
  float o[JW];
#pragma unroll
  for (int j = 0; j < JW; ++j) {
    float t = fmaf(S.I[P0][j], K.hi[j], m[j]);
    o[j] = fmaf(d, K.dm[j], t);
    if (j + 1 < JW) d = fmaf(d, K.dd[j], m[j]);
    S.I[P1][j] = fmaf(S.I[P0][j], K.ii[j], m[j]);
  }
  float oprev = __shfl_up_sync(0xffffffffu, o[JW - 1], 1);
  if (lane == 0) oprev = 0.f;                       // warps behind the first one take their lane 0 entry from shared memory after the pair
  S.W[P2][0] = xB + oprev;
#pragma unroll
  for (int j = 1; j < JW; ++j) S.W[P2][j] = xB + o[j - 1];
  wnext = xB + o[JW - 1];                                // lane 31: entry value of the next warp's first node
  S.xN[P0] = xN; S.xJ[P0] = xJ; S.xC[P0] = xC;
  R.xE = xE; R.xN = xN; R.xJ = xJ; R.xC = xC; R.xB = xB; R.scale = 1.0f;
}

template <int NW, int JW, int PH, bool XMX, int NS, bool HEAD>
__device__ __forceinline__ void mw_row_pair(int i, int lane, int warp, FwdState<JW> &S, const FwdConsts<JW> &K, float Q, const float (&PW)[NW],
                                            MwShared<NW> &sh, const char *__restrict__ emis_lane, unsigned rowbytes, MwRows<JW> &TA, MwRows<JW> &TB,
                                            uint32_t cwNA, uint32_t cwNB, bool have_next, float ploop, float pmove, float tEL, float tEM, float &totscale, float *__restrict__ xrow)
{
  constexpr int P2A = (PH + 2) & 3, P2B = (PH + 3) & 3;
  float mA[JW], mB[JW], eA, eB, aA, aB, dA, dB;
  mw_row_front<JW, PH, NS>(S, K, TA, mA, eA, aA, dA);
  mw_row_front<JW, PH + 1, NS>(S, K, TB, mB, eB, aB, dB);
  if (have_next) { mw_load_rows<JW>(emis_lane, rowbytes, cwNA, TA); mw_load_rows<JW>(emis_lane, rowbytes, cwNB, TB); }   // consumed by the next pair
  if (lane == 31) { sh.A[0][warp] = aA; sh.A[1][warp] = aB; }
  if (lane == 0)  { sh.E[0][warp] = eA; sh.E[1][warp] = eB; dA = 0.f; dB = 0.f; }
  if (BATHGPU_MW_PREFETCH && have_next) { mw_prefetch_rows(emis_lane, rowbytes, cwNA); mw_prefetch_rows(emis_lane, rowbytes, cwNB); }
  __syncthreads();
  float xEA = 0.f, xEB = 0.f, XA = 0.f, XB = 0.f;
#pragma unroll
  for (int v = 0; v < NW; ++v) {
    xEA += sh.E[0][v]; xEB += sh.E[1][v];
    if (v < warp) { XA = fmaf(PW[v], XA, sh.A[0][v]); XB = fmaf(PW[v], XB, sh.A[1][v]); }
  }
  dA = fmaf(XA, Q, dA); dB = fmaf(XB, Q, dB);
  RowOut A, B;
  float wnA, wnB;
  mw_row_back<JW, PH, HEAD>(i, lane, S, K, mA, xEA, dA, ploop, pmove, tEL, tEM, A, wnA);
  mw_row_back<JW, PH + 1, HEAD>(i + 1, lane, S, K, mB, xEB, dB, ploop, pmove, tEL, tEM, B, wnB);
  if (__builtin_expect(A.xE > 1.0e4f || B.xE > 1.0e4f, 0)) {          // rare, block-uniform
    if (A.xE > 1.0e4f) {
      const float sf = 1.0f / A.xE;
      scale_state<JW>(S, sf); wnA *= sf; wnB *= sf;
      A.scale = A.xE; A.xN *= sf; A.xJ *= sf; A.xC *= sf; A.xB *= sf;
      B.xE *= sf; B.xN *= sf; B.xJ *= sf; B.xC *= sf; B.xB *= sf;
      totscale += logf(A.xE);
      A.xE = 1.0f;
    }
    if (B.xE > 1.0e4f) {
      const float sf = 1.0f / B.xE;
      scale_state<JW>(S, sf); wnA *= sf; wnB *= sf;
      B.scale = B.xE; B.xN *= sf; B.xJ *= sf; B.xC *= sf; B.xB *= sf;
      totscale += logf(B.xE);
      B.xE = 1.0f;
    }
  }
  if (lane == 31) { sh.W[0][warp] = wnA; sh.W[1][warp] = wnB; }
  if (warp == 0) { store_xrow<XMX>(i, lane, A, xrow); store_xrow<XMX>(i + 1, lane, B, xrow); }
  __syncthreads();
  if (lane == 0 && warp > 0) { S.W[P2A][0] = sh.W[0][warp - 1]; S.W[P2B][0] = sh.W[1][warp - 1]; }
}

// JW nodes per lane, NW warps per window (32 NW JW >= M).  Resident blocks per SM the kernel is compiled for.
template <int NW, int JW> struct MwTune { static constexpr int kBlocks = (JW == 8) ? ((NW == 4) ? 2 : (NW == 3) ? 2 : 4) : ((NW >= 5) ? 2 : 4); };

template <int NW, int JW>
__device__ __forceinline__ void mw_load_consts(const float *__restrict__ cc, int vl, FwdConsts<JW> &K, float &Q, float (&PW)[NW])
{
  constexpr int VL = 32 * NW;
#pragma unroll
  for (int j = 0; j < JW; ++j) {
    K.qm[j] = __ldg(cc + (0 * JW + j) * VL + vl);
    K.dm[j] = __ldg(cc + (1 * JW + j) * VL + vl);
    K.dd[j] = __ldg(cc + (2 * JW + j) * VL + vl);
    K.hi[j] = __ldg(cc + (3 * JW + j) * VL + vl);
    K.ii[j] = __ldg(cc + (4 * JW + j) * VL + vl);
  }
#pragma unroll
  for (int s = 0; s < 5; ++s) K.bs[s] = __ldg(cc + (5 * JW + s) * VL + vl);
  Q = __ldg(cc + (5 * JW + 5) * VL + vl);
#pragma unroll
  for (int v = 0; v < NW; ++v) PW[v] = __ldg(cc + (5 * JW + 6) * VL + v);
}

// SET: as in fs3_forward_parser_kernel_v3 (the block's warps share one window, hence one profile)
template <int NW, int JW, bool XMX, int NS, bool SET = false>
__global__ void __launch_bounds__(32 * NW, MwTune<NW, JW>::kBlocks) fs3_forward_parser_kernel_mw(FsParserArgs a)
{
  __shared__ MwShared<NW> sh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, vl = threadIdx.x;

  FwdConsts<JW> K;
  float Q;
  float PW[NW];
  // this thread's JW nodes are JW/4 consecutive float4 chunks of real lane (JW vl) / (NW JW) of the one-warp table layout
  const int node0 = JW * vl, rl = node0 / (NW * JW), c0 = (node0 % (NW * JW)) / 4;
  const char    *emis_lane = nullptr;
  float          tEM = a.tEM, tEL = a.tEL;
  int            cur = -1;
  if constexpr (!SET) {
    mw_load_consts<NW, JW>(a.cellmw, vl, K, Q, PW);
    emis_lane = reinterpret_cast<const char *>(a.emis + ((size_t)c0 * 32 + rl) * 4);
  }
  const unsigned rowbytes  = (unsigned)a.mpad * 4u;

  for (;;) {
    if (threadIdx.x == 0) sh.win = atomicAdd(a.counter, 1);
    __syncthreads();
    const int w = sh.win;
    __syncthreads();
    if (w >= a.nwin) break;
    if constexpr (SET) {
      const int p = a.wprof[w];
      if (p != cur) {
        cur = p;
        const FsSetProfile sp = a.set[p];
        mw_load_consts<NW, JW>(sp.cellmw, vl, K, Q, PW);
        emis_lane = reinterpret_cast<const char *>(sp.emis + ((size_t)c0 * 32 + rl) * 4);
        tEM = sp.tEM; tEL = sp.tEL;
      }
    }

    const WindowDesc wd = a.wins[w];
    const int   L     = wd.L;
    const float pmove = wd.pmove, ploop = wd.ploop;
    float *xrow = nullptr;
    if constexpr (XMX) xrow = a.xmx + (size_t)a.xoff[w] * 6;

    FwdState<JW> S;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int j = 0; j < JW; ++j) { S.W[r][j] = 0.f; S.I[r][j] = 0.f; }
      S.xN[r] = 0.f; S.xJ[r] = 0.f; S.xC[r] = 0.f;
    }
    float totscale = 0.f;

    const int nq  = (L + 4) >> 2;
    const int pad = 4 * nq - (L + 1);
    long long nib = (wd.start - 1) + (long long)(lane - pad - 3) - 1 + 8;
    uint32_t lo = __ldg(a.dna4 + (nib >> 3)), hi = __ldg(a.dna4 + (nib >> 3) + 1);
    int i = -pad;

    // 32 rows per chunk: lane l prepares the codon word of row i + l; the next chunk's words are made one chunk ahead so that the
    // last pair of a chunk can request the first rows of the next one
    uint32_t cwl = codon_word(lo, hi, (int)(nib & 7) * 4, i + lane, L);
    nib += 32;
    if (8 < nq) { lo = __ldg(a.dna4 + (nib >> 3)); hi = __ldg(a.dna4 + (nib >> 3) + 1); }
    MwRows<JW> TA, TB;
    mw_load_rows<JW>(emis_lane, rowbytes, __shfl_sync(0xffffffffu, cwl, 0), TA);
    mw_load_rows<JW>(emis_lane, rowbytes, __shfl_sync(0xffffffffu, cwl, 1), TB);
#define BATHGPU_MW_CHUNK(HEAD_)                                                                                                   \
    {                                                                                                                             \
      const bool more = q0 + 8 < nq;                                                                                              \
      uint32_t cwn = 0;                                                                                                           \
      if (more) {                                                                                                                 \
        cwn = codon_word(lo, hi, (int)(nib & 7) * 4, i + 32 + lane, L);                                                           \
        nib += 32;                                                                                                                \
        if (q0 + 16 < nq) { lo = __ldg(a.dna4 + (nib >> 3)); hi = __ldg(a.dna4 + (nib >> 3) + 1); }                               \
      }                                                                                                                           \
      const int qn = min(8, nq - q0);                                                                                             \
      for (int qq = 0; qq < qn; ++qq) {                                                                                           \
        const uint32_t c2 = __shfl_sync(0xffffffffu, cwl, qq * 4 + 2);                                                            \
        const uint32_t c3 = __shfl_sync(0xffffffffu, cwl, qq * 4 + 3);                                                            \
        const uint32_t src = (qq < 7) ? cwl : cwn;                                                                                \
        const uint32_t n0 = __shfl_sync(0xffffffffu, src, (qq * 4 + 4) & 31);                                                     \
        const uint32_t n1 = __shfl_sync(0xffffffffu, src, (qq * 4 + 5) & 31);                                                     \
        mw_row_pair<NW, JW, 0, XMX, NS, HEAD_>(i, lane, warp, S, K, Q, PW, sh, emis_lane, rowbytes, TA, TB, c2, c3, true, ploop, pmove, tEL, tEM, totscale, xrow); i += 2; \
        mw_row_pair<NW, JW, 2, XMX, NS, HEAD_>(i, lane, warp, S, K, Q, PW, sh, emis_lane, rowbytes, TA, TB, n0, n1, (qq + 1 < qn) || more, ploop, pmove, tEL, tEM, totscale, xrow); i += 2; \
      }                                                                                                                           \
      cwl = cwn;                                                                                                                  \
    }
    int q0 = 0;
    BATHGPU_MW_CHUNK(true)
    for (q0 = 8; q0 < nq; q0 += 8) BATHGPU_MW_CHUNK(false)
#undef BATHGPU_MW_CHUNK

    if (threadIdx.x == 0) {
      float tot = S.xC[3] + S.xC[2] * ploop + S.xC[1] * ploop;
      int   st  = 0;
      float sc;
      if (isnan(tot) || isinf(tot))  { st = 16; sc = tot; }
      else if (L > 2 && tot == 0.0f) { st = 16; sc = -INFINITY; }
      else sc = totscale + logf(tot * pmove);
      a.fwdsc[w] = sc; a.status[w] = st;
    }
  }
}

}  // namespace bathgpu
