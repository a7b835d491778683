// fs_domain_mw.cuh -- the 5-codon envelope sweeps of fs_domain.cuh for LONG models (J > 32 nodes per lane, M <= 2048): several warps
// per envelope.
//
// The one-warp sweeps keep an envelope's whole row state in one warp's registers; at 48 or 64 nodes per lane that state is 20-100 KB of
// local memory per thread.  Here an envelope belongs to a block of NW = J/8 warps and every lane owns 8 nodes, node k = 8 (32 w + lane)
// + j + 1 -- the decomposition of the multi-warp parsers (fs_parser_mw.cuh, fs_backward_mw.cuh).  Recurrences, row order, scaling and
// the stored matrices are those of fs_domain.cuh: the matrix rows keep the one-warp layout for the profile's J ([cell][J/4][32][4]), so
// fs5_oatrace_kernel, the Forward export and the host read them unchanged.  Virtual lane v reads and writes the two float4 chunks
// 2 (v % NW) and 2 (v % NW) + 1 of real lane v / NW.
//
// Where a row couples the warps:
//   * Forward: E(i) is the sum of the warps' partial sums, and the delete chain enters warp w with X(w-1), X(w) = A31(w) + PW(w) X(w-1)
//     (A31: the warp's own scan with zero carry-in, PW: the product of the D->D odds over its 256 nodes); lane l adds X(w-1) Q(l), Q the
//     product over the lanes in front of it.  One barrier for both, a second one for the flow out of a warp's last node, which is the
//     entry value of the next warp's first node one row later.
//   * Backward: B(i) is the sum of the partial sums; the first product v of warp w+1 is the shifted product vn of warp w's last node,
//     and the downward delete chain enters warp w at its last node.  Every warp runs the chain with both unknowns at zero and publishes
//     B, v(first) and its chain value at its first node, A0(w); with U(w) = v_first(w+1) vdm(k_last) + X(w+1) dd(k_last), X(w) = A0(w)
//     + U(w) PWb(w) (PWb: dd over the warp's nodes but the last) and lane l adds U(w) QU(l) -- fs_backward_mw.cuh's algebra.  One
//     barrier; a second one for the posterior row's denominator.
//   * Optimal accuracy: the same two unknowns in max-plus form.  A warp's D chain is max(its own chain with entry -inf, Y) wherever
//     every D->D transition since its first node is allowed, Y = the D value its first node takes from the previous warp's last M and
//     D cells; a forbidden D->D restarts the chain at a value that does not depend on the entry.  Max is exact, so the cells are the
//     one-warp kernel's bit for bit.  One barrier for the exchange, one for the E maximum.
// Each exchange slot is written before a barrier, read between it and the next one and rewritten only after that next one.  Every
// warp computes the specials from the same shared values in the same order, so the rescale decisions are block-uniform.
#pragma once
#include "fs_domain.cuh"

namespace bathgpu {

constexpr int kMw5NodesPerLane = 8;

template <int NW> struct Mw5Shared {
  float A[NW], E[NW], W[NW], V[NW], M[NW], I[NW];
  float N2[21][NW];
  unsigned pass[NW];
  int   env;
};

// base of virtual lane vl's 8 nodes in a permuted row of the one-warp layout for J = 8 NW (in floats)
template <int NW> __device__ __forceinline__ int mw5_lane_base(int vl) { return ((2 * (vl % NW)) * kWarp + vl / NW) * 4; }

// Forward lane constants, multi-warp image: [F5_COUNT][8][32 NW] per node, [5][32 NW] scan multipliers, [32 NW] Q, [NW] PW
template <int NW>
__device__ __forceinline__ void load_fwd5_consts_mw(const float *__restrict__ cc, int vl, Fwd5Consts<kMw5NodesPerLane> &K, float &Q, float (&PW)[NW])
{
  constexpr int JW = kMw5NodesPerLane, VL = 32 * NW;
#pragma unroll
  for (int j = 0; j < JW; ++j) {
    K.mm[j] = __ldg(cc + (F5_MM * JW + j) * VL + vl);
    K.im[j] = __ldg(cc + (F5_IM * JW + j) * VL + vl);
    K.dm[j] = __ldg(cc + (F5_DM * JW + j) * VL + vl);
    K.md[j] = __ldg(cc + (F5_MD * JW + j) * VL + vl);
    K.dd[j] = __ldg(cc + (F5_DD * JW + j) * VL + vl);
    K.mi[j] = __ldg(cc + (F5_MI * JW + j) * VL + vl);
    K.ii[j] = __ldg(cc + (F5_II * JW + j) * VL + vl);
  }
#pragma unroll
  for (int s = 0; s < 5; ++s) K.bs[s] = __ldg(cc + (F5_COUNT * JW + s) * VL + vl);
  Q = __ldg(cc + (F5_COUNT * JW + 5) * VL + vl);
#pragma unroll
  for (int v = 0; v < NW; ++v) PW[v] = __ldg(cc + (F5_COUNT * JW + 6) * VL + v);
}

// Pull one stored matrix row towards L1 (prefetch_matrix_row for a block of NW warps)
template <int NW>
__device__ __forceinline__ void prefetch_matrix_row_mw(const float *row_base, int ncell, int mpad)
{
#ifndef BATHGPU_NO_ROW_PREFETCH
  const char *p = reinterpret_cast<const char *>(row_base);
  const int nbytes = ncell * mpad * 4;
  for (int off = threadIdx.x * 128; off < nbytes; off += 32 * NW * 128) asm volatile("prefetch.global.L1 [%0];" :: "l"(p + off));
#endif
}

// One Forward row (fwd5_row with the warps coupled)
template <int NW, int PH, bool STORE_D>
__device__ __forceinline__ void fwd5_row_mw(int i, int lane, int warp, Fwd5State<kMw5NodesPerLane> &S, const Fwd5Consts<kMw5NodesPerLane> &K,
                                            float Q, const float (&PW)[NW], Mw5Shared<NW> &sh,
                                            const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t codes,
                                            Fwd5Ctx &R, float *__restrict__ pprow_lane, int mpad,
                                            float *__restrict__ fxrow, float *__restrict__ lsfrow, float *__restrict__ drow_lane)
{
  constexpr int J = kMw5NodesPerLane, VEC = 4;
  constexpr int P0 = PH, P1 = (PH + 4) % 5, P2 = (PH + 3) % 5, P3 = (PH + 2) % 5, P4 = (PH + 1) % 5;
  int c[5];
  codon_rows5(nuc5_of(codes & 7u), nuc5_of((codes >> 3) & 7u), nuc5_of((codes >> 6) & 7u), nuc5_of((codes >> 9) & 7u),
              nuc5_of((codes >> 12) & 7u), c);

  float mc[5][J], m0[J];
  {
    float e[J];
    load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)c[0] * rowbytes), e);
#pragma unroll
    for (int j = 0; j < J; ++j) mc[0][j] = S.W[P0][j] * e[j];
    load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)c[1] * rowbytes), e);
#pragma unroll
    for (int j = 0; j < J; ++j) mc[1][j] = S.W[P1][j] * e[j];
    load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)c[2] * rowbytes), e);
#pragma unroll
    for (int j = 0; j < J; ++j) mc[2][j] = S.W[P2][j] * e[j];
    load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)c[3] * rowbytes), e);
#pragma unroll
    for (int j = 0; j < J; ++j) mc[3][j] = S.W[P3][j] * e[j];
    load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)c[4] * rowbytes), e);
#pragma unroll
    for (int j = 0; j < J; ++j) mc[4][j] = S.W[P4][j] * e[j];
  }
  float es = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    m0[j] = ((mc[0][j] + mc[1][j]) + (mc[2][j] + mc[3][j])) + mc[4][j];
    es += m0[j];
  }
  const float epart = warp_allsum(es);

  float a[J];
  float A = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j) { a[j] = m0[j] * K.md[j]; A = (j == 0) ? a[0] : fmaf(A, K.dd[j], a[j]); }
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    float up = __shfl_up_sync(0xffffffffu, A, 1 << s);
    A = fmaf(K.bs[s], up, A);
  }
  float d = __shfl_up_sync(0xffffffffu, A, 1);
  if (lane == 0) d = 0.f;
  if (lane == 31) sh.A[warp] = A;
  if (lane == 0)  sh.E[warp] = epart;
  __syncthreads();
  float xE = 0.f, X = 0.f;
#pragma unroll
  for (int v = 0; v < NW; ++v) {
    xE += sh.E[v];
    if (v < warp) X = fmaf(PW[v], X, sh.A[v]);
  }
  d = fmaf(X, Q, d);

  float xN = (i < 3) ? ((i >= 0) ? 1.0f : 0.0f) : S.xN[P3] * R.ploop;
  float xJ = fmaf(S.xJ[P3], R.ploop, xE * R.tEL);
  float xC = fmaf(S.xC[P3], R.ploop, xE * R.tEM);
  float xB = fmaf(xJ, R.pmove, xN * R.pmove);

  float o[J], icur[J];
  float dv[STORE_D ? J : 1];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    icur[j] = S.I[P0][j];
    float t = fmaf(icur[j], K.im[j], m0[j] * K.mm[j]);
    o[j] = fmaf(d, K.dm[j], t);
    if constexpr (STORE_D) dv[j] = d;
    if (j + 1 < J) d = fmaf(d, K.dd[j], a[j]);
    S.I[P2][j] = fmaf(icur[j], K.ii[j], m0[j] * K.mi[j]);
  }
  float oprev = __shfl_up_sync(0xffffffffu, o[J - 1], 1);
  if (lane == 0) oprev = 0.f;                      // warps behind the first take their lane 0 entry from shared memory below
  S.W[P4][0] = xB + oprev;
#pragma unroll
  for (int j = 1; j < J; ++j) S.W[P4][j] = xB + o[j - 1];
  float wnext = xB + o[J - 1];

  float scale = 1.0f;
  if (xE > 1.0e4f) {                               // block-uniform
    float sf = 1.0f / xE;
    scale = xE;
    xN *= sf; xJ *= sf; xC *= sf; xB *= sf; wnext *= sf;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
#pragma unroll
      for (int j = 0; j < J; ++j) { S.W[r][j] *= sf; S.I[r][j] *= sf; }
      S.xN[r] *= sf; S.xJ[r] *= sf; S.xC[r] *= sf;
    }
#pragma unroll
    for (int j = 0; j < J; ++j) {
      m0[j] *= sf; icur[j] *= sf;
      if constexpr (STORE_D) dv[j] *= sf;
#pragma unroll
      for (int cc = 0; cc < 5; ++cc) mc[cc][j] *= sf;
    }
    R.totscale += logf(xE);
    xE = 1.0f;
  }
  S.xN[P0] = xN; S.xJ[P0] = xJ; S.xC[P0] = xC;
  if (lane == 31) sh.W[warp] = wnext;

  if (i >= 0) {
    R.lsf = R.lsf + logf(scale);
    float *row = pprow_lane + (size_t)i * kPPCells * mpad;
    store_row<J, VEC>(row + PP_I * mpad, icur);
    store_row<J, VEC>(row + PP_C0 * mpad, m0);
#pragma unroll
    for (int cc = 0; cc < 5; ++cc) store_row<J, VEC>(row + (PP_C0 + 1 + cc) * mpad, mc[cc]);
    if constexpr (STORE_D) store_row<J, VEC>(drow_lane + (size_t)i * mpad, dv);
    if (warp == 0 && lane == 0) {
      float2 *x2 = reinterpret_cast<float2 *>(fxrow + (size_t)i * 6);
      x2[0] = make_float2(xE, xN);
      x2[1] = make_float2(xJ, xB);
      x2[2] = make_float2(xC, scale);
      lsfrow[i] = R.lsf;
    }
  }
  __syncthreads();
  if (lane == 0 && warp > 0) S.W[P4][0] = sh.W[warp - 1];
}

// fs5_forward_kernel for NW warps per envelope.  SET: FsSetProfile::cellmw holds the profile's multi-warp Forward constants.
template <int NW, bool STORE_D = false, bool SET = false>
__global__ void __launch_bounds__(32 * NW) fs5_forward_kernel_mw(DomainArgs a)
{
  constexpr int J = kMw5NodesPerLane;
  __shared__ Mw5Shared<NW> sh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, vl = threadIdx.x;
  const int lb = mw5_lane_base<NW>(vl);
  Fwd5Consts<J> K;
  float Q, PW[NW];
  const char *emis_lane = nullptr;
  float       tEM = a.tEM, tEL = a.tEL;
  int         cur = -1;
  if constexpr (!SET) {
    load_fwd5_consts_mw<NW>(a.cellfmw, vl, K, Q, PW);
    emis_lane = reinterpret_cast<const char *>(a.emis + lb);
  }
  const unsigned rowbytes = (unsigned)a.mpad * 4u;

  for (;;) {
    if (threadIdx.x == 0) sh.env = atomicAdd(a.counter, 1);
    __syncthreads();
    const int e = sh.env;
    __syncthreads();
    if (e >= a.nenv) break;
    if constexpr (SET) {
      const int p = a.wprof[e];
      if (p != cur) {
        cur = p;
        const FsSetProfile sp = a.set[p];
        load_fwd5_consts_mw<NW>(sp.cellmw, vl, K, Q, PW);
        emis_lane = reinterpret_cast<const char *>(sp.emis + lb);
        tEM = sp.tEM; tEL = sp.tEL;
      }
    }
    const EnvelopeDesc ed = a.envs[e];
    const int L = ed.L;
    Fwd5Ctx R;
    R.L = L; R.ploop = ed.ploop; R.pmove = ed.pmove; R.tEL = tEL; R.tEM = tEM; R.totscale = 0.f; R.lsf = 0.f;
    const long long xo = a.xoff[e];
    float *pprow_lane = a.pp + (size_t)xo * kPPCells * a.mpad + lb;
    float *fxrow = a.fx + (size_t)xo * 6;
    float *lsfrow = a.lsf + xo;
    float *drow_lane = STORE_D ? a.dcell + (size_t)xo * a.mpad + lb : nullptr;

    Fwd5State<J> S;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
#pragma unroll
      for (int j = 0; j < J; ++j) { S.W[r][j] = 0.f; S.I[r][j] = 0.f; }
      S.xN[r] = 0.f; S.xJ[r] = 0.f; S.xC[r] = 0.f;
    }

    const int n5  = (L + 5) / 5;
    const int pad = 5 * n5 - (L + 1);
    int i = -pad;
    for (int g0 = 0; g0 < n5; g0 += 6) {
      const uint32_t codes_l = (lane < 30) ? nuc_codes5(a.dna4, ed.start, i + lane - 4, L) : 0u;
      const int gn = min(6, n5 - g0);
      for (int g = 0; g < gn; ++g) {
#define BATHGPU_F5ROW(PH_)                                                                           \
        {                                                                                            \
          uint32_t codes = __shfl_sync(0xffffffffu, codes_l, g * 5 + PH_);                           \
          fwd5_row_mw<NW, PH_, STORE_D>(i, lane, warp, S, K, Q, PW, sh, emis_lane, rowbytes, codes, R, pprow_lane, a.mpad, fxrow, lsfrow, drow_lane); \
          ++i;                                                                                       \
        }
        BATHGPU_F5ROW(0) BATHGPU_F5ROW(1) BATHGPU_F5ROW(2) BATHGPU_F5ROW(3) BATHGPU_F5ROW(4)
#undef BATHGPU_F5ROW
      }
    }
    if (threadIdx.x == 0) {
      float tot = S.xC[4] + S.xC[3] * R.ploop + S.xC[2] * R.ploop;
      int   st  = 0;
      float sc;
      if (isnan(tot) || isinf(tot))  { st = 16; sc = tot; }
      else if (L > 1 && tot == 0.0f) { st = 16; sc = -INFINITY; }
      else sc = R.totscale + logf(tot * R.pmove);
      a.fwdsc[e] = sc; a.status[e] = st;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Backward + decoding + null2 sums.  Backward lane constants, multi-warp image: [BC_COUNT][8][32 NW] per node, [5][32 NW] scan
// multipliers (within a warp), [32 NW] QU, then per warp [NW] PWb, [NW] dd and [NW] vdm of the warp's last node.
template <int NW> struct Bck5MwConsts { float QU, PWb[NW], DDL[NW], VDML[NW]; };

template <int NW>
__device__ __forceinline__ void load_bck5_consts_mw(const float *__restrict__ cc, int vl, BckConsts<kMw5NodesPerLane> &K, Bck5MwConsts<NW> &C)
{
  constexpr int JW = kMw5NodesPerLane, VL = 32 * NW;
#pragma unroll
  for (int j = 0; j < JW; ++j) {
    K.vmm[j] = __ldg(cc + (BC_VMM * JW + j) * VL + vl);
    K.vim[j] = __ldg(cc + (BC_VIM * JW + j) * VL + vl);
    K.vdm[j] = __ldg(cc + (BC_VDM * JW + j) * VL + vl);
    K.dd[j]  = __ldg(cc + (BC_DD  * JW + j) * VL + vl);
    K.md[j]  = __ldg(cc + (BC_MD  * JW + j) * VL + vl);
    K.mi[j]  = __ldg(cc + (BC_MI  * JW + j) * VL + vl);
    K.ii[j]  = __ldg(cc + (BC_II  * JW + j) * VL + vl);
  }
#pragma unroll
  for (int s = 0; s < 5; ++s) K.bs[s] = __ldg(cc + (BC_COUNT * JW + s) * VL + vl);
  C.QU = __ldg(cc + (BC_COUNT * JW + 5) * VL + vl);
  const float *pw = cc + (BC_COUNT * JW + 6) * VL;
#pragma unroll
  for (int v = 0; v < NW; ++v) { C.PWb[v] = __ldg(pw + v); C.DDL[v] = __ldg(pw + NW + v); C.VDML[v] = __ldg(pw + 2 * NW + v); }
}

template <int NW, int PH>
__device__ __forceinline__ void bck5_row_mw(int i, int lane, int warp, Bck5State<kMw5NodesPerLane> &S, const BckConsts<kMw5NodesPerLane> &K,
                                            const Bck5MwConsts<NW> &C, Mw5Shared<NW> &sh,
                                            const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t codes,
                                            Bck5Ctx &R, float *__restrict__ pprow, float *__restrict__ pprow_lane, int mpad,
                                            const float *__restrict__ fxrow, const float *__restrict__ lsfrow,
                                            float *__restrict__ ppxrow, float (&accM)[kMw5NodesPerLane], float (&accI)[kMw5NodesPerLane])
{
  constexpr int J = kMw5NodesPerLane, VEC = 4;
  constexpr int S0 = PH, S1 = (PH + 1) % 5, S2 = (PH + 2) % 5, S3 = (PH + 3) % 5, S4 = (PH + 4) % 5;
  const int L = R.L;
  if (i > L) return;                               // block-uniform
  if (i >= 1) prefetch_matrix_row_mw<NW>(pprow + (size_t)(i - 1) * kPPCells * mpad, kPPCells, mpad);

  float xN, xJ, xC, xB, xE;
  const float fscale = fxrow[(size_t)i * 6 + 5];

  if (i == L) {
    xC = R.pmove; xN = 0.f; xJ = 0.f; xB = 0.f;
    xE = xC * R.tEM;
#pragma unroll
    for (int j = 0; j < J; ++j) { S.Mt[S0][j] = xE; S.I[S0][j] = 0.f; }
    S.xC[S1] = R.pmove; S.xC[S2] = R.pmove;
  } else {
    float v[J];
    {
      const int n1 = nuc5_of(codes & 7u), n2 = nuc5_of((codes >> 3) & 7u), n3 = nuc5_of((codes >> 6) & 7u),
                n4 = nuc5_of((codes >> 9) & 7u), n5 = nuc5_of((codes >> 12) & 7u);
      const int r1 = min(n1 * 341, 1366);
      const int r2 = min(n2 * 341 + n1 * 85 + 1, 1365);
      const int r3 = min(n3 * 341 + n2 * 85 + n1 * 21 + 2, 1364);
      const int r4 = min(n4 * 341 + n3 * 85 + n2 * 21 + n1 * 5 + 3, 1365);
      const int r5 = min(n5 * 341 + n4 * 85 + n3 * 21 + n2 * 5 + n1 + 4, 1366);
      float e[J];
      load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)r1 * rowbytes), e);
#pragma unroll
      for (int j = 0; j < J; ++j) v[j] = S.Mt[S1][j] * e[j];
      load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)r2 * rowbytes), e);
#pragma unroll
      for (int j = 0; j < J; ++j) v[j] = fmaf(S.Mt[S2][j], e[j], v[j]);
      load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)r3 * rowbytes), e);
#pragma unroll
      for (int j = 0; j < J; ++j) v[j] = fmaf(S.Mt[S3][j], e[j], v[j]);
      load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)r4 * rowbytes), e);
#pragma unroll
      for (int j = 0; j < J; ++j) v[j] = fmaf(S.Mt[S4][j], e[j], v[j]);
      load_emission_row<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)r5 * rowbytes), e);
#pragma unroll
      for (int j = 0; j < J; ++j) v[j] = fmaf(S.Mt[S0][j], e[j], v[j]);
    }
    float bsum = 0.f;
#pragma unroll
    for (int j = 0; j < J; ++j) bsum += v[j];
    const float bpart = warp_allsum(bsum);

    // the chain with both unknowns at the warp's upper end (next warp's first v, chain value entering from it) set to zero
    float vn[J];
    {
      float up = __shfl_down_sync(0xffffffffu, v[0], 1);
      if (lane == 31) up = 0.f;
#pragma unroll
      for (int j = 0; j + 1 < J; ++j) vn[j] = v[j + 1];
      vn[J - 1] = up;
    }
    float a[J];
    float A = 0.f;
#pragma unroll
    for (int j = J - 1; j >= 0; --j) { a[j] = vn[j] * K.vdm[j]; A = (j == J - 1) ? a[j] : fmaf(A, K.dd[j], a[j]); }
#pragma unroll
    for (int s = 0; s < 5; ++s) {
      float dn = __shfl_down_sync(0xffffffffu, A, 1 << s);
      A = fmaf(K.bs[s], dn, A);
    }
    float d = __shfl_down_sync(0xffffffffu, A, 1);
    if (lane == 31) d = 0.f;
    if (lane == 0) { sh.E[warp] = bpart; sh.A[warp] = A; sh.V[warp] = v[0]; }
    __syncthreads();
    xB = 0.f;
#pragma unroll
    for (int ww = 0; ww < NW; ++ww) xB += sh.E[ww];

    if (i == 0) {
      xN = fmaf(S.xN[S3], R.ploop, xB * R.pmove);
      S.xN[S0] = xN;
      return;
    }

    // the true values: X(w+1) (chain value at warp w's last node), U(w) (the value leaving that node downwards)
    float Xn = 0.f, U = 0.f;
#pragma unroll
    for (int ww = NW - 1; ww >= 0; --ww) {
      if (ww >= warp) {
        const float vf = (ww + 1 < NW) ? sh.V[ww + 1] : 0.f;
        const float u = fmaf(Xn, C.DDL[ww], vf * C.VDML[ww]);
        if (ww == warp) U = u;
        else Xn = fmaf(u, C.PWb[ww], sh.A[ww]);
      }
    }
    if (lane == 31) {
      vn[J - 1] = (warp + 1 < NW) ? sh.V[warp + 1] : 0.f;
      a[J - 1] = vn[J - 1] * K.vdm[J - 1];
      d = Xn;
    } else {
      d = fmaf(U, C.QU, d);
    }

    xC = S.xC[S3] * R.ploop;
    xJ = fmaf(S.xJ[S3], R.ploop, xB * R.pmove);
    xN = fmaf(S.xN[S3], R.ploop, xB * R.pmove);
    xE = fmaf(xJ, R.tEL, xC * R.tEM);

#pragma unroll
    for (int j = J - 1; j >= 0; --j) {
      float t = S.I[S3][j] * K.mi[j];
      t = fmaf(vn[j], K.vmm[j], t);
      float g = fmaf(d, K.md[j], t);
      d = fmaf(d, K.dd[j], a[j]);
      S.I[S0][j] = fmaf(S.I[S3][j], K.ii[j], vn[j] * K.vim[j]);
      S.Mt[S0][j] = xE + g;
    }
  }

  float scale = fscale;
  if (i < L) {
    if (R.own_scales) scale = (xB > 1.0e4f) ? xB : 1.0f;
    if (xB > 1.0e16f) R.own_scales = true;
  }
  if (scale > 1.0f) {
    float sf = 1.0f / scale;
    xN *= sf; xJ *= sf; xC *= sf; xB *= sf; xE *= sf;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
#pragma unroll
      for (int j = 0; j < J; ++j) { S.Mt[r][j] *= sf; S.I[r][j] *= sf; }
      if (i < L) { S.xN[r] *= sf; S.xJ[r] *= sf; S.xC[r] *= sf; }
    }
    R.totscale += logf(scale);
  }
  S.xN[S0] = xN; S.xJ[S0] = xJ; S.xC[S0] = xC;
  R.lsb = R.lsb + logf(scale);

  float *row = pprow_lane + (size_t)i * kPPCells * mpad;
  float fI[J], f0[J];
  load_row<J, VEC>(row + PP_I * mpad, fI);
  load_row<J, VEC>(row + PP_C0 * mpad, f0);
  float den = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    fI[j] = fI[j] * S.I[S0][j];
    f0[j] = f0[j] * S.Mt[S0][j];
    den += f0[j] + fI[j];
  }
  den = warp_allsum(den);
  if (lane == 0) sh.W[warp] = den;
  __syncthreads();
  float raw_denom = 0.f;
#pragma unroll
  for (int ww = 0; ww < NW; ++ww) raw_denom += sh.W[ww];
  const float lsf_i = lsfrow[i];
  const float factor_mdi = expf(lsf_i + R.lsb + R.liz);
  float N_pp, J_pp, C_pp;
  if (i > 2) {
    const float factor_njc = expf(lsfrow[i - 3] + R.lsb + R.liz);
    const float *f3 = fxrow + (size_t)(i - 3) * 6;
    N_pp = f3[1] * xN * R.ploop * factor_njc;
    J_pp = f3[2] * xJ * R.ploop * factor_njc;
    C_pp = f3[4] * xC * R.ploop * factor_njc;
  } else {
    N_pp = xN * expf(R.lsb + R.liz);
    J_pp = 0.f; C_pp = 0.f;
  }
  const float inv_denom = 1.0f / (raw_denom * factor_mdi + N_pp + J_pp + C_pp);
  if (isinf(factor_mdi) || isinf(inv_denom)) R.st = 16;
  const float scv = factor_mdi * inv_denom;
#pragma unroll
  for (int j = 0; j < J; ++j) { fI[j] *= scv; f0[j] *= scv; accM[j] += f0[j]; accI[j] += fI[j]; }
  store_row<J, VEC>(row + PP_I * mpad, fI);
  store_row<J, VEC>(row + PP_C0 * mpad, f0);
#pragma unroll
  for (int cc = 0; cc < 5; ++cc) {
    float fc[J];
    load_row<J, VEC>(row + (PP_C0 + 1 + cc) * mpad, fc);
#pragma unroll
    for (int j = 0; j < J; ++j) fc[j] = (fc[j] * S.Mt[S0][j]) * scv;
    store_row<J, VEC>(row + (PP_C0 + 1 + cc) * mpad, fc);
  }
  const float pN = N_pp * inv_denom, pJ = J_pp * inv_denom, pC = C_pp * inv_denom;
  R.accN += pN; R.accJ += pJ; R.accC += pC;
  if (warp == 0 && lane == 0) {
    float2 *x2 = reinterpret_cast<float2 *>(ppxrow + (size_t)i * 6);
    x2[0] = make_float2(0.f, pN);
    x2[1] = make_float2(pJ, 0.f);
    x2[2] = make_float2(pC, scale);
  }
}

template <int NW>
__global__ void __launch_bounds__(32 * NW) fs5_backward_decode_kernel_mw(DomainArgs a)
{
  constexpr int J = kMw5NodesPerLane, VEC = 4;
  __shared__ Mw5Shared<NW> sh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, vl = threadIdx.x;
  const int lb = mw5_lane_base<NW>(vl);
  BckConsts<J> K;
  Bck5MwConsts<NW> C;
  load_bck5_consts_mw<NW>(a.cellbmw, vl, K, C);
  const char    *emis_lane = reinterpret_cast<const char *>(a.emis + lb);
  const unsigned rowbytes  = (unsigned)a.mpad * 4u;

  for (;;) {
    if (threadIdx.x == 0) sh.env = atomicAdd(a.counter, 1);
    __syncthreads();
    const int e = sh.env;
    __syncthreads();
    if (e >= a.nenv) break;
    if (a.status[e] != 0) { if (threadIdx.x == 0) a.bcksc[e] = -INFINITY; continue; }
    const EnvelopeDesc ed = a.envs[e];
    const int L = ed.L;
    const long long xo = a.xoff[e];
    float *pprow = a.pp + (size_t)xo * kPPCells * a.mpad;
    float *pprow_lane = pprow + lb;
    const float *fxrow = a.fx + (size_t)xo * 6;
    const float *lsfrow = a.lsf + xo;
    float *ppxrow = a.ppx + (size_t)xo * 6;

    Bck5Ctx R;
    R.L = L; R.ploop = ed.ploop; R.pmove = ed.pmove; R.tEL = a.tEL; R.tEM = a.tEM;
    R.totscale = 0.f; R.lsb = 0.f; R.liz = -a.fwdsc[e]; R.own_scales = false; R.st = 0;
    R.accN = 0.f; R.accJ = 0.f; R.accC = 0.f;

    Bck5State<J> S;
    float accM[J], accI[J];
#pragma unroll
    for (int j = 0; j < J; ++j) { accM[j] = 0.f; accI[j] = 0.f; }
#pragma unroll
    for (int r = 0; r < 5; ++r) {
#pragma unroll
      for (int j = 0; j < J; ++j) { S.Mt[r][j] = 0.f; S.I[r][j] = 0.f; }
      S.xN[r] = 0.f; S.xJ[r] = 0.f; S.xC[r] = 0.f;
    }

    const int n5 = (L + 5) / 5;
    int i = 5 * n5 - 1;
    for (int g0 = 0; g0 < n5; g0 += 6) {
      const uint32_t codes_l = (lane < 30 && i - lane >= 0) ? nuc_codes5(a.dna4, ed.start, i - lane + 1, L) : 0u;
      const int gn = min(6, n5 - g0);
      for (int g = 0; g < gn; ++g) {
#define BATHGPU_B5ROW(PH_)                                                                           \
        {                                                                                            \
          uint32_t codes = __shfl_sync(0xffffffffu, codes_l, g * 5 + (4 - PH_));                     \
          bck5_row_mw<NW, PH_>(i, lane, warp, S, K, C, sh, emis_lane, rowbytes, codes, R, pprow, pprow_lane, a.mpad, fxrow, lsfrow, ppxrow, accM, accI); \
          --i;                                                                                       \
        }
        BATHGPU_B5ROW(4) BATHGPU_B5ROW(3) BATHGPU_B5ROW(2) BATHGPU_B5ROW(1) BATHGPU_B5ROW(0)
#undef BATHGPU_B5ROW
      }
    }

    {
      float tot = S.xN[0] + S.xN[1] + S.xN[2];
      float sc;
      if (isnan(tot) || isinf(tot)) { R.st = 16; sc = tot; }
      else if (tot == 0.0f)         { R.st = 16; sc = -INFINITY; }
      else sc = R.totscale + logf(tot);
      if (threadIdx.x == 0) { a.bcksc[e] = sc; if (R.st) a.status[e] = R.st; }
    }
    {
      float z[J];
#pragma unroll
      for (int j = 0; j < J; ++j) z[j] = 0.f;
#pragma unroll
      for (int cc = 0; cc < kPPCells; ++cc) store_row<J, VEC>(pprow_lane + (size_t)cc * a.mpad, z);
      if (threadIdx.x == 0) { for (int s = 0; s < 6; ++s) ppxrow[s] = 0.f; }
    }

    // null2 by expectation: the warps' partial sums through shared memory, finished by warp 0
    {
      const float norm = 1.0f / (float)L;
      const float xfactor = R.accN * norm + R.accC * norm + R.accJ * norm;
      float isum = 0.f;
#pragma unroll
      for (int j = 0; j < J; ++j) { accM[j] *= norm; accI[j] *= norm; isum += accI[j]; }
      isum = warp_allsum(isum);
      if (lane == 0) sh.N2[20][warp] = isum;
      for (int x = 0; x < 20; ++x) {
        float r[J];
        load_emission_row<J, VEC>(a.amino + (size_t)x * a.mpad + lb, r);
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < J; ++j) s = fmaf(accM[j], r[j], s);
        s = warp_allsum(s);
        if (lane == 0) sh.N2[x][warp] = s;
      }
      __syncthreads();
      if (warp == 0) {
        float itot = 0.f, n2 = 0.f;
#pragma unroll
        for (int ww = 0; ww < NW; ++ww) itot += sh.N2[20][ww];
        if (lane < 20) {
#pragma unroll
          for (int ww = 0; ww < NW; ++ww) n2 += sh.N2[lane][ww];
          n2 = n2 + itot + xfactor;
        }
        float out = 1.0f;
        const unsigned full = 0xffffffffu;
        float vals[20];
#pragma unroll
        for (int x = 0; x < 20; ++x) vals[x] = __shfl_sync(full, n2, x);
        if (lane < 20) out = n2;
        else if (lane == 21) out = (vals[2] + vals[11]) / 2.0f;
        else if (lane == 22) out = (vals[7] + vals[9]) / 2.0f;
        else if (lane == 23) out = (vals[3] + vals[13]) / 2.0f;
        else if (lane == 24) out = vals[8];
        else if (lane == 25) out = vals[1];
        else if (lane == 26) { float s = 0.f;
#pragma unroll
          for (int x = 0; x < 20; ++x) s += vals[x];
          out = s / 20.0f; }
        if (lane < 29) a.null2[(size_t)e * 29 + lane] = out;
      }
      __syncthreads();             // sh.N2 is rewritten by the next envelope
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Optimal-accuracy fill (oa_row with the warps coupled).  ppass: every D->D from the warp's first node up to this lane's first node is
// allowed (the warp's entry value Y reaches this lane's carry); dd0 / md0 / wpass per warp: the D->D and M->D masks of the warp's first
// node and whether every D->D after it inside the warp is allowed.
struct Oa5MwLane { bool ppass; float dpass[5]; };

template <int NW, int PH>
__device__ __forceinline__ void oa_row_mw(int i, int lane, int warp, OAState<kMw5NodesPerLane> &S, const uint32_t (&fl)[kMw5NodesPerLane],
                                          const Oa5MwLane &P, const bool (&dd0)[NW], const bool (&md0)[NW], const bool (&wpass)[NW],
                                          Mw5Shared<NW> &sh, const float *__restrict__ pprow, const float *__restrict__ pprow_lane,
                                          float *__restrict__ oarow_lane, int mpad,
                                          const float *__restrict__ ppxrow, float *__restrict__ oaxrow, int M, int J0,
                                          bool loopN, bool loopJ, bool loopC, bool loopE, bool moveE, bool moveN, bool moveJ)
{
  constexpr int J = kMw5NodesPerLane, VEC = 4;
  constexpr int P0 = PH, P1 = (PH + 4) % 5, P2 = (PH + 3) % 5, P3 = (PH + 2) % 5, P4 = (PH + 1) % 5;
  if (i < 1) return;
  const float *row = pprow_lane + (size_t)i * kPPCells * mpad;
  prefetch_matrix_row_mw<NW>(pprow + (size_t)(i + 1) * kPPCells * mpad, kPPCells, mpad);
  float pc[J], mnew[J], inew[J];
  load_row<J, VEC>(row + (PP_C0 + 1) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) mnew[j] = S.P[P1][j] + pc[j];
  float t2[J];
  load_row<J, VEC>(row + (PP_C0 + 2) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) mnew[j] = oa_max(mnew[j], S.P[P2][j] + pc[j]);
  load_row<J, VEC>(row + (PP_C0 + 3) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) t2[j] = S.P[P3][j] + pc[j];
  load_row<J, VEC>(row + (PP_C0 + 4) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) t2[j] = oa_max(t2[j], S.P[P4][j] + pc[j]);
  load_row<J, VEC>(row + (PP_C0 + 5) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) {
    t2[j] = oa_max(t2[j], S.P[P0][j] + pc[j]);
    mnew[j] = oa_max(mnew[j], t2[j]);
  }
  load_row<J, VEC>(row + PP_I * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) {
    float s = oa_mask(fl[j], OF_MI, S.Mr[P3][j]);
    s = oa_max(s, oa_mask(fl[j], OF_II, S.Ir[P3][j]));
    inew[j] = s + pc[j];
    const int k = J0 + j + 1;
    if (k == M) inew[j] = -INFINITY;
    if (k > M)  { inew[j] = -INFINITY; mnew[j] = -INFINITY; }
  }

  // D: the warp's own chain with entry -inf (oa_row's lane-serial pass and scan), then the entry from the previous warp
  float dnew[J];
  float mprev = __shfl_up_sync(0xffffffffu, mnew[J - 1], 1);
  if (lane == 0) mprev = -INFINITY;
  float carry;
  {
    float dd_ = -INFINITY, mm_ = mprev;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      float dv = oa_max(oa_mask(fl[j], OF_DD, dd_), oa_mask(fl[j], OF_MD, mm_));
      const int k = J0 + j + 1;
      if (k == 1) dv = -INFINITY;
      dd_ = dv; mm_ = mnew[j];
    }
    float A = dd_;
#pragma unroll
    for (int s = 0; s < 5; ++s) {
      float up = __shfl_up_sync(0xffffffffu, A, 1 << s);
      if (lane >= (1 << s) && P.dpass[s] != 0.f) A = oa_max(A, up);
    }
    carry = __shfl_up_sync(0xffffffffu, A, 1);
    if (lane == 0) carry = -INFINITY;
    if (lane == 31) { sh.A[warp] = A; sh.M[warp] = mnew[J - 1]; sh.I[warp] = inew[J - 1]; }
  }
  __syncthreads();
  float Xd = -INFINITY, Y = -INFINITY;             // D at the previous warp's last node; D that warp hands this warp's first node
#pragma unroll
  for (int v = 0; v < NW; ++v) {
    if (v <= warp) {
      const float y = (v == 0) ? -INFINITY : oa_max(dd0[v] ? Xd : -INFINITY, md0[v] ? sh.M[v - 1] : -INFINITY);
      if (v == warp) Y = y;
      else Xd = wpass[v] ? oa_max(sh.A[v], y) : sh.A[v];
    }
  }
  float mm_ = mprev;
  if (lane == 0) { if (warp > 0) { carry = Xd; mm_ = sh.M[warp - 1]; } }
  else if (P.ppass) carry = oa_max(carry, Y);
  {
    float dd_ = carry;
#pragma unroll
    for (int j = 0; j < J; ++j) {
      float dv = oa_max(oa_mask(fl[j], OF_DD, dd_), oa_mask(fl[j], OF_MD, mm_));
      const int k = J0 + j + 1;
      if (k == 1) dv = -INFINITY;
      if (k > M)  dv = -INFINITY;
      dnew[j] = dv;
      dd_ = dv; mm_ = mnew[j];
    }
  }

  float e = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j) e = oa_max(e, oa_max(mnew[j], dnew[j]));
#pragma unroll
  for (int dlt = 16; dlt >= 1; dlt >>= 1) e = oa_max(e, __shfl_xor_sync(0xffffffffu, e, dlt));

  // the previous warp's last M and I cells feed this warp's first node in the rows to come: read before the slots can be rewritten
  float mp = __shfl_up_sync(0xffffffffu, mnew[J - 1], 1);
  float ip = __shfl_up_sync(0xffffffffu, inew[J - 1], 1);
  float dp = __shfl_up_sync(0xffffffffu, dnew[J - 1], 1);
  if (lane == 0) {
    if (warp == 0) { mp = -INFINITY; ip = -INFINITY; dp = -INFINITY; }      // column 0 is -inf (:110-112)
    else { mp = sh.M[warp - 1]; ip = sh.I[warp - 1]; dp = Xd; }
  }
  if (lane == 0) sh.E[warp] = e;
  __syncthreads();
  float xE = sh.E[0];
#pragma unroll
  for (int v = 1; v < NW; ++v) xE = oa_max(xE, sh.E[v]);

  const float ppN = ppxrow[(size_t)i * 6 + 1], ppJ = ppxrow[(size_t)i * 6 + 2], ppC = ppxrow[(size_t)i * 6 + 4];
  float xN, xJ, xC, xB;
  if (i > 2) {
    xN = loopN ? S.xN[P3] + ppN : 0.0f;
    float t1 = loopJ ? S.xJ[P3] + ppJ : 0.0f, t2e = loopE ? xE : 0.0f;
    xJ = (t1 > t2e) ? t1 : t2e;
    t1 = loopC ? S.xC[P3] + ppC : 0.0f; t2e = moveE ? xE : 0.0f;
    xC = (t1 > t2e) ? t1 : t2e;
  } else {
    xN = loopN ? ppN : 0.0f;
    xJ = loopE ? xE : 0.0f;
    xC = moveE ? xE : 0.0f;
  }
  {
    float t1 = moveN ? xN : 0.0f, t2e = moveJ ? xJ : 0.0f;
    xB = (t1 > t2e) ? t1 : t2e;
  }
  S.xN[P0] = xN; S.xJ[P0] = xJ; S.xC[P0] = xC;
  // P(i)[k] for the rows to come: predecessors at node k-1 of this row
#pragma unroll
  for (int j = 0; j < J; ++j) {
    float s = oa_mask(fl[j], OF_BM, xB);
    s = oa_max(s, oa_mask(fl[j], OF_MM, mp));
    s = oa_max(s, oa_mask(fl[j], OF_IM, ip));
    s = oa_max(s, oa_mask(fl[j], OF_DM, dp));
    S.P[P0][j] = s;
    mp = mnew[j]; ip = inew[j]; dp = dnew[j];
  }
#pragma unroll
  for (int j = 0; j < J; ++j) { S.Mr[P0][j] = mnew[j]; S.Ir[P0][j] = inew[j]; }

  float *orow = oarow_lane + (size_t)i * kOACells * mpad;
  store_row<J, VEC>(orow + OA_M * mpad, mnew);
  store_row<J, VEC>(orow + OA_I * mpad, inew);
  store_row<J, VEC>(orow + OA_D * mpad, dnew);
  if (warp == 0 && lane == 0) {
    float2 *x2 = reinterpret_cast<float2 *>(oaxrow + (size_t)i * 6);
    x2[0] = make_float2(xE, xN);
    x2[1] = make_float2(xJ, xB);
    x2[2] = make_float2(xC, 0.f);
  }
}

template <int NW>
__global__ void __launch_bounds__(32 * NW) fs5_optacc_kernel_mw(DomainArgs a)
{
  constexpr int J = kMw5NodesPerLane, VEC = 4;
  __shared__ Mw5Shared<NW> sh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, vl = threadIdx.x;
  const int lb = mw5_lane_base<NW>(vl);
  const int J0 = vl * J, M = a.M;
  uint32_t fl[J];
#pragma unroll
  for (int j = 0; j < J; ++j) fl[j] = a.oaflags[J0 + j];
  // D->D pass-through flags (the loader's oapass, here for 8-node lanes): whole lane, and the lane without its first node
  bool lp = true, lp1 = true;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const bool ok = (J0 + j + 1 > M) || (fl[j] & OF_DD);
    lp = lp && ok;
    if (j > 0) lp1 = lp1 && ok;
  }
  Oa5MwLane P;
  {
    bool cur = lp;
#pragma unroll
    for (int s = 0; s < 5; ++s) {
      const int d = 1 << s;
      const bool upv = __shfl_up_sync(0xffffffffu, cur, d);
      P.dpass[s] = (lane >= d && cur) ? 1.0f : 0.0f;
      if (lane >= d) cur = cur && upv;
    }
    const unsigned bits = __ballot_sync(0xffffffffu, (lane == 0) ? lp1 : lp);
    const unsigned below = (lane == 0) ? 0u : ((1u << lane) - 1u);
    P.ppass = (bits & below) == below;
    if (lane == 0) sh.pass[warp] = bits;
  }
  __syncthreads();
  bool dd0[NW], md0[NW], wpass[NW];
#pragma unroll
  for (int v = 0; v < NW; ++v) {
    const uint32_t f0 = a.oaflags[256 * v];
    dd0[v] = (f0 & OF_DD) != 0; md0[v] = (f0 & OF_MD) != 0; wpass[v] = sh.pass[v] == 0xffffffffu;
  }

  for (;;) {
    __syncthreads();
    if (threadIdx.x == 0) sh.env = atomicAdd(a.counter, 1);
    __syncthreads();
    const int e = sh.env;
    if (e >= a.nenv) break;
    if (a.status[e] != 0) { if (threadIdx.x == 0) a.oasc[e] = -INFINITY; continue; }
    const EnvelopeDesc ed = a.envs[e];
    const int L = ed.L;
    const long long xo = a.xoff[e];
    const float *pprow = a.pp + (size_t)xo * kPPCells * a.mpad;
    const float *pprow_lane = pprow + lb;
    float *oarow_lane = a.oa + (size_t)xo * kOACells * a.mpad + lb;
    const float *ppxrow = a.ppx + (size_t)xo * 6;
    float *oaxrow = a.oax + (size_t)xo * 6;
    const bool loopN = ed.ploop != 0.f, loopJ = ed.ploop != 0.f, loopC = ed.ploop != 0.f;
    const bool moveN = ed.pmove != 0.f, moveJ = ed.pmove != 0.f;
    const bool loopE = a.tEL != 0.f, moveE = a.tEM != 0.f;

    OAState<J> S;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
#pragma unroll
      for (int j = 0; j < J; ++j) {
        float s = oa_mask(fl[j], OF_BM, (r == 0) ? 0.0f : -INFINITY);
        s = oa_max(s, oa_mask(fl[j], OF_MM, -INFINITY));
        s = oa_max(s, oa_mask(fl[j], OF_IM, -INFINITY));
        s = oa_max(s, oa_mask(fl[j], OF_DM, -INFINITY));
        S.P[r][j] = s; S.Mr[r][j] = -INFINITY; S.Ir[r][j] = -INFINITY;
      }
      S.xN[r] = 0.f; S.xJ[r] = -INFINITY; S.xC[r] = -INFINITY;
    }
    {
      float ninf[J];
#pragma unroll
      for (int j = 0; j < J; ++j) ninf[j] = -INFINITY;
#pragma unroll
      for (int cc = 0; cc < kOACells; ++cc) store_row<J, VEC>(oarow_lane + (size_t)cc * a.mpad, ninf);
      if (threadIdx.x == 0) { oaxrow[0] = -INFINITY; oaxrow[1] = 0.f; oaxrow[2] = -INFINITY; oaxrow[3] = 0.f; oaxrow[4] = -INFINITY; oaxrow[5] = 0.f; }
    }

    const int n5 = (L + 5) / 5;
    int i = 0;
    for (int g = 0; g < n5; ++g) {
#define BATHGPU_OAROW(PH_)                                                                                      \
      { if (i <= L) oa_row_mw<NW, PH_>(i, lane, warp, S, fl, P, dd0, md0, wpass, sh, pprow, pprow_lane, oarow_lane, a.mpad, \
                                       ppxrow, oaxrow, M, J0, loopN, loopJ, loopC, loopE, moveE, moveN, moveJ); \
        ++i; }
      BATHGPU_OAROW(0) BATHGPU_OAROW(1) BATHGPU_OAROW(2) BATHGPU_OAROW(3) BATHGPU_OAROW(4)
#undef BATHGPU_OAROW
    }
    __syncthreads();
    if (threadIdx.x == 0)
      a.oasc[e] = oaxrow[(size_t)L * 6 + 4] + oaxrow[(size_t)(L - 1) * 6 + 4] + oaxrow[(size_t)(L - 2) * 6 + 4];
  }
}

}  // namespace bathgpu
