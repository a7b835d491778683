// fs_backward_mw.cuh -- frameshift Backward parser for LONG models (M > 512): several warps per window.
//
// The multi-warp twin of fs3_backward_parser_kernel (fs_backward.cuh), built the way fs_parser_mw.cuh splits the Forward parser: a
// window belongs to a block of NW = J/8 warps, virtual lane vl = 32 w + lane owns the 8 nodes 8 vl + 1 .. 8 vl + 8, recurrence,
// folded table copy and scaled chains are the one-warp kernel's.  A Backward row couples the warps in three places, and all three go
// through ONE barrier per row:
//   * B(i) is the sum of the warps' partial sums;
//   * the shifted product vn(k) = v(k+1) of a warp's last node is the first product v of the next warp;
//   * the downward delete chain Ds(k) = vn(k) + Ds(k+1) dd(k) enters a warp at its last node with what the next warp's chain holds at
//     its first node.
// Every warp first runs its row with both unknowns at its upper end set to zero and publishes its partial B sum, its first product
// and its chain value at its first node, A0(w).  The chain is linear in the unknowns: with U(w) = v_first(w+1) + X(w+1) dd(k_last(w))
// -- the true chain value at the warp's last node -- the value at its first node is X(w) = A0(w) + U(w) PWb(w), PWb = product of dd over
// the warp's nodes but the last, and lane l's inflow grows by U(w) QU(l), QU = product of dd from the first node of lane l+1 to the
// warp's last node but one.  All warps evaluate that (NW <= 4 terms) from the same published values after the barrier, so B, the
// specials and the rescale decisions are block-uniform.  Two rows (i and i-1, which are independent of each other: the row-pair schedule
// of the one-warp kernel) go through one barrier together.  Exchange slots alternate between two sets from barrier to barrier: a slot
// is rewritten two barriers later, i.e. behind a barrier every warp has passed after reading it.
#pragma once
#include "fs_backward.cuh"

namespace bathgpu {

template <int NW> struct MwBckShared {
  float B[2][2][NW], A[2][2][NW], V[2][2][NW];      // [exchange set][row of the pair][warp]
  int   win;
};

template <int NW, int JW, int PH>
__device__ __forceinline__ void mw_bck_row(int i, int lane, int warp, BckState<JW> &S, const Bck3Consts<JW> &K, float QU,
                                           const float (&PWb)[NW], const float (&DDL)[NW], MwBckShared<NW> &sh,
                                           const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t cw, float fscale,
                                           BckRowCtx &R, float *__restrict__ xrow, int &xchg)
{
  constexpr int S0 = PH, S1 = (PH + 1) & 3, S2 = (PH + 2) & 3, S3 = (PH + 3) & 3;   // slots of rows i(=i+4), i+1, i+2, i+3
  const int L = R.L;
  const bool writer = (warp == 0 && lane == 0);

  if (i >= L - 1) {                 // block-uniform: pad rows above L do nothing, rows L and L-1 initialise (fwdback_fs.c:628-690)
    if (i <= L) {
      float xC = (i == L) ? R.pmove : R.ploop * R.pmove;
      float xE = xC * R.tEM;
      const float sc = fscale;
      if (sc > 1.0f) {
        const float sf = 1.0f / sc;
        xC *= sf; xE *= sf;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
#pragma unroll
          for (int j = 0; j < JW; ++j) { S.Mt[r][j] *= sf; S.I[r][j] *= sf; }
        }
        R.totscale += logf(sc);
      }
#pragma unroll
      for (int j = 0; j < JW; ++j) { S.Mt[S0][j] = xE; S.I[S0][j] = 0.f; }
      S.xN[S0] = 0.f; S.xJ[S0] = 0.f; S.xC[S0] = xC;
      if (i == L) S.xC[S1] = R.pmove;
      if (writer) {
        float2 *x2 = reinterpret_cast<float2 *>(xrow + (size_t)i * 6);
        x2[0] = make_float2(xE, 0.f);
        x2[1] = make_float2(0.f, 0.f);
        x2[2] = make_float2(xC, sc);
      }
    }
    return;
  }

  const int p = xchg & 1;           // exchange-slot set of this barrier
  xchg ^= 1;
  float e2[JW], e3[JW], e4[JW], v[JW];
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw & 511u) * rowbytes), e2);
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)((cw >> 9) & 511u) * rowbytes), e3);
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw >> 18) * rowbytes), e4);
  float bs0 = 0.f, bs1 = 0.f;
#pragma unroll
  for (int j = 0; j < JW; ++j) {
    float t = S.Mt[S2][j] * e2[j];
    t = fmaf(S.Mt[S3][j], e3[j], t);
    t = fmaf(S.Mt[S0][j], e4[j], t);
    v[j] = t;
    if (j == 0) bs0 = t * K.qb[0]; else if (j == 1) bs1 = t * K.qb[1]; else if (j & 1) bs1 = fmaf(t, K.qb[j], bs1); else bs0 = fmaf(t, K.qb[j], bs0);
  }
  const float bpart = warp_allsum(bs0 + bs1);

  float vn[JW];
  {
    float up = __shfl_down_sync(0xffffffffu, v[0], 1);
    if (lane == 31) up = 0.f;                           // the next warp's first product: unknown until the barrier
#pragma unroll
    for (int j = 0; j + 1 < JW; ++j) vn[j] = v[j + 1];
    vn[JW - 1] = up;
  }
  float A = 0.f;
#pragma unroll
  for (int j = JW - 1; j >= 0; --j) A = (j == JW - 1) ? vn[j] : fmaf(A, K.dd[j], vn[j]);
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    float dn = __shfl_down_sync(0xffffffffu, A, 1 << s);
    A = fmaf(K.bs[s], dn, A);
  }
  float d = __shfl_down_sync(0xffffffffu, A, 1);        // chain value at the first node of the next lane, zero inflow at the warp's end
  if (lane == 31) d = 0.f;
  if (lane == 0) { sh.B[p][0][warp] = bpart; sh.A[p][0][warp] = A; sh.V[p][0][warp] = v[0]; }
  __syncthreads();

  float xB = 0.f, Xn = 0.f, Uown = 0.f, Xnext = 0.f, vfnext = 0.f;
#pragma unroll
  for (int ww = 0; ww < NW; ++ww) xB += sh.B[p][0][ww];
#pragma unroll
  for (int ww = NW - 1; ww >= 0; --ww) {
    const float vf = (ww + 1 < NW) ? sh.V[p][0][ww + 1] : 0.f;
    const float U  = fmaf(Xn, DDL[ww], vf);
    if (ww == warp) { Uown = U; Xnext = Xn; vfnext = vf; }
    Xn = fmaf(U, PWb[ww], sh.A[p][0][ww]);
  }
  d = fmaf(Uown, QU, d);
  if (lane == 31) { d = Xnext; vn[JW - 1] = vfnext; }

  float g[JW];
#pragma unroll
  for (int j = JW - 1; j >= 0; --j) {
    float t = fmaf(S.I[S3][j], K.mi[j], vn[j]);
    g[j] = fmaf(d, K.md[j], t);
    d = fmaf(d, K.dd[j], vn[j]);
    S.I[S0][j] = fmaf(S.I[S3][j], K.ii[j], vn[j]);
  }
  float xC = S.xC[S3] * R.ploop;
  float xJ = fmaf(S.xJ[S3], R.ploop, xB * R.pmove);
  float xN = fmaf(S.xN[S3], R.ploop, xB * R.pmove);
  float xE = fmaf(xJ, R.tEL, xC * R.tEM);
#pragma unroll
  for (int j = 0; j < JW; ++j) S.Mt[S0][j] = xE + g[j];

  if (i == 0) {                     // termination (:951-987): only B and N are defined on row 0, no rescaling
    S.xN[S0] = xN;
    if (writer) {
      float2 *x2 = reinterpret_cast<float2 *>(xrow);
      x2[0] = make_float2(0.f, xN);
      x2[1] = make_float2(0.f, xB);
      x2[2] = make_float2(0.f, 1.0f);
    }
    return;
  }
  float scale = fscale;
  if (i < L - 2) {                  // (:910-916)
    if (xB > 1.0e16f) R.own_scales = true;
    if (R.own_scales) scale = (xB > 1.0e4f) ? xB : 1.0f;
  }
  if (scale > 1.0f) {               // block-uniform
    const float sf = 1.0f / scale;
    xN *= sf; xJ *= sf; xC *= sf; xB *= sf; xE *= sf;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int j = 0; j < JW; ++j) { S.Mt[r][j] *= sf; S.I[r][j] *= sf; }
      S.xN[r] *= sf; S.xJ[r] *= sf; S.xC[r] *= sf;
    }
    R.totscale += logf(scale);
  }
  S.xN[S0] = xN; S.xJ[S0] = xJ; S.xC[S0] = xC;
  if (writer) {
    float2 *x2 = reinterpret_cast<float2 *>(xrow + (size_t)i * 6);
    x2[0] = make_float2(xE, xN);
    x2[1] = make_float2(xJ, xB);
    x2[2] = make_float2(xC, scale);
  }
}

// ---- rows i (phase PH) and i-1 (phase PH-1) through one barrier (the row-pair schedule of fs_backward.cuh: row i-1 reads rows
// i+1 .. i+3 only, so both rows are computed from the same state and row i's rescaling is applied afterwards to what row i-1 produced)
template <int JW> struct MwBckFront { float vn[JW]; float d, bpart, A, v0; };

template <int JW, int PH>
__device__ __forceinline__ void mw_bck_front(int lane, const BckState<JW> &S, const Bck3Consts<JW> &K, const char *__restrict__ emis_lane,
                                             unsigned rowbytes, uint32_t cw, MwBckFront<JW> &F)
{
  constexpr int S0 = PH, S2 = (PH + 2) & 3, S3 = (PH + 3) & 3;
  float e2[JW], e3[JW], e4[JW], v[JW];
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw & 511u) * rowbytes), e2);
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)((cw >> 9) & 511u) * rowbytes), e3);
  load_emission_row<JW, 4>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw >> 18) * rowbytes), e4);
  float bs0 = 0.f, bs1 = 0.f;
#pragma unroll
  for (int j = 0; j < JW; ++j) {
    float t = S.Mt[S2][j] * e2[j];
    t = fmaf(S.Mt[S3][j], e3[j], t);
    t = fmaf(S.Mt[S0][j], e4[j], t);
    v[j] = t;
    if (j == 0) bs0 = t * K.qb[0]; else if (j == 1) bs1 = t * K.qb[1]; else if (j & 1) bs1 = fmaf(t, K.qb[j], bs1); else bs0 = fmaf(t, K.qb[j], bs0);
  }
  F.bpart = warp_allsum(bs0 + bs1);
  F.v0 = v[0];
  float up = __shfl_down_sync(0xffffffffu, v[0], 1);
  if (lane == 31) up = 0.f;
#pragma unroll
  for (int j = 0; j + 1 < JW; ++j) F.vn[j] = v[j + 1];
  F.vn[JW - 1] = up;
  float A = 0.f;
#pragma unroll
  for (int j = JW - 1; j >= 0; --j) A = (j == JW - 1) ? F.vn[j] : fmaf(A, K.dd[j], F.vn[j]);
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    float dn = __shfl_down_sync(0xffffffffu, A, 1 << s);
    A = fmaf(K.bs[s], dn, A);
  }
  F.A = A;
  F.d = __shfl_down_sync(0xffffffffu, A, 1);
  if (lane == 31) F.d = 0.f;
}

template <int NW, int JW, int PH>
__device__ __forceinline__ BckOut mw_bck_back(int lane, int warp, BckState<JW> &S, const Bck3Consts<JW> &K, float QU, const float (&PWb)[NW],
                                              const float (&DDL)[NW], const float (&sB)[NW], const float (&sA)[NW], const float (&sV)[NW],
                                              MwBckFront<JW> &F, const BckRowCtx &R)
{
  constexpr int S0 = PH, S3 = (PH + 3) & 3;
  float xB = 0.f, Xn = 0.f, Uown = 0.f, Xnext = 0.f, vfnext = 0.f;
#pragma unroll
  for (int ww = 0; ww < NW; ++ww) xB += sB[ww];
#pragma unroll
  for (int ww = NW - 1; ww >= 0; --ww) {
    const float vf = (ww + 1 < NW) ? sV[ww + 1] : 0.f;
    const float U  = fmaf(Xn, DDL[ww], vf);
    if (ww == warp) { Uown = U; Xnext = Xn; vfnext = vf; }
    Xn = fmaf(U, PWb[ww], sA[ww]);
  }
  float d = fmaf(Uown, QU, F.d);
  if (lane == 31) { d = Xnext; F.vn[JW - 1] = vfnext; }
  float g[JW];
#pragma unroll
  for (int j = JW - 1; j >= 0; --j) {
    float t = fmaf(S.I[S3][j], K.mi[j], F.vn[j]);
    g[j] = fmaf(d, K.md[j], t);
    d = fmaf(d, K.dd[j], F.vn[j]);
    S.I[S0][j] = fmaf(S.I[S3][j], K.ii[j], F.vn[j]);
  }
  float xC = S.xC[S3] * R.ploop;
  float xJ = fmaf(S.xJ[S3], R.ploop, xB * R.pmove);
  float xN = fmaf(S.xN[S3], R.ploop, xB * R.pmove);
  float xE = fmaf(xJ, R.tEL, xC * R.tEM);
#pragma unroll
  for (int j = 0; j < JW; ++j) S.Mt[S0][j] = xE + g[j];
  return BckOut{ xB, xN, xJ, xC, xE };
}

template <int NW, int JW, int PH>
__device__ __forceinline__ void mw_bck_row_pair(int i, int lane, int warp, BckState<JW> &S, const Bck3Consts<JW> &K, float QU,
                                                const float (&PWb)[NW], const float (&DDL)[NW], MwBckShared<NW> &sh,
                                                const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t cwA, uint32_t cwB,
                                                float fsA, float fsB, BckRowCtx &R, float *__restrict__ xrow, int &xchg)
{
  static_assert(PH == 3 || PH == 1, "pairs start on odd phases");
  const int p = xchg & 1;
  xchg ^= 1;
  MwBckFront<JW> FA, FB;
  mw_bck_front<JW, PH>(lane, S, K, emis_lane, rowbytes, cwA, FA);
  mw_bck_front<JW, PH - 1>(lane, S, K, emis_lane, rowbytes, cwB, FB);
  if (lane == 0) {
    sh.B[p][0][warp] = FA.bpart; sh.A[p][0][warp] = FA.A; sh.V[p][0][warp] = FA.v0;
    sh.B[p][1][warp] = FB.bpart; sh.A[p][1][warp] = FB.A; sh.V[p][1][warp] = FB.v0;
  }
  __syncthreads();
  BckOut A = mw_bck_back<NW, JW, PH>(lane, warp, S, K, QU, PWb, DDL, sh.B[p][0], sh.A[p][0], sh.V[p][0], FA, R);
  BckOut B = mw_bck_back<NW, JW, PH - 1>(lane, warp, S, K, QU, PWb, DDL, sh.B[p][1], sh.A[p][1], sh.V[p][1], FB, R);
  const int L = R.L;
  auto rescale_all = [&](float sf) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int j = 0; j < JW; ++j) { S.Mt[r][j] *= sf; S.I[r][j] *= sf; }
      S.xN[r] *= sf; S.xJ[r] *= sf; S.xC[r] *= sf;
    }
  };
  float scaleA = fsA;
  if (i < L - 2) {
    if (A.xB > 1.0e16f) R.own_scales = true;
    if (R.own_scales) scaleA = (A.xB > 1.0e4f) ? A.xB : 1.0f;
  }
  if (scaleA > 1.0f) {             // block-uniform
    const float sf = 1.0f / scaleA;
    A.xN *= sf; A.xJ *= sf; A.xC *= sf; A.xB *= sf; A.xE *= sf;
    B.xN *= sf; B.xJ *= sf; B.xC *= sf; B.xB *= sf; B.xE *= sf;
    rescale_all(sf);
    R.totscale += logf(scaleA);
  }
  S.xN[PH] = A.xN; S.xJ[PH] = A.xJ; S.xC[PH] = A.xC;
  float scaleB = fsB;
  if (i - 1 < L - 2) {
    if (B.xB > 1.0e16f) R.own_scales = true;
    if (R.own_scales) scaleB = (B.xB > 1.0e4f) ? B.xB : 1.0f;
  }
  if (scaleB > 1.0f) {
    const float sf = 1.0f / scaleB;
    B.xN *= sf; B.xJ *= sf; B.xC *= sf; B.xB *= sf; B.xE *= sf;
    rescale_all(sf);
    R.totscale += logf(scaleB);
  }
  S.xN[PH - 1] = B.xN; S.xJ[PH - 1] = B.xJ; S.xC[PH - 1] = B.xC;
  if (warp == 0 && lane == 0) {
    float2 *x2 = reinterpret_cast<float2 *>(xrow + (size_t)i * 6);
    x2[0] = make_float2(A.xE, A.xN);
    x2[1] = make_float2(A.xJ, A.xB);
    x2[2] = make_float2(A.xC, scaleA);
    x2 = reinterpret_cast<float2 *>(xrow + (size_t)(i - 1) * 6);
    x2[0] = make_float2(B.xE, B.xN);
    x2[1] = make_float2(B.xJ, B.xB);
    x2[2] = make_float2(B.xC, scaleB);
  }
}

// constant image (bathgpu.cu, cellbmw): [5 JW + 6][32 NW] floats (qb, dd, md, mi, ii per node; 5 scan multipliers; QU), then PWb[NW], DDL[NW]
// two blocks a multiprocessor up to NW = 4, one from NW = 6 up (two blocks allow 170 or 128 registers a thread there: 92 and 124 bytes spilled)
template <int NW, int JW>
__global__ void __launch_bounds__(32 * NW, (NW >= 5) ? 1 : 2) fs3_backward_parser_kernel_mw(FsBackwardArgs a)
{
  __shared__ MwBckShared<NW> sh;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, vl = threadIdx.x;
  constexpr int VL = 32 * NW;

  Bck3Consts<JW> K;
  const float *cc = a.cellbmw;
#pragma unroll
  for (int j = 0; j < JW; ++j) {
    K.qb[j] = __ldg(cc + (0 * JW + j) * VL + vl);
    K.dd[j] = __ldg(cc + (1 * JW + j) * VL + vl);
    K.md[j] = __ldg(cc + (2 * JW + j) * VL + vl);
    K.mi[j] = __ldg(cc + (3 * JW + j) * VL + vl);
    K.ii[j] = __ldg(cc + (4 * JW + j) * VL + vl);
  }
#pragma unroll
  for (int s = 0; s < 5; ++s) K.bs[s] = __ldg(cc + (5 * JW + s) * VL + vl);
  const float QU = __ldg(cc + (5 * JW + 5) * VL + vl);
  float PWb[NW], DDL[NW];
#pragma unroll
  for (int v = 0; v < NW; ++v) { PWb[v] = __ldg(cc + (5 * JW + 6) * VL + v); DDL[v] = __ldg(cc + (5 * JW + 6) * VL + NW + v); }
  const int node0 = JW * vl, rl = node0 / (NW * JW), c0 = (node0 % (NW * JW)) / 4;
  const char    *emis_lane = reinterpret_cast<const char *>(a.emis + ((size_t)c0 * 32 + rl) * 4);
  const unsigned rowbytes  = (unsigned)a.mpad * 4u;

  for (;;) {
    if (threadIdx.x == 0) sh.win = atomicAdd(a.counter, 1);
    __syncthreads();
    const int w = sh.win;
    __syncthreads();
    if (w >= a.nwin) break;

    const WindowDesc wd = a.wins[w];
    BckRowCtx R;
    R.L = wd.L; R.ploop = wd.ploop; R.pmove = wd.pmove; R.tEL = a.tEL; R.tEM = a.tEM;
    R.totscale = 0.f; R.own_scales = false;
    const float *fx   = a.fxmx + (size_t)a.xoff[w] * 6;
    float       *xrow = a.bxmx + (size_t)a.xoff[w] * 6;
    const int L = wd.L;

    BckState<JW> S;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int j = 0; j < JW; ++j) { S.Mt[r][j] = 0.f; S.I[r][j] = 0.f; }
      S.xN[r] = 0.f; S.xJ[r] = 0.f; S.xC[r] = 0.f;
    }

    const int nq = (L + 4) >> 2;
    int i = 4 * nq - 1;
    int xchg = 0;                                        // exchange-slot set of the next barrier (toggles with every barrier, block-uniform)
    for (int q0 = 0; q0 < nq; q0 += 8) {
      const int myrow = i - lane;                        // every warp prepares the same 32 rows
      uint32_t cwl = 0;
      float    fsl = 1.0f;
      if (myrow >= 0) {
        long long nib = (wd.start - 1) + (long long)myrow + 8;
        uint32_t lo = __ldg(a.dna4 + (nib >> 3)), hi = __ldg(a.dna4 + (nib >> 3) + 1);
        cwl = codon_word_bck(lo, hi, (int)(nib & 7) * 4, myrow, L);
        if (myrow <= L) fsl = __ldg(fx + (size_t)myrow * 6 + 5);
      }
      const int qn = min(8, nq - q0);
      for (int qq = 0; qq < qn; ++qq) {
#define BATHGPU_MWB_PAIR(PH_)                                                                                              \
        {                                                                                                                  \
          const int srcA = qq * 4 + (3 - PH_), srcB = srcA + 1;                                                            \
          const uint32_t cwA = __shfl_sync(0xffffffffu, cwl, srcA), cwB = __shfl_sync(0xffffffffu, cwl, srcB);             \
          const float    fsA = __shfl_sync(0xffffffffu, fsl, srcA), fsB = __shfl_sync(0xffffffffu, fsl, srcB);             \
          if (i <= L - 2 && i >= 2) mw_bck_row_pair<NW, JW, PH_>(i, lane, warp, S, K, QU, PWb, DDL, sh, emis_lane, rowbytes, cwA, cwB, fsA, fsB, R, xrow, xchg); \
          else {                                                                                                           \
            mw_bck_row<NW, JW, PH_>(i, lane, warp, S, K, QU, PWb, DDL, sh, emis_lane, rowbytes, cwA, fsA, R, xrow, xchg);  \
            mw_bck_row<NW, JW, PH_ - 1>(i - 1, lane, warp, S, K, QU, PWb, DDL, sh, emis_lane, rowbytes, cwB, fsB, R, xrow, xchg); \
          }                                                                                                                \
          i -= 2;                                                                                                          \
        }
        BATHGPU_MWB_PAIR(3) BATHGPU_MWB_PAIR(1)
#undef BATHGPU_MWB_PAIR
      }
    }
    if (threadIdx.x == 0) {
      float tot = S.xN[0] + S.xN[1] + S.xN[2];
      int   st  = 0;
      float sc;
      if (isnan(tot) || isinf(tot)) { st = 16; sc = tot; }
      else if (tot == 0.0f)         { st = 16; sc = -INFINITY; }
      else sc = R.totscale + logf(tot);
      a.bcksc[w] = sc; if (st) a.status[w] = st;
    }
  }
}

}  // namespace bathgpu
