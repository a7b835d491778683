// fs_parser_v4.cuh -- frameshift Forward parser, row-pair schedule on packed FP32 (FFMA2 / FMUL2 / FADD2).
//
// Same recurrence, carried quantities, tables and constants as fs_parser_v3.cuh (read fs_parser.cuh's header first).
// The v3 kernel is issue-bound: 113 warp-instructions per DP row at J = 6, 74 of them floating point, so even at full
// issue rate the FP32 pipe would be 52 % busy.  Blackwell's packed FP32 instructions do two FMAs per issue slot on an
// aligned register pair, and take a single register as a broadcast operand in any position (FFMA2 Rd, Ra.F32x2, Rb.F32, Rc.F32x2),
// so this kernel keeps every per-node array as pairs of NEIGHBOURING NODES (j, j+1) -- the layout the 64-bit table loads
// already deliver -- and issues one packed instruction per node pair wherever the work is elementwise over nodes:
//   * the match sum            m  = W(i-4) e4 + W(i-3) e3 + W(i-2) e2          3 per pair instead of 6
//   * the E partial sums       es = sum m qm                                    1 per pair instead of 2
//   * insert chain, outflow    t = Ih hi + m,  o = d dm + t,  Ih' = Ih ii + m   3 per pair instead of 6
// What stays scalar is what is serial over nodes: the lane-local delete chain A(j) = A(j-1) dd(j) + m(j).  The second
// serial pass of v3 (the chain re-run from the lane's true inflow) is replaced by d(j) = inflow * pd(j) + A(j-1) with
// pd(j) = dd(0) .. dd(j-1), a packed FMA per pair with the inflow as broadcast operand (the recurrence is linear).
// The E sums of the two rows of a pair are reduced together: one exchange puts row A's partials in the lower half-warp
// and row B's in the upper one, four butterfly steps finish both, two broadcasts hand them out (7 shuffles instead of 10).
// FP issue slots per row at J = 6: 74 -> 46.
#pragma once
#include "fs_parser_v3.cuh"

namespace bathgpu {

// packed FP32 (sm_100: FFMA2 / FMUL2 / FADD2); -ftz=true applies as to the scalar instructions
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 fmul2(float2 a, float2 b)           { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fadd2(float2 a, float2 b)           { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 bcast2(float x) { return make_float2(x, x); }     // ptxas turns this into a .F32 broadcast operand

// node pairs (2p, 2p+1) for p < JP, plus one scalar tail node when J is odd
template <int J> struct Pairs { static constexpr int JP = J / 2; static constexpr bool TAIL = (J & 1) != 0; static constexpr int NT = TAIL ? 1 : 1; };

template <int J>
struct FwdState4 {
  float2 W[4][Pairs<J>::JP > 0 ? Pairs<J>::JP : 1];
  float2 I[3][Pairs<J>::JP > 0 ? Pairs<J>::JP : 1];     // slot = row mod 3: Ih(i+3) overwrites Ih(i) in place
  float  Wt[4], It[3];                       // tail node (odd J)
  float  xN[4], xJ[4], xC[4];
};

template <int J>
struct FwdConsts4 {
  float2 qm[Pairs<J>::JP > 0 ? Pairs<J>::JP : 1], dm[Pairs<J>::JP > 0 ? Pairs<J>::JP : 1], hi[Pairs<J>::JP > 0 ? Pairs<J>::JP : 1],
         ii[Pairs<J>::JP > 0 ? Pairs<J>::JP : 1], pd[Pairs<J>::JP > 0 ? Pairs<J>::JP : 1];
  float  qmt, dmt, hit, iit, pdt;            // tail node
  float  dd[J];                              // serial chain multipliers
  float  bs[5];
};

template <int J>
__device__ __forceinline__ void load_fwd_consts4(const float *__restrict__ cc, int lane, FwdConsts4<J> &K)
{
  constexpr int JP = Pairs<J>::JP;
  float qm[J], dm[J], hi[J], ii[J], pd[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    qm[j]   = __ldg(cc + (FC_MM * J + j) * kWarp + lane);
    dm[j]   = __ldg(cc + (FC_DM * J + j) * kWarp + lane);
    K.dd[j] = __ldg(cc + (FC_DD * J + j) * kWarp + lane);
    hi[j]   = __ldg(cc + (FC_MI * J + j) * kWarp + lane);
    ii[j]   = __ldg(cc + (FC_II * J + j) * kWarp + lane);
  }
  pd[0] = 1.0f;
#pragma unroll
  for (int j = 1; j < J; ++j) pd[j] = pd[j - 1] * K.dd[j - 1];
#pragma unroll
  for (int p = 0; p < JP; ++p) {
    K.qm[p] = make_float2(qm[2 * p], qm[2 * p + 1]); K.dm[p] = make_float2(dm[2 * p], dm[2 * p + 1]);
    K.hi[p] = make_float2(hi[2 * p], hi[2 * p + 1]); K.ii[p] = make_float2(ii[2 * p], ii[2 * p + 1]);
    K.pd[p] = make_float2(pd[2 * p], pd[2 * p + 1]);
  }
  K.qmt = qm[J - 1]; K.dmt = dm[J - 1]; K.hit = hi[J - 1]; K.iit = ii[J - 1]; K.pdt = pd[J - 1];
#pragma unroll
  for (int s = 0; s < 5; ++s) K.bs[s] = __ldg(cc + FC_COUNT * J * kWarp + (FL_B0 + s) * kWarp + lane);
}

// emission row as node pairs (+ tail)
template <int J, int VEC>
__device__ __forceinline__ void load_emission_pairs(const float *__restrict__ row, float2 (&e)[Pairs<J>::JP > 0 ? Pairs<J>::JP : 1], float &et)
{
  constexpr int JP = Pairs<J>::JP;
  if constexpr (VEC == 4) {
#pragma unroll
    for (int g = 0; g < J / 4; ++g) {
      float4 t = __ldg(reinterpret_cast<const float4 *>(row) + g * kWarp);
      e[2 * g] = make_float2(t.x, t.y); e[2 * g + 1] = make_float2(t.z, t.w);
    }
  } else if constexpr (VEC == 2) {
#pragma unroll
    for (int g = 0; g < JP; ++g) e[g] = __ldg(reinterpret_cast<const float2 *>(row) + g * kWarp);
  } else {
    float s[J];
#pragma unroll
    for (int g = 0; g < J; ++g) s[g] = __ldg(row + g * kWarp);
#pragma unroll
    for (int p = 0; p < JP; ++p) e[p] = make_float2(s[2 * p], s[2 * p + 1]);
    et = s[J - 1];
  }
}

// first half of a row -- everything that does not wait for E(i): table loads, match values, this lane's partial E sum, the insert
// chain (t = Ih hi + m is the outflow without its delete term; Ih(i+3) = Ih ii + m, in place: slot IC = row mod 3) and the lane-local
// delete chain.  The entry values W live in a ring of 4 (slot PH = row mod 4; W(i) overwrites W(i-4) in place), so a loop body of
// 12 rows keeps every ring slot a fixed register: with a 4-slot insert ring ptxas moved 12 registers per row between slots.
template <int J, int VEC, int PH, int IC>
__device__ __forceinline__ float fwd4_match(FwdState4<J> &S, const FwdConsts4<J> &K, const char *__restrict__ emis_lane, unsigned rowbytes,
                                            uint32_t cw, float2 (&t)[Pairs<J>::JP > 0 ? Pairs<J>::JP : 1], float &tt, float (&q)[J + 1])
{
  constexpr int JP = Pairs<J>::JP;
  constexpr bool TAIL = Pairs<J>::TAIL;
  constexpr int P0 = PH, P1 = (PH + 3) & 3, P2 = (PH + 2) & 3;
  float2 e2[JP > 0 ? JP : 1], e3[JP > 0 ? JP : 1], e4[JP > 0 ? JP : 1], m[JP > 0 ? JP : 1];
  float  e2t = 0.f, e3t = 0.f, e4t = 0.f, mt = 0.f;
  load_emission_pairs<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw & 511u) * rowbytes), e2, e2t);
  load_emission_pairs<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)((cw >> 9) & 511u) * rowbytes), e3, e3t);
  load_emission_pairs<J, VEC>(reinterpret_cast<const float *>(emis_lane + (size_t)(cw >> 18) * rowbytes), e4, e4t);
  float2 es = make_float2(0.f, 0.f);
#pragma unroll
  for (int p = 0; p < JP; ++p) {
    float2 v = fmul2(S.W[P2][p], e4[p]);
    v = ffma2(S.W[P1][p], e3[p], v);
    v = ffma2(S.W[P0][p], e2[p], v);
    m[p] = v;
    es = (p == 0) ? fmul2(v, K.qm[0]) : ffma2(v, K.qm[p], es);
    t[p] = ffma2(S.I[IC][p], K.hi[p], v);
    S.I[IC][p] = ffma2(S.I[IC][p], K.ii[p], v);
  }
  float esum = (JP > 0) ? es.x + es.y : 0.f;
  if constexpr (TAIL) {
    float v = S.Wt[P2] * e4t;
    v = fmaf(S.Wt[P1], e3t, v);
    v = fmaf(S.Wt[P0], e2t, v);
    mt = v;
    esum = fmaf(v, K.qmt, esum);
    tt = fmaf(S.It[IC], K.hit, v);
    S.It[IC] = fmaf(S.It[IC], K.iit, v);
  }
  // lane-local delete chain for zero inflow: A(j) = A(j-1) dd(j) + m(j); q(j) = A(j-1) is what node j sees of it
  q[0] = 0.f;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const float mj = (TAIL && j == J - 1) ? mt : ((j & 1) ? m[j >> 1].y : m[j >> 1].x);
    q[j + 1] = (j == 0) ? mj : fmaf(q[j], K.dd[j], mj);
  }
  return esum;
}

// second half of a row: the warp scan of the delete chain, the outflow, and -- given E(i) -- the specials and the next entry values
template <int J, int PH, int NS, bool HEAD>
__device__ __forceinline__ void fwd4_flow(int i, int lane, FwdState4<J> &S, const FwdConsts4<J> &K, const float2 (&t)[Pairs<J>::JP > 0 ? Pairs<J>::JP : 1], float tt,
                                          const float (&q)[J + 1], float xE, float ploop, float pmove, float tEL, float tEM, RowOut &R)
{
  constexpr int JP = Pairs<J>::JP;
  constexpr bool TAIL = Pairs<J>::TAIL;
  constexpr int P0 = PH, P2 = (PH + 2) & 3, P3 = (PH + 1) & 3;
  float A = q[J];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    float up = __shfl_up_sync(0xffffffffu, A, 1 << s);
    A = fmaf(K.bs[s], up, A);
  }
  const float din = __shfl_up_sync(0xffffffffu, A, 1);   // lane 0 reads its own A: node 1 has no delete state, its dd and dm are 0 (bathgpu.cu)

  // d(j) = din pd(j) + q(j): the delete value node j sees; outflow o = d dm + t
  float2 o[JP > 0 ? JP : 1];
  float  ot = 0.f;
  const float2 din2 = bcast2(din);
#pragma unroll
  for (int p = 0; p < JP; ++p) {
    float2 d;
    if (p == 0) d = make_float2(din, fmaf(din, K.pd[0].y, q[1]));        // pd(0) = 1, q(0) = 0
    else        d = ffma2(din2, K.pd[p], make_float2(q[2 * p], q[2 * p + 1]));
    o[p] = ffma2(d, K.dm[p], t[p]);
  }
  if constexpr (TAIL) {
    const float d = (J == 1) ? din : fmaf(din, K.pdt, q[J - 1]);
    ot = fmaf(d, K.dmt, tt);
  }

  float xN = S.xN[P3] * ploop;
  if constexpr (HEAD) xN = (i < 3) ? ((i >= 0) ? 1.0f : 0.0f) : xN;
  float xJ = fmaf(S.xJ[P3], ploop, xE * tEL);
  float xC = fmaf(S.xC[P3], ploop, xE * tEM);
  float xB = fmaf(xJ, pmove, xN * pmove);

  // W(i+2)[k+1] = B(i) + flow out of node k: node pairs shift by one node
  float olast = TAIL ? ot : o[JP > 0 ? JP - 1 : 0].y;
  float oprev = __shfl_up_sync(0xffffffffu, olast, 1);
  if (lane == 0) oprev = 0.f;
#pragma unroll
  for (int p = 0; p < JP; ++p) {                    // halves of two different pairs: two scalar adds written straight into the pair
    const float lo = (p == 0) ? oprev : o[p - 1].y;
    S.W[P2][p] = make_float2(xB + lo, xB + o[p].x);
  }
  if constexpr (TAIL) S.Wt[P2] = xB + (JP > 0 ? o[JP > 0 ? JP - 1 : 0].y : oprev);
  S.xN[P0] = xN; S.xJ[P0] = xJ; S.xC[P0] = xC;
  R.xE = xE; R.xN = xN; R.xJ = xJ; R.xC = xC; R.xB = xB; R.scale = 1.0f;
}

template <int J>
__device__ __forceinline__ void scale_state4(FwdState4<J> &S, float sf)
{
  constexpr int JP = Pairs<J>::JP;
  const float2 sf2 = bcast2(sf);
#pragma unroll
  for (int r = 0; r < 4; ++r) {
#pragma unroll
    for (int p = 0; p < JP; ++p) { S.W[r][p] = fmul2(S.W[r][p], sf2); if (r < 3) S.I[r][p] = fmul2(S.I[r][p], sf2); }
    if constexpr (Pairs<J>::TAIL) { S.Wt[r] *= sf; if (r < 3) S.It[r] *= sf; }
    S.xN[r] *= sf; S.xJ[r] *= sf; S.xC[r] *= sf;
  }
}

// E(i) and E(i+1) from the two rows' per-lane partial sums, reduced together
__device__ __forceinline__ void warp_allsum_pair(int lane, float a, float b, float &sa, float &sb)
{
  const bool  up   = (lane & 16) != 0;
  const float send = up ? a : b;
  float       keep = up ? b : a;
  keep += __shfl_xor_sync(0xffffffffu, send, 16);         // lower half: partials of a; upper half: partials of b
#pragma unroll
  for (int d = 8; d >= 1; d >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, d);
  sa = __shfl_sync(0xffffffffu, keep, 0);
  sb = __shfl_sync(0xffffffffu, keep, 16);
}

// XMX (X rows handed out): the rescale test is the reference's, row by row (xE > 1e4: fwdback_fs.c:472-496), so that the SCALE
// column matches.  Scores only: the test moves to the end of the 12-row body (xemax = largest E seen in it) -- the score does not
// depend on where the scale factors are taken out, 12 rows cannot grow the state by more than ~1e7, and the body becomes one
// basic block: with a rare branch after every pair ptxas re-established its register assignment with ~12 MOVs per row.
template <int J, int VEC, int PH, int IC, bool XMX, int NS, bool HEAD>
__device__ __forceinline__ void fwd4_row_pair(int i, int lane, FwdState4<J> &S, const FwdConsts4<J> &K,
                                              const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t cwA, uint32_t cwB,
                                              float ploop, float pmove, float tEL, float tEM,
                                              float &totscale, float &xemax, float *__restrict__ xrow)
{
  constexpr int JP = Pairs<J>::JP;
  float2 tA[JP > 0 ? JP : 1], tB[JP > 0 ? JP : 1];
  float  tAt = 0.f, tBt = 0.f, qA[J + 1], qB[J + 1];
  // row i+1 reads rows <= i-1 only, so both rows' match values come first
  const float esA = fwd4_match<J, VEC, PH, IC>(S, K, emis_lane, rowbytes, cwA, tA, tAt, qA);
  const float esB = fwd4_match<J, VEC, PH + 1, (IC + 1) % 3>(S, K, emis_lane, rowbytes, cwB, tB, tBt, qB);
  float xEA, xEB;
  warp_allsum_pair(lane, esA, esB, xEA, xEB);
  RowOut A, B;
  fwd4_flow<J, PH, NS, HEAD>(i, lane, S, K, tA, tAt, qA, xEA, ploop, pmove, tEL, tEM, A);
  fwd4_flow<J, PH + 1, NS, HEAD>(i + 1, lane, S, K, tB, tBt, qB, xEB, ploop, pmove, tEL, tEM, B);
  if constexpr (!XMX) { xemax = fmaxf(xemax, fmaxf(A.xE, B.xE)); return; }
  if (__builtin_expect(A.xE > 1.0e4f || B.xE > 1.0e4f, 0)) {          // rare, warp-uniform
    if (A.xE > 1.0e4f) {
      const float sf = __fdividef(1.0f, A.xE);      // no subroutine call inside the row loop (see above)
      scale_state4<J>(S, sf);                    // includes what row i+1 has just written
      A.scale = A.xE; A.xN *= sf; A.xJ *= sf; A.xC *= sf; A.xB *= sf;
      B.xE *= sf; B.xN *= sf; B.xJ *= sf; B.xC *= sf; B.xB *= sf;
      totscale += __logf(A.xE);
      A.xE = 1.0f;
    }
    if (B.xE > 1.0e4f) {
      const float sf = __fdividef(1.0f, B.xE);
      scale_state4<J>(S, sf);
      B.scale = B.xE; B.xN *= sf; B.xJ *= sf; B.xC *= sf; B.xB *= sf;
      totscale += __logf(B.xE);
      B.xE = 1.0f;
    }
  }
  store_xrow<XMX>(i, lane, A, xrow);
  store_xrow<XMX>(i + 1, lane, B, xrow);
}

#ifndef BATHGPU_V4_WARPS
// resident warps per SM the kernel is compiled for (register budget 65536 / (32 n))
#define BATHGPU_V4_WARPS(J) ((J) <= 2 ? 20 : (J) == 3 ? 18 : (J) == 4 ? 16 : (J) == 5 ? 14 : (J) == 6 ? 12 : (J) == 7 ? 10 : (J) == 8 ? 9 : 8)
#endif

// SET: as in fs3_forward_parser_kernel_v3
template <int J, bool XMX, int NS = 5, bool SET = false>
__global__ void __launch_bounds__(32, BATHGPU_V4_WARPS(J)) fs3_forward_parser_kernel_v4(FsParserArgs a)
{
  constexpr int VEC = VecOf<J>::V;
  constexpr int JP = Pairs<J>::JP;
  const int lane = threadIdx.x & 31;

  FwdConsts4<J> K;
  const char    *emis_lane = nullptr;
  float          tEM = a.tEM, tEL = a.tEL;
  int            cur = -1;
  if constexpr (!SET) {
    load_fwd_consts4<J>(a.cellc, lane, K);
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
        load_fwd_consts4<J>(sp.cellc, lane, K);
        emis_lane = reinterpret_cast<const char *>(sp.emis + lane * VEC);
        tEM = sp.tEM; tEL = sp.tEL;
      }
    }

    const WindowDesc wd = a.wins[w];
    const int   L     = wd.L;
    const float pmove = wd.pmove, ploop = wd.ploop;
    float *xrow = nullptr;
    if constexpr (XMX) xrow = a.xmx + (size_t)a.xoff[w] * 6;

    FwdState4<J> S;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int p = 0; p < (JP > 0 ? JP : 1); ++p) { S.W[r][p] = make_float2(0.f, 0.f); if (r < 3) S.I[r][p] = make_float2(0.f, 0.f); }
      S.Wt[r] = 0.f; if (r < 3) S.It[r] = 0.f;
      S.xN[r] = 0.f; S.xJ[r] = 0.f; S.xC[r] = 0.f;
    }
    float totscale = 0.f, xemax = 0.f;

    // rows -pad .. L in bodies of 12 (all-zero pad rows in front, so that the last body ends exactly at row L); 24 rows per chunk:
    // lane l < 24 prepares the codon word of row i + l, rows pick theirs up with one shuffle; the first chunk runs the HEAD instantiation
    const int nb  = (L + 12) / 12;
    const int pad = 12 * nb - (L + 1);
    long long nib = (wd.start - 1) + (long long)(lane - pad - 3) - 1 + 8;
    // up to 11 pad rows in front: their nucleotides lie before the one guard word of the packed block and are never used
    uint32_t lo = (nib >= 0) ? __ldg(a.dna4 + (nib >> 3)) : 0u, hi = (nib >= -8) ? __ldg(a.dna4 + (nib >> 3) + 1) : 0u;
    int i = -pad;

#define BATHGPU_V4_PAIR(HEAD_, R_)                                                                                               \
        {                                                                                                                         \
          const uint32_t cA = __shfl_sync(0xffffffffu, cwl, bb * 12 + (R_));                                                      \
          const uint32_t cB = __shfl_sync(0xffffffffu, cwl, bb * 12 + (R_) + 1);                                                  \
          fwd4_row_pair<J, VEC, (R_) & 3, (R_) % 3, XMX, NS, HEAD_>(i, lane, S, K, emis_lane, rowbytes, cA, cB, ploop, pmove, tEL, tEM, totscale, xemax, xrow); \
          i += 2;                                                                                                                 \
        }
#define BATHGPU_V4_CHUNK(HEAD_)                                                                                                   \
    {                                                                                                                             \
      const uint32_t cwl = codon_word(lo, hi, (int)(nib & 7) * 4, i + lane, L);                                                   \
      nib += 24;                                                                                                                  \
      if (b0 + 2 < nb) { lo = __ldg(a.dna4 + (nib >> 3)); hi = __ldg(a.dna4 + (nib >> 3) + 1); }                                  \
      const int bn = min(2, nb - b0);                                                                                             \
      for (int bb = 0; bb < bn; ++bb) {                                                                                           \
        BATHGPU_V4_PAIR(HEAD_, 0) BATHGPU_V4_PAIR(HEAD_, 2) BATHGPU_V4_PAIR(HEAD_, 4)                                             \
        BATHGPU_V4_PAIR(HEAD_, 6) BATHGPU_V4_PAIR(HEAD_, 8) BATHGPU_V4_PAIR(HEAD_, 10)                                            \
        if constexpr (!XMX) {                                                                                                     \
          if (__builtin_expect(xemax > 1.0e4f, 0)) { scale_state4<J>(S, __fdividef(1.0f, xemax)); totscale += __logf(xemax); }    \
          xemax = 0.f;                                                                                                            \
        }                                                                                                                         \
      }                                                                                                                           \
    }
    int b0 = 0;
    BATHGPU_V4_CHUNK(true)
    for (b0 = 2; b0 < nb; b0 += 2) BATHGPU_V4_CHUNK(false)
#undef BATHGPU_V4_CHUNK
#undef BATHGPU_V4_PAIR

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
