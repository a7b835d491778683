// fs_domain.cuh -- the per-envelope stage of domain definition for sm_100a:
//   p7_Forward_Frameshift / p7_Backward_Frameshift (5 codon lengths, full matrices; reference
//   src/impl_sse/fwdback_fs.c:2054-2607, :2634-2980), p7_Decoding_Frameshift (decoding_fs.c:55-200),
//   p7_Null2_fs_ByExpectation (null2_fs.c:53-139), p7_OptimalAccuracy_Frameshift (optacc_fs.c:53-283) and
//   p7_OATrace_Frameshift (:300-593), as called by rescore_isolated_domain_frameshift (src/p7_domaindef.c:1022-1082).
//
// One warp per envelope, lane l owns J contiguous nodes, rows sequential -- the parsers' decomposition.
// Three sweeps over the envelope instead of the reference's six passes over stored matrices:
//   1. fs5_forward_kernel:  Forward, row state in registers; stores per cell {M_C0..M_C5 (times Z(k)), I}
//      and the X rows; the D cell is only ever read by the stochastic trace (stotrace_fs.c:72), so only the
//      fs5_forward_kernel<J, true> instantiation behind bathgpu_fs_forward_matrices keeps it;
//   2. fs5_backward_decode_kernel: Backward row state in registers; each Backward row is multiplied into the
//      stored Forward row at once and normalised, so the Backward matrix is never stored; the posterior
//      matrix overwrites the Forward one in place (as the reference does), and the null2 column sums
//      accumulate in registers during the same sweep;
//   3. fs5_optacc_kernel: max-plus fill from the posterior rows (a 5-row ring of "best way into node k"
//      values in registers), stores {M,I,D} per cell for the traceback;
//   4. fs5_oatrace_kernel: the reference's traceback state machine, one warp per envelope (lanes cooperate
//      on the E-state argmax, everything else is a short dependent chain of loads).
// Matrix rows are laid out [cell type][32*J] in the same lane-permuted order as the emission table, so
// every access in sweeps 1-3 is a coalesced 128/64/32-bit lane access.
//
// Posterior normalisation: every term of the per-row denominator carries the same factor 1/Z, so the
// posteriors do not depend on it (decoding_fs.c:152-174); the reference takes log Z from Backward's N cells
// after its sweep ends, this kernel takes it from the Forward score (they agree to 1e-4 nat, :3191), which
// is what lets the normalisation run inside the Backward sweep.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "fs_parser.cuh"
#include "fs_backward.cuh"

namespace bathgpu {

constexpr int kPPCells = 7;     // per node and row: I, M_C0, M_C1 .. M_C5
constexpr int kOACells = 3;     // per node and row: M, I, D
enum PPCell { PP_I = 0, PP_C0 = 1 };
enum OACell { OA_M = 0, OA_I = 1, OA_D = 2 };

enum Fwd5Const { F5_MM = 0, F5_IM, F5_DM, F5_MD, F5_DD, F5_MI, F5_II, F5_COUNT };      // + 5 scan multipliers (up)
// Backward uses BckCellConst / BckLaneConst of fs_backward.cuh

struct EnvelopeDesc {    // device copy of bathgpu_envelope
  long long start;
  int       L;
  float     pmove;
  float     ploop;
};

struct DomainArgs {
  const float    *emis;        // 5-codon table R[c][k] tBM(k-1) Z(k), permuted, [1367+29][mpad]
  const float    *amino;       // amino-acid odds rows, NOT folded: [20][mpad] permuted (null2)
  const float    *cellf;       // forward lane constants  [F5_COUNT][J][32] + [5][32]
  const float    *cellb;       // backward lane constants [BC_COUNT][J][32] + [5][32]
  const float    *cellfmw;     // the same two for the multi-warp sweeps (fs_domain_mw.cuh; J >= 16), or null
  const float    *cellbmw;
  const float    *oapass;      // [5][32]: scan step s may carry D through the lanes it spans (all DD allowed)
  const uint32_t *oaflags;     // per node: bit t set iff transition t has positive odds, t = BM,MM,IM,DM (source k-1), MD,DD (source k-1), MI,II (k)
  const uint32_t *dna4;
  const EnvelopeDesc *envs;
  int             nenv;
  int             M, mpad;
  float           tEM, tEL;    // E->MOVE, E->LOOP odds of the 5-codon profile as configured by the caller
  const long long *xoff;       // X-row offset of envelope e (rows), xoff[e+1]-xoff[e] = L+1
  float          *pp;          // [rows][7][mpad]   Forward cells, then posteriors
  float          *dcell;       // [rows][mpad]      Forward D cells (fs5_forward_kernel<J, true> only: the stochastic trace reads them)
  float          *oa;          // [rows][3][mpad]
  float          *fx;          // [rows][6] Forward X rows
  float          *ppx;         // [rows][6] posterior X rows (N,J,C used)
  float          *oax;         // [rows][6] OA X rows {E,N,J,B,C,-}
  float          *lsf;         // [rows] cumulative log Forward scales
  float          *fwdsc, *bcksc, *oasc;     // [nenv]
  float          *null2;       // [nenv][29]
  int            *status;      // [nenv]
  int            *counter;
  const FsSetProfile *set;     // fs5_forward_kernel<J, true, true>: envelope e is scored with profile set[wprof[e]] (emis, cellf, cellfmw, tEM, tEL unused)
  const int      *wprof;
};

template <int J, int VEC>
__device__ __forceinline__ void load_row(const float *__restrict__ row_lane, float (&v)[J])
{
#pragma unroll
  for (int g = 0; g < J / VEC; ++g) {
    if constexpr (VEC == 4) {
      float4 t = *(reinterpret_cast<const float4 *>(row_lane) + g * kWarp);
      v[4 * g + 0] = t.x; v[4 * g + 1] = t.y; v[4 * g + 2] = t.z; v[4 * g + 3] = t.w;
    } else if constexpr (VEC == 2) {
      float2 t = *(reinterpret_cast<const float2 *>(row_lane) + g * kWarp);
      v[2 * g + 0] = t.x; v[2 * g + 1] = t.y;
    } else {
      v[g] = row_lane[g * kWarp];
    }
  }
}

template <int J, int VEC>
__device__ __forceinline__ void store_row(float *__restrict__ row_lane, const float (&v)[J])
{
#pragma unroll
  for (int g = 0; g < J / VEC; ++g) {
    if constexpr (VEC == 4)      *(reinterpret_cast<float4 *>(row_lane) + g * kWarp) = make_float4(v[4 * g], v[4 * g + 1], v[4 * g + 2], v[4 * g + 3]);
    else if constexpr (VEC == 2) *(reinterpret_cast<float2 *>(row_lane) + g * kWarp) = make_float2(v[2 * g], v[2 * g + 1]);
    else                         row_lane[g * kWarp] = v[g];
  }
}

// 5-codon row indices (src/hmmer.h:306-310) with the clamps to the degenerate rows (fwdback_fs.c:2419-2429)
__device__ __forceinline__ int nuc5_of(uint32_t code3) { return code3 < 4u ? (int)code3 : 1367; }
__device__ __forceinline__ void codon_rows5(int t, int u, int v, int w, int x, int (&c)[5])
{
  c[0] = min(x * 341, 1366);
  c[1] = min(x * 341 + w * 85 + 1, 1365);
  c[2] = min(x * 341 + w * 85 + v * 21 + 2, 1364);
  c[3] = min(x * 341 + w * 85 + v * 21 + u * 5 + 3, 1365);
  c[4] = min(x * 341 + w * 85 + v * 21 + u * 5 + t + 4, 1366);
}

// 3-bit codes (0..3, 7 = degenerate or outside 1..L) of the five nucleotides n[p0 .. p0+4] of an envelope
__device__ __forceinline__ uint32_t nuc_codes5(const uint32_t *__restrict__ dna4, long long env_start, int p0, int L)
{
  // nibble index of n[p0] in the packed block: (env_start - 1) + (p0 - 1) + 8 guard nibbles
  long long nib = (env_start - 1) + (long long)(p0 - 1) + 8;
  if (nib < 0) nib = 0;          // never dereferenced meaningfully: all five positions are then outside the envelope
  uint32_t lo = __ldg(dna4 + (nib >> 3)), hi = __ldg(dna4 + (nib >> 3) + 1);
  uint32_t bits = __funnelshift_r(lo, hi, (int)(nib & 7) * 4);
  uint32_t out = 0;
#pragma unroll
  for (int b = 0; b < 5; ++b) {
    uint32_t n = (bits >> (4 * b)) & 15u;
    int p = p0 + b;
    uint32_t code = (n < 4u && p >= 1 && p <= L) ? n : 7u;
    out |= code << (3 * b);
  }
  return out;
}

// Pull the lines of one stored matrix row (ncell cells of mpad floats) towards L1 ahead of the sweep that will read it: these
// sweeps are one warp per envelope walking rows one after the other, so a row's loads are otherwise a full DRAM round trip on the
// critical path (the matrices of a batch of envelopes are far larger than L2).
__device__ __forceinline__ void prefetch_matrix_row(const float *row_base, int ncell, int mpad, int lane)
{
#ifndef BATHGPU_NO_ROW_PREFETCH
  const char *p = reinterpret_cast<const char *>(row_base);
  const int nbytes = ncell * mpad * 4;
  for (int off = lane * 128; off < nbytes; off += 32 * 128) asm volatile("prefetch.global.L1 [%0];" :: "l"(p + off));
#endif
}

template <int J>
struct Fwd5Consts { float mm[J], im[J], dm[J], md[J], dd[J], mi[J], ii[J]; float bs[5]; };

template <int J>
struct Fwd5State { float W[5][J]; float I[5][J]; float xN[5], xJ[5], xC[5]; };

struct Fwd5Ctx { int L; float ploop, pmove, tEL, tEM, totscale, lsf; };

// One Forward row.  PH = padded row mod 5 (compile time): ring slot of row i; row i-c sits in slot (PH+5-c)%5.
template <int J, int VEC, int PH, bool STORE_D>
__device__ __forceinline__ void fwd5_row(int i, int lane, Fwd5State<J> &S, const Fwd5Consts<J> &K,
                                         const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t codes,
                                         Fwd5Ctx &R, float *__restrict__ pprow_lane, int mpad,
                                         float *__restrict__ fxrow, float *__restrict__ lsfrow, float *__restrict__ drow_lane)
{
  constexpr int P0 = PH, P1 = (PH + 4) % 5, P2 = (PH + 3) % 5, P3 = (PH + 2) % 5, P4 = (PH + 1) % 5;   // rows i, i-1, .., i-4
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
  for (int j = 0; j < J; ++j) {            // (:2437-2441) ((c1+c2)+(c3+c4))+c5
    m0[j] = ((mc[0][j] + mc[1][j]) + (mc[2][j] + mc[3][j])) + mc[4][j];
    es += m0[j];
  }
  float xE = warp_allsum(es);

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

  // specials (:2476-2490): rows 0..2 hold N at 1
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
    S.I[P2][j] = fmaf(icur[j], K.ii[j], m0[j] * K.mi[j]);      // I(i+3): slot (i+3)%5 == (i-2)%5
  }
  float oprev = __shfl_up_sync(0xffffffffu, o[J - 1], 1);
  if (lane == 0) oprev = 0.f;
  // W(i+1)[k+1] = B(i) + flow out of node k; slot (i+1)%5 == (i-4)%5 was read above
  S.W[P4][0] = xB + oprev;
#pragma unroll
  for (int j = 1; j < J; ++j) S.W[P4][j] = xB + o[j - 1];

  float scale = 1.0f;
  if (xE > 1.0e4f) {               // (:2492-2513)
    float sf = 1.0f / xE;
    scale = xE;
    xN *= sf; xJ *= sf; xC *= sf; xB *= sf;
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

  if (i >= 0) {
    R.lsf = R.lsf + logf(scale);    // log_sfwd[i] (decoding_fs.c:83-85), float running sum
    float *row = pprow_lane + (size_t)i * kPPCells * mpad;
    store_row<J, VEC>(row + PP_I * mpad, icur);
    store_row<J, VEC>(row + PP_C0 * mpad, m0);
#pragma unroll
    for (int cc = 0; cc < 5; ++cc) store_row<J, VEC>(row + (PP_C0 + 1 + cc) * mpad, mc[cc]);
    if constexpr (STORE_D) store_row<J, VEC>(drow_lane + (size_t)i * mpad, dv);
    if (lane == 0) {
      float2 *x2 = reinterpret_cast<float2 *>(fxrow + (size_t)i * 6);
      x2[0] = make_float2(xE, xN);
      x2[1] = make_float2(xJ, xB);
      x2[2] = make_float2(xC, scale);
      lsfrow[i] = R.lsf;
    }
  }
}

template <int J>
__device__ __forceinline__ void load_fwd5_consts(const float *__restrict__ cc, int lane, Fwd5Consts<J> &K)
{
#pragma unroll
  for (int j = 0; j < J; ++j) {
    K.mm[j] = __ldg(cc + (F5_MM * J + j) * kWarp + lane);
    K.im[j] = __ldg(cc + (F5_IM * J + j) * kWarp + lane);
    K.dm[j] = __ldg(cc + (F5_DM * J + j) * kWarp + lane);
    K.md[j] = __ldg(cc + (F5_MD * J + j) * kWarp + lane);
    K.dd[j] = __ldg(cc + (F5_DD * J + j) * kWarp + lane);
    K.mi[j] = __ldg(cc + (F5_MI * J + j) * kWarp + lane);
    K.ii[j] = __ldg(cc + (F5_II * J + j) * kWarp + lane);
  }
#pragma unroll
  for (int s = 0; s < 5; ++s) K.bs[s] = __ldg(cc + F5_COUNT * J * kWarp + s * kWarp + lane);
}

// SET: the envelopes of a profile set (DomainArgs::set); constants and table re-read whenever a warp's next envelope has another
// profile.  Everything else is the kernel bathgpu_fs_forward_matrices runs, stores included: a copy that skips them is compiled
// into other floating-point contractions and misses the scores-only call's results by an ulp.
template <int J, bool STORE_D = false, bool SET = false>
__global__ void __launch_bounds__(32) fs5_forward_kernel(DomainArgs a)
{
  constexpr int VEC = VecOf<J>::V;
  const int lane = threadIdx.x & 31;
  Fwd5Consts<J> K;
  const char    *emis_lane = nullptr;
  float          tEM = a.tEM, tEL = a.tEL;
  int            cur = -1;
  if constexpr (!SET) {
    load_fwd5_consts<J>(a.cellf, lane, K);
    emis_lane = reinterpret_cast<const char *>(a.emis + lane * VEC);
  }
  const unsigned rowbytes  = (unsigned)a.mpad * 4u;

  for (;;) {
    int e = 0;
    if (lane == 0) e = atomicAdd(a.counter, 1);
    e = __shfl_sync(0xffffffffu, e, 0);
    if (e >= a.nenv) break;
    if constexpr (SET) {
      const int p = a.wprof[e];
      if (p != cur) {
        cur = p;
        const FsSetProfile sp = a.set[p];
        load_fwd5_consts<J>(sp.cellc, lane, K);
        emis_lane = reinterpret_cast<const char *>(sp.emis + lane * VEC);
        tEM = sp.tEM; tEL = sp.tEL;
      }
    }
    const EnvelopeDesc ed = a.envs[e];
    const int L = ed.L;
    Fwd5Ctx R;
    R.L = L; R.ploop = ed.ploop; R.pmove = ed.pmove; R.tEL = tEL; R.tEM = tEM; R.totscale = 0.f; R.lsf = 0.f;
    const long long xo = a.xoff[e];
    float *pprow_lane = a.pp + (size_t)xo * kPPCells * a.mpad + lane * VEC;
    float *fxrow = a.fx + (size_t)xo * 6;
    float *lsfrow = a.lsf + xo;
    float *drow_lane = STORE_D ? a.dcell + (size_t)xo * a.mpad + lane * VEC : nullptr;

    Fwd5State<J> S;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
#pragma unroll
      for (int j = 0; j < J; ++j) { S.W[r][j] = 0.f; S.I[r][j] = 0.f; }
      S.xN[r] = 0.f; S.xJ[r] = 0.f; S.xC[r] = 0.f;
    }

    const int n5  = (L + 5) / 5;                   // ceil((L+1)/5)
    const int pad = 5 * n5 - (L + 1);
    int i = -pad;
    for (int g0 = 0; g0 < n5; g0 += 6) {           // 30 rows per chunk: lane l prepares row i + l
      const uint32_t codes_l = (lane < 30) ? nuc_codes5(a.dna4, ed.start, i + lane - 4, L) : 0u;
      const int gn = min(6, n5 - g0);
      for (int g = 0; g < gn; ++g) {
#define BATHGPU_F5ROW(PH_)                                                                           \
        {                                                                                            \
          uint32_t codes = __shfl_sync(0xffffffffu, codes_l, g * 5 + PH_);                           \
          fwd5_row<J, VEC, PH_, STORE_D>(i, lane, S, K, emis_lane, rowbytes, codes, R, pprow_lane, a.mpad, fxrow, lsfrow, drow_lane); \
          ++i;                                                                                       \
        }
        BATHGPU_F5ROW(0) BATHGPU_F5ROW(1) BATHGPU_F5ROW(2) BATHGPU_F5ROW(3) BATHGPU_F5ROW(4)
#undef BATHGPU_F5ROW
      }
    }
    {   // row L sits in slot 4 (:2585-2601)
      float tot = S.xC[4] + S.xC[3] * R.ploop + S.xC[2] * R.ploop;
      int   st  = 0;
      float sc;
      if (isnan(tot) || isinf(tot))  { st = 16; sc = tot; }
      else if (L > 1 && tot == 0.0f) { st = 16; sc = -INFINITY; }
      else sc = R.totscale + logf(tot * R.pmove);
      if (lane == 0) { a.fwdsc[e] = sc; a.status[e] = st; }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Backward + decoding + null2 sums, one sweep from row L down to row 0.
template <int J>
struct Bck5State { float Mt[5][J]; float I[5][J]; float xN[5], xJ[5], xC[5]; };

struct Bck5Ctx {
  int   L;
  float ploop, pmove, tEL, tEM;
  float totscale;        // sum of log scales (score)
  float lsb;             // log_sbck[i]: float running sum of log scales of rows >= i (decoding_fs.c:86-88)
  float liz;             // -log Z
  bool  own_scales;
  int   st;
  float accN, accJ, accC;
};

template <int J, int VEC, int PH>
__device__ __forceinline__ void bck5_row(int i, int lane, Bck5State<J> &S, const BckConsts<J> &K,
                                         const char *__restrict__ emis_lane, unsigned rowbytes, uint32_t codes,
                                         Bck5Ctx &R, float *__restrict__ pprow_lane, int mpad,
                                         const float *__restrict__ fxrow, const float *__restrict__ lsfrow,
                                         float *__restrict__ ppxrow, float (&accM)[J], float (&accI)[J])
{
  // ring slot of row r is r mod 5; PH = i mod 5
  constexpr int S0 = PH, S1 = (PH + 1) % 5, S2 = (PH + 2) % 5, S3 = (PH + 3) % 5, S4 = (PH + 4) % 5;   // rows i(=i+5), i+1, .., i+4
  const int L = R.L;
  if (i > L) return;
  if (i >= 1) prefetch_matrix_row(pprow_lane - lane * VEC + (size_t)(i - 1) * kPPCells * mpad, kPPCells, mpad, lane);   // the row this sweep reads next

  float xN, xJ, xC, xB, xE;
  const float fscale = fxrow[(size_t)i * 6 + 5];

  if (i == L) {                    // (:2689-2741)
    xC = R.pmove; xN = 0.f; xJ = 0.f; xB = 0.f;
    xE = xC * R.tEM;
#pragma unroll
    for (int j = 0; j < J; ++j) { S.Mt[S0][j] = xE; S.I[S0][j] = 0.f; }
    S.xC[S1] = R.pmove; S.xC[S2] = R.pmove;       // xC_buf[L+1] = xC_buf[L+2] = tCM (:2684-2685)
  } else {
    // v'(k) = tBM(k-1) sum_c R[c][k] M(i+c,k); codes hold n[i+1..i+5] and the quasi-codon of length m is
    // n[i+1..i+m], last nucleotide most significant in the row index              (:2768-2800)
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
    xB = warp_allsum(bsum);

    if (i == 0) {                  // termination (:2899-2925)
      xN = fmaf(S.xN[S3], R.ploop, xB * R.pmove);
      S.xN[S0] = xN;
      return;
    }

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

  // scale of this row (:2741-2747, :2855-2862): the Forward row's, or Backward's own once xB has passed 1e16
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
      if (i < L) { S.xN[r] *= sf; S.xJ[r] *= sf; S.xC[r] *= sf; }     // row L leaves the buffers alone (:2722-2735)
    }
    R.totscale += logf(scale);
  }
  S.xN[S0] = xN; S.xJ[S0] = xJ; S.xC[S0] = xC;
  R.lsb = R.lsb + logf(scale);

  // ---- decoding of row i (decoding_fs.c:106-196)
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
  const float raw_denom = warp_allsum(den);
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
  if (lane == 0) {
    float2 *x2 = reinterpret_cast<float2 *>(ppxrow + (size_t)i * 6);
    x2[0] = make_float2(0.f, pN);
    x2[1] = make_float2(pJ, 0.f);
    x2[2] = make_float2(pC, scale);
  }
}

template <int J>
__global__ void __launch_bounds__(32) fs5_backward_decode_kernel(DomainArgs a)
{
  constexpr int VEC = VecOf<J>::V;
  const int lane = threadIdx.x & 31;
  BckConsts<J> K;
  load_bck_consts<J>(a.cellb, lane, K);
  const char    *emis_lane = reinterpret_cast<const char *>(a.emis + lane * VEC);
  const unsigned rowbytes  = (unsigned)a.mpad * 4u;

  for (;;) {
    int e = 0;
    if (lane == 0) e = atomicAdd(a.counter, 1);
    e = __shfl_sync(0xffffffffu, e, 0);
    if (e >= a.nenv) break;
    if (a.status[e] != 0) { if (lane == 0) a.bcksc[e] = -INFINITY; continue; }
    const EnvelopeDesc ed = a.envs[e];
    const int L = ed.L;
    const long long xo = a.xoff[e];
    float *pprow_lane = a.pp + (size_t)xo * kPPCells * a.mpad + lane * VEC;
    const float *fxrow = a.fx + (size_t)xo * 6;
    const float *lsfrow = a.lsf + xo;
    float *ppxrow = a.ppx + (size_t)xo * 6;

    Bck5Ctx R;
    R.L = L; R.ploop = ed.ploop; R.pmove = ed.pmove; R.tEL = a.tEL; R.tEM = a.tEM;
    R.totscale = 0.f; R.lsb = 0.f; R.liz = -a.fwdsc[e]; R.own_scales = false; R.st = 0;
    R.accN = 0.f; R.accJ = 0.f; R.accC = 0.f;
    // log Z from the Forward score: score = log(C_tot tCM) + totscale, and Z (decoding_fs.c:90-95) is the same
    // path sum seen from the N side, without the final C->T move both of them include.

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
    int i = 5 * n5 - 1;                            // >= L, i % 5 == 4
    for (int g0 = 0; g0 < n5; g0 += 6) {
      const uint32_t codes_l = (lane < 30 && i - lane >= 0) ? nuc_codes5(a.dna4, ed.start, i - lane + 1, L) : 0u;
      const int gn = min(6, n5 - g0);
      for (int g = 0; g < gn; ++g) {
#define BATHGPU_B5ROW(PH_)                                                                           \
        {                                                                                            \
          uint32_t codes = __shfl_sync(0xffffffffu, codes_l, g * 5 + (4 - PH_));                     \
          bck5_row<J, VEC, PH_>(i, lane, S, K, emis_lane, rowbytes, codes, R, pprow_lane, a.mpad, fxrow, lsfrow, ppxrow, accM, accI); \
          --i;                                                                                       \
        }
        BATHGPU_B5ROW(4) BATHGPU_B5ROW(3) BATHGPU_B5ROW(2) BATHGPU_B5ROW(1) BATHGPU_B5ROW(0)
#undef BATHGPU_B5ROW
      }
    }

    // Backward score (:2940-2975)
    {
      float tot = S.xN[0] + S.xN[1] + S.xN[2];
      float sc;
      if (isnan(tot) || isinf(tot)) { R.st = 16; sc = tot; }
      else if (tot == 0.0f)         { R.st = 16; sc = -INFINITY; }
      else sc = R.totscale + logf(tot);
      if (lane == 0) { a.bcksc[e] = sc; if (R.st) a.status[e] = R.st; }
    }
    // posterior row 0 is all zero (decoding_fs.c:99-104)
    {
      float z[J];
#pragma unroll
      for (int j = 0; j < J; ++j) z[j] = 0.f;
#pragma unroll
      for (int cc = 0; cc < kPPCells; ++cc) store_row<J, VEC>(pprow_lane + (size_t)cc * a.mpad, z);
      if (lane == 0) { for (int s = 0; s < 6; ++s) ppxrow[s] = 0.f; }
    }

    // null2 by expectation (null2_fs.c:78-133)
    {
      const float norm = 1.0f / (float)L;
      const float xfactor = R.accN * norm + R.accC * norm + R.accJ * norm;
      float isum = 0.f;
#pragma unroll
      for (int j = 0; j < J; ++j) { accM[j] *= norm; accI[j] *= norm; isum += accI[j]; }
      isum = warp_allsum(isum);
      float n2 = 0.f;              // lane x < 20 keeps null2[x]
      for (int x = 0; x < 20; ++x) {
        float r[J];
        load_emission_row<J, VEC>(a.amino + (size_t)x * a.mpad + lane * VEC, r);
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < J; ++j) s = fmaf(accM[j], r[j], s);
        s = warp_allsum(s) + isum + xfactor;
        if (lane == x) n2 = s;
      }
      // degenerate residues: average of the members' odds (esl_abc_FAvgScVec); gap, '*', '~' = 1
      float out = 1.0f;
      const unsigned full = 0xffffffffu;
      float vals[20];
#pragma unroll
      for (int x = 0; x < 20; ++x) vals[x] = __shfl_sync(full, n2, x);
      if (lane < 20) out = n2;
      else if (lane == 21) out = (vals[2] + vals[11]) / 2.0f;      // B = D,N
      else if (lane == 22) out = (vals[7] + vals[9]) / 2.0f;       // J = I,L
      else if (lane == 23) out = (vals[3] + vals[13]) / 2.0f;      // Z = E,Q
      else if (lane == 24) out = vals[8];                          // O = K
      else if (lane == 25) out = vals[1];                          // U = C
      else if (lane == 26) { float s = 0.f;
#pragma unroll
        for (int x = 0; x < 20; ++x) s += vals[x];
        out = s / 20.0f; }                                          // X = any
      if (lane < 29) a.null2[(size_t)e * 29 + lane] = out;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Optimal-accuracy fill (optacc_fs.c:53-283).  Max-plus, so given the posteriors the result is exact.
// P(r)[k] = best way into match k from row r = max(mask(BM) B(r), mask(MM) M(r,k-1), mask(IM) I(r,k-1), mask(DM) D(r,k-1))
// (a forbidden transition contributes 0.0, not -inf: the reference masks with _mm_and_ps, :140-181).
enum OAFlag { OF_BM = 1, OF_MM = 2, OF_IM = 4, OF_DM = 8, OF_MD = 16, OF_DD = 32, OF_MI = 64, OF_II = 128 };

template <int J>
struct OAState { float P[5][J]; float Mr[5][J]; float Ir[5][J]; float xN[5], xJ[5], xC[5]; };

__device__ __forceinline__ float oa_mask(uint32_t flags, uint32_t bit, float v) { return (flags & bit) ? v : 0.0f; }
__device__ __forceinline__ float oa_max(float a, float b) { return (a > b) ? a : b; }      // _mm_max_ps(a,b) = a > b ? a : b

template <int J, int VEC, int PH>
__device__ __forceinline__ void oa_row(int i, int lane, OAState<J> &S, const uint32_t (&fl)[J], const float (&dpass)[5],
                                       const float *__restrict__ pprow_lane, float *__restrict__ oarow_lane, int mpad,
                                       const float *__restrict__ ppxrow, float *__restrict__ oaxrow, int M, int J0,
                                       bool loopN, bool loopJ, bool loopC, bool loopE, bool moveE, bool moveN, bool moveJ)
{
  // ring slot of row r: r mod 5; PH = i mod 5; row i-c in slot (PH+5-c)%5
  constexpr int P0 = PH, P1 = (PH + 4) % 5, P2 = (PH + 3) % 5, P3 = (PH + 2) % 5, P4 = (PH + 1) % 5;
  if (i < 1) return;
  const float *row = pprow_lane + (size_t)i * kPPCells * mpad;
  prefetch_matrix_row(row - lane * VEC + (size_t)kPPCells * mpad, kPPCells, mpad, lane);       // row i+1 (one row past the end is still inside the buffer or its guard)
  float pc[J], mnew[J], inew[J];
  // M(i,k) = max_c ( P(i-c)[k] + pp_Cc(i,k) ); rows before 0 count as row 0 (:101-108) -- the ring holds row 0 there
  load_row<J, VEC>(row + (PP_C0 + 1) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) mnew[j] = S.P[P1][j] + pc[j];
  float t2[J];
  load_row<J, VEC>(row + (PP_C0 + 2) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) mnew[j] = oa_max(mnew[j], S.P[P2][j] + pc[j]);      // max(c1, c2)
  load_row<J, VEC>(row + (PP_C0 + 3) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) t2[j] = S.P[P3][j] + pc[j];
  load_row<J, VEC>(row + (PP_C0 + 4) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) t2[j] = oa_max(t2[j], S.P[P4][j] + pc[j]);          // max(c3, c4)
  load_row<J, VEC>(row + (PP_C0 + 5) * mpad, pc);
#pragma unroll
  for (int j = 0; j < J; ++j) {
    t2[j] = oa_max(t2[j], S.P[P0][j] + pc[j]);                                    // max(max(c3,c4), c5); slot P0 still holds row i-5
    mnew[j] = oa_max(mnew[j], t2[j]);
  }
  // I(i,k) = max(mask(MI) M(i-3,k), mask(II) I(i-3,k)) + pp_I(i,k); I(i,M) = -inf (:196-212)
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

  // D(i,k) = max(mask(MD(k-1)) M(i,k-1), mask(DD(k-1)) D(i,k-1)), D(i,1) = -inf (:214-247): lane-serial + warp scan.
  // The pass-through of a whole lane is a profile constant: dpass[s] is 1 when every DD between the two
  // partners of scan step s is allowed (then the carried value is taken as is), else the carry restarts at 0.0 or is blocked.
  float dnew[J];
  {
    // local pass with carry-in "nothing": use -inf for the incoming D and M of the previous lane
    float mprev = __shfl_up_sync(0xffffffffu, mnew[J - 1], 1);
    if (lane == 0) mprev = -INFINITY;
    // first the chain value at the END of this lane assuming carry-in cD = -inf
    float cD = -INFINITY, cM = mprev;
    float endv;
    {
      float dd_ = cD, mm_ = cM;
#pragma unroll
      for (int j = 0; j < J; ++j) {
        float dv = oa_max(oa_mask(fl[j], OF_DD, dd_), oa_mask(fl[j], OF_MD, mm_));
        const int k = J0 + j + 1;
        if (k == 1) dv = -INFINITY;
        dd_ = dv; mm_ = mnew[j];
      }
      endv = dd_;      // D at the last node of the lane, carry-in -inf
    }
    // warp scan of lane-end values: true_end(l) = max(endv(l), pass(l) ? true_end(l-1) : (blocked))
    // With masks that are all-true inside a lane, D passes through unchanged: max-scan with pass flags.
    float A = endv;
#pragma unroll
    for (int s = 0; s < 5; ++s) {
      float up = __shfl_up_sync(0xffffffffu, A, 1 << s);
      if (lane >= (1 << s) && dpass[s] != 0.f) A = oa_max(A, up);
    }
    float carry = __shfl_up_sync(0xffffffffu, A, 1);
    if (lane == 0) carry = -INFINITY;
    float dd_ = carry, mm_ = mprev;
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

  // E(i) = max_k max(M, D)
  float e = -INFINITY;
#pragma unroll
  for (int j = 0; j < J; ++j) e = oa_max(e, oa_max(mnew[j], dnew[j]));
#pragma unroll
  for (int dlt = 16; dlt >= 1; dlt >>= 1) e = oa_max(e, __shfl_xor_sync(0xffffffffu, e, dlt));
  const float xE = e;

  // specials (:251-279)
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

  // P(i)[k] for the rows to come: predecessors at node k-1 of THIS row
  {
    float mp = __shfl_up_sync(0xffffffffu, mnew[J - 1], 1);
    float ip = __shfl_up_sync(0xffffffffu, inew[J - 1], 1);
    float dp = __shfl_up_sync(0xffffffffu, dnew[J - 1], 1);
    if (lane == 0) { mp = -INFINITY; ip = -INFINITY; dp = -INFINITY; }     // column 0 is -inf (:110-112)
#pragma unroll
    for (int j = 0; j < J; ++j) {
      float s = oa_mask(fl[j], OF_BM, xB);
      s = oa_max(s, oa_mask(fl[j], OF_MM, mp));
      s = oa_max(s, oa_mask(fl[j], OF_IM, ip));
      s = oa_max(s, oa_mask(fl[j], OF_DM, dp));
      S.P[P0][j] = s;
      mp = mnew[j]; ip = inew[j]; dp = dnew[j];
    }
  }
#pragma unroll
  for (int j = 0; j < J; ++j) { S.Mr[P0][j] = mnew[j]; S.Ir[P0][j] = inew[j]; }

  float *orow = oarow_lane + (size_t)i * kOACells * mpad;
  store_row<J, VEC>(orow + OA_M * mpad, mnew);
  store_row<J, VEC>(orow + OA_I * mpad, inew);
  store_row<J, VEC>(orow + OA_D * mpad, dnew);
  if (lane == 0) {
    float2 *x2 = reinterpret_cast<float2 *>(oaxrow + (size_t)i * 6);
    x2[0] = make_float2(xE, xN);
    x2[1] = make_float2(xJ, xB);
    x2[2] = make_float2(xC, 0.f);
  }
}

template <int J>
__global__ void __launch_bounds__(32) fs5_optacc_kernel(DomainArgs a)
{
  constexpr int VEC = VecOf<J>::V;
  const int lane = threadIdx.x & 31;
  const int J0 = lane * J;
  uint32_t fl[J];
#pragma unroll
  for (int j = 0; j < J; ++j) fl[j] = a.oaflags[J0 + j];
  float dpass[5];
#pragma unroll
  for (int s = 0; s < 5; ++s) dpass[s] = a.oapass[s * 32 + lane];

  for (;;) {
    int e = 0;
    if (lane == 0) e = atomicAdd(a.counter, 1);
    e = __shfl_sync(0xffffffffu, e, 0);
    if (e >= a.nenv) break;
    if (a.status[e] != 0) { if (lane == 0) a.oasc[e] = -INFINITY; continue; }
    const EnvelopeDesc ed = a.envs[e];
    const int L = ed.L;
    const long long xo = a.xoff[e];
    const float *pprow_lane = a.pp + (size_t)xo * kPPCells * a.mpad + lane * VEC;
    float *oarow_lane = a.oa + (size_t)xo * kOACells * a.mpad + lane * VEC;
    const float *ppxrow = a.ppx + (size_t)xo * 6;
    float *oaxrow = a.oax + (size_t)xo * 6;
    // the length model of THIS envelope decides which special transitions exist (unihit: E->LOOP = 0, J unused)
    const bool loopN = ed.ploop != 0.f, loopJ = ed.ploop != 0.f, loopC = ed.ploop != 0.f;
    const bool moveN = ed.pmove != 0.f, moveJ = ed.pmove != 0.f;
    const bool loopE = a.tEL != 0.f, moveE = a.tEM != 0.f;

    OAState<J> S;
    // row 0 (:86-99): cells -inf, N = 0, B = 0, E = J = C = -inf.  P(0)[k] = max(mask(BM) 0, mask(..) -inf ..)
#pragma unroll
    for (int r = 0; r < 5; ++r) {
#pragma unroll
      for (int j = 0; j < J; ++j) {
        float s = oa_mask(fl[j], OF_BM, (r == 0) ? 0.0f : -INFINITY);      // rows before 0: xB counts as -inf (:101-108)
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
      if (lane == 0) { oaxrow[0] = -INFINITY; oaxrow[1] = 0.f; oaxrow[2] = -INFINITY; oaxrow[3] = 0.f; oaxrow[4] = -INFINITY; oaxrow[5] = 0.f; }
    }

    const int n5 = (L + 5) / 5;
    int i = 0;
    for (int g = 0; g < n5; ++g) {
#define BATHGPU_OAROW(PH_)                                                                                      \
      { if (i <= L) oa_row<J, VEC, PH_>(i, lane, S, fl, dpass, pprow_lane, oarow_lane, a.mpad, ppxrow, oaxrow, a.M, J0, \
                                        loopN, loopJ, loopC, loopE, moveE, moveN, moveJ);                      \
        ++i; }
      BATHGPU_OAROW(0) BATHGPU_OAROW(1) BATHGPU_OAROW(2) BATHGPU_OAROW(3) BATHGPU_OAROW(4)
#undef BATHGPU_OAROW
    }
    __syncwarp();
    if (lane == 0) {
      // ret_e = C(L) + C(L-1) + C(L-2) (:281)
      a.oasc[e] = oaxrow[(size_t)L * 6 + 4] + oaxrow[(size_t)(L - 1) * 6 + 4] + oaxrow[(size_t)(L - 2) * 6 + 4];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Traceback (optacc_fs.c:300-593).  One warp per envelope; every lane runs the same state machine on the
// same (broadcast) loads, and the lanes split the E-state argmax over nodes.
struct TraceStep { int32_t i; int16_t k; uint8_t st; uint8_t c; float pp; };
enum TraceState { TS_M = 1, TS_D = 2, TS_I = 3, TS_S = 4, TS_N = 5, TS_B = 6, TS_E = 7, TS_C = 8, TS_T = 9, TS_J = 10 };

struct TraceArgs {
  TraceStep       *steps;      // envelope e writes at steps + toff[e], in traceback order
  const long long *toff;
  int             *tlen;       // [nenv]
  const float     *tfv;        // un-permuted transition odds [8][M+1], BM,MM,IM,DM,MD,MI,II,DD (source-node indexed)
  int              J;
};

__device__ __forceinline__ int perm_of(int k, int J)      // position of node k inside a permuted row
{
  const int VEC = (J % 4 == 0) ? 4 : ((J % 2 == 0) ? 2 : 1);
  const int kk = k - 1, ln = kk / J, j = kk % J;
  return (j / VEC) * (32 * VEC) + ln * VEC + (j % VEC);
}

static __global__ void __launch_bounds__(128) fs5_oatrace_kernel(DomainArgs a, TraceArgs t)
{
  const int lane = threadIdx.x & 31;
  const int e    = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (e >= a.nenv) return;
  if (a.status[e] != 0) { if (lane == 0) t.tlen[e] = 0; return; }
  const EnvelopeDesc ed = a.envs[e];
  const int L = ed.L, M = a.M, mpad = a.mpad, J = t.J;
  const long long xo = a.xoff[e];
  const float *pp  = a.pp + (size_t)xo * kPPCells * mpad;
  const float *oa  = a.oa + (size_t)xo * kOACells * mpad;
  const float *ppx = a.ppx + (size_t)xo * 6;
  const float *oax = a.oax + (size_t)xo * 6;
  TraceStep *out = t.steps + t.toff[e];
  const int ld = M + 1;
  auto TF = [&](int tt, int k) -> float { return t.tfv[(size_t)tt * ld + k]; };
  auto OA = [&](int i, int k, int cell) -> float {
    if (k < 1) return -INFINITY;                   // column 0 (:110-112)
    return oa[((size_t)i * kOACells + cell) * mpad + perm_of(k, J)];
  };
  auto PP = [&](int i, int k, int cell) -> float { return pp[((size_t)i * kPPCells + cell) * mpad + perm_of(k, J)]; };
  const bool loopC = ed.ploop != 0.f, loopJ = ed.ploop != 0.f, moveN = ed.pmove != 0.f, moveJ = ed.pmove != 0.f;
  const bool loopE = a.tEL != 0.f, moveE = a.tEM != 0.f;

  int n = 0;
  int last_st = 0;
  auto emit = [&](int st, int k, int i, int c, float p) {      // p7_trace_fs_AppendWithPP: which fields each state keeps
    TraceStep s; s.st = (uint8_t)st; s.i = 0; s.k = 0; s.c = 0; s.pp = 0.f;
    if (st == TS_N || st == TS_C || st == TS_J) { if (last_st == st) { s.i = i; s.pp = p; } }
    else if (st == TS_D) s.k = (int16_t)k;
    else if (st == TS_M) { s.i = i; s.k = (int16_t)k; s.c = (uint8_t)c; s.pp = p; }
    else if (st == TS_I) { s.i = i; s.k = (int16_t)k; s.pp = p; }
    if (lane == 0) out[n] = s;
    last_st = st;
    ++n;
  };
  int i = L, k = 0, c = 0;
  emit(TS_T, k, i, c, 0.f);
  emit(TS_C, k, i, c, 0.f);
  int sprv = TS_C, scur = TS_C;
  const int max_steps = L + M + 8;
  bool bad = false;
  while (sprv != TS_S) {
    switch (sprv) {
    case TS_M: {                                   // select_m (:321-358): predecessors at row i, column k-1; order M > I > D > B
      float pm = (TF(1, k - 1) == 0.f) ? -INFINITY : OA(i, k - 1, OA_M);
      float pi = (TF(2, k - 1) == 0.f) ? -INFINITY : OA(i, k - 1, OA_I);
      float pd = (TF(3, k - 1) == 0.f) ? -INFINITY : OA(i, k - 1, OA_D);
      float pb = (TF(0, k - 1) == 0.f) ? -INFINITY : oax[(size_t)i * 6 + 3];
      scur = TS_M; float best = pm;
      if (pi > best) { best = pi; scur = TS_I; }
      if (pd > best) { best = pd; scur = TS_D; }
      if (pb > best) { best = pb; scur = TS_B; }
      k--; break; }
    case TS_D: {                                   // select_d (:360-376)
      float pm = (TF(4, k - 1) == 0.f) ? -INFINITY : OA(i, k - 1, OA_M);
      float pd = (TF(7, k - 1) == 0.f) ? -INFINITY : OA(i, k - 1, OA_D);
      scur = (pm >= pd) ? TS_M : TS_D;
      k--; break; }
    case TS_I: {                                   // select_i (:378-397)
      const int pi_ = (i >= 3) ? i - 3 : 0;
      float pm = (TF(5, k) == 0.f) ? -INFINITY : OA(pi_, k, OA_M);
      float pI = (TF(6, k) == 0.f) ? -INFINITY : OA(pi_, k, OA_I);
      scur = (pm >= pI) ? TS_M : TS_I;
      i -= 3; break; }
    case TS_N: scur = (i == 0) ? TS_S : TS_N; break;
    case TS_C: {                                   // select_c (:418-445)
      if (i < 4) { scur = TS_E; break; }
      float p0 = !loopC ? -INFINITY : oax[(size_t)(i - 3) * 6 + 4] + ppx[(size_t)i * 6 + 4];
      float p1 = (i < L     && loopC) ? oax[(size_t)(i - 2) * 6 + 4] + ppx[(size_t)(i + 1) * 6 + 4] : -INFINITY;
      float p2 = (i < L - 1 && loopC) ? oax[(size_t)(i - 1) * 6 + 4] + ppx[(size_t)(i + 2) * 6 + 4] : -INFINITY;
      float p3 = !moveE ? -INFINITY : oax[(size_t)i * 6 + 0];
      float best = p0; scur = TS_C;
      if (p1 > best) best = p1;
      if (p2 > best) best = p2;
      if (p3 > best) { best = p3; scur = TS_E; }
      break; }
    case TS_J: {                                   // select_j (:447-463)
      if (i <= 5) { scur = TS_E; break; }
      float p0 = !loopJ ? -INFINITY : oax[(size_t)i * 6 + 2] + ppx[(size_t)i * 6 + 2];
      float p1 = !loopE ? -INFINITY : oax[(size_t)i * 6 + 0];
      scur = (p1 > p0) ? TS_E : TS_J;
      break; }
    case TS_E: {                                   // select_e (:465-490): first maximum in the order M1,D1,M2,D2,...
      float best = -INFINITY; int bidx = 0x7fffffff;
      for (int kk = lane + 1; kk <= M; kk += 32) {
        float vm = OA(i, kk, OA_M), vd = OA(i, kk, OA_D);
        if (vm > best) { best = vm; bidx = 2 * kk; }
        if (vd > best) { best = vd; bidx = 2 * kk + 1; }
      }
#pragma unroll
      for (int dlt = 16; dlt >= 1; dlt >>= 1) {
        float ob = __shfl_xor_sync(0xffffffffu, best, dlt);
        int   oi = __shfl_xor_sync(0xffffffffu, bidx, dlt);
        if (ob > best || (ob == best && oi < bidx)) { best = ob; bidx = oi; }
      }
      if (bidx == 0x7fffffff || best == -INFINITY) { scur = TS_M; k = 1; }      // nothing beat -inf: the reference's initial values
      else { scur = (bidx & 1) ? TS_D : TS_M; k = bidx >> 1; }
      break; }
    case TS_B: {                                   // select_b (:492-502)
      float p0 = !moveN ? -INFINITY : oax[(size_t)i * 6 + 1];
      float p1 = !moveJ ? -INFINITY : oax[(size_t)i * 6 + 2];
      scur = (p0 > p1) ? TS_N : TS_J;
      break; }
    default: bad = true; break;
    }
    if (bad || i < 0 || k < 0 || n >= max_steps) { bad = true; break; }

    float postprob = 0.f;                          // get_postprob (:300-319)
    if (scur == TS_M)      postprob = PP(i, k, PP_C0);
    else if (scur == TS_I) postprob = PP(i, k, PP_I);
    else if (scur == sprv && scur == TS_N) postprob = ppx[(size_t)i * 6 + 1];
    else if (scur == sprv && scur == TS_C) postprob = ppx[(size_t)i * 6 + 4];
    else if (scur == sprv && scur == TS_J) postprob = ppx[(size_t)i * 6 + 2];
    c = 0;
    if (scur == TS_M) {                            // select_codon (:504-518): first maximum of the five per-length posteriors
      float bestc = PP(i, k, PP_C0 + 1); c = 1;
#pragma unroll
      for (int cc = 2; cc <= 5; ++cc) { float v = PP(i, k, PP_C0 + cc); if (v > bestc) { bestc = v; c = cc; } }
    }
    emit(scur, k, i, c, postprob);
    if ((scur == TS_N || scur == TS_C || scur == TS_J) && scur == sprv) i--;
    sprv = scur;
    i -= c;
  }
  __syncwarp();
  if (bad) { if (lane == 0) { t.tlen[e] = 0; a.status[e] = 11; } return; }
  if (lane == 0) t.tlen[e] = n;      // still in traceback order: the host pulls N/C/J residues back and reverses (p7_trace_fs_Reverse)
}

}  // namespace bathgpu
