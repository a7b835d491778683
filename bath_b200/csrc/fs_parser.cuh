// fs_parser.cuh -- frameshift Forward / Backward PARSER kernels (3 codon lengths) for sm_100a.
//
// What they compute is p7_ForwardParser_Frameshift_3Codons / p7_BackwardParser_Frameshift_3Codons
// (reference: src/impl_sse/fwdback_fs.c:97-533, :565-1013).  How they compute it is B200-first:
//
//  * one warp per DNA window; lane l owns J CONTIGUOUS model nodes k = l*J+1 .. l*J+J
//    (no striping -- striping exists to feed CPU SIMD lanes); all per-node state lives in registers;
//  * per-node state is the minimum the recurrence needs: the pre-emission entry values V(r)[k]
//    (the reference's IVX) for 4 rows and the insert values I(r)[k] for 3 rows -- 7 floats per node,
//    instead of the reference's 4x3 MDI ring + 3 IVX rows = 15;
//  * the D->D chain D(k+1) = M(k) tMD(k) + D(k) tDD(k) is a first-order linear recurrence: a serial
//    pass inside the lane plus a 5-step warp-shuffle scan whose multipliers are profile constants;
//  * E(i) = sum_k M(i,k)+D(i,k) equals sum_k M(i,k) Z(k) with the profile constant
//    Z(k) = 1 + tMD(k) (1 + tDD(k+1) + tDD(k+1) tDD(k+2) + ...), so E (hence B(i), hence row i+2)
//    does not wait for the D scan; Z(k) and the entry odds tBM(k-1) are folded into the emission
//    table once per profile, which removes two constants and two multiplies per node and row;
//  * the three emission rows of a DP row are read with coalesced 128/64/32-bit loads from a table laid
//    out [codon][J/VEC][lane][VEC]; the table is L1/L2 resident (0.3 MB at M=200);
//  * target nucleotides are 4-bit packed; each lane turns 4 nibbles into the three emission-row indices of
//    one DP row, 32 rows per step, and rows pick their word up with one shuffle;
//  * rows are unrolled by 4 so every ring slot is a compile-time register name; the window is entered
//    through 0..3 all-zero pad rows in front so that the last quad ends exactly at row L.
//
// Rescaling follows the reference: when E(i) > 1e4 everything live is divided by E(i) and log E(i)
// is accumulated (fwdback_fs.c:472-496).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bathgpu {

constexpr int kWarp = 32;

// lane-constant image: [NC][J][32] floats then [NL][32] floats
enum FwdCellConst { FC_MM = 0, FC_DM, FC_MD, FC_DD, FC_MI, FC_II, FC_COUNT };
enum FwdLaneConst { FL_B0 = 0, FL_B1, FL_B2, FL_B3, FL_B4, FL_COUNT };

struct WindowDesc {      // device copy of bathgpu_window
  long long start;       // 1-based block coordinate of window position 1
  int       L;
  float     pmove;
  float     ploop;
};

// One profile of a resident profile set (bathgpu_load_fs_profile_set): the pointers a kernel otherwise takes from its arguments,
// read per window in the kernels' SET instantiations.  Every profile of one launch has the same node count per lane J.
struct FsSetProfile {
  const float *emis;           // the table the kernel reads: emis_fwd (3 codon lengths) or emis (5)
  const float *cellc;          // lane constants: cellc (3) or cellf5 (5)
  const float *cellmw;         // multi-warp Forward constants (J >= 16: fs_parser_mw.cuh for 3 codon lengths, fs_domain_mw.cuh for 5), else null
  float        tEM, tEL;       // E->MOVE, E->LOOP odds of this profile
};

struct FsParserArgs {
  const float    *emis;        // [nrows][mpad] permuted odds table (3-codon profile)
  const float    *cellc;       // lane-constant image
  const uint32_t *dna4;        // 4-bit packed block, nt p (0-based) at word (p+8)>>3 (one guard word in front)
  const WindowDesc *wins;
  int             nwin;
  int             mpad;        // 32*J
  float           tEM, tEL;    // E->MOVE, E->LOOP odds
  float          *fwdsc;       // [nwin]
  int            *status;      // [nwin]
  float          *xmx;         // optional: X rows, window w at xmx + xoff[w]*6
  const long long *xoff;
  int            *counter;     // work-queue counter
  int             scan_steps;  // steps of the D->D warp scan this profile needs (5 = all; fewer when the D->D odds products die out)
  const float    *cellmw;      // lane-constant image of the multi-warp kernel (fs_parser_mw.cuh); null for models the one-warp kernels keep in registers
  int             mw_scan_steps;
  const FsSetProfile *set;     // SET instantiations: window w is scored with profile set[wprof[w]] (emis, cellc, cellmw, tEM, tEL unused)
  const int      *wprof;
};

template <int J> struct VecOf { static constexpr int V = (J % 4 == 0) ? 4 : ((J % 2 == 0) ? 2 : 1); };

// 3-codon index macros (src/hmmer.h:312-314) with the reference's clamp to the degenerate rows (:347-349)
__device__ __forceinline__ int codon2_fs3(int w, int x)               { int c = x * 84 + w * 21;                 return min(c, 337); }
__device__ __forceinline__ int codon3_fs3(int v, int w, int x)        { int c = x * 84 + w * 21 + v * 5 + 1;     return min(c, 336); }
__device__ __forceinline__ int codon4_fs3(int u, int v, int w, int x) { int c = x * 84 + w * 21 + v * 5 + u + 2; return min(c, 337); }

template <int J, int VEC>
__device__ __forceinline__ void load_emission_row(const float *__restrict__ row, float (&e)[J])
{
#pragma unroll
  for (int g = 0; g < J / VEC; ++g) {
    if constexpr (VEC == 4) {
      float4 t = __ldg(reinterpret_cast<const float4 *>(row) + g * kWarp);
      e[4 * g + 0] = t.x; e[4 * g + 1] = t.y; e[4 * g + 2] = t.z; e[4 * g + 3] = t.w;
    } else if constexpr (VEC == 2) {
      float2 t = __ldg(reinterpret_cast<const float2 *>(row) + g * kWarp);
      e[2 * g + 0] = t.x; e[2 * g + 1] = t.y;
    } else {
      e[g] = __ldg(row + g * kWarp);
    }
  }
}

__device__ __forceinline__ float warp_allsum(float v)
{
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  return v;
}

// fetch the 16 bits (4 nucleotides) for rows i..i+3 of a window; p0 = 0-based block index of row i
// Two warp-wide sums in one butterfly (the E sums of a Forward row pair, the B sums of a Backward one): lanes 0-15 collect row i, lanes 16-31 row i+1 (6 shuffles for the pair instead of 10); every
// lane ends with the same bits for each sum (the halves exchange their finished sums), so the rescale test stays warp-uniform.
__device__ __forceinline__ void pair_allsum(int lane, float a, float b, float &sa, float &sb)
{
  const bool lo = lane < 16;
  float mine = (lo ? a : b) + __shfl_xor_sync(0xffffffffu, lo ? b : a, 16);
  mine += __shfl_xor_sync(0xffffffffu, mine, 8);
  mine += __shfl_xor_sync(0xffffffffu, mine, 4);
  mine += __shfl_xor_sync(0xffffffffu, mine, 2);
  mine += __shfl_xor_sync(0xffffffffu, mine, 1);
  const float other = __shfl_xor_sync(0xffffffffu, mine, 16);
  sa = lo ? mine : other;
  sb = lo ? other : mine;
}

__device__ __forceinline__ uint32_t fetch_quad(const uint32_t *__restrict__ dna4, long long p0)
{
  long long q  = p0 + 8;                 // guard word in front
  long long wi = q >> 3;
  int       sh = (int)(q & 7) * 4;
  uint32_t lo = __ldg(dna4 + wi), hi = __ldg(dna4 + wi + 1);
  return __funnelshift_r(lo, hi, sh) & 0xffffu;
}

template <int J>
struct FwdState {
  float W[4][J];       // W(r)[k] = V(r)[k] / s(k), s(k) = tBM(k-1), in slot r&3   (V = the reference's IVX)
  float I[4][J];       // Ih(r)[k] = I(r,k) tIM(k) / (s(k+1) hi(k)) in slot r&3 (FwdConsts)
  float xN[4], xJ[4], xC[4];
};

// Per-node constants.  The Forward parsers read their own copy of the emission table (FsProfileImage::emis_fwd) with the entry
// odds s(k) = tBM(k-1), the E weight Z(k) and the match->match odds folded in:
//   T[c][k] = R[c][k] s(k) Z(k) mm(k),  mm(k) = tMM(k) / (Z(k) s(k+1))   =>   sum_c W T = Mq := M(i,k) Z(k) mm(k)
// so that the flow into node k+1 takes Mq with coefficient 1, and the other two chains are carried divided by whatever makes
// Mq enter them with coefficient 1 as well -- no chain multiplies the match value:
//   E(i)          = sum_k Mq qm,                 qm = 1 / mm(k)                       (an FMA where a plain sum would need an add)
//   Dg(k) = D(k) / g(k),  g(k+1) = tMD(k) / (Z(k) mm(k)),  g(1) = 1:
//   Dg(k+1)       = Dg(k) dd + Mq,               dd = g(k) tDD(k) / g(k+1)
//   Ih(k) = I(k) tIM(k) / (s(k+1) hi),           hi = tMI(k) tIM(k) / tMM(k):
//   Ih(i+3,k)     = Ih(i,k) ii + Mq,             ii = tII(k)
//   flow(k)       = Mq + Ih hi + Dg dm,          dm = g(k) tDM(k) / s(k+1)
// 10 floating-point instructions per cell against 12 with every transition applied where the reference applies it.
// Node M (no way out) and nodes with a vanishing tMM / tMD / tMI take tiny stand-ins for the divisors (bathgpu.cu).
template <int J>
struct FwdConsts {
  float qm[J], dm[J], dd[J], hi[J], ii[J];
  float bs[5];
};

template <int J>
__device__ __forceinline__ void load_fwd_consts(const float *__restrict__ cc, int lane, FwdConsts<J> &K)
{
#pragma unroll
  for (int j = 0; j < J; ++j) {
    K.qm[j] = __ldg(cc + (FC_MM * J + j) * kWarp + lane);
    K.dm[j] = __ldg(cc + (FC_DM * J + j) * kWarp + lane);
    K.dd[j] = __ldg(cc + (FC_DD * J + j) * kWarp + lane);
    K.hi[j] = __ldg(cc + (FC_MI * J + j) * kWarp + lane);
    K.ii[j] = __ldg(cc + (FC_II * J + j) * kWarp + lane);
  }
#pragma unroll
  for (int s = 0; s < 5; ++s) K.bs[s] = __ldg(cc + FC_COUNT * J * kWarp + (FL_B0 + s) * kWarp + lane);
}

// Codon words for 32 consecutive padded rows, one per lane: lane l handles padded row r0 + l, i.e.
// DP row i = r0 + l - pad.  n[p] for p outside 1..L or a degenerate code is the placeholder 338
// (fwdback_fs.c:176-178,344), which the index clamps turn into the degenerate emission rows (:347-349).
__device__ __forceinline__ uint32_t codon_word(uint32_t lo, uint32_t hi, int sh, int i, int L)
{
  uint32_t bits = __funnelshift_r(lo, hi, sh) & 0xffffu;       // nibbles n[i-3], n[i-2], n[i-1], n[i]
  int u = (int)(bits & 15u), v = (int)((bits >> 4) & 15u), w = (int)((bits >> 8) & 15u), x = (int)(bits >> 12);
  u = (u < 4 && i - 3 >= 1 && i - 3 <= L) ? u : 338;
  v = (v < 4 && i - 2 >= 1 && i - 2 <= L) ? v : 338;
  w = (w < 4 && i - 1 >= 1 && i - 1 <= L) ? w : 338;
  x = (x < 4 && i     >= 1 && i     <= L) ? x : 338;
  return (uint32_t)codon2_fs3(w, x) | ((uint32_t)codon3_fs3(v, w, x) << 9) | ((uint32_t)codon4_fs3(u, v, w, x) << 18);
}

}  // namespace bathgpu

// ---------------------------------------------------------------------------------------------
// Protein Forward parser over ORFs: p7_ForwardParser (reference src/impl_sse/fwdback.c:132, engine :256-466),
// the F3/F4 gate between the integer filters and the frameshift stage (src/p7_pipeline.c:1774-1789).
// Same carried quantities as the frameshift parser -- W = entry value / tBM, I~ = I tIM / s(k+1), E = sum M Z --
// with a one-row look-back; it reads the amino-acid rows (338 + x) of the SAME folded 3-codon emission table
// and the same lane constants, because the frameshift profile's amino rows and transitions are the protein
// profile's (src/modelconfig.c:343-352 vs :140-156).
namespace bathgpu {

struct OrfFwdArgs {
  const float    *emis;        // 3-codon image; amino rows start at row 338
  const float    *cellc;
  const uint8_t  *residues;
  const void     *orfs;        // OrfDesc[] (orf_filters.cuh): offset, L
  int             orf_stride;
  int             norf;
  int             mpad;
  float           nj;          // expected J uses of the protein profile (1 in bathsearch: multihit local)
  float           tEM, tEL;
  float          *fwdsc;
  int            *status;
  int            *counter;
};

template <int J>
__global__ void __launch_bounds__(32) orf_forward_parser_kernel(OrfFwdArgs a)
{
  constexpr int VEC = VecOf<J>::V;
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  FwdConsts<J> K;
  load_fwd_consts<J>(a.cellc, lane, K);
  const float *emis_lane = a.emis + (size_t)338 * a.mpad + lane * VEC;

  for (;;) {
    int o = 0;
    if (lane == 0) o = atomicAdd(a.counter, 1);
    o = __shfl_sync(full, o, 0);
    if (o >= a.norf) break;
    const char *od = reinterpret_cast<const char *>(a.orfs) + (size_t)o * a.orf_stride;
    const long long off = *reinterpret_cast<const long long *>(od);
    const int L = *reinterpret_cast<const int *>(od + 8);
    const float pmove = (2.0f + a.nj) / ((float)L + 2.0f + a.nj);      // p7_oprofile_ReconfigRestLength (p7_oprofile.c:1312-1313)
    const float ploop = 1.0f - pmove;

    float W[J], It[J];
#pragma unroll
    for (int j = 0; j < J; ++j) { W[j] = pmove; It[j] = 0.f; }         // row 0: B = tNM, nothing else (:281-285)
    float xN = 1.0f, xJ = 0.f, xC = 0.f, totscale = 0.f;

    int chunk = -64;
    unsigned myres = 0;
    for (int i = 1; i <= L; ++i) {
      if (i >= chunk + 32) { chunk = i; myres = (i + lane <= L) ? a.residues[off + i + lane - 1] : 0u; }
      const unsigned x = __shfl_sync(full, myres, i - chunk);
      float e[J], m[J];
      load_emission_row<J, VEC>(emis_lane + (size_t)x * a.mpad, e);
      float es = 0.f;
#pragma unroll
      for (int j = 0; j < J; ++j) { m[j] = W[j] * e[j]; es = fmaf(m[j], K.qm[j], es); }
      float xE = warp_allsum(es);

      float A = 0.f;
#pragma unroll
      for (int j = 0; j < J; ++j) A = (j == 0) ? m[0] : fmaf(A, K.dd[j], m[j]);
#pragma unroll
      for (int s = 0; s < 5; ++s) {
        float up = __shfl_up_sync(full, A, 1 << s);
        A = fmaf(K.bs[s], up, A);
      }
      float d = __shfl_up_sync(full, A, 1);
      if (lane == 0) d = 0.f;

      xN = xN * ploop;                                    // (:401-404)
      xC = fmaf(xC, ploop, xE * a.tEM);
      xJ = fmaf(xJ, ploop, xE * a.tEL);
      float xB = fmaf(xJ, pmove, xN * pmove);

      float ov[J];
#pragma unroll
      for (int j = 0; j < J; ++j) {
        float t = fmaf(It[j], K.hi[j], m[j]);
        ov[j] = fmaf(d, K.dm[j], t);
        if (j + 1 < J) d = fmaf(d, K.dd[j], m[j]);
        It[j] = fmaf(It[j], K.ii[j], m[j]);
      }
      float oprev = __shfl_up_sync(full, ov[J - 1], 1);
      if (lane == 0) oprev = 0.f;
      W[0] = xB + oprev;
#pragma unroll
      for (int j = 1; j < J; ++j) W[j] = xB + ov[j - 1];

      if (xE > 1.0e4f) {                                   // sparse rescaling (:407-423)
        const float sf = 1.0f / xE;
        xN *= sf; xC *= sf; xJ *= sf;
#pragma unroll
        for (int j = 0; j < J; ++j) { W[j] *= sf; It[j] *= sf; }
        totscale += logf(xE);
      }
    }
    int   st = 0;
    float sc;
    if (isnan(xC))                 { st = 16; sc = xC; }                 // (:447-449)
    else if (L > 0 && xC == 0.0f)  { st = 16; sc = -INFINITY; }
    else if (isinf(xC))            { st = 16; sc = xC; }
    else sc = totscale + logf(xC * pmove);
    if (lane == 0) { a.fwdsc[o] = sc; a.status[o] = st; }
  }
}

}  // namespace bathgpu
