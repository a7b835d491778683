// orf_filters.cuh -- the integer filters of the ORF stage for sm_100a:
//   p7_MSVFilter (+ its p7_SSVFilter shortcut)   reference src/impl_sse/msvfilter.c:74-208, ssvfilter.c:831-925
//   p7_SSVFilter_BATH (window finder)            src/impl_sse/msvfilter.c:250-427
//   p7_ViterbiFilter / p7_ViterbiFilter_BATH     src/impl_sse/vitfilter.c:83-248, :286-465
//
// One warp per ORF.  Lane l owns a CONTIGUOUS run of model nodes packed four uint8 (MSV) or two int16
// (Viterbi) per 32-bit register and uses the SIMD-in-a-word video instructions (__vmaxu4 / __vaddus4 /
// __vsubus4, __vmaxs2 / __vaddss2), which are exactly the saturating byte/word operations the CPU code
// issues, so every cell is bit-identical to the reference's.  The k-1 look-back is a funnel shift across
// the lane's registers plus one shuffle; row maxima are a byte/half fold plus one redux.sync.
// The score tables (byte costs 29 x Mpad, word scores 29 x Mpad, transitions 8 x Mpad) live in shared
// memory, loaded once per block.
//
// What is kept of the CPU's striped layout is only what shows in results: when a window finder must pick
// one cell among equals it scans in the reference's order k = q + Q z + 1 (q outer), Q = max(2, ceil(M / lanes)),
// with `lanes` the lanes per vector of the CPU build being matched (16/8 SSE, 32/16 AVX2).
//
// MSV: the reference first tries the J-less SSV shortcut and falls back to the full recursion when the J
// state could matter (ssvfilter.c:14-210).  The shortcut's cells equal max(MSV cell, begin score), so its answer
// is the full recursion's with the row maximum floored at the begin score; this kernel runs the full recursion
// and applies that floor when the shortcut would have answered.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace bathgpu {

struct OrfDesc {           // device copy of bathgpu_orf
  long long offset;        // index of the first residue in the uploaded residue buffer
  int       L;
  uint8_t   tjb_b;         // unbiased_byteify(logf(3/(L+3)))          p7_oprofile.c:1287
  uint8_t   ssv_thresh;    // sc_thresh of p7_SSVFilter_BATH            msvfilter.c:313
  int16_t   xw_move;       // wordify(logf(pmove))                      p7_oprofile.c:1320
  int16_t   vit_thresh;    // sc_thresh of p7_ViterbiFilter_BATH        vitfilter.c:315
  int16_t   flags;         // bit 0: emit Viterbi windows
  int       ext_thresh;    // sc_ext_thresh of p7_ViterbiFilter_BATH    vitfilter.c:319-321
};

struct WindowRec { int orf, n, k, length; float score; };
struct MsvSetProfile;
struct MsvSetTile;

struct FilterArgs {
  const uint8_t  *residues;
  int             res_stride;   // 1: residue buffer; 3: codon classes of the resident strand, one per nucleotide (orf_finder.cuh; MSV scores only)
  const OrfDesc  *orfs;
  int             norf;
  int             M;
  // bytes
  const uint32_t *rbv;       // [29][32*W] words, node k at byte k-1 of a row; pad bytes 255
  const uint32_t *nrb;       // [29][32*P] words, -cost of node k at half k-1 (msv16_filter_kernel); pad -255
  const uint8_t  *rbv_bytes; // same table, byte addressed (diagonal walks)
  int             rowwords_b;
  int             tbm_b, tec_b, base_b, bias_b;
  float           scale_b;
  // words
  const uint32_t *rwv;       // [29][32*P] words, node k at half k-1; pad -32768
  const uint32_t *twv;       // [8][32*P]: BM,MM,IM,DM aligned to the TARGET node (source k-1); MD,MI,II,DD to the source node
  const int      *ddsum;     // [5][32] + [32]: path sums of the DD scan (lane constants)
  int             rowwords_w;
  int             base_w, ddbound_w, xw_E_move, xw_E_loop;
  float           scale_w;
  int             lanes_u8, lanes_i16;
  // out
  float          *sc;
  int            *status;
  WindowRec      *wins;
  int            *nwins;
  int             max_wins;
  int            *counter;
  // msv16_filter_kernel<P, true>: the tiles of a profile-set screen and the set's profiles
  const MsvSetTile    *set_tiles;
  int                  set_ntiles;
  const MsvSetProfile *set_profiles;
};

__device__ __forceinline__ unsigned bytemax(unsigned v) { v = __vmaxu4(v, v >> 16); v = __vmaxu4(v, v >> 8); return v & 0xffu; }
__device__ __forceinline__ int halfmax(unsigned v) { int lo = (int)(short)(v & 0xffffu), hi = (int)(short)(v >> 16); return max(lo, hi); }

template <int W> __device__ __forceinline__ void lds_words(const uint32_t *p, uint32_t (&v)[W])
{
  if constexpr (W == 1)      v[0] = p[0];
  else if constexpr (W == 2) { uint2 t = *reinterpret_cast<const uint2 *>(p); v[0] = t.x; v[1] = t.y; }
  else if constexpr (W == 4) { uint4 t = *reinterpret_cast<const uint4 *>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
  else {
#pragma unroll
    for (int w = 0; w < W; ++w) v[w] = p[w];
  }
}

// reference scan order of node k among equal cells: q outer, lane-of-vector z inner, k = q + Q z + 1
__device__ __forceinline__ int stripe_key(int k, int Q, int lanes) { int q = (k - 1) % Q, z = (k - 1) / Q; return q * lanes + z; }
__device__ __forceinline__ int stripe_node(int key, int Q, int lanes) { int q = key / lanes, z = key % lanes; return q + Q * z + 1; }

// ---------------------------------------------------------------------------------------------
// MSV scores (MODE 0) and SSV windows (MODE 1).  W = words per lane (4 W nodes per lane).
template <int W, int MODE>
__global__ void __launch_bounds__(128) msv_filter_kernel(FilterArgs a)
{
  extern __shared__ uint32_t smem[];
  uint32_t *s_rbv = smem;                                  // [29][32*W]
  const int rowwords = 32 * W;
  for (int t = threadIdx.x; t < 29 * rowwords; t += blockDim.x) s_rbv[t] = a.rbv[t];
  __syncthreads();

  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  const unsigned biasv = (unsigned)a.bias_b * 0x01010101u;
  const int Q = max(2, (a.M - 1) / a.lanes_u8 + 1);

  for (;;) {
    int o = 0;
    if (lane == 0) o = atomicAdd(a.counter, 1);
    o = __shfl_sync(full, o, 0);
    if (o >= a.norf) break;
    const OrfDesc od = a.orfs[o];
    const int L = od.L;
    if (od.flags & 2) {                                    // wholly inside the block's overlap context: not scored (p7_pipeline.c:1634-1637)
      if (MODE == 0 && lane == 0) { a.sc[o] = -INFINITY; a.status[o] = 0; }
      continue;
    }
    const int tjbm = (int)(uint8_t)((int8_t)od.tjb_b + (int8_t)a.tbm_b);      // set1_epi8 of the 8-bit sum (:120)
    uint32_t m[W];
#pragma unroll
    for (int w = 0; w < W; ++w) m[w] = 0;
    int xJ = 0;
    int xB = max(a.base_b - tjbm, 0);
    unsigned xBv = (unsigned)xB * 0x01010101u;
    int st = 0;
    const int sc_thresh = od.ssv_thresh;

    int chunk = -64;                 // first residue held in myres (32 at a time, one per lane)
    unsigned myres = 0;
    for (int i = 1; i <= L; ++i) {
      {
        if (i >= chunk + 32 || i < chunk) {
          chunk = i;
          myres = (i + lane <= L) ? a.residues[od.offset + (long long)(i + lane - 1) * a.res_stride] : 0u;
        }
        const unsigned x = __shfl_sync(full, myres, i - chunk);
        uint32_t rb[W];
        lds_words<W>(s_rbv + x * rowwords + lane * W, rb);
        unsigned carry = __shfl_up_sync(full, m[W - 1], 1);
        if (lane == 0) carry = 0;                           // zeros shift in: -infinity (:139-143)
        unsigned rowmax = 0;
#pragma unroll
        for (int w = W - 1; w >= 0; --w) {
          unsigned lo = (w == 0) ? carry : m[w - 1];
          unsigned sv = __funnelshift_l(lo, m[w], 8);      // previous row, node k-1
          sv = __vmaxu4(sv, xBv);
          sv = __vaddus4(sv, biasv);
          sv = __vsubus4(sv, rb[w]);
          m[w] = sv;
          rowmax = __vmaxu4(rowmax, sv);
        }
        const int xE = (int)__reduce_max_sync(full, bytemax(rowmax));
        if constexpr (MODE == 0) {
          if (xE + a.bias_b >= 255) { st = 16; break; }    // overflow (:155-180)
          const int xEt = max(xE - a.tec_b, 0);
          xJ = max(xJ, xEt);
          xB = max(max(a.base_b, xJ) - tjbm, 0);
          xBv = (unsigned)xB * 0x01010101u;
        } else {
          if (xE >= sc_thresh) {                            // (:343-347) threshold reached: emit a window
            // the cell: highest value, first in the reference's scan order among equals (:352-364)
            unsigned best = 0xffffffffu;
#pragma unroll
            for (int w = 0; w < W; ++w)
#pragma unroll
              for (int b = 0; b < 4; ++b) {
                const int k = 4 * (lane * W + w) + b + 1;
                const int v = (int)((m[w] >> (8 * b)) & 0xffu);
                if (k <= a.M && v >= sc_thresh) best = min(best, ((unsigned)(255 - v) << 16) | (unsigned)stripe_key(k, Q, a.lanes_u8));
              }
            best = __reduce_min_sync(full, best);
            int end = stripe_node((int)(best & 0xffffu), Q, a.lanes_u8);
            int rem_sc = 255 - (int)(best >> 16);
#pragma unroll
            for (int w = 0; w < W; ++w) m[w] = 0;           // dp reset (:366)
            // walk the diagonal back to where it left the baseline, then extend it (:369-405); every lane
            // does the same scalar walk on broadcast loads
            const uint8_t *res = a.residues + od.offset - 1; // res[i] = residue i
            const int rw8 = a.rowwords_b * 4;
            int start = end, tstart = i, sc = rem_sc;
            while (rem_sc > a.base_b - (int)od.tjb_b - a.tbm_b) {
              rem_sc -= a.bias_b - (int)a.rbv_bytes[(size_t)res[tstart] * rw8 + (start - 1)];
              --start; --tstart;
            }
            start++; tstart++;
            int k = end + 1, n = i + 1, max_end = i, max_sc = sc, since = 0;
            while (k < a.M && n <= L) {
              sc += a.bias_b - (int)a.rbv_bytes[(size_t)res[n] * rw8 + (k - 1)];
              if (sc >= max_sc) { max_sc = sc; max_end = n; since = 0; }
              else if (++since == 5) break;
              k++; n++;
            }
            end += (max_end - i);
            float ret = ((float)(max_sc - (int)od.tjb_b) - (float)a.base_b);
            ret /= a.scale_b;
            ret -= 3.0f;
            if (lane == 0) {
              int slot = atomicAdd(a.nwins, 1);
              if (slot < a.max_wins) { WindowRec wr; wr.orf = o; wr.n = tstart; wr.k = end; wr.length = end - start + 1; wr.score = ret; a.wins[slot] = wr; }
            }
            i = max_end;                                      // skip forward (:424); the loop adds one
          }
        }
      }
    }
    if constexpr (MODE == 0) {
      if (lane == 0) {
        float sc;
        if (st) sc = INFINITY;
        else {                                               // (:203-205)
          // When the J state was never reachable the reference's answer comes from the SSV shortcut, whose cells are
          // floored at the begin score instead of at 0 (cellwise max(MSV cell, xB0): ssvfilter.c:130-170), so an ORF
          // with no cell above the begin score reports the begin score itself.  Same preconditions as the shortcut (:882-917).
          const int floorJ = a.base_b - (int)od.tjb_b - a.tbm_b - a.tec_b;
          if ((int)od.tjb_b + a.tbm_b + a.tec_b + a.bias_b < 127 && xJ <= a.base_b && floorJ >= 0) xJ = max(xJ, floorJ);
          sc = ((float)(xJ - (int)od.tjb_b) - (float)a.base_b);
          sc /= a.scale_b;
          sc -= 3.0f;
        }
        a.sc[o] = sc; a.status[o] = st;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// MSV scores on 16-bit lanes.  The byte-SIMD intrinsics above are emulated on this architecture (about seven integer
// instructions each), while the 16-bit min/max/add-then-clamp family (VIMNMX.S16x2, VIADDMNMX.S16x2, VIMNMX3) is native:
// carrying each uint8 cell in a 16-bit lane and clamping explicitly -- min(v + bias, 255), max(v - cost, 0) -- gives the
// same values as the saturating byte operations (msvfilter.c:145-148) in one instruction per step and two nodes per
// register.  P = words per lane (2 P nodes), the Viterbi filter's layout; costs are stored negated.
// One row of the recurrence on 16-bit lanes: returns the row's cells in m[] and folds them into rowmax.
template <int P>
__device__ __forceinline__ void msv16_row(const uint32_t *__restrict__ s_nrb_lane, unsigned x, int rowwords, int lane, uint32_t (&m)[P],
                                          unsigned xBv, unsigned biasv, unsigned &rowmax)
{
  uint32_t rb[P];
  lds_words<P>(s_nrb_lane + x * rowwords, rb);
  unsigned carry = __shfl_up_sync(0xffffffffu, m[P - 1], 1);
  if (lane == 0) carry = 0;                               // zeros shift in (:139-143)
#pragma unroll
  for (int w = P - 1; w >= 0; --w) {
    const unsigned lo = (w == 0) ? carry : m[w - 1];
    unsigned sv = __funnelshift_l(lo, m[w], 16);          // previous row, node k-1
    sv = __vmaxs2(sv, xBv);
    sv = __viaddmin_s16x2(sv, biasv, 0x00ff00ffu);        // adds_epu8(sv, bias)
    sv = __viaddmax_s16x2(sv, rb[w], 0u);                 // subs_epu8(sv, cost)
    m[w] = sv;
    rowmax = __vmaxs2(rowmax, sv);
  }
}

// A profile of a resident set (bathgpu_load_filter_profile_set): its MSV cost table and the byte parameters the recurrence reads.
struct MsvSetProfile {
  const uint32_t *nrb;       // [29][32*P] words, as FilterArgs::nrb
  int             P;
  int             tbm_b, tec_b, base_b, bias_b;
  float           scale_b;
};
// A run of consecutive ORFs of one job of bathgpu_orfs_msv_screen_set, all scored with one profile: descriptors orfs[desc0 ..
// desc0 + n - 1], scores written to sc[out0 ..].
struct MsvSetTile { int profile, n; long long desc0, out0; };
constexpr int kMsvSetTileOrfs = 256;

// One ORF of the MSV recurrence on 16-bit lanes: its score and status (meaningful in lane 0).
// Rows are taken 32 at a time (one residue per lane).  While the J state is out of reach -- E never exceeds base + tEC, so B keeps
// its initial value -- the per-row maximum is not needed row by row: a chunk runs without any reduction and its overall maximum is
// reduced once (this is the reference's SSV shortcut, ssvfilter.c:14-210, taken per chunk).  A chunk whose maximum shows that J
// became reachable or that a cell overflowed is re-run from its saved first row with the exact per-row recurrence (msvfilter.c:145-201).
template <int P>
__device__ __forceinline__ void msv16_orf(const FilterArgs &a, const OrfDesc &od, const uint32_t *__restrict__ s_nrb_lane, int lane,
                                          float &sc_out, int &st_out)
{
  const int rowwords = 32 * P;
  const unsigned full = 0xffffffffu;
  const unsigned biasv = (unsigned)a.bias_b * 0x00010001u;
  {
    const int L = od.L;
    if (od.flags & 2) {                                    // wholly inside the block's overlap context: not scored (p7_pipeline.c:1634-1637)
      sc_out = -INFINITY; st_out = 0;
      return;
    }
    const int tjbm = (int)(uint8_t)((int8_t)od.tjb_b + (int8_t)a.tbm_b);      // set1_epi8 of the 8-bit sum (:120)
    uint32_t m[P];
#pragma unroll
    for (int w = 0; w < P; ++w) m[w] = 0;
    int xJ = 0;
    int xB = max(a.base_b - tjbm, 0);
    unsigned xBv = (unsigned)xB * 0x00010001u;
    int st = 0;
    bool exact = false;                                    // J reachable: B moves with it, every row needs its own maximum

    for (int i0 = 1; i0 <= L && !st; i0 += 32) {
      const int nrow = min(32, L - i0 + 1);
      const unsigned myres = (lane < nrow) ? a.residues[od.offset + (long long)(i0 + lane - 1) * a.res_stride] : 0u;
      if (!exact) {
        uint32_t m0[P];
#pragma unroll
        for (int w = 0; w < P; ++w) m0[w] = m[w];
        unsigned cmax = 0;
        for (int r = 0; r < nrow; ++r)
          msv16_row<P>(s_nrb_lane, __shfl_sync(full, myres, r), rowwords, lane, m, xBv, biasv, cmax);
        const int xEc = (int)__reduce_max_sync(full, (int)max(cmax & 0xffffu, cmax >> 16));
        if (xEc + a.bias_b < 255 && xEc - a.tec_b <= a.base_b) { xJ = max(xJ, max(xEc - a.tec_b, 0)); continue; }
        exact = true;                                      // redo this chunk row by row
#pragma unroll
        for (int w = 0; w < P; ++w) m[w] = m0[w];
      }
      for (int r = 0; r < nrow; ++r) {
        unsigned rowmax = 0;
        msv16_row<P>(s_nrb_lane, __shfl_sync(full, myres, r), rowwords, lane, m, xBv, biasv, rowmax);
        const int xE = (int)__reduce_max_sync(full, (int)max(rowmax & 0xffffu, rowmax >> 16));
        if (xE + a.bias_b >= 255) { st = 16; break; }       // overflow (:155-180)
        const int xEt = max(xE - a.tec_b, 0);
        xJ = max(xJ, xEt);
        xB = max(max(a.base_b, xJ) - tjbm, 0);
        xBv = (unsigned)xB * 0x00010001u;
      }
    }
    float sc;
    if (st) sc = INFINITY;
    else {                                                   // (:203-205), with the SSV shortcut's floor (see msv_filter_kernel)
      const int floorJ = a.base_b - (int)od.tjb_b - a.tbm_b - a.tec_b;
      if ((int)od.tjb_b + a.tbm_b + a.tec_b + a.bias_b < 127 && xJ <= a.base_b && floorJ >= 0) xJ = max(xJ, floorJ);
      sc = ((float)(xJ - (int)od.tjb_b) - (float)a.base_b);
      sc /= a.scale_b;
      sc -= 3.0f;
    }
    sc_out = sc; st_out = st;
  }
}

// MSV scores of the ORFs a.orfs[0 .. norf-1] with the loaded profile (SET = false), or of the (job, ORF) runs a.set_tiles with the
// profiles of a resident set (SET = true): a block takes a tile, stages the tile's profile table unless it holds it already, and its
// warps take the tile's ORFs one at a time.  Both run the same recurrence (msv16_orf) on the same tables, so the scores are the same.
template <int P, bool SET>
__global__ void __launch_bounds__(128) msv16_filter_kernel(FilterArgs a)
{
  extern __shared__ uint32_t smem[];
  uint32_t *s_nrb = smem;                                  // [29][32*P] words: -cost of node k at half k-1
  const int rowwords = 32 * P;
  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  const uint32_t *s_nrb_lane = s_nrb + lane * P;
  if constexpr (!SET) {
    for (int t = threadIdx.x; t < 29 * rowwords; t += blockDim.x) s_nrb[t] = a.nrb[t];
    __syncthreads();
    for (;;) {
      int o = 0;
      if (lane == 0) o = atomicAdd(a.counter, 1);
      o = __shfl_sync(full, o, 0);
      if (o >= a.norf) break;
      const OrfDesc od = a.orfs[o];
      float sc; int st;
      msv16_orf<P>(a, od, s_nrb_lane, lane, sc, st);
      if (lane == 0) { a.sc[o] = sc; a.status[o] = st; }
    }
  } else {
    __shared__ int s_tile, s_next;
    int staged = -1;
    for (;;) {
      if (threadIdx.x == 0) { s_tile = atomicAdd(a.counter, 1); s_next = 0; }
      __syncthreads();
      const int t = s_tile;
      if (t >= a.set_ntiles) break;
      const MsvSetTile tl = a.set_tiles[t];
      const MsvSetProfile pr = a.set_profiles[tl.profile];
      if (tl.profile != staged) {                          // every thread sees the same tiles: the block agrees on `staged`
        for (int z = threadIdx.x; z < 29 * rowwords; z += blockDim.x) s_nrb[z] = pr.nrb[z];
        staged = tl.profile;
      }
      __syncthreads();
      FilterArgs pa = a;
      pa.tbm_b = pr.tbm_b; pa.tec_b = pr.tec_b; pa.base_b = pr.base_b; pa.bias_b = pr.bias_b; pa.scale_b = pr.scale_b;
      for (;;) {
        int j = 0;
        if (lane == 0) j = atomicAdd(&s_next, 1);
        j = __shfl_sync(full, j, 0);
        if (j >= tl.n) break;
        const OrfDesc od = a.orfs[tl.desc0 + j];
        float sc; int st;
        msv16_orf<P>(pa, od, s_nrb_lane, lane, sc, st);
        if (lane == 0) { a.sc[tl.out0 + j] = sc; a.status[tl.out0 + j] = st; }
      }
      __syncthreads();                                     // the tile and the table stay until every warp is done with them
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Viterbi filter.  P = words per lane (2 P nodes per lane).
enum VitT { VT_BM = 0, VT_MM, VT_IM, VT_DM, VT_MD, VT_MI, VT_II, VT_DD };

template <int P>
__global__ void __launch_bounds__(128) vit_filter_kernel(FilterArgs a)
{
  extern __shared__ uint32_t smem[];
  const int rowwords = 32 * P;
  uint32_t *s_rwv = smem;                                  // [29][32*P]
  uint32_t *s_twv = smem + 29 * rowwords;                  // [8][32*P]
  for (int t = threadIdx.x; t < 29 * rowwords; t += blockDim.x) s_rwv[t] = a.rwv[t];
  for (int t = threadIdx.x; t < 8 * rowwords; t += blockDim.x)  s_twv[t] = a.twv[t];
  __syncthreads();

  const int lane = threadIdx.x & 31;
  const unsigned full = 0xffffffffu;
  const unsigned NEG = 0x80008000u;                        // two -32768
  const int Q = max(2, (a.M - 1) / a.lanes_i16 + 1);

  // the transitions of this lane's nodes stay in registers
  uint32_t tBM[P], tMM[P], tIM[P], tDM[P], tMD[P], tMI[P], tII[P];
  lds_words<P>(s_twv + VT_BM * rowwords + lane * P, tBM);
  lds_words<P>(s_twv + VT_MM * rowwords + lane * P, tMM);
  lds_words<P>(s_twv + VT_IM * rowwords + lane * P, tIM);
  lds_words<P>(s_twv + VT_DM * rowwords + lane * P, tDM);
  lds_words<P>(s_twv + VT_MD * rowwords + lane * P, tMD);
  lds_words<P>(s_twv + VT_MI * rowwords + lane * P, tMI);
  lds_words<P>(s_twv + VT_II * rowwords + lane * P, tII);

  for (;;) {
    int o = 0;
    if (lane == 0) o = atomicAdd(a.counter, 1);
    o = __shfl_sync(full, o, 0);
    if (o >= a.norf) break;
    const OrfDesc od = a.orfs[o];
    const int L = od.L;
    const bool emit = (od.flags & 1) != 0;
    uint32_t m[P], iv[P], d[P];
#pragma unroll
    for (int w = 0; w < P; ++w) { m[w] = NEG; iv[w] = NEG; d[w] = NEG; }
    int xN = a.base_w;
    int xB = (int)(short)(xN + od.xw_move);
    int xJ = -32768, xC = -32768, xE = -32768;
    int st = 0, skip_until = 0;

    int chunk = -64;
    unsigned myres = 0;
    for (int i = 1; i <= L; ++i) {
      {
        if (i >= chunk + 32) {
          chunk = i;
          myres = (i + lane <= L) ? a.residues[od.offset + i + lane - 1] : 0u;
        }
        const unsigned x = __shfl_sync(full, myres, i - chunk);
        uint32_t rw[P];
        lds_words<P>(s_rwv + x * rowwords + lane * P, rw);
        const unsigned xBv = ((unsigned)xB & 0xffffu) * 0x00010001u;
        unsigned cm = __shfl_up_sync(full, m[P - 1], 1), ci = __shfl_up_sync(full, iv[P - 1], 1), cd = __shfl_up_sync(full, d[P - 1], 1);
        if (lane == 0) { cm = NEG; ci = NEG; cd = NEG; }     // -32768 shifts in (:140-142)
        unsigned xEv = NEG, Dmaxv = NEG;
        uint32_t mn[P], dc[P];
#pragma unroll
        for (int w = P - 1; w >= 0; --w) {
          const unsigned mp = __funnelshift_l((w == 0) ? cm : m[w - 1], m[w], 16);
          const unsigned ip = __funnelshift_l((w == 0) ? ci : iv[w - 1], iv[w], 16);
          const unsigned dp = __funnelshift_l((w == 0) ? cd : d[w - 1], d[w], 16);
          unsigned sv = __vaddss2(xBv, tBM[w]);
          sv = __vmaxs2(sv, __vaddss2(mp, tMM[w]));
          sv = __vmaxs2(sv, __vaddss2(ip, tIM[w]));
          sv = __vmaxs2(sv, __vaddss2(dp, tDM[w]));
          sv = __vaddss2(sv, rw[w]);
          xEv = __vmaxs2(xEv, sv);
          mn[w] = sv;
          dc[w] = __vaddss2(sv, tMD[w]);                     // D(i,k+1), M->D only
          Dmaxv = __vmaxs2(Dmaxv, dc[w]);
          iv[w] = __vmaxs2(__vaddss2(m[w], tMI[w]), __vaddss2(iv[w], tII[w]));
        }
#pragma unroll
        for (int w = 0; w < P; ++w) m[w] = mn[w];
        // new D row: the M->D values move up one node
        {
          unsigned c = __shfl_up_sync(full, dc[P - 1], 1);
          if (lane == 0) c = NEG;
#pragma unroll
          for (int w = P - 1; w >= 0; --w) d[w] = __funnelshift_l((w == 0) ? c : dc[w - 1], dc[w], 16);
        }
        xE = __reduce_max_sync(full, halfmax(xEv));
        if (xE >= 32767) { st = 16; break; }                 // (:176)
        // specials in int arithmetic, stored as int16 (:177-181)
        xN = (int)(short)(xN + 0);
        xC = (int)(short)max(xC + 0, xE + a.xw_E_move);
        xJ = (int)(short)max(xJ + 0, xE + a.xw_E_loop);
        xB = (int)(short)max(xJ + (int)od.xw_move, xN + (int)od.xw_move);

        if (emit && i > skip_until && xE >= (int)od.vit_thresh) {     // (:386-423)
          unsigned best = 0xffffffffu;
#pragma unroll
          for (int w = 0; w < P; ++w)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int k = 2 * (lane * P + w) + h + 1;
              const int v = (int)(short)((m[w] >> (16 * h)) & 0xffffu);
              if (k <= a.M && v == xE) best = min(best, (unsigned)stripe_key(k, Q, a.lanes_i16));
            }
          best = __reduce_min_sync(full, best);
          const int k_start = (best == 0xffffffffu) ? 0 : stripe_node((int)best, Q, a.lanes_i16);
          const uint8_t *res = a.residues + od.offset - 1;
          const int rw8 = a.rowwords_b * 4;
          int max_k_end = k_start, max_i_end = i, sc_ext = od.ext_thresh, max_sc_ext = sc_ext, since = 0;
          int kk = k_start + 1, nn = i + 1;
          while (kk <= a.M && nn <= L) {
            sc_ext += a.bias_b - (int)a.rbv_bytes[(size_t)res[nn] * rw8 + (kk - 1)];
            if (sc_ext >= max_sc_ext) { max_sc_ext = sc_ext; max_k_end = kk; max_i_end = nn; since = 0; }
            else if (++since == 5) break;
            kk++; nn++;
          }
          if (lane == 0) {
            int slot = atomicAdd(a.nwins, 1);
            if (slot < a.max_wins) { WindowRec wr; wr.orf = o; wr.n = i; wr.k = max_k_end; wr.length = max_k_end - k_start + 1; wr.score = 0.0f; a.wins[slot] = wr; }
          }
          skip_until = max_i_end;
        }

        // lazy F (:197-231): D->D paths only when they could beat B->M on the next row
        const int Dmax = __reduce_max_sync(full, halfmax(Dmaxv));
        if (Dmax + a.ddbound_w > xB) {
          // complete closure d[k] = max(d[k], d[k-1] + tDD(k-1)) in 32-bit, floor at -32768 at the end:
          // all tDD <= 0, so the floor commutes with the saturating adds of the reference
          uint32_t tDD[P];
          lds_words<P>(s_twv + VT_DD * rowwords + lane * P, tDD);
          int dv[2 * P], td[2 * P];
#pragma unroll
          for (int w = 0; w < P; ++w) {
            dv[2 * w] = (int)(short)(d[w] & 0xffffu); dv[2 * w + 1] = (int)(short)(d[w] >> 16);
            td[2 * w] = (int)(short)(tDD[w] & 0xffffu); td[2 * w + 1] = (int)(short)(tDD[w] >> 16);     // tDD of node k: k -> k+1
          }
          // lane-local closure with nothing coming in
          int e = dv[0];
#pragma unroll
          for (int j = 1; j < 2 * P; ++j) e = max(dv[j], e + td[j - 1]);
          // scan of lane-end values: end(l) = max(e(l), end(l-1) + T(l)), T(l) = tDD(last node of l-1) + sum of this lane's tDD but the last
          int A = e;
#pragma unroll
          for (int s = 0; s < 5; ++s) {
            int up = __shfl_up_sync(full, A, 1 << s);
            int T  = a.ddsum[s * 32 + lane];
            if (lane >= (1 << s)) A = max(A, up + T);
          }
          int cin = __shfl_up_sync(full, A, 1);              // closure value at the last node of the previous lane
          int tin = a.ddsum[5 * 32 + lane];                  // tDD of that node
          cin = (lane == 0) ? -(1 << 28) : cin + tin;
          int run = cin;
#pragma unroll
          for (int j = 0; j < 2 * P; ++j) {
            run = max(dv[j], run);
            dv[j] = max(run, -32768);
            run = run + td[j];
          }
#pragma unroll
          for (int w = 0; w < P; ++w) d[w] = ((unsigned)dv[2 * w] & 0xffffu) | ((unsigned)dv[2 * w + 1] << 16);
        }
      }
    }
    if (lane == 0) {
      float sc;
      if (st) sc = INFINITY;
      else if (xC > -32768) {                                // (:238-246)
        sc = (float)xC + (float)od.xw_move - (float)a.base_w;
        sc /= a.scale_w;
        sc -= 3.0f;
      } else sc = -INFINITY;
      a.sc[o] = sc; a.status[o] = st;
    }
  }
}

}  // namespace bathgpu
