// orf_finder.cuh -- six-frame translation on the device (SURVEY §8 f1): ORFs of every block of the resident strand,
// straight into the MSV filter's input, and the F1 screen that follows it.
//
// Replaces, for a GPU build, Easel's esl_gencode_ProcessStart/Piece/End as bathsearch calls them (src/bathsearch.c:385-392:
// maximal stop-free runs of whole codons, at least min_len residues, any codon may start one, a codon holding a degenerate
// nucleotide translates to X) and the per-ORF loop head of p7_Pipeline_BATH (src/p7_pipeline.c:1632-1652).
//
//   codon_class_kernel   cls[s] = amino-acid code of the codon starting at strand position s+1 (27 = stop): 1 B per nucleotide,
//                        shared by the three frames and by every block that covers the position;
//   orf_scan_kernel      a stop codon (or the end of the block) at block position p closes the ORF of its frame, which starts behind
//                        the previous stop of that frame: found by a max-scan over the tile (a walk back over cls only for the
//                        first ORF of each frame in a tile).  Pass 1 counts ORFs per tile of 2048 positions; after a scan of the tile counts, pass 2
//                        writes the descriptors in order of p -- the order in which a left-to-right scan finishes ORFs,
//                        which is the reference's ORF order inside a block (the window bookkeeping depends on it);
//   (the MSV kernel then reads residues from cls with stride 3: nothing is materialised for the 98 % of ORFs that fail)
//   orf_screen_kernel    keeps an ORF when its MSV score could pass F1 (the caller re-does the exact test) or overflowed,
//                        and gathers the survivors' residues into the unit-stride residue buffer the later stages use.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "orf_filters.cuh"

namespace bathgpu {

constexpr int kOrfTileThreads = 256;
constexpr int kOrfPosPerThread = 8;
constexpr int kOrfTile = kOrfTileThreads * kOrfPosPerThread;
constexpr uint8_t kStopCode = 27;

struct GeneticCode { uint8_t aa[64]; };

struct BlockDesc {         // device copy of bathgpu_block
  long long goff;          // block position p (1..n) is strand position goff + p
  int       n;
  int       C;             // context nucleotides in front (bottom strand: behind, in block coordinates): ORFs inside it are not scored
};

struct OrfMeta { int block, index, start, end, frame; };     // block-local coordinates, index = rank inside the block

struct OrfHit {            // device copy of bathgpu_orf_hit
  int       block, index, start, end, n, frame;
  long long offset;        // first residue in the unit-stride residue buffer
  float     usc;
  int       status;
};

struct OrfScanArgs {
  const uint8_t   *cls;
  const BlockDesc *blocks;
  const int       *tile_block;     // [ntiles]
  const int       *tile_p0;        // [ntiles] first block position of the tile
  int              ntiles;
  int              min_len;
  int              complement;
  // pass 1 out
  int             *tile_cnt;
  // pass 2 in / out
  const long long *tile_base;      // exclusive scan of tile_cnt
  const long long *block_first;    // [nblocks] rank of the block's first ORF
  const uint8_t   *tjb_of;         // [max_len + 1]
  int              max_len;
  OrfDesc         *descs;
  OrfMeta         *meta;
  unsigned long long *scored;      // += residues of the ORFs that will be scored (the MSV stage's cell count / M)
};

__global__ void __launch_bounds__(256) codon_class_kernel(const uint32_t *__restrict__ dna4, long long n, GeneticCode gc, uint8_t *__restrict__ cls)
{
  // the 64-entry code table in shared memory: 16 words in 16 banks, so any 32 lookups are conflict-free (indexing the kernel
  // parameter instead serialises the lanes of a warp in the constant cache)
  __shared__ uint8_t s_aa[64];
  if (threadIdx.x < 64) s_aa[threadIdx.x] = gc.aa[threadIdx.x];
  __syncthreads();
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // nucleotides 8t .. 8t+7 (0-based)
  if (t * 8 >= n) return;
  const uint32_t w0 = __ldg(dna4 + t + 1), w1 = __ldg(dna4 + t + 2);       // one guard word in front
  const unsigned long long bits = ((unsigned long long)w1 << 32) | w0;
  unsigned long long out = 0;
#pragma unroll
  for (int b = 0; b < 8; ++b) {
    const unsigned a = (unsigned)(bits >> (4 * b)) & 15u, c = (unsigned)(bits >> (4 * b + 4)) & 15u, g = (unsigned)(bits >> (4 * b + 8)) & 15u;
    unsigned aa = 26;                                   // X
    if (a < 4 && c < 4 && g < 4) aa = s_aa[16 * a + 4 * c + g];
    out |= (unsigned long long)aa << (8 * b);
  }
  *reinterpret_cast<unsigned long long *>(cls + t * 8) = out;
}

// One tile of 2048 block positions per thread block, 8 consecutive positions per thread.  The ORF that ends before position p starts
// behind the previous stop codon of p's frame: instead of every closing position walking back over the class bytes (21 dependent
// loads on average), each thread notes the last stop of each frame among its own positions, a block-wide max-scan hands every thread
// the last stop of each frame in front of it, and only the first ORF of each frame in a tile (whose stop lies in an earlier tile) walks.
template <bool EMIT>
__global__ void __launch_bounds__(kOrfTileThreads) orf_scan_kernel(OrfScanArgs a)
{
  __shared__ int s_warp[kOrfTileThreads / 32];
  __shared__ int s_last[3][kOrfTileThreads / 32];
  const int tile = blockIdx.x;
  const int b = a.tile_block[tile];
  const BlockDesc bd = a.blocks[b];
  const int p0 = a.tile_p0[tile] + threadIdx.x * kOrfPosPerThread;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const uint8_t *__restrict__ cls = a.cls + bd.goff - 1;          // cls[p] = class of the codon starting at block position p

  // is there a stop codon at block position p (whole codons only)?
  bool stop[kOrfPosPerThread];
  int  mine[3] = { -1, -1, -1 };                                   // last stop of each frame (p mod 3) among this thread's positions
#pragma unroll
  for (int z = 0; z < kOrfPosPerThread; ++z) {
    const int p = p0 + z;
    stop[z] = (p >= 1 && p + 2 <= bd.n) && (__ldg(cls + p) == kStopCode);
    if (stop[z]) mine[p % 3] = p;
  }
  // exclusive max-scan over the block, per frame
  int prev[3];
#pragma unroll
  for (int f = 0; f < 3; ++f) {
    int incl = mine[f];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl = max(incl, v); }
    if (lane == 31) s_last[f][wid] = incl;
    int excl = __shfl_up_sync(0xffffffffu, incl, 1);
    prev[f] = (lane == 0) ? -1 : excl;
  }
  __syncthreads();
#pragma unroll
  for (int f = 0; f < 3; ++f)
    for (int w = 0; w < wid; ++w) prev[f] = max(prev[f], s_last[f][w]);

  int lens[kOrfPosPerThread];
  int cnt = 0;
#pragma unroll
  for (int z = 0; z < kOrfPosPerThread; ++z) {
    const int p = p0 + z;
    int len = 0;
    if (p >= 1 && p <= bd.n + 1) {
      const bool ends = (p + 2 <= bd.n) ? stop[z] : true;          // the three positions without a whole codon close one frame each
      if (ends) {
        const int f = p % 3;
        if (prev[f] >= 0) len = (p - prev[f]) / 3 - 1;             // the stop is in this tile
        else {                                                     // it lies in an earlier tile (or the frame has none yet): walk
          const int t0 = a.tile_p0[tile];
          int q = p - 3;
          for (; q >= t0; q -= 3) ++len;                           // no stop of this frame in the tile before p
          for (; q >= 1 && __ldg(cls + q) != kStopCode; q -= 3) ++len;
        }
        if (len < a.min_len) len = 0;
      }
      if (stop[z]) prev[p % 3] = p;
    }
    lens[z] = len;
    cnt += len > 0;
  }
  // block-wide exclusive scan of cnt
  int incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
  if (lane == 31) s_warp[wid] = incl;
  __syncthreads();
  int wbase = 0, total = 0;
#pragma unroll
  for (int w = 0; w < kOrfTileThreads / 32; ++w) { if (w < wid) wbase += s_warp[w]; total += s_warp[w]; }
  if constexpr (!EMIT) {
    if (threadIdx.x == 0) a.tile_cnt[tile] = total;
  } else {
    long long r = a.tile_base[tile] + wbase + incl - cnt;
    unsigned scored = 0;
#pragma unroll
    for (int z = 0; z < kOrfPosPerThread; ++z) {
      if (lens[z] == 0) continue;
      const int p = p0 + z, len = lens[z];
      const int start = p - 3 * len, end = p - 1;
      const bool in_context = a.complement ? ((bd.n - start + 1) < bd.C) : (end < bd.C);     // (src/p7_pipeline.c:1634-1637)
      if (!in_context) scored += (unsigned)len;
      OrfDesc d;
      d.offset = bd.goff + start - 1;                   // index of the first codon in cls; residues follow with stride 3
      d.L = len; d.tjb_b = a.tjb_of[min(len, a.max_len)]; d.ssv_thresh = 0; d.xw_move = 0; d.vit_thresh = 0;
      d.flags = in_context ? 2 : 0; d.ext_thresh = 0;
      a.descs[r] = d;
      OrfMeta m;
      m.block = b; m.index = (int)(r - a.block_first[b]); m.start = start; m.end = end; m.frame = (start - 1) % 3;
      a.meta[r] = m;
      ++r;
    }
    scored = __reduce_add_sync(0xffffffffu, scored);
    if (lane == 0 && scored) atomicAdd(a.scored, (unsigned long long)scored);
  }
}

struct ScreenSetJob { long long item0, desc0; double min_bits; };    // one job of bathgpu_orfs_msv_screen_set, in item order

struct OrfScreenArgs {
  const uint8_t  *cls;
  const OrfDesc  *descs;
  const OrfMeta  *meta;
  const float    *usc;
  const int      *status;
  long long       norf;
  const float    *null_of;      // [max_len + 1] null1 score of an ORF of that length (p7_bg_NullOne)
  int             max_len;
  double          min_bits;     // keep when (usc - null) / ln 2 >= min_bits
  OrfHit         *hits;
  uint8_t        *residues;     // unit stride, survivors only
  unsigned long long *counters; // [0] hits, [1] residues
  // orf_screen_kernel<true> (bathgpu_orfs_msv_screen_set): item r is ORF r - item0 of job j's layout, whose descriptors start at
  // desc0; survivors past max_hits / max_res are counted, not written (the caller grows the buffers and runs the kernel again)
  const ScreenSetJob *jobs;
  int             njobs;
  int            *hit_job;      // [max_hits] job of each survivor
  unsigned long long *job_counters;   // [2 njobs] survivors and residues per job
  unsigned long long max_hits, max_res;
};

template <bool SET>
__global__ void __launch_bounds__(256) orf_screen_kernel(OrfScreenArgs a)
{
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= a.norf) return;
  long long di = r;
  int job = 0;
  double min_bits = a.min_bits;
  if constexpr (SET) {
    int lo = 0, hi = a.njobs - 1;                         // last job whose first item is <= r
    while (lo < hi) { const int mid = (lo + hi + 1) / 2; if (a.jobs[mid].item0 <= r) lo = mid; else hi = mid - 1; }
    job = lo;
    di = a.jobs[job].desc0 + (r - a.jobs[job].item0);
    min_bits = a.jobs[job].min_bits;
  }
  const OrfDesc d = a.descs[di];
  if (d.flags & 2) return;
  const int st = a.status[r];
  const float usc = a.usc[r];
  if (st == 0) {
    const double bits = ((double)usc - (double)a.null_of[min(d.L, a.max_len)]) / 0.69314718055994529;
    if (!(bits >= min_bits)) return;
  }
  const unsigned long long slot = atomicAdd(&a.counters[0], 1ull);
  const unsigned long long off  = atomicAdd(&a.counters[1], (unsigned long long)d.L);
  if constexpr (SET) {
    atomicAdd(&a.job_counters[2 * job], 1ull);
    atomicAdd(&a.job_counters[2 * job + 1], (unsigned long long)d.L);
    if (slot >= a.max_hits || off + d.L > a.max_res) return;
    a.hit_job[slot] = job;
  }
  const OrfMeta m = a.meta[di];
  OrfHit h;
  h.block = m.block; h.index = m.index; h.start = m.start; h.end = m.end; h.n = d.L; h.frame = m.frame;
  h.offset = (long long)off; h.usc = usc; h.status = st;
  a.hits[slot] = h;
  const uint8_t *src = a.cls + d.offset;
  uint8_t *dst = a.residues + off;
  for (int j = 0; j < d.L; ++j) dst[j] = src[3 * (size_t)j];
}

}  // namespace bathgpu
