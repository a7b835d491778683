/* bathgpu.h -- C ABI of libbathgpu.so: the B200 (sm_100a) engine for the
 * translated-search hot path of BATH's bathsearch.
 *
 * The reference has no FFI today; its replaceable boundary is the "impl" layer
 * (src/hmmer.h:1044-1052 includes one of impl_{sse,avx,neon}.h; impl_avx already
 * exposes every kernel as a patchable function pointer, src/impl_avx/fwdback_fs.c:21-22).
 * One-window-at-a-time calls cannot feed a GPU, so each entry point below is the
 * BATCHED form of one impl-layer function; the per-item semantics (inputs, outputs,
 * Easel status codes) are those of the function it replaces:
 *
 *   bathgpu_load_fs_profile   <- p7_fs_oprofile_Convert      src/impl_sse/p7_fs_oprofile.c:222-296
 *   bathgpu_upload_block      <- ESL_SQ block handed to p7_Pipeline_BATH  src/bathsearch.c:1261,1272
 *   bathgpu_fs_fwd_windows    <- p7_ForwardParser_Frameshift_3Codons      src/impl_sse/impl_sse.h:493
 *                                (call site src/p7_pipeline.c:1446-1450)
 *   bathgpu_fs_bck_decode     <- p7_BackwardParser_Frameshift_3Codons + p7_DomainDecoding_Frameshift
 *                                src/impl_sse/impl_sse.h:494,484 (call sites src/p7_pipeline.c:1470, src/p7_domaindef.c:320)
 *   bathgpu_fs_domains        <- p7_Forward_Frameshift, p7_Backward_Frameshift, p7_Decoding_Frameshift,
 *                                p7_OptimalAccuracy_Frameshift, p7_OATrace_Frameshift, p7_Null2_fs_ByExpectation
 *                                src/impl_sse/impl_sse.h:497-498,483,523-524,516 (call sites src/p7_domaindef.c:1022-1082)
 *   bathgpu_fs_forward_matrices <- p7_Forward_Frameshift with the matrix kept for p7_StochasticTrace_Frameshift
 *                                (call site src/p7_domaindef.c:411-414; the sampling and clustering stay host code)
 *
 * Plain pointers and sizes only.  All functions return an Easel-style status
 * (0 = eslOK); per-item status[] carries eslERANGE (16) exactly where the reference
 * function would have returned it.  There is no CPU fallback: every call fails with
 * BATHGPU_ENODEVICE if no CUDA device is usable.
 */
#ifndef BATHGPU_H
#define BATHGPU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BATHGPU_OK         0
#define BATHGPU_EMEM       5    /* eslEMEM   */
#define BATHGPU_EINVAL     11   /* eslEINVAL */
#define BATHGPU_ERANGE     16   /* eslERANGE */
#define BATHGPU_ENODEVICE  100
#define BATHGPU_ECUDA      101

#define BATHGPU_NXCELLS    6    /* E,N,J,B,C,SCALE  (impl_sse.h:324) */
#define BATHGPU_KP         29

typedef struct bathgpu_ctx bathgpu_ctx;

/* One DNA window of the uploaded block: nucleotides block[start .. start+L-1]
 * (1-based block coordinates, as dna_window->n / ->length in src/p7_pipeline.c:1376-1380).
 * pmove/ploop are the N/C/J odds p7_fs_oprofile_ReconfigLength(om_fs3, L/3) would set
 * (src/impl_sse/p7_fs_oprofile.c:636-651); the caller computes them so the length model
 * stays host-owned. */
typedef struct {
  int64_t start;
  int32_t L;
  float   pmove;
  float   ploop;
} bathgpu_window;

/* One trace step of an optimal-accuracy alignment (P7_TRACE st/k/i/c/pp; src/hmmer.h P7_TRACE). */
typedef struct {
  int32_t i;
  int16_t k;
  uint8_t st;
  uint8_t c;
  float   pp;
} bathgpu_trace_step;

/* One envelope to rescore: nucleotides block[start .. start+L-1]; pmove/ploop from
 * p7_fs_oprofile_ReconfigLength(om_fs5, L/3) in unihit mode (src/p7_domaindef.c:1018). */
typedef struct {
  int64_t start;
  int32_t L;
  float   pmove;
  float   ploop;
} bathgpu_envelope;

/* Per-envelope results of the domain stage (what rescore_isolated_domain_frameshift
 * reads back, src/p7_domaindef.c:1022-1082). */
typedef struct {
  float   envsc;        /* Forward score, nats            */
  float   bcksc;        /* Backward score, nats           */
  float   oasc;         /* optimal-accuracy expected score */
  int32_t status;       /* 0, or eslERANGE from fwd/bck/decoding */
  int32_t trace_offset; /* first step in the trace buffer  */
  int32_t trace_len;
  float   null2[BATHGPU_KP];
} bathgpu_domain_result;

/* ---- context ---------------------------------------------------------- */
int         bathgpu_create(int device, bathgpu_ctx **ret_ctx);
void        bathgpu_destroy(bathgpu_ctx *ctx);
const char *bathgpu_last_error(const bathgpu_ctx *ctx);
int         bathgpu_device_info(const bathgpu_ctx *ctx, int *sm_count, int *clock_khz, size_t *total_mem);

/* Page-locked host buffers for blocks, descriptors and results (so the copies inside the stage calls run at
 * full PCIe/C2C rate).  Any host pointer is accepted by the stage calls; pinned ones are just faster. */
void       *bathgpu_host_alloc(size_t bytes);
void        bathgpu_host_free(void *p);

/* ---- profile images ---------------------------------------------------- */
/* which = 3 or 5 codon lengths.  rfv: [nrows][M+1] emission odds ratios, row c as
 * P7_FS_OPROFILE->rfv[c] un-striped, column 0 unused; tfv: [8][M+1] transition odds,
 * order BM,MM,IM,DM,MD,MI,II,DD, SOURCE-node indexed (tfv[t][k] = exp(TSC(k,t)), 0 at k=M). */
int bathgpu_load_fs_profile(bathgpu_ctx *ctx, int which, int M, int nrows, const float *rfv, const float *tfv);

/* ---- protein (ORF-stage) filter profile: the integer parts of P7_OPROFILE, un-striped ------------------- */
/* Replaces reading om->rbv/rwv/twv in p7_MSVFilter / p7_ViterbiFilter (src/impl_sse/impl_sse.h:75-142).
 * rbv: [29][M+1] uint8 match costs (column 0 unused); rwv: [29][M+1] int16 match scores;
 * twv: [8][M+1] int16 transition scores, order BM,MM,IM,DM,MD,MI,II,DD, SOURCE-node indexed (0 .. M-1; column M = -32768).
 * cpu_lanes_u8 / cpu_lanes_i16: bytes / words per SIMD vector of the CPU build whose window tie-breaks are to be
 * reproduced (16 / 8 for SSE, 32 / 16 for AVX2; src/impl_sse/msvfilter.c:358-366, vitfilter.c:388-396). */
typedef struct {
  int32_t M;
  int32_t tbm_b, tec_b, base_b, bias_b;       /* om->tbm_b, tec_b, base_b, bias_b */
  float   scale_b;
  int32_t base_w, ddbound_w;                  /* om->base_w, ddbound_w            */
  int32_t xw_E_move, xw_E_loop;               /* om->xw[p7O_E][MOVE|LOOP]         */
  float   scale_w;
  int32_t cpu_lanes_u8, cpu_lanes_i16;
} bathgpu_filter_params;

int bathgpu_load_filter_profile(bathgpu_ctx *ctx, const bathgpu_filter_params *prm,
                                const uint8_t *rbv, const int16_t *rwv, const int16_t *twv);

/* One ORF of the uploaded residue buffer, with the per-length pieces of the score system the reference
 * re-derives per ORF on the host (p7_oprofile_ReconfigLength, src/impl_sse/p7_oprofile.c:1261-1326) and the
 * window thresholds (msvfilter.c:313, vitfilter.c:315-321), so that every float->integer rounding stays host-owned. */
typedef struct {
  int64_t offset;       /* index of the ORF's first residue in the residue buffer */
  int32_t L;
  uint8_t tjb_b;        /* unbiased_byteify(logf(3/(L+3)))                          */
  uint8_t ssv_thresh;   /* sc_thresh of p7_SSVFilter_BATH (uint8, as the reference stores it) */
  int16_t xw_move;      /* wordify(logf(pmove)), pmove = (2+nj)/(L+2+nj)            */
  int16_t vit_thresh;   /* sc_thresh of p7_ViterbiFilter_BATH                       */
  int16_t flags;        /* bit 0: emit windows from the Viterbi filter              */
  int32_t ext_thresh;   /* sc_ext_thresh of p7_ViterbiFilter_BATH                   */
} bathgpu_orf;

/* P7_HMM_WINDOW fields the pipeline reads (src/p7_hmmwindow.c:83): target position n, model position k,
 * diagonal length, score; orf = index of the ORF in the call. */
typedef struct { int32_t orf, n, k, length; float score; } bathgpu_orf_window;

/* residues: concatenated amino-acid codes (Easel digital alphabet, 0..28) of all ORFs of a block */
int bathgpu_upload_orfs(bathgpu_ctx *ctx, const uint8_t *residues, int64_t n);

/* a2: p7_MSVFilter over ORFs.  sc[n] nats (+inf with status eslERANGE on overflow, msvfilter.c:176-180). */
int bathgpu_msv_orfs(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, float *sc, int32_t *status);
/* a3: p7_SSVFilter_BATH over ORFs: windows only (sorted by ORF, then target position). */
int bathgpu_ssv_windows(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, bathgpu_orf_window *wins, int max_wins, int *nwins);
/* a4: p7_ViterbiFilter / p7_ViterbiFilter_BATH over ORFs: sc[n], status[n], and windows for ORFs with flags bit 0. */
int bathgpu_vit_orfs(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, float *sc, int32_t *status,
                     bathgpu_orf_window *wins, int max_wins, int *nwins);

/* a6: p7_ForwardParser over ORFs (src/impl_sse/impl_sse.h:488; call site src/p7_pipeline.c:1779): the protein
 * Forward score in nats.  Uses the amino-acid rows and transitions of the loaded 3-codon frameshift profile, which
 * are the protein profile's own (src/modelconfig.c:343-352); nj = expected J uses of the protein profile (1 for the
 * multihit local mode bathsearch configures), xfE = {E->MOVE, E->LOOP} odds. */
int bathgpu_fwd_orfs(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, float nj, const float xfE[2], float *fwdsc, int32_t *status);

/* ---- target block ------------------------------------------------------ */
/* Two resident targets (slot 0 / 1), e.g. the two strands of a sequence: uploads and every stage call act on the
 * selected slot, so the stages of both strands can be batched without re-uploading.  Slot 0 is selected at creation. */
int bathgpu_select_slot(bathgpu_ctx *ctx, int slot);

/* dsq: ESL_DSQ codes, dsq[1..n] valid (dsq[0], dsq[n+1] sentinels).  Packed to 4 bits/nt on device. */
int bathgpu_upload_block(bathgpu_ctx *ctx, const uint8_t *dsq, int64_t n);

/* The same block handed over as nseg pieces that follow one another on the device (seg[g]: the first nucleotide of piece g, seg_n[g]
 * nucleotides; e.g. the sequences of a multi-FASTA target that bathsearch reads one ESL_SQ at a time, src/bathsearch.c:1053-1113,
 * searched as one block): each piece crosses the host link from where it lies,
 * nothing is concatenated on the host.  The resident block has n = sum of seg_n nucleotides and sentinels at both ends. */
int bathgpu_upload_block_segments(bathgpu_ctx *ctx, const uint8_t *const *seg, const int64_t *seg_n, int nseg);

/* Host-packed blocks ("packed 2-bit/4-bit DNA windows" at the boundary): two nucleotides per byte -- dsq[2j+1] in the low nibble of byte j,
 * dsq[2j+2] in the high one, codes above 15 (Easel's '*' and '~') stored as 15 (N), an odd last nibble 15 -- which is the device's own
 * layout, so the block crosses the link at half the bytes and is not packed again.  bathgpu_pack_dna4 makes that form on the host
 * (packed: bathgpu_packed4_bytes(n) = (n+1)/2 bytes); a reader that digitises sequence files can emit it directly. */
int64_t bathgpu_packed4_bytes(int64_t n);
int bathgpu_pack_dna4(const uint8_t *dsq, int64_t n, uint8_t *packed);
int bathgpu_upload_block_packed4(bathgpu_ctx *ctx, const uint8_t *packed, int64_t n);

/* The reverse complement of slot src's resident sequence becomes slot dst's resident sequence (the bottom strand of a target whose
 * top strand was uploaded: bathsearch reverse-complements on the host, src/bathsearch.c:1087-1096, and would upload it again). */
int bathgpu_revcomp_slot(bathgpu_ctx *ctx, int src, int dst);

/* ---- a9: frameshift Forward parser (3 codon lengths) over windows ------- */
/* xfE = {E->MOVE, E->LOOP} odds (om_fs3->xf[p7O_E]).  Outputs: fwdsc[n] nats, status[n]. */
int bathgpu_fs_fwd_windows(bathgpu_ctx *ctx, const bathgpu_window *wins, int n, const float xfE[2],
                           float *fwdsc, int32_t *status);

/* bathgpu_upload_block + bathgpu_fs_fwd_windows in one call with the upload hidden behind the kernel: the block crosses the host
 * link in chunks while the windows that end inside the part already resident are being scored.  Any window order. */
int bathgpu_fs_fwd_block(bathgpu_ctx *ctx, const uint8_t *dsq, int64_t n, const bathgpu_window *wins, int nwin,
                         const float xfE[2], float *fwdsc, int32_t *status);

/* bathgpu_fs_fwd_block on a host-packed block (bathgpu_pack_dna4): same chunks, half the bytes, no packing kernel. */
int bathgpu_fs_fwd_block_packed4(bathgpu_ctx *ctx, const uint8_t *packed, int64_t n, const bathgpu_window *wins, int nwin,
                                 const float xfE[2], float *fwdsc, int32_t *status);

/* Same stage on descriptors already resident in device memory (set by
 * bathgpu_stage_windows); results stay on the device until bathgpu_fetch_scores.
 * Used to time the kernel with inputs resident in HBM. */
int bathgpu_stage_windows(bathgpu_ctx *ctx, const bathgpu_window *wins, int n);
int bathgpu_fs_fwd_staged(bathgpu_ctx *ctx, const float xfE[2]);
int bathgpu_fetch_scores(bathgpu_ctx *ctx, float *fwdsc, int32_t *status, int n);

/* ---- a10+a11: Backward parser + domain decoding ------------------------- */
/* For each window: re-runs the Forward parser keeping X rows, runs the Backward parser,
 * then DomainDecoding.  xf5_loop = {N,J,C}->LOOP odds of the profile the reference passes
 * to p7_DomainDecoding_Frameshift (om_fs5, src/p7_domaindef.c:320).  Outputs are
 * concatenated per window at out_offset[w] .. +L (L+1 floats each); bcksc[n]; status[n]. */
int bathgpu_fs_bck_decode(bathgpu_ctx *ctx, const bathgpu_window *wins, int n, const float xfE[2],
                          const float xf5_loop[3], const int64_t *out_offset,
                          float *mocc, float *btot, float *etot, float *fwdsc, float *bcksc, int32_t *status);

/* a10 without a11: Forward (X rows kept) + Backward parsers over windows.  fwd_xrows / bck_xrows: {E,N,J,B,C,SCALE} x (L+1)
 * per window, windows concatenated in call order (what P7_OMX->xmx holds, impl_sse.h:324), for a caller that runs
 * p7_DomainDecoding_Frameshift itself. */
int bathgpu_fs_fwd_bck_xrows(bathgpu_ctx *ctx, const bathgpu_window *wins, int n, const float xfE[2],
                             float *fwd_xrows, float *bck_xrows, float *fwdsc, float *bcksc, int32_t *status);

/* X rows {E,N,J,B,C,SCALE} x (L+1) per window, windows concatenated in call order, of the Forward (which = 0)
 * or Backward (which = 1) parser as left on the device by the last bathgpu_fs_bck_decode call (its last chunk):
 * what P7_OMX->xmx holds after p7_ForwardParser/BackwardParser_Frameshift_3Codons (impl_sse.h:324). */
int bathgpu_fs_fetch_xrows(bathgpu_ctx *ctx, int which, float *out, int64_t nrows);

/* ---- a12-a15: per-envelope Forward/Backward/Decoding/OA/trace/null2 ------ */
/* xfE5 = {E->MOVE, E->LOOP} odds of om_fs5 (unihit: {1,0}).  traces: caller-allocated buffer
 * of max_steps steps; results[e].trace_offset/len index into it. */
int bathgpu_fs_domains(bathgpu_ctx *ctx, const bathgpu_envelope *envs, int n, const float xfE5[2],
                       bathgpu_domain_result *results, bathgpu_trace_step *traces, int64_t max_steps);

/* ---- a16 (device part): the Forward matrix p7_StochasticTrace_Frameshift samples from ------ */
/* p7_Forward_Frameshift (src/impl_sse/impl_sse.h:497) over regions of the resident block, full matrix handed back as the
 * call at src/p7_domaindef.c:411-414 leaves it in pli->fwd_fs, un-striped: region r occupies rows off .. off + L of
 *   mx    [rows][(M+1)][8]  {D, I, M_C0, M_C1 .. M_C5} (impl_sse.h:296-314), node 0 all zero
 *   xrows [rows][6]         {E, N, J, B, C, SCALE}
 * with off = sum over earlier regions of (L+1); max_rows = rows the caller allocated.  xfE5 = {E->MOVE, E->LOOP} odds
 * (multihit: {0.5, 0.5}); the length model of each region is in its descriptor.  status[r] = eslERANGE as the reference.
 * mx = xrows = NULL: scores only -- what p7_ForwardParser_Frameshift_5Codons returns (src/impl_sse/impl_sse.h:495; its one
 * caller is the calibration p7_fs_Tau_5codons, src/evalues.c:759); max_rows is then ignored. */
int bathgpu_fs_forward_matrices(bathgpu_ctx *ctx, const bathgpu_envelope *regs, int n, const float xfE5[2],
                                float *mx, float *xrows, int64_t max_rows, float *fwdsc, int32_t *status);

/* ---- the frameshift Forward parsers over a resident profile set (calibration of many models at once) ------------------ */
/* The calibration runs p7_fs_Tau_3codons / p7_fs_Tau_5codons once per model (src/evalues.c:607-680, :703-776; 200 windows of
 * 300 nt each): a model alone fills a fraction of the device.  These two calls score the windows of MANY profiles in one launch
 * per kernel.
 * bathgpu_load_fs_profile_set: n profile images of one codon length (which = 3 or 5), profile p in the layout
 * bathgpu_load_fs_profile takes (M[p], nrows[p], rfv[p], tfv[p]).  Held beside the context's single loaded profile, which stays
 * untouched; loading a new set of the same codon length replaces the old one. */
int bathgpu_load_fs_profile_set(bathgpu_ctx *ctx, int which, int n, const int *M, const int *nrows,
                                const float *const *rfv, const float *const *tfv);

/* A window of the selected slot's block (as bathgpu_window) scored with profile `profile` of the set. */
typedef struct {
  int64_t start;
  int32_t L;
  float   pmove;
  float   ploop;
  int32_t profile;
} bathgpu_set_window;

/* xfE[2 p], xfE[2 p + 1] = {E->MOVE, E->LOOP} odds of profile p.  which = 3: fwdsc[w] is what bathgpu_fs_fwd_windows returns for
 * the window with that profile loaded alone (p7_ForwardParser_Frameshift_3Codons, call site src/evalues.c:649); which = 5: what
 * bathgpu_fs_forward_matrices returns in its scores-only mode (p7_ForwardParser_Frameshift_5Codons, :759).  Bit-identical to those
 * calls, status[w] = eslERANGE where they set it.  Windows of any mix of profiles and lengths, in any order. */
int bathgpu_fs_set_scores(bathgpu_ctx *ctx, int which, const bathgpu_set_window *wins, int n, const float *xfE,
                          float *fwdsc, int32_t *status);

/* Test/diagnostic: matrices of envelope e of the last chunk of the last bathgpu_fs_domains call, in the
 * reference's cell order: pp [(L+1)][(M+1)][8] {D,I,M_C0..M_C5} (impl_sse.h:296-314; D cells are 0 after
 * decoding), oa [(L+1)][(M+1)][3] {M,D,I}, ppx / oax [(L+1)][6] {E,N,J,B,C,SCALE}.  Any pointer may be NULL. */
int bathgpu_fs_fetch_domain_matrices(bathgpu_ctx *ctx, int e, float *pp, float *oa, float *ppx, float *oax);

/* ---- f1: six-frame translation, MSV and the F1 screen on the device -------------------------------------------- */
/* One block of the resident strand: block position p (1..n) is position goff + p of the uploaded sequence; C = nucleotides of
 * overlap context (dnasq->C): ORFs wholly inside it are not scored (src/p7_pipeline.c:1634-1637). */
typedef struct { int64_t goff; int32_t n; int32_t C; } bathgpu_block;
/* An ORF that survived the screen: block and rank inside the block (the reference's ORF order: by last nucleotide), block-local
 * nucleotide coordinates of its first and last nucleotide, residues, frame (0..2), offset of its residues in the device residue
 * buffer (what bathgpu_orf.offset of the later stage calls refers to), MSV score (nats) and status. */
typedef struct { int32_t block, index, start, end, n, frame; int64_t offset; float usc; int32_t status; } bathgpu_orf_hit;

/* Replaces, for a GPU build, the translation of each block (esl_gencode_Process*, src/bathsearch.c:385-392), the upload of ORF
 * residues and the head of the per-ORF loop (p7_MSVFilter and the cheap side of the F1 test, src/p7_pipeline.c:1632-1652) for ALL
 * blocks of the selected slot's sequence in one call.  complement: the uploaded sequence is the reverse complement (decides which
 * end the overlap context is at).  gcode[64]: amino-acid code (27 = stop) of codon 16 a + 4 b + c.  tjb_of[L], null_of[L] for
 * L = 0..max_len (longer ORFs use max_len): unbiased_byteify(logf(3/(L+3))) and p7_bg_NullOne for that length.  An ORF survives
 * when its MSV score overflowed or (usc - null_of[L]) / ln 2 >= min_bits; the caller then applies its exact P-value test.
 * Outputs: ORFs found per block, survivors and their residues (left in the device residue buffer; copy them out with
 * bathgpu_orfs_fetch, which returns them sorted by block and rank). */
int bathgpu_orfs_msv_screen(bathgpu_ctx *ctx, const bathgpu_block *blocks, int nblocks, int complement, const uint8_t gcode[64],
                            int min_len, const uint8_t *tjb_of, const float *null_of, int max_len, double min_bits,
                            int64_t *norfs_per_block, int64_t *nhits, int64_t *nres);
int bathgpu_orfs_fetch(bathgpu_ctx *ctx, bathgpu_orf_hit *hits, uint8_t *residues);
/* Measurement aid: CUDA-event time of the kernel groups of the last bathgpu_orfs_msv_screen call -- ms[0] codon classes, [1] ORF count
 * pass, [2] ORF emit pass, [3] MSV over every ORF, [4] F1 screen + residue gather -- with the number of ORFs found and the residues the
 * MSV kernel scored (its DP cells = residues x M). */
int bathgpu_orfs_stage_breakdown(bathgpu_ctx *ctx, float ms[5], int64_t *norfs, int64_t *residues_scored);

/* ---- a5: the bias-composition filter ---------------------------------------------------------------------------------- */
/* esl_hmm_Forward over the 2-state filter HMM of p7_bg_SetFilter (src/p7_bg.c:449-471), batched: what p7_bg_FilterScore computes
 * for an ORF (:491-500; call sites src/p7_pipeline.c:1659, :1697) and p7_bg_fs_FilterScore for each of the three reading frames of a
 * DNA window (:522-573, canonical residues only; call sites src/p7_pipeline.c:1432, :1437).
 *   kind 0: item = ORF of the selected slot's residue buffer (start = offset of its first residue); out[n]
 *   kind 1: item = DNA window of the selected slot (start = 1-based coordinate of its first nucleotide); out[3 n], frames 1..3
 * tables: [ntab][29][2] emission odds e[state][x] / f[x] as esl_hmm_Configure leaves them (table 0 = the model composition, others
 * the local compositions of p7_pli_ComputeLocalCompo); item.table picks one.  t00 = p1 of the null model at the item's length
 * (p7_bg_SetLength copies it into the filter HMM), t10/t11 = 1/(L1+1), L1/(L1+1) with L1 = M/8; state priors 0.999 / 0.001.
 * out = the summed log scale factors (esl_hmm_Forward's score); the caller adds the length terms and combines the frames as the
 * reference does.  Bit-identical to the host code for the same inputs (same operations in the same order, no fused multiply-adds). */
typedef struct { int64_t start; int32_t L; int32_t table; float t00; int32_t pad_; } bathgpu_bias_item;
int bathgpu_bias_forward(bathgpu_ctx *ctx, int kind, const bathgpu_bias_item *items, int n, const float *tables, int ntab,
                         float t10, float t11, const uint8_t gcode[64], float *out);

/* ---- f2: the standard-translation branch over ORFs ------------------------ */
/* p7_ForwardParser + p7_BackwardParser over ORFs of the uploaded residue buffer, X rows kept (what oxf_holder[i] and
 * pli->oxb hold at src/p7_pipeline.c:1492-1495 / :1762-1764): fwd_xrows / bck_xrows = {E,N,J,B,C,SCALE} x (L+1) per ORF,
 * ORFs concatenated in call order, for a caller that runs p7_DomainDecoding (an O(L) scalar pass) itself.  The length
 * model is p7_oprofile_ReconfigLength(om, L) with nj; xfE = {E->MOVE, E->LOOP} odds (multihit: {0.5, 0.5}).
 * Uses the amino-acid rows and transitions of the loaded frameshift profile, which are the protein profile's own. */
int bathgpu_orf_fwd_bck_xrows(bathgpu_ctx *ctx, const bathgpu_orf *orfs, int n, float nj, const float xfE[2],
                              float *fwd_xrows, float *bck_xrows, float *fwdsc, float *bcksc, int32_t *status);

/* rescore_isolated_domain_bath (src/p7_domaindef.c:1229-1370) over envelopes of ORFs: p7_Forward, p7_Backward, p7_Decoding,
 * p7_OptimalAccuracy, p7_OATrace and p7_Null2_ByExpectation (src/impl_sse/impl_sse.h:479-520).  envs[e].start is the 0-based
 * offset of the envelope's first residue in the uploaded residue buffer (like bathgpu_orf.offset), L its length in residues,
 * pmove/ploop from p7_oprofile_ReconfigLength(om, L) in unihit mode; xfE = {1, 0} there.  Trace steps carry i in envelope
 * coordinates (1..L) and c = 0; the caller maps them to nucleotides as p7_trace_fs_Convert does (src/p7_trace.c:405). */
int bathgpu_orf_domains(bathgpu_ctx *ctx, const bathgpu_envelope *envs, int n, const float xfE[2],
                        bathgpu_domain_result *results, bathgpu_trace_step *traces, int64_t max_steps);
/* p7_Forward over regions of ORFs with the whole matrix handed back, for the multi-domain branch of the standard-translation domain
 * definition: replaces p7_Forward(orfsq->dsq+i-1, j-i+1, om, fwd, NULL) at src/p7_domaindef.c:562 for all flagged regions of a batch
 * at once (om in multihit mode at the ORF's length: pmove / ploop of the descriptor, xfE = {0.5, 0.5}).  regs[r].start = 0-based
 * offset of the region's first residue in the slot's residue buffer.  mx: [(L+1)][(M+1)][4] = {M, D, I, 0} per region (what P7_OMX
 * dpf holds, un-striped), xrows: [(L+1)][6]; regions concatenated; max_rows = capacity of both in rows. */
int bathgpu_orf_forward_matrices(bathgpu_ctx *ctx, const bathgpu_envelope *regs, int n, const float xfE[2],
                                 float *mx, float *xrows, int64_t max_rows, float *fwdsc, int32_t *status);

/* Test/diagnostic: matrices of envelope e of the last chunk of the last bathgpu_orf_domains call, cell order {M,D,I}:
 * pp and oa [(L+1)][(M+1)][3], ppx / oax [(L+1)][6].  Any pointer may be NULL. */
int bathgpu_orf_fetch_domain_matrices(bathgpu_ctx *ctx, int e, float *pp, float *oa, float *ppx, float *oax);

/* ---- measurement helpers ------------------------------------------------ */
/* Device time (ms) of the kernels launched by the most recent stage call, measured with
 * CUDA events on the context's stream, and how many kernels that call launched. */
int bathgpu_last_stage_timing(const bathgpu_ctx *ctx, float *ms, int *launches);

/* FP32 FMA throughput of the device (TFLOP/s, best of several launches of a register-only FFMA kernel):
 * the roofline denominator for the frameshift Forward/Backward kernels, which are FP32-pipe bound. */
int bathgpu_measure_fp32_peak(bathgpu_ctx *ctx, double *tflops, double *sm_mhz_effective);
/* The same for the integer filters: 16-bit lane operations per second (saturating add and max on the two halves of a register, each
 * counted), 16 independent chains per thread. */
int bathgpu_measure_int16_peak(bathgpu_ctx *ctx, double *tera_ops);

#ifdef __cplusplus
}
#endif
#endif
