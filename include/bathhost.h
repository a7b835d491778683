/* bathhost.h -- C ABI of libbathhost.so: the HOST side of the translated-search path.
 *
 * In a GPU build of bathsearch these jobs stay in the reference's own C code (it has Easel);
 * this library restates them in C++ so that the path can be driven and measured end to end
 * without Easel: profile file reading, null model, frameshift profile construction and its
 * odds-ratio form, the length models, and (pipeline.cpp) the stage-batched translated pipeline.
 * Everything here runs once per query or per hit; the DP runs in libbathgpu.so (bathgpu.h).
 *
 *   bathhost_model_read       <- p7_hmmfile_Read (BATH3/f ASCII)              src/p7_hmmfile.c:1374-1690
 *                                + p7_bg_Create                                src/p7_bg.c:52-82
 *                                + p7_ProfileConfig_fs (3 and 5 codon lengths) src/modelconfig.c:220-698
 *                                + p7_fs_oprofile_Convert                      src/impl_sse/p7_fs_oprofile.c:222-296
 *                                as bathsearch sets a query up                 src/bathsearch.c:794-801
 *   bathhost_length_model     <- p7_fs_oprofile_ReconfigLength                 src/impl_sse/p7_fs_oprofile.c:636-651
 *   bathhost_calibrate        <- p7_Calibrate / bathconvert's frameshift taus  src/evalues.c:64-183; src/bathconvert.c:128-161
 *   bathhost_convert          <- bathconvert over a HMMER3/f library           src/bathconvert.c:128-161 per model
 */
#ifndef BATHHOST_H
#define BATHHOST_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BATHHOST_OK       0
#define BATHHOST_EFAIL    1
#define BATHHOST_EOF      3
#define BATHHOST_EMEM     5
#define BATHHOST_EFORMAT  7
#define BATHHOST_EINVAL  11

typedef struct bathhost_model bathhost_model;

/* evparam order: MMU, MLAMBDA, VMU, VLAMBDA, FTAU, FLAMBDA, FTAUFS3, FTAUFS5 (src/hmmer.h:67) */
typedef struct {
  int32_t M;
  int32_t max_length;     /* MAXL, amino units; -1 if absent */
  int32_t codon_table;    /* CODON TABLE; -1 if absent */
  float   fsprob;         /* FRAMESHIFT PROB; -1 if absent */
  float   evparam[8];
  int32_t has_fs3_stats, has_fs5_stats;
  char    name[128];
  char    acc[64];
} bathhost_model_info;

/* Reads the index-th model of a .bhmm file and configures it the way bathsearch does for a
 * query (p7_LOCAL, dummy L=100).  ct <= 0: use the file's CODON TABLE (1 if absent). */
int  bathhost_model_read(const char *path, int index, int ct, bathhost_model **ret_model);
int  bathhost_model_count(const char *path);
void bathhost_model_destroy(bathhost_model *m);
int  bathhost_model_get_info(const bathhost_model *m, bathhost_model_info *info);

/* p7_Builder_MaxLength(hmm, 1e-7) recomputed from the core model (what bathsearch uses when the file has no MAXL line,
 * src/bathsearch.c:761-762; bathhost_model_read already applies it) */
int  bathhost_model_computed_max_length(const bathhost_model *m);

/* Un-striped odds-ratio tables in the layout bathgpu_load_fs_profile takes.
 * which = 3 | 5.  rfv: [nrows][M+1], tfv: [8][M+1] (BM,MM,IM,DM,MD,MI,II,DD; source-node indexed). */
int          bathhost_model_nrows(const bathhost_model *m, int which);
const float *bathhost_model_rfv(const bathhost_model *m, int which);
const float *bathhost_model_tfv(const bathhost_model *m, int which);
/* best amino acid / indel pattern per (node, codon row): P7_FS_PROFILE codons[][] / indel_pos[][]
 * (src/hmmer.h:372-411), [(M+1)][maxcodons] */
const uint8_t *bathhost_model_codons(const bathhost_model *m, int which);
const uint8_t *bathhost_model_indel_pos(const bathhost_model *m, int which);
/* core-model match emission probabilities [(M+1)][20] (row 0 unused) and consensus [M+2] */
const float *bathhost_model_mat(const bathhost_model *m);
const char  *bathhost_model_consensus(const bathhost_model *m);

/* Integer filter score systems of the protein profile (P7_OPROFILE, src/impl_sse/p7_oprofile.c:773-921), in the
 * layout bathgpu_load_filter_profile takes: rbv [29][M+1] uint8, rwv [29][M+1] int16, twv [8][M+1] int16. */
typedef struct {
  int32_t M, tbm_b, tec_b, base_b, bias_b;
  float   scale_b;
  int32_t base_w, ddbound_w, xw_E_move, xw_E_loop;
  float   scale_w;
} bathhost_filter_params;
int            bathhost_model_filter_params(const bathhost_model *m, bathhost_filter_params *p);
const uint8_t *bathhost_model_rbv(const bathhost_model *m);
const int16_t *bathhost_model_rwv(const bathhost_model *m);
const int16_t *bathhost_model_twv(const bathhost_model *m);
/* per-ORF-length integers: tjb_b = unbiased_byteify(logf(3/(L+3))), xw_move = wordify(logf((2+nj)/(L+2+nj)))
 * (p7_oprofile_ReconfigLength, src/impl_sse/p7_oprofile.c:1261-1326) */
void           bathhost_orf_length_params(const bathhost_model *m, int L, uint8_t *tjb_b, int16_t *xw_move);

/* N/C/J move and loop odds for a target of L_amino residues with nj expected J uses
 * (multihit local: nj = 1; unihit: nj = 0), in float as the reference computes them. */
void bathhost_length_model(int L_amino, float nj, float *pmove, float *ploop);

/* ---- the stage-batched translated search (pipeline.cpp) -------------------------------------------------
 * Restates p7_Pipeline_BATH + p7_pli_Frameshift + frameshift domain definition + hit post-processing
 * (src/p7_pipeline.c:1583-1821, :1339-1522, :1005-1144; src/p7_domaindef.c:301-473, :993-1191;
 * src/p7_tophits.c:789-960) around batched calls into the device library.  The device library is handed in as a
 * table of function pointers with the signatures of include/bathgpu.h, so this library has no link-time dependency
 * on CUDA. */

typedef struct {
  void *ctx;                                      /* bathgpu_ctx* */
  const char *(*last_error)(const void *ctx);
  int (*load_fs_profile)(void *ctx, int which, int M, int nrows, const float *rfv, const float *tfv);
  int (*load_filter_profile)(void *ctx, const void *prm, const uint8_t *rbv, const int16_t *rwv, const int16_t *twv);
  int (*select_slot)(void *ctx, int slot);
  int (*upload_block)(void *ctx, const uint8_t *dsq, int64_t n);
  int (*upload_orfs)(void *ctx, const uint8_t *residues, int64_t n);
  int (*msv_orfs)(void *ctx, const void *orfs, int n, float *sc, int32_t *status);
  int (*ssv_windows)(void *ctx, const void *orfs, int n, void *wins, int max_wins, int *nwins);
  int (*vit_orfs)(void *ctx, const void *orfs, int n, float *sc, int32_t *status, void *wins, int max_wins, int *nwins);
  int (*fwd_orfs)(void *ctx, const void *orfs, int n, float nj, const float xfE[2], float *fwdsc, int32_t *status);
  int (*fs_fwd_windows)(void *ctx, const void *wins, int n, const float xfE[2], float *fwdsc, int32_t *status);
  int (*fs_fwd_bck_xrows)(void *ctx, const void *wins, int n, const float xfE[2], float *fwd_xrows, float *bck_xrows,
                          float *fwdsc, float *bcksc, int32_t *status);
  int (*fs_bck_decode)(void *ctx, const void *wins, int n, const float xfE[2], const float xf5_loop[3], const int64_t *out_offset,
                       float *mocc, float *btot, float *etot, float *fwdsc, float *bcksc, int32_t *status);
  int (*fs_domains)(void *ctx, const void *envs, int n, const float xfE5[2], void *results, void *traces, int64_t max_steps);
  int (*fs_forward_matrices)(void *ctx, const void *regs, int n, const float xfE5[2], float *mx, float *xrows, int64_t max_rows,
                             float *fwdsc, int32_t *status);
  int (*orf_fwd_bck_xrows)(void *ctx, const void *orfs, int n, float nj, const float xfE[2], float *fwd_xrows, float *bck_xrows,
                           float *fwdsc, float *bcksc, int32_t *status);
  int (*orf_domains)(void *ctx, const void *envs, int n, const float xfE[2], void *results, void *traces, int64_t max_steps);
  int (*orfs_msv_screen)(void *ctx, const void *blocks, int nblocks, int complement, const uint8_t gcode[64], int min_len,
                         const uint8_t *tjb_of, const float *null_of, int max_len, double min_bits,
                         int64_t *norfs_per_block, int64_t *nhits, int64_t *nres);
  int (*orfs_fetch)(void *ctx, void *hits, uint8_t *residues);
  int (*revcomp_slot)(void *ctx, int src, int dst);
  void *(*host_alloc)(size_t bytes);          /* optional (may be NULL): page-locked host memory for result buffers */
  void (*host_free)(void *p);
  /* optional (may be NULL: the host library then runs the same recursion on the host cores): bathgpu_bias_forward */
  int (*bias_forward)(void *ctx, int kind, const void *items, int n, const float *tables, int ntab, float t10, float t11,
                      const uint8_t gcode[64], float *out);
  /* optional (may be NULL: multi-domain regions of the standard branch are then rescored as one envelope and counted in
   * stats.n_multidomain_regions only): bathgpu_orf_forward_matrices */
  int (*orf_forward_matrices)(void *ctx, const void *regs, int n, const float xfE[2], float *mx, float *xrows, int64_t max_rows,
                              float *fwdsc, int32_t *status);
  /* optional (may be NULL: a chunk made of several sequences is then concatenated in a host buffer first and goes through
   * upload_block): bathgpu_upload_block_segments */
  int (*upload_block_segments)(void *ctx, const uint8_t *const *seg, const int64_t *seg_n, int nseg);
  /* optional pair (both NULL: bathhost_convert calibrates model by model through bathhost_calibrate):
   * bathgpu_load_fs_profile_set and bathgpu_fs_set_scores, the frameshift Forward parsers over many profiles at once */
  int (*load_fs_profile_set)(void *ctx, int which, int n, const int *M, const int *nrows, const float *const *rfv, const float *const *tfv);
  int (*fs_set_scores)(void *ctx, int which, const void *wins, int n, const float *xfE, float *fwdsc, int32_t *status);
} bathhost_backend;

/* 0 / unset fields take bathsearch's defaults (src/p7_pipeline.c:145-214; src/bathsearch.c:94) */
typedef struct {
  double  F1, F2, F3, F4, E;
  int32_t min_orf_len;        /* -l, 20 */
  int32_t block_length;       /* 262144 */
  int32_t cpu_lanes_u8, cpu_lanes_i16;   /* stripe geometry of the CPU build to match: 16/8 (SSE) */
  int32_t no_bias, no_null2, top_only, bottom_only;
  int32_t std_only;           /* 0: bathsearch --fs; 1: bathsearch's default pipeline (standard translation only) */
  int32_t show_frameline;     /* --frameline: the report's alignment blocks carry a FRAME line (src/p7_alidisplay.c:3998-4013) */
  int32_t reserved0;
  int64_t chunk_nt;           /* nucleotides per device-resident chunk of the target (0: chosen from the batch size and the number of
                                 device contexts; env BATHHOST_CHUNK_MBP overrides the choice).  Results do not depend on it. */
} bathhost_options;

typedef struct {
  int64_t seqidx;
  char    name[64];
  int32_t strand;             /* +1 top, -1 bottom */
  int64_t ali_from, ali_to, env_from, env_to, sq_len;
  int32_t hmm_from, hmm_to;
  double  evalue, lnP;
  float   score, bias, pre_score, envsc, oasc, pid;     /* score, bias, pre_score in bits, as the tables print them (src/p7_tophits.c:1325) */
  int32_t shifts, stops, trace_len;
  char    cigar[1024];          /* the first 1023 characters; bathhost_search_format_tblout prints the whole string */
} bathhost_hit;

typedef struct {
  int64_t nseqs, nres;                                      /* "Target sequence(s)", "residues searched"      */
  int64_t pos_past_msv, pos_past_bias, pos_past_vit, pos_past_fwd;   /* the footer's filter counters          */
  int64_t n_orfs, n_windows, n_std_windows, n_regions, n_multidomain_regions, n_envelopes, n_hits_reported;
  /* wall time per stage of the host pipeline, microseconds (host work + the device calls made from it) */
  int64_t us_orfs, us_upload, us_msv, us_bias, us_vit, us_fwd, us_windows, us_fs_fwd, us_fs_domains, us_std, us_xrows, us_decode, us_score;
} bathhost_stats;

/* ---- multi-domain regions (stotrace.cpp): p7_StochasticTrace_Frameshift x nsamples reduced to domain end points
 * (src/impl_sse/stotrace_fs.c:72; region_trace_ensemble_frameshift, src/p7_domaindef.c:892-954), then p7_spensemble_fs_Cluster
 * and the removal of dominated clusters (src/p7_spensemble.c:498; src/p7_domaindef.c:923-952).
 * mx / xrows: one region of bathgpu_fs_forward_matrices' output; tfv [8][M+1] odds {BM,MM,IM,DM,MD,MI,II,DD};
 * odds = {N/J/C->MOVE, N/J/C->LOOP, E->MOVE, E->LOOP}; segments come back in window coordinates (ireg = region start). */
typedef struct { int32_t idx, i, j, k, m; float prob; } bathhost_segment;
int bathhost_sample_region_segments(const float *mx, const float *xrows, int M, int L, const float *tfv, const float odds[4],
                                    uint32_t seed, int nsamples, int ireg, bathhost_segment *out, int max_out, int *nout);
int bathhost_cluster_region_segments(const bathhost_segment *sp, int n, int nsamples, bathhost_segment *out, int max_out, int *nout);
/* The standard-translation flavour (region_trace_ensemble, src/p7_domaindef.c:766-860; p7_StochasticTrace, src/impl_sse/stotrace.c;
 * p7_Null2_ByTrace, src/impl_sse/null2.c:131-219; p7_spensemble_Cluster with the protein link rule, src/p7_spensemble.c:191-218).
 * mx: one region of bathgpu_orf_forward_matrices' output [(L+1)][(M+1)][4] {M, D, I, 0}; rf: amino-acid emission odds [29][M+1];
 * res[1..L]: the region's residues; n2sc[0..L] receives the per-residue null2 scores (log of the ensemble mean odds). */
int bathhost_sample_region_segments_protein(const float *mx, const float *xrows, int M, int L, const float *tfv, const float *rf,
                                            const float odds[4], uint32_t seed, int nsamples, int ireg, const uint8_t *res,
                                            bathhost_segment *out, int max_out, int *nout, float *n2sc);
int bathhost_cluster_region_segments_protein(const bathhost_segment *sp, int n, int nsamples, bathhost_segment *out, int max_out, int *nout);

typedef struct bathhost_search bathhost_search;
int  bathhost_search_create(const bathhost_model *m, const bathhost_backend *be, const bathhost_options *opt, bathhost_search **ret);
/* The same search over SEVERAL device contexts (bathgpu_ctx on different GPUs, or more than one per GPU so that one context's host
 * stages run under another's kernels): the target is cut into chunks of consecutive blocks (src/bathsearch.c:1150,1198-1205 deals
 * blocks to worker threads the same way), chunks are dealt round-robin to the contexts, each context is driven by its own host thread,
 * and ONE hit list comes out -- E-values over the summed residue count, duplicates at block borders removed, as the reference merges
 * its workers' lists (src/bathsearch.c:869-921).  Everything the reference computes in block order (hit-window list, length-model
 * chain, early E-value cuts) is computed in that order on the host, so the list is identical whatever the number of contexts. */
int  bathhost_search_create_multi(const bathhost_model *m, const bathhost_backend *be, int nbackends, const bathhost_options *opt,
                                  bathhost_search **ret);
void bathhost_search_destroy(bathhost_search *s);
const char *bathhost_search_last_error(const bathhost_search *s);
/* dsq[1..n] Easel digital nucleotides with sentinels at [0] and [n+1]; both strands unless restricted.
 * bathhost_search_sequence searches one sequence at once.  bathhost_search_queue + bathhost_search_run search a whole set of
 * sequences in one stage-batched pass (larger device batches; the way to feed several GPUs): queued buffers must stay valid and
 * unchanged until bathhost_search_run returns.  Both ways give the same hits. */
int  bathhost_search_sequence(bathhost_search *s, const char *name, const uint8_t *dsq, int64_t n);
int  bathhost_search_queue(bathhost_search *s, const char *name, const uint8_t *dsq, int64_t n);
int  bathhost_search_run(bathhost_search *s);
/* E-values over the whole search space, duplicate removal, ordering, reporting threshold.  Runs anything still queued first;
 * calling it again without new sequences changes nothing. */
int  bathhost_search_finish(bathhost_search *s);
/* bathhost_search_finish of n different searches at once, one host thread each (e.g. the profiles of a query file, src/bathsearch.c:737,
 * each search created over device contexts of its own and fed the same target): the searches share nothing but the host pool, so each
 * returns the hit list it returns alone, and one search's serial host phases run under the others' device stages.  First non-zero
 * status, BATHHOST_EINVAL for a null or repeated search or two searches over the same device context. */
int  bathhost_search_finish_many(bathhost_search *const *searches, int n);
int  bathhost_search_nhits(const bathhost_search *s);
int  bathhost_search_get_hit(const bathhost_search *s, int idx, bathhost_hit *hit);
int  bathhost_search_get_stats(const bathhost_search *s, bathhost_stats *st);
/* The --tblout --cigar table of the reported hits as p7_tophits_TabularTargets writes it (src/p7_tophits.c:1603-1712): header
 * (if show_header) + one line per hit, NUL-terminated, without the trailer.  *needed = bytes required; call with buf = NULL to size. */
int  bathhost_search_format_tblout(const bathhost_search *s, int show_header, char *buf, size_t cap, size_t *needed);
/* The hit-dependent part of the main report, alignments included: "Scores for complete hits:" table (p7_tophits_Targets,
 * src/p7_tophits.c:1073-1227), two blank lines, "Annotation for each hit (and alignments):" with one block per reported hit
 * (p7_tophits_Domains, :1232-1410; alignment display built as p7_alidisplay_fs_Create / p7_alidisplay_nonfs_Create do,
 * src/p7_alidisplay.c:538-931 / :937-1232, and printed as p7_alidisplay_Print_BATH, :3758-4095), two blank lines -- what bathsearch
 * writes between the "Query:" block and "Internal pipeline statistics summary:" (src/bathsearch.c:960-961).  textw = --textw
 * (150 by default, 0 = unlimited).  Same sizing protocol as bathhost_search_format_tblout. */
int  bathhost_search_format_report(const bathhost_search *s, int textw, char *buf, size_t cap, size_t *needed);
/* The --fstblout table (p7_tophits_TabularFrameshifts, src/p7_tophits.c:1442-1600): one line per frameshift ('I' / 'D' and its length)
 * and per in-frame stop codon ('S') of the reported hits of the frameshift branch.  The reference ships no example of this table:
 * restated from the source, checked against the hit's CIGAR string. */
int  bathhost_search_format_fstblout(const bathhost_search *s, int show_header, char *buf, size_t cap, size_t *needed);
/* One query's section of bathsearch's output minus the run-dependent lines (banner, option echo, "# CPU time", "# Mc/sec", "//"):
 * "Query:" / "Accession:" / "Description:" (src/bathsearch.c:783-785), the report above, and p7_pli_Statistics from "Internal pipeline
 * statistics summary:" to "Total number of hits:" (src/p7_pipeline.c:1836-1874).  Call after bathhost_search_finish. */
int  bathhost_search_format_output(const bathhost_search *s, int textw, char *buf, size_t cap, size_t *needed);

/* ---- f4: E-value calibration by brief simulation (calibrate.cpp) ------------------------------------------------
 * p7_Calibrate with the frameshift branch (src/evalues.c:64-183: p7_Lambda, p7_MSVMu, p7_ViterbiMu, p7_Tau, p7_fs_Tau_3codons,
 * p7_fs_Tau_5codons), each simulation one batched stage call into the device library instead of 200 single-sequence kernel calls.
 *   convert_flow = 0  bathbuild: all five simulations from one generator seeded per model (src/p7_builder.c:130, evalues.c:94-98)
 *   convert_flow = 1  bathconvert / bathfetch (src/bathconvert.c:128-161; src/bathfetch.c:295-325): the two frameshift simulations
 *                     only, on a generator created once per run that keeps running from model to model: rng_state carries it
 *                     (0 = fresh generator from seed) and receives the state left behind.
 * seed 0 = 42 (the programs' default); which_mask bit 0 MSV, 1 Viterbi, 2 Forward, 3 FS3, 4 FS5 (0 = all; the generator is
 * advanced past skipped simulations); lambda <= 0: p7_Lambda of the model (flow 0) or the model file's lambda (flow 1).
 * evparam[8] in the order of bathhost_model_info.evparam; simulations not run stay -99999. */
typedef struct {
  uint32_t seed;
  uint32_t rng_state;
  int32_t  convert_flow;
  int32_t  which_mask;
  double   lambda;
} bathhost_calibration;
int    bathhost_calibrate(const bathhost_model *m, const bathhost_backend *be, bathhost_calibration *cal, double evparam[8]);
double bathhost_model_lambda(const bathhost_model *m);          /* p7_Lambda, src/evalues.c:243-250 */

/* ---- HMMER3/f -> BATH3/f (convert.cpp) ----------------------------------------------------------------------------
 * bathconvert for a library of hmmbuild models (read each model, add the frameshift parts, calibrate the two frameshift taus as
 * src/bathconvert.c:128-161 does, write): every model of in_path, read in one pass, is written to out_path as its own text with the first line
 * "BATH3/f", and "STATS LOCAL FS3 FORWARD", "STATS LOCAL FS5 FORWARD", "FRAMESHIFT PROB" and "CODON TABLE" lines after its
 * "STATS LOCAL FORWARD" line; every other byte is as the input has it.  ct (0 = 1) and fsprob (0 = 0.01) apply to every model.
 * The taus are those of bathhost_calibrate(convert_flow = 1, which_mask = FS3 | FS5) called model after model on one generator
 * (seed; rng_state carried), with the lambda of each model's STATS LOCAL FORWARD line.  With the backend's load_fs_profile_set /
 * fs_set_scores the simulations of many models share each device call (the output is the same).  BATHHOST_EFORMAT for anything but
 * HMMER3/f input, EINVAL for ct or fsprob; on failure out_path is not written.  *nmodels = models converted;
 * bathhost_convert_last_error() says why a call of this thread failed. */
int         bathhost_convert(const char *in_path, const char *out_path, int ct, float fsprob, uint32_t seed,
                             const bathhost_backend *be, int *nmodels);
const char *bathhost_convert_last_error(void);

#ifdef __cplusplus
}
#endif
#endif
