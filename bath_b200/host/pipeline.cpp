// pipeline.cpp -- host side of the translated-search path: the stage-batched frameshift pipeline (libbathhost.so).
//
// Restates the control flow of p7_Pipeline_BATH / p7_pli_Frameshift (src/p7_pipeline.c:1583-1821, :1339-1522),
// p7_domaindef_ByPosteriorHeuristics_Frameshift_BATH and rescore_isolated_domain_frameshift
// (src/p7_domaindef.c:301-473, :993-1191), p7_pli_postDomainDef_Frameshift_BATH (src/p7_pipeline.c:1005-1144)
// and the hit post-processing of bathsearch (src/bathsearch.c:869-921; src/p7_tophits.c:789-960), with every DP
// call replaced by ONE batched call per stage into the device library (include/bathgpu.h) through a table
// of function pointers.  P-values, thresholds, window merging, region heuristics, coordinates and hit records
// are computed here exactly as the reference computes them; nothing in this file does dynamic programming
// over model nodes except the 2-state bias filter (p7_bg_FilterScore), which the reference also runs on the host.
//
// Multi-domain regions of the frameshift branch are split as the reference splits them (src/p7_domaindef.c:395-453): Forward
// matrix from the device, 200 sampled tracebacks and their clustering in stotrace.cpp.  Not restated: the same step of the
// standard-translation branch (region_trace_ensemble, src/p7_domaindef.c:539-587) -- there such regions are rescored as one
// envelope and counted in the statistics.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <limits>
#include <map>
#include <tuple>
#include <string>
#include <thread>
#include <time.h>
#include <vector>
#include <memory>

#include "../../include/bathhost.h"
#include "../../include/bathgpu.h"
#include "host_internal.h"
#include "model_internal.h"

namespace bathhost {

static const double kLog2 = 0.69314718055994529;
static const float  kNegInfF = -std::numeric_limits<float>::infinity();

// ------------------------------------------------------------------------------------------
// p7_FLogsum (src/logsum.c:58-111)
static float g_logsum[16000];
static bool  g_logsum_ready = false;
static void flogsum_init()
{
  if (g_logsum_ready) return;
  for (int i = 0; i < 16000; ++i) g_logsum[i] = log(1. + exp((double) -i / 1000.f));
  g_logsum_ready = true;
}
static float flogsum(float a, float b)
{
  const float mx = (a > b) ? a : b, mn = (a > b) ? b : a;
  return (mn == kNegInfF || (mx - mn) >= 15.7f) ? mx : mx + g_logsum[(int) ((mx - mn) * 1000.f)];
}

// Easel statistics (esl_gumbel.c, esl_exponential.c; public Easel definitions)
static double gumbel_surv(double x, double mu, double lambda)
{
  const double y = lambda * (x - mu), ey = -exp(-y);
  return (fabs(ey) < 5e-9) ? -ey : 1 - exp(ey);
}
static double gumbel_invsurv(double p, double mu, double lambda)
{
  const double lp = (p < 5e-9) ? log(p) : log(-1. * log1p(-p));
  return mu - (lp / lambda);
}
static double exp_surv(double x, double mu, double lambda)    { return (x < mu) ? 1.0 : exp(-lambda * (x - mu)); }
static double exp_logsurv(double x, double mu, double lambda) { return (x < mu) ? 0.0 : -lambda * (x - mu); }

// ------------------------------------------------------------------------------------------
// null model with the 2-state bias filter (src/p7_bg.c:189-197, :356-384, :449-573; Easel esl_hmm.c)
struct Background {
  float f[kK];
  float p1, omega;
  float t[2][3], e[2][kK], eo[kKp][2], pi[2];

  explicit Background(const NullModel &n) { for (int x = 0; x < kK; ++x) f[x] = n.f[x]; p1 = n.p1; omega = n.omega; }
  static float p1_for_length(int L) { return (float) L / (float) (L + 1); }
  void set_length(int L) { p1 = p1_for_length(L); t[0][0] = p1; t[0][1] = 1.0f - p1; }
  float null_one(int L) const { return (float) L * log(p1) + log(1. - p1); }
  float fs_null_one(int La) const { float per_frame = (float) La * log(p1) + log(1. - p1); return per_frame + log(3.0); }

  void set_filter(int M, const float *compo)
  {
    const float L0 = 400.0, L1 = (float) M / 8.0;
    t[0][0] = L0 / (L0 + 1.0f); t[0][1] = 1.0f / (L0 + 1.0f); t[0][2] = 1.0f;
    t[1][0] = 1.0f / (L1 + 1.0f); t[1][1] = L1 / (L1 + 1.0f); t[1][2] = 1.0f;
    for (int x = 0; x < kK; ++x) { e[0][x] = f[x]; e[1][x] = compo[x]; }
    pi[0] = 0.999; pi[1] = 0.001;
    // esl_hmm_Configure: emission odds against the background; gap/'*'/'~' = 1; degenerates = summed e over summed f
    for (int x = 0; x < kK; ++x) for (int k = 0; k < 2; ++k) eo[x][k] = e[k][x] / f[x];
    for (int k = 0; k < 2; ++k) { eo[kK][k] = 1.0; eo[kKp - 2][k] = 1.0; eo[kKp - 1][k] = 1.0; }
    static const int members[6][2] = { { 2, 11 }, { 7, 9 }, { 3, 13 }, { 8, 8 }, { 1, 1 }, { -1, -1 } };
    for (int x = kK + 1; x <= kKp - 3; ++x)
      for (int k = 0; k < 2; ++k) {
        float num = 0.0f, den = 0.0f;
        for (int y = 0; y < kK; ++y) {
          const int *mb = members[x - kK - 1];
          const bool in = (mb[0] < 0) || y == mb[0] || y == mb[1];
          if (in) { num += e[k][y]; den += f[y]; }
        }
        eo[x][k] = (den > 0.0f) ? num / den : 0.0f;
      }
  }

  // esl_hmm_Forward, 2 states, per-row rescaling by the row maximum; eo = [kKp][2] emission odds, t00 = t[0][0] (the rest of row 0 follows),
  // t10/t11 = row 1.  Returns the summed log scale factors.  bathgpu_bias_forward runs exactly these operations in this order.
  static float hmm_forward_tab(const float *eo, float t00, float t10, float t11, const uint8_t *dsq, int L)
  {
    if (L == 0) return 0.0f;           // pi[M] is 0 in this model: log(0); never reached in the reference (L >= 1 everywhere it is called)
    const float t[2][2] = { { t00, 1.0f - t00 }, { t10, t11 } };
    const float pi[2] = { 0.999f, 0.001f };
    float prev[2], cur[2], logsc = 0;
    float mx = 0.0;
    for (int k = 0; k < 2; ++k) { prev[k] = eo[2 * dsq[1] + k] * pi[k]; mx = std::max(prev[k], mx); }
    for (int k = 0; k < 2; ++k) prev[k] /= mx;
    logsc += (float) log(mx);          // accumulated in float, in row order, as esl_hmm_Forward sums fwd->sc[]
    for (int i = 2; i <= L; ++i) {
      mx = 0.0;
      for (int k = 0; k < 2; ++k) {
        cur[k] = 0.0;
        for (int m = 0; m < 2; ++m) cur[k] += prev[m] * t[m][k];
        cur[k] *= eo[2 * dsq[i] + k];
        mx = std::max(cur[k], mx);
      }
      for (int k = 0; k < 2; ++k) prev[k] = cur[k] / mx;
      logsc += (float) log(mx);
    }
    float last = 0.0;
    for (int m = 0; m < 2; ++m) last += prev[m] * 1.0f;
    logsc += (float) log(last);
    return logsc;
  }
  float hmm_forward(const uint8_t *dsq, int L) const { return hmm_forward_tab(&eo[0][0], t[0][0], t[1][0], t[1][1], dsq, L); }
  // p7_bg_FilterScore: the Forward score with the null model's length distribution imposed (src/p7_bg.c:491-500)
  float filter_score_from(float fwd, int L) const { return fwd + (float) L * logf(p1) + logf(1. - p1); }
  float filter_score(const uint8_t *dsq, int L) const { return filter_score_from(hmm_forward(dsq, L), L); }

  // p7_bg_fs_FilterScore: three frames of the DNA window, canonical residues only (src/p7_bg.c:522-573)
  static int frame_residues(const uint8_t *dna, int L, int fr, const uint8_t gcode[64], uint8_t *orf)     // fills orf[1..], returns the count
  {
    int j = 1;
    for (int i = fr; i <= L - 2; i += 3) {
      const uint8_t a = dna[i], b = dna[i + 1], c = dna[i + 2];
      if (a < 4 && b < 4 && c < 4) {
        const uint8_t aa = gcode[16 * a + 4 * b + c];
        if (aa < kK) orf[j++] = aa;
      }
    }
    return j - 1;
  }
  float fs_filter_score_from(const float sc[3], int L) const
  {
    float sum = kNegInfF;
    for (int fr = 0; fr < 3; ++fr) sum = flogsum(sum, sc[fr]);
    return sum + ((float) (L / 3) * logf(p1) + logf(1. - p1) + log(3.0));
  }
  float fs_filter_score(const uint8_t *dna, int L, const uint8_t gcode[64]) const
  {
    std::vector<uint8_t> orf((size_t) L + 2);
    float sc[3];
    for (int fr = 1; fr <= 3; ++fr) sc[fr - 1] = hmm_forward(orf.data(), frame_residues(dna, L, fr, gcode, orf.data()));
    return fs_filter_score_from(sc, L);
  }
};

// ------------------------------------------------------------------------------------------
struct Orf {
  int start, end;            // nucleotide coordinates in the ORIENTED block, start < end
  int frame;
  long long offset;          // first residue in the block's residue buffer
  int n;                     // residues
  int window_idx = -1;       // orfsq->idx
  int local_idx = 0;         // rank among ALL ORFs of its block: the reference's index i (hit_windows ids)
};

struct OrfWin { int id, n, k, length; float score; };      // P7_HMM_WINDOW fields the pipeline reads
struct DnaWin { long long n; int k, length; };

struct Domain {
  int   ienv, jenv, iali, jali, ihmm, jhmm;   // window-relative until post-processing
  float envsc, oasc, domcorrection;
  std::vector<bathgpu_trace_step> tr;          // positions relative to the window
};

// P7_ALIDISPLAY as p7_alidisplay_fs_Create / p7_alidisplay_nonfs_Create fill it (src/p7_alidisplay.c:538-931, :937-1232):
// one character per core trace position (five for the nucleotide line); codon[] = codon length, 0 delete, 6 stop codon
struct AliDisplay {
  std::string model, mline, aseq, ntseq, ppline, csline, rfline;
  std::string cigar;                 // the whole CIGAR string (bathhost_hit::cigar holds its first 1023 characters)
  std::vector<uint8_t> codon;
  int N = 0;
  void size_for(int n, bool cs, bool rf)          // all lines are written by column index: one allocation each
  {
    N = n;
    model.assign(n, ' '); mline.assign(n, ' '); aseq.assign(n, ' '); ppline.assign(n, ' '); ntseq.assign((size_t) 5 * n, ' ');
    if (cs) csline.assign(n, ' ');
    if (rf) rfline.assign(n, ' ');
    codon.assign(n, 0);
  }
};

struct Hit {
  bathhost_hit pub;
  AliDisplay ad;
  bool from_fs_branch = false;      // P7_HIT::frameshift: made by p7_pli_postDomainDef_Frameshift_BATH (src/p7_pipeline.c:1114)
  double sortkey;
  bool duplicate = false, reported = false;
  bool evalue_done = false;         // lnP_raw holds the hit's own ln P; pub.lnP the search-space corrected one
  double lnP_raw = 0.0;
};

struct Options {
  double F1 = 0.02, F2 = 1e-3, F3 = 1e-5, F4 = 5e-4, E = 10.0;
  int    min_orf = 20, block_length = 262144, lanes_u8 = 16, lanes_i16 = 8;
  bool   do_bias = true, do_null2 = true, top = true, bottom = true;
  bool   frameline = false;           // --frameline: a FRAME line in every alignment block
  bool   fs = true;                   // --fs; false: bathsearch's default standard-translation pipeline (src/p7_pipeline.c:106-107)
};

}  // namespace bathhost

using namespace bathhost;

// grow-only host buffer for results the device writes: page-locked when the backend offers it (the copies then run at link rate)
struct HostBuf {
  float *p = nullptr; size_t cap = 0; void (*release)(void *) = nullptr;
  HostBuf() = default;
  HostBuf(const HostBuf &) = delete;                   // owns its block
  HostBuf &operator=(const HostBuf &) = delete;
  float *get(const bathhost_backend &be, size_t nfloats)
  {
    if (nfloats <= cap) return p;
    if (p) { if (release) release(p); else free(p); }
    size_t want = (size_t) 1 << 18;                       // powers of two: a buffer given back to the backend's cache fits the next request
    while (want < nfloats) want <<= 1;
    release = be.host_alloc ? be.host_free : nullptr;
    p = (float *) (be.host_alloc ? be.host_alloc(want * sizeof(float)) : malloc(want * sizeof(float)));
    cap = p ? want : 0;
    return p;
  }
  ~HostBuf() { if (p) { if (release) release(p); else free(p); } }
};

// Large scratch arrays of a batch (the decoding products of every window: ~80 bytes per window row, 0.5-0.7 GB per 1 Gbp profile) come
// from a process-wide free list instead of the heap: glibc hands freed blocks of this size back to the kernel, so every search paid
// for mapping and zeroing them again, from all host threads at once (page-fault storms: 35 -> 175 ms on the same phase).
class ScratchPool {
 public:
  static ScratchPool &get() { static ScratchPool p; return p; }
  std::vector<float> take(size_t n)
  {
    std::lock_guard<std::mutex> lk(mu_);
    size_t best = idle_.size();
    for (size_t z = 0; z < idle_.size(); ++z) if (idle_[z].capacity() >= n && (best == idle_.size() || idle_[z].capacity() < idle_[best].capacity())) best = z;
    std::vector<float> v;
    if (best < idle_.size()) { v.swap(idle_[best]); idle_.erase(idle_.begin() + (long) best); }
    return v;                                      // the caller resizes; contents are whatever the last user left
  }
  void give(std::vector<float> &&v)
  {
    std::lock_guard<std::mutex> lk(mu_);
    if (v.capacity() == 0) return;
    if (idle_.size() >= 64) { size_t small = 0; for (size_t z = 1; z < idle_.size(); ++z) if (idle_[z].capacity() < idle_[small].capacity()) small = z; idle_.erase(idle_.begin() + (long) small); }
    idle_.push_back(std::move(v));
  }
 private:
  std::mutex mu_;
  std::vector<std::vector<float>> idle_;
};

struct SeqRef {                                  // one queued target sequence (the caller keeps dsq alive until the batch has run)
  std::string name;
  const uint8_t *dsq = nullptr;                  // 1..n with sentinels
  int64_t n = 0, seqidx = 0;
  std::vector<uint8_t> own;                      // bathhost_search_sequence copies nothing; _queue_copy keeps the bytes here
};

struct bathhost_search {
  const bathhost_model *model;
  std::vector<bathhost_backend> bes;              // device contexts the stages are dealt to (one or more per GPU)
  std::vector<std::unique_ptr<HostBuf[]>> be_xbuf;   // per device context: X rows of the Forward / Backward parsers (page-locked, reused from unit to unit)
  Options               opt;
  Background            bg;
  std::vector<float>    compo;
  uint8_t               gcode[64];
  bathhost_stats        st{};
  std::vector<Hit>      hits;
  std::string           err;
  std::mutex            err_mu;
  std::vector<SeqRef>   queue;                    // sequences waiting for bathhost_search_run
  std::vector<uint8_t>  tjb_tab;                  // per ORF length L: the MSV filter's tjb byte cost and the null1 score (they depend on
  std::vector<float>    null_tab;                 // the profile and L only; grown to the longest block of a batch, kept across batches)
  std::vector<float>    compo_term;               // summands of the local composition per node and residue (compo_terms)
  bool                  finished = false;
  // ---- state the reference carries from one block-strand to the next, across sequences (src/bathsearch.c:817,1060-1105):
  // the hit_windows list is created once per query and never reset; by_id indexes it by ORF rank
  std::vector<OrfWin>   hit_windows;
  std::vector<std::vector<int>> by_id;
  // the length model left in om_fs5 by the last thing that reconfigured it (src/p7_domaindef.c:324, :1018):
  // p7_DomainDecoding_Frameshift reads its N/J/C loop odds (decoding_fs.c:309-349)
  float                 om5_nj = 1.0f;
  int                   om5_L = 100;
  int64_t               nseqs = 0;
  int64_t               chunk_nt = 0;             // 0: chosen per batch

  bathhost_search(const bathhost_model *m, const bathhost_backend *b, int nb) : model(m), bes(b, b + nb), bg(m->bg)
  {
    for (int k = 0; k < nb; ++k) be_xbuf.emplace_back(new HostBuf[2]);
  }
};

namespace {

int fail(bathhost_search *s, int code, const std::string &msg) { std::lock_guard<std::mutex> lk(s->err_mu); s->err = msg; return code; }

// The host threads of this process: ONE persistent pool shared by every search and every device driver thread (a pool per
// GPU-rank, re-spawned per stage, starved the 8-GPU search of cores).  BATHHOST_THREADS caps it (default: all cores, at most 64).
// parallel_chunks(n, min_chunk, fn) runs fn(a, b) over a partition of [0, n); the caller works too, and calls from several
// threads at once share the workers.
class HostPool {
 public:
  static HostPool &get() { static HostPool p; return p; }
  size_t size() const { return workers_.size() + 1; }
  struct Job { std::function<void(size_t, size_t)> fn; size_t n = 0, step = 1; std::atomic<size_t> next{ 0 }, done{ 0 }; size_t nchunks = 0; };
  void run(size_t n, size_t nthr, const std::function<void(size_t, size_t)> &fn)
  {
    auto job = std::make_shared<Job>();
    job->fn = fn; job->n = n;
    const size_t pieces = nthr * 4;                         // finer than the thread count: uneven items even out
    job->step = std::max<size_t>(1, (n + pieces - 1) / pieces);
    job->nchunks = (n + job->step - 1) / job->step;
    { std::lock_guard<std::mutex> lk(mu_); jobs_.push_back(job); }
    cv_.notify_all();
    work(*job);
    std::unique_lock<std::mutex> lk(mu_);
    done_cv_.wait(lk, [&] { return job->done.load() >= job->nchunks; });
    jobs_.erase(std::remove(jobs_.begin(), jobs_.end(), job), jobs_.end());
  }
 private:
  HostPool()
  {
    const char *e = getenv("BATHHOST_THREADS");
    const long v = e ? atol(e) : 0;
    const long hw = std::max<long>(1, v > 0 ? std::min<long>(v, 256) : std::min<long>((long) std::thread::hardware_concurrency(), 64));
    for (long t = 1; t < hw; ++t) workers_.emplace_back([this] { loop(); });
  }
  ~HostPool()
  {
    { std::lock_guard<std::mutex> lk(mu_); stop_ = true; }
    cv_.notify_all();
    for (auto &t : workers_) t.join();
  }
  void work(Job &j)
  {
    for (;;) {
      const size_t c = j.next.fetch_add(1);
      if (c >= j.nchunks) return;
      const size_t a = c * j.step, b = std::min(j.n, a + j.step);
      j.fn(a, b);
      if (j.done.fetch_add(1) + 1 >= j.nchunks) { std::lock_guard<std::mutex> lk(mu_); done_cv_.notify_all(); }
    }
  }
  void loop()
  {
    for (;;) {
      std::shared_ptr<Job> job;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] {
          if (stop_) return true;
          for (auto &j : jobs_) if (j->next.load() < j->nchunks) return true;
          return false;
        });
        if (stop_) return;
        for (auto &j : jobs_) if (j->next.load() < j->nchunks) { job = j; break; }
      }
      if (job) work(*job);
    }
  }
  std::vector<std::thread> workers_;
  std::vector<std::shared_ptr<Job>> jobs_;
  std::mutex mu_;
  std::condition_variable cv_, done_cv_;
  bool stop_ = false;
};

template <class F> void parallel_chunks(size_t n, size_t min_chunk, F &&fn)
{
  HostPool &pool = HostPool::get();
  const size_t nthr = std::max<size_t>(1, std::min(pool.size(), n / std::max<size_t>(1, min_chunk)));
  if (nthr <= 1) { fn((size_t) 0, n); return; }
  pool.run(n, nthr, std::function<void(size_t, size_t)>(std::ref(fn)));
}

struct StageTimer {              // adds the time since construction / last lap to a stats counter
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  void lap(int64_t &acc) {
    auto t1 = std::chrono::steady_clock::now();
    acc += std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
    t0 = t1;
  }
};

// BATHHOST_TRACE=1: wall time of every phase of run_batch on stderr (tuning aid)
struct PhaseTrace {
  bool on = getenv("BATHHOST_TRACE") != nullptr;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now(), t = t0;
  double cpu0 = cpu_ms();
  static double cpu_ms() { timespec ts; clock_gettime(CLOCK_PROCESS_CPUTIME_ID, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }
  void mark(const char *what)
  {
    if (!on) return;
    const auto n = std::chrono::steady_clock::now();
    const double c = cpu_ms();                              // CPU time of the whole process: meaningful with one search and BATHGPU_BLOCKING_SYNC=1
    fprintf(stderr, "[bathhost] %-34s %9.2f ms (at %9.2f)  cpu %9.2f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count(),
            std::chrono::duration<double, std::milli>(n - t0).count(), c - cpu0);
    t = n; cpu0 = c;
  }
};

// BE: the bathhost_backend the call goes to (a local reference at every call site)
static const bool g_trace_calls = [] { const char *e = getenv("BATHHOST_TRACE"); return e && atoi(e) >= 2; }();   // BATHHOST_TRACE=2: slow stage calls too
static const double g_trace_call_ms = [] { const char *e = getenv("BATHHOST_TRACE"); return e && atoi(e) >= 3 ? 0.2 : 5.0; }();   // =3: every call from 0.2 ms
#define BE_TRY(s, call, what)                                                                   \
  do { const auto t0_ = std::chrono::steady_clock::now();                                       \
       int st_ = (call);                                                                        \
       if (g_trace_calls) { const double ms_ = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0_).count(); \
         if (ms_ >= g_trace_call_ms) fprintf(stderr, "[bathhost]   ctx %p %-28s %9.2f ms\n", BE.ctx, what, ms_); } \
       if (st_ != 0) return fail(s, st_, std::string(what) + " failed: " +                      \
       (BE.last_error ? BE.last_error(BE.ctx) : "?")); } while (0)

// p7_pli_ComputeLocalCompo (src/p7_pipeline.c:427-458).  The summand of node k and residue x, f[x] * exp((base_b - rbv[x][k]) / scale_b),
// depends on the profile and the background only: compo_terms tabulates it once per search ([k][x], k = 0..M), and the sum below adds
// the tabulated floats in the reference's order -- the same additions on the same values as recomputing 20 exponentials per node for
// every ORF that reaches the local-composition test (which was the largest host cost of the filter phase).
std::vector<float> compo_terms(const bathhost_model *m, const Background &bg)
{
  const ProteinProfile &q = m->prot;
  const int M = q.M;
  std::vector<float> term((size_t) (M + 1) * kK, 0.0f);
  for (int k = 1; k <= M; ++k)
    for (int x = 0; x < kK; ++x) {
      const float log_odds = ((float) q.base_b - (float) q.rbv[(size_t) x * (M + 1) + k]) / q.scale_b;
      term[(size_t) k * kK + x] = bg.f[x] * expf(log_odds);
    }
  return term;
}

void local_compo(const bathhost_model *m, const float *term, int k_start, int k_end, float *compo)
{
  const int M = m->prot.M;
  int k_len = k_end - k_start + 1;
  if (k_len < 20) { k_start -= (20 - k_len) / 2; k_end += (20 - k_len) / 2; }
  k_start = std::max(1, k_start);
  k_end   = std::min(M, k_end);
  for (int x = 0; x < kK; ++x) compo[x] = 0.0f;
  for (int k = k_start; k <= k_end; ++k)
    for (int x = 0; x < kK; ++x) compo[x] += term[(size_t) k * kK + x];
  float sum = 0.0f;                                  // esl_vec_FNorm
  for (int x = 0; x < kK; ++x) sum += compo[x];
  if (sum != 0.0f) for (int x = 0; x < kK; ++x) compo[x] /= sum;
  else             for (int x = 0; x < kK; ++x) compo[x] = 1.0f / (float) kK;
}

int codon_index5(const uint8_t *dsq, int i, int c)      // quasi-codon of length c ending at i (src/p7_pipeline.c:819-871)
{
  for (int b = 0; b < c; ++b) if (dsq[i - b] >= 4) return c == 3 ? 1364 : (c == 2 || c == 4) ? 1365 : 1366;
  const int x = dsq[i];
  if (c == 1) return x * 341;
  const int w = dsq[i - 1];
  if (c == 2) return x * 341 + w * 85 + 1;
  const int v = dsq[i - 2];
  if (c == 3) return x * 341 + w * 85 + v * 21 + 2;
  const int u = dsq[i - 3];
  if (c == 4) return x * 341 + w * 85 + v * 21 + u * 5 + 3;
  const int t = dsq[i - 4];
  return x * 341 + w * 85 + v * 21 + u * 5 + t + 4;
}

enum { PXXx = 6, PXxX = 7, PxXX = 8 };
enum { P__X = 0, PX__ = 1, PXX_ = 2, PX_X = 3, P_XX = 4, PXXxX = 10, PXxXX = 11, PxXXX = 12, PXXxxX = 13, PXxxXX = 14, PxxXXX = 15 };
enum { TS_M = 1, TS_D = 2, TS_I = 3, TS_N = 5, TS_B = 6, TS_E = 7, TS_C = 8, TS_J = 10 };

// p7_pli_computeAliScores_BATH (src/p7_pipeline.c:781-985): sum of emission and transition log-odds along the core of the trace
float ali_score(const bathhost_model *m, const std::vector<bathgpu_trace_step> &tr, const uint8_t *dsq)
{
  const FsProfile &gm = m->gm5;
  const int M = gm.M;
  const size_t ld = (size_t) M + 1;
  int z1 = 0, z2 = (int) tr.size() - 1;
  while (z1 < (int) tr.size() && tr[z1].st != TS_M) ++z1;
  while (z2 >= 0 && tr[z2].st != TS_M) --z2;
  if (z1 > z2) return 0.0f;
  auto amino_sc = [&](int k, int i, int c) {
    const int ci = codon_index5(dsq, i, c);
    const int aa = gm.codons[(size_t) k * gm.maxcodons + ci];
    return gm.rsc[(size_t) (gm.maxcodons + aa) * ld + k];
  };
  auto tsc = [&](int k, int t) { return gm.tsc[(size_t) k * 8 + t]; };
  std::vector<float> per;
  int k = 0;
  while (z1 <= z2) {
    k = tr[z1].k;
    if (tr[z1].st == TS_M) {
      float v = amino_sc(k, tr[z1].i, tr[z1].c);
      if (z1 > 0 && tr[z1 - 1].st == TS_I)      v += tsc(k - 1, PT_IM);
      else if (z1 > 0 && tr[z1 - 1].st == TS_D) v += tsc(k - 1, PT_DM);
      per.push_back(v);
      k++; z1++;
      while (z1 < z2 && tr[z1].st == TS_M) {
        per.push_back(amino_sc(k, tr[z1].i, tr[z1].c) + tsc(k - 1, PT_MM));
        k++; z1++;
      }
    } else if (tr[z1].st == TS_I) {
      per.push_back(tsc(k, PT_MI));
      z1++;
      while (z1 < z2 && tr[z1].st == TS_I) { per.push_back(tsc(k, PT_II)); z1++; }
    } else if (tr[z1].st == TS_D) {
      per.push_back(tsc(k - 1, PT_MD));
      k++; z1++;
      while (z1 < z2 && tr[z1].st == TS_D) { per.push_back(tsc(k - 1, PT_DD)); k++; z1++; }
    } else break;
  }
  float s = 0.0f;
  for (float v : per) s += v;
  return s;
}

// the alignment summary p7_alidisplay_fs_Create derives from a trace (src/p7_alidisplay.c:696-895): frameshifts,
// stop codons, percent identity and the CIGAR string
static const char kDnaSym[]   = "ACGT-RYMKSWHBVDN*~";
static const char kAminoSym[] = "ACDEFGHIKLMNPQRSTVWY-BJZOUX*~";
enum { Pxxx = 9 };                                          // p7P_xxx: the fifth 3-nucleotide pattern (src/hmmer.h, enum p7p_indel_e)

static char encode_post_prob(float p) { return (p + 0.05 >= 1.0) ? '*' : (char) ((p + 0.05) * 10.0) + '0'; }     // p7_alidisplay_EncodePostProb

// nuc_one .. nuc_five (src/p7_alidisplay.c:107-213): the five display characters of a quasi-codon; bases the alignment
// treats as inserted are lower case, missing ones '-'
static void codon_chars(int c, int indel, const int n[5], char out[5])
{
  auto up = [&](int z) { return kDnaSym[n[z]]; };
  auto lo = [&](int z) { return (char) tolower(kDnaSym[n[z]]); };
  out[0] = (c < 4) ? ' ' : (indel == PxXXX || indel == PxxXXX || indel == Pxxx) ? lo(0) : up(0);
  if (c < 4) out[1] = (indel == P__X || indel == P_XX) ? '-' : (indel == PxXX || indel == Pxxx) ? lo(0) : up(0);
  else       out[1] = (indel == PXXxX || indel == PxXXX || indel == PXXxxX) ? up(1) : lo(1);
  if (c == 1 || indel == PX_X) out[2] = '-';
  else if (indel == P_XX)      out[2] = up(0);
  else if (c < 4)              out[2] = (indel == PXxX || indel == Pxxx) ? lo(1) : up(1);
  else                         out[2] = (indel == PXxXX || indel == PxXXX || indel == PxxXXX) ? up(2) : lo(2);
  if (indel == P__X)                        out[3] = up(0);
  else if (indel == PX_X || indel == P_XX)  out[3] = up(1);
  else if (c < 3)                           out[3] = '-';
  else if (c == 3)                          out[3] = (indel == PXXx || indel == Pxxx) ? lo(2) : up(2);
  else                                      out[3] = (indel == PXXxxX || indel == Pxxx) ? lo(3) : up(3);
  out[4] = (c < 5) ? ' ' : (indel == Pxxx) ? lo(4) : up(4);
}

void summarize_alignment(const bathhost_model *m, const std::vector<bathgpu_trace_step> &tr, const uint8_t *dsq, bathhost_hit &h, AliDisplay *ad = nullptr)
{
  const FsProfile &gm = m->gm5;
  const size_t ld = (size_t) gm.M + 1;
  std::vector<const bathgpu_trace_step *> core;
  for (const auto &s : tr) if (s.st == TS_M || s.st == TS_D || s.st == TS_I) core.push_back(&s);
  std::string cigar;
  int shifts = 0, stops = 0, exact = 0, n_count = 0;
  char buf[32];
  if (ad) ad->size_for((int) core.size(), !m->hmm.cs.empty(), !m->hmm.rf.empty());
  for (size_t z = 0; z < core.size(); ++z) {
    const bathgpu_trace_step &s = *core[z];
    const int nxt = (z + 1 < core.size()) ? core[z + 1]->st : TS_E;
    if (s.st == TS_M) {
      const int ci = codon_index5(dsq, s.i, s.c);
      const int aa = gm.codons[(size_t) s.k * gm.maxcodons + ci];
      const int indel = gm.indel_pos[(size_t) s.k * gm.maxcodons + ci];
      if (aa == amino_code(m->hmm.consensus[s.k])) exact++;
      if (ad) {
        int n[5] = { 0, 0, 0, 0, 0 };
        for (int z5 = 0; z5 < s.c; ++z5) n[z5] = dsq[s.i - (s.c - 1) + z5];
        char cc[5];
        codon_chars(s.c, indel, n, cc);
        memcpy(&ad->ntseq[5 * z], cc, 5);
        ad->model[z] = m->hmm.consensus[s.k];
        ad->mline[z] = (aa == amino_code(m->hmm.consensus[s.k])) ? m->hmm.consensus[s.k]
                       : (expf(gm.rsc[(size_t) (gm.maxcodons + aa) * ld + s.k]) > 1.0) ? '+' : ' ';
        ad->aseq[z] = (char) toupper(kAminoSym[aa]);
        ad->codon[z] = (uint8_t) ((s.c == 3 && (indel == PXXx || indel == PXxX || indel == PxXX)) ? 6 : s.c);
      }
      if (s.c != 3) shifts++;
      else if (indel == PXXx || indel == PXxX || indel == PxXX) stops++;
      if (nxt != TS_M || s.c != 3) {
        if (s.c == 3) n_count += 3;
        else if (indel == PXX_ || indel == PXXxX || indel == PXXxxX) n_count += 2;
        else if (indel == PX_X || indel == PX__ || indel == PXxXX || indel == PXxxXX) n_count += 1;
        snprintf(buf, sizeof buf, "%dM", n_count); cigar += buf;
        n_count = 0;
        if (s.c == 1) cigar += "2B"; else if (s.c == 2) cigar += "1B"; else if (s.c == 4) cigar += "1F"; else if (s.c == 5) cigar += "2F";
        if (indel == P__X || indel == PX_X || indel == PXXxX || indel == PXXxxX) n_count = 1;
        if (indel == P_XX || indel == PXxXX || indel == PXxxXX) n_count = 2;
        if (indel == PxXXX || indel == PxxXXX) n_count = 3;
        if (nxt != TS_M && n_count > 0) { snprintf(buf, sizeof buf, "%dM", n_count); cigar += buf; n_count = 0; }
      } else n_count += 3;
    } else if (s.st == TS_I) {
      const int ci = codon_index5(dsq, s.i, 3);
      const int indel = gm.indel_pos[(size_t) s.k * gm.maxcodons + ci];
      const bool stop = (indel == PXXx || indel == PXxX || indel == PxXX);
      if (stop) stops++;
      if (ad) {
        const int aa = stop ? 27 : gm.codons[(size_t) s.k * gm.maxcodons + ci];
        ad->model[z] = '.';
        ad->aseq[z] = (char) tolower(kAminoSym[aa]);
        const char cc[5] = { ' ', kDnaSym[dsq[s.i - 2]], kDnaSym[dsq[s.i - 1]], kDnaSym[dsq[s.i]], ' ' };
        memcpy(&ad->ntseq[5 * z], cc, 5);
        ad->codon[z] = stop ? 6 : 3;
      }
      n_count += 3;
      if (nxt != TS_I) { snprintf(buf, sizeof buf, "%dI", n_count); cigar += buf; n_count = 0; }
    } else {
      if (ad) { ad->model[z] = m->hmm.consensus[s.k]; ad->aseq[z] = '-'; memcpy(&ad->ntseq[5 * z], " --- ", 5); }
      n_count += 3;
      if (nxt != TS_D) { snprintf(buf, sizeof buf, "%dD", n_count); cigar += buf; n_count = 0; }
    }
    if (ad) {
      ad->ppline[z] = (s.st == TS_D) ? '.' : encode_post_prob(s.pp);
      if (!m->hmm.cs.empty()) ad->csline[z] = (s.st == TS_I) ? '.' : m->hmm.cs[s.k];
      if (!m->hmm.rf.empty()) ad->rfline[z] = (s.st == TS_I) ? '.' : m->hmm.rf[s.k];
    }
  }
  h.shifts = shifts; h.stops = stops;
  h.pid = core.empty() ? 0.0f : ((float) exact / (float) core.size()) * 100;
  snprintf(h.cigar, sizeof h.cigar, "%s", cigar.c_str());
  if (ad) ad->cigar = cigar;
}

// ---- a batch of target sequences, both strands, stage-batched and dealt to one or more devices ---------------------------
// The reference walks each sequence in blocks of block_length nucleotides carrying max_length*3 nucleotides of left
// context, top strand then bottom strand of each block (src/bathsearch.c:1060-1105).  Here the blocks of ALL queued
// sequences are cut into CHUNKS (runs of consecutive blocks, a few Mbp); a chunk's two strands are two UNITS, resident in two
// target slots of one device context.  Every DP stage runs once per unit over the work of all its blocks; units are dealt
// round-robin to the device contexts, each driven by its own host thread, and everything whose result depends on the
// order the reference visits blocks in is done on the host in exactly that order, whatever the number of devices:
//   * hit_windows is never reset between blocks, strands or sequences in the reference (info->hw, src/bathsearch.c:817,
//     1076,1090), so the window picked for an ORF (p7_pli_BuildDNAWindows) and the k-range scan of p7_pli_Frameshift see
//     every window stamped with the same ORF index by EARLIER blocks -- reproduced by appending in reference order;
//   * the length model left in om_fs5 by the previous window's rescoring feeds p7_DomainDecoding_Frameshift;
//   * the early E-value cuts use the residue count at the time the block is processed.
// So the merged hit list of N devices is the one-device list by construction: the same items go through the same kernels,
// only in different batches.
struct BlockInfo {
  long long b0, b1;          // original coordinates of the block on its sequence (context included)
  int       n, C, bw;        // dnasq->n, dnasq->C, dnasq->W
  long long nres_at[2];      // pli->nres when the top / bottom strand of this block is processed
  int       seq;             // index into the batch's sequence list
  long long coff;            // chunk coordinate (top strand, 0-based) of b0: the block is chunk positions coff+1 .. coff+n
};

// q with q[1..len] = positions local0+1 .. local0+len of the block in the strand's orientation (8 more on either side for
// look-backs): the caller's buffer itself on the top strand; on the bottom strand a reverse-complemented copy of the stretch --
// the bottom strand as a whole only ever exists on the device (bathgpu_revcomp_slot)
const uint8_t *oriented(const SeqRef &sq, const BlockInfo &blk, bool complement, long long local0, int len, std::vector<uint8_t> &buf)
{
  if (!complement) return sq.dsq + (blk.b0 - 1) + local0;
  static const uint8_t comp[18] = { 3, 2, 1, 0, 4, 6, 5, 8, 7, 9, 10, 14, 13, 12, 11, 15, 16, 17 };
  const int pad = 8;
  buf.resize((size_t) len + 2 * pad + 2);
  for (int p = -pad + 1; p <= len + pad; ++p) {
    const long long P = blk.b1 + 1 - (local0 + p);          // sequence coordinate of oriented block position local0 + p
    uint8_t c = 255;
    if (P >= 1 && P <= sq.n) { const uint8_t o = sq.dsq[P]; c = (o < 18) ? comp[o] : o; }
    buf[(size_t) (p + pad)] = c;
  }
  return buf.data() + pad;
}

// Stage 1 of one unit for one model, as a library search's set screen left it: ORFs per block, the survivors (sorted by block and
// rank), and the residue buffer their offsets index (shared by the models of the screen)
struct ScreenOut {
  std::vector<int64_t> norfs;
  std::vector<bathgpu_orf_hit> hits;
  std::shared_ptr<std::vector<uint8_t>> res;
};

// The reference's blocks of a batch of sequences (src/bathsearch.c:1060-1105) for a model of C context nucleotides, and the residue
// count as each block-strand is reached (nres: the count before the batch, then after it).  Block starts depend on W only.
std::vector<BlockInfo> cut_blocks(const std::vector<SeqRef> &seqs, int C, const Options &opt, long long &nres)
{
  std::vector<BlockInfo> blocks;
  const int W = opt.block_length;
  for (size_t sq = 0; sq < seqs.size(); ++sq) {
    const int64_t n = seqs[sq].n;
    int64_t pos = 1;
    bool first = true;
    while (pos <= n) {
      const int64_t ctx = first ? 0 : std::min<int64_t>(C, pos - 1);
      BlockInfo b;
      b.b0 = pos - ctx; b.b1 = std::min<int64_t>(n, pos + W - 1);
      b.n = (int) (b.b1 - b.b0 + 1); b.C = (int) ctx; b.bw = (int) (b.b1 - pos + 1);
      b.seq = (int) sq; b.coff = 0;
      b.nres_at[0] = b.nres_at[1] = nres;
      if (b.n >= 15) {
        if (opt.top)    { nres += b.bw; b.nres_at[0] = nres; }
        if (opt.bottom) { nres += b.bw; b.nres_at[1] = nres; }
      }
      blocks.push_back(b);
      pos = b.b1 + 1;
      first = false;
    }
  }
  return blocks;
}

// chunks: runs of consecutive blocks; a chunk's nucleotides are the concatenation of its SEGMENTS (one per sequence it touches: first
// block's b0 .. last block's b1), so blocks of one sequence keep their overlap and nothing is stored twice.  Sets blocks[].coff.
struct ChunkSeg { int seq; long long from, to, off; };     // sequence coordinates from..to at chunk offset off (0-based)
struct Chunk { int blk0, blk1; long long n; std::vector<ChunkSeg> segs; };
std::vector<Chunk> cut_chunks(std::vector<BlockInfo> &blocks, long long target)
{
  std::vector<Chunk> chunks;
  for (size_t b = 0; b < blocks.size(); ++b) {
    const BlockInfo &blk = blocks[b];
    const bool same_seq = !chunks.empty() && chunks.back().blk1 == (int) b && !chunks.back().segs.empty() && chunks.back().segs.back().seq == blk.seq;
    const long long grow = same_seq ? blk.b1 - chunks.back().segs.back().to : blk.n;
    if (chunks.empty() || chunks.back().n + grow > target) { chunks.push_back(Chunk{ (int) b, (int) b, 0, {} }); }
    Chunk &c = chunks.back();
    if (!c.segs.empty() && c.segs.back().seq == blk.seq && c.blk1 == (int) b) {      // the sequence's next block: extend its segment
      blocks[b].coff = c.segs.back().off + (blk.b0 - c.segs.back().from);
      c.n += blk.b1 - c.segs.back().to;
      c.segs.back().to = blk.b1;
    } else {
      c.segs.push_back(ChunkSeg{ blk.seq, blk.b0, blk.b1, c.n });
      blocks[b].coff = c.n;
      c.n += blk.n;
    }
    c.blk1 = (int) b + 1;
  }
  return chunks;
}

// Chunk positions of the blocks of one model in chunks cut for a library (cut_chunks over the blocks of its largest context): every
// block starts at or behind the segment's first nucleotide, so it lies inside the resident chunk.
void place_blocks(std::vector<BlockInfo> &blocks, const std::vector<Chunk> &chunks)
{
  for (const Chunk &c : chunks)
    for (int b = c.blk0; b < c.blk1; ++b)
      for (const ChunkSeg &g : c.segs)
        if (g.seq == blocks[(size_t) b].seq) { blocks[(size_t) b].coff = g.off + (blocks[(size_t) b].b0 - g.from); break; }
}

// The top strand of a chunk into slot_top, and its reverse complement made on the device in slot_bottom (bottom >= 0)
int upload_chunk(bathhost_search *s, const bathhost_backend &BE, const std::vector<SeqRef> &seqs, const Chunk &ch, int slot_top, int slot_bottom,
                 HostBuf &stage)
{
  BE_TRY(s, BE.select_slot(BE.ctx, slot_top), "bathgpu_select_slot");
  if (ch.segs.size() == 1) {                               // the caller's buffer as it is (the byte before and the one after are not read)
    const ChunkSeg &g = ch.segs[0];
    BE_TRY(s, BE.upload_block(BE.ctx, seqs[(size_t) g.seq].dsq + (g.from - 1), ch.n), "bathgpu_upload_block");
  } else if (BE.upload_block_segments) {                 // every piece crosses the link from the caller's buffer: no host copy of the chunk
    std::vector<const uint8_t *> sp(ch.segs.size());
    std::vector<int64_t> sn(ch.segs.size());
    for (size_t g = 0; g < ch.segs.size(); ++g) { sp[g] = seqs[(size_t) ch.segs[g].seq].dsq + ch.segs[g].from; sn[g] = ch.segs[g].to - ch.segs[g].from + 1; }
    BE_TRY(s, BE.upload_block_segments(BE.ctx, sp.data(), sn.data(), (int) sp.size()), "bathgpu_upload_block_segments");
  } else {
    uint8_t *buf = reinterpret_cast<uint8_t *>(stage.get(BE, ((size_t) ch.n + 2 + 3) / 4));
    if (!buf) return fail(s, BATHHOST_EMEM, "host allocation failed");
    buf[0] = 255; buf[ch.n + 1] = 255;
    parallel_chunks(ch.segs.size(), 1, [&](size_t ga, size_t gb) {
      for (size_t g = ga; g < gb; ++g) memcpy(buf + 1 + ch.segs[g].off, seqs[(size_t) ch.segs[g].seq].dsq + ch.segs[g].from, (size_t) (ch.segs[g].to - ch.segs[g].from + 1));
    });
    BE_TRY(s, BE.upload_block(BE.ctx, buf, ch.n), "bathgpu_upload_block");
  }
  if (slot_bottom >= 0) BE_TRY(s, BE.revcomp_slot(BE.ctx, slot_top, slot_bottom), "bathgpu_revcomp_slot");
  return 0;
}

// the default chunk length of a batch of total nucleotides over nbe device contexts
long long chunk_target(const bathhost_search *s, long long total)
{
  long long target = s->chunk_nt;
  if (target <= 0) {
    static const long long env_mbp = [] { const char *e = getenv("BATHHOST_CHUNK_MBP"); return e ? atoll(e) : 0LL; }();
    target = env_mbp > 0 ? env_mbp * 1000000LL
                         : std::max<long long>(4000000LL, std::min<long long>(128000000LL, total / (long long) s->bes.size() + 1));
  }
  return target;
}

struct Unit {                               // one strand of one chunk
  bool complement = false;
  int  sidx = 0, chunk = 0, be = 0, slot = 0;
  int  blk0 = 0, blk1 = 0;                  // its blocks: [blk0, blk1) of the batch's block list
  long long n_total = 0;                    // chunk length (both strands)
  bathhost_stats st{};                      // this unit's share of the counters and stage times
  std::vector<Orf> orfs;                    // of all blocks, block-local coordinates
  std::vector<int> orf_blk;                 // block of each ORF
  std::vector<int> orf_begin;               // [nblocks+1] range of each block's ORFs (index: block - blk0)
  std::vector<uint8_t> residues;
  const uint8_t *sres = nullptr;            // the survivors' residues, indexed by bathgpu_orf_hit.offset (residues, or a library screen's buffer)
  const ScreenOut *pre = nullptr;           // stage 1 of this unit already run by a library search's set screen (nullptr: run it here)
  std::vector<double> P_orf;
  std::vector<float>  fwdsc_orf;
  std::vector<std::vector<OrfWin>> wins_of_orf;     // windows of ORFs that reached the Forward stage, id = block-local ORF index
  std::vector<DnaWin> dwin;                 // DNA windows of all blocks, block-local coordinates
  std::vector<int>    dwin_blk;
  std::vector<int>    dwin_begin;           // [nblocks+1]
  std::vector<size_t> hw_count;             // [nblocks] length of the accumulated hit_windows list after this block-strand
  std::vector<bathgpu_window> gw;
  std::vector<float>   fs_fwd;
  std::vector<int32_t> fs_st;
  std::vector<int>     fsw;                 // windows that go down the frameshift branch
  std::vector<size_t>  xoff;
  float *fxr = nullptr, *bxr = nullptr;     // X rows of the Forward / Backward parsers (the device context's page-locked buffers; valid until its next unit)
  std::vector<int32_t> st2;
  struct Env { int win, i, j; };
  std::vector<Env> envs;
  std::vector<bathgpu_envelope> ge;
  std::vector<bathgpu_domain_result> res;
  std::vector<bathgpu_trace_step> traces;
  struct StdItem { int gi, w; };            // ORF sent down the standard-translation branch, and the DNA window it lost to (-1: none)
  std::vector<StdItem> stdq;
  std::vector<uint8_t> aligned;             // oxf_holder[i] == NULL: this ORF has been aligned already
  std::vector<std::pair<int, Hit>> hits_fs, hits_std;      // (block, hit) in the order the unit produces them
  int &ob(int b) { return orf_begin[(size_t) (b - blk0)]; }
  int &db(int b) { return dwin_begin[(size_t) (b - blk0)]; }
  size_t &hwc(int b) { return hw_count[(size_t) (b - blk0)]; }
  long long goff(const BlockInfo &b) const { return complement ? n_total - (b.coff + b.n) : b.coff; }   // slot coordinate = goff + block-local
  long long start_of(const BlockInfo &b) const { return complement ? b.b1 : b.b0; }                       // dnasq->start
};

// One batch of bias-filter Forward recursions (SURVEY 8 a5): on the device when the backend offers bathgpu_bias_forward, else on the host
// cores with the same operations (Background::hmm_forward_tab).  kind 0: items are ORFs of the selected slot's residue buffer, one
// score each; kind 1: DNA windows of the selected slot, three scores each (frames 1..3).  host_item(i, out) is the host path for item i.
static bool bias_on_device(const bathhost_backend &BE)
{
  static const bool off = [] { const char *e = getenv("BATHHOST_BIAS_HOST"); return e && atoi(e) != 0; }();
  return BE.bias_forward != nullptr && !off;
}
template <class HostItem>
int bias_batch(bathhost_search *s, const bathhost_backend &BE, int kind, const std::vector<bathgpu_bias_item> &items, const std::vector<float> &tables,
               const Background &bg, std::vector<float> &out, HostItem &&host_item)
{
  const size_t per = (kind == 1) ? 3 : 1;
  out.assign(items.size() * per, 0.0f);
  if (items.empty()) return 0;
  if (bias_on_device(BE)) {
    BE_TRY(s, BE.bias_forward(BE.ctx, kind, items.data(), (int) items.size(), tables.data(), (int) (tables.size() / (2 * kKp)), bg.t[1][0], bg.t[1][1],
                              s->gcode, out.data()), "bathgpu_bias_forward");
    return 0;
  }
  parallel_chunks(items.size(), kind == 1 ? 1 : 64, [&](size_t a, size_t b) { for (size_t i = a; i < b; ++i) host_item(i, &out[i * per]); });
  return 0;
}

// stages 1-3 for one unit: ORFs of every block, MSV, bias, Viterbi/SSV windows, local-composition re-check, protein Forward
int filter_unit(bathhost_search *s, Unit &S, const std::vector<BlockInfo> &blocks)
{
  const bathhost_model *m = s->model;
  const ProteinProfile &q = m->prot;
  const Options &opt = s->opt;
  const int M = q.M;
  const float *ev = m->hmm.evparam;
  const Background &bg = s->bg;
  const bathhost_backend &BE = s->bes[(size_t) S.be];
  StageTimer tm;

  // ---- stage 1: translation of every block, MSV over every ORF and the cheap side of the F1 test in ONE device call
  // (SURVEY 8 f1; src/bathsearch.c:385-392, src/p7_pipeline.c:1632-1652).  What comes back are the ORFs that can still pass F1,
  // with their block-local rank in the reference's ORF order (the window bookkeeping keys on it) and their residues.
  BE_TRY(s, BE.select_slot(BE.ctx, S.slot), "bathgpu_select_slot");      // the unit's nucleotides were made resident by the caller
  const size_t nblk = (size_t) (S.blk1 - S.blk0);
  S.orf_begin.assign(nblk + 1, 0);
  std::vector<bathgpu_block> bdesc(nblk);
  int maxlen = 1;
  for (size_t b = 0; b < nblk; ++b) {
    const BlockInfo &blk = blocks[(size_t) S.blk0 + b];
    bdesc[b].goff = S.goff(blk); bdesc[b].n = (blk.n >= 15) ? blk.n : 0; bdesc[b].C = blk.C;
    maxlen = std::max(maxlen, blk.n / 3 + 1);
  }
  // per-length integers and null1 scores depend on the ORF length only: tabulated once per search (run_batch grows the tables to the
  // longest block before the units start)
  const std::vector<uint8_t> &tjb_of = s->tjb_tab;
  const std::vector<float>   &null_of = s->null_tab;
  if ((int) tjb_of.size() < maxlen + 1) return fail(s, BATHHOST_EINVAL, "length tables shorter than the longest block");
  // the Gumbel tail is monotone: P > F1 exactly when the bit score is below x1 = invsurv(F1); the device keeps what is within a
  // margin of x1 or above it, the exact tail is evaluated here for those
  const double x1 = gumbel_invsurv(opt.F1, ev[EV_MMU], ev[EV_MLAMBDA]);
  std::vector<int64_t> norfs_blk(nblk, 0);
  std::vector<bathgpu_orf_hit> surv;
  if (S.pre) {
    norfs_blk = S.pre->norfs; surv = S.pre->hits; S.sres = S.pre->res->data();
  } else {
    int64_t nsurv = 0, nsres = 0;
    BE_TRY(s, BE.orfs_msv_screen(BE.ctx, bdesc.data(), (int) nblk, S.complement ? 1 : 0, s->gcode, opt.min_orf, tjb_of.data(), null_of.data(),
                                     maxlen, x1 - 0.02, norfs_blk.data(), &nsurv, &nsres), "bathgpu_orfs_msv_screen");
    surv.resize((size_t) nsurv);
    S.residues.resize((size_t) nsres);
    BE_TRY(s, BE.orfs_fetch(BE.ctx, surv.data(), S.residues.data()), "bathgpu_orfs_fetch");
    S.sres = S.residues.data();
  }
  for (size_t b = 0; b < nblk; ++b) S.st.n_orfs += norfs_blk[b];
  const int norf = (int) surv.size();
  S.orfs.resize((size_t) norf); S.orf_blk.resize((size_t) norf);
  {
    size_t z = 0;
    for (size_t b = 0; b < nblk; ++b) {
      S.orf_begin[b] = (int) z;
      while (z < surv.size() && surv[z].block == (int) b) {
        Orf &o = S.orfs[z];
        o.start = surv[z].start; o.end = surv[z].end; o.frame = surv[z].frame; o.offset = surv[z].offset; o.n = surv[z].n;
        o.local_idx = surv[z].index; o.window_idx = -1;
        S.orf_blk[z] = S.blk0 + (int) b;
        ++z;
      }
    }
    S.orf_begin[nblk] = (int) z;
  }
  S.P_orf.assign((size_t) norf, 1.0);
  S.fwdsc_orf.assign((size_t) norf, kNegInfF);
  S.wins_of_orf.assign((size_t) norf, {});
  tm.lap(S.st.us_msv);
  if (norf == 0) return 0;

  std::vector<Orf> &orfs = S.orfs;
  const uint8_t *residues = S.sres;
  auto orf_dsq = [&](const Orf &o, std::vector<uint8_t> &buf) {      // 1-based with sentinels, for the bias filter
    buf.assign((size_t) o.n + 2, 255);
    memcpy(buf.data() + 1, residues + o.offset, (size_t) o.n);
  };
  std::vector<int> live((size_t) norf);
  std::vector<float> usc((size_t) norf);
  for (int i = 0; i < norf; ++i) { live[i] = i; usc[i] = surv[i].usc; }
  struct Cand { int orf; float nullsc, usc, filtersc, vfsc; double P; bool need_vit; };
  std::vector<Cand> cand;
  std::vector<uint8_t> buf;
  {
    // the exact F1 test and the bias filter of each survivor are independent of one another: all host cores, then the
    // counters and the candidate list in ORF order
    struct Pre { uint8_t stage; float filtersc; double P; };       // stage 0: fails F1 on the MSV score, 1: fails after the bias filter, 2: passes
    std::vector<Pre> pre(live.size());
    parallel_chunks(live.size(), 256, [&](size_t ta, size_t tb) {
      for (size_t t = ta; t < tb; ++t) {
        const Orf &o = orfs[live[t]];
        const float nullsc = null_of[o.n];
        const float seqsc = (usc[t] - nullsc) / kLog2;
        Pre &r = pre[t];
        r.stage = 0; r.filtersc = nullsc; r.P = 1.0;
        if (seqsc < x1 - 0.01) continue;
        const double P = gumbel_surv(seqsc, ev[EV_MMU], ev[EV_MLAMBDA]);
        if (P > opt.F1) continue;
        r.stage = 2; r.P = P;
      }
    });
    if (opt.do_bias) {                                      // (:1657-1663) one batch over everything that passed F1 on the MSV score
      std::vector<int> bt;
      for (size_t t = 0; t < live.size(); ++t) if (pre[t].stage == 2) bt.push_back((int) t);
      std::vector<bathgpu_bias_item> items(bt.size());
      std::vector<float> tables(&bg.eo[0][0], &bg.eo[0][0] + 2 * kKp), fsc;
      for (size_t z = 0; z < bt.size(); ++z) {
        const Orf &o = orfs[live[bt[z]]];
        items[z] = bathgpu_bias_item{ o.offset, o.n, 0, Background::p1_for_length(o.n), 0 };
      }
      const int rc = bias_batch(s, BE, 0, items, tables, bg, fsc, [&](size_t z, float *out) {
        std::vector<uint8_t> lbuf;
        orf_dsq(orfs[live[bt[z]]], lbuf);
        *out = Background::hmm_forward_tab(tables.data(), items[z].t00, bg.t[1][0], bg.t[1][1], lbuf.data(), items[z].L);
      });
      if (rc != 0) return rc;
      parallel_chunks(bt.size(), 1024, [&](size_t za, size_t zb) {
        Background lbg = bg;
        for (size_t z = za; z < zb; ++z) {
          const size_t t = (size_t) bt[z];
          const Orf &o = orfs[live[t]];
          Pre &r = pre[t];
          lbg.set_length(o.n);
          r.filtersc = lbg.filter_score_from(fsc[z], o.n);
          const float seqsc = (usc[t] - r.filtersc) / kLog2;
          r.P = gumbel_surv(seqsc, ev[EV_MMU], ev[EV_MLAMBDA]);
          if (r.P > opt.F1) r.stage = 1;
        }
      });
    }
    for (size_t t = 0; t < live.size(); ++t) {
      if (pre[t].stage == 0) continue;
      const Orf &o = orfs[live[t]];
      S.st.pos_past_msv += (int64_t) o.n * 3;
      if (pre[t].stage == 1) continue;
      S.st.pos_past_bias += (int64_t) o.n * 3;
      Cand c; c.orf = live[t]; c.nullsc = null_of[o.n]; c.usc = usc[t]; c.filtersc = pre[t].filtersc; c.vfsc = kNegInfF; c.P = pre[t].P;
      c.need_vit = (c.P > opt.F2);
      cand.push_back(c);
    }
  }
  tm.lap(S.st.us_bias);
  if (cand.empty()) return 0;

  // ---- stage 2: Viterbi filter with windows, or the SSV window finder for ORFs already below F2 (:1666-1680)
  auto make_desc = [&](const Cand &c, bool windows) {
    const Orf &o = orfs[c.orf];
    bathgpu_orf d; memset(&d, 0, sizeof d);
    d.offset = o.offset; d.L = o.n; d.tjb_b = q.tjb_for_length(o.n); d.xw_move = q.xw_move_for_length(o.n);
    if (windows) {
      float invP = gumbel_invsurv(opt.F2, ev[EV_VMU], ev[EV_VLAMBDA]);          // vitfilter.c:313-321
      d.vit_thresh = (int16_t) ceil(((c.filtersc + kLog2 * invP + 3.0) * q.scale_w) - (float) q.xw_E_move - (float) d.xw_move + (float) q.base_w);
      invP = gumbel_invsurv(opt.F2, ev[EV_MMU], ev[EV_MLAMBDA]);
      d.ext_thresh = (int) ceil(((c.filtersc + kLog2 * invP + 3.0) * q.scale_b) + q.base_b + q.tec_b + d.tjb_b);
      d.flags = 1;
    } else {
      // p7_SSVFilter_BATH recomputes null1 for the ORF and inverts F1 (msvfilter.c:302-314)
      const float invP = gumbel_invsurv(opt.F1, ev[EV_MMU], ev[EV_MLAMBDA]);
      d.ssv_thresh = (uint8_t) (int) ceil(((c.nullsc + (invP * kLog2) + 3.0) * q.scale_b) + q.base_b + q.tec_b + d.tjb_b);
    }
    return d;
  };
  std::vector<int> vit_idx, ssv_idx;
  for (size_t t = 0; t < cand.size(); ++t) (cand[t].need_vit ? vit_idx : ssv_idx).push_back((int) t);
  std::vector<std::vector<OrfWin>> wins_of(cand.size());
  if (!vit_idx.empty()) {
    std::vector<bathgpu_orf> d(vit_idx.size());
    for (size_t z = 0; z < vit_idx.size(); ++z) d[z] = make_desc(cand[vit_idx[z]], true);
    std::vector<float> vsc(d.size());
    std::vector<int32_t> vst(d.size());
    int max_w = 0; for (auto &x : d) max_w += x.L / 2 + 4;
    std::vector<bathgpu_orf_window> w((size_t) max_w);
    int nw = 0;
    BE_TRY(s, BE.vit_orfs(BE.ctx, d.data(), (int) d.size(), vsc.data(), vst.data(), w.data(), max_w, &nw), "bathgpu_vit_orfs");
    for (size_t z = 0; z < vit_idx.size(); ++z) cand[vit_idx[z]].vfsc = vsc[z];
    for (int x = 0; x < nw; ++x) wins_of[vit_idx[w[x].orf]].push_back(OrfWin{ 0, w[x].n, w[x].k, w[x].length, w[x].score });
  }
  if (!ssv_idx.empty()) {
    std::vector<bathgpu_orf> d(ssv_idx.size());
    for (size_t z = 0; z < ssv_idx.size(); ++z) d[z] = make_desc(cand[ssv_idx[z]], false);
    int max_w = 0; for (auto &x : d) max_w += x.L / 2 + 4;
    std::vector<bathgpu_orf_window> w((size_t) max_w);
    int nw = 0;
    BE_TRY(s, BE.ssv_windows(BE.ctx, d.data(), (int) d.size(), w.data(), max_w, &nw), "bathgpu_ssv_windows");
    for (int x = 0; x < nw; ++x) wins_of[ssv_idx[w[x].orf]].push_back(OrfWin{ 0, w[x].n, w[x].k, w[x].length, w[x].score });
  }

  // ---- Viterbi decision, local-composition bias re-check (:1669-1718); ORFs that need a plain Viterbi re-run are batched
  std::vector<int> keep;                                  // candidate indices that go on to Forward
  std::vector<int> rerun;                                 // candidates needing p7_ViterbiFilter after the local bias raised filtersc
  {
    // per candidate: 0 = fails the Viterbi test, 1 = dropped by the local-composition re-check, 2 = needs a plain Viterbi re-run, 3 = kept.
    // Candidates are independent here (the null model is restored after each in the reference): all host cores, then the counters in order.
    std::vector<uint8_t> verdict(cand.size(), 0);
    std::vector<int> slot_of(cand.size(), -1);             // candidates whose local-composition filter score is needed -> their batch item
    parallel_chunks(cand.size(), 256, [&](size_t ta, size_t tb) {
      for (size_t t = ta; t < tb; ++t) {
        Cand &c = cand[t];
        verdict[t] = 3;
        if (c.need_vit) {
          const float seqsc = (c.vfsc - c.filtersc) / kLog2;
          c.P = gumbel_surv(seqsc, ev[EV_VMU], ev[EV_VLAMBDA]);
          if (c.P > opt.F2) { verdict[t] = 0; continue; }
        }
        if (opt.do_bias && !wins_of[t].empty()) slot_of[t] = 0;
      }
    });
    std::vector<int> bt;
    for (size_t t = 0; t < cand.size(); ++t) if (slot_of[t] == 0) { slot_of[t] = (int) bt.size(); bt.push_back((int) t); }
    if (!bt.empty()) {
      // the filter HMM of each candidate's local composition (p7_pli_ComputeLocalCompo over the nodes its windows cover), one table each
      std::vector<bathgpu_bias_item> items(bt.size());
      std::vector<float> tables(bt.size() * 2 * kKp), fsc;
      parallel_chunks(bt.size(), 64, [&](size_t za, size_t zb) {
        Background lbg = bg;
        float lcompo[kK];
        for (size_t z = za; z < zb; ++z) {
          const size_t t = (size_t) bt[z];
          const Orf &o = orfs[cand[t].orf];
          int k_max = wins_of[t][0].k, k_min = k_max - wins_of[t][0].length + 1;
          for (size_t w = 1; w < wins_of[t].size(); ++w) {
            k_max = std::max(k_max, wins_of[t][w].k);
            k_min = std::min(k_min, wins_of[t][w].k - wins_of[t][w].length + 1);
          }
          local_compo(m, s->compo_term.data(), k_min, k_max, lcompo);
          lbg.set_filter(M, lcompo);
          memcpy(&tables[z * 2 * kKp], &lbg.eo[0][0], sizeof(float) * 2 * kKp);
          items[z] = bathgpu_bias_item{ o.offset, o.n, (int32_t) z, Background::p1_for_length(o.n), 0 };
        }
      });
      const int rc = bias_batch(s, BE, 0, items, tables, bg, fsc, [&](size_t z, float *out) {
        std::vector<uint8_t> lbuf;
        orf_dsq(orfs[cand[(size_t) bt[z]].orf], lbuf);
        *out = Background::hmm_forward_tab(&tables[z * 2 * kKp], items[z].t00, bg.t[1][0], bg.t[1][1], lbuf.data(), items[z].L);
      });
      if (rc != 0) return rc;
      parallel_chunks(bt.size(), 1024, [&](size_t za, size_t zb) {
        Background lbg = bg;
        for (size_t z = za; z < zb; ++z) {
          const size_t t = (size_t) bt[z];
          Cand &c = cand[t];
          const Orf &o = orfs[c.orf];
          bool dropped = false, need_rerun = false;
          lbg.set_length(o.n);
          const float local_filtersc = lbg.filter_score_from(fsc[z], o.n);
          if (local_filtersc > c.filtersc) {
            c.filtersc = local_filtersc;
            if (c.vfsc == kNegInfF) {
              const float seqsc = (c.usc - c.filtersc) / kLog2;
              c.P = gumbel_surv(seqsc, ev[EV_MMU], ev[EV_MLAMBDA]);
              if (c.P > opt.F2) need_rerun = true;
            } else {
              const float seqsc = (c.vfsc - c.filtersc) / kLog2;
              c.P = gumbel_surv(seqsc, ev[EV_VMU], ev[EV_VLAMBDA]);
              if (c.P > opt.F2) dropped = true;
            }
          }
          verdict[t] = dropped ? 1 : need_rerun ? 2 : 3;
        }
      });
    }
    for (size_t t = 0; t < cand.size(); ++t) {
      if (verdict[t] == 0) { wins_of[t].clear(); continue; }
      S.st.pos_past_vit += (int64_t) orfs[cand[t].orf].n * 3;
      if (verdict[t] == 1) { wins_of[t].clear(); continue; }
      if (verdict[t] == 2) rerun.push_back((int) t); else keep.push_back((int) t);
    }
  }
  if (!rerun.empty()) {
    std::vector<bathgpu_orf> d(rerun.size());
    for (size_t z = 0; z < rerun.size(); ++z) { d[z] = make_desc(cand[rerun[z]], true); d[z].flags = 0; }
    std::vector<float> vsc(d.size());
    std::vector<int32_t> vst(d.size());
    int nw = 0;
    BE_TRY(s, BE.vit_orfs(BE.ctx, d.data(), (int) d.size(), vsc.data(), vst.data(), nullptr, 0, &nw), "bathgpu_vit_orfs");
    for (size_t z = 0; z < rerun.size(); ++z) {
      Cand &c = cand[rerun[z]];
      c.vfsc = vsc[z];
      const float seqsc = (c.vfsc - c.filtersc) / kLog2;
      c.P = gumbel_surv(seqsc, ev[EV_VMU], ev[EV_VLAMBDA]);
      if (c.P > opt.F2) wins_of[rerun[z]].clear(); else keep.push_back(rerun[z]);
    }
    std::sort(keep.begin(), keep.end());
  }
  tm.lap(S.st.us_vit);
  if (keep.empty()) return 0;

  // ---- stage 3: protein Forward over the survivors (:1774-1789)
  {
    std::vector<bathgpu_orf> d(keep.size());
    for (size_t z = 0; z < keep.size(); ++z) d[z] = make_desc(cand[keep[z]], true);
    std::vector<float> fsc(d.size());
    std::vector<int32_t> fst(d.size());
    const float xfE[2] = { expf(q.xsc_E_move), expf(q.xsc_E_loop) };
    BE_TRY(s, BE.fwd_orfs(BE.ctx, d.data(), (int) d.size(), q.nj, xfE, fsc.data(), fst.data()), "bathgpu_fwd_orfs");
    for (size_t z = 0; z < keep.size(); ++z) {
      const Cand &c = cand[keep[z]];
      const float seqsc = (fsc[z] - c.filtersc) / kLog2;
      S.P_orf[c.orf] = exp_surv(seqsc, ev[EV_FTAU], ev[EV_FLAMBDA]);
      S.fwdsc_orf[c.orf] = fsc[z] - c.nullsc;
      for (const OrfWin &w : wins_of[keep[z]]) { OrfWin x = w; x.id = S.orfs[c.orf].local_idx; S.wins_of_orf[c.orf].push_back(x); }
    }
  }

  tm.lap(S.st.us_fwd);
  return 0;
}

// positions in the accumulated hit_windows list of the entries stamped with each ORF index, in list order: the reference
// scans the whole list for an index (and the list is never reset, so earlier blocks' entries with the same index count too)
typedef std::vector<std::vector<int>> HitIndex;

// p7_pli_BuildDNAWindows (src/p7_pipeline.c:462-572) for one block-strand, against the accumulated hit_windows list.
// The ORF's window_idx mirrors orfsq->idx, stale values included: BuildDNAWindows leaves the pre-merge rank there (:545), and its
// merge loop then stamps "orf_block->list[i].idx = new_hit_cnt" on the ORF whose BLOCK RANK equals the window index i (:569) --
// p7_pli_Frameshift's standard-translation loop (:1484) reads idx of every ORF, also of those no window of the loop touched yet.
void build_dna_windows(bathhost_search *s, Unit &S, const BlockInfo &blk, int b, const std::vector<OrfWin> &hit_windows, const HitIndex &by_id)
{
  const ProteinProfile &q = s->model->prot;
  const Options &opt = s->opt;
  const int M = q.M;
  std::vector<DnaWin> dwin;
  for (int gi = S.ob(b); gi < S.ob(b + 1); ++gi) {
    const int f = S.orfs[gi].local_idx;
    if (S.P_orf[gi] > opt.F4) continue;
    Orf &o = S.orfs[gi];
    int best = -1; float best_score = kNegInfF;
    static const std::vector<int> kNone;
    for (int w : (f < (int) by_id.size() ? by_id[f] : kNone)) {
      if (hit_windows[w].score > best_score ||
          (hit_windows[w].score == best_score && hit_windows[w].length > (best >= 0 ? hit_windows[best].length : 0))) {
        best_score = hit_windows[w].score; best = (int) w;
      }
    }
    OrfWin cw;
    if (best >= 0) cw = hit_windows[best];
    else if (o.n >= M) { cw.n = (o.n - M) / 2 + 1; cw.k = M; cw.length = M; }
    else               { cw.n = 1; cw.k = M - ((M - o.n) / 2); cw.length = o.n; }
    long long ws = cw.n - (q.max_length * (0.1 + q.prefix_lengths[cw.k - cw.length + 1])) + 1;
    long long we = cw.n + cw.length + (q.max_length * (0.1 + q.suffix_lengths[cw.k])) - 2;
    ws = std::min<long long>(0, ws);
    we = std::max<long long>(o.n, we);
    ws = std::max<long long>(1, o.start + ws * 3);       // (n - start_ref + 1) == o.start on the bottom strand
    we = std::min<long long>(blk.n, o.start + we * 3);
    dwin.push_back(DnaWin{ ws, cw.k, (int) (we - ws + 1) });
    o.window_idx = (int) dwin.size() - 1;                // curr_orf->idx = windowlist->count - 1 (:545)
  }
  if (!dwin.empty()) {
    std::stable_sort(dwin.begin(), dwin.end(), [](const DnaWin &x, const DnaWin &y) { return x.n < y.n; });
    auto stamp = [&](int rank, int idx) {                // the survivor of block b whose rank in the block is `rank`, if it survived
      int lo = S.ob(b), hi = S.ob(b + 1);
      while (lo < hi) { const int mid = (lo + hi) / 2; if (S.orfs[mid].local_idx < rank) lo = mid + 1; else hi = mid; }
      if (lo < S.ob(b + 1) && S.orfs[lo].local_idx == rank) S.orfs[lo].window_idx = idx;
    };
    size_t nh = 0;
    for (size_t i = 1; i < dwin.size(); ++i) {
      DnaWin &pw = dwin[nh];
      const DnaWin &cw = dwin[i];
      const long long ov_s = std::max(pw.n, cw.n), ov_e = std::min(pw.n + pw.length - 1, cw.n + cw.length - 1);
      const long long ov_len = ov_e - ov_s + 1;
      const long long w_s = std::min(pw.n, cw.n), w_e = std::max(pw.n + pw.length - 1, cw.n + cw.length - 1);
      const long long w_len = w_e - w_s + 1;
      if (((float) ov_len / std::min(pw.length, cw.length) > 0.0f) && w_len < (2 * (q.max_length * 3))) { pw.n = w_s; pw.length = (int) w_len; }
      else { nh++; dwin[nh] = dwin[i]; }
      stamp((int) i, (int) nh);                          // orf_block->list[i].idx = new_hit_cnt (:569)
    }
    dwin.resize(nh + 1);
  }
  for (const DnaWin &d : dwin) { S.dwin.push_back(d); S.dwin_blk.push_back(b); }
}

// run fn(backend index) on one host thread per device context; the first failure is returned
template <class F> int for_each_backend(bathhost_search *s, F &&fn)
{
  const size_t nbe = s->bes.size();
  std::vector<int> rc(nbe, 0);
  if (nbe == 1) return fn(0);
  std::vector<std::thread> th;
  for (size_t k = 1; k < nbe; ++k) th.emplace_back([&, k] { rc[k] = fn((int) k); });
  rc[0] = fn(0);
  for (auto &t : th) t.join();
  for (int r : rc) if (r != 0) return r;
  return 0;
}

void add_stats(bathhost_stats &a, const bathhost_stats &b)
{
  a.pos_past_msv += b.pos_past_msv; a.pos_past_bias += b.pos_past_bias; a.pos_past_vit += b.pos_past_vit; a.pos_past_fwd += b.pos_past_fwd;
  a.n_orfs += b.n_orfs; a.n_windows += b.n_windows; a.n_std_windows += b.n_std_windows; a.n_regions += b.n_regions;
  a.n_multidomain_regions += b.n_multidomain_regions; a.n_envelopes += b.n_envelopes;
  a.us_orfs += b.us_orfs; a.us_upload += b.us_upload; a.us_msv += b.us_msv; a.us_bias += b.us_bias; a.us_vit += b.us_vit; a.us_fwd += b.us_fwd;
  a.us_windows += b.us_windows; a.us_fs_fwd += b.us_fs_fwd; a.us_fs_domains += b.us_fs_domains; a.us_std += b.us_std; a.us_xrows += b.us_xrows;
  a.us_decode += b.us_decode; a.us_score += b.us_score;
}

// The per-length tables of the filters (filter_unit: tjb byte cost and null1 score by ORF length), grown to the longest block
void grow_length_tables(bathhost_search *s, const std::vector<BlockInfo> &blocks)
{
  const ProteinProfile &q = s->model->prot;
  int maxlen = 1;
  for (const BlockInfo &blk : blocks) maxlen = std::max(maxlen, blk.n / 3 + 1);
  const size_t have = s->tjb_tab.size();
  if (have < (size_t) maxlen + 1) {
    s->tjb_tab.resize((size_t) maxlen + 1); s->null_tab.resize((size_t) maxlen + 1);
    if (have == 0) { s->tjb_tab[0] = q.tjb_for_length(1); s->null_tab[0] = 0.0f; }
    const size_t from = std::max<size_t>(have, 1);
    parallel_chunks((size_t) maxlen + 1 - from, 4096, [&](size_t a0, size_t a1) {
      Background lbg = s->bg;
      for (size_t L = from + a0; L < from + a1; ++L) { s->tjb_tab[L] = q.tjb_for_length((int) L); lbg.set_length((int) L); s->null_tab[L] = lbg.null_one((int) L); }
    });
  }
}

// Every queued sequence, both strands.  Stage times in the statistics are summed over units (device contexts work side by side,
// so with several of them the sum exceeds the wall time).
// A target already resident for the models of a library search (bathhost_library_search): the chunks cut once with the library's
// largest context and uploaded once per device context, dealt as run_batch deals them; screen[2 c + strand] = this model's stage 1.
struct SharedTarget {
  std::vector<Chunk> chunks;
  const std::vector<ScreenOut> *screen = nullptr;
};

int run_batch(bathhost_search *s, const SharedTarget *shared = nullptr)
{
  const bathhost_model *m = s->model;
  const ProteinProfile &q = m->prot;
  const Options &opt = s->opt;
  const int M = q.M;
  const float *ev = m->hmm.evparam;
  const Background &bg = s->bg;
  std::vector<SeqRef> seqs;
  seqs.swap(s->queue);
  if (seqs.empty()) return 0;
  PhaseTrace trace;

  // ---- the reference's blocks (src/bathsearch.c:1060-1105) and the residue count as each block-strand is reached
  long long nres = s->st.nres;
  std::vector<BlockInfo> blocks = cut_blocks(seqs, q.max_length * 3, opt, nres);
  s->st.nres = nres;
  const size_t nb = blocks.size();

  std::vector<Chunk> chunks;
  if (shared) {
    chunks = shared->chunks;
    place_blocks(blocks, chunks);
  } else {
    long long total = 0;
    for (const BlockInfo &b : blocks) total += b.n;
    chunks = cut_chunks(blocks, chunk_target(s, total));
  }

  // ---- units: the two strands of a chunk live in two slots of the same device context (the bottom strand is made from the top
  // one on the device); chunks are dealt round-robin to the contexts
  std::vector<int> active;
  if (opt.top)    active.push_back(0);
  if (opt.bottom) active.push_back(1);
  std::vector<std::unique_ptr<Unit>> units(chunks.size() * 2);
  std::vector<std::vector<int>> chunks_of_be(s->bes.size());
  for (size_t c = 0; c < chunks.size(); ++c) {
    const int be = (int) (c % s->bes.size());
    const int nth = (int) chunks_of_be[(size_t) be].size();
    chunks_of_be[(size_t) be].push_back((int) c);
    for (int sidx = 0; sidx < 2; ++sidx) {
      units[2 * c + sidx].reset(new Unit());
      Unit &U = *units[2 * c + sidx];
      U.complement = (sidx == 1); U.sidx = sidx; U.chunk = (int) c; U.be = be; U.slot = 2 * nth + sidx;
      U.blk0 = chunks[c].blk0; U.blk1 = chunks[c].blk1; U.n_total = chunks[c].n;
      if (shared && shared->screen) U.pre = &(*shared->screen)[2 * c + sidx];
    }
  }
  auto unit_of = [&](size_t c, int sidx) -> Unit & { return *units[2 * c + sidx]; };
  std::vector<int> chunk_of_block(nb);
  for (size_t c = 0; c < chunks.size(); ++c) for (int b = chunks[c].blk0; b < chunks[c].blk1; ++b) chunk_of_block[(size_t) b] = (int) c;

  if (s->compo_term.empty()) s->compo_term = compo_terms(m, bg);
  grow_length_tables(s, blocks);
  // ---- stages 1-3 per unit, device contexts side by side: upload (top) / reverse complement on the device (bottom), ORFs, filters
  // (Letting searches that run at the same time take this phase one after the other -- it holds the throughput-bound translation + MSV
  // pass -- was measured and lost 5-9 % on one B200: 4.07-4.39 against 4.46-4.54 Gbp/s; a search's filter phase does not fill the device.)
  int rc = for_each_backend(s, [&](int be) -> int {
    const bathhost_backend &BE = s->bes[(size_t) be];
    HostBuf stage;                                             // concatenation buffer for chunks of several sequences
    for (int c : chunks_of_be[(size_t) be]) {
      Unit &T = unit_of((size_t) c, 0), &B = unit_of((size_t) c, 1);
      StageTimer tm0;
      if (!shared) {                                           // a library search's target is resident already
        const int st = upload_chunk(s, BE, seqs, chunks[(size_t) c], T.slot, opt.bottom ? B.slot : -1, stage);
        if (st != 0) return st;
      }
      tm0.lap(T.st.us_upload);
      for (int sidx : active) {
        Unit &S = unit_of((size_t) c, sidx);
        const int st = filter_unit(s, S, blocks);
        if (st != 0) return st;
        S.aligned.assign(S.orfs.size(), 0);
        if (!opt.fs)                                            // default pipeline: every ORF past F3 is aligned by itself (:1720-1771)
          for (size_t gi = 0; gi < S.orfs.size(); ++gi)
            if (S.P_orf[gi] <= opt.F3) { S.st.pos_past_fwd += (int64_t) S.orfs[gi].n * 3; S.stdq.push_back(Unit::StdItem{ (int) gi, -1 }); }
      }
    }
    return 0;
  });
  if (rc != 0) return rc;
  trace.mark("upload + ORFs + filters (devices)");

  // ---- DNA windows, block by block in the reference's order, against the ever-growing hit_windows list (kept across batches)
  StageTimer tm;
  std::vector<OrfWin> &hit_windows = s->hit_windows;
  HitIndex &by_id = s->by_id;
  for (size_t c = 0; c < chunks.size(); ++c)
    for (int sidx : active) { Unit &S = unit_of(c, sidx); S.dwin_begin.assign((size_t) (S.blk1 - S.blk0) + 1, 0); S.hw_count.assign((size_t) (S.blk1 - S.blk0), 0); }
  for (size_t b = 0; b < nb; ++b)
    for (int sidx : active) {
      Unit &S = unit_of((size_t) chunk_of_block[b], sidx);
      S.db((int) b) = (int) S.dwin.size();
      if (blocks[b].n >= 15 && opt.fs) {
        for (int gi = S.ob((int) b); gi < S.ob((int) b + 1); ++gi)
          for (const OrfWin &w : S.wins_of_orf[gi]) {
            if ((size_t) w.id >= by_id.size()) by_id.resize((size_t) w.id + 1);
            by_id[w.id].push_back((int) hit_windows.size());
            hit_windows.push_back(w);
          }
        S.hwc((int) b) = hit_windows.size();
        build_dna_windows(s, S, blocks[b], (int) b, hit_windows, by_id);
      } else S.hwc((int) b) = hit_windows.size();
      S.db((int) b + 1) = (int) S.dwin.size();
    }
  tm.lap(s->st.us_windows);
  trace.mark("DNA windows (host, serial)");

  // ---- stages 4-5 per unit, device contexts side by side: frameshift Forward parser over every DNA window (:1446-1450), the
  // arbitration between window and ORFs (:1392-1465), Forward + Backward X rows of the windows that stay (:1469-1470), and the
  // part of p7_DomainDecoding_Frameshift that does not depend on the length-model chain
  const float xfE3[2] = { m->om3.xfE_move, m->om3.xfE_loop };
  struct Decoded { float *btot = nullptr, *etot = nullptr, *fb = nullptr, *e0 = nullptr; };   // btot, etot, e0: [L+1]; fb: [L+1][9]; views into the unit's block
  std::vector<std::vector<Decoded>> dec(units.size());
  struct DecBlocks {                                          // one block per unit, from the process-wide pool and back to it when the batch is done
    std::vector<std::vector<float>> v;
    explicit DecBlocks(size_t n) : v(n) {}
    ~DecBlocks() { for (auto &b : v) ScratchPool::get().give(std::move(b)); }
  } dec_blocks(units.size());
  rc = for_each_backend(s, [&](int be) -> int {
    const bathhost_backend &BE = s->bes[(size_t) be];
    for (int c : chunks_of_be[(size_t) be])
      for (int sidx : active) {
        Unit &S = unit_of((size_t) c, sidx);
        StageTimer tmu;
        const int nwin = (int) S.dwin.size();
        if (nwin == 0) continue;
        S.gw.resize((size_t) nwin);
        for (int w = 0; w < nwin; ++w) {
          S.gw[w].start = S.goff(blocks[(size_t) S.dwin_blk[w]]) + S.dwin[w].n; S.gw[w].L = S.dwin[w].length;
          bathhost_length_model(S.dwin[w].length / 3, 1.0f, &S.gw[w].pmove, &S.gw[w].ploop);
        }
        S.fs_fwd.resize((size_t) nwin); S.fs_st.resize((size_t) nwin);
        BE_TRY(s, BE.select_slot(BE.ctx, S.slot), "bathgpu_select_slot");
        BE_TRY(s, BE.fs_fwd_windows(BE.ctx, S.gw.data(), nwin, xfE3, S.fs_fwd.data(), S.fs_st.data()), "bathgpu_fs_fwd_windows");
        S.st.n_windows += nwin;
        tmu.lap(S.st.us_fs_fwd);

        // arbitration per window: the scores each window needs (ORF sums, null and bias filter scores) are independent of one
        // another and computed on all host cores; the decisions are then taken in the reference's order
        {
          const int nw = nwin;
          struct WinPre { int orf_cnt, k_min, k_max; double P_tot, P_min; float nullsc, filtersc; };
          std::vector<WinPre> pre((size_t) nw);
          auto inside_of = [&](const Orf &o, const DnaWin &dw) {
            return S.complement ? (o.start >= dw.n && o.end <= dw.n + dw.length + 1) : (o.start >= dw.n && o.end <= dw.n + dw.length - 1);
          };
          const std::vector<OrfWin> &hit_windows = s->hit_windows;
          const HitIndex &by_id = s->by_id;
          parallel_chunks((size_t) nw, 1, [&](size_t wa, size_t wb) {
            Background lbg = bg;
            for (size_t w = wa; w < wb; ++w) {
              const int b = S.dwin_blk[w];
              const DnaWin &dw = S.dwin[w];
              int orf_cnt = 0, k_min = M, k_max = 0;
              float tot_orfsc = kNegInfF;
              double P_min = std::numeric_limits<double>::infinity();
              size_t last_h = 0;
              const size_t hw_n = S.hwc(b);
              for (int gi = S.ob(b); gi < S.ob(b + 1); ++gi) {
                if (S.P_orf[gi] > opt.F4) continue;
                const Orf &o = S.orfs[gi];
                const int i = o.local_idx;
                if (!inside_of(o, dw)) continue;
                P_min = std::min(P_min, S.P_orf[gi]);
                tot_orfsc = flogsum(tot_orfsc, S.fwdsc_orf[gi]);
                orf_cnt++;
                size_t h = last_h;
                if ((size_t) i < by_id.size()) {                 // first entry stamped i at or after last_h (the reference scans forward for it)
                  const std::vector<int> &ix = by_id[i];
                  auto it = std::lower_bound(ix.begin(), ix.end(), (int) h);
                  h = (it == ix.end()) ? hw_n : std::min<size_t>(hw_n, (size_t) *it);
                } else h = hw_n;
                if (h < hw_n) {
                  while (h < hw_n && hit_windows[h].id == i) {
                    k_min = std::min(k_min, hit_windows[h].k - hit_windows[h].length + 1);
                    k_max = std::max(k_max, hit_windows[h].k);
                    h++;
                  }
                  last_h = h;
                }
              }
              WinPre &r = pre[w];
              r.orf_cnt = orf_cnt; r.P_min = P_min; r.k_min = k_min; r.k_max = k_max;
              r.P_tot = exp_surv(tot_orfsc / kLog2, ev[EV_FTAU], ev[EV_FLAMBDA]);
              lbg.set_length(dw.length / 3);
              r.nullsc = lbg.fs_null_one(dw.length / 3);
              r.filtersc = r.nullsc;
            }
          });
          if (opt.do_bias) {
            // p7_bg_fs_FilterScore of every window under the model composition, and under the local composition of the nodes its
            // ORFs' filter windows cover where there are any (:1432-1440): one batch, three frames per item
            std::vector<int> item_win, first_item((size_t) nw + 1, 0);
            for (int w = 0; w < nw; ++w) {
              first_item[(size_t) w] = (int) item_win.size();
              item_win.push_back(w);
              if (pre[(size_t) w].k_min <= pre[(size_t) w].k_max) item_win.push_back(w);
            }
            first_item[(size_t) nw] = (int) item_win.size();
            std::vector<bathgpu_bias_item> items(item_win.size());
            std::vector<float> tables((item_win.size() - (size_t) nw + 1) * 2 * kKp), fsc;
            {
              Background lbg = bg;
              lbg.set_filter(M, s->compo.data());
              memcpy(tables.data(), &lbg.eo[0][0], sizeof(float) * 2 * kKp);
              int ntab = 1;
              for (int w = 0; w < nw; ++w) {
                const float t00 = Background::p1_for_length(S.dwin[(size_t) w].length / 3);
                const int z = first_item[(size_t) w];
                items[(size_t) z] = bathgpu_bias_item{ S.gw[(size_t) w].start, S.dwin[(size_t) w].length, 0, t00, 0 };
                if (first_item[(size_t) w + 1] - z == 2) items[(size_t) z + 1] = bathgpu_bias_item{ S.gw[(size_t) w].start, S.dwin[(size_t) w].length, ntab++, t00, 0 };
              }
            }
            parallel_chunks((size_t) nw, 8, [&](size_t wa, size_t wb) {
              Background lbg = bg;
              float lcompo[kK];
              for (size_t w = wa; w < wb; ++w) {
                if (first_item[w + 1] - first_item[w] != 2) continue;
                local_compo(m, s->compo_term.data(), pre[w].k_min, pre[w].k_max, lcompo);
                lbg.set_filter(M, lcompo);
                memcpy(&tables[(size_t) items[(size_t) first_item[w] + 1].table * 2 * kKp], &lbg.eo[0][0], sizeof(float) * 2 * kKp);
              }
            });
            const int rcb = bias_batch(s, BE, 1, items, tables, bg, fsc, [&](size_t z, float *out) {
              const int w = item_win[z];
              const BlockInfo &blk = blocks[(size_t) S.dwin_blk[(size_t) w]];
              const DnaWin &dw = S.dwin[(size_t) w];
              std::vector<uint8_t> wbuf, orf((size_t) dw.length + 2);
              const uint8_t *wdsq = oriented(seqs[(size_t) blk.seq], blk, S.complement, dw.n - 1, dw.length, wbuf);        // window position p is wdsq[p]
              for (int fr = 1; fr <= 3; ++fr)
                out[fr - 1] = Background::hmm_forward_tab(&tables[(size_t) items[z].table * 2 * kKp], items[z].t00, bg.t[1][0], bg.t[1][1], orf.data(),
                                                          Background::frame_residues(wdsq, dw.length, fr, s->gcode, orf.data()));
            });
            if (rcb != 0) return rcb;
            Background lbg = bg;
            for (int w = 0; w < nw; ++w) {
              WinPre &r = pre[(size_t) w];
              const int L = S.dwin[(size_t) w].length;
              lbg.set_length(L / 3);
              for (int z = first_item[(size_t) w]; z < first_item[(size_t) w + 1]; ++z) {
                const float f = lbg.fs_filter_score_from(&fsc[(size_t) z * 3], L);
                if (z == first_item[(size_t) w] || f > r.filtersc) r.filtersc = f;
              }
            }
          }
          for (int w = 0; w < nw; ++w) {
            const int b = S.dwin_blk[w];
            const int wl = w - S.db(b);                         // the window's index in its block's list: what orfsq->idx holds
            const DnaWin &dw = S.dwin[w];
            const WinPre &r = pre[w];
            for (int gi = S.ob(b); gi < S.ob(b + 1); ++gi)
              if (S.P_orf[gi] <= opt.F4 && inside_of(S.orfs[gi], dw)) S.orfs[gi].window_idx = wl;
            const float fwdsc = S.fs_fwd[w];                      // on eslERANGE the score is -inf or NaN and the tests below fail, as in the reference
            const float seqscore = (fwdsc - r.filtersc) / kLog2;
            const double P_fs   = exp_surv(seqscore, ev[EV_FTAUFS3], ev[EV_FLAMBDA]);
            const double P_null = exp_surv((fwdsc - r.nullsc) / kLog2, ev[EV_FTAUFS3], ev[EV_FLAMBDA]);
            if (S.fs_st[w] == 0 && P_fs <= opt.F3 && (P_null < r.P_tot || (P_null == r.P_tot && r.orf_cnt > 1) || r.P_min > opt.F3)) {
              S.st.pos_past_fwd += dw.length;
              S.fsw.push_back(w);
            } else {                                              // standard-translation branch (:1480-1511)
              S.st.n_std_windows++;
              for (int gi = S.ob(b); gi < S.ob(b + 1); ++gi) {
                if (S.orfs[gi].window_idx != wl || S.P_orf[gi] > opt.F3 || S.aligned[gi]) continue;
                S.st.pos_past_fwd += (int64_t) S.orfs[gi].n * 3;
                S.aligned[gi] = 1;
                S.stdq.push_back(Unit::StdItem{ gi, w });
              }
            }
          }
        }
        tmu.lap(S.st.us_bias);

        // Forward (X rows kept) + Backward parsers over the frameshift-branch windows
        if (S.fsw.empty()) continue;
        std::vector<bathgpu_window> gf(S.fsw.size());
        S.xoff.assign(S.fsw.size() + 1, 0);
        for (size_t z = 0; z < S.fsw.size(); ++z) { gf[z] = S.gw[S.fsw[z]]; S.xoff[z + 1] = S.xoff[z] + (size_t) gf[z].L + 1; }
        // the X rows are consumed by the precomputation just below: one pair of page-locked buffers per device context serves all its units
        S.fxr = s->be_xbuf[(size_t) be][0].get(BE, S.xoff.back() * 6); S.bxr = s->be_xbuf[(size_t) be][1].get(BE, S.xoff.back() * 6); S.st2.resize(S.fsw.size());
        if (!S.fxr || !S.bxr) return fail(s, BATHHOST_EMEM, "host allocation failed");
        std::vector<float> f2(S.fsw.size()), b2(S.fsw.size());
        BE_TRY(s, BE.fs_fwd_bck_xrows(BE.ctx, gf.data(), (int) gf.size(), xfE3, S.fxr, S.bxr, f2.data(), b2.data(), S.st2.data()),
               "bathgpu_fs_fwd_bck_xrows");
        tmu.lap(S.st.us_xrows);

        // The transcendental part of p7_DomainDecoding_Frameshift does not depend on the length model the walk below chains from
        // window to window: it is precomputed for all windows on all host cores (cumulative log scales, Z, the btot/etot sums,
        // the nine forward x backward products and their scale factors per row)
        std::vector<Decoded> &DV = dec[(size_t) (2 * c + sidx)];
        DV.resize(S.fsw.size());
        {
          std::vector<float> &blk = dec_blocks.v[(size_t) (2 * c + sidx)];
          blk = ScratchPool::get().take(S.xoff.back() * 12);
          blk.resize(S.xoff.back() * 12);
          for (size_t z = 0; z < S.fsw.size(); ++z) {
            float *base = blk.data() + S.xoff[z] * 12;
            const size_t rows = S.xoff[z + 1] - S.xoff[z];     // Lw + 1
            DV[z].btot = base; DV[z].etot = base + rows; DV[z].fb = base + 2 * rows; DV[z].e0 = base + 11 * rows;
          }
        }
        // Per row i the reference multiplies three forward x backward products per special state by the scale factors
        // exp(lsf[i-3+o] + lsb[i+o] + liz), o = 0, 1, 2 (decoding_fs.c:309-352).  The factor of offset o at row i is the factor of offset 0
        // at row i+o -- the same expression on the same floats -- so one exponential per row is kept (e0) and read at i, i+1, i+2; the
        // btot / etot sums share theirs the same way (x[i] = exp(lsf[i] + lsb[i] + liz) serves etot[i] and btot[i+3]).  Entries the
        // walk never reads (rows below 3, offsets past the window end) are left unwritten.
        parallel_chunks(S.fsw.size(), 1, [&](size_t za, size_t zb) {
          std::vector<float> lsf, lsb, xd;
          for (size_t z = za; z < zb; ++z) {
            if (S.st2[z] != 0) continue;
            const int Lw = S.dwin[S.fsw[z]].length;
            const float *xf = S.fxr + S.xoff[z] * 6, *xb = S.bxr + S.xoff[z] * 6;
            Decoded &D = DV[z];
            lsf.resize((size_t) Lw + 2); lsb.resize((size_t) Lw + 2); xd.resize((size_t) Lw + 1);
            lsf[0] = logf(xf[5]);
            for (int i = 1; i <= Lw; ++i) lsf[i] = lsf[i - 1] + logf(xf[(size_t) i * 6 + 5]);
            lsb[Lw + 1] = 0.0f;
            for (int i = Lw; i >= 0; --i) lsb[i] = lsb[i + 1] + logf(xb[(size_t) i * 6 + 5]);
            const float liz = -flogsum(logf(xb[0 * 6 + 1]) + lsb[0], flogsum(logf(xb[1 * 6 + 1]) + lsb[1], logf(xb[2 * 6 + 1]) + lsb[2]));
            auto F = [&](int i, int cc) { return xf[(size_t) i * 6 + cc]; };
            auto B = [&](int i, int cc) { return xb[(size_t) i * 6 + cc]; };
            static const int cells[3] = { 1, 2, 4 };          // N, J, C
            for (int i = 0; i <= Lw; ++i) xd[i] = expf(lsf[i] + lsb[i] + liz);
            for (int i = 0; i < 3 && i <= Lw; ++i) { D.btot[i] = 0.f; D.etot[i] = 0.f; D.e0[i] = 0.f; }
            for (int i = 3; i <= Lw; ++i) {
              D.btot[i] = D.btot[i - 3] + F(i - 3, 3) * B(i - 3, 3) * xd[i - 3];
              D.etot[i] = D.etot[i - 3] + F(i, 0) * B(i, 0) * xd[i];
              D.e0[i] = expf(lsf[i - 3] + lsb[i] + liz);
              for (int cc = 0; cc < 3; ++cc) {
                float *fb = &D.fb[(size_t) i * 9 + 3 * cc];
                fb[0] = F(i - 3, cells[cc]) * B(i, cells[cc]);
                if (i < Lw)     fb[1] = F(i - 2, cells[cc]) * B(i + 1, cells[cc]);
                if (i < Lw - 1) fb[2] = F(i - 1, cells[cc]) * B(i + 2, cells[cc]);
              }
            }
          }
        });
        tmu.lap(S.st.us_decode);
      }
    return 0;
  });
  if (rc != 0) return rc;
  trace.mark("fs Forward, arbitration, X rows");
  tm = StageTimer();

  // ---- domain decoding and region finding on the host, in the reference's order (block, then strand, then window):
  // the length model of om_fs5 that p7_DomainDecoding_Frameshift reads is whatever the previous window's rescoring left
  // (src/p7_domaindef.c:320-325, :1018); the walk below only applies its loop odds to the precomputed products, in the
  // reference's operation order.
  const float rt1 = 0.25f, rt2 = 0.10f, rt3 = 0.20f;
  const uint32_t kStotraceSeed = 42; const int kStotraceSamples = 200;   // --seed default (src/bathsearch.c:131), ddef->nsamples (src/p7_domaindef.c:83)
  const int saveL = 100;                                    // gm_fs5->L: the dummy length bathsearch configures and never changes (src/bathsearch.c:797)
  // Multi-domain regions (is_multidomain_region_frameshift) are split by stochastic-trace clustering (src/p7_domaindef.c:395-453).
  // Their envelopes feed the length-model chain like any other, so the walk cannot simply skip them: it runs once with every
  // unresolved multi-domain region taken as one envelope, the Forward matrices of those regions are then filled on the device in
  // one batch and sampled and clustered here on all cores, and the walk is repeated with the clusters in place -- until it meets
  // no unresolved region (two passes unless a changed length model moves a later region's borders).
  struct RegionKey { int u, w, i, j; bool operator<(const RegionKey &o) const { return std::tie(u, w, i, j) < std::tie(o.u, o.w, o.i, o.j); } };   // u: unit
  std::map<RegionKey, std::vector<std::pair<int, int>>> resolved;
  const float walk_nj0 = s->om5_nj; const int walk_L0 = s->om5_L;
  const int64_t walk_regions0 = s->st.n_regions, walk_multi0 = s->st.n_multidomain_regions;
  // What a window's walk produces is a function of the length model it starts from (it enters only through the loop odds of the
  // decoding) and of the clusters known so far: envelopes, the length model it leaves behind, counters, unresolved regions.
  // That makes the chain speculative-parallel: every window is walked on all cores from a guessed input, the outputs are
  // chained, and whatever started from a wrong input is walked again -- until every window has been walked from the state its
  // predecessor really leaves, which is the sequential result.  Region borders hardly ever move with the loop odds, so this
  // settles in two or three rounds.
  struct WalkMemo { bool valid = false; float nj_in = 0, nj_out = 0; int L_in = 0, L_out = 0, nreg = 0, nmulti = 0;
                    std::vector<bathgpu_envelope> ge; std::vector<Unit::Env> envs; std::vector<RegionKey> pend; };
  std::vector<std::vector<WalkMemo>> memo(units.size());
  for (size_t u = 0; u < units.size(); ++u) memo[u].resize(units[u]->fsw.size());
  struct WalkItem { int u; size_t z; };
  std::vector<WalkItem> worder;                               // the reference's order: block, then strand, then window
  {
    std::vector<size_t> zpos(units.size(), 0);
    for (size_t b = 0; b < nb; ++b)
      for (int sidx : active) {
        const int u = 2 * chunk_of_block[b] + sidx;
        Unit &S = *units[(size_t) u];
        for (; zpos[u] < S.fsw.size() && S.dwin_blk[S.fsw[zpos[u]]] == (int) b; ++zpos[u])
          if (S.st2[zpos[u]] == 0) worder.push_back(WalkItem{ u, zpos[u] });   // backward underflow: no domain definition (:1471)
      }
  }
  auto walk_window = [&](int sidx, size_t z, float nj_in, int L_in, WalkMemo &wm) {      // sidx: the unit
    Unit &S = *units[(size_t) sidx];
    wm.valid = true; wm.nj_in = nj_in; wm.L_in = L_in; wm.nreg = 0; wm.nmulti = 0;
    wm.ge.clear(); wm.envs.clear(); wm.pend.clear();
    float om5_nj = nj_in; int om5_L = L_in;
          const int w = S.fsw[z];
          const int Lw = S.dwin[w].length;
          const float tL = 1.0f - (2.0f + om5_nj) / ((float) om5_L + 2.0f + om5_nj);
          // mocc[i] = 1 - sum over N,J,C and the three codon offsets of fwd * bck * loop odds * scale (decoding_fs.c:309-352)
          const Decoded &D = dec[(size_t) sidx][z];
          const float *btot = D.btot, *etot = D.etot;
          std::vector<float> mocc((size_t) Lw + 1, 0.f);
          for (int i = 3; i <= Lw; ++i) {
            float njcp = 0.;
            const float *fb = &D.fb[(size_t) i * 9], *e0 = &D.e0[i];       // e0[o]: the scale factor of codon offset o at this row
            for (int c = 0; c < 3; ++c) {
              njcp += fb[3 * c] * tL * e0[0];
              if (i < Lw)     njcp += fb[3 * c + 1] * tL * e0[1];
              if (i < Lw - 1) njcp += fb[3 * c + 2] * tL * e0[2];
            }
            mocc[i] = 1. - njcp;
          }
          om5_nj = 0.0f; om5_L = saveL / 3;                 // p7_fs_oprofile_ReconfigUnihit(om_fs5, saveL/3) (:325)
          // region finding (src/p7_domaindef.c:332-383)
          int i = -1, d = 0; bool triggered = false, start = false, end = false;
          for (int j = 1; j < Lw; ++j) {
            if (!triggered) { if (mocc[j] >= rt1) triggered = true; d = j; }
            else {
              while (d > 1 && !start) {
                d--;
                if (d > 3 && mocc[d] - (btot[d] - btot[d - 3]) < rt2) { d--;
                  if (d > 3 && mocc[d] - (btot[d] - btot[d - 3]) < rt2) { d--;
                    if (d > 3 && mocc[d] - (btot[d] - btot[d - 3]) < rt2) { d--; start = true; } } }
              }
              i = std::max(1, d - 3);
              d = j + 1;
              while (d < Lw && !end) {
                d++;
                if (d < Lw && mocc[d] - (etot[d] - etot[d - 3]) < rt2) { d++;
                  if (d < Lw && mocc[d] - (etot[d] - etot[d - 3]) < rt2) { d++;
                    if (d < Lw && mocc[d] - (etot[d] - etot[d - 3]) < rt2) { d++; end = true; } } }
              }
              j = std::min(Lw, d + 3);
              if (j - i + 1 >= 12) {
                wm.nreg++;
                float mx = -1.0f;                           // is_multidomain_region_frameshift (:684-714)
                auto scan = [&](int z0, int eoff, int f) {
                  for (int zz = z0; zz <= j - f; zz += 3) {
                    const float en = std::min(etot[zz] - etot[i + eoff], btot[j - f] - btot[zz - 3]);
                    mx = std::max(mx, en);
                  }
                };
                scan(i + 2, -1, (j - i + 1) % 3);
                scan(i + 3, 0, (j - i) % 3);
                scan(i + 4, 1, (j - i - 1) % 3);
                auto envelope = [&](int i2, int j2) {
                  const int Ld = j2 - i2 + 1;
                  if (Ld < 15) return;                       // rescore_isolated_domain_frameshift returns at once below 15 (:1012)
                  bathgpu_envelope g;
                  g.start = S.gw[w].start + i2 - 1; g.L = Ld;
                  bathhost_length_model(Ld / 3, 0.0f, &g.pmove, &g.ploop);
                  wm.ge.push_back(g); wm.envs.push_back(Unit::Env{ w, i2, j2 });
                  om5_nj = 0.0f; om5_L = Ld / 3;             // p7_fs_oprofile_ReconfigLength(om_fs5, Ld/3) (:1018)
                };
                const std::vector<std::pair<int, int>> *clusters = nullptr;
                if (mx >= rt3) {
                  wm.nmulti++;
                  const RegionKey key{ sidx, w, i, j };
                  auto it = resolved.find(key);
                  if (it != resolved.end()) clusters = &it->second; else wm.pend.push_back(key);
                }
                if (clusters) {
                  om5_nj = 0.0f; om5_L = saveL;              // ReconfigMultihit(saveL) .. ReconfigUnihit(om_fs5, saveL) (:409,:417)
                  for (const auto &c2 : *clusters) envelope(std::max(1, c2.first), c2.second);      // (:421-445)
                } else envelope(i, j);
              }
              i = -1; triggered = false; start = false; end = false;
            }
          }
    wm.nj_out = om5_nj; wm.L_out = om5_L;
  };
  static const bool walk_sequential = getenv("BATHHOST_SEQUENTIAL_WALK") != nullptr;
  for (int walk_pass = 0; ; ++walk_pass) {
    for (int round = 0; ; ++round) {
      std::vector<size_t> todo;
      float nj = walk_nj0; int L = walk_L0;
      for (size_t t = 0; t < worder.size(); ++t) {
        WalkMemo &wm = memo[(size_t) worder[t].u][worder[t].z];
        if (!wm.valid || wm.nj_in != nj || wm.L_in != L) { todo.push_back(t); wm.nj_in = nj; wm.L_in = L; }
        if (wm.valid) { nj = wm.nj_out; L = wm.L_out; } else { nj = 0.0f; L = saveL / 3; }   // first round: a guess for the successor
      }
      if (todo.empty()) break;
      if (trace.on) fprintf(stderr, "[bathhost]   walk pass %d round %d: %zu of %zu windows\n", walk_pass, round, todo.size(), worder.size());
      if (walk_sequential) todo.resize(1);                    // test hook: one window per round from its true input = the plain sequential walk
      if (round > (int) worder.size() + 2) return fail(s, BATHHOST_EINVAL, "the region walk does not settle");
      // Inside a piece of consecutive windows the chain is followed for real: a window starts from what its predecessor in the piece
      // has just left, so only the first window of a piece runs on a guess (the walk is bound by reading the decoding products,
      // 72 bytes per window row: walking nearly every window twice cost 10-34 ms per Gbp and profile).
      parallel_chunks(todo.size(), 4, [&](size_t ta, size_t tb) {
        for (size_t q = ta; q < tb; ++q) {
          const WalkItem &it = worder[todo[q]];
          WalkMemo &wm = memo[(size_t) it.u][it.z];
          if (q > ta && todo[q] == todo[q - 1] + 1) {
            const WalkItem &pit = worder[todo[q - 1]];
            const WalkMemo &pm = memo[(size_t) pit.u][pit.z];
            wm.nj_in = pm.nj_out; wm.L_in = pm.L_out;
          }
          walk_window(it.u, it.z, wm.nj_in, wm.L_in, wm);
        }
      });
    }
    trace.mark("  walk: rounds");
    std::vector<RegionKey> pending;
    for (const WalkItem &it : worder) { const WalkMemo &wm = memo[(size_t) it.u][it.z]; pending.insert(pending.end(), wm.pend.begin(), wm.pend.end()); }
    for (const WalkItem &it : worder) { WalkMemo &wm = memo[(size_t) it.u][it.z]; if (!wm.pend.empty()) wm.valid = false; }   // walked again once resolved
    if (pending.empty()) break;
    if (walk_pass > 64) return fail(s, BATHHOST_EINVAL, "multi-domain region resolution does not settle");
    // ---- Forward matrices of the unresolved regions (multihit, target length saveL: :409-412): one device call per unit that has any,
    // the device contexts side by side, then every region of every unit sampled and clustered on all cores at once (regions of this
    // kind are rare -- 10-20 per Gbp and profile -- but each costs a device call and 200 sampled traces, and they came one unit after
    // the other: 17-36 ms of a 110-150 ms profile on eight GPUs)
    const float xfE5m[2] = { 0.5f, 0.5f };
    float mh_pmove, mh_ploop;
    bathhost_length_model(saveL, 1.0f, &mh_pmove, &mh_ploop);
    struct UnitRegions { std::vector<bathgpu_envelope> regs; std::vector<RegionKey> keys; std::vector<int64_t> off; std::vector<float> fsc;
                         std::vector<int32_t> fst; HostBuf mx, xr; float *mxbuf = nullptr, *xrbuf = nullptr; };
    std::vector<UnitRegions> ur(units.size());
    for (const RegionKey &k : pending) {
      Unit &S = *units[(size_t) k.u];
      UnitRegions &R = ur[(size_t) k.u];
      if (R.off.empty()) R.off.push_back(0);
      bathgpu_envelope g;
      g.start = S.gw[k.w].start + k.i - 1; g.L = k.j - k.i + 1; g.pmove = mh_pmove; g.ploop = mh_ploop;
      R.regs.push_back(g); R.keys.push_back(k); R.off.push_back(R.off.back() + g.L + 1);
    }
    rc = for_each_backend(s, [&](int be) -> int {
      const bathhost_backend &BE = s->bes[(size_t) be];
      for (size_t sidx = 0; sidx < units.size(); ++sidx) {
        if (!units[sidx] || units[sidx]->be != be || ur[sidx].regs.empty()) continue;
        Unit &S = *units[sidx];
        UnitRegions &R = ur[sidx];
        R.mxbuf = R.mx.get(BE, (size_t) R.off.back() * (M + 1) * 8); R.xrbuf = R.xr.get(BE, (size_t) R.off.back() * 6);
        if (!R.mxbuf || !R.xrbuf) return fail(s, BATHHOST_EMEM, "host allocation failed");
        R.fsc.resize(R.regs.size()); R.fst.resize(R.regs.size());
        BE_TRY(s, BE.select_slot(BE.ctx, S.slot), "bathgpu_select_slot");
        if (!BE.fs_forward_matrices) return fail(s, BATHHOST_EINVAL, "the device library has no bathgpu_fs_forward_matrices");
        BE_TRY(s, BE.fs_forward_matrices(BE.ctx, R.regs.data(), (int) R.regs.size(), xfE5m, R.mxbuf, R.xrbuf, R.off.back(), R.fsc.data(), R.fst.data()),
               "bathgpu_fs_forward_matrices");
      }
      return 0;
    });
    if (rc != 0) return rc;
    trace.mark("  walk: region matrices (devices)");
    struct RegionRef { size_t u, r; };
    std::vector<RegionRef> all;
    for (size_t u = 0; u < ur.size(); ++u) for (size_t r = 0; r < ur[u].regs.size(); ++r) all.push_back(RegionRef{ u, r });
    std::vector<std::vector<std::pair<int, int>>> found(all.size());
    const SpecialOdds X{ mh_pmove, mh_ploop, xfE5m[0], xfE5m[1] };
    parallel_chunks(all.size(), 1, [&](size_t ra, size_t rb) {
      for (size_t q = ra; q < rb; ++q) {
        const UnitRegions &R = ur[all[q].u];
        const size_t r = all[q].r;
        if (R.fst[r] != 0) continue;                         // Forward out of range: no clusters (:412-413)
        const ForwardMatrix F{ R.mxbuf + (size_t) R.off[r] * (M + 1) * 8, R.xrbuf + (size_t) R.off[r] * 6, M, R.regs[r].L };
        std::vector<Segment> sp;
        if (!sample_region_segments(F, m->om5.tfv.data(), X, kStotraceSeed, kStotraceSamples, R.keys[r].i, sp)) continue;
        for (const Segment &g : cluster_region_segments(sp, kStotraceSamples)) found[q].push_back({ g.i, g.j });
      }
    });
    for (size_t q = 0; q < all.size(); ++q) resolved[ur[all[q].u].keys[all[q].r]] = std::move(found[q]);
    trace.mark("  walk: sampling + clustering");
  }
  s->st.n_regions = walk_regions0; s->st.n_multidomain_regions = walk_multi0;
  for (auto &U : units) { U->ge.clear(); U->envs.clear(); }
  for (const WalkItem &it : worder) {
    const WalkMemo &wm = memo[(size_t) it.u][it.z];
    Unit &S = *units[(size_t) it.u];
    S.ge.insert(S.ge.end(), wm.ge.begin(), wm.ge.end()); S.envs.insert(S.envs.end(), wm.envs.begin(), wm.envs.end());
    s->st.n_regions += wm.nreg; s->st.n_multidomain_regions += wm.nmulti;
    s->om5_nj = wm.nj_out; s->om5_L = wm.L_out;
  }
  tm.lap(s->st.us_windows);
  trace.mark("region walk (host)");

  // ---- stage 6 and everything after it, per unit, device contexts side by side: every envelope of the unit rescored in one
  // batched call (rescore_isolated_domain_frameshift, :993-1191), scoring and hit records, then the standard-translation branch
  const float xfE5[2] = { 1.0f, 0.0f };
  auto finish_unit = [&](Unit &S) -> int {
    const bathhost_backend &BE = s->bes[(size_t) S.be];
    const int sidx = S.sidx;
    StageTimer tm;
  if (!S.ge.empty()) {
    S.res.resize(S.ge.size());
    int64_t max_steps = 0; for (auto &g : S.ge) max_steps += g.L + M + 8;
    S.traces.resize((size_t) max_steps);
    BE_TRY(s, BE.select_slot(BE.ctx, S.slot), "bathgpu_select_slot");
    BE_TRY(s, BE.fs_domains(BE.ctx, S.ge.data(), (int) S.ge.size(), xfE5, S.res.data(), S.traces.data(), max_steps), "bathgpu_fs_domains");
    S.st.n_envelopes += (int64_t) S.ge.size();
  }
  tm.lap(S.st.us_fs_domains);
  // ---- scoring and hit records: envelopes are independent of one another (the early E-value cut uses the residue count fixed
  // for their block), so they are scored on all host cores and the hits kept in the reference's order
  {
    struct Item { size_t e; size_t b; };
    std::vector<Item> order;
    for (size_t e = 0; e < S.envs.size(); ++e) order.push_back(Item{ e, (size_t) S.dwin_blk[S.envs[e].win] });
    auto score_env = [&](const Item &it, Background &lbg, std::vector<uint8_t> &wbuf, Hit &h) -> bool {
      const size_t e = it.e, b = it.b;
      const std::vector<bathgpu_domain_result> &res = S.res;
      const std::vector<bathgpu_trace_step> &traces = S.traces;
          const BlockInfo &binfo = blocks[b];
          const DnaWin &dw = S.dwin[S.envs[e].win];
          const SeqRef &sq = seqs[(size_t) binfo.seq];
          const uint8_t *wdsq = oriented(sq, binfo, S.complement, dw.n - 1, dw.length, wbuf);
          const int Lw = dw.length;
          const long long nres_now = binfo.nres_at[sidx];
          struct { bool complement; long long start; const char *name; long long sq_len; } blk = { S.complement, S.start_of(binfo), sq.name.c_str(), (long long) sq.n };
          const int i = S.envs[e].i, j = S.envs[e].j, Ld = S.ge[e].L;
        const bathgpu_domain_result &r = res[e];
        if (r.status != 0 && r.trace_len == 0) return false;   // Forward/Backward range error: envelope dropped (:1022,1041)
        lbg.set_length(Ld / 3);
        const float env_null = lbg.fs_null_one(Ld / 3);
        const float seqsc = (r.envsc - env_null) / kLog2;
        const double P = exp_surv(seqsc, ev[EV_FTAUFS5], ev[EV_FLAMBDA]);
        const double Z = (float) nres_now / (float) q.max_length;
        if (P * Z > opt.E) return false;                         // early cut on the residues seen so far (:1033-1037)
        if (r.status != 0) return false;

        Domain dom;
        dom.tr.assign(traces.begin() + r.trace_offset, traces.begin() + r.trace_offset + r.trace_len);
        for (auto &ts : dom.tr) ts.i += i - 1;               // window coordinates (:1050-1051; every i >= 0 is shifted)
        const float aliscore = ali_score(m, dom.tr, wdsq);
        if (aliscore < 0.0f) return false;

        // null2 correction along the trace (:1084-1142)
        float domcorrection = 0.0f;
        {
          std::vector<float> n2((size_t) Lw + 2, 0.0f);
          int t5 = -1, u5 = -1, v5 = -1, w5 = -1, x5 = -1;
          size_t z = 0;
          int pos = i;
          auto cidx = [&](int c) {
            long long ci;
            if (c == 1)      { ci = (long long) x5 * 341;                                              return (int) std::min<long long>(ci, 1366); }
            else if (c == 2) { ci = (long long) x5 * 341 + w5 * 85 + 1;                                return (int) std::min<long long>(ci, 1365); }
            else if (c == 3) { ci = (long long) x5 * 341 + w5 * 85 + v5 * 21 + 2;                      return (int) std::min<long long>(ci, 1364); }
            else if (c == 4) { ci = (long long) x5 * 341 + w5 * 85 + v5 * 21 + u5 * 5 + 3;             return (int) std::min<long long>(ci, 1365); }
            ci = (long long) x5 * 341 + w5 * 85 + v5 * 21 + u5 * 5 + t5 + 4;                           return (int) std::min<long long>(ci, 1366);
          };
          const FsProfile &gm = m->gm5;
          while (pos <= j && z < dom.tr.size()) {
            x5 = (wdsq[pos] < 4) ? wdsq[pos] : 1367;
            const bathgpu_trace_step &ts = dom.tr[z];
            switch (ts.st) {
            case TS_N: case TS_C: case TS_J:
              n2[pos] = 0.0f;
              if (ts.i == pos && pos > i + 1) pos++;
              z++; break;
            case TS_M:
              if (ts.i == pos) {
                int ci = cidx(ts.c);
                if (ci < 0) ci = 0;                          // a look-back before the envelope start holds -1 in the reference too
                n2[pos] = logf(r.null2[gm.codons[(size_t) ts.k * gm.maxcodons + ci]]);
                if (n2[pos] == kNegInfF) n2[pos] = 0.0f;
                z++;
              } else n2[pos] = 0.0f;
              pos++; break;
            case TS_I:
              if (ts.i == pos) {
                int ci = cidx(3);
                if (ci < 0) ci = 0;
                n2[pos] = logf(r.null2[gm.codons[(size_t) ts.k * gm.maxcodons + ci]]);
                if (n2[pos] == kNegInfF) n2[pos] = 0.0f;
                z++;
              } else n2[pos] = 0.0f;
              pos++; break;
            default: z++; break;
            }
            t5 = u5; u5 = v5; v5 = w5; w5 = x5;
          }
          for (pos = i; pos <= j; ++pos) domcorrection += n2[pos];
        }
        dom.domcorrection = std::max(0.f, domcorrection);
        int z1 = 0, z2 = (int) dom.tr.size() - 1;
        while (z1 < (int) dom.tr.size() && dom.tr[z1].st != TS_M) ++z1;
        while (z2 >= 0 && dom.tr[z2].st != TS_M) --z2;
        if (z1 > z2) return false;
        dom.iali = dom.tr[z1].i - (dom.tr[z1].c - 1);
        dom.jali = dom.tr[z2].i;
        dom.ienv = i; dom.jenv = j;
        dom.ihmm = dom.tr[z1].k; dom.jhmm = dom.tr[z2].k;
        dom.envsc = r.envsc; dom.oasc = r.oasc;

        // ---- p7_pli_postDomainDef_Frameshift_BATH (src/p7_pipeline.c:1005-1144)
        const int ali_len = dom.jali - dom.iali + 1;
        if (ali_len < 12) return false;
        const int env_len = dom.jenv - dom.ienv + 1;
        const int ml = q.max_length;
        float bitscore = dom.envsc;
        bitscore -= 2 * log(2. / ((env_len / 3.) + 2));
        bitscore += 2 * log(2. / (ml + 2));
        bitscore -= ((env_len - ali_len) / 3.) * log((float) (env_len / 3.) / (float) ((env_len / 3.) + 2));
        bitscore += ((std::max(env_len, ml * 3) - ali_len) / 3.) * log((float) ml / (float) (ml + 2));
        const float dom_bias = opt.do_null2 ? flogsum(0.0, log(lbg.omega) + dom.domcorrection) : 0.0f;
        const int nl = std::max(env_len / 3, ml);
        lbg.set_length(nl);
        const float hit_null = lbg.fs_null_one(nl);
        const float dom_score = (bitscore - (hit_null + dom_bias)) / kLog2;
        const double dom_lnP = exp_logsurv(dom_score, ev[EV_FTAUFS5], ev[EV_FLAMBDA]);
        const double Z2 = (float) nres_now / (float) ml;
        if (!(exp(dom_lnP) * Z2 <= opt.E)) return false;

        h = Hit();
        memset(&h.pub, 0, sizeof h.pub);
        auto orig = [&](int wpos) -> long long {            // window position -> coordinate on the source sequence
          return blk.complement ? blk.start - (dw.n + wpos) + 2 : blk.start + dw.n + wpos - 2;
        };
        h.pub.seqidx = sq.seqidx;
        snprintf(h.pub.name, sizeof h.pub.name, "%s", blk.name ? blk.name : "");
        h.pub.strand = blk.complement ? -1 : 1;
        h.pub.env_from = orig(dom.ienv); h.pub.env_to = orig(dom.jenv);
        h.pub.ali_from = orig(dom.iali); h.pub.ali_to = orig(dom.jali);
        h.pub.hmm_from = dom.ihmm; h.pub.hmm_to = dom.jhmm;
        h.pub.sq_len = blk.sq_len;
        h.pub.score = dom_score; h.pub.bias = dom_bias / kLog2; h.pub.lnP = dom_lnP;
        h.pub.pre_score = bitscore / kLog2;
        h.pub.envsc = dom.envsc; h.pub.oasc = dom.oasc;
        h.pub.trace_len = (int32_t) dom.tr.size();
        summarize_alignment(m, dom.tr, wdsq, h.pub, &h.ad);
        h.from_fs_branch = true;
        h.sortkey = -dom_lnP;
        return true;
    };
    std::vector<Hit> out(order.size());
    std::vector<uint8_t> ok(order.size(), 0);
    parallel_chunks(order.size(), 8, [&](size_t za, size_t zb) {
      Background lbg = bg;
      std::vector<uint8_t> wbuf;
      for (size_t z = za; z < zb; ++z) ok[z] = score_env(order[z], lbg, wbuf, out[z]) ? 1 : 0;
    });
    for (size_t z = 0; z < order.size(); ++z) if (ok[z]) S.hits_fs.emplace_back((int) order[z].b, std::move(out[z]));
  }
  tm.lap(S.st.us_score);

  // ---- the standard-translation branch: ORFs whose DNA window lost the arbitration, or every ORF past F3 without --fs
  // (src/p7_pipeline.c:1480-1511, :1720-1771): BackwardParser + DomainDecoding + regions per ORF, then each envelope rescored
  if (!S.stdq.empty()) {
    Background ubg = bg;                                     // the null model's length is set per hit: a private copy per unit
    const size_t nq = S.stdq.size();
    const float xfEm[2] = { expf(q.xsc_E_move), expf(q.xsc_E_loop) };
    std::vector<bathgpu_orf> od(nq);
    std::vector<size_t> xo(nq + 1, 0);
    for (size_t z = 0; z < nq; ++z) {
      const Orf &o = S.orfs[S.stdq[z].gi];
      memset(&od[z], 0, sizeof od[z]);
      od[z].offset = o.offset; od[z].L = o.n;
      xo[z + 1] = xo[z] + (size_t) o.n + 1;
    }
    std::vector<float> fx(xo[nq] * 6), bx(xo[nq] * 6), fsc(nq), bsc(nq);
    std::vector<int32_t> pst(nq);
    BE_TRY(s, BE.select_slot(BE.ctx, S.slot), "bathgpu_select_slot");
    BE_TRY(s, BE.orf_fwd_bck_xrows(BE.ctx, od.data(), (int) nq, q.nj, xfEm, fx.data(), bx.data(), fsc.data(), bsc.data(), pst.data()),
           "bathgpu_orf_fwd_bck_xrows");

    // p7_DomainDecoding (src/impl_sse/decoding.c:160-196) and the region logic of p7_domaindef_ByPosteriorHeuristics_BATH
    // (src/p7_domaindef.c:500-618); ORFs are independent here (the length model is saved and restored around each)
    struct SEnv { int z, i, j; bool multi = false; std::shared_ptr<std::vector<float>> n2sc; };   // n2sc: per-ORF-position null2 scores from the trace ensemble
    std::vector<std::vector<SEnv>> env_of(nq);
    std::vector<int> nreg(nq, 0), nmulti(nq, 0);
    parallel_chunks(nq, 1, [&](size_t za, size_t zb) {
      for (size_t z = za; z < zb; ++z) {
        if (pst[z] != 0) continue;
        const int L = od[z].L;
        const float *xf = &fx[xo[z] * 6], *xb = &bx[xo[z] * 6];
        auto F = [&](int i, int c) { return xf[(size_t) i * 6 + c]; };
        auto B = [&](int i, int c) { return xb[(size_t) i * 6 + c]; };
        const float loop = 1.0f - (2.0f + q.nj) / ((float) L + 2.0f + q.nj);
        bool own = false;
        for (int i = 1; i < L; ++i) if (B(i, 5) != F(i, 5)) { own = true; break; }
        std::vector<float> btot((size_t) L + 1), etot((size_t) L + 1), mocc((size_t) L + 1);
        float scaleproduct = 1.0 / B(0, 1);
        btot[0] = etot[0] = mocc[0] = 0.0f;
        for (int i = 1; i <= L; ++i) {
          btot[i] = btot[i - 1] + (F(i - 1, 3) * B(i - 1, 3) * F(i - 1, 5) * scaleproduct);
          if (own) scaleproduct *= F(i - 1, 5) / B(i - 1, 5);
          etot[i] = etot[i - 1] + (F(i, 0) * B(i, 0) * F(i, 5) * scaleproduct);
          float njcp;
          njcp  = F(i - 1, 1) * B(i, 1) * loop * scaleproduct;
          njcp += F(i - 1, 2) * B(i, 2) * loop * scaleproduct;
          njcp += F(i - 1, 4) * B(i, 4) * loop * scaleproduct;
          mocc[i] = 1. - njcp;
        }
        if (std::isinf(scaleproduct)) continue;             // eslERANGE
        const float rt1 = 0.25f, rt2 = 0.10f, rt3 = 0.20f;
        int i = -1; bool triggered = false;
        for (int j = 1; j <= L; ++j) {
          if (!triggered) {
            if (mocc[j] - (btot[j] - btot[j - 1]) < rt2) i = j;
            else if (i == -1) i = j;
            if (mocc[j] >= rt1) triggered = true;
          } else if (mocc[j] - (etot[j] - etot[j - 1]) < rt2) {
            nreg[z]++;
            float mx = -1.0f;                               // is_multidomain_region (:652-664)
            for (int zz = i; zz <= j; ++zz) mx = std::max(mx, std::min(etot[zz] - etot[i - 1], btot[j] - btot[zz - 1]));
            if (mx >= rt3) nmulti[z]++;
            SEnv se; se.z = (int) z; se.i = i; se.j = j; se.multi = (mx >= rt3);
            env_of[z].push_back(se);
            i = -1; triggered = false;
          }
        }
      }
    });
    // ---- multi-domain regions (is_multidomain_region): resolved by clustering an ensemble of stochastic tracebacks
    // (src/p7_domaindef.c:551-600).  The Forward matrices of all flagged regions of the unit come from one device call (multihit
    // mode at the ORF's own length model: om's length was set to the ORF's, :510, :561); sampling, null2-by-trace and clustering on
    // the host cores (stotrace.cpp), one region per task; each cluster then takes the region's place as an envelope of its own.
    if (BE.orf_forward_matrices) {
      struct MReg { size_t z, e; };
      std::vector<MReg> mregs;
      for (size_t z = 0; z < nq; ++z) for (size_t e = 0; e < env_of[z].size(); ++e) if (env_of[z][e].multi) mregs.push_back(MReg{ z, e });
      if (!mregs.empty()) {
        std::vector<bathgpu_envelope> regs(mregs.size());
        std::vector<int64_t> off(mregs.size() + 1, 0);
        for (size_t r = 0; r < mregs.size(); ++r) {
          const SEnv &se = env_of[mregs[r].z][mregs[r].e];
          regs[r].start = od[mregs[r].z].offset + se.i - 1; regs[r].L = se.j - se.i + 1;
          bathhost_length_model(od[mregs[r].z].L, 1.0f, &regs[r].pmove, &regs[r].ploop);      // p7_oprofile_ReconfigMultihit(om, saveL)
          off[r + 1] = off[r] + regs[r].L + 1;
        }
        std::vector<float> mxbuf((size_t) off.back() * (M + 1) * 4), xrbuf((size_t) off.back() * 6), rsc(regs.size());
        std::vector<int32_t> rst(regs.size());
        const float xfEmh[2] = { 0.5f, 0.5f };
        BE_TRY(s, BE.orf_forward_matrices(BE.ctx, regs.data(), (int) regs.size(), xfEmh, mxbuf.data(), xrbuf.data(), off.back(), rsc.data(), rst.data()),
               "bathgpu_orf_forward_matrices");
        std::vector<std::vector<SEnv>> repl(mregs.size());
        const float *rf_amino = m->om3.rfv.data() + (size_t) (m->om3.nrows - kKp) * (M + 1);
        parallel_chunks(mregs.size(), 1, [&](size_t ra, size_t rb) {
          for (size_t r = ra; r < rb; ++r) {
            const SEnv &se = env_of[mregs[r].z][mregs[r].e];
            if (rst[r] != 0) continue;                       // Forward out of range: no clusters, no envelope
            const ForwardMatrix F{ mxbuf.data() + (size_t) off[r] * (M + 1) * 4, xrbuf.data() + (size_t) off[r] * 6, M, regs[r].L };
            const SpecialOdds X{ regs[r].pmove, regs[r].ploop, xfEmh[0], xfEmh[1] };
            const uint8_t *rres = S.sres + od[mregs[r].z].offset + se.i - 2;       // rres[p] = residue p of the region
            std::vector<Segment> sp;
            std::vector<float> n2r;
            if (!sample_region_segments_protein(F, m->om3.tfv.data(), rf_amino, X, 42u, 200, se.i, rres, sp, n2r)) continue;
            auto n2 = std::make_shared<std::vector<float>>((size_t) od[mregs[r].z].L + 2, 0.0f);
            for (int p = 1; p <= regs[r].L; ++p) (*n2)[(size_t) (se.i + p - 1)] = n2r[(size_t) p];
            for (const Segment &g : cluster_region_segments(sp, 200, true)) {
              SEnv c; c.z = se.z; c.i = g.i; c.j = g.j; c.multi = false; c.n2sc = n2;
              repl[r].push_back(c);
            }
          }
        });
        for (size_t r = mregs.size(); r-- > 0;) {              // back to front: positions in env_of[z] stay valid
          std::vector<SEnv> &v = env_of[mregs[r].z];
          v.erase(v.begin() + (long) mregs[r].e);
          v.insert(v.begin() + (long) mregs[r].e, repl[r].begin(), repl[r].end());
        }
      }
    }
    std::vector<SEnv> envs;
    std::vector<bathgpu_envelope> ge;
    int64_t max_steps = 0;
    for (size_t z = 0; z < nq; ++z) {
      S.st.n_regions += nreg[z]; S.st.n_multidomain_regions += nmulti[z];
      for (const SEnv &e : env_of[z]) {
        const int Ld = e.j - e.i + 1;
        bathgpu_envelope g;
        g.start = od[z].offset + e.i - 1; g.L = Ld;
        bathhost_length_model(Ld, 0.0f, &g.pmove, &g.ploop);     // p7_oprofile_ReconfigLength(om, Ld) in unihit mode (:1244)
        ge.push_back(g); envs.push_back(e);
        max_steps += Ld + M + 8;
      }
    }
    if (!ge.empty()) {
    std::vector<bathgpu_domain_result> res(ge.size());
    std::vector<bathgpu_trace_step> traces((size_t) max_steps);
    const float xfEu[2] = { 1.0f, 0.0f };
    BE_TRY(s, BE.orf_domains(BE.ctx, ge.data(), (int) ge.size(), xfEu, res.data(), traces.data(), max_steps), "bathgpu_orf_domains");
    S.st.n_envelopes += (int64_t) ge.size();

    std::vector<uint8_t> wbuf;
    for (size_t e = 0; e < envs.size(); ++e) {
      const bathgpu_domain_result &r = res[e];
      if (r.status != 0 || r.trace_len == 0) continue;       // eslFAIL (:1252)
      const Unit::StdItem &it = S.stdq[envs[e].z];
      const Orf &o = S.orfs[it.gi];
      const int b = S.orf_blk[it.gi];
      const BlockInfo &binfo = blocks[b];
      // windowsq: the DNA window (--fs) or the ORF's own nucleotides (default pipeline); block-local start
      // (an ORF sent here on a stale orfsq->idx need not lie inside that window: the stretch covers both)
      const SeqRef &sq = seqs[(size_t) binfo.seq];
      const long long n = sq.n;
      const char *name = sq.name.c_str();
      const long long win_n = (it.w >= 0) ? S.dwin[it.w].n : o.start;
      const long long win_e = (it.w >= 0) ? win_n + S.dwin[it.w].length - 1 : o.end;
      const long long lo0 = std::min<long long>(win_n, o.start) - 1, hi0 = std::max<long long>(win_e, o.end);
      const uint8_t *wdsq = oriented(sq, binfo, S.complement, lo0, (int) (hi0 - lo0), wbuf) + (lo0 - (win_n - 1));    // wdsq[p] = block position win_n - 1 + p
      const uint8_t *res_o = S.sres + o.offset - 1;           // ORF residue p is res_o[p]
      const int i = envs[e].i, j = envs[e].j;
      Domain dom;
      dom.tr.assign(traces.begin() + r.trace_offset, traces.begin() + r.trace_offset + r.trace_len);
      int orf_pos = 0;                                       // tr->sqfrom[0]: ORF position of the first match state (p7_trace_Index)
      for (auto &ts : dom.tr) {
        if (ts.i > 0) ts.i += i - 1;                         // (:1260-1261)
        if (orf_pos == 0 && ts.st == TS_M) orf_pos = ts.i;
      }
      {                                                      // p7_trace_fs_Convert (src/p7_trace.c:405-438)
        const int start = (int) (o.start - win_n);
        for (size_t z = 0; z < dom.tr.size(); ++z) {
          bathgpu_trace_step &ts = dom.tr[z];
          switch (ts.st) {
          case TS_N: case TS_C: case TS_J:
            if (z > 0 && dom.tr[z - 1].st == ts.st) ts.i = start + ts.i * 3;
            ts.c = 0; break;
          case TS_M: ts.i = start + ts.i * 3; ts.c = 3; break;
          case TS_I: ts.i = start + ts.i * 3; ts.c = 0; break;
          default: ts.c = 0; break;
          }
        }
      }
      const float aliscore = ali_score(m, dom.tr, wdsq);
      if (aliscore < 0.0f) continue;
      float domcorrection = 0.0f;                            // (:1296-1305)
      if (envs[e].n2sc) { for (int pos = i; pos <= j; ++pos) domcorrection += (*envs[e].n2sc)[(size_t) pos]; }   // null2_is_done (:1295)
      else for (int pos = i; pos <= j; ++pos) domcorrection += logf(r.null2[res_o[pos]]);
      dom.domcorrection = std::max(0.f, domcorrection);
      int z1 = 0, z2 = (int) dom.tr.size() - 1;
      while (z1 < (int) dom.tr.size() && dom.tr[z1].st != TS_M) ++z1;
      while (z2 >= 0 && dom.tr[z2].st != TS_M) --z2;
      if (z1 > z2) continue;
      dom.ihmm = dom.tr[z1].k; dom.jhmm = dom.tr[z2].k;
      dom.iali = dom.tr[z1].i - (dom.tr[z1].c - 1); dom.jali = dom.tr[z2].i;
      dom.ienv = i; dom.jenv = j; dom.envsc = r.envsc; dom.oasc = r.oasc;

      // ---- p7_pli_postDomainDef_BATH (src/p7_pipeline.c:1172-1290)
      const int env_len = dom.jenv - dom.ienv + 1;
      const int ali_len = (dom.jali - dom.iali + 1) / 3;
      if (ali_len < 4) continue;
      const int ml = q.max_length;
      float bitscore = dom.envsc;
      bitscore -= 2 * log(2. / (env_len + 2));
      bitscore += 2 * log(2. / (ml + 2));
      bitscore -= (env_len - ali_len) * log((float) env_len / (float) (env_len + 2));
      bitscore += (ml - ali_len) * log((float) ml / (float) (ml + 2));
      const float dom_bias = opt.do_null2 ? flogsum(0.0, log(ubg.omega) + dom.domcorrection) : 0.0f;
      ubg.set_length(ml);
      const float nullsc = ubg.null_one(ml);
      const float dom_score = (bitscore - (nullsc + dom_bias)) / kLog2;
      const double dom_lnP = exp_logsurv(dom_score, ev[EV_FTAU], ev[EV_FLAMBDA]);
      const double Z = (float) binfo.nres_at[sidx] / (float) ml;
      if (!(exp(dom_lnP) * Z <= opt.E)) continue;

      Hit h;
      memset(&h.pub, 0, sizeof h.pub);
      const long long bstart = S.start_of(binfo);            // dnasq->start
      auto orig = [&](int wpos) -> long long { return S.complement ? bstart - (win_n + wpos) + 2 : bstart + win_n + wpos - 2; };
      h.pub.seqidx = sq.seqidx;
      snprintf(h.pub.name, sizeof h.pub.name, "%s", name ? name : "");
      h.pub.strand = S.complement ? -1 : 1;
      if (!S.complement) { h.pub.env_from = bstart + o.start + dom.ienv * 3 - 4; h.pub.env_to = bstart + o.start + dom.jenv * 3 - 2; }
      else {                                                 // dnasq->end + orfsq->start, orfsq->start = dnasq->n - o.start + 1 on this strand
        const long long base = binfo.b0 + (binfo.n - o.start + 1);
        h.pub.env_from = base - dom.ienv * 3 + 2; h.pub.env_to = base - dom.jenv * 3;
      }
      h.pub.ali_from = orig(dom.iali); h.pub.ali_to = orig(dom.jali);
      h.pub.hmm_from = dom.ihmm; h.pub.hmm_to = dom.jhmm;
      h.pub.sq_len = (long long) n;
      h.pub.score = dom_score; h.pub.bias = dom_bias / kLog2; h.pub.lnP = dom_lnP;
      h.pub.pre_score = bitscore / kLog2;
      h.pub.envsc = dom.envsc; h.pub.oasc = dom.oasc;
      h.pub.trace_len = (int32_t) dom.tr.size();
      {                                                      // p7_alidisplay_nonfs_Create (src/p7_alidisplay.c:937-1230): PID and CIGAR
        std::string cigar;
        char buf[32];
        int exact = 0, ncore = 0, n_count = 0, pos = orf_pos;
        h.ad.size_for(z2 - z1 + 1, !m->hmm.cs.empty(), !m->hmm.rf.empty());
        for (int z = z1; z <= z2; ++z) {
          const bathgpu_trace_step &ts = dom.tr[z];
          const int nxt = dom.tr[z + 1].st;                 // z2 + 1 exists: the E state
          ncore++;
          {                                                  // display lines (:1128-1215)
            AliDisplay &ad = h.ad;
            const int y = z - z1;
            const char cons = m->hmm.consensus[ts.k];
            if (ts.st == TS_D) { ad.model[y] = cons; ad.aseq[y] = '-'; memcpy(&ad.ntseq[5 * y], " --- ", 5); }
            else {
              const int x = res_o[pos];
              const char cc[5] = { ' ', (char) toupper(kDnaSym[wdsq[ts.i - 2]]), (char) toupper(kDnaSym[wdsq[ts.i - 1]]), (char) toupper(kDnaSym[wdsq[ts.i]]), ' ' };
              memcpy(&ad.ntseq[5 * y], cc, 5);
              ad.aseq[y] = (char) toupper(kAminoSym[x]);
              if (ts.st == TS_M) {
                ad.model[y] = cons;
                ad.mline[y] = (x == amino_code(cons)) ? cons : (expf(q.msc[(size_t) x * (q.M + 1) + ts.k]) > 1.0) ? '+' : ' ';
                ad.codon[y] = ts.c;
              } else { ad.model[y] = '.'; ad.codon[y] = 3; }
            }
            ad.ppline[y] = (ts.st == TS_D) ? '.' : encode_post_prob(ts.pp);
            if (!m->hmm.cs.empty()) ad.csline[y] = (ts.st == TS_I) ? '.' : m->hmm.cs[ts.k];
            if (!m->hmm.rf.empty()) ad.rfline[y] = (ts.st == TS_I) ? '.' : m->hmm.rf[ts.k];
          }
          if (ts.st == TS_M) { if (res_o[pos] == amino_code(m->hmm.consensus[ts.k])) exact++; pos++; }
          else if (ts.st == TS_I) pos++;
          n_count += 3;
          if (nxt != ts.st) { snprintf(buf, sizeof buf, "%d%c", n_count, ts.st == TS_M ? 'M' : ts.st == TS_I ? 'I' : 'D'); cigar += buf; n_count = 0; }
        }
        h.pub.pid = ncore ? ((float) exact / ncore) * 100 : 0.0f;
        snprintf(h.pub.cigar, sizeof h.pub.cigar, "%s", cigar.c_str());
        h.ad.cigar = cigar;
      }
      h.sortkey = -dom_lnP;
      S.hits_std.emplace_back(b, std::move(h));
    }
    }
  }
  tm.lap(S.st.us_std);
  return 0;
  };   // finish_unit
  rc = for_each_backend(s, [&](int be) -> int {
    for (int c : chunks_of_be[(size_t) be])
      for (int sidx : active) { const int st = finish_unit(unit_of((size_t) c, sidx)); if (st != 0) return st; }
    return 0;
  });
  if (rc != 0) return rc;
  trace.mark("envelopes, scoring, std branch");

  // ---- hits in the reference's order: block by block, top strand then bottom strand; counters summed over units
  {
    std::vector<size_t> pf(units.size(), 0), ps(units.size(), 0);
    size_t more = 0;
    for (auto &U : units) more += U->hits_fs.size() + U->hits_std.size();
    s->hits.reserve(s->hits.size() + more);
    for (size_t b = 0; b < nb; ++b)
      for (int sidx : active) {
        const size_t u = 2 * (size_t) chunk_of_block[b] + (size_t) sidx;
        Unit &S = *units[u];
        for (; pf[u] < S.hits_fs.size() && S.hits_fs[pf[u]].first == (int) b; ++pf[u]) s->hits.push_back(std::move(S.hits_fs[pf[u]].second));
        for (; ps[u] < S.hits_std.size() && S.hits_std[ps[u]].first == (int) b; ++ps[u]) s->hits.push_back(std::move(S.hits_std[ps[u]].second));
      }
  }
  for (auto &U : units) add_stats(s->st, U->st);
  s->nseqs += (int64_t) seqs.size();
  s->st.nseqs = s->nseqs;
  trace.mark("hit list");
  return 0;
}

bathgpu_filter_params filter_params(const bathhost_search *s)
{
  const ProteinProfile &q = s->model->prot;
  bathgpu_filter_params fp;
  fp.M = s->model->hmm.M; fp.tbm_b = q.tbm_b; fp.tec_b = q.tec_b; fp.base_b = q.base_b; fp.bias_b = q.bias_b; fp.scale_b = q.scale_b;
  fp.base_w = q.base_w; fp.ddbound_w = q.ddbound_w; fp.xw_E_move = q.xw_E_move; fp.xw_E_loop = q.xw_E_loop; fp.scale_w = q.scale_w;
  fp.cpu_lanes_u8 = s->opt.lanes_u8; fp.cpu_lanes_i16 = s->opt.lanes_i16;
  return fp;
}

// device images: the three profiles of a query, replicated on every device context
int load_images(bathhost_search *s)
{
  const bathhost_model *m = s->model;
  const int M = m->hmm.M;
  const bathgpu_filter_params fp = filter_params(s);
  const ProteinProfile &q = m->prot;
  return for_each_backend(s, [&](int k) -> int {
    const bathhost_backend &BE = s->bes[(size_t) k];
    int rc;
    if ((rc = BE.load_fs_profile(BE.ctx, 3, M, m->om3.nrows, m->om3.rfv.data(), m->om3.tfv.data())) != 0 ||
        (rc = BE.load_fs_profile(BE.ctx, 5, M, m->om5.nrows, m->om5.rfv.data(), m->om5.tfv.data())) != 0 ||
        (rc = BE.load_filter_profile(BE.ctx, &fp, q.rbv.data(), q.rwv.data(), q.twv.data())) != 0) return rc;
    return 0;
  });
}

}  // namespace

// ------------------------------------------------------------------------------------------
extern "C" int bathhost_search_create_multi(const bathhost_model *m, const bathhost_backend *be, int nbackends, const bathhost_options *o, bathhost_search **ret)
{
  if (!m || !be || nbackends < 1 || nbackends > 256 || !ret) return BATHHOST_EINVAL;
  *ret = nullptr;
  if (!m->hmm.has_fs3 || !m->hmm.has_fs5 || !(m->hmm.fsprob > 0) || m->hmm.max_length < 1) return BATHHOST_EINVAL;   // src/bathsearch.c:747-759
  flogsum_init();
  bathhost_search *s = new (std::nothrow) bathhost_search(m, be, nbackends);
  if (!s) return BATHHOST_EMEM;
  if (o) {
    if (o->F1 > 0) s->opt.F1 = o->F1;
    if (o->F2 > 0) s->opt.F2 = o->F2;
    if (o->F3 > 0) s->opt.F3 = o->F3;
    if (o->F4 > 0) s->opt.F4 = o->F4;
    if (o->E > 0)  s->opt.E = o->E;
    if (o->min_orf_len > 0) s->opt.min_orf = o->min_orf_len;
    if (o->block_length > 0) s->opt.block_length = o->block_length;
    if (o->cpu_lanes_u8 > 0) s->opt.lanes_u8 = o->cpu_lanes_u8;
    if (o->cpu_lanes_i16 > 0) s->opt.lanes_i16 = o->cpu_lanes_i16;
    s->opt.do_bias = !o->no_bias; s->opt.do_null2 = !o->no_null2;
    s->opt.top = !o->bottom_only; s->opt.bottom = !o->top_only;
    s->opt.fs = !o->std_only;
    s->opt.frameline = o->show_frameline != 0;
    if (o->chunk_nt > 0) s->chunk_nt = o->chunk_nt;
  }
  if (!genetic_code(m->ct, s->gcode)) { delete s; return BATHHOST_EINVAL; }
  s->compo.assign(m->hmm.compo, m->hmm.compo + kK);
  s->bg.set_filter(m->hmm.M, s->compo.data());           // p7_pli_NewModel -> p7_bg_SetFilter(bg, om->M, om->compo)

  const int st = load_images(s);
  if (st != 0) { delete s; return st; }
  *ret = s;
  return BATHHOST_OK;
}

extern "C" int bathhost_search_create(const bathhost_model *m, const bathhost_backend *be, const bathhost_options *o, bathhost_search **ret)
{
  return bathhost_search_create_multi(m, be, 1, o, ret);
}

extern "C" void bathhost_search_destroy(bathhost_search *s) { delete s; }
extern "C" const char *bathhost_search_last_error(const bathhost_search *s) { return s ? s->err.c_str() : "no search"; }

// One more target sequence for the next bathhost_search_run: dsq[1..n] (sentinels at 0 and n+1), which the caller keeps alive
// and unchanged until that call returns.  Sequences are numbered in the order they are queued.
extern "C" int bathhost_search_queue(bathhost_search *s, const char *name, const uint8_t *dsq, int64_t n)
{
  if (!s || !dsq || n < 1) return BATHHOST_EINVAL;
  SeqRef r;
  r.name = name ? name : ""; r.dsq = dsq; r.n = n; r.seqidx = s->nseqs + (int64_t) s->queue.size();
  s->queue.push_back(std::move(r));
  return BATHHOST_OK;
}

// Every queued sequence, both strands unless restricted, through the whole pipeline: one stage-batched pass over all of them,
// dealt to the search's device contexts.  The state the reference carries from block to block (hit-window list, length model,
// residue count) continues from the previous run, so queueing everything and running once, or running after every sequence, gives
// the same hits.
extern "C" int bathhost_search_run(bathhost_search *s)
{
  if (!s) return BATHHOST_EINVAL;
  s->finished = false;
  return run_batch(s);
}

// One target sequence searched at once (queue + run).
extern "C" int bathhost_search_sequence(bathhost_search *s, const char *name, const uint8_t *dsq, int64_t n)
{
  const int st = bathhost_search_queue(s, name, dsq, n);
  return st != BATHHOST_OK ? st : bathhost_search_run(s);
}

// E-values over the whole search space, duplicate removal, final ordering and reporting threshold
// (src/bathsearch.c:869-921; src/p7_tophits.c:262-309, :789-960; src/p7_pipeline.c:584-602)
extern "C" int bathhost_search_finish(bathhost_search *s)
{
  if (!s) return BATHHOST_EINVAL;
  if (!s->queue.empty()) { const int st = bathhost_search_run(s); if (st != BATHHOST_OK) return st; }
  if (s->finished) return BATHHOST_OK;
  s->finished = true;
  const int Wn = s->model->prot.max_length * 3;
  for (Hit &h : s->hits) {
    if (!h.evalue_done) {                                   // hits of earlier finish calls keep the pre-correction value in lnP_raw
      h.lnP_raw = h.pub.lnP;
      h.evalue_done = true;
    }
    h.duplicate = false;
    h.pub.lnP = h.lnP_raw + log((float) s->st.nres / (float) Wn);      // p7_tophits_ComputeEvalues_BATH over the residues searched so far
    h.sortkey = -1.0 * h.pub.lnP;
    h.pub.evalue = exp(h.pub.lnP);
  }
  // The two sorts run on an index vector and the hits are moved once at the end: a Hit carries a kilobyte of fixed-size fields
  // (name, CIGAR), and sorting the records themselves cost 15-20 ms per profile and Gbp.
  std::vector<uint32_t> ord(s->hits.size());
  for (size_t z = 0; z < ord.size(); ++z) ord[z] = (uint32_t) z;
  const std::vector<Hit> &HV = s->hits;
  // p7_tophits_SortBySeqidxAndAlipos (hit_sorter_by_seqidx_aliposition, src/p7_tophits.c:286-306): seqidx, plus strand first, then
  // the smaller coordinate ascending and the larger one descending -- start and end are swapped on the minus strand first
  std::stable_sort(ord.begin(), ord.end(), [&HV](uint32_t x, uint32_t y) {
    const Hit &a = HV[x], &b = HV[y];
    if (a.pub.seqidx != b.pub.seqidx) return a.pub.seqidx < b.pub.seqidx;
    const int da = a.pub.ali_from < a.pub.ali_to ? 1 : -1, db = b.pub.ali_from < b.pub.ali_to ? 1 : -1;
    if (da != db) return da > db;
    const long long as = std::min(a.pub.ali_from, a.pub.ali_to), ae = std::max(a.pub.ali_from, a.pub.ali_to);
    const long long bs = std::min(b.pub.ali_from, b.pub.ali_to), be = std::max(b.pub.ali_from, b.pub.ali_to);
    if (as != bs) return as < bs;
    return ae > be;
  });
  if (ord.size() > 1) {                                     // p7_tophits_RemoveDuplicates
    size_t j = 0;
    for (size_t i = 1; i < ord.size(); ++i) {
      Hit &hj = s->hits[ord[j]], &hi = s->hits[ord[i]];
      long long s_j = hj.pub.ali_from, e_j = hj.pub.ali_to, s_i = hi.pub.ali_from, e_i = hi.pub.ali_to;
      const int dir_j = s_j < e_j ? 1 : -1, dir_i = s_i < e_i ? 1 : -1;
      if (dir_j == -1) std::swap(s_j, e_j);
      if (dir_i == -1) std::swap(s_i, e_i);
      const long long len_j = e_j - s_j + 1, len_i = e_i - s_i + 1;
      const long long is = std::max(s_i, s_j), ie = std::min(e_i, e_j), ilen = ie - is + 1;
      const int hs = std::max(hi.pub.hmm_from, hj.pub.hmm_from), he = std::min(hi.pub.hmm_to, hj.pub.hmm_to), hlen = he - hs + 1;
      const Hit &hp = s->hits[ord[i - 1]];
      if (hi.pub.seqidx == hp.pub.seqidx && dir_i == dir_j && hlen > 0 &&
          ((s_i >= s_j - 3 && s_i <= s_j + 3) || (e_i >= e_j - 3 && e_i <= e_j + 3) || (ilen >= len_i * 0.95) || (ilen >= len_j * 0.95))) {
        const size_t remove = hi.pub.lnP < hj.pub.lnP ? j : i;
        s->hits[ord[remove]].duplicate = true;
        j = (remove == j ? i : j);
      } else j = i;
    }
  }
  // p7_tophits_SortBySortkey: sortkey descending, then name, strand, position
  std::stable_sort(ord.begin(), ord.end(), [&HV](uint32_t x, uint32_t y) {
    const Hit &a = HV[x], &b = HV[y];
    if (a.sortkey != b.sortkey) return a.sortkey > b.sortkey;
    const int c = strcmp(a.pub.name, b.pub.name);
    if (c != 0) return c < 0;
    const int da = a.pub.ali_from < a.pub.ali_to ? 1 : -1, db = b.pub.ali_from < b.pub.ali_to ? 1 : -1;
    if (da != db) return da > db;
    return a.pub.ali_from < b.pub.ali_from;
  });
  {
    std::vector<Hit> moved;
    moved.reserve(s->hits.size());
    for (uint32_t z : ord) moved.push_back(std::move(s->hits[z]));
    s->hits.swap(moved);
  }
  s->st.n_hits_reported = 0;
  for (Hit &h : s->hits) {
    h.reported = !h.duplicate && (exp(h.pub.lnP) <= s->opt.E);      // Z forced to 1 for reporting (src/bathsearch.c:920)
    if (h.reported) s->st.n_hits_reported++;
  }
  return BATHHOST_OK;
}

// Several searches (one per query profile, each with device contexts of its own) finished at the same time, one host thread each:
// bathsearch's query loop (src/bathsearch.c:737) takes the profiles one after the other, but the searches share nothing, and run
// together one search's serial host phases (region walk, hit list) sit under the others' device stages.  Every search gives the hit
// list it gives alone.  Returns the first non-zero status.
extern "C" int bathhost_search_finish_many(bathhost_search *const *ss, int n)
{
  if (n < 0 || (n > 0 && !ss)) return BATHHOST_EINVAL;
  for (int k = 0; k < n; ++k) {
    if (!ss[k]) return BATHHOST_EINVAL;
    for (int q = 0; q < k; ++q) {
      if (ss[q] == ss[k]) return BATHHOST_EINVAL;
      for (const bathhost_backend &a : ss[q]->bes)          // a device context serves one search at a time
        for (const bathhost_backend &b : ss[k]->bes)
          if (a.ctx && a.ctx == b.ctx) return fail(ss[k], BATHHOST_EINVAL, "bathhost_search_finish_many: two searches share a device context");
    }
  }
  if (n == 0) return BATHHOST_OK;
  std::vector<int> st((size_t) n, BATHHOST_OK);
  std::vector<std::thread> th;
  for (int k = 1; k < n; ++k) th.emplace_back([&, k] { st[(size_t) k] = bathhost_search_finish(ss[k]); });
  st[0] = bathhost_search_finish(ss[0]);
  for (auto &t : th) t.join();
  for (int k = 0; k < n; ++k) if (st[(size_t) k] != BATHHOST_OK) return st[(size_t) k];
  return BATHHOST_OK;
}

extern "C" int bathhost_search_nhits(const bathhost_search *s) { return s ? (int) s->st.n_hits_reported : 0; }

extern "C" int bathhost_search_get_hit(const bathhost_search *s, int idx, bathhost_hit *hit)
{
  if (!s || !hit || idx < 0) return BATHHOST_EINVAL;
  int z = 0;
  for (const Hit &h : s->hits) if (h.reported) { if (z == idx) { *hit = h.pub; return BATHHOST_OK; } ++z; }
  return BATHHOST_EINVAL;
}

// p7_tophits_TabularTargets (src/p7_tophits.c:1603-1712) as bathsearch calls it with --tblout --cigar: the header and one line per
// reported hit, byte for byte (column widths grow with the longest name / coordinate exactly as there).  The trailer the
// reference appends (p7_tophits_TabularTail: program, files, command line, date) is the caller's.
extern "C" int bathhost_search_format_tblout(const bathhost_search *s, int show_header, char *buf, size_t cap, size_t *needed)
{
  if (!s || !needed || (!buf && cap > 0)) return BATHHOST_EINVAL;
  const bathhost_model *m = s->model;
  const std::string qname = m->hmm.name, qacc = m->hmm.acc;
  const bool fs_pipe = s->opt.fs;
  int tnamew = 20, posw = 9;
  for (const Hit &h : s->hits) {
    tnamew = std::max(tnamew, (int) strlen(h.pub.name));
    if (h.pub.ali_from > 0) {
      posw = std::max(posw, (int) std::to_string((long long) h.pub.ali_from).size());
      posw = std::max(posw, (int) std::to_string((long long) h.pub.ali_to).size());
    }
  }
  const int qnamew = std::max(20, (int) qname.size()), qaccw = std::max(10, (int) qacc.size()), taccw = 10;
  std::string out;
  char line[4096];
  auto put = [&](const char *fmt, auto... args) { snprintf(line, sizeof line, fmt, args...); out += line; };
  if (show_header) {
    put("#%7s %-*s %-*s %-*s %-*s %9s %9s %9s %9s %9s %9s", " hit ID", tnamew - 1, " target name", taccw, " accession", qnamew, " query name",
        qaccw, " accession", "  hmm len", " hmm from", "   hmm to", "  seq len", " ali from", "   ali to");
    put("  %9s %6s %5s %5s", "  E-value", " score", " bias", "  PID");
    if (fs_pipe) put(" %7s %6s", " shifts", " stops");
    put(" %s\n", "CIGAR");
    put("#%7s %-*s %-*s %-*s %-*s %9s %9s %9s %9s %9s %9s", "-------", tnamew - 1, "-------------------", taccw, "----------", qnamew,
        "--------------------", qaccw, "----------", "---------", "---------", "---------", "---------", "---------", "---------");
    put("  %9s %6s %5s %5s", "---------", "------", "-----", "-----");
    if (fs_pipe) put(" %7s %6s", "-------", "------");
    put(" %s\n", "---------------------");
  }
  int id = 0;
  for (const Hit &h : s->hits) {
    if (!h.reported) continue;
    ++id;
    put("%8d %-*s %-*s %-*s %-*s %8d  %8d  %8d  %*lld %*lld %*lld", id, tnamew, h.pub.name, taccw, "-", qnamew, qname.c_str(), qaccw,
        qacc.empty() ? "-" : qacc.c_str(), m->hmm.M, h.pub.hmm_from, h.pub.hmm_to, posw, (long long) h.pub.sq_len, posw, (long long) h.pub.ali_from,
        posw, (long long) h.pub.ali_to);
    put(" %9.2g %6.1f %5.1f %5.2f", h.pub.evalue, h.pub.score, h.pub.bias, h.pub.pid);
    if (fs_pipe) put(" %7d %6d", h.pub.shifts, h.pub.stops);
    put(" %s\n", h.ad.cigar.empty() ? h.pub.cigar : h.ad.cigar.c_str());
  }
  *needed = out.size() + 1;
  if (out.size() + 1 > cap) return buf ? BATHHOST_EINVAL : BATHHOST_OK;
  memcpy(buf, out.c_str(), out.size() + 1);
  return BATHHOST_OK;
}

// p7_alidisplay_Print_BATH (src/p7_alidisplay.c:3758-4095) without the spliced-alignment and --frameline branches: blocks of
// (CS) (RF) model / match / translation / codons / PP lines, each alignment column five characters wide
static void print_alidisplay(std::string &out, const AliDisplay &ad, const std::string &hmmname, const char *sqname, int hmmfrom, int hmmto,
                             long long sqfrom, long long sqto, int linewidth, bool show_frameline)
{
  char line[512];
  auto put = [&](const char *fmt, auto... args) { snprintf(line, sizeof line, fmt, args...); out += line; };
  auto textwidth = [](long long n) { int w = (n < 0) ? 1 : 0; while (n != 0) { n /= 10; w++; } return w; };
  const int max_namewidth = 30, min_aliwidth = 40;
  std::string show_hmm = hmmname, show_sq = sqname;
  int namewidth = (int) std::max(show_hmm.size(), show_sq.size());
  while (namewidth > max_namewidth + 3) {
    std::string &longer = (show_hmm.size() > show_sq.size()) ? show_hmm : show_sq;
    longer = longer.substr(0, max_namewidth) + "...";
    namewidth = (int) std::max(show_hmm.size(), show_sq.size());
  }
  namewidth = std::max(namewidth, 8);
  const int coordwidth = std::max(std::max(textwidth(hmmfrom), textwidth(hmmto)), std::max(textwidth(sqfrom), textwidth(sqto)));
  int max_aliwidth = (linewidth > 0) ? linewidth - namewidth - 2 * coordwidth - 5 : ad.N;
  if (max_aliwidth < ad.N && max_aliwidth < min_aliwidth) max_aliwidth = min_aliwidth;
  max_aliwidth -= 4;
  max_aliwidth /= 5;
  const bool fwd = sqfrom < sqto;
  long long i1 = sqfrom, i2 = fwd ? i1 - 1 : i1 + 1;
  int k1 = hmmfrom, pos = 0;
  auto row = [&](const std::string &chars, int w) { for (int i = 0; i < w && pos + i < (int) chars.size(); ++i) put("  %c  ", chars[pos + i]); };
  while (pos < ad.N) {
    if (pos > 0) out += "\n";
    const int w = max_aliwidth;
    int ni = 0, nk = 0;
    for (int z = pos; z < pos + w && z < ad.N; ++z) {
      if (ad.model[z] != '.' && ad.model[z] != ' ') nk++;
      if (ad.aseq[z] != '-') ni++;
    }
    const int k2 = k1 + nk - 1;
    if (!ad.csline.empty()) { put("  %*s ", namewidth + coordwidth + 1, " "); out += "  "; row(ad.csline, w); out += "  \n"; }
    if (!ad.rfline.empty()) { put("  %*s ", namewidth + coordwidth + 1, " "); out += "  "; row(ad.rfline, w); out += "   RF\n"; }
    put("  %*s %*d ", namewidth, show_hmm.c_str(), coordwidth, k1); out += "  "; row(ad.model, w); out += "  "; put(" %-*d\n", coordwidth, k2);
    put("  %*s ", namewidth + coordwidth + 1, " "); out += "  "; row(ad.mline, w); out += "  \n";
    put("  %*s ", namewidth + coordwidth + 1, " "); out += "  "; row(ad.aseq, w); out += "  \n";
    put("  %*s", namewidth, show_sq.c_str());
    if (ni > 0) put(" %*lld ", coordwidth, i1); else put(" %*s ", coordwidth, "-");
    out += "  ";
    std::vector<int> frameline;
    for (int j = 0; j < w && pos + j < ad.N; ++j) {
      out.append(ad.ntseq, (size_t) (pos + j) * 5, 5);
      const int c = ad.codon[pos + j] == 6 ? 3 : ad.codon[pos + j];
      const long long c1 = fwd ? i2 : i2 - 1;
      i2 += fwd ? c : -c;
      int frame = 0;                                         // p7_alidiplay_frame (:3719-3735)
      if (ad.codon[pos + j] != 0 && ad.codon[pos + j] != 6) {
        if (c1 < i2) { frame = (int) ((i2 + 1) % 3); if (frame == 0) frame = 3; }
        else         { frame = -(int) (i2 % 3);      if (frame == 0) frame = -3; }
      }
      frameline.push_back(frame);
    }
    out += "  ";
    if (ni > 0) put(" %-*lld\n", coordwidth, i2); else put(" %*s\n", coordwidth, "-");
    if (show_frameline) {                                    // --frameline (:3998-4013)
      put("  %*s ", namewidth + coordwidth + 1, ""); out += "  ";
      for (size_t j = 0; j < frameline.size(); ++j) {
        if (frameline[j] > 0)                put("  %d  ", frameline[j]);
        else if (frameline[j] < 0)           put(" %d  ", frameline[j]);
        else if (ad.codon[pos + j] == 6)     put("  %d  ", frameline[j]);
        else                                 out += "  .  ";
      }
      out += "  "; out += " FRAME\n";
    }
    put("  %*s ", namewidth + coordwidth + 1, ""); out += "  "; row(ad.ppline, w); out += "  "; out += " PP\n";
    k1 += nk;
    i1 = fwd ? i2 + 1 : i2 - 1;
    pos += w;
  }
}

// The hit-dependent part of bathsearch's report: p7_tophits_Targets, two blank lines, p7_tophits_Domains (with alignments), two blank
// lines (src/p7_tophits.c:1073-1227, :1232-1410 as called from src/bathsearch.c:960-961) -- everything between the "Query:" block and
// "Internal pipeline statistics summary:".  textw = --textw (150 by default; 0 = --notextw).
extern "C" int bathhost_search_format_report(const bathhost_search *s, int textw, char *buf, size_t cap, size_t *needed)
{
  if (!s || !needed || (!buf && cap > 0)) return BATHHOST_EINVAL;
  const bathhost_model *m = s->model;
  const bool fs_pipe = s->opt.fs;
  const double incE = 0.01;                                // --incE (src/p7_pipeline.c:166)
  int namew = 8, posw = 6, nreported = 0;
  for (const Hit &h : s->hits) {                           // p7_tophits_GetMaxNameLength / GetMaxPositionLength run over all hits
    namew = std::max(namew, (int) strlen(h.pub.name));
    if (h.pub.ali_from > 0) {
      posw = std::max(posw, (int) std::to_string((long long) h.pub.ali_from).size());
      posw = std::max(posw, (int) std::to_string((long long) h.pub.ali_to).size());
    }
    if (h.reported) nreported++;
  }
  std::string out;
  char line[4096];
  auto put = [&](const char *fmt, auto... args) { snprintf(line, sizeof line, fmt, args...); out += line; };

  out += "Scores for complete hits:\n";
  if (fs_pipe) {
    put("  %9s %6s %5s  %-*s %*s %*s  %6s  %5s  %s\n", "E-value", " score", " bias", namew, "Sequence", posw, "start", posw, "end", "shifts", "stops", "Description");
    put("  %9s %6s %5s  %-*s %*s %*s  %6s  %5s  %s\n", "-------", "------", "-----", namew, "--------", posw, "-----", posw, "-----", "------", "-----", "-----------");
  } else {
    put("  %9s %6s %5s  %-*s %*s %*s  %s\n", "E-value", " score", " bias", namew, "Sequence", posw, "start", posw, "end", "Description");
    put("  %9s %6s %5s  %-*s %*s %*s  %s\n", "-------", "------", "-----", namew, "--------", posw, "-----", posw, "-----", "-----------");
  }
  bool printed_incthresh = false;
  for (const Hit &h : s->hits) {
    if (!h.reported) continue;
    if (!(h.pub.evalue <= incE) && !printed_incthresh) { out += "  ------ inclusion threshold ------\n"; printed_incthresh = true; }
    put("%c %9.2g %6.1f %5.1f  %-*s %*lld %*lld  ", ' ', h.pub.evalue, h.pub.score, h.pub.bias, namew, h.pub.name, posw, (long long) h.pub.ali_from,
        posw, (long long) h.pub.ali_to);
    if (fs_pipe) put("%6d  %5d", h.pub.shifts, h.pub.stops);
    put("  %s\n", "");
  }
  if (nreported == 0) out += "\n   [No hits detected that satisfy reporting thresholds]\n";
  out += "\n\n";

  out += "Annotation for each hit (and alignments):\n";
  for (const Hit &h : s->hits) {
    if (!h.reported) continue;
    put(">> %s  %s\n", h.pub.name, "");
    if (fs_pipe) {
      put("   %6s %5s %9s %10s %9s    %9s %9s    %6s  %5s %9s   %4s\n", "score", "bias", "   Evalue", "hmm-from", " hmm-to", " ali-from", "   ali-to",
          "shifts", "stops", "   sq-len", "acc");
      put("   %6s %5s %9s %10s %9s    %9s %9s    %6s  %5s %9s   %4s\n", "------", "-----", "---------", "--------", "-------", "---------", "---------",
          "------", "-----", "---------", "----");
    } else {
      put("   %6s %5s %9s %10s %9s    %9s %9s    %9s   %4s\n", "score", "bias", "   Evalue", "hmm-from", " hmm-to", " ali-from", "   ali-to", "   sq-len", "acc");
      put("   %6s %5s %9s %10s %9s    %9s %9s    %9s   %4s\n", "------", "-----", "---------", "--------", "-------", "---------", "---------", "---------", "----");
    }
    put(" %c %6.1f %5.1f %9.2g %10d %9d %c%c %9lld %9lld %c%c", (h.pub.evalue <= incE) ? '!' : '?', h.pub.score, h.pub.bias, h.pub.evalue,
        h.pub.hmm_from, h.pub.hmm_to, (h.pub.hmm_from == 1) ? '[' : '.', (h.pub.hmm_to == m->hmm.M) ? ']' : '.',
        (long long) h.pub.ali_from, (long long) h.pub.ali_to, (h.pub.ali_from == 1) ? '[' : '.', (h.pub.ali_to == h.pub.sq_len) ? ']' : '.');
    if (fs_pipe) put(" %6d  %5d", h.pub.shifts, h.pub.stops);
    put(" %9lld   %4.2f\n", (long long) h.pub.sq_len, (h.pub.oasc / (1.0 + fabs((float) (h.pub.env_to - h.pub.env_from) / 3))));
    out += "\n  Alignment:\n";
    put("  score: %.1f bits", h.pub.score);
    out += "\n";
    print_alidisplay(out, h.ad, m->hmm.name, h.pub.name, h.pub.hmm_from, h.pub.hmm_to, h.pub.ali_from, h.pub.ali_to, textw, s->opt.frameline);
    out += "\n";
  }
  if (nreported == 0) out += "\n   [No hits detected that satisfy reporting thresholds]\n";
  out += "\n\n";

  *needed = out.size() + 1;
  if (out.size() + 1 > cap) return buf ? BATHHOST_EINVAL : BATHHOST_OK;
  memcpy(buf, out.c_str(), out.size() + 1);
  return BATHHOST_OK;
}

// p7_tophits_TabularFrameshifts (src/p7_tophits.c:1442-1600), the --fstblout table: one line per frameshift ('I' / 'D' with its length)
// and per in-frame stop codon ('S') of every reported hit of the frameshift branch, with its position in the alignment and on the
// target.  Walks the alignment display's codon lengths, which are the trace's c values (6 = stop codon in a match state).
extern "C" int bathhost_search_format_fstblout(const bathhost_search *s, int show_header, char *buf, size_t cap, size_t *needed)
{
  if (!s || !needed || (!buf && cap > 0)) return BATHHOST_EINVAL;
  const bathhost_model *m = s->model;
  const std::string qname = m->hmm.name, qacc = m->hmm.acc;
  int tnamew = 20, posw = 9, nhits = 0;
  for (const Hit &h : s->hits) {
    tnamew = std::max(tnamew, (int) strlen(h.pub.name));
    if (h.pub.ali_from > 0) {
      posw = std::max(posw, (int) std::to_string((long long) h.pub.ali_from).size());
      posw = std::max(posw, (int) std::to_string((long long) h.pub.ali_to).size());
    }
    nhits++;
  }
  const int qnamew = std::max(20, (int) qname.size()), qaccw = std::max(10, (int) qacc.size()), taccw = 10;
  std::string out;
  char line[4096];
  auto put = [&](const char *fmt, auto... args) { snprintf(line, sizeof line, fmt, args...); out += line; };
  if (show_header && nhits > 0) {
    put("#%-*s %-*s %-*s %-*s %-9s %-*s %-*s  %5s %6s %-*s %9s\n", tnamew - 1, " target name", taccw, " accession", qnamew, " query name", qaccw,
        " accession", " E-value", posw, " ali from", posw, " ali to", " I D S", " length", posw, " seq start", " ali start");
    put("#%*s %*s %*s %*s %9s %-*s %-*s  %5s  %6s  %-*s  %9s\n", tnamew - 1, "-------------------", taccw, "-----------", qnamew, "--------------------",
        qaccw, "----------", "---------", posw, "---------", posw, "---------", "-----", "------", posw, "---------", "---------");
  }
  for (const Hit &h : s->hits) {
    if (!h.reported || !h.from_fs_branch) continue;
    const long long seq_from = h.pub.ali_from, seq_to = h.pub.ali_to;
    int ali_pos = 1;
    for (int z = 0; z < h.ad.N; ++z) {
      const bool is_match = h.ad.model[z] != '.' && h.ad.aseq[z] != '-';
      const bool is_insert = h.ad.model[z] == '.';
      if (!is_match) { if (is_insert) ali_pos += 3; continue; }
      const int c = h.ad.codon[z];
      char type = 0; int len = 0, adv = 3;
      if      (c == 1) { type = 'D'; len = 2; adv = 1; }
      else if (c == 2) { type = 'D'; len = 1; adv = 2; }
      else if (c == 6) { type = 'S'; len = 0; adv = 3; }
      else if (c == 4) { type = 'I'; len = 1; adv = 4; }
      else if (c == 5) { type = 'I'; len = 2; adv = 5; }
      if (type) {
        const long long seq_start = (seq_from < seq_to) ? seq_from + ali_pos - 1 : seq_from - ali_pos + 1;
        put(" %-*s %-*s %-*s %-*s %9.2g %-*lld %-*lld  %5c  %6d  %-*lld  %9d\n", tnamew, h.pub.name, taccw, "-", qnamew, qname.c_str(), qaccw,
            qacc.empty() ? "-" : qacc.c_str(), h.pub.evalue, posw, seq_from, posw, seq_to, type, len, posw, seq_start, ali_pos);
      }
      ali_pos += adv;
    }
  }
  *needed = out.size() + 1;
  if (out.size() + 1 > cap) return buf ? BATHHOST_EINVAL : BATHHOST_OK;
  memcpy(buf, out.c_str(), out.size() + 1);
  return BATHHOST_OK;
}

// One query's section of bathsearch's output without the lines that depend on the run (banner, option echo, timings): the "Query:"
// block (src/bathsearch.c:783-785), bathhost_search_format_report, and p7_pli_Statistics up to "Total number of hits"
// (src/p7_pipeline.c:1836-1874; n_output / pos_output as src/bathsearch.c:950-957).
extern "C" int bathhost_search_format_output(const bathhost_search *s, int textw, char *buf, size_t cap, size_t *needed)
{
  if (!s || !needed || (!buf && cap > 0)) return BATHHOST_EINVAL;
  const bathhost_model *m = s->model;
  std::string out;
  char line[1024];
  auto put = [&](const char *fmt, auto... args) { snprintf(line, sizeof line, fmt, args...); out += line; };
  put("Query:       %s  [M=%d]\n", m->hmm.name.c_str(), m->hmm.M);
  if (!m->hmm.acc.empty())  put("Accession:   %s\n", m->hmm.acc.c_str());
  if (!m->hmm.desc.empty()) put("Description: %s\n", m->hmm.desc.c_str());
  size_t need = 0;
  int st = bathhost_search_format_report(s, textw, nullptr, 0, &need);
  if (st != BATHHOST_OK) return st;
  std::vector<char> rep(need);
  if ((st = bathhost_search_format_report(s, textw, rep.data(), need, &need)) != BATHHOST_OK) return st;
  out += rep.data();
  long long n_output = 0, pos_output = 0;
  for (const Hit &h : s->hits) {
    if (!h.reported) continue;
    n_output++;
    pos_output += 1 + std::llabs((long long) h.pub.ali_to - (long long) h.pub.ali_from);
  }
  const bathhost_stats &t = s->st;
  const double denom = (double) t.nres;                     // nres * nmodels, one model per search object
  out += "Internal pipeline statistics summary:\n-------------------------------------\n";
  put("Query model(s):              %15lld  (%lld nodes)\n", 1LL, (long long) m->hmm.M);
  put("Target %-12s          %15lld  (%lld residues searched)\n", "sequence(s):", (long long) t.nseqs, (long long) t.nres);
  put("Residues passing SSV filter: %15lld  (%.3g); expected (%.3g)\n", (long long) t.pos_past_msv, (double) t.pos_past_msv / denom, s->opt.F1);
  put("Residues passing bias filter:%15lld  (%.3g); expected (%.3g)\n", (long long) t.pos_past_bias, (double) t.pos_past_bias / denom, s->opt.F1);
  put("Residues passing Vit filter: %15lld  (%.3g); expected (%.3g)\n", (long long) t.pos_past_vit, (double) t.pos_past_vit / denom, s->opt.F2);
  put("Residues passing Fwd filter: %15lld  (%.3g); expected (%.3g)\n", (long long) t.pos_past_fwd, (double) t.pos_past_fwd / denom, s->opt.F3);
  put("Total number of hits:        %15d  (%.3g)\n", (int) n_output, (double) pos_output / denom);
  *needed = out.size() + 1;
  if (out.size() + 1 > cap) return buf ? BATHHOST_EINVAL : BATHHOST_OK;
  memcpy(buf, out.c_str(), out.size() + 1);
  return BATHHOST_OK;
}

extern "C" int bathhost_search_get_stats(const bathhost_search *s, bathhost_stats *st)
{
  if (!s || !st) return BATHHOST_EINVAL;
  *st = s->st;
  return BATHHOST_OK;
}

// ------------------------------------------------------------------------------------------
// A profile library against one target (bathhost.h): one search per model over shared device contexts and a target made resident once.
struct bathhost_library_search {
  std::vector<bathhost_search *> s;
  std::vector<SeqRef> queue;
  std::string err;
  ~bathhost_library_search() { for (bathhost_search *x : s) delete x; }
};

namespace {

thread_local std::string g_library_err;

// The ORF screen of models i0 .. i0+g-1 over every unit of the resident target, one set call per unit: out[k][2 c + strand]
int screen_group(bathhost_library_search *ls, const std::vector<SeqRef> &seqs, const std::vector<Chunk> &chunks, const std::vector<BlockInfo> &lib_blocks,
                 size_t i0, size_t g, std::vector<std::vector<ScreenOut>> &out)
{
  bathhost_search *s0 = ls->s[i0];
  const Options &opt = s0->opt;
  std::vector<std::vector<BlockInfo>> mb(g);
  std::vector<double> min_bits(g);
  std::vector<bathgpu_filter_params> prm(g);
  std::vector<const uint8_t *> rbv(g);
  for (size_t k = 0; k < g; ++k) {
    bathhost_search *s = ls->s[i0 + k];
    long long nres = s->st.nres;
    mb[k] = cut_blocks(seqs, s->model->prot.max_length * 3, opt, nres);
    place_blocks(mb[k], chunks);
    grow_length_tables(s, lib_blocks);                      // the library's blocks are the longest any model has
    const float *ev = s->model->hmm.evparam;
    min_bits[k] = gumbel_invsurv(s->opt.F1, ev[EV_MMU], ev[EV_MLAMBDA]) - 0.02;      // as filter_unit asks of bathgpu_orfs_msv_screen
    prm[k] = filter_params(s); rbv[k] = s->model->prot.rbv.data();
  }
  std::vector<int> active;
  if (opt.top)    active.push_back(0);
  if (opt.bottom) active.push_back(1);
  out.assign(g, std::vector<ScreenOut>(chunks.size() * 2));
  return for_each_backend(s0, [&](int be) -> int {
    bathhost_search *s = s0;
    const bathhost_backend &BE = s0->bes[(size_t) be];
    BE_TRY(s, BE.load_filter_profile_set(BE.ctx, (int) g, prm.data(), rbv.data()), "bathgpu_load_filter_profile_set");
    int nth = 0;
    for (size_t c = (size_t) be; c < chunks.size(); c += s0->bes.size(), ++nth) {
      const Chunk &ch = chunks[c];
      const size_t nblk = (size_t) (ch.blk1 - ch.blk0);
      for (int sidx : active) {
        std::vector<std::vector<bathgpu_block>> bd(g, std::vector<bathgpu_block>(nblk));
        std::vector<bathgpu_screen_job> jobs(g);
        int maxlen = 1;
        for (size_t k = 0; k < g; ++k) {
          for (size_t b = 0; b < nblk; ++b) {
            const BlockInfo &blk = mb[k][(size_t) ch.blk0 + b];
            bd[k][b].goff = sidx ? ch.n - (blk.coff + blk.n) : blk.coff; bd[k][b].n = (blk.n >= 15) ? blk.n : 0; bd[k][b].C = blk.C;
            maxlen = std::max(maxlen, blk.n / 3 + 1);
          }
          jobs[k] = bathgpu_screen_job{ (int32_t) k, (int32_t) nblk, bd[k].data(), min_bits[k] };
        }
        std::vector<int64_t> norfs(g * nblk), nh(g), nr(g);
        BE_TRY(s, BE.select_slot(BE.ctx, 2 * nth + sidx), "bathgpu_select_slot");
        BE_TRY(s, BE.orfs_msv_screen_set(BE.ctx, jobs.data(), (int) g, sidx, s0->gcode, opt.min_orf, s0->tjb_tab.data(), s0->null_tab.data(), maxlen,
                                         norfs.data(), nh.data(), nr.data()), "bathgpu_orfs_msv_screen_set");
        int64_t tot_h = 0, tot_r = 0;
        for (size_t k = 0; k < g; ++k) { tot_h += nh[k]; tot_r += nr[k]; }
        std::vector<bathgpu_orf_hit> hits((size_t) tot_h);
        auto res = std::make_shared<std::vector<uint8_t>>((size_t) tot_r);
        BE_TRY(s, BE.orfs_fetch_set(BE.ctx, hits.data(), res->data()), "bathgpu_orfs_fetch_set");
        size_t z = 0;
        for (size_t k = 0; k < g; ++k) {
          ScreenOut &o = out[k][2 * c + (size_t) sidx];
          o.norfs.assign(norfs.begin() + (long) (k * nblk), norfs.begin() + (long) ((k + 1) * nblk));
          o.hits.assign(hits.begin() + (long) z, hits.begin() + (long) (z + (size_t) nh[k]));
          o.res = res;
          z += (size_t) nh[k];
        }
      }
    }
    return 0;
  });
}

int library_fail(bathhost_library_search *ls, int code, const std::string &msg) { ls->err = msg; return code; }

int library_run(bathhost_library_search *ls)
{
  std::vector<SeqRef> seqs;
  seqs.swap(ls->queue);
  if (seqs.empty()) return 0;
  bathhost_search *s0 = ls->s[0];
  const Options &opt = s0->opt;
  // chunks cut once, at block starts, each resident range reaching back by the largest context of the library
  int Cmax = 0;
  for (bathhost_search *s : ls->s) Cmax = std::max(Cmax, s->model->prot.max_length * 3);
  long long nres_unused = 0, total = 0;
  std::vector<BlockInfo> lib_blocks = cut_blocks(seqs, Cmax, opt, nres_unused);
  for (const BlockInfo &b : lib_blocks) total += b.n;
  SharedTarget shared;
  shared.chunks = cut_chunks(lib_blocks, chunk_target(s0, total));
  // each chunk uploaded (and its bottom strand made) once, on the context and in the slots run_batch deals it to
  int rc = for_each_backend(s0, [&](int be) -> int {
    HostBuf stage;
    int nth = 0;
    for (size_t c = (size_t) be; c < shared.chunks.size(); c += s0->bes.size(), ++nth) {
      const int st = upload_chunk(s0, s0->bes[(size_t) be], seqs, shared.chunks[c], 2 * nth, opt.bottom ? 2 * nth + 1 : -1, stage);
      if (st != 0) return st;
    }
    return 0;
  });
  if (rc != 0) return library_fail(ls, rc, s0->err);
  auto run_model = [&](size_t i, const std::vector<ScreenOut> *screen) -> int {
    bathhost_search *s = ls->s[i];
    int st = load_images(s);
    if (st != 0) return library_fail(ls, st, "model " + std::to_string(i) + ": loading its profiles failed: " +
                                             (s->bes[0].last_error ? s->bes[0].last_error(s->bes[0].ctx) : "?"));
    for (size_t k = 0; k < seqs.size(); ++k) {
      SeqRef r;
      r.name = seqs[k].name; r.dsq = seqs[k].dsq; r.n = seqs[k].n; r.seqidx = s->nseqs + (int64_t) k;
      s->queue.push_back(std::move(r));
    }
    s->finished = false;
    SharedTarget sh;
    sh.chunks = shared.chunks; sh.screen = screen;
    st = run_batch(s, &sh);
    return st != 0 ? library_fail(ls, st, "model " + std::to_string(i) + ": " + s->err) : 0;
  };
  bool set_screen = true;
  for (const bathhost_backend &BE : s0->bes) set_screen = set_screen && BE.load_filter_profile_set && BE.orfs_msv_screen_set && BE.orfs_fetch_set;
  const size_t n = ls->s.size();
  if (!set_screen) {
    for (size_t i = 0; i < n; ++i) if ((rc = run_model(i, nullptr)) != 0) return rc;
    return 0;
  }
  size_t group = std::min<size_t>(n, BATHGPU_SCREEN_SET_MAX_JOBS);
  for (size_t i0 = 0; i0 < n;) {
    const size_t g = std::min(group, n - i0);
    std::vector<std::vector<ScreenOut>> screens;
    rc = screen_group(ls, seqs, shared.chunks, lib_blocks, i0, g, screens);
    if (rc == BATHHOST_EMEM && g > 1) { group = g / 2; continue; }       // the device cannot hold this many at once: half the group
    if (rc != 0) return library_fail(ls, rc, ls->s[i0]->err);
    for (size_t k = 0; k < g; ++k) if ((rc = run_model(i0 + k, &screens[k])) != 0) return rc;
    i0 += g;
  }
  return 0;
}

}  // namespace

extern "C" int bathhost_search_create_library(const bathhost_model *const *models, int n, const bathhost_backend *be, int nbackends,
                                              const bathhost_options *opt, bathhost_library_search **ret)
{
  g_library_err.clear();
  if (!ret) return BATHHOST_EINVAL;
  *ret = nullptr;
  if (!models || n < 1 || !be || nbackends < 1) { g_library_err = "bad arguments to bathhost_search_create_library"; return BATHHOST_EINVAL; }
  std::unique_ptr<bathhost_library_search> ls(new (std::nothrow) bathhost_library_search());
  if (!ls) return BATHHOST_EMEM;
  for (int i = 0; i < n; ++i) {
    bathhost_search *s = nullptr;
    const int st = models[i] ? bathhost_search_create_multi(models[i], be, nbackends, opt, &s) : BATHHOST_EINVAL;
    if (st != BATHHOST_OK) {
      bathhost_model_info info;
      const bool named = models[i] && bathhost_model_get_info(models[i], &info) == BATHHOST_OK;
      g_library_err = "model " + std::to_string(i) + (named ? std::string(" (") + info.name + ")" : std::string()) + " refused: " +
                      (be[0].last_error ? be[0].last_error(be[0].ctx) : "status " + std::to_string(st));
      return st;
    }
    ls->s.push_back(s);
  }
  *ret = ls.release();
  return BATHHOST_OK;
}

extern "C" void bathhost_library_search_destroy(bathhost_library_search *ls) { delete ls; }
extern "C" const char *bathhost_library_search_last_error(const bathhost_library_search *ls) { return ls ? ls->err.c_str() : g_library_err.c_str(); }

extern "C" int bathhost_library_search_queue(bathhost_library_search *ls, const char *name, const uint8_t *dsq, int64_t n)
{
  if (!ls || !dsq || n < 1) return BATHHOST_EINVAL;
  SeqRef r;
  r.name = name ? name : ""; r.dsq = dsq; r.n = n;
  ls->queue.push_back(std::move(r));
  return BATHHOST_OK;
}

extern "C" int bathhost_library_search_run(bathhost_library_search *ls) { return ls ? library_run(ls) : BATHHOST_EINVAL; }

extern "C" int bathhost_library_search_finish(bathhost_library_search *ls)
{
  if (!ls) return BATHHOST_EINVAL;
  int st = library_run(ls);
  for (size_t i = 0; st == BATHHOST_OK && i < ls->s.size(); ++i)
    if ((st = bathhost_search_finish(ls->s[i])) != BATHHOST_OK) ls->err = "model " + std::to_string(i) + ": " + ls->s[i]->err;
  return st;
}

extern "C" bathhost_search *bathhost_library_search_get(bathhost_library_search *ls, int i)
{
  return (ls && i >= 0 && (size_t) i < ls->s.size()) ? ls->s[(size_t) i] : nullptr;
}
