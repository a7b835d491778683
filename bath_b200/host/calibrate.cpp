// calibrate.cpp -- E-value calibration of a query model by brief simulation, batched onto the device library.
//
// What bathbuild (p7_Calibrate, src/evalues.c:64-183) and bathconvert / bathfetch (src/bathconvert.c:128-161,
// src/bathfetch.c:295-325) do once per model: score 200 random sequences with each of the hot-path kernels and fit the
// location of the score distribution.  The reference makes 1000 single-sequence kernel calls per model; here the host draws
// all sequences of a simulation first (the generator is one serial chain) and each simulation is ONE batched stage call:
//   p7_MSVMu           src/evalues.c:297-340   200 x 200 aa  -> bathgpu_msv_orfs
//   p7_ViterbiMu       src/evalues.c:366-411   200 x 200 aa  -> bathgpu_vit_orfs
//   p7_Tau             src/evalues.c:536-581   200 x 100 aa  -> bathgpu_fwd_orfs
//   p7_fs_Tau_3codons  src/evalues.c:607-680   200 x 300 nt  -> bathgpu_fs_fwd_windows
//   p7_fs_Tau_5codons  src/evalues.c:703-776   200 x 300 nt  -> bathgpu_fs_forward_matrices (scores only)
// A sequence whose frameshift Forward score overflows is replaced by the next one the generator yields (:649, :759), so the
// batch is topped up from the running generator until 200 scores are in.
//
// Easel pieces restated (Easel is not in the reference tree): esl_randomness_CreateFast / esl_random, esl_rsq_xfIID
// (esl_rnd_FChoose per residue), esl_rnd_Roll, esl_vec_FRelEntropy, esl_gumbel_FitComplete / FitCompleteLoc / invcdf.
// Pinned: the STATS lines of the shipped models come out to the printed precision (tests/test_calibration.py).
#include <cmath>
#include <cstring>
#include <vector>

#include "../../include/bathhost.h"
#include "../../include/bathgpu.h"
#include "host_internal.h"
#include "model_internal.h"

using namespace bathhost;

namespace {

constexpr double kLog2 = 0.69314718055994529;

struct FastRng {                       // esl_randomness_CreateFast: x <- 69069 x + 1, seed dispersed by Jenkins' mix
  uint32_t x;
  explicit FastRng(uint32_t seed)
  {
    uint32_t a = seed, b = 87654321u, c = 12345678u;
    a -= b; a -= c; a ^= (c >> 13);  b -= c; b -= a; b ^= (a << 8);   c -= a; c -= b; c ^= (b >> 13);
    a -= b; a -= c; a ^= (c >> 12);  b -= c; b -= a; b ^= (a << 16);  c -= a; c -= b; c ^= (b >> 5);
    a -= b; a -= c; a ^= (c >> 3);   b -= c; b -= a; b ^= (a << 10);  c -= a; c -= b; c ^= (b >> 15);
    x = c ? c : 42u;
  }
  double next() { x = x * 69069u + 1u; return (double) x / 4294967296.0; }
  int choose(const float *p, int n)    // esl_rnd_FChoose
  {
    const double roll = next();
    double sum = 0.0;
    for (int i = 0; i < n; ++i) { sum += p[i]; if (roll < sum) return i; }
    int i;
    do { i = (int) (next() * n); } while (p[i] == 0.0f);
    return i;
  }
  int roll(int n) { return (int) (next() * n); }   // esl_rnd_Roll
};

struct CodonTable {                    // p7_codontable_Create (src/hmmer.c:197-243): codons per amino acid in x, y, z order
  uint8_t nt[kK][6][3];
  int     n[kK];
  explicit CodonTable(const uint8_t gcode[64])
  {
    memset(n, 0, sizeof n);
    for (int c = 0; c < 64; ++c) {
      const int a = gcode[c];
      if (a < kK && n[a] < 6) { nt[a][n[a]][0] = (uint8_t) (c >> 4); nt[a][n[a]][1] = (uint8_t) ((c >> 2) & 3); nt[a][n[a]][2] = (uint8_t) (c & 3); ++n[a]; }
    }
  }
};

double fit_complete_loc(const std::vector<double> &x, double lambda)
{
  double esum = 0.0;
  for (double v : x) esum += exp(-lambda * v);
  return -log(esum / (double) x.size()) / lambda;
}

// esl_gumbel_FitComplete: Newton-Raphson on Lawless' eq. 4.1.6 from the method-of-moments start, then eq. 4.1.5
void fit_complete(const std::vector<double> &x, double *mu, double *lambda)
{
  const int n = (int) x.size();
  double mean = 0.0, var = 0.0;
  for (double v : x) mean += v;
  mean /= n;
  for (double v : x) var += (v - mean) * (v - mean);
  var /= (n - 1);
  double lam = 3.14159265358979323846 / sqrt(6.0 * var);
  for (int it = 0; it < 100; ++it) {
    double esum = 0., xesum = 0., xxesum = 0., xsum = 0.;
    for (double v : x) { const double e = exp(-lam * v); xsum += v; esum += e; xesum += v * e; xxesum += v * v * e; }
    const double fx  = (1.0 / lam) - (xsum / n) + (xesum / esum);
    const double dfx = ((xesum / esum) * (xesum / esum)) - (xxesum / esum) - (1.0 / (lam * lam));
    if (fabs(fx) < 1e-5) break;
    lam -= fx / dfx;
    if (lam <= 0.0) lam = 0.001;
  }
  *lambda = lam;
  *mu = fit_complete_loc(x, lam);
}

double tau_of(const std::vector<double> &x, double lambda, double tailp)     // src/evalues.c:561-568
{
  double gmu, glam;
  fit_complete(x, &gmu, &glam);
  return (gmu - log(-log(1.0 - tailp)) / glam) + log(tailp) / lambda;
}

// esl_rsq_xfIID of a random protein, reverse-translated with uniformly drawn synonymous codons (src/evalues.c:634-647): n sequences
// of 3 L nucleotides, one after the other from dst
void draw_reverse_translated(const bathhost_model *m, const CodonTable &tbl, FastRng &rng, int L, int n, uint8_t *dst)
{
  std::vector<uint8_t> amino(L);
  for (int i = 0; i < n; ++i) {
    for (int a = 0; a < L; ++a) amino[a] = (uint8_t) rng.choose(m->bg.f, kK);
    uint8_t *d = dst + (size_t) i * 3 * L;
    for (int a = 0; a < L; ++a, d += 3) memcpy(d, tbl.nt[amino[a]][rng.roll(tbl.n[amino[a]])], 3);
  }
}

float null_one(int L)      { const float p1 = (float) L / (float) (L + 1); return (float) L * log(p1) + log(1. - p1); }      // p7_bg_SetLength + p7_bg_NullOne
float fs_null_one(int La)  { return null_one(La) + log(3.0); }                                                               // p7_bg_fs_NullOne (src/p7_bg.c:377-384)

}  // namespace

// p7_Lambda (src/evalues.c:243-250): log 2 + 1.44 / (M H), H = mean relative entropy (bits) of the match emissions
extern "C" double bathhost_model_lambda(const bathhost_model *m)
{
  if (!m) return 0.0;
  const CoreModel &h = m->hmm;
  double KL = 0.0;
  for (int k = 1; k <= h.M; ++k) {
    float kl = 0.0f;
    const float *p = &h.mat[(size_t) k * kK];
    for (int x = 0; x < kK; ++x) if (p[x] > 0.0f) kl += p[x] * log(p[x] / m->bg.f[x]);
    KL += kl / kLog2;
  }
  KL /= (double) h.M;
  return kLog2 + 1.44 / ((double) h.M * KL);
}

extern "C" int bathhost_calibrate(const bathhost_model *m, const bathhost_backend *be, bathhost_calibration *cal, double evparam[8])
{
  if (!m || !be || !cal || !evparam || !be->ctx) return BATHHOST_EINVAL;
  const int EmL = 200, EmN = 200, EvL = 200, EvN = 200, EfL = 100, EfN = 200;     // p7_builder.c:116-122
  const double Eft = 0.04;
  const int mask = cal->which_mask ? cal->which_mask : 31;
  const ProteinProfile &q = m->prot;
  const int M = m->hmm.M;
  uint8_t gcode[64];
  if (!genetic_code(m->ct, gcode)) return BATHHOST_EINVAL;
  const CodonTable tbl(gcode);

  double lambda = cal->lambda;
  if (lambda <= 0.0) lambda = (cal->convert_flow && m->hmm.evparam[EV_FLAMBDA] > 0.0f) ? (double) m->hmm.evparam[EV_FLAMBDA] : bathhost_model_lambda(m);
  for (int z = 0; z < 8; ++z) evparam[z] = -99999.0;
  evparam[EV_MLAMBDA] = evparam[EV_VLAMBDA] = evparam[EV_FLAMBDA] = lambda;

  // device images of the query, as bathhost_search_create loads them
  int st;
  if ((st = be->load_fs_profile(be->ctx, 3, M, m->om3.nrows, m->om3.rfv.data(), m->om3.tfv.data())) != 0 ||
      (st = be->load_fs_profile(be->ctx, 5, M, m->om5.nrows, m->om5.rfv.data(), m->om5.tfv.data())) != 0) return st;
  bathgpu_filter_params fp;
  fp.M = M; fp.tbm_b = q.tbm_b; fp.tec_b = q.tec_b; fp.base_b = q.base_b; fp.bias_b = q.bias_b; fp.scale_b = q.scale_b;
  fp.base_w = q.base_w; fp.ddbound_w = q.ddbound_w; fp.xw_E_move = q.xw_E_move; fp.xw_E_loop = q.xw_E_loop; fp.scale_w = q.scale_w;
  fp.cpu_lanes_u8 = 16; fp.cpu_lanes_i16 = 8;
  if ((st = be->load_filter_profile(be->ctx, &fp, q.rbv.data(), q.rwv.data(), q.twv.data())) != 0) return st;

  FastRng rng(cal->seed ? cal->seed : 42u);
  if (cal->convert_flow && cal->rng_state) rng.x = cal->rng_state;

  std::vector<uint8_t> res;
  std::vector<bathgpu_orf> desc;
  std::vector<float> sc;
  std::vector<int32_t> status;
  std::vector<double> xv;

  // one protein simulation: N sequences of L residues drawn, uploaded and scored by one stage call
  auto protein_batch = [&](int L, int N, bool run) -> int {
    res.resize((size_t) N * L);
    for (size_t z = 0; z < res.size(); ++z) res[z] = (uint8_t) rng.choose(m->bg.f, kK);     // esl_rsq_xfIID
    if (!run) return 0;
    desc.assign(N, bathgpu_orf());
    for (int i = 0; i < N; ++i) {
      memset(&desc[i], 0, sizeof(bathgpu_orf));
      desc[i].offset = (int64_t) i * L; desc[i].L = L;
      desc[i].tjb_b = q.tjb_for_length(L); desc[i].xw_move = q.xw_move_for_length(L);      // p7_oprofile_ReconfigLength(om, L)
    }
    sc.assign(N, 0.0f); status.assign(N, 0);
    return be->upload_orfs(be->ctx, res.data(), (int64_t) res.size());
  };

  if (!cal->convert_flow) {
    // p7_MSVMu
    if ((st = protein_batch(EmL, EmN, mask & 1)) != 0) return st;
    if (mask & 1) {
      if ((st = be->msv_orfs(be->ctx, desc.data(), EmN, sc.data(), status.data())) != 0) return st;
      const float maxsc = (255 - q.base_b) / q.scale_b, nullsc = null_one(EmL);
      xv.resize(EmN);
      for (int i = 0; i < EmN; ++i) xv[i] = ((status[i] == BATHGPU_ERANGE ? maxsc : sc[i]) - nullsc) / kLog2;
      evparam[EV_MMU] = fit_complete_loc(xv, lambda);
    }
    // p7_ViterbiMu
    if ((st = protein_batch(EvL, EvN, mask & 2)) != 0) return st;
    if (mask & 2) {
      int nw = 0;
      if ((st = be->vit_orfs(be->ctx, desc.data(), EvN, sc.data(), status.data(), nullptr, 0, &nw)) != 0) return st;
      const float maxsc = (32767.0 - q.base_w) / q.scale_w, nullsc = null_one(EvL);
      xv.resize(EvN);
      for (int i = 0; i < EvN; ++i) xv[i] = ((status[i] == BATHGPU_ERANGE ? maxsc : sc[i]) - nullsc) / kLog2;
      evparam[EV_VMU] = fit_complete_loc(xv, lambda);
    }
    // p7_Tau
    if ((st = protein_batch(EfL, EfN, mask & 4)) != 0) return st;
    if (mask & 4) {
      const float xfE[2] = { expf(q.xsc_E_move), expf(q.xsc_E_loop) };
      if ((st = be->fwd_orfs(be->ctx, desc.data(), EfN, q.nj, xfE, sc.data(), status.data())) != 0) return st;
      const float nullsc = null_one(EfL);
      xv.resize(EfN);
      for (int i = 0; i < EfN; ++i) { if (status[i] != 0) return status[i]; xv[i] = (sc[i] - nullsc) / kLog2; }
      evparam[EV_FTAU] = tau_of(xv, lambda, Eft);
    }
  }

  // the two frameshift simulations: random proteins reverse-translated with uniformly drawn synonymous codons
  // (src/evalues.c:634-647); the length model is set from the AMINO length (:628), null model p7_bg_fs_NullOne(EfL)
  const int Ln = 3 * EfL;
  std::vector<uint8_t> dna;
  std::vector<bathgpu_window> wins;
  auto frameshift_simulation = [&](int which, bool run, double *tau) -> int {
    xv.clear();
    float pmove, ploop;
    bathhost_length_model(EfL, 1.0f, &pmove, &ploop);                 // p7_fs_oprofile_ReconfigLength(om_fs, EfL), multihit
    const float nullsc = fs_null_one(EfL);
    int need = EfN, rounds = 0;
    while (need > 0) {
      if (++rounds > 64) return BATHHOST_EFAIL;             // every score overflows: the reference would draw for ever (:649)
      dna.assign((size_t) need * Ln + 2, 255);
      draw_reverse_translated(m, tbl, rng, EfL, need, &dna[1]);
      if (!run) return 0;
      if ((st = be->select_slot(be->ctx, 0)) != 0 || (st = be->upload_block(be->ctx, dna.data(), (int64_t) need * Ln)) != 0) return st;
      sc.assign(need, 0.0f); status.assign(need, 0);
      if (which == 3) {
        wins.resize(need);
        for (int i = 0; i < need; ++i) { wins[i].start = 1 + (int64_t) i * Ln; wins[i].L = Ln; wins[i].pmove = pmove; wins[i].ploop = ploop; }
        const float xfE[2] = { m->om3.xfE_move, m->om3.xfE_loop };
        if ((st = be->fs_fwd_windows(be->ctx, wins.data(), need, xfE, sc.data(), status.data())) != 0) return st;
      } else {
        std::vector<bathgpu_envelope> env(need);
        for (int i = 0; i < need; ++i) { env[i].start = 1 + (int64_t) i * Ln; env[i].L = Ln; env[i].pmove = pmove; env[i].ploop = ploop; }
        const float xfE[2] = { m->om5.xfE_move, m->om5.xfE_loop };
        if ((st = be->fs_forward_matrices(be->ctx, env.data(), need, xfE, nullptr, nullptr, 0, sc.data(), status.data())) != 0) return st;
      }
      int got = 0;
      for (int i = 0; i < need; ++i) {
        if (status[i] == BATHGPU_ERANGE) continue;
        if (status[i] != 0) return status[i];
        xv.push_back((sc[i] - nullsc) / kLog2); ++got;
      }
      need -= got;
    }
    *tau = tau_of(xv, lambda, Eft);
    return 0;
  };
  if ((st = frameshift_simulation(3, mask & 8,  &evparam[EV_FTAUFS3])) != 0) return st;
  if ((st = frameshift_simulation(5, mask & 16, &evparam[EV_FTAUFS5])) != 0) return st;
  cal->rng_state = rng.x;
  return BATHHOST_OK;
}

uint32_t bathhost::calibration_generator(uint32_t seed) { return FastRng(seed ? seed : 42u).x; }

bool bathhost::draw_fs_sequences(const bathhost_model *m, uint32_t *state, int n, uint8_t *dna)
{
  uint8_t gcode[64];
  if (!genetic_code(m->ct, gcode)) return false;
  const CodonTable tbl(gcode);
  FastRng rng(42u);
  rng.x = *state;
  draw_reverse_translated(m, tbl, rng, kFsSimL, n, dna);
  *state = rng.x;
  return true;
}

double bathhost::fs_tau(const float *sc, int n, double lambda)
{
  const float nullsc = fs_null_one(kFsSimL);
  std::vector<double> xv(n);
  for (int i = 0; i < n; ++i) xv[i] = (sc[i] - nullsc) / kLog2;
  return tau_of(xv, lambda, 0.04);
}
