// convert.cpp -- HMMER3/f profile libraries to BATH3/f (libbathhost.so).
//
// What bathconvert does per model (src/bathconvert.c:128-161) over a whole library: a BATH3/f model is a HMMER3/f one plus the FS3 /
// FS5 Forward taus, the frameshift probability and the codon table.  The model text is spliced, not rewritten from parsed fields, so
// every other byte stays as hmmbuild wrote it.
//
// The taus come from bathconvert's two frameshift simulations on one generator that runs from model to model.  A model's draws depend
// on its scores only where a score overflows and the sequence is replaced by the next one drawn (src/evalues.c:649, :759), so the
// sequences of a batch of models are drawn optimistically in file order and scored by one set call per codon length.  If model j of
// the batch has an overflow, models before j stand, model j runs through bathhost_calibrate from the generator state it starts at,
// and the next batch starts after it: the output is that of the serial chain in every case.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../../include/bathhost.h"
#include "../../include/bathgpu.h"
#include "host_internal.h"
#include "model_internal.h"

using namespace bathhost;

namespace {

thread_local std::string g_err;

int failf(int code, const char *fmt, ...)
{
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

std::string first_token(const std::string &line)
{
  std::istringstream ss(line);
  std::string t;
  ss >> t;
  return t;
}

// The next model's lines, header to "//".  BATHHOST_EOF at the clean end of the file.
int next_record(std::istream &in, std::vector<std::string> &lines, long &lineno)
{
  lines.clear();
  std::string line;
  while (std::getline(in, line)) {
    ++lineno;
    if (line.find_first_not_of(" \t\r") == std::string::npos) continue;
    const std::string tag = first_token(line);
    if (tag != "HMMER3/f")
      return failf(BATHHOST_EFORMAT, "line %ld: format \"%s\" is not converted: the input must be HMMER3/f", lineno, tag.c_str());
    lines.push_back(line);
    while (std::getline(in, line)) {
      ++lineno;
      lines.push_back(line);
      if (line.rfind("//", 0) == 0) return BATHHOST_OK;
    }
    return failf(BATHHOST_EFORMAT, "line %ld: the model that starts at line %ld has no \"//\" line", lineno, lineno - (long) lines.size() + 1);
  }
  return BATHHOST_EOF;
}

std::string joined(const std::vector<std::string> &lines)
{
  std::string s;
  for (const std::string &l : lines) { s += l; s += '\n'; }
  return s;
}

// index of the model's "STATS LOCAL FORWARD" line in its header, -1 if it has none
int forward_stats_line(const std::vector<std::string> &lines)
{
  for (size_t z = 1; z < lines.size(); ++z) {
    std::istringstream ss(lines[z]);
    std::string a, b, c;
    ss >> a >> b >> c;
    if (a == "HMM") break;
    if (a == "STATS" && b == "LOCAL" && c == "FORWARD") return (int) z;
  }
  return -1;
}

std::string line_of(const char *fmt, ...)
{
  char buf[256];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  return buf;
}

struct Pending {
  std::vector<std::string> lines;
  bathhost_model *m = nullptr;
  int fwd_line = -1;
  double lambda = 0.0, tau3 = 0.0, tau5 = 0.0;
};

// the model's BATH3/f text: the evparam floats printed as the profile writer prints them
void write_model(std::ostream &out, const Pending &p, float fsprob, int ct)
{
  out << "BATH3/f\n";
  for (size_t z = 1; z < p.lines.size(); ++z) {
    out << p.lines[z] << '\n';
    if ((int) z == p.fwd_line) {
      out << line_of("STATS LOCAL FS3 FORWARD %8.4f %8.5f\n", (float) p.tau3, (float) p.lambda);
      out << line_of("STATS LOCAL FS5 FORWARD %8.4f %8.5f\n", (float) p.tau5, (float) p.lambda);
      out << line_of("FRAMESHIFT PROB  %8.4f\n", fsprob);
      out << line_of("CODON TABLE  %d\n", ct);
    }
  }
}

// Models scored together: at most this many, and at most this many bytes of the two codon lengths' odds tables (a 5-codon image is
// nrows x (M+1) floats).  A device that cannot hold a batch's set refuses the load (BATHGPU_EMEM) and the batch is halved.
constexpr int    kBatchModels = 128;
constexpr size_t kBatchBytes  = (size_t) 1 << 30;

size_t image_bytes(const bathhost_model *m)
{
  return (size_t) (m->om3.nrows + m->om5.nrows) * (size_t) (m->hmm.M + 1) * sizeof(float);
}

// One model by the serial path, from generator state *state
int calibrate_one(Pending &p, const bathhost_backend *be, uint32_t seed, uint32_t *state)
{
  bathhost_calibration cal;
  memset(&cal, 0, sizeof cal);
  cal.seed = seed; cal.rng_state = *state; cal.convert_flow = 1; cal.which_mask = 24;
  double ev[8];
  const int st = bathhost_calibrate(p.m, be, &cal, ev);
  if (st != BATHHOST_OK) return failf(st, "model %s: calibration failed (status %d)", p.m->hmm.name.c_str(), st);
  p.tau3 = ev[EV_FTAUFS3]; p.tau5 = ev[EV_FTAUFS5]; p.lambda = ev[EV_FLAMBDA];
  *state = cal.rng_state;
  return BATHHOST_OK;
}

const char *backend_error(const bathhost_backend *be) { return be->last_error ? be->last_error(be->ctx) : ""; }

// Models [0, n) of the batch, their set images loaded: scored together while nothing overflows (see the top of the file)
int calibrate_batch(std::vector<Pending> &B, int n, const bathhost_backend *be, uint32_t seed, uint32_t *state)
{
  const int N = kFsSimN, Ln = 3 * kFsSimL;
  float pmove, ploop;
  bathhost_length_model(kFsSimL, 1.0f, &pmove, &ploop);          // p7_fs_oprofile_ReconfigLength(om_fs, EfL), multihit
  std::vector<float> xf3(2 * (size_t) n), xf5(2 * (size_t) n);
  for (int j = 0; j < n; ++j) {
    xf3[2 * j] = B[j].m->om3.xfE_move; xf3[2 * j + 1] = B[j].m->om3.xfE_loop;
    xf5[2 * j] = B[j].m->om5.xfE_move; xf5[2 * j + 1] = B[j].m->om5.xfE_loop;
  }
  std::vector<uint8_t> dna;
  std::vector<uint32_t> start_state(n);
  std::vector<bathgpu_set_window> w3, w5;
  std::vector<float> sc3, sc5;
  std::vector<int32_t> st3, st5;
  int j0 = 0;
  while (j0 < n) {
    const int k = n - j0;
    // draws of models j0 .. n-1 in file order: FS3 then FS5 sequences of each, one block
    dna.assign((size_t) k * 2 * N * Ln + 2, 255);
    w3.resize((size_t) k * N); w5.resize((size_t) k * N);
    for (int j = j0; j < n; ++j) {
      if (*state == 0) *state = calibration_generator(seed);     // bathhost_calibrate's reading of rng_state 0
      start_state[j] = *state;
      const size_t base = (size_t) (j - j0) * 2 * N * Ln;
      if (!draw_fs_sequences(B[j].m, state, N, &dna[1 + base]) || !draw_fs_sequences(B[j].m, state, N, &dna[1 + base + (size_t) N * Ln]))
        return failf(BATHHOST_EINVAL, "model %s: codon table %d is not supported", B[j].m->hmm.name.c_str(), B[j].m->ct);
      for (int i = 0; i < N; ++i) {
        bathgpu_set_window &a = w3[(size_t) (j - j0) * N + i], &b = w5[(size_t) (j - j0) * N + i];
        a.start = 1 + (int64_t) (base + (size_t) i * Ln);       b.start = a.start + (int64_t) N * Ln;
        a.L = b.L = Ln; a.pmove = b.pmove = pmove; a.ploop = b.ploop = ploop; a.profile = b.profile = j;
      }
    }
    int st;
    if ((st = be->select_slot(be->ctx, 0)) != 0 || (st = be->upload_block(be->ctx, dna.data(), (int64_t) dna.size() - 2)) != 0)
      return failf(st, "block upload failed: %s", backend_error(be));
    const int nw = k * N;
    sc3.assign(nw, 0.0f); sc5.assign(nw, 0.0f); st3.assign(nw, 0); st5.assign(nw, 0);
    if ((st = be->fs_set_scores(be->ctx, 3, w3.data(), nw, xf3.data(), sc3.data(), st3.data())) != 0 ||
        (st = be->fs_set_scores(be->ctx, 5, w5.data(), nw, xf5.data(), sc5.data(), st5.data())) != 0)
      return failf(st, "set scores failed: %s", backend_error(be));
    int j = j0;
    for (; j < n; ++j) {
      const size_t o = (size_t) (j - j0) * N;
      bool overflow = false;
      for (int i = 0; i < N && !overflow; ++i) {
        if ((st3[o + i] != 0 && st3[o + i] != BATHGPU_ERANGE) || (st5[o + i] != 0 && st5[o + i] != BATHGPU_ERANGE))
          return failf(BATHHOST_EFAIL, "model %s: status %d / %d from the set scores", B[j].m->hmm.name.c_str(), st3[o + i], st5[o + i]);
        overflow = st3[o + i] == BATHGPU_ERANGE || st5[o + i] == BATHGPU_ERANGE;
      }
      if (overflow) break;
      B[j].tau3 = fs_tau(&sc3[o], N, B[j].lambda);
      B[j].tau5 = fs_tau(&sc5[o], N, B[j].lambda);
    }
    if (j == n) return BATHHOST_OK;                  // *state is where the last model's draws left the generator
    // model j saw an overflow: the serial path from its own start, then the rest drawn again from where it leaves the generator
    *state = start_state[j];
    if ((st = calibrate_one(B[j], be, seed, state)) != BATHHOST_OK) return st;
    j0 = j + 1;
  }
  return BATHHOST_OK;
}

int load_sets(std::vector<Pending> &B, int n, const bathhost_backend *be)
{
  std::vector<int> M(n), r3(n), r5(n);
  std::vector<const float *> f3(n), t3(n), f5(n), t5(n);
  for (int j = 0; j < n; ++j) {
    const bathhost_model *m = B[j].m;
    M[j] = m->hmm.M;
    r3[j] = m->om3.nrows; f3[j] = m->om3.rfv.data(); t3[j] = m->om3.tfv.data();
    r5[j] = m->om5.nrows; f5[j] = m->om5.rfv.data(); t5[j] = m->om5.tfv.data();
  }
  int st = be->load_fs_profile_set(be->ctx, 3, n, M.data(), r3.data(), f3.data(), t3.data());
  if (st == 0) st = be->load_fs_profile_set(be->ctx, 5, n, M.data(), r5.data(), f5.data(), t5.data());
  return st;
}

}  // namespace

extern "C" const char *bathhost_convert_last_error(void) { return g_err.c_str(); }

extern "C" int bathhost_convert(const char *in_path, const char *out_path, int ct, float fsprob, uint32_t seed,
                                const bathhost_backend *be, int *nmodels)
{
  g_err.clear();
  if (nmodels) *nmodels = 0;
  if (!in_path || !out_path || !be || !be->ctx) return failf(BATHHOST_EINVAL, "bad arguments to bathhost_convert");
  if (ct == 0) ct = 1;
  if (fsprob == 0.0f) fsprob = 0.01f;
  uint8_t gcode[64];
  if (!genetic_code(ct, gcode)) return failf(BATHHOST_EINVAL, "codon table %d is not supported", ct);
  if (!(fsprob > 0.0f && fsprob < 0.25f)) return failf(BATHHOST_EINVAL, "frameshift probability %g is outside (0, 0.25)", fsprob);
  const bool batched = be->load_fs_profile_set && be->fs_set_scores;

  std::ifstream in(in_path);
  if (!in) return failf(BATHHOST_EFAIL, "cannot open %s", in_path);
  const std::string tmp = std::string(out_path) + ".partial";
  std::ofstream out(tmp, std::ios::binary);
  if (!out) return failf(BATHHOST_EFAIL, "cannot write %s", tmp.c_str());
  std::vector<Pending> B;
  auto give_up = [&](int st) {
    for (Pending &p : B) bathhost_model_destroy(p.m);
    out.close();
    std::remove(tmp.c_str());
    return st;
  };

  uint32_t state = 0;                  // 0: a fresh generator from seed, as bathhost_calibrate reads it
  long lineno = 0;
  int done = 0, batch_cap = kBatchModels;
  bool eof = false;
  std::vector<std::vector<std::string>> texts;
  while (true) {
    // the next batch: records read in one pass, models set up on the host cores
    texts.clear();
    while (!eof && (int) (B.size() + texts.size()) < batch_cap) {
      std::vector<std::string> lines;
      const int st = next_record(in, lines, lineno);
      if (st == BATHHOST_EOF) { eof = true; break; }
      if (st != BATHHOST_OK) return give_up(st);
      texts.push_back(std::move(lines));
    }
    const size_t first_new = B.size();
    B.resize(first_new + texts.size());
    std::vector<int> status(texts.size(), BATHHOST_OK);
    std::atomic<size_t> next(0);
    auto worker = [&]() {
      for (size_t z; (z = next++) < texts.size();) {
        Pending &p = B[first_new + z];
        p.lines = std::move(texts[z]);
        p.fwd_line = forward_stats_line(p.lines);
        if (p.fwd_line < 0) { status[z] = BATHHOST_EFORMAT; continue; }
        status[z] = model_from_record(joined(p.lines), ct, fsprob, &p.m);
        if (status[z] == BATHHOST_OK)
          p.lambda = (p.m->hmm.evparam[EV_FLAMBDA] > 0.0f) ? (double) p.m->hmm.evparam[EV_FLAMBDA] : bathhost_model_lambda(p.m);
      }
    };
    const size_t nthr = std::max<size_t>(1, std::min<size_t>(texts.size(), std::max(1u, std::thread::hardware_concurrency())));
    std::vector<std::thread> pool;
    for (size_t t = 1; t < nthr; ++t) pool.emplace_back(worker);
    worker();
    for (std::thread &t : pool) t.join();
    for (size_t z = 0; z < texts.size(); ++z)
      if (status[z] != BATHHOST_OK)
        return give_up(failf(status[z], "model %d of %s: %s", done + (int) (first_new + z) + 1, in_path,
                             B[first_new + z].fwd_line < 0 ? "no STATS LOCAL FORWARD line" : "cannot be read or set up"));
    if (B.empty()) break;

    int n = 1;
    size_t bytes = image_bytes(B[0].m);
    while (n < (int) B.size() && bytes + image_bytes(B[n].m) <= kBatchBytes) bytes += image_bytes(B[n++].m);
    if (batched) {
      int st;
      while ((st = load_sets(B, n, be)) == BATHHOST_EMEM && n > 1) n = (n + 1) / 2;      // what the device holds
      if (st != 0) return give_up(failf(st, "loading a set of %d profiles failed: %s", n, backend_error(be)));
      if (n < batch_cap) batch_cap = n;
      if ((st = calibrate_batch(B, n, be, seed, &state)) != BATHHOST_OK) return give_up(st);
    } else {
      for (int j = 0; j < n; ++j) {
        const int st = calibrate_one(B[j], be, seed, &state);
        if (st != BATHHOST_OK) return give_up(st);
      }
    }
    for (int j = 0; j < n; ++j) {
      write_model(out, B[j], fsprob, ct);
      bathhost_model_destroy(B[j].m);
    }
    B.erase(B.begin(), B.begin() + n);
    done += n;
    if (eof && B.empty()) break;
  }
  out.close();
  if (!out) return give_up(failf(BATHHOST_EFAIL, "writing %s failed", tmp.c_str()));
  if (done == 0) return give_up(failf(BATHHOST_EFORMAT, "%s holds no model", in_path));
  if (std::rename(tmp.c_str(), out_path) != 0) return give_up(failf(BATHHOST_EFAIL, "cannot rename %s to %s", tmp.c_str(), out_path));
  if (nmodels) *nmodels = done;
  return BATHHOST_OK;
}
