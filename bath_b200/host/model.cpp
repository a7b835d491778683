// model.cpp -- host side of the translated-search path: query model set-up (libbathhost.so).
//
// Restates, without Easel, what bathsearch does once per query before any DP runs
// (src/bathsearch.c:794-801): read the BATH3/f profile, build the null model, configure the
// frameshift profiles for 3 and 5 codon lengths in local mode, and turn them into the un-striped
// odds-ratio tables libbathgpu.so consumes.  Arithmetic follows the reference operation for
// operation (float/double mix included) because these tables define every downstream score.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <limits>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/bathhost.h"
#include "host_internal.h"
#include "model_internal.h"

namespace bathhost {

static const float kNegInf = -std::numeric_limits<float>::infinity();

// ------------------------------------------------------------------------------------------
// alphabets and genetic codes (Easel esl_alphabet / esl_gencode; public Easel definitions)

const char kAminoSyms[] = "ACDEFGHIKLMNPQRSTVWY-BJZOUX*~";
const char kDnaSyms[]   = "ACGT-RYMKSWHBVDN*~";

int amino_code(char c)
{
  c = (char) std::toupper((unsigned char) c);
  if (c == '_' || c == '.') c = '-';
  const char *p = c ? std::strchr(kAminoSyms, c) : nullptr;
  return p ? (int) (p - kAminoSyms) : -1;
}

int dna_code(char c)
{
  c = (char) std::toupper((unsigned char) c);
  if (c == 'U') c = 'T';
  if (c == 'X') c = 'N';
  if (c == 'I') c = 'A';
  if (c == '_' || c == '.') c = '-';
  const char *p = c ? std::strchr(kDnaSyms, c) : nullptr;
  return p ? (int) (p - kDnaSyms) : -1;
}

// NCBI translation tables as edits of the standard code, codon index 16*n1 + 4*n2 + n3 in ACGT order
bool genetic_code(int ct, uint8_t out[64])
{
  std::string code = "KNKNTTTTRSRSIIMIQHQHPPPPRRRRLLLLEDEDAAAAGGGGVVVV*Y*YSSSS*CWCLFLF";
  auto set = [&](const char *codon, char aa) {
    code[16 * dna_code(codon[0]) + 4 * dna_code(codon[1]) + dna_code(codon[2])] = aa;
  };
  switch (ct) {
  case 1: case 11: break;
  case 2:  set("AGA", '*'); set("AGG", '*'); set("ATA", 'M'); set("TGA", 'W'); break;
  case 3:  set("ATA", 'M'); set("CTT", 'T'); set("CTC", 'T'); set("CTA", 'T'); set("CTG", 'T'); set("TGA", 'W'); break;
  case 4:  set("TGA", 'W'); break;
  case 5:  set("AGA", 'S'); set("AGG", 'S'); set("ATA", 'M'); set("TGA", 'W'); break;
  case 6:  set("TAA", 'Q'); set("TAG", 'Q'); break;
  case 9:  set("AAA", 'N'); set("AGA", 'S'); set("AGG", 'S'); set("TGA", 'W'); break;
  case 10: set("TGA", 'C'); break;
  case 12: set("CTG", 'S'); break;
  case 13: set("AGA", 'G'); set("AGG", 'G'); set("ATA", 'M'); set("TGA", 'W'); break;
  case 14: set("AAA", 'N'); set("AGA", 'S'); set("AGG", 'S'); set("TAA", 'Y'); set("TGA", 'W'); break;
  case 16: set("TAG", 'L'); break;
  case 21: set("TGA", 'W'); set("ATA", 'M'); set("AGA", 'S'); set("AGG", 'S'); set("AAA", 'N'); break;
  case 22: set("TCA", '*'); set("TAG", 'L'); break;
  case 23: set("TTA", '*'); break;
  case 24: set("AGA", 'S'); set("AGG", 'K'); set("TGA", 'W'); break;
  case 25: set("TGA", 'G'); break;
  default: return false;
  }
  for (int i = 0; i < 64; ++i) out[i] = (uint8_t) amino_code(code[i]);
  return true;
}

// members of the degenerate amino codes B J Z O U X (esl_alphabet.c)
static bool degenerate_has(int x, int y)
{
  switch (x) {
  case 21: return y == 2 || y == 11;
  case 22: return y == 7 || y == 9;
  case 23: return y == 3 || y == 13;
  case 24: return y == 8;
  case 25: return y == 1;
  case 26: return true;
  default: return false;
  }
}

// esl_abc_FExpectScVec: expected score of each degenerate code under the background
static void expected_degenerate_scores(float *sc, const float *bgf)
{
  for (int x = kK + 1; x <= kKp - 3; ++x) {
    float num = 0.0f, den = 0.0f;
    for (int y = 0; y < kK; ++y)
      if (degenerate_has(x, y)) { num += sc[y] * bgf[y]; den += bgf[y]; }
    sc[x] = num / den;
  }
}

// esl_sse_expf, one lane (Cephes expf): the reference exponentiates the score tables with it
// (src/impl_sse/p7_fs_oprofile.c:252,274,282), so libm's expf would differ in the last bits.
float simd_expf(float x)
{
  static const float P[6] = { 1.9875691500E-4f, 1.3981999507E-3f, 8.3334519073E-3f,
                              4.1665795894E-2f, 1.6666665459E-1f, 5.0000001201E-1f };
  if (x > 88.72283905206835f)    return std::numeric_limits<float>::infinity();
  if (x <= -103.27892990343185f) return 0.0f;
  if (x != x)                    return x;
  float fx = x * 1.44269504088896341f;
  fx = fx + 0.5f;
  float fl = (float) (int) fx;
  if (fl > fx) fl -= 1.0f;
  const int n = (int) fl;
  float hi = fl * 0.693359375f;
  float lo = fl * -2.12194440e-4f;
  x = x - hi;
  x = x - lo;
  const float z = x * x;
  float y = P[0];
  y = y * x; y = y + P[1];
  y = y * x; y = y + P[2];
  y = y * x; y = y + P[3];
  y = y * x; y = y + P[4];
  y = y * x; y = y + P[5];
  y = y * z;
  y = y + x;
  y = y + 1.0f;
  if (n + 127 <= 0) return 0.0f;
  union { int32_t i; float f; } pow2;
  pow2.i = (n + 127) << 23;
  return y * pow2.f;
}

// ------------------------------------------------------------------------------------------
// profile file

static float neglog_to_prob(const std::string &tok)
{
  return (tok[0] == '*') ? 0.0f : expf(-1.0 * atof(tok.c_str()));
}

static std::vector<std::string> split(const std::string &line)
{
  std::vector<std::string> out;
  std::istringstream ss(line);
  std::string t;
  while (ss >> t) out.push_back(t);
  return out;
}

// reads one model record from the stream; BATHHOST_EOF at clean end of file
static int read_record(std::istream &in, CoreModel &h)
{
  std::string line;
  std::vector<std::string> f;
  bool magic = false;
  while (std::getline(in, line)) {
    f = split(line);
    if (f.empty()) continue;
    if (f[0].rfind("BATH3/", 0) == 0 || f[0].rfind("HMMER3/", 0) == 0) { magic = true; break; }
    return BATHHOST_EFORMAT;
  }
  if (!magic) return BATHHOST_EOF;

  h = CoreModel();
  bool body = false, has_rf = false, has_cs = false;
  while (std::getline(in, line)) {
    f = split(line);
    if (f.empty()) continue;
    const std::string &tag = f[0];
    if      (tag == "NAME" && f.size() > 1) h.name = f[1];
    else if (tag == "ACC"  && f.size() > 1) h.acc = f[1];
    else if (tag == "DESC") { const size_t at = line.find_first_not_of(" \t", line.find("DESC") + 4); h.desc = (at == std::string::npos) ? "" : line.substr(at); }
    else if (tag == "RF" && f.size() > 1) has_rf = (f[1] == "yes");
    else if (tag == "CS" && f.size() > 1) has_cs = (f[1] == "yes");
    else if (tag == "LENG" && f.size() > 1) h.M = atoi(f[1].c_str());
    else if (tag == "MAXL" && f.size() > 1) h.max_length = atoi(f[1].c_str());
    else if (tag == "ALPH") { if (f.size() < 2 || f[1] != "amino") return BATHHOST_EFORMAT; }
    else if (tag == "STATS") {
      // "STATS LOCAL FS3 FORWARD tau lambda": token 4 is tau and lambda is never read (src/p7_hmmfile.c:1509-1510)
      if (f.size() < 5 || f[1] != "LOCAL") return BATHHOST_EFORMAT;
      const float a = (float) atof(f[3].c_str()), b = (float) atof(f[4].c_str());
      if      (f[2] == "MSV")     { h.evparam[EV_MMU] = a;  h.evparam[EV_MLAMBDA] = b; }
      else if (f[2] == "VITERBI") { h.evparam[EV_VMU] = a;  h.evparam[EV_VLAMBDA] = b; }
      else if (f[2] == "FORWARD") { h.evparam[EV_FTAU] = a; h.evparam[EV_FLAMBDA] = b; }
      else if (f[2] == "FS3")     { h.evparam[EV_FTAUFS3] = b; h.has_fs3 = true; }
      else if (f[2] == "FS5")     { h.evparam[EV_FTAUFS5] = b; h.has_fs5 = true; }
    }
    else if (tag == "FRAMESHIFT" && f.size() > 2) h.fsprob = (float) atof(f[2].c_str());
    else if (tag == "CODON" && f.size() > 2)      h.ct = atoi(f[2].c_str());
    else if (tag == "HMM") { body = true; break; }
  }
  if (!body || h.M <= 0) return BATHHOST_EFORMAT;
  if (!std::getline(in, line)) return BATHHOST_EFORMAT;        // transition column header

  const int M = h.M;
  h.t.assign((size_t) (M + 1) * 7, 0.0f);
  h.mat.assign((size_t) (M + 1) * kK, 0.0f);
  h.ins.assign((size_t) (M + 1) * kK, 0.0f);
  h.consensus.assign((size_t) M + 2, ' ');
  h.consensus[M + 1] = '\0';
  if (has_rf) h.rf.assign((size_t) M + 2, ' ');
  if (has_cs) h.cs.assign((size_t) M + 2, ' ');

  auto next_fields = [&](size_t need) -> bool {
    if (!std::getline(in, line)) return false;
    f = split(line);
    return f.size() >= need;
  };

  if (!next_fields(1)) return BATHHOST_EFORMAT;
  if (f[0] == "COMPO") {
    if (f.size() < 1 + kK) return BATHHOST_EFORMAT;
    for (int x = 0; x < kK; ++x) h.compo[x] = neglog_to_prob(f[1 + x]);
    h.has_compo = true;
    if (!next_fields(kK)) return BATHHOST_EFORMAT;
  }
  if (f.size() < (size_t) kK) return BATHHOST_EFORMAT;
  for (int x = 0; x < kK; ++x) h.ins[x] = neglog_to_prob(f[x]);
  if (!next_fields(7)) return BATHHOST_EFORMAT;
  for (int x = 0; x < 7; ++x) h.t[x] = neglog_to_prob(f[x]);

  for (int k = 1; k <= M; ++k) {
    if (!next_fields(1 + kK) || atoi(f[0].c_str()) != k) return BATHHOST_EFORMAT;
    for (int x = 0; x < kK; ++x) h.mat[(size_t) k * kK + x] = neglog_to_prob(f[1 + x]);
    h.consensus[k] = (f.size() > (size_t) (2 + kK)) ? f[2 + kK][0] : '-';
    if (has_rf) h.rf[k] = (f.size() > (size_t) (3 + kK)) ? f[3 + kK][0] : '-';       // match line: k, 20 emissions, MAP, CONS, RF, MM, CS
    if (has_cs) h.cs[k] = (f.size() > (size_t) (5 + kK)) ? f[5 + kK][0] : '-';
    if (!next_fields(kK)) return BATHHOST_EFORMAT;
    for (int x = 0; x < kK; ++x) h.ins[(size_t) k * kK + x] = neglog_to_prob(f[x]);
    if (!next_fields(7)) return BATHHOST_EFORMAT;
    for (int x = 0; x < 7; ++x) h.t[(size_t) k * 7 + x] = neglog_to_prob(f[x]);
  }
  if (!next_fields(1) || f[0] != "//") return BATHHOST_EFORMAT;
  return BATHHOST_OK;
}

// p7_Builder_MaxLength (src/p7_builder.c): the sequence length beyond which only a fraction <emit_thresh> of the
// model's emitted sequences fall; bathsearch computes it when the file has no MAXL line (src/bathsearch.c:761-762).
int builder_max_length(const CoreModel &h, double emit_thresh)
{
  const int M = h.M;
  if (M == 1) return 1;
  const int bound = std::max(M, std::min(20 * M, 100000));
  auto T = [&](int k, int t) -> double { return h.t[(size_t) k * 7 + t]; };
  std::vector<double> Mx[2], Ix[2], Dx[2];
  for (int c = 0; c < 2; ++c) { Mx[c].assign(M + 2, 0.0); Ix[c].assign(M + 2, 0.0); Dx[c].assign(M + 2, 0.0); }
  // column 1 (one residue emitted) in slot 0, column 2 in slot 1
  Mx[0][1] = 1.0;
  if (M >= 2) Dx[0][2] = T(1, HT_MD);
  for (int k = 3; k <= M; ++k) Dx[0][k] = T(k - 1, HT_DD) * Dx[0][k - 1];
  Ix[1][1] = T(1, HT_MI) * Mx[0][1];
  if (M >= 2) Mx[1][2] = T(1, HT_MM) * Mx[0][1];
  for (int k = 3; k <= M; ++k) {
    Mx[1][k] = T(k - 1, HT_DM) * Dx[0][k - 1];
    Ix[1][k] = 0;
    Dx[1][k] = T(k - 1, HT_MD) * Mx[1][k - 1] + T(k - 1, HT_DD) * Dx[1][k - 1];
  }
  double p_sum = Mx[0][M] + Mx[1][M] + Dx[0][M] + Dx[1][M];
  int cur = 0;
  for (int col = 3; col <= bound; ++col) {
    const int prev = 1 - cur;
    double surv = 0.0;
    Mx[cur][1] = Dx[cur][1] = 0;
    Ix[cur][1] = T(1, HT_II) * Ix[prev][1];
    surv += Ix[cur][1];
    for (int k = 2; k <= M; ++k) {
      Mx[cur][k] = T(k - 1, HT_MM) * Mx[prev][k - 1] + T(k - 1, HT_DM) * Dx[prev][k - 1] + T(k - 1, HT_IM) * Ix[prev][k - 1];
      Ix[cur][k] = T(k, HT_MI) * Mx[prev][k] + T(k, HT_II) * Ix[prev][k];
      Dx[cur][k] = T(k - 1, HT_MD) * Mx[cur][k - 1] + T(k - 1, HT_DD) * Dx[cur][k - 1];
      surv += Ix[cur][k] + Mx[cur][k] * (1 - T(k, HT_MD)) + Dx[cur][k] * (1 - T(k, HT_DD));
    }
    surv += Mx[cur][M] * T(M, HT_MD) + Dx[cur][M] * T(M, HT_DD) - Ix[cur][M];
    p_sum += Mx[cur][M] + Dx[cur][M];
    surv /= surv + p_sum;
    if (surv < emit_thresh) return col;
    cur = 1 - cur;
  }
  return bound;
}

// ------------------------------------------------------------------------------------------
// null model (src/p7_bg.c:52-82; frequencies src/hmmer.c:163-182)

NullModel::NullModel()
{
  static const float swissprot[kK] = {
    0.0787945, 0.0151600, 0.0535222, 0.0668298, 0.0397062, 0.0695071, 0.0229198, 0.0590092,
    0.0594422, 0.0963728, 0.0237718, 0.0414386, 0.0482904, 0.0395639, 0.0540978, 0.0683364,
    0.0540687, 0.0673417, 0.0114135, 0.0304133 };
  for (int x = 0; x < kK; ++x) f[x] = swissprot[x];
  p1 = 350. / 351.;
  omega = 1. / 256.;
}

// ------------------------------------------------------------------------------------------
// frameshift profile (src/modelconfig.c:220-698)

// match occupancy (src/p7_hmm.c:1349-1364)
static std::vector<float> match_occupancy(const CoreModel &h)
{
  std::vector<float> occ(h.M + 1, 0.0f);
  occ[1] = h.t[HT_MI] + h.t[HT_MM];
  for (int k = 2; k <= h.M; ++k)
    occ[k] = occ[k - 1] * (h.t[(size_t) (k - 1) * 7 + HT_MM] + h.t[(size_t) (k - 1) * 7 + HT_MI]) +
             (1.0 - occ[k - 1]) * h.t[(size_t) (k - 1) * 7 + HT_DM];
  return occ;
}

// index of a quasi-codon's emission row; same row numbering as src/hmmer.h:306-314
struct Rows3 {
  static constexpr int kRows = 338, kDegC = 336, kDegQ1 = 337;
  static int c2(int w, int x)               { return x * 84 + w * 21; }
  static int c3(int v, int w, int x)        { return x * 84 + w * 21 + v * 5 + 1; }
  static int c4(int u, int v, int w, int x) { return x * 84 + w * 21 + v * 5 + u + 2; }
};
struct Rows5 {
  static constexpr int kRows = 1367, kDegC = 1364, kDegQ1 = 1365, kDegQ2 = 1366;
  static int c1(int x)                             { return x * 341; }
  static int c2(int w, int x)                      { return x * 341 + w * 85 + 1; }
  static int c3(int v, int w, int x)               { return x * 341 + w * 85 + v * 21 + 2; }
  static int c4(int u, int v, int w, int x)        { return x * 341 + w * 85 + v * 21 + u * 5 + 3; }
  static int c5(int t, int u, int v, int w, int x) { return x * 341 + w * 85 + v * 21 + u * 5 + t + 4; }
};

// indel patterns (src/hmmer.h:251-268)
enum Pattern : uint8_t { P__X = 0, PX__, PXX_, PX_X, P_XX, PXXX, PXXx, PXxX, PxXX, Pxxx, PXXxX, PXxXX, PxXXX, PXXxxX, PXxxXX, PxxXXX };

void FsProfile::configure(const CoreModel &h, const NullModel &bg, const uint8_t gcode[64], int codon_lengths_)
{
  codon_lengths = codon_lengths_;
  M = h.M;
  maxcodons = (codon_lengths == 5) ? Rows5::kRows : Rows3::kRows;
  const int nrows = maxcodons + kKp;
  const size_t ld = (size_t) M + 1;
  rsc.assign((size_t) nrows * ld, kNegInf);
  tsc.assign((size_t) M * 8, kNegInf);
  codons.assign(ld * (size_t) (maxcodons + 1), 0);
  indel_pos.assign(ld * (size_t) (maxcodons + 1), 0);

  // local entry: uniform over fragments, weighted by occupancy (src/modelconfig.c:283-297)
  {
    std::vector<float> occ = match_occupancy(h);
    float Z = 0.;
    for (int k = 1; k <= M; ++k) Z += occ[k] * (float) (M - k + 1);
    for (int k = 1; k <= M; ++k) tsc[(size_t) (k - 1) * 8 + PT_BM] = log(occ[k] / Z);
  }
  // multihit local: E->C and E->J both 1/2 (:309-313)
  xsc[PX_E][PX_MOVE] = -0.69314718055994529;
  xsc[PX_E][PX_LOOP] = -0.69314718055994529;
  nj = 1.0f;
  for (int k = 1; k < M; ++k) {
    float *tp = &tsc[(size_t) k * 8];
    const float *ht = &h.t[(size_t) k * 7];
    tp[PT_MM] = log(ht[HT_MM]); tp[PT_MI] = log(ht[HT_MI]); tp[PT_MD] = log(ht[HT_MD]);
    tp[PT_IM] = log(ht[HT_IM]); tp[PT_II] = log(ht[HT_II]);
    tp[PT_DM] = log(ht[HT_DM]); tp[PT_DD] = log(ht[HT_DD]);
  }

  // amino-acid log-odds rows sit after the codon rows (:343-352)
  auto R = [&](int row, int k) -> float & { return rsc[(size_t) row * ld + k]; };
  auto amino = [&](int k, int a) -> float & { return rsc[(size_t) (maxcodons + a) * ld + k]; };
  for (int k = 1; k <= M; ++k) {
    float sc[kKp];
    sc[kK] = sc[kKp - 2] = sc[kKp - 1] = kNegInf;
    for (int x = 0; x < kK; ++x) sc[x] = log((double) h.mat[(size_t) k * kK + x] / bg.f[x]);
    expected_degenerate_scores(sc, bg.f);
    for (int x = 0; x < kKp; ++x) amino(k, x) = sc[x];
  }

  const float fs = h.fsprob;
  const float one_indel = log(fs), stop_cost = log(fs);
  const float two_indel = (codon_lengths == 5) ? (float) log(fs / 2.) : 0.0f;
  const float no_indel  = (codon_lengths == 5) ? (float) log(1. - fs * 4.) : (float) log(1. - fs * 3.);
  const int   STOP = kKp - 2, ANY = kKp - 3;

  for (int k = 1; k <= M; ++k) {
    // a quasi-codon row keeps the best-scoring amino acid it could be a damaged codon of
    auto offer = [&](int row, int a, Pattern pat) {
      if (amino(k, a) > R(row, k)) {
        R(row, k) = amino(k, a);
        codons[(size_t) k * maxcodons + row] = (uint8_t) a;
        indel_pos[(size_t) k * maxcodons + row] = pat;
      }
    };
    auto assign = [&](int row, int a, Pattern pat) {
      R(row, k) = amino(k, a);
      codons[(size_t) k * maxcodons + row] = (uint8_t) a;
      indel_pos[(size_t) k * maxcodons + row] = pat;
    };
    auto aa = [&](int n1, int n2, int n3) { return (int) gcode[16 * n1 + 4 * n2 + n3]; };

    for (int x = 0; x < 4; ++x)
      for (int w = 0; w < 4; ++w)
        for (int v = 0; v < 4; ++v) {
          const int a = aa(v, w, x);
          int row3;
          if (codon_lengths == 5) {
            offer(Rows5::c1(x), a, P__X);
            offer(Rows5::c1(v), a, PX__);
            offer(Rows5::c2(w, x), a, P_XX);
            offer(Rows5::c2(v, x), a, PX_X);
            offer(Rows5::c2(v, w), a, PXX_);
            row3 = Rows5::c3(v, w, x);
          } else {
            offer(Rows3::c2(w, x), a, P_XX);
            offer(Rows3::c2(v, x), a, PX_X);
            offer(Rows3::c2(v, w), a, PXX_);
            row3 = Rows3::c3(v, w, x);
          }
          if (a == STOP) {         // a stop codon scores as its best one-substitution neighbour (:395-425)
            for (int s = 0; s < 4; ++s) {
              offer(row3, aa(s, w, x), PxXX);
              offer(row3, aa(v, s, x), PXxX);
              offer(row3, aa(v, w, s), PXXx);
            }
          } else assign(row3, a, PXXX);
          for (int u = 0; u < 4; ++u) {
            const int row4 = (codon_lengths == 5) ? Rows5::c4(u, v, w, x) : Rows3::c4(u, v, w, x);
            offer(row4, aa(u, v, x), PXXxX);
            offer(row4, aa(u, w, x), PXxXX);
            offer(row4, aa(v, w, x), PxXXX);
            if (codon_lengths == 5)
              for (int t = 0; t < 4; ++t) {
                const int row5 = Rows5::c5(t, u, v, w, x);
                offer(row5, aa(t, u, x), PXXxxX);
                offer(row5, aa(t, w, x), PXxxXX);
                offer(row5, aa(v, w, x), PxxXXX);
              }
          }
        }

    // indel / stop costs on top (:497-519, :613-648)
    for (int x = 0; x < 4; ++x) {
      if (codon_lengths == 5) R(Rows5::c1(x), k) += two_indel;
      for (int w = 0; w < 4; ++w) {
        R(codon_lengths == 5 ? Rows5::c2(w, x) : Rows3::c2(w, x), k) += one_indel;
        for (int v = 0; v < 4; ++v) {
          const int a = aa(v, w, x);
          R(codon_lengths == 5 ? Rows5::c3(v, w, x) : Rows3::c3(v, w, x), k) += (a == STOP) ? stop_cost : no_indel;
          for (int u = 0; u < 4; ++u) {
            R(codon_lengths == 5 ? Rows5::c4(u, v, w, x) : Rows3::c4(u, v, w, x), k) += one_indel;
            if (codon_lengths == 5)
              for (int t = 0; t < 4; ++t) R(Rows5::c5(t, u, v, w, x), k) += two_indel;
          }
        }
      }
    }
    // rows for quasi-codons holding a degenerate nucleotide: residue X (:521-533, :650-658)
    auto degenerate = [&](int row, float cost) {
      R(row, k) = amino(k, ANY) + cost;
      codons[(size_t) k * maxcodons + row] = (uint8_t) ANY;
      indel_pos[(size_t) k * maxcodons + row] = Pxxx;
    };
    if (codon_lengths == 5) {
      degenerate(Rows5::kDegC, no_indel); degenerate(Rows5::kDegQ1, one_indel); degenerate(Rows5::kDegQ2, two_indel);
    } else {
      degenerate(Rows3::kDegC, no_indel); degenerate(Rows3::kDegQ1, one_indel);
    }
  }
}

// odds-ratio tables, un-striped (src/impl_sse/p7_fs_oprofile.c:222-296)
void FsOddsProfile::convert(const FsProfile &gm)
{
  M = gm.M;
  codon_lengths = gm.codon_lengths;
  nrows = gm.maxcodons + kKp;
  const size_t ld = (size_t) M + 1;
  rfv.assign((size_t) nrows * ld, 0.0f);
  tfv.assign(8 * ld, 0.0f);
  for (int c = 0; c < nrows; ++c)
    for (int k = 1; k <= M; ++k)
      rfv[(size_t) c * ld + k] = simd_expf(gm.rsc[(size_t) c * ld + k]);
  // order BM,MM,IM,DM,MD,MI,II,DD; source-node indexed; node M and (for the unrotated ones) node 0 carry 0
  static const int from[8] = { PT_BM, PT_MM, PT_IM, PT_DM, PT_MD, PT_MI, PT_II, PT_DD };
  for (int z = 0; z < 8; ++z)
    for (int k = (z < 4 ? 0 : 1); k < M; ++k)
      tfv[(size_t) z * ld + k] = simd_expf(gm.tsc[(size_t) k * 8 + from[z]]);
  xfE_move = expf(gm.xsc[PX_E][PX_MOVE]);
  xfE_loop = expf(gm.xsc[PX_E][PX_LOOP]);
}

// ------------------------------------------------------------------------------------------
// protein profile for the ORF filters

uint8_t ProteinProfile::unbiased_byteify(float sc) const
{
  sc = -1.0f * roundf(scale_b * sc);
  return (sc > 255.) ? 255 : (uint8_t) sc;
}
uint8_t ProteinProfile::biased_byteify(float sc) const
{
  sc = -1.0f * roundf(scale_b * sc);
  uint8_t b = (sc > 255 - bias_b) ? 255 : (uint8_t) sc + bias_b;
  return b;
}
int16_t ProteinProfile::wordify(float sc) const
{
  sc = roundf(scale_w * sc);
  if (sc >= 32767.0) return 32767;
  if (sc <= -32768.0) return -32768;
  return (int16_t) sc;
}
uint8_t ProteinProfile::tjb_for_length(int L) const { return unbiased_byteify(logf(3.0f / (float) (L + 3))); }
int16_t ProteinProfile::xw_move_for_length(int L) const
{
  const float pmove = (2.0f + nj) / ((float) L + 2.0f + nj);
  return wordify(logf(pmove));
}

// The protein profile's match scores and transitions are the frameshift profile's amino rows and
// transitions (same arithmetic, src/modelconfig.c:140-156 vs :343-352), so they are taken from there.
void ProteinProfile::configure(const CoreModel &h, const NullModel &bg, const FsProfile &gm_fs, const FsOddsProfile &om_fs)
{
  (void) bg;
  M = h.M; max_length = h.max_length; nj = 1.0f;
  const size_t ld = (size_t) M + 1;
  msc.assign((size_t) kKp * ld, kNegInf);
  for (int x = 0; x < kKp; ++x)
    for (int k = 1; k <= M; ++k) msc[(size_t) x * ld + k] = gm_fs.rsc[(size_t) (gm_fs.maxcodons + x) * ld + k];
  xsc_E_move = gm_fs.xsc[PX_E][PX_MOVE];
  xsc_E_loop = gm_fs.xsc[PX_E][PX_LOOP];

  // bytes (mf_conversion, :773-812): the bias is the highest score of a canonical residue; insert scores are 0
  float max = 0.0;
  for (int x = 0; x < kK; ++x)
    for (int k = 1; k <= M; ++k) if (msc[(size_t) x * ld + k] > max) max = msc[(size_t) x * ld + k];
  scale_b = 3.0 / 0.69314718055994529;
  base_b  = 190;
  bias_b  = unbiased_byteify(-1.0 * max);
  rbv.assign((size_t) kKp * ld, 255);
  for (int x = 0; x < kKp; ++x)
    for (int k = 1; k <= M; ++k) rbv[(size_t) x * ld + k] = biased_byteify(msc[(size_t) x * ld + k]);
  tbm_b = unbiased_byteify(logf(2.0f / ((float) M * (float) (M + 1))));
  tec_b = unbiased_byteify(logf(0.5f));

  // words (vf_conversion, :826-921)
  scale_w = 500.0 / 0.69314718055994529;
  base_w  = 12000;
  rwv.assign((size_t) kKp * ld, -32768);
  for (int x = 0; x < kKp; ++x)
    for (int k = 1; k <= M; ++k) rwv[(size_t) x * ld + k] = wordify(msc[(size_t) x * ld + k]);
  static const int from[8] = { PT_BM, PT_MM, PT_IM, PT_DM, PT_MD, PT_MI, PT_II, PT_DD };
  twv.assign(8 * ld, -32768);
  for (int t = 0; t < 8; ++t)
    for (int k = (t < 4 ? 0 : 1); k < M; ++k) {
      int16_t v = wordify(gm_fs.tsc[(size_t) k * 8 + from[t]]);
      const int16_t cap = (t == 6) ? -1 : 0;            // II may not cost 0 (:872-877)
      if (t != 7 && v > cap) v = cap;
      twv[(size_t) t * ld + k] = v;
    }
  xw_E_loop = wordify(xsc_E_loop);
  xw_E_move = wordify(xsc_E_move);
  ddbound_w = -32768;
  for (int k = 2; k < M - 1; ++k) {
    int dd = (int) wordify(gm_fs.tsc[(size_t) k * 8 + PT_DD]);
    dd    += (int) wordify(gm_fs.tsc[(size_t) (k + 1) * 8 + PT_DM]);
    dd    -= (int) wordify(gm_fs.tsc[(size_t) (k + 1) * 8 + PT_BM]);
    if (dd > ddbound_w) ddbound_w = dd;
  }

  // prefix / suffix lengths (p7_scoredata.c:358-375) from the odds-ratio MI and II transitions
  prefix_lengths.assign(ld, 0.0f);
  suffix_lengths.assign(ld, 0.0f);
  const float *t_mis = &om_fs.tfv[5 * ld], *t_iis = &om_fs.tfv[6 * ld];
  float sum = 0;
  for (int k = 1; k < M; ++k) {
    if (t_mis[k] == 0) prefix_lengths[k] = 1;
    else               prefix_lengths[k] = 1 + (int) (log(1e-7 / t_mis[k]) / log(t_iis[k]));
    sum += prefix_lengths[k];
  }
  prefix_lengths[0] = prefix_lengths[M] = 0;
  for (int k = 1; k < M; ++k) prefix_lengths[k] /= sum;
  suffix_lengths[M] = prefix_lengths[M - 1];
  for (int k = M - 1; k >= 1; --k) suffix_lengths[k] = suffix_lengths[k + 1] + prefix_lengths[k - 1];
  for (int k = 2; k < M; ++k) prefix_lengths[k] += prefix_lengths[k - 1];
}

}  // namespace bathhost

// ------------------------------------------------------------------------------------------
// C ABI

using namespace bathhost;


static int open_nth(const char *path, int index, CoreModel &h)
{
  std::ifstream in(path);
  if (!in) return BATHHOST_EFAIL;
  int st = BATHHOST_EOF;
  for (int n = 0; n <= index; ++n)
    if ((st = read_record(in, h)) != BATHHOST_OK) break;
  return st;
}

// everything after reading the core model: the query set-up of bathsearch (src/bathsearch.c:761-762, :794-801)
static int setup_model(bathhost_model *m, int ct)
{
  m->maxl_in_file = m->hmm.max_length;
  if (m->hmm.max_length == -1) m->hmm.max_length = builder_max_length(m->hmm, 1e-7);      // src/bathsearch.c:761-762
  m->ct = (ct > 0) ? ct : (m->hmm.ct > 0 ? m->hmm.ct : 1);
  uint8_t gcode[64];
  if (!genetic_code(m->ct, gcode) || !(m->hmm.fsprob > 0.0f)) return BATHHOST_EINVAL;
  m->gm3.configure(m->hmm, m->bg, gcode, 3);
  m->gm5.configure(m->hmm, m->bg, gcode, 5);
  m->om3.convert(m->gm3);
  m->om5.convert(m->gm5);
  m->prot.configure(m->hmm, m->bg, m->gm5, m->om5);
  return BATHHOST_OK;
}

extern "C" int bathhost_model_read(const char *path, int index, int ct, bathhost_model **ret_model)
{
  if (!path || index < 0 || !ret_model) return BATHHOST_EINVAL;
  *ret_model = nullptr;
  bathhost_model *m = new (std::nothrow) bathhost_model();
  if (!m) return BATHHOST_EMEM;
  int st = open_nth(path, index, m->hmm);
  if (st == BATHHOST_OK) st = setup_model(m, ct);
  if (st != BATHHOST_OK) { delete m; return st; }
  *ret_model = m;
  return BATHHOST_OK;
}

int bathhost::model_from_record(const std::string &text, int ct, float fsprob, bathhost_model **ret)
{
  *ret = nullptr;
  bathhost_model *m = new (std::nothrow) bathhost_model();
  if (!m) return BATHHOST_EMEM;
  std::istringstream in(text);
  int st = read_record(in, m->hmm);
  if (st == BATHHOST_EOF) st = BATHHOST_EFORMAT;
  if (st == BATHHOST_OK) {
    m->hmm.ct = ct;
    m->hmm.fsprob = fsprob;
    st = setup_model(m, ct);
  }
  if (st != BATHHOST_OK) { delete m; return st; }
  *ret = m;
  return BATHHOST_OK;
}

extern "C" int bathhost_model_count(const char *path)
{
  std::ifstream in(path);
  if (!in) return -1;
  CoreModel h;
  int n = 0;
  while (read_record(in, h) == BATHHOST_OK) ++n;
  return n;
}

extern "C" void bathhost_model_destroy(bathhost_model *m) { delete m; }

extern "C" int bathhost_model_get_info(const bathhost_model *m, bathhost_model_info *info)
{
  if (!m || !info) return BATHHOST_EINVAL;
  std::memset(info, 0, sizeof *info);
  info->M = m->hmm.M;
  info->max_length = m->hmm.max_length;
  info->codon_table = m->hmm.ct;
  info->fsprob = m->hmm.fsprob;
  for (int z = 0; z < 8; ++z) info->evparam[z] = m->hmm.evparam[z];
  info->has_fs3_stats = m->hmm.has_fs3;
  info->has_fs5_stats = m->hmm.has_fs5;
  std::strncpy(info->name, m->hmm.name.c_str(), sizeof info->name - 1);
  std::strncpy(info->acc, m->hmm.acc.c_str(), sizeof info->acc - 1);
  return BATHHOST_OK;
}

static const FsOddsProfile *odds(const bathhost_model *m, int which) { return !m ? nullptr : (which == 3 ? &m->om3 : which == 5 ? &m->om5 : nullptr); }
static const FsProfile     *prof(const bathhost_model *m, int which) { return !m ? nullptr : (which == 3 ? &m->gm3 : which == 5 ? &m->gm5 : nullptr); }

extern "C" int bathhost_model_nrows(const bathhost_model *m, int which) { auto *o = odds(m, which); return o ? o->nrows : 0; }
extern "C" const float *bathhost_model_rfv(const bathhost_model *m, int which) { auto *o = odds(m, which); return o ? o->rfv.data() : nullptr; }
extern "C" const float *bathhost_model_tfv(const bathhost_model *m, int which) { auto *o = odds(m, which); return o ? o->tfv.data() : nullptr; }
extern "C" const uint8_t *bathhost_model_codons(const bathhost_model *m, int which) { auto *p = prof(m, which); return p ? p->codons.data() : nullptr; }
extern "C" const uint8_t *bathhost_model_indel_pos(const bathhost_model *m, int which) { auto *p = prof(m, which); return p ? p->indel_pos.data() : nullptr; }
extern "C" const float *bathhost_model_mat(const bathhost_model *m) { return m ? m->hmm.mat.data() : nullptr; }
extern "C" const char *bathhost_model_consensus(const bathhost_model *m) { return m ? m->hmm.consensus.data() : nullptr; }

extern "C" void bathhost_length_model(int L_amino, float nj, float *pmove, float *ploop)
{
  const float pm = (2.0f + nj) / ((float) L_amino + 2.0f + nj);
  if (pmove) *pmove = pm;
  if (ploop) *ploop = 1.0f - pm;
}

extern "C" int bathhost_model_filter_params(const bathhost_model *m, bathhost_filter_params *p)
{
  if (!m || !p) return BATHHOST_EINVAL;
  const ProteinProfile &q = m->prot;
  p->M = q.M; p->tbm_b = q.tbm_b; p->tec_b = q.tec_b; p->base_b = q.base_b; p->bias_b = q.bias_b; p->scale_b = q.scale_b;
  p->base_w = q.base_w; p->ddbound_w = q.ddbound_w; p->xw_E_move = q.xw_E_move; p->xw_E_loop = q.xw_E_loop; p->scale_w = q.scale_w;
  return BATHHOST_OK;
}
extern "C" const uint8_t *bathhost_model_rbv(const bathhost_model *m) { return m ? m->prot.rbv.data() : nullptr; }
extern "C" const int16_t *bathhost_model_rwv(const bathhost_model *m) { return m ? m->prot.rwv.data() : nullptr; }
extern "C" const int16_t *bathhost_model_twv(const bathhost_model *m) { return m ? m->prot.twv.data() : nullptr; }
extern "C" void bathhost_orf_length_params(const bathhost_model *m, int L, uint8_t *tjb_b, int16_t *xw_move)
{
  if (!m) return;
  if (tjb_b)   *tjb_b   = m->prot.tjb_for_length(L);
  if (xw_move) *xw_move = m->prot.xw_move_for_length(L);
}

extern "C" int bathhost_model_computed_max_length(const bathhost_model *m)
{
  return m ? bathhost::builder_max_length(m->hmm, 1e-7) : -1;
}
