// model_internal.h -- the query model object shared by the host-side sources.
#pragma once
#include "host_internal.h"

struct bathhost_model {
  bathhost::CoreModel      hmm;
  bathhost::NullModel      bg;
  int                      ct = 1;
  int                      maxl_in_file = -1;
  bathhost::FsProfile      gm3, gm5;
  bathhost::FsOddsProfile  om3, om5;
  bathhost::ProteinProfile prot;
};

namespace bathhost {
// model.cpp: one model from the text of its record, set up as bathhost_model_read does, with the codon table and frameshift
// probability given (a HMMER3/f record carries neither).  BATHHOST_EFORMAT for a record that cannot be read, EINVAL for ct / fsprob.
int model_from_record(const std::string &text, int ct, float fsprob, bathhost_model **ret);

// calibrate.cpp: the pieces of bathconvert's frameshift simulations (src/evalues.c:607-680, :703-776) bathhost_convert batches
constexpr int kFsSimL = 100, kFsSimN = 200;        // EfL amino acids (300 nt) per sequence, EfN sequences per simulation
uint32_t calibration_generator(uint32_t seed);     // the state of a fresh generator (seed 0 = 42)
// n sequences of 3 kFsSimL nucleotides each, drawn as one simulation draws them, written one after the other from dna;
// *state is the generator before and after.  False for a model whose codon table is unknown.
bool draw_fs_sequences(const bathhost_model *m, uint32_t *state, int n, uint8_t *dna);
// the tau one simulation's kFsSimN scores (nats, none overflowed) give: the fit of p7_fs_Tau_*codons
double fs_tau(const float *sc, int n, double lambda);
}  // namespace bathhost
