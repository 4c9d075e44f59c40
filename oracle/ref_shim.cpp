// oracle/ref_shim.cpp -- TEST INFRASTRUCTURE, not product code.
//
// A thin C-ABI driver around the UNMODIFIED reference (soedinglab/hh-suite) compiled by
// oracle/ref_build.mk into oracle/_ref/libhhref.a.  It lets tests / bench.py's cpu_baseline
//   * run the reference's own HHM reader + PrepareQueryHMM / PrepareTemplateHMM
//     (src/hhfunc.cpp:121-202) and export the prepared fp32 DP inputs,
//   * feed arbitrary prepared profiles through the reference's own AVX2 kernel
//     Viterbi::Align (src/hhviterbi.cpp:163, src/hhviterbialgorithm.cpp:29-497),
//     Viterbi::Backtrace (src/hhviterbi.cpp:83) and ScoreForBacktrace (:195),
//   * call Prefilter::stripe_query_profile / ungapped_sse_score / swStripedByte
//     (src/hhprefilter.cpp:356,214,70),
//   * time the reference kernel on all host cores the way ViterbiRunner::alignment does
//     (src/hhviterbirunner.cpp:117-128: length-sorted batches of VECSIZE_FLOAT, OpenMP dynamic,1).
// Nothing here is linked into the product library (hh-suite_b200/csrc).  Only tests/,
// __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference may load the .so.
//
// This file contains no reference code: it only includes the reference headers at build time
// (-I/root/reference/src) and calls their API.  Private members are reached with the usual
// test-harness trick (#define private public) after the std headers are included.

#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <vector>
#include <omp.h>
#include <sys/mman.h>

#define private public
#define protected public
#include "hhdecl.h"
#include "hhhmm.h"
#include "hhhmmsimd.h"
#include "hhviterbi.h"
#include "hhviterbimatrix.h"
#include "hhmatrices.h"
#include "hhfunc.h"
#include "hhprefilter.h"
#include "hhhit.h"
#include "hhhitlist.h"
#include "hhviterbirunner.h"
#include "hhposteriordecoder.h"
#include "hhposteriordecoderrunner.h"
#include "hhposteriormatrix.h"
#include "hhalignment.h"
extern "C" {
#include "ffutil.h"
}
extern "C" {
#include "ffindex.h"
}
#include "cs219.lib.h"
#include "context_data.crf.h"
#undef private
#undef protected

namespace {

struct RefCtx {
  Parameters* par = nullptr;
  float pb[21] __attribute__((aligned(32)));
  float P[20][20] __attribute__((aligned(32)));
  float R[20][20] __attribute__((aligned(32)));
  float S[20][20] __attribute__((aligned(32)));
  float Sim[20][20] __attribute__((aligned(32)));
  float S73[NDSSP][NSSPRED][MAXCF];
  float S37[NSSPRED][MAXCF][NDSSP];
  float S33[NSSPRED][MAXCF][NSSPRED][MAXCF];
  cs::ContextLibrary<cs::AA>* context_lib = nullptr;
  cs::Crf<cs::AA>* crf = nullptr;
  cs::Pseudocounts<cs::AA>* pc_hhm_context_engine = nullptr;
  cs::Admix* pc_hhm_context_mode = nullptr;
  cs::Pseudocounts<cs::AA>* pc_prefilter_context_engine = nullptr;
  cs::Admix* pc_prefilter_context_mode = nullptr;
  int maxres = 0;
  HMM* q = nullptr;
  HMMSimd* q_simd = nullptr;
  // last batch state (for backtrace / scoring)
  std::vector<HMM*> t_hmm;
  HMMSimd* t_simd = nullptr;
  ViterbiMatrix* matrix = nullptr;
  Viterbi* viterbi = nullptr;
  Viterbi::ViterbiResult last;
  int last_ss_mode = 0;
  Prefilter* prefilter = nullptr;  // raw storage, ctor never run (needs an ffindex DB)
};

RefCtx* g = nullptr;
const char* kArgv[] = {"hhalign"};

// tr index map: caller uses the reference's HMM enum order M2M,M2I,M2D,I2M,I2I,D2M,D2D (src/hhdecl.h:68)
void fill_hmm(HMM* h, int L, const float* p, const float* tr, const unsigned char* ss_pred,
              const unsigned char* ss_conf, const unsigned char* ss_dssp) {
  h->L = L;
  for (int i = 0; i <= L + 1 && i < h->maxres; ++i) {
    for (int a = 0; a < 20; ++a) h->p[i][a] = p[(size_t)i * 20 + a];
  }
  for (int i = 0; i <= L; ++i)
    for (int k = 0; k < 7; ++k) h->tr[i][k] = tr[(size_t)i * 7 + k];
  h->nss_pred = h->nss_conf = h->nss_dssp = -1;
  for (int i = 0; i <= L + 1 && i < h->maxres; ++i) {
    h->ss_pred[i] = ss_pred ? (char)ss_pred[i] : 0;
    h->ss_conf[i] = ss_conf ? (char)ss_conf[i] : 0;
    h->ss_dssp[i] = ss_dssp ? (char)ss_dssp[i] : 0;
  }
  if (ss_pred) { h->nss_pred = 0; h->nss_conf = 0; }
  if (ss_dssp) h->nss_dssp = 0;
  h->mu = 0; h->lamda = 0;
}

void export_hmm(HMM* h, float* p, float* tr, float* pav, unsigned char* ss_pred,
                unsigned char* ss_conf, unsigned char* ss_dssp, float* neff) {
  const int L = h->L;
  if (p) for (int i = 0; i <= L + 1; ++i) for (int a = 0; a < 20; ++a) p[(size_t)i * 20 + a] = h->p[i][a];
  if (tr) for (int i = 0; i <= L; ++i) for (int k = 0; k < 7; ++k) tr[(size_t)i * 7 + k] = h->tr[i][k];
  if (pav) for (int a = 0; a < 20; ++a) pav[a] = h->pav[a];
  for (int i = 0; i <= L + 1; ++i) {
    if (ss_pred) ss_pred[i] = (h->nss_pred >= 0) ? (unsigned char)h->ss_pred[i] : 0;
    if (ss_conf) ss_conf[i] = (h->nss_conf >= 0) ? (unsigned char)h->ss_conf[i] : 0;
    if (ss_dssp) ss_dssp[i] = (h->nss_dssp >= 0) ? (unsigned char)h->ss_dssp[i] : 0;
  }
  if (neff) *neff = h->Neff_HMM;
}

}  // namespace

extern "C" {

// flags: bit0 = nocontxt (substitution-matrix pseudocounts for the query instead of the CRF)
int hhref_init(int nocontxt, int maxres) {
  if (g) return 0;
  Log::reporting_level() = WARNING;
  g = new RefCtx();
  g->par = new Parameters(1, kArgv);
  g->par->nocontxt = nocontxt ? 1 : 0;
  g->par->maxres = maxres;
  g->par->threads = 1;
  g->maxres = maxres;
  SetSubstitutionMatrix(g->par->matrix, g->pb, g->P, g->R, g->S, g->Sim);
  SetSecStrucSubstitutionMatrix(g->par->ssa, g->S73, g->S37, g->S33);
  if (!nocontxt)
    InitializePseudocountsEngine(*g->par, g->context_lib, g->crf, g->pc_hhm_context_engine,
                                 g->pc_hhm_context_mode, g->pc_prefilter_context_engine,
                                 g->pc_prefilter_context_mode);
  g->q = new HMM(MAXSEQDIS, maxres);
  g->q_simd = new HMMSimd(maxres);
  g->t_simd = new HMMSimd(maxres);
  g->matrix = new ViterbiMatrix();
  for (int i = 0; i < VECSIZE_FLOAT; ++i) g->t_hmm.push_back(new HMM(64, maxres));
  return 0;
}

int hhref_vecsize() { return VECSIZE_FLOAT; }

// Parameter getters so tests use the reference's own defaults (src/hhdecl.cpp:82-127)
float hhref_par_shift() { return g->par->shift; }
float hhref_par_ssw() { return g->par->ssw; }
float hhref_par_corr() { return g->par->corr; }
int hhref_par_ssm() { return g->par->ssm; }

// S33 table (for the SS variant): out[NSSPRED*MAXCF*NSSPRED*MAXCF]
void hhref_get_S33(float* out) { memcpy(out, g->S33, sizeof(g->S33)); }
void hhref_get_pb(float* out) { memcpy(out, g->pb, 20 * sizeof(float)); }
// R[a][b] = P(a|b), the pseudocount matrix of SetSubstitutionMatrix (src/hhfunc.cpp), out[400]
void hhref_get_R(float* out) { memcpy(out, g->R, 400 * sizeof(float)); }
// S[a][b]: substitution matrix in bits (Alignment::Filter2 qsc test)
void hhref_get_S(float* out) { memcpy(out, g->S, 400 * sizeof(float)); }
// the transition / aa pseudocount parameters PrepareTemplateHMM passes on (src/hhfunc.cpp:170-178)
void hhref_get_prep_params(float* out11) {
  Parameters& par = *g->par;
  float v[11] = {par.gapb, par.gapd, par.gape, par.gapf, par.gapg, par.gaph, par.gapi,
                 (float)par.pc_hhm_nocontext_mode, par.pc_hhm_nocontext_a, par.pc_hhm_nocontext_b,
                 par.pc_hhm_nocontext_c};
  memcpy(out11, v, sizeof(v));
}

// override par.pc_hhm_nocontext_mode / _a / _b / _c (the -pcm/-pca/-pcb/-pcc options) for the following preparations
extern "C" void hhref_set_pc(int mode, float a, float b, float c) {
  g->par->pc_hhm_nocontext_mode = mode; g->par->pc_hhm_nocontext_a = a; g->par->pc_hhm_nocontext_b = b;
  g->par->pc_hhm_nocontext_c = c;
}

// Read query HHM, add pseudocounts exactly like HHalign::run (src/hhalign.cpp:615-626), map to SIMD.
int hhref_load_query_hhm(const char* path) {
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  char pathbuf[NAMELEN];
  Pathname(pathbuf, const_cast<char*>(path));
  g->q->Read(f, g->par->maxcol, g->par->nseqdis, g->pb, pathbuf);
  fclose(f);
  char input_format = 0;
  PrepareQueryHMM(*g->par, input_format, g->q, g->pc_hhm_context_engine, g->pc_hhm_context_mode,
                  g->pb, g->R);
  g->q_simd->MapOneHMM(g->q);
  return g->q->L;
}

int hhref_get_query(float* p, float* tr, float* pav, unsigned char* ss_pred, unsigned char* ss_conf,
                    unsigned char* ss_dssp, float* neff) {
  export_hmm(g->q, p, tr, pav, ss_pred, ss_conf, ss_dssp, neff);
  return g->q->L;
}

// Install a synthetic, already prepared query.
int hhref_set_query(int L, const float* p, const float* tr, const float* pav,
                    const unsigned char* ss_pred, const unsigned char* ss_conf) {
  if (L + 2 > g->maxres) return -1;
  fill_hmm(g->q, L, p, tr, ss_pred, ss_conf, nullptr);
  if (pav) for (int a = 0; a < 20; ++a) g->q->pav[a] = pav[a];
  g->q_simd->MapOneHMM(g->q);
  return L;
}

// Read a template HHM and run PrepareTemplateHMM against the current query
// (src/hhviterbirunner.cpp:144-147); export the DP inputs.
int hhref_prepare_template_hhm(const char* path, float* p, float* tr, float* pav,
                               unsigned char* ss_pred, unsigned char* ss_conf,
                               unsigned char* ss_dssp, float* neff, int maxL) {
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  HMM* t = new HMM(MAXSEQDIS, g->maxres);
  char pathbuf[NAMELEN];
  Pathname(pathbuf, const_cast<char*>(path));
  t->Read(f, g->par->maxcol, g->par->nseqdis, g->pb, pathbuf);
  fclose(f);
  PrepareTemplateHMM(*g->par, g->q, t, 0, false, g->pb, g->R);
  int L = t->L;
  if (L > maxL) { delete t; return -2; }
  export_hmm(t, p, tr, pav, ss_pred, ss_conf, ss_dssp, neff);
  delete t;
  return L;
}

// Same as hhref_prepare_template_hhm but additionally exports the profile BEFORE the query-dependent
// null-model division (IncludeNullModelInHMM, src/hhhmm.cpp:2059-2081): the steps of PrepareTemplateHMM
// (src/hhfunc.cpp:165-202) are called one by one.  columnscore selects the null model (par.columnscore).
int hhref_prepare_template_hhm_raw(const char* path, int columnscore, float* p_raw, float* p_prep,
                                   float* tr, float* pav, int maxL) {
  FILE* f = fopen(path, "r");
  if (!f) return -1;
  HMM* t = new HMM(MAXSEQDIS, g->maxres);
  char pathbuf[NAMELEN];
  Pathname(pathbuf, const_cast<char*>(path));
  t->Read(f, g->par->maxcol, g->par->nseqdis, g->pb, pathbuf);
  fclose(f);
  Parameters& par = *g->par;
  t->AddTransitionPseudocounts(par.gapd, par.gape, par.gapf, par.gapg, par.gaph, par.gapi, par.gapb, par.gapb);
  t->PreparePseudocounts(g->R);
  t->AddAminoAcidPseudocounts(par.pc_hhm_nocontext_mode, par.pc_hhm_nocontext_a, par.pc_hhm_nocontext_b,
                              par.pc_hhm_nocontext_c);
  t->CalculateAminoAcidBackground(g->pb);
  int L = t->L;
  if (L > maxL) { delete t; return -2; }
  export_hmm(t, p_raw, tr, pav, nullptr, nullptr, nullptr, nullptr);
  t->IncludeNullModelInHMM(g->q, t, columnscore, par.half_window_size_local_aa_bg_freqs, g->pb);
  export_hmm(t, p_prep, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
  delete t;
  return L;
}

// ---------------------------------------------------------------------------------------------------
// MAC realignment of ONE hit (PosteriorDecoder::realign, src/hhposteriordecoder.cpp:85-118) around its
// Viterbi alignment.  Query = the loaded query (a copy is put into linear transition space exactly like
// PosteriorDecoderRunner::executeComputation, src/hhposteriordecoderrunner.cpp:48-52).
//   t_p/t_tr: prepared template as handed to the Viterbi kernel (null model included, log2 transitions)
//   vit_i/vit_j[1..nsteps]: the Viterbi path (Hit.i / Hit.j), i1..j2 its end points
//   excl_n previous MAC alignments of the same template: concatenated (i,j) lists, excl_off[excl_n+1]
// Outputs: MAC path out_i/out_j/out_states[1..nsteps'], P_posterior per step, res[6] = {i1,i2,j1,j2,nsteps,
// matched_cols}, fres[2] = {sum_of_probs, forward score before restoreHitValues}, *pforward,
// post[(Lq+1)*(Lt+1)] the posterior matrix (optional).
// par.exclstr / par.template_exclstr for the following hhref_mac_realign calls ("" = none)
static std::string g_mac_exclstr, g_mac_texclstr;
void hhref_set_mac_exclstr(const char* q, const char* t) { g_mac_exclstr = q ? q : ""; g_mac_texclstr = t ? t : ""; }

int hhref_mac_realign(int Lt, const float* t_p, const float* t_tr, int local, float shift, float mact, float corr,
                      int min_overlap, int i1, int i2, int j1, int j2, int nsteps, const int* vit_i,
                      const int* vit_j, int excl_n, const int* excl_off, const int* excl_i, const int* excl_j,
                      int* res, float* fres, double* pforward, int* out_i, int* out_j, char* out_states,
                      float* out_post_steps, float* post, float* t_tr_lin_out, float* q_tr_lin_out) {
  const int Lq = g->q->L;
  if (Lt + 2 > g->maxres) return -2;
  // query copy in linear space
  HMM* q = new HMM(MAXSEQDIS, g->maxres);
  *q = *g->q;
  q->trans_lin = 0;
  q->Log2LinTransitionProbs(1.0);
  {
    PosteriorDecoderRunner r(nullptr, nullptr, 1, 0.0f, g->S73, g->S33, g->S37);
    r.initializeQueryHMMTransitions(*q);
  }
  HMM* t = new HMM(MAXSEQDIS, g->maxres);
  fill_hmm(t, Lt, t_p, t_tr, nullptr, nullptr, nullptr);
  t->trans_lin = 0;
  t->Log2LinTransitionProbs(1.0);
  Hit hit;
  hit.L = Lt;
  hit.self = 0;
  hit.i1 = i1; hit.i2 = i2; hit.j1 = j1; hit.j2 = j2; hit.nsteps = nsteps;
  hit.i = new int[i2 + j2 + 2]; hit.j = new int[i2 + j2 + 2]; hit.states = new char[i2 + j2 + 2];
  for (int s = 1; s <= nsteps; ++s) { hit.i[s] = vit_i[s]; hit.j[s] = vit_j[s]; hit.states[s] = 0; }
  hit.ssm1 = hit.ssm2 = 0;
  hit.score = hit.score_ss = hit.score_aass = 0; hit.Pval = hit.Pvalt = hit.logPval = hit.logPvalt = 0;
  hit.Eval = hit.logEval = hit.Probab = 0;
  PosteriorMatrix pm;
  pm.allocateMatrix(Lq, Lt);
  ViterbiMatrix vm;
  vm.AllocateBacktraceMatrix(Lq, Lt);
  for (int i = 0; i <= Lq; ++i) memset(vm.getRow(i), 0, (size_t)(Lt + 1) * VECSIZE_FLOAT);
  PosteriorDecoder dec(Lt, local != 0, Lq, 0.0f, g->S73, g->S33, g->S37);
  std::vector<std::vector<int>*> keep;
  std::vector<PosteriorDecoder::MACBacktraceResult> excl;
  for (int e = 0; e < excl_n; ++e) {
    std::vector<int>* ai = new std::vector<int>(excl_i + excl_off[e], excl_i + excl_off[e + 1]);
    std::vector<int>* aj = new std::vector<int>(excl_j + excl_off[e], excl_j + excl_off[e + 1]);
    keep.push_back(ai); keep.push_back(aj);
    excl.push_back(PosteriorDecoder::MACBacktraceResult(ai, aj));
  }
  // realign() minus restoreHitValues' effect on what we export: run the public entry, then read the fields
  dec.realign(*q, *t, hit, pm, vm, excl, g_mac_exclstr.empty() ? nullptr : &g_mac_exclstr[0],
              g_mac_texclstr.empty() ? nullptr : &g_mac_texclstr[0], min_overlap, shift, mact, corr);
  res[0] = hit.i1; res[1] = hit.i2; res[2] = hit.j1; res[3] = hit.j2; res[4] = hit.nsteps; res[5] = hit.matched_cols;
  fres[0] = hit.sum_of_probs; fres[1] = 0;
  *pforward = hit.Pforward;
  for (int s = 0; s <= hit.nsteps; ++s) {
    out_i[s] = hit.i[s]; out_j[s] = hit.j[s]; out_states[s] = s ? hit.states[s] : 0;
    out_post_steps[s] = (s && hit.P_posterior) ? hit.P_posterior[s] : 0.f;
  }
  if (post)
    for (int i = 0; i <= Lq; ++i)
      for (int j = 0; j <= Lt; ++j) post[(size_t)i * (Lt + 1) + j] = (i && j) ? pm.getPosteriorValue(i, j) : 0.f;
  if (t_tr_lin_out) for (int i = 0; i <= Lt; ++i) for (int k = 0; k < 7; ++k) t_tr_lin_out[i * 7 + k] = t->tr[i][k];
  if (q_tr_lin_out) for (int i = 0; i <= Lq; ++i) for (int k = 0; k < 7; ++k) q_tr_lin_out[i * 7 + k] = q->tr[i][k];
  const int n = hit.nsteps;
  for (auto v : keep) delete v;
  pm.DeleteProbabilityMatrix();
  delete q; delete t;
  return n;
}

// Debug: forward pass only (same setup as hhref_mac_realign), exports the forward matrix and the scale factors.
int hhref_mac_forward_only(int Lt, const float* t_p, const float* t_tr, int local, float shift, int i1, int i2, int j1,
                           int j2, int nsteps, const int* vit_i, const int* vit_j, float* fwd, double* scale_out,
                           double* pforward) {
  const int Lq = g->q->L;
  HMM* q = new HMM(MAXSEQDIS, g->maxres);
  *q = *g->q;
  q->trans_lin = 0;
  q->Log2LinTransitionProbs(1.0);
  { PosteriorDecoderRunner r(nullptr, nullptr, 1, 0.0f, g->S73, g->S33, g->S37); r.initializeQueryHMMTransitions(*q); }
  HMM* t = new HMM(MAXSEQDIS, g->maxres);
  fill_hmm(t, Lt, t_p, t_tr, nullptr, nullptr, nullptr);
  t->trans_lin = 0;
  t->Log2LinTransitionProbs(1.0);
  Hit hit;
  hit.L = Lt; hit.self = 0;
  hit.i1 = i1; hit.i2 = i2; hit.j1 = j1; hit.j2 = j2; hit.nsteps = nsteps;
  hit.i = new int[i2 + j2 + 2]; hit.j = new int[i2 + j2 + 2]; hit.states = new char[i2 + j2 + 2];
  for (int s = 1; s <= nsteps; ++s) { hit.i[s] = vit_i[s]; hit.j[s] = vit_j[s]; hit.states[s] = 0; }
  hit.ssm1 = hit.ssm2 = 0;
  PosteriorMatrix pm; pm.allocateMatrix(Lq, Lt);
  ViterbiMatrix vm; vm.AllocateBacktraceMatrix(Lq, Lt);
  for (int i = 0; i <= Lq; ++i) memset(vm.getRow(i), 0, (size_t)(Lt + 1) * VECSIZE_FLOAT);
  PosteriorDecoder dec(Lt, local != 0, Lq, 0.0f, g->S73, g->S33, g->S37);
  dec.initializeForAlignment(*q, *t, hit, vm, 0, t->L, 0);
  dec.forwardAlgorithm(*q, *t, hit, pm, vm, shift, 0);
  for (int i = 0; i <= Lq; ++i)
    for (int j = 0; j <= Lt; ++j) fwd[(size_t)i * (Lt + 1) + j] = (i && j) ? pm.getPosteriorValue(i, j) : 0.f;
  for (int i = 0; i <= Lq + 1; ++i) scale_out[i] = dec.scale[i];
  *pforward = hit.Pforward;
  pm.DeleteProbabilityMatrix();
  delete q; delete t;
  return 0;
}

// fast_log2 of the reference (table-based, src/util-inl.h:108-128) and Score() (src/hhhit-inl.h:132)
float hhref_fast_log2(float x) { return fast_log2(x); }
float hhref_score_cols(const float* qi, const float* tj) {
  float q[20] __attribute__((aligned(32))), t[20] __attribute__((aligned(32)));
  memcpy(q, qi, 80); memcpy(t, tj, 80);
  return Score(q, t);
}

// Run the reference AVX2 kernel on one batch of n<=VECSIZE_FLOAT prepared targets.
//  t_p[k]: (Lt+2)*20, t_tr[k]: (Lt+1)*7 in HMM enum order, t_ss_pred/conf[k]: Lt+2 bytes or NULL
//  celloff[k]: (Lq+1)*(Lt_k+1) bytes (non-zero = cell off) or NULL
//  bt_out[k]:  (Lq+1)*(Lt_k+1) bytes, row-major [i][j], filled for 1<=i<=Lq,1<=j<=Lt_k
int hhref_viterbi_align(int n, const int* Lt, const float* const* t_p, const float* const* t_tr,
                        const unsigned char* const* t_ss_pred, const unsigned char* const* t_ss_conf,
                        const unsigned char* const* celloff, int use_ss, int local, float egq,
                        float egt, float shift, float ssw, float corr, float* score, int* i2,
                        int* j2, unsigned char* const* bt_out) {
  if (n < 1 || n > VECSIZE_FLOAT) return -1;
  const int Lq = g->q->L;
  int maxLt = 0;
  std::vector<HMM*> v;
  for (int k = 0; k < n; ++k) {
    if (Lt[k] + 2 > g->maxres) return -2;
    fill_hmm(g->t_hmm[k], Lt[k], t_p[k], t_tr[k], t_ss_pred ? t_ss_pred[k] : nullptr,
             t_ss_conf ? t_ss_conf[k] : nullptr, nullptr);
    v.push_back(g->t_hmm[k]);
    maxLt = std::max(maxLt, Lt[k]);
  }
  g->t_simd->MapHMMVector(v);
  g->matrix->AllocateBacktraceMatrix(Lq, maxLt);
  // clear all bytes (a fresh reference matrix is not zeroed; cell-off bits must be defined)
  for (int i = 0; i <= Lq; ++i) memset(g->matrix->getRow(i), 0, (size_t)(maxLt + 1) * VECSIZE_FLOAT);
  g->matrix->setCellOff(false);
  bool any_co = false;
  if (celloff)
    for (int k = 0; k < n; ++k)
      if (celloff[k])
        for (int i = 1; i <= Lq; ++i)
          for (int j = 1; j <= Lt[k]; ++j)
            if (celloff[k][(size_t)i * (Lt[k] + 1) + j]) { g->matrix->setCellOff(i, j, k, true); any_co = true; }
  (void)any_co;
  delete g->viterbi;
  g->viterbi = new Viterbi(g->maxres, local != 0, egq, egt, corr, g->par->min_overlap, shift,
                           g->par->ssm, ssw, g->S73, g->S33, g->S37);
  const int ss_hmm_mode = use_ss ? HMM::PRED_PRED : HMM::NO_SS_INFORMATION;
  g->last_ss_mode = ss_hmm_mode;
  Viterbi::ViterbiResult* r = g->viterbi->Align(g->q_simd, g->t_simd, g->matrix, n, ss_hmm_mode);
  g->last = *r;
  for (int k = 0; k < n; ++k) {
    score[k] = r->score[k]; i2[k] = r->i[k]; j2[k] = r->j[k];
    if (bt_out && bt_out[k])
      for (int i = 1; i <= Lq; ++i) {
        const unsigned char* row = g->matrix->getRow(i);
        for (int j = 1; j <= Lt[k]; ++j)
          bt_out[k][(size_t)i * (Lt[k] + 1) + j] = row[j * VECSIZE_FLOAT + k];
      }
  }
  delete r;
  return 0;
}

// Viterbi::Backtrace on lane `elem` of the last batch. Arrays sized >= i2+j2+2. Returns nsteps.
int hhref_backtrace(int elem, int* i_steps, int* j_steps, char* states, int* matched_cols) {
  Viterbi::BacktraceResult b = Viterbi::Backtrace(g->matrix, elem, g->last.i, g->last.j);
  for (int s = 0; s <= b.count; ++s) { i_steps[s] = s ? b.i_steps[s] : 0; j_steps[s] = s ? b.j_steps[s] : 0; states[s] = s ? b.states[s] : 0; }
  *matched_cols = b.matched_cols;
  int n = b.count;
  delete[] b.i_steps; delete[] b.j_steps; delete[] b.states;
  return n;
}

// Hit.score as the runner computes it (src/hhviterbirunner.cpp:29-42 -> hhviterbi.cpp:195-281)
int hhref_score_for_backtrace(int elem, float* score, float* score_ss) {
  Viterbi::BacktraceResult b = Viterbi::Backtrace(g->matrix, elem, g->last.i, g->last.j);
  Viterbi::BacktraceScore s = g->viterbi->ScoreForBacktrace(g->q_simd, g->t_simd, elem, &b,
                                                            g->last.score, g->last_ss_mode);
  *score = s.score; *score_ss = s.score_ss;
  delete[] s.S; delete[] s.S_ss;
  delete[] b.i_steps; delete[] b.j_steps; delete[] b.states;
  return b.count;
}

// CPU baseline: the reference AVX2 kernel over N prepared targets, batched/sorted like the runner
// (src/hhviterbirunner.cpp:117-128).  db_p: concatenated per-target (L+2)*20, db_tr: (L+1)*7.
// Returns seconds spent in Align(+Backtrace); *cells = Lq * sum(Lt).
double hhref_viterbi_bench(int N, const int* Lt, const long long* p_off, const long long* tr_off,
                           const float* db_p, const float* db_tr, int threads, int with_backtrace,
                           int repeats, double* cells, float* scores_out) {
  const int V = VECSIZE_FLOAT;
  const int Lq = g->q->L;
  std::vector<int> order(N);
  for (int i = 0; i < N; ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return Lt[a] > Lt[b]; });
  const int nb = (N + V - 1) / V;
  int maxL = 0;
  for (int i = 0; i < N; ++i) maxL = std::max(maxL, Lt[i]);
  // Pre-map every batch to its lane-interleaved form (BASELINE.md §3.2: time only Align+Backtrace)
  std::vector<HMMSimd*> simd(nb);
  std::vector<std::vector<HMM*>> hmms(nb);
  for (int b = 0; b < nb; ++b) {
    int n = std::min(V, N - b * V);
    int bl = 0;
    for (int k = 0; k < n; ++k) bl = std::max(bl, Lt[order[b * V + k]]);
    simd[b] = new HMMSimd(bl + 2);
    for (int k = 0; k < n; ++k) {
      int t = order[b * V + k];
      HMM* h = new HMM(2, Lt[t] + 2);
      fill_hmm(h, Lt[t], db_p + p_off[t], db_tr + tr_off[t], nullptr, nullptr, nullptr);
      hmms[b].push_back(h);
    }
    simd[b]->MapHMMVector(hmms[b]);
  }
  std::vector<Viterbi*> vit(threads);
  std::vector<ViterbiMatrix*> mat(threads);
  for (int t = 0; t < threads; ++t) {
    vit[t] = new Viterbi(maxL + 2, g->par->loc, g->par->egq, g->par->egt, g->par->corr,
                         g->par->min_overlap, g->par->shift, g->par->ssm, g->par->ssw, g->S73,
                         g->S33, g->S37);
    mat[t] = new ViterbiMatrix();
    mat[t]->AllocateBacktraceMatrix(Lq, maxL);
  }
  double c = 0;
  for (int i = 0; i < N; ++i) c += (double)Lq * Lt[i];
  *cells = c * repeats;
  auto t0 = std::chrono::steady_clock::now();
  for (int rep = 0; rep < repeats; ++rep) {
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads)
    for (int b = 0; b < nb; ++b) {
      int tid = omp_get_thread_num();
      int n = std::min(V, N - b * V);
      Viterbi::ViterbiResult* r = vit[tid]->Align(g->q_simd, simd[b], mat[tid], n, HMM::NO_SS_INFORMATION);
      if (with_backtrace)
        for (int k = 0; k < n; ++k) {
          Viterbi::BacktraceResult bt = Viterbi::Backtrace(mat[tid], k, r->i, r->j);
          delete[] bt.i_steps; delete[] bt.j_steps; delete[] bt.states;
        }
      if (scores_out)
        for (int k = 0; k < n; ++k) scores_out[order[b * V + k]] = r->score[k];
      delete r;
    }
  }
  auto t1 = std::chrono::steady_clock::now();
  for (int b = 0; b < nb; ++b) { for (HMM* h : hmms[b]) delete h; delete simd[b]; }
  for (int t = 0; t < threads; ++t) { delete vit[t]; delete mat[t]; }
  return std::chrono::duration<double>(t1 - t0).count();
}

// ---------------------------------------------------------------- prefilter pieces
static void ensure_prefilter() {
  if (g->prefilter) return;
  // Prefilter's ctor needs an ffindex DB; the three routines we call only use cs_lib.
  g->prefilter = (Prefilter*)calloc(1, sizeof(Prefilter));
  FILE* fin = fmemopen((void*)_binary_cs219_lib_start,
                       (size_t)(_binary_cs219_lib_end - _binary_cs219_lib_start), "r");
  g->prefilter->cs_lib = new cs::ContextLibrary<cs::AA>(fin);
  fclose(fin);
  cs::TransformToLin(*g->prefilter->cs_lib);
}

// 219 x 20 linear column-state probabilities (cs219.lib after TransformToLin, src/hhprefilter.cpp:41-44)
int hhref_get_cs219(float* out) {
  ensure_prefilter();
  const cs::ContextLibrary<cs::AA>& lib = *g->prefilter->cs_lib;
  for (int k = 0; k < (int)cs::AS219::kSize; ++k)
    for (int a = 0; a < 20; ++a) out[k * 20 + a] = lib[k].probs[0][a];
  return (int)cs::AS219::kSize;
}

// striped query profile from the CURRENT query HMM; qc must hold 220*(Lq+32) bytes. Returns W.
int hhref_stripe_query_profile(int score_offset, int bit_factor, unsigned char* qc) {
  ensure_prefilter();
  const int ec = VECSIZE_INT * 4;
  const int W = (g->q->L + ec - 1) / ec;
  g->prefilter->stripe_query_profile(g->q, score_offset, bit_factor, W, qc);
  return W;
}

int hhref_ungapped_score(const unsigned char* qc, int Lq, const unsigned char* dbseq, int L, int offset) {
  ensure_prefilter();
  const int ec = VECSIZE_INT * 4;
  simd_int* ws = (simd_int*)malloc_simd_int(3 * (Lq + ec) * sizeof(char));
  int s = g->prefilter->ungapped_sse_score(qc, Lq, dbseq, L, (unsigned char)offset, ws);
  free(ws);
  return s;
}

int hhref_sw_striped_byte(unsigned char* qc, int Lq, unsigned char* dbseq, int L, int gap_open,
                          int gap_extend, int offset) {
  ensure_prefilter();
  const int ec = VECSIZE_INT * 4;
  const int W = (Lq + ec - 1) / ec;
  simd_int* ws = (simd_int*)malloc_simd_int(3 * (Lq + ec) * sizeof(char));
  int s = g->prefilter->swStripedByte(qc, Lq, dbseq, L, (unsigned short)gap_open,
                                      (unsigned short)gap_extend, ws, ws + W, ws + 2 * W,
                                      (unsigned short)offset);
  free(ws);
  return s;
}

// Reference ungapped prefilter over a whole cs219 DB on `threads` cores (src/hhprefilter.cpp:466-482).
double hhref_ungapped_bench(const unsigned char* qc, int Lq, int N, const unsigned char* db,
                            const long long* off, const int* len, int offset, int threads,
                            int* scores) {
  ensure_prefilter();
  const int ec = VECSIZE_INT * 4;
  std::vector<simd_int*> ws(threads);
  for (int t = 0; t < threads; ++t) ws[t] = (simd_int*)malloc_simd_int(3 * (Lq + ec) * sizeof(char));
  auto t0 = std::chrono::steady_clock::now();
#pragma omp parallel for schedule(static) num_threads(threads)
  for (int n = 0; n < N; ++n)
    scores[n] = g->prefilter->ungapped_sse_score(qc, Lq, db + off[n], len[n], (unsigned char)offset,
                                                 ws[omp_get_thread_num()]);
  auto t1 = std::chrono::steady_clock::now();
  for (int t = 0; t < threads; ++t) free(ws[t]);
  return std::chrono::duration<double>(t1 - t0).count();
}

}  // extern "C"


// ---------------------------------------------------------------- hit-list statistics (a13)
// Build a HitList of n Hits carrying (score, score_ss, L, Neff_HMM, ssm2, file), run the reference's
// HitList::CalculatePvalues (src/hhhitlist.cpp:499) and optionally CalculateHHblitsEvalues (:465), return the per-hit
// values (indexed by input position via Hit.index) and the list order after each sort.
extern "C" int hhref_hitlist_stats(int n, const float* score, const float* score_ss, const int* L, const float* neff,
                                   const int* ssm2, const char* const* file, int qL, float qneff, int N_searched, int loc,
                                   int ssm, float ssw, int hhblits, int dbsize, float alphaa, float alphab, float alphac,
                                   double pf_evalue_thresh, double* pval, double* logpval, double* eval, double* logeval,
                                   float* score_aass, float* probab, int* order) {
  HitList* hl = new HitList();
  HMM q(2, qL + 2);
  q.L = qL;
  q.Neff_HMM = qneff;
  std::vector<char*> names(n);
  for (int k = 0; k < n; ++k) {
    Hit h;
    h.score = score[k]; h.score_ss = score_ss[k]; h.L = L[k]; h.Neff_HMM = neff[k];
    h.ssm1 = 0; h.ssm2 = ssm2 ? ssm2[k] : 0;
    h.nfirst = k;                 // carries the input position through the sorts
    names[k] = strdup(file ? file[k] : "x");
    h.file = names[k];
    hl->Push(h);
  }
  hl->N_searched = N_searched;
  hl->CalculatePvalues(&q, (char)loc, (char)ssm, ssw);
  if (hhblits) hl->CalculateHHblitsEvalues(&q, dbsize, alphaa, alphab, alphac, pf_evalue_thresh);
  int pos = 0;
  hl->Reset();
  while (!hl->End()) {
    Hit h = hl->ReadNext();
    const int k = h.nfirst;
    pval[k] = h.Pval; logpval[k] = h.logPval; eval[k] = h.Eval; logeval[k] = h.logEval;
    score_aass[k] = h.score_aass; probab[k] = h.Probab;
    order[pos++] = k;
  }
  for (char* p : names) free(p);
  delete hl;
  return pos;
}


// ViterbiRunner::calculateEarlyStop (src/hhviterbirunner.cpp:213) on synthetic hits
extern "C" float hhref_early_stop(int n, const float* score, const int* L, const float* neff, int qL, float qneff,
                                  int prefilter, int dbsize, float alphaa, float alphab, float alphac, double thresh) {
  Parameters par = *g->par;
  par.prefilter = prefilter; par.dbsize = dbsize; par.alphaa = alphaa; par.alphab = alphab; par.alphac = alphac;
  par.prefilter_evalue_thresh = thresh;
  HMM q(2, qL + 2);
  q.L = qL; q.Neff_HMM = qneff;
  std::vector<Hit> hits(n);
  for (int k = 0; k < n; ++k) { hits[k].score = score[k]; hits[k].L = L[k]; hits[k].Neff_HMM = neff[k]; }
  std::vector<HHblitsDatabase*> nodb;
  ViterbiRunner r(nullptr, nodb, 1);
  return r.calculateEarlyStop(par, &q, hits, 0);
}


// ---------------------------------------------------------------- A3M -> HMM (rows a10 / f1)
// The template branch of HHEntry::getTemplateHMM for an A3M record (src/hhdatabase.cpp:441-449): Alignment::Read,
// Compress (par.M_template), Filter (par.max_seqid_db / coverage_db / qid_db / qsc / Ndiff_db), FrequenciesAndTransitions.
// Exports the alignment as the reference holds it after filtering (X, I, keep, wg, nres, ksort) and the raw HMM
// (f, tr, Neff_M/I/D, Neff_HMM, ss); with prep != 0 PrepareTemplateHMM's query-independent steps are run as well and
// p / tr / pav exported like hhref_prepare_template_hhm_raw's p_raw.
// filt[5] = {max_seqid, coverage, qid, qsc, Ndiff} (NULL: the reference defaults); wg_mode = par.wg.
// dims[8] = {L, N_in, N_filtered, kfirst, kss_pred, kss_conf, kss_dssp, N_ss}
static int msa_export(Alignment* ali, const char* name, const float* filt, int wg_mode, int prep, int capL, int capN, int* dims,
                      unsigned char* X, unsigned short* I, signed char* keep, float* wg, int* nres, int* ksort,
                      float* f, float* tr, float* neff, float* neff_hmm, unsigned char* ss_pred,
                      unsigned char* ss_conf, float* p, float* tr_prep, float* pav) {
  Parameters& par = *g->par;
  char nm[NAMELEN];
  strncpy(nm, name, NAMELEN - 1); nm[NAMELEN - 1] = 0;
  ali->Compress(nm, par.cons, par.maxcol, par.M_template, par.Mgaps);
  const int max_seqid = filt ? (int)filt[0] : par.max_seqid_db;
  const int coverage = filt ? (int)filt[1] : par.coverage_db;
  const int qid = filt ? (int)filt[2] : par.qid_db;
  const float qsc = filt ? filt[3] : par.qsc_db;
  const int Ndiff = filt ? (int)filt[4] : par.Ndiff_db;
  ali->N_filtered = ali->Filter(max_seqid, g->S, coverage, qid, qsc, Ndiff);
  HMM* t = new HMM(MAXSEQDIS, g->maxres);
  t->name[0] = t->longname[0] = t->fam[0] = 0;
  ali->FrequenciesAndTransitions(t, (char)wg_mode, par.mark, par.cons, par.showcons, g->pb, g->Sim);
  const int L = ali->L, N = ali->N_in;
  dims[0] = L; dims[1] = N; dims[2] = ali->N_filtered; dims[3] = ali->kfirst; dims[4] = ali->kss_pred;
  dims[5] = ali->kss_conf; dims[6] = ali->kss_dssp; dims[7] = ali->N_ss;
  if (L > capL || N > capN) { delete t; return -2; }
  for (int k = 0; k < N; ++k) {
    for (int i = 0; i <= L + 1; ++i) X[(size_t)k * (L + 2) + i] = (unsigned char)ali->X[k][i];
    for (int i = 0; i <= L; ++i) I[(size_t)k * (L + 2) + i] = (ali->keep[k] || k == ali->kfirst) ? ali->I[k][i] : 0;
    keep[k] = ali->keep[k];
    wg[k] = ali->wg[k];
    nres[k] = ali->nres ? ali->nres[k] : -1;
    ksort[k] = ali->ksort ? ali->ksort[k] : -1;
  }
  for (int i = 0; i <= L + 1; ++i)
    for (int a = 0; a < 20; ++a) f[(size_t)i * 20 + a] = t->f[i][a];
  for (int i = 0; i <= L; ++i) {
    for (int k = 0; k < 7; ++k) tr[(size_t)i * 7 + k] = t->tr[i][k];
    neff[i] = t->Neff_M[i]; neff[(L + 1) + i] = t->Neff_I[i]; neff[2 * (L + 1) + i] = t->Neff_D[i];
  }
  *neff_hmm = t->Neff_HMM;
  for (int i = 0; i <= L + 1; ++i) {
    ss_pred[i] = (t->nss_pred >= 0 && i >= 1 && i <= L) ? (unsigned char)t->ss_pred[i] : 0;
    ss_conf[i] = (t->nss_pred >= 0 && i >= 1 && i <= L) ? (unsigned char)t->ss_conf[i] : 0;
  }
  if (prep) {
    t->AddTransitionPseudocounts(par.gapd, par.gape, par.gapf, par.gapg, par.gaph, par.gapi, par.gapb, par.gapb);
    t->PreparePseudocounts(g->R);
    t->AddAminoAcidPseudocounts(par.pc_hhm_nocontext_mode, par.pc_hhm_nocontext_a, par.pc_hhm_nocontext_b,
                                par.pc_hhm_nocontext_c);
    t->CalculateAminoAcidBackground(g->pb);
    export_hmm(t, p, tr_prep, pav, nullptr, nullptr, nullptr, nullptr);
  }
  delete t;
  return L;
}

extern "C" int hhref_msa_to_hmm(const char* path, const float* filt, int wg_mode, int prep, int capL, int capN, int* dims,
                                unsigned char* X, unsigned short* I, signed char* keep, float* wg, int* nres, int* ksort,
                                float* f, float* tr, float* neff, float* neff_hmm, unsigned char* ss_pred,
                                unsigned char* ss_conf, float* p, float* tr_prep, float* pav) {
  FILE* fh = fopen(path, "r");
  if (!fh) return -1;
  Parameters& par = *g->par;
  Alignment* ali = new Alignment(par.maxseq, g->maxres);
  char name[NAMELEN];
  strncpy(name, path, NAMELEN - 1); name[NAMELEN - 1] = 0;
  ali->Read(fh, name, par.mark, par.maxcol, par.nseqdis);
  fclose(fh);
  const int rc = msa_export(ali, path, filt, wg_mode, prep, capL, capN, dims, X, I, keep, wg, nres, ksort, f, tr, neff, neff_hmm,
                            ss_pred, ss_conf, p, tr_prep, pav);
  delete ali;
  return rc;
}

// The compressed branch of HHDatabaseEntry::getTemplateHMM (src/hhdatabase.cpp:303-326): entry `entry_name` of
// <prefix>_ca3m.ff{data,index}, decoded with <prefix>_sequence.ff* and <prefix>_header.ff* by Alignment::ReadCompressed.
extern "C" int hhref_ca3m_to_hmm(const char* prefix, const char* entry_name, const float* filt, int wg_mode, int prep, int capL,
                                 int capN, int* dims, unsigned char* X, unsigned short* I, signed char* keep, float* wg,
                                 int* nres, int* ksort, float* f, float* tr, float* neff, float* neff_hmm,
                                 unsigned char* ss_pred, unsigned char* ss_conf, float* p, float* tr_prep, float* pav) {
  struct FF { FILE* fd = nullptr; FILE* fi = nullptr; char* data = nullptr; size_t size = 0; ffindex_index_t* index = nullptr; };
  auto open_ff = [&](const char* suffix, FF& ff) {
    const std::string base = std::string(prefix) + suffix;
    ff.fd = fopen((base + ".ffdata").c_str(), "r");
    ff.fi = fopen((base + ".ffindex").c_str(), "r");
    if (!ff.fd || !ff.fi) return false;
    ff.data = ffindex_mmap_data(ff.fd, &ff.size);
    ff.index = ffindex_index_parse(ff.fi, ffcount_lines((base + ".ffindex").c_str()));   // 0 would reserve 200 M entries
    return ff.data && ff.index;
  };
  FF ca, sq, hd;
  if (!open_ff("_ca3m", ca) || !open_ff("_sequence", sq) || !open_ff("_header", hd)) return -1;
  ffindex_entry_t* entry = ffindex_get_entry_by_name(ca.index, const_cast<char*>(entry_name));
  if (!entry) return -3;
  Parameters& par = *g->par;
  Alignment* ali = new Alignment(par.maxseq, g->maxres);
  char* data = ffindex_get_data_by_entry(ca.data, entry);
  ali->ReadCompressed(entry, data, sq.index, sq.data, hd.index, hd.data, par.mark, par.maxcol);
  const int rc = msa_export(ali, entry->name, filt, wg_mode, prep, capL, capN, dims, X, I, keep, wg, nres, ksort, f, tr, neff,
                            neff_hmm, ss_pred, ss_conf, p, tr_prep, pav);
  delete ali;
  for (FF* ff : {&ca, &sq, &hd}) {
    if (ff->index) ffindex_index_free(ff->index);
    if (ff->data) munmap(ff->data, ff->size);
    if (ff->fd) fclose(ff->fd);
    if (ff->fi) fclose(ff->fi);
  }
  return rc;
}

// par.M_template / par.Mgaps (-M a2m | first | <percent>) for the following hhref_msa_to_hmm calls
extern "C" void hhref_set_M(int M, int Mgaps) { g->par->M_template = M; g->par->Mgaps = Mgaps; }

// _mm_rcp_ps of this host (Alignment::Amino_acid_frequencies_and_transitions_from_M_state uses simdf32_rcp,
// src/hhalignment.cpp:2531): lets a test compare the product's own sampled table with the reference build's view.
extern "C" void hhref_rcp_table(int n, float* out) {
  for (int m = 0; m < n; m += VECSIZE_FLOAT) {
    float in[VECSIZE_FLOAT] __attribute__((aligned(32))), res[VECSIZE_FLOAT] __attribute__((aligned(32)));
    for (int v = 0; v < VECSIZE_FLOAT; ++v) in[v] = (float)(m + v);
    simdf32_store(res, simdf32_rcp(simdf32_load(in)));
    for (int v = 0; v < VECSIZE_FLOAT && m + v < n; ++v) out[m + v] = res[v];
  }
}


// ---------------------------------------------------------------- context-specific pseudocounts (row a12)
// The CRF engine of the reference (InitializePseudocountsEngine, src/hhfunc.cpp:204-244) on demand, independent of the
// nocontxt flag the shim was initialised with.
static void ensure_context() {
  if (g->pc_hhm_context_engine) return;
  InitializePseudocountsEngine(*g->par, g->context_lib, g->crf, g->pc_hhm_context_engine, g->pc_hhm_context_mode,
                               g->pc_prefilter_context_engine, g->pc_prefilter_context_mode);
}

// par.clusterfile (-contxt <file>): rebuild the CRF engines from that .crf file instead of the embedded context_data.crf
extern "C" int hhref_set_contxt(const char* path) {
  g->par->clusterfile = path;
  InitializePseudocountsEngine(*g->par, g->context_lib, g->crf, g->pc_hhm_context_engine, g->pc_hhm_context_mode,
                               g->pc_prefilter_context_engine, g->pc_prefilter_context_mode);
  return g->crf ? (int)g->crf->size() : -1;
}

// state k of the CRF library in use: pc[20], bias, w[13*20]
extern "C" int hhref_crf_state(int k, double* pc, double* bias, double* w) {
  ensure_context();
  if (!g->crf || k < 0 || k >= (int)g->crf->size()) return -1;
  const cs::CrfState<cs::AA>& s = (*g->crf)[k];
  for (int a = 0; a < 20; ++a) pc[a] = s.pc[a];
  *bias = s.bias_weight;
  for (size_t j = 0; j < s.context_weights.length(); ++j)
    for (int a = 0; a < 20; ++a) w[j * 20 + a] = s.context_weights[j][a];
  return (int)g->crf->size();
}

// HMM::AddContextSpecificPseudocounts (src/hhhmm.cpp:1820) + CalculateAminoAcidBackground on an HMM with the given raw
// frequencies f[(L+2)*20] and Neff_M[L+1]; engine 0 = query HMM (par.pc_hhm_context_engine), 1 = prefilter profile.
extern "C" int hhref_context_pc(int L, const float* f, const float* neff_m, float neff_hmm, int engine, float* p, float* pav) {
  ensure_context();
  HMM* h = new HMM(MAXSEQDIS, g->maxres);
  h->L = L;
  h->has_pseudocounts = false;
  h->Neff_HMM = neff_hmm;
  for (int i = 0; i <= L + 1; ++i) for (int a = 0; a < 20; ++a) h->f[i][a] = f[(size_t)i * 20 + a];
  for (int i = 0; i <= L; ++i) h->Neff_M[i] = neff_m[i];
  if (engine == 0) h->AddContextSpecificPseudocounts(g->pc_hhm_context_engine, g->pc_hhm_context_mode);
  else h->AddContextSpecificPseudocounts(g->pc_prefilter_context_engine, g->pc_prefilter_context_mode);
  h->CalculateAminoAcidBackground(g->pb);
  for (int i = 0; i <= L + 1; ++i) for (int a = 0; a < 20; ++a) p[(size_t)i * 20 + a] = h->p[i][a];
  for (int a = 0; a < 20; ++a) pav[a] = h->pav[a];
  delete h;
  return L;
}

// the embedded context_data.crf text, so tests can hand it to the product without reading /root/reference
extern "C" const unsigned char* hhref_crf_text(long long* len) {
  *len = (long long)context_data_crf_len;
  return context_data_crf;
}
