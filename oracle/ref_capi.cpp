/*
 * ref_capi.cpp -- C ABI over the UNMODIFIED REFERENCE sources (TEST INFRASTRUCTURE ONLY).
 *
 * `make -C oracle ref` compiles /root/reference/src/{linalg,covfuncs,modandbase,fit}.cpp where they lie (nothing is
 * copied into this repository) against oracle/arma_shim/RcppArmadillo.h -- a header-only Armadillo subset written for
 * this purpose -- and links them with this file into oracle/_ref/libob_ref.so.  The library exports the ABI of
 * include/outerbase_b200.h with every `ob_` replaced by `ref_`, so the one Python binding (outerbase_b200/binding.py)
 * drives the reference itself: tests/test_oracle_ref.py pins the CPU oracle against it, bench.py's `--impl reference`
 * arm times it.  What is NOT the reference here, and why:
 *   - setcovfs / setknot live in src/interfaceR.cpp (an Rcpp module, cannot be compiled without R): restated below
 *     from interfaceR.cpp:53-73, 94-149;
 *   - eig_sym (LAPACK upstream) is the oracle's cyclic Jacobi, shuffle (R's RNG upstream) the oracle's tie-break
 *     policy: both sides of every comparison share them (SURVEY 8c "third-party arithmetic");
 *   - private members (rotmat, basescale, ...) are read through `#define private public` -- layout is unaffected.
 */
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "customconfig.h"
#include <RcppArmadillo.h>
using namespace arma;
#define private public
#include "covfuncs.h"
#include "modandbase.h"
#include "fit.h"
#undef private
#include "linalg.h"

#include "_gen/ref_api.h"

extern "C" void orc_eig_sym_jacobi(uint64_t n, const double* A, double* w, double* V);
extern "C" void arma_shim_eig_sym(std::uint64_t n, const double* A, double* w, double* V) { orc_eig_sym_jacobi(n, A, w, V); }

static thread_local std::string g_err;
#define REF_TRY try {
#define REF_CATCH                                                                      \
  }                                                                                    \
  catch (const std::range_error& e) { g_err = e.what(); return REF_ERR_INVALID; }      \
  catch (const std::invalid_argument& e) { g_err = e.what(); return REF_ERR_INVALID; } \
  catch (const std::exception& e) { g_err = e.what(); return REF_ERR_STATE; }          \
  return REF_OK;

struct ref_ctx { int nthreads; };
struct ref_outermod { outermod om; uint64_t select_seed = 0; };
struct ref_outerbase { std::unique_ptr<outerbase> ob; umat terms; };
/* optcg's iteration counter is a local of lpdf::optcg (fit.cpp:68): count the hessmult calls instead (one before the
 * loop, one per iteration) */
template <class Base> struct counting : Base {
  using Base::Base;
  unsigned hm_calls = 0;
  vec hessmult(const vec& g) override { ++hm_calls; return Base::hessmult(g); }
};
struct ref_lpdf {
  std::unique_ptr<lpdf> p;
  int kind = 0; /* 0 loglik_gauss, 1 logpr_gauss, 2 lpdfvec, 3 loglik_gda */
  uint64_t nhyp = 0, nrow = 0, d = 0, cg_iters = 0;
  unsigned* hm = nullptr;
  ref_lpdf *a = nullptr, *b = nullptr;
};
struct ref_predictor { std::unique_ptr<predictor> p; uint64_t d; };

static umat to_umat(const uint64_t* t, uint64_t K, uint64_t d) { return umat(reinterpret_cast<const uword*>(t), K, d); }
static mat to_mat(const double* x, uint64_t r, uint64_t c) { return mat(x, r, c); }
static vec to_vec(const double* x, uint64_t n) { return vec(x, n); }
template <class M> static void put(const M& m, double* out) { if (m.n_elem) std::memcpy(out, m.mem, m.n_elem * sizeof(double)); }

/* the OpenMP tuning outerbase::setloopvals_ derives (modandbase.cpp:504-513), for the stateless seam */
struct loopvals { bool vertpl; uword chunksize, loopsize; int nthreads; };
static loopvals default_lv(uint64_t N) {
  int T = 1;
#ifdef _OPENMP
  T = omp_get_num_procs();
#endif
  const uword chunk = std::max<uword>(32, std::min<uword>(1 + 2048 / T, N / (4 * T) + 1));
  const uword loops = (N + chunk - 1) / chunk;
  return {loops > 20, chunk, loops, T};
}

/* selectterms' tie-break (modandbase.cpp:406-409 shuffles with R's RNG): seed 0 = lowest index, else the oracle's
 * SplitMix64 stream -- the chosen candidate moves to the front, which is all selectterms reads (islarge(0)) */
static uint64_t g_rng = 0;
static uint64_t splitmix64(uint64_t& s) {
  uint64_t z = (s += 0x9E3779B97F4A7C15ull);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

extern "C" {

const char* ref_last_error(void) { return g_err.c_str(); }
int ref_version(void) { return 1; }
int ref_ctx_create(int, ref_ctx** out) {
  int nt = 1;
#ifdef _OPENMP
  nt = omp_get_num_procs();
#endif
  *out = new ref_ctx{nt};
  return REF_OK;
}
int ref_ctx_destroy(ref_ctx* c) { delete c; return REF_OK; }
int ref_ctx_synchronize(ref_ctx*) { return REF_OK; }
int ref_ctx_stream(ref_ctx*, void** s) { *s = nullptr; return REF_OK; }
int ref_comm_get_unique_id(void* id) { std::memset(id, 0, 128); return REF_OK; }
int ref_ctx_comm_init(ref_ctx*, int, int, const void*) { g_err = "the reference is single-rank"; return REF_ERR_STATE; }
int ref_ctx_comm_info(ref_ctx*, int* n, int* r) { *n = 1; *r = 0; return REF_OK; }
int ref_ctx_allreduce_dev(ref_ctx*, double*, uint64_t) { return REF_OK; }
int ref_ctx_fp64_peak(ref_ctx*, double* t) { *t = 0; return REF_OK; }
int ref_ctx_launch_count(ref_ctx*, uint64_t* c) { *c = 0; return REF_OK; }
int ref_ctx_set_option(ref_ctx*, const char*, double) { return REF_OK; }
int ref_outerbase_specialize(ref_outerbase*, const uint64_t*, uint64_t, double* s) { if (s) *s = 0; return REF_OK; }
int ref_outerbase_spec_state(ref_outerbase*, const uint64_t*, uint64_t, int* st) { if (st) *st = 0; return REF_OK; }
int ref_spec_source(const uint64_t*, uint64_t, uint64_t, const int*, char*, uint64_t*, uint64_t*) { g_err = "the reference has no kernels"; return REF_ERR_STATE; }
int ref_spec_source_dot(const uint64_t*, uint64_t, uint64_t, char*, uint64_t*, uint64_t*) { g_err = "the reference has no kernels"; return REF_ERR_STATE; }
int ref_spec_source_mat(const uint64_t*, uint64_t, uint64_t, char*, uint64_t*, uint64_t*) { g_err = "the reference has no kernels"; return REF_ERR_STATE; }
int ref_spec_source_tmat(const uint64_t*, uint64_t, uint64_t, char*, uint64_t*, uint64_t*) { g_err = "the reference has no kernels"; return REF_ERR_STATE; }
int ref_spec_compile_check(const char*, uint64_t*, double*) { g_err = "the reference has no kernels"; return REF_ERR_STATE; }
int ref_debug_terms_eval(const uint64_t*, uint64_t, uint64_t, const uint64_t*, int, int, const double*, const double*, const double*, double,
                         double*, double*, uint64_t*) { g_err = "the reference has no terms compiler"; return REF_ERR_STATE; }
int ref_outerbase_debug_phi_geometry(ref_outerbase*, const uint64_t*, uint64_t, int, int, int*) { g_err = "the reference has no kernels"; return REF_ERR_STATE; }
int ref_outerbase_debug_build_geometry(ref_outerbase*, int*) { g_err = "the reference has no kernels"; return REF_ERR_STATE; }
int ref_lpdf_debug_build_geometry(ref_lpdf*, int*) { g_err = "the reference has no kernels"; return REF_ERR_STATE; }

static covf* make_covf(const std::string& n) { /* interfaceR.cpp:60-68 */
  if (n == "mat25") return new covf_mat25();
  if (n == "mat25pow") return new covf_mat25pow();
  if (n == "mat25ang") return new covf_mat25ang();
  throw std::range_error("need to choose one of the existing cov functions");
}
int ref_covf_numhyp(const char* name, uint64_t* n) { REF_TRY std::unique_ptr<covf> c(make_covf(name)); *n = c->numhyp; REF_CATCH }
int ref_covf_cov(ref_ctx*, const char* name, const double* hyp, const double* x1, uint64_t n1, const double* x2, uint64_t n2, double* out) {
  REF_TRY
  std::unique_ptr<covf> c(make_covf(name));
  for (unsigned i = 0; i < c->numhyp; ++i) c->hyp[i] = hyp[i];
  put(c->cov(to_vec(x1, n1), to_vec(x2, n2)), out);
  REF_CATCH
}
int ref_covf_cov_gradhyp(ref_ctx*, const char* name, const double* hyp, const double* x1, uint64_t n1, const double* x2, uint64_t n2, double* out) {
  REF_TRY
  std::unique_ptr<covf> c(make_covf(name));
  for (unsigned i = 0; i < c->numhyp; ++i) c->hyp[i] = hyp[i];
  cube g = c->cov_gradhyp(to_vec(x1, n1), to_vec(x2, n2));
  std::copy(g.store.begin(), g.store.end(), out);
  REF_CATCH
}

/* ---- outermod ---- */
int ref_outermod_create(ref_outermod** out) { *out = new ref_outermod(); return REF_OK; }
int ref_outermod_destroy(ref_outermod* om) { delete om; return REF_OK; }
int ref_outermod_setcovfs(ref_outermod* h, uint64_t d, const char* const* names) { /* setcovfs, interfaceR.cpp:53-73 */
  REF_TRY
  outermod& om = h->om;
  std::vector<covf*> list;
  for (uint64_t k = 0; k < d; ++k) list.push_back(make_covf(names[k]));
  om.d = d;
  om.covflist = list;
  om.hyp_init();
  om.setcovfs = true;
  om.setknots = false;
  REF_CATCH
}
int ref_outermod_setknot(ref_outermod* h, const double* knots, const uint64_t* lens) { /* setknot, interfaceR.cpp:94-149 */
  REF_TRY
  outermod& om = h->om;
  if (!om.setcovfs) throw std::range_error("Need to set cov. funcs before setting knots.");
  std::vector<vec> L;
  const double* p = knots;
  for (uword l = 0; l < om.d; ++l) { L.push_back(to_vec(p, lens[l])); p += lens[l]; }
  for (unsigned int l = 0; l < om.d; ++l)
    if (!(*om.covflist[l]).inputcheck(L[l]))
      throw std::range_error(std::to_string(l + 1) + "knot point needs to be between " + std::to_string((*om.covflist[l]).lowbnd) + " and " +
                             std::to_string((*om.covflist[l]).uppbnd));
  om.knotptst.resize(om.d + 1);
  int currst = 0;
  for (unsigned int l = 0; l < om.d; ++l) { om.knotptst[l] = currst; currst += L[l].n_elem; }
  om.knotptst[om.d] = currst;
  om.knotpt.resize(currst);
  for (unsigned int l = 0; l < om.d; ++l) om.knotpt.subvec(om.knotptst[l], om.knotptst[l + 1] - 1) = L[l];
  om.setknots = true;
  om.knotptstge.resize(om.d + 1);
  om.gest.resize(om.hypst[om.d] + 1);
  currst = 0;
  int currstalt = 0;
  for (unsigned int l = 0; l < om.d; ++l) {
    om.knotptstge[l] = currst;
    for (unsigned int k = 0; k < (om.hypst[l + 1] - om.hypst[l]); ++k) {
      om.hypmatch[currstalt] = l;
      om.gest[currstalt] = currst;
      currst += om.knotptst[l + 1] - om.knotptst[l];
      currstalt += 1;
    }
  }
  om.knotptstge[om.d] = currst;
  om.gest[om.hypst[om.d]] = currst;
  om.build();
  REF_CATCH
}
int ref_outermod_updatehyp(ref_outermod* h, const double* hyp, uint64_t n) { REF_TRY h->om.hyp_set(to_vec(hyp, n)); REF_CATCH }
int ref_outermod_gethyp(ref_outermod* h, double* hyp) { put(h->om.hyp, hyp); return REF_OK; }
int ref_outermod_sizes(ref_outermod* h, uint64_t* d, uint64_t* nhyp, uint64_t* nknot, uint64_t* nge) {
  const outermod& om = h->om;
  *d = om.d; *nhyp = om.hyp.n_elem; *nknot = om.knotpt.n_elem; *nge = om.knotptstge.n_elem ? om.knotptstge[om.d] : 0;
  return REF_OK;
}
int ref_outermod_set_select_seed(ref_outermod* h, uint64_t seed) { h->select_seed = seed; return REF_OK; }
int ref_outermod_selectterms(ref_outermod* h, uint64_t numele, uint64_t* terms) {
  REF_TRY
  if (h->select_seed) {
    g_rng = h->select_seed;
    arma_shim_shuffle() = [](uword* perm, uword n) { if (n) std::swap(perm[0], perm[splitmix64(g_rng) % n]); };
  } else arma_shim_shuffle() = nullptr;
  umat t = h->om.selectterms((unsigned)numele);
  arma_shim_shuffle() = nullptr;
  std::memcpy(terms, t.mem, t.n_elem * sizeof(uint64_t));
  REF_CATCH
}
int ref_outermod_getvar(ref_outermod* h, const uint64_t* terms, uint64_t K, double* out) { REF_TRY put(h->om.getvar(to_umat(terms, K, h->om.d)), out); REF_CATCH }
int ref_outermod_getlvar_gradhyp(ref_outermod* h, const uint64_t* terms, uint64_t K, double* out) {
  REF_TRY put(h->om.getlvar_gradhyp(to_umat(terms, K, h->om.d)), out); REF_CATCH
}
int ref_outermod_hyplpdf(ref_outermod* h, const double* hyp, uint64_t n, double* out) { REF_TRY *out = h->om.hyplpdf(to_vec(hyp, n)); REF_CATCH }
int ref_outermod_hyplpdf_grad(ref_outermod* h, const double* hyp, uint64_t n, double* out) { REF_TRY put(h->om.hyplpdf_grad(to_vec(hyp, n)), out); REF_CATCH }
int ref_outermod_get_index(ref_outermod* h, const char* which, int64_t* out, uint64_t* n) {
  REF_TRY
  const std::string w = which;
  const outermod& m = h->om;
  std::vector<int64_t> v;
  auto cp = [&](const uvec& s) { v.assign(s.mem, s.mem + s.n_elem); };
  if (w == "knotptst") cp(m.knotptst);
  else if (w == "hypst") cp(m.hypst);
  else if (w == "hypmatch") cp(m.hypmatch);
  else if (w == "gest") cp(m.gest);
  else if (w == "knotptstge") cp(m.knotptstge);
  else if (w == "maxlevel") v.assign(m.maxlevel.mem, m.maxlevel.mem + m.maxlevel.n_elem);
  else throw std::invalid_argument("unknown index table " + w);
  *n = v.size();
  if (out) std::copy(v.begin(), v.end(), out);
  REF_CATCH
}
int ref_outermod_get_real(ref_outermod* h, const char* which, double* out, uint64_t* nrow, uint64_t* ncol) {
  REF_TRY
  const std::string w = which;
  const outermod& m = h->om;
  const mat* src = nullptr;
  if (w == "basisvar") src = &m.basisvar;
  else if (w == "knotpt") src = &m.knotpt;
  else if (w == "logbasisvar_gradhyp") src = &m.logbasisvar_gradhyp;
  else if (w == "rotmat") src = &m.rotmat;
  else if (w == "rotmat_gradhyp") src = &m.rotmat_gradhyp;
  else throw std::invalid_argument("unknown real table " + w);
  *nrow = src->n_rows; *ncol = src->n_cols;
  if (out) put(*src, out);
  REF_CATCH
}

/* ---- outerbase ---- */
int ref_outerbase_create(ref_ctx*, ref_outermod* om, const double* x, uint64_t N, int dograd, ref_outerbase** out) {
  REF_TRY
  if (!om->om.setknots) throw std::range_error("Need to set covfs and knots before building.");
  auto* h = new ref_outerbase();
  h->ob.reset(new outerbase(om->om, to_mat(x, N, om->om.d), dograd != 0));
  *out = h;
  REF_CATCH
}
int ref_outerbase_destroy(ref_outerbase* ob) { delete ob; return REF_OK; }
int ref_outerbase_build(ref_outerbase* ob) { REF_TRY ob->ob->build(); REF_CATCH }
int ref_outerbase_set_nthreads(ref_outerbase* ob, int n) { ob->ob->nthreads = n; return REF_OK; }
int ref_outerbase_loopvals(ref_outerbase* ob, uint64_t* nthreads, uint64_t* chunksize, uint64_t* loopsize, int* vertpl) {
  *nthreads = ob->ob->nthreads; *chunksize = ob->ob->chunksize; *loopsize = ob->ob->loopsize; *vertpl = ob->ob->vertpl;
  return REF_OK;
}
int ref_outerbase_get_real(ref_outerbase* ob, const char* which, double* out, uint64_t* nrow, uint64_t* ncol) {
  REF_TRY
  const std::string w = which;
  const outerbase& b = *ob->ob;
  const mat* src = nullptr;
  if (w == "basemat") src = &b.basemat;
  else if (w == "basemat_gradhyp") src = &b.basemat_gradhyp;
  else if (w == "basescale") src = &b.basescale;
  else if (w == "basescalemat") src = &b.basescalemat;
  else throw std::invalid_argument("unknown matrix " + w);
  *nrow = src->n_rows; *ncol = src->n_cols;
  if (out) put(*src, out);
  REF_CATCH
}
int ref_outerbase_getbase(ref_outerbase* ob, uint64_t dim, double* out) {
  REF_TRY
  if (dim < 1 || dim > ob->ob->d) throw std::range_error("dim out of range");
  put(ob->ob->getbase(dim), out);
  REF_CATCH
}
int ref_outerbase_getmat_gradhyp(ref_outerbase* ob, const uint64_t* terms, uint64_t K, double* out) {
  REF_TRY
  cube g = ob->ob->getmat_gradhyp(to_umat(terms, K, ob->ob->d));
  std::copy(g.store.begin(), g.store.end(), out);
  REF_CATCH
}
int ref_outerbase_getmat(ref_outerbase* ob, const uint64_t* terms, uint64_t K, double* out) { REF_TRY put(ob->ob->getmat(to_umat(terms, K, ob->ob->d)), out); REF_CATCH }
static void mm_impl(const outerbase& ob, int sq, const umat& t, const double* a, double* out) {
  vec o;
  if (sq) o = ob.sqmm(t, to_vec(a, t.n_rows)); else ob.mm(o, t, to_vec(a, t.n_rows));
  put(o, out);
}
static void tmm_impl(const outerbase& ob, int sq, const umat& t, const double* a, double* out) {
  vec o;
  if (sq) o = ob.sqtmm(t, to_vec(a, ob.n_row)); else ob.tmm(o, t, to_vec(a, ob.n_row));
  put(o, out);
}
int ref_outerbase_mm(ref_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* a, double* out) {
  REF_TRY mm_impl(*ob->ob, sq, to_umat(terms, K, ob->ob->d), a, out); REF_CATCH
}
int ref_outerbase_tmm(ref_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* a, double* out) {
  REF_TRY tmm_impl(*ob->ob, sq, to_umat(terms, K, ob->ob->d), a, out); REF_CATCH
}
int ref_outerbase_mm_gradhyp(ref_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* a, double* out, double* outge) {
  REF_TRY
  const outerbase& b = *ob->ob;
  umat t = to_umat(terms, K, b.d);
  vec o; mat g;
  if (sq) prodmmge_(o, g, t, to_vec(a, K), b.basematsq, b.basescalesq, b.knotptst, b.basematsq_gradhyp, b.gest, b.hypmatch, b.vertpl, b.chunksize, b.loopsize, b.nthreads);
  else b.mm_gradhyp(o, g, t, to_vec(a, K));
  if (out) put(o, out);
  put(g, outge);
  REF_CATCH
}
int ref_outerbase_tmm_gradhyp(ref_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* a, double* out, double* outge) {
  REF_TRY
  const outerbase& b = *ob->ob;
  umat t = to_umat(terms, K, b.d);
  vec o; mat g;
  if (sq) tprodmmge_(o, g, t, to_vec(a, b.n_row), b.basematsq, b.basescalesq, b.knotptst, b.basematsq_gradhyp, b.gest, b.hypmatch, b.vertpl, b.chunksize, b.loopsize, b.nthreads);
  else b.tmm_gradhyp(o, g, t, to_vec(a, b.n_row));
  if (out) put(o, out);
  put(g, outge);
  REF_CATCH
}
int ref_outerbase_mm_mat(ref_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* A, uint64_t C, double* out) {
  REF_TRY
  const outerbase& b = *ob->ob;
  mat o;
  prodmm_(o, to_umat(terms, K, b.d), to_mat(A, K, C), sq ? b.basematsq : b.basemat, sq ? b.basescalesq : b.basescale, b.knotptst, b.vertpl, b.chunksize, b.loopsize, b.nthreads);
  put(o, out);
  REF_CATCH
}
int ref_outerbase_tmm_mat(ref_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* A, uint64_t C, double* out) {
  REF_TRY
  const outerbase& b = *ob->ob;
  mat o;
  tprodmm_(o, to_umat(terms, K, b.d), to_mat(A, b.n_row, C), sq ? b.basematsq : b.basemat, sq ? b.basescalesq : b.basescale, b.knotptst, b.vertpl, b.chunksize, b.loopsize, b.nthreads);
  put(o, out);
  REF_CATCH
}
int ref_outerbase_residvar(ref_outerbase* ob, const uint64_t* terms, uint64_t K, double* out) { REF_TRY put(ob->ob->residvar(to_umat(terms, K, ob->ob->d)), out); REF_CATCH }
int ref_outerbase_residvar_gradhyp(ref_outerbase* ob, const uint64_t* terms, uint64_t K, double* out) {
  REF_TRY put(ob->ob->residvar_gradhyp(to_umat(terms, K, ob->ob->d)), out); REF_CATCH
}
int ref_outerbase_set_terms(ref_outerbase* ob, const uint64_t* terms, uint64_t K) { REF_TRY ob->terms = to_umat(terms, K, ob->ob->d); REF_CATCH }
int ref_outerbase_mm_dev(ref_outerbase* ob, int sq, const double* a, double* out) { REF_TRY mm_impl(*ob->ob, sq, ob->terms, a, out); REF_CATCH }
int ref_outerbase_tmm_dev(ref_outerbase* ob, int sq, const double* a, double* out) { REF_TRY tmm_impl(*ob->ob, sq, ob->terms, a, out); REF_CATCH }
int ref_outerbase_mm_mat_dev(ref_outerbase* ob, int sq, const double* A, uint64_t C, double* out) {
  return ref_outerbase_mm_mat(ob, sq, reinterpret_cast<const uint64_t*>(ob->terms.mem), ob->terms.n_rows, A, C, out);
}
int ref_outerbase_tmm_mat_dev(ref_outerbase* ob, int sq, const double* A, uint64_t C, double* out) {
  return ref_outerbase_tmm_mat(ob, sq, reinterpret_cast<const uint64_t*>(ob->terms.mem), ob->terms.n_rows, A, C, out);
}
int ref_outerbase_terms_stats(ref_outerbase* ob, uint64_t* W, uint64_t* Lcols, uint64_t* nodes, uint64_t* maxdepth) {
  REF_TRY
  const umat& t = ob->terms;
  uint64_t w = 0, lc = 0, md = 0;
  for (uword l = 0; l < t.n_cols; ++l) { uint64_t mx = 0; for (uword k = 0; k < t.n_rows; ++k) mx = std::max<uint64_t>(mx, t.at(k, l)); lc += mx; }
  for (uword k = 0; k < t.n_rows; ++k) { uint64_t nz = 0; for (uword l = 0; l < t.n_cols; ++l) nz += t.at(k, l) > 0; w += nz + 1; md = std::max(md, nz); }
  *W = w; *Lcols = lc; *nodes = t.n_rows; *maxdepth = md;
  REF_CATCH
}

/* ---- stateless linalg.h seam: the reference's free functions themselves (src/linalg.h:9-58) ---- */
static uvec to_uvec(const uint64_t* p, uint64_t n) { return uvec(reinterpret_cast<const uword*>(p), n); }
int ref_prodmm_vec(ref_ctx*, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* a, const double* basemat, uint64_t N, uint64_t M,
                   const double* basescale, const uint64_t* knotptst) {
  REF_TRY
  const loopvals lv = default_lv(N);
  vec o;
  prodmm_(o, to_umat(terms, K, d), to_vec(a, K), to_mat(basemat, N, M), to_vec(basescale, N), to_uvec(knotptst, d + 1), lv.vertpl, lv.chunksize, lv.loopsize, lv.nthreads);
  put(o, out);
  REF_CATCH
}
int ref_tprodmm_vec(ref_ctx*, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* a, const double* basemat, uint64_t N, uint64_t M,
                    const double* basescale, const uint64_t* knotptst) {
  REF_TRY
  const loopvals lv = default_lv(N);
  vec o;
  tprodmm_(o, to_umat(terms, K, d), to_vec(a, N), to_mat(basemat, N, M), to_vec(basescale, N), to_uvec(knotptst, d + 1), lv.vertpl, lv.chunksize, lv.loopsize, lv.nthreads);
  put(o, out);
  REF_CATCH
}
int ref_prodmm_mat(ref_ctx*, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* A, uint64_t C, const double* basemat, uint64_t N, uint64_t M,
                   const double* basescale, const uint64_t* knotptst) {
  REF_TRY
  const loopvals lv = default_lv(N);
  mat o;
  prodmm_(o, to_umat(terms, K, d), to_mat(A, K, C), to_mat(basemat, N, M), to_vec(basescale, N), to_uvec(knotptst, d + 1), lv.vertpl, lv.chunksize, lv.loopsize, lv.nthreads);
  put(o, out);
  REF_CATCH
}
int ref_tprodmm_mat(ref_ctx*, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* A, uint64_t C, const double* basemat, uint64_t N, uint64_t M,
                    const double* basescale, const uint64_t* knotptst) {
  REF_TRY
  const loopvals lv = default_lv(N);
  mat o;
  tprodmm_(o, to_umat(terms, K, d), to_mat(A, N, C), to_mat(basemat, N, M), to_vec(basescale, N), to_uvec(knotptst, d + 1), lv.vertpl, lv.chunksize, lv.loopsize, lv.nthreads);
  put(o, out);
  REF_CATCH
}
int ref_prodmmge(ref_ctx*, double* out, double* outge, const uint64_t* terms, uint64_t K, uint64_t d, const double* a, const double* basemat, uint64_t N, uint64_t M,
                 const double* basescale, const uint64_t* knotptst, const double* basematge, uint64_t Mge, const uint64_t* gest, const uint64_t* hypmatch, uint64_t H) {
  REF_TRY
  const loopvals lv = default_lv(N);
  vec o; mat g;
  prodmmge_(o, g, to_umat(terms, K, d), to_vec(a, K), to_mat(basemat, N, M), to_vec(basescale, N), to_uvec(knotptst, d + 1), to_mat(basematge, N, Mge),
            to_uvec(gest, H + 1), to_uvec(hypmatch, H), lv.vertpl, lv.chunksize, lv.loopsize, lv.nthreads);
  put(o, out); put(g, outge);
  REF_CATCH
}
int ref_tprodmmge(ref_ctx*, double* out, double* outge, const uint64_t* terms, uint64_t K, uint64_t d, const double* a, const double* basemat, uint64_t N, uint64_t M,
                  const double* basescale, const uint64_t* knotptst, const double* basematge, uint64_t Mge, const uint64_t* gest, const uint64_t* hypmatch, uint64_t H) {
  REF_TRY
  const loopvals lv = default_lv(N);
  vec o; mat g;
  tprodmmge_(o, g, to_umat(terms, K, d), to_vec(a, N), to_mat(basemat, N, M), to_vec(basescale, N), to_uvec(knotptst, d + 1), to_mat(basematge, N, Mge),
             to_uvec(gest, H + 1), to_uvec(hypmatch, H), lv.vertpl, lv.chunksize, lv.loopsize, lv.nthreads);
  put(o, out); put(g, outge);
  REF_CATCH
}
int ref_getmge(ref_ctx*, double* outge, const uint64_t* terms, uint64_t K, uint64_t d, const double* basemat, uint64_t N, uint64_t M, const double* basescale,
               const uint64_t* knotptst, const double* basematge, uint64_t Mge, const uint64_t* gest, const uint64_t* hypmatch, uint64_t H) {
  REF_TRY
  const loopvals lv = default_lv(N);
  cube g;
  /* the reference's function as it is; callers keep to unchunked shapes (its chunked branch cannot work, linalg.cpp:788-810) */
  getmge_(g, to_umat(terms, K, d), to_mat(basemat, N, M), to_vec(basescale, N), to_uvec(knotptst, d + 1), to_mat(basematge, N, Mge), to_uvec(gest, H + 1),
          to_uvec(hypmatch, H), lv.vertpl, lv.chunksize, lv.loopsize, lv.nthreads);
  std::copy(g.store.begin(), g.store.end(), outge);
  REF_CATCH
}
int ref_getm(ref_ctx*, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* basemat, uint64_t N, uint64_t M, const double* basescale,
             const uint64_t* knotptst) {
  REF_TRY
  const loopvals lv = default_lv(N);
  mat o;
  getm_(o, to_umat(terms, K, d), to_mat(basemat, N, M), to_vec(basescale, N), to_uvec(knotptst, d + 1), lv.vertpl, lv.chunksize, lv.loopsize, lv.nthreads);
  put(o, out);
  REF_CATCH
}

/* ---- lpdf family ---- */
int ref_loglik_gauss_create(ref_ctx*, ref_outermod* om, const uint64_t* terms, uint64_t K, const double* y, const double* x, uint64_t N, ref_lpdf** out) {
  REF_TRY
  auto* h = new ref_lpdf();
  auto* p = new counting<loglik_gauss>(om->om, to_umat(terms, K, om->om.d), to_vec(y, N), to_mat(x, N, om->om.d));
  h->p.reset(p); h->hm = &p->hm_calls; h->kind = 0; h->nhyp = om->om.hyp.n_elem; h->nrow = N; h->d = om->om.d;
  *out = h;
  REF_CATCH
}
int ref_loglik_std_create(ref_ctx*, ref_outermod* om, const uint64_t* terms, uint64_t K, const double* y, const double* x, uint64_t N, ref_lpdf** out) {
  REF_TRY
  auto* h = new ref_lpdf();
  auto* p = new counting<loglik_std>(om->om, to_umat(terms, K, om->om.d), to_vec(y, N), to_mat(x, N, om->om.d));
  h->p.reset(p); h->hm = &p->hm_calls; h->kind = 4; h->nhyp = om->om.hyp.n_elem; h->nrow = N; h->d = om->om.d;
  *out = h;
  REF_CATCH
}
int ref_loglik_gda_create(ref_ctx*, ref_outermod* om, const uint64_t* terms, uint64_t K, const double* y, const double* x, uint64_t N, ref_lpdf** out) {
  REF_TRY
  auto* h = new ref_lpdf();
  auto* p = new counting<loglik_gda>(om->om, to_umat(terms, K, om->om.d), to_vec(y, N), to_mat(x, N, om->om.d));
  h->p.reset(p); h->hm = &p->hm_calls; h->kind = 3; h->nhyp = om->om.hyp.n_elem; h->nrow = N; h->d = om->om.d;
  *out = h;
  REF_CATCH
}
int ref_logpr_gauss_create(ref_ctx*, ref_outermod* om, const uint64_t* terms, uint64_t K, ref_lpdf** out) {
  REF_TRY
  auto* h = new ref_lpdf();
  auto* p = new counting<logpr_gauss>(om->om, to_umat(terms, K, om->om.d));
  h->p.reset(p); h->hm = &p->hm_calls; h->kind = 1; h->nhyp = om->om.hyp.n_elem; h->nrow = 0; h->d = om->om.d;
  *out = h;
  REF_CATCH
}
int ref_lpdfvec_create(ref_lpdf* a, ref_lpdf* b, ref_lpdf** out) {
  REF_TRY
  auto* h = new ref_lpdf();
  auto* p = new counting<lpdfvec>(*a->p, *b->p);
  h->p.reset(p); h->hm = &p->hm_calls; h->kind = 2; h->nhyp = a->nhyp; h->nrow = std::max(a->nrow, b->nrow); h->d = a->d; h->a = a; h->b = b;
  *out = h;
  REF_CATCH
}
int ref_lpdf_destroy(ref_lpdf* l) { delete l; return REF_OK; }
int ref_lpdf_setnthreads(ref_lpdf* l, int k) { l->p->setnthreads(k); return REF_OK; }
int ref_lpdf_update(ref_lpdf* l, const double* coeff, uint64_t K) { REF_TRY l->p->update(to_vec(coeff, K)); REF_CATCH }
int ref_lpdf_updateom(ref_lpdf* l) { REF_TRY l->p->updateom(); REF_CATCH }
int ref_lpdf_updatepara(ref_lpdf* l, const double* para, uint64_t n) { REF_TRY l->p->updatepara(to_vec(para, n)); REF_CATCH }
int ref_lpdf_updateterms(ref_lpdf* l, const uint64_t* terms, uint64_t K) { REF_TRY l->p->updateterms(to_umat(terms, K, l->d)); REF_CATCH }
int ref_lpdf_optcg(ref_lpdf* l, double tol, uint64_t maxepch) {
  REF_TRY
  *l->hm = 0;
  l->p->optcg(tol, (unsigned)maxepch);
  l->cg_iters = *l->hm ? *l->hm - 1 : 0;
  REF_CATCH
}
int ref_lpdf_optnewton(ref_lpdf* l) { REF_TRY l->p->optnewton(); REF_CATCH }
static void put_cube(const cube& c, double* out, uint64_t* n) { *n = c.n_elem; std::copy(c.store.begin(), c.store.end(), out); }
int ref_lpdf_hess(ref_lpdf* l, double* out, uint64_t* n) { REF_TRY mat h = l->p->hess(); *n = h.n_elem; put(h, out); REF_CATCH }
int ref_lpdf_hessgradhyp(ref_lpdf* l, double* out, uint64_t* n) { REF_TRY put_cube(l->p->hessgradhyp(), out, n); REF_CATCH }
int ref_lpdf_hessgradpara(ref_lpdf* l, double* out, uint64_t* n) { REF_TRY put_cube(l->p->hessgradpara(), out, n); REF_CATCH }
int ref_lpdf_hessmult(ref_lpdf* l, const double* g, double* out) { REF_TRY put(l->p->hessmult(to_vec(g, l->p->nterms)), out); REF_CATCH }
int ref_lpdf_diaghess(ref_lpdf* l, double* out) { REF_TRY put(l->p->diaghess(), out); REF_CATCH }
int ref_lpdf_diaghessgradhyp(ref_lpdf* l, double* out) { REF_TRY put(l->p->diaghessgradhyp(), out); REF_CATCH }
int ref_lpdf_diaghessgradpara(ref_lpdf* l, double* out) { REF_TRY put(l->p->diaghessgradpara(), out); REF_CATCH }
int ref_lpdf_paralpdf(ref_lpdf* l, const double* para, uint64_t n, double* out) { REF_TRY *out = l->p->paralpdf(to_vec(para, n)); REF_CATCH }
int ref_lpdf_paralpdf_grad(ref_lpdf* l, const double* para, uint64_t n, double* out) { REF_TRY put(l->p->paralpdf_grad(to_vec(para, n)), out); REF_CATCH }
int ref_lpdf_set_flag(ref_lpdf* l, const char* which, int value) {
  REF_TRY
  const std::string w = which;
  if (w == "compute_val") l->p->compute_val = value;
  else if (w == "compute_grad") l->p->compute_grad = value;
  else if (w == "compute_gradhyp") l->p->compute_gradhyp = value;
  else if (w == "compute_gradpara") l->p->compute_gradpara = value;
  else if (w == "fullhess") l->p->fullhess = value;
  else if (w == "domarg") {
    auto* v = dynamic_cast<lpdfvec*>(l->p.get());
    if (!v) throw std::invalid_argument("domarg is a field of lpdfvec");
    v->domargadj = value;
  } else if (w == "dodiag") { /* R field name of loglik_gda::doda, interfaceR.cpp:748 */
    auto* v = dynamic_cast<loglik_gda*>(l->p.get());
    if (!v) throw std::invalid_argument("dodiag is a field of loglik_gda");
    v->doda = value; v->redostd = true;
  } else throw std::invalid_argument("unknown flag " + w);
  REF_CATCH
}
int ref_lpdf_sizes(ref_lpdf* l, uint64_t* nterms, uint64_t* npara, uint64_t* nhyp, uint64_t* nrow) {
  *nterms = l->p->nterms; *npara = l->p->para.n_elem; *nhyp = l->nhyp; *nrow = l->nrow;
  return REF_OK;
}
int ref_lpdf_get(ref_lpdf* l, const char* which, double* out, uint64_t* n) {
  REF_TRY
  const std::string w = which;
  vec v;
  if (w == "val") v = vec({l->p->val});
  else if (w == "grad") v = l->p->grad;
  else if (w == "gradhyp") v = l->p->gradhyp;
  else if (w == "gradpara") v = l->p->gradpara;
  else if (w == "coeff") v = l->p->coeff;
  else if (w == "para") v = l->p->para;
  else if (w == "totdiaghess") v = l->p->totdiaghess;
  else if (w == "tothess") { const mat& th = l->p->tothess; v.set_size(th.n_elem); std::copy(th.mem, th.mem + th.n_elem, v.mem); }
  else if (w == "cg_iters") v = vec({double(l->cg_iters)});
  else if (w == "yhat") {
    if (auto* g = dynamic_cast<loglik_gauss*>(l->p.get())) v = g->yhat;
    else if (auto* g2 = dynamic_cast<loglik_gda*>(l->p.get())) v = g2->yhat;
    else if (auto* g3 = dynamic_cast<loglik_std*>(l->p.get())) v = g3->yhat;
    else throw std::invalid_argument("yhat is a field of loglik_gauss / loglik_gda / loglik_std");
  } else if (w == "coeffsd") {
    auto* g = dynamic_cast<logpr_gauss*>(l->p.get());
    if (!g) throw std::invalid_argument("coeffsd is a field of logpr_gauss");
    v = g->coeffsd;
  } else throw std::invalid_argument("unknown field " + w);
  *n = v.n_elem;
  if (out) put(v, out);
  REF_CATCH
}
int ref_lpdf_set_coeff(ref_lpdf* l, const double* coeff, uint64_t K) { REF_TRY l->p->coeff = to_vec(coeff, K); REF_CATCH }

int ref_predictor_create(ref_lpdf* loglik, ref_predictor** out) {
  REF_TRY
  auto* h = new ref_predictor();
  h->p.reset(new predictor(*loglik->p)); /* lpdf::pred() throws std::invalid_argument for objects without one, fit.h:52-55 */
  h->d = loglik->d;
  *out = h;
  REF_CATCH
}
int ref_predictor_destroy(ref_predictor* p) { delete p; return REF_OK; }
int ref_predictor_update(ref_predictor* p, const double* x, uint64_t N) { REF_TRY p->p->update(to_mat(x, N, p->d)); REF_CATCH }
int ref_predictor_mean(ref_predictor* p, double* out) { REF_TRY put(p->p->mean(), out); REF_CATCH }
int ref_predictor_var(ref_predictor* p, double* out) { REF_TRY put(p->p->var(), out); REF_CATCH }

} // extern "C"
