/*
 * ob_capi.cu -- extern "C" layer of include/outerbase_b200.h over ob_engine.hpp.
 * Exceptions of the C++ core become status codes + ob_last_error(); nothing in here
 * computes: host model calls go to ob_model.hpp, everything N-sized to the CUDA kernels.
 */
#include "../../include/outerbase_b200.h"
#include "../../include/outerbase_b200_multi.h"
#include "../../include/outerbase_b200_multi_percol.h"
#include "../../include/outerbase_b200_multi_gda.h"

#include "ob_engine.hpp"

using obe::u64;

static thread_local std::string g_err;

#define OB_TRY try {
#define OB_CATCH                                                                          \
  }                                                                                       \
  catch (const obd::NoGpuError& e) { g_err = e.what(); return OB_ERR_NOGPU; }             \
  catch (const obd::CudaError& e) { g_err = e.what(); return OB_ERR_CUDA; }               \
  catch (const obd::NcclError& e) { g_err = e.what(); return OB_ERR_NCCL; }               \
  catch (const std::range_error& e) { g_err = e.what(); return OB_ERR_INVALID; }          \
  catch (const std::invalid_argument& e) { g_err = e.what(); return OB_ERR_INVALID; }     \
  catch (const std::exception& e) { g_err = e.what(); return OB_ERR_STATE; }              \
  return OB_OK;

struct ob_ctx { obd::Ctx c; explicit ob_ctx(int dev) : c(dev) {} };
struct ob_outermod { obh::OuterMod om; };
struct ob_outerbase { ob_ctx* ctx; std::unique_ptr<obe::OuterBase> ob; };
struct ob_lpdf { ob_ctx* ctx; std::unique_ptr<obe::Lpdf> p; };
struct ob_predictor { std::unique_ptr<obe::Pred> p; };

static void need(const void* p, const char* what) { if (!p) throw std::invalid_argument(std::string("null ") + what); }

extern "C" {

const char* ob_last_error(void) { return g_err.c_str(); }
int ob_version(void) { return 1; }

/* ---- context */
int ob_ctx_create(int device, ob_ctx** out) { OB_TRY need(out, "out"); *out = new ob_ctx(device); OB_CATCH }
int ob_ctx_destroy(ob_ctx* ctx) { OB_TRY delete ctx; OB_CATCH }
int ob_ctx_synchronize(ob_ctx* ctx) { OB_TRY need(ctx, "ctx"); ctx->c.sync(); OB_CATCH }
int ob_ctx_stream(ob_ctx* ctx, void** s) { OB_TRY need(ctx, "ctx"); *s = (void*)ctx->c.stream; OB_CATCH }
int ob_comm_get_unique_id(void* id128) {
  OB_TRY
  obd::NcclApi& api = obd::NcclApi::get();
  if (!api.GetUniqueId) throw obd::NcclError("libnccl.so.2 not found");
  obd::NcclUid uid;
  const int rc = api.GetUniqueId(&uid);
  if (rc != 0) throw obd::NcclError(std::string("ncclGetUniqueId: ") + api.GetErrorString(rc));
  std::memcpy(id128, uid.b, 128);
  OB_CATCH
}
int ob_ctx_comm_init(ob_ctx* ctx, int nranks, int rank, const void* id128) {
  OB_TRY
  need(ctx, "ctx");
  obd::NcclApi& api = obd::NcclApi::get();
  if (!api.CommInitRank) throw obd::NcclError("libnccl.so.2 not found");
  if (ctx->c.comm) throw std::logic_error("communicator already initialised");
  OB_CUDA(cudaSetDevice(ctx->c.device));
  obd::NcclUid uid;
  std::memcpy(uid.b, id128, 128);
  void* comm = nullptr;
  const int rc = api.CommInitRank(&comm, nranks, uid, rank);
  if (rc != 0) throw obd::NcclError(std::string("ncclCommInitRank: ") + api.GetErrorString(rc));
  ctx->c.comm = comm; ctx->c.nranks = nranks; ctx->c.rank = rank;
  ctx->c.p2p_init();
  OB_CATCH
}
int ob_ctx_comm_info(ob_ctx* ctx, int* nranks, int* rank) { OB_TRY need(ctx, "ctx"); *nranks = ctx->c.nranks; *rank = ctx->c.rank; OB_CATCH }
int ob_ctx_allreduce_dev(ob_ctx* ctx, double* buf_dev, uint64_t n) {
  OB_TRY need(ctx, "ctx"); if (n) need(buf_dev, "buf_dev"); ctx->c.allreduce_sum(buf_dev, n); OB_CATCH
}
int ob_ctx_fp64_peak(ob_ctx* ctx, double* tflops) { OB_TRY need(ctx, "ctx"); *tflops = obd::measure_fp64_peak(ctx->c); OB_CATCH }
int ob_ctx_launch_count(ob_ctx* ctx, uint64_t* count) { OB_TRY need(ctx, "ctx"); *count = ctx->c.launches; OB_CATCH }

/* ---- covf */
int ob_covf_numhyp(const char* name, uint64_t* n) { OB_TRY *n = (uint64_t)obh::cov_spec(name).numhyp; OB_CATCH }
static void cov_impl(ob_ctx* ctx, const char* name, const double* hyp, const double* x1, u64 n1, const double* x2, u64 n2,
                     double* out, bool grad) {
  need(ctx, "ctx");
  const obh::CovSpec sp = obh::cov_spec(name);
  obd::Ctx& c = ctx->c;
  obd::DevBuf<double> a, b, o, g;
  a.upload(x1, n1, c.stream); b.upload(x2, n2, c.stream);
  o.ensure(n1 * n2);
  if (grad) g.ensure(n1 * n2 * sp.numhyp);
  double h[2] = {hyp[0], sp.numhyp > 1 ? hyp[1] : 0.0};
  obd::launch_cov(c, sp.kind, h, a.p, n1, b.p, n2, o.p, grad ? g.p : nullptr);
  const obd::DevBuf<double>& src = grad ? g : o;
  const u64 n = grad ? n1 * n2 * sp.numhyp : n1 * n2;
  if (n) OB_CUDA(cudaMemcpyAsync(out, src.p, n * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
  c.sync();
}
int ob_covf_cov(ob_ctx* ctx, const char* name, const double* hyp, const double* x1, uint64_t n1, const double* x2,
                uint64_t n2, double* out) { OB_TRY cov_impl(ctx, name, hyp, x1, n1, x2, n2, out, false); OB_CATCH }
int ob_covf_cov_gradhyp(ob_ctx* ctx, const char* name, const double* hyp, const double* x1, uint64_t n1, const double* x2,
                        uint64_t n2, double* out) { OB_TRY cov_impl(ctx, name, hyp, x1, n1, x2, n2, out, true); OB_CATCH }

/* ---- outermod */
int ob_outermod_create(ob_outermod** out) { OB_TRY *out = new ob_outermod(); OB_CATCH }
int ob_outermod_destroy(ob_outermod* om) { OB_TRY delete om; OB_CATCH }
int ob_outermod_setcovfs(ob_outermod* om, uint64_t d, const char* const* names) {
  OB_TRY
  std::vector<std::string> v;
  for (u64 i = 0; i < d; ++i) v.push_back(names[i]);
  om->om.set_covfs(v);
  OB_CATCH
}
int ob_outermod_setknot(ob_outermod* om, const double* knots, const uint64_t* lens) { OB_TRY om->om.set_knot(knots, lens); OB_CATCH }
int ob_outermod_updatehyp(ob_outermod* om, const double* hyp, uint64_t n) { OB_TRY om->om.hyp_set(hyp, n); OB_CATCH }
int ob_outermod_gethyp(ob_outermod* om, double* hyp) { OB_TRY std::copy(om->om.hyp.begin(), om->om.hyp.end(), hyp); OB_CATCH }
int ob_outermod_sizes(ob_outermod* om, uint64_t* d, uint64_t* nhyp, uint64_t* nknot, uint64_t* nge) {
  OB_TRY *d = om->om.d; *nhyp = om->om.nhyp(); *nknot = om->om.nknot(); *nge = om->om.nge(); OB_CATCH
}
int ob_outermod_set_select_seed(ob_outermod* om, uint64_t seed) { OB_TRY om->om.select_seed = seed; OB_CATCH }
int ob_outermod_selectterms(ob_outermod* om, uint64_t numele, uint64_t* terms) { OB_TRY om->om.selectterms(numele, terms); OB_CATCH }
int ob_outermod_getvar(ob_outermod* om, const uint64_t* terms, uint64_t K, double* out) { OB_TRY om->om.getvar(terms, K, out); OB_CATCH }
int ob_outermod_getlvar_gradhyp(ob_outermod* om, const uint64_t* terms, uint64_t K, double* out) {
  OB_TRY om->om.getlvar_gradhyp(terms, K, out); OB_CATCH
}
int ob_outermod_hyplpdf(ob_outermod* om, const double* hyp, uint64_t n, double* out) { OB_TRY *out = om->om.hyplpdf(hyp, n); OB_CATCH }
int ob_outermod_hyplpdf_grad(ob_outermod* om, const double* hyp, uint64_t n, double* out) { OB_TRY om->om.hyplpdf_grad(hyp, n, out); OB_CATCH }
int ob_outermod_get_index(ob_outermod* om, const char* which, int64_t* out, uint64_t* n) {
  OB_TRY
  const std::string w = which;
  const obh::OuterMod& m = om->om;
  std::vector<int64_t> v;
  if (w == "knotptst") v.assign(m.knotptst.begin(), m.knotptst.end());
  else if (w == "hypst") v.assign(m.hypst.begin(), m.hypst.end());
  else if (w == "hypmatch") v.assign(m.hypmatch.begin(), m.hypmatch.end());
  else if (w == "gest") v.assign(m.gest.begin(), m.gest.end());
  else if (w == "knotptstge") v.assign(m.knotptstge.begin(), m.knotptstge.end());
  else if (w == "maxlevel") v.assign(m.maxlevel.begin(), m.maxlevel.end());
  else throw std::invalid_argument("unknown index table " + w);
  *n = v.size();
  if (out) std::copy(v.begin(), v.end(), out);
  OB_CATCH
}
int ob_outermod_get_real(ob_outermod* om, const char* which, double* out, uint64_t* nrow, uint64_t* ncol) {
  OB_TRY
  const std::string w = which;
  const obh::OuterMod& m = om->om;
  const std::vector<double>* src = nullptr;
  if (w == "basisvar") { src = &m.basisvar; *nrow = src->size(); *ncol = 1; }
  else if (w == "knotpt") { src = &m.knotpt; *nrow = src->size(); *ncol = 1; }
  else if (w == "logbasisvar_gradhyp") { src = &m.logbasisvar_gradhyp; *nrow = src->size(); *ncol = 1; }
  else if (w == "rotmat") { src = &m.rotmat.a; *nrow = m.rotmat.nr; *ncol = m.rotmat.nc; }
  else if (w == "rotmat_gradhyp") { src = &m.rotmat_gradhyp.a; *nrow = m.rotmat_gradhyp.nr; *ncol = m.rotmat_gradhyp.nc; }
  else throw std::invalid_argument("unknown real table " + w);
  if (out) std::copy(src->begin(), src->end(), out);
  OB_CATCH
}

/* ---- outerbase */
int ob_outerbase_create(ob_ctx* ctx, ob_outermod* om, const double* x, uint64_t N, int dograd, ob_outerbase** out) {
  OB_TRY
  need(ctx, "ctx"); need(om, "om");
  auto* h = new ob_outerbase();
  h->ctx = ctx;
  try { h->ob.reset(new obe::OuterBase(ctx->c, &om->om, x, N, dograd != 0)); } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_outerbase_destroy(ob_outerbase* ob) { OB_TRY delete ob; OB_CATCH }
int ob_outerbase_build(ob_outerbase* ob) { OB_TRY ob->ob->build(); OB_CATCH }
int ob_outerbase_set_nthreads(ob_outerbase* ob, int n) { OB_TRY ob->ob->nthreads = (u64)std::max(n, 1); OB_CATCH }
int ob_outerbase_loopvals(ob_outerbase* ob, uint64_t* nthreads, uint64_t* chunksize, uint64_t* loopsize, int* vertpl) {
  OB_TRY
  bool v;
  obh::loopvals(ob->ob->N, ob->ob->nthreads, *chunksize, *loopsize, v);
  *nthreads = ob->ob->nthreads; *vertpl = v;
  OB_CATCH
}
int ob_outerbase_get_real(ob_outerbase* ob, const char* which, double* out, uint64_t* nrow, uint64_t* ncol) {
  OB_TRY
  const std::string w = which;
  obe::OuterBase& b = *ob->ob;
  const double* src = nullptr;
  if (w == "basemat" || w == "basemat_gradhyp") b.ensure_all(); /* the reference's full layout (modandbase.cpp:521-539) */
  if (w == "basemat") { src = b.basemat.p; *nrow = b.N; *ncol = b.M; }
  else if (w == "basemat_gradhyp") { if (!b.dograd) throw std::invalid_argument("built without gradients"); src = b.basematge.p; *nrow = b.N; *ncol = b.Mge; }
  else if (w == "basescale") { src = b.scale.p; *nrow = b.N; *ncol = 1; }
  else if (w == "basescalemat") { src = b.scalemat.p; *nrow = b.N; *ncol = b.d; }
  else throw std::invalid_argument("unknown matrix " + w);
  if (out) { /* strip the 128-row padding of the device layout */
    for (u64 j = 0; j < *ncol; ++j)
      if (b.N) OB_CUDA(cudaMemcpyAsync(out + j * b.N, src + j * b.ld, b.N * sizeof(double), cudaMemcpyDeviceToHost, b.ctx.stream));
    b.ctx.sync();
  }
  OB_CATCH
}
int ob_outerbase_getbase(ob_outerbase* ob, uint64_t dim, double* out) { OB_TRY ob->ob->getbase(dim, out); OB_CATCH }
int ob_outerbase_getmat(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* out) { OB_TRY ob->ob->getmat(terms, K, out); OB_CATCH }
int ob_outerbase_getmat_gradhyp(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* out) { OB_TRY ob->ob->getmat_gradhyp(terms, K, out); OB_CATCH }
int ob_outerbase_mm(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* a, double* out) {
  OB_TRY ob->ob->mm(sq, terms, K, a, out); OB_CATCH
}
int ob_outerbase_tmm(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* a, double* out) {
  OB_TRY ob->ob->tmm(sq, terms, K, a, out); OB_CATCH
}
int ob_outerbase_mm_gradhyp(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* a, double* out, double* outge) {
  OB_TRY ob->ob->mm_gradhyp(sq, terms, K, a, out, outge); OB_CATCH
}
int ob_outerbase_tmm_gradhyp(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* a, double* out, double* outge) {
  OB_TRY ob->ob->tmm_gradhyp(sq, terms, K, a, out, outge); OB_CATCH
}
int ob_outerbase_mm_mat(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* A, uint64_t C, double* out) {
  OB_TRY ob->ob->mm_mat(sq, terms, K, A, C, out); OB_CATCH
}
int ob_outerbase_tmm_mat(ob_outerbase* ob, int sq, const uint64_t* terms, uint64_t K, const double* A, uint64_t C, double* out) {
  OB_TRY ob->ob->tmm_mat(sq, terms, K, A, C, out); OB_CATCH
}
int ob_outerbase_residvar(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* out) {
  OB_TRY need(ob, "ob"); ob->ob->residvar(terms, K, out); OB_CATCH
}
int ob_outerbase_residvar_gradhyp(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* out) {
  OB_TRY need(ob, "ob"); ob->ob->residvar_gradhyp(terms, K, out); OB_CATCH
}
int ob_outerbase_set_terms(ob_outerbase* ob, const uint64_t* terms, uint64_t K) {
  OB_TRY
  need(ob, "ob"); if (K) need(terms, "terms");
  obe::OuterBase& b = *ob->ob;
  b.cur_terms.assign(terms, terms + K * b.d);
  b.cur_K = K;
  b.coltable(b.program(b.cur_terms.data(), K, -1, 0), 0, -1);
  b.coltable(b.program(b.cur_terms.data(), K, -1, 1), 0, -1);
  b.terms_set = true;
  OB_CATCH
}
/* the object behind a *_dev call: a forgotten set_terms would otherwise run a zero-term program silently */
static obe::OuterBase& installed(ob_outerbase* ob) {
  need(ob, "ob");
  if (!ob->ob->terms_set) throw std::logic_error("set_terms has not been called on this outerbase");
  return *ob->ob;
}
int ob_outerbase_mm_dev(ob_outerbase* ob, int sq, const double* a_dev, double* out_dev) {
  OB_TRY obe::OuterBase& b = installed(ob); b.mm_dev(b.cur_terms.data(), b.cur_K, sq, a_dev, out_dev); OB_CATCH
}
int ob_outerbase_tmm_dev(ob_outerbase* ob, int sq, const double* a_dev, double* out_dev) {
  OB_TRY obe::OuterBase& b = installed(ob); b.tmm_dev(b.cur_terms.data(), b.cur_K, sq, a_dev, out_dev, true, b.N); OB_CATCH
}
int ob_outerbase_mm_mat_dev(ob_outerbase* ob, int sq, const double* A_dev, uint64_t C, double* out_dev) {
  OB_TRY obe::OuterBase& b = installed(ob); b.mm_mat_dev(b.cur_terms.data(), b.cur_K, sq, A_dev, C, out_dev, b.N); OB_CATCH
}
int ob_outerbase_tmm_mat_dev(ob_outerbase* ob, int sq, const double* A_dev, uint64_t C, double* out_dev) {
  OB_TRY obe::OuterBase& b = installed(ob); b.tmm_mat_dev(b.cur_terms.data(), b.cur_K, sq, A_dev, b.N, C, out_dev); OB_CATCH
}
int ob_outerbase_terms_stats(ob_outerbase* ob, uint64_t* W, uint64_t* Lcols, uint64_t* nodes, uint64_t* maxdepth) {
  OB_TRY
  obe::OuterBase& b = installed(ob);
  const obt::Program& P = b.program(b.cur_terms.data(), b.cur_K, -1)->host;
  *W = P.W; *Lcols = P.Lcols; *nodes = P.nodes; *maxdepth = P.maxdepth;
  OB_CATCH
}

int ob_ctx_set_option(ob_ctx* ctx, const char* name, double value) {
  OB_TRY
  need(ctx, "ctx"); need(name, "name");
  const std::string n(name);
  if (n == "spec") {
    if (value != 0 && value != 1 && value != 2) throw std::invalid_argument("spec must be 0, 1 or 2");
    ctx->c.spec_mode = (int)value;
  } else if (n == "spec_work") ctx->c.spec_work = value;
  else if (n == "dsweep") ctx->c.dsweep = value != 0;
  else if (n == "device_cg") ctx->c.device_cg = value != 0;
  else if (n == "overlap") ctx->c.overlap = value != 0;
  else if (n == "tmap") ctx->c.tmap = value != 0;
  else if (n == "p2p") ctx->c.p2p.enabled = value != 0; /* same value on every rank */
  else throw std::invalid_argument("unknown option " + n);
  OB_CATCH
}
int ob_outerbase_specialize(ob_outerbase* ob, const uint64_t* terms, uint64_t K, double* compile_seconds) {
  OB_TRY
  need(ob, "ob"); need(terms, "terms");
  obe::OuterBase::SpecEntry* e = ob->ob->spec_for(terms, K, /*force=*/true);
  if (!e) throw std::logic_error("specialisation did not produce a module");
  if (compile_seconds) *compile_seconds = obd::spec_compile_seconds(*e->k);
  OB_CATCH
}
int ob_outerbase_spec_state(ob_outerbase* ob, const uint64_t* terms, uint64_t K, int* state) {
  OB_TRY
  need(ob, "ob"); need(terms, "terms"); need(state, "state");
  *state = 0;
  for (const auto& e : ob->ob->specs)
    if (e.K == K && std::memcmp(e.terms.data(), terms, K * ob->ob->d * sizeof(u64)) == 0) *state = e.state;
  OB_CATCH
}
int ob_spec_source(const uint64_t* terms, uint64_t K, uint64_t d, const int* opts9, char* buf, uint64_t* len, uint64_t* info) {
  OB_TRY
  need(terms, "terms"); need(len, "len");
  obs::SpecOptions o = obd::spec_default_options();
  if (opts9) { o.ra = opts9[0]; o.qa = opts9[1]; o.tga = opts9[2]; o.cache_a = opts9[3]; o.wt = opts9[4]; o.rt = opts9[5]; o.pt = opts9[6]; o.cache_t = opts9[7]; o.acc_cap = opts9[8]; }
  const int types = obs::choose_types(terms, K, d, o);
  if (!types) throw std::invalid_argument("terms table is not trie-compilable (duplicate or too deep terms), or acc_cap is below one trie segment (32)");
  const obt::Program pa = obt::compile(terms, K, d, 1), pt = obt::compile(terms, K, d, types * o.wt);
  const obs::SpecSource S = obs::generate(&pa, &pt, types, o);
  if (!S.ok) throw std::invalid_argument(S.why);
  if (info) { info[0] = (u64)S.types; info[1] = (u64)S.nacc; info[2] = (u64)S.tr_a; info[3] = (u64)S.tr_t; }
  if (buf) {
    if (*len < S.src.size() + 1) throw std::range_error("buffer too small");
    std::memcpy(buf, S.src.c_str(), S.src.size() + 1);
  }
  *len = S.src.size() + 1;
  OB_CATCH
}
int ob_spec_source_dot(const uint64_t* terms, uint64_t K, uint64_t d, char* buf, uint64_t* len, uint64_t* info) {
  OB_TRY
  need(terms, "terms"); need(len, "len");
  const obs::SpecOptions o = obd::spec_default_options();
  const obt::Program pa = obt::compile(terms, K, d, 1);
  if (!pa.fast_ok) throw std::invalid_argument("terms table is not trie-compilable (duplicate or too deep terms)");
  const obs::SpecSource S = obs::generate_dot(pa, o);
  if (!S.ok) throw std::invalid_argument(S.why);
  if (info) { info[0] = (u64)S.nacc; info[1] = (u64)S.tr_a; }
  if (buf) {
    if (*len < S.src.size() + 1) throw std::range_error("buffer too small");
    std::memcpy(buf, S.src.c_str(), S.src.size() + 1);
  }
  *len = S.src.size() + 1;
  OB_CATCH
}
int ob_spec_source_tmat(const uint64_t* terms, uint64_t K, uint64_t d, char* buf, uint64_t* len, uint64_t* info) {
  OB_TRY
  need(terms, "terms"); need(len, "len");
  obs::SpecOptions o = obd::spec_default_options();
  o.wt = obs::kTmWarps; o.acc_cap = obs::kTmTerms;
  const int types = obs::choose_types(terms, K, d, o);
  if (!types) throw std::invalid_argument("terms table is not trie-compilable (duplicate or too deep terms)");
  const obt::Program pt = obt::compile(terms, K, d, types * obs::kTmWarps);
  const obs::SpecSource S = obs::generate_tmat(pt, types, o);
  if (!S.ok) throw std::invalid_argument(S.why);
  if (info) { info[0] = (u64)S.types; info[1] = (u64)S.maxcols_t; }
  if (buf) {
    if (*len < S.src.size() + 1) throw std::range_error("buffer too small");
    std::memcpy(buf, S.src.c_str(), S.src.size() + 1);
  }
  *len = S.src.size() + 1;
  OB_CATCH
}
int ob_spec_source_mat(const uint64_t* terms, uint64_t K, uint64_t d, char* buf, uint64_t* len, uint64_t* info) {
  OB_TRY
  need(terms, "terms"); need(len, "len");
  const obt::Program pa = obt::compile(terms, K, d, 1);
  const obs::SpecSource S = obs::generate_mat(pa, obd::spec_default_options());
  if (!S.ok) throw std::invalid_argument(S.why);
  if (info) { info[0] = (u64)S.nacc; info[1] = (u64)S.tr_a; }
  if (buf) {
    if (*len < S.src.size() + 1) throw std::range_error("buffer too small");
    std::memcpy(buf, S.src.c_str(), S.src.size() + 1);
  }
  *len = S.src.size() + 1;
  OB_CATCH
}
int ob_spec_compile_check(const char* source, uint64_t* cubin_bytes, double* seconds) {
  OB_TRY
  need(source, "source");
  const std::string cubin = obd::spec_compile_nocache(source, seconds);
  if (cubin_bytes) *cubin_bytes = cubin.size();
  OB_CATCH
}

int ob_debug_terms_eval(const uint64_t* terms, uint64_t K, uint64_t d, const uint64_t* knotptst, int ngroups, int aug_dim,
                        const double* bcols, const double* gcols0, const double* a, double b, double* out_phi_a,
                        double* out_phit, uint64_t* stats) {
  OB_TRY
  obt::Program P = obt::compile(terms, K, d, ngroups, aug_dim);
  if (stats) {
    stats[0] = P.W; stats[1] = P.Lcols; stats[2] = P.nodes; stats[3] = P.maxdepth; stats[4] = P.fast_ok;
    stats[5] = P.nslots(); stats[6] = P.fwd.size(); stats[7] = P.bwd.size();
  }
  if (!P.fast_ok) { if (out_phi_a) *out_phi_a = 0; return OB_OK; }
  std::vector<double> packed(P.cols.size());
  for (size_t c = 0; c < P.cols.size(); ++c) {
    const obt::ColRef& cr = P.cols[c];
    packed[c] = cr.aug ? gcols0[cr.level] : bcols[knotptst[cr.dim] + cr.level];
  }
  if (out_phi_a) *out_phi_a = obt::run_bwd_row(P, packed.data(), a);
  if (out_phit) { std::fill(out_phit, out_phit + K, 0.0); obt::run_fwd_row(P, packed.data(), b, out_phit); }
  OB_CATCH
}

int ob_outerbase_debug_phi_geometry(ob_outerbase* ob, const uint64_t* terms, uint64_t K, int transpose, int sq, int* out) {
  OB_TRY
  need(ob, "ob"); need(terms, "terms"); need(out, "out");
  obe::OuterBase& b = *ob->ob;
  obd::phi_geometry_info(b.ctx, b.plan(b.program(terms, K, -1, transpose ? 1 : 0), sq ? 1 : 0, -1), transpose == 0, out);
  OB_CATCH
}

static void build_geometry(const obe::OuterBase& b, int* out) {
  if (b.build_geom.size() != b.d) throw std::logic_error("this object has not built a basis");
  for (size_t l = 0; l < b.build_geom.size(); ++l) {
    const obd::BuildGeom& g = b.build_geom[l];
    out[4 * l] = g.mma; out[4 * l + 1] = g.tile; out[4 * l + 2] = g.mo; out[4 * l + 3] = g.smem;
  }
}
int ob_outerbase_debug_build_geometry(ob_outerbase* ob, int* out) {
  OB_TRY need(ob, "ob"); need(out, "out"); build_geometry(*ob->ob, out); OB_CATCH
}
int ob_lpdf_debug_build_geometry(ob_lpdf* l, int* out) {
  OB_TRY
  need(l, "l"); need(out, "out");
  if (auto* lik = dynamic_cast<obe::DevLik*>(l->p.get())) build_geometry(lik->ob, out);
  else if (auto* gda = dynamic_cast<obe::LoglikGda*>(l->p.get())) build_geometry(gda->ob, out);
  else throw std::invalid_argument("only a likelihood holds a basis");
  OB_CATCH
}

/* ---- stateless linalg.h seam */
#define SEAM_BASE(bmge, Mge, ge, hm, H) \
  need(ctx, "ctx");                     \
  obe::OuterBase ob(ctx->c, N, d, M, knotptst, basemat, basescale, bmge, Mge, ge, hm, H);
int ob_prodmm_vec(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* a, const double* basemat,
                  uint64_t N, uint64_t M, const double* basescale, const uint64_t* knotptst) {
  OB_TRY SEAM_BASE(nullptr, 0, nullptr, nullptr, 0) ob.mm(0, terms, K, a, out); OB_CATCH
}
int ob_tprodmm_vec(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* a, const double* basemat,
                   uint64_t N, uint64_t M, const double* basescale, const uint64_t* knotptst) {
  OB_TRY SEAM_BASE(nullptr, 0, nullptr, nullptr, 0) ob.tmm(0, terms, K, a, out); OB_CATCH
}
int ob_prodmm_mat(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* A, uint64_t C,
                  const double* basemat, uint64_t N, uint64_t M, const double* basescale, const uint64_t* knotptst) {
  OB_TRY SEAM_BASE(nullptr, 0, nullptr, nullptr, 0) ob.mm_mat(0, terms, K, A, C, out); OB_CATCH
}
int ob_tprodmm_mat(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* A, uint64_t C,
                   const double* basemat, uint64_t N, uint64_t M, const double* basescale, const uint64_t* knotptst) {
  OB_TRY SEAM_BASE(nullptr, 0, nullptr, nullptr, 0) ob.tmm_mat(0, terms, K, A, C, out); OB_CATCH
}
int ob_prodmmge(ob_ctx* ctx, double* out, double* outge, const uint64_t* terms, uint64_t K, uint64_t d, const double* a,
                const double* basemat, uint64_t N, uint64_t M, const double* basescale, const uint64_t* knotptst,
                const double* basematge, uint64_t Mge, const uint64_t* gest, const uint64_t* hypmatch, uint64_t H) {
  OB_TRY need(basematge, "basematge"); SEAM_BASE(basematge, Mge, gest, hypmatch, H) ob.mm_gradhyp(0, terms, K, a, out, outge); OB_CATCH
}
int ob_tprodmmge(ob_ctx* ctx, double* out, double* outge, const uint64_t* terms, uint64_t K, uint64_t d, const double* a,
                 const double* basemat, uint64_t N, uint64_t M, const double* basescale, const uint64_t* knotptst,
                 const double* basematge, uint64_t Mge, const uint64_t* gest, const uint64_t* hypmatch, uint64_t H) {
  OB_TRY need(basematge, "basematge"); SEAM_BASE(basematge, Mge, gest, hypmatch, H) ob.tmm_gradhyp(0, terms, K, a, out, outge); OB_CATCH
}
int ob_getm(ob_ctx* ctx, double* out, const uint64_t* terms, uint64_t K, uint64_t d, const double* basemat, uint64_t N, uint64_t M,
            const double* basescale, const uint64_t* knotptst) {
  OB_TRY SEAM_BASE(nullptr, 0, nullptr, nullptr, 0) ob.getmat(terms, K, out); OB_CATCH
}
int ob_getmge(ob_ctx* ctx, double* outge, const uint64_t* terms, uint64_t K, uint64_t d, const double* basemat, uint64_t N, uint64_t M,
              const double* basescale, const uint64_t* knotptst, const double* basematge, uint64_t Mge, const uint64_t* gest,
              const uint64_t* hypmatch, uint64_t H) {
  OB_TRY need(basematge, "basematge"); SEAM_BASE(basematge, Mge, gest, hypmatch, H) ob.getmat_gradhyp(terms, K, outge); OB_CATCH
}

/* ---- lpdf family */
int ob_loglik_gauss_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* y, const double* x,
                           uint64_t N, ob_lpdf** out) {
  OB_TRY
  need(ctx, "ctx"); need(om, "om");
  auto* h = new ob_lpdf();
  h->ctx = ctx;
  try { h->p.reset(new obe::LoglikGauss(ctx->c, &om->om, terms, K, y, x, N)); } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_loglik_std_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* y, const double* x,
                         uint64_t N, ob_lpdf** out) {
  OB_TRY
  need(ctx, "ctx"); need(om, "om");
  auto* h = new ob_lpdf();
  h->ctx = ctx;
  try { h->p.reset(new obe::LoglikStd(ctx->c, &om->om, terms, K, y, x, N)); } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_lpdf_optnewton(ob_lpdf* l) { OB_TRY l->p->optnewton(); OB_CATCH }
int ob_lpdf_hess(ob_lpdf* l, double* out, uint64_t* n) { OB_TRY auto o = l->p->hess(); std::copy(o.begin(), o.end(), out); *n = o.size(); OB_CATCH }
int ob_lpdf_hessgradhyp(ob_lpdf* l, double* out, uint64_t* n) { OB_TRY auto o = l->p->hessgradhyp(); std::copy(o.begin(), o.end(), out); *n = o.size(); OB_CATCH }
int ob_lpdf_hessgradpara(ob_lpdf* l, double* out, uint64_t* n) { OB_TRY auto o = l->p->hessgradpara(); std::copy(o.begin(), o.end(), out); *n = o.size(); OB_CATCH }
int ob_loglik_gda_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* y, const double* x,
                         uint64_t N, ob_lpdf** out) {
  OB_TRY
  need(ctx, "ctx"); need(om, "om");
  auto* h = new ob_lpdf();
  h->ctx = ctx;
  try { h->p.reset(new obe::LoglikGda(ctx->c, &om->om, terms, K, y, x, N)); } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_logpr_gauss_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, ob_lpdf** out) {
  OB_TRY
  need(om, "om");
  auto* h = new ob_lpdf();
  h->ctx = ctx;
  try { h->p.reset(new obe::LogprGauss(&om->om, terms, K)); } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_loglik_gauss_multi_create_ex(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* Y, uint64_t C,
                                    const double* x, uint64_t N, int para_per_column, ob_lpdf** out) {
  OB_TRY
  need(ctx, "ctx"); need(om, "om");
  if (C == 0) throw std::invalid_argument("ncol must be at least 1");
  auto* h = new ob_lpdf();
  h->ctx = ctx;
  try { h->p.reset(new obe::LoglikGaussMulti(ctx->c, &om->om, terms, K, Y, C, x, N, para_per_column != 0)); } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_loglik_gauss_multi_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* Y, uint64_t C,
                                 const double* x, uint64_t N, ob_lpdf** out) {
  return ob_loglik_gauss_multi_create_ex(ctx, om, terms, K, Y, C, x, N, 0, out);
}
int ob_loglik_gda_multi_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, const double* Y, uint64_t C,
                               const double* x, uint64_t N, ob_lpdf** out) {
  OB_TRY
  need(ctx, "ctx"); need(om, "om");
  if (C == 0) throw std::invalid_argument("ncol must be at least 1");
  auto* h = new ob_lpdf();
  h->ctx = ctx;
  try { h->p.reset(new obe::LoglikGdaMulti(ctx->c, &om->om, terms, K, Y, C, x, N)); } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_logpr_gauss_multi_create_ex(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, uint64_t C, int para_per_column,
                                   ob_lpdf** out) {
  OB_TRY
  need(om, "om");
  auto* h = new ob_lpdf();
  h->ctx = ctx;
  try { h->p.reset(new obe::LogprGaussMulti(&om->om, terms, K, C, para_per_column != 0)); } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_logpr_gauss_multi_create(ob_ctx* ctx, ob_outermod* om, const uint64_t* terms, uint64_t K, uint64_t C, ob_lpdf** out) {
  return ob_logpr_gauss_multi_create_ex(ctx, om, terms, K, C, 0, out);
}
int ob_lpdfvec_create(ob_lpdf* a, ob_lpdf* b, ob_lpdf** out) {
  OB_TRY
  need(a, "a"); need(b, "b");
  auto* h = new ob_lpdf();
  h->ctx = a->ctx;
  h->p.reset(new obe::LpdfVec(a->p.get(), b->p.get()));
  *out = h;
  OB_CATCH
}
int ob_lpdf_destroy(ob_lpdf* l) { OB_TRY delete l; OB_CATCH }
int ob_lpdf_setnthreads(ob_lpdf* l, int k) { OB_TRY l->p->setnthreads(k); OB_CATCH }
int ob_lpdf_update(ob_lpdf* l, const double* coeff, uint64_t K) { OB_TRY l->p->update(std::vector<double>(coeff, coeff + K)); OB_CATCH }
int ob_lpdf_updateom(ob_lpdf* l) { OB_TRY l->p->updateom(); OB_CATCH }
int ob_lpdf_updatepara(ob_lpdf* l, const double* para, uint64_t n) { OB_TRY l->p->updatepara(para, n); OB_CATCH }
int ob_lpdf_updateterms(ob_lpdf* l, const uint64_t* terms, uint64_t K) { OB_TRY l->p->updateterms(terms, K); OB_CATCH }
int ob_lpdf_optcg(ob_lpdf* l, double tol, uint64_t maxepch) { OB_TRY l->p->optcg(tol, maxepch); OB_CATCH }
int ob_lpdf_hessmult(ob_lpdf* l, const double* g, double* out) {
  OB_TRY
  std::vector<double> o = l->p->hessmult(std::vector<double>(g, g + l->p->nterms));
  std::copy(o.begin(), o.end(), out);
  OB_CATCH
}
int ob_lpdf_diaghess(ob_lpdf* l, double* out) { OB_TRY auto o = l->p->diaghess(); std::copy(o.begin(), o.end(), out); OB_CATCH }
int ob_lpdf_diaghessgradhyp(ob_lpdf* l, double* out) { OB_TRY auto o = l->p->diaghessgradhyp(); std::copy(o.begin(), o.end(), out); OB_CATCH }
int ob_lpdf_diaghessgradpara(ob_lpdf* l, double* out) { OB_TRY auto o = l->p->diaghessgradpara(); std::copy(o.begin(), o.end(), out); OB_CATCH }
int ob_lpdf_paralpdf(ob_lpdf* l, const double* para, uint64_t n, double* out) { OB_TRY *out = l->p->paralpdf(para, n); OB_CATCH }
int ob_lpdf_paralpdf_grad(ob_lpdf* l, const double* para, uint64_t n, double* out) { OB_TRY l->p->paralpdf_grad(para, n, out); OB_CATCH }
int ob_lpdf_set_flag(ob_lpdf* l, const char* which, int value) {
  OB_TRY
  const std::string w = which;
  if (w == "compute_val") l->p->compute_val = value;
  else if (w == "compute_grad") l->p->compute_grad = value;
  else if (w == "compute_gradhyp") l->p->compute_gradhyp = value;
  else if (w == "compute_gradpara") l->p->compute_gradpara = value;
  else if (w == "fullhess") l->p->fullhess = value;
  else if (w == "domarg") {
    auto* v = dynamic_cast<obe::LpdfVec*>(l->p.get());
    if (!v) throw std::invalid_argument("domarg is a field of lpdfvec");
    v->domargadj = value;
  } else if (w == "dodiag") { /* R field name of loglik_gda::doda, interfaceR.cpp:748 */
    if (auto* v = dynamic_cast<obe::LoglikGda*>(l->p.get())) { v->doda = value; v->redostd = true; }
    else if (auto* m = dynamic_cast<obe::LoglikGdaMulti*>(l->p.get())) { m->doda = value; m->redostd = true; }
    else throw std::invalid_argument("dodiag is a field of loglik_gda / loglik_gda_multi");
  } else throw std::invalid_argument("unknown flag " + w);
  OB_CATCH
}
int ob_lpdf_sizes(ob_lpdf* l, uint64_t* nterms, uint64_t* npara, uint64_t* nhyp, uint64_t* nrow) {
  OB_TRY *nterms = l->p->nterms; *npara = l->p->para.size(); *nhyp = l->p->nhyp(); *nrow = l->p->nrow(); OB_CATCH
}
int ob_lpdf_get(ob_lpdf* l, const char* which, double* out, uint64_t* n) {
  OB_TRY
  const std::string w = which;
  std::vector<double> v;
  if (w == "val") v = {l->p->val};
  else if (w == "grad") v = l->p->grad;
  else if (w == "gradhyp") v = l->p->gradhyp;
  else if (w == "gradpara") v = l->p->gradpara;
  else if (w == "coeff") v = l->p->coeff;
  else if (w == "para") v = l->p->para;
  else if (w == "totdiaghess") v = l->p->totdiaghess;
  else if (w == "tothess") v = l->p->tothess;
  else if (w == "cg_iters") {
    auto* mv = dynamic_cast<obe::LpdfVec*>(l->p.get());
    if (mv && mv->multi()) v.assign(mv->cg_iters_cols.begin(), mv->cg_iters_cols.end());
    else v = {double(l->p->cg_iters)};
  } else if (w == "ncol") v = {double(l->p->ncol())};
  else if (w == "predvar_ncol") {
    if (auto* g = dynamic_cast<obe::LoglikGaussBase*>(l->p.get())) v = {double(g->predvar_ncol())};
    else if (dynamic_cast<obe::LoglikGdaMulti*>(l->p.get())) v = {1.0};
    else throw std::invalid_argument("predvar_ncol is a field of loglik_gauss / loglik_gauss_multi / loglik_gda_multi");
  }
  else if (w == "yhat") {
    if (auto* g = dynamic_cast<obe::LoglikGauss*>(l->p.get())) v = g->get_yhat();
    else if (auto* g2 = dynamic_cast<obe::LoglikGda*>(l->p.get())) v = g2->yhat;
    else if (auto* g3 = dynamic_cast<obe::LoglikGdaMulti*>(l->p.get())) v = g3->get_yhat();
    else throw std::invalid_argument("yhat is a field of loglik_gauss / loglik_gda / loglik_gda_multi");
  } else if (w == "coeffsd") {
    auto* g = dynamic_cast<obe::LogprGauss*>(l->p.get());
    if (!g) throw std::invalid_argument("coeffsd is a field of logpr_gauss");
    v = g->coeffsd;
  } else throw std::invalid_argument("unknown field " + w);
  *n = v.size();
  if (out) std::copy(v.begin(), v.end(), out);
  OB_CATCH
}
int ob_lpdf_set_coeff(ob_lpdf* l, const double* coeff, uint64_t K) { OB_TRY l->p->coeff.assign(coeff, coeff + K); OB_CATCH }

int ob_predictor_create(ob_lpdf* loglik, ob_predictor** out) {
  OB_TRY
  auto* h = new ob_predictor();
  try {
    if (auto* g3 = dynamic_cast<obe::LoglikStd*>(loglik->p.get())) h->p.reset(new obe::PredrStd(*g3)); /* before its base class */
    else if (auto* g = dynamic_cast<obe::LoglikGaussBase*>(loglik->p.get())) h->p.reset(new obe::PredGauss(*g));
    else if (auto* g2 = dynamic_cast<obe::LoglikGda*>(loglik->p.get())) h->p.reset(new obe::PredGda(*g2));
    else if (auto* g4 = dynamic_cast<obe::LoglikGdaMulti*>(loglik->p.get())) h->p.reset(new obe::PredGda(*g4));
    else throw std::invalid_argument("cannot produce a predictor from this obj.");
  } catch (...) { delete h; throw; }
  *out = h;
  OB_CATCH
}
int ob_predictor_destroy(ob_predictor* p) { OB_TRY delete p; OB_CATCH }
int ob_predictor_update(ob_predictor* p, const double* x, uint64_t N) { OB_TRY p->p->update(x, N); OB_CATCH }
int ob_predictor_mean(ob_predictor* p, double* out) { OB_TRY p->p->mean(out); OB_CATCH }
int ob_predictor_var(ob_predictor* p, double* out) { OB_TRY p->p->var(out); OB_CATCH }

} // extern "C"
