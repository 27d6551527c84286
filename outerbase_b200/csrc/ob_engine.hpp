/*
 * ob_engine.hpp -- the reference's C++ classes re-hosted on the GPU kernels.
 *
 *   OuterBase         class outerbase   src/modandbase.h:57-125, src/modandbase.cpp:459-922
 *   Lpdf              class lpdf        src/fit.h:23-90,   optcg src/fit.cpp:37-96
 *   LogprGauss        logpr_gauss       src/lpdfs/logpr_gauss.cpp:41-145   (K-length, host)
 *   LoglikGaussBase   loglik_gauss      src/lpdfs/loglik_gauss.cpp:41-179  (N-length work on the GPU) on C responses;
 *                                       the products: LoglikGauss (one response), LoglikGaussMulti (C columns)
 *   LoglikStd         loglik_std        src/lpdfs/loglik_std.cpp:41-203
 *   LoglikGda         loglik_gda        src/lpdfs/loglik_gda.cpp:47-239
 *   LogprGaussMulti   logpr_gauss on each of C columns
 *   LoglikGdaMulti    loglik_gda on each of C columns (obfit_multi's stage 1)
 *   DevLik            what the device CG needs of a likelihood: LoglikGaussBase and LoglikGdaMulti derive from it
 *   LpdfVec           lpdfvec           src/fit.cpp:174-267,310-428,557-607 (diagonal branch), 269-299 (full branch)
 *   Pred              the predictors PredGauss (pred_gauss, loglik_gauss.cpp:196-227), PredrStd, PredGda
 *
 * State that is N-sized (x, basemat, basemat_gradhyp, basescale, y, yhat, residuals)
 * lives in HBM for the lifetime of the object; K- and H-sized state is mirrored on the
 * host, where the reference's K-vector algebra (CG scalars, prior, marginal
 * adjustment) is executed in the reference's own summation order.
 * basescalesq and basematsq_gradhyp are never stored: the kernels form them from the staged
 * tile in shared memory.  basematsq is materialised at the first squared product after a
 * build (OuterBase::sq_matrix).
 */
#pragma once
#include <cstring>
#include <list>

#include "ob_device.cuh"

namespace obe {

using obd::Ctx;
using obd::DevBuf;
using obh::OuterMod;
using u64 = uint64_t;

/* leading dimension of every N-row device matrix: whole 256-row tiles, pad rows zero */
inline u64 pad128(u64 n) { return ((n + 255) / 256) * 256; }

inline bool all_finite(const std::vector<double>& v) {
  for (double x : v) if (!std::isfinite(x)) return false;
  return true;
}

/* ------------------------------------------------------------------ outerbase */
struct OuterBase {
  Ctx& ctx;
  const OuterMod* om;
  u64 N = 0, ld = 0, d = 0, H = 0, M = 0, Mge = 0;
  bool dograd = true;
  u64 nthreads = 1;
  u64 om_version = 0;
  std::vector<u64> knotptst, gest, hypmatch, hypst;
  /* COMPACT column layout.  The reference builds and stores all m_l columns of every dimension (basemat N x M,
   * basemat_gradhyp N x sum H_l m_l: modandbase.cpp:521-539, 547-626), but the products read only levels up to the
   * highest one in `terms` -- 75 of 400 columns at C3 (SURVEY 8 a4).  Here dimension l holds mo[l] <= m_l columns
   * (levels 0 .. mo[l]-1) starting at column cst[l]; hyper-parameter h of dimension l holds mo[l] gradient columns
   * starting at cge[h].  mo grows on demand (need_levels: a terms table that reaches higher is built for before it is
   * multiplied) and is complete (mo = m, cst = knotptst, cge = gest) whenever somebody asks for the matrices
   * themselves (getbase, get_real: ensure_all).  Objects created from R-level `new(outerbase, om, x)` start complete;
   * the lpdf classes know their terms and start pruned. */
  std::vector<u64> mo, cst, cge;
  u64 Mc = 0, Mgec = 0;
  std::vector<obd::BuildGeom> build_geom; /* the kernel each dimension's last build ran on (a test hook reports it) */
  DevBuf<double> x, basemat, basematge, scalemat, scale;
  /* basematsq (modandbase.cpp:527-531), materialised at the first squared operator after a build: squaring the staged
   * tile inside the Phi kernels instead made every squared product 3x slower than the plain one, and a BFGS
   * evaluation runs 1 + 2H of them (diaghess, diaghessgradhyp) */
  DevBuf<double> basematsq;
  bool sq_valid = false;
  const double* sq_matrix() {
    if (!sq_valid) {
      basematsq.ensure(ld * Mc);
      obd::launch_square(ctx, basemat.p, ld * Mc, basematsq.p);
      sq_valid = true;
    }
    return basematsq.p;
  }
  DevBuf<double> knots_dev, rot_dev, rotg_dev;
  obd::Workspace ws;
  DevBuf<double> tmpK, tmpN, tmpN2, tmpP;

  struct ProgEntry { std::vector<u64> terms; u64 K; int aug; int G; int cap; std::unique_ptr<obd::DevProgram> prog; };
  std::list<ProgEntry> programs;
  struct ColEntry { const obd::DevProgram* prog; int sq; int h; std::unique_ptr<obd::ColTable> ct; };
  std::list<ColEntry> coltables;
  /* terms-specialised kernels of one table (ob_spec.hpp): its two programs (Phi a: G = wa streams,
   * Phi^T: types * wt streams) and the compiled module */
  struct SpecEntry {
    std::vector<u64> terms; u64 K = 0;
    std::unique_ptr<obd::DevProgram> pa, pt, ptm; /* ptm: streams of <= 32 terms for phi_tm_spec, built at first use */
    std::shared_ptr<obd::SpecKernels> k;
    int types = 0, types_m = 0;
    obs::SpecOptions opt;
    int state = 0;      /* 0 interpreter so far, 1 module ready, -1 not specialisable */
    bool probed = false; /* disk cache looked up */
    double work = 0;    /* row-terms sent through the interpreter kernels */
    std::string why;
    /* hyper-gradient products (gradcol_tables): per-dimension column tables whose dim-l entries point
     * into the scratch columns, and their host images */
    std::vector<std::unique_ptr<obd::ColTable>> gtab;
    std::vector<const double*> gsrc_host;
    std::vector<int> gops_host;
  };
  DevBuf<double> tmpC, tmpKd, tmpHp, tmpNg, tmpK2, tmpGe;
  DevBuf<unsigned char> tmpMask;
  std::list<SpecEntry> specs;
  /* terms installed by set_terms for the *_dev entry points; they refuse to run before it */
  std::vector<u64> cur_terms;
  u64 cur_K = 0;
  bool terms_set = false;

  /* hint_terms (K x d): the table the owner is going to multiply with -- the basis is built for its levels only */
  OuterBase(Ctx& c, const OuterMod* om_, const double* xh, u64 N_, bool dograd_, const u64* hint_terms = nullptr, u64 hint_K = 0)
      : ctx(c), om(om_), N(N_), dograd(dograd_) {
    if (!om->knots_set) throw std::range_error("Need to set covfs and knots before building.");
    d = om->d;
    static const bool prune = !(getenv("OB_PRUNE") && std::string(getenv("OB_PRUNE")) == "0");
    if (hint_terms && hint_K && prune) {
      mo.assign(d, 1);
      for (u64 l = 0; l < d; ++l) {
        u64 mx = 0;
        for (u64 k = 0; k < hint_K; ++k) mx = std::max(mx, hint_terms[k + l * hint_K]);
        mo[l] = mx + 1 + kLevelMargin;
      }
    }
    ld = pad128(N);
    nthreads = 1;
    /* x is copied (modandbase.h:60), column by column into the padded layout */
    x.ensure(ld * d);
    OB_CUDA(cudaMemsetAsync(x.p, 0, ld * d * sizeof(double), ctx.stream));
    for (u64 l = 0; l < d; ++l)
      if (N) OB_CUDA(cudaMemcpyAsync(x.p + l * ld, xh + l * N, N * sizeof(double), cudaMemcpyHostToDevice, ctx.stream));
    ctx.sync();
    build();
  }

  /* stateless linalg.h seam (src/linalg.h:9-58): wrap caller-provided basemat / basescale
   * (and optionally basematge) instead of building them; om stays null. */
  OuterBase(Ctx& c, u64 N_, u64 d_, u64 M_, const u64* kp, const double* bm, const double* bs,
            const double* bmge, u64 Mge_, const u64* ge, const u64* hm, u64 H_)
      : ctx(c), om(nullptr), N(N_), dograd(bmge != nullptr) {
    d = d_; M = M_; Mge = Mge_; H = H_;
    ld = pad128(N);
    knotptst.assign(kp, kp + d + 1);
    if (knotptst[d] > M) throw std::range_error("knotptst exceeds the columns of basemat");
    if (bmge) { gest.assign(ge, ge + H + 1); hypmatch.assign(hm, hm + H); }
    mo.resize(d);
    for (u64 l = 0; l < d; ++l) mo[l] = knotptst[l + 1] - knotptst[l];
    cst = knotptst; cge = gest; Mc = M; Mgec = Mge; /* the caller's matrices: complete layout */
    auto put = [&](DevBuf<double>& dst, const double* src, u64 ncol) {
      dst.ensure(ld * std::max<u64>(ncol, 1));
      OB_CUDA(cudaMemsetAsync(dst.p, 0, ld * std::max<u64>(ncol, 1) * sizeof(double), ctx.stream));
      for (u64 j = 0; j < ncol; ++j)
        if (N) OB_CUDA(cudaMemcpyAsync(dst.p + j * ld, src + j * N, N * sizeof(double), cudaMemcpyHostToDevice, ctx.stream));
    };
    put(basemat, bm, M);
    put(scale, bs, 1);
    if (bmge) put(basematge, bmge, Mge);
    ctx.sync();
  }

  void check_terms(const u64* terms, u64 K) const {
    for (u64 l = 0; l < d; ++l) {
      const u64 m = knotptst[l + 1] - knotptst[l];
      for (u64 k = 0; k < K; ++k)
        if (terms[k + l * K] >= m) throw std::range_error("terms level exceeds the number of knots");
    }
  }

  static constexpr u64 kLevelMargin = 2; /* levels built beyond the highest one seen: selectterms grows tables level by level */
  /* a new terms table: rebuild first when it reaches levels the compact layout does not hold */
  void need_levels(const u64* terms, u64 K) {
    if (!om) return;
    bool grow = false;
    for (u64 l = 0; l < d; ++l) {
      u64 mx = 0;
      for (u64 k = 0; k < K; ++k) mx = std::max(mx, terms[k + l * K]);
      if (mx + 1 > mo[l]) { mo[l] = mx + 1 + kLevelMargin; grow = true; }
    }
    if (grow) build();
  }
  bool complete() const {
    for (u64 l = 0; l < d; ++l) if (mo[l] < knotptst[l + 1] - knotptst[l]) return false;
    return true;
  }
  void ensure_all() { /* the matrices themselves are asked for: the reference's full layout */
    if (!om || complete()) return;
    for (u64 l = 0; l < d; ++l) mo[l] = knotptst[l + 1] - knotptst[l];
    build();
  }
  /* outerbase::build (modandbase.cpp:547-626): re-reads the CURRENT state of om */
  void build() {
    if (!om) throw std::logic_error("this outerbase wraps caller-provided matrices");
    if (knotptst != om->knotptst || d != om->d) { /* cached programs were bounds-checked against the OLD knot counts */
      coltables.clear(); programs.clear(); specs.clear();
      if (!knotptst.empty()) mo.clear(); /* the knot layout changed under us (setknot): start complete again */
    }
    d = om->d; hypmatch = om->hypmatch; hypst = om->hypst; gest = om->gest; knotptst = om->knotptst; /* setvals_ :492 */
    H = hypmatch.size();
    M = om->nknot();
    Mge = om->nge();
    if (mo.size() != d) { mo.resize(d); for (u64 l = 0; l < d; ++l) mo[l] = knotptst[l + 1] - knotptst[l]; }
    cst.assign(d + 1, 0); cge.assign(H + 1, 0);
    for (u64 l = 0; l < d; ++l) { mo[l] = std::max<u64>(1, std::min(mo[l], knotptst[l + 1] - knotptst[l])); cst[l + 1] = cst[l] + mo[l]; }
    for (u64 h = 0; h < H; ++h) cge[h + 1] = cge[h] + mo[hypmatch[h]];
    Mc = cst[d]; Mgec = cge[H];
    basemat.ensure(ld * Mc);
    if (dograd) basematge.ensure(ld * Mgec);
    scalemat.ensure(ld * d);
    scale.ensure(ld);
    knots_dev.upload(om->knotpt, ctx.stream);
    rot_dev.upload(om->rotmat.a, ctx.stream);
    if (dograd) rotg_dev.upload(om->rotmat_gradhyp.a, ctx.stream);
    std::vector<obd::BuildDims> dims(d);
    for (u64 l = 0; l < d; ++l) {
      obd::BuildDims& D = dims[l];
      D.kind = om->cov[l].kind; D.m = (int)om->mdim(l); D.nh = om->cov[l].numhyp;
      D.hyp[0] = om->hyp[hypst[l]]; D.hyp[1] = D.nh > 1 ? om->hyp[hypst[l] + 1] : 0.0;
      D.knot_off = knotptst[l]; D.col_off = cst[l]; D.rot_off = knotptst[l]; D.mo = (int)mo[l];
      for (int h = 0; h < D.nh; ++h) { D.ge_off[h] = cge[hypst[l] + h]; D.rotg_off[h] = gest[hypst[l] + h]; }
    }
    obd::launch_basis_build(ctx, dims, x.p, N, ld, knots_dev.p, rot_dev.p, om->rotmat.nr, rotg_dev.p, basemat.p,
                            dograd ? basematge.p : nullptr, scalemat.p, scale.p, dograd, build_geom);
    ctx.sync(); /* host vectors above must outlive the async uploads */
    coltables.clear(); /* buffers may have moved */
    sq_valid = false;
    om_version = om->version;
  }

  /* the program an INTERPRETER Phi kernel runs (dir 0 = Phi a, 1 = Phi^T): 16 term groups, one per compute warp.
   * Tables that prove hot run on the terms-specialised kernels instead (spec_for). */
  obd::DevProgram* program(const u64* terms, u64 K, int aug, int dir = 0) {
    (void)dir;
    return program_g(terms, K, aug, 16, 0);
  }
  obd::DevProgram* program_g(const u64* terms, u64 K, int aug, int G, int cap) {
    for (auto it = programs.begin(); it != programs.end(); ++it)
      if (it->K == K && it->aug == aug && it->G == G && it->cap == cap && std::memcmp(it->terms.data(), terms, K * d * sizeof(u64)) == 0) {
        programs.splice(programs.begin(), programs, it);
        return programs.front().prog.get();
      }
    check_terms(terms, K);
    need_levels(terms, K);
    ProgEntry e;
    e.terms.assign(terms, terms + K * d);
    e.K = K; e.aug = aug; e.G = G; e.cap = cap;
    e.prog.reset(new obd::DevProgram());
    e.prog->host = obt::compile(terms, K, d, G, aug, cap);
    e.prog->upload(ctx.stream);
    ctx.sync();
    programs.push_front(std::move(e));
    while (programs.size() > 96) {
      const obd::DevProgram* dead = programs.back().prog.get();
      coltables.remove_if([&](const ColEntry& c) { return c.prog == dead; });
      programs.pop_back();
    }
    return programs.front().prog.get();
  }

  /* ---- specialisation policy (Ctx::spec_mode): returns the ready entry or null (use the interpreter).
   * `force` compiles now whatever the mode (ob_outerbase_specialize). */
  SpecEntry* spec_for(const u64* terms, u64 K, bool force = false) {
    if ((ctx.spec_mode == 0 && !force) || K == 0 || N == 0) return nullptr;
    if (!om && ctx.spec_mode != 1 && !force) return nullptr; /* one-shot wrappers of the stateless seam */
    SpecEntry* e = nullptr;
    for (auto it = specs.begin(); it != specs.end(); ++it)
      if (it->K == K && std::memcmp(it->terms.data(), terms, K * d * sizeof(u64)) == 0) {
        specs.splice(specs.begin(), specs, it);
        e = &specs.front();
        break;
      }
    if (!e) {
      check_terms(terms, K);
      need_levels(terms, K);
      specs.emplace_front();
      e = &specs.front();
      e->terms.assign(terms, terms + K * d);
      e->K = K;
      while (specs.size() > 8) {
        const SpecEntry& dead = specs.back();
        coltables.remove_if([&](const ColEntry& c) { return c.prog == dead.pa.get() || c.prog == dead.pt.get() || c.prog == dead.ptm.get(); });
        specs.pop_back();
      }
    }
    if (e->state == 1) return e;
    if (e->state < 0) { if (force) throw std::runtime_error("terms table cannot be specialised: " + e->why); return nullptr; }
    const bool now = force || ctx.spec_mode == 1;
    e->work += (double)N * (double)K;
    const bool hot = e->work >= ctx.spec_work;
    const bool probe = !e->probed && (double)N * (double)K >= 1e8; /* large tables: a cached module is free */
    if (!now && !hot && !probe) return nullptr;
    try {
      if (!e->pa) {
        e->pa.reset(new obd::DevProgram());
        e->pa->host = obt::compile(terms, K, d, 1);
        if (!e->pa->host.fast_ok) throw std::runtime_error("not a trie-compilable table (duplicate or too deep terms)");
        e->opt = obd::spec_adapt_options(ctx, obd::spec_default_options(), (int)e->pa->host.cols.size(), e->pa->host.nslots());
        e->types = obs::choose_types(terms, K, d, e->opt);
        if (e->types == 0) throw std::runtime_error("not a trie-compilable table (duplicate or too deep terms)");
        e->pt.reset(new obd::DevProgram());
        e->pt->host = obt::compile(terms, K, d, e->types * e->opt.wt);
        e->pa->upload(ctx.stream);
        e->pt->upload(ctx.stream);
        ctx.sync();
      }
      const obs::SpecOptions& opt = e->opt;
      e->probed = true;
      e->k = obd::spec_build(ctx, e->pa->host, e->pt->host, e->types, opt, /*only_if_cached=*/!(now || hot));
      if (!e->k) return nullptr; /* not in the cache: stay on the interpreter until hot */
      if (!obd::spec_fits(ctx, *e->k, (int)e->pa->host.cols.size())) throw std::runtime_error("row tile does not fit in shared memory");
      e->state = 1;
      return e;
    } catch (const std::exception& ex) {
      e->state = -1;
      e->why = ex.what();
      e->k.reset();
      if (force) throw; /* ob_outerbase_specialize: fail loudly; under a policy the interpreter kernels take over */
      return nullptr;
    }
  }
  /* Phi a / Phi^T of the plain table (no hyper-gradient augmentation): specialised kernels when ready */
  void phi_a(const u64* terms, u64 K, int sq, const obd::PhiAArgs& a, int* grid_out) {
    if (SpecEntry* e = spec_for(terms, K)) { obd::launch_phi_a_spec(ctx, *e->k, plan(e->pa.get(), sq, -1), a, ws, grid_out); return; }
    obd::launch_phi_a(ctx, plan(program(terms, K, -1), sq, -1), a, ws, grid_out);
  }
  /* The specialised kernel stages the input vector with bulk copies of whole 128-row tiles, so it reads up to the
   * padded row count `ld` of a 16-byte aligned source.  Library buffers are padded; a caller's device buffer
   * (w_rows < ld) is used in place when the device allocation it lives in extends that far (the driver tells), and
   * copied to a padded buffer otherwise. */
  DevBuf<double> tmpW;
  /* `ready`: the input vector is still being copied in (Ctx::stream_rows_*); only the specialised kernel can consume
   * it that way -- returns false, having launched nothing, when the table is not specialised */
  bool phi_t(const u64* terms, u64 K, int sq, const double* w_dev, double* out_dev, u64 w_rows = ~(u64)0, const unsigned* ready = nullptr) {
    if (SpecEntry* e = spec_for(terms, K)) {
      const bool misaligned = reinterpret_cast<uintptr_t>(w_dev) & 15u;
      if (misaligned || (w_rows < ld && N % 256 != 0 && !obd::device_range_readable(w_dev, ld * sizeof(double)))) {
        tmpW.ensure(ld);
        OB_CUDA(cudaMemcpyAsync(tmpW.p, w_dev, N * sizeof(double), cudaMemcpyDeviceToDevice, ctx.stream));
        w_dev = tmpW.p;
      }
      obd::launch_phi_t_spec(ctx, *e->k, plan(e->pt.get(), sq, -1), w_dev, out_dev, ws, obd::spec_uses_cluster(*e->k) ? nullptr : ready);
      return !ready || !obd::spec_uses_cluster(*e->k);
    }
    if (ready) return false;
    obd::launch_phi_t(ctx, plan(program(terms, K, -1, 1), sq, -1), w_dev, out_dev, ws);
    return true;
  }

  /* H hyper-gradient dots from ONE sweep over the rows (phi_d_spec, ob_spec_scaffold.inc: reverse-mode walk of the trie,
   * d(Phi a)/dB for every basis column, contracted with the stored gradient columns per dimension), for the plain
   * (sq = 0: loglik_gauss::update, loglik_gauss.cpp:127) and the squared operator (sq = 1: sqmm_gradhyp,
   * modandbase.cpp:855-866, rows weighted by w or by one).  Option "dsweep" (Ctx::dsweep).  false: not available for
   * this table -- the caller uses one product per hyper-parameter. */
  bool gradhyp_sweep(const u64* terms, u64 K, int sq, const double* a_dev, const double* w_dev, double* out_dev /* H */) {
    if (!ctx.dsweep || !dograd || H == 0) return false;
    SpecEntry* e = spec_for(terms, K);
    if (!e) return false;
    obd::DotArgs g;
    g.gmat = basematge.p; g.bmat = sq ? basemat.p : nullptr; g.ld = ld; g.H = (int)H; g.d = (int)d;
    g.hypst = hypst.data(); g.gest = cge.data(); g.knotptst = cst.data();
    return obd::launch_phi_d_spec(ctx, *e->k, plan(e->pa.get(), sq, -1), a_dev, w_dev, g, out_dev);
  }
  /* The column tables of the hyper-gradient products on the specialised kernels, one per dimension l: program P with
   * dimension l's columns replaced by the scratch columns C_j of tmpC (launch_gradcols), every other column read from
   * the basis (squared operator: basematsq).  Uploaded on every call; the caller synchronises before it returns, so
   * the host images outlive the uploads.  Returns each dimension's highest level in P. */
  std::vector<u64> gradcol_tables(SpecEntry& e, const obt::Program& P, int sq) {
    const size_t nc = P.cols.size();
    std::vector<u64> lmax(d, 0);
    for (const obt::ColRef& cr : P.cols) lmax[cr.dim] = std::max<u64>(lmax[cr.dim], cr.level);
    u64 lall = 1;
    for (u64 l = 0; l < d; ++l) lall = std::max(lall, lmax[l]);
    tmpC.ensure(ld * lall);
    if (e.gtab.size() != d) { e.gtab.clear(); for (u64 l = 0; l < d; ++l) e.gtab.emplace_back(new obd::ColTable()); }
    e.gsrc_host.assign(d * nc, nullptr);
    e.gops_host.assign(nc, obd::COL_COPY);
    for (u64 l = 0; l < d; ++l) {
      for (size_t c = 0; c < nc; ++c) {
        const obt::ColRef& cr = P.cols[c];
        e.gsrc_host[l * nc + c] = cr.dim == l ? tmpC.p + (cr.level - 1) * ld : (sq ? sq_matrix() : basemat.p) + (cst[cr.dim] + cr.level) * ld;
      }
      obd::ColTable& ct = *e.gtab[l];
      ct.ncol = ct.nload = (int)nc; ct.has_ops = false;
      ct.load_src.upload(e.gsrc_host.data() + l * nc, nc, ctx.stream);
      ct.col_op.upload(e.gops_host.data(), nc, ctx.stream);
    }
    return lmax;
  }
  /* out[h] = gradhyp[h] = sum_n w_n * outge[n,h] for every hyper-parameter, outge = prodmmge_ (linalg.cpp:225-277)
   * of the coefficients a (host and device copies); local sums of this rank's rows.  In order of preference:
   *  - the sweep (gradhyp_sweep);
   *  - on the specialised kernels, the reference's own form (domultgesub_, linalg.cpp:139-163, 273-276):
   *      outge[:,h] = basescale % ( sum_{k: t_kl>0} a_k T_k^(-l) % (G_h[:,t_kl] - G_h[:,0] % B_l[:,t_kl]) ) + G_h[:,0] % yhat
   *    i.e. ONE plain product per hyper-parameter with the coefficients of the terms that skip dimension l zeroed and
   *    dimension l's columns replaced by C_j = G_j - G_0 % B_j.  Its PHI_DOT epilogue folds the dot with w, so yhatge
   *    is never stored;
   *  - one augmented interpreter product per hyper-parameter (ob_terms.hpp), then its dot with w. */
  void gradhyp_dots(const u64* terms, u64 K, const std::vector<double>& a_host, const double* a_dev, const double* w_dev,
                    const double* yhat_dev, double* out_dev /* H */) {
    if (H == 0) return;
    if (SpecEntry* e = dograd ? spec_for(terms, K) : nullptr) {
      if (ctx.dsweep) {
        tmpKd.upload(a_host, ctx.stream);
        const bool done = gradhyp_sweep(terms, K, 0, tmpKd.p, w_dev, out_dev);
        ctx.sync(); /* a_host must outlive the upload */
        if (done) return;
      }
      /* masked coefficients, one copy per dimension */
      std::vector<double> am(d * K);
      for (u64 l = 0; l < d; ++l)
        for (u64 k = 0; k < K; ++k) am[l * K + k] = terms[k + l * K] > 0 ? a_host[k] : 0.0;
      tmpKd.upload(am, ctx.stream);
      const std::vector<u64> lmax = gradcol_tables(*e, e->pa->host, 0);
      tmpHp.ensure(H * (u64)ctx.sms);
      for (u64 h = 0; h < H; ++h) {
        const u64 l = hypmatch[h];
        const double* G = basematge.p + cge[h] * ld;
        obd::launch_gradcols(ctx, basemat.p + cst[l] * ld, G, ld, lmax[l], tmpC.p);
        obd::PhiPlan pl;
        pl.prog = e->pa.get(); pl.cols = e->gtab[l].get(); pl.scale = scale.p; pl.sq = 0; pl.N = N;
        obd::PhiAArgs a;
        a.a = tmpKd.p + l * K; a.mode = obd::PHI_DOT; a.y = G; a.wdot = w_dev; a.yh = yhat_dev; a.ssq_partial = tmpHp.p + h * ctx.sms;
        int grid = 0;
        obd::launch_phi_a_spec(ctx, *e->k, pl, a, ws, &grid);
        obd::launch_sum_partials(ctx, tmpHp.p + h * ctx.sms, grid, out_dev + h);
      }
      ctx.sync(); /* the host images above must outlive the uploads */
      return;
    }
    tmpGe.ensure(ld + 4 * ctx.sms);
    for (u64 h = 0; h < H; ++h) {
      obd::PhiAArgs g; g.a = a_dev; g.out = tmpGe.p; g.mode = obd::PHI_PLAIN;
      obd::launch_phi_a(ctx, plan(program(terms, K, (int)hypmatch[h]), 0, (int)h), g, ws, nullptr);
      int nb = 0;
      obd::launch_dot_partials(ctx, w_dev, tmpGe.p, N, tmpGe.p + ld, &nb);
      obd::launch_sum_partials(ctx, tmpGe.p + ld, nb, out_dev + h);
    }
  }

  obd::ColTable* coltable(const obd::DevProgram* prog, int sq, int h) {
    for (auto& c : coltables) if (c.prog == prog && c.sq == sq && c.h == h) return c.ct.get();
    const obt::Program& P = prog->host;
    std::vector<const double*> src;
    std::vector<int> ops;
    std::vector<const double*> aux;
    for (const obt::ColRef& cr : P.cols) {
      if (!cr.aug) {
        src.push_back((sq ? sq_matrix() : basemat.p) + (cst[cr.dim] + cr.level) * ld);
        ops.push_back(obd::COL_COPY);
      } else {
        if (h < 0 || hypmatch[h] != cr.dim || !dograd) throw std::logic_error("gradient column without a hyper-parameter");
        src.push_back(basematge.p + (cge[h] + cr.level) * ld);
        if (sq) { /* basematsq_gradhyp = 2*(Rt % R), modandbase.cpp:588-590 */
          ops.push_back(obd::COL_TWO_G_B | (int)((P.cols.size() + aux.size()) << 8));
          aux.push_back(basemat.p + (cst[cr.dim] + cr.level) * ld);
        } else ops.push_back(obd::COL_COPY);
      }
    }
    ColEntry e;
    e.prog = prog; e.sq = sq; e.h = h;
    e.ct.reset(new obd::ColTable());
    e.ct->ncol = (int)src.size();
    src.insert(src.end(), aux.begin(), aux.end());
    e.ct->nload = (int)src.size();
    e.ct->has_ops = !aux.empty();
    e.ct->load_src.upload(src, ctx.stream);
    e.ct->col_op.upload(ops, ctx.stream);
    e.ct->src_host = src;
    ctx.sync();
    coltables.push_front(std::move(e));
    return coltables.front().ct.get();
  }

  obd::PhiPlan plan(const obd::DevProgram* prog, int sq, int h) {
    obd::PhiPlan pl;
    pl.prog = prog; pl.cols = coltable(prog, sq, h); pl.scale = scale.p; pl.sq = sq; pl.N = N; pl.ld = ld;
    return pl;
  }

  /* ---- device-pointer operations (stream ordered, not synchronised) */
  void mm_dev(const u64* terms, u64 K, int sq, const double* a_dev, double* out_dev) {
    obd::PhiAArgs a; a.a = a_dev; a.out = out_dev; a.mode = obd::PHI_PLAIN;
    phi_a(terms, K, sq, a, nullptr);
  }
  bool tmm_dev(const u64* terms, u64 K, int sq, const double* w_dev, double* out_dev, bool reduce_ranks = true, u64 w_rows = ~(u64)0,
               const unsigned* ready = nullptr) {
    if (!reduce_ranks) return phi_t(terms, K, sq, w_dev, out_dev, w_rows, ready);
    obd::Ctx::FuseScope fuse(ctx, K); /* cross-CTA and cross-rank reductions in one launch when peer memory is mapped */
    if (!phi_t(terms, K, sq, w_dev, out_dev, w_rows, ready)) return false;
    ctx.allreduce_after(out_dev, K);
    return true;
  }
  /* prodmmge_: outge column h = augmented-program product (ob_terms.hpp) */
  void mm_ge_dev(const u64* terms, u64 K, int sq, const double* a_dev, double* out_dev, double* outge_dev, u64 ldo) {
    if (!dograd) throw std::logic_error("outerbase was built without gradients");
    if (out_dev) mm_dev(terms, K, sq, a_dev, out_dev);
    for (u64 h = 0; h < H; ++h) {
      obd::PhiAArgs a; a.a = a_dev; a.out = outge_dev + h * ldo; a.mode = obd::PHI_PLAIN;
      obd::launch_phi_a(ctx, plan(program(terms, K, (int)hypmatch[h]), sq, (int)h), a, ws, nullptr);
    }
  }
  /* tprodmmge_'s outge (linalg.cpp:394-471) in the reference's own form (dotmultgesub_, :364-386) on the specialised
   * Phi^T kernel: column h = Phi^T (G_h[:,0] % w) + [t_kl > 0] % Phi_C^T w, where Phi_C is the plain product with
   * dimension l's columns replaced by C_j = G_j - G_0 % B_j (squared operators: 2 G_0, C_j = 2 B_j (G_j - G_0 B_j),
   * every other column squared in shared memory).  Two plain products per hyper-parameter on the same terms table. */
  bool tmm_ge_spec(const u64* terms, u64 K, int sq, const double* w_dev, double* outge_dev /* K x H, local sums */) {
    if (!dograd || H == 0) return false;
    SpecEntry* e = spec_for(terms, K);
    if (!e) return false;
    tmpNg.ensure(ld);
    tmpK2.ensure(2 * K);
    std::vector<unsigned char> mask(d * K);
    for (u64 l = 0; l < d; ++l)
      for (u64 k = 0; k < K; ++k) mask[l * K + k] = terms[k + l * K] > 0 ? 1 : 0;
    tmpMask.upload(mask, ctx.stream);
    const std::vector<u64> lmax = gradcol_tables(*e, e->pt->host, sq);
    for (u64 h = 0; h < H; ++h) {
      const u64 l = hypmatch[h];
      const double* G = basematge.p + cge[h] * ld;
      obd::launch_scaled_product(ctx, sq ? 2.0 : 1.0, G, w_dev, N, tmpNg.p); /* rows beyond N are masked by the kernel */
      obd::launch_phi_t_spec(ctx, *e->k, plan(e->pt.get(), sq, -1), tmpNg.p, tmpK2.p, ws);
      obd::launch_gradcols(ctx, basemat.p + cst[l] * ld, G, ld, lmax[l], tmpC.p, sq);
      obd::PhiPlan pl;
      pl.prog = e->pt.get(); pl.cols = e->gtab[l].get(); pl.scale = scale.p; pl.sq = sq; pl.N = N;
      obd::launch_phi_t_spec(ctx, *e->k, pl, w_dev, tmpK2.p + K, ws);
      obd::launch_masked_add(ctx, tmpK2.p, tmpK2.p + K, tmpMask.p + l * K, K, outge_dev + h * K);
    }
    ctx.sync(); /* the host images above must outlive the uploads */
    return true;
  }
  void tmm_ge_dev(const u64* terms, u64 K, int sq, const double* w_dev, double* out_dev /* K*(1+H): out | outge */) {
    if (!dograd) throw std::logic_error("outerbase was built without gradients");
    phi_t(terms, K, sq, w_dev, out_dev);
    if (!tmm_ge_spec(terms, K, sq, w_dev, out_dev + K))
      for (u64 h = 0; h < H; ++h)
        obd::launch_phi_t(ctx, plan(program(terms, K, (int)hypmatch[h], 1), sq, (int)h), w_dev, out_dev + (1 + h) * K, ws);
    ctx.allreduce_sum(out_dev, K * (1 + H));
  }

  /* ---- host-pointer operations (the reference's call signatures) */
  void d2h(double* dst, const double* src, u64 n) {
    if (n) OB_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDeviceToHost, ctx.stream));
    ctx.sync();
  }
  /* The host-pointer forms overlap their transfers with the kernel (bench.py's `e2e`): a page-locked, mapped result
   * buffer is written by the kernel itself while it computes; an input vector is copied in chunks on a second stream
   * while the Phi^T kernel already consumes the rows that have arrived. */
  static constexpr u64 kOverlapRows = 1u << 17;
  void mm(int sq, const u64* terms, u64 K, const double* a, double* out) {
    tmpK.upload(a, K, ctx.stream);
    if (ctx.overlap && N >= kOverlapRows)
      if (double* mapped = obd::Ctx::mapped_host_pointer(out)) {
        mm_dev(terms, K, sq, tmpK.p, mapped);
        ctx.sync();
        return;
      }
    tmpN.ensure(ld);
    mm_dev(terms, K, sq, tmpK.p, tmpN.p);
    d2h(out, tmpN.p, N);
  }
  void tmm(int sq, const u64* terms, u64 K, const double* a, double* out) {
    tmpN.ensure(ld);
    tmpK.ensure(K);
    bool done = false;
    if (ctx.overlap && N >= kOverlapRows && N < (1ull << 31)) {
      const unsigned* ready = ctx.stream_rows_begin();
      done = tmm_dev(terms, K, sq, tmpN.p, tmpK.p, true, ~(u64)0, ready);
      if (done) ctx.stream_rows_copy(tmpN.p, a, N); /* after the launch: a pageable source blocks the host per chunk */
      ctx.stream_rows_end();
    }
    if (!done) {
      if (N) OB_CUDA(cudaMemcpyAsync(tmpN.p, a, N * sizeof(double), cudaMemcpyHostToDevice, ctx.stream));
      tmm_dev(terms, K, sq, tmpN.p, tmpK.p);
    }
    d2h(out, tmpK.p, K);
  }
  void mm_gradhyp(int sq, const u64* terms, u64 K, const double* a, double* out, double* outge) {
    tmpK.upload(a, K, ctx.stream);
    tmpN.ensure(ld);
    tmpN2.ensure(ld * std::max<u64>(H, 1));
    mm_ge_dev(terms, K, sq, tmpK.p, out ? tmpN.p : nullptr, tmpN2.p, ld);
    if (out) d2h(out, tmpN.p, N);
    for (u64 h = 0; h < H; ++h) d2h(outge + h * N, tmpN2.p + h * ld, N);
  }
  void tmm_gradhyp(int sq, const u64* terms, u64 K, const double* a, double* out, double* outge) {
    tmpN.ensure(ld);
    if (N) OB_CUDA(cudaMemcpyAsync(tmpN.p, a, N * sizeof(double), cudaMemcpyHostToDevice, ctx.stream));
    tmpK.ensure(K * (1 + H));
    tmm_ge_dev(terms, K, sq, tmpN.p, tmpK.p);
    std::vector<double> h(K * (1 + H));
    d2h(h.data(), tmpK.p, K * (1 + H));
    if (out) std::copy(h.begin(), h.begin() + K, out);
    std::copy(h.begin() + K, h.end(), outge);
  }
  /* multi right-hand sides: one pass per column for now (DMMA kernel: DESIGN.md "next") */
  /* prodmm_(mat), linalg.cpp:527-557: eight or more columns run as ONE dense contraction on the FP64 tensor cores
   * (phi_am_spec) when the table is specialised; otherwise a column loop over the vector kernels */
  void mm_mat_dev(const u64* terms, u64 K, int sq, const double* A_dev, u64 C, double* out_dev, u64 ldo) {
    if (C >= 8)
      if (SpecEntry* e = spec_for(terms, K))
        if (obd::launch_phi_am_spec(ctx, *e->k, plan(e->pa.get(), sq, -1), A_dev, C, out_dev, ldo)) return;
    for (u64 c = 0; c < C; ++c) mm_dev(terms, K, sq, A_dev + c * K, out_dev + c * ldo);
  }
  /* tprodmm_(mat), linalg.cpp:583-637: eight or more columns run as dense contractions over the rows on the FP64 tensor
   * cores (phi_tm_spec) when the table is specialised; otherwise a column loop over the vector kernels */
  void tmm_mat_dev(const u64* terms, u64 K, int sq, const double* A_dev, u64 lda, u64 C, double* out_dev) {
    if (C >= 8)
      if (SpecEntry* e = spec_for(terms, K)) {
        if (!e->ptm && e->types_m >= 0) {
          obs::SpecOptions o = e->opt;
          o.wt = obs::kTmWarps; o.acc_cap = obs::kTmTerms;
          e->types_m = obs::choose_types(terms, K, d, o);
          if (e->types_m > 0 && e->types_m <= ctx.sms) {
            e->ptm.reset(new obd::DevProgram());
            e->ptm->host = obt::compile(terms, K, d, e->types_m * obs::kTmWarps);
            e->ptm->upload(ctx.stream);
            ctx.sync();
          } else e->types_m = -1;
        }
        if (e->ptm && obd::launch_phi_tm_spec(ctx, *e->k, plan(e->ptm.get(), sq, -1), e->types_m, A_dev, lda, C, out_dev)) {
          ctx.allreduce_sum(out_dev, K * C);
          return;
        }
      }
    for (u64 c = 0; c < C; ++c) tmm_dev(terms, K, sq, A_dev + c * lda, out_dev + c * K, false, std::min<u64>(ld, (C - c) * lda));
    ctx.allreduce_sum(out_dev, K * C);
  }
  void mm_mat(int sq, const u64* terms, u64 K, const double* A, u64 C, double* out) {
    tmpK.upload(A, K * C, ctx.stream);
    tmpN2.ensure(ld * C);
    mm_mat_dev(terms, K, sq, tmpK.p, C, tmpN2.p, ld);
    for (u64 c = 0; c < C; ++c) d2h(out + c * N, tmpN2.p + c * ld, N);
  }
  void tmm_mat(int sq, const u64* terms, u64 K, const double* A, u64 C, double* out) {
    tmpN2.ensure(ld * C);
    /* pad rows must be finite: the tensor-core kernel multiplies them by Phi = 0 */
    if (N < ld) OB_CUDA(cudaMemsetAsync(tmpN2.p, 0, ld * C * sizeof(double), ctx.stream));
    for (u64 c = 0; c < C; ++c)
      if (N) OB_CUDA(cudaMemcpyAsync(tmpN2.p + c * ld, A + c * N, N * sizeof(double), cudaMemcpyHostToDevice, ctx.stream));
    tmpK.ensure(K * C);
    tmm_mat_dev(terms, K, sq, tmpN2.p, ld, C, tmpK.p);
    d2h(out, tmpK.p, K * C);
  }
  /* outerbase::residvar / residvar_gradhyp, modandbase.cpp:889-922 (assume a correlation function) */
  void residvar(const u64* terms, u64 K, double* out /* N */) {
    if (!om) throw std::logic_error("residvar needs the outermod");
    std::vector<double> varc(K);
    om->getvar(terms, K, varc.data());
    mm(1, terms, K, varc.data(), out);
    for (u64 i = 0; i < N; ++i) out[i] = 1 - out[i];
  }
  void residvar_gradhyp(const u64* terms, u64 K, double* out /* N x H */) {
    if (!om) throw std::logic_error("residvar_gradhyp needs the outermod");
    std::vector<double> varc(K), l2(K * H), l3(N * H);
    om->getvar(terms, K, varc.data());
    mm_gradhyp(1, terms, K, varc.data(), nullptr, out);
    om->getlvar_gradhyp(terms, K, l2.data());
    for (u64 h = 0; h < H; ++h)
      for (u64 k = 0; k < K; ++k) l2[k + h * K] *= varc[k];
    mm_mat(1, terms, K, l2.data(), H, l3.data());
    for (u64 i = 0; i < N * H; ++i) out[i] = -out[i] - l3[i];
  }
  void getmat(const u64* terms, u64 K, double* out) {
    obd::DevProgram* pr = program(terms, K, -1);
    tmpP.ensure(ld * K);
    obd::launch_getmat(ctx, plan(pr, 0, -1), tmpP.p, ld);
    for (u64 k = 0; k < K; ++k) d2h(out + k * N, tmpP.p + k * ld, N);
  }
  /* the explicit basis matrix (h < 0, getmat :649) or its derivative in hyper-parameter h (one slice of
   * getmat_gradhyp :663, dogetmge_ linalg.cpp:741-750: the factor of dimension hypmatch[h] replaced by its gradient
   * column) in HBM: ld x K, pad rows zero */
  void getmat_dev(const u64* terms, u64 K, int h, double* out_dev) {
    if (h >= 0 && !dograd) throw std::logic_error("outerbase was built without gradients");
    if (N < ld) OB_CUDA(cudaMemsetAsync(out_dev, 0, ld * K * sizeof(double), ctx.stream));
    obd::DevProgram* pr = program(terms, K, h < 0 ? -1 : (int)hypmatch[h]);
    obd::launch_getmat(ctx, plan(pr, 0, h), out_dev, ld);
  }
  /* outerbase::getmat_gradhyp (modandbase.cpp:663-669; getmge_ linalg.cpp:778-822): N x K x H, slice after slice */
  void getmat_gradhyp(const u64* terms, u64 K, double* out) {
    tmpP.ensure(ld * std::max<u64>(K, 1));
    for (u64 h = 0; h < H; ++h) {
      getmat_dev(terms, K, (int)h, tmpP.p);
      for (u64 k = 0; k < K; ++k) d2h(out + (h * K + k) * N, tmpP.p + k * ld, N);
    }
  }
  void getbase(u64 dim1, double* out) {
    if (dim1 < 1 || dim1 > d) throw std::range_error("dim out of range");
    ensure_all();
    const u64 l = dim1 - 1, m = knotptst[l + 1] - knotptst[l];
    tmpP.ensure(N * m + 1);
    obd::launch_getbase(ctx, basemat.p, scalemat.p + l * ld, N, ld, cst[l], m, tmpP.p);
    d2h(out, tmpP.p, N * m);
  }
};

/* ------------------------------------------------------------------ lpdf family */
struct Lpdf {
  double val = 0;
  std::vector<double> grad, gradhyp, gradpara, para, coeff, totdiaghess, para0, paravar;
  std::vector<u64> terms; /* K x d */
  u64 d = 0;
  std::vector<double> tothess; /* K x K, fit.h:33 */
  bool didfulltothess = false, didnotothess = true, fullhess = false;
  bool compute_val = true, compute_grad = true, compute_gradhyp = false, compute_gradpara = false;
  u64 npara = 0, nterms = 0, cg_iters = 0;
  virtual ~Lpdf() {}
  virtual void setnthreads(int) {}
  virtual double paralpdf(const double* p, u64 n) const { /* fit.cpp:133-142 */
    if (npara != n) return -std::numeric_limits<double>::infinity();
    std::vector<double> t(n);
    for (u64 l = 0; l < n; ++l) { const double e = p[l] - para0[l]; t[l] = e * e / paravar[l]; }
    return 0.0 - 0.5 * obh::sum2(t.data(), n);
  }
  virtual void paralpdf_grad(const double* p, u64 n, double* out) const { /* fit.cpp:146-157 */
    for (u64 l = 0; l < para.size(); ++l) out[l] = 0.0;
    if (npara != n) return;
    for (u64 l = 0; l < n; ++l) out[l] -= (p[l] - para0[l]) / paravar[l];
  }
  virtual void updateom() {}
  virtual void updatepara(const double*, u64) {}
  virtual void updateterms(const u64*, u64) {}
  virtual void update(const std::vector<double>&) {}
  virtual std::vector<double> hessmult(const std::vector<double>&) { return {}; }
  virtual std::vector<double> diaghess() { return {}; }
  virtual std::vector<double> diaghessgradhyp() { return {}; } /* K x H */
  virtual std::vector<double> diaghessgradpara() { return {}; } /* K x npara */
  /* out[h] = sum_k c[k] * diaghessgradhyp[k, h] without forming the K x H matrix, when the object can (lpdfvec's
   * marginal adjustment, fit.cpp:259-263, only needs this contraction with c = 1 / diaghess) */
  virtual bool diaghessgradhyp_dot(const std::vector<double>&, std::vector<double>&) { return false; }
  virtual bool can_diaghessgradhyp_dot() const { return false; }
  /* out[j] = sum_k diaghessgradpara[k, j] / dh[k] (lpdfvec's marginal adjustment, fit.cpp:264-266) without forming the
   * nterms x npara matrix, when the object can; objects whose npara grows with the columns do */
  virtual bool diaghessgradpara_dot(const std::vector<double>&, std::vector<double>&) { return false; }
  virtual void settotdiaghess(const std::vector<double>& dh) { totdiaghess = dh; didfulltothess = false; didnotothess = false; }
  /* full Hessian, fit.h:81-88: K x K, K x K x H, K x K x npara (column-major, slice after slice); empty when the
   * object has none (loglik_gauss, loglik_gda) */
  virtual void settothess(const std::vector<double>& h) { tothess = h; didfulltothess = true; didnotothess = false; }
  virtual std::vector<double> hess() { return {}; }
  virtual std::vector<double> hessgradhyp() { return {}; }
  virtual std::vector<double> hessgradpara() { return {}; }
  virtual u64 nhyp() const { return 0; }
  virtual u64 nrow() const { return 0; }
  /* multi-response objects (loglik_gauss_multi, logpr_gauss_multi, an lpdfvec of them): ncol responses, coefficients
   * K x ncol column-major, nterms = K * ncol */
  virtual bool multi() const { return false; }
  virtual u64 ncol() const { return 1; }
  /* multi-response objects with one para entry per column (for an lpdfvec: either child) */
  virtual bool para_per_column() const { return false; }
  /* set with totdiaghess by an lpdfvec with a per-column child: the total diagonal's K-long column blocks then differ,
   * so a multi-response predictor gives one variance per column */
  bool totdiaghess_percol = false;

  /* dense K x K algebra of the full-Hessian branch: host side, like every other K-sized object of the lpdf family */
  /* solve A X = B by elimination with partial pivoting (Armadillo solve(): LAPACK dgesv); B is n x m */
  static std::vector<double> dense_solve(std::vector<double> A, std::vector<double> B, u64 n, u64 m) {
    if (A.size() != n * n || B.size() != n * m) throw std::invalid_argument("solve(): incompatible dimensions");
    for (u64 k = 0; k < n; ++k) {
      u64 piv = k;
      for (u64 i = k + 1; i < n; ++i) if (std::fabs(A[i + k * n]) > std::fabs(A[piv + k * n])) piv = i;
      if (A[piv + k * n] == 0.0) throw std::runtime_error("solve(): solution not found");
      if (piv != k) {
        for (u64 j = 0; j < n; ++j) std::swap(A[k + j * n], A[piv + j * n]);
        for (u64 j = 0; j < m; ++j) std::swap(B[k + j * n], B[piv + j * n]);
      }
      const double inv = 1.0 / A[k + k * n];
      for (u64 i = k + 1; i < n; ++i) A[i + k * n] *= inv; /* multipliers */
      for (u64 j = k + 1; j < n; ++j) {
        const double akj = A[k + j * n];
        if (akj == 0.0) continue;
        for (u64 i = k + 1; i < n; ++i) A[i + j * n] -= A[i + k * n] * akj;
      }
      for (u64 j = 0; j < m; ++j) {
        const double bkj = B[k + j * n];
        if (bkj == 0.0) continue;
        for (u64 i = k + 1; i < n; ++i) B[i + j * n] -= A[i + k * n] * bkj;
      }
    }
    for (u64 j = 0; j < m; ++j)
      for (u64 ii = n; ii-- > 0;) {
        const double x = B[ii + j * n] / A[ii + ii * n];
        B[ii + j * n] = x;
        for (u64 i = 0; i < ii; ++i) B[i + j * n] -= A[i + ii * n] * x;
      }
    return B;
  }
  static std::vector<double> dense_inv(const std::vector<double>& A, u64 n) {
    std::vector<double> I(n * n, 0.0);
    for (u64 i = 0; i < n; ++i) I[i + i * n] = 1.0;
    return dense_solve(A, std::move(I), n, n);
  }

  /* lpdf::optnewton, fit.cpp:98-131: one Newton step on the full Hessian */
  virtual void optnewton() {
    fullhess = true;
    compute_val = true; compute_grad = true; compute_gradhyp = false; compute_gradpara = false;
    if (coeff.size() != nterms) coeff.assign(nterms, 0.0);
    update(std::vector<double>(coeff));
    const std::vector<double> h = hess();
    const std::vector<double> r = grad;
    if (!all_finite(h) && !all_finite(r)) { val = -std::numeric_limits<double>::infinity(); return; }
    const std::vector<double> step = dense_solve(h, r, nterms, 1); /* throws on an empty Hessian as the reference's solve() does */
    for (u64 i = 0; i < nterms; ++i) coeff[i] += step[i];
    compute_gradhyp = true; compute_gradpara = true;
    update(std::vector<double>(coeff));
    compute_gradhyp = false; compute_gradpara = false;
  }

  /* lpdf::optcg, fit.cpp:37-96.  The K-length algebra runs on the host in the
   * reference's order (Armadillo's two-accumulator accu); update/hessmult are the GPU. */
  virtual void optcg(double tol, u64 maxepch) {
    fullhess = false;
    compute_val = true; compute_grad = true; compute_gradhyp = false; compute_gradpara = false;
    if (coeff.size() != nterms) coeff.assign(nterms, 0.0);
    update(std::vector<double>(coeff));
    std::vector<double> m = diaghess();
    cg_iters = 0;
    if (!all_finite(m) && !all_finite(grad)) { val = -std::numeric_limits<double>::infinity(); return; }
    const u64 K = nterms;
    std::vector<double> rm(K), t(K);
    for (u64 i = 0; i < K; ++i) rm[i] = grad[i] / m[i];
    std::vector<double> p = rm;
    std::vector<double> q = hessmult(p);
    double num = 0, beta = 0, denom = 1, alpha = 0, num2 = 0, valo = val, valdiff = 10;
    u64 k;
    for (k = 0; k < maxepch; k++) {
      for (u64 i = 0; i < K; ++i) t[i] = grad[i] * rm[i];
      num = obh::sum2(t.data(), K);
      if (num < tol && valdiff < tol) break;
      for (u64 i = 0; i < K; ++i) t[i] = q[i] * p[i];
      denom = obh::sum2(t.data(), K);
      alpha = num / denom;
      for (u64 i = 0; i < K; ++i) coeff[i] += alpha * p[i];
      valo = val;
      update(std::vector<double>(coeff));
      valdiff = val - valo;
      for (u64 i = 0; i < K; ++i) rm[i] = grad[i] / m[i];
      for (u64 i = 0; i < K; ++i) t[i] = (alpha * q[i]) * rm[i];
      num2 = -obh::sum2(t.data(), K);
      beta = num2 / num;
      for (u64 i = 0; i < K; ++i) p[i] = rm[i] + beta * p[i];
      q = hessmult(p);
    }
    cg_iters = k;
    compute_gradhyp = true; compute_gradpara = true;
    update(std::vector<double>(coeff));
    compute_gradhyp = false; compute_gradpara = false;
  }
};

struct LogprGauss : Lpdf { /* logpr_gauss.cpp:41-145 */
  const OuterMod* om;
  std::vector<double> coeffsd, coefflvarge, stdresid;
  double sca = 1;
  LogprGauss(const OuterMod* om_, const u64* t, u64 K) : om(om_) {
    d = om->d; npara = 1;
    terms.assign(t, t + K * d);
    para0 = {6}; paravar = {4};
    nterms = K;
    para = para0;
    sca = std::exp(para[0]);
    updateom();
  }
  void updateom() override {
    coeffsd.resize(nterms);
    om->getvar(terms.data(), nterms, coeffsd.data());
    for (double& v : coeffsd) v = std::sqrt(v);
    coefflvarge.resize(nterms * om->nhyp());
    om->getlvar_gradhyp(terms.data(), nterms, coefflvarge.data());
  }
  void updatepara(const double* p, u64 n) override { para.assign(p, p + n); sca = std::exp(para[0]); }
  void updateterms(const u64* t, u64 K) override { terms.assign(t, t + K * d); nterms = K; updateom(); }
  void update(const std::vector<double>& c) override {
    coeff = c;
    const u64 K = coeff.size(), H = om->nhyp();
    stdresid.resize(K);
    for (u64 i = 0; i < K; ++i) stdresid[i] = coeff[i] / (coeffsd[i] * sca);
    std::vector<double> t(K), t2(K);
    if (compute_val) {
      for (u64 i = 0; i < K; ++i) { t[i] = stdresid[i] * stdresid[i]; t2[i] = std::log(coeffsd[i] * sca); }
      val = -0.5 * obh::sum2(t.data(), K) - obh::sum2(t2.data(), K);
    }
    if (compute_gradhyp) {
      gradhyp.assign(H, 0.0);
      for (u64 i = 0; i < K; ++i) t[i] = stdresid[i] * stdresid[i] - 1;
      for (u64 h = 0; h < H; ++h) {
        double s1 = 0, s2 = 0;
        u64 j;
        const double* g = coefflvarge.data() + h * K;
        for (j = 1; j < K; j += 2) { s1 += (0.5 * g[j - 1]) * t[j - 1]; s2 += (0.5 * g[j]) * t[j]; }
        if ((j - 1) < K) s1 += (0.5 * g[j - 1]) * t[j - 1];
        gradhyp[h] = s1 + s2;
      }
    }
    if (compute_gradpara) {
      for (u64 i = 0; i < K; ++i) t[i] = stdresid[i] * stdresid[i];
      gradpara = {obh::sum2(t.data(), K) - double(coeffsd.size())};
    }
    if (compute_grad) {
      grad.resize(K);
      for (u64 i = 0; i < K; ++i) grad[i] = -1. * stdresid[i] / (coeffsd[i] * sca);
    }
  }
  std::vector<double> hessmult(const std::vector<double>& g) override {
    std::vector<double> o(g.size());
    for (u64 i = 0; i < g.size(); ++i) { const double s = coeffsd[i] * sca; o[i] = g[i] / (s * s); }
    return o;
  }
  std::vector<double> diaghess() override {
    std::vector<double> o(coeffsd.size());
    for (u64 i = 0; i < o.size(); ++i) { const double s = coeffsd[i] * sca; o[i] = 1. / (s * s); }
    return o;
  }
  std::vector<double> diaghessgradhyp() override {
    std::vector<double> o = coefflvarge;
    const u64 K = nterms, H = om->nhyp();
    for (u64 h = 0; h < H; ++h) for (u64 i = 0; i < K; ++i) { const double s = coeffsd[i] * sca; o[i + h * K] = -(o[i + h * K] / (s * s)); }
    return o;
  }
  bool can_diaghessgradhyp_dot() const override { return true; }
  bool diaghessgradhyp_dot(const std::vector<double>& c, std::vector<double>& out) override {
    const u64 K = nterms, H = om->nhyp();
    if (c.size() != K) return false;
    const std::vector<double> m = diaghessgradhyp();
    out.assign(H, 0.0);
    std::vector<double> t(K);
    for (u64 h = 0; h < H; ++h) {
      for (u64 i = 0; i < K; ++i) t[i] = m[i + h * K] * c[i];
      out[h] = obh::sum2(t.data(), K);
    }
    return true;
  }
  std::vector<double> diaghessgradpara() override {
    std::vector<double> o(nterms);
    for (u64 i = 0; i < nterms; ++i) { const double s = coeffsd[i] * sca; o[i] = -2. / (s * s); }
    return o;
  }
  /* hess / hessgradhyp / hessgradpara, logpr_gauss.cpp:153-186: the diagonal forms on the diagonal of K x K slices */
  static std::vector<double> on_diagonals(const std::vector<double>& dg, u64 K) {
    const u64 S = K ? dg.size() / K : 0;
    std::vector<double> o(K * K * S, 0.0);
    for (u64 s = 0; s < S; ++s) for (u64 i = 0; i < K; ++i) o[i + i * K + s * K * K] = dg[i + s * K];
    return o;
  }
  std::vector<double> hess() override { return on_diagonals(diaghess(), nterms); }
  std::vector<double> hessgradhyp() override { return on_diagonals(diaghessgradhyp(), nterms); }
  std::vector<double> hessgradpara() override { return on_diagonals(diaghessgradpara(), nterms); }
  u64 nhyp() const override { return om->nhyp(); }
};

[[noreturn]] inline void refuse_multi(const char* what) {
  throw std::invalid_argument(std::string(what) + " is not available for multi-response objects");
}
/* K x S -> (K C) x S: each length-K column repeated C times */
inline std::vector<double> tile_cols(const std::vector<double>& v, u64 K, u64 C) {
  const u64 S = K ? v.size() / K : 0;
  std::vector<double> o(K * C * S);
  for (u64 s = 0; s < S; ++s)
    for (u64 c = 0; c < C; ++c) std::copy(v.begin() + s * K, v.begin() + (s + 1) * K, o.begin() + (s * C + c) * K);
  return o;
}

/* A likelihood on C responses observed at the same rows that LpdfVec::optcg_device can drive: y, yhat and w are ld x C
 * on the device (pad rows zero), the update and the Hessian product run on the device (update_dev / hessmult_dev:
 * coefficients in, the likelihood part of grad or of the Hessian product in red[0 .. K C), nothing crosses to the host),
 * val_col(c) is column c's value of the last host update, and cg_params fills the likelihood's fields of the CG stage
 * kernel (its noise scale, and the device array of per-column sums of squared residuals for C columns). */
struct DevLik : Lpdf {
  Ctx& ctx;
  const OuterMod* om;
  OuterBase ob;
  std::vector<double> x_host; /* kept for predictor(loglik), loglik_gauss.cpp:198 */
  u64 N = 0, K = 0, C = 1;
  DevBuf<double> y, yhat, w, kbuf, red;
  std::vector<double> ssq_host; /* per-column sums of squared standardised residuals of the last update (all ranks) */

  DevLik(Ctx& c, const OuterMod* om_, const u64* t, u64 K_, const double* yh /* N x C */, u64 C_, const double* xh, u64 N_)
      : ctx(c), om(om_), ob(c, om_, xh, N_, true, t, K_), N(N_), K(K_), C(C_) {
    if (C == 0) throw std::invalid_argument("ncol must be at least 1");
    d = om->d;
    terms.assign(t, t + K * d);
    nterms = K * C;
    x_host.assign(xh, xh + N * d);
    const u64 ld = ob.ld;
    y.ensure(ld * C);
    OB_CUDA(cudaMemsetAsync(y.p, 0, ld * C * sizeof(double), ctx.stream));
    for (u64 j = 0; j < C; ++j)
      if (N) OB_CUDA(cudaMemcpyAsync(y.p + j * ld, yh + j * N, N * sizeof(double), cudaMemcpyHostToDevice, ctx.stream));
    yhat.ensure(ld * C); w.ensure(ld * C);
    ctx.sync();
  }
  static double arma_var(const double* x, u64 n) {
    if (n < 2) return 0.0;
    const double mean = obh::sum2(x, n) / double(n);
    double a2 = 0, a3 = 0;
    u64 i, j;
    for (i = 0, j = 1; j < n; i += 2, j += 2) { const double ti = mean - x[i], tj = mean - x[j]; a2 += ti * ti + tj * tj; a3 += ti + tj; }
    if (i < n) { const double ti = mean - x[i]; a2 += ti * ti; a3 += ti; }
    return (a2 - a3 * a3 / double(n)) / double(n - 1);
  }
  u64 ncol() const override { return C; }
  u64 nhyp() const override { return ob.H; }
  u64 nrow() const override { return N; }
  void setnthreads(int k) override { ob.nthreads = k; }
  virtual void update_dev(const double* coeff_dev) = 0;
  virtual void hessmult_dev(const double* g_dev) = 0;
  virtual double val_col(u64 c) const = 0;
  virtual void cg_params(obd::CgParams& c) const = 0;
};

/* loglik_gauss (loglik_gauss.cpp:41-179) on C responses observed at the same rows (C = 1: loglik_gauss itself), all but
 * the products.  Every column is the single-response model on its own response; the columns share the basis, the terms
 * table, the hyper-parameters and the para entry.  val, gradhyp and gradpara are the sums over the columns (in column
 * order) of what the single-response object returns at that column, grad is K x C, and the Hessian diagonals, which do
 * not depend on the response, are computed once and repeated C times.  With C = 1 every formula is the reference's
 * own.  The subclasses are the two paths of the products: LoglikGauss (one vector, fused epilogues) and
 * LoglikGaussMulti (matrix products over the columns).
 * percol (para per column, multi-response only): npara = C, para[c] is column c's noise log-sd with loglik_gauss's
 * default on that column; gradpara[c] is column c's own, and the Hessian diagonals are the one K-vector of squared
 * column sums scaled by each column's exp(-2 para[c]) (diaghessgradpara: (K C) x C, block-diagonal). */
struct LoglikGaussBase : DevLik {
  double Nglobal = 0;
  double obssd = 1;
  bool percol = false;
  std::vector<double> obssd_cols; /* C: column c's noise sd, exp(para[c]) (percol) or obssd */
  DevBuf<double> ones;
  std::vector<double> sqcs;      /* the last sqcolsums(); empty after updateom / updateterms */

  LoglikGaussBase(Ctx& c, const OuterMod* om_, const u64* t, u64 K_, const double* yh /* N x C */, u64 C_, const double* xh, u64 N_,
                  bool percol_ = false)
      : DevLik(c, om_, t, K_, yh, C_, xh, N_), percol(percol_) {
    npara = 1;
    /* para0 = log(0.01 * mean over the columns of var(y[:,c])), loglik_gauss.cpp:48 (Armadillo two-pass var); over ALL
     * ranks' rows */
    std::vector<double> var(C);
    if (ctx.nranks > 1) {
      std::vector<double> st(C + 1, 0.0), ss(C, 0.0);
      st[0] = double(N);
      for (u64 j = 0; j < C; ++j) for (u64 i = 0; i < N; ++i) st[1 + j] += yh[i + j * N];
      allreduce_host(st.data(), C + 1);
      Nglobal = st[0];
      for (u64 j = 0; j < C; ++j) {
        const double mean = st[1 + j] / st[0];
        for (u64 i = 0; i < N; ++i) ss[j] += (yh[i + j * N] - mean) * (yh[i + j * N] - mean);
      }
      allreduce_host(ss.data(), C);
      for (u64 j = 0; j < C; ++j) var[j] = ss[j] / (Nglobal - 1);
    } else {
      Nglobal = double(N);
      for (u64 j = 0; j < C; ++j) var[j] = arma_var(yh + j * N, N);
    }
    if (percol) { /* column c: loglik_gauss's own default on Y[:,c] */
      npara = C;
      para0.resize(C);
      for (u64 j = 0; j < C; ++j) para0[j] = std::log(0.01 * var[j]);
      paravar.assign(C, 1.0);
    } else {
      double vs = 0;
      for (double v : var) vs += v;
      para0 = {std::log(0.01 * (vs / double(C)))};
      paravar = {1};
    }
    para = para0;
    set_sds();
  }
  /* column c's entry of para */
  double para_col(u64 c) const { return para[percol ? c : 0]; }
  void set_sds() {
    obssd = std::exp(para[0]);
    obssd_cols.resize(C);
    for (u64 c = 0; c < C; ++c) obssd_cols[c] = percol ? std::exp(para[c]) : obssd;
  }
  void allreduce_host(double* v, u64 n) {
    red.upload(v, n, ctx.stream);
    ctx.allreduce_sum(red.p, n);
    OB_CUDA(cudaMemcpyAsync(v, red.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx.stream));
    ctx.sync();
  }
  void updateom() override { ob.build(); sqcs.clear(); }
  bool para_per_column() const override { return percol; }
  void updatepara(const double* p, u64 n) override {
    if (percol && n != C) throw std::range_error("para must have one entry per column");
    para.assign(p, p + n);
    set_sds();
  }
  void updateterms(const u64* t, u64 K_) override { terms.assign(t, t + K_ * d); K = K_; nterms = K * C; sqcs.clear(); }
  /* columns of the predictive variance of a predictor made from this likelihood now (PredGauss) */
  u64 predvar_ncol() const { return multi() && (percol || totdiaghess_percol) ? C : 1; }
  double val_col(u64 c) const override { return -0.5 * ssq_host[c] - Nglobal * std::log(obssd_cols[c]); }
  void cg_params(obd::CgParams& c) const override { c.obssd = obssd; c.nglobal = Nglobal; }
  /* val and gradpara of update() from ssq_host, loglik_gauss.cpp:121-129 */
  void set_val_gradpara() {
    if (compute_val) { val = 0; for (u64 c = 0; c < C; ++c) val += val_col(c); }
    if (compute_grad && compute_gradpara) {
      if (percol) { gradpara.resize(C); for (u64 c = 0; c < C; ++c) gradpara[c] = ssq_host[c] - Nglobal; }
      else { gradpara = {0.0}; for (u64 c = 0; c < C; ++c) gradpara[0] += ssq_host[c] - Nglobal; }
    }
  }

  /* device forms (DevLik), stream ordered, summed over ranks; update_dev also leaves each column's sum of squared
   * standardised residuals on the device */
  std::vector<double> hessmult(const std::vector<double>& g) override { /* :137-145 */
    if (g.size() != K * C) throw std::range_error("g must have K x ncol entries");
    kbuf.upload(g, ctx.stream);
    hessmult_dev(kbuf.p);
    std::vector<double> o(K * C);
    ob.d2h(o.data(), red.p, K * C);
    return o;
  }

  const double* ones_dev() {
    if (ones.cap < ob.ld) { ones.ensure(ob.ld); obd::launch_fill(ctx, ones.p, ob.ld, 1.0); }
    return ones.p;
  }
  /* the squared column sums Phi^2^T 1 (K), summed over ranks; kept in sqcs (they depend on the basis and the terms
   * table only, not on para) */
  std::vector<double> sqcolsums() {
    red.ensure(K);
    ob.tmm_dev(terms.data(), K, 1, ones_dev(), red.p);
    sqcs.resize(K);
    ob.d2h(sqcs.data(), red.p, K);
    return sqcs;
  }
  /* (K C) x S from a K x S matrix: column block c scaled by exp(-2 para_c) (shared para: the same block repeated) */
  std::vector<double> scale_cols(const std::vector<double>& v) const {
    const u64 S = K ? v.size() / K : 0;
    std::vector<double> o(K * C * S);
    for (u64 c = 0; c < C; ++c) {
      const double sc = std::exp(-2 * para_col(c));
      for (u64 s = 0; s < S; ++s) for (u64 i = 0; i < K; ++i) o[(s * C + c) * K + i] = sc * v[s * K + i];
    }
    return o;
  }
  std::vector<double> diaghess() override { return scale_cols(sqcolsums()); } /* :154-157 */
  std::vector<double> diaghessgradpara() override { /* :176-179 */
    std::vector<double> lh = diaghess();
    for (double& v : lh) v = -2 * v;
    if (!percol) return lh;
    std::vector<double> o(K * C * C, 0.0); /* block-diagonal: para c moves column c only */
    for (u64 c = 0; c < C; ++c) std::copy(lh.begin() + c * K, lh.begin() + (c + 1) * K, o.begin() + c * K * C + c * K);
    return o;
  }
  /* out[c] = sum_k diaghessgradpara[k, c] / dh[k] over column c's block, without the (K C) x C matrix; reuses the
   * squared column sums of the diaghess() that formed dh (lpdfvec's buildhess) */
  bool diaghessgradpara_dot(const std::vector<double>& dh, std::vector<double>& out) override {
    if (!percol || dh.size() != K * C) return false;
    const std::vector<double> lh = sqcs.size() == K ? sqcs : sqcolsums();
    out.assign(C, 0.0);
    std::vector<double> t(K);
    for (u64 c = 0; c < C; ++c) {
      const double sc = std::exp(-2 * para[c]);
      for (u64 i = 0; i < K; ++i) t[i] = -2 * (sc * lh[i]) / dh[c * K + i];
      out[c] = obh::sum2(t.data(), K);
    }
    return true;
  }
  std::vector<double> diaghessgradhyp() override { /* :165-168 */
    const u64 H = ob.H;
    red.ensure(K * (1 + H));
    ob.tmm_ge_dev(terms.data(), K, 1, ones_dev(), red.p);
    std::vector<double> all(K * (1 + H));
    ob.d2h(all.data(), red.p, K * (1 + H));
    return scale_cols(std::vector<double>(all.begin() + K, all.end()));
  }
  bool can_diaghessgradhyp_dot() const override { return ctx.dsweep; }
  /* sum_k c_k sum_n d(Phi^2)[n,k]/dhyp = sum_n d(Phi^2 c)[n]/dhyp: the hyper-gradient sweep on the squared operator.
   * Linear in c: the columns' weights (each scaled by its exp(-2 para_c) when para is per column) are summed first, then
   * ONE sweep.  The swept / not-swept decision is COLLECTIVE:
   * slot H of the reduction buffer counts the ranks whose sweep was unavailable (module build failure, table not
   * specialised, geometry), so every rank takes the same branch and the allreduce sequence stays aligned (the fallback
   * is a K*(1+H) allreduce in diaghessgradhyp()). */
  bool diaghessgradhyp_dot(const std::vector<double>& cv, std::vector<double>& out) override {
    const u64 H = ob.H;
    if (!ctx.dsweep || cv.size() != K * C || H == 0) return false;
    std::vector<double> s(K, 0.0);
    if (percol) /* each column's weights scaled by its own exp(-2 para_c); the result is then not scaled again */
      for (u64 c = 0; c < C; ++c) {
        const double sc = std::exp(-2 * para[c]);
        for (u64 i = 0; i < K; ++i) s[i] += sc * cv[c * K + i];
      }
    else /* shared para: plain sums, scaled once after the sweep */
      for (u64 c = 0; c < C; ++c) for (u64 i = 0; i < K; ++i) s[i] += cv[c * K + i];
    kbuf.upload(s, ctx.stream);
    red.ensure(H + 1);
    OB_CUDA(cudaMemsetAsync(red.p, 0, (H + 1) * sizeof(double), ctx.stream));
    bool done = false;
    try { done = ob.gradhyp_sweep(terms.data(), K, 1, kbuf.p, nullptr, red.p); } catch (const std::exception&) { done = false; }
    ctx.sync(); /* s must outlive the upload */
    if (ctx.nranks > 1) {
      if (!done) obd::launch_fill(ctx, red.p, H + 1, 0.0), obd::launch_fill(ctx, red.p + H, 1, 1.0);
      ctx.allreduce_sum(red.p, H + 1);
    } else if (!done) return false;
    std::vector<double> r(H + 1);
    ob.d2h(r.data(), red.p, H + 1);
    if (r[H] != 0.0) return false; /* some rank could not sweep: all ranks fall back together */
    out.assign(r.begin(), r.begin() + H);
    if (percol) return true;
    const double sc = std::exp(-2 * para[0]);
    for (double& v : out) v = sc * v;
    return true;
  }
};

/* the single-response path: Phi a and Phi^T w each ONE launch with the residual epilogues fused (PHI_UPDATE /
 * PHI_HESS), the sum of squared residuals reduced alongside the gradient */
struct LoglikGauss : LoglikGaussBase {
  std::vector<double> yhat_host;
  bool yhat_valid = false;

  LoglikGauss(Ctx& c, const OuterMod* om_, const u64* t, u64 K_, const double* yh, const double* xh, u64 N_)
      : LoglikGaussBase(c, om_, t, K_, yh, 1, xh, N_) {}

  void update(const std::vector<double>& c) override { /* loglik_gauss.cpp:110-130 */
    coeff = c;
    const u64 H = ob.H;
    if (c.size() != K) throw std::range_error("coeff must have one entry per term");
    kbuf.upload(coeff, ctx.stream);
    obd::PhiAArgs a;
    a.a = kbuf.p; a.out = yhat.p; a.w = w.p; a.y = y.p; a.sd = obssd; a.mode = obd::PHI_UPDATE;
    int grid = 0;
    ob.phi_a(terms.data(), K, 0, a, &grid);
    yhat_valid = false;
    /* reduction buffer: [grad (K) | ssq | gradhyp (H)] -> one allreduce */
    red.ensure(K + 1 + H);
    OB_CUDA(cudaMemsetAsync(red.p, 0, (K + 1 + H) * sizeof(double), ctx.stream));
    if (grid > 0) obd::launch_sum_partials(ctx, ob.ws.ssq.p, grid, red.p + K);
    if (compute_grad) ob.phi_t(terms.data(), K, 0, w.p, red.p);
    if (compute_grad && compute_gradhyp) ob.gradhyp_dots(terms.data(), K, coeff, kbuf.p, w.p, yhat.p, red.p + K + 1); /* :127 */
    ctx.allreduce_sum(red.p, K + 1 + H);
    std::vector<double> r(K + 1 + H);
    ob.d2h(r.data(), red.p, K + 1 + H);
    ssq_host.assign(1, r[K]);
    set_val_gradpara();
    if (compute_grad) {
      grad.assign(r.begin(), r.begin() + K);
      if (compute_gradhyp) gradhyp.assign(r.begin() + K + 1, r.end());
    }
  }
  /* red[K] = sum of squared standardised residuals, riding on the tail of the Phi^T launch (loglik_gauss.cpp:110-125) */
  void update_dev(const double* coeff_dev) override {
    obd::PhiAArgs a;
    a.a = coeff_dev; a.out = yhat.p; a.w = w.p; a.y = y.p; a.sd = obssd; a.mode = obd::PHI_UPDATE;
    int grid = 0;
    ob.phi_a(terms.data(), K, 0, a, &grid);
    yhat_valid = false;
    red.ensure(K + 2);
    bool fused;
    {
      obd::Ctx::FuseScope fuse(ctx, K + 1, ob.ws.ssq.p, grid);
      ob.phi_t(terms.data(), K, 0, w.p, red.p);
      fused = ctx.fused; ctx.fused = false;
    }
    if (!ctx.extra_done) {
      if (grid > 0) obd::launch_sum_partials(ctx, ob.ws.ssq.p, grid, red.p + K);
      else OB_CUDA(cudaMemsetAsync(red.p + K, 0, sizeof(double), ctx.stream));
    }
    if (!fused) ctx.allreduce_sum(red.p, K + 1);
  }
  void hessmult_dev(const double* g_dev) override { /* :137-145 */
    obd::PhiAArgs a;
    a.a = g_dev; a.w = w.p; a.sd = obssd; a.mode = obd::PHI_HESS;
    ob.phi_a(terms.data(), K, 0, a, nullptr);
    red.ensure(K + 2);
    obd::Ctx::FuseScope fuse(ctx, K);
    ob.phi_t(terms.data(), K, 0, w.p, red.p);
    ctx.allreduce_after(red.p, K);
  }
  const std::vector<double>& get_yhat() {
    if (!yhat_valid) { yhat_host.resize(N); ob.d2h(yhat_host.data(), yhat.p, N); yhat_valid = true; }
    return yhat_host;
  }
};

/* loglik_gda (src/lpdfs/loglik_gda.cpp:47-239): the stage-1 likelihood of obfit, built on a <= 3*numb-row subsample
 * (R/fitting.R:79-84).  Every Phi-type product runs on the GPU kernels through the outerbase operators; the
 * N-vector bookkeeping around them (per-row noise scale and its derivatives) follows the reference on the host. */
/* loglik_std, src/lpdfs/loglik_std.cpp:41-203: loglik_gauss's model (same value, gradients, Hessian products and
 * diagonals -- the formulas of :100-165 are loglik_gauss.cpp:110-179's) plus the full K x K Hessian that lpdf::optnewton
 * and the full branch of lpdfvec::buildhess need.  The reference keeps the explicit N x K basis and its N x K x H cube
 * for everything; here only the Hessians touch explicit matrices, and they are contractions over the rows on the FP64
 * tensor cores: hess = Phi^T . getmat (tprodmm_(mat) with K right-hand sides, phi_tm_spec), one more per
 * hyper-parameter for hessgradhyp.  Rows sharded over ranks like loglik_gauss (the products sum over ranks). */
struct LoglikStd : LoglikGauss {
  DevBuf<double> basis, hbuf;
  LoglikStd(Ctx& c, const OuterMod* om_, const u64* t, u64 K, const double* yh, const double* xh, u64 N_)
      : LoglikGauss(c, om_, t, K, yh, xh, N_) {}
  /* Phi^T . M for an explicit ld x K matrix M in `basis`; K x K on the host */
  std::vector<double> gram(int h) {
    const u64 K = nterms;
    basis.ensure(ob.ld * std::max<u64>(K, 1));
    hbuf.ensure(K * K + 1);
    ob.getmat_dev(terms.data(), K, h, basis.p);
    ob.tmm_mat_dev(terms.data(), K, 0, basis.p, ob.ld, K, hbuf.p);
    std::vector<double> o(K * K);
    ob.d2h(o.data(), hbuf.p, K * K);
    return o;
  }
  std::vector<double> hess() override { /* :173-176 */
    const u64 K = nterms;
    std::vector<double> g = gram(-1), o(K * K);
    const double c = std::exp(-2 * para[0]);
    /* Phi^T Phi is symmetric; the kernel's (i, j) and (j, i) differ in the last bit (one side is recomputed) */
    for (u64 j = 0; j < K; ++j) for (u64 i = 0; i < K; ++i) o[i + j * K] = c * (0.5 * (g[i + j * K] + g[j + i * K]));
    return o;
  }
  std::vector<double> hessgradhyp() override { /* :183-195 */
    const u64 K = nterms, H = ob.H;
    std::vector<double> o(K * K * H);
    const double c = std::exp(-2 * para[0]);
    for (u64 h = 0; h < H; ++h) {
      const std::vector<double> g = gram((int)h);
      for (u64 j = 0; j < K; ++j) for (u64 i = 0; i < K; ++i) o[i + j * K + h * K * K] = c * g[i + j * K] + c * g[j + i * K];
    }
    return o;
  }
  std::vector<double> hessgradpara() override { /* :202-206 */
    std::vector<double> o = hess();
    for (double& v : o) v = -2 * v;
    return o;
  }
};

/* loglik_gda's per-row noise sd and the host work that depends on it only, not on the response (shared by LoglikGda and
 * LoglikGdaMulti): the sd's derivatives (loglik_gda.cpp:226-235) and the Hessian diagonals (:172-211), all K- or
 * N-sized on the host around the GPU products, in the reference's operation order */
struct GdaSd {
  std::vector<double> obssd, obssd_gradhyp, obssd_gradpara;
  /* from obssd and rterms = residvar (read only with doda) */
  void sd_grads(OuterBase& ob, const u64* terms, u64 K, const std::vector<double>& para, bool doda, const std::vector<double>& rterms) {
    const u64 N = obssd.size(), H = ob.H;
    if (doda) {
      obssd_gradhyp.resize(N * H);
      ob.residvar_gradhyp(terms, K, obssd_gradhyp.data());
      for (u64 h = 0; h < H; ++h)
        for (u64 i = 0; i < N; ++i) obssd_gradhyp[i + h * N] *= (std::exp(2 * para[1]) * 0.5) / obssd[i];
    }
    obssd_gradpara.assign(N * 2, 0.0);
    for (u64 i = 0; i < N; ++i) {
      obssd_gradpara[i] = std::exp(2 * para[0]) / obssd[i];
      obssd_gradpara[i + N] = doda ? std::exp(2 * para[1]) * rterms[i] / obssd[i] : 0.0;
    }
  }
  std::vector<double> gda_diaghess(OuterBase& ob, const u64* terms, u64 K) const { /* :172-175 */
    const u64 N = obssd.size();
    std::vector<double> t(N), o(K);
    for (u64 i = 0; i < N; ++i) t[i] = 1 / (obssd[i] * obssd[i]);
    ob.tmm(1, terms, K, t.data(), o.data());
    return o;
  }
  std::vector<double> gda_diaghessgradhyp(OuterBase& ob, const u64* terms, u64 K, bool doda) const { /* :182-196 */
    const u64 N = obssd.size(), H = ob.H;
    std::vector<double> temp(N), lh(K * H);
    for (u64 i = 0; i < N; ++i) temp[i] = 1 / (obssd[i] * obssd[i]);
    ob.tmm_gradhyp(1, terms, K, temp.data(), nullptr, lh.data());
    for (u64 i = 0; i < N; ++i) temp[i] *= -2 / obssd[i];
    if (doda) {
      std::vector<double> t2(obssd_gradhyp), add(K * H);
      for (u64 h = 0; h < H; ++h)
        for (u64 i = 0; i < N; ++i) t2[i + h * N] *= temp[i];
      ob.tmm_mat(1, terms, K, t2.data(), H, add.data());
      for (u64 i = 0; i < K * H; ++i) lh[i] += add[i];
    }
    return lh;
  }
  std::vector<double> gda_diaghessgradpara(OuterBase& ob, const u64* terms, u64 K) const { /* :203-211 */
    const u64 N = obssd.size();
    std::vector<double> t2(obssd_gradpara), o(K * 2);
    for (u64 q = 0; q < 2; ++q)
      for (u64 i = 0; i < N; ++i) t2[i + q * N] *= (1 / (obssd[i] * obssd[i])) * (-2 / obssd[i]);
    ob.tmm_mat(1, terms, K, t2.data(), 2, o.data());
    return o;
  }
  /* Armadillo's two-accumulator dot */
  static double dot2(const double* a, const double* b, u64 n) {
    double s1 = 0, s2 = 0;
    u64 j;
    for (j = 1; j < n; j += 2) { s1 += a[j - 1] * b[j - 1]; s2 += a[j] * b[j]; }
    if ((j - 1) < n) s1 += a[j - 1] * b[j - 1];
    return s1 + s2;
  }
};

struct LoglikGda : Lpdf, GdaSd {
  Ctx& ctx;
  const OuterMod* om;
  OuterBase ob;
  std::vector<double> x_host, y;
  u64 N = 0;
  bool doda = true, redostd = true;
  std::vector<double> yhat, yhatge, residtemp, residtemp2;

  LoglikGda(Ctx& c, const OuterMod* om_, const u64* t, u64 K, const double* yh, const double* xh, u64 N_)
      : ctx(c), om(om_), ob(c, om_, xh, N_, true, t, K), N(N_) {
    if (ctx.nranks > 1) throw std::logic_error("loglik_gda is the single-rank subsample model of obfit stage 1");
    d = om->d; npara = 2;
    terms.assign(t, t + K * d);
    nterms = K;
    x_host.assign(xh, xh + N * d);
    y.assign(yh, yh + N);
    para0 = {0.5 * std::log(0.01 * DevLik::arma_var(yh, N)), 0.0};
    paravar = {4, 4};
    para = para0;
    buildstd();
  }
  void setnthreads(int k) override { ob.nthreads = k; }
  void updateom() override { ob.build(); if (doda) redostd = true; }
  void updatepara(const double* p, u64 n) override { para.assign(p, p + n); redostd = true; }
  void updateterms(const u64* t, u64 K) override { terms.assign(t, t + K * d); nterms = K; if (doda) redostd = true; }
  void buildstd() { /* :217-236 */
    if (redostd) {
      const u64 K = nterms;
      std::vector<double> rterms(N);
      ob.residvar(terms.data(), K, rterms.data());
      obssd.resize(N);
      for (u64 i = 0; i < N; ++i) {
        double v = std::exp(2 * para[0]);
        if (doda) v += std::exp(2 * para[1]) * rterms[i];
        obssd[i] = std::sqrt(v);
      }
      sd_grads(ob, terms.data(), K, para, doda, rterms);
    }
    redostd = false;
  }
  void update(const std::vector<double>& c) override { /* :116-149 */
    coeff = c;
    const u64 K = nterms, H = ob.H;
    if (c.size() != K) throw std::range_error("coeff must have one entry per term");
    yhat.resize(N);
    if (compute_gradhyp) { yhatge.resize(N * H); ob.mm_gradhyp(0, terms.data(), K, coeff.data(), yhat.data(), yhatge.data()); }
    else ob.mm(0, terms.data(), K, coeff.data(), yhat.data());
    buildstd();
    residtemp.resize(N); residtemp2.resize(N);
    for (u64 i = 0; i < N; ++i) { residtemp[i] = (yhat[i] - y[i]) / obssd[i]; residtemp2[i] = residtemp[i] * residtemp[i]; }
    if (compute_val) {
      std::vector<double> t(N);
      for (u64 i = 0; i < N; ++i) t[i] = std::log(obssd[i]);
      val = -0.5 * obh::sum2(residtemp2.data(), N) - obh::sum2(t.data(), N);
    }
    if (compute_grad) {
      std::vector<double> inv(N);
      for (u64 i = 0; i < N; ++i) { residtemp[i] = -1. * (residtemp[i] / obssd[i]); residtemp2[i] /= obssd[i]; inv[i] = 1 / obssd[i]; }
      grad.resize(K);
      ob.tmm(0, terms.data(), K, residtemp.data(), grad.data());
      if (compute_gradhyp) {
        gradhyp.assign(H, 0.0);
        for (u64 h = 0; h < H; ++h) {
          gradhyp[h] = dot2(residtemp.data(), yhatge.data() + h * N, N);
          if (doda) {
            gradhyp[h] += dot2(residtemp2.data(), obssd_gradhyp.data() + h * N, N);
            gradhyp[h] -= dot2(inv.data(), obssd_gradhyp.data() + h * N, N);
          }
        }
      }
      if (compute_gradpara) {
        gradpara.assign(2, 0.0);
        for (u64 q = 0; q < 2; ++q) {
          gradpara[q] = dot2(residtemp2.data(), obssd_gradpara.data() + q * N, N);
          gradpara[q] -= dot2(inv.data(), obssd_gradpara.data() + q * N, N);
        }
      }
    }
  }
  std::vector<double> hessmult(const std::vector<double>& g) override { /* :156-164 */
    const u64 K = nterms;
    std::vector<double> yt(N), o(K);
    ob.mm(0, terms.data(), K, g.data(), yt.data());
    for (u64 i = 0; i < N; ++i) { yt[i] /= obssd[i]; yt[i] /= obssd[i]; }
    ob.tmm(0, terms.data(), K, yt.data(), o.data());
    return o;
  }
  std::vector<double> diaghess() override { return gda_diaghess(ob, terms.data(), nterms); }
  std::vector<double> diaghessgradhyp() override { return gda_diaghessgradhyp(ob, terms.data(), nterms, doda); }
  std::vector<double> diaghessgradpara() override { return gda_diaghessgradpara(ob, terms.data(), nterms); }
  u64 nhyp() const override { return ob.H; }
  u64 nrow() const override { return N; }
};

/* ------------------------------------------------------------------ multi-response: C responses observed at the same rows
 * Every column is the single-response model on its own response, all columns share the basis, the terms table, the
 * hyper-parameters and both para entries (or, opted in per object, one para entry per column: its own noise scale or
 * coefficient scale).  val, gradhyp and gradpara are the sums over the columns (in column order) of what the
 * single-response object returns at that column, grad is K x C, the Hessian product is block-diagonal and the Hessian
 * diagonals are the single-response ones repeated C times (per-column para: each column's own).  The objective is meant for lpdfvec's diagonal
 * branch and its column-batched CG (LpdfVec::optcg_device); the full Hessian, optnewton and the host optcg are refused. */

/* an independent logpr_gauss on each column, shared coeffscale; percol: npara = C, para[c] is column c's coeffscale with
 * logpr_gauss's para0 and paravar, gradpara[c] is column c's own and the Hessian diagonals are per column
 * (diaghessgradpara: (K C) x C, block-diagonal) */
struct LogprGaussMulti : Lpdf {
  LogprGauss one;
  u64 K, C;
  bool percol;
  std::vector<double> val_cols;
  LogprGaussMulti(const OuterMod* om_, const u64* t, u64 K_, u64 C_, bool percol_ = false) : one(om_, t, K_), K(K_), C(C_), percol(percol_) {
    if (C == 0) throw std::invalid_argument("ncol must be at least 1");
    d = one.d; npara = one.npara; terms = one.terms; para0 = one.para0; paravar = one.paravar; para = one.para;
    if (percol) {
      npara = C;
      para0.assign(C, one.para0[0]); paravar.assign(C, one.paravar[0]); para = para0;
    }
    nterms = K * C;
  }
  /* point `one` at column c's para (shared para: it is always there) */
  void at(u64 c) { if (percol) one.updatepara(&para[c], 1); }
  double sca_col(u64 c) const { return percol ? std::exp(para[c]) : one.sca; }
  /* (K C) x S: column c's K x S result, for every c (shared para: one result repeated) */
  template <class F> std::vector<double> per_col(F f) {
    if (!percol) return tile_cols(f(), K, C);
    std::vector<double> o;
    for (u64 c = 0; c < C; ++c) {
      at(c);
      const std::vector<double> v = f();
      const u64 S = K ? v.size() / K : 0;
      o.resize(K * C * S);
      for (u64 s = 0; s < S; ++s) std::copy(v.begin() + s * K, v.begin() + (s + 1) * K, o.begin() + (s * C + c) * K);
    }
    return o;
  }
  bool multi() const override { return true; }
  u64 ncol() const override { return C; }
  bool para_per_column() const override { return percol; }
  u64 nhyp() const override { return one.nhyp(); }
  void updateom() override { one.updateom(); }
  void updatepara(const double* p, u64 n) override {
    if (!percol) { one.updatepara(p, n); para = one.para; return; }
    if (n != C) throw std::range_error("para must have one entry per column");
    para.assign(p, p + n);
  }
  void updateterms(const u64* t, u64 K_) override { one.updateterms(t, K_); terms = one.terms; K = K_; nterms = K * C; }
  std::vector<double> column(const std::vector<double>& v, u64 c) const { return std::vector<double>(v.begin() + c * K, v.begin() + (c + 1) * K); }
  void update(const std::vector<double>& cf) override {
    if (cf.size() != K * C) throw std::range_error("coeff must have K x ncol entries");
    coeff = cf;
    one.compute_val = compute_val; one.compute_grad = compute_grad; one.compute_gradhyp = compute_gradhyp; one.compute_gradpara = compute_gradpara;
    if (compute_val) { val = 0; val_cols.assign(C, 0.0); }
    if (compute_grad) grad.assign(K * C, 0.0);
    if (compute_gradhyp) gradhyp.assign(one.nhyp(), 0.0);
    if (compute_gradpara) gradpara.assign(percol ? C : 1, 0.0);
    for (u64 c = 0; c < C; ++c) {
      at(c);
      one.update(column(cf, c));
      if (compute_val) { val += one.val; val_cols[c] = one.val; }
      if (compute_grad) std::copy(one.grad.begin(), one.grad.end(), grad.begin() + c * K);
      if (compute_gradhyp) for (u64 h = 0; h < gradhyp.size(); ++h) gradhyp[h] += one.gradhyp[h];
      if (compute_gradpara) gradpara[percol ? c : 0] += one.gradpara[0];
    }
  }
  std::vector<double> hessmult(const std::vector<double>& g) override {
    if (g.size() != K * C) throw std::range_error("g must have K x ncol entries");
    std::vector<double> o(K * C);
    for (u64 c = 0; c < C; ++c) { at(c); const std::vector<double> h = one.hessmult(column(g, c)); std::copy(h.begin(), h.end(), o.begin() + c * K); }
    return o;
  }
  std::vector<double> diaghess() override { return per_col([&] { return one.diaghess(); }); }
  std::vector<double> diaghessgradhyp() override { return per_col([&] { return one.diaghessgradhyp(); }); }
  std::vector<double> diaghessgradpara() override {
    if (!percol) return tile_cols(one.diaghessgradpara(), K, C);
    std::vector<double> o(K * C * C, 0.0); /* block-diagonal: para c moves column c only */
    for (u64 c = 0; c < C; ++c) {
      at(c);
      const std::vector<double> v = one.diaghessgradpara();
      std::copy(v.begin(), v.end(), o.begin() + c * K * C + c * K);
    }
    return o;
  }
  bool diaghessgradpara_dot(const std::vector<double>& dh, std::vector<double>& out) override {
    if (!percol || dh.size() != K * C) return false;
    out.assign(C, 0.0);
    std::vector<double> t(K);
    for (u64 c = 0; c < C; ++c) {
      at(c);
      const std::vector<double> v = one.diaghessgradpara();
      for (u64 i = 0; i < K; ++i) t[i] = v[i] / dh[c * K + i];
      out[c] = obh::sum2(t.data(), K);
    }
    return true;
  }
  bool can_diaghessgradhyp_dot() const override { return true; }
  bool diaghessgradhyp_dot(const std::vector<double>& cv, std::vector<double>& out) override {
    if (cv.size() != K * C) return false;
    out.assign(one.nhyp(), 0.0);
    std::vector<double> o;
    for (u64 c = 0; c < C; ++c) {
      at(c);
      one.diaghessgradhyp_dot(column(cv, c), o);
      for (u64 h = 0; h < out.size(); ++h) out[h] += o[h];
    }
    return true;
  }
  std::vector<double> hess() override { refuse_multi("the full Hessian"); }
  std::vector<double> hessgradhyp() override { refuse_multi("the full Hessian"); }
  std::vector<double> hessgradpara() override { refuse_multi("the full Hessian"); }
  void optnewton() override { refuse_multi("optnewton"); }
  void optcg(double, u64) override { refuse_multi("optcg outside lpdfvec(logpr_gauss_multi, loglik_gauss_multi)"); }
};

/* the matrix path, also for C = 1: mm_mat_dev / tmm_mat_dev (the FP64 tensor-core kernels for C >= 8 on a specialised
 * table, else column loops) with the residual pass resid_multi between them */
struct LoglikGaussMulti : LoglikGaussBase {
  DevBuf<double> ssq, partial, gh;
  DevBuf<double> sd_dev; /* percol: obssd_cols on the device, refreshed by updatepara */

  LoglikGaussMulti(Ctx& c, const OuterMod* om_, const u64* t, u64 K_, const double* yh /* N x C */, u64 C_, const double* xh, u64 N_,
                   bool percol_ = false)
      : LoglikGaussBase(c, om_, t, K_, yh, C_, xh, N_, percol_) {
    ssq.ensure(C);
    upload_sds();
  }
  void cg_params(obd::CgParams& c) const override { LoglikGaussBase::cg_params(c); c.ssq = ssq.p; c.obssd_col = sd_cols_dev(); }
  bool multi() const override { return true; }
  void upload_sds() {
    if (!percol) return;
    sd_dev.upload(obssd_cols, ctx.stream);
    ctx.sync(); /* obssd_cols may change at the next updatepara */
  }
  void updatepara(const double* p, u64 n) override { LoglikGaussBase::updatepara(p, n); upload_sds(); }
  const double* sd_cols_dev() const { return percol ? sd_dev.p : nullptr; }

  /* ssq[c]: column c's sum of squared standardised residuals, summed over ranks */
  void update_dev(const double* coeff_dev) override {
    ob.mm_mat_dev(terms.data(), K, 0, coeff_dev, C, yhat.p, ob.ld);
    obd::launch_resid_multi(ctx, yhat.p, y.p, w.p, N, ob.ld, C, obssd, true, partial, ssq.p, sd_cols_dev());
    red.ensure(K * C);
    ob.tmm_mat_dev(terms.data(), K, 0, w.p, ob.ld, C, red.p);
    ctx.allreduce_sum(ssq.p, C);
  }
  void hessmult_dev(const double* g_dev) override { /* loglik_gauss.cpp:137-145 per column; w holds Phi g until the residual pass */
    ob.mm_mat_dev(terms.data(), K, 0, g_dev, C, w.p, ob.ld);
    obd::launch_resid_multi(ctx, w.p, nullptr, w.p, N, ob.ld, C, obssd, false, partial, nullptr, sd_cols_dev());
    red.ensure(K * C);
    ob.tmm_mat_dev(terms.data(), K, 0, w.p, ob.ld, C, red.p);
  }
  void update(const std::vector<double>& cf) override { /* loglik_gauss.cpp:110-130 per column */
    if (cf.size() != K * C) throw std::range_error("coeff must have K x ncol entries");
    coeff = cf;
    const u64 H = ob.H, ld = ob.ld;
    kbuf.upload(coeff, ctx.stream);
    update_dev(kbuf.p);
    ssq_host.resize(C);
    ob.d2h(ssq_host.data(), ssq.p, C);
    set_val_gradpara();
    if (!compute_grad) return;
    grad.resize(K * C);
    ob.d2h(grad.data(), red.p, K * C);
    if (compute_gradhyp) { /* one hyper-gradient pass per column (:127) */
      gh.ensure(std::max<u64>(H * C, 1));
      OB_CUDA(cudaMemsetAsync(gh.p, 0, std::max<u64>(H * C, 1) * sizeof(double), ctx.stream));
      for (u64 c = 0; c < C && H > 0; ++c) {
        const std::vector<double> a(coeff.begin() + c * K, coeff.begin() + (c + 1) * K);
        ob.gradhyp_dots(terms.data(), K, a, kbuf.p + c * K, w.p + c * ld, yhat.p + c * ld, gh.p + c * H);
      }
      ctx.allreduce_sum(gh.p, H * C);
      std::vector<double> r(H * C);
      ob.d2h(r.data(), gh.p, H * C);
      gradhyp.assign(H, 0.0);
      for (u64 c = 0; c < C; ++c) for (u64 h = 0; h < H; ++h) gradhyp[h] += r[c * H + h];
    }
  }
  std::vector<double> hess() override { refuse_multi("the full Hessian"); }
  std::vector<double> hessgradhyp() override { refuse_multi("the full Hessian"); }
  std::vector<double> hessgradpara() override { refuse_multi("the full Hessian"); }
  void optnewton() override { refuse_multi("optnewton"); }
  void optcg(double, u64) override { refuse_multi("optcg outside lpdfvec(logpr_gauss_multi, loglik_gauss_multi)"); }
};

/* loglik_gda (loglik_gda.cpp:47-239) on C responses observed at the same rows: column c is loglik_gda on Y[:,c].  The
 * columns share the basis, the terms table, the hyper-parameters, dodiag and both para entries, so the per-row noise
 * sd obssd is one N-vector; it is formed on the device (gda_obssd_kernel) from the squared product residvar runs, and
 * rebuilt where LoglikGda sets redostd.  val, gradhyp and gradpara are the sums over the columns (in column order) of
 * loglik_gda's, grad is K x C, hessmult is block-diagonal, and the Hessian diagonals, which do not depend on the
 * response, are loglik_gda's computed once and repeated C times.  The products are the matrix path of LoglikGaussMulti:
 * mm_mat_dev | resid_multi with the per-row sd | tmm_mat_dev; the sd's hyper-gradient bookkeeping stays on the host as in
 * LoglikGda and runs once per update with gradients.  Para is never per column; one rank only (obfit's stage-1
 * subsample). */
struct LoglikGdaMulti : DevLik, GdaSd {
  bool doda = true, redostd = true;
  double sumlogsd = 0; /* sum_i log obssd_i in obh::sum2 order: the likelihood's constant, the same for every column */
  std::vector<double> y_host;
  DevBuf<double> sd, phi2, ssq, partial, gh;

  LoglikGdaMulti(Ctx& c, const OuterMod* om_, const u64* t, u64 K_, const double* yh /* N x C */, u64 C_, const double* xh, u64 N_)
      : DevLik(c, om_, t, K_, yh, C_, xh, N_) {
    if (ctx.nranks > 1) throw std::logic_error("loglik_gda_multi is the single-rank subsample model of obfit stage 1");
    npara = 2;
    y_host.assign(yh, yh + N * C);
    double vs = 0; /* para0[0] = 0.5 log(0.01 mean_c var(Y[:,c])), loglik_gda.cpp:59 on the mean variance */
    for (u64 j = 0; j < C; ++j) vs += arma_var(yh + j * N, N);
    para0 = {0.5 * std::log(0.01 * (vs / double(C))), 0.0};
    paravar = {4, 4};
    para = para0;
    ssq.ensure(C);
    buildstd();
  }
  bool multi() const override { return true; }
  void updateom() override { ob.build(); if (doda) redostd = true; }
  void updatepara(const double* p, u64 n) override {
    if (n != 2) throw std::range_error("para must have two entries");
    para.assign(p, p + n);
    redostd = true;
  }
  void updateterms(const u64* t, u64 K_) override { terms.assign(t, t + K_ * d); K = K_; nterms = K * C; if (doda) redostd = true; }
  void buildstd() { /* loglik_gda.cpp:217-236 */
    if (!redostd) return;
    const u64 ld = ob.ld;
    std::vector<double> rterms;
    sd.ensure(std::max<u64>(ld, 1));
    if (doda) { /* residvar = 1 - Phi^2 varc */
      std::vector<double> varc(K);
      om->getvar(terms.data(), K, varc.data());
      kbuf.upload(varc, ctx.stream);
      phi2.ensure(std::max<u64>(ld, 1));
      ob.mm_dev(terms.data(), K, 1, kbuf.p, phi2.p);
      rterms.resize(N);
      ob.d2h(rterms.data(), phi2.p, N);
      for (u64 i = 0; i < N; ++i) rterms[i] = 1 - rterms[i];
    }
    obd::launch_gda_obssd(ctx, doda ? phi2.p : nullptr, N, ld, std::exp(2 * para[0]), std::exp(2 * para[1]), sd.p);
    obssd.resize(N);
    ob.d2h(obssd.data(), sd.p, N);
    sd_grads(ob, terms.data(), K, para, doda, rterms);
    std::vector<double> t(N);
    for (u64 i = 0; i < N; ++i) t[i] = std::log(obssd[i]);
    sumlogsd = obh::sum2(t.data(), N);
    redostd = false;
  }
  double val_col(u64 c) const override { return -0.5 * ssq_host[c] - sumlogsd; }
  void cg_params(obd::CgParams& c) const override { c.ssq = ssq.p; c.use_sumlogsd = 1; c.sumlogsd = sumlogsd; }
  /* ssq[c]: column c's sum of squared standardised residuals */
  void update_dev(const double* coeff_dev) override {
    ob.mm_mat_dev(terms.data(), K, 0, coeff_dev, C, yhat.p, ob.ld);
    obd::launch_resid_multi(ctx, yhat.p, y.p, w.p, N, ob.ld, C, 1.0, true, partial, ssq.p, nullptr, sd.p);
    red.ensure(K * C);
    ob.tmm_mat_dev(terms.data(), K, 0, w.p, ob.ld, C, red.p);
  }
  void hessmult_dev(const double* g_dev) override { /* loglik_gda.cpp:156-164 per column; w holds Phi g until the residual pass */
    ob.mm_mat_dev(terms.data(), K, 0, g_dev, C, w.p, ob.ld);
    obd::launch_resid_multi(ctx, w.p, nullptr, w.p, N, ob.ld, C, 1.0, false, partial, nullptr, nullptr, sd.p);
    red.ensure(K * C);
    ob.tmm_mat_dev(terms.data(), K, 0, w.p, ob.ld, C, red.p);
  }
  void update(const std::vector<double>& cf) override { /* loglik_gda.cpp:116-149 per column */
    if (cf.size() != K * C) throw std::range_error("coeff must have K x ncol entries");
    coeff = cf;
    buildstd();
    const u64 H = ob.H, ld = ob.ld;
    kbuf.upload(coeff, ctx.stream);
    update_dev(kbuf.p);
    ssq_host.resize(C);
    ob.d2h(ssq_host.data(), ssq.p, C);
    if (compute_val) { val = 0; for (u64 c = 0; c < C; ++c) val += val_col(c); }
    if (!compute_grad) return;
    grad.resize(K * C);
    ob.d2h(grad.data(), red.p, K * C);
    if (!compute_gradhyp && !compute_gradpara) return;
    std::vector<double> ghr(H * C, 0.0);
    if (compute_gradhyp && H > 0) { /* the residual term, one hyper-gradient pass per column (:136) */
      gh.ensure(H * C);
      OB_CUDA(cudaMemsetAsync(gh.p, 0, H * C * sizeof(double), ctx.stream));
      for (u64 c = 0; c < C; ++c) {
        const std::vector<double> a(coeff.begin() + c * K, coeff.begin() + (c + 1) * K);
        ob.gradhyp_dots(terms.data(), K, a, kbuf.p + c * K, w.p + c * ld, yhat.p + c * ld, gh.p + c * H);
      }
      ob.d2h(ghr.data(), gh.p, H * C);
    }
    /* the sd's terms (:137-147): the 1 / obssd dots do not depend on the response */
    std::vector<double> yh(N), inv(N), rt2(N), invh(H, 0.0), invp(2);
    for (u64 i = 0; i < N; ++i) inv[i] = 1 / obssd[i];
    if (doda) for (u64 h = 0; h < H; ++h) invh[h] = dot2(inv.data(), obssd_gradhyp.data() + h * N, N);
    for (u64 q = 0; q < 2; ++q) invp[q] = dot2(inv.data(), obssd_gradpara.data() + q * N, N);
    if (compute_gradhyp) gradhyp.assign(H, 0.0);
    if (compute_gradpara) gradpara.assign(2, 0.0);
    for (u64 c = 0; c < C; ++c) {
      ob.d2h(yh.data(), yhat.p + c * ld, N);
      const double* yc = y_host.data() + c * N;
      for (u64 i = 0; i < N; ++i) { const double r = (yh[i] - yc[i]) / obssd[i]; rt2[i] = r * r; rt2[i] /= obssd[i]; }
      if (compute_gradhyp)
        for (u64 h = 0; h < H; ++h) {
          double g = ghr[c * H + h];
          if (doda) { g += dot2(rt2.data(), obssd_gradhyp.data() + h * N, N); g -= invh[h]; }
          gradhyp[h] += g;
        }
      if (compute_gradpara)
        for (u64 q = 0; q < 2; ++q) {
          double g = dot2(rt2.data(), obssd_gradpara.data() + q * N, N);
          g -= invp[q];
          gradpara[q] += g;
        }
    }
  }
  std::vector<double> hessmult(const std::vector<double>& g) override {
    if (g.size() != K * C) throw std::range_error("g must have K x ncol entries");
    kbuf.upload(g, ctx.stream);
    hessmult_dev(kbuf.p);
    std::vector<double> o(K * C);
    ob.d2h(o.data(), red.p, K * C);
    return o;
  }
  /* N x C, the last update's */
  std::vector<double> get_yhat() {
    std::vector<double> o(N * C);
    for (u64 c = 0; c < C; ++c) ob.d2h(o.data() + c * N, yhat.p + c * ob.ld, N);
    return o;
  }
  std::vector<double> diaghess() override { return tile_cols(gda_diaghess(ob, terms.data(), K), K, C); }
  std::vector<double> diaghessgradhyp() override { return tile_cols(gda_diaghessgradhyp(ob, terms.data(), K, doda), K, C); }
  std::vector<double> diaghessgradpara() override { return tile_cols(gda_diaghessgradpara(ob, terms.data(), K), K, C); }
  std::vector<double> hess() override { refuse_multi("the full Hessian"); }
  std::vector<double> hessgradhyp() override { refuse_multi("the full Hessian"); }
  std::vector<double> hessgradpara() override { refuse_multi("the full Hessian"); }
  void optnewton() override { refuse_multi("optnewton"); }
  void optcg(double, u64) override { refuse_multi("optcg outside lpdfvec(logpr_gauss_multi, loglik_gda_multi)"); }
};

struct LpdfVec : Lpdf { /* fit.cpp:174-267,310-428,557-607 */
  double val_margadj = 0;
  std::vector<double> gradhyp_margadj, gradpara_margadj;
  bool domargadj = true;
  std::vector<double> diaghessv, diaghessgradhypv, diaghessgradparav;
  std::vector<double> hessv, hessgradhypv, hessgradparav; /* full-Hessian branch, fit.h:121-123 */
  bool hyp_matrix_stale = false; /* buildhess took the contracted route: the K x H matrix is formed on demand */
  bool para_matrix_stale = false; /* likewise for the nterms x npara matrix (per-column para) */
  bool redohess = true;
  Lpdf* kid[2];
  u64 parasrt[2], paraend[2];
  LpdfVec(Lpdf* a, Lpdf* b) {
    if (a->multi() != b->multi() || a->ncol() != b->ncol())
      throw std::invalid_argument("lpdfvec: children must both be single-response, or multi-response with the same number of columns");
    if ((dynamic_cast<LoglikGdaMulti*>(a) && b->para_per_column()) || (dynamic_cast<LoglikGdaMulti*>(b) && a->para_per_column()))
      throw std::invalid_argument("lpdfvec: loglik_gda_multi pairs with a shared-para logpr_gauss_multi only");
    kid[0] = a; kid[1] = b;
    terms = a->terms; d = a->d;
    nterms = a->nterms;
    parasrt[0] = 0; paraend[0] = a->npara - 1;
    parasrt[1] = paraend[0] + 1; paraend[1] = parasrt[1] + b->npara - 1;
    para.assign(1 + paraend[1], 0.0);
    std::copy(a->para.begin(), a->para.end(), para.begin() + parasrt[0]);
    std::copy(b->para.begin(), b->para.end(), para.begin() + parasrt[1]);
    npara = para.size();
  }
  void setnthreads(int k) override { for (Lpdf* l : kid) l->setnthreads(k); }
  void updateom() override { for (Lpdf* l : kid) l->updateom(); redohess = true; }
  void updatepara(const double* p, u64 n) override {
    if (n != para.size()) throw std::range_error("wrongsized para vector");
    for (int c = 0; c < 2; ++c) {
      std::copy(p + parasrt[c], p + paraend[c] + 1, para.begin() + parasrt[c]);
      kid[c]->updatepara(p + parasrt[c], paraend[c] + 1 - parasrt[c]);
    }
    redohess = true;
  }
  void updateterms(const u64* t, u64 K) override {
    terms.assign(t, t + K * d);
    for (Lpdf* l : kid) { l->updateterms(t, K); nterms = l->nterms; }
    redohess = true;
  }
  std::vector<double> diaghess_() {
    std::vector<double> out = kid[0]->diaghess(), h = kid[1]->diaghess();
    for (u64 i = 0; i < out.size(); ++i) out[i] += h[i];
    return out;
  }
  std::vector<double> diaghessgradhyp_() {
    std::vector<double> out = kid[0]->diaghessgradhyp(), h = kid[1]->diaghessgradhyp();
    for (u64 i = 0; i < out.size(); ++i) out[i] += h[i];
    return out;
  }
  std::vector<double> diaghessgradpara_() {
    std::vector<double> out(nterms * para.size(), 0.0);
    for (int c = 0; c < 2; ++c) {
      std::vector<double> h = kid[c]->diaghessgradpara();
      const u64 nc = paraend[c] + 1 - parasrt[c];
      for (u64 j = 0; j < nc; ++j) for (u64 i = 0; i < nterms; ++i) out[i + (parasrt[c] + j) * nterms] = h[i + j * nterms];
    }
    return out;
  }
  void settotdiaghess(const std::vector<double>& dh) override {
    totdiaghess = dh;
    for (Lpdf* l : kid) { l->settotdiaghess(dh); l->totdiaghess_percol = para_per_column(); }
  }
  void settothess(const std::vector<double>& h) override { tothess = h; for (Lpdf* l : kid) l->settothess(h); } /* :609-612 */
  std::vector<double> hess() override { return hessv; }
  std::vector<double> hessgradhyp() override { return hessgradhypv; }
  std::vector<double> hessgradpara() override { return hessgradparav; }
  static std::vector<double> sum_same_size(std::vector<double> a, const std::vector<double>& b, const char* what) {
    if (a.size() != b.size()) throw std::invalid_argument(std::string("addition: incompatible dimensions (") + what + ")");
    for (u64 i = 0; i < a.size(); ++i) a[i] += b[i];
    return a;
  }
  std::vector<double> hessgradpara_() { /* :539-549 */
    const u64 K = nterms, KK = K * K;
    std::vector<double> out(KK * para.size(), 0.0);
    for (int c = 0; c < 2; ++c) {
      const std::vector<double> h = kid[c]->hessgradpara();
      const u64 nc = paraend[c] + 1 - parasrt[c];
      if (h.size() != KK * nc) throw std::invalid_argument("copy into subcube: incompatible dimensions");
      std::copy(h.begin(), h.end(), out.begin() + parasrt[c] * KK);
    }
    return out;
  }
  /* the full branch of buildhess, fit.cpp:269-299.  log det and the inverse come from a Cholesky factor when the total
   * Hessian is positive definite (it is at every point optnewton reaches), else from the symmetric eigen-decomposition
   * the reference uses for both */
  void buildhess_full() {
    if (multi()) refuse_multi("the full-Hessian branch");
    const u64 K = nterms, KK = K * K;
    hessv = sum_same_size(kid[0]->hess(), kid[1]->hess(), "hess");
    settothess(hessv);
    if (!domargadj) return;
    hessgradhypv = sum_same_size(kid[0]->hessgradhyp(), kid[1]->hessgradhyp(), "hessgradhyp");
    hessgradparav = hessgradpara_();
    if (hessv.size() != KK) throw std::invalid_argument("eig_sym(): given matrix must be square sized");
    std::vector<double> L = hessv, hessi;
    bool pd = true;
    for (u64 j = 0; j < K && pd; ++j) { /* column Cholesky, lower triangle in place */
      double djj = L[j + j * K];
      for (u64 p = 0; p < j; ++p) djj -= L[j + p * K] * L[j + p * K];
      if (!(djj > 0.0)) { pd = false; break; }
      djj = std::sqrt(djj);
      L[j + j * K] = djj;
      for (u64 i = j + 1; i < K; ++i) {
        double v = L[i + j * K];
        for (u64 p = 0; p < j; ++p) v -= L[i + p * K] * L[j + p * K];
        L[i + j * K] = v / djj;
      }
    }
    if (pd) {
      std::vector<double> t(K);
      for (u64 i = 0; i < K; ++i) t[i] = 2.0 * std::log(L[i + i * K]);
      val_margadj = -0.5 * obh::sum2(t.data(), K);
      /* inverse = L^-T L^-1: invert the triangle column by column, then multiply */
      std::vector<double> Li(KK, 0.0);
      for (u64 j = 0; j < K; ++j) {
        Li[j + j * K] = 1.0 / L[j + j * K];
        for (u64 i = j + 1; i < K; ++i) {
          double v = 0.0;
          for (u64 p = j; p < i; ++p) v -= L[i + p * K] * Li[p + j * K];
          Li[i + j * K] = v / L[i + i * K];
        }
      }
      hessi.assign(KK, 0.0);
      for (u64 j = 0; j < K; ++j)
        for (u64 i = j; i < K; ++i) {
          double v = 0.0;
          for (u64 p = i; p < K; ++p) v += Li[p + i * K] * Li[p + j * K];
          hessi[i + j * K] = v; hessi[j + i * K] = v;
        }
    } else {
      obh::Mat S(K, K), V;
      S.a = hessv;
      std::vector<double> w;
      obh::sym_eig_desc(S, w, V);
      std::vector<double> t(K);
      for (u64 i = 0; i < K; ++i) t[i] = std::log(w[i]);
      val_margadj = -0.5 * obh::sum2(t.data(), K);
      hessi.assign(KK, 0.0);
      for (u64 j = 0; j < K; ++j)
        for (u64 i = 0; i < K; ++i) {
          double v = 0.0;
          for (u64 p = 0; p < K; ++p) v += V(i, p) * V(j, p) / w[p];
          hessi[i + j * K] = v;
        }
    }
    std::vector<double> tm(KK);
    const u64 H = KK ? hessgradhypv.size() / KK : 0, P = para.size();
    gradhyp_margadj.assign(H, 0.0);
    for (u64 l = 0; l < H; ++l) {
      for (u64 i = 0; i < KK; ++i) tm[i] = hessgradhypv[i + l * KK] * hessi[i];
      gradhyp_margadj[l] = -0.5 * obh::sum2(tm.data(), KK);
    }
    gradpara_margadj.assign(P, 0.0);
    for (u64 l = 0; l < P; ++l) {
      for (u64 i = 0; i < KK; ++i) tm[i] = hessgradparav[i + l * KK] * hessi[i];
      gradpara_margadj[l] = -0.5 * obh::sum2(tm.data(), KK);
    }
  }
  void buildhess() { /* fit.cpp:252-301 */
    if (redohess) {
      diaghessv = diaghess_();
      settotdiaghess(diaghessv);
      if (domargadj) {
        /* the marginal adjustment only needs diaghessgradhyp contracted with 1 / diaghess: children that can
         * deliver that contraction directly (loglik_gauss: one sweep instead of 2H products) skip the K x H matrix,
         * which is then formed lazily if somebody asks for it (diaghessgradhyp()) */
        const u64 K = diaghessv.size();
        std::vector<double> cinv(K), dot0, dot1;
        for (u64 i = 0; i < K; ++i) cinv[i] = 1.0 / diaghessv[i];
        const bool swept = kid[0]->can_diaghessgradhyp_dot() && kid[1]->can_diaghessgradhyp_dot() &&
                           kid[1]->diaghessgradhyp_dot(cinv, dot1) && kid[0]->diaghessgradhyp_dot(cinv, dot0) && dot0.size() == dot1.size();
        if (swept) { diaghessgradhypv.clear(); hyp_matrix_stale = true; }
        else { diaghessgradhypv = diaghessgradhyp_(); hyp_matrix_stale = false; }
        /* per-column children contract their para derivatives directly: with P growing with C, the dense
         * nterms x P matrix is what would dominate (formed on demand, diaghessgradpara()) */
        std::vector<double> pdot[2];
        bool pdone[2];
        for (int c = 0; c < 2; ++c) pdone[c] = kid[c]->diaghessgradpara_dot(diaghessv, pdot[c]);
        para_matrix_stale = pdone[0] || pdone[1];
        if (para_matrix_stale) diaghessgradparav.clear();
        else diaghessgradparav = diaghessgradpara_();
        const u64 H = swept ? dot0.size() : diaghessgradhypv.size() / std::max<u64>(K, 1), P = para.size();
        std::vector<double> t(K);
        for (u64 i = 0; i < K; ++i) t[i] = std::log(diaghessv[i]);
        val_margadj = -0.5 * obh::sum2(t.data(), K);
        gradhyp_margadj.assign(H, 0.0);
        for (u64 h = 0; h < H; ++h) {
          if (swept) { gradhyp_margadj[h] = -0.5 * (dot0[h] + dot1[h]); continue; }
          for (u64 i = 0; i < K; ++i) t[i] = diaghessgradhypv[i + h * K] / diaghessv[i];
          gradhyp_margadj[h] = -0.5 * obh::sum2(t.data(), K);
        }
        gradpara_margadj.assign(P, 0.0);
        if (!para_matrix_stale)
          for (u64 h = 0; h < P; ++h) {
            for (u64 i = 0; i < K; ++i) t[i] = diaghessgradparav[i + h * K] / diaghessv[i];
            gradpara_margadj[h] = -0.5 * obh::sum2(t.data(), K);
          }
        else
          for (int c = 0; c < 2; ++c) {
            const u64 nc = paraend[c] + 1 - parasrt[c];
            if (pdone[c]) { for (u64 j = 0; j < nc; ++j) gradpara_margadj[parasrt[c] + j] = -0.5 * pdot[c][j]; continue; }
            const std::vector<double> h = kid[c]->diaghessgradpara();
            for (u64 j = 0; j < nc; ++j) {
              for (u64 i = 0; i < K; ++i) t[i] = h[i + j * K] / diaghessv[i];
              gradpara_margadj[parasrt[c] + j] = -0.5 * obh::sum2(t.data(), K);
            }
          }
      }
      if (fullhess) buildhess_full();
    }
    redohess = false;
  }
  void update(const std::vector<double>& c) override { /* fit.cpp:323-361 */
    coeff = c;
    for (Lpdf* l : kid) {
      l->compute_val = compute_val; l->compute_grad = compute_grad;
      l->compute_gradhyp = compute_gradhyp; l->compute_gradpara = compute_gradpara;
    }
    for (Lpdf* l : kid) l->update(coeff);
    if (compute_val) val = 0;
    if (compute_grad) grad.assign(kid[0]->grad.size(), 0.0);
    if (compute_gradhyp) gradhyp.assign(kid[0]->gradhyp.size(), 0.0);
    if (compute_gradpara) gradpara.assign(para.size(), 0.0);
    buildhess();
    for (int cnt = 0; cnt < 2; ++cnt) {
      Lpdf* l = kid[cnt];
      if (compute_val) val += l->val;
      if (compute_grad) for (u64 i = 0; i < grad.size(); ++i) grad[i] += l->grad[i];
      if (compute_gradhyp) for (u64 i = 0; i < gradhyp.size(); ++i) gradhyp[i] += l->gradhyp[i];
      if (compute_gradpara) for (u64 i = parasrt[cnt]; i <= paraend[cnt]; ++i) gradpara[i] += l->gradpara[i - parasrt[cnt]];
    }
    if (domargadj) { /* margadj :371-380 */
      if (compute_val) val += val_margadj;
      if (compute_gradhyp) for (u64 i = 0; i < gradhyp.size(); ++i) gradhyp[i] += gradhyp_margadj[i];
      if (compute_gradpara) for (u64 i = 0; i < gradpara.size(); ++i) gradpara[i] += gradpara_margadj[i];
    }
  }
  std::vector<double> hessmult(const std::vector<double>& g) override {
    std::vector<double> out = kid[0]->hessmult(g), h = kid[1]->hessmult(g);
    for (u64 i = 0; i < out.size(); ++i) out[i] += h[i];
    return out;
  }
  /* lpdf::optcg (fit.cpp:37-96) with every K-vector and scalar of the loop in HBM, for lpdfvec(logpr_gauss,
   * loglik_gauss), lpdfvec(logpr_gauss_multi, loglik_gauss_multi) and lpdfvec(logpr_gauss_multi, loglik_gda_multi) in
   * either order (the likelihood is a DevLik).  The reference's sequence is kept
   * operation by operation -- first update() and diaghess() through the host path (they build the cached Hessian
   * diagonal and the marginal adjustment, fit.cpp:252-267), then per iteration: CG_STEP | stop test | update |
   * CG_POST_UPDATE | hessmult, each a few launches on the library stream; the host reads one value per iteration; the
   * final update() with gradients runs through the host path again.
   * Multi-response: C independent runs of lpdf::optcg, column c on column c's own objective (its loglik, its prior, the
   * single-response marginal adjustment) with its own num, alpha, beta, val / valdiff and stop test -- NOT one CG on the
   * K C system, which would share alpha and beta over the columns.  cg_stage_kernel runs one CTA per column; a column
   * whose stop test passes is frozen as the reference `break`s, and the loop ends when no column runs (the value the
   * host reads is the count of running columns) or after maxepch.  The products of an iteration run over all C columns,
   * frozen ones included.  When either child has per-column para, the columns' diagonals differ: each column's
   * marginal adjustment, coefficient scale and noise sd go to the kernel as C-entry device arrays, uploaded here once.
   * A single-response pairing returns false (the caller runs the host loop) without option device_cg, rows or a
   * specialised terms table, and for every other pairing; a multi-response object runs here or throws. */
  DevBuf<double> cg_coeff, cg_grad, cg_m, cg_rm, cg_p, cg_q, cg_sds, cg_scal, cg_sca, cg_vma;
  DevBuf<unsigned> cg_running;
  std::vector<u64> cg_iters_cols;
  bool optcg_device(double tol, u64 maxepch) {
    const bool mult = multi();
    auto* lk = dynamic_cast<DevLik*>(kid[0]);
    const bool lik_first = lk != nullptr;
    if (!lik_first) lk = dynamic_cast<DevLik*>(kid[1]);
    Lpdf* prior = kid[lik_first ? 1 : 0];
    auto* prm = dynamic_cast<LogprGaussMulti*>(prior);
    const LogprGauss* pr = prm ? &prm->one : dynamic_cast<LogprGauss*>(prior);
    if (!lk || !pr) {
      if (mult) throw std::invalid_argument("optcg on multi-response objects needs lpdfvec(logpr_gauss_multi, loglik_gauss_multi or loglik_gda_multi)");
      return false;
    }
    Ctx& ctx = lk->ctx;
    const u64 K = lk->K, C = lk->C, NS = obd::CG_NSCAL;
    if (!mult && (!ctx.device_cg || K == 0 || lk->N == 0 || !lk->ob.spec_for(terms.data(), K))) return false;
    compute_val = true; compute_grad = true; compute_gradhyp = false; compute_gradpara = false;
    if (coeff.size() != nterms) coeff.assign(nterms, 0.0);
    update(std::vector<double>(coeff));
    std::vector<double> m = diaghess();
    cg_iters = 0;
    if (mult) cg_iters_cols.assign(C, 0);
    if (!all_finite(m) && !all_finite(grad)) { val = -std::numeric_limits<double>::infinity(); return true; }
    /* the starting value of each run: single response, the lpdfvec's own; multi-response, column c's value as the
     * single-response lpdfvec forms it (fit.cpp:352-380): children in order, then its own marginal adjustment -- the
     * diagonal's column block c is column c's single-response diagonal (with shared para, every block is block 0) */
    const bool percol = mult && (lk->para_per_column() || prm->percol);
    std::vector<double> vma_cols(percol ? C : 1, val_margadj);
    if (mult)
      for (u64 c = 0; c < vma_cols.size(); ++c) {
        vma_cols[c] = 0;
        if (!domargadj) continue;
        std::vector<double> t(K);
        for (u64 i = 0; i < K; ++i) t[i] = std::log(diaghessv[c * K + i]);
        vma_cols[c] = -0.5 * obh::sum2(t.data(), K);
      }
    const double vma = vma_cols[0];
    std::vector<double> scal(C * NS, 0.0), sca_cols;
    for (u64 c = 0; c < C; ++c) {
      double v = val;
      if (mult) {
        const double vl = lk->val_col(c), vp = prm->val_cols[c];
        v = lik_first ? (0.0 + vl) + vp : (0.0 + vp) + vl;
        if (domargadj) v += vma_cols[percol ? c : 0];
      }
      if (percol) sca_cols.push_back(prm->sca_col(c));
      double* S = scal.data() + c * NS;
      S[obd::CG_VAL] = v; S[obd::CG_VALO] = v; S[obd::CG_VALDIFF] = 10; S[obd::CG_DENOM] = 1;
    }
    cg_coeff.upload(coeff, ctx.stream); cg_grad.upload(grad, ctx.stream); cg_m.upload(m, ctx.stream);
    cg_sds.upload(pr->coeffsd, ctx.stream);
    cg_rm.ensure(K * C); cg_p.ensure(K * C); cg_q.ensure(K * C);
    cg_scal.upload(scal, ctx.stream);
    if (percol) { cg_sca.upload(sca_cols, ctx.stream); cg_vma.upload(vma_cols, ctx.stream); }
    if (mult) cg_running.ensure(2);
    ctx.sync(); /* the host images above must outlive the uploads */
    obd::CgParams c{};
    c.K = (int)K; c.lik_first = lik_first ? 1 : 0; c.domarg = domargadj ? 1 : 0;
    c.coeff = cg_coeff.p; c.grad = cg_grad.p; c.m = cg_m.p; c.rm = cg_rm.p; c.p = cg_p.p; c.q = cg_q.p; c.sds = cg_sds.p;
    c.sca = pr->sca; c.val_margadj = vma; c.tol = tol; c.scal = cg_scal.p;
    lk->cg_params(c);
    if (mult) c.running = cg_running.p;
    if (percol) { c.sca_col = cg_sca.p; c.vma_col = cg_vma.p; }
    auto stage = [&](int st) { c.stage = st; c.red = lk->red.p; obd::launch_cg_stage(ctx, c, C); };
    stage(obd::CG_INIT);          /* rm = grad / m ; p = rm                       :58-60 */
    lk->hessmult_dev(cg_p.p);     /* q = hessmult(p), finished inside CG_STEP     :62 */
    u64 k;
    for (k = 0; k < maxepch; k++) {
      if (mult) {
        c.iter = (int)k;
        OB_CUDA(cudaMemsetAsync(cg_running.p + (k & 1), 0, sizeof(unsigned), ctx.stream));
      }
      stage(obd::CG_STEP);        /* q ; num ; stop test ; denom ; alpha ; coeff += alpha p ; valo   :72-77 */
      if (mult) OB_CUDA(cudaMemcpyAsync(ctx.pinned, cg_running.p + (k & 1), sizeof(unsigned), cudaMemcpyDeviceToHost, ctx.stream));
      else OB_CUDA(cudaMemcpyAsync(ctx.pinned, cg_scal.p + obd::CG_STOP, sizeof(double), cudaMemcpyDeviceToHost, ctx.stream));
      ctx.sync();
      unsigned running = 0;
      std::memcpy(&running, ctx.pinned, sizeof(running));
      if (mult ? running == 0 : ctx.pinned[0] != 0.0) break;
      lk->update_dev(cg_coeff.p); /* update(coeff)                                :78 */
      stage(obd::CG_POST_UPDATE); /* grad ; val ; valdiff ; rm ; beta ; p         :79-83 */
      lk->hessmult_dev(cg_p.p);   /* q = hessmult(p)                              :84 */
    }
    cg_iters = k;
    if (mult) OB_CUDA(cudaMemcpyAsync(scal.data(), cg_scal.p, C * NS * sizeof(double), cudaMemcpyDeviceToHost, ctx.stream));
    OB_CUDA(cudaMemcpyAsync(coeff.data(), cg_coeff.p, K * C * sizeof(double), cudaMemcpyDeviceToHost, ctx.stream));
    ctx.sync();
    if (mult)
      for (u64 j = 0; j < C; ++j) cg_iters_cols[j] = scal[j * NS + obd::CG_STOP] != 0.0 ? (u64)scal[j * NS + obd::CG_ITER] : k;
    compute_gradhyp = true; compute_gradpara = true;
    update(std::vector<double>(coeff));
    compute_gradhyp = false; compute_gradpara = false;
    return true;
  }
  void optcg(double tol, u64 maxepch) override {
    fullhess = false; /* fit.cpp:38 */
    if (!optcg_device(tol, maxepch)) Lpdf::optcg(tol, maxepch);
  }
  void optnewton() override {
    if (multi()) refuse_multi("optnewton");
    Lpdf::optnewton();
  }
  bool multi() const override { return kid[0]->multi(); }
  u64 ncol() const override { return kid[0]->ncol(); }
  bool para_per_column() const override { return kid[0]->para_per_column() || kid[1]->para_per_column(); }
  std::vector<double> diaghess() override { return diaghessv; }
  std::vector<double> diaghessgradhyp() override {
    if (hyp_matrix_stale) { diaghessgradhypv = diaghessgradhyp_(); hyp_matrix_stale = false; }
    return diaghessgradhypv;
  }
  std::vector<double> diaghessgradpara() override {
    if (para_matrix_stale) { diaghessgradparav = diaghessgradpara_(); para_matrix_stale = false; }
    return diaghessgradparav;
  }
  double paralpdf(const double* p, u64 n) const override {
    if (n != para.size()) return -std::numeric_limits<double>::infinity();
    double out = 0;
    for (int c = 0; c < 2; ++c) out += kid[c]->paralpdf(p + parasrt[c], paraend[c] + 1 - parasrt[c]);
    return out;
  }
  void paralpdf_grad(const double* p, u64 n, double* out) const override {
    for (u64 i = 0; i < para.size(); ++i) out[i] = 0.0;
    if (n != para.size()) return;
    for (int c = 0; c < 2; ++c) kid[c]->paralpdf_grad(p + parasrt[c], paraend[c] + 1 - parasrt[c], out + parasrt[c]);
  }
  u64 nhyp() const override { return kid[0]->nhyp(); }
  u64 nrow() const override { return std::max(kid[0]->nrow(), kid[1]->nrow()); }
};

/* a likelihood's predictor: its model on new inputs (update), the predictive mean (N x C for C responses) and variance */
struct Pred {
  Ctx& ctx;
  const OuterMod* om;
  std::vector<double> para, coeff;
  std::vector<u64> terms;
  u64 K, C;
  std::unique_ptr<OuterBase> ob;
  Pred(Ctx& c, const OuterMod* om_, const Lpdf& lk, const std::vector<double>& x, u64 N, u64 K_, u64 C_ = 1)
      : ctx(c), om(om_), para(lk.para), coeff(lk.coeff), terms(lk.terms), K(K_), C(C_) {
    ob.reset(new OuterBase(ctx, om, x.data(), N, false, terms.data(), K));
    if (coeff.size() != K * C) coeff.assign(K * C, 0.0);
  }
  virtual ~Pred() {}
  void update(const double* x, u64 N) { ob.reset(new OuterBase(ctx, om, x, N, false, terms.data(), K)); }
  void mean(double* out) {
    if (C == 1) ob->mm(0, terms.data(), K, coeff.data(), out);
    else ob->mm_mat(0, terms.data(), K, coeff.data(), C, out);
  }
  virtual void var(double* out) = 0;
  /* 1 / totdiaghess, zero before the total Hessian is set (loglik_gauss.cpp:205-209) */
  static std::vector<double> inv_totdiaghess(const Lpdf& lk) {
    if (lk.didnotothess) return std::vector<double>(lk.nterms, 0.0);
    std::vector<double> v(lk.totdiaghess.size());
    for (u64 i = 0; i < v.size(); ++i) v[i] = 1 / lk.totdiaghess[i];
    return v;
  }
};

struct PredGauss : Pred { /* loglik_gauss.cpp:196-227 */
  std::vector<double> coeffvar;
  bool percol, lik_percol;
  /* multi-response, shared para everywhere: the variance is one N-vector for all columns (the total Hessian diagonal is
   * the same K-vector repeated over the columns).  When the likelihood has per-column para, or its total diagonal came
   * from an lpdfvec with a per-column prior, the columns' diagonals differ: N x C, column c = Phi^2 V[:,c] +
   * exp(2 para_c) with V the K x C matrix of 1 / totdiaghess, as ONE squared multi-right-hand-side product. */
  PredGauss(LoglikGaussBase& lk)
      : Pred(lk.ctx, lk.om, lk, lk.x_host, lk.N, lk.K, lk.C), percol(lk.predvar_ncol() > 1), lik_percol(lk.percol) {
    if (!lk.multi() || percol) coeffvar = inv_totdiaghess(lk);
    else {
      coeffvar.assign(K, 0.0);
      if (!lk.didnotothess && lk.totdiaghess.size() >= K)
        for (u64 i = 0; i < K; ++i) coeffvar[i] = 1 / lk.totdiaghess[i];
    }
  }
  void var(double* out) override {
    if (percol) {
      if (coeffvar.size() != K * C) throw std::invalid_argument("predictor: the total Hessian diagonal must have K x ncol entries");
      ob->mm_mat(1, terms.data(), K, coeffvar.data(), C, out);
      for (u64 c = 0; c < C; ++c) {
        const double v = std::exp(2 * para[lik_percol ? c : 0]);
        for (u64 i = 0; i < ob->N; ++i) out[c * ob->N + i] += v;
      }
      return;
    }
    ob->mm(1, terms.data(), K, coeffvar.data(), out);
    const double c = std::exp(2 * para[0]);
    for (u64 i = 0; i < ob->N; ++i) out[i] += c;
  }
};

struct PredrStd : Pred { /* loglik_std.cpp:219-257 */
  std::vector<double> coeffcov; /* K x K */
  DevBuf<double> cov_dev, prod, basis, outv;
  PredrStd(LoglikStd& lk) : Pred(lk.ctx, lk.om, lk, lk.x_host, lk.N, lk.K) {
    coeffcov.assign(K * K, 0.0);
    if (!lk.didnotothess) {
      if (lk.didfulltothess) coeffcov = Lpdf::dense_inv(lk.tothess, K);
      /* as written in the reference (:229): the diagonal of the total Hessian itself, not its inverse */
      else for (u64 i = 0; i < K; ++i) coeffcov[i + i * K] = lk.totdiaghess[i];
    }
  }
  void var(double* out) override { /* rowsum((Phi coeffcov) % Phi) + exp(2 para) */
    const u64 N = ob->N, ld = ob->ld;
    if (N == 0) return;
    cov_dev.upload(coeffcov, ctx.stream);
    prod.ensure(ld * std::max<u64>(K, 1)); basis.ensure(ld * std::max<u64>(K, 1)); outv.ensure(ld);
    ob->mm_mat_dev(terms.data(), K, 0, cov_dev.p, K, prod.p, ld);
    ob->getmat_dev(terms.data(), K, -1, basis.p);
    obd::launch_rowdot(ctx, prod.p, basis.p, N, K, ld, std::exp(2 * para[0]), outv.p);
    ob->d2h(out, outv.p, N);
  }
};

/* multi-response (LoglikGdaMulti): the mean is N x C, the variance one N-vector for all columns from the first K entries
 * of 1 / totdiaghess (its column blocks are equal) */
struct PredGda : Pred { /* loglik_gda.cpp:249-283 */
  std::vector<double> coeffvar;
  bool doda;
  PredGda(LoglikGda& lk) : Pred(lk.ctx, lk.om, lk, lk.x_host, lk.N, lk.nterms), coeffvar(inv_totdiaghess(lk)), doda(lk.doda) {}
  PredGda(LoglikGdaMulti& lk) : Pred(lk.ctx, lk.om, lk, lk.x_host, lk.N, lk.K, lk.C), coeffvar(inv_totdiaghess(lk)), doda(lk.doda) {}
  void var(double* out) override {
    ob->mm(1, terms.data(), K, coeffvar.data(), out);
    std::vector<double> rv(ob->N);
    if (doda) ob->residvar(terms.data(), K, rv.data());
    for (u64 i = 0; i < ob->N; ++i) { out[i] += std::exp(2 * para[0]); if (doda) out[i] += std::exp(2 * para[1]) * rv[i]; }
  }
};

} // namespace obe
