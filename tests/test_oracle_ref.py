"""Pins the CPU oracle against the REFERENCE ITSELF (VERDICT r1, "a pinned oracle").

oracle/_ref/libob_ref.so is built by `make -C oracle ref` from the UNMODIFIED reference sources
(the reference's src/{linalg,covfuncs,modandbase,fit}.cpp + src/lpdfs/*.cpp) compiled against oracle/arma_shim -- a
header-only Armadillo subset written for this purpose -- and exports the same C ABI with prefix `ref_`
(oracle/ref_capi.cpp), so ONE binding drives reference and oracle on the same inputs.

With one OpenMP thread the reference is deterministic and the oracle must reproduce it BIT FOR BIT: terms, index tables,
eigenbasis, basis matrices, every linalg.h kernel on both `vertpl` branches, loglik_gauss / logpr_gauss / lpdfvec /
loglik_gda, optcg (iterates included), predictors.  With several threads both sides add thread-local partial sums under
`omp critical` in arrival order (linalg.cpp:334-335, 438-442, 616-617), so Phi^T-type results agree to rounding only
(<= 1e-14 relative asserted; ~1e-16 observed).

The two third-party stand-ins are SHARED by both sides, which is what makes bitwise equality meaningful: eig_sym (LAPACK
upstream) = the oracle's cyclic Jacobi, shuffle (R's RNG upstream) = the injectable tie-break.  BLAS order = netlib
reference BLAS (R's bundled libRblas).  The second build, libob_ref_noblas.so (Armadillo without BLAS: two-accumulator
inner products everywhere), shows what that third-party choice is worth: the linalg.h kernels on shared inputs do not
depend on it, the basis build does (eps * lambda_0 / lambda_j amplification, SURVEY 7 "hard parts").

The reference's sources are not part of this repository (with REFSRC=<checkout of the reference>/src in the
environment, the tests build oracle/_ref from it).  Without oracle/_ref these tests do NOT compare with the reference:
the reference side of every test runs on the oracle, so each assertion compares the oracle with itself, and what is
left is a pin of the oracle.  Every value that side returns is checked, in call order, against the oracle's own output
recorded in tests/golden/oracle_pin.npz: bit for bit (an 8-byte hash) in most tests; in the two tests whose sums arrive
in thread order (LOOSE), through its size, largest magnitude, 256 seeded samples and 32 block sums, to the tests' own
tolerances.  The pin is always taken from the oracle, never from oracle/_ref, because the oracle is what it is replayed
against: `OB_RECORD_ORACLE_PIN=1 pytest tests/test_oracle_ref.py` retakes it after a deliberate change to oracle/.
"""
import hashlib
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import one_cpu, REPO, make_problem, relerr

REFDIR = REPO / "oracle" / "_ref"
REFSRC = os.environ.get("REFSRC")  # src/ of a checkout of the reference
RECORD = REPO / "tests" / "golden" / "oracle_pin.npz"
RECORDING = os.environ.get("OB_RECORD_ORACLE_PIN") == "1"
# the libraries sum thread-local partial results in arrival order here: the values are reproducible to rounding only
LOOSE = {"test_kernels_with_all_threads", "test_stateless_seam_bitwise"}


def _ref_library(name):
    from outerbase_b200.binding import Library
    so = REFDIR / name
    if REFSRC and Path(REFSRC).exists():  # (re)build from the reference tree
        subprocess.run(["make", "-C", str(REPO / "oracle"), "ref", f"REFSRC={REFSRC}"], check=True, capture_output=True)
    return Library(so, "ref_") if so.exists() else None


LOOSE_SAMPLES, LOOSE_BLOCKS = 256, 32


def _fingerprint(v, loose):
    a = np.asarray(v, dtype=np.float64)
    if loose:  # size, largest magnitude, seeded samples (NaN-padded), sums of LOOSE_BLOCKS contiguous blocks
        flat = a.ravel()
        idx = np.random.default_rng(flat.size).choice(flat.size, size=min(flat.size, LOOSE_SAMPLES), replace=False)
        sample = np.full(LOOSE_SAMPLES, np.nan)
        sample[:idx.size] = flat[idx]
        sums = [b.sum() for b in np.array_split(flat, LOOSE_BLOCKS)]
        return np.concatenate([[flat.size, np.abs(flat).max() if flat.size else 0.0], sample, sums])
    h = hashlib.blake2b(repr(a.shape).encode() + np.ascontiguousarray(a).tobytes(), digest_size=8)
    return np.frombuffer(h.digest(), dtype=np.uint8)


class _Book:
    """The values one test reads from the reference side, in order: recorded, or checked against the pin."""

    def __init__(self, test, record, loose):
        self.test, self.loose, self.n = test, loose, 0
        self.seen = record.setdefault(test, []) if RECORDING else record.get(test, np.empty((0, 0)))

    def check(self, v):
        if v is None or isinstance(v, str):
            return v
        if isinstance(v, tuple):
            return tuple(self.check(u) for u in v)
        if self.loose and not isinstance(v, np.ndarray):  # loop sizes follow the host's core count
            return v
        key, fp = f"{self.test} value {self.n}", _fingerprint(v, self.loose)
        self.n += 1
        if RECORDING:
            self.seen.append(fp)
        elif self.n > len(self.seen):
            pytest.fail(f"{key}: the oracle pin has no such value")
        elif self.loose:
            # the tests' own tolerances: 1e-13 of the largest magnitude, or 1e-14 absolute where a 1 cancels (residvar)
            r = self.seen[self.n - 1]
            tol = max(1e-13 * r[1], 1e-14)
            assert fp[0] == r[0] and abs(fp[1] - r[1]) <= tol, key
            samples = slice(2, 2 + LOOSE_SAMPLES)
            assert np.nanmax(np.abs(fp[samples] - r[samples]), initial=0.0) <= tol, key
            block = -(-int(r[0]) // LOOSE_BLOCKS)
            assert np.abs(fp[samples.stop:] - r[samples.stop:]).max() <= tol * block, key
        else:
            assert np.array_equal(fp, self.seen[self.n - 1]), f"{key}: differs from the oracle pin"
        return v

    def wrap(self, v):
        from outerbase_b200.binding import _Handle
        return _Recorded(v, self) if isinstance(v, _Handle) else self.check(v)

    def finish(self):
        if not RECORDING and self.n != len(self.seen):
            pytest.fail(f"{self.test}: read {self.n} values, the oracle pin holds {len(self.seen)}")


def _unwrap(v):
    return object.__getattribute__(v, "_t") if isinstance(v, _Recorded) else v


class _Recorded:
    """A library or object standing on the reference side whose every returned value goes through a _Book."""

    def __init__(self, target, book):
        object.__setattr__(self, "_t", target)
        object.__setattr__(self, "_book", book)

    def __getattr__(self, name):
        v = getattr(self._t, name)
        if name.startswith("_"):
            return v
        if callable(v):
            return lambda *a, **k: self._book.wrap(v(*map(_unwrap, a), **{n: _unwrap(u) for n, u in k.items()}))
        return self._book.wrap(v)

    def __setattr__(self, name, value):
        setattr(self._t, name, _unwrap(value))


@pytest.fixture(scope="session")
def _record():
    if RECORDING:
        rec = {}
        yield rec
        np.savez_compressed(RECORD, **{test: np.stack(fps) for test, fps in rec.items() if fps})
    else:
        yield dict(np.load(RECORD)) if RECORD.exists() else {}


@pytest.fixture
def reference(request, oracle, _record):
    lib = _ref_library("libob_ref.so")
    if lib is not None and not RECORDING:
        yield lib
        return
    book = _Book(request.node.name, _record, request.function.__name__ in LOOSE)
    yield _Recorded(oracle, book)
    book.finish()


@pytest.fixture(scope="session")
def reference_noblas():
    lib = _ref_library("libob_ref_noblas.so")
    if lib is None:
        pytest.skip("oracle/_ref/libob_ref_noblas.so is not built: the reference without BLAS has no stand-in")
    return lib


def both(oracle, reference, N, K, threads=1, **kw):
    """The same problem on both libraries; outerbase rebuilt with `threads` OpenMP threads (setloopvals_, modandbase.cpp:504-513)."""
    omo, x, y, terms, rng = make_problem(oracle, N, K, **kw)
    omr, _, _, terms_r, _ = make_problem(reference, N, K, **kw)
    np.testing.assert_array_equal(terms, terms_r)
    obo, obr = oracle.outerbase(omo, x), reference.outerbase(omr, x)
    for ob in (obo, obr):
        ob.nthreads = threads
        ob.build()
    assert (obo.chunksize, obo.loopsize, obo.vertpl) == (obr.chunksize, obr.loopsize, obr.vertpl)
    return dict(omo=omo, omr=omr, x=x, y=y, terms=terms, rng=rng, obo=obo, obr=obr)


def operators(terms, a, r, A, R):
    return [("matmul", lambda ob: ob.matmul(terms, a)), ("tmatmul", lambda ob: ob.tmatmul(terms, r)),
            ("matmul_gradhyp", lambda ob: ob.matmul_gradhyp(terms, a)), ("tmatmul_gradhyp", lambda ob: ob.tmatmul_gradhyp(terms, r)),
            ("sqmm", lambda ob: ob.sqmm(terms, np.abs(a))), ("sqtmm", lambda ob: ob.sqtmm(terms, r)),
            ("sqcolsums", lambda ob: ob.sqcolsums(terms)), ("sqcolsums_gradhyp", lambda ob: ob.sqcolsums_gradhyp(terms)),
            ("sqmm_gradhyp", lambda ob: ob.sqmm_gradhyp(terms, a)), ("sqtmm_gradhyp", lambda ob: ob.sqtmm_gradhyp(terms, r)),
            ("matmul(mat)", lambda ob: ob.matmul(terms, A)), ("tmatmul(mat)", lambda ob: ob.tmatmul(terms, R)),
            ("getmat", lambda ob: ob.getmat(terms)), ("getbase", lambda ob: ob.getbase(2)),
            ("residvar", lambda ob: ob.residvar(terms)), ("residvar_gradhyp", lambda ob: ob.residvar_gradhyp(terms))]


@pytest.mark.parametrize("name,hyp", [("mat25", [0.3]), ("mat25pow", [-0.4, 0.6]), ("mat25ang", [0.2, -0.5])])
def test_covariances_bitwise(oracle, reference, name, hyp):
    """covf_*::cov / cov_gradhyp, src/covfuncs.cpp:113-347."""
    rng = np.random.default_rng(7)
    hi = 6.28 if name == "mat25ang" else 1.0
    x1, x2 = rng.uniform(0.001, hi, 257), rng.uniform(0.001, hi, 40)
    np.testing.assert_array_equal(oracle.covf_cov(name, hyp, x1, x2), reference.covf_cov(name, hyp, x1, x2))
    np.testing.assert_array_equal(oracle.covf_cov_gradhyp(name, hyp, x1, x2), reference.covf_cov_gradhyp(name, hyp, x1, x2))


@pytest.mark.parametrize("covs", [None, ["mat25pow"] * 8, ["mat25ang", "mat25", "mat25pow", "mat25", "mat25", "mat25", "mat25", "mat25pow"]])
def test_outermod_bitwise(oracle, reference, covs):
    """setcovfs / setknot / hyp_set / build / getvar / getlvar_gradhyp / selectterms / hyplpdf (modandbase.cpp:67-440)."""
    kn = None
    if covs and covs[0] == "mat25ang":
        kn = [np.arange(0.001, 0.999, 0.025)] * 8
        kn[0] = np.linspace(0.05, 6.2, 40)
    omo, x, y, terms, rng = make_problem(oracle, 50, 300, covs=covs, knots=kn)
    omr, *_ = make_problem(reference, 50, 300, covs=covs, knots=kn)
    hyp = omo.gethyp() + 0.05 * np.cos(np.arange(omo.gethyp().size))
    omo.updatehyp(hyp); omr.updatehyp(hyp)
    for w in ("knotptst", "hypst", "hypmatch", "gest", "knotptstge", "maxlevel"):
        np.testing.assert_array_equal(omo.index(w), omr.index(w), err_msg=w)
    for w in ("basisvar", "knotpt", "rotmat", "rotmat_gradhyp", "logbasisvar_gradhyp"):
        np.testing.assert_array_equal(omo.real(w), omr.real(w), err_msg=w)
    for K in (1, 20, 300, 1500):
        t = omo.selectterms(K)
        np.testing.assert_array_equal(t, omr.selectterms(K))
        np.testing.assert_array_equal(omo.getvar(t), omr.getvar(t))
        np.testing.assert_array_equal(omo.getlvar_gradhyp(t), omr.getlvar_gradhyp(t))
    for seed in (1, 12345):  # the randomised tie-break (modandbase.cpp:406-409) under the shared SplitMix64 policy
        omo.set_select_seed(seed); omr.set_select_seed(seed)
        np.testing.assert_array_equal(omo.selectterms(400), omr.selectterms(400))
    omo.set_select_seed(0); omr.set_select_seed(0)
    assert omo.hyplpdf(hyp) == omr.hyplpdf(hyp)
    np.testing.assert_array_equal(omo.hyplpdf_grad(hyp), omr.hyplpdf_grad(hyp))


# the reference's own test shapes (tests/testthat/test-obombasic.R, test-obomgrad.R, test-lpdf.R) + one shape that is tall
# (loopsize > 20) with ONE thread: chunksize = 2049 there, so N must exceed 20 * 2049
@pytest.mark.parametrize("N,K", [(15, 20), (200, 100), (10000, 100), (200, 1000), (10000, 2000), (45000, 60)])
def test_kernels_bitwise_with_one_thread(oracle, reference, N, K):
    """outerbase::build + every linalg.h kernel behind the outerbase operators (modandbase.cpp:547-922, linalg.cpp:57-715)."""
    P = both(oracle, reference, N, K, threads=1)
    assert P["obo"].vertpl == (N > 20 * 2049)
    for w in ("basemat", "basemat_gradhyp", "basescale", "basescalemat"):
        np.testing.assert_array_equal(P["obo"].real(w), P["obr"].real(w), err_msg=w)
    rng, terms = P["rng"], P["terms"]
    a = np.sqrt(P["omo"].getvar(terms) / 20) * rng.normal(size=K)
    r = rng.normal(size=N)
    A, R = np.asfortranarray(rng.normal(size=(K, 5))), np.asfortranarray(rng.normal(size=(N, 3)))
    for name, f in operators(terms, a, r, A, R):
        np.testing.assert_array_equal(f(P["obo"]), f(P["obr"]), err_msg=name)


@pytest.mark.parametrize("N,K", [(200, 100), (10000, 100), (10000, 2000)])
def test_kernels_with_all_threads(oracle, reference, N, K):
    """Default thread count (omp_get_num_procs, modandbase.cpp:464): row-local results stay bitwise, reductions over
    thread-local partial sums agree to rounding (the reference itself is not run-to-run reproducible there)."""
    threads = max(2, os.cpu_count() or 2)
    if N >= 10000:
        P = both(oracle, reference, N, K, threads=threads)
        assert P["obr"].vertpl or threads > 12  # row-chunk ("tall") branch
    else:
        # a short basis built by several threads races on basescale in the reference (modandbase.cpp:600-607, SURVEY 2.3):
        # build with one thread, then run the term-parallel ("wide") kernels with all of them
        P = both(oracle, reference, N, K, threads=1)
        P["obo"].nthreads = threads; P["obr"].nthreads = threads
        assert not P["obr"].vertpl
    rng, terms = P["rng"], P["terms"]
    a, r = rng.normal(size=K), rng.normal(size=N)
    A, R = np.asfortranarray(rng.normal(size=(K, 5))), np.asfortranarray(rng.normal(size=(N, 3)))
    # tall branch: every row is owned by one thread; wide branch: even Phi a sums thread-local vectors (linalg.cpp:77-92)
    row_local = {"matmul", "matmul_gradhyp", "sqmm", "sqmm_gradhyp", "matmul(mat)", "getmat", "getbase", "residvar", "residvar_gradhyp"} if P["obr"].vertpl else {"getmat", "getbase"}
    for name, f in operators(terms, a, r, A, R):
        u, v = f(P["obo"]), f(P["obr"])
        if name in row_local:
            np.testing.assert_array_equal(u, v, err_msg=name)
        elif name == "residvar":  # 1 - sqmm(...) (modandbase.cpp:889-896): the 1 cancels, rounding of the sums is absolute
            assert np.abs(u - v).max() < 1e-14, name
        else:
            assert relerr(u, v) < 1e-13, name


@pytest.mark.parametrize("N,K", [(200, 100), (10000, 100), (45000, 60)])
def test_stateless_seam_bitwise(oracle, reference, N, K):
    """The eight free functions of src/linalg.h:9-58 called directly (the reference's own symbols behind ref_prodmm_vec
    ...) on shared matrices: row-local ones bitwise, reductions to rounding (the seam runs with all threads)."""
    P = both(oracle, reference, N, K, threads=1)
    ob, om = P["obo"], P["omo"]
    bm, bs, bg = ob.real("basemat"), ob.real("basescale"), ob.real("basemat_gradhyp")
    kp, gest, hm = om.index("knotptst"), om.index("gest"), om.index("hypmatch")
    rng, terms = P["rng"], P["terms"]
    a, r = rng.normal(size=K), rng.normal(size=N)
    A, R = np.asfortranarray(rng.normal(size=(K, 4))), np.asfortranarray(rng.normal(size=(N, 4)))
    T = os.cpu_count() or 1  # the seam derives its tuning like setloopvals_ with omp_get_num_procs() threads
    chunk = max(32, min(1 + 2048 // T, N // (4 * T) + 1))
    tall = (N + chunk - 1) // chunk > 20

    def same(u, v, what):  # tall: each row belongs to one thread; wide: thread-local vectors are summed in arrival order
        if tall or T == 1:
            np.testing.assert_array_equal(u, v, err_msg=what)
        else:
            assert relerr(u, v) < 1e-13, what
    same(oracle.prodmm(terms, a, bm, bs, kp), reference.prodmm(terms, a, bm, bs, kp), "prodmm_")
    same(oracle.prodmm(terms, A, bm, bs, kp), reference.prodmm(terms, A, bm, bs, kp), "prodmm_(mat)")
    np.testing.assert_array_equal(oracle.getm(terms, bm, bs, kp), reference.getm(terms, bm, bs, kp))
    assert relerr(oracle.tprodmm(terms, r, bm, bs, kp), reference.tprodmm(terms, r, bm, bs, kp)) < 1e-14
    assert relerr(oracle.tprodmm(terms, R, bm, bs, kp), reference.tprodmm(terms, R, bm, bs, kp)) < 1e-14
    uo, ug = oracle.prodmmge(terms, a, bm, bs, kp, bg, gest, hm)
    vo, vg = reference.prodmmge(terms, a, bm, bs, kp, bg, gest, hm)
    same(uo, vo, "prodmmge_ out"); same(ug, vg, "prodmmge_ outge")
    uo, ug = oracle.tprodmmge(terms, r, bm, bs, kp, bg, gest, hm)
    vo, vg = reference.tprodmmge(terms, r, bm, bs, kp, bg, gest, hm)
    assert relerr(uo, vo) < 1e-13 and relerr(ug, vg) < 1e-13


def _lpdfs(lib, om, terms, y, x, order, threads):
    loglik, logpr = lib.loglik_gauss(om, terms, y, x), lib.logpr_gauss(om, terms)
    loglik.setnthreads(threads)
    loglik.updateom()  # rebuild the basis with that thread count
    vec = lib.lpdfvec(logpr, loglik) if order == "prior_first" else lib.lpdfvec(loglik, logpr)
    return loglik, logpr, vec


@pytest.mark.parametrize("order", ["prior_first", "loglik_first"])
@pytest.mark.parametrize("N,K", [(200, 100), (10000, 100), (200, 1000)])
def test_lpdf_family_and_optcg_bitwise(oracle, reference, N, K, order):
    """loglik_gauss, logpr_gauss, lpdfvec (both child orders, marginal adjustment) and lpdf::optcg -- src/fit.cpp:37-96,
    174-428, src/lpdfs/loglik_gauss.cpp, logpr_gauss.cpp -- at the shapes of tests/testthat/test-lpdf.R, one thread."""
    knots = [np.arange(0.001, 0.999, 0.05)] * 8
    omo, x, y, terms, rng = make_problem(oracle, N, K, covs=["mat25"] * 8, knots=knots)
    omr, *_ = make_problem(reference, N, K, covs=["mat25"] * 8, knots=knots)
    O, R = _lpdfs(oracle, omo, terms, y, x, order, 1), _lpdfs(reference, omr, terms, y, x, order, 1)
    coeff, g = rng.normal(size=K) / 100, rng.normal(size=K)
    for (lk, pr, vec) in (O, R):
        for l in (lk, pr, vec):
            l.compute_gradhyp = True; l.compute_gradpara = True
        lk.updatepara([np.log(0.1)])
        lk.update(coeff); pr.update(coeff)
    for i, name in enumerate(("loglik_gauss", "logpr_gauss")):
        o, r = O[i], R[i]
        assert o.val == r.val, name
        for f in ("grad", "gradhyp", "gradpara", "para"):
            np.testing.assert_array_equal(getattr(o, f), getattr(r, f), err_msg=f"{name}.{f}")
        np.testing.assert_array_equal(o.hessmult(g), r.hessmult(g), err_msg=name)
        np.testing.assert_array_equal(o.diaghess(), r.diaghess(), err_msg=name)
        np.testing.assert_array_equal(o.diaghessgradhyp(), r.diaghessgradhyp(), err_msg=name)
        np.testing.assert_array_equal(o.diaghessgradpara(), r.diaghessgradpara(), err_msg=name)
    np.testing.assert_array_equal(O[0].yhat, R[0].yhat)
    np.testing.assert_array_equal(O[1].coeffsd, R[1].coeffsd)
    vo, vr = O[2], R[2]
    for domarg in (True, False):
        vo.domarg = domarg; vr.domarg = domarg
        para = np.array(vo.para) + 0.1
        vo.updatepara(para); vr.updatepara(para)
        vo.set_coeff(np.zeros(K)); vr.set_coeff(np.zeros(K))
        vo.optcg(0.001, 100); vr.optcg(0.001, 100)
        assert vo.cg_iters == vr.cg_iters and vo.cg_iters > 0
        assert vo.val == vr.val
        for f in ("coeff", "grad", "gradhyp", "gradpara"):
            np.testing.assert_array_equal(getattr(vo, f), getattr(vr, f), err_msg=f"lpdfvec.{f} domarg={domarg}")
        assert vo.paralpdf(para) == vr.paralpdf(para)
        np.testing.assert_array_equal(vo.paralpdf_grad(para), vr.paralpdf_grad(para))
    # pred_gauss::update builds its outerbase with omp_get_num_procs() threads (loglik_gauss.cpp:214-218): 333 rows are a
    # "short" basis where the reference races on basescale (modandbase.cpp:600-607, SURVEY 2.3) -- one CPU for the duration
    with one_cpu():
        po, pr_ = oracle.predictor(O[0]), reference.predictor(R[0])
        xn = np.asfortranarray(np.random.default_rng(5).uniform(size=(333, 8)))
        po.update(xn); pr_.update(xn)
        np.testing.assert_array_equal(po.mean(), pr_.mean())
        np.testing.assert_array_equal(po.var(), pr_.var())


@pytest.mark.parametrize("N,K", [(300, 40), (2000, 150)])
def test_loglik_gda_bitwise(oracle, reference, N, K):
    """loglik_gda + pred_gda (src/lpdfs/loglik_gda.cpp:47-283): obfit's stage-1 model, one thread."""
    knots = [np.arange(0.001, 0.999, 0.05)] * 8
    out = {}
    for name, lib in (("o", oracle), ("r", reference)):
        om, x, y, terms, rng = make_problem(lib, N, K, covs=["mat25"] * 8, knots=knots)
        lk = lib.loglik_gda(om, terms, y, x)
        lk.setnthreads(1); lk.updateom()
        lk.compute_gradhyp = True; lk.compute_gradpara = True
        c, g = rng.normal(size=K) / 50, rng.normal(size=K)
        lk.updatepara([np.log(0.2), -0.5])
        lk.update(c)
        first = dict(val=lk.val, grad=np.array(lk.grad), gradhyp=np.array(lk.gradhyp), gradpara=np.array(lk.gradpara), yhat=np.array(lk.yhat),
                     hm=lk.hessmult(g), dh=lk.diaghess(), dhh=lk.diaghessgradhyp(), dhp=lk.diaghessgradpara())
        vec = lib.lpdfvec(lib.logpr_gauss(om, terms), lk)
        vec.optcg(0.001, 100)
        first.update(vval=vec.val, vcoeff=np.array(vec.coeff), iters=vec.cg_iters, vgh=np.array(vec.gradhyp), vgp=np.array(vec.gradpara))
        out[name] = first
    for k, v in out["o"].items():
        np.testing.assert_array_equal(v, out["r"][k], err_msg=k)


def _loglik_std_results(lib, N, K):
    knots = [np.arange(0.001, 0.999, 0.05)] * 8
    om, x, y, terms, rng = make_problem(lib, N, K, covs=["mat25"] * 8, knots=knots)
    lk, pr = lib.loglik_std(om, terms, y, x), lib.logpr_gauss(om, terms)
    c, g = rng.normal(size=K) / 50, rng.normal(size=K)
    for l in (lk, pr):
        l.compute_gradhyp = True; l.compute_gradpara = True
    lk.updatepara([np.log(0.2)])
    lk.update(c); pr.update(c)
    res = dict(val=lk.val, grad=np.array(lk.grad), gradhyp=np.array(lk.gradhyp), gradpara=np.array(lk.gradpara), yhat=np.array(lk.yhat),
               hm=lk.hessmult(g), dh=lk.diaghess(), dhh=lk.diaghessgradhyp(), dhp=lk.diaghessgradpara(),
               hess=lk.hess(), hgh=lk.hessgradhyp(), hgp=lk.hessgradpara(),
               pr_hess=pr.hess(), pr_hgh=pr.hessgradhyp(), pr_hgp=pr.hessgradpara())
    assert res["hess"].shape == (K, K) and res["hgh"].shape == (K, K, lk._sizes()[2]) and res["hgp"].shape == (K, K, 1)
    vec = lib.lpdfvec(lk, pr)
    for domarg in (True, False):
        vec.domarg = domarg
        vec.updatepara(np.array(vec.para) + 0.05)
        vec.set_coeff(np.zeros(K))
        vec.optnewton()
        res.update({f"v{domarg}_val": vec.val, f"v{domarg}_coeff": np.array(vec.coeff), f"v{domarg}_grad": np.array(vec.grad),
                    f"v{domarg}_gradhyp": np.array(vec.gradhyp), f"v{domarg}_gradpara": np.array(vec.gradpara),
                    f"v{domarg}_tothess": vec.tothess, f"v{domarg}_hess": vec.hess()})
    # a Newton step on a quadratic lands on the optimum: the gradient vanishes
    assert np.abs(vec.grad).max() < 1e-6 * np.abs(res["grad"]).max()
    pd = lib.predictor(lk)
    res.update(pm0=pd.mean(), pv0=pd.var())
    xn = np.asfortranarray(np.random.default_rng(5).uniform(size=(77, 8)))
    pd.update(xn)
    res.update(pm=pd.mean(), pv=pd.var())
    # objects without a full Hessian return empty matrices (fit.h:86-88)
    lg = lib.loglik_gauss(om, terms, y, x)
    assert lg.hess().size == 0 and lg.hessgradhyp().size == 0
    return res


@pytest.mark.parametrize("N,K", [(200, 60), (600, 150)])
def test_loglik_std_optnewton_full_hessian(oracle, reference, N, K):
    """loglik_std + predr_std (src/lpdfs/loglik_std.cpp:41-257), logpr_gauss::hess* (logpr_gauss.cpp:153-186), the
    full-Hessian branch of lpdfvec::buildhess (fit.cpp:269-299) and lpdf::optnewton (fit.cpp:98-131), as
    vignettes/learning.Rmd:92-160 uses them.  loglik_std has no setnthreads: its basis (and every predictor's) is built
    with omp_get_num_procs() threads, where the reference's short-basis branch races on basescale (modandbase.cpp:600-607)
    -- the process is pinned to one CPU for the duration (conftest.one_cpu).  1e-12: the dense products differ in order.
    N <= 600 keeps the basis unchunked -- getmge_'s chunked branch cannot work (linalg.cpp:788-810)."""
    out = {}
    for name, lib in (("o", oracle), ("r", reference)):
        with one_cpu():  # loglik_std and predr_std build their bases with omp_get_num_procs() threads: see conftest.one_cpu
            out[name] = _loglik_std_results(lib, N, K)
    for k, v in out["o"].items():
        if k.endswith("_grad"):  # the gradient AT the optimum is rounding noise: absolute, on the scale of the first gradient
            assert np.abs(v - out["r"][k]).max() < 1e-10 * np.abs(out["o"]["grad"]).max(), k
        else:
            assert relerr(v, out["r"][k]) < 1e-12, k


@pytest.mark.parametrize("N,K", [(200, 60), (600, 150)])
def test_getmge_bitwise(oracle, reference, N, K):
    """getmge_ (src/linalg.cpp:724-822, the eighth function of linalg.h) and outerbase::getmat_gradhyp on unchunked
    bases: bit for bit on shared inputs; each slice is the derivative of getmat in one hyper-parameter (finite
    differences of the basis)."""
    o = both(oracle, reference, N, K, threads=1)
    terms = o["terms"]
    go, gr = o["obo"].getmat_gradhyp(terms), o["obr"].getmat_gradhyp(terms)
    H = o["omo"].sizes()[1]
    assert go.shape == (N, K, H)
    np.testing.assert_array_equal(go, gr)
    ob = o["obo"]
    bm, bs, bg = ob.real("basemat"), ob.real("basescale"), ob.real("basemat_gradhyp")
    kp, gest, hm = o["omo"].index("knotptst"), o["omo"].index("gest"), o["omo"].index("hypmatch")
    so, sr = oracle.getmge(terms, bm, bs, kp, bg, gest, hm), reference.getmge(terms, bm, bs, kp, bg, gest, hm)
    np.testing.assert_array_equal(so, sr)
    np.testing.assert_array_equal(so, go)
    # slice h against a central difference of getmat in hyper-parameter h
    hyp = o["omo"].gethyp()
    h, eps = 3, 1e-6
    mats = []
    for sgn in (+1, -1):
        hp = hyp.copy(); hp[h] += sgn * eps
        o["omo"].updatehyp(hp); ob.build()
        mats.append(ob.getmat(terms))
    o["omo"].updatehyp(hyp); ob.build()
    fd = (mats[0] - mats[1]) / (2 * eps)
    assert relerr(go[:, :, h], fd) < 1e-3  # sanity only: the reference differentiates its eigenbasis approximately


@pytest.mark.parametrize("N,K", [(200, 60), (600, 150)])
def test_loglik_std_matches_loglik_gauss(oracle, N, K):
    """The two likelihoods are the same model (vignettes/speed.Rmd:66): values, gradients and the diagonal of the Hessian
    of loglik_std agree with loglik_gauss's, and diag(hess) is diaghess."""
    knots = [np.arange(0.001, 0.999, 0.05)] * 8
    om, x, y, terms, rng = make_problem(oracle, N, K, covs=["mat25"] * 8, knots=knots)
    ls, lg = oracle.loglik_std(om, terms, y, x), oracle.loglik_gauss(om, terms, y, x)
    c = rng.normal(size=K) / 50
    for l in (ls, lg):
        l.compute_gradhyp = True; l.compute_gradpara = True
        l.updatepara([np.log(0.3)])
        l.update(c)
    assert abs(ls.val - lg.val) < 1e-12 * abs(lg.val)
    for f in ("grad", "gradhyp", "gradpara", "yhat"):
        assert relerr(getattr(ls, f), getattr(lg, f)) < 1e-12, f
    assert relerr(ls.diaghess(), lg.diaghess()) < 1e-13 and relerr(ls.diaghessgradhyp(), lg.diaghessgradhyp()) < 1e-12
    assert relerr(np.diag(ls.hess()), ls.diaghess()) < 1e-14
    hgh = ls.hessgradhyp()
    assert relerr(np.stack([np.diag(hgh[:, :, h]) for h in range(hgh.shape[2])], axis=1), ls.diaghessgradhyp()) < 1e-12
    g = rng.normal(size=K)
    assert relerr(ls.hess() @ g, ls.hessmult(g)) < 1e-12


def test_blas_flavour_sensitivity(oracle, reference, reference_noblas):
    """What the unpinned BLAS under Armadillo is worth.  On SHARED basis matrices the linalg.h kernels do not depend on
    it beyond rounding; the basis build does (rotmat columns are divided by eigenvalues decaying like j^-6: SURVEY 7)."""
    P = both(oracle, reference, 2000, 150, threads=1)
    omn, *_ = make_problem(reference_noblas, 2000, 150)
    np.testing.assert_array_equal(P["omr"].real("rotmat"), omn.real("rotmat"))  # no inner products before the gradients
    obn = reference_noblas.outerbase(omn, P["x"]); obn.nthreads = 1; obn.build()
    bm_r, bm_n = P["obr"].real("basemat"), obn.real("basemat")
    kp = P["omr"].index("knotptst")
    low = np.concatenate([np.arange(kp[l], kp[l] + 6) for l in range(8)])  # levels 0..5 of every dimension
    assert relerr(bm_n[:, low], bm_r[:, low]) < 1e-9
    assert relerr(bm_n, bm_r) < 1e-2  # high levels: conditioning, not a bug -- hence parity is staged on shared inputs
    terms, rng = P["terms"], P["rng"]
    a, r = rng.normal(size=150), rng.normal(size=2000)
    bs, bg = P["obr"].real("basescale"), P["obr"].real("basemat_gradhyp")
    gest, hm = P["omr"].index("gest"), P["omr"].index("hypmatch")
    np.testing.assert_array_equal(reference.prodmm(terms, a, bm_r, bs, kp), reference_noblas.prodmm(terms, a, bm_r, bs, kp))
    assert relerr(reference.tprodmm(terms, r, bm_r, bs, kp), reference_noblas.tprodmm(terms, r, bm_r, bs, kp)) < 1e-14
    assert relerr(reference.tprodmmge(terms, r, bm_r, bs, kp, bg, gest, hm)[1], reference_noblas.tprodmmge(terms, r, bm_r, bs, kp, bg, gest, hm)[1]) < 1e-13


def test_bfgs_driver_on_the_reference(oracle, reference):
    """The R-level driver restated in outerbase_b200/fitting.py (BFGS_lpdf, R/outersupport.R:30-226) over the reference's
    own classes and over the oracle: same iterates => same optimum (one thread for determinism)."""
    from outerbase_b200 import fitting
    res = {}
    for name, lib in (("o", oracle), ("r", reference)):
        om, x, y, terms, rng = make_problem(lib, 400, 60, covs=["mat25"] * 8, knots=[np.arange(0.001, 0.999, 0.05)] * 8)
        lk = lib.loglik_gauss(om, terms, y, x)
        lk.setnthreads(1); lk.updateom()
        vec = lib.lpdfvec(lib.logpr_gauss(om, terms), lk)
        vec.domarg = True
        out = fitting.BFGS_lpdf(om, vec)
        res[name] = (out["optid"]["val"], np.array(out["parlist"]["hyp"]), np.array(out["parlist"]["para"]))
    assert res["o"][0] == res["r"][0]
    np.testing.assert_array_equal(res["o"][1], res["r"][1])
    np.testing.assert_array_equal(res["o"][2], res["r"][2])
