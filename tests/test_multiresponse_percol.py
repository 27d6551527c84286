"""Per-column para for the multi-response objects (include/outerbase_b200_multi_percol.h): each response column with its
own noise scale (loglik_gauss_multi) and coefficient scale (logpr_gauss_multi).

The reference is the definition written out: C single-response oracle objects, each at its own para
(tests/multiresponse_percol_reference.py).  GPU: the product's objects, column-batched CG and predictor against it."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import make_problem, relerr
from multiresponse_percol_reference import Reference
from outerbase_b200 import fitting

REPO = Path(__file__).resolve().parents[1]
N_REF, K_REF = 2000, 150
# (prior per column, likelihood per column): both, the noise alone, the coefficient scale alone
FORMS = [(True, True), (False, True), (True, False)]


def responses(x, y, C, seed=3):
    """C seeded responses at the same inputs whose noise levels differ from column to column (sd 0.02 to 0.32 on a
    unit-variance signal), so that each column's own noise scale matters"""
    rng = np.random.default_rng(seed)
    Y = np.empty((x.shape[0], C), order="F")
    for c in range(C):
        f = 1.0 + 0.5 * np.sin(1.7 * c)
        Y[:, c] = (f * y + (0.2 * (c % 5)) * np.cos(np.pi * (c + 1) * x[:, c % x.shape[1]])
                   + (0.02 + 0.1 * (c % 4)) * rng.normal(size=y.size))
    return Y


def objects(lib, N, K, C, seed=3):
    om, x, y, terms, rng = make_problem(lib, N, K)
    return om, x, responses(x, y, C, seed), terms, rng


def paras(C, lik_default, seed=11):
    """per-column (prior, likelihood) para near the defaults, every entry different"""
    rng = np.random.default_rng(seed)
    return 6.0 + rng.uniform(-1, 1, C), np.asarray(lik_default) + rng.uniform(-0.7, 0.7, C)


def vec_para(pp, pl, form, prior_first=True):
    """the lpdfvec's para for a form: a shared child takes the first column's entry"""
    a = pp if form[0] else pp[:1]
    b = pl if form[1] else pl[:1]
    return np.concatenate([a, b] if prior_first else [b, a])


def _flags(obj, on=True):
    obj.compute_val = on; obj.compute_grad = on; obj.compute_gradhyp = on; obj.compute_gradpara = on


def _update_all(obj, coeff):
    _flags(obj); obj.update(coeff)
    return obj.val, np.array(obj.grad), np.array(obj.gradhyp), np.array(obj.gradpara)


# ---------------------------------------------------------------------------------------------------- CPU
def test_product_exports_the_per_column_abi(product_symbols):
    import outerbase_b200 as ob
    syms = ob.header_symbols(ob.PERCOL_HEADER)
    assert syms == ["ob_loglik_gauss_multi_create_ex", "ob_logpr_gauss_multi_create_ex"]
    assert all(product_symbols.has(s) for s in syms)


def test_reference_is_the_single_response_model_per_column(oracle):
    """column c of the reference is the oracle's single-response object at column c's own para"""
    ref = Reference(oracle)
    C = 3
    om, x, Y, terms, rng = objects(oracle, 500, 40, C)
    lk = ref.loglik_gauss_multi(om, terms, Y, x, para_per_column=True)
    pr = ref.logpr_gauss_multi(om, terms, C, para_per_column=True)
    pp, pl = paras(C, lk.para)
    lk.updatepara(pl); pr.updatepara(pp)
    A = rng.normal(size=(40, C)) / 30
    got = _update_all(lk, A)
    for c in range(C):
        one = oracle.loglik_gauss(om, terms, Y[:, c], x)
        one.updatepara([pl[c]])
        v, g, _, gp = _update_all(one, A[:, c])
        np.testing.assert_array_equal(got[1][:, c], g)
        assert got[3][c] == gp[0]
        np.testing.assert_array_equal(lk.diaghess()[c * 40:(c + 1) * 40], one.diaghess())
    assert got[3].shape == (C,)
    for form in FORMS:
        vec = ref.lpdfvec(ref.logpr_gauss_multi(om, terms, C, para_per_column=form[0]),
                          ref.loglik_gauss_multi(om, terms, Y, x, para_per_column=form[1]))
        vec.domarg = True
        vec.updatepara(vec_para(pp, pl, form))
        vec.optcg(0.001, 100)
        for c in range(C):
            single = oracle.lpdfvec(oracle.logpr_gauss(om, terms), oracle.loglik_gauss(om, terms, Y[:, c], x))
            single.domarg = True
            single.updatepara([pp[c] if form[0] else pp[0], pl[c] if form[1] else pl[0]])
            single.optcg(0.001, 100)
            np.testing.assert_array_equal(vec.coeff[:, c], single.coeff)
            assert vec.cg_iters_per_column[c] == single.cg_iters


def test_para_layout_defaults_and_paralpdf(oracle):
    ref = Reference(oracle)
    C = 4
    om, x, Y, terms, _ = objects(oracle, 300, 30, C)
    lk = ref.loglik_gauss_multi(om, terms, Y, x, para_per_column=True)
    pr = ref.logpr_gauss_multi(om, terms, C, para_per_column=True)
    defaults = [oracle.loglik_gauss(om, terms, Y[:, c], x).para[0] for c in range(C)]
    np.testing.assert_array_equal(lk.para, defaults)
    np.testing.assert_allclose(lk.para, np.log(0.01 * np.var(Y, axis=0, ddof=1)), rtol=1e-13)
    np.testing.assert_array_equal(lk.paravar, np.ones(C))
    np.testing.assert_array_equal(pr.para, np.full(C, 6.0))
    np.testing.assert_array_equal(pr.paravar, np.full(C, 4.0))
    shared_lk = ref.loglik_gauss_multi(om, terms, Y, x)
    shared_pr = ref.logpr_gauss_multi(om, terms, C)
    for a, b in ((pr, lk), (lk, pr), (shared_pr, lk), (pr, shared_lk), (lk, shared_pr)):
        vec = ref.lpdfvec(a, b)
        np.testing.assert_array_equal(vec.para, np.concatenate([a.para, b.para]))
        p = vec.para + np.linspace(-0.5, 0.5, vec.para.size)
        want = sum(-0.5 * float(np.sum((q - k.para0) ** 2 / k.paravar))
                   for k, q in ((a, p[:a.para.size]), (b, p[a.para.size:])))
        assert vec.paralpdf(p) == pytest.approx(want, rel=1e-14)
        np.testing.assert_allclose(vec.paralpdf_grad(p), np.concatenate(
            [-(p[:a.para.size] - a.para0) / a.paravar, -(p[a.para.size:] - b.para0) / b.paravar]), rtol=1e-14)
        assert vec.paralpdf(p[:-1]) == -np.inf


def test_wrong_length_para_is_refused_by_the_reference(oracle):
    ref = Reference(oracle)
    om, x, Y, terms, _ = objects(oracle, 200, 20, 3)
    lk = ref.loglik_gauss_multi(om, terms, Y, x, para_per_column=True)
    pr = ref.logpr_gauss_multi(om, terms, 3, para_per_column=True)
    for obj, n in ((lk, 1), (lk, 4), (pr, 2), (ref.lpdfvec(pr, lk), 5)):
        with pytest.raises(ValueError):
            obj.updatepara(np.zeros(n))


def test_obfit_multi_per_column_and_obpred_on_the_reference(oracle):
    rng = np.random.default_rng(5)
    x = np.asfortranarray(rng.uniform(size=(400, 3)))
    f = lambda x: np.column_stack([np.sin(3 * x[:, 0]) + x[:, 1], 10 + 4 * x[:, 2] ** 2 - x[:, 0], np.cos(2 * x[:, 1]) * x[:, 2]])
    Y = f(x) + np.array([0.01, 0.3, 0.05]) * rng.normal(size=(400, 3))
    model = fitting.obfit_multi(Reference(oracle), x, Y, numb=30, numberopts=1, para_per_column=True)
    assert model["logpdf"].para.shape == (6,)
    xt = np.asfortranarray(rng.uniform(size=(100, 3)))
    Yt = f(xt)
    pred = fitting.obpred(model, xt)
    assert pred["mean"].shape == (100, 3) and pred["var"].shape == (100, 3)
    assert np.all(pred["var"] > 0)
    # each column's variance is its own predictor's, scaled by its own y_sca^2
    raw = model["predobj"].var()
    np.testing.assert_allclose(pred["var"], raw * model["y_sca"] ** 2, rtol=1e-15)
    for c in range(3):
        assert np.mean((pred["mean"][:, c] - Yt[:, c]) ** 2) < 0.05 * np.var(Yt[:, c])


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.fixture
def families(gpu):
    """the interpreter kernels (spec 0) and the terms-specialised ones compiled at first use (spec 1)"""
    def run(spec):
        gpu.set_option("spec", spec)
    yield run
    gpu.set_option("spec", 2)


def _build(lib, C, N=N_REF, K=K_REF):
    """the four children (prior / likelihood, shared / per column) and the seeded coefficients and para"""
    om, x, Y, terms, rng = objects(lib, N, K, C)
    kids = {}
    for pc in (False, True):
        kids["pr", pc] = lib.logpr_gauss_multi(om, terms, C, para_per_column=pc)
        kids["lk", pc] = lib.loglik_gauss_multi(om, terms, Y, x, para_per_column=pc)
    pp, pl = paras(C, kids["lk", True].para)
    A = np.asfortranarray(rng.normal(size=(K, C)) / 30)
    g = rng.normal(size=K * C)
    return kids, pp, pl, A, g


def _evaluate(lib, C):
    """everything the per-column objects compute at one seeded point, in a dict keyed by what it is"""
    kids, pp, pl, A, g = _build(lib, C)
    out = {"lk_para0": np.array(kids["lk", True].para)}
    for name, p in (("lk", pl), ("pr", pp)):
        obj = kids[name, True]
        obj.updatepara(p)
        out[name] = _update_all(obj, A) + (obj.hessmult(g), obj.diaghess(), obj.diaghessgradhyp(), obj.diaghessgradpara())
    for form in FORMS:
        for prior_first in (True, False):
            a, b = kids["pr", form[0]], kids["lk", form[1]]
            vec = lib.lpdfvec(a, b) if prior_first else lib.lpdfvec(b, a)
            vec.domarg = True
            vec.updatepara(vec_para(pp, pl, form, prior_first))
            r = _update_all(vec, A)
            first, second = (a, b) if prior_first else (b, a)
            margadj = r[3] - np.concatenate([np.atleast_1d(first.gradpara), np.atleast_1d(second.gradpara)])
            out[form, prior_first] = r + (margadj, vec.hessmult(g), vec.diaghess(), vec.diaghessgradhyp(), vec.diaghessgradpara())
    return out


_REF = {}  # the oracle's loops over the columns, shared by the two kernel families


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("C", [1, 3, 8, 70])
def test_gpu_per_column_objects_match_the_reference(gpu, oracle, families, spec, C):
    """update, hessmult and the Hessian diagonals of both per-column objects and of every lpdfvec form in both child
    orders.  spec 0 forms the lpdfvec's hyper-parameter adjustment from the K x H matrix, spec 1 by the sweep."""
    families(spec)
    if C not in _REF:
        _REF[C] = _evaluate(Reference(oracle), C)
    ref, got = _REF[C], _evaluate(gpu, C)
    np.testing.assert_allclose(got["lk_para0"], ref["lk_para0"], rtol=1e-13)
    for key in ref:
        if key == "lk_para0":
            continue
        gv, ov = got[key], ref[key]
        assert abs(gv[0] - ov[0]) <= 1e-8 * abs(ov[0]), key
        for i in (1, 2, 3):  # grad, gradhyp, gradpara
            assert np.shape(gv[i]) == np.shape(ov[i]), (key, i)
            assert relerr(gv[i], ov[i]) < 1e-8, (key, i)
        products = (4, 5, 7) if key in ("lk", "pr") else (5, 6, 8)  # hessmult, diaghess, diaghessgradpara
        for i in products:
            assert np.shape(gv[i]) == np.shape(ov[i]), (key, i)
            assert relerr(gv[i], ov[i]) < 1e-12, (key, i)
        i = 6 if key in ("lk", "pr") else 7  # a hyper-gradient: the single-response parity tests' tolerance
        assert relerr(gv[i], ov[i]) < 1e-7, (key, i)
        if key not in ("lk", "pr"):
            assert relerr(gv[4], ov[4]) < 1e-8, key  # the marginal adjustment's para gradient


def _optcg(lib, C, form, pp_pl=None, N=N_REF, K=K_REF, prior=None):
    om, x, Y, terms, _ = objects(lib, N, K, C)
    lk = lib.loglik_gauss_multi(om, terms, Y, x, para_per_column=form[1])
    vec = lib.lpdfvec(lib.logpr_gauss_multi(om, terms, C, para_per_column=form[0]), lk)
    vec.domarg = True
    pp, pl = pp_pl or paras(C, lib.loglik_gauss_multi(om, terms, Y, x, para_per_column=True).para)
    if prior is not None:
        pp = np.asarray(prior, dtype=float)
    vec.updatepara(vec_para(pp, pl, form))
    vec.optcg(0.001, 100)
    return vec, (om, x, Y, terms, pp, pl)


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("C,form", [(3, (True, True)), (8, (True, True)), (8, (False, True)), (8, (True, False)), (70, (True, True))])
def test_gpu_per_column_optcg_matches_the_reference(gpu, oracle, families, spec, C, form):
    families(spec)
    vec, _ = _optcg(gpu, C, form)
    ref, _ = _optcg(Reference(oracle), C, form)
    np.testing.assert_array_equal(vec.cg_iters_per_column, ref.cg_iters_per_column)
    assert relerr(vec.coeff, ref.coeff) < 1e-8
    assert abs(vec.val - ref.val) <= 1e-8 * abs(ref.val)
    assert relerr(vec.gradpara, ref.gradpara) < 1e-8
    assert len(set(vec.cg_iters_per_column.tolist())) > 1, vec.cg_iters_per_column


@pytest.mark.gpu
def test_gpu_columns_stop_at_different_iterations_because_their_noise_differs(gpu, oracle):
    """the same response in every column: with one shared para every column runs the same CG; with noise scales
    e^1.5 apart the columns stop at different iterations, each where its own single-response fit stops"""
    C = 3
    om, x, y, terms, _ = make_problem(gpu, N_REF, K_REF)
    Y = np.asfortranarray(np.column_stack([y] * C))
    shared = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, C), gpu.loglik_gauss_multi(om, terms, Y, x))
    shared.domarg = True
    shared.optcg(0.001, 100)
    assert len(set(shared.cg_iters_per_column.tolist())) == 1
    lk = gpu.loglik_gauss_multi(om, terms, Y, x, para_per_column=True)
    vec = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, C), lk)
    vec.domarg = True
    pl = lk.para + np.array([0.0, 1.5, 3.0])
    vec.updatepara(np.concatenate([[6.0], pl]))
    vec.optcg(0.001, 100)
    iters = vec.cg_iters_per_column
    assert len(set(iters.tolist())) == C, iters
    omr, xr, yr, termsr, _ = make_problem(oracle, N_REF, K_REF)
    for c in range(C):
        r = oracle.lpdfvec(oracle.logpr_gauss(omr, termsr), oracle.loglik_gauss(omr, termsr, yr, xr))
        r.domarg = True
        r.updatepara([6.0, pl[c]])
        r.optcg(0.001, 100)
        assert iters[c] == r.cg_iters, (c, iters[c], r.cg_iters)
        assert relerr(vec.coeff[:, c], r.coeff) < 1e-8, c


@pytest.mark.gpu
def test_gpu_per_column_launches_per_iteration_equal_the_shared_form(gpu, families):
    families(1)
    per = {}
    for C in (8, 64):
        for pc in (False, True):
            om, x, Y, terms, _ = objects(gpu, N_REF, K_REF, C)
            vec = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, C, para_per_column=pc),
                              gpu.loglik_gauss_multi(om, terms, Y, x, para_per_column=pc))
            vec.optcg(-1.0, 1)  # warm: modules, programs (tol < 0: no column ever stops)
            counts = []
            for epochs in (2, 6):
                vec.set_coeff(np.zeros(K_REF * C))
                n0 = gpu.launch_count()
                vec.optcg(-1.0, epochs)
                counts.append(gpu.launch_count() - n0)
            per[C, pc] = (counts[1] - counts[0]) / 4
    assert per[8, True] == per[8, False] == per[64, True] == per[64, False], per


def test_reference_predictor_of_a_shared_likelihood_under_a_per_column_prior(oracle):
    """each column's total diagonal holds its own prior scale (e^-2 to e^6 here), so the variance is N x C and its
    columns differ"""
    vec, (om, x, Y, terms, pp, pl) = _optcg(Reference(oracle), 3, (True, False), N=300, K=30, prior=[-2.0, 2.0, 6.0])
    p = Reference(oracle).predictor(vec.kids[1])
    p.update(x[:50])
    var = p.var()
    assert var.shape == (50, 3) and relerr(var[:, 0], var[:, 2]) > 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("spec,C,form", [(0, 3, (True, True)), (1, 8, (True, True)), (0, 3, (True, False)),
                                         (1, 8, (True, False)), (0, 3, (False, True))])
def test_gpu_per_column_predictor_matches_single_response_predictors(gpu, families, spec, C, form):
    """spec 1 with eight columns: the variance is one squared tensor-core product.  A shared likelihood under a
    per-column prior also gives one variance per column: the columns' total diagonals differ.  The prior scales span
    e^-2 to e^6, so that they move the variance visibly (by about 5 % between the first and the last column)"""
    families(spec)
    vec, (om, x, Y, terms, pp, pl) = _optcg(gpu, C, form, prior=np.linspace(-2.0, 6.0, C))
    pm = gpu.predictor(vec._children[1])
    xt = np.asfortranarray(np.random.default_rng(9).uniform(size=(700, x.shape[1])))
    pm.update(xt)
    mean, var = pm.mean(), pm.var()
    assert mean.shape == (700, C) and var.shape == (700, C)
    if form[0]:
        assert relerr(var[:, 0], var[:, -1]) > 1e-3
    for c in range(C):
        lk = gpu.loglik_gauss(om, terms, Y[:, c], x)
        v = gpu.lpdfvec(gpu.logpr_gauss(om, terms), lk)
        v.domarg = True
        v.updatepara([pp[c] if form[0] else pp[0], pl[c] if form[1] else pl[0]])
        v.optcg(0.001, 100)
        p = gpu.predictor(lk)
        p.update(xt)
        assert relerr(mean[:, c], p.mean()) < 1e-7, c
        assert relerr(var[:, c], p.var()) < 1e-12, c


@pytest.mark.gpu
def test_gpu_bfgs_on_the_per_column_objective_matches_the_reference(gpu, oracle):
    out = {}
    for name, lib in (("gpu", gpu), ("reference", Reference(oracle))):
        om, x, Y, terms, _ = objects(lib, 800, 60, 3)
        vec = lib.lpdfvec(lib.logpr_gauss_multi(om, terms, 3, para_per_column=True),
                          lib.loglik_gauss_multi(om, terms, Y, x, para_per_column=True))
        vec.domarg = True
        out[name] = fitting.BFGS_lpdf(om, vec)
    g, o = out["gpu"], out["reference"]
    assert g["parlist"]["para"].shape == (6,)
    assert abs(g["optid"]["val"] - o["optid"]["val"]) <= 1e-6 * abs(o["optid"]["val"])
    assert relerr(g["parlist"]["hyp"], o["parlist"]["hyp"]) < 1e-4
    assert relerr(g["parlist"]["para"], o["parlist"]["para"]) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("C", [3, 8])
def test_gpu_equal_entries_give_the_shared_object(gpu, C):
    """a per-column object with every entry at one value is the shared object up to rounding; its per-column gradpara
    sums to the shared one"""
    kids, pp, pl, A, g = _build(gpu, C)
    s = kids["lk", False].para[0]
    kids["lk", True].updatepara(np.full(C, s))
    kids["pr", True].updatepara(np.full(C, 6.0))
    for name in ("lk", "pr"):
        a, b = kids[name, True], kids[name, False]
        ra, rb = _update_all(a, A), _update_all(b, A)
        assert abs(ra[0] - rb[0]) <= 1e-13 * abs(rb[0]), name
        assert relerr(ra[1], rb[1]) < 1e-13 and relerr(ra[2], rb[2]) < 1e-13, name
        assert ra[3].shape == (C,) and abs(ra[3].sum() - rb[3][0]) <= 1e-12 * abs(rb[3][0]), name
        assert relerr(a.hessmult(g), b.hessmult(g)) < 1e-13, name
        np.testing.assert_array_equal(a.diaghess(), b.diaghess())
        assert relerr(a.diaghessgradhyp(), b.diaghessgradhyp()) < 1e-13, name
    va = gpu.lpdfvec(kids["pr", True], kids["lk", True])
    vb = gpu.lpdfvec(kids["pr", False], kids["lk", False])
    for v, p in ((va, np.concatenate([np.full(C, 6.0), np.full(C, s)])), (vb, np.array([6.0, s]))):
        v.domarg = True
        v.updatepara(p)
        v.optcg(0.001, 100)
    np.testing.assert_array_equal(va.cg_iters_per_column, vb.cg_iters_per_column)
    assert relerr(va.coeff, vb.coeff) < 1e-12
    assert abs(va.val - vb.val) <= 1e-12 * abs(vb.val)
    assert relerr(va.gradhyp, vb.gradhyp) < 1e-10
    gpa = va.gradpara
    assert relerr([gpa[:C].sum(), gpa[C:].sum()], vb.gradpara) < 1e-10


@pytest.mark.gpu
def test_gpu_one_column_is_loglik_gauss(gpu):
    om, x, Y, terms, rng = objects(gpu, N_REF, K_REF, 1)
    lk = gpu.loglik_gauss_multi(om, terms, Y, x, para_per_column=True)
    one = gpu.loglik_gauss(om, terms, Y[:, 0], x)
    np.testing.assert_array_equal(lk.para, one.para)
    a = rng.normal(size=K_REF) / 30
    ra, rb = _update_all(lk, a), _update_all(one, a)
    assert abs(ra[0] - rb[0]) <= 1e-13 * abs(rb[0])
    assert relerr(ra[1][:, 0], rb[1]) < 1e-12 and relerr(ra[3], rb[3]) < 1e-12 and relerr(ra[2], rb[2]) < 1e-10
    np.testing.assert_array_equal(lk.diaghess(), one.diaghess())
    np.testing.assert_array_equal(lk.diaghessgradpara(), one.diaghessgradpara())
    va = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, 1, para_per_column=True), lk)
    vb = gpu.lpdfvec(gpu.logpr_gauss(om, terms), one)
    for v in (va, vb):
        v.domarg = True
        v.optcg(0.001, 100)
    assert va.cg_iters_per_column[0] == vb.cg_iters
    assert relerr(va.coeff[:, 0], vb.coeff) < 1e-10
    assert abs(va.val - vb.val) <= 1e-10 * abs(vb.val)
    assert relerr(va.gradpara, vb.gradpara) < 1e-8


@pytest.mark.gpu
def test_gpu_per_column_fit_recovers_each_noise_level(gpu):
    """two columns of one smooth signal with noise sd 0.05 and 0.5: the per-column fit recovers each sd within a
    factor 1.25; the shared fit's one sd (in standardised units) lies between the two"""
    rng = np.random.default_rng(2024)
    N = 3000
    x = np.asfortranarray(rng.uniform(size=(N, 3)))
    s = np.sin(3 * x[:, 0]) + np.cos(2 * x[:, 1]) * x[:, 2] + x[:, 1] ** 2
    s = (s - s.mean()) / s.std()
    sd = np.array([0.05, 0.5])
    Y = np.column_stack([s, s]) + sd * rng.normal(size=(N, 2))
    per = fitting.obfit_multi(gpu, x, Y, numb=80, numberopts=1, para_per_column=True)
    shared = fitting.obfit_multi(gpu, x, Y, numb=80, numberopts=1)
    lp = per["logpdf"].para[2:]  # [prior C | likelihood C]
    est = np.exp(lp) * per["y_sca"]  # back to the response's units
    assert np.all(est / sd < 1.25) and np.all(sd / est < 1.25), (est, sd)
    one = np.exp(shared["logpdf"].para[1])
    assert np.exp(lp[0]) < one < np.exp(lp[1]), (np.exp(lp), one)
    pred = fitting.obpred(per, x[:500])
    assert pred["var"].shape == (500, 2) and np.all(pred["var"][:, 1] > pred["var"][:, 0])


@pytest.mark.gpu
def test_gpu_per_column_bad_input_is_refused(gpu):
    om, x, Y, terms, _ = objects(gpu, 300, 40, 3)
    lk = gpu.loglik_gauss_multi(om, terms, Y, x, para_per_column=True)
    pr = gpu.logpr_gauss_multi(om, terms, 3, para_per_column=True)
    for obj, n in ((lk, 1), (lk, 4), (pr, 1), (pr, 2)):
        with pytest.raises(ValueError):
            obj.updatepara(np.zeros(n))
    vec = gpu.lpdfvec(pr, lk)
    with pytest.raises(ValueError):
        vec.updatepara(np.zeros(5))
    assert vec.paralpdf(np.zeros(5)) == -np.inf
    with pytest.raises(ValueError):
        gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, 2, para_per_column=True), lk)


@pytest.mark.gpu
def test_gpu_per_column_row_sharding_two_ranks(gpu):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("single-GPU box")
    env = dict(os.environ, OMP_NUM_THREADS="2", OMP_WAIT_POLICY="passive")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29563", str(REPO / "tests" / "mgpu_multiresponse_percol_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert "mgpu_multiresponse_percol_worker world=2 OK" in res.stdout
