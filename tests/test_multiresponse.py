"""Multi-response loglik_gauss: C responses on one basis (include/outerbase_b200.h, ob_engine.hpp LoglikGaussMulti).

The reference is the definition itself: C single-response oracle objects and loops over them
(tests/multiresponse_reference.py).  GPU: the product's column-batched objects and CG against it, column by column."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import make_problem, relerr
from multiresponse_reference import Reference
from outerbase_b200 import fitting

REPO = Path(__file__).resolve().parents[1]
N_REF, K_REF = 2000, 150


def responses(x, y, C, seed=3):
    """C seeded responses at the same inputs: the base response scaled, plus a column-dependent smooth term and a
    little noise, so that the columns' CG runs stop after different numbers of iterations."""
    rng = np.random.default_rng(seed)
    Y = np.empty((x.shape[0], C), order="F")
    for c in range(C):
        f = 1.0 + 0.5 * np.sin(1.7 * c)
        Y[:, c] = f * y + (0.2 * (c % 5)) * np.cos(np.pi * (c + 1) * x[:, c % x.shape[1]]) + 0.05 * (c % 3) * rng.normal(size=y.size)
    return Y


def multi_objects(lib, N, K, C, seed=3):
    om, x, y, terms, rng = make_problem(lib, N, K)
    Y = responses(x, y, C, seed)
    return om, x, Y, terms, rng


def _flags(obj, on=True):
    obj.compute_val = on; obj.compute_grad = on; obj.compute_gradhyp = on; obj.compute_gradpara = on


def test_product_exports_the_extension_abi(product_symbols):
    import outerbase_b200 as ob
    syms = ob.header_symbols(ob.MULTI_HEADER)
    assert syms == ["ob_loglik_gauss_multi_create", "ob_logpr_gauss_multi_create"]
    assert all(product_symbols.has(s) for s in syms)


def test_binding_refuses_misaligned_responses(product_symbols):
    from outerbase_b200.binding import loglik_gauss_multi
    x, terms = np.zeros((10, 2)), np.zeros((3, 2), dtype=np.uint64)
    with pytest.raises(ValueError, match="align"):
        loglik_gauss_multi(product_symbols, None, terms, np.zeros((9, 2)), x)
    with pytest.raises(ValueError, match="N x C"):
        loglik_gauss_multi(product_symbols, None, terms, np.zeros(10), x)


def test_reference_is_the_single_response_model_per_column(oracle):
    """the reference's lpdfvec with C = 1 is the oracle's lpdfvec(logpr_gauss, loglik_gauss), and its optcg runs each
    column's own CG (the columns stop at different iterations)"""
    ref = Reference(oracle)
    om, x, Y, terms, _ = multi_objects(oracle, 600, 60, 3)
    vec = ref.lpdfvec(ref.logpr_gauss_multi(om, terms, 3), ref.loglik_gauss_multi(om, terms, Y, x))
    vec.domarg = True
    vec.optcg(0.001, 100)
    assert len(set(vec.cg_iters_per_column.tolist())) > 1, vec.cg_iters_per_column
    one = ref.lpdfvec(ref.logpr_gauss_multi(om, terms, 1), ref.loglik_gauss_multi(om, terms, Y[:, :1], x))
    single = oracle.lpdfvec(oracle.logpr_gauss(om, terms), oracle.loglik_gauss(om, terms, Y[:, 0], x))
    np.testing.assert_allclose(one.para, single.para, rtol=1e-14)
    for v in (one.vecs[0], single):
        v.domarg = True
        v.optcg(0.001, 100)
    np.testing.assert_array_equal(one.vecs[0].coeff, single.coeff)


def test_obfit_multi_and_obpred_on_the_reference(oracle):
    rng = np.random.default_rng(5)
    x = np.asfortranarray(rng.uniform(size=(400, 3)))
    f = lambda x: np.column_stack([np.sin(3 * x[:, 0]) + x[:, 1], 10 + 4 * x[:, 2] ** 2 - x[:, 0], np.cos(2 * x[:, 1]) * x[:, 2]])
    model = fitting.obfit_multi(Reference(oracle), x, f(x), numb=30, numberopts=1)
    xt = np.asfortranarray(rng.uniform(size=(100, 3)))
    Yt = f(xt)
    pred = fitting.obpred(model, xt)
    assert pred["mean"].shape == (100, 3) and pred["var"].shape == (100, 3)
    assert np.all(pred["var"] > 0)
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


def _update_all(obj, coeff):
    _flags(obj); obj.update(coeff)
    return obj.val, np.array(obj.grad), np.array(obj.gradhyp), np.array(obj.gradpara)


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("C", [1, 3, 8, 64, 70])
def test_gpu_update_and_products_match_the_oracle(gpu, oracle, families, spec, C):
    families(spec)
    res = {}
    for name, lib in (("gpu", gpu), ("reference", Reference(oracle))):
        om, x, Y, terms, rng = multi_objects(lib, N_REF, K_REF, C)
        A = np.asfortranarray(rng.normal(size=(K_REF, C)) / 30)
        lk = lib.loglik_gauss_multi(om, terms, Y, x)
        g = rng.normal(size=K_REF * C)
        res[name] = _update_all(lk, A) + (lk.hessmult(g), lk.diaghess(), lk.diaghessgradhyp(), lk.para)
    gv, ov = res["gpu"], res["reference"]
    assert abs(gv[0] - ov[0]) <= 1e-8 * abs(ov[0])
    for i in (1, 2, 3):
        assert relerr(gv[i], ov[i]) < 1e-8, i
    for i in (4, 5):  # products
        assert relerr(gv[i], ov[i]) < 1e-12, i
    assert relerr(gv[6], ov[6]) < 1e-7  # a hyper-gradient: the single-response parity tests' tolerance
    np.testing.assert_allclose(gv[7], ov[7], rtol=1e-13)


_C3_REF = {}  # the oracle's loop over the columns, shared by the two kernel families


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("C", [8, 70])
def test_gpu_update_on_the_c3_table(gpu, oracle, families, spec, C):
    """>= 20k rows of bench.py's C3 model (d = 10, K = 2000); the oracle side is the definition's loop, one
    single-response object at a time (C oracle bases would not fit in host memory)"""
    import bench
    families(spec)
    N = 20_000
    x = bench.synth_rows(0, N, 10)
    base = bench.wingweight(x)
    base = (base - base.mean()) / base.std()
    Y = responses(x, base, C)
    om, terms = bench.setup_model(gpu)
    A = np.asfortranarray(np.random.default_rng(1).normal(size=(terms.shape[0], C)) / 100)
    para = gpu.loglik_gauss_multi(om, terms, Y[:, :1], x).para  # any fixed para: both sides use the same
    if C not in _C3_REF:
        omr, termsr = bench.setup_model(oracle)
        np.testing.assert_array_equal(terms, termsr)
        val, grad, gh, gp = 0.0, [], 0.0, 0.0
        for c in range(C):
            lk = oracle.loglik_gauss(omr, termsr, Y[:, c], x)
            lk.updatepara(para)
            v, g, h, p = _update_all(lk, A[:, c])
            val += v; grad.append(g); gh = gh + h; gp = gp + p
        _C3_REF[C] = (val, np.column_stack(grad), gh, gp)
    val, grad, gh, gp = _C3_REF[C]
    lkg = gpu.loglik_gauss_multi(om, terms, Y, x)
    lkg.updatepara(para)
    gv = _update_all(lkg, A)
    assert abs(gv[0] - val) <= 1e-8 * abs(val)
    assert relerr(gv[1], grad) < 1e-8
    assert relerr(gv[2], gh) < 1e-8
    assert relerr(gv[3], gp) < 1e-8


def _optcg_columns(lib, C, N=N_REF, K=K_REF):
    om, x, Y, terms, rng = multi_objects(lib, N, K, C)
    vec = lib.lpdfvec(lib.logpr_gauss_multi(om, terms, C), lib.loglik_gauss_multi(om, terms, Y, x))
    vec.domarg = True
    vec.optcg(0.001, 100)
    return vec, (om, x, Y, terms)


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("C", [3, 8, 70])
def test_gpu_optcg_is_c_independent_runs(gpu, oracle, families, spec, C):
    families(spec)
    vec, (om, x, Y, terms) = _optcg_columns(gpu, C)
    iters = vec.cg_iters_per_column
    omr, xr, Yr, termsr, _ = multi_objects(oracle, N_REF, K_REF, C)
    para = vec.para
    for c in range(C):
        ref = oracle.lpdfvec(oracle.logpr_gauss(omr, termsr), oracle.loglik_gauss(omr, termsr, Yr[:, c], xr))
        ref.domarg = True
        ref.updatepara(para)
        ref.optcg(0.001, 100)
        assert iters[c] == ref.cg_iters, (c, iters[c], ref.cg_iters)
        assert relerr(vec.coeff[:, c], ref.coeff) < 1e-8, c
    assert len(set(iters.tolist())) > 1, iters  # columns froze at different iterations and stayed frozen
    # the whole log-density is the sum of the columns' (each with its own marginal adjustment)
    refs = []
    for c in range(C):
        r = oracle.lpdfvec(oracle.logpr_gauss(omr, termsr), oracle.loglik_gauss(omr, termsr, Yr[:, c], xr))
        r.domarg = True; r.updatepara(para); r.set_coeff(vec.coeff[:, c])
        _flags(r); r.update(vec.coeff[:, c])
        refs.append(r.val)
    assert abs(vec.val - sum(refs)) <= 1e-8 * abs(vec.val)
    # two runs from the same start are bit-identical
    first = vec.coeff.copy()
    vec.set_coeff(np.zeros(K_REF * C)); vec.optcg(0.001, 100)
    np.testing.assert_array_equal(vec.coeff, first)
    np.testing.assert_array_equal(vec.cg_iters_per_column, iters)


@pytest.mark.gpu
def test_gpu_launches_per_iteration_do_not_grow_with_c(gpu, families):
    """On a specialised table the products of C = 8 and C = 64 are single tensor-core passes: the same launches per
    CG iteration (a column loop would launch 8x more)."""
    families(1)
    per = {}
    for C in (8, 64):
        om, x, Y, terms, _ = multi_objects(gpu, N_REF, K_REF, C)
        vec = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, C), gpu.loglik_gauss_multi(om, terms, Y, x))
        vec.optcg(-1.0, 1)  # warm: modules, programs (tol < 0: no column ever stops)
        counts = []
        for epochs in (2, 6):
            vec.set_coeff(np.zeros(K_REF * C))
            n0 = gpu.launch_count()
            vec.optcg(-1.0, epochs)
            counts.append(gpu.launch_count() - n0)
        per[C] = (counts[1] - counts[0]) / 4
    assert per[8] == per[64], per


@pytest.mark.gpu
def test_gpu_predictor_matches_single_response_predictors(gpu):
    C = 3
    vec, (om, x, Y, terms) = _optcg_columns(gpu, C)
    lkm = vec._children[1]
    pm = gpu.predictor(lkm)
    xt = np.asfortranarray(np.random.default_rng(9).uniform(size=(700, x.shape[1])))
    pm.update(xt)
    mean, var = pm.mean(), pm.var()
    assert mean.shape == (700, C) and var.shape == (700,)
    for c in range(C):
        lk = gpu.loglik_gauss(om, terms, Y[:, c], x)
        v = gpu.lpdfvec(gpu.logpr_gauss(om, terms), lk)
        v.domarg = True
        v.updatepara(vec.para)
        v.optcg(0.001, 100)
        p = gpu.predictor(lk)
        p.update(xt)
        assert relerr(mean[:, c], p.mean()) < 1e-7, c
        assert relerr(var, p.var()) < 1e-12, c


@pytest.mark.gpu
def test_gpu_bfgs_on_the_multi_objective_matches_the_oracle(gpu, oracle):
    out = {}
    for name, lib in (("gpu", gpu), ("oracle", Reference(oracle))):
        om, x, Y, terms, _ = multi_objects(lib, 800, 60, 3)
        vec = lib.lpdfvec(lib.logpr_gauss_multi(om, terms, 3), lib.loglik_gauss_multi(om, terms, Y, x))
        vec.domarg = True
        out[name] = fitting.BFGS_lpdf(om, vec)
    g, o = out["gpu"], out["oracle"]
    assert abs(g["optid"]["val"] - o["optid"]["val"]) <= 1e-6 * abs(o["optid"]["val"])
    assert relerr(g["parlist"]["hyp"], o["parlist"]["hyp"]) < 1e-4
    assert relerr(g["parlist"]["para"], o["parlist"]["para"]) < 1e-4


@pytest.mark.gpu
def test_gpu_bad_input_is_refused(gpu):
    om, x, Y, terms, _ = multi_objects(gpu, 300, 40, 2)
    with pytest.raises(ValueError):
        gpu.loglik_gauss_multi(om, terms, Y[:, :0], x)
    with pytest.raises(ValueError):
        gpu.logpr_gauss_multi(om, terms, 0)
    lk = gpu.loglik_gauss_multi(om, terms, Y, x)
    with pytest.raises(ValueError):
        gpu.lpdfvec(gpu.logpr_gauss(om, terms), lk)
    with pytest.raises(ValueError):
        gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, 3), lk)
    vec = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, 2), lk)
    with pytest.raises(ValueError):
        vec.optnewton()
    with pytest.raises(ValueError):
        lk.optcg(0.001, 5)
    with pytest.raises(ValueError):
        lk.hess()


@pytest.mark.gpu
def test_gpu_row_sharding_two_ranks(gpu):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("single-GPU box")
    env = dict(os.environ, OMP_NUM_THREADS="2", OMP_WAIT_POLICY="passive")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29561", str(REPO / "tests" / "mgpu_multiresponse_worker.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    assert "mgpu_multiresponse_worker world=2 OK" in res.stdout
