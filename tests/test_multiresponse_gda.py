"""Multi-response loglik_gda: C responses on one basis with one per-row noise scale (include/outerbase_b200_multi_gda.h,
ob_engine.hpp LoglikGdaMulti), and the two-stage fitting.obfit_multi it makes possible.

The reference is the definition itself: C single-response oracle loglik_gda objects and loops over them
(tests/multiresponse_gda_reference.py).  GPU: the product's column-batched objects and CG against it."""
import numpy as np
import pytest

from conftest import make_problem, relerr
from multiresponse_gda_reference import Reference
from outerbase_b200 import fitting
from test_multiresponse import responses

N_GDA, K_GDA = 600, 80


def gda_objects(lib, C, N=N_GDA, K=K_GDA):
    """test_loglik_gda_parity's problem (mat25 everywhere, knots every 0.05) with C seeded responses"""
    om, x, y, terms, rng = make_problem(lib, N, K, covs=["mat25"] * 8, knots=[np.arange(0.001, 0.999, 0.05)] * 8)
    return om, x, responses(x, y, C), terms, rng


def _flags(obj, on=True):
    obj.compute_val = on; obj.compute_grad = on; obj.compute_gradhyp = on; obj.compute_gradpara = on


def _fit_data(n, seed):
    rng = np.random.default_rng(seed)
    x = np.asfortranarray(rng.uniform(size=(n, 3)))
    f = lambda x: np.column_stack([np.sin(3 * x[:, 0]) + x[:, 1] * x[:, 2] + 0.5 * x[:, 1] ** 2,
                                   10 + 4 * x[:, 2] ** 2 - x[:, 0], np.cos(2 * x[:, 1]) * x[:, 2]])
    return rng, x, f


def test_product_exports_the_gda_extension_abi(product_symbols):
    import outerbase_b200 as ob
    syms = ob.header_symbols(ob.MULTI_GDA_HEADER)
    assert syms == ["ob_loglik_gda_multi_create"]
    assert all(product_symbols.has(s) for s in syms)


def test_binding_refuses_misaligned_responses(product_symbols):
    from outerbase_b200.binding import loglik_gda_multi
    x, terms = np.zeros((10, 2)), np.zeros((3, 2), dtype=np.uint64)
    with pytest.raises(ValueError, match="align"):
        loglik_gda_multi(product_symbols, None, terms, np.zeros((9, 2)), x)
    with pytest.raises(ValueError, match="N x C"):
        loglik_gda_multi(product_symbols, None, terms, np.zeros(10), x)


def test_reference_is_loglik_gda_at_one_column(oracle):
    """C = 1: the reference's lpdfvec is the oracle's lpdfvec(logpr_gauss, loglik_gda), bit for bit"""
    ref = Reference(oracle)
    om, x, Y, terms, rng = gda_objects(oracle, 1, N=300, K=40)
    lk_r = ref.loglik_gda_multi(om, terms, Y, x)
    lk_o = oracle.loglik_gda(om, terms, Y[:, 0], x)
    np.testing.assert_array_equal(lk_r.para0, lk_o.para)
    lk_r.dodiag = True
    lk_o.dodiag = True
    vr = ref.lpdfvec(ref.logpr_gauss_multi(om, terms, 1), lk_r)
    vo = oracle.lpdfvec(oracle.logpr_gauss(om, terms), lk_o)
    for v in (vr, vo):
        v.domarg = True
        v.updatepara(np.array([5.0, np.log(0.3), -0.5]))
    c = rng.normal(size=40) / 30
    vr.update(c)
    _flags(vo); vo.update(c)
    assert vr.val == vo.val
    np.testing.assert_array_equal(vr.grad[:, 0], vo.grad)
    np.testing.assert_array_equal(vr.gradhyp, vo.gradhyp)
    np.testing.assert_array_equal(vr.gradpara, vo.gradpara)
    vr.optcg(0.001, 100)
    vo.optcg(0.001, 100)
    assert vr.cg_iters_per_column[0] == vo.cg_iters
    np.testing.assert_array_equal(vr.coeff[:, 0], vo.coeff)
    assert vr.val == vo.val


@pytest.mark.parametrize("seed", [0, 7])
def test_two_stage_obfit_multi_is_obfit_at_one_column(oracle, seed):
    rng, x, f = _fit_data(300, 11)
    y = f(x)[:, 0]
    multi = fitting.obfit_multi(Reference(oracle), x, y[:, None], numb=30, numberopts=1, stage1=True, seed=seed)
    single = fitting.obfit(oracle, x, y, numb=30, numberopts=1, seed=seed)
    np.testing.assert_array_equal(multi["stage1"]["rows"], single["stage1"]["rows"])
    np.testing.assert_array_equal(fitting.gethyp(multi["om"]), fitting.gethyp(single["om"]))
    np.testing.assert_array_equal(fitting.getpara(multi["logpdf"]), fitting.getpara(single["logpdf"]))
    assert multi["optinfo"]["optid"]["val"] == single["optinfo"]["optid"]["val"]


def test_two_stage_obfit_multi_predicts_on_the_reference(oracle):
    rng, x, f = _fit_data(400, 5)
    model = fitting.obfit_multi(Reference(oracle), x, f(x), numb=30, numberopts=1, stage1=True)
    assert model["stage1"]["rows"].size == min(400, 3 * 30)
    xt = np.asfortranarray(rng.uniform(size=(200, 3)))
    Yt = f(xt)
    pred = fitting.obpred(model, xt)
    assert pred["mean"].shape == (200, 3) and pred["var"].shape == (200, 3)
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


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [0, 1])
@pytest.mark.parametrize("dodiag", [True, False])
@pytest.mark.parametrize("C", [1, 3, 8, 70])
def test_gpu_likelihood_matches_the_reference(gpu, oracle, families, spec, dodiag, C):
    families(spec)
    res = {}
    for name, lib in (("gpu", gpu), ("reference", Reference(oracle))):
        om, x, Y, terms, rng = gda_objects(lib, C)
        lk = lib.loglik_gda_multi(om, terms, Y, x)
        lk.dodiag = dodiag
        lk.updatepara([np.log(0.2), -0.5])
        A = np.asfortranarray(rng.normal(size=(K_GDA, C)) / 50)
        g = rng.normal(size=K_GDA * C)
        _flags(lk)
        lk.update(A)
        res[name] = dict(val=lk.val, grad=np.array(lk.grad), gh=np.array(lk.gradhyp), gp=np.array(lk.gradpara), yhat=lk.yhat,
                         hm=lk.hessmult(g), dh=lk.diaghess(), dhh=lk.diaghessgradhyp(), dhp=lk.diaghessgradpara())
    g, o = res["gpu"], res["reference"]
    assert g["yhat"].shape == (N_GDA, C)
    assert abs(g["val"] - o["val"]) <= 1e-8 * abs(o["val"])
    assert relerr(g["grad"], o["grad"]) < 1e-8
    assert relerr(g["gh"], o["gh"]) < 1e-6 and relerr(g["gp"], o["gp"]) < 1e-7
    assert relerr(g["yhat"], o["yhat"]) < 1e-8
    assert relerr(g["hm"], o["hm"]) < 1e-8 and relerr(g["dh"], o["dh"]) < 1e-8
    assert relerr(g["dhh"], o["dhh"]) < 1e-7 and relerr(g["dhp"], o["dhp"]) < 1e-8


def test_reference_default_para_is_the_mean_variance(oracle):
    om, x, Y, terms, _ = gda_objects(oracle, 3, N=200, K=30)
    lk = Reference(oracle).loglik_gda_multi(om, terms, Y, x)
    np.testing.assert_allclose(lk.para0, [0.5 * np.log(0.01 * np.mean(np.var(Y, axis=0, ddof=1))), 0.0], rtol=1e-13)
    np.testing.assert_array_equal(lk.paravar, [4.0, 4.0])


@pytest.mark.gpu
def test_gpu_default_para_matches_the_reference(gpu, oracle):
    out = []
    for lib in (gpu, Reference(oracle)):
        om, x, Y, terms, _ = gda_objects(lib, 5)
        out.append(np.array(lib.loglik_gda_multi(om, terms, Y, x).para))
    np.testing.assert_array_equal(out[0], out[1])


@pytest.mark.gpu
@pytest.mark.parametrize("domarg", [True, False])
@pytest.mark.parametrize("lik_first", [False, True])
@pytest.mark.parametrize("C", [3, 8])
def test_gpu_optcg_is_c_independent_runs(gpu, oracle, families, C, lik_first, domarg):
    families(1)
    res = {}
    for name, lib in (("gpu", gpu), ("reference", Reference(oracle))):
        om, x, Y, terms, _ = gda_objects(lib, C)
        lk = lib.loglik_gda_multi(om, terms, Y, x)
        lk.dodiag = True
        pr = lib.logpr_gauss_multi(om, terms, C)
        vec = lib.lpdfvec(lk, pr) if lik_first else lib.lpdfvec(pr, lk)
        vec.domarg = domarg
        vec.updatepara(np.array([np.log(0.2), -0.5, 5.0]) if lik_first else np.array([5.0, np.log(0.2), -0.5]))
        vec.optcg(0.001, 100)
        res[name] = dict(iters=np.array(vec.cg_iters_per_column), coeff=np.array(vec.coeff), val=vec.val,
                         gh=np.array(vec.gradhyp), gp=np.array(vec.gradpara))
    g, o = res["gpu"], res["reference"]
    np.testing.assert_array_equal(g["iters"], o["iters"])
    assert relerr(g["coeff"], o["coeff"]) < 1e-8
    assert abs(g["val"] - o["val"]) <= 1e-8 * abs(o["val"])
    assert relerr(g["gh"], o["gh"]) < 1e-6 and relerr(g["gp"], o["gp"]) < 1e-7


@pytest.mark.gpu
def test_gpu_predictor_matches_the_reference(gpu, oracle):
    C = 3
    out = {}
    xt = None
    for name, lib in (("gpu", gpu), ("reference", Reference(oracle))):
        om, x, Y, terms, _ = gda_objects(lib, C)
        lk = lib.loglik_gda_multi(om, terms, Y, x)
        lk.dodiag = True
        vec = lib.lpdfvec(lib.logpr_gauss_multi(om, terms, C), lk)
        vec.domarg = True
        vec.optcg(0.001, 100)
        p = lib.predictor(lk)
        xt = np.asfortranarray(np.random.default_rng(5).uniform(size=(97, 8)))
        p.update(xt)
        out[name] = (p.mean(), p.var())
    g, o = out["gpu"], out["reference"]
    assert g[0].shape == (97, C) and g[1].shape == (97,)
    assert relerr(g[0], o[0]) < 1e-7 and relerr(g[1], o[1]) < 1e-7


@pytest.mark.gpu
def test_gpu_bad_input_is_refused(gpu):
    om, x, Y, terms, _ = gda_objects(gpu, 2, N=300, K=40)
    with pytest.raises(ValueError):
        gpu.loglik_gda_multi(om, terms, Y[:, :0], x)
    lk = gpu.loglik_gda_multi(om, terms, Y, x)
    with pytest.raises(ValueError):  # a per-column prior
        gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, 2, para_per_column=True), lk)
    with pytest.raises(ValueError):
        gpu.lpdfvec(lk, gpu.logpr_gauss_multi(om, terms, 2, para_per_column=True))
    with pytest.raises(ValueError):  # a single-response child
        gpu.lpdfvec(gpu.logpr_gauss(om, terms), lk)
    with pytest.raises(ValueError):  # a different C
        gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, 3), lk)
    with pytest.raises(ValueError):  # para is never per column
        lk.updatepara([0.0, 0.0, 0.0, 0.0])
    vec = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, 2), lk)
    with pytest.raises(ValueError):
        vec.optnewton()
    with pytest.raises(ValueError):
        lk.optnewton()
    with pytest.raises(ValueError):
        lk.optcg(0.001, 5)
    with pytest.raises(ValueError):
        lk.hess()
    two = gpu.lpdfvec(gpu.loglik_gauss_multi(om, terms, Y, x), lk)
    with pytest.raises(ValueError):  # optcg outside lpdfvec(logpr_gauss_multi, loglik_gda_multi)
        two.optcg(0.001, 5)


@pytest.mark.gpu
def test_gpu_two_stage_obfit_multi_matches_the_reference(gpu, oracle):
    """test_obfit_gpu_matches_oracle's bounds, at C = 3"""
    rng, x, f = _fit_data(600, 9)
    xt = np.asfortranarray(rng.uniform(size=(150, 3)))
    res = {}
    for name, lib in (("gpu", gpu), ("reference", Reference(oracle))):
        model = fitting.obfit_multi(lib, x, f(x), numb=40, covnames=["mat25pow"] * 3, numberopts=1, stage1=True, seed=3)
        res[name] = (fitting.gethyp(model["om"]), fitting.getpara(model["logpdf"]), fitting.obpred(model, xt),
                     model["optinfo"]["optid"]["val"], model["stage1"]["rows"])
    g, o = res["gpu"], res["reference"]
    np.testing.assert_array_equal(g[4], o[4])
    assert abs(g[3] - o[3]) <= 1e-4 * abs(o[3])
    assert relerr(g[0], o[0]) < 1e-3 and relerr(g[1], o[1]) < 1e-3
    assert relerr(g[2]["mean"], o[2]["mean"]) < 1e-4


@pytest.mark.gpu
def test_gpu_two_stage_obfit_multi_is_obfit_at_one_column(gpu):
    rng, x, f = _fit_data(600, 9)
    y = f(x)[:, 0]
    xt = np.asfortranarray(rng.uniform(size=(150, 3)))
    multi = fitting.obfit_multi(gpu, x, y[:, None], numb=40, covnames=["mat25pow"] * 3, numberopts=1, stage1=True, seed=3)
    single = fitting.obfit(gpu, x, y, numb=40, covnames=["mat25pow"] * 3, numberopts=1, seed=3)
    np.testing.assert_array_equal(multi["stage1"]["rows"], single["stage1"]["rows"])
    assert abs(multi["optinfo"]["optid"]["val"] - single["optinfo"]["optid"]["val"]) <= 1e-4 * abs(single["optinfo"]["optid"]["val"])
    assert relerr(fitting.gethyp(multi["om"]), fitting.gethyp(single["om"])) < 1e-3
    assert relerr(fitting.getpara(multi["logpdf"]), fitting.getpara(single["logpdf"])) < 1e-3
    assert relerr(fitting.obpred(multi, xt)["mean"][:, 0], fitting.obpred(single, xt)["mean"]) < 1e-4


@pytest.mark.gpu
def test_gpu_two_stage_obfit_multi_per_column_para(gpu):
    """para_per_column with stage 1: stage 2 starts each column from stage 1's two shared entries"""
    rng, x, f = _fit_data(600, 9)
    model = fitting.obfit_multi(gpu, x, f(x), numb=40, covnames=["mat25pow"] * 3, numberopts=1, stage1=True,
                                para_per_column=True, seed=3)
    assert fitting.getpara(model["logpdf"]).size == 6
    xt = np.asfortranarray(rng.uniform(size=(150, 3)))
    pred = fitting.obpred(model, xt)
    Yt = f(xt)
    assert pred["var"].shape == (150, 3) and np.all(pred["var"] > 0)
    for c in range(3):
        assert np.mean((pred["mean"][:, c] - Yt[:, c]) ** 2) < 0.05 * np.var(Yt[:, c])
