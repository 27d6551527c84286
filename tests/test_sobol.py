"""Sobol sensitivity indices of a tensor-product model (include/outerbase_b200_sobol.h, ob_engine.hpp sobol).

CPU: the exported ABI, and a numpy restatement of the header's forms against brute force on the full tensor grid of
X_q's columns, evaluated by the oracle.  GPU: the product against that restatement fed the product's own basis at X_q,
tables beyond the shared-memory staging size, brute force with the product's matmul, the semantics of the measure,
determinism, obsobol on a borehole fit against Monte Carlo on the true function, draws, multi-response fits and the
refusals."""
import types

import numpy as np
import pytest

from conftest import borehole8d
from outerbase_b200 import fitting
from outerbase_b200.binding import posterior_draws, sobol

# element-wise forward-error bound: |got - want| <= FWD * (|theta|^T A |theta|), A the pair factors of absolute values
FWD = 1e-10
STAGE_BYTES = 48 * 1024  # obd::kSobolStageBytes: larger tables are read through the cache


# ------------------------------------------------------------------------------------------ numpy restatement
def sobol_tables(lib, om, terms, xq):
    """mu_l, centred C_l and their absolute counterparts (mean |R|, mean |R - mu| |R' - mu'|) from getbase at xq."""
    terms = np.asarray(terms, dtype=np.int64)
    ob = lib.outerbase(om, np.asfortranarray(xq), dograd=False)
    tabs = []
    for l in range(terms.shape[1]):
        R = ob.getbase(l + 1)[:, :terms[:, l].max() + 1]
        mu = R.mean(axis=0)
        Rc = R - mu
        tabs.append(dict(mu=mu, C=Rc.T @ Rc / R.shape[0], mua=np.abs(R).mean(axis=0), Ca=np.abs(Rc).T @ np.abs(Rc) / R.shape[0]))
    return tabs


def sobol_reference(lib, om, terms, coeff, xq, tabs=None):
    """The header's table of forms, K x K pair matrices per dimension.  Also returns the bounds of the error check."""
    t = np.asarray(terms, dtype=np.int64)
    th = np.asarray(coeff, dtype=float).reshape((t.shape[0], -1), order="F")
    tabs = tabs or sobol_tables(lib, om, terms, xq)
    d = t.shape[1]
    p = [np.outer(T["mu"][t[:, l]], T["mu"][t[:, l]]) for l, T in enumerate(tabs)]
    c = [T["C"][np.ix_(t[:, l], t[:, l])] for l, T in enumerate(tabs)]
    g = [c[l] + p[l] for l in range(d)]

    def prod(ms, skip=None):
        out = np.ones((t.shape[0], t.shape[0]))
        for j, m in enumerate(ms):
            if j != skip:
                out = out * m
        return out

    def form(M):
        return ((M @ th) * th).sum(axis=0)

    var = form(sum(prod(g[:l]) * c[l] * prod(p[l + 1:]) for l in range(d)))
    first = np.array([form(c[l] * prod(p, skip=l)) for l in range(d)])
    total = np.array([form(c[l] * prod(g, skip=l)) for l in range(d)])
    pm = np.prod([T["mu"][t[:, l]] for l, T in enumerate(tabs)], axis=0)
    A = prod([np.outer(T["mua"][t[:, l]], T["mua"][t[:, l]]) + T["Ca"][np.ix_(t[:, l], t[:, l])] for l, T in enumerate(tabs)])
    pma = np.prod([T["mua"][t[:, l]] for l, T in enumerate(tabs)], axis=0)
    return dict(mean=th.T @ pm, var=var, first=first, total=total,
                bound=((A @ np.abs(th)) * np.abs(th)).sum(axis=0), bound_mean=np.abs(th).T @ pma)


def brute_force(lib, om, terms, coeff, xq):
    """mean, Var, Var_l(E[f | x_l]) and E[Var_l(f | x_-l)] on the full tensor grid of xq's columns."""
    n, d = xq.shape
    grid = np.stack(np.meshgrid(*[xq[:, l] for l in range(d)], indexing="ij"), axis=-1).reshape(-1, d)
    th = np.asarray(coeff, dtype=float).reshape((terms.shape[0], -1), order="F")
    f = lib.outerbase(om, np.asfortranarray(grid), dograd=False).matmul(terms, th)
    B = th.shape[1]
    F = f.reshape((n,) * d + (B,))
    axes = tuple(range(d))
    var = F.var(axis=axes)
    first = np.array([F.mean(axis=tuple(a for a in axes if a != l)).var(axis=0) for l in range(d)])
    total = np.array([F.var(axis=l).mean(axis=tuple(range(d - 1))) for l in range(d)])
    return dict(mean=F.mean(axis=axes), var=var, first=first, total=total)


def random_problem(lib, d, nknots, K, B, nq, seed, covs=None):
    rng = np.random.default_rng(seed)
    om = lib.outermod()
    om.setcovfs(covs or [("mat25", "mat25pow", "mat25ang")[l % 3] for l in range(d)])
    om.setknot([np.sort(rng.uniform(0.02, 0.98, size=m)) for m in nknots])
    terms = om.selectterms(K)
    coeff = np.asfortranarray(rng.normal(size=(terms.shape[0], B)) / (1 + terms.sum(axis=1))[:, None])
    xq = np.asfortranarray(rng.uniform(size=(nq, d)))
    return om, terms, coeff, xq


# ---------------------------------------------------------------------------------------------------- CPU
def test_product_exports_the_sobol_abi(product_symbols):
    import outerbase_b200 as ob
    syms = ob.header_symbols(ob.SOBOL_HEADER)
    assert syms == ["ob_sobol"]
    assert all(product_symbols.has(s) for s in syms)


@pytest.mark.parametrize("d,n,K,B,seed", [(3, 12, 40, 3, 1), (3, 8, 60, 2, 2), (4, 9, 60, 3, 3), (4, 10, 25, 4, 4)])
def test_reference_matches_brute_force_on_the_oracle(oracle, d, n, K, B, seed):
    om, terms, coeff, xq = random_problem(oracle, d, [12 + 3 * l for l in range(d)], K, B, n, seed)
    ref = sobol_reference(oracle, om, terms, coeff, xq)
    bf = brute_force(oracle, om, terms, coeff, xq)
    scale = np.max(bf["var"])
    assert scale > 0
    for key in ("mean", "var", "first", "total"):
        np.testing.assert_allclose(ref[key], bf[key], rtol=0, atol=1e-12 * scale, err_msg=key)
    # the forms are not trivially zero: every dimension carries some variance
    assert np.all(ref["first"] > 0) and np.all(ref["total"] >= ref["first"] - 1e-12 * scale)


# ---------------------------------------------------------------------------------------------------- GPU
def check_against_reference(gpu, om, terms, coeff, xq, what=""):
    got = sobol(gpu, om, terms, coeff, xq)
    ref = sobol_reference(gpu, om, terms, coeff, xq)
    bound = FWD * ref["bound"]
    assert np.all(np.abs(got["mean"] - ref["mean"]) <= FWD * ref["bound_mean"]), what + " mean"
    assert np.all(np.abs(got["var"] - ref["var"]) <= bound), what + " var"
    for key in ("first", "total"):
        assert np.all(np.abs(got[key] - ref[key]) <= bound[None, :]), what + " " + key
    return got, ref


CASES = [  # d, knots per dimension, K, B, n_q
    (3, [10, 14, 18], 1, 1, 1),
    (3, [10, 14, 18], 60, 7, 2),
    (8, [20] * 8, 60, 64, 127),
    (10, [16] * 10, 60, 65, 20_000),
    (8, [24, 12, 30, 16, 20, 40, 14, 18], 60, 7, 1_000_000),
]


@pytest.mark.gpu
@pytest.mark.parametrize("d,knots,K,B,nq", CASES)
def test_against_the_restatement(gpu, d, knots, K, B, nq):
    om, terms, coeff, xq = random_problem(gpu, d, knots, K, B, nq, seed=d * 1000 + K + B)
    got, _ = check_against_reference(gpu, om, terms, coeff, xq, what=f"d={d} K={K} B={B} nq={nq}")
    assert got["first"].shape == (d, B)


@pytest.mark.gpu
@pytest.mark.parametrize("B,nq", [(1, 1_000_000), (64, 20_000)])
def test_against_the_restatement_on_the_c3_table(gpu, B, nq):
    import bench
    om, terms = bench.setup_model(gpu)
    rng = np.random.default_rng(B)
    coeff = np.asfortranarray(rng.normal(size=(terms.shape[0], B)) / (1 + terms.sum(axis=1))[:, None])
    xq = bench.synth_rows(0, nq, bench.D)
    check_against_reference(gpu, om, terms, coeff, xq, what=f"C3 B={B} nq={nq}")


@pytest.mark.gpu
def test_tables_beyond_the_staging_size(gpu):
    """knot counts that differ per dimension, one of 100 knots whose levels reach 99: the tables exceed the staged size"""
    rng = np.random.default_rng(11)
    d = 4
    om = gpu.outermod()
    om.setcovfs(["mat25", "mat25pow", "mat25ang", "mat25"])
    om.setknot([np.sort(rng.uniform(0.01, 0.99, size=m)) for m in (100, 17, 33, 9)])
    base = om.selectterms(50)
    extra = np.array([[99, 0, 0, 0], [99, 1, 2, 0], [60, 0, 5, 3], [80, 4, 0, 1], [0, 16, 32, 8]], dtype=np.uint64)
    terms = np.asfortranarray(np.vstack([base, extra]))
    mo = terms.max(axis=0).astype(int) + 1
    assert mo[0] == 100 and 8 * (mo.sum() + (mo ** 2).sum()) > STAGE_BYTES
    coeff = np.asfortranarray(rng.normal(size=(terms.shape[0], 9)))
    xq = np.asfortranarray(rng.uniform(size=(5000, d)))
    check_against_reference(gpu, om, terms, coeff, xq, what="100 knots")


@pytest.mark.gpu
@pytest.mark.parametrize("d,n,K,B,seed", [(3, 12, 40, 3, 1), (4, 9, 60, 3, 3)])
def test_brute_force_on_the_gpu(gpu, d, n, K, B, seed):
    om, terms, coeff, xq = random_problem(gpu, d, [12 + 3 * l for l in range(d)], K, B, n, seed)
    got = sobol(gpu, om, terms, coeff, xq)
    bf = brute_force(gpu, om, terms, coeff, xq)
    scale = np.max(bf["var"])
    for key in ("mean", "var", "first", "total"):
        np.testing.assert_allclose(got[key], bf[key], rtol=0, atol=1e-11 * scale, err_msg=key)


@pytest.mark.gpu
def test_measure_semantics(gpu):
    om, terms, coeff, xq = random_problem(gpu, 6, [20] * 6, 60, 8, 3000, seed=5)
    a = sobol(gpu, om, terms, coeff, xq)
    scale = a["var"][None, :]
    # the measure is the empirical marginals: stacking X_q twice changes nothing
    b = sobol(gpu, om, terms, coeff, np.asfortranarray(np.vstack([xq, xq])))
    for key in ("var", "first", "total"):
        assert np.all(np.abs(a[key] - b[key]) <= 1e-13 * scale), key
    assert np.all(np.abs(a["mean"] - b["mean"]) <= 1e-13 * np.sqrt(a["var"]) + 1e-13 * np.abs(a["mean"]))
    # ... and the pairing within rows does not matter: each column permuted on its own
    rng = np.random.default_rng(0)
    xp = np.asfortranarray(np.stack([rng.permutation(xq[:, l]) for l in range(xq.shape[1])], axis=1))
    c = sobol(gpu, om, terms, coeff, xp)
    for key in ("var", "first", "total"):
        assert np.all(np.abs(a[key] - c[key]) <= 1e-12 * scale), key
    # 0 <= first <= total, sum first <= var <= sum total, within rounding
    tol = 1e-12 * a["var"]
    assert np.all(a["first"] >= -tol) and np.all(a["first"] <= a["total"] + tol)
    assert np.all(a["first"].sum(axis=0) <= a["var"] + tol) and np.all(a["var"] <= a["total"].sum(axis=0) + tol)


@pytest.mark.gpu
def test_determinism_and_column_independence(gpu):
    om, terms, coeff, xq = random_problem(gpu, 8, [20] * 8, 300, 65, 20_000, seed=9)
    a = sobol(gpu, om, terms, coeff, xq)
    b = sobol(gpu, om, terms, coeff, xq)
    for key in a:
        np.testing.assert_array_equal(a[key], b[key])
    for j in (0, 1, 31, 32, 33, 63, 64):
        one = sobol(gpu, om, terms, coeff[:, j], xq)
        assert one["mean"] == a["mean"][j] and one["var"] == a["var"][j], j
        np.testing.assert_array_equal(one["first"], a["first"][:, j])
        np.testing.assert_array_equal(one["total"], a["total"][:, j])


def pick_freeze(f, d, n, seed):
    """Saltelli's first-order and Jansen's total estimators on U(0,1)^d, n base samples"""
    rng = np.random.default_rng(seed)
    A, Bm = rng.uniform(size=(n, d)), rng.uniform(size=(n, d))
    fA, fB = f(A), f(Bm)
    var = np.var(np.concatenate([fA, fB]))
    first, total = np.empty(d), np.empty(d)
    for l in range(d):
        ABl = A.copy()
        ABl[:, l] = Bm[:, l]
        fAB = f(ABl)
        first[l] = np.mean(fB * (fAB - fA)) / var
        total[l] = 0.5 * np.mean((fA - fAB) ** 2) / var
    return first, total


@pytest.fixture(scope="module")
def borehole_fit(gpu):
    rng = np.random.default_rng(21)
    x = np.asfortranarray(rng.uniform(size=(3000, 8)))
    model = fitting.obfit(gpu, x, borehole8d(x), numb=200, numberopts=1, seed=1)
    xq = np.asfortranarray(np.random.default_rng(22).uniform(size=(20_000, 8)))
    return model, xq


@pytest.mark.gpu
def test_obsobol_on_the_borehole_function(borehole_fit):
    model, xq = borehole_fit
    res = fitting.obsobol(model, xq)
    first, total = pick_freeze(borehole8d, 8, 400_000, seed=3)
    # the known values of the borehole function (r_w dominates; r, T_u, T_l are inert)
    assert abs(first[0] - 0.83) < 0.02 and abs(total[0] - 0.87) < 0.02 and np.all(total[[1, 2, 4]] < 0.01)
    TOL = 0.03
    np.testing.assert_allclose(res["first"], first, atol=TOL)
    np.testing.assert_allclose(res["total"], total, atol=TOL)
    assert res["first"].shape == (8,) and np.isfinite(res["var"]) and res["var"] > 0
    yv = borehole8d(xq)
    assert abs(res["mean"] - yv.mean()) < 0.02 * yv.std() and abs(res["var"] / yv.var() - 1) < 0.05


@pytest.mark.gpu
def test_obsobol_draws_equal_sobol_on_the_draws(borehole_fit):
    model, xq = borehole_fit
    res = fitting.obsobol(model, xq, S=16, seed=4)
    dr = res["draws"]
    assert dr["first"].shape == (8, 16) and dr["var"].shape == (16,)
    coeff = posterior_draws(model["logpdf"]._lib, model["logpdf"], 16, 4).solve(0.001, 100).coeff
    for s in range(16):
        one = sobol(model["logpdf"]._lib, model["om"], model["terms"], coeff[:, s], xq)
        assert dr["var"][s] == model["y_sca"] ** 2 * one["var"]
        assert dr["mean"][s] == model["y_cent"] + model["y_sca"] * one["mean"]
        np.testing.assert_array_equal(dr["first"][:, s], one["first"] / one["var"])
        np.testing.assert_array_equal(dr["total"][:, s], one["total"] / one["var"])
    # the point estimate sits inside the spread of the draws
    assert np.all(np.abs(res["first"] - dr["first"].mean(axis=1)) < 5 * dr["first"].std(axis=1) + 1e-3)


@pytest.mark.gpu
def test_obsobol_on_a_multi_response_fit(gpu):
    rng = np.random.default_rng(31)
    x = np.asfortranarray(rng.uniform(size=(1500, 3)))
    Y = np.column_stack([np.sin(6 * x[:, 0]) + x[:, 1], x[:, 1] * x[:, 2] + 0.2 * x[:, 0], np.exp(x[:, 2])])
    model = fitting.obfit_multi(gpu, x, Y, numb=40, covnames=["mat25pow"] * 3, numberopts=1)
    xq = np.asfortranarray(rng.uniform(size=(4000, 3)))
    res = fitting.obsobol(model, xq)
    assert res["first"].shape == (3, 3) and res["var"].shape == (3,)
    coeff = model["logpdf"].coeff
    for c in range(3):
        one = sobol(gpu, model["om"], model["terms"], coeff[:, c], xq)
        np.testing.assert_array_equal(res["first"][:, c], one["first"] / one["var"])
        np.testing.assert_array_equal(res["total"][:, c], one["total"] / one["var"])
        assert res["var"][c] == model["y_sca"][c] ** 2 * one["var"]
    # column 0 depends on x_1 and x_2 additively, column 2 on x_3 alone
    assert res["first"][2, 2] > 0.95 and res["total"][2, 0] < 0.02
    with pytest.raises(ValueError, match="multi-response"):
        fitting.obsobol(model, xq, S=4)


@pytest.mark.gpu
def test_zero_variance_gives_nan_indices(gpu, recwarn):
    om, terms, coeff, xq = random_problem(gpu, 3, [10, 10, 10], 20, 2, 500, seed=8)
    fit = types.SimpleNamespace(_lib=gpu, coeff=np.zeros(terms.shape[0]))  # what obsobol reads of a fitted logpdf
    res = fitting.obsobol(dict(logpdf=fit, om=om, terms=terms, y_cent=0.0, y_sca=1.0), xq)
    assert res["var"] == 0 and np.all(np.isnan(res["first"])) and np.all(np.isnan(res["total"]))
    assert not [w for w in recwarn if issubclass(w.category, RuntimeWarning)]


@pytest.mark.gpu
def test_refusals(gpu):
    om, terms, coeff, xq = random_problem(gpu, 3, [10, 12, 14], 20, 2, 100, seed=6)
    with pytest.raises(ValueError, match="at least one column"):
        sobol(gpu, om, terms, np.zeros((terms.shape[0], 0)), xq)
    with pytest.raises(ValueError, match="at least one row"):
        sobol(gpu, om, terms, coeff, np.zeros((0, 3), order="F"))
    with pytest.raises(ValueError, match="columns, the outermod 3 dimensions"):
        sobol(gpu, om, np.zeros((5, 4), dtype=np.uint64), np.ones(5), xq)
    bad = terms.copy()
    bad[0, 1] = 12
    with pytest.raises(ValueError, match="exceeds the number of knots"):
        sobol(gpu, om, bad, coeff, xq)
