"""Shapley effects of a tensor-product model (include/outerbase_b200_sobol_shapley.h, ob_engine.hpp sobol_shapley,
ob_kernels.cu sobol_shapley_kernel).

CPU: the exported ABI, and a numpy restatement of the header's form against brute force on the full tensor grid of X_q's
columns (every ANOVA component variance from grid conditional means), evaluated by the oracle.  The restatement uses no
quadrature: it builds the coefficients of prod_{j != l} h_j(z) as K x K matrices by polynomial multiplication and weights
coefficient m by 1 / (m + 1), so it is independent of the product's nodes and weights.  GPU: the product against that
restatement fed the product's own basis at X_q, brute force with the product's matmul, the four outputs of ob_sobol bit
for bit, the identities, determinism and column independence, the semantics of the measure, obsobol(shapley=True) on
fits, and the refusals."""
import types

import numpy as np
import pytest

from outerbase_b200 import fitting
from outerbase_b200.binding import posterior_draws, sobol, sobol_pairs, sobol_shapley
from test_sobol import FWD, STAGE_BYTES, random_problem, sobol_tables
from test_sobol_pairs import PAIR_CASES, anova_brute_force, borehole_fit  # noqa: F401 (borehole_fit: a fixture)


# ------------------------------------------------------------------------------------------ numpy restatement
def factors(tabs, t):
    """p_j, c_j (K x K) of dimension j, and the pair factors of the absolute tables for the error bound"""
    p = lambda j: np.outer(tabs[j]["mu"][t[:, j]], tabs[j]["mu"][t[:, j]])  # noqa: E731
    c = lambda j: tabs[j]["C"][np.ix_(t[:, j], t[:, j])]  # noqa: E731
    a = lambda j: np.outer(tabs[j]["mua"][t[:, j]], tabs[j]["mua"][t[:, j]]) + tabs[j]["Ca"][np.ix_(t[:, j], t[:, j])]  # noqa: E731
    return p, c, a


def form(M, th):
    return ((M @ th) * th).sum(axis=0)


def shapley_reference(lib, om, terms, coeff, xq, tabs=None):
    """Sh_l = sum theta theta' c_l sum_m e_m / (m + 1), e_m the coefficient of z^m in prod_{j != l} (p_j + z c_j), built
    one dimension at a time.  Also returns the bound of the error check, |theta|^T A |theta| as in test_sobol."""
    t = np.asarray(terms, dtype=np.int64)
    th = np.asarray(coeff, dtype=float).reshape((t.shape[0], -1), order="F")
    tabs = tabs or sobol_tables(lib, om, terms, xq)
    d = t.shape[1]
    p, c, a = factors(tabs, t)
    sh = []
    for l in range(d):
        poly = [np.ones((t.shape[0], t.shape[0]))]
        for j in range(d):
            if j == l:
                continue
            pj, cj = p(j), c(j)
            nxt = [poly[0] * pj]
            nxt += [poly[m] * pj + poly[m - 1] * cj for m in range(1, len(poly))]
            nxt.append(poly[-1] * cj)
            poly = nxt
        sh.append(form(c(l) * sum(e / (m + 1) for m, e in enumerate(poly)), th))
    A = np.ones((t.shape[0], t.shape[0]))
    for j in range(d):
        A *= a(j)
    return dict(shapley=np.array(sh), bound=form(A, np.abs(th)))


def shapley_by_quadrature(lib, om, terms, coeff, xq, inputs):
    """Sh_l of the given inputs by an (n + 3)-node Gauss-Legendre rule in numpy: also exact, rounded differently, and
    needs a few K x K matrices only; with the bound as shapley_reference"""
    t = np.asarray(terms, dtype=np.int64)
    th = np.asarray(coeff, dtype=float).reshape((t.shape[0], -1), order="F")
    tabs = sobol_tables(lib, om, terms, xq)
    d = t.shape[1]
    p, c, a = factors(tabs, t)
    x, w = np.polynomial.legendre.leggauss(max(1, (d + 1) // 2) + 3)
    z, w = (1 + x) / 2, w / 2
    sh = {}
    for l in inputs:
        S = np.zeros((t.shape[0], t.shape[0]))
        for zi, wi in zip(z, w):
            M = np.full((t.shape[0], t.shape[0]), wi)
            for j in range(d):
                if j != l:
                    M *= p(j) + zi * c(j)
            S += M
        sh[l] = form(c(l) * S, th)
    A = np.ones((t.shape[0], t.shape[0]))
    for j in range(d):
        A *= a(j)
    return sh, form(A, np.abs(th))


def brute_shapley(sig, d):
    """sum of sigma2_u / |u| over the input sets u that contain l"""
    return np.array([sum(s / len(u) for u, s in sig.items() if l in u) for l in range(d)])


# ---------------------------------------------------------------------------------------------------- CPU
def test_product_exports_the_sobol_shapley_abi(product_symbols):
    import outerbase_b200 as ob
    syms = ob.header_symbols(ob.SOBOL_SHAPLEY_HEADER)
    assert syms == ["ob_sobol_shapley"]
    assert all(product_symbols.has(s) for s in syms)


@pytest.mark.parametrize("d,n,K,B,seed", [(1, 30, 12, 3, 5), (2, 14, 30, 3, 1), (3, 12, 40, 3, 2), (3, 8, 60, 2, 3),
                                          (4, 9, 60, 3, 4)])
def test_shapley_reference_matches_brute_force_on_the_oracle(oracle, d, n, K, B, seed):
    om, terms, coeff, xq = random_problem(oracle, d, [12 + 3 * l for l in range(d)], K, B, n, seed)
    ref = shapley_reference(oracle, om, terms, coeff, xq)
    sig, var = anova_brute_force(oracle, om, terms, coeff, xq)
    scale = np.max(var)
    assert scale > 0
    want = brute_shapley(sig, d)
    for l in range(d):
        np.testing.assert_allclose(ref["shapley"][l], want[l], rtol=0, atol=1e-12 * scale, err_msg=f"input {l}")
    np.testing.assert_allclose(ref["shapley"].sum(axis=0), var, rtol=0, atol=1e-12 * scale)
    if d == 1:
        np.testing.assert_allclose(ref["shapley"][0], var, rtol=0, atol=1e-12 * scale)
    assert np.all(ref["shapley"] > 0)


# ---------------------------------------------------------------------------------------------------- GPU
def check_against_reference(gpu, om, terms, coeff, xq, what=""):
    """sobol_shapley element-wise against the restatement, its four other outputs bit for bit against sobol"""
    got = sobol_shapley(gpu, om, terms, coeff, xq)
    one = sobol(gpu, om, terms, coeff, xq)
    for key in ("mean", "var", "first", "total"):
        np.testing.assert_array_equal(got[key], one[key], err_msg=what + " " + key)
    ref = shapley_reference(gpu, om, terms, coeff, xq)
    d = terms.shape[1]
    sh = got["shapley"].reshape((d, -1))
    bound = FWD * ref["bound"]
    for l in range(d):
        assert np.all(np.abs(sh[l] - ref["shapley"][l]) <= bound), f"{what} input {l}"
    return got, ref


@pytest.mark.gpu
@pytest.mark.parametrize("d,knots,K,B,nq", PAIR_CASES)
def test_shapley_against_the_restatement(gpu, d, knots, K, B, nq):
    om, terms, coeff, xq = random_problem(gpu, d, knots, K, B, nq, seed=d * 1000 + K + B)
    got, _ = check_against_reference(gpu, om, terms, coeff, xq, what=f"d={d} K={K} B={B} nq={nq}")
    assert got["shapley"].shape == (d, B)


@pytest.mark.gpu
def test_shapley_of_one_input_is_the_variance(gpu):
    om, terms, coeff, xq = random_problem(gpu, 1, [15], 10, 3, 200, seed=3)
    got, ref = check_against_reference(gpu, om, terms, coeff, xq, what="d=1")
    assert np.all(np.abs(got["shapley"][0] - got["var"]) <= FWD * ref["bound"])


@pytest.mark.gpu
def test_shapley_on_tables_beyond_the_staging_size(gpu):
    """knot counts that differ per dimension, one of 100 knots whose levels reach 99: the tables are not staged"""
    rng = np.random.default_rng(11)
    om = gpu.outermod()
    om.setcovfs(["mat25", "mat25pow", "mat25ang", "mat25"])
    om.setknot([np.sort(rng.uniform(0.01, 0.99, size=m)) for m in (100, 17, 33, 9)])
    extra = np.array([[99, 0, 0, 0], [99, 1, 2, 0], [60, 0, 5, 3], [80, 4, 0, 1], [0, 16, 32, 8]], dtype=np.uint64)
    terms = np.asfortranarray(np.vstack([om.selectterms(50), extra]))
    mo = terms.max(axis=0).astype(int) + 1
    assert mo[0] == 100 and 8 * (mo.sum() + (mo ** 2).sum()) > STAGE_BYTES
    coeff = np.asfortranarray(rng.normal(size=(terms.shape[0], 9)))
    xq = np.asfortranarray(rng.uniform(size=(5000, 4)))
    check_against_reference(gpu, om, terms, coeff, xq, what="100 knots")


@pytest.mark.gpu
def test_shapley_at_77_dimensions(gpu):
    """the largest d the forms kernel holds: ten row tiles, a segment of ten inputs per thread, 39 nodes"""
    om, terms, coeff, xq = random_problem(gpu, 77, [5] * 77, 100, 2, 50, seed=7)
    got, _ = check_against_reference(gpu, om, terms, coeff, xq, what="d=77")
    assert np.isfinite(got["shapley"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("B,nq", [(1, 1_000_000), (64, 20_000)])
def test_shapley_on_the_c3_table(gpu, B, nq):
    import bench
    om, terms = bench.setup_model(gpu)
    rng = np.random.default_rng(B)
    coeff = np.asfortranarray(rng.normal(size=(terms.shape[0], B)) / (1 + terms.sum(axis=1))[:, None])
    xq = bench.synth_rows(0, nq, bench.D)
    check_against_reference(gpu, om, terms, coeff, xq, what=f"C3 B={B} nq={nq}")


@pytest.mark.gpu
def test_shapley_on_the_c4_table_on_a_sample_of_inputs(gpu):
    """d = 20, K = 4000: the polynomial restatement would need d K x K layers; inputs 0, 7 and 19 by an (n + 3)-node rule"""
    import bench
    om, terms = bench.config_model(gpu, "c4share")
    assert terms.shape == (4000, 20)
    rng = np.random.default_rng(4)
    coeff = np.asfortranarray(rng.normal(size=(terms.shape[0], 64)) / (1 + terms.sum(axis=1))[:, None])
    xq = bench.config_rows("c4share", 0, 20_000)
    got = sobol_shapley(gpu, om, terms, coeff, xq)
    one = sobol(gpu, om, terms, coeff, xq)
    for key in ("mean", "var", "first", "total"):
        np.testing.assert_array_equal(got[key], one[key], err_msg=key)
    want, bound = shapley_by_quadrature(gpu, om, terms, coeff, xq, (0, 7, 19))
    for l, v in want.items():
        assert np.all(np.abs(got["shapley"][l] - v) <= FWD * bound), f"C4 input {l}"


@pytest.mark.gpu
def test_quadrature_restatement_agrees_with_the_polynomial_one(gpu):
    """the C4 check's restatement against the polynomial one, on a small case"""
    om, terms, coeff, xq = random_problem(gpu, 7, [12] * 7, 80, 3, 2000, seed=12)
    ref = shapley_reference(gpu, om, terms, coeff, xq)
    quad, _ = shapley_by_quadrature(gpu, om, terms, coeff, xq, range(7))
    for l in range(7):
        assert np.all(np.abs(quad[l] - ref["shapley"][l]) <= 1e-13 * ref["bound"]), l


@pytest.mark.gpu
@pytest.mark.parametrize("d,n,K,B,seed", [(3, 12, 40, 3, 1), (4, 9, 60, 3, 3)])
def test_shapley_brute_force_on_the_gpu(gpu, d, n, K, B, seed):
    om, terms, coeff, xq = random_problem(gpu, d, [12 + 3 * l for l in range(d)], K, B, n, seed)
    got = sobol_shapley(gpu, om, terms, coeff, xq)
    sig, var = anova_brute_force(gpu, om, terms, coeff, xq)
    want = brute_shapley(sig, d)
    for l in range(d):
        np.testing.assert_allclose(got["shapley"][l], want[l], rtol=0, atol=1e-11 * np.max(var))


@pytest.mark.gpu
@pytest.mark.parametrize("d,seed", [(2, 1), (3, 2), (6, 3), (20, 4)])
def test_shapley_identities(gpu, d, seed):
    om, terms, coeff, xq = random_problem(gpu, d, [14] * d, 80, 4, 3000, seed=seed)
    r = sobol_shapley(gpu, om, terms, coeff, xq)
    tol = 1e-10 * shapley_reference(gpu, om, terms, coeff, xq)["bound"] if d <= 6 else None
    if tol is None:
        t = np.asarray(terms, dtype=np.int64)
        _, _, a = factors(sobol_tables(gpu, om, terms, xq), t)
        A = np.ones((t.shape[0], t.shape[0]))
        for j in range(d):
            A *= a(j)
        tol = 1e-10 * form(A, np.abs(coeff))
    sh = r["shapley"]
    assert np.all(np.abs(sh.sum(axis=0) - r["var"]) <= tol)
    assert np.all(r["first"] <= sh + tol) and np.all(sh <= r["total"] + tol)
    if d in (2, 3):
        p = sobol_pairs(gpu, om, terms, coeff, xq)
        second = p["second"]
        if d == 2:
            for l in range(2):
                assert np.all(np.abs(sh[l] - (r["first"][l] + second[0, 1] / 2)) <= tol)
        else:
            l, m = np.triu_indices(3, 1)
            s012 = r["var"] - r["first"].sum(axis=0) - second[l, m].sum(axis=0)
            assert np.all(s012 > tol)  # the check is not vacuous
            for l in range(3):
                want = r["first"][l] + np.nansum(second[l], axis=0) / 2 + s012 / 3
                assert np.all(np.abs(sh[l] - want) <= 2 * tol), l


@pytest.mark.gpu
def test_shapley_of_an_input_held_constant_is_zero(gpu):
    om, terms, coeff, xq = random_problem(gpu, 5, [14] * 5, 80, 3, 3000, seed=13)
    xq[:, 2] = 0.37
    r = sobol_shapley(gpu, om, terms, coeff, xq)
    t = np.asarray(terms, dtype=np.int64)
    _, _, a = factors(sobol_tables(gpu, om, terms, xq), t)
    A = np.ones((t.shape[0], t.shape[0]))
    for j in range(5):
        A *= a(j)
    tol = FWD * form(A, np.abs(coeff))
    assert np.all(np.abs(r["shapley"][2]) <= tol)
    assert np.all(r["shapley"][[0, 1, 3, 4]] > 100 * tol)
    assert np.all(np.abs(r["shapley"].sum(axis=0) - r["var"]) <= tol)


@pytest.mark.gpu
def test_shapley_determinism_and_column_independence(gpu):
    om, terms, coeff, xq = random_problem(gpu, 12, [16] * 12, 300, 65, 20_000, seed=9)
    a = sobol_shapley(gpu, om, terms, coeff, xq)
    b = sobol_shapley(gpu, om, terms, coeff, xq)
    for key in a:
        np.testing.assert_array_equal(a[key], b[key])
    for j in (0, 1, 31, 32, 33, 63, 64):
        one = sobol_shapley(gpu, om, terms, coeff[:, j], xq)
        np.testing.assert_array_equal(one["shapley"], a["shapley"][:, j])


@pytest.mark.gpu
@pytest.mark.parametrize("d", [3, 20])
def test_shapley_column_independence_at_other_splits(gpu, d):
    """one row tile (eight k-step groups) and three row tiles (two groups) of the contraction"""
    om, terms, coeff, xq = random_problem(gpu, d, [12] * d, 200, 65, 5000, seed=d)
    a = sobol_shapley(gpu, om, terms, coeff, xq)
    for j in (0, 33, 64):
        np.testing.assert_array_equal(sobol_shapley(gpu, om, terms, coeff[:, j], xq)["shapley"], a["shapley"][:, j])


@pytest.mark.gpu
def test_shapley_measure_semantics(gpu):
    om, terms, coeff, xq = random_problem(gpu, 6, [20] * 6, 60, 8, 3000, seed=5)
    a = sobol_shapley(gpu, om, terms, coeff, xq)
    scale = a["var"][None, :]
    # stacking X_q twice changes nothing
    b = sobol_shapley(gpu, om, terms, coeff, np.asfortranarray(np.vstack([xq, xq])))
    assert np.all(np.abs(a["shapley"] - b["shapley"]) <= 1e-12 * scale)
    # ... and the pairing within rows does not matter: each column permuted on its own
    rng = np.random.default_rng(0)
    xp = np.asfortranarray(np.stack([rng.permutation(xq[:, l]) for l in range(xq.shape[1])], axis=1))
    c = sobol_shapley(gpu, om, terms, coeff, xp)
    assert np.all(np.abs(a["shapley"] - c["shapley"]) <= 1e-12 * scale)


@pytest.mark.gpu
def test_obsobol_shapley_on_the_borehole_function(borehole_fit):
    model, xq = borehole_fit
    lib = model["logpdf"]._lib
    res = fitting.obsobol(model, xq, shapley=True)
    plain = fitting.obsobol(model, xq)
    assert set(plain) == {"first", "total", "var", "mean"}
    assert set(res) == set(plain) | {"shapley"}
    for key in plain:
        np.testing.assert_array_equal(res[key], plain[key])
    r = sobol_shapley(lib, model["om"], model["terms"], model["logpdf"].coeff, xq)
    assert res["shapley"].shape == (8,)
    np.testing.assert_array_equal(res["shapley"], r["shapley"] / r["var"])
    # shapley=False is what obsobol returned before: sobol's forms over the variance
    one = sobol(lib, model["om"], model["terms"], model["logpdf"].coeff, xq)
    np.testing.assert_array_equal(plain["first"], one["first"] / one["var"])
    np.testing.assert_array_equal(plain["total"], one["total"] / one["var"])
    assert plain["var"] == model["y_sca"] ** 2 * one["var"]
    sh = res["shapley"]
    assert abs(sh.sum() - 1) < 1e-12
    assert np.all(res["first"] <= sh + 1e-12) and np.all(sh <= res["total"] + 1e-12)
    assert np.all(sh[[1, 2, 4]] < 0.01)  # r, T_u, T_l: inert
    assert np.argmax(sh) == np.argmax(res["total"])
    both = fitting.obsobol(model, xq, second=True, shapley=True)
    assert set(both) == set(plain) | {"second", "closed", "supset", "shapley"}
    np.testing.assert_array_equal(both["shapley"], res["shapley"])
    np.testing.assert_array_equal(both["second"], fitting.obsobol(model, xq, second=True)["second"])


@pytest.mark.gpu
def test_obsobol_shapley_draws_equal_sobol_shapley_on_the_draws(borehole_fit):
    model, xq = borehole_fit
    lib = model["logpdf"]._lib
    res = fitting.obsobol(model, xq, S=8, seed=4, shapley=True)
    dr = res["draws"]
    assert dr["shapley"].shape == (8, 8)
    coeff = posterior_draws(lib, model["logpdf"], 8, 4).solve(0.001, 100).coeff
    r = sobol_shapley(lib, model["om"], model["terms"], coeff, xq)
    np.testing.assert_array_equal(dr["shapley"], r["shapley"] / r["var"])
    np.testing.assert_array_equal(dr["first"], r["first"] / r["var"])


@pytest.mark.gpu
def test_obsobol_shapley_on_a_multi_response_fit(gpu):
    rng = np.random.default_rng(31)
    x = np.asfortranarray(rng.uniform(size=(1500, 3)))
    Y = np.column_stack([np.sin(6 * x[:, 0]) + x[:, 1], x[:, 1] * x[:, 2] + 0.2 * x[:, 0], np.exp(x[:, 2])])
    model = fitting.obfit_multi(gpu, x, Y, numb=40, covnames=["mat25pow"] * 3, numberopts=1)
    xq = np.asfortranarray(rng.uniform(size=(4000, 3)))
    res = fitting.obsobol(model, xq, shapley=True)
    assert res["shapley"].shape == (3, 3)
    coeff = model["logpdf"].coeff
    for c in range(3):
        one = sobol_shapley(gpu, model["om"], model["terms"], coeff[:, c], xq)
        np.testing.assert_array_equal(res["shapley"][:, c], one["shapley"] / one["var"])
    np.testing.assert_allclose(res["shapley"].sum(axis=0), 1, rtol=0, atol=1e-12)
    # column 2 depends on x_3 alone
    assert res["shapley"][2, 2] > 0.98


@pytest.mark.gpu
def test_zero_variance_gives_nan_shapley(gpu, recwarn):
    om, terms, coeff, xq = random_problem(gpu, 3, [10, 10, 10], 20, 2, 500, seed=8)
    fit = types.SimpleNamespace(_lib=gpu, coeff=np.zeros(terms.shape[0]))  # what obsobol reads of a fitted logpdf
    res = fitting.obsobol(dict(logpdf=fit, om=om, terms=terms, y_cent=0.0, y_sca=1.0), xq, shapley=True)
    assert res["var"] == 0
    assert res["shapley"].shape == (3,) and np.all(np.isnan(res["shapley"]))
    assert not [w for w in recwarn if issubclass(w.category, RuntimeWarning)]


@pytest.mark.gpu
def test_shapley_refusals(gpu):
    om, terms, coeff, xq = random_problem(gpu, 3, [10, 12, 14], 20, 2, 100, seed=6)
    with pytest.raises(ValueError, match="at least one column"):
        sobol_shapley(gpu, om, terms, np.zeros((terms.shape[0], 0)), xq)
    with pytest.raises(ValueError, match="at least one row"):
        sobol_shapley(gpu, om, terms, coeff, np.zeros((0, 3), order="F"))
    with pytest.raises(ValueError, match="terms table is empty"):
        sobol_shapley(gpu, om, np.zeros((0, 3), dtype=np.uint64), np.zeros(0), xq)
    with pytest.raises(ValueError, match="columns, the outermod 3 dimensions"):
        sobol_shapley(gpu, om, np.zeros((5, 4), dtype=np.uint64), np.ones(5), xq)
    with pytest.raises(ValueError, match="x must be nq x d"):
        sobol_shapley(gpu, om, terms, coeff, np.zeros((10, 4), order="F"))
    # levels beyond the knots
    bad = terms.copy()
    bad[0, 1] = 12
    with pytest.raises(ValueError, match="exceeds the number of knots"):
        sobol_shapley(gpu, om, bad, coeff, xq)
    # d = 78: beyond what the forms kernel holds
    om78, terms78, coeff78, xq78 = random_problem(gpu, 78, [5] * 78, 100, 1, 50, seed=7)
    with pytest.raises(ValueError, match="more dimensions"):
        sobol_shapley(gpu, om78, terms78, coeff78, xq78)
