"""Second-order Sobol indices of a tensor-product model (include/outerbase_b200_sobol_pairs.h, ob_engine.hpp sobol_pairs,
ob_kernels.cu sobol_pairs_kernel).

CPU: the exported ABI, and a numpy restatement of the header's second and supset forms against brute force on the full
tensor grid of X_q's columns (every ANOVA component variance from grid conditional means by inclusion-exclusion),
evaluated by the oracle.  GPU: the product against that restatement fed the product's own basis at X_q, brute force with
the product's matmul, the four outputs of ob_sobol bit for bit, determinism and column independence, the identities
between the forms, the semantics of the measure, obsobol(second=True) on fits, and the refusals."""
import itertools
import types

import numpy as np
import pytest

from conftest import borehole8d
from outerbase_b200 import fitting
from outerbase_b200.binding import _p, _u, posterior_draws, sobol, sobol_pairs
from test_sobol import CASES, FWD, STAGE_BYTES, random_problem, sobol_tables


# ------------------------------------------------------------------------------------------ numpy restatement
def pairs_reference(lib, om, terms, coeff, xq, pairs=None, tabs=None):
    """second[l, m] = sum theta theta' c_l c_m prod_{j not in {l,m}} p_j and supset[l, m] the same with g_j, from the K x K
    pair matrices, built one dimension at a time (memory for a few K x K matrices only).  pairs: the (l, m) to restate,
    default all.  Also returns the bound of the error check: |theta|^T A |theta|, A the pair factors of the absolute
    tables, as in test_sobol."""
    t = np.asarray(terms, dtype=np.int64)
    th = np.asarray(coeff, dtype=float).reshape((t.shape[0], -1), order="F")
    tabs = tabs or sobol_tables(lib, om, terms, xq)
    d = t.shape[1]
    pairs = [(l, m) for l in range(d) for m in range(l + 1, d)] if pairs is None else list(pairs)

    def p(j):
        return np.outer(tabs[j]["mu"][t[:, j]], tabs[j]["mu"][t[:, j]])

    def c(j):
        return tabs[j]["C"][np.ix_(t[:, j], t[:, j])]

    def form(M, a=th):
        return ((M @ a) * a).sum(axis=0)

    second, supset = {}, {}
    for l, m in pairs:
        S2 = c(l) * c(m)
        SU = S2.copy()
        for j in range(d):
            if j not in (l, m):
                pj = p(j)
                S2 *= pj
                SU *= c(j) + pj
        second[l, m], supset[l, m] = form(S2), form(SU)
    A = np.ones((t.shape[0], t.shape[0]))
    for j, T in enumerate(tabs):
        A *= np.outer(T["mua"][t[:, j]], T["mua"][t[:, j]]) + T["Ca"][np.ix_(t[:, j], t[:, j])]
    return dict(second=second, supset=supset, bound=form(A, np.abs(th)))


def anova_brute_force(lib, om, terms, coeff, xq):
    """sigma2_u of every non-empty input set u on the full tensor grid of xq's columns: the ANOVA component
    f_u = sum_{v subset of u} (-1)^{|u| - |v|} E[f | x_v] from the grid conditional means, sigma2_u = its mean square.
    Returns {u: sigma2_u (B)} and the grid variance."""
    n, d = xq.shape
    grid = np.stack(np.meshgrid(*[xq[:, l] for l in range(d)], indexing="ij"), axis=-1).reshape(-1, d)
    th = np.asarray(coeff, dtype=float).reshape((terms.shape[0], -1), order="F")
    F = lib.outerbase(om, np.asfortranarray(grid), dograd=False).matmul(terms, th).reshape((n,) * d + (-1,))
    axes = tuple(range(d))
    cond = {v: F.mean(axis=tuple(a for a in axes if a not in v), keepdims=True)
            for r in range(d + 1) for v in itertools.combinations(axes, r)}
    sig = {}
    for r in range(1, d + 1):
        for u in itertools.combinations(axes, r):
            fu = sum((-1) ** (len(u) - len(v)) * cond[v] for k in range(len(u) + 1) for v in itertools.combinations(u, k))
            sig[u] = (fu ** 2).mean(axis=axes)
    return sig, F.var(axis=axes)


def brute_pairs(sig, d):
    """second (sigma2_lm) and supset (sum of sigma2_u over u containing l and m) from the component variances"""
    second = {(l, m): sig[(l, m)] for l in range(d) for m in range(l + 1, d)}
    supset = {(l, m): sum(s for u, s in sig.items() if l in u and m in u) for l in range(d) for m in range(l + 1, d)}
    return second, supset


# ---------------------------------------------------------------------------------------------------- CPU
def test_product_exports_the_sobol_pairs_abi(product_symbols):
    import outerbase_b200 as ob
    syms = ob.header_symbols(ob.SOBOL_PAIRS_HEADER)
    assert syms == ["ob_sobol_pairs"]
    assert all(product_symbols.has(s) for s in syms)


@pytest.mark.parametrize("d,n,K,B,seed", [(2, 14, 30, 3, 1), (3, 12, 40, 3, 2), (3, 8, 60, 2, 3), (4, 9, 60, 3, 4)])
def test_pairs_reference_matches_brute_force_on_the_oracle(oracle, d, n, K, B, seed):
    om, terms, coeff, xq = random_problem(oracle, d, [12 + 3 * l for l in range(d)], K, B, n, seed)
    ref = pairs_reference(oracle, om, terms, coeff, xq)
    sig, var = anova_brute_force(oracle, om, terms, coeff, xq)
    scale = np.max(var)
    assert scale > 0
    # the components add up to the variance: the brute force itself is consistent
    np.testing.assert_allclose(sum(sig.values()), var, rtol=0, atol=1e-12 * scale)
    second, supset = brute_pairs(sig, d)
    for lm in second:
        np.testing.assert_allclose(ref["second"][lm], second[lm], rtol=0, atol=1e-12 * scale, err_msg=f"second {lm}")
        np.testing.assert_allclose(ref["supset"][lm], supset[lm], rtol=0, atol=1e-12 * scale, err_msg=f"supset {lm}")
    # the forms are not trivially zero
    assert all(np.all(ref["supset"][lm] > 0) for lm in second)


# ---------------------------------------------------------------------------------------------------- GPU
def check_against_reference(gpu, om, terms, coeff, xq, pairs=None, what=""):
    """sobol_pairs element-wise against the restatement on `pairs` (default all), its four other outputs bit for bit
    against sobol, and the diagonal and symmetry of the d x d arrays"""
    got = sobol_pairs(gpu, om, terms, coeff, xq)
    one = sobol(gpu, om, terms, coeff, xq)
    for key in ("mean", "var", "first", "total"):
        np.testing.assert_array_equal(got[key], one[key], err_msg=what + " " + key)
    d = terms.shape[1]
    B = np.asarray(coeff).reshape((terms.shape[0], -1), order="F").shape[1]
    S2 = got["second"].reshape((d, d, B))
    SU = got["supset"].reshape((d, d, B))
    assert np.all(np.isnan(S2[np.arange(d), np.arange(d)])) and np.all(np.isnan(SU[np.arange(d), np.arange(d)]))
    ref = pairs_reference(gpu, om, terms, coeff, xq, pairs=pairs)
    bound = FWD * ref["bound"]
    for (l, m), want in ref["second"].items():
        assert S2[l, m].tolist() == S2[m, l].tolist() and SU[l, m].tolist() == SU[m, l].tolist()
        assert np.all(np.abs(S2[l, m] - want) <= bound), f"{what} second ({l}, {m})"
        assert np.all(np.abs(SU[l, m] - ref["supset"][l, m]) <= bound), f"{what} supset ({l}, {m})"
    return got, ref


PAIR_CASES = CASES + [  # d, knots per dimension, K, B, n_q
    (2, [12, 17], 40, 5, 300),
    (40, [6] * 40, 120, 3, 500),  # 780 pairs: 13 output blocks per term-pair chunk
]


@pytest.mark.gpu
@pytest.mark.parametrize("d,knots,K,B,nq", PAIR_CASES)
def test_pairs_against_the_restatement(gpu, d, knots, K, B, nq):
    om, terms, coeff, xq = random_problem(gpu, d, knots, K, B, nq, seed=d * 1000 + K + B)
    got, _ = check_against_reference(gpu, om, terms, coeff, xq, what=f"d={d} K={K} B={B} nq={nq}")
    assert got["second"].shape == (d, d, B)


@pytest.mark.gpu
def test_one_dimension_writes_no_pair_output(gpu):
    """d = 1: P = 0, nothing is written (null pointers are accepted), and the other four outputs are sobol's"""
    om, terms, coeff, xq = random_problem(gpu, 1, [15], 10, 3, 200, seed=3)
    one = sobol(gpu, om, terms, coeff, xq)
    K, B = coeff.shape
    t = np.asfortranarray(terms.astype(np.uint64))
    for sentinel in (None, 7.25):
        mean, var = np.empty(B), np.empty(B)
        first, total = np.empty((1, B), order="F"), np.empty((1, B), order="F")
        second = None if sentinel is None else np.full(4, sentinel)
        supset = None if sentinel is None else np.full(4, sentinel)
        gpu.call("sobol_pairs", gpu.ctx, om._h, _p(t), _u(K), _p(coeff), _u(B), _p(xq), _u(xq.shape[0]), _p(mean),
                 _p(var), _p(first), _p(total), None if second is None else _p(second), None if supset is None else _p(supset))
        np.testing.assert_array_equal(mean, one["mean"])
        np.testing.assert_array_equal(var, one["var"])
        np.testing.assert_array_equal(first, one["first"])
        np.testing.assert_array_equal(total, one["total"])
        if sentinel is not None:
            assert np.all(second == sentinel) and np.all(supset == sentinel)
    got = sobol_pairs(gpu, om, terms, coeff, xq)
    assert got["second"].shape == (1, 1, B) and np.all(np.isnan(got["second"])) and np.all(np.isnan(got["supset"]))


@pytest.mark.gpu
def test_pairs_on_tables_beyond_the_staging_size(gpu):
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
@pytest.mark.parametrize("B,nq", [(1, 1_000_000), (64, 20_000)])
def test_pairs_on_the_c3_table(gpu, B, nq):
    import bench
    om, terms = bench.setup_model(gpu)
    rng = np.random.default_rng(B)
    coeff = np.asfortranarray(rng.normal(size=(terms.shape[0], B)) / (1 + terms.sum(axis=1))[:, None])
    xq = bench.synth_rows(0, nq, bench.D)
    check_against_reference(gpu, om, terms, coeff, xq, what=f"C3 B={B} nq={nq}")


@pytest.mark.gpu
def test_pairs_on_the_c4_table_on_a_sample_of_pairs(gpu):
    """d = 20, K = 4000: 190 pairs, three output blocks; the restatement on pairs from each block and the last"""
    import bench
    om, terms = bench.config_model(gpu, "c4share")
    assert terms.shape == (4000, 20)
    rng = np.random.default_rng(4)
    coeff = np.asfortranarray(rng.normal(size=(terms.shape[0], 64)) / (1 + terms.sum(axis=1))[:, None])
    xq = bench.config_rows("c4share", 0, 20_000)
    check_against_reference(gpu, om, terms, coeff, xq, pairs=[(0, 1), (3, 17), (7, 8), (12, 19), (18, 19)], what="C4")


@pytest.mark.gpu
@pytest.mark.parametrize("d,n,K,B,seed", [(3, 12, 40, 3, 1), (4, 9, 60, 3, 3)])
def test_pairs_brute_force_on_the_gpu(gpu, d, n, K, B, seed):
    om, terms, coeff, xq = random_problem(gpu, d, [12 + 3 * l for l in range(d)], K, B, n, seed)
    got = sobol_pairs(gpu, om, terms, coeff, xq)
    sig, var = anova_brute_force(gpu, om, terms, coeff, xq)
    scale = np.max(var)
    second, supset = brute_pairs(sig, d)
    for l, m in second:
        np.testing.assert_allclose(got["second"][l, m], second[l, m], rtol=0, atol=1e-11 * scale)
        np.testing.assert_allclose(got["supset"][l, m], supset[l, m], rtol=0, atol=1e-11 * scale)


@pytest.mark.gpu
def test_pairs_determinism_and_column_independence(gpu):
    om, terms, coeff, xq = random_problem(gpu, 12, [16] * 12, 300, 65, 20_000, seed=9)
    a = sobol_pairs(gpu, om, terms, coeff, xq)
    b = sobol_pairs(gpu, om, terms, coeff, xq)
    for key in a:
        np.testing.assert_array_equal(a[key], b[key])
    for j in (0, 1, 31, 32, 33, 63, 64):
        one = sobol_pairs(gpu, om, terms, coeff[:, j], xq)
        np.testing.assert_array_equal(one["second"], a["second"][:, :, j])
        np.testing.assert_array_equal(one["supset"], a["supset"][:, :, j])


def upper(M):
    d = M.shape[0]
    l, m = np.triu_indices(d, 1)
    return M[l, m]


@pytest.mark.gpu
@pytest.mark.parametrize("d,seed", [(2, 1), (3, 2), (6, 3)])
def test_pair_identities(gpu, d, seed):
    om, terms, coeff, xq = random_problem(gpu, d, [14] * d, 80, 4, 3000, seed=seed)
    r = sobol_pairs(gpu, om, terms, coeff, xq)
    tol = 1e-10 * pairs_reference(gpu, om, terms, coeff, xq, pairs=[])["bound"]
    second, supset = upper(r["second"]), upper(r["supset"])  # P x B
    l, m = np.triu_indices(d, 1)
    assert np.all(second >= -tol) and np.all(second <= supset + tol)
    assert np.all(supset <= np.minimum(r["total"][l], r["total"][m]) + tol)
    assert np.all(r["first"].sum(axis=0) + second.sum(axis=0) <= r["var"] + tol)
    if d == 2:
        rest = r["var"] - r["first"][0] - r["first"][1]
        assert np.all(np.abs(second[0] - rest) <= tol) and np.all(np.abs(supset[0] - rest) <= tol)
    if d == 3:
        s012 = r["var"] - r["first"].sum(axis=0) - second.sum(axis=0)  # sigma2 of {0, 1, 2}
        assert np.all(np.abs((supset - second) - s012[None, :]) <= 2 * tol)
        assert np.all(s012 > tol)  # the check is not vacuous


@pytest.mark.gpu
def test_pairs_measure_semantics(gpu):
    om, terms, coeff, xq = random_problem(gpu, 6, [20] * 6, 60, 8, 3000, seed=5)
    a = sobol_pairs(gpu, om, terms, coeff, xq)
    scale = a["var"][None, None, :]
    off = ~np.eye(6, dtype=bool)
    # stacking X_q twice changes nothing
    b = sobol_pairs(gpu, om, terms, coeff, np.asfortranarray(np.vstack([xq, xq])))
    for key in ("second", "supset"):
        assert np.all(np.abs(a[key] - b[key])[off] <= 1e-13 * np.broadcast_to(scale, a[key].shape)[off]), key
    # ... and the pairing within rows does not matter: each column permuted on its own
    rng = np.random.default_rng(0)
    xp = np.asfortranarray(np.stack([rng.permutation(xq[:, l]) for l in range(xq.shape[1])], axis=1))
    c = sobol_pairs(gpu, om, terms, coeff, xp)
    for key in ("second", "supset"):
        assert np.all(np.abs(a[key] - c[key])[off] <= 1e-12 * np.broadcast_to(scale, a[key].shape)[off]), key


@pytest.fixture(scope="module")
def borehole_fit(gpu):
    rng = np.random.default_rng(21)
    x = np.asfortranarray(rng.uniform(size=(3000, 8)))
    model = fitting.obfit(gpu, x, borehole8d(x), numb=200, numberopts=1, seed=1)
    xq = np.asfortranarray(np.random.default_rng(22).uniform(size=(20_000, 8)))
    return model, xq


def pair_indices_of(r):
    """what obsobol(second=True) derives from sobol_pairs, restated"""
    var = r["var"]
    f = r["first"]
    return dict(second=r["second"] / var, closed=(f[:, None] + f[None, :] + r["second"]) / var, supset=r["supset"] / var)


@pytest.mark.gpu
def test_obsobol_second_on_the_borehole_function(borehole_fit):
    model, xq = borehole_fit
    lib = model["logpdf"]._lib
    res = fitting.obsobol(model, xq, second=True)
    plain = fitting.obsobol(model, xq)
    assert set(plain) == {"first", "total", "var", "mean"}
    assert set(res) == set(plain) | {"second", "closed", "supset"}
    for key in plain:
        np.testing.assert_array_equal(res[key], plain[key])
    r = sobol_pairs(lib, model["om"], model["terms"], model["logpdf"].coeff, xq)
    for key, want in pair_indices_of(r).items():
        assert res[key].shape == (8, 8)
        np.testing.assert_array_equal(res[key], want)
    # second=False is what obsobol returned before: sobol's forms over the variance
    one = sobol(lib, model["om"], model["terms"], model["logpdf"].coeff, xq)
    np.testing.assert_array_equal(plain["first"], one["first"] / one["var"])
    np.testing.assert_array_equal(plain["total"], one["total"] / one["var"])
    assert plain["var"] == model["y_sca"] ** 2 * one["var"]
    # the borehole function: the interactions are small (total - first of r_w is about 0.04), the inert inputs
    # (r, T_u, T_l) take part in none, and the pure interaction indices fill the gap between sum first and 1
    off = ~np.eye(8, dtype=bool)
    assert np.nanmax(res["supset"][[1, 2, 4]]) < 0.01
    assert np.all(res["second"][off] >= -1e-12) and np.all(res["second"][off] <= res["supset"][off] + 1e-12)
    assert 0 < res["second"][off].sum() / 2 <= 1 - res["first"].sum() + 1e-9
    assert abs(res["closed"][0, 7] - (res["first"][0] + res["first"][7] + res["second"][0, 7])) < 1e-14


@pytest.mark.gpu
def test_obsobol_second_draws_equal_sobol_pairs_on_the_draws(borehole_fit):
    model, xq = borehole_fit
    lib = model["logpdf"]._lib
    res = fitting.obsobol(model, xq, S=8, seed=4, second=True)
    dr = res["draws"]
    assert dr["second"].shape == (8, 8, 8) and dr["first"].shape == (8, 8)
    coeff = posterior_draws(lib, model["logpdf"], 8, 4).solve(0.001, 100).coeff
    r = sobol_pairs(lib, model["om"], model["terms"], coeff, xq)
    for key, want in pair_indices_of(r).items():
        np.testing.assert_array_equal(dr[key], want)
    np.testing.assert_array_equal(dr["first"], r["first"] / r["var"])


@pytest.mark.gpu
def test_obsobol_second_on_a_multi_response_fit(gpu):
    rng = np.random.default_rng(31)
    x = np.asfortranarray(rng.uniform(size=(1500, 3)))
    Y = np.column_stack([np.sin(6 * x[:, 0]) + x[:, 1], x[:, 1] * x[:, 2] + 0.2 * x[:, 0], np.exp(x[:, 2])])
    model = fitting.obfit_multi(gpu, x, Y, numb=40, covnames=["mat25pow"] * 3, numberopts=1)
    xq = np.asfortranarray(rng.uniform(size=(4000, 3)))
    res = fitting.obsobol(model, xq, second=True)
    assert res["second"].shape == (3, 3, 3) and res["closed"].shape == (3, 3, 3) and res["first"].shape == (3, 3)
    coeff = model["logpdf"].coeff
    for c in range(3):
        one = sobol_pairs(gpu, model["om"], model["terms"], coeff[:, c], xq)
        for key, want in pair_indices_of(one).items():
            np.testing.assert_array_equal(res[key][:, :, c], want)
    # column 0 is additive, column 1 carries the x_2 x_3 interaction, column 2 depends on x_3 alone
    assert res["supset"][0, 1, 0] < 0.01 and res["second"][1, 2, 1] > 0.02 and res["supset"][0, 1, 2] < 0.01


@pytest.mark.gpu
def test_zero_variance_gives_nan_pair_indices(gpu, recwarn):
    om, terms, coeff, xq = random_problem(gpu, 3, [10, 10, 10], 20, 2, 500, seed=8)
    fit = types.SimpleNamespace(_lib=gpu, coeff=np.zeros(terms.shape[0]))  # what obsobol reads of a fitted logpdf
    res = fitting.obsobol(dict(logpdf=fit, om=om, terms=terms, y_cent=0.0, y_sca=1.0), xq, second=True)
    assert res["var"] == 0
    for key in ("second", "closed", "supset"):
        assert res[key].shape == (3, 3) and np.all(np.isnan(res[key])), key
    assert not [w for w in recwarn if issubclass(w.category, RuntimeWarning)]


@pytest.mark.gpu
def test_pairs_refusals(gpu):
    om, terms, coeff, xq = random_problem(gpu, 3, [10, 12, 14], 20, 2, 100, seed=6)
    with pytest.raises(ValueError, match="at least one column"):
        sobol_pairs(gpu, om, terms, np.zeros((terms.shape[0], 0)), xq)
    with pytest.raises(ValueError, match="at least one row"):
        sobol_pairs(gpu, om, terms, coeff, np.zeros((0, 3), order="F"))
    with pytest.raises(ValueError, match="terms table is empty"):
        sobol_pairs(gpu, om, np.zeros((0, 3), dtype=np.uint64), np.zeros(0), xq)
    with pytest.raises(ValueError, match="columns, the outermod 3 dimensions"):
        sobol_pairs(gpu, om, np.zeros((5, 4), dtype=np.uint64), np.ones(5), xq)
    with pytest.raises(ValueError, match="x must be nq x d"):
        sobol_pairs(gpu, om, terms, coeff, np.zeros((10, 4), order="F"))
    # d = 78: beyond what the forms kernel holds
    om78, terms78, coeff78, xq78 = random_problem(gpu, 78, [5] * 78, 100, 1, 50, seed=7)
    with pytest.raises(ValueError, match="more dimensions"):
        sobol_pairs(gpu, om78, terms78, coeff78, xq78)


@pytest.mark.gpu
def test_pairs_at_77_dimensions(gpu):
    """the largest d the forms kernel holds: 2926 pairs, 5852 pair outputs per column, 46 output blocks"""
    om, terms, coeff, xq = random_problem(gpu, 77, [5] * 77, 100, 2, 50, seed=7)
    got, _ = check_against_reference(gpu, om, terms, coeff, xq, pairs=[(0, 1), (0, 76), (37, 38), (75, 76)], what="d=77")
    assert np.isfinite(upper(got["second"][:, :, 0])).all()
