"""Posterior draws of a fitted model by perturb-and-MAP (include/outerbase_b200_draws.h, ob_engine.hpp Draws).

CPU: the generator (Philox4x32-10 + Box-Muller) against the Random123 known answers and a numpy restatement, the
statistics of its normals, and the prior mean of logpr_gauss_multi on the host path.  GPU: the device perturbations
against the host generator, each draw against numpy's dense solve of the perturbed system, the distribution of many
draws against the dense posterior, reproducibility, prediction, the C3 size and the refusals."""
import numpy as np
import pytest

from conftest import make_problem, relerr
from outerbase_b200 import fitting
from outerbase_b200.binding import posterior_draws

U32 = np.uint64(0xFFFFFFFF)


# ------------------------------------------------------------------------------------------ numpy restatement
def philox4x32_10(ctr, key):
    """Philox4x32-10 on arrays of counters (4 x n uint64 words < 2^32) and one key (2 words)."""
    c = [np.asarray(v, dtype=np.uint64) & U32 for v in ctr]
    k0, k1 = np.uint64(key[0]), np.uint64(key[1])
    for r in range(10):
        if r:
            k0 = (k0 + np.uint64(0x9E3779B9)) & U32
            k1 = (k1 + np.uint64(0xBB67AE85)) & U32
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & U32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & U32]
    return c


def normals(seed, stream, column, first, n):
    """Normals first .. first + n - 1 of (seed, stream, column), as the header defines them."""
    idx = np.arange(first, first + n, dtype=np.uint64)
    pair = np.unique(idx >> np.uint64(1))
    v = philox4x32_10([pair, np.full_like(pair, stream), np.full_like(pair, column), np.zeros_like(pair)],
                      [seed & 0xFFFFFFFF, seed >> 32])
    u1 = (((v[1] << np.uint64(32)) | v[0]) >> np.uint64(11)).astype(np.float64) + 1.0
    u2 = (((v[3] << np.uint64(32)) | v[2]) >> np.uint64(11)).astype(np.float64) + 1.0
    r = np.sqrt(-2.0 * np.log(u1 * 2.0 ** -53))
    th = 6.283185307179586 * (u2 * 2.0 ** -53)
    z = np.empty(2 * pair.size)
    z[0::2], z[1::2] = r * np.cos(th), r * np.sin(th)
    return z[(idx - 2 * pair[0]).astype(np.int64)]


# ---------------------------------------------------------------------------------------------------- CPU
def test_product_exports_the_draws_abi(product_symbols):
    import outerbase_b200 as ob
    syms = ob.header_symbols(ob.DRAWS_HEADER)
    assert syms == ["ob_draws_create", "ob_draws_destroy", "ob_draws_solve", "ob_draws_get", "ob_draws_predict",
                    "ob_debug_normals", "ob_logpr_gauss_multi_set_mean"]
    assert all(product_symbols.has(s) for s in syms)


def test_philox_known_answers():
    """Random123's known-answer vectors for Philox4x32-10"""
    cases = [([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
             ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
             ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
              [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]
    for ctr, key, want in cases:
        got = philox4x32_10([np.array([w], dtype=np.uint64) for w in ctr], key)
        assert [int(w[0]) for w in got] == want


def test_host_generator_matches_the_restatement(product_symbols):
    for seed, stream, column, first, n in [(0, 0, 0, 0, 1000), (12345, 1, 7, 3, 999), (2 ** 40 + 17, 0, 2 ** 31 + 5, 2 ** 32 + 1, 64),
                                           (7, 1, 0, 11, 1)]:
        got = product_symbols.debug_normals(seed, stream, column, first, n)
        want = normals(seed, stream, column, first, n)
        assert relerr(got, want) < 1e-14, (seed, stream, column, first)
    # a value depends on its index only, not on where the request starts
    a = product_symbols.debug_normals(5, 0, 3, 0, 101)
    np.testing.assert_array_equal(product_symbols.debug_normals(5, 0, 3, 37, 40), a[37:77])
    with pytest.raises(ValueError, match="32-bit"):
        product_symbols.debug_normals(0, 0, 2 ** 32, 0, 4)


def test_normal_statistics(product_symbols):
    n = 10 ** 6
    z = product_symbols.debug_normals(2024, 0, 3, 0, n)
    se = 1 / np.sqrt(n)
    assert abs(z.mean()) < 5 * se
    assert abs(z.var() - 1) < 5 * np.sqrt(2.0 / n)
    assert abs(np.mean(z[1:] * z[:-1])) < 5 * se  # lag 1: the two normals of one output
    assert abs(np.mean(z[2:] * z[:-2])) < 5 * se  # lag 2: neighbouring outputs
    w = product_symbols.debug_normals(2024, 1, 3, 0, n)  # the other stream, same column
    assert abs(np.mean(z * w)) < 5 * se
    v = product_symbols.debug_normals(2024, 0, 4, 0, n)  # the next column
    assert abs(np.mean(z * v)) < 5 * se
    assert abs(np.mean(z ** 4) - 3) < 5 * np.sqrt(96.0 / n)  # kurtosis of a normal (variance of z^4 is 96)
    assert not np.array_equal(z[:100], product_symbols.debug_normals(2025, 0, 3, 0, 100))
    assert not np.array_equal(z[:100], v[:100]) and not np.array_equal(z[:100], w[:100])


def test_prior_mean_on_the_host_path(product_symbols):
    """logpr_gauss_multi's update with a prior mean is the written-out formula; without one it is today's"""
    L = product_symbols
    om = L.outermod()
    om.setcovfs(["mat25pow", "mat25", "mat25"])
    om.setknot([np.arange(0.001, 0.999, 0.05)] * 3)
    terms = om.selectterms(40)
    K, C = terms.shape[0], 3
    rng = np.random.default_rng(4)
    theta = np.asfortranarray(rng.normal(size=(K, C)) * 0.1)
    M = np.asfortranarray(rng.normal(size=(K, C)) * 0.1)
    pr = L.logpr_gauss_multi(om, terms, C)
    pr.updatepara([0.3])
    plain = L.logpr_gauss_multi(om, terms, C)
    plain.updatepara([0.3])
    sd = np.sqrt(om.getvar(terms)) * np.exp(0.3)

    def evaluate(obj):
        obj.compute_val = True; obj.compute_grad = True
        obj.update(theta)
        return obj.val, obj.grad.copy()

    pr.set_mean(M)
    val, grad = evaluate(pr)
    st = (theta - M) / sd[:, None]
    assert abs(val - (-0.5 * np.sum(st ** 2) - C * np.sum(np.log(sd)))) <= 1e-13 * abs(val)
    np.testing.assert_allclose(grad, -st / sd[:, None], rtol=1e-14, atol=0)
    pr.set_mean(None)
    val0, grad0 = evaluate(pr)
    pv, pg = evaluate(plain)  # an object that never had a mean: today's values, bit for bit
    assert val0 == pv
    np.testing.assert_array_equal(grad0, pg)
    st0 = theta / sd[:, None]
    assert abs(val0 - (-0.5 * np.sum(st0 ** 2) - C * np.sum(np.log(sd)))) <= 1e-13 * abs(val0)
    with pytest.raises(ValueError, match="K x ncol"):
        pr.set_mean(np.zeros(K))


# ---------------------------------------------------------------------------------------------------- GPU
N_SMALL, K_SMALL, D_SMALL = 3000, 150, 6


@pytest.fixture
def families(gpu):
    """the interpreter kernels (spec 0) and the terms-specialised ones compiled at first use (spec 1)"""
    def run(spec):
        gpu.set_option("spec", spec)
    yield run
    gpu.set_option("spec", 2)


def small_fit(lib, lik_first=False):
    """the small model, fitted briefly: one optcg at the default hyper-parameters and para"""
    om, x, y, terms, rng = make_problem(lib, N_SMALL, K_SMALL, d=D_SMALL, covs=["mat25pow"] * D_SMALL)
    logpr, loglik = lib.logpr_gauss(om, terms), lib.loglik_gauss(om, terms, y, x)
    vec = lib.lpdfvec(loglik, logpr) if lik_first else lib.lpdfvec(logpr, loglik)
    vec.domarg = True
    vec.optcg(0.001, 100)
    return dict(om=om, x=x, y=y, terms=terms, logpr=logpr, loglik=loglik, vec=vec, rng=rng)


def dense_posterior(lib, fit):
    """Phi (getmat), sigma, the prior sds and H = Phi^T Phi / sigma^2 + D^-1"""
    Phi = lib.outerbase(fit["om"], fit["x"]).getmat(fit["terms"])
    sigma = float(np.exp(fit["loglik"].para[0]))
    sd = fit["logpr"].coeffsd * float(np.exp(fit["logpr"].para[0]))
    H = Phi.T @ Phi / sigma ** 2 + np.diag(1 / sd ** 2)
    return Phi, sigma, sd, H


@pytest.mark.gpu
def test_gpu_perturbations_match_the_host_generator(gpu):
    fit = small_fit(gpu)
    S, seed = 5, 11
    dr = posterior_draws(gpu, fit["vec"], S, seed)
    sigma = float(np.exp(fit["loglik"].para[0]))
    sd = fit["logpr"].coeffsd * float(np.exp(fit["logpr"].para[0]))
    Ys, D = dr.y, dr.prior_mean
    assert Ys.shape == (N_SMALL, S) and D.shape == (K_SMALL, S)
    for s in range(S):
        assert relerr((Ys[:, s] - fit["y"]) / sigma, gpu.debug_normals(seed, 0, s, 0, N_SMALL)) < 1e-14, s
        assert relerr(D[:, s] / sd, gpu.debug_normals(seed, 1, s, 0, K_SMALL)) < 1e-14, s


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [0, 1])
def test_gpu_each_draw_is_the_exact_perturbed_solve(gpu, families, spec):
    families(spec)
    fit = small_fit(gpu)
    Phi, sigma, sd, H = dense_posterior(gpu, fit)
    dr = posterior_draws(gpu, fit["vec"], 8, 3).solve(tol=1e-13, maxepch=2000)
    theta = np.linalg.solve(H, Phi.T @ dr.y / sigma ** 2 + dr.prior_mean / sd[:, None] ** 2)
    for s in range(8):
        assert relerr(dr.coeff[:, s], theta[:, s]) < 1e-8, (s, relerr(dr.coeff[:, s], theta[:, s]))
    assert np.all(dr.cg_iters > 0)


@pytest.mark.gpu
def test_gpu_draws_follow_the_dense_posterior(gpu):
    """S = 2048 draws at 20 new points: sample mean, variance and the covariance of two points against the dense
    posterior mean Phi* mu and covariance Phi* H^-1 Phi*^T, within 5 standard errors (fixed seed: deterministic)"""
    fit = small_fit(gpu)
    Phi, sigma, sd, H = dense_posterior(gpu, fit)
    Hi = np.linalg.inv(H)
    mu = Hi @ (Phi.T @ fit["y"]) / sigma ** 2
    xs = np.asfortranarray(np.random.default_rng(21).uniform(size=(20, D_SMALL)))
    Ps = gpu.outerbase(fit["om"], xs).getmat(fit["terms"])
    mean, cov = Ps @ mu, Ps @ Hi @ Ps.T
    S = 2048
    f = posterior_draws(gpu, fit["vec"], S, 77).solve(tol=1e-10, maxepch=2000).predict(xs)
    var = np.diag(cov)
    assert np.all(np.abs(f.mean(axis=1) - mean) < 5 * np.sqrt(var / S))
    assert np.all(np.abs(f.var(axis=1, ddof=1) - var) < 5 * var * np.sqrt(2.0 / (S - 1)))
    c01 = np.cov(f[0], f[1])[0, 1]
    assert abs(c01 - cov[0, 1]) < 5 * np.sqrt((var[0] * var[1] + cov[0, 1] ** 2) / S)


@pytest.mark.gpu
def test_gpu_draws_are_reproducible_and_independent_of_s(gpu):
    fit = small_fit(gpu, lik_first=True)
    a = posterior_draws(gpu, fit["vec"], 8, 5)
    b = posterior_draws(gpu, fit["vec"], 8, 5)
    c = posterior_draws(gpu, fit["vec"], 16, 5)
    # the object is a snapshot: later changes to the om and the fit do not reach it
    hyp = fit["om"].gethyp()
    fit["om"].updatehyp(hyp + 0.05)
    fit["vec"].updateom()
    fit["vec"].updatepara(fit["vec"].para + 0.1)
    for d in (a, b, c):
        d.solve()
    np.testing.assert_array_equal(a.y, b.y)
    np.testing.assert_array_equal(a.prior_mean, b.prior_mean)
    np.testing.assert_array_equal(a.coeff, b.coeff)
    np.testing.assert_array_equal(a.cg_iters, b.cg_iters)
    np.testing.assert_array_equal(c.y[:, :8], a.y)
    np.testing.assert_array_equal(c.prior_mean[:, :8], a.prior_mean)
    np.testing.assert_array_equal(c.cg_iters[:8], a.cg_iters)
    assert relerr(c.coeff[:, :8], a.coeff) < 1e-10
    assert not np.array_equal(posterior_draws(gpu, fit["vec"], 8, 6).y, a.y)


@pytest.mark.gpu
def test_gpu_predict_is_phi_times_the_draws(gpu):
    fit = small_fit(gpu)
    dr = posterior_draws(gpu, fit["vec"], 12, 1).solve()
    xs = np.asfortranarray(np.random.default_rng(8).uniform(size=(500, D_SMALL)))
    Ps = gpu.outerbase(fit["om"], xs).getmat(fit["terms"])
    assert relerr(dr.predict(xs), Ps @ dr.coeff) < 1e-12


@pytest.mark.gpu
def test_gpu_obdraws_in_the_units_of_y(gpu):
    rng = np.random.default_rng(5)
    x = np.asfortranarray(rng.uniform(size=(400, 3)))
    f = lambda x: 20 + 3 * (np.sin(3 * x[:, 0]) + x[:, 1] * x[:, 2])
    model = fitting.obfit_gauss(gpu, x, f(x) + 0.01 * rng.normal(size=400), numb=30, numberopts=1)
    xt = np.asfortranarray(rng.uniform(size=(50, 3)))
    draws = fitting.obdraws(model, xt, S=32, seed=4)
    assert draws.shape == (50, 32)
    f_std = posterior_draws(gpu, model["logpdf"], 32, 4).solve().predict(xt)
    np.testing.assert_array_equal(draws, model["y_cent"] + model["y_sca"] * f_std)
    # the draws scatter around the fit's prediction, in y's units
    pred = fitting.obpred(model, xt)["mean"]
    assert np.max(np.abs(draws.mean(axis=1) - pred)) < 0.1 * np.std(f(xt))


@pytest.mark.gpu
def test_gpu_draws_at_c3_size(gpu, families):
    """C3 rows (N = 1M, K = 2000, specialised) with S = 64: the solve finishes with finite draws, and a CG iteration
    takes the launches of the multi-response CG at the same C (nothing N x S goes through the host)"""
    import bench
    families(1)
    N, S = bench.N_TOTAL, 64
    x = bench.synth_rows(0, N, bench.D)
    y = bench.wingweight(x)
    y = (y - y.mean()) / y.std()
    om, terms = bench.setup_model(gpu)
    K = terms.shape[0]
    vec = gpu.lpdfvec(gpu.logpr_gauss(om, terms), gpu.loglik_gauss(om, terms, y, x))
    vec.domarg = True
    vec.optcg(0.001, 100)
    dr = posterior_draws(gpu, vec, S, 9).solve()
    assert dr.coeff.shape == (K, S) and np.all(np.isfinite(dr.coeff))
    assert np.all(dr.cg_iters > 0) and np.all(dr.cg_iters <= 100)

    def per_iteration(run):
        run(1)  # warm
        counts = []
        for epochs in (2, 6):
            n0 = gpu.launch_count()
            run(epochs)
            counts.append(gpu.launch_count() - n0)
        return (counts[1] - counts[0]) / 4

    draws_per = per_iteration(lambda e: dr.solve(-1.0, e))  # tol < 0: no column ever stops
    Y = np.asfortranarray(np.repeat(y[:, None], S, axis=1))
    multi = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, S), gpu.loglik_gauss_multi(om, terms, Y, x))
    del Y

    def run_multi(e):
        multi.set_coeff(np.zeros(K * S))
        multi.optcg(-1.0, e)
    assert draws_per == per_iteration(run_multi), draws_per


@pytest.mark.gpu
def test_gpu_refusals(gpu):
    om, x, y, terms, _ = make_problem(gpu, 400, 40)
    logpr = gpu.logpr_gauss(om, terms)
    vec = gpu.lpdfvec(logpr, gpu.loglik_gauss(om, terms, y, x))
    with pytest.raises(ValueError, match="S must be at least 1"):
        posterior_draws(gpu, vec, 0, 0)
    Y = np.asfortranarray(np.column_stack([y, 2 * y]))
    for percol in (False, True):
        mv = gpu.lpdfvec(gpu.logpr_gauss_multi(om, terms, 2, para_per_column=percol),
                         gpu.loglik_gauss_multi(om, terms, Y, x, para_per_column=percol))
        with pytest.raises(ValueError, match="multi-response and per-column-para fits are not supported"):
            posterior_draws(gpu, mv, 4, 0)
    with pytest.raises(ValueError, match="loglik_gda fits are not supported"):
        posterior_draws(gpu, gpu.lpdfvec(logpr, gpu.loglik_gda(om, terms, y, x)), 4, 0)
    with pytest.raises(ValueError, match="loglik_std fits are not supported"):
        posterior_draws(gpu, gpu.lpdfvec(logpr, gpu.loglik_std(om, terms, y, x)), 4, 0)
    with pytest.raises(ValueError, match=r"need a fitted lpdfvec\(logpr_gauss, loglik_gauss\)"):
        posterior_draws(gpu, gpu.loglik_gauss(om, terms, y, x), 4, 0)
    dr = posterior_draws(gpu, vec, 4, 0)
    with pytest.raises(RuntimeError, match="solve has not run"):
        dr.coeff
