"""The hyper-parameter gradients on every path that computes them (OuterBase::gradhyp_dots, ob_engine.hpp):

* the sweep: phi_d_spec (ob_spec.hpp emit_dot in the frame of ob_spec_scaffold.inc) + sum_rows_kernel, option dsweep;
* the reference's own form on the specialised kernels: gradcols_kernel + phi_a_spec (PHI_DOT) + sum_partials_kernel
  per hyper-parameter (dsweep = 0, or a table the sweep declines);
* the augmented interpreter program: phi_a + dot_partials_kernel + sum_partials_kernel per hyper-parameter (spec = 0).

A wrong hyper-gradient makes no fit fail -- BFGS still converges, elsewhere or later -- so each path is held here to a
plain restatement of prodmmge_'s outge (src/linalg.cpp:139-163, 225-277) in long double, evaluated on the GPU's own
basis (outerbase.real) and contracted with the likelihood's row weights:

    outge[:,h] = basescale % sum_{k: t_kl>0} a_k T_k^(-l) % (G_h[:,t_kl] - G_h[:,0] % B_l[:,t_kl]) + G_h[:,0] % yhat,

l = hypmatch[h], T_k^(-l) the product of term k's other factors; the squared operator reads basematsq, basescale^2 and
2 G % B (modandbase.cpp:588-590).  Every hyper-parameter is checked on its own,

    |got_h - want_h| <= 1e-12 * M_h,

M_h = the same sum with every factor replaced by its absolute value and the difference by |G_j| + |G_0| |B_j| -- a
norm-wise check cannot see a wrong entry orders of magnitude below the largest.  Each GPU case also asserts which
path ran, by the launches gradhyp adds to loglik_gauss.update: 2 for the sweep, 3 per hyper-parameter otherwise.

The likelihood builds its basis in the compact layout (levels up to those its table reaches), the restatement reads the
full layout of a second outerbase on the same rows.  The two hold the same bits: the same kernels give the same Phi a
on both (asserted), so the bound needs no allowance for the basis build.
"""
import contextlib

import numpy as np
import pytest

from conftest import make_problem

LD = np.longdouble
TOL = 1e-12
EPS = np.finfo(float).eps
PATHS = {"sweep": (1, 1), "gradcols": (1, 0), "interpreter": (0, 1)}  # (spec, dsweep)
SWEEP_MAX_COLS = 96  # SpecOptions::maxcols_d, ob_spec.hpp


# ------------------------------------------------------------------ the restatement

def basis_of(lib, om, x):
    """The basis a fresh outerbase builds on the rows x, in the reference's full layout."""
    ob = lib.outerbase(om, x)
    return dict(ob=ob, B=ob.real("basemat"), G=ob.real("basemat_gradhyp"), bs=ob.real("basescale"),
                kp=om.index("knotptst"), gest=om.index("gest"), hm=om.index("hypmatch"))


def _chunks(N, K, d):
    step = max(1, (1 << 20) // max(1, K * (d + 1)))
    for r0 in range(0, N, step):
        yield slice(r0, min(N, r0 + step))


def _factors(t, Bt):
    """Per dimension the N x K factor B_l[:, t_kl] (1 where the term skips l); prefix and suffix products over l."""
    K, d = t.shape
    F = [np.where(t[:, l] > 0, Bt[l][:, t[:, l]], LD(1)) for l in range(d)]
    pre, suf = [np.ones((Bt[0].shape[0], K), LD)], [None] * (d + 1)
    for l in range(d):
        pre.append(pre[-1] * F[l])
    suf[d] = np.ones_like(pre[0])
    for l in range(d - 1, -1, -1):
        suf[l] = F[l] * suf[l + 1]
    return pre, suf


def _dims(bas, r, sq):
    """B_l[r, :] per dimension (level 0 included) as long double, squared for the squared operator; and unsquared."""
    kp = bas["kp"]
    raw = [bas["B"][r, kp[l]:kp[l + 1]].astype(LD) for l in range(len(kp) - 1)]
    return ([b * b for b in raw] if sq else raw), raw


def restate(terms, a, bas, sq=False):
    """Per row: yhat = basescale % (Phi a) and outge (N x H) with their magnitudes (|.| of every factor)."""
    t = np.asarray(terms, dtype=np.int64)
    K, d = t.shape
    a = np.asarray(a, dtype=float).astype(LD)
    aa = np.abs(a)
    gest, hm = bas["gest"], bas["hm"]
    H, N = len(hm), bas["B"].shape[0]
    yhat, ymag = np.empty(N, LD), np.empty(N, LD)
    og, ogmag = np.empty((N, H), LD), np.empty((N, H), LD)
    for r in _chunks(N, K, d):
        Bt, Braw = _dims(bas, r, sq)
        sc = bas["bs"][r].astype(LD)
        if sq:
            sc = sc * sc
        pre, suf = _factors(t, Bt)
        phi = pre[d]
        yhat[r] = sc * (phi @ a)
        ymag[r] = np.abs(sc) * (np.abs(phi) @ aa)
        for h in range(H):
            l = int(hm[h])
            m = t[:, l] > 0
            j = t[m, l]
            Gr = bas["G"][r, gest[h]:gest[h + 1]].astype(LD)
            Gj, G0 = Gr[:, j], Gr[:, 0]
            if sq:  # basematsq_gradhyp = 2 G % B, level 0 included
                Gj, G0 = 2 * Gj * Braw[l][:, j], 2 * G0 * Braw[l][:, 0]
            Bj = Bt[l][:, j]
            T = (pre[l] * suf[l + 1])[:, m]
            S = (T * a[m] * (Gj - G0[:, None] * Bj)).sum(axis=1)
            Smag = (np.abs(T) * aa[m] * (np.abs(Gj) + np.abs(G0)[:, None] * np.abs(Bj))).sum(axis=1)
            og[r, h] = sc * S + G0 * yhat[r]
            ogmag[r, h] = np.abs(sc) * Smag + np.abs(G0) * ymag[r]
    return dict(yhat=yhat, ymag=ymag, og=og, ogmag=ogmag)


def restate_t(terms, bas, v, vmag=None, sq=False):
    """Phi^T (basescale % v) (K) and its magnitude |Phi|^T (|basescale| % vmag)."""
    t = np.asarray(terms, dtype=np.int64)
    K, d = t.shape
    v = np.asarray(v).astype(LD)
    vmag = np.abs(v) if vmag is None else np.asarray(vmag).astype(LD)
    out, mag = np.zeros(K, LD), np.zeros(K, LD)
    for r in _chunks(bas["B"].shape[0], K, d):
        Bt, _ = _dims(bas, r, sq)
        sc = bas["bs"][r].astype(LD)
        if sq:
            sc = sc * sc
        phi = _factors(t, Bt)[0][d]
        out += phi.T @ (sc * v[r])
        mag += np.abs(phi).T @ (np.abs(sc) * vmag[r])
    return out, mag


def check(got, want, mag, what):
    got, want, mag = np.asarray(got, dtype=LD), np.asarray(want, dtype=LD), np.asarray(mag, dtype=LD)
    assert got.shape == want.shape, what
    assert np.isfinite(got).all() and np.isfinite(want).all() and np.isfinite(mag).all(), what
    err = np.abs(got - want)
    bad = err > TOL * mag
    assert not bad.any(), (what, int(np.argmax(bad)), float(err[bad].max()), float(mag[bad][np.argmax(err[bad])]))


# ------------------------------------------------------------------ terms tables and models

COVS_ANG = ["mat25ang", "mat25", "mat25pow", "mat25ang", "mat25", "mat25pow", "mat25ang", "mat25"]


def column_table(ncols, d=8):
    """Root, single-dimension terms reaching exactly `ncols` basis columns, and interactions on columns already used."""
    per = [ncols // d + (1 if l < ncols % d else 0) for l in range(d)]
    rows = [np.zeros(d, dtype=np.uint64)]
    for l in range(d):
        for j in range(1, per[l] + 1):
            t = np.zeros(d, dtype=np.uint64); t[l] = j
            rows.append(t)
    for l in range(d - 1):
        t = np.zeros(d, dtype=np.uint64); t[l], t[l + 1] = 1, 2
        rows.append(t)
    for l in range(0, d - 2, 2):
        t = np.zeros(d, dtype=np.uint64); t[l], t[l + 1], t[l + 2] = 2, 1, 1
        rows.append(t)
    return np.asfortranarray(np.array(rows, dtype=np.uint64))


def model(lib, case, N):
    """(om, x, y, terms) of a named case on N rows."""
    if case == "c3":
        import bench
        om, terms = bench.setup_model(lib)
        x = bench.synth_rows(0, N, 10, seed=42)
        y = bench.wingweight(x)
        return om, x, (y - y.mean()) / y.std(ddof=1), terms
    if case == "empty_dim":  # dimension 3 of 9 used by no term: its hyper-parameters see G_h[:,0] * yhat only
        covs = ["mat25pow", "mat25", "mat25ang", "mat25pow", "mat25", "mat25", "mat25pow", "mat25", "mat25"]
        om, x, y, _, _ = make_problem(lib, N, 100, d=9, covs=covs)
        om8 = lib.outermod()
        om8.setcovfs(covs[:3] + covs[4:])
        om8.setknot([np.arange(0.001, 0.999, 0.025)] * 8)
        t8 = om8.selectterms(100)
        terms = np.asfortranarray(np.insert(t8, 3, 0, axis=1))
        return om, x, y, terms
    if case in ("cols96", "cols97"):
        om, x, y, _, _ = make_problem(lib, N, 10)
        return om, x, y, column_table(int(case[4:]))
    kw = {"mat25": dict(covs=["mat25"] * 8), "ang": dict(covs=COVS_ANG), "default": {}, "rootless": {},
          "d32": dict(d=32, covs=["mat25pow"] * 32), "d33pow": dict(d=33, covs=["mat25pow"] * 33),
          "d33": dict(d=33, covs=["mat25"] * 33)}[case]
    K = 100 if case.startswith("d3") else 120
    om, x, y, terms, _ = make_problem(lib, N, K, **kw)
    y = np.where(np.isfinite(y), y, 0.5)  # one row: make_problem's standardisation divides by zero
    if case == "rootless":
        assert not terms[0].any()
        terms = np.asfortranarray(terms[1:])
    return om, x, y, terms


def coefficients(om, terms, seed):
    rng = np.random.default_rng(seed)
    return 3 * np.sqrt(om.getvar(terms)) * rng.normal(size=terms.shape[0])


# ------------------------------------------------------------------ CPU: the restatement and the sweep's limits

@pytest.mark.parametrize("case", ["default", "ang", "empty_dim", "rootless"])
def test_restatement_matches_the_oracle(oracle, case):
    """The long-double restatement against the oracle's prodmmge_ / sqmm_gradhyp, row by row, on the oracle's basis."""
    om, x, y, terms = model(oracle, case, 300)
    bas = basis_of(oracle, om, x)
    a = coefficients(om, terms, 1)
    for sq in (False, True):
        ref = restate(terms, a, bas, sq=sq)
        out = (bas["ob"].sqmm if sq else bas["ob"].matmul)(terms, a)
        outge = (bas["ob"].sqmm_gradhyp if sq else bas["ob"].matmul_gradhyp)(terms, a)
        check(out, ref["yhat"], ref["ymag"], f"{case} sq={sq} yhat")
        check(outge, ref["og"], ref["ogmag"], f"{case} sq={sq} outge")


def test_sweep_generator_limits(product_symbols):
    """The sweep's module exists up to 96 basis columns and 32 dimensions; beyond, the generator declines and the
    engine keeps one product per hyper-parameter."""
    product_symbols.spec_source_dot(column_table(SWEEP_MAX_COLS))
    with pytest.raises(ValueError):
        product_symbols.spec_source_dot(column_table(SWEEP_MAX_COLS + 1))
    for case, ok in (("d32", True), ("d33", False)):
        _, _, _, terms = model(product_symbols, case, 10)
        if ok:
            product_symbols.spec_source_dot(terms)
        else:
            with pytest.raises(ValueError):
                product_symbols.spec_source_dot(terms)


# ------------------------------------------------------------------ GPU

@contextlib.contextmanager
def on_path(gpu, path):
    spec, dsweep = PATHS[path]
    gpu.set_option("spec", spec)
    gpu.set_option("dsweep", dsweep)
    try:
        yield
    finally:
        gpu.set_option("spec", 2)
        gpu.set_option("dsweep", 1)


def gradhyp_launches(gpu, lk, coeff):
    """Launches that compute_gradhyp adds to one update() (the first update compiles and sizes everything)."""
    lk.compute_grad = True
    lk.compute_gradhyp = True
    lk.update(coeff)
    lk.compute_gradhyp = False
    n0 = gpu.launch_count(); lk.update(coeff); n1 = gpu.launch_count()
    lk.compute_gradhyp = True
    lk.update(coeff); n2 = gpu.launch_count()
    return (n2 - n1) - (n1 - n0)


def expect_launches(path, om, terms, swept, ncol=1):
    """The sweep: phi_d_spec + sum_rows_kernel.  Otherwise per hyper-parameter a product and two reductions; on the
    specialised kernels the first is gradcols_kernel, which has nothing to do for a dimension no term uses."""
    if path == "sweep" and swept:
        return 2 * ncol
    hm = om.index("hypmatch")
    idle = 0 if path == "interpreter" else sum(1 for l in hm if not np.asarray(terms)[:, l].any())
    return ncol * (3 * len(hm) - idle)


def run_single(gpu, case, N, path, swept=True):
    om, x, y, terms = model(gpu, case, N)
    H = len(om.index("hypmatch"))
    a = coefficients(om, terms, N)
    bas = basis_of(gpu, om, x)
    with on_path(gpu, path):
        lk = gpu.loglik_gauss(om, terms, y, x)
        lk.updatepara([np.log(0.1)])
        n = gradhyp_launches(gpu, lk, a)
        assert n == expect_launches(path, om, terms, swept), (case, path, n, H)
        yhat, grad, gh = lk.yhat, lk.grad, lk.gradhyp
        ym = bas["ob"].matmul(terms, a)  # the same kernels on the full layout: the two layouts hold the same bits
        np.testing.assert_array_equal(ym, yhat)
    ref = restate(terms, a, bas)
    # the restatement holds the likelihood's basis: Phi a is its yhat, Phi^T w its gradient (loglik_gauss.cpp:110-130)
    check(yhat, ref["yhat"], ref["ymag"], f"{case} N={N} {path} yhat")
    sd = np.exp(lk.para[0])
    w = -(((yhat - y) / sd) / sd)
    g, gmag = restate_t(terms, bas, w)
    check(grad, g, gmag, f"{case} N={N} {path} grad")
    wl = w.astype(LD)
    check(gh, wl @ ref["og"], np.abs(wl) @ ref["ogmag"], f"{case} N={N} {path} gradhyp")


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("N", [1, 63, 64, 65, 127, 128, 129, 255, 257, 60_013])
def test_row_counts(gpu, N, path):
    """Ragged row counts against the 64-row tile (the rw < N weight mask), and 60 013 rows: every CTA works through
    several tiles with three in flight."""
    run_single(gpu, "default", N, path)


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("case,N,swept", [
    ("mat25", 1000, True),       # one hyper-parameter per dimension: the odd branch of the two-at-a-time epilogue
    ("ang", 1000, True),         # mat25ang mixed with mat25pow and mat25
    ("empty_dim", 1000, True),   # OBS_D_DIM_EMPTY
    ("rootless", 1000, True),    # no constant term
    ("cols96", 777, True),       # the sweep's last column count
    ("cols97", 777, False),      # one column more: one product per hyper-parameter
    ("d32", 500, True),          # 32 dimensions, 64 hyper-parameters: the last entries of DotParams' arrays
    ("d33pow", 500, False),      # 66 hyper-parameters
    ("d33", 500, False),         # 33 dimensions, 33 hyper-parameters
    ("c3", 3000, True),          # BASELINE C3's table (d = 10, K = 2000)
])
def test_tables(gpu, case, N, swept, path):
    run_single(gpu, case, N, path, swept)


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["sweep", "gradcols"])
@pytest.mark.parametrize("N", [65, 1000])
def test_marginal_adjustment(gpu, N, path):
    """The squared operator: lpdfvec(logpr_gauss, loglik_gauss)'s marginal adjustment (fit.cpp:259-263, buildhess),
    -0.5 sum_k (dhh_prior[k,h] + dhh_lik[k,h]) / diaghess[k], isolated as gradhyp with domarg minus without."""
    om, x, y, terms = model(gpu, "default", N)
    K, H = terms.shape[0], len(om.index("hypmatch"))
    a = coefficients(om, terms, 5) / 10
    para = [np.log(1.7), np.log(0.1)]
    bas = basis_of(gpu, om, x)
    with on_path(gpu, path):
        vec = gpu.lpdfvec(gpu.logpr_gauss(om, terms), gpu.loglik_gauss(om, terms, y, x))
        vec.compute_gradhyp = True
        vec.updatepara(para)
        vec.update(a)  # compiles the modules, squares the basis
        res = {}
        for dm in (True, False):
            vec.domarg = dm
            vec.updatepara(para)  # the Hessian diagonal and the adjustment are rebuilt at the next update
            n0 = gpu.launch_count()
            vec.update(a)
            res[dm] = (gpu.launch_count() - n0, np.array(vec.gradhyp, dtype=LD))
        dh = vec.diaghess()
    # domarg adds the adjustment's para derivative, whose diaghessgradpara re-reads Phi^2^T 1 (one launch), and the
    # hyper-parameter part: the sweep, or tmm_ge_dev's Phi^2^T 1 and five launches per hyper-parameter
    n = res[True][0] - res[False][0]
    assert n == (1 + 2 if path == "sweep" else 1 + 1 + 5 * H), (path, n, H)
    # the Hessian diagonal the adjustment divides by: prior 1 / (coeffsd sca)^2 plus exp(-2 para) Phi^2^T 1
    s = np.sqrt(om.getvar(terms)).astype(LD) * np.exp(LD(para[0]))
    lsc = np.exp(-2 * LD(para[1]))
    cs, csmag = restate_t(terms, bas, np.ones(N), sq=True)
    check(dh, 1 / s ** 2 + lsc * cs, 1 / s ** 2 + lsc * csmag, f"N={N} {path} diaghess")
    cinv = 1.0 / dh
    dhh0 = -om.getlvar_gradhyp(terms).astype(LD) / (s ** 2)[:, None]
    ref = restate(terms, cinv, bas, sq=True)
    want = -0.5 * (cinv.astype(LD) @ dhh0 + lsc * ref["og"].sum(axis=0))
    mag = 0.5 * (np.abs(cinv).astype(LD) @ np.abs(dhh0) + lsc * ref["ogmag"].sum(axis=0))
    got = res[True][1] - res[False][1]
    # the difference of two rounded sums carries their rounding: eps |gradhyp|
    mag = mag + EPS * (np.abs(res[True][1]) + np.abs(res[False][1])) / TOL
    check(got, want, mag, f"N={N} {path} marginal adjustment")


@pytest.mark.gpu
@pytest.mark.parametrize("path", list(PATHS))
@pytest.mark.parametrize("percol", [False, True])
def test_multi_response(gpu, percol, path):
    """loglik_gauss_multi with C = 3: gradhyp_dots per column on offset coefficient, weight and yhat vectors.  A column
    whose coefficients are zero adds exactly nothing, so each column's gradhyp is read on its own, then all three."""
    N, C = 1000, 3
    om, x, y, terms = model(gpu, "default", N)
    K, H = terms.shape[0], len(om.index("hypmatch"))
    Y = np.column_stack([y, np.sin(3 * x[:, 0]) + 0.3 * y, -0.5 * y + x[:, 1]])
    A = np.column_stack([coefficients(om, terms, 10 + c) for c in range(C)])
    para = [np.log(0.1), np.log(0.2), np.log(0.05)] if percol else [np.log(0.1)]
    sds = np.exp(para) if percol else np.exp(para * C)
    bas = basis_of(gpu, om, x)
    refs = [restate(terms, A[:, c], bas) for c in range(C)]
    with on_path(gpu, path):
        lk = gpu.loglik_gauss_multi(om, terms, Y, x, para_per_column=percol)
        lk.updatepara(para)
        n = gradhyp_launches(gpu, lk, A.ravel(order="F"))
        assert n == expect_launches(path, om, terms, True, ncol=C), (path, n, H)
        for cols in ([0], [1], [2], [0, 1, 2]):
            Ac = np.zeros_like(A)
            Ac[:, cols] = A[:, cols]
            lk.update(Ac.ravel(order="F"))
            gh, grad = lk.gradhyp, lk.grad
            want, mag = np.zeros(H, LD), np.zeros(H, LD)
            for c in range(C):
                ref = refs[c] if c in cols else dict(yhat=np.zeros(N, LD), ymag=np.zeros(N, LD))
                w = -(((ref["yhat"] - Y[:, c]) / sds[c]) / sds[c])
                # the kernel's w comes from its own yhat, within TOL * ymag of the restated one
                wmag = np.abs(w) + TOL * ref["ymag"] / sds[c] ** 2
                g, gmag = restate_t(terms, bas, w, wmag)
                check(grad[:, c], g, gmag, f"{path} percol={percol} cols={cols} grad[:, {c}]")
                if c in cols:
                    want += w @ ref["og"]
                    mag += wmag @ ref["ogmag"]
            check(gh, want, mag, f"{path} percol={percol} cols={cols} gradhyp")
