"""The basis build on the knot layouts obfit produces: every dimension its own knot count (16 to 70 in obfit's second
stage, fitting.py), mixed covariance kinds, with and without hyper-parameter gradients.

launch_basis_build (ob_kernels.cu) picks one of seven kernels per dimension from the knot count m, the columns built
mo and the number of hyper-parameter gradients nh (0 without gradients, 1 for mat25, 2 for mat25pow / mat25ang):
the tensor-core kernel with NT = 1, 2, 3, 5 or 9 column tiles of 8, or the FMA kernel with 64 or 32 rows per CTA.
outerbase.debug_build_geometry reports the choice; these tests assert it per dimension, reach every cell, and hold
each cell's values to the forward-error bound of the contraction, against the oracle and against an 80-bit
restatement of the covariance and the contraction.  The rotation blocks sit inside a max-m-row rotmat, so with
mixed knot counts a leading-dimension mix-up in the kernels shows.
"""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from conftest import relerr

pytestmark = pytest.mark.gpu

REPO = Path(__file__).resolve().parents[1]
EPS = np.finfo(float).eps
BOUNDS = {"mat25": (0.0, 1.0), "mat25pow": (0.0, 1.0), "mat25ang": (0.0, 6.283185)}  # fitting._COV_BOUNDS
KNOTS = {"mat25": (0.01, 0.99), "mat25pow": (0.01, 0.99), "mat25ang": (0.05, 6.0)}
# short length scales: the eigenvalues of 70-100 knots then span e^11 to e^16, and the likelihood comparisons at the
# deep levels stay at the rounding of the fits
HYP = {"mat25": [-1.5], "mat25pow": [-1.5, 0.3], "mat25ang": [-1.0, -1.0]}
NH = {"mat25": 1, "mat25pow": 2, "mat25ang": 2}
MODELS = {  # name: (covariances, knot counts)
    "small": (["mat25", "mat25pow", "mat25ang", "mat25", "mat25pow", "mat25ang"], [2, 3, 8, 9, 17, 25]),
    "mid": (["mat25pow", "mat25", "mat25ang", "mat25pow", "mat25", "mat25ang"], [40, 41, 64, 65, 72, 24]),
    "fma": (["mat25pow", "mat25ang", "mat25pow", "mat25", "mat25", "mat25pow"], [68, 69, 70, 73, 100, 16]),
}

# The dispatch on a B200 (227 KB of opt-in shared memory a block), DESIGN 3.5: the largest knot count of the NT = 9
# tensor-core kernel, of the 64-row FMA kernel and of the 32-row FMA kernel (the ceiling), per nh.
MMA9_MAX = {0: 72, 1: 72, 2: 64}
FMA64_MAX = {0: 137, 1: 89, 2: 68}
CEILING = {0: 152, 1: 102, 2: 80}
SMEM_OPTIN = 227 * 1024


def expected_kernel(m, mo, nh):
    if m <= 72:
        t = next(t for t in (1, 2, 3, 5, 9) if -(-mo // 8) <= t)
        if t < 9 or m <= MMA9_MAX[nh]:
            return ("dmma", t)
    return ("fma", 64 if m <= FMA64_MAX[nh] else 32)


def make_model(lib, name, ms=None):
    covs, m0 = MODELS[name]
    ms = ms or m0
    om = lib.outermod()
    om.setcovfs(covs)
    om.setknot([np.linspace(*KNOTS[c], m) for c, m in zip(covs, ms)])
    om.updatehyp(np.concatenate([HYP[c] for c in covs]))
    return om


def make_x(covs, N, seed=0, edges=True):
    """Uniform rows inside each covariance's bounds; with edges, row 0 and row N-1 at the lower and upper bound, rows 1
    and 2 at the upper and lower bound (the likelihoods and products go without: mat25pow's gradient is NaN at 0)."""
    rng = np.random.default_rng(seed)
    x = np.empty((N, len(covs)), order="F")
    for l, c in enumerate(covs):
        lo, hi = BOUNDS[c]
        x[:, l] = rng.uniform(lo, hi, N)
        if not edges:
            continue
        if N > 3:
            x[1, l], x[2, l] = hi, lo
        x[N - 1, l], x[0, l] = hi, lo
    return x


def check_rows(N):
    """64 rows (all when N <= 64): first and last, both sides of the 64-row tile edges, the rows at the bounds."""
    if N <= 64:
        return np.arange(N)
    must = [i for i in (0, 1, 2, 62, 63, 64, 65, 127, 128, N - 1) if i < N]
    rest = np.setdiff1d(np.arange(N), must)
    pick = np.random.default_rng(N).choice(rest, size=64 - len(must), replace=False)
    return np.sort(np.concatenate([must, pick]))


def basis(ob, dograd):
    out = dict(bm=ob.real("basemat"), sm=ob.real("basescalemat"), bs=ob.real("basescale"))
    if dograd:
        out["bg"] = ob.real("basemat_gradhyp")
    return out


def nan_match(got, want, what):
    """The reference's own NaN (mat25pow's gradient at x = 0: log(0) * 0): the same positions, finite elsewhere."""
    assert np.array_equal(np.isnan(got), np.isnan(want)), what
    assert np.isfinite(want[~np.isnan(want)]).all() and np.isfinite(got[~np.isnan(got)]).all(), what


def within_bound(got, want, bound, what):
    """Componentwise: the contraction's forward-error bound, with NaN where the reference has NaN."""
    nan_match(got, want, what)
    ok = np.isnan(want) | (np.abs(got - want) <= bound)
    assert ok.all(), (what, int(ok.size - ok.sum()), float(np.nanmax(np.abs(got - want) / np.maximum(bound, 1e-300))))


class Bounds:
    """The forward-error bound of test_gpu_parity.test_basis_build per dimension: column j of B_l is a length-m_l
    contraction divided by column 0, judged against gamma * sum_p |cov_p rot_pj| / |P0| (and the same for the
    divisor); the gradient blocks Rt = covg.rot + cov.rotg likewise.  The rotation blocks are the first m_l rows of
    the max-m-row rotmat.  rows: the rows of x to evaluate (C uses the double covariance of the oracle)."""

    def __init__(self, oracle, om, x, rows=None):
        self.om, self.oracle = om, oracle
        self.x = x if rows is None else x[rows]
        self.kp, self.hypst, self.gest = om.index("knotptst"), om.index("hypst"), om.index("gest")
        self.rot, self.rotg, self.kn, self.hyp = om.real("rotmat"), om.real("rotmat_gradhyp"), om.real("knotpt"), om.gethyp()
        self.covs = None

    def dims(self, covs):
        for l, c in enumerate(covs):
            m = int(self.kp[l + 1] - self.kp[l])
            hl = self.hyp[self.hypst[l]:self.hypst[l + 1]]
            kn = self.kn[self.kp[l]:self.kp[l + 1]]
            yield l, c, m, hl, kn, self.rot[:m, self.kp[l]:self.kp[l + 1]]

    def check(self, covs, got, want, what):
        """got / want: dicts of bm (N x M), sm (N x d), bs (N), optionally bg.  When want carries "cov_err" (basis80:
        an exact reference), the double covariance's own evaluation error enters the bound beside the contraction's."""
        sm = want["sm"]
        rel0 = np.zeros(self.x.shape[0])
        for l, c, m, hl, kn, R in self.dims(covs):
            Ca = np.abs(self.oracle.covf_cov(c, hl, self.x[:, l], kn))
            if "cov_err" in want:
                SV, SG = want["cov_err"][l]
            else:  # two double evaluations of the covariance: twice the error of one
                SV, SG = cov_error(c, hl, self.x[:, l], kn)
                SV, SG = 2 * SV, 2 * SG
            P0 = np.abs(sm[:, [l]])
            s0 = 8 * m * EPS * (Ca @ np.abs(R[:, [0]])) + SV @ np.abs(R[:, [0]])
            within_bound(got["sm"][:, l], want["sm"][:, l], s0[:, 0], f"{what} basescalemat dim {l}")
            r0 = s0 / P0
            rel0 += r0[:, 0]
            cols = slice(self.kp[l], self.kp[l + 1])
            bound = (8 * m * EPS * (Ca @ np.abs(R)) + SV @ np.abs(R)) / P0
            within_bound(got["bm"][:, cols], want["bm"][:, cols], bound + np.abs(want["bm"][:, cols]) * r0,
                         f"{what} basemat dim {l} ({c}, m = {m})")
            if "bg" in want:
                Cg = np.abs(self.oracle.covf_cov_gradhyp(c, hl, self.x[:, l], kn))
                for j, h in enumerate(range(self.hypst[l], self.hypst[l + 1])):
                    blk = slice(self.gest[h], self.gest[h] + m)
                    Rg = np.abs(self.rotg[:m, blk])
                    bound = 8 * m * EPS * (np.nan_to_num(Cg[:, :, j]) @ np.abs(R) + Ca @ Rg) + SG[:, :, j] @ np.abs(R) + SV @ Rg
                    within_bound(got["bg"][:, blk], want["bg"][:, blk], bound / P0 + np.abs(np.nan_to_num(want["bg"][:, blk])) * r0,
                                 f"{what} basemat_gradhyp dim {l} ({c}, m = {m}) hyper {j}")
        d = len(covs)
        within_bound(got["bs"], want["bs"], np.abs(want["bs"]) * (rel0 + 2 * d * EPS), f"{what} basescale")


# ---- an 80-bit restatement of cov / cov_gradhyp (ob_kernels.cu cov_transform_dev / cov_pair_dev, covfuncs.cpp) and of
# the contraction divided by column 0 (modandbase.cpp:285-327)
LD = np.longdouble


def _transform(kind, h, x, LD=LD):
    """(t, s) of cov_transform_dev, and the relative error bound of each in double: the rounding of exp / pow / sin /
    cos and of log(x) * t; pow(x, powv) carries powv |log x| times the rounding of powv."""
    x = np.asarray(x, dtype=LD)
    four = np.full(x.shape, 4 * EPS)
    if kind == "mat25":
        return x / np.exp(LD(2) * LD(h[0])), np.zeros_like(x), four, four
    if kind == "mat25pow":
        powv = np.exp(LD(0.25) * LD(h[1]))
        t = np.power(x, powv) / np.exp(LD(2) * LD(h[0]) + LD(0.25) * LD(h[1]))
        with np.errstate(divide="ignore", invalid="ignore"):
            lg = np.log(x)
            et = 4 * EPS * (1 + np.where(x > 0, np.abs(lg) * powv, 0)).astype(float)
            return t, lg * t, et, et + 4 * EPS * (1 + np.where(x > 0, 1 / np.abs(np.where(x == 1, 2, lg)), 0)).astype(float)
    return np.sin(x) / np.exp(LD(2) * LD(h[0])), np.cos(x) / np.exp(LD(2) * LD(h[1])), four, four


def _pair80(kind, h, at, as_, bt, bs):
    LD = at.dtype.type
    with np.errstate(invalid="ignore"):
        if kind == "mat25ang":
            hs, hc = at - bt, as_ - bs
            t = np.sqrt(hs * hs + hc * hc)
            e = np.exp(-t)
            v = (1 + t + t * t / 3) * e
            wv = e * (t + 1)
            return v, np.stack([LD(2) / 3 * hs * hs * wv, LD(2) / 3 * hc * hc * wv], axis=2)
        hh = at - bt
        ah = np.abs(hh)
        e = np.exp(-ah)
        v = (1 + ah + ah * ah / 3) * e
        h2 = hh * (1 + ah) * e
        if kind == "mat25":
            return v, (LD(2) / 3 * hh * h2)[:, :, None]
        powv = np.exp(LD(0.25) * LD(h[1]))
        g1 = (as_ - bs) * (-(LD(0.25) * powv / 3)) * h2 + LD(0.25) / 3 * hh * h2
        return v, np.stack([LD(2) / 3 * hh * h2, g1], axis=2)


def cov80(kind, h, x, knots, LD=LD):
    """N x m covariance and N x m x nh gradient in long double, and the first-order error of evaluating them in double
    from rounded transforms (|d cov / d u| |u| rel_u summed over the four transformed inputs u, by a difference
    quotient).  LD = np.float64 gives the error term alone at double speed."""
    tx, tk = _transform(kind, h, x, LD), _transform(kind, h, knots, LD)
    u = [tx[0][:, None], tx[1][:, None], tk[0][None, :], tk[1][None, :]]
    rel = [tx[2][:, None], tx[3][:, None], tk[2][None, :], tk[3][None, :]]
    V, G = _pair80(kind, h, *u)
    SV, SG = np.zeros(V.shape), np.zeros(G.shape)
    dl = LD(2) ** -24
    for i in range(4):
        w = list(u)
        w[i] = u[i] * (1 + dl)
        V2, G2 = _pair80(kind, h, *w)
        with np.errstate(invalid="ignore"):
            SV += np.nan_to_num((np.abs(V2 - V) / dl).astype(float)) * rel[i]
            SG += np.nan_to_num((np.abs(G2 - G) / dl).astype(float)) * rel[i][:, :, None]
    return V, G, SV, SG


def cov_error(kind, h, x, knots, chunk=4096):
    """cov80's evaluation-error terms alone, in double, row chunk by row chunk."""
    parts = [cov80(kind, h, x[i:i + chunk], knots, np.float64)[2:] for i in range(0, x.shape[0], chunk)]
    return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])


def basis80(om, covs, x, dograd):
    """basemat / basescalemat / basescale / basemat_gradhyp of rows x, the contraction in long double on the double
    rotmat blocks; "cov_err": per dimension the covariance evaluation error of cov80."""
    kp, hypst, gest = om.index("knotptst"), om.index("hypst"), om.index("gest")
    rot, rotg, kn, hyp = om.real("rotmat"), om.real("rotmat_gradhyp"), om.real("knotpt"), om.gethyp()
    N = x.shape[0]
    bm = np.zeros((N, kp[-1]), dtype=LD)
    bg = np.zeros((N, rotg.shape[1]), dtype=LD)
    sm = np.zeros((N, len(covs)), dtype=LD)
    cov_err = []
    for l, c in enumerate(covs):
        m = int(kp[l + 1] - kp[l])
        hl = hyp[hypst[l]:hypst[l + 1]]
        V, G, SV, SG = cov80(c, hl, x[:, l], kn[kp[l]:kp[l + 1]])
        cov_err.append((SV, SG))
        R = rot[:m, kp[l]:kp[l + 1]].astype(LD)
        P = V @ R
        sm[:, l] = P[:, 0]
        bm[:, kp[l]:kp[l + 1]] = P / P[:, [0]]
        if dograd:
            for j, h in enumerate(range(hypst[l], hypst[l + 1])):
                blk = slice(gest[h], gest[h] + m)
                with np.errstate(invalid="ignore"):
                    bg[:, blk] = (G[:, :, j] @ R + V @ rotg[:m, blk].astype(LD)) / P[:, [0]]
    out = dict(bm=bm.astype(float), sm=sm.astype(float), bs=np.prod(sm, axis=1).astype(float), cov_err=cov_err)
    if dograd:
        out["bg"] = bg.astype(float)
    return out


def rows_of(b, rows):
    return {k: v[rows] for k, v in b.items() if k != "cov_err"}


# ------------------------------------------------------------------ dispatch
def test_dispatch_reaches_every_kernel(gpu):
    """The hook's report per dimension on the three models, with and without gradients, against the B200 table of
    DESIGN 3.5; the union reaches all seven kernels, and the FMA kernel both with and without gradients."""
    reached = set()
    for name, (covs, ms) in MODELS.items():
        om = make_model(gpu, name)
        x = make_x(covs, 200)
        for dograd in (True, False):
            geo = gpu.outerbase(om, x, dograd=dograd).debug_build_geometry()
            for l, (c, m) in enumerate(zip(covs, ms)):
                nh = NH[c] if dograd else 0
                fam, tile, mo, smem = geo[l]
                assert (fam, tile) == expected_kernel(m, m, nh), (name, dograd, l, c, m, geo[l])
                assert mo == m and 0 < smem <= SMEM_OPTIN, (name, dograd, l, geo[l])
                reached.add((fam, tile, dograd))
            print(f"{name} dograd={dograd}: " + ", ".join(f"{c}({m}) {g[0]} {g[1]} {g[3]} B" for c, m, g in zip(covs, ms, geo)))
    cells = {(f, t) for f, t, _ in reached}
    assert cells == {("dmma", 1), ("dmma", 2), ("dmma", 3), ("dmma", 5), ("dmma", 9), ("fma", 64), ("fma", 32)}, cells
    assert {g for f, _, g in reached if f == "fma"} == {True, False}


# ------------------------------------------------------------------ values
VALUE_CASES = [(name, N, dograd) for name in MODELS for N in (1, 63, 65, 129) for dograd in (True,)]
VALUE_CASES += [(name, 700, dograd) for name in MODELS for dograd in (True, False)]
VALUE_CASES += [(name, 40_000, dograd) for name in ("mid", "fma") for dograd in (True, False)]  # 3-5 row tiles per CTA


@pytest.mark.parametrize("name,N,dograd", VALUE_CASES)
def test_basis_values(gpu, oracle, name, N, dograd):
    """basemat, basemat_gradhyp, basescalemat and basescale on every row against the oracle within the contraction's
    forward-error bound, and on 64 rows (tile edges, first and last row, x at the covariance bounds) against the 80-bit
    restatement within the same bound."""
    covs, ms = MODELS[name]
    omo, omg = make_model(oracle, name), make_model(gpu, name)
    np.testing.assert_array_equal(omo.real("rotmat"), omg.real("rotmat"))
    x = make_x(covs, N, seed=N)
    obg = gpu.outerbase(omg, x, dograd=dograd)
    got = basis(obg, dograd)
    want = basis(oracle.outerbase(omo, x, dograd=dograd), dograd)
    Bounds(oracle, omo, x).check(covs, got, want, f"{name} N={N} oracle")
    rows = check_rows(N)
    ref = basis80(omo, covs, x[rows], dograd)
    Bounds(oracle, omo, x, rows).check(covs, rows_of(got, rows), ref, f"{name} N={N} 80-bit")
    print(name, N, dograd, [g[:2] for g in obg.debug_build_geometry()])


_FMA_SCRIPT = r'''
import sys, numpy as np
sys.path.insert(0, "tests")
import outerbase_b200 as obp
from test_basis_layouts import MODELS, make_model, make_x, basis
gpu = obp.lib(0)
out = {}
for name in ("small", "mid"):
    covs, ms = MODELS[name]
    om = make_model(gpu, name)
    for dograd in (True, False):
        for N in (129, 700):
            ob = gpu.outerbase(om, make_x(covs, N, seed=N), dograd=dograd)
            geo = ob.debug_build_geometry()
            assert all(g[0] == "fma" for g in geo), geo
            for k, v in basis(ob, dograd).items():
                out[f"{name}_{int(dograd)}_{N}_{k}"] = v
np.savez(sys.argv[1], **out)
print("fma build OK")
'''


def test_fma_kernel_is_the_fallback(gpu, oracle, tmp_path):
    """OB_BUILD=fma (read once per process, so in a subprocess of its own) puts every dimension of the m <= 72 models
    on the FMA kernel; its bases agree with the default run (the tensor-core kernel wherever it fits) within the bound."""
    path = tmp_path / "fma.npz"
    res = subprocess.run([sys.executable, "-c", _FMA_SCRIPT, str(path)], capture_output=True, text=True, timeout=900,
                         cwd=str(REPO), env=dict(os.environ, OB_BUILD="fma"))
    assert res.returncode == 0 and "fma build OK" in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]
    fma = np.load(path)
    for name in ("small", "mid"):
        covs, ms = MODELS[name]
        omg, omo = make_model(gpu, name), make_model(oracle, name)
        for dograd in (True, False):
            for N in (129, 700):
                x = make_x(covs, N, seed=N)
                ob = gpu.outerbase(omg, x, dograd=dograd)
                geo = ob.debug_build_geometry()
                assert [g[:2] for g in geo] == [expected_kernel(m, m, NH[c] if dograd else 0) for c, m in zip(covs, ms)], geo
                got = {k: fma[f"{name}_{int(dograd)}_{N}_{k}"] for k in ("bm", "sm", "bs") + (("bg",) if dograd else ())}
                Bounds(oracle, omo, x).check(covs, got, basis(ob, dograd), f"{name} N={N} dograd={dograd} fma vs dmma")


# ------------------------------------------------------------------ compact layout growth
def _lik_state(lk, vec):
    return dict(val=lk.val, grad=np.array(lk.grad), gradhyp=np.array(lk.gradhyp), dh=lk.diaghess(), dhh=lk.diaghessgradhyp(),
                vval=vec.val, vgrad=np.array(vec.grad), vgradhyp=np.array(vec.gradhyp))


def _check_lik(g, o, what):
    assert abs(g["val"] - o["val"]) <= 1e-8 * abs(o["val"]), what
    assert relerr(g["grad"], o["grad"]) < 1e-8, what
    assert relerr(g["gradhyp"], o["gradhyp"]) < 1e-7, what
    assert relerr(g["dh"], o["dh"]) < 1e-8, what
    assert relerr(g["dhh"], o["dhh"]) < 1e-7, what
    assert abs(g["vval"] - o["vval"]) <= 1e-8 * abs(o["vval"]), what
    assert relerr(g["vgrad"], o["vgrad"]) < 1e-8, what
    assert relerr(g["vgradhyp"], o["vgradhyp"]) < 1e-7, what


def deep_terms(om, K, dims_levels):
    """selectterms(K) plus the single-dimension terms of each (dim, top level) up to that level."""
    t = np.asarray(om.selectterms(K), dtype=np.uint64)
    extra = []
    for l, top in dims_levels:
        for lev in range(1, top + 1):
            row = np.zeros(t.shape[1], dtype=np.uint64)
            row[l] = lev
            extra.append(row)
    t = np.vstack([t] + extra)
    _, first = np.unique(t, axis=0, return_index=True)
    return np.asfortranarray(t[np.sort(first)])


def test_compact_layout_grows_onto_the_fma_kernel(gpu, oracle):
    """loglik_gauss and lpdfvec(logpr_gauss, loglik_gauss) on the FMA model: the 70-knot mat25pow dimension (2) starts
    pruned on the NT = 5 tensor-core kernel (levels to 36: mo = 39), updateterms to a table reaching level 44 (mo = 47)
    moves it to the 32-row FMA kernel, updatehyp rebuilds it there, and the complete layout (getbase of an outerbase) builds all 70 columns on
    it; after each step the likelihood against the oracle at test_gpu_parity's loglik_gauss tolerances."""
    covs, ms = MODELS["fma"]
    N = 3000
    x = make_x(covs, N, seed=5, edges=False)
    y = np.sin(3 * x[:, 0]) + x[:, 2] ** 2 + 0.3 * np.cos(x[:, 1]) + 0.1 * x[:, 4]
    res, geo = {}, []
    for name, lib in (("o", oracle), ("g", gpu)):
        om = make_model(lib, name="fma")
        t_small = deep_terms(om, 40, [(2, 36)])
        t_deep = deep_terms(om, 200, [(2, 44), (4, 30)])
        rng = np.random.default_rng(3)
        c_small, c_deep = (rng.normal(size=t.shape[0]) * np.sqrt(om.getvar(t) / 20) for t in (t_small, t_deep))
        lk = lib.loglik_gauss(om, t_small, y, x)
        pr = lib.logpr_gauss(om, t_small)
        vec = lib.lpdfvec(pr, lk)
        for o in (lk, pr, vec):
            o.compute_gradhyp = True; o.compute_gradpara = True
        steps = []
        lk.update(c_small); vec.update(c_small)
        steps.append(_lik_state(lk, vec))
        if lib is gpu:
            geo.append(lk.debug_build_geometry())
        lk.updateterms(t_deep); pr.updateterms(t_deep)
        lk.update(c_deep); vec.update(c_deep)
        steps.append(_lik_state(lk, vec))
        if lib is gpu:
            geo.append(lk.debug_build_geometry())
        om.updatehyp(om.gethyp() + 0.03)
        lk.updateom(); pr.updateom()
        lk.update(c_deep); vec.update(c_deep)
        steps.append(_lik_state(lk, vec))
        if lib is gpu:
            geo.append(lk.debug_build_geometry())
        ob = lib.outerbase(om, x)
        steps.append(ob.getbase(3))
        if lib is gpu:
            geo.append(ob.debug_build_geometry())
        res[name] = steps
    print("dimension 2 through the steps:", [g[2] for g in geo])
    pruned, deep, rebuilt, complete = (g[2] for g in geo)
    assert pruned[:3] == ("dmma", 5, 39), pruned
    assert deep[:3] == ("fma", 32, 47), deep
    assert rebuilt[:3] == ("fma", 32, 47), rebuilt
    assert complete[:3] == ("fma", 32, 70), complete
    for i, what in enumerate(("pruned", "updateterms", "updatehyp")):
        _check_lik(res["g"][i], res["o"][i], what)
    # getbase: the un-normalised P_2 of the complete layout, the contraction's own bound
    gb, ob_ = res["g"][3], res["o"][3]
    om = make_model(oracle, "fma")
    om.updatehyp(om.gethyp() + 0.03)
    m = 70
    kp, hypst = om.index("knotptst"), om.index("hypst")
    h2, kn2 = om.gethyp()[hypst[2]:hypst[3]], om.real("knotpt")[kp[2]:kp[3]]
    Ca = np.abs(oracle.covf_cov("mat25pow", h2, x[:, 2], kn2))
    R = np.abs(om.real("rotmat")[:m, kp[2]:kp[3]])
    within_bound(gb, ob_, 8 * m * EPS * (Ca @ R) + 2 * cov_error("mat25pow", h2, x[:, 2], kn2)[0] @ R, "getbase(3)")


# ------------------------------------------------------------------ products on mixed layouts
@pytest.mark.parametrize("name", ["mid", "fma"])
def test_products_on_mixed_layouts(gpu, oracle, name):
    """The stateless products on the oracle's basis of a mixed model, with a table whose levels reach m-1 in two
    dimensions (selectterms plus single-dimension terms up to the top level): 1e-12 against the oracle on both kernel
    families."""
    covs, ms = MODELS[name]
    N = 3000
    om = make_model(oracle, name)
    x = make_x(covs, N, seed=9, edges=False)
    ob = oracle.outerbase(om, x)
    bm, bs, bg = ob.real("basemat"), ob.real("basescale"), ob.real("basemat_gradhyp")
    kp, gest, hm = om.index("knotptst"), om.index("gest"), om.index("hypmatch")
    terms = deep_terms(om, 300, [(2, ms[2] - 1), (4, ms[4] - 1)])
    K = terms.shape[0]
    assert terms.max(axis=0)[2] == ms[2] - 1 and terms.max(axis=0)[4] == ms[4] - 1
    rng = np.random.default_rng(11)
    a, r = rng.normal(size=K) / np.sqrt(K), rng.normal(size=N)
    omg = make_model(gpu, name)
    try:
        for spec in (0, 1):
            gpu.set_option("spec", spec)
            what = f"{name} spec={spec}"
            assert relerr(gpu.prodmm(terms, a, bm, bs, kp), oracle.prodmm(terms, a, bm, bs, kp)) < 1e-12, what
            assert relerr(gpu.tprodmm(terms, r, bm, bs, kp), oracle.tprodmm(terms, r, bm, bs, kp)) < 1e-12, what
            for f, v in (("prodmmge", a), ("tprodmmge", r)):
                out, outge = getattr(gpu, f)(terms, v, bm, bs, kp, bg, gest, hm)
                ro, rge = getattr(oracle, f)(terms, v, bm, bs, kp, bg, gest, hm)
                assert relerr(out, ro) < 1e-12, (what, f)
                for h in range(rge.shape[1]):
                    assert relerr(outge[:, h], rge[:, h]) < 1e-12, (what, f, h, relerr(outge[:, h], rge[:, h]))
            for Cn in (8, 64):
                A = np.asfortranarray(rng.normal(size=(K, Cn)) / np.sqrt(K))
                R = np.asfortranarray(rng.normal(size=(N, Cn)))
                assert relerr(gpu.prodmm(terms, A, bm, bs, kp), oracle.prodmm(terms, A, bm, bs, kp)) < 1e-12, (what, Cn)
                assert relerr(gpu.tprodmm(terms, R, bm, bs, kp), oracle.tprodmm(terms, R, bm, bs, kp)) < 1e-12, (what, Cn)
        # the generator takes the deep table: the specialised kernels ran (an object of the library's own, same table)
        obg = gpu.outerbase(omg, x, dograd=False)
        obg.matmul(terms, a)
        assert obg.spec_state(terms) == 1
    finally:
        gpu.set_option("spec", 2)


# ------------------------------------------------------------------ knot ceiling
def _create_fails(lib, fn, *args):
    h = C.c_void_p()
    rc = lib.fn(fn)(*args, C.byref(h))
    msg = lib.fn("last_error")().decode()
    assert rc == 1 and not h.value, (fn, rc, msg)
    return msg


@pytest.mark.parametrize("kind,m,ceiling", [("mat25pow", 81, 80), ("mat25", 103, 102)])
def test_knot_ceiling(gpu, oracle, kind, m, ceiling):
    """With gradients, more knots than the FMA kernel's shared memory holds fail at creation, for outerbase and for
    loglik_gauss, with a library error naming the dimension, its knot count and the ceiling, and no handle; the context
    keeps working, and the same model without gradients builds and matches the oracle."""
    covs = ["mat25", kind, "mat25ang"]
    ms = [20, m, 9]

    def model(lib):
        om = lib.outermod()
        om.setcovfs(covs)
        om.setknot([np.linspace(*KNOTS[c], k) for c, k in zip(covs, ms)])
        om.updatehyp(np.concatenate([HYP[c] for c in covs]))
        return om

    N = 300
    x = make_x(covs, N, seed=1)
    y = np.sin(3 * x[:, 1])
    om = model(gpu)
    xf, yf = np.asfortranarray(x), np.ascontiguousarray(y)
    terms = np.asfortranarray(om.selectterms(20))
    for fn, args in (("outerbase_create", (gpu.ctx, om._h, C.c_void_p(xf.ctypes.data), C.c_uint64(N), C.c_int(1))),
                     ("loglik_gauss_create", (gpu.ctx, om._h, C.c_void_p(terms.ctypes.data), C.c_uint64(terms.shape[0]),
                                              C.c_void_p(yf.ctypes.data), C.c_void_p(xf.ctypes.data), C.c_uint64(N)))):
        msg = _create_fails(gpu, fn, *args)
        assert f"dimension 2 has {m} knots" in msg and f"the {ceiling}" in msg, msg
    with pytest.raises(ValueError, match=f"dimension 2 has {m} knots"):
        gpu.outerbase(om, x)
    obg = gpu.outerbase(om, x, dograd=False)
    geo = obg.debug_build_geometry()
    assert geo[1][:3] == ("fma", 64, m), geo
    omo = model(oracle)
    Bounds(oracle, omo, x).check(covs, basis(obg, False), basis(oracle.outerbase(omo, x, dograd=False), False), f"{kind} {m} knots")
