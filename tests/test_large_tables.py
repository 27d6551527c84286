"""Phi and loglik_gauss on large terms tables and on tables the trie compiler refuses.

The interpreter Phi kernels choose their layout from the size of the table (phi_geometry, ob_kernels.cu): two tile
buffers with the program in shared memory, one buffer, the program left in global memory, and when nothing fits in
shared memory -- or the table has a duplicate row or a term deeper than the interpreter's stack -- the brute-force
kernels.  Here every one of those layouts runs on bench.py's C3 model (d = 10) at N = 3000 rows, and the layout each
table reaches is read back from the library (outerbase.debug_phi_geometry) and asserted, so that a threshold change
fails loudly instead of moving coverage.  At N = 3000 the kernels always use two rows per lane (R = 2); the smaller
inputs of the likelihood keep the CPU oracle's CG affordable at K = 20 000.

Products go through the stateless seam on the oracle's bit-identical basis (interpreter kernels, spec = 0); the
likelihood objects build their own basis on the GPU and are held to test_gpu_parity.py's tolerances.
"""
import numpy as np
import pytest

from conftest import relerr
from multiresponse_reference import Reference
from test_gpu_configs import GE_NORM_TOL, check
from test_multiresponse import responses

N, D = 3000, 10
EPS = np.finfo(float).eps
TWO, ONE, GLOBAL, BRUTE = "two buffers", "one buffer", "program in global memory", "brute force"
# the layout (Phi a, Phi^T) each K reaches on the C3 model at N = 3000 rows, as the library reports it on a B200
LARGE = {2000: (TWO, TWO), 9000: (ONE, ONE), 13000: (GLOBAL, GLOBAL), 16000: (BRUTE, GLOBAL), 20000: (BRUTE, BRUTE)}
NONTRIE = ("duplicate", "duplicate_intercept", "depth9", "depth8")
NONTRIE_LAYOUT = {"duplicate": (BRUTE, BRUTE), "duplicate_intercept": (BRUTE, BRUTE), "depth9": (BRUTE, BRUTE),
                  "depth8": (TWO, TWO)}
TABLES = list(LARGE) + list(NONTRIE)


def layout(g):
    if g["R"] == 0:
        return BRUTE
    if g["nbuf"] == 2:
        return TWO
    return ONE if g["prog_in_smem"] else GLOBAL


@pytest.fixture(scope="module")
def c3(oracle):
    """the oracle side: C3's model, N rows, the basis, and the tables (built once per module)"""
    import bench
    x = bench.synth_rows(0, N, D)
    y = bench.wingweight(x)
    y = (y - y.mean()) / y.std(ddof=1)
    omo, _ = bench.setup_model(oracle, K=300)
    ob = oracle.outerbase(omo, x)
    return dict(x=x, y=y, omo=omo, ob=ob, bm=ob.real("basemat"), bs=ob.real("basescale"), bg=ob.real("basemat_gradhyp"),
                kp=omo.index("knotptst"), gest=omo.index("gest"), hm=omo.index("hypmatch"), tables={})


@pytest.fixture(scope="module")
def c3g(c3, gpu):
    """the GPU side: the same model and an outerbase object on the same rows"""
    import bench
    omg, _ = bench.setup_model(gpu, K=300)
    return dict(omg=omg, obg=gpu.outerbase(omg, c3["x"]))


def table(c3, name):
    """K rows of selectterms, or C3's K = 300 table with one row the trie compiler cannot take"""
    if name not in c3["tables"]:
        om = c3["omo"]
        if isinstance(name, int):
            t = om.selectterms(name)
        else:
            base = om.selectterms(300)
            assert not base[0].any()  # row 0 is the intercept
            row = np.zeros((1, D), dtype=np.uint64)
            if name == "duplicate":
                row = base[5:6]
            elif name == "duplicate_intercept":
                row = base[0:1]
            else:
                row[0, :int(name[-1])] = 1
                assert not (base == row).all(1).any()
            t = np.asfortranarray(np.vstack([base, row]))
        c3["tables"][name] = t
    return c3["tables"][name]


@pytest.fixture
def spec(gpu):
    def set_spec(mode):
        gpu.set_option("spec", mode)
    yield set_spec
    gpu.set_option("spec", 2)
    gpu.set_option("spec_work", 4e12)
    gpu.set_option("device_cg", 1)


@pytest.mark.gpu
def test_layouts_cover_every_variant(c3, c3g, gpu):
    """every layout of both interpreter kernels, and the brute-force kernels, is reached by one of the tables below"""
    seen = set()
    for name in TABLES:
        t = table(c3, name)
        got = tuple(layout(c3g["obg"].debug_phi_geometry(t, transpose=tr)) for tr in (False, True))
        print(f"K = {t.shape[0]} ({name}): Phi a {got[0]}, Phi^T {got[1]}")
        want = LARGE[name] if name in LARGE else NONTRIE_LAYOUT[name]
        assert got == want, (name, got, want)
        seen.add(got)
    for need in ((TWO, TWO), (ONE, ONE), (GLOBAL, GLOBAL), (BRUTE, GLOBAL), (BRUTE, BRUTE)):
        assert need in seen, need


def test_depth8_term_mixes_trie_and_brute_force_programs(c3, product_symbols):
    """a term with 8 active dimensions fits the plain program; the hyper-gradient program of a dimension that term does
    not use adds one level and is refused, that of a dimension it uses is not"""
    t = table(c3, "depth8")
    kp = c3["kp"]
    ones = np.ones(int(kp[-1]))
    fast = {l: product_symbols.debug_terms_eval(t, kp, ones, np.ones(t.shape[0]), aug_dim=l, gcols0=ones)[2]["fast_ok"]
            for l in (0, 7, 8, 9)}
    assert product_symbols.debug_terms_eval(t, kp, ones, np.ones(t.shape[0]))[2]["fast_ok"] == 1
    assert fast == {0: 1, 7: 1, 8: 0, 9: 0}, fast


def phi_rows_longdouble(c3, terms, rows):
    """Phi[rows, :] = basescale * prod over the active dimensions of the basis columns, in 80-bit arithmetic"""
    bm = c3["bm"][rows].astype(np.longdouble)
    P = np.repeat(c3["bs"][rows].astype(np.longdouble)[:, None], terms.shape[0], axis=1)
    kp = c3["kp"]
    for l in range(D):
        lv = terms[:, l].astype(np.int64)
        on = lv > 0
        P[:, on] *= bm[:, kp[l] + lv[on]]
    return P


@pytest.mark.gpu
@pytest.mark.parametrize("name", TABLES)
def test_products_against_the_oracle(c3, c3g, gpu, oracle, spec, name):
    """prodmm_ / tprodmm_, the squared operators, prodmmge_ / tprodmmge_ on the interpreter kernels or the brute-force
    fallback: against the oracle, against an 80-bit evaluation on 64 rows, and bit for bit against a second call"""
    spec(0)
    terms = table(c3, name)
    K = terms.shape[0]
    bm, bs, kp, bg, gest, hm = c3["bm"], c3["bs"], c3["kp"], c3["bg"], c3["gest"], c3["hm"]
    abm, abs_ = np.abs(bm), np.abs(bs)
    rng = np.random.default_rng(17)
    a = np.sqrt(c3["omo"].getvar(terms) / 20) * rng.normal(size=K)
    r = rng.normal(size=N)
    runs = {}
    for sq, (B, S) in enumerate(((bm, bs), (bm * bm, bs * bs))):
        got = gpu.prodmm(terms, a, B, S, kp)
        check(got, oracle.prodmm(terms, a, B, S, kp), oracle.prodmm(terms, np.abs(a), np.abs(B), np.abs(S), kp), what=(name, sq, "prodmm"))
        runs[f"mm{sq}"] = got
        got = gpu.tprodmm(terms, r, B, S, kp)
        check(got, oracle.tprodmm(terms, r, B, S, kp), oracle.tprodmm(terms, np.abs(r), np.abs(B), np.abs(S), kp), what=(name, sq, "tprodmm"))
        runs[f"tmm{sq}"] = got
    a2 = rng.normal(size=K) / 100
    out, outge = gpu.prodmmge(terms, a2, bm, bs, kp, bg, gest, hm)
    ro, rge = oracle.prodmmge(terms, a2, bm, bs, kp, bg, gest, hm)
    check(out, ro, oracle.prodmm(terms, np.abs(a2), abm, abs_, kp), what=(name, "prodmmge"))
    for h in range(rge.shape[1]):
        assert relerr(outge[:, h], rge[:, h]) < GE_NORM_TOL, (name, "prodmmge", h)
    runs["mmge"] = (out, outge)
    out, outge = gpu.tprodmmge(terms, r, bm, bs, kp, bg, gest, hm)
    ro, rge = oracle.tprodmmge(terms, r, bm, bs, kp, bg, gest, hm)
    check(out, ro, oracle.tprodmm(terms, np.abs(r), abm, abs_, kp), what=(name, "tprodmmge"))
    for h in range(rge.shape[1]):
        assert relerr(outge[:, h], rge[:, h]) < GE_NORM_TOL, (name, "tprodmmge", h)
    runs["tmmge"] = (out, outge)

    # a plain 80-bit reference on 64 seeded rows: Phi a there, and Phi^T r for an r supported on those rows only.  The
    # brute-force Phi a adds the K terms one after another, as the oracle does (about 16 eps of the magnitude at K = 20 000)
    rows = np.sort(rng.choice(N, 64, replace=False))
    P = phi_rows_longdouble(c3, terms, rows)
    want = P @ a.astype(np.longdouble)
    mag = np.abs(P) @ np.abs(a).astype(np.longdouble)
    err = np.abs(runs["mm0"][rows].astype(np.longdouble) - want) / mag
    assert err.max() <= 32 * EPS, (name, "Phi a", float(err.max()) / EPS)
    rs = np.zeros(N)
    rs[rows] = rng.normal(size=64)
    got = gpu.tprodmm(terms, rs, bm, bs, kp)
    want = P.T @ rs[rows].astype(np.longdouble)
    mag = np.abs(P.T) @ np.abs(rs[rows]).astype(np.longdouble)
    err = np.abs(got.astype(np.longdouble) - want) / np.maximum(mag, np.finfo(float).tiny)
    assert err.max() <= 32 * EPS, (name, "Phi^T r", float(err.max()) / EPS)

    # the same call twice gives the same bits, the brute-force Phi^T included
    for sq, (B, S) in enumerate(((bm, bs), (bm * bm, bs * bs))):
        np.testing.assert_array_equal(gpu.prodmm(terms, a, B, S, kp), runs[f"mm{sq}"])
        np.testing.assert_array_equal(gpu.tprodmm(terms, r, B, S, kp), runs[f"tmm{sq}"])
    for key, got in (("mmge", gpu.prodmmge(terms, a2, bm, bs, kp, bg, gest, hm)), ("tmmge", gpu.tprodmmge(terms, r, bm, bs, kp, bg, gest, hm))):
        np.testing.assert_array_equal(got[0], runs[key][0])
        np.testing.assert_array_equal(got[1], runs[key][1])


@pytest.mark.gpu
def test_object_squared_operators(c3, c3g, gpu, oracle, spec):
    """sqmm / sqtmm of the device-resident object (the kernel squares the basis columns as it loads them) on the
    brute-force fallback, against the oracle's products on the object's own basis, squared on the host"""
    spec(0)
    terms = table(c3, 20000)
    obg, kp = c3g["obg"], c3["kp"]
    rng = np.random.default_rng(5)
    a = np.sqrt(c3["omo"].getvar(terms) / 20) * rng.normal(size=terms.shape[0])
    r = rng.normal(size=N)
    assert layout(obg.debug_phi_geometry(terms, sq=1)) == BRUTE
    B2, S2 = obg.real("basemat") ** 2, obg.real("basescale") ** 2
    check(obg.sqmm(terms, a), oracle.prodmm(terms, a, B2, S2, kp), oracle.prodmm(terms, np.abs(a), B2, S2, kp), what="sqmm")
    first = obg.sqtmm(terms, r)
    check(first, oracle.tprodmm(terms, r, B2, S2, kp), oracle.tprodmm(terms, np.abs(r), B2, S2, kp), what="sqtmm")
    np.testing.assert_array_equal(obg.sqtmm(terms, r), first)


# ---- loglik_gauss

LIK_TABLES = [2000, 9000, 13000, 16000, 20000] + list(NONTRIE)
_ORACLE = {}
XNEW = np.asfortranarray(np.random.default_rng(23).uniform(size=(333, D)))


def _lik_inputs(c3, name):
    terms = table(c3, name)
    rng = np.random.default_rng(29)
    coeff = np.sqrt(c3["omo"].getvar(terms) / 20) * rng.normal(size=terms.shape[0])
    return terms, coeff, rng.normal(size=terms.shape[0])


def _update_side(lib, om, c3, terms, coeff, g):
    lk = lib.loglik_gauss(om, terms, c3["y"], c3["x"])
    lk.compute_gradhyp = True; lk.compute_gradpara = True
    lk.updatepara([np.log(0.1)])
    lk.update(coeff)
    return dict(val=lk.val, grad=lk.grad, gradhyp=lk.gradhyp, gradpara=lk.gradpara, yhat=lk.yhat, hm=lk.hessmult(g),
                dh=lk.diaghess(), dhh=lk.diaghessgradhyp())


def _fit_side(lib, om, c3, terms):
    lk = lib.loglik_gauss(om, terms, c3["y"], c3["x"])
    vec = lib.lpdfvec(lib.logpr_gauss(om, terms), lk)
    vec.domarg = True
    return lk, vec


# On the tables of 9000 terms and more (K > N) the oracle's CG stops at the 100-iteration cap without meeting the
# tolerance.  Such an iterate depends on the rounding of every step, and the device loop adds its K-vector sums in
# another order than the oracle: after 100 steps two correct runs were measured 3e-6 apart in val (K = 9000, B200).  Those
# fits are compared after CAPPED_EPOCHS steps, before the rounding differences have grown to 1e-8.
CAPPED_EPOCHS = 30


def _fit(vec, K, epochs=100):
    vec.set_coeff(np.zeros(K))
    vec.optcg(0.001, epochs)
    return dict(coeff=vec.coeff, val=vec.val, iters=vec.cg_iters, epochs=epochs)


def oracle_lik(c3, oracle, name):
    if name not in _ORACLE:
        terms, coeff, g = _lik_inputs(c3, name)
        res = _update_side(oracle, c3["omo"], c3, terms, coeff, g)
        lk, vec = _fit_side(oracle, c3["omo"], c3, terms)
        res["fit"] = _fit(vec, terms.shape[0])
        if res["fit"]["iters"] == 100:
            res["fit"] = _fit(vec, terms.shape[0], CAPPED_EPOCHS)
        pr = oracle.predictor(lk)
        pr.update(XNEW)
        res["mean"], res["var"] = pr.mean(), pr.var()
        _ORACLE[name] = res
    return _ORACLE[name]


def check_update(got, want, name):
    assert abs(got["val"] - want["val"]) <= 1e-8 * abs(want["val"]), name
    assert relerr(got["grad"], want["grad"]) < 1e-8, name
    assert relerr(got["gradhyp"], want["gradhyp"]) < 1e-7, name
    assert relerr(got["gradpara"], want["gradpara"]) < 1e-8, name
    assert relerr(got["yhat"], want["yhat"]) < 1e-9, name
    assert relerr(got["hm"], want["hm"]) < 1e-8, name
    assert relerr(got["dh"], want["dh"]) < 1e-8, name
    # the squared operator's hyper-gradient on two independently built bases: 1.3e-7 measured at K = 20 000 (B200), the
    # high-level basis columns' gradients carry the build's rounding; the same product on one basis agrees to 1e-11
    assert relerr(got["dhh"], want["dhh"]) < 2e-7, name


def check_fit(got, want, name):
    assert got["iters"] == want["iters"], (name, got["iters"], want["iters"])
    assert abs(got["val"] - want["val"]) <= 1e-8 * abs(want["val"]), name
    assert relerr(got["coeff"], want["coeff"]) < 1e-8, name


@pytest.mark.gpu
@pytest.mark.parametrize("name", LIK_TABLES)
def test_loglik_gauss_against_the_oracle(c3, c3g, gpu, oracle, spec, name):
    """loglik_gauss update / hessmult / diaghess / diaghessgradhyp, optcg on lpdfvec(logpr_gauss, loglik_gauss) with the
    device-resident and the host CG loop, and the predictor, on the interpreter kernels or the brute-force fallback"""
    spec(0)
    want = oracle_lik(c3, oracle, name)
    terms, coeff, g = _lik_inputs(c3, name)
    K = terms.shape[0]
    check_update(_update_side(gpu, c3g["omg"], c3, terms, coeff, g), want, name)
    lk, vec = _fit_side(gpu, c3g["omg"], c3, terms)
    fits = {}
    for dcg in (1, 0):
        gpu.set_option("device_cg", dcg)
        fits[dcg] = _fit(vec, K, want["fit"]["epochs"])
        check_fit(fits[dcg], want["fit"], (name, dcg))
    gpu.set_option("device_cg", 1)
    again = _fit(vec, K, want["fit"]["epochs"])  # a second fit from zero: the same bits
    np.testing.assert_array_equal(again["coeff"], fits[1]["coeff"])
    assert again["iters"] == fits[1]["iters"] and again["val"] == fits[1]["val"]
    pr = gpu.predictor(lk)
    pr.update(XNEW)
    assert relerr(pr.mean(), want["mean"]) < 1e-7
    assert relerr(pr.var(), want["var"]) < 1e-7


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [1, 2])
def test_loglik_gauss_fallback_under_the_spec_policies(c3, c3g, gpu, oracle, spec, mode):
    """K = 16 000 (brute-force Phi a) with specialisation at first use, and under the automatic policy with a threshold
    that is crossed partway through the CG: whichever kernels serve the table, the fit is the oracle's"""
    name = 16000
    want = oracle_lik(c3, oracle, name)
    terms, coeff, g = _lik_inputs(c3, name)
    K = terms.shape[0]
    spec(mode)
    if mode == 2:
        # a CG iteration runs four products of N x K row-terms: the table turns hot in the third iteration
        assert want["fit"]["iters"] > 4
        gpu.set_option("spec_work", 10.0 * N * K)
    lk, vec = _fit_side(gpu, c3g["omg"], c3, terms)
    check_fit(_fit(vec, K, want["fit"]["epochs"]), want["fit"], (name, mode))
    if mode == 1:
        c3g["obg"].matmul(terms, coeff)
        state = c3g["obg"].spec_state(terms)
        print(f"K = {K}, spec = 1: spec_state {state} ({'specialised' if state == 1 else 'refused: interpreter / brute force'})")
        assert state in (1, -1)
    check_update(_update_side(gpu, c3g["omg"], c3, terms, coeff, g), want, (name, mode))


# ---- multi-response

@pytest.mark.gpu
@pytest.mark.parametrize("C", [3, 8])
def test_multi_response_on_a_duplicate_row_table(c3, c3g, gpu, oracle, spec, C):
    """loglik_gauss_multi builds its residuals after plain products, so it runs on the brute-force kernels too"""
    spec(0)
    terms = table(c3, "duplicate")
    K = terms.shape[0]
    Y = responses(c3["x"], c3["y"], C)
    ref = Reference(oracle)
    rv = ref.lpdfvec(ref.logpr_gauss_multi(c3["omo"], terms, C), ref.loglik_gauss_multi(c3["omo"], terms, Y, c3["x"]))
    rv.domarg = True
    rv.optcg(0.001, 100)
    vec = gpu.lpdfvec(gpu.logpr_gauss_multi(c3g["omg"], terms, C), gpu.loglik_gauss_multi(c3g["omg"], terms, Y, c3["x"]))
    vec.domarg = True
    vec.optcg(0.001, 100)
    np.testing.assert_array_equal(vec.cg_iters_per_column, rv.cg_iters_per_column)
    for c in range(C):
        assert relerr(vec.coeff[:, c], rv.coeff[:, c]) < 1e-8, c
    assert abs(vec.val - rv.val) <= 1e-8 * abs(rv.val)
    first, iters = vec.coeff.copy(), vec.cg_iters_per_column
    vec.set_coeff(np.zeros(K * C))
    vec.optcg(0.001, 100)
    np.testing.assert_array_equal(vec.coeff, first)
    np.testing.assert_array_equal(vec.cg_iters_per_column, iters)
