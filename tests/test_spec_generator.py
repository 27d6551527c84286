"""CPU tests of the kernel generator (outerbase_b200/csrc/ob_spec.hpp): the CUDA source it emits for
a terms table (a) compiles for sm_100a with NVRTC -- no GPU needed -- and (b) computes the right
numbers: the generated statements are lifted out of the source, compiled as HOST C++ with the three
load helpers stubbed, run on one random row and compared with the definition
Phi[n,k] = prod_{l: t_kl>0} B[n, l, t_kl] (src/linalg.cpp:70-75)."""
import ctypes as C
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import make_problem


def _terms(product_symbols, K, d=8):
    om, x, y, terms, rng = make_problem(product_symbols, 50, K, d=d)
    return np.asarray(terms), rng


@pytest.mark.parametrize("K", [1, 7, 120])
def test_generated_source_compiles_for_sm100a(product_symbols, K):
    terms, _ = _terms(product_symbols, K)
    src, info = product_symbols.spec_source(terms)
    assert "phi_a_spec" in src and "phi_t_spec" in src and info["types"] >= 1
    nbytes, seconds = product_symbols.spec_compile_check(src)
    assert nbytes > 10_000


def test_options_and_multicast_variant_compile(product_symbols):
    terms, _ = _terms(product_symbols, 300)
    # ra, qa, tga, cache_a, wt, rt, pt, cache_t, acc_cap [np, mc come from the defaults]
    src, info = product_symbols.spec_source(terms, [2, 2, 2, 16, 8, 2, 2, 8, 32])
    assert info["types"] >= 2 and info["tile_rows_a"] == 128 and info["tile_rows_t"] == 128
    product_symbols.spec_compile_check(src)
    with pytest.raises(ValueError):
        product_symbols.spec_source(terms, [1, 3, 2, 16, 8, 1, 4, 8, 32])  # 96-row tiles do not divide the row padding


def test_tensor_map_variant_layout_and_compile(product_symbols, monkeypatch):
    """Option tmap (22nd field of OB_SPEC_OPTS): Phi a's tile columns are ordered by (dimension, level), so that the levels
    of a dimension -- adjacent columns of the basis matrix -- are one 2-D tensor copy; the run table lists their first
    tile columns; the module compiles for sm_100a."""
    import re
    terms, _ = _terms(product_symbols, 300)
    monkeypatch.setenv("OB_SPEC_OPTS", "1,2,4,80,8,1,4,16,56,4,0,1,8,16,2,3,10,96,232,40,128,1")
    src, info = product_symbols.spec_source(terms)
    assert "#define OBS_TMAP_A 1" in src
    layout = [tuple(int(v) for v in m) for m in re.findall(r"// OBS_LAYOUT_A (\d+) (\d+) (\d+)", src)]
    assert [c for c, _, _ in layout] == list(range(len(layout)))
    assert [(d, l) for _, d, l in layout] == sorted((d, l) for _, d, l in layout)
    runs = [int(v) for v in re.search(r"obs_run_col_a\[\] = \{([\d,]+)\}", src).group(1).split(",")]
    starts = [c for c, d, l in layout if c == 0 or (layout[c - 1][1], layout[c - 1][2] + 1) != (d, l)]
    assert runs == starts + [len(layout)] and int(re.search(r"#define OBS_NRUNS_A (\d+)", src).group(1)) == len(starts)
    product_symbols.spec_compile_check(src)
    monkeypatch.delenv("OB_SPEC_OPTS")
    src0, _ = product_symbols.spec_source(terms)
    assert "#define OBS_TMAP_A 0" in src0


HARNESS = r"""
#include <cmath>
#include <cstdint>
static const double* TILE;
static const double* AS;
static inline double lds(uint32_t a) { return TILE[a / 8]; }
static inline double ldv(uint32_t a) { return TILE[a / 8]; }
template <int OFF> static inline double lda(uint32_t) { return AS[OFF / 8]; }
template <int OFF> static inline void lda2(uint32_t, double& x, double& y) { x = AS[OFF / 8]; y = AS[OFF / 8 + 1]; }
using std::fma;
extern "C" void run_a(const double* tile, const double* as_, double* out) {
  TILE = tile; AS = as_;
  const uint32_t tp = 0, as = 0; (void)as;
  double o[1] = {0.0};
  {
%(body_a)s
  }
  out[0] = o[0];
}
%(cases_t)s
"""
CASE_T = r"""
extern "C" void run_t_%(g)d(const double* tile, double bval, double* accs) {
  TILE = tile;
  const uint32_t tp = 0;
  double b[1] = {bval};
%(decl)s
  {
%(body)s
  }
%(store)s
}
"""


def test_generated_statements_compute_phi(product_symbols, tmp_path):
    K, d = 160, 8
    terms, rng = _terms(product_symbols, K, d)
    opts = [1, 4, 2, 12, 3, 1, 4, 6, 32]  # small streams: several CTA types, cached and uncached columns both occur
    src, info = product_symbols.spec_source(terms, opts)
    TRA, TRT = info["tile_rows_a"], info["tile_rows_t"]
    lay_a = [tuple(map(int, m)) for m in re.findall(r"// OBS_LAYOUT_A (\d+) (\d+) (\d+)", src)]
    slot_a = [tuple(map(int, m)) for m in re.findall(r"// OBS_SLOT_A (\d+) (-?\d+)", src)]
    lay_t = [tuple(map(int, m)) for m in re.findall(r"// OBS_LAYOUT_T (\d+) (\d+) (\d+) (\d+)", src)]
    streams = {int(g): (int(t), [int(v) for v in rest.split()]) for g, t, rest in re.findall(r"// OBS_STREAM_T (\d+) type (\d+) terms([ \d-]*)", src)}
    body_a = re.search(r"/\*BEGIN_BODY_A\*/(.*?)/\*END_BODY_A\*/", src, re.S).group(1)
    cases = {int(g): body for g, body in re.findall(r"/\*BEGIN_CASE_T (\d+)\*/(.*?)/\*END_CASE_T\*/", src, re.S)}
    assert len(cases) == len(streams) == info["types"] * opts[4]
    nacc = info["nacc"]
    cases_src = ""
    for g, body in cases.items():
        decl = "\n".join(f"  double acc{i} = 0.0;" for i in range(nacc))
        store = "\n".join(f"  accs[{i}] = acc{i};" for i in range(nacc))
        cases_src += CASE_T % dict(g=g, decl=decl, body=body, store=store)
    cpp = tmp_path / "harness.cpp"
    cpp.write_text(HARNESS % dict(body_a=body_a, cases_t=cases_src))
    so = tmp_path / "harness.so"
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), str(cpp)], check=True)
    lib = C.CDLL(str(so))
    # one random row of basis values B[dim][level] (level 0 unused) and its Phi row by the definition
    L = int(terms.max()) + 1
    B = rng.uniform(0.5, 1.5, size=(d, L))
    phi = np.array([np.prod([B[l, terms[k, l]] for l in range(d) if terms[k, l] > 0]) for k in range(K)])
    a = rng.normal(size=K)
    # --- Phi a
    tile = np.zeros((len(lay_a) + 1) * TRA)
    for pos, dim, lev in lay_a:
        tile[pos * TRA] = B[dim, lev]
    coef = np.array([a[t] if t >= 0 else 0.0 for _, t in sorted(slot_a)])
    out = np.zeros(1)
    lib.run_a(tile.ctypes.data_as(C.c_void_p), coef.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    assert abs(out[0] - phi @ a) <= 1e-12 * np.abs(phi * a).sum()
    # --- Phi^T: every stream's accumulators against b * Phi[k]
    bval = 0.37
    seen = []
    for g, (t, tlist) in streams.items():
        cols = [(pos, dim, lev) for (tt, pos, dim, lev) in lay_t if tt == t]
        tile = np.zeros((len(cols) + 2) * TRT)
        for pos, dim, lev in cols:
            tile[pos * TRT] = B[dim, lev]
        accs = np.zeros(nacc)
        getattr(lib, f"run_t_{g}")(tile.ctypes.data_as(C.c_void_p), C.c_double(bval), accs.ctypes.data_as(C.c_void_p))
        for i, k in enumerate(tlist):
            assert abs(accs[i] - bval * phi[k]) <= 1e-13 * abs(bval * phi[k]), (g, i, k)
        seen += tlist
    assert sorted(seen) == list(range(K))  # every term is owned by exactly one stream


HARNESS_M = r"""
#include <cstdint>
static const double* TILE;
static double PHI[64];
static double* OUT;
static inline double ldv(uint32_t a) { return TILE[a / 8]; }
#define OBS_NBLK %(nblk)d
#define OBS_M_EMIT(slot, value) PHI[slot] = (value)
#define OBS_M_BLOCK() { for (int i = 0; i < %(kc)d; ++i) { OUT[blk * %(kc)d + i] = PHI[i]; PHI[i] = -1.0; } }
extern "C" void run_m(const double* tile, double* out) {
  TILE = tile; OUT = out;
  const uint32_t tp = 0;
  {
%(body)s
  }
}
"""


@pytest.mark.parametrize("K,d", [(160, 8), (700, 10)])
def test_generated_multi_rhs_emits_compute_phi(product_symbols, tmp_path, K, d):
    """The forward program of phi_am_spec (blocks of KC emits with their basis-column loads hoisted to the top of the block,
    ob_spec.hpp emit_mat): executed on the host for one random row, every emit slot holds Phi[row, term of the slot]
    when its block is contracted, padding slots hold 0."""
    terms, rng = _terms(product_symbols, K, d)
    src, (nblk, tile_rows) = product_symbols.spec_source_mat(terms)
    kc = int(re.search(r"#define OBS_KC (\d+)", src).group(1))
    lay = [tuple(map(int, m)) for m in re.findall(r"// OBS_LAYOUT_M (\d+) (\d+) (\d+)", src)]
    slots = [t for _, t in sorted(tuple(map(int, m)) for m in re.findall(r"// OBS_SLOT_M (\d+) (-?\d+)", src))]
    body = re.search(r"/\*BEGIN_BODY_M\*/(.*?)/\*END_BODY_M\*/", src, re.S).group(1)
    assert body.count("OBS_M_BLOCK()") == 1  # ONE shared instance of the contraction
    cpp = tmp_path / "harness_m.cpp"
    cpp.write_text(HARNESS_M % dict(nblk=nblk, kc=kc, body=body))
    so = tmp_path / "harness_m.so"
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), str(cpp)], check=True)
    lib = C.CDLL(str(so))
    L = int(terms.max()) + 1
    B = rng.uniform(0.5, 1.5, size=(d, L))
    phi = np.array([np.prod([B[l, terms[k, l]] for l in range(d) if terms[k, l] > 0]) for k in range(K)])
    tile = np.zeros((len(lay) + 1) * tile_rows)
    for pos, dim, lev in lay:
        tile[pos * tile_rows] = B[dim, lev]
    out = np.full(nblk * kc, np.nan)
    lib.run_m(tile.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p))
    real = [t for t in slots if t >= 0]
    assert sorted(real) == list(range(K)) and len(slots) <= nblk * kc
    for i in range(nblk * kc):
        t = slots[i] if i < len(slots) else -1
        want = phi[t] if t >= 0 else 0.0
        assert abs(out[i] - want) <= 1e-13 * max(abs(want), 1.0), (i, t)


HARNESS_TM = r"""
#include <cstdint>
static const double* TILE;
static double* PHI;
static inline double lds(uint32_t a) { return TILE[a / 8]; }
static inline double ldv(uint32_t a) { return TILE[a / 8]; }
#define OBS_TM_PARK(slot, value) PHI[slot] = (value)
%(cases)s
"""
CASE_TM = r"""
extern "C" void run_tm_%(g)d(const double* tile, double bval, double* phi) {
  TILE = tile; PHI = phi;
  const uint32_t tp = 0;
  double b[1] = {bval};
  {
%(body)s
  }
}
"""


def test_generated_transposed_multi_rhs_parks_compute_phi(product_symbols, tmp_path):
    """The streams of phi_tm_spec (forward program with every emit parked, ob_spec.hpp emit_fwd park = true): executed on
    the host for one random row, stream g parks basescale * Phi[row, term] for its terms in order; every term belongs to
    exactly one stream of at most 32."""
    K, d = 300, 8
    terms, rng = _terms(product_symbols, K, d)
    src, info = product_symbols.spec_source_tmat(terms)
    streams = {int(g): (int(t), [int(v) for v in rest.split()]) for g, t, rest in re.findall(r"// OBS_STREAM_TM (\d+) type (\d+) terms([ \d-]*)", src)}
    lay = [tuple(map(int, m)) for m in re.findall(r"// OBS_LAYOUT_TM (\d+) (\d+) (\d+) (\d+)", src)]
    cases = {int(g): body for g, body in re.findall(r"/\*BEGIN_CASE_TM (\d+)\*/(.*?)/\*END_CASE_TM\*/", src, re.S)}
    assert len(cases) == len(streams) == info["types"] * 8
    cpp = tmp_path / "harness_tm.cpp"
    cpp.write_text(HARNESS_TM % dict(cases="".join(CASE_TM % dict(g=g, body=body) for g, body in cases.items())))
    so = tmp_path / "harness_tm.so"
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-o", str(so), str(cpp)], check=True)
    lib = C.CDLL(str(so))
    L = int(terms.max()) + 1
    B = rng.uniform(0.5, 1.5, size=(d, L))
    phi = np.array([np.prod([B[l, terms[k, l]] for l in range(d) if terms[k, l] > 0]) for k in range(K)])
    TR, bval, seen = 64, 0.41, []
    for g, (t, tlist) in streams.items():
        assert len(tlist) <= 32
        cols = [(pos, dim, lev) for (tt, pos, dim, lev) in lay if tt == t]
        tile = np.zeros((len(cols) + 2) * TR)
        for pos, dim, lev in cols:
            tile[pos * TR] = B[dim, lev]
        out = np.full(32, np.nan)
        getattr(lib, f"run_tm_{g}")(tile.ctypes.data_as(C.c_void_p), C.c_double(bval), out.ctypes.data_as(C.c_void_p))
        for i, k in enumerate(tlist):
            assert abs(out[i] - bval * phi[k]) <= 1e-13 * abs(bval * phi[k]), (g, i, k)
        seen += tlist
    assert sorted(seen) == list(range(K))


HARNESS_D = r"""
#include <cmath>
#include <cstddef>
#include <cstdint>
static const double* TILE;
static const double* AS;
static inline double lds(uint32_t a) { return TILE[a / 8]; }
static inline double ldv(uint32_t a) { return TILE[a / 8]; }
template <int OFF> static inline double lda(uint32_t) { return AS[OFF / 8]; }
template <int OFF> static inline void lda2(uint32_t, double& x, double& y) { x = AS[OFF / 8]; y = AS[OFF / 8 + 1]; }
using std::fma;
static inline void hyp_add(double* dst, double v, int) { *dst += v; }
struct DotParams { const double* gmat; const double* bmat; unsigned long long ld; int hst[33]; int gest[65]; int kst[33]; };
static struct { int ntiles = 1; } p;
%(macros)s
extern "C" void run_d(const double* tile, const double* as_, const double* gmat, const double* bmat, const int* hst, int nd,
                      const int* gest, int nh, const int* kst, double wv, double* hs, double* uroot_out) {
  TILE = tile; AS = as_;
  DotParams q{};
  q.gmat = gmat; q.bmat = bmat; q.ld = 1;
  for (int i = 0; i <= nd; ++i) { q.hst[i] = hst[i]; q.kst[i] = kst[i]; }
  for (int i = 0; i <= nh; ++i) q.gest[i] = gest[i];
  const uint32_t tp = 0, as = 0; (void)as;
  const int lane = 0; const unsigned long long rw = 0;
  {
%(body)s
  uroot_out[0] = uroot;
  }
}
"""


_SWEEP_CASES = [(160, 8, False, 2, True), (160, 8, True, 2, True), (160, 8, False, 1, True), (160, 8, True, 3, True),
                (2000, 10, False, 2, True), (120, 32, False, 2, True), (160, 8, False, 2, False)]


@pytest.mark.parametrize("K,d,unused_dim,nh,root", _SWEEP_CASES,
                         ids=["-".join(map(str, c[:4])) + ("" if c[4] else "-rootless") for c in _SWEEP_CASES])
def test_generated_hyper_gradient_sweep(product_symbols, tmp_path, K, d, unused_dim, nh, root):
    """phi_d_spec's generated body + epilogue macros (lifted to host C++) against the definition of prodmmge_'s outge
    (src/linalg.cpp:139-163, 273-276) for one row, plain and squared (basematsq_gradhyp = 2 G % B, modandbase.cpp:588-590);
    2000 x 10 has the size of BASELINE config C3's table, 32 dimensions with two hyper-parameters each fill DotParams'
    fixed arrays (hst[33], gest[65], kst[33]) to the last entry, and `root = False` drops the constant term."""
    terms, rng = _terms(product_symbols, K, d)
    if not root:
        assert not terms[0].any()
        terms = np.asfortranarray(terms[1:])
        K -= 1
    if unused_dim:  # a dimension no term uses: its hyper-parameters still see G_h[:,0] * yhat
        terms = np.asfortranarray(np.hstack([terms, np.zeros((K, 1), dtype=terms.dtype)]))
        d += 1
    src, info = product_symbols.spec_source_dot(terms)
    assert "phi_d_spec" in src and info["slots"] == K
    product_symbols.spec_compile_check(src)  # the real thing builds for sm_100a
    TR = info["tile_rows"]
    lay = [tuple(map(int, m)) for m in re.findall(r"// OBS_LAYOUT_D (\d+) (\d+) (\d+)", src)]
    slots = [tuple(map(int, m)) for m in re.findall(r"// OBS_SLOT_D (\d+) (-?\d+)", src)]
    body = re.search(r"/\*BEGIN_BODY_D\*/(.*?)/\*END_BODY_D\*/", src, re.S).group(1)
    macros = re.search(r"(#define OBS_D_HYP_BEGIN.*?)__device__ __forceinline__ void hyp_add", src, re.S).group(1)
    cpp = tmp_path / "harness_d.cpp"
    cpp.write_text(HARNESS_D % dict(macros=macros, body=body))
    so = tmp_path / "harness_d.so"
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off", "-Wno-unknown-pragmas", "-o", str(so), str(cpp)], check=True)
    lib = C.CDLL(str(so))
    L = int(terms.max()) + 1
    # nh hyper-parameters per dimension (mat25pow: 2, mat25: 1); the epilogue takes them two at a time
    B = rng.uniform(0.5, 1.5, size=(d, L)); B[:, 0] = 1.0
    G = rng.normal(size=(d * nh, L))  # G[h, j] = stored gradient column j of hyper h (level 0 included)
    a = rng.normal(size=K)
    T = np.array([np.prod([B[l, terms[k, l]] for l in range(d) if terms[k, l] > 0]) for k in range(K)])
    hst = np.arange(0, nh * (d + 1), nh, dtype=np.int32)
    gest = np.arange(0, L * (d * nh + 1), L, dtype=np.int32)
    kst = np.arange(0, L * (d + 1), L, dtype=np.int32)
    coef = np.zeros(K)
    for i, t in slots:
        coef[i] = a[t]
    wv = 0.83
    ptr = lambda v: v.ctypes.data_as(C.c_void_p)
    for squared in (False, True):
        Bt = B ** 2 if squared else B
        Gt = 2 * G * np.repeat(B, nh, axis=0) if squared else G  # 2 G % B, level 0: B = 1
        Tt = T ** 2 if squared else T
        tile = np.zeros((len(lay) + 1) * TR)
        for pos, dim, lev in lay:
            tile[pos * TR] = Bt[dim, lev]
        want = np.zeros(d * nh)
        for h in range(d * nh):
            l = h // nh
            j = terms[:, l].astype(int)
            m = j > 0
            s = np.sum(a[m] * Tt[m] / Bt[l, j[m]] * (Gt[h, j[m]] - Gt[h, 0] * Bt[l, j[m]]))
            want[h] = wv * (s + Gt[h, 0] * (Tt @ a))
        hs = np.zeros(d * nh); uroot = np.zeros(1)
        gflat = np.ascontiguousarray(G.ravel()); bflat = np.ascontiguousarray(B.ravel())
        lib.run_d(ptr(tile), ptr(coef), ptr(gflat), ptr(bflat) if squared else None, ptr(hst), C.c_int(d), ptr(gest), C.c_int(d * nh),
                  ptr(kst), C.c_double(wv), ptr(hs), ptr(uroot))
        assert abs(uroot[0] - Tt @ a) <= 1e-12 * np.abs(Tt * a).sum()
        scale = np.abs(want).max()
        assert np.abs(hs - want).max() <= 1e-11 * scale, (squared, np.abs(hs - want).max(), scale)


def test_hyper_gradient_sweep_refuses_tables_with_too_many_columns(product_symbols):
    """The derivative accumulators live in registers: beyond 96 basis columns the generator declines and the engine
    keeps one product per hyper-parameter (launch_phi_d_spec returns false)."""
    d, L = 8, 14  # 8 x 13 = 104 columns
    rows = [np.zeros(d, dtype=np.uint64)]
    for l in range(d):
        for j in range(1, L):
            t = np.zeros(d, dtype=np.uint64); t[l] = j
            rows.append(t)
    terms = np.asfortranarray(np.array(rows, dtype=np.uint64))
    with pytest.raises(ValueError):
        product_symbols.spec_source_dot(terms)
    product_symbols.spec_source(terms)  # the plain kernels have no such limit
