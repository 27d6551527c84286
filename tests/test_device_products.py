"""The device-pointer products of the C ABI -- ob_outerbase_set_terms, then mm_dev / tmm_dev / mm_mat_dev / tmm_mat_dev on
the caller's torch buffers, the calls bench.py times -- element-wise against the CPU oracle.

Reference: the oracle's stateless seam (prodmm_ / tprodmm_) on the basis read back from the object under test, so both
sides read the same bits; the squared operators on bm**2 and bs**2 (the library squares each stored entry; x*x is
correctly rounded on both sides).  Bound: check() of test_gpu_configs.py, |got - want| <= ELEM_TOL * (|Phi| |a|) per
entry plus the norm-wise 1e-12.

Caller buffers are not the library's padded layout: the ABI passes N rows and leading dimension N, the specialised
Phi^T stages whole row tiles and decides per call whether to read past N in place, to copy into a padded buffer or to
realign (OuterBase::phi_t, launch_phi_tm_spec).  Every input here has NaN after its last entry, every output starts as
a fixed NaN bit pattern: entries past the result keep their bits, every result entry is finite and correct.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import REPO, make_problem, relerr
from test_gpu_configs import ELEM_TOL, check

NAN_BITS = 0x7FF8_0000_DEAD_BEEF   # a quiet NaN with a payload: an entry still holding it was never written
TAIL = 512                         # NaN entries after each input / sentinels after each output: more than a row tile
K8 = 300                           # terms of the d = 8 make_problem tables
VEC_ROWS = [1, 63, 64, 65, 127, 128, 129, 255, 256, 257, 1000]
MAT_ROWS = [1, 65, 255, 256, 777, 4097]
MAT_COLS = [1, 7, 8, 9, 63, 64, 65, 128, 129]
LAYOUTS = ["padded", "poisoned", "misaligned"]


def ceil256(n):
    return ((n + 255) // 256) * 256


class OracleRef:
    """Oracle products on the basis read back from `ob` (bit-identical inputs); (want, magnitude) pairs."""

    def __init__(self, oracle, ob, om, terms):
        self.oracle, self.terms = oracle, terms
        self.kp = om.index("knotptst")
        self.bm, self.bs = ob.real("basemat"), ob.real("basescale")
        self._sq = None

    def _basis(self, sq):
        """(basis, |basis|) of the plain or the squared operator"""
        if not sq:
            return (self.bm, self.bs), (np.abs(self.bm), np.abs(self.bs))
        if self._sq is None:
            self._sq = (self.bm ** 2, self.bs ** 2)
        return self._sq, self._sq

    def mm(self, a, sq):
        (bm, bs), (abm, abs_) = self._basis(sq)
        return (self.oracle.prodmm(self.terms, a, bm, bs, self.kp), self.oracle.prodmm(self.terms, np.abs(a), abm, abs_, self.kp))

    def tmm(self, r, sq):
        (bm, bs), (abm, abs_) = self._basis(sq)
        return (self.oracle.tprodmm(self.terms, r, bm, bs, self.kp), self.oracle.tprodmm(self.terms, np.abs(r), abm, abs_, self.kp))


def nan_buffer(n):
    import torch
    return torch.full((n,), NAN_BITS, dtype=torch.int64, device="cuda").view(torch.float64)


def kept(buf, lo):
    """Entries [lo, end) of buf still hold the NaN pattern."""
    import torch
    return bool((buf.view(torch.int64)[lo:] == NAN_BITS).all())


def device_input(src, layout):
    """src (flat float64) on the device in a caller layout: `padded` exactly its length, `poisoned` followed by NaN,
    `misaligned` at an odd element offset (8- but not 16-byte aligned) and followed by NaN."""
    import torch
    src = torch.from_numpy(np.ascontiguousarray(src, dtype=np.float64).ravel(order="K"))
    if layout == "padded":
        return src.cuda()
    off = 1 if layout == "misaligned" else 0
    buf = nan_buffer(off + src.numel() + TAIL)
    v = buf[off:off + src.numel()]
    v.copy_(src)
    if layout == "misaligned":
        assert v.data_ptr() % 16 == 8
    return v


def device_output(n, layout, padded_len=None):
    """A NaN-filled output of at least n entries: the view the product writes, and the whole buffer."""
    if layout == "padded":
        buf = nan_buffer(padded_len if padded_len is not None else n + TAIL)
        return buf, buf
    off = 1 if layout == "misaligned" else 0
    buf = nan_buffer(off + n + TAIL)
    return buf[off:], buf


@pytest.fixture(params=[0, 1], ids=["interpreter", "specialised"])
def family(gpu, request):
    gpu.set_option("spec", request.param)
    yield request.param
    gpu.set_option("spec", 2)


@pytest.fixture()
def lib_stream(gpu):
    """torch work on the library's stream, as in bench.py."""
    import torch
    with torch.cuda.stream(torch.cuda.ExternalStream(gpu.stream())):
        yield gpu


_OBJ = {}


def d8_object(gpu, oracle, N, K=K8):
    """A d = 8 make_problem table on N rows: GPU object with its terms installed, oracle reference on its basis."""
    key = ("d8", N, K)
    if key not in _OBJ:
        om, x, _, terms, rng = make_problem(gpu, N, K)
        ob = gpu.outerbase(om, x, dograd=False)
        ob.set_terms(terms)
        ob.sqmm(terms, np.ones(K))  # materialise basematsq up front: launch counts below are the products' own
        _OBJ[key] = dict(om=om, ob=ob, terms=terms, ref=OracleRef(oracle, ob, om, terms), rng=rng, cache={})
    return _OBJ[key]


def c3_object(gpu, oracle, N):
    """bench.setup_model's C3 table (d = 10, K = 2000) on bench.synth_rows(0, N)."""
    import bench
    key = ("c3", N)
    if key not in _OBJ:
        for k in [k for k in _OBJ if k[0] == "c3"]:
            del _OBJ[k]  # one C3 basis resident at a time
        om, terms = bench.setup_model(gpu)
        ob = gpu.outerbase(om, bench.synth_rows(0, N, bench.D), dograd=False)
        ob.set_terms(terms)
        ob.sqmm(terms, np.ones(terms.shape[0]))
        ref = OracleRef(oracle, ob, om, terms) if oracle is not None else None
        _OBJ[key] = dict(om=om, ob=ob, terms=terms, ref=ref, rng=np.random.default_rng(N), cache={})
    return _OBJ[key]


def vector_products(lib, o, N, layouts=LAYOUTS, sqs=(0, 1), what=""):
    """mm_dev / tmm_dev in each caller layout against the oracle; entries past the result keep their NaN bits."""
    ob, ref, terms = o["ob"], o["ref"], o["terms"]
    K = terms.shape[0]
    if "vec" not in o["cache"]:
        rng = o["rng"]
        a = np.sqrt(o["om"].getvar(terms) / 20) * rng.normal(size=K)
        r = rng.normal(size=N)
        o["cache"]["vec"] = (a, r, {sq: (ref.mm(a, sq), ref.tmm(r, sq)) for sq in sqs})
    a, r, want = o["cache"]["vec"]
    for sq in sqs:
        (ya, ym), (ta, tm) = want[sq]
        for layout in layouts:
            tag = f"{what} N={N} sq={sq} {layout}"
            ad, rd = device_input(a, layout), device_input(r, layout)
            y, ybuf = device_output(N, layout, padded_len=ceil256(N))  # bench's yhat: padded to 256 rows
            g, gbuf = device_output(K, layout)
            ob.mm_dev(ad.data_ptr(), y.data_ptr(), sq)
            ob.tmm_dev(rd.data_ptr(), g.data_ptr(), sq)
            lib.synchronize()
            assert kept(y, N), tag + ": Phi a wrote past row N"
            assert kept(g, K), tag + ": Phi^T wrote past term K"
            yv, gv = y[:N].cpu().numpy(), g[:K].cpu().numpy()
            assert np.isfinite(yv).all() and np.isfinite(gv).all(), tag
            check(yv, ya, ym, what=tag + " mm_dev")
            check(gv, ta, tm, what=tag + " tmm_dev")


@pytest.mark.gpu
@pytest.mark.parametrize("N", VEC_ROWS)
def test_vector_products_in_caller_buffers(lib_stream, oracle, family, N):
    """mm_dev / tmm_dev, sq 0 and 1, on bench's layout (output padded to 256 rows, input exactly N), an input followed
    by NaN, and views at an odd element offset.  At N = 256 the caller's rows are the library's: nothing is staged."""
    vector_products(lib_stream, d8_object(lib_stream, oracle, N), N, what=f"d8 family={family}")


@pytest.mark.gpu
def test_vector_products_c3_table(lib_stream, oracle, family):
    N = 20_000
    vector_products(lib_stream, c3_object(lib_stream, oracle, N), N, what=f"c3 family={family}")


def matrix_products(lib, o, N, cols, family, what=""):
    """mm_mat_dev / tmm_mat_dev (leading dimension N, NaN after the inputs, NaN-filled outputs) and the host forms
    matmul / tmatmul / sqmm / sqtmmm with 2-D operands, against the oracle; routing asserted through launch counts."""
    ob, ref, terms = o["ob"], o["ref"], o["terms"]
    K = terms.shape[0]
    Cmax = max(cols)
    key = ("mat", Cmax)
    if key not in o["cache"]:
        rng = o["rng"]
        A = np.asfortranarray(rng.normal(size=(K, Cmax)) * np.sqrt(o["om"].getvar(terms) / 20)[:, None])
        R = np.asfortranarray(rng.normal(size=(N, Cmax)))
        o["cache"][key] = (A, R, {sq: (ref.mm(A, sq), ref.tmm(R, sq)) for sq in (0, 1)})
    A, R, want = o["cache"][key]
    for C in cols:
        counts = {}
        for sq in (0, 1):
            (ya, ym), (ta, tm) = want[sq]
            ya, ym, ta, tm = ya[:, :C], ym[:, :C], ta[:, :C], tm[:, :C]
            tag = f"{what} N={N} C={C} sq={sq}"
            Ad, Rd = device_input(A[:, :C].ravel(order="F"), "poisoned"), device_input(R[:, :C].ravel(order="F"), "poisoned")
            Y, G = nan_buffer(N * C + TAIL), nan_buffer(K * C + TAIL)
            lib.synchronize()
            n0 = lib.launch_count()
            ob.mm_mat_dev(Ad.data_ptr(), C, Y.data_ptr(), sq)
            n1 = lib.launch_count()
            ob.tmm_mat_dev(Rd.data_ptr(), C, G.data_ptr(), sq)
            counts[sq] = (n1 - n0, lib.launch_count() - n1)
            lib.synchronize()
            assert kept(Y, N * C) and kept(G, K * C), tag + ": wrote past the result"
            yv = Y[:N * C].cpu().numpy().reshape((N, C), order="F")
            gv = G[:K * C].cpu().numpy().reshape((K, C), order="F")
            assert np.isfinite(yv).all() and np.isfinite(gv).all(), tag
            check(yv, ya, ym, what=tag + " mm_mat_dev")
            check(gv, ta, tm, what=tag + " tmm_mat_dev")
            check(ob.sqmm(terms, A[:, :C]) if sq else ob.matmul(terms, A[:, :C]), ya, ym, what=tag + " host Phi A")
            check(ob.sqtmmm(terms, R[:, :C]) if sq else ob.tmatmul(terms, R[:, :C]), ta, tm, what=tag + " host Phi^T A")
        nmm, ntm = counts[0]
        chunks = (C + 63) // 64
        if family == 1 and C >= 8:  # tensor cores: gather + phi_am_spec / (pad copy +) phi_tm_spec + reduce per 64 columns
            assert 1 <= nmm <= 2 * chunks and 2 <= ntm <= 3 * chunks, (what, N, C, counts)
        else:  # the column loop over the vector kernels
            assert nmm >= C and ntm >= C, (what, N, C, counts)
        assert counts[1] == counts[0], (what, N, C, "squared operators read basematsq: same route", counts)


@pytest.mark.gpu
@pytest.mark.parametrize("N", MAT_ROWS)
def test_matrix_products_around_the_tensor_core_switch(lib_stream, oracle, family, N):
    """C around the switch to the tensor cores (8) and around the 64-column chunks, sq 0 and 1."""
    matrix_products(lib_stream, d8_object(lib_stream, oracle, N), N, MAT_COLS, family, what=f"d8 family={family}")


@pytest.mark.gpu
def test_matrix_products_c3_table(lib_stream, oracle, family):
    N = 20_000
    matrix_products(lib_stream, c3_object(lib_stream, oracle, N), N, [129], family, what=f"c3 family={family}")


@pytest.mark.gpu
def test_dev_calls_need_set_terms(lib_stream, oracle, family):
    """A fresh object refuses every *_dev call and terms_stats until set_terms, and enqueues nothing; after set_terms of
    another table the device forms give the host forms' bits on that table; terms_stats describes the installed table."""
    import bench
    N = 777
    om, x, _, terms, rng = make_problem(lib_stream, N, K8)
    ob = lib_stream.outerbase(om, x, dograd=False)
    a, r = device_input(rng.normal(size=K8), "padded"), device_input(rng.normal(size=N), "padded")
    out = nan_buffer(N * 9 + TAIL)
    for call in (lambda: ob.mm_dev(a.data_ptr(), out.data_ptr()), lambda: ob.tmm_dev(r.data_ptr(), out.data_ptr()),
                 lambda: ob.mm_mat_dev(a.data_ptr(), 1, out.data_ptr()), lambda: ob.tmm_mat_dev(r.data_ptr(), 1, out.data_ptr()),
                 ob.terms_stats):
        with pytest.raises(RuntimeError, match="set_terms"):
            call()
    lib_stream.synchronize()
    assert kept(out, 0)
    ob.set_terms(terms)
    t2 = np.asfortranarray(om.selectterms(120)[::-1])  # another table (fewer terms, other order)
    ob.set_terms(t2)
    K2 = t2.shape[0]
    W, Lcols = bench.term_stats(t2)
    st = ob.terms_stats()
    assert (st["W"], st["Lcols"], st["maxdepth"]) == (W, Lcols, int((t2 > 0).sum(1).max())), st
    a2, A2, R2 = rng.normal(size=K2), np.asfortranarray(rng.normal(size=(K2, 9))), np.asfortranarray(rng.normal(size=(N, 9)))
    for sq in (0, 1):
        host_mm = ob.sqmm if sq else ob.matmul
        host_tm = ob.sqtmmm if sq else ob.tmatmul
        y, g = nan_buffer(N + TAIL), nan_buffer(K2 + TAIL)
        Y, G = nan_buffer(N * 9 + TAIL), nan_buffer(K2 * 9 + TAIL)
        ad, rd, Ad, Rd = (device_input(v.ravel(order="F"), "poisoned") for v in (a2, r.cpu().numpy(), A2, R2))
        ob.mm_dev(ad.data_ptr(), y.data_ptr(), sq)
        ob.tmm_dev(rd.data_ptr(), g.data_ptr(), sq)
        ob.mm_mat_dev(Ad.data_ptr(), 9, Y.data_ptr(), sq)
        ob.tmm_mat_dev(Rd.data_ptr(), 9, G.data_ptr(), sq)
        lib_stream.synchronize()
        assert kept(y, N) and kept(g, K2) and kept(Y, 9 * N) and kept(G, 9 * K2)
        np.testing.assert_array_equal(y[:N].cpu().numpy(), host_mm(t2, a2))
        np.testing.assert_array_equal(g[:K2].cpu().numpy(), host_tm(t2, r.cpu().numpy()))
        np.testing.assert_array_equal(Y[:9 * N].cpu().numpy().reshape((N, 9), order="F"), host_mm(t2, A2))
        np.testing.assert_array_equal(G[:9 * K2].cpu().numpy().reshape((K2, 9), order="F"), host_tm(t2, R2))


def test_matmul_refuses_a_matrix_without_one_row_per_term(oracle):
    """outerbase._mm with a 2-D `a` checks its rows against the terms, as the 1-D form and _tmm do (the binding would
    otherwise upload K x C doubles from a smaller array)."""
    om, x, _, terms, rng = make_problem(oracle, 50, 20)
    ob = oracle.outerbase(om, x)
    for bad in (rng.normal(size=(19, 3)), rng.normal(size=(21, 3)), rng.normal(size=(3, 20))):
        with pytest.raises(ValueError, match="one row per term"):
            ob.matmul(terms, bad)
        with pytest.raises(ValueError, match="one row per term"):
            ob.sqmm(terms, bad)
    assert ob.matmul(terms, rng.normal(size=(20, 3))).shape == (50, 3)


def _run(script, env_extra, *args):
    env = dict(os.environ, **env_extra)
    res = subprocess.run([sys.executable, "-c", script, *map(str, args)], capture_output=True, text=True, env=env,
                         timeout=900, cwd=str(REPO))
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    return res.stdout


_FUSE_SCRIPT = r'''
import sys, numpy as np, torch
sys.path.insert(0, "tests")
from conftest import make_problem
import outerbase_b200 as obp
gpu = obp.lib(0)
gpu.set_option("spec", 1)
N, K = 5000, 300
om, x, y, terms, rng = make_problem(gpu, N, K)
ob = gpu.outerbase(om, x, dograd=False)
ob.set_terms(terms)
r = rng.normal(size=N)
with torch.cuda.stream(torch.cuda.ExternalStream(gpu.stream())):
    rd = torch.from_numpy(r).cuda()
    g = torch.empty(K, dtype=torch.float64, device="cuda")
    ob.tmm_dev(rd.data_ptr(), g.data_ptr())  # compiles the module
    gpu.synchronize()
    n0 = gpu.launch_count()
    ob.tmm_dev(rd.data_ptr(), g.data_ptr())
    gpu.synchronize()
    per_tmm = gpu.launch_count() - n0
    t_dev = g.cpu().numpy()
t_host = ob.tmatmul(terms, r)
lik = gpu.loglik_gauss(om, terms, y, x)
lik.compute_gradhyp = True
lik.update(rng.normal(size=K) / 100)
vec = gpu.lpdfvec(gpu.logpr_gauss(om, terms), gpu.loglik_gauss(om, terms, y, x))
vec.optcg(0.001, 100)
np.savez(sys.argv[1], per_tmm=per_tmm, t_dev=t_dev, t_host=t_host, r=r, terms=terms, bm=ob.real("basemat"),
         bs=ob.real("basescale"), kp=om.index("knotptst"), val=lik.val, grad=lik.grad, gradhyp=lik.gradhyp,
         fval=vec.val, fcoeff=vec.coeff, fgradhyp=vec.gradhyp, iters=vec.cg_iters)
'''


@pytest.mark.gpu
def test_unfused_phi_t_reduction(oracle, tmp_path):
    """OB_FUSE_TAIL=0 -- also what a refused cooperative launch falls back to: phi_t_spec ends without its cross-CTA tail
    and phi_t_reduce_kernel adds the per-CTA partial sums, and loglik_gauss sums its squared residuals in a kernel of
    its own instead of riding on the Phi^T launch.  Both reductions add in the same order as the fused tail (CTA
    partials in row-group order j = 0 .. J-1, a sequential sum from 0.0), so every product, the likelihood with its
    gradients and the CG fit carry the fused run's bits; the extra launch per Phi^T shows the path was taken."""
    runs = {}
    for name, env in (("fused", {}), ("unfused", {"OB_FUSE_TAIL": "0"})):
        _run(_FUSE_SCRIPT, env, tmp_path / f"{name}.npz")
        runs[name] = np.load(tmp_path / f"{name}.npz")
    f, u = runs["fused"], runs["unfused"]
    assert int(u["per_tmm"]) == int(f["per_tmm"]) + 1, (int(f["per_tmm"]), int(u["per_tmm"]))
    want = oracle.tprodmm(u["terms"], u["r"], u["bm"], u["bs"], u["kp"])
    mag = oracle.tprodmm(u["terms"], np.abs(u["r"]), np.abs(u["bm"]), np.abs(u["bs"]), u["kp"])
    check(u["t_dev"], want, mag, what="unfused tmm_dev")
    check(u["t_host"], want, mag, what="unfused tmatmul")
    for k in ("bm", "t_dev", "t_host", "val", "grad", "gradhyp", "fval", "fcoeff", "fgradhyp", "iters"):
        np.testing.assert_array_equal(u[k], f[k], err_msg=k)


_END_SCRIPT = r'''
import ctypes, sys, numpy as np, torch
sys.path.insert(0, "tests")
from conftest import make_problem, ORACLE_LIB
from outerbase_b200.binding import Library
import outerbase_b200 as obp
from test_device_products import OracleRef, nan_buffer, kept, TAIL, K8
from test_gpu_configs import check
cu = ctypes.CDLL("libcuda.so.1")
def address_range(p):
    base, size = ctypes.c_ulonglong(0), ctypes.c_size_t(0)
    rc = cu.cuMemGetAddressRange_v2(ctypes.byref(base), ctypes.byref(size), ctypes.c_ulonglong(p))
    return rc, base.value, size.value
def at_allocation_end(src):
    """src on the device in a buffer that ends exactly where its allocation ends: torch.empty(n) is its own cudaMalloc
    here; when the driver reports the allocation rounded up, a buffer of the reported size is allocated instead and
    src placed at its end"""
    n = src.size
    buf = torch.empty(n, dtype=torch.float64, device="cuda")
    rc, base, size = address_range(buf.data_ptr())
    assert rc == 0 and base == buf.data_ptr() and size >= 8 * n, (n, rc, base, size)
    exact = size == 8 * n
    if not exact:
        buf = torch.empty(size // 8, dtype=torch.float64, device="cuda")
        rc, base, size2 = address_range(buf.data_ptr())
        assert rc == 0 and base == buf.data_ptr() and size2 == size, (n, rc, base, size, size2)
    v = buf[buf.numel() - n:]
    v.copy_(torch.from_numpy(src))
    assert v.data_ptr() + 8 * n == base + size
    return v, exact
gpu = obp.lib(0)
oracle = Library(ORACLE_LIB, "orc_")
for spec in (0, 1):
    gpu.set_option("spec", spec)
    for N in (64, 200, 257, 1000, 4097):
        om, x, _, terms, rng = make_problem(gpu, N, K8)
        ob = gpu.outerbase(om, x, dograd=False)
        ob.set_terms(terms)
        ref = OracleRef(oracle, ob, om, terms)
        r = rng.normal(size=N)
        R = np.asfortranarray(rng.normal(size=(N, 9)))
        with torch.cuda.stream(torch.cuda.ExternalStream(gpu.stream())):
            rd, exact = at_allocation_end(r)
            Rd, _ = at_allocation_end(R.ravel(order="F"))
            for sq in (0, 1):
                g, G = nan_buffer(K8 + TAIL), nan_buffer(9 * K8 + TAIL)
                ob.tmm_dev(rd.data_ptr(), g.data_ptr(), sq)
                ob.tmm_mat_dev(Rd.data_ptr(), 9, G.data_ptr(), sq)
                gpu.synchronize()
                assert kept(g, K8) and kept(G, 9 * K8)
                want, mag = ref.tmm(r, sq)
                check(g[:K8].cpu().numpy(), want, mag, what=f"end of allocation spec={spec} N={N} sq={sq} tmm_dev")
                want, mag = ref.tmm(R, sq)
                check(G[:9 * K8].cpu().numpy().reshape((K8, 9), order="F"), want, mag, what=f"spec={spec} N={N} sq={sq} tmm_mat_dev")
        print(f"spec={spec} N={N} allocation size reported exactly: {exact}")
print("end of allocation OK")
'''


@pytest.mark.gpu
def test_input_at_the_end_of_its_allocation():
    """The Phi^T input ends exactly where its device allocation ends (caching allocator off, so a torch tensor is its
    own cudaMalloc): the specialised Phi^T cannot read whole row tiles in place (the driver reports the allocation too
    short) and copies to a padded buffer; odd N also takes the realigning copy; the tensor-core Phi^T stages the
    columns.  Against the oracle, both families."""
    out = _run(_END_SCRIPT, {"PYTORCH_NO_CUDA_MEMORY_CACHING": "1"})
    assert "end of allocation OK" in out, out
    print(out)


@pytest.mark.gpu
def test_bench_shard_shapes(lib_stream, oracle, family):
    """bench.py's layout (yhat padded to 256 rows, r exactly nloc rows) on the C3 table at the 8-GPU shard's 125 000 rows,
    every row against the oracle; C5's mm_mat_dev / tmm_mat_dev (C = 64, leading dimension nloc) likewise."""
    nloc = 125_000
    o = c3_object(lib_stream, oracle, nloc)
    vector_products(lib_stream, o, nloc, layouts=["padded"], sqs=(0,), what=f"c3 shard family={family}")
    matrix_products_plain(lib_stream, o, nloc, 64, what=f"c5 shard family={family}")


def matrix_products_plain(lib, o, N, C, what):
    ob, ref, terms = o["ob"], o["ref"], o["terms"]
    K = terms.shape[0]
    if ("c5", C) not in o["cache"]:
        rng = np.random.default_rng(1)
        A = np.asfortranarray(rng.normal(size=(K, C)) * np.sqrt(o["om"].getvar(terms) / 20)[:, None])
        R = np.asfortranarray(np.random.default_rng([7, 0]).normal(size=(N, C)))
        o["cache"][("c5", C)] = (A, R, ref.mm(A, 0), ref.tmm(R, 0))
    A, R, (ya, ym), (ta, tm) = o["cache"][("c5", C)]
    Ad, Rd = device_input(A.ravel(order="F"), "padded"), device_input(R.ravel(order="F"), "padded")
    Y, G = nan_buffer(ceil256(N) * C), nan_buffer(K * C + TAIL)  # bench's output buffer: C columns of 256-padded length
    ob.mm_mat_dev(Ad.data_ptr(), C, Y.data_ptr())
    ob.tmm_mat_dev(Rd.data_ptr(), C, G.data_ptr())
    lib.synchronize()
    assert kept(Y, N * C) and kept(G, K * C), what
    check(Y[:N * C].cpu().numpy().reshape((N, C), order="F"), ya, ym, what=what + " mm_mat_dev")
    check(G[:K * C].cpu().numpy().reshape((K, C), order="F"), ta, tm, what=what + " tmm_mat_dev")


@pytest.mark.gpu
def test_bench_one_gpu_shape(lib_stream, oracle):
    """bench.py's one-GPU shape (C3, 1 000 000 rows): both families agree norm-wise within 1e-12 on both products, and
    Phi a on a seeded sample of rows (4096, plus the first and last 256) is checked element-wise against the oracle on
    those rows' basis -- built by a second object on the sampled rows alone (the build is row by row)."""
    import bench
    N = 1_000_000
    lib = lib_stream
    o = c3_object(lib, None, N)
    ob, om, terms = o["ob"], o["om"], o["terms"]
    K = terms.shape[0]
    rng = np.random.default_rng(1)
    a = np.sqrt(om.getvar(terms) / 20) * rng.normal(size=K)
    r = np.random.default_rng([7, 0]).normal(size=N)
    ad, rd = device_input(a, "padded"), device_input(r, "padded")
    res = {}
    try:
        for spec in (0, 1):
            lib.set_option("spec", spec)
            y, g = nan_buffer(ceil256(N)), nan_buffer(K + TAIL)
            ob.mm_dev(ad.data_ptr(), y.data_ptr())
            ob.tmm_dev(rd.data_ptr(), g.data_ptr())
            lib.synchronize()
            assert kept(y, N) and kept(g, K)
            res[spec] = (y[:N].cpu().numpy(), g[:K].cpu().numpy())
            assert np.isfinite(res[spec][0]).all() and np.isfinite(res[spec][1]).all()
    finally:
        lib.set_option("spec", 2)
    assert ob.spec_state(terms) == 1
    assert relerr(res[1][0], res[0][0]) < 1e-12 and relerr(res[1][1], res[0][1]) < 1e-12
    idx = np.unique(np.concatenate([np.arange(256), np.arange(N - 256, N),
                                    np.random.default_rng(2024).choice(N, size=4096, replace=False)]))
    sub = lib.outerbase(om, np.asfortranarray(bench.synth_rows(0, N, bench.D)[idx]), dograd=False)
    ref = OracleRef(oracle, sub, om, terms)
    want, mag = ref.mm(a, 0)
    for spec in (0, 1):
        check(res[spec][0][idx], want, mag, what=f"1M rows, sampled rows, spec={spec}")
