"""ctypes binding over the C ABI of include/outerbase_b200.h.

The classes mirror the reference's Rcpp module `obmod` (src/interfaceR.cpp:661-793)
name for name -- `outermod`, `outerbase`, `loglik_gauss`, `logpr_gauss`, `lpdfvec`,
`predictor`, and the free functions `setcovfs`, `setknot`, `gethyp`, `getpara` -- so
tests and drivers read like the reference's R code.  Matrices are numpy float64 in
Fortran order (Armadillo column-major), `terms` is uint64 Fortran order.

`Library(path, prefix)` binds one shared library exporting that ABI under a symbol
prefix.  The product package binds its own CUDA library (prefix `ob_`); tests also
bind the CPU oracle (prefix `orc_`) through this same class.  Nothing in this module
knows where the oracle lives.
"""
from __future__ import annotations

import ctypes as C
import re
from pathlib import Path

import numpy as np

_ERR = {1: ValueError, 2: RuntimeError, 3: RuntimeError, 4: RuntimeError, 5: RuntimeError}


def header_symbols(header: Path, prefix: str = "ob_") -> list[str]:
    """Every function name include/outerbase_b200.h declares (renamed to `prefix`)."""
    txt = Path(header).read_text()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    names = re.findall(r"\b(?:int|const char\*)\s+(ob_[a-z0-9_]+)\s*\(", txt)
    return [prefix + n[3:] for n in names]


def _f64(a, order="F"):
    return np.require(np.asarray(a, dtype=np.float64), requirements=["F_CONTIGUOUS" if order == "F" else "C_CONTIGUOUS", "ALIGNED"])


def _terms(t):
    t = np.asarray(t)
    if t.ndim != 2:
        raise ValueError("terms must be a K x d table")
    return np.require(t.astype(np.uint64, copy=False), requirements=["F_CONTIGUOUS", "ALIGNED"])


def _p(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


def _u(x):
    return C.c_uint64(int(x))


class Library:
    def __init__(self, path, prefix="ob_", device=0, create_ctx=True):
        self.path = str(path)
        self.prefix = prefix
        self.lib = C.CDLL(self.path, mode=C.RTLD_GLOBAL if False else C.RTLD_LOCAL)
        self.fn("last_error").restype = C.c_char_p
        self.ctx = None
        if create_ctx:
            h = C.c_void_p()
            self.call("ctx_create", C.c_int(device), C.byref(h))
            self.ctx = h

    # -- plumbing
    def fn(self, name):
        return getattr(self.lib, self.prefix + name)

    def has(self, name):
        return hasattr(self.lib, name)

    def call(self, name, *args):
        f = self.fn(name)
        f.restype = C.c_int
        rc = f(*args)
        if rc != 0:
            msg = self.fn("last_error")()
            raise _ERR.get(rc, RuntimeError)(f"{self.prefix}{name}: {msg.decode() if msg else rc}")

    # -- context
    def synchronize(self):
        self.call("ctx_synchronize", self.ctx)

    def stream(self) -> int:
        s = C.c_void_p()
        self.call("ctx_stream", self.ctx, C.byref(s))
        return s.value or 0

    def set_option(self, name: str, value: float):
        """Context options; "spec" = 0 never | 1 at first use | 2 auto (terms-specialised kernels)."""
        self.call("ctx_set_option", self.ctx, name.encode(), C.c_double(value))

    def spec_source(self, terms, opts=None):
        """CUDA source the generator emits for a terms table (host only) -> (source, info)."""
        t = _terms(terms)
        o = (C.c_int * 9)(*opts) if opts is not None else None
        n = C.c_uint64(0)
        info = (C.c_uint64 * 4)()
        self.call("spec_source", _p(t), _u(t.shape[0]), _u(t.shape[1]), o, None, C.byref(n), info)
        buf = C.create_string_buffer(n.value)
        self.call("spec_source", _p(t), _u(t.shape[0]), _u(t.shape[1]), o, buf, C.byref(n), info)
        return buf.value.decode(), dict(types=info[0], nacc=info[1], tile_rows_a=info[2], tile_rows_t=info[3])

    def spec_source_tmat(self, terms):
        """Source of the tensor-core Phi^T.A module (phi_tm_spec) for a table; info = {types, maxcols}."""
        t = np.asfortranarray(terms, dtype=np.uint64)
        n = C.c_uint64(0)
        info = (C.c_uint64 * 2)()
        self.call("spec_source_tmat", _p(t), _u(t.shape[0]), _u(t.shape[1]), None, C.byref(n), info)
        buf = C.create_string_buffer(n.value)
        self.call("spec_source_tmat", _p(t), _u(t.shape[0]), _u(t.shape[1]), buf, C.byref(n), info)
        return buf.value.decode(), {"types": info[0], "maxcols": info[1]}

    def spec_source_mat(self, terms):
        """Source of the multi-right-hand-side kernel (phi_am_spec) for a table; info = (blocks per pass, tile rows)."""
        t = _terms(terms)
        n = C.c_uint64(0)
        info = (C.c_uint64 * 2)()
        self.call("spec_source_mat", _p(t), _u(t.shape[0]), _u(t.shape[1]), None, C.byref(n), info)
        buf = C.create_string_buffer(n.value)
        self.call("spec_source_mat", _p(t), _u(t.shape[0]), _u(t.shape[1]), buf, C.byref(n), info)
        return buf.value.decode(), tuple(int(v) for v in info)

    def spec_source_dot(self, terms):
        """CUDA source of the hyper-gradient sweep kernel (phi_d_spec) for a terms table (host only) -> (source, info)."""
        t = _terms(terms)
        n = C.c_uint64(0)
        info = (C.c_uint64 * 2)()
        self.call("spec_source_dot", _p(t), _u(t.shape[0]), _u(t.shape[1]), None, C.byref(n), info)
        buf = C.create_string_buffer(n.value)
        self.call("spec_source_dot", _p(t), _u(t.shape[0]), _u(t.shape[1]), buf, C.byref(n), info)
        return buf.value.decode(), dict(slots=info[0], tile_rows=info[1])

    def spec_compile_check(self, source: str):
        """NVRTC-compile a generated source for sm_100a (no GPU needed) -> (cubin bytes, seconds)."""
        nb, sec = C.c_uint64(0), C.c_double(0)
        self.call("spec_compile_check", source.encode(), C.byref(nb), C.byref(sec))
        return nb.value, sec.value

    def debug_normals(self, seed, stream, column, first, n):
        """n standard normals of the posterior draws' generator (seed, stream, column) from index `first` on, computed
        on the host (include/outerbase_b200_draws.h); no GPU needed."""
        out = np.empty(int(n))
        self.call("debug_normals", _u(seed), C.c_uint32(int(stream)), _u(column), _u(first), _u(n), _p(out))
        return out

    def fp64_peak(self) -> float:
        v = C.c_double()
        self.call("ctx_fp64_peak", self.ctx, C.byref(v))
        return v.value

    def launch_count(self) -> int:
        n = C.c_uint64()
        self.call("ctx_launch_count", self.ctx, C.byref(n))
        return n.value

    def comm_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        self.call("comm_get_unique_id", buf)
        return buf.raw

    def comm_init(self, nranks: int, rank: int, uid: bytes):
        buf = C.create_string_buffer(uid, 128)
        self.call("ctx_comm_init", self.ctx, C.c_int(nranks), C.c_int(rank), buf)

    def allreduce_dev(self, buf_ptr: int, n: int):
        """In-place sum over ranks of n doubles at a device pointer, on the library's stream (not synchronised)."""
        self.call("ctx_allreduce_dev", self.ctx, C.c_void_p(buf_ptr), C.c_uint64(n))

    def comm_info(self):
        n, r = C.c_int(), C.c_int()
        self.call("ctx_comm_info", self.ctx, C.byref(n), C.byref(r))
        return n.value, r.value

    # -- covf (src/covfuncs.cpp)
    def covf_numhyp(self, name):
        n = C.c_uint64()
        self.call("covf_numhyp", name.encode(), C.byref(n))
        return n.value

    def covf_cov(self, name, hyp, x1, x2):
        hyp, x1, x2 = _f64(hyp), _f64(x1), _f64(x2)
        out = np.empty((x1.size, x2.size), order="F")
        self.call("covf_cov", self.ctx, name.encode(), _p(hyp), _p(x1), _u(x1.size), _p(x2), _u(x2.size), _p(out))
        return out

    def covf_cov_gradhyp(self, name, hyp, x1, x2):
        hyp, x1, x2 = _f64(hyp), _f64(x1), _f64(x2)
        nh = self.covf_numhyp(name)
        out = np.empty((x1.size, x2.size, nh), order="F")
        self.call("covf_cov_gradhyp", self.ctx, name.encode(), _p(hyp), _p(x1), _u(x1.size), _p(x2), _u(x2.size), _p(out))
        return out

    # -- host-side self check of the terms compiler (product only)
    def debug_terms_eval(self, terms, knotptst, bcols, a, b=1.0, ngroups=16, aug_dim=-1, gcols0=None):
        t = _terms(terms)
        K, d = t.shape
        kp = np.ascontiguousarray(knotptst, dtype=np.uint64)
        bc, a = _f64(bcols), _f64(a)
        g0 = _f64(gcols0) if gcols0 is not None else None
        phia = C.c_double()
        phit = np.empty(K)
        stats = np.zeros(8, dtype=np.uint64)
        self.call("debug_terms_eval", _p(t), _u(K), _u(d), _p(kp), C.c_int(ngroups), C.c_int(aug_dim), _p(bc), _p(g0),
                  _p(a), C.c_double(b), C.byref(phia), _p(phit), _p(stats))
        names = ("W", "Lcols", "nodes", "maxdepth", "fast_ok", "nslots", "nwords_fwd", "nwords_bwd")
        return phia.value, phit, dict(zip(names, map(int, stats)))

    # -- object factories, named as in the Rcpp module
    def outermod(self):
        return outermod(self)

    def outerbase(self, om, x, dograd=True):
        return outerbase(self, om, x, dograd)

    def loglik_gauss(self, om, terms, y, x):
        return loglik_gauss(self, om, terms, y, x)

    def loglik_gda(self, om, terms, y, x):
        return loglik_gda(self, om, terms, y, x)

    def loglik_std(self, om, terms, y, x):
        return loglik_std(self, om, terms, y, x)

    def logpr_gauss(self, om, terms):
        return logpr_gauss(self, om, terms)

    def loglik_gauss_multi(self, om, terms, Y, x, para_per_column=False):
        return loglik_gauss_multi(self, om, terms, Y, x, para_per_column)

    def logpr_gauss_multi(self, om, terms, ncol, para_per_column=False):
        return logpr_gauss_multi(self, om, terms, ncol, para_per_column)

    def loglik_gda_multi(self, om, terms, Y, x):
        return loglik_gda_multi(self, om, terms, Y, x)

    def lpdfvec(self, a, b):
        if isinstance(a, _multi) or isinstance(b, _multi):
            return lpdfvec_multi(self, a, b)
        return lpdfvec(self, a, b)

    def predictor(self, loglik):
        if isinstance(loglik, (loglik_gauss_multi, loglik_gda_multi)):
            return predictor_multi(self, loglik)
        return predictor(self, loglik)

    # -- stateless linalg.h seam (src/linalg.h:9-58)
    def prodmm(self, terms, a, basemat, basescale, knotptst):
        t, a, bm, bs = _terms(terms), _f64(a), _f64(basemat), _f64(basescale)
        kp = np.ascontiguousarray(knotptst, dtype=np.uint64)
        N, M = bm.shape
        if a.ndim == 1:
            out = np.empty(N)
            self.call("prodmm_vec", self.ctx, _p(out), _p(t), _u(t.shape[0]), _u(t.shape[1]), _p(a), _p(bm), _u(N), _u(M), _p(bs), _p(kp))
        else:
            out = np.empty((N, a.shape[1]), order="F")
            self.call("prodmm_mat", self.ctx, _p(out), _p(t), _u(t.shape[0]), _u(t.shape[1]), _p(a), _u(a.shape[1]), _p(bm), _u(N), _u(M), _p(bs), _p(kp))
        return out

    def tprodmm(self, terms, a, basemat, basescale, knotptst):
        t, a, bm, bs = _terms(terms), _f64(a), _f64(basemat), _f64(basescale)
        kp = np.ascontiguousarray(knotptst, dtype=np.uint64)
        N, M = bm.shape
        K = t.shape[0]
        if a.ndim == 1:
            out = np.empty(K)
            self.call("tprodmm_vec", self.ctx, _p(out), _p(t), _u(K), _u(t.shape[1]), _p(a), _p(bm), _u(N), _u(M), _p(bs), _p(kp))
        else:
            out = np.empty((K, a.shape[1]), order="F")
            self.call("tprodmm_mat", self.ctx, _p(out), _p(t), _u(K), _u(t.shape[1]), _p(a), _u(a.shape[1]), _p(bm), _u(N), _u(M), _p(bs), _p(kp))
        return out

    def _ge(self, name, terms, a, basemat, basescale, knotptst, basematge, gest, hypmatch, nout):
        t, a, bm, bs, bg = _terms(terms), _f64(a), _f64(basemat), _f64(basescale), _f64(basematge)
        kp = np.ascontiguousarray(knotptst, dtype=np.uint64)
        ge = np.ascontiguousarray(gest, dtype=np.uint64)
        hm = np.ascontiguousarray(hypmatch, dtype=np.uint64)
        N, M = bm.shape
        H = hm.size
        out = np.empty(nout)
        outge = np.empty((nout, H), order="F")
        self.call(name, self.ctx, _p(out), _p(outge), _p(t), _u(t.shape[0]), _u(t.shape[1]), _p(a), _p(bm), _u(N), _u(M), _p(bs), _p(kp),
                  _p(bg), _u(bg.shape[1]), _p(ge), _p(hm), _u(H))
        return out, outge

    def prodmmge(self, terms, a, basemat, basescale, knotptst, basematge, gest, hypmatch):
        return self._ge("prodmmge", terms, a, basemat, basescale, knotptst, basematge, gest, hypmatch, np.asarray(basemat).shape[0])

    def tprodmmge(self, terms, a, basemat, basescale, knotptst, basematge, gest, hypmatch):
        return self._ge("tprodmmge", terms, a, basemat, basescale, knotptst, basematge, gest, hypmatch, np.asarray(terms).shape[0])

    def getmge(self, terms, basemat, basescale, knotptst, basematge, gest, hypmatch):
        """getmge_, src/linalg.cpp:778-822: N x K x H cube."""
        t, bm, bs, bg = _terms(terms), _f64(basemat), _f64(basescale), _f64(basematge)
        kp, ge, hm = (np.ascontiguousarray(v, dtype=np.uint64) for v in (knotptst, gest, hypmatch))
        N, M = bm.shape
        out = np.empty((N, t.shape[0], hm.size), order="F")
        self.call("getmge", self.ctx, _p(out), _p(t), _u(t.shape[0]), _u(t.shape[1]), _p(bm), _u(N), _u(M), _p(bs), _p(kp), _p(bg), _u(bg.shape[1]),
                  _p(ge), _p(hm), _u(hm.size))
        return out

    def getm(self, terms, basemat, basescale, knotptst):
        t, bm, bs = _terms(terms), _f64(basemat), _f64(basescale)
        kp = np.ascontiguousarray(knotptst, dtype=np.uint64)
        N, M = bm.shape
        out = np.empty((N, t.shape[0]), order="F")
        self.call("getm", self.ctx, _p(out), _p(t), _u(t.shape[0]), _u(t.shape[1]), _p(bm), _u(N), _u(M), _p(bs), _p(kp))
        return out


class _Handle:
    _destroy = None

    def __init__(self, lib: Library):
        self._lib = lib
        self._h = C.c_void_p()

    def __del__(self):
        try:
            if self._h and self._destroy:
                self._lib.call(self._destroy, self._h)
                self._h = C.c_void_p()
        except Exception:
            pass


def _build_geometry(lib, name, h, d):
    out = (C.c_int * (4 * d))()
    lib.call(name, h, out)
    return [("dmma" if out[4 * l] else "fma", out[4 * l + 1], out[4 * l + 2], out[4 * l + 3]) for l in range(d)]


class outermod(_Handle):
    """new(outermod) -- src/modandbase.h:9-54."""
    _destroy = "outermod_destroy"

    def __init__(self, lib):
        super().__init__(lib)
        lib.call("outermod_create", C.byref(self._h))
        self._keep = []

    def setcovfs(self, names):
        arr = (C.c_char_p * len(names))(*[n.encode() for n in names])
        self._lib.call("outermod_setcovfs", self._h, _u(len(names)), arr)

    def setknot(self, knotlist):
        ks = [np.asarray(k, dtype=np.float64).ravel() for k in knotlist]
        flat = np.ascontiguousarray(np.concatenate(ks)) if ks else np.zeros(0)
        lens = np.ascontiguousarray([k.size for k in ks], dtype=np.uint64)
        self._lib.call("outermod_setknot", self._h, _p(flat), _p(lens))

    def sizes(self):
        d, h, m, g = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._lib.call("outermod_sizes", self._h, C.byref(d), C.byref(h), C.byref(m), C.byref(g))
        return d.value, h.value, m.value, g.value

    @property
    def d(self):
        return self.sizes()[0]

    def updatehyp(self, hyp):
        hyp = _f64(hyp)
        self._lib.call("outermod_updatehyp", self._h, _p(hyp), _u(hyp.size))

    def gethyp(self):
        out = np.empty(self.sizes()[1])
        self._lib.call("outermod_gethyp", self._h, _p(out))
        return out

    def set_select_seed(self, seed):
        self._lib.call("outermod_set_select_seed", self._h, _u(seed))

    def selectterms(self, numele):
        out = np.empty((int(numele), self.d), dtype=np.uint64, order="F")
        self._lib.call("outermod_selectterms", self._h, _u(numele), _p(out))
        return out

    def getvar(self, terms):
        t = _terms(terms)
        out = np.empty(t.shape[0])
        self._lib.call("outermod_getvar", self._h, _p(t), _u(t.shape[0]), _p(out))
        return out

    def getlvar_gradhyp(self, terms):
        t = _terms(terms)
        out = np.empty((t.shape[0], self.sizes()[1]), order="F")
        self._lib.call("outermod_getlvar_gradhyp", self._h, _p(t), _u(t.shape[0]), _p(out))
        return out

    def hyplpdf(self, hyp):
        hyp = _f64(hyp)
        out = C.c_double()
        self._lib.call("outermod_hyplpdf", self._h, _p(hyp), _u(hyp.size), C.byref(out))
        return out.value

    def hyplpdf_grad(self, hyp):
        hyp = _f64(hyp)
        out = np.empty(self.sizes()[1])
        self._lib.call("outermod_hyplpdf_grad", self._h, _p(hyp), _u(hyp.size), _p(out))
        return out

    def index(self, which):
        n = C.c_uint64()
        self._lib.call("outermod_get_index", self._h, which.encode(), C.c_void_p(0), C.byref(n))
        out = np.empty(n.value, dtype=np.int64)
        self._lib.call("outermod_get_index", self._h, which.encode(), _p(out), C.byref(n))
        return out

    def real(self, which):
        r, c = C.c_uint64(), C.c_uint64()
        self._lib.call("outermod_get_real", self._h, which.encode(), C.c_void_p(0), C.byref(r), C.byref(c))
        out = np.empty((r.value, c.value), order="F")
        self._lib.call("outermod_get_real", self._h, which.encode(), _p(out), C.byref(r), C.byref(c))
        return out[:, 0].copy() if c.value == 1 else out


def setcovfs(om: outermod, names):  # src/interfaceR.cpp:53
    om.setcovfs(list(names))


def setknot(om: outermod, knotlist):  # src/interfaceR.cpp:94
    om.setknot(knotlist)


def gethyp(om: outermod):  # src/interfaceR.cpp:151
    return om.gethyp()


def getpara(logpdf):  # src/interfaceR.cpp:168
    return logpdf.para


class outerbase(_Handle):
    """new(outerbase, om, x) -- src/modandbase.h:57-125, src/interfaceR.cpp:680-694."""
    _destroy = "outerbase_destroy"

    def __init__(self, lib, om, x, dograd=True):
        super().__init__(lib)
        self._om = om
        x = _f64(x)
        if x.ndim != 2:
            raise ValueError("x must be N x d")
        self.n_row, self.d = x.shape
        lib.call("outerbase_create", lib.ctx, om._h, _p(x), _u(x.shape[0]), C.c_int(1 if dograd else 0), C.byref(self._h))

    def build(self):
        self._lib.call("outerbase_build", self._h)

    def specialize(self, terms) -> float:
        """Compile the terms-specialised kernels for this table now; returns the compile seconds."""
        t = _terms(terms)
        sec = C.c_double(0)
        self._lib.call("outerbase_specialize", self._h, _p(t), _u(t.shape[0]), C.byref(sec))
        return sec.value

    def spec_state(self, terms) -> int:
        t = _terms(terms)
        st = C.c_int(0)
        self._lib.call("outerbase_spec_state", self._h, _p(t), _u(t.shape[0]), C.byref(st))
        return st.value

    def debug_phi_geometry(self, terms, transpose=False, sq=0):
        """Layout of the interpreter Phi a (Phi^T with transpose) kernel for this object's rows and a terms table:
        R (rows per lane; 0 = brute-force kernels), nbuf (tile buffers), prog_in_smem, smem (bytes). Product only."""
        t = _terms(terms)
        out = (C.c_int * 4)()
        self._lib.call("outerbase_debug_phi_geometry", self._h, _p(t), _u(t.shape[0]), C.c_int(1 if transpose else 0), C.c_int(sq), out)
        return dict(zip(("R", "nbuf", "prog_in_smem", "smem"), map(int, out)))

    def debug_build_geometry(self):
        """The kernel each dimension's last basis build ran on: one (family, tile, mo, smem) per dimension, family
        "dmma" (tile = column tiles of 8) or "fma" (tile = rows per CTA). Product only."""
        return _build_geometry(self._lib, "outerbase_debug_build_geometry", self._h, self.d)

    def _loopvals(self):
        nt, cs, ls, vp = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_int()
        self._lib.call("outerbase_loopvals", self._h, C.byref(nt), C.byref(cs), C.byref(ls), C.byref(vp))
        return nt.value, cs.value, ls.value, bool(vp.value)

    nthreads = property(lambda s: s._loopvals()[0], lambda s, k: s._lib.call("outerbase_set_nthreads", s._h, C.c_int(int(k))))
    chunksize = property(lambda s: s._loopvals()[1])
    loopsize = property(lambda s: s._loopvals()[2])
    vertpl = property(lambda s: s._loopvals()[3])

    def real(self, which):
        r, c = C.c_uint64(), C.c_uint64()
        self._lib.call("outerbase_get_real", self._h, which.encode(), C.c_void_p(0), C.byref(r), C.byref(c))
        out = np.empty((r.value, c.value), order="F")
        self._lib.call("outerbase_get_real", self._h, which.encode(), _p(out), C.byref(r), C.byref(c))
        return out[:, 0].copy() if which == "basescale" else out

    def getbase(self, dim):
        kp = self._om.index("knotptst")
        if not 1 <= dim <= self.d:
            raise ValueError("dim out of range")
        out = np.empty((self.n_row, int(kp[dim] - kp[dim - 1])), order="F")
        self._lib.call("outerbase_getbase", self._h, _u(dim), _p(out))
        return out

    def getmat(self, terms):
        t = _terms(terms)
        out = np.empty((self.n_row, t.shape[0]), order="F")
        self._lib.call("outerbase_getmat", self._h, _p(t), _u(t.shape[0]), _p(out))
        return out

    def getmat_gradhyp(self, terms):
        """outerbase::getmat_gradhyp, src/modandbase.cpp:663-669: N x K x H cube (loglik_std's basismat_gradhyp)."""
        t = _terms(terms)
        out = np.empty((self.n_row, t.shape[0], self._om.sizes()[1]), order="F")
        self._lib.call("outerbase_getmat_gradhyp", self._h, _p(t), _u(t.shape[0]), _p(out))
        return out

    def _mm(self, sq, terms, a, out=None):
        t, a = _terms(terms), _f64(a)
        if a.ndim == 2:
            if a.shape[0] != t.shape[0]:
                raise ValueError("a must have one row per term")
            out = np.empty((self.n_row, a.shape[1]), order="F")
            self._lib.call("outerbase_mm_mat", self._h, C.c_int(sq), _p(t), _u(t.shape[0]), _p(a), _u(a.shape[1]), _p(out))
            return out
        if a.size != t.shape[0]:
            raise ValueError("a must have one entry per term")
        if out is None:
            out = np.empty(self.n_row)
        elif out.dtype != np.float64 or out.size != self.n_row or not out.flags.c_contiguous:
            raise ValueError("out must be a contiguous float64 vector with one entry per row")
        self._lib.call("outerbase_mm", self._h, C.c_int(sq), _p(t), _u(t.shape[0]), _p(a), _p(out))
        return out

    def _tmm(self, sq, terms, a, out=None):
        t, a = _terms(terms), _f64(a)
        if a.shape[0] != self.n_row:
            raise ValueError("a must have one entry per row")
        if a.ndim == 2:
            out = np.empty((t.shape[0], a.shape[1]), order="F")
            self._lib.call("outerbase_tmm_mat", self._h, C.c_int(sq), _p(t), _u(t.shape[0]), _p(a), _u(a.shape[1]), _p(out))
            return out
        if out is None:
            out = np.empty(t.shape[0])
        elif out.dtype != np.float64 or out.size != t.shape[0] or not out.flags.c_contiguous:
            raise ValueError("out must be a contiguous float64 vector with one entry per term")
        self._lib.call("outerbase_tmm", self._h, C.c_int(sq), _p(t), _u(t.shape[0]), _p(a), _p(out))
        return out

    def _mmge(self, sq, terms, a):
        t, a = _terms(terms), _f64(a)
        H = self._om.sizes()[1]
        out, outge = np.empty(self.n_row), np.empty((self.n_row, H), order="F")
        self._lib.call("outerbase_mm_gradhyp", self._h, C.c_int(sq), _p(t), _u(t.shape[0]), _p(a), _p(out), _p(outge))
        return out, outge

    def _tmmge(self, sq, terms, a):
        t, a = _terms(terms), _f64(a)
        H = self._om.sizes()[1]
        out, outge = np.empty(t.shape[0]), np.empty((t.shape[0], H), order="F")
        self._lib.call("outerbase_tmm_gradhyp", self._h, C.c_int(sq), _p(t), _u(t.shape[0]), _p(a), _p(out), _p(outge))
        return out, outge

    # R-visible methods (interfaceR.cpp:686-693)
    def matmul(self, terms, a, out=None):
        """obj$matmul(terms, a); `out` (optional) receives the result in place, e.g. a pinned buffer."""
        return self._mm(0, terms, a, out)

    def tmatmul(self, terms, a, out=None):
        return self._tmm(0, terms, a, out)

    def matmul_gradhyp(self, terms, a):
        return self._mmge(0, terms, a)[1]

    def tmatmul_gradhyp(self, terms, a):
        return self._tmmge(0, terms, a)[1]

    # C++-only methods (modandbase.h:100-111)
    def sqmm(self, terms, a):
        return self._mm(1, terms, a)

    def sqtmm(self, terms, a):
        return self._tmm(1, terms, a)

    def sqtmmm(self, terms, a):
        return self._tmm(1, terms, a)

    def residvar(self, terms):
        """outerbase::residvar, src/modandbase.cpp:889-896."""
        t = _terms(terms)
        out = np.empty(self.n_row)
        self._lib.call("outerbase_residvar", self._h, _p(t), _u(t.shape[0]), _p(out))
        return out

    def residvar_gradhyp(self, terms):
        """outerbase::residvar_gradhyp, src/modandbase.cpp:904-922."""
        t = _terms(terms)
        out = np.empty((self.n_row, self._om.sizes()[1]), order="F")
        self._lib.call("outerbase_residvar_gradhyp", self._h, _p(t), _u(t.shape[0]), _p(out))
        return out

    def sqmm_gradhyp(self, terms, a):
        return self._mmge(1, terms, a)[1]

    def sqtmm_gradhyp(self, terms, a):
        return self._tmmge(1, terms, a)[1]

    def sqcolsums(self, terms):
        return self._tmm(1, terms, np.ones(self.n_row))

    def sqcolsums_gradhyp(self, terms):
        return self._tmmge(1, terms, np.ones(self.n_row))[1]

    # device-pointer forms (ints are raw device addresses, e.g. torch .data_ptr())
    def set_terms(self, terms):
        t = _terms(terms)
        self._lib.call("outerbase_set_terms", self._h, _p(t), _u(t.shape[0]))

    def mm_dev(self, a_ptr, out_ptr, sq=0):
        self._lib.call("outerbase_mm_dev", self._h, C.c_int(sq), C.c_void_p(a_ptr), C.c_void_p(out_ptr))

    def tmm_dev(self, a_ptr, out_ptr, sq=0):
        self._lib.call("outerbase_tmm_dev", self._h, C.c_int(sq), C.c_void_p(a_ptr), C.c_void_p(out_ptr))

    def mm_mat_dev(self, A_ptr, ncol, out_ptr, sq=0):
        self._lib.call("outerbase_mm_mat_dev", self._h, C.c_int(sq), C.c_void_p(A_ptr), _u(ncol), C.c_void_p(out_ptr))

    def tmm_mat_dev(self, A_ptr, ncol, out_ptr, sq=0):
        self._lib.call("outerbase_tmm_mat_dev", self._h, C.c_int(sq), C.c_void_p(A_ptr), _u(ncol), C.c_void_p(out_ptr))

    def terms_stats(self):
        w, lc, nd, md = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._lib.call("outerbase_terms_stats", self._h, C.byref(w), C.byref(lc), C.byref(nd), C.byref(md))
        return {"W": w.value, "Lcols": lc.value, "nodes": nd.value, "maxdepth": md.value}


class lpdf(_Handle):
    """class lpdf -- src/fit.h:23-90, src/interfaceR.cpp:696-723."""
    _destroy = "lpdf_destroy"

    def _sizes(self):
        k, p, h, n = C.c_uint64(), C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._lib.call("lpdf_sizes", self._h, C.byref(k), C.byref(p), C.byref(h), C.byref(n))
        return k.value, p.value, h.value, n.value

    def _get(self, which):
        n = C.c_uint64()
        self._lib.call("lpdf_get", self._h, which.encode(), C.c_void_p(0), C.byref(n))
        out = np.empty(n.value)
        self._lib.call("lpdf_get", self._h, which.encode(), _p(out), C.byref(n))
        return out

    def _flag(self, which, v):
        self._lib.call("lpdf_set_flag", self._h, which.encode(), C.c_int(1 if v else 0))

    nterms = property(lambda s: s._sizes()[0])
    val = property(lambda s: float(s._get("val")[0]))
    grad = property(lambda s: s._get("grad"))
    gradhyp = property(lambda s: s._get("gradhyp"))
    gradpara = property(lambda s: s._get("gradpara"))
    coeff = property(lambda s: s._get("coeff"))
    para = property(lambda s: s._get("para"))
    totdiaghess = property(lambda s: s._get("totdiaghess"))
    tothess = property(lambda s: (lambda v: v.reshape((int(round(v.size ** 0.5)),) * 2, order="F"))(s._get("tothess")))
    fullhess = property(fset=lambda s, v: s._flag("fullhess", v))
    cg_iters = property(lambda s: int(s._get("cg_iters")[0]))
    # C++ member names; the R module swaps gradhyp/gradpara (interfaceR.cpp:700-701)
    compute_val = property(fset=lambda s, v: s._flag("compute_val", v))
    compute_grad = property(fset=lambda s, v: s._flag("compute_grad", v))
    compute_gradhyp = property(fset=lambda s, v: s._flag("compute_gradhyp", v))
    compute_gradpara = property(fset=lambda s, v: s._flag("compute_gradpara", v))

    def debug_build_geometry(self):
        """outerbase.debug_build_geometry for the basis a likelihood holds. Product only."""
        return _build_geometry(self._lib, "lpdf_debug_build_geometry", self._h, self._om.d)

    def setnthreads(self, k):
        self._lib.call("lpdf_setnthreads", self._h, C.c_int(int(k)))

    def update(self, coeff):
        c = _f64(coeff)
        self._lib.call("lpdf_update", self._h, _p(c), _u(c.size))

    def updateom(self):
        self._lib.call("lpdf_updateom", self._h)

    def updatepara(self, para):
        p = _f64(np.atleast_1d(para))
        self._lib.call("lpdf_updatepara", self._h, _p(p), _u(p.size))

    def updateterms(self, terms):
        t = _terms(terms)
        self._lib.call("lpdf_updateterms", self._h, _p(t), _u(t.shape[0]))

    def optcg(self, tol, epoch):
        self._lib.call("lpdf_optcg", self._h, C.c_double(tol), _u(epoch))

    def optnewton(self):
        """lpdf$optnewton() -- src/fit.cpp:98-131, src/interfaceR.cpp:715."""
        self._lib.call("lpdf_optnewton", self._h)

    def set_coeff(self, coeff):
        c = _f64(coeff)
        self._lib.call("lpdf_set_coeff", self._h, _p(c), _u(c.size))

    def _cube(self, name, nslices):
        k = self.nterms
        out = np.empty((k, k, max(nslices, 1)), order="F")
        n = C.c_uint64()
        self._lib.call(name, self._h, _p(out), C.byref(n))
        if n.value == 0:  # the reference returns an empty matrix / cube (fit.h:86-88)
            return np.empty((0, 0, 0), order="F")
        if n.value != k * k * nslices:
            raise RuntimeError(f"{name}: {n.value} values for a {k} x {k} x {nslices} result")
        return out[:, :, :nslices]

    def hess(self):
        h = self._cube("lpdf_hess", 1)
        return h[:, :, 0] if h.size else np.empty((0, 0))

    def hessgradhyp(self):
        return self._cube("lpdf_hessgradhyp", self._sizes()[2])

    def hessgradpara(self):
        return self._cube("lpdf_hessgradpara", self._sizes()[1])

    def hessmult(self, g):
        g = _f64(g)
        out = np.empty(self.nterms)
        self._lib.call("lpdf_hessmult", self._h, _p(g), _p(out))
        return out

    def diaghess(self):
        out = np.empty(self.nterms)
        self._lib.call("lpdf_diaghess", self._h, _p(out))
        return out

    def diaghessgradhyp(self):
        k, _, h, _ = self._sizes()
        out = np.empty((k, h), order="F")
        self._lib.call("lpdf_diaghessgradhyp", self._h, _p(out))
        return out

    def diaghessgradpara(self):
        k, p, _, _ = self._sizes()
        out = np.empty((k, p), order="F")
        self._lib.call("lpdf_diaghessgradpara", self._h, _p(out))
        return out

    def paralpdf(self, para):
        p = _f64(np.atleast_1d(para))
        out = C.c_double()
        self._lib.call("lpdf_paralpdf", self._h, _p(p), _u(p.size), C.byref(out))
        return out.value

    def paralpdf_grad(self, para):
        p = _f64(np.atleast_1d(para))
        out = np.empty(self._sizes()[1])
        self._lib.call("lpdf_paralpdf_grad", self._h, _p(p), _u(p.size), _p(out))
        return out


class loglik_gauss(lpdf):
    """new(loglik_gauss, om, terms, y, x) -- src/lpdfs/loglik_gauss.cpp:41."""

    def __init__(self, lib, om, terms, y, x):
        super().__init__(lib)
        self._om = om
        t, y, x = _terms(terms), _f64(y), _f64(x)
        if x.shape[0] != y.size:
            raise ValueError("x and y dims do not align")
        lib.call("loglik_gauss_create", lib.ctx, om._h, _p(t), _u(t.shape[0]), _p(y), _p(x), _u(y.size), C.byref(self._h))

    yhat = property(lambda s: s._get("yhat"))


class loglik_std(lpdf):
    """new(loglik_std, om, terms, y, x) -- src/lpdfs/loglik_std.cpp:41, src/interfaceR.cpp:733-737."""

    def __init__(self, lib, om, terms, y, x):
        super().__init__(lib)
        self._om = om
        t, y, x = _terms(terms), _f64(y), _f64(x)
        if x.shape[0] != y.size:
            raise ValueError("x and y dims do not align")
        lib.call("loglik_std_create", lib.ctx, om._h, _p(t), _u(t.shape[0]), _p(y), _p(x), _u(y.size), C.byref(self._h))

    yhat = property(lambda s: s._get("yhat"))


class loglik_gda(lpdf):
    """new(loglik_gda, om, terms, y, x) -- src/lpdfs/loglik_gda.cpp:47, src/interfaceR.cpp:745-750."""

    def __init__(self, lib, om, terms, y, x):
        super().__init__(lib)
        self._om = om
        t, y, x = _terms(terms), _f64(y), _f64(x)
        if x.shape[0] != y.size:
            raise ValueError("x and y dims do not align")
        lib.call("loglik_gda_create", lib.ctx, om._h, _p(t), _u(t.shape[0]), _p(y), _p(x), _u(y.size), C.byref(self._h))

    yhat = property(lambda s: s._get("yhat"))
    dodiag = property(fset=lambda s, v: s._flag("dodiag", v))


class logpr_gauss(lpdf):
    """new(logpr_gauss, om, terms) -- src/lpdfs/logpr_gauss.cpp:41."""

    def __init__(self, lib, om, terms):
        super().__init__(lib)
        self._om = om
        t = _terms(terms)
        lib.call("logpr_gauss_create", lib.ctx, om._h, _p(t), _u(t.shape[0]), C.byref(self._h))

    coeffsd = property(lambda s: s._get("coeffsd"))


class lpdfvec(lpdf):
    """new(lpdfvec, a, b) -- src/fit.cpp:174."""

    def __init__(self, lib, a, b):
        super().__init__(lib)
        self._children = (a, b)  # keep alive: lpdfvec holds references (fit.h:133)
        lib.call("lpdfvec_create", a._h, b._h, C.byref(self._h))

    domarg = property(fset=lambda s, v: s._flag("domarg", v))


class _multi:
    """Multi-response objects (C responses on one basis): coefficients and gradients are K x C (column c belongs to
    response c); every other quantity is as for the flat K*C vector of the C ABI."""
    ncol = property(lambda s: int(s._get("ncol")[0]))
    coeff = property(lambda s: s._get("coeff").reshape((-1, s.ncol), order="F"))
    grad = property(lambda s: s._get("grad").reshape((-1, s.ncol), order="F"))


class loglik_gauss_multi(_multi, lpdf):
    """loglik_gauss on each column of Y (N x C), all columns on one basis (include/outerbase_b200_multi.h).
    para_per_column: one noise log-sd per column (include/outerbase_b200_multi_percol.h) instead of one shared."""

    def __init__(self, lib, om, terms, Y, x, para_per_column=False):
        super().__init__(lib)
        self._om = om
        self.para_per_column = bool(para_per_column)
        t, Y, x = _terms(terms), _f64(Y), _f64(x)
        if Y.ndim != 2:
            raise ValueError("Y must be N x C")
        if x.shape[0] != Y.shape[0]:
            raise ValueError("x and Y dims do not align")
        if self.para_per_column:
            lib.call("loglik_gauss_multi_create_ex", lib.ctx, om._h, _p(t), _u(t.shape[0]), _p(Y), _u(Y.shape[1]), _p(x),
                     _u(Y.shape[0]), C.c_int(1), C.byref(self._h))
        else:
            lib.call("loglik_gauss_multi_create", lib.ctx, om._h, _p(t), _u(t.shape[0]), _p(Y), _u(Y.shape[1]), _p(x),
                     _u(Y.shape[0]), C.byref(self._h))


class logpr_gauss_multi(_multi, lpdf):
    """An independent logpr_gauss on each of ncol coefficient columns, shared coeffscale (para_per_column: one
    coeffscale per column)."""

    def __init__(self, lib, om, terms, ncol, para_per_column=False):
        super().__init__(lib)
        self._om = om
        self.para_per_column = bool(para_per_column)
        t = _terms(terms)
        if self.para_per_column:
            lib.call("logpr_gauss_multi_create_ex", lib.ctx, om._h, _p(t), _u(t.shape[0]), _u(ncol), C.c_int(1), C.byref(self._h))
        else:
            lib.call("logpr_gauss_multi_create", lib.ctx, om._h, _p(t), _u(t.shape[0]), _u(ncol), C.byref(self._h))

    def set_mean(self, mean=None):
        """Centre column c's prior at mean[:, c] (K x ncol); None: every prior centred at 0."""
        m = _f64(mean) if mean is not None else None
        self._lib.call("logpr_gauss_multi_set_mean", self._h, _p(m), _u(0 if m is None else m.size))


class loglik_gda_multi(_multi, lpdf):
    """loglik_gda on each column of Y (N x C), all columns on one basis with one per-row noise scale
    (include/outerbase_b200_multi_gda.h): the stage-1 likelihood of a two-stage multi-response fit."""

    def __init__(self, lib, om, terms, Y, x):
        super().__init__(lib)
        self._om = om
        t, Y, x = _terms(terms), _f64(Y), _f64(x)
        if Y.ndim != 2:
            raise ValueError("Y must be N x C")
        if x.shape[0] != Y.shape[0]:
            raise ValueError("x and Y dims do not align")
        lib.call("loglik_gda_multi_create", lib.ctx, om._h, _p(t), _u(t.shape[0]), _p(Y), _u(Y.shape[1]), _p(x),
                 _u(Y.shape[0]), C.byref(self._h))

    yhat = property(lambda s: s._get("yhat").reshape((-1, s.ncol), order="F"))
    dodiag = property(fset=lambda s, v: s._flag("dodiag", v))


class lpdfvec_multi(_multi, lpdfvec):
    """lpdfvec of two multi-response children; optcg runs one independent CG per column."""
    cg_iters_per_column = property(lambda s: s._get("cg_iters").astype(int))
    cg_iters = property(lambda s: int(s._get("cg_iters").max()))


class posterior_draws(_Handle):
    """S joint draws from the posterior of a fitted lpdfvec(logpr_gauss, loglik_gauss), by perturb-and-MAP
    (include/outerbase_b200_draws.h): the object copies the fit when it is made; `solve` runs the S perturbed fits,
    `coeff` is K x S, `predict(x)` the N x S draws of the latent function at new inputs."""
    _destroy = "draws_destroy"

    def __init__(self, lib, logpdf, S, seed=0):
        super().__init__(lib)
        self.S = int(S)
        lib.call("draws_create", logpdf._h, _u(S), _u(seed), C.byref(self._h))

    def _get(self, which, nrow=None):
        n = C.c_uint64()
        self._lib.call("draws_get", self._h, which.encode(), C.c_void_p(0), C.byref(n))
        out = np.empty(n.value)
        self._lib.call("draws_get", self._h, which.encode(), _p(out), C.byref(n))
        return out if nrow is None else out.reshape((-1, self.S), order="F")

    def solve(self, tol=0.001, maxepch=100):
        self._lib.call("draws_solve", self._h, C.c_double(tol), _u(maxepch))
        return self

    coeff = property(lambda s: s._get("coeff", True))
    cg_iters = property(lambda s: s._get("cg_iters").astype(int))
    y = property(lambda s: s._get("y", True))  # the perturbed responses, N x S
    prior_mean = property(lambda s: s._get("prior_mean", True))  # the prior centres delta_s, K x S

    def predict(self, x):
        x = _f64(x)
        if x.ndim != 2:
            raise ValueError("x must be N x d")
        out = np.empty((x.shape[0], self.S), order="F")
        self._lib.call("draws_predict", self._h, _p(x), _u(x.shape[0]), _p(out))
        return out


def sobol(lib, om, terms, coeff, x):
    """Mean, variance, first-order and total-effect variances of f_b = sum_k coeff[k, b] Phi_k under the product of the
    empirical marginals of x's columns (include/outerbase_b200_sobol.h).  coeff is a K-vector (mean and var are floats,
    first and total have d entries) or K x B (mean and var have B entries, first and total are d x B).  The indices are
    first / var and total / var."""
    t = _terms(terms)
    K, d = t.shape
    if d != om.d:
        raise ValueError(f"terms has {d} columns, the outermod {om.d} dimensions")
    x = _f64(x)
    if x.ndim != 2 or x.shape[1] != d:
        raise ValueError("x must be nq x d")
    c = _f64(coeff)
    vec = c.ndim == 1
    if vec:
        c = c.reshape((-1, 1), order="F")
    if c.ndim != 2 or c.shape[0] != K:
        raise ValueError("coeff must have one row per term")
    B = c.shape[1]
    mean, var = np.empty(B), np.empty(B)
    first, total = np.empty((d, B), order="F"), np.empty((d, B), order="F")
    lib.call("sobol", lib.ctx, om._h, _p(t), _u(K), _p(c), _u(B), _p(x), _u(x.shape[0]), _p(mean), _p(var), _p(first),
             _p(total))
    if vec:
        return dict(mean=float(mean[0]), var=float(var[0]), first=first[:, 0].copy(), total=total[:, 0].copy())
    return dict(mean=mean, var=var, first=first, total=total)


def sobol_pairs(lib, om, terms, coeff, x):
    """binding.sobol's four outputs (the same bits) and, for every input pair l < m, second (the pure second-order
    variance sigma2_lm) and supset (Liu-Owen superset importance: the variance of every interaction that involves both)
    (include/outerbase_b200_sobol_pairs.h).  second and supset are symmetric d x d for a K-vector coeff, d x d x B for a
    K x B coeff, with NaN on the diagonal."""
    t = _terms(terms)
    K, d = t.shape
    if d != om.d:
        raise ValueError(f"terms has {d} columns, the outermod {om.d} dimensions")
    x = _f64(x)
    if x.ndim != 2 or x.shape[1] != d:
        raise ValueError("x must be nq x d")
    c = _f64(coeff)
    vec = c.ndim == 1
    if vec:
        c = c.reshape((-1, 1), order="F")
    if c.ndim != 2 or c.shape[0] != K:
        raise ValueError("coeff must have one row per term")
    B = c.shape[1]
    P = d * (d - 1) // 2
    mean, var = np.empty(B), np.empty(B)
    first, total = np.empty((d, B), order="F"), np.empty((d, B), order="F")
    second, supset = np.empty((max(P, 1), B), order="F"), np.empty((max(P, 1), B), order="F")
    lib.call("sobol_pairs", lib.ctx, om._h, _p(t), _u(K), _p(c), _u(B), _p(x), _u(x.shape[0]), _p(mean), _p(var),
             _p(first), _p(total), _p(second), _p(supset))
    l, m = np.triu_indices(d, 1)  # row-major over l < m: row r of second / supset
    S2, SU = np.full((d, d, B), np.nan), np.full((d, d, B), np.nan)
    S2[l, m], S2[m, l] = second[:P], second[:P]
    SU[l, m], SU[m, l] = supset[:P], supset[:P]
    if vec:
        return dict(mean=float(mean[0]), var=float(var[0]), first=first[:, 0].copy(), total=total[:, 0].copy(),
                    second=S2[:, :, 0].copy(), supset=SU[:, :, 0].copy())
    return dict(mean=mean, var=var, first=first, total=total, second=S2, supset=SU)


def sobol_shapley(lib, om, terms, coeff, x):
    """binding.sobol's four outputs (the same bits) and shapley, the Shapley effect of every input: the variance of
    each ANOVA component split equally among its inputs, sum_{u containing l} sigma2_u / |u|
    (include/outerbase_b200_sobol_shapley.h).  shapley has d entries for a K-vector coeff, d x B for a K x B coeff; it
    adds up to var, and first <= shapley <= total."""
    t = _terms(terms)
    K, d = t.shape
    if d != om.d:
        raise ValueError(f"terms has {d} columns, the outermod {om.d} dimensions")
    x = _f64(x)
    if x.ndim != 2 or x.shape[1] != d:
        raise ValueError("x must be nq x d")
    c = _f64(coeff)
    vec = c.ndim == 1
    if vec:
        c = c.reshape((-1, 1), order="F")
    if c.ndim != 2 or c.shape[0] != K:
        raise ValueError("coeff must have one row per term")
    B = c.shape[1]
    mean, var = np.empty(B), np.empty(B)
    first, total, shapley = (np.empty((d, B), order="F") for _ in range(3))
    lib.call("sobol_shapley", lib.ctx, om._h, _p(t), _u(K), _p(c), _u(B), _p(x), _u(x.shape[0]), _p(mean), _p(var),
             _p(first), _p(total), _p(shapley))
    if vec:
        return dict(mean=float(mean[0]), var=float(var[0]), first=first[:, 0].copy(), total=total[:, 0].copy(),
                    shapley=shapley[:, 0].copy())
    return dict(mean=mean, var=var, first=first, total=total, shapley=shapley)


class predictor(_Handle):
    """new(predictor, loglik) -- src/fit.h:352-361."""
    _destroy = "predictor_destroy"

    def __init__(self, lib, loglik):
        super().__init__(lib)
        self._loglik = loglik
        self._n = loglik._sizes()[3]
        lib.call("predictor_create", loglik._h, C.byref(self._h))

    def update(self, x):
        x = _f64(x)
        self._n = x.shape[0]
        self._lib.call("predictor_update", self._h, _p(x), _u(x.shape[0]))

    def mean(self):
        out = np.empty(self._n)
        self._lib.call("predictor_mean", self._h, _p(out))
        return out

    def var(self):
        out = np.empty(self._n)
        self._lib.call("predictor_var", self._h, _p(out))
        return out


class predictor_multi(predictor):
    """predictor(loglik_gauss_multi or loglik_gda_multi): mean N x C; var is one N-vector shared by all columns, or
    N x C when the likelihood has a noise scale per column or was fitted under a prior with a coefficient scale per
    column."""

    def __init__(self, lib, loglik):
        super().__init__(lib, loglik)
        self._var_ncol = int(loglik._get("predvar_ncol")[0])  # fixed when the predictor is made, as its variance

    def mean(self):
        out = np.empty((self._n, self._loglik.ncol), order="F")
        self._lib.call("predictor_mean", self._h, _p(out))
        return out

    def var(self):
        if self._var_ncol == 1:
            return super().var()
        out = np.empty((self._n, self._loglik.ncol), order="F")
        self._lib.call("predictor_var", self._h, _p(out))
        return out
