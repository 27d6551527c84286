"""The multi-response objects of include/outerbase_b200_multi.h written literally as their definition: C
single-response objects of a library (the CPU oracle in the tests), one per response column, and loops over them.

`Reference(lib)` offers the factories `fitting.obfit_multi` and `fitting.BFGS_lpdf` use (outermod, loglik_gauss_multi,
logpr_gauss_multi, lpdfvec, predictor), so one driver runs on the CUDA product and on this reference.  Coefficients and
gradients are K x C like the product's binding.  Sums over the columns are formed in column order; the marginal
adjustment of the multi-response lpdfvec is the sum of the columns' single-response adjustments (the product forms
it on the K*C-long vectors: equal up to summation order)."""
import numpy as np


class _Multi:
    def __init__(self, cols, K):
        self.cols, self.K, self.ncol = cols, K, len(cols)
        self.compute_val = self.compute_grad = True
        self.compute_gradhyp = self.compute_gradpara = False

    nterms = property(lambda s: s.K * s.ncol)
    val = property(lambda s: float(sum(c.val for c in s.cols)))
    grad = property(lambda s: np.column_stack([c.grad for c in s.cols]))
    gradhyp = property(lambda s: np.sum([c.gradhyp for c in s.cols], axis=0))
    gradpara = property(lambda s: np.sum([c.gradpara for c in s.cols], axis=0))

    def _col(self, v, c):
        return np.asarray(v, dtype=float).reshape((self.K, self.ncol), order="F")[:, c]

    def update(self, coeff):
        for c, o in enumerate(self.cols):
            o.compute_val, o.compute_grad = self.compute_val, self.compute_grad
            o.compute_gradhyp, o.compute_gradpara = self.compute_gradhyp, self.compute_gradpara
            o.update(self._col(coeff, c))

    def hessmult(self, g):
        return np.concatenate([o.hessmult(self._col(g, c)) for c, o in enumerate(self.cols)])

    def diaghess(self):
        return np.concatenate([o.diaghess() for o in self.cols])

    def diaghessgradhyp(self):
        return np.vstack([o.diaghessgradhyp() for o in self.cols])

    def updatepara(self, para):
        self.para = np.atleast_1d(np.asarray(para, dtype=float)).copy()
        for o in self.cols:
            o.updatepara(self.para)

    def paralpdf(self, p):  # fit.cpp:133-142 with this object's own defaults
        p = np.atleast_1d(np.asarray(p, dtype=float))
        return -0.5 * float(np.sum((p - self.para0) ** 2 / self.paravar)) if p.size == self.para0.size else -np.inf

    def paralpdf_grad(self, p):
        return -(np.atleast_1d(np.asarray(p, dtype=float)) - self.para0) / self.paravar


class loglik_gauss_multi(_Multi):
    def __init__(self, lib, om, terms, Y, x):
        Y = np.asarray(Y, dtype=float)
        if Y.ndim != 2 or Y.shape[0] != np.asarray(x).shape[0] or Y.shape[1] == 0:
            raise ValueError("Y must be N x C with C >= 1 and one row per row of x")
        super().__init__([lib.loglik_gauss(om, terms, Y[:, c], x) for c in range(Y.shape[1])], np.asarray(terms).shape[0])
        self.para0 = np.array([np.log(0.01 * np.mean(np.var(Y, axis=0, ddof=1)))])
        self.paravar = np.array([1.0])
        self.updatepara(self.para0)


class logpr_gauss_multi(_Multi):
    def __init__(self, lib, om, terms, ncol):
        if ncol < 1:
            raise ValueError("ncol must be at least 1")
        super().__init__([lib.logpr_gauss(om, terms) for _ in range(ncol)], np.asarray(terms).shape[0])
        self.para0, self.paravar = np.array([6.0]), np.array([4.0])  # logpr_gauss.cpp
        self.para = self.para0.copy()


class lpdfvec:
    """lpdfvec(a, b) of two multi-response children: one single-response lpdfvec per column."""

    def __init__(self, lib, a, b):
        if not (isinstance(a, _Multi) and isinstance(b, _Multi)) or a.ncol != b.ncol:
            raise ValueError("lpdfvec: children must be multi-response with the same number of columns")
        self.kids, self.K, self.ncol = (a, b), a.K, a.ncol
        self.vecs = [lib.lpdfvec(a.cols[c], b.cols[c]) for c in range(a.ncol)]
        self.cg_iters_per_column = np.zeros(a.ncol, dtype=int)

    para = property(lambda s: np.concatenate([s.kids[0].para, s.kids[1].para]))
    val = property(lambda s: float(sum(v.val for v in s.vecs)))
    coeff = property(lambda s: np.column_stack([v.coeff for v in s.vecs]))
    grad = property(lambda s: np.column_stack([v.grad for v in s.vecs]))
    gradhyp = property(lambda s: np.sum([v.gradhyp for v in s.vecs], axis=0))
    gradpara = property(lambda s: np.sum([v.gradpara for v in s.vecs], axis=0))
    cg_iters = property(lambda s: int(s.cg_iters_per_column.max()))

    @property
    def domarg(self):
        raise AttributeError("write-only")

    @domarg.setter
    def domarg(self, v):
        for x in self.vecs:
            x.domarg = v

    def _split(self, p):
        n0 = self.kids[0].para.size
        return p[:n0], p[n0:]

    def updatepara(self, para):
        p = np.atleast_1d(np.asarray(para, dtype=float))
        for k, q in zip(self.kids, self._split(p)):
            k.para = q.copy()
        for v in self.vecs:
            v.updatepara(p)

    def updateom(self):
        for v in self.vecs:
            v.updateom()

    def updateterms(self, terms):
        for v in self.vecs:
            v.updateterms(terms)
        self.K = np.asarray(terms).shape[0]
        for k in self.kids:
            k.K = self.K

    def set_coeff(self, coeff):
        A = np.asarray(coeff, dtype=float).reshape((self.K, self.ncol), order="F")
        for c, v in enumerate(self.vecs):
            v.set_coeff(A[:, c])

    def update(self, coeff):
        A = np.asarray(coeff, dtype=float).reshape((self.K, self.ncol), order="F")
        for c, v in enumerate(self.vecs):
            v.compute_val = v.compute_grad = v.compute_gradhyp = v.compute_gradpara = True
            v.update(A[:, c])

    def optcg(self, tol, epochs):
        for c, v in enumerate(self.vecs):
            v.optcg(tol, epochs)
            self.cg_iters_per_column[c] = v.cg_iters

    def paralpdf(self, p):
        p = np.atleast_1d(np.asarray(p, dtype=float))
        return sum(k.paralpdf(q) for k, q in zip(self.kids, self._split(p)))

    def paralpdf_grad(self, p):
        p = np.atleast_1d(np.asarray(p, dtype=float))
        return np.concatenate([k.paralpdf_grad(q) for k, q in zip(self.kids, self._split(p))])


class predictor:
    """one single-response predictor per column: mean N x C, the shared variance"""

    def __init__(self, lib, loglik):
        self.preds = [lib.predictor(o) for o in loglik.cols]

    def update(self, x):
        for p in self.preds:
            p.update(x)

    def mean(self):
        return np.column_stack([p.mean() for p in self.preds])

    def var(self):
        return self.preds[0].var()


class Reference:
    def __init__(self, lib):
        self.lib = lib

    def outermod(self):
        return self.lib.outermod()

    def loglik_gauss_multi(self, om, terms, Y, x):
        return loglik_gauss_multi(self.lib, om, terms, Y, x)

    def logpr_gauss_multi(self, om, terms, ncol):
        return logpr_gauss_multi(self.lib, om, terms, ncol)

    def lpdfvec(self, a, b):
        return lpdfvec(self.lib, a, b)

    def predictor(self, loglik):
        return predictor(self.lib, loglik)
