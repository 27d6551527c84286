"""The per-column form of the multi-response objects (include/outerbase_b200_multi_percol.h) written literally as its
definition: C single-response objects of a library (the CPU oracle in the tests), one per response column, each at its
own para, and loops over them.

`Reference(lib)` offers the factories `fitting.obfit_multi` and `fitting.BFGS_lpdf` use, with the `para_per_column`
option of the product's binding; without it the objects are those of tests/multiresponse_reference.py.  An lpdfvec is one
single-response lpdfvec per column; its para is laid out as [child 0's entries | child 1's entries], where a per-column
child has C entries (entry c is column c's) and a shared child one entry that serves every column."""
import numpy as np

import multiresponse_reference as R


class _PerColumn:
    """para entry c belongs to column c"""

    def updatepara(self, para):
        p = np.atleast_1d(np.asarray(para, dtype=float))
        if p.size != self.ncol:
            raise ValueError("para must have one entry per column")
        self.para = p.copy()
        for o, q in zip(self.cols, p):
            o.updatepara([q])

    gradpara = property(lambda s: np.array([o.gradpara[0] for o in s.cols]))

    def diaghessgradpara(self):  # (K C) x C, block-diagonal
        K, C = self.K, self.ncol
        out = np.zeros((K * C, C))
        for c, o in enumerate(self.cols):
            out[c * K:(c + 1) * K, c] = np.asarray(o.diaghessgradpara())[:, 0]
        return out


class loglik_gauss_multi(_PerColumn, R._Multi):
    def __init__(self, lib, om, terms, Y, x):
        Y = np.asarray(Y, dtype=float)
        if Y.ndim != 2 or Y.shape[0] != np.asarray(x).shape[0] or Y.shape[1] == 0:
            raise ValueError("Y must be N x C with C >= 1 and one row per row of x")
        R._Multi.__init__(self, [lib.loglik_gauss(om, terms, Y[:, c], x) for c in range(Y.shape[1])], np.asarray(terms).shape[0])
        self.para0 = np.array([o.para[0] for o in self.cols])  # each column's own loglik_gauss default
        self.paravar = np.ones(self.ncol)
        self.para = self.para0.copy()


class logpr_gauss_multi(_PerColumn, R._Multi):
    def __init__(self, lib, om, terms, ncol):
        if ncol < 1:
            raise ValueError("ncol must be at least 1")
        R._Multi.__init__(self, [lib.logpr_gauss(om, terms) for _ in range(ncol)], np.asarray(terms).shape[0])
        self.para0, self.paravar = np.full(ncol, 6.0), np.full(ncol, 4.0)  # logpr_gauss.cpp, per column
        self.para = self.para0.copy()


def per_column(obj):
    return isinstance(obj, _PerColumn)


class lpdfvec(R.lpdfvec):
    """one single-response lpdfvec per column, column c at [child 0's entry for c, child 1's entry for c]"""

    def __init__(self, lib, a, b):
        super().__init__(lib, a, b)
        for k in self.kids:  # the columns' total diagonals differ when either child is per-column
            k.fitted_per_column = per_column(a) or per_column(b)

    def _col_para(self, p, c):
        return np.array([q[c] if per_column(k) else q[0] for k, q in zip(self.kids, self._split(p))])

    def updatepara(self, para):
        p = np.atleast_1d(np.asarray(para, dtype=float))
        if p.size != sum(k.para.size for k in self.kids):
            raise ValueError("wrongsized para vector")
        for k, q in zip(self.kids, self._split(p)):
            k.para = q.copy()
        for c, v in enumerate(self.vecs):
            v.updatepara(self._col_para(p, c))

    @property
    def gradpara(self):
        out = []
        for j, k in enumerate(self.kids):
            g = np.array([v.gradpara[j] for v in self.vecs])  # column c's derivative in child j's entry
            out.append(g if per_column(k) else np.array([g.sum()]))
        return np.concatenate(out)

    def hessmult(self, g):
        G = np.asarray(g, dtype=float).reshape((self.K, self.ncol), order="F")
        return np.concatenate([v.hessmult(G[:, c]) for c, v in enumerate(self.vecs)])

    def diaghess(self):
        return np.concatenate([v.diaghess() for v in self.vecs])

    def diaghessgradhyp(self):
        return np.vstack([v.diaghessgradhyp() for v in self.vecs])

    def diaghessgradpara(self):
        K, C = self.K, self.ncol
        sizes = [k.para.size for k in self.kids]
        out = np.zeros((K * C, sum(sizes)))
        for c, v in enumerate(self.vecs):
            d = np.asarray(v.diaghessgradpara())
            for j, k in enumerate(self.kids):
                out[c * K:(c + 1) * K, j * sizes[0] + (c if per_column(k) else 0)] = d[:, j]
        return out


class predictor(R.predictor):
    """one single-response predictor per column: mean N x C; variance N x C for a per-column likelihood or one fitted
    in an lpdfvec with a per-column child (each column's predictor has its own column's total diagonal)"""

    def __init__(self, lib, loglik):
        super().__init__(lib, loglik)
        self.percol = per_column(loglik) or getattr(loglik, "fitted_per_column", False)

    def var(self):
        return np.column_stack([p.var() for p in self.preds]) if self.percol else super().var()


class Reference(R.Reference):
    def loglik_gauss_multi(self, om, terms, Y, x, para_per_column=False):
        return (loglik_gauss_multi if para_per_column else R.loglik_gauss_multi)(self.lib, om, terms, Y, x)

    def logpr_gauss_multi(self, om, terms, ncol, para_per_column=False):
        return (logpr_gauss_multi if para_per_column else R.logpr_gauss_multi)(self.lib, om, terms, ncol)

    def lpdfvec(self, a, b):
        return lpdfvec(self.lib, a, b)

    def predictor(self, loglik):
        return predictor(self.lib, loglik)
