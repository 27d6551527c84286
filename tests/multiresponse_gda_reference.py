"""loglik_gda_multi (include/outerbase_b200_multi_gda.h) written literally as its definition: C single-response
loglik_gda objects of a library (the CPU oracle in the tests), one per response column, and loops over them.

`Reference(lib)` extends the factories of tests/multiresponse_reference.py with `loglik_gda_multi`, so that
`fitting.obfit_multi(..., stage1=True)` runs on it as on the CUDA product.  The columns share both para entries and
dodiag; val, gradhyp and gradpara are the column sums in column order, grad is K x C, yhat is N x C and the Hessian
diagonals are stacked column by column."""
import math

import numpy as np

import multiresponse_reference as mr


def _sum2(x):
    """Armadillo's two-accumulator sum (np.cumsum adds strictly in order)."""
    s1 = float(np.cumsum(x[0::2])[-1]) if x.size > 0 else 0.0
    s2 = float(np.cumsum(x[1::2])[-1]) if x.size > 1 else 0.0
    return s1 + s2


def arma_var(x):
    """arma::var (op_var::direct_var) in its own operation order: what loglik_gda's default para0 is built from."""
    x = np.asarray(x, dtype=float)
    n = x.size
    if n < 2:
        return 0.0
    t = _sum2(x) / n - x
    m = 2 * (n // 2)
    a2 = np.cumsum(t[0:m:2] * t[0:m:2] + t[1:m:2] * t[1:m:2])[-1]
    a3 = np.cumsum(t[0:m:2] + t[1:m:2])[-1]
    if n % 2:
        a2 += t[-1] * t[-1]
        a3 += t[-1]
    return float((a2 - a3 * a3 / n) / (n - 1))


class loglik_gda_multi(mr._Multi):
    def __init__(self, lib, om, terms, Y, x):
        Y = np.asarray(Y, dtype=float)
        if Y.ndim != 2 or Y.shape[0] != np.asarray(x).shape[0] or Y.shape[1] == 0:
            raise ValueError("Y must be N x C with C >= 1 and one row per row of x")
        C = Y.shape[1]
        super().__init__([lib.loglik_gda(om, terms, Y[:, c], x) for c in range(C)], np.asarray(terms).shape[0])
        vs = 0.0
        for c in range(C):
            vs += arma_var(Y[:, c])
        self.para0 = np.array([0.5 * math.log(0.01 * (vs / C)), 0.0])
        self.paravar = np.array([4.0, 4.0])
        self.updatepara(self.para0)

    yhat = property(lambda s: np.column_stack([o.yhat for o in s.cols]))

    @property
    def dodiag(self):
        raise AttributeError("write-only")

    @dodiag.setter
    def dodiag(self, v):
        for o in self.cols:
            o.dodiag = v

    def diaghessgradpara(self):
        return np.vstack([o.diaghessgradpara() for o in self.cols])


class Reference(mr.Reference):
    def loglik_gda_multi(self, om, terms, Y, x):
        return loglik_gda_multi(self.lib, om, terms, Y, x)
