"""R-level drivers of the reference, re-hosted in Python over the C ABI (SURVEY 8f rank 1).

The reference keeps hyper-parameter learning in R (`R/outersupport.R`, `R/fitting.R`); R is
not available next to this library, so the same control flow lives here, statement for
statement, on top of the binding classes (`outerbase_b200.binding`), which work identically
over the CUDA product and over the CPU oracle -- that is how the parity tests run ONE driver
on both.  Nothing N-sized happens in this file: every objective evaluation is
`om.updatehyp -> logpdf.updateom (basis rebuild on the GPU) -> logpdf.optcg (CG on the GPU)`.

  BFGS_std      R/outersupport.R:30-176   line-searched BFGS with the reference's restart rules
  BFGS_lpdf     R/outersupport.R:195-204  (cgsteps / cgtol are accepted and NOT forwarded, as upstream: SURVEY A9.i)
  lpdfwrapper   R/outersupport.R:209-226  negated log-posterior and its gradient in (hyp, para)
  genknotlist   R/fitting.R:177-185       type-7 quantile knots
  getsteps      R/fitting.R:188-195
  obfit         R/fitting.R:27-137        both stages: loglik_gda on a subsample, then loglik_gauss on all rows
  obfit_gauss   R/fitting.R:100-136       the stage-2 loop alone, started from the constructor defaults
  obfit_multi                             obfit_gauss for C responses at the same inputs (no reference counterpart);
                                          stage1=True: obfit's two stages, stage 1 on loglik_gda_multi over one row
                                          subsample shared by the columns
  obpred        R/fitting.R:149-155
  obdraws                                 S joint posterior draws of a fitted model at new inputs (no reference
                                          counterpart)
  obsobol                                 Sobol first-order and total indices of a fitted model, exact from its
                                          coefficients, optionally the second-order indices of every input pair and
                                          the Shapley effects, and of S posterior draws (no reference counterpart)
"""
from __future__ import annotations

import math

import numpy as np

from .binding import gethyp, getpara, posterior_draws, sobol, sobol_pairs, sobol_shapley


def _flatten(parlist):
    keys = list(parlist.keys())
    return keys, np.concatenate([np.atleast_1d(np.asarray(parlist[k], dtype=float)) for k in keys])


def _relist(vec, parlist):
    out, pos = {}, 0
    for k, v in parlist.items():
        n = np.atleast_1d(np.asarray(v)).size
        out[k] = np.array(vec[pos:pos + n], dtype=float)
        pos += n
    return out


def _isna(v):
    return v is None or (isinstance(v, float) and math.isnan(v))


def BFGS_std(funcw, parlist, B=None, lr=0.1, verbose=0, **kw):
    """R/outersupport.R:30-176.  `funcw(parlist, **kw)` returns {"val": float, "gval": dict or None}."""
    c1, c2, numatte0 = 0.0001, 0.9, 5
    _, parv = _flatten(parlist)

    def gvec(optid):
        return None if optid["gval"] is None else _flatten(optid["gval"])[1]

    def wolfe(optid, step, dirc, go, valo, c2_):
        g = gvec(optid)
        w1 = (optid["val"] - valo) - c1 * step * float(np.sum(dirc * go))
        # gval = NULL (objective = Inf): R's sum(dirc * unlist(NULL)) is 0, not NA
        w2 = -(0.0 if g is None else float(np.sum(dirc * g))) + c2_ * float(np.sum(dirc * go))
        return w1, w2

    optid = funcw(_relist(parv, parlist), **kw)
    valo = optid["val"]
    go = gvec(optid)
    resetB = True
    if go is None or np.any(np.isnan(go)):
        raise RuntimeError("initial gradient was undefined, stopping.")
    if B is None:
        B = np.diag(1 / np.sqrt(go ** 2 + 0.001))
    else:
        B = np.array(B, dtype=float)
        resetB = False
    twice = False
    lr0 = lr00 = lr
    history = [dict(iter=0, obj=valo, wolfe1=None, wolfe2=None, lr=lr)]
    dirc = -B @ go
    k = 0
    for k in range(1, 101):
        dirc = -B @ go
        st = lr * dirc
        parvp = parv + st
        optid = funcw(_relist(parvp, parlist), **kw)
        wolfcond1, wolfcond2 = wolfe(optid, lr, dirc, go, valo, c2)
        numatte, lrlb, lrub, lrh = numatte0, 0.0, math.inf, lr
        optidh = optid
        while numatte > 0 and (_isna(wolfcond1) or _isna(wolfcond2) or wolfcond1 > 0 or wolfcond2 > 0):
            if _isna(wolfcond1) or _isna(wolfcond2) or wolfcond1 > 0:
                lrub = lrh
                lrh = 0.5 * (lrlb + lrub)
            else:
                lrlb = lrh
                lrh = 0.5 * (lrlb + lrub) if math.isfinite(lrub) else 2 * lrlb
            parvp = parv + lrh * dirc
            optidh = funcw(_relist(parvp, parlist), **kw)
            wolfcond1, wolfcond2 = wolfe(optidh, lrh, dirc, go, valo, c2)
            numatte -= 1
        if _isna(wolfcond1) or _isna(wolfcond2):
            raise RuntimeError("something is very wrong... stuck on NAs")
        if wolfcond1 > 0:
            if resetB:
                c2 = c2 ** 0.5
                lr0 = lr0 / 10
                lr = lr0
            if lr0 < lr00 / (10 ** 2 + 1):
                break
            optid = funcw(_relist(parv, parlist), **kw)  # do not feed it extra info
            valo = optid["val"]
            go = gvec(optid)
            B = np.diag(1 / np.sqrt(0.001 + go ** 2))
            resetB = True
            history.append(dict(iter=k, obj=None, wolfe1=None, wolfe2=None, lr=lr))
            if verbose > 0:
                print("restarted hessian")
        else:
            if lr != lrh:
                lr = lrh
                st = parvp - parv
                parv = parvp
                optid = optidh
            else:
                parv = parvp
            if k > 2 and float(np.sum(st * go)) > -go.size / 4 and twice:
                break
            elif k > 2 and float(np.sum(st * go)) > -go.size / 4:
                twice = True
            goo = go
            valo = optid["val"]
            go = gvec(optid)
            yv = go - goo
            history.append(dict(iter=k, obj=valo, wolfe1=wolfcond1, wolfe2=wolfcond2, lr=lr))
            if verbose > 1:
                print(history[-1])
            if resetB:
                B = float(np.sum(st * yv)) / float(np.sum(yv * yv)) * np.eye(parv.size)
                resetB = False
            cvh = 1 / float(np.sum(st * yv))
            M1 = np.eye(go.size) - cvh * np.outer(st, yv)
            B = M1 @ B @ M1.T + cvh * np.outer(st, st)
            lr = lr ** 0.9  # drift toward 1
    optid = funcw(_relist(parv, parlist), **kw)  # finish by evaluating
    if verbose > 0:
        print(f"num iter: {k}  obj start: {history[0]['obj']}  obj end: {optid['val']}\nfinal learning rate: {lr}")
    return dict(parlist=_relist(parv, parlist), B=B, lr=lr, optid=optid, history=history, iters=k)


def lpdfwrapper(parlist, om, logpdf, newt=False, cgsteps=100, cgtol=0.001):
    """.lpdfwrapper, R/outersupport.R:209-226: the NEGATED log-posterior in (hyp, para) and its gradient."""
    regpara = logpdf.paralpdf(parlist["para"])
    reghyp = om.hyplpdf(parlist["hyp"])
    if math.isfinite(regpara) and math.isfinite(reghyp):
        om.updatehyp(parlist["hyp"])
        logpdf.updateom()
        logpdf.updatepara(parlist["para"])
        if newt:
            logpdf.optnewton()  # :218 -- needs a likelihood with a full Hessian (loglik_std)
        else:
            logpdf.optcg(cgtol, cgsteps)
        gval = dict(parlist)
        gval["hyp"] = -np.asarray(logpdf.gradhyp) - np.asarray(om.hyplpdf_grad(parlist["hyp"]))
        gval["para"] = -np.asarray(logpdf.gradpara) - np.asarray(logpdf.paralpdf_grad(parlist["para"]))
        return dict(val=-logpdf.val - reghyp - regpara, gval=gval)
    return dict(val=math.inf, gval=None)


def BFGS_lpdf(om, logpdf, parlist=None, newt=False, cgsteps=100, cgtol=0.001, **kw):
    """R/outersupport.R:195-204.  om and logpdf are left at the optimal parameters."""
    parlist = dict(parlist or {})
    if parlist.get("hyp") is None:
        parlist["hyp"] = gethyp(om)
    if parlist.get("para") is None:
        parlist["para"] = getpara(logpdf)
    parlist = {"hyp": np.asarray(parlist["hyp"], dtype=float), "para": np.asarray(parlist["para"], dtype=float)}
    lpdfwrapper(parlist, om, logpdf, newt=newt)  # start by aligning para with
    # upstream never forwards cgsteps / cgtol to the wrapper (SURVEY A9.i): every evaluation runs optcg(0.001, 100)
    return BFGS_std(lpdfwrapper, parlist, om=om, newt=newt, logpdf=logpdf, **kw)


def genknotlist(bassize, x):
    """.genknotlist, R/fitting.R:177-185 (R's default type-7 quantile = numpy's default 'linear')."""
    x = np.asarray(x)
    out = []
    for k in range(x.shape[1]):
        b = int(bassize[k])
        out.append(np.quantile(x[:, k], np.linspace(0, 1, b) * b / (b + 1) + 0.5 / (b + 1)))
    return out


# bounds of the covariance classes (covfuncs.cpp:109-110, 193-194, 281-282)
_COV_BOUNDS = {"mat25": (0.0, 1.0), "mat25pow": (0.0, 1.0), "mat25ang": (0.0, 6.283185)}


def checkcov(covname, x):
    """.checkcov, R/fitting.R:158-175: the column must lie inside the covariance's bounds and span 1/20 of them."""
    if covname not in _COV_BOUNDS:
        raise ValueError("\n covariances must be from listcov()")
    lo, hi = _COV_BOUNDS[covname]
    x = np.asarray(x)
    if x.min() < lo or x.max() > hi:
        raise ValueError(f"\n x ranges exceed limits of covariance functions \n the limits are between {lo} and {hi} \n try rescaling")
    if x.max() - x.min() < (hi - lo) / 20:
        raise ValueError(f"\n x are too small for ranges\n the limits are between {lo} and {hi} \n try rescaling")


def getsteps(numb, sampsize, sigtonoiseratio=1e-3, tol=0.001):
    """.getsteps, R/fitting.R:188-195 (its result is unused upstream: SURVEY A9.i)."""
    r = math.sqrt(numb / sampsize)
    kapp = 1000.0 if r == 1.0 else min(1000.0, (1 + r) ** 2 / (1 - r) ** 2)  # R: x/0 = Inf, min(1000, Inf) = 1000
    iterest = 0.5 * math.sqrt(kapp) * math.log(2 * sampsize * sigtonoiseratio / tol)
    return math.ceil(2 * iterest)


def obfit_gauss(lib, x, y, numb=100, covnames=None, hyp=None, numberopts=2, verbose=0, knots=40):
    """Stage 2 of obfit (R/fitting.R:100-136) started from the constructor defaults instead of the
    loglik_gda warm start of stage 1 (R/fitting.R:76-98, SURVEY 8f rank 2): standardise y, 40 quantile knots,
    `numberopts` rounds of selectterms + BFGS_lpdf on lpdfvec(logpr_gauss, loglik_gauss) with domarg."""
    x = np.asfortranarray(np.asarray(x, dtype=float))
    y = np.asarray(y, dtype=float)
    if x.shape[0] != y.size:
        raise ValueError("x and y dims do not align")
    d = x.shape[1]
    if numb < 2 * d:
        raise ValueError("number of basis functions should be less than twice the dimension")
    y_cent, y_sca = float(y.mean()), float(y.std(ddof=1))
    ys = (y - y_cent) / y_sca
    om = lib.outermod()
    om.setcovfs(list(covnames) if covnames is not None else ["mat25pow"] * d)
    if hyp is not None and len(hyp) == gethyp(om).size:
        om.updatehyp(hyp)
    om.setknot(genknotlist([knots] * d, x))
    terms = om.selectterms(numb)
    logpr = lib.logpr_gauss(om, terms)
    loglik = lib.loglik_gauss(om, terms, ys, x)
    logpdf = lib.lpdfvec(logpr, loglik)  # prior first (R/fitting.R:86,107)
    logpdf.domarg = True
    optinfo = dict(B=None, lr=0.2)
    for k in range(numberopts):
        terms = om.selectterms(numb)
        logpdf.updateterms(terms)
        optinfo = BFGS_lpdf(om, logpdf, verbose=verbose, B=optinfo["B"], lr=optinfo["lr"] / 2)
    return dict(y_cent=y_cent, y_sca=y_sca, om=om, terms=terms, logpdf=logpdf, loglik=loglik, logpr=logpr,
                predobj=lib.predictor(loglik), optinfo=optinfo)


def obfit(lib, x, y, numb=100, verbose=0, covnames=None, hyp=None, numberopts=2, nthreads=None, seed=0):
    """obfit, R/fitting.R:27-137.  The row subsample of stage 1 is drawn with numpy's generator (`seed`) where the
    reference uses R's `sample`; everything else follows the R code line by line."""
    x = np.asfortranarray(np.asarray(x, dtype=float))
    y = np.asarray(y, dtype=float)
    n, d = x.shape
    if n != y.size:
        raise ValueError("x and y dims do not align")
    if n < d:
        raise ValueError("dimension larger than sample size has not been tested")
    if d == 1:
        raise ValueError("dimension must be larger than 1")
    if d == 2:
        raise ValueError("dimension 2 has not been tested")
    if numb < 2 * d:
        raise ValueError("number of basis functions should be less than twice the dimension")
    if numb > 100000:
        raise ValueError("number of basis functions is beyond testing")
    # R/fitting.R:33 stops for n > 1e6 (SURVEY A9.ii); the GPU path has no such limit
    y_cent, y_sca = float(y.mean()), float(y.std(ddof=1))
    ys = (y - y_cent) / y_sca
    covnames = list(covnames) if covnames is not None else ["mat25pow"] * d
    if len(covnames) != d:
        raise ValueError("cov names must be same size as columns in x")
    for k in range(d):  # R/fitting.R:68
        checkcov(covnames[k], x[:, k])
    om = lib.outermod()
    om.setcovfs(covnames)
    if hyp is not None and len(hyp) == gethyp(om).size:
        om.updatehyp(hyp)
    om.setknot(genknotlist([40] * d, x))  # 40 knot point for each dim
    # ---- stage 1: few terms, row subsample, loglik_gda (R/fitting.R:76-98)
    numbr = min(n // 2, numb, 80 * d)
    terms = om.selectterms(numbr)
    ssr = min(n, 3 * numbr)
    logpr = lib.logpr_gauss(om, terms)
    subset = np.sort(np.random.default_rng(seed).choice(n, size=ssr, replace=False))
    loglik = lib.loglik_gda(om, terms, ys[subset], np.asfortranarray(x[subset]))
    loglik.dodiag = True
    logpdf = lib.lpdfvec(logpr, loglik)
    if nthreads is not None:
        logpdf.setnthreads(int(math.ceil(nthreads)))
    if verbose > 0:
        print("doing partial optimization")
    optinfo = BFGS_lpdf(om, logpdf, verbose=verbose, cgsteps=100)
    # ---- stage 2: all rows, loglik_gauss (R/fitting.R:100-136)
    terms = om.selectterms(numb)
    bassize = np.ceil(np.maximum(16, np.minimum(70, 2 * np.asarray(terms).max(axis=0)))).astype(int)
    om.setknot(genknotlist(bassize, x))
    loglik_faster = lib.loglik_gauss(om, terms, ys, x)
    logpdf_faster = lib.lpdfvec(logpr, loglik_faster)
    logpdf_faster.domarg = True
    B = np.asarray(optinfo["B"])[:-1, :-1]          # one fewer para, so we strip that one off
    B = ssr / n * B                                  # decrease scale
    logpdf_faster.updatepara(getpara(logpdf)[:2])
    if nthreads is not None:
        logpdf_faster.setnthreads(int(math.ceil(nthreads)))
    lr = optinfo["lr"]
    for k in range(numberopts):
        if verbose > 0:
            print("doing optimization", k + 1)
        terms = om.selectterms(numb)
        logpdf_faster.updateterms(terms)
        optinfo = BFGS_lpdf(om, logpdf_faster, verbose=verbose, B=B, lr=lr / 2,
                            cgsteps=getsteps(numb, n, float(np.var(ys, ddof=1)) / math.exp(2 * getpara(logpdf_faster)[1])))
        B, lr = optinfo["B"], optinfo["lr"]
    return dict(y_cent=y_cent, y_sca=y_sca, om=om, terms=terms, logpdf=logpdf_faster, loglik=loglik_faster, logpr=logpr,
                predobj=lib.predictor(loglik_faster), optinfo=optinfo, stage1=dict(logpdf=logpdf, loglik=loglik, rows=subset))


def obfit_multi(lib, x, Y, numb=100, covnames=None, hyp=None, numberopts=2, verbose=0, knots=40, para_per_column=False,
                stage1=False, seed=0):
    """obfit_gauss for C responses observed at the same inputs (Y is N x C): each column standardised on its own, then
    the same stage-2 loop on lpdfvec(logpr_gauss_multi, loglik_gauss_multi) with domarg -- one basis, one terms table,
    shared hyper-parameters and para, one independent CG per column inside every objective evaluation.
    para_per_column: each column gets its own noise scale and coefficient scale (para has 2 C entries), for outputs
    whose signal-to-noise ratios differ; the hyper-parameters stay shared.
    stage1: obfit's two stages (R/fitting.R:27-137) instead of stage 2 alone.  Stage 1 fits the hyper-parameters on
    lpdfvec(logpr_gauss_multi, loglik_gda_multi) over ONE seeded subsample of at most 3 numbr rows shared by all columns
    (`knots` is then unused: 40 knots, as obfit); stage 2 starts from its hyper-parameters, its two shared para entries
    (each repeated C times with para_per_column) and its BFGS metric scaled by ssr / n (none with para_per_column: the
    stage-1 metric has no per-column para block).  With C = 1 this is obfit itself."""
    x = np.asfortranarray(np.asarray(x, dtype=float))
    Y = np.asarray(Y, dtype=float)
    if Y.ndim != 2:
        raise ValueError("Y must be N x C")
    if x.shape[0] != Y.shape[0]:
        raise ValueError("x and Y dims do not align")
    n, d = x.shape
    C = Y.shape[1]
    if stage1:  # obfit's checks, R/fitting.R:30-68
        if n < d:
            raise ValueError("dimension larger than sample size has not been tested")
        if d == 1:
            raise ValueError("dimension must be larger than 1")
        if d == 2:
            raise ValueError("dimension 2 has not been tested")
    if numb < 2 * d:
        raise ValueError("number of basis functions should be less than twice the dimension")
    if stage1 and numb > 100000:
        raise ValueError("number of basis functions is beyond testing")
    y_cent, y_sca = Y.mean(axis=0), Y.std(axis=0, ddof=1)
    Ys = np.asfortranarray((Y - y_cent) / y_sca)
    covnames = list(covnames) if covnames is not None else ["mat25pow"] * d
    if stage1:
        if len(covnames) != d:
            raise ValueError("cov names must be same size as columns in x")
        for k in range(d):
            checkcov(covnames[k], x[:, k])
    om = lib.outermod()
    om.setcovfs(covnames)
    if hyp is not None and len(hyp) == gethyp(om).size:
        om.updatehyp(hyp)
    percol = {"para_per_column": True} if para_per_column else {}
    if not stage1:
        om.setknot(genknotlist([knots] * d, x))
        terms = om.selectterms(numb)
        logpr = lib.logpr_gauss_multi(om, terms, C, **percol)
        loglik = lib.loglik_gauss_multi(om, terms, Ys, x, **percol)
        logpdf = lib.lpdfvec(logpr, loglik)  # prior first, as obfit_gauss
        logpdf.domarg = True
        optinfo = dict(B=None, lr=0.2)
        for k in range(numberopts):
            terms = om.selectterms(numb)
            logpdf.updateterms(terms)
            optinfo = BFGS_lpdf(om, logpdf, verbose=verbose, B=optinfo["B"], lr=optinfo["lr"] / 2)
        return dict(y_cent=y_cent, y_sca=y_sca, om=om, terms=terms, logpdf=logpdf, loglik=loglik, logpr=logpr,
                    predobj=lib.predictor(loglik), optinfo=optinfo)
    om.setknot(genknotlist([40] * d, x))
    # ---- stage 1: few terms, one row subsample for every column, loglik_gda_multi (R/fitting.R:76-98)
    numbr = min(n // 2, numb, 80 * d)
    terms = om.selectterms(numbr)
    ssr = min(n, 3 * numbr)
    logpr = lib.logpr_gauss_multi(om, terms, C)
    subset = np.sort(np.random.default_rng(seed).choice(n, size=ssr, replace=False))
    loglik = lib.loglik_gda_multi(om, terms, np.asfortranarray(Ys[subset]), np.asfortranarray(x[subset]))
    loglik.dodiag = True
    logpdf = lib.lpdfvec(logpr, loglik)
    if verbose > 0:
        print("doing partial optimization")
    optinfo = BFGS_lpdf(om, logpdf, verbose=verbose, cgsteps=100)
    # ---- stage 2: all rows, loglik_gauss_multi (R/fitting.R:100-136)
    terms = om.selectterms(numb)
    bassize = np.ceil(np.maximum(16, np.minimum(70, 2 * np.asarray(terms).max(axis=0)))).astype(int)
    om.setknot(genknotlist(bassize, x))
    if para_per_column:
        logpr = lib.logpr_gauss_multi(om, terms, C, **percol)
    loglik_faster = lib.loglik_gauss_multi(om, terms, Ys, x, **percol)
    logpdf_faster = lib.lpdfvec(logpr, loglik_faster)
    logpdf_faster.domarg = True
    para = np.asarray(getpara(logpdf))[:2]
    if para_per_column:
        B, para = None, np.repeat(para, C)
    else:
        B = np.asarray(optinfo["B"])[:-1, :-1]      # one fewer para, so we strip that one off
        B = ssr / n * B                              # decrease scale
    logpdf_faster.updatepara(para)
    lr = optinfo["lr"]
    for k in range(numberopts):
        if verbose > 0:
            print("doing optimization", k + 1)
        terms = om.selectterms(numb)
        logpdf_faster.updateterms(terms)
        optinfo = BFGS_lpdf(om, logpdf_faster, verbose=verbose, B=B, lr=lr / 2)
        B, lr = optinfo["B"], optinfo["lr"]
    return dict(y_cent=y_cent, y_sca=y_sca, om=om, terms=terms, logpdf=logpdf_faster, loglik=loglik_faster, logpr=logpr,
                predobj=lib.predictor(loglik_faster), optinfo=optinfo, stage1=dict(logpdf=logpdf, loglik=loglik, rows=subset))


def obpred(obmodel, x):
    """R/fitting.R:149-155.  A model of obfit_multi gives an N x C mean and an N x C variance: the shared variance
    (or, with para per column, each column's own) scaled by each column's y_sca^2."""
    obmodel["predobj"].update(np.asfortranarray(np.asarray(x, dtype=float)))
    if np.ndim(obmodel["y_sca"]):
        var = obmodel["predobj"].var()
        var = var * obmodel["y_sca"] ** 2 if var.ndim == 2 else np.outer(var, obmodel["y_sca"] ** 2)
        return dict(mean=obmodel["y_cent"] + obmodel["y_sca"] * obmodel["predobj"].mean(), var=var)
    return dict(mean=obmodel["y_cent"] + obmodel["y_sca"] * obmodel["predobj"].mean(),
                var=obmodel["y_sca"] ** 2 * obmodel["predobj"].var())


def obdraws(obmodel, x, S=64, seed=0, tol=0.001, maxepch=100):
    """S joint posterior draws of the latent function at the rows of x (N x S, in y's units: y_cent + y_sca f) for a model
    of obfit / obfit_gauss, conditional on its hyper-parameters, terms and para (posterior_draws: perturb-and-MAP, exact
    at CG convergence; tol is the CG tolerance of the S solves).  Observation noise at x is not included."""
    draws = posterior_draws(obmodel["logpdf"]._lib, obmodel["logpdf"], S, seed).solve(tol, maxepch)
    return obmodel["y_cent"] + obmodel["y_sca"] * draws.predict(np.asfortranarray(np.asarray(x, dtype=float)))


def _indices(r):
    """first / var and total / var; a column whose variance is 0 gets NaN indices"""
    var = np.asarray(r["var"], dtype=float)
    with np.errstate(divide="ignore", invalid="ignore"):
        first = np.where(var != 0, r["first"] / np.where(var != 0, var, 1.0), np.nan)
        total = np.where(var != 0, r["total"] / np.where(var != 0, var, 1.0), np.nan)
    return first, total


def _pair_indices(r):
    """second / var, closed = (first_l + first_m + second_lm) / var and supset / var (d x d or d x d x B, NaN on the
    diagonal); a column whose variance is 0 gets NaN indices"""
    var = np.asarray(r["var"], dtype=float)
    f = np.asarray(r["first"], dtype=float)
    closed = f[:, None] + f[None, :] + r["second"]
    den = np.where(var != 0, var, 1.0)
    with np.errstate(divide="ignore", invalid="ignore"):
        return {k: np.where(var != 0, v / den, np.nan) for k, v in (("second", r["second"]), ("closed", closed),
                                                                    ("supset", r["supset"]))}


def _shapley_indices(r):
    """shapley / var (d or d x B, adding up to 1); a column whose variance is 0 gets NaN"""
    var = np.asarray(r["var"], dtype=float)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(var != 0, r["shapley"] / np.where(var != 0, var, 1.0), np.nan)


def obsobol(obmodel, x, S=0, seed=0, tol=0.001, maxepch=100, second=False, shapley=False):
    """Sobol indices of the latent function of a model of obfit / obfit_gauss / obfit_multi under the product of the
    empirical marginals of x's columns (binding.sobol: exact quadratic forms in the fitted coefficients).  Returns first and
    total (the first-order and total indices, d or d x C), var (Var f in y's units, y_sca^2 var) and mean (y_cent +
    y_sca E f).  second=True adds, from binding.sobol_pairs, the input-pair indices second (pure second-order), closed
    (first_l + first_m + second_lm) and supset (superset importance), each d x d or d x d x C with NaN on the diagonal.
    shapley=True adds, from binding.sobol_shapley, shapley: the Shapley effects over the variance (d or d x C), which
    add up to 1 and lie between first and total.
    S > 0 adds `draws`: the same keys for each of S posterior draws (d x S, d x d x S, S), conditional on the
    hyper-parameters, terms and para (posterior_draws; single-response models only)."""
    logpdf = obmodel["logpdf"]
    lib, om, terms = logpdf._lib, obmodel["om"], obmodel["terms"]
    x = np.asfortranarray(np.asarray(x, dtype=float))
    y_cent, y_sca = obmodel["y_cent"], obmodel["y_sca"]
    forms = sobol_pairs if second else sobol

    def indices(coeff):
        r = forms(lib, om, terms, coeff, x)
        first, total = _indices(r)
        out = dict(first=first, total=total, var=y_sca ** 2 * r["var"], mean=y_cent + y_sca * r["mean"])
        if second:
            out.update(_pair_indices(r))
        if shapley:
            out["shapley"] = _shapley_indices(sobol_shapley(lib, om, terms, coeff, x))
        return out

    out = indices(logpdf.coeff)
    if S > 0:
        out["draws"] = indices(posterior_draws(lib, logpdf, S, seed).solve(tol, maxepch).coeff)
    return out
