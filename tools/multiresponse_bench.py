"""Multi-response fit on the C3 model (bench.setup_model, synth_rows, N = 1M, K = 2000, one B200): C seeded responses
(the wing-weight-style response plus a column-dependent smooth term) fitted as ONE lpdfvec(logpr_gauss_multi,
loglik_gauss_multi), against the same C fits run one after another with single-response objects in the same process.
Prints one JSON line per C in {8, 64}:
  optcg_ms / cg_iters_per_column   warm optcg(0.001, 100) from zero coefficients, and the iteration spread (the batched
                                   run lasts as long as its slowest column)
  ms_per_iter / launches_per_iter  from two no-stop runs (tol < 0) of 2 and 6 iterations
  bfgs_eval_ms                     one BFGS objective evaluation: updatehyp -> updateom -> optcg (fitting.lpdfwrapper)
  separate_*                       the C single-response fits one after another: total with object construction,
                                   and the optcg of each new object
The GPU name and power limit are read in the same run.

--para-per-column compares the shared form with the per-column one (each column its own noise scale and coefficient
scale) instead: for each C, both objects are built once and measured alternately, three rounds each, so that both see
the same clocks; one JSON line per C with, per form, every round's ms_per_iter, launches_per_iter and bfgs_eval_ms (no
separate fits)."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
import torch  # noqa: E402

import bench  # noqa: E402
import outerbase_b200 as obp  # noqa: E402
from outerbase_b200 import fitting  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def responses(x, C):
    base = bench.wingweight(x)
    base = (base - base.mean()) / base.std()
    Y = np.empty((x.shape[0], C), order="F")
    for c in range(C):
        Y[:, c] = (1 + 0.5 * np.sin(1.7 * c)) * base + 0.3 * np.cos(np.pi * (1 + c % 7) * x[:, c % x.shape[1]])
    return Y


def timed(lib, f):
    lib.synchronize()
    t0 = time.perf_counter()
    r = f()
    lib.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def percol_main(lib, name, power, om, terms, x, N, K):
    for C in (8, 64):
        Y = responses(x, C)
        vecs = {}
        for form, pc in (("shared", False), ("per_column", True)):
            vec = lib.lpdfvec(lib.logpr_gauss_multi(om, terms, C, para_per_column=pc),
                              lib.loglik_gauss_multi(om, terms, Y, x, para_per_column=pc))
            vec.domarg = True
            vec.optcg(0.001, 100)  # warm: module compilation, programs, buffers
            vecs[form] = (vec, vec.coeff.copy(), dict(hyp=np.array(om.gethyp()), para=np.array(vec.para)))
        rounds = {f: dict(ms_per_iter=[], launches_per_iter=[], bfgs_eval_ms=[]) for f in vecs}
        for _ in range(3):
            for form, (vec, coeff, parlist) in vecs.items():
                per = []
                for ep in (2, 6):
                    vec.set_coeff(np.zeros(K * C))
                    n0 = lib.launch_count()
                    ms, _ = timed(lib, lambda: vec.optcg(-1.0, ep))
                    per.append((ms, lib.launch_count() - n0))
                rounds[form]["ms_per_iter"].append(round((per[1][0] - per[0][0]) / 4, 3))
                rounds[form]["launches_per_iter"].append((per[1][1] - per[0][1]) / 4)
                vec.set_coeff(coeff)
                ms, _ = timed(lib, lambda: fitting.lpdfwrapper(parlist, om, vec))
                rounds[form]["bfgs_eval_ms"].append(round(ms, 2))
        out = {"workload": f"multi-response optcg on the C3 model, N={N} K={K} C={C}, shared vs per-column para",
               "gpu": name, "power_limit": power}
        for form, r in rounds.items():
            out[form] = dict(r, cg_iters_per_column=vecs[form][0].cg_iters_per_column.tolist(),
                             ms_per_iter_median=float(np.median(r["ms_per_iter"])),
                             bfgs_eval_ms_median=float(np.median(r["bfgs_eval_ms"])))
        print(json.dumps(out), flush=True)
        del vecs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--para-per-column", action="store_true", help="shared against per-column para, alternately")
    args = ap.parse_args()
    lib = obp.lib(0)
    lib.set_option("spec", 1)
    name, power = gpu_info()
    om, terms = bench.setup_model(lib)
    N, K = bench.N_TOTAL, terms.shape[0]
    x = bench.synth_rows(0, N, bench.D)
    if args.para_per_column:
        return percol_main(lib, name, power, om, terms, x, N, K)
    for C in (8, 64):
        Y = responses(x, C)
        lk = lib.loglik_gauss_multi(om, terms, Y, x)
        vec = lib.lpdfvec(lib.logpr_gauss_multi(om, terms, C), lk)
        vec.domarg = True
        vec.optcg(0.001, 100)  # warm: module compilation, programs, buffers
        vec.set_coeff(np.zeros(K * C))
        optcg_ms, _ = timed(lib, lambda: vec.optcg(0.001, 100))
        iters = vec.cg_iters_per_column
        coeff = vec.coeff.copy()
        per = []
        for ep in (2, 6):
            vec.set_coeff(np.zeros(K * C))
            n0 = lib.launch_count()
            ms, _ = timed(lib, lambda: vec.optcg(-1.0, ep))
            per.append((ms, lib.launch_count() - n0))
        ms_it, launch_it = (per[1][0] - per[0][0]) / 4, (per[1][1] - per[0][1]) / 4
        vec.set_coeff(coeff)
        parlist = dict(hyp=np.array(om.gethyp()), para=np.array(vec.para))
        bfgs_ms, _ = timed(lib, lambda: fitting.lpdfwrapper(parlist, om, vec))
        del vec, lk
        # the same C fits, one single-response fit after another
        sep_total, sep_optcg, sep_iters = 0.0, 0.0, []
        for c in range(C):
            t0 = time.perf_counter()
            lk1 = lib.loglik_gauss(om, terms, Y[:, c], x)
            v1 = lib.lpdfvec(lib.logpr_gauss(om, terms), lk1)
            v1.domarg = True
            v1.updatepara(parlist["para"])
            ms, _ = timed(lib, lambda: v1.optcg(0.001, 100))
            sep_total += (time.perf_counter() - t0) * 1e3
            sep_optcg += ms
            sep_iters.append(v1.cg_iters)
            del v1, lk1
        print(json.dumps({
            "workload": f"multi-response optcg on the C3 model, N={N} K={K} C={C}", "gpu": name, "power_limit": power,
            "optcg_ms": round(optcg_ms, 2), "cg_iters_per_column": iters.tolist(),
            "cg_iters_min_median_max": [int(iters.min()), float(np.median(iters)), int(iters.max())],
            "ms_per_iter": round(ms_it, 3), "launches_per_iter": launch_it, "bfgs_eval_ms": round(bfgs_ms, 2),
            "separate_fits_total_ms": round(sep_total, 2), "separate_optcg_sum_ms": round(sep_optcg, 2),
            "separate_cg_iters": sep_iters,
            "separate_iters_match": sep_iters == iters.tolist()}), flush=True)


if __name__ == "__main__":
    main()
