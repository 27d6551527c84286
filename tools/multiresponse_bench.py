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
The GPU name and power limit are read in the same run."""
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


def main():
    lib = obp.lib(0)
    lib.set_option("spec", 1)
    name, power = gpu_info()
    om, terms = bench.setup_model(lib)
    N, K = bench.N_TOTAL, terms.shape[0]
    x = bench.synth_rows(0, N, bench.D)
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
