"""Posterior draws on the C3 model (bench.setup_model, synth_rows, N = 1M, K = 2000, terms-specialised kernels, one GPU).

The model is fitted briefly (one optcg(0.001, 100) of lpdfvec(logpr_gauss, loglik_gauss) at bench.setup_model's
hyper-parameters); then for S in {8, 64} a posterior_draws object is made and measured:
  solve_ms            warm solve(0.001, 100) from the fit's coefficients, median of three (one cold solve first)
  cg_iters_per_column the iterations each column took in that solve (the batched run lasts as long as its slowest column)
  ms_per_iter         from two no-stop solves (tol < 0) of 2 and 6 iterations; launches_per_iter likewise
  predict_ms          warm predict at 1M new points: basis build, one Phi.A with S columns, the N x S copy to the host
The GPU name and power limit are read in the same run; the result goes to --out as JSON."""
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
from outerbase_b200.binding import posterior_draws  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(0), "unknown"
    return name, power


def timed(lib, f):
    lib.synchronize()
    t0 = time.perf_counter()
    r = f()
    lib.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r06_posterior_draws.json"))
    ap.add_argument("--S", default="8,64")
    args = ap.parse_args()
    name, power = gpu_info()
    lib = obp.lib(0)
    lib.set_option("spec", 1)
    N = bench.N_TOTAL
    x = bench.synth_rows(0, N, bench.D)
    y = bench.wingweight(x)
    y = (y - y.mean()) / y.std()
    om, terms = bench.setup_model(lib)
    K = terms.shape[0]
    vec = lib.lpdfvec(lib.logpr_gauss(om, terms), lib.loglik_gauss(om, terms, y, x))
    vec.domarg = True
    fit_ms, _ = timed(lib, lambda: vec.optcg(0.001, 100))
    xs = bench.synth_rows(N, 2 * N, bench.D)  # new points
    res = {"workload": f"posterior draws on the C3 model, N={N} K={K}", "gpu": name, "power_limit": power,
           "fit": {"optcg_ms_cold": fit_ms, "cg_iters": vec.cg_iters}, "runs": []}
    for S in (int(s) for s in args.S.split(",")):
        dr = posterior_draws(lib, vec, S, seed=0)
        cold_ms, _ = timed(lib, lambda: dr.solve(0.001, 100))
        solves = sorted(timed(lib, lambda: dr.solve(0.001, 100))[0] for _ in range(3))
        iters = dr.cg_iters.tolist()
        assert np.all(np.isfinite(dr.coeff))
        per = {}
        for epochs in (2, 6):
            dr.solve(-1.0, epochs)  # warm this length once
            n0 = lib.launch_count()
            per[epochs] = (timed(lib, lambda: dr.solve(-1.0, epochs))[0], lib.launch_count() - n0)
        ms_per_iter = (per[6][0] - per[2][0]) / 4
        launches_per_iter = (per[6][1] - per[2][1]) / 4
        dr.solve(0.001, 100)
        dr.predict(xs)  # warm: the module for the new rows' object
        pred_ms = sorted(timed(lib, lambda: dr.predict(xs))[0] for _ in range(3))
        run = {"S": S, "solve_ms_cold": cold_ms, "solve_ms": solves[1], "solve_ms_all": solves, "cg_iters_per_column": iters,
               "cg_iters_max": max(iters), "ms_per_iter": ms_per_iter, "launches_per_iter": launches_per_iter,
               "predict_points": int(xs.shape[0]), "predict_ms": pred_ms[1], "predict_ms_all": pred_ms}
        res["runs"].append(run)
        print(json.dumps(run), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({"gpu": name, "power_limit": power, "out": args.out}))


if __name__ == "__main__":
    main()
