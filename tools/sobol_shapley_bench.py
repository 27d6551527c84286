"""Shapley effects (binding.sobol_shapley) on the benchmark's tables, one GPU.

Workloads (those of tools/sobol_pairs_bench.py, and a shape check at the largest d):
  c3_B1, c3_B64   the C3 table (bench.setup_model: d = 10, K = 2000) with X_q = the 1M training rows (bench.synth_rows)
  c4_B64          the C4-size table (bench.config_model "c4share": d = 20, K = 4000) on 125k rows
  d77_B64         d = 77 (five knots per dimension), K = 100, seeded uniform X_q of 20k rows: the one-CTA-per-SM variant
Coefficients are seeded normals scaled by 1 / (1 + level sum); the forms do not depend on their values.
Recorded per workload:
  call_ms            warm wall time of the whole call (basis build of X_q, both moment stages, the first-order and
                     total forms, the Shapley forms, the copies), ended by a device synchronise; median of three after
                     one cold call; sobol_call_ms the same for binding.sobol, in the same run
  kernels_us         device time of each kernel in one further call, from torch.profiler in a run of its own
  shapley_flop       per term pair (K (K + 1) / 2 of them) 5 d n FP64 operations to form the d factors over the
                     n = max(1, ceil(d / 2)) nodes and 2 d B in the contraction: an operation count of the algorithm, not
                     of the instructions the kernel issues
  shapley_tflops     shapley_flop over the Shapley kernel's device time, and its share of the FP64 peak measured in the
                     same run (Library.fp64_peak: DFMA, the same pipe and rate as DMMA, DESIGN §3.3b)
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
from outerbase_b200.binding import sobol, sobol_shapley  # noqa: E402


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


def kernel_times(f):
    """device microseconds per kernel name over one call of f"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        f()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        if us and any(t in e.key for t in ("sobol_", "colsum_partials", "basis_build", "basescale")):
            out[e.key] = {"us": float(us), "count": int(e.count)}
    return out


def d77_model(lib):
    rng = np.random.default_rng(77)
    om = lib.outermod()
    om.setcovfs([("mat25", "mat25pow", "mat25ang")[l % 3] for l in range(77)])
    om.setknot([np.sort(rng.uniform(0.02, 0.98, size=5)) for _ in range(77)])
    return om, om.selectterms(100), np.asfortranarray(rng.uniform(size=(20_000, 77)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(REPO / "profiles" / "r09_sobol_shapley.json"))
    args = ap.parse_args()
    name, power = gpu_info()
    lib = obp.lib(0)
    peak = lib.fp64_peak()
    res = {"gpu": name, "power_limit": power, "fp64_peak_tflops": peak, "runs": []}
    om3, t3 = bench.setup_model(lib)
    x3 = bench.synth_rows(0, bench.N_TOTAL, bench.D)
    om4, t4 = bench.config_model(lib, "c4share")
    x4 = bench.config_rows("c4share", 0, 125_000)
    om7, t7, x7 = d77_model(lib)
    for tag, om, terms, xq, B in (("c3_B1", om3, t3, x3, 1), ("c3_B64", om3, t3, x3, 64), ("c4_B64", om4, t4, x4, 64),
                                  ("d77_B64", om7, t7, x7, 64)):
        K, d = terms.shape
        rng = np.random.default_rng(B)
        coeff = np.asfortranarray(rng.normal(size=(K, B)) / (1 + terms.sum(axis=1))[:, None])
        call = lambda: sobol_shapley(lib, om, terms, coeff, xq)  # noqa: E731
        cold_ms, r = timed(lib, call)
        calls = sorted(timed(lib, call)[0] for _ in range(3))
        base = sorted(timed(lib, lambda: sobol(lib, om, terms, coeff, xq))[0] for _ in range(3))
        assert np.all(np.isfinite(r["var"])) and np.all(r["var"] > 0)
        kt = kernel_times(call)
        shap_us = sum(v["us"] for k, v in kt.items() if "sobol_shapley" in k)
        forms_us = sum(v["us"] for k, v in kt.items() if "sobol_forms" in k)
        build_us = sum(v["us"] for k, v in kt.items() if "basis_build" in k or "basescale" in k)
        moments_us = sum(v["us"] for k, v in kt.items() if "sobol_moments" in k)
        n = max(1, (d + 1) // 2)
        npairs = K * (K + 1) / 2
        flop_form, flop_mma = 5.0 * d * n * npairs, 2.0 * d * B * npairs
        flop = flop_form + flop_mma
        sh = r["shapley"][:, 0] / r["var"][0]
        run = {"workload": tag, "K": K, "d": d, "B": B, "nodes": n, "nq": int(xq.shape[0]), "call_ms_cold": cold_ms,
               "call_ms": calls[1], "call_ms_all": calls, "sobol_call_ms": base[1], "kernels_us": kt,
               "basis_build_us": build_us, "moments_us": moments_us, "forms_us": forms_us, "shapley_us": shap_us,
               "shapley_flop_form": flop_form, "shapley_flop_contraction": flop_mma, "shapley_flop": flop,
               "shapley_tflops": flop / (shap_us * 1e-6) / 1e12 if shap_us else None,
               "shapley_frac_of_fp64_peak": flop / (shap_us * 1e-6) / 1e12 / peak if shap_us else None,
               "shapley_sum_minus_1": float(sh.sum() - 1.0)}
        res["runs"].append(run)
        print(json.dumps(run), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({"gpu": name, "power_limit": power, "out": args.out}))


if __name__ == "__main__":
    main()
