#!/usr/bin/env python
"""bench.py -- Phi a + Phi^T r matvec pairs/s of the outerbase hot path (BASELINE.json metric).

Workload (config C3 of BASELINE.json): wing-weight-style d=10 inputs, N = 1,000,000 rows in
total, K = 2000 terms from selectterms, `mat25pow` covariances with 40 quantile knots per
dimension, spread hyper-parameters.  With --gpus G the N rows are sharded over G ranks
(strong scaling) and every Phi^T r ends in one NCCL allreduce of K doubles.

A "step" is one CG iteration's worth of the path (src/fit.cpp:71-85): two (Phi a, Phi^T r)
pairs.  `value` is pairs/s with every operand resident in HBM (device-pointer C ABI), timed
with CUDA events on the library's stream, max over ranks.  `e2e` is the same metric through
the reference-facing calls outerbase::mm / outerbase::tmm with HOST buffers (coefficients and
residuals copied in, results copied out, every call).  `--impl reference` times the REFERENCE'S OWN
code on the host cores: oracle/_ref/libob_ref.so, the unmodified linalg/modandbase sources compiled
against the Armadillo-subset shim (kind "reference"); only where that library is absent the CPU
oracle's restatement (kind "port").

`--config` selects the BASELINE.json configuration (default c3, the one the metric is quoted on):
  c2       borehole d=8, N=100k, K=1000                      same metric, same JSON line
  c3       d=10, N=1M, K=2000                                (default)
  c4share  one GPU's share of C4: d=20, N=1.25M, K=4000      same metric
  c5       Phi.A with 64 right-hand sides on C3's table      metric phi_mat_products_per_s, roofline = DMMA pipe
  build    basis rebuild with gradients at C3's shape        metric basis_builds_per_s, roofline = DMMA pipe + HBM writes
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

D, N_TOTAL, K_TERMS, KNOTS = 10, 1_000_000, 2000, 40


def synth_rows(lo: int, hi: int, d: int, seed: int = 42) -> np.ndarray:
    """Rows [lo, hi) of the synthetic U(0,1)^d design; identical for any sharding."""
    blk = 1 << 16
    out = np.empty((hi - lo, d), order="F")
    b0 = lo // blk
    pos = 0
    while pos < hi - lo:
        start = b0 * blk
        rng = np.random.default_rng([seed, b0])
        chunk = rng.uniform(size=(blk, d))
        a = max(lo, start) - start
        b = min(hi, start + blk) - start
        out[pos:pos + (b - a)] = chunk[a:b]
        pos += b - a
        b0 += 1
    return out


def wingweight(x: np.ndarray) -> np.ndarray:
    """Wing-weight-style 10-input closed form (Forrester et al. 2008), inputs scaled from [0,1]."""
    Sw = 150 + 50 * x[:, 0]; Wfw = 220 + 80 * x[:, 1]; A = 6 + 4 * x[:, 2]
    Lam = (-10 + 20 * x[:, 3]) * np.pi / 180; q = 16 + 29 * x[:, 4]; lam = 0.5 + 0.5 * x[:, 5]
    tc = 0.08 + 0.1 * x[:, 6]; Nz = 2.5 + 3.5 * x[:, 7]; Wdg = 1700 + 800 * x[:, 8]; Wp = 0.025 + 0.055 * x[:, 9]
    return (0.036 * Sw ** 0.758 * Wfw ** 0.0035 * (A / np.cos(Lam) ** 2) ** 0.6 * q ** 0.006 * lam ** 0.04
            * (100 * tc / np.cos(Lam)) ** (-0.3) * (Nz * Wdg) ** 0.49 + Sw * Wp)


def setup_model(lib, d=D, K=K_TERMS):
    """outermod with the obfit defaults (R/fitting.R:66-75): mat25pow, 40 quantile knots per dim."""
    om = lib.outermod()
    om.setcovfs(["mat25pow"] * d)
    sample = synth_rows(0, 100_000, d)
    q = np.linspace(0, 1, KNOTS) * KNOTS / (KNOTS + 1) + 0.5 / (KNOTS + 1)  # .genknotlist, R/fitting.R:177-185
    om.setknot([np.quantile(sample[:, l], q) for l in range(d)])
    hyp = om.gethyp()
    hyp[0::2] = np.linspace(-0.6, 0.4, d)  # anisotropic terms (SURVEY 8d)
    om.updatehyp(hyp)
    terms = om.selectterms(K)
    return om, terms


CONFIGS = {
    "c2": dict(d=8, N=100_000, K=1000, name="C2 borehole d=8"),
    "c3": dict(d=10, N=N_TOTAL, K=K_TERMS, name="C3 wingweight-style d=10"),
    "c4share": dict(d=20, N=1_250_000, K=4000, name="C4 (one GPU's share of N=10M) synthetic d=20"),
    "c5": dict(d=10, N=N_TOTAL, K=K_TERMS, name="C5 multi-RHS (64 columns) on C3's table"),
    "build": dict(d=10, N=N_TOTAL, K=K_TERMS, name="basis rebuild with gradients at C3's shape"),
}


def config_model(lib, cfg):
    """outermod + terms of a BASELINE configuration (the obfit defaults, R/fitting.R:66-75)."""
    c = CONFIGS[cfg]
    if c["d"] == D:
        return setup_model(lib)
    seed = 7 if c["d"] == 20 else 42
    om = lib.outermod()
    om.setcovfs(["mat25pow"] * c["d"])
    sample = synth_rows(0, 100_000, c["d"], seed=seed)
    q = np.linspace(0, 1, KNOTS) * KNOTS / (KNOTS + 1) + 0.5 / (KNOTS + 1)
    om.setknot([np.quantile(sample[:, l], q) for l in range(c["d"])])
    hyp = om.gethyp()
    hyp[0::2] = np.linspace(-0.6, 0.4, c["d"])
    om.updatehyp(hyp)
    return om, om.selectterms(c["K"])


def config_rows(cfg, lo, hi):
    c = CONFIGS[cfg]
    return synth_rows(lo, hi, c["d"], seed=7 if c["d"] == 20 else 42)


def measured_traffic(cfg, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture of
    this configuration (profiles/r02_traffic.json, written by tools/ncu_traffic.py), or (None, None)."""
    f = REPO / "profiles" / "r02_traffic.json"
    try:
        e = json.loads(f.read_text())[cfg]
        return float(e["kernels"][kernel]["dram_bytes_per_launch"]), f"ncu --set full, profiles/r02_traffic.json[{cfg}] ({e['source']})"
    except Exception:
        return None, None


DUMP_MAX = 1 << 21  # elements per array written by --dump-outputs (16 MB of float64; at most three arrays per run)


def dump_rows(n_rows, ncols):
    """Global row indices that --dump-outputs keeps of an n_rows x ncols output: all of them when the output fits
    DUMP_MAX, else a fixed, seeded sample (the same for every build and every sharding)."""
    k = max(1, DUMP_MAX // max(1, ncols))
    if n_rows <= k:
        return np.arange(n_rows)
    return np.sort(np.random.default_rng(0).choice(n_rows, size=k, replace=False))


def write_outputs(outdir, rank, world, lo, hi, N, sharded, whole):
    """--dump-outputs: `sharded` maps names to this rank's rows [lo, hi) of an N-row output, `whole` to outputs that
    every rank holds in full.  Rank 0 writes each as DIR/<name>.npy in float64, rows sampled by dump_rows."""
    arrays = {}
    for name, a in sharded.items():
        a = np.asarray(a, dtype=np.float64)
        idx = dump_rows(N, a.size // max(1, a.shape[0]))
        part = a[idx[(idx >= lo) & (idx < hi)] - lo]
        if world > 1:
            import torch.distributed as dist
            parts = [None] * world if rank == 0 else None
            dist.gather_object(part, parts, dst=0)
            part = np.concatenate(parts) if rank == 0 else None
        arrays[name] = part
    if rank != 0:
        return
    arrays.update((name, np.asarray(a, dtype=np.float64)) for name, a in whole.items())
    outdir = Path(outdir)
    outdir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(outdir / f"{name}.npy", a)


def term_stats(terms):
    nnz = (terms > 0).sum(1)
    return int((nnz + 1).sum()), int(terms.max(0).sum())


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        self.t0 = self.t1 = None

    def mark(self, which):
        setattr(self, which, time.time())

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.split(", ") for r in Path(self.f.name).read_text().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); smax = float(r[2])
            except Exception:
                continue
            for nm, v in zip(names, r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(nm)
        # the sampler runs across the whole bench; the under-load clock is the top half of the samples
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_lib():
    """The CPU implementation that is timed beside the GPU: the reference itself when oracle/_ref holds it, else the port."""
    from outerbase_b200.binding import Library
    ref = REPO / "oracle" / "_ref" / "libob_ref.so"
    if ref.exists():
        return Library(ref, "ref_"), "reference", "unmodified reference sources (linalg.cpp, modandbase.cpp, covfuncs.cpp) on the Armadillo-subset shim, -O2 -fopenmp"
    so = REPO / "oracle" / "_build" / "libob_oracle.so"
    if not so.exists():
        subprocess.run(["make", "-C", str(REPO / "oracle")], check=True, capture_output=True)
    return Library(so, "orc_"), "port", "OpenMP row-chunk path of the oracle's restatement, -O2 -fopenmp"


def cpu_pairs_per_s(cfg, rows: int, steps: int, warmup: int, budget_s: float):
    """(Phi a, Phi^T r) pairs/s of the CPU implementation on `rows` rows of the configuration, all host threads;
    returns (pairs/s on those rows, threads, steps done, seconds, kind, what)."""
    L, kind, what = cpu_lib()
    om, terms = config_model(L, cfg)
    x = config_rows(cfg, 0, rows)
    ob = L.outerbase(om, x, dograd=False)
    rng = np.random.default_rng(1)
    a = np.sqrt(om.getvar(terms) / 20) * rng.normal(size=terms.shape[0])
    r = rng.normal(size=rows)
    cores = ob.nthreads
    for _ in range(max(0, warmup)):
        ob.matmul(terms, a); ob.tmatmul(terms, r)
    t0 = time.time()
    done = 0
    for _ in range(max(1, steps)):
        for _ in range(2):
            ob.matmul(terms, a); ob.tmatmul(terms, r)
        done += 1
        if time.time() - t0 > budget_s:
            break
    dt = time.time() - t0
    return 2 * done / dt, cores, done, dt, kind, what


def run_reference(args):
    """The reference arm: the reference's own CPU path on the FULL row count of the configuration (steps are cut to the
    time budget, rows are not: the number is a measurement, not an extrapolation)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.config if args.config in ("c2", "c3", "c4share") else "c3"
    c = CONFIGS[cfg]
    N = args.rows or c["N"]
    val, cores, done, dt, kind, what = cpu_pairs_per_s(cfg, N, args.steps, min(args.warmup, 1), budget_s=90.0)
    line = {
        "impl": "reference", "metric": "phi_matvec_pairs_per_s", "value": val, "unit": "pairs/s", "n_gpus": args.gpus,
        "steps": done, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * dt / max(done, 1),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{c['name']} N={N} K={c['K']} mat25pow {KNOTS} knots/dim (all {N} rows; step = 2 pairs)"},
        "cpu_baseline": {"value": val, "unit": "pairs/s", "cores": int(cores), "kind": kind,
                         "sample": f"all {N} rows, {done} steps of 2 pairs in {dt:.1f} s; {what}"},
        "e2e": {"value": val, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def config_response(x):
    """Synthetic responses of the non-C3 configurations: borehole on the first 8 inputs (+ smooth terms for d = 20)."""
    rw = x[:, 0] * 0.10 + 0.05; r = x[:, 1] * 49900 + 100; Tu = x[:, 2] * 52530 + 63070; Hu = x[:, 3] * 120 + 990  # obtest_borehole8d,
    Tl = x[:, 4] * 52.9 + 63.1; Hl = x[:, 5] * 120 + 700; L = x[:, 6] * 560 + 1120; Kw = x[:, 7] * 2190 + 9855     # R/testfuncs.R:32-46
    m2 = np.log(r / rw)
    y = 2 * np.pi * Tu * (Hu - Hl) / m2 / (1 + 2 * L * Tu / (m2 * rw ** 2 * Kw) + Tu / Tl) - 77
    if x.shape[1] > 10:
        y = y + 20 * np.sin(3 * x[:, 8]) * x[:, 9] + 10 * x[:, 10:].sum(1)
    return y


def hbm_peak():
    mp = REPO / "MEASURED_PEAKS.json"
    if mp.exists():
        return float(json.loads(mp.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def run_special(args, lib, om, terms, x, cfg, rank, world, local, N, W, Lcols, lo, hi):
    """c5: Phi.A with 64 right-hand sides (prodmm_(mat), src/linalg.cpp:527-557) and its transpose; build: the basis
    rebuild with gradients (outerbase::build, src/modandbase.cpp:547-626).  Same JSON contract, own metric."""
    import torch
    import torch.distributed as dist
    dev = torch.device("cuda", local)
    stream = torch.cuda.ExternalStream(lib.stream())
    nloc, K = x.shape[0], terms.shape[0]
    fp64_peak = lib.fp64_peak()
    clocks = ClockSampler(local) if rank == 0 else None

    def barrier():
        lib.synchronize(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed(f, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0 = lib.launch_count()
        e0.record(stream)
        for _ in range(steps):
            f()
        e1.record(stream)
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.cpu()[0]) / steps, lib.launch_count() - n0

    if cfg == "c5":
        Ccols = 64
        ob = lib.outerbase(om, x, dograd=False)
        ob.set_terms(terms); ob.specialize(terms)
        rng = np.random.default_rng(1)
        A = torch.from_numpy(np.asfortranarray(rng.normal(size=(K, Ccols)) * np.sqrt(om.getvar(terms) / 20)[:, None]).T.copy()).to(dev)  # column-major K x C
        ld = ((nloc + 255) // 256) * 256
        out = torch.empty(Ccols * ld, dtype=torch.float64, device=dev)
        R = torch.from_numpy(np.random.default_rng([7, rank]).normal(size=(Ccols, nloc))).to(dev)  # column-major N x C
        G = torch.empty(Ccols * K, dtype=torch.float64, device=dev)
        f_mm = lambda: ob.mm_mat_dev(A.data_ptr(), Ccols, out.data_ptr())
        f_tm = lambda: ob.tmm_mat_dev(R.data_ptr(), Ccols, G.data_ptr())
        for _ in range(max(3, args.warmup)):
            f_mm(); f_tm()
        barrier()
        ms_mm, l1 = timed(f_mm, args.steps)
        ms_tm, l2 = timed(f_tm, args.steps)
        if args.dump_outputs:  # the last timed products: Phi.A (column-major, leading dimension nloc) and Phi^T.R (K x C)
            dumped = ({"phi_a_mat": out[:Ccols * nloc].view(Ccols, nloc).T.cpu().numpy()}, {"phi_t_mat": G.view(Ccols, K).T.cpu().numpy()})
        # e2e: host matrices in, host results out, every call
        Ah = np.asfortranarray(rng.normal(size=(K, Ccols))); Rh = np.asfortranarray(rng.normal(size=(nloc, Ccols)))
        ob.matmul(terms, Ah); barrier()
        t0 = time.perf_counter(); n_e2e = 3
        for _ in range(n_e2e):
            ob.matmul(terms, Ah)
        barrier(); e2e_ms = (time.perf_counter() - t0) / n_e2e * 1e3
        clk = clocks.stop() if clocks else None
        if args.dump_outputs:
            write_outputs(args.dump_outputs, rank, world, lo, hi, N, *dumped)
        if rank != 0:
            return
        flop = 2.0 * (-(-N // world)) * K * Ccols
        achieved = flop / (ms_mm * 1e-3) / 1e12
        traffic, tsrc = measured_traffic(cfg, "phi_am_spec") if world == 1 else (None, None)
        hp, hs = hbm_peak()
        line = {"metric": "phi_mat_products_per_s", "value": 1e3 / ms_mm, "unit": "products/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms_mm, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"{CONFIGS[cfg]['name']}: Phi.A, N={N} K={K} C={Ccols}, rows sharded over {world} GPU(s)", "step": "one Phi.A product (prodmm_(mat))",
                           "l2": "inputs exceed L2 (0.6 GB of basis columns + 0.5 GB of output per product)"},
                "e2e": {"value": 1e3 / e2e_ms, "unit": "products/s", "h2d_bytes_per_step": K * Ccols * 8, "d2h_bytes_per_step": nloc * Ccols * 8},
                "gpu_launches": int(l1),
                "roofline": {"bound": "tensor", "kernel": "phi_am_spec", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                             "frac": achieved / fp64_peak, "traffic": traffic, "traffic_source": tsrc,
                             "peak_source": "FP64 pipe (DFMA micro-benchmark of this process; DMMA shares the pipe and its peak, profiles/r01_dmma_bench.txt)",
                             "algorithmic_flop_per_launch": flop, "hbm": {"peak_gbs": hp, "peak_source": hs}},
                "transpose": {"ms": ms_tm, "launches": int(l2), "note": "Phi^T.A (tprodmm_(mat), linalg.cpp:583-637), same shapes"},
                "clocks": clk}
        print(json.dumps(line))
        return
    # ---- build
    ob = lib.outerbase(om, x, dograd=True)
    for _ in range(max(3, args.warmup)):
        ob.build()
    barrier()
    t0 = time.perf_counter(); n0 = lib.launch_count()
    for _ in range(args.steps):
        ob.build()
    barrier()
    ms = (time.perf_counter() - t0) / args.steps * 1e3
    launches = lib.launch_count() - n0
    if args.dump_outputs:  # the basis the last timed rebuild left in the object
        dumped = ({"basemat": ob.real("basemat"), "basescale": ob.real("basescale")}, {})
    # what a BFGS objective evaluation pays (R/outersupport.R:215-216 -> loglik_gauss::updateom): the same rebuild on the
    # columns the terms table reads (compact layout, DESIGN 2)
    yv = wingweight(x); yv = (yv - yv.mean()) / yv.std(ddof=1)
    loglik = lib.loglik_gauss(om, terms, yv, x)
    for _ in range(3):
        loglik.updateom()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        loglik.updateom()
    barrier()
    ms_pruned = (time.perf_counter() - t0) / args.steps * 1e3
    clk = clocks.stop() if clocks else None
    if args.dump_outputs:
        write_outputs(args.dump_outputs, rank, world, lo, hi, N, *dumped)
    if rank != 0:
        return
    d, H, M, nge = om.sizes()
    m = M // d
    nmax = -(-N // world)
    flop = 2.0 * nmax * d * m * m * (1 + 2 * (H // d))  # SURVEY 8d
    bytes_w = 8.0 * nmax * (M + nge + d + 1)
    hp, hs = hbm_peak()
    achieved = flop / (ms * 1e-3) / 1e12
    line = {"metric": "basis_builds_per_s", "value": 1e3 / ms, "unit": "builds/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{CONFIGS[cfg]['name']}: N={N} d={d} m={m} H={H}, rows sharded over {world} GPU(s)", "step": "one outerbase::build with gradients",
                       "l2": f"writes {bytes_w / 1e9:.1f} GB per build"},
            "e2e": {"value": 1e3 / ms, "unit": "builds/s", "h2d_bytes_per_step": int(8 * (M * m + nge * m)), "d2h_bytes_per_step": 0},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "basis_build_mma_kernel", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s", "frac": achieved / fp64_peak,
                         "traffic": None, "peak_source": "FP64 pipe (DFMA micro-benchmark of this process; DMMA shares it)", "algorithmic_flop_per_launch": flop / d,
                         "hbm": {"achieved_gbs": bytes_w / (ms * 1e-3) / 1e9, "peak_gbs": hp, "peak_source": hs, "algorithmic_bytes_per_build": bytes_w}},
            "pruned": {"ms": ms_pruned, "columns": int(np.asarray(terms).max(0).sum() + 3 * d), "of": int(M),
                       "note": "loglik_gauss::updateom: levels the terms table reads (+2), the layout every objective evaluation rebuilds"},
            "clocks": clk}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the measured path (--impl reference stops after 90 s; the e2e and optcg "
                         "side measurements use their own counts)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=0, help="total rows over all ranks (default: the configuration's)")
    ap.add_argument("--config", default="c3", choices=sorted(CONFIGS), help="BASELINE.json configuration (default c3)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-optcg", action="store_true")
    ap.add_argument("--spec", default="1", choices=["0", "1"],
                    help="1: terms-specialised kernels, compiled during set-up (default); 0: interpreter kernels only")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float64; outputs "
                         "above 2M elements as a fixed, seeded sample of their rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the B200 path computed: not available with --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    import outerbase_b200 as obp
    if not obp.LIBPATH.exists():
        obp.build()
    lib = obp.lib(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        box = [lib.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        lib.comm_init(world, rank, box[0])

    cfg = args.config
    C = CONFIGS[cfg]
    N = args.rows or C["N"]
    K_TERMS_ = C["K"]
    lo, hi = (N * rank) // world, (N * (rank + 1)) // world
    nloc = hi - lo
    om, terms = config_model(lib, cfg)
    W, Lcols = term_stats(terms)
    x = config_rows(cfg, lo, hi)
    lib.set_option("spec", float(args.spec))
    if cfg in ("c5", "build"):
        run_special(args, lib, om, terms, x, cfg, rank, world, local, N, W, Lcols, lo, hi)
        if world > 1:
            dist.destroy_process_group()
        return
    ob = lib.outerbase(om, x, dograd=False)
    ob.set_terms(terms)
    # set-up, untimed like the basis build: compile the kernels for this terms table (NVRTC, cached on disk)
    spec_compile_s = ob.specialize(terms) if args.spec == "1" else None
    rng = np.random.default_rng(1)
    K_TERMS = K_TERMS_  # noqa: N806 -- the configuration's term count from here on
    a_h = np.sqrt(om.getvar(terms) / 20) * rng.normal(size=K_TERMS)
    r_h = np.random.default_rng([7, rank]).normal(size=nloc)

    stream = torch.cuda.ExternalStream(lib.stream())
    dev = torch.device("cuda", local)
    a_d = torch.from_numpy(a_h).to(dev)
    r_d = torch.from_numpy(r_h).to(dev)
    yhat_d = torch.empty(((nloc + 255) // 256) * 256, dtype=torch.float64, device=dev)
    g_d = torch.empty(K_TERMS, dtype=torch.float64, device=dev)
    torch.cuda.synchronize()

    def step_dev(ev=None):
        for i in range(2):
            if ev is not None: ev[0][i].record(stream)
            ob.mm_dev(a_d.data_ptr(), yhat_d.data_ptr())
            if ev is not None: ev[1][i].record(stream)
            ob.tmm_dev(r_d.data_ptr(), g_d.data_ptr())
            if ev is not None: ev[2][i].record(stream)

    def barrier():
        lib.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    fp64_peak = lib.fp64_peak()
    clocks = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        step_dev()
    barrier()
    # ---- value: device-resident operands
    evs = [[[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(3)] for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = lib.launch_count()
    e0.record(stream)
    t_issue = time.perf_counter()
    for s in range(args.steps):
        step_dev(evs[s])
    e1.record(stream)
    t_issue = (time.perf_counter() - t_issue) / args.steps * 1e3  # host time to ISSUE one step (launch-bound check)
    barrier()
    launches = lib.launch_count() - n0
    if args.dump_outputs:  # what the last timed step returned: Phi a on this rank's rows, Phi^T r summed over the ranks
        dumped = ({"phi_a": yhat_d[:nloc].cpu().numpy()}, {"phi_t": g_d.cpu().numpy()})
    ms = e0.elapsed_time(e1)
    t_a = float(np.mean([evs[s][0][i].elapsed_time(evs[s][1][i]) for s in range(args.steps) for i in range(2)]))
    t_t = float(np.mean([evs[s][1][i].elapsed_time(evs[s][2][i]) for s in range(args.steps) for i in range(2)]))
    tms = torch.tensor([ms, t_a, t_t], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms, t_a, t_t = [float(v) for v in tms.cpu()]
    value = 2 * args.steps / (ms * 1e-3)

    # ---- the cross-GPU sum on its own: K doubles, back to back (ranks in lockstep), both implementations
    allreduce = None
    if world > 1:
        allreduce = {}
        buf = torch.zeros(K_TERMS, dtype=torch.float64, device=dev)
        for name, p2p in (("p2p_us", 1), ("nccl_us", 0)):
            lib.set_option("p2p", p2p)
            for _ in range(20):
                lib.allreduce_dev(buf.data_ptr(), K_TERMS)
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            for _ in range(200):
                lib.allreduce_dev(buf.data_ptr(), K_TERMS)
            a1.record(stream)
            barrier()
            allreduce[name] = a0.elapsed_time(a1) / 200 * 1e3
            for _ in range(5):
                ob.tmm_dev(r_d.data_ptr(), g_d.data_ptr())
            barrier()
            a0.record(stream)
            for _ in range(100):
                ob.tmm_dev(r_d.data_ptr(), g_d.data_ptr())
            a1.record(stream)
            barrier()
            allreduce["phi_t_" + name] = a0.elapsed_time(a1) / 100 * 1e3
        lib.set_option("p2p", 1)
        allreduce["note"] = "K doubles, 200 back-to-back calls on the library stream; p2p falls back to NCCL when peer memory is not mapped"

    # ---- e2e: the reference-facing calls outerbase::mm / outerbase::tmm with HOST buffers, every call
    # copying its inputs in and its result out (pinned host memory on both sides, as the contract asks)
    def pinned(n, src=None):
        t = torch.empty(n, dtype=torch.float64).pin_memory()
        v = t.numpy()
        if src is not None:
            v[:] = src
        return t, v
    _ka, a_p = pinned(K_TERMS, a_h)
    _kr, r_p = pinned(nloc, r_h)
    _ky, y_p = pinned(nloc)
    _kg, g_p = pinned(K_TERMS)
    for _ in range(2):
        ob.matmul(terms, a_p, out=y_p); ob.tmatmul(terms, r_p, out=g_p)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(3, min(args.steps, 10))
    for _ in range(e2e_steps):
        for _ in range(2):
            yh = ob.matmul(terms, a_p, out=y_p)
            gh = ob.tmatmul(terms, r_p, out=g_p)
    barrier()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = 2 * e2e_steps / float(dt.cpu()[0])
    h2d = 2 * (K_TERMS * 8 + nloc * 8)
    d2h = 2 * (nloc * 8 + K_TERMS * 8)

    # ---- obfit's CG solve on the same shard: lpdfvec(logpr_gauss, loglik_gauss).optcg(0.001, 100)
    optcg = None
    if not args.no_optcg:
        yv = wingweight(x) if C["d"] == D else config_response(x)
        stats = torch.tensor([yv.sum(), (yv ** 2).sum(), float(nloc)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(stats)
        s1, s2, n = [float(v) for v in stats.cpu()]
        mean = s1 / n
        sd = np.sqrt((s2 - n * mean * mean) / (n - 1))
        yv = (yv - mean) / sd
        logpr = lib.logpr_gauss(om, terms)
        loglik = lib.loglik_gauss(om, terms, yv, x)
        vec = lib.lpdfvec(logpr, loglik)  # prior first, as obfit does (R/fitting.R:86,107)
        barrier()
        t0 = time.perf_counter()
        vec.optcg(0.001, 100)
        barrier()
        t_cg = time.perf_counter() - t0
        # the same solve again from zero coefficients: what every further objective evaluation of a
        # BFGS_lpdf run costs (compiled programs, column tables and kernels are cached in the object)
        vec.set_coeff(np.zeros(K_TERMS))
        barrier()
        t0 = time.perf_counter()
        vec.optcg(0.001, 100)
        barrier()
        t_cg2 = time.perf_counter() - t0
        optcg = {"wall_s": t_cg2, "first_call_wall_s": t_cg, "iters": vec.cg_iters, "val": vec.val,
                 "pairs": 2 * vec.cg_iters + 2, "extra": "one diaghess (squared Phi^T) and H hyper-gradient Phi a passes per call"}
        del vec, loglik, logpr

    clk = clocks.stop() if clocks else None
    if args.dump_outputs:
        write_outputs(args.dump_outputs, rank, world, lo, hi, N, *dumped)
    if rank == 0:
        hbm_peak, hbm_src = 6650.0, "fallback"
        mp = REPO / "MEASURED_PEAKS.json"
        if mp.exists():
            hbm_peak, hbm_src = float(json.loads(mp.read_text())["hbm_gbs"]), "measured"
        # dominant kernel: the slower of the two Phi kernels; algorithmic work N*W flop (+N), SURVEY 8d
        kn = ("phi_t_spec", "phi_a_spec") if args.spec == "1" else ("phi_t2_kernel", "phi_a_kernel")
        dom, t_dom = (kn[0], t_t) if t_t >= t_a else (kn[1], t_a)
        nmax = -(-N // world)
        flop = nmax * (W + 1)
        achieved = flop / (t_dom * 1e-3) / 1e12
        bytes_alg = nmax * 8 * (Lcols + 1) + nmax * 8
        # dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
        # `ncu --set full` capture of this exact workload (profiles/r01_spec_ncu_summary.md); other shapes: null
        traffic, traffic_src = (measured_traffic(cfg, dom) if args.spec == "1" and world == 1 and N == C["N"] else (None, None))
        roofline = {"bound": "fp64", "kernel": dom, "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                    "frac": achieved / fp64_peak if fp64_peak else None, "traffic": traffic,
                    "traffic_source": traffic_src,
                    "peak_source": "DFMA micro-benchmark run in this process (nominal 37.2 TFLOP/s at 1965 MHz)",
                    "algorithmic_flop_per_launch": flop, "W": W, "Lcols": Lcols,
                    "ms_phi_a": t_a, "ms_phi_t": t_t, "host_issue_ms_per_step": t_issue,
                    "hbm": {"achieved_gbs": bytes_alg / (t_dom * 1e-3) / 1e9, "peak_gbs": hbm_peak, "peak_source": hbm_src,
                            "algorithmic_bytes_per_launch": bytes_alg}}
        line = {
            "metric": "phi_matvec_pairs_per_s", "value": value, "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{C['name']} N={N} K={K_TERMS} mat25pow {KNOTS} knots/dim, rows sharded over {world} GPU(s)",
                       "step": "one CG iteration of fit.cpp:71-85 = 2 x (Phi a, Phi^T r [+allreduce])",
                       "kernels": ("terms-specialised (run-time compiled for this table during set-up: "
                                   f"{spec_compile_s:.1f} s, 0 = disk-cache hit)") if args.spec == "1" else "interpreter",
                       "l2": f"inputs exceed L2: {nmax * 8 * (Lcols + 2) / 1e6:.0f} MB of basis columns per pass vs 126 MB"},
            "e2e": {"value": e2e_value, "unit": "pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "roofline": roofline, "clocks": clk, "optcg": optcg, "allreduce": allreduce,
        }
        if world == 1 and not args.no_cpu_baseline:
            try:
                sample = min(N, 250_000)  # ~10-20 s of CPU work on the box's host cores; `--impl reference` times all rows
                v, cores, done, dtc, kind, what = cpu_pairs_per_s(cfg, sample, 40, 1, budget_s=15.0)
                line["cpu_baseline"] = {"value": v * sample / N, "unit": "pairs/s", "cores": int(cores), "kind": kind,
                                        "sample": f"{sample} of {N} rows, {done} steps of 2 pairs in {dtc:.1f} s, scaled by rows; {what}"}
            except Exception as e:  # the oracle is only the reported baseline
                line["cpu_baseline"] = {"value": None, "unit": "pairs/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
