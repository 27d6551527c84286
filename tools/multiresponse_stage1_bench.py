"""Does obfit's stage 1 shorten a multi-response fit?  fitting.obfit_multi on the C3 model (bench.synth_rows, N = 1M, the
hyper-parameters of bench.setup_model, numb = 2000, numberopts = 1, one B200) with the responses of
tools/multiresponse_bench.py, run with stage1=False (stage 2 alone from the constructor defaults) and stage1=True
(loglik_gda_multi on a shared subsample of at most 3 numbr rows first).  Prints one JSON line per C in {8, 64} with,
per run:
  wall_ms                               the whole obfit_multi call (the CG measurement below excluded)
  stage1_ms                             from the call to the end of the last stage-1 objective evaluation (the
                                        CG measurement below excluded)
  evals_stage1 / evals_stage2           objective evaluations (fitting.lpdfwrapper calls) in each stage
  eval_ms_stage1 / eval_ms_stage2       their summed times
  final_val / hyp / para                the optimum (-log-posterior) and where it is
  stage1_cg_ms_per_iter / _launches_per_iter
                                        one stage-1 CG iteration, from two no-stop runs (tol < 0) of 2 and 6 iterations
                                        at the first stage-1 evaluation's point
The GPU name and power limit are read in the same run."""
import json
import sys
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "tools"))
import bench  # noqa: E402
import outerbase_b200 as obp  # noqa: E402
from multiresponse_bench import gpu_info, responses, timed  # noqa: E402
from outerbase_b200 import binding, fitting  # noqa: E402


class Counter:
    """wraps fitting.lpdfwrapper: counts and times each objective evaluation by stage (the likelihood child's type)"""

    def __init__(self, lib):
        self.lib, self.inner = lib, fitting.lpdfwrapper
        self.reset()

    def reset(self):
        self.evals = {1: [], 2: []}
        self.t_start, self.t_stage1_end, self.excluded_ms, self.cg = time.perf_counter(), None, 0.0, None

    def __call__(self, parlist, om, logpdf, **kw):
        stage = 1 if isinstance(logpdf._children[1], binding.loglik_gda_multi) else 2
        ms, out = timed(self.lib, lambda: self.inner(parlist, om, logpdf, **kw))
        self.evals[stage].append(ms)
        if stage == 1:
            if self.cg is None:
                t0 = time.perf_counter()
                self.cg = self.cg_per_iter(logpdf)
                self.excluded_ms += (time.perf_counter() - t0) * 1e3
            self.t_stage1_end = time.perf_counter()
        return out

    def cg_per_iter(self, vec):
        coeff = vec.coeff.copy()
        per = []
        for ep in (2, 6):
            vec.set_coeff(np.zeros(coeff.size))
            n0 = self.lib.launch_count()
            ms, _ = timed(self.lib, lambda: vec.optcg(-1.0, ep))
            per.append((ms, self.lib.launch_count() - n0))
        vec.set_coeff(coeff)
        return round((per[1][0] - per[0][0]) / 4, 3), (per[1][1] - per[0][1]) / 4


def main():
    lib = obp.lib(0)
    lib.set_option("spec", 1)
    name, power = gpu_info()
    om, _ = bench.setup_model(lib)
    hyp = np.array(om.gethyp())
    N, numb = bench.N_TOTAL, 2000
    x = bench.synth_rows(0, N, bench.D)
    counter = Counter(lib)
    fitting.lpdfwrapper = counter
    for C in (8, 64):
        Y = responses(x, C)
        out = {"workload": f"obfit_multi on the C3 model, N={N} numb={numb} C={C} numberopts=1", "gpu": name, "power_limit": power}
        for stage1 in (False, True):
            counter.reset()
            ms, model = timed(lib, lambda: fitting.obfit_multi(lib, x, Y, numb=numb, hyp=hyp, numberopts=1, stage1=stage1))
            r = {"wall_ms": round(ms - counter.excluded_ms, 1), "evals_stage1": len(counter.evals[1]), "evals_stage2": len(counter.evals[2]),
                 "eval_ms_stage1": round(sum(counter.evals[1]), 1), "eval_ms_stage2": round(sum(counter.evals[2]), 1),
                 "final_val": model["optinfo"]["optid"]["val"], "hyp": fitting.gethyp(model["om"]).tolist(),
                 "para": np.asarray(fitting.getpara(model["logpdf"])).tolist()}
            if stage1:
                r["stage1_ms"] = round((counter.t_stage1_end - counter.t_start) * 1e3 - counter.excluded_ms, 1)
                r["stage1_rows"] = int(model["stage1"]["rows"].size)
                r["stage1_terms"] = int(model["stage1"]["loglik"].nterms // C)
                r["stage1_cg_ms_per_iter"], r["stage1_cg_launches_per_iter"] = counter.cg
            out["stage1" if stage1 else "stage2_only"] = r
            del model
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
