"""Two-rank worker for the per-column multi-response objects (tests/test_multiresponse_percol.py): rows sharded over the
ranks, one B200 per rank.  Every rank also runs the 1-rank fit on all rows on its own GPU (before the communicator
exists); the per-column defaults, which are variances over all ranks' rows, and the sharded fit must match it and be
bit-identical across the ranks."""
import os
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

REPO = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "tests"))
from conftest import relerr  # noqa: E402
from test_multiresponse_percol import objects  # noqa: E402

N, K, C = 6001, 150, 8


def fit(lib, rows):
    om, x, Y, terms, _ = objects(lib, N, K, C)
    lk = lib.loglik_gauss_multi(om, terms, np.asfortranarray(Y[rows]), np.asfortranarray(x[rows]), para_per_column=True)
    vec = lib.lpdfvec(lib.logpr_gauss_multi(om, terms, C, para_per_column=True), lk)
    vec.domarg = True
    default = np.array(vec.para)
    vec.updatepara(default + np.linspace(-0.3, 0.3, 2 * C))
    vec.optcg(0.001, 100)
    return dict(default=default, coeff=np.array(vec.coeff), val=vec.val, gradhyp=np.array(vec.gradhyp),
                gradpara=np.array(vec.gradpara), iters=np.array(vec.cg_iters_per_column))


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    import outerbase_b200 as obp
    lib = obp.lib(local)
    ref = fit(lib, slice(0, N))
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    box = [lib.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    lib.comm_init(world, rank, box[0])
    lo, hi = (N * rank) // world, (N * (rank + 1)) // world
    got = fit(lib, slice(lo, hi))
    assert relerr(got["default"], ref["default"]) < 1e-12  # per-column defaults over all ranks' rows
    np.testing.assert_array_equal(got["iters"], ref["iters"])
    assert relerr(got["coeff"], ref["coeff"]) < 1e-8
    assert abs(got["val"] - ref["val"]) <= 1e-8 * abs(ref["val"])
    assert relerr(got["gradpara"], ref["gradpara"]) < 1e-8
    assert relerr(got["gradhyp"], ref["gradhyp"]) < 1e-6
    for v in (got["coeff"].ravel(order="F"), np.array([got["val"]]), got["gradhyp"], got["gradpara"]):
        t = torch.from_numpy(v.copy()).cuda()
        tmax, tmin = t.clone(), t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX); dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        assert torch.equal(tmax, tmin)
    dist.barrier()
    if rank == 0:
        print(f"mgpu_multiresponse_percol_worker world={world} OK")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
