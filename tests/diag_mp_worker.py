"""Worker of tests/test_diag_gpu.py::test_two_ranks_give_the_numbers_of_one_handle: one process per GPU under
torch.distributed.run.  mq_diag_summary(collective=1) over the ranks' chains equals the summary of one handle that runs
all of them (a chain's trajectory does not depend on the GPU it runs on), to 1e-12 relative."""
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def run(mq, cfg, pk, n, device, seed, rank=None, world=None, ident=None):
    smp = mq.Sampler(cfg, pk, n, device, seed)
    if ident is not None:
        smp.comm_init(ident, rank, world)          # also sets the chain offset to rank * n
    smp.diag_begin(5, 8)
    smp.init_chains()
    for _ in range(20):
        smp.step(10)
        smp.drain()
    s = smp.diag_summary(collective=ident is not None)
    if ident is not None:
        smp.comm_destroy()
    smp.close()
    return s


def main():
    import torch
    import torch.distributed as dist
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import dist as mqd
    from mcmc_eq_b200._lib import comm_unique_id
    from tests import inputs
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    d = tempfile.mkdtemp(prefix=f"mqdiag{rank}_")
    cfgp, pkp = inputs.materialise("example2", d, j_max_start=10, j_max_main=100000, deci=2, true_random=3)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    n, seed = 8, 41
    ident = mqd.exchange_unique_id(dist, comm_unique_id, device=f"cuda:{local}")
    got = run(mq, cfg, pk, n, local, seed, rank, world, ident)
    parts = [None] * world
    dist.all_gather_object(parts, {k: got[k] for k in ("mean", "sd", "rhat", "ess", "n_models", "chains_used")})
    ok = {}
    if rank == 0:
        one = run(mq, cfg, pk, n * world, local, seed)
        ok["chains_used"] = one["chains_used"] == got["chains_used"] == n * world
        ok["n_models"] = one["n_models"] == got["n_models"] > 0
        ok["ranks_agree"] = all(np.array_equal(p[k], parts[0][k], equal_nan=True) for p in parts for k in ("mean", "sd", "rhat", "ess"))
        for k in ("mean", "sd", "rhat", "ess"):
            a, b = got[k], one[k]
            same = np.array_equal(np.isfinite(a), np.isfinite(b)) and np.array_equal(a[~np.isfinite(a)], b[~np.isfinite(b)], equal_nan=True)
            f = np.isfinite(b)
            scale = np.maximum(np.abs(b[f]), np.nan_to_num(one["sd"][f]))
            ok[k] = bool(same and (np.abs(a[f] - b[f]) <= 1e-12 * scale + 1e-300).all())
        print("DIAGRESULT " + json.dumps(ok))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
