"""bench.py --config fine: the fine-grid stress case (BASELINE.json configs[4], SURVEY.md section 8d item 5): 0.1 km grid to
200 km depth (eikonal plane 565 x 2001), 50 stations x 200 events on a 40 km array, 512 chains as 8 temperatures x 64
replicas with parallel-tempering swap rounds.  A step is one Metropolis-Hastings iteration of every chain with a velocity
proposal: 2 x 2001 eikonal solves of 1.13 M nodes per chain, then the misfit.  Planes of this size take eik_fine_kernel
(per-lane arrays in global memory); the generic kernel is timed beside it on a few chains in a subprocess
(MCMCEQ_EIKONAL=generic is read once per process)."""
from __future__ import annotations

import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))


def oracle_rows(cfg, st, ps, iz, rows):
    """rows of the oracle's field for source depth iz of phase ps: [len(rows)][nxmod]"""
    import ctypes as C
    from tests import util
    from tests import fwd_helpers as fh
    L = util.oracle()
    g = fh.fm_grid(cfg)
    nz, nxmod = cfg.grid.nz, L.fm_nxmod(C.byref(g))
    slow = np.zeros(nz, np.float32)
    L.fm_rasterise(C.byref(g), len(st["z"]), util.ptr(util.f32(st["z"])), util.ptr(util.f32(st["vp"])), util.ptr(util.f32(st["vpvs"])), ps,
                   util.ptr(slow))
    t0 = time.perf_counter()
    field, rc = util.oracle_time_2d(slow, nxmod, iz)
    dt = time.perf_counter() - t0
    assert rc == 0
    return field.T[rows], dt


def main(args, rank, world, local, dist):
    import bench as B
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    n_gpus = max(world, 1)
    total = 512
    chains = args.chains or total // n_gpus
    events, stations = args.events or 200, args.stations or 50
    device = local
    W = max(args.warmup, 1)
    cfg, pk, truth = synth.workload(events, stations, 33, device, fine=True, j_max_start=0, j_max_main=2**30, deci=2**30)
    nz, nxmod = cfg.grid.nz, int(np.sqrt(cfg.grid.nx ** 2 + cfg.grid.ny ** 2))
    workload = (f"fine-grid: {chains * n_gpus} chains ({chains}/GPU, 8 temperatures x {chains * n_gpus // 8} replicas) x {events} events x "
                f"{stations} stations, grid h=0.1 km 400x400x{nz} (eikonal plane {nxmod}x{nz}), <=20 layers, proposal 'P' (P_full: 2*nz "
                f"eikonal solves of {nxmod * nz} nodes + full misfit per proposal), tempering swap round after every step")
    config = {"workload": workload, "baseline_config": "configs[4]", "chains_per_gpu": chains, "events": events, "stations": stations,
              "grid": f"{nxmod}x{nz}", "proposal_string": "P", "parallelism": f"chains sharded x{n_gpus}; tempering all-gather over NCCL when N > 1",
              "l2": "per-step working set (tables 73 MB per chain, solver windows 145 MB per warp) exceeds the 126 MB L2"}
    smp = mq.Sampler(cfg, pk, chains, device, 1000)
    if dist is not None:
        import torch
        from mcmc_eq_b200 import dist as mqd
        from mcmc_eq_b200._lib import comm_unique_id
        smp.comm_init(mqd.exchange_unique_id(dist, comm_unique_id, torch.device("cuda", device)), rank, world)
    else:
        smp.set_chain_offset(0)
    ladder = np.array([1.0, 0.8, 0.64, 0.5, 0.4, 0.32, 0.25, 0.2], np.float32)
    smp.init_chains()
    smp.set_beta(ladder[(np.arange(chains) + rank * chains) % 8].copy())
    for _ in range(W):
        smp.step(1, "P")
    smp.sync()
    clocks = B.ClockSampler(device)
    clocks.start()
    launches0 = mq.lib().mq_launch_count()
    smp.profile(True)
    B.barrier_max(dist, 0.0, device)
    smp.sync()
    swaps, swap_ms = 0, []
    smp.timer_start(0)
    for k in range(args.steps):
        smp.step(1, "P")
        t0 = time.perf_counter()
        swaps += smp.temper_swap(k)           # one swap round per step: all-gather of (log-likelihood, beta) when N > 1
        swap_ms.append(1000.0 * (time.perf_counter() - t0))
    ms = smp.timer_stop(0)
    smp.sync()
    ms = B.barrier_max(dist, ms, device)
    launches = mq.lib().mq_launch_count() - launches0
    eik_ms, eik_n, spl = smp.profile(False)
    kernels = smp.profile_kernels()
    clk = clocks.stop()
    counts, ll, rms = smp.stats()
    if args.dump_outputs and rank == 0:
        B.dump_outputs(smp, (counts, ll, rms), args.dump_outputs)
    value = chains * n_gpus * args.steps / (ms / 1000.0)
    n_rows = mq.lib().mq_get_rows(smp.h, 0, 1, None, None)
    roofline = B.roofline_block(cfg, smp, ms, eik_ms, eik_n, spl, kernels, clk, device, n_rows) if eik_n else None
    if roofline:
        roofline["node_updates_per_s"] = float(nxmod) * nz * spl / (eik_ms / eik_n / 1000.0)

    # ---- parity: sampled (chain, phase, source depth) fields against the CPU oracle, after the timed region
    m = smp.get_models()
    rng = np.random.default_rng(5 + rank)
    ok, worst, n_checked, t_solve = True, 0.0, 0, []
    for c in sorted(int(x) for x in rng.choice(chains, size=min(2, chains), replace=False)):
        d = int(m.dim[c])
        st = dict(z=m.z[c, :d], vp=m.vp[c, :d], vpvs=m.vpvs[c, :d])
        for ph in (1, 2):
            rows, idx = smp.rows(c, ph)
            for iz in sorted(int(x) for x in rng.choice(nz, size=3, replace=False)) + [0]:
                ref, dt = oracle_rows(cfg, st, ph, iz, idx)
                t_solve.append(dt)
                err = np.abs(rows[:, iz, :] - ref)
                ok = ok and bool((err <= np.maximum(1e-4, 5e-6 * np.abs(ref))).all())
                worst = max(worst, float(err.max()))
                n_checked += 1
    parity = {"chains": min(2, chains), "fields": n_checked, "max_row_dt": worst, "tolerance": "max(1e-4 s, 5e-6 T) per stored table node",
              "against": "oracle/ (CPU restatement of time_2d, bit-identical to the compiled reference)", "ok": ok}

    # ---- end to end: one forward through the host-buffer call
    import torch
    keep = []
    for name in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise", "origin"):
        t = torch.from_numpy(getattr(m, name).copy()).pin_memory()
        keep.append(t)
        setattr(m, name, t.numpy())
    mf = np.zeros((chains, 8), np.float32)
    org = np.zeros((chains, pk.n_events), np.float32)
    B.barrier_max(dist, 0.0, device)
    t0 = time.perf_counter()
    smp.forward_host(m, 3, mf, org)
    e2e_s = B.barrier_max(dist, time.perf_counter() - t0, device)
    e2e = {"value": chains * n_gpus / e2e_s, "unit": B.UNIT, "steps": 1,
           "h2d_bytes_per_step": int(sum(getattr(m, k).nbytes for k in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise"))),
           "d2h_bytes_per_step": int(mf.nbytes + org.nbytes), "call": "mq_forward_host(calct=3)"}
    smp.close()

    # ---- the generic kernel on the same plane (a few chains, own process), and the oracle's solve time on one host core
    generic = None
    if rank == 0 and not args.no_extras and "MCMCEQ_EIKONAL" not in os.environ:
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--config", "fine", "--chains", "8", "--steps", "1", "--warmup", "1", "--no-extras"]
        r = subprocess.run(cmd, env=dict(os.environ, MCMCEQ_EIKONAL="generic", CUDA_VISIBLE_DEVICES=str(device), RANK="0", WORLD_SIZE="1"),
                           capture_output=True, text=True, timeout=3000)
        try:
            g = json.loads(r.stdout.strip().split("\n")[-1])
            per_solve = g["roofline"]["avg_launch_ms"] / g["roofline"]["solves_per_launch"]
            mine = roofline["avg_launch_ms"] / roofline["solves_per_launch"]
            generic = {"kernel": g["roofline"]["kernel"], "chains": 8, "us_per_solve": 1000.0 * per_solve, "fine_kernel_us_per_solve": 1000.0 * mine,
                       "speedup": per_solve / mine}
        except Exception as e:          # the comparison is informative; the headline does not depend on it
            generic = {"error": f"{type(e).__name__}: {e}", "stderr": r.stderr[-300:]}
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    t1 = float(np.median(t_solve))
    base = {"value": 1.0 / (2 * nz * t1), "unit": B.UNIT, "cores": 1, "kind": "port",
            "sample": f"{len(t_solve)} eikonal solves of the oracle port on this plane, {1000 * t1:.1f} ms each on one host core; a proposal is "
                      f"2*nz = {2 * nz} of them (misfit and the reference's table copies not counted).  The reference program itself "
                      f"cannot run this configuration: its four tables ttt[nz][nz][nxmod] (src/mcmc_eq.c:525-528) are 36 GB per chain"}
    line = {"metric": B.METRIC, "value": value, "unit": B.UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": W, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong" if not args.chains else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config, "clocks": clk, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": base,
            "parity_check": parity, "tempering": {"rounds": args.steps, "swaps_this_rank": int(swaps), "swap_round_us": 1000.0 * float(np.median(swap_ms)),
                                                  "ladder": [float(x) for x in ladder], "transport": "ncclAllGather" if dist is not None else "one GPU"},
            "generic_kernel": generic, "acceptance_rate": float(counts[:, 17].sum()) / max(float(counts[:, 17].sum() + counts[:, 18].sum()), 1.0),
            "median_rms_s": float(np.median(rms))}
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    if not ok:
        sys.exit(3)
