"""Reciprocal travel-time tables against parity tables on the GPU (mq_set_tables; DESIGN.md sections 3 and 6).

    python tools/recip_bench.py [--out FILE.json] [--steps K] [--mix M] [--sample S] [--only config3,config4_shard,fine]

Cases: config 3 (1024 chains x 200 events x 50 stations, Example grid 282 x 62), one 1024-chain shard of config 4
(2000 events x 100 stations on the same grid) and the 0.1 km fine grid (565 x 2001, a few chains).  Per case and mode:
  * P_full: proposals/s of 'P' steps (both tables of every chain rebuilt, then the full misfit), device-timed;
  * eikonal ms per launch and the kernel taken (mq_profile / mq_profile_kernels), misfit ms per launch (mq_profile_misfit);
and once per case the per-pick |t_pred(reciprocal) - t_pred(parity)| (max, mean, p99) on S sampled chains, evaluated on
the same models in both modes after M mixed iterations (the config's proposal strings) of a reciprocal sampler, so that
the models look like posterior models.  Prints one JSON object (and writes it to --out); the GPU's name and power limit
are part of it.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = {
    "config3": dict(chains=1024, events=200, stations=50, fine=False),
    "config4_shard": dict(chains=1024, events=2000, stations=100, fine=False),
    "fine": dict(chains=8, events=200, stations=50, fine=True),
}


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().split("\n")[0]
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def timed_p(smp, steps):
    """K 'P' steps -> (ms per step, eikonal ms per launch, launches, solves per full launch, kernels, misfit ms per launch)."""
    smp.profile(True)
    smp.sync()
    smp.timer_start(0)
    for _ in range(steps):
        smp.step(1, "P")
    ms = smp.timer_stop(0)
    smp.sync()
    eik_ms, eik_n, spl = smp.profile(False)
    mis_n, mis_ms = smp.profile_misfit()
    return dict(ms_per_step=ms / steps, eikonal_ms_per_launch=eik_ms / max(eik_n, 1), eikonal_launches=eik_n,
                solves_per_launch=spl, kernels=smp.profile_kernels(), misfit_ms_per_launch=mis_ms / max(mis_n, 1))


def run_case(name, case, steps, mix, n_sample, warmup=2):
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    n = case["chains"]
    cfg, pk, _truth = synth.workload(case["events"], case["stations"], 33, 0, fine=case["fine"], j_max_start=0, j_max_main=2**30,
                                     deci=2**30)
    out = {"chains": n, "events": case["events"], "stations": case["stations"], "picks": int(pk.n_picks),
           "grid": f"{cfg.grid.nx}x{cfg.grid.ny}x{cfg.grid.nz}, h = {cfg.grid.h} km"}
    # ---- P_full per mode (each mode on its own chains, same seed)
    for mode in ("parity", "reciprocal"):
        smp = mq.Sampler(cfg, pk, n, 0, 1000)
        smp.set_tables(mode)
        smp.init_chains()
        for _ in range(warmup):
            smp.step(1, "P")
        r = timed_p(smp, steps)
        r["p_full"] = n / (r["ms_per_step"] / 1000.0)
        out[mode] = r
        if mode == "reciprocal":
            out["n_rows"] = int(r["solves_per_launch"] // (2 * n))
            # ---- mixing, then the models every chain holds, for the error measurement
            t0 = time.time()
            smp.step(mix, None)
            smp.sync()
            out["mix_iterations"] = mix
            out["mix_s"] = time.time() - t0
            models = smp.get_models()
        smp.close()
    out["speedup_p_full"] = out["reciprocal"]["p_full"] / out["parity"]["p_full"]
    # ---- per-pick error on sampled chains: the same models through both modes
    rng = np.random.default_rng(5)
    sample = sorted(int(c) for c in rng.choice(n, size=min(n_sample, n), replace=False))
    tp = {}
    for mode in ("parity", "reciprocal"):
        smp = mq.Sampler(cfg, pk, n, 0, 1000)
        smp.set_tables(mode)
        smp.forward_host(models, 3)
        tp[mode] = np.stack([smp.predictions(c)[1] for c in sample]).astype(np.float64)
        smp.close()
    ok = (tp["parity"] < 1e29) & (tp["reciprocal"] < 1e29)
    e = np.abs(tp["reciprocal"] - tp["parity"])[ok]
    dims = models.dim[sample]
    out["error"] = {"chains": len(sample), "picks": int(e.size), "max_s": float(e.max()), "mean_s": float(e.mean()),
                    "p99_s": float(np.percentile(e, 99)), "mean_layers": float(np.mean(dims)),
                    "picks_outside_table": int((~ok).sum())}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--mix", type=int, default=1500)
    ap.add_argument("--sample", type=int, default=64)
    ap.add_argument("--only", default=",".join(CASES))
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "cases": {}}
    for name in args.only.split(","):
        case = CASES[name]
        steps = 3 if case["fine"] else args.steps
        mix = min(args.mix, 300) if case["fine"] else args.mix
        res["cases"][name] = run_case(name, case, steps, mix, args.sample)
        print(name, json.dumps(res["cases"][name]), file=sys.stderr, flush=True)
    text = json.dumps(res)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
