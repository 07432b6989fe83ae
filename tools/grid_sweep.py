"""P_full on planes of growing depth: the pipelined eikonal kernel (MCMCEQ_EIKONAL_PIPE=1) against the fused one (=0).

    python tools/grid_sweep.py --out DIR [--nz 62,63,94,121,123,126,127] [--example2] [--chains 1024] [--repeats 3]

Every plane spans the Example extent (200 x 200 x 62 nodes at h = 2 km: x, y in [-200, 198] km, z in [-4, 118] km) at the
spacing h = 122 km / (nz - 1), with the bench workload's 200 events x 50 stations (synth.workload); --example2 adds the
Example2 inputs at h = 0.25 km (plane 272 x 121).  Each (plane, kernel setting, repeat) runs in a subprocess of its own (the
switch is read once per process), the two settings alternating; a run warms up with --warmup P steps, then times --steps P
steps with CUDA events on the library's stream (mq_timer) and the eikonal launches with mq_profile, reads the kernel taken
from mq_profile_kernels, and checks 4 chains against the CPU oracle (tests/test_bench_scale_gpu.py: predictions, class sums,
origin times, receiver rows), so that a fast but wrong plane does not pass.  The environment passes through to the
subprocesses (MCMCEQ_LIB, MCMCEQ_PIPE_LC, ...).  Writes DIR/runs.jsonl (one line per run), DIR/summary.json and
DIR/summary.md (median and spread of the repeats per plane and setting), with the card name and power limit."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CHILD = r"""
import json, sys, tempfile
import numpy as np
sys.path.insert(0, %r)
import mcmc_eq_b200 as mq
from mcmc_eq_b200 import synth
from tests import inputs, test_bench_scale_gpu as tb
a = json.loads(sys.argv[1])
if a["plane"] == "example2":
    d = tempfile.mkdtemp(prefix="mqsweep_")
    cfgp, pkp = inputs.materialise("example2", d, h=0.25, nx=193, ny=193, nz=121)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
else:
    cfg, pk, _truth = synth.workload(200, 50, 33, 0, j_max_start=0, j_max_main=2**30, deci=2**30, **a["grid"])
n = a["chains"]
smp = mq.Sampler(cfg, pk, n, 0, 1000)
smp.init_chains()
for _ in range(a["warmup"]):
    smp.step(1, "P")
smp.sync()
smp.profile(True)
smp.timer_start(0)
for _ in range(a["steps"]):
    smp.step(1, "P")
ms = smp.timer_stop(0)
smp.sync()
eik_ms, eik_n, per_launch = smp.profile(False)
kernels = {k: v[0] for k, v in smp.profile_kernels().items()}
m = smp.get_models()
mf, origin = smp.forward_host(m, 3)
chains = [0, n // 3, 2 * n // 3, n - 1]
try:
    worst = tb._check(cfg, pk, smp, m, mf, origin, chains)
    parity = dict(ok=True, chains=chains, **worst)
except AssertionError as e:
    parity = dict(ok=False, chains=chains, error=str(e)[:300])
nodes = smp.nxmod * cfg.grid.nz
print(json.dumps(dict(nxmod=smp.nxmod, nz=cfg.grid.nz, ms=ms, eik_ms=eik_ms, eik_launches=eik_n, solves_per_launch=per_launch,
                      kernels=kernels, parity=parity, nodes=nodes)))
smp.close()
"""


def example_extent(nz: int) -> dict:
    h = 122.0 / (nz - 1)
    n = 1 + int(round(398.0 / h))
    return dict(h=h, nx=n, ny=n, nz=nz, x0=-200.0, y0=-200.0, z0=-4.0)


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown (nvidia-smi failed)"


def run_one(plane, grid, pipe: str, args) -> dict:
    env = dict(os.environ, MCMCEQ_EIKONAL_PIPE=pipe)
    a = dict(plane=plane, grid=grid, chains=args.chains, warmup=args.warmup, steps=args.steps)
    r = subprocess.run([sys.executable, "-c", CHILD % ROOT, json.dumps(a)], env=env, capture_output=True, text=True, timeout=3600)
    if r.returncode != 0:
        return dict(plane=plane, pipe=pipe, failed=True, stderr=r.stderr[-1500:])
    res = json.loads(r.stdout.strip().splitlines()[-1])
    launches = max(res["eik_launches"], 1)
    eik_launch_ms = res["eik_ms"] / launches
    res.update(plane=plane, pipe=pipe, failed=False, eik_ms_per_launch=eik_launch_ms,
               us_per_solve=1000.0 * eik_launch_ms / res["solves_per_launch"],
               node_updates_per_s=res["solves_per_launch"] * res["nodes"] / (eik_launch_ms / 1000.0),
               proposals_per_s=args.chains * args.steps / (res["ms"] / 1000.0))
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--nz", default="62,63,94,121,123,126,127")
    ap.add_argument("--example2", action="store_true", help="add the Example2 inputs at h = 0.25 km (plane 272 x 121)")
    ap.add_argument("--pipe", default="1,0", help="kernel settings to alternate (MCMCEQ_EIKONAL_PIPE values)")
    ap.add_argument("--chains", type=int, default=1024)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--tag", default="", help="label of this sweep in the summary (e.g. the library variant)")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    card = gpu_info()
    planes = [(f"example_nz{nz}", example_extent(int(nz))) for nz in args.nz.split(",") if nz]
    if args.example2:
        planes.append(("example2", None))
    settings = args.pipe.split(",")
    runs = []
    with open(os.path.join(args.out, "runs.jsonl"), "a") as f:
        for plane, grid in planes:
            for rep in range(args.repeats):
                for pipe in (settings if rep % 2 == 0 else settings[::-1]):
                    res = run_one(plane, grid, pipe, args)
                    res.update(repeat=rep, tag=args.tag, card=card)
                    runs.append(res)
                    f.write(json.dumps(res) + "\n")
                    f.flush()
                    print(plane, "pipe", pipe, "rep", rep, "FAILED" if res["failed"] else
                          f"{res['kernels']} {res['eik_ms_per_launch']:.2f} ms/launch parity {res['parity']['ok']}", flush=True)
    rows = []
    for plane, _grid in planes:
        for pipe in settings:
            rs = [r for r in runs if r["plane"] == plane and r["pipe"] == pipe and not r["failed"]]
            if not rs:
                rows.append(dict(plane=plane, pipe=pipe, failed=True))
                continue
            e = sorted(r["eik_ms_per_launch"] for r in rs)
            p = sorted(r["proposals_per_s"] for r in rs)
            med = e[len(e) // 2]
            rows.append(dict(plane=plane, pipe=pipe, failed=False, plane_shape=f"{rs[0]['nxmod']} x {rs[0]['nz']}",
                             kernels=sorted({k for r in rs for k in r["kernels"]}), repeats=len(rs),
                             eik_ms_median=med, eik_ms_min=e[0], eik_ms_max=e[-1],
                             us_per_solve=1000.0 * med / rs[0]["solves_per_launch"],
                             node_updates_per_s=rs[0]["solves_per_launch"] * rs[0]["nodes"] / (med / 1000.0),
                             proposals_per_s_median=p[len(p) // 2], parity_ok=all(r["parity"]["ok"] for r in rs)))
    summary = dict(card=card, tag=args.tag, chains=args.chains, steps=args.steps, warmup=args.warmup, rows=rows)
    with open(os.path.join(args.out, "summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    lines = [f"card, power limit: {card}; {args.chains} chains, {args.steps} timed P steps after {args.warmup}; {args.tag}", "",
             "| plane | nxmod x nz | PIPE | kernel | eikonal ms/launch (median, min - max) | us/solve | node updates/s | P_full proposals/s | parity |",
             "|---|---|---|---|---|---|---|---|---|"]
    for r in rows:
        if r["failed"]:
            lines.append(f"| {r['plane']} | | {r['pipe']} | FAILED | | | | | |")
            continue
        lines.append(f"| {r['plane']} | {r['plane_shape']} | {r['pipe']} | {', '.join(r['kernels'])} | {r['eik_ms_median']:.2f} "
                     f"({r['eik_ms_min']:.2f} - {r['eik_ms_max']:.2f}) | {r['us_per_solve']:.3f} | {r['node_updates_per_s']:.3g} | "
                     f"{r['proposals_per_s_median']:.0f} | {'ok' if r['parity_ok'] else 'FAILED'} |")
    with open(os.path.join(args.out, "summary.md"), "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
