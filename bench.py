#!/usr/bin/env python
"""bench.py -- MCMC proposals/s including the full FD travel-time forward, on N B200s of one node.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --gpus 1 --steps K --warmup W      # the reference's own CPU path

Workload (BASELINE.json configs[2], SURVEY.md section 8d item 3): 1024 chains per GPU x 200 events x 50
stations (20 000 picks), Example grid (282 x 62 eikonal plane), models of up to 20 layers.  A step is one
Metropolis-Hastings iteration of every chain with a velocity-model proposal ('P': both travel-time tables are
rebuilt = 2*nz eikonal solves, then the full misfit) -- "P_full" of SURVEY.md section 8d.  Chains are
independent, so N GPUs run N*1024 chains with no data-path collective (weak scaling).

value = whole-job proposals/s with the chain state resident in HBM (device-timed, max over ranks);
e2e   = forward evaluations/s through the batched drop-in of cal_fit_newx (mq_forward_host): models are
        copied from pinned host memory every call and the class sums + origin times are read back.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mcmc_proposals_per_sec_incl_fd_traveltime_forward"
UNIT = "proposals/s"
SMEM_PEAK_GBS = 148 * 128 * 1.965   # 148 SM x 128 B/clk x 1.965 GHz = 37.2 TB/s (SURVEY.md section 8d)


def kernel_traffic(kernel, solves_per_launch):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture (profiles/traffic.json:
    dram__bytes_read.sum + dram__bytes_write.sum of one launch of the same workload), scaled to this run's launch size."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    t = json.load(open(p)).get(kernel)
    if not t:
        return None
    return float(t["dram_bytes_per_launch"]) * solves_per_launch / float(t["solves_per_launch"])


def kernel_instructions(kernel, solves_per_launch):
    """Warp instructions per launch of the dominant kernel (smsp__inst_executed.sum of the same ncu capture), scaled."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    t = json.load(open(p)).get(kernel)
    if not t or "warp_instructions_per_launch" not in t:
        return None
    return float(t["warp_instructions_per_launch"]) * solves_per_launch / float(t["solves_per_launch"])


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def torch_sm_count(device):
    import torch
    return torch.cuda.get_device_properties(device).multi_processor_count


class ClockSampler:
    """SM clock, power and throttle reasons sampled through NVML every 10 ms while the timed region runs
    (nvidia-smi -lms as the fallback when the NVML binding is missing)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}

    def __init__(self, index):
        self.index, self.proc, self.rows, self.stop_flag, self.t, self.nvml = index, None, [], False, None, None

    def _nvml_loop(self):
        n, h = self.nvml
        while not self.stop_flag:
            try:
                sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
                pw = n.nvmlDeviceGetPowerUsage(h) / 1000.0
                try:
                    rs = n.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((float(sm), pw, int(rs)))
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        try:
            import pynvml as n
            n.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.index
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                idx = int(vis.split(",")[self.index])
            h = n.nvmlDeviceGetHandleByIndex(idx)
            self.max_sm = float(n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM))
            self.nvml = (n, h)
            self.t = threading.Thread(target=self._nvml_loop, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag = True
            self.t.join(timeout=1)
            if not self.rows:
                return None
            sm = sorted(r[0] for r in self.rows)
            reasons = [k for k, b in self.BITS.items() if any(r[2] & b for r in self.rows)]
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_sm, "power_w_max": max(r[1] for r in self.rows),
                    "samples": len(self.rows), "reasons": reasons, "source": "nvml, 10 ms"}
        if not self.proc:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = [r for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not rows:
            return None
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "power_w_max": max(float(r[2]) for r in rows),
                "samples": len(rows), "reasons": reasons, "source": "nvidia-smi -lms 50"}


def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def barrier_max(dist, value, device):
    """barrier + max over ranks of a python float"""
    if dist is None:
        return value
    import torch
    t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{device}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------------------------------------------
# the reference's own CPU path: oracle/_ref/mcmc_eq (unmodified sources, gcc -O4), one process per host core
# ------------------------------------------------------------------------------------------------------
def reference_exe():
    p = os.path.join(ROOT, "oracle", "_ref", "mcmc_eq")
    return p if os.path.exists(p) else None


def count_proposals(text):
    """Iterations of src/mcmc_eq.c:845 a chain file reports: the sum of the accepted / rejected pairs of its `cnt ... a/r`
    lines (src/mcmc_eq.c:1199-1207)."""
    n = 0
    for ln in text.split("\n"):
        if ln.startswith("cnt") and "a/r" in ln:
            a, r = ln.split()[-2:]
            n += int(a) + int(r)
    return n


def run_reference_batch(workdir, exe, cfg_dict, procs_n, accepted, seed0, string, picks="picks"):
    """`procs_n` concurrent chains of `accepted` accepted models each, proposal string `string` in both phases
    (None: the config's own strings).  Returns (proposals, wall seconds)."""
    from mcmc_eq_b200.io import write_config
    procs = []
    t0 = time.perf_counter()
    for k in range(procs_n):
        cfgp = os.path.join(workdir, f"cfg_{k}.dat")
        a = max(1, accepted // 3)
        over = dict(j_max_start=a, j_max_main=max(1, accepted - a), deci=10**8, true_random=seed0 + k)
        if string:
            over.update(dstring_start=string, dstring_main=string)
        write_config(cfg_dict, cfgp, **over)
        cmd = [exe, cfgp, os.path.join(workdir, f"rjx-{k:03d}.out"), os.path.join(workdir, picks)]
        if shutil.which("taskset"):
            cmd = ["taskset", "-c", str(k % (os.cpu_count() or 1))] + cmd
        procs.append(subprocess.Popen(cmd, cwd=workdir, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
    for p in procs:
        p.wait()
    wall = time.perf_counter() - t0
    proposals = 0
    for k in range(procs_n):
        proposals += count_proposals(open(os.path.join(workdir, f"rjx-{k:03d}.out")).read())
    return proposals, wall


def oracle_port_batch(cfg, pk, truth, seconds):
    """Fallback when the compiled reference is absent: time the oracle port (1 core) of a full forward."""
    from tests import fwd_helpers as fh
    t0 = time.perf_counter()
    n = 0
    while time.perf_counter() - t0 < seconds:
        fh.oracle_forward(cfg, pk, truth["z"], truth["vp"], truth["vpvs"], truth["eq"], truth["pres"], truth["sres"])
        n += 1
    return n, time.perf_counter() - t0


def cpu_timed(exe, d, cd, cores, accepted, string, budget_s, steps=1, warmup=0, seed0=2000):
    """Batches of `cores` fresh reference chains until `budget_s` is used; -> (proposals, wall, batches) of the timed steps."""
    per_step = budget_s / max(steps + warmup, 1)
    tot_p, tot_w, batches = 0, 0.0, 0
    for s in range(warmup + steps):
        t_step, k = 0.0, 0
        while t_step < per_step * 0.85 or k == 0:
            p, w = run_reference_batch(d, exe, cd, cores, accepted, seed0 + 1000 * s + 17 * k, string)
            t_step += w
            k += 1
            if s >= warmup:
                tot_p += p
                tot_w += w
                batches += 1
    return tot_p, tot_w, batches


def cpu_baseline(cfg, pk, truth, budget_s, steps=1, warmup=0, string="P", accepted=40):
    """Reference CPU path on this box's host cores, bounded sample.  -> dict for the JSON line + wall seconds."""
    from mcmc_eq_b200.io import config_to_dict, write_picks
    exe = reference_exe()
    cores = os.cpu_count() or 1
    if exe is None:
        n, wall = oracle_port_batch(cfg, pk, truth, min(budget_s, 20.0))
        return {"value": n / wall, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": f"{n} full forwards (2*nz eikonal solves + misfit) of the oracle port, one chain, {wall:.1f} s"}, wall
    d = tempfile.mkdtemp(prefix="mqref_")
    try:
        write_picks(pk, os.path.join(d, "picks"), truth["t64"])
        cd = config_to_dict(cfg)
        # The reference's loop counter is ACCEPTED models (src/mcmc_eq.c:845), so the run time of a long chain is not
        # bounded by its configuration.  Bounded sample: short fresh chains (`accepted` accepted models each, one process
        # per core), batch after batch until the time budget of a step is used; proposals = sum of the cnt a/r lines.
        tot_p, tot_w, batches = cpu_timed(exe, d, cd, cores, accepted, string, budget_s, steps, warmup)
        per_proc = tot_p / max(batches * cores, 1)
        return {"value": tot_p / tot_w, "unit": UNIT, "cores": cores, "kind": "reference",
                "sample": f"{batches} batch(es) of {cores} concurrent unmodified mcmc_eq processes (gcc -O4, one per core, fresh "
                          f"chains of {accepted} accepted models), proposal string '{string or 'config line 33'}' on the same "
                          f"synthetic picks: {tot_p} proposals in {tot_w:.1f} s; each process's start-up (exec, pick parsing and "
                          f"the initial forward = one full-forward proposal's worth of work) is inside the wall time: about "
                          f"1/{per_proc + 1:.0f} of it for the {per_proc:.0f} proposals a process makes"}, tot_w
    finally:
        shutil.rmtree(d, ignore_errors=True)


def cpu_small(name, budget_s):
    """Configs 1-2 the way the reference runs them: 10 concurrent chains on the shipped example inputs (P_mix)."""
    from tests import inputs
    exe = reference_exe()
    if exe is None:
        return None
    d = tempfile.mkdtemp(prefix="mqref_")
    try:
        cfg_d, arr = inputs.load(name)
        inputs.write_picks(arr, os.path.join(d, "picks"))
        t0, tot_p, tot_w, k = time.perf_counter(), 0, 0.0, 0
        while time.perf_counter() - t0 < budget_s * 0.7 or k == 0:
            p, w = run_reference_batch(d, exe, cfg_d, 10, 240, 500 + 31 * k, cfg_d["dstring_main"])
            tot_p += p; tot_w += w; k += 1
        return {"value": tot_p / tot_w, "unit": UNIT, "chains": 10, "cores": min(10, os.cpu_count() or 1),
                "sample": f"{k} batch(es) of 10 concurrent unmodified mcmc_eq processes, 240 accepted models each, main-phase string"}
    finally:
        shutil.rmtree(d, ignore_errors=True)


# ------------------------------------------------------------------------------------------------------
# pieces of the repo arm
# ------------------------------------------------------------------------------------------------------
def timed_steps(smp, dist, device, steps, iters, proposals):
    """K steps, device-timed on the library's stream, max over ranks.  -> (ms, eik_ms, eik_n, solves_per_launch, kernels)"""
    smp.profile(True)
    barrier_max(dist, 0.0, device)
    smp.sync()
    smp.timer_start(0)
    for _ in range(steps):
        smp.step(iters, proposals)
    ms = smp.timer_stop(0)
    smp.sync()
    ms = barrier_max(dist, ms, device)
    eik_ms, eik_n, solves_per_launch = smp.profile(False)
    return ms, eik_ms, eik_n, solves_per_launch, smp.profile_kernels()


DUMP_LIMIT_BYTES = 60 * 10**6


def dump_outputs(smp, stats, out_dir, seed=0):
    """What the timed steps left for a caller of mq_step, written as out_dir/<name>.npy: the chain states (mq_get_models),
    the per-chain statistics `stats` = smp.stats() and the tempering betas.  Integers are written as float64; nucleus slots past a
    chain's dimension are not part of its model and are written as 0.  When all chains would take more than
    DUMP_LIMIT_BYTES, a seeded sample of chains is written, the same for every run; chain.npy holds their indices."""
    m = smp.get_models()
    counts, ll, rms = stats
    live = np.arange(m.md)[None, :] < m.dim[:, None]
    out = {"dim": m.dim.astype(np.float64), "z": np.where(live, m.z, np.float32(0)), "vp": np.where(live, m.vp, np.float32(0)),
           "vpvs": np.where(live, m.vpvs, np.float32(0)), "eq": m.eq, "origin": m.origin, "pres": m.pres, "sres": m.sres,
           "noise": m.noise, "counts": counts.astype(np.float64), "loglik": ll, "rms": rms, "beta": smp.get_beta()}
    per_chain = 8 + sum(a.nbytes for a in out.values()) // smp.n
    keep = min(smp.n, DUMP_LIMIT_BYTES // per_chain)
    idx = np.arange(smp.n) if keep == smp.n else np.sort(np.random.default_rng(seed).choice(smp.n, keep, replace=False))
    out["chain"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a if name == "chain" else a[idx])


def roofline_block(cfg, smp, ms, eik_ms, eik_n, solves_per_launch, kernels, clk, device, n_rows):
    """Roofline of the dominant kernel (eikonal) from the live CUDA-event time of its launches."""
    nz, nxmod = cfg.grid.nz, smp.nxmod
    alg_bytes_per_solve = 4 * nz + 4 * nxmod * nz            # read nz slownesses, write the field (SURVEY 8d)
    peak, peak_src = measured_peak()
    t_launch = eik_ms / eik_n / 1000.0
    achieved = alg_bytes_per_solve * solves_per_launch / t_launch / 1e9
    smem_alg = 32.0 * nxmod * nz * solves_per_launch / t_launch / 1e9
    # the kernel every counted launch took, as the library reports it (mq_profile_kernels), not as the environment suggests
    kernel = max(kernels.items(), key=lambda kv: kv[1][1])[0] if kernels else "?"
    roofline = {"bound": "hbm", "kernel": kernel, "kernels_launched": {k: v[0] for k, v in kernels.items()},
                "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": kernel_traffic(kernel, solves_per_launch), "peak_source": peak_src,
                "algorithmic_bytes_per_solve": alg_bytes_per_solve, "solves_per_launch": int(solves_per_launch),
                "avg_launch_ms": eik_ms / eik_n, "share_of_step": eik_ms / ms,
                "layout": f"receiver rows only are stored ({n_rows} of {nz} rows); algorithmic bytes count the full field as the reference materialises it",
                "smem": {"achieved": smem_alg, "peak": SMEM_PEAK_GBS, "unit": "GB/s", "frac": smem_alg / SMEM_PEAK_GBS,
                         "algorithmic_bytes_per_node_update": 32}}
    winst = kernel_instructions(kernel, solves_per_launch)
    if winst:
        sm_ghz = float((clk or {}).get("sm_mhz") or 1965.0) / 1000.0
        issue_peak = torch_sm_count(device) * 4 * sm_ghz
        roofline["issue"] = {"achieved": winst / t_launch / 1e9, "peak": issue_peak, "unit": "G warp-instructions/s",
                             "frac": winst / t_launch / 1e9 / issue_peak, "warp_instructions_per_launch": winst,
                             "source": "smsp__inst_executed.sum of the committed ncu capture (profiles/traffic.json)"}
    return roofline


def e2e_block(smp, pk, dist, device, chains, n_gpus, steps):
    """The same metric through the plugin call with HOST buffers: models from pinned memory in, class sums + origins out."""
    import torch
    m = smp.get_models()
    keep = []
    for name in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise", "origin"):
        t = torch.from_numpy(getattr(m, name).copy()).pin_memory()
        keep.append(t)
        setattr(m, name, t.numpy())
    mf_t = torch.zeros((chains, 8), dtype=torch.float32).pin_memory()
    org_t = torch.zeros((chains, pk.n_events), dtype=torch.float32).pin_memory()
    h2d = sum(getattr(m, k).nbytes for k in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise"))
    d2h = mf_t.numpy().nbytes + org_t.numpy().nbytes
    e2e_steps = max(3, min(steps, 10))
    for _ in range(2):
        smp.forward_host(m, 3, mf_t.numpy(), org_t.numpy())
    barrier_max(dist, 0.0, device)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        smp.forward_host(m, 3, mf_t.numpy(), org_t.numpy())      # synchronous: returns with the results on the host
    e2e_s = barrier_max(dist, time.perf_counter() - t0, device)
    return {"value": chains * n_gpus * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
            "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "call": "mq_forward_host(calct=3): batched drop-in of cal_fit_newx"}, m, mf_t.numpy()


def parity_block(cfg, pk, truth, smp, m, mf, n_sample, seed):
    """After the timed region: sampled chains of the benched state against the CPU oracle -- per-pick predictions
    (1e-4 s), class sums (2e-5 relative), stored receiver rows (max(1e-4 s, 2e-6 T)) -- and the synthetic picks'
    noise-free predictions (made by this library) against the oracle's, which the reference arm uses."""
    from tests import fwd_helpers as fh
    rng = np.random.default_rng(seed)
    chains = sorted(int(c) for c in rng.choice(smp.n, size=min(n_sample, smp.n), replace=False))
    max_dt, max_rel, max_row = 0.0, 0.0, 0.0
    ok = True
    for c in chains:
        d = int(m.dim[c])
        rmf, _org, _res, rpred, tabs = fh.oracle_forward(cfg, pk, m.z[c, :d], m.vp[c, :d], m.vpvs[c, :d], m.eq[c], m.pres[c],
                                                          m.sres[c], want_tables=True)
        _r, tpred = smp.predictions(c)
        fin = np.isfinite(rpred) & (np.abs(rpred) < 1e20)
        dt = float(np.abs(tpred[fin] - rpred[fin]).max()) if fin.any() else 0.0
        big = rmf > 0
        rel = float((np.abs(mf[c][big] - rmf[big]) / rmf[big]).max()) if big.any() else 0.0
        if not np.isfinite(rmf).all():      # an event outside the table: both sides must say so
            rel = 0.0 if (np.isfinite(mf[c]) == np.isfinite(rmf)).all() else float("inf")
        max_dt, max_rel = max(max_dt, dt), max(max_rel, rel)
        for ph in (1, 2):
            rows, idx = smp.rows(c, ph)
            ref = tabs[ph - 1][idx]
            err = np.abs(rows - ref)
            tol = np.maximum(1e-4, 2e-6 * np.abs(ref))
            max_row = max(max_row, float(err.max()))
            ok = ok and bool((err <= tol).all())
        ok = ok and dt <= 1e-4 and rel <= 2e-5
    out = {"chains": len(chains), "max_dt": max_dt, "max_rel_class_sum": max_rel, "max_row_dt": max_row,
           "tolerance": "1e-4 s per pick, 2e-5 relative per class sum, max(1e-4 s, 2e-6 T) per stored table node",
           "against": "oracle/ (CPU restatement, bit-identical to the compiled reference)", "ok": ok}
    if truth is not None and "tpred" in truth:
        ref = fh.oracle_forward(cfg, pk, truth["z"], truth["vp"], truth["vpvs"], truth["eq"], truth["pres"], truth["sres"])[3]
        out["synthetic_picks_max_dt"] = float(np.abs(ref - truth["tpred"]).max())
        out["ok"] = out["ok"] and out["synthetic_picks_max_dt"] <= 1e-4
    return out


def pmix_block(smp, dist, device, chains, n_gpus, iters=480):
    """P_mix: the reference's own balanced proposal string (src/mcmc_eq.c:803-834), desynchronised stepping."""
    smp.step(48, None)
    barrier_max(dist, 0.0, device)
    smp.sync()
    smp.timer_start(1)
    smp.step(iters, None)
    ms = barrier_max(dist, smp.timer_stop(1), device)
    return {"value": chains * n_gpus * iters / (ms / 1000.0), "unit": UNIT, "iterations_per_call": iters, "ms_per_iteration": ms / iters,
            "string": "config line 33 balanced as src/mcmc_eq.c:803-834, main phase", "stepping": "desynchronised (bit-identical to lock-step)"}


def small_block(device, with_cpu, budget_s):
    """Configs 1-2: 10 chains on the shipped example inputs (tests/golden copies), P_mix and P_full."""
    import mcmc_eq_b200 as mq
    from tests import inputs
    out = {}
    for name in ("example", "example2"):
        d = tempfile.mkdtemp(prefix="mqsmall_")
        try:
            cfgp, pkp = inputs.materialise(name, d, j_max_start=0, j_max_main=2**30, deci=2**30)
            cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
            smp = mq.Sampler(cfg, pk, 10, device, 7)
            smp.init_chains()
            smp.step(48, None)
            smp.sync()
            smp.timer_start(2)
            smp.step(480, None)
            ms_mix = smp.timer_stop(2)
            smp.timer_start(2)
            for _ in range(20):
                smp.step(1, "P")
            ms_full = smp.timer_stop(2)
            smp.close()
            out[name] = {"chains": 10, "picks": int(pk.n_picks), "p_mix": 10 * 480 / (ms_mix / 1000.0), "p_full": 10 * 20 / (ms_full / 1000.0),
                         "unit": UNIT}
            if with_cpu:
                out[name]["cpu"] = cpu_small(name, budget_s)
        finally:
            shutil.rmtree(d, ignore_errors=True)
    return out


def class_counts(pk):
    """picks per class code 2*class + phase (P picks come first in every event)"""
    ev = np.repeat(np.arange(pk.n_events), np.diff(pk.ev_off))
    is_s = (np.arange(pk.n_picks) - pk.ev_off[:-1][ev]) >= pk.n_p[ev]
    return np.bincount(2 * pk.cls + is_s.astype(np.int64), minlength=8)[:8]


def collectives_block(pk, dist, rank, world, device, seed, n=64):
    """The library's own NCCL paths under the driver's eyes (a 64-chain handle per rank on the same picks, every accepted
    model a record): tempering swap rounds -- one all-gather of (log-likelihood, beta) per chain, identical decisions on
    every rank -- checked against the host statement of the rule (mcmc_eq_b200.dist.swap_plan) on numbers gathered through
    torch.distributed, and the posterior all-reduce checked against the sum of the per-rank accumulators."""
    import torch
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import dist as mqd, synth
    from mcmc_eq_b200._lib import comm_unique_id
    cfg = synth.config(j_max_start=0, j_max_main=2**30, deci=1)
    smp = mq.Sampler(cfg, pk, n, device, seed)
    uid = mqd.exchange_unique_id(dist, comm_unique_id, torch.device("cuda", device))
    smp.comm_init(uid, rank, world)          # also numbers the chains globally: chain offset = rank * n
    smp.posterior_begin(0.05, 0.02, -1)
    smp.init_chains()
    smp.step(8, "QRN")
    smp.drain()
    ok = True
    n_class = class_counts(pk)
    ladder = np.array([1.0, 0.8, 0.64, 0.5, 0.4, 0.32, 0.25, 0.2], np.float32)   # 8 temperatures x replicas, as config 5 asks
    smp.set_beta(ladder[(np.arange(n) + rank * n) % 8].copy())
    rounds, swapped, temper_ms = 6, 0, []
    for r in range(rounds):
        smp.step(2, "QN")
        smp.drain()
        _c, ll, _ = smp.stats()
        full = mqd.full_loglik(ll, smp.get_models().noise, n_class)
        t_ll = torch.tensor(full, dtype=torch.float64, device=f"cuda:{device}")
        t_b = torch.tensor(smp.get_beta(), dtype=torch.float32, device=f"cuda:{device}")
        g_ll = [torch.zeros_like(t_ll) for _ in range(world)]
        g_b = [torch.zeros_like(t_b) for _ in range(world)]
        dist.all_gather(g_ll, t_ll)
        dist.all_gather(g_b, t_b)
        want, _k = mqd.swap_plan(torch.cat(g_ll).cpu().numpy(), torch.cat(g_b).cpu().numpy(), r, seed)
        smp.sync()
        t0 = time.perf_counter()
        swapped += smp.temper_swap(r)        # synchronous: returns with the swap count on the host
        temper_ms.append(1000.0 * (time.perf_counter() - t0))
        ok = ok and bool(np.array_equal(smp.get_beta(), want[rank * n:(rank + 1) * n]))
    smp.set_beta(np.ones(n, np.float32))
    local = smp.posterior_get()
    pack = lambda d: np.concatenate([d["hist_vp"].ravel().astype(np.float64), d["hist_vpvs"].ravel().astype(np.float64),
                                     d["eqsum"].ravel(), d["ressum"].ravel(), d["noisesum"].ravel(), [float(d["n_models"])]])
    t_loc = torch.tensor(pack(local), dtype=torch.float64, device=f"cuda:{device}")
    dist.all_reduce(t_loc)
    smp.sync()
    t0 = time.perf_counter()
    smp.posterior_allreduce()                # two ncclAllReduce (int32 histograms, double moment sums) + a synchronise
    allreduce_ms = 1000.0 * (time.perf_counter() - t0)
    tot = smp.posterior_get()
    ok = ok and bool(np.allclose(pack(tot), t_loc.cpu().numpy(), rtol=1e-12, atol=1e-9)) and tot["n_models"] > 0
    smp.comm_destroy()
    smp.close()
    flag = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device=f"cuda:{device}")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return {"temper_us": 1000.0 * float(np.median(temper_ms)), "temper_rounds": rounds, "temper_swaps_this_rank": int(swapped),
            "allreduce_us": 1000.0 * allreduce_ms, "posterior_models": int(tot["n_models"]), "ranks": world, "chains_per_rank": n,
            "timed": "host wall time of the synchronous call (pack kernel + ncclAllGather + swap kernel + count read-back; "
                     "two ncclAllReduce + synchronise)",
            "checked_against": "mcmc_eq_b200.dist.swap_plan on the all-gathered (log-likelihood, beta); sum of the per-rank accumulators",
            "ok": bool(flag.item() > 0.5)}


# ------------------------------------------------------------------------------------------------------
CONFIG3 = dict(chains=1024, events=200, stations=50)        # BASELINE.json configs[2]: the configuration the metric is quoted on
CONFIG4 = dict(chains=8192, events=2000, stations=100)      # BASELINE.json configs[3]: sharded by chain over 1/2/4/8 GPUs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto", "3", "4", "fine"],
                    help="auto: config 3 (synth-1024) on one GPU, config 4 (synth-8192 sharded by chain, strong scaling) on several")
    ap.add_argument("--chains", type=int, default=0, help="chains per GPU (overrides the configuration's)")
    ap.add_argument("--events", type=int, default=0)
    ap.add_argument("--stations", type=int, default=0)
    ap.add_argument("--proposals", default="P", help="proposal letters of a step (P = full forward recomputation)")
    ap.add_argument("--iters-per-step", type=int, default=1,
                    help="Metropolis-Hastings iterations per chain in one mq_step call (>= 4: desynchronised stepping, for mixed proposal strings)")
    ap.add_argument("--cpu-budget", type=float, default=20.0, help="seconds of host time for the cpu_baseline leg")
    ap.add_argument("--ref-budget", type=float, default=110.0, help="seconds of host time for the headline of --impl reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline, roofline, e2e and parity check only (profiling runs)")
    ap.add_argument("--parity-chains", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the chain states and statistics they computed as DIR/<name>.npy "
                         "(rank 0's chains when several GPUs run)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this library computed: it needs --impl ours")
    W = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        # the reference is a CPU program: rank 0 alone times it, the other ranks leave without joining any group
        rank, world, local, dist = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), 0, None
        if rank != 0:
            return
    else:
        rank, world, local, dist = dist_setup(args.gpus)
    n_gpus = max(world, 1)
    if args.config == "fine":
        import bench_fine
        return bench_fine.main(args, rank, world, local, dist)
    which = args.config if args.config != "auto" else ("3" if n_gpus == 1 else "4")
    base_cfg = CONFIG3 if which == "3" else CONFIG4
    strong = which == "4"
    total_chains = base_cfg["chains"]
    chains = args.chains or (total_chains // n_gpus if strong else total_chains)
    events, stations = args.events or base_cfg["events"], args.stations or base_cfg["stations"]
    scaling = "strong" if (strong and not args.chains) else "weak"
    if which == "3":
        workload = (f"synth-{chains}: {chains} chains/GPU x {events} events x {stations} stations "
                    f"({2 * events * stations} picks), Example grid h=2 km 200x200x62 (eikonal plane 282x62), "
                    f"<=20 layers, proposal '{args.proposals}' (P_full: 2*nz eikonal solves + full misfit per proposal)")
        par = f"chains sharded x{n_gpus}, {chains} per GPU (weak scaling), no data-path collective"
    else:
        workload = (f"synth-8192 sharded: {chains * n_gpus} chains in total = {chains} chains/GPU on {n_gpus} GPU(s) x {events} events x "
                    f"{stations} stations ({2 * events * stations} picks), Example grid h=2 km 200x200x62 (eikonal plane 282x62), "
                    f"<=20 layers, proposal '{args.proposals}' (P_full: 2*nz eikonal solves + full misfit per proposal)")
        par = f"{chains * n_gpus} chains sharded by chain over {n_gpus} GPU(s) ({scaling} scaling), no data-path collective"
    config = {"workload": workload, "baseline_config": f"configs[{2 if which == '3' else 3}]", "chains_per_gpu": chains, "events": events,
              "stations": stations, "grid": "282x62", "proposal_string": args.proposals, "iterations_per_step": args.iters_per_step,
              "parallelism": par,
              "l2": "per-step working set (tables 0.9 MB per chain + solver scratch > 1 GB per GPU) exceeds the 126 MB L2"}

    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth

    if args.impl == "reference":
        def oracle_predict(cfg, pk0, st):   # synthetic picks without touching the GPU library
            from tests import fwd_helpers as fh
            return fh.oracle_forward(cfg, pk0, st["z"], st["vp"], st["vpvs"], st["eq"], st["pres"], st["sres"])[3]
        cfg, pk, truth = synth.workload(events, stations, 33, 0, predictor=oracle_predict)
        base, wall = cpu_baseline(cfg, pk, truth, args.ref_budget, steps=max(args.steps, 1), warmup=args.warmup)
        line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1000.0 * wall / max(args.steps, 1), "higher_is_better": True,
                "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": base, "gpu_launches": 0,
                "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        if not args.no_extras:
            # CPU counterparts of the repo arm's extra keys: P_mix on the same picks, and configs 1-2 (10 chains)
            pm, _ = cpu_baseline(cfg, pk, truth, 25.0, string=synth.EXAMPLE_LIKE["dstring_main"], accepted=200)
            line["p_mix"] = pm
            line["small"] = {name: cpu_small(name, 15.0) for name in ("example", "example2")}
        print(json.dumps(line))
        return

    device = local
    cfg, pk, truth = synth.workload(events, stations, 33, device, j_max_start=0, j_max_main=2**30, deci=2**30)
    smp = mq.Sampler(cfg, pk, chains, device, 1000)
    smp.set_chain_offset(rank * chains)     # chain g of the job draws from stream (seed, g) on whichever GPU it runs
    smp.init_chains()
    # the timed steps start from valid chain states W proposals away from the start models, as a fresh reference chain does
    # (the reference arm times fresh chains too); "p_full_after_mixing" repeats the measurement on burned-in chains
    for _ in range(W):
        smp.step(1, args.proposals)
    smp.sync()

    # ---- timed region: K steps, device-timed on the library's stream --------------------------------------
    clocks = ClockSampler(device)
    clocks.start()
    launches0 = mq.lib().mq_launch_count()
    ms, eik_ms, eik_n, solves_per_launch, kernels = timed_steps(smp, dist, device, args.steps, args.iters_per_step, args.proposals)
    launches = mq.lib().mq_launch_count() - launches0
    clk = clocks.stop()
    counts, ll, rms = smp.stats()
    if args.dump_outputs and rank == 0:
        dump_outputs(smp, (counts, ll, rms), args.dump_outputs)
    proposals = chains * n_gpus * args.steps * args.iters_per_step
    value = proposals / (ms / 1000.0)

    # the roofline figure needs the exact number of solves per launch: only a pure 'P' string rebuilds both tables of every
    # chain in every step (V rebuilds one, B/D/M can be ineligible, Q/R/N rebuild none)
    roofline = None
    n_rows = mq.lib().mq_get_rows(smp.h, 0, 1, None, None)
    if eik_n > 0 and set(args.proposals) <= {"P"}:
        roofline = roofline_block(cfg, smp, ms, eik_ms, eik_n, solves_per_launch, kernels, clk, device, n_rows)

    e2e, m_host, mf_host = e2e_block(smp, pk, dist, device, chains, n_gpus, args.steps)

    # ---- parity of what was just timed: sampled chains of the e2e call's models against the CPU oracle ------------
    parity = parity_block(cfg, pk, truth if rank == 0 else None, smp, m_host, mf_host, args.parity_chains if n_gpus == 1 else 2, 77 + rank)
    if dist is not None:
        import torch
        flag = torch.tensor([1.0 if parity["ok"] else 0.0], dtype=torch.float64, device=f"cuda:{device}")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity["ok_all_ranks"] = bool(flag.item() > 0.5)
        parity["chains"] = parity["chains"] * n_gpus

    extras = {}
    if not args.no_extras:
        extras["p_mix"] = pmix_block(smp, dist, device, chains, n_gpus)
        if n_gpus == 1 and set(args.proposals) <= {"P"}:
            # The work of a solve depends on the model (number of layers, contrasts: a one-layer model is a homogeneous
            # medium with analytic solves).  The headline is timed on chains a few proposals away from their start models, as
            # a fresh reference chain is; the same P_full step on the same chains after the mixed iterations above plus 1500
            # more, with the mean number of layers next to it, shows how much that matters.
            smp.step(1500, None)
            k2 = max(3, min(args.steps, 20))
            ms2, e2, n2, _spl2, kern2 = timed_steps(smp, dist, device, k2, 1, "P")
            extras["p_full_after_mixing"] = {"value": chains * k2 / (ms2 / 1000.0), "unit": UNIT, "steps": k2, "ms_per_step": ms2 / k2,
                                             "eikonal_ms_per_launch": e2 / max(n2, 1), "mixed_iterations_before": 48 + 480 + 1500,
                                             "median_rms_s": float(np.median(smp.stats()[2])),
                                             "mean_layers": float(np.mean(smp.get_models().dim)),
                                             "mean_layers_headline": float(np.mean(m_host.dim)),
                                             "kernels_launched": {k: v[0] for k, v in kern2.items()}}
            if roofline and n2 > 0:
                t2 = e2 / n2 / 1000.0
                peak2, _src2 = measured_peak()
                extras["p_full_after_mixing"]["roofline"] = {
                    "hbm_algorithmic_frac": roofline["algorithmic_bytes_per_solve"] * roofline["solves_per_launch"] / t2 / 1e9 / peak2,
                    "smem_algorithmic_frac": 32.0 * smp.nxmod * cfg.grid.nz * roofline["solves_per_launch"] / t2 / 1e9 / SMEM_PEAK_GBS}
        if dist is not None:
            extras["collectives"] = collectives_block(pk, dist, rank, world, device, 1000)
    base = None
    if rank == 0 and n_gpus == 1 and not args.no_cpu_baseline:
        base, _ = cpu_baseline(cfg, pk, truth, args.cpu_budget)
    smp.close()

    if not args.no_extras and rank == 0 and n_gpus == 1:
        extras["small"] = small_block(device, False, 0.0)
    if not args.no_extras and n_gpus == 1 and which == "3" and not args.chains:
        # config 4 on ONE GPU (8192 chains x 2000 events x 100 stations): the N = 1 point of the strong-scaling series that
        # `--gpus N` runs for N > 1
        c4cfg, c4pk, _t = synth.workload(CONFIG4["events"], CONFIG4["stations"], 33, device, j_max_start=0, j_max_main=2**30, deci=2**30)
        s4 = mq.Sampler(c4cfg, c4pk, CONFIG4["chains"], device, 1000)
        s4.init_chains()
        for _ in range(3):
            s4.step(1, "P")
        k4 = max(3, min(args.steps, 10))
        ms4, e4, n4, spl4, kern4 = timed_steps(s4, None, device, k4, 1, "P")
        extras["config4"] = {"workload": "synth-8192 on one GPU: 8192 chains x 2000 events x 100 stations (400 000 picks), P_full",
                             "value": CONFIG4["chains"] * k4 / (ms4 / 1000.0), "unit": UNIT, "steps": k4, "ms_per_step": ms4 / k4,
                             "eikonal_ms_per_launch": e4 / max(n4, 1), "eikonal_share_of_step": e4 / ms4,
                             "kernels_launched": {k: v[0] for k, v in kern4.items()}}
        s4.close()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    acc = float(counts[:, 17].sum()) / max(float(counts[:, 17].sum() + counts[:, 18].sum()), 1.0)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": W,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": config, "clocks": clk, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roofline, "cpu_baseline": base, "parity_check": parity, "acceptance_rate": acc,
            "median_rms_s": float(np.median(rms))}
    line.update(extras)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    if not parity["ok"] or not parity.get("ok_all_ranks", True):
        sys.exit(3)


if __name__ == "__main__":
    main()
