"""Cost of the convergence diagnostics (mq_diag_*, DESIGN.md section 4d), three measurements:

  step    device time per round of `chunk` P_mix iterations (the configuration's balanced strings, desynchronised
          stepping) with and without diagnostics, config 3 inputs (synth.workload(200, 50)) at each --chains count, deci 25,
          each round drained as the command line drains (mq_drain_begin, a writer thread finishes the batch; the
          tools/output_bench.py workload).  Off and on alternate in fresh subprocesses, --repeats times each.
  summary mq_diag_summary at config 3 (1024 chains x 200 events x 50 stations) and config 4 (8192 x 2000 x 100), K = 16,
          after enough iterations (deci 1) that every chain has its slots filled; median of --calls calls, host clock
          around a call that ends in a device synchronise.  Bytes: the accumulators the summary reads (ref, the k_c sums and
          2 floor(k_c/2) sums of squares of every used chain) and the sequence means it writes and reads again.
  state   state size, mq_state_save and mq_state_load with diagnostics on, config 3.

The GPU's name and power limit are read in the same run.

    python tools/diag_bench.py [--chains 1024,8192] [--rounds 4] [--repeats 2] [--calls 5] [--out result.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CONFIGS = {3: (1024, 200, 50), 4: (8192, 2000, 100)}


def gpu_info() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().split("\n")[0]
        name, power = [x.strip() for x in q.split(",")]
        return dict(gpu=name, power_limit=power)
    except Exception as e:   # the numbers still stand, without their attribution
        return dict(gpu=f"unknown ({e})", power_limit="unknown")


def step_child(n: int, diag: bool, rounds: int, chunk: int = 100) -> dict:
    """One process: ms per round of `chunk` iterations + drain, diagnostics on or off."""
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    cfg, pk, _ = synth.workload(200, 50, 33, 0, j_max_start=0, j_max_main=2**30, deci=25)
    smp = mq.Sampler(cfg, pk, n, 0, 1000)
    smp.set_ring(8)
    if diag:
        smp.diag_begin(0, 16)
    smp.init_chains()
    smp.step(chunk)
    smp.drain()
    threads, stats = [], dict(records=0, lost=0)

    def finish(batch):
        recs, lost = smp.drain_finish(batch)
        stats["records"] += len(recs)
        stats["lost"] += lost

    smp.sync()
    smp.timer_start(5)
    for _ in range(rounds):
        smp.step(chunk)
        if len(threads) >= 2:
            threads.pop(0).join()
        t = threading.Thread(target=finish, args=(smp.drain_begin(),))
        t.start()
        threads.append(t)
    ms = smp.timer_stop(5)
    for t in threads:
        t.join()
    out = dict(ms_per_round=ms / rounds, records=stats["records"], lost=stats["lost"])
    if diag:
        out["diag_models"] = int(smp.diag_summary()["n_models"])
    smp.close()
    return out


def step_bench(chains: list[int], rounds: int, repeats: int) -> list[dict]:
    res = []
    for n in chains:
        runs = {False: [], True: []}
        for _ in range(repeats):
            for diag in (False, True):
                r = subprocess.run([sys.executable, __file__, "--child", f"{n},{int(diag)},{rounds}"], capture_output=True,
                                   text=True, timeout=1800)
                if r.returncode != 0:
                    raise RuntimeError(r.stderr[-2000:])
                runs[diag].append(json.loads(r.stdout.strip().split("\n")[-1]))
        off = [x["ms_per_round"] for x in runs[False]]
        on = [x["ms_per_round"] for x in runs[True]]
        res.append(dict(chains=n, iterations_per_round=100, deci=25, rounds=rounds, ms_per_round_off=off, ms_per_round_on=on,
                        overhead=statistics.median(on) / statistics.median(off) - 1.0,
                        lost=sum(x["lost"] for x in runs[False] + runs[True]), diag_models=runs[True][-1]["diag_models"]))
    return res


def summary_bench(config: int, calls: int, state: bool) -> dict:
    import numpy as np
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    from mcmc_eq_b200._lib import check, lib, dp, ip, lp
    n, ne, ns = CONFIGS[config]
    cfg, pk, _ = synth.workload(ne, ns, 33, 0, j_max_start=0, j_max_main=2**30, deci=1)
    smp = mq.Sampler(cfg, pk, n, 0, 1)
    dims = smp.diag_begin(0, 16)
    smp.init_chains()
    smp.step(64)
    smp.drain()
    Q, K = dims.n_quantities, dims.n_batches
    k = np.zeros(n, np.int32)
    check(lib().mq_diag_chains(smp.h, None, None, None, None, k.ctypes.data_as(ip), None))
    used = k[k >= 4].astype(np.int64)
    read_acc = int(Q * 8 * (used + 1 + 2 * (used // 2)).sum())
    mu_bytes = int(2 * 2 * Q * 8 * len(used))            # written by pass 1, read by pass 3
    mean, sd, rhat, ess = (np.zeros(Q) for _ in range(4))
    N, cu = C.c_int64(0), C.c_int32(0)
    args = [smp.h, 0] + [a.ctypes.data_as(dp) for a in (mean, sd, rhat, ess)] + [C.byref(N), C.byref(cu)]
    check(lib().mq_diag_summary(*args))                  # warm-up (and the work space)
    times = []
    for _ in range(calls):
        t0 = time.perf_counter()
        check(lib().mq_diag_summary(*args))
        times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    out = dict(config=config, chains=n, events=ne, stations=ns, quantities=Q, n_batches=K,
               accumulator_bytes=int(n * Q * (2 * K + 1) * 8 + 16 * n), chains_used=int(cu.value), n_models=int(N.value),
               full_batches_min=int(k.min()), full_batches_max=int(k.max()), summary_ms=round(1e3 * t, 3),
               summary_ms_all=[round(1e3 * x, 3) for x in times], bytes_read_accumulators=read_acc, bytes_mu=mu_bytes,
               gbps_accumulators=round(read_acc / t / 1e9, 1), gbps_all=round((read_acc + mu_bytes) / t / 1e9, 1))
    if state:
        size = C.c_uint64(0)
        check(lib().mq_state_size(smp.h, C.byref(size)))
        buf = C.create_string_buffer(size.value)
        got = C.c_uint64(0)
        check(lib().mq_state_save(smp.h, buf, size.value, C.byref(got)))
        check(lib().mq_state_load(smp.h, buf, got.value))
        save, load = [], []
        for _ in range(3):
            t0 = time.perf_counter()
            check(lib().mq_state_save(smp.h, buf, size.value, C.byref(got)))
            save.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            check(lib().mq_state_load(smp.h, buf, got.value))
            load.append(time.perf_counter() - t0)
        out.update(state_bytes=int(got.value), state_save_ms=round(1e3 * statistics.median(save), 2),
                   state_load_ms=round(1e3 * statistics.median(load), 2))
    smp.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", default="1024,8192")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--configs", default="3,4")
    ap.add_argument("--skip-step", action="store_true")
    ap.add_argument("--child")
    ap.add_argument("--out")
    a = ap.parse_args()
    if a.child:
        n, diag, rounds = (int(x) for x in a.child.split(","))
        print(json.dumps(step_child(n, bool(diag), rounds)))
        return
    res = dict(gpu_info())
    res["summary"] = [summary_bench(int(c), a.calls, state=int(c) == 3) for c in a.configs.split(",")]
    if not a.skip_step:
        res["step"] = step_bench([int(x) for x in a.chains.split(",")], a.rounds, a.repeats)
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
