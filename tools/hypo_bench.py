"""Cost of the hypocentre uncertainty accumulators (mq_hypo_*, DESIGN.md section 4e), three measurements:

  step    device time per round of `chunk` P_mix iterations (the configuration's balanced strings, desynchronised
          stepping) with and without the accumulators, config 3 inputs (synth.workload(200, 50)) at each --chains count,
          deci 25, each round drained as the command line drains (mq_drain_begin, a writer thread finishes the batch; the
          tools/diag_bench.py workload).  Off and on alternate in fresh subprocesses, --repeats times each.
  summary mq_hypo_summary at config 3 (1024 chains x 200 events x 50 stations) and config 4 (8192 x 2000 x 100), bins of
          grid h / 10 (the command line's), after 64 iterations at deci 1; median of --calls calls, host clock around a
          call that ends in a device synchronise.  Bytes: the per-chain accumulators (read twice) and the histograms.
  state   accumulator memory, and state size, mq_state_save and mq_state_load with the accumulators on, config 3.

The GPU's name and power limit are read in the same run.

    python tools/hypo_bench.py [--chains 1024,8192] [--rounds 4] [--repeats 2] [--calls 5] [--out result.json]
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

from tools.diag_bench import CONFIGS, gpu_info  # noqa: E402


def step_child(n: int, on: bool, rounds: int, chunk: int = 100) -> dict:
    """One process: ms per round of `chunk` iterations + drain, accumulators on or off."""
    import numpy as np
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    cfg, pk, _ = synth.workload(200, 50, 33, 0, j_max_start=0, j_max_main=2**30, deci=25)
    smp = mq.Sampler(cfg, pk, n, 0, 1000)
    smp.set_ring(8)
    if on:
        smp.hypo_begin(np.float32(cfg.grid.h) / np.float32(10), 0)
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
    if on:
        out["hypo_models"] = int(smp.hypo_summary()["n_models"])
    smp.close()
    return out


def step_bench(chains: list[int], rounds: int, repeats: int) -> list[dict]:
    res = []
    for n in chains:
        runs = {False: [], True: []}
        for _ in range(repeats):
            for on in (False, True):
                r = subprocess.run([sys.executable, __file__, "--child", f"{n},{int(on)},{rounds}"], capture_output=True,
                                   text=True, timeout=1800)
                if r.returncode != 0:
                    raise RuntimeError(r.stderr[-2000:])
                runs[on].append(json.loads(r.stdout.strip().split("\n")[-1]))
        off = [x["ms_per_round"] for x in runs[False]]
        on_ = [x["ms_per_round"] for x in runs[True]]
        res.append(dict(chains=n, iterations_per_round=100, deci=25, rounds=rounds, ms_per_round_off=off, ms_per_round_on=on_,
                        overhead=statistics.median(on_) / statistics.median(off) - 1.0,
                        lost=sum(x["lost"] for x in runs[False] + runs[True]), hypo_models=runs[True][-1]["hypo_models"]))
    return res


def summary_bench(config: int, calls: int, state: bool) -> dict:
    import numpy as np
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    from mcmc_eq_b200._lib import check, lib, dp, lp
    n, ne, ns = CONFIGS[config]
    cfg, pk, _ = synth.workload(ne, ns, 33, 0, j_max_start=0, j_max_main=2**30, deci=1)
    smp = mq.Sampler(cfg, pk, n, 0, 1)
    dims = smp.hypo_begin(np.float32(cfg.grid.h) / np.float32(10), 0)
    smp.init_chains()
    smp.step(64)
    smp.drain()
    nbt = int(sum(dims.n_bins))
    acc_bytes = int(n * ne * 18 * 8 + 8 * n)
    hist_bytes = int(ne * (nbt + 3) * 4)
    out_arrays = [np.zeros(ne * k) for k in (4, 16, 15, 3, 3, 9)]
    N = C.c_int64(0)
    args = [smp.h, 0] + [a.ctypes.data_as(dp) for a in out_arrays] + [C.byref(N)]
    check(lib().mq_hypo_summary(*args))                   # warm-up (and the work space)
    times = []
    for _ in range(calls):
        t0 = time.perf_counter()
        check(lib().mq_hypo_summary(*args))
        times.append(time.perf_counter() - t0)
    t = statistics.median(times)
    read = 2 * n * ne * 18 * 8 - n * ne * 10 * 8 + ne * nbt * 4     # round 1 reads ref, sum, cross; round 2 ref and sum
    res = dict(config=config, chains=n, events=ne, stations=ns, bin_km=float(dims.bin_km), n_bins=list(dims.n_bins),
               accumulator_bytes=acc_bytes, histogram_bytes=hist_bytes, n_models=int(N.value), summary_ms=round(1e3 * t, 3),
               summary_ms_all=[round(1e3 * x, 3) for x in times], bytes_read=read, gbps=round(read / t / 1e9, 1))
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
        res.update(state_bytes=int(got.value), state_save_ms=round(1e3 * statistics.median(save), 2),
                   state_load_ms=round(1e3 * statistics.median(load), 2))
    smp.close()
    return res


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
        n, on, rounds = (int(x) for x in a.child.split(","))
        print(json.dumps(step_child(n, bool(on), rounds)))
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
