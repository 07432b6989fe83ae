"""Cost of a checkpoint: mq_state_save (device -> host buffer), writing the state to a file (write + fsync), mq_state_load
(host -> device, table rebuild of every chain and hash check) and the size of the state, for the bench workloads:

    config 3: 1024 chains x synth.workload(200 events, 50 stations)
    config 4: 8192 chains x synth.workload(2000 events, 100 stations)

each after a few mixed iterations (config strings).  Every time is the median of --repeats calls measured with a host
clock around a call that ends in a device synchronise.  The GPU's name and power limit are read in the same run.

    python tools/state_bench.py [--configs 3,4] [--repeats 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
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


def run(config: int, repeats: int) -> dict:
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    from mcmc_eq_b200._lib import check, lib
    n, ne, ns = CONFIGS[config]
    cfg, pk, _truth = synth.workload(ne, ns, 33, 0)
    smp = mq.Sampler(cfg, pk, n, 0, 1)
    smp.init_chains()
    smp.step(12)
    smp.drain()
    size = C.c_uint64(0)
    check(lib().mq_state_size(smp.h, C.byref(size)))
    buf = C.create_string_buffer(size.value)
    got = C.c_uint64(0)
    save, write, load = [], [], []
    check(lib().mq_state_save(smp.h, buf, size.value, C.byref(got)))       # warm-up of every call
    check(lib().mq_state_load(smp.h, buf, size.value))
    with tempfile.TemporaryDirectory(prefix="mqstate_bench_") as d:
        path = os.path.join(d, "state")
        for _ in range(repeats):
            t0 = time.perf_counter()
            check(lib().mq_state_save(smp.h, buf, size.value, C.byref(got)))
            save.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            with open(path, "wb") as f:
                f.write(memoryview(buf)[:got.value])
                f.flush()
                os.fsync(f.fileno())
            write.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            check(lib().mq_state_load(smp.h, buf, got.value))
            load.append(time.perf_counter() - t0)
    smp.step(2)     # the loaded handle steps on
    smp.sync()
    smp.close()
    ms = lambda v: round(1e3 * statistics.median(v), 2)
    return dict(config=config, chains=n, events=ne, stations=ns, state_bytes=got.value,
                bytes_per_chain=round(got.value / n), save_ms=ms(save), write_ms=ms(write), load_ms=ms(load),
                save_ms_all=[round(1e3 * x, 2) for x in save], load_ms_all=[round(1e3 * x, 2) for x in load])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="3,4")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out")
    a = ap.parse_args()
    res = dict(gpu_info(), results=[run(int(c), a.repeats) for c in a.configs.split(",")])
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
