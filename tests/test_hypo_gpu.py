"""Hypocentre uncertainty on the device (mq_hypo_*, csrc/hypo.cu).  The accumulators equal hypo.accumulate and
hypo.histogram over the drained records BIT FOR BIT, the device summary equals hypo.summarise on those accumulators to
1e-12, a coordinate fixed by the pick file has variance 0, lock-step and desynchronised stepping give the same
accumulators, they survive a save / load bit for bit, the command line's -L file agrees with the library and is
byte-identical after a kill and resume, and two ranks give the numbers of one handle."""
import json
import os
import signal
import subprocess
import sys

import numpy as np
import pytest

from tests import inputs, util

pytestmark = pytest.mark.gpu

MQ_ERR_ARG, MQ_ERR_STATE = -1, -7


def _host(mqh, cfg, recs, n, burn, bin_km):
    """hypo.py's accumulators over the used drained records: per-chain dicts and the histograms of all of them."""
    lo, hi = mqh.box(cfg)
    per, allv = [], []
    for c in range(n):
        mine = [mqh.record_values(r) for r in recs if r["chain"] == c and r["number"] > burn]
        per.append(mqh.accumulate(np.stack(mine)))
        allv += mine
    hist, outside = mqh.histogram(np.stack(allv), lo, hi, bin_km)
    return per, hist, outside


def _close(a, b, scale, rtol=1e-12):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    f = ~np.isnan(b)
    s = np.maximum(np.abs(b[f]), np.broadcast_to(scale, b.shape)[f])
    assert (np.abs(a[f] - b[f]) <= rtol * s + 1e-300).all(), float(np.max(np.abs(a[f] - b[f]) / np.maximum(s, 1e-300)))


def _compare_summary(dev, want):
    assert dev["n_models"] == want["n_models"]
    sd = np.sqrt(np.abs(np.diagonal(want["cov"], axis1=1, axis2=2)))            # [ne, 4]
    _close(dev["mean"], want["mean"], sd)
    _close(dev["cov"], want["cov"], np.sqrt(sd[:, :, None] * sd[:, None, :]))
    _close(dev["quant"], want["quant"], 0.0)
    _close(dev["mode"], want["mode"], 0.0)
    _close(dev["axes"], want["axes"], want["axes"][:, :1])
    # axis vectors where the axes are well separated (elsewhere any rotation inside the degenerate plane is right)
    sep = np.min(np.abs(np.diff(want["axes"] ** 2, axis=1)), axis=1) > 1e-6 * want["axes"][:, 0] ** 2
    assert np.allclose(dev["axis_dir"][sep], want["axis_dir"][sep], rtol=0, atol=1e-9)


def _summarise(mqh, cfg, dims, acc):
    lo, _hi = mqh.box(cfg)
    return mqh.summarise(lo=lo, bin_km=dims.bin_km, n_bins=list(dims.n_bins), **acc)


@pytest.mark.parametrize("tria", [0, 1])
def test_accumulators_equal_the_host_rule_on_the_drained_records(tria, tmp_path):
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import hypo as mqh
    cfgp, pkp = inputs.materialise("example2", str(tmp_path), j_max_start=20, j_max_main=100000, deci=2, true_random=5, tria=tria)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    n, burn, bin_km = 6, 20, np.float32(cfg.grid.h) / np.float32(10)
    smp = mq.Sampler(cfg, pk, n, 0, 5)
    smp.set_ring(16)
    dims = smp.hypo_begin(bin_km, burn)
    lo, hi = mqh.box(cfg)
    assert dims.n_events == pk.n_events and list(dims.n_bins) == list(mqh.n_bins(lo, hi, bin_km))
    assert np.array_equal(np.float32(dims.lo[:]), lo)
    smp.init_chains()
    recs = []
    for _ in range(40):
        smp.step(10)
        r, lost = smp.drain()
        assert lost == 0
        recs += r
    dev = smp.hypo_chains()
    summ = smp.hypo_summary()
    again = smp.hypo_summary()
    smp.close()
    per, hist, outside = _host(mqh, cfg, recs, n, burn, bin_km)
    assert min(p["n_models"] for p in per) >= 100
    for c in range(n):
        for key in ("ref", "sum", "cross", "n_models"):
            assert np.array_equal(dev[key][c], per[c][key]), (c, key)
    assert np.array_equal(dev["hist"], hist) and np.array_equal(dev["outside"], outside)
    for key in ("mean", "cov", "quant", "mode", "axes", "axis_dir"):   # the same accumulators give the same bits
        assert np.array_equal(summ[key], again[key], equal_nan=True), key
    want = _summarise(mqh, cfg, dims, dict(hist=dev["hist"], **mqh.stack(per)))
    _compare_summary(summ, want)
    assert np.isfinite(summ["cov"]).all() and (summ["axes"][:, 0] >= summ["axes"][:, 2]).all()


def test_a_coordinate_fixed_by_the_pick_file_has_no_variance(tmp_path):
    import mcmc_eq_b200 as mq
    cfgp, pkp = inputs.materialise("example2", str(tmp_path), j_max_start=10, j_max_main=100000, deci=2)
    cfg, pk0 = mq.read_config(cfgp), mq.Picks.read(pkp)
    fix = pk0.fix.copy()
    fix[0, 2] = 5.0                                                 # event 0: depth fixed by the pick file
    pk = mq.Picks(pk0.ev_off, pk0.n_p, pk0.st_id, pk0.x, pk0.y, pk0.z, pk0.t, pk0.cls, pk0.reftime, fix, pk0.n_stations)
    smp = mq.Sampler(cfg, pk, 16, 0, 9)
    dims = smp.hypo_begin(np.float32(cfg.grid.h) / np.float32(10), 0)
    smp.init_chains()
    for _ in range(20):
        smp.step(10)
        smp.drain()
    s = smp.hypo_summary()
    smp.close()
    c = s["cov"][0]
    assert (c[2, :] == 0.0).all() and (c[:, 2] == 0.0).all() and c[0, 0] > 0.0 and c[3, 3] > 0.0
    assert s["mean"][0, 2] == 5.0
    assert (np.abs(s["quant"][0, 2] - 5.0) <= dims.bin_km).all() and abs(s["mode"][0, 2] - 5.0) <= dims.bin_km
    assert np.isfinite(s["cov"]).all() and (s["axes"][0] >= 0).all()


def _bench_sampler(mq, n, seed=1000, deci=2):
    from mcmc_eq_b200 import synth
    cfg, pk, _truth = synth.workload(200, 50, 33, 0, j_max_start=0, j_max_main=2**30, deci=deci)
    return mq.Sampler(cfg, pk, n, 0, seed), cfg, pk


def test_lockstep_and_desynchronised_stepping_give_the_same_accumulators():
    import mcmc_eq_b200 as mq
    res = []
    for call, calls in ((3, 160), (480, 1)):
        smp, cfg, _pk = _bench_sampler(mq, 256, seed=77)
        smp.hypo_begin(np.float32(cfg.grid.h) / np.float32(10), 10)
        smp.init_chains()
        for _ in range(calls):
            smp.step(call)                                         # the ring overflows: dropped records count all the same
        res.append((smp.hypo_chains(), smp.stats()[0]))
        smp.close()
    (a, ca), (b, cb) = res
    assert np.array_equal(ca, cb)
    assert (a["n_models"] > 16).all()
    for key in a:
        assert np.array_equal(a[key], b[key]), key


def test_bench_scale_summary_through_the_pipelined_kernel():
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import hypo as mqh
    n = 1024
    smp, cfg, pk = _bench_sampler(mq, n)
    smp.set_ring(64)
    dims = smp.hypo_begin(np.float32(cfg.grid.h) / np.float32(10), 0)
    smp.init_chains()
    smp.profile(True)
    for _ in range(10):
        smp.step(48)                                                # P_mix: the configuration's balanced strings
        _r, lost = smp.drain()
        assert lost == 0
    smp.profile(False)
    assert "eik_pipe_kernel" in smp.profile_kernels(), smp.profile_kernels()
    dev = smp.hypo_chains()
    summ = smp.hypo_summary()
    smp.close()
    assert summ["mean"].shape == (200, 4) and summ["n_models"] == int(dev["n_models"].sum()) > n
    _compare_summary(summ, _summarise(mqh, cfg, dims, dev))


# ---- checkpoint and resume ---------------------------------------------------------------------------------------------
def _sections(blob):
    import ctypes as C
    from mcmc_eq_b200._lib import MqStateHeader, MqStateSection
    head = MqStateHeader.from_buffer_copy(blob[:C.sizeof(MqStateHeader)])
    secs = [MqStateSection.from_buffer_copy(blob, C.sizeof(MqStateHeader) + k * C.sizeof(MqStateSection)) for k in range(head.n_sections)]
    return head, secs


def test_a_loaded_state_continues_the_accumulators_bit_for_bit(tmp_path):
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200._lib import STATE_HYPO
    from tests.test_state_gpu import _reseal
    cfgp, pkp = inputs.materialise("example2", str(tmp_path), j_max_start=10, j_max_main=100000, deci=3)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    n, bin_km = 12, np.float32(cfg.grid.h) / np.float32(10)
    a = mq.Sampler(cfg, pk, n, 0, 4)
    a.init_chains()
    a.step(30)
    a.drain()
    plain = a.save_state()                                          # feature off: flags and sections as before
    head, secs = _sections(plain)
    assert not head.flags & STATE_HYPO and {s.id for s in secs} <= {1, 2, 3, 4, 5} and head.format == 1
    a.diag_begin(5, 8)                                              # next to the diagnostics section
    a.hypo_begin(bin_km, 15)
    for _ in range(10):
        a.step(9)
        a.drain()
    blob = a.save_state()
    head, secs = _sections(blob)
    assert head.flags & STATE_HYPO and [s.id for s in secs][-2:] == [5, 6]
    saved = a.hypo_chains()
    for _ in range(6):
        a.step(9)
        a.drain()
    b = mq.Sampler(cfg, pk, n, 0, 99)
    b.load_state(blob)
    for key, v in b.hypo_chains().items():
        assert np.array_equal(v, saved[key]), key
    for _ in range(6):
        b.step(9)
        b.drain()
    da, db = a.hypo_chains(), b.hypo_chains()
    for key in da:
        assert np.array_equal(da[key], db[key]), key
    sa, sb = a.hypo_summary(), b.hypo_summary()
    for key in sa:
        assert np.array_equal(sa[key], sb[key], equal_nan=True), key
    # a hypocentre section whose bin counts or bin width do not fit is refused and leaves the handle as it was
    sec = secs[-1]
    before = b.hypo_chains()
    for at, value in ((sec.offset + 12, (int(before["hist"].shape[1]) + 7).to_bytes(4, "little")),     # n_bins[0]
                      (sec.offset + 8, np.float32(bin_km * 2).tobytes()),                              # bin_km
                      (sec.offset + 8, np.float32(-1.0).tobytes())):
        bad = bytearray(blob)
        bad[at:at + 4] = value
        with pytest.raises(mq.MqError) as e:
            b.load_state(_reseal(bad))
        assert e.value.code == MQ_ERR_ARG
        for key, v in b.hypo_chains().items():
            assert np.array_equal(v, before[key]), key
    # a state without the section loads and frees the handle's accumulators
    b.load_state(plain)
    with pytest.raises(mq.MqError) as e:
        b.hypo_summary()
    assert e.value.code == MQ_ERR_STATE
    a.close(); b.close()


def test_arguments_and_order(tmp_path):
    import mcmc_eq_b200 as mq
    cfgp, pkp = inputs.materialise("example2", str(tmp_path), j_max_start=10, j_max_main=100000, deci=3)
    cfg = mq.read_config(cfgp)
    s = mq.Sampler(cfg, mq.Picks.read(pkp), 4, 0, 1)
    s._hbins = (1, 1, 1)
    for call in (s.hypo_chains, s.hypo_summary):
        with pytest.raises(mq.MqError) as e:
            call()
        assert e.value.code == MQ_ERR_STATE
    span = max(cfg.grid.nx, cfg.grid.ny, cfg.grid.nz) * cfg.grid.h
    for w, burn in ((0.0, 0), (-1.0, 0), (float("nan"), 0), (0.1, -1), (span / 2**21, 0)):
        with pytest.raises(mq.MqError) as e:
            s.hypo_begin(w, burn)
        assert e.value.code == MQ_ERR_ARG
    s.hypo_begin(cfg.grid.h, 0)                                     # before mq_init_chains
    summ = s.hypo_summary()                                         # no model yet: NaN everywhere
    assert summ["n_models"] == 0 and np.isnan(summ["mean"]).all() and np.isnan(summ["quant"]).all()
    s.init_chains()
    s.step(6)
    assert s.hypo_summary()["n_models"] == int(s.hypo_chains()["n_models"].sum())
    s.close()


# ---- the command line --------------------------------------------------------------------------------------------------
EXE = os.path.join(util.ROOT, "mcmc_eq_b200", "host", "mcmc_eq")


def _files(d, n):
    return [open(os.path.join(d, f"rjx-{k:03d}.out"), "rb").read() for k in range(1, n + 1)]


def _parse(path):
    lines = open(path).read().split("\n")
    head = lines[0].split()
    rows = np.array([[float(x) for x in ln.split()] for ln in lines[1:] if ln])
    return head, rows


def test_the_command_line_file_agrees_with_the_library_and_survives_a_kill(tmp_path):
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import hypo as mqh
    kw = dict(j_max_start=60, j_max_main=6000, deci=20, true_random=77)
    runs = {}
    for name in ("A", "B", "P"):
        runs[name] = str(tmp_path / name)
        inputs.materialise("example2", runs[name], **kw)
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "16", "-q", "-k", "ck", "-K", "0", "-L", "loc.txt"],
                       cwd=runs["A"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    want, want_loc = _files(runs["A"], 16), open(os.path.join(runs["A"], "loc.txt"), "rb").read()
    head, rows = _parse(os.path.join(runs["A"], "loc.txt"))
    cfg, pk = mq.read_config(os.path.join(runs["A"], "config_eqx.dat")), mq.Picks.read(os.path.join(runs["A"], "picks"))
    assert head[:3] == ["#", "events", str(pk.n_events)] and head[5:7] == ["burn_in", "60"]
    assert float(head[8]) == np.float32(cfg.grid.h) / np.float32(10)
    assert rows.shape == (pk.n_events, 2 + 4 + 4 + 1 + 15 + 3 + 9 + 3) and np.array_equal(rows[:, 0], np.arange(pk.n_events))
    # the last checkpoint is one chunk (2 deci iterations) before the end: load it, step that chunk, summarise
    ck = open(os.path.join(runs["A"], "ck"), "rb").read()
    smp = mq.Sampler(cfg, pk, 16, 0, 1)
    smp.load_state(ck[48 + 8 * 16:])                                # after the CLI's header and 16 chain file lengths
    smp.step(2 * kw["deci"])
    smp.drain()
    s = smp.hypo_summary()
    outside = smp.hypo_chains()["outside"]
    smp.close()
    assert (rows[:, 1] == s["n_models"]).all() and int(head[4]) == s["n_models"]
    sd = np.sqrt(np.diagonal(s["cov"], axis1=1, axis2=2))
    corr = s["cov"][:, 2, 3] / np.sqrt(s["cov"][:, 2, 2] * s["cov"][:, 3, 3])
    axes = [np.array([[s["axes"][e, k], *mqh.azimuth_plunge(s["axis_dir"][e, k])] for k in range(3)]).ravel() for e in range(pk.n_events)]
    expect = np.concatenate([s["mean"], sd, corr[:, None], s["quant"].reshape(-1, 15), s["mode"], np.array(axes), outside], 1)
    assert np.allclose(rows[:, 2:], expect, rtol=1e-8, atol=1e-6, equal_nan=True), np.nanmax(np.abs(rows[:, 2:] - expect))
    assert ((rows[:, 31:38:3] >= 0) & (rows[:, 31:38:3] <= 90)).all()                              # plunges
    assert ((rows[:, 30:37:3] >= 0) & (rows[:, 30:37:3] < 360)).all()                              # azimuths
    # killed after its first checkpoint and resumed: the same -L file and chain files
    d = runs["B"]
    p = subprocess.Popen([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "16", "-k", "ck", "-K", "0", "-L", "loc.txt"], cwd=d,
                         stderr=subprocess.PIPE, stdout=subprocess.DEVNULL, text=True)
    seen_ck, killed = False, False
    for line in p.stderr:
        if line.startswith("Test"):
            if seen_ck:
                p.send_signal(signal.SIGKILL)
                killed = True
                break
            seen_ck = os.path.exists(os.path.join(d, "ck"))
    p.wait(timeout=300)
    p.stderr.close()
    assert killed, "run B ended before it could be killed"
    assert os.path.exists(os.path.join(d, "loc.txt"))              # written at the checkpoint
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-R", "ck", "-q", "-L", "loc.txt"], cwd=d,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    assert open(os.path.join(d, "loc.txt"), "rb").read() == want_loc
    assert _files(d, 16) == want
    # -L with a checkpoint of a run without it fails before any chain file is touched
    pdir = runs["P"]
    p = subprocess.Popen([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "4", "-k", "ck", "-K", "0"], cwd=pdir,
                         stderr=subprocess.PIPE, stdout=subprocess.DEVNULL, text=True)
    for line in p.stderr:
        if line.startswith("Test") and os.path.exists(os.path.join(pdir, "ck")):
            p.send_signal(signal.SIGKILL)
            break
    p.wait(timeout=300)
    p.stderr.close()
    stamp = [os.stat(os.path.join(pdir, f"rjx-{k:03d}.out")).st_mtime_ns for k in range(1, 5)]
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-R", "ck", "-q", "-L", "loc.txt"], cwd=pdir,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "holds no hypocentre accumulators" in r.stderr, r.stderr
    assert [os.stat(os.path.join(pdir, f"rjx-{k:03d}.out")).st_mtime_ns for k in range(1, 5)] == stamp
    assert not os.path.exists(os.path.join(pdir, "loc.txt"))


# ---- two ranks ---------------------------------------------------------------------------------------------------------
def test_two_ranks_give_the_numbers_of_one_handle():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29539", os.path.join(util.ROOT, "tests", "hypo_mp_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=util.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.split("\n") if ln.startswith("HYPORESULT ")][0]
    res = json.loads(line[len("HYPORESULT "):])
    assert res and all(res.values()), res
