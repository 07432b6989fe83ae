"""Convergence diagnostics on the device (mq_diag_*, csrc/diag.cu).  The accumulators equal diag.accumulate over the
quantities of the drained records BIT FOR BIT, the device summary equals diag.summarise on those accumulators to 1e-12,
lock-step and desynchronised stepping give the same accumulators, the accumulators survive a save / load bit for bit,
a command-line run killed and resumed writes the same diagnostics file, and two ranks give the numbers of one handle."""
import json
import os
import signal
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from tests import inputs, util
from tests.test_posterior_gpu import _nearest, _tria_profile

pytestmark = pytest.mark.gpu

MQ_ERR_ARG, MQ_ERR_STATE = -1, -7


def _velocity(cfg):
    """rec -> (vp[nz], vpvs[nz]) as the posterior bins them: nearest nucleus or TRIA = 1 profile, clipped."""
    g = cfg.grid
    lo_v, hi_v, lo_r, hi_r = (np.float32(x) for x in (cfg.vpmin, cfg.vpmax, cfg.vpvsmin, cfg.vpvsmax))

    def f(r):
        if cfg.tria == 1:
            pv, pr = _tria_profile(r["z"], r["vp"], g.nz, g.h, g.z0), _tria_profile(r["z"], r["vpvs"], g.nz, g.h, g.z0)
        else:
            pv, pr = np.zeros(g.nz, np.float32), np.zeros(g.nz, np.float32)
            for i in range(g.nz):
                k = _nearest(r["z"], np.float32(np.float32(i) * np.float32(g.h) + np.float32(g.z0)))
                pv[i], pr[i] = r["vp"][k], r["vpvs"][k]
        return np.minimum(np.maximum(pv, lo_v), hi_v), np.minimum(np.maximum(pr, lo_r), hi_r)
    return f


def _host_accumulators(mq_diag, cfg, recs, n, burn, K, chains=None):
    vel = _velocity(cfg)
    out = []
    for c in (range(n) if chains is None else chains):
        mine = [r for r in recs if r["chain"] == c and r["number"] > burn]
        trace = np.stack([mq_diag.record_quantities(r, cfg, vel) for r in mine]) if mine else np.zeros((0, 0))
        out.append(mq_diag.accumulate(trace, K) if mine else None)
    return out


def _same_chain(dev, c, host):
    for key in ("ref", "sum", "sumsq", "batch_len", "full_batches", "n_models"):
        assert np.array_equal(dev[key][c], host[key]), (c, key)


def _close(a, b, sd, rtol=1e-12):
    """equal to rtol relative to max(|b|, sd): NaN and inf in the same places"""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.isinf(a), np.isinf(b))
    assert np.array_equal(a[np.isinf(a)], b[np.isinf(b)])
    f = np.isfinite(b)
    scale = np.maximum(np.abs(b[f]), np.nan_to_num(np.asarray(sd, np.float64)[f]))
    assert (np.abs(a[f] - b[f]) <= rtol * scale + 1e-300).all(), float(np.max(np.abs(a[f] - b[f]) / np.maximum(scale, 1e-300)))


def _compare_summary(dev, host):
    assert dev["chains_used"] == host["chains_used"] and dev["n_models"] == host["n_models"]
    for key in ("mean", "sd", "rhat", "ess"):
        _close(dev[key], host[key], host["sd"])


@pytest.mark.parametrize("tria", [0, 1])
def test_accumulators_equal_the_host_rule_on_the_drained_records(tria):
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import diag as mqd
    d = tempfile.mkdtemp(prefix="mqd_")
    cfgp, pkp = inputs.materialise("example2", d, j_max_start=20, j_max_main=100000, deci=2, true_random=5, tria=tria)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    n, burn, K = 6, 20, 8
    smp = mq.Sampler(cfg, pk, n, 0, 5)
    smp.set_ring(16)
    dims = smp.diag_begin(burn, K)
    assert (dims.n_quantities, dims.n_batches) == (10 + 2 * cfg.grid.nz + 4 * pk.n_events + 2 * pk.n_stations, K)
    smp.init_chains()
    recs = []
    for _ in range(80):
        smp.step(10)
        r, lost = smp.drain()
        assert lost == 0
        recs += r
    dev = smp.diag_chains()
    summ = smp.diag_summary()
    smp.close()
    host = _host_accumulators(mqd, cfg, recs, n, burn, K)
    assert min(h["n_models"] for h in host) >= 100                 # several doublings of the batch length
    assert (dev["batch_len"] >= 8).all()
    for c in range(n):
        _same_chain(dev, c, host[c])
    want = mqd.summarise(**mqd.stack(host))
    _compare_summary(summ, want)
    assert summ["names"][0] == "rms" and len(summ["names"]) == dims.n_quantities


def _bench_sampler(mq, n, seed=1000, deci=2):
    from mcmc_eq_b200 import synth
    cfg, pk, _truth = synth.workload(200, 50, 33, 0, j_max_start=0, j_max_main=2**30, deci=deci)
    return mq.Sampler(cfg, pk, n, 0, seed), cfg, pk


def test_bench_scale_summary_and_sampled_chains():
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import diag as mqd
    n, K = 1024, 16
    smp, cfg, pk = _bench_sampler(mq, n)
    smp.set_ring(64)
    smp.diag_begin(0, K)
    smp.init_chains()
    sample = [0, 1, 137, 500, 511, 512, 900, 1023]
    recs = []
    smp.profile(True)
    for _ in range(10):
        smp.step(48)                                                # P_mix: the configuration's balanced strings
        r, lost = smp.drain()
        assert lost == 0
        recs += [x for x in r if x["chain"] in sample]
    _ms, _launches, _per = smp.profile(False)
    assert "eik_pipe_kernel" in smp.profile_kernels(), smp.profile_kernels()   # full rebuild passes take it
    dev = smp.diag_chains()
    summ = smp.diag_summary()
    again = smp.diag_summary()
    smp.close()
    assert len(summ["mean"]) == 1034 and summ["chains_used"] > 900
    for key in ("mean", "sd", "rhat", "ess"):                      # the same accumulators give the same bits
        assert np.array_equal(summ[key], again[key], equal_nan=True)
    _compare_summary(summ, mqd.summarise(**dev))
    host = _host_accumulators(mqd, cfg, recs, n, 0, K, chains=sample)
    for c, h in zip(sample, host):
        _same_chain(dev, c, h)


def test_lockstep_and_desynchronised_stepping_give_the_same_accumulators():
    import mcmc_eq_b200 as mq
    res = []
    for call, calls in ((3, 160), (480, 1)):
        smp, _cfg, _pk = _bench_sampler(mq, 256, seed=77)
        smp.diag_begin(10, 16)
        smp.init_chains()
        for _ in range(calls):
            smp.step(call)                                         # the ring overflows: dropped records count all the same
        res.append((smp.diag_chains(), smp.stats()[0]))
        smp.close()
    (a, ca), (b, cb) = res
    assert np.array_equal(ca, cb)
    assert (a["n_models"] > 16).all()
    for key in a:
        assert np.array_equal(a[key], b[key]), key


def test_hypocentres_that_never_move_have_infinite_or_undefined_rhat(tmp_path):
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import diag as mqd
    cfgp, pkp = inputs.materialise("example2", str(tmp_path), j_max_start=10, j_max_main=100000, deci=2)
    cfg, pk0 = mq.read_config(cfgp), mq.Picks.read(pkp)
    fix = pk0.fix.copy()
    free = fix == -9999.0
    fix[0, 2] = 5.0                                                 # event 0: depth fixed by the pick file
    free[0, 2] = False
    pk = mq.Picks(pk0.ev_off, pk0.n_p, pk0.st_id, pk0.x, pk0.y, pk0.z, pk0.t, pk0.cls, pk0.reftime, fix, pk0.n_stations)
    smp = mq.Sampler(cfg, pk, 16, 0, 9)
    smp.diag_begin(0, 8)
    smp.init_chains()
    for _ in range(20):
        smp.step(10, "PVN")
        smp.drain()
    s = smp.diag_summary()
    smp.close()
    assert s["chains_used"] == 16
    nz, ne = cfg.grid.nz, pk.n_events
    at = 10 + 2 * nz
    rhat = s["rhat"][at:at + 4 * ne].reshape(ne, 4)
    assert (rhat[:, :3][free] == np.inf).all()
    assert np.isnan(rhat[:, :3][~free]).all() and np.isnan(s["ess"][at:at + 4 * ne].reshape(ne, 4)[:, :3][~free]).all()
    assert np.isfinite(rhat[:, 3]).all()                            # origin times move with the velocity model
    assert mqd.quantity_names(nz, ne, pk.n_stations)[at + 2] == "z[0]"


# ---- checkpoint and resume ---------------------------------------------------------------------------------------------
def _sections(blob):
    import ctypes as C
    from mcmc_eq_b200._lib import MqStateHeader, MqStateSection
    head = MqStateHeader.from_buffer_copy(blob[:C.sizeof(MqStateHeader)])
    secs = [MqStateSection.from_buffer_copy(blob, C.sizeof(MqStateHeader) + k * C.sizeof(MqStateSection)) for k in range(head.n_sections)]
    return head, secs


def test_a_loaded_state_continues_the_accumulators_bit_for_bit(tmp_path):
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200._lib import STATE_DIAG
    from tests.test_state_gpu import _reseal
    cfgp, pkp = inputs.materialise("example2", str(tmp_path), j_max_start=10, j_max_main=100000, deci=3)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    n = 12
    a = mq.Sampler(cfg, pk, n, 0, 4)
    a.init_chains()
    a.step(30)
    a.drain()
    plain = a.save_state()                                          # diagnostics off: flags and sections as before
    head, secs = _sections(plain)
    assert not head.flags & STATE_DIAG and {s.id for s in secs} <= {1, 2, 3, 4} and head.format == 1
    a.diag_begin(15, 8)
    for _ in range(10):
        a.step(9)
        a.drain()
    blob = a.save_state()
    head, secs = _sections(blob)
    assert head.flags & STATE_DIAG and secs[-1].id == 5 and len(blob) - len(plain) == secs[-1].bytes + 24   # + its table entry
    saved = a.diag_chains()
    for _ in range(6):
        a.step(9)
        a.drain()
    b = mq.Sampler(cfg, pk, n, 0, 99)
    b.load_state(blob)
    for key, v in b.diag_chains().items():
        assert np.array_equal(v, saved[key]), key
    for _ in range(6):
        b.step(9)
        b.drain()
    da, db = a.diag_chains(), b.diag_chains()
    for key in da:
        assert np.array_equal(da[key], db[key]), key
    sa, sb = a.diag_summary(), b.diag_summary()
    for key in ("mean", "sd", "rhat", "ess", "n_models", "chains_used"):
        assert np.array_equal(sa[key], sb[key], equal_nan=True), key
    assert sa["chains_used"] == n
    # a diagnostics section of another quantity count is refused and leaves the handle as it was
    bad = bytearray(blob)
    sec = secs[-1]
    bad[sec.offset + 12:sec.offset + 16] = (int.from_bytes(bad[sec.offset + 12:sec.offset + 16], "little") + 1).to_bytes(4, "little")
    before = b.diag_chains()
    with pytest.raises(mq.MqError) as e:
        b.load_state(_reseal(bad))
    assert e.value.code == MQ_ERR_ARG
    for key, v in b.diag_chains().items():
        assert np.array_equal(v, before[key]), key
    # a state without diagnostics frees the handle's
    b.load_state(plain)
    with pytest.raises(mq.MqError) as e:
        b.diag_summary()
    assert e.value.code == MQ_ERR_STATE
    a.close(); b.close()


def test_arguments_and_order():
    import mcmc_eq_b200 as mq
    cfg_d = tempfile.mkdtemp(prefix="mqd_")
    cfgp, pkp = inputs.materialise("example2", cfg_d, j_max_start=10, j_max_main=100000, deci=3)
    s = mq.Sampler(mq.read_config(cfgp), mq.Picks.read(pkp), 4, 0, 1)
    s._ddims = (1, 8)
    for call in (s.diag_chains, s.diag_summary):
        with pytest.raises(mq.MqError) as e:
            call()
        assert e.value.code == MQ_ERR_STATE
    for burn, k in ((-1, 16), (0, 7), (0, 9), (0, 66), (0, 6)):
        with pytest.raises(mq.MqError) as e:
            s.diag_begin(burn, k)
        assert e.value.code == MQ_ERR_ARG
    s.diag_begin(0, 64)                                            # before mq_init_chains
    s.init_chains()
    s.step(6)
    assert s.diag_summary()["chains_used"] == 0                    # no chain has four full batches yet: all NaN
    s.close()


# ---- the command line --------------------------------------------------------------------------------------------------
EXE = os.path.join(util.ROOT, "mcmc_eq_b200", "host", "mcmc_eq")


def _files(d, n):
    return [open(os.path.join(d, f"rjx-{k:03d}.out"), "rb").read() for k in range(1, n + 1)]


def test_a_killed_run_resumed_from_its_checkpoint_writes_the_same_diagnostics(tmp_path):
    kw = dict(j_max_start=60, j_max_main=6000, deci=20, true_random=77)
    runs = {}
    for name in ("A", "B", "P"):
        runs[name] = str(tmp_path / name)
        inputs.materialise("example2", runs[name], **kw)
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "16", "-q", "-D", "diag.txt"], cwd=runs["A"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    assert "max R-hat" in r.stderr
    want, want_diag = _files(runs["A"], 16), open(os.path.join(runs["A"], "diag.txt"), "rb").read()
    lines = want_diag.decode().split("\n")
    assert lines[0].startswith("# chains_used 16 burn_in 60 batches 16 iterations ")
    import mcmc_eq_b200 as mq
    cfg, pk = mq.read_config(os.path.join(runs["A"], "config_eqx.dat")), mq.Picks.read(os.path.join(runs["A"], "picks"))
    assert len([x for x in lines[1:] if x]) == 10 + 2 * cfg.grid.nz + 4 * pk.n_events + 2 * pk.n_stations
    names = [x.split()[0] for x in lines[1:] if x]
    assert names[:3] == ["rms", "dim", "noise"] and set(names) == {"rms", "dim", "noise", "vp", "vpvs", "x", "y", "z", "t", "pres", "sres"}
    d = runs["B"]
    p = subprocess.Popen([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "16", "-k", "ck", "-K", "0", "-D", "diag.txt"], cwd=d,
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
    assert os.path.exists(os.path.join(d, "diag.txt"))             # written at the checkpoint
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-R", "ck", "-q", "-D", "diag.txt"], cwd=d,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    assert open(os.path.join(d, "diag.txt"), "rb").read() == want_diag
    assert _files(d, 16) == want
    # -D with a checkpoint of a run without diagnostics fails before any chain file is touched
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
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-R", "ck", "-q", "-D", "diag.txt"], cwd=pdir,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "holds no diagnostics" in r.stderr, r.stderr
    assert [os.stat(os.path.join(pdir, f"rjx-{k:03d}.out")).st_mtime_ns for k in range(1, 5)] == stamp
    assert not os.path.exists(os.path.join(pdir, "diag.txt"))


# ---- two ranks ---------------------------------------------------------------------------------------------------------
def test_two_ranks_give_the_numbers_of_one_handle():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29537", os.path.join(util.ROOT, "tests", "diag_mp_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=util.ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.split("\n") if ln.startswith("DIAGRESULT ")][0]
    res = json.loads(line[len("DIAGRESULT "):])
    assert res and all(res.values()), res
