"""Checkpoint and resume (mq_state_save / mq_state_load, csrc/state.cu): a sampler that loads a saved state continues every
chain with the same proposals, decisions and records as the sampler that saved it, BIT FOR BIT -- counters, likelihoods,
models, decimated records, best models, posterior accumulators and temperatures.  A state that does not fit the handle
is refused and leaves the handle as it was; a rebuilt travel-time table whose hash differs from the saved one is named.
The command line's -k / -R resume a killed run to chain files byte-identical to an uninterrupted run's."""
import ctypes as C
import json
import os
import signal
import subprocess
import sys
import time

import numpy as np
import pytest

from tests import inputs, util

pytestmark = pytest.mark.gpu

MQ_ERR_ARG, MQ_ERR_STATE, MQ_ERR_BUSY = -1, -7, -9

SCRIPT = r"""
import json, sys, tempfile, numpy as np
sys.path.insert(0, %r)
import mcmc_eq_b200 as mq
from tests import inputs
case = json.loads(sys.argv[2])
d = tempfile.mkdtemp(prefix="mqstate_")
cfgp, pkp = inputs.materialise(case["input"], d, j_max_start=30, j_max_main=100000, deci=7, tria=case["tria"])
cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
n, temper = case["n"], case["temper"]
out = {}

def recs_to(prefix, recs):
    for f in ("chain", "kind", "number", "dim", "rms"):
        out[prefix + "rec_" + f] = np.array([r[f] for r in recs])
    out[prefix + "rec_code"] = np.array([ord(r["code"]) for r in recs])
    for f in ("noise", "z", "vp", "vpvs", "eq", "origin", "pres", "sres"):
        out[prefix + "rec_" + f] = np.concatenate([np.ravel(r[f]) for r in recs]) if recs else np.zeros(0)

def state_to(prefix, s):
    c, ll, rms = s.stats()
    out[prefix + "counts"] = c; out[prefix + "ll"] = ll; out[prefix + "rms"] = rms
    m = s.get_models()
    for f in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise", "origin"):
        out[prefix + "m_" + f] = getattr(m, f)
    best = s.snapshot_all(1)
    for f in ("number", "dim", "rms"):
        out[prefix + "best_" + f] = np.array([b[f] for b in best])
    for f in ("noise", "z", "vp", "vpvs", "eq", "origin", "pres", "sres"):
        out[prefix + "best_" + f] = np.concatenate([np.ravel(b[f]) for b in best])
    out[prefix + "beta"] = s.get_beta()
    if case["posterior"]:
        for k, v in s.posterior_get().items():
            out[prefix + "post_" + k] = np.asarray(v)

def drained(s, recs):
    r, lost = s.drain()
    assert lost == 0
    recs += r

def continuation(s, recs):
    for i, chunk in enumerate((6, 5)):
        s.step(chunk); drained(s, recs)
        if temper: s.temper_swap(10 + i)
    s.step(6, "QVRPBDMN"); drained(s, recs)
    s.step(5, "P"); drained(s, recs)
    if temper: s.temper_swap(12)

a = mq.Sampler(cfg, pk, n, 0, 21)
if case["offset"]: a.set_chain_offset(case["offset"])
a.init_chains()
if case["posterior"]: a.posterior_begin(0.1, 0.02, 3)
if temper: a.set_beta(np.linspace(1.0, 0.3, n).astype(np.float32))
pre = []
for i, chunk in enumerate((7, 5, 7, 7)):
    a.step(chunk); drained(a, pre)
    if temper: a.temper_swap(i)
blob = a.save_state()
state_to("a0_", a)
ra = []
continuation(a, ra)
state_to("a_", a); recs_to("a_", ra)
a.close()

b = mq.Sampler(cfg, pk, n, 0, 5)          # another seed, no chain offset, posterior or betas: the state's replace them
b.load_state(blob)
state_to("b0_", b)
out["resave_equal"] = np.array(b.save_state() == blob)
rb = []
continuation(b, rb)
state_to("b_", b); recs_to("b_", rb)
out["n_pre_records"] = np.array(len(pre)); out["n_records"] = np.array(len(rb))
np.savez(sys.argv[1], **out)
"""

CASES = {
    "example2_97_voronoi": dict(input="example2", n=97, tria=0, posterior=False, temper=False, offset=0, desync="1"),
    "example2_8_tria": dict(input="example2", n=8, tria=1, posterior=False, temper=False, offset=0, desync="1"),
    "example_40_posterior_tempering": dict(input="example", n=40, tria=0, posterior=True, temper=True, offset=0, desync="1"),
    "example2_97_lockstep": dict(input="example2", n=97, tria=0, posterior=False, temper=False, offset=0, desync="0"),
    "example2_8_chain_offset": dict(input="example2", n=8, tria=0, posterior=False, temper=False, offset=1000, desync="1"),
}


def _compare(res, x, y):
    keys = sorted(k[len(x):] for k in res if k.startswith(x))
    assert keys
    for k in keys:
        a, b = res[x + k], res[y + k]
        if k.startswith("post_") and a.dtype == np.float64:
            # the moment sums are double atomics from every chain's block (snapshot_kernel): their order, and so their last
            # bits, differ between any two runs, resumed or not.  The histograms and the model count are exact.
            assert np.allclose(a, b, rtol=1e-12, atol=0), (x, y, k, float(np.abs(a - b).max()))
        else:
            assert np.array_equal(a, b), (x, y, k)


@pytest.mark.parametrize("name", sorted(CASES))
def test_a_loaded_state_continues_bit_for_bit(tmp_path, name):
    case = CASES[name]
    env = dict(os.environ, MCMCEQ_DESYNC=case["desync"])
    path = str(tmp_path / "state.npz")
    r = subprocess.run([sys.executable, "-c", SCRIPT % util.ROOT, path, json.dumps(case)], env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    res = dict(np.load(path))
    _compare(res, "a0_", "b0_")        # right after the load: the saved state
    _compare(res, "a_", "b_")          # after the continuation
    assert bool(res["resave_equal"])   # a loaded state saves to the same bytes
    assert int(res["n_records"]) > 0 and int(res["n_pre_records"]) > 0
    if case["posterior"]:
        assert res["a_post_n_models"] > res["a0_post_n_models"] > 0
    if case["temper"]:
        assert not np.array_equal(res["a_beta"], np.linspace(1.0, 0.3, case["n"]).astype(np.float32))


# ---- bench scale: the rebuild of the load runs the benched kernels -------------------------------------------------------
def _continue_and_compare(a, b, p_steps):
    a.step(p_steps, "P")
    b.step(p_steps, "P")
    for x, y in zip(a.stats(), b.stats()):
        assert np.array_equal(x, y)
    ma, mb = a.get_models(), b.get_models()
    for f in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise", "origin"):
        assert np.array_equal(getattr(ma, f), getattr(mb, f)), f
    for ra, rb in zip(a.snapshot_all(1), b.snapshot_all(1)):
        for f in ("number", "dim", "rms", "noise", "z", "vp", "vpvs", "eq", "origin", "pres", "sres"):
            assert np.array_equal(ra[f], rb[f]), f


def _save_load(mq, cfg, pk, n):
    a = mq.Sampler(cfg, pk, n, 0, 3)
    a.init_chains()
    a.step(6, "QVRPBDMN")
    a.drain()
    blob = a.save_state()
    b = mq.Sampler(cfg, pk, n, 0, 3)
    b.profile(True)
    b.load_state(blob)
    _ms, launches, _per = b.profile(False)
    return a, b, launches, b.profile_kernels()


def test_bench_workload_resumes_bit_for_bit_through_the_pipelined_kernel():
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    cfg, pk, _truth = synth.workload(200, 50, 33, 0, j_max_start=0, j_max_main=2**30, deci=2**30)
    a, b, launches, kernels = _save_load(mq, cfg, pk, 1024)
    assert launches == 1 and list(kernels) == ["eik_pipe_kernel"], kernels
    _continue_and_compare(a, b, 4)
    a.close(); b.close()


def test_deep_plane_resumes_bit_for_bit_through_the_deep_pipelined_kernel(tmp_path):
    import mcmc_eq_b200 as mq
    cfgp, pkp = inputs.materialise("example2", str(tmp_path), h=0.25, nx=193, ny=193, nz=121, j_max_start=30,
                                   j_max_main=100000, deci=2**30)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    a, b, launches, kernels = _save_load(mq, cfg, pk, 1000)
    assert launches == 1 and list(kernels) == ["eik_pipe_kernel"], kernels
    _continue_and_compare(a, b, 3)
    a.close(); b.close()


# ---- refusals, preconditions, the hash check -----------------------------------------------------------------------------
def _sum64(data: bytes, h=0x9E3779B97F4A7C15):
    """The checksum of include/mcmceq_b200.h (mq_state_*)."""
    data = data + b"\0" * (-len(data) % 8)
    m = (1 << 64) - 1
    for w in np.frombuffer(data, "<u8").tolist():
        h = ((h ^ w) * 0x100000001B3) & m
        h ^= h >> 32
    return h


def _reseal(blob: bytearray) -> bytes:
    blob[-8:] = _sum64(bytes(blob[:-8])).to_bytes(8, "little")
    return bytes(blob)


def _example2(tmp_path, n=8, **over):
    import mcmc_eq_b200 as mq
    kw = dict(j_max_start=30, j_max_main=100000, deci=7)
    kw.update(over)
    d = str(tmp_path / ("in_" + "_".join(f"{k}{v}" for k, v in sorted(over.items()))))
    cfgp, pkp = inputs.materialise("example2", d, **kw)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    s = mq.Sampler(cfg, pk, n, 0, 7)
    s.init_chains()
    s.step(9)
    s.drain()
    return s


def _snapshot(s):
    c, ll, rms = s.stats()
    m = s.get_models()
    return [c, ll, rms] + [getattr(m, f) for f in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise", "origin")]


def test_refused_states_leave_the_handle_unchanged(tmp_path):
    import mcmc_eq_b200 as mq
    a = _example2(tmp_path)
    blob = a.save_state()
    foreign = {"n_chains": _example2(tmp_path, n=9).save_state(), "deci": _example2(tmp_path, deci=8).save_state()}
    pk2 = mq.Picks.read(os.path.join(str(tmp_path), "in_", "picks"))
    pk2.t[0] += 0.001
    pk2 = mq.Picks(pk2.ev_off, pk2.n_p, pk2.st_id, pk2.x, pk2.y, pk2.z, pk2.t, pk2.cls, pk2.reftime, pk2.fix, pk2.n_stations)
    p = mq.Sampler(a.cfg, pk2, 8, 0, 7)
    p.init_chains()
    foreign["pick_time"] = p.save_state()
    foreign["truncated"] = blob[:-8]
    flipped = bytearray(blob)
    flipped[len(blob) // 2] ^= 0x10
    foreign["flipped_byte"] = bytes(flipped)
    bad = bytearray(blob)
    bad[0:1] = b"X"
    foreign["magic"] = _reseal(bad)
    bad = bytearray(blob)
    bad[8:12] = (2).to_bytes(4, "little")
    foreign["format"] = _reseal(bad)
    before = _snapshot(a)
    for what, other in foreign.items():
        with pytest.raises(mq.MqError) as e:
            a.load_state(other)
        assert e.value.code == MQ_ERR_ARG, (what, str(e.value))
        for x, y in zip(before, _snapshot(a)):
            assert np.array_equal(x, y), what
    a.step(5)                     # and it steps on from where it was
    c, _ll, _rms = a.stats()
    assert (c[:, 17] + c[:, 18] == 9 + 5).all()


def test_save_needs_a_state_and_a_drained_ring(tmp_path):
    import mcmc_eq_b200 as mq
    cfgp, pkp = inputs.materialise("example2", str(tmp_path), j_max_start=30, j_max_main=100000, deci=3)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    s = mq.Sampler(cfg, pk, 16, 0, 7)
    with pytest.raises(mq.MqError) as e:
        s.save_state()
    assert e.value.code == MQ_ERR_STATE
    s.init_chains()
    s.step(12)                    # accepted models since: records wait in the ring
    with pytest.raises(mq.MqError) as e:
        s.save_state()
    assert e.value.code == MQ_ERR_STATE and "undrained" in str(e.value)
    b1 = s.drain_begin()
    s.step(12)
    b2 = s.drain_begin()
    with pytest.raises(mq.MqError) as e:
        s.save_state()
    assert e.value.code == MQ_ERR_BUSY
    r1, _ = s.drain_finish(b1)
    s.drain_finish(b2)
    assert r1
    assert len(s.save_state()) > 0


def test_a_table_hash_that_differs_is_named(tmp_path):
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200._lib import MqStateHeader, MqStateSection
    a = _example2(tmp_path)
    blob = bytearray(a.save_state())
    head = MqStateHeader.from_buffer_copy(bytes(blob[:C.sizeof(MqStateHeader)]))
    secs = [MqStateSection.from_buffer_copy(bytes(blob[C.sizeof(MqStateHeader) + k * C.sizeof(MqStateSection):]))
            for k in range(head.n_sections)]
    tab = [s for s in secs if s.id == 2][0]
    assert tab.bytes == 2 * 8 * 8
    at = tab.offset + 8 * (2 * 3 + 1)                                # chain 3, phase S
    blob[at:at + 8] = ((int.from_bytes(blob[at:at + 8], "little") + 1) % 2**64).to_bytes(8, "little")
    b = mq.Sampler(a.cfg, a.picks, 8, 0, 7)
    with pytest.raises(mq.MqError) as e:
        b.load_state(_reseal(blob))
    assert e.value.code == MQ_ERR_STATE and "S table of chain 3 " in str(e.value), str(e.value)
    b.load_state(bytes(a.save_state()))                            # the untouched state loads
    assert np.array_equal(b.stats()[0], a.stats()[0])


# ---- the command line ------------------------------------------------------------------------------------------------
EXE = os.path.join(util.ROOT, "mcmc_eq_b200", "host", "mcmc_eq")


def _files(d, n):
    return [open(os.path.join(d, f"rjx-{k:03d}.out"), "rb").read() for k in range(1, n + 1)]


def test_a_killed_run_resumed_from_its_checkpoint_writes_the_same_files(tmp_path):
    kw = dict(j_max_start=60, j_max_main=6000, deci=20, true_random=77)
    runs = {}
    for name in ("A", "B"):
        d = str(tmp_path / name)
        runs[name] = d
        cfgp, pkp = inputs.materialise("example2", d, **kw)
    # A: to the end
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "16", "-q"], cwd=runs["A"], capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    want = _files(runs["A"], 16)
    # B: checkpoints after every chunk, killed once a checkpoint exists and a further chunk has run
    d = runs["B"]
    ck = os.path.join(d, "ck")
    p = subprocess.Popen([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "16", "-k", "ck", "-K", "0"], cwd=d,
                         stderr=subprocess.PIPE, stdout=subprocess.DEVNULL, text=True)
    seen_ck = False
    killed = False
    for line in p.stderr:
        if line.startswith("Test"):
            if seen_ck:
                p.send_signal(signal.SIGKILL)
                killed = True
                break
            seen_ck = os.path.exists(ck)
    p.wait(timeout=300)
    p.stderr.close()
    assert killed and p.returncode == -signal.SIGKILL, "run B ended before it could be killed"
    assert os.path.exists(ck)
    partial = _files(d, 16)
    assert any(len(x) < len(y) for x, y in zip(partial, want))
    # C: resumed
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-R", "ck", "-q"], cwd=d, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr
    got = _files(d, 16)
    for k, (x, y) in enumerate(zip(got, want)):
        assert x == y, f"chain file {k + 1} differs"
    # a checkpoint of another configuration is refused before the chain files are touched
    o = str(tmp_path / "other")
    inputs.materialise("example2", o, **dict(kw, deci=21))
    stamp = [os.stat(os.path.join(d, f"rjx-{k:03d}.out")).st_mtime_ns for k in range(1, 17)]
    time.sleep(0.01)
    r = subprocess.run([EXE, os.path.join(o, "config_eqx.dat"), "rjx-%03d.out", "picks", "-R", "ck", "-q"], cwd=d,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "mq_state_load" in r.stderr, r.stderr
    assert _files(d, 16) == want
    assert [os.stat(os.path.join(d, f"rjx-{k:03d}.out")).st_mtime_ns for k in range(1, 17)] == stamp
