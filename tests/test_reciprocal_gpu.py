"""Reciprocal travel-time tables on the device (mq_set_tables, MQ_TABLES_RECIPROCAL): one solve per receiver row with the
source at that row, every row of its field stored (csrc/eikonal.cu: EikBatch::src_rows).

Implementation parity is exact: the stored rows of a reciprocal handle (mq_get_rows) are the axis-swapped full table of a
parity handle with the same models (mq_get_table), R[r][y][x] = P[y][row_index[r]][x], BIT FOR BIT -- on every kernel,
each case asserting through mq_profile_kernels which one ran.  The forward on those tables matches the oracle's reciprocal
forward (tests/test_reciprocal_cpu.py) within the misfit tolerances (1e-4 s per pick, 2e-5 relative on class sums).  The
sampler keeps its invariants in this mode (lock-step = desynchronised, maintained = fresh likelihood, save / load /
continue bit for bit), a state of one mode is refused by a handle of the other, and the command line's -x works end to
end."""
import ctypes as C
import os
import signal
import subprocess
import sys
import tempfile
import time

import numpy as np
import pytest

from tests import fwd_helpers as fh
from tests import inputs, util
from tests.test_reciprocal_cpu import fixture_states, reciprocal_forward
from tests.test_receiver_rows_gpu import EX2, HALVED, TALL, make_case, _states

pytestmark = pytest.mark.gpu

MQ_ERR_ARG, MQ_ERR_UNSUPPORTED, MQ_ERR_STATE = -1, -3, -7
EXE = os.path.join(util.ROOT, "mcmc_eq_b200", "host", "mcmc_eq")
FW_MOD = os.path.join(util.ROOT, "mcmc_eq_b200", "host", "fw_mod")


def _forward(cfg, pk, states, n, mode):
    """A handle of `mode` with the states loaded and forwarded -> (sampler, mf, origin, kernels of the table launch)."""
    import mcmc_eq_b200 as mq
    smp = mq.Sampler(cfg, pk, n, 0, 1)
    smp.set_tables(mode)
    smp.profile(True)
    mf, org = smp.forward_host(fh.fill_models(smp.new_models(), states), 3)
    smp.profile(False)
    return smp, mf, org, list(smp.profile_kernels())


def _check_swapped(rec, par, sample):
    """rows of the reciprocal handle == the axis-swapped full tables of the parity handle, bit for bit."""
    for c in sample:
        for ph in (1, 2):
            rows, idx = rec.rows(c, ph)
            full = par.table(c, ph)                       # [row][source][x]
            want = np.ascontiguousarray(np.transpose(full, (1, 0, 2))[idx])
            assert np.array_equal(rows.view(np.uint32), want.view(np.uint32)), (c, ph, int((rows != want).sum()))


def _check_oracle(cfg, pk, states, rec, mf, org, sample):
    for c in sample:
        rmf, rorg, rtp = reciprocal_forward(cfg, pk, states[c])
        tp = rec.predictions(c)[1]
        assert np.abs(tp - rtp).max() <= 1e-4, (c, float(np.abs(tp - rtp).max()))
        assert np.allclose(mf[c], rmf, rtol=2e-5, atol=1e-6), (c, mf[c], rmf)
        assert np.abs(org[c] - rorg).max() <= 1e-4


@pytest.mark.parametrize("name", ["example", "example2", "example2_tria"])
def test_fixture_models_fused_kernel(name):
    """The committed fixture models (Example, Example2, TRIA = 1): fused kernel, exact tables, oracle forward."""
    cfg, pk, states = fixture_states(name)
    n = len(states)
    rec, mf, org, kernels = _forward(cfg, pk, states, n, "reciprocal")
    assert kernels == ["eik_fast_kernel"]
    par = _forward(cfg, pk, states, n, "parity")[0]
    _check_swapped(rec, par, range(n))
    _check_oracle(cfg, pk, states, rec, mf, org, range(n))
    # no parity table exists in this mode
    with pytest.raises(Exception) as ei:
        rec.table(0, 1)
    assert ei.value.code == MQ_ERR_UNSUPPORTED
    rec.close()
    par.close()


@pytest.mark.parametrize("grid, which, n, kernel, sample", [
    ("EX2", "dozen", 2000, "eik_pipe_kernel", [0, 1, 1999]),       # CA = 64: 2000 x 2 x 16 rows = 2000 warp tasks
    ("HALVED", "all", 170, "eik_pipe_kernel", [0, 169]),           # CA = 128: 170 x 2 x 121 rows = 1286 warp tasks
    ("EX2", "dozen", 8, "eik_fast_kernel", [0, 1, 7]),
    ("TALL", "deep", 2, "eik_fine_kernel", [0, 1]),                # 90 x 700 plane, global-memory slices
])
def test_every_kernel_stores_the_axis_swapped_parity_table(grid, which, n, kernel, sample):
    g = {"EX2": EX2, "HALVED": HALVED, "TALL": TALL}[grid]
    cfg, pk, _rows = make_case(g, which)
    states = _states(cfg, pk, n, 12)
    rec, mf, org, kernels = _forward(cfg, pk, states, n, "reciprocal")
    assert kernels == [kernel]
    par = _forward(cfg, pk, states, n, "parity")[0]
    _check_swapped(rec, par, sample)
    _check_oracle(cfg, pk, states, rec, mf, org, sample[:2])
    rec.close()
    par.close()


GENERIC_SCRIPT = r"""
import sys, numpy as np
sys.path.insert(0, %r)
from tests.test_reciprocal_gpu import _forward, _check_swapped, _check_oracle
from tests.test_reciprocal_cpu import fixture_states
cfg, pk, states = fixture_states("example2")
n = len(states)
rec, mf, org, kernels = _forward(cfg, pk, states, n, "reciprocal")
assert kernels == ["eik_generic_kernel"], kernels
par = _forward(cfg, pk, states, n, "parity")[0]
_check_swapped(rec, par, range(n))
_check_oracle(cfg, pk, states, rec, mf, org, range(n))
print("ok")
"""


def test_generic_kernel():
    r = subprocess.run([sys.executable, "-c", GENERIC_SCRIPT % util.ROOT], env=dict(os.environ, MCMCEQ_EIKONAL="generic"),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stderr[-3000:]


# ---- the sampler in reciprocal mode ----------------------------------------------------------------------------------------
SAMPLER_SCRIPT = r"""
import sys, tempfile, numpy as np
sys.path.insert(0, %r)
import mcmc_eq_b200 as mq
from tests import inputs
d = tempfile.mkdtemp(prefix="mqrs_")
cfgp, pkp = inputs.materialise("example2", d, j_max_start=30, j_max_main=100000, deci=7)
cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
smp = mq.Sampler(cfg, pk, 97, 0, 21)
smp.set_tables("reciprocal")
smp.init_chains()
try:
    smp.set_tables("parity")
    raise SystemExit("mq_set_tables after mq_init_chains was accepted")
except mq.MqError as e:
    assert e.code == -7, e.code
recs = []
for chunk in (7, 5, 7, 7, 4, 6):
    smp.step(chunk)
    r, lost = smp.drain()
    assert lost == 0
    recs += r
smp.step(6, "QVRPBDMN")
smp.step(5, "P")
c, ll, rms = smp.stats()
m = smp.get_models()
out = dict(c=c, ll=ll, rms=rms, rec_number=np.array([r["number"] for r in recs]), rec_rms=np.array([r["rms"] for r in recs]))
for f in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise", "origin"):
    out[f] = getattr(m, f)
smp.forward(3)
c2, ll2, rms2 = smp.stats()
out["ll_fresh"] = ll2; out["rms_fresh"] = rms2
np.savez(sys.argv[1], **out)
"""


def test_lock_step_and_desynchronised_agree_and_keep_the_likelihood(tmp_path):
    res = {}
    for desync in ("0", "1"):
        path = str(tmp_path / f"d{desync}.npz")
        r = subprocess.run([sys.executable, "-c", SAMPLER_SCRIPT % util.ROOT, path], env=dict(os.environ, MCMCEQ_DESYNC=desync),
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        res[desync] = dict(np.load(path))
    a, b = res["0"], res["1"]
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert a["rec_number"].size > 0 and a["c"][:, 17].sum() > 0
    # the maintained likelihood is the one a fresh reciprocal forward gives
    assert np.allclose(a["ll_fresh"], a["ll"], rtol=2e-5, atol=1e-3), np.abs(a["ll_fresh"] - a["ll"]).max()
    assert np.allclose(a["rms_fresh"], a["rms"], rtol=1e-5)


def _sampler(tmp_path, mode, n=12, seed=3):
    import mcmc_eq_b200 as mq
    d = str(tmp_path / "in")
    if not os.path.exists(d):
        inputs.materialise("example2", d, j_max_start=30, j_max_main=100000, deci=7)
    cfg, pk = mq.read_config(os.path.join(d, "config_eqx.dat")), mq.Picks.read(os.path.join(d, "picks"))
    s = mq.Sampler(cfg, pk, n, 0, seed)
    s.set_tables(mode)
    return s


def test_save_load_continue_and_mode_refusals(tmp_path):
    import mcmc_eq_b200 as mq
    from tests.test_state_gpu import _continue_and_compare
    a = _sampler(tmp_path, "reciprocal")
    a.init_chains()
    a.step(9, "QVRPBDMN")
    a.drain()
    blob = a.save_state()
    head = mq._lib.MqStateHeader.from_buffer_copy(blob[:C.sizeof(mq._lib.MqStateHeader)])
    assert head.flags & mq._lib.STATE_RECIPROCAL and head.flags & mq._lib.STATE_TABLES and head.format == 1
    b = _sampler(tmp_path, "reciprocal", seed=5)
    b.profile(True)
    b.load_state(blob)
    b.profile(False)
    assert list(b.profile_kernels()) == ["eik_fast_kernel"]
    assert b.save_state() == blob
    _continue_and_compare(a, b, 4)
    with pytest.raises(mq.MqError) as ei:
        b.set_tables("parity")                  # the handle holds a state now
    assert ei.value.code == MQ_ERR_STATE
    # a parity handle refuses the reciprocal state and stays usable; and the reverse
    p = _sampler(tmp_path, "parity")
    with pytest.raises(mq.MqError) as ei:
        p.load_state(blob)
    assert ei.value.code == MQ_ERR_ARG
    p.init_chains()
    p.step(4)
    p.drain()
    pblob = p.save_state()
    assert not mq._lib.MqStateHeader.from_buffer_copy(pblob[:C.sizeof(mq._lib.MqStateHeader)]).flags & mq._lib.STATE_RECIPROCAL
    r = _sampler(tmp_path, "reciprocal")
    with pytest.raises(mq.MqError) as ei:
        r.load_state(pblob)
    assert ei.value.code == MQ_ERR_ARG
    r.load_state(blob)                          # still fresh: the state of its own mode loads
    r.step(2)
    with pytest.raises(ValueError):
        _sampler(tmp_path, "transposed")
    for s in (a, b, p, r):
        s.close()


# ---- the command line --------------------------------------------------------------------------------------------------------
def _files(d, n):
    return [open(os.path.join(d, f"rjx-{k:03d}.out"), "rb").read() for k in range(1, n + 1)]


def test_mcmc_eq_x_killed_and_resumed_writes_the_same_files(tmp_path):
    kw = dict(j_max_start=60, j_max_main=3000, deci=20, true_random=77)
    runs = {}
    for name in ("A", "B", "P"):
        runs[name] = str(tmp_path / name)
        inputs.materialise("example2", runs[name], **kw)
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "8", "-q", "-x"], cwd=runs["A"], capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    assert sum("reciprocal travel-time tables" in line for line in r.stderr.split("\n")) == 1, r.stderr
    want = _files(runs["A"], 8)
    d = runs["B"]
    p = subprocess.Popen([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "8", "-x", "-k", "ck", "-K", "0"], cwd=d,
                         stderr=subprocess.PIPE, stdout=subprocess.DEVNULL, text=True)
    seen_ck = killed = False
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
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-R", "ck", "-q"], cwd=d, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr
    assert "reciprocal travel-time tables" in r.stderr       # the mode came from the checkpoint
    assert _files(d, 8) == want
    # a parity run's checkpoint with -x: refused before the chain files are touched
    dp = runs["P"]
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "8", "-q", "-k", "ck", "-K", "0"], cwd=dp,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr
    files = _files(dp, 8)
    stamp = [os.stat(os.path.join(dp, f"rjx-{k:03d}.out")).st_mtime_ns for k in range(1, 9)]
    time.sleep(0.01)
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-R", "ck", "-q", "-x"], cwd=dp, capture_output=True,
                       text=True, timeout=300)
    assert r.returncode != 0 and "parity tables" in r.stderr and "mq_create" not in r.stderr, r.stderr
    assert _files(dp, 8) == files
    assert [os.stat(os.path.join(dp, f"rjx-{k:03d}.out")).st_mtime_ns for k in range(1, 9)] == stamp


def test_fw_mod_x_matches_the_oracle_reciprocal_forward():
    sys.path.insert(0, os.path.join(util.ROOT, "tools"))
    from make_golden import last_block
    import mcmc_eq_b200 as mq
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=77)
        blk = os.path.join(d, "block")
        block = last_block(open(os.path.join(util.GOLDEN, "chain_ref_example2.out")).read())
        open(blk, "w").write(block)
        out = {}
        for x in (False, True):
            r = subprocess.run([FW_MOD, cfgp, blk, pkp] + (["-x"] if x else []), cwd=d, capture_output=True, text=True, timeout=300)
            assert r.returncode == 0, r.stderr
            assert ("reciprocal travel-time tables" in r.stderr) == x
            out[x] = [ln.split() for ln in r.stdout.strip().split("\n")]
        cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    # the model block as the oracle wants it
    lines = block.strip().split("\n")
    tok = lines[0].split()
    dim = int(tok[3])
    nuc = np.array([float(v) for v in tok[13:13 + 3 * dim]], np.float32).reshape(dim, 3)
    ne, ns = pk.n_events, pk.n_stations
    eq = np.array([[float(v) for v in ln.split()[5:8]] for ln in lines[1:1 + ne]], np.float32)
    res = np.array([[float(v) for v in ln.split()[5:7]] for ln in lines[1 + ne:1 + ne + ns]], np.float32)
    s = dict(z=nuc[:, 0], vp=nuc[:, 1], vpvs=nuc[:, 2], eq=eq, pres=res[:, 0], sres=res[:, 1])
    _rmf, _rorg, rtp = reciprocal_forward(cfg, pk, s)
    got = np.array([float(t[5]) for t in out[True] if t[0] != "EVENT"], np.float32)
    par = np.array([float(t[5]) for t in out[False] if t[0] != "EVENT"], np.float32)
    assert got.size == rtp.size == pk.n_picks
    assert np.abs(got - rtp).max() < 1e-4 + 1e-5, float(np.abs(got - rtp).max())   # printed with %f: 1e-6 s
    assert np.abs(got - par).max() > 0.0                 # -x is not the parity forward
