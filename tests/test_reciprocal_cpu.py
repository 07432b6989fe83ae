"""Reciprocal travel-time tables without a GPU: the oracle's reciprocal forward, its error against the parity forward on
the committed fixture models, and the command line's checks of a checkpoint's table mode.

The reciprocal table of a (chain, phase) is the field of a solve with its source at each receiver row j, read at every node:
R[j][y][x] = time from (0, j) to (x, y).  It is the parity table with every row kept and its receiver-row and source-depth
axes swapped, R[j][y][x] = P[y][j][x], and built by the same solver from the same sources, so that identity is exact.  The
misfit then reads R[layer][event depth] where the parity forward reads P[layer][event depth]: the difference is the finite-
difference scheme's reciprocity error, |T(a -> b) - T(b -> a)|, measured here per pick (DESIGN.md section 6)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

from tests import fwd_helpers as fh
from tests import inputs, util

EXE = os.path.join(util.ROOT, "mcmc_eq_b200", "host", "mcmc_eq")
STATES = ("z", "vp", "vpvs", "eq", "pres", "sres", "noise")

# Per-pick |t_pred(reciprocal) - t_pred(parity)| on the fixture models below, measured with this oracle (DESIGN.md
# section 6): Example (h = 2 km) max 0.139 s, mean 0.0253 s; Example2 (h = 0.5 km) max 0.0255 s, mean 0.0049 s, and with
# TRIA = 1 max 0.0532 s, mean 0.0057 s.  The bounds are those values rounded up.
ERR_BOUND = {"example": (0.15, 0.03), "example2": (0.03, 0.006), "example2_tria": (0.06, 0.007)}   # (max, mean) s


def oracle_table_reciprocal(g, slow, rows):
    """Reciprocal tables by the oracle's solver, in the layout fm_misfit reads: ttt[j][y][x] = time from a source at
    (0, j) to node (x, y) for every receiver row j in rows (other rows stay zero: the misfit never reads them)."""
    L = util.oracle()
    nz, nxmod = g.nz, L.fm_nxmod(C.byref(g))
    ttt = np.zeros((nz, nz, nxmod), np.float32)
    worst = 0
    for j in rows:
        field, rc = util.oracle_time_2d(slow, nxmod, int(j))
        worst = min(worst, rc)
        ttt[j] = field.T
    return ttt, worst


def _slowness(cfg, g, s, ps):
    L = util.oracle()
    slow = np.zeros(cfg.grid.nz, np.float32)
    (L.fm_rasterise_tria if cfg.tria == 1 else L.fm_rasterise)(C.byref(g), len(s["z"]), util.ptr(util.f32(s["z"])),
                                                               util.ptr(util.f32(s["vp"])), util.ptr(util.f32(s["vpvs"])), ps,
                                                               util.ptr(slow))
    return slow


def _misfit(cfg, pk, s, tabs):
    L = util.oracle()
    g, p = fh.fm_grid(cfg), fh.fm_picks(pk)
    mf, origin = np.zeros(8, np.float32), np.zeros(pk.n_events, np.float32)
    resid, tpred = np.zeros(pk.n_picks, np.float32), np.zeros(pk.n_picks, np.float32)
    rc = L.fm_misfit(C.byref(g), C.byref(p), util.ptr(util.f32(s["eq"])), util.ptr(util.f32(s["pres"])),
                     util.ptr(util.f32(s["sres"])), util.ptr(tabs[0]), util.ptr(tabs[1]), 1, len(s["z"]),
                     util.ptr(util.f32(s["z"])), util.ptr(util.f32(s["vp"])), util.ptr(util.f32(s["vpvs"])), util.ptr(mf),
                     util.ptr(origin), util.ptr(resid), util.ptr(tpred))
    assert rc == 0
    return mf, origin, tpred


def receiver_rows(cfg, pk):
    """The rows the library keeps: layer and layer + 1 of every station, in the library's float arithmetic."""
    lay = ((pk.z - np.float32(cfg.grid.z0)) / np.float32(cfg.grid.h)).astype(np.int32)
    return sorted(set(lay.tolist()) | set((lay + 1).tolist()))


def reciprocal_forward(cfg, pk, s):
    """(mf, origin, tpred) of one chain state through the oracle with reciprocal tables."""
    g = fh.fm_grid(cfg)
    rows = receiver_rows(cfg, pk)
    tabs = []
    for ps in (1, 2):
        t, rc = oracle_table_reciprocal(g, _slowness(cfg, g, s, ps), rows)
        assert rc == 0
        tabs.append(t)
    return _misfit(cfg, pk, s, tabs)


def fixture_states(name):
    """(cfg, picks, states) of the committed forward fixtures: Example / Example2 with TRIA = 0, Example2 with TRIA = 1."""
    import mcmc_eq_b200 as mq
    d = tempfile.mkdtemp(prefix="mqrecip_")
    if name == "example2_tria":
        cfgp, pkp = inputs.materialise("example2", d, tria=1)
        f = np.load(os.path.join(util.GOLDEN, "forward_ref_tria.npz"))
        states = [{k: f[f"{i}_{k}"] for k in STATES} for i in range(int(f["n"]))]
    else:
        cfgp, pkp = inputs.materialise(name, d)
        f = np.load(os.path.join(util.GOLDEN, "forward_ref.npz"))
        states = [{k: f[f"{name}_{i}_{k}"] for k in STATES} for i in range(int(f[f"{name}_n"]))]
    return mq.read_config(cfgp), mq.Picks.read(pkp), states


@pytest.mark.parametrize("name", ["example", "example2", "example2_tria"])
def test_reciprocal_table_is_the_axis_swapped_parity_table(name, oracle):
    cfg, pk, states = fixture_states(name)
    g = fh.fm_grid(cfg)
    nz, nxmod = cfg.grid.nz, oracle.fm_nxmod(C.byref(g))
    row_sets = [receiver_rows(cfg, pk), [0, 1, nz // 2, nz - 2, nz - 1]]
    assert 0 in row_sets[0] + row_sets[1] and nz - 2 in row_sets[1]
    for s in states[:2]:
        for ps in (1, 2):
            slow = _slowness(cfg, g, s, ps)
            par = np.zeros((nz, nz, nxmod), np.float32)
            assert oracle.fm_build_table(C.byref(g), util.ptr(slow), util.ptr(par)) == 0
            swapped = np.transpose(par, (1, 0, 2))          # [source][row][x]
            for rows in row_sets:
                rec, rc = oracle_table_reciprocal(g, slow, rows)
                assert rc == 0
                assert np.array_equal(rec[rows].view(np.uint32), swapped[rows].view(np.uint32)), (name, ps, rows)


@pytest.mark.parametrize("name", ["example", "example2", "example2_tria"])
def test_reciprocity_error_per_pick(name, oracle):
    """What the approximation costs: per-pick predictions of the reciprocal forward against the parity forward."""
    cfg, pk, states = fixture_states(name)
    errs = []
    for s in states:
        _mf, _org, _res, tp = fh.oracle_forward(cfg, pk, s["z"], s["vp"], s["vpvs"], s["eq"], s["pres"], s["sres"])
        _rmf, _rorg, rtp = reciprocal_forward(cfg, pk, s)
        ok = (tp < 1e29) & (rtp < 1e29)
        assert np.array_equal(ok, tp < 1e29)            # the same picks fall outside the table in both modes
        errs.append(np.abs(rtp[ok] - tp[ok]).astype(np.float64))
    e = np.concatenate(errs)
    emax, emean = ERR_BOUND[name]
    print(f"{name}: {e.size} picks, max {e.max():.5f} s, mean {e.mean():.5f} s, p99 {np.percentile(e, 99):.5f} s")
    assert e.max() <= emax and e.mean() <= emean, (name, float(e.max()), float(e.mean()))
    assert e.max() > 0.0                                 # the two modes are not the same forward


# ---- the command line: a checkpoint's table mode is checked before a handle exists ------------------------------------
def _checkpoint(path, flags, n_chains=4):
    """A checkpoint file whose sampler state is a bare header with the given flags: it passes every check the command
    line makes without the library (the library refuses it later: bad checksum)."""
    from mcmc_eq_b200._lib import MqStateHeader
    head = MqStateHeader()
    head.magic = b"MQSTATE"
    head.format = 1
    head.header_bytes = C.sizeof(MqStateHeader)
    head.n_chains = n_chains
    head.flags = flags
    state = bytes(head) + bytes(64)
    ck = b"MQCKPT1\0" + np.array([n_chains, 0], np.int32).tobytes() + np.array([7], np.uint64).tobytes() + \
        np.array([20, 0], np.int64).tobytes() + np.array([len(state)], np.uint64).tobytes()
    with open(path, "wb") as f:
        f.write(ck + np.zeros(n_chains, np.int64).tobytes() + state)


def _resume(d, *extra):
    assert os.path.exists(EXE), "host/mcmc_eq not built (python -m mcmc_eq_b200.build)"
    return subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-R", "ck", "-q", *extra], cwd=d, capture_output=True,
                          text=True, timeout=120)


@pytest.mark.parametrize("flags, x, refused", [
    (4 | 16, False, False),     # reciprocal checkpoint: -R takes the mode from it
    (4 | 16, True, False),      # ... and -x agrees with it
    (4, True, True),            # -x against a parity checkpoint
    (4, False, False),          # parity checkpoint, no -x
])
def test_resume_checks_the_table_mode_first(tmp_path, flags, x, refused):
    from mcmc_eq_b200._lib import STATE_RECIPROCAL, STATE_TABLES
    assert (STATE_TABLES, STATE_RECIPROCAL) == (4, 16)
    d = str(tmp_path)
    inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=77)
    _checkpoint(os.path.join(d, "ck"), flags)
    r = _resume(d, *(["-x"] if x else []))
    assert r.returncode != 0                              # the bare state never loads
    assert not [f for f in os.listdir(d) if f.startswith("rjx-")]
    if refused:
        assert "parity tables" in r.stderr and "mq_create" not in r.stderr, r.stderr
    else:
        # past every host-side check: what fails is the library (no device here, or the state's checksum on a GPU)
        assert "parity tables" not in r.stderr and ("mq_create" in r.stderr or "mq_state_load" in r.stderr), r.stderr


# ---- the reciprocal instantiations of the pipelined kernel, from the compiler alone ----------------------------------------
def test_reciprocal_pipe_kernels_fit_their_warps():
    """eik_pipe_recip_kernel (CA = 64 with 12 warps, CA = 128 with 8) keeps the parity kernel's resource limits: registers
    within what its warps per CTA allow, no stack frame, no local memory from the generic sweep."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("sass_footprint", os.path.join(util.ROOT, "tools", "sass_footprint.py"))
    sf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(sf)
    if not all(sf.cuda_bin(t) for t in ("nvcc", "cuobjdump", "nvdisasm")):
        pytest.skip("needs nvcc, cuobjdump and nvdisasm")
    with tempfile.TemporaryDirectory() as d:
        cubin = sf.compile_cubin(util.ROOT, os.path.join(d, "eikonal.cubin"))
        fp = [e for e in sf.footprint(cubin) if "eik_pipe_recip_kernel" in e["mangled"]]
    ca = {e["mangled"]: 64 if "ILi64E" in e["mangled"] else 128 for e in fp}
    assert sorted(ca.values()) == [64, 128]
    for e in fp:
        w = {64: 12, 128: 8}[ca[e["mangled"]]]
        assert e["registers"] <= min(255, (65536 // (w * 32)) // 8 * 8), (e["kernel"], e["registers"])
        assert e["stack"] == 0 and e["local_by_file"].get("eik_core.cuh", 0) == 0, e["kernel"]
