"""The CPU oracle (oracle/*.c) is pinned here: bit-for-bit against fixtures generated from the
unmodified reference (tests/golden, tools/make_golden.py) and, when oracle/_ref is present,
against the compiled reference itself on fresh seeded inputs."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import util, inputs
from tests.util import f32, ptr


def test_eikonal_oracle_matches_golden_bitwise(oracle):
    d, meta = util.golden_eikonal()
    st = util.PlStats()
    for i, (gname, kind, iz) in enumerate(meta):
        s, tref = d[f"s_{i}"], d[f"t_{i}"]
        t, rc = util.oracle_time_2d(s, tref.shape[0], int(iz), C.byref(st))
        assert rc == 0
        assert np.array_equal(t.view(np.uint32), tref.view(np.uint32)), (i, gname, kind, iz)
    # the fixtures exercise every irregular branch of the solver
    assert st.recursive_init > 0 and st.nearest_init > 0 and st.box_init > 0
    assert st.headwaves > 0 and st.reverse_sweeps > 0


def test_eikonal_oracle_matches_reference_live(oracle, reflib):
    rng = np.random.default_rng(11)
    for trial in range(24):
        nz, nx = int(rng.integers(6, 66)), int(rng.integers(8, 290))
        kind = ["posterior", "contrast", "lvz", "gradient"][trial % 4]
        z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(1, 21)), 0.0, (nz - 1) * 2.0, kind)
        s = util.rasterise_np(z, vp, vpvs, 2.0, 0.0, nz, 1 + trial % 2)
        for iz in rng.integers(0, nz, 5):
            t1, r1 = util.oracle_time_2d(s, nx, int(iz))
            t2, r2 = util.ref_time_2d(s, nx, int(iz))
            assert r1 == r2
            assert np.array_equal(t1.view(np.uint32), t2.view(np.uint32))


def test_eikonal_oracle_general_media_live(oracle, reflib):
    """2-D heterogeneous media and interior sources: the restatement is the full algorithm."""
    rng = np.random.default_rng(12)
    for trial in range(40):
        nx, ny = int(rng.integers(3, 50)), int(rng.integers(3, 50))
        hs = f32(rng.uniform(0.2, 1.0, (nx, ny))) if trial % 2 else f32(np.kron(rng.uniform(0.2, 1, (nx // 5 + 1, ny // 5 + 1)), np.ones((5, 5)))[:nx, :ny])
        xs, ys = float(rng.integers(0, nx)), float(rng.integers(0, ny))
        t1 = np.zeros((nx, ny), np.float32)
        t2 = np.zeros((nx, ny), np.float32)
        h2 = hs.copy()
        r1 = oracle.pl_time_2d(ptr(hs), ptr(t1), nx, ny, xs, ys, 0.001, None)
        r2 = reflib.time_2d(ptr(h2), ptr(t2), nx, ny, xs, ys, 0.001, 0)
        assert r1 == r2 and np.array_equal(t1.view(np.uint32), t2.view(np.uint32))


def test_eikonal_oracle_error_codes(oracle):
    hs = np.full((4, 4), 0.5, np.float32)
    t = np.zeros((4, 4), np.float32)
    assert oracle.pl_time_2d(ptr(hs), ptr(t), 1, 4, 0.0, 0.0, 0.001, None) == -8     # ERR_DIM
    assert oracle.pl_time_2d(ptr(hs), ptr(t), 4, 4, 0.0, 0.0, 2.0, None) == -5       # ERR_EPS
    bad = hs.copy(); bad[1, 1] = -1.0
    assert oracle.pl_time_2d(ptr(bad), ptr(t), 4, 4, 0.0, 0.0, 0.001, None) == -7    # ERR_PHYS
    bad[1, 1] = 1e19
    assert oracle.pl_time_2d(ptr(bad), ptr(t), 4, 4, 0.0, 0.0, 0.001, None) == -6    # ERR_RANGE


def _example(name):
    import mcmc_eq_b200 as mq
    import tempfile
    d = tempfile.mkdtemp(prefix="mqin_")
    cfgp, pkp = inputs.materialise(name, d)
    return mq.read_config(cfgp), mq.Picks.read(pkp)


@pytest.mark.parametrize("name", ["example2", "example"])
def test_forward_oracle_matches_golden_bitwise(oracle, name):
    """Rasteriser + nz eikonal solves + lookup + residual loop == the reference's cal_fit_newx."""
    from tests import fwd_helpers as fh
    cfg, pk = _example(name)
    d = np.load(os.path.join(util.GOLDEN, "forward_ref.npz"))
    for i in range(int(d[f"{name}_n"])):
        s = {k: d[f"{name}_{i}_{k}"] for k in ("z", "vp", "vpvs", "eq", "pres", "sres")}
        mf, origin, _r, _t, tabs = fh.oracle_forward(cfg, pk, s["z"], s["vp"], s["vpvs"], s["eq"], s["pres"], s["sres"], True)
        assert np.array_equal(mf.view(np.uint32), d[f"{name}_{i}_mf"].view(np.uint32)), (name, i, mf, d[f"{name}_{i}_mf"])
        assert np.array_equal(origin.view(np.uint32), d[f"{name}_{i}_origin"].view(np.uint32))
        if i == 0:
            assert np.array_equal(tabs[0][1:3], d[f"{name}_{i}_tabP_rows12"])


def test_inputs_roundtrip():
    """materialise() -> our readers gives back the stored arrays (format of src/mcmc_eq.c:1238-1294)."""
    for name, ne, npk, ns in (("example", 220, 15081, 130), ("example2", 225, 3600, 8)):
        cfg, pk = _example(name)
        _c, arr = inputs.load(name)
        assert (pk.n_events, pk.n_picks, pk.n_stations) == (ne, npk, ns)
        assert np.array_equal(pk.ev_off, arr["ev_off"]) and np.array_equal(pk.n_p, arr["n_p"])
        assert np.array_equal(pk.x, arr["x"]) and np.array_equal(pk.t, arr["t64"].astype(np.float32))
        assert np.array_equal(pk.cls, arr["cls"]) and np.array_equal(pk.st_id, arr["st_id"])
    assert cfg.grid.nz == 61 and abs(cfg.grid.h - 0.5) < 1e-7 and cfg.dstring_main == b"QVRPBDMN"


def test_chain_scalars_match_reference_live(oracle, reflib):
    rng = np.random.default_rng(5)
    reflib.nexp.restype = C.c_float
    reflib.nexp.argtypes = [C.c_float]
    for v in list(rng.uniform(-200, 200, 200)) + [81.8, 81.9, 88.0, 1e9, -1e9]:
        assert oracle.ch_nexp(v) == reflib.nexp(v)
    from tests import refapi
    reflib.model_valid.argtypes = [C.POINTER(refapi.Model), C.c_float, C.c_float, C.c_float, C.c_float]
    n_valid = 0
    for trial in range(300):
        dim = int(rng.integers(1, 25))
        kind = "gradient" if trial % 2 else "lvz"
        z, vp, vpvs = util.voronoi_model(rng, dim, -4.0, 118.0, kind)
        inv = float(rng.choice([-1.0, -0.05, 0.05, 1.0]))
        m = refapi.Model()
        m.dimension = dim
        for i in range(dim):
            m.z[i], m.vp[i], m.vpvs[i] = float(z[i]), float(vp[i]), float(vpvs[i])
        a = reflib.model_valid(C.byref(m), 2.0, -4.0, 118.0, inv)
        b = oracle.ch_model_valid(dim, ptr(z), ptr(vp), ptr(vpvs), 2.0, -4.0, 118.0, inv)
        assert a == b
        n_valid += (a == 0)
    assert 20 < n_valid < 280


def test_chain_oracle_reproduces_every_recorded_decision(oracle):
    """Chain level of the oracle: the reference's proposal stream (tests/golden/replay_example2.npz, recorded from the
    unmodified reference by oracle/replay_log.c) scored with the oracle's restatement -- class sums from fm_misfit +
    tables for a sample of the proposals, likelihood / proposal ratio / alpha from oracle/chain.c for all of them --
    must give the reference's accept/reject decision for all 312 evaluated proposals."""
    import tempfile
    import mcmc_eq_b200 as mq
    from tests import replay, fwd_helpers as fh
    log = replay.load("example2")
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=77)
        cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    assert len(log["u"]) == 313 and int(log["accepted"][1:].sum()) == 200
    old_ll = replay.loglik(log["mf"][0], log["noise"][0])
    kinds = {}
    for i, kind, q, lf, u, acc, cur, prop in replay.proposals(log, cfg, pk.n_class):
        kinds[kind] = kinds.get(kind, 0) + 1
        new_ll = replay.loglik(log["mf"][i], prop["noise"])
        alpha = oracle.ch_alpha(lf, new_ll, old_ll)
        assert (u < alpha) == acc, (i, kind, u, alpha, acc)
        if acc:
            old_ll = new_ll
        if i % 40 == 1 or kind in "BD":   # full forward of the oracle on a sample (each costs ~2 x 61 eikonal solves)
            mf, origin, _r, _t = fh.oracle_forward(cfg, pk, prop["z"], prop["vp"], prop["vpvs"], prop["eq"], prop["pres"], prop["sres"])
            assert np.array_equal(mf, log["mf"][i]), (i, kind)
            assert np.array_equal(origin, prop["origin"])
    assert set(kinds) == set("QRPVMBDN"), kinds     # every arm of the proposal switch occurs in the recorded chain


# ---- the linear-gradient parameterisation (config line 29 = 1) ---------------------------------------------------------
def test_tria_forward_oracle_matches_golden_bitwise(oracle):
    """fm_rasterise_tria (src/misfit.c:217-250) + tables + residual loop == cal_fit_newx of the compiled reference with
    TRIA = 1 (tests/golden/forward_ref_tria.npz): states with nuclei at equal depths and with the two end nuclei only."""
    import tempfile
    import mcmc_eq_b200 as mq
    from tests import fwd_helpers as fh
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, tria=1)
        cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    assert cfg.tria == 1
    d = np.load(os.path.join(util.GOLDEN, "forward_ref_tria.npz"))
    for i in range(int(d["n"])):
        s = {k: d[f"{i}_{k}"] for k in ("z", "vp", "vpvs", "eq", "pres", "sres")}
        mf, origin, _r, _t, tabs = fh.oracle_forward(cfg, pk, s["z"], s["vp"], s["vpvs"], s["eq"], s["pres"], s["sres"], True)
        assert np.array_equal(mf.view(np.uint32), d[f"{i}_mf"].view(np.uint32)), (i, mf, d[f"{i}_mf"])
        assert np.array_equal(origin.view(np.uint32), d[f"{i}_origin"].view(np.uint32))
        if i == 0:
            assert np.array_equal(tabs[0][1:3], d["0_tabP_rows12"]) and np.array_equal(tabs[1][1:3], d["0_tabS_rows12"])


def test_tria_chain_oracle_reproduces_every_recorded_decision(oracle):
    """The recorded TRIA = 1 chain of the unmodified reference (tests/golden/replay_example2_tria.npz): decisions from
    oracle/chain.c for every proposal, class sums from the oracle's forward for a sample; the two end nuclei are never
    moved or removed (src/mcmc_eq.c:990-998,1059-1067)."""
    import tempfile
    import mcmc_eq_b200 as mq
    from tests import replay, fwd_helpers as fh
    log = replay.load("example2_tria")
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=78, tria=1)
        cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    g = cfg.grid
    zmin, zmax = np.float32(g.z0), np.float32(g.z0 + (g.nz - 1) * g.h)
    old_ll = replay.loglik(log["mf"][0], log["noise"][0])
    kinds = {}
    for i, kind, q, lf, u, acc, cur, prop in replay.proposals(log, cfg, pk.n_class):
        kinds[kind] = kinds.get(kind, 0) + 1
        assert prop["dim"] >= 2 and prop["z"][0] == zmin and prop["z"][1] == zmax, (i, kind)
        new_ll = replay.loglik(log["mf"][i], prop["noise"])
        alpha = oracle.ch_alpha(lf, new_ll, old_ll)
        assert (u < alpha) == acc, (i, kind, u, alpha, acc)
        if acc:
            old_ll = new_ll
        if i % 40 == 1 or kind in "BDM":
            mf, origin, _r, _t = fh.oracle_forward(cfg, pk, prop["z"], prop["vp"], prop["vpvs"], prop["eq"], prop["pres"], prop["sres"])
            assert np.array_equal(mf, log["mf"][i]), (i, kind)
            assert np.array_equal(origin, prop["origin"])
    assert set(kinds) >= set("QRPVBN"), kinds
