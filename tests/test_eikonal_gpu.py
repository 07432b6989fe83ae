"""Parity of the CUDA eikonal path (through the C ABI) with the oracle and the reference fixtures.
Tolerance: |dT| <= max(1e-4 s, 2e-6 T) -- FP32 restatement bound, SURVEY.md Appendix A.5."""

import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu


def test_batch_matches_golden_reference_fields():
    import mcmc_eq_b200 as mq
    d, meta = util.golden_eikonal()
    groups = {}
    for i, m in enumerate(meta):
        tref = d[f"t_{i}"]
        groups.setdefault(tref.shape, []).append((d[f"s_{i}"], int(m[2]), tref))
    worst = 0.0
    for (nx, nz), items in groups.items():
        t = mq.eikonal_batch(np.array([s for s, _, _ in items]), [iz for _, iz, _ in items], nx)
        for k, (_s, _iz, tref) in enumerate(items):
            err = np.abs(t[k] - tref)
            assert (err <= util.eikonal_tol(tref)).all(), (nx, nz, _iz, err.max())
            worst = max(worst, float(err.max()))
    assert worst < 1e-4


@pytest.mark.parametrize("grid,kind,seed", [(util.EXAMPLE_GRID, "posterior", 1), (util.EXAMPLE_GRID, "contrast", 2),
                                            (util.EXAMPLE2_GRID, "posterior", 3), (util.EXAMPLE2_GRID, "lvz", 4),
                                            (util.EXAMPLE_GRID, "gradient", 5)])
def test_full_tables_match_oracle(oracle, grid, kind, seed):
    """Every source depth of seeded models, both phases (what setup_table_new computes)."""
    import mcmc_eq_b200 as mq
    rng = np.random.default_rng(seed)
    nx, nz = util.nxmod_of(grid), grid["nz"]
    slows, izs = [], []
    for _ in range(3):
        z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(1, 21)), grid["z0"], grid["z0"] + (nz - 1) * grid["h"], kind)
        for ps in (1, 2):
            s = util.rasterise_np(z, vp, vpvs, grid["h"], grid["z0"], nz, ps)
            slows += [s] * nz
            izs += list(range(nz))
    t, st, rc = mq.eikonal_batch(np.array(slows), izs, nx, return_status=True)
    assert rc == 0 and (st == 0).all()
    nbad = 0
    stats = util.PlStats()
    import ctypes as C
    for k in range(len(izs)):
        tref, _ = util.oracle_time_2d(slows[k], nx, izs[k], C.byref(stats))
        nbad += int((np.abs(t[k] - tref) > util.eikonal_tol(tref)).any())
    assert nbad == 0
    assert stats.recursive_init > 0


@pytest.mark.parametrize("nz", [61, 62, 63])
def test_source_in_the_middle_of_its_layer_at_mid_depth(oracle, nz):
    """The widest box the solver's shared row buffer has to hold (top and bottom row at full length in the same round): a
    source in the middle of a layer that is itself in the middle of the depth range.  With a row buffer of nz + 4 nodes an
    odd nz (the Example2 grid has 61) lost the top row's newest node to the bottom row's: 2.7 s off along the top of the
    plane.  tests/test_emu_cpu.py holds the same case on the host build."""
    import mcmc_eq_b200 as mq
    nx = util.nxmod_of(util.EXAMPLE2_GRID)
    mid = (nz - 1) // 2
    slows, izs = [], []
    for half in (7, 11, 12):
        for iz in (mid - 1, mid, mid + 1):
            s = np.full(nz, 0.1263643, np.float32)
            s[:iz - half] = 0.2491149
            s[iz - half:iz + half + 1] = 0.2100524
            slows.append(s)
            izs.append(iz)
    t, st, rc = mq.eikonal_batch(np.array(slows), izs, nx, return_status=True)
    assert rc == 0 and (st == 0).all()
    for k in range(len(izs)):
        tref, _ = util.oracle_time_2d(slows[k], nx, izs[k])
        err = np.abs(t[k] - tref)
        assert (err <= util.eikonal_tol(tref)).all(), (nz, izs[k], float(err.max()))


def test_edge_grids_and_ragged_batches(oracle):
    import mcmc_eq_b200 as mq
    rng = np.random.default_rng(9)
    for nx, nz, n in ((2, 2, 1), (2, 7, 5), (7, 2, 33), (11, 12, 64), (12, 11, 95), (300, 9, 3)):
        z, vp, vpvs = util.voronoi_model(rng, 3, 0.0, float(nz - 1), "contrast")
        s = util.rasterise_np(z, vp, vpvs, 1.0, 0.0, nz, 1)
        izs = rng.integers(0, nz, n)
        t = mq.eikonal_batch(np.tile(s, (n, 1)), izs, nx)
        for k in range(n):
            tref, rc = util.oracle_time_2d(s, nx, int(izs[k]))
            assert rc == 0 and (np.abs(t[k] - tref) <= util.eikonal_tol(tref)).all(), (nx, nz, izs[k])
    # empty batch and bad arguments
    assert mq.eikonal_batch(np.zeros((0, 5), np.float32), [], 6).shape == (0, 6, 5)
    with pytest.raises(mq.MqError):
        mq.eikonal_batch(np.ones((1, 5), np.float32), [7], 6)


def test_time_2d_dropin_signature(oracle):
    """mq_time_2d takes the reference's own argument list (src/fdtimes.h:6-7)."""
    import mcmc_eq_b200 as mq
    rng = np.random.default_rng(2)
    g = util.EXAMPLE2_GRID
    nx, nz = util.nxmod_of(g), g["nz"]
    z, vp, vpvs = util.voronoi_model(rng, 7, g["z0"], g["z0"] + (nz - 1) * g["h"], "posterior")
    s = util.rasterise_np(z, vp, vpvs, g["h"], g["z0"], nz, 1)
    hs = np.ascontiguousarray(np.tile(s, (nx, 1)))
    keep = hs.copy()
    t = mq.time_2d(hs, 0.0, 17.0)
    assert np.array_equal(hs, keep)                      # input never modified
    tref, _ = util.oracle_time_2d(s, nx, 17)
    assert (np.abs(t - tref) <= util.eikonal_tol(tref)).all()
    with pytest.raises(mq.MqError) as e:
        mq.time_2d(hs, 3.0, 17.0)
    assert e.value.code == -3


def test_size_independent_properties_at_scale():
    """1024 solves on the Example grid: source node is zero, times grow away from it, and scaling the
    slowness by 2 (an exact operation in binary floating point) scales every time by exactly 2."""
    import mcmc_eq_b200 as mq
    rng = np.random.default_rng(4)
    g = util.EXAMPLE_GRID
    nx, nz = util.nxmod_of(g), g["nz"]
    slows, izs = [], []
    for _ in range(16):
        z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(9, 21)), g["z0"], g["z0"] + (nz - 1) * g["h"], "posterior")
        s = util.rasterise_np(z, vp, vpvs, g["h"], g["z0"], nz, 1)
        slows += [s] * 64
        izs += list(rng.integers(0, nz, 64))
    slows = np.array(slows)
    t1 = mq.eikonal_batch(slows, izs, nx)
    t2 = mq.eikonal_batch(2.0 * slows, izs, nx)
    assert np.array_equal(t2, 2.0 * t1)
    k = np.arange(len(izs))
    assert (t1[k, 0, izs] == 0).all() and (t1 >= 0).all() and np.isfinite(t1).all() and (t1 < 1e4).all()
    # last column is later than the first one everywhere
    assert (t1[:, -1, :] > t1[:, 0, :]).all()
