"""The CUDA solver core (csrc/eik_core.cuh) compiled for the HOST: the same FP32, restructured
algorithm the GPU runs, checked against the oracle on CPU.  Tolerance: |dT| <= max(1e-4 s, 2e-6 T)
(SURVEY.md Appendix A.5).  This is a test of the algorithm, not a product path."""
import ctypes as C

import numpy as np
import pytest

from tests import util
from tests.util import ptr, fp


@pytest.fixture(scope="module")
def emu():
    from mcmc_eq_b200 import build
    L = C.CDLL(build.build_emu())
    L.emu_time_2d.argtypes = [fp, C.c_int, C.c_int, C.c_int, fp, C.POINTER(C.c_int)]
    L.emu_fast_time_2d.argtypes = [fp, C.c_int, C.c_int, C.c_int, fp, C.POINTER(C.c_int), C.c_int, fp]
    L.emu_set_gm.argtypes = [C.c_int]
    return L


@pytest.fixture(scope="module")
def emu_mt():
    from mcmc_eq_b200 import build
    L = C.CDLL(build.build_emu_mt())
    ip = C.POINTER(C.c_int)
    L.emu_mt_time_2d.argtypes = [fp, C.c_int, C.c_int, ip, fp, ip, C.c_int, fp, ip, C.c_int, C.c_int]
    L.emu_mt_set_fill.argtypes = [C.c_float]
    return L


def _run(emu, s, nx, iz):
    s = util.f32(s)
    t = np.zeros((nx, len(s)), np.float32)
    cnt = np.zeros(7, np.int32)
    rc = emu.emu_time_2d(ptr(s), nx, len(s), iz, ptr(t), cnt.ctypes.data_as(C.POINTER(C.c_int)))
    return t, rc, cnt


def test_core_matches_golden(emu):
    d, meta = util.golden_eikonal()
    worst = 0.0
    tot = np.zeros(7, np.int64)
    for i, m in enumerate(meta):
        s, tref = d[f"s_{i}"], d[f"t_{i}"]
        t, rc, cnt = _run(emu, s, tref.shape[0], int(m[2]))
        assert rc == 0
        err = np.abs(t - tref)
        assert (err <= util.eikonal_tol(tref)).all(), (m, err.max())
        worst = max(worst, float(err.max()))
        tot += cnt
    assert worst < 1e-4
    assert tot[2] > 0 and tot[3] > 0 and tot[4] > 0 and tot[5] > 0 and tot[6] > 0   # every branch taken


@pytest.mark.parametrize("grid,kind", [(util.EXAMPLE2_GRID, "posterior"), (util.EXAMPLE_GRID, "posterior"),
                                       (util.EXAMPLE_GRID, "contrast"), (util.EXAMPLE2_GRID, "lvz")])
def test_core_matches_oracle_all_depths(emu, oracle, grid, kind):
    rng = np.random.default_rng(abs(hash((grid["nz"], kind))) % 2**32)
    nx, nz = util.nxmod_of(grid), grid["nz"]
    z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(2, 21)), grid["z0"], grid["z0"] + (nz - 1) * grid["h"], kind)
    for ps in (1, 2):
        s = util.rasterise_np(z, vp, vpvs, grid["h"], grid["z0"], nz, ps)
        for iz in range(nz):
            tref, _ = util.oracle_time_2d(s, nx, iz)
            t, rc, _ = _run(emu, s, nx, iz)
            assert rc == 0
            assert (np.abs(t - tref) <= util.eikonal_tol(tref)).all()


def test_core_small_and_degenerate_grids(emu, oracle):
    rng = np.random.default_rng(3)
    for nx, nz in ((2, 2), (2, 9), (9, 2), (3, 3), (11, 5), (12, 23), (40, 8)):
        z, vp, vpvs = util.voronoi_model(rng, 3, 0.0, float(nz - 1), "contrast")
        s = util.rasterise_np(z, vp, vpvs, 1.0, 0.0, nz, 1)
        for iz in range(nz):
            tref, r1 = util.oracle_time_2d(s, nx, iz)
            t, r2, _ = _run(emu, s, nx, iz)
            assert r1 == 0 and r2 == 0
            assert (np.abs(t - tref) <= util.eikonal_tol(tref)).all(), (nx, nz, iz)


def _run_fast(emu, s, nx, iz, rows):
    s = util.f32(s)
    t = np.full((nx, len(s)), -1.0, np.float32)
    rows = np.ascontiguousarray(rows, np.int32)
    ro = np.zeros((len(rows), nx), np.float32)
    rc = emu.emu_fast_time_2d(ptr(s), nx, len(s), iz, ptr(t), rows.ctypes.data_as(C.POINTER(C.c_int)), len(rows), ptr(ro))
    return t, ro, rc


@pytest.mark.parametrize("seed,grid", [(1, None), (2, util.EXAMPLE_GRID), (3, util.EXAMPLE2_GRID)])
def test_fast_path_is_bit_identical_to_generic_core(emu, seed, grid):
    """The shared-memory, in-place / ping-pong solver (eik_fast.cuh) visits the nodes in the same order with the
    same arithmetic as the generic core: identical bits, whole field and receiver rows, every source depth."""
    rng = np.random.default_rng(seed)
    for trial in range(10 if grid is None else 3):
        if grid is None:
            nx, nz, h, z0 = int(rng.integers(2, 200)), int(rng.integers(2, 70)), 2.0, 0.0
        else:
            nx, nz, h, z0 = util.nxmod_of(grid), grid["nz"], grid["h"], grid["z0"]
        kind = ["posterior", "contrast", "lvz", "gradient"][trial % 4]
        z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(1, 21)), z0, z0 + (nz - 1) * h, kind)
        s = util.rasterise_np(z, vp, vpvs, h, z0, nz, 1 + trial % 2)
        rows = sorted({0, min(1, nz - 1), min(2, nz - 1), nz - 1})
        for iz in range(nz):
            t1, rc1, _ = _run(emu, s, nx, iz)
            t2, ro, rc2 = _run_fast(emu, s, nx, iz, rows)
            assert rc1 == rc2 == 0, (nx, nz, iz, rc1, rc2)
            assert np.array_equal(t1.view(np.uint32), t2.view(np.uint32)), (nx, nz, kind, iz)
            assert np.array_equal(ro, t1[:, rows].T)


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("seed,shape", [(21, None), (22, (40, 260)), (23, (12, 90)), (24, (282, 62))])
def test_global_memory_variant_is_bit_identical(emu, seed, shape, mode):
    """The solver as eik_fine_kernel instantiates it (slices in global memory: read-ahead row sweeps, columns of the growing
    box swept by the two-chain loop with the real cells beyond the ends of the range, rows that run along the masked right
    edge) against the generic core: identical bits for every source depth, on planes that are taller than wide (the box
    reaches the right edge long before the top and the bottom), with head waves, low-velocity zones and random models."""
    rng = np.random.default_rng(seed)
    for trial in range(8 if shape is None else 4):
        if shape is None:
            nx, nz = int(rng.integers(2, 120)), int(rng.integers(2, 150))
        else:
            nx, nz = shape
        h, z0 = 1.0, 0.0
        kind = ["posterior", "contrast", "lvz", "gradient"][trial % 4]
        z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(1, 21)), z0, z0 + (nz - 1) * h, kind)
        s = util.rasterise_np(z, vp, vpvs, h, z0, nz, 1 + trial % 2)
        rows = sorted({0, min(1, nz - 1), nz - 1})
        step = 1 if nz <= 100 else 7
        for iz in list(range(0, nz, step)) + [nz - 1]:
            t1, rc1, _ = _run(emu, s, nx, iz)
            emu.emu_set_gm(mode)
            t2, ro, rc2 = _run_fast(emu, s, nx, iz, rows)
            emu.emu_set_gm(0)
            assert rc1 == rc2 == 0, (nx, nz, iz, rc1, rc2)
            assert np.array_equal(t1.view(np.uint32), t2.view(np.uint32)), (nx, nz, kind, iz, float(np.abs(t1 - t2).max()))
            assert np.array_equal(ro, t1[:, rows].T)
            # receiver rows only (the table build): the homogeneous seed box is filled lazily, outline and receiver rows first
            emu.emu_set_gm(mode)
            ro2 = np.zeros((len(rows), nx), np.float32)
            rc3 = emu.emu_fast_time_2d(ptr(util.f32(s)), nx, nz, iz, None, np.ascontiguousarray(rows, np.int32).ctypes.data_as(C.POINTER(C.c_int)),
                                       len(rows), ptr(ro2))
            emu.emu_set_gm(0)
            assert rc3 == 0 and np.array_equal(ro2, t1[:, rows].T), (nx, nz, kind, iz)


def _three_layers(nz, lo, hi, s_top=0.2491149, s_mid=0.2100524, s_bot=0.1263643):
    s = np.full(nz, s_bot, np.float32)
    s[:lo] = s_top
    s[lo:hi + 1] = s_mid
    return s


@pytest.mark.parametrize("nz", [31, 45, 61, 62, 63])
def test_row_buffer_holds_both_rows_of_the_widest_box(emu, nz):
    """The top and the bottom row of the growing box share one buffer (top from the front, bottom from the back).  Both are
    longest when the seed box failed above and below in the same round of seed_search (a source in the middle of its layer:
    the box is 2.5 nodes wider than half its height) and reaches the top and the bottom of the grid in the same round (source
    at mid depth): nz + 5 nodes for an odd nz.  With nz + 4 the last top-row sweep read the bottom row's newest node
    (2.7 s off at the Example2 grid's nz = 61)."""
    nx = 4 * nz
    mid = (nz - 1) // 2
    for half in (3, 7, 11, 12):
        for iz in (mid - 1, mid, mid + 1):
            if iz - half < 1 or iz + half > nz - 3:
                continue
            s = _three_layers(nz, iz - half, iz + half)
            t1, rc1, _ = _run(emu, s, nx, iz)
            t2, ro, rc2 = _run_fast(emu, s, nx, iz, [0, nz - 1])
            assert rc1 == rc2 == 0
            assert np.array_equal(t1.view(np.uint32), t2.view(np.uint32)), (nz, half, iz, float(np.abs(t1 - t2).max()))
            emu.emu_set_gm(1)
            t3, ro, rc3 = _run_fast(emu, s, nx, iz, [0, nz - 1])
            emu.emu_set_gm(0)
            assert rc3 == 0 and np.array_equal(t1.view(np.uint32), t3.view(np.uint32)), (nz, half, iz, "gm")


@pytest.mark.parametrize("mode,split", [(0, 0), (0, 1), (1, 0), (2, 0), (2, 1)])
def test_a_warp_of_lanes_is_bit_identical_to_the_generic_core(emu, emu_mt, mode, split):
    """The solver with a warp of 8 host threads as its lanes (tests/emu/host_warp.h: the collectives are barriers), one model
    per lane, all modes of the device code: per-lane in-place columns (0), slices in global memory (1: eik_fine_kernel),
    lock-step columns over the UNION of the lanes' ranges with sentinels outside a lane's own range (1, 2: Dims::lock_cols),
    and the hand-over of the last box-phase column (split: what eik_pipe_kernel's tensor-memory march starts from).  What a
    lane computes must not depend on its neighbours: identical bits to the one-lane generic core."""
    ip = C.POINTER(C.c_int)
    W = emu_mt.emu_mt_lanes()
    g = util.EXAMPLE2_GRID
    nx, nz, h, z0 = util.nxmod_of(g), g["nz"], g["h"], g["z0"]
    rng = np.random.default_rng(100 + 10 * mode + split)
    rows = np.array([0, 1, 2, nz - 1], np.int32)
    # the scratch arrays start as garbage (on the GPU: what the previous task left): nothing may depend on it
    emu_mt.emu_mt_set_fill(float("nan") if (split or mode != 1) else 7.25)
    for trial, kind in enumerate(["lvz", "posterior", "contrast"]):
        S = np.zeros((W, nz), np.float32)
        for l in range(W):
            z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(2, 21)), z0, z0 + (nz - 1) * h, kind)
            S[l] = util.rasterise_np(z, vp, vpvs, h, z0, nz, 1 + l % 2)
        if trial == 0:
            S[W - 1] = _three_layers(nz, 19, 41, 0.2219247)     # the widest box (see the row-buffer test), next to other lanes
        ref = {}
        for iz in list(range(0, nz, 3)) + [30, nz - 1]:
            izs = np.full(W, iz, np.int32)
            if trial == 1:
                izs[1] = -1                                      # a lane without a solve (ragged last warp)
            full = np.full((W, nx, nz), -1, np.float32)
            ro = np.zeros((W, len(rows), nx), np.float32)
            st = np.zeros(W, np.int32)
            emu_mt.emu_mt_time_2d(ptr(S), nx, nz, izs.ctypes.data_as(ip), ptr(full), rows.ctypes.data_as(ip), len(rows), ptr(ro),
                                  st.ctypes.data_as(ip), mode, split)
            for l in range(W):
                if izs[l] < 0:
                    continue
                t, rc, _ = _run(emu, S[l], nx, iz)
                assert rc == 0 and st[l] == 0, (kind, iz, l, rc, st[l])
                assert np.array_equal(ro[l].view(np.uint32), t[:, rows].T.view(np.uint32)), (kind, iz, l, float(np.abs(ro[l] - t[:, rows].T).max()))
                if not split:
                    assert np.array_equal(full[l].view(np.uint32), t.view(np.uint32)), (kind, iz, l)
    # every collective was reached by all lanes from the same call site (anything else is undefined on the GPU)
    assert emu_mt.emu_mt_site_mismatches() == 0


def test_a_warp_of_lanes_on_the_example_plane(emu, emu_mt):
    """The benched configuration of the pipelined kernel (lock-step box-phase columns, hand-over to the march) on the Example
    plane (282 x 62, even nz) with eight posterior-like models per warp: identical bits to the one-lane generic core."""
    ip = C.POINTER(C.c_int)
    W = emu_mt.emu_mt_lanes()
    g = util.EXAMPLE_GRID
    nx, nz, h, z0 = util.nxmod_of(g), g["nz"], g["h"], g["z0"]
    rng = np.random.default_rng(7)
    rows = np.array([1, 2], np.int32)
    emu_mt.emu_mt_set_fill(float("nan"))
    S = np.zeros((W, nz), np.float32)
    for l in range(W):
        z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(1, 8)), z0, z0 + (nz - 1) * h, "posterior" if l % 2 else "lvz")
        S[l] = util.rasterise_np(z, vp, vpvs, h, z0, nz, 1 + l % 2)
    for iz in (0, 7, 19, 30, 31, 44, nz - 1):
        izs = np.full(W, iz, np.int32)
        full = np.zeros((W, 1), np.float32)
        ro = np.zeros((W, len(rows), nx), np.float32)
        st = np.zeros(W, np.int32)
        emu_mt.emu_mt_time_2d(ptr(S), nx, nz, izs.ctypes.data_as(ip), ptr(full), rows.ctypes.data_as(ip), len(rows), ptr(ro),
                              st.ctypes.data_as(ip), 2, 1)
        for l in range(W):
            t, rc, _ = _run(emu, S[l], nx, iz)
            assert rc == 0 and st[l] == 0
            assert np.array_equal(ro[l].view(np.uint32), t[:, rows].T.view(np.uint32)), (iz, l, float(np.abs(ro[l] - t[:, rows].T).max()))
    assert emu_mt.emu_mt_site_mismatches() == 0
