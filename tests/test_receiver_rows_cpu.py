"""Receiver rows anywhere in the plane, on the host builds of the warp-synchronous solver (csrc/eik_fast.cuh).

The example inputs only ever ask for rows 0..3 (stations at the surface), but a borehole or ocean-bottom network asks for
rows at any depth: more than the eight rows a lane keeps in registers during the march (the rest come from rows[]), rows
inside a deep source's homogeneous seed box or refined-init region (copied from the window up to xbox_end, or written
lazily in the global-memory variant), and rows that a homogeneous model fills in closed form.  Every variant must give the
receiver rows of the generic core's full field bit for bit, for every source depth."""
import ctypes as C

import numpy as np
import pytest

from tests import util
from tests.util import ptr, fp

IP = C.POINTER(C.c_int)
KINDS = ("posterior", "contrast", "lvz", "gradient")


@pytest.fixture(scope="module")
def emu():
    from mcmc_eq_b200 import build
    L = C.CDLL(build.build_emu())
    L.emu_time_2d.argtypes = [fp, C.c_int, C.c_int, C.c_int, fp, IP]
    L.emu_fast_time_2d.argtypes = [fp, C.c_int, C.c_int, C.c_int, fp, IP, C.c_int, fp]
    L.emu_set_gm.argtypes = [C.c_int]
    return L


@pytest.fixture(scope="module")
def emu_mt():
    from mcmc_eq_b200 import build
    L = C.CDLL(build.build_emu_mt())
    L.emu_mt_time_2d.argtypes = [fp, C.c_int, C.c_int, IP, fp, IP, C.c_int, fp, IP, C.c_int, C.c_int]
    L.emu_mt_set_fill.argtypes = [C.c_float]
    return L


def _generic(emu, s, nx, iz):
    t = np.zeros((nx, len(s)), np.float32)
    assert emu.emu_time_2d(ptr(s), nx, len(s), iz, ptr(t), None) == 0
    return t


def _rows_only(emu, s, nx, iz, rows, gm):
    """Receiver rows alone (no full field), as the table build asks for them."""
    rows = np.ascontiguousarray(rows, np.int32)
    ro = np.full((len(rows), nx), np.nan, np.float32)
    emu.emu_set_gm(gm)
    try:
        rc = emu.emu_fast_time_2d(ptr(s), nx, len(s), iz, None, rows.ctypes.data_as(IP), len(rows), ptr(ro))
    finally:
        emu.emu_set_gm(0)
    assert rc == 0
    return ro


def row_sets(nz, iz):
    """all rows; ~12 scattered rows (the source row and its neighbours, mid-plane, the last two); the rows below the source."""
    scattered = {iz - 1, iz, iz + 1, 0, 5, nz // 4, nz // 2, nz // 2 + 3, (3 * nz) // 4, nz - 3, nz - 2, nz - 1}
    out = {"all": list(range(nz)), "scattered": sorted(r for r in scattered if 0 <= r < nz)}
    if iz + 1 < nz:
        out["below"] = list(range(iz + 1, nz))
    return out


def _models(rng, nz, h=1.0):
    """Slowness columns of the four model families (P and S alternating) and a single-layer model (homogeneous: the
    solver's closed-form `whole` branch)."""
    out = []
    for k, kind in enumerate(KINDS):
        z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(2, 16)), 0.0, (nz - 1) * h, kind)
        out.append((kind, util.rasterise_np(z, vp, vpvs, h, 0.0, nz, 1 + k % 2)))
    out.append(("single", np.full(nz, np.float32(h / 5.8), np.float32)))
    return out


def _bits_equal(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


PLANES = [(136, 61), (282, 62), (101, 37), (272, 121)]


@pytest.mark.parametrize("nx,nz", PLANES)
def test_single_lane_rows_anywhere(emu, nx, nz):
    """The one-lane build in its three slice layouts (shared memory, global memory as eik_fine_kernel uses it, lock-step
    columns), receiver rows only, against the generic core's field."""
    rng = np.random.default_rng(1000 + nx + nz)
    for kind, s in _models(rng, nz):
        step = 1 if nz <= 62 else 2
        for iz in sorted(set(range(0, nz, step)) | {nz - 2, nz - 1}):
            t = _generic(emu, s, nx, iz)
            for name, rows in row_sets(nz, iz).items():
                want = t[:, rows].T
                for gm in (0, 1, 2):
                    got = _rows_only(emu, s, nx, iz, rows, gm)
                    assert _bits_equal(got, want), (nx, nz, kind, iz, name, gm, float(np.nanmax(np.abs(got - want))))


@pytest.mark.parametrize("nx,nz", PLANES)
@pytest.mark.parametrize("mode,split", [(0, 0), (0, 1), (1, 0), (1, 1), (2, 0), (2, 1)])
def test_a_warp_of_lanes_rows_anywhere(emu, emu_mt, nx, nz, mode, split):
    """A warp of host threads, one model per lane (all families and the single-layer model side by side), every source depth;
    split: the box phase hands its last column to the march (eik_pipe_kernel's data flow).  Scratch starts as NaN."""
    W = emu_mt.emu_mt_lanes()
    rng = np.random.default_rng(2000 + nx + nz + 10 * mode + split)
    models = _models(rng, nz)
    S = np.stack([models[l % len(models)][1] for l in range(W)]).astype(np.float32)
    emu_mt.emu_mt_set_fill(float("nan"))
    step = 1 if nz <= 62 else 3
    for iz in sorted(set(range(0, nz, step)) | {nz - 2, nz - 1}):
        ts = [_generic(emu, S[l], nx, iz) for l in range(W)]
        izs = np.full(W, iz, np.int32)
        for name, rows in row_sets(nz, iz).items():
            r = np.ascontiguousarray(rows, np.int32)
            full = np.full((W, nx, nz), -1, np.float32)
            ro = np.full((W, len(r), nx), np.nan, np.float32)
            st = np.zeros(W, np.int32)
            emu_mt.emu_mt_time_2d(ptr(S), nx, nz, izs.ctypes.data_as(IP), ptr(full), r.ctypes.data_as(IP), len(r), ptr(ro),
                                  st.ctypes.data_as(IP), mode, split)
            for l in range(W):
                assert st[l] == 0
                want = ts[l][:, rows].T
                assert _bits_equal(ro[l], want), (nx, nz, models[l % len(models)][0], iz, name, l,
                                                  float(np.nanmax(np.abs(ro[l] - want))))
                if not split:
                    assert _bits_equal(full[l], ts[l])
    assert emu_mt.emu_mt_site_mismatches() == 0


def _layered_around(nz, lo, hi, h=1.0):
    """A thick homogeneous layer lo..hi between two others: a source inside it gets a large homogeneous seed box."""
    s = np.full(nz, np.float32(h / 7.9), np.float32)
    s[:lo] = np.float32(h / 4.1)
    s[lo:hi + 1] = np.float32(h / 6.2)
    return s


def test_global_memory_rows_inside_the_seed_box(emu, emu_mt):
    """eik_fine_kernel's layout on a tall plane (90 x 700): with rows only, the homogeneous seed box is filled lazily (outline
    first, receiver rows strictly inside it next), so rows 349 / 350 / 351 around a source at 350 -- and every row of the
    box, in the all-rows set -- come from that path."""
    nx, nz = 90, 700
    W = emu_mt.emu_mt_lanes()
    rng = np.random.default_rng(77)
    models = _models(rng, nz)
    models += [("layer300-400", _layered_around(nz, 300, 400)), ("layer340-362", _layered_around(nz, 340, 362))]
    emu_mt.emu_mt_set_fill(float("nan"))
    depths = [0, 1, 120, 345, 349, 350, 351, 356, 600, nz - 2, nz - 1]
    for kind, s in models:
        for iz in depths:
            t = _generic(emu, s, nx, iz)
            sets = dict(row_sets(nz, iz), box=[349, 350, 351])
            for name, rows in sets.items():
                want = t[:, rows].T
                got = _rows_only(emu, s, nx, iz, rows, 1)
                assert _bits_equal(got, want), (kind, iz, name, float(np.nanmax(np.abs(got - want))))
        # the same through a warp of lanes (slices in global memory, hand-over to the march), depths side by side
        izs = np.array([depths[k % len(depths)] for k in range(3, 3 + W)], np.int32)
        S = np.tile(s, (W, 1)).astype(np.float32)
        rows = np.array([3, 200, 348, 349, 350, 351, 352, 500, nz - 2, nz - 1], np.int32)
        ro = np.full((W, len(rows), nx), np.nan, np.float32)
        st = np.zeros(W, np.int32)
        emu_mt.emu_mt_time_2d(ptr(S), nx, nz, izs.ctypes.data_as(IP), None, rows.ctypes.data_as(IP), len(rows), ptr(ro),
                              st.ctypes.data_as(IP), 1, 1)
        for l in range(W):
            assert st[l] == 0
            want = _generic(emu, s, nx, int(izs[l]))[:, rows].T
            assert _bits_equal(ro[l], want), (kind, int(izs[l]), l)
    assert emu_mt.emu_mt_site_mismatches() == 0
