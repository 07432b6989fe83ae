"""The box phase and the hand-over of the pipelined eikonal kernel on the planes of the grids refined by halving the spacing,
which take its CA = 128 instantiation (88 <= nz <= 126): the warp-synchronous solver with a warp of 8 host threads as its
lanes (tests/emu/host_warp.h) in the benched configuration -- lock-step box-phase columns (Dims::lock_cols) and the hand-over
of the last box-phase column that the tensor-memory march starts from -- must give identical bits to the one-lane generic
core.  The tensor-memory march itself runs on the GPU only (tests/test_pipe_deep_gpu.py compares it with the fused kernel)."""
import ctypes as C

import numpy as np
import pytest

from tests import util
from tests.test_emu_cpu import _run, _three_layers
from tests.util import fp, ptr

# (nxmod, nz, h, z0): Example at h = 1 km (399 x 399 x 123), Example2 at h = 0.25 km (193 x 193 x 121), the deepest plane
# of the instantiation (even nz)
PLANES = {
    "example_half": (util.nxmod_of(dict(nx=399, ny=399)), 123, 1.0, -4.0),
    "example2_half": (util.nxmod_of(dict(nx=193, ny=193)), 121, 0.25, -2.0),
    "nz126": (282, 126, 1.0, -4.0),
}


@pytest.fixture(scope="module")
def emu():
    from mcmc_eq_b200 import build
    L = C.CDLL(build.build_emu())
    L.emu_time_2d.argtypes = [fp, C.c_int, C.c_int, C.c_int, fp, C.POINTER(C.c_int)]
    return L


@pytest.fixture(scope="module")
def emu_mt():
    from mcmc_eq_b200 import build
    L = C.CDLL(build.build_emu_mt())
    ip = C.POINTER(C.c_int)
    L.emu_mt_time_2d.argtypes = [fp, C.c_int, C.c_int, ip, fp, ip, C.c_int, fp, ip, C.c_int, C.c_int]
    L.emu_mt_set_fill.argtypes = [C.c_float]
    return L


@pytest.mark.parametrize("plane", sorted(PLANES))
def test_a_warp_of_lanes_on_a_deep_plane(emu, emu_mt, plane):
    """Seven posterior-like and low-velocity-zone models and the widest box of the three-layer model (a source in the middle
    of a layer at mid depth, see tests/test_emu_cpu.py) in one warp, on a NaN-filled scratch."""
    ip = C.POINTER(C.c_int)
    W = emu_mt.emu_mt_lanes()
    nx, nz, h, z0 = PLANES[plane]
    rng = np.random.default_rng(nz)
    rows = np.array([0, 1, 2, nz - 1], np.int32)
    emu_mt.emu_mt_set_fill(float("nan"))
    S = np.zeros((W, nz), np.float32)
    for l in range(W):
        z, vp, vpvs = util.voronoi_model(rng, int(rng.integers(1, 21)), z0, z0 + (nz - 1) * h, "posterior" if l % 2 else "lvz")
        S[l] = util.rasterise_np(z, vp, vpvs, h, z0, nz, 1 + l % 2)
    mid = (nz - 1) // 2
    S[W - 1] = _three_layers(nz, mid - 11, mid + 11, 0.2219247)
    for iz in (0, 1, 13, 40, mid - 1, mid, mid + 1, 97, nz - 2, nz - 1):
        izs = np.full(W, iz, np.int32)
        full = np.zeros((W, 1), np.float32)
        ro = np.zeros((W, len(rows), nx), np.float32)
        st = np.zeros(W, np.int32)
        emu_mt.emu_mt_time_2d(ptr(S), nx, nz, izs.ctypes.data_as(ip), ptr(full), rows.ctypes.data_as(ip), len(rows), ptr(ro),
                              st.ctypes.data_as(ip), 2, 1)
        for l in range(W):
            t, rc, _ = _run(emu, S[l], nx, iz)
            assert rc == 0 and st[l] == 0, (plane, iz, l, rc, st[l])
            assert np.array_equal(ro[l].view(np.uint32), t[:, rows].T.view(np.uint32)), \
                (plane, iz, l, float(np.abs(ro[l] - t[:, rows].T).max()))
    assert emu_mt.emu_mt_site_mismatches() == 0
