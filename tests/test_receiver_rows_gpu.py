"""Stations at any depth through every table kernel: borehole and ocean-bottom stations ask for receiver rows far below the
top four rows the example inputs use.  A station in layer k needs rows k and k + 1 of every table (src/misfit.c:91); the
handle stores only those rows (capi.cu) and the misfit kernel reads row r0 and the next one.

Station sets: one station in every layer (n_rows = nz), about a dozen non-contiguous layers, one deep pair (rows nz - 2 and
nz - 1), with hand-placed stations at z = z0, exactly on a grid node (w2 = 0) and in layer nz - 2.  Each case asserts the
eikonal kernel it ran (fused, pipelined with CA = 64 and CA = 128, global-memory fine kernel) and checks sampled chains, the
first and the last always: every stored row against the oracle's table (util.eikonal_tol), per-pick predictions 1e-4 s, class
sums 2e-5 relative, origin times 1e-4 s.  The all-rows set on the pipelined plane is also bit-identical to the fused kernel."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import fwd_helpers as fh
from tests import util

pytestmark = pytest.mark.gpu

EX2 = dict(h=0.5, nx=97, ny=97, nz=61, x0=-24.0, y0=-24.0, z0=-2.0)          # 137 x 61
HALVED = dict(h=0.25, nx=193, ny=193, nz=121, x0=-24.0, y0=-24.0, z0=-2.0)   # 272 x 121
TALL = dict(h=0.25, nx=64, ny=64, nz=700, x0=-8.0, y0=-8.0, z0=-1.0)        # 90 x 700
N_EVENTS = 6


def station_layers(nz, which):
    if which == "all":
        return list(range(nz - 1))
    if which == "dozen":
        return sorted({0, 5, 11, 18, 26, nz // 2, nz - 9, nz - 2})
    if which == "deep":
        return [nz - 2, nz - 2, nz - 2]
    raise ValueError(which)


def make_case(grid, which, seed=11):
    """-> (cfg, picks): stations of the set at their layers (a node, z0 and layer nz - 2 hand-placed), N_EVENTS events."""
    from mcmc_eq_b200 import synth
    cfg = synth.config(**grid)
    h, z0, nz = np.float32(grid["h"]), np.float32(grid["z0"]), grid["nz"]
    layers = station_layers(nz, which)
    geo = synth.geometry(N_EVENTS, len(layers), seed, aperture=min(0.15, 0.4 * (grid["nx"] - 1) * grid["h"] / 240.0))
    rng = np.random.default_rng(seed)
    frac = rng.uniform(0.1, 0.9, len(layers)).astype(np.float32)
    frac[0] = 0.0                                   # layer 0 at z = z0
    if len(layers) > 3:
        frac[2] = 0.0                               # exactly on a node: w2 = 0
    if which == "deep":
        frac[1] = 0.0                               # on node nz - 2
    sz = (z0 + (np.array(layers, np.float32) + frac) * h).astype(np.float32)
    geo["sz"] = sz
    pk = synth.picks_from(geo, rng.uniform(1.0, 30.0, N_EVENTS * 2 * len(layers)).astype(np.float32))
    # the layer the library computes for each station (capi.cu), in the same float arithmetic
    lay = ((sz - z0) / h).astype(np.int32)
    assert np.array_equal(lay, layers), (lay, layers)
    want_rows = sorted(set(layers) | set(l + 1 for l in layers))
    return cfg, pk, want_rows


def _states(cfg, pk, n, seed):
    rng = np.random.default_rng(seed)
    st = fh.random_states(rng, cfg, pk, n, "posterior", 14)
    st[-1] = fh.random_states(rng, cfg, pk, 1, "contrast", 5)[0]     # head waves
    st[min(1, n - 1)] = fh.random_states(rng, cfg, pk, 1, "lvz", 9)[0]
    return st


def run_forward(grid, which, n, sample, seed=12):
    import mcmc_eq_b200 as mq
    cfg, pk, want_rows = make_case(grid, which)
    st = _states(cfg, pk, n, seed)
    smp = mq.Sampler(cfg, pk, n, 0, 1)
    smp.profile(True)
    mf, org = smp.forward_host(fh.fill_models(smp.new_models(), st), 3)
    smp.profile(False)
    kernels = list(smp.profile_kernels())
    out = dict(mf=mf, org=org)
    for c in sample:
        out[f"tp{c}"] = smp.predictions(c)[1]
        for ph in (1, 2):
            rows, idx = smp.rows(c, ph)
            assert list(idx) == want_rows, (list(idx), want_rows)
            out[f"rows{c}_{ph}"] = rows
    smp.close()
    return cfg, pk, st, out, kernels


def _oracle_sparse(cfg, pk, s, rows, depths):
    """Oracle forward with tables that hold only the source depths the picks read (the others stay zero, never read)."""
    L = util.oracle()
    g = fh.fm_grid(cfg)
    nz, nxmod = cfg.grid.nz, L.fm_nxmod(C.byref(g))
    tabs = []
    for ps in (1, 2):
        slow = np.zeros(nz, np.float32)
        L.fm_rasterise(C.byref(g), len(s["z"]), util.ptr(util.f32(s["z"])), util.ptr(util.f32(s["vp"])),
                       util.ptr(util.f32(s["vpvs"])), ps, util.ptr(slow))
        t = np.zeros((max(rows) + 1, nz, nxmod), np.float32)
        for iz in depths:
            field, rc = util.oracle_time_2d(slow, nxmod, iz)
            assert rc == 0
            t[rows, iz, :] = field.T[rows]
        tabs.append(t)
    p = fh.fm_picks(pk)
    mf, origin = np.zeros(8, np.float32), np.zeros(pk.n_events, np.float32)
    resid, tpred = np.zeros(pk.n_picks, np.float32), np.zeros(pk.n_picks, np.float32)
    rc = L.fm_misfit(C.byref(g), C.byref(p), util.ptr(util.f32(s["eq"])), util.ptr(util.f32(s["pres"])), util.ptr(util.f32(s["sres"])),
                     util.ptr(tabs[0]), util.ptr(tabs[1]), 1, len(s["z"]), util.ptr(util.f32(s["z"])), util.ptr(util.f32(s["vp"])),
                     util.ptr(util.f32(s["vpvs"])), util.ptr(mf), util.ptr(origin), util.ptr(resid), util.ptr(tpred))
    assert rc == 0
    return mf, origin, tpred, tabs


def _stored_rows(pk, cfg):
    lay = ((pk.z - np.float32(cfg.grid.z0)) / np.float32(cfg.grid.h)).astype(np.int32)
    return sorted(set(lay) | set(lay + 1))


def check(cfg, pk, st, out, sample, sparse=False):
    rows = _stored_rows(pk, cfg)
    for c in sample:
        s = st[c]
        if sparse:
            iz1 = ((s["eq"][:, 2] - np.float32(cfg.grid.z0)) / np.float32(cfg.grid.h)).astype(np.int32)
            depths = sorted(set(iz1) | set(iz1 + 1))
            rmf, rorg, rtp, tabs = _oracle_sparse(cfg, pk, s, rows, depths)
        else:
            depths = slice(None)
            rmf, rorg, _rres, rtp, tabs = fh.oracle_forward(cfg, pk, s["z"], s["vp"], s["vpvs"], s["eq"], s["pres"], s["sres"], True)
        for ph in (1, 2):
            ref = tabs[ph - 1][rows][:, depths, :]
            err = np.abs(out[f"rows{c}_{ph}"][:, depths, :] - ref)
            assert (err <= util.eikonal_tol(ref)).all(), (c, ph, float(err.max()))
        tp = out[f"tp{c}"]
        assert np.abs(tp - rtp).max() <= 1e-4, (c, float(np.abs(tp - rtp).max()))
        assert np.allclose(out["mf"][c], rmf, rtol=2e-5, atol=1e-6), (c, out["mf"][c], rmf)
        assert np.abs(out["org"][c] - rorg).max() <= 1e-4


@pytest.mark.parametrize("which", ["all", "dozen", "deep"])
def test_fused_kernel_rows_anywhere(which):
    n = 8
    sample = [0, 1, 5, n - 1]
    cfg, pk, st, out, kernels = run_forward(EX2, which, n, sample)
    assert kernels == ["eik_fast_kernel"]
    n_rows = out["rows0_1"].shape[0]
    assert {"all": n_rows == EX2["nz"], "dozen": 9 < n_rows < 25, "deep": n_rows == 2}[which]
    check(cfg, pk, st, out, sample)


PIPE_SCRIPT = ("import sys, numpy as np; sys.path.insert(0, %r); from tests.test_receiver_rows_gpu import run_forward, EX2; "
               "cfg, pk, st, out, k = run_forward(EX2, 'all', int(sys.argv[2]), [0, 233, int(sys.argv[2]) - 1]); "
               "out['kernel'] = np.array(k[0]); np.savez(sys.argv[1], **out)")


@pytest.mark.parametrize("which", ["all", "dozen", "deep"])
def test_pipelined_kernel_rows_anywhere(which, tmp_path):
    """eik_pipe_kernel with CA = 64 (its march emits rows from tensor memory): 480 chains x 2 phases x 61 depths is work for
    every warp of the launch (148 x 12 warp tasks)."""
    n = 480
    sample = [0, 233, n - 1]
    cfg, pk, st, out, kernels = run_forward(EX2, which, n, sample)
    assert kernels == ["eik_pipe_kernel"]
    check(cfg, pk, st, out, sample)
    if which == "all":
        path = str(tmp_path / "fused.npz")
        r = subprocess.run([sys.executable, "-c", PIPE_SCRIPT % util.ROOT, path, str(n)], capture_output=True, text=True,
                           env=dict(os.environ, MCMCEQ_EIKONAL_PIPE="0"), timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        fused = dict(np.load(path))
        assert str(fused.pop("kernel")) == "eik_fast_kernel"
        for k in fused:
            assert np.array_equal(fused[k].view(np.uint32), out[k].view(np.uint32)), (k, int((fused[k] != out[k]).sum()))


@pytest.mark.parametrize("which", ["dozen", "deep"])
def test_deep_pipelined_kernel_rows_anywhere(which):
    """eik_pipe_kernel with CA = 128 on the halved Example2 plane (272 x 121)."""
    n = 170
    sample = [0, n - 1]
    cfg, pk, st, out, kernels = run_forward(HALVED, which, n, sample)
    assert kernels == ["eik_pipe_kernel"]
    check(cfg, pk, st, out, sample)


@pytest.mark.parametrize("which", ["dozen", "deep"])
def test_fine_kernel_rows_anywhere(which):
    """eik_fine_kernel (slices in global memory) on a 90 x 700 plane; the oracle's tables hold the depths the picks read."""
    n = 2
    sample = [0, 1]
    cfg, pk, st, out, kernels = run_forward(TALL, which, n, sample)
    assert kernels == ["eik_fine_kernel"]
    check(cfg, pk, st, out, sample, sparse=True)


# ---- refusals ------------------------------------------------------------------------------------------------------------

def _create(cfg, pk):
    import mcmc_eq_b200 as mq
    L = mq.lib()
    h = C.c_void_p()
    before = L.mq_launch_count()
    rc = L.mq_create(C.byref(cfg), C.byref(pk.view), 1, 0, 1, C.byref(h))
    if rc == 0:
        L.mq_destroy(h)
    return rc, L.mq_launch_count() - before, L.mq_last_error().decode()


def test_station_sets_the_handle_refuses():
    """A pick whose receiver rows do not fit the packed record (row index 256 or more: a set of over 257 rows) and a
    station in the last layer (the reference reads ttt[layer + 1] unchecked) are refused with MQ_ERR_ARG, no table built."""
    from mcmc_eq_b200 import synth
    MQ_ERR_ARG = -1
    grid = dict(h=0.5, nx=20, ny=20, nz=300, x0=-5.0, y0=-5.0, z0=0.0)
    cfg = synth.config(**grid)
    h = np.float32(0.5)

    def picks(layers):
        geo = synth.geometry(2, len(layers), 3, aperture=0.02)
        geo["sz"] = (np.array(layers, np.float32) + np.float32(0.5)) * h
        return synth.picks_from(geo)

    rc, launches, msg = _create(cfg, picks(list(range(0, 299))))          # 300 rows
    assert rc == MQ_ERR_ARG and launches == 0 and "packed record" in msg, (rc, msg)
    rc, launches, msg = _create(cfg, picks(list(range(0, 256)) + [258]))  # rows 0..256, 258, 259: index 257 for layer 258
    assert rc == MQ_ERR_ARG and launches == 0 and "packed record" in msg, (rc, msg)
    rc, _l, msg = _create(cfg, picks(list(range(0, 256))))               # rows 0..256: the last pick's row index is 255
    assert rc == 0, msg
    rc, launches, msg = _create(cfg, picks([0, 7, 299]))                  # a station in layer nz - 1
    assert rc == MQ_ERR_ARG and launches == 0 and "outside the depth grid" in msg, (rc, msg)
