"""The misfit kernel (forward.cu: misfit_kernel) at the edges the example inputs never reach.

- Pick counts: events of 1 .. 513 picks.  Up to 256 picks an event's residuals stay in shared memory (KEEP); a handle with a
  larger event runs every event through the global per-pick scratch.  P-only and S-only events and events with missing
  classes are included.  Both paths against the oracle per pick, per class sum and per origin time; KEEP against the forced
  scratch path (MCMCEQ_MISFIT_SCRATCH=1) bit for bit; the scratch path inside the sampler (single-event proposals write the
  event's sums from it).
- Spacing: non-power-of-two grid spacings take bilinear_depth / bilinear_dist with the division and, where the float
  difference x2 - x1 is not the spacing itself, the per-pick prefactor; the power-of-two instantiation against the general
  one (MCMCEQ_MISFIT_POW2=0) bit for bit; mq_traveltimet against the oracle's lookup bit for bit.
- Geometry: hypocentres at z0, on a depth node, in the last depth cell, under a station, in the last distance cell; a
  station outside the model box (1e30 from distance, not depth).

Each environment switch is read once per process, so those comparisons run in subprocesses (run_case below)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import fwd_helpers as fh
from tests import util

pytestmark = pytest.mark.gpu

EX2 = dict(h=0.5, nx=97, ny=97, nz=61, x0=-24.0, y0=-24.0, z0=-2.0)
SIZES = [1, 2, 31, 32, 33, 64, 255, 256, 257, 300, 513]
N_STATIONS = 520


def _config(**grid):
    from mcmc_eq_b200 import synth
    return synth.config(**grid)


def count_picks(big: bool, seed=5):
    """Events of every size in SIZES (those over 256 only when big): P-only, S-only, mixed, some with classes missing."""
    import mcmc_eq_b200 as mq
    rng = np.random.default_rng(seed)
    r = 20.0 * np.sqrt(rng.uniform(0, 1, N_STATIONS))
    th = rng.uniform(0, 2 * np.pi, N_STATIONS)
    sx, sy = (r * np.cos(th)).astype(np.float32), (r * np.sin(th)).astype(np.float32)
    sz = rng.uniform(-1.9, 0.4, N_STATIONS).astype(np.float32)
    ev_off, n_p, st, cls = [0], [], [], []
    for k, size in enumerate(s for s in SIZES if big or s <= 256):
        mode = k % 4            # 0: mixed, 1: P only, 2: S only (n_p = 0), 3: mixed with classes 1 and 2 missing
        npk = {0: (size + 1) // 2, 1: size, 2: 0, 3: size // 2}[mode]
        nsk = size - npk
        assert npk <= N_STATIONS and nsk <= N_STATIONS
        st += list(rng.choice(N_STATIONS, npk, replace=False)) + list(rng.choice(N_STATIONS, nsk, replace=False))
        cls += list(rng.choice([0, 3] if mode == 3 else [0, 1, 2, 3], size))
        n_p.append(npk)
        ev_off.append(ev_off[-1] + size)
    st = np.array(st, np.int32)
    t = rng.uniform(2.0, 12.0, len(st)).astype(np.float32)
    return mq.Picks(np.array(ev_off), np.array(n_p), st, sx[st], sy[st], sz[st], t, np.array(cls), n_stations=N_STATIONS)


def geometry_picks(cfg):
    """Ten events at the edges of the lookup, 9 stations, one of them outside the model box."""
    import mcmc_eq_b200 as mq
    g = cfg.grid
    h, z0, nz = np.float32(g.h), np.float32(g.z0), g.nz
    nxmod = util.nxmod_of(dict(nx=g.nx, ny=g.ny))
    sx = np.array([0.0, 5.25, -7.5, -23.0, 12.0, -3.0, 8.5, 60.0, 1.0], np.float32)
    sy = np.array([0.0, -4.0, 9.0, -23.0, 3.5, -11.0, 8.5, 60.0, 1.0], np.float32)
    sz = np.array([-1.5, -1.0, -0.25, -1.75, 0.0, -2.0, -0.5, -1.0, float(z0 + 2 * h)], np.float32)
    far = 7
    d_last = (nxmod - 2 + 0.4) * float(h)          # inside the last distance cell from station 3
    e = np.array([
        [1.0, 2.0, z0],                             # z = z0
        [-2.0, 1.5, z0 + 9 * h],                    # exactly on a depth node
        [3.0, -2.0, z0 + (nz - 2) * h + 0.2],       # iz1 = nz - 2 (the last valid depth cell)
        [0.0, 0.0, 6.3],                            # directly under station 0 (dist = 0)
        [5.25, -4.0, z0 + 17 * h],                  # under station 1, on a node
        [-23.0 + d_last / np.sqrt(2), -23.0 + d_last / np.sqrt(2), 4.0],   # last distance cell from station 3
        [2.0, 2.0, 11.1], [-6.0, 4.0, 20.2], [7.0, -8.0, 3.3], [0.5, 0.5, 1.1],
    ], np.float32)
    ev_off, n_p, st = [0], [], []
    for k in range(len(e)):
        stations = [s for s in range(len(sx)) if s != far or k in (6, 7)]   # the far station is picked in events 6 and 7
        st += stations + stations[::2]
        n_p.append(len(stations))
        ev_off.append(len(st))
    st = np.array(st, np.int32)
    rng = np.random.default_rng(9)
    cls = rng.integers(0, 4, len(st))
    cls[ev_off[6]:ev_off[8]] = 0        # the events with out-of-table picks hold class 0 only: the other sums stay finite
    t = rng.uniform(2.0, 12.0, len(st)).astype(np.float32)
    return mq.Picks(np.array(ev_off), np.array(n_p), st, sx[st], sy[st], sz[st], t, cls, n_stations=len(sx)), e


def _states(cfg, pk, n, seed):
    rng = np.random.default_rng(seed)
    st = fh.random_states(rng, cfg, pk, n, "posterior", 12)
    st[1 % n] = fh.random_states(rng, cfg, pk, 1, "contrast", 5)[0]
    return st


def case(name):
    """-> (cfg, picks, states) of a named case; deterministic, so that a subprocess rebuilds the same inputs."""
    if name in ("keep", "scratch"):
        cfg = _config(**EX2)
        pk = count_picks(name == "scratch")
        return cfg, pk, _states(cfg, pk, 6, 31)
    if name in ("example", "example2"):
        import tempfile
        import mcmc_eq_b200 as mq
        from tests import inputs
        d = tempfile.mkdtemp(prefix="mqme_")
        cfgp, pkp = inputs.materialise(name, d)
        cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
        return cfg, pk, _states(cfg, pk, 12, 32)
    raise ValueError(name)


def run_case(name, out_path):
    """Forward of the case's states: sums and origin times without per-pick output, then predictions of every chain, then
    the sums again (the predictions pass re-runs the kernel with per-pick output on)."""
    import mcmc_eq_b200 as mq
    cfg, pk, st = case(name)
    n = len(st)
    smp = mq.Sampler(cfg, pk, n, 0, 1)
    mf, org = smp.forward_host(fh.fill_models(smp.new_models(), st), 3)
    tp = np.stack([smp.predictions(c)[1] for c in range(n)])
    res = np.stack([smp.predictions(c)[0] for c in range(n)])
    mf2, org2 = smp.forward(0)
    smp.close()
    np.savez(out_path, mf=mf, org=org, tp=tp, res=res, mf2=mf2, org2=org2)


SCRIPT = "import sys; sys.path.insert(0, %r); from tests.test_misfit_edges_gpu import run_case; run_case(sys.argv[1], sys.argv[2])"


def _run(tmp_path, name, **env):
    path = str(tmp_path / f"{name}_{'_'.join(env) or 'default'}.npz")
    r = subprocess.run([sys.executable, "-c", SCRIPT % util.ROOT, name, path], env=dict(os.environ, **env), capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return dict(np.load(path))


def _check_oracle(cfg, pk, st, mf, org, tp, chains):
    for c in chains:
        s = st[c]
        rmf, rorg, rres, rtp = fh.oracle_forward(cfg, pk, s["z"], s["vp"], s["vpvs"], s["eq"], s["pres"], s["sres"])
        assert np.abs(tp[c] - rtp).max() <= 1e-4, (c, float(np.abs(tp[c] - rtp).max()))
        assert np.array_equal(np.isinf(mf[c]), np.isinf(rmf)), (c, mf[c], rmf)
        fin = np.isfinite(rmf)
        assert np.allclose(mf[c][fin], rmf[fin], rtol=2e-5, atol=1e-6), (c, mf[c], rmf)
        ok = np.abs(rorg) < 1e20          # events with a 1e30 prediction have origin times of order -1e29
        assert np.array_equal(np.abs(org[c]) < 1e20, ok)
        assert np.abs(org[c][ok] - rorg[ok]).max() <= 1e-4


# ---- pick counts ---------------------------------------------------------------------------------------------------------

def test_events_of_every_size_match_the_oracle(tmp_path):
    """Both handles against the oracle, and the in-shared-memory path bit for bit against the forced scratch path, with and
    without per-pick output."""
    for name in ("keep", "scratch"):
        cfg, pk, st = case(name)
        ev = np.diff(pk.ev_off)
        assert (ev.max() > 256) == (name == "scratch")
        assert (pk.n_p == 0).any() and (pk.n_p == ev).any()
        a = _run(tmp_path, name)
        _check_oracle(cfg, pk, st, a["mf"], a["org"], a["tp"], range(len(st)))
        assert np.array_equal(a["mf"], a["mf2"]) and np.array_equal(a["org"], a["org2"])
        if name == "keep":
            b = _run(tmp_path, name, MCMCEQ_MISFIT_SCRATCH="1")
            for k in a:
                assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), (k, int((a[k] != b[k]).sum()))


def test_scratch_path_in_the_sampler():
    """Every proposal kind on the handle with events over 256 picks: single-event proposals (Q) write the event's sums and
    origin time from the scratch path; the maintained likelihood must equal a fresh forward."""
    import mcmc_eq_b200 as mq
    cfg = _config(**EX2, j_max_start=0, j_max_main=100000)
    pk = count_picks(True)
    smp = mq.Sampler(cfg, pk, 16, 0, 7)
    smp.init_chains()
    smp.step(60, "QVRPBDMN")
    counts, ll, rms = smp.stats()
    assert counts[:, 1:17].reshape(16, 8, 2)[:, 3, 0].sum() > 0        # accepted Q proposals
    m = smp.get_models()
    _mf, origin = smp.forward(3)
    _c, ll2, rms2 = smp.stats()
    assert np.array_equal(ll2, ll), float(np.abs(ll2 - ll).max())
    assert np.array_equal(rms2, rms) and np.array_equal(origin, m.origin)
    smp.close()


# ---- spacing -------------------------------------------------------------------------------------------------------------

def _dxf_differs(cfg, pk, st):
    """How many lookups of a state take the per-pick prefactor (float x2 - x1 != h), by numpy float32."""
    h = np.float32(cfg.grid.h)
    e = st["eq"][np.repeat(np.arange(pk.n_events), np.diff(pk.ev_off))]
    dx, dy = (pk.x - e[:, 0]).astype(np.float32), (pk.y - e[:, 1]).astype(np.float32)
    dist = np.sqrt((dx * dx + dy * dy).astype(np.float32)).astype(np.float32)
    m1 = (dist / h).astype(np.int32)
    return int(((np.float32(m1 + 1) * h - np.float32(m1) * h).astype(np.float32) != h).sum())


@pytest.mark.parametrize("h,z0", [(0.3, -1.1), (0.75, -1.3), (1.5, -2.2)])
def test_non_power_of_two_spacing(h, z0):
    """Per pick against the oracle through both table kernels: the fused one (8 chains) and the pipelined one (600 chains:
    work for every warp of the launch)."""
    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    nz = 50
    cfg = _config(h=h, nx=60, ny=60, nz=nz, x0=-30 * h, y0=-30 * h, z0=z0)
    geo = synth.geometry(8, 20, 41, aperture=0.12 * h, elev=(z0 + 0.01, 0.5))
    pk = synth.picks_from(geo, np.random.default_rng(3).uniform(1, 9, 8 * 40).astype(np.float32))
    for n, kernel in ((8, "eik_fast_kernel"), (600, "eik_pipe_kernel")):
        smp = mq.Sampler(cfg, pk, n, 0, 1)
        st = _states(cfg, pk, n, 50 + n)
        smp.profile(True)
        mf, org = smp.forward_host(fh.fill_models(smp.new_models(), st), 3)
        smp.profile(False)
        assert list(smp.profile_kernels()) == [kernel]
        chains = [0, 1, n // 2, n - 1]
        tp = {c: smp.predictions(c)[1] for c in chains}
        smp.close()
        _check_oracle(cfg, pk, st, mf, org, tp, chains)
        if h == 0.3:      # 0.3 is not exact in binary: the float cell width x2 - x1 differs from h for some cells
            assert sum(_dxf_differs(cfg, pk, st[c]) for c in chains) > 0


def test_power_of_two_instantiation_is_bit_identical_to_the_general_one(tmp_path):
    """The claim at forward.cu (misfit kernel, POW2): with a power-of-two spacing y / h == y * (1/h) and every bilinear
    prefactor is a power of two, so the float path equals the double one bit for bit -- on Example (h = 2) and Example2
    (h = 0.5), every pick, class sum and origin time."""
    for name in ("example2", "example"):
        a = _run(tmp_path, name)
        b = _run(tmp_path, name, MCMCEQ_MISFIT_POW2="0")
        for k in a:
            assert np.array_equal(a[k].view(np.uint32), b[k].view(np.uint32)), (name, k, int((a[k] != b[k]).sum()))


@pytest.mark.parametrize("h,z0", [(0.3, -1.1), (0.75, -1.3), (1.5, -2.2), (0.5, -2.0)])
def test_traveltimet_on_cell_boundaries_and_past_the_table(oracle, h, z0):
    """mq_traveltimet against the oracle's lookup (reference src/interpol.c:43-83) bit for bit: the same float corner products
    and the same double prefactor.  Points on cell boundaries, inside the last valid cell, and past it (the sentinel)."""
    import mcmc_eq_b200 as mq
    g = dict(h=h, nx=40, ny=30, nz=37, x0=0.0, y0=0.0, z0=z0)
    nx = util.nxmod_of(g)
    nz = g["nz"]
    rng = np.random.default_rng(int(h * 100))
    tab = np.cumsum(rng.uniform(0.01, 0.3, (nz, nx)).astype(np.float32), axis=1)
    rows = (C.POINTER(C.c_float) * nz)(*[tab[k].ctypes.data_as(C.POINTER(C.c_float)) for k in range(nz)])
    L = mq.lib()
    L.mq_traveltimet.argtypes = [C.POINTER(C.POINTER(C.c_float)), C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float,
                                 C.c_float, C.POINTER(C.c_float), C.c_int]
    fg = util.FmGrid(h, g["nx"], g["ny"], nz, 0.0, 0.0, z0)
    hf, z0f = np.float32(h), np.float32(z0)
    k_x, k_z = np.arange(nx + 2), np.arange(nz + 2)
    pts = [(np.float32(k) * hf, z0f + np.float32(j) * hf) for k, j in zip(rng.choice(k_x, 150), rng.choice(k_z, 150))]
    pts += [(np.float32(k) * hf, np.float32(rng.uniform(z0, z0 + (nz - 1) * h))) for k in k_x]            # dist = k h
    pts += [(np.float32(rng.uniform(0, (nx - 1) * h)), z0f + np.float32(j) * hf) for j in k_z]            # z = z0 + k h
    last_x, last_z = (nx - 2) * h, (nz - 2) * h
    pts += [(np.float32(last_x + f * h), np.float32(z0 + last_z + u * h)) for f, u in rng.uniform(0, 1, (100, 2))]   # last cell
    pts += [(np.float32(last_x + h + f), np.float32(z0 + u * (nz - 1) * h)) for f, u in rng.uniform(0, 2, (60, 2))]  # past it
    pts += [(np.float32(f * (nx - 1) * h), np.float32(z0 + last_z + h + u)) for f, u in rng.uniform(0, 1, (60, 2))]
    n_sentinel = 0
    for dist, z in pts:
        out = C.c_float(0)
        assert L.mq_traveltimet(rows, g["nx"], g["ny"], nz, h, float(dist), float(z), z0, C.byref(out), 0) == 0
        want = oracle.fm_traveltime(util.ptr(tab), C.byref(fg), float(dist), float(z))
        assert np.float32(out.value).view(np.uint32) == np.float32(want).view(np.uint32), (h, float(dist), float(z), out.value, want)
        n_sentinel += want == np.float32(1e30)
    assert 100 < n_sentinel < len(pts) - 250


# ---- geometry ------------------------------------------------------------------------------------------------------------

def test_hypocentres_at_the_edges_of_the_lookup():
    """Hypocentres at z0, on a depth node, in the last depth cell, under a station and in the last distance cell, plus one
    station outside the model box: per-pick predictions and the pattern of infinite class sums against the oracle."""
    import mcmc_eq_b200 as mq
    cfg = _config(**EX2)
    pk, e = geometry_picks(cfg)
    st = _states(cfg, pk, 3, 61)
    for s in st:
        s["eq"] = e.copy()
    smp = mq.Sampler(cfg, pk, 3, 0, 1)
    mf, org = smp.forward_host(fh.fill_models(smp.new_models(), st), 3)
    tp = {c: smp.predictions(c)[1] for c in range(3)}
    smp.close()
    _check_oracle(cfg, pk, st, mf, org, tp, range(3))
    # what the edges are: the far station's picks (and only those) are out of the table by distance
    h, nxmod = np.float32(cfg.grid.h), util.nxmod_of(dict(nx=cfg.grid.nx, ny=cfg.grid.ny))
    ev = np.repeat(np.arange(pk.n_events), np.diff(pk.ev_off))
    dist = np.sqrt(((pk.x - e[ev, 0]) ** 2 + (pk.y - e[ev, 1]) ** 2).astype(np.float32))
    m1 = (dist / h).astype(np.int32)
    assert (m1 >= nxmod - 1).sum() > 0 and set(ev[m1 >= nxmod - 1]) == {6, 7}
    assert (m1 == nxmod - 2).any() and (dist == 0).any()
    assert np.isinf(mf[0]).any() and np.isfinite(mf[0]).any()
