"""The most deeply nesting columns of tests/golden/deep_nesting.npz (head-wave reverse propagation, see
tests/test_reverse_depth_cpu.py) through every eikonal kernel: every node of every solve within level 1 of the oracle,
|dT| <= max(1e-4 s, 2e-6 T), and status 0.  The warp kernels (fused, pipelined) are bit-identical to each other; the
generic kernel rounds its square roots correctly where they take the hardware approximation (eik_fast.cuh), so it is
held to the oracle's tolerance, not to their bits.

  generic    mq_eikonal_batch with MCMCEQ_EIKONAL=generic, in a subprocess (the switch is read once per process);
  fused      mq_eikonal_batch on the fixture's own planes (282 x 62, 137 x 61, 272 x 121: all fit a shared-memory slice,
             and a batch never takes the pipelined kernel, so eik_fast_kernel runs);
  fine       mq_eikonal_batch on the 90 x 700 plane of test_receiver_rows_gpu.py, columns resampled to it (no shared-memory
             slice holds that plane: eik_fine_kernel runs);
  pipelined  table rebuilds of a sampler whose chains carry the fixture's admissible models, enough of them for every warp
             of the launch (mq_profile_kernels says eik_pipe_kernel ran): CA = 64 on the Example and Example2 planes, CA =
             128 on the halved plane."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import util
from tests.test_receiver_rows_gpu import TALL, make_case

pytestmark = pytest.mark.gpu

TALL_NX = util.nxmod_of(TALL)
TALL_DEPTHS = list(range(0, TALL["nz"], 5)) + [TALL["nz"] - 1]
PLANES = {"example": util.EXAMPLE_GRID, "example2": util.EXAMPLE2_GRID,
          "halved": dict(h=0.25, nx=193, ny=193, nz=121, x0=-24.0, y0=-24.0, z0=-2.0)}
PIPE_CHAINS = {"example": 1230, "example2": 480, "halved": 170}


def _fixture():
    d = np.load(os.path.join(util.GOLDEN, "deep_nesting.npz"))
    out = []
    for i, m in enumerate(d["meta"]):
        search, k, plane, tria, ps = m.split("|")
        rec = dict(search=search, k=int(k), plane=plane, tria=int(tria), ps=int(ps), slow=d[f"slow_{i}"], depth=d[f"depth_{i}"])
        if f"z_{i}" in d:
            rec.update(z=d[f"z_{i}"], vp=d[f"vp_{i}"], vpvs=d[f"vpvs_{i}"])
        out.append(rec)
    return out


def _tall(rec):
    """The column stretched over the 700 depth nodes of the tall plane, same velocities."""
    g = PLANES[rec["plane"]]
    v = np.float32(g["h"]) / rec["slow"]
    idx = (np.arange(TALL["nz"]) * len(v)) // TALL["nz"]
    return (np.float32(TALL["h"]) / v[idx]).astype(np.float32)


def batches():
    """{name: (slow[n, nz], iz[n], nxmod)}: every source depth of the fixture's columns on each plane, and the resampled
    columns on the tall plane."""
    fx = _fixture()
    out = {}
    for plane, g in PLANES.items():
        cols = [r["slow"] for r in fx if r["plane"] == plane]
        if cols:
            nz = g["nz"]
            out[plane] = (np.repeat(np.array(cols), nz, axis=0), np.tile(np.arange(nz, dtype=np.int32), len(cols)), util.nxmod_of(g))
    tall = [_tall(r) for r in fx]
    out["tall"] = (np.repeat(np.array(tall), len(TALL_DEPTHS), axis=0), np.tile(np.array(TALL_DEPTHS, np.int32), len(tall)), TALL_NX)
    return out


GENERIC_SCRIPT = ("import sys, numpy as np; sys.path.insert(0, %r); import mcmc_eq_b200 as mq; "
                  "from tests.test_reverse_depth_gpu import batches; out = {}\n"
                  "for name, (s, iz, nx) in batches().items():\n"
                  "    t, st, rc = mq.eikonal_batch(s, iz, nx, return_status=True); out[name] = t; out[name + '_st'] = st; out[name + '_rc'] = np.array(rc)\n"
                  "np.savez(sys.argv[1], **out)")


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    """{name: (fields from the default kernels, fields from the generic kernel)} for every batch."""
    import mcmc_eq_b200 as mq
    path = str(tmp_path_factory.mktemp("revdepth") / "generic.npz")
    r = subprocess.run([sys.executable, "-c", GENERIC_SCRIPT % util.ROOT, path], capture_output=True, text=True,
                       env=dict(os.environ, MCMCEQ_EIKONAL="generic"), timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    gen = dict(np.load(path))
    out = {}
    for name, (s, iz, nx) in batches().items():
        t, st, rc = mq.eikonal_batch(s, iz, nx, return_status=True)
        assert rc == 0 and (st == 0).all(), (name, rc, np.flatnonzero(st)[:8])
        assert int(gen[name + "_rc"]) == 0 and (gen[name + "_st"] == 0).all(), name
        out[name] = (t, gen[name])
    return out


def _against_oracle(s, iz, nx, fields):
    """fields: {kernel: t[n, nx, nz]} -> ({kernel: worst |dT|}, deepest nesting of the oracle)"""
    import ctypes as C
    worst, deepest = {k: 0.0 for k in fields}, 0
    for k in range(len(iz)):
        st = util.PlStats()
        tref, rc = util.oracle_time_2d(s[k], nx, int(iz[k]), C.byref(st))
        assert rc == 0
        tol = util.eikonal_tol(tref)
        for name, t in fields.items():
            err = np.abs(t[k] - tref)
            assert (err <= tol).all(), (name, k, int(iz[k]), float(err.max()))
            worst[name] = max(worst[name], float(err.max()))
        deepest = max(deepest, int(st.max_rev_depth))
    return worst, deepest


@pytest.mark.parametrize("name", ["example", "example2", "halved", "tall"])
def test_fused_fine_and_generic_kernels(runs, name):
    """Fused kernel (fixture planes) or fine kernel (tall plane), and the generic kernel, against the oracle."""
    if name not in runs:
        pytest.skip(f"no fixture column on the {name} plane")
    s, iz, nx = batches()[name]
    t, t_gen = runs[name]
    worst, deepest = _against_oracle(s, iz, nx, {"fine" if name == "tall" else "fused": t, "generic": t_gen})
    print(f"\n{name}: {len(iz)} solves, worst |dT| {worst} s, deepest nesting {deepest}")
    if name != "tall":
        assert deepest >= 2


@pytest.mark.parametrize("plane", ["example", "example2", "halved"])
def test_pipelined_kernel(runs, plane):
    """Table rebuilds on eik_pipe_kernel with the fixture's Voronoi and TRIA = 1 models of the plane replicated over the
    chains: the receiver rows the handle stores are the bits of the fused kernel's fields for the same columns."""
    import mcmc_eq_b200 as mq
    from tests import fwd_helpers as fh
    grid = PLANES[plane]
    fx = [r for r in _fixture() if r["plane"] == plane and "z" in r]
    if not fx:
        pytest.skip(f"no admissible model on the {plane} plane")
    t_fused = runs[plane][0]
    cols = [r["slow"] for r in _fixture() if r["plane"] == plane]
    nz = grid["nz"]
    n = PIPE_CHAINS[plane]
    checked = 0
    for tria in (0, 1):
        models = [r for r in fx if r["tria"] == tria]
        if not models:
            continue
        cfg, pk, want_rows = make_case(grid, "dozen")
        cfg.tria = tria
        cfg.max_dim = 200                                     # the shipped configs' layer cap, which the search used
        rng = np.random.default_rng(5)
        st = fh.random_states(rng, cfg, pk, n, "posterior", 4)
        for c in range(n):
            r = models[c % len(models)]
            st[c].update(z=r["z"], vp=r["vp"], vpvs=r["vpvs"])
        smp = mq.Sampler(cfg, pk, n, 0, 1)
        try:
            smp.profile(True)
            smp.forward_host(fh.fill_models(smp.new_models(), st), 3)
            smp.profile(False)
            assert list(smp.profile_kernels()) == ["eik_pipe_kernel"], (plane, tria, list(smp.profile_kernels()))
            for c in list(range(len(models))) + [n - 1]:
                r = models[c % len(models)]
                rows, idx = smp.rows(c, r["ps"])
                assert list(idx) == want_rows
                j = next(i for i, s in enumerate(cols) if np.array_equal(s, r["slow"]))
                ref = t_fused[j * nz:(j + 1) * nz][:, :, idx].transpose(2, 0, 1)     # [row, source depth, x]
                assert np.array_equal(rows.view(np.uint32), ref.view(np.uint32)), (plane, tria, c, int((rows != ref).sum()))
                checked += 1
        finally:
            smp.close()
    assert checked > 0
