"""Oracle-side forward model for the tests: tables + misfit of a chain state."""
from __future__ import annotations

import ctypes as C

import numpy as np

from tests import util
from tests.util import FmGrid, FmPicks, f32, ptr, ip


def fm_grid(cfg) -> FmGrid:
    g = cfg.grid
    return FmGrid(g.h, g.nx, g.ny, g.nz, g.x0, g.y0, g.z0)


def fm_picks(pk) -> FmPicks:
    return FmPicks(pk.n_events, pk.n_picks, ptr(pk.ev_off, ip), ptr(pk.n_p, ip), ptr(pk.st_id, ip), ptr(pk.cls, ip),
                   ptr(pk.x), ptr(pk.y), ptr(pk.z), ptr(pk.t))


def oracle_forward(cfg, pk, z, vp, vpvs, eq, pres, sres, want_tables=False):
    """(mf[8], origin[ne], resid[np], tpred[np]) of one chain state through the CPU oracle."""
    L = util.oracle()
    g = fm_grid(cfg)
    nz = cfg.grid.nz
    nxmod = L.fm_nxmod(C.byref(g))
    z, vp, vpvs = f32(z), f32(vp), f32(vpvs)
    dim = len(z)
    tabs = []
    for ps in (1, 2):
        slow = np.zeros(nz, np.float32)
        (L.fm_rasterise_tria if cfg.tria == 1 else L.fm_rasterise)(C.byref(g), dim, ptr(z), ptr(vp), ptr(vpvs), ps, ptr(slow))
        t = np.zeros((nz, nz, nxmod), np.float32)
        rc = L.fm_build_table(C.byref(g), ptr(slow), ptr(t))
        assert rc == 0
        tabs.append(t)
    p = fm_picks(pk)
    eq, pres, sres = f32(eq), f32(pres), f32(sres)
    mf = np.zeros(8, np.float32)
    origin = np.zeros(pk.n_events, np.float32)
    resid = np.zeros(pk.n_picks, np.float32)
    tpred = np.zeros(pk.n_picks, np.float32)
    rc = L.fm_misfit(C.byref(g), C.byref(p), ptr(eq), ptr(pres), ptr(sres), ptr(tabs[0]), ptr(tabs[1]), cfg.eikonal, dim,
                     ptr(z), ptr(vp), ptr(vpvs), ptr(mf), ptr(origin), ptr(resid), ptr(tpred))
    assert rc == 0, rc
    if want_tables:
        return mf, origin, resid, tpred, tabs
    return mf, origin, resid, tpred


def random_states(rng, cfg, pk, n, kind="posterior", max_layers=20):
    """n random chain states (dict of arrays) inside the prior box of cfg."""
    g = cfg.grid
    zmin, zmax = g.z0, g.z0 + (g.nz - 1) * g.h
    xmin, xmax = g.x0, g.x0 + (g.nx - 1) * g.h
    ymin, ymax = g.y0, g.y0 + (g.ny - 1) * g.h
    out = []
    for _ in range(n):
        nl = int(rng.integers(1, max_layers + 1))
        z, vp, vpvs = util.voronoi_model(rng, nl, zmin, zmax, kind)
        cx, cy = 0.5 * (xmin + xmax), 0.5 * (ymin + ymax)
        eq = np.stack([rng.uniform(cx - 0.25 * (xmax - xmin), cx + 0.25 * (xmax - xmin), pk.n_events),
                       rng.uniform(cy - 0.25 * (ymax - ymin), cy + 0.25 * (ymax - ymin), pk.n_events),
                       rng.uniform(max(zmin, 0.0), 0.8 * zmax, pk.n_events)], axis=1).astype(np.float32)
        pres = rng.normal(0, 0.2, pk.n_stations).astype(np.float32)
        sres = rng.normal(0, 0.3, pk.n_stations).astype(np.float32)
        noise = rng.uniform(0.05, 1.0, 8).astype(np.float32)
        out.append(dict(z=z, vp=vp, vpvs=vpvs, eq=eq, pres=pres, sres=sres, noise=noise))
    return out


def tria_states(rng, cfg, pk, n, max_layers=12):
    """Random chain states of the linear-gradient parameterisation (config line 29 = 1): nuclei 0 and 1 sit at the top
    and the bottom of the model (src/mcmc_eq.c:577-588), velocities increase with depth plus scatter."""
    g = cfg.grid
    zmin, zmax = g.z0, g.z0 + (g.nz - 1) * g.h
    out = random_states(rng, cfg, pk, n, "posterior", max_layers)
    for s in out:
        nl = len(s["z"]) + 2
        z = np.concatenate([[zmin, zmax], s["z"]]).astype(np.float32)
        vp = (4.5 + 0.04 * (z - zmin) + rng.normal(0, 0.25, nl)).astype(np.float32)
        vpvs = (1.73 + rng.normal(0, 0.05, nl)).astype(np.float32)
        s.update(z=z, vp=vp, vpvs=vpvs)
    return out


def fill_models(m, states):
    for c, s in enumerate(states):
        d = len(s["z"])
        m.dim[c] = d
        m.z[c, :d], m.vp[c, :d], m.vpvs[c, :d] = s["z"], s["vp"], s["vpvs"]
        m.eq[c], m.pres[c], m.sres[c], m.noise[c] = s["eq"], s["pres"], s["sres"], s["noise"]
    return m
