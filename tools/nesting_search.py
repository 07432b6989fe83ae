#!/usr/bin/env python
"""Search for velocity columns whose head waves nest the eikonal solver's reverse propagation deeply; writes
tests/golden/deep_nesting.npz.

The reference re-times the lines behind a head wave by recursion without a depth limit (src/time_2d.c:1128-1143); the
CUDA solver keeps that recursion in a fixed stack of eik::kMaxReverseDepth frames (csrc/eik_core.cuh).  This tool
measures how deep real and constructed columns nest, with the oracle's counter pl_stats.max_rev_depth, by hill-climbing:

  objective   the worst nesting over all source depths of a column (ties: more source depths at that nesting win);
  mutations   move a nucleus, change a velocity, add or remove a nucleus; a mutant is kept when it does not score lower.

Two searches, fixed seeds, fixed iteration counts (so the file is reproducible):
  admissible     Voronoi and TRIA = 1 models inside the priors of the shipped configs (velocity and vp/vs bounds, layer
                 cap), P and S columns, on the Example (282 x 62), Example2 (137 x 61) and halved Example2 (272 x 121)
                 planes;
  unconstrained  Voronoi columns of any positive velocity (log-uniform 0.05-50 km/s) on the Example plane: can a column
                 nest deeper than the stack at all?

For each climb (search, plane, parameterisation) and each nesting depth from 2 upward that it reached, the worst column
found (most source depths at that nesting) is saved with its plane, its model where it has one, and the oracle's nesting
per source depth.

Usage: python tools/nesting_search.py [--iters-scale F] [--out PATH]   (CPU only, about 4 minutes on 8 cores)
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import util  # noqa: E402

HALVED_GRID = dict(h=0.25, nx=193, ny=193, nz=121, x0=-24.0, y0=-24.0, z0=-2.0)   # Example2 at half spacing


def _priors(name):
    with open(os.path.join(util.GOLDEN, f"inputs_{name}.json")) as f:
        c = json.load(f)
    return dict(vpmin=c["vpmin"], vpmax=c["vpmax"], vpvsmin=c["vpvsmin"], vpvsmax=c["vpvsmax"], max_dim=c["max_dim"])


PLANES = {"example": (util.EXAMPLE_GRID, "example"), "example2": (util.EXAMPLE2_GRID, "example2"),
          "halved": (HALVED_GRID, "example2")}

# (search, plane, tria, seed, iterations)
CLIMBS = [("admissible", "example", 0, 1, 6000), ("admissible", "example", 1, 2, 6000),
          ("admissible", "example2", 0, 3, 6000), ("admissible", "example2", 1, 4, 6000),
          ("admissible", "halved", 0, 5, 1200), ("admissible", "halved", 1, 6, 1200),
          ("unconstrained", "example", 0, 7, 12000), ("unconstrained", "example", 0, 8, 12000)]


def nesting(s, nx):
    """The oracle's nesting of head-wave reverse propagation for every source depth of column s: int[nz]."""
    out = np.zeros(len(s), np.int32)
    for iz in range(len(s)):
        st = util.PlStats()
        _, rc = util.oracle_time_2d(s, nx, iz, C.byref(st))
        assert rc == 0, rc
        out[iz] = st.max_rev_depth
    return out


def rasterise(g, model, ps, tria):
    L = util.oracle()
    fg = util.FmGrid(g["h"], g["nx"], g["ny"], g["nz"], g["x0"], g["y0"], g["z0"])
    z, vp, vpvs = (util.f32(a) for a in model)
    slow = np.zeros(g["nz"], np.float32)
    (L.fm_rasterise_tria if tria else L.fm_rasterise)(C.byref(fg), len(z), util.ptr(z), util.ptr(vp), util.ptr(vpvs), ps,
                                                       util.ptr(slow))
    return slow


class Space:
    """Models of one search: nucleus depths in the plane, velocities and vp/vs in their bounds."""

    def __init__(self, search, plane, tria):
        self.g, pri = PLANES[plane][0], _priors(PLANES[plane][1])
        self.zmin, self.zmax = self.g["z0"], self.g["z0"] + (self.g["nz"] - 1) * self.g["h"]
        self.tria = tria
        self.free = 2 if tria else 0          # TRIA = 1: nuclei 0 and 1 sit at the top and the bottom of the model
        if search == "admissible":
            self.vlo, self.vhi, self.rlo, self.rhi, self.cap = pri["vpmin"], pri["vpmax"], pri["vpvsmin"], pri["vpvsmax"], pri["max_dim"]
            self.phases = (1, 2)
        else:
            self.vlo, self.vhi, self.rlo, self.rhi, self.cap = 0.05, 50.0, 1.0, 1.0, 200
            self.phases = (1,)

    def velocity(self, rng, n=None):
        return np.exp(rng.uniform(np.log(self.vlo), np.log(self.vhi), n))

    def start(self, rng):
        n = int(rng.integers(2, 12))
        z = rng.uniform(self.zmin, self.zmax, n)
        if self.tria:
            z[:2] = self.zmin, self.zmax
        return [z, self.velocity(rng, n), rng.uniform(self.rlo, self.rhi, n)]

    def mutate(self, rng, m):
        z, vp, r = (a.copy() for a in m)
        n, op = len(z), int(rng.integers(4))
        if op == 0 and n > self.free:          # move a nucleus
            i = int(rng.integers(self.free, n))
            z[i] = np.clip(z[i] + rng.normal(0, 0.1 * (self.zmax - self.zmin)), self.zmin, self.zmax)
        elif op == 1:                          # change a velocity (or vp/vs)
            i = int(rng.integers(n))
            if rng.random() < 0.7:
                vp[i] = self.velocity(rng)
            else:
                r[i] = rng.uniform(self.rlo, self.rhi)
        elif op == 2 and n < self.cap:         # add a nucleus
            z, vp, r = np.append(z, rng.uniform(self.zmin, self.zmax)), np.append(vp, self.velocity(rng)), np.append(r, rng.uniform(self.rlo, self.rhi))
        elif op == 3 and n > max(1, self.free + (1 if self.tria else 0)):   # remove one (TRIA keeps its two ends)
            i = int(rng.integers(self.free, n))
            z, vp, r = np.delete(z, i), np.delete(vp, i), np.delete(r, i)
        return [z.astype(np.float32), vp.astype(np.float32), r.astype(np.float32)]

    def columns(self, m):
        return [(ps, rasterise(self.g, m, ps, self.tria)) for ps in self.phases]


def climb(args):
    search, plane, tria, seed, iters = args
    sp = Space(search, plane, tria)
    nx = util.nxmod_of(sp.g)
    rng = np.random.default_rng(seed)
    best = {}                                   # nesting depth -> (sources at it, record)

    def score(m):
        top = (-1, 0)
        for ps, s in sp.columns(m):
            d = nesting(s, nx)
            worst = int(d.max())
            key = (worst, int((d == worst).sum()))
            for k in range(2, worst + 1):       # the column nests exactly k deep at (d == k).sum() source depths
                cnt = int((d == k).sum())
                if cnt and (k not in best or cnt > best[k][0]):
                    best[k] = (cnt, dict(search=search, plane=plane, tria=tria, ps=ps, slow=s, depth=d,
                                         z=m[0], vp=m[1], vpvs=m[2]))
            top = max(top, key)
        return top

    m = sp.start(rng)
    cur = score(m)
    for _ in range(iters):
        m2 = sp.mutate(rng, m)
        sc = score(m2)
        if sc >= cur:
            m, cur = m2, sc
    return search, plane, tria, cur, {k: v[1] for k, v in best.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters-scale", type=float, default=1.0)
    ap.add_argument("--out", default=os.path.join(util.GOLDEN, "deep_nesting.npz"))
    a = ap.parse_args()
    util.oracle()
    jobs = [(s, p, t, seed, max(1, int(n * a.iters_scale))) for s, p, t, seed, n in CLIMBS]
    t0 = time.time()
    with mp.Pool(min(len(jobs), os.cpu_count() or 1)) as pool:
        results = pool.map(climb, jobs)
    worst = {}                                  # (search, plane, tria, depth) -> record with the most sources at that depth
    for search, plane, tria, cur, best in results:
        print(f"{search:13s} {plane:8s} tria={tria}: worst nesting {cur[0]} at {cur[1]} source depths")
        for k, rec in best.items():
            key = (search, plane, tria, k)
            if key not in worst or int((rec["depth"] == k).sum()) > int((worst[key]["depth"] == k).sum()):
                worst[key] = rec
    out, meta = {}, []
    for i, ((search, _, _, k), rec) in enumerate(sorted(worst.items())):
        g = PLANES[rec["plane"]][0]
        meta.append(f"{search}|{k}|{rec['plane']}|{rec['tria']}|{rec['ps']}")
        out[f"slow_{i}"] = util.f32(rec["slow"])
        out[f"depth_{i}"] = rec["depth"].astype(np.int8)
        out[f"plane_{i}"] = np.array([util.nxmod_of(g), g["nz"], g["h"], g["z0"], g["nx"], g["ny"], g["x0"], g["y0"]], np.float64)
        if search == "admissible":
            out[f"z_{i}"], out[f"vp_{i}"], out[f"vpvs_{i}"] = util.f32(rec["z"]), util.f32(rec["vp"]), util.f32(rec["vpvs"])
    out["meta"] = np.array(meta)
    np.savez_compressed(a.out, **out)
    print(f"{len(meta)} columns -> {a.out} ({os.path.getsize(a.out)} bytes, {time.time() - t0:.0f} s)")
    for m in meta:
        print("  ", m)


if __name__ == "__main__":
    main()
