"""Test helpers: ctypes views of the CPU oracle (oracle/liboracle.so), of the compiled
reference (oracle/_ref, when present) and seeded model / geometry generators."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_DIR = os.path.join(ORACLE_DIR, "_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden")

fp = C.POINTER(C.c_float)
ip = C.POINTER(C.c_int)


class PlStats(C.Structure):
    _fields_ = [(n, C.c_long) for n in
                ("col_sweeps", "row_sweeps", "reverse_sweeps", "headwaves", "recursive_init", "nearest_init", "box_init")]


class FmGrid(C.Structure):
    _fields_ = [("h", C.c_float), ("nx", C.c_int), ("ny", C.c_int), ("nz", C.c_int),
                ("x0", C.c_float), ("y0", C.c_float), ("z0", C.c_float)]


class FmPicks(C.Structure):
    _fields_ = [("n_events", C.c_int), ("n_picks", C.c_int), ("ev_off", ip), ("n_p", ip), ("st_id", ip), ("cls", ip),
                ("x", fp), ("y", fp), ("z", fp), ("t", fp)]


_oracle = None
_ref = None


def oracle() -> C.CDLL:
    global _oracle
    if _oracle is None:
        so = os.path.join(ORACLE_DIR, "liboracle.so")
        srcs = [os.path.join(ORACLE_DIR, f) for f in os.listdir(ORACLE_DIR) if f.endswith((".c", ".h"))]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
            subprocess.run(["make", "-C", ORACLE_DIR, "liboracle.so"], check=True, stdout=subprocess.DEVNULL)
        L = C.CDLL(so)
        L.pl_time_2d.argtypes = [fp, fp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.POINTER(PlStats)]
        L.fm_nxmod.argtypes = [C.POINTER(FmGrid)]
        L.fm_find_in_cell.argtypes = [fp, C.c_int, C.c_float]
        L.fm_find_neighbor_cell.argtypes = [fp, C.c_int, C.c_int]
        L.fm_dst.argtypes = [C.c_float] * 4
        L.fm_dst.restype = C.c_float
        L.fm_receiver.argtypes = [C.POINTER(FmGrid), C.c_float, ip, fp, fp]
        L.fm_rasterise.argtypes = [C.POINTER(FmGrid), C.c_int, fp, fp, fp, C.c_int, fp]
        L.fm_rasterise_tria.argtypes = [C.POINTER(FmGrid), C.c_int, fp, fp, fp, C.c_int, fp]
        L.fm_build_table.argtypes = [C.POINTER(FmGrid), fp, fp]
        L.fm_traveltime.argtypes = [fp, C.POINTER(FmGrid), C.c_float, C.c_float]
        L.fm_traveltime.restype = C.c_float
        L.fm_misfit.argtypes = [C.POINTER(FmGrid), C.POINTER(FmPicks), fp, fp, fp, fp, fp, C.c_int, C.c_int, fp, fp, fp,
                                fp, fp, fp, fp]
        L.ch_nexp.argtypes = [C.c_float]
        L.ch_nexp.restype = C.c_float
        L.ch_model_valid.argtypes = [C.c_int, fp, fp, fp, C.c_float, C.c_float, C.c_float, C.c_float]
        L.ch_misfit.argtypes = [fp, fp]
        L.ch_misfit.restype = C.c_double
        L.ch_rms.argtypes = [fp, C.c_int]
        L.ch_rms.restype = C.c_double
        L.ch_alpha.argtypes = [C.c_double] * 3
        L.ch_alpha.restype = C.c_float
        L.ch_logfac_birth.argtypes = [C.c_float] * 10
        L.ch_logfac_birth.restype = C.c_double
        L.ch_logfac_death.argtypes = [C.c_float] * 10
        L.ch_logfac_death.restype = C.c_double
        L.ch_logfac_noise.argtypes = [ip, fp, fp]
        L.ch_logfac_noise.restype = C.c_double
        _oracle = L
    return _oracle


def reflib():
    """The unmodified reference as a shared library (oracle/_ref), or None."""
    global _ref
    if _ref is None:
        so = os.path.join(REF_DIR, "libmcmceq_ref.so")
        if not os.path.exists(so):
            return None
        L = C.CDLL(so)
        L.time_2d.argtypes = [fp, fp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int]
        _ref = L
    return _ref


def golden_eikonal():
    """time_2d fields of the compiled reference for seeded models (tools/make_golden.py): ({"s_i", "t_i"}, meta), where
    meta[i] = [grid, kind, source iz].  The fields are stored in two files to keep each under 1 MB."""
    d = {}
    for part in (1, 2):
        d.update(np.load(os.path.join(GOLDEN, f"eikonal_ref_{part}.npz")))
    return d, [m.split("|") for m in d["meta"]]


def f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def ptr(a, t=fp):
    return a.ctypes.data_as(t)


def oracle_time_2d(s, nx, iz, stats=None):
    """Oracle field for a depth-only medium s[nz], source (0, iz): returns t[nx, nz]."""
    L = oracle()
    s = f32(s)
    nz = s.shape[0]
    hs = np.ascontiguousarray(np.tile(s, (nx, 1)))
    t = np.zeros((nx, nz), np.float32)
    rc = L.pl_time_2d(ptr(hs), ptr(t), nx, nz, 0.0, float(iz), 0.001, stats)
    return t, rc


def ref_time_2d(s, nx, iz):
    L = reflib()
    s = f32(s)
    nz = s.shape[0]
    hs = np.ascontiguousarray(np.tile(s, (nx, 1)))
    t = np.zeros((nx, nz), np.float32)
    rc = L.time_2d(ptr(hs), ptr(t), nx, nz, 0.0, float(iz), 0.001, 0)
    return t, rc


# ---- seeded Voronoi models --------------------------------------------------------------

def voronoi_model(rng, nlayers, zmin, zmax, kind="posterior"):
    """(z, vp, vpvs) of `nlayers` nuclei.  kind: posterior | gradient | lvz | contrast."""
    z = rng.uniform(zmin, zmax, nlayers).astype(np.float32)
    if kind == "posterior":      # SURVEY Appendix C (6)
        vp = 5.0 + 0.03 * (z - zmin) + rng.normal(0, 0.15, nlayers)
        vpvs = rng.choice([1.65, 1.73, 1.8, 1.85], nlayers) + rng.normal(0, 0.02, nlayers)
    elif kind == "gradient":
        vp = np.sort(rng.uniform(2.5, 8.5, nlayers))[np.argsort(np.argsort(z))]
        vpvs = np.full(nlayers, 1.73)
    elif kind == "lvz":
        vp = rng.uniform(2.0, 9.0, nlayers)
        vpvs = rng.uniform(1.5, 2.2, nlayers)
    elif kind == "contrast":     # few layers, large jumps: head waves + reverse propagation
        vp = np.sort(rng.choice([2.0, 3.5, 5.0, 6.5, 8.0, 9.5], nlayers))[np.argsort(np.argsort(z))]
        vp = vp + rng.normal(0, 0.01, nlayers)
        vpvs = np.full(nlayers, 1.8)
    else:
        raise ValueError(kind)
    return z, vp.astype(np.float32), vpvs.astype(np.float32)


def rasterise_np(z, vp, vpvs, h, z0, nz, ps):
    """numpy twin of the Voronoi rasteriser (ties -> highest index), float32 arithmetic."""
    z = f32(z)
    zq = (np.float32(z0) + np.arange(nz, dtype=np.float32) * np.float32(h)).astype(np.float32)
    d = (z[None, :] - zq[:, None]).astype(np.float32)
    d2 = (d * d).astype(np.float32)
    k = d2.shape[1] - 1 - np.argmin(d2[:, ::-1], axis=1)
    v = f32(vp)[k] if ps == 1 else (f32(vp)[k] / f32(vpvs)[k]).astype(np.float32)
    return (np.float32(h) / v).astype(np.float32)


EXAMPLE_GRID = dict(h=2.0, nx=200, ny=200, nz=62, x0=-200.0, y0=-200.0, z0=-4.0)   # Example/config_eqx.dat:1-7
EXAMPLE2_GRID = dict(h=0.5, nx=97, ny=97, nz=61, x0=-24.0, y0=-24.0, z0=-2.0)      # Example2/config_eqx.dat:1-7


def nxmod_of(g):
    return int(np.sqrt(g["nx"] * g["nx"] + g["ny"] * g["ny"]))


def eikonal_tol(t_ref):
    """|dT| <= max(1e-4 s, 2e-6 T): the FP32 restatement bound of SURVEY.md Appendix A.5."""
    return np.maximum(1e-4, 2e-6 * np.abs(t_ref))
