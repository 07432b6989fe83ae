"""Hypocentre uncertainty without a GPU: the library exports mq_hypo_*, and hypo.py -- the statement the device is checked
against -- pools per-chain shifted sums into np.cov of the concatenated samples, reads quantiles and the mode off the
histograms by its documented rules, gives np.linalg.eigh's ellipsoid with the documented signs, azimuths and plunges,
and the documented NaN / 0 in every edge case."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from mcmc_eq_b200 import hypo
from tests import util

LIB = os.path.join(util.ROOT, "mcmc_eq_b200", "libmcmceq_b200.so")


def test_library_exports_the_hypo_entry_points():
    assert os.path.exists(LIB), "libmcmceq_b200.so not built (python -m mcmc_eq_b200.build)"
    lib = C.CDLL(LIB)
    for name in ("mq_hypo_begin", "mq_hypo_chains", "mq_hypo_summary"):
        assert hasattr(lib, name), name
    syms = subprocess.run(["nm", "-D", "--defined-only", LIB], capture_output=True, text=True, check=True).stdout.split()
    for name in ("mq_hypo_begin", "mq_hypo_chains", "mq_hypo_summary"):
        assert name in syms, name


def _summary_of(chains, lo=(0.0, 0.0, 0.0), w=1.0, hi=(100.0, 100.0, 100.0)):
    accs = [hypo.accumulate(x) for x in chains]
    acc = hypo.stack(accs)
    allv = np.concatenate(chains, 0)
    lo32, hi32 = np.float32(lo), np.float32(hi)
    hist, outside = hypo.histogram(allv, lo32, hi32, w)
    return hypo.summarise(hist, lo=lo32, bin_km=w, n_bins=hypo.n_bins(lo32, hi32, w), **acc), allv, outside


@pytest.mark.parametrize("offset", [0.0, 200.0])
def test_pooled_covariance_equals_np_cov_of_the_concatenated_samples(offset):
    """A spread of 10 m at up to 230 km; chains of one model, and a chain whose first model (its ref) is 40 km off."""
    rng = np.random.default_rng(7)
    A = np.array([[1.0, 0.3, -0.2, 0.5], [0.0, 0.8, 0.1, 0.0], [0.0, 0.0, 0.5, 0.9], [0.0, 0.0, 0.0, 0.2]]) * 0.01
    chains = []
    for m in (1, 1, 2, 17, 300, 41):
        shift = rng.standard_normal(4) * 0.02
        x = offset + 30.0 + shift + rng.standard_normal((m, 1, 4)) @ A.T
        x = np.concatenate([x, x[:, :, ::-1] + 1.0], 1)              # two events
        chains.append(x.astype(np.float32))
    far = chains[-1].copy()
    far[0] += 40.0
    chains.append(far)
    s, allv, _ = _summary_of(chains, hi=(offset + 100.0,) * 3)
    assert s["n_models"] == len(allv)
    for e in range(2):
        v = allv[:, e, :].astype(np.float64)
        want = np.cov(v.T)
        assert np.allclose(s["mean"][e], v.mean(0), rtol=1e-12, atol=0)
        scale = np.sqrt(np.outer(np.diag(want), np.diag(want)))
        assert (np.abs(s["cov"][e] - want) <= 1e-12 * np.maximum(scale, np.abs(want))).all(), (s["cov"][e], want)
        assert np.array_equal(s["cov"][e], s["cov"][e].T)


def test_accumulate_uses_the_first_model_as_reference():
    x = (200.0 + 0.01 * np.random.default_rng(1).standard_normal((50, 3, 4))).astype(np.float32)
    a = hypo.accumulate(x)
    assert np.array_equal(a["ref"], x[0].T.astype(np.float64)) and a["n_models"] == 50
    d = x.astype(np.float64) - x[0].astype(np.float64)
    assert np.allclose(a["sum"], d.sum(0).T, rtol=0, atol=1e-12)
    assert np.allclose(a["cross"][hypo.PAIRS.index((2, 3))], (d[:, :, 2] * d[:, :, 3]).sum(0), rtol=1e-12, atol=1e-18)


def test_quantiles_of_a_dense_uniform_sample():
    rng = np.random.default_rng(3)
    lo, hi, w = 2.0, 12.0, 0.01
    v = rng.uniform(lo + 1.0, lo + 9.0, 2_000_000).astype(np.float32)
    trace = np.zeros((len(v), 1, 3), np.float32)
    trace[:, 0, :] = v[:, None]
    hist, outside = hypo.histogram(trace, np.float32([lo] * 3), np.float32([hi] * 3), w)
    assert not outside.any()
    nb = hypo.n_bins(np.float32([lo] * 3), np.float32([hi] * 3), w)
    assert nb[0] == int(np.float32(10.0) / np.float32(0.01)) + 1
    q = hypo.quantiles(hist[0, :nb[0]], lo, w)
    assert np.allclose(q, np.quantile(v.astype(np.float64), hypo.PROBS), rtol=0, atol=2 * w)
    # exact on a histogram whose bins hold equal counts: the rule interpolates linearly inside a bin
    flat = np.full(100, 10)
    assert np.allclose(hypo.quantiles(flat, 0.0, 0.5), [50.0 * p for p in hypo.PROBS], rtol=0, atol=1e-12)


def test_histogram_clamps_and_counts_values_outside_the_box():
    lo, hi = np.float32([0.0, 0.0, 0.0]), np.float32([10.0, 10.0, 10.0])
    trace = np.float32([[[-3.0, 10.0, 10.5]], [[0.0, 9.99, 4.0]]])
    hist, outside = hypo.histogram(trace, lo, hi, 1.0)
    assert list(outside[0]) == [1, 0, 1]
    nb = hypo.n_bins(lo, hi, 1.0)
    assert list(nb) == [11, 11, 11]
    x, y, z = hist[0, :11], hist[0, 11:22], hist[0, 22:]
    assert x[0] == 2 and y[9] == 1 and y[10] == 1 and z[10] == 1 and z[4] == 1


def test_mode_takes_the_lowest_of_equal_bins():
    assert hypo.mode([0, 3, 1, 3, 0], 10.0, 2.0) == 10.0 + 2.0 * 1.5
    assert hypo.mode([5], -1.0, 0.5) == -0.75
    assert math.isnan(hypo.mode([0, 0], 0.0, 1.0))


def _rot(ax, ang):
    c, s = math.cos(ang), math.sin(ang)
    i, j = [(1, 2), (0, 2), (0, 1)][ax]
    r = np.eye(3)
    r[i, i], r[i, j], r[j, i], r[j, j] = c, -s, s, c
    return r


@pytest.mark.parametrize("seed", range(6))
def test_ellipsoid_against_eigh(seed):
    rng = np.random.default_rng(seed)
    R = _rot(0, rng.uniform(-3, 3)) @ _rot(1, rng.uniform(-3, 3)) @ _rot(2, rng.uniform(-3, 3))
    lam = np.sort(rng.uniform(0.01, 4.0, 3))[::-1] ** 2 * (1e-4 if seed % 2 else 1.0)
    cov = R @ np.diag(lam) @ R.T
    axes, dirs = hypo.ellipsoid(cov)
    wl, wv = np.linalg.eigh(cov)
    assert np.allclose(axes ** 2, wl[::-1], rtol=0, atol=1e-10 * wl[-1])
    gaps = np.abs(np.diff(wl[::-1]))
    if gaps.min() > 1e-3 * wl[-1]:
        for k in range(3):
            assert np.allclose(dirs[k], hypo.sign_rule(wv[:, 2 - k]), rtol=0, atol=1e-8)
    for k in range(3):
        assert abs(np.linalg.norm(dirs[k]) - 1.0) < 1e-12 and dirs[k][2] >= 0.0
    assert np.allclose(dirs @ dirs.T, np.eye(3), atol=1e-12)


def test_axis_aligned_and_rotated_azimuth_and_plunge():
    axes, dirs = hypo.ellipsoid(np.diag([4.0, 9.0, 1.0]))           # sd 2 along x, 3 along y, 1 along z
    assert np.array_equal(axes, [3.0, 2.0, 1.0])
    assert np.array_equal(dirs, [[0, 1, 0], [1, 0, 0], [0, 0, 1]])
    assert hypo.azimuth_plunge(dirs[0]) == (0.0, 0.0)               # north
    assert hypo.azimuth_plunge(dirs[1]) == (90.0, 0.0)              # east
    assert hypo.azimuth_plunge(dirs[2])[1] == 90.0                  # straight down
    # the sign rule: horizontal axes point to +y, or to +x when they lie on the x axis
    assert np.array_equal(hypo.sign_rule([-1.0, 0.0, 0.0]), [1.0, 0.0, 0.0])
    assert np.array_equal(hypo.sign_rule([0.5, -0.5, 0.0]), [-0.5, 0.5, 0.0])
    assert np.array_equal(hypo.sign_rule([0.5, 0.5, -0.1]), [-0.5, -0.5, 0.1])
    # the long axis rotated 30 degrees clockwise from +y and dipping 20 degrees down
    az, pl = math.radians(30.0), math.radians(20.0)
    u = np.array([math.sin(az) * math.cos(pl), math.cos(az) * math.cos(pl), math.sin(pl)])
    cov = 9.0 * np.outer(u, u) + 0.25 * np.eye(3)
    axes, dirs = hypo.ellipsoid(cov)
    a0, p0 = hypo.azimuth_plunge(dirs[0])
    assert abs(a0 - 30.0) < 1e-9 and abs(p0 - 20.0) < 1e-9 and abs(axes[0] - math.sqrt(9.25)) < 1e-12
    # an axis in the south-west quadrant, pointing up before the sign rule: azimuth 225 - 180 = 45 after it
    v = hypo.sign_rule([-math.sqrt(0.5) * 0.8, -math.sqrt(0.5) * 0.8, -0.6])
    a, p = hypo.azimuth_plunge(v)
    assert abs(a - 45.0) < 1e-9 and abs(p - math.degrees(math.asin(0.6))) < 1e-9
    assert hypo.azimuth_plunge([-1e-300, 1.0, 0.0])[0] < 360.0


def test_edge_cases():
    lo, hi = np.float32([0.0] * 3), np.float32([10.0] * 3)
    nb = hypo.n_bins(lo, hi, 1.0)
    empty = dict(ref=np.zeros((2, 4, 1)), sum=np.zeros((2, 4, 1)), cross=np.zeros((2, 10, 1)), n_models=np.zeros(2, np.int64))
    s = hypo.summarise(np.zeros((1, int(nb.sum())), np.int32), lo=lo, bin_km=1.0, n_bins=nb, **empty)     # N = 0
    assert s["n_models"] == 0
    for k in ("mean", "cov", "quant", "mode", "axes", "axis_dir"):
        assert np.isnan(s[k]).all(), k
    one = [np.float32([[[1.0, 2.0, 3.0, 4.0]]])]                     # N = 1: a mean and quantiles, no covariance
    s, _, _ = _summary_of(one, hi=(10.0,) * 3)
    assert s["n_models"] == 1 and np.array_equal(s["mean"][0], [1.0, 2.0, 3.0, 4.0])
    assert np.isnan(s["cov"]).all() and np.isnan(s["axes"]).all() and np.isnan(s["axis_dir"]).all()
    assert np.isfinite(s["quant"]).all() and np.array_equal(s["mode"][0], [1.5, 2.5, 3.5])
    # z never moves (fixed by the pick file) in chains that disagree on x: variance and covariances exactly 0
    rng = np.random.default_rng(5)
    chains = []
    for m in (5, 9, 1, 30):
        x = np.empty((m, 1, 4), np.float32)
        x[:, 0, 0] = 3.0 + rng.standard_normal() + rng.standard_normal(m)
        x[:, 0, 1] = 4.0 + rng.standard_normal(m)
        x[:, 0, 2] = np.float32(7.3)
        x[:, 0, 3] = rng.standard_normal(m)
        chains.append(x)
    s, _, _ = _summary_of(chains, hi=(10.0,) * 3, w=0.1)
    c = s["cov"][0]
    assert (c[2, :] == 0.0).all() and (c[:, 2] == 0.0).all() and c[0, 0] > 0
    assert s["mean"][0, 2] == np.float32(7.3)
    assert abs(s["quant"][0, 2, 2] - np.float32(7.3)) <= 0.1
    assert s["axes"][0, 2] == 0.0 and np.array_equal(s["axis_dir"][0, 2], [0.0, 0.0, 1.0])
