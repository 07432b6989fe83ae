"""Convergence diagnostics without a GPU: the library exports mq_diag_*, diag.accumulate is the slot and doubling rule
(checked against direct sums of the same trace), and diag.summarise gives R-hat near 1 and the right ESS on synthetic
chains with known autocorrelation, flags chains that disagree, and gives the documented NaN / inf in every edge case."""
import ctypes as C
import os

import numpy as np
import pytest

from mcmc_eq_b200 import diag
from tests import util

LIB = os.path.join(util.ROOT, "mcmc_eq_b200", "libmcmceq_b200.so")


def test_library_exports_the_diag_entry_points():
    assert os.path.exists(LIB), "libmcmceq_b200.so not built (python -m mcmc_eq_b200.build)"
    lib = C.CDLL(LIB)
    for name in ("mq_diag_begin", "mq_diag_chains", "mq_diag_summary"):
        assert hasattr(lib, name), name


def test_quantity_names_follow_the_device_order():
    names = diag.quantity_names(3, 2, 2)
    assert len(names) == 10 + 2 * 3 + 4 * 2 + 2 * 2
    assert names[:3] == ["rms", "dim", "noise[0]"]
    assert names[10:16] == ["vp[0]", "vp[1]", "vp[2]", "vpvs[0]", "vpvs[1]", "vpvs[2]"]
    assert names[16:24] == ["x[0]", "y[0]", "z[0]", "t[0]", "x[1]", "y[1]", "z[1]", "t[1]"]
    assert names[24:] == ["pres[0]", "sres[0]", "pres[1]", "sres[1]"]
    assert len(diag.quantity_names(62, 200, 50)) == 1034 and len(diag.quantity_names(62, 2000, 100)) == 8334


@pytest.mark.parametrize("m", [0, 1, 7, 8, 9, 33, 100, 257, 1000])
def test_accumulate_matches_direct_sums(m):
    K = 8
    rng = np.random.default_rng(m)
    x = 200.0 + 0.01 * rng.standard_normal((m, 3))
    a = diag.accumulate(x, K)
    assert a["n_models"] == m
    k, L = int(a["full_batches"]), int(a["batch_len"])
    if m:
        assert np.array_equal(a["ref"], x[0])
    # the invariant: k full batches of L models, the rest in the open slot k, every later slot empty
    assert k * L <= m < k * L + L and (m < K or K // 2 <= k < K)
    d = x - (x[0] if m else 0.0)
    for b in range(k + 1):
        seg = d[b * L:min((b + 1) * L, m)]
        assert np.allclose(a["sum"][b], seg.sum(0), rtol=0, atol=1e-12)
        assert np.allclose(a["sumsq"][b], (seg ** 2).sum(0), rtol=1e-12, atol=1e-18)
    assert not a["sum"][k + 1:].any() and not a["sumsq"][k + 1:].any()
    # the chain axis form gives the same bits
    b3 = diag.accumulate(np.stack([x, x]), K)
    for key in a:
        assert np.array_equal(b3[key][1], a[key]), key


def test_accumulate_keeps_the_variance_of_a_large_offset():
    """Sums of d = x - ref: a hypocentre at 200 km with an sd of 0.01 km keeps its variance."""
    rng = np.random.default_rng(3)
    x = 200.0 + 0.01 * rng.standard_normal((64, 4096, 1))
    acc = diag.accumulate(x, 16)
    s = diag.summarise(**acc)
    assert abs(s["sd"][0] / 0.01 - 1.0) < 0.01
    assert abs(s["mean"][0] - 200.0) < 1e-3


def _ar1(n_chains, n, rho, rng):
    e = rng.standard_normal((n_chains, n))
    x = np.empty_like(e)
    x[:, 0] = e[:, 0] / np.sqrt(1.0 - rho * rho)
    for t in range(1, n):
        x[:, t] = rho * x[:, t - 1] + e[:, t]
    return x


@pytest.fixture(scope="module")
def synthetic():
    rng = np.random.default_rng(2024)
    n, m = 2000, 4096
    iid = rng.standard_normal((n, m))
    ar = _ar1(n, m, 0.9, rng)
    shifted = rng.standard_normal((n, m))
    shifted[: n // 2] += 1.0
    return {name: diag.summarise(**diag.accumulate(x[:, :, None], 16)) for name, x in
            (("iid", iid), ("ar", ar), ("shifted", shifted))}


def test_iid_chains_have_rhat_one_and_ess_n(synthetic):
    s = synthetic["iid"]
    assert s["chains_used"] == 2000
    assert abs(s["rhat"][0] - 1.0) < 0.01
    assert abs(s["ess"][0] / s["n_models"] - 1.0) < 0.10


def test_ar1_ess_follows_the_autocorrelation(synthetic):
    s = synthetic["ar"]
    rho = 0.9
    want = (1 - rho) / (1 + rho)
    assert abs(s["ess"][0] / s["n_models"] / want - 1.0) < 0.15
    assert abs(s["rhat"][0] - 1.0) < 0.01


def test_chains_that_disagree_have_a_large_rhat(synthetic):
    assert synthetic["shifted"]["rhat"][0] > 1.1


def _acc(k, L, S, T, ref=0.0):
    """accumulators of one chain with k full batches of L models: S, T lists of k per-batch sums (one quantity)"""
    K = 16
    s, t = np.zeros((K, 1)), np.zeros((K, 1))
    s[:k, 0], t[:k, 0] = S, T
    return dict(ref=np.array([ref]), sum=s, sumsq=t, batch_len=L, full_batches=k, n_models=k * L)


def test_edge_cases_give_their_documented_values():
    # no chain with four full batches: everything NaN
    s = diag.summarise(**diag.stack([_acc(3, 1, [0, 1, 2], [0, 1, 4])]))
    assert s["chains_used"] == 0 and all(np.isnan(s[k][0]) for k in ("mean", "sd", "rhat", "ess"))
    # constant everywhere: var+ == 0, rhat and ess NaN, mean and sd finite
    const = [_acc(4, 2, [0] * 4, [0] * 4, ref=5.0), _acc(4, 2, [0] * 4, [0] * 4, ref=5.0)]
    s = diag.summarise(**diag.stack(const))
    assert s["chains_used"] == 2 and s["mean"][0] == 5.0 and s["sd"][0] == 0.0
    assert np.isnan(s["rhat"][0]) and np.isnan(s["ess"][0])
    # constant within each chain, different between chains: W == 0 < var+, rhat +inf; sigma2 == 0, ess +inf
    s = diag.summarise(**diag.stack([_acc(4, 2, [0] * 4, [0] * 4, ref=1.0), _acc(4, 2, [0] * 4, [0] * 4, ref=2.0)]))
    assert s["rhat"][0] == np.inf and s["ess"][0] == np.inf and s["sd"][0] > 0
    # batch means all equal but values vary inside the batches: sigma2 == 0 < var+ (W > 0), ess +inf, rhat finite
    s = diag.summarise(**diag.stack([_acc(4, 2, [0] * 4, [2] * 4), _acc(4, 2, [0] * 4, [2] * 4)]))
    assert np.isfinite(s["rhat"][0]) and s["ess"][0] == np.inf
