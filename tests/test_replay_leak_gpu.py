"""A replayed iteration (mq_replay_step) leaves no trace in the free-running steps after it.

mq_replay_step hands the kernels the reference's uniform deviates in place of the chain's own draws.  Once it has
returned, every mq_step pass -- lock-step and desynchronised -- must draw its accept tests from the chain's counter-based
stream again: a pass that still sees the injected deviates would accept on them and consume no draw.  So two handles
that differ only by one replayed iteration in which no chain proposes anything must step on bit for bit alike."""
import tempfile

import numpy as np
import pytest

from tests import inputs

pytestmark = pytest.mark.gpu

N = 64


def _run(cfg, pk, replay):
    import mcmc_eq_b200 as mq
    smp = mq.Sampler(cfg, pk, N, 0, 5)
    try:
        smp.init_chains()
        if replay:   # no chain proposes: the replayed iteration changes no state of its own
            u = np.random.default_rng(3).random(N, np.float32)
            smp.replay_step(["\0"] * N, smp.get_models(), np.zeros(N, np.int32), np.zeros(N), u)
        recs, lost = [], []
        for n_iters, override in ((3, "P"), (24, None)):   # lock-step passes, then desynchronised ones (config strings)
            smp.step(n_iters, override)
            r, n_lost = smp.drain()
            recs += r
            lost.append(n_lost)
        c, ll, rms = smp.stats()
        m = smp.get_models()
        return c, ll, rms, m, recs, lost
    finally:
        smp.close()


def test_replay_step_leaves_free_running_steps_unchanged():
    import mcmc_eq_b200 as mq
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, j_max_start=10, j_max_main=100000, deci=5)
        cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    a = _run(cfg, pk, replay=True)
    b = _run(cfg, pk, replay=False)
    for name, x, y in zip(("counts", "loglik", "rms"), a[:3], b[:3]):
        assert np.array_equal(x, y), name
    assert a[0][:, 17].sum() > 0 and a[0][:, 18].sum() > 0   # both accepted and rejected proposals occurred
    for f in ("dim", "z", "vp", "vpvs", "eq", "pres", "sres", "noise", "origin"):
        assert np.array_equal(getattr(a[3], f), getattr(b[3], f)), f
    ra, rb = a[4], b[4]
    assert a[5] == b[5] == [0, 0], (a[5], b[5])   # records dropped by a full ring
    assert len(ra) == len(rb) > 0
    for x, y in zip(ra, rb):
        for k in x:
            assert np.array_equal(x[k], y[k]), (k, x["chain"], x["number"])
