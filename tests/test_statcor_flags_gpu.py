"""Every station-correction flag (config scor_flag, src/mcmc_eq.c:910-928) through the batched sampler.

 0: corrections keep their mean (+dx at the chosen station, -dx/(ns-1) everywhere else);
-1: S corrections never move; -2: P corrections never move (the perturbation also gets a second addition at the station);
 1: the reference station's P correction is held at ref_statcor_P, one station moves per accepted step;
 2: both corrections of the reference station are held (ref_statcor_P / ref_statcor_S).

The proposal is scored through the misfit kernel's correction override (forward.cu), the accept applies it to the stored
corrections (chain.cu) with the same float operations, so the maintained likelihood equals a fresh forward of the stored
state bit for bit.  A difference means a proposal was scored on corrections other than the ones it stored."""
import tempfile

import numpy as np
import pytest

from tests import inputs

pytestmark = pytest.mark.gpu

REF = 3
REF_P, REF_S = 0.125, -0.375


def _sampler(flag, n=32, seed=17):
    import mcmc_eq_b200 as mq
    d = tempfile.mkdtemp(prefix="mqsc_")
    cfgp, pkp = inputs.materialise("example2", d, scor_flag=flag, reference_station=REF, ref_statcor_P=REF_P,
                                   ref_statcor_S=REF_S, j_max_start=0, j_max_main=100000, sdev_start_delay=0.2)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    assert cfg.scor_flag == flag and cfg.reference_station == REF and pk.n_stations > REF + 1
    return cfg, pk, mq.Sampler(cfg, pk, n, 0, seed)


def _check_fresh_forward(smp):
    """mf / ll / rms / origin maintained by the sampler against a from-scratch forward of the stored state."""
    _c, ll, rms = smp.stats()
    m = smp.get_models()
    _mf, origin = smp.forward(3)
    _c2, ll2, rms2 = smp.stats()
    assert np.array_equal(ll2, ll), (np.abs(ll2 - ll).max(), int((ll2 != ll).sum()))
    assert np.array_equal(rms2, rms)
    assert np.array_equal(origin, m.origin)


@pytest.mark.parametrize("flag", [-2, -1, 0, 1, 2])
def test_station_correction_flag(flag):
    cfg, pk, smp = _sampler(flag)
    smp.init_chains()
    m0 = smp.get_models()
    n = smp.n
    # start values (src/mcmc_eq.c:585-600): the reference station starts at the given corrections under flags 1 and 2
    if flag in (1, 2):
        assert (m0.pres[:, REF] == np.float32(REF_P)).all()
    if flag == 2:
        assert (m0.sres[:, REF] == np.float32(REF_S)).all()
    # start corrections are drawn (sdev_start_delay > 0): the invariants below are not about zeros
    assert np.abs(m0.pres).max() > 0.01 and np.abs(m0.sres).max() > 0.01

    iters = 60
    if flag in (1, 2):      # one iteration at a time: at most one station changes per step
        prev = m0
        for _ in range(iters):
            smp.step(1, "RRRRQN")
            cur = smp.get_models()
            changed = (cur.pres != prev.pres) | (cur.sres != prev.sres)
            assert (changed.sum(1) <= 1).all(), np.nonzero(changed.sum(1) > 1)
            prev = cur
    else:
        smp.step(iters, "RRRRQN")
    counts, _ll, _rms = smp.stats()
    r_acc = counts[:, 1:17].reshape(n, 8, 2)[:, :, 0]     # accepted, per proposal kind (N P V Q R M B D)
    m = smp.get_models()
    dp, ds = m.pres != m0.pres, m.sres != m0.sres
    if flag == -1:
        assert np.array_equal(m.sres, m0.sres) and dp.any()
    if flag == -2:
        assert np.array_equal(m.pres, m0.pres) and ds.any()
    if flag == 0:
        assert dp.any() and ds.any()
        assert np.abs(m.pres.mean(1) - m0.pres.mean(1)).max() < 1e-5
        assert np.abs(m.sres.mean(1) - m0.sres.mean(1)).max() < 1e-5
    if flag == 1:
        assert (m.pres[:, REF] == np.float32(REF_P)).all()
        assert ds[:, REF].any(), "the reference station's S correction must still move under flag 1"
        assert dp[:, np.arange(pk.n_stations) != REF].any()
    if flag == 2:
        assert (m.pres[:, REF] == np.float32(REF_P)).all() and (m.sres[:, REF] == np.float32(REF_S)).all()
        assert dp.any() and ds.any()
    assert r_acc[:, 4].sum() > 0                     # R proposals were accepted
    _check_fresh_forward(smp)
    smp.close()
