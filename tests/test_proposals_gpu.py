"""The device sampler against the host restatement of the reference (tests/sampler_ref.py), draw for draw.

tests/test_sampler_ref_cpu.py ties the restatement to the reference: driven by libc rand() it walks both recorded reference
chains bit for bit.  Here the restatement is driven by the device's own Philox streams and must reproduce what the device
does: the start models of mq_init_chains, and every iteration of mq_step(1) from the device's saved state -- the arm, its
bounded Gaussian draws, retry loops, eligibility rules, the epi_search factor of the start phase, the LVZ switch, the
proposal ratios of B, D and N, and the accept draw.  Every step starts from the device's own state, so a difference is
found at the iteration that made it.

Compared bit for bit: dim, z / vp / vpvs, hypocentres, station corrections, sigmas, inv_control; exactly: draws, acce,
reject and the 20 counters.  The one allowed difference is a Gaussian deviate whose double value lies within 2^-52 of a
float rounding boundary (the device's double log is not glibc's): the prediction is then redone with that deviate rounded
the other way and must match exactly; such cases are counted and reported.  Decisions whose log-likelihood comes from the
FP32 forward are compared with the near-tie rule of tests/test_replay_gpu.py."""
import math
import multiprocessing as mp
import os
import tempfile
import time

import numpy as np
import pytest

from tests import inputs, sampler_ref as S

pytestmark = pytest.mark.gpu

NO_RECORDS = 10**9          # deci: no decimated record is ever written, so a state can be saved after every step
TOTALS = dict(chain_iterations=0, near_ties=0, one_ulp=0)


@pytest.fixture(scope="module")
def pool():
    # the workers run the restatement only (no CUDA call), so a fork of a process that holds a CUDA context is safe
    p = mp.get_context("fork").Pool(max(1, min(16, (os.cpu_count() or 2) - 1)))
    t0 = time.time()
    yield p
    p.close()
    p.join()
    print(f"\nproposals: {TOTALS['chain_iterations']} chain-iterations compared, {TOTALS['near_ties']} near-ties declared, "
          f"{TOTALS['one_ulp']} one-ulp Gaussian deviates, {time.time() - t0:.0f} s")


def _setup(name, n, seed=1, picks_fix=None, **over):
    import mcmc_eq_b200 as mq
    over.setdefault("deci", NO_RECORDS)
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise(name, d, **over)
        cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    if picks_fix is not None:
        nc = pk.n_class
        pk = mq.Picks(pk.ev_off, pk.n_p, pk.st_id, pk.x, pk.y, pk.z, pk.t, pk.cls, pk.reftime, picks_fix, pk.n_stations)
        pk.n_class = nc
    smp = mq.Sampler(cfg, pk, n, 0, seed)
    return smp, cfg, pk, S.make_cfg(cfg, pk)


def _bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def _diff(want: S.State, B: S.SavedState, ch: int):
    """-> [] when device chain ch of state B equals the prediction, else the names of the fields that differ, floats
    bit for bit."""
    got = B.chain(ch)
    bad = []
    if got.dim != want.dim:
        return ["dim"]
    for k in ("z", "vp", "vpvs", "eq", "pres", "sres", "noise"):
        if not np.array_equal(_bits(getattr(got, k)), _bits(getattr(want, k))):
            bad.append(k)
    if _bits(got.inv) != _bits(want.inv):
        bad.append("inv_control")
    for k in ("draws", "acce", "reject", "counts"):
        if getattr(got, k) != getattr(want, k):
            bad.append(k)
    return bad


# ---- start models ------------------------------------------------------------------------------------------------------

def _fixed_components(name):
    _c, arr = inputs.load(name)
    fix = np.array(arr["fix"], np.float64).reshape(-1, 3)
    fix[0] = (1.25, -3.5, 4.0)           # all three fixed
    fix[3, 2] = 7.75                     # depth only
    fix[10, 0] = -2.0                    # x only
    return fix


START_CASES = [
    ("example", dict(), {}),
    ("example2", dict(), {}),
    ("example2", dict(tria=1), {}),
    ("example2", dict(start_cell_number=1), {}),
    ("example2", dict(scor_flag=1, reference_station=2, ref_statcor_P=0.3125, sdev_start_delay=0.1), {}),
    ("example2", dict(scor_flag=2, reference_station=5, ref_statcor_P=-0.25, ref_statcor_S=0.4375, sdev_start_delay=0.1), {}),
    ("example2", dict(), dict(fix=True)),
    ("example2", dict(), dict(seed=(0xDEADBEEF << 32) | 12345, offset=1000)),
]


@pytest.mark.parametrize("name,over,extra", START_CASES, ids=[f"{n}-{i}" for i, (n, _o, _e) in enumerate(START_CASES)])
def test_start_models_equal_the_restatement(pool, name, over, extra):
    n = 1024
    seed = extra.get("seed", 1)
    smp, _cfg, _pk, c = _setup(name, n, seed=seed, picks_fix=_fixed_components(name) if extra.get("fix") else None, aflag=1, **over)
    off = extra.get("offset", 0)
    if off:
        smp.set_chain_offset(off)
    smp.init_chains()
    B = S.SavedState(smp.save_state())
    assert B.seed == seed and B.chain_offset == off
    preds = pool.map(S.init_job, [(c, seed, off + ch) for ch in range(n)], chunksize=16)
    bad = []
    for ch, (want, ok) in enumerate(preds):
        assert ok
        d = _diff(want, B, ch)
        if d:
            bad.append((ch, d))
    TOTALS["chain_iterations"] += n
    assert not bad, bad[:8]
    smp.close()


# ---- stepping ----------------------------------------------------------------------------------------------------------

def _loglik_of_proposals(fwd, preds, B, c):
    """new log-likelihood of every chain's proposal: from the saved class sums for N (exact), from mq_forward_host on a
    second handle for the others (FP32 forward: near-tie rule)."""
    m = fwd.new_models(c.md)
    exact = np.zeros(B.n, bool)
    for ch, (st, P, _r) in enumerate(preds):
        s = P.new if (P.new is not None and P.eligible and P.ok) else st
        m.dim[ch] = s.dim
        m.z[ch, :s.dim], m.vp[ch, :s.dim], m.vpvs[ch, :s.dim] = s.z, s.vp, s.vpvs
        m.eq[ch], m.pres[ch], m.sres[ch], m.noise[ch] = s.eq, s.pres, s.sres, s.noise
        exact[ch] = P.kind == "N"
    mf, _o = fwd.forward_host(m, 3)
    out = []
    for ch, (st, P, _r) in enumerate(preds):
        if P.kind == "N":
            out.append(S.loglik(B.head["mf"][ch], P.new.noise))
        else:
            out.append(S.loglik(mf[ch], m.noise[ch]))
    return out, exact


def _run(smp, c, pool, iters, override=None, beta=None, fwd=None, max_ties=0):
    """Steps the device `iters` times with mq_step(1); before each step the restatement predicts every chain's next state
    from the saved one.  beta: the inverse temperature of every chain (mq_set_beta), None = 1.  fwd: a second handle for
    the likelihood of the proposals (aflag = 0, beta = 1).  -> the kinds of the proposals seen."""
    if beta is not None:
        smp.set_beta(np.full(smp.n, beta, np.float32))
    b = 1.0 if beta is None else float(np.float32(beta))
    kinds = {}
    ties = one_ulp = 0
    for it in range(iters):
        A = S.SavedState(smp.save_state())
        jobs = [(A.chain(ch), c, A.seed, A.chain_offset + ch, override, ()) for ch in range(A.n)]
        preds = pool.map(S.propose_job, jobs, chunksize=8)
        if c.aflag == 1:
            new_ll, exact = [0.0] * A.n, np.ones(A.n, bool)
        elif fwd is not None:
            new_ll, exact = _loglik_of_proposals(fwd, preds, A, c)
        else:     # beta so small that the likelihoods do not move alpha: any value does
            new_ll, exact = [st.ll for st, _P, _r in preds], np.ones(A.n, bool)
        wants = []
        for ch, (st, P, rng) in enumerate(preds):
            before = st.copy()
            acc, u, _alpha = S.decide(st, P, c, rng, new_ll[ch], b)
            st.draws = rng.draws
            wants.append((st, P, acc, u, before))
            if P.kind:
                kinds[P.kind] = kinds.get(P.kind, 0) + 1
        smp.step(1, override)
        B = S.SavedState(smp.save_state())
        for ch, (want, P, acc, u, before) in enumerate(wants):
            d = _diff(want, B, ch)
            if not d:
                continue
            got = B.chain(ch)
            if not exact[ch] and set(d) <= {"acce", "reject", "counts", "dim", "z", "vp", "vpvs", "eq", "pres", "sres"} \
                    and (got.acce == want.acce - 1 if acc else got.acce == want.acce + 1):
                # a decision taken the other way: allowed at a near-tie only, then the state must be the other outcome's
                margin = abs(math.log(max(u, 1e-30)) - (P.log_fac + new_ll[ch] - before.ll))
                assert margin <= 2e-5 * max(abs(new_ll[ch]), abs(before.ll)) + 1e-3, (it, ch, P.kind, margin, d)
                alt = before.copy()
                S.decide(alt, P, c, S.Rand(S.Philox(0, 0, 0)), 1e30 if not acc else -1e30, 1.0, u=u)
                alt.draws = want.draws
                assert not _diff(alt, B, ch), (it, ch, P.kind, _diff(alt, B, ch))
                ties += 1
                continue
            # a Gaussian deviate near a float rounding boundary: redo the prediction with it rounded the other way
            redone = False
            rng0 = S.Rand(S.Philox(A.seed, A.chain_offset + ch, A.chain(ch).draws))
            S.propose(A.chain(ch), c, rng0, override)
            for k in rng0.fragile:
                st2, P2, r2 = S.propose_job((A.chain(ch), c, A.seed, A.chain_offset + ch, override, (k,)))
                S.decide(st2, P2, c, r2, new_ll[ch], b)
                st2.draws = r2.draws
                if not _diff(st2, B, ch):
                    redone = True
                    break
            assert redone, f"iteration {it}, chain {ch}, arm {P.kind!r}: {d} differ (acce {want.acce}, draws {before.draws})"
            one_ulp += 1
        TOTALS["chain_iterations"] += A.n
    assert ties <= max_ties, ties
    TOTALS["near_ties"] += ties
    TOTALS["one_ulp"] += one_ulp
    return kinds


PRIOR_CASES = [
    ("example2", 256, 300, "QRPVMBDN", dict()),
    ("example2", 256, 300, None, dict()),
    ("example2", 64, 150, "QRPVMBDN", dict(tria=1, j_max_start=40, j_max_main=80)),
] + [("example2", 64, 120, "RRRQPN", dict(scor_flag=f, reference_station=1, ref_statcor_P=0.25, ref_statcor_S=-0.125,
                                          j_max_start=40, j_max_main=60)) for f in (-2, -1, 0, 1, 2)]


@pytest.mark.parametrize("name,n,iters,override,over", PRIOR_CASES, ids=[f"prior{i}" for i in range(len(PRIOR_CASES))])
def test_prior_regime_every_arm_draw_for_draw(pool, name, n, iters, override, over):
    """aflag = 1: every eligible proposal is accepted, so every arm's output is visible.  j_max_start is crossed (the
    epi_search factor and the start string end) and j_max_main is reached by some chains (finished chains draw nothing)."""
    over = dict(dict(j_max_start=100, j_max_main=150), **over)
    smp, _cfg, _pk, c = _setup(name, n, seed=11, aflag=1, **over)
    smp.init_chains()
    kinds = _run(smp, c, pool, iters, override)
    want = set(override or (c.ps_start + c.ps_main))
    assert set(kinds) == want, kinds
    counts, _ll, _rms = smp.stats()
    acce = S.SavedState(smp.save_state()).head["acce"]
    assert (acce > c.j_max_start).any(), "the main phase was never reached"
    if iters >= c.j_max_start + c.j_max_main:
        assert (acce == c.j_max_start + c.j_max_main).any(), "no chain finished"
    smp.close()


def test_proposal_ratios_decide_alone(pool):
    """aflag = 0 and beta = 1e-30: alpha is 1 for P V M Q R N and nexp(log_fac) for B and D, so the decisions test the
    device's birth and death log_fac with no likelihood involved.  max_dim = 8 with inv_control = -1 makes B ineligible
    from three nuclei on (dim + 1 < max_dim / (1 + |inv|))."""
    smp, _cfg, _pk, c = _setup("example2", 64, seed=5, max_dim=8, j_max_start=20, j_max_main=400)
    smp.init_chains()
    kinds = _run(smp, c, pool, 150, "BDBDBDPVMQRN", beta=1e-30)
    assert {"B", "D"} <= set(kinds)
    counts, _ll, _rms = smp.stats()
    assert counts[:, 13].sum() > 0 and counts[:, 14].sum() > 0 and counts[:, 15].sum() > 0 and counts[:, 16].sum() > 0
    smp.close()


REAL_CASES = [
    ("example2", 64, 300, dict(j_max_start=60, j_max_main=1000)),
    ("example", 64, 300, dict(tria=1, j_max_start=60, j_max_main=1000)),
    # inv_control > 0: the LVZ switch at acce == revert = 20 + 30 / 2 fires on every iteration the chain sits there (Q1)
    ("example2", 64, 200, dict(inv_control=1.0, j_max_start=20, j_max_main=30)),
]


@pytest.mark.parametrize("name,n,iters,over", REAL_CASES, ids=["example2", "example-tria", "lvz"])
def test_the_real_sampler_draw_for_draw(pool, name, n, iters, over):
    """beta = 1, aflag = 0: the likelihood of N exactly from the class sums, of the other arms from mq_forward_host on a
    second handle (FP32 forward), a decision differing only at a declared near-tie."""
    smp, cfg, pk, c = _setup(name, n, seed=21, **over)
    import mcmc_eq_b200 as mq
    fwd = mq.Sampler(cfg, pk, n, 0, 21)
    smp.init_chains()
    inv0 = S.SavedState(smp.save_state()).head["inv_control"].copy()
    _run(smp, c, pool, iters, fwd=fwd, max_ties=max(2, n * iters // 2000))
    A = S.SavedState(smp.save_state())
    if "inv_control" in over:
        assert (A.head["acce"] > c.revert).any()
        assert (A.head["inv_control"] != inv0).any()
    fwd.close()
    smp.close()


# ---- edges -------------------------------------------------------------------------------------------------------------

def _models(smp, c, dim, z, vp, vpvs, noise=None):
    m = smp.new_models(c.md)
    m.dim[:] = dim
    for ch in range(smp.n):
        m.z[ch, :dim], m.vp[ch, :dim], m.vpvs[ch, :dim] = z, vp, vpvs
    m.eq[:] = np.array([[(c.xmin + c.xmax) / 2, (c.ymin + c.ymax) / 2, 5.0]], np.float32)
    m.noise[:] = 1.0 if noise is None else noise
    return m


@pytest.mark.parametrize("case", ["dim1", "tria-dim3", "birth-bound"])
def test_ineligible_moves_are_rejected_and_consume_their_uniform(pool, case):
    if case == "dim1":
        smp, _cfg, _pk, c = _setup("example2", 16, seed=3)
        smp.set_models(_models(smp, c, 1, [5.0], [5.0], [1.7]))
        over = "MD"
    elif case == "tria-dim3":
        smp, _cfg, _pk, c = _setup("example2", 16, seed=3, tria=1)
        smp.set_models(_models(smp, c, 3, [c.zmin, c.zmax, 10.0], [3.0, 9.0, 6.0], [1.7, 1.7, 1.7]))
        over = "MD"
    else:   # max_dim 6, |inv| = 1: dim + 1 < 3 fails at dim = 2
        smp, _cfg, _pk, c = _setup("example2", 16, seed=3, max_dim=6)
        smp.set_models(_models(smp, c, 2, [3.0, 15.0], [4.0, 6.0], [1.7, 1.7]))
        over = "B"
    smp.step(1, over)
    A = S.SavedState(smp.save_state())
    _run(smp, c, pool, 4, over)
    B = S.SavedState(smp.save_state())
    assert (B.head["acce"] == A.head["acce"]).all() and (B.head["reject"] == A.head["reject"] + 4).all()
    assert (B.head["draws"] == A.head["draws"] + 8).all()      # the arm and the accept test: two draws each
    smp.close()


@pytest.mark.parametrize("aflag", [0, 1])
def test_a_proposal_that_cannot_succeed_gives_up_and_is_rejected(pool, aflag):
    """A sigma far outside [noise_min, noise_max] (20 against 10, sdevn 0.01): the N arm's bounded draw gives up after 10^5
    tries.  The device must stop after exactly the restatement's draws and reject it, also when sampling the prior."""
    smp, _cfg, _pk, c = _setup("example2", 4, seed=9, aflag=aflag)
    noise = np.ones(8, np.float32)
    noise[3] = 20.0
    smp.set_models(_models(smp, c, 2, [3.0, 15.0], [4.0, 6.0], [1.7, 1.7], noise))
    smp.step(1, "Q")
    A = S.SavedState(smp.save_state())
    _run(smp, c, pool, 1, "N")
    B = S.SavedState(smp.save_state())
    assert (B.head["reject"] == A.head["reject"] + 1).all() and (B.head["acce"] == A.head["acce"]).all()
    assert (B.head["draws"] - A.head["draws"] > 200000).all()
    assert (B.head["noise"] == A.head["noise"]).all()
    smp.close()


def test_a_stream_position_past_two_to_the_34_draws(pool):
    """draws moved to just below 2^34 in a saved state: the block index then has a non-zero high word (ctr[1])."""
    smp, _cfg, _pk, c = _setup("example2", 32, seed=(7 << 32) | 7, aflag=1, j_max_start=100, j_max_main=150)
    smp.init_chains()
    A = S.SavedState(smp.save_state())
    A.head["draws"][:] = (1 << 34) - 5 + np.arange(smp.n) % 4
    smp.load_state(A.edited())
    assert (S.SavedState(smp.save_state()).head["draws"] == A.head["draws"]).all()
    _run(smp, c, pool, 20, "QRPVMBDN")
    assert (S.SavedState(smp.save_state()).head["draws"] > (1 << 34)).all()
    smp.close()
