"""The pipelined eikonal kernel on planes of 88 - 126 depth nodes (its CA = 128 instantiation: 128-node column arrays in tensor
memory), the planes of the two example grids refined by halving the spacing.  Against the fused kernel (MCMCEQ_EIKONAL_PIPE=0)
bit for bit, as tests/test_pipe_gpu.py does for the Example plane, on which kernel the dispatch picks, and at bench scale on
the halved Example grid against the CPU oracle."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu

N_CHAINS = 1000          # not a multiple of 32 (ragged last warp); 2 x 1000 x 88 solves fill 148 x 8 warps and more
LOWEST_DEEP_NZ = 88      # the lowest nz the dispatch sends to the CA = 128 instantiation (eikonal.cu: kPipeDeepMinNz)

# name -> (input set, config override): halved Example2 (plane 272 x 121), halved Example (564 x 123), the deepest plane of
# the instantiation (272 x 126, even nz), the lowest nz it takes (272 x 88).  Example2's start models (3.5 km/s + 0.25 km/s
# per km) must stay below its vpmax = 12 km/s: at h = 0.25 km these planes end at 19.75 - 29.25 km depth
PLANES = {
    "example2_half": ("example2", dict(h=0.25, nx=193, ny=193, nz=121)),
    "example_half": ("example", dict(h=1.0, nx=399, ny=399, nz=123)),
    "nz126": ("example2", dict(h=0.25, nx=193, ny=193, nz=126)),
    "nz_lowest": ("example2", dict(h=0.25, nx=193, ny=193, nz=LOWEST_DEEP_NZ)),
}
KINDS = ("lvz", "posterior", "contrast", "gradient")

SCRIPT = r"""
import json, sys, tempfile, numpy as np
sys.path.insert(0, %r)
import mcmc_eq_b200 as mq
from tests import inputs, fwd_helpers as fh
planes, kinds, n = json.loads(sys.argv[2]), sys.argv[3].split(","), int(sys.argv[4])
out = {}
for name, (inp, over) in planes.items():
    d = tempfile.mkdtemp(prefix="mqdeep_")
    cfgp, pkp = inputs.materialise(inp, d, **over)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    for kind in kinds:
        smp = mq.Sampler(cfg, pk, n, 0, 1)
        rng = np.random.default_rng(4)
        st = fh.random_states(rng, cfg, pk, n, kind=kind)
        smp.profile(True)
        mf, org = smp.forward_host(fh.fill_models(smp.new_models(32), st), 3)
        smp.profile(False)
        ks = sorted(smp.profile_kernels())
        res, tp = smp.predictions(3)
        _r, tp_last = smp.predictions(n - 1)
        smp.init_chains(); smp.step(6, "PVMBDQ")
        c, ll, rms = smp.stats()
        key = name + "_" + kind
        out[key + "_mf"] = mf; out[key + "_org"] = org; out[key + "_tp"] = tp; out[key + "_tpl"] = tp_last
        out[key + "_ll"] = ll; out[key + "_c"] = c; out[key + "_kernels"] = np.array(ks)
        smp.close()
np.savez(sys.argv[1], **out)
"""


def _run(path, pipe, planes=PLANES, kinds=KINDS):
    import json
    env = dict(os.environ, MCMCEQ_EIKONAL_PIPE="1" if pipe else "0")
    r = subprocess.run([sys.executable, "-c", SCRIPT % util.ROOT, path, json.dumps(planes), ",".join(kinds), str(N_CHAINS)],
                       env=env, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-1500:]
    return dict(np.load(path))


def test_deep_pipelined_kernel_is_bit_identical_to_the_fused_kernel(tmp_path):
    """Class sums, origin times, per-pick predictions of the first and the last chain, counters and log-likelihoods after a
    few mixed steps: identical bits, on every plane and model family."""
    a = _run(str(tmp_path / "fused.npz"), False)
    b = _run(str(tmp_path / "pipe.npz"), True)
    for k in a:
        if k.endswith("_kernels"):
            assert list(a[k]) == ["eik_fast_kernel"], (k, a[k])
            assert list(b[k]) == ["eik_pipe_kernel"], (k, b[k])
            continue
        assert np.array_equal(a[k], b[k]), (k, int((a[k] != b[k]).sum()), a[k].size,
                                            float(np.nanmax(np.abs(a[k].astype(float) - b[k].astype(float)))))


def _kernels_taken(directory, name, nz_override=None):
    import mcmc_eq_b200 as mq
    from tests import fwd_helpers as fh
    from tests import inputs
    inp, over = PLANES[name]
    if nz_override is not None:
        over = dict(over, nz=nz_override)
    cfgp, pkp = inputs.materialise(inp, str(directory), **over)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    smp = mq.Sampler(cfg, pk, N_CHAINS, 0, 1)
    st = fh.random_states(np.random.default_rng(2), cfg, pk, N_CHAINS, kind="posterior")
    smp.profile(True)
    smp.forward_host(fh.fill_models(smp.new_models(32), st), 3)
    _ms, launches, per_launch = smp.profile(False)
    kernels = smp.profile_kernels()
    smp.close()
    assert launches == 1 and per_launch == 2 * N_CHAINS * cfg.grid.nz
    return list(kernels)


@pytest.mark.parametrize("name", sorted(PLANES))
def test_deep_planes_take_the_pipelined_kernel(tmp_path, name):
    assert _kernels_taken(tmp_path, name) == ["eik_pipe_kernel"]


def test_one_node_deeper_takes_the_fused_kernel(tmp_path):
    """nz = 127: a column array of 128 nodes holds nodes -1 .. 126, one too few."""
    assert _kernels_taken(tmp_path, "nz126", nz_override=127) == ["eik_fast_kernel"]


def test_one_node_shallower_than_the_deep_range_takes_the_fused_kernel(tmp_path):
    """Below LOWEST_DEEP_NZ a plane fills too little of a 128-node column array: the fused kernel is faster there."""
    assert _kernels_taken(tmp_path, "nz_lowest", nz_override=LOWEST_DEEP_NZ - 1) == ["eik_fast_kernel"]


def _generic_core_rows(slow, nxmod, iz, rows):
    """Receiver rows of one solve by the host build of the generic solver core (tests/emu), the arithmetic every kernel
    shares: [n_rows][nxmod]."""
    import ctypes as C
    from mcmc_eq_b200 import build
    from tests.util import fp, ptr
    L = C.CDLL(build.build_emu())
    L.emu_time_2d.argtypes = [fp, C.c_int, C.c_int, C.c_int, fp, C.POINTER(C.c_int)]
    t = np.zeros((nxmod, len(slow)), np.float32)
    cnt = np.zeros(7, np.int32)
    assert L.emu_time_2d(ptr(util.f32(slow)), nxmod, len(slow), iz, ptr(t), cnt.ctypes.data_as(C.POINTER(C.c_int))) == 0
    return t[:, rows].T


def test_deep_pipelined_kernel_at_bench_scale_matches_the_oracle():
    """The bench workload's events and stations on the Example grid at h = 1 km (plane 564 x 123), 1024 chains through
    mq_forward_host(calct = 3), chain states as tests/test_bench_scale_gpu.py prepares them; sampled chains, the first and the
    last warp-tasks included, against the CPU oracle: predictions (1e-4 s), class sums (2e-5 relative), origin times
    (1e-4 s), and every stored receiver-row node within util.eikonal_tol.  On a plane this wide the FP32 restatement of the
    solver itself can leave that bound late in a solve: the host build of the generic core (tests/emu), the arithmetic all
    kernels share, is 3.6e-4 s off at T = 87 s on one three-layer model here.  The rows of such a solve must then lie within
    util.eikonal_tol of that host build instead."""
    import ctypes as C

    import mcmc_eq_b200 as mq
    from mcmc_eq_b200 import synth
    from tests import fwd_helpers as fh
    from tests.test_bench_scale_gpu import _chain_states
    n = 1024
    cfg, pk, truth = synth.workload(200, 50, h=1.0, nx=399, ny=399, nz=123)
    assert util.nxmod_of(dict(nx=399, ny=399)) == 564
    ref_pred = fh.oracle_forward(cfg, pk, truth["z"], truth["vp"], truth["vpvs"], truth["eq"], truth["pres"], truth["sres"])[3]
    assert np.abs(ref_pred - truth["tpred"]).max() <= 1e-4
    smp, m = _chain_states(mq, synth, cfg, pk, n, 5)
    smp.profile(True)
    mf, origin = smp.forward_host(m, 3)
    _ms, launches, per_launch = smp.profile(False)
    assert launches == 1 and per_launch == 2 * n * cfg.grid.nz
    assert list(smp.profile_kernels()) == ["eik_pipe_kernel"]
    O = util.oracle()
    g = fh.fm_grid(cfg)
    rng = np.random.default_rng(11)
    chains = sorted(int(c) for c in rng.choice(n, size=12, replace=False)) + [0, 1, n - 2, n - 1]
    worst, outside = 0.0, 0
    for c in chains:
        d = int(m.dim[c])
        rmf, rorg, _res, rpred, tabs = fh.oracle_forward(cfg, pk, m.z[c, :d], m.vp[c, :d], m.vpvs[c, :d], m.eq[c], m.pres[c],
                                                          m.sres[c], want_tables=True)
        _r, tpred = smp.predictions(c)
        ok = np.abs(rpred) < 1e20
        assert ok.any() and (np.abs(tpred[ok] - rpred[ok]) <= 1e-4).all(), (c, np.abs(tpred[ok] - rpred[ok]).max())
        assert ((np.abs(tpred) > 1e20) == ~ok).all()
        fin = np.isfinite(rmf)
        assert (np.isfinite(mf[c]) == fin).all()
        assert np.allclose(mf[c][fin], rmf[fin], rtol=2e-5, atol=1e-6), (c, mf[c], rmf)
        if ok.all():
            assert np.abs(origin[c] - rorg).max() <= 1e-4, c
        for ph in (1, 2):
            rows, idx = smp.rows(c, ph)
            ref = tabs[ph - 1][idx]                     # [row][source depth][x]
            err = np.abs(rows - ref)
            worst = max(worst, float(err.max()))
            bad = np.unique(np.nonzero(err > util.eikonal_tol(ref))[1])
            if len(bad):
                slow = np.zeros(cfg.grid.nz, np.float32)
                (O.fm_rasterise_tria if cfg.tria == 1 else O.fm_rasterise)(
                    C.byref(g), d, util.ptr(util.f32(m.z[c, :d])), util.ptr(util.f32(m.vp[c, :d])), util.ptr(util.f32(m.vpvs[c, :d])),
                    ph, util.ptr(slow))
                for iz in bad:
                    outside += 1
                    core = _generic_core_rows(slow, smp.nxmod, int(iz), idx)
                    assert (np.abs(rows[:, iz] - core) <= util.eikonal_tol(core)).all(), (c, ph, int(iz), float(err[:, iz].max()))
    print(f"deep bench-scale parity (564 x 123, {len(chains)} chains): max |dT| row {worst:.2e} s; {outside} solves with row "
          f"nodes outside util.eikonal_tol of the oracle, all within it of the host build of the generic core")
    smp.close()
