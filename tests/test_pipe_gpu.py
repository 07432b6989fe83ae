"""The two eikonal kernels against each other: the pipelined kernel (default: box phases on a pool of shared-memory slices,
column marches in tensor memory, csrc/eik_march.cuh: tcgen05.ld/st 32x32b) and the fused kernel (MCMCEQ_EIKONAL_PIPE=0:
everything in shared memory).  Same arithmetic, so class sums, origin times, per-pick predictions and chain trajectories must
be IDENTICAL bit for bit; each runs in its own subprocess because the switch is read once per process."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu

SCRIPT = r"""
import sys, tempfile, numpy as np
sys.path.insert(0, %r)
import mcmc_eq_b200 as mq
from tests import inputs, fwd_helpers as fh
out = {}
for name in ("example2", "example"):
    d = tempfile.mkdtemp(prefix="mqsp_")
    cfgp, pkp = inputs.materialise(name, d)
    cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    n = int(sys.argv[2])                          # not a multiple of 32: ragged last warp
    smp = mq.Sampler(cfg, pk, n, 0, 1)
    rng = np.random.default_rng(4)
    kinds = sys.argv[3].split(",") if len(sys.argv) > 3 else ["lvz", "posterior"]      # example2, example
    st = fh.random_states(rng, cfg, pk, n, kind=kinds[1] if name == "example" else kinds[0])
    mf, org = smp.forward_host(fh.fill_models(smp.new_models(32), st), 3)
    res, tp = smp.predictions(3)
    smp.init_chains(); smp.step(6, "PVMBDQ")
    c, ll, rms = smp.stats()
    out[name + "_mf"] = mf; out[name + "_org"] = org; out[name + "_tp"] = tp; out[name + "_ll"] = ll; out[name + "_c"] = c
    smp.close()
np.savez(sys.argv[1], **out)
"""


def _run(path, pipe, n, row_march=True, kinds="lvz,posterior"):
    env = dict(os.environ, MCMCEQ_EIKONAL_PIPE="1" if pipe else "0", MCMCEQ_ROW_MARCH="1" if row_march else "0")
    r = subprocess.run([sys.executable, "-c", SCRIPT % util.ROOT, path, str(n), kinds], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-1500:]
    return dict(np.load(path))


def test_pipelined_kernel_is_bit_identical_to_the_fused_kernel(tmp_path):
    """One persistent CTA per SM, 16 warps sharing a pool of shared-memory slices (box phase) and a pool of TMEM sets (march)."""
    # the pipelined kernel only takes launches with work for all 148 x 12 warps: 1230 chains x 2 phases x 61 depths
    a = _run(str(tmp_path / "fused.npz"), False, 1230)
    b = _run(str(tmp_path / "pipe.npz"), True, 1230)
    for k in a:
        assert np.array_equal(a[k], b[k]), (k, int((a[k] != b[k]).sum()), a[k].size, float(np.nanmax(np.abs(a[k].astype(float) - b[k].astype(float)))))


@pytest.mark.parametrize("kinds", ["posterior,contrast", "contrast,lvz", "gradient,gradient"])
def test_pipelined_kernel_is_bit_identical_on_other_model_families(tmp_path, kinds):
    """The box phase is inlined into the pipelined kernel since round 2; the compiler fault that kept it out of line in
    round 1 (eikonal.cu, solve_warp_call) gave wrong times on one model family and right ones on another, so the comparison
    runs on all of them (Example2 grid, Example grid): low-velocity zones, posterior-like, high-contrast, gradient models."""
    a = _run(str(tmp_path / "fused.npz"), False, 1230, kinds=kinds)
    b = _run(str(tmp_path / "pipe.npz"), True, 1230, kinds=kinds)
    for k in a:
        assert np.array_equal(a[k], b[k]), (kinds, k, int((a[k] != b[k]).sum()), a[k].size)


def test_lock_step_row_sweeps_are_bit_identical_to_the_general_walk(tmp_path):
    """Rows whose past times do not decrease away from the axis are swept in lock-step (eik_fast.cuh: row_march) instead of by
    the per-lane walk (MCMCEQ_ROW_MARCH=0): the same nodes from the same neighbours, so identical bits -- in both kernels."""
    a = _run(str(tmp_path / "walk.npz"), False, 70, row_march=False)
    b = _run(str(tmp_path / "rows.npz"), False, 70)
    c = _run(str(tmp_path / "pipe_walk.npz"), True, 1230, row_march=False)
    d = _run(str(tmp_path / "pipe_rows.npz"), True, 1230)
    for x, y in ((a, b), (c, d)):
        for k in x:
            assert np.array_equal(x[k], y[k]), k
