"""Checkpoint and resume without a GPU: the library exports the three state entry points, and the command line checks a
checkpoint given to -R before it creates a handle or touches a chain file."""
import ctypes as C
import os
import subprocess

from tests import inputs, util

LIB = os.path.join(util.ROOT, "mcmc_eq_b200", "libmcmceq_b200.so")
EXE = os.path.join(util.ROOT, "mcmc_eq_b200", "host", "mcmc_eq")


def test_library_exports_the_state_entry_points():
    assert os.path.exists(LIB), "libmcmceq_b200.so not built (python -m mcmc_eq_b200.build)"
    lib = C.CDLL(LIB)
    for name in ("mq_state_size", "mq_state_save", "mq_state_load"):
        assert hasattr(lib, name), name


def test_resume_from_a_garbage_file_fails_before_a_handle_exists(tmp_path):
    assert os.path.exists(EXE), "host/mcmc_eq not built (python -m mcmc_eq_b200.build)"
    d = str(tmp_path)
    inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=77)
    with open(os.path.join(d, "ck"), "wb") as f:
        f.write(b"this is not a checkpoint" * 40)
    r = subprocess.run([EXE, "config_eqx.dat", "rjx-%03d.out", "picks", "-n", "4", "-R", "ck", "-q"], cwd=d, capture_output=True,
                       text=True, timeout=120)
    assert r.returncode != 0
    assert "not a checkpoint" in r.stderr and "mq_create" not in r.stderr, r.stderr
    assert not [f for f in os.listdir(d) if f.startswith("rjx-")]
