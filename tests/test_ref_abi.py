"""host/ref_abi.h re-declares the struct layouts that cross the reference's function seam (src/mc.h:61-134).  Every size
and member offset is compared with tests/refapi.py, the ctypes mirror of those structs through which the compiled
reference wrote the fixtures under tests/golden, and, where the reference sources are present (REF_SRC, as for
oracle/Makefile), with the compiler's view of the reference header itself."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest

from tests import util

REF_SRC = os.environ.get("REF_SRC", "")     # the reference's src/ directory, as `make -C oracle REF_SRC=...` takes it

PROBE = r"""
#include <stdio.h>
#include <stddef.h>
%s
#define P(T, m) printf(#T "." #m " %%zu\n", offsetof(struct T, m))
int main(void)
{
    printf("Model %%zu\nDATA %%zu\nOBS %%zu\nGRDHEAD %%zu\nQUAKE %%zu\n", sizeof(struct Model), sizeof(struct DATA), sizeof(struct OBS),
           sizeof(struct GRDHEAD), sizeof(struct QUAKE));
    P(Model, number); P(Model, dimension); P(Model, noq); P(Model, nos); P(Model, pres); P(Model, sres); P(Model, origin);
    P(Model, %s); P(Model, z); P(Model, vp); P(Model, vpvs); P(Model, eq);
    P(GRDHEAD, nx); P(GRDHEAD, ny); P(GRDHEAD, nz); P(GRDHEAD, h); P(GRDHEAD, x0); P(GRDHEAD, y0); P(GRDHEAD, z0);
    P(OBS, st_id); P(OBS, x); P(OBS, y); P(OBS, z); P(OBS, t); P(OBS, cl); P(OBS, layer); P(OBS, w1); P(OBS, w2);
    P(DATA, eq_id); P(DATA, reftime); P(DATA, xfix); P(DATA, yfix); P(DATA, zfix); P(DATA, nobs_p); P(DATA, nobs_s);
    P(DATA, %s); P(DATA, p_picks); P(DATA, s_picks);
    return 0;
}
"""


def _offsets(d, name, include, noise_member, class_member, flags):
    src = os.path.join(d, name + ".c")
    open(src, "w").write(PROBE % (include, noise_member, class_member))
    exe = os.path.join(d, name)
    subprocess.run(["gcc", "-w", src, "-o", exe] + flags, check=True)
    out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    # the first noise sigma / class counter goes by different names in the two headers: compare by position
    return [ln.split()[-1] for ln in out.strip().split("\n")]


def _ours(d):
    return _offsets(d, "ours", '#include "%s"' % os.path.join(util.ROOT, "mcmc_eq_b200", "host", "ref_abi.h"), "noise", "nobs_class", [])


def test_ref_abi_header_matches_the_ctypes_mirror():
    from tests import refapi as R
    off = lambda T, *ms: [str(getattr(T, m).offset) for m in ms]
    mirror = ([str(C.sizeof(T)) for T in (R.Model, R.DATA, R.OBS, R.GRDHEAD, R.QUAKE)]
              + off(R.Model, "number", "dimension", "noq", "nos", "pres", "sres", "origin", "p_noise0", "z", "vp", "vpvs", "eq")
              + off(R.GRDHEAD, "nx", "ny", "nz", "h", "x0", "y0", "z0")
              + off(R.OBS, "st_id", "x", "y", "z", "t", "cl", "layer", "w1", "w2")
              + off(R.DATA, "eq_id", "reftime", "xfix", "yfix", "zfix", "nobs_p", "nobs_s", "nobs_p0", "p_picks", "s_picks"))
    with tempfile.TemporaryDirectory() as d:
        assert _ours(d) == mirror


def test_ref_abi_header_matches_the_reference_layout():
    if not os.path.isdir(REF_SRC):
        pytest.skip("reference sources absent (REF_SRC names their src/ directory)")
    with tempfile.TemporaryDirectory() as d:
        ours = _ours(d)
        ref = _offsets(d, "ref", '#include "mc.h"', "p_noise0", "nobs_p0", ["-I", REF_SRC])
    assert ours == ref
