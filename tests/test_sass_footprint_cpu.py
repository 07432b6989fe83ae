"""Instruction footprint of the pipelined eikonal kernel, from the compiler alone (tools/sass_footprint.py).

The kernel's warps wait on instruction fetch when its code is large, and the generic sweep (eik_core.cuh) runs on the
slow path at a few active lanes, where every local-memory access is paid in full.  So, for both instantiations of
eik_pipe_kernel:
  * no LDL/STL comes from eik_core.cuh (the sweep keeps its grid view and its reverse-propagation stack in registers);
  * the register count allows the kernel's warps per CTA (12 at CA = 64, 8 at CA = 128);
  * the SASS, callees included, stays within a budget set from the achieved size (about 16 300 instructions with
    nvcc 12.9, against 23 700 when the kernel also carried the per-lane in-place box-phase column walk and 32 944 when the
    slow path was inlined at every site) plus a margin for compiler versions.
"""
import importlib.util
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("sass_footprint", os.path.join(ROOT, "tools", "sass_footprint.py"))
sf = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(sf)

INSTRUCTION_BUDGET = 18000

pytestmark = pytest.mark.skipif(not all(sf.cuda_bin(t) for t in ("nvcc", "cuobjdump", "nvdisasm")),
                                reason="needs nvcc, cuobjdump and nvdisasm")


@pytest.fixture(scope="module")
def pipe_kernels(tmp_path_factory):
    cubin = sf.compile_cubin(ROOT, str(tmp_path_factory.mktemp("sass") / "eikonal.cubin"))
    fp = {e["mangled"]: e for e in sf.footprint(cubin) if "eik_pipe_kernel" in e["mangled"]}
    assert sorted(e["warps_per_cta"] for e in fp.values()) == [8, 12]
    return fp


def test_no_local_memory_in_generic_sweep(pipe_kernels):
    for e in pipe_kernels.values():
        assert e["local_by_file"].get("eik_core.cuh", 0) == 0, (e["kernel"], e["local_by_file"])
        assert e["stack"] == 0, e["kernel"]


def test_registers_allow_warps_per_cta(pipe_kernels):
    for e in pipe_kernels.values():
        assert e["registers"] <= e["register_limit"], (e["kernel"], e["registers"], e["register_limit"])


def test_instruction_budget(pipe_kernels):
    for e in pipe_kernels.values():
        assert e["instructions"] <= INSTRUCTION_BUDGET, (e["kernel"], e["instructions"])
