"""Head-wave reverse propagation at depth, on the host builds of the solver (no GPU).

The reference re-times the lines behind a head wave by recursion without a limit (src/time_2d.c:1128-1143; the oracle's
sweep_line).  eik::sweep_line (csrc/eik_core.cuh) unrolls that recursion into a stack of kMaxReverseDepth frames held in
a shift register, and a head wave that would open one frame more is dropped with status kErrReverseDepth (-30).

tests/golden/deep_nesting.npz (tools/nesting_search.py) holds the most deeply nesting columns a hill-climb found, inside
the shipped priors and without them.  Real columns nest only a few frames deep, so most of the stack never runs at the
library's bound of 12.  Here the solver is also built with a lowered bound B (-DEIK_MAX_REVERSE_DEPTH=B, into a temporary
directory), so that on the same columns every frame, every shift of the register and the overflow are exercised:
  * where the oracle nests at most B frames deep the B build must give the bits of the full build, status 0, and its
    event counts (line sweeps, reverse sweeps, head waves), which pin which lines were re-timed and how often;
  * where it nests deeper: status -30 exactly.
The FP32 solver is not bit-identical to the oracle (the oracle keeps the reference's double sqrt, so an adoption by one
ulp can differ and with it a re-timed line more or less); against the oracle the bound is level 1,
|dT| <= max(1e-4 s, 2e-6 T) (SURVEY.md Appendix A.5)."""
import ctypes as C
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from tests import util
from tests.util import fp, ptr

ip = C.POINTER(C.c_int)
ERR_REVERSE_DEPTH = -30
LIB_BOUND = 12
MODES = {0: "per-lane columns", 1: "global-memory slices", 2: "lock-step columns"}


def fixture_columns():
    """[(search, depth, plane (nx, nz), slowness column, oracle's nesting per source depth)] of deep_nesting.npz."""
    d = np.load(os.path.join(util.GOLDEN, "deep_nesting.npz"))
    out = []
    for i, m in enumerate(d["meta"]):
        search, k = m.split("|")[:2]
        pl = d[f"plane_{i}"]
        out.append((search, int(k), (int(pl[0]), int(pl[1])), d[f"slow_{i}"], d[f"depth_{i}"].astype(int)))
    return out


COLUMNS = fixture_columns()
WORST = max(int(c[4].max()) for c in COLUMNS)
BOUNDS = sorted(set(range(1, 4)) | set(range(1, min(WORST, LIB_BOUND) + 1)))


def _compile(src, bound, out, extra=()):
    cmd = ["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", "-Wno-unused-but-set-variable",
           *extra, src, "-o", out]
    if bound is not None:
        cmd.insert(1, f"-DEIK_MAX_REVERSE_DEPTH={bound}")
    subprocess.run(cmd, check=True)
    return out


def _load(so, mt):
    L = C.CDLL(so)
    if mt:
        L.emu_mt_time_2d.argtypes = [fp, C.c_int, C.c_int, ip, fp, ip, C.c_int, fp, ip, C.c_int, C.c_int]
        L.emu_mt_set_fill.argtypes = [C.c_float]
        L.emu_mt_set_fill(float("nan"))
    else:
        L.emu_time_2d.argtypes = [fp, C.c_int, C.c_int, C.c_int, fp, ip]
    return L


@pytest.fixture(scope="module")
def builds(tmp_path_factory):
    """{bound: (one-lane library, warp-of-8-threads library)}: the library's bound (None: the macro left undefined) and
    every lowered bound, compiled from tests/emu into a temporary directory."""
    d = tmp_path_factory.mktemp("emu_bounds")
    emu = os.path.join(util.ROOT, "tests", "emu")
    jobs = {}
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 2) as ex:
        for b in [None] + BOUNDS:
            tag = "lib" if b is None else str(b)
            jobs[b] = (ex.submit(_compile, os.path.join(emu, "eik_emu.cpp"), b, str(d / f"emu_{tag}.so")),
                       ex.submit(_compile, os.path.join(emu, "eik_emu_mt.cpp"), b, str(d / f"emu_mt_{tag}.so"), ("-pthread",)))
        return {b: (_load(f1.result(), False), _load(f2.result(), True)) for b, (f1, f2) in jobs.items()}


def _oracle(s, nx, iz):
    st = util.PlStats()
    t, rc = util.oracle_time_2d(s, nx, iz, C.byref(st))
    assert rc == 0
    return t, st


def _one_lane(L, s, nx, iz):
    s = util.f32(s)
    t = np.zeros((nx, len(s)), np.float32)
    cnt = np.zeros(7, np.int32)
    rc = L.emu_time_2d(ptr(s), nx, len(s), iz, ptr(t), cnt.ctypes.data_as(ip))
    return t, rc, cnt


def _warp(L, cases, nx, nz, mode):
    """cases: [(column, iz)], at most one per lane of the warp -> fields [lanes, nx, nz], status [lanes]."""
    W = L.emu_mt_lanes()
    assert len(cases) <= W
    S = np.zeros((W, nz), np.float32)
    izs = np.full(W, -1, np.int32)
    for l, (s, iz) in enumerate(cases):
        S[l], izs[l] = s, iz
    rows = np.array([0, nz - 1], np.int32)
    full = np.full((W, nx, nz), -1, np.float32)
    ro = np.zeros((W, len(rows), nx), np.float32)
    st = np.zeros(W, np.int32)
    L.emu_mt_time_2d(ptr(S), nx, nz, izs.ctypes.data_as(ip), ptr(full), rows.ctypes.data_as(ip), len(rows), ptr(ro),
                     st.ctypes.data_as(ip), mode, 0)
    assert L.emu_mt_site_mismatches() == 0
    return full, st


@pytest.fixture(scope="module")
def reference():
    """Per fixture column and source depth: the oracle's field and its nesting."""
    out = []
    for search, k, (nx, nz), s, depth in COLUMNS:
        per = []
        for iz in range(nz):
            t, st = _oracle(s, nx, iz)
            per.append((t, int(st.max_rev_depth)))
        out.append(per)
    return out


def test_fixture_still_reaches_its_depths(reference):
    """Every column of the fixture nests, source depth by source depth, as deep as the search recorded, and the column saved
    for depth k reaches k: the file cannot go stale while the oracle changes under it."""
    assert {"admissible", "unconstrained"} <= {c[0] for c in COLUMNS}
    for (search, k, (nx, nz), s, depth), per in zip(COLUMNS, reference):
        assert len(s) == nz and depth.shape == (nz,)
        assert [p[1] for p in per] == list(depth), (search, k)
        assert int(depth.max()) >= k and (depth == k).any(), (search, k)
    for k in range(2, WORST + 1):
        assert any(c[1] == k for c in COLUMNS), k
    print(f"\nfixture: {len(COLUMNS)} columns, worst nesting {WORST}")


def test_counter_reads_zero_without_head_waves_and_counts_a_low_velocity_zone(oracle):
    g = util.EXAMPLE_GRID
    nx, nz, h = util.nxmod_of(g), g["nz"], g["h"]
    flat = np.full(nz, h / 6.0, np.float32)
    assert all(_oracle(flat, nx, iz)[1].max_rev_depth == 0 for iz in range(nz))
    # 6 km/s over a 3 km/s channel over 8 km/s: head waves along both interfaces of the channel
    lvz = np.full(nz, h / 8.0, np.float32)
    lvz[:20] = h / 6.0
    lvz[20:30] = h / 3.0
    depth = [_oracle(lvz, nx, iz)[1].max_rev_depth for iz in range(nz)]
    assert max(depth) >= 1, depth


@pytest.mark.parametrize("idx", range(len(COLUMNS)), ids=[f"{c[0]}-{c[1]}" for c in COLUMNS])
def test_library_bound_against_the_oracle(builds, reference, idx):
    """With the library's bound, every source depth of every fixture column: level 1 of the oracle and status 0; the warp
    of eight host threads in all three modes gives the one-lane build's bits."""
    search, k, (nx, nz), s, depth = COLUMNS[idx]
    one, warp = builds[None]
    fields = []
    for iz in range(nz):
        tref, dep = reference[idx][iz]
        assert dep <= LIB_BOUND
        t, rc, cnt = _one_lane(one, s, nx, iz)
        assert rc == 0, (search, k, iz, rc)
        assert (np.abs(t - tref) <= util.eikonal_tol(tref)).all(), (search, k, iz, float(np.abs(t - tref).max()))
        fields.append(t)
    W = warp.emu_mt_lanes()
    for mode in MODES:
        for iz0 in range(0, nz, W):
            izs = list(range(iz0, min(nz, iz0 + W)))
            full, st = _warp(warp, [(s, iz) for iz in izs], nx, nz, mode)
            for l, iz in enumerate(izs):
                assert st[l] == 0, (search, k, MODES[mode], iz, st[l])
                assert np.array_equal(full[l].view(np.uint32), fields[iz].view(np.uint32)), (search, k, MODES[mode], iz)


@pytest.mark.parametrize("bound", BOUNDS)
def test_lowered_bound_runs_every_frame_and_its_overflow(builds, reference, bound):
    """Stack of `bound` frames: solves that nest at most that deep are the full build's bits with its event counts (every
    frame up to the top one runs, and the top one is shifted in and out), solves that nest deeper fail with -30 -- in the
    one-lane build and in the warp of eight host threads (global-memory slices, lock-step columns), where a lane that
    overflows sits next to lanes that do not.  The warp builds may get through a solve that overflows the one-lane core
    (they meet fewer nested head waves in the generic sweep), never the other way round."""
    one, warp = builds[bound]
    full_one = builds[None][0]
    W = warp.emu_mt_lanes()
    n_exact = n_shallower = n_over = n_warp_over = 0
    for idx, (search, k, (nx, nz), s, depth) in enumerate(COLUMNS):
        want = {}
        for iz in range(nz):
            tref, dep = reference[idx][iz]
            t, rc, cnt = _one_lane(one, s, nx, iz)
            if dep <= bound:
                t_lib, _, cnt_lib = _one_lane(full_one, s, nx, iz)
                assert rc == 0, (bound, search, k, iz, dep, rc)
                assert np.array_equal(t.view(np.uint32), t_lib.view(np.uint32)), (bound, search, k, iz, dep)
                assert np.array_equal(cnt, cnt_lib), (bound, search, k, iz, dep, cnt, cnt_lib)
                want[iz] = (0, t_lib)
                n_exact += dep == bound
                n_shallower += dep < bound
            else:
                assert rc == ERR_REVERSE_DEPTH, (bound, search, k, iz, dep, rc)
                want[iz] = (ERR_REVERSE_DEPTH, None)
                n_over += 1
        for mode in (1, 2):
            for iz0 in range(0, nz, W):
                izs = list(range(iz0, min(nz, iz0 + W)))
                full, st = _warp(warp, [(s, iz) for iz in izs], nx, nz, mode)
                for l, iz in enumerate(izs):
                    rc, t_lib = want[iz]
                    if rc == ERR_REVERSE_DEPTH:
                        # the warp solver enters the generic sweep only on the lines its own sweeps hand over, so it can
                        # get through a solve that overflows the one-lane core; then it must still give the full bits
                        assert st[l] in (0, ERR_REVERSE_DEPTH), (bound, search, k, MODES[mode], iz, st[l])
                        n_warp_over += st[l] == ERR_REVERSE_DEPTH
                        if st[l] == 0:
                            t_lib = _one_lane(full_one, s, nx, iz)[0]
                        else:
                            continue
                    else:
                        assert st[l] == 0, (bound, search, k, MODES[mode], iz, st[l])
                    assert np.array_equal(full[l].view(np.uint32), t_lib.view(np.uint32)), (bound, search, k, MODES[mode], iz)
    print(f"\nbound {bound}: {n_exact} solves exactly {bound} deep (bits), {n_shallower} shallower (bits), "
          f"{n_over} deeper (status -30; the warp builds: {n_warp_over} of {2 * n_over})")
    assert n_exact > 0, "no fixture solve fills the stack"
    if bound < WORST:
        assert n_over > 0, "no fixture solve overflows the stack"
