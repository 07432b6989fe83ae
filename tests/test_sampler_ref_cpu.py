"""The sampler restatement (tests/sampler_ref.py) against the unmodified reference, without a GPU.

Its random-number sources are checked first: Philox4x32-10 against the Random123 known-answer vectors, the glibc rand()
restatement against libc itself.  Then, driven by srand(seed) as the reference is, the restatement must walk both
recorded reference chains (tests/golden/replay_*.npz, oracle/replay_log.c) draw for draw: the start state, every proposal
the reference evaluated, every uniform deviate of an accept test and every decision bit for bit, and the counters the
reference printed at the end of its chain file.  One libc stream feeds every draw of the reference, so a single draw
missing or added anywhere shifts everything after it."""
import ctypes as C
import ctypes.util
import os
import re
import tempfile

import numpy as np
import pytest

from tests import inputs, replay, sampler_ref as S
from tests.util import GOLDEN

# (counter; key) -> output of philox4x32-10, the known-answer vectors of Random123 (kat_vectors)
PHILOX_KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


@pytest.mark.parametrize("ctr,key,out", PHILOX_KAT)
def test_philox_reproduces_the_known_answer_vectors(ctr, key, out):
    assert S.philox_block(ctr, key) == out


def test_philox_stream_takes_the_words_of_each_block_in_order_and_the_block_index_in_two_words():
    seed, chain = 0x1234_5678_9abc_def0, 77
    key = (seed & S.M32, seed >> 32)
    for draws in (0, 1, 5, (1 << 34) - 3):
        p = S.Philox(seed, chain, draws)
        got = [p.next31() for _ in range(9)]
        want = []
        for d in range(draws, draws + 9):
            b = d >> 2
            want.append(S.philox_block((b & S.M32, b >> 32, chain, 0x6d636d63), key)[d & 3] >> 1)
        assert got == want and p.draws == draws + 9


def _libc():
    return C.CDLL(ctypes.util.find_library("c") or "libc.so.6")


@pytest.mark.parametrize("seed", [1, 77, 78, 2**31 + 5])
def test_glibc_restatement_equals_libc_rand(seed):
    libc = _libc()
    libc.srand.argtypes = [C.c_uint]
    libc.rand.restype = C.c_int
    libc.srand(seed)
    n = 1_000_000 if seed in (77, 78) else 20_000
    want = np.fromiter((libc.rand() for _ in range(n)), np.int64, n)
    g = S.Glibc(seed)
    got = np.fromiter((g.next31() for _ in range(n)), np.int64, n)
    assert np.array_equal(got, want)


def _bits(a):
    return np.asarray(a, np.float32).view(np.uint32)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _cnt_lines(name):
    """(tested, [accepted, rejected] per arm N P V Q R M B D) from the end of the reference's chain file."""
    with open(os.path.join(GOLDEN, f"chain_ref_{name}.out")) as f:
        lines = [l for l in f if l.startswith("cnt")]
    tested = int(re.search(r"tested\s+(\d+)", lines[0]).group(1))
    ar = [tuple(int(x) for x in l.split()[-2:]) for l in lines[1:]]
    return tested, ar


# (fixture, chain seed, TRIA, evaluated proposals): the configuration of tests/test_replay_gpu.py
CHAINS = [("example2", 77, 0, 312), ("example2_tria", 78, 1, 343)]


@pytest.mark.parametrize("fixture,seed,tria,n_props", CHAINS)
def test_restatement_walks_the_recorded_reference_chain_draw_for_draw(fixture, seed, tria, n_props):
    import mcmc_eq_b200 as mq
    log = replay.load(fixture)
    with tempfile.TemporaryDirectory() as d:
        cfgp, pkp = inputs.materialise("example2", d, j_max_start=60, j_max_main=140, deci=20, true_random=seed, tria=tria)
        cfg, pk = mq.read_config(cfgp), mq.Picks.read(pkp)
    c = S.make_cfg(cfg, pk)
    rng = S.Rand(S.Glibc(seed))
    st, ok = S.init_chain(c, rng)
    assert ok
    r0 = replay.state_of(log, 0)
    assert st.dim == r0["dim"], "the start model has another dimension: a draw of the start phase is missing or extra"
    for k in ("z", "vp", "vpvs", "eq", "pres", "sres", "noise"):
        assert _same(getattr(st, k), r0[k]), k
    st.ll = replay.loglik(log["mf"][0], log["noise"][0])
    i, n_walked, n_not_evaluated = 1, 0, 0
    kinds = set()
    while st.acce < c.j_max_start + c.j_max_main:
        P = S.propose(st, c, rng)
        n_walked += 1
        if not (P.eligible and P.ok):                 # not evaluated by the reference: still consumes a uniform
            acc, _u, _a = S.decide(st, P, c, rng, None)
            assert not acc
            n_not_evaluated += 1
            continue
        assert i < len(log["u"]), "more evaluated proposals than the reference made"
        prop = replay.state_of(log, i)
        new = P.new
        assert new.dim == prop["dim"], (i, P.kind)
        for k in ("z", "vp", "vpvs", "eq", "pres", "sres", "noise"):
            assert _same(getattr(new, k), prop[k]), (i, P.kind, k)
        new_ll = replay.loglik(log["mf"][i], prop["noise"])
        acc, u, _alpha = S.decide(st, P, c, rng, new_ll)
        assert _same(u, log["u"][i]), (i, P.kind, u, log["u"][i])
        assert acc == bool(log["accepted"][i]), (i, P.kind)
        kinds.add(P.kind)
        i += 1
    assert i == len(log["u"]) == n_props + 1
    assert kinds == set("QRPVMBDN")
    tested, ar = _cnt_lines(fixture)
    assert st.counts[0] == tested == n_props
    assert [(st.counts[1 + 2 * k], st.counts[2 + 2 * k]) for k in range(8)] == ar
    assert st.counts[17] == c.j_max_start + c.j_max_main and st.counts[18] == sum(r for _a, r in ar)
    print(f"{fixture}: {n_walked} proposals walked, {n_props} evaluated and {n_not_evaluated} not, {rng.draws} libc draws")


def test_saved_state_editor_recomputes_the_checksum():
    """The chains section is read and written back through the documented record layout; an unedited blob comes back
    byte for byte, an edited one carries the sum64 of its new bytes."""
    from mcmc_eq_b200._lib import MqStateHeader, MqStateSection
    n, md, ne, ns = 3, 4, 2, 3
    nf = 9 * md + 16 * ne + 4 * ns
    rec_bytes = (S.HEAD.itemsize + 4 * nf + 7) // 8 * 8
    H = MqStateHeader(magic=b"MQSTATE", format=1, header_bytes=C.sizeof(MqStateHeader), n_chains=n, max_dim=md, n_events=ne,
                      n_stations=ns, seed=5, n_sections=1)
    off = C.sizeof(MqStateHeader) + C.sizeof(MqStateSection)
    sec = MqStateSection(id=1, offset=off, bytes=n * rec_bytes)
    payload = np.random.default_rng(0).integers(0, 255, n * rec_bytes, dtype=np.uint8).tobytes()
    body = bytes(H) + bytes(sec) + payload
    blob = body + S.sum64(body).to_bytes(8, "little")
    s = S.SavedState(blob)
    assert s.edited() == blob
    s.head["draws"][1] = (1 << 34) - 2
    s.z[2, 1] = 7.5
    out = S.SavedState(s.edited())
    assert int(out.head["draws"][1]) == (1 << 34) - 2 and out.z[2, 1] == 7.5
    raw = out.edited()
    assert int.from_bytes(raw[-8:], "little") == S.sum64(raw[:-8]) != S.sum64(blob[:-8])
