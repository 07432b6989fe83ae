"""Host restatement of the sampler's arithmetic (TEST INFRASTRUCTURE ONLY): the start models, every proposal arm and the
accept decision of src/mcmc_eq.c, as csrc/chain.cu states them, in float32 / float64 with the device's operation order.

One restatement, two sources of random numbers:
  Glibc(seed)                   libc rand() after srand(seed): drives the reference, so the restatement must reproduce the
                                recorded reference chains (tests/golden/replay_*.npz, chain_ref_*.out) draw for draw;
  Philox(seed, chain, draws)    the device's counter-based stream (chain.cu: struct Philox): drives the library, so the
                                restatement must reproduce what the device does from any saved state.

Float32 arithmetic is done on Python floats rounded with f32() after every operation: a sum, difference, product or
quotient of two float32 values computed in double and rounded once to float32 is the float32 result (double carries more
than 2 x 24 + 2 bits).  model_valid, find_in_cell / find_neighbor, the log_fac expressions and nexp come from the CPU
oracle (oracle/chain.c, oracle/fwd_model.c), which is pinned to the reference separately (tests/test_oracle_pin.py).

The device's double log() is not correctly rounded, glibc's is (to the last bit in practice): a Gaussian deviate whose
double value lies within 2^-52 of a float32 rounding boundary can round the other way on the device.  gauss() notes
every such deviate (Rand.fragile); a caller that sees a one-ulp difference can redo the prediction with that deviate
rounded the other way (Rand.flip) and so tell this case from a real one."""
from __future__ import annotations

import ctypes as C
import math
import struct
from dataclasses import dataclass, field

import numpy as np

from tests import util
from tests.util import ptr, f32 as f32a

_F = struct.Struct("<f")
M32 = 0xFFFFFFFF
MAX_TRIES = 100000          # chain.cu: kMaxTries, and the give-up bound of gauss_bounded


def f32(x: float) -> float:
    """x rounded to float32 (round to nearest even), as a Python float."""
    return _F.unpack(_F.pack(x))[0]


def ulp_step(x: float, up: bool) -> float:
    """The float32 neighbour of float32 x towards +inf (up) or -inf."""
    b = struct.unpack("<I", _F.pack(x))[0]
    if x == 0.0:
        b = 1 if up else 0x80000001
    elif (x > 0) == up:
        b += 1
    else:
        b -= 1
    return struct.unpack("<f", struct.pack("<I", b & M32))[0]


# ---- random-number sources: next31() -> 31 random bits --------------------------------------------------------------

class Glibc:
    """glibc random() / rand() with the default TYPE_3 state (degree 31, separation 3) after srand(seed): the seeding
    LCG 16807 mod 2^31 - 1 in Schrage's form, 310 discarded outputs, then r[i] = r[i-31] + r[i-3] mod 2^32, output >> 1."""

    def __init__(self, seed: int):
        seed &= M32
        if seed == 0:
            seed = 1
        word = seed - (1 << 32) if seed & 0x80000000 else seed      # int32_t word = seed
        r = [word & M32]
        for _ in range(30):
            hi = int(word / 127773)                                  # C division truncates towards zero
            lo = word - hi * 127773
            word = 16807 * lo - 2836 * hi
            if word < 0:
                word += 2147483647
            r.append(word & M32)
        self.r = r                                                   # the 31 state words
        self.f, self.b = 3, 0                                        # front and rear of the additive generator
        self.draws = 0
        for _ in range(310):
            self._step()
        self.draws = 0

    def _step(self) -> int:
        r = self.r
        v = (r[self.f] + r[self.b]) & M32
        r[self.f] = v
        self.f = (self.f + 1) % 31
        self.b = (self.b + 1) % 31
        return v >> 1

    def next31(self) -> int:
        self.draws += 1
        return self._step()


def philox_block(ctr, key):
    """Philox4x32-10 of chain.cu (Philox::block): counter words c0..c3, key k0, k1 -> four output words."""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for _ in range(10):
        p0 = 0xD2511F53 * c0
        p1 = 0xCD9E8D57 * c2
        c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & M32, p1 & M32, ((p0 >> 32) ^ c3 ^ k1) & M32, p0 & M32
        k0 = (k0 + 0x9E3779B9) & M32
        k1 = (k1 + 0xBB67AE85) & M32
    return (c0, c1, c2, c3)


class Philox:
    """The stream of device chain `chain` (= chain offset + index in the handle) under `seed`, from word `draws` on:
    key (seed low, seed high), counter (block low, block high, chain, 0x6d636d63), word out[draws & 3] of block draws >> 2."""

    def __init__(self, seed: int, chain: int, draws: int = 0):
        self.key = (seed & M32, (seed >> 32) & M32)
        self.chain = chain & M32
        self.draws = draws
        self._set_block(draws >> 2)

    def _set_block(self, b: int):
        self.out = philox_block((b & M32, (b >> 32) & M32, self.chain, 0x6d636d63), self.key)

    def next31(self) -> int:
        w = self.out[self.draws & 3]
        self.draws += 1
        if (self.draws & 3) == 0:
            self._set_block(self.draws >> 2)
        return w >> 1


# ---- the rand_* helpers (src/mcmc_eq.c:122-178, chain.cu: Philox::uniform ... gauss_bounded) ------------------------

class Rand:
    """uniform / below / between / gauss / gauss_bounded over a source."""

    def __init__(self, src, flip=()):
        self.src = src
        self.n_gauss = 0          # gauss() calls so far
        self.fragile = []         # indices of the deviates within 2^-52 of a float rounding boundary
        self.flip = set(flip)     # indices of the deviates to round the other way

    @property
    def draws(self) -> int:
        return self.src.draws

    def next31(self) -> int:
        return self.src.next31()

    def uniform(self) -> float:              # (float)rand() / RAND_MAX in float: RAND_MAX rounds to 2^31
        return f32(f32(float(self.src.next31())) / 2147483648.0)

    def below(self, n: int) -> int:          # rand_eq_int, clamped to n - 1
        i = int(f32(self.uniform() * float(n)))
        return i if i < n else n - 1

    def between(self, lo: float, hi: float) -> float:
        return f32(lo + f32(f32(f32(hi - lo) * f32(float(self.src.next31()))) / 2147483648.0))

    def gauss(self) -> float:
        while True:
            v1 = f32(f32(2.0 * self.uniform()) - 1.0)
            v2 = f32(f32(2.0 * self.uniform()) - 1.0)
            s = f32(f32(v1 * v1) + f32(v2 * v2))
            if s < 1.0:
                break
        k = self.n_gauss
        self.n_gauss += 1
        if s == 0.0:
            return 0.0
        g = v1 * math.sqrt(-2.0 * math.log(s) / s)
        r = f32(g)
        # the two float32 values around g and the midpoint between them: a device log one ulp off can cross it
        other = ulp_step(r, g > r) if g != r else r
        mid = (r + other) / 2.0
        if g != r and abs(g - mid) <= 2.0 ** -52 * abs(g):
            self.fragile.append(k)
            if k in self.flip:
                r = other
        return r

    def gauss_bounded(self, v0: float, sdev: float, lo: float, hi: float):
        """-> (dv, ok): the first dv = gauss * sdev with lo < v0 + dv < hi; (0, False) after 10^5 tries."""
        for _ in range(MAX_TRIES):
            dv = f32(self.gauss() * sdev)
            x = f32(v0 + dv)
            if lo < x < hi:
                return dv, True
        return 0.0, False


# ---- configuration -------------------------------------------------------------------------------------------------

class Cfg:
    """The configuration fields the sampler reads (plain Python numbers, float32-exact) and the handle's derived values
    (capi.cu: mq_create): md, xmin .. zmax, lvz_flag, inv0 (the start inv_control), revert, the balanced proposal strings,
    n_class and fix (the picks' fixed hypocentre components, -9999 = free).  Picklable, for worker processes."""

    def __init__(self, cfg, picks):
        import types
        for name, _t in type(cfg)._fields_:
            v = getattr(cfg, name)
            if name == "grid":
                v = types.SimpleNamespace(**{k: getattr(v, k) for k, _ in type(v)._fields_})
            elif isinstance(v, bytes):
                v = v.decode()
            setattr(self, name, v)
        self.n_class = np.ascontiguousarray(picks.n_class, np.int32)
        self.fix = np.asarray(picks.fix, np.float64).reshape(-1, 3)
        self.ne, self.ns = int(picks.n_events), int(picks.n_stations)


def balance(letters: str, noq: int, nos: int, per: int) -> str:
    """Balanced proposal string (src/mcmc_eq.c:769-834, chain.cu: balance): Q and R once per `per` events / stations."""
    out = []
    for q in letters:
        if q == "Q":
            out += ["Q"] * len(range(0, noq, per))
        elif q == "R":
            out += ["R"] * len(range(0, nos, per))
        elif q in "NMVPBD":
            out.append(q)
    return "".join(out)


def make_cfg(cfg, picks) -> Cfg:
    g = cfg.grid
    c = Cfg(cfg, picks)
    c.md = min(cfg.max_dim, 1000)
    c.xmin, c.xmax = g.x0, f32(g.x0 + f32((g.nx - 1) * g.h))
    c.ymin, c.ymax = g.y0, f32(g.y0 + f32((g.ny - 1) * g.h))
    c.zmin, c.zmax = g.z0, f32(g.z0 + f32((g.nz - 1) * g.h))
    c.lvz_flag = 1 if cfg.inv_control > 0 else 0
    c.inv0 = -cfg.inv_control if cfg.inv_control > 0 else cfg.inv_control
    c.revert = int(cfg.j_max_start + cfg.j_max_main // 2)                       # src/mcmc_eq.c:840
    c.ps_start = balance(c.dstring_start, c.ne, c.ns, 10)
    c.ps_main = balance(c.dstring_main, c.ne, c.ns, 20)
    return c


# ---- the oracle's pieces -------------------------------------------------------------------------------------------

def _fa(a) -> np.ndarray:
    return f32a(a)


def model_valid(dim, z, vp, vpvs, cfg: Cfg, inv: float) -> bool:
    L = util.oracle()
    return L.ch_model_valid(dim, ptr(_fa(z)), ptr(_fa(vp)), ptr(_fa(vpvs)), cfg.grid.h, cfg.zmin, cfg.zmax, inv) == 0


def find_in_cell(z, dim, zq) -> int:
    return util.oracle().fm_find_in_cell(ptr(_fa(z)), dim, zq)


def find_neighbor(z, dim, n) -> int:
    return util.oracle().fm_find_neighbor_cell(ptr(_fa(z)), dim, n)


# ---- chain state -------------------------------------------------------------------------------------------------

@dataclass
class State:
    """One chain: the current model (lists of float32-exact floats), hypocentres [ne][3], station corrections, sigmas,
    and the sampler's bookkeeping."""
    dim: int
    z: list
    vp: list
    vpvs: list
    eq: list
    pres: list
    sres: list
    noise: list
    inv: float
    acce: int = 0
    reject: int = 0
    counts: list = field(default_factory=lambda: [0] * 20)
    draws: int = 0
    ll: float = 0.0
    mf: list = field(default_factory=lambda: [0.0] * 8)

    def copy(self) -> "State":
        return State(self.dim, list(self.z), list(self.vp), list(self.vpvs), [list(q) for q in self.eq], list(self.pres),
                     list(self.sres), list(self.noise), self.inv, self.acce, self.reject, list(self.counts), self.draws, self.ll,
                     list(self.mf))


# ---- start models (src/mcmc_eq.c:559-630, chain.cu: init_chains_kernel) ---------------------------------------------

def init_chain(cfg: Cfg, rng: Rand) -> tuple[State, bool]:
    """-> (start state, ok); ok is False when a start value could not be drawn inside its bounds."""
    g = cfg
    ok = True
    inv = cfg.inv0

    def gb(*a):
        nonlocal ok
        dv, good = rng.gauss_bounded(*a)
        ok = ok and good
        return dv

    dim = 1
    z, vp, vpvs = [], [], []
    for _attempt in range(MAX_TRIES):
        if g.start_cell_number > 1:
            dim = g.start_cell_number + int(gb(float(g.start_cell_number), float(g.sdev_start_cell_number), 1.0, float(g.grid.nz)))
        else:
            dim = 1
        if dim < 1:
            dim = 1
        first = 0
        z = z[:2] if g.tria == 1 else []
        if g.tria == 1:     # two fixed nuclei at the top and the bottom of the model (src/mcmc_eq.c:577-588)
            dim += 2
            first = 2
            z = [g.zmin, g.zmax]
            vp, vpvs = [0.0, 0.0], [0.0, 0.0]
            for i in range(2):
                value = f32(g.start_vp + f32(f32(z[i] - g.grid.z0) * g.start_vp_grad))
                vp[i] = f32(value + gb(value, g.sdev_start_vp, g.vpmin, g.vpmax))
                vpvs[i] = f32(g.start_vpvs + gb(g.start_vpvs, g.sdev_start_vpvs, g.vpvsmin, g.vpvsmax))
        else:
            vp, vpvs = [], []
        if dim > g.md:
            dim = g.md
        for i in range(first, dim):
            z.append(rng.between(g.zmin, g.zmax))
        for i in range(first, dim):
            value = f32(g.start_vp + f32(f32(z[i] - g.grid.z0) * g.start_vp_grad))
            vp.append(f32(value + gb(value, g.sdev_start_vp, g.vpmin, g.vpmax)))
            vpvs.append(f32(g.start_vpvs + gb(g.start_vpvs, g.sdev_start_vpvs, g.vpvsmin, g.vpvsmax)))
        if model_valid(dim, z, vp, vpvs, cfg, inv):
            break
    z, vp, vpvs = z[:dim], vp[:dim], vpvs[:dim]
    hx = f32(f32(g.xmax - g.xmin) / 2.0)
    hy = f32(f32(g.ymax - g.ymin) / 2.0)
    eq = [[0.0, 0.0, 0.0] for _ in range(g.ne)]
    lo, hi = f32(g.xmin + f32(hx * f32(1.0 - g.r_start_eqh))), f32(g.xmin + f32(hx * f32(1.0 + g.r_start_eqh)))
    for q in range(g.ne):
        eq[q][0] = rng.between(lo, hi)
    lo, hi = f32(g.ymin + f32(hy * f32(1.0 - g.r_start_eqh))), f32(g.ymin + f32(hy * f32(1.0 + g.r_start_eqh)))
    for q in range(g.ne):
        eq[q][1] = rng.between(lo, hi)
    zhi = f32(g.zmax * g.r_start_eqv)
    for q in range(g.ne):
        eq[q][2] = rng.between(g.zmin, zhi)
    for q in range(g.ne):
        for k in range(3):
            if g.fix[q, k] != -9999.0:
                eq[q][k] = f32(float(g.fix[q, k]))
    pres = [f32(g.start_delay + gb(g.start_delay, g.sdev_start_delay, g.residual_min, g.residual_max)) for _ in range(g.ns)]
    sres = [f32(g.start_delay + gb(g.start_delay, g.sdev_start_delay, g.residual_min, g.residual_max)) for _ in range(g.ns)]
    if g.scor_flag in (1, 2):
        pres[g.reference_station] = g.ref_statcor_P
    if g.scor_flag == 2:
        sres[g.reference_station] = g.ref_statcor_S
    st = State(dim, z, vp, vpvs, eq, pres, sres, [g.start_noise] * 8, inv)
    st.draws = rng.draws
    return st, ok


# ---- one proposal (src/mcmc_eq.c:845-1130, chain.cu: propose_kernel) ------------------------------------------------

@dataclass
class Proposal:
    kind: str             # the arm, '' for a finished chain
    eligible: bool = True
    ok: bool = True       # False: a retry loop gave up
    new: State = None     # the chain with the proposal applied (None: nothing to apply)
    log_fac: float = 0.0
    q_idx: int = -1       # Q: the event moved; R: the station


def propose(st: State, cfg: Cfg, rng: Rand, override: str | None = None) -> Proposal:
    """The proposal of the chain in state `st`; st.inv takes the LVZ switch (Q1) in place."""
    g = cfg
    j = st.acce
    if j >= g.j_max_start + g.j_max_main:             # finished chain (src/mcmc_eq.c:845): draws nothing
        return Proposal("", eligible=False)
    if j == g.revert and g.lvz_flag == 1:            # Q1: on every iteration while acce == revert (:849-853)
        st.inv = -st.inv
    inv = st.inv
    if override:
        kind = override[rng.below(len(override))]
        fac = g.epi_search if j <= g.j_max_start else 1.0
    elif j <= g.j_max_start:
        kind = g.ps_start[rng.below(len(g.ps_start))]
        fac = g.epi_search
    else:
        kind = g.ps_main[rng.below(len(g.ps_main))]
        fac = 1.0
    P = Proposal(kind)
    ok = True

    def gb(*a):
        nonlocal ok
        dv, good = rng.gauss_bounded(*a)
        ok = ok and good
        return dv

    dim, z, vp, vpvs = st.dim, st.z, st.vp, st.vpvs
    new = st.copy()
    if kind == "Q":
        idx = rng.below(g.ne)
        q = st.eq[idx]
        dx = gb(q[0], f32(g.sdevxs * fac), g.xmin, g.xmax)
        dy = gb(q[1], f32(g.sdevys * fac), g.ymin, g.ymax)
        dz = gb(q[2], f32(g.sdevzs * fac), g.zmin, g.zmax)
        d = [dx, dy, dz]
        for k in range(3):
            if g.fix[idx, k] != -9999.0:
                d[k] = 0.0
        new.eq[idx] = [f32(q[k] + d[k]) for k in range(3)]
        P.q_idx = idx
    elif kind == "R":
        idx = rng.below(g.ns)
        dx = gb(st.pres[idx], g.sdevresidual, g.residual_min, g.residual_max)
        dy = gb(st.sres[idx], g.sdevresidual, g.residual_min, g.residual_max)
        if g.scor_flag == -1:
            dy = 0.0
        if g.scor_flag == -2:
            dx = 0.0
        dx2 = dy2 = 0.0
        if g.scor_flag != 0:      # second addition of the reference (:919-928): for flags -1 / -2 dx is applied twice (Q4)
            dx2, dy2 = dx, dy
            if g.reference_station == idx:
                if g.scor_flag == 1:
                    dx2 = 0.0
                if g.scor_flag == 2:
                    dx2 = dy2 = 0.0
        nsm1 = float(g.ns - 1)
        if g.scor_flag <= 0:      # zero-mean compensation over the other stations (:905-915)
            for k in range(g.ns):
                if k == idx:
                    new.pres[k] = f32(st.pres[k] + dx)
                    new.sres[k] = f32(st.sres[k] + dy)
                else:
                    new.pres[k] = f32(st.pres[k] - f32(dx / nsm1))
                    new.sres[k] = f32(st.sres[k] - f32(dy / nsm1))
        if g.scor_flag != 0:
            new.pres[idx] = f32(new.pres[idx] + dx2)
            new.sres[idx] = f32(new.sres[idx] + dy2)
        P.q_idx = idx
    elif kind in "PVM":
        fixed = 2 if g.tria == 1 else 0          # the two end nuclei of TRIA = 1 are never moved (:990-998)
        if kind == "M" and not (dim > 1 + fixed):
            P.eligible = False
            return P
        for _t in range(MAX_TRIES):
            nz_, nvp, nvs = list(z), list(vp), list(vpvs)
            idx = fixed + rng.below(dim - fixed) if kind == "M" else rng.below(dim)
            if kind == "P":
                nvp[idx] = f32(vp[idx] + gb(vp[idx], g.sdevvp, g.vpmin, g.vpmax))
            elif kind == "V":
                nvs[idx] = f32(vpvs[idx] + gb(vpvs[idx], g.sdevvpvs, g.vpvsmin, g.vpvsmax))
            else:
                nz_[idx] = f32(z[idx] + gb(z[idx], g.sdevz, g.zmin, g.zmax))
            if model_valid(dim, nz_, nvp, nvs, cfg, inv):
                break
        else:
            ok = False
        new.z, new.vp, new.vpvs = nz_, nvp, nvs
    elif kind == "B":
        if not ((dim + 1) < (g.max_dim / (1.0 + math.sqrt(f32(inv * inv))))) or dim + 1 > g.md:
            P.eligible = False
            return P
        for _t in range(MAX_TRIES):
            newz = rng.between(g.zmin, g.zmax)
            idx = find_in_cell(z, dim, newz)
            dvp = gb(vp[idx], g.sdevvp, g.vpmin, g.vpmax)
            dvs = gb(vpvs[idx], g.sdevvpvs, g.vpvsmin, g.vpvsmax)
            nz_, nvp, nvs = list(z) + [newz], list(vp) + [f32(vp[idx] + dvp)], list(vpvs) + [f32(vpvs[idx] + dvs)]
            if model_valid(dim + 1, nz_, nvp, nvs, cfg, inv):
                break
        else:
            ok = False
        L = util.oracle()
        P.log_fac = L.ch_logfac_birth(g.sdevvp, g.vpmin, g.vpmax, nvp[dim], vp[idx], g.sdevvpvs, g.vpvsmin, g.vpvsmax,
                                      nvs[dim], vpvs[idx])
        new.dim, new.z, new.vp, new.vpvs = dim + 1, nz_, nvp, nvs
    elif kind == "D":
        fixed = 2 if g.tria == 1 else 0          # ... nor removed (:1059-1067)
        if not (dim > 1 + fixed):
            P.eligible = False
            return P
        L = util.oracle()
        for _t in range(MAX_TRIES):
            dead = fixed + rng.below(dim - fixed)
            nb = find_neighbor(z, dim, dead)
            lf = L.ch_logfac_death(g.sdevvp, g.vpmin, g.vpmax, vp[dead], vp[nb], g.sdevvpvs, g.vpvsmin, g.vpvsmax,
                                   vpvs[dead], vpvs[nb])
            keep = [i for i in range(dim) if i != dead]
            nz_, nvp, nvs = [z[i] for i in keep], [vp[i] for i in keep], [vpvs[i] for i in keep]
            if model_valid(dim - 1, nz_, nvp, nvs, cfg, inv):
                break
        else:
            ok = False
        P.log_fac = lf
        new.dim, new.z, new.vp, new.vpvs = dim - 1, nz_, nvp, nvs
    elif kind == "N":
        o = st.noise
        nn = [f32(o[k] + gb(o[k], g.sdevn, g.noise_min, g.noise_max)) for k in range(8)]   # p0 s0 p1 s1 ... (:1097-1112)
        P.log_fac = util.oracle().ch_logfac_noise(ptr(cfg.n_class, util.ip), ptr(_fa(o)), ptr(_fa(nn)))
        new.noise = nn
    P.ok = ok
    P.new = new
    return P


SLOT = {"N": 0, "P": 1, "V": 2, "Q": 3, "R": 4, "M": 5, "B": 6, "D": 7}


def alpha_of(log_fac: float, new_ll: float, old_ll: float) -> float:
    return util.oracle().ch_alpha(log_fac, new_ll, old_ll)


def loglik(mf, noise) -> float:
    return -util.oracle().ch_misfit(ptr(_fa(mf)), ptr(_fa(noise))) / 2.0


def decide(st: State, P: Proposal, cfg: Cfg, rng: Rand, new_ll: float | None, beta: float = 1.0, u: float | None = None):
    """The accept test (src/mcmc_eq.c:1135-1164, chain.cu: accept_kernel) -> (accepted, u, alpha); updates st's
    acce / reject / counts in place and, when accepted, its model, hypocentres, corrections and sigmas.  new_ll: the
    proposal's log-likelihood (ignored under aflag = 1, or for a proposal that is not evaluated).  beta: the chain's
    inverse temperature, on both likelihoods and, for N only, on log_fac.  u: a recorded deviate instead of a draw."""
    if not P.kind:
        return None, None, None
    g = cfg
    slot = SLOT[P.kind]
    evaluated = P.eligible and P.ok
    if evaluated:
        st.counts[0] += 1                           # nmod: models whose misfit was evaluated
        nl = 0.0 if g.aflag == 1 else new_ll
        lf = beta * P.log_fac if P.kind == "N" else P.log_fac
        alpha = alpha_of(lf, beta * nl, beta * st.ll)
    else:
        alpha = 0.0
    if g.aflag == 1:
        alpha = 1.0                                 # prior sampling; also an ineligible M / B / D (:1137-1141), unverified
    if not P.eligible and g.aflag == 0:
        alpha = 0.0                                 # Q5: rejected, and still consumes its uniform
    if not P.ok:
        alpha = 0.0                                 # a retry loop that gave up is rejected under every aflag
    if u is None:
        u = rng.uniform()
    if u < alpha:
        st.acce += 1
        st.counts[1 + 2 * slot] += 1
        st.counts[17] += 1
        if P.new is not None:
            n = P.new
            st.dim, st.z, st.vp, st.vpvs = n.dim, n.z, n.vp, n.vpvs
            st.eq, st.pres, st.sres, st.noise = n.eq, n.pres, n.sres, n.noise
        if evaluated:
            st.ll = 0.0 if g.aflag == 1 else new_ll
        return True, u, alpha
    st.reject += 1
    st.counts[2 + 2 * slot] += 1
    st.counts[18] += 1
    return False, u, alpha


# ---- saved states (state.cu, include/mcmceq_b200.h) ---------------------------------------------------------------

HEAD = np.dtype([("ll", "<f8"), ("rms", "<f8"), ("misfit", "<f8"), ("best_rms", "<f8"), ("best_snap_rms", "<f8"),
                 ("acce", "<i8"), ("reject", "<i8"), ("best_number", "<i8"), ("draws", "<u8"), ("counts", "<i8", (20,)),
                 ("dim", "<i4"), ("best_dim", "<i4"), ("best_code", "<i4"), ("best_flag", "<i4"),
                 ("inv_control", "<f4"), ("pad", "<f4"), ("mf", "<f4", (8,)), ("noise", "<f4", (8,)), ("best_noise", "<f4", (8,))])
assert HEAD.itemsize == 352


def sum64(data: bytes, h: int = 0x9E3779B97F4A7C15) -> int:
    """The blob checksum: h = (h ^ w) * 0x100000001B3, h ^= h >> 32 over the little-endian words, last one zero-padded."""
    M = (1 << 64) - 1
    pad = (-len(data)) % 8
    words = np.frombuffer(bytes(data) + b"\0" * pad, "<u8").tolist()
    for w in words:
        h = ((h ^ w) * 0x100000001B3) & M
        h ^= h >> 32
    return h


class SavedState:
    """The chains section of a saved state: head [n] (HEAD) and the float arrays of every chain in state.cu order
    (cur / prop models [md], eq [ne][3], origin, pres, sres, evsum [ne][8], the best-model snapshot)."""

    def __init__(self, blob: bytes):
        from mcmc_eq_b200._lib import MqStateHeader, MqStateSection
        self.blob = bytearray(blob)
        H = MqStateHeader.from_buffer_copy(self.blob[:C.sizeof(MqStateHeader)])
        self.header = H
        self.n, self.md, self.ne, self.ns = H.n_chains, H.max_dim, H.n_events, H.n_stations
        self.seed, self.chain_offset = H.seed, H.chain_offset
        off = None
        for k in range(H.n_sections):
            s = MqStateSection.from_buffer_copy(self.blob, C.sizeof(MqStateHeader) + k * C.sizeof(MqStateSection))
            if s.id == 1:
                off = s.offset
        assert off is not None
        md, ne, ns = self.md, self.ne, self.ns
        nf = 9 * md + 16 * ne + 4 * ns
        self.rec_bytes = (HEAD.itemsize + 4 * nf + 7) // 8 * 8
        self.off = off
        rec = np.dtype([("head", HEAD), ("f", "<f4", (nf,)), ("pad", "u1", (self.rec_bytes - HEAD.itemsize - 4 * nf,))])
        self.rec = np.frombuffer(self.blob, rec, self.n, off).copy()
        self.head = self.rec["head"]
        f = self.rec["f"]
        o = 0

        def take(k):
            nonlocal o
            a = f[:, o:o + k]
            o += k
            return a
        self.z, self.vp, self.vpvs = take(md), take(md), take(md)
        take(3 * md)
        self.eq = take(3 * ne).reshape(self.n, ne, 3)
        self.origin = take(ne)
        self.pres, self.sres = take(ns), take(ns)

    def chain(self, c: int) -> State:
        h = self.head[c]
        d = int(h["dim"])
        return State(d, self.z[c, :d].tolist(), self.vp[c, :d].tolist(), self.vpvs[c, :d].tolist(), self.eq[c].tolist(),
                     self.pres[c].tolist(), self.sres[c].tolist(), h["noise"].tolist(), float(h["inv_control"]),
                     int(h["acce"]), int(h["reject"]), [int(x) for x in h["counts"]], int(h["draws"]), float(h["ll"]),
                     h["mf"].tolist())

    def edited(self) -> bytes:
        """The blob with this object's (edited) chain records and a recomputed checksum."""
        b = bytearray(self.blob)
        b[self.off:self.off + self.rec.nbytes] = self.rec.tobytes()
        b[-8:] = struct.pack("<Q", sum64(bytes(b[:-8])))
        return bytes(b)


# ---- jobs for worker processes ---------------------------------------------------------------------------------------

def init_job(job):
    """(cfg, seed, chain) -> (start state, ok) of device chain `chain` (chain offset included)."""
    cfg, seed, chain = job
    return init_chain(cfg, Rand(Philox(seed, chain, 0)))


def propose_job(job):
    """(state, cfg, seed, chain, override, flip) -> (state after the LVZ switch, proposal, rng after the proposal)."""
    st, cfg, seed, chain, override, flip = job
    rng = Rand(Philox(seed, chain, st.draws), flip)
    P = propose(st, cfg, rng, override)
    return st, P, rng
