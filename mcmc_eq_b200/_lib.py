"""ctypes binding of libmcmceq_b200.so (include/mcmceq_b200.h, host/mq_io.h)."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
# MCMCEQ_LIB: an alternative build of the same library (A/B experiments, tools/ab_build.py); the default is the in-tree build
LIB_PATH = os.environ.get("MCMCEQ_LIB") or os.path.join(_PKG, "libmcmceq_b200.so")
_lib = None

fp = C.POINTER(C.c_float)
dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int32)
lp = C.POINTER(C.c_int64)


class MqError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libmcmceq_b200 error {code}: {msg}")
        self.code = code


class MqGrid(C.Structure):
    _fields_ = [("h", C.c_float), ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32),
                ("x0", C.c_float), ("y0", C.c_float), ("z0", C.c_float)]


class MqConfig(C.Structure):
    _fields_ = [("grid", MqGrid), ("max_dim", C.c_int32),
                ("vpmin", C.c_float), ("vpmax", C.c_float), ("vpvsmin", C.c_float), ("vpvsmax", C.c_float),
                ("noise_min", C.c_float), ("noise_max", C.c_float), ("residual_min", C.c_float), ("residual_max", C.c_float),
                ("sdevx", C.c_float), ("sdevy", C.c_float), ("sdevz", C.c_float),
                ("sdevvp", C.c_float), ("sdevvpvs", C.c_float), ("sdevn", C.c_float),
                ("sdevxs", C.c_float), ("epi_search", C.c_float), ("sdevys", C.c_float), ("sdevzs", C.c_float),
                ("sdevresidual", C.c_float), ("inv_control", C.c_float),
                ("reference_station", C.c_int32), ("scor_flag", C.c_int32),
                ("ref_statcor_P", C.c_float), ("ref_statcor_S", C.c_float), ("tria", C.c_int32),
                ("j_max_start", C.c_int32), ("j_max_main", C.c_int32), ("deci", C.c_int32),
                ("true_random", C.c_int32), ("eikonal", C.c_int32),
                ("dstring_start", C.c_char * 64), ("dstring_main", C.c_char * 64),
                ("aflag", C.c_int32), ("inp_model_switch", C.c_char * 16),
                ("start_vp", C.c_float), ("sdev_start_vp", C.c_float), ("start_vp_grad", C.c_float),
                ("start_vpvs", C.c_float), ("sdev_start_vpvs", C.c_float),
                ("start_cell_number", C.c_int32), ("sdev_start_cell_number", C.c_int32),
                ("start_noise", C.c_float), ("start_delay", C.c_float), ("sdev_start_delay", C.c_float),
                ("r_start_eqh", C.c_float), ("r_start_eqv", C.c_float)]


class MqPicks(C.Structure):
    _fields_ = [("n_events", C.c_int32), ("n_picks", C.c_int32), ("n_stations", C.c_int32),
                ("ev_off", ip), ("n_p", ip), ("st_id", ip), ("x", fp), ("y", fp), ("z", fp), ("t", fp), ("cls", ip),
                ("reftime", dp), ("fix", dp)]


class MqioPicks(C.Structure):
    _fields_ = [("view", MqPicks), ("ev_off", ip), ("n_p", ip), ("st_id", ip), ("cls", ip), ("eq_id", ip),
                ("x", fp), ("y", fp), ("z", fp), ("t", fp), ("reftime", dp), ("fix", dp), ("n_class", C.c_int32 * 8)]


class MqModels(C.Structure):
    _fields_ = [("n_chains", C.c_int32), ("max_dim", C.c_int32), ("n_events", C.c_int32), ("n_stations", C.c_int32),
                ("dim", ip), ("z", fp), ("vp", fp), ("vpvs", fp), ("eq", fp), ("pres", fp), ("sres", fp), ("noise", fp),
                ("origin", fp)]


class MqRecord(C.Structure):
    _fields_ = [("chain", C.c_int32), ("kind", C.c_int32), ("code", C.c_char), ("number", C.c_int64), ("dim", C.c_int32),
                ("rms", C.c_double), ("noise", fp), ("z", fp), ("vp", fp), ("vpvs", fp), ("eq", fp), ("origin", fp),
                ("pres", fp), ("sres", fp)]


class MqReplay(C.Structure):
    _fields_ = [("n_chains", C.c_int32), ("kind", C.c_char_p), ("proposed", C.POINTER(MqModels)), ("q_idx", ip),
                ("log_fac", dp), ("u", fp), ("accepted", ip), ("alpha", fp), ("new_ll", dp), ("mf", fp)]


class MqPosteriorDims(C.Structure):
    _fields_ = [("ndv", C.c_int32), ("ndvpvs", C.c_int32), ("nz", C.c_int32), ("n_events", C.c_int32), ("n_stations", C.c_int32)]


class MqDiagDims(C.Structure):
    _fields_ = [("n_quantities", C.c_int32), ("nz", C.c_int32), ("n_events", C.c_int32), ("n_stations", C.c_int32),
                ("n_batches", C.c_int32)]


class MqHypoDims(C.Structure):
    _fields_ = [("n_events", C.c_int32), ("n_bins", C.c_int32 * 3), ("bin_km", C.c_float), ("lo", C.c_float * 3)]


class MqStateHeader(C.Structure):
    """Start of a saved sampler state (include/mcmceq_b200.h: mq_state_header)."""
    _fields_ = [("magic", C.c_char * 8), ("format", C.c_uint32), ("header_bytes", C.c_uint32), ("version", C.c_char * 48),
                ("n_chains", C.c_int32), ("max_dim", C.c_int32), ("n_events", C.c_int32), ("n_stations", C.c_int32),
                ("n_picks", C.c_int32), ("nz", C.c_int32), ("nxmod", C.c_int32), ("n_rows", C.c_int32),
                ("seed", C.c_uint64), ("chain_offset", C.c_int64), ("flags", C.c_uint32), ("n_sections", C.c_uint32),
                ("post_dv", C.c_float), ("post_dvpvs", C.c_float), ("post_ndv", C.c_int32), ("post_ndvpvs", C.c_int32),
                ("post_burn_in", C.c_int64), ("config_sum", C.c_uint64), ("picks_sum", C.c_uint64)]


class MqStateSection(C.Structure):
    _fields_ = [("id", C.c_uint32), ("reserved", C.c_uint32), ("offset", C.c_uint64), ("bytes", C.c_uint64)]


STATE_POSTERIOR, STATE_BETA, STATE_TABLES, STATE_DIAG, STATE_RECIPROCAL, STATE_HYPO = 1, 2, 4, 8, 16, 32
TABLES_PARITY, TABLES_RECIPROCAL = 0, 1     # mq_set_tables
STATE_SEC_DIAG, STATE_SEC_HYPO = 5, 6


RECORD_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(MqRecord))


def lib() -> C.CDLL:
    """Load the CUDA library.  Fails loudly when it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(f"{LIB_PATH} not built: run `python -m mcmc_eq_b200.build`")
        L = C.CDLL(LIB_PATH)
        L.mq_version.restype = C.c_char_p
        L.mq_last_error.restype = C.c_char_p
        L.mqio_last_error.restype = C.c_char_p
        L.mq_launch_count.restype = C.c_int64
        L.mq_time_2d.argtypes = [fp, fp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int]
        L.mq_eikonal_batch.argtypes = [fp, ip, C.c_int, C.c_int, C.c_int, fp, ip, C.c_int]
        L.mq_create.argtypes = [C.POINTER(MqConfig), C.POINTER(MqPicks), C.c_int, C.c_int, C.c_uint64, C.POINTER(C.c_void_p)]
        L.mq_destroy.argtypes = [C.c_void_p]
        L.mq_set_models.argtypes = [C.c_void_p, C.POINTER(MqModels)]
        L.mq_get_models.argtypes = [C.c_void_p, C.POINTER(MqModels)]
        L.mq_forward.argtypes = [C.c_void_p, C.c_int, fp, fp]
        L.mq_forward_host.argtypes = [C.c_void_p, C.POINTER(MqModels), C.c_int, fp, fp]
        u8p = C.POINTER(C.c_uint8)
        L.mq_set_chain_offset.argtypes = [C.c_void_p, C.c_int64]
        L.mq_posterior_begin.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_int64, C.POINTER(MqPosteriorDims)]
        L.mq_posterior_get.argtypes = [C.c_void_p, ip, ip, ip, dp, dp, dp, dp, lp]
        L.mq_posterior_allreduce.argtypes = [C.c_void_p]
        L.mq_diag_begin.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.POINTER(MqDiagDims)]
        L.mq_diag_chains.argtypes = [C.c_void_p, dp, dp, dp, ip, ip, lp]
        L.mq_diag_summary.argtypes = [C.c_void_p, C.c_int, dp, dp, dp, dp, lp, ip]
        L.mq_hypo_begin.argtypes = [C.c_void_p, C.c_float, C.c_int64, C.POINTER(MqHypoDims)]
        L.mq_hypo_chains.argtypes = [C.c_void_p, ip, ip, dp, dp, dp, lp]
        L.mq_hypo_summary.argtypes = [C.c_void_p, C.c_int, dp, dp, dp, dp, dp, dp, lp]
        L.mq_comm_unique_id.argtypes = [u8p]
        L.mq_comm_init.argtypes = [C.c_void_p, u8p, C.c_int, C.c_int]
        L.mq_comm_destroy.argtypes = [C.c_void_p]
        L.mq_set_beta.argtypes = [C.c_void_p, fp]
        L.mq_get_beta.argtypes = [C.c_void_p, fp]
        L.mq_temper_swap.argtypes = [C.c_void_p, C.c_int64, ip]
        L.mq_tables_save.argtypes = [C.c_void_p]
        L.mq_tables_restore.argtypes = [C.c_void_p]
        L.mq_get_table.argtypes = [C.c_void_p, C.c_int, C.c_int, fp]
        L.mq_get_rows.argtypes = [C.c_void_p, C.c_int, C.c_int, fp, C.POINTER(C.c_int32)]
        L.mq_set_tables.argtypes = [C.c_void_p, C.c_int]
        L.mq_get_predictions.argtypes = [C.c_void_p, C.c_int, fp, fp]
        L.mq_init_chains.argtypes = [C.c_void_p]
        L.mq_step.argtypes = [C.c_void_p, C.c_int, C.c_char_p]
        L.mq_replay_step.argtypes = [C.c_void_p, C.POINTER(MqReplay)]
        L.mq_get_stats.argtypes = [C.c_void_p, lp, dp, dp]
        L.mq_drain.argtypes = [C.c_void_p, RECORD_FN, C.c_void_p, C.POINTER(C.c_int)]
        L.mq_set_ring.argtypes = [C.c_void_p, C.c_int]
        L.mq_drain_begin.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.mq_batch_wait.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.mq_batch_deliver.argtypes = [C.c_void_p, RECORD_FN, C.c_void_p]
        L.mq_batch_release.argtypes = [C.c_void_p]
        L.mq_snapshot.argtypes = [C.c_void_p, C.c_int, C.c_int, RECORD_FN, C.c_void_p]
        L.mq_snapshot_all.argtypes = [C.c_void_p, C.c_int, RECORD_FN, C.c_void_p]
        L.mq_profile_kernels.argtypes = [C.c_void_p, lp, dp]
        L.mq_profile_misfit.argtypes = [C.c_void_p, lp, dp]
        L.mq_eikonal_kernel_name.argtypes = [C.c_int]
        L.mq_eikonal_kernel_name.restype = C.c_char_p
        L.mq_sync.argtypes = [C.c_void_p]
        L.mq_timer.argtypes = [C.c_void_p, C.c_int, C.c_int, dp]
        L.mq_profile.argtypes = [C.c_void_p, C.c_int, dp, lp, lp]
        L.mq_state_size.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        L.mq_state_save.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
        L.mq_state_load.argtypes = [C.c_void_p, C.c_char_p, C.c_uint64]
        L.mqio_read_config.argtypes = [C.c_char_p, C.POINTER(MqConfig)]
        L.mqio_read_picks.argtypes = [C.c_char_p, C.POINTER(MqioPicks)]
        L.mqio_free_picks.argtypes = [C.POINTER(MqioPicks)]
        _lib = L
    return _lib


def comm_unique_id() -> bytes:
    """128 bytes identifying a new NCCL communicator (rank 0 calls this and distributes them)."""
    buf = (C.c_uint8 * 128)()
    check(lib().mq_comm_unique_id(buf))
    return bytes(buf)


def check(rc: int) -> None:
    if rc != 0:
        raise MqError(rc, lib().mq_last_error().decode())


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a, t=fp):
    return a.ctypes.data_as(t)


def eikonal_batch(slow, src_iz, nxmod: int, device: int = 0, return_status: bool = False):
    """n solves: slow[n, nz] (h/v per depth cell), src_iz[n] -> t[n, nxmod, nz]."""
    slow = _f32(slow)
    n, nz = slow.shape
    iz = np.ascontiguousarray(src_iz, dtype=np.int32)
    assert iz.shape == (n,)
    t = np.empty((n, nxmod, nz), np.float32)
    st = np.zeros(n, np.int32)
    rc = lib().mq_eikonal_batch(_p(slow), _p(iz, ip), n, nxmod, nz, _p(t), _p(st, ip), device)
    if return_status:
        return t, st, rc
    check(rc)
    return t


def time_2d(hs, xs: float, ys: float, eps_init: float = 0.001) -> np.ndarray:
    """Drop-in call of the reference's time_2d signature (hs[nx, ny] -> t[nx, ny])."""
    hs = _f32(hs)
    nx, ny = hs.shape
    t = np.zeros((nx, ny), np.float32)
    check(lib().mq_time_2d(_p(hs), _p(t), nx, ny, xs, ys, eps_init, 0))
    return t


def read_config(path: str) -> MqConfig:
    cfg = MqConfig()
    rc = lib().mqio_read_config(path.encode(), C.byref(cfg))
    if rc != 0:
        raise MqError(rc, lib().mqio_last_error().decode())
    return cfg


class Picks:
    """Flattened pick set (numpy arrays) + the C view of it."""

    def __init__(self, ev_off, n_p, st_id, x, y, z, t, cls, reftime=None, fix=None, n_stations=None):
        self.ev_off = np.ascontiguousarray(ev_off, np.int32)
        self.n_p = np.ascontiguousarray(n_p, np.int32)
        self.st_id = np.ascontiguousarray(st_id, np.int32)
        self.x, self.y, self.z, self.t = _f32(x), _f32(y), _f32(z), _f32(t)
        self.cls = np.ascontiguousarray(cls, np.int32)
        self.n_events = len(self.n_p)
        self.n_picks = len(self.st_id)
        self.n_stations = int(self.st_id.max()) + 1 if n_stations is None else int(n_stations)
        self.reftime = np.ascontiguousarray(reftime if reftime is not None else np.zeros(self.n_events), np.float64)
        self.fix = np.ascontiguousarray(fix if fix is not None else np.full((self.n_events, 3), -9999.0), np.float64)
        self.view = MqPicks(self.n_events, self.n_picks, self.n_stations, _p(self.ev_off, ip), _p(self.n_p, ip),
                            _p(self.st_id, ip), _p(self.x), _p(self.y), _p(self.z), _p(self.t), _p(self.cls, ip),
                            _p(self.reftime, dp), _p(self.fix, dp))

    @staticmethod
    def read(path: str) -> "Picks":
        raw = MqioPicks()
        rc = lib().mqio_read_picks(path.encode(), C.byref(raw))
        if rc != 0:
            raise MqError(rc, lib().mqio_last_error().decode())
        v = raw.view
        ne, npk = v.n_events, v.n_picks
        arr = lambda p, n, dt: np.ctypeslib.as_array(p, shape=(n,)).astype(dt, copy=True)
        out = Picks(arr(v.ev_off, ne + 1, np.int32), arr(v.n_p, ne, np.int32), arr(v.st_id, npk, np.int32),
                    arr(v.x, npk, np.float32), arr(v.y, npk, np.float32), arr(v.z, npk, np.float32),
                    arr(v.t, npk, np.float32), arr(v.cls, npk, np.int32), arr(v.reftime, ne, np.float64),
                    arr(v.fix, 3 * ne, np.float64).reshape(ne, 3), v.n_stations)
        out.n_class = np.array(list(raw.n_class), np.int32)
        lib().mqio_free_picks(C.byref(raw))
        return out


class Models:
    """Host SoA mirror of `struct Model` for n chains."""

    def __init__(self, n_chains, max_dim, n_events, n_stations):
        self.n, self.md, self.ne, self.ns = n_chains, max_dim, n_events, n_stations
        self.dim = np.ones(n_chains, np.int32)
        self.z = np.zeros((n_chains, max_dim), np.float32)
        self.vp = np.ones((n_chains, max_dim), np.float32)
        self.vpvs = np.ones((n_chains, max_dim), np.float32)
        self.eq = np.zeros((n_chains, n_events, 3), np.float32)
        self.pres = np.zeros((n_chains, n_stations), np.float32)
        self.sres = np.zeros((n_chains, n_stations), np.float32)
        self.noise = np.ones((n_chains, 8), np.float32)
        self.origin = np.zeros((n_chains, n_events), np.float32)

    def view(self) -> MqModels:
        return MqModels(self.n, self.md, self.ne, self.ns, _p(self.dim, ip), _p(self.z), _p(self.vp), _p(self.vpvs),
                        _p(self.eq), _p(self.pres), _p(self.sres), _p(self.noise), _p(self.origin))


class Sampler:
    """One handle = n_chains chains on one GPU."""

    def __init__(self, cfg: MqConfig, picks: Picks, n_chains: int, device: int = 0, seed: int = 1):
        self.cfg, self.picks, self.n = cfg, picks, n_chains
        self.h = C.c_void_p()
        check(lib().mq_create(C.byref(cfg), C.byref(picks.view), n_chains, device, seed, C.byref(self.h)))
        self.nz = cfg.grid.nz
        self.nxmod = int(np.sqrt(cfg.grid.nx * cfg.grid.nx + cfg.grid.ny * cfg.grid.ny))

    def close(self):
        if self.h:
            lib().mq_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def new_models(self, max_dim=None) -> Models:
        return Models(self.n, max_dim or min(self.cfg.max_dim, 1000), self.picks.n_events, self.picks.n_stations)

    def set_models(self, m: Models):
        v = m.view()
        check(lib().mq_set_models(self.h, C.byref(v)))

    def get_models(self, max_dim=None) -> Models:
        m = self.new_models(max_dim)
        v = m.view()
        check(lib().mq_get_models(self.h, C.byref(v)))
        return m

    def forward(self, calct=3, want_origin=True):
        mf = np.zeros((self.n, 8), np.float32)
        org = np.zeros((self.n, self.picks.n_events), np.float32) if want_origin else None
        check(lib().mq_forward(self.h, calct, _p(mf), _p(org) if want_origin else None))
        return mf, org

    def forward_host(self, m: Models, calct=3, mf=None, origin=None):
        mf = np.zeros((self.n, 8), np.float32) if mf is None else mf
        origin = np.zeros((self.n, self.picks.n_events), np.float32) if origin is None else origin
        v = m.view()
        check(lib().mq_forward_host(self.h, C.byref(v), calct, _p(mf), _p(origin)))
        return mf, origin

    def tables_save(self):
        check(lib().mq_tables_save(self.h))

    def tables_restore(self):
        check(lib().mq_tables_restore(self.h))

    def set_tables(self, mode: str):
        """How tables are built: "parity" (the default, one solve per source depth) or "reciprocal" (one solve per receiver
        row, an approximation: DESIGN.md section 6).  Before set_models / init_chains / load_state."""
        modes = {"parity": TABLES_PARITY, "reciprocal": TABLES_RECIPROCAL}
        if mode not in modes:
            raise ValueError(f"table mode {mode!r}: 'parity' or 'reciprocal'")
        check(lib().mq_set_tables(self.h, modes[mode]))

    def table(self, chain: int, phase: int) -> np.ndarray:
        t = np.zeros((self.nz, self.nz, self.nxmod), np.float32)
        check(lib().mq_get_table(self.h, chain, phase, _p(t)))
        return t

    def rows(self, chain: int, phase: int):
        """(rows[n_rows][nz][nxmod], row_index[n_rows]): the stored receiver rows of a chain's table."""
        n = lib().mq_get_rows(self.h, chain, phase, None, None)
        if n < 0:
            check(n)
        t = np.zeros((n, self.nz, self.nxmod), np.float32)
        idx = np.zeros(n, np.int32)
        n2 = lib().mq_get_rows(self.h, chain, phase, _p(t), idx.ctypes.data_as(C.POINTER(C.c_int32)))
        if n2 < 0:
            check(n2)
        return t, idx

    def predictions(self, chain: int):
        r = np.zeros(self.picks.n_picks, np.float32)
        t = np.zeros(self.picks.n_picks, np.float32)
        check(lib().mq_get_predictions(self.h, chain, _p(r), _p(t)))
        return r, t

    def init_chains(self):
        check(lib().mq_init_chains(self.h))

    def step(self, n_iters: int, override: str | None = None):
        check(lib().mq_step(self.h, n_iters, override.encode() if override else None))

    def replay_step(self, kinds, proposed: "Models", q_idx, log_fac, u):
        """One iteration driven by recorded proposals (mq_replay_step): kinds = one letter per chain ('\\0' skips)."""
        n = self.n
        kb = C.create_string_buffer(bytes(ord(k) if isinstance(k, str) else int(k) for k in kinds), n)
        q = np.ascontiguousarray(q_idx, np.int32)
        lf = np.ascontiguousarray(log_fac, np.float64)
        uu = _f32(u)
        acc, alpha, ll, mf = np.zeros(n, np.int32), np.zeros(n, np.float32), np.zeros(n, np.float64), np.zeros((n, 8), np.float32)
        v = proposed.view()
        r = MqReplay(n, C.cast(kb, C.c_char_p), C.pointer(v), _p(q, ip), _p(lf, dp), _p(uu), _p(acc, ip), _p(alpha), _p(ll, dp), _p(mf))
        check(lib().mq_replay_step(self.h, C.byref(r)))
        return dict(accepted=acc, alpha=alpha, new_ll=ll, mf=mf)

    # ---- more than one GPU / posterior / tempering -------------------------------------------------------
    def set_chain_offset(self, first_chain: int):
        check(lib().mq_set_chain_offset(self.h, first_chain))

    def posterior_begin(self, dv: float, dvpvs: float, burn_in: int = 0):
        d = MqPosteriorDims()
        check(lib().mq_posterior_begin(self.h, dv, dvpvs, burn_in, C.byref(d)))
        self._pdims = d
        return d

    def posterior_get(self):
        d = self._pdims
        out = dict(hist_vp=np.zeros((d.ndv, d.nz), np.int32), hist_vpvs=np.zeros((d.ndvpvs, d.nz), np.int32),
                   boundary=np.zeros(d.nz, np.int32), vsum=np.zeros((d.nz, 4)), eqsum=np.zeros((d.n_events, 8)),
                   ressum=np.zeros((d.n_stations, 4)), noisesum=np.zeros(16))
        n = C.c_int64(0)
        check(lib().mq_posterior_get(self.h, _p(out["hist_vp"], ip), _p(out["hist_vpvs"], ip), _p(out["boundary"], ip),
                                     _p(out["vsum"], dp), _p(out["eqsum"], dp), _p(out["ressum"], dp), _p(out["noisesum"], dp),
                                     C.byref(n)))
        out["n_models"] = n.value
        return out

    def posterior_allreduce(self):
        check(lib().mq_posterior_allreduce(self.h))

    # ---- convergence diagnostics (mq_diag_*, mcmc_eq_b200/diag.py) ------------------------------------------------
    def diag_begin(self, burn_in: int = 0, n_batches: int = 16) -> MqDiagDims:
        """Split R-hat and ESS of every posterior quantity from the decimated models with number > burn_in."""
        d = MqDiagDims()
        check(lib().mq_diag_begin(self.h, burn_in, n_batches, C.byref(d)))
        self._ddims = (d.n_quantities, d.n_batches)
        return d

    def diag_chains(self) -> dict:
        """Raw per-chain accumulators: ref [n, Q], sum / sumsq [n, K, Q], batch_len, full_batches, n_models [n]."""
        Q, K = self._ddims
        out = dict(ref=np.zeros((self.n, Q)), sum=np.zeros((self.n, K, Q)), sumsq=np.zeros((self.n, K, Q)),
                   batch_len=np.zeros(self.n, np.int32), full_batches=np.zeros(self.n, np.int32), n_models=np.zeros(self.n, np.int64))
        check(lib().mq_diag_chains(self.h, _p(out["ref"], dp), _p(out["sum"], dp), _p(out["sumsq"], dp), _p(out["batch_len"], ip),
                                   _p(out["full_batches"], ip), _p(out["n_models"], lp)))
        return out

    def diag_summary(self, collective: bool = False) -> dict:
        """mean, sd, rhat, ess [Q], n_models (N), chains_used and the quantity names (diag.quantity_names)."""
        from .diag import quantity_names
        Q, _K = self._ddims
        out = {k: np.zeros(Q) for k in ("mean", "sd", "rhat", "ess")}
        n, used = C.c_int64(0), C.c_int32(0)
        check(lib().mq_diag_summary(self.h, int(collective), _p(out["mean"], dp), _p(out["sd"], dp), _p(out["rhat"], dp),
                                    _p(out["ess"], dp), C.byref(n), C.byref(used)))
        out["n_models"], out["chains_used"] = n.value, used.value
        out["names"] = quantity_names(self.nz, self.picks.n_events, self.picks.n_stations)
        return out

    # ---- hypocentre uncertainty (mq_hypo_*, mcmc_eq_b200/hypo.py) -------------------------------------------------
    def hypo_begin(self, bin_km: float, burn_in: int = 0) -> MqHypoDims:
        """Per-event covariance, quantiles, mode and error ellipsoid of the hypocentres of the decimated models with
        number > burn_in; histograms of x, y and z with bins of bin_km."""
        d = MqHypoDims()
        check(lib().mq_hypo_begin(self.h, bin_km, burn_in, C.byref(d)))
        self._hbins = tuple(d.n_bins)
        return d

    def hypo_chains(self) -> dict:
        """Raw accumulators: hist [ne, Bx + By + Bz], outside [ne, 3], ref / sum [n, 4, ne], cross [n, 10, ne], n_models [n]."""
        ne = self.picks.n_events
        out = dict(hist=np.zeros((ne, sum(self._hbins)), np.int32), outside=np.zeros((ne, 3), np.int32),
                   ref=np.zeros((self.n, 4, ne)), sum=np.zeros((self.n, 4, ne)), cross=np.zeros((self.n, 10, ne)),
                   n_models=np.zeros(self.n, np.int64))
        check(lib().mq_hypo_chains(self.h, _p(out["hist"], ip), _p(out["outside"], ip), _p(out["ref"], dp), _p(out["sum"], dp),
                                   _p(out["cross"], dp), _p(out["n_models"], lp)))
        return out

    def hypo_summary(self, collective: bool = False) -> dict:
        """mean [ne, 4], cov [ne, 4, 4], quant [ne, 3, 5], mode [ne, 3], axes [ne, 3], axis_dir [ne, 3, 3], n_models (N)."""
        ne = self.picks.n_events
        out = dict(mean=np.zeros((ne, 4)), cov=np.zeros((ne, 4, 4)), quant=np.zeros((ne, 3, 5)), mode=np.zeros((ne, 3)),
                   axes=np.zeros((ne, 3)), axis_dir=np.zeros((ne, 3, 3)))
        n = C.c_int64(0)
        check(lib().mq_hypo_summary(self.h, int(collective), *[_p(out[k], dp) for k in ("mean", "cov", "quant", "mode", "axes", "axis_dir")],
                                    C.byref(n)))
        out["n_models"] = n.value
        return out

    def comm_init(self, unique_id: bytes, rank: int, world: int):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        check(lib().mq_comm_init(self.h, buf, rank, world))

    def comm_destroy(self):
        check(lib().mq_comm_destroy(self.h))

    def set_beta(self, beta):
        b = _f32(beta)
        assert b.shape == (self.n,)
        check(lib().mq_set_beta(self.h, _p(b)))

    def get_beta(self) -> np.ndarray:
        b = np.zeros(self.n, np.float32)
        check(lib().mq_get_beta(self.h, _p(b)))
        return b

    def temper_swap(self, round_: int) -> int:
        k = C.c_int32(0)
        check(lib().mq_temper_swap(self.h, round_, C.byref(k)))
        return k.value

    def save_state(self) -> bytes:
        """Sampler state of every chain (mq_state_save): what step() needs to continue each chain exactly where it is.
        Drain the decimated records first."""
        size = C.c_uint64(0)
        check(lib().mq_state_size(self.h, C.byref(size)))
        buf = C.create_string_buffer(size.value)
        check(lib().mq_state_save(self.h, buf, size.value, C.byref(size)))
        return buf.raw[:size.value]

    def load_state(self, blob: bytes):
        """Continue from a state of save_state (mq_state_load); the state's seed, chain offset, posterior and betas
        replace this sampler's."""
        blob = bytes(blob)
        check(lib().mq_state_load(self.h, blob, len(blob)))
        head = MqStateHeader.from_buffer_copy(blob[:C.sizeof(MqStateHeader)])
        if head.flags & STATE_POSTERIOR:
            self._pdims = MqPosteriorDims(head.post_ndv, head.post_ndvpvs, self.nz, self.picks.n_events, self.picks.n_stations)
        if head.flags & STATE_DIAG:   # the section starts with int64 burn_in, int32 n_batches, int32 n_quantities
            for k in range(head.n_sections):
                sec = MqStateSection.from_buffer_copy(blob, C.sizeof(MqStateHeader) + k * C.sizeof(MqStateSection))
                if sec.id == STATE_SEC_DIAG:
                    K, Q = np.frombuffer(blob, np.int32, 2, sec.offset + 8)
                    self._ddims = (int(Q), int(K))
        if head.flags & STATE_HYPO:   # the section starts with int64 burn_in, float bin_km, int32 n_bins[3]
            for k in range(head.n_sections):
                sec = MqStateSection.from_buffer_copy(blob, C.sizeof(MqStateHeader) + k * C.sizeof(MqStateSection))
                if sec.id == STATE_SEC_HYPO:
                    self._hbins = tuple(int(b) for b in np.frombuffer(blob, np.int32, 3, sec.offset + 12))

    def sync(self):
        check(lib().mq_sync(self.h))

    def timer_start(self, slot=0):
        check(lib().mq_timer(self.h, slot, 0, None))

    def timer_stop(self, slot=0) -> float:
        ms = C.c_double(0)
        check(lib().mq_timer(self.h, slot, 1, C.byref(ms)))
        return ms.value

    def profile(self, enable=True):
        ms, n, per = C.c_double(0), C.c_int64(0), C.c_int64(0)
        check(lib().mq_profile(self.h, int(enable), C.byref(ms), C.byref(n), C.byref(per)))
        return ms.value, n.value, per.value

    def stats(self):
        counts = np.zeros((self.n, 20), np.int64)
        ll = np.zeros(self.n, np.float64)
        rms = np.zeros(self.n, np.float64)
        check(lib().mq_get_stats(self.h, _p(counts, lp), _p(ll, dp), _p(rms, dp)))
        return counts, ll, rms

    def _collect(self, call):
        out = []
        ne, ns = self.picks.n_events, self.picks.n_stations

        def cb(_user, rp):
            r = rp.contents
            a = lambda p, n: np.ctypeslib.as_array(p, shape=(n,)).copy()
            out.append(dict(chain=r.chain, kind=r.kind, code=r.code.decode(), number=r.number, dim=r.dim, rms=r.rms,
                            noise=a(r.noise, 8), z=a(r.z, r.dim), vp=a(r.vp, r.dim), vpvs=a(r.vpvs, r.dim),
                            eq=a(r.eq, 3 * ne).reshape(ne, 3), origin=a(r.origin, ne), pres=a(r.pres, ns), sres=a(r.sres, ns)))
            return 0

        call(RECORD_FN(cb))
        return out

    def drain(self):
        lost = C.c_int(0)
        recs = self._collect(lambda fn: check(lib().mq_drain(self.h, fn, None, C.byref(lost))))
        return recs, lost.value

    def set_ring(self, slots: int):
        check(lib().mq_set_ring(self.h, slots))

    def drain_begin(self):
        """Start an asynchronous drain; returns the batch (finish it with drain_finish, possibly on another thread)."""
        b = C.c_void_p()
        check(lib().mq_drain_begin(self.h, C.byref(b)))
        return b

    def drain_finish(self, batch):
        """-> (records, n_lost) of a batch begun with drain_begin; releases the batch."""
        n, lost = C.c_int(0), C.c_int(0)
        check(lib().mq_batch_wait(batch, C.byref(n), C.byref(lost)))
        recs = self._collect(lambda fn: check(lib().mq_batch_deliver(batch, fn, None)))
        check(lib().mq_batch_release(batch))
        assert len(recs) == n.value
        return recs, lost.value

    def snapshot(self, chain: int, which: int = 0):
        return self._collect(lambda fn: check(lib().mq_snapshot(self.h, chain, which, fn, None)))[0]

    def snapshot_all(self, which: int = 0):
        return self._collect(lambda fn: check(lib().mq_snapshot_all(self.h, which, fn, None)))

    def profile_misfit(self):
        """(launches, ms) of the misfit kernel over the accumulation the last profile() call read."""
        n, ms = C.c_int64(0), C.c_double(0)
        check(lib().mq_profile_misfit(self.h, C.byref(n), C.byref(ms)))
        return n.value, ms.value

    def profile_kernels(self):
        """{kernel name: (launches, ms)} of the eikonal launches counted by the last profile() call."""
        n = np.zeros(4, np.int64)
        ms = np.zeros(4, np.float64)
        check(lib().mq_profile_kernels(self.h, _p(n, lp), _p(ms, dp)))
        return {lib().mq_eikonal_kernel_name(k).decode(): (int(n[k]), float(ms[k])) for k in range(4) if n[k] > 0}
