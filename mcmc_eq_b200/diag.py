"""Host statement of the convergence diagnostics (include/mcmceq_b200.h: mq_diag_*, csrc/diag.cu, DESIGN.md section 4d).

`accumulate` is the slot and doubling rule of the device's per-chain accumulators in float64 and in the device's order, so
that it gives the same bits from the same quantities; `summarise` is split R-hat, the batch-means ESS, mean and sd from
those accumulators.  The tests compare the device with these functions, as `dist.swap_plan` is for tempering.
"""
from __future__ import annotations

import numpy as np

def quantity_table(nz: int, ne: int, ns: int) -> list[tuple[str, int]]:
    """(name, index) of each of the Q = 10 + 2 nz + 4 ne + 2 ns quantities, in the device's order."""
    out = [("rms", 0), ("dim", 0)] + [("noise", k) for k in range(8)]
    out += [("vp", i) for i in range(nz)] + [("vpvs", i) for i in range(nz)]
    out += [(w, e) for e in range(ne) for w in ("x", "y", "z", "t")]
    out += [(w, s) for s in range(ns) for w in ("pres", "sres")]
    return out


def quantity_names(nz: int, ne: int, ns: int) -> list[str]:
    """'rms', 'dim', 'noise[k]', 'vp[i]', 'vpvs[i]', 'x[e]' .. 't[e]', 'pres[s]', 'sres[s]'."""
    return [w if w in ("rms", "dim") else f"{w}[{i}]" for w, i in quantity_table(nz, ne, ns)]


def record_quantities(rec: dict, cfg, velocity) -> np.ndarray:
    """The Q quantities of one drained record (Sampler.drain's dict) as float64.  velocity(rec) -> (vp[nz], vpvs[nz]) is
    the rasterisation (nearest nucleus or TRIA = 1 profile, clipped to the prior range) the caller states."""
    vp, vpvs = velocity(rec)
    eq = np.concatenate([np.asarray(rec["eq"], np.float32), np.asarray(rec["origin"], np.float32)[:, None]], 1)
    st = np.stack([np.asarray(rec["pres"], np.float32), np.asarray(rec["sres"], np.float32)], 1)
    parts = [np.float64([rec["rms"], rec["dim"]]), np.asarray(rec["noise"], np.float32), np.asarray(vp, np.float32),
             np.asarray(vpvs, np.float32), eq.ravel(), st.ravel()]
    return np.concatenate([np.asarray(p).astype(np.float64) for p in parts])


def accumulate(trace, K: int = 16) -> dict:
    """Accumulators of the device from a chain's used models in order: trace [n_models, Q], or [n_chains, n_models, Q]
    for chains with the same number of models.  -> ref, sum [K, Q], sumsq [K, Q], batch_len, full_batches, n_models (with a
    leading chain axis for a 3-d trace)."""
    x = np.asarray(trace, np.float64)
    one = x.ndim == 2
    if one:
        x = x[None]
    n, m, Q = x.shape
    ref = x[:, 0, :].copy() if m else np.zeros((n, Q))
    S, T = np.zeros((n, K, Q)), np.zeros((n, K, Q))
    k, L = 0, 1
    for j in range(m):
        d = x[:, j, :] - ref
        S[:, k] = S[:, k] + d
        T[:, k] = T[:, k] + d * d
        if j + 1 - k * L == L:            # the model fills the open slot
            k += 1
            if k == K:                    # pairs merge, i ascending; slots K/2 .. K-1 are empty again
                for i in range(K // 2):
                    S[:, i] = S[:, 2 * i] + S[:, 2 * i + 1]
                    T[:, i] = T[:, 2 * i] + T[:, 2 * i + 1]
                S[:, K // 2:] = 0.0
                T[:, K // 2:] = 0.0
                k, L = K // 2, 2 * L
    out = dict(ref=ref, sum=S, sumsq=T, batch_len=np.full(n, L, np.int32), full_batches=np.full(n, k, np.int32),
               n_models=np.full(n, m, np.int64))
    return {a: v[0] for a, v in out.items()} if one else out


def stack(accs: list[dict]) -> dict:
    """One accumulator dict with a chain axis from per-chain dicts of `accumulate`."""
    return {a: np.stack([np.asarray(x[a]) for x in accs]) for a in accs[0]}


def summarise(ref, sum, sumsq, batch_len, full_batches, **_ignored) -> dict:
    """Split R-hat, batch-means ESS, mean and sd per quantity from per-chain accumulators (shapes of mq_diag_chains).
    Extra keys (n_models) are ignored, so summarise(**acc) works.  -> mean, sd, rhat, ess [Q], n_models (N), chains_used."""
    ref, S, T = np.asarray(ref, np.float64), np.asarray(sum, np.float64), np.asarray(sumsq, np.float64)
    L_all, k_all = np.asarray(batch_len, np.int64), np.asarray(full_batches, np.int64)
    Q = ref.shape[1]
    used = np.nonzero(k_all >= 4)[0]
    nan = np.full(Q, np.nan)
    if len(used) == 0:
        return dict(mean=nan, sd=nan.copy(), rhat=nan.copy(), ess=nan.copy(), n_models=0, chains_used=0)
    mus, s2s, ns = [], [], []
    sig_num, sig_den, N, mean_num = np.zeros(Q), 0.0, 0.0, np.zeros(Q)
    for c in used:                        # per chain in the device's order: batch sums added one slot after the other
        k, L = int(k_all[c]), float(L_all[c])
        h = k // 2
        nj = h * L
        for lo in (0, h):
            Sj, Tj = np.zeros(Q), np.zeros(Q)
            for b in range(lo, lo + h):
                Sj, Tj = Sj + S[c, b], Tj + T[c, b]
            m = Sj / nj
            s2s.append((Tj - Sj * m) / (nj - 1.0))
            mus.append(ref[c] + m)
            ns.append(nj)
        sall, ysum, dev = np.zeros(Q), np.zeros(Q), np.zeros(Q)
        for b in range(k):
            sall, ysum = sall + S[c, b], ysum + S[c, b] / L
        ybar = ysum / k
        for b in range(k):
            dev = dev + (S[c, b] / L - ybar) ** 2
        sig_num += L * dev
        sig_den += k - 1
        N += k * L
        mean_num += k * L * ref[c] + sall
    mus, s2s = np.array(mus), np.array(s2s)
    M = len(mus)
    W = s2s.mean(0)
    mubar = mus.mean(0)
    Bv = ((mus - mubar) ** 2).sum(0) / (M - 1)
    nbar = float(np.mean(ns))
    varp = (nbar - 1.0) / nbar * W + Bv
    sig = sig_num / sig_den
    with np.errstate(divide="ignore", invalid="ignore"):
        rhat = np.where(varp > 0, np.where(W > 0, np.sqrt(varp / np.where(W > 0, W, 1.0)), np.inf), np.nan)
        ess = np.where(varp > 0, np.where(sig > 0, N * varp / np.where(sig > 0, sig, 1.0), np.inf), np.nan)
    return dict(mean=mean_num / N, sd=np.sqrt(varp), rhat=rhat, ess=ess, n_models=int(N), chains_used=len(used))
