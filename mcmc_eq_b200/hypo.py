"""Host statement of the hypocentre uncertainty (include/mcmceq_b200.h: mq_hypo_*, csrc/hypo.cu, DESIGN.md section 4e).

`accumulate` and `histogram` are the device's per-chain sums and per-event histograms, in float64 / float32 and in the
device's operation order, so that they give the same bits from the same drained records; `summarise` is the mean, the
covariance, the quantiles, the mode and the error ellipsoid from those accumulators, with `jacobi3` the device's
eigen-decomposition operation for operation.  The tests compare the device with these functions, as `diag.py` is for
mq_diag_*.  These statistics are this library's own; they are not analyse_eq's EZ / EM.
"""
from __future__ import annotations

import math

import numpy as np

PROBS = (0.025, 0.16, 0.5, 0.84, 0.975)
PAIRS = [(i, j) for i in range(4) for j in range(i, 4)]   # xx xy xz xt yy yz yt zz zt tt
JACOBI_SWEEPS = 32


def box(cfg) -> tuple[np.ndarray, np.ndarray]:
    """lo, hi (float32 [3]) of the box the sampler keeps hypocentres in: grid origin to origin + (n - 1) h."""
    g = cfg.grid
    h = np.float32(g.h)
    lo = np.array([g.x0, g.y0, g.z0], np.float32)
    n = np.array([g.nx - 1, g.ny - 1, g.nz - 1], np.float32)
    return lo, (lo + n * h).astype(np.float32)


def n_bins(lo, hi, bin_km: float) -> np.ndarray:
    """Bins per axis: (int)((hi - lo) / w) + 1 in float32."""
    lo, hi, w = np.asarray(lo, np.float32), np.asarray(hi, np.float32), np.float32(bin_km)
    return (np.trunc((hi - lo) / w).astype(np.int64) + 1).astype(np.int32)


def record_values(rec: dict) -> np.ndarray:
    """(x, y, z, t) of every event of one drained record (Sampler.drain's dict): float32 [ne, 4]."""
    return np.concatenate([np.asarray(rec["eq"], np.float32).reshape(-1, 3), np.asarray(rec["origin"], np.float32)[:, None]], 1)


def accumulate(trace) -> dict:
    """A chain's sums from its used models in record order: trace float32 [m, ne, 4] -> ref, sum [4, ne], cross [10, ne],
    n_models."""
    x = np.asarray(trace, np.float32).astype(np.float64)
    m, ne = x.shape[0], x.shape[1]
    ref = x[0].T.copy() if m else np.zeros((4, ne))
    S, Cx = np.zeros((4, ne)), np.zeros((10, ne))
    for k in range(m):
        d = x[k].T - ref
        S = S + d
        for p, (i, j) in enumerate(PAIRS):
            Cx[p] = Cx[p] + d[i] * d[j]
    return dict(ref=ref, sum=S, cross=Cx, n_models=m)


def histogram(trace, lo, hi, bin_km: float) -> tuple[np.ndarray, np.ndarray]:
    """Histograms of x, y, z of used models (trace float32 [m, ne, >= 3]) -> hist [ne, Bx + By + Bz], outside [ne, 3]."""
    v = np.asarray(trace, np.float32)
    lo, hi, w = np.asarray(lo, np.float32), np.asarray(hi, np.float32), np.float32(bin_km)
    nb = n_bins(lo, hi, w)
    m, ne = v.shape[0], v.shape[1]
    hist = np.zeros((ne, int(nb.sum())), np.int32)
    outside = np.zeros((ne, 3), np.int32)
    off = 0
    for a in range(3):
        q = ((v[:, :, a] - lo[a]) / w).astype(np.float32)
        j = np.trunc(np.clip(q, -1.0, float(nb[a]))).astype(np.int64)
        j = np.clip(j, 0, nb[a] - 1)
        outside[:, a] = (~((v[:, :, a] >= lo[a]) & (v[:, :, a] <= hi[a]))).sum(0)
        for e in range(ne):
            hist[e, off:off + nb[a]] += np.bincount(j[:, e], minlength=int(nb[a])).astype(np.int32)
        off += int(nb[a])
    return hist, outside


def quantiles(counts, lo: float, bin_km: float) -> np.ndarray:
    """The quantiles at PROBS of one histogram: target = p N, j = the smallest bin with cum_j >= target,
    value = lo + w (j + (target - cum_{j-1}) / count_j)."""
    c = np.asarray(counts, np.int64)
    cum = np.cumsum(c)
    N = int(cum[-1]) if len(c) else 0
    if N == 0:
        return np.full(len(PROBS), np.nan)
    lo, w = float(np.float32(lo)), float(np.float32(bin_km))
    out = []
    for p in PROBS:
        t = p * N
        j = int(np.argmax(cum >= t))
        prev = int(cum[j - 1]) if j else 0
        out.append(lo + w * (j + (t - prev) / int(c[j])))
    return np.array(out)


def mode(counts, lo: float, bin_km: float) -> float:
    """Centre of the fullest bin, the lowest index on a tie; NaN for an empty histogram."""
    c = np.asarray(counts)
    if c.sum() == 0:
        return math.nan
    return float(np.float32(lo)) + float(np.float32(bin_km)) * (int(np.argmax(c)) + 0.5)


def jacobi3(a) -> tuple[np.ndarray, np.ndarray]:
    """Cyclic Jacobi on a symmetric 3 x 3 matrix, as the device runs it: -> eigenvalues [3] (unsorted), vectors [3, 3]
    (columns)."""
    a = [[float(a[i][j]) for j in range(3)] for i in range(3)]
    v = [[1.0 if i == j else 0.0 for j in range(3)] for i in range(3)]
    for sweep in range(JACOBI_SWEEPS):
        if a[0][1] == 0.0 and a[0][2] == 0.0 and a[1][2] == 0.0:
            break
        for p, q in ((0, 1), (0, 2), (1, 2)):
            o = 3 - p - q
            apq = a[p][q]
            if apq == 0.0:
                continue
            g = 100.0 * abs(apq)
            if sweep > 3 and abs(a[p][p]) + g == abs(a[p][p]) and abs(a[q][q]) + g == abs(a[q][q]):
                a[p][q] = a[q][p] = 0.0
                continue
            hd = a[q][q] - a[p][p]
            if abs(hd) + g == abs(hd):
                t = apq / hd
            else:
                theta = 0.5 * hd / apq
                t = 1.0 / (abs(theta) + math.sqrt(1.0 + theta * theta))
                if theta < 0.0:
                    t = -t
            c = 1.0 / math.sqrt(1.0 + t * t)
            s = t * c
            tau = s / (1.0 + c)
            h = t * apq
            a[p][p] -= h
            a[q][q] += h
            a[p][q] = a[q][p] = 0.0
            gp, gq = a[o][p], a[o][q]
            a[o][p] = a[p][o] = gp - s * (gq + gp * tau)
            a[o][q] = a[q][o] = gq + s * (gp - gq * tau)
            for k in range(3):
                vp, vq = v[k][p], v[k][q]
                v[k][p] = vp - s * (vq + vp * tau)
                v[k][q] = vq + s * (vp - vq * tau)
    return np.array([a[0][0], a[1][1], a[2][2]]), np.array(v)


def sign_rule(v) -> np.ndarray:
    """v with v_z >= 0; v_y >= 0 when v_z == 0; v_x >= 0 when both are 0."""
    x, y, z = (float(t) for t in v)
    if z < 0.0 or (z == 0.0 and (y < 0.0 or (y == 0.0 and x < 0.0))):
        x, y, z = -x, -y, -z
    return np.array([x, y, z])


def ellipsoid(cov3) -> tuple[np.ndarray, np.ndarray]:
    """1-sigma semi-axes (descending; a negative rounding residue gives 0) and unit axis vectors [axis, xyz] of a 3 x 3
    covariance.  Multiply the axes by sqrt(chi2_3(P)) for confidence level P."""
    lam, vec = jacobi3(cov3)
    order = [0, 1, 2]
    for i in range(2):                     # the device's bubble sort: descending, the lower index first on a tie
        for j in range(2 - i):
            if lam[order[j + 1]] > lam[order[j]]:
                order[j], order[j + 1] = order[j + 1], order[j]
    axes = np.array([math.sqrt(lam[c]) if lam[c] > 0.0 else 0.0 for c in order])
    dirs = np.array([sign_rule(vec[:, c]) for c in order])
    return axes, dirs


def azimuth_plunge(v) -> tuple[float, float]:
    """Azimuth (degrees clockwise from +y, in [0, 360)) and plunge (degrees towards +z, down) of an axis vector signed by
    sign_rule (plunge in [0, 90])."""
    x, y, z = (float(t) for t in v)
    az = math.degrees(math.atan2(x, y))
    if az < 0.0:
        az += 360.0
    if az >= 360.0:
        az -= 360.0
    return az, math.degrees(math.atan2(z, math.hypot(x, y)))


def stack(accs: list[dict]) -> dict:
    """Accumulators with a chain axis (the shapes of mq_hypo_chains) from per-chain dicts of `accumulate`."""
    return {k: np.stack([np.asarray(a[k]) for a in accs]) for k in ("ref", "sum", "cross", "n_models")}


def summarise(hist, ref, sum, cross, n_models, lo, bin_km, n_bins, **_ignored) -> dict:
    """mean [ne, 4], cov [ne, 4, 4], quant [ne, 3, 5], mode [ne, 3], axes [ne, 3], axis_dir [ne, 3, 3] and n_models (N)
    from the accumulators (ref / sum [n, 4, ne], cross [n, 10, ne], n_models [n], hist [ne, sum n_bins])."""
    ref, S, Cx = np.asarray(ref, np.float64), np.asarray(sum, np.float64), np.asarray(cross, np.float64)
    nm = np.asarray(n_models, np.int64)
    ne = ref.shape[2]
    N, A, W = 0.0, np.zeros((4, ne)), np.zeros((10, ne))
    for c in range(len(nm)):
        n = float(nm[c])
        if n == 0.0:
            continue
        N += n
        A += n * ref[c] + S[c]
        for p, (i, j) in enumerate(PAIRS):
            W[p] += Cx[c, p] - S[c, i] * S[c, j] / n
    mean = (A / N).T if N > 0 else np.full((ne, 4), np.nan)
    B = np.zeros((10, ne))
    if N > 0:
        for c in range(len(nm)):
            n = float(nm[c])
            if n == 0.0:
                continue
            d = ref[c] + S[c] / n - mean.T
            for p, (i, j) in enumerate(PAIRS):
                B[p] += n * (d[i] * d[j])
    cov = np.full((ne, 4, 4), np.nan)
    axes, dirs = np.full((ne, 3), np.nan), np.full((ne, 3, 3), np.nan)
    if N > 1:
        for p, (i, j) in enumerate(PAIRS):
            cov[:, i, j] = cov[:, j, i] = (W[p] + B[p]) / (N - 1.0)
        for e in range(ne):
            axes[e], dirs[e] = ellipsoid(cov[e, :3, :3])
    hist = np.asarray(hist)
    nb = [int(b) for b in n_bins]
    quant, md = np.full((ne, 3, 5), np.nan), np.full((ne, 3), np.nan)
    off = 0
    for a in range(3):
        for e in range(ne):
            h = hist[e, off:off + nb[a]]
            quant[e, a] = quantiles(h, lo[a], bin_km)
            md[e, a] = mode(h, lo[a], bin_km)
        off += nb[a]
    return dict(mean=mean, cov=cov, quant=quant, mode=md, axes=axes, axis_dir=dirs, n_models=int(N))
