"""Reference for weighted ensemble statistics: :func:`tests.group_stats_ref.grouped_temperature_stats` with an integer
weight per member (include/ufair.h, ufair_stats_pass_weighted_*).  Member m adds weights[m] to its bin instead of 1
and enters the moments as wv = weights[m] * T (sum of wv, sum of wv * T); weight 0 counts it nowhere, min and max
included, like a negative label.  Binning and the non-finite rule are those of the unweighted reference."""
import numpy as np


def weighted_temperature_stats(T, lo, hi, bins, labels, n_groups, weights):
    """(hist uint64 [n_groups][n_t][bins], moments float64 [n_groups][n_t][4] = sum w T, sum w T^2, min, max).
    ``labels`` None pools every member in one group (n_groups must then be 1)."""
    T = np.asarray(T)
    ft = T.dtype.type
    n_t, M = T.shape
    lab = np.zeros(M, dtype=np.int64) if labels is None else np.asarray(labels, dtype=np.int64)
    w = np.asarray(weights).astype(np.uint64)
    inv_w = ft(ft(bins) / (ft(hi) - ft(lo)))
    x = (T - ft(lo)) * inv_w                                  # subtract, then multiply, each rounded
    nan = np.isnan(x)
    idx = np.clip(np.floor(np.where(nan, 0, x)), 0, bins - 1).astype(np.int64)
    member_in = (lab >= 0) & (lab < n_groups) & (w > 0)
    ok = ~nan & member_in[None, :]
    key = (np.where(member_in, lab, 0)[None, :] * n_t + np.arange(n_t)[:, None]) * bins + idx
    hist = np.zeros(n_groups * n_t * bins, dtype=np.uint64)
    np.add.at(hist, key[ok], np.broadcast_to(w, T.shape)[ok])
    T64 = T.astype(np.float64)
    mom = np.empty((n_groups, n_t, 4))
    mom[..., 0:2], mom[..., 2], mom[..., 3] = 0.0, np.inf, -np.inf
    for g in range(n_groups):
        sel = (lab == g) & (w > 0)
        Tg = T64[:, sel]
        if not Tg.shape[1]:
            continue
        wv = w[sel].astype(np.float64) * Tg                   # (double)w * v, rounded
        with np.errstate(invalid="ignore"):                   # inf + -inf in a sum is NaN, as on the device
            mom[g] = np.stack([wv.sum(axis=1), (wv * Tg).sum(axis=1), np.fmin.reduce(Tg, axis=1, initial=np.inf),
                               np.fmax.reduce(Tg, axis=1, initial=-np.inf)], axis=1)
    return hist.reshape(n_groups, n_t, bins), mom


def weights_with_extremes(M, seed, zeros=0.25, total=2 ** 32 - 1):
    """uint32 weights [M >= 64]: mostly 0..3 (about `zeros` of them 0), plus three large weights that bring the sum
    to exactly `total` (the largest sum one call may have)."""
    rng = np.random.default_rng(seed)
    w = rng.integers(1, 4, M).astype(np.int64)
    w[rng.random(M) < zeros] = 0
    rest = total - int(w.sum())
    w[7] += rest // 2
    w[40] += rest // 4
    w[M - 3] += rest - rest // 2 - rest // 4
    assert int(w.sum()) == total and w.max() <= 2 ** 32 - 1
    return w.astype(np.uint32)
