"""Reference for grouped ensemble statistics: a per-group recount of T[n_t][M] with the kernel's binning rule
(the rule of oracle.ufair_oracle.temperature_stats, restated here for all groups in one pass).  Member m counts in
group labels[m] when 0 <= labels[m] < n_groups and nowhere otherwise; NaN is not binned."""
import numpy as np


def grouped_temperature_stats(T, lo, hi, bins, labels, n_groups):
    """(hist uint64 [n_groups][n_t][bins], moments float64 [n_groups][n_t][4] = sum, sumsq, min, max).
    An empty group has sum 0, min +inf and max -inf, as the device buffers are initialised."""
    T = np.asarray(T)
    ft = T.dtype.type
    n_t = T.shape[0]
    lab = np.asarray(labels, dtype=np.int64)
    inv_w = ft(ft(bins) / (ft(hi) - ft(lo)))
    x = (T - ft(lo)) * inv_w                                  # subtract, then multiply, each rounded
    nan = np.isnan(x)
    idx = np.clip(np.floor(np.where(nan, 0, x)), 0, bins - 1).astype(np.int64)
    member_in = (lab >= 0) & (lab < n_groups)
    ok = ~nan & member_in[None, :]
    key = (np.where(member_in, lab, 0)[None, :] * n_t + np.arange(n_t)[:, None]) * bins + idx
    hist = np.bincount(key[ok], minlength=n_groups * n_t * bins).reshape(n_groups, n_t, bins).astype(np.uint64)
    T64 = T.astype(np.float64)
    mom = np.empty((n_groups, n_t, 4))
    mom[..., 0:2], mom[..., 2], mom[..., 3] = 0.0, np.inf, -np.inf
    for g in range(n_groups):
        Tg = T64[:, lab == g]
        if Tg.shape[1]:
            mom[g] = np.stack([Tg.sum(axis=1), (Tg * Tg).sum(axis=1), Tg.min(axis=1), Tg.max(axis=1)], axis=1)
    return hist, mom
