"""Reference for grouped ensemble statistics: a per-group recount of T[n_t][M] with the kernel's binning rule
(the rule of oracle.ufair_oracle.temperature_stats, restated here for all groups in one pass).  Member m counts in
group labels[m] when 0 <= labels[m] < n_groups and nowhere otherwise.  Non-finite T follows the same rule as the
pooled oracle: NaN is neither binned nor in min / max but makes the sums NaN; +-inf land in the edge bins and enter
every moment."""
import numpy as np


def grouped_temperature_stats(T, lo, hi, bins, labels, n_groups):
    """(hist uint64 [n_groups][n_t][bins], moments float64 [n_groups][n_t][4] = sum, sumsq, min, max).
    An empty group (or an all-NaN step) has min +inf and max -inf, as the device buffers are initialised; an empty
    group has sum 0."""
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
            mom[g] = np.stack([Tg.sum(axis=1), (Tg * Tg).sum(axis=1), np.fmin.reduce(Tg, axis=1, initial=np.inf),
                               np.fmax.reduce(Tg, axis=1, initial=-np.inf)], axis=1)
    return hist, mom


def plant_non_finite(T, lo, hi, bins):
    """Overwrite entries of T[n_t >= 6][M >= 256] (in place; returned) with the values the binning and the moments
    must handle: NaN, +-inf, exactly lo, exactly hi, one ulp below hi and inner bin edges, both infinities in one
    step, and an all-NaN step (3).  Bin edges are exact when (hi - lo) / bins is a power of two."""
    ft = T.dtype.type
    w = (hi - lo) / bins
    T[0, 3], T[0, 10], T[0, 11] = np.nan, np.inf, -np.inf
    T[1, 0], T[1, 1], T[1, 2] = ft(lo), ft(hi), np.nextafter(ft(hi), ft(-np.inf))
    T[1, 3:8] = [ft(lo + k * w) for k in (1, 4, 7, bins // 2, bins - 1)]
    T[2, 100], T[2, 101] = np.inf, -np.inf
    T[3, :] = np.nan
    T[4, 200], T[4, 201] = np.nan, np.inf
    T[5, 255] = -np.inf
    return T
