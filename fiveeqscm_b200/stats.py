"""Ensemble statistics read off the per-step temperature histograms / moments (SURVEY.md 8 a8).

Pure array post-processing of what the kernel produced (works on numpy arrays or torch tensors
moved to numpy); the histogram itself is built on the GPU inside the integrator.
"""
from __future__ import annotations

import numpy as np


def _np(x):
    try:
        import torch
        if isinstance(x, torch.Tensor):
            return x.detach().cpu().numpy()
    except ImportError:  # pragma: no cover
        pass
    return np.asarray(x)


def _torch_of(x):
    """The torch module if x is a torch tensor, else None."""
    try:
        import torch
    except ImportError:  # pragma: no cover
        return None
    return torch if isinstance(x, torch.Tensor) else None


WEIGHT_MAX = 2 ** 32 - 1   # the largest member weight, and the largest sum of one call's weights (include/ufair.h)


def integer_weights(w, scale: float):
    """Integer member weights for ``run_ensemble(stat_weight=)`` from real ones (e.g. likelihoods):
    ``floor(w * scale + 0.5)`` elementwise, in float64.  Elementwise, so every rank of a multi-GPU run that uses the
    same ``scale`` agrees on each member's weight.  Works on numpy arrays (returns int64 numpy) and torch tensors
    (returns int64 on the same device).

    Resolution: a weight is rounded to a multiple of 1 / ``scale``, at most 0.5 / ``scale`` off.  A member whose
    weight rounds to 0 (w < 0.5 / scale) is dropped, so the total weight lost that way is at most M / (2 scale) for
    M members.  Choose ``scale`` so that the sum of the results stays <= 2^32 - 1 (``run_ensemble`` checks it), e.g.
    ``scale = (2**32 - 1) / w.sum() * 0.999`` for weights normalised to their total.

    Raises ValueError for a NaN or negative weight, a non-positive or non-finite ``scale``, and a result > 2^32 - 1."""
    scale = float(scale)
    if not (scale > 0 and np.isfinite(scale)):
        raise ValueError(f"scale must be finite and > 0, got {scale!r}")
    torch = _torch_of(w)
    if torch is not None:   # one synchronise for the three checks
        x = w.to(torch.float64)
        q = torch.floor(x * scale + 0.5)
        top = q.nan_to_num(0.0).max() if q.numel() else x.new_zeros(())
        bad_nan, bad_neg, top = torch.stack([torch.isnan(x).any(), (x < 0).any(), top]).tolist()
    else:
        x = np.asarray(w, dtype=np.float64)
        q = np.floor(x * scale + 0.5)
        bad_nan, bad_neg = bool(np.isnan(x).any()), bool((x < 0).any())
        top = float(np.nan_to_num(q, nan=0.0).max()) if q.size else 0.0
    if bad_nan:
        raise ValueError("integer_weights: a weight is NaN")
    if bad_neg:
        raise ValueError("integer_weights: a weight is negative")
    if top > WEIGHT_MAX:
        raise ValueError(f"integer_weights: a weight times scale rounds to {top:.6g} > 2^32 - 1; lower the scale")
    return q.to(torch.int64) if torch is not None else q.astype(np.int64)


def percentiles(hist, lo: float, hi: float, pcts):
    """Percentiles of T per time step from counts [..., n_t][bins] (leading axes: statistics groups); linear
    inside the bin.  Returns [..., n_t][len(pcts)].  For a weighted run (``stat_weight=``) the counts are weight
    totals, and these are the weighted percentiles."""
    h = _np(hist).astype(np.float64)
    lead = h.shape[:-1]
    h = h.reshape(-1, h.shape[-1])
    n_t, bins = h.shape
    w = (hi - lo) / bins
    cdf = np.cumsum(h, axis=1)
    tot = cdf[:, -1]
    rows = np.arange(n_t)
    out = np.empty((n_t, len(pcts)))
    for j, pct in enumerate(pcts):
        target = tot * (pct / 100.0)
        k = np.minimum((cdf < target[:, None]).sum(axis=1), bins - 1)
        prev = np.where(k > 0, cdf[rows, np.maximum(k - 1, 0)], 0.0)
        cnt = h[rows, k]
        frac = np.where(cnt > 0, (target - prev) / np.where(cnt > 0, cnt, 1.0), 0.0)
        out[:, j] = lo + (k + np.clip(frac, 0.0, 1.0)) * w
    return out.reshape(lead + (len(pcts),))


def percentiles_device(hist, lo: float, hi: float, pcts):
    """Same as :func:`percentiles`, computed on the GPU (libufair `ufair_hist_percentiles`) from a
    device histogram [..., n_t][bins] (int64 counts, e.g. the all-reduced one; leading axes are statistics groups,
    all rows go in one call); returns a device tensor [..., n_t][len(pcts)].  Bit-identical to the host version.
    Counts are weight totals when the run was weighted (``stat_weight=``)."""
    import torch

    from . import _abi
    if not (isinstance(hist, torch.Tensor) and hist.is_cuda and hist.dtype == torch.int64):
        raise ValueError("hist must be a CUDA int64 tensor [..., n_t][bins]")
    lead = tuple(hist.shape[:-1])
    h = hist.contiguous().reshape(-1, hist.shape[-1])
    p = torch.as_tensor(list(pcts), dtype=torch.float64, device=h.device)
    out = torch.empty(h.shape[0], p.numel(), dtype=torch.float64, device=h.device)
    with torch.cuda.device(h.device):
        _abi.check(_abi.lib().ufair_hist_percentiles(h.data_ptr(), h.shape[0], h.shape[1], float(lo), float(hi),
                                                     p.data_ptr(), p.numel(), out.data_ptr(),
                                                     torch.cuda.current_stream(h.device).cuda_stream))
    return out.reshape(*lead, p.numel())


def mean_std(moments, n_member):
    """(mean, std) per step from moments [..., n_t][4] = sum, sumsq, min, max.  ``n_member``: the member count,
    or an array of per-row counts [..., n_t] -- for grouped statistics a group's histogram row sums
    (``hist.sum(-1)``).  For a weighted run (``stat_weight=``) pass ``hist.sum(-1)``, the weight totals: the moments
    hold sum w T and sum w T^2, so these are the weighted mean and the weighted (population) std."""
    m = _np(moments)
    if not np.isscalar(n_member):
        n_member = _np(n_member)
    mean = m[..., 0] / n_member
    var = np.maximum(m[..., 1] / n_member - mean * mean, 0.0)
    return mean, np.sqrt(var)
