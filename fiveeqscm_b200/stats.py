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


def percentiles(hist, lo: float, hi: float, pcts):
    """Percentiles of T per time step from counts [..., n_t][bins] (leading axes: statistics groups); linear
    inside the bin.  Returns [..., n_t][len(pcts)]."""
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
    all rows go in one call); returns a device tensor [..., n_t][len(pcts)].  Bit-identical to the host version."""
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
    (``hist.sum(-1)``)."""
    m = _np(moments)
    if not np.isscalar(n_member):
        n_member = _np(n_member)
    mean = m[..., 0] / n_member
    var = np.maximum(m[..., 1] / n_member - mean * mean, 0.0)
    return mean, np.sqrt(var)
