"""Reference for period means (include/ufair.h, out_every = k): row p is the sum of steps p k .. p k + k - 1 in step
order, starting from zero, in the rows' own precision, times (Real)(1.0 / k)."""
import numpy as np


def period_mean(x, k):
    """Per-step rows x[..., n_t, M] (any float dtype) -> period means [..., n_t / k, M] of the same dtype."""
    x = np.asarray(x)
    ft = x.dtype.type
    v = x.reshape(x.shape[:-2] + (x.shape[-2] // k, k, x.shape[-1]))
    s = np.zeros(v.shape[:-2] + v.shape[-1:], dtype=x.dtype)
    for j in range(k):
        s = s + v[..., j, :]
    return s * ft(1.0 / k)
