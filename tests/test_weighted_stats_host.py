"""CPU tests of weighted ensemble statistics: the weighted reference against the unweighted one (all-ones weights,
replicated members), stats.integer_weights, the argument checks of stat_weight= in the Python layer, and the C ABI's
weighted entry points (binding and NULL-weight rejection)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import concentrations as conc
from fiveeqscm_b200 import params as P
from fiveeqscm_b200 import stats as S
from tests.group_stats_ref import grouped_temperature_stats, plant_non_finite
from tests.weighted_stats_ref import weighted_temperature_stats, weights_with_extremes

WMAX = 2 ** 32 - 1


def _T(n_t, M, seed, dtype=np.float64):
    rng = np.random.default_rng(seed)
    return (rng.normal(1.5, 0.8, size=(n_t, M)) + np.linspace(0, 2, n_t)[:, None]).astype(dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("G", [1, 4, 13])
def test_all_ones_weights_are_the_unweighted_reference(dtype, G):
    n_t, M = 7, 3001
    T = plant_non_finite(_T(n_t, M, 1, dtype), -1.0, 6.0, 28)
    labels = np.random.default_rng(2).integers(-1, G + 1, M)     # negatives and labels >= G count nowhere
    h, m = grouped_temperature_stats(T, -1.0, 6.0, 28, labels, G)
    hw, mw = weighted_temperature_stats(T, -1.0, 6.0, 28, labels, G, np.ones(M, dtype=np.uint32))
    assert hw.dtype == np.uint64 and np.array_equal(hw, h)
    np.testing.assert_array_equal(mw, m)                           # NaN where NaN, bit for bit elsewhere


def test_pooled_reference_takes_no_labels():
    T = _T(5, 700, 3)
    w = np.random.default_rng(4).integers(0, 5, 700)
    a = weighted_temperature_stats(T, -1.0, 6.0, 64, None, 1, w)
    b = weighted_temperature_stats(T, -1.0, 6.0, 64, np.zeros(700), 1, w)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_weight_k_is_k_copies_of_the_member(dtype):
    """Counts exactly those of the ensemble with member m repeated w[m] times; moments to summation order; weight 0
    is the member left out, min and max included."""
    n_t, M, G = 9, 2000, 5
    T = _T(n_t, M, 5, dtype)
    rng = np.random.default_rng(6)
    w = rng.integers(0, 6, M)
    w[:50] = 0
    T[:, :50] = 100.0                                              # weight 0: out of max (and the last bin)
    labels = rng.integers(-1, G, M)
    rep = np.repeat(np.arange(M), w)
    h_rep, m_rep = grouped_temperature_stats(T[:, rep], -1.0, 6.0, 200, labels[rep], G)
    h, m = weighted_temperature_stats(T, -1.0, 6.0, 200, labels, G, w)
    assert np.array_equal(h, h_rep)
    assert h.sum() == n_t * int(w[(labels >= 0)].sum())
    np.testing.assert_array_equal(m[..., 2:], m_rep[..., 2:])
    np.testing.assert_allclose(m[..., :2], m_rep[..., :2], rtol=1e-12)
    assert (m[..., 3] < 100.0).all()


def test_weights_with_extremes_reach_the_bound():
    w = weights_with_extremes(3001, 1)
    assert w.dtype == np.uint32 and int(w.astype(np.int64).sum()) == WMAX
    assert (w == 0).any() and (w == 1).any() and int(w.max()) > 2 ** 30
    T = _T(3, 3001, 2)
    h, _ = weighted_temperature_stats(T, -1.0, 6.0, 16, None, 1, w)
    assert (h.sum(axis=-1) == WMAX).all()


def test_integer_weights_rounds_half_up_elementwise():
    w = np.array([0.0, 0.49, 0.5, 1.0, 1.5, 2.4999, 7.25])
    got = S.integer_weights(w, 2.0)
    assert got.dtype == np.int64 and got.tolist() == [0, 1, 1, 2, 3, 5, 15]
    assert S.integer_weights(w, 1.0).tolist() == [0, 0, 1, 1, 2, 2, 7]
    t = S.integer_weights(torch.from_numpy(w), 2.0)
    assert isinstance(t, torch.Tensor) and t.dtype == torch.int64 and t.tolist() == got.tolist()
    assert S.integer_weights(w.astype(np.float32), 2.0).tolist() == got.tolist()
    assert S.integer_weights(np.zeros(0), 3.0).shape == (0,)
    # the largest weight that fits, and elementwise: a rank's slice gets its members' weights of the whole array
    assert S.integer_weights(np.array([WMAX / 10.0]), 10.0)[0] == WMAX
    big = np.random.default_rng(0).random(1000)
    assert np.array_equal(S.integer_weights(big, 1e6)[300:700], S.integer_weights(big[300:700], 1e6))
    # the resolution: members below 0.5 / scale are dropped, and so at most M / (2 scale) of the weight is lost
    lik = np.random.default_rng(1).random(5000) ** 8
    scale = 100.0
    q = S.integer_weights(lik, scale)
    assert (q[lik < 0.5 / scale] == 0).all()
    assert lik[q == 0].sum() <= lik.size / (2 * scale)
    assert np.abs(q / scale - lik).max() <= 0.5 / scale


@pytest.mark.parametrize("kind", ["numpy", "torch"])
def test_integer_weights_rejections(kind):
    wrap = (lambda a: a) if kind == "numpy" else torch.from_numpy
    for w, scale, match in ((np.array([1.0, np.nan]), 1.0, "NaN"), (np.array([1.0, -0.25]), 1.0, "negative"),
                            (np.array([1.0, np.inf]), 1.0, "2\\^32"), (np.array([WMAX + 0.5]), 1.0, "2\\^32"),
                            (np.array([1.0]), 0.0, "scale"), (np.array([1.0]), -2.0, "scale"),
                            (np.array([1.0]), np.inf, "scale"), (np.array([1.0]), np.nan, "scale")):
        with pytest.raises(ValueError, match=match):
            S.integer_weights(wrap(w), scale)


def _prep(M=9, **kw):
    """_prepare of a small host run, which checks every keyword before anything touches CUDA"""
    G, n_t = 3, 6
    E = np.random.default_rng(0).random((G, n_t, M))
    gp, tp = P.default_params(M)
    return conc._prepare(conc._HostArrays(np.float64), E, gp, tp, **kw)


def test_stat_weight_argument_errors_are_raised_before_any_cuda_work():
    M, spec = 9, conc.HistSpec(bins=16)
    ok = np.ones(M, dtype=np.int64)
    cases = [(dict(stat_weight=ok), "needs stats"),
             (dict(stats=spec, stat_weight=np.ones(M - 1, dtype=np.int64)), "one weight per member"),
             (dict(stats=spec, stat_weight=np.ones((M, 1), dtype=np.int64)), "one weight per member"),
             (dict(stats=spec, stat_weight=np.ones(M)), "integers"),
             (dict(stats=spec, stat_weight=np.ones(M, dtype=bool)), "integers"),
             (dict(stats=spec, stat_weight=torch.ones(M)), "integers"),
             (dict(stats=spec, stat_weight=np.r_[ok[:-1], -1]), "negative"),
             (dict(stats=spec, stat_weight=torch.tensor(np.r_[ok[:-1], -3])), "negative"),
             (dict(stats=spec, stat_weight=np.r_[ok[:-1], 2 ** 32]), "2\\^32 - 1"),
             (dict(stats=spec, stat_weight=np.array([1] * (M - 1) + [2 ** 64 - 1], dtype=np.uint64)), "2\\^32 - 1"),
             (dict(stats=spec, stat_weight=torch.tensor(np.r_[ok[:-1], 2 ** 40])), "2\\^32 - 1"),
             (dict(stats=spec, stat_weight=np.r_[np.zeros(M - 2, np.int64), WMAX, 1]), "sums to 4294967296"),
             (dict(stats=spec, stat_weight=np.full(M, 2 ** 31, dtype=np.uint32)), "sums to")]
    for kw, match in cases:
        with pytest.raises(ValueError, match=match):
            _prep(M, **kw)
    # uint64 beyond 2^63 through torch too (seen through int64)
    with pytest.raises(ValueError, match="2\\^32 - 1"):
        conc._check_weights(torch.tensor([1, 2 ** 63 + 5], dtype=torch.uint64), 2, spec)


def test_stat_weight_is_placed_as_the_runs_own_uint32_array():
    M, spec = 9, conc.HistSpec(bins=16)
    src = np.arange(M, dtype=np.int64)
    d, placed, _, _, _ = _prep(M, stats=spec, stat_weight=src)
    w = placed["stat_weight"]
    assert w.dtype == np.uint32 and w.flags.c_contiguous and w.tolist() == src.tolist()
    assert not np.shares_memory(w, src)
    assert "stat_weight" not in [f[0] for f in _abi.UfairDesc._fields_]     # carried beside the descriptor
    for x in (src.astype(np.uint32), torch.from_numpy(src), list(range(M)), src.astype(np.uint64)):
        assert _prep(M, stats=spec, stat_weight=x)[1]["stat_weight"].tolist() == src.tolist()
    # the largest total that fits
    top = np.r_[np.zeros(M - 1, np.int64), WMAX]
    assert int(_prep(M, stats=spec, stat_weight=top)[1]["stat_weight"][-1]) == WMAX
    assert "stat_weight" not in _prep(M, stats=spec)[1]
    assert conc.EnsembleResult().weighted is False


def test_binding_declares_the_weighted_entry_points():
    for name in ("ufair_stats_pass_weighted_f64", "ufair_stats_pass_weighted_f32", "ufair_run_host_weighted_f64",
                 "ufair_run_host_weighted_f32"):
        assert name in _abi.SIGNATURES
    assert len(_abi.SIGNATURES["ufair_stats_pass_weighted_f64"][1]) == 3
    assert len(_abi.SIGNATURES["ufair_run_host_weighted_f64"][1]) == 5


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_abi.lib_path()):
        import __graft_entry__ as g
        g.build()
    return _abi.lib()


def _desc(**kw):
    d = _abi.UfairDesc(n_gas=1, n_t=4, n_member=4, ld_member=4, stats=1, hist_bins=8, hist_copies=1, hist_lo=0.0,
                       hist_hi=1.0, hist_rows=4, hist_private=16, moments_private=16)
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def test_abi_rejects_a_null_weight_before_touching_the_device(lib):
    w = (ctypes.c_uint32 * 4)(1, 1, 1, 1)
    for fn in (lib.ufair_stats_pass_weighted_f64, lib.ufair_stats_pass_weighted_f32):
        assert fn(ctypes.byref(_desc()), None, None) == _abi.ERR_ARG
        assert b"weight is NULL" in lib.ufair_last_error()
        assert fn(ctypes.byref(_desc(n_member=0)), None, None) == _abi.ERR_ARG   # even with nothing to count
    ws = ctypes.c_void_p(1)   # rejected before the workspace is used
    for fn in (lib.ufair_run_host_weighted_f64, lib.ufair_run_host_weighted_f32):
        assert fn(ws, ctypes.byref(_desc()), None, 16, 16) == _abi.ERR_ARG
        assert b"weight is NULL" in lib.ufair_last_error()
        assert fn(ws, ctypes.byref(_desc(stats=0, n_member=0)), ctypes.addressof(w), None, None) == _abi.ERR_ARG
        assert b"stats == 1" in lib.ufair_last_error()


def test_abi_weighted_entry_points_keep_the_unweighted_rules(lib):
    """Every other fault: the unweighted twin's code and message."""
    w = (ctypes.c_uint32 * 4)(1, 1, 1, 1)
    labels = (ctypes.c_int32 * 4)()
    faults = (dict(n_stat_groups=-1), dict(n_stat_groups=4), dict(stats=0), dict(struct_size=8),
              dict(ld_member=3, n_member=3), dict(stat_group=ctypes.addressof(labels), n_stat_groups=2, out_T=None),
              dict(out_every=3))
    for kw in faults:
        for twin, weighted in ((lib.ufair_stats_pass_f64, lib.ufair_stats_pass_weighted_f64),
                               (lib.ufair_stats_pass_f32, lib.ufair_stats_pass_weighted_f32)):
            rc = twin(ctypes.byref(_desc(**kw)), None)
            msg = lib.ufair_last_error()
            assert rc != 0, kw
            assert weighted(ctypes.byref(_desc(**kw)), ctypes.addressof(w), None) == rc, kw
            assert lib.ufair_last_error() == msg, kw
    ws = ctypes.c_void_p(1)
    for kw in (dict(n_stat_groups=-1), dict(n_stat_groups=4), dict(struct_size=8), dict(alpha_mode=9)):
        for twin, weighted in ((lib.ufair_run_host_f64, lib.ufair_run_host_weighted_f64),
                               (lib.ufair_run_host_f32, lib.ufair_run_host_weighted_f32)):
            rc = twin(ws, ctypes.byref(_desc(**kw)), 16, 16)
            msg = lib.ufair_last_error()
            assert rc != 0, kw
            assert weighted(ws, ctypes.byref(_desc(**kw)), ctypes.addressof(w), 16, 16) == rc, kw
            assert lib.ufair_last_error() == msg, kw
