"""CPU tests of grouped ensemble statistics: the per-group reference against the pooled oracle, the
post-processing with a leading group axis, the grouped summary frame, the two-rank gloo reduction of a 3-D
histogram, and argument checking in the C ABI and the Python layer."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import concentrations as conc
from fiveeqscm_b200 import stats as S
from oracle import ufair_oracle as o
from tests.group_stats_ref import grouped_temperature_stats, plant_non_finite

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _T(n_t, M, seed, dtype=np.float64):
    rng = np.random.default_rng(seed)
    return (rng.normal(1.5, 0.8, size=(n_t, M)) + np.linspace(0, 2, n_t)[:, None]).astype(dtype)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_grouped_reference_equals_a_loop_of_the_pooled_oracle_nan_outside_min_max(dtype):
    """Group by group, the grouped reference is the pooled oracle on the group's members, and both keep a NaN out of
    the histogram and out of min / max while it makes the sums NaN (the device's rule)."""
    n_t, M, G = 7, 5003, 13
    T = _T(n_t, M, 1, dtype)
    T[3, 17] = np.nan                                           # NaN is not binned
    labels = np.random.default_rng(2).integers(-2, G + 2, M)    # negatives and labels >= G count nowhere
    labels[labels == 5] = 6                                     # group 5 is empty
    hist, mom = grouped_temperature_stats(T, -1.0, 6.0, 300, labels, G)
    assert hist.shape == (G, n_t, 300) and mom.shape == (G, n_t, 4)
    for g in range(G):
        sel = labels == g
        if not sel.any():
            assert not hist[g].any() and (mom[g, :, :2] == 0).all()
            assert (mom[g, :, 2] == np.inf).all() and (mom[g, :, 3] == -np.inf).all()
            continue
        h, m = o.temperature_stats(T[:, sel], -1.0, 6.0, 300)
        assert np.array_equal(hist[g], h)
        np.testing.assert_array_equal(mom[g], m)
    g17 = int(labels[17])
    assert 0 <= g17 < G                                         # the NaN member is in a group
    Tg = T[3, labels == g17].astype(np.float64)
    assert np.isnan(mom[g17, 3, :2]).all()
    assert mom[g17, 3, 2] == np.nanmin(Tg) and mom[g17, 3, 3] == np.nanmax(Tg)
    # every member with a label in range counted once per step, except the NaN
    n_in = int(((labels >= 0) & (labels < G)).sum())
    assert (hist.sum(axis=(0, 2)) == n_in - (np.arange(n_t) == 3) * int(0 <= labels[17] < G)).all()


def test_percentiles_and_mean_std_take_a_leading_group_axis():
    G, n_t, M = 4, 9, 4000
    T = _T(n_t, M, 3)
    labels = np.arange(M) % G
    hist, mom = grouped_temperature_stats(T, -1.0, 6.0, 256, labels, G)
    p = S.percentiles(hist, -1.0, 6.0, (5, 50, 95))
    assert p.shape == (G, n_t, 3)
    n = hist.sum(axis=-1)
    mean, std = S.mean_std(mom, n)
    assert mean.shape == (G, n_t)
    for g in range(G):
        assert np.array_equal(p[g], S.percentiles(hist[g], -1.0, 6.0, (5, 50, 95)))
        mg, sg = S.mean_std(mom[g], int(n[g, 0]))
        assert np.array_equal(mean[g], mg) and np.array_equal(std[g], sg)
        np.testing.assert_allclose(mean[g], T[:, labels == g].mean(axis=1), rtol=1e-12)
    # the plain 2-D call is unchanged
    h2, m2 = o.temperature_stats(T, -1.0, 6.0, 256)
    assert S.percentiles(h2, -1.0, 6.0, (50,)).shape == (n_t, 1)
    assert np.array_equal(S.mean_std(m2, M)[0], m2[:, 0] / M)


def test_grouped_summary_frame():
    from fiveeqscm_b200 import frames
    from fiveeqscm_b200.concentrations import EnsembleResult, HistSpec
    G, n_t, M = 3, 12, 3000
    T = _T(n_t, M, 4)
    labels = np.arange(M) % 4 - 1                              # -1 = left out; groups of 750 members
    spec = HistSpec(lo=-1.0, hi=6.0, bins=200, groups=G)
    hist, mom = grouped_temperature_stats(T, spec.lo, spec.hi, spec.bins, labels, G)
    years = 2000 + np.arange(n_t)
    res = EnsembleResult(T=T, hist=hist.astype(np.int64), moments=mom, spec=spec, n_member=M, stat_group="scenario")
    sf = frames.summary_frame(res, years, pcts=(5, 50, 95), group_names=["ssp119", "ssp245", "ssp585"])
    assert list(sf.columns) == ["scenario", "year", "members", "T_mean", "T_std", "T_min", "T_max", "T_p5", "T_p50",
                                "T_p95"]
    assert len(sf) == G * n_t and (sf["members"] == 750).all()
    for g, name in enumerate(["ssp119", "ssp245", "ssp585"]):
        part = sf[sf["scenario"] == name]
        assert np.array_equal(part["year"], years)
        np.testing.assert_allclose(part["T_mean"], T[:, labels == g].mean(axis=1), rtol=1e-12)
        assert np.array_equal(part["T_max"], T[:, labels == g].max(axis=1))
        assert np.array_equal(part["T_p50"], S.percentiles(hist[g], spec.lo, spec.hi, (50,))[:, 0])
    res.stat_group = "labels"
    sf2 = frames.summary_frame(res, years, pcts=(50,))
    assert list(sf2.columns[:2]) == ["group", "year"] and list(sf2["group"].unique()) == [0, 1, 2]
    with pytest.raises(ValueError, match="group_names"):
        frames.summary_frame(res, years, group_names=["a"])


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
from fiveeqscm_b200 import dist as D
from tests.group_stats_ref import grouped_temperature_stats, plant_non_finite
rank, world = int(sys.argv[1]), int(sys.argv[2])
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=sys.argv[3], RANK=str(rank), WORLD_SIZE=str(world))
dist.init_process_group("gloo", rank=rank, world_size=world)
M, n_t, G = 1001, 30, 5
rng = np.random.default_rng(7)
T = rng.normal(1.0, 0.9, size=(n_t, M))
labels = rng.integers(-1, G, M)
lo, hi = D.shard_bounds(M, world, rank)
h, m = grouped_temperature_stats(T[:, lo:hi], -5.0, 25.0, 256, labels[lo:hi], G)
hist = torch.from_numpy(h.astype(np.int64)); mom = torch.from_numpy(m)
D.allreduce_stats(hist, mom)
h_all, m_all = grouped_temperature_stats(T, -5.0, 25.0, 256, labels, G)
assert hist.shape == (G, n_t, 256) and np.array_equal(hist.numpy().astype(np.uint64), h_all), "histogram"
assert np.allclose(mom.numpy()[..., :2], m_all[..., :2], rtol=1e-12)
assert np.array_equal(mom.numpy()[..., 2:], m_all[..., 2:])
dist.barrier(); dist.destroy_process_group()
print("RANK_OK", rank)
"""


def test_two_rank_gloo_reduction_of_grouped_statistics(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    port = str(31500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), "2", port], stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in range(2)]
    for r, p in enumerate(procs):
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0 and f"RANK_OK {r}" in out, err[-2000:]


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_abi.lib_path()):
        import __graft_entry__ as g
        g.build()
    return _abi.lib()


def test_abi_rejects_bad_group_arguments(lib):
    """Checked before anything touches the device."""
    labels = (ctypes.c_int32 * 4)()

    def desc(**kw):
        d = _abi.UfairDesc(n_gas=1, n_t=4, n_member=4, ld_member=4, stats=1, hist_bins=8, hist_copies=1, hist_lo=0.0,
                           hist_hi=1.0, hist_rows=4, hist_private=16, moments_private=16)
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    for kw, what in ((dict(n_stat_groups=-1), b"n_stat_groups"), (dict(n_stat_groups=_abi.MAX_STAT_GROUPS + 1), b"n_stat_groups"),
                     (dict(n_stat_groups=4), b"stat_group"), (dict(stats=0, stat_group=ctypes.addressof(labels)), b"stats == 0")):
        d = desc(**kw)
        for fn in (lib.ufair_run_f64, lib.ufair_stats_pass_f32, lib.ufair_stats_reset):
            assert fn(ctypes.byref(d), None) == _abi.ERR_ARG, (kw, fn)
            assert what in lib.ufair_last_error(), (kw, lib.ufair_last_error())
    d = desc(n_stat_groups=2, stat_group=ctypes.addressof(labels), hist_rows=2 ** 30)
    assert lib.ufair_stats_reset(ctypes.byref(d), None) == _abi.ERR_ARG and b"32 bits" in lib.ufair_last_error()
    ws = ctypes.c_void_p(1)   # rejected before the workspace is used
    assert lib.ufair_run_host_f64(ws, ctypes.byref(desc(n_stat_groups=3)), 16, 16) == _abi.ERR_ARG
    assert b"stat_group" in lib.ufair_last_error()


def test_python_group_resolution():
    H = conc.HistSpec
    assert conc._resolve_groups(None, None, False, 1) == (None, None)
    assert conc._resolve_groups(H(), None, True, 4) == (H(), None)
    spec, src = conc._resolve_groups(H(), "scenario", True, 4)
    assert (spec.groups, src) == (4, "scenario")
    assert conc._resolve_groups(H(groups=6), "scenario", True, 4)[0].groups == 6
    assert conc._resolve_groups(H(groups=3), np.zeros(5), False, 1) == (H(groups=3), "labels")
    for args, match in (((H(groups=2), None, True, 4), "needs stat_group"),
                        ((None, "scenario", True, 4), "needs stats"),
                        ((H(), "scenario", False, 1), "needs scen_idx"),
                        ((H(), "members", True, 4), "stat_group must be"),
                        ((H(), np.zeros(5), False, 1), "not inferred"),
                        ((H(groups=-1), np.zeros(5), False, 1), "groups must be"),
                        ((H(groups=_abi.MAX_STAT_GROUPS + 1), np.zeros(5), False, 1), "groups must be"),
                        ((H(), "scenario", True, _abi.MAX_STAT_GROUPS + 1), "at most")):
        with pytest.raises(ValueError, match=match):
            conc._resolve_groups(*args)
    conc._check_labels(2, 3, "x")
    with pytest.raises(ValueError, match="label 3 >= groups 3"):
        conc._check_labels(3, 3, "x")


def _same_moments(a, b):
    """min / max exactly, sum / sumsq to summation order (assert_allclose: NaN where the other has NaN, inf equal)"""
    np.testing.assert_array_equal(a[..., 2:], b[..., 2:])
    np.testing.assert_allclose(a[..., :2], b[..., :2], rtol=1e-12)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_one_rule_for_non_finite_temperatures(dtype):
    """NaN: not binned, not in min / max, makes sum and sumsq NaN; +-inf: edge bins and every moment.  The numpy
    oracle, the grouped reference and (for float64, which it bins in) the C oracle agree on it."""
    from oracle import c_oracle as co
    lo, hi, bins = -1.0, 6.0, 28
    T = plant_non_finite(_T(6, 257, 5, dtype), lo, hi, bins)
    n_t, M = T.shape
    hist, mom = o.temperature_stats(T, lo, hi, bins)
    fin = np.where(np.isfinite(T), T, np.nan).astype(np.float64)
    nan = np.isnan(T)
    assert (hist.sum(axis=1) == M - nan.sum(axis=1)).all()
    assert hist[0, -1] >= 1 and hist[0, 0] >= 1 and hist[2, -1] >= 1 and hist[2, 0] >= 1     # infinities: edge bins
    assert hist[1, 0] >= 1 and hist[1, -1] >= 2                             # lo -> bin 0; hi and hi - 1 ulp -> last bin
    assert not hist[3].any()
    assert np.array_equal(np.isnan(mom[:, 0]), nan.any(axis=1) | (np.isposinf(T).any(axis=1) & np.isneginf(T).any(axis=1)))
    assert np.isnan(mom[[0, 3, 4], 1]).all() and mom[2, 1] == np.inf
    assert mom[0, 2] == -np.inf and mom[0, 3] == np.inf and mom[4, 3] == np.inf
    assert mom[3, 2] == np.inf and mom[3, 3] == -np.inf                     # all-NaN: the sentinels
    assert mom[1, 2] == np.nanmin(fin[1]) and mom[1, 3] == np.nanmax(fin[1])
    assert mom[5, 0] == -np.inf and mom[5, 1] == np.inf and mom[5, 2] == -np.inf and mom[5, 3] == np.nanmax(fin[5])
    mean, _ = S.mean_std(mom, hist.sum(axis=1))
    assert np.isnan(mean[[0, 2, 3, 4]]).all() and np.isfinite(mean[1]) and mean[5] == -np.inf
    gh, gm = grouped_temperature_stats(T, lo, hi, bins, np.zeros(M, dtype=np.int32), 1)
    assert np.array_equal(gh[0], hist)
    _same_moments(gm[0], mom)
    if dtype == np.float64:
        ch, cm = co.temperature_stats(T, lo, hi, bins)
        assert np.array_equal(ch, hist)
        _same_moments(cm, mom)
    # grouped: every group sees the rule, an empty group keeps the empty identities
    lab = np.arange(M) % 4
    lab[lab == 3] = -1
    gh, gm = grouped_temperature_stats(T, lo, hi, bins, lab, 4)
    for g in range(3):
        h, m = o.temperature_stats(T[:, lab == g], lo, hi, bins)
        assert np.array_equal(gh[g], h)
        _same_moments(gm[g], m)
    assert not gh[3].any() and (gm[3, :, :2] == 0).all() and (gm[3, :, 2] == np.inf).all() and (gm[3, :, 3] == -np.inf).all()
