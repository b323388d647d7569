"""Weighted ensemble statistics on the device: weighted counts against a recount of the kernel's own T, the unweighted
pass reproduced by all-ones weights and by 0/1 weights against negative labels, replicated members, determinism, the
host pipeline, member chunks into one set of private buffers, the packed reduction, period means, non-finite
temperatures, guard bands around the private buffers, and argument errors."""
import ctypes as C

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import params as P
from tests.group_stats_ref import plant_non_finite
from tests.test_gpu_guard import POISON64, _desc_and_buffers
from tests.util import ensemble, to_dev, to_np
from tests.weighted_stats_ref import weighted_temperature_stats, weights_with_extremes

pytestmark = pytest.mark.gpu

WMAX = 2 ** 32 - 1


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    from fiveeqscm_b200 import concentrations as c
    _abi.lib()
    return c


def _plan(api, M, n_t, prec, spec, stat_group, weight, seed=5, gp_idx=None, **kw):
    """Sampler -> integrator with T output and weighted statistics, on the device.  gp_idx: the members of the
    sampled ensemble to run (repeats allowed)."""
    gp, tp, esc, scen = P.sample_on_device(M, seed, precision=prec)
    if gp_idx is not None:
        gp, tp, esc, scen = gp[..., gp_idx], tp[:, gp_idx], esc[:, gp_idx], scen[gp_idx]
    return api.DevicePlan(to_dev(P.scenario_emissions(n_t)), gp.contiguous(), tp.contiguous(),
                          scen_idx=scen.contiguous(), e_scale=esc.contiguous(), stats=spec, stat_group=stat_group,
                          stat_weight=weight, outputs=("T",), return_state=False, precision=prec, **kw)


def _labels(M, G, seed):
    return np.random.default_rng(seed).integers(-1, G, M).astype(np.int32)


def _grouping(api, M, G, seed):
    """(stat_group argument, HistSpec groups, labels for the reference or None): pooled (G == 0), the four scenario
    groups (G == "s") or G random groups with negative labels."""
    if G == 0:
        return None, 0, None
    if G == "s":
        return "scenario", 0, None
    lab = _labels(M, G, seed)
    return lab, G, lab


def _lead(res):
    """hist, moments with a leading group axis"""
    h, m = to_np(res.hist), to_np(res.moments)
    return (h, m) if h.ndim == 3 else (h[None], m[None])


def _check_moments(mom, ref, T, labels, w):
    """min / max exact; sum within 1e-12 of sum w |T| of the group, sum of squares within 1e-12 relative"""
    assert np.array_equal(mom[..., 2:], ref[..., 2:]), "min / max exact"
    G = ref.shape[0]
    lab = np.zeros(T.shape[1], dtype=np.int64) if labels is None else labels
    wf = w.astype(np.float64)
    cnt = [(lab == g) & (w > 0) for g in range(G)]
    absw = np.stack([(np.abs(T[:, c].astype(np.float64)) * wf[c]).sum(axis=1) for c in cnt])
    assert np.all(np.abs(mom[..., 0] - ref[..., 0]) <= 1e-12 * absw), "sum"
    assert np.all(np.abs(mom[..., 1] - ref[..., 1]) <= 1e-12 * ref[..., 1]), "sum of squares"


def _bits(x):
    return to_np(x).view(np.uint64) if hasattr(x, "detach") else np.asarray(x).view(np.uint64)


CASES = [  # prec, out_dtype, M, grouping (0 pooled, "s" four scenarios, else labels with negatives), bins, copies
    ("f64", None, 3001, 0, 256, 3),
    ("f64", None, 5003, "s", 1024, 5),
    ("f32", None, 4099, 4, 512, 3),
    ("f64", "f32", 4001, 16, 300, 4),
    ("f32", None, 2999, 16, 128, 2),
    ("f64", "f32", 1999, 0, 512, 3),
    ("f64", None, 3001, 0, 20000, 3),     # past the 16 384-slot shared-memory budget: global atomics, pooled
    ("f32", None, 2001, 4, 8192, 2),      # 4 x 8192 slots: global atomics, 4-group tile
    ("f64", None, 2003, 16, 4096, 3),     # 8 x 4096 slots: global atomics, 8-group tile
]


@pytest.mark.parametrize("prec,out_dtype,M,G,bins,copies", CASES, ids=lambda v: str(v))
def test_weighted_counts_equal_a_recount_of_the_kernels_T(api, prec, out_dtype, M, G, bins, copies):
    """Weights 0, 1..3 and three large ones, summing to exactly 2^32 - 1 (the most one call may count)."""
    import torch
    n_t = 41
    w = weights_with_extremes(M, seed=M)
    stat_group, groups, lab = _grouping(api, M, G, seed=M + 1)
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=bins, copies=copies, groups=groups)
    plan = _plan(api, M, n_t, prec, spec, stat_group, to_dev(w), out_dtype=out_dtype)
    res = plan.run()
    torch.cuda.synchronize()
    assert res.weighted and plan.stat_weight.dtype == torch.uint32
    T = to_np(res.T)
    assert T.dtype == (np.float32 if "f32" in (prec, out_dtype) else np.float64)
    if G == "s":
        lab = to_np(plan.scen_idx)
    ng = 1 if G == 0 else (4 if G == "s" else G)
    h_ref, m_ref = weighted_temperature_stats(T, spec.lo, spec.hi, bins, lab, ng, w)
    hist, mom = _lead(res)
    assert hist.shape == (ng, n_t, bins) and res.hist.dtype == torch.int64
    assert np.array_equal(hist.astype(np.uint64), h_ref)
    _check_moments(mom, m_ref, T, lab, w)
    if G == 0:
        assert (hist.sum(axis=-1) == WMAX).all()      # every T finite: each row counts the whole weight


@pytest.mark.parametrize("prec,G,bins", [("f64", 0, 512), ("f32", 0, 512), ("f64", "s", 512), ("f32", 13, 300),
                                         ("f64", 0, 20000), ("f64", 13, 4096)], ids=lambda v: str(v))
def test_all_ones_weights_are_the_unweighted_pass_bit_for_bit(api, prec, G, bins):
    import torch
    M, n_t = 4001, 37
    stat_group, groups, _ = _grouping(api, M, G, seed=3)
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=bins, copies=5, groups=groups)
    plain = _plan(api, M, n_t, prec, spec, stat_group, None).run()
    wplan = _plan(api, M, n_t, prec, spec, stat_group, torch.ones(M, dtype=torch.int64, device="cuda"))
    ones = wplan.run()
    torch.cuda.synchronize()
    assert not plain.weighted and ones.weighted
    assert torch.equal(ones.T, plain.T) and torch.equal(ones.hist, plain.hist)
    assert np.array_equal(_bits(ones.moments), _bits(plain.moments))
    # the plan's weights are its own buffer: overwritten in place, a re-run takes them
    wplan.stat_weight.view(torch.int32).fill_(2)
    twos = wplan.run()
    torch.cuda.synchronize()
    assert torch.equal(twos.hist, 2 * plain.hist)


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("G", [0, 4, 13])
def test_zero_one_weights_are_negative_labels(api, prec, G):
    """Weight 0 counts a member nowhere, exactly like a negative label; weight 1 like its own label."""
    import torch
    M, n_t = 3001, 29
    w = (np.random.default_rng(G + 7).random(M) < 0.6).astype(np.int32)
    lab = _labels(M, G, 8) if G else np.zeros(M, dtype=np.int32)
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=256, copies=4, groups=G)
    weighted = _plan(api, M, n_t, prec, spec, lab if G else None, to_dev(w)).run()
    by_label = _plan(api, M, n_t, prec, api.HistSpec(lo=-0.5, hi=3.5, bins=256, copies=4, groups=max(G, 1)),
                     np.where(w == 0, -1, lab).astype(np.int32), None).run()
    torch.cuda.synchronize()
    hw, mw = _lead(weighted)
    hl, ml = _lead(by_label)
    assert np.array_equal(hw, hl) and np.array_equal(mw.view(np.uint64), ml.view(np.uint64))


@pytest.mark.parametrize("G", [0, "s"])
def test_weight_k_is_k_copies_of_the_member(api, G):
    """A weighted run's histogram and device percentiles are those of the unweighted run in which member m appears
    weight[m] times (same parameters, so the same T), bit for bit."""
    import torch
    from fiveeqscm_b200 import stats
    M, n_t, seed = 1500, 45, 12
    w = np.random.default_rng(2).integers(0, 4, M)
    rep = torch.from_numpy(np.repeat(np.arange(M), w)).cuda()
    stat_group = None if G == 0 else "scenario"
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=400, copies=3)
    a = _plan(api, M, n_t, "f64", spec, stat_group, to_dev(w), seed=seed, gas_form=None).run()
    b = _plan(api, M, n_t, "f64", spec, stat_group, None, seed=seed, gp_idx=rep, gas_form=None).run()
    torch.cuda.synchronize()
    assert torch.equal(b.T, a.T[:, rep]), "the duplicated members integrate to the same T"
    assert torch.equal(a.hist, b.hist)
    pcts = (5.0, 17.0, 50.0, 83.0, 95.0)
    pa, pb = stats.percentiles_device(a.hist, spec.lo, spec.hi, pcts), stats.percentiles_device(b.hist, spec.lo, spec.hi, pcts)
    torch.cuda.synchronize()
    assert torch.equal(pa, pb)
    assert torch.equal(a.moments[..., 2:], b.moments[..., 2:])
    assert torch.allclose(a.moments[..., :2], b.moments[..., :2], rtol=1e-12, atol=0)


def test_moments_are_deterministic(api):
    import torch
    M, n_t, G = 6007, 29, 13
    plan = _plan(api, M, n_t, "f64", api.HistSpec(lo=-0.5, hi=3.5, bins=256, groups=G), _labels(M, G, 1),
                 to_dev(weights_with_extremes(M, 3)))
    a = plan.run()
    h1, m1 = a.hist.clone(), a.moments.clone()
    b = plan.run()
    torch.cuda.synchronize()
    assert torch.equal(h1, b.hist) and np.array_equal(_bits(m1), _bits(b.moments))


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_host_pipeline_matches_the_device_path(api, prec):
    """Chunks of 384 members cut the weights (and their large entries) unevenly: the histogram and min / max are the
    device path's bit for bit, the sums to summation order (members fold into other copies)."""
    import torch
    M, n_t, G = 5003, 33, 6
    gp, tp, esc, scen = (to_np(x) for x in P.sample_on_device(M, 9, precision=prec))
    scen = np.ascontiguousarray(scen, dtype=np.int32)
    E = P.scenario_emissions(n_t)
    w = weights_with_extremes(M, 4)
    lab = _labels(M, G, 4)
    for stat_group, groups in ((None, 0), (lab, G), ("scenario", 0)):
        spec = api.HistSpec(lo=-0.5, hi=3.5, bins=300, copies=3, groups=groups)
        ws = api.Workspace(torch.cuda.current_device(), 384)
        try:
            host = api.run_ensemble(E, gp, tp, scen_idx=scen, e_scale=esc, stats=spec, stat_group=stat_group,
                                    stat_weight=w, outputs=("T",), return_state=False, workspace=ws, precision=prec)
        finally:
            ws.close()
        dev = api.run_ensemble(to_dev(E), to_dev(gp), to_dev(tp), scen_idx=to_dev(scen), e_scale=to_dev(esc),
                               stats=spec, stat_group=stat_group if not isinstance(stat_group, np.ndarray) else to_dev(lab),
                               stat_weight=to_dev(w), outputs=("T",), return_state=False, precision=prec)
        torch.cuda.synchronize()
        assert host.weighted and dev.weighted
        assert np.array_equal(host.hist, to_np(dev.hist))
        assert np.array_equal(host.moments[..., 2:], to_np(dev.moments)[..., 2:])
        np.testing.assert_allclose(host.moments[..., :2], to_np(dev.moments)[..., :2], rtol=1e-12)
        labels = None if stat_group is None else (scen if isinstance(stat_group, str) else lab)
        ng = 1 if stat_group is None else (4 if isinstance(stat_group, str) else G)
        h_ref, _ = weighted_temperature_stats(host.T, spec.lo, spec.hi, 300, labels, ng, w)
        assert np.array_equal(host.hist.reshape(h_ref.shape).astype(np.uint64), h_ref)


def test_member_chunks_accumulate_into_one_set_of_private_buffers(api):
    """Two weighted passes over member chunks [0, m1) and [m1, M), into the same private buffers, finalise to the
    whole run's histogram and min / max; the packed fold of the same buffers holds the counts exactly."""
    import torch
    L = _abi.lib()
    M, n_t, G, m1, bins = 5001, 23, 5, 2048, 300
    lab = _labels(M, G, 6)
    w = weights_with_extremes(M, 6)
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=bins, copies=3, groups=G)
    plan = _plan(api, M, n_t, "f64", spec, lab, to_dev(w))
    whole = plan.run()
    d = _abi.UfairDesc.from_buffer_copy(plan.desc)
    _abi.check(L.ufair_stats_reset(C.byref(d), None))
    wt = plan.stat_weight
    for lo, hi in ((0, m1), (m1, M)):
        dc = _abi.UfairDesc.from_buffer_copy(d)
        dc.n_member = hi - lo
        dc.out_T = d.out_T + lo * 8
        dc.stat_group = d.stat_group + lo * 4
        _abi.check(L.ufair_stats_pass_weighted_f64(C.byref(dc), wt.data_ptr() + lo * 4, None))
    rows = G * n_t
    hist = torch.empty(G, n_t, bins, dtype=torch.int64, device="cuda")
    mom = torch.empty(G, n_t, 4, dtype=torch.float64, device="cuda")
    _abi.check(L.ufair_stats_finalize(C.byref(d), hist.data_ptr(), mom.data_ptr(), None))
    sums = torch.empty(rows, bins + 2, dtype=torch.float64, device="cuda")
    ext = torch.empty(rows, 2, dtype=torch.float64, device="cuda")
    _abi.check(L.ufair_stats_finalize_packed(C.byref(d), sums.data_ptr(), ext.data_ptr(), None))
    h2 = torch.empty_like(hist)
    m2 = torch.empty_like(mom)
    _abi.check(L.ufair_stats_unpack(sums.data_ptr(), ext.data_ptr(), rows, bins, h2.data_ptr(), m2.data_ptr(), None))
    torch.cuda.synchronize()
    assert torch.equal(hist, whole.hist) and torch.equal(mom[..., 2:], whole.moments[..., 2:])
    assert torch.allclose(mom[..., :2], whole.moments[..., :2], rtol=1e-12, atol=0)
    # the packed layout: counts as exact doubles, then the sums; unpack gives the finalised buffers back
    assert torch.equal(sums[:, :bins], hist.reshape(rows, bins).to(torch.float64))
    assert torch.equal(sums[:, :bins].to(torch.int64), hist.reshape(rows, bins))
    assert torch.equal(sums[:, bins], mom.reshape(rows, 4)[:, 0]) and torch.equal(sums[:, bins + 1], mom.reshape(rows, 4)[:, 1])
    assert torch.equal(h2, hist) and np.array_equal(_bits(m2), _bits(mom))
    assert int(hist.sum(dim=(0, 2)).max()) <= WMAX


@pytest.mark.parametrize("G", [0, "s"])
def test_period_means_are_binned_weighted(api, G):
    import torch
    M, n_t, k = 3001, 40, 10
    w = weights_with_extremes(M, 9)
    stat_group, groups, lab = _grouping(api, M, G, 9)
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=256, copies=3, groups=groups)
    plan = _plan(api, M, n_t, "f64", spec, stat_group, to_dev(w), out_every=k)
    res = plan.run()
    torch.cuda.synchronize()
    T = to_np(res.T)
    assert T.shape == (n_t // k, M)
    if G == "s":
        lab = to_np(plan.scen_idx)
    h_ref, m_ref = weighted_temperature_stats(T, spec.lo, spec.hi, 256, lab, 1 if G == 0 else 4, w)
    hist, mom = _lead(res)
    assert np.array_equal(hist.astype(np.uint64), h_ref)
    _check_moments(mom, m_ref, T, lab, w)


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("G", [0, 3, 9], ids=["pooled", "G3", "G9"])
def test_non_finite_temperatures_follow_the_rule(api, prec, G):
    """plant_non_finite's NaN, +-inf, edge and all-NaN rows, written between the integrator and the weighted pass.
    The members with weight > 0 follow the unweighted rule; a NaN or inf on a weight-0 member changes nothing."""
    import torch
    from fiveeqscm_b200 import stats
    from oracle import ufair_oracle as o
    M, n_t, lo, hi, bins = 1003, 8, -1.0, 6.0, 28
    lab = _labels(M, G, 17) if G else None
    if G:
        lab[[3, 10, 11, 100, 101, 200, 201, 255]] = np.arange(8) % G     # every planted value in a group
    w = np.random.default_rng(5).integers(1, 5, M).astype(np.uint32)
    w[[3, 10, 101, 201]] = 0                       # NaN, +inf, -inf, +inf on weight-0 members
    w[::13] = 0
    spec = api.HistSpec(lo=lo, hi=hi, bins=bins, copies=3, groups=G)
    plan = _plan(api, M, n_t, prec, spec, lab, to_dev(w))
    plan.reset_stats()
    plan.launch()
    T = plant_non_finite(to_np(plan.result.T).copy(), lo, hi, bins)

    def stats_of(T):
        plan.reset_stats()
        plan.result.T.copy_(torch.from_numpy(T))
        plan.stats_pass()
        plan.finalize_stats()
        torch.cuda.synchronize()
        return _lead(plan.result)

    hist, mom = stats_of(T)
    h_ref, m_ref = weighted_temperature_stats(T, lo, hi, bins, lab, max(G, 1), w)
    assert np.array_equal(hist.astype(np.uint64), h_ref)
    assert np.array_equal(mom[..., 2:], m_ref[..., 2:]), "min / max exact"
    labs = np.zeros(M, dtype=np.int64) if lab is None else lab
    cnt = [(labs == g) & (w > 0) for g in range(max(G, 1))]   # the members that count: no NaN from weight-0 ones
    absw = np.stack([(np.abs(T[:, c].astype(np.float64)) * w[c]).sum(axis=1) for c in cnt])
    for j in (0, 1):
        got, want = mom[..., j], m_ref[..., j]
        fin = np.isfinite(want)
        assert np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(got[np.isinf(want)], want[np.isinf(want)])
        tol = 1e-12 * (absw if j == 0 else want)
        assert np.all(np.abs(got[fin] - want[fin]) <= tol[fin])
    assert not hist[:, 3].any() and (mom[:, 3, 2] == np.inf).all() and (mom[:, 3, 3] == -np.inf).all()
    pcts = (0.0, 5.0, 50.0, 95.0, 100.0)
    pd = to_np(stats.percentiles_device(plan.result.hist, lo, hi, pcts)).reshape(-1, n_t, len(pcts))
    for g in range(hist.shape[0]):
        assert np.array_equal(pd[g], o.percentiles_from_hist(hist[g], lo, hi, pcts)), g
    # the weight-0 members' values do not matter: finite ones there give the same bits
    T_fin = T.copy()
    T_fin[:, w == 0] = 1.0
    hist2, mom2 = stats_of(T_fin)
    assert np.array_equal(hist2, hist) and np.array_equal(mom2.view(np.uint64), mom.view(np.uint64))


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("Gs", [0, 11])
def test_weighted_buffers_stay_inside_their_rows(prec, Gs):
    import torch
    L = _abi.lib()
    M, n_t, bins, copies, ld = 1003, 19, 96, 3, 1008
    ens = ensemble(M, n_t=n_t, seed=13)
    d, b = _desc_and_buffers(ens, M, n_t, 3, ld, prec, True, outputs=("T",), stats=True)
    G = max(Gs, 1)
    lab = _labels(M, G, 2)
    labels = torch.from_numpy(lab).cuda()
    w = weights_with_extremes(M, 2)
    # the weights inside a poisoned allocation too: the pass reads [n_member] of them and writes none
    wfull = np.full(M + 64, 0x5EADBEEF, dtype=np.uint32)
    wfull[32:32 + M] = w
    wbuf = torch.from_numpy(wfull).cuda()
    rows = G * n_t
    d.hist_bins, d.hist_copies, d.hist_lo, d.hist_hi, d.hist_t0, d.hist_rows = bins, copies, -0.5, 3.5, 0, n_t
    if Gs:
        d.n_stat_groups, d.stat_group = Gs, labels.data_ptr()
    hp = torch.full((copies + 2, rows, bins), 0x5EADBEEF, dtype=torch.int32, device="cuda")
    mp = torch.full((copies + 2, rows, 4), float(POISON64), dtype=torch.float64, device="cuda")
    d.hist_private = hp.data_ptr() + rows * bins * 4
    d.moments_private = mp.data_ptr() + rows * 4 * 8
    hist = torch.full((rows + 2, bins), -7, dtype=torch.int64, device="cuda")
    mom = torch.full((rows + 2, 4), float(POISON64), dtype=torch.float64, device="cuda")
    _abi.check(L.ufair_stats_reset(C.byref(d), None))
    _abi.check((L.ufair_run_f64 if prec == "f64" else L.ufair_run_f32)(C.byref(d), None))
    weighted = L.ufair_stats_pass_weighted_f64 if prec == "f64" else L.ufair_stats_pass_weighted_f32
    _abi.check(weighted(C.byref(d), wbuf.data_ptr() + 32 * 4, None))
    _abi.check(L.ufair_stats_finalize(C.byref(d), hist[1].data_ptr(), mom[1].data_ptr(), None))
    torch.cuda.synchronize()
    pb = np.array([POISON64]).view(np.uint64)[0]
    h = hp.cpu().numpy()
    assert (h[0] == 0x5EADBEEF).all() and (h[-1] == 0x5EADBEEF).all(), "hist_private guard blocks"
    m = mp.cpu().numpy().view(np.uint64)
    assert (m[0] == pb).all() and (m[-1] == pb).all(), "moments_private guard blocks"
    hh, mm = hist.cpu().numpy(), mom.cpu().numpy()
    assert (hh[0] == -7).all() and (hh[-1] == -7).all(), "finalised hist guard rows"
    assert (mm[[0, -1]].view(np.uint64) == pb).all(), "finalised moments guard rows"
    wb = wbuf.cpu().numpy()
    assert (wb[:32] == 0x5EADBEEF).all() and (wb[32 + M:] == 0x5EADBEEF).all() and np.array_equal(wb[32:32 + M], w)
    for name, buf in b.items():
        buf.check(name, written=name.startswith("o") or name == "state")
    T = b["oT"].data()
    h_ref, m_ref = weighted_temperature_stats(T, -0.5, 3.5, bins, lab if Gs else None, G, w)
    assert np.array_equal(hh[1:-1].reshape(G, n_t, bins).astype(np.uint64), h_ref)
    _check_moments(mm[1:-1].reshape(G, n_t, 4), m_ref, T, lab if Gs else None, w)


def test_argument_errors(api):
    import torch
    M, n_t = 600, 10
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=64)
    ones = torch.ones(M, dtype=torch.int64, device="cuda")
    for w, match in ((ones[:-1], "one weight per member"), (ones.double(), "integers"),
                     (torch.cat([ones[:-1], -ones[:1]]), "negative"),
                     (torch.cat([ones[:-1], ones[:1] * 2 ** 32]), "2\\^32 - 1"),
                     (torch.full((M,), 2 ** 23, dtype=torch.int32, device="cuda"), "sums to")):
        with pytest.raises(ValueError, match=match):
            _plan(api, M, n_t, "f64", spec, None, w)
    gp, tp, esc, scen = P.sample_on_device(M, 1)
    E = P.scenario_emissions(n_t)
    with pytest.raises(ValueError, match="needs stats"):
        api.run_ensemble(to_dev(E), gp, tp, scen_idx=scen, e_scale=esc, stat_weight=ones)
    with pytest.raises(ValueError, match="needs stats"):     # host path too
        api.run_ensemble(E, to_np(gp), to_np(tp), scen_idx=to_np(scen), e_scale=to_np(esc), stat_weight=np.ones(M, int))
    with pytest.raises(ValueError, match="sums to"):
        api.run_ensemble(E, to_np(gp), to_np(tp), scen_idx=to_np(scen), e_scale=to_np(esc), stats=spec,
                         stat_weight=np.full(M, 2 ** 23, dtype=np.int64))
    # the C ABI on a real plan: a NULL weight, and the unweighted pass's own rules
    plan = _plan(api, M, n_t, "f64", spec, None, ones)
    L = _abi.lib()
    d = _abi.UfairDesc.from_buffer_copy(plan.desc)
    assert L.ufair_stats_pass_weighted_f64(C.byref(d), None, None) == _abi.ERR_ARG
    d.stats = 0
    assert L.ufair_stats_pass_weighted_f64(C.byref(d), plan.stat_weight.data_ptr(), None) == _abi.ERR_ARG
    assert b"stats == 0" in L.ufair_last_error()
    torch.cuda.synchronize()
