"""Grouped ensemble statistics on the device: per-group counts against a recount of the kernel's own T, the pooled
pass reproduced by one group, determinism, sharding and the packed reduction, the host pipeline, device
percentiles, non-finite temperatures, guard bands around every grouped buffer, and argument errors."""
import ctypes as C

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import params as P
from oracle import ufair_oracle as o
from tests.group_stats_ref import grouped_temperature_stats, plant_non_finite
from tests.test_gpu_guard import POISON64, _desc_and_buffers
from tests.util import ensemble, to_dev, to_np

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    from fiveeqscm_b200 import concentrations as c
    _abi.lib()
    return c


def _plan(api, M, n_t, prec, spec, stat_group, seed=5, first=0, **kw):
    """Sampler -> integrator with T output and statistics, on the device."""
    gp, tp, esc, scen = P.sample_on_device(M, seed, first_member=first, precision=prec)
    plan = api.DevicePlan(to_dev(P.scenario_emissions(n_t)), gp, tp, scen_idx=scen, e_scale=esc, stats=spec,
                          stat_group=stat_group, outputs=("T",), return_state=False, precision=prec, **kw)
    return plan, scen


def _labels(M, G, neg, seed):
    rng = np.random.default_rng(seed)
    lab = rng.integers(-1 if neg else 0, G, M).astype(np.int32)
    return lab


def _check_moments(mom, ref, absT):
    assert np.array_equal(mom[..., 2:], ref[..., 2:]), "min / max exact"
    assert np.all(np.abs(mom[..., 0] - ref[..., 0]) <= 1e-12 * absT), "sum"
    assert np.all(np.abs(mom[..., 1] - ref[..., 1]) <= 1e-12 * ref[..., 1]), "sum of squares"


def _abs_sums(T, labels, G):
    return np.stack([np.abs(T[:, labels == g].astype(np.float64)).sum(axis=1) for g in range(G)])


CASES = [  # prec, M, groups, bins, copies, negative labels; groups <= 4 take the 4-group tile, more the 8-group one
    ("f64", 3001, 1, 256, 3, False),
    ("f64", 5003, 4, 1024, 5, True),
    ("f32", 4099, 4, 512, 3, True),
    ("f64", 2999, 13, 300, 4, True),     # two tiles, the last one partial
    ("f32", 3333, 40, 128, 3, True),     # five tiles
    ("f64", 3001, 13, 4096, 3, True),    # 8 x 4096 bins > shared-memory budget: global atomics
    ("f64", 2001, 4, 8192, 2, False),    # 4 x 8192 bins: global atomics
    ("f32", 1999, 40, 2500, 3, True),
]


@pytest.mark.parametrize("prec,M,G,bins,copies,neg", CASES, ids=lambda v: str(v))
def test_grouped_counts_equal_a_recount_of_the_kernels_T(api, prec, M, G, bins, copies, neg):
    import torch
    n_t = 41
    lab = _labels(M, G, neg, seed=M + G)
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=bins, copies=copies, groups=G)
    plan, _ = _plan(api, M, n_t, prec, spec, lab)
    if neg:   # labels >= groups are counted nowhere either (Python rejects them; the kernel must still skip them)
        plan.stat_group[::17] = G + 3
        lab = to_np(plan.stat_group)
    res = plan.run()
    torch.cuda.synchronize()
    T = to_np(res.T)
    assert res.hist.shape == (G, n_t, bins) and res.moments.shape == (G, n_t, 4)
    h_ref, m_ref = grouped_temperature_stats(T, spec.lo, spec.hi, bins, lab, G)
    assert np.array_equal(to_np(res.hist).astype(np.uint64), h_ref)
    _check_moments(to_np(res.moments), m_ref, _abs_sums(T, lab, G))


@pytest.mark.parametrize("prec,bins", [pytest.param("f64", 512, id="f64"), pytest.param("f32", 512, id="f32"),
                                       # past the 16 384-slot shared-memory budget: the pooled pass's global atomics
                                       pytest.param("f64", 20000, id="f64-20000"),
                                       pytest.param("f32", 20000, id="f32-20000")])
def test_one_group_is_the_pooled_pass_and_groups_sum_to_it(api, prec, bins):
    import torch
    M, n_t = 4001, 37
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=bins, copies=5)
    pooled = _plan(api, M, n_t, prec, spec, None)[0].run()
    one = _plan(api, M, n_t, prec, api.HistSpec(lo=-0.5, hi=3.5, bins=bins, copies=5, groups=1),
                np.zeros(M, dtype=np.int32))[0].run()
    four = _plan(api, M, n_t, prec, spec, "scenario")[0].run()
    torch.cuda.synchronize()
    assert torch.equal(one.T, pooled.T)
    assert torch.equal(one.hist[0], pooled.hist) and torch.equal(one.moments[0], pooled.moments)   # bit for bit
    assert four.hist.shape[0] == 4 and torch.equal(four.hist.sum(dim=0), pooled.hist)
    if bins > 16384:
        h_ref, _ = grouped_temperature_stats(to_np(pooled.T), spec.lo, spec.hi, bins, np.zeros(M, dtype=np.int32), 1)
        assert np.array_equal(to_np(pooled.hist).astype(np.uint64), h_ref[0])


def test_moments_are_deterministic(api):
    import torch
    M, n_t, G = 6007, 29, 13
    plan, _ = _plan(api, M, n_t, "f64", api.HistSpec(lo=-0.5, hi=3.5, bins=256, groups=G), _labels(M, G, True, 1))
    a = plan.run()
    h1, m1 = a.hist.clone(), a.moments.clone()
    b = plan.run()
    torch.cuda.synchronize()
    assert torch.equal(h1, b.hist)
    assert np.array_equal(to_np(m1).view(np.uint64), to_np(b.moments).view(np.uint64))


def test_per_scenario_shards_sum_to_the_whole_run_and_the_packed_reduction(api):
    import torch
    L = _abi.lib()
    M, n_t, seed = 6000, 60, 11
    spec = api.HistSpec(lo=-1.0, hi=6.0, bins=256)

    def shard(first, n):
        plan, _ = _plan(api, n, n_t, "f64", spec, "scenario", seed=seed, first=first)
        res = plan.run()
        rows = 4 * n_t
        sums = torch.empty(rows, spec.bins + 2, dtype=torch.float64, device="cuda")
        ext = torch.empty(rows, 2, dtype=torch.float64, device="cuda")
        _abi.check(L.ufair_stats_finalize_packed(C.byref(plan.desc), sums.data_ptr(), ext.data_ptr(), None))
        torch.cuda.synchronize()
        return res, sums, ext

    def unpack(sums, ext):
        hist = torch.empty(4, n_t, spec.bins, dtype=torch.int64, device="cuda")
        mom = torch.empty(4, n_t, 4, dtype=torch.float64, device="cuda")
        _abi.check(L.ufair_stats_unpack(sums.data_ptr(), ext.data_ptr(), 4 * n_t, spec.bins, hist.data_ptr(),
                                        mom.data_ptr(), None))
        torch.cuda.synchronize()
        return hist, mom

    whole, s_w, e_w = shard(0, M)
    (a, s_a, e_a), (b, s_b, e_b) = shard(0, 2500), shard(2500, M - 2500)
    assert whole.hist.shape == (4, n_t, spec.bins) and whole.spec.groups == 4 and whole.stat_group == "scenario"
    assert torch.equal(a.hist + b.hist, whole.hist)
    assert torch.equal(torch.minimum(a.moments[..., 2], b.moments[..., 2]), whole.moments[..., 2])
    assert torch.equal(torch.maximum(a.moments[..., 3], b.moments[..., 3]), whole.moments[..., 3])
    assert torch.allclose(a.moments[..., :2] + b.moments[..., :2], whole.moments[..., :2], rtol=1e-12, atol=1e-12)
    h, m = unpack(s_w, e_w)
    assert torch.equal(h, whole.hist) and torch.equal(m, whole.moments)
    h2, m2 = unpack(s_a + s_b, torch.maximum(e_a, e_b))
    assert torch.equal(h2, whole.hist) and torch.equal(m2[..., 2:], whole.moments[..., 2:])


def test_host_pipeline_matches_the_device_path(api):
    import torch
    M, n_t, G = 5003, 33, 6
    gp, tp, esc, scen = (to_np(x) for x in P.sample_on_device(M, 9))
    scen = np.ascontiguousarray(scen, dtype=np.int32)
    E = P.scenario_emissions(n_t)
    lab = _labels(M, G, True, 4)
    for stat_group, groups in ((lab, G), (scen, 4), ("scenario", 0)):   # own labels; scen_idx itself twice
        spec = api.HistSpec(lo=-0.5, hi=3.5, bins=300, copies=3, groups=groups)
        ws = api.Workspace(torch.cuda.current_device(), 384)                  # 384 does not divide 5003
        try:
            host = api.run_ensemble(E, gp, tp, scen_idx=scen, e_scale=esc, stats=spec, stat_group=stat_group,
                                    outputs=("T",), return_state=False, workspace=ws)
        finally:
            ws.close()
        dev = api.run_ensemble(to_dev(E), to_dev(gp), to_dev(tp), scen_idx=to_dev(scen), e_scale=to_dev(esc),
                               stats=spec, stat_group=stat_group if isinstance(stat_group, str) else to_dev(stat_group),
                               outputs=("T",), return_state=False)
        torch.cuda.synchronize()
        ng = groups or 4
        assert host.hist.shape == (ng, n_t, 300) and np.array_equal(host.hist, to_np(dev.hist))
        assert np.array_equal(host.moments[..., 2:], to_np(dev.moments)[..., 2:])
        labels = stat_group if not isinstance(stat_group, str) else scen
        h_ref, _ = grouped_temperature_stats(host.T, spec.lo, spec.hi, 300, labels, ng)
        assert np.array_equal(host.hist.astype(np.uint64), h_ref)


def test_device_percentiles_of_grouped_histograms(api):
    import torch
    from fiveeqscm_b200 import stats
    plan, _ = _plan(api, 3000, 45, "f64", api.HistSpec(lo=-0.5, hi=3.5, bins=400), "scenario")
    res = plan.run()
    pd = stats.percentiles_device(res.hist, -0.5, 3.5, (5, 17, 50, 83, 95))
    torch.cuda.synchronize()
    assert pd.shape == (4, 45, 5)
    assert np.array_equal(to_np(pd), stats.percentiles(res.hist, -0.5, 3.5, (5, 17, 50, 83, 95)))


@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("G", [0, 3, 9], ids=["pooled", "G3", "G9"])   # 3 groups: the 4-group tile; 9: the 8-group one
def test_non_finite_temperatures_follow_the_rule(api, prec, G):
    """T rows carrying NaN, +-inf, exactly lo / hi, one ulp below hi, bin edges and an all-NaN step, written between
    the integrator and the statistics pass: NaN is neither binned nor in min / max and makes its row's sum and sumsq
    NaN; the infinities land in the edge bins and enter every moment (include/ufair.h, statistics block)."""
    import torch
    from fiveeqscm_b200 import stats
    M, n_t, lo, hi, bins = 1003, 8, -1.0, 6.0, 28
    lab = _labels(M, G, True, 17) if G else None
    spec = api.HistSpec(lo=lo, hi=hi, bins=bins, copies=3, groups=G)
    plan, _ = _plan(api, M, n_t, prec, spec, lab)
    plan.reset_stats()
    plan.launch()
    T = plant_non_finite(to_np(plan.result.T).copy(), lo, hi, bins)
    plan.result.T.copy_(torch.from_numpy(T))                # the T rows the statistics pass reads
    plan.stats_pass()
    plan.finalize_stats()
    torch.cuda.synchronize()
    hist, mom = to_np(plan.result.hist), to_np(plan.result.moments)
    if G:
        h_ref, m_ref = grouped_temperature_stats(T, lo, hi, bins, lab, G)
        absT = _abs_sums(T, lab, G)
    else:
        h_ref, m_ref = o.temperature_stats(T, lo, hi, bins)
        absT = np.abs(T.astype(np.float64)).sum(axis=1)
    assert np.array_equal(hist.astype(np.uint64), h_ref)
    assert np.array_equal(mom[..., 2:], m_ref[..., 2:]), "min / max exact"
    for j in (0, 1):                                      # sum, sumsq: NaN and inf where the reference has them
        got, want = mom[..., j], m_ref[..., j]
        fin = np.isfinite(want)
        assert np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(got[np.isinf(want)], want[np.isinf(want)])
        tol = 1e-12 * (absT if j == 0 else want)
        assert np.all(np.abs(got[fin] - want[fin]) <= tol[fin])
    assert np.isnan(mom[..., 3, 0]).all() and (mom[..., 3, 2] == np.inf).all() and (mom[..., 3, 3] == -np.inf).all()
    assert not hist[..., 3, :].any()
    pcts = (0.0, 5.0, 50.0, 95.0, 100.0)
    pd = to_np(stats.percentiles_device(plan.result.hist, lo, hi, pcts)).reshape(-1, n_t, len(pcts))
    for g, h in enumerate(hist.reshape(-1, n_t, bins)):
        assert np.array_equal(pd[g], o.percentiles_from_hist(h, lo, hi, pcts)), g
        assert np.array_equal(pd[g, 3], o.percentiles_from_hist(h[3:4], lo, hi, pcts)[0])   # the all-NaN step


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_grouped_buffers_stay_inside_their_rows(prec):
    import torch
    L = _abi.lib()
    M, n_t, Gs, bins, copies, ld = 1003, 19, 11, 96, 3, 1008
    ens = ensemble(M, n_t=n_t, seed=13)
    d, b = _desc_and_buffers(ens, M, n_t, 3, ld, prec, True, outputs=("T",), stats=True)
    lab = _labels(M, Gs, True, 2)
    labels = torch.from_numpy(lab).cuda()
    rows = Gs * n_t
    d.hist_bins, d.hist_copies, d.hist_lo, d.hist_hi, d.hist_t0, d.hist_rows = bins, copies, -0.5, 3.5, 0, n_t
    d.n_stat_groups, d.stat_group = Gs, labels.data_ptr()
    hp = torch.full((copies + 2, rows, bins), 0x5EADBEEF, dtype=torch.int32, device="cuda")
    mp = torch.full((copies + 2, rows, 4), float(POISON64), dtype=torch.float64, device="cuda")
    d.hist_private = hp.data_ptr() + rows * bins * 4
    d.moments_private = mp.data_ptr() + rows * 4 * 8
    hist = torch.full((rows + 2, bins), -7, dtype=torch.int64, device="cuda")
    mom = torch.full((rows + 2, 4), float(POISON64), dtype=torch.float64, device="cuda")
    sums = torch.full((rows + 2, bins + 2), float(POISON64), dtype=torch.float64, device="cuda")
    ext = torch.full((rows + 2, 2), float(POISON64), dtype=torch.float64, device="cuda")
    _abi.check(L.ufair_stats_reset(C.byref(d), None))
    _abi.check((L.ufair_run_f64 if prec == "f64" else L.ufair_run_f32)(C.byref(d), None))
    _abi.check((L.ufair_stats_pass_f64 if prec == "f64" else L.ufair_stats_pass_f32)(C.byref(d), None))
    _abi.check(L.ufair_stats_finalize(C.byref(d), hist[1].data_ptr(), mom[1].data_ptr(), None))
    _abi.check(L.ufair_stats_finalize_packed(C.byref(d), sums[1].data_ptr(), ext[1].data_ptr(), None))
    torch.cuda.synchronize()
    pb = np.array([POISON64]).view(np.uint64)[0]
    h = hp.cpu().numpy()
    assert (h[0] == 0x5EADBEEF).all() and (h[-1] == 0x5EADBEEF).all(), "hist_private guard blocks"
    m = mp.cpu().numpy().view(np.uint64)
    assert (m[0] == pb).all() and (m[-1] == pb).all(), "moments_private guard blocks"
    hh, mm = hist.cpu().numpy(), mom.cpu().numpy()
    assert (hh[0] == -7).all() and (hh[-1] == -7).all(), "finalised hist guard rows"
    assert (mm[[0, -1]].view(np.uint64) == pb).all(), "finalised moments guard rows"
    ss, ee = sums.cpu().numpy().view(np.uint64), ext.cpu().numpy().view(np.uint64)
    assert (ss[[0, -1]] == pb).all() and (ee[[0, -1]] == pb).all(), "packed guard rows"
    for name, buf in b.items():
        buf.check(name, written=name.startswith("o") or name == "state")
    T = b["oT"].data()
    h_ref, m_ref = grouped_temperature_stats(T, -0.5, 3.5, bins, lab, Gs)
    assert np.array_equal(hh[1:-1].reshape(Gs, n_t, bins).astype(np.uint64), h_ref)
    _check_moments(mm[1:-1].reshape(Gs, n_t, 4), m_ref, _abs_sums(T, lab, Gs))


def test_argument_errors(api):
    import torch
    M, n_t = 600, 10
    spec = api.HistSpec(lo=-0.5, hi=3.5, bins=64, groups=3)
    with pytest.raises(ValueError, match="label 3 >= groups 3"):
        _plan(api, M, n_t, "f64", spec, np.full(M, 3, dtype=np.int32))
    with pytest.raises(ValueError, match="one label per member"):
        _plan(api, M, n_t, "f64", spec, np.zeros(M - 1, dtype=np.int32))
    with pytest.raises(ValueError, match="not inferred"):
        _plan(api, M, n_t, "f64", api.HistSpec(), np.zeros(M, dtype=np.int32))
    with pytest.raises(ValueError, match="label 3 >= groups 3"):    # four scenarios, three groups
        _plan(api, M, n_t, "f64", spec, "scenario")
    gp, tp, esc, scen = P.sample_on_device(M, 1)
    with pytest.raises(ValueError, match="needs scen_idx"):
        api.run_ensemble(to_dev(P.scenario_emissions(n_t)[:, :, :1]), gp, tp, stats=api.HistSpec(), stat_group="scenario")
    with pytest.raises(ValueError, match="label 3 >= groups 3"):    # host path too
        api.run_ensemble(P.scenario_emissions(n_t), to_np(gp), to_np(tp), scen_idx=to_np(scen), stats=spec,
                         stat_group=np.full(M, 3, dtype=np.int32))
    # the C ABI: a NULL label array with several groups, and too many groups, on a real plan
    plan, _ = _plan(api, M, n_t, "f64", spec, np.zeros(M, dtype=np.int32))
    L = _abi.lib()
    d = _abi.UfairDesc.from_buffer_copy(plan.desc)
    d.stat_group = None
    assert L.ufair_stats_pass_f64(C.byref(d), None) == _abi.ERR_ARG
    d = _abi.UfairDesc.from_buffer_copy(plan.desc)
    d.n_stat_groups = _abi.MAX_STAT_GROUPS + 1
    assert L.ufair_stats_pass_f64(C.byref(d), None) == _abi.ERR_ARG
    torch.cuda.synchronize()
