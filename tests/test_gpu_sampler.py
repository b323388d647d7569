"""On-device ensemble sampler (SURVEY.md 8f-3) against its numpy restatement: the integer stream and
the scenario indices bit-exact, the floating-point transforms to a few ulp, sharding invariance, and
an end-to-end run from sampled parameters."""
import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import params as P
from oracle import c_oracle as co
from oracle import ufair_oracle as o
from tests.util import assert_parity, to_dev, to_np

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    from fiveeqscm_b200 import concentrations as c
    _abi.lib()
    return c


def _close(got, ref, rtol):
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return bool(np.all(np.abs(got - ref) <= rtol * np.abs(ref)))


@pytest.mark.parametrize("dense,gases", [(False, P.GASES), (True, P.GASES), (False, ("co2", "ch4", "n2o", "hfc")), (False, ("hfc",))])
def test_device_sampler_matches_oracle(api, dense, gases):
    M, seed, first = 10_007, 20261018, 123_456_789_012     # global indices beyond 2^32: high counter word in use
    t = P.sampler_tables(gases, dense_pools=dense)
    gp, tp, esc, scen = P.sample_on_device(M, seed, first_member=first, tables=t)
    rgp, rtp, resc, rscen = o.sample_ensemble(seed, first, M, n_scen=4, **t)
    assert np.array_equal(to_np(scen), rscen)                                   # integer path: bit-exact
    assert _close(to_np(gp), rgp, 1e-14) and _close(to_np(tp), rtp, 1e-14) and _close(to_np(esc), resc, 1e-14)
    assert np.array_equal(to_np(gp)[:, _abi.GP_C0], rgp[:, _abi.GP_C0])         # fixed rows: the table, exactly
    assert np.array_equal(to_np(gp) == 0.0, rgp == 0.0)                         # absent pools / terms stay absent


def test_sharding_invariance_and_fp32(api):
    import torch
    t = P.sampler_tables()
    whole = P.sample_on_device(5000, 99, tables=t)
    parts = [P.sample_on_device(n, 99, first_member=f, tables=t) for f, n in ((0, 1234), (1234, 2001), (3235, 1765))]
    for k in range(4):
        assert torch.equal(torch.cat([p[k] for p in parts], dim=-1), whole[k])
    f32 = P.sample_on_device(5000, 99, tables=t, precision="f32")
    for k in range(3):
        assert f32[k].dtype == torch.float32 and torch.equal(f32[k], whole[k].to(torch.float32))   # rounded once, on store
    assert torch.equal(f32[3], whole[3])


def test_run_from_sampled_ensemble_matches_oracle(api):
    """Sampler -> integrator on the device (scenario-shared emissions: nothing per-member ever crosses
    PCIe) against oracle sampler -> oracle integrator."""
    import torch
    M, n_t, seed = 3000, 200, 5
    t = P.sampler_tables()
    scen_E = P.scenario_emissions(n_t)
    gp, tp, esc, scen = P.sample_on_device(M, seed, tables=t)
    res = api.run_ensemble(to_dev(scen_E), gp, tp, scen_idx=scen, e_scale=esc)
    torch.cuda.synchronize()
    rgp, rtp, resc, rscen = o.sample_ensemble(seed, 0, M, n_scen=4, **t)
    ref = co.oxfair(scen_E, rgp, rtp, scen_idx=rscen, e_scale=resc)
    assert_parity(res, ref, ("C", "RF", "T", "state"))


def test_sampler_argument_errors(api):
    import ctypes as C
    L = _abi.lib()
    sp = _abi.UfairSampler(n_gas=3, n_scen=4)
    assert L.ufair_sample_f64(C.byref(sp), 0, 0, 0, None, None, None, None, None) == _abi.OK      # empty: no launch
    assert L.ufair_sample_f64(C.byref(sp), -1, 4, 4, None, None, None, None, None) == _abi.ERR_ARG
    sp.n_scen = 0
    assert L.ufair_sample_f64(C.byref(sp), 0, 4, 4, None, None, None, None, None) == _abi.ERR_ARG
    sp.n_scen, sp.struct_size = 4, 8
    assert L.ufair_sample_f64(C.byref(sp), 0, 4, 4, None, None, None, None, None) == _abi.ERR_ARG
    bad = _abi.UfairSampler(n_gas=2, n_scen=1)
    bad.gas_dist[1][3] = 7
    assert L.ufair_sample_f64(C.byref(bad), 0, 4, 4, None, None, None, None, None) == _abi.ERR_ARG


def test_sharded_ensemble_statistics_equal_the_single_gpu_run(api):
    """SURVEY 8e: integer histogram counts make the reduced statistics independent of how the member
    axis is split.  Two 'ranks' (run one after the other here) sample their blocks of the global
    ensemble by global index, integrate, and their summed histograms are the single run's, bit for bit."""
    import torch
    M, n_t, seed = 6000, 150, 11
    scen_E = to_dev(P.scenario_emissions(n_t))
    spec = api.HistSpec(lo=-1.0, hi=6.0, bins=512)

    def shard(first, n):
        gp, tp, esc, scen = P.sample_on_device(n, seed, first_member=first)
        r = api.run_ensemble(scen_E, gp, tp, scen_idx=scen, e_scale=esc, stats=spec, outputs=("T",))
        torch.cuda.synchronize()
        return r

    whole = shard(0, M)
    a, b = shard(0, 2500), shard(2500, 3500)
    assert torch.equal(a.hist + b.hist, whole.hist)
    assert torch.equal(torch.cat([a.T, b.T], dim=1), whole.T)
    mom = whole.moments
    assert torch.allclose(a.moments[:, :2] + b.moments[:, :2], mom[:, :2], rtol=1e-12, atol=1e-12)
    assert torch.equal(torch.minimum(a.moments[:, 2], b.moments[:, 2]), mom[:, 2])
    assert torch.equal(torch.maximum(a.moments[:, 3], b.moments[:, 3]), mom[:, 3])
    from fiveeqscm_b200 import stats
    pw = stats.percentiles_device(whole.hist, spec.lo, spec.hi, (5, 50, 95))
    ps = stats.percentiles_device(a.hist + b.hist, spec.lo, spec.hi, (5, 50, 95))
    assert torch.equal(pw, ps)


def test_packed_statistics_layout_round_trips_and_reduces_like_the_plain_one(api):
    """The cross-GPU reduce works on two packed buffers (ufair_stats_finalize_packed: counts as doubles + moment
    sums -> SUM; max and -min -> MAX).  On one GPU: packed -> unpack equals the plain finalize bit for bit, and
    'reducing' two shards' packed buffers the way the collectives would (elementwise sum / max) and unpacking
    gives the single run's histogram and extrema bit for bit -- the arithmetic of dist.StatsReducer without NCCL."""
    import ctypes as C

    import torch
    L = _abi.lib()
    M, n_t, seed = 5000, 60, 3
    scen_E = to_dev(P.scenario_emissions(n_t))
    spec = api.HistSpec(lo=-1.0, hi=6.0, bins=256)

    def packed(first, n):
        gp, tp, esc, scen = P.sample_on_device(n, seed, first_member=first)
        plan = api.DevicePlan(scen_E, gp, tp, scen_idx=scen, e_scale=esc, stats=spec, outputs=("T",), return_state=False)
        plan.reset_stats(); plan.launch(); plan.stats_pass(); plan.finalize_stats()
        sums = torch.empty(n_t, spec.bins + 2, dtype=torch.float64, device="cuda")
        ext = torch.empty(n_t, 2, dtype=torch.float64, device="cuda")
        _abi.check(L.ufair_stats_finalize_packed(C.byref(plan.desc), sums.data_ptr(), ext.data_ptr(), None))
        torch.cuda.synchronize()
        return plan.result, sums, ext

    def unpack(sums, ext):
        hist = torch.empty(n_t, spec.bins, dtype=torch.int64, device="cuda")
        mom = torch.empty(n_t, 4, dtype=torch.float64, device="cuda")
        _abi.check(L.ufair_stats_unpack(sums.data_ptr(), ext.data_ptr(), n_t, spec.bins, hist.data_ptr(), mom.data_ptr(), None))
        torch.cuda.synchronize()
        return hist, mom

    whole, s_w, e_w = packed(0, M)
    h, m = unpack(s_w, e_w)
    assert torch.equal(h, whole.hist) and torch.equal(m, whole.moments)
    (ra, s_a, e_a), (rb, s_b, e_b) = packed(0, 2048), packed(2048, M - 2048)
    h2, m2 = unpack(s_a + s_b, torch.maximum(e_a, e_b))
    assert torch.equal(h2, whole.hist) and torch.equal(m2[:, 2:], whole.moments[:, 2:])
    assert torch.allclose(m2[:, :2], whole.moments[:, :2], rtol=1e-12, atol=1e-12)
