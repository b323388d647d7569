"""Period means (``out_every`` = k >= 2): one row of C, RF and T per period of k steps, the mean over its steps.

The rule (include/ufair.h) is exact -- s = 0; s = s + x_t in step order in the run's precision; mean = s * (Real)(1 / k)
-- so most checks here are bitwise: the period loop against the per-step loop's own rows averaged by that rule.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from oracle import c_oracle as co
from tests.group_stats_ref import grouped_temperature_stats
from tests.period_mean_ref import period_mean
from tests.test_gpu_guard import GASES, Guarded
from tests.util import ensemble, output_relerr, to_dev, to_np

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fiveeqscm_b200 import concentrations
    return concentrations


def _inputs(ens, layout, fext, G):
    """run_ensemble inputs (device tensors) for one emission layout and one external-forcing mode."""
    kw = {}
    if layout == "member":
        E = ens["E"]
    else:
        E = ens["scen"]
        kw.update(scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]))
    if fext == "shared":
        kw["f_ext"] = to_dev(ens["f_ext"])
    elif fext == "member":
        M = ens["gas_params"].shape[2]
        kw.update(f_ext=to_dev(ens["f_ext"][:, None] * (1.0 + 0.01 * np.arange(M))), fext_per_member=True)
    return to_dev(E), kw


def _run(api, ens, E, **kw):
    return api.run_ensemble(E, to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), **kw)


def _assert_means_equal(per_step, mean_run, k, keys=("C", "RF", "T")):
    for key in keys:
        want = period_mean(to_np(getattr(per_step, key)), k)
        np.testing.assert_array_equal(to_np(getattr(mean_run, key)), want, err_msg=f"{key}, k={k}")
    np.testing.assert_array_equal(to_np(mean_run.state), to_np(per_step.state), err_msg=f"state, k={k}")


# ------------------------------------------------------------------ 1. bitwise against the per-step run
@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("alpha_mode", ["exp", "sinh", "newton", "one"])
@pytest.mark.parametrize("G", [1, 2, 3, 4])
def test_period_means_equal_the_mean_of_the_per_step_rows(api, prec, alpha_mode, G):
    n_t, M = 20, 203
    ens = ensemble(M, n_t=n_t, gases=GASES[G], dense=True, seed=100 + G)
    common = dict(precision=prec, alpha_mode=alpha_mode, newton_iters=2)
    for layout in ("member", "scenario"):
        for fext in ("none", "shared", "member"):
            E, kw = _inputs(ens, layout, fext, G)
            for iirf_max in (None, 45.0):   # 45: the iIRF ceiling binds for most members
                one = _run(api, ens, E, iirf_max=iirf_max, **common, **kw)
                for k in (2, 10, n_t):
                    got = _run(api, ens, E, iirf_max=iirf_max, out_every=k, **common, **kw)
                    assert got.out_every == k and got.T.shape == (n_t // k, M) and got.C.shape == (G, n_t // k, M)
                    _assert_means_equal(one, got, k)


# ------------------------------------------------------------------ 2. the oracle
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_period_means_match_the_oracle(api, prec):
    n_t, M, k, dt = 200, 1500, 10, 0.1
    ens = ensemble(M, n_t=n_t, dt=dt, dense=True, seed=5)
    got = _run(api, ens, to_dev(ens["scen"]), dt=dt, scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]),
               f_ext=to_dev(ens["f_ext"]), out_every=k, precision=prec)
    ref = co.oxfair(ens["scen"], ens["gas_params"], ens["thermal_params"], dt=dt, scen_idx=ens["scen_idx"],
                    e_scale=ens["e_scale"], f_ext=ens["f_ext"])
    for key in ("C", "RF", "T"):
        want = period_mean(ref[key], k)
        if prec == "f64":
            assert output_relerr(key, to_np(getattr(got, key)), want) <= 1e-10, key
    if prec == "f32":
        assert np.max(np.abs(to_np(got.T).astype(np.float64) - period_mean(ref["T"], k))) <= 1e-4
        assert output_relerr("C", to_np(got.C).astype(np.float64), period_mean(ref["C"], k)) <= 2e-5
    else:
        assert output_relerr("state", to_np(got.state), ref["state"]) <= 1e-10


# ------------------------------------------------------------------ 3. specialised forms and the variant report
@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("G", [1, 2, 3, 4])
def test_specialised_forms_give_the_dense_period_loop_bits(api, prec, G):
    n_t, M, k = 40, 700, 4
    gases = ("ch4",) if G == 1 else GASES[G]   # literature parameters: one-pool gases have a specialised form
    ens = ensemble(M, n_t=n_t, gases=gases, dense=False, seed=40 + G)
    E = to_dev(ens["E"])
    plan = api.DevicePlan(E, to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), out_every=k, precision=prec,
                          f_ext=to_dev(ens["f_ext"]))
    form, _, _ = plan.kernel_variant()
    assert plan.loop_variant == "period_mean" and plan.n_out == n_t // k and any(form)
    sparse = plan.run()
    dense = _run(api, ens, E, out_every=k, precision=prec, f_ext=to_dev(ens["f_ext"]), gas_form=None)
    for key in ("C", "RF", "T", "state"):
        np.testing.assert_array_equal(to_np(getattr(sparse, key)), to_np(getattr(dense, key)), err_msg=key)


def test_variant_report_names_the_period_loop_only_for_k_of_two_and_more(api):
    ens = ensemble(64, n_t=8, dense=True, seed=1)
    mk = lambda **kw: api.DevicePlan(to_dev(ens["E"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), **kw)
    for kw, k, want in ((dict(), 0, "plain"), (dict(), 1, "plain"), (dict(iirf_max=97.0), 1, "general"),
                        (dict(), 2, "period_mean"), (dict(alpha_mode="sinh"), 8, "period_mean"),
                        (dict(outputs=("T",), stats=api.HistSpec()), 4, "period_mean")):
        p = mk(out_every=k, **kw)
        _, gpl, _ = p.kernel_variant()
        assert p.loop_variant == want, (kw, k)
        if k >= 2:
            assert gpl == 3   # all gases per lane: no small-ensemble mapping for the period loop


# ------------------------------------------------------------------ 4. resume
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_two_time_chunks_equal_one_call(api, prec):
    import torch
    n_t, n1, M, k = 60, 24, 900, 6
    ens = ensemble(M, n_t=n_t, dense=True, seed=9)
    spec = api.HistSpec(lo=-1.0, hi=3.0, bins=256, copies=3)
    gp, tp = to_dev(ens["gas_params"]), to_dev(ens["thermal_params"])
    full = api.DevicePlan(to_dev(ens["E"]), gp, tp, out_every=k, precision=prec, stats=spec).run()
    p1 = api.DevicePlan(to_dev(ens["E"][:, :n1]), gp, tp, out_every=k, precision=prec, stats=spec)
    r1 = p1.result
    p1.launch()
    p2 = api.DevicePlan(to_dev(ens["E"][:, n1:]), gp, tp, out_every=k, precision=prec, stats=spec, state_in=r1.state)
    # both chunks count into one set of statistics buffers: rows [0, n1 / k) and [n1 / k, n_t / k)
    n_out = n_t // k
    hp = torch.empty(spec.copies, n_out, spec.bins, dtype=torch.int32, device="cuda")
    mp = torch.empty(spec.copies, n_out, _abi.MOM_COUNT, dtype=torch.float64, device="cuda")
    hist = torch.empty(n_out, spec.bins, dtype=torch.int64, device="cuda")
    mom = torch.empty(n_out, _abi.MOM_COUNT, dtype=torch.float64, device="cuda")
    for p, t0 in ((p1, 0), (p2, n1 // k)):
        p.desc.hist_private, p.desc.moments_private = hp.data_ptr(), mp.data_ptr()
        p.desc.hist_rows, p.desc.hist_t0 = n_out, t0
    L, s = _abi.lib(), torch.cuda.current_stream().cuda_stream
    _abi.check(L.ufair_stats_reset(C.byref(p1.desc), s))
    p1.stats_pass()
    p2.launch()
    p2.stats_pass()
    _abi.check(L.ufair_stats_finalize(C.byref(p2.desc), hist.data_ptr(), mom.data_ptr(), s))
    r2 = p2.result
    torch.cuda.synchronize()
    for key, axis in (("C", 1), ("RF", 1), ("T", 0)):
        np.testing.assert_array_equal(np.concatenate([to_np(getattr(r1, key)), to_np(getattr(r2, key))], axis=axis),
                                      to_np(getattr(full, key)), err_msg=key)
    np.testing.assert_array_equal(to_np(r2.state), to_np(full.state))
    np.testing.assert_array_equal(to_np(hist), to_np(full.hist))
    np.testing.assert_array_equal(to_np(mom), to_np(full.moments))


# ------------------------------------------------------------------ 5. statistics
@pytest.mark.parametrize("prec", ["f64", "f32"])
@pytest.mark.parametrize("grouped", [False, True])
def test_statistics_bin_the_period_mean_rows(api, prec, grouped):
    n_t, M, k = 120, 20_000, 10
    ens = ensemble(M, n_t=n_t, dense=True, seed=12)
    spec = api.HistSpec(lo=-1.0, hi=3.0, bins=512, copies=5)
    kw = dict(stat_group="scenario") if grouped else {}
    res = _run(api, ens, to_dev(ens["scen"]), scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]),
               f_ext=to_dev(ens["f_ext"]), out_every=k, precision=prec, stats=spec, **kw)
    T = to_np(res.T)
    n_g = ens["scen"].shape[2] if grouped else 1
    labels = ens["scen_idx"] if grouped else np.zeros(M, dtype=np.int64)
    h_ref, m_ref = grouped_temperature_stats(T, spec.lo, spec.hi, spec.bins, labels, n_g)
    hist, mom = to_np(res.hist), to_np(res.moments)
    if not grouped:
        h_ref, m_ref = h_ref[0], m_ref[0]
    assert hist.shape == h_ref.shape and hist.shape[-2] == n_t // k
    np.testing.assert_array_equal(hist.astype(np.uint64), h_ref)
    np.testing.assert_allclose(mom, m_ref, rtol=1e-12)


# ------------------------------------------------------------------ 6. host pipeline
@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_host_pipeline_equals_the_device_path(api, prec):
    n_t, M, k = 80, 1003, 8
    ens = ensemble(M, n_t=n_t, dense=True, seed=21)
    spec = api.HistSpec(copies=4)
    kw = dict(scen_idx=ens["scen_idx"], e_scale=ens["e_scale"], f_ext=ens["f_ext"], out_every=k, precision=prec,
              stats=spec)
    dev = _run(api, ens, to_dev(ens["scen"]), **{key: to_dev(v) if isinstance(v, np.ndarray) else v
                                                 for key, v in kw.items()})
    host = api.run_ensemble(ens["scen"], ens["gas_params"], ens["thermal_params"], chunk_members=384, **kw)
    out = api.pinned_result(3, n_t, M, stats=spec, precision=prec, out_every=k)
    ws = api.Workspace(0, 256)
    reused = api.run_ensemble(ens["scen"], ens["gas_params"], ens["thermal_params"], workspace=ws, out=out, **kw)
    ws.close()
    assert reused is out and out.T.shape == (n_t // k, M)
    for r in (host, reused):
        for key in ("C", "RF", "T", "state", "hist"):
            np.testing.assert_array_equal(getattr(r, key), to_np(getattr(dev, key)), err_msg=key)
        np.testing.assert_allclose(r.moments, to_np(dev.moments), rtol=1e-12)


# ------------------------------------------------------------------ 7. guard bands
GUARD_CASES = [  # (n_gas, M, ld slack, n_t, k, precision, per-member emissions, form)
    (3, 1003, 6, 40, 8, "f64", True, False),
    (1, 95, 2, 18, 3, "f64", False, False),
    (4, 259, 6, 20, 20, "f64", True, False),
    (3, 515, 2, 24, 2, "f64", True, True),
    (2, 1003, 4, 30, 5, "f32", False, False),
    (4, 70, 4, 12, 4, "f32", True, True),
]


@pytest.mark.parametrize("G,M,slack,n_t,k,prec,e_member,form", GUARD_CASES, ids=lambda v: str(v).replace(" ", ""))
def test_period_outputs_stay_inside_their_rows(api, G, M, slack, n_t, k, prec, e_member, form):
    import torch
    npdt = np.float64 if prec == "f64" else np.float32
    q = 16 // npdt().itemsize
    ld = (M + q - 1) // q * q + slack // q * q
    n_out = n_t // k
    ens = ensemble(M, n_t=n_t, gases=GASES[G], dense=not form, seed=7 + M)
    mk = lambda rows: Guarded(rows, M, ld, npdt, True)
    b = {"gp": mk(G * _abi.GP_COUNT).fill(ens["gas_params"].astype(npdt)),
         "tp": mk(_abi.TP_COUNT).fill(ens["thermal_params"].astype(npdt)),
         "oC": mk(G * n_out), "oRF": mk(G * n_out), "oT": mk(n_out), "state": mk(_abi.state_rows(G))}
    d = _abi.UfairDesc(n_gas=G, n_t=n_t, n_member=M, ld_member=ld, out_mask=_abi.OUT_C | _abi.OUT_RF | _abi.OUT_T,
                       out_every=k, gas_params=b["gp"].ptr, thermal_params=b["tp"].ptr, out_C=b["oC"].ptr,
                       out_RF=b["oRF"].ptr, out_T=b["oT"].ptr, state_out=b["state"].ptr)
    keep = []
    if e_member:
        b["E"] = mk(G * n_t).fill(ens["E"].astype(npdt))
        d.emissions, d.e_mode = b["E"].ptr, _abi.E_MEMBER
    else:
        keep = [to_dev(ens["scen"].astype(npdt)), to_dev(ens["scen_idx"].astype(np.int32))]
        b["esc"] = mk(G).fill(ens["e_scale"].astype(npdt))
        d.emissions, d.scen_idx, d.e_scale, d.e_mode = keep[0].data_ptr(), keep[1].data_ptr(), b["esc"].ptr, _abi.E_SCENARIO
        d.n_scen = ens["scen"].shape[2]
    if form:
        from fiveeqscm_b200.concentrations import _detect_form_host
        for g, f in enumerate(_detect_form_host(ens["gas_params"], None)):
            d.gas_form[g] = f
    L = _abi.lib()
    _abi.check((L.ufair_run_f64 if prec == "f64" else L.ufair_run_f32)(C.byref(d), None))
    torch.cuda.synchronize()
    for name, buf in b.items():
        buf.check(name, written=name.startswith("o") or name == "state")
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"])
    if prec == "f64":
        for key, rows in (("C", (G, n_out, M)), ("RF", (G, n_out, M)), ("T", (n_out, M))):
            assert output_relerr(key, b["o" + key].data().reshape(rows), period_mean(ref[key], k)) < 1e-10, key
    else:
        assert np.max(np.abs(b["oT"].data().astype(np.float64) - period_mean(ref["T"], k))) < 1e-4


# ------------------------------------------------------------------ 8. the checked build (libufair_dbg.so)
_DBG = os.path.join(os.path.dirname(_abi.lib_path()), "libufair_dbg.so")
_TRIP = """
import numpy as np, torch
from fiveeqscm_b200 import concentrations as api
from tests.util import ensemble, to_dev
ens = ensemble(70, n_t=12)
res = api.run_ensemble(to_dev(ens["E"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), out_every=3)
torch.cuda.synchronize()
print("completed")
"""


@pytest.mark.skipif(not os.path.exists(_DBG), reason="libufair_dbg.so not built (make -C fiveeqscm_b200/csrc debug)")
def test_period_loop_on_the_debug_bounds_build():
    """The guard and parity cases of this file on the build whose kernels check every output store against its
    array (n_out rows in the period loop) and every ring read; then its negative control: with UFAIR_DEBUG_TRIP=1
    the store check pretends the last output row is missing and must count the period loop's stores there (it counts,
    it never traps)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, UFAIR_LIB=_DBG, PYTHONPATH=root)
    env.pop("UFAIR_DEBUG_TRIP", None)
    sel = ["tests/test_gpu_period_means.py::test_period_outputs_stay_inside_their_rows",
           "tests/test_gpu_period_means.py::test_period_means_equal_the_mean_of_the_per_step_rows"]
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider"] + sel,
                       cwd=root, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    ok = subprocess.run([sys.executable, "-c", _TRIP], cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert ok.returncode == 0 and "completed" in ok.stdout, ok.stderr[-2000:]
    trip = subprocess.run([sys.executable, "-c", _TRIP], cwd=root, env=dict(env, UFAIR_DEBUG_TRIP="1"),
                          capture_output=True, text=True, timeout=600)
    assert trip.returncode != 0 and "completed" not in trip.stdout
    assert "debug bounds check" in trip.stderr and "output stores in the last 1 row(s)" in trip.stderr, trip.stderr[-2000:]


# ------------------------------------------------------------------ 9. full size: configs[4]
def test_full_size_annual_means_of_a_tenth_of_a_year_run(api):
    """configs[4]: 10^6 members x 7360 steps of 0.1 yr, scenario-shared emissions and forcing.  Annual means of C, RF
    and T plus statistics in one device-resident call (41 GB of outputs instead of 412); its T equals, bit for bit,
    the sequential mean of the per-step T-only run's rows, computed on the device."""
    import torch

    from fiveeqscm_b200 import params as P
    M, n_t, dt, k = 1_000_000, 7360, 0.1, 10
    torch.cuda.empty_cache()
    ens = P.sample_ensemble(M, n_t=n_t, dt=dt, seed=4, dense_pools=True)   # scenario tables: no per-member expansion
    kw = dict(dt=dt, scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]), f_ext=to_dev(ens["f_ext"]))
    gp, tp, E = to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), to_dev(ens["scen"])
    spec = api.HistSpec(lo=-1.0, hi=4.0)
    mean = api.run_ensemble(E, gp, tp, out_every=k, stats=spec, **kw)
    assert mean.C.shape == (3, n_t // k, M) and mean.hist.shape == (n_t // k, spec.bins)
    one = api.run_ensemble(E, gp, tp, outputs=("T",), **kw)
    v = one.T.reshape(n_t // k, k, M)
    s = torch.zeros(n_t // k, M, dtype=torch.float64, device="cuda")
    for j in range(k):
        s = s + v[:, j]
    s = s * (1.0 / k)
    assert torch.equal(mean.T, s)
    assert torch.equal(mean.state, one.state)
    assert bool((mean.hist.sum(dim=1) == M).all())
    assert torch.isfinite(mean.C).all() and torch.isfinite(mean.RF).all()
