"""Float32 outputs of FP64 runs (``out_dtype="f32"``, UFAIR_OUTTYPE_F32): the integration stays FP64 and every stored
C, RF and T value is the round-to-nearest-even float32 of the value the same run stores in FP64.

That rule is exact, so the checks here are bitwise: the float32-output run against the FP64-output run of the same
descriptor, cast to float32.  The state stays FP64 and must not move at all."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from tests.group_stats_ref import grouped_temperature_stats
from tests.test_gpu_guard import GASES, Guarded
from tests.util import ensemble, to_dev, to_np

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fiveeqscm_b200 import concentrations
    return concentrations


def _np(x):
    return x if isinstance(x, np.ndarray) else to_np(x)


def _cast_equal(got, want64, what):
    """got (float32) is want64 (float64) rounded to float32, bit for bit, with NaN in the same places."""
    got, want64 = _np(got), _np(want64)
    assert got.dtype == np.float32 and want64.dtype == np.float64, what
    want = want64.astype(np.float32)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan, err_msg=f"{what}: NaN positions")
    np.testing.assert_array_equal(got.view(np.uint32)[~nan], want.view(np.uint32)[~nan], err_msg=what)


def _assert_run_cast(f32, f64, keys=("C", "RF", "T"), what=""):
    for key in keys:
        _cast_equal(getattr(f32, key), getattr(f64, key), f"{what} {key}")
    if f64.state is not None:
        np.testing.assert_array_equal(to_np(f32.state).view(np.uint64), to_np(f64.state).view(np.uint64),
                                      err_msg=f"{what} state")


def _inputs(ens, layout, fext):
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


def _plan(api, ens, E, **kw):
    return api.DevicePlan(E, to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), **kw)


def _pair(api, ens, E, **kw):
    """(float32-output plan, its result, the FP64-output result) of one descriptor."""
    p = _plan(api, ens, E, out_dtype="f32", **kw)
    return p, p.run(), _plan(api, ens, E, **kw).run()


# ------------------------------------------------------------------ 1. bitwise against the cast FP64 run
@pytest.mark.parametrize("alpha_mode", ["exp", "sinh", "newton", "one"])
@pytest.mark.parametrize("G", [1, 2, 3, 4])
def test_f32_outputs_equal_the_cast_fp64_run(api, alpha_mode, G):
    n_t, M = 20, 203
    ens = ensemble(M, n_t=n_t, gases=GASES[G], dense=True, seed=300 + G)
    for layout in ("member", "scenario"):
        for fext in ("none", "shared", "member"):
            E, kw = _inputs(ens, layout, fext)
            for iirf_max in (None, 45.0):   # 45: the iIRF ceiling binds for most members
                p, f32, f64 = _pair(api, ens, E, alpha_mode=alpha_mode, newton_iters=2, iirf_max=iirf_max, **kw)
                assert f32.T.dtype == f32.C.dtype == f32.RF.dtype == p.out_dtype and f32.state.dtype == f64.state.dtype
                assert p.kernel_variant()[1] == G   # all gases per lane
                _assert_run_cast(f32, f64, what=f"{layout} {fext} {iirf_max}")


# ------------------------------------------------------------------ 2. every loop, the forms, the variant report
LOOPS = [  # (run_ensemble keywords, the loop that must run)
    (dict(iirf_max=60.0), "general"),
    (dict(), "plain"),
    (dict(f_ext="shared"), "plain_fext"),
    (dict(f_ext="member"), "plain_fext"),
    (dict(outputs=(), stats="spec"), "plain_subset"),   # statistics only: a float32 T scratch
    (dict(outputs=("C", "RF"), f_ext="shared"), "plain_subset"),
    (dict(out_every=10), "period_mean"),
    (dict(out_every=10, outputs=("T",), iirf_max=60.0, f_ext="member"), "period_mean"),
]


@pytest.mark.parametrize("kw,loop", LOOPS, ids=[f"{lp}-{i}" for i, (_, lp) in enumerate(LOOPS)])
@pytest.mark.parametrize("dense", [True, False], ids=["dense", "forms"])
def test_every_loop_and_form(api, kw, loop, dense):
    n_t, M = 40, 517
    ens = ensemble(M, n_t=n_t, dense=dense, seed=77)
    kw = dict(kw)
    fext = kw.pop("f_ext", "none")
    if kw.get("stats") == "spec":
        kw["stats"] = api.HistSpec(lo=-1.0, hi=3.0, bins=64, copies=2)
    E, extra = _inputs(ens, "member", fext)
    p, f32, f64 = _pair(api, ens, E, **kw, **extra)
    form, gpl, _ = p.kernel_variant()
    assert p.loop_variant == loop and gpl == 3
    if not dense:
        assert any(form)   # literature parameters: the specialised forms
    outs = kw.get("outputs", ("C", "RF", "T"))
    _assert_run_cast(f32, f64, keys=outs, what=loop)
    if "stats" in kw:   # FP32 binning of the stored float32 rows, not of the FP64 ones
        scratch = to_np(p._t_scratch)[:, :M]
        _cast_equal(scratch, _plan(api, ens, E, outputs=("T",), **extra).run().T, "T scratch")
        h_ref, _ = grouped_temperature_stats(scratch, -1.0, 3.0, 64, np.zeros(M, np.int64), 1)
        np.testing.assert_array_equal(to_np(f32.hist).astype(np.uint64), h_ref[0])


@pytest.mark.parametrize("M", [100_000, 100_032])
def test_both_sides_of_the_small_ensemble_mapping(api, M):
    """At most UFAIR_SMALL_ENSEMBLE FP64 members run one gas per lane with FP64 outputs; float32 outputs never do."""
    n_t = 16
    ens = ensemble(M, n_t=n_t, dense=True, seed=5)
    E = to_dev(ens["E"])
    p, f32, f64 = _pair(api, ens, E, f_ext=to_dev(ens["f_ext"]))
    assert _plan(api, ens, E).kernel_variant()[1] == (1 if M <= 100_000 else 3)
    assert p.kernel_variant()[1] == 3
    _assert_run_cast(f32, f64)


@pytest.mark.parametrize("k", [10])
def test_period_means_are_rounded_once_at_the_store(api, k):
    n_t, M = 120, 1001
    ens = ensemble(M, n_t=n_t, dense=True, seed=8)
    E, kw = _inputs(ens, "scenario", "shared")
    p, f32, f64 = _pair(api, ens, E, out_every=k, **kw)
    p.kernel_variant()
    assert f32.T.shape == (n_t // k, M) and p.loop_variant == "period_mean"
    _assert_run_cast(f32, f64, what=f"out_every={k}")


def test_f32_run_accepts_f32_outputs_and_changes_nothing(api):
    ens = ensemble(300, n_t=12, dense=True, seed=2)
    E = to_dev(ens["E"])
    a = _plan(api, ens, E, precision="f32", out_dtype="f32", outputs=("C", "T", "alpha")).run()
    b = _plan(api, ens, E, precision="f32", outputs=("C", "T", "alpha")).run()
    for key in ("C", "T", "alpha", "state"):
        np.testing.assert_array_equal(to_np(getattr(a, key)), to_np(getattr(b, key)), err_msg=key)


# ------------------------------------------------------------------ 3. composition
def test_two_time_chunks_equal_one_call(api):
    import torch
    n_t, n1, M = 60, 24, 900
    ens = ensemble(M, n_t=n_t, dense=True, seed=9)
    spec = api.HistSpec(lo=-1.0, hi=3.0, bins=256, copies=3)
    gp, tp = to_dev(ens["gas_params"]), to_dev(ens["thermal_params"])
    kw = dict(out_dtype="f32", stats=spec)
    full = api.DevicePlan(to_dev(ens["E"]), gp, tp, **kw).run()
    p1 = api.DevicePlan(to_dev(ens["E"][:, :n1]), gp, tp, **kw)
    r1 = p1.result
    p1.launch()
    assert r1.state.dtype == torch.float64   # the resume state stays FP64
    p2 = api.DevicePlan(to_dev(ens["E"][:, n1:]), gp, tp, state_in=r1.state, **kw)
    hp = torch.empty(spec.copies, n_t, spec.bins, dtype=torch.int32, device="cuda")
    mp = torch.empty(spec.copies, n_t, _abi.MOM_COUNT, dtype=torch.float64, device="cuda")
    hist = torch.empty(n_t, spec.bins, dtype=torch.int64, device="cuda")
    mom = torch.empty(n_t, _abi.MOM_COUNT, dtype=torch.float64, device="cuda")
    for p, t0 in ((p1, 0), (p2, n1)):
        p.desc.hist_private, p.desc.moments_private = hp.data_ptr(), mp.data_ptr()
        p.desc.hist_rows, p.desc.hist_t0 = n_t, t0
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


@pytest.mark.parametrize("chunk", [1024, 65536], ids=["no-ramp", "ramp"])
def test_host_pipeline_equals_the_device_path(api, chunk):
    """1024-member chunks start at full size; 65 536-member ones ramp up from 8192 over the 20 003 members."""
    n_t, M = 50, 20_003
    ens = ensemble(M, n_t=n_t, dense=True, seed=21)
    spec = api.HistSpec(copies=4)
    kw = dict(scen_idx=ens["scen_idx"], e_scale=ens["e_scale"], f_ext=ens["f_ext"], out_dtype="f32", stats=spec)
    dev = api.run_ensemble(to_dev(ens["scen"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]),
                           **{key: to_dev(v) if isinstance(v, np.ndarray) else v for key, v in kw.items()})
    host = api.run_ensemble(ens["scen"], ens["gas_params"], ens["thermal_params"], chunk_members=chunk, **kw)
    out = api.pinned_result(3, n_t, M, stats=spec, out_dtype="f32")
    ws = api.Workspace(0, chunk)
    reused = api.run_ensemble(ens["scen"], ens["gas_params"], ens["thermal_params"], workspace=ws, out=out, **kw)
    ws.close()
    assert reused is out and out.T.dtype == np.float32 and out.state.dtype == np.float64
    for r in (host, reused):
        for key in ("C", "RF", "T", "state", "hist"):
            np.testing.assert_array_equal(getattr(r, key), to_np(getattr(dev, key)), err_msg=key)
        np.testing.assert_allclose(r.moments, to_np(dev.moments), rtol=1e-12)


# ------------------------------------------------------------------ 4. statistics
@pytest.mark.parametrize("grouping", ["pooled", "scenario", "labels"])
def test_statistics_recount_the_stored_float32_rows(api, grouping):
    import torch
    n_t, M = 60, 30_000
    ens = ensemble(M, n_t=n_t, dense=True, seed=12)
    spec = api.HistSpec(lo=-1.0, hi=3.0, bins=512, copies=5)
    kw = dict(scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]), f_ext=to_dev(ens["f_ext"]))
    n_g, labels = 1, np.zeros(M, dtype=np.int64)
    if grouping == "scenario":
        kw["stat_group"], n_g, labels = "scenario", ens["scen"].shape[2], ens["scen_idx"]
    elif grouping == "labels":
        labels = np.random.default_rng(4).integers(-2, 7, M)   # negative labels are counted nowhere
        n_g, kw["stat_group"] = 7, to_dev(labels.astype(np.int32))
        spec.groups = 7
    E = to_dev(ens["scen"])
    res = _plan(api, ens, E, out_dtype="f32", stats=spec, **kw).run()
    only = _plan(api, ens, E, out_dtype="f32", stats=spec, outputs=(), **kw).run()   # a float32 T scratch
    T = to_np(res.T)
    assert T.dtype == np.float32
    h_ref, m_ref = grouped_temperature_stats(T, spec.lo, spec.hi, spec.bins, labels, n_g)
    hist, mom = to_np(res.hist), to_np(res.moments)
    if grouping == "pooled":
        h_ref, m_ref = h_ref[0], m_ref[0]
    np.testing.assert_array_equal(hist.astype(np.uint64), h_ref)
    np.testing.assert_allclose(mom, m_ref, rtol=1e-12)
    np.testing.assert_array_equal(to_np(only.hist), hist)
    np.testing.assert_array_equal(to_np(only.moments), mom)
    torch.cuda.synchronize()


# ------------------------------------------------------------------ 5. guard bands
GUARD_CASES = [  # (n_gas, M, ld, n_t, out_every, per-member emissions, form, stats); ld = 2 (mod 4): 8-byte f32 rows
    (3, 1003, 1006, 30, 1, True, False, True),
    (1, 95, 98, 18, 3, False, False, True),
    (4, 259, 262, 20, 1, True, True, False),
    (2, 515, 522, 24, 4, False, False, True),
    (3, 70, 74, 16, 1, True, True, True),
]


@pytest.mark.parametrize("G,M,ld,n_t,k,e_member,form,stats", GUARD_CASES, ids=lambda v: str(v).replace(" ", ""))
def test_f32_outputs_stay_inside_their_rows(api, G, M, ld, n_t, k, e_member, form, stats):
    import torch
    assert ld % 4 == 2
    n_out = n_t // k
    ens = ensemble(M, n_t=n_t, gases=GASES[G], dense=not form, seed=7 + M)
    run = {}
    for out_type, odt in ((_abi.OUTTYPE_F32, np.float32), (_abi.OUTTYPE_RUN, np.float64)):
        mk = lambda rows, dt=np.float64: Guarded(rows, M, ld, dt, True)
        b = {"gp": mk(G * _abi.GP_COUNT).fill(ens["gas_params"]), "tp": mk(_abi.TP_COUNT).fill(ens["thermal_params"]),
             "oC": mk(G * n_out, odt), "oRF": mk(G * n_out, odt), "oT": mk(n_out, odt), "state": mk(_abi.state_rows(G))}
        d = _abi.UfairDesc(n_gas=G, n_t=n_t, n_member=M, ld_member=ld, out_mask=_abi.OUT_C | _abi.OUT_RF | _abi.OUT_T,
                           out_every=k, out_type=out_type, gas_params=b["gp"].ptr, thermal_params=b["tp"].ptr,
                           out_C=b["oC"].ptr, out_RF=b["oRF"].ptr, out_T=b["oT"].ptr, state_out=b["state"].ptr)
        keep = []
        if e_member:
            b["E"] = mk(G * n_t).fill(ens["E"])
            d.emissions, d.e_mode = b["E"].ptr, _abi.E_MEMBER
        else:
            keep = [to_dev(ens["scen"]), to_dev(ens["scen_idx"].astype(np.int32))]
            b["esc"] = mk(G).fill(ens["e_scale"])
            d.emissions, d.scen_idx, d.e_scale, d.e_mode = keep[0].data_ptr(), keep[1].data_ptr(), b["esc"].ptr, _abi.E_SCENARIO
            d.n_scen = ens["scen"].shape[2]
        if form:
            from fiveeqscm_b200.concentrations import _detect_form_host
            for g, f in enumerate(_detect_form_host(ens["gas_params"], None)):
                d.gas_form[g] = f
        L = _abi.lib()
        if stats:   # the statistics pass over the 8-byte-aligned float32 rows
            spec = dict(bins=128, copies=3, lo=-1.0, hi=3.0)
            hp = torch.empty(spec["copies"], n_out, spec["bins"], dtype=torch.int32, device="cuda")
            mp = torch.empty(spec["copies"], n_out, _abi.MOM_COUNT, dtype=torch.float64, device="cuda")
            hist = torch.empty(n_out, spec["bins"], dtype=torch.int64, device="cuda")
            mom = torch.empty(n_out, _abi.MOM_COUNT, dtype=torch.float64, device="cuda")
            d.stats, d.hist_bins, d.hist_copies, d.hist_lo, d.hist_hi = 1, spec["bins"], spec["copies"], spec["lo"], spec["hi"]
            d.hist_rows, d.hist_private, d.moments_private = n_out, hp.data_ptr(), mp.data_ptr()
            _abi.check(L.ufair_stats_reset(C.byref(d), None))
        _abi.check(L.ufair_run_f64(C.byref(d), None))
        if stats:
            _abi.check(L.ufair_stats_pass_f64(C.byref(d), None))
            _abi.check(L.ufair_stats_finalize(C.byref(d), hist.data_ptr(), mom.data_ptr(), None))
        torch.cuda.synchronize()
        for name, buf in b.items():
            buf.check(name, written=name.startswith("o") or name == "state")
        run[out_type] = {name: buf.data() for name, buf in b.items() if name.startswith("o") or name == "state"}
        if stats and out_type == _abi.OUTTYPE_F32:
            h_ref, m_ref = grouped_temperature_stats(run[out_type]["oT"], spec["lo"], spec["hi"], spec["bins"],
                                                     np.zeros(M, np.int64), 1)
            np.testing.assert_array_equal(to_np(hist).astype(np.uint64), h_ref[0])
            np.testing.assert_allclose(to_np(mom), m_ref[0], rtol=1e-12)
    f32, f64 = run[_abi.OUTTYPE_F32], run[_abi.OUTTYPE_RUN]
    for name in ("oC", "oRF", "oT"):
        _cast_equal(f32[name], f64[name], name)
    np.testing.assert_array_equal(f32["state"], f64["state"])


# ------------------------------------------------------------------ 6. the checked build (libufair_dbg.so)
_DBG = os.path.join(os.path.dirname(_abi.lib_path()), "libufair_dbg.so")
_TRIP = """
import numpy as np, torch
from fiveeqscm_b200 import concentrations as api
from tests.util import ensemble, to_dev
ens = ensemble(70, n_t=12)
res = api.run_ensemble(to_dev(ens["E"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), out_dtype="f32")
torch.cuda.synchronize()
print("completed")
"""


@pytest.mark.skipif(not os.path.exists(_DBG), reason="libufair_dbg.so not built (make -C fiveeqscm_b200/csrc debug)")
def test_f32_outputs_on_the_debug_bounds_build():
    """The guard and cast cases of this file on the build whose kernels check every output store against its array
    (float32 pointers here), then its negative control: with UFAIR_DEBUG_TRIP=1 the store check pretends the last
    output row is missing and must count the float32 stores there (it counts, it never traps)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, UFAIR_LIB=_DBG, PYTHONPATH=root)
    env.pop("UFAIR_DEBUG_TRIP", None)
    sel = ["tests/test_gpu_f32_outputs.py::test_f32_outputs_stay_inside_their_rows",
           "tests/test_gpu_f32_outputs.py::test_every_loop_and_form"]
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider"] + sel,
                       cwd=root, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    ok = subprocess.run([sys.executable, "-c", _TRIP], cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert ok.returncode == 0 and "completed" in ok.stdout, ok.stderr[-2000:]
    trip = subprocess.run([sys.executable, "-c", _TRIP], cwd=root, env=dict(env, UFAIR_DEBUG_TRIP="1"),
                          capture_output=True, text=True, timeout=600)
    assert trip.returncode != 0 and "completed" not in trip.stdout
    assert "debug bounds check" in trip.stderr and "output stores in the last 1 row(s)" in trip.stderr, trip.stderr[-2000:]


# ------------------------------------------------------------------ 7. full size: the configs[3] shard
def test_full_size_shard_with_f32_outputs(api):
    """1.25e6 members x 736 steps x 3 gases, device-resident, float32 C, RF and T (26 GB instead of 52) plus
    statistics; a member block equals the FP64-output run of the same members, cast, bit for bit."""
    import torch

    from fiveeqscm_b200 import params as P
    M, n_t, lo, hi = 1_250_000, 736, 0, 131_072
    torch.cuda.empty_cache()
    ens = P.sample_ensemble(M, n_t=n_t, seed=11, dense_pools=True)   # scenario tables: no per-member expansion
    gp, tp = to_dev(ens["gas_params"]), to_dev(ens["thermal_params"])
    kw = dict(f_ext=to_dev(ens["f_ext"]))
    spec = api.HistSpec(lo=-1.0, hi=4.0)
    full = api.run_ensemble(to_dev(ens["scen"]), gp, tp, scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]),
                            out_dtype="f32", stats=spec, **kw)
    assert full.C.dtype == torch.float32 and full.C.shape == (3, n_t, M) and full.state.dtype == torch.float64
    assert bool((full.hist.sum(dim=1) == M).all())
    blk = api.run_ensemble(to_dev(ens["scen"]), gp[..., lo:hi].contiguous(), tp[..., lo:hi].contiguous(),
                           scen_idx=to_dev(ens["scen_idx"][lo:hi]), e_scale=to_dev(ens["e_scale"][:, lo:hi]), **kw)
    for key in ("C", "RF", "T"):
        got, want = getattr(full, key)[..., lo:hi], getattr(blk, key)
        assert torch.equal(torch.isnan(got), torch.isnan(want)), key
        assert torch.equal(got, want.to(torch.float32)), key
    assert torch.equal(full.state[:, lo:hi], blk.state)
