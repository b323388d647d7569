"""GPU parity tests: the CUDA path, called through the C ABI (ctypes binding), against the CPU oracle
on identical seeded inputs.  Tolerances (BASELINE.json north_star):
  FP64: <= 1e-10 relative vs the float64 oracle, each output on its own scale: C, RF and alpha gas by gas,
        the state row by row, T as a whole (tests/util.py output_relerr; RF, T and the temperature rows of
        the state with a 0.01 W m-2 / K floor on the scale);
  FP32: <= 1e-4 K in temperature, each gas's concentrations within 2e-5 of that gas's scale.
Integer work (histogram counts) is bit-exact.
"""
import os
from types import SimpleNamespace

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import params as P
from oracle import c_oracle as co
from oracle import ufair_oracle as o
from tests.util import TOL64, assert_parity, ensemble, field_relerr, slice_relerr, to_dev, to_np

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "hfc_reference.npz")


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    from fiveeqscm_b200 import concentrations as c
    _abi.lib()  # the CUDA library must be present: no fallback
    return c


def _run_dev(api, ens, *, E=None, **kw):
    import torch
    E = ens["E"] if E is None else E
    res = api.run_ensemble(to_dev(E), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), **kw)
    torch.cuda.synchronize()
    return res


def _check(res, ref, keys=("C", "RF", "T"), tol=TOL64):
    assert_parity(res, ref, keys, tol)


def _check32(res, ref):
    """FP32: T within 1e-4 K of the float64 oracle, each gas's C within 2e-5 of that gas's own scale."""
    assert res.T.dtype.itemsize == 4
    err_T = np.max(np.abs(to_np(res.T).astype(np.float64) - ref["T"]))
    assert err_T <= 1e-4, f"T off by {err_T:.3e} K"
    err_C = slice_relerr(to_np(res.C), ref["C"])
    assert err_C < 2e-5, f"C relative error {err_C:.3e}"


# ------------------------------------------------------------------ a1: the reference's function
def _golden_cases():
    z = np.load(GOLDEN)
    names = sorted({k.split("__")[0] for k in z.files})
    return [(n, z[f"{n}__emissions"], z[f"{n}__time"], float(z[f"{n}__lifetime"]), z[f"{n}__expected"]) for n in names]


def test_reference_test_file_itself_passes_unmodified(api):
    """The reference's own test FILE (tests/unit/test_hfcs.py, vendored byte for byte as
    tests/golden/ref_test_hfcs.py -- sha256 pinned in tests/test_host_logic.py), run by pytest in a
    fresh interpreter against this repo's U_FaIR package: the drop-in claim of SURVEY.md 8b."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-c", os.devnull, "--rootdir", root,
                        os.path.join(root, "tests", "golden", "ref_test_hfcs.py")],
                       cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "1 passed" in r.stdout, r.stdout + r.stderr
    # ... and it really was this repo's CUDA implementation that answered
    import U_FaIR.concentrations as uc
    assert os.path.dirname(os.path.abspath(uc.__file__)) == os.path.join(root, "U_FaIR")


def test_reference_test_reads_unchanged(api):
    # reference tests/unit/test_hfcs.py:5-13, through the drop-in module path
    from U_FaIR.concentrations import calculate_hfc_conc
    time = np.array([0, 1, 2, 3])
    input_emissions = np.array([10, 0, 0, 0])
    expected = 10 * np.exp(-time)
    result = calculate_hfc_conc(input_emissions, time, lifetime=1.0)
    np.testing.assert_allclose(result, expected)


@pytest.mark.parametrize("case", _golden_cases(), ids=lambda c: c[0])
def test_hfc_matches_reference_fixtures(api, case):
    _, e, t, life, expected = case
    got = api.calculate_hfc_conc(e, t, life)
    assert got.dtype == np.float64 and got.shape == expected.shape
    np.testing.assert_allclose(got, expected, rtol=4.5e-16, atol=0)   # CUDA exp vs numpy exp: <= 2 ulp


def test_hfc_physical_opt_in(api):
    # reference TODOs (tests/unit/test_hfcs.py:15-16): constant emissions; pulse not in year zero
    t = np.arange(0.0, 30.0, 0.5)
    got = api.calculate_hfc_conc(np.full(t.size, 2.0), t, 7.0, strict=False)
    np.testing.assert_allclose(got, 2.0 * 7.0 * (1 - np.exp(-(t + 0.5) / 7.0)), rtol=1e-13)
    e = np.zeros(t.size)
    e[4] = 3.0
    got = api.calculate_hfc_conc(e, t, 7.0, strict=False)
    assert np.all(got[:4] == 0.0)
    first = 3.0 * 7.0 * (1 - np.exp(-0.5 / 7.0))
    np.testing.assert_allclose(got[4:], first * np.exp(-(t[4:] - t[4]) / 7.0), rtol=1e-13)


# ------------------------------------------------------------------ configs[0], configs[1]
def test_config0_single_co2_default_params(api):
    """BASELINE configs[0]: CO2 only, one default parameter set, annual emissions 1765-2500."""
    gp, tp = P.default_params(1, gases=("co2",))
    E = P.scenario_emissions(736, gases=("co2",))[:, :, 1:2]          # [1][736][1]
    ens = dict(gas_params=gp, thermal_params=tp)
    res = _run_dev(api, ens, E=E)
    ref_c = co.oxfair(E, gp, tp)
    ref_np = o.oxfair(E, gp, tp)
    _check(res, ref_c)
    _check(res, ref_np)
    assert 500 < ref_np["C"][0, -1, 0] < 2000 and 1.0 < ref_np["T"][-1, 0] < 8.0   # sane physics


@pytest.mark.parametrize("dense", [True, False])
def test_config1_3gas_1e4_members(api, dense):
    """BASELINE configs[1]: CO2/CH4/N2O, 10^4-member sampled ensemble, 736 annual steps."""
    ens = ensemble(10_000, dense=dense)
    res = _run_dev(api, ens, f_ext=to_dev(ens["f_ext"]), outputs=("C", "RF", "T", "alpha"))
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=ens["f_ext"], want_alpha=True)
    _check(res, ref, keys=("C", "RF", "T", "alpha", "state"))
    # elementwise too, where the field is not near zero
    T, Tr = to_np(res.T), ref["T"]
    big = np.abs(Tr) > 0.1
    assert np.max(np.abs(T[big] - Tr[big]) / np.abs(Tr[big])) < TOL64


# ------------------------------------------------------------------ every mode, small sizes
MODES = [
    dict(alpha_mode="exp"),
    dict(alpha_mode="exp", iirf_max=60.0, t_mode="end"),
    dict(alpha_mode="sinh"),
    dict(alpha_mode="newton", newton_iters=3, iirf_max=97.0),
    dict(alpha_mode="newton", newton_iters=0),
    dict(alpha_mode="one", t_mode="end"),
]
_OKW = {"exp": o.ALPHA_EXP, "sinh": o.ALPHA_SINH, "newton": o.ALPHA_NEWTON, "one": o.ALPHA_ONE}


def _oracle_kw(kw):
    out = dict(kw)
    out["alpha_mode"] = _OKW[kw["alpha_mode"]]
    if "t_mode" in out:
        out["t_mode"] = o.T_END if out["t_mode"] == "end" else o.T_MID
    return out


@pytest.mark.parametrize("kw", MODES, ids=lambda k: "-".join(f"{a}={b}" for a, b in k.items()))
@pytest.mark.parametrize("n_gas", [1, 2, 3, 4])
def test_modes_and_gas_counts(api, kw, n_gas):
    gases = ("co2", "ch4", "n2o", "hfc")[:n_gas]
    ens = ensemble(777, n_t=300, dense=True, gases=gases, seed=11 + n_gas)
    res = _run_dev(api, ens, f_ext=to_dev(ens["f_ext"]), outputs=("C", "RF", "T", "alpha"), **kw)
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=ens["f_ext"], want_alpha=True,
                    **_oracle_kw(kw))
    _check(res, ref, keys=("C", "RF", "T", "alpha", "state"))


@pytest.mark.parametrize("kw", MODES, ids=lambda k: "-".join(f"{a}={b}" for a, b in k.items()))
@pytest.mark.parametrize("n_gas", [1, 2, 3, 4])
def test_modes_and_gas_counts_fp32(api, kw, n_gas):
    """The same runs on the FP32 instantiations (the general loop where alpha is an output)."""
    gases = ("co2", "ch4", "n2o", "hfc")[:n_gas]
    ens = ensemble(777, n_t=300, dense=True, gases=gases, seed=11 + n_gas)
    res = _run_dev(api, ens, f_ext=to_dev(ens["f_ext"]), outputs=("C", "RF", "T", "alpha"), precision="f32", **kw)
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=ens["f_ext"], **_oracle_kw(kw))
    _check32(res, ref)


@pytest.mark.parametrize("M", [1, 2, 3, 31, 127, 128, 129, 255, 1001])
def test_ragged_member_counts(api, M):
    ens = ensemble(M, n_t=97, dense=True, seed=M)          # 97: also a ragged last time tile
    res = _run_dev(api, ens)
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"])
    _check(res, ref, keys=("C", "RF", "T", "state"))
    assert res.C.shape == (3, 97, M) and res.T.shape == (97, M)


def test_empty_inputs(api):
    ens = ensemble(4, n_t=5)
    res = _run_dev(api, ens, E=ens["E"][:, :0])      # zero time steps
    assert res.T.shape == (0, 4)
    import torch
    z = lambda *s: torch.zeros(*s, dtype=torch.float64, device="cuda")
    res = api.run_ensemble(z(3, 5, 0), z(3, 17, 0), z(4, 0))   # zero members
    assert res.T.shape == (5, 0)
    res = api.run_ensemble(np.zeros((3, 5, 2)), np.zeros((3, 17, 0)), np.zeros((4, 0)),   # host pipeline, scenario inputs
                           scen_idx=np.zeros(0, dtype=np.int32))
    assert res.T.shape == (5, 0)


def test_scenario_shared_emissions_and_forcing(api):
    """configs[2] layout: emissions shared per scenario, per-member scenario index and scale."""
    ens = ensemble(5000, n_t=400, dense=True)
    n_s = ens["scen"].shape[2]
    fx = np.stack([ens["f_ext"] * (1 + 0.1 * s) for s in range(n_s)], axis=1)
    res = api.run_ensemble(to_dev(ens["scen"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]),
                           scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]), f_ext=to_dev(fx))
    ref = co.oxfair(ens["scen"], ens["gas_params"], ens["thermal_params"], scen_idx=ens["scen_idx"],
                    e_scale=ens["e_scale"], f_ext=fx)
    _check(res, ref, keys=("C", "RF", "T", "state"))
    # and it is the same thing as expanding the emissions per member
    fx_m = fx[:, ens["scen_idx"]]
    res2 = _run_dev(api, ens, f_ext=to_dev(fx_m), fext_per_member=True)
    for k in ("C", "RF", "T"):
        np.testing.assert_array_equal(to_np(getattr(res, k)), to_np(getattr(res2, k)))


def test_subannual_timestep(api):
    """configs[4] shape: dt = 0.1 yr, 7360 steps (fewer members so the oracle stays fast)."""
    ens = ensemble(512, n_t=7360, dt=0.1, dense=True)
    res = _run_dev(api, ens, dt=0.1, f_ext=to_dev(ens["f_ext"]))
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], dt=0.1, f_ext=ens["f_ext"])
    _check(res, ref, keys=("C", "RF", "T", "state"))


def test_time_chunked_resume_is_bitwise(api):
    ens = ensemble(1000, n_t=200)
    full = _run_dev(api, ens)
    a = _run_dev(api, ens, E=ens["E"][:, :77])
    b = _run_dev(api, ens, E=ens["E"][:, 77:], state_in=a.state)
    np.testing.assert_array_equal(np.concatenate([to_np(a.T), to_np(b.T)]), to_np(full.T))
    np.testing.assert_array_equal(np.concatenate([to_np(a.C), to_np(b.C)], axis=1), to_np(full.C))
    np.testing.assert_array_equal(to_np(b.state), to_np(full.state))


def test_member_independence_is_bitwise(api):
    """Any member block integrates to the same bits alone as inside a larger launch."""
    ens = ensemble(3000, n_t=150)
    full = _run_dev(api, ens)
    sl = slice(1000, 1700)
    sub = dict(gas_params=ens["gas_params"][:, :, sl], thermal_params=ens["thermal_params"][:, sl])
    part = _run_dev(api, sub, E=ens["E"][:, :, sl])
    np.testing.assert_array_equal(to_np(part.T), to_np(full.T)[:, sl])
    np.testing.assert_array_equal(to_np(part.RF), to_np(full.RF)[:, :, sl])


# ------------------------------------------------------------------ statistics
def test_histogram_bit_exact_and_moments(api):
    ens = ensemble(20_000, n_t=300, dense=True)
    spec = api.HistSpec(lo=-5.0, hi=25.0, bins=1024, copies=7)
    res = _run_dev(api, ens, stats=spec)
    T = to_np(res.T)
    h_ref, m_ref = co.temperature_stats(T, spec.lo, spec.hi, spec.bins)
    np.testing.assert_array_equal(to_np(res.hist).astype(np.uint64), h_ref)     # integer work: bit-exact
    assert np.all(to_np(res.hist).sum(axis=1) == 20_000)
    mom = to_np(res.moments)
    np.testing.assert_allclose(mom[:, :2], m_ref[:, :2], rtol=1e-12)
    np.testing.assert_array_equal(mom[:, 2:], m_ref[:, 2:])                     # min / max: exact
    # against the oracle's own T the histogram may differ only where T sits on a bin edge
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"])
    h_or, _ = co.temperature_stats(ref["T"], spec.lo, spec.hi, spec.bins)
    assert np.abs(to_np(res.hist).astype(np.int64) - h_or.astype(np.int64)).sum() <= 4
    from fiveeqscm_b200 import stats as S
    pct = S.percentiles(res.hist, spec.lo, spec.hi, [5, 50, 95])
    direct = np.percentile(T, [5, 50, 95], axis=1).T
    assert np.max(np.abs(pct - direct)) < 2 * (spec.hi - spec.lo) / spec.bins
    # the device percentile kernel is bit-identical to the oracle's CDF walk (and to the host one)
    pcts = [0.0, 1.0, 5.0, 17.0, 50.0, 83.0, 95.0, 99.9, 100.0]
    pct_dev = to_np(S.percentiles_device(res.hist, spec.lo, spec.hi, pcts))
    np.testing.assert_array_equal(pct_dev, o.percentiles_from_hist(to_np(res.hist), spec.lo, spec.hi, pcts))
    np.testing.assert_array_equal(pct_dev, S.percentiles(res.hist, spec.lo, spec.hi, pcts))


def test_histogram_outliers_and_narrow_range(api):
    ens = ensemble(4096, n_t=64)
    spec = api.HistSpec(lo=0.2, hi=0.6, bins=16, copies=3)     # most values fall outside: edge bins
    res = _run_dev(api, ens, stats=spec, outputs=("T",))
    h_ref, _ = co.temperature_stats(to_np(res.T), spec.lo, spec.hi, spec.bins)
    np.testing.assert_array_equal(to_np(res.hist).astype(np.uint64), h_ref)


# ------------------------------------------------------------------ FP32 mode
def test_fp32_mode_temperature_within_1e4_K(api):
    ens = ensemble(10_000, dense=True)
    res = _run_dev(api, ens, f_ext=to_dev(ens["f_ext"]), precision="f32")
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=ens["f_ext"])
    _check32(res, ref)


# ------------------------------------------------------------------ host pipeline == device path
@pytest.mark.parametrize("chunk", [256, 4096])
def test_host_pipeline_matches_device_path(api, chunk):
    ens = ensemble(1000, n_t=120, dense=True)
    spec = api.HistSpec(copies=4)
    dev = _run_dev(api, ens, f_ext=to_dev(ens["f_ext"]), stats=spec, outputs=("C", "RF", "T", "alpha"))
    host = api.run_ensemble(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=ens["f_ext"], stats=spec,
                            outputs=("C", "RF", "T", "alpha"), chunk_members=chunk)
    for k in ("C", "RF", "T", "alpha", "state"):
        assert isinstance(getattr(host, k), np.ndarray)
        np.testing.assert_array_equal(getattr(host, k), to_np(getattr(dev, k)))
    np.testing.assert_array_equal(host.hist, to_np(dev.hist))
    np.testing.assert_allclose(host.moments, to_np(dev.moments), rtol=1e-12)


def test_host_pipeline_scenario_mode_and_resume(api):
    ens = ensemble(900, n_t=90)
    a = api.run_ensemble(ens["scen"], ens["gas_params"], ens["thermal_params"], scen_idx=ens["scen_idx"],
                         e_scale=ens["e_scale"], chunk_members=384)
    ref = co.oxfair(ens["scen"], ens["gas_params"], ens["thermal_params"], scen_idx=ens["scen_idx"],
                    e_scale=ens["e_scale"])
    _check(a, ref, keys=("C", "RF", "T", "state"))
    b1 = api.run_ensemble(ens["scen"][:, :40], ens["gas_params"], ens["thermal_params"], scen_idx=ens["scen_idx"],
                          e_scale=ens["e_scale"], chunk_members=384)
    b2 = api.run_ensemble(ens["scen"][:, 40:], ens["gas_params"], ens["thermal_params"], scen_idx=ens["scen_idx"],
                          e_scale=ens["e_scale"], state_in=b1.state, chunk_members=384)
    np.testing.assert_array_equal(np.concatenate([b1.T, b2.T]), a.T)


# ------------------------------------------------------------------ parameter prep kernels
def test_g1g0_and_kq_kernels(api):
    import ctypes
    import torch
    L = _abi.lib()
    rng = np.random.default_rng(5)
    n = 1000
    a = rng.dirichlet(np.ones(4), size=n).T.copy()
    tau = np.exp(rng.uniform(0, 7, size=(4, n)))     # 1..1100 yr: g1's 1-(1+z)e^-z cancels for tau >> h
    a_d, tau_d = to_dev(a), to_dev(tau)      # keep the device arrays alive across the launches
    for mode in (_abi.ALPHA_EXP, _abi.ALPHA_SINH):
        g1 = torch.empty(n, dtype=torch.float64, device="cuda")
        g0 = torch.empty_like(g1)
        _abi.check(L.ufair_g1g0_f64(a_d.data_ptr(), tau_d.data_ptr(), n, n, 100.0, mode,
                                    g1.data_ptr(), g0.data_ptr(), None))
        torch.cuda.synchronize()
        np.testing.assert_allclose(to_np(g1), o.g_1(a, tau), rtol=1e-9)   # 1-(1+z)e^-z cancels for tau >> h
        np.testing.assert_allclose(to_np(g0), o.g_0(a, tau, alpha_mode=mode), rtol=1e-8)
    tcr, ecs = rng.uniform(1, 2.5, n), rng.uniform(2, 5, n)
    d1, d2 = rng.uniform(150, 400, n), rng.uniform(2, 8, n)
    q1 = torch.empty(n, dtype=torch.float64, device="cuda")
    q2 = torch.empty_like(q1)
    ins = [to_dev(x) for x in (tcr, ecs, d1, d2)]
    _abi.check(L.ufair_kq_f64(*(x.data_ptr() for x in ins), 3.74, n, q1.data_ptr(), q2.data_ptr(), None))
    torch.cuda.synchronize()
    r1, r2 = o.k_q(tcr, ecs, d1, d2, 3.74)
    np.testing.assert_allclose(to_np(q1), r1, rtol=1e-12)
    np.testing.assert_allclose(to_np(q2), r2, rtol=1e-12)
    assert ctypes.sizeof(_abi.UfairDesc) > 0


# ------------------------------------------------------------------ error behaviour
def test_python_errors(api):
    ens = ensemble(8, n_t=4)
    with pytest.raises(ValueError):
        _run_dev(api, ens, alpha_mode="bogus")
    with pytest.raises(ValueError):
        _run_dev(api, ens, outputs=("C", "nope"))
    with pytest.raises(ValueError):
        api.run_ensemble(to_dev(ens["E"]), to_dev(ens["gas_params"][:, :5]), to_dev(ens["thermal_params"]))
    with pytest.raises(ValueError):
        api.run_ensemble(to_dev(ens["scen"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]),
                         scen_idx=to_dev(np.full(8, 99, dtype=np.int32)))


# ------------------------------------------------------------------ full-size properties (configs[3] shard)
def test_full_size_shard_properties(api):
    """One GPU's shard of configs[3] is 1.25e6 members x 736 steps.  The oracle cannot finish that in
    seconds, so check size-independent properties: histogram rows each count every member, the
    kernel's histogram equals a recount of its own T on the device, a member block cut out of the
    big launch matches the oracle, and stats-only mode reproduces the same histogram."""
    import torch
    M, n_t = 1_250_048 // 4, 736     # a quarter shard keeps the test's memory and time modest
    g = torch.Generator(device="cuda").manual_seed(1234)
    ens = ensemble(4096, dense=True)
    reps = (M + 4095) // 4096
    tile = lambda x: to_dev(x).repeat(*([1] * (x.ndim - 1)), reps)[..., :M].contiguous()
    gp, tp = tile(ens["gas_params"]), tile(ens["thermal_params"])
    gp[:, _abi.GP_R0] *= 1 + 0.02 * torch.randn(3, M, generator=g, device="cuda", dtype=torch.float64)
    E = tile(ens["E"])
    spec = api.HistSpec()
    res = api.run_ensemble(E, gp, tp, stats=spec)
    torch.cuda.synchronize()
    hist = res.hist
    assert bool((hist.sum(dim=1) == M).all())
    invw = spec.bins / (spec.hi - spec.lo)
    idx = torch.floor((res.T - spec.lo) * invw).clamp_(0, spec.bins - 1).to(torch.int64)
    recount = torch.zeros(n_t, spec.bins, dtype=torch.int64, device="cuda")
    recount.scatter_add_(1, idx, torch.ones_like(idx))
    assert torch.equal(recount, hist)
    sl = slice(777_000 // 4, 777_000 // 4 + 512)
    ref = co.oxfair(to_np(E[:, :, sl]), to_np(gp[:, :, sl]), to_np(tp[:, sl]))
    _check(SimpleNamespace(**{k: getattr(res, k)[..., sl] for k in ("C", "RF", "T")}), ref)
    res2 = api.run_ensemble(E, gp, tp, stats=spec, outputs=(), return_state=False)
    torch.cuda.synchronize()
    assert torch.equal(res2.hist, hist)


def test_config2_full_size_fp64_vs_fp32(api):
    """BASELINE configs[2]: 10^6-member perturbed-parameter ensemble x 4 scenarios, FP64 vs FP32.
    Full size on the device (scenario-shared emissions, T + statistics only); the oracle checks a
    slice, the two precisions are compared with each other everywhere (<= 1e-4 K)."""
    import torch
    M, n_t = 1_000_000, 736
    ens = ensemble(8192, dense=True, seed=42)
    reps = (M + 8191) // 8192
    tile = lambda x: to_dev(x).repeat(*([1] * (x.ndim - 1)), reps)[..., :M].contiguous()
    g = torch.Generator(device="cuda").manual_seed(7)
    gp, tp = tile(ens["gas_params"]), tile(ens["thermal_params"])
    gp[:, _abi.GP_R0] *= 1 + 0.02 * torch.randn(3, M, generator=g, device="cuda", dtype=torch.float64)
    idx = torch.randint(0, 4, (M,), generator=g, device="cuda", dtype=torch.int32)
    esc = 1 + 0.05 * torch.randn(3, M, generator=g, device="cuda", dtype=torch.float64)
    scen = to_dev(ens["scen"])
    kw = dict(scen_idx=idx, e_scale=esc, outputs=("T",), stats=api.HistSpec(), return_state=False)
    r64 = api.run_ensemble(scen, gp, tp, precision="f64", **kw)
    r32 = api.run_ensemble(scen, gp, tp, precision="f32", **kw)
    torch.cuda.synchronize()
    assert bool((r64.hist.sum(dim=1) == M).all()) and bool((r32.hist.sum(dim=1) == M).all())
    assert float((r64.T - r32.T.double()).abs().max()) <= 1e-4
    sl = slice(123_456, 123_456 + 256)
    ref = co.oxfair(ens["scen"], to_np(gp[:, :, sl]), to_np(tp[:, sl]), scen_idx=to_np(idx[sl]), e_scale=to_np(esc[:, sl]))
    assert field_relerr(to_np(r64.T[:, sl]), ref["T"]) < TOL64
    # per-scenario means are ordered like the scenarios' cumulative emissions in 2500
    T_end = r64.T[-1]
    means = [float(T_end[idx == s].mean()) for s in range(4)]
    assert means[1] > means[0] and means[2] > means[0] and means[3] < means[0]


def test_config4_full_size_subannual(api):
    """BASELINE configs[4]: dt = 0.1 yr, 10^6 members x 7360 steps (scenario-shared emissions, T only).
    Size-independent properties: every histogram row counts every member, and two time chunks joined
    through state_out/state_in reproduce the one-shot run bit for bit."""
    import torch
    M, n_t, dt = 1_000_000, 7360, 0.1
    ens = ensemble(4096, n_t=n_t, dt=dt, dense=True, seed=9)
    reps = (M + 4095) // 4096
    tile = lambda x: to_dev(x).repeat(*([1] * (x.ndim - 1)), reps)[..., :M].contiguous()
    gp, tp = tile(ens["gas_params"]), tile(ens["thermal_params"])
    g = torch.Generator(device="cuda").manual_seed(11)
    gp[:, _abi.GP_R0] *= 1 + 0.02 * torch.randn(3, M, generator=g, device="cuda", dtype=torch.float64)
    idx = torch.randint(0, 4, (M,), generator=g, device="cuda", dtype=torch.int32)
    scen = to_dev(ens["scen"])
    spec = api.HistSpec(copies=8)
    one = api.run_ensemble(scen, gp, tp, dt=dt, scen_idx=idx, outputs=("T",), stats=spec)
    torch.cuda.synchronize()
    assert bool((one.hist.sum(dim=1) == M).all())
    T_one_tail = one.T[-64:].clone()
    state_one = one.state.clone()
    del one
    cut = 3333                       # not a multiple of the tile length
    a = api.run_ensemble(scen[:, :cut].contiguous(), gp, tp, dt=dt, scen_idx=idx, outputs=())
    b = api.run_ensemble(scen[:, cut:].contiguous(), gp, tp, dt=dt, scen_idx=idx, outputs=("T",), state_in=a.state)
    torch.cuda.synchronize()
    assert torch.equal(b.T[-64:], T_one_tail) and torch.equal(b.state, state_one)
    sl = slice(500_000, 500_000 + 64)
    ref = co.oxfair(ens["scen"], to_np(gp[:, :, sl]), to_np(tp[:, sl]), dt=dt, scen_idx=to_np(idx[sl]))
    assert field_relerr(to_np(b.T[-64:, sl]), ref["T"][-64:]) < TOL64


def test_host_pipeline_fp32_and_output_reuse(api):
    """FP32 through the host pipeline == FP32 on the device; `out=` reuses the caller's (pinned) buffers."""
    ens = ensemble(3000, n_t=64, dense=True)
    spec = api.HistSpec(copies=5)
    dev = _run_dev(api, ens, precision="f32", stats=spec)
    out = api.pinned_result(3, 64, 3000, stats=spec, precision="f32")
    ws = api.Workspace(0, 1024)
    r1 = api.run_ensemble(ens["E"], ens["gas_params"], ens["thermal_params"], precision="f32", stats=spec,
                          workspace=ws, out=out)
    assert r1 is out and r1.T.dtype == np.float32
    t_ptr = r1.T.ctypes.data
    for k in ("C", "RF", "T", "state"):
        np.testing.assert_array_equal(getattr(r1, k), to_np(getattr(dev, k)))
    np.testing.assert_array_equal(r1.hist, to_np(dev.hist))
    r2 = api.run_ensemble(ens["E"], ens["gas_params"], ens["thermal_params"], precision="f32", stats=spec,
                          workspace=ws, out=out)
    assert r2.T.ctypes.data == t_ptr            # same buffer, refilled
    np.testing.assert_array_equal(r2.T, to_np(dev.T))
    ws.close()


def test_step_is_cuda_graph_capturable(api):
    """reset + integrate + statistics pass + finalize are plain stream work (no allocation, no
    synchronisation, tensor maps passed by value): a whole step can be captured once and replayed."""
    import torch
    ens = ensemble(4000, n_t=64, dense=True, seed=6)
    spec = api.HistSpec(lo=-1.0, hi=3.0, bins=128)
    plan = api.DevicePlan(to_dev(ens["E"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), stats=spec)
    eager = plan.run()
    torch.cuda.synchronize()
    want = {k: getattr(eager, k).clone() for k in ("C", "RF", "T", "hist", "moments", "state")}
    for k in want:
        getattr(eager, k).zero_()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        plan.run()                                  # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        plan.run()
    for _ in range(2):
        for k in want:
            getattr(plan.result, k).zero_()
        graph.replay()
        torch.cuda.synchronize()
        for k, v in want.items():
            assert torch.equal(getattr(plan.result, k), v), k


@pytest.mark.parametrize("dense", [True, False])
@pytest.mark.parametrize("alpha_mode", ["exp", "sinh", "newton", "one"])
def test_plain_variant_is_bitwise_the_general_kernel(api, dense, alpha_mode):
    """Runs with no external forcing, no iIRF ceiling and outputs exactly C + RF + T take a kernel
    instantiation without those run-time switches; asking for alpha as well takes the general one.
    Same arithmetic, so the same bits (and both match the oracle)."""
    import torch
    ens = ensemble(1234, n_t=77, dense=dense, seed=31)
    kw = dict(alpha_mode=alpha_mode, newton_iters=2 if alpha_mode == "newton" else 0)
    plain = _run_dev(api, ens, outputs=("C", "RF", "T"), **kw)
    general = _run_dev(api, ens, outputs=("C", "RF", "T", "alpha"), **kw)
    for k in ("C", "RF", "T", "state"):
        assert torch.equal(getattr(plain, k), getattr(general, k)), k
    t_only = _run_dev(api, ens, outputs=("T",), **kw)       # the output-subset instantiation (default alpha mode)
    rf_only = _run_dev(api, ens, outputs=("RF",), stats=api.HistSpec(), **kw)
    assert torch.equal(t_only.T, general.T) and t_only.C is None and torch.equal(t_only.state, general.state)
    assert torch.equal(rf_only.RF, general.RF) and int(rf_only.hist.sum()) == 1234 * 77
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], **_oracle_kw(kw))
    _check(plain, ref, keys=("C", "RF", "T", "state"))


@pytest.mark.parametrize("dense", [True, False])
@pytest.mark.parametrize("fext", ["shared", "scenario", "member"])
def test_plain_variant_with_external_forcing_is_bitwise_the_general_kernel(api, dense, fext):
    """The production configuration -- external forcing present, everything else plain -- has its own
    instantiation (default alpha mode); asking for alpha as well takes the general kernel."""
    import torch
    M, n_t = 999, 61
    ens = ensemble(M, n_t=n_t, dense=dense, seed=17)
    S = ens["scen"].shape[2]
    if fext == "member":
        fx = ens["f_ext"][:, None] * (1 + 0.01 * np.arange(M))[None, :]
        E, kw, okw = ens["E"], dict(f_ext=to_dev(fx), fext_per_member=True), dict(f_ext=fx, fext_per_member=True)
    elif fext == "scenario":
        fx = np.stack([ens["f_ext"] * (1 + 0.2 * s) for s in range(S)], axis=1)
        E = ens["scen"]
        kw = dict(f_ext=to_dev(fx), scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]))
        okw = dict(f_ext=fx, scen_idx=ens["scen_idx"], e_scale=ens["e_scale"])
    else:
        E, kw, okw = ens["E"], dict(f_ext=to_dev(ens["f_ext"])), dict(f_ext=ens["f_ext"])
    plain = _run_dev(api, ens, E=E, outputs=("C", "RF", "T"), **kw)
    general = _run_dev(api, ens, E=E, outputs=("C", "RF", "T", "alpha"), **kw)
    for k in ("C", "RF", "T", "state"):
        assert torch.equal(getattr(plain, k), getattr(general, k)), k
    ref = co.oxfair(E, ens["gas_params"], ens["thermal_params"], **okw)
    _check(plain, ref, keys=("C", "RF", "T", "state"))


def test_more_than_65535_steps_with_statistics(api):
    """A long sub-annual run: 70 000 steps of dt = 0.01 yr (the step count exceeds a CUDA grid's y / z limit,
    which the statistics pass must not depend on)."""
    import torch
    M, n_t, dt = 64, 70_000, 0.01
    ens = ensemble(M, n_t=n_t, dt=dt, dense=True, gases=("co2",), seed=3)
    spec = api.HistSpec(lo=-1.0, hi=9.0, bins=200, copies=4)
    res = api.run_ensemble(to_dev(ens["E"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), dt=dt, stats=spec)
    torch.cuda.synchronize()
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], dt=dt)
    _check(res, ref, keys=("C", "RF", "T", "state"))
    hist, mom = co.temperature_stats(to_np(res.T), spec.lo, spec.hi, spec.bins)
    assert np.array_equal(to_np(res.hist), hist.astype(np.int64))
    assert np.allclose(to_np(res.moments), mom, rtol=1e-12, atol=1e-12)


def test_host_pipeline_long_run_shrinks_its_chunks(api):
    """Staging memory grows with the step count; for long runs the pipeline cuts the chunk size down
    (8 GB budget) instead of allocating chunk x n_t rows -- same results as the device path."""
    M, n_t, dt = 6000, 12_000, 0.05
    ens = ensemble(M, n_t=n_t, dt=dt, dense=False, gases=("co2", "ch4"), seed=8)
    dev = _run_dev(api, ens, dt=dt, outputs=("C", "RF", "T", "alpha"))
    host = api.run_ensemble(ens["E"], ens["gas_params"], ens["thermal_params"], dt=dt, outputs=("C", "RF", "T", "alpha"))
    for k in ("C", "RF", "T", "alpha", "state"):
        np.testing.assert_array_equal(getattr(host, k), to_np(getattr(dev, k)))


def test_loop_variant_selection(api):
    """Which instantiation of the time loop the dispatcher takes (include/ufair.h UFAIR_LOOP_*)."""
    ens = ensemble(64, n_t=8, dense=True, seed=1)
    mk = lambda **kw: api.DevicePlan(to_dev(ens["E"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), **kw)

    def loop(**kw):
        p = mk(**kw)
        p.kernel_variant()
        return p.loop_variant

    fx = to_dev(ens["f_ext"])
    assert loop() == "plain" and loop(stats=api.HistSpec()) == "plain" and loop(alpha_mode="sinh") == "plain"
    assert loop(f_ext=fx) == "plain_fext" and loop(f_ext=fx, alpha_mode="newton", newton_iters=1) == "general"
    assert loop(iirf_max=97.0) == "general" and loop(outputs=("C", "RF", "T", "alpha")) == "general"
    assert loop(outputs=("T",)) == "plain_subset" and loop(outputs=(), stats=api.HistSpec(), f_ext=fx) == "plain_subset"
    assert loop(outputs=("T",), alpha_mode="sinh") == "general"
    assert loop(conc_driven=True) == "conc_driven" and loop(outputs=("C", "RF", "T", "E")) == "conc_driven"


def test_alpha_saturation_keeps_the_decay_argument_in_its_domain(api):
    """ADVICE r1: with alpha driven to its lower saturation (iIRF hugely negative) and a fast pool,
    x = (dt / tau) / alpha used to run past the range-reduction's 32-bit integer and the pools blew up
    silently.  alpha's floor is now raised per lane so that x stays below 7.6e8: the run stays finite, the
    fast pools simply equilibrate (m = 1), and the concentrations stay pinned near C0."""
    import torch
    ens = ensemble(64, n_t=30, dense=True)
    gp = ens["gas_params"].copy()
    gp[:, _abi.GP_R0] = -5000.0                      # alpha -> exp(-hundreds): saturates
    gp[0, _abi.GP_TAU0 + 3] = 0.002                  # dt / tau = 500
    for mode in ("exp", "newton"):
        res = api.run_ensemble(to_dev(ens["E"]), to_dev(gp), to_dev(ens["thermal_params"]), alpha_mode=mode, newton_iters=3,
                               outputs=("C", "RF", "T", "alpha"))
        torch.cuda.synchronize()
        for k in ("C", "RF", "T", "alpha", "state"):
            assert bool(torch.isfinite(getattr(res, k)).all()), (mode, k)
        if mode == "exp":   # (Newton's safeguarded steps walk alpha back up from the saturated seed)
            al = to_np(res.alpha)
            assert al.max() < 2.0 ** -19 and al.min() > 0.0   # gas 0: floor 2^(ilogb(500) - 28) = 2^-20, mantissa < 2
            C0 = gp[:, _abi.GP_C0][:, None, :]
            assert np.all(np.abs(to_np(res.C) - C0) < 1e-2 * C0)
