"""Per-gas specialised kernels (SURVEY.md 8f-1: one-pool gases, the reference's own HFC case
U_FaIR/concentrations.py:4-5, next to four-pool CO2): same results as the general kernel and as the
(always general) CPU oracle, through the C ABI."""
import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import params as P
from oracle import c_oracle as co
from tests.util import assert_parity, ensemble, to_dev, to_np

pytestmark = pytest.mark.gpu

LOG, LIN, SQRT = _abi.TERM_LOG, _abi.TERM_LIN, _abi.TERM_SQRT
GASES4 = ("co2", "ch4", "n2o", "hfc")
DETECTED = {"co2": _abi.form(4, LOG), "ch4": _abi.form(1, SQRT), "n2o": _abi.form(1, SQRT), "hfc": _abi.form(1, LIN)}
KERNEL = {"co2": 0, "ch4": _abi.form(1, LIN | SQRT), "n2o": _abi.form(1, LIN | SQRT), "hfc": _abi.form(1, LIN)}


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    from fiveeqscm_b200 import concentrations as c
    _abi.lib()
    return c


def _plan(api, ens, **kw):
    return api.DevicePlan(to_dev(ens["E"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), **kw)


def _sync():
    import torch
    torch.cuda.synchronize()


@pytest.mark.parametrize("gases", [GASES4[:1], GASES4[:2], GASES4[:3], GASES4, ("hfc",), ("ch4",)], ids="+".join)
def test_detected_form_selects_specialised_kernel_same_bits_as_general(api, gases):
    ens = ensemble(1500, n_t=200, dense=False, gases=gases, seed=5)
    G = len(gases)
    auto = _plan(api, ens, f_ext=to_dev(ens["f_ext"]), outputs=("C", "RF", "T", "alpha"))
    assert auto.gas_form == tuple(DETECTED[g] for g in gases)
    form, gpl, mw = auto.kernel_variant()
    if gases == ("co2",):                      # nothing to skip: the general kernel
        assert form == (0,)
    else:
        assert form == tuple(KERNEL[g] for g in gases) and gpl == G and mw == 32
    dense = _plan(api, ens, f_ext=to_dev(ens["f_ext"]), outputs=("C", "RF", "T", "alpha"), gas_form=None)
    assert dense.gas_form == (0,) * G and dense.kernel_variant()[0] == (0,) * G
    ra, rd = auto.run(), dense.run()
    _sync()
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=ens["f_ext"], want_alpha=True)
    assert_parity(ra, ref, ("C", "RF", "T", "alpha", "state"))
    for k in ("C", "RF", "T", "alpha", "state"):
        assert np.array_equal(to_np(getattr(ra, k)), to_np(getattr(rd, k))), f"{k}: specialised != general bits"


def test_declared_form_and_superset_fallback(api):
    ens = ensemble(333, n_t=64, dense=False, seed=9)
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"])
    # the caller's own declaration, in the tuple spelling
    p = _plan(api, ens, gas_form=[None, (1, "sqrt"), (1, "lin+sqrt")])
    assert p.kernel_variant()[0] == (0, KERNEL["ch4"], KERNEL["n2o"])
    r = p.run(); _sync()
    assert_parity(r, ref)
    # a form no instantiated kernel covers (two pools in CH4) runs on the general kernel
    q = _plan(api, ens, gas_form=[None, (2, "sqrt"), (1, "sqrt")])
    assert q.kernel_variant()[0] == (0, 0, 0)
    r2 = q.run(); _sync()
    assert np.array_equal(to_np(r2.T), to_np(r.T))
    # other alpha modes have no specialised instantiation: general kernel, same oracle parity
    n = _plan(api, ens, alpha_mode="sinh")
    assert n.gas_form[1] == DETECTED["ch4"] and n.kernel_variant()[0] == (0, 0, 0)


def test_dense_parameters_detect_as_general(api):
    ens = ensemble(400, n_t=16, dense=True, seed=2)
    p = _plan(api, ens)
    assert p.gas_form == (_abi.form(4, LOG | LIN | SQRT),) * 3 and p.kernel_variant()[0] == (0, 0, 0)


def test_nonzero_initial_state_in_a_skipped_pool_is_detected(api):
    ens = ensemble(256, n_t=16, dense=False, seed=3)
    st = np.zeros((_abi.state_rows(3), 256))
    st[5 * 1 + 2, 17] = 1.0e-3                       # CH4 pool 3 of one member carries mass
    p = _plan(api, ens, state_in=to_dev(st))
    assert p.gas_form[1] == _abi.form(3, SQRT) and p.kernel_variant()[0] == (0, 0, 0)
    r = p.run(); _sync()
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], state_in=st)
    assert_parity(r, ref, ("C",))


def test_specialised_scenario_emissions_stats_and_resume(api):
    import torch
    M, n_t = 5000, 120
    ens = ensemble(M, n_t=n_t, dense=False, seed=21)
    spec = api.HistSpec(lo=-2.0, hi=8.0, bins=256)
    kw = dict(scen_idx=to_dev(ens["scen_idx"]), e_scale=to_dev(ens["e_scale"]), f_ext=to_dev(ens["f_ext"]))
    run = lambda E, **k: api.run_ensemble(to_dev(E), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), **k)
    full = run(ens["scen"], stats=spec, **kw)
    gen = run(ens["scen"], stats=spec, gas_form=None, **kw)
    torch.cuda.synchronize()
    assert torch.equal(full.hist, gen.hist) and torch.equal(full.T, gen.T) and torch.equal(full.moments, gen.moments)
    ref = co.oxfair(ens["scen"], ens["gas_params"], ens["thermal_params"], scen_idx=ens["scen_idx"],
                    e_scale=ens["e_scale"], f_ext=ens["f_ext"])
    assert_parity(full, ref, ("C", "RF", "T", "state"))
    # two half-length calls chained through the state == one call, bit for bit
    h = n_t // 2
    kw1 = dict(kw, f_ext=to_dev(ens["f_ext"][:h]))
    kw2 = dict(kw, f_ext=to_dev(ens["f_ext"][h:]))
    a = run(ens["scen"][:, :h], **kw1)
    b = run(ens["scen"][:, h:], state_in=a.state, **kw2)
    torch.cuda.synchronize()
    assert torch.equal(torch.cat([a.T, b.T]), full.T) and torch.equal(b.state, full.state)


def test_specialised_fp32_within_1e4_K(api):
    ens = ensemble(4096, dense=False, seed=4)
    p = _plan(api, ens, precision="f32", outputs=("T",))
    assert p.kernel_variant()[0] == (0, KERNEL["ch4"], KERNEL["n2o"])
    r = p.run(); _sync()
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"])
    assert np.max(np.abs(to_np(r.T).astype(np.float64) - ref["T"])) < 1e-4


def test_reference_todo_cases_one_pool_gas(api):
    """The reference's own open test TODOs (tests/unit/test_hfcs.py:15-16): constant emissions and
    a pulse that is not in year zero, for the one-box gas its function models -- against the
    closed forms, on the one-pool kernel."""
    n_t, tau, c = 40, 7.5, 0.3
    gp = np.zeros((1, _abi.GP_COUNT, 2)); gp[0, _abi.GP_A0] = 1.0
    gp[0, _abi.GP_TAU0:_abi.GP_TAU0 + 4] = np.array([tau, 1.0, 1.0, 1.0])[:, None]
    gp[0, _abi.GP_EMIS2CONC], gp[0, _abi.GP_F2] = c, 0.5
    tp = np.array([0.33, 0.41, 239.0, 4.1])[:, None] * np.ones((1, 2))
    E = np.zeros((1, n_t, 2)); E[0, :, 0] = 2.0; E[0, 5, 1] = 10.0      # member 0 constant, member 1 pulse in year 5
    p = api.DevicePlan(to_dev(E), to_dev(gp), to_dev(tp), alpha_mode="exp")
    assert p.kernel_variant()[0] == (_abi.form(1, LIN),)
    # r0 = rU = rT = rA = 0 -> iIRF = 0 -> alpha = g0 (state independent): a fixed-lifetime box
    r = p.run(); _sync()
    ref = co.oxfair(E, gp, tp)
    assert_parity(r, ref, ("C",))
    alpha = float(to_np(api.run_ensemble(to_dev(E), to_dev(gp), to_dev(tp), outputs=("alpha",)).alpha)[0, 0, 0])
    k = np.exp(-1.0 / (alpha * tau))
    t = np.arange(1, n_t + 1)
    const = 2.0 * c * alpha * tau * (1.0 - k ** t)                       # relaxation to E c alpha tau
    pulse = np.where(t >= 6, 10.0 * c * alpha * tau * (1.0 - k) * k ** (t - 6.0), 0.0)
    C = to_np(r.C)[0]
    assert np.allclose(C[:, 0], const, rtol=1e-12, atol=0) and np.allclose(C[:, 1], pulse, rtol=1e-12, atol=1e-300)


@pytest.mark.parametrize("gases,M,n_t", [(GASES4[:3], 1001, 97), (GASES4, 33, 1), (GASES4[:2], 2, 7), (("ch4",), 129, 3)],
                         ids=lambda v: "+".join(v) if isinstance(v, tuple) else str(v))
def test_specialised_ragged_tiles_and_per_member_forcing(api, gases, M, n_t):
    """Odd step counts (a ragged last 2-step tile), ragged member counts (a partial last warp) and the
    2-D tensor-map path of per-member external forcing, all on the specialised kernels."""
    ens = ensemble(M, n_t=n_t, dense=False, gases=gases, seed=M + n_t)
    fx = ens["f_ext"][:, None] * (1 + 0.01 * np.arange(M))[None, :]
    p = _plan(api, ens, f_ext=to_dev(fx), fext_per_member=True, outputs=("C", "RF", "T", "alpha"))
    assert any(p.kernel_variant()[0]) and p.kernel_variant()[2] == 32
    r = p.run(); _sync()
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=fx, fext_per_member=True, want_alpha=True)
    assert_parity(r, ref, ("C", "RF", "T", "alpha", "state"))
    g = _plan(api, ens, f_ext=to_dev(fx), fext_per_member=True, outputs=("C", "RF", "T", "alpha"), gas_form=None).run(); _sync()
    for k in ("C", "RF", "T", "alpha", "state"):
        assert np.array_equal(to_np(getattr(r, k)), to_np(getattr(g, k))), k
