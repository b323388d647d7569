"""Concentration-driven gases (SURVEY.md 8f-4, concentrations -> emissions): the kernel against the
oracle's invert_conc, and the round trip emissions -> C -> emissions the domain offers."""
import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from oracle import c_oracle as co
from oracle import ufair_oracle as o
from tests.util import TOL64, assert_parity, ensemble, field_relerr, output_relerr, to_dev, to_np

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    from fiveeqscm_b200 import concentrations as c
    _abi.lib()
    return c


def _dev(api, E, ens, **kw):
    import torch
    r = api.run_ensemble(to_dev(E), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]), **kw)
    torch.cuda.synchronize()
    return r


@pytest.mark.parametrize("n_gas", [1, 2, 3, 4])
@pytest.mark.parametrize("alpha_mode", ["exp", "sinh", "newton", "one"])
def test_round_trip_and_oracle_parity(api, n_gas, alpha_mode):
    gases = ("co2", "ch4", "n2o", "hfc")[:n_gas]
    ens = ensemble(600, n_t=150, dense=True, gases=gases, seed=40 + n_gas)
    kw = dict(alpha_mode=alpha_mode, newton_iters=2 if alpha_mode == "newton" else 0, f_ext=to_dev(ens["f_ext"]))
    fwd = _dev(api, ens["E"], ens, **kw)
    inv = _dev(api, to_np(fwd.C), ens, conc_driven=True, **kw)
    # the round trip: emissions come back, and with them the whole trajectory
    assert output_relerr("E", inv.E, ens["E"]) < TOL64
    assert_parity(inv, {k: to_np(getattr(fwd, k)) for k in ("C", "RF", "T", "state")}, ("C", "RF", "T", "state"))
    # and the diagnosed emissions are the oracle's
    okw = dict(alpha_mode={"exp": o.ALPHA_EXP, "sinh": o.ALPHA_SINH, "newton": o.ALPHA_NEWTON, "one": o.ALPHA_ONE}[alpha_mode],
               newton_iters=kw["newton_iters"], f_ext=ens["f_ext"])
    ref = co.oxfair(to_np(fwd.C), ens["gas_params"], ens["thermal_params"], conc_driven=(1 << n_gas) - 1, **okw)
    assert_parity(inv, ref, ("E", "C", "RF", "T", "state"))


def test_mixed_drive_only_co2_concentration_driven(api):
    ens = ensemble(1000, n_t=200, dense=True, seed=8)
    fwd = _dev(api, ens["E"], ens)
    mixed = np.array(ens["E"])
    mixed[0] = to_np(fwd.C)[0]                                   # CO2 rows: concentrations; CH4, N2O: emissions
    inv = _dev(api, mixed, ens, conc_driven=[True, False, False])
    ref = co.oxfair(mixed, ens["gas_params"], ens["thermal_params"], conc_driven=1)
    assert_parity(inv, ref, ("E",))
    assert output_relerr("E", inv.E, ens["E"]) < TOL64
    assert np.array_equal(to_np(inv.E)[1:], ens["E"][1:])        # emission-driven gases: the input, untouched
    assert output_relerr("T", inv.T, to_np(fwd.T)) < TOL64
    assert_parity(inv, ref, ("C", "RF", "T", "state"))


def test_prescribed_concentration_pathway(api):
    """A pathway that is not the image of any forward run: 1 %/yr CO2 growth from pre-industrial."""
    M, n_t = 257, 140
    ens = ensemble(M, n_t=n_t, dense=False, gases=("co2",), seed=2)
    C0 = ens["gas_params"][0, _abi.GP_C0]
    path = (C0[None, :] * 1.01 ** np.arange(1, n_t + 1)[:, None])[None]
    inv = _dev(api, path, ens, conc_driven=True, outputs=("C", "T"))
    ref = co.oxfair(path, ens["gas_params"], ens["thermal_params"], conc_driven=1)
    assert field_relerr(to_np(inv.C), path) < 1e-13                       # the pathway is met
    assert_parity(inv, ref, ("E", "T"))
    assert float(to_np(inv.E)[0, -1].min()) > 0 and 1.0 < float(np.median(to_np(inv.T)[69])) < 2.5   # TCR-scale warming at doubling


def test_scenario_shared_pathways_host_pipeline_and_fp32(api):
    ens = ensemble(3000, n_t=100, dense=True, seed=12)
    fwd = _dev(api, ens["E"], ens)
    Cn = to_np(fwd.C)
    # host pipeline (numpy in, numpy out), ragged chunks
    host = api.run_ensemble(Cn, ens["gas_params"], ens["thermal_params"], conc_driven=True, chunk_members=1024)
    dev = _dev(api, Cn, ens, conc_driven=True)
    for k in ("E", "C", "T"):
        assert np.array_equal(host.__dict__[k], to_np(getattr(dev, k))), k
    # scenario-shared concentration pathways (4 columns) picked per member
    S = 4
    paths = np.stack([Cn[:, :, s] for s in range(S)], axis=2)
    idx = (np.arange(3000) % S).astype(np.int32)
    sh = _dev(api, paths, ens, scen_idx=to_dev(idx), conc_driven=True)
    ref = co.oxfair(paths, ens["gas_params"], ens["thermal_params"], scen_idx=idx, conc_driven=7)
    assert_parity(sh, ref, ("E", "C", "RF", "T", "state"))
    # FP32 mode: temperature within 1e-4 K of the float64 oracle when driven by the same pathway
    r32 = _dev(api, Cn, ens, conc_driven=True, precision="f32", outputs=("T",))
    ref_all = co.oxfair(Cn, ens["gas_params"], ens["thermal_params"], conc_driven=7)
    assert np.max(np.abs(to_np(r32.T).astype(np.float64) - ref_all["T"])) < 1e-4


def test_inverse_argument_errors(api):
    ens = ensemble(8, n_t=4, seed=1)
    with pytest.raises(ValueError):
        _dev(api, ens["E"], ens, conc_driven=[True, False])          # one flag per gas
    d = _abi.UfairDesc(n_gas=3, n_t=4, n_member=8, ld_member=8, conc_driven=8)
    assert _abi.lib().ufair_run_f64(d, None) == _abi.ERR_ARG          # names gas 3 of 3


def test_full_shard_round_trip(api):
    """BASELINE configs[3], one GPU's shard (1.25e6 members x 736 steps x 3 gases): the oracle cannot
    run that in seconds, the round trip can -- emissions -> concentrations (forward kernel) ->
    emissions (concentration-driven kernel) must return the input, and the temperatures must agree."""
    import torch
    M, n_t = 1_250_000, 736
    ens = ensemble(5000, n_t=n_t, dense=True, seed=77)
    reps = (M + 4999) // 5000
    tile = lambda x: to_dev(x).repeat(*([1] * (x.ndim - 1)), reps)[..., :M].contiguous()
    gp, tp, E = tile(ens["gas_params"]), tile(ens["thermal_params"]), tile(ens["E"])
    g = torch.Generator(device="cuda").manual_seed(99)
    E *= 1 + 0.05 * torch.rand(3, 1, M, generator=g, device="cuda", dtype=torch.float64)   # members differ
    fwd = api.run_ensemble(E, gp, tp, outputs=("C", "T"), return_state=False)
    inv = api.run_ensemble(fwd.C, gp, tp, conc_driven=True, outputs=("T",), return_state=False)
    torch.cuda.synchronize()
    for gas in range(3):
        scale = float(E[gas].abs().max())
        err = float((inv.E[gas] - E[gas]).abs().max()) / scale
        assert err < TOL64, f"gas {gas}: emissions come back with relative error {err:.2e}"
    assert float((inv.T - fwd.T).abs().max()) / float(fwd.T.abs().max()) < TOL64
