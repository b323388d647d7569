"""The parity rule of tests/util.py on a real 4-gas oracle result: a whole-field criterion lets the small slices of
a stacked output drift, the per-gas / per-state-row rule does not."""
import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from oracle import c_oracle as co
from tests.util import FLOOR, TOL64, ensemble, field_relerr, output_relerr, slice_relerr, state_floors

GASES4 = ("co2", "ch4", "n2o", "hfc")


@pytest.fixture(scope="module")
def ref():
    ens = ensemble(500, n_t=300, dense=False, gases=GASES4)
    return co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=ens["f_ext"], want_alpha=True)


def test_the_smallest_slices_sit_far_below_the_field_scale(ref):
    """The premise: HFC's concentration and the temperature rows of the state are orders of magnitude below the
    largest slice of their field, so 1e-10 of the field is much more than 1e-10 of theirs."""
    C, st = ref["C"], ref["state"]
    assert np.abs(C[3]).max() < 1e-2 * np.abs(C).max()
    s1 = 5 * 4
    assert np.abs(st[s1:]).max() < 1e-3 * np.abs(st).max()


def test_a_wrong_small_gas_or_state_row_passes_the_field_rule_and_fails_the_slice_rule(ref):
    C = ref["C"].copy()
    C[3] *= 1 + 1e-8                                  # HFC concentrations off by 1e-8 of their own size
    assert field_relerr(C, ref["C"]) < TOL64
    assert output_relerr("C", C, ref["C"]) > TOL64
    st = ref["state"].copy()
    st[5 * 4] *= 1 + 1e-7                             # S1 off by 1e-7 of its own size
    assert field_relerr(st, ref["state"]) < TOL64
    assert output_relerr("state", st, ref["state"]) > TOL64
    for k in ("C", "RF", "T", "alpha", "state"):      # and the oracle's own result passes
        assert output_relerr(k, ref[k], ref[k]) == 0.0


def test_slice_relerr_and_the_floors():
    ref = np.array([[1e4, -2e4], [1e-3, 2e-3]])
    got = ref + np.array([[1.0, 0.0], [0.0, 1e-9]])
    assert slice_relerr(got, ref) == pytest.approx(max(1.0 / 2e4, 1e-9 / 2e-3))
    assert slice_relerr(got, ref, floor=[0.0, 1.0]) == pytest.approx(1.0 / 2e4)      # the floor bounds the scale below
    assert field_relerr(got, ref) == pytest.approx(1.0 / 2e4)
    rows = _abi.state_rows(4)
    f = state_floors(rows)
    assert f.shape == (rows,) and (f[:20] == 0).all() and (f[20:] == FLOOR["T"]).all()
    # T is judged whole, with its floor; a run of tiny temperatures is measured on the floor
    T = np.full((2, 3), 1e-6)
    assert output_relerr("T", T + 1e-13, T) == pytest.approx(1e-13 / FLOOR["T"])
    assert output_relerr("RF", np.zeros((2, 1, 1)) + 1e-13, np.zeros((2, 1, 1))) == pytest.approx(1e-13 / FLOOR["RF"])
