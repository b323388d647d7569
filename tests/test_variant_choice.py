"""Which integrator instantiation a descriptor selects, read through ufair_kernel_variant (no GPU needed).

ufair_kernel_variant validates the descriptor but never touches its arrays, so fake non-NULL addresses stand in
for them.  The report is the same Variant the launch dispatches on."""
import ctypes
import os

import pytest

from fiveeqscm_b200 import _abi

FAKE = 4096  # a 16-byte-aligned address that is never dereferenced
ONE_SQRT, ONE_LIN = _abi.form(1, _abi.TERM_SQRT), _abi.form(1, _abi.TERM_LIN)


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_abi.lib_path()):
        import __graft_entry__ as g
        g.build()
    return _abi.lib()


def _desc(n_gas, n_member, outputs=_abi.OUT_C | _abi.OUT_RF | _abi.OUT_T, alpha_mode=_abi.ALPHA_EXP,
          fext_mode=_abi.FEXT_NONE, gas_form=(), conc_driven=0, iirf_max=0.0):
    d = _abi.UfairDesc(n_gas=n_gas, n_t=16, n_member=n_member, ld_member=-(-n_member // 4) * 4, out_mask=outputs,
                       alpha_mode=alpha_mode, newton_iters=1, fext_mode=fext_mode, conc_driven=conc_driven,
                       iirf_max=iirf_max)
    for name in ("emissions", "gas_params", "thermal_params", "f_ext", "out_C", "out_RF", "out_T", "out_alpha",
                 "out_E"):
        setattr(d, name, FAKE)
    for g, f in enumerate(gas_form):
        d.gas_form[g] = f
    return d


def _variant(lib, elem, d):
    form, gpl, mw, loop = ctypes.c_uint32(), ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    rc = lib.ufair_kernel_variant(ctypes.byref(d), elem, ctypes.byref(form), ctypes.byref(gpl), ctypes.byref(mw),
                                  ctypes.byref(loop))
    assert rc == _abi.OK, lib.ufair_last_error()
    return form.value, gpl.value, mw.value, _abi.LOOP_NAMES[loop.value]


SINH, NEWTON, ONE = _abi.ALPHA_SINH, _abi.ALPHA_NEWTON, _abi.ALPHA_ONE
T_ONLY = _abi.OUT_T
COVERED = (0, ONE_SQRT, ONE_SQRT)          # the instantiated 3-gas form 0x616100 covers it
NOT_COVERED = (0, _abi.form(2, _abi.TERM_SQRT), ONE_SQRT)

# (elem, n_gas, n_member, descriptor fields) -> (form, gases per lane, members per warp, loop)
CASES = [
    # the small-ensemble threshold: FP64, default alpha mode, several gases
    (8, 3, 100_000, {}, (0x0, 1, 10, "plain")),
    (8, 3, 100_001, {}, (0x0, 3, 32, "plain")),
    (8, 2, 1000, {}, (0x0, 1, 16, "plain")),
    (8, 4, 1000, {}, (0x0, 1, 8, "plain")),
    (8, 1, 1000, {}, (0x0, 1, 32, "plain")),
    (4, 3, 1000, {}, (0x0, 3, 32, "plain")),
    (4, 1, 1000, {}, (0x0, 1, 32, "plain")),
    (8, 3, 1000, dict(alpha_mode=SINH), (0x0, 3, 32, "plain")),
    (8, 3, 1000, dict(alpha_mode=ONE), (0x0, 3, 32, "plain")),
    # forms: covering, not covering, outside the EXP mode, ignored by the inverse loop
    (8, 3, 1000, dict(gas_form=COVERED), (0x616100, 3, 32, "plain")),
    (8, 3, 1000, dict(gas_form=COVERED, fext_mode=_abi.FEXT_SCENARIO), (0x616100, 3, 32, "plain_fext")),
    (8, 3, 1000, dict(gas_form=COVERED, outputs=T_ONLY), (0x616100, 3, 32, "plain_subset")),
    (8, 3, 1000, dict(gas_form=COVERED, iirf_max=97.0), (0x616100, 3, 32, "general")),
    (8, 3, 1000, dict(gas_form=COVERED, alpha_mode=SINH), (0x0, 3, 32, "plain")),
    (8, 3, 1000, dict(gas_form=COVERED, conc_driven=1), (0x0, 3, 32, "conc_driven")),
    (8, 3, 1000, dict(gas_form=NOT_COVERED), (0x0, 1, 10, "plain")),
    (4, 3, 1000, dict(gas_form=COVERED), (0x616100, 3, 32, "plain")),
    (8, 1, 1000, dict(gas_form=(ONE_LIN,)), (0x21, 1, 32, "plain")),
    (8, 1, 1000, dict(gas_form=(ONE_SQRT,)), (0x61, 1, 32, "plain")),
    (8, 2, 1000, dict(gas_form=(0, ONE_SQRT)), (0x6100, 2, 32, "plain")),
    (8, 4, 1000, dict(gas_form=(0, ONE_SQRT, ONE_SQRT, ONE_LIN)), (0x21616100, 4, 32, "plain")),
    # every loop, and the loops that exist only in the EXP mode falling back to the general one
    (8, 3, 1000, dict(conc_driven=1), (0x0, 3, 32, "conc_driven")),
    (8, 3, 1000, dict(outputs=_abi.OUT_C | _abi.OUT_RF | _abi.OUT_T | _abi.OUT_E), (0x0, 3, 32, "conc_driven")),
    (8, 3, 1000, dict(alpha_mode=NEWTON, conc_driven=2), (0x0, 3, 32, "conc_driven")),
    (8, 3, 1000, dict(outputs=T_ONLY), (0x0, 1, 10, "plain_subset")),
    (8, 3, 1000, dict(outputs=T_ONLY, alpha_mode=SINH), (0x0, 3, 32, "general")),
    (4, 3, 1000, dict(outputs=T_ONLY), (0x0, 3, 32, "plain_subset")),
    (8, 3, 1000, dict(fext_mode=_abi.FEXT_MEMBER), (0x0, 1, 10, "plain_fext")),
    (8, 3, 1000, dict(fext_mode=_abi.FEXT_SCENARIO, alpha_mode=NEWTON), (0x0, 3, 32, "general")),
    (4, 2, 1000, dict(fext_mode=_abi.FEXT_SCENARIO), (0x0, 2, 32, "plain_fext")),
    (8, 3, 1000, dict(iirf_max=97.0), (0x0, 1, 10, "general")),
    (8, 3, 1000, dict(outputs=_abi.OUT_C | _abi.OUT_RF | _abi.OUT_T | _abi.OUT_ALPHA), (0x0, 1, 10, "general")),
]


@pytest.mark.parametrize("elem,n_gas,n_member,fields,want", CASES)
def test_kernel_variant_choice(lib, elem, n_gas, n_member, fields, want):
    assert _variant(lib, elem, _desc(n_gas, n_member, **fields)) == want
