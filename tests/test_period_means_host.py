"""Period means (out_every) without a GPU: the library's argument checks and variant report (ufair_kernel_variant
validates a descriptor without touching its arrays), the Python layer's checks and result sizes, and the reference
rule itself."""
import ctypes
import os

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import concentrations as api
from tests.period_mean_ref import period_mean

FAKE = 4096  # a 16-byte-aligned address that is never dereferenced
CRT = _abi.OUT_C | _abi.OUT_RF | _abi.OUT_T


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_abi.lib_path()):
        import __graft_entry__ as g
        g.build()
    return _abi.lib()


def _desc(out_every, n_t=24, outputs=CRT, **fields):
    d = _abi.UfairDesc(n_gas=3, n_t=n_t, n_member=1000, ld_member=1000, out_mask=outputs, out_every=out_every)
    for name in ("emissions", "gas_params", "thermal_params", "out_C", "out_RF", "out_T", "out_alpha", "out_E",
                 "hist_private", "moments_private"):
        setattr(d, name, FAKE)
    for k, v in fields.items():
        setattr(d, k, v)
    return d


def _variant(lib, d, elem=8):
    form, gpl, mw, loop = ctypes.c_uint32(), ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    rc = lib.ufair_kernel_variant(ctypes.byref(d), elem, ctypes.byref(form), ctypes.byref(gpl), ctypes.byref(mw),
                                  ctypes.byref(loop))
    return rc, (form.value, gpl.value, _abi.LOOP_NAMES[loop.value] if rc == _abi.OK else None)


@pytest.mark.parametrize("fields,rc,msg", [
    (dict(out_every=-1), _abi.ERR_ARG, b"out_every -1 < 0"),
    (dict(out_every=5), _abi.ERR_ARG, b"not a multiple of out_every 5"),
    (dict(out_every=4, outputs=CRT | _abi.OUT_ALPHA), _abi.ERR_UNSUPPORTED, b"alpha and emissions outputs"),
    (dict(out_every=4, outputs=CRT | _abi.OUT_E), _abi.ERR_UNSUPPORTED, b"alpha and emissions outputs"),
    (dict(out_every=4, conc_driven=1), _abi.ERR_UNSUPPORTED, b"concentration-driven"),
    # statistics rows count output rows: 24 steps / 4 = 6 rows from hist_t0
    (dict(out_every=4, stats=1, hist_bins=8, hist_copies=1, hist_lo=0.0, hist_hi=1.0, hist_t0=3, hist_rows=8),
     _abi.ERR_ARG, b"hist_rows 8 < hist_t0 3 + output rows 6"),
])
def test_the_library_rejects_what_period_means_do_not_support(lib, fields, rc, msg):
    d = _desc(**fields)
    assert lib.ufair_run_f64(ctypes.byref(d), None) == rc
    assert msg in lib.ufair_last_error(), lib.ufair_last_error()
    assert _variant(lib, d)[0] == rc


def test_period_means_accept_what_they_support(lib):
    # n_out rows of statistics suffice (per-step runs need n_t); every alpha mode; 0 and 1 are the per-step loops
    stats = dict(stats=1, hist_bins=8, hist_copies=1, hist_lo=0.0, hist_hi=1.0, hist_t0=2, hist_rows=8)
    assert _variant(lib, _desc(4, **stats)) == (_abi.OK, (0, 3, "period_mean"))
    assert _variant(lib, _desc(1, **stats))[0] == _abi.ERR_ARG
    for mode in (_abi.ALPHA_EXP, _abi.ALPHA_SINH, _abi.ALPHA_NEWTON, _abi.ALPHA_ONE):
        assert _variant(lib, _desc(24, alpha_mode=mode, iirf_max=90.0)) == (_abi.OK, (0, 3, "period_mean"))
        assert _variant(lib, _desc(2, alpha_mode=mode, fext_mode=_abi.FEXT_MEMBER, f_ext=FAKE))[1][2] == "period_mean"
    assert _variant(lib, _desc(0))[1][2] == "plain" and _variant(lib, _desc(1))[1][2] == "plain"
    assert _variant(lib, _desc(1, outputs=CRT | _abi.OUT_ALPHA))[1][2] == "general"
    # the specialised forms of the default mode, FP64 and FP32
    one_sqrt = _abi.form(1, _abi.TERM_SQRT)
    d = _desc(3)
    d.gas_form[1], d.gas_form[2] = one_sqrt, one_sqrt
    assert _variant(lib, d) == (_abi.OK, (0x616100, 3, "period_mean"))
    assert _variant(lib, d, elem=4) == (_abi.OK, (0x616100, 3, "period_mean"))


def test_python_checks_match_the_library():
    assert api._out_rows(24) == 24 and api._out_rows(24, 0) == 24 and api._out_rows(24, 1) == 24
    assert api._out_rows(24, 4) == 6 and api._out_rows(24, 24) == 1
    for k, kw, match in ((-1, {}, "integer >= 0"), (2.5, {}, "integer >= 0"), (5, {}, "not a multiple"),
                         (4, dict(outputs=("T", "alpha")), "not supported"), (4, dict(outputs=("C", "E")), "not supported"),
                         (4, dict(conc_driven=True), "not supported"), (4, dict(conc_driven=[False, True]), "not supported")):
        with pytest.raises(ValueError, match=match):
            api._out_rows(24, k, **kw)
    assert api._out_rows(24, 4, conc_driven=[False, False]) == 6


def test_result_layout_and_chunk_size_follow_the_output_rows():
    spec = api.HistSpec(bins=16, groups=2)
    layout = {name: shape for name, _, shape, _ in api._result_layout(3, 7360, 5, ("C", "RF", "T"), True, spec, 10)}
    assert layout == {"C": (3, 736, 5), "RF": (3, 736, 5), "T": (736, 5), "state": (18, 5), "hist": (2, 736, 16),
                      "moments": (2, 736, 4)}
    assert api._result_layout(3, 7360, 5, ("T",), False, None, 1) == api._result_layout(3, 7360, 5, ("T",), False, None)
    # scenario-table inputs, T trajectories back: link-bound per step, kernel-bound with annual means of 0.1-yr steps
    kw = dict(e_member=False, fext_member=False, outputs=("T",), e_scale=True)
    assert api.auto_chunk_members(3, 7360, **kw) == 16384
    assert api.auto_chunk_members(3, 7360, out_every=10, **kw) == 131072
    assert api.auto_chunk_members(3, 7360, out_every=1, **kw) == 16384
    # C, RF and T of 3 gases: still link-bound at k = 10 (41 KB back per member against 220 ns of integration)
    assert api.auto_chunk_members(3, 7360, out_every=10, **dict(kw, outputs=("C", "RF", "T"))) == 16384


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_reference_mean_rule(dtype):
    """period_mean is the sequential sum from zero in the rows' precision times (Real)(1.0 / k): checked element by
    element against scalar arithmetic in that precision."""
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((2, 30, 7)) * 10.0 ** rng.integers(-3, 4, (2, 30, 7))).astype(dtype)
    ft = np.dtype(dtype).type
    for k in (2, 3, 10, 30):
        got = period_mean(x, k)
        assert got.dtype == dtype and got.shape == (2, 30 // k, 7)
        for g in range(2):
            for p in range(30 // k):
                for m in range(7):
                    s = ft(0)
                    for t in range(p * k, p * k + k):
                        s = ft(s + x[g, t, m])
                    assert got[g, p, m] == ft(s * ft(1.0 / k))
