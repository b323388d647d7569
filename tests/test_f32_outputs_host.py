"""Float32 outputs (out_type / ``out_dtype``) without a GPU: the descriptor field, the library's argument checks and
variant report (ufair_kernel_variant validates a descriptor without touching its arrays), and the Python layer's
checks, result layout and chunk size."""
import ctypes
import os

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from fiveeqscm_b200 import concentrations as api

FAKE = 4096  # a 16-byte-aligned address that is never dereferenced
CRT = _abi.OUT_C | _abi.OUT_RF | _abi.OUT_T
F32 = _abi.OUTTYPE_F32


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_abi.lib_path()):
        import __graft_entry__ as g
        g.build()
    return _abi.lib()


def _desc(out_type=F32, outputs=CRT, n_member=1000, **fields):
    d = _abi.UfairDesc(n_gas=3, n_t=24, n_member=n_member, ld_member=n_member, out_mask=outputs, out_type=out_type)
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


def test_descriptor_field_replaces_the_padding_word():
    assert _abi.ABI_VERSION == 5 and (_abi.OUTTYPE_RUN, _abi.OUTTYPE_F32) == (0, 1)
    assert _abi.UfairDesc.out_type.offset == 4 and _abi.UfairDesc.out_type.size == 4
    assert _abi.UfairDesc.n_gas.offset == 8
    assert _abi.UfairDesc().out_type == _abi.OUTTYPE_RUN   # the default: outputs in the run's precision
    assert _abi.UfairDesc(out_type=-1).out_type == -1      # signed, as the header declares it
    d = api._build_desc(3, 10, 5, 6, 1, False, 0, "exp", 0, "mid", ("T",), 1.0, 100.0, None, None, out_kind="float32")
    assert d.out_type == F32
    d = api._build_desc(3, 10, 5, 6, 1, False, 0, "exp", 0, "mid", ("T",), 1.0, 100.0, None, None)
    assert d.out_type == _abi.OUTTYPE_RUN


@pytest.mark.parametrize("fields,rc,msg", [
    (dict(out_type=2), _abi.ERR_ARG, b"out_type 2 is not"),
    (dict(out_type=-1), _abi.ERR_ARG, b"out_type -1 is not"),
    (dict(outputs=CRT | _abi.OUT_ALPHA), _abi.ERR_UNSUPPORTED, b"alpha and emissions outputs"),
    (dict(outputs=CRT | _abi.OUT_E), _abi.ERR_UNSUPPORTED, b"alpha and emissions outputs"),
    (dict(conc_driven=4), _abi.ERR_UNSUPPORTED, b"concentration-driven"),
])
def test_the_library_rejects_what_f32_outputs_do_not_support(lib, fields, rc, msg):
    d = _desc(**fields)
    assert lib.ufair_run_f64(ctypes.byref(d), None) == rc
    assert msg in lib.ufair_last_error(), lib.ufair_last_error()
    assert _variant(lib, d)[0] == rc
    assert lib.ufair_stats_pass_f64(ctypes.byref(d), None) == rc
    if fields.get("out_type", F32) != F32:   # an unknown type is an error in either precision
        assert _variant(lib, d, elem=4)[0] == rc
        assert lib.ufair_run_f32(ctypes.byref(d), None) == rc


def test_f32_runs_accept_f32_outputs_as_their_own(lib):
    for fields in (dict(), dict(outputs=CRT | _abi.OUT_ALPHA), dict(conc_driven=1, outputs=CRT | _abi.OUT_E)):
        assert _variant(lib, _desc(**fields), elem=4)[0] == _abi.OK, fields
        assert _variant(lib, _desc(**fields), elem=4)[1] == _variant(lib, _desc(out_type=0, **fields), elem=4)[1]


def test_variant_report(lib):
    # every loop but the inverse one; all gases per lane on both sides of UFAIR_SMALL_ENSEMBLE (100 000 members)
    for n_member in (1000, 100_000, 100_032):
        assert _variant(lib, _desc(n_member=n_member)) == (_abi.OK, (0, 3, "plain"))
        assert _variant(lib, _desc(out_type=0, n_member=n_member))[1][1] == (1 if n_member <= 100_000 else 3)
    for fields, loop in ((dict(iirf_max=50.0), "general"), (dict(fext_mode=_abi.FEXT_SCENARIO, f_ext=FAKE), "plain_fext"),
                         (dict(outputs=_abi.OUT_T), "plain_subset"), (dict(out_every=4), "period_mean")):
        assert _variant(lib, _desc(**fields)) == (_abi.OK, (0, 3, loop)), fields
    for mode in (_abi.ALPHA_SINH, _abi.ALPHA_NEWTON, _abi.ALPHA_ONE):   # the loops those modes have
        assert _variant(lib, _desc(alpha_mode=mode, outputs=_abi.OUT_T))[1][2] == "general"
        assert _variant(lib, _desc(alpha_mode=mode, out_every=2))[1][2] == "period_mean"
    one_sqrt = _abi.form(1, _abi.TERM_SQRT)
    d = _desc(n_member=500)
    d.gas_form[1], d.gas_form[2] = one_sqrt, one_sqrt
    assert _variant(lib, d) == (_abi.OK, (0x616100, 3, "plain"))


def test_python_checks_match_the_library():
    assert api._out_kind() == "real" and api._out_kind("f64", "f64") == "real" and api._out_kind("f32", "f32") == "real"
    assert api._out_kind("f64", "f32") == "float32"
    assert api._out_kind("f32", "f32", outputs=("C", "alpha"), conc_driven=True) == "real"   # FP32 run: nothing changes
    assert api._out_kind("f64", "f32", conc_driven=[False, False]) == "float32"
    for args, kw, match in ((("f64", "f16"), {}, "out_dtype must be"), (("f64", np.float32), {}, "out_dtype must be"),
                            (("f32", "f64"), {}, "never wider"),
                            (("f64", "f32"), dict(outputs=("T", "alpha")), "not supported"),
                            (("f64", "f32"), dict(outputs=("C", "E")), "not supported"),
                            (("f64", "f32"), dict(conc_driven=True), "not supported"),
                            (("f64", "f32"), dict(conc_driven=[False, True]), "not supported")):
        with pytest.raises(ValueError, match=match):
            api._out_kind(*args, **kw)


def test_prepare_sets_the_descriptor_field_from_run_keywords():
    from fiveeqscm_b200 import params as P
    G, n_t, M = 3, 6, 9
    E = np.random.default_rng(0).random((G, n_t, M))
    gp, tp = P.default_params(M)
    prep = lambda **kw: api._prepare(api._HostArrays(np.float64), E, gp, tp, **kw)[0]
    assert prep(out_dtype="f32").out_type == F32 and prep().out_type == _abi.OUTTYPE_RUN
    assert prep(precision="f32", out_dtype="f32").out_type == _abi.OUTTYPE_RUN
    assert api._desc_out_kind(prep(out_dtype="f32")) == "float32"
    with pytest.raises(ValueError, match="not supported"):
        prep(out_dtype="f32", conc_driven=True)
    with pytest.raises(ValueError, match="not supported"):
        prep(out_dtype="f32", outputs=("T", "alpha"))


def test_result_layout_keeps_the_state_in_the_run_precision():
    spec = api.HistSpec(bins=16)
    layout = {name: (shape, kind) for name, _, shape, kind in
              api._result_layout(3, 20, 5, ("C", "RF", "T"), True, spec, 4, "float32")}
    assert layout == {"C": ((3, 5, 5), "float32"), "RF": ((3, 5, 5), "float32"), "T": ((5, 5), "float32"),
                      "state": ((18, 5), "real"), "hist": ((5, 16), "int64"), "moments": ((5, 4), "float64")}
    assert api._result_layout(3, 20, 5, ("T",), True, None) == api._result_layout(3, 20, 5, ("T",), True, None, 1, "real")


def test_chunk_size_counts_four_bytes_per_output_element():
    # scenario inputs, T of 4-step means back: 2 bytes of T per member-step in FP64 (link-bound against ~0.03 ns of
    # integration per member-step), 1 in float32 (kernel-bound)
    kw = dict(e_member=False, fext_member=False, outputs=("T",), e_scale=True, return_state=False, out_every=4)
    assert api.auto_chunk_members(3, 7360, **kw) == 16384
    assert api.auto_chunk_members(3, 7360, out_dtype="f32", **kw) == 131072
    assert api.auto_chunk_members(3, 7360, out_dtype="f64", **kw) == 16384
    assert api.auto_chunk_members(3, 7360, precision="f32", out_dtype="f32", **kw) == \
        api.auto_chunk_members(3, 7360, precision="f32", **kw)
