"""One statement of what a run's descriptor must satisfy.  The run rules (what the caller asked for) hold for host and
device arrays alike: ufair_run_host_* applies them to the caller's descriptor before it touches the workspace or a
device, with the code and message of ufair_run_* and ufair_kernel_variant.  The placement rules (row pitch, alignment,
the statistics buffers, row offset and T rows of the statistics pass) are for device arrays only: the host pipeline
owns those fields and stages its chunks to satisfy them, as the GPU test at the end shows."""
import ctypes
import os

import numpy as np
import pytest

from fiveeqscm_b200 import _abi

FAKE = 4096  # a 16-byte-aligned address that is never dereferenced
CRT = _abi.OUT_C | _abi.OUT_RF | _abi.OUT_T
STATS = dict(stats=1, hist_bins=8, hist_copies=1, hist_lo=0.0, hist_hi=1.0, hist_t0=0, hist_rows=24)
SPEC = b"stats requested but histogram spec/buffers incomplete"


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_abi.lib_path()):
        import __graft_entry__ as g
        g.build()
    return _abi.lib()


def _desc(**fields):
    d = _abi.UfairDesc(n_gas=3, n_t=24, n_member=1000, ld_member=1000, out_mask=CRT)
    for name in ("emissions", "gas_params", "thermal_params", "out_C", "out_RF", "out_T", "out_alpha", "out_E",
                 "hist_private", "moments_private"):
        setattr(d, name, FAKE)
    for k, v in fields.items():
        setattr(d, k, v)
    return d


def _id(fields):
    """a test id: the fields a case sets, beyond the statistics defaults it builds on"""
    if fields is None:
        return "NULL"
    return ",".join(f"{k}={v}" for k, v in fields.items() if k not in STATS or STATS[k] != v) or "stats"


def _variant(lib, d, elem):
    form, gpl, mw, loop = ctypes.c_uint32(), ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    return lib.ufair_kernel_variant(d, elem, ctypes.byref(form), ctypes.byref(gpl), ctypes.byref(mw), ctypes.byref(loop))


def _calls(lib, d, elem):
    """(rc, message) of every entry point that checks a run of element size elem."""
    p = ctypes.byref(d) if d is not None else None
    run, host = (lib.ufair_run_f64, lib.ufair_run_host_f64) if elem == 8 else (lib.ufair_run_f32, lib.ufair_run_host_f32)
    ws = ctypes.c_void_p(1)   # rejected before the workspace is used
    out = {}
    for name, call in (("run", lambda: run(p, None)), ("variant", lambda: _variant(lib, p, elem)),
                       ("host", lambda: host(ws, p, FAKE, FAKE))):
        rc = call()
        out[name] = (rc, lib.ufair_last_error())
    return out


RUN_FAULTS = [  # (fields, or None for a NULL descriptor; code; message fragment)
    (None, _abi.ERR_ARG, b"descriptor is NULL"),
    (dict(struct_size=8), _abi.ERR_ARG, b"struct_size 8"),
    (dict(n_gas=0), _abi.ERR_ARG, b"n_gas 0 outside"),
    (dict(n_gas=5), _abi.ERR_ARG, b"n_gas 5 outside"),
    (dict(n_t=-1), _abi.ERR_ARG, b"negative n_t"),
    (dict(n_member=-1), _abi.ERR_ARG, b"negative n_t / n_member"),
    (dict(ld_member=999), _abi.ERR_ARG, b"ld_member < n_member"),
    (dict(ld_member=2 ** 31), _abi.ERR_ARG, b"split the member axis"),
    (dict(e_mode=2), _abi.ERR_ARG, b"bad e_mode"),
    (dict(fext_mode=3), _abi.ERR_ARG, b"bad fext_mode"),
    (dict(alpha_mode=7), _abi.ERR_ARG, b"bad alpha_mode"),
    (dict(t_mode=2), _abi.ERR_ARG, b"bad t_mode"),
    (dict(alpha_mode=_abi.ALPHA_NEWTON, newton_iters=9), _abi.ERR_ARG, b"newton_iters 9"),
    (dict(n_scen=0), _abi.ERR_ARG, b"n_scen"),
    (dict(dt=0.0), _abi.ERR_ARG, b"dt and iirf_h"),
    (dict(iirf_h=float("nan")), _abi.ERR_ARG, b"dt and iirf_h"),
    (dict(n_stat_groups=_abi.MAX_STAT_GROUPS + 1, **STATS), _abi.ERR_ARG, b"n_stat_groups"),
    (dict(n_stat_groups=4, **STATS), _abi.ERR_ARG, b"needs stat_group labels"),
    (dict(stat_group=FAKE), _abi.ERR_ARG, b"stat_group set but stats == 0"),
    (dict(out_every=-1), _abi.ERR_ARG, b"out_every -1 < 0"),
    (dict(out_every=5), _abi.ERR_ARG, b"not a multiple of out_every 5"),
    (dict(out_every=4, out_mask=CRT | _abi.OUT_ALPHA), _abi.ERR_UNSUPPORTED, b"per step only"),
    (dict(out_type=2), _abi.ERR_ARG, b"out_type 2"),
    (dict(emissions=None), _abi.ERR_ARG, b"must not be NULL"),
    (dict(gas_params=None), _abi.ERR_ARG, b"must not be NULL"),
    (dict(thermal_params=None), _abi.ERR_ARG, b"must not be NULL"),
    (dict(fext_mode=_abi.FEXT_MEMBER), _abi.ERR_ARG, b"f_ext is NULL"),
    (dict(fext_mode=_abi.FEXT_SCENARIO), _abi.ERR_ARG, b"f_ext is NULL"),
    (dict(out_C=None), _abi.ERR_ARG, b"out_C requested but NULL"),
    (dict(out_RF=None), _abi.ERR_ARG, b"out_RF requested but NULL"),
    (dict(out_T=None), _abi.ERR_ARG, b"out_T requested but NULL"),
    (dict(out_mask=CRT | _abi.OUT_ALPHA, out_alpha=None), _abi.ERR_ARG, b"out_alpha requested but NULL"),
    (dict(out_mask=CRT | _abi.OUT_E, out_E=None), _abi.ERR_ARG, b"out_E requested but NULL"),
    (dict(conc_driven=1 << 5), _abi.ERR_ARG, b"conc_driven 0x20 names a gas"),
    (dict(conc_driven=-1), _abi.ERR_ARG, b"names a gas"),
    (dict(STATS, hist_bins=0), _abi.ERR_ARG, SPEC),
    (dict(STATS, hist_hi=0.0), _abi.ERR_ARG, SPEC),
    (dict(STATS, hist_hi=-1.0), _abi.ERR_ARG, SPEC),
]


@pytest.mark.parametrize("elem", [8, 4])
@pytest.mark.parametrize("fields,rc,msg", RUN_FAULTS, ids=[_id(f) for f, _, _ in RUN_FAULTS])
def test_host_and_device_entry_points_reject_a_bad_run_alike(lib, fields, rc, msg, elem):
    got = _calls(lib, _desc(**fields) if fields is not None else None, elem)
    assert got["run"][0] == rc and msg in got["run"][1], got
    assert got["variant"] == got["run"] and got["host"] == got["run"], got


def test_an_empty_run_is_accepted_without_its_arrays(lib):
    for fields in (dict(n_member=0, ld_member=0), dict(n_t=0)):
        d = _desc(emissions=None, gas_params=None, thermal_params=None, out_C=None, out_RF=None, out_T=None, **fields)
        for elem in (8, 4):
            assert {k: rc for k, (rc, _) in _calls(lib, d, elem).items()} == {"run": 0, "variant": 0, "host": 0}


PLACEMENT_FAULTS = [  # today's code and message of the device entry points
    (dict(ld_member=1001), _abi.ERR_ALIGN, b"ld_member 1001: rows must be a multiple of 16 bytes"),
    (dict(emissions=FAKE + 4), _abi.ERR_ALIGN, b"emissions must be 16-byte aligned"),
    (dict(fext_mode=_abi.FEXT_MEMBER, f_ext=FAKE + 8), _abi.ERR_ALIGN, b"f_ext must be 16-byte aligned"),
    (dict(STATS, hist_copies=0), _abi.ERR_ARG, SPEC),
    (dict(STATS, hist_private=None), _abi.ERR_ARG, SPEC),
    (dict(STATS, moments_private=None), _abi.ERR_ARG, SPEC),
    (dict(STATS, out_mask=_abi.OUT_C, out_T=None), _abi.ERR_ARG, b"stats need out_T (the moments pass reads the T rows)"),
    (dict(STATS, hist_rows=23), _abi.ERR_ARG, b"hist_rows 23 < hist_t0 0 + output rows 24"),
    (dict(STATS, hist_t0=-1), _abi.ERR_ARG, b"hist_rows 24 < hist_t0 -1 + output rows 24"),
]


@pytest.mark.parametrize("fields,rc,msg", PLACEMENT_FAULTS, ids=[_id(f) for f, _, _ in PLACEMENT_FAULTS])
def test_device_entry_points_keep_the_placement_rules(lib, fields, rc, msg):
    d = _desc(**fields)
    p = ctypes.byref(d)
    scratch = form = None
    for name, call in (("run_f64", lambda: lib.ufair_run_f64(p, None)), ("run_f32", lambda: lib.ufair_run_f32(p, None)),
                       ("stats_pass_f64", lambda: lib.ufair_stats_pass_f64(p, None)),
                       ("stats_pass_f32", lambda: lib.ufair_stats_pass_f32(p, None)),
                       ("detect_form_f64", lambda: lib.ufair_detect_form_f64(p, scratch, form, None)),
                       ("variant_f64", lambda: _variant(lib, p, 8)), ("variant_f32", lambda: _variant(lib, p, 4))):
        assert call() == rc, name
        assert lib.ufair_last_error() == msg, (name, lib.ufair_last_error())


def test_statistics_buffer_entry_points_check_the_buffers(lib):
    """ufair_stats_reset / _finalize / _finalize_packed: a spec of bins and rows, and the private buffers the pass
    uses (no histogram range: they never bin)."""
    for fields in (dict(hist_bins=0), dict(hist_rows=0), dict(hist_copies=0), dict(hist_private=None),
                   dict(moments_private=None)):
        p = ctypes.byref(_desc(**dict(STATS, **fields)))
        for name, call in (("reset", lambda: lib.ufair_stats_reset(p, None)),
                           ("finalize", lambda: lib.ufair_stats_finalize(p, FAKE, FAKE, None)),
                           ("finalize_packed", lambda: lib.ufair_stats_finalize_packed(p, FAKE, FAKE, None))):
            assert call() == _abi.ERR_ARG, (fields, name)
            assert b"histogram spec/buffers incomplete" in lib.ufair_last_error(), (fields, name)


@pytest.mark.gpu
def test_host_pipeline_takes_host_arrays_that_break_every_placement_rule():
    """Emissions at an address 4 bytes past 16-byte alignment, an odd row pitch (4020-byte rows), and statistics with
    hist_copies = 0, no private buffers, no hist_rows and no T output: the pipeline owns all of these.  Its T histogram
    and moments are those of the same FP32 run through the device path (sums to summation order)."""
    import torch
    from fiveeqscm_b200 import concentrations as api
    from tests.util import ensemble, to_dev, to_np

    M, n_t, ld, bins = 1003, 21, 1005, 64
    ens = ensemble(M, n_t=n_t, seed=31)
    E, gp, tp = (ens[k].astype(np.float32) for k in ("E", "gas_params", "thermal_params"))
    G = E.shape[0]

    def rows(x, offset=0):
        """x as [rows][ld] float32 rows in a host buffer that starts `offset` elements into its allocation"""
        buf = np.zeros(offset + x.size // M * ld, dtype=np.float32)
        r = buf[offset:].reshape(-1, ld)
        r[:, :M] = x.reshape(-1, M)
        return r

    hE, hgp, htp, hC = rows(E, 1), rows(gp), rows(tp), np.zeros((G * n_t, ld), dtype=np.float32)
    assert hE.ctypes.data % 16 == 4 and ld * 4 % 16 != 0
    d = _abi.UfairDesc(n_gas=G, n_t=n_t, n_member=M, ld_member=ld, out_mask=_abi.OUT_C, stats=1, hist_bins=bins,
                       hist_copies=0, hist_lo=-5.0, hist_hi=25.0, emissions=hE.ctypes.data, gas_params=hgp.ctypes.data,
                       thermal_params=htp.ctypes.data, out_C=hC.ctypes.data)
    hist = np.zeros((n_t, bins), dtype=np.uint64)
    mom = np.zeros((n_t, _abi.MOM_COUNT))
    L = _abi.lib()
    ws = ctypes.c_void_p()
    _abi.check(L.ufair_workspace_create(torch.cuda.current_device(), 384, ctypes.byref(ws)))
    try:
        _abi.check(L.ufair_run_host_f32(ws, ctypes.byref(d), hist.ctypes.data, mom.ctypes.data))
    finally:
        L.ufair_workspace_destroy(ws)

    dev = api.run_ensemble(to_dev(E), to_dev(gp), to_dev(tp), precision="f32", outputs=("C",), return_state=False,
                           gas_form=None, stats=api.HistSpec(lo=-5.0, hi=25.0, bins=bins, copies=3))
    torch.cuda.synchronize()
    assert (hist.sum(axis=1) == M).all()
    assert np.array_equal(hist, to_np(dev.hist).astype(np.uint64))
    dmom = to_np(dev.moments)
    assert np.array_equal(mom[:, 2:], dmom[:, 2:]), "min / max exact"
    np.testing.assert_allclose(mom[:, :2], dmom[:, :2], rtol=1e-12)
    np.testing.assert_allclose(hC[:, :M].reshape(G, n_t, M), to_np(dev.C), rtol=1e-6)
