"""Memory-safety evidence without compute-sanitizer (closed on this GPU pool): guard-band tests.

Every buffer the library writes -- C, RF, T, alpha, E, the final state, the private histogram / moment
copies, and on the host pipeline the caller's host arrays -- is allocated with one poisoned row before
and after it and poisoned tail columns between n_member and the row pitch.  The ragged cases (member
counts that fill no warp, no TMA box and no chunk evenly; 1-4 gases; specialised forms; the
concentration-driven variant; FP32; a chunk size that does not divide M) run through the C ABI with
pointers into those buffers, and afterwards every guard word must still hold the poison pattern
while every word inside has been written.  Inputs get the same treatment: a read past their end
would pull in the NaN poison and show up in the comparison with the oracle.
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from fiveeqscm_b200 import _abi
from oracle import c_oracle as co
from tests.util import ensemble, output_relerr

pytestmark = pytest.mark.gpu

POISON64 = np.frombuffer(np.array([0x7FF8DEADBEEFCAFE], dtype=np.uint64).tobytes(), dtype=np.float64)[0]
POISON32 = np.frombuffer(np.array([0x7FC0BEEF], dtype=np.uint32).tobytes(), dtype=np.float32)[0]
GASES = {1: ("co2",), 2: ("co2", "ch4"), 3: ("co2", "ch4", "n2o"), 4: ("co2", "ch4", "n2o", "hfc")}


class Guarded:
    """[rows][M] data inside a poisoned [rows + 2][ld] allocation (device tensor or host array)."""

    def __init__(self, rows, M, ld, dtype, device):
        import torch
        self.rows, self.M, self.ld, self.device = rows, M, ld, device
        poison = POISON64 if dtype == np.float64 else POISON32
        full = np.full((rows + 2, ld), poison, dtype=dtype)
        if device:
            self.t = torch.from_numpy(full).cuda()
            self.ptr = self.t.data_ptr() + ld * full.itemsize
        else:
            self.t = torch.from_numpy(full).pin_memory()
            self.ptr = self.t.data_ptr() + ld * full.itemsize
        self.itype = np.uint64 if dtype == np.float64 else np.uint32
        self.pbits = np.array([poison]).view(self.itype)[0]

    def fill(self, data):
        import torch
        src = torch.from_numpy(np.ascontiguousarray(data.reshape(self.rows, self.M)))
        self.t[1:-1, :self.M] = src.cuda() if self.device else src
        return self

    def host(self):
        return self.t.cpu().numpy() if self.device else self.t.numpy()

    def data(self):
        return self.host()[1:-1, :self.M]

    def check(self, name, written=True):
        bits = self.host().view(self.itype)
        assert (bits[0] == self.pbits).all() and (bits[-1] == self.pbits).all(), f"{name}: a guard ROW was overwritten"
        assert (bits[1:-1, self.M:] == self.pbits).all(), f"{name}: tail columns >= n_member were overwritten"
        if written:
            assert not (bits[1:-1, :self.M] == self.pbits).any(), f"{name}: some element inside was never written"


def _desc_and_buffers(ens, M, n_t, G, ld, prec, device, *, outputs, stats, conc_driven=0, fext_member=False,
                      gas_form=None, state_in=None):
    npdt = np.float64 if prec == "f64" else np.float32
    mk = lambda rows: Guarded(rows, M, ld, npdt, device)
    b = {"E": mk(G * n_t).fill(ens["E"].astype(npdt)), "gp": mk(G * _abi.GP_COUNT).fill(ens["gas_params"].astype(npdt)),
         "tp": mk(_abi.TP_COUNT).fill(ens["thermal_params"].astype(npdt))}
    mask = sum(getattr(_abi, "OUT_" + ("ALPHA" if o == "alpha" else o)) for o in outputs)
    d = _abi.UfairDesc(n_gas=G, n_t=n_t, n_member=M, ld_member=ld, n_scen=1, e_mode=_abi.E_MEMBER, out_mask=mask,
                       stats=1 if stats else 0, conc_driven=conc_driven, emissions=b["E"].ptr, gas_params=b["gp"].ptr,
                       thermal_params=b["tp"].ptr)
    if fext_member:
        fx = np.broadcast_to(ens["f_ext"][:, None], (n_t, M)) * (1.0 + 0.01 * np.arange(M))
        b["fx"] = mk(n_t).fill(np.ascontiguousarray(fx).astype(npdt))
        d.f_ext, d.fext_mode = b["fx"].ptr, _abi.FEXT_MEMBER
    if state_in is not None:
        b["sin"] = mk(_abi.state_rows(G)).fill(state_in.astype(npdt))
        d.state_in = b["sin"].ptr
    for o, rows in (("C", G * n_t), ("RF", G * n_t), ("T", n_t), ("alpha", G * n_t), ("E", G * n_t)):
        if o in outputs or (o == "T" and stats):
            b["o" + o] = mk(rows)
            setattr(d, {"C": "out_C", "RF": "out_RF", "T": "out_T", "alpha": "out_alpha", "E": "out_E"}[o], b["o" + o].ptr)
    b["state"] = mk(_abi.state_rows(G))
    d.state_out = b["state"].ptr
    if gas_form is not None:
        for g, f in enumerate(gas_form):
            d.gas_form[g] = f
    return d, b


def _run_device(d, b, prec, stats_spec=None):
    import torch
    L = _abi.lib()
    hp = mp = None
    if stats_spec is not None:
        bins, copies = stats_spec
        d.hist_bins, d.hist_copies, d.hist_lo, d.hist_hi, d.hist_t0, d.hist_rows = bins, copies, -5.0, 25.0, 0, d.n_t
        # private statistics buffers with a poisoned row-block either side
        hp = torch.full((copies + 2, d.n_t, bins), 0x5EADBEEF, dtype=torch.int32, device="cuda")
        mp = torch.full((copies + 2, d.n_t, _abi.MOM_COUNT), float(POISON64), dtype=torch.float64, device="cuda")
        d.hist_private = hp.data_ptr() + d.n_t * bins * 4
        d.moments_private = mp.data_ptr() + d.n_t * _abi.MOM_COUNT * 8
        _abi.check(L.ufair_stats_reset(C.byref(d), None))
    run = L.ufair_run_f64 if prec == "f64" else L.ufair_run_f32
    _abi.check(run(C.byref(d), None))
    if stats_spec is not None:
        sp = L.ufair_stats_pass_f64 if prec == "f64" else L.ufair_stats_pass_f32
        _abi.check(sp(C.byref(d), None))
    torch.cuda.synchronize()
    if stats_spec is not None:
        h = hp.cpu().numpy()
        assert (h[0] == 0x5EADBEEF).all() and (h[-1] == 0x5EADBEEF).all(), "hist_private guard blocks overwritten"
        assert (h[1:-1].sum(axis=(0, 2)) == d.n_member).all(), "every member counted once per step"
        m = mp.cpu().numpy().view(np.uint64)
        pb = np.array([POISON64]).view(np.uint64)[0]
        assert (m[0] == pb).all() and (m[-1] == pb).all(), "moments_private guard blocks overwritten"


CASES = [  # (n_gas, M, ld slack, n_t, precision, extra)
    (3, 1003, 6, 37, "f64", {}),                       # ragged warp, ragged 8-step tile (37 = 4 tiles + 5)
    (3, 1, 2, 9, "f64", {}),                           # one member
    (3, 37, 4, 8, "f64", dict(alpha=True)),            # general loop (alpha output), 3 full + 1 ragged 10-member warp
    (1, 95, 2, 17, "f64", {}),
    (2, 1000, 0, 12, "f64", dict(fext_member=True)),   # per-member forcing through the second TMA map
    (4, 259, 6, 19, "f64", {}),
    (3, 515, 2, 23, "f64", dict(sparse=True)),         # specialised per-gas forms (32 members per warp)
    (3, 333, 2, 16, "f64", dict(inverse=True)),        # concentration-driven variant + emissions output
    (3, 1003, 4, 37, "f32", {}),
    (4, 70, 4, 11, "f32", dict(sparse=True)),
]


@pytest.mark.parametrize("G,M,slack,n_t,prec,extra", CASES, ids=lambda v: str(v).replace(" ", ""))
def test_device_outputs_stay_inside_their_rows(G, M, slack, n_t, prec, extra):
    es = 8 if prec == "f64" else 4
    q = 16 // es
    ld = (M + q - 1) // q * q + slack // q * q
    ens = ensemble(M, n_t=n_t, gases=GASES[G], dense=not extra.get("sparse"), seed=7 + M)
    outputs = ("C", "RF", "T") + (("alpha",) if extra.get("alpha") else ()) + (("E",) if extra.get("inverse") else ())
    form = None
    if extra.get("sparse"):
        from fiveeqscm_b200.concentrations import _detect_form_host
        form = _detect_form_host(ens["gas_params"], None)
    kw = {}
    if extra.get("inverse"):   # drive gas 0 by the concentrations an emission-driven run produces
        fwd = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"])
        ens = dict(ens, E=np.concatenate([fwd["C"][:1], ens["E"][1:]]))
        kw["conc_driven"] = 1
    d, b = _desc_and_buffers(ens, M, n_t, G, ld, prec, True, outputs=outputs, stats=True,
                             fext_member=bool(extra.get("fext_member")), gas_form=form, **kw)
    _run_device(d, b, prec, stats_spec=(64, 3))
    for name, buf in b.items():
        buf.check(name, written=name.startswith("o") or name == "state")
    # the run is also right (a read past an input row would have pulled the NaN poison in)
    fx = None
    if extra.get("fext_member"):
        fx = b["fx"].data().astype(np.float64)
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"], f_ext=fx, fext_per_member=fx is not None,
                    conc_driven=kw.get("conc_driven", 0), want_alpha=True)
    T = b["oT"].data().astype(np.float64)
    if prec == "f64":
        for k in outputs:
            assert output_relerr(k, b["o" + k].data().reshape(ref[k].shape), ref[k]) < 1e-10, k
        assert output_relerr("state", b["state"].data(), ref["state"]) < 1e-10
    else:
        assert np.max(np.abs(T - ref["T"])) < 1e-4


def test_resume_state_buffers_are_guarded_too():
    G, M, n_t, ld = 3, 77, 10, 80
    ens = ensemble(M, n_t=n_t, seed=3)
    d1, b1 = _desc_and_buffers(ens, M, n_t, G, ld, "f64", True, outputs=("T",), stats=False)
    _run_device(d1, b1, "f64")
    b1["state"].check("state_out")
    st = b1["state"].data()
    d2, b2 = _desc_and_buffers(ens, M, n_t, G, ld, "f64", True, outputs=("C", "RF", "T"), stats=False, state_in=st)
    _run_device(d2, b2, "f64")
    for name, buf in b2.items():
        buf.check(name, written=name.startswith("o") or name == "state")


@pytest.mark.parametrize("prec", ["f64", "f32"])
def test_host_pipeline_with_a_chunk_that_does_not_divide_M(prec):
    """ufair_run_host_*: chunks of 384 members over 1003 (2 full chunks + 235), host arrays with a row
    pitch larger than M: every D2H copy must land inside its row, in the right columns."""
    import torch
    G, M, n_t, ld = 3, 1003, 21, 1010
    ens = ensemble(M, n_t=n_t, seed=21)
    d, b = _desc_and_buffers(ens, M, n_t, G, ld, prec, False, outputs=("C", "RF", "T"), stats=True)
    d.hist_bins, d.hist_copies, d.hist_lo, d.hist_hi = 64, 2, -5.0, 25.0
    hist = np.full((n_t + 2, 64), -7, dtype=np.int64)
    mom = np.full((n_t + 2, 4), float(POISON64))
    ws = C.c_void_p()
    L = _abi.lib()
    _abi.check(L.ufair_workspace_create(torch.cuda.current_device(), 384, C.byref(ws)))
    try:
        run = L.ufair_run_host_f64 if prec == "f64" else L.ufair_run_host_f32
        _abi.check(run(ws, C.byref(d), hist[1:].ctypes.data, mom[1:].ctypes.data))
    finally:
        L.ufair_workspace_destroy(ws)
    for name, buf in b.items():
        buf.check(name, written=name.startswith("o") or name == "state")
    assert (hist[0] == -7).all() and (hist[-1] == -7).all() and (hist[1:-1].sum(axis=1) == M).all()
    ref = co.oxfair(ens["E"], ens["gas_params"], ens["thermal_params"])
    T = b["oT"].data().astype(np.float64)
    if prec == "f64":
        assert output_relerr("T", T, ref["T"]) < 1e-10
        for k in ("C", "RF"):
            assert output_relerr(k, b["o" + k].data().reshape(G, n_t, M), ref[k]) < 1e-10, k
        assert output_relerr("state", b["state"].data(), ref["state"]) < 1e-10
    else:
        assert np.max(np.abs(T - ref["T"])) < 1e-4


# ------------------------------------------------------------------ the checked build (libufair_dbg.so)
_DBG = os.path.join(os.path.dirname(_abi.lib_path()), "libufair_dbg.so")
_TRIP = """
import numpy as np, torch
from fiveeqscm_b200 import concentrations as api
from tests.util import ensemble, to_dev
ens = ensemble(70, n_t=9)
res = api.run_ensemble(to_dev(ens["E"]), to_dev(ens["gas_params"]), to_dev(ens["thermal_params"]))
torch.cuda.synchronize()
print("completed")
"""


@pytest.mark.skipif(not os.path.exists(_DBG), reason="libufair_dbg.so not built (make -C fiveeqscm_b200/csrc debug)")
def test_debug_bounds_build_never_traps_and_its_checks_are_live():
    """The same library compiled with -DUFAIR_DEBUG_BOUNDS traps on any output store outside its array
    (or in a column >= n_member) and on any read of the shared-memory emission / forcing rings outside
    the box the TMA delivered.  The ragged cases of this file and of the parity suite run on it in a
    subprocess (a trap poisons the CUDA context) and must pass; then the negative control: with
    UFAIR_DEBUG_TRIP=1 the store check pretends the last row of every array is missing, and the very
    same run must fail with the check's error -- so the checks are really compiled in and reached.  The
    control counts the stores it finds in the cut rows instead of trapping, so it never faults the device."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, UFAIR_LIB=_DBG, PYTHONPATH=root)
    env.pop("UFAIR_DEBUG_TRIP", None)
    sel = ["tests/test_gpu_guard.py", "tests/test_gpu_parity.py::test_ragged_member_counts",
           "tests/test_gpu_parity.py::test_modes_and_gas_counts", "tests/test_gpu_parity.py::test_scenario_shared_emissions_and_forcing",
           "tests/test_gpu_parity.py::test_subannual_timestep", "tests/test_gpu_inverse.py", "tests/test_gpu_forms.py"]
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-k", "not debug_bounds", "-p", "no:cacheprovider"] + sel,
                       cwd=root, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    ok = subprocess.run([sys.executable, "-c", _TRIP], cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert ok.returncode == 0 and "completed" in ok.stdout, ok.stderr[-2000:]
    trip = subprocess.run([sys.executable, "-c", _TRIP], cwd=root, env=dict(env, UFAIR_DEBUG_TRIP="1"), capture_output=True,
                          text=True, timeout=600)
    assert trip.returncode != 0 and "completed" not in trip.stdout
    assert "debug bounds check" in trip.stderr and "output stores in the last 1 row(s)" in trip.stderr, trip.stderr[-2000:]
