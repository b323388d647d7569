"""Host-side mirror of the reference's ``U_FaIR/concentrations.py`` call surface, on the B200.

* :func:`calculate_hfc_conc` -- the one function the reference ships
  (reference U_FaIR/concentrations.py:4-5; same name, argument order and ``lifetime=`` keyword
  as its caller uses, reference tests/unit/test_hfcs.py:3,10).  Strict-compat by default:
  ``emissions[0] * exp(-time)``, ``lifetime`` ignored, numpy broadcasting of the operands.
* :func:`run_ensemble` -- the batched 5-equation integrator the reference only names
  (.coveragerc:12-19: step_conc, step_forc, step_temp, g_1, g_0, alpha_val, k_q, oxfair):
  emissions plus gas / thermal parameters in; concentrations, radiative forcing and temperature
  out, with the ensemble-member axis added as the fastest axis.

Everything numeric runs in libufair.so (hand-written sm_100a CUDA).  There is no CPU path: the
functions raise if the library or a CUDA device is missing.  Device (torch.cuda) tensors in ->
device tensors out, on the current stream, no copies; numpy / CPU tensors in -> the C++ host
pipeline (chunked, H2D / kernel / D2H overlapped) and numpy out.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import math
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _abi

_ALPHA = {"exp": _abi.ALPHA_EXP, "sinh": _abi.ALPHA_SINH, "newton": _abi.ALPHA_NEWTON, "one": _abi.ALPHA_ONE}
_TMODE = {"mid": _abi.T_MID, "end": _abi.T_END}
_OUT = {"C": _abi.OUT_C, "RF": _abi.OUT_RF, "T": _abi.OUT_T, "alpha": _abi.OUT_ALPHA, "E": _abi.OUT_E}


def _torch():
    import torch
    return torch


def _require_cuda():
    torch = _torch()
    if not torch.cuda.is_available():
        raise RuntimeError("fiveeqscm_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


@dataclass
class HistSpec:
    """Per-time-step temperature histogram: `bins` equal bins on [lo, hi) (edge bins absorb outliers).

    ``groups`` > 0 builds one histogram and one set of moments per member label (``stat_group=`` of
    :func:`run_ensemble`): results are then [groups][n_t][..].  0 pools every member (results [n_t][..]).
    The private histogram scales with it: copies x groups x n_t x bins x 4 bytes on the device."""
    lo: float = -5.0
    hi: float = 25.0
    bins: int = 1024
    copies: int = 16  # privatised copies the kernel spreads its atomics over
    groups: int = 0   # 0 = pooled; with stat_group="scenario", 0 means one group per scenario

    def lead_shape(self, n_t):
        """Leading axes of every statistics array (results and private copies): [groups][n_t], or [n_t] pooled."""
        return (self.groups, n_t) if self.groups else (n_t,)


@dataclass
class EnsembleResult:
    C: object = None        # [n_gas][n_t][n_member]
    RF: object = None       # [n_gas][n_t][n_member]
    T: object = None        # [n_t][n_member]
    alpha: object = None    # [n_gas][n_t][n_member] (diagnostic)
    E: object = None        # [n_gas][n_t][n_member] emission rates (diagnosed for concentration-driven gases)
    state: object = None    # [5 n_gas + 3][n_member]  -> pass as state_in to continue the run
    hist: object = None     # [n_t][bins] int64 counts (this rank's members); [groups][n_t][bins] when grouped
    moments: object = None  # [n_t][4] float64: sum, sumsq, min, max of T over members; [groups][n_t][4] when grouped
    spec: Optional[HistSpec] = None
    n_member: int = 0
    stat_group: Optional[str] = None  # what the statistics are grouped by: None (pooled), "scenario" or "labels"


# ------------------------------------------------------------------------------------------------
# a1: the reference's function
# ------------------------------------------------------------------------------------------------
def calculate_hfc_conc(emissions, time, lifetime, *, strict=True):
    """Concentration response of a one-box gas (reference U_FaIR/concentrations.py:4-5).

    strict=True (default) reproduces the reference exactly, quirks included: only
    ``emissions[0]`` is read and ``lifetime`` is ignored (unit lifetime), i.e.
    ``emissions[0] * exp(-time)`` with numpy broadcasting, returned as float64.
    strict=False is the physical reading: the whole emission series is integrated with
    e-folding time ``lifetime`` on the (uniform) grid ``time`` through the general integrator,
    and the concentration at the END of each step is returned.
    """
    torch = _require_cuda()
    L = _abi.lib()
    is_torch = isinstance(emissions, torch.Tensor) or isinstance(time, torch.Tensor)
    if strict:
        if is_torch:
            e0 = torch.as_tensor(emissions)[0].to("cuda", torch.float64)
            tt = torch.as_tensor(time).to("cuda", torch.float64)
            e0, tt = torch.broadcast_tensors(e0, tt)
        else:
            e0_np, tt_np = np.broadcast_arrays(np.asarray(emissions)[0], np.asarray(time))
            e0 = torch.from_numpy(np.ascontiguousarray(e0_np, dtype=np.float64)).cuda()
            tt = torch.from_numpy(np.ascontiguousarray(tt_np, dtype=np.float64)).cuda()
        e0 = e0.contiguous()
        tt = tt.contiguous()
        out = torch.empty_like(e0)
        _abi.check(L.ufair_hfc_pulse_f64(e0.data_ptr(), tt.data_ptr(), out.data_ptr(), e0.numel(),
                                         torch.cuda.current_stream().cuda_stream))
        return out if is_torch else out.cpu().numpy()
    # physical opt-in: one gas, one pool, alpha == 1, C0 = 0, c = 1
    e = np.asarray(emissions.cpu() if is_torch else emissions, dtype=np.float64)
    t = np.asarray(time.cpu() if is_torch else time, dtype=np.float64).reshape(-1)
    if e.shape[0] != t.shape[0] or t.shape[0] < 2:
        raise ValueError("strict=False needs emissions and time of equal length >= 2 along axis 0")
    dts = np.diff(t)
    if not np.allclose(dts, dts[0], rtol=1e-12, atol=0):
        raise ValueError("strict=False needs a uniform time grid")
    lead = e.shape[1:]
    e2 = e.reshape(e.shape[0], -1)
    M = e2.shape[1]
    gp = np.zeros((1, _abi.GP_COUNT, M))
    gp[0, _abi.GP_A0] = 1.0
    gp[0, _abi.GP_TAU0:_abi.GP_TAU0 + 4] = np.broadcast_to(np.asarray(lifetime, dtype=np.float64).reshape(-1), (M,))
    gp[0, _abi.GP_EMIS2CONC] = 1.0
    gp[0, _abi.GP_F2] = 1.0
    tp = np.array([0.0, 0.0, 1.0, 1.0])[:, None] * np.ones((4, M))
    res = run_ensemble(e2[None], gp, tp, dt=float(dts[0]), alpha_mode="one", outputs=("C",))
    out = res.C[0].reshape((e.shape[0],) + lead)
    return torch.from_numpy(out).cuda() if is_torch else out


# ------------------------------------------------------------------------------------------------
# the batched integrator
# ------------------------------------------------------------------------------------------------
def _round_up(n, m):
    return (n + m - 1) // m * m


def _build_desc(G, n_t, M, ld, n_scen, e_scen, fext_mode, alpha_mode, newton_iters, t_mode, outputs, dt, iirf_h,
                iirf_max, stats: Optional[HistSpec], gas_form=None, conc_driven=None):
    if alpha_mode not in _ALPHA:
        raise ValueError(f"alpha_mode must be one of {sorted(_ALPHA)}")
    if t_mode not in _TMODE:
        raise ValueError(f"t_mode must be one of {sorted(_TMODE)}")
    mask = 0
    for o in outputs:
        if o not in _OUT:
            raise ValueError(f"unknown output {o!r}; choose from {sorted(_OUT)}")
        mask |= _OUT[o]
    d = _abi.UfairDesc(n_gas=G, n_t=n_t, n_member=M, ld_member=ld, n_scen=n_scen,
                       e_mode=_abi.E_SCENARIO if e_scen else _abi.E_MEMBER, fext_mode=fext_mode,
                       alpha_mode=_ALPHA[alpha_mode], newton_iters=int(newton_iters), t_mode=_TMODE[t_mode],
                       out_mask=mask, stats=1 if stats is not None else 0, dt=float(dt), iirf_h=float(iirf_h),
                       iirf_max=0.0 if iirf_max is None else float(iirf_max))
    if stats is not None:
        d.hist_bins, d.hist_copies = int(stats.bins), int(stats.copies)
        d.hist_lo, d.hist_hi = float(stats.lo), float(stats.hi)
        d.hist_t0, d.hist_rows = 0, n_t
        d.n_stat_groups = int(stats.groups)
    d.conc_driven = _driven_mask(conc_driven, G)
    if gas_form is not None and not isinstance(gas_form, str):
        if len(gas_form) != G:
            raise ValueError("gas_form must have one entry per gas")
        for g, f in enumerate(gas_form):
            d.gas_form[g] = _form_byte(f)
    return d


def _resolve_groups(stats: Optional[HistSpec], stat_group, has_scen_idx: bool, n_scen: int):
    """(HistSpec with ``groups`` settled, source) for ``stat_group=``: source is None (pooled), "scenario" (the
    members' scen_idx, one group per scenario unless ``groups`` says otherwise) or "labels" (an array [M]; its group
    count is never inferred from the data, so that every rank of a multi-GPU run agrees on it)."""
    if stats is not None and not 0 <= int(stats.groups) <= _abi.MAX_STAT_GROUPS:
        raise ValueError(f"HistSpec.groups must be 0..{_abi.MAX_STAT_GROUPS}")
    if stat_group is None:
        if stats is not None and stats.groups:
            raise ValueError("HistSpec.groups > 0 needs stat_group ('scenario' or one label per member)")
        return stats, None
    if stats is None:
        raise ValueError("stat_group needs stats=HistSpec(...)")
    if isinstance(stat_group, str):
        if stat_group != "scenario":
            raise ValueError("stat_group must be None, 'scenario' or one label per member")
        if not has_scen_idx:
            raise ValueError("stat_group='scenario' needs scen_idx")
        groups = int(stats.groups) or int(n_scen)
        if groups > _abi.MAX_STAT_GROUPS:
            raise ValueError(f"{groups} scenario groups: at most {_abi.MAX_STAT_GROUPS}")
        return dataclasses.replace(stats, groups=groups), "scenario"
    if stats.groups < 1:
        raise ValueError("stat_group labels need HistSpec(groups=G), G >= 1 (it is not inferred from the labels)")
    return stats, "labels"


def _check_labels(top: int, groups: int, name: str):
    """The largest label must stay below the group count (negative ones mean "not counted")."""
    if top >= groups:
        raise ValueError(f"{name} has a label {top} >= groups {groups}")


def _driven_mask(conc_driven, G) -> int:
    """None / False -> 0; True -> every gas; else one truth value per gas."""
    if conc_driven is None or conc_driven is False:
        return 0
    if conc_driven is True:
        return (1 << G) - 1
    flags = list(conc_driven)
    if len(flags) != G:
        raise ValueError("conc_driven must be a bool or one flag per gas")
    return sum(1 << g for g, f in enumerate(flags) if f)


def _with_E(outputs, conc_driven):
    """Concentration-driven runs always return the diagnosed emissions."""
    outputs = tuple(outputs)
    if conc_driven is None or isinstance(conc_driven, bool):
        driven = bool(conc_driven)
    else:
        driven = any(bool(f) for f in conc_driven)
    return outputs + ("E",) if driven and "E" not in outputs else outputs


def _any_nonzero(row) -> bool:
    """Is any element of a 1-D array non-zero?  Dense parameter sets answer from the first element; an all-zero
    row costs one pass without a temporary (the comparison ``row != 0`` allocated one per row: 8 ms per call on a
    786 432-member ensemble, on the critical path of every host-pipeline call)."""
    return bool(row.size) and (bool(row[0] != 0) or bool(np.count_nonzero(row)))


def _detect_form_host(gp, state_in):
    """gas_form from HOST parameter arrays: the numpy twin of ufair_detect_form_* (same rule)."""
    out = []
    for g in range(gp.shape[0]):
        used = [_any_nonzero(gp[g, _abi.GP_A0 + q]) or (state_in is not None and _any_nonzero(state_in[5 * g + q]))
                for q in range(1, 4)]
        n_pool = 4 if used[2] else 3 if used[1] else 2 if used[0] else 1
        terms = sum(bit for bit, row in ((_abi.TERM_LOG, _abi.GP_F1), (_abi.TERM_LIN, _abi.GP_F2),
                                         (_abi.TERM_SQRT, _abi.GP_F3)) if _any_nonzero(gp[g, row]))
        out.append(_abi.form(n_pool, terms or _abi.TERM_LIN))
    return out


def auto_chunk_members(n_gas, n_t, *, e_member, fext_member, outputs, return_state=True, state_in=False, e_scale=False,
                       precision="f64") -> int:
    """Members per chunk of the host pipeline when the caller does not say.  What matters is which side of the
    pipeline a member keeps busy longer: the host link (bytes per member up or down at ~50 GB/s) or the integrator
    (~10 ns per member and 1000 gas-steps in FP64, a third of that in FP32).  Link-bound calls -- per-member emissions
    in, trajectories out -- want SMALL chunks (16 384: the fill and drain of the pipeline are one chunk each, and the
    link is busy whatever the kernel's efficiency); kernel-bound calls -- scenario-table inputs, statistics or T
    only out -- want chunks that fill the GPU for several waves (131 072; measured 1.8 / 2.2 / 2.2 / 1.9e10
    member-steps/s at 32 768 / 131 072 / 262 144 / 786 432 on a 786 432-member call)."""
    es = 8 if precision == "f64" else 4
    gt = n_gas * n_t
    up = (gt if e_member else 0) + (n_t if fext_member else 0) + n_gas * _abi.GP_COUNT + _abi.TP_COUNT + \
        (n_gas if e_scale else 0) + (_abi.state_rows(n_gas) if state_in else 0)
    down = sum(math.prod(shape) for _, _, shape, _ in _result_layout(n_gas, n_t, 1, outputs, return_state, None))
    link_ns = max(up, down) * es / 50.0                       # ns per member at 50 GB/s, the busier direction
    kernel_ns = gt * (0.010 if precision == "f64" else 0.0035)   # ns per member: 27 ms / 9 ms per 1.25e6 x 736 x 3 on B200
    return 16384 if link_ns >= kernel_ns else 131072


def _form_byte(f) -> int:
    """One gas_form entry: None / 0 (unspecified), a raw UFAIR_FORM byte, or (n_pool, "log+lin+sqrt")."""
    if f is None:
        return 0
    if isinstance(f, (int, np.integer)):
        if not 0 <= int(f) <= 0x7f or (int(f) & 7) > 4:
            raise ValueError(f"bad gas_form byte {f!r}")
        return int(f)
    n_pool, terms = f
    if not 1 <= int(n_pool) <= 4:
        raise ValueError("gas_form n_pool must be 1..4")
    bits = {"log": _abi.TERM_LOG, "lin": _abi.TERM_LIN, "sqrt": _abi.TERM_SQRT}
    t = 0
    for name in (terms.split("+") if isinstance(terms, str) else terms):
        if name not in bits:
            raise ValueError(f"unknown forcing term {name!r}; choose from {sorted(bits)}")
        t |= bits[name]
    return _abi.form(int(n_pool), t)


def run_ensemble(emissions, gas_params, thermal_params, *, dt=1.0, scen_idx=None, e_scale=None, f_ext=None,
                 fext_per_member=False, state_in=None, alpha_mode="exp", newton_iters=0, iirf_max=None,
                 iirf_h=100.0, t_mode="mid", outputs: Sequence[str] = ("C", "RF", "T"), stats: Optional[HistSpec] = None,
                 precision="f64", return_state=True, chunk_members=None, workspace=None, out=None,
                 gas_form="auto", conc_driven=None, stat_group=None) -> EnsembleResult:
    """Integrate the 5-equation model for an ensemble (oxfair, .coveragerc:19, as one kernel launch).

    emissions      [G][n_t][M] per-member emission RATES, or [G][n_t][S] scenario-shared with
                   ``scen_idx`` [M] int32 (optional per-member multiplier ``e_scale`` [G][M]).
    gas_params     [G][17][M] raw parameters (rows: include/ufair.h UFAIR_GP_*).
    thermal_params [4][M]: q1, q2, d1, d2.
    f_ext          optional external forcing: [n_t] / [n_t][S] (shared) or, with
                   ``fext_per_member=True``, [n_t][M].
    state_in       optional [5G+3][M] state from a previous call's ``.state`` (resume).
    alpha_mode     "exp" | "sinh" | "newton" (``newton_iters`` fixed steps) | "one".
    outputs        any of "C", "RF", "T", "alpha".   stats: HistSpec -> per-step T histogram + moments.
    stat_group     statistics per member group instead of pooled: "scenario" (by ``scen_idx``; one group per
                   scenario unless ``stats.groups`` says otherwise) or labels [M] int with ``stats.groups`` = G:
                   label g in [0, G) counts the member in group g, a negative label leaves it out of the
                   statistics.  ``.hist`` is then [G][n_t][bins] and ``.moments`` [G][n_t][4].
    precision      "f64" (default; <= 1e-10 relative vs the float64 oracle) or "f32" (<= 1e-4 K in T).
    conc_driven    None, True (every gas) or one flag per gas: those gases' ``emissions`` rows are the
                   CONCENTRATION to reach at the end of each step; the emission rate that does so
                   is diagnosed (step_conc inverted exactly) and returned as ``.E`` (all gases).
    gas_form       per-gas specialisation (include/ufair.h UFAIR_FORM): "auto" scans the parameters on
                   the device and lets the library skip pools with a_i == 0 and forcing terms whose
                   coefficient is zero for every member; None = no specialisation; or one entry per gas, e.g.
                   [None, (1, "lin+sqrt"), (1, "lin+sqrt")] -- a promise the caller makes.

    torch.cuda tensors -> results are torch.cuda tensors (current stream, asynchronous);
    numpy / CPU tensors -> chunked host pipeline, results are numpy arrays.  For repeated host
    calls pass ``workspace=Workspace(...)`` (device staging reuse) and ``out=previous_result``
    (host output reuse; allocate those with :func:`pinned_result` for full-speed D2H).
    ``chunk_members`` (host pipeline without a workspace): None picks 16 384 for link-bound calls and
    131 072 for kernel-bound ones (:func:`auto_chunk_members`).
    """
    torch = _require_cuda()
    if precision not in ("f64", "f32"):
        raise ValueError("precision must be 'f64' or 'f32'")
    kw = dict(dt=dt, scen_idx=scen_idx, e_scale=e_scale, f_ext=f_ext, fext_per_member=fext_per_member, state_in=state_in,
              alpha_mode=alpha_mode, newton_iters=newton_iters, iirf_max=iirf_max, iirf_h=iirf_h, t_mode=t_mode,
              outputs=outputs, stats=stats, precision=precision, return_state=return_state, gas_form=gas_form,
              conc_driven=conc_driven, stat_group=stat_group)
    if isinstance(emissions, torch.Tensor) and emissions.is_cuda:
        return DevicePlan(emissions, gas_params, thermal_params, **kw).run()
    return _run_host(emissions, gas_params, thermal_params, chunk_members=chunk_members, workspace=workspace, out=out,
                     **kw)


def _shapes(E_shape, gp_shape, tp_shape, scen_idx, fext_shape, fext_per_member, e_scale_shape=None, state_shape=None):
    if len(E_shape) != 3 or len(gp_shape) != 3 or len(tp_shape) != 2:
        raise ValueError("emissions must be [G][n_t][M|S], gas_params [G][17][M], thermal_params [4][M]")
    G, n_t = E_shape[0], E_shape[1]
    M = gp_shape[2]
    if not (1 <= G <= _abi.MAX_GAS):
        raise ValueError(f"n_gas must be 1..{_abi.MAX_GAS}")
    if gp_shape[0] != G or gp_shape[1] != _abi.GP_COUNT or tuple(tp_shape) != (_abi.TP_COUNT, M):
        raise ValueError("gas_params must be [G][17][M] and thermal_params [4][M]")
    # scenario-shared emissions are explicit: a scen_idx, or a single column every member shares
    e_scen = scen_idx is not None or (E_shape[2] == 1 and M != 1)
    if not e_scen and E_shape[2] != M:
        raise ValueError(f"emissions last axis is {E_shape[2]}: per-member emissions need {M} columns (one per member); "
                         "scenario-shared emissions [G][n_t][S] need scen_idx [M] (or S == 1)")
    n_scen = E_shape[2] if e_scen else 1
    if e_scale_shape is not None:
        if not e_scen:
            raise ValueError("e_scale applies to scenario-shared emissions only")
        if tuple(e_scale_shape) != (G, M):
            raise ValueError(f"e_scale must be [G][M] = ({G}, {M}), got {tuple(e_scale_shape)}")
    if state_shape is not None and tuple(state_shape) != (_abi.state_rows(G), M):
        raise ValueError("state_in must be [5G+3][M]")
    fext_mode = _abi.FEXT_NONE
    if fext_shape is not None:
        if fext_per_member:
            if tuple(fext_shape) != (n_t, M):
                raise ValueError("per-member f_ext must be [n_t][M]")
            fext_mode = _abi.FEXT_MEMBER
        else:
            cols = 1 if len(fext_shape) == 1 else fext_shape[1]
            if fext_shape[0] != n_t:
                raise ValueError("f_ext must have n_t rows")
            if e_scen and cols != n_scen:
                if cols != 1:
                    raise ValueError("shared f_ext must be [n_t] or [n_t][S] with S matching the emissions")
            if not e_scen:
                n_scen = cols
            fext_mode = _abi.FEXT_SCENARIO
    return G, n_t, M, e_scen, n_scen, fext_mode


def _result_layout(n_gas, n_t, M, outputs, return_state, stats: Optional[HistSpec]):
    """(result field, descriptor field, shape, dtype) of every array a run returns.  dtype "real" is the run's
    precision; hist and moments have no descriptor field (ufair_stats_finalize and ufair_run_host_* take them)."""
    layout = [(o, "out_" + o, (n_t, M) if o == "T" else (n_gas, n_t, M), "real") for o in _OUT if o in outputs]
    if return_state:
        layout.append(("state", "state_out", (_abi.state_rows(n_gas), M), "real"))
    if stats is not None:
        lead = stats.lead_shape(n_t)
        layout += [("hist", None, lead + (stats.bins,), "int64"), ("moments", None, lead + (_abi.MOM_COUNT,), "float64")]
    return layout


def _numpy(x):
    return x.detach().cpu().numpy() if isinstance(x, _torch().Tensor) else x


class _DeviceArrays:
    """Places a run's arrays on `device`: tensors of the run dtype; member rows padded to a 16-byte pitch (ld) and
    16-byte aligned, as the integrator's bulk loads need."""

    def __init__(self, torch, device, dtype):
        self.torch, self.device, self.dtype = torch, device, dtype

    def ld(self, M):
        return _round_up(max(M, 1), 16 // self.dtype.itemsize)

    def array(self, x):
        return self.torch.as_tensor(x, device=self.device).to(self.dtype).contiguous()

    def rows(self, x, ld):
        if x.shape[-1] != ld:
            x = self.torch.nn.functional.pad(x, (0, ld - x.shape[-1]))
        return x.clone() if x.data_ptr() % 16 else x

    def labels(self, x):
        return self.torch.as_tensor(x, device=self.device).to(self.torch.int32).contiguous().reshape(-1)

    @staticmethod
    def ptr(x):
        return x.data_ptr()


class _HostArrays:
    """Places a run's arrays for the host pipeline: contiguous numpy arrays of the run dtype, row pitch ld = M."""

    def __init__(self, dtype):
        self.dtype = dtype

    @staticmethod
    def ld(M):
        return M

    def array(self, x):
        return np.ascontiguousarray(_numpy(x), dtype=self.dtype)

    @staticmethod
    def rows(x, ld):
        return x

    @staticmethod
    def labels(x):
        return np.ascontiguousarray(_numpy(x), dtype=np.int32).reshape(-1)

    @staticmethod
    def ptr(x):
        return x.ctypes.data


def _prepare(arrays, E, gp, tp, *, dt=1.0, scen_idx=None, e_scale=None, f_ext=None, fext_per_member=False,
             state_in=None, alpha_mode="exp", newton_iters=0, iirf_max=None, iirf_h=100.0, t_mode="mid",
             outputs=("C", "RF", "T"), stats=None, gas_form="auto", conc_driven=None, stat_group=None):
    """Checks a run's inputs (keywords of :func:`run_ensemble`) and places them with `arrays` (:class:`_DeviceArrays`
    or :class:`_HostArrays`).  Returns (descriptor with every input wired, the placed arrays by descriptor field,
    the outputs with "E" added for concentration-driven runs, the HistSpec with its group count settled, the label
    source of :func:`_resolve_groups`).  ``gas_form="auto"`` is left to the caller: it scans the placed arrays."""
    if isinstance(gas_form, str) and gas_form != "auto":
        raise ValueError("gas_form must be 'auto', None or one entry per gas")
    E, gp, tp, e_scale, f_ext, state_in = (None if x is None else arrays.array(x)
                                           for x in (E, gp, tp, e_scale, f_ext, state_in))
    shape = lambda x: None if x is None else tuple(x.shape)
    G, n_t, M, e_scen, n_scen, fext_mode = _shapes(E.shape, gp.shape, tp.shape, scen_idx, shape(f_ext), fext_per_member,
                                                   shape(e_scale), shape(state_in))
    stats, source = _resolve_groups(stats, stat_group, scen_idx is not None, n_scen)
    outputs = _with_E(outputs, conc_driven)
    ld = arrays.ld(M)
    d = _build_desc(G, n_t, M, ld, n_scen, e_scen, fext_mode, alpha_mode, newton_iters, t_mode, outputs, dt, iirf_h,
                    iirf_max, stats, gas_form, conc_driven)
    placed = dict(emissions=E if e_scen else arrays.rows(E, ld), gas_params=arrays.rows(gp, ld),
                  thermal_params=arrays.rows(tp, ld))
    if scen_idx is not None:
        si = placed["scen_idx"] = arrays.labels(scen_idx)
        if si.shape[0] != M:
            raise ValueError("scen_idx must have one entry per member")
        if M and (int(si.min()) < 0 or int(si.max()) >= n_scen):
            raise ValueError("scen_idx out of range")
    if source is not None:   # "scenario": the labels ARE scen_idx (no copy; they follow in-place updates of it)
        lab = placed["stat_group"] = placed["scen_idx"] if source == "scenario" else arrays.labels(stat_group)
        if lab.shape[0] != M:
            raise ValueError("stat_group must have one label per member")
        if M:
            _check_labels(int(lab.max()), stats.groups, "scen_idx" if source == "scenario" else "stat_group")
    if e_scale is not None:
        placed["e_scale"] = arrays.rows(e_scale, ld)
    if f_ext is not None:
        if fext_per_member:
            f_ext = arrays.rows(f_ext, ld)
        elif math.prod(f_ext.shape) == n_t and n_scen > 1:   # [n_t] -> [n_t][S]: the one column repeated
            f_ext = arrays.array(f_ext.reshape(n_t, 1)[:, [0] * n_scen])
        placed["f_ext"] = f_ext
    if state_in is not None:
        placed["state_in"] = arrays.rows(state_in, ld)
    for field, x in placed.items():
        setattr(d, field, arrays.ptr(x))
    return d, placed, outputs, stats, source


class DevicePlan:
    """A prepared device-resident run: descriptor + buffers.  ``run_ensemble`` on CUDA tensors is
    ``plan = DevicePlan(...); plan.reset_stats(); plan.launch(); plan.finalize_stats()``; callers
    that repeat the same run (benchmarks, time-chunked drivers) keep the plan and re-launch it.
    Keywords are those of :func:`run_ensemble` but the host pipeline's ``chunk_members``, ``workspace`` and ``out``."""

    def __init__(self, E, gp, tp, *, precision="f64", return_state=True, gas_form="auto", **inputs):
        torch = _require_cuda()
        self._L = _abi.lib()
        dtype = torch.float64 if precision == "f64" else torch.float32
        dev = E.device
        d, placed, outputs, stats, source = _prepare(_DeviceArrays(torch, dev, dtype), E, gp, tp, gas_form=gas_form,
                                                     **inputs)
        G, n_t, M, ld = d.n_gas, d.n_t, d.n_member, d.ld_member
        self.device, self.precision, self.stats = dev, precision, stats
        self.n_gas, self.n_t, self.n_member = G, n_t, M
        self.scen_idx = placed.get("scen_idx")   # the plan's own copy: callers that re-launch may overwrite it in place
        self.stat_group = placed.get("stat_group")

        res = EnsembleResult(spec=stats, n_member=M, stat_group=source)
        for name, field, shape, kind in _result_layout(G, n_t, M, outputs, return_state, stats):
            if field is None:
                setattr(res, name, torch.empty(shape, dtype=getattr(torch, kind), device=dev))
                continue
            buf = torch.empty(shape[:-1] + (ld,), dtype=dtype, device=dev)
            setattr(d, field, buf.data_ptr())
            setattr(res, name, buf[..., :M])
        if stats is not None:
            if "T" not in outputs:  # the moments pass reads the T rows: scratch the caller never sees
                self._t_scratch = torch.empty(n_t, ld, dtype=dtype, device=dev)
                d.out_T = self._t_scratch.data_ptr()
            rows = math.prod(stats.lead_shape(n_t))
            self._hp = torch.empty(stats.copies, rows, stats.bins, dtype=torch.int32, device=dev)
            self._mp = torch.empty(stats.copies, rows, _abi.MOM_COUNT, dtype=torch.float64, device=dev)
            d.hist_private, d.moments_private = self._hp.data_ptr(), self._mp.data_ptr()
        keep = list(placed.values())
        res._keep = keep  # inputs stay alive as long as the result does
        self.desc, self.result, self._keep = d, res, keep
        self._run = self._L.ufair_run_f64 if precision == "f64" else self._L.ufair_run_f32
        if isinstance(gas_form, str) and M:  # "auto": one scan (synchronises the current stream once, at plan time)
            scratch = torch.empty(_abi.MAX_GAS, dtype=torch.int32, device=dev)
            form = (C.c_uint8 * _abi.MAX_GAS)()
            detect = self._L.ufair_detect_form_f64 if precision == "f64" else self._L.ufair_detect_form_f32
            with torch.cuda.device(dev):
                _abi.check(detect(C.byref(d), scratch.data_ptr(), form, self._stream()))
            for g in range(G):
                d.gas_form[g] = form[g]
        self.gas_form = tuple(int(d.gas_form[g]) for g in range(G))

    def _stream(self):
        return _torch().cuda.current_stream(self.device).cuda_stream

    def kernel_variant(self):
        """(form, gases_per_lane, members_per_warp) of the integrator variant this plan launches;
        form is one UFAIR_FORM byte per gas, 0 everywhere = the general kernel."""
        f, g, mw, loop = C.c_uint32(), C.c_int32(), C.c_int32(), C.c_int32()
        _abi.check(self._L.ufair_kernel_variant(C.byref(self.desc), 8 if self.precision == "f64" else 4, f, g, mw, loop))
        self.loop_variant = _abi.LOOP_NAMES[loop.value]   # one of _abi.LOOP_NAMES (UFAIR_LOOP_*)
        return tuple((f.value >> (8 * k)) & 0xff for k in range(self.n_gas)), g.value, mw.value

    def reset_stats(self):
        if self.stats is not None:
            _abi.check(self._L.ufair_stats_reset(C.byref(self.desc), self._stream()))

    def launch(self):
        """One launch of the fused integrator on the current stream (asynchronous)."""
        _abi.check(self._run(C.byref(self.desc), self._stream()))

    def stats_pass(self):
        """Statistics pass: histogram and moments of the T rows the integrator just wrote."""
        if self.stats is not None:
            fn = self._L.ufair_stats_pass_f64 if self.precision == "f64" else self._L.ufair_stats_pass_f32
            _abi.check(fn(C.byref(self.desc), self._stream()))

    def finalize_stats(self):
        if self.stats is not None:
            r = self.result
            _abi.check(self._L.ufair_stats_finalize(C.byref(self.desc), r.hist.data_ptr(), r.moments.data_ptr(),
                                                    self._stream()))

    def run(self) -> EnsembleResult:
        with _torch().cuda.device(self.device):
            self.reset_stats()
            self.launch()
            self.stats_pass()
            self.finalize_stats()
        return self.result


class Workspace:
    """Device staging buffers + streams of the host pipeline (reuse across calls to avoid re-allocation)."""

    def __init__(self, device: int = 0, chunk_members: int = 16384):
        self._h = C.c_void_p()
        _abi.check(_abi.lib().ufair_workspace_create(int(device), int(chunk_members), C.byref(self._h)))

    def close(self):
        if self._h:
            _abi.lib().ufair_workspace_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _run_host(E, gp, tp, *, precision="f64", return_state=True, gas_form="auto", chunk_members=None, workspace=None,
              out=None, **inputs):
    torch = _torch()
    npdt = np.float64 if precision == "f64" else np.float32
    d, placed, outputs, stats, source = _prepare(_HostArrays(npdt), E, gp, tp, gas_form=gas_form, **inputs)
    G, n_t, M = d.n_gas, d.n_t, d.n_member
    if isinstance(gas_form, str) and M:
        for g, f in enumerate(_detect_form_host(placed["gas_params"], placed.get("state_in"))):
            d.gas_form[g] = f
    res = out if out is not None else EnsembleResult()
    res.spec, res.n_member, res.stat_group = stats, M, source
    for name, field, shape, kind in _result_layout(G, n_t, M, outputs, return_state, stats):
        cur = getattr(res, name)   # out= reuse: an array of the right shape and dtype is written in place
        if isinstance(cur, torch.Tensor):
            cur = cur.numpy()
        dtype = npdt if kind == "real" else np.dtype(kind)
        if not (isinstance(cur, np.ndarray) and cur.shape == shape and cur.dtype == dtype and cur.flags.c_contiguous):
            cur = np.empty(shape, dtype=dtype)
        setattr(res, name, cur)
        if field is not None:
            setattr(d, field, cur.ctypes.data)
    stat_out = (res.hist.ctypes.data, res.moments.ctypes.data) if stats is not None else (None, None)
    own = workspace is None
    if own and chunk_members is None:
        chunk_members = auto_chunk_members(G, n_t, e_member=d.e_mode == _abi.E_MEMBER,
                                           fext_member=d.fext_mode == _abi.FEXT_MEMBER, outputs=outputs,
                                           return_state=return_state, state_in="state_in" in placed,
                                           e_scale="e_scale" in placed, precision=precision)
    ws = Workspace(torch.cuda.current_device(), chunk_members) if own else workspace
    try:
        L = _abi.lib()
        run = L.ufair_run_host_f64 if precision == "f64" else L.ufair_run_host_f32
        _abi.check(run(ws._h, C.byref(d), *stat_out))
    finally:
        if own:
            ws.close()
    return res


def pinned_result(n_gas, n_t, n_member, outputs=("C", "RF", "T"), stats: Optional[HistSpec] = None, precision="f64",
                  return_state=True) -> EnsembleResult:
    """Page-locked host output buffers for :func:`run_ensemble` ``out=`` (D2H at full PCIe speed).  Grouped
    statistics need ``stats.groups`` set to the group count here (``HistSpec(groups=S)`` for per-scenario ones)."""
    torch = _require_cuda()
    real = torch.float64 if precision == "f64" else torch.float32
    r = EnsembleResult(spec=stats, n_member=n_member)
    for name, _, shape, kind in _result_layout(n_gas, n_t, n_member, outputs, return_state, stats):
        dtype = real if kind == "real" else getattr(torch, kind)
        setattr(r, name, torch.empty(shape, dtype=dtype, pin_memory=True).numpy())
    return r
