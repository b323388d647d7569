"""ctypes binding of include/ufair.h (libufair.so).

There is no CPU fallback: if the CUDA library is missing, :func:`lib` raises.
"""
from __future__ import annotations

import ctypes as C
import os

ABI_VERSION = 5
MAX_GAS = 4
N_POOL = 4
MAX_STAT_GROUPS = 256

# gas_params rows (include/ufair.h UFAIR_GP_*)
GP_A0, GP_TAU0, GP_R0, GP_RU, GP_RT, GP_RA, GP_C0, GP_EMIS2CONC, GP_F1, GP_F2, GP_F3 = (
    0, 4, 8, 9, 10, 11, 12, 13, 14, 15, 16)
GP_COUNT = 17
TERM_LOG, TERM_LIN, TERM_SQRT = 1, 2, 4


def form(n_pool: int, terms: int) -> int:
    """UFAIR_FORM(n_pool, terms) of include/ufair.h."""
    return (n_pool & 7) | ((terms & 7) << 4)
TP_Q1, TP_Q2, TP_D1, TP_D2 = 0, 1, 2, 3
TP_COUNT = 4

E_MEMBER, E_SCENARIO = 0, 1
FEXT_NONE, FEXT_SCENARIO, FEXT_MEMBER = 0, 1, 2
ALPHA_EXP, ALPHA_SINH, ALPHA_NEWTON, ALPHA_ONE = 0, 1, 2, 3
T_MID, T_END = 0, 1
OUT_C, OUT_RF, OUT_T, OUT_ALPHA, OUT_E = 1, 2, 4, 8, 16
OUTTYPE_RUN, OUTTYPE_F32 = 0, 1
MOM_SUM, MOM_SUMSQ, MOM_MIN, MOM_MAX, MOM_COUNT = 0, 1, 2, 3, 4

OK, ERR_ARG, ERR_ALIGN, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOMEM = 0, -1, -2, -3, -4, -5


def state_rows(n_gas: int) -> int:
    return 5 * n_gas + 3


class UfairDesc(C.Structure):
    """Mirror of `struct ufair_desc` (include/ufair.h); field order and types must match."""
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("out_type", C.c_int32),
        ("n_gas", C.c_int32),
        ("n_t", C.c_int32),
        ("n_member", C.c_int64),
        ("ld_member", C.c_int64),
        ("n_scen", C.c_int32),
        ("e_mode", C.c_int32),
        ("fext_mode", C.c_int32),
        ("alpha_mode", C.c_int32),
        ("newton_iters", C.c_int32),
        ("t_mode", C.c_int32),
        ("out_mask", C.c_int32),
        ("stats", C.c_int32),
        ("dt", C.c_double),
        ("iirf_h", C.c_double),
        ("iirf_max", C.c_double),
        ("emissions", C.c_void_p),
        ("scen_idx", C.c_void_p),
        ("e_scale", C.c_void_p),
        ("f_ext", C.c_void_p),
        ("gas_params", C.c_void_p),
        ("thermal_params", C.c_void_p),
        ("state_in", C.c_void_p),
        ("out_C", C.c_void_p),
        ("out_RF", C.c_void_p),
        ("out_T", C.c_void_p),
        ("out_alpha", C.c_void_p),
        ("state_out", C.c_void_p),
        ("hist_bins", C.c_int32),
        ("hist_copies", C.c_int32),
        ("hist_lo", C.c_double),
        ("hist_hi", C.c_double),
        ("hist_t0", C.c_int32),
        ("hist_rows", C.c_int32),
        ("hist_private", C.c_void_p),
        ("moments_private", C.c_void_p),
        ("gas_form", C.c_uint8 * 4),
        ("conc_driven", C.c_int32),
        ("out_E", C.c_void_p),
        ("n_stat_groups", C.c_int32),
        ("out_every", C.c_int32),
        ("stat_group", C.c_void_p),
    ]

    def __init__(self, **kw):
        super().__init__()
        self.struct_size = C.sizeof(UfairDesc)
        self.n_scen = 1
        self.dt = 1.0
        self.iirf_h = 100.0
        self.iirf_max = 0.0
        for k, v in kw.items():
            setattr(self, k, v)


DIST_FIXED, DIST_LOGNORMAL, DIST_NORMAL = 0, 1, 2
LOOP_NAMES = ("general", "conc_driven", "plain", "plain_fext", "plain_subset", "period_mean")   # UFAIR_LOOP_*


class UfairSampler(C.Structure):
    """Mirror of `struct ufair_sampler` (include/ufair.h)."""
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("n_gas", C.c_int32),
        ("seed", C.c_uint64),
        ("n_scen", C.c_int32),
        ("reserved", C.c_int32),
        ("e_scale_sigma", C.c_double),
        ("gas_base", (C.c_double * GP_COUNT) * MAX_GAS),
        ("gas_sigma", (C.c_double * GP_COUNT) * MAX_GAS),
        ("thermal_base", C.c_double * TP_COUNT),
        ("thermal_sigma", C.c_double * TP_COUNT),
        ("gas_dist", (C.c_uint8 * 24) * MAX_GAS),
        ("thermal_dist", C.c_uint8 * 8),
    ]

    def __init__(self, **kw):
        super().__init__()
        self.struct_size = C.sizeof(UfairSampler)
        self.n_scen = 1
        for k, v in kw.items():
            setattr(self, k, v)


class UfairError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libufair error {code}: {msg}")
        self.code = code


_LIB = None
# UFAIR_LIB selects a tuning variant of the same library (perf experiments); default: the in-tree build
_LIB_PATH = os.environ.get("UFAIR_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libufair.so")

# every symbol include/ufair.h declares, with (restype, argtypes)
_vp, _i32, _i64, _dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
_pd = C.POINTER(C.c_double)
SIGNATURES = {
    "ufair_abi_version": (C.c_int, []),
    "ufair_last_error": (C.c_char_p, []),
    "ufair_block_members": (_i64, []),
    "ufair_run_f64": (C.c_int, [C.POINTER(UfairDesc), _vp]),
    "ufair_run_f32": (C.c_int, [C.POINTER(UfairDesc), _vp]),
    "ufair_detect_form_f64": (C.c_int, [C.POINTER(UfairDesc), _vp, C.POINTER(C.c_uint8), _vp]),
    "ufair_detect_form_f32": (C.c_int, [C.POINTER(UfairDesc), _vp, C.POINTER(C.c_uint8), _vp]),
    "ufair_kernel_variant": (C.c_int, [C.POINTER(UfairDesc), _i32, C.POINTER(C.c_uint32), C.POINTER(_i32),
                                       C.POINTER(_i32), C.POINTER(_i32)]),
    "ufair_stats_reset": (C.c_int, [C.POINTER(UfairDesc), _vp]),
    "ufair_stats_pass_f64": (C.c_int, [C.POINTER(UfairDesc), _vp]),
    "ufair_stats_pass_f32": (C.c_int, [C.POINTER(UfairDesc), _vp]),
    "ufair_stats_finalize": (C.c_int, [C.POINTER(UfairDesc), _vp, _vp, _vp]),
    "ufair_stats_finalize_packed": (C.c_int, [C.POINTER(UfairDesc), _vp, _vp, _vp]),
    "ufair_stats_unpack": (C.c_int, [_vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "ufair_hist_percentiles": (C.c_int, [_vp, _i32, _i32, _dbl, _dbl, _vp, _i32, _vp, _vp]),
    "ufair_g1g0_f64": (C.c_int, [_vp, _vp, _i64, _i64, _dbl, _i32, _vp, _vp, _vp]),
    "ufair_kq_f64": (C.c_int, [_vp, _vp, _vp, _vp, _dbl, _i64, _vp, _vp, _vp]),
    "ufair_hfc_pulse_f64": (C.c_int, [_vp, _vp, _vp, _i64, _vp]),
    "ufair_sample_f64": (C.c_int, [C.POINTER(UfairSampler), _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ufair_sample_f32": (C.c_int, [C.POINTER(UfairSampler), _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ufair_workspace_create": (C.c_int, [C.c_int, _i64, C.POINTER(_vp)]),
    "ufair_workspace_destroy": (C.c_int, [_vp]),
    "ufair_run_host_f64": (C.c_int, [_vp, C.POINTER(UfairDesc), _vp, _vp]),
    "ufair_run_host_f32": (C.c_int, [_vp, C.POINTER(UfairDesc), _vp, _vp]),
    "ufair_link_probe": (C.c_int, [C.c_int, _i64, _i64, _i32, _i32, _pd, _pd]),
    "ufair_math_probe_f64": (C.c_int, [C.c_int, _vp, _vp, _i64, _vp]),
    "ufair_math_probe_f32": (C.c_int, [C.c_int, _vp, _vp, _i64, _vp]),
    "ufair_peak_fp64": (C.c_int, [C.c_int, _pd, _pd, _vp]),
    "ufair_peak_fp32": (C.c_int, [C.c_int, _pd, _pd, _vp]),
    "ufair_peak_mufu": (C.c_int, [C.c_int, _pd, _pd, _vp]),
}


def lib_path() -> str:
    return _LIB_PATH


def lib():
    """Load libufair.so (built in-tree by `make -C fiveeqscm_b200/csrc` / __graft_entry__.build())."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(_LIB_PATH):
            raise ImportError(
                f"{_LIB_PATH} is missing: the CUDA library has not been built "
                "(run `python -c 'import __graft_entry__ as g; g.build()'` or `make -C fiveeqscm_b200/csrc`). "
                "There is no CPU fallback.")
        L = C.CDLL(_LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here = header/library mismatch: loud
            fn.restype = res
            fn.argtypes = args
        v = L.ufair_abi_version()
        if v != ABI_VERSION:
            raise ImportError(f"libufair ABI version {v} != binding {ABI_VERSION}")
        _LIB = L
    return _LIB


def check(code: int) -> None:
    if code != 0:
        msg = lib().ufair_last_error()
        raise UfairError(code, msg.decode() if msg else "?")
