"""Shared helpers for the GPU parity tests: the oracle is the checker, the CUDA path (through the
C ABI / ctypes binding) is the thing under test."""
import numpy as np

from fiveeqscm_b200 import params as P

TOL64 = 1e-10
# Forcing and temperature of a run that lasts one or two steps from pre-industrial are ~1e-6 W m-2 / K,
# and f1 ln(C / C0) at C = C0 (1 + 1e-7) is ill-conditioned in float64 whoever evaluates it (one
# rounding of the argument is 1e-16 / 1e-7 = 1e-9 of the result; the kernel multiplies by 1/C0 where
# the oracle divides).  The 1e-10 criterion is therefore applied to max(field scale, 0.01 W m-2 or K):
# an absolute 1e-12 W m-2 / K for such runs, the plain relative criterion for every run of normal length.
# The state rows S1, S2 and T_prev are temperatures too and take T's floor (see output_relerr).
FLOOR = {"RF": 1e-2, "T": 1e-2}


def ensemble(M, n_t=736, dt=1.0, seed=20261018, dense=True, gases=P.GASES):
    ens = P.sample_ensemble(M, n_t=n_t, dt=dt, seed=seed, gases=gases, dense_pools=dense)
    ens["E"] = P.member_emissions(ens["scen"], ens["scen_idx"], ens["e_scale"])
    return ens


def field_relerr(got, ref, floor=0.0):
    """max |got - ref| / max |ref|: error relative to the field's own scale (the 1e-10 criterion).
    `floor` bounds the scale from below for fields that can be arbitrarily small (see FLOOR)."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    scale = max(float(np.max(np.abs(ref))) if ref.size else 0.0, floor)
    return float(np.max(np.abs(got - ref)) / (scale if scale > 0 else 1.0))


def slice_relerr(got, ref, floor=0.0):
    """The largest field_relerr over the leading-axis slices: each slice (a gas, a state row) is measured on
    its own scale, so a small slice stacked under a large one is not checked against the large one's scale.
    `floor` is one value for every slice or one per slice."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    floors = np.broadcast_to(np.asarray(floor, dtype=np.float64), ref.shape[:1])
    return max((field_relerr(got[i], ref[i], float(floors[i])) for i in range(ref.shape[0])), default=0.0)


def state_floors(n_rows):
    """Per-row floors of a state [5 G + 3][M]: four pools and cumulative emissions per gas (no floor), then
    S1, S2 and T_prev (T's floor)."""
    return np.array([0.0] * (n_rows - 3) + [FLOOR["T"]] * 3)


def output_relerr(name, got, ref):
    """The parity error of output `name` by the repository's rule: C, RF, alpha and E per gas, the state per
    row, T as a whole; RF, T and the temperature rows of the state with their floor."""
    got, ref = _host(got), np.asarray(ref)
    if name == "T":
        return field_relerr(got, ref, FLOOR["T"])
    if name == "state":
        return slice_relerr(got, ref, state_floors(ref.shape[0]))
    assert name in ("C", "RF", "alpha", "E"), name
    return slice_relerr(got, ref, FLOOR.get(name, 0.0))


def assert_parity(res, ref, keys=("C", "RF", "T"), tol=TOL64, what=""):
    """Every output in `keys` of `res` (attributes: tensors or arrays) within `tol` of `ref[key]` by output_relerr."""
    for k in keys:
        err = output_relerr(k, getattr(res, k), ref[k])
        assert err < tol, f"{what}{k}: relative error {err:.3e} > {tol}"


def _host(x):
    return to_np(x) if hasattr(x, "detach") else np.asarray(x)


def to_dev(x):
    import torch
    return None if x is None else torch.from_numpy(np.ascontiguousarray(x)).cuda()


def to_np(x):
    return None if x is None else x.detach().cpu().numpy()
