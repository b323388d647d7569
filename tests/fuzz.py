"""Seeded random configurations checked against the C oracle: every combination of gas count,
member / step counts (ragged tiles and warps), emission layout, external-forcing layout, alpha mode,
clamp, temperature mode, resume state, concentration-driven gases, sparse or dense parameters
(specialised or general kernel) that the dedicated tests only sample by hand.  Shared by the GPU
tests (the CUDA path, FP64 and FP32) and a CPU test (the numpy oracle through the same harness)."""
import os

import numpy as np

from oracle import c_oracle as co
from oracle import ufair_oracle as o
from tests.util import TOL64, ensemble, output_relerr, slice_relerr

TOL32_T = 1e-4       # FP32: K, absolute, against the float64 oracle
TOL32_C = 2e-5       # FP32: each gas's concentrations relative to that gas's own scale
GASES = ("co2", "ch4", "n2o", "hfc")
_AM = {"exp": o.ALPHA_EXP, "sinh": o.ALPHA_SINH, "newton": o.ALPHA_NEWTON, "one": o.ALPHA_ONE}
N_CASES = int(os.environ.get("UFAIR_FUZZ_CASES", "40"))   # a one-off wider sweep: UFAIR_FUZZ_CASES=400 pytest ...


def _case(seed):
    """The configuration a seed stands for."""
    r = np.random.default_rng(1000 + seed)
    G = int(r.integers(1, 5))
    M = int(r.choice([1, 2, 7, 31, 32, 33, 100, 321, 640, 1000, 2049]))
    n_t = int(r.choice([1, 2, 7, 8, 9, 16, 17, 50, 129]))
    c = dict(G=G, M=M, n_t=n_t, dense=bool(r.integers(0, 2)), dt=float(r.choice([1.0, 0.25, 0.1])),
             alpha_mode=str(r.choice(["exp", "exp", "sinh", "newton", "one"])), newton_iters=int(r.integers(0, 4)),
             iirf_max=[None, 97.0, 40.0][int(r.integers(0, 3))], t_mode=str(r.choice(["mid", "end"])),
             e_layout=str(r.choice(["member", "scenario", "scenario+scale"])),
             fext=str(r.choice(["none", "shared", "scenario", "member"])), resume=bool(r.integers(0, 2)),
             driven=int(r.integers(0, 1 << G)) if r.random() < 0.3 else 0, stats=bool(r.integers(0, 2)))
    return c


def check_case(seed, run_ensemble, HistSpec, to_dev, to_np, precision="f64"):
    """Build configuration `seed`, run it through `run_ensemble` (the public API's signature) in `precision` and
    check every output against the C oracle.  Returns the errors it measured, by output.

    FP64: every output by the per-gas / per-state-row rule of tests.util.output_relerr, <= 1e-10.
    FP32: T within 1e-4 K (absolute); each emission-driven gas's C within 2e-5 of that gas's own scale.  RF is
    not checked beyond what T implies (FP32 log2 of 1 + tiny is not 2e-5-accurate in runs of a few steps), and
    a concentration-driven gas is checked through T only (its diagnosed emissions cancel in FP32)."""
    c = _case(seed)
    G, M, n_t = c["G"], c["M"], c["n_t"]
    ens = ensemble(M, n_t=n_t, dt=c["dt"], dense=c["dense"], gases=GASES[:G], seed=seed)
    gp, tp = ens["gas_params"], ens["thermal_params"]
    kw, okw = {}, {}
    if c["e_layout"] == "member":
        E = ens["E"]
    else:
        E = ens["scen"]
        kw["scen_idx"], okw["scen_idx"] = to_dev(ens["scen_idx"]), ens["scen_idx"]
        if c["e_layout"] == "scenario+scale" and not c["driven"]:
            kw["e_scale"], okw["e_scale"] = to_dev(ens["e_scale"]), ens["e_scale"]
    S = ens["scen"].shape[2]
    if c["fext"] == "shared":
        fx = ens["f_ext"]
    elif c["fext"] == "scenario" and c["e_layout"] != "member":
        fx = np.stack([ens["f_ext"] * (1 + 0.2 * s) for s in range(S)], axis=1)
    elif c["fext"] == "scenario":                           # per-member emissions: one shared series
        fx = ens["f_ext"]
    elif c["fext"] == "member":
        fx = ens["f_ext"][:, None] * (1 + 0.01 * np.arange(M))[None, :]
        kw["fext_per_member"] = okw["fext_per_member"] = True
    if c["fext"] != "none":
        kw["f_ext"], okw["f_ext"] = to_dev(fx), fx
    modes = dict(alpha_mode=c["alpha_mode"], newton_iters=c["newton_iters"], iirf_max=c["iirf_max"], t_mode=c["t_mode"])
    omodes = dict(modes, alpha_mode=_AM[c["alpha_mode"]], t_mode=o.T_END if c["t_mode"] == "end" else o.T_MID)
    state = None
    if c["resume"]:   # a spun-up state from a short forward run of the same members
        state = co.oxfair(ens["E"][:, : max(1, n_t // 2)], gp, tp, dt=c["dt"], **{k: v for k, v in omodes.items()})["state"]
        kw["state_in"], okw["state_in"] = to_dev(state), state
    if c["driven"]:   # concentration-driven gases: feed them the concentrations of a forward run
        fwd = co.oxfair(E, gp, tp, dt=c["dt"], **okw, **omodes)
        Cf = fwd["C"]
        E = np.array(E)
        for g in range(G):
            if (c["driven"] >> g) & 1:
                if c["e_layout"] == "member":
                    E[g] = Cf[g]
                else:       # scenario-shared pathways: take each scenario's first member as its pathway
                    first = [int(np.argmax(ens["scen_idx"] == s)) if np.any(ens["scen_idx"] == s) else 0 for s in range(S)]
                    E[g] = Cf[g][:, first]
        kw["conc_driven"] = [bool((c["driven"] >> g) & 1) for g in range(G)]
        okw["conc_driven"] = c["driven"]
    spec = HistSpec(lo=-1.0, hi=6.0, bins=64, copies=3) if c["stats"] else None
    res = run_ensemble(to_dev(E), to_dev(gp), to_dev(tp), dt=c["dt"], stats=spec, precision=precision,
                       outputs=("C", "RF", "T", "alpha"), **kw, **modes)
    ref = co.oxfair(E, gp, tp, dt=c["dt"], want_alpha=True, **okw, **omodes)
    errs = {}
    if precision == "f64":
        for k in ("C", "RF", "T", "alpha", "state"):
            errs[k] = output_relerr(k, to_np(getattr(res, k)), ref[k])
            assert errs[k] < TOL64, f"{c}: {k} relative error {errs[k]:.3e}"
        if c["driven"]:
            errs["E"] = output_relerr("E", to_np(res.E), ref["E"])
            assert errs["E"] < 1e-9, f"{c}: E relative error {errs['E']:.3e}"
    else:
        T = to_np(res.T)
        assert T.dtype == np.float32
        errs["T"] = float(np.max(np.abs(T.astype(np.float64) - ref["T"]))) if T.size else 0.0
        assert errs["T"] <= TOL32_T, f"{c}: T off by {errs['T']:.3e} K"
        emitted = [g for g in range(G) if not (c["driven"] >> g) & 1]
        if emitted:
            errs["C"] = slice_relerr(to_np(res.C)[emitted], ref["C"][emitted])
            assert errs["C"] <= TOL32_C, f"{c}: C relative error {errs['C']:.3e} (gases {emitted})"
    if spec is not None:
        T = to_np(res.T)
        # binned in T's own precision: the C oracle's recount casts to float64 first, so it serves FP64 only
        hist, mom = (co if precision == "f64" else o).temperature_stats(T, spec.lo, spec.hi, spec.bins)
        assert np.array_equal(to_np(res.hist), hist.astype(np.int64)), f"{c}: histogram"
        assert np.allclose(to_np(res.moments), mom, rtol=1e-12, atol=1e-11), f"{c}: moments"
    return errs
