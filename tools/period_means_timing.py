"""Time the period-mean loop (out_every = k) against the per-step loops it stands in for.

(a) bench shard at 740 steps (736 is not a multiple of 10; both loops run the same 740): 1.25e6 members x 3 gases,
    FP64, per-member emissions from the device sampler (22 GB, larger than L2): k = 1 C / RF / T (the plain loop)
    against k = 10 C / RF / T (the period-mean loop), kernel ms.
(b) configs[4] device-resident: 10^6 members x 7360 steps of 0.1 yr, scenario-shared emissions: k = 1 T + statistics
    (what bench.py runs) against k = 10 C / RF / T + statistics, ms of one integration plus its statistics pass.
(c) host pipeline end to end: scenario-table inputs from host memory, C / RF / T of every member back into pinned
    host buffers, k = 1 against k = 10, member-steps/s beside the device-to-host link rate the link probe measures
    in the same call (the rate a link-bound call cannot exceed: D2H GB/s over bytes back per member-step).
Each pair alternates after a warm-up of both; (a) and (b) time with CUDA events, (c) with the host clock around the
synchronous call.  Medians are reported with min and max.  One JSON line, with the card and its power limit.

    python tools/period_means_timing.py [--reps 7] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = (x.strip() for x in out.split(",", 1))
        return name, power
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        return "unknown", "unknown"


def stats_of(ms):
    import numpy as np
    ms = np.asarray(ms, dtype=float)
    return {"median": round(float(np.median(ms)), 3), "min": round(float(ms.min()), 3), "max": round(float(ms.max()), 3)}


def alternate(torch, plans, reps, with_stats):
    """CUDA-event ms of each plan's launch (+ statistics pass), plans alternating; the statistics reset is outside
    the timed window."""
    def one(p, timed):
        p.reset_stats()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        p.launch()
        if with_stats:
            p.stats_pass()
        b.record()
        return (a, b) if timed else None

    for p in plans.values():
        one(p, False)
    torch.cuda.synchronize()
    ev = {k: [] for k in plans}
    for _ in range(reps):
        for k, p in plans.items():
            ev[k].append(one(p, True))
    torch.cuda.synchronize()
    return {k: stats_of([a.elapsed_time(b) for a, b in v]) for k, v in ev.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--host-members", type=int, default=262_144)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    from fiveeqscm_b200 import _abi
    from fiveeqscm_b200 import concentrations as conc
    from fiveeqscm_b200 import params as P

    assert torch.cuda.is_available(), "the timing needs a GPU"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    name, power = card()
    out = {"tool": "period_means_timing", "device": name, "power_limit": power, "precision": "f64", "reps": args.reps}
    k = 10

    # ---- (a) bench shard: per-member emissions, C / RF / T, equal work
    M, n_t = 1_250_000, 740
    gp, tp, scale, idx = P.sample_on_device(M, 20261018, n_scen=4, dense_pools=True)
    scen = torch.from_numpy(P.scenario_emissions(n_t)).to(dev)
    E = (scen[:, :, idx.long()] * scale[:, None, :]).contiguous()
    plans = {"k1": conc.DevicePlan(E, gp.contiguous(), tp.contiguous(), return_state=False),
             "k10": conc.DevicePlan(E, gp.contiguous(), tp.contiguous(), return_state=False, out_every=k)}
    loops = {}
    for key, p in plans.items():
        p.kernel_variant()
        loops[key] = p.loop_variant
    t = alternate(torch, plans, args.reps, False)
    out["a_bench_shard"] = {"members": M, "n_t": n_t, "n_gas": 3, "outputs": "C,RF,T", "loops": loops, "ms": t,
                            "ratio_k10_over_k1": round(t["k10"]["median"] / t["k1"]["median"], 3)}
    del plans, E, gp, tp, scale, idx, scen
    torch.cuda.empty_cache()

    # ---- (b) configs[4], device-resident, with statistics
    M, n_t, dt = 1_000_000, 7360, 0.1
    gp, tp, scale, idx = P.sample_on_device(M, 20261018, n_scen=4, dense_pools=True)
    scen = torch.from_numpy(P.scenario_emissions(n_t, dt)).to(dev)
    kw = dict(dt=dt, scen_idx=idx.contiguous(), e_scale=scale.contiguous(), stats=conc.HistSpec(), return_state=False)
    plans = {"k1_T_stats": conc.DevicePlan(scen, gp.contiguous(), tp.contiguous(), outputs=("T",), **kw),
             "k10_CRFT_stats": conc.DevicePlan(scen, gp.contiguous(), tp.contiguous(), out_every=k, **kw)}
    t = alternate(torch, plans, max(3, args.reps // 2), True)
    out["b_configs4_device"] = {
        "members": M, "n_t": n_t, "dt": dt, "ms": t,
        "output_GB": {"k1_T_stats": round(n_t * M * 8 / 1e9, 1), "k10_CRFT_stats": round(7 * (n_t // k) * M * 8 / 1e9, 1)},
        "ratio_k10_over_k1": round(t["k10_CRFT_stats"]["median"] / t["k1_T_stats"]["median"], 3)}
    del plans, gp, tp, scale, idx, scen
    torch.cuda.empty_cache()

    # ---- (c) host pipeline end to end: scenario tables in, full trajectories out
    M, n_t = args.host_members, 740
    ens = P.sample_ensemble(M, n_t=n_t, dense_pools=True)
    hkw = dict(scen_idx=ens["scen_idx"], e_scale=ens["e_scale"], return_state=False)
    outs = {kk: conc.pinned_result(3, n_t, M, return_state=False, out_every=kk) for kk in (1, k)}
    chunk = {kk: conc.auto_chunk_members(3, n_t, e_member=False, fext_member=False, outputs=("C", "RF", "T"),
                                         return_state=False, e_scale=True, out_every=kk) for kk in (1, k)}
    wss = {kk: conc.Workspace(0, chunk[kk]) for kk in (1, k)}

    def host_run(kk):
        t0 = time.perf_counter()
        conc.run_ensemble(ens["scen"], ens["gas_params"], ens["thermal_params"], out_every=kk, out=outs[kk],
                          workspace=wss[kk], **hkw)
        return time.perf_counter() - t0

    for kk in (1, k):
        host_run(kk)
    secs = {1: [], k: []}
    for _ in range(args.reps):
        for kk in (1, k):
            secs[kk].append(host_run(kk))
    for ws in wss.values():
        ws.close()
    L = _abi.lib()
    gbs, s = (C.c_double * 2)(), C.c_double()
    nbytes = 1 << 30
    _abi.check(L.ufair_link_probe(0, 0, nbytes, 0, 8, gbs, C.byref(s)))
    _abi.check(L.ufair_link_probe(0, 0, 0, 0, 0, gbs, None))
    d2h = gbs[1]
    res = {"members": M, "n_t": n_t, "d2h_GBps": round(d2h, 2), "chunk_members": {str(kk): chunk[kk] for kk in chunk}}
    import numpy as np
    for kk in (1, k):
        med = float(np.median(secs[kk]))
        bytes_per_ms = 7 * 8 / kk                      # C, RF of 3 gases and T, per member-step
        res[f"k{kk}"] = {"s": stats_of(secs[kk]), "member_steps_per_s": float(f"{M * n_t / med:.4g}"),
                         "bytes_back_per_member_step": round(bytes_per_ms, 2),
                         "link_bound_member_steps_per_s": float(f"{d2h * 1e9 / bytes_per_ms:.4g}")}
    res["speedup_k10_over_k1"] = round(res[f"k{k}"]["member_steps_per_s"] / res["k1"]["member_steps_per_s"], 2)
    out["c_host_pipeline"] = res

    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
