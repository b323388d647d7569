"""Time float32 outputs of FP64 runs (out_dtype="f32") against FP64 outputs.

(a) host pipeline end to end: 262 144 members x 740 steps, scenario-table inputs from host memory, C / RF / T of every
    member back into pinned host buffers; FP64 and float32 outputs, each per step (k = 1) and as period means (k = 10).
    Member-steps/s beside the link-bound rate: the device-to-host GB/s the link probe measures in the same call over
    the bytes back per member-step (7 values x 8 or 4 bytes / k).
(b) device-resident, the bench shard: 1.25e6 members x 736 steps x 3 gases, per-member emissions from the device
    sampler (22 GB, larger than L2), C / RF / T + statistics: integrator ms and statistics-pass ms, FP64 against
    float32 outputs.
Each set of arms alternates after a warm-up of every arm; (a) times with the host clock around the synchronous call,
(b) with CUDA events.  Medians are reported with min and max.  One JSON line, with the card and its power limit.

    python tools/f32_outputs_timing.py [--reps 7] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.period_means_timing import card, stats_of  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--host-members", type=int, default=262_144)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import numpy as np
    import torch

    from fiveeqscm_b200 import _abi
    from fiveeqscm_b200 import concentrations as conc
    from fiveeqscm_b200 import params as P

    assert torch.cuda.is_available(), "the timing needs a GPU"
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    name, power = card()
    out = {"tool": "f32_outputs_timing", "device": name, "power_limit": power, "precision": "f64", "reps": args.reps}

    # ---- (a) host pipeline end to end: scenario tables in, full trajectories out
    M, n_t = args.host_members, 740
    ens = P.sample_ensemble(M, n_t=n_t, dense_pools=True)
    hkw = dict(scen_idx=ens["scen_idx"], e_scale=ens["e_scale"], return_state=False)
    arms = [(od, k) for k in (1, 10) for od in ("f64", "f32")]
    key = lambda od, k: f"{od}_k{k}"
    outs = {key(od, k): conc.pinned_result(3, n_t, M, return_state=False, out_every=k, out_dtype=od) for od, k in arms}
    chunk = {key(od, k): conc.auto_chunk_members(3, n_t, e_member=False, fext_member=False, outputs=("C", "RF", "T"),
                                                 return_state=False, e_scale=True, out_every=k, out_dtype=od)
             for od, k in arms}
    wss = {kk: conc.Workspace(0, c) for kk, c in chunk.items()}

    def host_run(od, k):
        t0 = time.perf_counter()
        conc.run_ensemble(ens["scen"], ens["gas_params"], ens["thermal_params"], out_every=k, out_dtype=od,
                          out=outs[key(od, k)], workspace=wss[key(od, k)], **hkw)
        return time.perf_counter() - t0

    for od, k in arms:
        host_run(od, k)
    secs = {key(od, k): [] for od, k in arms}
    for _ in range(args.reps):
        for od, k in arms:
            secs[key(od, k)].append(host_run(od, k))
    for ws in wss.values():
        ws.close()
    L = _abi.lib()
    gbs, s = (C.c_double * 2)(), C.c_double()
    _abi.check(L.ufair_link_probe(0, 0, 1 << 30, 0, 8, gbs, C.byref(s)))
    _abi.check(L.ufair_link_probe(0, 0, 0, 0, 0, gbs, None))
    d2h = gbs[1]
    res = {"members": M, "n_t": n_t, "d2h_GBps": round(d2h, 2), "chunk_members": chunk}
    for od, k in arms:
        med = float(np.median(secs[key(od, k)]))
        per = 7 * (8 if od == "f64" else 4) / k             # bytes back per member-step: C, RF of 3 gases and T
        rate, bound = M * n_t / med, d2h * 1e9 / per
        res[key(od, k)] = {"s": stats_of(secs[key(od, k)]), "member_steps_per_s": float(f"{rate:.4g}"),
                           "bytes_back_per_member_step": round(per, 2),
                           "link_bound_member_steps_per_s": float(f"{bound:.4g}"),
                           "fraction_of_link_bound": round(rate / bound, 3)}
    for k in (1, 10):
        res[f"speedup_f32_over_f64_k{k}"] = round(res[key("f32", k)]["member_steps_per_s"] /
                                                   res[key("f64", k)]["member_steps_per_s"], 2)
    out["a_host_pipeline"] = res
    del outs, ens
    torch.cuda.empty_cache()

    # ---- (b) the bench shard, device-resident: integrator and statistics pass, FP64 against float32 outputs
    M, n_t = 1_250_000, 736
    gp, tp, scale, idx = P.sample_on_device(M, 20261018, n_scen=4, dense_pools=True)
    scen = torch.from_numpy(P.scenario_emissions(n_t)).to(dev)
    E = (scen[:, :, idx.long()] * scale[:, None, :]).contiguous()
    plans = {od: conc.DevicePlan(E, gp.contiguous(), tp.contiguous(), stats=conc.HistSpec(), return_state=False,
                                 out_dtype=od) for od in ("f64", "f32")}
    loops = {}
    for od, p in plans.items():
        p.kernel_variant()
        loops[od] = p.loop_variant

    def one(p):
        p.reset_stats()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        p.launch()
        ev[1].record()
        p.stats_pass()
        ev[2].record()
        return ev

    for p in plans.values():
        one(p)
    torch.cuda.synchronize()
    evs = {od: [] for od in plans}
    for _ in range(args.reps):
        for od, p in plans.items():
            evs[od].append(one(p))
    torch.cuda.synchronize()
    res = {"members": M, "n_t": n_t, "n_gas": 3, "outputs": "C,RF,T + statistics", "loops": loops}
    for od, v in evs.items():
        res[od] = {"integrator_ms": stats_of([a.elapsed_time(b) for a, b, _ in v]),
                   "stats_pass_ms": stats_of([b.elapsed_time(c) for _, b, c in v]),
                   "output_GB": round(7 * n_t * M * (8 if od == "f64" else 4) / 1e9, 1)}
    for part in ("integrator_ms", "stats_pass_ms"):
        res[f"ratio_f32_over_f64_{part}"] = round(res["f32"][part]["median"] / res["f64"][part]["median"], 3)
    out["b_bench_shard_device"] = res

    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
