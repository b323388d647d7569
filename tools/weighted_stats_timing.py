"""Time the weighted statistics pass against the unweighted one on the bench shard's T.

The bench shard: 1.25e6 members x 736 steps from the device sampler (four scenarios), FP64, so T is 7.4 GB --
larger than L2, every pass reads it from HBM.  One integration writes T; then every arm's pass reads that same T
through its own descriptor and private buffers:
    pooled             stat_group = NULL, ufair_stats_pass_f64 (the pass bench.py times)
    pooled_weighted    the same with integer member weights, ufair_stats_pass_weighted_f64
    scenario4          stat_group = scen_idx, 4 groups
    scenario4_weighted the same with the weights
The weights are integers 0 .. 1000 (about 10 % of them 0), as stats.integer_weights makes them from likelihoods.
After a warm-up of every arm the arms alternate, `--reps` rounds, each pass timed with CUDA events (the reset of the
private buffers is outside the timed window).  Prints one JSON line: the card and its power limit, median ms per
pass, the spread, GB/s of T read, and each weighted arm against its unweighted twin.

    python tools/weighted_stats_timing.py [--reps 20] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--members", type=int, default=1_250_000)
    ap.add_argument("--n-t", type=int, default=736)
    ap.add_argument("--reps", type=int, default=20)
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
    L = _abi.lib()
    M, n_t = args.members, args.n_t
    gp, tp, scale, idx = P.sample_on_device(M, 20261018, n_scen=4, dense_pools=True)
    scen = torch.from_numpy(P.scenario_emissions(n_t)).to(dev)
    spec = conc.HistSpec()
    rng = np.random.default_rng(1)
    w = rng.integers(0, 1001, M)
    w[rng.random(M) < 0.1] = 0
    plan = conc.DevicePlan(scen, gp.contiguous(), tp.contiguous(), scen_idx=idx.contiguous(), e_scale=scale.contiguous(),
                           stats=spec, outputs=("T",), return_state=False, stat_weight=torch.from_numpy(w).to(dev))
    plan.launch()                                   # T, once: every arm reads these rows
    torch.cuda.synchronize()
    weight = plan.stat_weight.data_ptr()

    arms = {"pooled": (None, 0, False), "pooled_weighted": (None, 0, True),
            "scenario4": (plan.scen_idx, 4, False), "scenario4_weighted": (plan.scen_idx, 4, True)}
    descs, keep = {}, []
    for name, (lab, G, _) in arms.items():
        d = _abi.UfairDesc.from_buffer_copy(plan.desc)
        rows = max(1, G) * n_t
        hp = torch.empty(spec.copies, rows, spec.bins, dtype=torch.int32, device=dev)
        mp = torch.empty(spec.copies, rows, _abi.MOM_COUNT, dtype=torch.float64, device=dev)
        d.hist_private, d.moments_private = hp.data_ptr(), mp.data_ptr()
        d.n_stat_groups, d.stat_group = G, (lab.data_ptr() if lab is not None else None)
        keep += [hp, mp]
        descs[name] = d

    stream = torch.cuda.current_stream().cuda_stream

    def one(name, timed):
        d, weighted = descs[name], arms[name][2]
        _abi.check(L.ufair_stats_reset(C.byref(d), stream))
        if timed:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
        if weighted:
            _abi.check(L.ufair_stats_pass_weighted_f64(C.byref(d), weight, stream))
        else:
            _abi.check(L.ufair_stats_pass_f64(C.byref(d), stream))
        if timed:
            b.record()
            return a, b

    for name in descs:                              # warm-up: module load, smem attributes, first touch
        one(name, False)
        one(name, False)
    torch.cuda.synchronize()
    ev = {name: [] for name in descs}
    for _ in range(args.reps):
        for name in descs:
            ev[name].append(one(name, True))
    torch.cuda.synchronize()
    t_bytes = M * n_t * 8
    name, power = card()
    out = {"tool": "weighted_stats_timing", "device": name, "power_limit": power, "members": M, "n_t": n_t,
           "precision": "f64", "bins": spec.bins, "copies": spec.copies, "reps": args.reps, "T_bytes": t_bytes,
           "weights": "integers 0..1000, 10 % zero", "weight_total": int(w.sum()), "variants": {}}
    for k, pairs in ev.items():
        ms = np.array([a.elapsed_time(b) for a, b in pairs])
        med = float(np.median(ms))
        out["variants"][k] = {"ms_median": round(med, 4), "ms_min": round(float(ms.min()), 4),
                              "ms_max": round(float(ms.max()), 4), "T_GBps": round(t_bytes / med / 1e6, 1)}
    for k in ("pooled", "scenario4"):
        v = out["variants"][k + "_weighted"]
        v["vs_unweighted"] = round(v["ms_median"] / out["variants"][k]["ms_median"], 3)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
