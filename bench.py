#!/usr/bin/env python
"""bench.py -- headline benchmark of the Universal-FaIR ensemble integrator on B200.

Metric (BASELINE.json): ensemble member-timesteps/sec.  Workload: one GPU's shard of configs[3]
(10^7-member x 736-year 3-gas ensemble over 8 GPUs = 1.25e6 members per GPU), FP64, per-member
emissions resident in HBM, full C/RF/T output to HBM, per-step temperature histogram + moments,
NCCL all-reduce of the statistics when N > 1.  Weak scaling: per-GPU work is fixed.

    python bench.py [--gpus N] [--steps K] [--warmup W]            our arm
    python bench.py --impl reference ...                             the CPU arm (oracle on host cores)
    torchrun --nproc-per-node N bench.py --gpus N ...                N > 1
    python bench.py ... --dump-outputs DIR                           also write the last timed step's outputs

One JSON line on stdout (rank 0).  `value` = device-resident throughput; `e2e` = the same metric
through the public host-buffer API (pinned host inputs -> H2D -> kernel -> D2H of all outputs), stated
against the host-link ceiling measured in the same run with the same number of ranks copying at once;
`roofline` = the integrate kernel against the FP64-pipe peak measured in this run (and the HBM view);
`configs` = the other BASELINE.json configurations (N = 1); `cpu_baseline` = the CPU rendering of the
loop timed on this box's cores on a bounded sample.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402,F401

N_GAS = 3
# algorithmic work per member-step (BASELINE.md section 5 / DESIGN.md): 3 gases
#   bytes: 3 E in + 3 C + 3 RF + 1 T out = 10 words (80 B in f64, 40 B in f32)
FLOPS_PER_STEP = 751.0               # 163 simple + 15 exp(28) + 3 log(36) + 3 sqrt(10) + 3 div(10)
METRIC = "ensemble member-timesteps/sec"
CPU_SAMPLE_MEMBERS = 65536           # the CPU arm's sample, the same in both legs (cpu_baseline and --impl reference)
DUMP_BYTES = 63_000_000              # --dump-outputs writes at most this much in all (64 MB with the .npy headers)
DUMP_SEED = 0                        # ... and samples larger outputs with this seed


def algorithmic_flops(gas_form, newton_iters=0):
    """SURVEY.md 8(d) convention (exp = 28, log = 36, sqrt = 10, div = 10 FP64 flops), per member-step,
    for the pools and forcing terms the parameters actually use: per gas 18 + 8 n_pool simple flops,
    1 + n_pool exponentials, one division, a log / sqrt where that term exists; 13 for the thermal
    step.  Four pools and all three terms in every gas give the survey's 751.  Newton mode adds, per
    iteration and gas, n_pool exponentials and ~30 simple flops (SURVEY.md 8a, row a3)."""
    total = 13.0
    for f in gas_form:
        n_pool = (f & 7) or 4
        terms = (f >> 4) & 7 or 7
        total += 18 + 8 * n_pool + 28 * (1 + n_pool) + 10 + (36 if terms & 1 else 0) + (10 if terms & 4 else 0)
        total += newton_iters * (28 * n_pool + 30)
    return total


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--members-per-gpu", type=int, default=1_250_000)
    ap.add_argument("--n-t", type=int, default=736)
    ap.add_argument("--precision", default="f64", choices=["f64", "f32"])
    ap.add_argument("--e2e-members", type=int, default=-1, help="members per GPU of the e2e leg (0: the whole shard; default: "
                    "786432 at N <= 2, 393216 at N = 4, 262144 at N = 8 -- page-locking the shard's 74 GB of host buffers takes "
                    "~35 s per rank alone and more with 8 ranks at once, which would be most of the run, and at N >= 4 this "
                    "platform's shared host link makes the same bytes take 3-5x as long; always within a third of free host memory)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-chunk", type=int, default=16384, help="members per chunk of the host pipeline")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU work for the cpu_baseline sample")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-lit", action="store_true", help="skip the secondary literature-parameter measurement")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE.json configurations")
    ap.add_argument("--configs-scale", type=float, default=1.0, help="test hook: shrink the member counts of `configs`")
    ap.add_argument("--sparse", action="store_true", help="literature-style sparse parameters (1-pool CH4/N2O)")
    ap.add_argument("--general-kernel", action="store_true", help="experiment: never pick a specialised per-gas form")
    ap.add_argument("--fext", action="store_true", help="experiment: add a shared external-forcing series")
    ap.add_argument("--iirf-max", type=float, default=None, help="experiment: switch the iIRF ceiling on (general kernel)")
    ap.add_argument("--no-stats", action="store_true", help="experiment: integrate without histogram/moments")
    ap.add_argument("--outputs", default="C,RF,T", help="experiment: comma list of outputs written to HBM ('' = none)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32 / float64, "
                         "rank 0's members; a fixed seeded sample of members, and of steps if need be, keeps it under 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_config(args, n_gpus):
    return {
        "workload": "configs[3] shard: 3-gas (CO2/CH4/N2O) x %d steps x %d members per GPU (x%d GPUs = %d members), "
                    "per-member emissions, full C/RF/T output + per-step T histogram (1024 bins) and moments"
                    % (args.n_t, args.members_per_gpu, n_gpus, args.members_per_gpu * n_gpus),
        "members_per_gpu": args.members_per_gpu, "n_t": args.n_t, "n_gas": N_GAS, "dt_years": 1.0,
        "alpha_mode": "exp", "t_mode": "mid", "parameters": "sparse" if args.sparse else "dense (4 active pools, 3 forcing terms per gas)",
        "sharding": "member axis, %d rank(s), no data-path collective; one all-reduce group of histogram+moments per step, "
                    "overlapped with the next step's integration" % n_gpus,
        "l2": "inputs (%.1f GB per step) exceed L2; no explicit flush" % (N_GAS * args.n_t * args.members_per_gpu * 8 / 1e9),
    }


# ------------------------------------------------------------------------------------------------
# synthetic inputs on the device (the product's own sampler)
# ------------------------------------------------------------------------------------------------
def device_ensemble(torch, M, n_t, first_member, dense, dt=1.0, expand=True):
    """Synthetic inputs generated on the GPU by the product's own sampler (ufair_sample_f64: Philox
    stream keyed by the GLOBAL member index, so the N ranks together hold the one ensemble a single
    GPU would generate): perturbed parameters, a scenario index and an emission scale per member.
    expand=True returns per-member emission rows (scenario rows times the scale), else the scenario
    table with the index and scale."""
    from fiveeqscm_b200 import params as P
    dev = torch.device("cuda", torch.cuda.current_device())
    gp, tp, scale, idx = P.sample_on_device(M, 20261018, first_member=first_member, n_scen=4, dense_pools=dense)
    scen = torch.from_numpy(P.scenario_emissions(n_t, dt)).to(dev)               # [3][n_t][4]
    if not expand:
        return scen, gp.contiguous(), tp.contiguous(), idx.contiguous(), scale.contiguous()
    E = scen[:, :, idx.long()]                                                    # [3][n_t][M]
    E *= scale[:, None, :]
    return E.contiguous(), gp.contiguous(), tp.contiguous()


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "power_w_max": None, "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1])); pw.append(float(c[2]))
            except ValueError:
                continue
            for nme, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            busy = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons),
                       power_w_max=max(pw), samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle on the host cores (the only place bench.py executes oracle/)
# ------------------------------------------------------------------------------------------------
def host_threads():
    """Host threads the CPU arm may use: the cores this process can run on (torchrun exports
    OMP_NUM_THREADS=1, which is about the GPU ranks, not about this leg)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_rates(E, gp, tp, target_seconds):
    """member-steps/s on this box's cores of (a) the blocked, vectorised CPU rendering of the loop
    (oracle/ufair_oracle_fast.c: tiles of 64 members, libmvec, OpenMP -- the baseline) and (b) the textbook
    scalar loop the parity tests check against, both on the same fixed sample, C/RF/T written to host memory."""
    from oracle import c_oracle as co
    n_thr = host_threads()
    n, n_t = E.shape[2], E.shape[1]
    run = lambda blocked: co.oxfair(E, gp, tp, outputs=("C", "RF", "T"), n_threads=n_thr, blocked=blocked)
    run(True)                                                # warm-up: page the sample in, spin the threads up
    t0 = time.perf_counter(); run(True); dt1 = max(time.perf_counter() - t0, 1e-6)
    reps = max(1, int(target_seconds / dt1))
    t0 = time.perf_counter()
    for _ in range(reps):
        out = run(True)
    fast = reps * n * n_t / (time.perf_counter() - t0)
    n_txt = min(n, 64 * n_thr * 4)                           # the scalar loop is ~20x slower: a slice of the sample
    t0 = time.perf_counter()
    co.oxfair(E[:, :, :n_txt], gp[:, :, :n_txt], tp[:, :n_txt], outputs=("C", "RF", "T"), n_threads=n_thr)
    textbook = n_txt * n_t / (time.perf_counter() - t0)
    return fast, textbook, out["threads"], reps


def cpu_sample(n_t, dense, n=CPU_SAMPLE_MEMBERS):
    from fiveeqscm_b200 import params as P
    ens = P.sample_ensemble(n, n_t=n_t, dense_pools=dense)
    E = P.member_emissions(ens["scen"], ens["scen_idx"], ens["e_scale"])
    return E, ens["gas_params"], ens["thermal_params"]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import c_oracle as co
    n_thr = host_threads()
    n = CPU_SAMPLE_MEMBERS
    E, gp, tp = cpu_sample(args.n_t, not args.sparse)
    run = lambda: co.oxfair(E, gp, tp, n_threads=n_thr, blocked=True)
    out = run()
    t0 = time.perf_counter(); out = run(); dt0 = time.perf_counter() - t0
    reps = max(1, int(1.0 / max(dt0, 1e-3)))                 # ~1 s of work per step

    def step():
        for _ in range(reps):
            out = run()
            co.temperature_stats(out["T"][:, :4096], -5.0, 25.0, 1024)   # histogram of a slice (serial helper; not the point)
        return out
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step()
    el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: out[k] for k in ("C", "RF", "T", "state")}, {})
    work = args.steps * reps * n * args.n_t
    val = work / el
    sample = ("%d members x %d steps x %d passes per step; blocked + vectorised C rendering of the loop "
              "(oracle/ufair_oracle_fast.c, OpenMP, libmvec), C/RF/T written to host memory" % (n, args.n_t, reps))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "member-timesteps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, args.gpus),
            "cpu_baseline": {"value": val, "unit": "member-timesteps/s", "cores": n_thr, "kind": "port", "sample": sample,
                             "host_cpus": os.cpu_count()},
            "e2e": {"value": val, "unit": "member-timesteps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "the reference ships no implementation of the 5-equation loop (SURVEY.md 0); this arm times the "
                    "in-repo CPU rendering of it (the fast blocked one, not the textbook checker) on the host cores"}
    emit(line)


# ------------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def claim_stdout():
    """Keep stdout for the ONE JSON line: everything else any library prints to fd 1 (NCCL's version
    banner, for one) is sent to stderr for the life of the process."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def dump_outputs(out_dir, per_member, per_step):
    """--dump-outputs: write the arrays the timed path returned in its last step as out_dir/<name>.npy, float32 or
    float64 (integer counts as float64).  per_member maps names to arrays whose last axis is the member axis, per_step
    to arrays whose first axis is the time step; torch tensors are sampled on their device before the copy.  To stay
    under DUMP_BYTES the per-step arrays keep at most a quarter of it (a sample of steps beyond that) and the
    per-member arrays share the rest (a sample of members).  Samples are sorted indices drawn with DUMP_SEED, so the
    same arguments give the same sample."""
    rng = np.random.default_rng(DUMP_SEED)

    def sample(n, k):
        return None if k >= n else np.sort(rng.choice(n, size=max(k, 1), replace=False))

    def take(x, idx, axis):
        if idx is not None:
            if hasattr(x, "index_select"):
                import torch
                x = x.index_select(axis, torch.as_tensor(idx, device=x.device))
            else:
                x = np.take(x, idx, axis=axis)
        x = np.asarray(x.cpu() if hasattr(x, "cpu") else x)
        return x if x.dtype in (np.float32, np.float64) else x.astype(np.float64)

    size = lambda shape: 8 * int(np.prod(shape, dtype=np.int64))       # bytes, counted as float64
    steps, used = None, 0
    if per_step:
        n_t, row = next(iter(per_step.values())).shape[0], sum(size(x.shape[1:]) for x in per_step.values())
        steps = sample(n_t, DUMP_BYTES // 4 // row)
        used = row * (n_t if steps is None else len(steps))
    members = None
    if per_member:
        n_member, column = next(iter(per_member.values())).shape[-1], sum(size(x.shape[:-1]) for x in per_member.values())
        members = sample(n_member, (DUMP_BYTES - used) // column)
    os.makedirs(out_dir, exist_ok=True)
    for name, x in per_step.items():
        np.save(os.path.join(out_dir, name + ".npy"), take(x, steps, 0))
    for name, x in per_member.items():
        np.save(os.path.join(out_dir, name + ".npy"), take(x, members, -1))


# ------------------------------------------------------------------------------------------------
# measured peaks and the roofline of one launch
# ------------------------------------------------------------------------------------------------
def measured_peaks(L, _abi):
    """HBM: MEASURED_PEAKS.json (driver-written).  FP64 / FP32 FMA and MUFU: measured here -- the first launch
    is the BURST figure (cold, full clock); steps are seconds long and run under the power cap, so the
    denominator is the SUSTAINED one: the same microbenchmark back to back, median of launches 6-10."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    out = {"hbm_gbs": float(peaks.get("hbm_gbs", 6650.0)),
           "hbm_source": "MEASURED_PEAKS.json (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"}
    msd, fl = ctypes.c_double(), ctypes.c_double()
    for key, fn, iters in (("fp64_tflops", L.ufair_peak_fp64, 400_000), ("fp32_tflops", L.ufair_peak_fp32, 800_000),
                           ("mufu_tops", L.ufair_peak_mufu, 800_000)):
        rates = []
        for _ in range(10 if key == "fp64_tflops" else 4):
            _abi.check(fn(iters, msd, fl, None))
            rates.append(fl.value / (msd.value * 1e-3) / 1e12)
        out[key + "_burst"] = rates[0]
        out[key] = statistics.median(rates[len(rates) // 2:])
    out["fma_source"] = ("FMA / MUFU.EX2 microbenchmarks in this run (ufair_peak_*): sustained = median of the second half "
                         "of back-to-back launches, burst = the first")
    return out


def roofline_of(kernel_ms, member_steps, bytes_step, flops_step, peaks, precision):
    """The binding roofline of one launch: max(bytes / HBM peak, flops / FMA-pipe peak) / measured time.  FP32
    mode evaluates exp / log / sqrt / reciprocal on the MUFU pipe, so the FMA-flop convention does not
    describe it: its binding roofline is HBM (SURVEY.md 8d)."""
    a_hbm = bytes_step * member_steps / (kernel_ms * 1e-3) / 1e9
    fpeak = peaks["fp64_tflops"] if precision == "f64" else peaks["fp32_tflops"]
    a_fp = flops_step * member_steps / (kernel_ms * 1e-3) / 1e12
    t_hbm, t_fp = bytes_step / (peaks["hbm_gbs"] * 1e9), flops_step / (fpeak * 1e12)
    name = "fp64" if precision == "f64" else "fp32"
    if t_hbm > t_fp or precision == "f32":
        r = {"bound": "hbm", "achieved": a_hbm, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": a_hbm / peaks["hbm_gbs"]}
    else:
        r = {"bound": name, "achieved": a_fp, "peak": fpeak, "unit": "TFLOP/s", "frac": a_fp / fpeak}
    r["hbm_frac"], r[name + "_frac"] = a_hbm / peaks["hbm_gbs"], a_fp / fpeak
    return r


def time_launches(torch, plan, n, warm=2, with_stats=True):
    """ms per integrator launch (CUDA events on the launching stream) and ms per whole step."""
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def step(k=None):
        plan.reset_stats()
        if k is not None:
            k[0].record()
        plan.launch()
        if k is not None:
            k[1].record()
        if with_stats:
            plan.stats_pass()
            plan.finalize_stats()
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    ks = [(ev(), ev()) for _ in range(n)]
    e0, e1 = ev(), ev()
    e0.record()
    for k in ks:
        step(k)
    e1.record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ks) / n, e0.elapsed_time(e1) / n


def variant_of(plan):
    f, g, m = plan.kernel_variant()
    return {"form": list(f), "gases_per_lane": g, "members_per_warp": m, "loop": plan.loop_variant}


def other_configs(torch, conc, peaks, spec, shrink=1.0):
    """BASELINE.json configs[1], [2], [4] and the Newton mode of north_star, each on its own line of the
    `configs` key: integrator ms per launch (CUDA events), member-steps/s of the whole step (integrator +
    statistics), roofline fraction, kernel variant.  One GPU."""
    out = {}
    free = torch.cuda.empty_cache
    sz = lambda m: m if shrink == 1.0 else max(2048, int(m * shrink) // 128 * 128)

    def entry(plan, M, n_t, kms, sms, bytes_step, flops_step, precision, what):
        r = roofline_of(kms, float(M) * n_t, bytes_step, flops_step, peaks, precision)
        return {"what": what, "members": M, "n_t": n_t, "dtype": precision, "kernel_ms": kms, "step_ms": sms,
                "value": float(M) * n_t / (sms * 1e-3), "unit": "member-timesteps/s",
                "roofline": r, "frac": r["frac"], "algorithmic_bytes_per_member_step": bytes_step,
                "algorithmic_flops_per_member_step": flops_step, "kernel_variant": variant_of(plan)}

    # ---- configs[1]: 10^4-member ensemble x 736 steps -- latency-bound: 1000 ten-member warps on a GPU that holds 2368
    try:
        M, n_t = sz(10_000), 736
        E, gp, tp = device_ensemble(torch, M, n_t, 0, True)
        plan = conc.DevicePlan(E, gp, tp, stats=spec)
        kms, sms = time_launches(torch, plan, 20, warm=3)
        v = variant_of(plan)
        e = entry(plan, M, n_t, kms, sms, 80, FLOPS_PER_STEP, "f64", "configs[1]: 3-gas 10^4-member ensemble x 736 steps, per-member "
                  "emissions, C/RF/T + statistics")
        warps = -(-M // v["members_per_warp"])
        e["occupancy"] = {"warps": warps, "sm_count": 148, "warps_per_sm": warps / 148.0,
                          "note": "latency-bound by construction (SURVEY.md H4): the ensemble is a fraction of one wave, so the "
                                  "serial 736-step chain of a warp sets the time, not the FP64 pipe"}
        out["configs1_1e4_members"] = e
        del plan, E, gp, tp
    except Exception as exc:
        out["configs1_1e4_members"] = {"error": repr(exc)}
    free()

    # ---- configs[2]: 10^6 members x 4 scenarios, scenario-shared emissions (+ per-member scale), FP64 and FP32
    for prec in ("f64", "f32"):
        key = "configs2_1e6x4_scenario_shared_" + prec
        try:
            M, n_t = sz(1_000_000), 736
            scen, gp, tp, idx, scale = device_ensemble(torch, M, n_t, 0, True, expand=False)
            idx.zero_()
            plan = conc.DevicePlan(scen, gp, tp, scen_idx=idx, e_scale=scale, stats=spec, precision=prec)
            ev = lambda: torch.cuda.Event(enable_timing=True)
            for s in range(2):
                plan.run()
            torch.cuda.synchronize()
            ks, e0, e1 = [], ev(), ev()
            e0.record()
            for s in range(4):                                # one launch per scenario: every member runs all four
                plan.scen_idx.fill_(s)
                plan.reset_stats()
                a, b = ev(), ev()
                a.record(); plan.launch(); b.record()
                plan.stats_pass(); plan.finalize_stats()
                ks.append((a, b))
            e1.record()
            torch.cuda.synchronize()
            kms, tot = sum(a.elapsed_time(b) for a, b in ks) / 4, e0.elapsed_time(e1)
            es = 8 if prec == "f64" else 4
            e = entry(plan, M, n_t, kms, tot / 4, 7 * es, FLOPS_PER_STEP, prec,
                      "configs[2]: 3-gas 10^6-member perturbed-parameter ensemble x 4 scenarios = 4 launches, scenario-shared "
                      "emissions [3][736][4] + per-member scale (no per-member input is read in the loop), C/RF/T + statistics")
            e["member_runs"] = 4 * M
            out[key] = e
            del plan, scen, gp, tp, idx, scale
        except Exception as exc:
            out[key] = {"error": repr(exc)}
        free()

    # ---- configs[4]: dt = 0.1 yr, 7360 steps
    try:   # (i) the whole 10^6-member ensemble in one launch: scenario-shared emissions, T + statistics device-resident
        M, n_t = sz(1_000_000), 7360
        scen, gp, tp, idx, scale = device_ensemble(torch, M, n_t, 0, True, dt=0.1, expand=False)
        plan = conc.DevicePlan(scen, gp, tp, dt=0.1, scen_idx=idx, e_scale=scale, stats=spec, outputs=("T",), return_state=False)
        kms, sms = time_launches(torch, plan, 2, warm=1)
        out["configs4_dt0.1_T_and_statistics"] = entry(
            plan, M, n_t, kms, sms, 8, FLOPS_PER_STEP, "f64",
            "configs[4]: 10^6 members x 7360 steps (dt = 0.1 yr) in ONE launch, scenario-shared emissions, T rows (59 GB) + "
            "per-step histogram / moments stay on the device")
        del plan, scen, gp, tp, idx, scale
    except Exception as exc:
        out["configs4_dt0.1_T_and_statistics"] = {"error": repr(exc)}
    free()
    try:   # (ii) full C/RF/T: 412 GB for the whole ensemble, so it runs as 8 member chunks of 125 000; one chunk timed
        M, n_t = sz(125_000), 7360
        E, gp, tp = device_ensemble(torch, M, n_t, 0, True, dt=0.1)
        plan = conc.DevicePlan(E, gp, tp, dt=0.1, stats=spec)
        kms, sms = time_launches(torch, plan, 3, warm=1)
        e = entry(plan, M, n_t, kms, sms, 80, FLOPS_PER_STEP, "f64",
                  "configs[4]: one of the 8 member chunks (125 000 members x 7360 steps, dt = 0.1 yr) the full-output run is cut "
                  "into: per-member emissions streamed from HBM (22 GB), C/RF/T written (52 GB), + statistics")
        e["chunks_for_1e6_members"] = 8
        out["configs4_dt0.1_full_output_chunk"] = e
        del plan, E, gp, tp
    except Exception as exc:
        out["configs4_dt0.1_full_output_chunk"] = {"error": repr(exc)}
    free()

    # ---- Newton mode (north_star: "fixed iteration count, deterministic"), K = 3, the headline shard
    try:
        M, n_t, K = sz(1_250_000), 736, 3
        E, gp, tp = device_ensemble(torch, M, n_t, 0, True)
        plan = conc.DevicePlan(E, gp, tp, stats=spec, alpha_mode="newton", newton_iters=K)
        kms, sms = time_launches(torch, plan, 3, warm=1)
        fl = algorithmic_flops((0,) * N_GAS, newton_iters=K)
        e = entry(plan, M, n_t, kms, sms, 80, fl, "f64",
                  "alpha mode NEWTON, K = 3 fixed iterations on iIRF100(alpha) = iIRF, on the configs[3] shard")
        e["newton_iters"] = K
        out["newton_k3"] = e
        del plan, E, gp, tp
    except Exception as exc:
        out["newton_k3"] = {"error": repr(exc)}
    free()
    return out


def canary_bitwise(torch, dist, conc, D, spec, rank, world, n_canary=65536):
    """SURVEY.md 8e "test this", on hardware: a 65 536-member canary ensemble is split over the ranks (the
    sampler is keyed by the global member index), integrated, reduced with the production StatsReducer; rank 0
    also integrates the whole canary alone.  Histogram, extrema and percentiles must agree bit for bit."""
    from fiveeqscm_b200 import stats as S
    n_t = 200
    lo, hi = D.shard_bounds(n_canary, world, rank)
    E, gp, tp = device_ensemble(torch, hi - lo, n_t, lo, True)
    plan = conc.DevicePlan(E, gp, tp, stats=spec, outputs=("T",), return_state=False)
    red = D.StatsReducer(plan)
    plan.reset_stats(); plan.launch(); plan.stats_pass(); red.submit(); red.wait()
    torch.cuda.synchronize()
    ok = None
    if rank == 0:
        E1, gp1, tp1 = device_ensemble(torch, n_canary, n_t, 0, True)
        one = conc.DevicePlan(E1, gp1, tp1, stats=spec, outputs=("T",), return_state=False).run()
        torch.cuda.synchronize()
        pcts = (5.0, 17.0, 50.0, 83.0, 95.0)
        pa = S.percentiles_device(plan.result.hist, spec.lo, spec.hi, pcts)
        pb = S.percentiles_device(one.hist, spec.lo, spec.hi, pcts)
        ok = bool(torch.equal(plan.result.hist, one.hist)) and bool(torch.equal(pa, pb)) and \
            bool(torch.equal(plan.result.moments[:, 2:], one.moments[:, 2:]))
    return ok


def main():
    claim_stdout()
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    import torch
    import torch.distributed as dist
    from fiveeqscm_b200 import _abi, concentrations as conc, dist as D

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (our arm) needs a GPU; there is no CPU fallback"
    torch.cuda.set_device(local)
    # one rank per GPU: on a multi-node host keep each rank (and the pinned host buffers it is about to allocate)
    # next to its GPU.  Not at N = 1, where the CPU-baseline leg wants every core of the box.
    binding = D.bind_rank_to_cpus(local, world) if world > 1 else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_gpus = world
    L = _abi.lib()
    M, n_t = args.members_per_gpu, args.n_t

    E, gp, tp = device_ensemble(torch, M, n_t, rank * M, dense=not args.sparse)
    spec = None if args.no_stats else conc.HistSpec()
    outs = tuple(o for o in args.outputs.split(",") if o)
    fx = None
    if args.fext:
        yr = torch.arange(n_t, device=E.device, dtype=torch.float64)
        fx = 0.1 * torch.sin(2.0 * 3.141592653589793 * yr / 11.0)
    plan = conc.DevicePlan(E, gp, tp, stats=spec, precision=args.precision, outputs=outs, f_ext=fx,
                           iirf_max=args.iirf_max, gas_form=None if args.general_kernel else "auto")
    vform, vgpl, vmw = plan.kernel_variant()
    loop_variant = plan.loop_variant
    flops_step = algorithmic_flops(plan.gas_form if not args.general_kernel else (0,) * N_GAS)
    assert args.sparse or flops_step == FLOPS_PER_STEP
    res = plan.result
    reducer = D.StatsReducer(plan)

    ev = lambda: torch.cuda.Event(enable_timing=True)
    kern_ev = [(ev(), ev()) for _ in range(args.steps)]

    def step(i=None):
        plan.reset_stats()
        if i is not None:
            kern_ev[i][0].record()
        plan.launch()                      # the fused integrator: the dominant kernel
        if i is not None:
            kern_ev[i][1].record()
        plan.stats_pass()                  # statistics pass over the T rows
        reducer.submit()                   # fold (+ with N > 1: the two all-reduces, on a side stream, under the next step)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 0)):
        step()
    reducer.wait()
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    e0, e1 = ev(), ev()
    e0.record()
    for i in range(args.steps):
        step(i)
    reducer.wait()                         # the last step's reduction is inside the timed region
    e1.record()
    barrier()
    clk = clocks.stop() if clocks else None
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    kms = torch.tensor([sum(a.elapsed_time(b) for a, b in kern_ev) / args.steps], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(kms, op=dist.ReduceOp.MAX)
    total_ms, kernel_ms = float(ms.item()), float(kms.item())
    ms_per_step = total_ms / args.steps
    units_per_step = float(M) * n_t * n_gpus
    value = units_per_step / (ms_per_step * 1e-3)

    # sanity on the result of the last step (cheap, outside the timed region)
    if spec is not None:
        assert bool((res.hist.sum(dim=1) == M * n_gpus).all()), "histogram rows must count every member"
    if res.T is not None:
        assert bool(torch.isfinite(res.T[-1]).all())
    if args.dump_outputs and rank == 0:
        pick = lambda names: {k: getattr(res, k) for k in names if getattr(res, k) is not None}
        dump_outputs(args.dump_outputs, pick(("C", "RF", "T", "state")), pick(("hist", "moments")))

    line = {"metric": METRIC, "value": value, "unit": "member-timesteps/s", "n_gpus": n_gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": args.precision, "data": "synthetic", "config": workload_config(args, n_gpus),
            # per step: stats_reset, ufair_integrate_kernel, stats_pass, stats_finalize[_packed] (+ stats_unpack with N > 1)
            "gpu_launches": ((4 if world == 1 else 5) if spec is not None else 1) * args.steps,
            "kernel_ms_per_launch": kernel_ms}

    peaks = None
    es = 8 if args.precision == "f64" else 4
    if rank == 0:
        line["clocks"] = clk
        peaks = measured_peaks(L, _abi)
        line["peaks"] = peaks
        # ---- roofline of the dominant kernel (ufair_integrate_kernel), measured live
        bytes_step = (N_GAS + 2 * N_GAS + 1) * es
        roof = roofline_of(kernel_ms, float(M) * n_t, bytes_step, flops_step, peaks, args.precision)
        traffic, traffic_src = None, None  # DRAM bytes per launch: NOT measured in this run (that needs ncu)
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(args.precision)
            if tj and spec is not None and outs == ("C", "RF", "T") and not args.sparse:
                traffic = tj["bytes_per_member_step"] * float(M) * n_t
                traffic_src = "not measured in this run: scaled from the committed ncu --set full capture (%s), %.2f B per member-step" % (
                    tj.get("capture", "profiles/"), tj["bytes_per_member_step"])
        except Exception:
            pass
        bound = "fp64" if args.precision == "f64" else "fp32"
        fpeak = peaks[bound + "_tflops"]
        a_hbm = bytes_step * float(M) * n_t / (kernel_ms * 1e-3) / 1e9
        a_fp = flops_step * float(M) * n_t / (kernel_ms * 1e-3) / 1e12
        roof.update({
            "traffic": traffic, "traffic_source": traffic_src,
            "kernel": "ufair_integrate_kernel<%s,3,EXP>" % ("double" if es == 8 else "float"),
            "kernel_ms": kernel_ms, "kernel_share_of_step": kernel_ms / ms_per_step,
            "algorithmic_bytes_per_member_step": bytes_step, "algorithmic_flops_per_member_step": flops_step,
            "kernel_variant": {"form": list(vform), "gases_per_lane": vgpl, "members_per_warp": vmw, "loop": loop_variant},
            "hbm": {"achieved": a_hbm, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": a_hbm / peaks["hbm_gbs"],
                    "peak_source": peaks["hbm_source"]},
            bound: {"achieved": a_fp, "peak": fpeak, "unit": "TFLOP/s", "frac": a_fp / fpeak,
                    "peak_burst": peaks[bound + "_tflops_burst"], "frac_of_burst": a_fp / peaks[bound + "_tflops_burst"],
                    "peak_source": peaks["fma_source"]},
        })
        # The FMA peak is measured by a pure DFMA / FFMA loop, which draws less power than the integrator and therefore
        # runs at a higher clock under the board's power cap.  `frac` stays against that measured peak; this entry only
        # says how much of the gap is the clock (informational).
        try:
            per_sm = 128.0 if bound == "fp64" else 256.0      # FMA flops per cycle and SM: 64 FP64 / 128 FP32 lanes
            implied = fpeak * 1e12 / (torch.cuda.get_device_properties(local).multi_processor_count * per_sm) / 1e6
            if clk and clk.get("sm_mhz"):
                roof["clock_note"] = {"peak_measured_at_mhz": implied, "kernel_ran_at_mhz": clk["sm_mhz"],
                                      "frac_of_pipe_at_kernel_clock": (a_fp / fpeak) * implied / float(clk["sm_mhz"]),
                                      "what": "the pipe peak scaled to the SM clock sampled during the timed region (median, nvidia-smi)"}
        except Exception:
            pass
        line["roofline"] = roof
    del plan, res, reducer
    torch.cuda.empty_cache()

    # ---- hardware evidence that the reduced statistics do not depend on the GPU count (SURVEY.md 8e)
    if world > 1 and spec is not None:
        try:
            ok = canary_bitwise(torch, dist, conc, D, spec, rank, world)
            if rank == 0:
                line["multi_gpu_bitwise"] = ok
        except Exception as exc:
            if rank == 0:
                line["multi_gpu_bitwise"] = {"error": repr(exc)}

    # ---- the same shard with literature-style (sparse) parameters: one-pool CH4 / N2O, one forcing term
    # per gas, on the specialised kernel the library picks for them.  Secondary figure; the headline
    # above keeps the dense parameters, where nothing can be skipped.
    side = (rank == 0 and world == 1 and not args.sparse and not args.general_kernel and spec is not None
            and not args.fext and args.iirf_max is None and outs == ("C", "RF", "T") and args.precision == "f64")
    if side and not args.no_lit:
        try:
            from fiveeqscm_b200 import params as P
            gp2, tp2, _, _ = P.sample_on_device(M, 20261018, dense_pools=False, precision="f64")
            plan2 = conc.DevicePlan(E, gp2.contiguous(), tp2.contiguous(), stats=spec, precision=args.precision, outputs=outs)
            ms2, _ = time_launches(torch, plan2, 5, warm=3)
            fl2 = algorithmic_flops(plan2.gas_form)
            line["literature_parameters"] = {
                "what": "same shard and outputs, CH4 / N2O with one pool and the sqrt term only, CO2 four pools and "
                        "the log term: integrator launches only",
                "kernel_ms": ms2, "value": float(M) * n_t / (ms2 * 1e-3), "unit": "member-timesteps/s",
                "kernel_variant": variant_of(plan2), "algorithmic_flops_per_member_step": fl2,
                "frac_of_fp64_peak": fl2 * float(M) * n_t / (ms2 * 1e-3) / 1e12 / peaks["fp64_tflops"]}
            del plan2, gp2, tp2
            torch.cuda.empty_cache()
        except Exception as exc:  # never lose the headline line to the secondary figure
            line["literature_parameters"] = {"error": repr(exc)}

    # ---- e2e: the public host-buffer API, pinned host inputs, H2D + kernel + D2H of every output
    if not args.no_e2e:
        row_bytes = (N_GAS * n_t + N_GAS * 17 + 4) * es + ((2 * N_GAS + 1) * n_t + 18) * es   # host bytes per member
        auto = {1: 786432, 2: 786432, 4: 393216}.get(world, 262144)
        Me = M if args.e2e_members == 0 else min(args.e2e_members if args.e2e_members > 0 else auto, M)
        try:
            avail = [int(ln.split()[1]) * 1024 for ln in open("/proc/meminfo") if ln.startswith("MemAvailable")][0]
            fit = int(avail / 3 / world / row_bytes) // 1024 * 1024
            if fit < Me:
                Me = max(fit, 16384)
        except Exception:
            pass
        hdt = torch.float64 if args.precision == "f64" else torch.float32
        t_pin = time.perf_counter()
        def pin(x):   # page-locked host copy in the run's precision, filled straight from the device (no pageable detour)
            h = torch.empty(x.shape, dtype=hdt, pin_memory=True)
            h.copy_(x)
            return h
        Eh, gph, tph = pin(E[:, :, :Me]), pin(gp[:, :, :Me]), pin(tp[:, :Me])
        outs_e = ("C", "RF", "T")
        out = conc.pinned_result(N_GAS, n_t, Me, outputs=outs_e, stats=spec, precision=args.precision)
        t_pin = time.perf_counter() - t_pin
        del E
        torch.cuda.empty_cache()
        ws = conc.Workspace(local, args.e2e_chunk)
        call = lambda: conc.run_ensemble(Eh, gph, tph, stats=spec, outputs=outs_e, precision=args.precision,
                                         workspace=ws, out=out)
        call()  # warm-up: staging allocation
        h2d = (N_GAS * n_t + N_GAS * 17 + 4) * Me * es
        d2h = ((2 * N_GAS + 1) * n_t + 18) * Me * es + (n_t * spec.bins * 8 + n_t * 32 if spec is not None else 0)

        # the link ceiling, measured now, with every rank copying at once: pitched copies of the pipeline's shape,
        # both directions together in the pipeline's byte ratio, and each direction alone
        g2, secs = (ctypes.c_double * 2)(), ctypes.c_double()
        rows = N_GAS * n_t

        def probe(up, down, reps=4):
            if world > 1:
                dist.barrier()
            _abi.check(L.ufair_link_probe(local, up // rows * rows, down // rows * rows, rows, reps, g2, secs))
            v = torch.tensor([g2[0], g2[1], secs.value], device="cuda", dtype=torch.float64)
            if world > 1:
                allv = [torch.zeros_like(v) for _ in range(world)]
                dist.all_gather(allv, v)
                v = torch.stack(allv)
            else:
                v = v[None]
            return v.cpu().numpy()
        unit = 192 << 20
        up_b, down_b = int(unit * h2d / d2h), unit
        # long enough that the ranks' start skew after the barrier (milliseconds) does not let the early ones see an idle
        # link: 0.8 GB per direction at N = 1 (15 ms), 6 GB at N = 8 (0.4 s at the ~15 GB/s a rank gets there)
        reps = 4 * world
        mix = probe(up_b, down_b, reps)
        solo_up, solo_down = probe(unit, 0, reps), probe(0, unit, reps)
        L.ufair_link_probe(local, 0, 0, 0, 1, g2, None)
        t_mix = float(mix[:, 2].max())                         # the slowest rank sets the step, as in e2e
        mix_value = float(Me) * n_t * n_gpus / (t_mix * (d2h / (down_b // rows * rows * float(reps))))
        # the ceiling proper: no pipeline can beat the busier direction moving its bytes at the rate that direction
        # reaches ALONE with every rank copying (aggregate over ranks: all of them have to finish)
        per_probe = float(unit // rows * rows) * reps
        agg_up = world * per_probe / float(solo_up[:, 2].max())
        agg_down = world * per_probe / float(solo_down[:, 2].max())
        ceiling_value = float(Me) * n_t * n_gpus / max(world * d2h / agg_down, world * h2d / agg_up)

        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            r = call()
            if world > 1 and spec is not None:
                hh, mm = torch.from_numpy(r.hist).cuda(), torch.from_numpy(r.moments).cuda()
                D.allreduce_stats(hh, mm)
                torch.cuda.synchronize()
        mine = time.perf_counter() - t0
        el = torch.tensor([mine], device="cuda", dtype=torch.float64)
        if world > 1:
            allt = [torch.zeros_like(el) for _ in range(world)]
            dist.all_gather(allt, el)
            times = torch.stack(allt).cpu().numpy().ravel()
        else:
            times = el.cpu().numpy().ravel()
        t_max = float(times.max())
        e2e_value = float(Me) * n_t * n_gpus * args.e2e_steps / t_max
        triple = lambda col: [float(col.min()), float(col.max()), float(col.sum())]
        line["e2e"] = {
            "value": e2e_value, "unit": "member-timesteps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "members_per_gpu": Me, "steps": args.e2e_steps, "cpu_binding": binding, "pin_seconds": t_pin,
            "pcie_ceiling_gbs": {
                "what": "ufair_link_probe, all %d rank(s) copying at once, pitched copies of %d rows; [slowest rank, fastest rank, sum over ranks]" % (world, rows),
                "h2d_alone": triple(solo_up[:, 0]), "d2h_alone": triple(solo_down[:, 1]),
                "h2d_in_pipeline_mix": triple(mix[:, 0]), "d2h_in_pipeline_mix": triple(mix[:, 1])},
            "ceiling_value": ceiling_value, "frac_of_ceiling": e2e_value / ceiling_value,
            "mix_estimate_value": mix_value, "frac_of_mix_estimate": e2e_value / mix_value,
            "achieved_gbs_per_rank": {"d2h_min": d2h * args.e2e_steps / float(times.max()) / 1e9,
                                      "d2h_max": d2h * args.e2e_steps / float(times.min()) / 1e9,
                                      "h2d_min": h2d * args.e2e_steps / float(times.max()) / 1e9,
                                      "h2d_max": h2d * args.e2e_steps / float(times.min()) / 1e9},
            "what": "run_ensemble(host pinned E/params -> all of C, RF, T, state + histogram back on the host), "
                    "chunked %d members, H2D/kernel/D2H overlapped on 3 streams; wall clock, max over ranks; "
                    "ceiling_value = the busier direction's bytes at the aggregate rate that direction reaches alone with all "
                    "ranks copying, measured just before (an upper bound: no interference between the directions); "
                    "mix_estimate_value = the same bytes at the rates of a probe that drives both directions flat out at once in "
                    "the pipeline's %.2f : 1 down : up ratio (pessimistic: the pipeline's copy-in is spread out)" % (args.e2e_chunk, d2h / h2d)}
        # secondary: the configs[3] use case proper -- host inputs in, only the ensemble statistics back
        # (histogram + moments; no trajectory leaves the GPU), same chunked pipeline
        if spec is not None:
            try:
                out2 = conc.pinned_result(N_GAS, n_t, Me, outputs=(), stats=spec, precision=args.precision, return_state=False)
                call2 = lambda: conc.run_ensemble(Eh, gph, tph, stats=spec, outputs=(), precision=args.precision,
                                                  workspace=ws, out=out2, return_state=False)
                call2()
                barrier()
                t0 = time.perf_counter()
                for _ in range(args.e2e_steps):
                    call2()
                el2 = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(el2, op=dist.ReduceOp.MAX)
                v2 = float(Me) * n_t * n_gpus * args.e2e_steps / float(el2.item())
                line["e2e_statistics_only"] = {
                    "value": v2, "unit": "member-timesteps/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": n_t * spec.bins * 8 + n_t * 32,
                    "frac_of_h2d_ceiling": v2 / (float(solo_up[:, 0].min()) * 1e9 * world / (h2d / (float(Me) * n_t))),
                    "what": "same host inputs, outputs=(): only the per-step T histogram and moments return to the host"}
            except Exception as exc:
                line["e2e_statistics_only"] = {"error": repr(exc)}
        # secondary: the same ensemble the way configs[3] would be fed in production -- the emissions ARE scenario rows
        # times a per-member scale, so the host holds the 4-scenario table, an index and a scale per member and the
        # parameters; nothing else crosses the link, only the statistics come back
        if spec is not None and not args.sparse:
            try:
                ws.close()
                chunk3 = conc.auto_chunk_members(N_GAS, n_t, e_member=False, fext_member=False, outputs=(), return_state=False,
                                                 e_scale=True, precision=args.precision)   # what run_ensemble picks by itself
                ws = conc.Workspace(local, chunk3)
                from fiveeqscm_b200 import params as P
                gp3, tp3, esc3, idx3 = P.sample_on_device(Me, 20261018, first_member=rank * M, n_scen=4, dense_pools=True,
                                                          precision=args.precision)
                scen_h = torch.from_numpy(P.scenario_emissions(n_t)).to(hdt).pin_memory()
                gp3h, tp3h, esc3h = pin(gp3), pin(tp3), pin(esc3)
                idx3h = torch.empty(idx3.shape, dtype=torch.int32, pin_memory=True); idx3h.copy_(idx3)
                out3 = conc.pinned_result(N_GAS, n_t, Me, outputs=(), stats=spec, precision=args.precision, return_state=False)
                call3 = lambda: conc.run_ensemble(scen_h, gp3h, tp3h, scen_idx=idx3h.numpy(), e_scale=esc3h, stats=spec, outputs=(),
                                                  precision=args.precision, workspace=ws, out=out3, return_state=False)
                call3()
                barrier()
                t0 = time.perf_counter()
                for _ in range(args.e2e_steps):
                    call3()
                el3 = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
                if world > 1:
                    dist.all_reduce(el3, op=dist.ReduceOp.MAX)
                up3 = (N_GAS * 17 + 4 + N_GAS) * Me * es + Me * 4 + N_GAS * n_t * 4 * es
                line["e2e_scenario_inputs"] = {
                    "value": float(Me) * n_t * n_gpus * args.e2e_steps / float(el3.item()), "unit": "member-timesteps/s",
                    "h2d_bytes_per_step": up3, "d2h_bytes_per_step": n_t * spec.bins * 8 + n_t * 32,
                    "what": "host inputs = scenario table [3][n_t][4] + per-member scenario index, emission scale and parameters "
                            "(%.2f B per member-step), outputs = per-step histogram and moments; chunks of %d members (the library's own choice for a "
                            "kernel-bound call), the first ones shorter" % (up3 / (float(Me) * n_t), chunk3)}
                del gp3, tp3, esc3, idx3
            except Exception as exc:
                line["e2e_scenario_inputs"] = {"error": repr(exc)}
        ws.close()
        del Eh, gph, tph, out
    else:
        del E
    torch.cuda.empty_cache()

    # ---- the other BASELINE.json configurations (N = 1)
    if side and not args.no_configs:
        line["configs"] = other_configs(torch, conc, peaks, spec, args.configs_scale)

    # ---- CPU baseline: the loop on this box's cores, fixed bounded sample of the same workload
    if rank == 0 and world == 1 and not args.no_cpu:   # reported at N = 1 only
        Ec, gpc, tpc = cpu_sample(n_t, not args.sparse)
        fast, textbook, thr, reps = cpu_rates(Ec, gpc, tpc, args.cpu_seconds)
        line["cpu_baseline"] = {
            "value": fast, "unit": "member-timesteps/s", "cores": thr, "kind": "port", "host_cpus": os.cpu_count(),
            "sample": "%d members x %d steps x %d passes: blocked + vectorised C rendering of the loop "
                      "(oracle/ufair_oracle_fast.c: 64-member tiles, libmvec, OpenMP)" % (CPU_SAMPLE_MEMBERS, n_t, reps),
            "textbook_scalar_loop": {"value": textbook, "what": "oracle/ufair_oracle.c, the parity checker, same threads"}}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        emit(line)


if __name__ == "__main__":
    main()
