"""CPU tests of the host-side logic: sharding plan, statistics post-processing, the
world_size-2 reduction over gloo, argument validation and the loud no-fallback behaviour."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from fiveeqscm_b200 import concentrations as conc
from fiveeqscm_b200 import dist as D
from fiveeqscm_b200 import params as P
from fiveeqscm_b200 import stats as S
from oracle import c_oracle as co
from oracle import ufair_oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_bounds_cover_and_align():
    for n in (0, 1, 127, 128, 129, 10_000, 10_000_000):
        for w in (1, 2, 4, 8):
            edges = [D.shard_bounds(n, w, r) for r in range(w)]
            assert edges[0][0] == 0 and edges[-1][1] == n
            for (lo, hi), (lo2, _) in zip(edges, edges[1:]):
                assert hi == lo2 and lo <= hi
            for lo, hi in edges[:-1]:
                assert lo % 128 == 0 and hi % 128 == 0
    lo, hi = D.shard_bounds(10_000_000, 8, 3)
    assert abs((hi - lo) - 1_250_000) <= 128
    with pytest.raises(ValueError):
        D.shard_bounds(10, 2, 2)


def test_percentiles_and_moments_postprocessing():
    rng = np.random.default_rng(0)
    T = rng.normal(2.0, 0.7, size=(5, 50_000))
    hist, mom = o.temperature_stats(T, -5.0, 25.0, 1024)
    pct = S.percentiles(hist, -5.0, 25.0, [5, 50, 95])
    np.testing.assert_allclose(pct, o.percentiles_from_hist(hist, -5.0, 25.0, [5, 50, 95]))
    assert np.max(np.abs(pct - np.percentile(T, [5, 50, 95], axis=1).T)) < 2 * 30 / 1024
    mean, std = S.mean_std(mom, T.shape[1])
    np.testing.assert_allclose(mean, T.mean(axis=1), rtol=1e-12)
    np.testing.assert_allclose(std, T.std(axis=1), rtol=1e-9)


def test_shape_validation():
    sh = conc._shapes
    assert sh((3, 10, 8), (3, 17, 8), (4, 8), None, None, False) == (3, 10, 8, False, 1, 0)
    assert sh((3, 10, 4), (3, 17, 8), (4, 8), object(), (10, 4), False)[3:] == (True, 4, 1)
    assert sh((3, 10, 8), (3, 17, 8), (4, 8), None, (10, 8), True)[5] == 2
    with pytest.raises(ValueError):
        sh((3, 10, 8), (2, 17, 8), (4, 8), None, None, False)
    with pytest.raises(ValueError):
        sh((5, 10, 8), (5, 17, 8), (4, 8), None, None, False)
    with pytest.raises(ValueError):
        sh((3, 10, 8), (3, 17, 8), (4, 8), None, (9,), False)
    with pytest.raises(ValueError):
        conc._build_desc(3, 1, 1, 2, 1, False, 0, "exp", 0, "sideways", ("T",), 1.0, 100.0, None, None)


def test_default_parameters_are_sane():
    gp, tp = P.default_params(2)
    assert gp.shape == (3, 17, 2) and tp.shape == (4, 2)
    np.testing.assert_allclose(gp[:, 0:4].sum(axis=1), 1.0)
    ens = P.sample_ensemble(100, n_t=50, dense_pools=True)
    assert np.all(ens["gas_params"][:, 4:8] > 0) and np.all(ens["gas_params"][:, 14:17] != 0)
    np.testing.assert_allclose(ens["gas_params"][:, 0:4].sum(axis=1), 1.0, rtol=1e-12)
    E = P.scenario_emissions(736)
    assert E.shape == (3, 736, 4) and abs(E[0, 255, 1] - 10.0) < 0.2       # ~10 GtC/yr in 2020


def test_no_cpu_fallback_without_cuda():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    ens = P.sample_ensemble(4, n_t=3)
    E = P.member_emissions(ens["scen"], ens["scen_idx"], ens["e_scale"])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        conc.run_ensemble(E, ens["gas_params"], ens["thermal_params"])
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        conc.calculate_hfc_conc(np.array([10, 0]), np.array([0, 1]), 1.0)


def test_missing_library_fails_loudly(tmp_path):
    code = textwrap.dedent(f"""
        import sys; sys.path.insert(0, {ROOT!r})
        from fiveeqscm_b200 import _abi
        _abi._LIB_PATH = {str(tmp_path / 'nope.so')!r}
        try:
            _abi.lib()
        except ImportError as e:
            assert 'no CPU fallback' in str(e); print('LOUD')
    """)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert "LOUD" in out.stdout, out.stderr


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
from fiveeqscm_b200 import dist as D, params as P, stats as S
from oracle import c_oracle as co
rank, world = int(sys.argv[1]), int(sys.argv[2])
os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=sys.argv[3], RANK=str(rank), WORLD_SIZE=str(world))
dist.init_process_group("gloo", rank=rank, world_size=world)
M, n_t = 1000, 40
ens = P.sample_ensemble(M, n_t=n_t, seed=5)
E = P.member_emissions(ens["scen"], ens["scen_idx"], ens["e_scale"])
lo, hi = D.shard_bounds(M, world, rank)
# each rank integrates ITS members (here with the CPU checker standing in for the GPU kernel,
# which cannot run on this box) and builds its local statistics ...
T = co.oxfair(E[:, :, lo:hi], ens["gas_params"][:, :, lo:hi], ens["thermal_params"][:, lo:hi])["T"]
h, m = co.temperature_stats(T, -5.0, 25.0, 256)
hist = torch.from_numpy(h.astype(np.int64)); mom = torch.from_numpy(m)
# ... and the product's reduction combines them
D.allreduce_stats(hist, mom)
Tall = co.oxfair(E, ens["gas_params"], ens["thermal_params"])["T"]
h_all, m_all = co.temperature_stats(Tall, -5.0, 25.0, 256)
assert np.array_equal(hist.numpy().astype(np.uint64), h_all), "histogram not bitwise equal to single-rank"
assert np.allclose(mom.numpy()[:, :2], m_all[:, :2], rtol=1e-12)
assert np.array_equal(mom.numpy()[:, 2:], m_all[:, 2:])
dist.barrier(); dist.destroy_process_group()
print("RANK_OK", rank)
"""


def test_two_rank_gloo_reduction_matches_single_rank(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER.format(root=ROOT))
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), str(r), "2", port], stdout=subprocess.PIPE,
                              stderr=subprocess.PIPE, text=True) for r in range(2)]
    for r, p in enumerate(procs):
        out, err = p.communicate(timeout=300)
        assert p.returncode == 0 and f"RANK_OK {r}" in out, err[-2000:]


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm: the C oracle on the host cores) prints ONE JSON line
    with the contract's keys."""
    import json
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ensemble member-timesteps/sec" and d["value"] > 0
    assert d["higher_is_better"] is True and d["unit"] == "member-timesteps/s"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]
    assert "workload" in d["config"]


def test_gas_form_spelling_and_flop_convention():
    from fiveeqscm_b200 import _abi
    from fiveeqscm_b200.concentrations import _form_byte
    import bench
    assert _form_byte(None) == 0 and _form_byte(0) == 0
    assert _form_byte((1, "lin+sqrt")) == _abi.form(1, _abi.TERM_LIN | _abi.TERM_SQRT) == 0x61
    assert _form_byte((4, ("log",))) == 0x14 and _form_byte(0x21) == 0x21
    for bad in ((0, "lin"), (5, "lin"), (1, "cube"), 0x85, 0x06):
        with pytest.raises(ValueError):
            _form_byte(bad)
    # the survey's 751 flops per member-step is the four-pool, three-term case of the per-form count
    assert bench.algorithmic_flops((0, 0, 0)) == bench.FLOPS_PER_STEP == 751.0
    assert bench.algorithmic_flops((0x14, 0x41, 0x41)) == 236 + 2 * 102 + 13


def test_scenario_tables_and_summary_frames(tmp_path):
    import pandas as pd
    from fiveeqscm_b200 import frames
    from fiveeqscm_b200 import params as P
    from fiveeqscm_b200.concentrations import EnsembleResult, HistSpec
    from oracle import ufair_oracle as o
    n_t = 30
    scen = P.scenario_emissions(n_t)                                            # [3][n_t][4]
    rows = [dict(year=1765 + t, scenario=f"s{s}", co2=scen[0, t, s], ch4=scen[1, t, s], n2o=scen[2, t, s])
            for s in (2, 0, 1) for t in reversed(range(n_t))]                   # shuffled on purpose
    path = tmp_path / "scen.csv"
    pd.DataFrame(rows).to_csv(path, index=False)
    years, names, E, dt = frames.scenarios_from_csv(path)
    assert names == ["s2", "s0", "s1"] and dt == 1.0 and np.array_equal(years, 1765.0 + np.arange(n_t))
    assert np.allclose(E, scen[:, :, [2, 0, 1]], rtol=1e-15)
    with pytest.raises(ValueError):
        frames.scenarios_from_frame(pd.DataFrame(rows).drop(columns="ch4"))
    with pytest.raises(ValueError):
        frames.scenarios_from_frame(pd.DataFrame(rows[:-1]))                    # one scenario a year short
    with pytest.raises(ValueError):
        frames.scenarios_from_frame(pd.DataFrame([dict(year=y, co2=1, ch4=1, n2o=1) for y in (2000, 2001, 2003)]))
    # summaries from an (oracle-made) result
    gp, tp = P.sample_params(500, np.random.default_rng(0))
    run = o.oxfair(E, gp, tp, scen_idx=np.arange(500) % 3)
    spec = HistSpec(lo=-1.0, hi=4.0, bins=500)
    hist, mom = o.temperature_stats(run["T"], spec.lo, spec.hi, spec.bins)
    res = EnsembleResult(C=run["C"], RF=run["RF"], T=run["T"], hist=hist.astype(np.int64), moments=mom, spec=spec, n_member=500)
    sf = frames.summary_frame(res, years, pcts=(5, 50, 95))
    assert list(sf.columns) == ["year", "members", "T_mean", "T_std", "T_min", "T_max", "T_p5", "T_p50", "T_p95"]
    assert np.allclose(sf["T_mean"], run["T"].mean(axis=1), atol=1e-12) and np.all(sf["members"] == 500)
    assert np.all(sf["T_p5"] <= sf["T_p50"]) and np.all(sf["T_p50"] <= sf["T_p95"])
    assert np.max(np.abs(sf["T_p50"] - np.median(run["T"], axis=1))) < 2 * (spec.hi - spec.lo) / spec.bins
    mf = frames.member_frame(res, years, member=7)
    assert np.array_equal(mf["C_co2"], run["C"][0, :, 7]) and np.array_equal(mf["T"], run["T"][:, 7]) and "E_co2" not in mf
    with pytest.raises(ValueError):
        frames.summary_frame(EnsembleResult(T=run["T"]), years)


def test_host_side_form_detection_matches_the_device_rule():
    from fiveeqscm_b200 import _abi
    from fiveeqscm_b200 import params as P
    from fiveeqscm_b200.concentrations import _detect_form_host
    LOG, LIN, SQRT = _abi.TERM_LOG, _abi.TERM_LIN, _abi.TERM_SQRT
    gp, _ = P.sample_params(64, np.random.default_rng(1), ("co2", "ch4", "n2o", "hfc"))
    assert _detect_form_host(gp, None) == [_abi.form(4, LOG), _abi.form(1, SQRT), _abi.form(1, SQRT), _abi.form(1, LIN)]
    st = np.zeros((_abi.state_rows(4), 64))
    st[5 * 2 + 1, 3] = 1e-9                                  # N2O pool 2 carries mass in one member
    assert _detect_form_host(gp, st)[2] == _abi.form(2, SQRT)
    gpd, _ = P.sample_params(8, np.random.default_rng(1), dense_pools=True)
    assert _detect_form_host(gpd, None) == [_abi.form(4, LOG | LIN | SQRT)] * 3
    gp0 = np.array(gp[3:4]); gp0[0, _abi.GP_F2] = 0.0       # no forcing at all: the linear term stands in
    assert _detect_form_host(gp0, None) == [_abi.form(1, LIN)]


def test_numa_lookup_reads_sysfs(tmp_path):
    from fiveeqscm_b200 import dist as D
    assert D._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11} and D._parse_cpulist("") == set()
    dev = tmp_path / "bus/pci/devices/0000:1b:00.0"
    dev.mkdir(parents=True)
    (dev / "numa_node").write_text("1\n")
    node = tmp_path / "devices/system/node/node1"
    node.mkdir(parents=True)
    (node / "cpulist").write_text("32-63,96-127\n")
    n, cpus = D.numa_cpus_of_gpu(0, 0x1b, 0, sysfs=str(tmp_path))
    assert n == 1 and len(cpus) == 64 and 32 in cpus and 127 in cpus and 0 not in cpus
    (dev / "numa_node").write_text("-1\n")                          # single-socket host
    assert D.numa_cpus_of_gpu(0, 0x1b, 0, sysfs=str(tmp_path)) == (-1, set())
    assert D.numa_cpus_of_gpu(0, 0x99, 0, sysfs=str(tmp_path)) == (-1, set())     # unknown device


def test_vendored_reference_test_file_is_verbatim():
    """tests/golden/ref_test_hfcs.py is the reference's tests/unit/test_hfcs.py, byte for byte, as pinned by its
    sha256 (test infrastructure: the GPU suite runs the FILE against this repo's U_FaIR package)."""
    import hashlib
    here = os.path.dirname(os.path.abspath(__file__))
    data = open(os.path.join(here, "golden", "ref_test_hfcs.py"), "rb").read()
    assert hashlib.sha256(data).hexdigest() == "5eeed8cd25a7b55f38006f3f6e3baa3a3fb5910040da14d71b5ab49e355e1d64"


def test_shape_validation_of_scenario_inputs():
    """ADVICE r1: e_scale must be [G][M] (a short array would be read past its end by the copy loop), and a
    member axis that is neither M nor backed by scen_idx is an error, not a silent scenario run."""
    from fiveeqscm_b200.concentrations import _shapes
    G, n_t, M = 3, 10, 64
    ok = _shapes((G, n_t, 4), (G, 17, M), (4, M), object(), None, False, (G, M))
    assert ok[3] is True and ok[4] == 4
    for bad in ((M,), (1, M), (G, M - 1), (G + 1, M)):
        with pytest.raises(ValueError, match="e_scale"):
            _shapes((G, n_t, 4), (G, 17, M), (4, M), object(), None, False, bad)
    with pytest.raises(ValueError, match="e_scale"):
        _shapes((G, n_t, M), (G, 17, M), (4, M), None, None, False, (G, M))      # per-member emissions: no scale
    with pytest.raises(ValueError, match="scen_idx"):
        _shapes((G, n_t, 5), (G, 17, M), (4, M), None, None, False)              # 5 columns, 64 members, no index
    assert _shapes((G, n_t, 1), (G, 17, M), (4, M), None, None, False)[3] is True   # one shared column is fine
    assert _shapes((G, n_t, M), (G, 17, M), (4, M), None, None, False)[3] is False


def test_any_nonzero_and_auto_chunk_choice():
    """The host-side form scan answers dense rows from their first element and all-zero rows in one pass, with the
    answers of the plain comparison; the host pipeline's own chunk choice is small for link-bound calls and large for
    kernel-bound ones."""
    from fiveeqscm_b200 import concentrations as api
    rng = np.random.default_rng(3)
    for row in (np.zeros(1000), np.ones(1000), np.r_[np.zeros(999), 1e-300], np.r_[0.0, rng.standard_normal(5)], np.zeros(0),
                np.array([-0.0, 0.0]), np.array([np.nan])):
        assert api._any_nonzero(row) == bool(np.any(row != 0))
    full = api.auto_chunk_members(3, 736, e_member=True, fext_member=False, outputs=("C", "RF", "T"))
    stats_only = api.auto_chunk_members(3, 736, e_member=True, fext_member=False, outputs=(), return_state=False)
    t_only = api.auto_chunk_members(3, 736, e_member=False, fext_member=False, outputs=("T",), return_state=False, e_scale=True)
    scenario = api.auto_chunk_members(3, 736, e_member=False, fext_member=False, outputs=(), return_state=False, e_scale=True)
    scenario32 = api.auto_chunk_members(3, 736, e_member=False, fext_member=False, outputs=(), return_state=False, e_scale=True,
                                        precision="f32")
    assert (full, stats_only, t_only) == (16384, 16384, 16384) and scenario == 131072 and scenario32 == 131072
    short = api.auto_chunk_members(3, 10, e_member=False, fext_member=False, outputs=(), return_state=False)
    assert short == 16384     # ten steps: the parameters going up outweigh the integration
