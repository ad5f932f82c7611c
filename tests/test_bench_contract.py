"""bench.py: the workloads follow BASELINE.json's configs, the pair sharding is a partition, the reference arm (`--impl reference`,
the CPU restatement on the host cores) prints a line with every key of the measurement contract, and `--dump-outputs` writes what
the timed path computed (on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_workloads_follow_baseline_configs():
    import bench
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert bench.METRIC.startswith("flow_residual_constraints_per_sec") and "constraints/sec" in base["metric"]
    wl = bench.WORKLOADS
    spec2 = wl["config2_300f_384x224_grid16x12_sep10"]
    assert (spec2["frames"], spec2["w"], spec2["h"], spec2["gx"], spec2["gy"], spec2["sep"]) == (300, 384, 224, 16, 12, 10)      # configs[1]
    assert wl["config3_300f_384x224_grid16x12_sep10_maskratio0.20"]["mask_ratio"] == 0.20                                       # configs[2]
    s4 = wl["config4_1000f_640x384_grid32x24_sep10_huber"]
    assert (s4["frames"], s4["w"], s4["h"], s4["gx"], s4["gy"]) == (1000, 640, 384, 32, 24) and s4["cfg"]["robust_type"] == bench.abi.ROBUST_HUBER   # configs[3]
    assert wl["config5_300f_384x224_grid16x12_sep10_holes50_dolly"]["scene"]["hole_fraction"] > 0                                # configs[4]
    # config 1 builds in a blink: records, pair list and medians have consistent shapes; the overlap filter and the holes act
    spec, sc, cfg, pairs, offs, rec, med = bench.build_case("config1_8f_128x96_grid4x4_sep10")
    assert rec.shape[1] == 6 and offs[-1] == rec.shape[0] and len(pairs) == len(offs) - 1 == 30 and med.shape == (8,)
    from robust_cvd_b200 import synthetic
    fast = synthetic.Scene(40, 128, 96, seed=2, rot_deg=6.0, motion=0.15)
    kept = fast.filtered_pairs(0.2)
    assert 0 < len(kept) < len(synthetic.hierarchical2_pairs(40)) and all(fast.mask_ratio(a, b) > 0.2 for a, b in kept[:5])
    holes = synthetic.Scene(6, 128, 96, seed=2, hole_fraction=0.29, dolly=0.008)
    py, px = np.mgrid[0:96, 0:128]
    assert 0.55 < holes.visible(3, px.ravel(), py.ravel()).mean() < 0.85
    assert holes.constraints(sep=10)[2].shape[0] < 0.8 * synthetic.Scene(6, 128, 96, seed=2, dolly=0.008).constraints(sep=10)[2].shape[0]


def test_pair_sharding_is_a_balanced_partition():
    import bench
    spec, sc, cfg, pairs, offs, rec, med = bench.build_case("config1_8f_128x96_grid4x4_sep10")
    seen = []
    counts = []
    for r in range(3):
        lp, lo, lr = bench.shard_pairs(pairs, offs, rec, r, 3)
        seen += [tuple(p) for p in lp]; counts.append(lr.shape[0])
        assert lo[-1] == lr.shape[0]
    assert sorted(seen) == sorted(tuple(p) for p in pairs) and sum(counts) == rec.shape[0]
    assert max(counts) - min(counts) <= np.diff(offs).max()


def test_dump_outputs_keeps_a_fixed_sample_under_the_limit(tmp_path, monkeypatch):
    import bench
    rng = np.random.default_rng(1)
    arrays = {"a": rng.normal(size=(100, 30)), "b": rng.normal(size=(100, 30)).astype(np.float32), "costs": np.array([2.0, 1.0])}
    bench.dump_outputs(str(tmp_path / "full"), arrays)
    assert sorted(os.listdir(tmp_path / "full")) == ["a.npy", "b.npy", "costs.npy"]
    np.testing.assert_array_equal(np.load(tmp_path / "full" / "a.npy"), arrays["a"])
    assert np.load(tmp_path / "full" / "b.npy").dtype == np.float64
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4096 + 20 * (2 * 30 * 8 + 8) + 16)       # room for 20 of the 100 frames
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    got = {f: np.load(tmp_path / "s1" / f) for f in os.listdir(tmp_path / "s1")}
    rows = got["sampled_frames.npy"].astype(int)
    assert len(rows) == 20 and np.all(np.diff(rows) > 0) and rows[-1] < 100
    np.testing.assert_array_equal(got["a.npy"], arrays["a"][rows]); np.testing.assert_array_equal(got["costs.npy"], arrays["costs"])
    assert sum(v.nbytes for v in got.values()) <= bench.DUMP_LIMIT_BYTES
    np.testing.assert_array_equal(np.load(tmp_path / "s2" / "sampled_frames.npy"), got["sampled_frames.npy"])


@pytest.mark.gpu
def test_bench_dumps_what_the_timed_steps_computed(tmp_path):
    """`--steps` sets the number of timed steps and `--dump-outputs` writes the arrays of the last one and of the last e2e call."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "config1_8f_128x96_grid4x4_sep10", "--steps", "4", "--warmup", "1",
                          "--skip-cpu", "--skip-pose-opt", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == 4
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(got) == ["candidate_state", "costs", "e2e_costs", "e2e_state", "gradient", "step"]
    stride = d["config"]["structure"]["stride"]
    for k in ("candidate_state", "e2e_state", "gradient", "step"):
        assert got[k].shape == (8, stride) and got[k].dtype == np.float64 and np.isfinite(got[k]).all(), k
    assert 0 < got["e2e_costs"][1] < got["e2e_costs"][0] and abs(got["costs"][0] - got["e2e_costs"][0]) <= 1e-11 * got["costs"][0]


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` needs no GPU: smallest workload, one step."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "config1_8f_128x96_grid4x4_sep10", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["kind"] == "port" and d["config"]["workload"].startswith("config1")
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
