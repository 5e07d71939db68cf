"""bench.py contract (task statement, "Measurement"): the reference arm runs on the host here, the committed JSON line of
this repo's arm (profiles/r01_bench_v6.json, taken on a B200) carries every key the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline")


def test_reference_arm_prints_one_json_line_on_the_host():
    """`bench.py --impl reference` = the oracle port of main.py:161-291 on the host cores: one JSON line, impl=reference,
    the arm's own metric / unit, e2e == value with zero transfer bytes, no GPU launches."""
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "target nodes/sec (sample+train)" and d["unit"] == "nodes/s"
    for k in BASE_KEYS:
        assert k in d, k
    assert d["e2e"] == {"value": d["value"], "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["gpu_launches"] == 0 and d["higher_is_better"] is True and d["vs_baseline"] is None


def test_bench_rejects_zero_steps_and_dumps_of_the_reference_arm(tmp_path):
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path / "d")]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny"] + extra,
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert res.returncode == 2 and not res.stdout.strip(), res.stderr[-2000:]
    assert not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step_repeat_across_runs(cuda_device, tmp_path):
    """`--dump-outputs DIR`: the last timed step's losses, sampler statistics, sampled nodes, logits and updated parameters
    as float32 / float64 .npy files.  The optimisers counted prime + warm-up + `--steps` steps, the dumped batch holds the
    targets of the batch the last timed step ran (not those of the prefetched next one), and two runs with the same
    arguments dump the same numbers."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from grapes_b200.dist import shard_batches
    prime, warmup, steps = 2, 3, 4
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "small",
                              "--steps", str(steps), "--warmup", str(warmup), "--prime", str(prime), "--no-cpu-baseline",
                              "--no-spmm", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-4000:]
        d = json.loads(res.stdout.strip().splitlines()[-1])
        assert d["steps"] == steps and d["warmup"] == warmup and d["prime_steps"] == prime
        arrays = {p.stem: np.load(p) for p in sorted(out.glob("*.npy"))}
        assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
        assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
        dumps.append(arrays)
    a, b = dumps
    assert a.keys() == b.keys()
    for key in ("loss_c", "loss_gfn", "log_z", "tot_log_prob", "sampler_stats", "all_nodes", "logits_c", "adam_steps",
                "gcn_c.gcn_layers.0.lin.weight", "gcn_gf.gcn_layers.1.bias", "gcn_z.gcn_layers.1.lin.weight"):
        assert key in a, key
    assert a["adam_steps"].tolist() == [prime + warmup + steps] * 2
    # the batches in the order bench.py runs them (same seeded workload, warm-up and timed steps only)
    cfg, _, _, _, _, train_idx = bench.build_workload("small", 0, cuda_device)
    B = cfg["batch_size"]
    mine = shard_batches(train_idx.numel() // B, 0, 1)
    batch = lambda j: set(train_idx[mine[j % len(mine)] * B:(mine[j % len(mine)] + 1) * B].tolist())
    last = warmup + steps - 1
    dumped = set(a["all_nodes"].astype(np.int64).tolist())
    assert batch(last) <= dumped and not batch(last + 1) <= dumped and not batch(last - 1) <= dumped
    assert a["sampler_stats"].shape == (cfg["sampling_hops"], 4) and a["logits_c"].shape == (len(dumped), cfg["C"])
    for h in range(cfg["sampling_hops"]):
        s = a[f"sampled_hop{h}"]
        assert 0 < s.size <= cfg["num_samples"] and np.array_equal(s, np.round(s)) and set(s.astype(np.int64).tolist()) <= dumped
    assert np.isfinite(a["loss_c"]).all() and np.isfinite(a["logits_c"]).all()
    for key in a:
        assert np.array_equal(a[key], b[key]), key


def test_committed_bench_line_carries_the_contract():
    d = json.loads(open(os.path.join(ROOT, "profiles", "r01_bench_v6.json")).read().strip().splitlines()[-1])
    for k in BASE_KEYS + ("clocks", "roofline"):
        assert k in d, k
    assert d["metric"] == "target nodes/sec (sample+train)" and d["unit"] == "nodes/s" and d["scaling"] == "weak"
    assert "products" in d["config"]["workload"] and "l2_policy" in d["config"] and "model" not in d["config"]
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0
    e = d["e2e"]
    assert e["unit"] == "nodes/s" and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] < d["value"]
    r = d["roofline"]
    for k in ("bound", "achieved", "peak", "unit", "frac", "traffic", "kernel"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["unit"] == "nodes/s" and c["sample"]
    ck = d["clocks"]
    assert ck["sm_mhz"] > 0 and ck["sm_max_mhz"] >= ck["sm_mhz"] and isinstance(ck["reasons"], list)
    assert not set(ck["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_round2_bench_lines_carry_the_round2_keys():
    """Round-2 additions: per-rank step-time percentiles, the priming steps, where `traffic` was read from, how the gradient is
    exchanged; the 8-GPU line was taken under the driver's own command (--steps 20 --warmup 5)."""
    d = json.load(open(os.path.join(ROOT, "profiles", "r02_bench_v3.json")))
    for k in ("step_times", "prime_steps", "gradient_exchange", "rooflines", "clocks", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["n_gpus"] == 1 and len(d["step_times"]) == 1 and d["step_times"][0]["p50_ms"] > 0
    assert d["roofline"]["traffic_source"]["commit"] and d["roofline"]["traffic"] > 0
    assert d["e2e"]["value"] < d["value"] and d["launches_per_step"] == 69
    s = json.load(open(os.path.join(ROOT, "profiles", "r02_scale_products_n8_peer_20a.json")))
    assert s["n_gpus"] == 8 and s["steps"] == 20 and s["warmup"] == 5 and len(s["step_times"]) == 8
    assert "peer memory" in s["gradient_exchange"] and s["scaling"] == "weak"
    assert s["value"] > 6.5 * d["value"]                       # the north star's 8-GPU target against this round's 1-GPU line
    assert max(t["p50_ms"] for t in s["step_times"]) < 1.02 * min(t["p50_ms"] for t in s["step_times"])
