"""The JSON lines bench.py printed on the B200 (committed under profiles/) carry every
key of the driver's contract; keeps the line format from drifting.  (bench.py itself
needs a GPU; its output is what can be checked here.)"""

import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
             "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "e2e",
             "clocks", "gpu_launches"}


def _line(name):
    text = open(os.path.join(ROOT, "profiles", name)).read().strip().splitlines()[-1]
    return json.loads(text)


@pytest.mark.parametrize("name,n", [("r01_bench_n1.json", 1), ("r01_bench_n2.json", 2),
                                    ("r01_bench_n4.json", 4), ("r01_bench_n8.json", 8),
                                    ("r02_bench_n1_call3.json", 1), ("r02_bench_n1_final.json", 1),
                                    ("r02_bench_n2.json", 2),
                                    ("r02_bench_n4_gpus0-3.json", 4), ("r02_bench_n8.json", 8)])
def test_our_arm_line(name, n):
    d = _line(name)
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    assert d["n_gpus"] == n and d["unit"] == "GB/s" and d["higher_is_better"] is True
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "u8"
    assert d["data"] == "synthetic" and "workload" in d["config"] and "l2" in d["config"]
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["e2e"]["d2h_bytes_per_step"] == 16_060_522_496
    assert 0 < d["e2e"]["value"] <= d["value"] * 1.02      # e2e cannot beat the raw path
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r)
    assert r["bound"] == "hbm" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["frac"] >= 0.70                                  # north_star: >= 70 % of the HBM roofline
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown",
                                               "sw_thermal_slowdown"}
    if n == 1:
        c = d["cpu_baseline"]
        assert {"value", "unit", "cores", "kind", "sample"} <= set(c) and c["kind"] == "port"
        assert d["stall_ms"]["async"] < 50.0                  # north_star: < 50 ms stall
    if name.startswith("r02"):
        assert r["traffic_source"].startswith("static:")      # a committed capture, says so
        if n == 1:
            fresh = d["restore_fresh_process"]
            assert fresh["ours"]["bit_exact_probe"] and fresh["reference_style"]["bit_exact_probe"]
            assert fresh["ours"]["restore_call_s"] < 1.0 < fresh["reference_style"]["restore_call_s"]
        else:
            coop = d["ddp_cooperative"]
            assert coop["image_matches_replicas"] and coop["restore"]["bit_exact_spot_check"]
            # n PCIe links instead of one: the ONE image lands faster than over a single link
            assert coop["ms_per_save"] < coop["single_link_reference_policy_ms"]
            if d.get("fsdp"):
                assert d["fsdp"]["segment_matches_local_shards"]
    # whole-job aggregate: per-rank PCIe Gen5 x16 cannot exceed ~58 GB/s
    assert d["value"] / n < 58.0


def test_reference_arm_runs_on_every_rank():
    """The N-rank reference arm is like for like: every rank runs the reference's loop."""
    d = _line("r02_bench_reference_n2.json")
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["ranks_run"] == 2
    assert d["cpu_baseline"]["cores"] == 2


def test_reference_arm_line():
    d = _line("r01_bench_reference.json")
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["metric"] == _line("r01_bench_n1.json")["metric"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["e2e"]["value"] == d["value"]
    assert {"kind", "cores", "sample", "value"} <= set(d["cpu_baseline"])


def test_dump_segment_is_bit_exact_seeded_and_bounded(tmp_path, monkeypatch):
    """--dump-outputs: bf16 words come back widened bit-exactly to float32; a segment larger
    than the sample is sampled at the same positions every time."""
    import sys

    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    t = torch.randn(1000, dtype=torch.float32).to(torch.bfloat16)
    buf = bytearray(t.view(torch.uint16).numpy().tobytes())
    bench.dump_segment(str(tmp_path / "a"), "seg", buf)
    got = np.load(tmp_path / "a" / "seg.npy")
    assert got.dtype == np.float32 and np.array_equal(got, t.float().numpy())

    monkeypatch.setattr(bench, "DUMP_WORDS", 64)
    big = bytearray(np.arange(5000, dtype=np.uint16).tobytes())
    for d in ("b", "c"):
        bench.dump_segment(str(tmp_path / d), "seg", big)
    b, c = np.load(tmp_path / "b" / "seg.npy"), np.load(tmp_path / "c" / "seg.npy")
    assert b.shape == (64,) and np.array_equal(b.view(np.uint32), c.view(np.uint32))
    words = b.view(np.uint32) >> 16
    assert np.all(np.diff(words.astype(np.int64)) >= 0) and words.max() < 5000
