"""The measurement contract of bench.py on a GPU, at a size that takes seconds: ONE JSON line with the roofline, cpu_baseline, e2e,
clocks and gpu_launches objects the driver reads (the CPU suite checks the reference arm, tests/test_abi.py)."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(arguments):
    result = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + arguments, capture_output=True, text=True, timeout=900)
    assert result.returncode == 0, result.stderr[-2000:]
    lines = [line for line in result.stdout.splitlines() if line.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def check_common(line):
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "roofline", "e2e", "gpu_launches", "clocks"):
        assert key in line, key
    assert line["n_gpus"] == 1 and line["warmup"] >= 3 and line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["gpu_launches"] > 0 and "workload" in line["config"] and "l2" in line["config"]
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in line["roofline"], key
    for key in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"):
        assert key in line["e2e"], key
    for key in ("sm_mhz", "sm_max_mhz", "reasons"):
        assert key in line["clocks"], key


def test_trace_bench_line():
    rays = 1 << 18
    line = run_bench(["--workload", "trace", "--steps", "2", "--quads", "128", "64", "--rays", str(rays), "--cpu-sample", "65536", "--no-secondary"])
    check_common(line)
    assert line["unit"] == "Mrays/s" and line["scaling"] == "weak" and line["dtype"] == "f32"
    roofline = line["roofline"]
    assert roofline["bound"] == "hbm" and roofline["unit"] == "GB/s" and roofline["achieved"] > 0
    assert roofline["frac"] == pytest.approx(roofline["achieved"] / roofline["peak"], rel=1e-6)
    assert line["e2e"]["value"] > 0 and line["e2e"]["h2d_bytes_per_step"] == 2 * rays * 32 and line["e2e"]["d2h_bytes_per_step"] == rays * 16 + rays
    assert line["gpu_launches"] == 2 * line["steps"]
    baseline = line["cpu_baseline"]
    assert baseline["kind"] == "port" and baseline["cores"] >= 1 and baseline["value"] > 0 and baseline["unit"] == "Mrays/s" and baseline["sample"]
    assert baseline["single_thread"]["value"] > 0 and baseline["single_thread"]["cores"] == 1
    assert roofline["frac_nominal_8tbs"] == pytest.approx(roofline["achieved"] / 8000.0, rel=1e-6)
    # the plugin-call leg from page-locked memory (echo_b200_host_alloc) and from pageable memory
    assert "page-locked" in line["e2e"]["host_memory"] and line["e2e_pageable"]["value"] > 0
    # the on-chip ceilings are measured live by the library and the same algorithmic bytes are set against them
    assert roofline["frac_l2"] == pytest.approx(roofline["achieved"] / roofline["l2_peak_gbs"], rel=1e-6) and roofline["l2_peak_gbs"] > 0
    assert roofline["l1_sector_peak_gbs"] > 0 and "L1" in roofline["bound_measured"]
    # the device SweepBuilder beside the host mirror of the recursive build: the same bytes
    build = line["tree_build"]
    assert build["identical_to_host_mirror"] and build["nodes"] == line["config"]["tree"]["nodes"] and build["device_build_ms"] > 0 and build["host_mirror_ms"] > 0


def check_render_record(record, width, height, spp):
    assert record["unit"] == "samples/s" and record["scaling"] == "strong" and record["value"] > 0
    assert record["samples_per_step"] == width * height * spp
    roofline = record["roofline"]
    assert roofline["achieved"] > 0 and roofline["frac"] == pytest.approx(roofline["achieved"] / roofline["peak"], rel=1e-6)
    assert roofline["algorithmic_bytes_per_sample"] == pytest.approx(sum(roofline["bytes_per_sample_parts"].values()), rel=1e-9)
    assert roofline["per_sample_counters"]["node_visits"] > 1 and roofline["per_sample_counters"]["trace_queries"] >= 1
    e2e = record["e2e"]
    assert e2e["value"] > 0 and e2e["d2h_bytes_per_step"] >= width * height * 16 and "echo_b200_render_tiles" in e2e["call"]
    assert record["rank_step_ms"]["min"] > 0 and len(record["rank_step_ms"]["per_rank"]) == 1 and record["all_reduce"]["count"] >= 1
    baseline = record["cpu_baseline"]
    assert baseline["kind"] == "port" and baseline["value"] > 0 and baseline["unit"] == "samples/s" and baseline["cores"] >= 1


def test_render_bench_line():
    line = run_bench(["--workload", "render", "--scene", "cornell", "--width", "256", "--height", "256", "--spp", "4", "--steps", "2", "--bounce-limit", "8"])
    check_common(line)
    check_render_record(line, 256, 256, 4)
    assert line["stats_last_step"]["Sample/Evaluated"] == 256 * 256 * 4


def test_default_line_carries_the_render_records(tmp_path):
    """`python bench.py` (the default run): the C2 headline plus `render.c1 / c3 / c4 / c5` with roofline, cpu_baseline and the
    plugin-call e2e, every record timed over --steps steps, and --dump-outputs writing the last step's outputs. Shrunk through the
    environment so that the whole default path runs in seconds."""
    environment = {**os.environ, "ECHO_BENCH_SHRINK": "1"}
    outputs = tmp_path / "outputs"
    result = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "6", "--quads", "128", "64", "--rays", str(1 << 18), "--cpu-sample", "65536", "--no-secondary",
                             "--dump-outputs", str(outputs)], capture_output=True, text=True, timeout=1200, env=environment)
    assert result.returncode == 0, result.stderr[-2000:]
    lines = [line for line in result.stdout.splitlines() if line.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    check_common(line)
    assert line["unit"] == "Mrays/s" and set(line["render"]) >= {"c1", "c3", "c4", "c5"}
    for key in ("c1", "c3", "c4", "c5"):
        record = line["render"][key]
        check_render_record(record, record["config"]["width"], record["config"]["height"], record["config"]["spp_per_step"])
    assert "all-reduce every 4" in line["render"]["c5"]["config"]["parallelism"] and line["render"]["c5"]["all_reduce"]["count"] == 2  # after step 4 and the last
    assert line["gpu_launches"] > 2 * line["steps"]
    assert all(line["render"][key]["steps"] == line["steps"] == 6 for key in ("c1", "c3", "c4", "c5"))

    import numpy as np
    from echorenderer_b200 import structs
    dumped = {path.stem: np.load(path) for path in outputs.iterdir()}
    assert set(dumped) == {"trace_token", "trace_distance", "trace_uv", "occluded", "frame_cornell", "frame_mixed", "frame_lights", "frame_large"}
    assert all(array.dtype in (np.float32, np.float64) and np.isfinite(array).all() for array in dumped.values()) and sum(array.nbytes for array in dumped.values()) <= 64 << 20
    rays = 1 << 18  # fewer than the sample size: every ray is kept, in order
    assert dumped["trace_token"].shape == dumped["trace_distance"].shape == dumped["occluded"].shape == (rays,) and dumped["trace_uv"].shape == (rays, 2)
    assert set(np.unique(dumped["occluded"])) <= {0.0, 1.0} and 0 < (dumped["trace_token"] != structs.TOKEN_EMPTY).sum() < rays
    miss = dumped["trace_token"] == structs.TOKEN_EMPTY
    assert (dumped["trace_distance"][miss] == -1).all() and (dumped["trace_distance"][~miss] >= 0).all()
    for key in ("c1", "c3", "c4", "c5"):
        config = line["render"][key]["config"]
        frame = dumped["frame_" + {"c1": "cornell", "c3": "mixed", "c4": "lights", "c5": "large"}[key]]
        assert frame.shape == (min(config["width"] * config["height"], 1 << 18), 4) and np.isfinite(frame).all() and frame[:, :3].max() > 0, key
