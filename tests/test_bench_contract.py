"""bench.py prints exactly one JSON line on stdout with the keys the driver reads (both arms)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--width", "160", "--height", "90", "--spp", "4", "--steps", "1", "--warmup", "1", "--cpu-seconds", "0.5", "--c3-spp", "2", "--c5-spp", "2"]
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
             "config", "e2e", "gpu_launches", "cpu_baseline"}


def run_bench(extra):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + SMALL + extra, capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, f"stdout must hold exactly one line, got {len(lines)}"
    return json.loads(lines[0])


def test_reference_arm_line():
    """--impl reference: the oracle port on the host cores; runs without a GPU."""
    line = run_bench(["--impl", "reference"])
    assert BASE_KEYS <= set(line) and line["impl"] == "reference"
    assert line["unit"] == "Msamples/s" and line["higher_is_better"] is True and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"] + SMALL, capture_output=True, text=True,
                         cwd=ROOT, env=env, timeout=120)
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_bench_rejects_what_it_cannot_time_or_dump():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, cwd=ROOT, timeout=120)
        assert res.returncode == 2 and "error" in res.stderr, extra


def test_dump_frame_samples_a_large_frame_the_same_way_every_time(tmp_path, monkeypatch):
    import bench
    frame = np.random.default_rng(5).random((20, 30, 3))
    bench.dump_frame(str(tmp_path / "whole"), frame)
    assert np.array_equal(np.load(tmp_path / "whole" / "frame.npy"), frame)
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * 24)
    bench.dump_frame(str(tmp_path / "a"), frame)
    bench.dump_frame(str(tmp_path / "b"), frame.copy())
    a, b = np.load(tmp_path / "a" / "frame.npy"), np.load(tmp_path / "b" / "frame.npy")
    assert a.shape == (100, 3) and a.dtype == np.float64 and np.array_equal(a, b)
    rows = [int(np.nonzero((frame.reshape(-1, 3) == p).all(axis=1))[0][0]) for p in a]
    assert rows == sorted(set(rows))                       # distinct pixels of the frame, in pixel order


@pytest.mark.gpu
def test_dumped_frame_is_the_same_for_any_number_of_steps(tmp_path):
    """--dump-outputs writes the last timed step's frame; every step renders the same seeded frame, so --steps does not change
    it, while the timed region holds exactly --steps frames' worth of kernel launches."""
    quick = ["--no-extras", "--no-e2e", "--no-cpu-baseline"]
    one = run_bench(quick + ["--dump-outputs", str(tmp_path / "one")])
    three = run_bench(quick + ["--steps", "3", "--dump-outputs", str(tmp_path / "three")])
    assert (one["steps"], three["steps"]) == (1, 3)
    assert one["gpu_launches"] > 0 and three["gpu_launches"] == 3 * one["gpu_launches"]
    assert three["rays_per_path"] == one["rays_per_path"]
    a, b = np.load(tmp_path / "one" / "frame.npy"), np.load(tmp_path / "three" / "frame.npy")
    assert a.shape == (90, 160, 3) and a.dtype == np.float64 and np.isfinite(a).all() and a.max() > 0
    assert np.array_equal(a, b)
    assert np.allclose(a.mean(axis=(0, 1)), one["mean_radiance"], rtol=1e-12, atol=0)


@pytest.mark.gpu
def test_gpu_arm_line():
    line = run_bench([])
    assert BASE_KEYS | {"clocks", "roofline"} <= set(line) and "impl" not in line
    assert line["n_gpus"] == 1 and line["dtype"] == "f64" and line["data"] == "synthetic" and line["vs_baseline"] is None
    assert line["scaling"] == "strong"
    assert line["gpu_launches"] > 0 and line["value"] > 0 and line["e2e"]["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] == 160 * 90 * 24
    r = line["roofline"]
    assert r["bound"] in ("issue", "hbm") and r["peak"] > 0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["unit"] == ("Gwarp-inst/s" if r["bound"] == "issue" else "GB/s")
    # the contract's HBM roofline on algorithmic bytes and the other ceilings, as flat keys the driver keeps
    assert r["hbm_peak_gbs"] > 0 and abs(r["hbm_frac"] - r["hbm_achieved_gbs"] / r["hbm_peak_gbs"]) < 1e-9
    assert all(not isinstance(v, (dict, list)) for v in r.values())
    c = line["cpu_baseline"]
    assert c["kind"] == "port" and c["value"] > 0 and c["cores"] >= 1 and "spp" in c["sample"]
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"])
    oc = line["other_configs"]
    assert oc["c3_reflective_spheres_dof_1920x1080_tiles"]["seconds"] > 0 and oc["c5_gold_dragon_3840x2160_progressive"]["seconds"] > 0
    # both arms describe the workload with the SAME config dict
    ref = run_bench(["--impl", "reference"])
    assert ref["config"] == line["config"] and ref["metric"] == line["metric"] and ref["unit"] == line["unit"]
