"""Per-tile adaptive sampling, measured (one GPU process; writes JSON lines).

1. Overhead of RM_FLAG_MOMENTS on the bench frame (GoldDragon stand-in, 1920x1080, 500 spp, scene resident): frames rendered
   alternately without and with the flag; CUDA-event time of the accumulator kernel (stage kind 3, RM_FLAG_STAGE_TIMING) and
   of the whole frame.
2. Adaptive against uniform on GoldDragon (stand-in) and ReflectiveSpheres at 1920x1080, sample_count 500, samples_per_iteration
   16, thresholds 0.05 / 0.02 / 0.01: fraction of samples rendered, wall time of render_tiled + await, and the RMSE (8-bit
   levels) of the tonemapped frame against a 4096-spp frame of another seed, next to the RMSE of a uniform render with the
   same number of samples.

    python scripts/adaptive_bench.py --out /tmp/r3_adaptive.jsonl [--small]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from raymond_b200 import api as A  # noqa: E402
from raymond_b200 import fixtures as F  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def scene_of(name: str, small: bool) -> A.Scene:
    if name == "reflective_spheres":
        return A.Scene.from_fixture(F.reflective_spheres())
    objs = F.gold_dragon(F.dragon_standin(160, 40) if small else F.dragon_standin())
    s = A.Scene()
    for o in objs:
        if o[0] == "sphere":
            s.push_sphere(o[1], o[2], A.Material.from_fixture(o[3]))
        elif o[0] == "plane":
            s.push_plane(o[1], o[2], A.Material.from_fixture(o[3]))
        else:
            s.push_grid(A.AccGrid.build_from_mesh(A.Mesh.new(o[1]), device=0), A.Material.from_fixture(o[2]))
    return s


def moments_overhead(scene, W, H, spp, frames):
    st = A.Settings(A.CameraSettings.from_fixture(F.camera(W, H)), spp, (32, 32), 5)
    ds = A.DeviceScene(scene, 0)
    runs = {0: [], A.FLAG_MOMENTS: []}
    rs = {f: A.Renderer(ds, st, A.GpuOptions(seed=1, flags=A.FLAG_STAGE_TIMING | f)) for f in runs}
    for r in rs.values():           # warm-up frame
        r.render(0, spp)
        r.sync()
    for i in range(frames):
        for f, r in rs.items():
            before, acc0 = r.stats()["device_ms"], r.stage_stats()["ms"]["accumulate"][0]
            r.clear()
            r.render(0, spp)
            r.sync()
            runs[f].append({"frame_ms": r.stats()["device_ms"] - before, "accumulate_ms": r.stage_stats()["ms"]["accumulate"][0] - acc0})
    for r in rs.values():
        r.close()
    out = {}
    for f, label in ((0, "default"), (A.FLAG_MOMENTS, "moments")):
        fr = [x["frame_ms"] for x in runs[f]]
        ac = [x["accumulate_ms"] for x in runs[f]]
        out[label] = {"frame_ms": fr, "accumulate_ms": ac, "frame_ms_median": float(np.median(fr)), "accumulate_ms_median": float(np.median(ac))}
    out["frame_overhead_pct"] = 100.0 * (out["moments"]["frame_ms_median"] / out["default"]["frame_ms_median"] - 1.0)
    out["accumulate_overhead_ms"] = out["moments"]["accumulate_ms_median"] - out["default"]["accumulate_ms_median"]
    return out


def timed(scene, st, seed, adaptive=None):
    t0 = time.perf_counter()
    task = A.render_tiled(scene, st, A.GpuOptions(seed=seed), adaptive)
    frame = task.await_()
    wall = time.perf_counter() - t0
    return frame, task.stats(), wall


def rmse8(a, b) -> float:
    return float(np.sqrt(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)))


def adaptive_vs_uniform(scene, name, W, H, spp, spi, ref_spp, thresholds):
    cam = A.CameraSettings.from_fixture(F.camera(W, H))
    ref, _, ref_wall = timed(scene, A.Settings(cam, ref_spp, (32, 32), 5), seed=1000)
    ref8 = A.tonemap(ref)
    st = A.Settings(cam, spp, (32, 32), 5, spi)
    timed(scene, st, seed=1)                                 # warm-up of this frame layout
    uni, ustats, uwall = timed(scene, st, seed=1)
    rows = [{"scene": name, "mode": "uniform", "spp": spp, "samples": ustats["samples"], "fraction": 1.0, "wall_s": uwall,
             "rmse8_vs_ref": rmse8(A.tonemap(uni), ref8)}]
    for tau in thresholds:
        frame, stats, wall = timed(scene, st, seed=1, adaptive=A.AdaptiveSettings(tau, 2 * spi))
        eq_spp = max(1, int(round(stats["samples"] / (W * H))))
        eq, estats, ewall = timed(scene, A.Settings(cam, eq_spp, (32, 32), 5, spi), seed=1)
        rows.append({"scene": name, "mode": "adaptive", "threshold": tau, "min_samples": 2 * spi, "spp": spp, "samples": stats["samples"],
                     "fraction": stats["samples"] / float(W * H * spp), "wall_s": wall, "rmse8_vs_ref": rmse8(A.tonemap(frame), ref8),
                     "equal_samples_uniform": {"spp": eq_spp, "samples": estats["samples"], "wall_s": ewall, "rmse8_vs_ref": rmse8(A.tonemap(eq), ref8)}})
    rows.append({"scene": name, "mode": "reference", "spp": ref_spp, "seed": 1000, "wall_s": ref_wall})
    return rows


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True)
    p.add_argument("--small", action="store_true", help="a tiny run of the whole script (check that it works end to end)")
    a = p.parse_args()
    W, H, spp, ref_spp, frames = (192, 108, 32, 128, 2) if a.small else (1920, 1080, 500, 4096, 4)
    info = card()
    lines = []
    dragon = scene_of("gold_dragon", a.small)
    rec = {"measurement": "moments_overhead", "scene": "gold_dragon_standin", "width": W, "height": H, "spp": spp, **info}
    rec.update(moments_overhead(dragon, W, H, spp, frames))
    lines.append(rec)
    print(json.dumps(rec), flush=True)
    for name in ("gold_dragon", "reflective_spheres"):
        sc = dragon if name == "gold_dragon" else scene_of(name, a.small)
        for row in adaptive_vs_uniform(sc, name, W, H, spp, 16 if not a.small else 4, ref_spp, (0.05, 0.02, 0.01)):
            row.update({"measurement": "adaptive_vs_uniform", "width": W, "height": H, **info})
            lines.append(row)
            print(json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for r in lines:
            f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()
