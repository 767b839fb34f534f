"""Cost of colour textures, measured (one GPU process; writes JSON lines).

The open GoldDragon stand-in (floor, red sphere, dragon; no walls) under the procedural sky of fixtures.sky(), at 1920x1080,
bounce limit 5, rendered by two renderers whose frames alternate:
    plain     the scene without textures
    textured  a 2048 x 1024 texture on the dragon (its surface parameter as uv, fixtures.dragon_standin(uv=True)) and a
              64 x 64 checker tiled on the floor (scale 2 per unit); the colours are those of the plain scene's materials
Per variant: Msamples/s from the CUDA-event time of the frame (frames without RM_FLAG_STAGE_TIMING), and per-stage k_shade and
total times from a second set of frames with RM_FLAG_STAGE_TIMING.

    python scripts/texture_bench.py --out /tmp/r10_texture.jsonl [--spp 64] [--frames 5] [--small]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from raymond_b200 import api as A  # noqa: E402
from raymond_b200 import fixtures as F  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def dragon_texture(W: int = 2048, H: int = 1024) -> np.ndarray:
    """Stripes along the tube and rings around it, values in [0.35, 1]."""
    u = (np.arange(W) + 0.5) / W
    v = (np.arange(H) + 0.5) / H
    U, V = np.meshgrid(u, v)
    a = 0.5 + 0.5 * np.sin(2.0 * np.pi * 40.0 * U)
    b = 0.5 + 0.5 * np.cos(2.0 * np.pi * 8.0 * V)
    img = np.stack([0.35 + 0.65 * a, 0.35 + 0.65 * b, 0.35 + 0.65 * a * b], axis=-1)
    return np.ascontiguousarray(img, dtype=np.float32)


def floor_texture(n: int = 64) -> np.ndarray:
    c = (np.indices((n, n)).sum(axis=0) // 8) % 2
    return np.ascontiguousarray(np.stack([0.3 + 0.7 * c] * 3, axis=-1), dtype=np.float32)


def open_dragon(small: bool, sky, textured: bool) -> A.Scene:
    s = A.Scene()
    for o in F.open_dragon(F.dragon_standin(160, 40, uv=True) if small else F.dragon_standin(uv=True)):
        if o[0] == "sphere":
            s.push_sphere(o[1], o[2], A.Material.from_fixture(o[3]))
        elif o[0] == "plane":
            s.push_plane(o[1], o[2], A.Material.from_fixture(o[3]))
        else:
            s.push_grid(A.AccGrid.build_from_mesh(A.Mesh.new(o[1]), device=0), A.Material.from_fixture(o[2]))
    s.set_environment(sky)
    if textured:
        s.set_texture(1, dragon_texture(256, 128) if small else dragon_texture())
        s.set_texture(2, floor_texture(), scale=(2.0, 2.0))
    return s


def renderer(scene, st, flags):
    return A.Renderer(A.DeviceScene(scene, 0), st, A.GpuOptions(seed=1, flags=flags))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--spp", type=int, default=64)
    ap.add_argument("--frames", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="160x96 and a small mesh: a rehearsal of the script, not a measurement")
    a = ap.parse_args()
    W, H = (160, 96) if a.small else (1920, 1080)
    st = A.Settings(A.CameraSettings.from_fixture(F.camera(W, H)), a.spp, (32, 32), 5)
    sky = F.sky()
    variants = {"plain": open_dragon(a.small, sky, False), "textured": open_dragon(a.small, sky, True)}
    info = card()
    lines = []
    for timing in (0, A.FLAG_STAGE_TIMING):
        rs = {k: renderer(sc, st, timing) for k, sc in variants.items()}
        for r in rs.values():       # warm-up frame
            r.render(0, a.spp)
            r.sync()
        runs = {k: [] for k in rs}
        for _ in range(a.frames):
            for k, r in rs.items():
                before = r.stats()["device_ms"]
                shade0 = np.array(r.stage_stats()["ms"]["shade"])
                r.clear()
                r.render(0, a.spp)
                r.sync()
                runs[k].append((r.stats()["device_ms"] - before, np.array(r.stage_stats()["ms"]["shade"]) - shade0))
        for k, r in rs.items():
            frame = [x[0] for x in runs[k]]
            rec = {"variant": k, "stage_timing": bool(timing), "width": W, "height": H, "spp": a.spp, "bounce_limit": 5,
                   "sky": list(sky.shape[:2]), "frame_ms": frame, "frame_ms_median": float(np.median(frame)),
                   "msamples_per_s": W * H * a.spp / (float(np.median(frame)) * 1e-3) / 1e6, "rays": r.stats()["rays"], "upload_bytes": r.stats()["upload_bytes"], **info}
            if timing:
                shade = np.median(np.stack([x[1] for x in runs[k]]), axis=0)
                rec["shade_ms_by_depth"] = [float(x) for x in shade[1:6]]
                rec["shade_ms_total"] = float(shade.sum())
            lines.append(rec)
            r.close()
    with open(a.out, "w") as f:
        for rec in lines:
            f.write(json.dumps(rec) + "\n")
            print(json.dumps({k: v for k, v in rec.items() if k != "frame_ms"}))


if __name__ == "__main__":
    main()
