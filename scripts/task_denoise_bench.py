"""The filter on the task path (rm_render_tiled_denoised), measured (one process; writes JSON lines, each with the card's name and
power limit read in the same run).

Scene: the GoldDragon stand-in at 1920x1080 and 500 spp, on 1, 2, 4 and 8 GPUs (device_count; counts above the GPUs of the box are
written as "not measured"), plus two shares on GPU 0 (device_list [0, 0]: the sliced filter's data path on a one-GPU box).

1. e2e: host time of render_tiled(...).await_() for the plain task and for denoised tasks (1 and 3 passes), alternated, tracing
   off.  A denoised task is finished once its filtered frame is on the host, so the difference is the whole cost: Q and the feature
   sums kept on every share, plus the filter.
2. filter: from the raw frame on the host to the filtered frame on the host, from the driver's RM_TRACE marks ("accumulators
   summed, frame on the host" -> "denoised frame on the host"), in separate traced runs.
3. one GPU only: Renderer.read_denoised on a renderer that rendered the same samples, host time of the call, next to the task's
   filter time; and whether the two frames are equal bit for bit.

    python scripts/task_denoise_bench.py [--out profiles/r6_task_denoise.jsonl] [--reps 4]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from raymond_b200 import api as A  # noqa: E402
from raymond_b200 import fixtures as F  # noqa: E402

W, H, SPP, SEED = 1920, 1080, 500, 2026
TRACE = re.compile(r"\[rm_trace\]\s+([0-9.]+) ms\s+(.*)")


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [l for l in q.stdout.splitlines() if l.strip()]
    name, power = [x.strip() for x in rows[0].split(",")]
    return {"gpu": name, "power_limit": power, "gpus_on_box": len(rows)}


def settings():
    return A.Settings(A.CameraSettings.from_fixture(F.camera(W, H)), SPP, (32, 32), 5)


def options(devices):
    return A.GpuOptions(seed=SEED, device_list=devices)


def e2e(scene, st, devices, denoise):
    t0 = time.perf_counter()
    task = A.render_tiled(scene, st, options(devices), denoise=denoise)
    task.await_()
    return (time.perf_counter() - t0) * 1e3, task


def traced_filter_ms(scene, st, devices, denoise):
    """(raw frame on the host -> filtered frame on the host) from the driver's trace marks, and the task."""
    os.environ["RM_TRACE"] = "1"
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as log:
        os.dup2(log.fileno(), 2)
        try:
            task = A.render_tiled(scene, st, options(devices), denoise=denoise)
            task.stats()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["RM_TRACE"]
        log.seek(0)
        marks = {}
        for line in log:
            m = TRACE.match(line.strip())
            if m:
                marks[m.group(2)] = float(m.group(1))
    return marks["driver: denoised frame on the host"] - marks["driver: devices done, accumulators summed, frame on the host"], task


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_task_denoise.jsonl"))
    p.add_argument("--reps", type=int, default=4)
    args = p.parse_args()
    info = card()
    scene = A.Scene.from_fixture(F.gold_dragon(F.dragon_standin()))
    st = settings()
    configs = [("gpus1", None), ("shares2_on_gpu0", [0, 0])] + [(f"gpus{g}", list(range(g))) for g in (2, 4, 8)]
    variants = {"plain": None, "denoise_1": A.DenoiseSettings(1), "denoise_3": A.DenoiseSettings(3)}
    with open(args.out, "w") as out:
        def emit(row):
            out.write(json.dumps(row) + "\n")
            out.flush()
            print(json.dumps(row), flush=True)

        for name, devices in configs:
            if devices and max(devices) >= info["gpus_on_box"]:
                emit(dict(info, kind="e2e", config=name, result="not measured", reason=f"{len(set(devices))} GPUs needed"))
                continue
            for v in variants.values():                  # warm-up of every variant
                e2e(scene, st, devices, v)
            times = {k: [] for k in variants}
            for _ in range(args.reps):
                for k, v in variants.items():
                    times[k].append(e2e(scene, st, devices, v)[0])
            med = {k: float(np.median(t)) for k, t in times.items()}
            emit(dict(info, kind="e2e", config=name, devices=devices or [0], size=f"{W}x{H}", spp=SPP, reps=args.reps, ms_median=med, ms_all=times,
                      denoise_1_over_plain=med["denoise_1"] / med["plain"] - 1.0, denoise_3_over_plain=med["denoise_3"] / med["plain"] - 1.0))
            for k in ("denoise_1", "denoise_3"):
                ms = []
                for _ in range(args.reps):
                    t, task = traced_filter_ms(scene, st, devices, variants[k])
                    ms.append(t)
                row = dict(info, kind="filter", config=name, devices=devices or [0], size=f"{W}x{H}", spp=SPP, iterations=variants[k].iterations,
                           reps=args.reps, raw_to_filtered_ms_median=float(np.median(ms)), raw_to_filtered_ms_all=ms)
                if devices is None:
                    # the old one-renderer path on the same samples: one renderer, the whole frame in one call
                    r = A.Renderer(scene, st, A.GpuOptions(seed=SEED, flags=A.FLAG_AOV | A.FLAG_MOMENTS))
                    r.render(0, SPP)
                    r.sync()
                    r.read_denoised(SPP, variants[k])
                    host = []
                    for _ in range(args.reps):
                        t0 = time.perf_counter()
                        frame = r.read_denoised(SPP, variants[k])
                        host.append((time.perf_counter() - t0) * 1e3)
                    r.close()
                    row.update(read_denoised_ms_median=float(np.median(host)), read_denoised_ms_all=host,
                               task_frame_equals_read_denoised=bool(np.array_equal(task.await_denoised().view(np.uint64), frame.view(np.uint64))))
                emit(row)


if __name__ == "__main__":
    main()
