"""First-hit feature buffers and the a-trous denoiser, measured (one GPU process; writes JSON lines, each with the card's name and
power limit).

1. Cost of the flags: GoldDragon stand-in, 1920x1080, one 32-spp batch per call, renderers without flags, with RM_FLAG_MOMENTS and
   with RM_FLAG_AOV | RM_FLAG_MOMENTS on one resident scene, called in turn; host time of render + sync per batch.
2. Cost of the denoiser at 1920x1080: host time of read_denoised (kernels, D2H, conversion), CUDA events on the renderer's
   stream around the call, and the kernel times torch.profiler reports.
3. Benefit at 320x240 on GoldDragon (stand-in) and ReflectiveSpheres: RMSE (linear, clamped to [0, 10]) against a 4096-spp render
   of another seed, raw and denoised, at 4 / 16 / 64 spp; the raw spp whose RMSE matches the denoised 16-spp one; and a sweep of
   the filter settings at 16 spp, RMSE ratio and mean-luminance shift per setting (what the defaults in include/raymond.h were
   chosen from).

    python scripts/denoise_bench.py [--out profiles/r5_denoise.jsonl] [--reps 10]
"""
import argparse
import itertools
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

FLAGS = A.FLAG_AOV | A.FLAG_MOMENTS
LUMA = np.array([0.2126, 0.7152, 0.0722])


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power}


def settings(cam, spp):
    return A.Settings(A.CameraSettings.from_fixture(cam), spp, (32, 32), 5)


def rmse(a, b):
    return float(np.sqrt(np.mean((np.clip(a, 0.0, 10.0) - np.clip(b, 0.0, 10.0)) ** 2)))


def flag_cost(out, info, reps):
    ds = A.DeviceScene(A.Scene.from_fixture(F.gold_dragon(F.dragon_standin())))
    s = settings(F.camera(1920, 1080), 32)
    variants = {"none": 0, "moments": A.FLAG_MOMENTS, "aov_moments": FLAGS}
    rs = {k: A.Renderer(ds, s, A.GpuOptions(seed=2026, batch_spp=32, flags=f)) for k, f in variants.items()}
    times = {k: [] for k in variants}
    for rep in range(reps + 2):
        for k, r in rs.items():
            t0 = time.perf_counter()
            r.render(rep * 32, 32)
            r.sync()
            if rep >= 2:                     # two warm-up batches each
                times[k].append((time.perf_counter() - t0) * 1e3)
    med = {k: float(np.median(v)) for k, v in times.items()}
    row = dict(info, kind="flag_cost", scene="gold_dragon_standin", size="1920x1080", batch_spp=32, reps=reps,
               ms_per_batch_median=med, ms_per_batch_all=times,
               aov_overhead_vs_moments=med["aov_moments"] / med["moments"] - 1.0, aov_moments_overhead_vs_none=med["aov_moments"] / med["none"] - 1.0)
    out.write(json.dumps(row) + "\n")
    print(json.dumps({k: v for k, v in row.items() if k != "ms_per_batch_all"}), flush=True)
    for r in rs.values():
        r.close()


def denoise_time(out, info, reps):
    import torch
    stream = torch.cuda.Stream()
    scene = A.Scene.from_fixture(F.gold_dragon(F.dragon_standin()))
    r = A.Renderer(scene, settings(F.camera(1920, 1080), 32), A.GpuOptions(seed=2026, flags=FLAGS, stream=stream.cuda_stream))
    r.render(0, 32)
    r.sync()
    r.read_denoised(32)                      # warm-up
    host, event = [], []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        t0 = time.perf_counter()
        r.read_denoised(32)
        host.append((time.perf_counter() - t0) * 1e3)
        e1.record(stream)
        e1.synchronize()
        event.append(e0.elapsed_time(e1))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            r.read_denoised(32)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        if "k_atrous" in e.key or "k_denoise_pack" in e.key:
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            kernels["k_atrous" if "k_atrous" in e.key else "k_denoise_pack"] = {"calls": e.count, "us_per_read": t / reps}
    r.close()
    row = dict(info, kind="denoise_time", scene="gold_dragon_standin", size="1920x1080", iterations="default", reps=reps,
               host_ms_median=float(np.median(host)), event_ms_median=float(np.median(event)), kernels=kernels)
    out.write(json.dumps(row) + "\n")
    print(json.dumps(row), flush=True)


def quality(out, info):
    scenes = {"gold_dragon_standin": F.gold_dragon(F.dragon_standin()), "reflective_spheres": F.reflective_spheres()}
    cam = F.camera(320, 240)
    sweep = {}
    for name, objs in scenes.items():
        scene = A.DeviceScene(A.Scene.from_fixture(objs))
        ref = A.Renderer(scene, settings(cam, 4096), A.GpuOptions(seed=1))
        ref.render(0, 4096)
        reference = ref.read_frame(4096)
        ref.close()
        raw_rmse = {}
        den16 = None
        for spp in (4, 16, 64):
            r = A.Renderer(scene, settings(cam, spp), A.GpuOptions(seed=2, flags=FLAGS))
            r.render(0, spp)
            raw, den = r.read_frame(spp), r.read_denoised(spp)
            raw_rmse[spp] = rmse(raw, reference)
            row = dict(info, kind="quality", scene=name, size="320x240", spp=spp, reference_spp=4096, rmse_raw=raw_rmse[spp],
                       rmse_denoised=rmse(den, reference), ratio=rmse(den, reference) / raw_rmse[spp],
                       luma_reference=float((reference @ LUMA).mean()), luma_raw=float((raw @ LUMA).mean()), luma_denoised=float((den @ LUMA).mean()))
            out.write(json.dumps(row) + "\n")
            print(json.dumps(row), flush=True)
            if spp == 16:
                den16 = row["rmse_denoised"]
                sweep[name] = []
                for it, sc, sn, sa, sz in itertools.product((1, 2, 3, 5), (1.0, 4.0, 16.0, 1e3, 1e4), (0.1, 0.25, 0.5), (0.1, 0.3), (0.2, 1.0)):
                    d = r.read_denoised(16, A.DenoiseSettings(it, sc, sn, sa, sz))
                    sweep[name].append(((it, sc, sn, sa, sz), rmse(d, reference) / raw_rmse[16], float((d @ LUMA).mean()) / row["luma_raw"] - 1.0))
            r.close()
        ladder = {}
        for spp in (32, 128, 256, 512, 1024):
            r = A.Renderer(scene, settings(cam, spp), A.GpuOptions(seed=2))
            r.render(0, spp)
            ladder[spp] = rmse(r.read_frame(spp), reference)
            r.close()
        ladder.update(raw_rmse)
        matched = min((s for s, e in ladder.items() if e <= den16), default=None)
        row = dict(info, kind="match", scene=name, size="320x240", rmse_denoised_16spp=den16, raw_rmse_by_spp=dict(sorted(ladder.items())),
                   first_measured_raw_spp_at_or_below=matched, raw_spp_estimate_1_over_sqrt=16.0 * (raw_rmse[16] / den16) ** 2)
        out.write(json.dumps(row) + "\n")
        print(json.dumps(row), flush=True)
    names = list(sweep)
    rows = []
    for k in range(len(sweep[names[0]])):
        s = sweep[names[0]][k][0]
        rows.append(dict(settings=dict(zip(("iterations", "sigma_color", "sigma_normal", "sigma_albedo", "sigma_depth"), s)),
                         ratio={n: sweep[n][k][1] for n in names}, luma_shift={n: sweep[n][k][2] for n in names}))
    # the bars of tests/test_gpu_denoise.py: RMSE <= 0.6 x raw and mean luminance within 1 % of raw, on both scenes
    passes = lambda r: max(r["ratio"].values()) <= 0.6 and max(abs(x) for x in r["luma_shift"].values()) <= 0.01
    rows.sort(key=lambda r: (not passes(r), max(r["ratio"].values())))
    row = dict(info, kind="sweep", size="320x240", spp=16, reference_spp=4096, settings_tried=len(rows), settings_passing=sum(map(passes, rows)),
               results=rows)
    out.write(json.dumps(row) + "\n")
    print(json.dumps(row)[:3000], flush=True)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_denoise.jsonl"))
    p.add_argument("--reps", type=int, default=10)
    args = p.parse_args()
    info = card()
    with open(args.out, "w") as out:
        flag_cost(out, info, args.reps)
        denoise_time(out, info, args.reps)
        quality(out, info)


if __name__ == "__main__":
    main()
