#!/usr/bin/env python
"""bench.py — GoldDragon 1920x1080, 500 spp, 5 bounces (BASELINE.json configs[1]) on N B200s.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference ...                    # the reference's algorithm on the host cores (the oracle port)
    python bench.py ... --dump-outputs DIR                  # also DIR/frame.npy, the frame of the last timed step (same seed, same inputs)

A step = one pass of the hot path over one frame: W*H*spp paths through camera ray generation,
Scene::intersect (sphere / planes / uniform-grid DDA), the BRDF bounce loop and the tile accumulator.
Metric: Msamples/s (paths per second, whole job).  The dragon mesh is missing from the reference
snapshot, so the scene uses the documented STAND-IN mesh (raymond_b200.fixtures.dragon_standin).

N > 1 (torchrun, one rank per GPU): STRONG scaling — the job stays the 1920x1080 x 500 spp frame; rank g renders
the global samples g, g+N, ... of every pixel and the per-rank f64 accumulators are summed onto rank 0 with an
NCCL reduce inside the timed region.  `e2e` is the same frame through the reference-facing call with host buffers:
render_tiled(scene, settings).await() — at N > 1 with rm_gpu_options.device_count = N, i.e. ONE process (rank 0)
driving the N GPUs through the C ABI, which is what a Rust caller of the FFI crate gets; the one-process-per-GPU
variant of the same frame is reported beside it as `e2e_torchrun`.  BASELINE configs[2] and configs[4] are timed at
the same N in `other_configs`, configs[3] (1 M-triangle soup, primary-hit query) at N = 1.

One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

METRIC = "Msamples/sec (paths x 5 bounces), GoldDragon 1920x1080 500 spp"
UNIT = "Msamples/s"
# Per-unit constants of the dominant kernel taken from the ncu --set full capture under profiles/ (dram bytes, warp instructions, ...):
# written by scripts/ncu_constants.py from the .ncu-rep and the bench line of the same command, never edited by hand.
NCU_CONSTANTS = os.path.join(ROOT, "profiles", "ncu_constants.json")

print_line = None


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--width", type=int, default=1920)
    p.add_argument("--height", type=int, default=1080)
    p.add_argument("--spp", type=int, default=500)
    p.add_argument("--bounces", type=int, default=5)
    p.add_argument("--scene", default="gold_dragon", choices=["gold_dragon", "reflective_spheres", "reflective_spheres_dof"])
    p.add_argument("--seed", type=int, default=2026)
    p.add_argument("--precision", default="f64", choices=["f64", "f32shade"],
                   help="arithmetic of the statistical scope (BRDF sampling / weights); the intersection code is always the reference's f64 sequence")
    p.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU work of the cpu_baseline sample")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-extras", action="store_true", help="skip BASELINE configs[2] / configs[4] (other_configs)")
    p.add_argument("--c3-spp", type=int, default=1000, help="samples of the configs[2] run in other_configs (tests shrink it)")
    p.add_argument("--c5-spp", type=int, default=4096, help="samples of the configs[4] run in other_configs (tests shrink it)")
    p.add_argument("--no-c4", action="store_true", help="skip the configs[3] leg of other_configs")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="write the frame of the last timed step to DIR/frame.npy (f64 H x W x 3; above 64 MB a fixed sample of its pixels)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        p.error("--dump-outputs records the CUDA path; the reference arm picks its sample count from its own speed")
    return args


def scene_objects(name):
    from raymond_b200 import fixtures as F
    if name == "gold_dragon":
        return F.gold_dragon(F.dragon_standin()), "GoldDragon (STAND-IN mesh, 871200 triangles; dragon_vrip.ply is missing from the reference snapshot)"
    if name == "reflective_spheres":
        return F.reflective_spheres(), "ReflectiveSpheres"
    return F.reflective_spheres(), "ReflectiveSpheres + aperture sampling (focal 2.5, radius 0.5)"


def camera_for(args):
    from raymond_b200 import fixtures as F
    if args.scene == "reflective_spheres_dof":
        return F.camera(args.width, args.height, focal_length=2.5, aperture_radius=0.5)
    return F.camera(args.width, args.height)


def config_of(args, label):
    """The workload description — the SAME dict from both arms (what each arm actually sampled goes into cpu_baseline.sample)."""
    return {"workload": f"{label} {args.width}x{args.height}, {args.spp} spp, {args.bounces} bounces", "scene": args.scene,
            "width": args.width, "height": args.height, "spp": args.spp, "bounces": args.bounces, "tile": [32, 32],
            "mesh": "stand-in" if args.scene == "gold_dragon" else "analytic",
            "parallelism": f"sample-split x{args.gpus} + ncclReduce(sum)" if args.gpus > 1 else "1 GPU",
            "l2": "inputs exceed L2 (scene ~290 MB + ~10 GB of wavefront queues per 16-spp batch); no explicit flush",
            "precision": args.precision}


# ------------------------------------------------------------------------------- clocks

class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons every 200 ms during the timed region (NVML)."""

    def __init__(self, device_index: int):
        super().__init__(daemon=True)
        self.idx = device_index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[device_index]) if vis and vis.split(",")[device_index].isdigit() else device_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            log(f"[bench] NVML unavailable: {e}")

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:  # noqa: BLE001
                pass
            self._stop_evt.wait(0.2)

    def finish(self) -> dict:
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------- CPU arm (oracle port)

def oracle_scene(objs):
    from oracle import oracle as O
    s = O.Scene()
    for o in objs:
        if o[0] == "sphere":
            s.add_sphere(o[1], o[2], o[3])
        elif o[0] == "plane":
            s.add_plane(o[1], o[2], o[3])
        else:
            s.add_grid(O.AccGrid.build_from_mesh(O.Mesh.from_triangles(o[1])), o[2])
    return s


def cpu_sample_plan(sc, cam, bounces, target_s, cores):
    """Pick a bounded sample (full frame, k spp) worth about `target_s` seconds of CPU work."""
    from oracle import oracle as O
    small = dict(cam, width=max(cam["width"] // 4, 16), height=max(cam["height"] // 4, 16))
    O.render(sc, small, 1, seed=1, bounce_limit=bounces, worker_count=cores)          # page-in / warm caches
    t0 = time.perf_counter()
    O.render(sc, small, 1, seed=2, bounce_limit=bounces, worker_count=cores)
    rate = small["width"] * small["height"] / (time.perf_counter() - t0)
    frame = cam["width"] * cam["height"]
    spp = int(max(1, min(64, round(rate * target_s / frame))))
    return spp, rate


def run_cpu(sc, cam, spp, bounces, cores, seed):
    from oracle import oracle as O
    t0 = time.perf_counter()
    _, cnt = O.render(sc, cam, spp, seed=seed, bounce_limit=bounces, worker_count=cores)
    dt = time.perf_counter() - t0
    return cnt["samples"] / dt / 1e6, dt, cnt


def bench_reference(args):
    """The reference's own algorithm on the host cores: the C++ oracle port (no rustc here, so the reference
    itself cannot be built), reference threading model (worker threads over a FIFO tile queue, 1 spp per pass)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    objs, label = scene_objects(args.scene)
    cam = camera_for(args)
    sc = oracle_scene(objs)
    per_step_target = max(2.0, min(20.0, 150.0 / max(args.steps + args.warmup, 1)))
    spp, _ = cpu_sample_plan(sc, cam, args.bounces, per_step_target, cores)
    for i in range(args.warmup):
        run_cpu(sc, cam, spp, args.bounces, cores, args.seed + i)
    t0 = time.perf_counter()
    n = 0
    for i in range(args.steps):
        _, _, cnt = run_cpu(sc, cam, spp, args.bounces, cores, args.seed + 100 + i)
        n += cnt["samples"]
    dt = time.perf_counter() - t0
    value = n / dt / 1e6
    sample = (f"each step = {cam['width']}x{cam['height']} x {spp} spp of the workload's frame on {cores} host threads (the full frame at reduced spp: "
              f"Msamples/s does not depend on spp); f64, -ffp-contract=off, the reference's threading model")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_of(args, label),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print_line(json.dumps(line))


# ------------------------------------------------------------------------------- GPU arm

def ncu_constants(kernel: str):
    try:
        return json.load(open(NCU_CONSTANTS)).get(kernel)
    except Exception:  # noqa: BLE001
        return None


def roofline_record(A, args, scene, settings, local, world, st0, st1, samples_rank0, clocks):
    """Roofline of the dominant kernel on rank 0: live CUDA-event time per (kernel, depth) over the timed region; algorithmic
    bytes / operations from an instrumented pass of the same rays (C cells visited, T triangle tests); DRAM bytes, warp
    instructions and cache hit rates per unit from the ncu capture under profiles/ (profiles/ncu_constants.json)."""
    W, H = args.width, args.height
    kinds = A.KERNEL_KINDS
    d_ms = {k: [b - a for a, b in zip(st0["ms"][k], st1["ms"][k])] for k in kinds}
    d_launch = {k: [b - a for a, b in zip(st0["launches"][k], st1["launches"][k])] for k in kinds}
    d_rays = [b - a for a, b in zip(st0["rays"], st1["rays"])]
    d_grid = [b - a for a, b in zip(st0["grid_rays"], st1["grid_rays"])]
    d_shtri = [b - a for a, b in zip(st0["shaded_triangles"], st1["shaded_triangles"])]
    counted = A.Renderer(scene, A.Settings(settings.camera_settings, 4, (32, 32), args.bounces),
                         A.GpuOptions(device=local, seed=args.seed, flags=A.FLAG_COUNT_WORK, batch_spp=4, precision=PRECISIONS[args.precision]))
    counted.render(0, 4)
    cs = counted.stage_stats()
    counted.close()
    total_ms = sum(sum(v) for v in d_ms.values())
    stages, per_kernel = [], {}
    kernel_bytes, kernel_flops = 0.0, 0.0
    for d in range(0, A.STAGE_SLOTS):
        for k in kinds:
            if d_launch[k][d] == 0:
                continue
            C_ = T_ = None
            if k == "accumulate":
                # reads 24 B per path, reads + writes 24 B per pixel per batch
                units, per_unit = samples_rank0, 24.0 + 48.0 * W * H * d_launch[k][d] / max(samples_rank0, 1)
            elif k == "setup":
                # ray in (48 B; depth 1 generates it and writes it instead) + hit record out (16 B) + a 128-B traversal record per grid ray
                units = d_rays[d]
                per_unit = 48.0 + 16.0 + 128.0 * d_grid[d] / max(d_rays[d], 1)
            elif k == "traverse":
                # SURVEY 8d: B(ray) = 64 + 8 C + 76 T  (48-B ray in, 16-B hit out, 8 B per visited cell, 4 + 72 B per triangle test)
                g_ = max(cs["grid_rays"][d], 1)
                C_, T_ = cs["cells"][d] / g_, cs["triangle_tests"][d] / g_
                units, per_unit = d_grid[d], 64.0 + 8.0 * C_ + 76.0 * T_
                # what THIS kernel has to move for the same decisions: 128-B record + 16-B hit, a 4-B occupancy word per cell, an 8-B record
                # per occupied cell, a 16-B bounding sphere + 4-B triangle index per candidate, the 96-B positions per candidate not proven a miss
                kernel_bytes += (144.0 + 4.0 * C_ + 8.0 * cs["occupied_cells"][d] / g_ + 20.0 * T_ + 96.0 * cs["evaluated_tests"][d] / g_) * d_grid[d]
                # f64 add/sub/mul/div this kernel executes per grid ray: 1 per cell step (t_max += t_delta), 19 per bounding-sphere
                # pre-test, and the counted exits (20 / 30 / 46 / 52) of the Triangle::intersects calls it evaluates
                kernel_flops += (C_ + 19.0 * T_ + cs["evaluated_test_flops"][d] / g_) * d_grid[d]
            else:
                # shade (+ the next depth's set-up when fused): ray + throughput + id + hit in (92 B), next ray out (76 B) or radiance out (24 B);
                # +144 B (positions, normals) per shaded triangle
                units = d_rays[d]
                cont = d_rays[d + 1] if d + 1 < A.STAGE_SLOTS and d < args.bounces else 0
                per_unit = 92.0 + (76.0 * cont + 24.0 * (d_rays[d] - cont) + 144.0 * d_shtri[d]) / max(d_rays[d], 1)
            bytes_total = per_unit * units
            ms_ = d_ms[k][d]
            stages.append({"kernel": "k_" + k, "depth": d, "ms": ms_, "launches": d_launch[k][d], "units": units,
                           "alg_bytes_per_unit": per_unit, "cells_per_ray": C_, "tests_per_ray": T_,
                           "achieved_gbs": bytes_total / (ms_ * 1e-3) / 1e9 if ms_ > 0 else None, "share": ms_ / max(total_ms, 1e-9)})
            pk = per_kernel.setdefault(k, {"ms": 0.0, "launches": 0, "bytes": 0.0, "units": 0})
            pk["ms"] += ms_; pk["launches"] += d_launch[k][d]; pk["bytes"] += bytes_total; pk["units"] += units
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    top = max(per_kernel, key=lambda k: per_kernel[k]["ms"])
    pk = per_kernel[top]
    secs = pk["ms"] * 1e-3
    hbm_ach = pk["bytes"] / secs / 1e9 if secs > 0 else 0.0
    nc = ncu_constants("k_" + top) or {}
    sms = 148
    try:
        import torch
        sms = torch.cuda.get_device_properties(local).multi_processor_count
    except Exception:  # noqa: BLE001
        pass
    mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965.0
    issue_peak = sms * 4 * mhz * 1e6 / 1e9                        # one warp instruction per scheduler per clock, G warp-inst/s
    rec = {"kernel": "k_" + top, "unit_name": "grid ray" if top == "traverse" else ("path" if top == "accumulate" else "ray"),
           "launch_ms_avg": pk["ms"] / max(pk["launches"], 1), "launches": pk["launches"], "share_of_step": pk["ms"] / max(total_ms, 1e-9),
           "units_per_launch": pk["units"] / max(pk["launches"], 1)}
    for k, v in per_kernel.items():
        rec["share_k_" + k] = v["ms"] / max(total_ms, 1e-9)
    # --- the HBM roofline the contract defines: ALGORITHMIC bytes of the reference's algorithm / time / measured copy bandwidth
    rec.update({"hbm_achieved_gbs": hbm_ach, "hbm_peak_gbs": hbm_peak, "hbm_frac": hbm_ach / hbm_peak, "hbm_peak_source": hbm_src,
                "alg_bytes_per_unit": pk["bytes"] / max(pk["units"], 1), "alg_bytes_per_launch": pk["bytes"] / max(pk["launches"], 1)})
    traffic = None
    if nc.get("dram_bytes_per_unit") is not None:
        traffic = nc["dram_bytes_per_unit"] * pk["units"] / max(pk["launches"], 1)
        rec["dram_bytes_per_unit_ncu"] = nc["dram_bytes_per_unit"]
        rec["dram_frac"] = nc["dram_bytes_per_unit"] * pk["units"] / secs / 1e9 / hbm_peak     # real DRAM traffic against the HBM peak
    if top == "traverse":
        rec["kernel_bytes_per_unit"] = kernel_bytes / max(pk["units"], 1)
        rec["kernel_bytes_frac_of_hbm"] = kernel_bytes / secs / 1e9 / hbm_peak
        fp64_peak = A.measure_fp64_rate(local)
        rec.update({"fp64_peak_gops": fp64_peak, "fp64_achieved_gops": kernel_flops / secs / 1e9, "fp64_frac": kernel_flops / secs / 1e9 / fp64_peak,
                    "fp64_ops_per_unit": kernel_flops / max(pk["units"], 1)})
    for key in ("l1_hit", "l2_hit", "threads_per_inst", "fp64_pipe_active", "issue_active_ncu", "registers", "source"):
        if key in nc:
            rec["ncu_" + key] = nc[key]
    # --- which ceiling binds.  The traversal set is L2-resident (DRAM at a few % of peak) and the arithmetic is 0.1 of the f64 rate:
    # the largest fraction is instruction issue, so that is the roofline reported in bound / achieved / peak / frac.
    if nc.get("warp_inst_per_unit") is not None:
        inst_ach = nc["warp_inst_per_unit"] * pk["units"] / secs / 1e9
        rec.update({"bound": "issue", "achieved": inst_ach, "peak": issue_peak, "unit": "Gwarp-inst/s", "frac": inst_ach / issue_peak,
                    "warp_inst_per_unit_ncu": nc["warp_inst_per_unit"],
                    "peak_source": f"{sms} SMs x 4 schedulers x {mhz:.0f} MHz (median SM clock sampled during the timed region), 1 warp instruction per scheduler per clock",
                    "note": "binding ceiling = instruction issue: warp instructions per unit (ncu smsp__inst_executed of the same kernel, profiles/) x units / live kernel time; "
                            "the contract's HBM roofline on algorithmic bytes is in hbm_achieved_gbs / hbm_peak_gbs / hbm_frac, real DRAM traffic in dram_frac, arithmetic in fp64_frac"})
    else:
        rec.update({"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak, "peak_source": hbm_src})
    rec["traffic"] = traffic
    return rec, stages


PRECISIONS = {"f64": 0, "f32shade": 1}
DUMP_BYTES = 60_000_000          # under 64 MB with the .npy header; a 1920x1080 f64 frame is 49.8 MB


def dump_frame(out_dir: str, frame: np.ndarray) -> None:
    """frame.npy: the whole frame when it fits in DUMP_BYTES, otherwise the pixels of a seeded sample (rows of a (k, 3) array,
    in pixel order), the same pixels for every run at the same resolution so that two builds can be compared."""
    os.makedirs(out_dir, exist_ok=True)
    out = np.ascontiguousarray(frame, dtype=np.float64)
    if out.nbytes > DUMP_BYTES:
        pixels = out.reshape(-1, out.shape[-1])
        keep = np.random.default_rng(0).choice(pixels.shape[0], DUMP_BYTES // pixels[0].nbytes, replace=False)
        out = pixels[np.sort(keep)]
    np.save(os.path.join(out_dir, "frame.npy"), out)


def bench_ours(args):
    import torch
    import torch.distributed as dist

    from raymond_b200 import api as A
    from raymond_b200 import build as B
    from raymond_b200 import distributed as D
    from raymond_b200 import fixtures as F

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this implementation has no CPU path")
    torch.cuda.set_device(local)
    side = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        side = dist.new_group(backend="gloo")      # host-side waits (while rank 0 alone drives all GPUs) must not spin on the devices
    B.build()
    precision = PRECISIONS[args.precision]

    objs, label = scene_objects(args.scene)
    cam = camera_for(args)
    W, H, spp = args.width, args.height, args.spp
    t0 = time.perf_counter()
    scene = A.Scene.from_fixture(objs)                   # host side: Mesh::new + AccGrid::build_from_mesh
    host_build_s = time.perf_counter() - t0
    settings = A.Settings(A.CameraSettings.from_fixture(cam), spp, (32, 32), args.bounces)

    def barrier():
        if world > 1:
            dist.barrier()

    def host_barrier():
        if world > 1:
            dist.barrier(group=side)

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- resident-scene throughput (`value`): scene in HBM, accumulators in HBM, this rank's share of the 500 samples, then the
    #      accumulator exchange (copy + ncclReduce onto rank 0) — all inside the timed region
    dr = D.DistributedRenderer(scene, settings, device=local, seed=args.seed, flags=A.FLAG_STAGE_TIMING, precision=precision)
    for _ in range(args.warmup):
        dr.clear()
        dr.render(spp)
        dr.checkpoint()
    dr.synchronize()
    s0 = dr.stats()
    st0 = dr.renderer.stage_stats()
    sampler = ClockSampler(local)
    sampler.start()
    barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(dr.stream)
    for _ in range(args.steps):
        dr.clear()
        dr.render(spp)
        dr.checkpoint()
    ev1.record(dr.stream)
    torch.cuda.synchronize()
    barrier()
    clocks = sampler.finish()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    s1 = dr.stats()
    st1 = dr.renderer.stage_stats()
    samples_total = W * H * spp * args.steps
    value = samples_total / ms_total / 1e3
    launches = int(sum_over_ranks(float(s1["kernel_launches"] - s0["kernel_launches"])))
    rays = int(sum_over_ranks(float(s1["rays"] - s0["rays"])))
    frame = dr.frame(spp)               # the running sums of the last timed step over spp (a view of a buffer the legs below reuse)
    if frame is not None and args.dump_outputs:
        dump_frame(args.dump_outputs, frame)
    mean_radiance = [float(x) for x in frame.mean(axis=(0, 1))] if frame is not None else None

    roofline = stages = None
    if rank == 0:
        roofline, stages = roofline_record(A, args, scene, settings, local, world, st0, st1, int(s1["samples"] - s0["samples"]), clocks)
    dr.close()
    del dr

    # ---- the same frame with the statistical scope (BRDF sampling / weights) in f32 (rm_precision 1), reported beside the headline
    f32_mode = None
    if not args.no_extras and precision == 0:
        d32 = D.DistributedRenderer(scene, settings, device=local, seed=args.seed, precision=A.PRECISION_F32_SHADING)
        d32.render(spp); d32.checkpoint(); d32.synchronize()
        n32 = max(1, min(args.steps, 3))
        barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(d32.stream)
        for _ in range(n32):
            d32.clear(); d32.render(spp); d32.checkpoint()
        e1.record(d32.stream)
        torch.cuda.synchronize(); barrier()
        ms32 = max_over_ranks(e0.elapsed_time(e1))
        f32frame = d32.frame(spp)
        f32_mode = {"value": W * H * spp * n32 / ms32 / 1e3, "unit": UNIT, "ms_per_step": ms32 / n32, "steps": n32,
                    "mean_radiance": None if f32frame is None else [float(x) for x in f32frame.mean(axis=(0, 1))],
                    "what": "rm_gpu_options.precision = RM_PRECISION_F32_SHADING: lobe sampling, Fresnel, GGX and Smith terms in f32 with FMA; camera rays, "
                            "Scene::intersect, hit points, normals and ray origins stay the reference's f64 sequence (tests: noise floor of SURVEY 8d)"}
        d32.close()
        del d32

    # ---- BASELINE configs[2] and configs[4] at this N (scene resident, exchange inside, wall clock around barriers, max over ranks)
    other = None
    if not args.no_extras:
        other = {}
        sp = A.Scene.from_fixture(F.reflective_spheres())
        c3 = A.Settings(A.CameraSettings.from_fixture(F.camera(1920, 1080, focal_length=2.5, aperture_radius=0.5)), args.c3_spp, (32, 32), 5)
        d3 = D.DistributedRenderer(sp, c3, device=local, seed=args.seed, partition=A.PARTITION_TILES, precision=precision)
        d3.render(min(50, args.c3_spp)); d3.sums()                # warm-up
        barrier(); torch.cuda.synchronize(); t0 = time.perf_counter()
        d3.clear(); d3.render(args.c3_spp); f3 = d3.frame(args.c3_spp)
        torch.cuda.synchronize(); barrier()
        sec = max_over_ranks(time.perf_counter() - t0)
        other["c3_reflective_spheres_dof_1920x1080_tiles"] = {
            "spp": args.c3_spp, "seconds": sec, "msamples_per_s": 1920 * 1080 * args.c3_spp / sec / 1e6, "partition": f"tiles round-robin over {world} GPU(s)",
            "mean_radiance": None if f3 is None else float(f3.mean())}
        d3.close()
        del d3
        spi5 = max(1, args.c5_spp // 16)                           # 16 checkpoints (256 at the full 4096 spp)
        c5 = A.Settings(A.CameraSettings.from_fixture(F.camera(3840, 2160)), args.c5_spp, (32, 32), 5, samples_per_iteration=spi5)
        d5 = D.DistributedRenderer(scene, c5, device=local, seed=args.seed, precision=precision)
        d5.render(min(8, args.c5_spp)); d5.sums()                 # warm-up
        barrier(); torch.cuda.synchronize(); t0 = time.perf_counter()
        f5 = d5.render_progressive(None)                          # 16 checkpoints: copy + ncclReduce each, D2H of the final frame
        torch.cuda.synchronize(); barrier()
        sec = max_over_ranks(time.perf_counter() - t0)
        other["c5_gold_dragon_3840x2160_progressive"] = {
            "spp": args.c5_spp, "samples_per_iteration": spi5, "seconds": sec, "msamples_per_s": 3840 * 2160 * args.c5_spp / sec / 1e6,
            "checkpoints": (args.c5_spp + spi5 - 1) // spi5, "partition": f"sample-split over {world} GPU(s)",
            "mean_radiance": None if f5 is None else float(f5.mean())}
        d5.close()
        del d5, f5

    # ---- BASELINE configs[3] (rank 0 of an N = 1 run): the 1 M-triangle soup, 1920x1080 pixel-centre primaries through the
    #      device-resident Scene::intersect query; C and T of the byte model counted by the instrumented kernels on the jittered
    #      camera rays of the same frame (1 spp, 1 bounce).  Its hit indices are held bit-exact to the oracle by tests/ (1-10 M).
    if other is not None and rank == 0 and world == 1 and not args.no_c4:
        try:
            tris = F.triangle_soup(1_000_000, F.SOUP_BOX_CUBIC)
            t0 = time.perf_counter()
            sgrid = A.AccGrid.build_from_mesh(A.Mesh.new(tris), device=local)
            build_s = time.perf_counter() - t0
            del tris
            soup = A.Scene()
            soup.push_grid(sgrid, A.Material.from_fixture(F.DRAGON_MATERIAL))
            cs4 = A.CameraSettings.from_fixture(F.camera(1920, 1080))
            cnt = A.Renderer(soup, A.Settings(cs4, 1, (32, 32), 1), A.GpuOptions(device=local, seed=args.seed, flags=A.FLAG_COUNT_WORK))
            cnt.render(0, 1)
            c4s = cnt.stage_stats()
            cnt.close()
            g4 = max(c4s["grid_rays"][1], 1)
            C4, T4 = c4s["cells"][1] / g4, c4s["triangle_tests"][1] / g4
            ds4 = A.DeviceScene(soup, local)
            n4 = 1920 * 1080
            rays4 = torch.empty((n4, 6), dtype=torch.float64, device=f"cuda:{local}")
            obj4 = torch.empty(n4, dtype=torch.int64, device=f"cuda:{local}")
            sub4 = torch.empty(n4, dtype=torch.int64, device=f"cuda:{local}")
            t4 = torch.zeros(n4, dtype=torch.float64, device=f"cuda:{local}")
            st4 = torch.cuda.current_stream().cuda_stream
            A.primary_rays_device(cs4, local, rays4.data_ptr(), st4)
            for _ in range(3):
                ds4.intersect_device(rays4.data_ptr(), n4, obj4.data_ptr(), sub4.data_ptr(), t4.data_ptr(), st4)
            torch.cuda.synchronize()
            best4 = None
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                ds4.intersect_device(rays4.data_ptr(), n4, obj4.data_ptr(), sub4.data_ptr(), t4.data_ptr(), st4)
                e1.record()
                torch.cuda.synchronize()
                best4 = e0.elapsed_time(e1) if best4 is None else min(best4, e0.elapsed_time(e1))
            hitf = float((obj4 >= 0).float().mean())
            entering = g4 / n4                                  # fraction of the frame's rays that enter the grid's box
            alg_bytes = (64.0 + 8.0 * C4 + 76.0 * T4) * entering * n4
            hbm_peak4 = 6650.0
            try:
                hbm_peak4 = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
            except Exception:  # noqa: BLE001
                pass
            other["c4_triangle_soup_1m_primary_hits"] = {
                "triangles": 1_000_000, "rays": n4, "ms": best4, "mrays_per_s": n4 / best4 / 1e3, "hit_fraction": hitf, "device_grid_build_s": build_s,
                "cells_per_grid_ray": C4, "tests_per_grid_ray": T4, "alg_gbs": alg_bytes / (best4 * 1e-3) / 1e9, "hbm_frac_on_alg_bytes": alg_bytes / (best4 * 1e-3) / 1e9 / hbm_peak4,
                "what": "k_setup + k_traverse + k_export_hits of one rm_device_scene_intersect call (best of 5, CUDA events); algorithmic bytes = 64 + 8 C + 76 T per grid ray "
                        "(SURVEY 8d); 4 M / 10 M soups and the ncu capture of this regime: profiles/r2_c4_soup_*"}
            del ds4, soup, sgrid, rays4, obj4, sub4, t4
        except Exception as e:  # noqa: BLE001
            log(f"[bench] configs[3] leg failed: {e!r}")
            other["c4_triangle_soup_1m_primary_hits"] = None

    # ---- end to end through the reference-facing call with host buffers: render_tiled(scene, settings).await() — scene flatten +
    #      H2D inside, D2H of the f64 frame + tile slicing + averaging inside.  N > 1: (1) one process per GPU (torchrun), every
    #      rank creates its renderer (scene upload), renders its share, exchange, frame on rank 0's host; (2) THE C-ABI call with
    #      device_count = N from rank 0's process alone (the other ranks hand their cached device memory back and wait on the host).
    e2e = e2e_torchrun = None
    if not args.no_e2e:
        e2e_steps = max(1, args.steps)
        d2h = W * H * 24
        if world > 1:
            times, h2d = [], 0
            for i in range(1 + e2e_steps):
                barrier(); torch.cuda.synchronize(); t0 = time.perf_counter()
                dre = D.DistributedRenderer(scene, settings, device=local, seed=args.seed + i, precision=precision)
                dre.render(spp)
                out = dre.frame(spp)
                stt = dre.stats()
                dre.close()
                torch.cuda.synchronize(); barrier()
                if i > 0:
                    times.append(time.perf_counter() - t0)
                h2d = int(stt["upload_bytes"])
            tt = max_over_ranks(sum(times))
            e2e_torchrun = {"value": W * H * spp * e2e_steps / tt / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(sum_over_ranks(float(h2d))),
                            "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": 1e3 * tt / e2e_steps,
                            "call": "per rank: DistributedRenderer(scene upload) + render(share) + ncclReduce + frame() on rank 0"}
            A.release_cached_memory()
        # the library's device-memory caches start empty (the legs above left blocks of other sizes in them); the first,
        # untimed frame below fills them again the way a process that renders this frame repeatedly has them
        A.release_cached_memory()
        host_barrier()
        if rank == 0:
            times, h2d = [], 0
            opts = dict(seed=args.seed, precision=precision)
            if world > 1:
                opts["device_list"] = list(range(world))
            else:
                opts["device"] = local
            frame_buf = np.zeros((H, W, 3))                      # the caller's frame buffer, kept across frames
            for i in range(1 + e2e_steps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                task = A.render_tiled(scene, settings, A.GpuOptions(**dict(opts, seed=args.seed + i)))
                out = task.await_(frame_buf)
                dt = time.perf_counter() - t0
                stt = task.stats()
                del task
                h2d = int(stt["upload_bytes"])
                if i > 0:
                    times.append(dt)
            e2e = {"value": W * H * spp * e2e_steps / sum(times) / 1e6, "unit": UNIT, "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": 1e3 * sum(times) / e2e_steps,
                   "ms_per_step_min": 1e3 * min(times), "ms_per_step_max": 1e3 * max(times), "ms_steps": [round(1e3 * t, 1) for t in times][:32],
                   "device_ms_last_step": float(stt["device_ms"]),
                   "call": "render_tiled(scene, settings).await()" + (f" with rm_gpu_options.device_count = {world} (one process drives all GPUs through the C ABI)" if world > 1 else ""),
                   "mean_radiance": float(out.mean())}
        host_barrier()

    # ---- CPU baseline: the oracle port on this box's host cores, bounded sample (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        osc = oracle_scene(objs)
        cspp, _ = cpu_sample_plan(osc, cam, args.bounces, args.cpu_seconds, cores)
        v, dt, cnt = run_cpu(osc, cam, cspp, args.bounces, cores, args.seed)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{W}x{H} x {cspp} spp of the same scene ({dt:.1f} s; reference threading model, f64, -ffp-contract=off)",
               "rays_per_path": cnt["rays"] / max(cnt["samples"], 1)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / max(args.steps, 1), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64" if args.precision == "f64" else "f64 intersection + f32 shading", "data": "synthetic",
            "config": config_of(args, label),
            "e2e": e2e, "e2e_torchrun": e2e_torchrun, "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "other_configs": other, "f32_shading": f32_mode,
            "mrays_per_s": rays / ms_total / 1e3, "rays_per_path": rays / max(samples_total, 1),
            "stages": stages, "host_grid_build_s": host_build_s, "mean_radiance": mean_radiance,
            "nonfinite_samples": int(s1["nonfinite_samples"]),
        }
        print_line(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    # stdout carries exactly ONE JSON line: anything libraries write to file descriptor 1 meanwhile (NCCL prints its version
    # banner and, with NCCL_DEBUG=INFO, its log there) is sent to stderr, and the descriptor is restored for the final print
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    real_stdout = os.fdopen(saved, "w")
    global print_line
    print_line = lambda text: (real_stdout.write(text + "\n"), real_stdout.flush())
    if args.impl == "reference":
        bench_reference(args)
    else:
        bench_ours(args)


if __name__ == "__main__":
    main()
