"""Census of the rays of the last wavefront stage (depth == bounce_limit) of the bench frame, on the CPU.

    python scripts/last_bounce_census.py [--width 480 --height 270 --spp 4 --bounces 5 --seed 2026 --out profiles/r4_last_bounce_census.json]

In the default (drop) mode a path at depth bounce_limit delivers its throughput times the emission of the closest object if that
object is an emitter, and an exact 0 otherwise.  On GoldDragon the grid (the dragon) is Metal, so a last-depth ray whose closest
analytic object (sphere / planes) is not an emitter is decided before its grid traversal.  This script counts, for the
last-depth rays of a reduced GoldDragon frame (the bench scene, camera and seed at fewer pixels and samples):
  rays         the rays of the stage (paths still alive after depth bounce_limit - 1)
  box          ... whose line enters the grid's bounding box ahead of the origin (AABB::intersects)
  grid_rays    ... of those, the ones k_setup queues for traversal: not already hit by another object before the box entry
               (the `tmin > best_t + bound` rule of k_setup)
  emissive     ... of those, the ones whose closest analytic hit is an emitter: they still need the traversal
  skippable    grid_rays - emissive, and its share of grid_rays
Every Scene::intersect is the oracle's (the reference's f64 sequence); the bounce is the f64 lobe of k_shade / the reference
(src/trace.rs:256-319) in numpy with the same counter-based draws, so the paths are the ones the renderer follows up to
last-bit differences of sin / cos / acos.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np

from oracle import oracle as O
from raymond_b200 import fixtures as F

M32 = np.uint64(0xFFFFFFFF)


def philox(seed: int, c0, c1, c2, c3):
    """Philox4x32-10 of rm_kernels.cuh / the oracle, vectorised (uint32 lanes carried in uint64)."""
    c = [np.asarray(x, dtype=np.uint64) & M32 for x in (c0, c1, c2, c3)]
    c = np.broadcast_arrays(*c)
    c0, c1, c2, c3 = [x.copy() for x in c]
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & M32
        k0 = (k0 + 0x9E3779B9) & 0xFFFFFFFF
        k1 = (k1 + 0xBB67AE85) & 0xFFFFFFFF
    return c0, c1, c2, c3


def draw(hi, lo):
    """u52: 52 bits -> (k + 0.5) * 2^-52"""
    return ((((hi << np.uint64(32)) | lo) >> np.uint64(12)).astype(np.float64) + 0.5) * (1.0 / 4503599627370496.0)


def dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def normalize(a):
    return a * (1.0 / np.sqrt(dot(a, a)))[..., None]


def onb(n):
    sign = np.where(n[:, 2] > 0.0, 1.0, -1.0)
    a = -1.0 / (sign + n[:, 2])
    bb = n[:, 0] * n[:, 1] * a
    t = np.stack([1.0 + sign * n[:, 0] * n[:, 0] * a, sign * bb, -sign * n[:, 0]], axis=1)
    b = np.stack([bb, sign + n[:, 1] * n[:, 1] * a, -n[:, 1]], axis=1)
    return t, b


def heron(a, b, c):
    ab, ac, bc = np.linalg.norm(b - a, axis=1), np.linalg.norm(c - a, axis=1), np.linalg.norm(c - b, axis=1)
    s = (ab + ac + bc) / 2.0
    return np.sqrt(s * (s - ab) * (s - ac) * (s - bc))


def lobe(seed, normal, view_from, color, rough, metal, pixel, sample, depth):
    """lobe_f64: next direction, weight, offset along the normal."""
    view = normalize(view_from)
    f0 = 0.04 + metal[:, None] * (color - 0.04)
    w0, w1, w2, w3 = philox(seed, pixel, sample, depth, 0)
    r, ra = draw(w0, w1), draw(w2, w3)
    w0, w1, _, _ = philox(seed, pixel, sample, depth, 1)
    rb = draw(w0, w1)
    prob_d = 0.5 + metal * (0.0 - 0.5)
    diff = r < prob_d
    refl = normalize(-view - 2.0 * ((-dot(view, normal))[:, None] * normal))
    axis = np.where(diff[:, None], normal, refl)
    a = rough * rough
    with np.errstate(all="ignore"):
        theta = a * np.sqrt(rb / (1.0 - rb))
        c_t = np.where(diff, np.sqrt(ra), np.cos(theta))
        s_t = np.where(diff, np.sqrt(1.0 - ra), np.sin(theta))
        phi = 2.0 * np.pi * np.where(diff, rb, ra)
        tg, bt = onb(axis)
        local = np.stack([s_t * np.cos(phi), c_t, s_t * np.sin(phi)], axis=1)
        d = normalize((tg * local[:, :1] + axis * local[:, 1:2]) + bt * local[:, 2:3])
        ndl = dot(normal, d)
        half = normalize(d + view)
        hv = dot(half, view)
        one = 1.0
        fres_d = f0 + (one - f0) * (1.0 - np.fmax(hv, 0.0))[:, None] ** 5
        w_d = (((one - fres_d) * (1.0 - metal)[:, None]) * color * np.fmax(ndl, 0.0)[:, None]) / (prob_d * c_t)[:, None]
        F_s = f0 + (one - f0) * (1.0 - hv)[:, None] ** 5
        nh = dot(normal, half)
        den = np.fmax(np.pi * ((nh * nh) * (a - 1.0) + 1.0) ** 2, 1e-7)
        D = a / den
        k = a / 8.0
        nv, nl = np.fmax(dot(normal, view), 0.0), np.fmax(ndl, 0.0)
        G = (nv / (nv * (1.0 - k) + k)) * (nl / (nl * (1.0 - k) + k))
        denom = 4.0 * dot(normal, view) * ndl + 0.001
        pdf = (D * nh) / (4.0 * hv) + 0.0001
        w_s = ((((D * G)[:, None] * F_s) / denom[:, None]) * ndl[:, None] / (1.0 - prob_d)[:, None]) / pdf[:, None]
    wgt = np.where(diff[:, None], w_d, w_s)
    eps = np.where(diff, 0.00001, 0.0001)
    return d, wgt, eps


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--width", type=int, default=480)
    p.add_argument("--height", type=int, default=270)
    p.add_argument("--spp", type=int, default=4)
    p.add_argument("--bounces", type=int, default=5)
    p.add_argument("--seed", type=int, default=2026)
    p.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_last_bounce_census.json"))
    args = p.parse_args()
    t0 = time.time()

    tris = F.translate(F.dragon_standin(), F.DRAGON_TRANSLATE)
    objs = F.gold_dragon(F.dragon_standin())
    full, analytic = O.Scene(), O.Scene()
    kinds, mats = [], []
    analytic_index = []            # full-scene index of each object of the analytic-only scene
    for i, o in enumerate(objs):
        if o[0] == "sphere":
            full.add_sphere(o[1], o[2], o[3]); analytic.add_sphere(o[1], o[2], o[3]); analytic_index.append(i)
        elif o[0] == "plane":
            full.add_plane(o[1], o[2], o[3]); analytic.add_plane(o[1], o[2], o[3]); analytic_index.append(i)
        else:
            grid = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(o[1]))
            bounds = grid.info()["bounds"]
            full.add_grid(grid, o[2])
        kinds.append(o[0])
        mats.append(o[-1])
    analytic_index = np.array(analytic_index)
    emissive = np.array([m[0] == "Emission" for m in mats])
    color = np.array([m[1] for m in mats], dtype=np.float64)
    rough = np.array([0.0 if m[0] == "Emission" else m[2] for m in mats])
    metal = np.array([1.0 if m[0] == "Metal" else 0.0 for m in mats])
    grid_obj = kinds.index("grid")
    shd = tris.reshape(-1, 3, 11)         # per vertex: position (0:3), normal (3:6), ...
    diag = float(np.linalg.norm(bounds[1] - bounds[0]))
    diag2 = diag * diag

    cam = F.camera(args.width, args.height)
    cpos = np.array(cam["position"])
    n_pix = args.width * args.height
    rays = np.concatenate([O.camera_rays(cam, args.seed, s) for s in range(args.spp)])
    pixel = np.tile(np.arange(n_pix, dtype=np.uint64), args.spp)
    sample = np.repeat(np.arange(args.spp, dtype=np.uint64), n_pix)
    T = np.ones((rays.shape[0], 3))
    per_depth = []
    for depth in range(1, args.bounces + 1):
        obj, sub, t, _ = full.intersect(rays, threads=args.threads)
        row = {"depth": depth, "rays": int(rays.shape[0])}
        if depth == args.bounces:
            o, d = rays[:, :3], rays[:, 3:]
            aobj, _, at, _ = analytic.intersect(rays, threads=args.threads)
            best = np.where(aobj >= 0, analytic_index[np.maximum(aobj, 0)], -1)
            with np.errstate(all="ignore"):
                inv = 1.0 / d
                t1, t2 = (bounds[0] - o) * inv, (bounds[1] - o) * inv
                tmin = np.fmin(t1, t2).max(axis=1)
                tmax = np.fmax(t1, t2).min(axis=1)
            box = tmax > np.fmax(tmin, 0.0)
            pushed = box & ~((best >= 0) & (tmin > at + (1e-6 + 4e-7 * (np.fmax(tmin, 0.0) + diag) * diag2)))
            emit = pushed & (best >= 0) & emissive[np.maximum(best, 0)]
            n_push, n_emit = int(pushed.sum()), int(emit.sum())
            row.update({"box": int(box.sum()), "grid_rays": n_push, "emissive": n_emit, "skippable": n_push - n_emit,
                        "skippable_share": (n_push - n_emit) / max(n_push, 1),
                        "closest_is_emitter": int(((obj >= 0) & emissive[np.maximum(obj, 0)]).sum())})
            per_depth.append(row)
            break
        hit = obj >= 0
        emit = hit & emissive[np.maximum(obj, 0)]
        go = hit & ~emit
        o, d, ti, ob = rays[go, :3], rays[go, 3:], t[go], obj[go]
        frag = o + d * ti[:, None]
        normal = np.empty_like(frag)
        is_plane = np.array([k == "plane" for k in kinds])[ob]
        is_sphere = np.array([k == "sphere" for k in kinds])[ob]
        is_grid = ob == grid_obj
        normal[is_plane] = np.array([objs[k][2] for k in ob[is_plane]]).reshape(-1, 3)
        normal[is_sphere] = normalize(frag[is_sphere] - np.array([objs[k][1] for k in ob[is_sphere]]).reshape(-1, 3))
        if is_grid.any():
            v = shd[sub[go][is_grid].astype(np.int64)]
            v0, v1, v2 = v[:, 0, 0:3], v[:, 1, 0:3], v[:, 2, 0:3]
            n0, n1, n2 = v[:, 0, 3:6], v[:, 1, 3:6], v[:, 2, 3:6]
            fp = frag[is_grid]
            with np.errstate(all="ignore"):
                abc = heron(v0, v1, v2)
                ba, bb = heron(v0, v1, fp) / abc, heron(v0, v2, fp) / abc
                bc = 1.0 - (ba + bb)
                normal[is_grid] = normalize(n2 * ba[:, None] + n1 * bb[:, None] + n0 * bc[:, None])
        nd, w, eps = lobe(args.seed, normal, cpos - frag, color[ob], rough[ob], metal[ob], pixel[go], sample[go], depth)
        Tn = T[go] * w
        alive = ~np.all(Tn == 0.0, axis=1)
        row.update({"emitter_hits": int(emit.sum()), "misses": int((~hit).sum()), "zero_throughput": int((~alive).sum())})
        per_depth.append(row)
        rays = np.concatenate([frag + normal * eps[:, None], nd], axis=1)[alive]
        T, pixel, sample = Tn[alive], pixel[go][alive], sample[go][alive]

    last = per_depth[-1]
    rec = {"what": "last-depth census, GoldDragon (stand-in mesh), oracle intersections, CPU", "width": args.width, "height": args.height,
           "spp": args.spp, "bounces": args.bounces, "seed": args.seed, "per_depth": per_depth,
           "last_depth_skippable_share": last.get("skippable_share"), "seconds": round(time.time() - t0, 1)}
    print(json.dumps(rec))
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
