"""CPU census of grouped bounding-sphere culling in k_traverse: would testing one sphere around a run of G consecutive references
of a cell's list, before the references' own spheres, cut the stage-1 items of the pooled loop?

    python scripts/ref_group_census.py [--width 480 --height 270 --spp 4 --seed 2026 --soup-width 480 --soup-height 270]

Rays: the grid rays of depths 1 and 2 of a reduced bench frame (the GoldDragon stand-in, its camera and seed at fewer pixels
and samples; the bounce is last_bounce_census.py's f64 lobe), and the pixel-centre-jittered primaries of the 1 M-triangle
soup of configs[3].  The occupied cells each ray visits come from the oracle's own walk (ref_group_census.cpp).  Per
(ray, visited occupied cell):
  items     today's stage-1 items: the length of the cell's list
  grouped   ceil(count / G) group tests, plus the members of the groups that pass
  survivors references whose own sphere test passes (today), and those of them inside a passing group (grouped): equal
            unless a member escapes the `lim < r2` guard of cull_sphere while its group does not
Spheres are the library's (cover_census.spheres: prepare_grid_image's rule).  A group sphere has an f32 centre at the middle
of the members' sphere boxes and the radius (max |c_g - c_i| + R_i) (1 + 2e-6), in f64 rounded up to f32, infinite when a
member's is: every member sphere lies inside it with a margin, so a group the line misses holds no survivor.  The cull test
is cull_sphere's, f64, with its per-ray `lim` guard.  The last row, G = cell, is one sphere per occupied cell: k_traverse tests it
in the lane that reaches the cell, so its group test costs no pooled round (profiles/README.md, round 11).
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402

from oracle import oracle as O  # noqa: E402
from raymond_b200 import fixtures as F  # noqa: E402
from cover_census import spheres  # noqa: E402
from last_bounce_census import heron, lobe, normalize  # noqa: E402

WHOLE_CELL = 1 << 30            # a group as long as any list: one sphere per occupied cell (what k_traverse tests)
GROUPS = (2, 4, 8, WHOLE_CELL)


def walker():
    src = os.path.join(ROOT, "scripts", "ref_group_census.cpp")
    h = hashlib.sha256()
    for p in (src, os.path.join(ROOT, "oracle", "raymond_oracle.cpp")):
        with open(p, "rb") as f:
            h.update(f.read())
    out_dir = os.path.join(tempfile.gettempdir(), f"raymond_ref_group_census_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"libref_group_census_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-shared", "-o", tmp,
                        src, "-lm"], check=True)
        os.replace(tmp, so)
    L = C.CDLL(so, mode=os.RTLD_LOCAL)
    vp, sz = C.c_void_p, C.c_size_t
    L.rmo_mesh_from_triangles.restype = vp
    L.rmo_mesh_from_triangles.argtypes = [vp, sz]
    L.rmo_mesh_destroy.argtypes = [vp]
    L.rmo_grid_build.restype = vp
    L.rmo_grid_build.argtypes = [vp, C.POINTER(C.c_int)]
    L.rmo_grid_destroy.argtypes = [vp]
    L.rmoc_walk_grid.restype = vp
    L.rmoc_walk_grid.argtypes = [vp, vp, sz, C.c_int, C.POINTER(sz)]
    L.rmoc_walk_take.argtypes = [vp, vp, vp]
    return L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def visited_cells(L, tris, rays, threads):
    """(ray index, cell index) of every occupied cell the rays visit, for the oracle's grid of `tris`."""
    t = np.ascontiguousarray(tris, dtype=np.float64).reshape(-1, O.TRI_DOUBLES)
    mesh = L.rmo_mesh_from_triangles(_ptr(t), t.shape[0])
    st = C.c_int(0)
    g = L.rmo_grid_build(mesh, C.byref(st))
    L.rmo_mesh_destroy(mesh)
    assert g, f"grid build: oracle status {st.value}"
    r = np.ascontiguousarray(rays, dtype=np.float64)
    n = C.c_size_t(0)
    w = L.rmoc_walk_grid(g, _ptr(r), r.shape[0], threads, C.byref(n))
    ray, cell = np.zeros(n.value, np.uint64), np.zeros(n.value, np.uint64)
    L.rmoc_walk_take(w, _ptr(ray), _ptr(cell))
    L.rmo_grid_destroy(g)
    return ray.astype(np.int64), cell.astype(np.int64)


def round_up_f32(r):
    rf = r.astype(np.float32)
    low = ~(rf.astype(np.float64) >= r)
    rf[low] = np.nextafter(rf[low], np.float32(np.inf))
    return rf.astype(np.float64)


def group_spheres(c, R, start, G):
    """Group spheres of runs of G consecutive references of each cell's list (c, R: per-reference spheres in reference order;
    start: the cells' list starts, n_cells + 1).  Returns (centre, radius, first reference) per group, and the group base per cell."""
    cnt = np.diff(start)
    ng = (cnt + G - 1) // G
    gbase = np.zeros(cnt.shape[0] + 1, np.int64)
    np.cumsum(ng, out=gbase[1:])
    cell_of_group = np.repeat(np.arange(cnt.shape[0]), ng)
    first = start[cell_of_group] + (np.arange(gbase[-1]) - gbase[cell_of_group]) * G
    with np.errstate(invalid="ignore"):
        lo = np.minimum.reduceat(c - R[:, None], first, axis=0) if first.size else np.zeros((0, 3))
        hi = np.maximum.reduceat(c + R[:, None], first, axis=0) if first.size else np.zeros((0, 3))
        cg = ((lo + hi) * 0.5).astype(np.float32).astype(np.float64)
        member_group = np.repeat(np.arange(first.size), np.diff(np.append(first, start[-1])))
        reach = np.sqrt(((cg[member_group] - c) ** 2).sum(1)) + R
        rg = np.maximum.reduceat(reach, first) * (1.0 + 2e-6) if first.size else np.zeros(0)
    inf = np.maximum.reduceat(~np.isfinite(R), first) if first.size else np.zeros(0, bool)
    rg = round_up_f32(rg)
    rg[inf | ~np.isfinite(rg)] = np.inf
    cg[inf] = 0.0
    return cg, rg, first, gbase


def culled(cs, rs, o, d, dd, lim):
    """cull_sphere: |cross(c - o, d)|^2 > R^2 |d|^2 and lim < R^2 (f64)."""
    oc = cs - o
    cr = np.cross(oc, d)
    r2 = rs * rs
    with np.errstate(invalid="ignore", over="ignore"):
        return ((cr * cr).sum(1) > r2 * dd) & (lim < r2)


def census(L, tris, rays, bounds, threads, chunk=1 << 21):
    P = np.asarray(F.positions(tris), dtype=np.float64)
    ray_i, cell_i = visited_cells(L, tris, rays, threads)
    mesh = O.Mesh.from_triangles(tris)
    start, refs = O.AccGrid.build_from_mesh(mesh).csr()
    start, refs = start.astype(np.int64), refs.astype(np.int64)
    tc, tR = spheres(P)
    c, R = tc[refs], tR[refs]
    o, d = rays[:, :3], rays[:, 3:]
    dd = (d * d).sum(1)
    m = np.maximum(np.abs(bounds[0] - o), np.abs(bounds[1] - o))
    lim = (m * m).sum(1) * 1.01e-17
    grp = {G: group_spheres(c, R, start, G) for G in GROUPS}
    cnt = start[cell_i + 1] - start[cell_i]
    out = {"rays": int(np.unique(ray_i).size), "cells": int(ray_i.size), "items": int(cnt.sum()), "survivors": 0}
    for G in GROUPS:
        out[f"G{G}"] = {"group_tests": 0, "members": 0, "survivors": 0}
    lo = 0
    while lo < ray_i.size:                                   # chunks of pairs holding about `chunk` items
        hi = min(ray_i.size, lo + max(1, int(np.searchsorted(np.cumsum(cnt[lo:]), chunk))))
        pr, pc, pn = ray_i[lo:hi], cell_i[lo:hi], cnt[lo:hi]
        item_pair = np.repeat(np.arange(pr.size), pn)
        pos = start[pc][item_pair] + (np.arange(item_pair.size) - np.repeat(np.cumsum(pn) - pn, pn))
        ir = pr[item_pair]
        own = ~culled(c[pos], R[pos], o[ir], d[ir], dd[ir], lim[ir])
        out["survivors"] += int(own.sum())
        for G in GROUPS:
            cg, rg, first, gbase = grp[G]
            gi = gbase[pc][item_pair] + (pos - start[pc][item_pair]) // G        # group of each item
            heads = pos == first[gi]                                              # one group test per group
            gpass = ~culled(cg[gi[heads]], rg[gi[heads]], o[ir[heads]], d[ir[heads]], dd[ir[heads]], lim[ir[heads]])
            member_pass = np.repeat(gpass, np.diff(np.append(np.flatnonzero(heads), gi.size)))
            s = out[f"G{G}"]
            s["group_tests"] += int(heads.sum())
            s["members"] += int(member_pass.sum())
            s["survivors"] += int((own & member_pass).sum())
        lo = hi
    for G in GROUPS:
        s = out[f"G{G}"]
        s["grouped_items"] = s["group_tests"] + s["members"]
        s["ratio"] = round(s["grouped_items"] / max(out["items"], 1), 4)
        s["group_pass_rate"] = round(s["members"] / max(out["items"], 1), 4)
    return out


def bounce(seed, objs, kinds, tris, rays, obj, sub, t, pixel, sample, cpos, mats, depth):
    """The depth+1 rays of the paths that hit a non-emitter at `depth` (last_bounce_census.py's bounce)."""
    emissive = np.array([m[0] == "Emission" for m in mats])
    color = np.array([m[1] for m in mats], dtype=np.float64)
    rough = np.array([0.0 if m[0] == "Emission" else m[2] for m in mats])
    metal = np.array([1.0 if m[0] == "Metal" else 0.0 for m in mats])
    go = (obj >= 0) & ~emissive[np.maximum(obj, 0)]
    o, d, ti, ob = rays[go, :3], rays[go, 3:], t[go], obj[go]
    frag = o + d * ti[:, None]
    normal = np.empty_like(frag)
    is_plane = np.array([k == "plane" for k in kinds])[ob]
    is_sphere = np.array([k == "sphere" for k in kinds])[ob]
    is_grid = np.array([k == "grid" for k in kinds])[ob]
    normal[is_plane] = np.array([objs[k][2] for k in ob[is_plane]]).reshape(-1, 3)
    normal[is_sphere] = normalize(frag[is_sphere] - np.array([objs[k][1] for k in ob[is_sphere]]).reshape(-1, 3))
    shd = tris.reshape(-1, 3, 11)
    if is_grid.any():
        v = shd[sub[go][is_grid].astype(np.int64)]
        with np.errstate(all="ignore"):
            abc = heron(v[:, 0, 0:3], v[:, 1, 0:3], v[:, 2, 0:3])
            ba = heron(v[:, 0, 0:3], v[:, 1, 0:3], frag[is_grid]) / abc
            bb = heron(v[:, 0, 0:3], v[:, 2, 0:3], frag[is_grid]) / abc
            bc = 1.0 - (ba + bb)
            normal[is_grid] = normalize(v[:, 2, 3:6] * ba[:, None] + v[:, 1, 3:6] * bb[:, None] + v[:, 0, 3:6] * bc[:, None])
    nd, w, eps = lobe(seed, normal, cpos - frag, color[ob], rough[ob], metal[ob], pixel[go], sample[go], depth)
    alive = ~np.all(w == 0.0, axis=1)
    return np.concatenate([frag + normal * eps[:, None], nd], axis=1)[alive], pixel[go][alive], sample[go][alive]


def grid_rays(analytic, rays, bounds, threads):
    """The rays k_setup queues for traversal: the line enters the grid's box ahead of the origin, and no analytic object is hit
    before the box entry (k_setup's `tmin > best_t + bound` rule)."""
    o, d = rays[:, :3], rays[:, 3:]
    aobj, _, at, _ = analytic.intersect(rays, threads=threads)
    diag = float(np.linalg.norm(bounds[1] - bounds[0]))
    with np.errstate(all="ignore"):
        inv = 1.0 / d
        t1, t2 = (bounds[0] - o) * inv, (bounds[1] - o) * inv
        tmin, tmax = np.fmin(t1, t2).max(axis=1), np.fmax(t1, t2).min(axis=1)
    box = tmax > np.fmax(tmin, 0.0)
    return rays[box & ~((aobj >= 0) & (tmin > at + (1e-6 + 4e-7 * (np.fmax(tmin, 0.0) + diag) * diag * diag)))]


def show(name, r):
    print(f"{name}: {r['rays']} rays, {r['cells']} occupied cells visited, {r['items']} stage-1 items "
          f"({r['items'] / max(r['rays'], 1):.1f} per ray), {r['survivors']} survivors")
    for G in GROUPS:
        s = r[f"G{G}"]
        same = "identical" if s["survivors"] == r["survivors"] else f"DIFFER by {r['survivors'] - s['survivors']}"
        print(f"  G={'cell' if G == WHOLE_CELL else G}: {s['group_tests']} group tests + {s['members']} members of passing groups = {s['grouped_items']} items, "
              f"{s['ratio']:.3f} x today; members pass {s['group_pass_rate']:.3f}; survivors {s['survivors']} ({same})")


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--width", type=int, default=480)
    p.add_argument("--height", type=int, default=270)
    p.add_argument("--spp", type=int, default=4)
    p.add_argument("--seed", type=int, default=2026)
    p.add_argument("--soup-width", type=int, default=480)
    p.add_argument("--soup-height", type=int, default=270)
    p.add_argument("--threads", type=int, default=os.cpu_count() or 1)
    a = p.parse_args()
    t0 = time.time()
    L = walker()

    tris = F.translate(F.dragon_standin(), F.DRAGON_TRANSLATE)
    objs = F.gold_dragon(F.dragon_standin())
    full, analytic = O.Scene(), O.Scene()
    kinds, mats = [], []
    for ob in objs:
        if ob[0] == "sphere":
            full.add_sphere(ob[1], ob[2], ob[3]); analytic.add_sphere(ob[1], ob[2], ob[3])
        elif ob[0] == "plane":
            full.add_plane(ob[1], ob[2], ob[3]); analytic.add_plane(ob[1], ob[2], ob[3])
        else:
            grid = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(ob[1]))
            bounds = grid.info()["bounds"]
            full.add_grid(grid, ob[2])
        kinds.append(ob[0])
        mats.append(ob[-1])
    cam = F.camera(a.width, a.height)
    n_pix = a.width * a.height
    rays = np.concatenate([O.camera_rays(cam, a.seed, s) for s in range(a.spp)])
    pixel = np.tile(np.arange(n_pix, dtype=np.uint64), a.spp)
    sample = np.repeat(np.arange(a.spp, dtype=np.uint64), n_pix)
    print(f"GoldDragon stand-in, {tris.shape[0]} triangles, {a.width}x{a.height} x {a.spp} spp, seed {a.seed}")
    for depth in (1, 2):
        show(f"depth {depth}", census(L, tris, grid_rays(analytic, rays, bounds, a.threads), bounds, a.threads))
        if depth == 1:
            obj, sub, t, _ = full.intersect(rays, threads=a.threads)
            rays, pixel, sample = bounce(a.seed, objs, kinds, tris, rays, obj, sub, t, pixel, sample, np.array(cam["position"]), mats, depth)

    soup = F.triangle_soup(1_000_000, F.SOUP_BOX_CUBIC)
    sb = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(soup)).info()["bounds"]
    srays = O.camera_rays(F.camera(a.soup_width, a.soup_height), a.seed, 0)
    print(f"1 M-triangle soup (configs[3]), {a.soup_width}x{a.soup_height} primaries")
    show("primary", census(L, soup, srays, sb, a.threads))
    print(f"({time.time() - t0:.0f} s)")


if __name__ == "__main__":
    main()
