"""Regenerate tests/golden/* from a checkout of the reference project (Nyrox/raymond).

    RAYMOND_REFERENCE_DIR=<reference checkout> python scripts/make_golden.py

1. reference_png_blocks.json — 16x16-pixel block means (8-bit RGB) of the reference's OWN renders
   examples/ReflectiveSpheres.png and examples/GoldDragon.png (592x340, 500 spp, 5 bounces, README.md:24-28).
   They are the only outputs of the reference itself that exist (it has no tests and cannot be built here);
   tests/test_oracle.py renders the same scene with the oracle and compares block means.
2. reference_mesh_kats.json — what the ORACLE computes on the reference's shipped PLY meshes (assets/meshes):
   bounds, grid resolution, cell/reference counts, CRC32 of the cell lists and of the hit results of a fixed
   160x120 primary-ray frame.  Not reference truth — a regression pin, checked by the tests when the reference's
   meshes are at hand.
"""
import json
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REF = os.environ.get("RAYMOND_REFERENCE_DIR") or sys.exit("make_golden.py: set RAYMOND_REFERENCE_DIR to a checkout of the reference project (Nyrox/raymond)")
OUT = os.path.join(ROOT, "tests", "golden")


def png_blocks(path, block=16):
    from PIL import Image
    im = np.asarray(Image.open(path).convert("RGB"), dtype=np.float64)
    H, W, _ = im.shape
    hb, wb = H // block, W // block
    b = im[:hb * block, :wb * block].reshape(hb, block, wb, block, 3).mean(axis=(1, 3))
    return {"width": W, "height": H, "block": block, "rows": hb, "cols": wb, "mean_rgb8": np.round(b, 3).tolist(),
            "image_mean_rgb8": np.round(im.mean(axis=(0, 1)), 4).tolist(), "pure_black_pixels": int((im.sum(axis=-1) == 0).sum()),
            "ceiling_pixel_296_10": im[10, 296].astype(int).tolist()}


def mesh_kats():
    from oracle import oracle as O
    from raymond_b200 import fixtures as F
    out = {}
    cam = F.camera(160, 120, position=(0.0, 0.0, -4.0))
    rays = O.primary_rays(cam)
    for name in ("cube", "ico_sphere", "monkeysmooth", "suzanne", "suzanne_flat"):
        m = O.Mesh.load_ply(f"{REF}/assets/meshes/{name}.ply")
        e = {"triangles": len(m), "bounds": m.bounds.tolist()}
        brute_tri, brute_t = m.intersects(rays)
        e["brute_hits"] = int((brute_tri >= 0).sum())
        try:
            g = O.AccGrid.build_from_mesh(m)
        except O.OracleError as err:
            e["build_status"] = err.status
            out[name] = e
            continue
        i = g.info()
        start, refs = g.csr()
        tri, t, cnt = g.intersects(rays)
        e.update({"build_status": 0, "resolution": i["resolution"], "cell_size": i["cell_size"].tolist(), "cells": i["cell_count"],
                  "references": i["reference_count"], "max_per_cell": int(np.diff(start.astype(np.int64)).max()),
                  "empty_cells": int((np.diff(start.astype(np.int64)) == 0).sum()),
                  "csr_crc32": zlib.crc32(start.tobytes() + refs.tobytes()),
                  "hits": int((tri >= 0).sum()), "hit_tri_crc32": zlib.crc32(tri.tobytes()),
                  "hit_t_crc32": zlib.crc32(np.where(tri >= 0, t, 0.0).tobytes()),
                  "grid_equals_brute_force": bool(np.array_equal(tri, brute_tri) and np.array_equal(t[tri >= 0], brute_t[tri >= 0])),
                  "cells_visited": cnt["cells"], "triangle_tests": cnt["tri_tests"]})
        out[name] = e
    return out


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    blocks = {n: png_blocks(f"{REF}/examples/{n}.png") for n in ("ReflectiveSpheres", "GoldDragon")}
    json.dump(blocks, open(os.path.join(OUT, "reference_png_blocks.json"), "w"))
    json.dump(mesh_kats(), open(os.path.join(OUT, "reference_mesh_kats.json"), "w"), indent=1)
    print("wrote", os.listdir(OUT))
