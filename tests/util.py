"""Shared helpers: instantiate a fixture scene in the product (CUDA) and in the oracle (CPU)."""
import os

import numpy as np

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

# A checkout of the reference project (Nyrox/raymond): its PLY meshes and renders are not part of this repository, so the
# tests that read them skip unless RAYMOND_REFERENCE_DIR names one.
REFERENCE_DIR = os.environ.get("RAYMOND_REFERENCE_DIR", "")
REFERENCE_MESHES = os.path.join(REFERENCE_DIR, "assets", "meshes")
NEEDS_REFERENCE = "needs a checkout of the reference project in RAYMOND_REFERENCE_DIR"


def have_reference_assets() -> bool:
    return bool(REFERENCE_DIR) and os.path.isdir(REFERENCE_MESHES)


def oracle_scene(objects) -> O.Scene:
    s = O.Scene()
    for o in objects:
        if o[0] == "sphere":
            s.add_sphere(o[1], o[2], o[3])
        elif o[0] == "plane":
            s.add_plane(o[1], o[2], o[3])
        else:
            s.add_grid(O.AccGrid.build_from_mesh(O.Mesh.from_triangles(o[1])), o[2])
    return s


def product_scene(objects) -> A.Scene:
    return A.Scene.from_fixture(objects)


def settings(cam: dict, spp: int, tile=(32, 32), bounce_limit=5, spi=0) -> A.Settings:
    return A.Settings(A.CameraSettings.from_fixture(cam), spp, tile, bounce_limit, spi)


def assert_hits_equal(got, want, what=""):
    """Bit-exact: object index, subobject (triangle) index and — on hits — the distance bits."""
    gobj, gsub, gt = got
    wobj, wsub, wt = want[:3]
    bad = np.nonzero(gobj != wobj)[0]
    assert bad.size == 0, f"{what}: {bad.size} object-index mismatches, first ray {bad[:5]}"
    hit = wobj >= 0
    bad = np.nonzero(gsub[hit] != wsub[hit])[0]
    assert bad.size == 0, f"{what}: {bad.size} subobject-index mismatches"
    gb = gt[hit].view(np.uint64)
    wb = wt[hit].view(np.uint64)
    bad = np.nonzero(gb != wb)[0]
    assert bad.size == 0, f"{what}: {bad.size} distances differ in their bits (max rel {np.max(np.abs(gt[hit]-wt[hit])/np.abs(wt[hit]))})"


def small_meshes() -> dict:
    """Generated meshes (travel to the GPU box) covering cubic and aliased (res.y > res.z) grids."""
    return {
        "cube": F.cube(),
        "bumpy": F.bumpy_sphere(),
        "bumpy_fine": F.bumpy_sphere(60, 120, 1.0, 0.1, (1.0, 0.7, 0.45)),
        "tube": F.dragon_standin(96, 24),
    }
