"""Scenes and cameras outside the few material and camera settings the benchmark scenes use, for the same-stream tests of
test_gpu_shading_space.py; test_shading_space_oracle.py checks on the CPU that each fixture reaches the regime it is for.

Every fixture is 96x72 (unless its camera says otherwise) at 4 spp, seed 7.  The regimes (`tags`):

* "nonfinite": roughness 0.  k = 0 in geometry_schlick_ggx, so it divides 0 by 0 whenever n.v <= 0 or n.l <= 0, and the view
  vector always points at the camera (A8): the reference's samples are NaN on many paths.
* "negative": colours outside [0, 1] give negative path values.
* "bright": non-unit plane normals scale both the weight and the ray offset by |n|; path values above 100.
* "camera": the frame differs from the one the origin camera with fov 55 (and no depth of field) sees.
* "shape": a frame far from 4:3 (pixel index to (x, y) and the aspect ratio); its pixels are not all alike.
* "f32": also rendered in the f32 shading mode (roughness sweep, colours, non-unit normals).
* "last_bounce": the last-depth shortcut must not change a bit (non-emissive grids in front of an emitter).
"""
from dataclasses import dataclass, field

import numpy as np

from raymond_b200 import fixtures as F

from test_gpu_edges import two_mesh_scene

W, H, SPP, SEED = 96, 72, 4, 7
BOX = F.BOX_PLANES
EMISSION_1E3 = ("Emission", (1e-3, 1e-3, 1e-3), (1.0, 1.0, 1.0), 0.0, 0.0)


@dataclass
class Fixture:
    objs: list
    cam: dict = field(default_factory=lambda: F.camera(W, H))
    limit: int = 5
    tags: tuple = ()


def two_spheres(kind: str, rough: float, colour=(0.9, 0.6, 0.3)) -> list:
    return [("sphere", (0.0, -0.2, 3.0), 0.8, (kind, colour, rough)),
            ("sphere", (-1.2, -0.6, 2.6), 0.4, (kind, (0.8, 0.8, 0.8), rough))] + BOX


def bumpy_mesh() -> np.ndarray:
    return F.translate(F.bumpy_sphere(20, 40, 0.6), (0.2, -0.3, 3.0))


ROUGHNESS = (0.0, 1e-3, 0.3, 1.0, 1.5, 3.0)       # at 3.0 the GGX angle reaches ~6e8 rad: CUDA sincos against glibc far out


def fixtures() -> dict:
    fx = {}
    for kind in ("Metal", "Diffuse"):
        for rough in ROUGHNESS:
            fx[f"{kind.lower()}_rough_{rough:g}"] = Fixture(two_spheres(kind, rough), tags=("f32",) + (("nonfinite",) if rough == 0.0 else ()))
    for rough in (0.3, 1.5):
        for limit in (1, 2, 8):
            fx[f"metal_rough_{rough:g}_limit_{limit}"] = Fixture(two_spheres("Metal", rough), limit=limit)
    mesh = bumpy_mesh()
    fx["mesh_metal_rough_0"] = Fixture([("grid", mesh, ("Metal", (0.9, 0.7, 0.3), 0.0))] + BOX, tags=("nonfinite",))
    fx["mesh_metal_rough_0.8"] = Fixture([("grid", mesh, ("Metal", (0.9, 0.7, 0.3), 0.8))] + BOX)
    ball = ("sphere", (0.0, -0.2, 3.0), 0.8)
    # the 0.04 channel makes the Metal f0 equal the colour there
    fx["colour_diffuse"] = Fixture([ball + (("Diffuse", (1.7, 0.04, -0.3), 0.5),)] + BOX, tags=("negative", "f32"))
    fx["colour_metal"] = Fixture([ball + (("Metal", (-0.5, 2.0, 0.04), 0.4),)] + BOX, tags=("negative", "f32"))
    fx["emitter_sphere_fov_120"] = Fixture([("sphere", (0.5, 0.3, 2.5), 0.3, ("Emission", (40.0, 20.0, 5.0), (1.0, 1.0, 1.0), 0.0, 0.0)),
                                            ("sphere", (-0.5, -0.5, 3.0), 0.5, ("Diffuse", (0.8, 0.8, 0.8), 0.3))] + BOX,
                                           cam=F.camera(W, H, fov_vert=120.0), tags=("camera",))
    fx["emitter_1e-3"] = Fixture(two_spheres("Metal", 0.3)[:2] + [BOX[0], ("plane", (0.0, 2.0, 0.0), (0.0, -1.0, 0.0), EMISSION_1E3)] + BOX[2:])
    fx["emitter_behind_grid"] = Fixture([("grid", mesh, ("Metal", (0.9, 0.9, 0.9), 0.3)),
                                         ("sphere", (0.1, -0.2, 4.3), 0.6, ("Emission", (6.0, 5.0, 4.0), (1.0, 1.0, 1.0), 0.0, 0.0))] + BOX,
                                        tags=("last_bounce",))
    fx["normals_non_unit"] = Fixture([("plane", (0.0, -1.0, 0.0), (0.0, 3.0, 0.0), ("Diffuse", (0.75, 0.75, 0.75), 0.5)),
                                      ("plane", (0.0, 2.0, 0.0), (0.0, -0.5, 0.0), BOX[1][3])] + BOX[2:], tags=("bright", "f32"))
    fx["normals_tilted_metal_floor"] = Fixture([("plane", (0.0, -1.0, 0.0), (0.3, 2.0, -0.4), ("Metal", (0.9, 0.8, 0.7), 0.2))] + BOX[1:], tags=("f32",))
    spheres = F.reflective_spheres()
    fx["camera_position"] = Fixture(spheres, cam=F.camera(W, H, position=(0.8, 1.2, 1.0)), tags=("camera",))
    # the camera looks along +z at a small sphere near the back wall, and sees the big one only in reflections; n.v <= 0 is common
    fx["camera_behind_metal"] = Fixture([("sphere", (1.3, 1.2, 4.6), 0.3, ("Metal", (0.9, 0.9, 0.9), 0.6))] + two_spheres("Metal", 0.6),
                                        cam=F.camera(W, H, position=(1.5, 1.5, 4.0)), tags=("camera",))
    fx["camera_fov_10"] = Fixture(spheres, cam=F.camera(W, H, fov_vert=10.0), tags=("camera",))
    fx["camera_fov_120"] = Fixture(spheres, cam=F.camera(W, H, fov_vert=120.0), tags=("camera",))
    fx["camera_portrait_48x128"] = Fixture(spheres, cam=F.camera(48, 128), tags=("shape",))
    fx["camera_200x1"] = Fixture(spheres, cam=F.camera(200, 1), tags=("shape",))
    fx["dof_off_origin"] = Fixture(spheres, cam=F.camera(W, H, position=(0.3, -0.2, -1.0), focal_length=4.0, aperture_radius=0.2), tags=("camera",))
    fx["dof_aperture_2"] = Fixture(spheres, cam=F.camera(W, H, aperture_radius=2.0), tags=("camera",))
    fx["dof_focal_0"] = Fixture(spheres, cam=F.camera(W, H, focal_length=0.0, aperture_radius=0.5), tags=("camera",))
    fx["two_grids_emitter"] = Fixture(two_mesh_scene()[:3] + [("sphere", (0.0, 0.9, 4.0), 0.35, ("Emission", (8.0, 8.0, 8.0), (1.0, 1.0, 1.0), 0.0, 0.0))]
                                      + BOX, tags=("last_bounce",))
    return fx


FIXTURES = fixtures()


def tagged(tag: str) -> list:
    return [k for k, f in FIXTURES.items() if tag in f.tags]


def origin_camera(cam: dict) -> dict:
    """The camera every other scene test uses, at this fixture's frame size."""
    return F.camera(cam["width"], cam["height"])
