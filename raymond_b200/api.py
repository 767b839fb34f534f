"""Python host mirror of the reference's scene / camera / render-tile API over the C ABI.

Same names and argument meaning as the reference (Nyrox/raymond):
    Scene, Object push order, Geometry {Plane, Sphere, Grid}      core/src/scene.rs
    Mesh.load_ply / Mesh.new / bake_transform                     core/src/geometry/mesh.rs
    AccGrid.build_from_mesh                                       core/src/geometry/acc_grid.rs
    Material {Diffuse, Metal, Emission}                           core/src/lib.rs:21-26
    CameraSettings, Settings, render_tiled, TaskHandle, Message   src/trace.rs:32-230
    Tile                                                          core/src/tile.rs

Everything that computes goes through libraymond_cuda.so (include/raymond.h); there is no
CPU implementation here.  Importing this module loads the library and raises if it is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# RAYMOND_CUDA_LIB selects another build of the same library (kernel tuning experiments); there is still no CPU path
LIB_PATH = os.environ.get("RAYMOND_CUDA_LIB") or os.path.join(_HERE, "libraymond_cuda.so")

TRI_DOUBLES = 33


class RaymondError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"raymond status {status}: {message}")
        self.status = status


# status codes (include/raymond.h)
RM_OK = 0
RM_ERR_INVALID_ARGUMENT = -1
RM_ERR_IO = -2
RM_ERR_PLY = -3
RM_ERR_GRID_INDEX_OOB = -4
RM_ERR_DEGENERATE_BOUNDS = -5
RM_ERR_GRID_CAST = -6
RM_ERR_CUDA = -7
RM_ERR_UNSUPPORTED = -8
RM_ERR_PROJECT = -11

PARTITION_SAMPLES = 0
PARTITION_TILES = 1
FLAG_KEEP_NONFINITE = 1
FLAG_STAGE_TIMING = 2
FLAG_COUNT_WORK = 4
FLAG_NO_RAY_BINNING = 8     # 8, 16, 32: reserved values, accepted with no effect
FLAG_FUSE_SETUP = 16
FLAG_SPLIT_SETUP = 32
PRECISION_F64 = 0
PRECISION_F32_SHADING = 1
STAGE_SLOTS = 16


class Vec3C(C.Structure):
    _fields_ = [("x", C.c_double), ("y", C.c_double), ("z", C.c_double)]


class AabbC(C.Structure):
    _fields_ = [("min", Vec3C), ("max", Vec3C)]


class MaterialC(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("reserved", C.c_uint32), ("a", Vec3C), ("b", Vec3C), ("p0", C.c_double), ("p1", C.c_double)]


class GridInfoC(C.Structure):
    _fields_ = [("resolution", C.c_size_t * 3), ("cell_size", Vec3C), ("bounds", AabbC), ("cell_count", C.c_size_t),
                ("reference_count", C.c_size_t), ("triangle_count", C.c_size_t)]


class CameraSettingsC(C.Structure):
    _fields_ = [("backbuffer_width", C.c_size_t), ("backbuffer_height", C.c_size_t), ("fov_vert", C.c_double), ("position", Vec3C),
                ("focal_length", C.c_double), ("aperture_radius", C.c_double)]


class SettingsC(C.Structure):
    _fields_ = [("worker_count", C.c_size_t), ("camera_settings", CameraSettingsC), ("sample_count", C.c_size_t),
                ("samples_per_iteration", C.c_size_t), ("tile_size", C.c_size_t * 2), ("bounce_limit", C.c_size_t)]


class GpuOptionsC(C.Structure):
    _fields_ = [("device", C.c_int32), ("rank", C.c_int32), ("world_size", C.c_int32), ("partition", C.c_uint32), ("seed", C.c_uint64),
                ("stream", C.c_void_p), ("accum_device", C.c_void_p), ("batch_spp", C.c_size_t), ("flags", C.c_uint32), ("device_count", C.c_uint32),
                ("device_list", C.POINTER(C.c_int32)), ("precision", C.c_uint32), ("reserved", C.c_uint32)]


class TileC(C.Structure):
    _fields_ = [("sample_count", C.c_size_t), ("width", C.c_size_t), ("height", C.c_size_t), ("left", C.c_size_t), ("top", C.c_size_t),
                ("data", C.POINTER(Vec3C))]


class MessageC(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("reserved", C.c_uint32), ("tile", TileC)]


class StatsC(C.Structure):
    _fields_ = [("samples", C.c_uint64), ("rays", C.c_uint64), ("nonfinite_samples", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("device_ms", C.c_double), ("upload_ms", C.c_double), ("upload_bytes", C.c_uint64)]

    def as_dict(self) -> dict:
        return {n: getattr(self, n) for n, _ in self._fields_}


KERNEL_KINDS = ("setup", "traverse", "shade", "accumulate", "bin")      # kind 4 ("bin") is reserved and stays zero


class StageStatsC(C.Structure):
    _fields_ = [("ms", (C.c_double * STAGE_SLOTS) * len(KERNEL_KINDS)), ("launches", (C.c_uint64 * STAGE_SLOTS) * len(KERNEL_KINDS))] + \
               [(n, C.c_uint64 * STAGE_SLOTS) for n in ("rays", "grid_rays", "cells", "triangle_tests", "shaded_triangles", "evaluated_tests", "occupied_cells", "evaluated_test_flops")]

    def as_dict(self) -> dict:
        d = {"ms": {k: list(self.ms[i]) for i, k in enumerate(KERNEL_KINDS)},
             "launches": {k: list(self.launches[i]) for i, k in enumerate(KERNEL_KINDS)}}
        for n in ("rays", "grid_rays", "cells", "triangle_tests", "shaded_triangles", "evaluated_tests", "occupied_cells", "evaluated_test_flops"):
            d[n] = list(getattr(self, n))
        return d


TILE_CALLBACK = C.CFUNCTYPE(None, C.POINTER(TileC), C.c_void_p)

# every symbol include/raymond.h declares (tests check the library exports them all)
ABI_SYMBOLS = [
    "rm_last_error", "rm_last_status", "rm_abi_version",
    "rm_mesh_from_triangles", "rm_mesh_load_ply", "rm_mesh_translate", "rm_mesh_triangle_count", "rm_mesh_bounds", "rm_mesh_triangles",
    "rm_mesh_destroy", "rm_grid_build", "rm_grid_build_on_device", "rm_grid_retain", "rm_grid_release", "rm_grid_get_info", "rm_grid_get_cells",
    "rm_scene_create", "rm_scene_add_sphere", "rm_scene_add_plane", "rm_scene_add_grid", "rm_scene_object_count", "rm_scene_destroy",
    "rm_scene_intersect", "rm_tile_free", "rm_render_tiled", "rm_task_poll", "rm_task_await", "rm_task_set_callback", "rm_task_pump",
    "rm_task_finished", "rm_task_stats", "rm_task_destroy", "rm_device_scene_create", "rm_device_scene_destroy",
    "rm_device_scene_intersect", "rm_primary_rays_device", "rm_renderer_create", "rm_renderer_create_on", "rm_renderer_render",
    "rm_renderer_accum_device", "rm_renderer_clear", "rm_renderer_sync", "rm_renderer_read_sums", "rm_renderer_read_frame",
    "rm_renderer_stats", "rm_renderer_stage_stats", "rm_renderer_destroy", "rm_tile_layout", "rm_renderer_read_rgb8", "rm_tonemap_rgb8",
    "rm_write_png", "rm_project_load_scene", "rm_message_to_json", "rm_release_cached_memory", "rm_measure_fp64_rate",
]

_lib = None


def lib():
    """Load libraymond_cuda.so (built in-tree by raymond_b200.build). No fallback: missing library = error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RaymondError(RM_ERR_CUDA, f"{LIB_PATH} is missing — build it with `python -m raymond_b200.build` (there is no CPU path)")
    L = C.CDLL(LIB_PATH, mode=os.RTLD_LOCAL)
    vp, sz, i32 = C.c_void_p, C.c_size_t, C.c_int
    P = C.POINTER
    sig = {
        "rm_last_error": (C.c_char_p, []),
        "rm_last_status": (i32, []),
        "rm_abi_version": (i32, []),
        "rm_mesh_from_triangles": (vp, [vp, sz]),
        "rm_mesh_load_ply": (vp, [C.c_char_p]),
        "rm_mesh_translate": (i32, [vp, Vec3C]),
        "rm_mesh_triangle_count": (sz, [vp]),
        "rm_mesh_bounds": (i32, [vp, P(AabbC)]),
        "rm_mesh_triangles": (i32, [vp, sz, sz, vp]),
        "rm_mesh_destroy": (None, [vp]),
        "rm_grid_build": (vp, [vp, P(i32)]),
        "rm_grid_build_on_device": (vp, [vp, i32, P(i32)]),
        "rm_grid_retain": (vp, [vp]),
        "rm_grid_release": (None, [vp]),
        "rm_grid_get_info": (i32, [vp, P(GridInfoC)]),
        "rm_grid_get_cells": (i32, [vp, vp, vp]),
        "rm_scene_create": (vp, []),
        "rm_scene_add_sphere": (i32, [vp, Vec3C, C.c_double, P(MaterialC)]),
        "rm_scene_add_plane": (i32, [vp, Vec3C, Vec3C, P(MaterialC)]),
        "rm_scene_add_grid": (i32, [vp, vp, P(MaterialC)]),
        "rm_scene_object_count": (sz, [vp]),
        "rm_scene_destroy": (None, [vp]),
        "rm_scene_intersect": (i32, [vp, i32, vp, sz, vp, vp, vp]),
        "rm_tile_free": (None, [P(TileC)]),
        "rm_render_tiled": (vp, [vp, P(SettingsC), P(GpuOptionsC)]),
        "rm_task_poll": (i32, [vp, P(MessageC)]),
        "rm_task_await": (i32, [vp, vp]),
        "rm_task_set_callback": (i32, [vp, TILE_CALLBACK, vp]),
        "rm_task_pump": (i32, [vp]),
        "rm_task_finished": (i32, [vp]),
        "rm_task_stats": (i32, [vp, P(StatsC)]),
        "rm_task_destroy": (None, [vp]),
        "rm_device_scene_create": (vp, [vp, i32]),
        "rm_device_scene_destroy": (None, [vp]),
        "rm_device_scene_intersect": (i32, [vp, vp, sz, vp, vp, vp, vp]),
        "rm_primary_rays_device": (i32, [P(CameraSettingsC), i32, vp, vp]),
        "rm_renderer_create": (vp, [vp, P(SettingsC), P(GpuOptionsC)]),
        "rm_renderer_create_on": (vp, [vp, P(SettingsC), P(GpuOptionsC)]),
        "rm_renderer_render": (i32, [vp, sz, sz, sz]),
        "rm_renderer_accum_device": (vp, [vp]),
        "rm_renderer_clear": (i32, [vp]),
        "rm_renderer_sync": (i32, [vp]),
        "rm_renderer_read_sums": (i32, [vp, vp]),
        "rm_renderer_read_frame": (i32, [vp, sz, vp]),
        "rm_renderer_read_rgb8": (i32, [vp, sz, C.c_double, C.c_double, vp]),
        "rm_tonemap_rgb8": (i32, [vp, sz, C.c_double, C.c_double, i32, vp]),
        "rm_write_png": (i32, [C.c_char_p, vp, sz, sz]),
        "rm_project_load_scene": (vp, [C.c_char_p, P(i32)]),
        "rm_message_to_json": (sz, [P(MessageC), C.c_char_p, sz]),
        "rm_release_cached_memory": (i32, []),
        "rm_measure_fp64_rate": (i32, [i32, C.POINTER(C.c_double)]),
        "rm_renderer_stats": (i32, [vp, P(StatsC)]),
        "rm_renderer_stage_stats": (i32, [vp, P(StageStatsC)]),
        "rm_renderer_destroy": (None, [vp]),
        "rm_tile_layout": (sz, [P(SettingsC), vp, sz]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def last_error() -> str:
    return (lib().rm_last_error() or b"").decode("utf-8", "replace")


def _check(status: int) -> None:
    if status < 0:
        raise RaymondError(status, last_error())


def _require(handle, what: str, status: int = RM_ERR_CUDA):
    if not handle:
        st = lib().rm_last_status()
        raise RaymondError(st if st < 0 else status, f"{what}: {last_error()}")
    return handle


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _v3(v) -> Vec3C:
    return Vec3C(float(v[0]), float(v[1]), float(v[2]))


# ---------------------------------------------------------------------------- Material

@dataclass(frozen=True)
class Material:
    """enum Material (core/src/lib.rs:21-26)."""
    kind: int
    a: tuple
    b: tuple = (0.0, 0.0, 0.0)
    p0: float = 0.0
    p1: float = 0.0

    @staticmethod
    def Diffuse(color, roughness: float) -> "Material":
        return Material(0, tuple(map(float, color)), (0.0, 0.0, 0.0), float(roughness), 0.0)

    @staticmethod
    def Metal(color, roughness: float) -> "Material":
        return Material(1, tuple(map(float, color)), (0.0, 0.0, 0.0), float(roughness), 0.0)

    @staticmethod
    def Emission(e, b=(1.0, 1.0, 1.0), p0: float = 0.0, p1: float = 0.0) -> "Material":
        return Material(2, tuple(map(float, e)), tuple(map(float, b)), float(p0), float(p1))

    @staticmethod
    def from_fixture(m) -> "Material":
        if m[0] == "Diffuse":
            return Material.Diffuse(m[1], m[2])
        if m[0] == "Metal":
            return Material.Metal(m[1], m[2])
        if m[0] == "Emission":
            return Material.Emission(m[1], m[2], m[3], m[4])
        raise ValueError(f"unknown material {m[0]!r}")

    def _c(self) -> MaterialC:
        return MaterialC(self.kind, 0, _v3(self.a), _v3(self.b), self.p0, self.p1)


# ---------------------------------------------------------------------------- Mesh / AccGrid

class Mesh:
    """Mesh (core/src/geometry/mesh.rs:10-13)."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def new(cls, triangles: np.ndarray) -> "Mesh":
        """Mesh::new(Vec<Triangle>): triangles as (n, 33) f64 in the reference's Triangle layout."""
        t = np.ascontiguousarray(triangles, dtype=np.float64).reshape(-1, TRI_DOUBLES)
        return cls(_require(lib().rm_mesh_from_triangles(_ptr(t), t.shape[0]), "Mesh::new", RM_ERR_INVALID_ARGUMENT))

    @classmethod
    def load_ply(cls, path: str) -> "Mesh":
        h = lib().rm_mesh_load_ply(os.fsencode(path))
        if not h:
            msg = last_error()
            raise RaymondError(RM_ERR_IO if "cannot read" in msg else RM_ERR_PLY, msg)
        return cls(h)

    def bake_transform(self, translate) -> None:
        _check(lib().rm_mesh_translate(self._h, _v3(translate)))

    def __len__(self) -> int:
        return int(lib().rm_mesh_triangle_count(self._h))

    @property
    def bounding_box(self) -> np.ndarray:
        b = AabbC()
        _check(lib().rm_mesh_bounds(self._h, C.byref(b)))
        return np.array([[b.min.x, b.min.y, b.min.z], [b.max.x, b.max.y, b.max.z]])

    def triangles(self) -> np.ndarray:
        out = np.zeros((len(self), TRI_DOUBLES))
        _check(lib().rm_mesh_triangles(self._h, 0, len(self), _ptr(out)))
        return out

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rm_mesh_destroy(self._h)
            self._h = None


class AccGrid:
    """Arc<AccGrid> (core/src/geometry/acc_grid.rs:27-33)."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def build_from_mesh(cls, mesh: Mesh, device: Optional[int] = None) -> "AccGrid":
        """Consumes the mesh's triangles, like the Rust move.  `device` = CUDA ordinal builds the cell lists on the GPU
        (same grid, bit for bit); None = the host build."""
        st = C.c_int(0)
        if device is None:
            h = lib().rm_grid_build(mesh._h, C.byref(st))
        else:
            h = lib().rm_grid_build_on_device(mesh._h, int(device), C.byref(st))
        if not h:
            raise RaymondError(st.value, last_error())
        return cls(h)

    def info(self) -> dict:
        i = GridInfoC()
        _check(lib().rm_grid_get_info(self._h, C.byref(i)))
        return {"resolution": [int(x) for x in i.resolution], "cell_size": np.array([i.cell_size.x, i.cell_size.y, i.cell_size.z]),
                "bounds": np.array([[i.bounds.min.x, i.bounds.min.y, i.bounds.min.z], [i.bounds.max.x, i.bounds.max.y, i.bounds.max.z]]),
                "cell_count": int(i.cell_count), "reference_count": int(i.reference_count), "triangle_count": int(i.triangle_count)}

    def cells(self):
        """(cell_start[cell_count + 1], references[reference_count]) — compressed-row image of cells/mapping_table."""
        i = self.info()
        start = np.zeros(i["cell_count"] + 1, dtype=np.uint32)
        refs = np.zeros(max(i["reference_count"], 1), dtype=np.uint32)
        _check(lib().rm_grid_get_cells(self._h, _ptr(start), _ptr(refs)))
        return start, refs[:i["reference_count"]]

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rm_grid_release(self._h)
            self._h = None


# ---------------------------------------------------------------------------- Scene

class Scene:
    """Scene { objects } (core/src/scene.rs:42-52); objects are pushed in order."""

    def __init__(self):
        self._h = _require(lib().rm_scene_create(), "Scene::new", RM_ERR_INVALID_ARGUMENT)
        self._grids = []

    def push_sphere(self, origin, radius: float, material: Material) -> None:
        m = material._c()
        _check(lib().rm_scene_add_sphere(self._h, _v3(origin), float(radius), C.byref(m)))

    def push_plane(self, origin, normal, material: Material) -> None:
        m = material._c()
        _check(lib().rm_scene_add_plane(self._h, _v3(origin), _v3(normal), C.byref(m)))

    def push_grid(self, grid: AccGrid, material: Material) -> None:
        m = material._c()
        _check(lib().rm_scene_add_grid(self._h, grid._h, C.byref(m)))
        self._grids.append(grid)

    @classmethod
    def from_fixture(cls, objects: Sequence) -> "Scene":
        """Build from raymond_b200.fixtures object tuples."""
        s = cls()
        for o in objects:
            if o[0] == "sphere":
                s.push_sphere(o[1], o[2], Material.from_fixture(o[3]))
            elif o[0] == "plane":
                s.push_plane(o[1], o[2], Material.from_fixture(o[3]))
            elif o[0] == "grid":
                s.push_grid(AccGrid.build_from_mesh(Mesh.new(o[1])), Material.from_fixture(o[2]))
            else:
                raise ValueError(f"unknown object {o[0]!r}")
        return s

    @classmethod
    def load_project(cls, path: str) -> "Scene":
        """Project::load(path)?.build_scene() (core/src/project.rs:33-57)."""
        st = C.c_int(0)
        h = lib().rm_project_load_scene(os.fsencode(path), C.byref(st))
        if not h:
            raise RaymondError(st.value, last_error())
        s = cls.__new__(cls)
        s._h = h
        s._grids = []
        return s

    def __len__(self) -> int:
        return int(lib().rm_scene_object_count(self._h))

    def intersect(self, rays: np.ndarray, device: int = 0):
        """Scene::intersect over (n, 6) f64 host rays -> (object index or -1, subobject index, distance)."""
        r = np.ascontiguousarray(rays, dtype=np.float64).reshape(-1, 6)
        n = r.shape[0]
        obj = np.full(n, -1, dtype=np.int64)
        sub = np.zeros(n, dtype=np.uint64)
        t = np.zeros(n)
        _check(lib().rm_scene_intersect(self._h, device, _ptr(r), n, _ptr(obj), _ptr(sub), _ptr(t)))
        return obj, sub, t

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rm_scene_destroy(self._h)
            self._h = None


# ---------------------------------------------------------------------------- settings

@dataclass
class Transform:
    """Transform { position } (src/transform.rs:3-14)."""
    position: tuple = (0.0, 0.0, 0.0)

    @staticmethod
    def identity() -> "Transform":
        return Transform((0.0, 0.0, 0.0))


@dataclass
class CameraSettings:
    """CameraSettings (src/trace.rs:32-40)."""
    backbuffer_width: int
    backbuffer_height: int
    fov_vert: float
    transform: Transform = field(default_factory=Transform.identity)
    focal_length: float = 2.5
    aperture_radius: float = 0.0

    @staticmethod
    def from_fixture(cam: dict) -> "CameraSettings":
        return CameraSettings(cam["width"], cam["height"], cam["fov_vert"], Transform(tuple(cam.get("position", (0.0, 0.0, 0.0)))),
                              cam.get("focal_length", 2.5), cam.get("aperture_radius", 0.0))

    def _c(self) -> CameraSettingsC:
        return CameraSettingsC(int(self.backbuffer_width), int(self.backbuffer_height), float(self.fov_vert), _v3(self.transform.position),
                               float(self.focal_length), float(self.aperture_radius))


@dataclass
class Settings:
    """Settings (src/trace.rs:42-55)."""
    camera_settings: CameraSettings
    sample_count: int
    tile_size: tuple = (32, 32)
    bounce_limit: int = 5
    samples_per_iteration: int = 0
    worker_count: int = 0   # CPU threads in the reference (default num_cpus); unused by the GPU path

    def _c(self) -> SettingsC:
        return SettingsC(int(self.worker_count or (os.cpu_count() or 1)), self.camera_settings._c(), int(self.sample_count),
                         int(self.samples_per_iteration), (C.c_size_t * 2)(int(self.tile_size[0]), int(self.tile_size[1])), int(self.bounce_limit))


@dataclass
class GpuOptions:
    """rm_gpu_options: knobs with no counterpart in the reference."""
    device: int = 0
    rank: int = 0
    world_size: int = 1
    partition: int = PARTITION_SAMPLES
    seed: int = 0
    stream: int = 0
    accum_device: int = 0
    batch_spp: int = 0
    flags: int = 0
    device_count: int = 0     # render_tiled only: > 1 = that many GPUs driven from this process
    device_list: Optional[Sequence[int]] = None   # the ordinals to use (may repeat one); None = device, device+1, ...
    precision: int = PRECISION_F64

    def _c(self) -> GpuOptionsC:
        count = self.device_count
        lst = None
        if self.device_list is not None:
            count = len(self.device_list)
            lst = (C.c_int32 * max(count, 1))(*[int(d) for d in self.device_list])
        o = GpuOptionsC(self.device, self.rank, self.world_size, self.partition, self.seed, self.stream or None, self.accum_device or None,
                        self.batch_spp, self.flags, count, lst, self.precision, 0)
        o._keep = lst            # the array must outlive the call that reads the struct
        return o


def tile_layout(settings: Settings) -> np.ndarray:
    """Tile rectangles (left, top, width, height) in the reference's queue order (src/trace.rs:142-173)."""
    s = settings._c()
    n = lib().rm_tile_layout(C.byref(s), None, 0)
    out = np.zeros((max(n, 1), 4), dtype=np.uint64)
    lib().rm_tile_layout(C.byref(s), _ptr(out), n)
    return out[:n].astype(np.int64)


# ---------------------------------------------------------------------------- Tile / Message / TaskHandle

@dataclass
class Tile:
    """Tile (core/src/tile.rs:6-14): `data` is the running SUM, (height, width, 3) f64."""
    sample_count: int
    width: int
    height: int
    left: int
    top: int
    data: np.ndarray


@dataclass
class Message:
    """enum Message { TileFinished(Tile), TileProgressed(Tile) } (src/trace.rs:62-66)."""
    kind: str
    tile: Tile


def message_to_json(kind: str, tile: Tile) -> str:
    """The tile message as the reference puts it on the wire (server/src/protocol.rs:9-14)."""
    data = np.ascontiguousarray(tile.data, dtype=np.float64)
    m = MessageC(0 if kind == "TileFinished" else 1, 0,
                 TileC(tile.sample_count, tile.width, tile.height, tile.left, tile.top, C.cast(data.ctypes.data, C.POINTER(Vec3C))))
    n = lib().rm_message_to_json(C.byref(m), None, 0)
    buf = C.create_string_buffer(n + 1)
    lib().rm_message_to_json(C.byref(m), buf, n + 1)
    return buf.value.decode("ascii")


def _tile_from_c(t: TileC) -> Tile:
    n = t.width * t.height
    data = np.ctypeslib.as_array(C.cast(t.data, C.POINTER(C.c_double)), shape=(n * 3,)).copy().reshape(t.height, t.width, 3) if n else np.zeros((0, 0, 3))
    return Tile(int(t.sample_count), int(t.width), int(t.height), int(t.left), int(t.top), data)


class TaskHandle:
    """TaskHandle (src/trace.rs:70-135)."""

    def __init__(self, handle, settings: Settings, keepalive=None):
        self._h = handle
        self.settings = settings
        self._callback = None
        self._c_callback = None
        self._keepalive = keepalive

    def poll(self) -> Optional[Message]:
        m = MessageC()
        got = lib().rm_task_poll(self._h, C.byref(m))
        _check(got)
        if not got:
            return None
        msg = Message("TileFinished" if m.kind == 0 else "TileProgressed", _tile_from_c(m.tile))
        lib().rm_tile_free(C.byref(m.tile))
        return msg

    def await_(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        """r#await(): block, then the averaged frame as (H, W, 3) f64 (row-major W*H Vec<Vector3>).  `out` = a C-contiguous f64
        array of that shape to write into (a caller rendering frame after frame keeps one, as the C ABI's caller does)."""
        cs = self.settings.camera_settings
        shape = (cs.backbuffer_height, cs.backbuffer_width, 3)
        if out is None:
            out = np.zeros(shape)
        elif out.shape != shape or out.dtype != np.float64 or not out.flags.c_contiguous:
            raise ValueError(f"await_: out must be a C-contiguous float64 array of shape {shape}")
        _check(lib().rm_task_await(self._h, _ptr(out)))
        return out

    def set_callback(self, callback: Optional[Callable[[Tile], None]]) -> None:
        self._callback = callback
        if callback is None:
            self._c_callback = C.cast(None, TILE_CALLBACK)
        else:
            self._c_callback = TILE_CALLBACK(lambda tp, _u: callback(_tile_from_c(tp.contents)))
        _check(lib().rm_task_set_callback(self._h, self._c_callback, None))

    def async_await(self) -> int:
        """Deliver queued TileProgressed tiles to the callback (src/trace.rs:119-134)."""
        n = lib().rm_task_pump(self._h)
        _check(n)
        return n

    def finished(self) -> bool:
        return bool(lib().rm_task_finished(self._h))

    def stats(self) -> dict:
        s = StatsC()
        _check(lib().rm_task_stats(self._h, C.byref(s)))
        return s.as_dict()

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rm_task_destroy(self._h)
            self._h = None


def render_tiled(scene: Scene, settings: Settings, options: Optional[GpuOptions] = None) -> TaskHandle:
    """render_tiled(scene, settings) -> TaskHandle (src/trace.rs:137-230). Returns immediately."""
    s = settings._c()
    o = (options or GpuOptions())._c()
    h = _require(lib().rm_render_tiled(scene._h, C.byref(s), C.byref(o)), "render_tiled")
    return TaskHandle(h, settings)


def tonemap(frame: np.ndarray, exposure: float = 1.0, gamma: float = 2.2, device: int = 0) -> np.ndarray:
    """cli_old's display transform (cli_old/src/main.rs:157-181) of an averaged (H, W, 3) f64 frame -> uint8, on the GPU."""
    f = np.ascontiguousarray(frame, dtype=np.float64)
    out = np.zeros(f.shape, dtype=np.uint8)
    _check(lib().rm_tonemap_rgb8(_ptr(f), f.size // 3, exposure, gamma, device, _ptr(out)))
    return out


def release_cached_memory() -> None:
    """Return the cached device pool and pinned staging blocks to the driver."""
    _check(lib().rm_release_cached_memory())


def measure_fp64_rate(device: int = 0) -> float:
    """Sustained f64 operation rate (independent DADD / DMUL, no FMA) of `device` in Gop/s: the roofline's compute ceiling."""
    g = C.c_double(0.0)
    _check(lib().rm_measure_fp64_rate(device, C.byref(g)))
    return g.value


def write_png(path: str, rgb8: np.ndarray) -> None:
    """image.save(path) (cli_old/src/main.rs:194-197): (H, W, 3) uint8 -> 8-bit RGB PNG."""
    a = np.ascontiguousarray(rgb8, dtype=np.uint8)
    _check(lib().rm_write_png(os.fsencode(path), _ptr(a), a.shape[1], a.shape[0]))


# ---------------------------------------------------------------------------- device-level interface

class DeviceScene:
    """A Scene flattened and resident in HBM."""

    def __init__(self, scene: Scene, device: int = 0):
        self._h = _require(lib().rm_device_scene_create(scene._h, device), "rm_device_scene_create")
        self.device = device

    def intersect_device(self, rays_ptr: int, count: int, obj_ptr: int, sub_ptr: int, dist_ptr: int, stream: int = 0) -> None:
        """Scene::intersect on device-resident rays/results (raw device pointers); asynchronous on `stream`."""
        _check(lib().rm_device_scene_intersect(self._h, rays_ptr, count, obj_ptr or None, sub_ptr or None, dist_ptr or None, stream or None))

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rm_device_scene_destroy(self._h)
            self._h = None


def primary_rays_device(camera: CameraSettings, device: int, rays_ptr: int, stream: int = 0) -> None:
    c = camera._c()
    _check(lib().rm_primary_rays_device(C.byref(c), device, rays_ptr, stream or None))


class Renderer:
    """The wavefront path tracer on one GPU: render sample ranges into a device accumulator."""

    def __init__(self, scene, settings: Settings, options: Optional[GpuOptions] = None):
        self.settings = settings
        self.options = options or GpuOptions()
        s = settings._c()
        o = self.options._c()
        if isinstance(scene, DeviceScene):
            self._scene = scene
            self._h = _require(lib().rm_renderer_create_on(scene._h, C.byref(s), C.byref(o)), "rm_renderer_create_on")
        else:
            self._scene = None
            self._h = _require(lib().rm_renderer_create(scene._h, C.byref(s), C.byref(o)), "rm_renderer_create")

    def render(self, first_sample: int, count: int, stride: int = 1) -> None:
        _check(lib().rm_renderer_render(self._h, first_sample, count, stride))

    @property
    def accum_ptr(self) -> int:
        return int(lib().rm_renderer_accum_device(self._h) or 0)

    def clear(self) -> None:
        _check(lib().rm_renderer_clear(self._h))

    def sync(self) -> None:
        _check(lib().rm_renderer_sync(self._h))

    def _frame(self) -> np.ndarray:
        cs = self.settings.camera_settings
        return np.zeros((cs.backbuffer_height, cs.backbuffer_width, 3))

    def read_sums(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        out = self._frame() if out is None else out
        _check(lib().rm_renderer_read_sums(self._h, _ptr(out)))
        return out

    def read_frame(self, sample_count: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        out = self._frame() if out is None else out
        _check(lib().rm_renderer_read_frame(self._h, sample_count, _ptr(out)))
        return out

    def read_rgb8(self, sample_count: int, exposure: float = 1.0, gamma: float = 2.2) -> np.ndarray:
        """sum / sample_count -> cli_old's tonemap (src cli_old/src/main.rs:157-181) on the GPU -> (H, W, 3) uint8."""
        cs = self.settings.camera_settings
        out = np.zeros((cs.backbuffer_height, cs.backbuffer_width, 3), dtype=np.uint8)
        _check(lib().rm_renderer_read_rgb8(self._h, sample_count, exposure, gamma, _ptr(out)))
        return out

    def stats(self) -> dict:
        s = StatsC()
        _check(lib().rm_renderer_stats(self._h, C.byref(s)))
        return s.as_dict()

    def stage_stats(self) -> dict:
        """Per wavefront stage and kernel kind: ms / launches (FLAG_STAGE_TIMING); rays, grid_rays, shaded_triangles;
        cells / triangle_tests (FLAG_COUNT_WORK)."""
        s = StageStatsC()
        _check(lib().rm_renderer_stage_stats(self._h, C.byref(s)))
        return s.as_dict()

    def close(self) -> None:
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rm_renderer_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()
