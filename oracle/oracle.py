"""ctypes binding of the CPU oracle (oracle/raymond_oracle.cpp).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  Nothing under raymond_b200/
imports this module.  PARITY UNPINNED — see the header of raymond_oracle.cpp.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libraymond_oracle.so")

TRI_DOUBLES = 33  # 3 vertices x (position 3, normal 3, uv 2, tangent 3) — reference Triangle, 264 B


class Vec3(C.Structure):
    _fields_ = [("x", C.c_double), ("y", C.c_double), ("z", C.c_double)]


class MaterialC(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("reserved", C.c_uint32), ("a", Vec3), ("b", Vec3), ("p0", C.c_double), ("p1", C.c_double)]


class CameraC(C.Structure):
    _fields_ = [("width", C.c_size_t), ("height", C.c_size_t), ("fov_vert", C.c_double), ("position", Vec3),
                ("focal_length", C.c_double), ("aperture_radius", C.c_double)]


class SettingsC(C.Structure):
    _fields_ = [("worker_count", C.c_size_t), ("camera", CameraC), ("sample_count", C.c_size_t),
                ("samples_per_iteration", C.c_size_t), ("tile_size", C.c_size_t * 2), ("bounce_limit", C.c_size_t)]


class CountersC(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays", "cells", "tri_tests", "grid_hits", "aabb_tests", "shaded_tri", "nonfinite", "samples")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


def build(force: bool = False) -> str:
    """Compile the oracle with its Makefile (g++ -O2 -ffp-contract=off)."""
    src = os.path.join(_HERE, "raymond_oracle.cpp")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE, "-B" if force else "-s"], check=True, stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_LIB_PATH, mode=os.RTLD_LOCAL)
    vp, dp, sz = C.c_void_p, C.POINTER(C.c_double), C.c_size_t
    L.rmo_mesh_load_ply.restype = vp
    L.rmo_mesh_load_ply.argtypes = [C.c_char_p, C.POINTER(C.c_int)]
    L.rmo_mesh_from_triangles.restype = vp
    L.rmo_mesh_from_triangles.argtypes = [vp, sz]
    L.rmo_mesh_translate.argtypes = [vp, C.c_double, C.c_double, C.c_double]
    L.rmo_mesh_count.restype = sz
    L.rmo_mesh_count.argtypes = [vp]
    L.rmo_mesh_bounds.argtypes = [vp, vp]
    L.rmo_mesh_triangles.argtypes = [vp, vp]
    L.rmo_mesh_destroy.argtypes = [vp]
    L.rmo_mesh_intersect.argtypes = [vp, vp, sz, vp, vp]
    L.rmo_grid_build.restype = vp
    L.rmo_grid_build.argtypes = [vp, C.POINTER(C.c_int)]
    L.rmo_grid_destroy.argtypes = [vp]
    L.rmo_grid_info.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.rmo_grid_tables.argtypes = [vp, vp, vp]
    L.rmo_grid_intersect.argtypes = [vp, vp, sz, vp, vp, C.POINTER(CountersC)]
    L.rmo_scene_create.restype = vp
    L.rmo_scene_destroy.argtypes = [vp]
    L.rmo_scene_add_sphere.argtypes = [vp, Vec3, C.c_double, C.POINTER(MaterialC)]
    L.rmo_scene_add_plane.argtypes = [vp, Vec3, Vec3, C.POINTER(MaterialC)]
    L.rmo_scene_add_grid.argtypes = [vp, vp, C.POINTER(MaterialC)]
    L.rmo_scene_intersect.argtypes = [vp, vp, sz, vp, vp, vp, C.POINTER(CountersC), C.c_int]
    L.rmo_scene_normal.argtypes = [vp, vp, C.c_int64, C.c_uint64, C.c_double, vp]
    L.rmo_primary_rays.argtypes = [C.POINTER(CameraC), vp, vp]
    L.rmo_camera_rays.argtypes = [C.POINTER(CameraC), C.c_uint64, C.c_uint32, vp]
    L.rmo_rng_draw.restype = C.c_double
    L.rmo_rng_draw.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
    L.rmo_rng_draw_f32.restype = C.c_double
    L.rmo_rng_draw_f32.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
    L.rmo_tile_layout.restype = sz
    L.rmo_tile_layout.argtypes = [C.POINTER(SettingsC), vp, sz]
    L.rmo_render.restype = C.c_int
    L.rmo_render.argtypes = [vp, C.POINTER(SettingsC), C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, vp, C.POINTER(CountersC)]
    L.rmo_trace_samples.argtypes = [vp, C.POINTER(SettingsC), C.c_uint64, vp, vp, sz, vp]
    _lib = L
    return L


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _rays(rays) -> np.ndarray:
    r = np.ascontiguousarray(rays, dtype=np.float64)
    assert r.ndim == 2 and r.shape[1] == 6
    return r


class OracleError(RuntimeError):
    def __init__(self, status: int, what: str):
        super().__init__(f"{what}: oracle status {status}")
        self.status = status


class Mesh:
    """Mesh (core/src/geometry/mesh.rs)."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def load_ply(cls, path: str) -> "Mesh":
        st = C.c_int(0)
        h = lib().rmo_mesh_load_ply(os.fsencode(path), C.byref(st))
        if not h:
            raise OracleError(st.value, f"load_ply({path})")
        return cls(h)

    @classmethod
    def from_triangles(cls, tris: np.ndarray) -> "Mesh":
        t = np.ascontiguousarray(tris, dtype=np.float64).reshape(-1, TRI_DOUBLES)
        return cls(lib().rmo_mesh_from_triangles(_ptr(t), t.shape[0]))

    def bake_transform(self, translate) -> None:
        lib().rmo_mesh_translate(self._h, *map(float, translate))

    def __len__(self) -> int:
        return int(lib().rmo_mesh_count(self._h))

    @property
    def bounds(self) -> np.ndarray:
        out = np.zeros(6)
        lib().rmo_mesh_bounds(self._h, _ptr(out))
        return out.reshape(2, 3)

    def triangles(self) -> np.ndarray:
        out = np.zeros((len(self), TRI_DOUBLES))
        lib().rmo_mesh_triangles(self._h, _ptr(out))
        return out

    def intersects(self, rays):
        """Brute-force Mesh::intersects (mesh.rs:23-42)."""
        r = _rays(rays)
        tri = np.full(r.shape[0], -1, dtype=np.int64)
        t = np.zeros(r.shape[0])
        lib().rmo_mesh_intersect(self._h, _ptr(r), r.shape[0], _ptr(tri), _ptr(t))
        return tri, t

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rmo_mesh_destroy(self._h)
            self._h = None


class AccGrid:
    """AccGrid (core/src/geometry/acc_grid.rs)."""

    def __init__(self, handle):
        self._h = handle

    @classmethod
    def build_from_mesh(cls, mesh: Mesh) -> "AccGrid":
        st = C.c_int(0)
        h = lib().rmo_grid_build(mesh._h, C.byref(st))
        if not h:
            raise OracleError(st.value, "AccGrid::build_from_mesh")
        return cls(h)

    def info(self) -> dict:
        res = np.zeros(3, dtype=np.uint64)
        cs = np.zeros(3)
        b = np.zeros(6)
        n = (C.c_uint64 * 3)()
        lib().rmo_grid_info(self._h, _ptr(res), _ptr(cs), _ptr(b), C.addressof(n), C.addressof(n) + 8, C.addressof(n) + 16)
        return {"resolution": [int(x) for x in res], "cell_size": cs, "bounds": b.reshape(2, 3),
                "cell_count": int(n[0]), "table_len": int(n[1]), "reference_count": int(n[1]) - int(n[0]),
                "triangle_count": int(n[2])}

    def tables(self):
        """(cells, mapping_table) exactly as the reference stores them."""
        i = self.info()
        cells = np.zeros(i["cell_count"], dtype=np.uint64)
        table = np.zeros(i["table_len"], dtype=np.uint64)
        lib().rmo_grid_tables(self._h, _ptr(cells), _ptr(table))
        return cells, table

    def csr(self):
        """The same contents as (cell_start[ncells+1], references[nrefs])."""
        cells, table = self.tables()
        n = cells.shape[0]
        counts = table[cells].astype(np.int64)
        start = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(counts, out=start[1:])
        mask = np.ones(table.shape[0], dtype=bool)
        mask[cells] = False
        return start.astype(np.uint32), table[mask].astype(np.uint32)

    def intersects(self, rays):
        """AccGrid::intersects; tri -1 = miss, -2 = the reference would panic."""
        r = _rays(rays)
        tri = np.full(r.shape[0], -1, dtype=np.int64)
        t = np.zeros(r.shape[0])
        cnt = CountersC()
        lib().rmo_grid_intersect(self._h, _ptr(r), r.shape[0], _ptr(tri), _ptr(t), C.byref(cnt))
        return tri, t, cnt.as_dict()

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rmo_grid_destroy(self._h)
            self._h = None


def _mat(m) -> MaterialC:
    kind = {"Diffuse": 0, "Metal": 1, "Emission": 2}[m[0]]
    if kind == 2:
        e, b, p0, p1 = m[1], m[2], m[3], m[4]
        return MaterialC(kind, 0, Vec3(*e), Vec3(*b), p0, p1)
    return MaterialC(kind, 0, Vec3(*m[1]), Vec3(0, 0, 0), m[2], 0.0)


class Scene:
    """Scene (core/src/scene.rs). Objects are given as fixture tuples, see raymond_b200/fixtures.py."""

    def __init__(self):
        self._h = lib().rmo_scene_create()
        self._keep = []
        self.n_objects = 0

    def add_sphere(self, origin, radius, material):
        m = _mat(material)
        lib().rmo_scene_add_sphere(self._h, Vec3(*origin), float(radius), C.byref(m))
        self.n_objects += 1

    def add_plane(self, origin, normal, material):
        m = _mat(material)
        lib().rmo_scene_add_plane(self._h, Vec3(*origin), Vec3(*normal), C.byref(m))
        self.n_objects += 1

    def add_grid(self, grid: AccGrid, material):
        m = _mat(material)
        lib().rmo_scene_add_grid(self._h, grid._h, C.byref(m))
        self._keep.append(grid)
        self.n_objects += 1

    def intersect(self, rays, threads: int = 1):
        r = _rays(rays)
        n = r.shape[0]
        obj = np.full(n, -1, dtype=np.int64)
        sub = np.zeros(n, dtype=np.uint64)
        t = np.zeros(n)
        cnt = CountersC()
        lib().rmo_scene_intersect(self._h, _ptr(r), n, _ptr(obj), _ptr(sub), _ptr(t), C.byref(cnt), threads)
        return obj, sub, t, cnt.as_dict()

    def normal(self, ray, obj, sub, t) -> np.ndarray:
        r = np.ascontiguousarray(ray, dtype=np.float64).reshape(6)
        out = np.zeros(3)
        lib().rmo_scene_normal(self._h, _ptr(r), int(obj), int(sub), float(t), _ptr(out))
        return out

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rmo_scene_destroy(self._h)
            self._h = None


def camera_c(cam: dict) -> CameraC:
    return CameraC(int(cam["width"]), int(cam["height"]), float(cam["fov_vert"]), Vec3(*cam.get("position", (0.0, 0.0, 0.0))),
                   float(cam.get("focal_length", 2.5)), float(cam.get("aperture_radius", 0.0)))


def settings_c(cam: dict, sample_count: int, tile_size=(32, 32), bounce_limit: int = 5, worker_count: int = 0,
               samples_per_iteration: int = 0) -> SettingsC:
    wc = worker_count or (os.cpu_count() or 1)
    return SettingsC(wc, camera_c(cam), int(sample_count), int(samples_per_iteration),
                     (C.c_size_t * 2)(int(tile_size[0]), int(tile_size[1])), int(bounce_limit))


def primary_rays(cam: dict, jitter: np.ndarray | None = None) -> np.ndarray:
    """generate_primary_ray for the whole frame (row-major). jitter None = pixel centres."""
    c = camera_c(cam)
    n = c.width * c.height
    out = np.zeros((n, 6))
    j = None
    if jitter is not None:
        j = np.ascontiguousarray(jitter, dtype=np.float64).reshape(n, 2)
    lib().rmo_primary_rays(C.byref(c), _ptr(j) if j is not None else None, _ptr(out))
    return out


def camera_rays(cam: dict, seed: int, sample: int) -> np.ndarray:
    c = camera_c(cam)
    out = np.zeros((c.width * c.height, 6))
    lib().rmo_camera_rays(C.byref(c), seed, sample, _ptr(out))
    return out


DRAWS = ("f64", "f32")


def rng_draw(seed, pixel, sample, depth, index, draws: str = "f64") -> float:
    """Draw `index` of (seed; pixel, sample, depth).  draws="f32": the stream of the product's f32 shading mode (23-bit
    uniforms, all three shading draws of a depth from one Philox block); its camera draws (depth 0) are the f64 ones."""
    assert draws in DRAWS, draws
    f = lib().rmo_rng_draw_f32 if draws == "f32" else lib().rmo_rng_draw
    return float(f(seed, pixel, sample, depth, index))


def tile_layout(cam: dict, tile_size) -> np.ndarray:
    s = settings_c(cam, 1, tile_size)
    n = lib().rmo_tile_layout(C.byref(s), None, 0)
    out = np.zeros((n, 4), dtype=np.uint64)
    lib().rmo_tile_layout(C.byref(s), _ptr(out), n)
    return out.astype(np.int64)


def render(scene: Scene, cam: dict, sample_count: int, *, seed: int = 0, tile_size=(32, 32), bounce_limit: int = 5,
           worker_count: int = 0, first_sample: int = 0, sample_stride: int = 1, drop_nonfinite: bool = True, draws: str = "f64"):
    """render_tiled + await.  Returns (running sums H x W x 3, counters).  draws="f32": the shading draws are those of the
    product's f32 shading mode (see rng_draw), so that mode can be compared path for path; the arithmetic stays f64."""
    assert draws in DRAWS, draws
    s = settings_c(cam, sample_count, tile_size, bounce_limit, worker_count)
    W, H = s.camera.width, s.camera.height
    out = np.zeros((H, W, 3))
    cnt = CountersC()
    rc = lib().rmo_render(scene._h, C.byref(s), seed, first_sample, sample_stride,
                          (1 if drop_nonfinite else 0) | (2 if draws == "f32" else 0), _ptr(out), C.byref(cnt))
    if rc != 0:
        raise OracleError(rc, "render")
    return out, cnt.as_dict()


def trace_samples(scene: Scene, cam: dict, pixels, samples, *, seed: int = 0, bounce_limit: int = 5) -> np.ndarray:
    s = settings_c(cam, 1, (32, 32), bounce_limit, 1)
    p = np.ascontiguousarray(pixels, dtype=np.uint32)
    q = np.ascontiguousarray(samples, dtype=np.uint32)
    out = np.zeros((p.shape[0], 3))
    lib().rmo_trace_samples(scene._h, C.byref(s), seed, _ptr(p), _ptr(q), p.shape[0], _ptr(out))
    return out
