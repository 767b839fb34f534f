"""ctypes binding of tests/tex_oracle.cpp: the CPU oracle with colour textures (test infrastructure only).

The library is compiled on first use into a directory under the system's temporary directory (keyed by the hash of the
sources), so the test tree is never written to.  It contains its own copy of the oracle, so its scenes are built through it.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "tex_oracle.cpp")
_DEPS = (_SRC, os.path.join(_HERE, "env_oracle.cpp"), os.path.join(os.path.dirname(_HERE), "oracle", "raymond_oracle.cpp"))
_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    h = hashlib.sha256()
    for p in _DEPS:
        with open(p, "rb") as f:
            h.update(f.read())
    out_dir = os.path.join(tempfile.gettempdir(), f"raymond_tex_oracle_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, f"libtex_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        tmp = f"{so}.{os.getpid()}.tmp"
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-shared", "-o", tmp,
                        _SRC, "-lm"], check=True)
        os.replace(tmp, so)
    L = C.CDLL(so, mode=os.RTLD_LOCAL)
    vp, sz = C.c_void_p, C.c_size_t
    L.rmo_mesh_from_triangles.restype = vp
    L.rmo_mesh_from_triangles.argtypes = [vp, sz]
    L.rmo_mesh_destroy.argtypes = [vp]
    L.rmo_grid_build.restype = vp
    L.rmo_grid_build.argtypes = [vp, C.POINTER(C.c_int)]
    L.rmo_grid_destroy.argtypes = [vp]
    L.rmo_scene_create.restype = vp
    L.rmo_scene_destroy.argtypes = [vp]
    L.rmo_scene_add_sphere.argtypes = [vp, O.Vec3, C.c_double, C.POINTER(O.MaterialC)]
    L.rmo_scene_add_plane.argtypes = [vp, O.Vec3, O.Vec3, C.POINTER(O.MaterialC)]
    L.rmo_scene_add_grid.argtypes = [vp, vp, C.POINTER(O.MaterialC)]
    L.rmoe_env_create.restype = vp
    L.rmoe_env_create.argtypes = [vp, sz, sz, C.c_double, C.c_double]
    L.rmoe_env_destroy.argtypes = [vp]
    L.rmot_tex_create.restype = vp
    L.rmot_tex_create.argtypes = [vp, sz, sz, C.c_double, C.c_double]
    L.rmot_tex_destroy.argtypes = [vp]
    L.rmot_tex_lookup.argtypes = [vp, vp, sz, vp]
    L.rmot_sphere_uv.argtypes = [vp, sz, vp]
    L.rmot_plane_uv.argtypes = [vp, vp, vp, sz, vp]
    L.rmot_triangle_uv.argtypes = [vp, vp, sz, vp]
    L.rmot_render_sample.restype = C.c_int
    L.rmot_render_sample.argtypes = [vp, vp, vp, sz, C.POINTER(O.SettingsC), C.c_uint64, C.c_uint32, C.c_uint32, C.c_int, vp,
                                     C.POINTER(O.CountersC)]
    _lib = L
    return L


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _f64(a, cols):
    return np.ascontiguousarray(a, dtype=np.float64).reshape(-1, cols)


class Texture:
    """The texture of rm_texture (include/raymond.h): (H, W, 3) texels, taken as f32, and the uv scale (su, sv)."""

    def __init__(self, image, scale=(1.0, 1.0)):
        t = np.ascontiguousarray(image, dtype=np.float32)
        assert t.ndim == 3 and t.shape[2] == 3
        self.image, self.scale = t, (float(scale[0]), float(scale[1]))
        self._h = lib().rmot_tex_create(_ptr(t), t.shape[1], t.shape[0], *self.scale)

    def lookup(self, st) -> np.ndarray:
        """T(s, t) for (n, 2) uv pairs."""
        d = _f64(st, 2)
        out = np.zeros((d.shape[0], 3))
        lib().rmot_tex_lookup(self._h, _ptr(d), d.shape[0], _ptr(out))
        return out

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.rmot_tex_destroy(self._h)
            self._h = None


def sphere_uv(normals) -> np.ndarray:
    n = _f64(normals, 3)
    out = np.zeros((n.shape[0], 2))
    lib().rmot_sphere_uv(_ptr(n), n.shape[0], _ptr(out))
    return out


def plane_uv(origin, normal, frags) -> np.ndarray:
    o, nn, p = _f64(origin, 3), _f64(normal, 3), _f64(frags, 3)
    out = np.zeros((p.shape[0], 2))
    lib().rmot_plane_uv(_ptr(o), _ptr(nn), _ptr(p), p.shape[0], _ptr(out))
    return out


def triangle_uv(tris, points) -> np.ndarray:
    """(s, t) of point i on (n, 33) reference-layout triangle record i."""
    t, p = _f64(tris, O.TRI_DOUBLES), _f64(points, 3)
    assert t.shape[0] == p.shape[0]
    out = np.zeros((p.shape[0], 2))
    lib().rmot_triangle_uv(_ptr(t), _ptr(p), p.shape[0], _ptr(out))
    return out


class Scene:
    """A fixture scene (raymond_b200.fixtures object tuples) with textures {object index: Texture} and an environment map
    ((image, scale, rotation), or None: a 1 x 1 black map, which renders as the oracle without one)."""

    def __init__(self, objects, textures: dict, env=None):
        L = lib()
        self.textures = dict(textures)
        img, scale, rot = env if env is not None else (np.zeros((1, 1, 3), dtype=np.float32), 1.0, 0.0)
        self._env_img = np.ascontiguousarray(img, dtype=np.float32)
        self._env = L.rmoe_env_create(_ptr(self._env_img), self._env_img.shape[1], self._env_img.shape[0], float(scale), float(rot))
        self._h = L.rmo_scene_create()
        self._grids = []
        self.n = len(objects)
        for o in objects:
            if o[0] == "sphere":
                m = O._mat(o[3])
                L.rmo_scene_add_sphere(self._h, O.Vec3(*o[1]), float(o[2]), C.byref(m))
            elif o[0] == "plane":
                m = O._mat(o[3])
                L.rmo_scene_add_plane(self._h, O.Vec3(*o[1]), O.Vec3(*o[2]), C.byref(m))
            else:
                t = np.ascontiguousarray(o[1], dtype=np.float64).reshape(-1, O.TRI_DOUBLES)
                mesh = L.rmo_mesh_from_triangles(_ptr(t), t.shape[0])
                st = C.c_int(0)
                g = L.rmo_grid_build(mesh, C.byref(st))
                L.rmo_mesh_destroy(mesh)
                assert g, f"grid build: oracle status {st.value}"
                self._grids.append(g)
                m = O._mat(o[2])
                L.rmo_scene_add_grid(self._h, g, C.byref(m))

    def render_sample(self, cam: dict, sample: int, *, seed: int, bounce_limit: int = 5, drop_nonfinite: bool = True,
                      draws: str = "f64", threads: int = 0):
        """One sample per pixel (global sample index `sample`): (H x W x 3 radiance, counters)."""
        assert draws in O.DRAWS, draws
        s = O.settings_c(cam, 1, (32, 32), bounce_limit, 1)
        out = np.zeros((s.camera.height, s.camera.width, 3))
        cnt = O.CountersC()
        flags = (1 if drop_nonfinite else 0) | (2 if draws == "f32" else 0)
        handles = (C.c_void_p * max(self.n, 1))(*[self.textures[i]._h if i in self.textures else None for i in range(self.n)])
        lib().rmot_render_sample(self._h, self._env, handles, self.n, C.byref(s), seed, sample, flags, threads or (os.cpu_count() or 1),
                                 _ptr(out), C.byref(cnt))
        return out, cnt.as_dict()

    def __del__(self):
        if _lib is not None:
            if getattr(self, "_h", None):
                _lib.rmo_scene_destroy(self._h)
                self._h = None
            if getattr(self, "_env", None):
                _lib.rmoe_env_destroy(self._env)
                self._env = None
            for g in getattr(self, "_grids", []):
                _lib.rmo_grid_destroy(g)
            self._grids = []
