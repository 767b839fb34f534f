"""numpy restatement of the colour-texture lookup and the uv of each geometry kind of include/raymond.h (rm_texture), for the
tests.

Every operation is one f64 numpy ufunc call in the header's order (numpy never fuses a multiply-add), so the result differs
from the oracle's (glibc) and the GPU's (CUDA libdevice) only by what their atan2 / acos return, which only the sphere uses.
"""
from __future__ import annotations

import numpy as np


def tex_lookup(image, st, scale=(1.0, 1.0)) -> np.ndarray:
    """T(s, t) for (n, 2) uv pairs `st` of the (H, W, 3) texture `image` (taken as f32, widened exactly)."""
    tex = np.asarray(image, dtype=np.float32).astype(np.float64)
    H, W = tex.shape[0], tex.shape[1]
    st = np.asarray(st, dtype=np.float64).reshape(-1, 2)
    with np.errstate(invalid="ignore", over="ignore"):
        sp = st[:, 0] * float(scale[0])
        tp = st[:, 1] * float(scale[1])
    bad = ~(np.isfinite(sp) & np.isfinite(tp))
    sp = np.where(bad, 0.0, sp)
    tp = np.where(bad, 0.0, tp)
    sp = sp - np.floor(sp)
    tp = tp - np.floor(tp)
    x = sp * float(W) - 0.5
    y = (1.0 - tp) * float(H) - 0.5
    x0 = np.floor(x)
    y0 = np.floor(y)
    fx = (x - x0)[:, None]
    fy = (y - y0)[:, None]
    ix0 = x0.astype(np.int64) % W
    ix1 = (x0.astype(np.int64) + 1) % W
    iy0 = y0.astype(np.int64) % H
    iy1 = (y0.astype(np.int64) + 1) % H
    t00, t01, t10, t11 = tex[iy0, ix0], tex[iy0, ix1], tex[iy1, ix0], tex[iy1, ix1]
    top = t00 + fx * (t01 - t00)
    bot = t10 + fx * (t11 - t10)
    out = top + fy * (bot - top)
    out[bad] = np.nan
    return out


def sphere_uv(normals) -> np.ndarray:
    n = np.asarray(normals, dtype=np.float64).reshape(-1, 3)
    with np.errstate(invalid="ignore"):
        s = 0.5 + np.arctan2(n[:, 0], n[:, 2]) / (2.0 * np.pi)
        cy = np.where(n[:, 1] < -1.0, -1.0, np.where(n[:, 1] > 1.0, 1.0, n[:, 1]))
        t = 1.0 - np.arccos(cy) / np.pi
    return np.stack([s, t], axis=-1)


def onb(n):
    """create_coordinate_system_of_n (src/trace.rs:408-416) as the kernels and the oracle evaluate it."""
    n = np.asarray(n, dtype=np.float64)
    sign = np.where(n[..., 2] > 0.0, 1.0, -1.0)
    a = -1.0 / (sign + n[..., 2])
    b = n[..., 0] * n[..., 1] * a
    tg = np.stack([1.0 + sign * n[..., 0] * n[..., 0] * a, sign * b, -sign * n[..., 0]], axis=-1)
    bt = np.stack([b, sign + n[..., 1] * n[..., 1] * a, -n[..., 1]], axis=-1)
    return tg, bt


def _dot(a, b):
    return (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]


def plane_uv(origin, normal, frags) -> np.ndarray:
    tg, bt = onb(np.asarray(normal, dtype=np.float64).reshape(3))
    p = np.asarray(frags, dtype=np.float64).reshape(-1, 3) - np.asarray(origin, dtype=np.float64).reshape(3)
    return np.stack([_dot(p, tg), _dot(p, bt)], axis=-1)


def _dist(a, b):
    d = b - a
    return np.sqrt(_dot(d, d))


def _heron(a, b, c):
    ab, ac, bc = _dist(a, b), _dist(a, c), _dist(b, c)
    s = (ab + ac + bc) / 2.0
    with np.errstate(invalid="ignore"):
        return np.sqrt(s * (s - ab) * (s - ac) * (s - bc))


def triangle_uv(tris, points) -> np.ndarray:
    """(s, t) of point i on (n, 33) reference-layout triangle record i: the Heron weights of the surface normal, then
    ((uv2 ba) + (uv1 bb)) + (uv0 bc)."""
    t = np.asarray(tris, dtype=np.float64).reshape(-1, 3, 11)
    p = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    v0, v1, v2 = t[:, 0, 0:3], t[:, 1, 0:3], t[:, 2, 0:3]
    with np.errstate(invalid="ignore", divide="ignore"):
        abc = _heron(v0, v1, v2)
        ba = (_heron(v0, v1, p) / abc)[:, None]
        bb = (_heron(v0, v2, p) / abc)[:, None]
        bc = 1.0 - (ba + bb)
    return ((t[:, 2, 6:8] * ba) + (t[:, 1, 6:8] * bb)) + (t[:, 0, 6:8] * bc)
