"""numpy restatement of the environment-map lookup of include/raymond.h (rm_environment), for the tests.

Every operation is one f64 numpy ufunc call in the header's order (numpy never fuses a multiply-add), so the result differs
from the oracle's (glibc) and the GPU's (CUDA libdevice) only by what their atan2 / acos return.
"""
from __future__ import annotations

import numpy as np


def env_lookup(image, dirs, scale: float = 1.0, rotation: float = 0.0) -> np.ndarray:
    """L(d) for (n, 3) directions `dirs` of the (H, W, 3) map `image` (taken as f32, widened exactly)."""
    tex = np.asarray(image, dtype=np.float32).astype(np.float64)
    H, W = tex.shape[0], tex.shape[1]
    d = np.asarray(dirs, dtype=np.float64).reshape(-1, 3)
    with np.errstate(invalid="ignore"):
        u = 0.5 + (np.arctan2(d[:, 0], d[:, 2]) + float(rotation)) / (2.0 * np.pi)
        u = u - np.floor(u)
        cy = np.where(d[:, 1] < -1.0, -1.0, np.where(d[:, 1] > 1.0, 1.0, d[:, 1]))
        v = np.arccos(cy) / np.pi
    nan = np.isnan(u) | np.isnan(v)
    u = np.where(nan, 0.0, u)
    v = np.where(nan, 0.0, v)
    x = u * float(W) - 0.5
    y = v * float(H) - 0.5
    x0 = np.floor(x)
    y0 = np.floor(y)
    fx = (x - x0)[:, None]
    fy = (y - y0)[:, None]
    ix0 = x0.astype(np.int64) % W
    ix1 = (x0.astype(np.int64) + 1) % W
    iy0 = np.clip(y0.astype(np.int64), 0, H - 1)
    iy1 = np.clip(y0.astype(np.int64) + 1, 0, H - 1)
    t00, t01, t10, t11 = tex[iy0, ix0], tex[iy0, ix1], tex[iy1, ix0], tex[iy1, ix1]
    top = t00 + fx * (t01 - t00)
    bot = t10 + fx * (t11 - t10)
    out = float(scale) * (top + fy * (bot - top))
    out[nan] = np.nan
    return out


def sky_dirs_edge_cases() -> np.ndarray:
    """Directions on the u seam, at both poles, with signed zeros and off the unit sphere."""
    s = np.sqrt(0.5)
    return np.array([
        [0.0, 0.0, 1.0], [0.0, 0.0, -1.0], [-0.0, 0.0, -1.0], [0.0, -0.0, -1.0], [1e-300, 0.0, -1.0], [-1e-300, 0.0, -1.0],
        [0.0, 1.0, 0.0], [0.0, -1.0, 0.0], [0.0, 1.0, -0.0], [-0.0, -1.0, -0.0], [1e-17, 1.0, 0.0], [0.0, -1.0, 1e-17],
        [s, 0.0, s], [-s, 0.0, s], [s, s, 0.0], [0.0, s, -s], [-1.0, 0.0, 0.0], [1.0, 0.0, 0.0],
        [0.0, 2.0, 0.0], [0.0, -3.0, 0.0], [3.0, 4.0, 0.0], [0.1, 0.2, 0.3], [-0.0, -0.0, -0.0], [0.0, 0.0, 0.0],
    ])
