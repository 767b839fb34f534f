"""CPU census of the coverage mask of the camera rays (DESIGN §3.7) on the bench frame: how many pixel-centre camera rays
enter the grid's box, and how many of those come from pixels the mask leaves uncovered (their traversal is skipped).

    python scripts/cover_census.py [--width 1920] [--height 1080] [--pad 1]

The bounding spheres are restated from the library's construction (prepare_grid_image): f32 centre at the middle of the
triangle's vertex box, radius to the farthest vertex times (1 + 1e-6) plus 1e-9 (1 + max |centre|), rounded up to f32;
the mask rule is k_cover_rects' (sphere box projected, `pad` pixels added, clamped to the frame).
"""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from raymond_b200 import fixtures as F  # noqa: E402


def spheres(P: np.ndarray):
    c = ((P.min(1) + P.max(1)) / 2).astype(np.float32)
    cd = c.astype(np.float64)
    r = np.sqrt(((P - cd[:, None, :]) ** 2).sum(-1).max(1)) * (1.0 + 1e-6) + 1e-9 * (1.0 + np.abs(cd).max(1))
    rf = r.astype(np.float32)
    low = rf.astype(np.float64) < r
    rf[low] = np.nextafter(rf[low], np.float32(np.inf))
    return cd, rf.astype(np.float64)


def mask(c, R, W, H, th, pad):
    lo, hi = c - R[:, None], c + R[:, None]
    assert (lo[:, 2] > 0).all(), "a sphere box is not in front of the camera: the library would build no mask"
    xr = np.stack([lo[:, 0] / lo[:, 2], lo[:, 0] / hi[:, 2], hi[:, 0] / lo[:, 2], hi[:, 0] / hi[:, 2]], 1)
    yr = np.stack([lo[:, 1] / lo[:, 2], lo[:, 1] / hi[:, 2], hi[:, 1] / lo[:, 2], hi[:, 1] / hi[:, 2]], 1)
    sx, sy = th * W / H, th
    X0, X1 = (xr.min(1) / sx + 1) * 0.5 * W, (xr.max(1) / sx + 1) * 0.5 * W
    Y0, Y1 = (1 - yr.max(1) / sy) * 0.5 * H, (1 - yr.min(1) / sy) * 0.5 * H
    x0 = np.clip(np.floor(X0) - pad, 0, W - 1).astype(int)
    x1 = np.clip(np.floor(X1) + pad, -1, W - 1).astype(int)
    y0 = np.clip(np.floor(Y0) - pad, 0, H - 1).astype(int)
    y1 = np.clip(np.floor(Y1) + pad, -1, H - 1).astype(int)
    ok = (x0 <= x1) & (y0 <= y1)
    d = np.zeros((H + 1, W + 1), np.int64)
    np.add.at(d, (y0[ok], x0[ok]), 1)
    np.add.at(d, (y0[ok], x1[ok] + 1), -1)
    np.add.at(d, (y1[ok] + 1, x0[ok]), -1)
    np.add.at(d, (y1[ok] + 1, x1[ok] + 1), 1)
    return d.cumsum(0).cumsum(1)[:H, :W] > 0, X1 - X0, Y1 - Y0


def main() -> None:
    p = argparse.ArgumentParser()
    p.add_argument("--width", type=int, default=1920)
    p.add_argument("--height", type=int, default=1080)
    p.add_argument("--pad", type=int, default=1)
    a = p.parse_args()
    W, H = a.width, a.height
    th = np.tan(55.0 / 2.0 * np.pi / 180.0)        # the bench camera: fov 55, at the origin, looking along +z
    P = np.asarray(F.positions(F.translate(F.dragon_standin(), F.DRAGON_TRANSLATE)), dtype=np.float64)
    c, R = spheres(P)
    cover, w, h = mask(c, R, W, H, th, a.pad)
    bmin, bmax = P.reshape(-1, 3).min(0), P.reshape(-1, 3).max(0)
    xs, ys = np.arange(W) + 0.5, np.arange(H) + 0.5
    px, py = (2 * (xs / W) - 1) * th * W / H, (1 - 2 * (ys / H)) * th
    D = np.stack(np.broadcast_arrays(px[None, :], py[:, None], np.ones((H, W))), -1)
    D /= np.linalg.norm(D, axis=-1, keepdims=True)
    with np.errstate(divide="ignore", invalid="ignore"):
        t1, t2 = bmin / D, bmax / D
    enter = np.minimum(t1, t2).max(-1) < np.maximum(t1, t2).min(-1)
    skipped = enter & ~cover
    print(f"GoldDragon stand-in, {P.shape[0]} triangles, camera {W}x{H}, pad {a.pad} px")
    print(f"projected sphere boxes: median {np.median(w):.2f} x {np.median(h):.2f} px, max {w.max():.2f} x {h.max():.2f} px")
    print(f"pixels covered by the mask: {cover.sum()} of {W * H} ({cover.mean():.4f})")
    print(f"pixel-centre rays entering the grid box: {enter.sum()}")
    print(f"  of those from uncovered pixels (traversal skipped): {skipped.sum()} ({skipped.sum() / enter.sum():.4f})")


if __name__ == "__main__":
    main()
