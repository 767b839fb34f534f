"""The coverage mask of the camera rays (DESIGN §3.7).

Without depth of field every camera ray starts at the camera, so a pixel outside the screen-space box of every triangle's
bounding sphere (plus a pixel) cannot see the first grid object: k_setup<SRC_CAMERA> pushes no traversal record for its rays
and their hit records keep the analytic answer.  RM_NO_COVER_MASK=1 in the environment (read when a renderer is created)
turns the mask off; with and without it the frame and the statistics must be the same to the last bit, and fewer depth-1
rays enter the grid with it.  The mask switches itself off where its argument does not hold.
"""
import os

import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from test_gpu_env import env_scene
from util import oracle_scene, product_scene, settings

pytestmark = pytest.mark.gpu

SEED = 2026
THREADS = os.cpu_count() or 1


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def mask_env(monkeypatch, on):
    if on:
        monkeypatch.delenv("RM_NO_COVER_MASK", raising=False)
    else:
        monkeypatch.setenv("RM_NO_COVER_MASK", "1")


def render(make_scene, cam, spp, monkeypatch, on, bounce_limit=5, **opt):
    """Running sums, stats, stage stats and coverage mask of one Renderer, with the mask allowed or not."""
    mask_env(monkeypatch, on)
    r = A.Renderer(make_scene(), settings(cam, spp, bounce_limit=bounce_limit), A.GpuOptions(seed=SEED, **opt))
    cover = r.coverage()
    r.render(0, spp)
    out = r.read_sums(), r.stats(), r.stage_stats(), cover
    r.close()
    monkeypatch.delenv("RM_NO_COVER_MASK", raising=False)
    return out


def assert_same(on, off, what):
    (s1, st1, ss1, c1), (s0, st0, ss0, c0) = on, off
    assert c0 is None, f"{what}: RM_NO_COVER_MASK left a mask"
    assert bits_equal(s1, s0), f"{what}: the frames differ"
    for k in ("rays", "samples", "nonfinite_samples"):
        assert st1[k] == st0[k], f"{what}: {k}"
    assert ss1["rays"] == ss0["rays"] and ss1["shaded_triangles"] == ss0["shaded_triangles"], what
    assert ss1["grid_rays"][2:] == ss0["grid_rays"][2:], what


def gold_dragon():
    return product_scene(F.gold_dragon(F.dragon_standin()))


@pytest.mark.parametrize("precision", [A.PRECISION_F64, A.PRECISION_F32_SHADING])
@pytest.mark.parametrize("flags", [0, A.FLAG_KEEP_NONFINITE], ids=["drop", "keep"])
def test_gold_dragon_bit_identical(precision, flags, monkeypatch):
    """GoldDragon (full stand-in mesh) at 640x360 x 8 spp: the same frame and statistics, fewer depth-1 grid rays."""
    cam, spp = F.camera(640, 360), 8
    on = render(gold_dragon, cam, spp, monkeypatch, True, precision=precision, flags=flags)
    off = render(gold_dragon, cam, spp, monkeypatch, False, precision=precision, flags=flags)
    assert on[3] is not None and 0 < on[3].mean() < 1
    assert_same(on, off, f"precision {precision}, flags {flags}")
    g1, g0 = on[2]["grid_rays"][1], off[2]["grid_rays"][1]
    assert g1 < 0.75 * g0, (g1, g0)
    print(f"depth-1 grid rays {g0} -> {g1} ({g1 / g0:.3f}); {on[3].mean():.3f} of the frame covered")


def test_open_dragon_with_environment(monkeypatch):
    """The open dragon under an environment map: rays that miss everything see the map, the mask changes nothing."""
    cam, spp = F.camera(320, 180), 6
    make = lambda: env_scene(F.open_dragon(F.dragon_standin(240, 60)))
    on = render(make, cam, spp, monkeypatch, True)
    off = render(make, cam, spp, monkeypatch, False)
    assert on[3] is not None
    assert_same(on, off, "open dragon, environment map")
    assert on[2]["grid_rays"][1] < off[2]["grid_rays"][1]


def gold_dragon_small():
    return product_scene(F.gold_dragon(F.dragon_standin(240, 60)))


@pytest.mark.parametrize("kind", ["samples", "tiles", "adaptive", "denoised"])
def test_tasks_bit_identical(kind, monkeypatch):
    """render_tiled with two shares on device 0 (sample and tile partitions), an adaptive task and a denoised task: every
    share builds its own mask, and the awaited frame and the statistics are the same to the last bit."""
    cam = F.camera(160, 120)
    st = settings(cam, 8, tile=(32, 32), spi=4 if kind == "adaptive" else 0)
    extra, await_fn = {}, (lambda t: t.await_())
    if kind == "samples":
        opt = A.GpuOptions(seed=SEED, device_list=[0, 0], partition=A.PARTITION_SAMPLES)
    elif kind == "tiles":
        opt = A.GpuOptions(seed=SEED, device_list=[0, 0], partition=A.PARTITION_TILES)
    elif kind == "adaptive":
        opt = A.GpuOptions(seed=SEED)
        extra = {"adaptive": A.AdaptiveSettings(0.05, 4)}
    else:
        opt = A.GpuOptions(seed=SEED, device_list=[0, 0], partition=A.PARTITION_SAMPLES)
        extra, await_fn = {"denoise": True}, (lambda t: t.await_denoised())
    out = []
    for on in (True, False):
        mask_env(monkeypatch, on)
        task = A.render_tiled(gold_dragon_small(), st, opt, **extra)
        out.append((await_fn(task), task.stats()))
    monkeypatch.delenv("RM_NO_COVER_MASK", raising=False)
    (f1, s1), (f0, s0) = out
    assert bits_equal(f1, f0), kind
    for k in ("rays", "samples", "nonfinite_samples"):
        assert s1[k] == s0[k], (kind, k)


# ---------------------------------------------------------------------------- the mask against the oracle's hits


def sphere_mask(tris, cam, pad, radius_scale):
    """The mask restated in numpy from the triangles: f32 centre of each vertex box, radius to the farthest vertex (no
    inflation), the sphere's box projected, `pad` pixels added (the library: pad 1 and inflated, rounded-up radii)."""
    P = F.positions(tris).astype(np.float64)
    c = ((P.min(1) + P.max(1)) / 2).astype(np.float32).astype(np.float64)
    R = np.linalg.norm(P - c[:, None, :], axis=-1).max(1) * radius_scale
    W, H = cam["width"], cam["height"]
    th = np.tan(cam["fov_vert"] / 2 * np.pi / 180)
    sx, sy = th * W / H, th
    lo, hi = c - R[:, None] - np.array(cam["position"]), c + R[:, None] - np.array(cam["position"])
    assert (lo[:, 2] > 0).all()
    xr = np.stack([lo[:, 0] / lo[:, 2], lo[:, 0] / hi[:, 2], hi[:, 0] / lo[:, 2], hi[:, 0] / hi[:, 2]], 1)
    yr = np.stack([lo[:, 1] / lo[:, 2], lo[:, 1] / hi[:, 2], hi[:, 1] / lo[:, 2], hi[:, 1] / hi[:, 2]], 1)
    X0, X1 = (xr.min(1) / sx + 1) * W / 2, (xr.max(1) / sx + 1) * W / 2
    Y0, Y1 = (1 - yr.max(1) / sy) * H / 2, (1 - yr.min(1) / sy) * H / 2
    x0 = np.clip(np.floor(X0) - pad, 0, W - 1).astype(int)
    x1 = np.clip(np.floor(X1) + pad, -1, W - 1).astype(int)
    y0 = np.clip(np.floor(Y0) - pad, 0, H - 1).astype(int)
    y1 = np.clip(np.floor(Y1) + pad, -1, H - 1).astype(int)
    d = np.zeros((H + 1, W + 1), np.int64)
    ok = (x0 <= x1) & (y0 <= y1)
    np.add.at(d, (y0[ok], x0[ok]), 1)
    np.add.at(d, (y0[ok], x1[ok] + 1), -1)
    np.add.at(d, (y1[ok] + 1, x0[ok]), -1)
    np.add.at(d, (y1[ok] + 1, x1[ok] + 1), 1)
    return d.cumsum(0).cumsum(1)[:H, :W] > 0


@pytest.mark.parametrize("mesh", [(24, 6), (1320, 330)], ids=["coarse", "standin"])
def test_every_grid_hit_comes_from_a_covered_pixel(mesh):
    """Every jittered camera ray whose closest hit (oracle Scene::intersect) is the dragon comes from a covered pixel.  The
    check has teeth: on the coarse mesh (triangles many pixels wide) the same mask with pad 0 and halved radii leaves some
    of those pixels uncovered; on the full stand-in the triangles' boxes overlap so densely that it would not."""
    cam, spp = F.camera(480, 270), 8
    mesh = F.dragon_standin(*mesh)
    objs = F.gold_dragon(mesh)
    r = A.Renderer(product_scene(objs), settings(cam, 1), A.GpuOptions(seed=SEED))
    cover = r.coverage()
    r.close()
    assert cover is not None
    osc = oracle_scene(objs)
    hit = np.zeros(cover.shape, bool)
    for s in range(spp):
        obj = osc.intersect(O.camera_rays(cam, SEED, s), THREADS)[0]
        hit |= (obj == 1).reshape(cover.shape)
    assert hit.sum() > 1000
    assert not (hit & ~cover).any(), f"{(hit & ~cover).sum()} pixels see the dragon but are not covered"
    tris = F.translate(mesh, F.DRAGON_TRANSLATE)
    assert not (hit & ~sphere_mask(tris, cam, 1, 1.0)).any()
    missed = (hit & ~sphere_mask(tris, cam, 0, 0.5)).sum()
    if mesh.shape[0] < 1000:
        assert missed > 0, "pad 0 and half radii should leave a hit pixel uncovered"
    print(f"covered {cover.mean():.3f}, hit {hit.mean():.3f}, missed by pad 0 and half radii {missed}")


# ---------------------------------------------------------------------------- where the mask switches itself off


def nan_dragon(coords):
    """The coarse dragon with NaN in some position coordinates of triangle 5 (layout of fixtures.positions)."""
    m = F.dragon_standin(96, 24).copy()
    for k in coords:
        m[5, 11 * (k // 3) + k % 3] = np.nan
    return F.gold_dragon(m)


OFF_CASES = {
    # (objects, camera)
    "camera_inside_the_box": (lambda: F.gold_dragon(F.dragon_standin(96, 24)), F.camera(64, 48, position=F.DRAGON_TRANSLATE)),
    "mesh_partly_behind": (lambda: F.gold_dragon(F.dragon_standin(96, 24)), F.camera(64, 48, position=(1.5, -0.3, 2.9))),
    # the grid's box is in front, but the spheres of the triangles on its near face reach behind the camera: k_cover_rects
    # flags them and the renderer drops the mask
    "camera_at_the_near_face": (lambda: F.gold_dragon(F.dragon_standin(96, 24)),
                                F.camera(64, 48, position=(0.0, -0.3, F.positions(F.translate(F.dragon_standin(96, 24), F.DRAGON_TRANSLATE))[..., 2].min() - 1e-4))),
    "depth_of_field": (lambda: F.gold_dragon(F.dragon_standin(96, 24)), F.camera(64, 48, aperture_radius=0.05)),
}


@pytest.mark.parametrize("case", sorted(OFF_CASES))
def test_mask_switches_itself_off(case, monkeypatch):
    objs, cam = OFF_CASES[case]
    on = render(lambda: product_scene(objs()), cam, 4, monkeypatch, True)
    off = render(lambda: product_scene(objs()), cam, 4, monkeypatch, False)
    assert on[3] is None, f"{case}: the renderer built a mask"
    assert_same(on, off, case)
    assert on[2]["grid_rays"] == off[2]["grid_rays"], case


def test_no_mask_when_counting_work(monkeypatch):
    """RM_FLAG_COUNT_WORK keeps the per-stage cells and triangle tests comparable with the oracle's (DESIGN §3.4)."""
    mask_env(monkeypatch, True)
    r = A.Renderer(gold_dragon_small(), settings(F.camera(64, 48), 1), A.GpuOptions(seed=SEED, flags=A.FLAG_COUNT_WORK))
    assert r.coverage() is None
    r.close()


def test_one_nan_coordinate_keeps_the_mask(monkeypatch):
    """A NaN vertex coordinate leaves a finite sphere around the rest of the triangle (fmin / fmax skip the NaN), and that
    triangle can never be hit: its a, u, v and t are NaN, and every comparison that would accept the hit is false.  The
    mask stays on and the frame is the same to the last bit.  (A triangle whose sphere is not finite needs a NaN on one
    axis of all three vertices, and the grid build refuses such a mesh.)"""
    cam = F.camera(160, 120)
    on = render(lambda: product_scene(nan_dragon([0])), cam, 4, monkeypatch, True)
    off = render(lambda: product_scene(nan_dragon([0])), cam, 4, monkeypatch, False)
    assert on[3] is not None
    assert_same(on, off, "one NaN coordinate")
