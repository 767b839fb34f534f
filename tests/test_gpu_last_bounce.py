"""The last wavefront stage (depth == bounce_limit) in the default (drop) mode.

There a path delivers T (*) emission when its closest object is an emitter and an exact 0 otherwise, so the renderer runs a
last-depth k_shade that reads only the hit object, and k_setup queues no grid traversal for a ray whose closest analytic hit
is not an emitter, as long as no grid object emits and RM_FLAG_COUNT_WORK is off.  RM_FULL_LAST_BOUNCE=1 in the environment
(read when a renderer is created) renders the last stage like every other; with it the frame must be the same to the last bit.
In keep mode, with an emissive grid and under RM_FLAG_COUNT_WORK the grid traversal is not skipped, and the frame still
matches the reference path for path.
"""
import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from test_gpu_configs import compare_paths, gpu_sample_frames
from test_gpu_nonfinite import SCENES as NAN_SCENES
from util import oracle_scene, product_scene, settings

pytestmark = pytest.mark.gpu

SEED = 2026
EMISSIVE_GRID = ("Emission", (0.9, 0.6, 0.2), (1.0, 1.0, 1.0), 0.0, 0.0)


def gold_dragon(nu=240, nv=60):
    return F.gold_dragon(F.dragon_standin(nu, nv))


def oracle_frames(objs, cam, spp, limit):
    """One frame per sample index, as test_gpu_configs.oracle_sample_frames, at any bounce limit."""
    osc = oracle_scene(objs)
    return [O.render(osc, cam, 1, seed=SEED, first_sample=s, bounce_limit=limit)[0] for s in range(spp)]


def render(objs, cam, spp, bounce_limit, monkeypatch, full_last, flags=0, **opt):
    """Running sums, stats and stage stats of one Renderer, with or without the last-depth shortcut."""
    if full_last:
        monkeypatch.setenv("RM_FULL_LAST_BOUNCE", "1")
    else:
        monkeypatch.delenv("RM_FULL_LAST_BOUNCE", raising=False)
    r = A.Renderer(product_scene(objs), settings(cam, spp, bounce_limit=bounce_limit), A.GpuOptions(seed=SEED, flags=flags, **opt))
    r.render(0, spp)
    out = r.read_sums(), r.stats(), r.stage_stats()
    r.close()
    monkeypatch.delenv("RM_FULL_LAST_BOUNCE", raising=False)
    return out


def assert_same_bits(a, b, what):
    assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), f"{what}: the frames differ"


@pytest.mark.parametrize("precision", [A.PRECISION_F64, A.PRECISION_F32_SHADING])
@pytest.mark.parametrize("limit", [1, 5])
def test_skip_is_bit_identical(limit, precision, monkeypatch):
    """GoldDragon (full stand-in mesh) at 320x240 x 8 spp: the same frame and statistics with and without the shortcut, and
    fewer grid rays in the last stage only."""
    objs, cam, spp = F.gold_dragon(F.dragon_standin()), F.camera(320, 240), 8
    g, gs, gst = render(objs, cam, spp, limit, monkeypatch, False, precision=precision)
    f, fs, fst = render(objs, cam, spp, limit, monkeypatch, True, precision=precision)
    assert_same_bits(g, f, f"bounce_limit {limit}")
    for k in ("rays", "samples", "nonfinite_samples"):
        assert gs[k] == fs[k], k
    assert gst["rays"] == fst["rays"]
    assert gst["shaded_triangles"] == fst["shaded_triangles"]
    assert gst["grid_rays"][:limit] == fst["grid_rays"][:limit]
    assert gst["grid_rays"][limit] < fst["grid_rays"][limit]
    print(f"bounce_limit {limit}: last-stage grid rays {fst['grid_rays'][limit]} -> {gst['grid_rays'][limit]}")


def test_skip_render_tiled_two_shares(monkeypatch):
    """The task driver with two shares (sample partition, peer reduce) takes the shortcut too and awaits the same frame."""
    objs, cam, spp = gold_dragon(), F.camera(160, 120), 4
    st = settings(cam, spp)
    frames = []
    monkeypatch.delenv("RM_FULL_LAST_BOUNCE", raising=False)
    for full_last in (False, True):
        if full_last:
            monkeypatch.setenv("RM_FULL_LAST_BOUNCE", "1")
        task = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=SEED, device_list=[0, 0]))
        frames.append((task.await_(), task.stats()))
    assert_same_bits(frames[0][0], frames[1][0], "render_tiled")
    assert frames[0][1]["rays"] == frames[1][1]["rays"]


@pytest.mark.parametrize("limit", [1, 5, 40])
def test_skip_paths_match_the_oracle(limit):
    """With the shortcut on, path for path against the reference: GoldDragon (the Metal dragon can hide the ceiling), and
    bounce_limit 40 (far deeper than the paths of this frame reach: four of the six walls are black, so the last stage is empty)."""
    objs, cam, spp = gold_dragon(), F.camera(96, 72), 2
    g, _ = gpu_sample_frames(product_scene(objs), settings(cam, spp, bounce_limit=limit), spp, seed=SEED)
    compare_paths(g, oracle_frames(objs, cam, spp, limit), f"GoldDragon bounce_limit {limit}")


def assert_skip_off(objs, cam, spp, limit, monkeypatch, flags, what):
    """The last stage traverses the same grid rays as RM_FULL_LAST_BOUNCE and the frame is the same to the last bit."""
    g, gs, gst = render(objs, cam, spp, limit, monkeypatch, False, flags=flags)
    f, fs, fst = render(objs, cam, spp, limit, monkeypatch, True, flags=flags)
    assert gst["grid_rays"] == fst["grid_rays"], what
    assert_same_bits(g, f, what)
    assert gs["rays"] == fs["rays"] and gs["nonfinite_samples"] == fs["nonfinite_samples"], what
    return gst


def test_no_skip_with_an_emissive_grid(monkeypatch):
    """A grid that emits can itself be the answer of a last-depth ray: no ray is left out of its traversal."""
    objs = [F.RED_SPHERE, ("grid", F.translate(F.dragon_standin(240, 60), F.DRAGON_TRANSLATE), EMISSIVE_GRID)] + F.BOX_PLANES
    cam, spp, limit = F.camera(96, 72), 2, 5
    st = assert_skip_off(objs, cam, spp, limit, monkeypatch, 0, "emissive grid")
    assert st["grid_rays"][limit] > 0
    g, _ = gpu_sample_frames(product_scene(objs), settings(cam, spp, bounce_limit=limit), spp, seed=SEED)
    compare_paths(g, oracle_frames(objs, cam, spp, limit), "emissive grid")


def test_no_skip_when_counting_work(monkeypatch):
    """RM_FLAG_COUNT_WORK keeps the per-stage cells and triangle tests comparable with the reference's at every depth."""
    objs, cam, spp, limit = gold_dragon(), F.camera(96, 72), 2, 5
    st = assert_skip_off(objs, cam, spp, limit, monkeypatch, A.FLAG_COUNT_WORK, "count work")
    assert st["cells"][limit] > 0
    g, _ = gpu_sample_frames(product_scene(objs), settings(cam, spp, bounce_limit=limit), spp, seed=SEED, flags=A.FLAG_COUNT_WORK)
    compare_paths(g, oracle_frames(objs, cam, spp, limit), "count work")


@pytest.mark.parametrize("limit", [1, 5])
def test_no_skip_in_keep_mode(limit, monkeypatch):
    """Keep mode computes the last weight, and a NaN weight (a NaN shading normal of the mesh) must poison the sample: the
    last stage is rendered in full, NaN for NaN.  The path values of a finite keep-mode frame match the reference's."""
    cam, spp = F.camera(64, 48), 4
    assert_skip_off(NAN_SCENES["box"], cam, spp, limit, monkeypatch, A.FLAG_KEEP_NONFINITE, f"keep, NaN normals, bounce_limit {limit}")
    objs = gold_dragon()
    assert_skip_off(objs, cam, spp, limit, monkeypatch, A.FLAG_KEEP_NONFINITE, f"keep, GoldDragon, bounce_limit {limit}")
    g, _ = gpu_sample_frames(product_scene(objs), settings(cam, spp, bounce_limit=limit), spp, seed=SEED, flags=A.FLAG_KEEP_NONFINITE)
    compare_paths(g, oracle_frames(objs, cam, spp, limit), f"keep, GoldDragon, bounce_limit {limit}")
