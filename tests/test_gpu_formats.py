"""GPU half of the SURVEY §8f rows: a JSON-project scene traces exactly like the same scene pushed through the API, and
the display transform kernel matches the reference front-end's tonemap (cli_old/src/main.rs:157-181)."""
import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from test_formats import write_project
from util import assert_hits_equal, product_scene, settings

pytestmark = pytest.mark.gpu


def test_project_scene_traces_like_the_api_scene(tmp_path):
    objs = F.gold_dragon(F.dragon_standin(120, 30))
    path = str(tmp_path / "scene.json")
    write_project(path, objs, str(tmp_path))
    loaded = A.Scene.load_project(path)
    # the same scene pushed object by object through the API (the mesh from the PLY text the project names)
    direct = A.Scene()
    for i, o in enumerate(objs):
        m = A.Material.from_fixture(o[-1])
        if o[0] == "sphere":
            direct.push_sphere(o[1], o[2], m)
        elif o[0] == "plane":
            direct.push_plane(o[1], o[2], m)
        else:
            direct.push_grid(A.AccGrid.build_from_mesh(A.Mesh.load_ply(str(tmp_path / f"mesh{i}.ply"))), m)
    rays = np.concatenate([O.primary_rays(F.camera(200, 120)), F.random_rays(20000, 3, ((-1.9, 1.9), (-0.9, 1.9), (-1.9, 4.9)))])
    assert_hits_equal(loaded.intersect(rays), direct.intersect(rays) + (None,), "project-loaded scene")
    st = settings(F.camera(96, 54), 4)
    a = A.Renderer(loaded, st, A.GpuOptions(seed=3)); a.render(0, 4)
    b = A.Renderer(direct, st, A.GpuOptions(seed=3)); b.render(0, 4)
    assert np.array_equal(a.read_sums(), b.read_sums())


def tonemap_test_frame():
    rng = np.random.default_rng(2)
    frame = rng.gamma(0.7, 0.6, size=(270, 480, 3))
    frame[0, 0] = (0.0, 0.0, 0.0)
    frame[0, 1] = (1.5, 1.5, 1.5)            # the ceiling: 227
    frame[0, 2] = (np.nan, 0.5, 0.5)         # cast fails -> whole pixel stays 0
    frame[0, 3] = (-0.5, 0.5, 0.5)           # 1 - exp(+0.5) < 0 -> powf -> NaN -> 0
    frame[0, 4] = (1e6, 0.0, 1e-12)
    return frame


def assert_tonemap_close(got, want, what, max_fraction=1e-5):
    """At most 1 level, on at most `max_fraction` of the values: a last-ulp libm difference landing on an integer boundary."""
    diff = np.abs(got.astype(int) - want.astype(int))
    assert diff.max() <= 1 and (diff > 0).mean() <= max_fraction, f"{what}: {int((diff > 0).sum())} values differ, by up to {diff.max()}"


def assert_tonemap_close_saturated(got, want, frame, exposure, what, max_fraction=1e-5):
    """assert_tonemap_close, except for values whose t = 1 - exp(-exposure p) is 1 - k 2^-53 with 1 <= k <= 4: there
    pow(t, 1 / gamma) rounds to 1.0 or to the double below it, and CUDA's pow and glibc's differ by that one ulp, so the value
    is 255 or 254.  At exposure 10, 156 values of tonemap_test_frame() are such; measured on a B200, 66 of them differ at gamma 2.2 and 38 at
    gamma 4.  They may differ by that one level; every other value is held to the bar."""
    with np.errstate(over="ignore", invalid="ignore"):
        edge = (1.0 - np.exp(frame * -1.0 * exposure)) >= 1.0 - 4.0 * 2.0 ** -53
    diff = np.abs(got.astype(int) - want.astype(int))
    assert (np.minimum(got, want)[edge & (diff > 0)] == 254).all() and diff[edge].max(initial=0) <= 1, f"{what}: saturated values"
    assert_tonemap_close(np.where(edge, want, got), want, what, max_fraction)


def test_tonemap_kernel_matches_the_reference_transform():
    """8-bit values equal F.tonemap (numpy restatement of cli_old's loop, glibc exp/pow) except where a last-ulp libm
    difference lands on an integer boundary: at most 1 level, on at most 1 pixel in 10^5."""
    frame = tonemap_test_frame()
    got = A.tonemap(frame)
    want = F.tonemap(frame)
    assert got[0, 1].tolist() == [227, 227, 227] and got[0, 2].tolist() == [0, 0, 0] and got[0, 3].tolist() == [0, 0, 0]
    assert_tonemap_close(got, want, "exposure 1, gamma 2.2")


# exposure 0 maps every finite pixel to 0; a negative exposure makes 1 - exp(+p) negative, so pow is NaN and the pixel is 0
# (except p = 0); gamma 1 is linear, 0.5 squares, 4 lifts the dark end
@pytest.mark.parametrize("exposure,gamma", [(0.0, 2.2), (1e-3, 2.2), (10.0, 2.2), (-1.0, 2.2), (1.0, 1.0), (1.0, 0.5), (1.0, 4.0),
                                            (1e-3, 0.5), (10.0, 4.0)])
def test_tonemap_kernel_exposure_and_gamma(exposure, gamma):
    """rm_tonemap_rgb8 and Renderer.read_rgb8 take the reference's exposure and gamma: both against the numpy restatement."""
    frame = tonemap_test_frame()
    want = F.tonemap(frame, exposure, gamma)
    got = A.tonemap(frame, exposure, gamma)
    assert_tonemap_close_saturated(got, want, frame, exposure, f"rm_tonemap_rgb8 exposure {exposure}, gamma {gamma}")
    if exposure == 0.0:
        assert not want.any()
    elif exposure > 0.0 and gamma >= 1.0:
        assert (want > 0).mean() > 0.3
    objs, cam, spp = F.reflective_spheres(), F.camera(96, 54), 4
    r = A.Renderer(product_scene(objs), settings(cam, spp), A.GpuOptions(seed=4))
    r.render(0, spp)
    rgb = r.read_rgb8(spp, exposure, gamma)
    mean = r.read_frame(spp)
    r.close()
    # the bar of test_renderer_rgb8_epilogue_and_png: this frame has only 15 552 values
    assert_tonemap_close_saturated(rgb, F.tonemap(mean, exposure, gamma), mean, exposure, f"read_rgb8 exposure {exposure}, gamma {gamma}", max_fraction=1e-4)


def test_renderer_rgb8_epilogue_and_png(tmp_path):
    from PIL import Image
    objs, cam, spp = F.reflective_spheres(), F.camera(160, 90), 8
    r = A.Renderer(product_scene(objs), settings(cam, spp), A.GpuOptions(seed=4))
    r.render(0, spp)
    rgb = r.read_rgb8(spp)
    want = F.tonemap(r.read_frame(spp))
    diff = np.abs(rgb.astype(int) - want.astype(int))
    assert diff.max() <= 1 and (diff > 0).mean() <= 1e-4
    assert rgb[2, 80].tolist() == [227, 227, 227]              # the emitting ceiling, as in examples/*.png
    path = str(tmp_path / "output.png")
    A.write_png(path, rgb)
    assert np.array_equal(np.asarray(Image.open(path)), rgb)
