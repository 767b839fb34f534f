"""rm_precision: the f32 mode of the statistical scope against the f64 mode.

The two modes draw their uniforms from the same Philox blocks but not from the same words (the f32 mode makes one Philox call
per bounce instead of two), so they are different sample streams of the same estimator: what must hold is that the f32 image
is as close to an f64 image as two f64 images with different seeds are to each other (the noise floor of SURVEY 8d), that the
mean agrees (no bias), that the path-length statistics agree — and that the bit-exact scope is untouched.  The same-stream,
path-for-path comparison of the f32 mode is test_gpu_f32_paths.py, against the oracle given the f32 mode's own draws."""
import numpy as np
import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import product_scene, settings

pytestmark = pytest.mark.gpu

LUMA = np.array([0.2126, 0.7152, 0.0722])


def render(ps, cam, spp, precision, seed, limit=5):
    r = A.Renderer(ps, settings(cam, spp, bounce_limit=limit), A.GpuOptions(seed=seed, precision=precision))
    r.render(0, spp)
    out, stats = r.read_sums() / spp, r.stats()
    r.close()
    return out, stats


@pytest.mark.parametrize("scene", ["spheres", "dof", "dragon"])
def test_f32_shading_is_the_same_estimator(scene):
    if scene == "dragon":
        ps, cam, spp = product_scene(F.gold_dragon(F.dragon_standin(480, 120))), F.camera(320, 180), 64
    elif scene == "dof":
        ps, cam, spp = product_scene(F.reflective_spheres()), F.camera(320, 180, focal_length=2.5, aperture_radius=0.5), 64
    else:
        ps, cam, spp = product_scene(F.reflective_spheres()), F.camera(320, 180), 64
    a, sa = render(ps, cam, spp, A.PRECISION_F64, 5)
    b, sb = render(ps, cam, spp, A.PRECISION_F32_SHADING, 5)
    c, _ = render(ps, cam, spp, A.PRECISION_F64, 6)                 # another stream: the noise floor
    assert sa["samples"] == sb["samples"] and sb["nonfinite_samples"] <= sa["nonfinite_samples"] + 8
    clip = lambda x: np.clip(x, 0, 10)
    la, lb, lc = clip(a) @ LUMA, clip(b) @ LUMA, clip(c) @ LUMA
    # the f32 image is no farther from an f64 image than another f64 stream is (1.15 x the noise floor, SURVEY 8d)
    same, floor = np.sqrt(((la - lb) ** 2).mean()), np.sqrt(((la - lc) ** 2).mean())
    assert same <= 1.15 * floor, (same, floor)
    # no bias: |mean luminance difference| <= max(0.5 %, 3 standard errors)
    se = np.sqrt(la.var() / la.size + lb.var() / lb.size)
    assert abs(la.mean() - lb.mean()) <= max(5e-3 * la.mean(), 3 * se), (la.mean(), lb.mean(), se)
    # the same lobe probabilities: rays per path agree to 0.5 %
    assert abs(sa["rays"] - sb["rays"]) <= 0.005 * sa["rays"]


def test_f32_shading_leaves_directly_visible_emitters_exact():
    """bounce_limit 1: only emission seen by camera rays contributes; nothing of that is in the statistical scope."""
    ps, cam = product_scene(F.reflective_spheres()), F.camera(96, 64)
    a, _ = render(ps, cam, 2, A.PRECISION_F64, 3, limit=1)
    b, _ = render(ps, cam, 2, A.PRECISION_F32_SHADING, 3, limit=1)
    assert np.array_equal(a, b) and a.any()


def test_unknown_precision_is_rejected():
    with pytest.raises(A.RaymondError) as e:
        A.Renderer(product_scene(F.reflective_spheres()), settings(F.camera(8, 8), 1), A.GpuOptions(precision=7))
    assert e.value.status == A.RM_ERR_INVALID_ARGUMENT
