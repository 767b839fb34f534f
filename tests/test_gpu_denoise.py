"""rm_renderer_read_denoised: the library's filter against the numpy float32 restatement (tests/denoise_ref.py) on the renderer's
own sums, the quality of the default settings against a high-sample render, and the argument and state errors."""
import numpy as np
import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

import denoise_ref as D
from test_gpu_nonfinite import SCENES as NONFINITE_SCENES
from util import product_scene, settings

pytestmark = pytest.mark.gpu

FLAGS = A.FLAG_AOV | A.FLAG_MOMENTS
SCENES = {"spheres": F.reflective_spheres, "dragon_standin": lambda: F.gold_dragon(F.dragon_standin())}
LUMA = np.array([0.2126, 0.7152, 0.0722])


def rendered(objs, cam, spp, seed=7, flags=FLAGS):
    r = A.Renderer(product_scene(objs), settings(cam, spp, (32, 32)), A.GpuOptions(seed=seed, flags=flags))
    r.render(0, spp)
    return r


@pytest.mark.parametrize("denoise", [None, A.DenoiseSettings(3, 1.5, 0.3, 0.4, 0.05), A.DenoiseSettings(10, 8.0, 2.0, 1.0, 1.0)],
                         ids=["defaults", "three", "ten"])
@pytest.mark.parametrize("name", ["spheres", "dragon_small", "nonfinite_box"])
def test_denoised_is_the_restatement(name, denoise):
    """nonfinite_box keeps NaN / Inf samples (RM_FLAG_KEEP_NONFINITE): those pixels are copied and their neighbours skip them."""
    n = 8
    if name == "nonfinite_box":
        r = rendered(NONFINITE_SCENES["box"], F.camera(64, 48), n, seed=3, flags=FLAGS | A.FLAG_KEEP_NONFINITE)
    else:
        objs = F.reflective_spheres() if name == "spheres" else F.gold_dragon(F.dragon_standin(96, 24))
        r = rendered(objs, F.camera(128, 96), n)
    got = r.read_denoised(n, denoise)
    S, Q = r.read_sums(), r.read_moments()
    albedo, normal, depth = r.read_aovs(n)
    r.close()
    kw = D.DEFAULTS if denoise is None else dict(iterations=denoise.iterations, sigma_color=denoise.sigma_color,
                                                 sigma_normal=denoise.sigma_normal, sigma_albedo=denoise.sigma_albedo,
                                                 sigma_depth=denoise.sigma_depth)
    want = D.denoise(S, Q, albedo, normal, depth, n, **kw).astype(np.float64)
    for f in (np.isnan, np.isposinf, np.isneginf):
        assert np.array_equal(f(got), f(want)), f.__name__
    if name == "nonfinite_box":
        assert np.isnan(want).any() and np.isfinite(want).mean() > 0.5
    fin = np.isfinite(want)
    err = np.abs(got[fin] - want[fin])
    rel = err / np.maximum(np.abs(want[fin]), 1e-30)
    print(f"{name} {kw}: largest difference {err.max():.3g} absolute, {rel[err > 1e-6].max(initial=0.0):.3g} relative beyond 1e-6 absolute")
    assert (err <= 1e-4 * np.abs(want[fin]) + 1e-6).all()
    assert np.abs(got - S / n)[fin].max() > 1e-3       # the filter did something


def rmse(a, b):
    return float(np.sqrt(np.mean((np.clip(a, 0.0, 10.0) - np.clip(b, 0.0, 10.0)) ** 2)))


@pytest.mark.parametrize("name", list(SCENES))
def test_default_settings_quality(name):
    """At 16 spp the defaults bring the RMSE against a 4096-spp render (linear, clamped to [0, 10]) to <= 0.6 x the raw one,
    and keep the mean luminance of the raw frame within 1 %."""
    objs, cam = SCENES[name](), F.camera(320, 240)
    ref = rendered(objs, cam, 4096, seed=1, flags=0)
    reference = ref.read_frame(4096)
    ref.close()
    r = rendered(objs, cam, 16, seed=2)
    raw = r.read_frame(16)
    den = r.read_denoised(16)
    r.close()
    e_raw, e_den = rmse(raw, reference), rmse(den, reference)
    l_raw, l_den = float((raw @ LUMA).mean()), float((den @ LUMA).mean())
    print(f"{name}: RMSE raw {e_raw:.4g}, denoised {e_den:.4g} ({e_den / e_raw:.3f} x); mean luminance raw {l_raw:.5g}, denoised {l_den:.5g}")
    assert e_den <= 0.6 * e_raw
    assert abs(l_den - l_raw) <= 0.01 * l_raw


def test_errors():
    objs, cam = F.reflective_spheres(), F.camera(32, 24)
    r = rendered(objs, cam, 4)
    for bad in (A.DenoiseSettings(iterations=0), A.DenoiseSettings(iterations=11), A.DenoiseSettings(sigma_color=0.0),
                A.DenoiseSettings(sigma_normal=-1.0), A.DenoiseSettings(sigma_albedo=float("nan")), A.DenoiseSettings(sigma_depth=float("inf")),
                # finite and > 0 in f64, but not usable in f32: the square underflows or overflows, or the value itself does
                A.DenoiseSettings(sigma_normal=1e-25), A.DenoiseSettings(sigma_albedo=1e20), A.DenoiseSettings(sigma_color=1e39),
                A.DenoiseSettings(sigma_depth=1e-40)):
        with pytest.raises(A.RaymondError) as e:
            r.read_denoised(4, bad)
        assert e.value.status == A.RM_ERR_INVALID_ARGUMENT, bad
    for count in (0, 1):
        with pytest.raises(A.RaymondError) as e:
            r.read_denoised(count)
        assert e.value.status == A.RM_ERR_INVALID_ARGUMENT
    r.read_denoised(4, A.DenoiseSettings(iterations=10))
    assert np.isfinite(r.read_denoised(4, A.DenoiseSettings(sigma_normal=2e-19, sigma_albedo=1e19, sigma_color=3e38, sigma_depth=2e-38))).all()
    r.close()
    for flags in (0, A.FLAG_AOV, A.FLAG_MOMENTS):
        r = rendered(objs, cam, 4, flags=flags)
        with pytest.raises(A.RaymondError) as e:
            r.read_denoised(4)
        assert e.value.status == A.RM_ERR_STATE
        r.close()
    r = A.Renderer(product_scene(objs), settings(cam, 4, (8, 8)), A.GpuOptions(flags=FLAGS, world_size=2, rank=0, partition=A.PARTITION_TILES))
    r.render(0, 4)
    with pytest.raises(A.RaymondError) as e:
        r.read_denoised(4)
    assert e.value.status == A.RM_ERR_UNSUPPORTED
    r.close()
