"""rm_render_tiled_denoised (no GPU): bad arguments fail before any device work, with the statuses include/raymond.h gives, and the
Python mirror refuses adaptive sampling together with the filter."""
import ctypes as C

import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import settings

BAD_SETTINGS = [A.DenoiseSettings(iterations=0), A.DenoiseSettings(iterations=11), A.DenoiseSettings(sigma_color=0.0),
                A.DenoiseSettings(sigma_normal=-1.0), A.DenoiseSettings(sigma_albedo=float("nan")),
                A.DenoiseSettings(sigma_depth=float("inf")),
                # finite and > 0 in f64, but not usable in f32: the square underflows or overflows, or the value itself does
                A.DenoiseSettings(sigma_normal=1e-25), A.DenoiseSettings(sigma_albedo=1e20), A.DenoiseSettings(sigma_color=1e39),
                A.DenoiseSettings(sigma_depth=1e-40)]


def refused(spp=4, options=None, denoise=True):
    with pytest.raises(A.RaymondError) as e:
        A.render_tiled(A.Scene(), settings(F.camera(8, 4), spp), options, denoise=denoise)
    return e.value


@pytest.mark.parametrize("bad", BAD_SETTINGS, ids=lambda s: repr(s))
def test_bad_settings(bad):
    e = refused(denoise=bad)
    assert e.status == A.RM_ERR_INVALID_ARGUMENT
    assert "rm_render_tiled_denoised" in str(e)


@pytest.mark.parametrize("spp", [0, 1])
def test_sample_count_below_two(spp):
    e = refused(spp)
    assert e.status == A.RM_ERR_INVALID_ARGUMENT
    assert "sample_count" in str(e)


def test_sample_count_is_checked_before_the_settings():
    assert "sample_count" in str(refused(1, denoise=A.DenoiseSettings(iterations=0)))


def test_one_rank_of_a_multi_process_job():
    e = refused(options=A.GpuOptions(world_size=2, rank=0))
    assert e.status == A.RM_ERR_UNSUPPORTED
    # invalid settings are reported first
    assert refused(options=A.GpuOptions(world_size=2, rank=0), denoise=A.DenoiseSettings(iterations=0)).status == A.RM_ERR_INVALID_ARGUMENT


def test_null_arguments():
    L = A.lib()
    s = settings(F.camera(8, 4), 4)._c()
    assert not L.rm_render_tiled_denoised(None, C.byref(s), None, None)
    assert L.rm_last_status() == A.RM_ERR_INVALID_ARGUMENT
    sc = A.Scene()
    assert not L.rm_render_tiled_denoised(sc._h, None, None, None)
    assert L.rm_last_status() == A.RM_ERR_INVALID_ARGUMENT
    assert L.rm_task_await_denoised(None, None) == A.RM_ERR_INVALID_ARGUMENT


def test_camera_checks_come_first():
    st = settings(F.camera(8, 4), 1)
    st.camera_settings.aperture_radius = float("inf")      # a camera rm_render_tiled refuses
    with pytest.raises(A.RaymondError) as e:
        A.render_tiled(A.Scene(), st, None, denoise=A.DenoiseSettings(iterations=0))
    assert e.value.status == A.RM_ERR_INVALID_ARGUMENT
    assert "sample_count" not in str(e.value) and "sigma" not in str(e.value)


def test_adaptive_and_denoise_do_not_combine():
    with pytest.raises(ValueError):
        A.render_tiled(A.Scene(), settings(F.camera(8, 4), 4, spi=2), None, A.AdaptiveSettings(0.05), denoise=True)


def test_the_other_entry_points_keep_refusing_the_feature_buffers():
    for adaptive in (None, A.AdaptiveSettings(0.05)):
        with pytest.raises(A.RaymondError) as e:
            A.render_tiled(A.Scene(), settings(F.camera(8, 4), 4, spi=2), A.GpuOptions(flags=A.FLAG_AOV), adaptive)
        assert e.value.status == A.RM_ERR_UNSUPPORTED and "RM_FLAG_AOV" in str(e.value)
