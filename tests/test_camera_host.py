"""CPU tests of the depth-of-field camera settings the renderer refuses.

The reference's aperture sampling (src/trace.rs:335-360) draws points until one lies strictly inside the aperture disk, and
then unwraps the focal-plane hit.  An infinite aperture radius, one whose dx² + dy² overflows, or a non-finite camera position
makes that loop endless (on the GPU: a kernel that never returns); a negative or NaN focal length makes the unwrap panic.
Such settings are RM_ERR_INVALID_ARGUMENT before any device work, so the statuses hold on a box without a GPU.  No test here
renders with a refused setting."""
import math

import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import settings

INF, NAN = math.inf, math.nan

REFUSED = {
    "aperture_inf": dict(aperture_radius=INF),
    "aperture_1e154": dict(aperture_radius=1e154),
    "aperture_above_1e150": dict(aperture_radius=1.0000000000000002e150),
    "position_inf": dict(aperture_radius=0.5, position=(INF, 0.0, 0.0)),
    "position_minus_inf": dict(aperture_radius=0.5, position=(0.0, 0.0, -INF)),
    "position_nan": dict(aperture_radius=0.5, position=(0.0, NAN, 0.0)),
    "focal_negative": dict(aperture_radius=0.5, focal_length=-1.0),
    "focal_minus_tiny": dict(aperture_radius=0.5, focal_length=-5e-324),
    "focal_nan": dict(aperture_radius=0.5, focal_length=NAN),
    "focal_minus_inf": dict(aperture_radius=0.5, focal_length=-INF),
}

# accepted as far as the device probe: the largest radius whose square cannot overflow, and a focal plane through the camera
ACCEPTED = {
    "aperture_1e150": dict(aperture_radius=1e150),
    "focal_zero": dict(aperture_radius=0.5, focal_length=0.0),
    "focal_minus_zero": dict(aperture_radius=0.5, focal_length=-0.0),
    # without depth of field none of the three values is used by the camera ray, as in the reference
    "pinhole_nan_focal": dict(aperture_radius=0.0, focal_length=NAN),
    "pinhole_negative_aperture": dict(aperture_radius=-INF, focal_length=-1.0),
}


def _status_of(fn):
    with pytest.raises(A.RaymondError) as e:
        fn()
    return e.value.status


def _renderer(cam):
    return A.Renderer(A.Scene(), settings(cam, 1), A.GpuOptions())


def _tiled(cam):
    return A.render_tiled(A.Scene(), settings(cam, 1), A.GpuOptions())


def _tiled_adaptive(cam):
    return A.render_tiled(A.Scene(), settings(cam, 4, spi=2), A.GpuOptions(), A.AdaptiveSettings(0.05))


def _tiled_two_shares(cam):
    return A.render_tiled(A.Scene(), settings(cam, 1), A.GpuOptions(device_list=[0, 0]))


ENTRY_POINTS = {"renderer": _renderer, "render_tiled": _tiled, "render_tiled_adaptive": _tiled_adaptive,
                "render_tiled_two_shares": _tiled_two_shares}


@pytest.mark.parametrize("entry", list(ENTRY_POINTS))
@pytest.mark.parametrize("case", list(REFUSED))
def test_refused_camera_is_invalid_argument(case, entry):
    cam = F.camera(8, 4, **REFUSED[case])
    assert _status_of(lambda: ENTRY_POINTS[entry](cam)) == A.RM_ERR_INVALID_ARGUMENT


def _finish(handle):
    """On a box with a GPU the accepted settings create a renderer, or render an empty 8x4 scene."""
    if isinstance(handle, A.Renderer):
        handle.close()
    else:
        handle.await_()


@pytest.mark.parametrize("entry", list(ENTRY_POINTS))
@pytest.mark.parametrize("case", list(ACCEPTED))
def test_accepted_camera_reaches_the_device_probe(case, entry):
    cam = F.camera(8, 4, **ACCEPTED[case])
    try:
        _finish(ENTRY_POINTS[entry](cam))
    except A.RaymondError as e:
        assert e.status == A.RM_ERR_CUDA, f"{case} through {entry}: status {e.status} ({e})"
