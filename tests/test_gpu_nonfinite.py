"""Non-finite samples against the oracle: scenes whose shading normals are NaN, so that the reference's samples are NaN.

The scenes of the other parity tests never produce a non-finite sample, so their `nonfinite_samples == oracle` checks compare
0 with 0.  Here every fixture does (test_oracle_produces_nonfinite_samples holds the oracle to that on the CPU):

* "nobox": a bumpy sphere whose every 5th triangle has zero vertex normals (the interpolated normal normalises to NaN), Metal
  like the dragon, under the emissive ceiling of the box;
* "box": the same mesh in the full box with the red sphere, so paths also reach NaN hits after a black wall zeroed their
  throughput;
* "sliver": needle triangles 1e9 times longer than high.  Heron's formula (triangle.rs:47-68) computes their area as
  s (s - a) (s - b) (s - c) with s - a cancelling to 0 (or below), so the barycentric weights are 0 / 0 and the normal is NaN —
  the source the reference itself is exposed to on real meshes (SURVEY A17).

A Metal surface with a NaN normal gives a NaN lobe weight.  The reference multiplies the child's radiance by it, and the child
returns 0 (the continuation ray has a NaN direction and misses), so the sample is NaN.  RM_FLAG_KEEP_NONFINITE must reproduce
that sample for sample; the default mode drops non-finite samples, so its frame equals the reference's drop-mode frame.
"""
import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import oracle_scene, product_scene, settings

CAM = F.camera(64, 48)
SPP, SEED = 4, 3


def nan_normal_mesh() -> np.ndarray:
    m = F.translate(F.bumpy_sphere(20, 40, 0.6, 0.1, (1.0, 0.8, 0.6)), (0.3, -0.3, 3.2))
    m.reshape(-1, 3, 11)[::5, :, 3:6] = 0.0
    return m


def sliver_mesh(n: int = 12, length: float = 5e7, height: float = 0.05, z: float = 2.0) -> np.ndarray:
    """`n` needle triangles across the view at depth `z`, each `height` high and 2 `length` wide (height / length = 1e-9: at
    1e-7 the same layout has finite normals), plus two small triangles at opposite corners of a cube around them, so that the
    grid resolution estimate gives every axis at least one cell."""
    ys = np.linspace(-0.4, 0.4, n) * z
    p0 = np.stack([np.full(n, -length), ys, np.full(n, z)], axis=1)
    p1 = np.stack([np.full(n, length), ys, np.full(n, z)], axis=1)
    p2 = np.stack([np.zeros(n), ys + height, np.full(n, z)], axis=1)
    corners = np.array([[-length, -length, -length], [length, length, length]])
    anchors = F.make_triangles(corners, corners + [1.0, 0.0, 0.0], corners + [0.0, 1.0, 0.0])
    return np.concatenate([F.make_triangles(p0, p1, p2), anchors])


def scenes() -> dict:
    m = nan_normal_mesh()
    ceiling = F.BOX_PLANES[1]
    return {
        "nobox": [("grid", m, F.DRAGON_MATERIAL), ceiling],
        "box": [F.RED_SPHERE, ("grid", m, F.DRAGON_MATERIAL)] + F.BOX_PLANES,
        "sliver": [("grid", sliver_mesh(), F.DRAGON_MATERIAL), ceiling],
    }


SCENES = scenes()


def gpu_sums(objs, bounce_limit, flags=0, precision=A.PRECISION_F64):
    r = A.Renderer(product_scene(objs), settings(CAM, SPP, bounce_limit=bounce_limit),
                   A.GpuOptions(seed=SEED, flags=flags, precision=precision))
    r.render(0, SPP)
    sums = r.read_sums()
    stats = r.stats()
    r.close()
    return sums, stats


def oracle_sums(objs, bounce_limit, keep):
    return O.render(oracle_scene(objs), CAM, SPP, seed=SEED, bounce_limit=bounce_limit, drop_nonfinite=not keep)


def nonfinite_pixels(x):
    return ~np.isfinite(x).all(axis=-1)


def assert_nonfinite_classes_equal(g, o, what):
    """Per channel: NaN where the oracle is NaN, +Inf / -Inf where it is."""
    for name, f in (("NaN", np.isnan), ("+Inf", np.isposinf), ("-Inf", np.isneginf)):
        bad = np.argwhere(f(g) != f(o))
        assert bad.size == 0, f"{what}: {len(bad)} channels differ in being {name}, first (y, x, c) {bad[:5].tolist()}"


def assert_finite_pixels_close(g, o, what):
    """Where the oracle's pixel is finite, the GPU's is finite and agrees to 1e-9 relative (the same measure and the same
    room for one libm-flipped branch as test_gpu_render.compare_same_stream)."""
    fin = ~nonfinite_pixels(o)
    assert np.isfinite(g[fin]).all(), f"{what}: non-finite GPU values on finite oracle pixels"
    gm, om = g[fin] / SPP, o[fin] / SPP
    rel = np.abs(gm - om).max(axis=-1) / np.maximum(np.abs(om).max(axis=-1), 1e-3)
    outliers = int((rel > 1e-9).sum())
    assert outliers <= max(1, int(1e-4 * rel.size)), f"{what}: {outliers} finite pixels differ beyond 1e-9 relative (largest {rel.max():.3g})"


@pytest.mark.parametrize("name", list(SCENES))
def test_oracle_produces_nonfinite_samples(name):
    """The fixtures below are only meaningful if the reference's samples on them are non-finite (CPU only)."""
    objs = SCENES[name]
    for limit in (1, 5):
        sums, cnt = oracle_sums(objs, limit, keep=True)
        assert cnt["nonfinite"] > 0, f"{name}, bounce_limit {limit}: the oracle produced no non-finite sample"
        assert np.isnan(sums).any(axis=-1).sum() >= 1, f"{name}, bounce_limit {limit}: no NaN pixel"
        dropped, dcnt = oracle_sums(objs, limit, keep=False)
        assert np.isfinite(dropped).all() and dcnt["nonfinite"] == cnt["nonfinite"]


@pytest.mark.gpu
@pytest.mark.parametrize("limit", [1, 5])
@pytest.mark.parametrize("name", list(SCENES))
def test_keep_nonfinite_same_stream(name, limit):
    """RM_FLAG_KEEP_NONFINITE against render(drop_nonfinite=False): the same pixels are NaN / Inf, the finite pixels agree, and
    the statistics are the reference's — nonfinite_samples, and rays, since no path is stopped early in this mode."""
    objs = SCENES[name]
    g, gs = gpu_sums(objs, limit, flags=A.FLAG_KEEP_NONFINITE)
    o, oc = oracle_sums(objs, limit, keep=True)
    what = f"{name} bounce_limit {limit} keep"
    assert_nonfinite_classes_equal(g, o, what)
    assert np.array_equal(nonfinite_pixels(g), nonfinite_pixels(o))
    assert_finite_pixels_close(g, o, what)
    assert gs["samples"] == oc["samples"] == CAM["width"] * CAM["height"] * SPP
    assert gs["nonfinite_samples"] == oc["nonfinite"] > 0
    assert gs["rays"] == oc["rays"]


@pytest.mark.gpu
@pytest.mark.parametrize("limit", [1, 5])
@pytest.mark.parametrize("name", list(SCENES))
def test_drop_nonfinite_same_stream(name, limit):
    """The default mode: finite sums equal to the reference's drop-mode sums.  nonfinite_samples counts the non-finite values
    the GPU's own paths deliver, a lower bound of the reference's count (include/raymond.h).  On these scenes it is exactly 0:
    every non-finite reference sample comes from a NaN normal, the path's continuation ray has a NaN origin and direction and
    misses, and a missed path delivers an exact 0 where the reference multiplies 0 by the NaN weight."""
    objs = SCENES[name]
    g, gs = gpu_sums(objs, limit)
    o, oc = oracle_sums(objs, limit, keep=False)
    assert np.isfinite(g).all()
    assert_finite_pixels_close(g, o, f"{name} bounce_limit {limit} drop")
    assert gs["nonfinite_samples"] <= oc["nonfinite"]
    assert gs["nonfinite_samples"] == 0
    assert gs["rays"] <= oc["rays"]


@pytest.mark.gpu
def test_keep_nonfinite_render_tiled_two_shares():
    """Keep mode through render_tiled with two shares on one GPU (peer reduce of the accumulators and the fused finalize):
    the awaited frame is NaN exactly where the reference's is; the GPU tonemap epilogue shows those pixels as (0, 0, 0)."""
    objs, limit = SCENES["box"], 5
    st = settings(CAM, SPP, bounce_limit=limit)
    task = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=SEED, flags=A.FLAG_KEEP_NONFINITE, device_list=[0, 0]))
    frame = task.await_()
    stats = task.stats()
    o, oc = oracle_sums(objs, limit, keep=True)
    mask = nonfinite_pixels(o)
    assert mask.sum() > 0
    assert np.array_equal(nonfinite_pixels(frame), mask)
    assert_nonfinite_classes_equal(frame, o / SPP, "render_tiled keep")
    assert_finite_pixels_close(frame * SPP, o, "render_tiled keep")
    assert stats["nonfinite_samples"] == oc["nonfinite"]
    assert stats["rays"] == oc["rays"]

    r = A.Renderer(product_scene(objs), st, A.GpuOptions(seed=SEED, flags=A.FLAG_KEEP_NONFINITE))
    r.render(0, SPP)
    rgb = r.read_rgb8(SPP)
    mean = r.read_frame(SPP)
    r.close()
    assert np.array_equal(nonfinite_pixels(mean), mask)
    assert not rgb[mask].any(), "a non-finite pixel is not (0, 0, 0) in the 8-bit view"
    # everywhere else the epilogue is cli_old's tonemap of the frame (within one level: GPU expf / powf)
    diff = np.abs(rgb.astype(int) - F.tonemap(mean).astype(int))
    assert diff.max() <= 1
    assert rgb[~mask].any(axis=-1).mean() > 0.3


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENES))
def test_keep_nonfinite_f32_shading(name):
    """RM_PRECISION_F32_SHADING in keep mode at bounce_limit 1: camera rays, hits and normals are f64 in both modes and the
    lobe of a NaN normal is NaN in either arithmetic, so the NaN pixels and the count are the f64 mode's (and the reference's).
    At this depth every finite sample is an emission seen directly or a zero, so the finite sums are identical as well."""
    objs, limit = SCENES[name], 1
    g32, s32 = gpu_sums(objs, limit, flags=A.FLAG_KEEP_NONFINITE, precision=A.PRECISION_F32_SHADING)
    g64, s64 = gpu_sums(objs, limit, flags=A.FLAG_KEEP_NONFINITE)
    o, oc = oracle_sums(objs, limit, keep=True)
    assert_nonfinite_classes_equal(g32, g64, f"{name} f32shade vs f64")
    assert np.array_equal(nonfinite_pixels(g32), nonfinite_pixels(o))
    assert s32["nonfinite_samples"] == s64["nonfinite_samples"] == oc["nonfinite"]
    fin = ~nonfinite_pixels(g64)
    assert np.array_equal(g32[fin], g64[fin])
    assert s32["rays"] == s64["rays"] == oc["rays"]
