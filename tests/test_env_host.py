"""Environment maps without a GPU: the oracle with a map (tests/env_oracle.cpp) against the numpy restatement of the lookup
(tests/env_ref.py) and, with a black map, against the oracle itself; the validation of rm_scene_set_environment; and
rm_load_hdr on Radiance files generated here."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

import env_oracle as EO
import env_ref

SHAPES = [(1, 1), (1, 9), (7, 1), (16, 32), (33, 17)]


def _dirs(rng, n=4000):
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([d, env_ref.sky_dirs_edge_cases()])


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_oracle_lookup_matches_numpy(shape):
    rng = np.random.default_rng(shape[0] * 100 + shape[1])
    img = (rng.random(shape + (3,)) * 4.0).astype(np.float32)
    for scale, rotation in ((1.0, 0.0), (2.5, 1.3), (0.75, -7.0)):
        e = EO.Environment(img, scale, rotation)
        d = _dirs(rng)
        got, want = e.lookup(d), env_ref.env_lookup(img, d, scale, rotation)
        assert np.all(np.isfinite(got))
        rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
        assert rel.max() <= 1e-12, (scale, rotation, rel.max())


def test_constant_map_is_exact():
    texel = np.array([[[0.3, 1.7, 123.456]]], dtype=np.float32)
    d = _dirs(np.random.default_rng(3))
    for scale in (1.0, 0.1, 3.0):
        e = EO.Environment(texel, scale, 0.4)
        want = scale * texel.reshape(3).astype(np.float64)
        assert np.array_equal(e.lookup(d), np.broadcast_to(want, d.shape))
        assert np.array_equal(env_ref.env_lookup(texel, d, scale, 0.4), np.broadcast_to(want, d.shape))


def test_centre_column_is_plus_z_and_row_zero_is_up():
    H, W = 4, 8
    img = np.zeros((H, W, 3), dtype=np.float32)
    img[..., 0] = np.arange(W)[None, :]
    img[..., 1] = np.arange(H)[:, None]
    e = EO.Environment(img)
    # +z lands between the columns W/2 - 1 and W/2; straight up is row 0 only (clamped), straight down the last row
    assert e.lookup([[0.0, 0.0, 1.0]])[0, 0] == (W / 2 - 1 + W / 2) / 2
    assert e.lookup([[0.0, 1.0, 0.0]])[0, 1] == 0.0
    assert e.lookup([[0.0, -1.0, 0.0]])[0, 1] == H - 1


def test_nan_direction_gives_nan():
    img = np.ones((2, 4, 3), dtype=np.float32)
    e = EO.Environment(img)
    d = np.array([[np.nan, 0.0, 1.0], [0.0, np.nan, 1.0], [0.0, 0.0, np.nan]])
    assert np.all(np.isnan(e.lookup(d)))
    assert np.all(np.isnan(env_ref.env_lookup(img, d)))


@pytest.mark.parametrize("draws", O.DRAWS)
@pytest.mark.parametrize("keep", [False, True], ids=["drop", "keep"])
@pytest.mark.parametrize("name", ["box", "open"])
def test_black_map_is_the_oracle(name, keep, draws):
    """trace_env restates the oracle's trace with one change on a miss: with an all-zero map every sample and counter is the
    oracle's own (a miss delivers 0 * weights there, as the reference's trace does)."""
    objs = F.reflective_spheres() if name == "box" else F.open_spheres()
    cam = F.camera(24, 16, focal_length=2.0, aperture_radius=0.3)
    osc, esc = O.Scene(), EO.Scene(objs, EO.Environment(np.zeros((4, 8, 3), dtype=np.float32)))
    for o in objs:
        (osc.add_sphere if o[0] == "sphere" else osc.add_plane)(o[1], o[2], o[3])
    for sample in (0, 3):
        want, wc = O.render(osc, cam, 1, seed=9, first_sample=sample, bounce_limit=4, drop_nonfinite=not keep, draws=draws, worker_count=2)
        got, gc = esc.render_sample(cam, sample, seed=9, bounce_limit=4, drop_nonfinite=not keep, draws=draws, threads=2)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
        assert {k: gc[k] for k in ("rays", "shaded_tri", "nonfinite", "samples")} == {k: wc[k] for k in ("rays", "shaded_tri", "nonfinite", "samples")}


# ---------------------------------------------------------------------------- rm_scene_set_environment


def _set_raw(scene, texels, w, h, scale=1.0, rotation=0.0):
    t = np.ascontiguousarray(texels, dtype=np.float32)
    env = A.EnvironmentC(t.ctypes.data if t.size else None, w, h, scale, rotation)
    return A.lib().rm_scene_set_environment(scene._h, C.byref(env))


BAD = {
    "nan_texel": (np.array([[[1.0, np.nan, 1.0]]]), 1, 1, 1.0, 0.0),
    "inf_texel": (np.array([[[1.0, 1.0, np.inf]]]), 1, 1, 1.0, 0.0),
    "negative_texel": (np.array([[[1.0, -1e-30, 1.0]]]), 1, 1, 1.0, 0.0),
    "zero_width": (np.ones((1, 1, 3)), 0, 1, 1.0, 0.0),
    "zero_height": (np.ones((1, 1, 3)), 1, 0, 1.0, 0.0),
    "width_above_32768": (np.ones((1, 32769, 3)), 32769, 1, 1.0, 0.0),
    "height_above_32768": (np.ones((32769, 1, 3)), 1, 32769, 1.0, 0.0),
    "negative_scale": (np.ones((1, 1, 3)), 1, 1, -1.0, 0.0),
    "nan_scale": (np.ones((1, 1, 3)), 1, 1, np.nan, 0.0),
    "inf_scale": (np.ones((1, 1, 3)), 1, 1, np.inf, 0.0),
    "nan_rotation": (np.ones((1, 1, 3)), 1, 1, 1.0, np.nan),
    "inf_rotation": (np.ones((1, 1, 3)), 1, 1, 1.0, -np.inf),
    "null_texels": (np.zeros((0,)), 1, 1, 1.0, 0.0),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_invalid_environment_is_refused(case):
    s = A.Scene()
    assert _set_raw(s, *BAD[case]) == A.RM_ERR_INVALID_ARGUMENT
    assert "rm_scene_set_environment" in A.last_error()


def test_python_mirror_validates():
    s = A.Scene()
    with pytest.raises(A.RaymondError) as e:
        s.set_environment(np.ones((2, 2, 3), dtype=np.float32), scale=-2.0)
    assert e.value.status == A.RM_ERR_INVALID_ARGUMENT
    with pytest.raises(A.RaymondError):
        s.set_environment(np.ones((2, 2), dtype=np.float32))
    s.set_environment(np.ones((2, 2, 3), dtype=np.float32), scale=0.0, rotation=-3.0)
    s.set_background((0.1, 0.2, 0.3))
    s.clear_environment()
    assert A.lib().rm_scene_set_environment(None, None) == A.RM_ERR_INVALID_ARGUMENT
    assert A.lib().rm_scene_set_environment(s._h, None) == A.RM_OK      # NULL clears, also with nothing set


def test_limits_are_accepted():
    s = A.Scene()
    assert _set_raw(s, np.zeros((1, 32768, 3)), 32768, 1) == A.RM_OK
    assert _set_raw(s, np.zeros((32768, 1, 3)), 1, 32768) == A.RM_OK


# ---------------------------------------------------------------------------- rm_load_hdr


def _roundtrip(tmp_path, img, rle=True, name="m.hdr"):
    p = str(tmp_path / name)
    F.write_hdr(p, img, rle)
    return p, F.rgbe_decode(F.rgbe_encode(img))


@pytest.mark.parametrize("shape,rle", [((5, 3), False), ((4, 7), True), ((3, 8), True), ((6, 40), True), ((6, 40), False),
                                       ((2, 300), True), ((1, 32767), True), ((2, 32768), True), ((1, 40000), True)],
                         ids=lambda x: str(x))
def test_load_hdr_decodes_exactly(tmp_path, shape, rle):
    rng = np.random.default_rng(shape[1])
    img = np.exp(rng.normal(0.0, 3.0, size=shape + (3,)))
    img[:, : shape[1] // 3] = img[:, :1]                 # long runs (crossing 128 when the row is wide)
    img[0, 0] = 0.0                                      # e == 0
    p, want = _roundtrip(tmp_path, img, rle)
    got = A.load_hdr(p)
    assert got.dtype == np.float32 and got.shape == shape + (3,)
    assert np.array_equal(got, want)
    # wider than 32767 or narrower than 8: the writer stores flat, the loader must read flat
    flat = shape[1] < 8 or shape[1] > 32767 or not rle
    assert (os.path.getsize(p) == len(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n") + len(f"-Y {shape[0]} +X {shape[1]}\n") + 4 * img.size // 3) == flat


def test_load_hdr_runs_and_literals_of_every_length(tmp_path):
    W = 600
    row = np.concatenate([np.full(200, 3), np.arange(130) % 256, np.full(127, 9), np.full(128, 10), np.arange(15)])[:W]
    img = np.ldexp((row[None, :, None].astype(np.float64) + 0.5) / 256.0, 1) * np.ones((2, W, 3))
    p, want = _roundtrip(tmp_path, img, True)
    assert np.array_equal(A.load_hdr(p), want)


def test_load_hdr_rgbe_header_and_rgbe_magic(tmp_path):
    img = np.full((2, 9, 3), 0.75)
    p, want = _roundtrip(tmp_path, img, True)
    data = open(p, "rb").read().replace(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n", b"#?RGBE\n# comment\nEXPOSURE=1.0\n")
    q = tmp_path / "rgbe.hdr"
    q.write_bytes(data)
    assert np.array_equal(A.load_hdr(str(q)), want)


def _bad_file(tmp_path, data: bytes):
    p = tmp_path / "bad.hdr"
    p.write_bytes(data)
    with pytest.raises(A.RaymondError) as e:
        A.load_hdr(str(p))
    return e.value.status


def test_load_hdr_malformed(tmp_path):
    img = np.full((3, 12, 3), 2.0)
    p, _ = _roundtrip(tmp_path, img, True, "good.hdr")
    good = open(p, "rb").read()
    for cut in (5, len(good) // 2, len(good) - 1):
        assert _bad_file(tmp_path, good[:cut]) == A.RM_ERR_IMAGE, cut
    assert _bad_file(tmp_path, good.replace(b"#?RADIANCE", b"#?RADIANSE")) == A.RM_ERR_IMAGE
    assert _bad_file(tmp_path, b"P6\n" + good) == A.RM_ERR_IMAGE
    assert _bad_file(tmp_path, good.replace(b"-Y 3 +X 12", b"+Y 3 +X 12")) == A.RM_ERR_IMAGE
    assert _bad_file(tmp_path, good.replace(b"-Y 3 +X 12", b"-Y 3 -X 12")) == A.RM_ERR_IMAGE
    assert _bad_file(tmp_path, good.replace(b"-Y 3 +X 12", b"+X 12 -Y 3")) == A.RM_ERR_IMAGE
    assert _bad_file(tmp_path, good.replace(b"32-bit_rle_rgbe", b"32-bit_rle_xyze")) == A.RM_ERR_IMAGE
    assert _bad_file(tmp_path, good.replace(b"-Y 3 +X 12", b"-Y 0 +X 12")) == A.RM_ERR_IMAGE
    # a run-length scanline whose width field disagrees with the resolution line
    hdr_end = good.index(b"+X 12\n") + len(b"+X 12\n")
    assert good[hdr_end:hdr_end + 4] == bytes([2, 2, 0, 12])
    assert _bad_file(tmp_path, good[:hdr_end] + bytes([2, 2, 0, 13]) + good[hdr_end + 4:]) == A.RM_ERR_IMAGE


def test_load_hdr_missing_file(tmp_path):
    with pytest.raises(A.RaymondError) as e:
        A.load_hdr(str(tmp_path / "missing.hdr"))
    assert e.value.status == A.RM_ERR_IO


def test_sky_fixture_roundtrips(tmp_path):
    sky = F.sky(128, 64)
    assert sky.shape == (64, 128, 3) and sky.dtype == np.float32 and np.all(sky >= 0) and sky.max() > 100.0
    p, want = _roundtrip(tmp_path, sky, True)
    assert np.array_equal(A.load_hdr(p), want)
