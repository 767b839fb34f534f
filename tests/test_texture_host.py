"""Colour textures without a GPU: the oracle with textures (tests/tex_oracle.cpp) against the numpy restatement of the lookup
and of the uv of each geometry kind (tests/tex_ref.py), to the bit; with all-ones textures, against the oracle itself; and the
validation of rm_scene_set_texture."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

import tex_oracle as TO
import tex_ref
from util import oracle_scene

SHAPES = [(1, 1), (1, 9), (7, 1), (16, 32), (33, 17)]
SCALES = [(1.0, 1.0), (3.0, 0.5), (-2.0, 7.25), (0.0, 1.0)]


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def _uvs(rng, n=3000):
    """Random uv, the seams, values just below 0 and 1 (s' - floor(s') rounds to 1 there), large and negative uv."""
    tiny = np.nextafter(0.0, -1.0)
    edges = [[0.0, 0.0], [1.0, 1.0], [0.5, 0.5], [-0.0, -0.0], [tiny, tiny], [-1e-17, 0.3], [0.3, -1e-17],
             [np.nextafter(1.0, 0.0), np.nextafter(1.0, 0.0)], [1.0 + 2e-16, 2.0], [-1.0, -3.0], [1e15 + 0.25, -1e15 - 0.75],
             [1e300, 0.5], [-1e300, 0.5], [123456.789, -98765.4321], [1e-300, -1e-300]]
    return np.concatenate([rng.uniform(-3.0, 4.0, size=(n, 2)), np.array(edges)])


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_oracle_lookup_matches_numpy_to_the_bit(shape):
    rng = np.random.default_rng(shape[0] * 100 + shape[1])
    img = (rng.random(shape + (3,)) * 4.0).astype(np.float32)
    for scale in SCALES:
        st = _uvs(rng)
        got, want = TO.Texture(img, scale).lookup(st), tex_ref.tex_lookup(img, st, scale)
        fin = np.isfinite(want).all(axis=1)
        assert np.isnan(got[~fin]).all()
        assert bits_equal(got, want), scale


def test_nonfinite_uv_gives_nan():
    img = np.ones((2, 4, 3), dtype=np.float32)
    st = np.array([[np.nan, 0.0], [0.0, np.nan], [np.inf, 0.5], [0.5, -np.inf], [1e200, 0.5]])
    for scale in ((1.0, 1.0), (1e200, 1e200)):
        got, want = TO.Texture(img, scale).lookup(st), tex_ref.tex_lookup(img, st, scale)
        assert bits_equal(got, want)
    assert np.isnan(TO.Texture(img).lookup(st[:4])).all()
    assert np.isnan(TO.Texture(img, (1e200, 1e200)).lookup(st)).all()        # s' = 1e200 * 1e200 overflows


def test_single_texel_and_all_ones_are_exact():
    texel = np.array([[[0.3, 1.7, 123.456]]], dtype=np.float32)
    st = _uvs(np.random.default_rng(3))[:-3]
    want = texel.reshape(3).astype(np.float64)
    for scale in SCALES:
        assert np.array_equal(TO.Texture(texel, scale).lookup(st), np.broadcast_to(want, st.shape[:1] + (3,)))
        ones = np.ones((5, 7, 3), dtype=np.float32)
        assert np.array_equal(TO.Texture(ones, scale).lookup(st), np.ones((st.shape[0], 3)))


def test_texel_centres_and_orientation():
    H, W = 4, 8
    img = np.zeros((H, W, 3), dtype=np.float32)
    img[..., 0] = np.arange(W)[None, :]
    img[..., 1] = np.arange(H)[:, None]
    t = TO.Texture(img)
    # the centre of texel (row r, column c) is at s = (c + 0.5) / W, t = 1 - (r + 0.5) / H: row 0 is the top (t = 1)
    for r, c in ((0, 0), (3, 7), (1, 5)):
        got = t.lookup([[(c + 0.5) / W, 1.0 - (r + 0.5) / H]])[0]
        assert got[0] == c and got[1] == r
    # half-way across the u seam: the mean of the last and the first column (repeat)
    assert t.lookup([[0.0, 1.0 - 0.5 / H]])[0, 0] == (W - 1 + 0) / 2
    assert t.lookup([[0.5 / W, 1.0]])[0, 1] == (H - 1 + 0) / 2


def test_sphere_uv_matches_numpy():
    rng = np.random.default_rng(5)
    n = rng.normal(size=(4000, 3))
    n /= np.linalg.norm(n, axis=1, keepdims=True)
    s = np.sqrt(0.5)
    edges = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, -1.0], [-0.0, 0.0, -1.0], [1e-300, 0.0, -1.0], [-1e-300, 0.0, -1.0],
                      [0.0, 1.0, 0.0], [0.0, -1.0, 0.0], [0.0, 1.0 + 1e-16, 0.0], [s, 0.0, s], [-s, 0.0, -s], [0.0, -3.0, 0.0]])
    n = np.concatenate([n, edges])
    got, want = TO.sphere_uv(n), tex_ref.sphere_uv(n)
    # glibc's atan2 / acos against numpy's: the same to an ulp or two
    assert np.abs(got - want).max() <= 4e-16
    assert bits_equal(TO.sphere_uv(edges), tex_ref.sphere_uv(edges))
    assert np.isnan(TO.sphere_uv([[np.nan, 0.0, 1.0]])[:, 0]).all() and np.isnan(TO.sphere_uv([[0.0, np.nan, 1.0]])[:, 1]).all()


@pytest.mark.parametrize("normal", [(0.0, 1.0, 0.0), (0.0, 0.0, -1.0), (0.0, 0.0, 1.0), (-1.0, 0.0, 0.0), (0.3, 0.4, -0.866)])
def test_plane_uv_matches_numpy_to_the_bit(normal):
    rng = np.random.default_rng(7)
    origin = (0.5, -1.0, 2.0)
    frags = rng.uniform(-50.0, 50.0, size=(2000, 3))
    assert bits_equal(TO.plane_uv(origin, normal, frags), tex_ref.plane_uv(origin, normal, frags))


def test_triangle_uv_matches_numpy_to_the_bit():
    rng = np.random.default_rng(11)
    tris = F.bumpy_sphere(uv=True)
    k = rng.integers(0, tris.shape[0], size=3000)
    pos = F.positions(tris[k])
    w = rng.dirichlet((1.0, 1.0, 1.0), size=k.size)
    pts = (pos * w[:, :, None]).sum(axis=1)
    got, want = TO.triangle_uv(tris[k], pts), tex_ref.triangle_uv(tris[k], pts)
    assert bits_equal(got, want)
    uv = tris[k].reshape(-1, 3, 11)[:, :, 6:8]
    assert np.abs(got - (uv * w[:, :, None]).sum(axis=1)).max() < 1e-6       # the weights are the barycentrics


def test_fixture_uv_leaves_the_default_arrays():
    for mk in (lambda **kw: F.dragon_standin(40, 12, **kw), F.bumpy_sphere):
        a, b = mk(), mk(uv=True)
        cols = np.ones(F.TRI_DOUBLES, bool)
        cols[[6, 7, 17, 18, 28, 29]] = False
        assert np.array_equal(a[:, cols], b[:, cols]) and not a[:, ~cols].any()
        assert 0.0 <= b[:, ~cols].min() and b[:, ~cols].max() == 1.0


def _ones_textures(objs):
    return {i: TO.Texture(np.ones((1, 1, 3), dtype=np.float32), (2.0, 3.0)) for i, o in enumerate(objs)
            if o[-1][0] in ("Diffuse", "Metal")}


@pytest.mark.parametrize("draws", O.DRAWS)
@pytest.mark.parametrize("keep", [False, True], ids=["drop", "keep"])
@pytest.mark.parametrize("name", ["spheres", "dragon"])
def test_all_ones_textures_are_the_oracle(name, keep, draws):
    """trace_tex restates trace_env with one change, the colour of a textured object: all-ones textures on every Diffuse and
    Metal object give the oracle's own samples and counters."""
    mesh = F.dragon_standin(48, 12, uv=True)
    objs = F.reflective_spheres() if name == "spheres" else F.gold_dragon(mesh)
    cam = F.camera(24, 16)
    osc, tsc = oracle_scene(objs), TO.Scene(objs, _ones_textures(objs))
    for sample in (0, 3):
        want, wc = O.render(osc, cam, 1, seed=9, first_sample=sample, bounce_limit=4, drop_nonfinite=not keep, draws=draws, worker_count=2)
        got, gc = tsc.render_sample(cam, sample, seed=9, bounce_limit=4, drop_nonfinite=not keep, draws=draws, threads=2)
        assert bits_equal(got, want)
        keys = ("rays", "shaded_tri", "nonfinite", "samples")
        assert {k: gc[k] for k in keys} == {k: wc[k] for k in keys}


def test_textures_change_the_frame():
    objs = F.reflective_spheres()
    cam = F.camera(24, 16)
    plain, _ = TO.Scene(objs, {}).render_sample(cam, 0, seed=9, threads=2)
    checker = np.indices((4, 4)).sum(axis=0) % 2
    img = np.stack([checker, 1 - checker, checker], axis=-1).astype(np.float32)
    textured, _ = TO.Scene(objs, {0: TO.Texture(img), 2: TO.Texture(img, (4.0, 4.0))}).render_sample(cam, 0, seed=9, threads=2)
    assert not np.array_equal(plain, textured)


# ---------------------------------------------------------------------------- rm_scene_set_texture


def _set_raw(scene, index, texels, w, h, su=1.0, sv=1.0):
    t = np.ascontiguousarray(texels, dtype=np.float32)
    tex = A.TextureC(t.ctypes.data if t.size else None, w, h, su, sv)
    return A.lib().rm_scene_set_texture(scene._h if scene is not None else None, index, C.byref(tex))


BAD = {
    "nan_texel": (0, np.array([[[1.0, np.nan, 1.0]]]), 1, 1, 1.0, 1.0),
    "inf_texel": (0, np.array([[[1.0, 1.0, np.inf]]]), 1, 1, 1.0, 1.0),
    "negative_texel": (0, np.array([[[1.0, -1e-30, 1.0]]]), 1, 1, 1.0, 1.0),
    "zero_width": (0, np.ones((1, 1, 3)), 0, 1, 1.0, 1.0),
    "zero_height": (0, np.ones((1, 1, 3)), 1, 0, 1.0, 1.0),
    "width_above_32768": (0, np.ones((1, 32769, 3)), 32769, 1, 1.0, 1.0),
    "height_above_32768": (0, np.ones((32769, 1, 3)), 1, 32769, 1.0, 1.0),
    "nan_scale_u": (0, np.ones((1, 1, 3)), 1, 1, np.nan, 1.0),
    "inf_scale_v": (0, np.ones((1, 1, 3)), 1, 1, 1.0, -np.inf),
    "null_texels": (0, np.zeros((0,)), 1, 1, 1.0, 1.0),
    "index_out_of_range": (8, np.ones((1, 1, 3)), 1, 1, 1.0, 1.0),
}


@pytest.mark.parametrize("case", sorted(BAD))
def test_invalid_texture_is_refused(case):
    s = A.Scene.from_fixture(F.reflective_spheres())
    assert _set_raw(s, *BAD[case]) == A.RM_ERR_INVALID_ARGUMENT
    assert "rm_scene_set_texture" in A.last_error()


def test_null_scene_is_refused():
    assert _set_raw(None, 0, np.ones((1, 1, 3)), 1, 1) == A.RM_ERR_INVALID_ARGUMENT
    assert "rm_scene_set_texture" in A.last_error()
    assert A.lib().rm_scene_set_texture(None, 0, None) == A.RM_ERR_INVALID_ARGUMENT


def test_emission_object_is_unsupported():
    s = A.Scene.from_fixture(F.reflective_spheres())
    ceiling = 3                                          # BOX_PLANES[1], after the two spheres
    assert F.reflective_spheres()[ceiling][3][0] == "Emission"
    assert _set_raw(s, ceiling, np.ones((1, 1, 3)), 1, 1) == A.RM_ERR_UNSUPPORTED
    assert "rm_scene_set_texture" in A.last_error()
    with pytest.raises(A.RaymondError) as e:
        s.set_texture(ceiling, np.ones((2, 2, 3), dtype=np.float32))
    assert e.value.status == A.RM_ERR_UNSUPPORTED
    # unbinding is always allowed
    s.clear_texture(ceiling)


def test_valid_textures_and_unbinding():
    s = A.Scene.from_fixture(F.reflective_spheres())
    for i in (0, 1, 2, 4, 7):
        assert _set_raw(s, i, np.ones((3, 5, 3)), 5, 3, -2.0, 0.0) == A.RM_OK
    s.set_texture(0, np.zeros((32768, 1, 3), dtype=np.float32), scale=(1e300, -1e300))
    s.clear_texture(0)
    s.clear_texture(0)
    with pytest.raises(A.RaymondError):
        s.clear_texture(8)
    with pytest.raises(A.RaymondError):
        s.set_texture(0, np.ones((2, 2), dtype=np.float32))
    assert len(s) == 8


def test_ctypes_mirror_has_the_header_layout():
    assert C.sizeof(A.TextureC) == 40
    assert [A.TextureC.__dict__[f].offset for f in ("texels", "width", "height", "scale_u", "scale_v")] == [0, 8, 16, 24, 32]
