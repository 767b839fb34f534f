"""Colour textures on the GPU (rm_scene_set_texture, include/raymond.h).

At a hit on a textured object the material's colour a becomes a (*) T(s, t).  Nothing else changes: the draws, the hits and
the ray counts are those of the scene without textures, so all-ones textures render to the same bits, and textured scenes
are held path for path against the oracle with textures (tests/tex_oracle.cpp)."""
import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

import denoise_ref as D
import tex_oracle as TO
import tex_ref
from test_gpu_configs import THREADS, compare_paths, gpu_sample_frames
from test_gpu_f32_paths import compare_f32_paths
from util import product_scene, settings

pytestmark = pytest.mark.gpu

SEED = 91
SKY = F.sky(128, 64, sun_radiance=40.0)
SKY_SCALE, SKY_ROT = 1.3, 0.7
PRECISIONS = [A.PRECISION_F64, A.PRECISION_F32_SHADING]
# Path-for-path bar of the f64 mode: hits are bit-exact, and the uv of a plane or a grid hit is the same expression on both
# sides, so paths differ only by what CUDA's and glibc's atan2 / acos return (the sphere mapping and the sky).  Largest
# per-path relative difference measured on one B200 (1000 W power limit) over every case of test_textured_paths_f64 and
# test_textured_paths_keep: 3.3e-10 (textured open spheres, bounce limit 5; 4.1e-12 for the open dragon, 3.9e-14 for the
# closed box, 3.4e-15 or less at limit 1).  The bar is about 20x that.
PATH_REL_BAR = 7e-9
# Bars of the f32 mode against the oracle on the f32 draws (compare_f32_paths): the textured colour is rounded to f32 where
# the plain materials' colours were exact in f32.  Measured on one B200 over every case of test_textured_paths_f32: 99th
# percentile 1.1e-5 and 7.8e-4 of the paths beyond 1e-3 (both open dragon, limit 5).  The bars are about 3x that.
F32_P99_BAR, F32_GROSS_BAR = 3e-5, 2e-3


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def stripes(W=64, H=32):
    """A texture with edges in both directions, values in [0.1, 1]."""
    u = (np.arange(W) + 0.5) / W
    v = (np.arange(H) + 0.5) / H
    U, V = np.meshgrid(u, v)
    c = (np.floor(U * 8) + np.floor(V * 4)) % 2
    img = np.stack([0.1 + 0.9 * c, 0.2 + 0.8 * U, 0.3 + 0.7 * (1.0 - V)], axis=-1)
    return np.ascontiguousarray(img, dtype=np.float32)


TEX = stripes()
FLOOR_TEX = stripes(16, 16)


def dragon_mesh():
    return F.dragon_standin(96, 24, uv=True)


# scene name -> (objects, {object index: (image, scale)}, environment map or None, camera)
def scene_case(name):
    if name == "spheres":
        objs = F.open_spheres()
        return objs, {0: (TEX, (1.0, 1.0)), 1: (TEX, (2.0, 1.0)), 3: (TEX, (-1.0, 3.0)), 4: (FLOOR_TEX, (0.5, 0.5))}, True, F.camera(64, 48)
    if name == "dragon":
        objs = F.open_dragon(dragon_mesh())
        return objs, {0: (TEX, (1.0, 1.0)), 1: (TEX, (4.0, 1.0)), 2: (FLOOR_TEX, (2.0, 2.0))}, True, F.camera(64, 40)
    objs = F.gold_dragon(dragon_mesh())            # the closed box: textured sphere, dragon, floor and front wall
    return objs, {0: (TEX, (1.0, 1.0)), 1: (TEX, (4.0, 1.0)), 2: (FLOOR_TEX, (2.0, 2.0)), 4: (TEX, (0.25, 0.25))}, False, F.camera(64, 40)


CASES = ["spheres", "dragon", "box"]


def gpu_scene(objs, tex, env):
    s = product_scene(objs)
    for i, (img, sc) in tex.items():
        s.set_texture(i, img, scale=sc)
    if env:
        s.set_environment(SKY, SKY_SCALE, SKY_ROT)
    return s


def oracle_scene(objs, tex, env):
    return TO.Scene(objs, {i: TO.Texture(img, sc) for i, (img, sc) in tex.items()}, (SKY, SKY_SCALE, SKY_ROT) if env else None)


def oracle_frames(osc, cam, spp, limit, keep=False, draws="f64"):
    o, oc = [], {}
    for s in range(spp):
        f, c = osc.render_sample(cam, s, seed=SEED, bounce_limit=limit, drop_nonfinite=not keep, draws=draws, threads=THREADS)
        o.append(f)
        oc = {k: oc.get(k, 0) + v for k, v in c.items()}
    return o, oc


def _render(scene, st, spp, **opt):
    r = A.Renderer(scene, st, A.GpuOptions(seed=SEED, flags=A.FLAG_MOMENTS | opt.pop("flags", 0), **opt))
    r.render(0, spp)
    out = r.read_sums(), r.read_moments(), r.stats()
    r.close()
    return out


# ---------------------------------------------------------------------------- all-ones textures: nothing changes


@pytest.mark.parametrize("keep", [False, True], ids=["drop", "keep"])
@pytest.mark.parametrize("precision", PRECISIONS, ids=["f64", "f32"])
@pytest.mark.parametrize("name", ["spheres", "dragon"])
def test_all_ones_textures_are_the_same_frame(name, precision, keep):
    objs = F.reflective_spheres() if name == "spheres" else F.gold_dragon(dragon_mesh())
    ones = {i: (np.ones((3, 5, 3), dtype=np.float32), (1.7, -2.3)) for i, o in enumerate(objs) if o[-1][0] != "Emission"}
    st, spp = settings(F.camera(96, 64), 6), 6
    flags = A.FLAG_KEEP_NONFINITE if keep else 0
    S0, Q0, s0 = _render(product_scene(objs), st, spp, precision=precision, flags=flags)
    S1, Q1, s1 = _render(gpu_scene(objs, ones, False), st, spp, precision=precision, flags=flags)
    assert bits_equal(S1, S0) and bits_equal(Q1, Q0)
    for k in ("rays", "samples", "nonfinite_samples"):
        assert s1[k] == s0[k], k


# ---------------------------------------------------------------------------- path for path against trace_tex


@pytest.mark.parametrize("limit", [1, 3, 5])
@pytest.mark.parametrize("name", CASES)
def test_textured_paths_f64(name, limit):
    objs, tex, env, cam = scene_case(name)
    spp = 3
    g, gs = gpu_sample_frames(gpu_scene(objs, tex, env), settings(cam, spp, bounce_limit=limit), spp, SEED)
    o, oc = oracle_frames(oracle_scene(objs, tex, env), cam, spp, limit)
    plain, _ = oracle_frames(oracle_scene(objs, {}, env), cam, 1, limit)
    g, o = np.stack(g), np.stack(o)
    rel = np.abs(g - o).max(axis=-1) / np.maximum(np.abs(o).max(axis=-1), 1e-3)
    print(f"texture paths | {name} limit {limit} | largest relative difference {rel.max():.3g}")
    if limit > 1:
        assert not np.array_equal(o[0], plain[0])           # the textures change the frame
    # no path may differ by more than 1e-3; PATH_REL_BAR bounds all of them
    compare_paths(list(g), list(o), f"{name} textured limit {limit}", max_differing=1.0, max_gross=0.0)
    assert rel.max() <= PATH_REL_BAR
    assert gs["samples"] == oc["samples"] and gs["rays"] <= oc["rays"]


@pytest.mark.parametrize("limit", [2, 5])
@pytest.mark.parametrize("name", CASES)
def test_textured_paths_keep(name, limit):
    objs, tex, env, cam = scene_case(name)
    spp = 2
    g, gs = gpu_sample_frames(gpu_scene(objs, tex, env), settings(cam, spp, bounce_limit=limit), spp, SEED, flags=A.FLAG_KEEP_NONFINITE)
    o, oc = oracle_frames(oracle_scene(objs, tex, env), cam, spp, limit, keep=True)
    g, o = np.stack(g), np.stack(o)
    assert gs["rays"] == oc["rays"] and gs["nonfinite_samples"] == oc["nonfinite"]
    for f in (np.isnan, np.isposinf, np.isneginf):
        assert np.array_equal(f(g), f(o))
    fin = np.isfinite(o).all(axis=-1)
    rel = np.abs(g[fin] - o[fin]).max(axis=-1) / np.maximum(np.abs(o[fin]).max(axis=-1), 1e-3)
    print(f"texture paths | {name} keep limit {limit} | largest relative difference {rel.max():.3g} | non-finite {gs['nonfinite_samples']}")
    assert rel.max() <= PATH_REL_BAR, rel.max()


@pytest.mark.parametrize("limit", [1, 3, 5])
@pytest.mark.parametrize("name", CASES)
def test_textured_paths_f32(name, limit):
    objs, tex, env, cam = scene_case(name)
    spp = 3
    g, gs = gpu_sample_frames(gpu_scene(objs, tex, env), settings(cam, spp, bounce_limit=limit), spp, SEED, precision=A.PRECISION_F32_SHADING)
    o, oc = oracle_frames(oracle_scene(objs, tex, env), cam, spp, limit, draws="f32")
    compare_f32_paths(np.stack(g), np.stack(o), f"{name} textured limit {limit} f32", p99_max=F32_P99_BAR, gross_max=F32_GROSS_BAR)
    assert gs["samples"] == oc["samples"]


# ---------------------------------------------------------------------------- the albedo feature buffer


def _normalize(a):
    return a * (1.0 / np.sqrt((a[:, 0] * a[:, 0] + a[:, 1] * a[:, 1]) + a[:, 2] * a[:, 2]))[:, None]


@pytest.mark.parametrize("name", ["spheres", "dragon"])
def test_albedo_is_the_textured_colour(name):
    """RM_FLAG_AOV at 1 spp: the albedo of every pixel is a (*) T(s, t) at its camera ray's first hit, with (s, t) and T from
    tex_ref.py — the direct check of the device lookup and of the three mappings."""
    objs, tex, env, cam = scene_case(name)
    s = gpu_scene(objs, tex, env)
    r = A.Renderer(s, settings(cam, 1), A.GpuOptions(seed=SEED, flags=A.FLAG_AOV))
    r.render(0, 1)
    alb = r.read_aovs(1)[0].reshape(-1, 3)
    r.close()
    rays = O.camera_rays(cam, SEED, 0)
    obj, sub, t = s.intersect(rays)
    want = np.zeros_like(alb)
    frag = rays[:, 0:3] + rays[:, 3:6] * t[:, None]
    kinds = set()
    for i, o in enumerate(objs):
        m = obj == i
        if not m.any():
            continue
        a = np.asarray(o[-1][1], dtype=np.float64)
        if i not in tex:
            want[m] = a
            continue
        if o[0] == "sphere":
            st = tex_ref.sphere_uv(_normalize(frag[m] - np.asarray(o[1])))
        elif o[0] == "plane":
            st = tex_ref.plane_uv(o[1], o[2], frag[m])
        else:
            st = tex_ref.triangle_uv(np.asarray(o[1])[sub[m]], frag[m])
        kinds.add(o[0])
        want[m] = a * tex_ref.tex_lookup(tex[i][0], st, tex[i][1])
    rel = np.abs(alb - want).max(axis=-1) / np.maximum(np.abs(want).max(axis=-1), 1e-3)
    print(f"albedo | {name} | {sorted(kinds)} | largest relative difference from tex_ref {rel.max():.3g}")
    assert kinds == ({"sphere", "plane"} if name == "spheres" else {"sphere", "plane", "grid"})
    assert rel.max() <= 1e-12
    assert np.unique(want.round(6), axis=0).shape[0] > 50       # the textures vary across the frame


# ---------------------------------------------------------------------------- the other features


@pytest.mark.parametrize("switch", ["RM_FULL_LAST_BOUNCE", "RM_NO_COVER_MASK"])
@pytest.mark.parametrize("precision", PRECISIONS, ids=["f64", "f32"])
@pytest.mark.parametrize("name", CASES)
def test_switches_give_the_same_bits(name, precision, switch, monkeypatch):
    objs, tex, env, cam = scene_case(name)
    out = []
    for on in (False, True):
        if on:
            monkeypatch.setenv(switch, "1")
        else:
            monkeypatch.delenv(switch, raising=False)
        r = A.Renderer(gpu_scene(objs, tex, env), settings(cam, 4, bounce_limit=3), A.GpuOptions(seed=SEED, precision=precision))
        r.render(0, 4)
        out.append((r.read_sums(), r.stats()))
        r.close()
    monkeypatch.delenv(switch, raising=False)
    (a, sa), (b, sb) = out
    assert bits_equal(a, b)
    assert sa["rays"] == sb["rays"] and sa["nonfinite_samples"] == sb["nonfinite_samples"]


def test_placements_keep_the_textures_they_were_made_with():
    objs, tex, env, cam = scene_case("spheres")
    st, spp = settings(cam, 3), 3
    plain = A.render_tiled(gpu_scene(objs, {}, env), st, A.GpuOptions(seed=SEED)).await_()
    textured = A.render_tiled(gpu_scene(objs, tex, env), st, A.GpuOptions(seed=SEED)).await_()
    assert not bits_equal(plain, textured)
    s = gpu_scene(objs, {}, env)
    r = A.Renderer(s, st, A.GpuOptions(seed=SEED))
    task = A.render_tiled(s, st, A.GpuOptions(seed=SEED))
    for i, (img, sc) in tex.items():
        s.set_texture(i, img, scale=sc)
    r.render(0, spp)
    assert bits_equal(r.read_frame(spp), plain)
    r.close()
    assert bits_equal(task.await_(), plain)
    assert bits_equal(A.render_tiled(s, st, A.GpuOptions(seed=SEED)).await_(), textured)
    # a refused texture leaves the one that was bound; clearing every texture renders the plain scene
    with pytest.raises(A.RaymondError):
        s.set_texture(0, np.full((2, 2, 3), np.nan, dtype=np.float32))
    assert bits_equal(A.render_tiled(s, st, A.GpuOptions(seed=SEED)).await_(), textured)
    for i in tex:
        s.clear_texture(i)
    assert bits_equal(A.render_tiled(s, st, A.GpuOptions(seed=SEED)).await_(), plain)


def _texture_bytes(objs, tex):
    texels = sum(img.shape[0] * img.shape[1] for img, _ in tex.values()) * 16
    grids = {i for i in tex if objs[i][0] == "grid"}
    return texels + sum(np.asarray(objs[i][1]).shape[0] * 48 for i in grids)


@pytest.mark.parametrize("name", ["spheres", "dragon"])
def test_texels_and_uvs_count_in_upload_bytes(name):
    objs, tex, env, cam = scene_case(name)
    st = settings(cam, 1)
    _render(gpu_scene(objs, {}, env), st, 1)              # the pixel map of this layout is cached from here on
    _, _, with_tex = _render(gpu_scene(objs, tex, env), st, 1)
    _, _, without = _render(gpu_scene(objs, {}, env), st, 1)
    assert with_tex["upload_bytes"] - without["upload_bytes"] == _texture_bytes(objs, tex)


def test_tile_shares_match_one_share():
    objs, tex, env, _ = scene_case("dragon")
    st = settings(F.camera(96, 64), 6, spi=3)
    ref = A.render_tiled(gpu_scene(objs, tex, env), st, A.GpuOptions(seed=5)).await_()
    opt = A.GpuOptions(seed=5, device_list=[0, 0], partition=A.PARTITION_TILES)
    A.render_tiled(gpu_scene(objs, {}, env), st, opt).await_()      # the shares' pixel maps of this layout are cached from here on
    plain = A.render_tiled(gpu_scene(objs, {}, env), st, opt)
    plain.await_()
    many = A.render_tiled(gpu_scene(objs, tex, env), st, opt)
    assert bits_equal(many.await_(), ref)
    assert many.stats()["upload_bytes"] - plain.stats()["upload_bytes"] == 2 * _texture_bytes(objs, tex)


def test_adaptive_task_completes():
    objs, tex, env, _ = scene_case("spheres")
    st = settings(F.camera(96, 64), 32, spi=4)
    task = A.render_tiled(gpu_scene(objs, tex, env), st, A.GpuOptions(seed=3), adaptive=A.AdaptiveSettings(threshold=0.05, min_samples=4))
    frame = task.await_()
    assert np.isfinite(frame).all() and frame.max() > 0.1
    assert 0 < task.stats()["samples"] <= 96 * 64 * 32


def test_denoised_task_is_the_restatement():
    objs, tex, env, _ = scene_case("dragon")
    cam, spp = F.camera(96, 64), 8
    st = settings(cam, spp)
    task = A.render_tiled(gpu_scene(objs, tex, env), st, A.GpuOptions(seed=4, device_list=[0, 0], partition=A.PARTITION_SAMPLES), denoise=True)
    got = task.await_denoised()
    S = Q = alb = nrm = dep = None
    for g in range(2):
        r = A.Renderer(gpu_scene(objs, tex, env), st, A.GpuOptions(seed=4, world_size=2, rank=g, partition=A.PARTITION_SAMPLES,
                                                                    flags=A.FLAG_AOV | A.FLAG_MOMENTS))
        r.render(g, len(range(g, spp, 2)), 2)
        parts = (r.read_sums(), r.read_moments()) + r.read_aovs(1)
        r.close()
        S, Q, alb, nrm, dep = parts if S is None else tuple(a + b for a, b in zip((S, Q, alb, nrm, dep), parts))
    # the albedo guide is the textured colour: it differs from the plain scene's
    r = A.Renderer(gpu_scene(objs, {}, env), st, A.GpuOptions(seed=4, flags=A.FLAG_AOV))
    r.render(0, spp)
    assert not np.allclose(r.read_aovs(1)[0], alb)
    r.close()
    want = D.denoise(S, Q, alb / spp, nrm / spp, dep / spp, spp, **D.DEFAULTS).astype(np.float64)
    assert np.isfinite(got).all() and np.isfinite(want).all()
    assert (np.abs(got - want) <= 1e-4 * np.abs(want) + 1e-6).all()
