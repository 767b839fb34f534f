"""Environment maps on the GPU (rm_scene_set_environment, include/raymond.h).

A ray that leaves the scene delivers T (*) L(d).  Nothing else changes: the draws, the hits and the ray counts are those of the
scene without a map, so a scene whose every ray is caught renders to the same bits with or without one, and open scenes are
held path for path against the oracle with a map (tests/env_oracle.cpp), whose trace looks the map up with glibc's atan2 / acos
on a miss."""
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

import denoise_ref as D
import env_oracle as EO
import env_ref
from test_gpu_configs import THREADS, compare_paths, gpu_sample_frames
from test_gpu_f32_paths import compare_f32_paths
from util import product_scene, settings

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SEED = 77
SKY = F.sky(128, 64, sun_radiance=40.0)
SKY_SCALE, SKY_ROT = 1.3, 0.7
PRECISIONS = [A.PRECISION_F64, A.PRECISION_F32_SHADING]
# Path-for-path bar of the f64 mode on open scenes: hits are bit-exact, so paths differ only by what CUDA's and glibc's
# atan2 / acos return.  Largest per-path relative difference measured on one B200 (1000 W power limit) over every case of
# test_open_scene_paths_f64: 4.6e-13 (open dragon, bounce limit >= 3; 5e-16 at limit 1, where only camera rays see the map).
# The bar is about 20x that.
PATH_REL_BAR = 1e-11


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def env_scene(objs, image=SKY, scale=SKY_SCALE, rotation=SKY_ROT):
    s = product_scene(objs)
    if image is not None:
        s.set_environment(image, scale, rotation)
    return s


def env_oracle(objs, image=SKY, scale=SKY_SCALE, rotation=SKY_ROT):
    return EO.Scene(objs, EO.Environment(image, scale, rotation))


def open_dragon():
    return F.open_dragon(F.dragon_standin(96, 24))


# ---------------------------------------------------------------------------- empty scene


@pytest.mark.parametrize("keep", [False, True], ids=["drop", "keep"])
@pytest.mark.parametrize("precision", PRECISIONS, ids=["f64", "f32"])
def test_constant_map_fills_the_frame(precision, keep):
    c, scale = np.array([0.3, 1.7, 42.5], dtype=np.float32), 0.37
    want = scale * c.astype(np.float64)
    cam = F.camera(40, 24)
    for limit in (0, 1, 2, 5):
        s = A.Scene()
        s.set_background(c, scale)
        frames, stats = gpu_sample_frames(s, settings(cam, 2, bounce_limit=limit), 2, SEED, precision=precision,
                                          flags=A.FLAG_KEEP_NONFINITE if keep else 0)
        for f in frames:
            if limit == 0:
                assert not f.any()
            else:
                assert np.array_equal(f, np.broadcast_to(want, f.shape)), limit
        assert stats["nonfinite_samples"] == 0


@pytest.mark.parametrize("cam", [F.camera(64, 40), F.camera(48, 32, fov_vert=120.0, position=(0.2, -0.1, 0.3)),
                                 F.camera(40, 30, focal_length=2.0, aperture_radius=0.4)], ids=["pinhole", "wide", "dof"])
def test_equirect_map_on_camera_rays(cam):
    spp = 3
    frames, _ = gpu_sample_frames(env_scene([]), settings(cam, spp), spp, SEED)
    worst = 0.0
    for s, f in enumerate(frames):
        rays = O.camera_rays(cam, SEED, s)
        want = env_ref.env_lookup(SKY, rays[:, 3:], SKY_SCALE, SKY_ROT).reshape(f.shape)
        rel = np.abs(f - want) / np.maximum(np.abs(want), 1e-300)
        worst = max(worst, rel.max())
    print(f"camera rays {cam['width']}x{cam['height']}: largest relative difference from env_ref {worst:.3g}")
    assert worst <= 1e-12


# ---------------------------------------------------------------------------- closed box: nothing changes


def _render(scene, st, spp, **opt):
    r = A.Renderer(scene, st, A.GpuOptions(seed=SEED, flags=A.FLAG_MOMENTS | opt.pop("flags", 0), **opt))
    r.render(0, spp)
    out = r.read_sums(), r.read_moments(), r.stats()
    r.close()
    return out


@pytest.mark.parametrize("keep", [False, True], ids=["drop", "keep"])
@pytest.mark.parametrize("precision", PRECISIONS, ids=["f64", "f32"])
@pytest.mark.parametrize("name", ["spheres", "dragon"])
def test_closed_box_ignores_the_map(name, precision, keep):
    objs = F.reflective_spheres() if name == "spheres" else F.gold_dragon(F.dragon_standin(160, 40))
    st, spp = settings(F.camera(96, 64), 6), 6
    flags = A.FLAG_KEEP_NONFINITE if keep else 0
    S0, Q0, s0 = _render(product_scene(objs), st, spp, precision=precision, flags=flags)
    S1, Q1, s1 = _render(env_scene(objs, scale=1e3), st, spp, precision=precision, flags=flags)
    assert s1["rays"] == s0["rays"] and s1["samples"] == s0["samples"]
    assert bits_equal(S1, S0) and bits_equal(Q1, Q0)
    if keep:
        assert s1["nonfinite_samples"] == s0["nonfinite_samples"]
    else:
        # a ray gets past the six planes only with a NaN origin (a NaN Heron normal, SURVEY A17) or when within 1e-6 of
        # parallel to two axes: a path whose throughput is already NaN then delivers NaN where it delivered an exact 0.  Such
        # paths are non-finite in the reference too, so the count stays at or below the oracle's.
        assert s1["nonfinite_samples"] >= s0["nonfinite_samples"]
        if s1["nonfinite_samples"] > s0["nonfinite_samples"]:
            _, oc = oracle_frames(env_oracle(objs, scale=1e3), F.camera(96, 64), spp, 5)
            assert s1["nonfinite_samples"] <= oc["nonfinite"], (s0["nonfinite_samples"], s1["nonfinite_samples"], oc["nonfinite"])


def test_texels_count_in_upload_bytes():
    objs, st = F.reflective_spheres(), settings(F.camera(32, 16), 1)
    _render(product_scene(objs), st, 1)              # the pixel map of this layout is cached from here on
    _, _, with_map = _render(env_scene(objs), st, 1)
    _, _, without = _render(product_scene(objs), st, 1)
    assert with_map["upload_bytes"] - without["upload_bytes"] == SKY.shape[0] * SKY.shape[1] * 16


# ---------------------------------------------------------------------------- open scenes, path for path


OPEN = {"spheres": (F.open_spheres, F.camera(64, 48)), "dragon": (open_dragon, F.camera(64, 40))}


def oracle_frames(osc, cam, spp, limit, keep=False, draws="f64"):
    o, oc = [], {}
    for s in range(spp):
        f, c = osc.render_sample(cam, s, seed=SEED, bounce_limit=limit, drop_nonfinite=not keep, draws=draws, threads=THREADS)
        o.append(f)
        oc = {k: oc.get(k, 0) + v for k, v in c.items()}
    return o, oc


@pytest.mark.parametrize("limit", [1, 2, 3, 4, 5])
@pytest.mark.parametrize("name", list(OPEN))
def test_open_scene_paths_f64(name, limit):
    mk, cam = OPEN[name]
    objs, spp = mk(), 3
    g, gs = gpu_sample_frames(env_scene(objs), settings(cam, spp, bounce_limit=limit), spp, SEED)
    o, oc = oracle_frames(env_oracle(objs), cam, spp, limit)
    g, o = np.stack(g), np.stack(o)
    rel = np.abs(g - o).max(axis=-1) / np.maximum(np.abs(o).max(axis=-1), 1e-3)
    print(f"env paths | {name} limit {limit} | largest relative difference {rel.max():.3g} | lit {(o != 0).any(axis=-1).mean():.0%}")
    assert (o > 0).any(axis=-1).mean() > 0.4          # the map lights the frame (at limit 1 only the sky is lit)
    compare_paths(list(g), list(o), f"{name} env limit {limit}", max_differing=0.0, max_gross=0.0)
    assert rel.max() <= PATH_REL_BAR
    assert gs["samples"] == oc["samples"] and gs["rays"] <= oc["rays"]


@pytest.mark.parametrize("limit", [2, 5])
@pytest.mark.parametrize("name", list(OPEN))
def test_open_scene_paths_keep(name, limit):
    mk, cam = OPEN[name]
    objs, spp = mk(), 2
    g, gs = gpu_sample_frames(env_scene(objs), settings(cam, spp, bounce_limit=limit), spp, SEED, flags=A.FLAG_KEEP_NONFINITE)
    o, oc = oracle_frames(env_oracle(objs), cam, spp, limit, keep=True)
    g, o = np.stack(g), np.stack(o)
    assert gs["rays"] == oc["rays"] and gs["nonfinite_samples"] == oc["nonfinite"]
    for f in (np.isnan, np.isposinf, np.isneginf):
        assert np.array_equal(f(g), f(o))
    fin = np.isfinite(o).all(axis=-1)
    rel = np.abs(g[fin] - o[fin]).max(axis=-1) / np.maximum(np.abs(o[fin]).max(axis=-1), 1e-3)
    print(f"env paths | {name} keep limit {limit} | largest relative difference {rel.max():.3g} | non-finite {gs['nonfinite_samples']}")
    assert rel.max() <= PATH_REL_BAR, rel.max()


@pytest.mark.parametrize("limit", [1, 3, 5])
@pytest.mark.parametrize("name", list(OPEN))
def test_open_scene_paths_f32(name, limit):
    mk, cam = OPEN[name]
    objs, spp = mk(), 3
    g, gs = gpu_sample_frames(env_scene(objs), settings(cam, spp, bounce_limit=limit), spp, SEED, precision=A.PRECISION_F32_SHADING)
    o, oc = oracle_frames(env_oracle(objs), cam, spp, limit, draws="f32")
    compare_f32_paths(np.stack(g), np.stack(o), f"{name} env limit {limit} f32")
    assert gs["samples"] == oc["samples"]


# ---------------------------------------------------------------------------- last depth


@pytest.mark.parametrize("precision", PRECISIONS, ids=["f64", "f32"])
@pytest.mark.parametrize("name", list(OPEN) + ["box"])
def test_full_last_bounce_is_the_same_frame(name, precision, monkeypatch):
    objs = F.reflective_spheres() if name == "box" else OPEN[name][0]()
    cam = OPEN["spheres"][1]
    out = []
    for full in (False, True):
        if full:
            monkeypatch.setenv("RM_FULL_LAST_BOUNCE", "1")
        else:
            monkeypatch.delenv("RM_FULL_LAST_BOUNCE", raising=False)
        for limit in (1, 3):
            r = A.Renderer(env_scene(objs), settings(cam, 4, bounce_limit=limit), A.GpuOptions(seed=SEED, precision=precision))
            r.render(0, 4)
            out.append((r.read_sums(), r.stats()))
            r.close()
    monkeypatch.delenv("RM_FULL_LAST_BOUNCE", raising=False)
    for (a, sa), (b, sb) in zip(out[:2], out[2:]):
        assert bits_equal(a, b)
        assert sa["rays"] == sb["rays"] and sa["nonfinite_samples"] == sb["nonfinite_samples"]


# ---------------------------------------------------------------------------- snapshots


def test_placements_keep_the_map_they_were_made_with():
    objs, st, spp = F.open_spheres(), settings(F.camera(48, 32), 3), 3
    want = A.render_tiled(env_scene(objs), st, A.GpuOptions(seed=SEED)).await_()
    s = env_scene(objs)
    r = A.Renderer(s, st, A.GpuOptions(seed=SEED))
    task = A.render_tiled(s, st, A.GpuOptions(seed=SEED))
    s.set_background((5.0, 0.0, 0.0))
    r.render(0, spp)
    assert bits_equal(r.read_frame(spp), want)
    r.close()
    assert bits_equal(task.await_(), want)
    # a refused map leaves the red background; clearing it renders the scene without a map
    with pytest.raises(A.RaymondError):
        s.set_environment(np.full((2, 2, 3), -1.0, dtype=np.float32))
    red = A.render_tiled(s, st, A.GpuOptions(seed=SEED)).await_()
    assert not bits_equal(red, want)
    s.clear_environment()
    plain = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=SEED)).await_()
    assert bits_equal(A.render_tiled(s, st, A.GpuOptions(seed=SEED)).await_(), plain)
    bad = product_scene(objs)
    with pytest.raises(A.RaymondError):
        bad.set_environment(np.full((2, 2, 3), np.nan, dtype=np.float32))
    assert bits_equal(A.render_tiled(bad, st, A.GpuOptions(seed=SEED)).await_(), plain)


# ---------------------------------------------------------------------------- tasks


@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]], ids=["gpus00", "gpus000"])
@pytest.mark.parametrize("partition", [A.PARTITION_SAMPLES, A.PARTITION_TILES], ids=["samples", "tiles"])
def test_task_shares_match_one_share(partition, devices):
    objs, st = open_dragon(), settings(F.camera(96, 64), 6, spi=3)
    ref = A.render_tiled(env_scene(objs), st, A.GpuOptions(seed=5)).await_()
    many = A.render_tiled(env_scene(objs), st, A.GpuOptions(seed=5, device_list=devices, partition=partition))
    got = many.await_()
    if partition == A.PARTITION_TILES:
        assert bits_equal(got, ref)
    else:
        assert np.allclose(got, ref, rtol=1e-12, atol=1e-12)
    assert many.stats()["upload_bytes"] >= len(devices) * SKY.shape[0] * SKY.shape[1] * 16
    assert ref.max() > 0.1


def test_adaptive_task_completes():
    objs, st = F.open_spheres(), settings(F.camera(96, 64), 32, spi=4)
    task = A.render_tiled(env_scene(objs), st, A.GpuOptions(seed=3), adaptive=A.AdaptiveSettings(threshold=0.05, min_samples=4))
    frame = task.await_()
    assert np.isfinite(frame).all() and frame.max() > 0.1
    assert 0 < task.stats()["samples"] <= 96 * 64 * 32


def test_denoised_task_is_the_restatement():
    objs, cam, spp = F.open_spheres(), F.camera(96, 64), 8
    st = settings(cam, spp)
    task = A.render_tiled(env_scene(objs), st, A.GpuOptions(seed=4, device_list=[0, 0], partition=A.PARTITION_SAMPLES), denoise=True)
    got = task.await_denoised()
    S = Q = alb = nrm = dep = None
    for g in range(2):
        r = A.Renderer(env_scene(objs), st, A.GpuOptions(seed=4, world_size=2, rank=g, partition=A.PARTITION_SAMPLES,
                                                          flags=A.FLAG_AOV | A.FLAG_MOMENTS))
        r.render(g, len(range(g, spp, 2)), 2)
        parts = (r.read_sums(), r.read_moments()) + r.read_aovs(1)
        r.close()
        S, Q, alb, nrm, dep = parts if S is None else tuple(a + b for a, b in zip((S, Q, alb, nrm, dep), parts))
    want = D.denoise(S, Q, alb / spp, nrm / spp, dep / spp, spp, **D.DEFAULTS).astype(np.float64)
    assert np.isfinite(got).all() and np.isfinite(want).all()
    assert (np.abs(got - want) <= 1e-4 * np.abs(want) + 1e-6).all()
    assert np.abs(got - S / spp).max() > 1e-3


# ---------------------------------------------------------------------------- cli_old


def test_cli_old_open_env(tmp_path):
    from PIL import Image
    exe = str(tmp_path / "cli_old")
    lib_dir = os.path.join(ROOT, "raymond_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "cli_old.cpp"),
                    "-L", lib_dir, "-lraymond_cuda", f"-Wl,-rpath,{lib_dir}", "-o", exe], check=True)
    mesh = F.dragon_standin(160, 40)
    ply, hdr, out = str(tmp_path / "dragon.ply"), str(tmp_path / "sky.hdr"), str(tmp_path / "output.png")
    F.write_ply(ply, mesh)
    F.write_hdr(hdr, SKY)
    subprocess.run([exe, "--mesh", ply, "--out", out, "--width", "160", "--height", "90", "--spp", "6", "--seed", "11", "--open",
                    "--env", hdr, "--env-scale", "0.8", "--env-rotation", "1.5"], check=True, capture_output=True, text=True)
    got = np.asarray(Image.open(out))
    m = A.Mesh.load_ply(ply)
    m.bake_transform(F.DRAGON_TRANSLATE)
    scene = A.Scene()
    scene.push_sphere(*F.RED_SPHERE[1:3], A.Material.from_fixture(F.RED_SPHERE[3]))
    scene.push_grid(A.AccGrid.build_from_mesh(m), A.Material.from_fixture(F.DRAGON_MATERIAL))
    scene.push_plane(F.FLOOR[1], F.FLOOR[2], A.Material.from_fixture(F.FLOOR[3]))
    scene.set_environment(A.load_hdr(hdr), 0.8, 1.5)
    frame = A.render_tiled(scene, settings(F.camera(160, 90), 6), A.GpuOptions(seed=11)).await_()
    assert np.array_equal(got, A.tonemap(frame))
    assert got.shape == (90, 160, 3) and got.mean() > 50
