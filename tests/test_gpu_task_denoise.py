"""rm_render_tiled_denoised: the feature-guided filter on the task path, sliced by rows across the shares of a task.

One share is rm_renderer_read_denoised bit for bit.  Under the tile partition every pixel's sums come from one share plus zeros, so
any number of shares gives the one-share frame bit for bit.  Under the sample partition the shares' own sums, rebuilt in numpy in
share order and filtered by the float32 restatement (tests/denoise_ref.py), are the reference.  The raw path (messages, await)
is the plain render's."""
import os
import subprocess

import numpy as np
import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

import denoise_ref as D
from conftest import cuda_device_count
from test_gpu_nonfinite import SCENES as NONFINITE_SCENES
from util import product_scene, settings

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

FLAGS = A.FLAG_AOV | A.FLAG_MOMENTS
TEN = A.DenoiseSettings(10, 8.0, 2.0, 1.0, 1.0)


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def ref_kwargs(denoise):
    if denoise is True or denoise is None:
        return D.DEFAULTS
    return dict(iterations=denoise.iterations, sigma_color=denoise.sigma_color, sigma_normal=denoise.sigma_normal,
                sigma_albedo=denoise.sigma_albedo, sigma_depth=denoise.sigma_depth)


def dragon():
    return F.gold_dragon(F.dragon_standin(160, 40))


@pytest.mark.parametrize("denoise", [True, TEN], ids=["defaults", "ten"])
@pytest.mark.parametrize("name", ["spheres", "dragon"])
def test_one_device_is_read_denoised(name, denoise):
    objs = F.reflective_spheres() if name == "spheres" else dragon()
    cam, spp = F.camera(128, 96), 8
    st = settings(cam, spp)
    task = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=7), denoise=denoise)
    got = task.await_denoised()
    r = A.Renderer(product_scene(objs), st, A.GpuOptions(seed=7, flags=FLAGS))
    r.render(0, spp)
    want = r.read_denoised(spp, None if denoise is True else denoise)
    assert bits_equal(task.await_(), r.read_frame(spp))
    r.close()
    assert bits_equal(got, want)
    assert np.isfinite(got).all() and got.max() > 0.1


def device_lists():
    lists = [[0, 0], [0, 0, 0]]
    n = cuda_device_count()
    if n >= 2:
        lists += [[0, 1]]
    if n >= 4:
        lists += [[0, 1, 2, 3]]
    return lists


@pytest.mark.parametrize("denoise", [True, A.DenoiseSettings(5, 2.0, 0.3, 0.4, 0.5), TEN], ids=["defaults", "five", "ten"])
@pytest.mark.parametrize("devices", device_lists(), ids=lambda d: "gpus" + "".join(map(str, d)))
def test_tile_partition_is_the_one_share_frame(devices, denoise):
    objs, st = dragon(), settings(F.camera(160, 96), 6, spi=3)
    one = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=5), denoise=denoise).await_denoised()
    many = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=5, device_list=devices, partition=A.PARTITION_TILES), denoise=denoise)
    assert bits_equal(many.await_denoised(), one)


def share_sums(objs, st, spp, seed, G, flags, shares=None):
    """S, Q and the raw feature sums of the task's shares (world_size G, rank g: global samples g, g + G, ...) added in share
    order, as the task adds them.  `shares`: how many of them render anything (the rest hold zeros, which add exactly)."""
    S = Q = alb = nrm = dep = None
    for g in range(G if shares is None else shares):
        r = A.Renderer(product_scene(objs), st, A.GpuOptions(seed=seed, world_size=G, rank=g, partition=A.PARTITION_SAMPLES, flags=flags))
        count = len(range(g, spp, G))
        if count:
            r.render(g, count, G)
        parts = (r.read_sums(), r.read_moments()) + r.read_aovs(1)       # read_aovs(1): the raw sums
        r.close()
        if S is None:
            S, Q, alb, nrm, dep = parts
        else:
            S, Q, alb, nrm, dep = (a + b for a, b in zip((S, Q, alb, nrm, dep), parts))
    return S, Q, alb, nrm, dep


def assert_matches_restatement(got, sums, spp, denoise):
    S, Q, alb, nrm, dep = sums
    want = D.denoise(S, Q, alb / spp, nrm / spp, dep / spp, spp, **ref_kwargs(denoise)).astype(np.float64)
    for f in (np.isnan, np.isposinf, np.isneginf):
        assert np.array_equal(f(got), f(want)), f.__name__
    fin = np.isfinite(want)
    err = np.abs(got[fin] - want[fin])
    print(f"largest difference {err.max(initial=0.0):.3g} absolute")
    assert (err <= 1e-4 * np.abs(want[fin]) + 1e-6).all()
    assert np.abs(got - S / spp)[fin].max() > 1e-3        # the filter did something


SAMPLE_CASES = {
    # name: (scene, camera, spp, seed, device list, settings, extra flags)
    "spheres_2": (F.reflective_spheres, F.camera(96, 64), 8, 3, [0, 0], True, 0),
    "dragon_3_ten": (dragon, F.camera(160, 96), 6, 4, [0, 0, 0], TEN, 0),
    "nonfinite_box_2": (lambda: NONFINITE_SCENES["box"], F.camera(64, 48), 8, 3, [0, 0], A.DenoiseSettings(3, 1.5, 0.3, 0.4, 0.05),
                        A.FLAG_KEEP_NONFINITE),
    # 8 rows a share: the taps of passes 2..4 (up to 32 rows away) reach across several slices
    "rows24_shares3_five": (F.reflective_spheres, F.camera(64, 24), 8, 9, [0, 0, 0], A.DenoiseSettings(5, 2.0, 0.3, 0.4, 0.5), 0),
    # fewer rows than shares: one share owns no row at all
    "rows2_shares3": (F.reflective_spheres, F.camera(64, 2), 8, 2, [0, 0, 0], A.DenoiseSettings(3, 2.0, 0.3, 0.4, 0.5), 0),
}
if cuda_device_count() >= 2:
    SAMPLE_CASES["spheres_gpus01"] = (F.reflective_spheres, F.camera(96, 64), 8, 3, [0, 1], TEN, 0)


@pytest.mark.parametrize("name", list(SAMPLE_CASES))
def test_sample_partition_is_the_restatement_of_the_summed_sums(name):
    scene, cam, spp, seed, devices, denoise, flags = SAMPLE_CASES[name]
    objs, st = scene(), settings(cam, spp)
    task = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=seed, device_list=devices, partition=A.PARTITION_SAMPLES, flags=flags),
                          denoise=denoise)
    got = task.await_denoised()
    sums = share_sums(objs, st, spp, seed, len(devices), FLAGS | flags)
    if name.startswith("nonfinite"):
        assert np.isnan(got).any() and np.isfinite(got).mean() > 0.5
    assert_matches_restatement(got, sums, spp, denoise)


def test_staged_fallback_with_more_shares_than_one_kernel_takes():
    objs, cam, spp, seed = F.reflective_spheres(), F.camera(64, 48), 6, 8
    st = settings(cam, spp)
    devices = [0] * 65
    task = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=seed, device_list=devices), denoise=TEN)
    got = task.await_denoised()
    assert_matches_restatement(got, share_sums(objs, st, spp, seed, len(devices), FLAGS, shares=spp), spp, TEN)


def messages(task):
    out = []
    while (m := task.poll()) is not None:
        out.append(m)
    return out


@pytest.mark.parametrize("partition", [A.PARTITION_SAMPLES, A.PARTITION_TILES], ids=["samples", "tiles"])
@pytest.mark.parametrize("devices", [None, [0, 0], [0, 0, 0]], ids=["one", "gpus00", "gpus000"])
def test_the_raw_path_is_the_plain_render(devices, partition):
    objs, st, denoise = dragon(), settings(F.camera(160, 96), 7, spi=3), A.DenoiseSettings(2)
    opts = A.GpuOptions(seed=6, device_list=devices, partition=partition)
    plain = A.render_tiled(product_scene(objs), st, opts)
    den = A.render_tiled(product_scene(objs), st, opts, denoise=denoise)
    s_plain, s_den = plain.stats(), den.stats()
    assert den.finished()
    assert s_den["samples"] == s_plain["samples"] == 160 * 96 * 7
    shares = len(devices) if devices else 1
    assert s_den["kernel_launches"] >= s_plain["kernel_launches"] + (1 + denoise.iterations) * shares
    filtered = den.await_denoised()        # does not consume the messages
    m_plain, m_den = messages(plain), messages(den)
    assert [(m.kind, m.tile.sample_count, m.tile.left, m.tile.top, m.tile.width, m.tile.height) for m in m_den] == \
           [(m.kind, m.tile.sample_count, m.tile.left, m.tile.top, m.tile.width, m.tile.height) for m in m_plain]
    assert all(bits_equal(a.tile.data, b.tile.data) for a, b in zip(m_den, m_plain))
    assert {m.tile.sample_count for m in m_den if m.kind == "TileProgressed"} == {3, 6}
    # await_() takes the messages, so it reads a second pair of tasks; the second denoised task filters the same frame
    again = A.render_tiled(product_scene(objs), st, opts, denoise=denoise)
    assert bits_equal(again.await_(), A.render_tiled(product_scene(objs), st, opts).await_())
    assert bits_equal(again.await_denoised(), filtered)
    assert bits_equal(again.await_denoised(), filtered)      # the filtered frame stays readable


def test_await_denoised_needs_a_denoised_task():
    task = A.render_tiled(product_scene(F.reflective_spheres()), settings(F.camera(32, 24), 2), A.GpuOptions())
    with pytest.raises(A.RaymondError) as e:
        task.await_denoised()
    assert e.value.status == A.RM_ERR_STATE
    task.await_()


def cli_devices():
    return [1, 2] if cuda_device_count() >= 2 else [1]


@pytest.mark.parametrize("gpus", cli_devices())
def test_cli_old_twin_writes_the_filtered_frame(tmp_path, gpus):
    from PIL import Image
    exe = str(tmp_path / "cli_old")
    lib_dir = os.path.join(ROOT, "raymond_b200")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "examples", "cli_old.cpp"),
                    "-L", lib_dir, "-lraymond_cuda", f"-Wl,-rpath,{lib_dir}", "-o", exe], check=True)
    out = str(tmp_path / "denoised.png")
    res = subprocess.run([exe, "--out", out, "--width", "160", "--height", "90", "--spp", "6", "--seed", "11", "--gpus", str(gpus),
                          "--denoise", "1"], check=True, capture_output=True, text=True)
    assert "Total render time" in res.stdout
    got = np.asarray(Image.open(out))
    scene = product_scene(F.reflective_spheres())     # cli_old without --mesh
    task = A.render_tiled(scene, settings(F.camera(160, 90), 6), A.GpuOptions(seed=11, device_count=gpus), denoise=A.DenoiseSettings(1))
    frame = task.await_denoised()
    assert np.array_equal(got, A.tonemap(frame))
    assert not np.array_equal(got, A.tonemap(task.await_()))
