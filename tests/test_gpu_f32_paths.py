"""Path-for-path parity of the f32 shading mode (RM_PRECISION_F32_SHADING) with the oracle on the f32 mode's own draws.

lobe_f32 draws its three shading uniforms from 23 bits of one Philox block per bounce, so it is a different sample stream from
the f64 mode, and the statistical tests of test_gpu_precision / test_gpu_shading_space cannot see a wrong term that only some
paths reach.  The oracle's f32-draw stream (`draws="f32"`, checked on the CPU by test_oracle_f32_draws) hands the reference's
f64 integrator exactly those uniforms, so the only difference left between a GPU path and the oracle's is the f32 arithmetic of
the lobe: hits, normals, camera rays and lobe choices are the same on both sides until a rounding difference moves a
continuation ray across a silhouette or a triangle edge.

Per path, rel = max_c |g - o| / max(max_c |o|, 1e-3) (the measure of test_gpu_configs.compare_paths).  `compare_f32_paths`
holds the bulk to the size of f32 rounding through a few bounces (99th percentile), bounds the fraction of paths off by more
than 1e-3 (divergent paths, and GGX angles far beyond 2 pi at roughness >= 1.5), and holds those to the reference's range and to
no bias.  The bars are stated multiples of the values measured on a B200 (profiles/r7_f32_paths.log)."""
import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from shading_space import FIXTURES, SEED, SPP, tagged
from test_gpu_configs import LUMA, THREADS, gpu_sample_frames
from test_gpu_nonfinite import CAM as NF_CAM, SCENES as NF_SCENES, SEED as NF_SEED, SPP as NF_SPP
from test_gpu_shading_space import VALUE_SCALE
from util import oracle_scene, product_scene, settings

pytestmark = pytest.mark.gpu

F32 = A.PRECISION_F32_SHADING

# Bars, each a stated multiple of what the B200 measured (profiles/r7_f32_paths.log: 60 comparisons, 1.7 M paths).
# 99th percentile of rel: largest measured 1.4e-6 (metal_rough_3), 5e-7 typical; the bar is 7x that.  A wrong term in the
# weight moves it to 1e-2 and beyond.
P99_MAX = 1e-5
# Fraction of paths with rel > 1e-3: largest measured 2.0e-4 (5 of 24 576 paths of camera_portrait_48x128, divergent at a
# silhouette), 0 or 1 path elsewhere; the bar is 2x that.
GROSS_MAX = 4e-4
# Keep mode: paths whose NaN / +Inf / -Inf class differs in some channel, and |GPU - oracle| of nonfinite_samples and of rays.
# Measured: 0 on all 12 cases.  1e-4 of the paths (2 of 27 648) is left for an n.v or n.l whose sign f32 and f64 see
# differently within rounding of 0.
KEEP_DIFF_MAX = 1e-4
# The bias of the tail is tested when it has this many paths; a smaller tail is held by the range bound alone.
MIN_TAIL_FOR_BIAS = 10


def frames(objs, cam, spp, seed, limit, keep=False):
    """The GPU's f32-mode frames and the oracle's f32-draw frames, one per global sample, and both sides' counters."""
    g, gs = gpu_sample_frames(product_scene(objs), settings(cam, spp, bounce_limit=limit), spp, seed=seed, precision=F32,
                              flags=A.FLAG_KEEP_NONFINITE if keep else 0)
    osc = oracle_scene(objs)
    o, oc = [], {}
    for s in range(spp):
        f, c = O.render(osc, cam, 1, seed=seed, first_sample=s, bounce_limit=limit, drop_nonfinite=not keep, draws="f32",
                        worker_count=THREADS)
        o.append(f)
        oc = {k: oc.get(k, 0) + v for k, v in c.items()}
    return np.stack(g), gs, np.stack(o), oc


def path_rel(g, o):
    return np.abs(g - o).max(axis=-1) / np.maximum(np.abs(o).max(axis=-1), 1e-3)


def compare_f32_paths(g, o, what, signed=False, p99_max=P99_MAX, gross_max=GROSS_MAX):
    """Asserts, over finite paths g / o [..., 3] of the same stream:
      * the bulk: the 99th percentile of rel is at most `p99_max`;
      * the tails: at most `gross_max` of the paths have rel > 1e-3; every such GPU path is finite and within 2 max|o| of 0
        (non-negative unless `signed`), and, when there are MIN_TAIL_FOR_BIAS or more, their mean luminance difference is
        within 4 standard errors of 0;
      * the frame: mean luminance agrees to 0.2 %.
    Prints the measured table row.  Returns rel."""
    assert np.isfinite(g).all(), f"{what}: non-finite path value"
    rel = path_rel(g, o)
    p50, p99, p9999 = np.percentile(rel, [50, 99, 99.99])
    lit = (o != 0).any(axis=-1)             # paths that deliver radiance (most others are exact zeros on both sides)
    lit50 = np.median(rel[lit]) if lit.any() else 0.0
    f4, f3 = (rel > 1e-4).mean(), (rel > 1e-3).mean()
    print(f"f32 paths | {what:44s} | {rel.size:7d} paths | rel p50 {p50:.2g} p99 {p99:.2g} p99.99 {p9999:.2g} max {rel.max():.3g}"
          f" | p50 of {lit.mean():.0%} lit {lit50:.2g} | >1e-4 {f4:.3g} | >1e-3 {f3:.3g} ({int((rel > 1e-3).sum())})")
    assert p99 <= p99_max, f"{what}: 99th percentile of the per-path relative difference {p99:.3g} > {p99_max:g}"
    assert f3 <= gross_max, f"{what}: {f3:.3g} of the paths differ by more than 1e-3 relative (bar {gross_max:g})"
    gross = rel > 1e-3
    clip = (lambda x: x) if signed else (lambda x: np.clip(x, 0, 10))
    if gross.any():
        gd, od = g[gross], o[gross]
        bound = 2.0 * np.abs(o).max()
        lo = -bound if signed else 0.0
        assert gd.min() >= lo and gd.max() <= bound, f"{what}: a differing path value is outside [{lo}, {bound}]"
        dl = clip(gd) @ LUMA - clip(od) @ LUMA
        se = dl.std() / np.sqrt(dl.size)
        assert dl.size < MIN_TAIL_FOR_BIAS or abs(dl.mean()) <= 4.0 * se + 1e-12, f"{what}: differing paths are biased: mean {dl.mean()} vs standard error {se} over {dl.size} paths"
    gl, ol = (clip(g) @ LUMA).mean(), (clip(o) @ LUMA).mean()
    assert abs(gl - ol) <= 0.002 * abs(ol) + 1e-12, f"{what}: mean luminance {gl} vs {ol}"
    return rel


def check_drop(objs, cam, spp, seed, limit, what, scale=1.0, signed=False):
    g, gs, o, oc = frames(objs, cam, spp, seed, limit)
    compare_f32_paths(g * scale, o * scale, what, signed=signed)
    assert gs["samples"] == oc["samples"] == cam["width"] * cam["height"] * spp
    assert gs["nonfinite_samples"] <= oc["nonfinite"]           # D4: the GPU's own non-finite paths, a lower bound
    assert gs["rays"] <= oc["rays"]                             # the GPU stops paths whose throughput became exactly 0
    return g, o


def check_keep(objs, cam, spp, seed, limit, what):
    g, gs, o, oc = frames(objs, cam, spp, seed, limit, keep=True)
    classes = np.zeros(g.shape[:-1], dtype=bool)
    for f in (np.isnan, np.isposinf, np.isneginf):
        classes |= (f(g) != f(o)).any(axis=-1)
    dn, dr = abs(gs["nonfinite_samples"] - oc["nonfinite"]), abs(gs["rays"] - oc["rays"])
    print(f"f32 paths | {what:44s} | class differs on {int(classes.sum())} paths | non-finite {gs['nonfinite_samples']} vs"
          f" {oc['nonfinite']} | rays {gs['rays']} vs {oc['rays']}")
    allowance = KEEP_DIFF_MAX * classes.size
    assert classes.sum() <= allowance, f"{what}: {int(classes.sum())} paths differ in their NaN / Inf class"
    assert dn <= allowance, (gs["nonfinite_samples"], oc["nonfinite"])
    assert oc["nonfinite"] > 0
    assert dr <= allowance, (gs["rays"], oc["rays"])
    assert gs["samples"] == oc["samples"]
    fin = np.isfinite(o).all(axis=-1) & np.isfinite(g).all(axis=-1)
    compare_f32_paths(g[fin], o[fin], f"{what}, finite paths")


@pytest.mark.parametrize("name", list(FIXTURES))
def test_drop_mode_paths(name):
    """Every fixture of shading_space.py: roughness 0 to 3, colours outside [0, 1], non-unit normals, meshes, cameras, depth of
    field, two grids."""
    fx = FIXTURES[name]
    check_drop(fx.objs, fx.cam, SPP, SEED, fx.limit, f"{name} drop", scale=VALUE_SCALE.get(name, 1.0), signed="negative" in fx.tags)


BENCH_SCENES = {
    # the sizes of the f64 same-stream tests of test_gpu_render.py
    "ReflectiveSpheres 160x120x8": (F.reflective_spheres, F.camera(160, 120), 8, 3),
    "GoldDragon stand-in 160x90x4": (lambda: F.gold_dragon(F.dragon_standin(240, 60)), F.camera(160, 90), 4, 5),
    "DoF 120x80x4": (F.reflective_spheres, F.camera(120, 80, focal_length=2.5, aperture_radius=0.5), 4, 9),
}


@pytest.mark.parametrize("what", list(BENCH_SCENES))
def test_benchmark_scene_paths(what):
    objs, cam, spp, seed = BENCH_SCENES[what]
    check_drop(objs(), cam, spp, seed, 5, what)


@pytest.mark.parametrize("limit", [1, 2, 5, 8])
@pytest.mark.parametrize("name", ["metal_rough_1", "diffuse_rough_0.3"])
def test_bounce_limits(name, limit):
    fx = FIXTURES[name]
    g, o = check_drop(fx.objs, fx.cam, SPP, SEED, limit, f"{name} bounce_limit {limit}")
    if limit == 1:
        # only emission seen by camera rays counts, and nothing of it is f32
        assert np.array_equal(g, o)


KEEP_SCENES = {name: (FIXTURES[name].objs, FIXTURES[name].cam, SPP, SEED) for name in tagged("nonfinite")}
KEEP_SCENES.update({f"nan_normals_{k}": (v, NF_CAM, NF_SPP, NF_SEED) for k, v in NF_SCENES.items()})


@pytest.mark.parametrize("limit", [2, 5])
@pytest.mark.parametrize("name", list(KEEP_SCENES))
def test_keep_mode_paths(name, limit):
    """RM_FLAG_KEEP_NONFINITE past depth 1: the NaN / +Inf / -Inf class of every path and channel is the oracle's, except on
    the few paths where f32 and f64 disagree on the sign of an n.v or n.l within rounding of 0; rays are the oracle's up to the
    same paths, because the lobe choices are identical."""
    objs, cam, spp, seed = KEEP_SCENES[name]
    check_keep(objs, cam, spp, seed, limit, f"{name} keep bounce_limit {limit}")


@pytest.mark.parametrize("partition", [A.PARTITION_TILES, A.PARTITION_SAMPLES], ids=["tiles", "samples"])
@pytest.mark.parametrize("devices", [[0, 0], [0, 0, 0]], ids=["two", "three"])
def test_device_list_matches_one_device(partition, devices):
    """render_tiled in the f32 mode over repeated device ordinals gives the one-device frame: bit-identical when the shares own
    disjoint tiles, within 1e-12 when they own samples (the same samples summed in another association)."""
    objs, cam, spp = F.gold_dragon(F.dragon_standin(160, 40)), F.camera(160, 96), 7
    st = settings(cam, spp)
    ps = product_scene(objs)
    one = A.render_tiled(ps, st, A.GpuOptions(seed=5, precision=F32)).await_()
    many = A.render_tiled(ps, st, A.GpuOptions(seed=5, precision=F32, device_list=devices, partition=partition))
    got = many.await_()
    assert many.stats()["samples"] == 160 * 96 * spp
    if partition == A.PARTITION_TILES:
        assert np.array_equal(got, one)
    else:
        assert np.allclose(got, one, rtol=1e-12, atol=1e-12)
    f64 = A.render_tiled(ps, st, A.GpuOptions(seed=5)).await_()
    assert not np.array_equal(one, f64)          # the f32 mode is in effect
