"""Path-for-path parity with the oracle on the materials and cameras of shading_space.py: roughness 0 to 3, colours outside
[0, 1], emitters other than the ceiling, non-unit plane normals, off-origin and wide / narrow cameras, odd frame shapes, depth
of field and two grids.

lobe_f64 does not repeat the reference's trace operation for operation (a re-associated throughput product, sqrt closed forms
for cos / sin(acos(x)), pow5, div0, a shared lobe frame, the D5 stop); every fixture here holds those choices to the same
bars as the benchmark scenes: in drop mode no path may differ beyond 1e-9 relative, in keep mode the NaN / +Inf / -Inf
classes are equal per path and channel.  The f32 shading mode is held to test_gpu_precision's estimator checks here, and
path for path on every fixture by test_gpu_f32_paths.py, against the oracle given the f32 mode's own draws."""
import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from shading_space import FIXTURES, SEED, SPP, tagged
from test_gpu_configs import LUMA, THREADS, compare_paths, gpu_sample_frames
from test_gpu_last_bounce import assert_same_bits, render as last_bounce_render
from test_gpu_nonfinite import assert_nonfinite_classes_equal
from util import oracle_scene, product_scene, settings

pytestmark = pytest.mark.gpu

# compare_paths' relative measure has an absolute floor of 1e-3 per path; with an emitter of 1e-3 the path values are ~1e-4,
# so that fixture is compared at 1000 times its values (path values scale with the emission, the relative measure does not)
VALUE_SCALE = {"emitter_1e-3": 1e3}


def compare_signed_paths(gpu_frames, ora_frames, what, max_differing=1e-5, max_gross=2e-6):
    """compare_paths for fixtures whose paths may be negative (colours outside [0, 1]): the same differing-path bars, a
    differing GPU path bounded by |g| <= 2 max|o|, and no bias in the unclipped luminance."""
    g, o = np.stack(gpu_frames), np.stack(ora_frames)
    assert np.isfinite(g).all(), f"{what}: non-finite path value"
    rel = np.abs(g - o).max(axis=-1) / np.maximum(np.abs(o).max(axis=-1), 1e-3)
    differing, gross = rel > 1e-9, rel > 1e-3
    report = f"{what}: {int(differing.sum())} of {differing.size} paths differ = {differing.mean():.5%} (by more than 1e-3: {int(gross.sum())}; largest relative difference {rel.max():.3g})"
    print(report)
    assert differing.mean() <= max_differing and gross.mean() <= max_gross, report
    gd, od = g[differing], o[differing]
    if gd.size:
        bound = 2.0 * np.abs(o).max()
        assert np.abs(gd).max() <= bound, f"{what}: a differing path value {np.abs(gd).max()} is outside [-{bound}, {bound}]"
        dl = gd @ LUMA - od @ LUMA
        se = dl.std() / np.sqrt(dl.size)
        assert abs(dl.mean()) <= 4.0 * se + 1e-12, f"{what}: differing paths are biased: mean {dl.mean()} vs standard error {se}"
    gl, ol = (g @ LUMA).mean(), (o @ LUMA).mean()
    assert abs(gl - ol) <= 0.002 * abs(ol) + 1e-12, f"{what}: mean luminance {gl} vs {ol}"


def compare(name, g, o, what):
    s = VALUE_SCALE.get(name, 1.0)
    g, o = np.asarray(g) * s, np.asarray(o) * s
    (compare_signed_paths if "negative" in FIXTURES[name].tags else compare_paths)(g, o, what)


def oracle_frames(name, keep):
    fx = FIXTURES[name]
    osc = oracle_scene(fx.objs)
    frames = [O.render(osc, fx.cam, 1, seed=SEED, first_sample=s, bounce_limit=fx.limit, drop_nonfinite=not keep, worker_count=THREADS)[0]
              for s in range(SPP)]
    _, cnt = O.render(osc, fx.cam, SPP, seed=SEED, bounce_limit=fx.limit, drop_nonfinite=not keep, worker_count=THREADS)
    return frames, cnt


def gpu_frames(name, flags=0):
    fx = FIXTURES[name]
    return gpu_sample_frames(product_scene(fx.objs), settings(fx.cam, SPP, bounce_limit=fx.limit), SPP, seed=SEED, flags=flags)


@pytest.mark.parametrize("name", list(FIXTURES))
def test_drop_mode_paths(name):
    g, gs = gpu_frames(name)
    o, oc = oracle_frames(name, keep=False)
    compare(name, g, o, f"{name} drop")
    assert gs["samples"] == oc["samples"]
    assert gs["nonfinite_samples"] <= oc["nonfinite"]          # D4: the GPU's own non-finite paths, a lower bound


@pytest.mark.parametrize("name", list(FIXTURES))
def test_keep_mode_paths(name):
    g, gs = gpu_frames(name, flags=A.FLAG_KEEP_NONFINITE)
    o, oc = oracle_frames(name, keep=True)
    g, o = np.stack(g), np.stack(o)
    assert_nonfinite_classes_equal(g, o, f"{name} keep")
    finite = np.isfinite(o).all(axis=-1)
    assert np.isfinite(g[finite]).all()
    compare(name, g[finite], o[finite], f"{name} keep, finite paths")
    assert gs["nonfinite_samples"] == oc["nonfinite"]
    assert gs["rays"] == oc["rays"]
    if "nonfinite" in FIXTURES[name].tags:
        assert oc["nonfinite"] > 0


@pytest.mark.parametrize("limit", [1, 2, 5])
@pytest.mark.parametrize("name", tagged("last_bounce"))
def test_last_bounce_shortcut_is_bit_identical(name, limit, monkeypatch):
    fx = FIXTURES[name]
    g, gs, gst = last_bounce_render(fx.objs, fx.cam, SPP, limit, monkeypatch, False)
    f, fs, fst = last_bounce_render(fx.objs, fx.cam, SPP, limit, monkeypatch, True)
    assert_same_bits(g, f, f"{name} bounce_limit {limit}")
    assert gs["rays"] == fs["rays"] and gs["nonfinite_samples"] == fs["nonfinite_samples"]
    assert gst["grid_rays"][:limit] == fst["grid_rays"][:limit]
    assert 0 < gst["grid_rays"][limit] <= fst["grid_rays"][limit]
    print(f"{name} bounce_limit {limit}: last-stage grid rays {fst['grid_rays'][limit]} -> {gst['grid_rays'][limit]}")


def f32_render(ps, cam, spp, precision, seed, limit):
    r = A.Renderer(ps, settings(cam, spp, bounce_limit=limit), A.GpuOptions(seed=seed, precision=precision))
    r.render(0, spp)
    out, stats = r.read_sums() / spp, r.stats()
    r.close()
    return out, stats


@pytest.mark.parametrize("name", tagged("f32"))
def test_f32_shading_is_the_same_estimator(name):
    """test_gpu_precision's checks at 128x96 x 64 spp: the f32 image is within 1.15 times the noise floor of two f64 seeds, the
    mean luminance agrees, rays per path agree to 0.5 %, and the fraction of non-finite samples is the f64 mode's within 4
    standard errors of the difference of two binomial proportions (plus 8 samples, for fixtures that have almost none)."""
    fx = FIXTURES[name]
    ps, cam, spp = product_scene(fx.objs), F.camera(128, 96), 64
    a, sa = f32_render(ps, cam, spp, A.PRECISION_F64, 5, fx.limit)
    b, sb = f32_render(ps, cam, spp, A.PRECISION_F32_SHADING, 5, fx.limit)
    c, _ = f32_render(ps, cam, spp, A.PRECISION_F64, 6, fx.limit)
    assert sa["samples"] == sb["samples"]
    n = sa["samples"]
    pa, pb = sa["nonfinite_samples"] / n, sb["nonfinite_samples"] / n
    p = (pa + pb) / 2
    se = np.sqrt(2.0 * p * (1.0 - p) / n)
    print(f"{name} f32: non-finite samples {sb['nonfinite_samples']} vs f64 {sa['nonfinite_samples']} of {n}")
    assert abs(pa - pb) <= 4.0 * se + 8.0 / n, (sa["nonfinite_samples"], sb["nonfinite_samples"], n)
    if "nonfinite" in fx.tags:
        assert sa["nonfinite_samples"] > 0
    clip = lambda x: np.clip(x, 0, 10)
    la, lb, lc = clip(a) @ LUMA, clip(b) @ LUMA, clip(c) @ LUMA
    same, floor = np.sqrt(((la - lb) ** 2).mean()), np.sqrt(((la - lc) ** 2).mean())
    assert same <= 1.15 * floor, (same, floor)
    se = np.sqrt(la.var() / la.size + lb.var() / lb.size)
    assert abs(la.mean() - lb.mean()) <= max(5e-3 * la.mean(), 3 * se), (la.mean(), lb.mean(), se)
    assert abs(sa["rays"] - sb["rays"]) <= 0.005 * sa["rays"]
