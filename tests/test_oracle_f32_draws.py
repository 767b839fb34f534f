"""The oracle's f32-draw stream (CPU): the same-stream reference of the product's f32 shading mode (RM_PRECISION_F32_SHADING).

That mode makes one Philox call per bounce and builds its three shading uniforms from 23 bits of words 0, 2 and 1
(lobe_f32 in rm_kernels.cuh).  The oracle's `draws="f32"` gives its f64 integrator exactly those uniforms, so that the GPU's
f32 mode can be compared with it path for path (test_gpu_f32_paths.py).  Checked here against an independent numpy Philox."""
import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import fixtures as F

from shading_space import FIXTURES
from util import oracle_scene

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF


def philox4x32_10(seed: np.ndarray, c: np.ndarray) -> np.ndarray:
    """Philox4x32-10 (Salmon et al., SC'11) on N counters c[N, 4] under N 64-bit keys; returns the words [N, 4]."""
    c = c.astype(np.uint64)
    k0, k1 = seed.astype(np.uint64) & MASK, seed.astype(np.uint64) >> np.uint64(32)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c[:, 0], np.uint64(M1) * c[:, 2]
        c = np.stack([(p1 >> np.uint64(32)) ^ c[:, 1] ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ c[:, 3] ^ k1, p0 & MASK], axis=1)
        k0, k1 = (k0 + np.uint64(W0)) & MASK, (k1 + np.uint64(W1)) & MASK
    return c


def u23(x: np.ndarray) -> np.ndarray:
    return ((x >> np.uint64(9)).astype(np.float64) + 0.5) * 2.0 ** -23


def u52(hi: np.ndarray, lo: np.ndarray) -> np.ndarray:
    return (((hi << np.uint64(32)) | lo) >> np.uint64(12)).astype(np.float64) * 2.0 ** -52 + 2.0 ** -53


def tuples(n: int = 300) -> np.ndarray:
    """(seed, pixel, sample, depth) spread over the whole range of each counter word, plus a few corners."""
    rng = np.random.default_rng(20261021)
    t = np.stack([rng.integers(0, 2 ** 64, n, dtype=np.uint64), rng.integers(0, 2 ** 32, n, dtype=np.uint64),
                  rng.integers(0, 2 ** 32, n, dtype=np.uint64), rng.integers(1, 9, n, dtype=np.uint64)], axis=1)
    corners = np.array([[0, 0, 0, 1], [2 ** 64 - 1, 2 ** 32 - 1, 2 ** 32 - 1, 2 ** 32 - 1], [7, 5, 3, 1], [7, 5, 3, 8]], dtype=np.uint64)
    return np.concatenate([t, corners])


def test_f32_draws_are_the_f32_shading_mode_uniforms():
    """Draws 0, 1, 2 of depth >= 1 are u23 of words 0, 2, 1 of Philox(seed; pixel, sample, depth, 0), bit for bit."""
    t = tuples()
    w = philox4x32_10(t[:, 0], np.concatenate([t[:, 1:], np.zeros((len(t), 1), np.uint64)], axis=1))
    want = np.stack([u23(w[:, 0]), u23(w[:, 2]), u23(w[:, 1])], axis=1)
    got = np.array([[O.rng_draw(int(s), int(p), int(q), int(d), i, draws="f32") for i in range(3)] for s, p, q, d in t])
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    assert ((got > 0) & (got < 1)).all()
    # a draw of the f32 stream is a multiple of 2^-24 (23 bits and the half step), which no f64 draw is
    assert np.array_equal(got * 2 ** 24, np.round(got * 2 ** 24))
    # the f64 stream of the same tuples still matches the numpy Philox (draws 0 and 1 of block 0, draw 2 of block 1)
    w1 = philox4x32_10(t[:, 0], np.concatenate([t[:, 1:], np.ones((len(t), 1), np.uint64)], axis=1))
    want64 = np.stack([u52(w[:, 0], w[:, 1]), u52(w[:, 2], w[:, 3]), u52(w1[:, 0], w1[:, 1])], axis=1)
    got64 = np.array([[O.rng_draw(int(s), int(p), int(q), int(d), i) for i in range(3)] for s, p, q, d in t])
    assert np.array_equal(got64.view(np.uint64), want64.view(np.uint64))


def test_camera_draws_are_the_f64_ones():
    """Depth 0 (the pixel jitter and every round of the aperture rejection loop) is the same stream in both modes."""
    for s, p, q, _ in tuples(60):
        for i in range(8):
            a = O.rng_draw(int(s), int(p), int(q), 0, i)
            assert O.rng_draw(int(s), int(p), int(q), 0, i, draws="f32") == a


def render(fx, limit, draws, keep=False):
    return O.render(oracle_scene(fx.objs), fx.cam, 2, seed=7, bounce_limit=limit, drop_nonfinite=not keep, draws=draws)


@pytest.mark.parametrize("name", ["metal_rough_0.3", "diffuse_rough_0.3", "dof_aperture_2", "mesh_metal_rough_0"])
def test_bounce_limit_1_is_the_f64_render(name):
    """At bounce_limit 1 only emission seen by camera rays counts: the shading draws never reach the frame, so the two
    streams give the same sums bit for bit (NaN samples included in keep mode).  From limit 2 on they differ."""
    fx = FIXTURES[name]
    for keep in (False, True):
        a, ca = render(fx, 1, "f64", keep)
        b, cb = render(fx, 1, "f32", keep)
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64)) and ca == cb
    a, _ = render(fx, 2, "f64")
    b, _ = render(fx, 2, "f32")
    assert not np.array_equal(a, b)


def test_lobe_choices_are_exact_in_both_precisions():
    """The lobe choice `r < prob_d` is the same in f32 and f64: a u23 draw is exact in f32, and prob_d is 0.5 (Diffuse) or 0
    (Metal), exact in both.  So the GPU's f32 mode and the f32-draw oracle choose the same lobe on every path whose hits agree."""
    t = tuples()
    r = np.array([O.rng_draw(int(s), int(p), int(q), int(d), 0, draws="f32") for s, p, q, d in t])
    assert np.array_equal(r.astype(np.float32).astype(np.float64), r)
    for prob_d in (0.5, 0.0):
        assert np.array_equal(r < prob_d, r.astype(np.float32) < np.float32(prob_d))
    assert 0 < (r < 0.5).sum() < len(r)


def test_f32_draws_render_the_same_estimator():
    """An f32-draw render is another sample of the reference's estimator: its mean luminance over the ReflectiveSpheres frame
    is the f64-draw render's within the noise of the two streams."""
    objs, cam, spp = F.reflective_spheres(), F.camera(48, 36), 16
    osc = oracle_scene(objs)
    luma = np.array([0.2126, 0.7152, 0.0722])
    la = np.clip(O.render(osc, cam, spp, seed=3)[0] / spp, 0, 10) @ luma
    lb = np.clip(O.render(osc, cam, spp, seed=3, draws="f32")[0] / spp, 0, 10) @ luma
    se = np.sqrt(la.var() / la.size + lb.var() / lb.size)
    assert abs(la.mean() - lb.mean()) <= max(0.02 * la.mean(), 4 * se), (la.mean(), lb.mean(), se)
