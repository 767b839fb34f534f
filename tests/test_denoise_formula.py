"""The a-trous denoiser's formula (include/raymond.h, rm_renderer_read_denoised) on synthetic inputs, through the numpy float32
restatement the GPU test compares the library with (tests/denoise_ref.py).  No GPU."""
import numpy as np

import denoise_ref as D

F = np.float32


def inputs(H=12, W=16, n=16, colour=0.5, var=0.01, seed=0):
    """Sums as the renderer keeps them: S, Q (per-channel sample variance `var`), and feature means of a flat grey wall."""
    S = np.full((H, W, 3), colour * n)
    Q = S * colour + var * (n - 1)
    albedo = np.full((H, W, 3), 0.5)
    normal = np.tile(np.array([0.0, 0.0, -1.0]), (H, W, 1))
    depth = np.full((H, W), 3.0)
    return S, Q, albedo, normal, depth, n


def scalar_denoise(S, Q, albedo, normal, depth, n, iterations, sc, sn, sa, sz):
    """The same filter one pixel and one tap at a time, as written in the header."""
    c, v, a, m, z = D.pack(S, Q, albedo, normal, depth, n)
    H, W = v.shape
    for it in range(iterations):
        step = 1 << it
        c2, v2 = c.copy(), v.copy()
        for y in range(H):
            for x in range(W):
                if not (np.isfinite(c[y, x]).all() and np.isfinite(v[y, x]) and np.isfinite(a[y, x]).all() and np.isfinite(m[y, x]).all()
                        and np.isfinite(z[y, x])):
                    continue
                rc = F(1) / (F(sc) * np.sqrt(v[y, x]) + F(1e-6))
                rn = F(1) / (F(sn) * F(sn))
                ra = F(1) / (F(sa) * F(sa))
                rz = F(1) / (F(sz) * F(step) * z[y, x] + F(1e-6))
                sw, acc, sv = F(0), np.zeros(3, F), F(0)
                for dy in range(-2, 3):
                    for dx in range(-2, 3):
                        qy, qx = y + dy * step, x + dx * step
                        if not (0 <= qy < H and 0 <= qx < W):
                            continue
                        if not (np.isfinite(c[qy, qx]).all() and np.isfinite(v[qy, qx]) and np.isfinite(a[qy, qx]).all()
                                and np.isfinite(m[qy, qx]).all() and np.isfinite(z[qy, qx])):
                            continue
                        dc, dn, da = c[y, x] - c[qy, qx], m[y, x] - m[qy, qx], a[y, x] - a[qy, qx]
                        sq = lambda u: (u[0] * u[0] + u[1] * u[1]) + u[2] * u[2]
                        e = ((np.sqrt(sq(dc)) * rc + sq(dn) * rn) + sq(da) * ra) + abs(z[y, x] - z[qy, qx]) * rz
                        w = D.KERNEL[dx + 2] * D.KERNEL[dy + 2] * np.exp(-e)
                        sw = sw + w
                        acc = acc + w * c[qy, qx]
                        sv = sv + (w * w) * v[qy, qx]
                c2[y, x] = acc / sw
                v2[y, x] = sv / (sw * sw)
        c, v = c2, v2
    return c


def test_restatement_is_the_per_pixel_formula():
    """The vectorised restatement equals a one-tap-at-a-time evaluation on random inputs with edges, including the frame border."""
    rng = np.random.default_rng(3)
    H, W, n = 9, 11, 8
    S = rng.uniform(0.0, 2.0, (H, W, 3)) * n
    Q = S * S / n + rng.uniform(0.0, 0.5, (H, W, 3)) * (n - 1)
    albedo = np.where(rng.random((H, W, 1)) < 0.5, 0.2, 0.7) * np.ones(3)
    normal = rng.normal(size=(H, W, 3))
    normal /= np.linalg.norm(normal, axis=-1, keepdims=True)
    depth = rng.uniform(1.0, 4.0, (H, W))
    S[4, 5, 1] = np.nan
    got = D.denoise(S, Q, albedo, normal, depth, n, 3, 2.0, 0.7, 0.3, 0.5)
    want = scalar_denoise(S, Q, albedo, normal, depth, n, 3, 2.0, 0.7, 0.3, 0.5)
    assert got.dtype == np.float32
    np.testing.assert_allclose(got, want, rtol=2e-6, atol=1e-7)


def test_constant_image_is_unchanged():
    S, Q, albedo, normal, depth, n = inputs()
    out = D.denoise(S, Q, albedo, normal, depth, n, **D.DEFAULTS)
    np.testing.assert_allclose(out, 0.5, rtol=1e-6)


def test_noise_free_albedo_step_does_not_bleed():
    """Left half albedo and colour 0.2, right half 0.8.  Without noise, and with noise large enough that the colour term alone
    would let the halves mix, the albedo term keeps every pixel within 1e-4 of its own side's value."""
    H, W, n = 12, 16, 16
    for var in (0.0, 4.0):
        S, Q, albedo, normal, depth, _ = inputs(H, W, n, var=var)
        side = np.where(np.arange(W) < W // 2, 0.2, 0.8)[None, :, None] * np.ones((H, 1, 3))
        S = side * n
        Q = S * side + var * (n - 1)
        albedo = side.copy()
        out = D.denoise(S, Q, albedo, normal, depth, n, **D.DEFAULTS)
        np.testing.assert_allclose(out, side.astype(np.float32), rtol=1e-4, err_msg=f"variance {var}")
        if var:      # the colour term alone does mix them: the albedo term is what holds the edge
            mixed = D.denoise(S, Q, np.full_like(albedo, 0.5), normal, depth, n, **D.DEFAULTS)
            assert np.abs(mixed - side).max() > 0.01


def test_nonfinite_pixels_are_copied_and_skipped():
    """A pixel with any non-finite value keeps its colour, and its neighbours ignore it as a tap."""
    S, Q, albedo, normal, depth, n = inputs()
    S[3, 4, 0] = np.nan
    normal[6, 7, 2] = np.nan
    S[8, 2, 1] = np.inf
    Q[8, 10, 2] = np.inf            # infinite variance: the pixel is copied as it is
    out = D.denoise(S, Q, albedo, normal, depth, n, **D.DEFAULTS)
    c, *_ = D.pack(S, Q, albedo, normal, depth, n)
    for y, x in ((3, 4), (6, 7), (8, 2), (8, 10)):
        np.testing.assert_array_equal(out[y, x], c[y, x])
    assert np.isnan(out[3, 4, 0]) and np.isposinf(out[8, 2, 1])
    others = np.ones(out.shape[:2], bool)
    others[[3, 6, 8, 8], [4, 7, 2, 10]] = False
    np.testing.assert_allclose(out[others], 0.5, rtol=1e-6)
