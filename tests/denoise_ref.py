"""numpy float32 restatement of the feature-guided a-trous denoiser of rm_renderer_read_denoised (include/raymond.h).

The inputs are what the renderer's own readers return: S (read_sums), Q (read_moments) and the feature means of read_aovs.  They
are packed in f64 exactly as the library packs them and rounded to f32 once; every later operation is f32, in the library's order.
"""
import numpy as np

F = np.float32
KERNEL = np.array([1.0 / 16.0, 1.0 / 4.0, 3.0 / 8.0, 1.0 / 4.0, 1.0 / 16.0], dtype=np.float32)
DEFAULTS = dict(iterations=1, sigma_color=1e4, sigma_normal=0.1, sigma_albedo=0.3, sigma_depth=1.0)     # include/raymond.h


def pack(S, Q, albedo, normal, depth, n):
    """(colour (H, W, 3), variance (H, W), albedo, normal, depth) in f32: c = S / n, v = se2_R + se2_G + se2_B."""
    n = float(n)
    m = S / n
    d = Q - S * m
    se2 = np.where(d < 0.0, 0.0, d) / (n - 1.0) / n
    v = (se2[..., 0] + se2[..., 1]) + se2[..., 2]
    return m.astype(F), v.astype(F), albedo.astype(F), normal.astype(F), depth.astype(F)


def _finite(c, v, a, m, z):
    return np.isfinite(c).all(-1) & np.isfinite(v) & np.isfinite(a).all(-1) & np.isfinite(m).all(-1) & np.isfinite(z)


def _sq3(x):
    return (x[..., 0] * x[..., 0] + x[..., 1] * x[..., 1]) + x[..., 2] * x[..., 2]


def atrous(c, v, a, m, z, step, sigma_color, sigma_normal, sigma_albedo, sigma_depth):
    """One pass at tap distance `step` over f32 arrays; returns (c', v')."""
    H, W = v.shape
    sc, sn, sa, sz = F(sigma_color), F(sigma_normal), F(sigma_albedo), F(sigma_depth)
    ok = _finite(c, v, a, m, z)
    one = F(1.0)
    rc = one / (sc * np.sqrt(v) + F(1e-6))
    rn = one / (sn * sn)
    ra = one / (sa * sa)
    rz = one / (sz * F(step) * z + F(1e-6))
    sw = np.zeros((H, W), F)
    acc = np.zeros((H, W, 3), F)
    sv = np.zeros((H, W), F)
    ys, xs = np.arange(H)[:, None], np.arange(W)[None, :]
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            qy, qx = ys + dy * step, xs + dx * step
            inside = (qy >= 0) & (qy < H) & (qx >= 0) & (qx < W)
            qyc, qxc = np.clip(qy, 0, H - 1), np.clip(qx, 0, W - 1)
            cq, vq, aq, mq, zq = c[qyc, qxc], v[qyc, qxc], a[qyc, qxc], m[qyc, qxc], z[qyc, qxc]
            use = inside & ok[qyc, qxc] & ok
            with np.errstate(all="ignore"):
                e = ((np.sqrt(_sq3(c - cq)) * rc + _sq3(m - mq) * rn) + _sq3(a - aq) * ra) + np.abs(z - zq) * rz
                w = (KERNEL[dx + 2] * KERNEL[dy + 2]) * np.exp(-e)
            w = np.where(use, w, F(0.0)).astype(F)
            sw = sw + w
            acc = acc + w[..., None] * np.where(use[..., None], cq, F(0.0))
            sv = sv + (w * w) * np.where(use, vq, F(0.0))
    with np.errstate(all="ignore"):
        c2 = acc / sw[..., None]
        v2 = sv / (sw * sw)
    return np.where(ok[..., None], c2, c).astype(F), np.where(ok, v2, v).astype(F)


def denoise(S, Q, albedo, normal, depth, n, iterations, sigma_color, sigma_normal, sigma_albedo, sigma_depth):
    """The final colour (H, W, 3) f32 of rm_renderer_read_denoised."""
    c, v, a, m, z = pack(S, Q, albedo, normal, depth, n)
    for i in range(iterations):
        c, v = atrous(c, v, a, m, z, 1 << i, sigma_color, sigma_normal, sigma_albedo, sigma_depth)
    return c
