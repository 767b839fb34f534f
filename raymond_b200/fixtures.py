"""Scene and mesh fixtures for the benchmark configurations (harness data, numpy only).

The two benchmark scenes are the ones `cli_old` hard-codes (reference
cli_old/src/main.rs:45-150, SURVEY.md Appendix D).  A scene is described as plain
data — a list of object tuples — so the same description can be instantiated
through the product C ABI (raymond_b200.api) and through the CPU oracle (tests).

    ("sphere", origin, radius, material)
    ("plane",  origin, normal, material)
    ("grid",   triangles ndarray (n, 33) f64, material)      # reference Triangle layout, 264 B
    material = ("Diffuse", colour, roughness) | ("Metal", colour, roughness)
             | ("Emission", e, b, p0, p1)

The GoldDragon mesh (assets/meshes/dragon_vrip.ply) is missing from the reference
snapshot (.MISSING_LARGE_BLOBS); `dragon_standin()` generates a documented stand-in
of the same triangle count class and bounding box regime.  Every number measured
on it is flagged "stand-in".
"""
from __future__ import annotations

import numpy as np

TRI_DOUBLES = 33
# offsets inside one 33-double triangle record: vertex k starts at 11*k
_POS, _NRM, _UV, _TAN = 0, 3, 6, 8

# ---------------------------------------------------------------------------- scenes

# cli_old/src/main.rs:77-127 — the box; order matters for ties (scene.rs:61)
BOX_PLANES = [
    ("plane", (0.0, -1.0, 0.0), (0.0, 1.0, 0.0), ("Diffuse", (0.75, 0.75, 0.75), 0.5)),                       # floor
    ("plane", (0.0, 2.0, 0.0), (0.0, -1.0, 0.0), ("Emission", (1.5, 1.5, 1.5), (1.0, 1.0, 1.0), 0.27, 0.0)),  # ceiling
    ("plane", (0.0, 0.0, -2.0), (0.0, 0.0, 1.0), ("Diffuse", (1.0, 1.0, 1.0), 0.4)),                          # front wall
    ("plane", (0.0, 0.0, 5.0), (0.0, 0.0, -1.0), ("Diffuse", (0.0, 0.0, 0.0), 0.9)),                          # back wall
    ("plane", (-2.0, 0.0, 0.0), (1.0, 0.0, 0.0), ("Diffuse", (0.0, 0.0, 0.0), 0.3)),                          # left wall
    ("plane", (2.0, 0.0, 0.0), (-1.0, 0.0, 0.0), ("Diffuse", (0.0, 0.0, 0.0), 0.3)),                          # right wall
]
RED_SPHERE = ("sphere", (-1.0, -0.5, 3.5), 0.5, ("Diffuse", (1.0, 0.0, 0.0), 0.02))       # cli_old/src/main.rs:48-55
BLUE_SPHERE = ("sphere", (0.74, -0.25, 3.5), 0.75, ("Metal", (0.05, 0.25, 1.00), 0.01))   # cli_old/src/main.rs:56-58 (commented out there)
DRAGON_MATERIAL = ("Metal", (1.0, 1.0, 0.1), 0.15)                                        # cli_old/src/main.rs:74
DRAGON_TRANSLATE = (0.0, -0.3, 2.9)                                                       # cli_old/src/main.rs:61


def camera(width: int, height: int, *, fov_vert: float = 55.0, position=(0.0, 0.0, 0.0), focal_length: float = 2.5,
           aperture_radius: float = 0.0) -> dict:
    """CameraSettings as cli_old builds them (cli_old/src/main.rs:134-142)."""
    return {"width": int(width), "height": int(height), "fov_vert": float(fov_vert), "position": tuple(map(float, position)),
            "focal_length": float(focal_length), "aperture_radius": float(aperture_radius)}


def reflective_spheres() -> list:
    """ReflectiveSpheres: red diffuse + blue metal sphere in the box (README image; SURVEY Appendix D)."""
    return [RED_SPHERE, BLUE_SPHERE] + BOX_PLANES


def gold_dragon(triangles: np.ndarray) -> list:
    """GoldDragon as cli_old builds it: red sphere, Grid(mesh translated by (0,-0.3,2.9)), box."""
    return [RED_SPHERE, ("grid", translate(triangles, DRAGON_TRANSLATE), DRAGON_MATERIAL)] + BOX_PLANES


FLOOR = BOX_PLANES[0]


def open_dragon(triangles: np.ndarray) -> list:
    """The GoldDragon scene without its walls and ceiling: floor, red sphere and the dragon under the open sky (the scene
    `cli_old --open` builds).  Rays that leave it see the environment map, if the scene has one."""
    return [RED_SPHERE, ("grid", translate(triangles, DRAGON_TRANSLATE), DRAGON_MATERIAL), FLOOR]


def open_spheres() -> list:
    """Spheres on a floor under the open sky: diffuse and metal, rough and smooth."""
    return [RED_SPHERE, BLUE_SPHERE,
            ("sphere", (0.0, -0.6, 4.6), 0.4, ("Metal", (0.9, 0.9, 0.9), 0.6)),
            ("sphere", (1.3, -0.7, 2.8), 0.3, ("Diffuse", (0.2, 0.8, 0.3), 0.9)), FLOOR]


def sky(width: int = 256, height: int = 128, *, sun_dir=(0.4, 0.6, 0.7), sun_radius_deg: float = 2.5, sun_radiance: float = 400.0) -> np.ndarray:
    """Procedural equirectangular sky, (height, width, 3) float32 in the layout of include/raymond.h's rm_environment: a
    horizon-to-zenith gradient above, a dim ground below, and a small bright sun disc in direction `sun_dir`."""
    v = (np.arange(height) + 0.5) / height
    u = (np.arange(width) + 0.5) / width
    V, U = np.meshgrid(v, u, indexing="ij")
    theta = V * np.pi                              # 0 = +y
    phi = (U - 0.5) * 2.0 * np.pi                  # atan2(d.x, d.z)
    d = np.stack([np.sin(theta) * np.sin(phi), np.cos(theta), np.sin(theta) * np.cos(phi)], axis=-1)
    up = np.clip(d[..., 1], 0.0, 1.0)[..., None]
    horizon = np.array([0.9, 0.95, 1.0])
    zenith = np.array([0.25, 0.45, 0.95])
    ground = np.array([0.18, 0.16, 0.14])
    img = np.where(d[..., 1:2] >= 0.0, horizon + (zenith - horizon) * np.sqrt(up), ground)
    sd = np.asarray(sun_dir, dtype=np.float64)
    sd = sd / np.linalg.norm(sd)
    sun = (d @ sd) >= np.cos(np.radians(sun_radius_deg))
    img[sun] = sun_radiance * np.array([1.0, 0.95, 0.85])
    return np.ascontiguousarray(img, dtype=np.float32)


def write_hdr(path: str, image: np.ndarray, rle: bool = True) -> None:
    """Write (H, W, 3) radiance as a Radiance RGBE (.hdr) file ("-Y H +X W"); scanlines run-length encoded when `rle` and
    8 <= W <= 32767 (the only widths the format encodes), else flat."""
    img = np.asarray(image, dtype=np.float64)
    H, W = img.shape[:2]
    rgbe = rgbe_encode(img)
    with open(path, "wb") as f:
        f.write(b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n" + f"-Y {H} +X {W}\n".encode())
        for y in range(H):
            row = rgbe[y]
            if rle and 8 <= W <= 32767:
                f.write(bytes([2, 2, W >> 8, W & 255]))
                for c in range(4):
                    f.write(_rle_channel(row[:, c]))
            else:
                f.write(row.tobytes())


def rgbe_encode(img: np.ndarray) -> np.ndarray:
    """(…, 3) radiance -> (…, 4) uint8 RGBE (m = floor(v * 256 / 2^e'), exponent of the largest channel)."""
    img = np.asarray(img, dtype=np.float64)
    mx = img.max(axis=-1)
    m, e = np.frexp(mx)                            # mx = m * 2^e, m in [0.5, 1)
    scale = np.where(mx > 1e-32, np.ldexp(256.0, -e), 0.0)
    out = np.zeros(img.shape[:-1] + (4,), dtype=np.uint8)
    out[..., :3] = np.clip(np.floor(img * scale[..., None]), 0, 255).astype(np.uint8)
    out[..., 3] = np.where(mx > 1e-32, np.clip(e + 128, 0, 255), 0).astype(np.uint8)
    return out


def rgbe_decode(rgbe: np.ndarray) -> np.ndarray:
    """uint8 RGBE -> float32 radiance: (m + 0.5) * 2^(e - 136), 0 for e == 0 (include/raymond.h, rm_load_hdr)."""
    q = np.asarray(rgbe, dtype=np.uint8)
    e = q[..., 3:4].astype(np.int64)
    v = np.ldexp(q[..., :3].astype(np.float64) + 0.5, e - 136)
    return np.where(e == 0, 0.0, v).astype(np.float32)


def _rle_channel(vals: np.ndarray) -> bytes:
    """New-style RLE of one channel of a scanline: runs of >= 3 equal bytes as (128 + n, value), n <= 127; the rest as
    literal spans (n, bytes...), n <= 128."""
    out = bytearray()
    v = np.asarray(vals, dtype=np.uint8)
    n = len(v)
    i = 0
    lit = []
    while i < n:
        j = i
        while j < n and j - i < 127 and v[j] == v[i]:
            j += 1
        if j - i >= 3:
            while lit:
                out += bytes([min(len(lit), 128)]) + bytes(lit[:128])
                lit = lit[128:]
            out += bytes([128 + (j - i), int(v[i])])
            i = j
        else:
            lit.append(int(v[i]))
            i += 1
    while lit:
        out += bytes([min(len(lit), 128)]) + bytes(lit[:128])
        lit = lit[128:]
    return bytes(out)


def soup_scene(triangles: np.ndarray) -> list:
    """C4: one Grid object, Metal((1,1,0.1), 0.15) (SURVEY §8d)."""
    return [("grid", triangles, DRAGON_MATERIAL)]


# ---------------------------------------------------------------------------- mesh helpers

def make_triangles(p0, p1, p2, n0=None, n1=None, n2=None) -> np.ndarray:
    """Pack positions (and vertex normals; default = unit face normal) into (n, 33) reference-layout records."""
    p0 = np.asarray(p0, dtype=np.float64).reshape(-1, 3)
    p1 = np.asarray(p1, dtype=np.float64).reshape(-1, 3)
    p2 = np.asarray(p2, dtype=np.float64).reshape(-1, 3)
    n = p0.shape[0]
    if n0 is None:
        fn = np.cross(p1 - p0, p2 - p0)
        ln = np.linalg.norm(fn, axis=1, keepdims=True)
        fn = fn / np.where(ln > 0, ln, 1.0)
        n0 = n1 = n2 = fn
    out = np.zeros((n, TRI_DOUBLES))
    for k, (p, nn) in enumerate(((p0, n0), (p1, n1), (p2, n2))):
        out[:, 11 * k + _POS:11 * k + _POS + 3] = p
        out[:, 11 * k + _NRM:11 * k + _NRM + 3] = np.asarray(nn, dtype=np.float64).reshape(-1, 3)
    return out


def positions(tris: np.ndarray) -> np.ndarray:
    """(n, 3, 3) vertex positions of (n, 33) triangle records."""
    t = np.asarray(tris).reshape(-1, 3, 11)
    return t[:, :, 0:3]


def normals(tris: np.ndarray) -> np.ndarray:
    t = np.asarray(tris).reshape(-1, 3, 11)
    return t[:, :, 3:6]


def translate(tris: np.ndarray, offset) -> np.ndarray:
    """Mesh::bake_transform (mesh.rs:48-56): position += translate, one IEEE add per component."""
    out = np.array(tris, dtype=np.float64, copy=True).reshape(-1, 3, 11)
    out[:, :, 0:3] += np.asarray(offset, dtype=np.float64)
    return out.reshape(-1, TRI_DOUBLES)


def write_ply(path: str, tris: np.ndarray, with_uv: bool = False) -> None:
    """Blender-style ASCII PLY (x y z nx ny nz [s t]; one vertex per corner) that Mesh::load_ply accepts."""
    t = np.asarray(tris).reshape(-1, 3, 11)
    n = t.shape[0]
    with open(path, "w") as f:
        f.write("ply\nformat ascii 1.0\ncomment generated by raymond_b200.fixtures\n")
        f.write(f"element vertex {3 * n}\n")
        for name in ("x", "y", "z", "nx", "ny", "nz") + (("s", "t") if with_uv else ()):
            f.write(f"property float {name}\n")
        f.write(f"element face {n}\nproperty list uchar uint vertex_indices\nend_header\n")
        cols = 8 if with_uv else 6
        for v in t.reshape(-1, 11)[:, :cols]:
            f.write(" ".join(f"{x:.6f}" for x in v) + "\n")
        for i in range(n):
            f.write(f"3 {3 * i} {3 * i + 1} {3 * i + 2}\n")


def cube(half: float = 0.521075) -> np.ndarray:
    """Axis-aligned cube, 12 triangles, flat normals (same shape as the reference's cube asset)."""
    h = half
    faces = []
    for axis in range(3):
        for sgn in (1.0, -1.0):
            u, v = (axis + 1) % 3, (axis + 2) % 3
            c = np.zeros((4, 3))
            c[:, axis] = sgn * h
            c[:, u] = [h, -h, -h, h]
            c[:, v] = [h, h, -h, -h]
            if sgn < 0:
                c = c[::-1]
            faces.append((c[0], c[1], c[2]))
            faces.append((c[0], c[2], c[3]))
    p = np.array(faces)
    return make_triangles(p[:, 0], p[:, 1], p[:, 2])


def bumpy_sphere(n_lat: int = 24, n_lon: int = 48, radius: float = 1.0, bump: float = 0.12, squash=(1.0, 0.8, 0.6), *,
                 uv: bool = False) -> np.ndarray:
    """Closed bumpy ellipsoid with smooth vertex normals — a small anisotropic test mesh
    (res.y > res.z after the grid resolution estimate => exercises the aliasing quirk A1).  `uv`: see _grid_surface."""
    th = np.linspace(0.0, np.pi, n_lat + 1)
    ph = np.linspace(0.0, 2.0 * np.pi, n_lon, endpoint=False)
    T, P = np.meshgrid(th, ph, indexing="ij")
    r = radius * (1.0 + bump * np.sin(5.0 * T) * np.cos(4.0 * P) + 0.5 * bump * np.cos(3.0 * T + 1.0))
    pts = np.stack([r * np.sin(T) * np.cos(P), r * np.cos(T), r * np.sin(T) * np.sin(P)], axis=-1) * np.asarray(squash)
    return _grid_surface(pts, wrap_u=False, wrap_v=True, uv=uv)


def _grid_surface(pts: np.ndarray, wrap_u: bool, wrap_v: bool, uv: bool = False) -> np.ndarray:
    """Triangulate a (nu, nv, 3) point grid; smooth vertex normals from central differences.  `uv`: every vertex carries its
    surface parameter as its uv, (i, j) / (the number of cells along u, along v), so the texture of rm_texture spans the
    surface once; the last cell of a wrapped axis ends at 1, not 0.  Without `uv` the uvs stay zero (the arrays the fixtures
    always had)."""
    nu, nv, _ = pts.shape
    du = np.roll(pts, -1, axis=0) - np.roll(pts, 1, axis=0)
    dv = np.roll(pts, -1, axis=1) - np.roll(pts, 1, axis=1)
    if not wrap_u:
        du[0] = pts[1] - pts[0]
        du[-1] = pts[-1] - pts[-2]
    if not wrap_v:
        dv[:, 0] = pts[:, 1] - pts[:, 0]
        dv[:, -1] = pts[:, -1] - pts[:, -2]
    nrm = np.cross(dv, du)
    ln = np.linalg.norm(nrm, axis=-1, keepdims=True)
    # poles of a lat/long grid have a zero derivative: fall back to the radial direction
    rad = pts / np.maximum(np.linalg.norm(pts, axis=-1, keepdims=True), 1e-300)
    nrm = np.where(ln > 1e-12, nrm / np.maximum(ln, 1e-300), rad)
    iu = np.arange(nu if wrap_u else nu - 1)
    iv = np.arange(nv if wrap_v else nv - 1)
    I, J = np.meshgrid(iu, iv, indexing="ij")
    I1, J1 = (I + 1) % nu, (J + 1) % nv
    a = (I, J); b = (I1, J); c = (I1, J1); d = (I, J1)
    p = lambda ij: pts[ij[0], ij[1]].reshape(-1, 3)
    n = lambda ij: nrm[ij[0], ij[1]].reshape(-1, 3)
    t1 = make_triangles(p(a), p(b), p(c), n(a), n(b), n(c))
    t2 = make_triangles(p(a), p(c), p(d), n(a), n(c), n(d))
    if uv:
        cu, cv = float(len(iu)), float(len(iv))
        st = lambda i, j: np.stack([i.reshape(-1) / cu, j.reshape(-1) / cv], axis=-1)
        for t, corners in ((t1, (st(I, J), st(I + 1, J), st(I + 1, J + 1))), (t2, (st(I, J), st(I + 1, J + 1), st(I, J + 1)))):
            for k, c2 in enumerate(corners):
                t[:, 11 * k + _UV:11 * k + _UV + 2] = c2
    out = np.empty((t1.shape[0] * 2, TRI_DOUBLES))
    out[0::2] = t1
    out[1::2] = t2
    # drop degenerate (zero-area) triangles at poles
    pos = positions(out)
    area2 = np.linalg.norm(np.cross(pos[:, 1] - pos[:, 0], pos[:, 2] - pos[:, 0]), axis=1)
    return np.ascontiguousarray(out[area2 > 1e-14])


def dragon_standin(nu: int = 1320, nv: int = 330, *, uv: bool = False) -> np.ndarray:
    """STAND-IN for the missing dragon_vrip.ply: a closed, bumpy tube around a closed space curve.

    Default 1320 x 330 x 2 = 871 200 triangles (the Stanford dragon has 871 414), smooth vertex
    normals, mesh-local bounding box ~ x[-1.14, 1.14] y[-0.63, 0.85] z[-0.50, 0.50] — the regime
    SURVEY.md Appendix D estimates from examples/GoldDragon.png (res.y > res.z, so the grid's
    index aliasing A1 is exercised; rests near the floor after the (0, -0.3, 2.9) translate).
    Deterministic (no RNG).  `uv`: the tube's (curve, around) parameter as the vertices' uv (see _grid_surface).
    """
    s = np.linspace(0.0, 2.0 * np.pi, nu, endpoint=False)
    ph = np.linspace(0.0, 2.0 * np.pi, nv, endpoint=False)
    c = np.stack([0.92 * np.cos(s), 0.11 + 0.50 * np.sin(2.0 * s + 0.4), 0.28 * np.sin(3.0 * s)], axis=-1)
    dc = np.stack([-0.92 * np.sin(s), 1.00 * np.cos(2.0 * s + 0.4), 0.84 * np.cos(3.0 * s)], axis=-1)
    T = dc / np.linalg.norm(dc, axis=1, keepdims=True)
    z = np.array([0.0, 0.0, 1.0])
    n1 = np.cross(z, T)
    n1 /= np.linalg.norm(n1, axis=1, keepdims=True)     # T is never parallel to z on this curve
    n2 = np.cross(T, n1)
    S, P = np.meshgrid(s, ph, indexing="ij")
    r = 0.17 + 0.045 * np.sin(5.0 * S) + 0.012 * np.sin(40.0 * S) * np.sin(24.0 * P) + 0.004 * np.sin(130.0 * S + 7.0 * P)
    pts = c[:, None, :] + r[..., None] * (np.cos(P)[..., None] * n1[:, None, :] + np.sin(P)[..., None] * n2[:, None, :])
    return _grid_surface(pts, wrap_u=True, wrap_v=True, uv=uv)


# ---------------------------------------------------------------------------- triangle soup (C4)

def _splitmix64(seed: int, n: int) -> np.ndarray:
    """First n outputs of SplitMix64(seed), vectorised."""
    with np.errstate(over="ignore"):
        i = np.arange(1, n + 1, dtype=np.uint64)
        z = np.uint64(seed) + i * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def _uniform(seed: int, n: int) -> np.ndarray:
    return (_splitmix64(seed, n) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


SOUP_BOX_CUBIC = ((-1.0, 1.0), (-1.0, 1.0), (2.0, 4.0))      # B1: cubic grid, index formula exact
SOUP_BOX_FLAT = ((-1.0, 1.0), (-0.7, 0.7), (2.55, 3.45))     # B2: res.y > res.z => aliasing path


def triangle_soup(n: int, box=SOUP_BOX_CUBIC, seed: int | None = None) -> np.ndarray:
    """SURVEY §8d C4 soup: n triangles, centres uniform in `box`, vertices = centre + U[-s, s]^3 with
    s = 0.5 (vol/n)^(1/3); vertex normals = unit face normal; SplitMix64 seed 0x5EED0000 + n."""
    seed = (0x5EED0000 + n) if seed is None else seed
    u = _uniform(seed, 12 * n).reshape(n, 12)
    lo = np.array([b[0] for b in box]); hi = np.array([b[1] for b in box])
    vol = float(np.prod(hi - lo))
    s = 0.5 * (vol / n) ** (1.0 / 3.0)
    centre = lo + u[:, 0:3] * (hi - lo)
    off = (u[:, 3:12].reshape(n, 3, 3) * 2.0 - 1.0) * s
    p = centre[:, None, :] + off
    return make_triangles(p[:, 0], p[:, 1], p[:, 2])


def random_rays(n: int, seed: int = 0xD1CE, origin_box=((-2.0, 2.0), (-1.0, 2.0), (-2.0, 5.0))) -> np.ndarray:
    """SURVEY §8d C4 (ii): origins uniform in a box, directions uniform on the sphere; (n, 6) f64."""
    u = _uniform(seed, 5 * n).reshape(n, 5)
    lo = np.array([b[0] for b in origin_box]); hi = np.array([b[1] for b in origin_box])
    o = lo + u[:, 0:3] * (hi - lo)
    zc = 2.0 * u[:, 3] - 1.0
    ph = 2.0 * np.pi * u[:, 4]
    rr = np.sqrt(np.maximum(0.0, 1.0 - zc * zc))
    d = np.stack([rr * np.cos(ph), rr * np.sin(ph), zc], axis=-1)
    return np.ascontiguousarray(np.concatenate([o, d], axis=1))


# ---------------------------------------------------------------------------- display transform

def tonemap(linear: np.ndarray, exposure: float = 1.0, gamma: float = 2.2) -> np.ndarray:
    """cli_old/src/main.rs:157-181: 1 - exp(p * -1 * exposure), ^(1 / gamma), x255, truncate; out-of-range/NaN pixel stays 0."""
    p = np.asarray(linear, dtype=np.float64)
    with np.errstate(invalid="ignore", over="ignore", divide="ignore"):
        c = np.power(1.0 - np.exp(p * -1.0 * exposure), 1.0 / gamma) * 255.0
    ok = np.all(np.isfinite(c) & (c > -1.0) & (c < 256.0), axis=-1, keepdims=True)
    return np.where(ok, np.nan_to_num(c), 0.0).astype(np.uint8)
