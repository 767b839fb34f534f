"""CPU tests of the ORACLE (oracle/raymond_oracle.cpp) — what pins the checker itself.

The reference has no tests, golden vectors or fixtures (SURVEY §4, §8c) and cannot be compiled here, so the
oracle is anchored by everything that IS available:
  * the reference's own rendered output, examples/ReflectiveSpheres.png (block means in tests/golden/, made by
    scripts/make_golden.py) — the only output of the reference itself;
  * an independent pure-Python restatement of the intersection code written from the Rust sources (tests/pyref.py),
    compared bit for bit;
  * the reference's brute-force Mesh::intersects (mesh.rs:23-42) as a cross-check of the grid on camera-side rays;
  * known answers on the reference's shipped meshes (SURVEY Appendix C; tests/golden/reference_mesh_kats.json).
"""
import json
import os
import zlib

import numpy as np
import pytest

import pyref
from oracle import oracle as O
from raymond_b200 import fixtures as F

from util import NEEDS_REFERENCE, REFERENCE_DIR, REFERENCE_MESHES, have_reference_assets, oracle_scene

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_reference = pytest.mark.skipif(not have_reference_assets(), reason=NEEDS_REFERENCE)


def _tri_positions(tris):
    p = F.positions(tris)
    return [tuple(tuple(float(c) for c in v) for v in t) for t in p]


def _same_bits(a: float, b: float) -> bool:
    return pyref.bits(a) == pyref.bits(b)


# ------------------------------------------------------------------ independent restatement, bit for bit

@pytest.mark.parametrize("name,tris", [("cube", F.cube()), ("bumpy", F.bumpy_sphere(10, 20)), ("tube", F.dragon_standin(40, 10))])
def test_grid_build_matches_python_restatement(name, tris):
    g = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(tris))
    pg = pyref.Grid(_tri_positions(tris))
    info = g.info()
    assert info["resolution"] == list(pg.res)
    assert [pyref.bits(x) for x in info["cell_size"]] == [pyref.bits(x) for x in pg.cell]
    cells, table = g.tables()
    assert cells.tolist() == pg.cells and table.tolist() == pg.table


@pytest.mark.parametrize("name,tris", [("cube", F.cube()), ("bumpy", F.bumpy_sphere(10, 20)), ("tube", F.dragon_standin(40, 10))])
def test_grid_traversal_matches_python_restatement(name, tris):
    g = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(tris))
    pg = pyref.Grid(_tri_positions(tris))
    rays = np.concatenate([O.primary_rays(F.camera(24, 18, position=(0.0, 0.0, -4.0))), F.random_rays(1500, 3, ((-2, 2), (-2, 2), (-2, 2)))])
    # aim a third of the random rays at the mesh so that inside / fix-up / +side starts are all hit
    aim = F.random_rays(rays.shape[0], 5, ((-0.5, 0.5), (-0.3, 0.3), (-0.3, 0.3)))[:, :3] - rays[:, :3]
    aim /= np.linalg.norm(aim, axis=1, keepdims=True)
    rays[500::3, 3:] = aim[500::3]
    rays[7, 3:] = (0.0, 0.0, 1.0)
    rays[8, 3:] = (-0.0, 1.0, 0.0)
    tri, t, _ = g.intersects(rays)
    hits = 0
    for i, r in enumerate(rays):
        want = pg.intersects(tuple(r[:3]), tuple(r[3:]))
        if want is None:
            assert tri[i] == -1, f"ray {i}: oracle hit {tri[i]}, python restatement missed"
        else:
            hits += 1
            assert tri[i] == want[0] and _same_bits(t[i], want[1]), f"ray {i}: oracle ({tri[i]}, {t[i]!r}) vs python {want}"
    assert hits > 50


def test_scene_intersect_matches_python_restatement():
    objs = F.gold_dragon(F.dragon_standin(40, 10))
    sc = oracle_scene(objs)
    pobjs = []
    for o in objs:
        if o[0] == "sphere":
            pobjs.append(("sphere", tuple(map(float, o[1])), float(o[2])))
        elif o[0] == "plane":
            pobjs.append(("plane", tuple(map(float, o[1])), tuple(map(float, o[2]))))
        else:
            pobjs.append(("grid", pyref.Grid(_tri_positions(o[1]))))
    rays = np.concatenate([O.primary_rays(F.camera(32, 18)), F.random_rays(800, 9, ((-1.9, 1.9), (-0.9, 1.9), (-1.9, 4.9)))])
    obj, sub, t, _ = sc.intersect(rays)
    seen = set()
    for i, r in enumerate(rays):
        want = pyref.scene_intersect(pobjs, tuple(r[:3]), tuple(r[3:]))
        if want is None:
            assert obj[i] == -1
        else:
            seen.add(want[0])
            assert (obj[i], sub[i]) == (want[0], want[1]) and _same_bits(t[i], want[2]), f"ray {i}"
    assert len(seen) >= 6


def test_primary_rays_match_python_restatement():
    for cam in (F.camera(31, 17), F.camera(16, 9, fov_vert=90.0, position=(1.0, -2.0, 0.5))):
        rays = O.primary_rays(cam)
        jit = np.random.default_rng(1).random((cam["width"] * cam["height"], 2))
        jrays = O.primary_rays(cam, jit)
        for y in range(cam["height"]):
            for x in range(cam["width"]):
                i = y * cam["width"] + x
                o, d = pyref.primary_ray(x, y, cam)
                assert [pyref.bits(v) for v in rays[i]] == [pyref.bits(v) for v in (*o, *d)]
                o, d = pyref.primary_ray(x, y, cam, jit[i, 0] - 0.5, jit[i, 1] - 0.5)
                assert [pyref.bits(v) for v in jrays[i]] == [pyref.bits(v) for v in (*o, *d)]


def test_tile_layout_matches_python_restatement():
    for (w, h, tw, th) in ((592, 340, 32, 32), (100, 70, 32, 32), (64, 64, 64, 64), (65, 1, 8, 8), (7, 300, 16, 7)):
        assert O.tile_layout(F.camera(w, h), (tw, th)).tolist() == [list(r) for r in pyref.tile_layout(w, h, tw, th)]


# ------------------------------------------------------------------ known answers (SURVEY Appendix C)

def test_cube_known_answers():
    """Generated cube with the half-extent of the reference's cube.ply: res [3,3,3], quirks A1/A3 visible."""
    g = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(F.cube()))
    assert g.info()["resolution"] == [3, 3, 3] and g.info()["cell_count"] == 27
    assert g.info()["cell_size"][0] == 0.3473833333333333
    rays = np.array([[0.1, 0.05, -3, 0, 0, 1], [-2, 0.03, 0.02, 1, 0, 0], [0.1, -3, 0.05, 0, 1, 0],
                     [2, 0, 0, -1, 0, 0], [0.1, 0.05, 3, 0, 0, -1], [0.1, 3, 0.05, 0, -1, 0]], dtype=np.float64)
    tri, t, _ = g.intersects(rays)
    assert (tri[:3] >= 0).all() and (tri[3:] == -1).all()          # +side origins miss (A3 / index out of range)
    assert t[0] == 2.4789250000000003 and t[1] == 1.4789249999999998 and t[2] == 2.4789250000000003
    # the brute force (mesh.rs:23-42) does see the +side hits — the grid's misses are the reference's behaviour, not ours
    btri, bt = O.Mesh.from_triangles(F.cube()).intersects(rays)
    assert (btri >= 0).all() and bt[3] == 1.4789249999999998


@needs_reference
def test_reference_meshes_known_answers():
    kats = json.load(open(os.path.join(GOLDEN, "reference_mesh_kats.json")))
    # SURVEY Appendix C
    assert kats["monkeysmooth"]["resolution"] == [15, 10, 9] and kats["monkeysmooth"]["references"] == 3678
    assert kats["suzanne_flat"]["resolution"] == [18, 13, 11] and kats["suzanne_flat"]["references"] == 6036
    assert kats["ico_sphere"]["resolution"] == [6, 6, 6] and kats["ico_sphere"]["references"] == 825
    assert (kats["monkeysmooth"]["hits"], kats["suzanne_flat"]["hits"], kats["ico_sphere"]["hits"]) == (2276, 2308, 494)
    assert kats["suzanne"]["build_status"] == -4                    # the reference panics at acc_grid.rs:61
    rays = O.primary_rays(F.camera(160, 120, position=(0.0, 0.0, -4.0)))
    for name, k in kats.items():
        m = O.Mesh.load_ply(f"{REFERENCE_MESHES}/{name}.ply")
        assert len(m) == k["triangles"] and m.bounds.tolist() == k["bounds"]
        btri, bt = m.intersects(rays)
        if k["build_status"] != 0:
            with pytest.raises(O.OracleError) as e:
                O.AccGrid.build_from_mesh(m)
            assert e.value.status == k["build_status"]
            continue
        g = O.AccGrid.build_from_mesh(m)
        start, refs = g.csr()
        assert zlib.crc32(start.tobytes() + refs.tobytes()) == k["csr_crc32"]
        tri, t, cnt = g.intersects(rays)
        assert zlib.crc32(tri.tobytes()) == k["hit_tri_crc32"]
        assert zlib.crc32(np.where(tri >= 0, t, 0.0).tobytes()) == k["hit_t_crc32"]
        # grid == brute force on camera-side primaries (SURVEY Appendix C)
        assert np.array_equal(tri, btri) and np.array_equal(t[tri >= 0], bt[tri >= 0])


@needs_reference
def test_reference_mesh_traversal_matches_python_restatement():
    """The Blender-exported meshes with aliased (res.y > res.z) grids through both restatements."""
    m = O.Mesh.load_ply(f"{REFERENCE_MESHES}/monkeysmooth.ply")
    tris = m.triangles()
    g = O.AccGrid.build_from_mesh(m)
    pg = pyref.Grid(_tri_positions(tris))
    cells, table = g.tables()
    assert cells.tolist() == pg.cells and table.tolist() == pg.table
    rays = F.random_rays(1200, 21, ((-3, 3), (-3, 3), (-3, 3)))
    aim = F.random_rays(1200, 22, ((-1.0, 1.0), (-0.7, 0.7), (-0.6, 0.6)))[:, :3] - rays[:, :3]
    rays[:, 3:] = aim / np.linalg.norm(aim, axis=1, keepdims=True)
    tri, t, _ = g.intersects(rays)
    for i, r in enumerate(rays):
        want = pg.intersects(tuple(r[:3]), tuple(r[3:]))
        assert (tri[i] == -1) if want is None else (tri[i] == want[0] and _same_bits(t[i], want[1]))
    assert (tri >= 0).sum() > 300


def test_grid_agrees_with_brute_force_from_the_camera_side():
    """Where the quirks do not bite (origins below the box on every axis it is entered from), grid == brute force."""
    for tris in (F.bumpy_sphere(), F.translate(F.dragon_standin(96, 24), (0.0, 0.0, 0.0))):
        m = O.Mesh.from_triangles(tris)
        rays = O.primary_rays(F.camera(120, 90, position=(-0.2, -0.1, -5.0)))
        btri, bt = m.intersects(rays)
        tri, t, _ = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(tris)).intersects(rays)
        same = tri == btri
        # A2 (first cell with a hit wins, no in-cell check) may pick a different triangle on a few rays of an aliased grid
        assert same.mean() > 0.995
        assert np.array_equal(t[same & (tri >= 0)], bt[same & (tri >= 0)])


# ------------------------------------------------------------------ RNG stream (a documented deviation: counter-based)

def test_rng_stream_properties():
    u = np.array([O.rng_draw(7, p, s, d, i) for p in range(40) for s in range(5) for d in range(3) for i in range(4)])
    assert ((u > 0.0) & (u < 1.0)).all()
    assert abs(u.mean() - 0.5) < 0.02 and abs(u.var() - 1 / 12) < 0.01
    assert O.rng_draw(7, 1, 2, 3, 0) == O.rng_draw(7, 1, 2, 3, 0)
    assert len({O.rng_draw(7, 1, 2, 3, 0), O.rng_draw(8, 1, 2, 3, 0), O.rng_draw(7, 2, 2, 3, 0), O.rng_draw(7, 1, 3, 3, 0),
                O.rng_draw(7, 1, 2, 4, 0), O.rng_draw(7, 1, 2, 3, 1)}) == 6


# ------------------------------------------------------------------ the reference's own output

def _block_means(img8, block):
    H, W, _ = img8.shape
    hb, wb = H // block, W // block
    return img8[:hb * block, :wb * block].astype(np.float64).reshape(hb, block, wb, block, 3).mean(axis=(1, 3))


def test_integrator_against_the_reference_render():
    """Oracle render of the reconstructed ReflectiveSpheres scene (SURVEY Appendix D) vs the block means of the
    reference's examples/ReflectiveSpheres.png (592x340, 500 spp).  Tolerances (8-bit levels after the reference's
    tonemap, cli_old/src/main.rs:157-181): image mean within 2.0 per channel; 16x16-block means: median |diff| <= 2.0,
    95th percentile <= 8.0 (the oracle runs 48 spp, and the concave tonemap biases a noisier image darker)."""
    gold = json.load(open(os.path.join(GOLDEN, "reference_png_blocks.json")))["ReflectiveSpheres"]
    spp = 48
    sums, cnt = O.render(oracle_scene(F.reflective_spheres()), F.camera(gold["width"], gold["height"]), spp, seed=2024)
    img = F.tonemap(sums / spp)
    assert cnt["nonfinite"] == 0
    want = np.array(gold["mean_rgb8"])
    got = _block_means(img, gold["block"])
    diff = np.abs(got - want)
    assert np.abs(img.reshape(-1, 3).mean(axis=0) - np.array(gold["image_mean_rgb8"])).max() <= 2.0
    assert np.median(diff) <= 2.0 and np.percentile(diff, 95) <= 8.0, (np.median(diff), np.percentile(diff, 95))
    assert img[10, 296].tolist() == gold["ceiling_pixel_296_10"] == [227, 227, 227]      # 1 - exp(-1.5), gamma 2.2
    # paths end by emission, depth or the absorbing walls: rays per path as in SURVEY Appendix C
    assert 3.6 < cnt["rays"] / cnt["samples"] < 4.0


@pytest.fixture(scope="module")
def reflective_spheres_500spp():
    """The oracle's tonemapped ReflectiveSpheres frame at the reference's own 592x340 x 500 spp, and its counters."""
    gold = json.load(open(os.path.join(GOLDEN, "reference_png_blocks.json")))["ReflectiveSpheres"]
    spp = 500
    sums, cnt = O.render(oracle_scene(F.reflective_spheres()), F.camera(gold["width"], gold["height"]), spp, seed=77)
    return F.tonemap(sums / spp), cnt


def test_integrator_matches_the_reference_render_at_matched_spp(reflective_spheres_500spp):
    """At the reference's own 500 spp the oracle's image differs from examples/ReflectiveSpheres.png by exactly the oracle's
    seed-to-seed noise: measured 16x16-block mean |diff| 0.21 levels (oracle seed A vs seed B: 0.22), image means within 0.03
    levels per channel.  Bounds below leave ~30 % headroom over those."""
    gold = json.load(open(os.path.join(GOLDEN, "reference_png_blocks.json")))["ReflectiveSpheres"]
    img, cnt = reflective_spheres_500spp
    assert np.abs(img.reshape(-1, 3).mean(axis=0) - np.array(gold["image_mean_rgb8"])).max() <= 0.15
    bd = np.abs(_block_means(img, gold["block"]) - np.array(gold["mean_rgb8"]))
    assert bd.mean() <= 0.30 and np.percentile(bd, 95) <= 0.85 and bd.max() <= 2.5, (bd.mean(), np.percentile(bd, 95), bd.max())
    assert cnt["nonfinite"] == 0 and abs(cnt["rays"] / cnt["samples"] - 3.81) < 0.03          # SURVEY Appendix C: 3.81 rays per path


@needs_reference
def test_integrator_matches_the_reference_png_pixel_for_pixel(reflective_spheres_500spp):
    """The same frame against every pixel of examples/ReflectiveSpheres.png: measured pixel mean |diff| 3.47 (noise floor 3.49).
    Only the block means of that image are stored in tests/golden/, so the per-pixel check needs the reference checkout."""
    from PIL import Image
    img, _ = reflective_spheres_500spp
    ref = np.asarray(Image.open(os.path.join(REFERENCE_DIR, "examples", "ReflectiveSpheres.png")).convert("RGB")).astype(float)
    d = np.abs(img.astype(float) - ref)
    assert d.mean() <= 3.9 and np.median(d) <= 2.0


def test_gold_dragon_box_against_the_reference_render():
    """The dragon mesh is missing from the snapshot, but the box around it is not: blocks of examples/GoldDragon.png
    along the top of the frame (ceiling and upper walls, far from the mesh) must agree within 3 levels at 16 spp
    (the concave tonemap biases a noisier image darker), the upper-left corner within 6 on average."""
    gold = json.load(open(os.path.join(GOLDEN, "reference_png_blocks.json")))["GoldDragon"]
    spp = 16
    objs = F.gold_dragon(F.dragon_standin(330, 82))
    sums, _ = O.render(oracle_scene(objs), F.camera(gold["width"], gold["height"]), spp, seed=5)
    got = _block_means(F.tonemap(sums / spp), gold["block"])
    want = np.array(gold["mean_rgb8"])
    assert np.abs(got[0] - want[0]).max() <= 3.0            # top block row
    assert np.abs(got[:4, :4] - want[:4, :4]).mean() <= 6.0  # upper-left corner: ceiling + left wall
