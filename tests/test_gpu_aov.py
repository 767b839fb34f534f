"""First-hit feature buffers (RM_FLAG_AOV) against the oracle on the same random stream.

Every sample's camera ray (oracle.camera_rays, depth of field included) goes through the oracle's Scene::intersect and its
shading normal; albedo is the hit object's material colour, depth the hit distance, a miss adds zeros.  Summed in sample order,
the depth and albedo sums are the library's to the bit, and the normal sums agree within 1e-9 relative.
"""
import functools

import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import oracle_scene, product_scene, settings

pytestmark = pytest.mark.gpu

SEED, SPP, BATCH = 11, 4, 3          # two batches per render
TILE = (16, 16)
SETUPS = {
    "spheres_c1": (F.reflective_spheres(), F.camera(160, 120)),
    "spheres_dof": (F.reflective_spheres(), F.camera(120, 80, focal_length=2.5, aperture_radius=0.5)),       # the C3 camera
    "dragon_standin": (F.gold_dragon(F.dragon_standin(96, 24)), F.camera(96, 64)),
}


@functools.lru_cache(maxsize=None)
def oracle_aovs(name, first=0, count=SPP):
    """Sums over samples first .. first+count-1 of albedo (H, W, 3), normal (H, W, 3) and depth (H, W)."""
    objs, cam = SETUPS[name]
    osc = oracle_scene(objs)
    colour = np.array([(o[2] if o[0] == "grid" else o[3])[1] for o in objs], dtype=np.float64)
    W, H = cam["width"], cam["height"]
    sa, sn, sz = np.zeros((H * W, 3)), np.zeros((H * W, 3)), np.zeros(H * W)
    for s in range(first, first + count):
        rays = O.camera_rays(cam, SEED, s)
        obj, sub, t, _ = osc.intersect(rays)
        a, n, z = np.zeros((H * W, 3)), np.zeros((H * W, 3)), np.zeros(H * W)
        hit = obj >= 0
        a[hit] = colour[obj[hit]]
        z[hit] = t[hit]
        for i in np.nonzero(hit)[0]:
            n[i] = osc.normal(rays[i], obj[i], sub[i], t[i])
        sa, sn, sz = sa + a, sn + n, sz + z
    return sa.reshape(H, W, 3), sn.reshape(H, W, 3), sz.reshape(H, W)


def renderer(name, flags=A.FLAG_AOV, limit=5, **opt):
    objs, cam = SETUPS[name]
    return A.Renderer(product_scene(objs), settings(cam, SPP, TILE, bounce_limit=limit), A.GpuOptions(seed=SEED, batch_spp=BATCH, flags=flags, **opt))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def assert_normals_close(g, o, what):
    assert np.array_equal(np.isnan(g), np.isnan(o)), f"{what}: NaN elements differ"
    fin = np.isfinite(o)
    err = np.abs(g[fin] - o[fin]) / np.maximum(np.abs(o[fin]), 1e-3)
    print(f"{what}: largest relative normal difference {err.max():.3g}")
    assert err.max() <= 1e-9, f"{what}: normal sums differ by {err.max():.3g} relative"


@pytest.mark.parametrize("limit", [5, 1])
@pytest.mark.parametrize("name", list(SETUPS))
def test_aovs_are_the_oracles(name, limit):
    """bounce_limit 1 makes depth 1 the last depth, where drop mode would skip the grid for rays whose closest analytic hit is not
    an emitter: with the flag set it must not."""
    r = renderer(name, limit=limit)
    r.render(0, SPP)
    ga, gn, gz = r.read_aovs(1)
    r.close()
    oa, on, oz = oracle_aovs(name)
    assert np.array_equal(bits(gz), bits(oz)), f"{name}: {int((bits(gz) != bits(oz)).sum())} depth sums differ in their bits"
    assert np.array_equal(bits(ga), bits(oa)), f"{name}: {int((bits(ga) != bits(oa)).sum())} albedo sums differ in their bits"
    assert_normals_close(gn, on, name)
    assert (oz > 0).mean() > 0.9
    # read_aovs divides by sample_count
    r = renderer(name, limit=limit)
    r.render(0, SPP)
    ma, mn, mz = r.read_aovs(SPP)
    r.close()
    assert np.array_equal(bits(ma), bits(oa / SPP)) and np.array_equal(bits(mz), bits(oz / SPP))


@pytest.mark.parametrize("limit", [1, 5])
def test_sums_unchanged_by_the_flag(limit):
    """S, Q, rays and the per-stage statistics are bit-identical with and without RM_FLAG_AOV; k_aov adds one launch per batch.
    At bounce_limit 1 the flag turns off the last-depth grid skip of stage 1, so more of its rays enter the grid there."""
    out = {}
    for flags in (A.FLAG_MOMENTS, A.FLAG_MOMENTS | A.FLAG_AOV):
        r = renderer("dragon_standin", flags=flags, limit=limit)
        r.render(0, SPP)
        out[flags] = (r.read_sums(), r.read_moments(), r.stats(), r.stage_stats())
        r.close()
    (S0, Q0, st0, ss0), (S1, Q1, st1, ss1) = out.values()
    assert np.array_equal(bits(S0), bits(S1)) and np.array_equal(bits(Q0), bits(Q1))
    assert (st0["samples"], st0["rays"], st0["nonfinite_samples"]) == (st1["samples"], st1["rays"], st1["nonfinite_samples"])
    assert st1["kernel_launches"] == st0["kernel_launches"] + -(-SPP // BATCH)
    assert ss0["launches"] == ss1["launches"] and not any(ss1["launches"]["bin"])
    assert ss0["rays"] == ss1["rays"] and ss0["shaded_triangles"] == ss1["shaded_triangles"]
    if limit == 1:
        assert ss1["grid_rays"][1] > ss0["grid_rays"][1] and ss1["grid_rays"][2:] == ss0["grid_rays"][2:]
    else:
        assert ss0["grid_rays"] == ss1["grid_rays"]


def test_tile_partition_and_active_tiles():
    """A tile share holds the full renderer's sums on its own tiles and zeros elsewhere; after set_active_tiles only the active
    tiles take the later samples."""
    name = "spheres_c1"
    full = renderer(name)
    full.render(0, SPP)
    fa, fn, fz = full.read_aovs(1)
    full.close()
    part = renderer(name, rank=1, world_size=2, partition=A.PARTITION_TILES)
    part.render(0, SPP)
    pa, pn, pz = part.read_aovs(1)
    layout = A.tile_layout(part.settings)
    part.close()
    owned = np.zeros(fz.shape, bool)
    for t, (l, top, w, h) in enumerate(layout):
        owned[top:top + h, l:l + w] = t % 2 == 1
    for g, f in ((pa, fa), (pn, fn), (pz, fz)):
        assert np.array_equal(bits(g[owned]), bits(f[owned]))
        assert not g[~owned].any()

    active = np.arange(len(layout)) % 3 == 0
    r = renderer(name)
    r.render(0, 2)
    r.set_active_tiles(active)
    r.render(2, SPP - 2)
    ra, rn, rz = r.read_aovs(1)
    r.close()
    first = renderer(name)
    first.render(0, 2)
    ea, en, ez = first.read_aovs(1)
    first.close()
    on = np.zeros(fz.shape, bool)
    for t, (l, top, w, h) in enumerate(layout):
        on[top:top + h, l:l + w] = active[t]
    for g, f, e in ((ra, fa, ea), (rn, fn, en), (rz, fz, ez)):
        assert np.array_equal(bits(g[on]), bits(f[on]))
        assert np.array_equal(bits(g[~on]), bits(e[~on]))


def test_clear_and_state():
    r = renderer("spheres_c1")
    r.render(0, SPP)
    assert r.read_aovs(1)[2].any()
    r.clear()
    assert not any(a.any() for a in r.read_aovs(1))
    r.render(0, SPP)
    oa, on, oz = oracle_aovs("spheres_c1")
    assert np.array_equal(bits(r.read_aovs(1)[2]), bits(oz))
    with pytest.raises(A.RaymondError) as e:
        r.read_aovs(0)
    assert e.value.status == A.RM_ERR_INVALID_ARGUMENT
    r.close()

    r = renderer("spheres_c1", flags=A.FLAG_MOMENTS)
    r.render(0, 1)
    with pytest.raises(A.RaymondError) as e:
        r.read_aovs(1)
    assert e.value.status == A.RM_ERR_STATE
    r.close()


def test_no_depth_one_stage_leaves_zeros():
    r = renderer("spheres_c1", limit=0)
    r.render(0, SPP)
    assert not any(a.any() for a in r.read_aovs(1))
    r.close()
