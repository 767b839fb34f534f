"""The instrumented kernels (RM_FLAG_COUNT_WORK: k_setup / k_traverse<true>) against the oracle's own counters.

bench.py's roofline and the algorithmic-bytes model (DESIGN §3: C = grid cells visited, T = triangle tests) rest on these
counts, and they come from separate instantiations of the traversal kernel.  The oracle counts the same quantities for the
same rays (`cells` per cell entered, `tri_tests` per list entry of an occupied cell, acc_grid.rs:127-184), so with every
ray traced by both sides the totals must be equal, not merely close.
"""
import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import assert_hits_equal, oracle_scene, product_scene, settings

pytestmark = pytest.mark.gpu

CAM = F.camera(160, 90)
DIFFUSE = ("Diffuse", (0.8, 0.7, 0.6), 0.4)


def cube_stack() -> np.ndarray:
    """40 identical copies of the cube: every triangle is tied with 39 others at every hit, and the occupied cells hold
    80 to 240 references — many pooled rounds per cell, wrapping the traversal kernel's 64-slot survivor ring."""
    return np.concatenate([F.cube()] * 40)


def depth1_meshes() -> dict:
    return {
        "bumpy_fine": F.translate(F.bumpy_sphere(60, 120, 1.0, 0.1, (1.0, 0.7, 0.45)), (0.0, 0.0, 3.0)),   # res.y > res.z (A1)
        "dragon": F.translate(F.dragon_standin(240, 60), F.DRAGON_TRANSLATE),
        "soup200k": F.triangle_soup(200_000, F.SOUP_BOX_FLAT),
        "cube40": F.translate(cube_stack(), (0.2, -0.1, 2.5)),
    }


def gpu_render(objs, spp, bounce_limit, flags, seed=7, cam=CAM):
    r = A.Renderer(product_scene(objs), settings(cam, spp, bounce_limit=bounce_limit), A.GpuOptions(seed=seed, flags=flags))
    r.render(0, spp)
    sums = r.read_sums()
    stats, stages = r.stats(), r.stage_stats()
    r.close()
    return sums, stats, stages


def check_stage_relations(stages, what):
    """Per stage: occupied cells are cells, evaluated tests are tests, and an evaluated Triangle::intersects costs 20 to 52
    f64 operations depending on its exit (include/raymond.h)."""
    for d in range(len(stages["cells"])):
        c, t = stages["cells"][d], stages["triangle_tests"][d]
        occ, ev, fl = stages["occupied_cells"][d], stages["evaluated_tests"][d], stages["evaluated_test_flops"][d]
        assert occ <= c, f"{what} stage {d}: {occ} occupied of {c} cells"
        assert ev <= t, f"{what} stage {d}: {ev} evaluated of {t} tests"
        assert 20 * ev <= fl <= 52 * ev, f"{what} stage {d}: {fl} flops for {ev} evaluated tests"


@pytest.mark.parametrize("scene", ["gold_dragon", "reflective_spheres"])
def test_flags_do_not_change_the_frame(scene):
    """Timing, counting and the reserved flag values (8, 16, 32: accepted, no effect) leave every bit of the frame and the
    ray count as they are.  Cells and triangle tests are counted only with RM_FLAG_COUNT_WORK, and only where there is a grid."""
    has_grid = scene == "gold_dragon"
    objs = F.gold_dragon(F.dragon_standin(240, 60)) if has_grid else F.reflective_spheres()
    spp = 3
    ref, ref_stats, _ = gpu_render(objs, spp, 5, 0)
    assert ref.any()
    for flags in (A.FLAG_STAGE_TIMING, A.FLAG_COUNT_WORK, A.FLAG_NO_RAY_BINNING, A.FLAG_FUSE_SETUP, A.FLAG_SPLIT_SETUP,
                  A.FLAG_STAGE_TIMING | A.FLAG_COUNT_WORK):
        got, stats, stages = gpu_render(objs, spp, 5, flags)
        assert np.array_equal(got.view(np.uint64), ref.view(np.uint64)), f"flags {flags}: the frame changed"
        assert stats["rays"] == ref_stats["rays"] and stats["nonfinite_samples"] == ref_stats["nonfinite_samples"]
        if flags & A.FLAG_COUNT_WORK and has_grid:
            assert sum(stages["cells"]) > 0 and sum(stages["triangle_tests"]) > 0
        else:
            assert sum(stages["cells"]) == 0 and sum(stages["triangle_tests"]) == 0


@pytest.mark.parametrize("name", list(depth1_meshes()))
def test_depth1_counts_are_exact(name):
    """One grid and nothing else (so no ray skips the grid in k_setup), camera rays only: the summed cells and triangle tests
    are the oracle's exactly."""
    objs = [("grid", depth1_meshes()[name], DIFFUSE)]
    _, stats, stages = gpu_render(objs, 2, 1, A.FLAG_COUNT_WORK)
    _, oc = O.render(oracle_scene(objs), CAM, 2, seed=7, bounce_limit=1)
    assert stats["rays"] == oc["rays"] == CAM["width"] * CAM["height"] * 2
    assert sum(stages["grid_rays"]) >= oc["grid_hits"] > 0
    assert sum(stages["cells"]) == oc["cells"], f"{name}: cells {sum(stages['cells'])} vs oracle {oc['cells']}"
    assert sum(stages["triangle_tests"]) == oc["tri_tests"], f"{name}: triangle tests {sum(stages['triangle_tests'])} vs oracle {oc['tri_tests']}"
    check_stage_relations(stages, name)


def test_full_depth_counts_single_grid():
    """Every depth on one grid with a non-black Diffuse material.  With RM_FLAG_KEEP_NONFINITE no path is stopped early, so
    the GPU traces exactly the reference's rays and the totals are equal; without it, paths whose throughput became zero
    stop, and the totals can only be smaller."""
    objs = [("grid", F.translate(F.dragon_standin(240, 60), F.DRAGON_TRANSLATE), DIFFUSE)]
    spp = 2
    _, oc = O.render(oracle_scene(objs), CAM, spp, seed=7, bounce_limit=5, drop_nonfinite=False)
    _, stats, stages = gpu_render(objs, spp, 5, A.FLAG_COUNT_WORK | A.FLAG_KEEP_NONFINITE)
    assert stats["rays"] == oc["rays"] > CAM["width"] * CAM["height"] * spp
    assert sum(stages["cells"]) == oc["cells"]
    assert sum(stages["triangle_tests"]) == oc["tri_tests"]
    assert stages["cells"][2] > 0, "bounced rays should traverse the grid"
    check_stage_relations(stages, "single grid, keep")
    _, stats, stages = gpu_render(objs, spp, 5, A.FLAG_COUNT_WORK)
    assert stats["rays"] <= oc["rays"]
    assert sum(stages["cells"]) <= oc["cells"] and sum(stages["triangle_tests"]) <= oc["tri_tests"]
    check_stage_relations(stages, "single grid")


def test_full_depth_counts_gold_dragon():
    """GoldDragon: rays whose analytic hit lies before the grid's box skip the traversal, and D5 stops zero-throughput paths,
    so the GPU's totals are at most the oracle's."""
    objs = F.gold_dragon(F.dragon_standin(240, 60))
    spp = 2
    _, oc = O.render(oracle_scene(objs), CAM, spp, seed=7, bounce_limit=5)
    _, stats, stages = gpu_render(objs, spp, 5, A.FLAG_COUNT_WORK)
    assert stats["rays"] <= oc["rays"]
    assert 0 < sum(stages["cells"]) <= oc["cells"]
    assert 0 < sum(stages["triangle_tests"]) <= oc["tri_tests"]
    check_stage_relations(stages, "GoldDragon")


def test_tied_copies_first_wins():
    """40 identical cubes through Scene::intersect: bit-exact against the oracle, and every hit reports a triangle of the
    first copy (indices < 12): the strict `<` in list order keeps the earliest of equal distances."""
    objs = [("grid", F.translate(cube_stack(), (0.2, -0.1, 2.5)), DIFFUSE)]
    rays = np.concatenate([O.primary_rays(CAM),
                           F.random_rays(20_000, origin_box=((-1.0, 1.4), (-1.3, 1.1), (1.3, 3.7)))])
    want = oracle_scene(objs).intersect(rays)
    got = product_scene(objs).intersect(rays, device=0)
    assert_hits_equal(got, want, "cube x40")
    hit = want[0] >= 0
    assert hit.sum() > 4_000
    assert (got[1][hit] < 12).all()
