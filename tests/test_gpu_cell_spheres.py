"""Cell spheres in k_traverse (DESIGN §3.1): the lane that reaches an occupied cell tests one bounding sphere around the
reference spheres of the cell's list, and a ray whose line provably misses it skips the cell's list.  The cull is exact, so
with and without it (RM_NO_CELL_SPHERES=1 in the environment when the scene is placed) frames, statistics and the per-stage
cells, tests and survivors are the same to the last bit.  The host-side test checks the sphere rule, restated in numpy.
"""
import os
import sys

import numpy as np
import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import product_scene, settings

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
from ref_group_census import group_spheres  # noqa: E402
from cover_census import spheres  # noqa: E402

SEED = 2026
WHOLE_CELL = 1 << 30          # a group as long as any cell's list: one sphere per occupied cell


def bits_equal(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def render(make_scene, cam, spp, monkeypatch, on, flags):
    if on:
        monkeypatch.delenv("RM_NO_CELL_SPHERES", raising=False)
    else:
        monkeypatch.setenv("RM_NO_CELL_SPHERES", "1")
    r = A.Renderer(make_scene(), settings(cam, spp), A.GpuOptions(seed=SEED, flags=flags))
    r.render(0, spp)
    out = r.read_sums(), r.stats(), r.stage_stats()
    r.close()
    monkeypatch.delenv("RM_NO_CELL_SPHERES", raising=False)
    return out


def compare(make_scene, cam, spp, monkeypatch, keep=False):
    for flags in (0, A.FLAG_COUNT_WORK):
        flags |= A.FLAG_KEEP_NONFINITE if keep else 0
        (s1, st1, ss1), (s0, st0, ss0) = (render(make_scene, cam, spp, monkeypatch, on, flags) for on in (True, False))
        assert bits_equal(s1, s0), f"flags {flags}: the frames differ"
        for k in ("rays", "samples", "nonfinite_samples"):
            assert st1[k] == st0[k], (flags, k)
        for k in ("rays", "grid_rays", "cells", "triangle_tests", "evaluated_tests", "occupied_cells", "shaded_triangles"):
            assert ss1[k] == ss0[k], (flags, k)
        if flags & A.FLAG_COUNT_WORK:
            assert not any(ss0["cell_sphere_tests"])
            assert ss1["cell_sphere_tests"] == ss1["occupied_cells"], "every occupied cell a ray reaches is tested"


@pytest.mark.gpu
def test_gold_dragon(monkeypatch):
    compare(lambda: product_scene(F.gold_dragon(F.dragon_standin())), F.camera(160, 90), 4, monkeypatch)


@pytest.mark.gpu
def test_soup(monkeypatch):
    compare(lambda: product_scene(F.soup_scene(F.triangle_soup(100_000, F.SOUP_BOX_CUBIC))), F.camera(160, 90), 2, monkeypatch)


@pytest.mark.gpu
@pytest.mark.parametrize("keep", [False, True], ids=["drop", "keep"])
@pytest.mark.parametrize("name", ["nobox", "box", "sliver"])
def test_nonfinite_fixtures(name, keep, monkeypatch):
    from test_gpu_nonfinite import CAM, scenes
    compare(lambda: product_scene(scenes()[name]), CAM, 4, monkeypatch, keep=keep)


def test_cell_sphere_rule_on_a_small_mesh():
    """One sphere per occupied cell; every member sphere lies inside it with the (1 + 2e-6) margin; a member with an
    infinite radius makes its cell's infinite."""
    from oracle import oracle as O
    tris = F.translate(F.dragon_standin(48, 12), F.DRAGON_TRANSLATE)
    start, refs = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(tris)).csr()
    start, refs = start.astype(np.int64), refs.astype(np.int64)
    tc, tR = spheres(np.asarray(F.positions(tris), dtype=np.float64))
    c, R = tc[refs], tR[refs].copy()
    inf_at = int(start[np.flatnonzero(np.diff(start) > 1)[0]]) + 1
    R[inf_at] = np.inf
    cg, rg, first, gbase = group_spheres(c, R, start, WHOLE_CELL)
    occupied = np.flatnonzero(np.diff(start) > 0)
    assert np.array_equal(first, start[occupied]), "one sphere per occupied cell, at its first reference"
    assert np.array_equal(cg.astype(np.float32).astype(np.float64), cg) and np.array_equal(rg.astype(np.float32).astype(np.float64), rg)
    member = np.repeat(np.arange(first.size), np.diff(start)[occupied])
    fin = np.isfinite(rg[member])
    reach = np.sqrt(((cg[member] - c) ** 2).sum(1)) + R
    assert (rg[member][fin] >= reach[fin] * (1.0 + 2e-6)).all()
    assert np.isinf(rg[member[inf_at]]) and np.isfinite(rg).sum() == rg.size - 1
