"""CPU tests of the product's host side (no GPU, no compute calls): the C-ABI library loads and exports every
symbol include/raymond.h declares; the host half of the path (Mesh::new, Mesh::load_ply, bake_transform,
AccGrid::build_from_mesh, tile layout) produces exactly what the oracle produces; failures are statuses, and a
compute call without a CUDA device is a loud error, never a CPU fallback."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import oracle as O
from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import NEEDS_REFERENCE, REFERENCE_MESHES, have_reference_assets, settings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = pytest.mark.skipif(not have_reference_assets(), reason=NEEDS_REFERENCE)


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "raymond.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = set(re.findall(r"\b(rm_[a-z0-9_]+)\s*\(", text))
    names -= {"rm_tile_callback"}          # a function-pointer typedef, not an entry point
    return sorted(names)


def test_library_exports_every_declared_symbol():
    L = A.lib()
    declared = _declared_functions()
    assert len(declared) >= 40
    missing = [n for n in declared if not hasattr(L, n)]
    assert not missing, f"libraymond_cuda.so does not export {missing}"
    assert sorted(A.ABI_SYMBOLS) == declared, "api.ABI_SYMBOLS and include/raymond.h disagree"
    assert L.rm_abi_version() == 2


def test_struct_layouts_match_the_header():
    """ctypes mirrors vs the sizes the C compiler gives include/raymond.h (checked by compiling a probe)."""
    import subprocess
    import tempfile
    probe = r'''
    #include <stdio.h>
    #include "raymond.h"
    int main(void) {
        printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(rm_triangle), sizeof(rm_material), sizeof(rm_camera_settings), sizeof(rm_settings),
               sizeof(rm_gpu_options), sizeof(rm_tile), sizeof(rm_message), sizeof(rm_stats), sizeof(rm_stage_stats), sizeof(rm_grid_info));
        return 0;
    }'''
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "probe.c")
        open(src, "w").write(probe)
        exe = os.path.join(d, "probe")
        subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        sizes = [int(x) for x in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert sizes == [264, C.sizeof(A.MaterialC), C.sizeof(A.CameraSettingsC), C.sizeof(A.SettingsC), C.sizeof(A.GpuOptionsC),
                     C.sizeof(A.TileC), C.sizeof(A.MessageC), C.sizeof(A.StatsC), C.sizeof(A.StageStatsC), C.sizeof(A.GridInfoC)]
    assert A.TRI_DOUBLES * 8 == 264            # Triangle(Vertex x3), vertex.rs:5-10


def _same_grid(tris):
    og = O.AccGrid.build_from_mesh(O.Mesh.from_triangles(tris))
    pg = A.AccGrid.build_from_mesh(A.Mesh.new(tris))
    oi, pi = og.info(), pg.info()
    assert oi["resolution"] == pi["resolution"]
    assert np.array_equal(oi["cell_size"].view(np.uint64), pi["cell_size"].view(np.uint64))
    assert np.array_equal(oi["bounds"], pi["bounds"])
    assert (oi["cell_count"], oi["reference_count"], oi["triangle_count"]) == (pi["cell_count"], pi["reference_count"], pi["triangle_count"])
    ostart, orefs = og.csr()
    pstart, prefs = pg.cells()
    assert np.array_equal(ostart, pstart) and np.array_equal(orefs, prefs)
    return pi


@pytest.mark.parametrize("name", ["cube", "bumpy", "bumpy_fine", "tube", "soup_cubic", "soup_flat"])
def test_grid_build_is_the_oracles(name):
    """AccGrid::build_from_mesh (acc_grid.rs:36-83): same resolution, cell size bits, and per-cell reference lists
    (contents AND order) as the oracle — cell contents decide which triangle a ray reports."""
    tris = {"cube": F.cube, "bumpy": F.bumpy_sphere, "bumpy_fine": lambda: F.bumpy_sphere(60, 120, 1.0, 0.1, (1.0, 0.7, 0.45)),
            "tube": lambda: F.dragon_standin(96, 24), "soup_cubic": lambda: F.triangle_soup(20000, F.SOUP_BOX_CUBIC),
            "soup_flat": lambda: F.triangle_soup(20000, F.SOUP_BOX_FLAT)}[name]()
    info = _same_grid(tris)
    if name == "cube":
        assert info["resolution"] == [3, 3, 3]
    if name in ("bumpy_fine", "soup_flat"):
        assert info["resolution"][1] > info["resolution"][2]      # the aliased regime (A1)


def test_mesh_bounds_and_translate():
    tris = F.bumpy_sphere(8, 16)
    pm, om = A.Mesh.new(tris), O.Mesh.from_triangles(tris)
    assert np.array_equal(pm.bounding_box, om.bounds)
    pm.bake_transform((0.25, -0.3, 2.9))
    om.bake_transform((0.25, -0.3, 2.9))
    assert np.array_equal(pm.bounding_box, om.bounds)
    assert np.array_equal(pm.triangles(), om.triangles())
    # empty mesh: the reference's sentinels (mesh.rs:124-125)
    assert A.Mesh.new(np.zeros((0, 33))).bounding_box.tolist() == [[125125.0, 1251251.0, 12512512.0], [-123125.0, -125123.0, -512123.0]]


def test_grid_build_errors_are_statuses():
    # zero-extent axis: res 0 -> the reference underflows `grid_res[i] - 1` (acc_grid.rs:54)
    flat = F.make_triangles(np.array([[0.0, 0, 0]]), np.array([[1.0, 0, 0]]), np.array([[0.0, 1, 0]]))
    with pytest.raises(A.RaymondError) as e:
        A.AccGrid.build_from_mesh(A.Mesh.new(flat))
    assert e.value.status == A.RM_ERR_DEGENERATE_BOUNDS
    with pytest.raises(O.OracleError) as oe:
        O.AccGrid.build_from_mesh(O.Mesh.from_triangles(flat))
    assert oe.value.status == A.RM_ERR_DEGENERATE_BOUNDS
    # a deep grid (res.z > res.y) with triangles at the far end: index out of bounds (acc_grid.rs:61 panics)
    tall = F.bumpy_sphere(20, 40, 1.0, 0.05, (0.5, 0.45, 1.6))
    with pytest.raises(A.RaymondError) as e:
        A.AccGrid.build_from_mesh(A.Mesh.new(tall))
    assert e.value.status == A.RM_ERR_GRID_INDEX_OOB
    with pytest.raises(O.OracleError) as oe:
        O.AccGrid.build_from_mesh(O.Mesh.from_triangles(tall))
    assert oe.value.status == A.RM_ERR_GRID_INDEX_OOB


def test_ply_loader_round_trip(tmp_path):
    """Mesh::load_ply (mesh.rs:58-121): ASCII, x y z nx ny nz [s t]; non-triangles dropped; same triangles as the oracle's loader."""
    tris = F.bumpy_sphere(6, 12)
    for with_uv in (False, True):
        path = str(tmp_path / f"m{int(with_uv)}.ply")
        F.write_ply(path, tris, with_uv=with_uv)
        pm, om = A.Mesh.load_ply(path), O.Mesh.load_ply(path)
        assert len(pm) == len(om) == tris.shape[0]
        pt, ot = pm.triangles(), om.triangles()
        assert np.array_equal(pt.view(np.uint64), ot.view(np.uint64))       # includes the NaN tangents when uv = 0
        assert np.allclose(F.positions(pt), F.positions(tris), rtol=0, atol=1e-6)
    # a quad face is silently dropped, a short vertex line is an error, a missing file is an IO error
    quad = tmp_path / "quad.ply"
    quad.write_text("ply\nformat ascii 1.0\nelement vertex 4\nproperty float x\nelement face 2\nend_header\n"
                    "0 0 0 0 0 1\n1 0 0 0 0 1\n1 1 0 0 0 1\n0 1 0 0 0 1\n4 0 1 2 3\n3 0 1 2\n")
    assert len(A.Mesh.load_ply(str(quad))) == len(O.Mesh.load_ply(str(quad))) == 1
    short = tmp_path / "short.ply"
    short.write_text("ply\nelement vertex 1\nend_header\n0 0 0\n")
    with pytest.raises(A.RaymondError) as e:
        A.Mesh.load_ply(str(short))
    assert e.value.status == A.RM_ERR_PLY
    with pytest.raises(A.RaymondError) as e:
        A.Mesh.load_ply(str(tmp_path / "nope.ply"))
    assert e.value.status == A.RM_ERR_IO


@needs_reference
def test_reference_ply_meshes_load_and_build_like_the_oracle():
    for name in ("cube", "ico_sphere", "monkeysmooth", "suzanne_flat"):
        path = f"{REFERENCE_MESHES}/{name}.ply"
        pm, om = A.Mesh.load_ply(path), O.Mesh.load_ply(path)
        assert np.array_equal(pm.triangles().view(np.uint64), om.triangles().view(np.uint64))
        _same_grid(om.triangles())
    # suzanne.ply: res [13,12,16] -> index out of bounds, the reference panics (SURVEY Appendix C)
    with pytest.raises(A.RaymondError) as e:
        A.AccGrid.build_from_mesh(A.Mesh.load_ply(f"{REFERENCE_MESHES}/suzanne.ply"))
    assert e.value.status == A.RM_ERR_GRID_INDEX_OOB


def test_tile_layout_is_the_references():
    for (w, h, tw, th) in ((592, 340, 32, 32), (1920, 1080, 32, 32), (100, 70, 32, 32), (64, 64, 64, 64), (65, 1, 8, 8), (7, 300, 16, 7)):
        got = A.tile_layout(settings(F.camera(w, h), 1, tile=(tw, th)))
        assert got.tolist() == O.tile_layout(F.camera(w, h), (tw, th)).tolist()
        assert got[:, 2].dot(got[:, 3]) == w * h
    assert len(A.tile_layout(settings(F.camera(1920, 1080), 1))) == 2040       # SURVEY §8 a3


def test_scene_object_order_and_materials():
    s = A.Scene.from_fixture(F.reflective_spheres())
    assert len(s) == 8
    with pytest.raises(A.RaymondError):
        m = A.MaterialC(7, 0, A.Vec3C(0, 0, 0), A.Vec3C(0, 0, 0), 0.0, 0.0)
        A._check(A.lib().rm_scene_add_sphere(s._h, A.Vec3C(0, 0, 0), 1.0, C.byref(m)))


_WITHOUT_A_DEVICE = r'''
import os, sys
sys.path[:0] = [sys.argv[1], os.path.join(sys.argv[1], "tests")]
import numpy as np
import pytest
from raymond_b200 import api as A
from raymond_b200 import fixtures as F
from util import settings
sc = A.Scene.from_fixture(F.reflective_spheres())
with pytest.raises(A.RaymondError) as e:
    sc.intersect(np.array([[0, 0, 0, 0, 0, 1.0]]))
assert e.value.status == A.RM_ERR_CUDA and "no CPU path" in str(e.value)
with pytest.raises(A.RaymondError):
    A.render_tiled(sc, settings(F.camera(8, 8), 1))
with pytest.raises(A.RaymondError):
    A.Renderer(sc, settings(F.camera(8, 8), 1))
with pytest.raises(A.RaymondError):
    A.DeviceScene(sc, 0)
with pytest.raises(A.RaymondError):
    A.measure_fp64_rate(0)
'''


def test_compute_without_a_device_is_an_error_not_a_fallback():
    """Without a CUDA device every compute entry point must fail with RM_ERR_CUDA and say so.  The checks run in a child
    process that sees no device (CUDA_VISIBLE_DEVICES empty), so they hold on machines with GPUs as well."""
    import subprocess
    import sys
    res = subprocess.run([sys.executable, "-c", _WITHOUT_A_DEVICE, ROOT], capture_output=True, text=True,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=300)
    assert res.returncode == 0, res.stderr[-3000:]


def test_product_does_not_import_the_oracle():
    """oracle/ is test infrastructure: nothing under raymond_b200/ may import, load or link it."""
    pkg = os.path.join(ROOT, "raymond_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".cuh", ".hpp", ".h")):
                text = open(os.path.join(dirpath, f), errors="replace").read()
                assert "raymond_oracle" not in text and "from oracle" not in text and "import oracle" not in text, f
