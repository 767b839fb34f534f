"""Several shares of a frame driven from ONE process through the C ABI (rm_gpu_options.device_count / device_list): samples
or tiles are split between the devices, the scene crosses the bus once in slices (one per share) and is gathered device to
device, and the accumulators are combined over peer memory.  The device list may name an ordinal more than once, so the whole
data path — sliced upload + gather, peer reduce, progressive tiles — runs on a 1-GPU box too; with >= 2 GPUs (gpurun --gpus 2) the same tests also use real peers."""
import numpy as np
import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from conftest import cuda_device_count
from util import product_scene, settings

pytestmark = pytest.mark.gpu


def device_lists():
    """[0, 0] (two shares on one GPU), three shares, 65 (more than one exchange kernel takes: the staged exchange), and — when
    the box has them — distinct GPUs."""
    lists = [[0, 0], [0, 0, 0], [0] * 65]
    n = cuda_device_count()
    if n >= 2:
        lists += [[0, 1], [1, 0, 1]]
    if n >= 4:
        lists += [[0, 1, 2, 3]]
    return lists


@pytest.mark.parametrize("devices", device_lists(), ids=lambda d: "gpus" + "".join(map(str, d)))
@pytest.mark.parametrize("partition", [A.PARTITION_SAMPLES, A.PARTITION_TILES])
def test_device_list_matches_one_device(partition, devices):
    objs, cam, spp = F.gold_dragon(F.dragon_standin(160, 40)), F.camera(160, 96), 7
    st = settings(cam, spp, spi=3)
    one = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=5))
    ref = one.await_()
    many = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=5, device_list=devices, partition=partition))
    stats = many.stats()
    msgs = []
    while (m := many.poll()) is not None:
        msgs.append(m)
    assert stats["samples"] == 160 * 96 * spp
    prog = sorted({m.tile.sample_count for m in msgs if m.kind == "TileProgressed"})
    assert prog == [3, 6]
    layout = A.tile_layout(st)
    assert len([m for m in msgs if m.kind == "TileFinished"]) == len(layout)
    assert len([m for m in msgs if m.kind == "TileProgressed"]) == 2 * len(layout)
    got = np.zeros_like(ref)
    for m in msgs:
        if m.kind == "TileFinished":
            t = m.tile
            got[t.top:t.top + t.height, t.left:t.left + t.width] = t.data / t.sample_count
    if partition == A.PARTITION_TILES:
        assert np.array_equal(got, ref)                        # disjoint tiles: identical sums
    else:
        assert np.allclose(got, ref, rtol=1e-12, atol=1e-12)   # same samples, different association across devices
    # await() of a second task gives the same frame
    again = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=5, device_list=devices, partition=partition)).await_()
    assert np.array_equal(again, got)


def test_progressive_tiles_are_running_sums_of_all_devices():
    """TileProgressed (src/trace.rs:214-219) with several devices: the tile at checkpoint k holds the first k samples of ALL shares."""
    objs, cam, spp = F.reflective_spheres(), F.camera(96, 64), 8
    st = settings(cam, spp, spi=4)
    task = A.render_tiled(product_scene(objs), st, A.GpuOptions(seed=3, device_list=[0, 0]))
    task.stats()
    half = A.Renderer(product_scene(objs), settings(cam, 4), A.GpuOptions(seed=3))
    half.render(0, 4)
    want = half.read_sums()
    half.close()
    seen = 0
    while (m := task.poll()) is not None:
        if m.kind == "TileProgressed":
            t = m.tile
            assert t.sample_count == 4
            assert np.allclose(t.data, want[t.top:t.top + t.height, t.left:t.left + t.width], rtol=1e-12, atol=1e-12)
            seen += 1
    assert seen == len(A.tile_layout(st))


def test_device_count_rejects_single_device_options():
    sc = product_scene(F.reflective_spheres())
    with pytest.raises(A.RaymondError) as e:
        A.render_tiled(sc, settings(F.camera(16, 16), 2), A.GpuOptions(device_count=2, device_list=[0, 0], world_size=2, rank=0))
    assert e.value.status == A.RM_ERR_INVALID_ARGUMENT
    with pytest.raises(A.RaymondError) as e:
        A.render_tiled(sc, settings(F.camera(16, 16), 2), A.GpuOptions(device_count=64))
    assert e.value.status == A.RM_ERR_CUDA
    with pytest.raises(A.RaymondError) as e:
        A.render_tiled(sc, settings(F.camera(16, 16), 2), A.GpuOptions(device_list=[0, 99]))
    assert e.value.status == A.RM_ERR_CUDA
