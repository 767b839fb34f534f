"""CPU: every fixture of shading_space.py reaches the regime it is there for, so that none of the GPU comparisons of
test_gpu_shading_space.py turns into comparing 0 with 0."""
import os

import numpy as np
import pytest

from oracle import oracle as O

from shading_space import FIXTURES, SEED, SPP, origin_camera, tagged
from util import oracle_scene

THREADS = os.cpu_count() or 8


def oracle_sums(name, cam=None, keep=False):
    fx = FIXTURES[name]
    return O.render(oracle_scene(fx.objs), cam or fx.cam, SPP, seed=SEED, bounce_limit=fx.limit, drop_nonfinite=not keep, worker_count=THREADS)


@pytest.mark.parametrize("name", tagged("nonfinite"))
def test_roughness_0_gives_nonfinite_samples(name):
    sums, cnt = oracle_sums(name, keep=True)
    assert cnt["nonfinite"] >= 0.01 * cnt["samples"], f"{name}: {cnt['nonfinite']} non-finite samples of {cnt['samples']}"
    assert np.isnan(sums).any()


@pytest.mark.parametrize("name", tagged("negative"))
def test_negative_colours_give_negative_path_values(name):
    fx = FIXTURES[name]
    osc = oracle_scene(fx.objs)
    per_sample = np.stack([O.render(osc, fx.cam, 1, seed=SEED, first_sample=s, bounce_limit=fx.limit, worker_count=THREADS)[0] for s in range(SPP)])
    assert (per_sample < 0).sum() >= 100, f"{name}: {(per_sample < 0).sum()} negative path channels"


@pytest.mark.parametrize("name", tagged("bright"))
def test_non_unit_normals_give_bright_paths(name):
    fx = FIXTURES[name]
    osc = oracle_scene(fx.objs)
    per_sample = np.stack([O.render(osc, fx.cam, 1, seed=SEED, first_sample=s, bounce_limit=fx.limit, worker_count=THREADS)[0] for s in range(SPP)])
    assert per_sample.max() > 100.0


@pytest.mark.parametrize("name", tagged("camera"))
def test_camera_fixture_sees_another_frame(name):
    fx = FIXTURES[name]
    got, _ = oracle_sums(name)
    base, _ = oracle_sums(name, cam=origin_camera(fx.cam))
    assert got.any()
    assert not np.array_equal(got, base), f"{name}: the same frame as the origin camera's"


@pytest.mark.parametrize("name", tagged("shape"))
def test_frame_shape_fixture_is_not_uniform(name):
    got, _ = oracle_sums(name)
    luma = got.sum(axis=-1)
    assert len(np.unique(luma)) > luma.size // 4, f"{name}: {len(np.unique(luma))} distinct pixel values of {luma.size}"


def test_fixture_table_covers_the_regimes():
    for tag in ("nonfinite", "negative", "bright", "camera", "shape", "f32", "last_bounce"):
        assert tagged(tag), tag
