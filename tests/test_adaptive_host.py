"""CPU tests of rm_render_tiled_adaptive: its arguments are checked before any device work, so the statuses hold on a box
without a GPU, and the ctypes mirror of rm_adaptive_settings has the header's layout."""
import ctypes as C
import math
import os
import subprocess
import tempfile

import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import settings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _status_of(fn):
    with pytest.raises(A.RaymondError) as e:
        fn()
    return e.value.status


@pytest.mark.parametrize("threshold", [0.0, -0.01, math.nan, math.inf, -math.inf])
def test_bad_threshold_is_invalid_argument(threshold):
    st = settings(F.camera(32, 16), 8, spi=2)
    assert _status_of(lambda: A.render_tiled(A.Scene(), st, A.GpuOptions(), A.AdaptiveSettings(threshold))) == A.RM_ERR_INVALID_ARGUMENT


def test_zero_samples_per_iteration_is_invalid_argument():
    st = settings(F.camera(32, 16), 8, spi=0)
    assert _status_of(lambda: A.render_tiled(A.Scene(), st, A.GpuOptions(), A.AdaptiveSettings(0.05))) == A.RM_ERR_INVALID_ARGUMENT


@pytest.mark.parametrize("device_count", [0, 1])
def test_one_rank_of_a_multi_process_job_is_unsupported(device_count):
    st = settings(F.camera(32, 16), 8, spi=2)
    o = A.GpuOptions(rank=1, world_size=2, device_count=device_count)
    assert _status_of(lambda: A.render_tiled(A.Scene(), st, o, A.AdaptiveSettings(0.05))) == A.RM_ERR_UNSUPPORTED


def test_adaptive_settings_layout_matches_the_header():
    probe = r'''
    #include <stddef.h>
    #include <stdio.h>
    #include "raymond.h"
    int main(void) {
        printf("%zu %zu %zu\n", sizeof(rm_adaptive_settings), offsetof(rm_adaptive_settings, threshold), offsetof(rm_adaptive_settings, min_samples));
        return 0;
    }'''
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "probe.c")
        open(src, "w").write(probe)
        exe = os.path.join(d, "probe")
        subprocess.run(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), src, "-o", exe], check=True)
        got = [int(x) for x in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(A.AdaptiveSettingsC), A.AdaptiveSettingsC.threshold.offset, A.AdaptiveSettingsC.min_samples.offset]
