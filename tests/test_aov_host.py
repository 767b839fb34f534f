"""RM_FLAG_AOV on the task path (no GPU): a task cannot read the feature sums, so rm_render_tiled and rm_render_tiled_adaptive
refuse the flag before any device work."""
import pytest

from raymond_b200 import api as A
from raymond_b200 import fixtures as F

from util import settings


@pytest.mark.parametrize("adaptive", [None, A.AdaptiveSettings(0.05)], ids=["render_tiled", "render_tiled_adaptive"])
def test_task_path_refuses_the_feature_buffers(adaptive):
    with pytest.raises(A.RaymondError) as e:
        A.render_tiled(A.Scene(), settings(F.camera(8, 4), 4, spi=2), A.GpuOptions(flags=A.FLAG_AOV | A.FLAG_MOMENTS), adaptive)
    assert e.value.status == A.RM_ERR_UNSUPPORTED
    assert "RM_FLAG_AOV" in str(e.value)
