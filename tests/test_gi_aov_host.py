"""CPU: the GI planes entry points (vrt_gi_render_aov) -- struct layout, and no CPU fallback without a device."""
import ctypes

import numpy as np
import pytest

from tests.common import CAM_MAIN, GI_KD
from voxelraytrace20190722_b200 import capi


def test_gi_aov_layout_matches_header():
    assert ctypes.sizeof(capi.vrt_gi_aov) == 40
    assert [f for f, _ in capi.vrt_gi_aov._fields_] == list(capi.GI_AOV_PLANES)
    assert capi.vrt_gi_aov.hits.offset == 32


def test_gi_render_aov_without_device_raises():
    capi.load()
    if capi.device_count() > 0:
        pytest.skip("CUDA device present")
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], 8, 4, 1)
    tree = capi.Octree(None)  # no device: no octree can be built, and the entry point must not compute anything
    with pytest.raises(capi.VrtError):
        tree.gi_render_aov(cam, GI_KD, np.float32(0.01))
    with pytest.raises(capi.VrtError):
        tree.gi_render_aov_dev(cam, GI_KD, np.float32(0.01), 0, {"albedo": 16})
    with pytest.raises(ValueError):
        tree.gi_render_aov(cam, GI_KD, np.float32(0.01), planes=("albedo", "depth"))
