"""CPU: the banded and multi-GPU GI plane entry points (vrt_gi_render_aov_bands_async, vrt_mgpu_gi_render_aov*) --
no CPU fallback without a device, and plane names checked before the library is called."""
import numpy as np
import pytest

from tests.common import CAM_MAIN, GI_KD
from voxelraytrace20190722_b200 import capi


def _handles():
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], 8, 4, 1)
    tree = capi.Octree(None)  # without a device no octree or replica can be made
    mg = capi.MultiGpu.__new__(capi.MultiGpu)
    mg._h = None
    return cam, tree, mg


def test_gi_plane_frames_without_device_raise():
    capi.load()
    if capi.device_count() > 0:
        pytest.skip("CUDA device present")
    cam, tree, mg = _handles()
    res = np.float32(0.01)
    with pytest.raises(capi.VrtError):
        tree.gi_render_aov_bands_async(cam, GI_KD, res, 0, {"albedo": 16}, 8, 0, 1)
    with pytest.raises(capi.VrtError):
        mg.gi_render_aov_async(cam, GI_KD, res, 0, {"albedo": 16})
    with pytest.raises(capi.VrtError):
        mg.gi_render_aov(cam, GI_KD, res, 0, {"hits": 16})


def test_gi_plane_frames_reject_unknown_planes():
    cam, tree, mg = _handles()
    res = np.float32(0.01)
    with pytest.raises(ValueError):
        tree.gi_render_aov_bands_async(cam, GI_KD, res, 0, {"albedo": 16, "depth": 32}, 8, 0, 1)
    with pytest.raises(ValueError):
        mg.gi_render_aov_async(cam, GI_KD, res, 0, {"depth": 16})
    with pytest.raises(ValueError):
        mg.gi_render_aov(cam, GI_KD, res, 0, {"film": 16})
