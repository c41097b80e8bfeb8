"""CPU: the GI entry points refuse a `res` (cone_trace's min_voxel_size) on which the cone march never ends, and a
float32 simulation of that march shows where the boundary lies.

For res = 0, a negative or a subnormal res the marching distance stops advancing (0.1 * diam rounds away), so every
cone of every thread would loop forever on the device.  Each entry point that takes res checks it first, before the
handle: a null handle therefore reports the res error, which pins the check without a device."""
import ctypes as C

import numpy as np
import pytest

from tests.common import CAM_MAIN, GI_KD, gi_march, gi_maxdist
from voxelraytrace20190722_b200 import capi

F32 = np.finfo(np.float32)
VRT_ERR_ARG = -1  # include/vrt.h
# -0.0078125: -gi_res of a unit cube at depth 7
BAD_RES = [0.0, -0.0, -0.0078125, 1e-45, F32.tiny / 2, float("nan"), float("inf"), float("-inf")]


def _calls(L, cam, kd, res, tree=None, mg=None):
    """Every entry point that takes res, called with `res` on the tree handle `tree` / replica set `mg` (null by
    default) and otherwise valid arguments: name -> a call returning the rc."""
    f32 = np.zeros((cam.ny, cam.nx, 3), np.float32)
    pos = np.zeros((1, 3), np.float32)
    nrm = np.array([[0, 1, 0]], np.float32)
    out = np.zeros((1, 3), np.float32)
    aov = capi.vrt_gi_aov(albedo=f32.ctypes.data)
    b = capi.vrt_bands(cam.ny, 0, 1)
    p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    cp, kp, fp, r = C.byref(cam.c), p(kd), p(f32), float(res)
    return {
        "vrt_gi_cone_trace": lambda: L.vrt_gi_cone_trace(tree, p(pos), p(nrm), 1, r, p(out)),
        "vrt_gi_render_camera": lambda: L.vrt_gi_render_camera(tree, cp, kp, r, 0, 0, cam.nx, cam.ny, fp),
        "vrt_gi_render_camera_dev": lambda: L.vrt_gi_render_camera_dev(tree, cp, kp, r, 0, 0, cam.nx, cam.ny, fp),
        "vrt_gi_render_aov": lambda: L.vrt_gi_render_aov(tree, cp, kp, r, 0, 0, cam.nx, cam.ny, fp, C.byref(aov)),
        "vrt_gi_render_aov_dev": lambda: L.vrt_gi_render_aov_dev(tree, cp, kp, r, 0, 0, cam.nx, cam.ny, fp,
                                                                 C.byref(aov)),
        "vrt_gi_render_bands_async": lambda: L.vrt_gi_render_bands_async(tree, cp, kp, r, C.byref(b), fp),
        "vrt_gi_render_aov_bands_async": lambda: L.vrt_gi_render_aov_bands_async(tree, cp, kp, r, C.byref(b), fp,
                                                                                 C.byref(aov)),
        "vrt_mgpu_gi_render": lambda: L.vrt_mgpu_gi_render(mg, cp, kp, r, fp),
        "vrt_mgpu_gi_render_async": lambda: L.vrt_mgpu_gi_render_async(mg, cp, kp, r, fp),
        "vrt_mgpu_gi_render_aov": lambda: L.vrt_mgpu_gi_render_aov(mg, cp, kp, r, fp, C.byref(aov)),
        "vrt_mgpu_gi_render_aov_async": lambda: L.vrt_mgpu_gi_render_aov_async(mg, cp, kp, r, fp, C.byref(aov)),
    }


def res_refused(L, call):
    """(rc, message) of one call, and whether it is the res refusal."""
    rc = call()
    msg = L.vrt_last_error().decode(errors="replace")
    return rc, msg, rc == VRT_ERR_ARG and msg.startswith("res ")


@pytest.mark.parametrize("res", BAD_RES)
def test_every_gi_entry_refuses_res_without_a_march(res):
    L = capi.load()
    res = np.float32(res)
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], 8, 4, 1)
    calls = _calls(L, cam, GI_KD, res)
    assert len(calls) == 11
    for name, call in calls.items():
        rc, msg, ok = res_refused(L, call)
        assert ok, f"{name}(res={res!r}) -> {rc} '{msg}', not the res refusal"
        assert "FLT_MIN" in msg
    # a valid res passes the check and fails on the null handle instead
    calls = _calls(L, cam, GI_KD, np.float32(0.0078125))
    for name, call in calls.items():
        rc, msg, ok = res_refused(L, call)
        assert rc != 0 and not ok, f"{name}: a valid res is refused ('{msg}')"


def test_march_ends_exactly_for_normal_res():
    """The march ends in well under 2,000 steps for res = FLT_MIN whatever the root box, and does not advance at all
    for 0, a negative or the smallest subnormal res; the steps of the cases the GPU tests rely on."""
    tiny = np.float32(F32.tiny)
    for maxdist in (np.float32(1e-30), np.float32(1e-3), np.float32(3.4641016), np.float32(1e20), F32.max,
                    np.float32(np.inf)):
        lv, ended = gi_march(maxdist, tiny)
        assert ended and 0 < len(lv) < 2000, (maxdist, len(lv))
    for res in (0.0, -0.0, -1e-3, 1e-45):
        lv, ended = gi_march(np.float32(3.4641016), np.float32(res))
        assert not ended and len(lv) == 1, res
    # cube root box of edge 2 (maxdist 2 sqrt 3): the steps quoted in include/vrt.h and the GPU tests
    md = gi_maxdist([-1, -1, -1, 1, 1, 1])
    assert md == np.sqrt(np.float32(12), dtype=np.float32)
    steps = {r: len(gi_march(md, np.float32(r))[0]) for r in (4.2e-45, F32.tiny, 1e-30, 1e-24, 2.0 ** -9, 3.0)}
    assert steps == {4.2e-45: 941, F32.tiny: 807, 1e-30: 640, 1e-24: 513, 2.0 ** -9: 64, 3.0: 0}
    assert len(gi_march(np.float32(np.inf), tiny)[0]) == 1608 and len(gi_march(F32.max, tiny)[0]) == 1607
    # NaN and inf end at once: the device would return zeros, they are refused as never meant
    for res in (np.nan, np.inf):
        assert gi_march(md, np.float32(res)) == ([], True)
