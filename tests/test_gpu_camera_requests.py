"""GPU: the return code of every camera entry point for every malformed request that applies to it, and that a refused
or empty request launches nothing (vrt_launch_count does not move).

The entry points differ in where the empty-request return sits among the argument checks, and these tables pin each
one's answer: the rectangle and banded forms return VRT_OK for an empty request before they look at the outputs, the
one-shot GI forms (vrt_gi_render_camera*, vrt_gi_render_aov*) refuse a missing output, kd or GI state even then.  The
vrt_mgpu_* forms run on a replica set of one device repeated three times."""
import ctypes as C

import numpy as np
import pytest

from tests.common import CAM_MAIN, CAM_LIGHT, GI_KD, gi_res
from voxelraytrace20190722_b200 import scenes

pytestmark = pytest.mark.gpu
OK, ARG = 0, -1  # include/vrt.h
NX, NY, SPP, BAND_H = 16, 16, 4, 8
BUF = NX * NY * SPP * 48  # bytes: enough for any output of this camera

RECT = {"vrt_trace_camera", "vrt_trace_camera_dev", "vrt_trace_camera16_dev", "vrt_render_camera",
        "vrt_render_camera_dev", "vrt_render_camera_async", "vrt_gi_render_camera", "vrt_gi_render_camera_dev",
        "vrt_gi_render_aov", "vrt_gi_render_aov_dev"}
BANDS = {"vrt_render_bands_dev", "vrt_trace_bands16_dev", "vrt_render_bands_async", "vrt_gi_render_bands_async",
         "vrt_gi_render_aov_bands_async", "vrt_frame_bands_dev", "vrt_frame_bands_peer_dev"}
MGPU = {"vrt_mgpu_render_async", "vrt_mgpu_render", "vrt_mgpu_gi_render_async", "vrt_mgpu_gi_render",
        "vrt_mgpu_gi_render_aov_async", "vrt_mgpu_gi_render_aov"}
SHADE = {"vrt_render_camera", "vrt_render_camera_dev", "vrt_render_camera_async", "vrt_render_bands_dev",
         "vrt_render_bands_async", "vrt_frame_bands_dev", "vrt_frame_bands_peer_dev", "vrt_mgpu_render_async",
         "vrt_mgpu_render"}
AOV = {"vrt_gi_render_aov", "vrt_gi_render_aov_dev", "vrt_gi_render_aov_bands_async", "vrt_mgpu_gi_render_aov_async",
       "vrt_mgpu_gi_render_aov"}
GI = AOV | {"vrt_gi_render_camera", "vrt_gi_render_camera_dev", "vrt_gi_render_bands_async",
            "vrt_mgpu_gi_render_async", "vrt_mgpu_gi_render"}
ONE_SHOT_GI = GI & RECT
FRAME = {"vrt_frame_bands_dev", "vrt_frame_bands_peer_dev"}
ENTRIES = sorted(RECT | BANDS | MGPU)
# these two used to launch the cone-trace step table before they refused a rectangle outside the film or returned for
# an empty one: test_refused_gi_film_launches_nothing
STEP_TABLE = {"vrt_gi_render_camera", "vrt_gi_render_camera_dev"}
STEP_TABLE_CASES = {"rect outside the film", "rect with a negative corner", "rect with x1 < x0", "empty rect"}


@pytest.fixture(scope="module")
def env(gpu):
    import torch
    L = gpu.load()
    tri, nrm = scenes.atrium(detail=0.3)
    depth = 6
    tree = gpu.Octree.build(tri, nrm, depth)
    lcam = gpu.Camera(CAM_LIGHT[0], CAM_LIGHT[1:4], CAM_LIGHT[4:7], CAM_LIGHT[7:10], 64, 64, 4)

    def lit(h):
        h.gi_init()
        h.gi_splat(lcam, GI_KD)
        h.gi_filter()
        return h

    lit(tree)
    unlit = gpu.Octree.from_blob_dev(*tree.blob_dev())
    mg = lit(gpu.MultiGpu(tree, [0, 0, 0]))
    mg_unlit = gpu.MultiGpu(tree, [0, 0, 0])
    cam = gpu.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], NX, NY, SPP)
    host = [torch.zeros(BUF, dtype=torch.uint8).pin_memory() for _ in range(7)]
    dev = [torch.zeros(BUF, dtype=torch.uint8, device="cuda") for _ in range(7)]
    torch.cuda.synchronize()
    kd = np.ascontiguousarray(GI_KD)
    yield dict(L=L, tree=tree, unlit=unlit, mg=mg, mg_unlit=mg_unlit, cam=cam, host=host, dev=dev, kd=kd,
               res=float(gi_res(tree.info()["root_aabb"], depth)), shade=gpu._shade(None, 0.8, 0.0), gpu=gpu)
    for h in (mg_unlit, mg, unlit, tree):
        h.close()


def _args(env, name):
    """The valid arguments of entry point `name`."""
    mgpu = name in MGPU
    bufs = env["dev"] if name.endswith("_dev") else env["host"]
    ptr = [C.c_void_p(b.data_ptr()) for b in bufs]
    return dict(h=(env["mg"] if mgpu else env["tree"])._h, cam=C.byref(env["cam"].c), rect=(0, 0, NX, NY),
                b=env["gpu"].vrt_bands(BAND_H, 0, 2), out=ptr[0], out2=ptr[1], sh=C.byref(env["shade"]),
                kd=env["kd"].ctypes.data_as(C.c_void_p), res=env["res"],
                aov=env["gpu"].vrt_gi_aov(*(p.value for p in ptr[2:7])), aov_null=False)


def _call(L, name, a):
    h, cam, out, out2, sh, kd, res = a["h"], a["cam"], a["out"], a["out2"], a["sh"], a["kd"], a["res"]
    r = a["rect"]
    b = None if a["b"] is None else C.byref(a["b"])
    aov = None if a["aov_null"] else C.byref(a["aov"])
    fn = getattr(L, name)
    if name in ("vrt_trace_camera", "vrt_trace_camera_dev", "vrt_trace_camera16_dev"):
        return fn(h, cam, *r, out)
    if name in ("vrt_render_camera", "vrt_render_camera_dev", "vrt_render_camera_async"):
        return fn(h, cam, sh, *r, out)
    if name in ("vrt_gi_render_camera", "vrt_gi_render_camera_dev"):
        return fn(h, cam, kd, res, *r, out)
    if name in ("vrt_gi_render_aov", "vrt_gi_render_aov_dev"):
        return fn(h, cam, kd, res, *r, out, aov)
    if name in ("vrt_render_bands_dev", "vrt_render_bands_async"):
        return fn(h, cam, sh, b, out)
    if name == "vrt_trace_bands16_dev":
        return fn(h, cam, b, out)
    if name == "vrt_gi_render_bands_async":
        return fn(h, cam, kd, res, b, out)
    if name == "vrt_gi_render_aov_bands_async":
        return fn(h, cam, kd, res, b, out, aov)
    if name in FRAME:
        return fn(h, cam, sh, b, out, out2)
    if name in ("vrt_mgpu_render_async", "vrt_mgpu_render"):
        return fn(h, cam, sh, out)
    if name in ("vrt_mgpu_gi_render_async", "vrt_mgpu_gi_render"):
        return fn(h, cam, kd, res, out)
    assert name in ("vrt_mgpu_gi_render_aov_async", "vrt_mgpu_gi_render_aov")
    return fn(h, cam, kd, res, out, aov)


def _cases(env, name):
    """(what, argument overrides, expected rc) of every malformed or empty request that applies to `name`."""
    gpu = env["gpu"]
    empty = (3, 2, 3, NY)
    c = [("null handle", dict(h=None), ARG), ("null camera", dict(cam=None), ARG)]
    out = "aov_null" if name in AOV else "out"
    null_out = {out: True} if out == "aov_null" else {out: None}
    if name in RECT:
        c += [("rect outside the film", dict(rect=(0, 0, NX + 1, NY)), ARG),
              ("rect with a negative corner", dict(rect=(-1, 0, NX, NY)), ARG),
              ("rect with x1 < x0", dict(rect=(5, 0, 4, NY)), ARG),
              ("empty rect", dict(rect=empty), OK),
              ("empty rect, null output", dict(rect=empty, **null_out), ARG if name in ONE_SHOT_GI else OK)]
        if name in SHADE:
            c += [("empty rect, null shade", dict(rect=empty, sh=None), OK)]
        if name in ONE_SHOT_GI:
            c += [("empty rect, handle without vrt_gi_init", dict(rect=empty, h=env["unlit"]._h), ARG),
                  ("empty rect, null kd", dict(rect=empty, kd=None), ARG)]
    if name in BANDS:
        no_rows = gpu.vrt_bands(BAND_H, NY // BAND_H, 1)
        c += [(f"bands {bb}", dict(b=gpu.vrt_bands(*bb)), ARG)
              for bb in ((0, 0, 1), (-1, 0, 1), (BAND_H, 0, 0), (BAND_H, 0, -2), (BAND_H, -1, 1))]
        # the pipelined GI forms check kd and the planes before the handle, the rest of the request after the rows
        c += [("null bands", dict(b=None), ARG), ("no rows", dict(b=no_rows), OK),
              ("no rows, null output", dict(b=no_rows, **null_out), ARG if name in AOV else OK)]
        if name in SHADE:
            c += [("no rows, null shade", dict(b=no_rows, sh=None), OK)]
        if name in GI:
            c += [("no rows, handle without vrt_gi_init", dict(b=no_rows, h=env["unlit"]._h), OK),
                  ("no rows, null kd", dict(b=no_rows, kd=None), ARG)]
        if name in AOV:
            c += [("no rows, every plane NULL", dict(b=no_rows, aov=gpu.vrt_gi_aov()), ARG)]
    c += [("null output", null_out, ARG)]
    if name in FRAME:
        c += [("null film", dict(out2=None), ARG)]
    if name in SHADE:
        c += [("null shade", dict(sh=None), ARG)]
    if name in GI:
        c += [("handle without vrt_gi_init", dict(h=(env["mg_unlit"] if name in MGPU else env["unlit"])._h), ARG),
              ("null kd", dict(kd=None), ARG), ("res 0", dict(res=0.0), ARG), ("res NaN", dict(res=float("nan")), ARG),
              ("res 0, null handle", dict(res=0.0, h=None), ARG)]
    if name in AOV:
        c += [("every plane NULL", dict(aov=gpu.vrt_gi_aov()), ARG)]
    return c


def _sync(env):
    env["tree"].sync()
    env["mg"].sync()


@pytest.mark.parametrize("name", ENTRIES)
def test_request_checks(gpu, env, name):
    L = env["L"]
    valid = _args(env, name)
    n0 = L.vrt_launch_count()
    assert _call(L, name, valid) == OK, L.vrt_last_error()
    assert L.vrt_launch_count() > n0, f"{name}: the valid request launched nothing"
    _sync(env)
    for what, over, want in _cases(env, name):
        n0 = L.vrt_launch_count()
        rc = _call(L, name, dict(valid, **over))
        _sync(env)
        assert rc == want, f"{name}, {what}: rc {rc} ({L.vrt_last_error().decode()}), expected {want}"
        if name in STEP_TABLE and what in STEP_TABLE_CASES:
            continue
        assert L.vrt_launch_count() == n0, f"{name}, {what}: launched {L.vrt_launch_count() - n0} kernels"
    # the handle still works after the refusals
    assert _call(L, name, valid) == OK
    _sync(env)


@pytest.mark.parametrize("name", sorted(STEP_TABLE))
@pytest.mark.parametrize("rect", [(3, 2, 3, NY), (0, 0, NX, 0), (0, 0, NX + 1, NY), (0, 3, NX, 2)])
def test_refused_gi_film_launches_nothing(gpu, env, name, rect):
    """An empty rectangle or one outside the film no longer launches the cone-trace step table."""
    L = env["L"]
    n0 = L.vrt_launch_count()
    rc = _call(L, name, dict(_args(env, name), rect=rect))
    _sync(env)
    assert rc == (OK if rect[2] >= rect[0] and rect[3] >= rect[1] and rect[2] <= NX else ARG)
    assert L.vrt_launch_count() == n0, f"{name} {rect}: launched {L.vrt_launch_count() - n0} kernels"
