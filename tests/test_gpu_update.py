"""GPU: animated geometry -- vrt_update_triangles(_dev), vrt_update_xform and their vrt_mgpu_* forms.

After an update a handle must be bytewise the handle a fresh build makes from the new pose: the blob (the checkpoint
bytes of vrt_tree_save), the exported leaf set and the info, and therefore every frame.  A transform update must
produce exactly the pose a float32 numpy evaluation of ((m0*x + m1*y) + m2*z) + m3 gives.  Updates between enqueued
pipelined frames must order themselves: frames before render the old pose, frames after the new one."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests.common import CAM_LIGHT, CAM_MAIN, CAM_SPHERE, GI_KD, assert_bits_equal, gi_res
from voxelraytrace20190722_b200 import scenes

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CPP = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "voxelraytrace20190722_b200", "cpp")
OFF_TRI4, OFF_NRM = 240, 248  # byte offsets of BlobHeader::off_tri4 / off_nrm (csrc/vrt_internal.h)


# ---- the pose a transform update must produce, restated in float32 numpy ------------------------------------------
def _rows(m, p, w):
    """((m0*x + m1*y) + m2*z) [+ m3] per row of m for points p [..., 3], every operation rounded to float32."""
    m = np.asarray(m, np.float32)
    out = np.empty_like(p)
    for r in range(3):
        s = (m[r, 0] * p[..., 0]).astype(np.float32) + (m[r, 1] * p[..., 1]).astype(np.float32)
        s = s.astype(np.float32) + (m[r, 2] * p[..., 2]).astype(np.float32)
        s = s.astype(np.float32)
        out[..., r] = (s + m[r, 3]).astype(np.float32) if w == 4 else s
    return out


def _pose(tri, nrm, xforms):
    """The current pose for rest pose (tri, nrm) [T, 9] and xforms [(first, count, M[, N])]."""
    from voxelraytrace20190722_b200 import capi
    t = np.array(tri, np.float32).reshape(-1, 3, 3)
    n = None if nrm is None else np.array(nrm, np.float32).reshape(-1, 3, 3)
    for x in xforms:
        a, b = x[0], x[0] + x[1]
        t[a:b] = _rows(np.asarray(x[2], np.float32).reshape(3, 4), t[a:b], 4)
        if n is not None:
            nm = np.asarray(x[3], np.float32) if len(x) == 4 else capi.xform_normal_matrix(x[2])
            n[a:b] = _rows(nm.reshape(3, 3), n[a:b], 3)
    return t.reshape(-1, 9), None if n is None else n.reshape(-1, 9)


def _rot(axis, ang, centre=(0, 0, 0), shift=(0, 0, 0)):
    """3x4 float32: rotation by `ang` about `axis` through `centre`, then a translation."""
    a = np.asarray(axis, np.float64)
    a = a / np.linalg.norm(a)
    k = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    r = np.eye(3) + np.sin(ang) * k + (1 - np.cos(ang)) * (k @ k)
    c = np.asarray(centre, np.float64)
    return np.concatenate([r, (c - r @ c + np.asarray(shift))[:, None]], 1).astype(np.float32)


# ---- handles --------------------------------------------------------------------------------------------------------
def _build(gpu, tri, nrm, depth, unit=False):
    """vrt_build, or vrt_build_ex with VRT_BUILD_UNIT_NORMALS."""
    if not unit:
        return gpu.Octree.build(tri, nrm, depth)
    L = gpu.load()
    tri = np.ascontiguousarray(tri, np.float32)
    nrm = np.ascontiguousarray(nrm, np.float32)
    L.vrt_build_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_uint32, C.POINTER(C.c_void_p)]
    h = C.c_void_p()
    gpu._check(L.vrt_build_ex(tri.ctypes.data, nrm.ctypes.data, len(tri), depth, 1, C.byref(h)))
    return gpu.Octree(h.value)


def _blob(tree, tmp_path, name="b"):
    """The blob up to hdr.bytes (the checkpoint vrt_tree_save writes)."""
    p = str(tmp_path / f"{name}.vrt")
    tree.save(p)
    return open(p, "rb").read()


def _blob_pose(blob, T):
    """(tri [T, 9], nrm [T, 9]) from the blob's tri4 and nrm sections."""
    o4, on = (int(np.frombuffer(blob[o:o + 8], np.uint64)[0]) for o in (OFF_TRI4, OFF_NRM))
    tri = np.frombuffer(blob[o4:o4 + 48 * T], np.float32).reshape(T, 3, 4)[:, :, :3].reshape(T, 9)
    return tri, np.frombuffer(blob[on:on + 36 * T], np.float32).reshape(T, 9)


def _info(tree):
    i = tree.info()
    i.pop("build_ms")
    i.pop("device_bytes")
    i["root_aabb"] = i["root_aabb"].tobytes()
    return i


def _assert_fresh(gpu, tree, tri, nrm, depth, tmp_path, unit=False, what=""):
    """`tree` is bytewise what a fresh build of (tri, nrm) makes: blob, export and info."""
    fresh = _build(gpu, tri, nrm, depth, unit)
    try:
        assert _blob(tree, tmp_path, "u") == _blob(fresh, tmp_path, "f"), f"{what}: blob differs"
        for a, b in zip(tree.leaves(nodes=True), fresh.leaves(nodes=True)):
            assert_bits_equal(a, b, f"{what}: export")
        assert _info(tree) == _info(fresh), f"{what}: info"
    finally:
        fresh.close()


def _cam(gpu, c, nx, ny, spp):
    return gpu.Camera(c[0], c[1:4], c[4:7], c[7:10], nx, ny, spp)


def _lit(tree, lcam):
    tree.gi_init()
    tree.gi_splat(lcam, GI_KD)
    tree.gi_filter()


def _pinned(shape, dtype):
    import torch
    return torch.full(shape, 7, dtype=dtype).pin_memory()


SCENES = {
    "sphere": (lambda: scenes.uv_sphere(64, 32), 6, CAM_SPHERE),
    "soup": (lambda: scenes.soup(6000, e=0.03), 6, CAM_SPHERE),
    "atrium": (lambda: scenes.atrium(detail=0.3), 6, CAM_MAIN),
}


def _moved(tri, seed):
    """A full new pose of the same triangles: every vertex displaced a little (a deforming mesh)."""
    rng = np.random.default_rng(seed)
    return (np.asarray(tri, np.float32) + rng.uniform(-0.02, 0.02, np.shape(tri)).astype(np.float32)).astype(np.float32)


# ---- full update ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("normals", ["none", "given", "unit"])
def test_full_update_equals_fresh_build(gpu, tmp_path, name, normals):
    maker, depth, _ = SCENES[name]
    tri, nrm = maker()
    nrm = None if normals == "none" else nrm
    unit = normals == "unit"
    if unit:  # VRT_BUILD_UNIT_NORMALS keeps normals verbatim: hand it unnormalised ones to see that they are kept
        nrm = (np.asarray(nrm, np.float32) * np.float32(1.5)).astype(np.float32)
    tree = _build(gpu, tri, nrm, depth, unit)
    try:
        tri2 = _moved(tri, 1)
        nrm2 = None if nrm is None else np.roll(nrm, 1, axis=0)
        tree.update(tri2, nrm2)
        _assert_fresh(gpu, tree, tri2, nrm2, depth, tmp_path, unit, f"{name} host")
        tree.update(tri, nrm, max_depth=depth + 1)  # back to the first pose, one level deeper
        _assert_fresh(gpu, tree, tri, nrm, depth + 1, tmp_path, unit, f"{name} depth")
        import torch
        d_tri = torch.from_numpy(np.ascontiguousarray(tri2, np.float32)).cuda()
        d_nrm = None if nrm2 is None else torch.from_numpy(np.ascontiguousarray(nrm2, np.float32)).cuda()
        torch.cuda.synchronize()
        tree.update_dev(d_tri.data_ptr(), 0 if d_nrm is None else d_nrm.data_ptr(), len(tri2), max_depth=depth)
        _assert_fresh(gpu, tree, tri2, nrm2, depth, tmp_path, unit, f"{name} dev")
    finally:
        tree.close()


# ---- transform update ---------------------------------------------------------------------------------------------------
def _xform_cases(T):
    c = (0.1, -0.2, 0.3)
    return {
        "all": [(0, T, _rot((0, 1, 0), 0.7, c, (0.05, 0.01, -0.03)))],
        "disjoint": [(T // 2, T // 5, _rot((1, 1, 0), -1.1, c, (0.2, 0, 0))),
                     (3, T // 4, _rot((0, 0, 1), 0.3), _rot((0, 1, 0), 2.0)[:, :3]),  # an explicit (odd) N
                     (T - 7, 7, np.concatenate([np.eye(3) * 1.25, np.ones((3, 1)) * 0.01], 1).astype(np.float32))],
        "one": [(T // 3, 1, _rot((0, 1, 1), 1.3, c, (0.0, 0.5, 0.0)))],
        "outside": [(0, T // 2, _rot((1, 0, 0), 0.4, c, (3.0, -2.0, 1.5)))],  # leaves the old root box
    }


@pytest.mark.parametrize("name", sorted(SCENES))
@pytest.mark.parametrize("case", ["all", "disjoint", "one", "outside"])
def test_xform_pose_is_float32_restatement(gpu, tmp_path, name, case):
    maker, depth, _ = SCENES[name]
    tri, nrm = maker()
    tree = gpu.Octree.build(tri, nrm, depth)
    try:
        box0 = tree.info()["root_aabb"]
        xf = _xform_cases(len(tri))[case]
        tree.update_xform(xf)
        ptri, pnrm = _pose(tri, nrm, xf)
        blob = _blob(tree, tmp_path, "x")
        btri, _ = _blob_pose(blob, len(tri))
        assert_bits_equal(btri, ptri, f"{name}/{case}: tri4 section vs numpy pose")
        _assert_fresh(gpu, tree, ptri, pnrm, depth, tmp_path, what=f"{name}/{case}")
        if case == "outside":
            assert not np.array_equal(tree.info()["root_aabb"], box0)
        tree.update_xform(xf)  # absolute: the same table again gives the same tree
        assert _blob(tree, tmp_path, "y") == blob
        tree.rebuild(depth)  # vrt_rebuild rebuilds the current pose
        assert _blob(tree, tmp_path, "z") == blob
        tree.update(tri, nrm)  # a full update is the new rest pose
        tree.update_xform([(0, 1, np.eye(3, 4, dtype=np.float32))])
        _assert_fresh(gpu, tree, tri, nrm, depth, tmp_path, what=f"{name}/{case} rest")
    finally:
        tree.close()


def test_xform_unit_normals_and_no_normals(gpu, tmp_path):
    tri, nrm = scenes.uv_sphere(48, 24)
    xf = _xform_cases(len(tri))["disjoint"]
    for unit, n in ((True, nrm), (False, None)):
        tree = _build(gpu, tri, n, 6, unit)
        try:
            tree.update_xform(xf)
            ptri, pnrm = _pose(tri, n, xf)
            _assert_fresh(gpu, tree, ptri, pnrm, 6, tmp_path, unit, f"unit={unit}")
            if unit:  # kept verbatim: the blob's nrm section is the numpy pose itself
                assert_bits_equal(_blob_pose(_blob(tree, tmp_path), len(tri))[1], pnrm, "unit normals")
        finally:
            tree.close()


# ---- images -----------------------------------------------------------------------------------------------------------
def _textured_scene(gpu):
    z = np.load(os.path.join(G, "gi_textured.npz"))
    mats = (z["uv"], z["mtl"], z["kd"], z["mtl_tex"], [z["tex0_seen"], z["tex1_seen"]])
    return z, mats, int(z["depth"]), np.float32(z["res"]), np.asarray(z["cam10"], np.float32)


def test_images_after_update_equal_fresh_handle(gpu):
    z, mats, depth, res, cam10 = _textured_scene(gpu)
    tri, nrm = z["tri"], z["nrm"]
    T = len(tri)
    lnx, lny, lspp = (int(v) for v in z["light_dims"])
    lcam = _cam(gpu, z["light_cam10"], lnx, lny, lspp)
    cam = _cam(gpu, cam10, 96, 64, 4)
    xf = [(0, T // 2, _rot((0, 1, 0), 0.5, (0, 0, 0), (0.1, 0, 0)))]
    ptri, pnrm = _pose(tri, nrm, xf)
    tree = gpu.Octree.build(tri, nrm, depth)
    fresh = gpu.Octree.build(ptri, pnrm, depth)
    try:
        tree.set_materials(*mats)
        tree.set_film_format("rgbe")
        _lit(tree, lcam)
        tree.update_xform(xf)
        _lit(tree, lcam)
        fresh.set_materials(*mats)
        fresh.set_film_format("rgbe")
        _lit(fresh, lcam)
        assert_bits_equal(tree.render(cam), fresh.render(cam), "primary film")
        import torch
        d = [torch.zeros(96 * 64 * 4 * 16, dtype=torch.uint8, device="cuda") for _ in range(2)]
        tree.trace_camera_dev(cam, d[0].data_ptr(), compact=True)
        fresh.trace_camera_dev(cam, d[1].data_ptr(), compact=True)
        tree.sync()
        fresh.sync()
        assert torch.equal(d[0], d[1]), "hit16 records"
        assert_bits_equal(tree.gi_render(cam, GI_KD, res), fresh.gi_render(cam, GI_KD, res), "GI film")
        f0, p0 = tree.gi_render_aov(cam, GI_KD, res)
        f1, p1 = fresh.gi_render_aov(cam, GI_KD, res)
        assert_bits_equal(f0, f1, "GI film of the planes call")
        for n in p0:
            assert p0[n].tobytes() == p1[n].tobytes(), f"GI plane {n}"
    finally:
        tree.close()
        fresh.close()


# ---- pipeline ordering --------------------------------------------------------------------------------------------------
def _expected(gpu, tri, nrm, depth, cam, lcam, res, kind):
    t = gpu.Octree.build(tri, nrm, depth)
    try:
        if kind == "film":
            return t.render(cam)
        _lit(t, lcam)
        if kind == "gi":
            return t.gi_render(cam, GI_KD, res)
        return t.gi_render_aov(cam, GI_KD, res, planes=("albedo",), film=False)[1]["albedo"]
    finally:
        t.close()


@pytest.mark.parametrize("first_odd", [False, True])
def test_updates_between_pipelined_frames(gpu, first_odd):
    """Frames of every pipelined kind, updates and relighting enqueued without a sync; each film is the frame of the
    pose in force when it was enqueued."""
    import torch
    tri, nrm = scenes.atrium(detail=0.3)
    depth, T = 6, len(tri)
    nx, ny = 128, 96
    cam = _cam(gpu, CAM_MAIN, nx, ny, 4)
    lcam = _cam(gpu, CAM_LIGHT, 96, 96, 4)
    poses = [[], [(0, T // 3, _rot((0, 1, 0), 0.6, (0, 0.5, 0), (0.1, 0, 0)))],
             [(T // 3, T // 3, _rot((1, 0, 0), -0.4, (0, 0.5, 0), (0, 0.05, 0)))]]
    kinds = ["film", "gi", "aov", "film", "gi"]
    tree = gpu.Octree.build(tri, nrm, depth)
    frames = []  # (pose index, kind, host buffer)
    res = gi_res(tree.info()["root_aabb"], depth)
    try:
        _lit(tree, lcam)
        for k, xf in enumerate(poses):
            if k:
                tree.update_xform(xf)
                _lit(tree, lcam)  # relight: the GI state belongs to the previous octree
            nframes = 3 if (k == 0 and first_odd) else 2
            for j in range(nframes):
                kind = kinds[(k + j) % len(kinds)]
                buf = _pinned((ny, nx, 3), torch.float32)
                if kind == "film":
                    tree.render_async(cam, buf.numpy())
                elif kind == "gi":
                    tree.gi_render_bands_async(cam, GI_KD, res, buf.data_ptr(), ny, 0, 1)
                else:
                    tree.gi_render_aov_bands_async(cam, GI_KD, res, 0, {"albedo": buf.data_ptr()}, ny, 0, 1)
                frames.append((k, kind, buf))
        tree.sync()
        for k, kind, buf in frames:
            ptri, pnrm = _pose(tri, nrm, poses[k])
            exp = _expected(gpu, ptri, pnrm, depth, cam, lcam, res, kind)
            assert_bits_equal(buf.numpy(), exp, f"pose {k} {kind}")
    finally:
        tree.close()


# ---- multi-GPU ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("devices", [[0], [0, 0]])
def test_mgpu_update_equals_fresh(gpu, tmp_path, devices):
    import torch
    tri, nrm = scenes.atrium(detail=0.3)
    depth, T = 6, len(tri)
    nx, ny = 128, 96
    cam = _cam(gpu, CAM_MAIN, nx, ny, 4)
    lcam = _cam(gpu, CAM_LIGHT, 96, 96, 4)
    xf = [(0, T // 2, _rot((0, 1, 0), -0.8, (0, 0.5, 0), (0, 0, 0.2)))]
    ptri, pnrm = _pose(tri, nrm, xf)
    src = gpu.Octree.build(tri, nrm, depth)
    mg = gpu.MultiGpu(src, devices)
    src.close()  # the replica set keeps its own rest pose
    fresh = gpu.Octree.build(ptri, pnrm, depth)
    try:
        mg.gi_init()
        mg.update_xform(xf)
        mg.gi_init()
        mg.gi_splat(lcam, GI_KD)
        mg.gi_filter()
        _lit(fresh, lcam)
        res = gi_res(fresh.info()["root_aabb"], depth)
        buf = _pinned((ny, nx, 3), torch.float32)
        mg.gi_render(cam, GI_KD, res, buf.data_ptr())
        assert_bits_equal(buf.numpy(), fresh.gi_render(cam, GI_KD, res), "replica GI film")
        mg.render(cam, buf.data_ptr())  # every replica renders its 8-row bands: every replica holds the fresh octree
        assert_bits_equal(buf.numpy(), fresh.render(cam), "replica primary film")
        # a replica set made from a loaded tree has no rest pose until a full update
        path = str(tmp_path / "t.vrt")
        fresh.save(path)
        loaded = gpu.Octree.load(path)
        mg2 = gpu.MultiGpu(loaded, devices)
        loaded.close()
        with pytest.raises(gpu.VrtError) as e:
            mg2.update_xform(xf)
        assert e.value.code == -5
        mg2.render(cam, buf.data_ptr())
        assert_bits_equal(buf.numpy(), fresh.render(cam), "loaded set unchanged")
        mg2.update(tri, nrm)
        mg2.update_xform(xf)
        mg2.render(cam, buf.data_ptr())
        assert_bits_equal(buf.numpy(), fresh.render(cam), "loaded set after update + xform")
        mg2.close()
    finally:
        mg.close()
        fresh.close()


# ---- errors ---------------------------------------------------------------------------------------------------------------
def test_errors_change_nothing(gpu, tmp_path):
    L = gpu.load()
    tri, nrm = scenes.uv_sphere(48, 24)
    T, depth = len(tri), 6
    tree = gpu.Octree.build(tri, nrm, depth)
    cam = _cam(gpu, CAM_SPHERE, 64, 48, 1)
    blob, film = _blob(tree, tmp_path), tree.render(cam)
    f32 = np.ascontiguousarray(tri, np.float32)
    n32 = np.ascontiguousarray(nrm, np.float32)
    ok = _rot((0, 1, 0), 0.3)

    def table(*rows):
        arr = (gpu.vrt_xform * max(len(rows), 1))()
        for k, (a, n, m) in enumerate(rows):
            arr[k] = gpu.vrt_xform(a, n, (C.c_float * 12)(*np.asarray(m, np.float32).reshape(-1)),
                                   (C.c_float * 9)(*np.eye(3, dtype=np.float32).reshape(-1)))
        return arr

    bad_m = ok.copy()
    bad_m[1, 2] = np.nan
    inf_m = ok.copy()
    inf_m[0, 3] = np.inf
    calls = {
        "null handle": (L.vrt_update_triangles, (None, f32.ctypes.data, n32.ctypes.data, T, depth), -1),
        "null tri": (L.vrt_update_triangles, (tree._h, None, n32.ctypes.data, T, depth), -1),
        "wrong count": (L.vrt_update_triangles, (tree._h, f32.ctypes.data, n32.ctypes.data, T - 1, depth), -1),
        "normals missing": (L.vrt_update_triangles, (tree._h, f32.ctypes.data, None, T, depth), -1),
        "depth 0": (L.vrt_update_triangles, (tree._h, f32.ctypes.data, n32.ctypes.data, T, 0), -1),
        "depth 18": (L.vrt_update_triangles_dev, (tree._h, f32.ctypes.data, n32.ctypes.data, T, 18), -1),
        "xf null handle": (L.vrt_update_xform, (None, C.cast(table((0, 1, ok)), C.c_void_p), 1, depth), -1),
        "xf null table": (L.vrt_update_xform, (tree._h, None, 1, depth), -1),
        "num_xf 0": (L.vrt_update_xform, (tree._h, C.cast(table((0, 1, ok)), C.c_void_p), 0, depth), -1),
        "xf depth": (L.vrt_update_xform, (tree._h, C.cast(table((0, 1, ok)), C.c_void_p), 1, 18), -1),
        "range past end": (L.vrt_update_xform, (tree._h, C.cast(table((T - 1, 2, ok)), C.c_void_p), 1, depth), -1),
        "range start past end": (L.vrt_update_xform, (tree._h, C.cast(table((T, 1, ok)), C.c_void_p), 1, depth), -1),
        "empty range": (L.vrt_update_xform, (tree._h, C.cast(table((3, 0, ok)), C.c_void_p), 1, depth), -1),
        "overlap": (L.vrt_update_xform, (tree._h, C.cast(table((10, 5, ok), (0, 11, ok)), C.c_void_p), 2, depth), -1),
        "nan m": (L.vrt_update_xform, (tree._h, C.cast(table((0, 4, bad_m)), C.c_void_p), 1, depth), -1),
        "inf m": (L.vrt_update_xform, (tree._h, C.cast(table((0, 4, inf_m)), C.c_void_p), 1, depth), -1),
    }
    nan_n = table((0, 4, ok))
    nan_n[0].n[4] = float("nan")
    calls["nan n"] = (L.vrt_update_xform, (tree._h, C.cast(nan_n, C.c_void_p), 1, depth), -1)
    path = str(tmp_path / "l.vrt")
    tree.save(path)
    loaded = gpu.Octree.load(path)
    calls["loaded: triangles"] = (L.vrt_update_triangles, (loaded._h, f32.ctypes.data, n32.ctypes.data, T, depth), -5)
    calls["loaded: xform"] = (L.vrt_update_xform, (loaded._h, C.cast(table((0, 1, ok)), C.c_void_p), 1, depth), -5)
    mg = gpu.MultiGpu(tree, [0])
    calls["mgpu count"] = (L.vrt_mgpu_update_triangles, (mg._h, f32.ctypes.data, n32.ctypes.data, T + 1, depth), -1)
    calls["mgpu null"] = (L.vrt_mgpu_update_xform, (None, C.cast(table((0, 1, ok)), C.c_void_p), 1, depth), -1)
    calls["mgpu overlap"] = (L.vrt_mgpu_update_xform, (mg._h, C.cast(table((0, 5, ok), (4, 1, ok)), C.c_void_p), 2,
                                                       depth), -1)
    try:
        launches = gpu.launch_count()
        for what, (fn, args, code) in calls.items():
            assert fn(*args) == code, what
            assert gpu.launch_count() == launches, f"{what}: enqueued work"
            assert_bits_equal(tree.render(cam), film, f"{what}: frame after the rejected call")
            launches = gpu.launch_count()
        assert _blob(tree, tmp_path, "after") == blob
        assert_bits_equal(loaded.render(cam), film, "loaded handle unchanged")
        buf = np.zeros((48, 64, 3), np.float32)
        gpu.host_register(buf.ctypes.data, buf.nbytes)
        mg.render(cam, buf.ctypes.data)
        gpu.host_unregister(buf.ctypes.data)
        assert_bits_equal(buf, film, "replicas unchanged")
        with pytest.raises(ValueError):
            tree.update(tri[:-1], nrm[:-1])
        with pytest.raises(ValueError):
            tree.update(tri, nrm[:-1])
    finally:
        mg.close()
        loaded.close()
        tree.close()


# ---- the C++ mirror and the demo ------------------------------------------------------------------------------------------
def _write_obj(path, tri, nrm):
    with open(path, "w") as f:
        for t, n in zip(tri, nrm):
            for v in t:
                f.write("v %.9g %.9g %.9g\n" % tuple(v))
            for v in n:
                f.write("vn %.9g %.9g %.9g\n" % tuple(v))
        for i in range(len(tri)):
            a = 3 * i + 1
            f.write(f"f {a}//{a} {a + 1}//{a + 1} {a + 2}//{a + 2}\n")


def _read_hdr(path, nx, ny):
    raw = open(path, "rb").read()
    head = b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y %d +X %d\n" % (ny, nx)
    assert raw.startswith(head) and len(raw) == len(head) + nx * ny * 4
    return np.frombuffer(raw[len(head):], np.uint8).reshape(ny, nx, 4)


def _unit(nrm):
    """gi::Triangle's ctor normalisation (voxel_octree.cc:426): v / sqrtf(((0 + x*x) + y*y) + z*z), float32."""
    n = np.asarray(nrm, np.float32).reshape(-1, 3)
    s = np.float32(0) + (n[:, 0] * n[:, 0]).astype(np.float32)
    s = (s + (n[:, 1] * n[:, 1]).astype(np.float32)).astype(np.float32)
    s = (s + (n[:, 2] * n[:, 2]).astype(np.float32)).astype(np.float32)
    return (n / np.sqrt(s)[:, None]).astype(np.float32).reshape(-1, 9)


def test_demo_main_animate(tmp_path, gpu):
    """demo_main --animate p: four GI frames of the scene turned by 1..4 quarter turns about the vertical axis through
    the root-box centre (gi::transform_gpu + relighting).  Frame k's HDR pixels are film_encode('rgbe') of the GI film
    Python renders from a fresh build of the pre-turned mesh, and the mirror's ray_march reports that build's leaf."""
    subprocess.check_call(["make", "-s", "-C", CPP])
    tri, nrm = scenes.uv_sphere(64, 32)
    tri = (np.asarray(tri, np.float32) + np.float32(0.25) * np.array([1, 0, 0], np.float32)).astype(np.float32)
    tri[: len(tri) // 4] = (tri[: len(tri) // 4] * np.float32(1.3)).astype(np.float32)  # not symmetric under the turn
    obj = tmp_path / "scene.obj"
    _write_obj(obj, tri, nrm)
    nx, ny, depth = 96, 67, 6
    prefix = tmp_path / "anim"
    out = subprocess.run([os.path.join(CPP, "demo_main"), str(tmp_path / "o.bmp"), str(depth), str(nx), str(ny),
                          str(obj), "--animate", str(prefix)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "animation written" in out.stdout
    fov = np.float32(60.0) * np.float32(3.1415926535897932384626) / np.float32(180.0)
    cam = _cam(gpu, np.concatenate([[fov], CAM_SPHERE[1:]]).astype(np.float32), nx, ny, 4)
    lcam = _cam(gpu, np.concatenate([[fov], CAM_LIGHT[1:]]).astype(np.float32), nx, ny, 4)
    # the demo's Triangle objects hold ctor-normalised normals, handed over with VRT_BUILD_UNIT_NORMALS
    un = _unit(nrm)
    box = gpu.Octree.build(tri, nrm, depth).info()["root_aabb"]
    cx = ((box[0] + box[3]) * np.float32(0.5)).astype(np.float32)
    cz = ((box[2] + box[5]) * np.float32(0.5)).astype(np.float32)
    centre = cam.gen_rays(rect=(nx // 2, ny // 2, nx // 2 + 1, ny // 2 + 1))[:1]
    lines = [ln for ln in out.stdout.splitlines() if "centre ray:" in ln and ln.startswith("frame")]
    assert len(lines) == 4
    for k, (c, s) in enumerate([(0, 1), (-1, 0), (0, -1), (1, 0)]):
        c, s = np.float32(c), np.float32(s)
        tx = (cx - ((c * cx).astype(np.float32) + (s * cz).astype(np.float32))).astype(np.float32)
        tz = (cz - ((-s * cx).astype(np.float32) + (c * cz).astype(np.float32))).astype(np.float32)
        m = np.array([[c, 0, s, tx], [0, 1, 0, 0], [-s, 0, c, tz]], np.float32)
        n = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]], np.float32)
        ptri, pnrm = _pose(tri, un, [(0, len(tri), m, n)])
        t = _build(gpu, ptri, pnrm, depth, unit=True)
        try:
            _lit(t, lcam)
            res = gi_res(t.info()["root_aabb"], depth)
            film = t.gi_render(cam, GI_KD, res)
            assert_bits_equal(_read_hdr(f"{prefix}.{k}.hdr", nx, ny), t.film_encode(film, "rgbe"), f"frame {k}")
            h = t.trace_rays(centre)[0]
            if h["hit"]:
                cell, cnt, _ = t.leaves()
                li = np.flatnonzero((cell == h["cell"]).all(1))[0]
                assert lines[k] == (f"frame {k} centre ray: leaf cell ({h['cell'][0]},{h['cell'][1]},{h['cell'][2]}) "
                                    f"with {cnt[li]} triangles, triangle {h['tri']}"), lines[k]
            else:
                assert lines[k] == f"frame {k} centre ray: miss"
        finally:
            t.close()
