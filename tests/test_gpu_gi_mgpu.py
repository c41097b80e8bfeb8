"""GPU: the cone-traced GI film (main.cc:117-126) on several GPUs -- the banded, pipelined form of one handle
(vrt_gi_render_bands_async, one call per rank into one shared host frame) and the single-process multi-GPU form
(vrt_mgpu_set_materials / vrt_mgpu_gi_* on the replicas of a vrt_mgpu).

The single-device GI film is pinned to the oracle and to reference-generated vectors (test_gpu_gi.py); these tests
require the multi-GPU films to equal it bytewise.  On a box with one GPU the "devices" are several replicas on
device 0, plus every visible device once when there are more."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests.common import CAM_LIGHT, CAM_MAIN, CAM_SPHERE, GI_KD, assert_bits_equal, gi_res, textured_case
from voxelraytrace20190722_b200 import dist as vdist
from voxelraytrace20190722_b200 import scenes

pytestmark = pytest.mark.gpu
CPP = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "voxelraytrace20190722_b200", "cpp")


def _cam(gpu, c, nx, ny, spp, shift=0.0):
    return gpu.Camera(c[0], c[1:4] + np.float32(shift), c[4:7], c[7:10], nx, ny, spp)


def _light(gpu, shift=0.0, n=128):
    return _cam(gpu, CAM_LIGHT, n, n, 4, shift)


def _lit(tree, lcam):
    tree.gi_init()
    tree.gi_splat(lcam, GI_KD)
    tree.gi_filter()


def _replica(gpu, tree, lcam):
    """A rank's own copy of the octree (what a multi-process host receives), lit by its own light pass."""
    p, n = tree.blob_dev()
    r = gpu.Octree.from_blob_dev(p, n)
    _lit(r, lcam)
    return r


def _device_lists(gpu, reps):
    ndev = gpu.device_count()
    return [[0] * reps] + ([list(range(ndev))] if ndev > 1 else [])


def _pinned(shape, dtype="float32"):
    import torch
    dt = {"float32": torch.float32, "uint8": torch.uint8}[dtype]
    return torch.full(shape, 7, dtype=dt).pin_memory()


def _expect(tree, cam, res, fmt="f32"):
    f = tree.gi_render(cam, GI_KD, res)
    return f if fmt == "f32" else tree.film_encode(f, fmt)


@pytest.fixture(scope="module")
def atrium(gpu):
    """The untextured atrium at detail 0.3, depth 8, lit from main.cc's light camera."""
    tri, nrm = scenes.atrium(detail=0.3)
    depth = 8
    tree = gpu.Octree.build(tri, nrm, depth)
    _lit(tree, _light(gpu))
    yield dict(tree=tree, res=gi_res(tree.info()["root_aabb"], depth), cam10=CAM_MAIN, mats=None)
    tree.close()


@pytest.fixture(scope="module")
def textured(gpu):
    """A textured sphere (four materials, two textures) at depth 7."""
    z = textured_case()
    depth = 7
    tree = gpu.Octree.build(z["tri"], z["nrm"], depth)
    mats = (z["uv"], z["mtl"], z["kd"], z["mtl_tex"], [z["tex0"], z["tex1"]])
    tree.set_materials(*mats)
    _lit(tree, _light(gpu))
    yield dict(tree=tree, res=gi_res(tree.info()["root_aabb"], depth), cam10=CAM_SPHERE, mats=mats)
    tree.close()


@pytest.mark.parametrize("world", [1, 3])
@pytest.mark.parametrize("fmt", ["f32", "rgbe"])
def test_banded_gi_frames_assemble_the_host_frame(gpu, atrium, world, fmt):
    """Every rank renders its bands of the GI film with gi_render_bands_async into ONE shared host frame; two frames
    with different cameras in flight, twice; 99 rows (the last band is short)."""
    tree, res = atrium["tree"], atrium["res"]
    nx, ny, spp = 160, 99, 4
    cams = [_cam(gpu, CAM_MAIN, nx, ny, spp, 0.01 * k) for k in range(4)]
    want = [_expect(tree, c, res, fmt) for c in cams]
    ranks = [tree] + [_replica(gpu, tree, _light(gpu)) for _ in range(world - 1)]
    shf = vdist.SharedHostFrame(ny, nx, nbuf=2, fmt=fmt)
    try:
        for r in ranks:
            r.set_film_format(fmt)
        for k0 in (0, 2):
            for k in (k0, k0 + 1):
                shf.frame(k)[:] = 7
                for rank, r in enumerate(ranks):
                    r.gi_render_bands_async(cams[k], GI_KD, res, shf.ptr(k), vdist.BAND_H, rank, world)
            for r in ranks:
                r.sync()
            for k in (k0, k0 + 1):
                assert_bits_equal(shf.frame(k), want[k], f"world {world} {fmt} frame {k}")
    finally:
        tree.set_film_format("f32")
        for r in ranks[1:]:
            r.close()
        shf.close()


@pytest.mark.parametrize("scene", ["textured", "atrium"])
def test_multi_gpu_gi_film_equals_the_single_device_film(gpu, request, scene):
    """MultiGpu: materials and the light pass on the replicas, then pipelined GI frames on two pinned host frames,
    bytewise equal to Octree.gi_render on the source tree."""
    case = request.getfixturevalue(scene)
    tree, res = case["tree"], case["res"]
    nx, ny, spp = 200, 133, 4
    cams = [_cam(gpu, case["cam10"], nx, ny, spp, 0.01 * k) for k in range(4)]
    want = [_expect(tree, c, res) for c in cams]
    assert (want[0] != want[0][0, 0]).any(axis=2).mean() > 0.05  # (the scene is in view)
    for devices in _device_lists(gpu, 3):
        mg = gpu.MultiGpu(tree, devices)
        try:
            if case["mats"] is not None:
                mg.set_materials(*case["mats"])
            mg.gi_init()
            mg.gi_splat(_light(gpu), GI_KD)
            mg.gi_filter()
            bufs = [_pinned((ny, nx, 3)) for _ in range(2)]
            for k0 in (0, 2):
                for k in (k0, k0 + 1):
                    mg.gi_render_async(cams[k], GI_KD, res, bufs[k & 1].data_ptr())
                mg.sync()
                for k in (k0, k0 + 1):
                    assert_bits_equal(bufs[k & 1].numpy(), want[k], f"{scene} {devices} frame {k}")
            mg.gi_render(cams[1], GI_KD, res, bufs[0].data_ptr())
            assert_bits_equal(bufs[0].numpy(), want[1], f"{scene} {devices} gi_render")
            assert all(mg.mean_kernel_ms(i, 2) > 0 for i in range(len(devices)))
            assert mg.mean_kernel_ms(len(devices), 2) == 0.0
        finally:
            mg.close()


def test_relighting_between_pipelined_frames(gpu, atrium):
    """Three GI frames enqueued (both kernel streams busy), then -- without a sync -- a new light pass under a second
    light camera and two more frames at another cone-trace resolution: every frame equals the synchronous film under
    its own light and resolution.  On one handle (gi_render_bands_async over the whole film) and on MultiGpu."""
    src, res1 = atrium["tree"], atrium["res"]
    res2 = np.float32(res1 * 2)
    l1, l2 = _light(gpu), _light(gpu, shift=-4.0)
    nx, ny, spp = 160, 99, 4
    cams = [_cam(gpu, CAM_MAIN, nx, ny, spp, 0.01 * k) for k in range(5)]
    ress = [res1, res1, res1, res2, res2]
    tree = _replica(gpu, src, l2)
    try:
        want = [None] * 5
        for k in (3, 4):
            want[k] = _expect(tree, cams[k], ress[k])
        _lit(tree, l1)
        for k in (0, 1, 2):
            want[k] = _expect(tree, cams[k], ress[k])
        assert not np.array_equal(want[2], _expect(src, cams[2], res2))  # the resolution matters ...
        assert not np.array_equal(want[3], _expect(src, cams[3], res2))  # ... and so does the light
        bufs = [_pinned((ny, nx, 3)) for _ in range(5)]

        def run(enqueue, relight, sync):
            for k in (0, 1, 2):
                enqueue(k)
            relight()
            for k in (3, 4):
                enqueue(k)
            sync()
            for k in range(5):
                assert_bits_equal(bufs[k].numpy(), want[k], f"frame {k}")
                bufs[k].fill_(7)

        run(lambda k: tree.gi_render_bands_async(cams[k], GI_KD, ress[k], bufs[k].data_ptr(), ny, 0, 1),
            lambda: _lit(tree, l2), tree.sync)
        for devices in _device_lists(gpu, 2):
            mg = gpu.MultiGpu(src, devices)
            try:
                _lit(mg, l1)
                run(lambda k: mg.gi_render_async(cams[k], GI_KD, ress[k], bufs[k].data_ptr()), lambda: _lit(mg, l2),
                    mg.sync)
            finally:
                mg.close()
    finally:
        tree.close()


def test_full_size_gi_film_on_replicas(gpu):
    """main.cc's image at full size: the atrium at 1024^3, light film 512^2 x 4, GI film 3840 x 2160 x 4 in RGBE
    through MultiGpu -- bytewise the single device's gi_render_dev film."""
    import torch
    depth = 11
    tri, nrm = scenes.atrium()
    tree = gpu.Octree.build(tri, nrm, depth)
    res = gi_res(tree.info()["root_aabb"], depth)
    lcam = _light(gpu, n=512)
    nx, ny, spp = 3840, 2160, 4
    cam = _cam(gpu, CAM_MAIN, nx, ny, spp)
    try:
        _lit(tree, lcam)
        tree.set_film_format("rgbe")
        d_film = torch.empty(ny * nx * 4, dtype=torch.uint8, device="cuda")
        tree.gi_render_dev(cam, GI_KD, res, d_film.data_ptr())
        tree.sync()
        want = d_film.cpu().numpy().reshape(ny, nx, 4)
        del d_film
        assert (want != want[0, 0]).any(axis=2).mean() > 0.05
        host = _pinned((ny, nx, 4), "uint8")
        for devices in _device_lists(gpu, 2):
            mg = gpu.MultiGpu(tree, devices)
            try:
                mg.set_film_format("rgbe")
                _lit(mg, lcam)
                mg.gi_render(cam, GI_KD, res, host.data_ptr())
                assert_bits_equal(host.numpy(), want, f"4K RGBE GI film on {devices}")
                host.fill_(7)
            finally:
                mg.close()
    finally:
        tree.close()


def test_gi_multi_gpu_arguments_and_edge_cases(gpu, atrium):
    tree, res = atrium["tree"], atrium["res"]
    L = gpu.load()
    nx, ny, spp = 64, 12, 4
    cam = _cam(gpu, CAM_MAIN, nx, ny, spp)
    mg = gpu.MultiGpu(tree, [0, 0, 0])
    host = _pinned((ny, nx, 3))
    try:
        # the replicas hold geometry only: no GI film before their light pass
        with pytest.raises(gpu.VrtError) as e:
            mg.gi_render(cam, GI_KD, res, host.data_ptr())
        assert e.value.code == -1
        unlit = gpu.Octree.from_blob_dev(*tree.blob_dev())
        with pytest.raises(gpu.VrtError):
            unlit.gi_render_bands_async(cam, GI_KD, res, host.data_ptr(), ny, 0, 1)
        unlit.close()
        mg.gi_init()
        bad = _light(gpu)
        bad.c.spp = 3
        with pytest.raises(gpu.VrtError):
            mg.gi_splat(bad, GI_KD)
        with pytest.raises(gpu.VrtError):
            tree.gi_splat(bad, GI_KD)
        mg.gi_splat(_light(gpu), GI_KD)
        mg.gi_filter()
        # 12 rows = two bands for three replicas: the third has nothing to render
        want = _expect(tree, cam, res)
        mg.gi_render(cam, GI_KD, res, host.data_ptr())
        assert_bits_equal(host.numpy(), want, "more replicas than bands")
        # rgb8 (Film::to_byte_array) through the replicas
        mg.set_film_format("rgb8")
        h8 = _pinned((ny, nx, 3), "uint8")
        mg.gi_render(cam, GI_KD, res, h8.data_ptr())
        assert_bits_equal(h8.numpy(), _expect(tree, cam, res, "rgb8"), "rgb8")
        mg.set_film_format("f32")
        # null kd / null frame: VRT_ERR_ARG, like vrt_gi_render_camera
        kd = np.ascontiguousarray(GI_KD)
        fres = float(res)
        b = gpu.vrt_bands(ny, 0, 1)
        assert L.vrt_mgpu_gi_render_async(mg._h, C.byref(cam.c), None, fres, C.c_void_p(host.data_ptr())) == -1
        assert L.vrt_mgpu_gi_render_async(mg._h, C.byref(cam.c), kd.ctypes.data_as(C.c_void_p), fres, None) == -1
        assert L.vrt_gi_render_bands_async(tree._h, C.byref(cam.c), None, fres, C.byref(b),
                                           C.c_void_p(host.data_ptr())) == -1
        assert L.vrt_gi_render_bands_async(tree._h, C.byref(cam.c), kd.ctypes.data_as(C.c_void_p), fres, C.byref(b),
                                           None) == -1
        assert L.vrt_gi_render_camera(tree._h, C.byref(cam.c), None, fres, 0, 0, nx, ny, C.c_void_p(host.data_ptr())) == -1
        assert L.vrt_mgpu_gi_init(None) == -1 and L.vrt_mgpu_mean_kernel_ms(None, 0, 1) == 0.0
        # the handles are still usable after the rejected calls
        mg.gi_render(cam, GI_KD, res, host.data_ptr())
        assert_bits_equal(host.numpy(), want, "after rejected calls")
    finally:
        mg.close()


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


def test_demo_main_gi_devices(tmp_path, gpu):
    """The C++ mirror: demo_main --gi-devices 0,0 renders main.cc's GI film again through gi::MultiGpu
    (light_map_gpu / cone_trace_init_filter / render_gi_gpu on the replicas); it equals the single-device film."""
    subprocess.check_call(["make", "-s", "-C", CPP])
    tri, nrm = scenes.uv_sphere(64, 32)
    obj = tmp_path / "sphere.obj"
    _write_obj(obj, tri, nrm)
    nx, ny, depth = 96, 67, 6
    gi_dump = tmp_path / "gi_film.bin"
    out = subprocess.run([os.path.join(CPP, "demo_main"), str(tmp_path / "o.bmp"), str(depth), str(nx), str(ny),
                          str(obj), "--gi", str(gi_dump), "--gi-devices", "0,0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "GI film on 2 replicas" in out.stdout and "success." in out.stdout
    single = np.fromfile(gi_dump, np.float32)
    multi = np.fromfile(str(gi_dump) + ".mgpu", np.float32)
    assert single.size == nx * ny * 3 and single.max() > 0
    assert_bits_equal(multi, single, "demo_main GI film on gi::MultiGpu")
