"""GPU: the GI film's planes (albedo, direct, indirect, normal, hit records) in the banded, pipelined frame loop of one
handle (vrt_gi_render_aov_bands_async) and on the replicas of a vrt_mgpu (vrt_mgpu_gi_render_aov(_async)).

Every output lands in a FULL pinned host frame pre-filled with a sentinel byte.  The reference is the single-device
Octree.gi_render_aov on the source tree (whose planes test_gpu_gi_aov.py pins to the point entry points and the
oracle): every byte a call writes must equal it, and every byte it must not write must still hold the sentinel.  On a
box with one GPU the "devices" are several replicas on device 0, plus every visible device once when there are more."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from tests.common import CAM_MAIN, CAM_SPHERE, GI_KD, assert_bits_equal, gi_res, textured_case
from tests.test_gpu_gi_mgpu import _cam, _device_lists, _light, _lit, _replica, _write_obj
from voxelraytrace20190722_b200 import scenes

pytestmark = pytest.mark.gpu
CPP = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "voxelraytrace20190722_b200", "cpp")
SENTINEL = np.uint8(7)
PLANES = ("albedo", "direct", "indirect", "normal", "hits")
OUTS = ("film",) + PLANES
BAND_H = 8  # the bands vrt_mgpu deals


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
    """A textured sphere (four materials, two textures) at depth 7: the albedo plane reads the textures."""
    z = textured_case()
    depth = 7
    tree = gpu.Octree.build(z["tri"], z["nrm"], depth)
    mats = (z["uv"], z["mtl"], z["kd"], z["mtl_tex"], [z["tex0"], z["tex1"]])
    tree.set_materials(*mats)
    _lit(tree, _light(gpu))
    yield dict(tree=tree, res=gi_res(tree.info()["root_aabb"], depth), cam10=CAM_SPHERE, mats=mats)
    tree.close()


class Frames:
    """One set of full pinned host frames, one per output, every byte the sentinel."""

    def __init__(self, gpu, cam, fmt="f32"):
        import torch
        self.ny = cam.ny
        row = {"film": gpu.film_pixel_bytes(fmt), "hits": 16 * cam.spp}
        self.t = {n: torch.full((cam.ny * cam.nx * row.get(n, 12),), int(SENTINEL), dtype=torch.uint8).pin_memory()
                  for n in OUTS}

    def film(self, req=OUTS):
        return self.t["film"].data_ptr() if "film" in req else 0

    def planes(self, req=OUTS):
        return {n: self.t[n].data_ptr() for n in PLANES if n in req}

    def reset(self):
        for t in self.t.values():
            t.fill_(int(SENTINEL))

    def check(self, want, req=OUTS, rows=None, what=""):
        """The requested outputs hold `want` on `rows` (every row by default) and the sentinel elsewhere; the others
        hold the sentinel only."""
        for n, t in self.t.items():
            got = t.numpy().reshape(self.ny, -1)
            if n not in req:
                exp = np.full_like(got, SENTINEL)
            elif rows is None:
                exp = want[n]
            else:
                exp = np.where(rows[:, None], want[n], SENTINEL)
            assert_bits_equal(got, exp, f"{what} {n}")


def _want(tree, cam, res):
    """Every output of the single-device call, as bytes per frame row."""
    film, pl = tree.gi_render_aov(cam, GI_KD, res)
    pl["film"] = film
    return {n: np.ascontiguousarray(a).view(np.uint8).reshape(cam.ny, -1) for n, a in pl.items()}


def _rank_rows(ny, band_h, first, stride):
    return (np.arange(ny) // band_h) % stride == first


@pytest.mark.parametrize("world", [1, 3])
@pytest.mark.parametrize("fmt", ["f32", "rgbe", "rgb8"])
def test_banded_planes_assemble_the_host_frames(gpu, atrium, world, fmt):
    """Every rank renders its bands of the film and all five planes into ONE set of full host frames; two frames with
    different cameras in flight, twice; 99 rows (the last band is short)."""
    tree, res = atrium["tree"], atrium["res"]
    nx, ny, spp = 160, 99, 4
    cams = [_cam(gpu, CAM_MAIN, nx, ny, spp, 0.01 * k) for k in range(4)]
    ranks = [tree] + [_replica(gpu, tree, _light(gpu)) for _ in range(world - 1)]
    try:
        for r in ranks:
            r.set_film_format(fmt)
        want = [_want(tree, c, res) for c in cams]
        sets = [Frames(gpu, cams[0], fmt) for _ in range(2)]
        for k0 in (0, 2):
            for k in (k0, k0 + 1):
                for rank, r in enumerate(ranks):
                    f = sets[k & 1]
                    r.gi_render_aov_bands_async(cams[k], GI_KD, res, f.film(), f.planes(), BAND_H, rank, world)
            for r in ranks:
                r.sync()
            for k in (k0, k0 + 1):
                sets[k & 1].check(want[k], what=f"world {world} {fmt} frame {k}")
                sets[k & 1].reset()
    finally:
        tree.set_film_format("f32")
        for r in ranks[1:]:
            r.close()


def test_plane_subsets_leave_other_bytes_untouched(gpu, atrium):
    tree, res = atrium["tree"], atrium["res"]
    nx, ny, spp = 160, 99, 4
    cam = _cam(gpu, CAM_MAIN, nx, ny, spp)
    want = _want(tree, cam, res)
    f = Frames(gpu, cam)
    for req in (("hits",), ("normal",), ("film", "albedo"), PLANES):
        tree.gi_render_aov_bands_async(cam, GI_KD, res, f.film(req), f.planes(req), BAND_H, 0, 1)
        tree.sync()
        f.check(want, req, what=f"request {req}")
        f.reset()
    # three ranks of which only rank 1 renders: only its rows change
    tree.gi_render_aov_bands_async(cam, GI_KD, res, f.film(), f.planes(), BAND_H, 1, 3)
    tree.sync()
    f.check(want, rows=_rank_rows(ny, BAND_H, 1, 3), what="rank 1 of 3")


@pytest.mark.parametrize("spp", [1, 4])
@pytest.mark.parametrize("band_h", [1, 5, 8, None])
def test_band_shapes(gpu, textured, band_h, spp):
    """band_h 1, 5, 8 and ny, with more ranks than bands: the ranks without rows return VRT_OK and write nothing."""
    tree, res = textured["tree"], textured["res"]
    nx, ny = 64, 37
    band_h = band_h or ny
    cam = _cam(gpu, textured["cam10"], nx, ny, spp)
    want = _want(tree, cam, res)
    assert want["albedo"].any()  # (the sphere is in view)
    nbands = -(-ny // band_h)
    stride = nbands + 2
    L = gpu.load()
    f = Frames(gpu, cam)
    kd = np.ascontiguousarray(GI_KD)
    aov = gpu.vrt_gi_aov(**f.planes())
    for first in (nbands, nbands + 1):
        b = gpu.vrt_bands(band_h, first, stride)
        assert L.vrt_gi_render_aov_bands_async(tree._h, C.byref(cam.c), kd.ctypes.data_as(C.c_void_p), float(res),
                                               C.byref(b), C.c_void_p(f.film()), C.byref(aov)) == 0
    tree.sync()
    f.check(want, rows=np.zeros(ny, bool), what=f"band_h {band_h}: ranks without rows")
    for first in range(stride):
        tree.gi_render_aov_bands_async(cam, GI_KD, res, f.film(), f.planes(), band_h, first, stride)
    tree.sync()
    f.check(want, what=f"band_h {band_h} spp {spp}")


def test_mixed_pipeline_on_one_handle(gpu, atrium):
    """GI film -> AOV frame -> harness film -> AOV frame at a larger resolution (buffer growth) -> a new light pass
    under a second light camera -> two AOV frames at another cone-trace resolution, no sync in between: every frame
    equals the synchronous result for the GI state at its enqueue."""
    import torch
    src, res1 = atrium["tree"], atrium["res"]
    res2 = np.float32(res1 * 2)
    l1, l2 = _light(gpu), _light(gpu, shift=-4.0)
    small, big = (160, 99), (240, 150)
    cams = [_cam(gpu, CAM_MAIN, *(big if k >= 3 else small), 4, 0.01 * k) for k in range(6)]
    tree = _replica(gpu, src, l2)
    try:
        want = {k: _want(tree, cams[k], res2) for k in (4, 5)}
        _lit(tree, l1)
        want.update({k: _want(tree, cams[k], res1) for k in (1, 3)})
        want_gi = tree.gi_render(cams[0], GI_KD, res1)
        want_h = tree.render(cams[2])
        assert not np.array_equal(want[4]["indirect"], _want(tree, cams[4], res2)["indirect"])  # the light matters
        gi_buf = torch.full((small[1], small[0], 3), 7, dtype=torch.float32).pin_memory()
        h_buf = torch.full((small[1], small[0], 3), 7, dtype=torch.float32).pin_memory()
        sets = {k: Frames(gpu, cams[k]) for k in (1, 3, 4, 5)}

        def aov(k, res):
            f = sets[k]
            tree.gi_render_aov_bands_async(cams[k], GI_KD, res, f.film(), f.planes(), BAND_H, 0, 1)

        tree.gi_render_bands_async(cams[0], GI_KD, res1, gi_buf.data_ptr(), small[1], 0, 1)
        aov(1, res1)
        tree.render_bands_async(cams[2], h_buf.data_ptr(), small[1], 0, 1)
        aov(3, res1)
        _lit(tree, l2)
        aov(4, res2)
        aov(5, res2)
        tree.sync()
        assert_bits_equal(gi_buf.numpy(), want_gi, "GI film")
        assert_bits_equal(h_buf.numpy(), want_h, "harness film")
        for k, f in sets.items():
            f.check(want[k], what=f"AOV frame {k}")
    finally:
        tree.close()


@pytest.mark.parametrize("scene", ["textured", "atrium"])
def test_multi_gpu_planes_equal_the_single_device_planes(gpu, request, scene):
    """MultiGpu: pipelined AOV frames alternating between two sets of host frames, the sync form, and more replicas
    than bands (8 rows, three replicas)."""
    case = request.getfixturevalue(scene)
    tree, res = case["tree"], case["res"]
    nx, ny, spp = 200, 133, 4
    cams = [_cam(gpu, case["cam10"], nx, ny, spp, 0.01 * k) for k in range(4)]
    want = [_want(tree, c, res) for c in cams]
    cam8 = _cam(gpu, case["cam10"], nx, 8, spp)
    want8 = _want(tree, cam8, res)
    for devices in _device_lists(gpu, 3):
        mg = gpu.MultiGpu(tree, devices)
        try:
            if case["mats"] is not None:
                mg.set_materials(*case["mats"])
            _lit(mg, _light(gpu))
            sets = [Frames(gpu, cams[0]) for _ in range(2)]
            for k0 in (0, 2):
                for k in (k0, k0 + 1):
                    f = sets[k & 1]
                    mg.gi_render_aov_async(cams[k], GI_KD, res, f.film(), f.planes())
                mg.sync()
                for k in (k0, k0 + 1):
                    sets[k & 1].check(want[k], what=f"{scene} {devices} frame {k}")
                    sets[k & 1].reset()
            f = sets[0]
            mg.gi_render_aov(cams[1], GI_KD, res, f.film(), f.planes())
            f.check(want[1], what=f"{scene} {devices} gi_render_aov")
            f8 = Frames(gpu, cam8)
            mg.gi_render_aov(cam8, GI_KD, res, f8.film(), f8.planes())
            f8.check(want8, what=f"{scene} {devices} more replicas than bands")
        finally:
            mg.close()


def test_plane_frame_arguments_and_errors(gpu, atrium):
    """Every rejected call returns VRT_ERR_ARG and enqueues nothing: the valid frame enqueued after each one (no sync
    in between) is still correct."""
    tree, res = atrium["tree"], atrium["res"]
    L = gpu.load()
    nx, ny, spp = 64, 12, 4
    cam = _cam(gpu, CAM_MAIN, nx, ny, spp)
    want = _want(tree, cam, res)
    kd = np.ascontiguousarray(GI_KD).ctypes.data_as(C.c_void_p)
    fres = float(res)
    mg = gpu.MultiGpu(tree, [0, 0, 0])
    unlit = gpu.Octree.from_blob_dev(*tree.blob_dev())
    sets = []
    try:
        def single(h, c, k, b, f, a):
            return L.vrt_gi_render_aov_bands_async(h, c, k, fres, b, f, a)

        def multi(h, c, k, _b, f, a, sync=False):
            return (L.vrt_mgpu_gi_render_aov if sync else L.vrt_mgpu_gi_render_aov_async)(h, c, k, fres, f, a)

        def valid(enqueue):
            f = Frames(gpu, cam)
            sets.append(f)
            enqueue(f)

        good_b = gpu.vrt_bands(BAND_H, 0, 1)
        none = gpu.vrt_gi_aov()
        for name, call, h, enqueue in (
                ("tree", single, tree._h,
                 lambda f: tree.gi_render_aov_bands_async(cam, GI_KD, res, f.film(), f.planes(), BAND_H, 0, 1)),
                ("mgpu", multi, mg._h, lambda f: mg.gi_render_aov_async(cam, GI_KD, res, f.film(), f.planes()))):
            if name == "mgpu":
                # the replicas hold geometry only: no plane frame before their light pass
                f = Frames(gpu, cam)
                aov = gpu.vrt_gi_aov(**f.planes())
                assert call(h, C.byref(cam.c), kd, C.byref(good_b), C.c_void_p(f.film()), C.byref(aov)) == -1
                _lit(mg, _light(gpu))
            else:
                f = Frames(gpu, cam)
                aov = gpu.vrt_gi_aov(**f.planes())
                assert call(unlit._h, C.byref(cam.c), kd, C.byref(good_b), C.c_void_p(f.film()), C.byref(aov)) == -1
            valid(enqueue)
            f = Frames(gpu, cam)
            aov = gpu.vrt_gi_aov(**f.planes())
            film = C.c_void_p(f.film())
            bad = [("every plane NULL", (h, C.byref(cam.c), kd, C.byref(good_b), film, C.byref(none))),
                   ("null cam", (h, None, kd, C.byref(good_b), film, C.byref(aov))),
                   ("null kd", (h, C.byref(cam.c), None, C.byref(good_b), film, C.byref(aov))),
                   ("null aov", (h, C.byref(cam.c), kd, C.byref(good_b), film, None))]
            if name == "tree":
                bad += [(f"bands {bb}", (h, C.byref(cam.c), kd, C.byref(gpu.vrt_bands(*bb)), film, C.byref(aov)))
                        for bb in ((0, 0, 1), (BAND_H, 0, 0), (BAND_H, -1, 1))]
            else:
                bad += [("null handle", (None, C.byref(cam.c), kd, None, film, C.byref(aov)))]
            for what, args in bad:
                assert call(*args) == -1, f"{name}: {what}"
                if name == "mgpu":
                    assert multi(*args, sync=True) == -1, f"{name} sync: {what}"
                valid(enqueue)
            f.check(want, req=(), what=f"{name}: nothing written by the rejected calls")
        tree.sync()
        mg.sync()
        for i, f in enumerate(sets):
            f.check(want, what=f"valid frame {i} after a rejected call")
    finally:
        unlit.close()
        mg.close()


def test_full_size_planes_on_replicas(gpu):
    """main.cc's image at full size: the atrium at 1024^3, light film 2048^2 x 4, 3840 x 2160 x 4, the RGBE film
    and every plane through MultiGpu([0, 0]): bytewise gi_render_aov_dev's, compared on the host."""
    import torch
    depth = 11
    tri, nrm = scenes.atrium()
    tree = gpu.Octree.build(tri, nrm, depth)
    res = gi_res(tree.info()["root_aabb"], depth)
    lcam = _light(gpu, n=2048)
    nx, ny, spp = 3840, 2160, 4
    cam = _cam(gpu, CAM_MAIN, nx, ny, spp)
    try:
        _lit(tree, lcam)
        tree.set_film_format("rgbe")
        f = Frames(gpu, cam, "rgbe")
        d = {n: torch.empty(t.numel(), dtype=torch.uint8, device="cuda") for n, t in f.t.items()}
        tree.gi_render_aov_dev(cam, GI_KD, res, d["film"].data_ptr(), {n: d[n].data_ptr() for n in PLANES})
        tree.sync()
        want = {n: t.cpu().numpy().reshape(ny, -1) for n, t in d.items()}
        del d
        film = want["film"].reshape(ny, nx, 4)
        assert (film != film[0, 0]).any(axis=2).mean() > 0.05
        mg = gpu.MultiGpu(tree, [0, 0])
        try:
            mg.set_film_format("rgbe")
            _lit(mg, lcam)
            mg.gi_render_aov(cam, GI_KD, res, f.film(), f.planes())
            f.check(want, what="4K RGBE film and planes on [0, 0]")
        finally:
            mg.close()
    finally:
        tree.close()


def test_demo_main_gi_aov_devices(tmp_path, gpu):
    """The C++ mirror: demo_main --gi f --gi-aov p --gi-devices 0,0 also writes p.mgpu.*.hdr through the MultiGpu
    overload of render_gi_aov_gpu, byte-identical to the single-device p.*.hdr."""
    subprocess.check_call(["make", "-s", "-C", CPP])
    tri, nrm = scenes.uv_sphere(64, 32)
    obj = tmp_path / "sphere.obj"
    _write_obj(obj, tri, nrm)
    nx, ny, depth = 96, 67, 6
    prefix = tmp_path / "p"
    out = subprocess.run([os.path.join(CPP, "demo_main"), str(tmp_path / "o.bmp"), str(depth), str(nx), str(ny),
                          str(obj), "--gi", str(tmp_path / "f.bin"), "--gi-aov", str(prefix), "--gi-devices", "0,0"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "GI planes on 2 replicas written" in out.stdout and "success." in out.stdout
    for n in ("albedo", "direct", "indirect", "normal"):
        single = (tmp_path / f"p.{n}.hdr").read_bytes()
        multi = (tmp_path / f"p.mgpu.{n}.hdr").read_bytes()
        assert len(single) > nx * ny * 4 and multi == single, n
