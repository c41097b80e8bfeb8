"""GPU: what the cone-traced GI film is made of (vrt_gi_render_aov): albedo, the leaf's direct light, the cone-traced
indirect light, the ISect normal and the 16-byte hit records, from the film's own launch.

The planes are pinned three ways: the film is bytewise the film of gi_render (so nothing else changed), every term is
bit-exact against the point entry points of the library evaluated on trace_camera's hits (albedo, gi_cone_trace,
the hit normal, and compute_illum of the hit leaf's light-map row) accumulated like the film, and the terms agree
with the oracle's restatement of main.cc's trace() loop (the indirect term up to the log2f caveat of
test_gpu_gi.py).  The oracle side is the loop of the oracle's orc_gi_render built from the oracle's own ray march,
albedo, cone trace and light-map rows, with VoxelOctree::compute_illum restated below in float32."""
import os
import subprocess

import numpy as np
import pytest

from tests.common import CAM_LIGHT, CAM_MAIN, CAM_SPHERE, GI_KD, assert_bits_equal, gi_res
from tests.test_gpu_gi import _lit, mostly_bits_equal
from tests.test_gpu_gi_mgpu import _write_obj
from voxelraytrace20190722_b200 import scenes

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CPP = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "voxelraytrace20190722_b200", "cpp")
FLOAT_PLANES = ("albedo", "direct", "indirect", "normal")
NX, NY = 64, 48


def _cam(gpu, c, nx, ny, spp):
    return gpu.Camera(c[0], c[1:4], c[4:7], c[7:10], nx, ny, spp)


def _textured(gpu, port):
    z = np.load(os.path.join(G, "gi_textured.npz"))
    depth = int(z["depth"])
    texs = [z["tex0_seen"], z["tex1_seen"]]
    tree = gpu.Octree.build(z["tri"], z["nrm"], depth)
    tree.set_materials(z["uv"], z["mtl"], z["kd"], z["mtl_tex"], texs)
    orc = port.build(z["tri"], z["nrm"], depth)
    orc.set_materials(z["uv"], z["mtl"], z["kd"], z["mtl_tex"], texs)
    lnx, lny, lspp = (int(v) for v in z["light_dims"])
    lc = z["light_cam10"]
    tree.gi_init()
    tree.gi_splat(_cam(gpu, lc, lnx, lny, lspp), GI_KD)
    tree.gi_filter()
    orc.gi_reset()
    orc.gi_splat(lc, 1.0, lnx, lny, lspp, GI_KD)
    orc.gi_filter()
    return tree, orc, depth, np.float32(z["res"]), np.asarray(z["cam10"], np.float32)


SCENES = {
    "atrium_d6": (lambda: scenes.atrium(detail=0.3), 6, CAM_MAIN),
    "sphere_d7": (lambda: scenes.uv_sphere(96, 48), 7, CAM_SPHERE),
    "soup_d6": (lambda: scenes.soup(6000, e=0.03), 6, CAM_SPHERE),
    "textured": None,
}


@pytest.fixture(scope="module")
def lit(gpu, port):
    """name -> (tree, oracle tree, depth, res, cam10), lit as in test_gi_rows_vs_oracle; built on first use."""
    cache = {}

    def get(name):
        if name not in cache:
            if name == "textured":
                cache[name] = _textured(gpu, port)
            else:
                maker, depth, cam10 = SCENES[name]
                tri, nrm = maker()
                tree, orc = _lit(gpu, port, tri, nrm, depth)
                cache[name] = (tree, orc, depth, gi_res(orc.root_aabb(), depth), cam10)
        return cache[name]

    yield get
    for tree, *_ in cache.values():
        tree.close()


def _u32(a):
    """The bits of a float plane or of hit records."""
    return np.ascontiguousarray(a).view(np.uint32)


def _accumulate(v, spp):
    """film->add(c * (1/spp)) in sample order from +0 (main.cc:119-122), float32: v [npix * spp, 3] -> [npix, 3]."""
    w = np.float32(0.25) if spp == 4 else np.float32(1)
    v = np.asarray(v, np.float32).reshape(-1, spp, 3)
    acc = np.zeros((v.shape[0], 3), np.float32)
    for s in range(spp):
        acc = (acc + (v[:, s] * w).astype(np.float32)).astype(np.float32)
    return acc


ILLUM_D = np.array([[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, 0, 0], [0, -1, 0], [0, 0, -1]], np.float32)  # voxel_octree.cc:19-20


def _compute_illum(illum, d):
    """VoxelOctree::compute_illum (voxel_octree.h:71-81) of leaf rows illum [n, 6, 3] toward d [n, 3], in float32 with
    the oracle's operation order (vrt_oracle.c orc_compute_illum): out = +0, then for i = 0..5
    out += clamp(((0 + a0 d0) + a1 d1) + a2 d2, 0, 1) * illum[i], a = illum_d[i]."""
    f32 = np.float32
    il = np.asarray(illum, f32).reshape(-1, 6, 3)
    d = np.asarray(d, f32).reshape(-1, 3)
    out = np.zeros((len(d), 3), f32)
    for i in range(6):
        a = ILLUM_D[i]
        s = (f32(0) + a[0] * d[:, 0]).astype(f32)
        s = (s + a[1] * d[:, 1]).astype(f32)
        s = (s + a[2] * d[:, 2]).astype(f32)
        c = np.where(s > 1, f32(1), np.where(s < 0, f32(0), s)).astype(f32)
        out = (out + (c[:, None] * il[:, i]).astype(f32)).astype(f32)
    return out


def _oracle_planes(port, orc, depth, cam10, nx, ny, spp, res):
    """The loop of the oracle's orc_gi_render (main.cc:10-30,117-123) writing the factors of trace() instead of the
    film: the oracle's ray march, albedo and cone trace per sample, compute_illum of the hit leaf's row of the
    oracle's light map, accumulated like the film.  {plane: [ny, nx, 3]}."""
    rays = port.gen_rays(cam10, 1.0, nx, ny, spp)
    h = orc.trace(rays)
    m = h.hit.astype(bool)
    cells, _, il = orc.gi_level(depth - 1)  # the non-empty leaves, the only ones a ray can hit
    side = 1 << (depth - 1)

    def key(c):
        c = c.astype(np.int64)
        return (c[:, 0] * side + c[:, 1]) * side + c[:, 2]

    k = key(cells)
    order = np.argsort(k)
    hk = key(h.cell[m])
    at = np.minimum(np.searchsorted(k[order], hk), len(k) - 1)
    assert np.array_equal(k[order][at], hk), "hit leaf without a light-map row"
    v = {n: np.zeros((len(rays), 3), np.float32) for n in FLOAT_PLANES}
    v["albedo"][m] = orc.albedo(h.tri[m], h.pos[m], GI_KD)
    v["indirect"][m] = orc.gi_cone_trace(h.pos[m], h.nrm[m], res)
    v["direct"][m] = _compute_illum(il[order[at]], -rays[m, 3:6])
    v["normal"][m] = h.nrm[m]
    return {n: _accumulate(v[n], spp).reshape(ny, nx, 3) for n in FLOAT_PLANES}


def _point_terms(tree, depth, res, rays, hits48, hits16):
    """Per-sample terms from the point entry points on 48-byte hits (misses +0): {plane: [n, 3]}."""
    m = hits48["hit"].astype(bool)
    assert np.array_equal(m, hits16["hit"].astype(bool))
    assert np.array_equal(hits48["tri"][m], hits16["tri"][m])
    pos, nrm, tri = hits48["pos"][m], hits48["nrm"][m], hits48["tri"][m]
    _, il = tree.gi_level(depth - 1)
    d = rays["d"][m]
    out = {n: np.zeros((len(hits48), 3), np.float32) for n in FLOAT_PLANES}
    out["albedo"][m] = tree.albedo(tri, pos, GI_KD)
    out["indirect"][m] = tree.gi_cone_trace(pos, nrm, res)
    out["normal"][m] = nrm
    out["direct"][m] = _compute_illum(il[hits16["leaf"][m]], -d)
    return out


def _dev_hits16(gpu, tree, cam, rect=None):
    import torch
    x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
    n = (x1 - x0) * (y1 - y0) * cam.spp
    d = torch.empty(n * 16, dtype=torch.uint8, device="cuda")
    tree.trace_camera_dev(cam, d.data_ptr(), rect=rect, compact=True)
    tree.sync()
    return d.cpu().numpy().view(gpu.HIT16_DTYPE)


@pytest.mark.parametrize("spp", [1, 4])
@pytest.mark.parametrize("name", list(SCENES))
def test_gi_planes_exact(gpu, port, lit, name, spp):
    tree, orc, depth, res, cam10 = lit(name)
    cam = _cam(gpu, cam10, NX, NY, spp)
    film, pl = tree.gi_render_aov(cam, GI_KD, res)
    assert set(pl) == set(gpu.GI_AOV_PLANES)
    # 1. the film is gi_render's, in every film format; the float planes do not depend on the format
    assert_bits_equal(film, tree.gi_render(cam, GI_KD, res), f"{name} f32 film")
    try:
        for fmt in ("rgbe", "rgb8"):
            tree.set_film_format(fmt)
            f2, p2 = tree.gi_render_aov(cam, GI_KD, res)
            want = tree.gi_render(cam, GI_KD, res).view(np.uint8).reshape(-1)[: f2.size]
            assert_bits_equal(f2.reshape(-1), want, f"{name} {fmt} film")
            for n in gpu.GI_AOV_PLANES:
                assert_bits_equal(_u32(p2[n]), _u32(pl[n]), f"{name} {fmt} {n}")
    finally:
        tree.set_film_format("f32")
    # 2. the hit records are trace_camera16's
    h16 = pl["hits"].reshape(-1)
    assert_bits_equal(_u32(h16), _u32(_dev_hits16(gpu, tree, cam)), f"{name} hits")
    # 3. every term against the point entry points, accumulated like the film: no tolerance
    m48 = tree.trace_camera(cam)
    assert m48["hit"].sum() > 100
    terms = _point_terms(tree, depth, res, cam.gen_rays(), m48, h16)
    for n in FLOAT_PLANES:
        assert_bits_equal(pl[n].reshape(-1, 3), _accumulate(terms[n], spp), f"{name} {n} vs point entry points")
    assert pl["indirect"].max() > 0 and pl["direct"].max() > 0
    # 4. against the oracle's trace() loop
    ref = _oracle_planes(port, orc, depth, cam10, NX, NY, spp, res)
    for n in ("albedo", "normal", "direct"):
        assert_bits_equal(pl[n], ref[n], f"{name} {n} vs oracle")
    mostly_bits_equal(pl["indirect"].reshape(-1, 3), ref["indirect"].reshape(-1, 3), f"{name} indirect vs oracle")
    # 5. one sample per pixel: the film is albedo * (indirect + direct) on hits, the sky elsewhere
    if spp == 1:
        hit = h16["hit"].reshape(NY, NX).astype(bool)
        a, i, d = pl["albedo"], pl["indirect"], pl["direct"]
        prod = (a * (i + d).astype(np.float32)).astype(np.float32)
        assert_bits_equal(film[hit], prod[hit], f"{name} film = A * (I + D)")
        assert_bits_equal(film[~hit], tree.render(cam)[~hit], f"{name} film = sky on misses")


@pytest.mark.parametrize("spp", [1, 4])
def test_gi_planes_rectangles_and_subsets(gpu, lit, spp):
    tree, _, _, res, cam10 = lit("atrium_d6")
    cam = _cam(gpu, cam10, NX, NY, spp)
    film, pl = tree.gi_render_aov(cam, GI_KD, res)
    x0, y0, x1, y1 = rect = (5, 3, 50, 40)
    f2, p2 = tree.gi_render_aov(cam, GI_KD, res, rect=rect)
    assert_bits_equal(f2, film[y0:y1, x0:x1], "rect film")
    for n in gpu.GI_AOV_PLANES:
        assert_bits_equal(_u32(p2[n]), _u32(pl[n][y0:y1, x0:x1]), f"rect {n}")
    for n in gpu.GI_AOV_PLANES:
        f3, p3 = tree.gi_render_aov(cam, GI_KD, res, planes=(n,), film=False)
        assert f3 is None and list(p3) == [n]
        assert_bits_equal(_u32(p3[n]), _u32(pl[n]), f"{n} alone")
    _, p4 = tree.gi_render_aov(cam, GI_KD, res, film=False)
    for n in FLOAT_PLANES:
        assert_bits_equal(p4[n], pl[n], f"{n} without film")


def test_gi_planes_errors_and_empty_scene(gpu, lit):
    tree, _, _, res, cam10 = lit("sphere_d7")
    cam = _cam(gpu, cam10, NX, NY, 4)
    unlit = gpu.Octree.from_blob_dev(*tree.blob_dev())
    try:
        with pytest.raises(gpu.VrtError):
            unlit.gi_render_aov(cam, GI_KD, res)  # no vrt_gi_init
    finally:
        unlit.close()
    with pytest.raises(gpu.VrtError) as e:
        tree.gi_render_aov(cam, GI_KD, res, planes=())  # the film alone is gi_render
    assert e.value.code == -1
    with pytest.raises(gpu.VrtError) as e:
        tree.gi_render_aov(cam, GI_KD, res, rect=(0, 0, NX + 1, NY))
    assert e.value.code == -1
    with pytest.raises(gpu.VrtError):
        tree.gi_render_aov_dev(cam, GI_KD, res, 0, {})
    # the handle is usable after the rejected calls
    film, _ = tree.gi_render_aov(cam, GI_KD, res, planes=("albedo",))
    assert_bits_equal(film, tree.gi_render(cam, GI_KD, res), "after rejected calls")
    empty = gpu.Octree.build(np.zeros((0, 3, 3), np.float32), np.zeros((0, 3, 3), np.float32), 5)
    try:
        empty.gi_init()
        empty.gi_splat(_cam(gpu, CAM_LIGHT, 32, 32, 4), GI_KD)
        empty.gi_filter()
        film, pl = empty.gi_render_aov(cam, GI_KD, np.float32(0.01))
        for n in FLOAT_PLANES:
            assert pl[n].view(np.uint32).max() == 0, n  # +0, not -0
        assert (pl["hits"]["leaf"] == gpu.VRT_NO_TRI).all() and (pl["hits"]["hit"] == 0).all()
        assert_bits_equal(film, empty.render(cam), "empty scene: the film is the sky")
    finally:
        empty.close()


def test_gi_planes_dev_ordered_between_pipelined_frames(gpu, lit):
    """Pipelined GI frame -> device planes at another cone-trace resolution and film size -> frame, no sync between:
    each equals its isolated run (the planes use the handle stream's step table)."""
    import torch
    tree, _, _, res, cam10 = lit("atrium_d6")
    nx, ny, spp = 160, 99, 4
    cam1 = _cam(gpu, cam10, nx, ny, spp)
    cam2 = _cam(gpu, cam10, 96, 72, spp)
    res2 = np.float32(res * 2)
    want_frame = tree.gi_render(cam1, GI_KD, res)
    want_film, want = tree.gi_render_aov(cam2, GI_KD, res2)
    assert not np.array_equal(want_film, tree.gi_render(cam2, GI_KD, res))  # the resolution matters
    frames = [torch.full((ny, nx, 3), 7, dtype=torch.float32).pin_memory() for _ in range(2)]
    d_film = torch.full((72, 96, 3), 7, dtype=torch.float32, device="cuda")
    d = {n: torch.full((72, 96, 3), 7, dtype=torch.float32, device="cuda") for n in FLOAT_PLANES}
    d["hits"] = torch.full((72 * 96 * spp * 4,), 7, dtype=torch.int32, device="cuda")
    tree.gi_render_bands_async(cam1, GI_KD, res, frames[0].data_ptr(), ny, 0, 1)
    tree.gi_render_aov_dev(cam2, GI_KD, res2, d_film.data_ptr(), {n: t.data_ptr() for n, t in d.items()})
    tree.gi_render_bands_async(cam1, GI_KD, res, frames[1].data_ptr(), ny, 0, 1)
    tree.sync()
    for k in range(2):
        assert_bits_equal(frames[k].numpy(), want_frame, f"frame {k}")
    assert_bits_equal(d_film.cpu().numpy(), want_film, "device film")
    for n in FLOAT_PLANES:
        assert_bits_equal(d[n].cpu().numpy(), want[n], f"device {n}")
    assert_bits_equal(_u32(d["hits"].cpu().numpy()), _u32(want["hits"].reshape(-1)), "device hits")


def test_gi_planes_full_size(gpu):
    """main.cc's image at full size: the atrium at 1024^3, light film 2048^2 x 4, GI film 3840 x 2160 x 4.  Film and
    hits are bytewise gi_render_dev's and trace_camera16_dev's; the terms are exact against the point entry points
    on a seeded sample of 65,536 pixels."""
    import torch
    depth = 11
    tri, nrm = scenes.atrium()
    tree = gpu.Octree.build(tri, nrm, depth)
    try:
        res = gi_res(tree.info()["root_aabb"], depth)
        tree.gi_init()
        tree.gi_splat(_cam(gpu, CAM_LIGHT, 2048, 2048, 4), GI_KD)
        tree.gi_filter()
        nx, ny, spp = 3840, 2160, 4
        cam = _cam(gpu, CAM_MAIN, nx, ny, spp)
        d_film = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
        d = {n: torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda") for n in FLOAT_PLANES}
        d["hits"] = torch.empty((ny * nx * spp * 4,), dtype=torch.int32, device="cuda")
        tree.gi_render_aov_dev(cam, GI_KD, res, d_film.data_ptr(), {n: t.data_ptr() for n, t in d.items()})
        tree.sync()
        ref = torch.empty_like(d_film)
        tree.gi_render_dev(cam, GI_KD, res, ref.data_ptr())
        tree.sync()
        assert torch.equal(d_film.view(torch.int32), ref.view(torch.int32)), "4K film differs from gi_render_dev"
        del ref
        h16_ref = torch.empty_like(d["hits"])
        tree.trace_camera_dev(cam, h16_ref.data_ptr(), compact=True)
        tree.sync()
        assert torch.equal(d["hits"], h16_ref), "4K hits differ from trace_camera16_dev"
        del h16_ref
        pl = {n: d[n].cpu().numpy() for n in FLOAT_PLANES}
        h16 = d["hits"].cpu().numpy().view(gpu.HIT16_DTYPE).reshape(ny, nx, spp)
        del d, d_film
        rng = np.random.default_rng(2026)
        pix = np.sort(rng.choice(nx * ny, 65536, replace=False))
        py, px = pix // nx, pix % nx
        rays = []
        for y0 in range(0, ny, 216):  # gen_rays in row chunks, keeping the sampled pixels
            sel = (py >= y0) & (py < y0 + 216)
            r = cam.gen_rays((0, y0, nx, min(ny, y0 + 216))).reshape(-1, nx, spp)
            rays.append(r[py[sel] - y0, px[sel]])
        rays = np.concatenate(rays).reshape(-1)
        h48 = tree.trace_rays(rays)
        terms = _point_terms(tree, depth, res, rays, h48, h16[py, px].reshape(-1))
        assert h48["hit"].mean() > 0.5
        for n in FLOAT_PLANES:
            assert_bits_equal(pl[n][py, px], _accumulate(terms[n], spp), f"4K {n} vs point entry points")
    finally:
        tree.close()


def _read_hdr(path, nx, ny):
    raw = open(path, "rb").read()
    head = b"#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y %d +X %d\n" % (ny, nx)
    assert raw.startswith(head) and len(raw) == len(head) + nx * ny * 4
    return np.frombuffer(raw[len(head):], np.uint8).reshape(ny, nx, 4)


def test_demo_main_gi_aov(tmp_path, gpu):
    """The C++ mirror: demo_main --gi f --gi-aov p writes p.{albedo,direct,indirect,normal}.hdr through
    render_gi_aov_gpu; their RGBE pixels are film_encode(plane, 'rgbe') of the same planes through Python."""
    subprocess.check_call(["make", "-s", "-C", CPP])
    tri, nrm = scenes.uv_sphere(64, 32)
    obj = tmp_path / "sphere.obj"
    _write_obj(obj, tri, nrm)
    nx, ny, depth = 96, 67, 6
    gi_dump, prefix = tmp_path / "gi_film.bin", tmp_path / "p"
    out = subprocess.run([os.path.join(CPP, "demo_main"), str(tmp_path / "o.bmp"), str(depth), str(nx), str(ny),
                          str(obj), "--gi", str(gi_dump), "--gi-aov", str(prefix)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "GI planes written" in out.stdout and "success." in out.stdout
    fov = np.float32(60.0) * np.float32(3.1415926535897932384626) / np.float32(180.0)  # the demo's jql::to_radian
    tree = gpu.Octree.build(tri, nrm, depth)
    try:
        tree.gi_init()
        tree.gi_splat(_cam(gpu, np.concatenate([[fov], CAM_LIGHT[1:]]).astype(np.float32), nx, ny, 4), GI_KD)
        tree.gi_filter()
        res = gi_res(tree.info()["root_aabb"], depth)
        cam = _cam(gpu, np.concatenate([[fov], CAM_SPHERE[1:]]).astype(np.float32), nx, ny, 4)
        film, pl = tree.gi_render_aov(cam, GI_KD, res, planes=FLOAT_PLANES)
        # (the same scene and light as the demo's: its film is this film)
        assert_bits_equal(np.fromfile(gi_dump, np.float32).reshape(ny, nx, 3), film, "demo GI film")
        for n in FLOAT_PLANES:
            assert_bits_equal(_read_hdr(f"{prefix}.{n}.hdr", nx, ny), tree.film_encode(pl[n], "rgbe"), f"demo {n}.hdr")
    finally:
        tree.close()
