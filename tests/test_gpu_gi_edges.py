"""GPU: the cone march of the GI rows (vrt_gi.cuh gi_cone_one / gi_cone_sample / gi_locate) at the edges where its
fast paths differ from the reference's loop, bit for bit against the oracle.

The oracle runs in exact mode (Port.exact_log2): split_level = int(log2f(x)) with the correctly rounded log2f, which
is the device's definition, so no sample may differ.  Where NaN can appear the comparison is NaN-aware (the same NaN
positions, every other bit equal): device NaNs are canonical, x86 NaNs are not.

* the march length: res from deeper than the tree down to 1e-30 (a march longer than the step table, continued by the
  per-sample loop) and FLT_MIN, all samples at level 0, no sample at all;
* the step table against the per-sample loop it replaced (VRT_GI_STEPS=0, read once per process: a child process);
* the six-lobe sum (TreeDev::gi_ok = 0: a splat after the filter, non-finite light) against the three-lobe path;
* points exactly on node mid-planes and outside the root box; trees 12 and 17 (VRT_MAX_DEPTH) levels deep;
* res changing between in-flight pipelined frames; a planar scene (zero-thickness root box);
* the refusal of every res on which the march would not end, with nothing launched."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.common import (CAM_LIGHT, CAM_MAIN, CAM_SPHERE, GI_KD, assert_bits_equal, compare_hits, gi_march,
                          gi_maxdist, gi_res, leaves_equal)
from tests.test_gi_march_host import BAD_RES, _calls, res_refused
from tests.test_gpu_gi import _lit, node_cells
from tests.test_gpu_gi_aov import _oracle_planes
from tests.test_gpu_gi_mgpu import _pinned
from voxelraytrace20190722_b200 import scenes

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F32 = np.finfo(np.float32)
SCENES = {
    "atrium_d6": (lambda: scenes.atrium(detail=0.3), 6, CAM_MAIN),
    "sphere_d7": (lambda: scenes.uv_sphere(96, 48), 7, CAM_SPHERE),
}


def _cam(gpu, c, nx, ny, spp):
    return gpu.Camera(c[0], c[1:4], c[4:7], c[7:10], nx, ny, spp)


def assert_nan_equal(a, b, what):
    """The same NaN positions, and bitwise equality everywhere else."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    na, nb = np.isnan(a), np.isnan(b)
    assert np.array_equal(na, nb), f"{what}: NaN at {int((na != nb).sum())} differing positions"
    zero = np.float32(0)
    assert_bits_equal(np.where(na, zero, a), np.where(nb, zero, b), what)


def _levels_vs_oracle(tree, orc, depth, what, cmp=assert_bits_equal):
    cells = node_cells(tree.leaves(nodes=True)[3], tree.info()["level_offset"], depth - 1)
    for level in range(depth):
        ocells, ocov, oil = orc.gi_level(level)
        cov, il = tree.gi_level(level)
        assert_bits_equal(cells[level], ocells, f"{what} level {level} cells")
        cmp(cov, ocov, f"{what} level {level} coverage")
        cmp(il, oil, f"{what} level {level} illum")


def _hits(port, orc, cam10, nx, ny, spp=1):
    h = orc.trace(port.gen_rays(cam10, 1.0, nx, ny, spp))
    m = h.hit.astype(bool)
    assert m.sum() > 100
    return h.pos[m], h.nrm[m]


@pytest.fixture(scope="module")
def lit(gpu, port):
    """name -> (tree, oracle tree, depth, res, cam10), lit as in test_gi_rows_vs_oracle; built on first use."""
    cache = {}

    def get(name):
        if name not in cache:
            maker, depth, cam10 = SCENES[name]
            tri, nrm = maker()
            tree, orc = _lit(gpu, port, tri, nrm, depth)
            assert_bits_equal(tree.info()["root_aabb"], orc.root_aabb(), "root box")
            cache[name] = (tree, orc, depth, gi_res(orc.root_aabb(), depth), cam10)
        return cache[name]

    yield get
    for tree, *_ in cache.values():
        tree.close()


# ---- a. res sweep ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(SCENES))
def test_res_sweep_vs_exact_oracle(gpu, port, lit, name):
    tree, orc, depth, res0, cam10 = lit(name)
    maxdist = gi_maxdist(orc.root_aabb())
    pos, nrm = _hits(port, orc, cam10, 48, 32)
    f32 = np.float32
    cases = {
        "gi_res": res0,
        "gi_res/3": f32(res0 / f32(3)),
        "gi_res/4096": f32(res0 * f32(2.0 ** -12)),
        "1e-30": f32(1e-30),
        "FLT_MIN": f32(F32.tiny),
        "maxdist/2.5": f32(maxdist / f32(2.5)),
        "maxdist": maxdist,
    }
    marches = {k: gi_march(maxdist, r) for k, r in cases.items()}
    assert all(ended for _, ended in marches.values())
    L = depth - 1
    assert max(marches["gi_res/4096"][0]) > L        # samples deeper than the tree
    assert len(marches["1e-30"][0]) > 511            # the step table truncates, the per-sample loop continues
    assert len(marches["FLT_MIN"][0]) > 511
    lv0 = marches["maxdist/2.5"][0]
    assert len(lv0) > 0 and set(lv0) == {0}          # every sample at level 0 (the root)
    assert marches["maxdist"][0] == []               # no sample at all
    with port.exact_log2():
        for k, r in cases.items():
            got = tree.gi_cone_trace(pos, nrm, r)
            assert_bits_equal(got, orc.gi_cone_trace(pos, nrm, r), f"{name} cone_trace res={k}")
            if k == "maxdist":
                assert not got.view(np.uint32).any(), "no step: exact +0"
            elif k in ("gi_res", "maxdist/2.5"):
                assert got.max() > 0
        nx, ny, spp = 32, 24, 4
        cam = _cam(gpu, cam10, nx, ny, spp)
        for k in ("gi_res/3", "1e-30"):
            assert_bits_equal(tree.gi_render(cam, GI_KD, cases[k]),
                              orc.gi_render(cam10, 1.0, nx, ny, spp, cases[k], GI_KD), f"{name} film res={k}")


# ---- b. step table vs the per-sample loop -------------------------------------------------------------------------
def _step_outputs(gpu):
    """Cone traces at three res values, a GI film and a film with every plane, on the lit atrium -- GPU only."""
    tri, nrm = scenes.atrium(detail=0.3)
    depth = 6
    tree = gpu.Octree.build(tri, nrm, depth)
    try:
        tree.gi_init()
        tree.gi_splat(_cam(gpu, CAM_LIGHT, 128, 128, 4), GI_KD)
        tree.gi_filter()
        res = gi_res(tree.info()["root_aabb"], depth)
        cam = _cam(gpu, CAM_MAIN, 40, 30, 4)
        h = tree.trace_camera(cam)
        m = h["hit"].astype(bool)
        out = {}
        for k, r in (("res", res), ("res3", np.float32(res / np.float32(3))), ("tiny", np.float32(1e-30))):
            out["cone_" + k] = tree.gi_cone_trace(h["pos"][m], h["nrm"][m], r)
        out["film"] = tree.gi_render(cam, GI_KD, res)
        film, planes = tree.gi_render_aov(cam, GI_KD, np.float32(1e-30))
        out["aov_film"] = film
        for n, a in planes.items():
            out["aov_" + n] = np.ascontiguousarray(a).view(np.uint32)
        return out
    finally:
        tree.close()


def test_step_table_equals_per_sample_loop(gpu, tmp_path):
    assert os.environ.get("VRT_GI_STEPS", "1")[:1] != "0", "this process must run with the step table"
    path = tmp_path / "loop.npz"
    code = ("import sys; sys.path.insert(0, sys.argv[1]); import numpy as np; "
            "from voxelraytrace20190722_b200 import capi; from tests.test_gpu_gi_edges import _step_outputs; "
            "capi.load(); np.savez(sys.argv[2], **_step_outputs(capi))")
    subprocess.run([sys.executable, "-c", code, ROOT, str(path)], check=True, cwd=ROOT, timeout=600,
                   env=dict(os.environ, VRT_GI_STEPS="0"))
    loop = np.load(path)
    table = _step_outputs(gpu)
    assert sorted(loop.files) == sorted(table)
    assert table["cone_res"].max() > 0 and table["cone_tiny"].max() > 0
    for k, v in table.items():
        assert_bits_equal(v, loop[k], f"{k}: step table vs per-sample loop")


# ---- c. the six-lobe path -----------------------------------------------------------------------------------------
def _away(gpu, n=64):
    """A light camera that looks away from every scene here (no ray hits)."""
    return gpu.Camera(CAM_LIGHT[0], (1, 10, 1), (1, 20, 1), (0, 0, 1), n, n, 4)


@pytest.mark.parametrize("name", list(SCENES))
def test_six_lobe_sum_equals_three_lobe_path(gpu, port, lit, name):
    """The same filtered lobes read by the three facing lobes (gi_ok = 1) and by the full sum (gi_ok = 0 after a splat
    that adds nothing): bytewise the same cone traces, films and indirect planes, over every cone direction,
    including the +-0 components of axis-aligned normals."""
    tree, orc, depth, res, cam10 = lit(name)
    pos, nrm = _hits(port, orc, cam10, 48, 32)
    axes = np.concatenate([np.eye(3), -np.eye(3)]).astype(np.float32)
    pos = np.concatenate([pos, np.repeat(pos[:50], 6, axis=0)])
    nrm = np.concatenate([nrm, np.tile(axes, (50, 1))])
    cam = _cam(gpu, cam10, 40, 30, 4)
    before = [tree.gi_level(level) for level in range(depth)]
    rec = (tree.gi_cone_trace(pos, nrm, res), tree.gi_render(cam, GI_KD, res),
           tree.gi_render_aov(cam, GI_KD, res, planes=("indirect",), film=False)[1]["indirect"])
    away = _away(gpu)
    assert not tree.trace_camera(away)["hit"].any()
    try:
        tree.gi_splat(away, GI_KD)
        for level, (c0, i0) in enumerate(before):
            c1, i1 = tree.gi_level(level)
            assert_bits_equal(c1, c0, f"{name} level {level} coverage")
            assert_bits_equal(i1, i0, f"{name} level {level} illum")
        got = (tree.gi_cone_trace(pos, nrm, res), tree.gi_render(cam, GI_KD, res),
               tree.gi_render_aov(cam, GI_KD, res, planes=("indirect",), film=False)[1]["indirect"])
        for what, a, b in zip(("cone_trace", "film", "indirect"), got, rec):
            assert_bits_equal(a, b, f"{name} six lobes vs three: {what}")
        assert rec[0].max() > 0
    finally:
        tree.gi_filter()  # the module's tree is shared: back to the filtered state


def test_stale_levels_vs_oracle(gpu, port):
    """Splat A, filter, splat B without a filter: leaves hold A + B, the upper levels A's filter (gi_ok = 0)."""
    tri, nrm = scenes.atrium(detail=0.3)
    depth = 6
    tree = gpu.Octree.build(tri, nrm, depth)
    orc = port.build(tri, nrm, depth)
    b10 = np.array([CAM_LIGHT[0], -3, 8, 2, 0, 0, 0, 0, 1, 0], np.float32)
    try:
        tree.gi_init()
        tree.gi_splat(_cam(gpu, CAM_LIGHT, 128, 128, 4), GI_KD)
        tree.gi_filter()
        tree.gi_splat(_cam(gpu, b10, 96, 96, 4), GI_KD)
        orc.gi_reset()
        orc.gi_splat(CAM_LIGHT, 1.0, 128, 128, 4, GI_KD)
        orc.gi_filter()
        orc.gi_splat(b10, 1.0, 96, 96, 4, GI_KD)
        _levels_vs_oracle(tree, orc, depth, "stale")
        res = gi_res(orc.root_aabb(), depth)
        pos, nrm_h = _hits(port, orc, CAM_MAIN, 48, 32)
        nx, ny, spp = 40, 30, 4
        with port.exact_log2():
            got = tree.gi_cone_trace(pos, nrm_h, res)
            assert got.max() > 0
            assert_bits_equal(got, orc.gi_cone_trace(pos, nrm_h, res), "stale cone_trace")
            assert_bits_equal(tree.gi_render(_cam(gpu, CAM_MAIN, nx, ny, spp), GI_KD, res),
                              orc.gi_render(CAM_MAIN, 1.0, nx, ny, spp, res, GI_KD), "stale film")
    finally:
        tree.close()


def test_non_finite_lobes_vs_oracle(gpu, port):
    """kd near +-3e38: leaf sums overflow to +-inf, opposite signs meet in NaN above them, the root is not finite, so
    gi_ok = 0 and every cone sample takes the six-lobe sum (0 * inf = NaN on the lobes facing away)."""
    tri, nrm = scenes.atrium(detail=0.3)
    depth = 6
    tree = gpu.Octree.build(tri, nrm, depth)
    orc = port.build(tri, nrm, depth)
    big = np.array([3e38, -3e38, 3e38], np.float32)
    b10 = np.array([CAM_LIGHT[0], -3, 8, 2, 0, 0, 0, 0, 1, 0], np.float32)
    try:
        tree.gi_init()
        tree.gi_splat(_cam(gpu, CAM_LIGHT, 96, 96, 4), big)
        tree.gi_splat(_cam(gpu, b10, 96, 96, 4), -big)
        tree.gi_filter()
        orc.gi_reset()
        orc.gi_splat(CAM_LIGHT, 1.0, 96, 96, 4, big)
        orc.gi_splat(b10, 1.0, 96, 96, 4, -big)
        orc.gi_filter()
        _, root_il = tree.gi_level(0)
        assert np.isnan(root_il).any(), "the root must be non-finite for the fallback to be taken"
        assert np.isinf(tree.gi_level(depth - 1)[1]).any()
        _levels_vs_oracle(tree, orc, depth, "non-finite", cmp=assert_nan_equal)
        res = gi_res(orc.root_aabb(), depth)
        pos, nrm_h = _hits(port, orc, CAM_MAIN, 48, 32)
        nx, ny, spp = 40, 30, 4
        with port.exact_log2():
            got = tree.gi_cone_trace(pos, nrm_h, res)
            assert np.isnan(got).any()
            assert_nan_equal(got, orc.gi_cone_trace(pos, nrm_h, res), "non-finite cone_trace")
            assert_nan_equal(tree.gi_render(_cam(gpu, CAM_MAIN, nx, ny, spp), GI_KD, res),
                             orc.gi_render(CAM_MAIN, 1.0, nx, ny, spp, res, GI_KD), "non-finite film")
    finally:
        tree.close()


# ---- d. mid-planes and points outside the root box ----------------------------------------------------------------
@pytest.mark.parametrize("name", list(SCENES))
def test_mid_planes_and_outside_points(gpu, port, lit, name):
    """Cone origins whose coordinates are node centres (leaf centres, and leaf faces = the centres of their ancestors,
    all from the reference's float recurrence of the oracle's boxes), on the root faces and half a root size outside
    every face; axis normals, so cone 0 keeps two coordinates on those planes at every step (n_z = -1 takes the
    s = -1 branch of orthonormal_basis).  Where p equals a centre the reference's `p > c` must send it low."""
    tree, orc, depth, res, _ = lit(name)
    bx = orc.leaves(boxes=True)[3]
    rng = np.random.default_rng(5)
    pick = bx[rng.choice(len(bx), min(len(bx), 120), replace=False)]
    half = np.float32(0.5)
    centres = ((pick[:, :3] + pick[:, 3:]) * half).astype(np.float32)
    origins = [centres, pick[:, :3], pick[:, 3:],
               np.stack([pick[:, 0], centres[:, 1], pick[:, 5]], axis=1)]
    root = orc.root_aabb()
    rc = ((root[:3] + root[3:]) * half).astype(np.float32)
    size = (root[3:] - root[:3]).astype(np.float32)
    faces = []
    for a in range(3):
        for side, sgn in ((root[a], -1), (root[3 + a], 1)):
            on = rc.copy()
            on[a] = side
            out = on.copy()
            out[a] = np.float32(side + np.float32(sgn) * size[a] * half)
            faces += [on, out]
    origins.append(np.array(faces, np.float32))
    o = np.concatenate(origins).astype(np.float32)
    axes = np.concatenate([np.eye(3), -np.eye(3)]).astype(np.float32)
    pos = np.repeat(o, 6, axis=0)
    nrm = np.tile(axes, (len(o), 1))
    with port.exact_log2():
        for r in (res, np.float32(res * np.float32(4))):
            got = tree.gi_cone_trace(pos, nrm, r)
            assert_bits_equal(got, orc.gi_cone_trace(pos, nrm, r), f"{name} mid-plane cone_trace res={r}")
            assert got.max() > 0


# ---- e. deep trees ------------------------------------------------------------------------------------------------
def _deep_scene(depth, scale):
    """Four small, far-apart, nearly horizontal triangles with tilted vertex normals (so that cones of every direction
    see lit lobes) in a root box of about 1 x 1 x 1; light and film cameras close above the second one."""
    rng = np.random.default_rng(depth)
    centres = np.array([[-0.5, -0.5, -0.5], [0.5, 0.4, 0.3], [0.1, -0.2, 0.45], [-0.3, 0.5, -0.1]], np.float32)
    shape = np.array([[-1, 0, -1], [1, 0, -0.6], [0, 0, 1]], np.float32)
    off = (shape + rng.uniform(-0.2, 0.2, (4, 3, 3))).astype(np.float32) * np.float32(scale)
    tri = (centres[:, None, :] + off).astype(np.float32)
    n = np.concatenate([rng.uniform(-0.8, 0.8, (4, 3, 1)), np.ones((4, 3, 1)), rng.uniform(-0.8, 0.8, (4, 3, 1))],
                       axis=2)
    nrm = (n / np.linalg.norm(n, axis=2, keepdims=True)).astype(np.float32)
    c = tri[1].mean(axis=0).astype(np.float32)
    s = np.float32(scale)
    light10 = np.array([CAM_LIGHT[0], *(c + s * np.array([1, 3, 0.5], np.float32)), *c, 0, 0, 1], np.float32)
    cam10 = np.array([CAM_LIGHT[0], *(c + s * np.array([-1, 2.5, 1.5], np.float32)), *c, 0, 0, 1], np.float32)
    return tri, nrm, light10, cam10


@pytest.mark.parametrize("depth,scale", [(12, 3e-2), (17, 3e-3)])
def test_deep_trees_vs_oracle(gpu, port, depth, scale):
    """The path cache at L = 11 and L = 16 (7 L words per thread: in k_gi_cone_points' shared memory, and in the film
    kernel's traversal-stack column)."""
    assert depth <= gpu.VRT_MAX_DEPTH
    tri, nrm, light10, cam10 = _deep_scene(depth, scale)
    tree = gpu.Octree.build(tri, nrm, depth)
    orc = port.build(tri, nrm, depth)
    try:
        assert tree.info()["max_depth"] == depth
        leaves_equal(tree.leaves(), orc.leaves())
        tree.gi_init()
        tree.gi_splat(_cam(gpu, light10, 128, 128, 4), GI_KD)
        tree.gi_filter()
        orc.gi_reset()
        orc.gi_splat(light10, 1.0, 128, 128, 4, GI_KD)
        orc.gi_filter()
        assert (tree.gi_level(depth - 1)[1] > 0).any(), "the leaf level must be lit"
        _levels_vs_oracle(tree, orc, depth, f"depth {depth}")
        res = gi_res(orc.root_aabb(), depth)
        pos, nrm_h = _hits(port, orc, cam10, 48, 48)
        nx, ny, spp = 24, 24, 4
        cam = _cam(gpu, cam10, nx, ny, spp)
        with port.exact_log2():
            got = tree.gi_cone_trace(pos, nrm_h, res)
            assert got.max() > 0
            assert_bits_equal(got, orc.gi_cone_trace(pos, nrm_h, res), f"depth {depth} cone_trace")
            film, pl = tree.gi_render_aov(cam, GI_KD, res, planes=("indirect",))
            assert_bits_equal(film, orc.gi_render(cam10, 1.0, nx, ny, spp, res, GI_KD), f"depth {depth} film")
            ref = _oracle_planes(port, orc, depth, cam10, nx, ny, spp, res)
            assert pl["indirect"].max() > 0
            assert_bits_equal(pl["indirect"], ref["indirect"], f"depth {depth} indirect")
    finally:
        tree.close()


# ---- f. res changing between in-flight frames ---------------------------------------------------------------------
def test_res_changes_between_pipelined_frames(gpu, lit):
    """Six pipelined GI frames alternating three res values (1e-30 among them: a march past the step table), so the
    step tables of both kernel streams are rewritten while frames are in flight, and a point cone trace at a fourth
    res between two enqueues: every frame is the synchronous film of its own res.  On one handle and on
    MultiGpu([0, 0])."""
    tree, _, depth, res, cam10 = lit("atrium_d6")
    nx, ny, spp = 64, 40, 4
    cam = _cam(gpu, cam10, nx, ny, spp)
    ress = [res, np.float32(1e-30), np.float32(res * np.float32(3))] * 2
    want = [tree.gi_render(cam, GI_KD, r) for r in ress]
    assert not np.array_equal(want[0], want[1]) and not np.array_equal(want[0], want[2])
    pts = tree.trace_camera(_cam(gpu, cam10, 16, 16, 1))
    m = pts["hit"].astype(bool)
    res4 = np.float32(res / np.float32(2))
    cone_want = tree.gi_cone_trace(pts["pos"][m], pts["nrm"][m], res4)
    bufs = [_pinned((ny, nx, 3)) for _ in range(6)]

    def run(enqueue, sync, what):
        for k in range(6):
            enqueue(k)
            if k == 2:
                assert_bits_equal(tree.gi_cone_trace(pts["pos"][m], pts["nrm"][m], res4), cone_want,
                                  f"{what}: cone trace between enqueues")
        sync()
        for k in range(6):
            assert_bits_equal(bufs[k].numpy(), want[k], f"{what}: frame {k}")
            bufs[k].fill_(7)

    run(lambda k: tree.gi_render_bands_async(cam, GI_KD, ress[k], bufs[k].data_ptr(), ny, 0, 1), tree.sync,
        "one handle")
    mg = gpu.MultiGpu(tree, [0, 0])
    try:
        mg.gi_init()
        mg.gi_splat(_cam(gpu, CAM_LIGHT, 192, 192, 4), GI_KD)
        mg.gi_filter()
        run(lambda k: mg.gi_render_async(cam, GI_KD, ress[k], bufs[k].data_ptr()), mg.sync, "MultiGpu([0, 0])")
    finally:
        mg.close()


# ---- g. planar scene ----------------------------------------------------------------------------------------------
def _planar():
    """Triangles at z = 0: the unit square in two halves and two smaller ones inside it."""
    tri = np.array([[[0, 0, 0], [1, 0, 0], [1, 1, 0]], [[0, 0, 0], [1, 1, 0], [0, 1, 0]],
                    [[0.2, 0.3, 0], [0.7, 0.25, 0], [0.4, 0.8, 0]], [[0.55, 0.6, 0], [0.9, 0.7, 0], [0.6, 0.95, 0]]],
                   np.float32)
    rng = np.random.default_rng(3)
    n = np.concatenate([rng.uniform(-0.6, 0.6, (4, 3, 2)), np.ones((4, 3, 1))], axis=2)
    return tri, (n / np.linalg.norm(n, axis=2, keepdims=True)).astype(np.float32)


def _res_xy(root, depth):
    """main.cc's Res over the axes of non-zero size only."""
    s = (root[3:] - root[:3]).astype(np.float32) / np.float32(2.0 ** depth)
    return np.float32(s[s > 0].min())


def _guarded_refusals(gpu, cam, res, tree_h=None, mg_h=None):
    """Every res entry point on a real handle refuses `res` -- each first probed on a null handle, so that a library
    without the check fails here and never launches a march that does not end.  Nothing is launched."""
    L = gpu.load()
    probe = _calls(L, cam, GI_KD, res)
    calls = _calls(L, cam, GI_KD, res, tree=tree_h, mg=mg_h)
    n0 = gpu.launch_count()
    for name in probe:
        rc, msg, ok = res_refused(L, probe[name])
        if not ok:
            pytest.fail(f"{name} does not refuse res={res!r} ('{msg}'): not calling it on a real handle")
        if name.startswith("vrt_mgpu") and mg_h is None:
            continue
        rc, msg, ok = res_refused(L, calls[name])
        assert ok, f"{name}(real handle, res={res!r}) -> {rc} '{msg}'"
    assert gpu.launch_count() == n0, "a refused call launched a kernel"


def test_planar_scene(gpu, port):
    tri, nrm = _planar()
    depth = 6
    tree = gpu.Octree.build(tri, nrm, depth)
    orc = port.build(tri, nrm, depth)
    try:
        root = orc.root_aabb()
        assert_bits_equal(root, np.array([0, 0, 0, 1, 1, 0], np.float32), "root box")
        assert_bits_equal(tree.info()["root_aabb"], root, "GPU root box")
        leaves_equal(tree.leaves(), orc.leaves())
        cam10 = np.array([CAM_LIGHT[0], 0.3, 0.4, 1.2, 0.5, 0.5, 0, 0, 1, 0], np.float32)
        nx, ny, spp = 40, 30, 4
        cam = _cam(gpu, cam10, nx, ny, spp)
        rays = port.gen_rays(cam10, 1.0, nx, ny, spp)
        exp = orc.trace(rays)
        assert exp.hit.sum() > 1000
        assert compare_hits(tree.trace_camera(cam), exp, "planar") == 0
        light10 = np.array([CAM_LIGHT[0], 0.6, 0.4, 2.0, 0.5, 0.5, 0, 0, 1, 0], np.float32)
        tree.gi_init()
        tree.gi_splat(_cam(gpu, light10, 128, 128, 4), GI_KD)
        tree.gi_filter()
        orc.gi_reset()
        orc.gi_splat(light10, 1.0, 128, 128, 4, GI_KD)
        orc.gi_filter()
        _levels_vs_oracle(tree, orc, depth, "planar")
        assert gi_res(root, depth) == 0
        _guarded_refusals(gpu, cam, gi_res(root, depth), tree_h=tree._h)
        res = _res_xy(root, depth)
        assert res == np.float32(1 / 64)
        m = exp.hit.astype(bool)
        with port.exact_log2():
            got = tree.gi_cone_trace(exp.pos[m], exp.nrm[m], res)
            assert got.max() > 0
            assert_bits_equal(got, orc.gi_cone_trace(exp.pos[m], exp.nrm[m], res), "planar cone_trace")
            assert_bits_equal(tree.gi_render(cam, GI_KD, res), orc.gi_render(cam10, 1.0, nx, ny, spp, res, GI_KD),
                              "planar film")
    finally:
        tree.close()


# ---- h. refusals on real handles ----------------------------------------------------------------------------------
def test_refusals_on_real_handles(gpu, lit):
    tree, _, depth, res, cam10 = lit("atrium_d6")
    nx, ny, spp = 32, 24, 4
    cam = _cam(gpu, cam10, nx, ny, spp)
    want = tree.gi_render(cam, GI_KD, res)
    mg = gpu.MultiGpu(tree, [0, 0])
    try:
        mg.gi_init()
        mg.gi_splat(_cam(gpu, CAM_LIGHT, 192, 192, 4), GI_KD)
        mg.gi_filter()
        mg.sync()
        for bad in BAD_RES + [-res]:
            _guarded_refusals(gpu, cam, np.float32(bad), tree_h=tree._h, mg_h=mg._h)
        buf = _pinned((ny, nx, 3))
        tree.gi_render_bands_async(cam, GI_KD, res, buf.data_ptr(), ny, 0, 1)
        tree.sync()
        assert_bits_equal(buf.numpy(), want, "pipelined frame after the refusals")
        buf.fill_(7)
        mg.gi_render_async(cam, GI_KD, res, buf.data_ptr())
        mg.sync()
        assert_bits_equal(buf.numpy(), want, "MultiGpu frame after the refusals")
    finally:
        mg.close()
