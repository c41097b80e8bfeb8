"""CPU: the C restatement (oracle/vrt_oracle.c) against the golden vectors generated from
the UNMODIFIED reference (tests/golden/make_golden.py).  This is what pins the oracle."""
import glob
import os

import numpy as np
import pytest

from tests.common import assert_bits_equal

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_predicates_golden(port):
    z = np.load(os.path.join(G, "predicates.npz"))
    assert_bits_equal(port.tribox(z["centers"], z["halves"], z["tris"]), z["tribox"], "triBoxOverlap")
    assert_bits_equal(port.tri_overlap_aabb(z["boxes"], z["tris"]), z["tri_overlap_aabb"], "is_overlap")
    res, tuv = port.raytri(z["raytri_in"])
    assert_bits_equal(res, z["raytri_res"], "intersect_triangle3")
    tuv[res == 0] = 0
    assert_bits_equal(tuv, z["raytri_tuv"], "t,u,v")
    assert_bits_equal(port.aabb_isect(z["boxes"], z["slab_rays"]), z["slab"], "AABB::isect")
    assert 100 < z["tribox"].sum() < len(z["tribox"]) - 100
    assert z["raytri_res"].sum() > 50 and z["slab"].sum() > 100


def test_camera_golden(port):
    z = np.load(os.path.join(G, "camera.npz"))
    for name in ("sphere", "main", "light"):
        cam10 = z[name + "_cam10"]
        nx, ny, spp = (int(v) for v in z[name + "_dims"])
        assert_bits_equal(port.camera_matrix(cam10), z[name + "_C"], name + " C_")
        assert_bits_equal(port.gen_rays(cam10, 1.0, nx, ny, spp), z[name + "_rays"], name + " rays")


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(G, "scene_*.npz"))), ids=os.path.basename)
def test_scene_golden(port, path):
    z = np.load(path)
    tree = port.build(z["tri"], z["nrm"], int(z["depth"]))
    assert_bits_equal(tree.root_aabb(), z["root_aabb"], "root AABB")
    cells, counts, refs, boxes = tree.leaves(boxes=True)
    assert_bits_equal(cells, z["leaf_cell"], "leaf cells")
    assert_bits_equal(counts, z["leaf_count"], "leaf counts")
    assert_bits_equal(refs, z["leaf_refs"], "leaf refs")
    assert_bits_equal(boxes, z["leaf_boxes"], "leaf boxes (split recurrence)")
    h = tree.trace(z["rays"])
    assert_bits_equal(h.hit, z["hit"], "hit")
    assert_bits_equal(h.cell, z["hit_cell"], "leaf")
    assert_bits_equal(h.tri, z["hit_tri"], "triangle")
    assert_bits_equal(h.pos, z["hit_pos"], "ISect.hit")
    assert_bits_equal(h.nrm, z["hit_nrm"], "ISect.normal")


def test_gi_golden(port):
    """SURVEY.md 8(f) rows: splat -> filter -> cone trace -> trace() film against vectors produced by
    the reference's own functions (tests/golden/make_golden.py)."""
    z = np.load(os.path.join(G, "gi_atrium.npz"))
    depth = int(z["depth"])
    tree = port.build(z["tri"], z["nrm"], depth)
    lnx, lny, lspp = (int(v) for v in z["light_dims"])
    tree.gi_reset()
    tree.gi_splat(z["light_cam10"], 1.0, lnx, lny, lspp, z["kd"])
    tree.gi_filter()
    for level in range(depth):
        cells, cov, il = tree.gi_level(level)
        assert_bits_equal(cells, z[f"l{level}_cells"], f"level {level} cells")
        assert_bits_equal(cov, z[f"l{level}_cov"], f"level {level} coverage")
        assert_bits_equal(il, z[f"l{level}_illum"], f"level {level} illum")
    res = np.float32(z["res"])
    assert_bits_equal(tree.gi_cone_trace(z["cone_pos"], z["cone_nrm"], res), z["cone"], "cone_trace")
    nx, ny, spp = (int(v) for v in z["dims"])
    assert_bits_equal(tree.gi_render(z["cam10"], 1.0, nx, ny, spp, res, z["kd"]), z["film"], "trace() film")
    # the correctly rounded log2f of the device (Port.exact_log2) takes the same split levels on these vectors
    with port.exact_log2():
        assert_bits_equal(tree.gi_cone_trace(z["cone_pos"], z["cone_nrm"], res), z["cone"], "exact-mode cone_trace")
        assert_bits_equal(tree.gi_render(z["cam10"], 1.0, nx, ny, spp, res, z["kd"]), z["film"],
                          "exact-mode trace() film")


def test_textured_golden(port):
    """Triangle::get_albedo with textures and the GI rows on a textured sphere against vectors produced by the
    reference (textures as the reference's stbi_load returned them)."""
    z = np.load(os.path.join(G, "gi_textured.npz"))
    depth = int(z["depth"])
    tree = port.build(z["tri"], z["nrm"], depth)
    tree.set_materials(z["uv"], z["mtl"], z["kd"], z["mtl_tex"], [z["tex0_seen"], z["tex1_seen"]])
    assert_bits_equal(tree.albedo(z["alb_tri"], z["alb_pos"]), z["albedo"], "get_albedo")
    lnx, lny, lspp = (int(v) for v in z["light_dims"])
    tree.gi_reset()
    tree.gi_splat(z["light_cam10"], 1.0, lnx, lny, lspp, np.array([0.7, 0.6, 0.5], np.float32))
    tree.gi_filter()
    for level in range(depth):
        _, cov, il = tree.gi_level(level)
        assert_bits_equal(cov, z[f"l{level}_cov"], f"level {level} coverage")
        assert_bits_equal(il, z[f"l{level}_illum"], f"level {level} illum")
    nx, ny, spp = (int(v) for v in z["dims"])
    assert_bits_equal(tree.gi_render(z["cam10"], 1.0, nx, ny, spp, np.float32(z["res"]), np.array([0.7, 0.6, 0.5], np.float32)),
                      z["film"], "textured trace() film")


def test_film_export_golden(port):
    """Film::to_byte_array and stbi_write_hdr(Film::to_float_array) of the reference (tests/golden/make_golden_film.py)
    against the restatement's per-pixel encoders and the product's host-side .hdr writer (vrt_hdr_file: header +
    per-component RLE, no device involved)."""
    from voxelraytrace20190722_b200 import capi
    z = np.load(os.path.join(G, "film_export.npz"))
    for name in ("wide", "big", "narrow"):
        film = z[name]
        assert_bits_equal(port.film_rgb8(film), z[name + "_rgb8"], name + " to_byte_array")
        hdr = capi.hdr_file(port.film_rgbe(film))
        assert hdr == z[name + "_hdr"].tobytes(), name + ": .hdr file differs from stbi_write_hdr's"
    # the narrow film is written flat: its payload IS the per-pixel RGBE encoding
    nar = z["narrow_hdr"].tobytes()
    assert nar.endswith(port.film_rgbe(z["narrow"]).tobytes())
