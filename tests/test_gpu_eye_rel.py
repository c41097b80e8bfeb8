"""GPU: eye-relative hull records and triangle terms of the camera launches (csrc/vrt_trace.cu eye_rel_for_launch).

Every result must be bytewise the one of the per-ray subtraction (vrt_debug_set_eye_rel off): the hit records and the
film of the headline frame, the RGBE film, pipelined frames of a moving camera whose slots are refilled while the other
stream may still read, an eye outside the root box, and a frame after vrt_update_xform has moved triangles."""
import numpy as np
import pytest

from tests.common import CAM_MAIN

pytestmark = pytest.mark.gpu


def _frame(tree, cam, torch, film_bytes_per_px=12, shadow_eps=None):
    hits = torch.zeros(cam.nx * cam.ny * cam.spp * 16, dtype=torch.uint8, device="cuda")
    film = torch.zeros(cam.nx * cam.ny * film_bytes_per_px, dtype=torch.uint8, device="cuda")
    tree.frame_bands_dev(cam, hits.data_ptr(), film.data_ptr(), 8, 0, 1, full_frame=True, shadow_eps=shadow_eps)
    tree.sync()
    return hits, film


def _on_off(tree, cam, torch, **kw):
    """The frame with the eye-relative records and without.  (A small launch with a new eye keeps the per-ray
    subtraction; the records are filled from the second launch with the same eye on, so the first one is repeated.)"""
    out = []
    for on in (True, False):
        tree.debug_set_eye_rel(on)
        if on:
            _frame(tree, cam, torch, **kw)
        n0 = tree.debug_eye_rel_launches()
        out.append(_frame(tree, cam, torch, **kw))
        assert tree.debug_eye_rel_launches() == n0 + (1 if on else 0), "records used exactly when switched on"
    tree.debug_set_eye_rel(True)
    return out


def torch_equal(x, y):
    """Bytewise equality of two device buffers as a plain bool (no tensor reaches an assertion message)."""
    return x.shape == y.shape and bool((x == y).all())


def _assert_same(a, b, what):
    for x, y, name in zip(a, b, ("hit records", "film")):
        same = torch_equal(x, y)
        assert same, f"{what}: {name} differ with the eye-relative records"


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


@pytest.fixture(scope="module")
def atrium():
    from voxelraytrace20190722_b200 import scenes
    return scenes.atrium()


def test_headline_frame_f32_and_rgbe(torch, atrium):
    from voxelraytrace20190722_b200 import capi
    tree = capi.Octree.build(*atrium, 11)
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], 3840, 2160, 4)
    before = tree.info()["device_bytes"]
    on, off = _on_off(tree, cam, torch)
    _assert_same(on, off, "headline f32")
    assert int(on[0].view(torch.int32)[3::4].sum()) > 10_000_000  # (hit flags: the frame is mostly hits)
    # the two slots of eye-relative records are counted (32 bytes per interior node, 112 per triangle)
    i = tree.info()
    assert i["device_bytes"] - before >= 2 * ((i["num_nodes"] - i["num_leaves"]) * 32 + i["num_tris"] * 112)
    tree.set_film_format("rgbe")
    on, off = _on_off(tree, cam, torch, film_bytes_per_px=4)
    _assert_same(on, off, "headline rgbe")
    tree.close()


def test_orbit_pipelined_two_streams(torch, atrium):
    """Eight frames of the config 5 orbit (2048^3, 7680x4320 x 4; primary rays only: launches with shadow rays do not
    use the records), one new eye per frame, alternating between two streams: every frame refills a slot another frame
    used two frames earlier."""
    from voxelraytrace20190722_b200 import capi
    tree = capi.Octree.build(*atrium, 12)
    n, c, r, h = 64, np.array([0.0, 0.4, 0.0]), 0.9, 0.6
    cams = []
    for k in range(8):
        a = 2 * np.pi * k / n
        eye = c + np.array([r * np.cos(a), h, r * np.sin(a)])
        cams.append(capi.Camera(CAM_MAIN[0], eye.astype(np.float32), c.astype(np.float32), (0, 1, 0), 7680, 4320, 4))
    S = [torch.cuda.Stream(), torch.cuda.Stream()]
    res = {}
    for on in (True, False):
        tree.debug_set_eye_rel(on)
        n0 = tree.debug_eye_rel_launches()
        outs = [(torch.zeros(cam.nx * cam.ny * cam.spp * 16, dtype=torch.uint8, device="cuda"),
                 torch.zeros(cam.nx * cam.ny * 12, dtype=torch.uint8, device="cuda")) for cam in cams]
        torch.cuda.synchronize()  # (the buffers are cleared on the default stream)
        for i, cam in enumerate(cams):
            hits, film = outs[i]
            with torch.cuda.stream(S[i & 1]):
                tree.set_stream(S[i & 1].cuda_stream)
                tree.frame_bands_dev(cam, hits.data_ptr(), film.data_ptr(), 8, 0, 1, full_frame=True)
        torch.cuda.synchronize()
        tree.set_stream(0)
        res[on] = outs
        assert tree.debug_eye_rel_launches() - n0 == (len(cams) if on else 0)
        if not on:
            for i in range(len(cams)):
                _assert_same(res[True][i], outs[i], f"orbit frame {i}")
    tree.close()


def test_eye_outside_root_box(torch, atrium):
    from voxelraytrace20190722_b200 import capi
    tree = capi.Octree.build(*atrium, 9)
    lo, hi = np.array(tree.info()["root_aabb"][:3]), np.array(tree.info()["root_aabb"][3:])
    eye = (hi + (hi - lo) * 0.7).astype(np.float32)
    cam = capi.Camera(CAM_MAIN[0], eye, ((lo + hi) / 2).astype(np.float32), (0, 1, 0), 640, 360, 4)
    on, off = _on_off(tree, cam, torch)
    _assert_same(on, off, "eye outside")
    assert int(on[0].view(torch.int32)[3::4].sum()) > 1000
    tree.close()


def test_frame_after_update(torch, atrium):
    """A slot filled before vrt_update_xform must not be reused after it: the same eye again gives the frame of the
    new pose."""
    from voxelraytrace20190722_b200 import capi
    tree = capi.Octree.build(*atrium, 9)
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], 640, 360, 4)
    _frame(tree, cam, torch)
    first = _frame(tree, cam, torch)  # (the second launch with this eye fills a slot)
    T = tree.info()["num_tris"]
    m = np.eye(3, 4, dtype=np.float32)
    m[:, 3] = (0.03, 0.05, -0.02)
    tree.update_xform([(0, T // 2, m)])
    on, off = _on_off(tree, cam, torch)
    _assert_same(on, off, "after update")
    moved = not torch_equal(first[0], on[0])
    assert moved, "the update moved nothing the camera sees"
    tree.close()


def test_slot_read_on_both_streams_then_refilled(torch, atrium):
    """A slot read by launches on two streams is refilled only after both: stream A fills slot 0 for eye E (8K frame),
    stream B reads it in a small launch, A fills slot 1 for a new eye, then B refills slot 0 for another new eye while
    A's first launch may still be reading it.  Every launch must give the result of the per-ray path."""
    from voxelraytrace20190722_b200 import capi
    tree = capi.Octree.build(*atrium, 12)
    c, r, h = np.array([0.0, 0.4, 0.0]), 0.9, 0.6
    cams = []
    for k in range(3):
        a = 2 * np.pi * k / 64
        eye = c + np.array([r * np.cos(a), h, r * np.sin(a)])
        cams.append(capi.Camera(CAM_MAIN[0], eye.astype(np.float32), c.astype(np.float32), (0, 1, 0), 7680, 4320, 4))
    # (stream index, camera, rect)
    seq = [(0, cams[0], None), (1, cams[0], (0, 0, 64, 64)), (0, cams[1], None), (1, cams[2], None)]
    S = [torch.cuda.Stream(), torch.cuda.Stream()]
    res = {}
    for on in (True, False):
        tree.debug_set_eye_rel(on)
        n0 = tree.debug_eye_rel_launches()
        # (zeroed: a rect launch writes only the head of its buffer)
        outs = [torch.zeros(cam.nx * cam.ny * cam.spp * 16, dtype=torch.uint8, device="cuda") for _, cam, _ in seq]
        torch.cuda.synchronize()  # (the buffers are cleared on the default stream)
        for (si, cam, rect), out in zip(seq, outs):
            with torch.cuda.stream(S[si]):
                tree.set_stream(S[si].cuda_stream)
                tree.trace_camera_dev(cam, out.data_ptr(), rect=rect, compact=True)
        torch.cuda.synchronize()
        tree.set_stream(0)
        assert tree.debug_eye_rel_launches() - n0 == (len(seq) if on else 0)
        res[on] = outs
    for i, (a, b) in enumerate(zip(res[True], res[False])):
        same = torch_equal(a, b)
        assert same, f"launch {i}: hit records differ with the eye-relative records"
    tree.close()
