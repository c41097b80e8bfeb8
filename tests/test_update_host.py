"""CPU: the animated-geometry calls of the Python binding (Octree.update / update_dev / update_xform, MultiGpu.update /
update_xform) -- no CPU fallback without a device, and malformed triangle arrays and transform tuples rejected before
the library is called."""
import numpy as np
import pytest

from voxelraytrace20190722_b200 import capi

M = np.eye(3, 4, dtype=np.float32)


def _handles():
    tree = capi.Octree(None)  # without a device no octree or replica can be made
    mg = capi.MultiGpu.__new__(capi.MultiGpu)
    mg._h, mg.max_depth, mg.num_tris = None, 6, 2
    return tree, mg


def test_updates_without_device_raise():
    capi.load()
    if capi.device_count() > 0:
        pytest.skip("CUDA device present")
    tree, mg = _handles()
    tri = np.zeros((2, 9), np.float32)
    with pytest.raises(capi.VrtError):
        tree.update(tri)
    with pytest.raises(capi.VrtError):
        tree.update_dev(16, 0, 2)
    with pytest.raises(capi.VrtError):
        tree.update_xform([(0, 1, M)])
    with pytest.raises(capi.VrtError):
        mg.update(tri)
    with pytest.raises(capi.VrtError):
        mg.update_xform([(0, 1, M)])


@pytest.mark.parametrize("xforms", [
    [],
    [(0, 1)],
    [(0, 1, M, np.eye(3), "extra")],
    [(0, 1, np.eye(3, dtype=np.float32))],
    [(0, 1, np.eye(4, dtype=np.float32))],
    [(0, 1, M, np.eye(4, dtype=np.float32))],
    [(-1, 1, M)],
    [(0, -2, M)],
    [(0, 2 ** 32, M)],
    ["not a tuple"],
])
def test_bad_xform_tuples_rejected(xforms):
    tree, mg = _handles()
    with pytest.raises(ValueError):
        tree.update_xform(xforms)
    with pytest.raises(ValueError):
        mg.update_xform(xforms)


def test_bad_triangle_shapes_rejected():
    tree, mg = _handles()
    for tri, nrm in ((np.zeros((2, 8), np.float32), None), (np.zeros(0, np.float32), None),
                     (np.zeros((2, 9), np.float32), np.zeros((1, 9), np.float32))):
        with pytest.raises(ValueError):
            tree.update(tri, nrm)
        with pytest.raises(ValueError):
            mg.update(tri, nrm)
    with pytest.raises(ValueError):  # the replicas' triangle count
        mg.update(np.zeros((3, 9), np.float32))


def test_default_normal_matrix_is_inverse_transpose():
    m = np.array([[2, 0, 0, 1], [0, 0.5, 0, 2], [0, 0, 4, 3]], np.float32)
    n = capi.xform_normal_matrix(m)
    assert n.dtype == np.float32
    assert np.array_equal(n, np.diag([0.5, 2, 0.25]).astype(np.float32))
    t = capi._xform_table([(3, 4, m)])
    assert (t[0].first_tri, t[0].num_tris) == (3, 4)
    assert np.array_equal(np.array(t[0].m[:], np.float32), m.reshape(-1))
    assert np.array_equal(np.array(t[0].n[:], np.float32), n.reshape(-1))
