"""ctypes binding of libvrt.so (include/vrt.h) -- the host-side mirror used by
tests and bench.py.  Python is only plumbing here: every compute call lands in
the CUDA library; if the library or a CUDA device is missing the calls raise
:class:`VrtError` (there is no CPU fallback and no route into oracle/).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

VRT_MAX_DEPTH = 17
VRT_NO_TRI = 0xFFFFFFFF


class VrtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libvrt error {code}: {msg}")
        self.code = code


class vrt_camera(C.Structure):
    _fields_ = [("C", C.c_float * 16), ("z", C.c_float), ("tmin", C.c_float), ("tmax", C.c_float),
                ("nx", C.c_int32), ("ny", C.c_int32), ("spp", C.c_int32)]


class vrt_shade(C.Structure):
    _fields_ = [("light_dir", C.c_float * 3), ("kd", C.c_float), ("shadow_eps", C.c_float), ("shadow", C.c_int32)]


class vrt_bands(C.Structure):
    _fields_ = [("band_h", C.c_int32), ("band_first", C.c_int32), ("band_stride", C.c_int32)]


class vrt_texture(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("channels", C.c_int32), ("data", C.c_void_p)]


class vrt_gi_aov(C.Structure):
    """The per-pixel planes of vrt_gi_render_aov(_dev); a null member is not written."""
    _fields_ = [("albedo", C.c_void_p), ("direct", C.c_void_p), ("indirect", C.c_void_p), ("normal", C.c_void_p),
                ("hits", C.c_void_p)]


GI_AOV_PLANES = ("albedo", "direct", "indirect", "normal", "hits")


class vrt_xform(C.Structure):
    """One range of vrt_update_xform: p' = M[:, :3] p + M[:, 3], n' = N n for triangles [first_tri, +num_tris)."""
    _fields_ = [("first_tri", C.c_uint32), ("num_tris", C.c_uint32), ("m", C.c_float * 12), ("n", C.c_float * 9)]


class vrt_tree_info(C.Structure):
    _fields_ = [("num_tris", C.c_uint32), ("max_depth", C.c_int32), ("root_aabb", C.c_float * 6),
                ("num_nodes", C.c_uint64), ("num_leaves", C.c_uint64), ("num_refs", C.c_uint64),
                ("level_offset", C.c_uint64 * (VRT_MAX_DEPTH + 1)), ("device_bytes", C.c_uint64),
                ("build_ms", C.c_double)]


class vrt_tree_view(C.Structure):
    _fields_ = [("leaf_cell", C.c_void_p), ("leaf_count", C.c_void_p), ("leaf_refs", C.c_void_p),
                ("nodes", C.c_void_p)]


HIT_DTYPE = np.dtype([("hit", "<u4"), ("tri", "<u4"), ("cell", "<u4", (3,)), ("t", "<f4"),
                      ("pos", "<f4", (3,)), ("nrm", "<f4", (3,))])
HIT16_DTYPE = np.dtype([("leaf", "<u4"), ("tri", "<u4"), ("t", "<f4"), ("hit", "<u4")])
RAY_DTYPE = np.dtype([("o", "<f4", (3,)), ("d", "<f4", (3,)), ("tmin", "<f4"), ("tmax", "<f4")])
assert HIT_DTYPE.itemsize == 48 and HIT16_DTYPE.itemsize == 16 and RAY_DTYPE.itemsize == 32

# every symbol include/vrt.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "vrt_abi_version", "vrt_last_error", "vrt_device_count", "vrt_launch_count",
    "vrt_build", "vrt_build_dev", "vrt_build_indexed", "vrt_rebuild", "vrt_tree_free", "vrt_tree_get_info",
    "vrt_tree_export", "vrt_tree_import", "vrt_tree_set_stream", "vrt_tree_blob_dev",
    "vrt_tree_from_blob_dev", "vrt_tree_save", "vrt_tree_load", "vrt_camera_init", "vrt_gen_rays", "vrt_trace_rays",
    "vrt_trace_rays_dev", "vrt_trace_camera", "vrt_trace_camera_dev", "vrt_trace_camera16_dev",
    "vrt_render_camera", "vrt_render_camera_dev", "vrt_render_camera_async", "vrt_band_rows", "vrt_render_bands_dev", "vrt_render_bands_async",
    "vrt_trace_bands16_dev", "vrt_count_camera", "vrt_frame_bands_dev", "vrt_frame_bands_peer_dev",
    "vrt_dev_alloc", "vrt_dev_free", "vrt_host_register", "vrt_host_unregister", "vrt_ipc_export", "vrt_ipc_open", "vrt_ipc_close", "vrt_tree_sync",
    "vrt_last_kernel_ms", "vrt_mean_kernel_ms", "vrt_debug_general_order_calls", "vrt_debug_param_check", "vrt_debug_pair_total", "vrt_debug_set_hull", "vrt_debug_set_eye_rel", "vrt_debug_eye_rel_launches", "vrt_debug_hull_stats", "vrt_build_ex", "vrt_mgpu_create", "vrt_mgpu_num_devices",
    "vrt_mgpu_render_async", "vrt_mgpu_sync", "vrt_mgpu_render", "vrt_mgpu_free", "vrt_set_film_format",
    "vrt_film_pixel_bytes", "vrt_hdr_file", "vrt_mgpu_set_film_format", "vrt_film_encode", "vrt_set_materials", "vrt_albedo", "vrt_gi_init", "vrt_gi_splat_camera", "vrt_gi_filter",
    "vrt_gi_get_level", "vrt_gi_cone_trace", "vrt_gi_render_camera", "vrt_gi_render_camera_dev", "vrt_tribox_batch",
    "vrt_tri_overlap_aabb_batch", "vrt_raytri_batch", "vrt_aabb_isect_batch",
    "vrt_gi_render_bands_async", "vrt_mgpu_set_materials", "vrt_mgpu_gi_init", "vrt_mgpu_gi_splat_camera",
    "vrt_mgpu_gi_filter", "vrt_mgpu_gi_render_async", "vrt_mgpu_gi_render", "vrt_mgpu_mean_kernel_ms",
    "vrt_gi_render_aov", "vrt_gi_render_aov_dev",
    "vrt_gi_render_aov_bands_async", "vrt_mgpu_gi_render_aov_async", "vrt_mgpu_gi_render_aov",
    "vrt_update_triangles", "vrt_update_triangles_dev", "vrt_update_xform", "vrt_mgpu_update_triangles",
    "vrt_mgpu_update_xform",
]

_lib = None


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """dlopen libvrt.so (building it in-tree with nvcc when stale and possible)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB
    if build_if_missing and _build.is_stale():
        try:
            _build.build_native()
        except Exception as e:  # keep a prebuilt .so if nvcc is unavailable
            if not os.path.exists(path):
                raise VrtError(-2, f"libvrt.so missing and cannot be built: {e}") from e
    if not os.path.exists(path):
        raise VrtError(-2, "libvrt.so missing (no CPU fallback exists)")
    L = C.CDLL(path)
    vp, u32, u64, i32, f32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int, C.c_float
    L.vrt_abi_version.restype = i32
    L.vrt_last_error.restype = C.c_char_p
    L.vrt_device_count.restype = i32
    L.vrt_launch_count.restype = u64
    L.vrt_build.argtypes = [vp, vp, u32, i32, C.POINTER(vp)]
    L.vrt_build_dev.argtypes = [vp, vp, u32, i32, C.POINTER(vp)]
    L.vrt_rebuild.argtypes = [vp, i32]
    L.vrt_tree_free.argtypes = [vp]
    L.vrt_tree_free.restype = None
    L.vrt_tree_get_info.argtypes = [vp, C.POINTER(vrt_tree_info)]
    L.vrt_tree_export.argtypes = [vp, C.POINTER(vrt_tree_view)]
    L.vrt_tree_import.argtypes = [vp, vp, u32, i32, vp, u64, vp, vp, vp, C.POINTER(vp)]
    L.vrt_tree_set_stream.argtypes = [vp, vp]
    L.vrt_tree_blob_dev.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.vrt_tree_from_blob_dev.argtypes = [vp, u64, C.POINTER(vp)]
    L.vrt_tree_save.argtypes = [vp, C.c_char_p]
    L.vrt_tree_load.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.vrt_camera_init.argtypes = [vp, f32, i32, i32, i32, C.POINTER(vrt_camera)]
    L.vrt_gen_rays.argtypes = [C.POINTER(vrt_camera), i32, i32, i32, i32, vp]
    L.vrt_trace_rays.argtypes = [vp, vp, u64, vp]
    L.vrt_trace_rays_dev.argtypes = [vp, vp, u64, vp]
    for name in ("vrt_trace_camera", "vrt_trace_camera_dev", "vrt_trace_camera16_dev"):
        getattr(L, name).argtypes = [vp, C.POINTER(vrt_camera), i32, i32, i32, i32, vp]
    for name in ("vrt_render_camera", "vrt_render_camera_dev", "vrt_render_camera_async"):
        getattr(L, name).argtypes = [vp, C.POINTER(vrt_camera), C.POINTER(vrt_shade), i32, i32, i32, i32, vp]
    L.vrt_band_rows.argtypes = [C.POINTER(vrt_camera), C.POINTER(vrt_bands)]
    L.vrt_render_bands_dev.argtypes = [vp, C.POINTER(vrt_camera), C.POINTER(vrt_shade), C.POINTER(vrt_bands), vp]
    L.vrt_render_bands_async.argtypes = L.vrt_render_bands_dev.argtypes
    L.vrt_trace_bands16_dev.argtypes = [vp, C.POINTER(vrt_camera), C.POINTER(vrt_bands), vp]
    L.vrt_count_camera.argtypes = [vp, C.POINTER(vrt_camera), i32, i32, i32, i32, vp]
    L.vrt_frame_bands_dev.argtypes = [vp, C.POINTER(vrt_camera), C.POINTER(vrt_shade), C.POINTER(vrt_bands), vp, vp]
    L.vrt_frame_bands_peer_dev.argtypes = L.vrt_frame_bands_dev.argtypes
    L.vrt_dev_alloc.argtypes = [u64, C.POINTER(vp)]
    L.vrt_dev_free.argtypes = [vp]
    L.vrt_host_register.argtypes = [vp, u64]
    L.vrt_host_unregister.argtypes = [vp]
    L.vrt_ipc_export.argtypes = [vp, vp]
    L.vrt_ipc_open.argtypes = [vp, C.POINTER(vp)]
    L.vrt_ipc_close.argtypes = [vp]
    L.vrt_debug_general_order_calls.restype = u64
    L.vrt_debug_param_check.argtypes = [vp]
    L.vrt_debug_pair_total.argtypes = [vp, u64, vp]
    L.vrt_debug_set_hull.argtypes = [vp, i32]
    L.vrt_debug_set_eye_rel.argtypes = [vp, i32]
    L.vrt_debug_eye_rel_launches.argtypes = [vp, vp]
    L.vrt_debug_hull_stats.argtypes = [vp]
    L.vrt_mgpu_create.argtypes = [vp, i32, vp, C.POINTER(vp)]
    L.vrt_mgpu_num_devices.argtypes = [vp]
    L.vrt_set_film_format.argtypes = [vp, C.c_int32]
    L.vrt_mgpu_set_film_format.argtypes = [vp, C.c_int32]
    L.vrt_film_pixel_bytes.argtypes = [C.c_int32]
    L.vrt_film_encode.argtypes = [vp, vp, C.c_uint64, C.c_int32, vp]
    L.vrt_hdr_file.restype = C.c_int64
    L.vrt_hdr_file.argtypes = [vp, C.c_int32, C.c_int32, vp, C.c_uint64]
    L.vrt_mgpu_render_async.argtypes = [vp, C.POINTER(vrt_camera), C.POINTER(vrt_shade), vp]
    L.vrt_mgpu_render.argtypes = [vp, C.POINTER(vrt_camera), C.POINTER(vrt_shade), vp]
    L.vrt_mgpu_sync.argtypes = [vp]
    L.vrt_mgpu_free.argtypes = [vp]
    L.vrt_mgpu_free.restype = None
    L.vrt_gi_init.argtypes = [vp]
    L.vrt_build_indexed.argtypes = [vp, u64, vp, u64, vp, C.c_uint32, i32, C.POINTER(vp)]
    L.vrt_set_materials.argtypes = [vp, vp, vp, C.c_uint32, vp, vp, C.c_uint32, vp]
    L.vrt_albedo.argtypes = [vp, vp, vp, u64, vp, vp]
    L.vrt_gi_splat_camera.argtypes = [vp, C.POINTER(vrt_camera), vp]
    L.vrt_gi_filter.argtypes = [vp]
    L.vrt_gi_get_level.argtypes = [vp, i32, vp, vp]
    L.vrt_gi_cone_trace.argtypes = [vp, vp, vp, u64, f32, vp]
    L.vrt_gi_render_camera.argtypes = [vp, C.POINTER(vrt_camera), vp, f32, i32, i32, i32, i32, vp]
    L.vrt_gi_render_camera_dev.argtypes = L.vrt_gi_render_camera.argtypes
    L.vrt_gi_render_bands_async.argtypes = [vp, C.POINTER(vrt_camera), vp, f32, C.POINTER(vrt_bands), vp]
    L.vrt_gi_render_aov.argtypes = [vp, C.POINTER(vrt_camera), vp, f32, i32, i32, i32, i32, vp, C.POINTER(vrt_gi_aov)]
    L.vrt_gi_render_aov_dev.argtypes = L.vrt_gi_render_aov.argtypes
    L.vrt_gi_render_aov_bands_async.argtypes = [vp, C.POINTER(vrt_camera), vp, f32, C.POINTER(vrt_bands), vp,
                                                C.POINTER(vrt_gi_aov)]
    L.vrt_mgpu_gi_render_aov_async.argtypes = [vp, C.POINTER(vrt_camera), vp, f32, vp, C.POINTER(vrt_gi_aov)]
    L.vrt_mgpu_gi_render_aov.argtypes = L.vrt_mgpu_gi_render_aov_async.argtypes
    L.vrt_mgpu_set_materials.argtypes = [vp, vp, vp, C.c_uint32, vp, vp, C.c_uint32, vp]
    L.vrt_mgpu_gi_init.argtypes = [vp]
    L.vrt_mgpu_gi_splat_camera.argtypes = [vp, C.POINTER(vrt_camera), vp]
    L.vrt_mgpu_gi_filter.argtypes = [vp]
    L.vrt_mgpu_gi_render_async.argtypes = [vp, C.POINTER(vrt_camera), vp, f32, vp]
    L.vrt_mgpu_gi_render.argtypes = L.vrt_mgpu_gi_render_async.argtypes
    L.vrt_mgpu_mean_kernel_ms.restype = C.c_double
    L.vrt_mgpu_mean_kernel_ms.argtypes = [vp, i32, i32]
    L.vrt_tree_sync.argtypes = [vp]
    L.vrt_update_triangles.argtypes = [vp, vp, vp, u32, i32]
    L.vrt_update_triangles_dev.argtypes = [vp, vp, vp, u32, i32]
    L.vrt_update_xform.argtypes = [vp, vp, u32, i32]
    L.vrt_mgpu_update_triangles.argtypes = [vp, vp, vp, u32, i32]
    L.vrt_mgpu_update_xform.argtypes = [vp, vp, u32, i32]
    L.vrt_mean_kernel_ms.restype = C.c_double
    L.vrt_mean_kernel_ms.argtypes = [vp, i32]
    L.vrt_last_kernel_ms.restype = C.c_double
    L.vrt_last_kernel_ms.argtypes = [vp]
    L.vrt_tribox_batch.argtypes = [vp, vp, vp, u64, vp]
    L.vrt_tri_overlap_aabb_batch.argtypes = [vp, vp, u64, vp]
    L.vrt_raytri_batch.argtypes = [vp, u64, vp, vp]
    L.vrt_aabb_isect_batch.argtypes = [vp, vp, u64, vp]
    for s in SYMBOLS:
        f = getattr(L, s)
        if f.restype is C.c_int and s not in ("vrt_abi_version", "vrt_device_count"):
            pass
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise VrtError(rc, load().vrt_last_error().decode(errors="replace"))


def _check_pos(rc):
    if rc < 0:
        raise VrtError(rc, load().vrt_last_error().decode(errors="replace"))
    return rc


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, np.float32)
    return a if shape is None else a.reshape(shape)


def _shade(light, kd, shadow_eps):
    """vrt_shade: light direction (default main.cc:72), kd, optional shadow rays (eps > 0)."""
    return vrt_shade((C.c_float * 3)(*(default_light() if light is None else light)), float(kd),
                     float(shadow_eps or 0.0), 1 if shadow_eps else 0)


def device_count() -> int:
    return int(load().vrt_device_count())


def launch_count() -> int:
    return int(load().vrt_launch_count())


def default_light():
    """normalize(Vec3{1,10,1}) with the reference's float arithmetic (main.cc:72)."""
    v = np.array([1, 10, 1], np.float32)
    s = np.float32(0)
    for k in range(3):
        s = np.float32(s + np.float32(v[k] * v[k]))
    return (v / np.sqrt(s, dtype=np.float32)).astype(np.float32)


class Camera:
    """Mirror of the reference's ``Camera(fov, eye, spot, up)`` + ``Film(w,h,nx,ny)``
    (camera.h:24-29,70-83)."""

    def __init__(self, fov, eye, spot, up, nx, ny, spp=1, film_h=1.0):
        self.cam10 = np.array([fov, *eye, *spot, *up], np.float32)
        self.c = vrt_camera()
        _check(load().vrt_camera_init(_ptr(self.cam10), float(film_h), int(nx), int(ny), int(spp), C.byref(self.c)))
        self.nx, self.ny, self.spp, self.film_h = int(nx), int(ny), int(spp), float(film_h)

    @property
    def matrix(self):
        return np.array(self.c.C[:], np.float32)

    def gen_rays(self, rect=None):
        """gen_rays1/gen_rays4 for every pixel of ``rect`` -> structured RAY array."""
        x0, y0, x1, y1 = rect if rect else (0, 0, self.nx, self.ny)
        out = np.zeros((y1 - y0) * (x1 - x0) * self.spp, RAY_DTYPE)
        _check(load().vrt_gen_rays(C.byref(self.c), x0, y0, x1, y1, _ptr(out)))
        return out


class Octree:
    """Owner of a ``vrt_tree*`` -- mirror of ``gi::VoxelOctree`` + ``ray_march_init``."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle)

    # ---- construction ------------------------------------------------------
    @classmethod
    def build(cls, tri_xyz, tri_nrm, max_depth):
        """gi::ray_march_init(&root, voxels, max_depth) -- host arrays in."""
        tri = _f32(tri_xyz, (-1, 9))
        nrm = None if tri_nrm is None else _f32(tri_nrm, (-1, 9))
        h = C.c_void_p()
        _check(load().vrt_build(_ptr(tri), _ptr(nrm), tri.shape[0], int(max_depth), C.byref(h)))
        return cls(h.value)

    @classmethod
    def build_indexed(cls, vertices, normals, index3, max_depth):
        """tinyobj-style arrays: vertices [nv,3], normals [nn,3] or None, index3 [T,3,3] int32
        (vertex_index, normal_index, texcoord_index per face vertex)."""
        v = np.ascontiguousarray(vertices, np.float32).reshape(-1, 3)
        n = None if normals is None else np.ascontiguousarray(normals, np.float32).reshape(-1, 3)
        idx = np.ascontiguousarray(index3, np.int32).reshape(-1, 3, 3)
        h = C.c_void_p()
        _check(load().vrt_build_indexed(_ptr(v), len(v), None if n is None else _ptr(n), 0 if n is None else len(n),
                                        _ptr(idx), len(idx), int(max_depth), C.byref(h)))
        return cls(h.value)

    @classmethod
    def build_dev(cls, d_tri_ptr, d_nrm_ptr, num_tris, max_depth):
        h = C.c_void_p()
        _check(load().vrt_build_dev(C.c_void_p(d_tri_ptr), C.c_void_p(d_nrm_ptr) if d_nrm_ptr else None,
                                    int(num_tris), int(max_depth), C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_leaves(cls, tri_xyz, tri_nrm, max_depth, root_aabb, leaf_cell, leaf_count, leaf_refs):
        tri = _f32(tri_xyz, (-1, 9))
        nrm = None if tri_nrm is None else _f32(tri_nrm, (-1, 9))
        root = _f32(root_aabb)
        cell = np.ascontiguousarray(leaf_cell, np.uint32)
        cnt = np.ascontiguousarray(leaf_count, np.uint32)
        refs = np.ascontiguousarray(leaf_refs, np.uint32)
        h = C.c_void_p()
        _check(load().vrt_tree_import(_ptr(tri), _ptr(nrm), tri.shape[0], int(max_depth), _ptr(root), len(cnt),
                                      _ptr(cell), _ptr(cnt), _ptr(refs), C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_blob_dev(cls, d_ptr, nbytes):
        h = C.c_void_p()
        _check(load().vrt_tree_from_blob_dev(C.c_void_p(d_ptr), int(nbytes), C.byref(h)))
        return cls(h.value)

    @classmethod
    def load(cls, path):
        """Octree checkpoint written by :meth:`save` -> a usable handle (no rebuild)."""
        h = C.c_void_p()
        _check(load().vrt_tree_load(os.fsencode(path), C.byref(h)))
        return cls(h.value)

    def save(self, path):
        _check(load().vrt_tree_save(self._h, os.fsencode(path)))

    def rebuild(self, max_depth):
        _check(load().vrt_rebuild(self._h, int(max_depth)))

    # ---- animated geometry (include/vrt.h vrt_update_*) ------------------------------------------------------------
    def _update_args(self, num_tris, max_depth):
        """max_depth None -> the handle's current depth; a triangle count other than the handle's raises."""
        i = self.info()
        if num_tris is not None and num_tris != i["num_tris"]:
            raise ValueError(f"update needs {i['num_tris']} triangles (the handle's count), got {num_tris}")
        return i["max_depth"] if max_depth is None else int(max_depth)

    def update(self, tri_xyz, tri_nrm=None, max_depth=None):
        """Replace the handle's triangles (same count; normals exactly when it was built with them) and rebuild at
        max_depth (None: the current depth).  Materials and film format stay; call gi_init again."""
        tri, nrm = _update_arrays(tri_xyz, tri_nrm)
        depth = self._update_args(tri.shape[0], max_depth)
        _check(load().vrt_update_triangles(self._h, _ptr(tri), _ptr(nrm), tri.shape[0], depth))

    def update_dev(self, d_tri_ptr, d_nrm_ptr, num_tris, max_depth=None):
        """update() from device arrays [num_tris, 9] float32 (d_nrm_ptr 0 / None: no normals)."""
        depth = self._update_args(int(num_tris), max_depth)
        _check(load().vrt_update_triangles_dev(self._h, C.c_void_p(int(d_tri_ptr or 0) or None),
                                               C.c_void_p(int(d_nrm_ptr or 0) or None), int(num_tris), depth))

    def update_xform(self, xforms, max_depth=None):
        """Set the pose to the rest pose (the triangles of the last build or update()) with ranges moved: xforms is a
        list of (first, count, M 3x4[, N 3x3]); N defaults to the float64 inverse transpose of M[:, :3]."""
        arr = _xform_table(xforms)
        depth = self._update_args(None, max_depth)
        _check(load().vrt_update_xform(self._h, C.cast(arr, C.c_void_p), len(arr), depth))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            load().vrt_tree_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # interpreter shutdown: module globals are already gone
            pass

    def set_stream(self, cuda_stream_ptr):
        _check(load().vrt_tree_set_stream(self._h, C.c_void_p(cuda_stream_ptr)))

    # ---- inspection --------------------------------------------------------
    def info(self):
        i = vrt_tree_info()
        _check(load().vrt_tree_get_info(self._h, C.byref(i)))
        return dict(num_tris=i.num_tris, max_depth=i.max_depth, root_aabb=np.array(i.root_aabb[:], np.float32),
                    num_nodes=int(i.num_nodes), num_leaves=int(i.num_leaves), num_refs=int(i.num_refs),
                    level_offset=[int(v) for v in i.level_offset], device_bytes=int(i.device_bytes),
                    build_ms=float(i.build_ms))

    def leaves(self, nodes=False):
        """(leaf_cell [L,3], leaf_count [L], leaf_refs [R]) in Morton order."""
        i = self.info()
        cell = np.zeros((i["num_leaves"], 3), np.uint32)
        cnt = np.zeros(i["num_leaves"], np.uint32)
        refs = np.zeros(i["num_refs"], np.uint32)
        nd = np.zeros((i["num_nodes"], 2), np.uint32) if nodes else None
        v = vrt_tree_view(_ptr(cell), _ptr(cnt), _ptr(refs), _ptr(nd))
        _check(load().vrt_tree_export(self._h, C.byref(v)))
        return (cell, cnt, refs, nd) if nodes else (cell, cnt, refs)

    def blob_dev(self):
        p, n = C.c_void_p(), C.c_uint64()
        _check(load().vrt_tree_blob_dev(self._h, C.byref(p), C.byref(n)))
        return p.value, int(n.value)

    @property
    def last_kernel_ms(self):
        return float(load().vrt_last_kernel_ms(self._h))

    # ---- queries -----------------------------------------------------------
    def trace_rays(self, rays):
        """gi::ray_march for a batch of rays (structured RAY array or [R,8] float32)."""
        rays = np.ascontiguousarray(rays)
        if rays.dtype != RAY_DTYPE:
            rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8).view(RAY_DTYPE).reshape(-1)
        out = np.zeros(len(rays), HIT_DTYPE)
        _check(load().vrt_trace_rays(self._h, _ptr(rays), len(rays), _ptr(out)))
        return out

    def trace_rays_dev(self, d_rays_ptr, n, d_out_ptr):
        _check(load().vrt_trace_rays_dev(self._h, C.c_void_p(d_rays_ptr), int(n), C.c_void_p(d_out_ptr)))

    def trace_camera(self, cam: Camera, rect=None):
        """render_mt loop replaced by one launch: gen_rays + ray_march per pixel sample."""
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        out = np.zeros((y1 - y0) * (x1 - x0) * cam.spp, HIT_DTYPE)
        _check(load().vrt_trace_camera(self._h, C.byref(cam.c), x0, y0, x1, y1, _ptr(out)))
        return out

    def trace_camera_dev(self, cam: Camera, d_out_ptr, rect=None, compact=False):
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        fn = load().vrt_trace_camera16_dev if compact else load().vrt_trace_camera_dev
        _check(fn(self._h, C.byref(cam.c), x0, y0, x1, y1, C.c_void_p(d_out_ptr)))

    def set_film_format(self, fmt):
        """'f32' (default), 'rgbe' (stbi_write_hdr's pixel encoding) or 'rgb8' (Film::to_byte_array): how every
        film-writing call of this handle stores a finished pixel."""
        self.film_format = FILM_FORMATS[fmt] if isinstance(fmt, str) else int(fmt)
        _check(load().vrt_set_film_format(self._h, self.film_format))

    def film_encode(self, film, fmt):
        """Encode a float film [..., 3] on the device: 'rgbe' -> uint8 [..., 4], 'rgb8' -> uint8 [..., 3]."""
        f = np.ascontiguousarray(film, np.float32)
        code = FILM_FORMATS[fmt]
        out = np.zeros(f.shape[:-1] + (4 if code == 1 else 3,), np.uint8)
        _check(load().vrt_film_encode(self._h, _ptr(f), f.size // 3, code, _ptr(out)))
        return out

    def _film_array(self, h, w):
        fmt = getattr(self, "film_format", 0)
        return np.zeros((h, w, 3), np.float32) if fmt == 0 else np.zeros((h, w, 4 if fmt == 1 else 3), np.uint8)

    def render(self, cam: Camera, light=None, kd=0.8, rect=None, out=None, shadow_eps=None):
        """Harness-shaded film ([h,w,3] float, or the handle's film format) through HOST buffers."""
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        sh = _shade(light, kd, shadow_eps)
        if out is None:
            out = self._film_array(y1 - y0, x1 - x0)
        _check(load().vrt_render_camera(self._h, C.byref(cam.c), C.byref(sh), x0, y0, x1, y1, _ptr(out)))
        return out

    def render_bands_dev(self, cam: Camera, d_film_ptr, band_h, band_first, band_stride, light=None, kd=0.8,
                         shadow_eps=None):
        """Rank `band_first` of `band_stride` in a row-interleaved multi-GPU frame."""
        sh = _shade(light, kd, shadow_eps)
        b = vrt_bands(int(band_h), int(band_first), int(band_stride))
        _check(load().vrt_render_bands_dev(self._h, C.byref(cam.c), C.byref(sh), C.byref(b), C.c_void_p(d_film_ptr)))

    def render_bands_async(self, cam: Camera, host_frame_ptr, band_h, band_first, band_stride, light=None, kd=0.8,
                           shadow_eps=None):
        """Rank `band_first` of `band_stride`: render this rank's bands and DMA them to their final rows
        of the full (pinned, possibly shared between the ranks) host frame; asynchronous, see sync()."""
        sh = _shade(light, kd, shadow_eps)
        b = vrt_bands(int(band_h), int(band_first), int(band_stride))
        _check(load().vrt_render_bands_async(self._h, C.byref(cam.c), C.byref(sh), C.byref(b),
                                             C.c_void_p(int(host_frame_ptr))))

    def frame_bands_dev(self, cam: Camera, d_hits_ptr, d_film_ptr, band_h, band_first, band_stride, light=None,
                        kd=0.8, full_frame=False, shadow_eps=None):
        """One frame step of rank `band_first` of `band_stride`: hit16 records + film (async).
        full_frame=True: d_film_ptr is the whole [ny][nx][3] frame (possibly peer-mapped from
        rank 0) and pixels are stored at their final place."""
        sh = _shade(light, kd, shadow_eps)
        b = vrt_bands(int(band_h), int(band_first), int(band_stride))
        fn = load().vrt_frame_bands_peer_dev if full_frame else load().vrt_frame_bands_dev
        _check(fn(self._h, C.byref(cam.c), C.byref(sh), C.byref(b), C.c_void_p(d_hits_ptr), C.c_void_p(d_film_ptr)))

    def sync(self):
        _check(load().vrt_tree_sync(self._h))

    def debug_set_hull(self, on: bool):
        """Test hook: content-hull pruning of the ray kernels off / on for this handle."""
        _check(load().vrt_debug_set_hull(self._h, 1 if on else 0))

    def debug_set_eye_rel(self, on: bool):
        """Test hook: eye-relative hull records and triangle terms of the camera launches on / off for this handle."""
        _check(load().vrt_debug_set_eye_rel(self._h, 1 if on else 0))

    def debug_eye_rel_launches(self):
        """Test hook: camera launches of this handle that read eye-relative records so far."""
        n = C.c_uint64()
        _check(load().vrt_debug_eye_rel_launches(self._h, C.byref(n)))
        return int(n.value)

    def mean_kernel_ms(self, last_n):
        return float(load().vrt_mean_kernel_ms(self._h, int(last_n)))

    def trace_bands16_dev(self, cam: Camera, d_out_ptr, band_h, band_first, band_stride):
        b = vrt_bands(int(band_h), int(band_first), int(band_stride))
        _check(load().vrt_trace_bands16_dev(self._h, C.byref(cam.c), C.byref(b), C.c_void_p(d_out_ptr)))

    def count_camera(self, cam: Camera, rect=None):
        """Work counters of the reference algorithm over a frame (SURVEY.md 8d)."""
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        c = np.zeros(8, np.uint64)
        _check(load().vrt_count_camera(self._h, C.byref(cam.c), x0, y0, x1, y1, _ptr(c)))
        return dict(rays=int(c[0]), n_int=int(c[1]), n_leaf=int(c[2]), n_tri=int(c[3]), hits=int(c[4]),
                    n_param=int(c[5]), n_tie=int(c[6]), n_unsafe=int(c[7]))

    # ---- materials / textures (SURVEY.md 8f row 3) -------------------------------
    def set_materials(self, tri_uv, tri_mtl, kd, mtl_tex, textures):
        """textures: list of uint8 arrays [h, w, channels] (as stbi_load returns them)."""
        _set_materials(load().vrt_set_materials, self._h, tri_uv, tri_mtl, kd, mtl_tex, textures)

    def albedo(self, tri, pos, kd_default=(0.8, 0.8, 0.8)):
        tri = np.ascontiguousarray(tri, np.uint32)
        pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 3)
        kd = np.ascontiguousarray(kd_default, np.float32)
        out = np.zeros((len(tri), 3), np.float32)
        _check(load().vrt_albedo(self._h, _ptr(tri), _ptr(pos), len(tri), _ptr(kd), _ptr(out)))
        return out

    # ---- GI rows (SURVEY.md 8f) ------------------------------------------------
    def gi_init(self):
        _check(load().vrt_gi_init(self._h))

    def gi_splat(self, light_cam: Camera, kd):
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_gi_splat_camera(self._h, C.byref(light_cam.c), _ptr(kd)))

    def gi_filter(self):
        _check(load().vrt_gi_filter(self._h))

    def gi_level(self, level):
        """(coverage[n], illum[n,6,3]) of tree level `level`, node (= Morton) order."""
        off = self.info()["level_offset"]
        n = int(off[level + 1] - off[level])
        cov = np.zeros(n, np.float32)
        il = np.zeros((n, 6, 3), np.float32)
        _check(load().vrt_gi_get_level(self._h, int(level), _ptr(cov), _ptr(il)))
        return cov, il

    def gi_cone_trace(self, pos, nrm, res):
        pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 3)
        nrm = np.ascontiguousarray(nrm, np.float32).reshape(-1, 3)
        out = np.zeros((len(pos), 3), np.float32)
        _check(load().vrt_gi_cone_trace(self._h, _ptr(pos), _ptr(nrm), len(pos), float(np.float32(res)), _ptr(out)))
        return out

    def gi_render(self, cam: Camera, kd, res, rect=None):
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        kd = np.ascontiguousarray(kd, np.float32)
        out = np.zeros((y1 - y0, x1 - x0, 3), np.float32)
        _check(load().vrt_gi_render_camera(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)), x0, y0, x1, y1,
                                           _ptr(out)))
        return out

    def gi_render_bands_async(self, cam: Camera, kd, res, host_frame_ptr, band_h, band_first, band_stride):
        """The GI film's bands `band_first`, `band_first + band_stride`, ... DMA-copied to their final rows of the
        full (pinned, possibly shared between the ranks) host frame in the handle's film format; asynchronous, see
        sync().  (band_h = ny, 0, 1: the whole film as one pipelined frame.)"""
        kd = np.ascontiguousarray(kd, np.float32)
        b = vrt_bands(int(band_h), int(band_first), int(band_stride))
        _check(load().vrt_gi_render_bands_async(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)), C.byref(b),
                                                C.c_void_p(int(host_frame_ptr))))

    def gi_render_dev(self, cam: Camera, kd, res, d_film_ptr, rect=None):
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_gi_render_camera_dev(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)), x0, y0, x1,
                                               y1, C.c_void_p(d_film_ptr)))

    def gi_render_aov(self, cam: Camera, kd, res, rect=None, planes=GI_AOV_PLANES, film=True):
        """The GI film (gi_render's, in the handle's film format; None with film=False) and what it is made of, from
        one launch: {name: array} for the requested planes -- 'albedo', 'direct', 'indirect', 'normal' as float32
        [h, w, 3] sample means, 'hits' as HIT16_DTYPE [h, w, spp] (include/vrt.h vrt_gi_aov)."""
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        h, w = y1 - y0, x1 - x0
        unknown = set(planes) - set(GI_AOV_PLANES)
        if unknown:
            raise ValueError(f"unknown GI planes {sorted(unknown)}")
        out = {n: (np.zeros((h, w, cam.spp), HIT16_DTYPE) if n == "hits" else np.zeros((h, w, 3), np.float32))
               for n in planes}
        f = self._film_array(h, w) if film else None
        aov = vrt_gi_aov(**{n: a.ctypes.data for n, a in out.items()})
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_gi_render_aov(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)), x0, y0, x1, y1,
                                        _ptr(f), C.byref(aov)))
        return f, out

    def gi_render_aov_dev(self, cam: Camera, kd, res, d_film_or_0, d_planes: dict, rect=None):
        """gi_render_aov into device memory, enqueued on the handle's stream: d_planes maps plane names to device
        pointers (float32 [h, w, 3], hits vrt_hit16 [h, w, spp]); d_film_or_0 = 0 writes no film."""
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        aov = _gi_aov(d_planes)
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_gi_render_aov_dev(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)), x0, y0, x1,
                                            y1, C.c_void_p(int(d_film_or_0) or None), C.byref(aov)))

    def gi_render_aov_bands_async(self, cam: Camera, kd, res, host_film_ptr_or_0, host_planes: dict, band_h,
                                  band_first, band_stride):
        """gi_render_aov in the banded, pipelined form of gi_render_bands_async: host_planes maps plane names to
        (pinned) FULL host frames (float32 [ny, nx, 3], hits vrt_hit16 [ny, nx, spp]), of which only this handle's
        band rows are written, like the film's (host_film_ptr_or_0 = 0: no film); asynchronous, see sync()."""
        aov = _gi_aov(host_planes)
        kd = np.ascontiguousarray(kd, np.float32)
        b = vrt_bands(int(band_h), int(band_first), int(band_stride))
        _check(load().vrt_gi_render_aov_bands_async(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)),
                                                    C.byref(b), C.c_void_p(int(host_film_ptr_or_0) or None),
                                                    C.byref(aov)))

    def render_async(self, cam: Camera, out, light=None, kd=0.8, rect=None, shadow_eps=None):
        """Pipelined frame loop: enqueue one frame whose film lands in the (pinned) host array
        `out`; call sync() before reading.  Alternate between two host arrays."""
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        sh = _shade(light, kd, shadow_eps)
        _check(load().vrt_render_camera_async(self._h, C.byref(cam.c), C.byref(sh), x0, y0, x1, y1, _ptr(out)))

    def render_dev(self, cam: Camera, d_film_ptr, light=None, kd=0.8, rect=None, shadow_eps=None):
        x0, y0, x1, y1 = rect if rect else (0, 0, cam.nx, cam.ny)
        sh = _shade(light, kd, shadow_eps)
        _check(load().vrt_render_camera_dev(self._h, C.byref(cam.c), C.byref(sh), x0, y0, x1, y1,
                                            C.c_void_p(d_film_ptr)))


def debug_general_order_calls() -> int:
    return int(load().vrt_debug_general_order_calls())


def debug_param_check():
    """(expansions cross-checked, mismatches) -- non-zero only with a -DVRT_PARAM_CHECK build."""
    c = np.zeros(2, np.uint64)
    _check(load().vrt_debug_param_check(_ptr(c)))
    return int(c[0]), int(c[1])


FILM_FORMATS = {"f32": 0, "rgbe": 1, "rgb8": 2}


def film_pixel_bytes(fmt) -> int:
    return int(_check_pos(load().vrt_film_pixel_bytes(FILM_FORMATS[fmt] if isinstance(fmt, str) else int(fmt))))


def hdr_file(film_rgbe) -> bytes:
    """The bytes stbi_write_hdr writes for a film, from its RGBE encoding [ny][nx][4] (host code)."""
    a = np.ascontiguousarray(film_rgbe, np.uint8)
    ny, nx = a.shape[0], a.shape[1]
    n = int(_check_pos(load().vrt_hdr_file(_ptr(a), nx, ny, None, 0)))
    out = np.zeros(n, np.uint8)
    _check_pos(load().vrt_hdr_file(_ptr(a), nx, ny, _ptr(out), n))
    return out.tobytes()


class MultiGpu:
    """vrt_mgpu_*: one process, N devices -- replicas of a built octree, every frame's 8-row bands dealt round-robin
    to the devices and DMA-copied to their final rows of one (pinned) host frame."""

    def __init__(self, tree: "Octree", devices):
        dv = np.ascontiguousarray(devices, np.int32)
        h = C.c_void_p()
        _check(load().vrt_mgpu_create(tree._h, len(dv), _ptr(dv), C.byref(h)))
        self._h = h
        i = tree.info()
        self.max_depth, self.num_tris = i["max_depth"], i["num_tris"]

    @property
    def num_devices(self):
        return int(load().vrt_mgpu_num_devices(self._h))

    def render_async(self, cam: Camera, host_frame_ptr, light=None, kd=0.8, shadow_eps=None):
        sh = _shade(light, kd, shadow_eps)
        _check(load().vrt_mgpu_render_async(self._h, C.byref(cam.c), C.byref(sh), C.c_void_p(int(host_frame_ptr))))

    def render(self, cam: Camera, host_frame_ptr, light=None, kd=0.8, shadow_eps=None):
        sh = _shade(light, kd, shadow_eps)
        _check(load().vrt_mgpu_render(self._h, C.byref(cam.c), C.byref(sh), C.c_void_p(int(host_frame_ptr))))

    def sync(self):
        _check(load().vrt_mgpu_sync(self._h))

    def set_film_format(self, fmt):
        _check(load().vrt_mgpu_set_film_format(self._h, FILM_FORMATS[fmt] if isinstance(fmt, str) else int(fmt)))

    # ---- GI film on the replicas (the replicas hold geometry only until these calls) ----------------------------
    def set_materials(self, tri_uv, tri_mtl, kd, mtl_tex, textures):
        """Octree.set_materials on every replica."""
        _set_materials(load().vrt_mgpu_set_materials, self._h, tri_uv, tri_mtl, kd, mtl_tex, textures)

    def gi_init(self):
        _check(load().vrt_mgpu_gi_init(self._h))

    def gi_splat(self, light_cam: Camera, kd):
        """The light pass on every replica (deterministic: every replica holds the same bits)."""
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_mgpu_gi_splat_camera(self._h, C.byref(light_cam.c), _ptr(kd)))

    def gi_filter(self):
        _check(load().vrt_mgpu_gi_filter(self._h))

    def gi_render_async(self, cam: Camera, kd, res, host_frame_ptr):
        """Enqueue one GI film: 8-row bands round-robin over the replicas, each DMA-copied to its final rows of the
        (pinned) host frame in the replicas' film format; call sync() before reading."""
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_mgpu_gi_render_async(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)),
                                               C.c_void_p(int(host_frame_ptr))))

    def gi_render(self, cam: Camera, kd, res, host_frame_ptr):
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_mgpu_gi_render(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)),
                                         C.c_void_p(int(host_frame_ptr))))

    def gi_render_aov_async(self, cam: Camera, kd, res, host_film_ptr_or_0, host_planes: dict):
        """Enqueue one GI film (host_film_ptr_or_0 = 0: none) and its planes (Octree.gi_render_aov_bands_async's
        host_planes) over the replicas, 8-row bands round-robin; call sync() before reading."""
        aov = _gi_aov(host_planes)
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_mgpu_gi_render_aov_async(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)),
                                                   C.c_void_p(int(host_film_ptr_or_0) or None), C.byref(aov)))

    def gi_render_aov(self, cam: Camera, kd, res, host_film_ptr_or_0, host_planes: dict):
        aov = _gi_aov(host_planes)
        kd = np.ascontiguousarray(kd, np.float32)
        _check(load().vrt_mgpu_gi_render_aov(self._h, C.byref(cam.c), _ptr(kd), float(np.float32(res)),
                                             C.c_void_p(int(host_film_ptr_or_0) or None), C.byref(aov)))

    def update(self, tri_xyz, tri_nrm=None, max_depth=None):
        """Octree.update on the replicas: the first one rebuilds, the others copy its blob (max_depth None: the
        replicas' current depth)."""
        tri, nrm = _update_arrays(tri_xyz, tri_nrm)
        if tri.shape[0] != self.num_tris:
            raise ValueError(f"update needs {self.num_tris} triangles (the replicas' count), got {tri.shape[0]}")
        depth = self.max_depth if max_depth is None else int(max_depth)
        _check(load().vrt_mgpu_update_triangles(self._h, _ptr(tri), _ptr(nrm), tri.shape[0], depth))
        self.max_depth = depth

    def update_xform(self, xforms, max_depth=None):
        """Octree.update_xform on the replicas (rest pose: the source tree's triangles, or the last update())."""
        arr = _xform_table(xforms)
        depth = self.max_depth if max_depth is None else int(max_depth)
        _check(load().vrt_mgpu_update_xform(self._h, C.cast(arr, C.c_void_p), len(arr), depth))
        self.max_depth = depth

    def mean_kernel_ms(self, index, last_n):
        """Mean device time of the last `last_n` kernels of replica `index` (waits for them)."""
        return float(load().vrt_mgpu_mean_kernel_ms(self._h, int(index), int(last_n)))

    def close(self):
        if self._h:
            load().vrt_mgpu_free(self._h)
            self._h = None


def _update_arrays(tri_xyz, tri_nrm):
    """float32 [T, 9] triangles (and normals of the same shape) for the update calls; shape errors raise here."""
    tri = np.ascontiguousarray(tri_xyz, np.float32)
    if tri.size % 9 or tri.size == 0:
        raise ValueError(f"tri_xyz must hold [T, 9] floats, got shape {tri.shape}")
    tri = tri.reshape(-1, 9)
    if tri_nrm is None:
        return tri, None
    nrm = np.ascontiguousarray(tri_nrm, np.float32)
    if nrm.size != tri.size:
        raise ValueError(f"tri_nrm must have the shape of tri_xyz {tri.shape}, got {nrm.shape}")
    return tri, nrm.reshape(-1, 9)


def xform_normal_matrix(m):
    """The default normal matrix of a 3x4 transform: the float64 inverse transpose of M[:, :3], as float32."""
    return np.linalg.inv(np.asarray(m, np.float64).reshape(3, 4)[:, :3]).T.astype(np.float32)


def _xform_table(xforms):
    """vrt_xform array from (first, count, M 3x4[, N 3x3]) tuples; malformed tuples raise ValueError."""
    xforms = list(xforms)
    if not xforms:
        raise ValueError("update_xform needs at least one transform")
    arr = (vrt_xform * len(xforms))()
    for k, x in enumerate(xforms):
        if not isinstance(x, (tuple, list)) or len(x) not in (3, 4):
            raise ValueError(f"transform {k}: expected (first, count, M[, N]), got {x!r}")
        first, count = int(x[0]), int(x[1])
        if first < 0 or count < 0 or first >= 2 ** 32 or count >= 2 ** 32:
            raise ValueError(f"transform {k}: bad range ({first}, {count})")
        m = np.asarray(x[2], np.float32)
        if m.shape != (3, 4):
            raise ValueError(f"transform {k}: M must be 3x4, got shape {m.shape}")
        n = np.asarray(x[3], np.float32) if len(x) == 4 and x[3] is not None else xform_normal_matrix(x[2])
        if n.shape != (3, 3):
            raise ValueError(f"transform {k}: N must be 3x3, got shape {n.shape}")
        arr[k] = vrt_xform(first, count, (C.c_float * 12)(*m.reshape(-1)), (C.c_float * 9)(*n.reshape(-1)))
    return arr


def _gi_aov(planes: dict) -> vrt_gi_aov:
    """A vrt_gi_aov of the pointers in `planes` (names of GI_AOV_PLANES; 0 / None: not written)."""
    unknown = set(planes) - set(GI_AOV_PLANES)
    if unknown:
        raise ValueError(f"unknown GI planes {sorted(unknown)}")
    return vrt_gi_aov(**{n: int(p) for n, p in planes.items() if p})


def _set_materials(fn, h, tri_uv, tri_mtl, kd, mtl_tex, textures):
    """vrt_set_materials / vrt_mgpu_set_materials on handle `h` (textures: uint8 arrays [h, w, channels])."""
    tri_uv = np.ascontiguousarray(tri_uv, np.float32).reshape(-1, 6)
    tri_mtl = np.ascontiguousarray(tri_mtl, np.uint32)
    kd = np.ascontiguousarray(kd, np.float32).reshape(-1, 3)
    mtl_tex = np.ascontiguousarray(mtl_tex, np.int32)
    texs = [np.ascontiguousarray(t, np.uint8) for t in textures]
    arr = (vrt_texture * max(len(texs), 1))()
    for i, t in enumerate(texs):
        arr[i] = vrt_texture(t.shape[1], t.shape[0], t.shape[2], t.ctypes.data)
    _check(fn(h, _ptr(tri_uv), _ptr(tri_mtl), len(kd), _ptr(kd), _ptr(mtl_tex), len(texs), C.cast(arr, C.c_void_p)))


def debug_hull_stats():
    """[level][expansions, interior children visited, hull tests, prunes] (-DVRT_HULL_STATS builds)."""
    c = np.zeros(80, np.uint64)
    _check(load().vrt_debug_hull_stats(_ptr(c)))
    return c.reshape(20, 4)


def debug_pair_total(block_counts) -> int:
    """64-bit device sum of 32-bit block counts (the build's pair-total overflow guard)."""
    c = np.ascontiguousarray(block_counts, np.uint32)
    out = np.zeros(1, np.uint64)
    _check(load().vrt_debug_pair_total(_ptr(c), len(c), _ptr(out)))
    return int(out[0])


def dev_alloc(nbytes: int) -> int:
    p = C.c_void_p()
    _check(load().vrt_dev_alloc(int(nbytes), C.byref(p)))
    return p.value


def dev_free(ptr: int):
    _check(load().vrt_dev_free(C.c_void_p(ptr)))


def host_register(ptr: int, nbytes: int):
    _check(load().vrt_host_register(C.c_void_p(ptr), int(nbytes)))


def host_unregister(ptr: int):
    _check(load().vrt_host_unregister(C.c_void_p(ptr)))


def ipc_export(ptr: int) -> bytes:
    h = (C.c_uint8 * 64)()
    _check(load().vrt_ipc_export(C.c_void_p(ptr), h))
    return bytes(h)


def ipc_open(handle: bytes) -> int:
    h = (C.c_uint8 * 64).from_buffer_copy(handle)
    p = C.c_void_p()
    _check(load().vrt_ipc_open(h, C.byref(p)))
    return p.value


def ipc_close(ptr: int):
    _check(load().vrt_ipc_close(C.c_void_p(ptr)))


def band_rows(cam: Camera, band_h, band_first, band_stride) -> int:
    b = vrt_bands(int(band_h), int(band_first), int(band_stride))
    r = load().vrt_band_rows(C.byref(cam.c), C.byref(b))
    if r < 0:
        _check(r)
    return int(r)


# ---- predicates (device KATs) ------------------------------------------------
def tribox(centers, halves, tris):
    """triBoxOverlap(boxcenter, boxhalfsize, triverts) (tribox2.h:15), batched."""
    c, h, t = _f32(centers, (-1, 3)), _f32(halves, (-1, 3)), _f32(tris, (-1, 9))
    out = np.zeros(len(c), np.uint8)
    _check(load().vrt_tribox_batch(_ptr(c), _ptr(h), _ptr(t), len(c), _ptr(out)))
    return out


def tri_overlap_aabb(aabbs, tris):
    b, t = _f32(aabbs, (-1, 6)), _f32(tris, (-1, 9))
    out = np.zeros(len(b), np.uint8)
    _check(load().vrt_tri_overlap_aabb_batch(_ptr(b), _ptr(t), len(b), _ptr(out)))
    return out


def raytri(in15):
    """intersect_triangle3(orig, dir, v0, v1, v2, &t, &u, &v) (raytri.h:5-7), batched."""
    a = np.ascontiguousarray(in15, np.float64).reshape(-1, 15)
    res = np.zeros(len(a), np.uint8)
    tuv = np.zeros((len(a), 3), np.float64)
    _check(load().vrt_raytri_batch(_ptr(a), len(a), _ptr(res), _ptr(tuv)))
    return res, tuv


def aabb_isect(aabbs, rays):
    b = _f32(aabbs, (-1, 6))
    r = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
    out = np.zeros(len(b), np.uint8)
    _check(load().vrt_aabb_isect_batch(_ptr(b), _ptr(r), len(b), _ptr(out)))
    return out
