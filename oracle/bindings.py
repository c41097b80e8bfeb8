"""ctypes bindings for the two CPU checkers -- TEST INFRASTRUCTURE.

* :class:`Port`  -> oracle/libvrt_oracle.so  (vrt_oracle.c, the C restatement)
* :class:`Ref`   -> oracle/_ref/libvrt_ref.so (the UNMODIFIED reference sources +
  ref_harness.cc, built by oracle/build_ref.sh)

Only tests/, ``__graft_entry__.smoke()`` and bench.py's ``cpu_baseline`` /
``--impl reference`` legs may import this module.  The product package
(voxelraytrace20190722_b200) never does.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "libvrt_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libvrt_ref.so")

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")


def _opt(arr):
    return None if arr is None else arr.ctypes.data_as(C.c_void_p)


def build_port(force: bool = False) -> str:
    src = os.path.join(HERE, "vrt_oracle.c")
    if force or not os.path.exists(PORT_SO) or os.path.getmtime(PORT_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", HERE, "-B" if force else "-s", "libvrt_oracle.so"])
    return PORT_SO


def build_ref(force: bool = False) -> str | None:
    """Build oracle/_ref when the reference sources are present; else keep prebuilt."""
    have_src = os.path.exists(os.path.join(
        os.environ.get("VRT_REFERENCE_DIR", "/root/reference"), "VoxelRayTrace20190722", "voxel_octree.cc"))
    harness = os.path.join(HERE, "ref_harness.cc")
    # (the same recipe also links the reference's main.cc against libvrt.so: oracle/_ref/main_dropin*)
    dropin = os.path.join(HERE, "_ref", "main_dropin")
    deps = [harness, os.path.join(HERE, "build_ref.sh"),
            os.path.join(HERE, "..", "voxelraytrace20190722_b200", "cpp", "vrt_dropin.cc"),
            os.path.join(HERE, "..", "include", "vrt.h")]
    outs = [REF_SO] + ([dropin] if os.path.exists(os.path.join(HERE, "..", "voxelraytrace20190722_b200", "libvrt.so")) else [])
    stale = any(not os.path.exists(o) for o in outs) or \
        min(os.path.getmtime(o) for o in outs) < max(os.path.getmtime(d) for d in deps if os.path.exists(d))
    if have_src and (force or stale):
        subprocess.check_call(["bash", os.path.join(HERE, "build_ref.sh")])
    return REF_SO if os.path.exists(REF_SO) else None


def ref_available() -> bool:
    return os.path.exists(REF_SO)


def _as_tri(tri):
    tri = np.ascontiguousarray(tri, np.float32).reshape(-1, 9)
    return tri


class _HitArrays:
    def __init__(self, R, with_t=True):
        self.hit = np.zeros(R, np.uint8)
        self.cell = np.zeros((R, 3), np.uint32)
        self.tri = np.zeros(R, np.uint32)
        self.t = np.zeros(R, np.float32) if with_t else None
        self.pos = np.zeros((R, 3), np.float32)
        self.nrm = np.zeros((R, 3), np.float32)


# ----------------------------------------------------------------------------
class Port:
    """The C restatement (oracle/vrt_oracle.c)."""

    def __init__(self):
        self.lib = C.CDLL(build_port())
        L = self.lib
        L.orc_build.restype = C.c_void_p
        L.orc_build.argtypes = [_f32p, C.c_void_p, C.c_uint32, C.c_int]
        L.orc_free.argtypes = [C.c_void_p]
        L.orc_root_aabb.argtypes = [C.c_void_p, _f32p]
        L.orc_stats.argtypes = [C.c_void_p, _u64p]
        L.orc_dump_leaves.argtypes = [C.c_void_p, _u32p, _u32p, _u32p, C.c_void_p]
        L.orc_trace_rays.argtypes = [C.c_void_p, _f32p, C.c_uint64, _u8p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_camera_matrix.argtypes = [_f32p, _f32p]
        L.orc_camera_z.restype = C.c_float
        L.orc_camera_z.argtypes = [C.c_float, C.c_float]
        L.orc_gen_rays.argtypes = [_f32p, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, _f32p]
        L.orc_tribox_batch.argtypes = [_f32p, _f32p, _f32p, C.c_uint64, _u8p]
        L.orc_tri_overlap_aabb_batch.argtypes = [_f32p, _f32p, C.c_uint64, _u8p]
        L.orc_raytri_batch.argtypes = [_f64p, C.c_uint64, _u8p, _f64p]
        L.orc_aabb_isect_batch.argtypes = [_f32p, _f32p, C.c_uint64, _u8p]
        # GI rows (SURVEY.md 8f)
        L.orc_gi_reset.argtypes = [C.c_void_p]
        L.orc_gi_splat.argtypes = [C.c_void_p, _f32p, C.c_float, C.c_int, C.c_int, C.c_int, _f32p]
        L.orc_gi_filter.argtypes = [C.c_void_p]
        L.orc_gi_dump_level.restype = C.c_uint64
        L.orc_gi_dump_level.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.orc_gi_cone_trace.argtypes = [C.c_void_p, _f32p, _f32p, C.c_uint64, C.c_float, _f32p]
        L.orc_gi_render.argtypes = [C.c_void_p, _f32p, C.c_float, C.c_int, C.c_int, C.c_int, C.c_float, _f32p, _f32p]
        L.orc_gi_set_exact_log2.argtypes = [C.c_int]
        # materials / textures (SURVEY.md 8f row 3)
        L.orc_set_materials.argtypes = [C.c_void_p, _f32p, _u32p, C.c_uint32, _f32p, C.c_void_p, C.c_uint32, C.c_void_p,
                                        C.c_void_p]
        L.orc_film_rgb8.argtypes = [_f32p, C.c_uint64, _u8p]
        L.orc_film_rgbe.argtypes = [_f32p, C.c_uint64, _u8p]
        L.orc_albedo.argtypes = [C.c_void_p, _u32p, _f32p, C.c_uint64, _f32p, _f32p]

    @contextlib.contextmanager
    def exact_log2(self):
        """Within the block the cone trace (gi_cone_trace, gi_render) takes split_level = int(log2f(x)) with the
        correctly rounded log2f, (float)log2((double)x), instead of libm's -- the definition the device evaluates,
        so GPU results compare bit for bit.  Outside it the oracle keeps the reference's libm expression."""
        self.lib.orc_gi_set_exact_log2(1)
        try:
            yield self
        finally:
            self.lib.orc_gi_set_exact_log2(0)

    # -- film export ----------------------------------------------------------
    def film_rgb8(self, film):
        """Film::to_byte_array (camera.cc:27-48) of a float film [..., 3] -> uint8 [..., 3]."""
        f = np.ascontiguousarray(film, np.float32)
        out = np.zeros(f.shape, np.uint8)
        self.lib.orc_film_rgb8(f.reshape(-1), f.size // 3, out.reshape(-1))
        return out

    def film_rgbe(self, film):
        """stbiw__linear_to_rgbe (stb_image_write.h:601-616) per pixel: float [..., 3] -> uint8 [..., 4]."""
        f = np.ascontiguousarray(film, np.float32)
        out = np.zeros(f.shape[:-1] + (4,), np.uint8)
        self.lib.orc_film_rgbe(f.reshape(-1), f.size // 3, out.reshape(-1))
        return out

    # -- tree ---------------------------------------------------------------
    def build(self, tri, nrm, max_depth):
        tri = _as_tri(tri)
        nrm_c = None if nrm is None else np.ascontiguousarray(nrm, np.float32).reshape(-1, 9)
        h = self.lib.orc_build(tri, _opt(nrm_c), tri.shape[0], int(max_depth))
        return PortTree(self, h, int(max_depth))

    # -- camera -------------------------------------------------------------
    def camera_matrix(self, cam10):
        out = np.zeros(16, np.float32)
        self.lib.orc_camera_matrix(np.ascontiguousarray(cam10, np.float32), out)
        return out

    def camera_z(self, fov, film_h):
        return np.float32(self.lib.orc_camera_z(float(np.float32(fov)), float(np.float32(film_h))))

    def gen_rays(self, cam10, film_h, nx, ny, spp, rect=None):
        x0, y0, x1, y1 = rect if rect else (0, 0, nx, ny)
        Cm = self.camera_matrix(cam10)
        z = self.camera_z(cam10[0], film_h)
        out = np.zeros(((y1 - y0) * (x1 - x0) * spp, 8), np.float32)
        self.lib.orc_gen_rays(Cm, float(z), nx, ny, spp, x0, y0, x1, y1, out)
        return out

    # -- predicates -----------------------------------------------------------
    def tribox(self, centers, halves, tris):
        n = len(centers)
        out = np.zeros(n, np.uint8)
        self.lib.orc_tribox_batch(np.ascontiguousarray(centers, np.float32),
                                  np.ascontiguousarray(halves, np.float32), _as_tri(tris), n, out)
        return out

    def tri_overlap_aabb(self, aabbs, tris):
        n = len(aabbs)
        out = np.zeros(n, np.uint8)
        self.lib.orc_tri_overlap_aabb_batch(np.ascontiguousarray(aabbs, np.float32), _as_tri(tris), n, out)
        return out

    def raytri(self, in15):
        in15 = np.ascontiguousarray(in15, np.float64)
        n = len(in15)
        res = np.zeros(n, np.uint8)
        tuv = np.zeros((n, 3), np.float64)
        self.lib.orc_raytri_batch(in15, n, res, tuv)
        return res, tuv

    def aabb_isect(self, aabbs, rays):
        n = len(aabbs)
        out = np.zeros(n, np.uint8)
        self.lib.orc_aabb_isect_batch(np.ascontiguousarray(aabbs, np.float32),
                                      np.ascontiguousarray(rays, np.float32), n, out)
        return out


class PortTree:
    def __init__(self, port, handle, max_depth):
        self.port, self.h, self.max_depth = port, handle, max_depth

    def __del__(self):
        if getattr(self, "h", None):
            self.port.lib.orc_free(self.h)
            self.h = None

    def stats(self):
        s = np.zeros(6, np.uint64)
        self.port.lib.orc_stats(self.h, s)
        return dict(nodes=int(s[0]), interior=int(s[1]), leaves=int(s[2]), refs=int(s[3]),
                    max_leaf_refs=int(s[4]), nonempty_nodes=int(s[5]))

    def root_aabb(self):
        out = np.zeros(6, np.float32)
        self.port.lib.orc_root_aabb(self.h, out)
        return out

    def leaves(self, boxes=False):
        st = self.stats()
        cells = np.zeros((st["leaves"], 3), np.uint32)
        counts = np.zeros(st["leaves"], np.uint32)
        refs = np.zeros(st["refs"], np.uint32)
        bx = np.zeros((st["leaves"], 6), np.float32) if boxes else None
        self.port.lib.orc_dump_leaves(self.h, cells, counts, refs, _opt(bx))
        return (cells, counts, refs, bx) if boxes else (cells, counts, refs)

    def trace(self, rays, counters=False):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
        R = len(rays)
        o = _HitArrays(R)
        cn = np.zeros(6, np.uint64) if counters else None
        self.port.lib.orc_trace_rays(self.h, rays, R, o.hit, _opt(o.cell), _opt(o.tri), _opt(o.t),
                                     _opt(o.pos), _opt(o.nrm), _opt(cn))
        if counters:
            o.counters = dict(n_slab=int(cn[0]), n_int=int(cn[1]), n_leaf_all=int(cn[2]),
                              n_leaf=int(cn[3]), n_tri=int(cn[4]), max_stack=int(cn[5]))
        return o

    def _gi(self, name):
        return getattr(self.port.lib, "orc_gi_" + name)

    # -- GI rows (SURVEY.md 8f): same method names on PortTree and RefScene -----------------
    def gi_reset(self):
        self._gi("reset")(self.h)

    def gi_filter(self):
        self._gi("filter")(self.h)

    def gi_level(self, level):
        """(cells[n,3], coverage[n], illum[n,6,3]) of the nodes of `level` with coverage > 0, Morton order."""
        f = self._gi("dump_level")
        n = int(f(self.h, int(level), None, None, None, 0))
        cells = np.zeros((n, 3), np.uint32)
        cov = np.zeros(n, np.float32)
        il = np.zeros((n, 6, 3), np.float32)
        if n:
            f(self.h, int(level), cells.ctypes.data, cov.ctypes.data, il.ctypes.data, n)
        return cells, cov, il

    def gi_cone_trace(self, pos, nrm, res):
        pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 3)
        nrm = np.ascontiguousarray(nrm, np.float32).reshape(-1, 3)
        out = np.zeros((len(pos), 3), np.float32)
        self._gi("cone_trace")(self.h, pos, nrm, len(pos), float(np.float32(res)), out)
        return out

    def set_materials(self, tri_uv, tri_mtl, kd, mtl_tex, textures):
        """textures: list of uint8 arrays [h, w, channels] as the reference's stbi_load returns them."""
        tri_uv = np.ascontiguousarray(tri_uv, np.float32).reshape(-1, 6)
        tri_mtl = np.ascontiguousarray(tri_mtl, np.uint32)
        kd = np.ascontiguousarray(kd, np.float32).reshape(-1, 3)
        mtl_tex = np.ascontiguousarray(mtl_tex, np.int32)
        texs = [np.ascontiguousarray(t, np.uint8) for t in textures]
        whc = np.array([[t.shape[1], t.shape[0], t.shape[2]] for t in texs], np.int32).reshape(-1, 3)
        ptrs = (C.c_void_p * max(len(texs), 1))(*[t.ctypes.data for t in texs])
        self.port.lib.orc_set_materials(self.h, tri_uv, tri_mtl, len(kd), kd, mtl_tex.ctypes.data, len(texs),
                                        whc.ctypes.data, C.cast(ptrs, C.c_void_p))

    def albedo(self, tri, pos, kd_default=(0.8, 0.8, 0.8)):
        tri = np.ascontiguousarray(tri, np.uint32)
        pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 3)
        out = np.zeros((len(tri), 3), np.float32)
        self.port.lib.orc_albedo(self.h, tri, pos, len(tri), np.ascontiguousarray(kd_default, np.float32), out)
        return out

    def gi_splat(self, cam10, film_h, nx, ny, spp, kd):
        self.kd = np.ascontiguousarray(kd, np.float32)
        self.port.lib.orc_gi_splat(self.h, np.ascontiguousarray(cam10, np.float32), float(film_h), nx, ny, spp,
                                   self.kd)

    def gi_render(self, cam10, film_h, nx, ny, spp, res, kd=None, nthreads=1):
        kd = self.kd if kd is None else np.ascontiguousarray(kd, np.float32)
        film = np.zeros((ny, nx, 3), np.float32)
        self.port.lib.orc_gi_render(self.h, np.ascontiguousarray(cam10, np.float32), float(film_h), nx, ny, spp,
                                    float(np.float32(res)), kd, film)
        return film

    def gi_render_counted(self, cam10, film_h, nx, ny, spp, res, kd=None):
        """gi_render plus the cone trace's work counters: (film, {samples, descent_steps, located})."""
        lib = self.port.lib
        lib.orc_gi_counters_reset()
        film = self.gi_render(cam10, film_h, nx, ny, spp, res, kd)
        c = np.zeros(3, np.uint64)
        lib.orc_gi_counters(c.ctypes.data_as(C.c_void_p))
        return film, {"samples": int(c[0]), "descent_steps": int(c[1]), "located": int(c[2])}


# ----------------------------------------------------------------------------
class Ref:
    """The unmodified reference, through oracle/ref_harness.cc."""

    def __init__(self):
        so = build_ref()
        if so is None:
            raise FileNotFoundError("oracle/_ref/libvrt_ref.so not built and reference sources absent")
        self.lib = C.CDLL(so)
        L = self.lib
        L.ref_scene_create.restype = C.c_void_p
        L.ref_scene_create.argtypes = [_f32p, C.c_void_p, C.c_uint32]
        L.ref_scene_free.argtypes = [C.c_void_p]
        L.ref_scene_build.restype = C.c_double
        L.ref_scene_build.argtypes = [C.c_void_p, C.c_int]
        L.ref_scene_stats.argtypes = [C.c_void_p, _u64p]
        L.ref_scene_root_aabb.argtypes = [C.c_void_p, _f32p]
        L.ref_scene_dump_leaves.argtypes = [C.c_void_p, _u32p, C.c_void_p, _u32p, _u32p, C.c_void_p]
        L.ref_trace_rays.argtypes = [C.c_void_p, _f32p, C.c_uint64, C.c_int, _u8p, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p]
        L.ref_gen_rays.argtypes = [_f32p, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_int, _f32p]
        L.ref_render_mt.restype = C.c_double
        L.ref_render_mt.argtypes = [C.c_void_p, _f32p, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p]
        L.ref_hardware_concurrency.restype = C.c_int
        L.ref_tribox_batch.argtypes = [_f32p, _f32p, _f32p, C.c_uint64, _u8p]
        L.ref_tri_overlap_aabb_batch.argtypes = [_f32p, _f32p, C.c_uint64, _u8p]
        L.ref_raytri_batch.argtypes = [_f64p, C.c_uint64, _u8p, _f64p]
        L.ref_aabb_isect_batch.argtypes = [_f32p, _f32p, C.c_uint64, _u8p]
        L.ref_camera_matrix.argtypes = [_f32p, _f32p]
        # GI rows (SURVEY.md 8f)
        L.ref_scene_set_diffuse.argtypes = [C.c_void_p, _f32p]
        L.ref_gi_reset.argtypes = [C.c_void_p]
        L.ref_gi_splat.argtypes = [C.c_void_p, _f32p, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int]
        L.ref_gi_filter.argtypes = [C.c_void_p]
        L.ref_gi_dump_level.restype = C.c_uint64
        L.ref_gi_dump_level.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]
        L.ref_gi_cone_trace.argtypes = [C.c_void_p, _f32p, _f32p, C.c_uint64, C.c_float, _f32p]
        L.ref_scene_create_mat.restype = C.c_void_p
        L.ref_scene_create_mat.argtypes = [_f32p, _f32p, _f32p, _u32p, C.c_uint32, C.c_uint32, _f32p, C.c_void_p]
        L.ref_albedo.argtypes = [C.c_void_p, _u32p, _f32p, C.c_uint64, _f32p]
        L.ref_load_image.restype = C.c_uint64
        L.ref_load_image.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p,
                                     C.c_uint64]
        L.ref_film_to_bytes.argtypes = [_f32p, C.c_int, C.c_int, _u8p]
        L.ref_write_hdr.restype = C.c_uint64
        L.ref_write_hdr.argtypes = [_f32p, C.c_int, C.c_int, C.c_void_p, C.c_uint64]
        L.ref_gi_render.restype = C.c_double
        L.ref_gi_render.argtypes = [C.c_void_p, _f32p, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, C.c_float,
                                    _f32p, C.c_int]

    def hardware_concurrency(self):
        return int(self.lib.ref_hardware_concurrency())

    def scene(self, tri, nrm=None):
        tri = _as_tri(tri)
        nrm_c = None if nrm is None else np.ascontiguousarray(nrm, np.float32).reshape(-1, 9)
        h = self.lib.ref_scene_create(tri, _opt(nrm_c), tri.shape[0])
        return RefScene(self, h)

    def build(self, tri, nrm, max_depth):
        s = self.scene(tri, nrm)
        s.build(max_depth)
        return s

    def scene_mat(self, tri, nrm, tri_uv, tri_mtl, kd, texpaths):
        """Triangles with texture coordinates and per-triangle materials; texpaths[m] = image file or ''."""
        tri = _as_tri(tri)
        nrm_c = np.ascontiguousarray(nrm, np.float32).reshape(-1, 9)
        uv = np.ascontiguousarray(tri_uv, np.float32).reshape(-1, 6)
        mt = np.ascontiguousarray(tri_mtl, np.uint32)
        kd = np.ascontiguousarray(kd, np.float32).reshape(-1, 3)
        arr = (C.c_char_p * len(kd))(*[os.fsencode(p) for p in texpaths])
        h = self.lib.ref_scene_create_mat(tri, nrm_c, uv, mt, tri.shape[0], len(kd), kd, C.cast(arr, C.c_void_p))
        sc = RefScene(self, h)
        sc._keep = arr
        return sc

    def load_image(self, path):
        """The bytes the reference's load_image() sees (stbi_load): uint8 [h, w, channels]."""
        w, h, c = C.c_int(0), C.c_int(0), C.c_int(0)
        n = self.lib.ref_load_image(os.fsencode(path), C.byref(w), C.byref(h), C.byref(c), None, 0)
        if n == 0:
            raise FileNotFoundError(path)
        out = np.zeros(int(n), np.uint8)
        self.lib.ref_load_image(os.fsencode(path), C.byref(w), C.byref(h), C.byref(c), out.ctypes.data, int(n))
        return out.reshape(h.value, w.value, c.value)

    def film_to_bytes(self, film):
        """Film::to_byte_array() of the reference's own Film filled with `film` [n][n][3] (square: Film::set
        indexes y*ny + x, camera.cc:12-15, which only addresses a square film correctly)."""
        f = np.ascontiguousarray(film, np.float32)
        ny, nx = f.shape[0], f.shape[1]
        assert nx == ny
        out = np.zeros((ny, nx, 3), np.uint8)
        self.lib.ref_film_to_bytes(f.reshape(-1), nx, ny, out.reshape(-1))
        return out

    def write_hdr(self, film) -> bytes:
        """The file stbi_write_hdr writes for Film::to_float_array() (main.cc:125-126)."""
        f = np.ascontiguousarray(film, np.float32)
        ny, nx = f.shape[0], f.shape[1]
        assert nx == ny
        n = int(self.lib.ref_write_hdr(f.reshape(-1), nx, ny, None, 0))
        out = np.zeros(n, np.uint8)
        self.lib.ref_write_hdr(f.reshape(-1), nx, ny, out.ctypes.data, n)
        return out.tobytes()

    def camera_matrix(self, cam10):
        out = np.zeros(16, np.float32)
        self.lib.ref_camera_matrix(np.ascontiguousarray(cam10, np.float32), out)
        return out

    def gen_rays(self, cam10, film_h, nx, ny, spp, rect=None, film_w=1.0):
        x0, y0, x1, y1 = rect if rect else (0, 0, nx, ny)
        out = np.zeros(((y1 - y0) * (x1 - x0) * spp, 8), np.float32)
        self.lib.ref_gen_rays(np.ascontiguousarray(cam10, np.float32), film_w, film_h, nx, ny, spp,
                              x0, y0, x1, y1, out)
        return out

    def tribox(self, centers, halves, tris):
        n = len(centers)
        out = np.zeros(n, np.uint8)
        self.lib.ref_tribox_batch(np.ascontiguousarray(centers, np.float32),
                                  np.ascontiguousarray(halves, np.float32), _as_tri(tris), n, out)
        return out

    def tri_overlap_aabb(self, aabbs, tris):
        n = len(aabbs)
        out = np.zeros(n, np.uint8)
        self.lib.ref_tri_overlap_aabb_batch(np.ascontiguousarray(aabbs, np.float32), _as_tri(tris), n, out)
        return out

    def raytri(self, in15):
        in15 = np.ascontiguousarray(in15, np.float64)
        n = len(in15)
        res = np.zeros(n, np.uint8)
        tuv = np.zeros((n, 3), np.float64)
        self.lib.ref_raytri_batch(in15, n, res, tuv)
        return res, tuv

    def aabb_isect(self, aabbs, rays):
        n = len(aabbs)
        out = np.zeros(n, np.uint8)
        self.lib.ref_aabb_isect_batch(np.ascontiguousarray(aabbs, np.float32),
                                      np.ascontiguousarray(rays, np.float32), n, out)
        return out


class RefScene:
    def __init__(self, ref, handle):
        self.ref, self.h = ref, handle
        self.build_seconds = None
        self.max_depth = None

    def __del__(self):
        if getattr(self, "h", None):
            self.ref.lib.ref_scene_free(self.h)
            self.h = None

    def build(self, max_depth):
        self.build_seconds = float(self.ref.lib.ref_scene_build(self.h, int(max_depth)))
        self.max_depth = int(max_depth)
        return self.build_seconds

    def stats(self):
        s = np.zeros(6, np.uint64)
        self.ref.lib.ref_scene_stats(self.h, s)
        return dict(nodes=int(s[0]), interior=int(s[1]), leaves=int(s[2]), refs=int(s[3]),
                    max_leaf_refs=int(s[4]), nonempty_nodes=int(s[1] + s[2]))

    def root_aabb(self):
        out = np.zeros(6, np.float32)
        self.ref.lib.ref_scene_root_aabb(self.h, out)
        return out

    def leaves(self, boxes=False):
        st = self.stats()
        cells = np.zeros((st["leaves"], 3), np.uint32)
        levels = np.zeros(st["leaves"], np.uint32)
        counts = np.zeros(st["leaves"], np.uint32)
        refs = np.zeros(st["refs"], np.uint32)
        bx = np.zeros((st["leaves"], 6), np.float32) if boxes else None
        self.ref.lib.ref_scene_dump_leaves(self.h, cells, _opt(levels), counts, refs, _opt(bx))
        assert (levels == self.max_depth - 1).all() or st["leaves"] == 0
        return (cells, counts, refs, bx) if boxes else (cells, counts, refs)

    def trace(self, rays, nthreads=1):
        rays = np.ascontiguousarray(rays, np.float32).reshape(-1, 8)
        R = len(rays)
        o = _HitArrays(R, with_t=False)
        self.ref.lib.ref_trace_rays(self.h, rays, R, int(nthreads), o.hit, _opt(o.cell), _opt(o.tri),
                                    _opt(o.pos), _opt(o.nrm))
        return o

    def render_mt(self, cam10, film_h, nx, ny, spp, outputs=True, film_w=1.0):
        """The reference's own thread-pool render loop; returns (seconds, rays, hits|None)."""
        R = nx * ny * spp
        o = _HitArrays(R, with_t=False) if outputs else None
        n = C.c_uint64(0)
        sec = self.ref.lib.ref_render_mt(
            self.h, np.ascontiguousarray(cam10, np.float32), film_w, film_h, nx, ny, spp,
            _opt(o.hit) if o else None, _opt(o.cell) if o else None, _opt(o.tri) if o else None,
            _opt(o.pos) if o else None, _opt(o.nrm) if o else None, C.byref(n))
        return float(sec), int(n.value), o

    def _gi(self, name):
        return getattr(self.ref.lib, "ref_gi_" + name)

    # -- GI rows (SURVEY.md 8f): same method names on PortTree and RefScene -----------------
    def gi_reset(self):
        self._gi("reset")(self.h)

    def gi_filter(self):
        self._gi("filter")(self.h)

    def gi_level(self, level):
        """(cells[n,3], coverage[n], illum[n,6,3]) of the nodes of `level` with coverage > 0, Morton order."""
        f = self._gi("dump_level")
        n = int(f(self.h, int(level), None, None, None, 0))
        cells = np.zeros((n, 3), np.uint32)
        cov = np.zeros(n, np.float32)
        il = np.zeros((n, 6, 3), np.float32)
        if n:
            f(self.h, int(level), cells.ctypes.data, cov.ctypes.data, il.ctypes.data, n)
        return cells, cov, il

    def gi_cone_trace(self, pos, nrm, res):
        pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 3)
        nrm = np.ascontiguousarray(nrm, np.float32).reshape(-1, 3)
        out = np.zeros((len(pos), 3), np.float32)
        self._gi("cone_trace")(self.h, pos, nrm, len(pos), float(np.float32(res)), out)
        return out

    def albedo(self, tri, pos):
        tri = np.ascontiguousarray(tri, np.uint32)
        pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 3)
        out = np.zeros((len(tri), 3), np.float32)
        self.ref.lib.ref_albedo(self.h, tri, pos, len(tri), out)
        return out

    def gi_splat(self, cam10, film_h, nx, ny, spp, kd, film_w=1.0):
        self.ref.lib.ref_scene_set_diffuse(self.h, np.ascontiguousarray(kd, np.float32))
        self.ref.lib.ref_gi_splat(self.h, np.ascontiguousarray(cam10, np.float32), float(film_w), float(film_h),
                                  nx, ny, spp)

    def gi_render(self, cam10, film_h, nx, ny, spp, res, kd=None, nthreads=1, film_w=1.0):
        if kd is not None:
            self.ref.lib.ref_scene_set_diffuse(self.h, np.ascontiguousarray(kd, np.float32))
        film = np.zeros((ny, nx, 3), np.float32)
        self.seconds = float(self.ref.lib.ref_gi_render(self.h, np.ascontiguousarray(cam10, np.float32), float(film_w),
                                                        float(film_h), nx, ny, spp, float(np.float32(res)), film,
                                                        int(nthreads)))
        return film
