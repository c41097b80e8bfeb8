"""Shared helpers for the parity tests (inputs, comparison, harness pixel)."""
import numpy as np

from voxelraytrace20190722_b200 import scenes

RAD = np.pi / 180.0
CAM_SPHERE = np.array([60 * RAD, 0, 1, 3, 0, 0, 0, 0, 1, 0], np.float32)       # SURVEY 8d config 2
CAM_MAIN = np.array([90 * RAD, 1, 1.3, -.2, 0, .4, 0, 0, 1, 0], np.float32)     # main.cc:112-115
CAM_LIGHT = np.array([60 * RAD, 1, 10, 1, 0, 0, 0, 0, 1, 0], np.float32)        # main.cc:76-78


def bits(a):
    a = np.ascontiguousarray(a)
    if a.dtype == np.float32:
        return a.view(np.uint32)
    if a.dtype == np.float64:
        return a.view(np.uint64)
    return a


def assert_bits_equal(a, b, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    ne = bits(a) != bits(b)
    assert not ne.any(), f"{what}: {int(ne.sum())} of {ne.size} elements differ (first at {np.argwhere(ne)[0]})"


def leaves_equal(a, b):
    """(cells, counts, refs) triples, both in Morton order."""
    for x, y, nm in zip(a, b, ("leaf cells", "leaf counts", "leaf refs")):
        assert_bits_equal(x, y, nm)


def compare_hits(gpu_hits, orc, what="", allow_mismatch=0.0):
    """gpu_hits: structured HIT array; orc: oracle _HitArrays.  Bit-exact by default."""
    n = len(gpu_hits)
    bad = (gpu_hits["hit"] != orc.hit)
    bad |= gpu_hits["tri"] != orc.tri
    bad |= (gpu_hits["cell"] != orc.cell).any(axis=1)
    frac = bad.sum() / max(n, 1)
    assert frac <= allow_mismatch, f"{what}: {int(bad.sum())}/{n} rays differ in (hit, leaf cell, triangle)"
    ok = ~bad
    assert_bits_equal(gpu_hits["pos"][ok], orc.pos[ok], what + " ISect.hit")
    assert_bits_equal(gpu_hits["nrm"][ok], orc.nrm[ok], what + " ISect.normal")
    if getattr(orc, "t", None) is not None:
        assert_bits_equal(gpu_hits["t"][ok], orc.t[ok], what + " t")
    return int(bad.sum())


def shadow_rays(orc_hits, light, eps):
    """Harness shadow rays (config 5): origin = hit + eps*normal (float32 ops), direction = light."""
    f32 = np.float32
    o = (orc_hits.pos + (f32(eps) * orc_hits.nrm).astype(np.float32)).astype(np.float32)
    r = np.zeros((len(o), 8), np.float32)
    r[:, 0:3] = o
    r[:, 3:6] = np.asarray(light, np.float32)
    r[:, 7] = np.finfo(np.float32).max
    return r


def harness_film(rays, orc_hits, light, kd, spp, visibility=None):
    """The harness pixel of SURVEY.md 8(d) evaluated on ORACLE hits with numpy float32
    (sky: main.cc:18-20; samples added in order with weight 1/spp: main.cc:119-122)."""
    f32 = np.float32
    d = rays.reshape(-1, 8)[:, 3:6].astype(np.float32)
    t = (0.5 * (d[:, 1].astype(np.float64) + 1.0)).astype(np.float32)
    v1 = np.array([0.6, 0.8, 1.0], np.float32)
    sky = (f32(1.0) + (v1[None, :] - f32(1.0)) * t[:, None]).astype(np.float32)
    n = orc_hits.nrm.astype(np.float32)
    L = np.asarray(light, np.float32)
    dot = (f32(0) + n[:, 0] * L[0]).astype(np.float32)
    dot = (dot + n[:, 1] * L[1]).astype(np.float32)
    dot = (dot + n[:, 2] * L[2]).astype(np.float32)
    dot = np.where(dot > 1, f32(1), np.where(dot < 0, f32(0), dot)).astype(np.float32)
    c = (f32(kd) * dot).astype(np.float32)
    if visibility is not None:
        c = (c * visibility.astype(np.float32)).astype(np.float32)
    col = np.where(orc_hits.hit[:, None].astype(bool), c[:, None].repeat(3, 1), sky).astype(np.float32)
    w = f32(0.25) if spp == 4 else f32(1)
    col = (col * w).astype(np.float32).reshape(-1, spp, 3)
    acc = np.zeros((col.shape[0], 3), np.float32)
    for s in range(spp):
        acc = (acc + col[:, s]).astype(np.float32)
    return acc


def to_u8(film):
    """Film::to_byte_array (camera.cc:25-47): v*255.9 -> uint8 cast."""
    return np.clip(film.astype(np.float32) * np.float32(255.9), 0, 255).astype(np.uint8)


def small_scenes():
    """(name, tri, nrm, depth, cam10) cases that the oracle finishes in seconds."""
    out = []
    tri, nrm = scenes.uv_sphere(64, 32)
    out.append(("sphere64_d6", tri, nrm, 6, CAM_SPHERE))
    tri, nrm = scenes.uv_sphere()
    out.append(("sphere256_d8", tri, nrm, 8, CAM_SPHERE))
    tri, nrm = scenes.soup(20000, e=0.02)
    out.append(("soup20k_d7", tri, nrm, 7, CAM_SPHERE))
    tri, nrm = scenes.atrium(detail=0.35)
    out.append(("atrium_d7", tri, nrm, 7, CAM_MAIN))
    return out


def gi_res(root_aabb, max_depth):
    """main.cc:69-70: Res = min over axes of root.aabb.size() / powf(2, max_depth)."""
    root = np.asarray(root_aabb, np.float32)
    return np.float32(((root[3:] - root[:3]) / np.float32(2.0 ** max_depth)).min())


def gi_maxdist(root_aabb):
    """cone_trace's maxdist = length(root.aabb.size()), float32 with jql::dot's order (voxel_octree.cc:250)."""
    root = np.asarray(root_aabb, np.float32)
    s = (root[3:] - root[:3]).astype(np.float32)
    d = np.float32(0)
    for k in range(3):
        d = np.float32(d + np.float32(s[k] * s[k]))
    return np.sqrt(d, dtype=np.float32)


def gi_march(maxdist, res, limit=100000):
    """The march of cone_trace (voxel_octree.cc:252-281) in float32: the level int(log2f(maxdist / diam)) sampled at
    each step (log2f correctly rounded; None where the ratio is not a positive float), and whether the march ends --
    False when dist stops advancing (0, negative or subnormal res) or `limit` steps pass.  It depends on res and the
    root box only, not on the cone."""
    f32 = np.float32
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        maxdist, res = f32(maxdist), f32(res)
        mindist = f32(f32(1.414) * res)
        ap2 = f32(f32(0.577350269) * f32(2))
        dist = mindist
        levels = []
        while dist < maxdist:
            a = f32(ap2 * dist)
            diam = a if mindist < a else mindist
            if maxdist < diam:
                break
            if len(levels) == limit:
                return levels, False
            q = f32(maxdist / diam)
            levels.append(int(f32(np.log2(np.float64(q)))) if 0 < q < np.inf else None)
            nxt = f32(dist + f32(f32(0.1) * diam))
            if not nxt > dist:
                return levels, False
            dist = nxt
    return levels, True


GI_KD = np.array([0.7, 0.6, 0.5], np.float32)  # the scene's single untextured material (material_t::diffuse)


def write_tga(path, img):
    """Uncompressed top-left-origin TGA (24/32-bit true colour or 8-bit grey) from a uint8 [h, w, c] array --
    a format the reference's stb_image decodes back to exactly these bytes."""
    img = np.ascontiguousarray(img, np.uint8)
    h, w, c = img.shape
    hdr = bytearray(18)
    hdr[2] = 2 if c >= 3 else 3
    hdr[12], hdr[13], hdr[14], hdr[15] = w & 255, w >> 8, h & 255, h >> 8
    hdr[16] = 8 * c
    hdr[17] = 0x20 | (8 if c == 4 else 0)
    data = img[..., [2, 1, 0, 3][:c]] if c >= 3 else img
    with open(path, "wb") as f:
        f.write(bytes(hdr) + np.ascontiguousarray(data).tobytes())


def textured_case(seed=3, nu=48, nv=24):
    """A sphere with random texture coordinates (outside [0,1] too: unit_cycle), four materials, two of them
    textured (3- and 4-channel images).  Returns a dict of plain arrays."""
    rng = np.random.default_rng(seed)
    tri, nrm = scenes.uv_sphere(nu, nv)
    T = len(tri)
    uv = rng.uniform(-0.5, 2.5, (T, 3, 2)).astype(np.float32)
    uv[: T // 8] = np.round(uv[: T // 8] * 4) / 4   # coordinates exactly on texel / cycle boundaries
    return dict(tri=tri, nrm=nrm, uv=uv, mtl=rng.integers(0, 4, T).astype(np.uint32),
                kd=rng.uniform(0.2, 0.9, (4, 3)).astype(np.float32), mtl_tex=np.array([-1, 0, -1, 1], np.int32),
                tex0=rng.integers(0, 256, (17, 23, 3), dtype=np.uint8), tex1=rng.integers(0, 256, (8, 8, 4), dtype=np.uint8))


def export_test_film(ny=64, nx=64, seed=3):
    """A float film [ny][nx][3] (square when it goes through the reference, see Ref.film_to_bytes) that exercises the export encodings: plain [0,1)
    colours, constant runs of every length class of the RLE (3, 127, 128, 129 ...), exact zeros, values below the
    1e-32 cut, powers of two and their neighbours, bright (> 1) and huge values, and a few negative components."""
    rng = np.random.default_rng(seed)
    f = rng.uniform(0.0, 1.0, (ny, nx, 3)).astype(np.float32)
    if ny < 14:  # a small film: just the value classes, row by row as far as they fit
        f[0, :, :] = rng.uniform(0, 3e-32, (nx, 3)).astype(np.float32)
        f[1, :, :] = rng.uniform(1.0, 40.0, (nx, 3)).astype(np.float32)
        f[2, :, 2] = -rng.uniform(0, 2.0, nx).astype(np.float32)
        f[3, :, :] = 0.0
        return f
    f[1, :, :] = 0.25                       # one run over the whole row
    f[2, 3:6, :] = f[2, 3, :]               # run of exactly 3
    f[3, : nx - 1, 1] = 0.5                 # run that stops one short of the row end
    f[4, :, :] = 0.0
    f[5, :, :] = rng.uniform(0, 3e-32, (nx, 3)).astype(np.float32)
    p2 = np.float32(2.0) ** rng.integers(-20, 12, nx).astype(np.float32)
    f[6, :, 0] = p2
    f[7, :, 0] = np.nextafter(p2, np.float32(0))
    f[8, :, 0] = np.nextafter(p2, np.float32(np.inf))
    f[9, :, :] = rng.uniform(1.0, 40.0, (nx, 3)).astype(np.float32)
    f[10, :, :] = rng.uniform(0, 1e10, (nx, 3)).astype(np.float32)
    f[11, :, 2] = -rng.uniform(0, 2.0, nx).astype(np.float32)
    f[12, :, :] = 1.0
    f[13, ::2, :] = 0.999999
    if ny > 20:
        f[14:20, :, :] = (f[14:20, :, :] * 4).astype(np.int32).astype(np.float32) / 4  # quantised: many short runs
    return f
