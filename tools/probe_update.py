"""Animated geometry: what moving one object costs per frame.  Scene: the atrium at 1024^3 (depth 11) plus the
config-2 UV sphere (65,024 triangles) scaled to r = 0.15 and appended as the last triangles; the sphere moves on a
circle, turning as it goes, one step per frame.  Prints one JSON line (and writes it to --out when given).

Variants, alternated within the run (--reps blocks, each with warm-up):
  1. update cost (host clock around each call; every one returns synchronised):
       xform        Octree.update_xform of the sphere's range (vrt_update_xform)
       rebuild      Octree.rebuild of the same handle (vrt_rebuild)
       fresh        what callers had to do before: Octree.build from host triangles + set_materials + film format
  2. primary film, pipelined 3840 x 2160 x 4 RGBE (render_async into two pinned host frames):
       film_static  the loop alone;   film_xform  the loop with update_xform before every frame
  3. GI film, pipelined 3840 x 2160 x 4 RGBE (gi_render_bands_async, bands {ny, 0, 1}):
       gi_static    the loop alone;   gi_xform    + update_xform, gi_init, the 2048^2 x 4 splat and the filter per frame
  4. the last frame of every animated variant against the same frame of a fresh build of that pose (bytewise)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.common import CAM_LIGHT, CAM_MAIN, GI_KD, gi_res  # noqa: E402
from voxelraytrace20190722_b200 import capi, scenes  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except Exception as e:  # noqa: BLE001
        out = [f"nvidia-smi failed: {e}"]
    return out


def sphere_xform(k, first, count, centre, radius):
    """Frame k's transform of the sphere (rest pose: centred on the origin): a turn of 0.2 rad per frame about y,
    then the point k / 16 of the way round a horizontal circle about `centre`."""
    a = 0.2 * k
    c, s = np.cos(a), np.sin(a)
    r = np.array([[c, 0, s], [0, 1, 0], [-s, 0, c]])
    b = 2 * np.pi * k / 16
    p = np.asarray(centre, np.float64) + radius * np.array([np.cos(b), 0.0, np.sin(b)])
    return (first, count, np.concatenate([r, p[:, None]], 1).astype(np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depth", type=int, default=11)
    ap.add_argument("--light", type=int, default=2048)
    ap.add_argument("--nx", type=int, default=3840)
    ap.add_argument("--ny", type=int, default=2160)
    ap.add_argument("--frames", type=int, default=12)
    ap.add_argument("--updates", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    capi.load()
    if capi.device_count() < 1:
        raise SystemExit("probe_update needs a CUDA device")
    info = gpu_info()
    atri, anrm = scenes.atrium()
    stri, snrm = scenes.uv_sphere()
    stri = (np.asarray(stri, np.float32) * np.float32(0.15)).astype(np.float32)
    tri = np.concatenate([np.asarray(atri, np.float32).reshape(-1, 9), stri.reshape(-1, 9)])
    nrm = np.concatenate([np.asarray(anrm, np.float32).reshape(-1, 9), np.asarray(snrm, np.float32).reshape(-1, 9)])
    T, S = len(tri), len(stri)
    first = T - S
    box = capi.Octree.build(atri, anrm, 4).info()["root_aabb"].astype(np.float64)
    centre = (box[:3] + box[3:]) / 2
    radius = 0.25 * min(box[3] - box[0], box[5] - box[2])
    mats = (np.zeros((T, 6), np.float32), np.zeros(T, np.uint32), GI_KD.reshape(1, 3), np.array([-1], np.int32), [])

    def xf(k):
        return [sphere_xform(k, first, S, centre, radius)]

    def setup(t):
        t.set_materials(*mats)
        t.set_film_format("rgbe")

    tree = capi.Octree.build(tri, nrm, a.depth)
    setup(tree)
    tree.update_xform(xf(0))
    res = gi_res(tree.info()["root_aabb"], a.depth)
    lcam = capi.Camera(CAM_LIGHT[0], CAM_LIGHT[1:4], CAM_LIGHT[4:7], CAM_LIGHT[7:10], a.light, a.light, 4)
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], a.nx, a.ny, 4)
    frames = [torch.full((a.ny, a.nx, 4), 7, dtype=torch.uint8).pin_memory() for _ in range(2)]

    def lit(t):
        t.gi_init()
        t.gi_splat(lcam, GI_KD)
        t.gi_filter()

    lit(tree)
    clock = [1]  # pose counter of the animated loops

    # ---- 1. update cost ----
    def pose(k):
        """frame k's pose as the kernel computes it: ((m0*x + m1*y) + m2*z) + m3 in float32, normals by the inverse
        transpose (= the rotation)"""
        f, n, m = xf(k)[0]
        nm = capi.xform_normal_matrix(m)
        t, q = tri.copy(), nrm.copy()
        for arr, mat, w in ((t, m, 4), (q, nm, 3)):
            p = arr[f:f + n].reshape(-1, 3)
            o = np.empty_like(p)
            for r in range(3):
                v = (mat[r, 0] * p[:, 0]).astype(np.float32) + (mat[r, 1] * p[:, 1]).astype(np.float32)
                v = v.astype(np.float32) + (mat[r, 2] * p[:, 2]).astype(np.float32)
                o[:, r] = (v.astype(np.float32) + mat[r, 3]).astype(np.float32) if w == 4 else v
            arr[f:f + n] = o.reshape(-1, 9)
        return t, q

    fresh_pose = pose(1)

    def fresh_build():  # (the pose is computed outside the timed call)
        t = capi.Octree.build(*fresh_pose, a.depth)
        setup(t)
        t.close()

    def do_xform():
        tree.update_xform(xf(clock[0]))
        clock[0] += 1

    cost = {"xform": do_xform, "rebuild": lambda: tree.rebuild(a.depth), "fresh": fresh_build}
    cost_runs = {n: [] for n in cost}

    # ---- 2./3. pipelined loops ----
    def film_frame(i, animate):
        if animate:
            do_xform()
        tree.render_async(cam, frames[i & 1].numpy())

    def gi_frame(i, animate):
        if animate:
            do_xform()
            lit(tree)
        tree.gi_render_bands_async(cam, GI_KD, res, frames[i & 1].data_ptr(), a.ny, 0, 1)

    loops = {"film_static": (film_frame, False), "film_xform": (film_frame, True),
             "gi_static": (gi_frame, False), "gi_xform": (gi_frame, True)}
    loop_runs = {n: [] for n in loops}
    checks = {}

    def check_last(kind):
        """last frame of an animated loop vs the frame of a fresh build of the pose it rendered"""
        tree.sync()
        got = frames[(a.frames - 1) & 1].numpy().copy()
        fresh = capi.Octree.build(*pose(clock[0] - 1), a.depth)
        setup(fresh)
        buf = torch.full((a.ny, a.nx, 4), 7, dtype=torch.uint8).pin_memory()
        if kind == "film":
            fresh.render_async(cam, buf.numpy())
        else:
            lit(fresh)
            fresh.gi_render_bands_async(cam, GI_KD, res, buf.data_ptr(), a.ny, 0, 1)
        fresh.sync()
        fresh.close()
        return bool(np.array_equal(got, buf.numpy()))

    for rep in range(a.reps):
        for name, fn in cost.items():
            for _ in range(a.warmup):
                fn()
            for _ in range(a.updates):
                t0 = time.perf_counter()
                fn()
                cost_runs[name].append((time.perf_counter() - t0) * 1e3)
            print(json.dumps(dict(rep=rep, variant=name, ms=float(np.median(cost_runs[name][-a.updates:])))),
                  file=sys.stderr, flush=True)
        for name, (frame, animate) in loops.items():
            for i in range(a.warmup):
                frame(i, animate)
            tree.sync()
            t0 = time.perf_counter()
            for i in range(a.frames):
                frame(i, animate)
            tree.sync()
            ms = (time.perf_counter() - t0) * 1e3 / a.frames
            loop_runs[name].append(ms)
            if animate:
                ok = check_last("film" if name.startswith("film") else "gi")
                checks[name] = checks.get(name, True) and ok
            print(json.dumps(dict(rep=rep, variant=name, frame_ms=ms)), file=sys.stderr, flush=True)
            if name == "film_xform" or name == "gi_xform":
                lit(tree)  # the static GI loop after an animated one needs a lit tree

    out = dict(
        update_ms={n: dict(median=float(np.median(v)), min=float(np.min(v)), runs=len(v)) for n, v in cost_runs.items()},
        frame_ms={n: dict(median=float(np.median(v)), runs=v) for n, v in loop_runs.items()},
        last_frame_equals_fresh_build=checks,
    )
    out["film_xform_over_static"] = out["frame_ms"]["film_xform"]["median"] / out["frame_ms"]["film_static"]["median"]
    out["gi_xform_over_static"] = out["frame_ms"]["gi_xform"]["median"] / out["frame_ms"]["gi_static"]["median"]
    line = dict(probe="update", gpus=info, visible_devices=capi.device_count(),
                scene=f"atrium + uv_sphere(256,128) r=0.15, depth {a.depth}", num_tris=T, moving_tris=S,
                light_film=[a.light, a.light, 4], film=[a.nx, a.ny, 4], film_format="rgbe", frames=a.frames,
                updates=a.updates, warmup=a.warmup, reps=a.reps, tree_nodes=tree.info()["num_nodes"], **out,
                not_measured="several GPUs (MultiGpu updates): one GPU visible" if capi.device_count() < 2 else "")
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    tree.close()


if __name__ == "__main__":
    main()
