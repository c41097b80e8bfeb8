"""The GI film's planes in the pipelined frame loop: main.cc's image (atrium 1024^3, light film 2048^2 x 4, GI film
3840 x 2160 x 4, f32 film) enqueued frame after frame into pinned host frames.  Prints one JSON line (and writes it
to --out when given).

Variants, alternated within the run (--reps blocks of --warmup + --frames frames each):
  film_only       Octree.gi_render_bands_async with bands {ny, 0, 1} (the film alone)
  aov_bands       Octree.gi_render_aov_bands_async with {ny, 0, 1}: the film plus all five planes
  aov_mgpu_[0]    MultiGpu([0]).gi_render_aov_async: the same frame through one replica
  aov_mgpu_[0,0]  MultiGpu([0, 0]).gi_render_aov_async: through two replicas on one device
Per variant: the frame time (host clock around the enqueued frames, ending in a sync), the mean kernel time of every
device's handle over those frames, the bytes copied to the host per frame (from the shapes), and whether the last
frame equals gi_render_aov_dev on the source tree bytewise.  Frames alternate between two sets of host frames."""
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

PLANES = capi.GI_AOV_PLANES


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except Exception as e:  # noqa: BLE001
        out = [f"nvidia-smi failed: {e}"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depth", type=int, default=11)
    ap.add_argument("--light", type=int, default=2048)
    ap.add_argument("--nx", type=int, default=3840)
    ap.add_argument("--ny", type=int, default=2160)
    ap.add_argument("--frames", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    capi.load()
    if capi.device_count() < 1:
        raise SystemExit("probe_gi_aov_mgpu needs a CUDA device")
    info = gpu_info()
    tri, nrm = scenes.atrium()
    tree = capi.Octree.build(tri, nrm, a.depth)
    res = gi_res(tree.info()["root_aabb"], a.depth)
    lcam = capi.Camera(CAM_LIGHT[0], CAM_LIGHT[1:4], CAM_LIGHT[4:7], CAM_LIGHT[7:10], a.light, a.light, 4)
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], a.nx, a.ny, 4)
    npix, F = a.nx * a.ny, a.frames
    nbytes = {"film": npix * 12, "hits": npix * 4 * 16, **{n: npix * 12 for n in PLANES[:4]}}

    tree.gi_init()
    tree.gi_splat(lcam, GI_KD)
    tree.gi_filter()
    # the reference: the film and every plane into device memory in one launch
    d = {n: torch.empty(b, dtype=torch.uint8, device="cuda") for n, b in nbytes.items()}
    tree.gi_render_aov_dev(cam, GI_KD, res, d["film"].data_ptr(), {n: d[n].data_ptr() for n in PLANES})
    tree.sync()
    ref = {n: t.cpu().numpy() for n, t in d.items()}
    del d
    sets = [{n: torch.full((b,), 7, dtype=torch.uint8).pin_memory() for n, b in nbytes.items()} for _ in range(2)]

    def planes(s):
        return {n: s[n].data_ptr() for n in PLANES}

    mgs = {}
    for devices in ([0], [0, 0]):
        mg = capi.MultiGpu(tree, devices)
        mg.gi_init()
        mg.gi_splat(lcam, GI_KD)
        mg.gi_filter()
        mg.sync()
        mgs[str(devices).replace(" ", "")] = mg

    def tree_kernel_ms():
        return [tree.mean_kernel_ms(F)]

    variants = {
        "film_only": (lambda s: tree.gi_render_bands_async(cam, GI_KD, res, s["film"].data_ptr(), a.ny, 0, 1),
                      tree.sync, tree_kernel_ms, ("film",)),
        "aov_bands": (lambda s: tree.gi_render_aov_bands_async(cam, GI_KD, res, s["film"].data_ptr(), planes(s),
                                                               a.ny, 0, 1),
                      tree.sync, tree_kernel_ms, tuple(nbytes)),
    }
    for key, mg in mgs.items():
        variants[f"aov_mgpu_{key}"] = (
            lambda s, mg=mg: mg.gi_render_aov_async(cam, GI_KD, res, s["film"].data_ptr(), planes(s)), mg.sync,
            lambda mg=mg: [mg.mean_kernel_ms(i, F) for i in range(mg.num_devices)], tuple(nbytes))

    runs = {name: [] for name in variants}
    checks = {}
    for rep in range(a.reps):
        for name, (enqueue, sync, kernel_ms, outs) in variants.items():
            for s in sets:
                for t in s.values():
                    t.fill_(7)
            for i in range(a.warmup):
                enqueue(sets[i & 1])
            sync()
            t0 = time.perf_counter()
            for i in range(F):
                enqueue(sets[i & 1])
            sync()
            ms = (time.perf_counter() - t0) * 1e3 / F
            runs[name].append(dict(frame_ms=ms, mean_kernel_ms=kernel_ms()))
            last = sets[(F - 1) & 1]
            checks[name] = checks.get(name, True) and all(np.array_equal(last[n].numpy(), ref[n]) for n in outs)
            print(json.dumps(dict(rep=rep, variant=name, **runs[name][-1])), file=sys.stderr, flush=True)

    out = {}
    for name, (_, _, _, outs) in variants.items():
        fr = [r["frame_ms"] for r in runs[name]]
        out[name] = dict(frame_ms=float(np.median(fr)), frame_ms_runs=fr,
                         mean_kernel_ms=[float(np.median(k)) for k in zip(*[r["mean_kernel_ms"] for r in runs[name]])],
                         bytes_to_host_per_frame=int(sum(nbytes[n] for n in outs)),
                         last_frame_equals_gi_render_aov_dev=bool(checks[name]))
    base = out["film_only"]["frame_ms"]
    for name in out:
        out[name]["frame_ms_over_film_only"] = out[name]["frame_ms"] / base
    line = dict(probe="gi_aov_mgpu", gpus=info, visible_devices=capi.device_count(), scene=f"atrium depth {a.depth}",
                light_film=[a.light, a.light, 4], gi_film=[a.nx, a.ny, 4], film_format="f32", frames=F,
                warmup=a.warmup, reps=a.reps, variants=out, tree_nodes=tree.info()["num_nodes"],
                not_measured=f"frame times on 2, 4 and 8 GPUs ({capi.device_count()} visible)")
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    for mg in mgs.values():
        mg.close()
    tree.close()


if __name__ == "__main__":
    main()
