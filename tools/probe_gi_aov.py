"""GI film with its planes (vrt_gi_render_aov_dev) against the GI film alone (vrt_gi_render_camera_dev) on main.cc's
image: the atrium at 1024^3, light film 2048^2 x 4, GI film 3840 x 2160 x 4 (f32 film), all device-resident.
Prints one JSON line (and writes it to --out when given).

Three calls alternate frame by frame in one process: the film alone, the film plus every plane (albedo, direct,
indirect, normal, hits) and the film plus the hit records only.  After --warmup rounds, each is timed over --frames
rounds: the kernel with the CUDA events the library records around every trace launch (mean_kernel_ms), and the
whole call with a host clock around call + sync.  The outputs of the last round are checked bytewise: films against
the film alone, hits against trace_camera16_dev, and the planes of the two AOV calls against each other."""
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--depth", type=int, default=11)
    ap.add_argument("--light", type=int, default=2048)
    ap.add_argument("--nx", type=int, default=3840)
    ap.add_argument("--ny", type=int, default=2160)
    ap.add_argument("--frames", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    capi.load()
    if capi.device_count() < 1:
        raise SystemExit("probe_gi_aov needs a CUDA device")
    tri, nrm = scenes.atrium()
    tree = capi.Octree.build(tri, nrm, a.depth)
    res = gi_res(tree.info()["root_aabb"], a.depth)
    lcam = capi.Camera(CAM_LIGHT[0], CAM_LIGHT[1:4], CAM_LIGHT[4:7], CAM_LIGHT[7:10], a.light, a.light, 4)
    spp = 4
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], a.nx, a.ny, spp)
    tree.gi_init()
    tree.gi_splat(lcam, GI_KD)
    tree.gi_filter()
    tree.sync()

    shape = (a.ny, a.nx, 3)
    films = {k: torch.empty(shape, dtype=torch.float32, device="cuda") for k in ("film", "all", "hits")}
    planes = {n: torch.empty(shape, dtype=torch.float32, device="cuda") for n in ("albedo", "direct", "indirect", "normal")}
    hits = {k: torch.empty((a.ny * a.nx * spp * 4,), dtype=torch.int32, device="cuda") for k in ("all", "hits")}
    planes_ptr = {n: t.data_ptr() for n, t in planes.items()}
    calls = {
        "film": lambda: tree.gi_render_dev(cam, GI_KD, res, films["film"].data_ptr()),
        "all": lambda: tree.gi_render_aov_dev(cam, GI_KD, res, films["all"].data_ptr(),
                                              dict(planes_ptr, hits=hits["all"].data_ptr())),
        "hits": lambda: tree.gi_render_aov_dev(cam, GI_KD, res, films["hits"].data_ptr(),
                                               {"hits": hits["hits"].data_ptr()}),
    }
    kernel = {k: [] for k in calls}
    call = {k: [] for k in calls}
    for r in range(a.warmup + a.frames):
        for k, fn in calls.items():
            t0 = time.perf_counter()
            fn()
            tree.sync()
            t1 = time.perf_counter()
            if r >= a.warmup:
                kernel[k].append(tree.mean_kernel_ms(1))
                call[k].append((t1 - t0) * 1e3)

    ref_hits = torch.empty_like(hits["all"])
    tree.trace_camera_dev(cam, ref_hits.data_ptr(), compact=True)
    tree.sync()
    checks = dict(
        film_all_eq_film=bool(torch.equal(films["all"].view(torch.int32), films["film"].view(torch.int32))),
        film_hits_eq_film=bool(torch.equal(films["hits"].view(torch.int32), films["film"].view(torch.int32))),
        hits_all_eq_trace_camera16=bool(torch.equal(hits["all"], ref_hits)),
        hits_only_eq_trace_camera16=bool(torch.equal(hits["hits"], ref_hits)),
    )
    stats = {}
    for k in calls:
        kk, cc = np.array(kernel[k]), np.array(call[k])
        stats[k] = dict(kernel_ms_mean=float(kk.mean()), kernel_ms_min=float(kk.min()), kernel_ms_max=float(kk.max()),
                        call_ms_mean=float(cc.mean()))
    base = stats["film"]["kernel_ms_mean"]
    for k in ("all", "hits"):
        stats[k]["kernel_ratio_vs_film"] = stats[k]["kernel_ms_mean"] / base
    line = dict(probe="gi_aov", gpus=gpu_info(), scene=f"atrium depth {a.depth}", light_film=[a.light, a.light, 4],
                gi_film=[a.nx, a.ny, spp], film_format="f32", frames=a.frames, warmup=a.warmup, res=float(res),
                stats=stats, target="all-planes kernel <= 1.05 x film kernel",
                target_met=bool(stats["all"]["kernel_ratio_vs_film"] <= 1.05), checks=checks,
                tree_nodes=tree.info()["num_nodes"])
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    tree.close()


if __name__ == "__main__":
    main()
