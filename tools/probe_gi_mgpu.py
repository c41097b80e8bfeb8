"""GI film on several GPUs: main.cc's image (atrium 1024^3, light film 2048^2 x 4, GI film 3840 x 2160 x 4) through
MultiGpu for the device lists [0], [0,0] and [0..N-1] (N = 2, 4, 8 as available), against gi_render_dev on the
source tree.  Prints one JSON line (and writes it to --out when given).

Per device list: the light pass on all replicas (host clock around gi_init / gi_splat / gi_filter + sync), the
pipelined frame time (host clock around F frames enqueued on two pinned host frames, ending in MultiGpu.sync(); RGBE
and f32 films), the mean kernel time of every replica over those frames, and whether the frame equals the
one-device frame bytewise."""
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
    ndev = capi.device_count()
    if ndev < 1:
        raise SystemExit("probe_gi_mgpu needs a CUDA device")
    tri, nrm = scenes.atrium()
    tree = capi.Octree.build(tri, nrm, a.depth)
    res = gi_res(tree.info()["root_aabb"], a.depth)
    lcam = capi.Camera(CAM_LIGHT[0], CAM_LIGHT[1:4], CAM_LIGHT[4:7], CAM_LIGHT[7:10], a.light, a.light, 4)
    cam = capi.Camera(CAM_MAIN[0], CAM_MAIN[1:4], CAM_MAIN[4:7], CAM_MAIN[7:10], a.nx, a.ny, 4)
    F = a.frames

    # one device, whole film into device memory (no copy): the reference point
    tree.gi_init()
    tree.gi_splat(lcam, GI_KD)
    tree.gi_filter()
    tree.sync()
    dev = {}
    ref_rgbe = None
    for fmt in ("rgbe", "f32"):
        tree.set_film_format(fmt)
        d_film = torch.empty(a.ny * a.nx * capi.film_pixel_bytes(fmt), dtype=torch.uint8, device="cuda")
        for _ in range(a.warmup):
            tree.gi_render_dev(cam, GI_KD, res, d_film.data_ptr())
        tree.sync()
        t0 = time.perf_counter()
        for _ in range(F):
            tree.gi_render_dev(cam, GI_KD, res, d_film.data_ptr())
        tree.sync()
        dev[fmt] = dict(frame_ms=(time.perf_counter() - t0) * 1e3 / F, kernel_ms=tree.mean_kernel_ms(F))
        if fmt == "rgbe":
            ref_rgbe = d_film.cpu().numpy()
        del d_film
    tree.set_film_format("f32")

    lists = [[0], [0, 0]] + [list(range(n)) for n in (2, 4, 8) if n <= ndev]
    rows = []
    one_dev = None
    for devices in lists:
        mg = capi.MultiGpu(tree, devices)
        row = dict(devices=devices)
        t0 = time.perf_counter()
        mg.gi_init()
        mg.gi_splat(lcam, GI_KD)
        mg.gi_filter()
        mg.sync()
        row["light_pass_ms"] = (time.perf_counter() - t0) * 1e3
        for fmt in ("rgbe", "f32"):
            mg.set_film_format(fmt)
            pb = capi.film_pixel_bytes(fmt)
            bufs = [torch.full((a.ny * a.nx * pb,), 7, dtype=torch.uint8).pin_memory() for _ in range(2)]
            for i in range(a.warmup):
                mg.gi_render_async(cam, GI_KD, res, bufs[i & 1].data_ptr())
            mg.sync()
            t0 = time.perf_counter()
            for i in range(F):
                mg.gi_render_async(cam, GI_KD, res, bufs[i & 1].data_ptr())
            mg.sync()
            ms = (time.perf_counter() - t0) * 1e3 / F
            k = [mg.mean_kernel_ms(i, F) for i in range(len(devices))]
            row[fmt] = dict(frame_ms=ms, kernel_ms_per_device=k, kernel_max_over_mean=max(k) / (sum(k) / len(k)))
            if fmt == "rgbe":
                frame = bufs[(F - 1) & 1].numpy().copy()
                if devices == [0]:
                    one_dev = frame
                    row["frame_check_vs_gi_render_dev"] = bool(np.array_equal(frame, ref_rgbe))
                row["frame_check"] = bool(np.array_equal(frame, one_dev))
            del bufs
        mg.close()
        rows.append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)

    base = rows[0]
    for row in rows:
        for fmt in ("rgbe", "f32"):
            r = row[fmt]
            r["speedup_vs_list0"] = base[fmt]["frame_ms"] / r["frame_ms"]
            r["speedup_vs_gi_render_dev"] = dev[fmt]["frame_ms"] / r["frame_ms"]
            n = len(set(row["devices"]))
            r["target_ms"] = 1.15 * base[fmt]["frame_ms"] / n  # <= 1.15 x (1-device time / N)
    line = dict(probe="gi_mgpu", gpus=gpu_info(), visible_devices=ndev, scene=f"atrium depth {a.depth}",
                light_film=[a.light, a.light, 4], gi_film=[a.nx, a.ny, 4], frames=F, warmup=a.warmup,
                gi_render_dev=dev, lists=rows, tree_nodes=tree.info()["num_nodes"])
    s = json.dumps(line)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    tree.close()


if __name__ == "__main__":
    main()
