"""Cost of the per-eye work of the camera launches (eye-relative hull records and triangle terms): device time of a
hit16 launch plus everything the library enqueues before it, with a fixed eye (slots reused) and with a new eye on
every launch (slots refilled), eye-relative records on and off.  Usage: probe_eye_rel.py [depth ...]"""
import sys

import numpy as np
import torch

sys.path.insert(0, '.')
from voxelraytrace20190722_b200 import capi, scenes  # noqa: E402

capi.load()
tri, nrm = scenes.atrium()
for D in [int(a) for a in sys.argv[1:]] or [11, 12]:
    tree = capi.Octree.build(tri, nrm, D)
    nx, ny, spp = 3840, 2160, 4
    c, r, h = np.array([0.0, 0.4, 0.0]), 0.9, 0.6
    cams = []
    for k in range(16):
        a = 2 * np.pi * k / 64
        eye = c + np.array([r * np.cos(a), h, r * np.sin(a)])
        cams.append(capi.Camera(np.pi / 2, eye.astype(np.float32), c.astype(np.float32), (0, 1, 0), nx, ny, spp))
    out = torch.empty(nx * ny * spp * 16, dtype=torch.uint8, device='cuda')
    i = tree.info()
    line = [f"depth {D}: {i['num_nodes'] - i['num_leaves']} interior nodes, {i['num_tris']} tris"]
    for on in (True, False):
        tree.debug_set_eye_rel(on)
        for moving in (False, True):
            ms, kern = [], []
            for rep in range(2):
                for k in range(len(cams)):
                    cam = cams[k] if moving else cams[0]
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    tree.trace_camera_dev(cam, out.data_ptr(), compact=True)
                    e1.record()
                    torch.cuda.synchronize()
                    if rep:
                        ms.append(e0.elapsed_time(e1))
                        kern.append(tree.last_kernel_ms)
            line.append(f"eye_rel {'on ' if on else 'off'} {'new eye' if moving else 'same eye'}: call {np.mean(ms):.3f} ms "
                        f"kernel {np.mean(kern):.3f} ms (fill+queue {np.mean(ms) - np.mean(kern):.3f})")
    tree.debug_set_eye_rel(True)
    line.append(f"device_bytes {tree.info()['device_bytes']}")
    print("\n  ".join(line), flush=True)
    tree.close()
