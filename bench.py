#!/usr/bin/env python
"""bench.py -- headline benchmark of the octree hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): the "Sponza 1024^3 @4K" configuration of BASELINE.json
on the procedural atrium stand-in (sponza.obj is absent from the reference checkout,
SURVEY.md 0): 266,156 triangles voxelized at max_depth 11 (1024^3 leaf grid), main.cc's
final camera (main.cc:112-115), 3840x2160 film, gen_rays4 -> 33,177,600 primary rays
per step.  A step = one frame = one launch of the persistent ray kernel per GPU.

  value     Mrays/s with everything resident in HBM: per step every rank traces its 8-row
            bands and writes 16-byte hit records to HBM and the shaded pixels straight into
            rank 0's frame (peer stores over NVLink inside the ray kernel; --assemble gather:
            NCCL gather + re-order copy instead), all inside the timed region
  e2e       Mrays/s through the host-buffer C-ABI call (vrt_render_camera_async; N>1:
            vrt_render_bands_async on every rank): camera in, shaded film copied back to
            pinned host memory inside the timed region (N>1: one host frame shared by the ranks,
            every rank DMA-copies its own bands).  The film travels as main.cc writes it
            (stbi_write_hdr's RGBE pixels, encoded in the ray kernel); e2e_f32 is the same
            loop with the float film (12 B/pixel), which the host's PCIe ingest caps at 8 GPUs
  config5   BASELINE.json configs[4] in the same run: 2048^3, 7680x4320, orbit, primary +
            shadow rays (a few frames; the full line: --workload atrium2048_8k_orbit_shadow)
  parity    the bench's CPU sample (640x360x4 rays) and the leaf sets of the 1024^3 octrees,
            compared with the unmodified reference inside the run
  roofline  algorithmic bytes per ray (SURVEY.md 8d: 8*N_int + 8*N_leaf + 40*N_tri + 16,
            N_* counted on the same frame) * rays / kernel time, against the measured HBM
            copy bandwidth of MEASURED_PEAKS.json
  build     voxelization + octree build throughput (Mtris/s), device-timed and end to end
  cpu_baseline  the UNMODIFIED reference (oracle/_ref) on the host cores: ray_march_init
            (1 thread by construction) and render_mt (thread pool) on a bounded sample

--impl reference times the reference's own CPU implementation on the same workload
(bounded sample per step) and prints the same JSON shape with "impl": "reference".

--dump-outputs DIR writes what the last timed step computed, for comparing two builds output for
output: the film and the 16-byte hit records of a fixed, seeded sample of the frame's pixels
(DUMP_PIXELS of them, every sample ray of each), as DIR/<name>.npy in float32 / float64.
The orbit workloads move the camera every step (the last timed step shows camera (steps - 1) % 64),
so their dumps depend on --steps; the fixed-camera workloads dump the same frame for any --steps.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

RAD = np.pi / 180.0
WORKLOADS = {
    # name: (scene, scene kwargs, max_depth, cam10, nx, ny, spp)
    "atrium1024_4k_spp4": ("atrium", {}, 11, [90 * RAD, 1, 1.3, -.2, 0, .4, 0, 0, 1, 0], 3840, 2160, 4),
    "atrium1024_4k_spp1": ("atrium", {}, 11, [90 * RAD, 1, 1.3, -.2, 0, .4, 0, 0, 1, 0], 3840, 2160, 1),
    "sphere256_1080p_spp1": ("sphere", {}, 9, [60 * RAD, 0, 1, 3, 0, 0, 0, 0, 1, 0], 1920, 1080, 1),
    "atrium32_1k_spp4": ("atrium", {}, 6, [90 * RAD, 1, 1.3, -.2, 0, .4, 0, 0, 1, 0], 1024, 1024, 4),
    # BASELINE config 4 geometry traced: 2M-triangle random soup voxelized at 2048^3, 4K, camera outside the cloud
    "soup2m_2048_4k_spp4": ("soup", {}, 12, [60 * RAD, 0, 1, 3, 0, 0, 0, 0, 1, 0], 3840, 2160, 4),
    # BASELINE config 5: 2048^3, 8K, 64-frame camera orbit, primary + one shadow ray per hit
    "atrium2048_8k_orbit_shadow": ("atrium", {}, 12, [90 * RAD, 1, 1.3, -.2, 0, .4, 0, 0, 1, 0], 7680, 4320, 4),
}
# per-workload extras: camera orbit (eye(k) = c + (r cos 2 pi k/n, h, r sin 2 pi k/n) looking at c) and shadow rays
EXTRAS = {"atrium2048_8k_orbit_shadow": {"orbit": 64, "orbit_c": (0.0, 0.4, 0.0), "orbit_r": 0.9, "orbit_h": 0.6,
                                          "shadow_eps": 1e-3}}
DEFAULT_WORKLOAD = "atrium1024_4k_spp4"
CPU_SAMPLE = (640, 360)  # film used for the bounded CPU sample (same scene, camera, spp)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self, name):
        self.marks = getattr(self, "marks", {})
        self.marks[name] = time.perf_counter()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        marks = getattr(self, "marks", {})
        windows = [(marks[a], marks[b]) for a, b in (("t0", "t1"), ("e0_f32", "e1_f32"), ("e0_rgbe", "e1_rgbe")) if a in marks and b in marks]
        for ts, r in self.rows:
            if windows and not any(lo <= ts <= hi + 0.06 for lo, hi in windows):
                continue  # only samples taken while a timed region (value loop, e2e loop) was running
            c = [x.strip() for x in r.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[0]))
                mx.append(float(c[1]))
            except ValueError:
                continue
            for nm, v in zip(names, c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


OBJ_SCENE = {}  # filled by make_scene when the geometry comes from an OBJ file (--obj / Asset/sponza/sponza.obj)


def make_scene(wl, obj=None):
    """Geometry of the workload.  The "Sponza" workloads use the real asset when it is there (--obj PATH, or
    Asset/sponza/sponza.obj next to the repo / $VRT_SPONZA_OBJ: SURVEY.md 7 step 2) -- OBJ + MTL + TGA read on the
    host (voxelraytrace20190722_b200/assets.py), materials handed to vrt_set_materials -- else the procedural
    atrium stand-in."""
    from voxelraytrace20190722_b200 import assets, scenes
    scene, kw, depth, cam10, nx, ny, spp = WORKLOADS[wl]
    if obj is None and scene == "atrium":
        obj = assets.default_sponza_obj()
    if obj:
        sc = assets.load_scene(obj)
        tri, nrm = assets.expand_triangles(sc)
        if nrm is None:
            raise SystemExit(f"bench.py: {obj} has faces without normals (obj2voxel asserts them, voxel_octree.cc:346)")
        OBJ_SCENE.update(path=obj, scene=sc)
        return tri, nrm, depth, np.asarray(cam10, np.float32), nx, ny, spp
    tri, nrm = scenes.make_scene(scene, **kw)
    return tri, nrm, depth, np.asarray(cam10, np.float32), nx, ny, spp


# ----------------------------------------------------------------------------
# reference arm / cpu baseline (oracle/_ref = the unmodified reference)
# ----------------------------------------------------------------------------
GI_KD = [0.7, 0.6, 0.5]        # the single untextured material of the GI rows
GI_LIGHT_CAM = [60 * RAD, 1, 10, 1, 0, 0, 0, 0, 1, 0]  # main.cc:76-78
GI_LIGHT_FILM = (2048, 2048, 4)                          # main.cc:75 + gen_rays4
GI_CPU_SAMPLE = (160, 90)
GI_CPU_LIGHT = (256, 256)


def gi_res_of(root_aabb, depth):
    """main.cc:69-70: Res = min over axes of root.aabb.size() / powf(2, max_depth)."""
    r = np.asarray(root_aabb, np.float32)
    return float(np.float32(((r[3:] - r[:3]) / np.float32(2.0 ** depth)).min()))


def parity_vs_reference(scene, tree, wl, cam10, nx, ny, spp):
    """Parity of the CUDA path against the UNMODIFIED reference on the benched octree: every ray of the CPU sample
    film (the reference's own render_mt + gen_rays + gi::ray_march, hit records kept) against tree.trace_camera on
    the same camera -- hit flag, leaf cell, triangle, ISect.hit, ISect.normal, all bitwise -- and the leaf sets of
    the two octrees (cells, counts, triangle lists).  The oracle is the checker here, never the thing measured."""
    from voxelraytrace20190722_b200 import capi
    _, rays, o = scene.render_mt(cam10, 1.0, nx, ny, spp, outputs=True)
    cam = capi.Camera(cam10[0], cam10[1:4], cam10[4:7], cam10[7:10], nx, ny, spp)
    g = tree.trace_camera(cam)
    bad = (g["hit"] != o.hit) | (g["tri"] != o.tri) | (g["cell"] != o.cell).any(axis=1)
    bad |= (g["pos"].view(np.uint32) != o.pos.view(np.uint32)).any(axis=1)
    bad |= (g["nrm"].view(np.uint32) != o.nrm.view(np.uint32)).any(axis=1)
    ours, theirs = tree.leaves(), scene.leaves()
    leaf_ok = all(a.shape == b.shape and np.array_equal(a, b) for a, b in zip(ours, theirs))
    return {"config": wl, "against": "oracle/_ref (unmodified reference): render_mt + gi::ray_march, gi::ray_march_init",
            "film": f"{nx}x{ny}x{spp}", "rays": int(rays), "hits": int(o.hit.sum()), "mismatches": int(bad.sum()),
            "compared": "hit, leaf cell, triangle, ISect.hit, ISect.normal (bitwise)",
            "leaf_sets_bit_exact": bool(leaf_ok), "leaves": int(len(theirs[1])), "refs": int(len(theirs[2]))}


def cpu_reference(tri, nrm, depth, cam10, spp, steps, warmup, sample=CPU_SAMPLE, gi=False, parity_tree=None, wl=None):
    from oracle.bindings import Ref
    ref = Ref()
    scene = ref.scene(tri, nrm)
    build_s = scene.build(depth)
    nx, ny = sample
    times, rays = [], 0
    for i in range(warmup + steps):
        sec, rays, _ = scene.render_mt(cam10, 1.0, nx, ny, spp, outputs=False)
        if i >= warmup:
            times.append(sec)
    cores = ref.hardware_concurrency()
    parity = parity_vs_reference(scene, parity_tree, wl, cam10, nx, ny, spp) if parity_tree is not None else None
    gi_out = None
    if gi:
        # GI rows on the reference: splat (sequential, bounded light film), filter, then the final trace() loop on
        # a bounded film with all host threads (the tree is read-only there)
        lx, ly = GI_CPU_LIGHT
        t0 = time.perf_counter()
        scene.gi_reset()
        scene.gi_splat(GI_LIGHT_CAM, 1.0, lx, ly, 4, GI_KD)
        t1 = time.perf_counter()
        scene.gi_filter()
        t2 = time.perf_counter()
        gx, gy = GI_CPU_SAMPLE
        scene.gi_render(cam10, 1.0, gx, gy, spp, gi_res_of(scene.root_aabb(), depth), GI_KD, nthreads=cores)
        gi_out = {"splat_mrays_per_s": lx * ly * 4 / (t1 - t0) / 1e6, "splat_threads": 1,
                  "filter_s": t2 - t1, "render_mrays_per_s": gx * gy * spp / scene.seconds / 1e6,
                  "render_threads": cores,
                  "sample": f"light film {lx}x{ly}x4 (sequential, as the deterministic order requires), trace() film {gx}x{gy}x{spp}"}
    return dict(build_s=build_s, mtris=len(tri) / build_s / 1e6, ms_per_step=1e3 * float(np.mean(times)), gi=gi_out,
                parity=parity,
                mrays=rays / float(np.mean(times)) / 1e6, rays=rays, cores=cores,
                sample=f"same scene/camera/spp at {nx}x{ny} ({rays} rays per step) through render_mt + gen_rays{spp} + "
                       f"gi::ray_march on {min(cores, 64)} pool threads; octree built once by gi::ray_march_init "
                       f"(1 thread, {build_s:.1f} s, {len(tri) / build_s / 1e6:.4f} Mtris/s)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    tri, nrm, depth, cam10, nx, ny, spp = make_scene(args.workload, args.obj)
    r = cpu_reference(tri, nrm, depth, cam10, spp, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": "Mrays/s octree traversal", "value": r["mrays"], "unit": "Mrays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": dict(workload_config(args.workload, len(tri), args.gpus),
                       film=f"{CPU_SAMPLE[0]}x{CPU_SAMPLE[1]} sample of the {WORKLOADS[args.workload][4]}x"
                            f"{WORKLOADS[args.workload][5]} film (same scene, camera, spp; rate metric)",
                       rays_per_step=r["rays"],
                       sharding="host threads: render_mt's 64 tiles on the thread pool (no GPU)"),
        "cpu_baseline": {"value": r["mrays"], "unit": "Mrays/s", "cores": r["cores"], "kind": "reference",
                         "sample": r["sample"]},
        "e2e": {"value": r["mrays"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "build": {"mtris_per_s": r["mtris"], "seconds": r["build_s"], "threads": 1},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def workload_config(wl, ntris, gpus):
    scene, kw, depth, cam10, nx, ny, spp = WORKLOADS[wl]
    if OBJ_SCENE:
        sc = OBJ_SCENE["scene"]
        scene_desc = (f"obj {OBJ_SCENE['path']} ({ntris} tris, {len(sc['materials'])} materials, {len(sc['textures'])} textures"
                      + (f", missing textures {sc['missing_textures']}" if sc["missing_textures"] else "") + ")")
    else:
        scene_desc = f"{scene} ({ntris} tris" + ("; procedural Sponza stand-in, sponza.obj absent from the reference checkout)"
                                                 if scene == "atrium" else ")")
    return {"workload": wl,
            "scene": scene_desc,
            "max_depth": depth, "leaf_grid": f"{2 ** (depth - 1)}^3", "film": f"{nx}x{ny}", "spp": spp,
            "rays_per_step": nx * ny * spp,
            "camera": ("64-frame orbit (SURVEY 8d config 5), one frame per step; value counts primary rays, every hit "
                       "also traces one shadow ray in the same launch" if wl in EXTRAS else
                       "main.cc:112-115" if scene == "atrium" else "SURVEY 8d config 2"),
            "sharding": f"8-row bands round-robin over {gpus} GPU(s), replicated octree (one NCCL broadcast), frame assembled on rank 0",
            "l2": "inputs larger than L2: octree blob > 126 MB and every step writes 16 B/ray of hit records + 12 B/pixel of film"}


def make_cams(capi, wl, cam10, nx, ny, spp):
    """The workload's cameras: one fixed camera, or the frames of an orbit (EXTRAS)."""
    extra = EXTRAS.get(wl, {})
    if not extra.get("orbit"):
        return [capi.Camera(cam10[0], cam10[1:4], cam10[4:7], cam10[7:10], nx, ny, spp)]
    n_orb, c, r, h = extra["orbit"], np.asarray(extra["orbit_c"]), extra["orbit_r"], extra["orbit_h"]
    cams = []
    for k in range(n_orb):
        a = 2 * np.pi * k / n_orb
        eye = c + np.array([r * np.cos(a), h, r * np.sin(a)])
        cams.append(capi.Camera(cam10[0], eye.astype(np.float32), c.astype(np.float32), (0, 1, 0), nx, ny, spp))
    return cams


DUMP_PIXELS = 1 << 18  # pixels of the --dump-outputs sample: about 34 MB at 4 spp
DUMP_SEED = 20190722


def sample_outputs(torch, film, hit_rows, ny, nx, spp):
    """--dump-outputs: the film values and the hit records (vrt_hit16: leaf, tri, t, hit) of every sample ray of a
    fixed, seeded set of pixels.  film: [ny, nx, 3] float32 on the device; hit_rows: film-ordered [>= ny, nx*spp*4]
    int32 on the device.  Integer fields are widened to float64 (exact), so every array is float32 or float64."""
    n = min(DUMP_PIXELS, ny * nx)
    idx = np.sort(np.random.default_rng(DUMP_SEED).choice(ny * nx, n, replace=False))
    sel = torch.from_numpy(idx).to(film.device)
    px = film.reshape(ny * nx, 3).index_select(0, sel).cpu().numpy()
    rec = hit_rows[:ny].reshape(ny * nx, spp, 4).index_select(0, sel).cpu().numpy().view(np.uint32)
    return {"pixel_index": idx.astype(np.float64), "film": px.astype(np.float32),
            "hit_leaf": rec[..., 0].astype(np.float64), "hit_tri": rec[..., 1].astype(np.float64),
            "hit_t": rec[..., 2].view(np.float32).copy(), "hit_flag": rec[..., 3].astype(np.float64)}


def config5_block(args, capi, vdist, torch, world, rank, dev, tri, nrm):
    """BASELINE.json configs[4] inside the default run (every rank calls this): the same triangles voxelized at 2048^3,
    7680x4320 x 4 spp, camera orbit, primary rays + one shadow ray per hit, bands over all GPUs, frames assembled on
    rank 0 by the kernel's own stores.  A few frames only (the full line: --workload atrium2048_8k_orbit_shadow)."""
    wl = "atrium2048_8k_orbit_shadow"
    _, _, depth, cam10, nx, ny, spp = WORKLOADS[wl]
    shadow_eps = EXTRAS[wl]["shadow_eps"]
    if world > 1:
        import torch.distributed as td
    tree = capi.Octree.build(tri, nrm, depth) if rank == 0 else None
    if world > 1:
        tree = vdist.replicate_octree(tree, dev)
    cams = make_cams(capi, wl, cam10, nx, ny, spp)
    rows = vdist.max_band_rows(ny, world)
    hits = [torch.empty((rows, nx * spp * 4), dtype=torch.int32, device=dev) for _ in range(2)]
    pf = vdist.PeerFrame(ny, nx, dev)
    stream = torch.cuda.current_stream(dev)
    S = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]

    def step(i):
        with torch.cuda.stream(S[i & 1]):
            tree.set_stream(S[i & 1].cuda_stream)
            tree.frame_bands_dev(cams[i % len(cams)], hits[i & 1].data_ptr(), pf.ptr(i & 1), vdist.BAND_H, rank, world,
                                 full_frame=True, shadow_eps=shadow_eps)

    def sync_all():
        stream.wait_stream(S[0])
        stream.wait_stream(S[1])
        torch.cuda.synchronize(dev)
        if world > 1:
            td.barrier()
            torch.cuda.synchronize(dev)

    steps = max(2, min(args.steps, 8))
    for i in range(3):
        step(i)
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    S[0].wait_stream(stream)
    S[1].wait_stream(stream)
    for i in range(steps):
        step(i)
    stream.wait_stream(S[0])
    stream.wait_stream(S[1])
    e1.record(stream)
    sync_all()
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    if world > 1:
        td.all_reduce(t, op=td.ReduceOp.MAX)
    ms = float(t[0])
    # the frame assembled last (single-stream loop: step `steps - 1` again) against rank 0 alone
    tree.set_stream(stream.cuda_stream)
    tree.frame_bands_dev(cams[(steps - 1) % len(cams)], hits[0].data_ptr(), pf.ptr(0), vdist.BAND_H, rank, world,
                         full_frame=True, shadow_eps=shadow_eps)
    sync_all()
    ok = None
    if rank == 0:
        tree.set_stream(0)
        alone = torch.empty((ny, nx, 3), dtype=torch.float32, device=dev)
        tree.render_dev(cams[(steps - 1) % len(cams)], alone.data_ptr(), shadow_eps=shadow_eps)
        tree.sync()
        ok = bool(torch.equal(pf.frame(0).view(torch.int32), alone.view(torch.int32)))
        del alone
    info = tree.info()
    sync_all()
    if rank != 0:
        pf.close()  # (the peers unmap before rank 0 frees)
    sync_all()
    if rank == 0:
        pf.close()
    del hits
    tree.close()
    return {"workload": wl, "config": "BASELINE.json configs[4]: atrium at 2048^3, 7680x4320, gen_rays4, 64-frame orbit, "
                                      "primary + one shadow ray per hit (traced in the same launch)",
            "steps": steps, "ms_per_frame": ms, "primary_mrays_per_s": nx * ny * spp / (ms * 1e-3) / 1e6,
            "n_gpu_frame_equals_1_gpu_frame_bytewise": ok, "octree_nodes": info["num_nodes"],
            "octree_device_bytes": info["device_bytes"]}


# ----------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------
def run_ours(args):
    import torch
    from voxelraytrace20190722_b200 import capi, dist as vdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (libvrt has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as td
        td.init_process_group("nccl", device_id=dev)
    capi.load()
    sampler = ClockSampler(local)  # runs for the whole job; only samples inside the timed regions are kept
    if rank == 0:
        sampler.start()

    tri, nrm, depth, cam10, nx, ny, spp = make_scene(args.workload, args.obj)
    T = len(tri)
    rays_per_step = nx * ny * spp
    launches0 = capi.launch_count()

    # ---- build on rank 0 (end to end: host triangles -> octree in HBM), replicate ----
    build = {}
    tree = None
    if rank == 0:
        capi.Octree.build(tri[:1024], nrm[:1024], 4).close()  # CUDA context + module load, outside the timing
        # host triangles in -> octree resident in HBM, on a fresh handle.  The first full-size build of a
        # process also grows the stream-ordered memory pool from nothing (reported as e2e_first_s); e2e_s is
        # the same call on another fresh handle once the pool holds the scratch memory of a build, i.e. what
        # a long-running process pays per scene
        t0 = time.perf_counter()
        capi.Octree.build(tri, nrm, depth).close()
        build["e2e_first_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        tree = capi.Octree.build(tri, nrm, depth)
        build["e2e_s"] = time.perf_counter() - t0
        ms = []
        for _ in range(args.build_reps + 1):
            tree.rebuild(depth)
            ms.append(tree.info()["build_ms"])
        build["ms"] = float(np.mean(ms[1:])) if len(ms) > 1 else ms[0]
    if world > 1:
        tree = vdist.replicate_octree(tree, dev)
    if OBJ_SCENE and rank == 0 and world == 1:
        sc = OBJ_SCENE["scene"]  # Triangle::get_albedo data for the GI rows (voxel_octree.cc:471-484)
        tree.set_materials(sc["tri_uv"], sc["tri_mtl"], sc["kd"], sc["mtl_tex"], sc["textures"])
    info = tree.info()
    extra = EXTRAS.get(args.workload, {})
    shadow_eps = extra.get("shadow_eps")
    cams = make_cams(capi, args.workload, cam10, nx, ny, spp)
    cam = cams[0]
    stream = torch.cuda.current_stream(dev)
    tree.set_stream(stream.cuda_stream)

    # One step = one frame: this rank's 8-row bands through the ray kernel, which writes the
    # compact per-ray hit records (kept sharded in HBM) AND the shaded pixels.  Framebuffer
    # assembly on rank 0 is fused into the kernel (default, --assemble peer): the pixels are
    # stored straight into rank 0's double-buffered frame over NVLink (CUDA-IPC mapped), so
    # there is no collective and no re-order pass.  --assemble gather uses the NCCL gather
    # (double-buffered, asynchronous) + one re-order copy instead.
    rows = vdist.max_band_rows(ny, world)  # padded to the largest shard so the gather is uniform
    hits = [torch.empty((rows, nx * spp * 4), dtype=torch.int32, device=dev) for _ in range(2)]
    use_gather = (args.assemble == "gather") and world > 1
    fg = vdist.FrameGather(ny, nx, 3, torch.float32, dev) if use_gather else None
    pf = None if use_gather else vdist.PeerFrame(ny, nx, dev)
    # two streams, alternating per frame: the head of frame k+1 fills the SMs that the tail of
    # frame k (a few long rays) leaves idle.  (Not with NCCL in the loop: its kernels cannot
    # become resident while two persistent grids own every SM.)
    S = [torch.cuda.Stream(dev)]
    S.append(S[0] if use_gather else torch.cuda.Stream(dev))

    def step(i):
        k = i & 1
        with torch.cuda.stream(S[k]):
            tree.set_stream(S[k].cuda_stream)
            if use_gather:
                film = fg.buffer(k)
                tree.frame_bands_dev(cams[i % len(cams)], hits[k].data_ptr(), film.data_ptr(), vdist.BAND_H, rank, world,
                                     shadow_eps=shadow_eps)
                if i > 0:
                    fg.assemble(k ^ 1)  # frame i-1 (its gather ran under this frame's kernel)
                fg.gather_async(k)
            else:
                tree.frame_bands_dev(cams[i % len(cams)], hits[k].data_ptr(), pf.ptr(k), vdist.BAND_H, rank, world,
                                     full_frame=True, shadow_eps=shadow_eps)

    def drain(i_last):
        if use_gather:
            with torch.cuda.stream(S[0]):
                fg.assemble(i_last & 1)
                fg.finish()
        stream.wait_stream(S[0])
        stream.wait_stream(S[1])

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            td.barrier()
            torch.cuda.synchronize(dev)

    for i in range(args.warmup):
        step(i)
    drain(args.warmup - 1)
    sync_all()
    sampler.mark("t0")
    l0 = capi.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    S[0].wait_stream(stream)
    S[1].wait_stream(stream)
    for i in range(args.steps):
        step(i)
    drain(args.steps - 1)
    e1.record(stream)
    sync_all()
    sampler.mark("t1")
    launches = capi.launch_count() - l0
    total_ms = e0.elapsed_time(e1)
    t = torch.tensor([total_ms, tree.mean_kernel_ms(min(args.steps, 64))], dtype=torch.float64, device=dev)
    if world > 1:
        if os.environ.get("VRT_BENCH_DEBUG"):
            allt = [torch.zeros_like(t) for _ in range(world)]
            td.all_gather(allt, t)
            if rank == 0:
                sys.stderr.write("per-rank [total_ms, kernel_ms]: " + str([[round(float(v), 3) for v in a] for a in allt]) + "\n")
        td.all_reduce(t, op=td.ReduceOp.MAX)
    total_ms, kern_ms_events = float(t[0]), float(t[1])
    ms_per_step = total_ms / args.steps
    # launches of consecutive frames overlap (two streams), so a launch's own event pair also
    # spans the time it waits behind its predecessor; the average launch duration over the
    # timed region is the CUDA-event time of the region / launches
    kern_ms = ms_per_step
    value = rays_per_step / (ms_per_step * 1e-3) / 1e6

    # ---- --dump-outputs: the last timed step's frame and hit records, before anything below overwrites them ----
    if args.dump_outputs:
        k_last = (args.steps - 1) & 1
        hit_rows = hits[k_last] if world == 1 else vdist.gather_rows(hits[k_last], ny)  # collective
        if rank == 0:
            film = fg.frame if use_gather else pf.frame(k_last)
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in sample_outputs(torch, film, hit_rows, ny, nx, spp).items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
        del hit_rows

    # ---- the dominant kernel alone: one stream, CUDA events around every launch (no overlap with a neighbour) ----
    tree.set_stream(stream.cuda_stream)
    with torch.cuda.stream(stream):
        for i in range(args.steps):
            tree.frame_bands_dev(cams[i % len(cams)], hits[0].data_ptr(), (fg.buffer(0).data_ptr() if use_gather else pf.ptr(0)),
                                 vdist.BAND_H, rank, world, full_frame=not use_gather, shadow_eps=shadow_eps)
    tk = torch.tensor([tree.mean_kernel_ms(min(args.steps, 64))], dtype=torch.float64, device=dev)
    sync_all()
    if world > 1:
        td.all_reduce(tk, op=td.ReduceOp.MAX)
    kern_ms_isolated = float(tk[0])

    # ---- e2e: host-buffer C-ABI call, film copied back to pinned host memory every step ----
    # Measured for two film formats (include/vrt.h vrt_set_film_format): "rgbe" -- the film as main.cc:125-126
    # delivers it (stbi_write_hdr's pixel encoding, 4 B/pixel, encoded in the ray kernel's pixel store) -- is the
    # headline `e2e`; "f32" (Film::to_float_array, 12 B/pixel; round 1's e2e) is reported beside it as `e2e_f32`.
    # The float film saturates this box's device->host ingest at 8 GPUs (DESIGN.md 6), the encoded one does not.
    def measure_e2e(fmt):
        note, host_ok, sync_ms = None, None, None
        bpp = capi.film_pixel_bytes(fmt)
        tree.set_film_format(fmt)
        try:
            if world == 1:
                # frame loop through the host-buffer C ABI: vrt_render_camera_async enqueues the frame and its
                # device->host copy (pinned film, alternating between two host buffers); the copy of frame k
                # overlaps the kernel of frame k+1; every frame's film is in host memory when the timed region
                # ends (vrt_tree_sync)
                film_hosts = [torch.empty((ny, nx, 3), dtype=torch.float32).pin_memory() if fmt == "f32" else
                              torch.empty((ny, nx, bpp), dtype=torch.uint8).pin_memory() for _ in range(2)]
                film_nps = [f.numpy() for f in film_hosts]
                tree.set_stream(0)
                for i in range(max(2, args.warmup // 2)):
                    tree.render_async(cams[i % len(cams)], film_nps[i & 1], shadow_eps=shadow_eps)
                tree.sync()
                sampler.mark("e0_" + fmt)
                t0 = time.perf_counter()
                for i in range(args.steps):
                    tree.render_async(cams[i % len(cams)], film_nps[i & 1], shadow_eps=shadow_eps)
                tree.sync()
                ms = (time.perf_counter() - t0) * 1e3 / args.steps
                sampler.mark("e1_" + fmt)
                # the last frame of the loop against the synchronous single-frame call (also timed, for reference)
                k_last = args.steps - 1
                t0 = time.perf_counter()
                for _ in range(min(args.steps, 5)):
                    alone = tree.render(cams[k_last % len(cams)], shadow_eps=shadow_eps)
                sync_ms = (time.perf_counter() - t0) * 1e3 / min(args.steps, 5)
                host_ok = bool(np.array_equal(film_nps[k_last & 1].view(np.uint8), alone.view(np.uint8)))
                return ms, ny * nx * bpp, host_ok, note, sync_ms
            # N ranks: the same frame loop through vrt_render_bands_async -- every rank renders its bands and
            # DMA-copies them to their final rows of a host frame that all ranks of the node map (POSIX shared
            # memory, pinned in every process): N PCIe links in parallel, the copy of frame k overlapping the
            # kernel of frame k+1; every frame is complete in host memory when the timed region ends
            # (vrt_tree_sync on every rank + barrier)
            try:
                shf = vdist.SharedHostFrame(ny, nx, nbuf=2, fmt=fmt)
            except RuntimeError as ex:  # raised on every rank or on none
                shf = None
                note = f"no shared pinned host frame ({ex}): per-frame barrier + copy from rank 0's GPU (float film)"
            if shf is not None:
                tree.set_stream(0)

                def e2e_step(i):
                    tree.render_bands_async(cams[i % len(cams)], shf.ptr(i), vdist.BAND_H, rank, world,
                                            shadow_eps=shadow_eps)

                def e2e_drain():
                    tree.sync()
            else:
                tree.set_film_format("f32")
                bpp = 12
                film_host = torch.empty((ny, nx, 3), dtype=torch.float32).pin_memory() if rank == 0 else None
                tree.set_stream(stream.cuda_stream)

                def e2e_step(i):
                    if use_gather:
                        tree.render_bands_dev(cams[i % len(cams)], fg.buffer(0).data_ptr(), vdist.BAND_H, rank, world,
                                              shadow_eps=shadow_eps)
                        fg.gather_async(0)
                        full = fg.assemble(0)
                    else:
                        tree.frame_bands_dev(cams[i % len(cams)], hits[0].data_ptr(), pf.ptr(0), vdist.BAND_H, rank, world,
                                             full_frame=True, shadow_eps=shadow_eps)
                        torch.cuda.synchronize(dev)
                        td.barrier()  # every rank's pixels have landed in rank 0's frame
                        full = pf.frame(0)
                    if rank == 0:
                        film_host.copy_(full, non_blocking=True)
                    torch.cuda.synchronize(dev)

                def e2e_drain():
                    pass
            for i in range(max(2, args.warmup // 2)):
                e2e_step(i)
            e2e_drain()
            sync_all()
            sampler.mark("e0_" + fmt)
            t0 = time.perf_counter()
            for i in range(args.steps):
                e2e_step(i)
            e2e_drain()
            sync_all()
            sampler.mark("e1_" + fmt)
            tt = torch.tensor([(time.perf_counter() - t0) * 1e3 / args.steps], dtype=torch.float64, device=dev)
            td.all_reduce(tt, op=td.ReduceOp.MAX)
            ms = float(tt[0])
            # the last host frame of the loop against the same camera rendered by rank 0 alone
            if rank == 0:
                k_last = args.steps - 1
                alone = tree.render(cams[k_last % len(cams)], shadow_eps=shadow_eps)
                got_host = shf.frame(k_last) if shf is not None else film_host.numpy()
                host_ok = bool(np.array_equal(got_host.view(np.uint8), alone.view(np.uint8)))
            if shf is not None:
                sync_all()
                shf.close()
            return ms, ny * nx * bpp, host_ok, note, sync_ms
        finally:
            tree.set_film_format("f32")
            tree.set_stream(stream.cuda_stream)

    f32_ms, f32_d2h, f32_ok, f32_note, f32_sync_ms = measure_e2e("f32")
    e2e_ms, d2h, e2e_host_frame_ok, e2e_note, e2e_sync_ms = measure_e2e("rgbe")
    e2e_f32 = {"value": rays_per_step / (f32_ms * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": f32_ms,
               "d2h_bytes_per_step": int(f32_d2h), "film": "f32 (Film::to_float_array, 12 B/pixel): round 1's e2e",
               "host_frame_equals_1_gpu_render_bytewise": f32_ok, "sync_single_frame_ms": f32_sync_ms, "note": f32_note}
    e2e_value = rays_per_step / (e2e_ms * 1e-3) / 1e6
    clocks = sampler.stop() if rank == 0 else None

    # ---- N-GPU frame == 1-GPU frame, bytewise (outside every timed region) ----
    frame_check = None
    if rank == 0:
        tree.set_stream(0)
        ref_film = torch.empty((ny, nx, 3), dtype=torch.float32, device=dev)
        # the frame that was assembled last (timed loop with the gather, the single-stream loop with peer stores)
        # shows the camera of step `steps - 1` (orbit workloads move the camera every step)
        tree.render_dev(cams[(args.steps - 1) % len(cams)], ref_film.data_ptr(), shadow_eps=shadow_eps)
        tree.sync()
        got = fg.frame if use_gather else pf.frame(0)
        frame_check = bool(torch.equal(got.view(torch.int32), ref_film.view(torch.int32)))
        del ref_film

    # ---- BASELINE config 5 in the same run (default workload only; all ranks) ----
    cfg5 = None
    if args.workload == DEFAULT_WORKLOAD and not args.no_config5 and not OBJ_SCENE:
        try:
            cfg5 = config5_block(args, capi, vdist, torch, world, rank, dev, tri, nrm)
        except Exception as ex:  # noqa: BLE001 -- reported in the line, the headline numbers stand
            cfg5 = {"workload": "atrium2048_8k_orbit_shadow", "error": repr(ex)}

    if rank != 0:
        if world > 1:
            td.destroy_process_group()
        return 0

    # ---- roofline: algorithmic bytes of the reference algorithm on this very frame ----
    tree.set_stream(0)
    cnt = tree.count_camera(cam)
    n_int, n_leaf, n_tri = (cnt[k] / cnt["rays"] for k in ("n_int", "n_leaf", "n_tri"))
    b_ray = 8 * n_int + 8 * n_leaf + 40 * n_tri + 16
    peaks, peak_src = measured_peaks()
    rays_per_launch = rays_per_step / world
    achieved = b_ray * rays_per_launch / (kern_ms * 1e-3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(tp):
        try:
            with open(tp) as f:
                traffic = json.load(f).get(args.workload, {}).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "peak_source": peak_src,
                "kernel": "k_trace_camera<HIT16_FILM>", "kernel_ms": kern_ms,
                "kernel_ms_isolated": kern_ms_isolated,
                "frac_isolated": b_ray * rays_per_launch / (kern_ms_isolated * 1e-3) / 1e9 / peaks["hbm_gbs"],
                "timing": ("kernel_ms = CUDA-event time of the timed region / launches (consecutive frames alternate between "
                           "two streams, so the tail of one launch overlaps the head of the next); kernel_ms_isolated = mean "
                           "of per-launch CUDA-event pairs of the same launches issued on ONE stream after the timed region "
                           "(comparable with the ncu launch list under profiles/)"),
                "bytes_per_ray": b_ray,
                "n_int": n_int, "n_leaf": n_leaf, "n_tri": n_tri, "hit_fraction": cnt["hits"] / cnt["rays"]}

    # ---- build metric ----
    b_tri = None
    rho = info["num_refs"] / max(T, 1)
    nu = info["num_nodes"] / max(T, 1)
    b_tri = 36 + 12 * rho + 8 * nu
    build_out = {"mtris_per_s": T / (build["ms"] * 1e-3) / 1e6, "ms": build["ms"],
                 "e2e_mtris_per_s": T / build["e2e_s"] / 1e6, "e2e_s": build["e2e_s"],
                 "e2e_first_s": build["e2e_first_s"],
                 "h2d_bytes": int(tri.nbytes + nrm.nbytes), "bytes_per_tri": b_tri,
                 "roofline_frac": b_tri * T / (build["ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"],
                 "leaves": info["num_leaves"], "nodes": info["num_nodes"], "refs": info["num_refs"]}

    # ---- BASELINE config 4: the 2 M-triangle soup voxelized at 2048^3 (build throughput), rank 0, N=1 ----
    build_soup = None
    if world == 1 and not args.no_build_soup and args.workload != "soup2m_2048_4k_spp4":
        from voxelraytrace20190722_b200 import scenes as _sc
        stri, snrm = _sc.make_scene("soup")
        t0 = time.perf_counter()
        stree = capi.Octree.build(stri, snrm, 12)
        s_e2e = time.perf_counter() - t0
        sms = []
        for _ in range(args.build_reps + 1):
            stree.rebuild(12)
            sms.append(stree.info()["build_ms"])
        sinfo = stree.info()
        s_ms = float(np.mean(sms[1:])) if len(sms) > 1 else sms[0]
        s_btri = 36 + 12 * sinfo["num_refs"] / len(stri) + 8 * sinfo["num_nodes"] / len(stri)
        build_soup = {"workload": "soup 2,000,000 tris (PCG seed 12345) at max_depth 12 (2048^3)",
                      "mtris_per_s": len(stri) / (s_ms * 1e-3) / 1e6, "ms": s_ms, "e2e_s": s_e2e,
                      "e2e_mtris_per_s": len(stri) / s_e2e / 1e6, "bytes_per_tri": s_btri,
                      "roofline_frac": s_btri * len(stri) / (s_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                      "leaves": sinfo["num_leaves"], "nodes": sinfo["num_nodes"], "refs": sinfo["num_refs"]}
        stree.close()
        del stri, snrm

    # ---- GI rows (SURVEY.md 8f "next"): splat / filter / trace() film, device-timed (rank 0, N=1) ----
    gi_out = None
    if world == 1 and not args.no_gi:
        tree.set_stream(0)
        lx, ly, lspp = GI_LIGHT_FILM
        lcam = capi.Camera(GI_LIGHT_CAM[0], GI_LIGHT_CAM[1:4], GI_LIGHT_CAM[4:7], GI_LIGHT_CAM[7:10], lx, ly, lspp)
        res = gi_res_of(info["root_aabb"], depth)
        gfilm = torch.empty((ny, nx, 3), dtype=torch.float32, device=dev)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        tree.gi_init()
        tree.gi_splat(lcam, GI_KD)      # warm-up (allocations)
        tree.gi_render_dev(cam, GI_KD, res, gfilm.data_ptr())
        tree.gi_init()
        tree.sync()
        ev[0].record()
        tree.gi_splat(lcam, GI_KD)
        ev[1].record()
        tree.gi_filter()
        ev[2].record()
        tree.gi_render_dev(cam, GI_KD, res, gfilm.data_ptr())
        ev[3].record()
        tree.gi_render_dev(cam, GI_KD, res, gfilm.data_ptr())
        ev[4].record()
        tree.sync()
        torch.cuda.synchronize(dev)
        splat_ms, filter_ms = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
        render_ms = min(ev[2].elapsed_time(ev[3]), ev[3].elapsed_time(ev[4]))
        # roofline entry of the GI film kernel: algorithmic bytes of the reference's cone trace (voxel_octree.cc:247-283)
        # per ray = the primary traversal's bytes + 8 B per descent step of every sample's point location (the
        # reference walks down from the root at every step) + 80 B per sample that reaches its level (coverage +
        # illum[6]), counted by the instrumented oracle on a bounded film of the same scene / camera
        gi_roof = None
        if not args.no_cpu_baseline:
            try:
                from oracle.bindings import Port
                t0 = time.perf_counter()
                ptree = Port().build(tri, nrm, depth)
                ptree.gi_reset()
                ptree.gi_filter()
                gx, gy = GI_CPU_SAMPLE
                _, cc = ptree.gi_render_counted(cam10, 1.0, gx, gy, spp, res, GI_KD)
                n_gi = gx * gy * spp
                b_gi = b_ray + (8 * cc["descent_steps"] + 80 * cc["located"]) / n_gi
                ach = b_gi * rays_per_step / (render_ms * 1e-3) / 1e9
                gi_roof = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                           "frac": ach / peaks["hbm_gbs"], "bytes_per_ray": b_gi,
                           "samples_per_ray": cc["samples"] / n_gi, "descent_steps_per_ray": cc["descent_steps"] / n_gi,
                           "located_per_ray": cc["located"] / n_gi,
                           "counted_on": f"{gx}x{gy}x{spp} film, oracle port (coverage from the filter; the counts do not "
                                         f"depend on the light map), {time.perf_counter() - t0:.1f} s",
                           "kernel": "k_trace_camera<GI_FILM>"}
                del ptree
            except Exception as e:  # the roofline entry is a report, never a reason to fail the bench
                gi_roof = {"error": str(e)}
        gi_out = {"roofline": gi_roof,
                  "splat_ms": splat_ms, "splat_mrays_per_s": lx * ly * lspp / (splat_ms * 1e-3) / 1e6,
                  "light_film": f"{lx}x{ly}x{lspp} (main.cc:75-78)", "filter_ms": filter_ms,
                  "render_ms": render_ms, "render_mrays_per_s": rays_per_step / (render_ms * 1e-3) / 1e6,
                  "render": "trace() of main.cc:10-30 per sample: ray march + 6 cones + direct + albedo, same film as the headline",
                  "res": res, "film_mean": [float(v) for v in gfilm.mean(dim=(0, 1)).cpu()]}
        del gfilm

    # ---- cpu baseline (rank 0, N=1 only) ----
    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            tree.set_stream(0)
            r = cpu_reference(tri, nrm, depth, cam10, spp, steps=1, warmup=0, gi=not args.no_gi, parity_tree=tree,
                              wl=args.workload)
            parity = r["parity"]
            cpu = {"value": r["mrays"], "unit": "Mrays/s", "cores": r["cores"], "kind": "reference",
                   "sample": r["sample"], "build_mtris_per_s": r["mtris"], "build_seconds": r["build_s"],
                   "gi": r["gi"]}
        except Exception as e:  # oracle/_ref missing on this box
            cpu = {"value": None, "unit": "Mrays/s", "cores": None, "kind": "reference",
                   "sample": f"unavailable: {e}"}

    line = {
        "metric": "Mrays/s octree traversal", "value": value, "unit": "Mrays/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": workload_config(args.workload, T, world),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": 92, "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_ms,
                "film": "rgbe: the film as main.cc:125-126 delivers it (stbi_write_hdr's pixel encoding, stb_image_write.h:"
                        "601-616, 4 B/pixel), encoded in the ray kernel's pixel store (vrt_set_film_format); bytewise equal to "
                        "the reference encoder on the float film (tests/test_gpu_film_export.py)",
                "call": ("vrt_render_camera_async per frame + vrt_tree_sync (camera struct in, shaded film out to pinned "
                         "host; frame k's copy overlaps frame k+1's kernel)" if world == 1 else
                         "vrt_render_bands_async per rank and frame + vrt_tree_sync + barrier (camera struct in; every rank "
                         "DMA-copies its bands to their final rows of one host frame shared and pinned by all ranks; "
                         "frame k's copy overlaps frame k+1's kernel)"),
                "sync_single_frame_ms": e2e_sync_ms if world == 1 else None, "note": e2e_note},
        "e2e_f32": e2e_f32,
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": cpu,
        "parity": parity,
        "build": build_out,
        "build_soup": build_soup,
        "config5": cfg5,
        "gi": gi_out,
        "octree": {"device_bytes": info["device_bytes"], "nodes": info["num_nodes"], "leaves": info["num_leaves"]},
        "frame_check": {"n_gpu_frame_equals_1_gpu_frame_bytewise": frame_check,
                        "e2e_host_frame_equals_1_gpu_render_bytewise": e2e_host_frame_ok},
        "assemble": ("nccl gather + re-order copy" if use_gather else
                     "fused: peer stores into rank 0's IPC-mapped frame over NVLink" if world > 1 else "local frame"),
    }
    print(json.dumps(line))
    if world > 1:
        td.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--build-reps", type=int, default=3)
    ap.add_argument("--obj", default=None,
                    help="Wavefront OBJ (+ MTL + TGA) to use as the scene instead of the procedural stand-in; default: "
                         "Asset/sponza/sponza.obj next to the repo or $VRT_SPONZA_OBJ when present")
    ap.add_argument("--assemble", default="peer", choices=["peer", "gather"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gi", action="store_true", help="skip the GI rows (splat/filter/cone-trace film)")
    ap.add_argument("--no-build-soup", action="store_true", help="skip the 2 M-triangle soup build (BASELINE config 4)")
    ap.add_argument("--no-config5", action="store_true", help="skip the BASELINE config 5 block (2048^3, 8K orbit + shadow rays)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the film and hit records of a seeded sample of the last step's "
                         "pixels to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
