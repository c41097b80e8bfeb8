"""GPU: the C++ host mirror (cpp/vrt_gi.*) -- the reference's own signatures on top of the
C ABI -- driven by the main.cc-like demo, checked against the oracle."""
import os
import subprocess

import numpy as np
import pytest

from tests.common import CAM_LIGHT, GI_KD, assert_bits_equal, compare_hits, gi_res
from voxelraytrace20190722_b200 import capi, scenes

pytestmark = pytest.mark.gpu
CPP = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "voxelraytrace20190722_b200", "cpp")


def _write_obj(path, tri, nrm):
    with open(path, "w") as f:
        for t, n in zip(tri, nrm):
            for v in t:
                f.write("v %.9g %.9g %.9g\n" % tuple(v))
            for v in n:
                f.write("vn %.9g %.9g %.9g\n" % tuple(v))
        for i in range(len(tri)):
            a = 3 * i + 1
            f.write(f"f {a}//{a} {a + 1}//{a + 1} {a + 2}//{a + 2}\n")


def test_demo_main_matches_oracle(tmp_path, port, gpu):
    subprocess.check_call(["make", "-s", "-C", CPP])
    tri, nrm = scenes.uv_sphere(64, 32)
    obj = tmp_path / "sphere.obj"
    _write_obj(obj, tri, nrm)
    nx, ny, depth, spp = 96, 64, 6, 4
    dump = tmp_path / "hits.bin"
    gi_dump = tmp_path / "gi_film.bin"
    out = subprocess.run([os.path.join(CPP, "demo_main"), str(tmp_path / "o.bmp"), str(depth), str(nx), str(ny),
                          str(obj), "--dump", str(dump), "--gi", str(gi_dump)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "success." in out.stdout and f"#tris={len(tri)}" in out.stdout
    hits = np.fromfile(dump, capi.HIT_DTYPE)
    assert len(hits) == nx * ny * spp
    fov = np.float32(60.0) * np.float32(3.1415926535897932384626) / np.float32(180.0)  # jql::to_radian
    cam10 = np.array([fov, 0, 1, 3, 0, 0, 0, 0, 1, 0], np.float32)
    orc = port.build(tri, nrm, depth)
    exp = orc.trace(port.gen_rays(cam10, 1.0, nx, ny, spp))
    assert exp.hit.sum() > 100
    assert compare_hits(hits, exp, "demo_main") == 0
    assert os.path.getsize(tmp_path / "o.bmp") == 54 + nx * ny * 3
    # the GI half of main.cc through the mirror (light_map_gpu, gi::cone_trace_init_filter, render_gi_gpu)
    film = np.fromfile(gi_dump, np.float32).reshape(ny, nx, 3)
    orc.gi_reset()
    orc.gi_splat(np.concatenate([[fov], CAM_LIGHT[1:]]).astype(np.float32), 1.0, nx, ny, 4, GI_KD)
    orc.gi_filter()
    with port.exact_log2():
        exp_film = orc.gi_render(cam10, 1.0, nx, ny, spp, gi_res(orc.root_aabb(), depth), GI_KD)
    assert_bits_equal(film, exp_film, "demo_main GI film")
    assert "centre ray indirect light" in out.stdout
    with open(str(gi_dump) + ".hdr", "rb") as f:  # the stbi_write_hdr step of main.cc:125-126
        hdr = f.read()
    assert hdr.startswith(b"#?RADIANCE") and hdr.endswith(hdr[-4 * nx * ny:]) and len(hdr) > 4 * nx * ny
