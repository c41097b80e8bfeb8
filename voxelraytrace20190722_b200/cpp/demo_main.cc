// demo_main.cc -- the hot-path half of the reference's main.cc (main.cc:32-129) written
// against the mirror API: triangles -> gi::ray_march_init -> per-pixel gen_rays4 +
// gi::ray_march, rendered by ONE GPU launch instead of render_mt + thread pool, image
// written as BMP.  Geometry: a procedural UV sphere (sponza.obj is not in the reference
// checkout), or "v/vn/f" triangles from an OBJ given on the command line.
//   demo_main [out.bmp] [max_depth] [nx] [ny] [scene.obj]
// With --dump <file> it also writes (hit,tri,cell,pos,nrm) per ray for the parity test.
// With --gi <file> it also writes main.cc's cone-traced GI film (float, plus <file>.hdr); with --gi-devices 0,0,...
// as well, the same film rendered through gi::MultiGpu on those devices goes to <file>.mgpu; with --gi-aov <prefix> as
// well, what that film is made of goes to <prefix>.{albedo,direct,indirect,normal}.hdr (and, with --gi-devices, the
// same planes rendered through the replicas to <prefix>.mgpu.{albedo,direct,indirect,normal}.hdr).
// With --animate <prefix> it renders four GI frames, the scene turned by one more quarter turn about the vertical
// axis through the centre of its root box before each (gi::transform_gpu, then the light map and filter again), and
// writes frame k to <prefix>.<k>.hdr.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>

#include "vrt_gi.h"

using jql::Vec3;

static std::vector<gi::Triangle> make_sphere(int nu, int nv)
{
        std::vector<gi::Triangle> tris;
        auto vert = [&](int i, int j) {
                const double th = M_PI * j / nv, ph = 2.0 * M_PI * (i % nu) / nu;
                const double st = (j == 0 || j == nv) ? 0.0 : std::sin(th);
                return Vec3{ (float)(st * std::cos(ph)), (float)std::cos(th), (float)(st * std::sin(ph)) };
        };
        for (int i = 0; i < nu; ++i)
                for (int j = 0; j < nv; ++j) {
                        Vec3 a = vert(i, j), b = vert(i + 1, j), c = vert(i + 1, j + 1), d = vert(i, j + 1);
                        if (j != 0) tris.emplace_back(a, b, c, a, b, c);
                        if (j != nv - 1) tris.emplace_back(a, c, d, a, c, d);
                }
        return tris;
}

static std::vector<gi::Triangle> load_obj(const char* path)
{
        std::ifstream f(path);
        if (!f) { std::fprintf(stderr, "cannot open %s\n", path); std::exit(1); }
        std::vector<Vec3> v, vn;
        std::vector<gi::Triangle> tris;
        std::string line;
        while (std::getline(f, line)) {
                std::istringstream s(line);
                std::string tag;
                s >> tag;
                if (tag == "v") { Vec3 p; s >> p.x >> p.y >> p.z; v.push_back(p); }
                else if (tag == "vn") { Vec3 p; s >> p.x >> p.y >> p.z; vn.push_back(p); }
                else if (tag == "f") {
                        std::vector<std::pair<int, int>> idx;
                        std::string tok;
                        while (s >> tok) {
                                int vi = 0, ti = 0, ni = 0;
                                if (std::sscanf(tok.c_str(), "%d/%d/%d", &vi, &ti, &ni) != 3 &&
                                    std::sscanf(tok.c_str(), "%d//%d", &vi, &ni) != 2)
                                        std::sscanf(tok.c_str(), "%d", &vi);
                                idx.push_back({ vi < 0 ? (int)v.size() + vi : vi - 1, ni < 0 ? (int)vn.size() + ni : ni - 1 });
                        }
                        for (size_t k = 1; k + 1 < idx.size(); ++k) {  // fan triangulation
                                Vec3 p0 = v[idx[0].first], p1 = v[idx[k].first], p2 = v[idx[k + 1].first];
                                Vec3 g{ (p1.y - p0.y) * (p2.z - p0.z) - (p2.y - p0.y) * (p1.z - p0.z),
                                        (p1.z - p0.z) * (p2.x - p0.x) - (p2.z - p0.z) * (p1.x - p0.x),
                                        (p1.x - p0.x) * (p2.y - p0.y) - (p2.x - p0.x) * (p1.y - p0.y) };
                                auto nrm = [&](int ni) { return (ni >= 0 && ni < (int)vn.size()) ? vn[ni] : g; };
                                tris.emplace_back(p0, p1, p2, nrm(idx[0].second), nrm(idx[k].second), nrm(idx[k + 1].second));
                        }
                }
        }
        return tris;
}

static void write_bmp(const char* path, const Film& film)
{
        const auto rgb = film.to_byte_array();
        const int w = film.nx, h = film.ny, row = (3 * w + 3) & ~3;
        std::vector<unsigned char> img((size_t)row * h, 0);
        for (int y = 0; y < h; ++y)
                for (int x = 0; x < w; ++x)
                        for (int c = 0; c < 3; ++c)
                                img[(size_t)(h - 1 - y) * row + 3 * x + (2 - c)] = rgb[((size_t)y * w + x) * 3 + c];
        unsigned char hdr[54] = { 'B', 'M' };
        auto put = [&](int off, uint32_t v) { std::memcpy(hdr + off, &v, 4); };
        put(2, 54 + (uint32_t)img.size()); put(10, 54); put(14, 40); put(18, (uint32_t)w); put(22, (uint32_t)h);
        hdr[26] = 1; hdr[28] = 24; put(34, (uint32_t)img.size());
        FILE* f = std::fopen(path, "wb");
        if (!f) return;
        std::fwrite(hdr, 1, 54, f);
        std::fwrite(img.data(), 1, img.size(), f);
        std::fclose(f);
}

// Radiance .hdr (RGBE, no run-length encoding) of the float film -- the host-side job stbi_write_hdr does in
// main.cc:125-126.
static void write_hdr(const char* path, const Film& film)
{
        const auto d = film.to_float_array();
        FILE* f = std::fopen(path, "wb");
        if (!f) return;
        std::fprintf(f, "#?RADIANCE\nFORMAT=32-bit_rle_rgbe\n\n-Y %d +X %d\n", film.ny, film.nx);
        for (size_t i = 0; i < (size_t)film.nx * film.ny; ++i) {
                const float r = d[3 * i], g = d[3 * i + 1], b = d[3 * i + 2];
                const float m = std::max(r, std::max(g, b));
                unsigned char px[4] = { 0, 0, 0, 0 };
                if (m >= 1e-32f) {
                        int e;
                        const float sc = std::frexp(m, &e) * 256.0f / m;
                        px[0] = (unsigned char)(r * sc);
                        px[1] = (unsigned char)(g * sc);
                        px[2] = (unsigned char)(b * sc);
                        px[3] = (unsigned char)(e + 128);
                }
                std::fwrite(px, 1, 4, f);
        }
        std::fclose(f);
}

int main(int argc, char** argv)
{
        const char* out = "demo.bmp";
        const char* dump = nullptr;
        const char* gi_dump = nullptr;  // --gi <file>: also run main.cc's light map + filter + cone-traced film
        std::vector<int> gi_devices;    // --gi-devices 0,0,...: the GI film again on these replicas -> <file>.mgpu
        const char* gi_aov = nullptr;   // --gi-aov <prefix>: the GI film's planes -> <prefix>.<plane>.hdr
        const char* animate = nullptr;  // --animate <prefix>: four GI frames of the turning scene -> <prefix>.<k>.hdr
        const char* obj = nullptr;
        int depth = 6, nx = 1024, ny = 1024, pos = 0;  // main.cc:34-35,67
        for (int i = 1; i < argc; ++i) {
                if (!std::strcmp(argv[i], "--dump") && i + 1 < argc) { dump = argv[++i]; continue; }
                if (!std::strcmp(argv[i], "--gi") && i + 1 < argc) { gi_dump = argv[++i]; continue; }
                if (!std::strcmp(argv[i], "--gi-aov") && i + 1 < argc) { gi_aov = argv[++i]; continue; }
                if (!std::strcmp(argv[i], "--animate") && i + 1 < argc) { animate = argv[++i]; continue; }
                if (!std::strcmp(argv[i], "--gi-devices") && i + 1 < argc) {
                        for (const char* p = argv[++i]; *p;) {
                                char* end = nullptr;
                                gi_devices.push_back((int)std::strtol(p, &end, 10));
                                p = (*end == ',') ? end + 1 : end;
                                if (end == p && *p) { std::fprintf(stderr, "bad --gi-devices list\n"); return 1; }
                        }
                        continue;
                }
                switch (pos++) {
                case 0: out = argv[i]; break;
                case 1: depth = std::atoi(argv[i]); break;
                case 2: nx = std::atoi(argv[i]); break;
                case 3: ny = std::atoi(argv[i]); break;
                case 4: obj = argv[i]; break;
                }
        }
        try {
                std::printf("voxelizer...\n");
                auto voxels = obj ? load_obj(obj) : make_sphere(256, 128);
                std::printf("#tris=%zu\noctree...\n", voxels.size());
                std::vector<gi::VoxelBase*> voxel_ptrs;
                for (auto& v : voxels) voxel_ptrs.push_back(&v);
                gi::VoxelOctree root;
                gi::ray_march_init(&root, voxel_ptrs, depth);  // main.cc:67
                std::printf("tracing...\n");
                Camera cam{ 60.f * 3.1415926535897932384626f / 180.f, { 0, 1, 3 }, { 0, 0, 0 }, { 0, 1, 0 } };
                Film film(1.f, 1.f, nx, ny);
                const float l = std::sqrt(1.f + 100.f + 1.f);
                std::vector<vrt_hit> hits;
                render_gpu(&film, cam, &root, 4, Vec3{ 1 / l, 10 / l, 1 / l }, 0.8f, dump ? &hits : nullptr);  // main.cc:118-123
                // spot check through the per-ray reference signatures (main.cc:16)
                auto rays = cam.gen_rays4(film, nx / 2, ny / 2);
                gi::VoxelOctree* leaf = nullptr;
                gi::VoxelBase* vox = nullptr;
                jql::ISect is{};
                const bool hit = gi::ray_march(&root, rays[0], &leaf, &vox, &is);
                std::printf("centre ray: hit=%d", (int)hit);
                if (hit) std::printf(" leaf cell (%u,%u,%u) with %zu triangles, hit (%g,%g,%g)", leaf->cell[0], leaf->cell[1],
                                     leaf->cell[2], leaf->voxels.size(), is.hit.x, is.hit.y, is.hit.z);
                std::printf("\n");
                write_bmp(out, film);
                if (dump) {
                        FILE* f = std::fopen(dump, "wb");
                        std::fwrite(hits.data(), sizeof(vrt_hit), hits.size(), f);
                        std::fclose(f);
                }
                if (gi_dump) {
                        // main.cc:69-123 on the GPU: light map (Film(1,1,2048,2048) there; nx x ny here), filter,
                        // then the cone-traced film of the same camera
                        std::printf("light map...\n");
                        Film sfilm(1.f, 1.f, nx, ny);
                        Camera scam{ 60.f * 3.1415926535897932384626f / 180.f, { 1, 10, 1 }, { 0, 0, 0 }, { 0, 1, 0 } };
                        const Vec3 kd{ 0.7f, 0.6f, 0.5f };
                        light_map_gpu(sfilm, scam, &root, 4, kd);
                        std::printf("filtering...\n");
                        gi::cone_trace_init_filter(&root);
                        std::printf("cone tracing...\n");
                        // main.cc's Res over the axes of non-zero size: a planar scene's Res would be 0, which the GI
                        // entry points refuse (the cone march would not advance)
                        float res = 3.4e38f;
                        for (int k = 0; k < 3; ++k)
                                if (root.aabb.max[k] > root.aabb.min[k])
                                        res = std::min(res, (root.aabb.max[k] - root.aabb.min[k]) / std::pow(2.f, (float)depth));
                        Film gfilm(1.f, 1.f, nx, ny);
                        render_gi_gpu(&gfilm, cam, &root, 4, kd, res);
                        if (hit) {
                                const Vec3 c = gi::cone_trace(root, is, res);
                                std::printf("centre ray indirect light (%g,%g,%g)\n", c.x, c.y, c.z);
                        }
                        write_hdr((std::string(gi_dump) + ".hdr").c_str(), gfilm);  // main.cc:125-126
                        const auto d = gfilm.to_float_array();
                        FILE* f = std::fopen(gi_dump, "wb");
                        std::fwrite(d.data(), sizeof(float), d.size(), f);
                        std::fclose(f);
                        // the film's factors (a denoiser's albedo and normal guides, the light terms), rendered by
                        // `render` and written to <prefix><infix>.<plane>.hdr
                        auto write_planes = [&](const char* infix, auto&& render) {
                                Film albedo(1.f, 1.f, nx, ny), direct(1.f, 1.f, nx, ny), indirect(1.f, 1.f, nx, ny),
                                        normal(1.f, 1.f, nx, ny);
                                gi::GiAov aov;
                                aov.albedo = &albedo;
                                aov.direct = &direct;
                                aov.indirect = &indirect;
                                aov.normal = &normal;
                                render(aov);
                                const std::pair<const char*, const Film*> planes[4] = {
                                        { "albedo", &albedo }, { "direct", &direct }, { "indirect", &indirect }, { "normal", &normal }
                                };
                                for (const auto& pl : planes)
                                        write_hdr((std::string(gi_aov) + infix + "." + pl.first + ".hdr").c_str(), *pl.second);
                        };
                        if (gi_aov) {
                                write_planes("", [&](gi::GiAov& aov) { render_gi_aov_gpu(nullptr, cam, &root, 4, kd, res, aov); });
                                std::printf("GI planes written\n");
                        }
                        if (!gi_devices.empty()) {
                                // the same three GI statements on the replicas of gi::MultiGpu
                                std::printf("GI film on %zu replicas...\n", gi_devices.size());
                                gi::MultiGpu replicas(&root, gi_devices);
                                light_map_gpu(sfilm, scam, replicas, 4, kd);
                                gi::cone_trace_init_filter(replicas);
                                Film mfilm(1.f, 1.f, nx, ny);
                                render_gi_gpu(&mfilm, cam, replicas, 4, kd, res);
                                const auto md = mfilm.to_float_array();
                                FILE* mf = std::fopen((std::string(gi_dump) + ".mgpu").c_str(), "wb");
                                std::fwrite(md.data(), sizeof(float), md.size(), mf);
                                std::fclose(mf);
                                if (gi_aov) {
                                        write_planes(".mgpu", [&](gi::GiAov& aov) {
                                                render_gi_aov_gpu(nullptr, cam, replicas, 4, kd, res, aov);
                                        });
                                        std::printf("GI planes on %zu replicas written\n", gi_devices.size());
                                }
                        }
                }
                if (animate) {
                        // a moving scene: per frame one transform update (the pose is absolute: a turn of (k+1)
                        // quarters from the rest pose), the light map and filter again, the GI film
                        const Vec3 kd{ 0.7f, 0.6f, 0.5f };
                        Film sfilm(1.f, 1.f, nx, ny);
                        Camera scam{ 60.f * 3.1415926535897932384626f / 180.f, { 1, 10, 1 }, { 0, 0, 0 }, { 0, 1, 0 } };
                        const float cx = (root.aabb.min.x + root.aabb.max.x) * 0.5f;
                        const float cz = (root.aabb.min.z + root.aabb.max.z) * 0.5f;
                        const float cs[4][2] = { { 0, 1 }, { -1, 0 }, { 0, -1 }, { 1, 0 } };  // cos, sin of (k+1) * 90 deg
                        for (int k = 0; k < 4; ++k) {
                                const float c = cs[k][0], s = cs[k][1];
                                // p' = R (p - centre) + centre about the y axis: R = [[c,0,s],[0,1,0],[-s,0,c]]
                                vrt_xform xf{};
                                xf.first_tri = 0;
                                xf.num_tris = (uint32_t)voxels.size();
                                const float m[12] = { c, 0, s, cx - (c * cx + s * cz), 0, 1, 0, 0, -s, 0, c, cz - (-s * cx + c * cz) };
                                const float n[9] = { c, 0, s, 0, 1, 0, -s, 0, c };
                                std::memcpy(xf.m, m, sizeof m);
                                std::memcpy(xf.n, n, sizeof n);
                                gi::transform_gpu(&root, { xf });
                                light_map_gpu(sfilm, scam, &root, 4, kd);
                                gi::cone_trace_init_filter(&root);
                                float res = 3.4e38f;
                                for (int a = 0; a < 3; ++a)
                                        if (root.aabb.max[a] > root.aabb.min[a])
                                                res = std::min(res, (root.aabb.max[a] - root.aabb.min[a]) /
                                                                            std::pow(2.f, (float)depth));
                                Film afilm(1.f, 1.f, nx, ny);
                                render_gi_gpu(&afilm, cam, &root, 4, kd, res);
                                write_hdr((std::string(animate) + "." + std::to_string(k) + ".hdr").c_str(), afilm);
                                // the per-ray mirror sees the new leaves: the centre ray's leaf and triangle
                                gi::VoxelOctree* aleaf = nullptr;
                                gi::VoxelBase* avox = nullptr;
                                jql::ISect ais{};
                                if (gi::ray_march(&root, rays[0], &aleaf, &avox, &ais))
                                        std::printf("frame %d centre ray: leaf cell (%u,%u,%u) with %zu triangles, triangle %td\n", k,
                                                    aleaf->cell[0], aleaf->cell[1], aleaf->cell[2], aleaf->voxels.size(),
                                                    static_cast<gi::Triangle*>(avox) - voxels.data());
                                else
                                        std::printf("frame %d centre ray: miss\n", k);
                        }
                        std::printf("animation written\n");
                }
                std::printf("success.\n");
        } catch (const std::exception& e) {
                std::fprintf(stderr, "error: %s\n", e.what());
                return 2;
        }
        return 0;
}
