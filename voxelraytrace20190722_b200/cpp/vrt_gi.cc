// vrt_gi.cc -- implementation of the C++ host mirror (vrt_gi.h) on top of libvrt.so.
// No arithmetic of the hot path happens here: geometry is packed into flat arrays and
// handed to the C ABI; results are mapped back onto the reference's object model.
#include "vrt_gi.h"

#include <cmath>
#include <cstring>
#include <mutex>
#include <stdexcept>
#include <string>

namespace {
[[noreturn]] void fail(const char* what)
{
        throw std::runtime_error(std::string(what) + ": " + vrt_last_error());
}
void check(int rc, const char* what)
{
        if (rc != VRT_OK)
                fail(what);
}
vrt_ray to_native(const jql::Ray& r)
{
        vrt_ray n;
        n.o[0] = r.o.x; n.o[1] = r.o.y; n.o[2] = r.o.z;
        n.d[0] = r.d.x; n.d[1] = r.d.y; n.d[2] = r.d.z;
        n.tmin = r.tmin;
        n.tmax = r.tmax;
        return n;
}
}  // namespace

namespace gi {

struct GpuTree {
        vrt_tree* tree = nullptr;
        int max_depth = 0;
        std::vector<VoxelBase*> voxels;  // index -> object (triangle index == insertion index)
        // leaf set exported once (Morton order) for on-demand materialisation
        std::vector<uint32_t> leaf_cell, leaf_count, leaf_start, leaf_refs;
        std::unordered_map<uint64_t, std::unique_ptr<VoxelOctree>> leaves;  // key = packed cell
        std::unordered_map<uint64_t, uint32_t> leaf_index;
        std::mutex mu;
        ~GpuTree() { vrt_tree_free(tree); }
        static uint64_t key(const uint32_t c[3]) { return ((uint64_t)c[0] << 42) | ((uint64_t)c[1] << 21) | c[2]; }
        VoxelOctree* leaf(const uint32_t c[3]);
};

VoxelOctree* GpuTree::leaf(const uint32_t c[3])
{
        std::lock_guard<std::mutex> lock(mu);
        if (leaf_index.empty() && !leaf_count.empty()) {
                uint32_t run = 0;
                leaf_start.resize(leaf_count.size());
                for (size_t i = 0; i < leaf_count.size(); ++i) {
                        leaf_start[i] = run;
                        run += leaf_count[i];
                        leaf_index[key(&leaf_cell[3 * i])] = (uint32_t)i;
                }
        }
        const uint64_t k = key(c);
        auto it = leaves.find(k);
        if (it != leaves.end())
                return it->second.get();
        auto node = std::make_unique<VoxelOctree>();
        node->depth = max_depth;
        std::memcpy(node->cell, c, sizeof node->cell);
        auto li = leaf_index.find(k);
        if (li != leaf_index.end()) {
                const uint32_t i = li->second;
                for (uint32_t j = 0; j < leaf_count[i]; ++j)
                        node->voxels.push_back(voxels[leaf_refs[leaf_start[i] + j]]);
        }
        VoxelOctree* p = node.get();
        leaves[k] = std::move(node);
        return p;
}

Triangle::Triangle(Vec3 p0, Vec3 p1, Vec3 p2, Vec3 n0, Vec3 n1, Vec3 n2)
        : p_{ p0, p1, p2 }, n_{ n0, n1, n2 }
{
        // normals normalised like the reference ctor (voxel_octree.cc:426; jql::normalize = v / sqrtf(dot(v,v)),
        // value_sum from 0; this file is compiled with -ffp-contract=off) -- ray_march_init hands them to the GPU
        // build verbatim (VRT_BUILD_UNIT_NORMALS).  AABB = min/max of the vertices (voxel_octree.cc:430).
        for (int v = 0; v < 3; ++v) {
                float s = 0.f;
                s += n_[v].x * n_[v].x;
                s += n_[v].y * n_[v].y;
                s += n_[v].z * n_[v].z;
                const float l = std::sqrt(s);
                n_[v] = Vec3{ n_[v].x / l, n_[v].y / l, n_[v].z / l };
        }
        aabb_.min = aabb_.max = p0;
        for (int v = 1; v < 3; ++v)
                for (int k = 0; k < 3; ++k) {
                        if (p_[v][k] < aabb_.min[k]) aabb_.min[k] = p_[v][k];
                        if (aabb_.max[k] < p_[v][k]) aabb_.max[k] = p_[v][k];
                }
}

bool Triangle::is_overlap(const AABB3D& aabb) const
{
        const float box[6] = { aabb.min.x, aabb.min.y, aabb.min.z, aabb.max.x, aabb.max.y, aabb.max.z };
        uint8_t out = 0;
        check(vrt_tri_overlap_aabb_batch(box, vertices(), 1, &out), "Triangle::is_overlap");
        return out != 0;
}

bool Triangle::isect(const Ray& ray, ISect* isect) const
{
        // Triangle::isect (voxel_octree.cc:438-460) is part of the leaf stage of the ray
        // kernel; a stand-alone call builds a depth-1 tree around this triangle (the root
        // is then the only leaf) -- but the root slab test would interfere, so the public
        // predicate is used instead and only the hit flag + position are reported.
        double in[15] = { ray.o.x, ray.o.y, ray.o.z, ray.d.x, ray.d.y, ray.d.z };
        for (int k = 0; k < 9; ++k)
                in[6 + k] = vertices()[k];
        uint8_t res = 0;
        double tuv[3];
        check(vrt_raytri_batch(in, 1, &res, tuv), "Triangle::isect");
        if (res != 1)
                return false;
        if (isect) {
                // the FP32 shell of Triangle::isect (voxel_octree.cc:449-454) around the GPU's FP64 result:
                // u,v,w = clamp(.,0,1); normal = normalize(n0*w + n1*u + n2*v); hit = o + (float)t * d
                auto clamp01 = [](float s) { return s > 1.f ? 1.f : (s < 0.f ? 0.f : s); };
                const float u = clamp01((float)tuv[1]), v = clamp01((float)tuv[2]);
                const float w = clamp01(1 - u - v);
                Vec3 n;
                for (int k = 0; k < 3; ++k)
                        n[k] = (n_[0][k] * w + n_[1][k] * u) + n_[2][k] * v;
                float s = 0.f;
                s += n.x * n.x;
                s += n.y * n.y;
                s += n.z * n.z;
                const float l = std::sqrt(s);
                isect->normal = Vec3{ n.x / l, n.y / l, n.z / l };
                const float t = (float)tuv[0];
                isect->hit = Vec3{ ray.o.x + t * ray.d.x, ray.o.y + t * ray.d.y, ray.o.z + t * ray.d.z };
        }
        return true;
}

static GpuTree* gpu_tree(VoxelOctree* root, const char* what)
{
        if (!root || !root->gpu)
                throw std::runtime_error(std::string(what) + ": octree not initialised (call ray_march_init)");
        return root->gpu.get();
}

// the root box, depth and exported leaf set of the handle's current octree; the leaves materialised from an earlier
// one are dropped (after an update their cells and triangle lists no longer hold)
static void load_leaf_set(VoxelOctree* root)
{
        GpuTree* g = root->gpu.get();
        vrt_tree_info info;
        check(vrt_tree_get_info(g->tree, &info), "vrt_tree_get_info");
        root->aabb.min = Vec3{ info.root_aabb[0], info.root_aabb[1], info.root_aabb[2] };
        root->aabb.max = Vec3{ info.root_aabb[3], info.root_aabb[4], info.root_aabb[5] };
        std::lock_guard<std::mutex> lock(g->mu);
        g->max_depth = info.max_depth;
        g->leaf_cell.assign(3 * info.num_leaves, 0);
        g->leaf_count.assign(info.num_leaves, 0);
        g->leaf_refs.assign(info.num_refs, 0);
        g->leaf_start.clear();
        g->leaf_index.clear();
        g->leaves.clear();
        vrt_tree_view view{ g->leaf_cell.data(), g->leaf_count.data(), g->leaf_refs.data(), nullptr };
        check(vrt_tree_export(g->tree, &view), "vrt_tree_export");
}

void ray_march_init(VoxelOctree* root, std::vector<VoxelBase*>& voxels, int max_depth)
{
        auto g = std::make_shared<GpuTree>();
        g->max_depth = max_depth;
        g->voxels = voxels;
        std::vector<float> tri(9 * voxels.size()), nrm(9 * voxels.size());
        for (size_t i = 0; i < voxels.size(); ++i) {
                std::memcpy(&tri[9 * i], voxels[i]->vertices(), 36);
                std::memcpy(&nrm[9 * i], voxels[i]->normals(), 36);
        }
        check(vrt_build_ex(tri.data(), nrm.data(), (uint32_t)voxels.size(), max_depth, VRT_BUILD_UNIT_NORMALS, &g->tree),
              "gi::ray_march_init");
        root->depth = 1;
        root->gpu = std::move(g);
        load_leaf_set(root);
}

void update_triangles_gpu(VoxelOctree* root, const std::vector<float>& tri_xyz, const std::vector<float>& tri_nrm,
                          int max_depth)
{
        GpuTree* g = gpu_tree(root, "gi::update_triangles_gpu");
        if (tri_xyz.size() != 9 * g->voxels.size() || (!tri_nrm.empty() && tri_nrm.size() != tri_xyz.size()))
                throw std::runtime_error("gi::update_triangles_gpu: expected 9 floats per triangle of the octree");
        check(vrt_update_triangles(g->tree, tri_xyz.data(), tri_nrm.empty() ? nullptr : tri_nrm.data(),
                                   (uint32_t)g->voxels.size(), max_depth ? max_depth : g->max_depth),
              "gi::update_triangles_gpu");
        load_leaf_set(root);
}

void transform_gpu(VoxelOctree* root, const std::vector<vrt_xform>& xf, int max_depth)
{
        GpuTree* g = gpu_tree(root, "gi::transform_gpu");
        check(vrt_update_xform(g->tree, xf.data(), (uint32_t)xf.size(), max_depth ? max_depth : g->max_depth),
              "gi::transform_gpu");
        load_leaf_set(root);
}

void update_triangles_gpu(MultiGpu& replicas, const std::vector<float>& tri_xyz, const std::vector<float>& tri_nrm,
                          int max_depth)
{
        if (tri_xyz.empty() || tri_xyz.size() % 9 || (!tri_nrm.empty() && tri_nrm.size() != tri_xyz.size()))
                throw std::runtime_error("gi::update_triangles_gpu: expected 9 floats per triangle");
        check(vrt_mgpu_update_triangles(replicas.native(), tri_xyz.data(), tri_nrm.empty() ? nullptr : tri_nrm.data(),
                                        (uint32_t)(tri_xyz.size() / 9), max_depth),
              "gi::update_triangles_gpu");
}

void transform_gpu(MultiGpu& replicas, const std::vector<vrt_xform>& xf, int max_depth)
{
        check(vrt_mgpu_update_xform(replicas.native(), xf.data(), (uint32_t)xf.size(), max_depth), "gi::transform_gpu");
}

const vrt_tree* native_handle(const VoxelOctree* root)
{
        return (root && root->gpu) ? root->gpu->tree : nullptr;
}

static void fill(GpuTree* g, const vrt_hit& h, MarchResult* r)
{
        r->hit = h.hit != 0;
        r->leaf = nullptr;
        r->voxel = nullptr;
        if (!r->hit)
                return;
        r->leaf = g->leaf(h.cell);
        r->voxel = g->voxels[h.tri];
        r->isect.hit = Vec3{ h.pos[0], h.pos[1], h.pos[2] };
        r->isect.normal = Vec3{ h.nrm[0], h.nrm[1], h.nrm[2] };
}

void ray_march_batch(VoxelOctree* root, const std::vector<Ray>& rays, std::vector<MarchResult>* out)
{
        if (!root || !root->gpu)
                throw std::runtime_error("gi::ray_march: octree not initialised (call ray_march_init)");
        std::vector<vrt_ray> nr(rays.size());
        for (size_t i = 0; i < rays.size(); ++i)
                nr[i] = to_native(rays[i]);
        std::vector<vrt_hit> hits(rays.size());
        check(vrt_trace_rays(root->gpu->tree, nr.data(), nr.size(), hits.data()), "gi::ray_march");
        out->resize(rays.size());
        for (size_t i = 0; i < rays.size(); ++i)
                fill(root->gpu.get(), hits[i], &(*out)[i]);
}

bool ray_march(VoxelOctree* root, const Ray& ray, VoxelOctree** leaf_ptr, VoxelBase** voxel_ptr, ISect* isect,
               bool /*even_invisible: Triangle::is_visible() is always true, voxel_octree.cc:493-496*/)
{
        if (!root || !root->gpu)
                throw std::runtime_error("gi::ray_march: octree not initialised (call ray_march_init)");
        const vrt_ray nr = to_native(ray);
        vrt_hit h;
        check(vrt_trace_rays(root->gpu->tree, &nr, 1, &h), "gi::ray_march");
        if (!h.hit)
                return false;  // outputs are written only on `true`, like the reference
        MarchResult r;
        fill(root->gpu.get(), h, &r);
        if (leaf_ptr) *leaf_ptr = r.leaf;
        if (voxel_ptr) *voxel_ptr = r.voxel;
        if (isect) *isect = r.isect;
        return true;
}

}  // namespace gi

// ---- Film (camera.cc:3-63) -----------------------------------------------------------
Film::Film(float w_, float h_, int nx_, int ny_) : w{ w_ }, h{ h_ }, nx{ nx_ }, ny{ ny_ }
{
        data_.assign((size_t)nx * ny, jql::Vec3{ 0, 0, 0 });
}

void Film::add(int x, int y, const jql::Vec3& c)
{
        jql::Vec3& d = data_[(size_t)y * nx + x];
        d.x += c.x;
        d.y += c.y;
        d.z += c.z;
}

std::vector<std::uint8_t> Film::to_byte_array() const
{
        std::vector<std::uint8_t> d((size_t)nx * ny * 3);
        for (size_t i = 0; i < data_.size(); ++i) {
                d[3 * i + 0] = static_cast<std::uint8_t>(data_[i].x * 255.9f);
                d[3 * i + 1] = static_cast<std::uint8_t>(data_[i].y * 255.9f);
                d[3 * i + 2] = static_cast<std::uint8_t>(data_[i].z * 255.9f);
        }
        return d;
}

std::vector<float> Film::to_float_array() const
{
        std::vector<float> d((size_t)nx * ny * 3);
        std::memcpy(d.data(), data_.data(), d.size() * sizeof(float));
        return d;
}

// ---- Camera (camera.cc:65-112) ---------------------------------------------------------
Camera::Camera(float fov_, jql::Vec3 eye, jql::Vec3 spot, jql::Vec3 up, float near_, float far_)
        : fov{ fov_ }, near{ near_ }, far{ far_ }
{
        const float c[10] = { fov_, eye.x, eye.y, eye.z, spot.x, spot.y, spot.z, up.x, up.y, up.z };
        std::memcpy(cam10_, c, sizeof c);
}

vrt_camera Camera::native(const Film& film, int spp) const
{
        vrt_camera c;
        check(vrt_camera_init(cam10_, film.h, film.nx, film.ny, spp, &c), "Camera");
        c.tmin = near;
        c.tmax = far;
        return c;
}

static std::vector<jql::Ray> gen_pixel(const Camera& cam, const Film& film, int px, int py, int spp)
{
        const vrt_camera c = cam.native(film, spp);
        std::vector<vrt_ray> r((size_t)spp);
        check(vrt_gen_rays(&c, px, py, px + 1, py + 1, r.data()), "Camera::gen_rays");  // range-checked like the asserts
        std::vector<jql::Ray> out((size_t)spp);
        for (int k = 0; k < spp; ++k) {
                out[k].o = jql::Vec3{ r[k].o[0], r[k].o[1], r[k].o[2] };
                out[k].d = jql::Vec3{ r[k].d[0], r[k].d[1], r[k].d[2] };
                out[k].tmin = r[k].tmin;
                out[k].tmax = r[k].tmax;
        }
        return out;
}

std::vector<jql::Ray> Camera::gen_rays1(const Film& film, int px, int py) { return gen_pixel(*this, film, px, py, 1); }
std::vector<jql::Ray> Camera::gen_rays4(const Film& film, int px, int py) { return gen_pixel(*this, film, px, py, 4); }

void render_gpu(Film* film, Camera& cam, gi::VoxelOctree* root, int spp, const jql::Vec3& light_dir, float kd,
                std::vector<vrt_hit>* hits)
{
        if (!root || !root->gpu)
                throw std::runtime_error("render_gpu: octree not initialised (call ray_march_init)");
        const vrt_camera c = cam.native(*film, spp);
        vrt_shade sh{ { light_dir.x, light_dir.y, light_dir.z }, kd, 0.f, 0 };
        check(vrt_render_camera(root->gpu->tree, &c, &sh, 0, 0, film->nx, film->ny, &film->data()->x), "render_gpu");
        if (hits) {
                hits->resize((size_t)film->nx * film->ny * spp);
                check(vrt_trace_camera(root->gpu->tree, &c, 0, 0, film->nx, film->ny, hits->data()), "render_gpu");
        }
}

// ---- GI rows (voxel_octree.h:90-92, main.cc:75-97,117-123) ------------------------------------
namespace gi {
static vrt_tree* gi_tree(const VoxelOctree* root, const char* what)
{
        if (!root || !root->gpu)
                throw std::runtime_error(std::string(what) + ": octree not initialised (call ray_march_init)");
        return root->gpu->tree;
}

void cone_trace_init_filter(VoxelOctree* root)
{
        check(vrt_gi_filter(gi_tree(root, "cone_trace_init_filter")), "cone_trace_init_filter");
}

void cone_trace_batch(const VoxelOctree& root, const std::vector<ISect>& isects, float min_voxel_size, std::vector<Vec3>* out)
{
        std::vector<float> pos(3 * isects.size()), nrm(3 * isects.size());
        for (size_t i = 0; i < isects.size(); ++i)
                for (int k = 0; k < 3; ++k) {
                        pos[3 * i + k] = isects[i].hit[k];
                        nrm[3 * i + k] = isects[i].normal[k];
                }
        out->resize(isects.size());
        check(vrt_gi_cone_trace(gi_tree(&root, "cone_trace"), pos.data(), nrm.data(), isects.size(), min_voxel_size,
                                out->empty() ? nullptr : &(*out)[0].x),
              "cone_trace");
}

Vec3 cone_trace(const VoxelOctree& root, const ISect& isect, float min_voxel_size)
{
        std::vector<Vec3> out;
        cone_trace_batch(root, { isect }, min_voxel_size, &out);
        return out[0];
}

MultiGpu::MultiGpu(const VoxelOctree* root, const std::vector<int>& devices)
{
        check(vrt_mgpu_create(gi_tree(root, "gi::MultiGpu"), (int)devices.size(), devices.data(), &m_), "gi::MultiGpu");
}

MultiGpu::~MultiGpu() { vrt_mgpu_free(m_); }

void cone_trace_init_filter(MultiGpu& replicas)
{
        check(vrt_mgpu_gi_filter(replicas.native()), "cone_trace_init_filter");
}
}  // namespace gi

void light_map_gpu(const Film& sfilm, Camera& scam, gi::VoxelOctree* root, int spp, const jql::Vec3& kd)
{
        vrt_tree* t = gi::gi_tree(root, "light_map_gpu");
        const vrt_camera c = scam.native(sfilm, spp);
        const float k[3] = { kd.x, kd.y, kd.z };
        check(vrt_gi_init(t), "light_map_gpu");
        check(vrt_gi_splat_camera(t, &c, k), "light_map_gpu");
}

void render_gi_gpu(Film* film, Camera& cam, gi::VoxelOctree* root, int spp, const jql::Vec3& kd, float res)
{
        vrt_tree* t = gi::gi_tree(root, "render_gi_gpu");
        const vrt_camera c = cam.native(*film, spp);
        const float k[3] = { kd.x, kd.y, kd.z };
        check(vrt_gi_render_camera(t, &c, k, res, 0, 0, film->nx, film->ny, &film->data()->x), "render_gi_gpu");
}

// The film geometry of a render_gi_aov_gpu call (the film, else the first float plane; all of one size), with
// aov.hits resized for it; returns the vrt_gi_aov of aov's buffers.
static vrt_gi_aov gi_aov_native(const Film* film_or_null, int spp, gi::GiAov& aov, const Film** geometry)
{
        Film* const planes[4] = { aov.albedo, aov.direct, aov.indirect, aov.normal };
        const Film* geo = film_or_null;
        for (Film* p : planes)
                if (!geo)
                        geo = p;
        if (!geo)
                throw std::runtime_error("render_gi_aov_gpu: neither a film nor a float plane gives the film size");
        for (Film* p : planes)
                if (p && (p->nx != geo->nx || p->ny != geo->ny))
                        throw std::runtime_error("render_gi_aov_gpu: the planes and the film differ in size");
        if (aov.hits)
                aov.hits->resize((size_t)geo->nx * geo->ny * spp);
        float* dst[4];
        for (int i = 0; i < 4; ++i)
                dst[i] = planes[i] ? &planes[i]->data()->x : nullptr;
        *geometry = geo;
        return vrt_gi_aov{ dst[0], dst[1], dst[2], dst[3], aov.hits ? aov.hits->data() : nullptr };
}

void render_gi_aov_gpu(Film* film_or_null, Camera& cam, gi::VoxelOctree* root, int spp, const jql::Vec3& kd, float res,
                       gi::GiAov& aov)
{
        vrt_tree* t = gi::gi_tree(root, "render_gi_aov_gpu");
        const Film* geo = nullptr;
        const vrt_gi_aov a = gi_aov_native(film_or_null, spp, aov, &geo);
        const vrt_camera c = cam.native(*geo, spp);
        const float k[3] = { kd.x, kd.y, kd.z };
        check(vrt_gi_render_aov(t, &c, k, res, 0, 0, geo->nx, geo->ny, film_or_null ? &film_or_null->data()->x : nullptr,
                                &a),
              "render_gi_aov_gpu");
}

void light_map_gpu(const Film& sfilm, Camera& scam, gi::MultiGpu& replicas, int spp, const jql::Vec3& kd)
{
        const vrt_camera c = scam.native(sfilm, spp);
        const float k[3] = { kd.x, kd.y, kd.z };
        check(vrt_mgpu_gi_init(replicas.native()), "light_map_gpu");
        check(vrt_mgpu_gi_splat_camera(replicas.native(), &c, k), "light_map_gpu");
}

void render_gi_gpu(Film* film, Camera& cam, gi::MultiGpu& replicas, int spp, const jql::Vec3& kd, float res)
{
        const vrt_camera c = cam.native(*film, spp);
        const float k[3] = { kd.x, kd.y, kd.z };
        // the devices DMA their bands into the film; page-locked for the call, they copy in parallel (if the range
        // cannot be locked, e.g. because the caller already did, the copies still land, staged by the driver)
        float* dst = &film->data()->x;
        const uint64_t bytes = (uint64_t)film->nx * film->ny * 3 * sizeof(float);
        const bool locked = vrt_host_register(dst, bytes) == VRT_OK;
        const int rc = vrt_mgpu_gi_render(replicas.native(), &c, k, res, dst);
        if (locked)
                vrt_host_unregister(dst);
        check(rc, "render_gi_gpu");
}

void render_gi_aov_gpu(Film* film_or_null, Camera& cam, gi::MultiGpu& replicas, int spp, const jql::Vec3& kd, float res,
                       gi::GiAov& aov)
{
        const Film* geo = nullptr;
        const vrt_gi_aov a = gi_aov_native(film_or_null, spp, aov, &geo);
        const vrt_camera c = cam.native(*geo, spp);
        const float k[3] = { kd.x, kd.y, kd.z };
        float* const film = film_or_null ? &film_or_null->data()->x : nullptr;
        // every output page-locked for the call, as in render_gi_gpu (a range that cannot be locked still receives
        // its bands, staged by the driver)
        const uint64_t plane_bytes = (uint64_t)geo->nx * geo->ny * 3 * sizeof(float);
        void* const dst[6] = { film, a.albedo, a.direct, a.indirect, a.normal, a.hits };
        const uint64_t bytes[6] = { plane_bytes, plane_bytes, plane_bytes, plane_bytes, plane_bytes,
                                    (uint64_t)geo->nx * geo->ny * spp * sizeof(vrt_hit16) };
        bool locked[6] = {};
        for (int i = 0; i < 6; ++i)
                locked[i] = dst[i] && vrt_host_register(dst[i], bytes[i]) == VRT_OK;
        const int rc = vrt_mgpu_gi_render_aov(replicas.native(), &c, k, res, film, &a);
        for (int i = 0; i < 6; ++i)
                if (locked[i])
                        vrt_host_unregister(dst[i]);
        check(rc, "render_gi_aov_gpu");
}

// vrt_set_materials / vrt_mgpu_set_materials with the mirror's material records
template <class H, class Fn>
static void set_materials_native(Fn fn, H* h, const std::vector<jql::Vec2>& uv, const std::vector<std::uint32_t>& tri_material,
                                 const std::vector<GpuMaterial>& materials, const std::vector<GpuTexture>& textures)
{
        std::vector<float> kd(3 * materials.size());
        std::vector<int32_t> mt(materials.size());
        for (size_t m = 0; m < materials.size(); ++m) {
                kd[3 * m] = materials[m].diffuse.x;
                kd[3 * m + 1] = materials[m].diffuse.y;
                kd[3 * m + 2] = materials[m].diffuse.z;
                mt[m] = materials[m].texture;
        }
        std::vector<vrt_texture> tx(textures.size());
        for (size_t i = 0; i < textures.size(); ++i)
                tx[i] = vrt_texture{ textures[i].width, textures[i].height, textures[i].channels, textures[i].data };
        check(fn(h, uv.empty() ? nullptr : &uv[0].x, tri_material.data(), (uint32_t)materials.size(), kd.data(), mt.data(),
                 (uint32_t)tx.size(), tx.data()),
              "set_materials_gpu");
}

void set_materials_gpu(gi::VoxelOctree* root, const std::vector<jql::Vec2>& uv, const std::vector<std::uint32_t>& tri_material,
                       const std::vector<GpuMaterial>& materials, const std::vector<GpuTexture>& textures)
{
        set_materials_native(vrt_set_materials, gi::gi_tree(root, "set_materials_gpu"), uv, tri_material, materials, textures);
}

void set_materials_gpu(gi::MultiGpu& replicas, const std::vector<jql::Vec2>& uv, const std::vector<std::uint32_t>& tri_material,
                       const std::vector<GpuMaterial>& materials, const std::vector<GpuTexture>& textures)
{
        set_materials_native(vrt_mgpu_set_materials, replicas.native(), uv, tri_material, materials, textures);
}

// ---- predicates ----------------------------------------------------------------------------
int triBoxOverlap(float boxcenter[3], float boxhalfsize[3], float triverts[3][3])
{
        uint8_t out = 0;
        check(vrt_tribox_batch(boxcenter, boxhalfsize, &triverts[0][0], 1, &out), "triBoxOverlap");
        return out;
}

int intersect_triangle3(double orig[3], double dir[3], double vert0[3], double vert1[3], double vert2[3], double* t,
                        double* u, double* v)
{
        double in[15];
        std::memcpy(in, orig, 24);
        std::memcpy(in + 3, dir, 24);
        std::memcpy(in + 6, vert0, 24);
        std::memcpy(in + 9, vert1, 24);
        std::memcpy(in + 12, vert2, 24);
        uint8_t res = 0;
        double tuv[3];
        check(vrt_raytri_batch(in, 1, &res, tuv), "intersect_triangle3");
        if (res == 1) {
                *t = tuv[0];
                *u = tuv[1];
                *v = tuv[2];
        }
        return res;
}
