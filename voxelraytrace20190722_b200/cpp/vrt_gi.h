// vrt_gi.h -- C++ host mirror of the reference's surface for the octree hot path, on
// top of the C ABI (include/vrt.h).  Same names, argument meaning and error behaviour
// as the reference headers it mirrors (paths relative to VoxelRayTrace20190722/):
//
//   jql::Vec2/Vec3/Ray/ISect/AABB3D      graphics_math.h:44-88,1132-1167,1220-1266
//   gi::VoxelBase / gi::Triangle         voxel_octree.h:36-59,94-113
//   gi::VoxelOctree                      voxel_octree.h:61-83
//   gi::ray_march_init / gi::ray_march   voxel_octree.h:85-89
//   Film / Camera / render_mt            camera.h:24-83
//   triBoxOverlap / intersect_triangle3  tribox2.h:15 / raytri.h:5-7
//
// Nothing here computes on the CPU: every call lands in libvrt.so (CUDA); without a
// device the calls throw std::runtime_error with vrt_last_error().  A maintainer of
// the reference keeps main.cc and swaps camera.cc/voxel_octree.cc/tribox2.cc/raytri.cc
// for this translation unit (INTEGRATION.md).
#ifndef VRT_GI_H
#define VRT_GI_H

#include <cstdint>
#include <limits>
#include <memory>
#include <unordered_map>
#include <vector>

#include "../../include/vrt.h"

namespace jql {
struct Vec2 { float x, y; };
struct Vec3 {
        float x, y, z;
        float& operator[](int i) { return (&x)[i]; }
        const float& operator[](int i) const { return (&x)[i]; }
};
struct Ray {  // graphics_math.h:1150-1167.  NOTE: like vrt_ray, d is taken verbatim here;
              // use Ray::make() for the reference ctor's normalisation (done on the GPU).
        Vec3 o, d;
        float tmin = 0.f, tmax = std::numeric_limits<float>::max();
};
struct ISect { Vec3 hit, normal; };
struct AABB3D { Vec3 min, max; };
}  // namespace jql

namespace gi {
using jql::AABB3D;
using jql::ISect;
using jql::Ray;
using jql::Vec2;
using jql::Vec3;

class VoxelBase {  // voxel_octree.h:36-59 (hot-path half)
public:
        virtual ~VoxelBase() = default;
        virtual AABB3D get_aabb() const = 0;
        virtual bool is_overlap(const AABB3D& aabb) const = 0;            // GPU: vrt_tri_overlap_aabb_batch
        virtual bool isect(const Ray& ray, ISect* isect) const = 0;       // GPU: vrt_raytri_batch
        virtual bool is_visible() const { return true; }
        // the flat geometry the GPU path needs (the reference keeps p_/n_ private)
        virtual const float* vertices() const = 0;  // 9 floats
        virtual const float* normals() const = 0;   // 9 floats
};

class Triangle : public VoxelBase {  // voxel_octree.h:94-113 (geometry half; no material)
public:
        Triangle(Vec3 p0, Vec3 p1, Vec3 p2, Vec3 n0, Vec3 n1, Vec3 n2);
        AABB3D get_aabb() const override { return aabb_; }
        bool is_overlap(const AABB3D& aabb) const override;
        bool isect(const Ray& ray, ISect* isect) const override;
        const float* vertices() const override { return &p_[0].x; }
        const float* normals() const override { return &n_[0].x; }

private:
        Vec3 p_[3];
        Vec3 n_[3];
        AABB3D aabb_;
};

struct GpuTree;  // owns the vrt_tree* and the leaf materialisation tables

class VoxelOctree {  // voxel_octree.h:61-83
public:
        AABB3D aabb{};
        std::vector<VoxelBase*> voxels;               // leaf: triangles in insertion order
        std::unique_ptr<VoxelOctree> children[8];     // not materialised on the GPU path (see leaf())
        float coverage{};
        int depth{};
        Vec3 illum[6]{};
        // GPU side (root only)
        std::shared_ptr<GpuTree> gpu;
        uint32_t cell[3]{};                           // leaf cell coordinates at level max_depth-1
};

// voxel_octree.h:85-86.  Packs the triangles, runs vrt_build; root->aabb is filled.
void ray_march_init(VoxelOctree* root, std::vector<VoxelBase*>& voxels, int max_depth);
// voxel_octree.h:87-89.  One ray = one kernel launch (link-compatible spot checks);
// *leaf_ptr is a host VoxelOctree materialised on demand (aabb, voxels, cell filled).
bool ray_march(VoxelOctree* root, const Ray& ray, VoxelOctree** leaf_ptr, VoxelBase** voxel_ptr, ISect* isect,
               bool even_invisible = false);
// Batched form of the same call: out[i] mirrors (return value, *leaf_ptr, *voxel_ptr, *isect).
struct MarchResult {
        bool hit;
        VoxelOctree* leaf;
        VoxelBase* voxel;
        ISect isect;
};
void ray_march_batch(VoxelOctree* root, const std::vector<Ray>& rays, std::vector<MarchResult>* out);
const vrt_tree* native_handle(const VoxelOctree* root);
// voxel_octree.h:90-92 (GI rows): the filter runs over the GPU-resident per-node state that
// light_map_gpu() filled; cone_trace evaluates one surface point (one launch), cone_trace_batch many.
void cone_trace_init_filter(VoxelOctree* root);
Vec3 cone_trace(const VoxelOctree& root, const ISect& isect, float min_voxel_size);
void cone_trace_batch(const VoxelOctree& root, const std::vector<ISect>& isects, float min_voxel_size,
                      std::vector<Vec3>* out);

// Replicas of a built octree on several devices (vrt_mgpu_*; a device may be listed more than once), for main.cc's
// GI statements on N GPUs: light_map_gpu / cone_trace_init_filter / render_gi_gpu below take one in place of the
// root.  The replicas hold the geometry only; the light pass runs on each of them.  Owns the vrt_mgpu*.
class MultiGpu {
public:
        MultiGpu(const VoxelOctree* root, const std::vector<int>& devices);
        ~MultiGpu();
        MultiGpu(const MultiGpu&) = delete;
        MultiGpu& operator=(const MultiGpu&) = delete;
        vrt_mgpu* native() const { return m_; }
        int num_devices() const { return vrt_mgpu_num_devices(m_); }

private:
        vrt_mgpu* m_ = nullptr;
};
void cone_trace_init_filter(MultiGpu& replicas);

// Animated geometry (vrt_update_triangles / vrt_update_xform): move the triangles of a built octree and revoxelise.
// tri_xyz and tri_nrm hold 9 floats per triangle in the order of the voxels given to ray_march_init (tri_nrm: the
// normals as Triangle stores them, or empty exactly when the octree has no input normals); xf ranges index that
// order too.  The VoxelBase objects stay the caller's and are not changed.  max_depth 0: the current depth.  The
// root box and the leaf set ray_march reads follow the new octree; leaf pointers from earlier calls are invalid.
// The GI state is dropped: light the scene again (light_map_gpu, cone_trace_init_filter).
void update_triangles_gpu(VoxelOctree* root, const std::vector<float>& tri_xyz, const std::vector<float>& tri_nrm,
                          int max_depth = 0);
void transform_gpu(VoxelOctree* root, const std::vector<vrt_xform>& xf, int max_depth = 0);
// the same on the replicas (every replica ends up with the first one's octree); max_depth is required
void update_triangles_gpu(MultiGpu& replicas, const std::vector<float>& tri_xyz, const std::vector<float>& tri_nrm,
                          int max_depth);
void transform_gpu(MultiGpu& replicas, const std::vector<vrt_xform>& xf, int max_depth);
}  // namespace gi

class Film {  // camera.h:24-39 -- storage is y*nx+x (the reference's y*ny+x is only right for nx==ny)
public:
        const float w, h;
        const int nx, ny;
        Film(float w, float h, int nx, int ny);
        jql::Vec3 get(int x, int y) const { return data_[(size_t)y * nx + x]; }
        void set(int x, int y, const jql::Vec3& c) { data_[(size_t)y * nx + x] = c; }
        void add(int x, int y, const jql::Vec3& c);
        std::vector<std::uint8_t> to_byte_array() const;
        std::vector<float> to_float_array() const;
        jql::Vec3* data() { return data_.data(); }

private:
        std::vector<jql::Vec3> data_;
};

class Camera {  // camera.h:70-83
public:
        const float fov;
        const float near;
        const float far;
        Camera(float fov, jql::Vec3 eye, jql::Vec3 spot, jql::Vec3 up, float near = 0,
               float far = std::numeric_limits<float>::max());
        std::vector<jql::Ray> gen_rays1(const Film& film, int px, int py);
        std::vector<jql::Ray> gen_rays4(const Film& film, int px, int py);
        // whole-film forms used by the GPU render loop
        vrt_camera native(const Film& film, int spp) const;

private:
        float cam10_[10];
};

// Replacement of the two render_mt loops of main.cc (camera.h:41-68): one launch for the
// whole film.  hits (optional) receives film.nx*film.ny*spp records, row-major by pixel,
// then sample.  The film receives the harness pixel (sky / kd*n.l, SURVEY.md 8d).
void render_gpu(Film* film, Camera& cam, gi::VoxelOctree* root, int spp, const jql::Vec3& light_dir, float kd,
                std::vector<vrt_hit>* hits = nullptr);

// Replacement of the light-map render_mt loop of main.cc:81-96: every sample of the light camera's
// film splats clamp(dot(illum_d[i], n)) * get_diffuse(...) into its leaf, in the sequential loop
// order (deterministic; the reference races here).  kd = the material's diffuse colour.
void light_map_gpu(const Film& sfilm, Camera& scam, gi::VoxelOctree* root, int spp, const jql::Vec3& kd);
// Replacement of the final render_mt loop of main.cc:117-123 (trace() per sample, film += c / spp).
void render_gi_gpu(Film* film, Camera& cam, gi::VoxelOctree* root, int spp, const jql::Vec3& kd, float res);
// The same two statements on the replicas of a gi::MultiGpu: the light map is splatted on every replica, and the
// film's 8-row bands are dealt round-robin to the devices, each copying its bands straight into film->data().
// Both return when the work is done; the film equals the single-device one bytewise.
void light_map_gpu(const Film& sfilm, Camera& scam, gi::MultiGpu& replicas, int spp, const jql::Vec3& kd);
void render_gi_gpu(Film* film, Camera& cam, gi::MultiGpu& replicas, int spp, const jql::Vec3& kd, float res);

namespace gi {
// What main.cc's GI film is made of, per pixel (vrt_gi_aov in include/vrt.h): the sample means of the albedo, the
// leaf's direct light, the cone-traced indirect light and the ISect normal (a miss adds 0), and the 16-byte hit
// record of every sample.  Every member is optional (nullptr: not written).
struct GiAov {
        Film* albedo = nullptr;
        Film* direct = nullptr;
        Film* indirect = nullptr;
        Film* normal = nullptr;
        std::vector<vrt_hit16>* hits = nullptr;  // resized to nx * ny * spp (pixel row-major, then sample)
};
}  // namespace gi
// render_gi_gpu plus the planes of `aov`, from one launch.  film_or_null (when given) receives the same film as
// render_gi_gpu; the film and the float planes must have one size, and at least one of them gives the camera's film
// geometry.
void render_gi_aov_gpu(Film* film_or_null, Camera& cam, gi::VoxelOctree* root, int spp, const jql::Vec3& kd, float res,
                       gi::GiAov& aov);
// The same on the replicas of a gi::MultiGpu: 8-row bands dealt round-robin, each device copying its bands straight
// into the film and the planes (page-locked for the call).  Returns when the work is done; every output equals the
// single-device one bytewise.
void render_gi_aov_gpu(Film* film_or_null, Camera& cam, gi::MultiGpu& replicas, int spp, const jql::Vec3& kd, float res,
                       gi::GiAov& aov);

// Materials for the GI passes (the half of gi::Triangle the geometry mirror leaves out: t_[3] and
// tinyobj::material_t::diffuse / diffuse_texname, voxel_octree.h:110-111).  uv holds three texture
// coordinates per triangle in the order of the voxels given to ray_march_init; a material with
// texture < 0 is untextured.  Texture bytes are what stbi_load returns (row 0 = top).
struct GpuMaterial {
        jql::Vec3 diffuse;
        int texture;  // index into the textures, or -1
};
struct GpuTexture {
        int width, height, channels;
        const std::uint8_t* data;
};
void set_materials_gpu(gi::VoxelOctree* root, const std::vector<jql::Vec2>& uv, const std::vector<std::uint32_t>& tri_material,
                       const std::vector<GpuMaterial>& materials, const std::vector<GpuTexture>& textures);
// the same materials on every replica
void set_materials_gpu(gi::MultiGpu& replicas, const std::vector<jql::Vec2>& uv, const std::vector<std::uint32_t>& tri_material,
                       const std::vector<GpuMaterial>& materials, const std::vector<GpuTexture>& textures);

// tribox2.h:15 and raytri.h:5-7 -- same signatures, evaluated on the GPU.
int triBoxOverlap(float boxcenter[3], float boxhalfsize[3], float triverts[3][3]);
int intersect_triangle3(double orig[3], double dir[3], double vert0[3], double vert1[3], double vert2[3], double* t,
                        double* u, double* v);

#endif  // VRT_GI_H
