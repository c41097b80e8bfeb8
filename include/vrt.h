/* include/vrt.h -- C ABI of libvrt.so, the B200 (sm_100a) implementation of the
 * sparse-voxel-octree hot path of jqly/VoxelRayTrace20190722.
 *
 * The reference has no FFI layer; its boundary for this path is the C++
 * function surface below (paths relative to VoxelRayTrace20190722/).  Each
 * entry point names the reference interface it replaces.  C++ adapters with
 * the reference's exact signatures live in
 * voxelraytrace20190722_b200/cpp/vrt_gi.{h,cc}; INTEGRATION.md shows how
 * main.cc binds to them.
 *
 * Conventions
 *   - every function returns VRT_OK (0) or a negative vrt_status; the message
 *     of the last failure on the calling thread is vrt_last_error().  Nothing
 *     in the library calls exit()/abort() (the reference does: voxel_octree.cc:329).
 *   - handles (vrt_tree*) are allocated and freed by the library; every `out`
 *     buffer is caller-allocated; input arrays are borrowed for the call only.
 *   - functions without a suffix take HOST pointers, copy in/out inside the call
 *     and return when the result is in the caller's buffer; functions ending in
 *     _dev take DEVICE pointers (current CUDA device) and only ENQUEUE work on the
 *     tree's stream (vrt_tree_sync / vrt_last_kernel_ms wait for it).
 *   - there is no CPU fallback: without a usable CUDA device every compute
 *     entry point fails with VRT_ERR_CUDA.
 *   - triangle index == index into tri_xyz == OBJ face order
 *     (voxel_octree.cc:334-368); it is the tie-break key of the reference.
 *   - max_depth is the reference's 1-based depth (voxel_octree.cc:74):
 *     leaves live at level max_depth-1, leaf grid = 2^(max_depth-1) per axis.
 */
#ifndef VRT_H
#define VRT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* libvrt.so is built with -fvisibility=hidden; only this header is exported. */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define VRT_ABI_VERSION 1

typedef enum vrt_status {
        VRT_OK = 0,
        VRT_ERR_ARG = -1,      /* bad argument (null pointer, depth out of range, ...) */
        VRT_ERR_CUDA = -2,     /* CUDA runtime failure or no device                    */
        VRT_ERR_NOMEM = -3,    /* device or host allocation failed                     */
        VRT_ERR_CAPACITY = -4, /* key packing does not fit 64 bit (T, depth too large) */
        VRT_ERR_STATE = -5     /* handle not built / wrong device                      */
} vrt_status;

#define VRT_MAX_DEPTH 17u      /* 1-based; 3*(max_depth-1) Morton bits + tri bits <= 64 */
#define VRT_NO_TRI 0xffffffffu

typedef struct vrt_tree vrt_tree;

/* jql::Ray (graphics_math.h:1150-1167), 32 bytes, copied verbatim: d is NOT
 * re-normalised by the library (the reference normalises in the Ray ctor; a
 * caller that builds rays through vrt_gen_rays gets that for free). */
typedef struct vrt_ray {
        float o[3];
        float d[3];
        float tmin;
        float tmax;
} vrt_ray;

/* Result of gi::ray_march (voxel_octree.h:87-89) for one ray.  48 bytes.
 * (leaf_ptr, voxel_ptr, ISect) -> (cell, tri, pos/nrm); `t` is (float)dt of
 * Triangle::isect (voxel_octree.cc:454). */
typedef struct vrt_hit {
        uint32_t hit;      /* 1 = ray_march returned true                        */
        uint32_t tri;      /* index of *voxel_ptr in the input array, VRT_NO_TRI  */
        uint32_t cell[3];  /* *leaf_ptr as cell coordinates at level max_depth-1  */
        float t;
        float pos[3];      /* ISect::hit                                          */
        float nrm[3];      /* ISect::normal                                       */
} vrt_hit;

/* Compact per-ray record (16 bytes) -- the "hit record" SURVEY.md 8(d) counts. */
typedef struct vrt_hit16 {
        uint32_t leaf;     /* index into the Morton-sorted leaf array, VRT_NO_TRI on miss */
        uint32_t tri;
        float t;
        uint32_t hit;
} vrt_hit16;

/* Camera as the reference constructs it: Camera(fov,eye,spot,up) camera.cc:65-75
 * + Film(w,h,nx,ny) camera.h:24-29.  C is the column-major camera-to-world
 * matrix C_ (private member of the reference's Camera); z is
 * -(film_h/(2*tanf(fov/2))) (camera.cc:82,100) -- tanf stays on the host. */
typedef struct vrt_camera {
        float C[16];
        float z;
        float tmin, tmax;  /* Camera::near / Camera::far (camera.h:76-77): 0, FLT_MAX */
        int32_t nx, ny;    /* film resolution                                         */
        int32_t spp;       /* 1 = gen_rays1, 4 = gen_rays4                            */
} vrt_camera;

typedef struct vrt_tree_info {
        uint32_t num_tris;
        int32_t max_depth;
        float root_aabb[6];    /* min xyz, max xyz (voxel_octree.cc:70-72)             */
        uint64_t num_nodes;    /* non-empty nodes, all levels (interior + leaves)      */
        uint64_t num_leaves;   /* non-empty leaves at level max_depth-1                */
        uint64_t num_refs;     /* sum of leaf triangle-list lengths                    */
        uint64_t level_offset[VRT_MAX_DEPTH + 1]; /* node index range of each level   */
        uint64_t device_bytes; /* HBM held by the handle                               */
        double build_ms;       /* device time of the last vrt_build (CUDA events)      */
} vrt_tree_info;

/* Host view of the flat octree (caller-allocated arrays, sizes from vrt_tree_info):
 *   leaf_cell [num_leaves][3]  cell coordinates, Morton (= reference child) order
 *   leaf_count[num_leaves]     triangles per leaf
 *   leaf_refs [num_refs]       triangle indices, ascending inside each leaf
 *   nodes     [num_nodes][2]   {child_mask | first_child<<?} see DESIGN.md; may be NULL
 */
typedef struct vrt_tree_view {
        uint32_t* leaf_cell;
        uint32_t* leaf_count;
        uint32_t* leaf_refs;
        uint32_t* nodes;
} vrt_tree_view;

/* ---- library ------------------------------------------------------------- */
int vrt_abi_version(void);
const char* vrt_last_error(void);
/* number of CUDA devices visible; <0 on failure */
int vrt_device_count(void);
/* kernels launched by this process so far (bench.py's gpu_launches claim) */
uint64_t vrt_launch_count(void);

/* ---- build: replaces gi::ray_march_init (voxel_octree.h:85-86,
 *      voxel_octree.cc:67-75) + Triangle ctor/get_aabb/is_overlap
 *      (voxel_octree.cc:423-436,486-492) + triBoxOverlap (tribox2.cc:112) ----
 * tri_nrm may be NULL (geometric normal cross(p1-p0,p2-p0) per triangle). */
int vrt_build(const float* tri_xyz, const float* tri_nrm, uint32_t num_tris,
              int max_depth, vrt_tree** out);
int vrt_build_dev(const float* d_tri_xyz, const float* d_tri_nrm, uint32_t num_tris,
                  int max_depth, vrt_tree** out);
/* vrt_build with flags.  VRT_BUILD_UNIT_NORMALS: tri_nrm holds Triangle::n_ as the reference's Triangle
 * objects store it (already normalised by the ctor, voxel_octree.cc:426) and is kept verbatim -- what a
 * binding that reads existing gi::Triangle objects must pass (cpp/vrt_dropin.cc). */
#define VRT_BUILD_UNIT_NORMALS 1u
int vrt_build_ex(const float* tri_xyz, const float* tri_nrm, uint32_t num_tris, int max_depth,
                 uint32_t flags, vrt_tree** out);
/* Indexed ingest (obj2voxel, voxel_octree.cc:305-371): the arrays tinyobj::LoadObj returns --
 * attrib.vertices[num_vertices][3], attrib.normals[num_normals][3] (NULL: geometric normals) and the
 * per-face-vertex tinyobj::index_t records index3[T][3] = {vertex_index, normal_index,
 * texcoord_index} -- are uploaded as they are and gathered into triangles on the device. */
int vrt_build_indexed(const float* vertices, uint64_t num_vertices, const float* normals,
                      uint64_t num_normals, const int32_t* index3, uint32_t num_tris, int max_depth,
                      vrt_tree** out);
/* Re-run the build on the triangles already held by the handle (timing loops). */
int vrt_rebuild(vrt_tree* tree, int max_depth);
void vrt_tree_free(vrt_tree* tree);
int vrt_tree_get_info(const vrt_tree* tree, vrt_tree_info* out);
int vrt_tree_export(const vrt_tree* tree, vrt_tree_view* out);
/* Build a handle from an externally produced leaf set (e.g. the oracle's tree):
 * lets the ray kernel be checked independently of the voxelizer. */
int vrt_tree_import(const float* tri_xyz, const float* tri_nrm, uint32_t num_tris,
                    int max_depth, const float root_aabb[6], uint64_t num_leaves,
                    const uint32_t* leaf_cell, const uint32_t* leaf_count,
                    const uint32_t* leaf_refs, vrt_tree** out);
/* Use `stream` (a cudaStream_t) for all work of this handle; NULL = default. */
int vrt_tree_set_stream(vrt_tree* tree, void* stream);

/* Raw device arrays of a built tree, for replication over NCCL (SURVEY.md 8e):
 * blob = one contiguous device allocation holding everything the ray kernel
 * reads; a replica is created from a received copy with vrt_tree_from_blob_dev. */
int vrt_tree_blob_dev(const vrt_tree* tree, const void** d_blob, uint64_t* bytes);
int vrt_tree_from_blob_dev(const void* d_blob, uint64_t bytes, vrt_tree** out);

/* Checkpoint of a built octree (SURVEY.md 5: the reference rebuilds its tree on every run;
 * the flat blob IS a serialisable format): the whole device blob, byte for byte. */
int vrt_tree_save(const vrt_tree* tree, const char* path);
int vrt_tree_load(const char* path, vrt_tree** out);

/* ---- ray generation: replaces Camera::Camera + gen_rays1/gen_rays4
 *      (camera.cc:65-112) ---------------------------------------------------- */
/* cam10 = fov, eye[3], spot[3], up[3]; fills C, z, tmin/tmax (host arithmetic,
 * identical to the reference ctor). */
int vrt_camera_init(const float cam10[10], float film_h, int nx, int ny, int spp,
                    vrt_camera* out);
/* rays_out[(y1-y0)][(x1-x0)][spp] */
int vrt_gen_rays(const vrt_camera* cam, int x0, int y0, int x1, int y1,
                 vrt_ray* rays_out);

/* ---- query: replaces gi::ray_march (voxel_octree.cc:131-188) and the
 *      render_mt pixel loop (camera.h:41-68) --------------------------------- */
int vrt_trace_rays(const vrt_tree* tree, const vrt_ray* rays, uint64_t num_rays,
                   vrt_hit* out);
int vrt_trace_rays_dev(const vrt_tree* tree, const vrt_ray* d_rays, uint64_t num_rays,
                       vrt_hit* d_out);
/* Ray generation fused into the traversal kernel; pixel rectangle [x0,x1)x[y0,y1);
 * out[(y1-y0)][(x1-x0)][spp]. */
int vrt_trace_camera(const vrt_tree* tree, const vrt_camera* cam, int x0, int y0,
                     int x1, int y1, vrt_hit* out);
int vrt_trace_camera_dev(const vrt_tree* tree, const vrt_camera* cam, int x0, int y0,
                         int x1, int y1, vrt_hit* d_out);
int vrt_trace_camera16_dev(const vrt_tree* tree, const vrt_camera* cam, int x0, int y0,
                           int x1, int y1, vrt_hit16* d_out);

/* Harness pixel (SURVEY.md 8d): miss -> sky lerp of main.cc:18-20; hit ->
 * kd*clamp(dot(normal,light),0,1); spp samples * (1/spp) accumulated in sample
 * order (main.cc:119-122).  film_rgb[(y1-y0)][(x1-x0)][3] float. */
typedef struct vrt_shade {
        float light_dir[3]; /* normalised on the host, main.cc:72 */
        float kd;
        float shadow_eps;   /* shadow ray origin = hit + shadow_eps * normal              */
        int32_t shadow;     /* 1: one shadow ray per hit toward light_dir (config 5 of
                               BASELINE.json; harness-defined, same ray_march semantics) */
} vrt_shade;
int vrt_render_camera(const vrt_tree* tree, const vrt_camera* cam, const vrt_shade* sh,
                      int x0, int y0, int x1, int y1, float* film_rgb);
int vrt_render_camera_dev(const vrt_tree* tree, const vrt_camera* cam,
                          const vrt_shade* sh, int x0, int y0, int x1, int y1,
                          float* d_film_rgb);
/* Frame-sequence form of vrt_render_camera: returns once the frame is ENQUEUED; the
 * kernel of the next frame overlaps this frame's device->host copy (two device films, a
 * copy stream).  film_rgb should be pinned host memory and must stay valid until
 * vrt_tree_sync() returns; alternate between (at least) two host buffers. */
int vrt_render_camera_async(const vrt_tree* tree, const vrt_camera* cam,
                            const vrt_shade* sh, int x0, int y0, int x1, int y1,
                            float* film_rgb);
/* Film export encodings, fused into the store of a finished pixel (every film-writing entry point of the handle:
 * vrt_render_camera*, vrt_render_bands*, vrt_frame_bands*, vrt_gi_render_camera*, vrt_gi_render_bands_async,
 * vrt_mgpu_render*, vrt_mgpu_gi_render*).  The reference
 * keeps a float film and converts it after the render loop; on a multi-GPU node the float film is what saturates
 * the host's device->host ingest, so the conversion runs in the ray kernel and the encoded film crosses PCIe:
 *   VRT_FILM_F32   [ny][nx][3] float            Film::to_float_array, camera.cc:50-63 (default)
 *   VRT_FILM_RGBE  [ny][nx][4] uint8 (R,G,B,E)  the pixel encoding stbi_write_hdr applies to that array
 *                                               (main.cc:125-126; stbiw__linear_to_rgbe, stb_image_write.h:601-616);
 *                                               vrt_hdr_file() turns it into the bytes of test2.hdr
 *   VRT_FILM_RGB8  [ny][nx][3] uint8            Film::to_byte_array, camera.cc:27-48 (v * 255.9f, cast to uint8)
 * With a format other than F32 the `float*` film arguments address bytes of that layout. */
typedef enum vrt_film_format { VRT_FILM_F32 = 0, VRT_FILM_RGBE = 1, VRT_FILM_RGB8 = 2 } vrt_film_format;
int vrt_set_film_format(vrt_tree* tree, int32_t format);
int vrt_film_pixel_bytes(int32_t format); /* 12 / 4 / 3, or VRT_ERR_ARG */
/* The same encodings applied on the device to a float film the caller already holds (host pointers;
 * format = VRT_FILM_RGBE or VRT_FILM_RGB8; out = npix * vrt_film_pixel_bytes(format) bytes). */
int vrt_film_encode(const vrt_tree* tree, const float* film_rgb, uint64_t npix, int32_t format, uint8_t* out);
/* The file stbi_write_hdr(name, nx, ny, 3, film) writes (stb_image_write.h:635-740: header, then per scanline the
 * 4-byte marker and the four components run-length encoded separately; flat pixels for nx < 8 or nx >= 32768),
 * from the RGBE film.  Host code, no device involved.  Returns the number of bytes of the file, which are written
 * to `out` if cap is large enough (call with cap = 0 to size the buffer); negative vrt_status on bad arguments. */
int64_t vrt_hdr_file(const uint8_t* film_rgbe, int32_t nx, int32_t ny, uint8_t* out, uint64_t cap);
/* Row-interleaved shard of the film for multi-GPU runs (SURVEY.md 8e; replaces the
 * static 8x8 tile split of render_mt, camera.h:45-55): the film is cut into bands
 * of band_h rows; the call renders bands band_first, band_first+band_stride, ...
 * over the full film width and writes them compactly, out[local_row][nx][...]
 * with vrt_band_rows() local rows. */
typedef struct vrt_bands {
        int32_t band_h;
        int32_t band_first;
        int32_t band_stride;
} vrt_bands;
int vrt_band_rows(const vrt_camera* cam, const vrt_bands* bands);
int vrt_render_bands_dev(const vrt_tree* tree, const vrt_camera* cam, const vrt_shade* sh,
                         const vrt_bands* bands, float* d_film_rgb);
int vrt_trace_bands16_dev(const vrt_tree* tree, const vrt_camera* cam,
                          const vrt_bands* bands, vrt_hit16* d_out);
/* The multi-GPU form of vrt_render_camera_async (render_mt camera.h:41-68 with the film in
 * host memory): film_rgb_full is the FULL [ny][nx][3] host frame -- on a multi-process node a
 * shared mapping that every rank has pinned (cudaHostRegister) -- and this rank's bands are
 * DMA-copied straight to their final rows, asynchronously (two device band buffers per handle:
 * the copy of frame k overlaps the kernel of frame k+1).  vrt_tree_sync() on every rank, then a
 * process barrier, and the frame is complete.  Alternate between two host frames. */
int vrt_render_bands_async(const vrt_tree* tree, const vrt_camera* cam, const vrt_shade* sh,
                           const vrt_bands* bands, float* film_rgb_full);
/* Single-process multi-GPU render for C / C++ hosts (the thread pool of render_mt, camera.h:41-68, becomes N
 * devices): replicate a built octree onto `num_devices` devices (devices == NULL: 0..num_devices-1; peer copies of
 * the blob), then per frame deal the film's 8-row bands round-robin to the devices.  Every device runs the
 * vrt_render_bands_async pipeline and DMA-copies its bands to their final rows of film_rgb_full (pinned host
 * memory, e.g. vrt_host_register'ed); vrt_mgpu_sync (or the synchronous vrt_mgpu_render) completes the frame.
 * The source tree stays the caller's and may be freed after vrt_mgpu_create.  vrt_mgpu_create copies the
 * geometry only; materials and the GI state of the replicas are set through the vrt_mgpu_* GI calls below. */
typedef struct vrt_mgpu vrt_mgpu;
int vrt_mgpu_create(const vrt_tree* tree, int num_devices, const int* devices, vrt_mgpu** out);
int vrt_mgpu_num_devices(const vrt_mgpu* m);
int vrt_mgpu_set_film_format(vrt_mgpu* m, int32_t format); /* vrt_set_film_format on every replica */
int vrt_mgpu_render_async(vrt_mgpu* m, const vrt_camera* cam, const vrt_shade* sh, float* film_rgb_full);
int vrt_mgpu_sync(vrt_mgpu* m);
int vrt_mgpu_render(vrt_mgpu* m, const vrt_camera* cam, const vrt_shade* sh, float* film_rgb_full);
void vrt_mgpu_free(vrt_mgpu* m);
/* Work counters of the reference algorithm for a camera frame (SURVEY.md 8d):
 * counts[0..4] = rays traced, interior nodes expanded (travorder calls), non-empty
 * leaves visited, triangle tests, hits; counts[5..7] = kernel statistics: expansions done
 * by the parametric fast path, slab fallbacks caused by a tie, slab expansions at levels
 * that are not key-safe for the ray.  Host pointer out. */
int vrt_count_camera(const vrt_tree* tree, const vrt_camera* cam, int x0, int y0, int x1,
                     int y1, uint64_t counts[8]);
/* One frame step of the multi-GPU render loop: this rank's bands, writing BOTH the
 * compact per-ray hit records (kept sharded in this GPU's HBM) and the shaded film
 * bands (the piece the framebuffer gather collects).  d_hits[local_row][nx][spp],
 * d_film_rgb[local_row][nx][3]. */
int vrt_frame_bands_dev(const vrt_tree* tree, const vrt_camera* cam, const vrt_shade* sh,
                        const vrt_bands* bands, vrt_hit16* d_hits, float* d_film_rgb);
/* Same step with the framebuffer assembly FUSED into the ray kernel (SURVEY.md 5/8e,
 * the alternative to gather): d_frame_rgb is the FULL [ny][nx][3] frame, normally rank
 * 0's buffer mapped into this process with vrt_ipc_open, and the kernel stores every
 * finished pixel straight to its final place over NVLink (peer stores; no NCCL, no
 * staging, no re-order pass).  On rank 0 / a single GPU it is just a local pointer. */
int vrt_frame_bands_peer_dev(const vrt_tree* tree, const vrt_camera* cam, const vrt_shade* sh,
                             const vrt_bands* bands, vrt_hit16* d_hits, float* d_frame_rgb);
/* Plain device memory that can be shared between the processes of one node
 * (cudaMalloc + CUDA IPC): export a 64-byte handle on the owner, open it on the peers. */
int vrt_dev_alloc(uint64_t bytes, void** d_ptr);
int vrt_dev_free(void* d_ptr);
/* Page-lock a host range for DMA (e.g. a frame in POSIX shared memory that all ranks of a node
 * map: the target of vrt_render_bands_async). */
int vrt_host_register(void* ptr, uint64_t bytes);
int vrt_host_unregister(void* ptr);
int vrt_ipc_export(const void* d_ptr, uint8_t handle[64]);
int vrt_ipc_open(const uint8_t handle[64], void** d_ptr);
int vrt_ipc_close(void* d_ptr);
/* Test hook: how many node expansions of this process took the general (>4 candidate
 * children) ordering path of the ray kernel. */
uint64_t vrt_debug_general_order_calls(void);
/* ---- GI rows (SURVEY.md 8f "next"): light-map splat (main.cc:75-97), cone_trace_init_filter
 *      and cone_trace (voxel_octree.cc:190-303), the final trace() pixel (main.cc:10-30).
 *      One untextured material: kd = tinyobj material_t::diffuse (voxel_octree.cc:474-476).
 *      Per-node state (coverage, illum[6]) lives beside the node array; it belongs to one
 *      build: call vrt_gi_init again after vrt_rebuild, vrt_update_triangles(_dev) or
 *      vrt_update_xform (and their vrt_mgpu_* forms).
 *      `res` (cone_trace's min_voxel_size) must be finite and >= FLT_MIN: every entry point
 *      that takes it returns VRT_ERR_ARG otherwise, before it looks at its other arguments.
 *      For a normal res every step of a cone grows its distance by at least 11.5 %, so the
 *      march ends (in about 1,600 steps even for res = FLT_MIN and an infinite root box); for
 *      0, a negative or a subnormal res the distance stops advancing and the march never ends.
 *      main.cc's Res (min over axes of root size / 2^max_depth) is 0 for a planar scene: take
 *      the minimum over the axes of non-zero size. ------------------------------------------ */
/* Materials (Triangle::get_albedo, voxel_octree.cc:471-484): tri_uv[T][3][2] per-vertex texture
 * coordinates, tri_mtl[T] material ids, per material kd[m][3] (tinyobj material_t::diffuse) and
 * mtl_tex[m] = index into tex[] or -1 (empty diffuse_texname).  Textures are the bytes stbi_load
 * returns (row 0 = top, `channels` interleaved).  Without this call every triangle has the colour
 * passed to the GI entry points.  Host pointers; the data is copied. */
typedef struct vrt_texture {
        int32_t width, height, channels;
        const uint8_t* data;
} vrt_texture;
int vrt_set_materials(vrt_tree* tree, const float* tri_uv, const uint32_t* tri_mtl, uint32_t num_mtl,
                      const float* kd, const int32_t* mtl_tex, uint32_t num_tex, const vrt_texture* tex);
/* Triangle::get_albedo(ISect{hit = pos[i]}) of triangle tri[i] (barycentric + unit_cycle + nearest
 * texel with the vertical flip, texel_fetch voxel_octree.cc:401-422); host pointers */
int vrt_albedo(const vrt_tree* tree, const uint32_t* tri, const float* pos, uint64_t n,
               const float kd_default[3], float* out_rgb);
/* allocate + zero the per-node GI state (VoxelOctree::coverage / illum, voxel_octree.h:66-70) */
int vrt_gi_init(vrt_tree* tree);
/* The light-map lambda of main.cc:81-96 for every sample of the light camera's film:
 * leaf.illum[i] += clamp(dot(illum_d[i], normal),0,1) * get_diffuse(isect, ray, (1,1,1)).
 * Contributions are added per leaf in the order of the sequential loop (py, px, sample), which
 * makes the result deterministic (the reference races on the += from its pool threads). */
int vrt_gi_splat_camera(vrt_tree* tree, const vrt_camera* light_cam, const float kd[3]);
/* gi::cone_trace_init_filter(root): coverage 1 on non-empty leaves, parents = child sum / 8 */
int vrt_gi_filter(vrt_tree* tree);
/* host copies of one level's state, node order (= Morton order): coverage[n], illum18[n][6][3];
 * n = level_offset[level+1] - level_offset[level] (vrt_tree_get_info) */
int vrt_gi_get_level(const vrt_tree* tree, int level, float* coverage, float* illum18);
/* gi::cone_trace(root, ISect{hit=pos, normal=nrm}, res) for n surface points; host pointers */
int vrt_gi_cone_trace(const vrt_tree* tree, const float* pos, const float* nrm, uint64_t n, float res,
                      float* out_rgb);
/* The final image loop of main.cc:117-123: per sample trace() = sky | albedo * (cone_trace +
 * leaf.compute_illum(-ray.d)), film += colour / spp.  film_rgb[(y1-y0)][(x1-x0)][3]. */
int vrt_gi_render_camera(const vrt_tree* tree, const vrt_camera* cam, const float kd[3], float res, int x0,
                         int y0, int x1, int y1, float* film_rgb);
int vrt_gi_render_camera_dev(const vrt_tree* tree, const vrt_camera* cam, const float kd[3], float res,
                             int x0, int y0, int x1, int y1, float* d_film_rgb);
/* The GI film of vrt_gi_render_camera in the banded, pipelined form of vrt_render_bands_async: this handle's
 * bands of the film are cone-traced into one of two device band buffers (kernels alternating between two
 * streams) and DMA-copied to their final rows of film_rgb_full, the FULL [ny][nx][...] host frame in the
 * handle's film format (pinned; on a multi-process node a shared mapping every rank has registered).  kd is a
 * host pointer.  Returns once the frame is ENQUEUED; the frame is complete after vrt_tree_sync() (and, with
 * several ranks, a process barrier).  Requires vrt_gi_init (VRT_ERR_ARG otherwise).  bands = {ny, 0, 1} is the
 * single-GPU pipelined GI loop (main.cc:117-123 frame after frame): alternate between two host frames.
 * vrt_set_materials, vrt_gi_init, vrt_gi_splat_camera and vrt_gi_filter may be called between enqueued frames
 * without a vrt_tree_sync: they run after every frame enqueued before them and before every frame after. */
int vrt_gi_render_bands_async(const vrt_tree* tree, const vrt_camera* cam, const float kd[3], float res,
                              const vrt_bands* bands, float* film_rgb_full);
/* What the GI film is made of: the per-pixel planes of one vrt_gi_render_camera launch (for a denoiser's albedo and
 * normal guides, a compositor, or tuning octree depth, light-film resolution and textures).  For a sample that hits,
 * with d the ray direction, the library computes exactly the terms the film is built from:
 *   A  albedo    Triangle::get_albedo at the hit, kd the untextured colour (what vrt_albedo returns);
 *   I  indirect  gi::cone_trace(root, isect, res), six cones (what vrt_gi_cone_trace returns);
 *   D  direct    the hit leaf's VoxelOctree::compute_illum(-d) (voxel_octree.h:71-81);
 *   N  normal    the ISect normal the cone basis is built from;
 * and the film sample is A * (I + D).  A miss adds +0 to every plane; the sky goes into the film only.
 * Every float plane is [(y1-y0)][(x1-x0)][3] float32 whatever the film format, accumulated like the film
 * (main.cc:119-122): acc = +0, then acc += v_s * (1/spp) in sample order, so the normal plane is the sample mean and
 * is not renormalised.  hits is [(y1-y0)][(x1-x0)][spp] vrt_hit16, bytewise the records of the 16-byte camera
 * trace for the same camera and rectangle.  Every member is optional (NULL: not written). */
typedef struct vrt_gi_aov {
        float* albedo;    /* [rows][cols][3] */
        float* direct;    /* [rows][cols][3] */
        float* indirect;  /* [rows][cols][3] */
        float* normal;    /* [rows][cols][3] */
        vrt_hit16* hits;  /* [rows][cols][spp] */
} vrt_gi_aov;
/* The GI film of the camera-film GI call plus any of the planes above, in one launch.  The film (in the handle's
 * film format, bytewise that call's film) may be NULL; a request with every plane NULL is VRT_ERR_ARG (the film
 * alone is that call).  Otherwise requirements and errors are those of the camera-film GI call: vrt_gi_init first,
 * and a rectangle outside the film is VRT_ERR_ARG.  The first form takes host pointers and returns when they are
 * filled; the _dev form takes device pointers and is enqueued on the handle's stream (with that stream's cone-trace
 * step table, like the _dev camera-film GI call). */
int vrt_gi_render_aov(const vrt_tree* tree, const vrt_camera* cam, const float kd[3], float res, int x0, int y0,
                      int x1, int y1, float* film_or_null, const vrt_gi_aov* aov);
int vrt_gi_render_aov_dev(const vrt_tree* tree, const vrt_camera* cam, const float kd[3], float res, int x0, int y0,
                          int x1, int y1, float* d_film_or_null, const vrt_gi_aov* d_aov);
/* The GI film and its planes (vrt_gi_render_aov) in the banded, pipelined form of vrt_gi_render_bands_async, for a
 * denoiser or compositor that reads the planes in host memory every frame.  aov_full holds HOST pointers to FULL
 * frames: each float plane [ny][nx][3] float32, hits [ny][nx][spp] vrt_hit16, and film_full_or_null (NULL: no film)
 * [ny][nx][...] in the handle's film format.  This handle's bands of every non-NULL output are rendered by one launch
 * into one of two device buffers and DMA-copied to their final rows; every other byte of those frames, and every
 * NULL member, is left untouched.  Every byte written equals vrt_gi_render_aov for the same camera, kd, res, film
 * format and GI state; the film is bytewise vrt_gi_render_bands_async's.  The frames should be pinned (on a
 * multi-process node: shared mappings every rank has registered) and stay valid until vrt_tree_sync; the
 * vrt_gi_aov struct, cam and kd are read during the call only.  A request with every plane NULL is VRT_ERR_ARG
 * (the film alone is vrt_gi_render_bands_async); so are a missing vrt_gi_init, bad bands and a NULL cam, kd or
 * aov_full.  A handle with no rows in `bands` returns VRT_OK and enqueues nothing, and a rejected call enqueues
 * nothing.  The frames share the pipeline (two kernel streams, one copy stream) of vrt_render_camera_async,
 * vrt_render_bands_async and vrt_gi_render_bands_async, so the four calls may be interleaved on one handle, and
 * the light-map calls may be issued between enqueued frames without a sync, as for vrt_gi_render_bands_async. */
int vrt_gi_render_aov_bands_async(const vrt_tree* tree, const vrt_camera* cam, const float kd[3], float res,
                                  const vrt_bands* bands, float* film_full_or_null, const vrt_gi_aov* aov_full);
/* The GI rows on the replicas of a vrt_mgpu (main.cc:75-126 over N devices).  vrt_mgpu_create copies the
 * geometry only: materials and the GI state are set through these calls, each of which runs the single-device
 * call on every replica (host pointers, like the single-device calls).  The light pass runs on every replica --
 * the splat is deterministic, so every replica holds the same bits -- and the replicas work concurrently.
 *   vrt_mgpu_set_materials    vrt_set_materials on every replica
 *   vrt_mgpu_gi_init          vrt_gi_init                  (main.cc:75)
 *   vrt_mgpu_gi_splat_camera  vrt_gi_splat_camera          (main.cc:81-96, the light-map render_mt loop)
 *   vrt_mgpu_gi_filter        vrt_gi_filter                (gi::cone_trace_init_filter, main.cc:97)
 *   vrt_mgpu_gi_render_async  the GI film (main.cc:117-123): the 8-row bands dealt round-robin, each replica's
 *                             through vrt_gi_render_bands_async into film_rgb_full (pinned host memory); the
 *                             frame is complete after vrt_mgpu_sync.  Alternate between two host frames.
 *   vrt_mgpu_gi_render        vrt_mgpu_gi_render_async + vrt_mgpu_sync
 *   vrt_mgpu_gi_render_aov_async  the GI film (optional) and its planes: the same 8-row bands, each replica's
 *                             through vrt_gi_render_aov_bands_async into the full host frames of film_full_or_null
 *                             and aov_full (pinned); complete after vrt_mgpu_sync.  Alternate between two sets.
 *   vrt_mgpu_gi_render_aov    vrt_mgpu_gi_render_aov_async + vrt_mgpu_sync */
int vrt_mgpu_set_materials(vrt_mgpu* m, const float* tri_uv, const uint32_t* tri_mtl, uint32_t num_mtl,
                           const float* kd, const int32_t* mtl_tex, uint32_t num_tex, const vrt_texture* tex);
int vrt_mgpu_gi_init(vrt_mgpu* m);
int vrt_mgpu_gi_splat_camera(vrt_mgpu* m, const vrt_camera* light_cam, const float kd[3]);
int vrt_mgpu_gi_filter(vrt_mgpu* m);
int vrt_mgpu_gi_render_async(vrt_mgpu* m, const vrt_camera* cam, const float kd[3], float res, float* film_rgb_full);
int vrt_mgpu_gi_render(vrt_mgpu* m, const vrt_camera* cam, const float kd[3], float res, float* film_rgb_full);
int vrt_mgpu_gi_render_aov_async(vrt_mgpu* m, const vrt_camera* cam, const float kd[3], float res,
                                 float* film_full_or_null, const vrt_gi_aov* aov_full);
int vrt_mgpu_gi_render_aov(vrt_mgpu* m, const vrt_camera* cam, const float kd[3], float res, float* film_full_or_null,
                           const vrt_gi_aov* aov_full);
/* vrt_mean_kernel_ms of replica `index` (0 for a bad index): the per-device balance of a multi-GPU frame loop */
double vrt_mgpu_mean_kernel_ms(vrt_mgpu* m, int index, int last_n);

/* ---- animated geometry: new triangles for a built handle, then the build of vrt_rebuild at max_depth ----------
 * Full update: vrt_update_triangles(_dev) replaces the handle's triangles (its REST pose) and rebuilds.  num_tris must
 *   equal the handle's count (the per-triangle materials stay valid), tri_nrm must be given exactly when the handle
 *   was built with normals, and the handle's VRT_BUILD_UNIT_NORMALS flag is kept.  The _dev form copies from the
 *   caller's device arrays on the handle's stream; like every build both forms return when the build is done, so the
 *   arrays may be reused at once.
 * Transform update: vrt_update_xform sets the current pose to the rest pose with each range moved by its transform,
 *     p' = M[:, :3] p + M[:, 3]   for the three vertices   (m: row-major 3x4)
 *     n' = N n                    for the three normals    (n: row-major 3x3, normally the inverse transpose of
 *                                                           M[:, :3]; ignored when the handle has no normals)
 *   each coordinate evaluated as ((m0*x + m1*y) + m2*z) + m3 in float32 without fused multiply-add (and the same
 *   for n), and rebuilds.  Triangles outside every range keep their rest pose.  Ranges are non-empty, lie inside
 *   [0, num_tris) and do not overlap; transforms are absolute (the same table twice gives the same tree).  The rest
 *   pose is the triangles of the last build or full update; vrt_rebuild after a transform update rebuilds the
 *   current pose.
 * After either call the handle is bytewise the one vrt_build_ex with the same flags makes from the current pose (the
 * blob up to its size, vrt_tree_export, vrt_tree_get_info but build_ms and device_bytes).  Materials, film format,
 * stream and the pipelined-frame state are kept; the GI state is dropped as after every build (vrt_gi_init again).
 * Each update runs after every frame already enqueued on the handle (both kernel streams of the pipelined loops)
 * and before every frame enqueued later, as the GI writers do: frames enqueued before it render the old geometry,
 * frames after it the new, with no vrt_tree_sync in between.
 * Errors: VRT_ERR_ARG for a NULL handle or array, a wrong count, normals given or missing against the handle,
 * max_depth out of range, num_xf == 0, an empty, out-of-range or overlapping range, and a non-finite m or n entry;
 * VRT_ERR_STATE for a handle without input triangles (vrt_tree_load, vrt_tree_from_blob_dev) or on another
 * device.  A rejected call changes nothing and enqueues nothing.  A build failure (VRT_ERR_NOMEM, VRT_ERR_CAPACITY)
 * leaves what a failed vrt_rebuild leaves: the new pose is the handle's input and vrt_rebuild builds it, while the
 * octree is whatever the failed build left (the previous blob when it failed before assembly, none when the blob
 * could not be allocated: then every other call returns VRT_ERR_STATE); render nothing from it before a
 * successful update or vrt_rebuild. */
typedef struct vrt_xform {
        uint32_t first_tri, num_tris;
        float m[12]; /* row-major 3x4 */
        float n[9];  /* row-major 3x3 */
} vrt_xform;
int vrt_update_triangles(vrt_tree* tree, const float* tri_xyz, const float* tri_nrm, uint32_t num_tris,
                         int max_depth);
int vrt_update_triangles_dev(vrt_tree* tree, const float* d_tri_xyz, const float* d_tri_nrm, uint32_t num_tris,
                             int max_depth);
int vrt_update_xform(vrt_tree* tree, const vrt_xform* xf, uint32_t num_xf, int max_depth);
/* The same on the replicas of a vrt_mgpu: the first replica rebuilds, every other one then takes a copy of its blob
 * after its own enqueued frames, so every replica is bytewise the fresh build.  vrt_mgpu_create copies the source
 * tree's input triangles (about 72 bytes per triangle) as the rest pose; a replica set made from a tree without
 * them returns VRT_ERR_STATE from vrt_mgpu_update_xform until vrt_mgpu_update_triangles has given it triangles
 * (with or without normals; without VRT_BUILD_UNIT_NORMALS).  Host pointers.  On a failure the other replicas keep
 * their previous octree. */
int vrt_mgpu_update_triangles(vrt_mgpu* m, const float* tri_xyz, const float* tri_nrm, uint32_t num_tris,
                              int max_depth);
int vrt_mgpu_update_xform(vrt_mgpu* m, const vrt_xform* xf, uint32_t num_xf, int max_depth);

/* out = {node expansions cross-checked against the slab expansion, mismatches}; counts only in
 * a library built with -DVRT_PARAM_CHECK (tests), {0,0} otherwise. */
int vrt_debug_param_check(uint64_t out[2]);
/* Test hook: switch the content-hull pruning of the ray kernels off / on for this handle (the hulls stay
 * allocated), so that the pruned traversal can be compared with the unpruned one on the same tree. */
int vrt_debug_set_hull(vrt_tree* tree, int on);
/* Test hook: camera launches of this handle read eye-relative hull records and triangle terms (on, the default) or
 * subtract the eye per ray (off); both give the same results bit for bit. */
int vrt_debug_set_eye_rel(vrt_tree* tree, int on);
/* Test hook: number of camera launches of this handle that read eye-relative records so far. */
int vrt_debug_eye_rel_launches(const vrt_tree* tree, uint64_t* out);
/* Diagnostic (libraries built with -DVRT_HULL_STATS only, zeros otherwise): per tree level {node expansions, interior
 * children visited, hull tests, hull prunes} of the per-ray kernel since the last call. */
int vrt_debug_hull_stats(uint64_t out80[80]);
/* Test hook of the build's overflow guard: the per-level (triangle, cell) pair totals are 32-bit block
 * counts; whenever a level could produce 2^32 pairs they are also summed in 64 bits on the device and the
 * build returns VRT_ERR_CAPACITY instead of wrapping.  This runs that 64-bit sum on `n` host counts. */
int vrt_debug_pair_total(const uint32_t* block_counts, uint64_t n, uint64_t* total);
/* _dev launches are asynchronous with respect to the host: they return once the work is
 * enqueued on the tree's stream.  vrt_tree_sync waits for it. */
int vrt_tree_sync(const vrt_tree* tree);
/* device time (ms, CUDA events on the tree's stream) of the last trace/render kernel
 * launched through this handle, and the mean over the last n launches (n <= 64); both
 * wait for those launches to finish. */
double vrt_last_kernel_ms(const vrt_tree* tree);
double vrt_mean_kernel_ms(const vrt_tree* tree, int last_n);

/* ---- predicates (device KATs; each call launches a kernel) ---------------- */
/* triBoxOverlap (tribox2.h:15): centers[n][3], halves[n][3], tris[n][3][3] */
int vrt_tribox_batch(const float* centers, const float* halves, const float* tris,
                     uint64_t n, uint8_t* out);
/* Triangle::is_overlap (voxel_octree.cc:486-492): aabbs[n][6] */
int vrt_tri_overlap_aabb_batch(const float* aabbs, const float* tris, uint64_t n,
                               uint8_t* out);
/* intersect_triangle3 (raytri.h:5-7): in[n][15]=orig,dir,v0,v1,v2; tuv[n][3] */
int vrt_raytri_batch(const double* in, uint64_t n, uint8_t* result, double* tuv);
/* AABB<Vec3>::isect(ray,nullptr) (graphics_math.h:1312-1332) */
int vrt_aabb_isect_batch(const float* aabbs, const vrt_ray* rays, uint64_t n,
                         uint8_t* out);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* VRT_H */
