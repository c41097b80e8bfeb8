// vrt_internal.h -- handle layout, HBM blob layout and helpers shared by the
// translation units of libvrt.so.  Not part of the public ABI.
#pragma once

#include <cstdint>
#include <cstdio>
#include <string>
#include <cuda_runtime.h>

#include "../../include/vrt.h"

namespace vrt {

// ---------------------------------------------------------------------------
// HBM layout ("blob"): ONE contiguous device allocation holding everything the
// ray kernel reads, so that a replica is a single ncclBroadcast.  All section
// offsets are 256-byte aligned byte offsets from the start of the blob.
//
//   header      BlobHeader (512 B)
//   nodes       uint2[num_nodes], BFS order: level 0 (root) first, each level
//               sorted by Morton code, children of one node contiguous.
//                 interior (level < L): .x = index of first non-empty child,
//                                       .y = 8-bit child mask (bit c = child c
//                                            non-empty; c: x bit2, y bit1, z bit0)
//                 leaf     (level == L): .x = first triangle ref, .y = ref count
//   leaf_morton uint64[num_leaves]  Morton code of leaf i (3 bits per level)
//   leaf_refs   uint32[num_refs]    triangle indices, ascending per leaf
//   tri4        float4[3*num_tris]  vertices padded to 16 B (v0,_)(v1,_)(v2,_)
//   nrm         float[9*num_tris]   per-vertex normals, normalised like the
//                                   Triangle ctor (voxel_octree.cc:426)
//   axis_tab    float2[3][2^(L+1)]  per-axis cell bounds: entry (1<<l)+i of
//               axis a = (min,max) of cell i at level l along a, produced by the
//               reference's float recurrence (voxel_octree.cc:30-37).  Boxes are
//               products of three 1-D intervals, so this table IS the set of all
//               node AABBs ("pointerless and box-less" node array).
// ---------------------------------------------------------------------------
struct BlobHeader {
        uint64_t magic;
        uint64_t bytes;
        uint32_t num_tris;
        int32_t max_depth;  // reference's 1-based depth; L = max_depth-1
        float root_aabb[6];
        uint64_t num_nodes;
        uint64_t num_leaves;
        uint64_t num_refs;
        uint64_t level_offset[VRT_MAX_DEPTH + 1];
        uint64_t off_nodes;
        uint64_t off_leaf_morton;
        uint64_t off_leaf_refs;
        uint64_t off_tri4;
        uint64_t off_nrm;
        uint64_t off_axis_tab;
        uint64_t axis_tab_stride;  // float2 entries per axis = 2^(L+1)
};
static_assert(sizeof(BlobHeader) <= 512, "header grew");
constexpr uint64_t kBlobMagic = 0x3142305452565856ull;  // "VXVRT0B1"
constexpr uint64_t kHeaderBytes = 512;
// floats of GI state per node (vrt_gi.cuh): six lobes (+x +y +z -x -y -z), each one float4 {illum r, g, b, coverage}
// -- the node's coverage is repeated in every lobe so that a cone sample, which needs the three lobes facing the cone
// and the coverage, is three LDG.128
constexpr int kGiStride = 24;
constexpr int kGiCoverage = 3;

inline uint64_t align256(uint64_t x) { return (x + 255ull) & ~255ull; }

// Device-side view handed to kernels by value.
struct TreeDev {
        const uint2* nodes;
        const unsigned long long* leaf_morton;
        const uint32_t* leaf_refs;
        const float4* tri4;
        const float* nrm;
        const float4* tab4[3];  // axis table viewed as float4: entry (1<<l)+x =
                                // (lo.min, lo.max, hi.min, hi.max) of the two
                                // children of cell x at level l
        const float2* tab2[3];
        const float* gi;  // per-node GI state (vrt_gi.cuh), or null before vrt_gi_init
        // one word behind the GI state: 1 when cone_trace_init_filter has run since the last change of the light map AND
        // the root's filtered values are all finite -- then EVERY node's values are finite (a non-finite value
        // propagates up the sums of the filter), which is what lets a cone sample skip its zero-coefficient lobes
        const uint32_t* gi_ok;
        // content hull of every INTERIOR node (round 2), fused with a copy of its node record into one
        // 32-byte sector: float4 {first_child bits, child mask bits, x.min, x.max}, float4 {y.min, y.max, z.min,
        // z.max}; the bounds are the extreme leaf-cell planes (floats of the axis table) over the node's
        // non-empty leaves.  A ray whose slab interval over the hull is empty cannot pass the slab test of any
        // leaf below (monotone rounding), so the subtree is skipped without changing any result.  Null: no pruning.
        const float4* hull;
        // per interior node: bit c = child c's hull is worth testing (k_hull_level); the hull records of the other
        // children are never touched, their 8-byte node records are read instead
        const uint8_t* tight8;
        uint32_t rec_mask;  // 0xffff: hull tests on; 0x00ff: the tight flags are cleared from every record read (off)
        // triangles widened for the leaf test (round 2): per triangle ten doubles v0, e1 = v1 - v0, e2 = v2 - v0, pad --
        // the first operations of intersect_triangle3 (raytri.cc:205-207) on the widened vertices, done once per
        // build instead of once per (ray, triangle) test.  Every tree with triangles has them (compute_hulls).
        const double* tri64;
        // materials (vrt_set_materials), all null when unset: per-vertex texture coordinates, material id per
        // triangle, per material (kd.xyz, texture id or -1 as int bits), per texture (byte offset, w, h, channels)
        const float2* mat_uv;
        const uint32_t* mat_tri;
        const float4* mat_kd;
        const int4* mat_tex;
        const uint8_t* mat_texels;
        uint32_t num_nodes;
        uint32_t num_leaves;
        int L;  // leaf level = max_depth-1
        int tame;  // root box valid and |coords| <= 1e18: the FMNMX fast path is exact
};

void set_error(const char* fmt, ...);
bool cuda_ok(cudaError_t e, const char* what);
void count_launch(int n = 1);
// frees the scratch buffers parked by Scratch::release (one device synchronisation for all of them)
void scratch_flush_deferred();

#define VRT_CUDA(expr)                                  \
        do {                                            \
                if (!::vrt::cuda_ok((expr), #expr))     \
                        return VRT_ERR_CUDA;            \
        } while (0)

// Growable device scratch buffer (kept across rebuilds so timing loops do not
// hit cudaMalloc).
struct Scratch {
        void* p = nullptr;
        size_t cap = 0;
        int reserve(size_t bytes);
        void release();
        template <class T>
        T* as() const { return static_cast<T*>(p); }
};

}  // namespace vrt

struct vrt_tree {
        int device = 0;
        cudaStream_t stream = nullptr;
        bool own_blob = true;
        void* blob = nullptr;  // device
        uint64_t blob_bytes = 0;
        vrt::BlobHeader hdr{};  // host copy
        vrt::TreeDev dev{};
        // inputs kept for vrt_rebuild
        float* d_tri_in = nullptr;  // [T][9] as given
        float* d_nrm_in = nullptr;  // [T][9] as given, or null
        bool unit_normals = false;  // VRT_BUILD_UNIT_NORMALS: d_nrm_in is stored verbatim
        // build scratch
        vrt::Scratch keys_a, keys_b, tmp_a, tmp_b, tmp_c, hist, refs_s, tab_s, level_morton[VRT_MAX_DEPTH + 1],
            level_first[VRT_MAX_DEPTH + 1], level_mask[VRT_MAX_DEPTH + 1];
        uint32_t* d_counter = nullptr;  // small device counter block
        uint32_t* h_counter = nullptr;  // pinned mirror (also mapped: words 16..19 are the build's host mailbox)
        uint32_t mailbox_ticket = 0;
        // per-SM tile queues of the camera kernels: 8 launch slots x kTileQueues counters (vrt_trace.cu)
        static constexpr int kTileQueues = 256;
        uint32_t* d_tile_queues = nullptr;
        // trace scratch (host-pointer entry points)
        vrt::Scratch io_in, io_out;
        // GI rows (SURVEY.md 8f): per-node coverage + illum[6], see vrt_gi.cuh
        vrt::Scratch gi_buf, gi_recs, mat_buf;
        // step table of the last cone trace launch, one per kernel stream ([0] `stream`, [1] `alt_stream`): a GI frame
        // on one stream never overwrites the table a frame on the other stream may still read
        mutable vrt::Scratch gi_steps[2];
        vrt::Scratch hull_buf;  // TreeDev::hull
        vrt::Scratch tri64_buf;  // TreeDev::tri64
        // pipelined host-film path (vrt_render_camera_async): two device films, a copy stream
        vrt::Scratch film_dev[2];
        cudaStream_t copy_stream = nullptr;
        // the async frame loops alternate their kernels between `stream` and `alt_stream`, so that the head of
        // frame k+1 fills the SMs the long-ray tail of frame k leaves idle; launch_stream (when set) overrides
        // `stream` for the next trace launch
        cudaStream_t alt_stream = nullptr;
        mutable cudaStream_t launch_stream = nullptr;
        cudaEvent_t film_ready[2] = {}, film_copied[2] = {};
        // recorded on `stream` when a GI / material writer returns; alt_stream waits on it (vrt_api.cu gi_writer_end)
        cudaEvent_t gi_written = nullptr;
        mutable uint64_t n_async_frames = 0;
        cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // build timing
        // trace launches are asynchronous: each one records a (start, stop) pair in this ring
        static constexpr int kEvRing = 64;
        cudaEvent_t ring0[kEvRing] = {}, ring1[kEvRing] = {};
        mutable uint64_t n_trace_launches = 0;
        // L2 access-policy window over the top levels of the node array (vrt_trace.cu)
        mutable void* l2_window_stream = nullptr;
        mutable const void* l2_window_nodes = nullptr;
        mutable uint64_t l2_window_bytes = 0;
        // origin-relative axis tables of the camera launches (vrt_trace.cu tab_rel_for_launch)
        static constexpr int kRelSlots = 8;
        struct RelSlot {
                float eye[3] = { 0, 0, 0 };
                bool valid = false, done = false;
                cudaEvent_t ev = nullptr, ev_read = nullptr;  // table filled / last launch that reads it enqueued
                cudaStream_t stream = nullptr;
                uint64_t last_use = 0;
        };
        mutable uint64_t tabrel_clock = 0;
        mutable int tabrel_cur = 0;
        mutable vrt::Scratch tabrel_buf;
        mutable RelSlot tabrel_slot[kRelSlots];
        mutable const void* tabrel_blob = nullptr;
        mutable uint64_t tabrel_build = ~0ull;
        uint64_t n_builds = 0;  // bumped whenever the blob's contents change (tree_bind_views)
        int film_fmt = 0;  // VRT_FILM_* of every film this handle's kernels write (vrt_set_film_format)
        double build_ms = 0;
        mutable double last_kernel_ms = 0;
        uint64_t scratch_bytes() const;
};

namespace vrt {
int tree_alloc(vrt_tree** out);
void tree_bind_views(vrt_tree* t);
// build pipeline (vrt_build.cu)
int build_tree(vrt_tree* t, int max_depth);
// 64-bit sum of n device uint32 (the overflow guard of the per-level pair totals); synchronises the stream
int sum_u32_as_u64(vrt_tree* t, const uint32_t* d_v, uint64_t n, uint64_t* out);
// per-node content hulls beside the blob (after tree_bind_views; every build / import / replica)
int compute_hulls(vrt_tree* t);
int import_leaves(vrt_tree* t, int max_depth, const float root_aabb[6], uint64_t num_leaves,
                  const uint32_t* leaf_cell, const uint32_t* leaf_count,
                  const uint32_t* leaf_refs);
// trace (vrt_trace.cu)
enum OutMode { OUT_HIT48 = 0, OUT_HIT16 = 1, OUT_FILM = 2, OUT_COUNT = 3, OUT_HIT16_FILM = 4, OUT_SPLAT = 5, OUT_GI_FILM = 6 };
int launch_trace_rays(const vrt_tree* t, const vrt_ray* d_rays, uint64_t n, vrt_hit* d_out);
// band_h > 0: rows [y0,y1) are LOCAL rows of a banded shard; local row r maps to film row
// y0_film + (r / band_h) * band_pitch + r % band_h (y0 then carries y0_film, y1 = y0 + local rows).
struct GiArgs {  // OUT_SPLAT / OUT_GI_FILM: default material colour, cone-trace min_voxel_size
        float kd[3];
        float res;
        const float4* steps = nullptr;  // step table of the cone trace for (res, root box), see gi_step_table
};
int launch_trace_camera(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, int x0,
                        int y0, int x1, int y1, void* d_out, OutMode mode, int band_h = 0,
                        int band_pitch = 0, void* d_out2 = nullptr, int film_full = 0,
                        const GiArgs* gi = nullptr);
int launch_film_encode(const vrt_tree* t, const float* d_film, uint64_t npix, int fmt, uint8_t* d_out);
// mean device time (ms) of the last n trace launches (waits for them)
int trace_ms_mean(const vrt_tree* t, int last_n, double* ms);
int general_order_calls(unsigned long long* out);
int hull_stats(unsigned long long* out80);
// GI (vrt_gi.cu)
int gi_init(vrt_tree* t);
int gi_splat_camera(vrt_tree* t, const vrt_camera* cam, const float kd[3]);
int gi_filter(vrt_tree* t);
// fills the tree's step table for `res` on its launch stream (vrt_gi.cuh) -- the table of that kernel stream --
// and returns the device pointer
int gi_step_table(const vrt_tree* t, float res, const float4** d_steps);
int gi_cone_points(const vrt_tree* t, const float* d_pos, const float* d_nrm, uint64_t n, float res, float* d_out);
int gi_albedo_points(const vrt_tree* t, const uint32_t* d_tri, const float* d_pos, uint64_t n, const float kd[3], float* d_out);
// sort `n` 64-bit keys held in t->keys_a on bits [lo,hi) with the build's radix sort (vrt_build.cu)
int sort_keys_u64(vrt_tree* t, uint64_t n, int lo, int hi, unsigned long long** sorted);
int param_check_counts(unsigned long long out[2]);
}  // namespace vrt
