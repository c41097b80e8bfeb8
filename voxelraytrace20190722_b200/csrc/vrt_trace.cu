// vrt_trace.cu -- octree traversal + leaf triangle hits + fused ray generation.
//
// Replaces gi::ray_march / travorder / ray_march_isect (voxel_octree.cc:77-188),
// Triangle::isect -> intersect_triangle3 (voxel_octree.cc:438-460,
// raytri.cc:197-249), AABB<Vec3>::isect (graphics_math.h:1312-1332),
// Camera::gen_rays1/4 (camera.cc:77-112) and the render_mt pixel loop
// (camera.h:41-68).
//
// Reference semantics kept (SURVEY.md 8a):
//   1. children are visited in ascending dot(d, centre-o), ties by child index
//      (libstdc++ insertion sort of 8 items is stable);
//   2. a child is entered only if its slab test passes; empty children can never
//      produce a hit and are dropped up front (child mask);
//   3. the first leaf (in that order) with ANY accepted triangle ends the ray;
//      inside the leaf the smallest float length(hit-o) wins, first index on ties;
//      no t>0 / tmin / tmax test on triangle hits, hit not clipped to the leaf;
//   4. slab and key arithmetic are FMA-free and use the reference's operation
//      order; child boxes come from the recurrence table (vrt_internal.h).
//
// Work decomposition: one ray per thread, 32 rays of one warp form an 8x4 pixel
// tile (spp=1) or a 4x2 pixel tile x 4 samples (spp=4); warps pull tiles from an
// atomic queue (persistent threads).  The traversal stack (one 12-byte record
// per level) lives in shared memory, indexed [level][thread] -> conflict free.
#include <algorithm>
#include <cfloat>
#include <cstdlib>
#include <cstring>

#include "vrt_exact.cuh"
#include "vrt_gi.cuh"
#include "vrt_internal.h"

namespace vrt {

#ifndef VRT_TRACE_THREADS
#define VRT_TRACE_THREADS 128
#endif
#ifndef VRT_TRACE_MIN_BLOCKS
#define VRT_TRACE_MIN_BLOCKS 6  // k_trace_rays (48-byte records)
#endif
#ifndef VRT_EYE_ALL
#define VRT_EYE_ALL 0
#endif
#ifndef VRT_ER_EYE
#define VRT_ER_EYE 1
#endif
constexpr int kTraceThreads = VRT_TRACE_THREADS;
#ifndef VRT_TILE_BLOCK_LOG
#define VRT_TILE_BLOCK_LOG 3
#endif
constexpr uint32_t kTileBlockLog = VRT_TILE_BLOCK_LOG;  // the tile order runs over (1 << log) x (1 << log)-tile blocks
constexpr uint32_t kQueueBitmap = 248;  // per-SM tile queues: counters [0, 248), exhausted-queue bitmap [248, 256)
constexpr int kMaxLevels = VRT_MAX_DEPTH;  // stack records per thread

struct TraceParams {
        TreeDev tree;
        CameraParams cam;
        int x0, y0, x1, y1;  // pixel rectangle (camera modes); y range is LOCAL rows when banded
        int band_h, band_pitch;  // local row r -> film row y0 + (r/band_h)*band_pitch + r%band_h
        const vrt_ray* rays;  // explicit-ray mode
        unsigned long long num_rays;
        void* out;
        void* out2;  // film when MODE == OUT_HIT16_FILM
        int film_full;  // out2 is the full [ny][nx][3] frame (peer-mapped): address by film row
        int film_fmt;   // VRT_FILM_F32 / VRT_FILM_RGBE / VRT_FILM_RGB8: how a finished pixel is stored (include/vrt.h)
        uint32_t* queue;  // tile counter(s)
        uint32_t num_tiles;
        // camera kernels: one tile queue per SM over a blocked tile order (see k_trace_camera)
        uint32_t num_queues, queue_chunk, blocks_x, tiles_y;
        float light[3];
        float kd;
        float shadow_eps;
        int shadow;  // harness shadow ray per hit (BASELINE config 5)
        float root[6];
        float kd3[3];  // GI modes: the material's diffuse colour (untextured albedo)
        float gi_res;  // GI film: min_voxel_size of cone_trace (main.cc:69-70)
        const float4* gi_steps;  // GI film: the launch's step table (vrt_gi.cuh), or null
        uint32_t lut_off;  // warp-synchronous kernels: byte offset of the mask table in dynamic shared memory
        float eye[3];      // camera modes: the rays' common origin (camera_eye_host), bit-identical to gen_ray_origin
        // camera modes: the axis tables with the common origin already subtracted, rel[a][i] = tab4[a][i] - eye[a]
        // (k_tab_rel: the reference's (plane - o) of every slab test, evaluated once per table entry instead of once
        // per ray and node); null: the expansion subtracts itself
        const float4* tabrel[3];
        // camera modes, k_trace_camera<.., ER = true>: the hull records and the triangle terms relative to eye
        // (k_hull_eye_rel, k_tri_eye_rel)
        const float4* hull_eye;
        const double* tri_eye;
        vrt_gi_aov aov;  // OUT_GI_AOV: the per-pixel planes (include/vrt.h); a null member is not written
};

struct HitState {
        uint32_t tri;
        uint32_t leaf;  // global node index of the leaf
        uint32_t cx, cy, cz;
        float t, u, v;
        bool hit;
};

// Per-ray work counters of the reference algorithm (SURVEY.md 8d): interior nodes
// expanded (travorder calls), non-empty leaves visited, triangle tests.
struct WorkCount {
        uint32_t n_int, n_leaf, n_tri;
        // how the interior expansions were evaluated (kernel statistics, not reference work):
        // parametric fast path / slab fallback because of a tie / slab because the level is
        // not key-safe for this ray
        uint32_t n_param, n_tie, n_unsafe;
};

// Eye-relative triangle terms of a camera launch (k_tri_eye_rel): per triangle 14 doubles (112 bytes, seven 16-byte
// loads) e2, e1, tv = eye - v0, qv = tv x e1, tq = e2 . qv, pad.
constexpr uint32_t kTriEyeDoubles = 14;

// Triangle::isect + ray_march_isect for one leaf (voxel_octree.cc:99-129,438-460); rec = the leaf's node
// record {first reference, reference count}.  EYE: the terms come from tri_eye, the launch's eye-relative triangle
// terms (o is then the launch's eye).
template <bool COUNT, bool EYE = false>
__device__ __forceinline__ bool leaf_isect_rec(const TreeDev& tr, const uint2 rec, const float o[3],
                                               const float d[3], HitState& hs, WorkCount& wc,
                                               const double* tri_eye = nullptr)
{
        if (COUNT) {
                wc.n_leaf += 1;
                wc.n_tri += rec.y;
        }
        const double od[3] = { (double)o[0], (double)o[1], (double)o[2] };
        const double dd[3] = { (double)d[0], (double)d[1], (double)d[2] };
        bool found = false;
        float best = 0.f;
        for (uint32_t i = 0; i < rec.y; ++i) {
                const uint32_t ti = __ldg(&tr.leaf_refs[rec.x + i]);
                double dt, du, dv;
                if (EYE) {
                        const double2* q = reinterpret_cast<const double2*>(tri_eye + kTriEyeDoubles * (uint64_t)ti);
                        const double2 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);
                        const double2 q4 = __ldg(q + 4), q5 = __ldg(q + 5);
                        const double tq = __ldg(tri_eye + kTriEyeDoubles * (uint64_t)ti + 12);
                        const double e2[3] = { q0.x, q0.y, q1.x }, e1[3] = { q1.y, q2.x, q2.y };
                        const double tv[3] = { q3.x, q3.y, q4.x }, qv[3] = { q4.y, q5.x, q5.y };
                        if (ray_triangle3_eye(dd, e1, e2, tv, qv, tq, dt, du, dv) != 1)
                                continue;
                } else {  // v0, e1, e2 already widened and subtracted (k_tri64, every tree with triangles has them)
                        const double2* q = reinterpret_cast<const double2*>(tr.tri64 + 10ull * ti);  // 80-byte records
                        const double2 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3);
                        const double q4 = __ldg(tr.tri64 + 10ull * ti + 8);
                        const double a[3] = { q0.x, q0.y, q1.x }, e1[3] = { q1.y, q2.x, q2.y }, e2[3] = { q3.x, q3.y, q4 };
                        if (ray_triangle3_edges(od, dd, a, e1, e2, dt, du, dv) != 1)
                                continue;
                }
                // hit = o + (float)dt * d ; depth = length(hit - o)   voxel_octree.cc:454,114
                const float tf = __double2float_rn(dt);
                const float hx = fadd(o[0], fmul(tf, d[0]));
                const float hy = fadd(o[1], fmul(tf, d[1]));
                const float hz = fadd(o[2], fmul(tf, d[2]));
                const float ex = fsub(hx, o[0]), ey = fsub(hy, o[1]), ez = fsub(hz, o[2]);
                const float depth = __fsqrt_rn(dot3(ex, ey, ez, ex, ey, ez));
                if (!found || depth < best) {  // std::min_element: first minimum
                        found = true;
                        best = depth;
                        hs.tri = ti;
                        hs.t = tf;
                        hs.u = __double2float_rn(du);
                        hs.v = __double2float_rn(dv);
                }
        }
        return found;
}

template <bool COUNT>
__device__ __forceinline__ bool leaf_isect(const TreeDev& tr, uint32_t leaf_node, const float o[3],
                                           const float d[3], HitState& hs, WorkCount& wc)
{
        return leaf_isect_rec<COUNT>(tr, __ldg(&tr.nodes[leaf_node]), o, d, hs, wc);
}

// ISect of the winning triangle (voxel_octree.cc:449-454).
__device__ __forceinline__ void finish_isect(const TreeDev& tr, const HitState& hs, const float o[3],
                                             const float d[3], float pos[3], float nrm[3])
{
        const float u = clampf(hs.u, 0.f, 1.f);
        const float v = clampf(hs.v, 0.f, 1.f);
        const float w = clampf(fsub(fsub(1.f, u), v), 0.f, 1.f);
        const float* n = tr.nrm + 9ull * hs.tri;
#pragma unroll
        for (int k = 0; k < 3; ++k)
                nrm[k] = fadd(fadd(fmul(__ldg(n + k), w), fmul(__ldg(n + 3 + k), u)), fmul(__ldg(n + 6 + k), v));
        normalize3(nrm[0], nrm[1], nrm[2]);
#pragma unroll
        for (int k = 0; k < 3; ++k)
                pos[k] = fadd(o[k], fmul(hs.t, d[k]));
}

// EXACT path: one ray through the octree with every min/max/first-extremum rule of
// the reference restated literally (NaN/Inf/denormal-safe).  Only rays that fail the
// `ray_is_tame` test below take it, so it is kept out of line.
// s_first/s_meta/s_list: the three words of this thread's stack record 0; record r, word w lives
// at s_first[(3 * r + w) * blockDim.x] (see the kernels).
template <bool COUNT>
__device__ __noinline__ void trace_one_exact(const TreeDev& tr, const float* root, const float* o,
                                             const float* d, float tmin, float tmax, uint32_t* s_first,
                                             uint32_t* s_meta, uint32_t* s_list, HitState& hs, WorkCount& wc)
{
        float dinv[3];
#pragma unroll
        for (int k = 0; k < 3; ++k)
                dinv[k] = slab_dinv(d[k]);
        {
                const float mn[3] = { root[0], root[1], root[2] };
                const float mx[3] = { root[3], root[4], root[5] };
                if (!aabb_isect(mn, mx, o, dinv, tmin, tmax))  // voxel_octree.cc:134
                        return;
        }
        const int L = tr.L;
        if (L == 0) {  // root is the only leaf (voxel_octree.cc:137-144)
                if (leaf_isect<COUNT>(tr, 0, o, d, hs, wc)) {
                        hs.hit = true;
                        hs.leaf = 0;
                        hs.cx = hs.cy = hs.cz = 0;
                }
                return;
        }
        const int stride = blockDim.x;
        int level = 0;           // level of the node whose children are being iterated
        uint32_t x = 0, y = 0, z = 0;
        uint32_t node = 0;       // node to expand
        uint32_t first = 0, mask = 0, list = 0, cnt = 0;
        bool need_expand = true;
        for (;;) {
                if (need_expand) {
                        // ---- expand `node` at (level; x,y,z): order + slab-test its 8 children ----
                        const uint2 rec = __ldg(&tr.nodes[node]);
                        if (COUNT)
                                wc.n_int += 1;
                        first = rec.x;
                        mask = rec.y & 0xffu;
                        const uint32_t ti = (1u << level) + 0u;
                        const float4 bx = __ldg(&tr.tab4[0][ti + x]);
                        const float4 by = __ldg(&tr.tab4[1][ti + y]);
                        const float4 bz = __ldg(&tr.tab4[2][ti + z]);
                        // per axis, per half (lo/hi child): slab interval and centre key term
                        float smin[3][2], smax[3][2], kterm[3][2];
                        const float4 bb[3] = { bx, by, bz };
#pragma unroll
                        for (int a = 0; a < 3; ++a) {
                                const float mnv[2] = { bb[a].x, bb[a].z };
                                const float mxv[2] = { bb[a].y, bb[a].w };
#pragma unroll
                                for (int hsel = 0; hsel < 2; ++hsel) {
                                        const float t_a = fmul(fsub(mnv[hsel], o[a]), dinv[a]);
                                        const float t_b = fmul(fsub(mxv[hsel], o[a]), dinv[a]);
                                        smin[a][hsel] = std_min(t_a, t_b);
                                        smax[a][hsel] = std_max(t_a, t_b);
                                        // travorder key term: d * (centre - o), centre=(min+max)*.5f
                                        const float ctr = fmul(fadd(mnv[hsel], mxv[hsel]), .5f);
                                        kterm[a][hsel] = fmul(d[a], fsub(ctr, o[a]));
                                }
                        }
                        float key[8];
                        uint32_t valid = 0;
#pragma unroll
                        for (int c = 0; c < 8; ++c) {
                                const int hx = (c >> 2) & 1, hy = (c >> 1) & 1, hz = c & 1;
                                const float t0 = max_element3(smin[0][hx], smin[1][hy], smin[2][hz]);
                                const float t1 = min_element3(smax[0][hx], smax[1][hy], smax[2][hz]);
                                if (((mask >> c) & 1u) && slab_accept(t0, t1, tmin, tmax))
                                        valid |= 1u << c;
                                key[c] = fadd(fadd(fadd(0.f, kterm[0][hx]), kterm[1][hy]), kterm[2][hz]);
                        }
                        // stable rank of every valid child among the valid children
                        uint32_t rank[8];
#pragma unroll
                        for (int c = 0; c < 8; ++c)
                                rank[c] = 0;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
#pragma unroll
                                for (int j = i + 1; j < 8; ++j) {
                                        const bool j_first = key[j] < key[i];  // else i (lower index) first
                                        rank[i] += (j_first && ((valid >> j) & 1u)) ? 1u : 0u;
                                        rank[j] += (!j_first && ((valid >> i) & 1u)) ? 1u : 0u;
                                }
                        }
                        list = 0;
#pragma unroll
                        for (int c = 0; c < 8; ++c)
                                if ((valid >> c) & 1u)
                                        list |= (uint32_t)c << (3u * rank[c]);
                        cnt = __popc(valid);
                        need_expand = false;
                }
                if (cnt == 0) {
                        if (level == 0)
                                return;  // miss
                        --level;
                        x >>= 1;
                        y >>= 1;
                        z >>= 1;
                        first = s_first[level * 3 * stride];
                        const uint32_t m = s_meta[level * 3 * stride];
                        mask = m & 0xffu;
                        cnt = m >> 8;
                        list = s_list[level * 3 * stride];
                        continue;
                }
                const uint32_t c = list & 7u;
                list >>= 3;
                --cnt;
                const uint32_t child = first + __popc(mask & ((1u << c) - 1u));
                const uint32_t cx = 2u * x + ((c >> 2) & 1u);
                const uint32_t cy = 2u * y + ((c >> 1) & 1u);
                const uint32_t cz = 2u * z + (c & 1u);
                if (level + 1 == L) {
                        if (leaf_isect<COUNT>(tr, child, o, d, hs, wc)) {
                                hs.hit = true;
                                hs.leaf = child;
                                hs.cx = cx;
                                hs.cy = cy;
                                hs.cz = cz;
                                return;
                        }
                } else {
                        s_first[level * 3 * stride] = first;
                        s_meta[level * 3 * stride] = mask | (cnt << 8);
                        s_list[level * 3 * stride] = list;
                        ++level;
                        x = cx;
                        y = cy;
                        z = cz;
                        node = child;
                        need_expand = true;
                }
        }
}

// ---------------------------------------------------------------------------
// TAME rays (finite, moderately sized origin/direction whose direction components are zero or
// normal floats) take trace_one_fast.  For such rays no NaN can appear in the slab or key
// arithmetic -- (plane-o) is finite and 1/d' is finite and non-zero -- so
// std::min/std::max/min_element/max_element coincide with FMNMX up to the sign of a zero, which
// none of the comparisons below can observe.  Two node expansions exist for them:
//   * expand_slab (out of line, the fallback): the reference's eight per-child slab tests in
//     FMNMX form -- hi.min of a child pair is bitwise lo.max (both are min+size in the
//     recurrence), so 3 planes per axis instead of 4; children that pass are inserted into a
//     4-slot list kept sorted by key (stable), the rare 5th candidate falls back to a general
//     packed-rank ordering of all 8 (order_children_general);
//   * the parametric expansion inside trace_one_fast (see there), used whenever it is provably
//     equivalent.
// Packed FADD2/FMUL2 carry the per-axis plane arithmetic; only levels that still have unvisited
// children are pushed on the (shared-memory) return stack.
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool ray_is_tame(const TreeDev& tr, const float o[3], const float d[3])
{
        bool ok = tr.tame != 0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                const float ad = fabsf(d[k]);
                ok = ok && (fabsf(o[k]) <= 1e18f) && (ad <= 1e18f) && (ad == 0.f || ad >= FLT_MIN);
        }
        return ok;
}

__device__ __forceinline__ float fmax3(float a, float b, float c)
{
        float r;
        asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
        return r;
}
__device__ __forceinline__ float fmin3(float a, float b, float c)
{
        float r;
        asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
        return r;
}

// Packed FP32x2 arithmetic (sm_100+ FADD2/FMUL2): two independently rounded IEEE
// operations per issued instruction.  ptxas contracts a packed mul feeding a packed
// add/sub into FFMA2 even with explicit .rn and --fmad=false (observed with CUDA 12.9),
// so these helpers are ONLY used where the consumer of a product is not an add/sub:
// sub->mul and add->mul chains.  The SASS of the expansion block is checked for FFMA2.
__device__ __forceinline__ float2 sub2s(float ax, float ay, float b)
{
        float2 r;
        asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%4}; sub.rn.f32x2 rc, ra, rb; mov.b64 {%0,%1}, rc;}"
            : "=f"(r.x), "=f"(r.y) : "f"(ax), "f"(ay), "f"(b));
        return r;
}
__device__ __forceinline__ float2 add2(float ax, float ay, float bx, float by)
{
        float2 r;
        asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; add.rn.f32x2 rc, ra, rb; mov.b64 {%0,%1}, rc;}"
            : "=f"(r.x), "=f"(r.y) : "f"(ax), "f"(ay), "f"(bx), "f"(by));
        return r;
}
__device__ __forceinline__ float2 mul2s(float2 a, float b)
{
        float2 r;
        asm("{.reg .b64 ra, rb, rc; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%4}; mul.rn.f32x2 rc, ra, rb; mov.b64 {%0,%1}, rc;}"
            : "=f"(r.x), "=f"(r.y) : "f"(a.x), "f"(a.y), "f"(b));
        return r;
}

// General ordering of a node's children (any number of valid children): the packed-rank
// method.  Only reached when more than four children of one node pass the slab test
// (a ray through shared faces/edges); kept out of line.  Returns the visiting order as a
// list of 3-bit child ids (lowest bits first) and the count.
__device__ unsigned long long g_general_calls = 0;  // how often the >4-candidate path ran (tests)

__device__ __noinline__ uint32_t order_children_general(const float* smin6, const float* smax6, const float* kt6,
                                                        uint32_t mask, float tmin, float tmax, uint32_t* cnt_out)
{
        const float inf = __int_as_float(0x7f800000);
        atomicAdd(&g_general_calls, 1ull);
        float key[8];
        uint32_t cnt = 0;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
                const int hx = c >> 2, hy = (c >> 1) & 1, hz = c & 1;
                const float t0 = fmaxf(fmaxf(smin6[hx], smin6[2 + hy]), smin6[4 + hz]);
                const float t1 = fminf(fminf(smax6[hx], smax6[2 + hy]), smax6[4 + hz]);
                key[c] = inf;
                if (((mask >> c) & 1u) && slab_accept(t0, t1, tmin, tmax)) {
                        key[c] = fadd(fadd(kt6[hx], kt6[2 + hy]), kt6[4 + hz]);
                        cnt += 1u;
                }
        }
        uint32_t ranks = 0x76543210u;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
#pragma unroll
                for (int j = i + 1; j < 8; ++j)
                        ranks += (key[j] < key[i]) ? ((1u << (4 * i)) - (1u << (4 * j))) : 0u;
        }
        uint32_t list = 0;
#pragma unroll
        for (int c = 0; c < 8; ++c)
                list |= (uint32_t)c << (3u * ((ranks >> (4 * c)) & 15u));  // invalid ones land behind the valid ones
        *cnt_out = cnt;
        return list;
}

// Slab expansion of one node for a tame ray: the reference's per-child test and key order
// evaluated for all 8 children (FMNMX form).  Used by the parametric expansion below as its
// fallback (ties, key-unsafe levels), so it is kept out of line.  Returns the visiting order
// as 3-bit child ids, lowest bits first.
__device__ __noinline__ uint32_t expand_slab(float4 b0, float4 b1, float4 b2, float ox, float oy, float oz,
                                             float dx, float dy, float dz, float ix, float iy, float iz,
                                             uint32_t mask, float tmin, float tmax, uint32_t* cnt_out)
{
        const float inf = __int_as_float(0x7f800000);
        const float4 bb[3] = { b0, b1, b2 };
        const float o[3] = { ox, oy, oz }, d[3] = { dx, dy, dz }, dinv[3] = { ix, iy, iz };
        float smin[3][2], smax[3][2], kt[3][2];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
                // b = (p0, p1, p1, p2): lo child [p0,p1], hi child [p1,p2]
                const float2 t01 = mul2s(sub2s(bb[a].x, bb[a].y, o[a]), dinv[a]);  // (p-o)*dinv
                const float2 t12 = mul2s(sub2s(bb[a].z, bb[a].w, o[a]), dinv[a]);
                smin[a][0] = fminf(t01.x, t01.y);
                smax[a][0] = fmaxf(t01.x, t01.y);
                smin[a][1] = fminf(t12.x, t12.y);
                smax[a][1] = fmaxf(t12.x, t12.y);
                // travorder key terms d*((min+max)*.5f - o); the subtraction stays scalar
                // so that it cannot be contracted with the *.5f
                const float2 h = mul2s(add2(bb[a].x, bb[a].y, bb[a].z, bb[a].w), .5f);
                kt[a][0] = fmul(d[a], fsub(h.x, o[a]));
                kt[a][1] = fmul(d[a], fsub(h.y, o[a]));
        }
        float kxy[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
                kxy[q] = fadd(kt[0][q >> 1], kt[1][q & 1]);
        // candidates are inserted into a 4-slot list sorted by key; a later child
        // (higher index) goes behind equal keys -- the stable order of the
        // reference's insertion sort.  A line meets at most 4 of the 8 octants,
        // so a 5th candidate is rare and handled by the general method.
        float sk0 = inf, sk1 = inf, sk2 = inf, sk3 = inf;
        uint32_t si0 = 0, si1 = 0, si2 = 0, si3 = 0;
        uint32_t cnt = 0;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
                const float t0 = fmax3(smin[0][c >> 2], smin[1][(c >> 1) & 1], smin[2][c & 1]);
                const float t1 = fmin3(smax[0][c >> 2], smax[1][(c >> 1) & 1], smax[2][c & 1]);
                if (((mask >> c) & 1u) && slab_accept(t0, t1, tmin, tmax)) {
                        float ck = fadd(kxy[c >> 1], kt[2][c & 1]);
                        uint32_t ci = c;
                        cnt += 1u;
                        bool p;
                        float tk;
                        uint32_t tiq;
                        p = ck < sk0; tk = sk0; tiq = si0; sk0 = p ? ck : sk0; si0 = p ? ci : si0; ck = p ? tk : ck; ci = p ? tiq : ci;
                        p = ck < sk1; tk = sk1; tiq = si1; sk1 = p ? ck : sk1; si1 = p ? ci : si1; ck = p ? tk : ck; ci = p ? tiq : ci;
                        p = ck < sk2; tk = sk2; tiq = si2; sk2 = p ? ck : sk2; si2 = p ? ci : si2; ck = p ? tk : ck; ci = p ? tiq : ci;
                        p = ck < sk3; sk3 = p ? ck : sk3; si3 = p ? ci : si3;
                }
        }
        uint32_t list = si0 | (si1 << 3) | (si2 << 6) | (si3 << 9);
        if (cnt > 4u) {
                const float a_min[6] = { smin[0][0], smin[0][1], smin[1][0], smin[1][1], smin[2][0], smin[2][1] };
                const float a_max[6] = { smax[0][0], smax[0][1], smax[1][0], smax[1][1], smax[2][0], smax[2][1] };
                const float a_kt[6] = { kt[0][0], kt[0][1], kt[1][0], kt[1][1], kt[2][0], kt[2][1] };
                uint32_t cnt_general = 0;
                list = order_children_general(a_min, a_max, a_kt, mask, tmin, tmax, &cnt_general);
                cnt = cnt_general;
        }
        *cnt_out = cnt;
        return list;
}

// expand_slab with the result in the fast path's list format: 4 bits per entry, lowest first,
// entry = 8 | child id, empty list = 0 (at most 8 entries).
__device__ __noinline__ uint32_t expand_slab4(float4 b0, float4 b1, float4 b2, float ox, float oy, float oz,
                                              float dx, float dy, float dz, float ix, float iy, float iz,
                                              uint32_t mask, float tmin, float tmax)
{
        uint32_t cnt = 0;
        const uint32_t l3 = expand_slab(b0, b1, b2, ox, oy, oz, dx, dy, dz, ix, iy, iz, mask, tmin, tmax, &cnt);
        uint32_t l4 = 0;
        for (uint32_t i = cnt; i-- > 0u;)
                l4 = (l4 << 4) | 8u | ((l3 >> (3u * i)) & 7u);
        return l4;
}

// Number of tree levels at which the PARAMETRIC expansion (below) provably visits the
// children in the reference's key order for this ray: consecutive cells along the ray differ
// in one axis a, their travorder keys differ by |d_a| * (centre step) before rounding, and
// every rounding in  ((0 + dx*(cx-ox)) + dy*(cy-oy)) + dz*(cz-oz)  is monotone, so the float
// keys are ordered like the cells as soon as that step exceeds the accumulated rounding
// error (< 8 * 2^-24 * B, B bounding every intermediate magnitude).  We ask for
// |d_a| * extent_a * 2^-(l+1) >= 2^-18 * B (4x margin) at expansion level l; below that the slab
// expansion is used.  Axis-parallel rays (d_a == 0) and flat scenes (extent_a == 0) get 0.
__device__ __forceinline__ int param_safe_levels(const float root[6], const float o[3], const float d[3])
{
        float B = 0.f, pm = 0.f, q = __int_as_float(0x7f800000);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
                B += fmaxf(fabsf(root[a] - o[a]), fabsf(root[3 + a] - o[a]));
                pm = fmaxf(pm, fmaxf(fabsf(root[a]), fabsf(root[3 + a])));
                q = fminf(q, fabsf(d[a]) * (root[3 + a] - root[a]));
        }
        B = (B + pm) * 3.814697265625e-06f;  // 2^-18
        if (!(B > 0.f) || !(q > 0.f))
                return 0;
        const float r = q / B;  // <= 2^19
        if (!(r >= 2.f))
                return 0;
        return (int)(__float_as_uint(r) >> 23) - 127;  // r >= 2^e: levels 0..e-1 are safe
}

#ifdef VRT_PARAM_CHECK
__device__ unsigned long long g_param_check[4] = { 0, 0, 0, 0 };  // checked, mismatches, -, -
#endif
#ifdef VRT_HULL_STATS  // diagnostic build: [level][0..3] = expansions, visited interior children, hull tests, prunes
__device__ unsigned long long g_hull_stats[20][4];
#endif

// Can the (tame) ray reach any non-empty leaf below interior node `node`?  Slab interval of the ray
// over the node's content hull (TreeDev::hull) against the window, as an OVERLAP test: every leaf
// cell below lies inside the hull plane by plane and rounding is monotone, so a leaf that passes the
// reference's slab test implies max(t0,tmin) <= min(t1,tmax) here.  false = the subtree cannot
// produce a hit; skipping it changes no result.  ER: the record is eye-relative (k_hull_eye_rel: the planes already
// minus the launch's eye, which is o), so only the products remain.
template <bool ER = false>
__device__ __forceinline__ bool hull_reachable(const float4 ha, const float4 hb, const float o[3], const float dinv[3],
                                               float tmin, float tmax, float& t0, float& t1)
{
        const float2 ax = mul2s(ER ? make_float2(ha.z, ha.w) : sub2s(ha.z, ha.w, o[0]), dinv[0]);
        const float2 ay = mul2s(ER ? make_float2(hb.x, hb.y) : sub2s(hb.x, hb.y, o[1]), dinv[1]);
        const float2 az = mul2s(ER ? make_float2(hb.z, hb.w) : sub2s(hb.z, hb.w, o[2]), dinv[2]);
        t0 = fmax3(fminf(ax.x, ax.y), fminf(ay.x, ay.y), fminf(az.x, az.y));
        t1 = fmin3(fmaxf(ax.x, ax.y), fmaxf(ay.x, ay.y), fmaxf(az.x, az.y));
        return fmaxf(t0, tmin) <= fminf(t1, tmax);
}

// FAST path.  Node expansion is PARAMETRIC: with t(p) = (p-o)*dinv the nine child-plane
// parameters of a node (three planes per axis; exactly the floats the reference's eight slab
// tests are made of), a child's slab interval is the intersection of three per-axis intervals
// [e0,em] or [em,e1] (e0/e1 = near/far plane, em = mid plane; rounding is monotone so
// e0 <= em <= e1 holds in floats).  The children with t0 <= t1 are therefore exactly the cells
// of a 2x2x2 grid met by the diagonal t -> (t,t,t) on [T0,T1] = [max e0, min e1]: a start cell
// (axis a is in its far half iff em_a < T0) followed by one flip per axis whose em_a lies in
// [T0,T1], in ascending em_a.  Closed intervals make this exact unless two flipping axes have
// EQUAL em (the ray meets a shared edge: extra cells touch) -- then, and at levels that are
// not key-safe (param_safe_levels), the node is expanded by expand_slab instead.  Each cell
// knows its own t0 (entry breakpoint) and t1 (next breakpoint), so the reference's window test
// slab_accept(t0,t1,tmin,tmax) is evaluated on the same values.
// ER (camera launches, o = the launch's eye): the hull records are read from hull_eye and the leaf tests take
// their eye-dependent terms from tri_eye (EyeRel below) instead of subtracting the origin per ray.
template <bool COUNT, bool REL, bool ER>
__device__ __forceinline__ void trace_one_fast(const TreeDev& tr, const float root[6], const float o[3],
                                               const float d[3], float tmin, float tmax, uint32_t* s_first,
                                               uint32_t* s_meta, uint32_t* s_list, HitState& hs, WorkCount& wc,
                                               const float4* const* rel, const float4* hull_eye,
                                               const double* tri_eye)
{
        const float4* const hull = ER ? hull_eye : tr.hull;
        float dinv[3];
#pragma unroll
        for (int k = 0; k < 3; ++k)
                dinv[k] = slab_dinv(d[k]);
        {
                const float mn[3] = { root[0], root[1], root[2] };
                const float mx[3] = { root[3], root[4], root[5] };
                if (!aabb_isect(mn, mx, o, dinv, tmin, tmax))  // voxel_octree.cc:134
                        return;
        }
        const int L = tr.L;
        if (L == 0) {  // root is the only leaf (voxel_octree.cc:137-144)
                if (leaf_isect<COUNT>(tr, 0, o, d, hs, wc)) {
                        hs.hit = true;
                        hs.leaf = 0;
                        hs.cx = hs.cy = hs.cz = 0;
                }
                return;
        }
        constexpr int stride = kTraceThreads;
        // per-ray constants of the parametric expansion in ONE register: bits 0-2 negmask (near
        // half of axis a is the HIGH child when d_a < 0; child id: x bit 2, y bit 1, z bit 0),
        // bit 3 always set (the "entry present" bit of a visiting-list entry, see below), bit 4
        // default window [0, FLT_MAX], bits 5.. number of key-safe levels
        uint32_t rayflags = (d[0] < 0.f ? 4u : 0u) | (d[1] < 0.f ? 2u : 0u) | (d[2] < 0.f ? 1u : 0u) | 8u |
                            (((tmin == 0.f) && (tmax == FLT_MAX)) ? 16u : 0u) |
                            ((uint32_t)param_safe_levels(root, o, d) << 5);
        asm volatile("" : "+r"(rayflags));  // keep it in its register (do not rematerialise per node)
        // x,y,z are HEAP indices into the per-axis table: (1 << level) + cell coordinate, so a
        // child is 2*i + bit and an ancestor i >> k.  The return stack is addressed through one
        // register holding this thread's shared-memory byte address of the next free record.
        int level = 0;
        uint32_t x = 1, y = 1, z = 1;
        // record of the node to expand (a tested child's comes with its hull record) and its node index (for the
        // per-node flags of which children's hulls are worth testing)
        // (outside the counting mode every interior node's record is read from its hull record, whose mask word also
        // carries the tight-children flags in bits 8-15: the expansion needs no second per-node load; tr.rec_mask
        // = 0x00ff clears the flags -- the "hulls off" switch of the tests)
        uint2 rec;
        if (!COUNT) {
                const float4 h0 = __ldg(&hull[0]);
                rec = make_uint2(__float_as_uint(h0.x), __float_as_uint(h0.y) & tr.rec_mask);
        } else {
                rec = __ldg(&tr.nodes[0]);
                rec.y &= 0xffu;
        }
        // visiting list of the node being iterated: 4 bits per entry, lowest first, entry =
        // 8 | child id -- an empty list is the value 0, so no separate count is carried
        uint32_t first, mask, list;
        uint32_t sp = (uint32_t)__cvta_generic_to_shared(s_first);
        // bottom-of-stack sentinel (meta bit 31): popping it means the ray left the tree
        asm volatile("st.shared.u32 [%0+%1], %2;" ::"r"(sp), "n"(stride * 4u), "r"(0x80000000u) : "memory");
        sp += 3u * stride * 4u;
        constexpr uint32_t kCol = stride * 4u;  // bytes between the three words of a record
        constexpr uint32_t kRec = 3u * kCol;    // bytes between records of one thread
        for (;;) {
                // ---- expand the node of `rec` (level; x,y,z) ---------------------------------
                {
                        if (COUNT)
                                wc.n_int += 1;
#ifdef VRT_HULL_STATS
                        atomicAdd(&g_hull_stats[level][0], 1ull);
#endif
                        first = rec.x;
                        mask = rec.y;  // bits 0-7 child mask; bits 8-15 children whose hull is worth testing (0 without hulls)
                        // REL: (plane - o) comes from the launch's table (the same subtraction, done once per entry)
                        float4 bx, by, bz;
                        if (REL) {
                                bx = __ldg(&rel[0][x]);
                                by = __ldg(&rel[1][y]);
                                bz = __ldg(&rel[2][z]);
                        } else {
                                bx = __ldg(&tr.tab4[0][x]);
                                by = __ldg(&tr.tab4[1][y]);
                                bz = __ldg(&tr.tab4[2][z]);
                        }
                        bool use_slab = false;
                        {
                                // t(p0), t(p1) packed, t(p2) scalar -- the reference's (plane-o)*dinv
                                const float2 ax = mul2s(REL ? make_float2(bx.x, bx.y) : sub2s(bx.x, bx.y, o[0]), dinv[0]);
                                const float2 ay = mul2s(REL ? make_float2(by.x, by.y) : sub2s(by.x, by.y, o[1]), dinv[1]);
                                const float2 az = mul2s(REL ? make_float2(bz.x, bz.y) : sub2s(bz.x, bz.y, o[2]), dinv[2]);
                                const float ax2 = fmul(REL ? bx.w : fsub(bx.w, o[0]), dinv[0]);
                                const float ay2 = fmul(REL ? by.w : fsub(by.w, o[1]), dinv[1]);
                                const float az2 = fmul(REL ? bz.w : fsub(bz.w, o[2]), dinv[2]);
                                const float emx = ax.y, emy = ay.y, emz = az.y;
                                const float T0 = fmax3(fminf(ax.x, ax2), fminf(ay.x, ay2), fminf(az.x, az2));
                                const float T1 = fmin3(fmaxf(ax.x, ax2), fmaxf(ay.x, ay2), fmaxf(az.x, az2));
                                // mid-plane parameters in ascending order s0 <= s1 <= s2
                                const bool yx = emy < emx, zx = emz < emx, zy = emz < emy;
                                const float s0 = fmin3(emx, emy, emz), s2 = fmax3(emx, emy, emz);
                                // median = the one that is neither: a ^ b ^ c ^ min ^ max on the bit patterns
                                const float s1 = __uint_as_float(__float_as_uint(emx) ^ __float_as_uint(emy) ^ __float_as_uint(emz) ^
                                                                 __float_as_uint(s0) ^ __float_as_uint(s2));
                                // slab expansion instead: the ray may touch a shared edge (extra cells),
                                // or this level is not key-safe for the ray (level >= safe levels)
                                const bool unsafe = (uint32_t)(level * 32 + 31) >= rayflags;
                                if (s0 == s1 || s1 == s2 || unsafe) {
                                        use_slab = true;
                                        if (COUNT) {
                                                wc.n_unsafe += unsafe ? 1u : 0u;
                                                wc.n_tie += unsafe ? 0u : 1u;
                                        }
                                } else {
                                        if (COUNT)
                                                wc.n_param += 1;
                                        // axis bit (x 4, y 2, z 1) of the smallest / largest mid-plane parameter
                                        const uint32_t b0 = (!yx && !zx) ? 4u : ((yx && !zy) ? 2u : 1u);
                                        const uint32_t b2 = (yx && zx) ? 4u : ((!yx && zy) ? 2u : 1u);
                                        // the diagonal visits, in this order, the cells {}, {b0}, {b0,b1}, {all}
                                        // (set = axes already in their far half); as child ids:
                                        // (each with the entry bit 8 of the visiting list already set)
                                        const uint32_t c0 = rayflags & 15u, c1 = c0 ^ b0, c3 = c0 ^ 7u, c2 = c3 ^ b2;
                                        // cell j spans [max(T0, s_(j-1)), min(T1, s_j)] -- the very t0/t1 the
                                        // reference's slab test computes for that child
                                        bool a0, a1, a2, a3;
                                        if (rayflags & 16u) {
                                                // window [0, FLT_MAX] and finite t0 <= t1: accepted iff t1 >= 0.  With
                                                // s0 <= s1 <= s2:  max(T0,s_(j-1)) <= min(T1,s_j)  <=>  T0 <= T1 and
                                                // s_(j-1) <= T1 and T0 <= s_j;  min(T1,s_j) >= 0  <=>  T1 >= 0 and s_j >= 0.
                                                // The two lower bounds fold into TL = max(T0, 0):  T0 <= x and 0 <= x  <=>
                                                // TL <= x  (no NaN on this path; the sign of a zero is invisible to <=)
                                                const float TL = fmaxf(T0, 0.f);
                                                const bool vw = TL <= T1;
                                                a0 = vw && (TL <= s0);
                                                a1 = vw && (s0 <= T1) && (TL <= s1);
                                                a2 = vw && (s1 <= T1) && (TL <= s2);
                                                a3 = vw && (s2 <= T1);
                                        } else {
                                                const float h0 = fminf(T1, s0), h1 = fminf(T1, s1), h2 = fminf(T1, s2);
                                                const float l1 = fmaxf(T0, s0), l2 = fmaxf(T0, s1), l3 = fmaxf(T0, s2);
                                                a0 = slab_accept(T0, h0, tmin, tmax);
                                                a1 = slab_accept(l1, h1, tmin, tmax);
                                                a2 = slab_accept(l2, h2, tmin, tmax);
                                                a3 = slab_accept(l3, T1, tmin, tmax);
                                        }
                                        // child present?  (c_j carries the entry bit 8, so test bit 8+id of mask << 8)
                                        const uint32_t m8 = mask << 8;
                                        a0 = a0 && ((m8 & (1u << c0)) != 0u);
                                        a1 = a1 && ((m8 & (1u << c1)) != 0u);
                                        a2 = a2 && ((m8 & (1u << c2)) != 0u);
                                        a3 = a3 && ((m8 & (1u << c3)) != 0u);
                                        // visiting order = chain order; packed lowest bits first
                                        list = a3 ? c3 : 0u;
                                        list = a2 ? ((list << 4) | c2) : list;
                                        list = a1 ? ((list << 4) | c1) : list;
                                        list = a0 ? ((list << 4) | c0) : list;
#ifdef VRT_PARAM_CHECK
                                        {
                                                if (REL) {
                                                        bx = __ldg(&tr.tab4[0][x]);
                                                        by = __ldg(&tr.tab4[1][y]);
                                                        bz = __ldg(&tr.tab4[2][z]);
                                                }
                                                const uint32_t list_s = expand_slab4(bx, by, bz, o[0], o[1], o[2], d[0], d[1], d[2], dinv[0],
                                                                                     dinv[1], dinv[2], mask, tmin, tmax);
                                                atomicAdd(&g_param_check[0], 1ull);
                                                if (list_s != list)
                                                        atomicAdd(&g_param_check[1], 1ull);
                                        }
#endif
                                }
                        }
                        if (use_slab) {
                                if (REL) {  // the slab expansion works on the planes themselves
                                        bx = __ldg(&tr.tab4[0][x]);
                                        by = __ldg(&tr.tab4[1][y]);
                                        bz = __ldg(&tr.tab4[2][z]);
                                }
                                list = expand_slab4(bx, by, bz, o[0], o[1], o[2], d[0], d[1], d[2], dinv[0], dinv[1], dinv[2],
                                                    mask, tmin, tmax);
                        }
                }
                // ---- visit children in order until we descend, hit, or run out -----------------
                for (;;) {
                        if (list == 0u) {
                                sp -= kRec;
                                uint32_t m;
                                asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(m) : "r"(sp), "n"(kCol));
                                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(first) : "r"(sp));
                                asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(list) : "r"(sp), "n"(2u * kCol));
                                if ((int32_t)m < 0)
                                        return;  // miss
                                mask = m & 0xffffu;
                                const int nl = (int)(m >> 16);
                                x >>= (level - nl);
                                y >>= (level - nl);
                                z >>= (level - nl);
                                level = nl;
                                // (fall through: only levels with children left are ever pushed, so the popped list is not
                                // empty and the lane takes its next child in this same iteration -- lanes that pop and
                                // lanes that do not then run the visit step together instead of one warp iteration apart)
                        }
                        const uint32_t c = list & 7u;
                        list >>= 4;
                        const uint32_t child = first + __popc(mask & ((1u << c) - 1u));
                        const uint32_t cx = 2u * x + ((c >> 2) & 1u);
                        const uint32_t cy = 2u * y + ((c >> 1) & 1u);
                        const uint32_t cz = 2u * z + (c & 1u);
                        if (level + 1 == L) {
                                if (leaf_isect_rec<COUNT, ER>(tr, __ldg(&tr.nodes[child]), o, d, hs, wc, tri_eye)) {
                                        hs.hit = true;
                                        hs.leaf = child;
                                        hs.cx = cx - (1u << L);
                                        hs.cy = cy - (1u << L);
                                        hs.cz = cz - (1u << L);
                                        return;
                                }
                                continue;
                        }
                        // the child's node record, fused with its content hull: skip a child under which the
                        // ray cannot reach a non-empty leaf (not in the counting mode, which reports the
                        // reference algorithm's work)
                        // (only children flagged "tight" by the build are tested -- where the content fills most of
                        // the cell the test rarely prunes -- and only their 32-byte hull records are read; the bits
                        // are 0 without hulls and in the counting mode)
#ifdef VRT_HULL_STATS
                        atomicAdd(&g_hull_stats[level][1], 1ull);
#endif
                        if (!COUNT) {
                                const float4 ha = __ldg(&hull[2ull * child]);
                                if ((mask >> (8u + c)) & 1u) {
                                        const float4 hb = __ldg(&hull[2ull * child + 1]);
                                        float h0, h1;
#ifdef VRT_HULL_STATS
                                        atomicAdd(&g_hull_stats[level][2], 1ull);
                                        if (!hull_reachable<ER>(ha, hb, o, dinv, tmin, tmax, h0, h1))
                                                atomicAdd(&g_hull_stats[level][3], 1ull);
#endif
                                        if (!hull_reachable<ER>(ha, hb, o, dinv, tmin, tmax, h0, h1))
                                                continue;
                                }
                                rec = make_uint2(__float_as_uint(ha.x), __float_as_uint(ha.y) & tr.rec_mask);
                        } else {
                                rec = __ldg(&tr.nodes[child]);
                                rec.y &= 0xffu;
                        }
                        if (list != 0u) {  // remember this level only if it has children left
                                asm volatile("st.shared.u32 [%0], %1;" ::"r"(sp), "r"(first) : "memory");
                                asm volatile("st.shared.u32 [%0+%1], %2;" ::"r"(sp), "n"(kCol),
                                             "r"(mask + ((uint32_t)level << 16))
                                             : "memory");
                                asm volatile("st.shared.u32 [%0+%1], %2;" ::"r"(sp), "n"(2u * kCol), "r"(list) : "memory");
                                sp += kRec;
                        }
                        ++level;
                        x = cx;
                        y = cy;
                        z = cz;
                        break;
                }
        }
}

template <bool COUNT, bool REL = false, bool ER = false>
__device__ __forceinline__ void trace_one(const TreeDev& tr, const float root[6], const float o[3],
                                          const float d[3], float tmin, float tmax, uint32_t* s_first,
                                          uint32_t* s_meta, uint32_t* s_list, HitState& hs, WorkCount& wc,
                                          const float4* const* rel = nullptr, const float4* hull_eye = nullptr,
                                          const double* tri_eye = nullptr)
{
        hs.hit = false;
        hs.tri = VRT_NO_TRI;
        hs.leaf = VRT_NO_TRI;
        hs.cx = hs.cy = hs.cz = 0xffffffffu;
        hs.t = hs.u = hs.v = 0.f;
        if (tr.num_nodes == 0)
                return;
        if (ray_is_tame(tr, o, d))
                trace_one_fast<COUNT, REL, ER>(tr, root, o, d, tmin, tmax, s_first, s_meta, s_list, hs, wc, rel, hull_eye,
                                               tri_eye);
        else
                trace_one_exact<COUNT>(tr, root, o, d, tmin, tmax, s_first, s_meta, s_list, hs, wc);
}

// Out-of-line copy of the per-ray traversal: the fallback of the warp-synchronous kernels (and
// their shadow rays), so that the per-ray code exists once and off the hot path.  Everything goes
// in and out BY VALUE: the caller's ray and hit state never have their address taken and stay
// in registers on the hot path.
struct PtResult {
        HitState hs;
        WorkCount wc;
};
template <bool COUNT>
__device__ __noinline__ PtResult trace_one_nl(const TreeDev& tr, const float* root, float ox, float oy, float oz,
                                              float dx, float dy, float dz, float tmin, float tmax, uint32_t* s_first)
{
        PtResult r;
        r.wc = WorkCount{ 0, 0, 0, 0, 0, 0 };
        const float o3[3] = { ox, oy, oz }, d3[3] = { dx, dy, dz };
        const float r6[6] = { root[0], root[1], root[2], root[3], root[4], root[5] };
        trace_one<COUNT>(tr, r6, o3, d3, tmin, tmax, s_first, s_first + kTraceThreads, s_first + 2 * kTraceThreads, r.hs,
                         r.wc);
        return r;
}

// ---------------------------------------------------------------------------
// WARP-SYNCHRONOUS traversal (round 2).  The 32 rays of a warp tile share one traversal: the
// warp walks the UNION of the nodes its rays visit with one stack, every lane evaluates the
// node expansion for its own ray, and a lane takes part in a subtree only if its own ray would
// enter it.  Measured on the headline frame (instrumented oracle): a ray expands 29.8 nodes, the
// union over a 4x2-pixel x 4-sample tile is 33.4 nodes (28.5 rays per union node), so the warp
// runs ONE instruction stream without divergence, node records and plane tables are loaded once
// per warp, and the visit / stack bookkeeping is paid once per warp instead of once per lane.
//
// Why the shared visiting order is every ray's own order.  In the frame of the ray's direction
// signs (S = child id ^ negmask; bit a of S set = far half of axis a) the children a ray enters
// on a key-safe level without mid-plane ties are a CHAIN {} c {b0} c {b0,b1} c {x,y,z} visited in
// that order (see trace_one_fast).  Ascending numeric S is a linear extension of set inclusion, so
// a warp whose rays have the same direction signs can visit the children 0..7 in ascending S
// and every lane sees its own children in its own (= the reference's travorder) order; depth
// first recursion keeps that true for the leaves.  A lane stops at its first leaf with an
// accepted triangle, exactly like ray_march (voxel_octree.cc:181-185).
//
// Node expansion per lane, without any ordering work: child S of the node is entered iff its
// slab interval passes the reference's test.  With e0 <= em <= e1 the near / mid / far plane
// parameters per axis (the very floats of the per-child slab tests), TL = max(e0x,e0y,e0z,0),
// T1 = min(e1x,e1y,e1z):   t0_S = max(TL, em_a : a in S),  t1_S = min(T1, em_a : a not in S),
// accepted (window [0,FLT_MAX], finite values) iff t0_S <= t1_S.
//
// Eligibility of a tile (else every lane runs the per-ray path): all rays tame, default window,
// the same direction signs, every level key-safe for every ray.  A lane that meets a mid-plane
// tie (ray through a shared edge: the closed test admits cells outside the chain, whose order is
// the key order) leaves the warp traversal and is re-traced by the per-ray path afterwards.
//
// Children's node records are prefetched with cp.async into the warp's stack record while the
// expansion arithmetic runs, so a descent (or a leaf visit) starts from shared memory instead
// of a dependent global load.  Stack record r of a warp = two rows of 32 words:
//   A[r][lane] = the lane's 8 accept bits at that node;   B[r][0..15] = the children's records,
//   B[r][16..18] = first child, child mask | level << 8, children still to visit
// (the rows are the warp's own slice of the per-ray stack columns, see below).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void cp_async8(uint32_t saddr, const void* g)
{
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all()
{
        asm volatile("cp.async.wait_all;" ::: "memory");
}

constexpr uint32_t kFull = 0xffffffffu;
constexpr uint32_t kWsRedo = 0xfffffffeu;  // HitState::tri of a lane that left the warp traversal (mid-plane tie)
constexpr int kWsLutBytes = 8 * 256;  // child mask -> mask in the S frame, per negmask

// lut: the CTA's table [negmask][mask] -> bit S = mask bit (S ^ negmask)
__device__ __forceinline__ void ws_fill_lut(uint8_t* lut)
{
        for (int i = threadIdx.x; i < 8 * 256; i += blockDim.x) {
                const uint32_t ng = (uint32_t)i >> 8, m = (uint32_t)i & 255u;
                uint32_t r = 0;
#pragma unroll
                for (uint32_t S = 0; S < 8; ++S)
                        r |= ((m >> (S ^ ng)) & 1u) << S;
                lut[i] = (uint8_t)r;
        }
        __syncthreads();
}

template <bool COUNT>
__device__ __forceinline__ void trace_tile_ws(const TreeDev& tr, const float root[6], const float o[3],
                                              const float d[3], bool active, uint32_t neg, uint32_t* wsm,
                                              const uint8_t* lut, HitState& hs, WorkCount& wc)
{
        const uint32_t lane = threadIdx.x & 31u;
        hs.hit = false;
        hs.tri = VRT_NO_TRI;
        hs.leaf = VRT_NO_TRI;
        hs.cx = hs.cy = hs.cz = 0xffffffffu;
        hs.t = hs.u = hs.v = 0.f;
        float dinv[3];
#pragma unroll
        for (int k = 0; k < 3; ++k)
                dinv[k] = slab_dinv(d[k]);
        bool alive = active;
        {
                const float mn[3] = { root[0], root[1], root[2] };
                const float mx[3] = { root[3], root[4], root[5] };
                alive = alive && aabb_isect(mn, mx, o, dinv, 0.f, FLT_MAX);  // voxel_octree.cc:134
        }
        if (!__any_sync(kFull, alive))
                return;
        const uint32_t L = (uint32_t)tr.L;
        const uint8_t* lutn = lut + neg * 256u;
        // shared-memory byte addresses of this warp's rows: the warp only uses the words of its own
        // lanes' per-ray stack columns (other warps of the CTA may be on the per-ray path), i.e. rows of
        // 32 words every kTraceThreads words: A[r] = base + r * kWsRec, B[r] = A[r] + kWsRow
        constexpr uint32_t kWsRow = kTraceThreads * 4u, kWsRec = 2u * kWsRow;
        const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(wsm);
        uint32_t level = 0, x = 1, y = 1, z = 1, sp = 0;
        uint2 rec = __ldg(&tr.nodes[0]);
        bool in = alive;
        uint32_t first, mask, any8, acc8;
        for (;;) {
                // ---- expand the node whose record is `rec` (level; x,y,z) ---------------------
                first = rec.x;
                mask = rec.y & 0xffu;
                {
                        const float4 bx = __ldg(&tr.tab4[0][x]);
                        const float4 by = __ldg(&tr.tab4[1][y]);
                        const float4 bz = __ldg(&tr.tab4[2][z]);
                        // children's records -> B[sp][0..15]; at most one batch per lane in flight
                        cp_async_wait_all();
                        __syncwarp();  // every lane has read its child record out of this row
                        if (lane < (uint32_t)__popc(mask))
                                cp_async8(sbase + sp * kWsRec + kWsRow + lane * 8u, &tr.nodes[first + lane]);
                        const float2 ax = mul2s(sub2s(bx.x, bx.y, o[0]), dinv[0]);  // t(p0), t(pm)
                        const float2 ay = mul2s(sub2s(by.x, by.y, o[1]), dinv[1]);
                        const float2 az = mul2s(sub2s(bz.x, bz.y, o[2]), dinv[2]);
                        const float ax2 = fmul(fsub(bx.w, o[0]), dinv[0]);  // t(p2)
                        const float ay2 = fmul(fsub(by.w, o[1]), dinv[1]);
                        const float az2 = fmul(fsub(bz.w, o[2]), dinv[2]);
                        const float emx = ax.y, emy = ay.y, emz = az.y;
                        const float TL = fmaxf(fmax3(fminf(ax.x, ax2), fminf(ay.x, ay2), fminf(az.x, az2)), 0.f);
                        const float T1 = fmin3(fmaxf(ax.x, ax2), fmaxf(ay.x, ay2), fmaxf(az.x, az2));
                        // S bits: x 4, y 2, z 1 (far half of that axis)
                        const float lo1 = fmaxf(TL, emz), lo2 = fmaxf(TL, emy), lo4 = fmaxf(TL, emx);
                        const float lo3 = fmax3(TL, emy, emz), lo5 = fmax3(TL, emx, emz), lo6 = fmax3(TL, emx, emy);
                        const float lo7 = fmaxf(lo6, emz);
                        const float hi6 = fminf(T1, emz), hi5 = fminf(T1, emy), hi3 = fminf(T1, emx);
                        const float hi4 = fmin3(T1, emy, emz), hi2 = fmin3(T1, emx, emz), hi1 = fmin3(T1, emx, emy);
                        const float hi0 = fminf(hi1, emz);
                        uint32_t a = (TL <= hi0 ? 1u : 0u) | (lo1 <= hi1 ? 2u : 0u) | (lo2 <= hi2 ? 4u : 0u) |
                                     (lo3 <= hi3 ? 8u : 0u) | (lo4 <= hi4 ? 16u : 0u) | (lo5 <= hi5 ? 32u : 0u) |
                                     (lo6 <= hi6 ? 64u : 0u) | (lo7 <= T1 ? 128u : 0u);
                        a &= (uint32_t)lutn[mask];
                        const bool tie = (emx == emy) || (emy == emz) || (emx == emz);
                        if (in && tie) {  // the chain argument does not hold: re-trace this ray alone
                                hs.tri = kWsRedo;
                                alive = false;
                        }
                        const bool use = in && !tie;
                        acc8 = use ? a : 0u;
                        if (COUNT && use) {
                                wc.n_int += 1;
                                wc.n_param += 1;
                        }
#ifdef VRT_PARAM_CHECK
                        if (use) {
                                const uint32_t list_s = expand_slab4(bx, by, bz, o[0], o[1], o[2], d[0], d[1], d[2], dinv[0],
                                                                     dinv[1], dinv[2], mask, 0.f, FLT_MAX);
                                uint32_t list_w = 0;
                                for (int S = 7; S >= 0; --S)
                                        if ((a >> S) & 1u)
                                                list_w = (list_w << 4) | 8u | ((uint32_t)S ^ neg);
                                atomicAdd(&g_param_check[0], 1ull);
                                if (list_s != list_w)
                                        atomicAdd(&g_param_check[1], 1ull);
                        }
#endif
                        any8 = __reduce_or_sync(kFull, acc8);
                }
                // ---- visit the children in ascending S until the warp descends or is done ------
                for (;;) {
                        if (any8 == 0u) {
                                if (sp == 0u)
                                        return;
                                --sp;
                                const uint32_t ra = sbase + sp * kWsRec;
                                uint32_t ml;
                                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(acc8) : "r"(ra + lane * 4u));
                                asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(first) : "r"(ra), "n"(kWsRow + 64u));
                                asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(ml) : "r"(ra), "n"(kWsRow + 68u));
                                asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(any8) : "r"(ra), "n"(kWsRow + 72u));
                                mask = ml & 0xffu;
                                const uint32_t nl = ml >> 8;
                                x >>= (level - nl);
                                y >>= (level - nl);
                                z >>= (level - nl);
                                level = nl;
                                continue;
                        }
                        const uint32_t S = (uint32_t)__ffs((int)any8) - 1u;
                        any8 &= any8 - 1u;
                        const bool inc = alive && (((acc8 >> S) & 1u) != 0u);
                        if (!__any_sync(kFull, inc))
                                continue;  // (every ray that wanted this child has finished meanwhile)
                        const uint32_t c = S ^ neg;
                        const uint32_t k = (uint32_t)__popc(mask & ((1u << c) - 1u));
                        cp_async_wait_all();
                        __syncwarp();
                        uint2 crec;
                        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2+%3];"
                                     : "=r"(crec.x), "=r"(crec.y)
                                     : "r"(sbase + sp * kWsRec + k * 8u), "n"(kWsRow));
                        const uint32_t cx = 2u * x + ((c >> 2) & 1u);
                        const uint32_t cy = 2u * y + ((c >> 1) & 1u);
                        const uint32_t cz = 2u * z + (c & 1u);
                        if (level + 1u == L) {
                                bool found = false;
                                if (inc)
                                        found = leaf_isect_rec<COUNT>(tr, crec, o, d, hs, wc);
                                if (found) {
                                        hs.hit = true;
                                        hs.leaf = first + k;
                                        hs.cx = cx - (1u << L);
                                        hs.cy = cy - (1u << L);
                                        hs.cz = cz - (1u << L);
                                        alive = false;
                                }
                                if (!__any_sync(kFull, alive))
                                        return;
                                continue;
                        }
                        // content hull of the child (see hull_reachable): lanes whose ray cannot reach a non-empty
                        // leaf below leave the subtree; the warp skips it when no lane is left
                        bool incr = inc;
                        if (!COUNT && (tr.rec_mask & 0x100u)) {
                                const float4 ha = __ldg(&tr.hull[2ull * (first + k)]), hb = __ldg(&tr.hull[2ull * (first + k) + 1]);
                                float h0, h1;
                                incr = inc && hull_reachable(ha, hb, o, dinv, 0.f, FLT_MAX, h0, h1);
                                if (!__any_sync(kFull, incr))
                                        continue;
                        }
                        if (any8 != 0u) {  // remember this node only if it has children left
                                const uint32_t ra = sbase + sp * kWsRec;
                                asm volatile("st.shared.u32 [%0], %1;" ::"r"(ra + lane * 4u), "r"(acc8) : "memory");
                                if (lane == 0u)
                                        asm volatile("st.shared.v4.u32 [%0+%4], {%1,%2,%3,%3};" ::"r"(ra), "r"(first),
                                                     "r"(mask | (level << 8)), "r"(any8), "n"(kWsRow + 64u)
                                                     : "memory");
                                __syncwarp();
                                ++sp;
                        }
                        ++level;
                        x = cx;
                        y = cy;
                        z = cz;
                        rec = crec;
                        in = incr;
                        break;
                }
        }
}

__device__ __forceinline__ void store_hit48(vrt_hit* out, const TreeDev& tr, const HitState& hs,
                                            const float o[3], const float d[3])
{
        float pos[3] = { 0.f, 0.f, 0.f }, nrm[3] = { 0.f, 0.f, 0.f };
        if (hs.hit)
                finish_isect(tr, hs, o, d, pos, nrm);
        float4* q = reinterpret_cast<float4*>(out);
        q[0] = make_float4(__uint_as_float(hs.hit ? 1u : 0u), __uint_as_float(hs.tri), __uint_as_float(hs.cx),
                           __uint_as_float(hs.cy));
        q[1] = make_float4(__uint_as_float(hs.cz), hs.hit ? hs.t : 0.f, pos[0], pos[1]);
        q[2] = make_float4(pos[2], nrm[0], nrm[1], nrm[2]);
}

// Harness pixel (SURVEY.md 8d; main.cc:18-20 for the sky): miss -> sky lerp; hit ->
// kd * clamp(dot(normal, light), 0, 1) * visibility.  With p.shadow the visibility is a
// second ray_march-semantics query from hit + eps*normal toward the light (config 5 of
// BASELINE.json; harness-defined -- the reference itself has no shadow rays); it runs in
// the same kernel, reusing the thread's traversal stack.
template <bool COUNT, bool NL>
__device__ __forceinline__ void shade(const TraceParams& p, const HitState& hs, const float o[3],
                                      const float d[3], uint32_t* s_first, uint32_t* s_meta, uint32_t* s_list,
                                      WorkCount& wc, float rgb[3])
{
        if (!hs.hit) {
                // float t = 0.5 * (ray.d.y + 1.0)  -- double arithmetic, then lerp in float
                const float t = __double2float_rn(dmul(0.5, dadd((double)d[1], 1.0)));
                const float v1[3] = { 0.6f, 0.8f, 1.0f };
#pragma unroll
                for (int k = 0; k < 3; ++k)
                        rgb[k] = fadd(1.0f, fmul(fsub(v1[k], 1.0f), t));
                return;
        }
        float pos[3], nrm[3];
        finish_isect(p.tree, hs, o, d, pos, nrm);
        const float nl = clampf(dot3(nrm[0], nrm[1], nrm[2], p.light[0], p.light[1], p.light[2]), 0.f, 1.f);
        float c = fmul(p.kd, nl);
        if (p.shadow) {
                const float so[3] = { fadd(pos[0], fmul(p.shadow_eps, nrm[0])), fadd(pos[1], fmul(p.shadow_eps, nrm[1])),
                                      fadd(pos[2], fmul(p.shadow_eps, nrm[2])) };
                const float sd[3] = { p.light[0], p.light[1], p.light[2] };
                HitState sh;
                if (NL) {
                        const PtResult r = trace_one_nl<COUNT>(p.tree, p.root, so[0], so[1], so[2], sd[0], sd[1], sd[2], 0.f,
                                                               FLT_MAX, s_first);
                        sh.hit = r.hs.hit;
                        if (COUNT) {
                                wc.n_int += r.wc.n_int;
                                wc.n_leaf += r.wc.n_leaf;
                                wc.n_tri += r.wc.n_tri;
                                wc.n_param += r.wc.n_param;
                                wc.n_tie += r.wc.n_tie;
                                wc.n_unsafe += r.wc.n_unsafe;
                        }
                } else {
                        trace_one<COUNT>(p.tree, p.root, so, sd, 0.f, FLT_MAX, s_first, s_meta, s_list, sh, wc);
                }
                c = fmul(c, sh.hit ? 0.f : 1.f);
        }
        rgb[0] = rgb[1] = rgb[2] = c;
}

// The per-ray records, the film and the GI planes are written once and never read by the kernel: streaming stores
// (st.global.cs) keep them from displacing octree lines in L2 (-DVRT_PLAIN_STORES: ordinary stores).
#ifdef VRT_PLAIN_STORES
#define VRT_STORE_OUT(ptr, val) (*(ptr) = (val))
#else
#define VRT_STORE_OUT(ptr, val) __stcs((ptr), (val))
#endif

// The factors of one trace() sample that hits (main.cc:10-30): the ISect normal the cone basis is built from, the
// albedo, the cone-traced indirect light and the hit leaf's direct light toward the eye.  A miss leaves them +0.
struct GiTerms {
        float nrm[3], albedo[3], ind[3], dir[3];
};

// trace() of main.cc:10-30: sky on a miss, else albedo * (cone-traced indirect light + the leaf's
// direct light toward the eye); Triangle::is_visible() is true, albedo = material diffuse.
// g receives the factors (OUT_GI_AOV); the film mode discards them.
__device__ __forceinline__ void shade_gi(const TraceParams& p, const HitState& hs, const float o[3], const float d[3],
                                         uint32_t* s_col, float rgb[3], GiTerms& g)
{
        if (!hs.hit) {
                const float t = __double2float_rn(dmul(0.5, dadd((double)d[1], 1.0)));
                const float v1[3] = { 0.6f, 0.8f, 1.0f };
#pragma unroll
                for (int k = 0; k < 3; ++k)
                        rgb[k] = fadd(1.0f, fmul(fsub(v1[k], 1.0f), t));
                return;
        }
        float pos[3];
        finish_isect(p.tree, hs, o, d, pos, g.nrm);
        gi_albedo(p.tree, hs.tri, pos, p.kd3, g.albedo);
        // the traversal is over: this thread's stack column doubles as the cone trace's path cache
        gi_cone_trace_point(p.tree, p.root, reinterpret_cast<float*>(s_col), kTraceThreads, pos, g.nrm, p.gi_res,
                            p.gi_steps, g.ind);
        const float nd[3] = { -d[0], -d[1], -d[2] };
        gi_compute_illum(p.tree.gi + (size_t)kGiStride * hs.leaf, nd, g.dir);
#pragma unroll
        for (int k = 0; k < 3; ++k)
                rgb[k] = fmul(g.albedo[k], fadd(g.ind[k], g.dir[k]));
}

// film->add(px,py, v * (1/spp)) in sample order (main.cc:119-122), acc = +0 first: the pixel's sum, in the lane
// of sample 0.  Every lane of the warp takes part (shuffles).
__device__ __forceinline__ void accumulate_samples(const float v[3], int spp, float acc[3])
{
        const float wgt = (spp == 4) ? .25f : 1.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                const float c = fmul(v[k], wgt);
                if (spp == 4) {
                        const float c1 = __shfl_down_sync(0xffffffffu, c, 1);
                        const float c2 = __shfl_down_sync(0xffffffffu, c, 2);
                        const float c3 = __shfl_down_sync(0xffffffffu, c, 3);
                        acc[k] = fadd(fadd(fadd(fadd(0.f, c), c1), c2), c3);
                } else {
                        acc[k] = fadd(0.f, c);
                }
        }
}

// ---------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kTraceThreads, VRT_TRACE_MIN_BLOCKS)
k_trace_rays(const __grid_constant__ TraceParams p)
{
        extern __shared__ uint32_t s_stack[];
        uint32_t* s_first = s_stack + threadIdx.x;
        uint32_t* s_meta = s_first + kTraceThreads;  // record r, word w: s_first[(3 * r + w) * threads]
        uint32_t* s_list = s_meta + kTraceThreads;
        const unsigned long long nwarp_items = (p.num_rays + 31ull) / 32ull;
        const int lane = threadIdx.x & 31;
        for (;;) {
                uint32_t tile = 0;
                if (lane == 0)
                        tile = atomicAdd(p.queue, 1u);
                tile = __shfl_sync(0xffffffffu, tile, 0);
                if (tile >= nwarp_items)
                        break;
                const unsigned long long r = (unsigned long long)tile * 32ull + lane;
                if (r < p.num_rays) {
                        const float4* rp = reinterpret_cast<const float4*>(p.rays + r);
                        const float4 r0 = __ldg(rp), r1 = __ldg(rp + 1);
                        const float o[3] = { r0.x, r0.y, r0.z };
                        const float d[3] = { r0.w, r1.x, r1.y };
                        HitState hs;
                        WorkCount wc;
                        trace_one<false>(p.tree, p.root, o, d, r1.z, r1.w, s_first, s_meta, s_list, hs, wc);
                        store_hit48(static_cast<vrt_hit*>(p.out) + r, p.tree, hs, o, d);
                }
                __syncwarp();
        }
}

// Round 2: every mode ran best at 72 registers (7 CTAs/SM).  Round 1 had the compact outputs at 64 registers (8 CTAs/SM);
// since the tiles of an SM are neighbours on the film (per-SM queues below: L1 hit rate 73 -> 87 %) the warps wait
// less on memory, and the 1/d values that 64 registers push into local memory (re-read in every expansion and hull
// test) cost more than the eighth CTA hides: hit16 5.92 -> 5.72 ms per headline frame.
template <int MODE, bool WS, bool ER>
// Round 3: the instantiations with eye-relative records (ER: the film, hit16 and hit16 + film modes) no longer need
// the origin in registers during the traversal, and one more CTA per SM (64 registers) is faster for them: headline
// frame 5.51 -> 5.39 ms (B200, DESIGN.md section 5).
#ifndef VRT_FILM_MIN_BLOCKS
#define VRT_FILM_MIN_BLOCKS 7
#endif
#ifndef VRT_HIT16_MIN_BLOCKS
#define VRT_HIT16_MIN_BLOCKS 7
#endif
#ifndef VRT_GI_MIN_BLOCKS
#define VRT_GI_MIN_BLOCKS 5
#endif
__global__ void __launch_bounds__(kTraceThreads, (MODE == OUT_HIT16 || MODE == OUT_COUNT) ? VRT_HIT16_MIN_BLOCKS + (ER ? 1 : 0)
                                                 : (MODE == OUT_GI_FILM || MODE == OUT_GI_AOV) ? VRT_GI_MIN_BLOCKS
                                                                                          : VRT_FILM_MIN_BLOCKS + (ER ? 1 : 0))
k_trace_camera(const __grid_constant__ TraceParams p)
{
        extern __shared__ uint32_t s_stack[];
        uint32_t* s_first = s_stack + threadIdx.x;
        uint32_t* s_meta = s_first + kTraceThreads;  // record r, word w: s_first[(3 * r + w) * threads]
        uint32_t* s_list = s_meta + kTraceThreads;
        const int lane = threadIdx.x & 31;
        const int W = p.x1 - p.x0, H = p.y1 - p.y0;
        const int spp = p.cam.spp;
        // warp-synchronous path: this warp's stack rows and the CTA's child-mask table
        uint32_t* wsm = s_stack + (threadIdx.x & ~31u);
        const uint8_t* lut = reinterpret_cast<const uint8_t*>(s_stack) + p.lut_off;
        const bool ws_ok = WS && p.tree.L >= 1 && p.tree.num_nodes != 0 && p.tree.tame != 0 && p.cam.tmin == 0.f &&
                           p.cam.tmax == FLT_MAX;
        if (WS)
                ws_fill_lut(reinterpret_cast<uint8_t*>(s_stack) + p.lut_off);
        // warp tile: 8x4 pixels (spp 1) or 4x2 pixels x 4 samples (spp 4)
        const int tw = (spp == 4) ? 4 : 8, th = (spp == 4) ? 2 : 4;
        const int tiles_x = (W + tw - 1) / tw;
        // the next tile index is fetched while the current tile is traced (the atomic's round
        // trip to L2 stays off the critical path)
#ifndef VRT_TILE_GLOBAL
        // Tile order and queues.  The tile sequence runs block by block over 8x8-tile blocks (row-major inside a
        // block), and is cut into one contiguous range per SM; the warps of an SM pull from their SM's own counter, so
        // the tiles in flight on one SM are neighbours on the film and their rays share node, hull and triangle
        // records in that SM's L1 (hit rate 73 -> 87 % on the headline frame).  A warp that finds its queue exhausted
        // marks it in a bitmap behind the counters (p.queue[kQueueBitmap..]) and moves to the next queue that is not
        // marked -- at the end of a frame a warp reads eight words instead of probing every queue.
        // s_queue: the warp's current queue (shared, not a register: it is only touched between tiles).
        __shared__ uint32_t s_queue[kTraceThreads / 32];
        uint32_t* const my_queue = &s_queue[threadIdx.x >> 5];
        {
                uint32_t smid;
                asm("mov.u32 %0, %%smid;" : "=r"(smid));
                if (lane == 0)
                        *my_queue = smid % p.num_queues;
                __syncwarp();
        }
        // the ticket for the next tile is drawn while the current tile is traced (the atomic's round trip to L2
        // stays off the critical path); everything but the atomic itself is warp-uniform
        uint32_t next = 0;
        if (lane == 0)
                next = atomicAdd(p.queue + *my_queue, 1u);
        for (;;) {
                uint32_t n = __shfl_sync(0xffffffffu, next, 0);
                uint32_t qv = *my_queue;
                uint32_t tile = qv * p.queue_chunk + n;
                if (n >= p.queue_chunk || tile >= p.num_tiles) {  // this queue is exhausted: move on (rare)
                        tile = 0xffffffffu;
                        for (;;) {
                                if (lane == 0)
                                        atomicOr(p.queue + kQueueBitmap + (qv >> 5), 1u << (qv & 31u));
                                __syncwarp();
                                // lanes 0..7 hold the bitmap (read past L1: other SMs set the bits); a set bit or a bit
                                // beyond the last queue = nothing to fetch there
                                uint32_t w = 0xffffffffu;
                                if (lane < 8) {
                                        w = __ldcg(p.queue + kQueueBitmap + lane);
                                        const uint32_t first = (uint32_t)lane * 32u;
                                        if (p.num_queues < first + 32u)
                                                w |= (p.num_queues > first) ? (0xffffffffu << (p.num_queues - first)) : 0xffffffffu;
                                }
                                const uint32_t open = ~w;
                                // first open queue behind qv, else the first open queue at all
                                const uint32_t wl = qv >> 5;
                                const uint32_t behind = (lane > (int)wl) ? open
                                                        : (lane == (int)wl) ? (open & ~((2u << (qv & 31u)) - 1u))
                                                                            : 0u;
                                uint32_t vote = __ballot_sync(0xffffffffu, behind != 0u);
                                uint32_t pick = behind;
                                if (!vote) {
                                        vote = __ballot_sync(0xffffffffu, open != 0u);
                                        pick = open;
                                }
                                if (!vote)
                                        break;  // every queue is exhausted
                                const int src = __ffs((int)vote) - 1;
                                qv = (uint32_t)src * 32u + (uint32_t)(__ffs((int)__shfl_sync(0xffffffffu, pick, src)) - 1);
                                if (lane == 0)
                                        n = atomicAdd(p.queue + qv, 1u);
                                n = __shfl_sync(0xffffffffu, n, 0);
                                if (n < p.queue_chunk && qv * p.queue_chunk + n < p.num_tiles) {
                                        tile = qv * p.queue_chunk + n;
                                        break;
                                }
                        }
                        __syncwarp();
                        if (lane == 0)
                                *my_queue = qv;
                        __syncwarp();
                }
                if (tile == 0xffffffffu)
                        break;
                if (lane == 0)
                        next = atomicAdd(p.queue + qv, 1u);
                const uint32_t blk = tile >> (2 * kTileBlockLog);
                const uint32_t bly = blk / p.blocks_x, blx = blk - bly * p.blocks_x;
                const int ty = (int)((bly << kTileBlockLog) + ((tile >> kTileBlockLog) & ((1u << kTileBlockLog) - 1u))),
                          tx = (int)((blx << kTileBlockLog) + (tile & ((1u << kTileBlockLog) - 1u)));
                // (tiles in the padding of the blocked order lie beyond x1 / H: all their lanes are inactive)
#else
        uint32_t next = 0;
        if (lane == 0)
                next = atomicAdd(p.queue, 1u);
        for (;;) {
                const uint32_t tile = __shfl_sync(0xffffffffu, next, 0);
                if (tile >= p.num_tiles)
                        break;
                if (lane == 0)
                        next = atomicAdd(p.queue, 1u);
                const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
#endif
                int s, lx, ly;
                if (spp == 4) {
                        s = lane & 3;
                        lx = (lane >> 2) & 3;
                        ly = lane >> 4;
                } else {
                        s = 0;
                        lx = lane & 7;
                        ly = lane >> 3;
                }
                const int px = p.x0 + tx * tw + lx;
                const int ry = ty * th + ly;  // local row
                const int py = p.y0 + (ry / p.band_h) * p.band_pitch + (ry % p.band_h);
                const bool active = (px < p.x1) && (ry < H);
                float o[3] = { 0, 0, 0 }, d[3] = { 0, 0, 1 };
                HitState hs;
                hs.hit = false;
                WorkCount wc = { 0, 0, 0, 0, 0, 0 };
                if (WS) {
                        if (active)
                                gen_ray(p.cam, px, py, s, o, d);
                        // the tile is traced by the warp as a whole when every ray qualifies (see trace_tile_ws)
                        const uint32_t neg = (d[0] < 0.f ? 4u : 0u) | (d[1] < 0.f ? 2u : 0u) | (d[2] < 0.f ? 1u : 0u);
                        const uint32_t am = __ballot_sync(0xffffffffu, active);
                        const uint32_t neg0 = __shfl_sync(0xffffffffu, neg, am ? (__ffs((int)am) - 1) : 0);
                        const bool elig = !active || (neg == neg0 && ray_is_tame(p.tree, o, d) &&
                                                      param_safe_levels(p.root, o, d) >= p.tree.L);
                        const bool tile_ws = ws_ok && am != 0u && __all_sync(0xffffffffu, elig);
                        bool redo = false;
                        if (tile_ws) {
                                trace_tile_ws<MODE == OUT_COUNT>(p.tree, p.root, o, d, active, neg0, wsm, lut, hs, wc);
                                redo = !hs.hit && hs.tri == kWsRedo;
                        }
                        if (active && (!tile_ws || redo)) {
                                const PtResult r = trace_one_nl<MODE == OUT_COUNT>(p.tree, p.root, o[0], o[1], o[2], d[0], d[1],
                                                                                   d[2], p.cam.tmin, p.cam.tmax, s_first);
                                hs = r.hs;
                                if (MODE == OUT_COUNT)
                                        wc = r.wc;
                        }
                } else if (active) {
                        // the common origin comes precomputed from the host in the record-only modes (-3.5 % there);
                        // the film modes keep computing it (measured: with it precomputed ptxas spills more in those
                        // instantiations and the frame step gets 5 % slower) unless the eye-relative records are in use
                        // (ER: the traversal then needs the origin only in the rare slab fallback and the hit distance)
                        if (VRT_EYE_ALL || MODE == OUT_HIT16 || MODE == OUT_HIT48 || (ER && VRT_ER_EYE)) {
                                o[0] = p.eye[0];
                                o[1] = p.eye[1];
                                o[2] = p.eye[2];
                                gen_ray_dir(p.cam, px, py, s, d);
                        } else {
                                gen_ray(p.cam, px, py, s, o, d);
                        }
                        // (every camera launch carries the origin-relative plane table, see launch_trace_camera)
                        trace_one<MODE == OUT_COUNT, MODE != OUT_COUNT, ER>(p.tree, p.root, o, d, p.cam.tmin, p.cam.tmax,
                                                                            s_first, s_meta, s_list, hs, wc, p.tabrel,
                                                                            p.hull_eye, p.tri_eye);
                }
                const unsigned long long pix = (unsigned long long)ry * W + (px - p.x0);
                if (MODE == OUT_HIT48) {
                        if (active)
                                store_hit48(static_cast<vrt_hit*>(p.out) + pix * spp + s, p.tree, hs, o, d);
                } else if (MODE == OUT_COUNT) {
                        // out = uint64[8]: rays, n_int, n_leaf, n_tri, hits, n_param, n_tie, n_unsafe
                        unsigned long long v[8] = { active ? 1ull : 0ull, wc.n_int, wc.n_leaf, wc.n_tri,
                                                    (active && hs.hit) ? 1ull : 0ull, wc.n_param, wc.n_tie, wc.n_unsafe };
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
#pragma unroll
                                for (int o2 = 16; o2 > 0; o2 >>= 1)
                                        v[k] += __shfl_down_sync(0xffffffffu, v[k], o2);
                                if (lane == 0)
                                        atomicAdd(static_cast<unsigned long long*>(p.out) + k, v[k]);
                        }
                } else if (MODE == OUT_SPLAT) {
                        // light-map pass (main.cc:81-96): key = (leaf, ray index in the reference's sequential
                        // loop order), record = ISect.normal and illum = get_diffuse(isect, ray, (1,1,1)) =
                        // albedo * clamp(dot(normal, -ray.d), 0, 1) * color (voxel_octree.cc:462-469)
                        if (active) {
                                unsigned long long key = ~0ull;
                                float4 rec0 = make_float4(0.f, 0.f, 0.f, 0.f), rec1 = rec0;
                                if (hs.hit) {
                                        float pos[3], nrm[3], albedo[3];
                                        finish_isect(p.tree, hs, o, d, pos, nrm);
                                        gi_albedo(p.tree, hs.tri, pos, p.kd3, albedo);
                                        const float tmp = clampf(dot3(nrm[0], nrm[1], nrm[2], -d[0], -d[1], -d[2]), 0.f, 1.f);
                                        rec0 = make_float4(nrm[0], nrm[1], nrm[2], fmul(fmul(albedo[0], tmp), 1.f));
                                        rec1 = make_float4(fmul(fmul(albedo[1], tmp), 1.f), fmul(fmul(albedo[2], tmp), 1.f), 0.f, 0.f);
                                        key = ((unsigned long long)(hs.leaf - (p.tree.num_nodes - p.tree.num_leaves)) << 32) |
                                              (unsigned long long)(pix * spp + s);
                                }
                                static_cast<unsigned long long*>(p.out)[pix * spp + s] = key;
                                static_cast<float4*>(p.out2)[2 * (pix * spp + s)] = rec0;
                                static_cast<float4*>(p.out2)[2 * (pix * spp + s) + 1] = rec1;
                        }
                } else if (MODE == OUT_HIT16) {  // (OUT_HIT16_FILM handled below)
                        if (active) {
                                uint4 q;
                                q.x = hs.hit ? (hs.leaf - p.tree.num_nodes + p.tree.num_leaves) : VRT_NO_TRI;
                                q.y = hs.tri;
                                q.z = __float_as_uint(hs.hit ? hs.t : 0.f);
                                q.w = hs.hit ? 1u : 0u;
                                VRT_STORE_OUT(reinterpret_cast<uint4*>(p.out) + (pix * spp + s), q);
                        }
                } else {
                        // the hit records of OUT_HIT16_FILM and OUT_GI_AOV, stored before shading (hs is then dead
                        // during the cone trace)
                        if ((MODE == OUT_HIT16_FILM || (MODE == OUT_GI_AOV && p.aov.hits)) && active) {
                                uint4 q;
                                q.x = hs.hit ? (hs.leaf - p.tree.num_nodes + p.tree.num_leaves) : VRT_NO_TRI;
                                q.y = hs.tri;
                                q.z = __float_as_uint(hs.hit ? hs.t : 0.f);
                                q.w = hs.hit ? 1u : 0u;
                                VRT_STORE_OUT(reinterpret_cast<uint4*>(MODE == OUT_GI_AOV ? (void*)p.aov.hits : p.out) +
                                                      (pix * spp + s),
                                              q);
                        }
                        float rgb[3] = { 0, 0, 0 };
                        GiTerms g = {};
                        if (active) {
                                if (MODE == OUT_GI_FILM || MODE == OUT_GI_AOV)
                                        shade_gi(p, hs, o, d, s_first, rgb, g);
                                else
                                        shade<MODE == OUT_COUNT, WS>(p, hs, o, d, s_first, s_meta, s_list, wc, rgb);
                        }
                        float acc[3];
                        accumulate_samples(rgb, spp, acc);
                        void* const film = (MODE == OUT_HIT16_FILM) ? p.out2 : p.out;
                        if (active && s == 0 && (MODE != OUT_GI_AOV || film)) {
                                const unsigned long long fpix = (MODE == OUT_HIT16_FILM && p.film_full)
                                                                    ? (unsigned long long)py * p.cam.nx + px
                                                                    : pix;
                                if (p.film_fmt == VRT_FILM_F32) {
                                        float* f = static_cast<float*>(film) + fpix * 3ull;
                                        VRT_STORE_OUT(f + 0, acc[0]);
                                        VRT_STORE_OUT(f + 1, acc[1]);
                                        VRT_STORE_OUT(f + 2, acc[2]);
                                } else if (p.film_fmt == VRT_FILM_RGBE) {  // the film as stbi_write_hdr encodes it
                                        VRT_STORE_OUT(static_cast<uint32_t*>(film) + fpix, film_rgbe(acc));
                                } else {  // Film::to_byte_array
                                        const uint32_t v = film_rgb8(acc);
                                        uint8_t* f = static_cast<uint8_t*>(film) + fpix * 3ull;
                                        f[0] = (uint8_t)v;
                                        f[1] = (uint8_t)(v >> 8);
                                        f[2] = (uint8_t)(v >> 16);
                                }
                        }
                        if (MODE == OUT_GI_AOV) {
                                // the planes accumulate exactly as the film does (f32 whatever the film format); the
                                // null tests are uniform
                                float* const planes[4] = { p.aov.albedo, p.aov.direct, p.aov.indirect, p.aov.normal };
                                const float* const terms[4] = { g.albedo, g.dir, g.ind, g.nrm };
#pragma unroll
                                for (int i = 0; i < 4; ++i) {
                                        if (!planes[i])
                                                continue;
                                        accumulate_samples(terms[i], spp, acc);
                                        if (active && s == 0) {
                                                float* f = planes[i] + pix * 3ull;
                                                VRT_STORE_OUT(f + 0, acc[0]);
                                                VRT_STORE_OUT(f + 1, acc[1]);
                                                VRT_STORE_OUT(f + 2, acc[2]);
                                        }
                                }
                        }
                }
                __syncwarp();
        }
}

// Origin-relative axis tables of a camera launch: rel[i] = tab[i] - eye[axis] for the three axes (contiguous:
// n4 float4 entries per axis).  fsub = the reference's (plane - o), rounded once, exactly as the expansion would.
__global__ void __launch_bounds__(256) k_tab_rel(const float4* __restrict__ tab, uint32_t n4, float ex, float ey, float ez,
                                                 float4* __restrict__ rel)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= 3u * n4)
                return;
        const float e = (i < n4) ? ex : (i < 2u * n4) ? ey : ez;
        const float4 t = tab[i];
        rel[i] = make_float4(fsub(t.x, e), fsub(t.y, e), fsub(t.z, e), fsub(t.w, e));
}

// Eye-relative hull records of a camera launch: the records of TreeDev::hull (n interior nodes) with their six planes
// minus the eye -- fsub, the (plane - o) of hull_reachable rounded once -- and the first-child and mask words unchanged,
// so that a record is still the node record of the expansion.
__global__ void __launch_bounds__(256) k_hull_eye_rel(const float4* __restrict__ hull, uint64_t n, float ex, float ey,
                                                      float ez, float4* __restrict__ out)
{
        const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        const float4 a = hull[2 * i], b = hull[2 * i + 1];
        out[2 * i] = make_float4(a.x, a.y, fsub(a.z, ex), fsub(a.w, ex));
        out[2 * i + 1] = make_float4(fsub(b.x, ey), fsub(b.y, ey), fsub(b.z, ez), fsub(b.w, ez));
}

// Eye-relative triangle terms (kTriEyeDoubles per triangle, see leaf_isect_rec): from tri64's v0, e1, e2 the tv, qv and
// e2 . qv that ray_triangle3_edges evaluates for a ray from the eye, with its operations in its order.
__global__ void __launch_bounds__(256) k_tri_eye_rel(const double* __restrict__ tri64, uint32_t T, float ex, float ey,
                                                     float ez, double* __restrict__ out)
{
        const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= T)
                return;
        const double* q = tri64 + 10ull * t;
        const double a[3] = { q[0], q[1], q[2] }, e1[3] = { q[3], q[4], q[5] }, e2[3] = { q[6], q[7], q[8] };
        const double o[3] = { (double)ex, (double)ey, (double)ez };
        double tv[3], qv[3];
#pragma unroll
        for (int k = 0; k < 3; ++k)
                tv[k] = dsub(o[k], a[k]);
        dcross(qv, tv, e1);
        const double r[kTriEyeDoubles] = { e2[0], e2[1], e2[2], e1[0], e1[1], e1[2], tv[0],
                                           tv[1], tv[2], qv[0], qv[1], qv[2], ddot3(e2, qv), 0.0 };
        double2* w = reinterpret_cast<double2*>(out + kTriEyeDoubles * (uint64_t)t);
#pragma unroll
        for (int k = 0; k < (int)kTriEyeDoubles / 2; ++k)
                w[k] = make_double2(r[2 * k], r[2 * k + 1]);
}

// The slot of `slots` whose records are those of `eye`: a slot that holds them, else the least recently used one,
// refilled on `ls` by fill(k) once every launch that read it since its last fill (on any stream, rel_slot_read) is
// done.  Launches of consecutive frames may overlap on two streams: a launch on another stream than the one that
// filled the slot waits for the fill through the slot's event.
template <class Fill>
static int rel_slot_for_launch(vrt_tree::RelSlot* slots, int n, uint64_t& clock, const float eye[3], cudaStream_t ls,
                               Fill fill, int* out)
{
        int k = -1;
        for (int i = 0; i < n; ++i)
                if (slots[i].valid && memcmp(slots[i].eye, eye, 12) == 0)
                        k = i;
        if (k < 0) {
                k = 0;
                for (int i = 1; i < n; ++i)
                        if (slots[i].last_use < slots[k].last_use)
                                k = i;
                auto& s = slots[k];
                if (!s.ev)
                        VRT_CUDA(cudaEventCreateWithFlags(&s.ev, cudaEventDisableTiming));
                for (int i = 0; i < s.n_read; ++i)
                        VRT_CUDA(cudaStreamWaitEvent(ls, s.read_ev[i], 0));
                s.n_read = 0;
                s.valid = false;
                if (int rc = fill(k))
                        return rc;
                VRT_CUDA(cudaEventRecord(s.ev, ls));
                memcpy(s.eye, eye, 12);
                s.valid = true;
                s.done = false;
                s.stream = ls;
        }
        auto& s = slots[k];
        if (!s.done) {
                if (cudaEventQuery(s.ev) == cudaSuccess)
                        s.done = true;
                else if (s.stream != ls)
                        VRT_CUDA(cudaStreamWaitEvent(ls, s.ev, 0));
                cudaGetLastError();  // (cudaErrorNotReady is not an error here)
        }
        s.last_use = ++clock;
        *out = k;
        return VRT_OK;
}

// After a launch on `ls` that reads slot s: the slot's read event of that stream is recorded behind it.  When every
// entry belongs to another stream, this stream takes over entry 0 after waiting for its event, so that the new event
// still completes only after that stream's readers.
static int rel_slot_read(vrt_tree::RelSlot& s, cudaStream_t ls)
{
        int i = 0;
        while (i < s.n_read && s.read_stream[i] != ls)
                ++i;
        if (i == vrt_tree::RelSlot::kReaders) {
                i = 0;
                VRT_CUDA(cudaStreamWaitEvent(ls, s.read_ev[0], 0));
        } else if (i == s.n_read) {
                s.n_read++;
        }
        if (!s.read_ev[i])
                VRT_CUDA(cudaEventCreateWithFlags(&s.read_ev[i], cudaEventDisableTiming));
        s.read_stream[i] = ls;
        VRT_CUDA(cudaEventRecord(s.read_ev[i], ls));
        return VRT_OK;
}

// The origin-relative axis tables for (tree contents, eye), cached per handle: a frame loop with a fixed camera builds
// them once.
static int tab_rel_for_launch(const vrt_tree* t, const float eye[3], cudaStream_t ls, const float4* out[3])
{
        const uint64_t n4 = t->hdr.axis_tab_stride / 2;  // float4 entries per axis
        const uint64_t slot_bytes = 3 * n4 * sizeof(float4);
        if (t->tabrel_buf.cap < vrt_tree::kRelSlots * slot_bytes || t->tabrel_blob != t->blob ||
            t->tabrel_build != t->n_builds) {
                VRT_CUDA(cudaDeviceSynchronize());  // (first launch after a build: nothing may still read the old tables)
                for (auto& s : t->tabrel_slot) {
                        s.valid = false;
                        s.n_read = 0;
                }
                if (t->tabrel_buf.reserve(vrt_tree::kRelSlots * slot_bytes))
                        return VRT_ERR_NOMEM;
                t->tabrel_blob = t->blob;
                t->tabrel_build = t->n_builds;
        }
        auto fill = [&](int k) -> int {
                float4* dst = reinterpret_cast<float4*>(static_cast<char*>(t->tabrel_buf.p) + k * slot_bytes);
                k_tab_rel<<<(unsigned)((3 * n4 + 255) / 256), 256, 0, ls>>>(t->dev.tab4[0], (uint32_t)n4, eye[0], eye[1], eye[2], dst);
                count_launch();
                VRT_CUDA(cudaGetLastError());
                return VRT_OK;
        };
        int k = 0;
        if (int rc = rel_slot_for_launch(t->tabrel_slot, vrt_tree::kRelSlots, t->tabrel_clock, eye, ls, fill, &k))
                return rc;
        t->tabrel_cur = k;
        const float4* base = reinterpret_cast<const float4*>(static_cast<const char*>(t->tabrel_buf.p) + k * slot_bytes);
        for (int a = 0; a < 3; ++a)
                out[a] = base + a * n4;
        return VRT_OK;
}

// The eye-relative hull records and triangle terms for (tree contents, eye), cached per handle like the tables above
// (fewer slots: a slot is 32 bytes per interior node and 112 per triangle).  vrt_update_* rebuilds, which bumps n_builds.
// VRT_ERR_NOMEM: no room for the slots; the caller launches with the absolute records instead, and the reservation is
// not tried again before the next build.
static uint64_t eye_rel_hull_bytes(const vrt_tree* t)
{
        return align256((t->hdr.num_nodes - t->hdr.num_leaves) * 2 * sizeof(float4));
}
static uint64_t eye_rel_slot_bytes(const vrt_tree* t)
{
        return eye_rel_hull_bytes(t) + align256((uint64_t)t->hdr.num_tris * kTriEyeDoubles * sizeof(double));
}
static bool eye_rel_cached(const vrt_tree* t, const float eye[3])
{
        if (t->eyerel_blob != t->blob || t->eyerel_build != t->n_builds)
                return false;
        for (const auto& s : t->eyerel_slot)
                if (s.valid && memcmp(s.eye, eye, 12) == 0)
                        return true;
        return false;
}
static int eye_rel_for_launch(const vrt_tree* t, const float eye[3], cudaStream_t ls, const float4** hull_eye,
                              const double** tri_eye)
{
        const uint64_t interior = t->hdr.num_nodes - t->hdr.num_leaves, T = t->hdr.num_tris;
        const uint64_t hull_bytes = eye_rel_hull_bytes(t), slot_bytes = eye_rel_slot_bytes(t);
        const bool current = t->eyerel_blob == t->blob && t->eyerel_build == t->n_builds;
        if (current && t->eyerel_nomem)
                return VRT_ERR_NOMEM;
        if (!current || t->eyerel_buf.cap < vrt_tree::kEyeRelSlots * slot_bytes) {
                VRT_CUDA(cudaDeviceSynchronize());  // (first launch after a build: nothing may still read the old records)
                for (auto& s : t->eyerel_slot) {
                        s.valid = false;
                        s.n_read = 0;
                }
                t->eyerel_blob = t->blob;
                t->eyerel_build = t->n_builds;
                t->eyerel_nomem = t->eyerel_buf.reserve(vrt_tree::kEyeRelSlots * slot_bytes) != 0;
                if (t->eyerel_nomem)
                        return VRT_ERR_NOMEM;
        }
        auto fill = [&](int k) -> int {
                char* base = static_cast<char*>(t->eyerel_buf.p) + k * slot_bytes;
                if (interior) {
                        k_hull_eye_rel<<<(unsigned)((interior + 255) / 256), 256, 0, ls>>>(t->dev.hull, interior, eye[0], eye[1],
                                                                                          eye[2], reinterpret_cast<float4*>(base));
                        count_launch();
                }
                if (T) {
                        k_tri_eye_rel<<<(unsigned)((T + 255) / 256), 256, 0, ls>>>(t->dev.tri64, (uint32_t)T, eye[0], eye[1], eye[2],
                                                                                  reinterpret_cast<double*>(base + hull_bytes));
                        count_launch();
                }
                VRT_CUDA(cudaGetLastError());
                return VRT_OK;
        };
        int k = 0;
        if (int rc = rel_slot_for_launch(t->eyerel_slot, vrt_tree::kEyeRelSlots, t->eyerel_clock, eye, ls, fill, &k))
                return rc;
        t->eyerel_cur = k;
        const char* base = static_cast<const char*>(t->eyerel_buf.p) + k * slot_bytes;
        *hull_eye = reinterpret_cast<const float4*>(base);
        *tri_eye = reinterpret_cast<const double*>(base + hull_bytes);
        return VRT_OK;
}

// The film encodings of the camera kernels applied to a float film that already exists (vrt_film_encode).
__global__ void __launch_bounds__(256) k_film_encode(const float* __restrict__ film, unsigned long long npix, int fmt,
                                                     uint8_t* __restrict__ out)
{
        const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= npix)
                return;
        const float c[3] = { film[3 * i], film[3 * i + 1], film[3 * i + 2] };
        if (fmt == VRT_FILM_RGBE) {
                reinterpret_cast<uint32_t*>(out)[i] = film_rgbe(c);
        } else {
                const uint32_t v = film_rgb8(c);
                out[3 * i] = (uint8_t)v;
                out[3 * i + 1] = (uint8_t)(v >> 8);
                out[3 * i + 2] = (uint8_t)(v >> 16);
        }
}

int launch_film_encode(const vrt_tree* t, const float* d_film, uint64_t npix, int fmt, uint8_t* d_out)
{
        if (!npix)
                return VRT_OK;
        k_film_encode<<<(unsigned)((npix + 255) / 256), 256, 0, t->stream>>>(d_film, npix, fmt, d_out);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        return VRT_OK;
}

// ---------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------
static int g_sm_count = 0;

static int persistent_grid(const void* kernel, size_t smem)
{
        if (!g_sm_count) {
                int dev = 0;
                cudaGetDevice(&dev);
                cudaDeviceGetAttribute(&g_sm_count, cudaDevAttrMultiProcessorCount, dev);
                if (g_sm_count <= 0)
                        g_sm_count = 148;
        }
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kTraceThreads, smem) != cudaSuccess ||
            per_sm < 1) {
                cudaGetLastError();
                per_sm = 4;
        }
        return g_sm_count * per_sm;
}

// Traversal stack: one 3-word record per thread for the bottom sentinel and for every level
// that can be left with unvisited children (levels 0 .. L-1).
static size_t stack_bytes(const vrt_tree* t, OutMode mode = OUT_HIT48)
{
        const int L = std::max(t->dev.L, 1);
        size_t words = (size_t)3 * (size_t)(L + 1);
        if (mode == OUT_GI_FILM || mode == OUT_GI_AOV)  // the same column then holds the cone trace's path cache (vrt_gi.cuh)
                words = std::max(words, (size_t)kGiPathWords * (size_t)L);
        return words * kTraceThreads * sizeof(uint32_t);
}

// L2 access-policy window (north star: "top octree levels pinned in L2"): the node array is in BFS order,
// so the records of the top levels are one contiguous prefix.  The prefix that fits the device's persisting
// L2 carve-out (and the window limit) is marked persisting on the launch stream, everything else -- above all
// the 16 B/ray + 12 B/pixel output stream -- is left normal.  Measured on the headline frame (ncu, profiles/
// r1q_l2_window_ab.txt): node reads already hit L2 (82 %) and DRAM reads are 40 MB per frame either way,
// while the carve-out takes L2 away from the output stream (DRAM writes 0.60 -> 1.26 GB); 7.72 vs 7.73 ms.
// It is therefore OFF by default; VRT_L2_WINDOW=1 turns it on.
static void apply_l2_window(const vrt_tree* t)
{
        static int enabled = -1, max_window = 0, max_persist = 0;
        if (enabled < 0) {
                const char* e = getenv("VRT_L2_WINDOW");
                enabled = (e && e[0] == '1') ? 1 : 0;
                int dev = 0;
                cudaGetDevice(&dev);
                cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev);
                cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
                if (enabled && max_persist > 0)
                        cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)max_persist);
                cudaGetLastError();
        }
        if (!enabled || max_window <= 0 || max_persist <= 0 || t->hdr.num_nodes == 0)
                return;
        if (t->l2_window_stream == (void*)t->stream && t->l2_window_nodes == (const void*)t->dev.nodes)
                return;
        // whole levels from the root down while they fit
        const uint64_t cap = std::min<uint64_t>((uint64_t)max_window, (uint64_t)max_persist);
        uint64_t bytes = 0;
        for (int l = 0; l <= t->hdr.max_depth - 1; ++l) {
                const uint64_t upto = t->hdr.level_offset[l + 1] * 8ull;
                if (upto > cap)
                        break;
                bytes = upto;
        }
        if (!bytes)
                return;
        cudaStreamAttrValue v{};
        v.accessPolicyWindow.base_ptr = const_cast<uint2*>(t->dev.nodes);
        v.accessPolicyWindow.num_bytes = bytes;
        v.accessPolicyWindow.hitRatio = 1.0f;
        v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        v.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
        if (cudaStreamSetAttribute(t->stream, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess)
                cudaGetLastError();
        t->l2_window_stream = (void*)t->stream;
        t->l2_window_nodes = (const void*)t->dev.nodes;
        t->l2_window_bytes = bytes;
}

// every tree with interior levels carries hull records (compute_hulls after every build / import / replica): the
// ray kernels read the node records from them
static int check_hull_records(const vrt_tree* t)
{
        if (t->hdr.num_nodes != 0 && ((t->dev.L >= 1 && t->dev.hull == nullptr) || (t->hdr.num_tris && t->dev.tri64 == nullptr))) {
                set_error("octree has no hull / widened-triangle records (compute_hulls did not run)");
                return VRT_ERR_STATE;
        }
        return VRT_OK;
}

static void fill_common(const vrt_tree* t, TraceParams& p)
{
        apply_l2_window(t);
        p.tree = t->dev;
        for (int k = 0; k < 6; ++k)
                p.root[k] = t->hdr.root_aabb[k];
        // one work-queue counter per in-flight launch (launches on alternating streams may
        // overlap): 8 slots
        p.queue = t->d_counter + 16 + 2 * (t->n_trace_launches % 8);
}

int launch_trace_rays(const vrt_tree* t, const vrt_ray* d_rays, uint64_t n, vrt_hit* d_out)
{
        if (n == 0)
                return VRT_OK;
        if ((n + 31) / 32 >= 0xffffffffull) {
                set_error("too many rays for one launch");
                return VRT_ERR_ARG;
        }
        if (int rc = check_hull_records(t))
                return rc;
        TraceParams p{};
        fill_common(t, p);
        p.rays = d_rays;
        p.num_rays = n;
        p.out = d_out;
        const size_t smem = stack_bytes(t);
        VRT_CUDA(cudaFuncSetAttribute(k_trace_rays, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const uint64_t warps = (n + 31) / 32;
        int grid = persistent_grid((const void*)k_trace_rays, smem);
        grid = (int)std::min<uint64_t>((uint64_t)grid, (warps + 3) / 4);
        VRT_CUDA(cudaMemsetAsync(p.queue, 0, 4, t->stream));
        const int slot = (int)(t->n_trace_launches % vrt_tree::kEvRing);
        VRT_CUDA(cudaEventRecord(t->ring0[slot], t->stream));
        k_trace_rays<<<grid, kTraceThreads, smem, t->stream>>>(p);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        VRT_CUDA(cudaEventRecord(t->ring1[slot], t->stream));
        t->n_trace_launches++;
        return VRT_OK;
}

// gen_ray_origin on the host: the same IEEE single-precision operations in the same order (this file's host code is
// compiled without contraction or fast-math, so x * 0.f and the sums of zeros are evaluated, not folded)
static void camera_eye_host(const vrt_camera* cam, float eye[3])
{
        volatile float o4[4];
        for (int r = 0; r < 4; ++r) {
                volatile float a = 0.f + cam->C[r] * 0.f;
                a = a + cam->C[4 + r] * 0.f;
                a = a + cam->C[8 + r] * 0.f;
                a = a + cam->C[12 + r] * 1.f;
                o4[r] = a;
        }
        for (int k = 0; k < 3; ++k)
                eye[k] = o4[k] / o4[3];
}

int launch_trace_camera(const vrt_tree* t, const CameraLaunch& l)
{
        const vrt_camera* cam = l.cam;
        const int x0 = l.x0, y0 = l.y0, x1 = l.x1, y1 = l.y1;
        const OutMode mode = l.mode;
        if (x1 <= x0 || y1 <= y0)
                return VRT_OK;
        if (int rc = check_hull_records(t))
                return rc;
        TraceParams p{};
        fill_common(t, p);
        for (int k = 0; k < 16; ++k)
                p.cam.C[k] = cam->C[k];
        camera_eye_host(cam, p.eye);
        p.cam.z = cam->z;
        p.cam.tmin = cam->tmin;
        p.cam.tmax = cam->tmax;
        p.cam.nx = cam->nx;
        p.cam.ny = cam->ny;
        p.cam.spp = cam->spp;
        p.x0 = x0;
        p.y0 = y0;
        p.x1 = x1;
        p.y1 = y1;
        p.band_h = l.band_h > 0 ? l.band_h : (y1 - y0);
        p.band_pitch = l.band_h > 0 ? l.band_pitch : 0;
        p.out = l.out;
        p.out2 = l.out2;
        p.film_full = l.film_full;
        p.film_fmt = t->film_fmt;
        p.kd3[0] = l.kd[0];
        p.kd3[1] = l.kd[1];
        p.kd3[2] = l.kd[2];
        p.gi_res = l.res;
        p.aov = l.aov;
        if (l.sh) {
                p.light[0] = l.sh->light_dir[0];
                p.light[1] = l.sh->light_dir[1];
                p.light[2] = l.sh->light_dir[2];
                p.kd = l.sh->kd;
                p.shadow = l.sh->shadow;
                p.shadow_eps = l.sh->shadow_eps;
        }
        const int tw = (cam->spp == 4) ? 4 : 8, th = (cam->spp == 4) ? 2 : 4;
        const uint64_t tiles = (uint64_t)((x1 - x0 + tw - 1) / tw) * (uint64_t)((y1 - y0 + th - 1) / th);
        if (tiles >= 0xfff00000ull) {  // (the prefetching queue overshoots by one fetch per warp)
                set_error("too many tiles for one launch");
                return VRT_ERR_ARG;
        }
        p.num_tiles = (uint32_t)tiles;
#ifndef VRT_TILE_GLOBAL
        {
                const uint32_t tiles_x = (uint32_t)((x1 - x0 + tw - 1) / tw), tiles_y = (uint32_t)((y1 - y0 + th - 1) / th);
                constexpr uint32_t bs = 1u << kTileBlockLog;
                p.blocks_x = (tiles_x + bs - 1u) / bs;
                p.tiles_y = tiles_y;
                const uint64_t padded = (uint64_t)p.blocks_x * ((tiles_y + bs - 1u) / bs) * (uint64_t)(bs * bs);
                if (padded >= 0xfff00000ull) {
                        set_error("too many tiles for one launch");
                        return VRT_ERR_ARG;
                }
                p.num_tiles = (uint32_t)padded;
                persistent_grid((const void*)k_trace_rays, 0);  // (g_sm_count)
                p.num_queues = (uint32_t)std::min(g_sm_count, (int)kQueueBitmap);
                p.queue_chunk = (p.num_tiles + p.num_queues - 1u) / p.num_queues;
                p.queue = t->d_tile_queues + (size_t)vrt_tree::kTileQueues * (t->n_trace_launches % 8);
        }
#endif
        // per-ray kernels by default; VRT_TRACE_WS=1 selects the warp-synchronous kernels (measured slower so
        // far, see DESIGN.md): the child-mask table of trace_tile_ws follows the stack in dynamic shared memory
        static int use_ws = -1;
        if (use_ws < 0) {
                const char* e = getenv("VRT_TRACE_WS");
                use_ws = (e && e[0] == '1') ? 1 : 0;
        }
        const bool ws = use_ws != 0;
        cudaStream_t ls = l.stream;
        // every camera launch but the counting mode reads the origin-relative tables; the per-ray kernels of the film
        // and hit16 modes (the ones measured with them) also the eye-relative hull records and triangle terms, unless
        // they are switched off or do not fit in memory
        const bool use_rel = mode != OUT_COUNT && t->hdr.num_nodes != 0 && t->dev.L >= 1;
        const bool er_mode = mode == OUT_HIT16 || mode == OUT_HIT16_FILM || mode == OUT_FILM;
        bool er = false;
        if (use_rel) {
                const int rc = tab_rel_for_launch(t, p.eye, ls, p.tabrel);
                if (rc)
                        return rc;
                // (launches with shadow rays keep them off: measured on config 5, 2048^3 8K orbit + shadow rays, with
                // them the frame went from 56.28 to 56.59 ms on B200, DESIGN.md section 5)
                if (!ws && er_mode && t->eyerel_on && !(l.sh && l.sh->shadow)) {
                        // a slot fill reads and writes about a slot's bytes; it pays for itself from about one ray per
                        // 13 slot bytes (B200, DESIGN.md section 5: the 2048^3 tree's 595 MB slot costs 0.22 ms, a ray
                        // saves 5 ps).  Smaller launches with a new eye keep the per-ray subtraction; an eye seen by the
                        // previous launch (a fixed camera) is filled on its second launch and reused from then on.
                        const uint64_t rays = (uint64_t)(x1 - x0) * (uint64_t)(y1 - y0) * (uint64_t)cam->spp;
                        if (rays * 13 >= eye_rel_slot_bytes(t) || memcmp(t->eyerel_last, p.eye, 12) == 0 ||
                            eye_rel_cached(t, p.eye)) {
                                const int rc2 = eye_rel_for_launch(t, p.eye, ls, &p.hull_eye, &p.tri_eye);
                                if (rc2 && rc2 != VRT_ERR_NOMEM)
                                        return rc2;
                                er = rc2 == VRT_OK;
                        }
                        memcpy(t->eyerel_last, p.eye, 12);
                }
        }
        p.lut_off = (uint32_t)stack_bytes(t, mode);
        const size_t smem = stack_bytes(t, mode) + (ws ? (size_t)kWsLutBytes : 0);
        const void* kern = nullptr;
#define VRT_PICK(M) kern = ws ? (const void*)k_trace_camera<M, true, false> : (const void*)k_trace_camera<M, false, false>
#define VRT_PICK_ER(M) \
        kern = er ? (const void*)k_trace_camera<M, false, true> : ws ? (const void*)k_trace_camera<M, true, false> \
                                                                      : (const void*)k_trace_camera<M, false, false>
        switch (mode) {
        case OUT_HIT48: VRT_PICK(OUT_HIT48); break;
        case OUT_HIT16: VRT_PICK_ER(OUT_HIT16); break;
        case OUT_COUNT: VRT_PICK(OUT_COUNT); break;
        case OUT_HIT16_FILM: VRT_PICK_ER(OUT_HIT16_FILM); break;
        case OUT_SPLAT: VRT_PICK(OUT_SPLAT); break;
        case OUT_GI_FILM: VRT_PICK(OUT_GI_FILM); break;
        case OUT_GI_AOV: VRT_PICK(OUT_GI_AOV); break;
        default: VRT_PICK_ER(OUT_FILM); break;
        }
#undef VRT_PICK_ER
#undef VRT_PICK
        VRT_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int grid = persistent_grid(kern, smem);
        grid = (int)std::min<uint64_t>((uint64_t)grid, (tiles + 3) / 4);
        if (mode == OUT_GI_FILM || mode == OUT_GI_AOV) {
                const int rc = gi_step_table(t, l.res, ls, &p.gi_steps);
                if (rc)
                        return rc;
        }
#ifndef VRT_TILE_GLOBAL
        VRT_CUDA(cudaMemsetAsync(p.queue, 0, sizeof(uint32_t) * vrt_tree::kTileQueues, ls));
#else
        VRT_CUDA(cudaMemsetAsync(p.queue, 0, 4, ls));
#endif
        const int slot = (int)(t->n_trace_launches % vrt_tree::kEvRing);
        VRT_CUDA(cudaEventRecord(t->ring0[slot], ls));
        void* args[] = { &p };
        VRT_CUDA(cudaLaunchKernel(kern, dim3(grid), dim3(kTraceThreads), args, smem, ls));
        count_launch();
        VRT_CUDA(cudaEventRecord(t->ring1[slot], ls));
        // (a later launch that re-fills these slots waits for this reader)
        if (use_rel)
                if (int rc = rel_slot_read(t->tabrel_slot[t->tabrel_cur], ls))
                        return rc;
        if (er) {
                if (int rc = rel_slot_read(t->eyerel_slot[t->eyerel_cur], ls))
                        return rc;
                t->n_eyerel_launches++;
        }
        t->n_trace_launches++;
        return VRT_OK;
}

int hull_stats(unsigned long long* out80)
{
#ifdef VRT_HULL_STATS
        VRT_CUDA(cudaDeviceSynchronize());
        VRT_CUDA(cudaMemcpyFromSymbol(out80, g_hull_stats, sizeof(unsigned long long) * 80));
        unsigned long long z[80] = { 0 };
        VRT_CUDA(cudaMemcpyToSymbol(g_hull_stats, z, sizeof z));
#else
        for (int i = 0; i < 80; ++i)
                out80[i] = 0;
#endif
        return VRT_OK;
}

int general_order_calls(unsigned long long* out)
{
        VRT_CUDA(cudaDeviceSynchronize());
        VRT_CUDA(cudaMemcpyFromSymbol(out, g_general_calls, sizeof(unsigned long long)));
        return VRT_OK;
}

// {expansions cross-checked against expand_slab, mismatches}; only a library built with
// -DVRT_PARAM_CHECK counts (tests/test_gpu_param_check.py), otherwise {0, 0}.
int param_check_counts(unsigned long long out[2])
{
        out[0] = out[1] = 0;
#ifdef VRT_PARAM_CHECK
        unsigned long long v[4];
        VRT_CUDA(cudaDeviceSynchronize());
        VRT_CUDA(cudaMemcpyFromSymbol(v, g_param_check, sizeof v));
        out[0] = v[0];
        out[1] = v[1];
#endif
        return VRT_OK;
}

int trace_ms_mean(const vrt_tree* t, int last_n, double* ms)
{
        *ms = 0;
        const uint64_t n = t->n_trace_launches;
        if (n == 0)
                return VRT_OK;
        const int cnt = (int)std::min<uint64_t>({ (uint64_t)std::max(last_n, 1), n, (uint64_t)vrt_tree::kEvRing });
        double sum = 0;
        for (int i = 0; i < cnt; ++i) {
                const int slot = (int)((n - 1 - i) % vrt_tree::kEvRing);
                VRT_CUDA(cudaEventSynchronize(t->ring1[slot]));
                float e = 0;
                VRT_CUDA(cudaEventElapsedTime(&e, t->ring0[slot], t->ring1[slot]));
                sum += e;
        }
        *ms = sum / cnt;
        return VRT_OK;
}

}  // namespace vrt
