// vrt_build.cu -- GPU voxelization + sparse-octree construction.
//
// Replaces gi::ray_march_init / insert / split (voxel_octree.cc:27-75) and the
// Triangle::is_overlap -> triBoxOverlap calls it makes (voxel_octree.cc:486-492,
// tribox2.cc:112-186).  Semantics reproduced exactly (SURVEY.md 8a):
//   * root AABB = union of all triangle AABBs; child boxes by the reference's
//     float recurrence, NOT a closed form (voxel_octree.cc:30-37);
//   * a triangle reaches a leaf cell iff the SAT test passes for that cell AND
//     for every ancestor including the root (hierarchical insert,
//     voxel_octree.cc:43) -- hence a level-synchronous top-down expansion, which
//     is exact by construction;
//   * leaves hold triangle indices in ascending order.
// Pipeline: root AABB reduction -> per-axis interval table -> root filter ->
// L x expand (8 lanes per (triangle, cell) pair, one SAT test per lane; mask pass,
// scan, emit pass: deterministic) -> flat pointerless node array, by one of two drivers:
//   ranked (default, depth >= 5): the frontier carries node ranks, the node arrays come out
//     of the expansion itself, the leaf reference lists out of a counting sort (see
//     "RANKED top-down build" below);
//   sorted (shallow trees, imports, oversize leaves): keys Morton<<tb | tri stay sorted by
//     (triangle, Morton) -> stable LSD radix sort on the Morton bits -> unique -> bottom-up
//     parent derivation.
// Both produce the same bytes.
#include <algorithm>
#include <cfloat>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "vrt_exact.cuh"
#include "vrt_internal.h"
#include "vrt_prims.cuh"

namespace vrt {

// ---------------------------------------------------------------------------
// Morton helpers: 3 bits per level, child digit c = (x<<2)|(y<<1)|z
// (voxel_octree.cc:33: mask = (i&4, i&2, i&1) for (x,y,z)).
// ---------------------------------------------------------------------------
__host__ __device__ inline uint32_t compact1by2(unsigned long long v)
{
        v &= 0x1249249249249249ull;
        v = (v ^ (v >> 2)) & 0x10c30c30c30c30c3ull;
        v = (v ^ (v >> 4)) & 0x100f00f00f00f00full;
        v = (v ^ (v >> 8)) & 0x001f0000ff0000ffull;
        v = (v ^ (v >> 16)) & 0x001f00000000ffffull;
        v = (v ^ (v >> 32)) & 0x00000000001fffffull;
        return (uint32_t)v;
}

__host__ __device__ inline unsigned long long spread1by2(uint32_t x)
{
        unsigned long long v = x & 0x1fffffull;
        v = (v | (v << 32)) & 0x001f00000000ffffull;
        v = (v | (v << 16)) & 0x001f0000ff0000ffull;
        v = (v | (v << 8)) & 0x100f00f00f00f00full;
        v = (v | (v << 4)) & 0x10c30c30c30c30c3ull;
        v = (v | (v << 2)) & 0x1249249249249249ull;
        return v;
}

__host__ __device__ inline unsigned long long morton_encode(uint32_t x, uint32_t y, uint32_t z)
{
        return (spread1by2(x) << 2) | (spread1by2(y) << 1) | spread1by2(z);
}

// ---------------------------------------------------------------------------
// Root AABB: min/max over all vertices in index order, std::min/std::max
// semantics (ties keep the EARLIEST element, which only matters for the sign
// of a zero) -- graphics_math.h:1228-1266 via voxel_octree.cc:70-72,430.
// ---------------------------------------------------------------------------
struct MinMaxIdx {
        float v;
        uint32_t i;
};
__device__ __forceinline__ void mm_min(MinMaxIdx& a, float v, uint32_t i)
{
        if (v < a.v || (v == a.v && i < a.i)) {
                a.v = v;
                a.i = i;
        }
}
__device__ __forceinline__ void mm_max(MinMaxIdx& a, float v, uint32_t i)
{
        if (a.v < v || (v == a.v && i < a.i)) {
                a.v = v;
                a.i = i;
        }
}

// partial[block][12] as (value bits, index) pairs: 3 mins then 3 maxes
__global__ void __launch_bounds__(256)
k_aabb_partial(const float* __restrict__ tri, uint32_t num_verts, uint2* __restrict__ partial)
{
        MinMaxIdx mn[3], mx[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                mn[k] = { FLT_MAX, 0xffffffffu };
                mx[k] = { -FLT_MAX, 0xffffffffu };
        }
        for (uint32_t v = blockIdx.x * blockDim.x + threadIdx.x; v < num_verts;
             v += gridDim.x * blockDim.x) {
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                        float f = tri[3ull * v + k];
                        mm_min(mn[k], f, v);
                        mm_max(mx[k], f, v);
                }
        }
        __shared__ MinMaxIdx sh[6][8];
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                        float ov = __shfl_down_sync(0xffffffffu, mn[k].v, o);
                        uint32_t oi = __shfl_down_sync(0xffffffffu, mn[k].i, o);
                        mm_min(mn[k], ov, oi);
                        ov = __shfl_down_sync(0xffffffffu, mx[k].v, o);
                        oi = __shfl_down_sync(0xffffffffu, mx[k].i, o);
                        mm_max(mx[k], ov, oi);
                }
                if (lane == 0) {
                        sh[k][w] = mn[k];
                        sh[3 + k][w] = mx[k];
                }
        }
        __syncthreads();
        if (threadIdx.x < 6) {
                MinMaxIdx a = sh[threadIdx.x][0];
                for (int i = 1; i < 8; ++i) {
                        if (threadIdx.x < 3)
                                mm_min(a, sh[threadIdx.x][i].v, sh[threadIdx.x][i].i);
                        else
                                mm_max(a, sh[threadIdx.x][i].v, sh[threadIdx.x][i].i);
                }
                partial[blockIdx.x * 6 + threadIdx.x] = make_uint2(__float_as_uint(a.v), a.i);
        }
}

__global__ void k_aabb_final(const uint2* __restrict__ partial, int nblocks, float* __restrict__ out6)
{
        // warp q reduces quantity q (3 mins, 3 maxes) over the block partials
        const int q = threadIdx.x >> 5, lane = threadIdx.x & 31;
        if (q >= 6)
                return;
        MinMaxIdx a = { q < 3 ? FLT_MAX : -FLT_MAX, 0xffffffffu };
        for (int b = lane; b < nblocks; b += 32) {
                uint2 p = partial[b * 6 + q];
                if (q < 3)
                        mm_min(a, __uint_as_float(p.x), p.y);
                else
                        mm_max(a, __uint_as_float(p.x), p.y);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
                float ov = __shfl_down_sync(0xffffffffu, a.v, o);
                uint32_t oi = __shfl_down_sync(0xffffffffu, a.i, o);
                if (q < 3)
                        mm_min(a, ov, oi);
                else
                        mm_max(a, ov, oi);
        }
        if (lane == 0)
                out6[q] = a.v;
}

// ---------------------------------------------------------------------------
// Per-axis interval table (float recurrence of split(), voxel_octree.cc:30-37):
//   size = (max-min)/2 ; child b: min' = min + (float)b*size ; max' = min' + size
// tab[a][(1<<l)+i] = (min,max) of cell i at level l.  One block, level by level.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(1024)
k_axis_table(const float* __restrict__ root6, float2* __restrict__ tab, uint64_t stride, int L)
{
        for (int a = threadIdx.x; a < 3; a += blockDim.x) {
                tab[a * stride + 0] = make_float2(0.f, 0.f);
                tab[a * stride + 1] = make_float2(root6[a], root6[3 + a]);
        }
        __syncthreads();
        for (int l = 0; l < L; ++l) {
                const uint32_t n = 1u << l;
                for (uint32_t j = threadIdx.x; j < 3 * n; j += blockDim.x) {
                        const uint32_t a = j / n, i = j - a * n;
                        const float2 p = tab[a * stride + n + i];
                        const float s = fdiv(fsub(p.y, p.x), 2.f);
                        float2 c0, c1;
                        c0.x = fadd(p.x, fmul(0.f, s));
                        c0.y = fadd(c0.x, s);
                        c1.x = fadd(p.x, fmul(1.f, s));
                        c1.y = fadd(c1.x, s);
                        tab[a * stride + 2 * n + 2 * i] = c0;
                        tab[a * stride + 2 * n + 2 * i + 1] = c1;
                }
                __syncthreads();
        }
}

// ---------------------------------------------------------------------------
// Hierarchical voxelization, one level per step, in two deterministic passes:
//   mask pass : 8 lanes per (triangle, cell) pair, lane c runs the SAT test against
//               child c; the 8 verdicts are stored as one mask byte per pair and the
//               survivors are counted per block (no atomics);
//   (exclusive scan of the block counts)
//   emit pass : every pair writes its surviving children, in child order, at its exact
//               position.
// The output order is (input order, child index).  The level-0 frontier is in triangle
// order, so by induction every frontier is sorted by (triangle, Morton code) -- which lets
// the final sort run on the Morton bits only (stable LSD passes keep the triangle order
// inside a leaf = the reference's insertion order).
// ---------------------------------------------------------------------------
constexpr int kPairsPerBlock = 256;

__device__ __forceinline__ uint32_t block_sum_256(uint32_t v)
{
        __shared__ uint32_t s_w[8];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
                v += __shfl_down_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0)
                s_w[threadIdx.x >> 5] = v;
        __syncthreads();
        uint32_t tot = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
                tot += s_w[i];
        __syncthreads();
        return tot;
}

// exclusive prefix of v over the 256 threads of the block
__device__ __forceinline__ uint32_t block_excl_scan_256(uint32_t v)
{
        __shared__ uint32_t s_w[8];
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        uint32_t inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
                uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o)
                        inc += t;
        }
        if (lane == 31)
                s_w[w] = inc;
        __syncthreads();
        uint32_t woff = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
                woff += (i < w) ? s_w[i] : 0u;
        __syncthreads();
        return woff + inc - v;
}

// Level 0: triangles that overlap the root box (insert's first test at the root,
// voxel_octree.cc:43).  One thread per triangle.
__global__ void __launch_bounds__(256)
k_root_mask(const float* __restrict__ tri, uint32_t T, const float* __restrict__ root6,
            uint8_t* __restrict__ masks, uint32_t* __restrict__ block_counts)
{
        const uint32_t t = blockIdx.x * kPairsPerBlock + threadIdx.x;
        bool ov = false;
        if (t < T) {
                const float* p = tri + 9ull * t;
                float v0[3] = { p[0], p[1], p[2] }, v1[3] = { p[3], p[4], p[5] }, v2[3] = { p[6], p[7], p[8] };
                float mn[3] = { root6[0], root6[1], root6[2] };
                float mx[3] = { root6[3], root6[4], root6[5] };
                ov = tri_overlaps_aabb(mn, mx, v0, v1, v2);
                masks[t] = ov ? 1 : 0;
        }
        const uint32_t tot = block_sum_256(ov ? 1u : 0u);
        if (threadIdx.x == 0)
                block_counts[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(256)
k_root_emit(uint32_t T, const uint8_t* __restrict__ masks, const uint32_t* __restrict__ block_offs,
            unsigned long long* __restrict__ out)
{
        const uint32_t t = blockIdx.x * kPairsPerBlock + threadIdx.x;
        const uint32_t m = (t < T) ? masks[t] : 0u;
        const uint32_t off = block_excl_scan_256(m);
        if (m)
                out[block_offs[blockIdx.x] + off] = (unsigned long long)t;  // Morton code of the root is empty
}

// One level of the hierarchical insert, mask pass.  in keys = morton<<tb | tri.
__global__ void __launch_bounds__(256)
k_expand_mask(const float* __restrict__ tri, const float2* __restrict__ tab, uint64_t stride,
              const unsigned long long* __restrict__ in, uint32_t n_in, int level /* of the input cells */,
              int tb, uint8_t* __restrict__ masks, uint32_t* __restrict__ block_counts)
{
        const uint32_t c = threadIdx.x & 7;
        const uint32_t lane = threadIdx.x & 31;
        const unsigned long long tmask = (1ull << tb) - 1ull;
        const uint32_t child_base = 2u << level;  // table offset of level+1
        uint32_t cnt = 0;
#pragma unroll 1
        for (int it = 0; it < kPairsPerBlock / 32; ++it) {
                const uint32_t idx = blockIdx.x * kPairsPerBlock + it * 32 + (threadIdx.x >> 3);
                bool ov = false;
                if (idx < n_in) {
                        const unsigned long long key = in[idx];
                        const uint32_t t = (uint32_t)(key & tmask);
                        const unsigned long long m = key >> tb;
                        const uint32_t cx = 2u * compact1by2(m >> 2) + ((c >> 2) & 1u);
                        const uint32_t cy = 2u * compact1by2(m >> 1) + ((c >> 1) & 1u);
                        const uint32_t cz = 2u * compact1by2(m) + (c & 1u);
                        const float2 bx = tab[0 * stride + child_base + cx];
                        const float2 by = tab[1 * stride + child_base + cy];
                        const float2 bz = tab[2 * stride + child_base + cz];
                        const float* p = tri + 9ull * t;
                        float v0[3] = { p[0], p[1], p[2] }, v1[3] = { p[3], p[4], p[5] }, v2[3] = { p[6], p[7], p[8] };
                        float mn[3] = { bx.x, by.x, bz.x };
                        float mx[3] = { bx.y, by.y, bz.y };
                        ov = tri_overlaps_aabb(mn, mx, v0, v1, v2);
                }
                const uint32_t bal = __ballot_sync(0xffffffffu, ov);
                if (c == 0 && idx < n_in)
                        masks[idx] = (uint8_t)((bal >> (lane & 24u)) & 0xffu);
                cnt += ov ? 1u : 0u;
        }
        const uint32_t tot = block_sum_256(cnt);
        if (threadIdx.x == 0)
                block_counts[blockIdx.x] = tot;
}

// Emit pass: thread t handles pair blockIdx*256+t and writes its surviving children.
__global__ void __launch_bounds__(256)
k_expand_emit(const unsigned long long* __restrict__ in, uint32_t n_in, int tb,
              const uint8_t* __restrict__ masks, const uint32_t* __restrict__ block_offs,
              unsigned long long* __restrict__ out)
{
        const uint32_t idx = blockIdx.x * kPairsPerBlock + threadIdx.x;
        uint32_t m = 0;
        unsigned long long key = 0;
        if (idx < n_in) {
                m = masks[idx];
                key = in[idx];
        }
        uint32_t pos = block_offs[blockIdx.x] + block_excl_scan_256(__popc(m));
        const unsigned long long t = key & ((1ull << tb) - 1ull);
        const unsigned long long mo = (key >> tb) << 3;
        while (m) {
                const uint32_t c = __ffs((int)m) - 1;
                m &= m - 1u;
                out[pos++] = ((mo | c) << tb) | t;
        }
}

// ---------------------------------------------------------------------------
// After the sort: leaves, refs and the bottom-up parent derivation.
// ---------------------------------------------------------------------------
// flag[i] = 1 where a new code starts ; code(i) = keys[i] >> shift
__global__ void k_head_flags(const unsigned long long* __restrict__ keys, uint64_t n, int shift,
                             uint32_t* __restrict__ flag)
{
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        flag[i] = (i == 0 || (keys[i] >> shift) != (keys[i - 1] >> shift)) ? 1u : 0u;
}

// leaves from sorted keys: pos = exclusive scan of flags.
__global__ void k_emit_leaves(const unsigned long long* __restrict__ keys, uint64_t n, int tb,
                              const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos,
                              unsigned long long* __restrict__ leaf_morton,
                              uint32_t* __restrict__ leaf_start, uint32_t* __restrict__ refs)
{
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        const unsigned long long k = keys[i];
        refs[i] = (uint32_t)(k & ((1ull << tb) - 1ull));
        if (flag[i]) {
                leaf_morton[pos[i]] = k >> tb;
                leaf_start[pos[i]] = (uint32_t)i;
        }
}

// parents of a sorted child-code list: flag where code>>3 changes.
__global__ void k_parent_flags(const unsigned long long* __restrict__ child, uint64_t n,
                               uint32_t* __restrict__ flag)
{
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        flag[i] = (i == 0 || (child[i] >> 3) != (child[i - 1] >> 3)) ? 1u : 0u;
}

__global__ void k_emit_parents(const unsigned long long* __restrict__ child, uint64_t n,
                               const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos,
                               unsigned long long* __restrict__ parent_morton,
                               uint32_t* __restrict__ parent_first, uint32_t* __restrict__ parent_mask)
{
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n || !flag[i])
                return;
        const unsigned long long pm = child[i] >> 3;
        uint32_t mask = 0;
        for (uint64_t j = i; j < n && j < i + 8 && (child[j] >> 3) == pm; ++j)
                mask |= 1u << (uint32_t)(child[j] & 7ull);
        const uint32_t p = pos[i];
        parent_morton[p] = pm;
        parent_first[p] = (uint32_t)i;
        parent_mask[p] = mask;
}

// final node array
__global__ void k_write_interior(const uint32_t* __restrict__ first, const uint32_t* __restrict__ mask,
                                 uint32_t n, uint32_t child_level_offset, uint2* __restrict__ nodes)
{
        uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i < n)
                nodes[i] = make_uint2(first[i] + child_level_offset, mask[i]);
}

__global__ void k_write_leaves(const uint32_t* __restrict__ start, uint32_t n, uint32_t num_refs,
                               uint2* __restrict__ nodes)
{
        uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i < n) {
                uint32_t s = start[i];
                uint32_t e = (i + 1 < n) ? start[i + 1] : num_refs;
                nodes[i] = make_uint2(s, e - s);
        }
}

// vertices -> float4 x3 ; normals normalised like the Triangle ctor
// (voxel_octree.cc:426); NULL normals -> geometric normal cross(p1-p0,p2-p0).
__global__ void k_pack_tris(const float* __restrict__ tri, const float* __restrict__ nrm_in, uint32_t T,
                            float4* __restrict__ tri4, float* __restrict__ nrm_out, int unit_normals)
{
        uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= T)
                return;
        const float* p = tri + 9ull * t;
        float v[9];
#pragma unroll
        for (int k = 0; k < 9; ++k)
                v[k] = p[k];
        tri4[3ull * t + 0] = make_float4(v[0], v[1], v[2], 0.f);
        tri4[3ull * t + 1] = make_float4(v[3], v[4], v[5], 0.f);
        tri4[3ull * t + 2] = make_float4(v[6], v[7], v[8], 0.f);
        float n[9];
        if (nrm_in) {
#pragma unroll
                for (int k = 0; k < 9; ++k)
                        n[k] = nrm_in[9ull * t + k];
        } else {
                // jql::cross(p1-p0, p2-p0) graphics_math.h:588-592
                float a[3] = { fsub(v[3], v[0]), fsub(v[4], v[1]), fsub(v[5], v[2]) };
                float b[3] = { fsub(v[6], v[0]), fsub(v[7], v[1]), fsub(v[8], v[2]) };
                float g[3];
                g[0] = fsub(fmul(a[1], b[2]), fmul(b[1], a[2]));
                g[1] = fsub(fmul(a[2], b[0]), fmul(b[2], a[0]));
                g[2] = fsub(fmul(a[0], b[1]), fmul(b[0], a[1]));
#pragma unroll
                for (int k = 0; k < 9; ++k)
                        n[k] = g[k % 3];
        }
        // (unit_normals: the caller hands over Triangle::n_ itself, already normalised by the Triangle ctor --
        // normalising again would move the last bit)
        if (!(unit_normals && nrm_in)) {
#pragma unroll
                for (int k = 0; k < 3; ++k)
                        normalize3(n[3 * k], n[3 * k + 1], n[3 * k + 2]);
        }
#pragma unroll
        for (int k = 0; k < 9; ++k)
                nrm_out[9ull * t + k] = n[k];
}

// ---------------------------------------------------------------------------
// host orchestration
// ---------------------------------------------------------------------------
static inline unsigned grid_for(uint64_t n, unsigned block)
{
        return (unsigned)std::max<uint64_t>(1, (n + block - 1) / block);
}

// Pair totals are carried in 32 bits (block counts, their scan, the frontier indices).  A level with n pairs can
// produce up to 8n: whenever 8n could reach 2^32 the block counts are ALSO summed in 64 bits before the scan, and
// the build stops with VRT_ERR_CAPACITY instead of sizing the next frontier from a wrapped total.
__global__ void __launch_bounds__(256)
k_sum_u32_u64(const uint32_t* __restrict__ v, uint64_t n, unsigned long long* __restrict__ out)
{
        unsigned long long acc = 0;
        for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
                acc += v[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
                acc += __shfl_down_sync(0xffffffffu, acc, o);
        if ((threadIdx.x & 31) == 0 && acc)
                atomicAdd(out, acc);
}

// sum of `n` device uint32 as a 64-bit host value (synchronises the stream)
int sum_u32_as_u64(vrt_tree* t, const uint32_t* d_v, uint64_t n, uint64_t* out)
{
        unsigned long long* d_sum = reinterpret_cast<unsigned long long*>(t->d_counter + 58);
        VRT_CUDA(cudaMemsetAsync(d_sum, 0, 8, t->stream));
        if (n) {
                k_sum_u32_u64<<<(unsigned)std::min<uint64_t>(1184, (n + 255) / 256), 256, 0, t->stream>>>(d_v, n, d_sum);
                count_launch();
        }
        unsigned long long h = 0;
        VRT_CUDA(cudaMemcpyAsync(&h, d_sum, 8, cudaMemcpyDeviceToHost, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        *out = h;
        return VRT_OK;
}

// true when the totals of a level fed by n pairs need the 64-bit check
static inline bool pair_total_may_wrap(uint64_t n) { return n >= (1ull << 29); }

// ---------------------------------------------------------------------------
// RANKED top-down build (the default for trees of depth >= 5).  The level-synchronous expansion
// above already visits every (triangle, non-empty cell) pair of every level, so the node arrays
// can be produced on the way down instead of being re-derived bottom-up from sorted leaf keys:
//   * a frontier pair carries the RANK of its cell among the non-empty cells of its level (the
//     cell's index in the BFS node array) instead of the cell's Morton code;
//   * the mask pass records "child c of node i exists" as one flag byte per (node, child) -- plain
//     stores of the constant 1, no atomics, the result cannot depend on any order;
//   * an exclusive scan of popc(mask) over the nodes of the level gives first_child, hence the
//     rank of every child = first_child + popc(mask & below(c)) -- children of one node are
//     contiguous and nodes stay in Morton order level by level (induction from the root);
//   * the leaf reference lists are a counting sort of the last frontier by leaf rank (atomic
//     cursors) followed by an ascending sort of every leaf's short list, which restores the
//     reference's insertion order (ascending triangle index) whatever order the atomics took.
// No radix sort, no head flags, no bottom-up pass; the output arrays are the same ones
// assemble_blob() consumes, bit for bit (tests: leaf sets, node records, checkpoint bytes).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_expand_mask_r(const float* __restrict__ tri, const float2* __restrict__ tab, uint64_t stride,
                const unsigned long long* __restrict__ in, uint32_t n_in, int level /* of the input cells */,
                const unsigned long long* __restrict__ node_morton,
                uint8_t* __restrict__ child_seen /* [nodes][8], zeroed */, int crowded, int iters,
                uint8_t* __restrict__ masks, uint32_t* __restrict__ block_counts)
{
        // a block handles 32 * iters pairs (iters = 8: kPairsPerBlock; small frontiers use iters = 1, i.e. 8x
        // the blocks and no serial loop -- those levels are bound by the latency of one pair's load chain)
        const uint32_t c = threadIdx.x & 7;
        const uint32_t lane = threadIdx.x & 31;
        const uint32_t child_base = 2u << level;  // table offset of level+1
        uint32_t cnt = 0;
#pragma unroll 1
        for (int it = 0; it < iters; ++it) {
                const uint32_t idx = (blockIdx.x * iters + it) * 32 + (threadIdx.x >> 3);
                bool ov = false;
                uint32_t node = 0;
                if (idx < n_in) {
                        const unsigned long long key = in[idx];
                        const uint32_t t = (uint32_t)key;
                        node = (uint32_t)(key >> 32);
                        const unsigned long long m = node_morton[node];
                        const uint32_t cx = 2u * compact1by2(m >> 2) + ((c >> 2) & 1u);
                        const uint32_t cy = 2u * compact1by2(m >> 1) + ((c >> 1) & 1u);
                        const uint32_t cz = 2u * compact1by2(m) + (c & 1u);
                        const float2 bx = tab[0 * stride + child_base + cx];
                        const float2 by = tab[1 * stride + child_base + cy];
                        const float2 bz = tab[2 * stride + child_base + cz];
                        const float* p = tri + 9ull * t;
                        float v0[3] = { p[0], p[1], p[2] }, v1[3] = { p[3], p[4], p[5] }, v2[3] = { p[6], p[7], p[8] };
                        float mn[3] = { bx.x, by.x, bz.x };
                        float mx[3] = { bx.y, by.y, bz.y };
                        ov = tri_overlaps_aabb(mn, mx, v0, v1, v2);
                }
                const uint32_t bal = __ballot_sync(0xffffffffu, ov);
                if (c == 0 && idx < n_in)
                        masks[idx] = (uint8_t)((bal >> (lane & 24u)) & 0xffu);
                // "child c of this node exists": a plain byte store -- every writer stores the same 1, so no
                // atomic is needed; the 8 lanes of a pair hit one 8-byte word
                // (`crowded` levels -- near the root thousands of pairs share a node -- read first: re-storing
                // a flag that is already set would only queue up behind the other writers of the same sector)
                if (ov) {
                        uint8_t* f = child_seen + 8ull * node + c;
                        if (!crowded || !__ldcg(f))
                                *f = 1;
                }
                cnt += ov ? 1u : 0u;
        }
        const uint32_t tot = block_sum_256(cnt);
        if (threadIdx.x == 0)
                block_counts[blockIdx.x] = tot;
}

// Round 2: the mask pass with ONE thread per (triangle, cell) pair.  The thread evaluates all eight
// children's tests at once (tri_overlaps_children8: the sub-expressions that are identical between children
// are computed once -- about a third of the arithmetic of eight separate calls, and no 8-lane groups that
// diverge at the early exits).  Same outputs as k_expand_mask_r; a block handles kPairsPerBlock pairs.
__global__ void __launch_bounds__(256)
k_expand_mask_r8(const float* __restrict__ tri, const float2* __restrict__ tab, uint64_t stride,
                 const unsigned long long* __restrict__ in, uint32_t n_in, int level /* of the input cells */,
                 const unsigned long long* __restrict__ node_morton, uint8_t* __restrict__ child_seen /* [nodes][8], zeroed */,
                 int crowded, uint8_t* __restrict__ masks, uint32_t* __restrict__ block_counts)
{
        const uint32_t idx = blockIdx.x * kPairsPerBlock + threadIdx.x;
        uint32_t m8 = 0;
        if (idx < n_in) {
                const unsigned long long key = in[idx];
                const uint32_t t = (uint32_t)key;
                const uint32_t node = (uint32_t)(key >> 32);
                const unsigned long long m = node_morton[node];
                // float4 view of the table: entry (1<<level)+x of an axis = (lo.min, lo.max, hi.min, hi.max) of
                // the two children of cell x at `level`
                const float4* tab4 = reinterpret_cast<const float4*>(tab);
                const uint64_t s4 = stride >> 1;
                const uint32_t base = 1u << level;
                const float4 bx = tab4[0 * s4 + base + compact1by2(m >> 2)];
                const float4 by = tab4[1 * s4 + base + compact1by2(m >> 1)];
                const float4 bz = tab4[2 * s4 + base + compact1by2(m)];
                const float* p = tri + 9ull * t;
                const float v0[3] = { p[0], p[1], p[2] }, v1[3] = { p[3], p[4], p[5] }, v2[3] = { p[6], p[7], p[8] };
                m8 = tri_overlaps_children8(bx, by, bz, v0, v1, v2);
                masks[idx] = (uint8_t)m8;
                // "child c of this node exists": plain byte stores of the constant 1 (see k_expand_mask_r)
                uint32_t mm = m8;
                while (mm) {
                        const uint32_t c = __ffs((int)mm) - 1;
                        mm &= mm - 1u;
                        uint8_t* f = child_seen + 8ull * node + c;
                        if (!crowded || !__ldcg(f))
                                *f = 1;
                }
        }
        const uint32_t tot = block_sum_256((uint32_t)__popc(m8));
        if (threadIdx.x == 0)
                block_counts[blockIdx.x] = tot;
}

// child mask (the 8 flag bytes packed into 8 bits) and children per node; *dead_ends counts the nodes
// none of whose children any triangle reached
__global__ void k_node_counts(const unsigned long long* __restrict__ child_seen, uint32_t n,
                              uint32_t* __restrict__ mask, uint32_t* __restrict__ cnt, uint32_t* __restrict__ dead_ends)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i < n) {
                // byte c (0 or 1) -> bit c: the eight products land on distinct bit positions, no carries
                const unsigned long long x = child_seen[i] & 0x0101010101010101ull;
                const uint32_t m = (uint32_t)((x * 0x0102040810204080ull) >> 56);
                mask[i] = m;
                cnt[i] = __popc(m);
                if (!m)
                        atomicAdd(dead_ends, 1u);
        }
}

// totals of one level in one place: out[0] = pairs produced, out[1] = nodes of the next level
// (out[2] = dead ends so far, accumulated by k_node_counts)
// `mailbox` (may be null) is page-locked HOST memory mapped into the device's address space: the three totals and
// then a ticket are stored there directly, so the host learns them by polling one word instead of a copy + a
// stream synchronisation per level (the stream never drains: the host enqueues the next level as soon as the
// ticket shows up).
__global__ void k_publish_totals(const uint32_t* __restrict__ pairs_total, const uint32_t* __restrict__ first_last,
                                 const uint32_t* __restrict__ cnt_last, uint32_t* __restrict__ out,
                                 volatile uint32_t* mailbox, uint32_t ticket)
{
        const uint32_t a = *pairs_total, b = *first_last + *cnt_last;
        out[0] = a;
        out[1] = b;
        if (mailbox) {
                mailbox[0] = a;
                mailbox[1] = b;
                mailbox[2] = out[2];
                __threadfence_system();
                mailbox[3] = ticket;
        }
}

// Host side of the mailbox: spin until the ticket arrives (with a periodic look at the stream, so that a failed
// launch cannot hang the host).  Returns false when the stream finished without delivering the ticket.
static bool wait_mailbox(cudaStream_t s, volatile uint32_t* mailbox, uint32_t ticket)
{
        for (uint64_t spin = 1;; ++spin) {
                if (mailbox[3] == ticket)
                        return true;
                if ((spin & 0xfffffull) == 0 && cudaStreamQuery(s) != cudaErrorNotReady)
                        return mailbox[3] == ticket;
        }
}

// ---- dead ends.  A triangle can pass a cell's SAT test and fail all eight children's; the reference
// then holds an interior node with eight empty leaves, which can never produce a hit, and the flat
// array does not store such nodes (nor ancestors left without any stored child) -- exactly what the
// bottom-up derivation of the sorted path yields.  The ranked path removes them afterwards: alive
// masks bottom-up (in place), an exclusive scan of the alive flags per level = the new ranks, one
// compaction per level.
__global__ void k_alive_mask(uint32_t* __restrict__ mask, const uint32_t* __restrict__ first, uint32_t n,
                             const uint32_t* __restrict__ mask_next)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        uint32_t m = mask[i], out = 0, pos = first[i];
        while (m) {
                const uint32_t c = __ffs((int)m) - 1;
                m &= m - 1u;
                if (mask_next[pos++])
                        out |= 1u << c;
        }
        mask[i] = out;
}

__global__ void k_alive_flags(const uint32_t* __restrict__ mask, uint32_t n, uint32_t* __restrict__ flag)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i <= n)
                flag[i] = (i < n && mask[i]) ? 1u : 0u;  // flag[n] = 0: the scan leaves the total there
}

struct LevelOffsets {
        uint32_t total_at[VRT_MAX_DEPTH + 1];  // index (into the new-rank buffer) of every level's total
};
__global__ void k_collect_totals(const uint32_t* __restrict__ idx_buf, LevelOffsets lo, int levels,
                                 uint32_t* __restrict__ out)
{
        const int l = threadIdx.x;
        if (l < levels)
                out[l] = idx_buf[lo.total_at[l]];
}

__global__ void k_compact_level(const unsigned long long* __restrict__ morton, const uint32_t* __restrict__ mask,
                                const uint32_t* __restrict__ first, const uint32_t* __restrict__ newidx,
                                const uint32_t* __restrict__ newidx_next /* null: children are leaves */, uint32_t n,
                                unsigned long long* __restrict__ out_morton, uint32_t* __restrict__ out_mask,
                                uint32_t* __restrict__ out_first)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        const uint32_t m = mask[i];
        if (!m)
                return;
        const uint32_t j = newidx[i];
        out_morton[j] = morton[i];
        out_mask[j] = m;
        // new rank of the first stored child: the exclusive scan counts the stored nodes before first[i]
        out_first[j] = newidx_next ? newidx_next[first[i]] : first[i];
}

// Morton codes of the next level's nodes: child c of node i sits at first[i] + popc(mask & below(c))
__global__ void k_children_morton(const unsigned long long* __restrict__ morton, const uint32_t* __restrict__ mask,
                                  const uint32_t* __restrict__ first, uint32_t n,
                                  unsigned long long* __restrict__ child_morton)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        uint32_t m = mask[i];
        uint32_t pos = first[i];
        const unsigned long long base = morton[i] << 3;
        while (m) {
                const uint32_t c = __ffs((int)m) - 1;
                m &= m - 1u;
                child_morton[pos++] = base | c;
        }
}

// Emit pass of the ranked expansion: out key = child rank << 32 | triangle.  At the last level
// (leaf_cnt != null) it also counts the references of every leaf.
__global__ void __launch_bounds__(256)
k_expand_emit_r(const unsigned long long* __restrict__ in, uint32_t n_in, const uint8_t* __restrict__ masks,
                const uint32_t* __restrict__ block_offs, const uint32_t* __restrict__ node_mask,
                const uint32_t* __restrict__ node_first, unsigned long long* __restrict__ out,
                uint32_t* __restrict__ leaf_cnt, uint32_t offs_per_block /* mask-pass blocks per 256 pairs */)
{
        const uint32_t idx = blockIdx.x * kPairsPerBlock + threadIdx.x;
        uint32_t m = 0;
        unsigned long long key = 0;
        if (idx < n_in) {
                m = masks[idx];
                key = in[idx];
        }
        uint32_t pos = block_offs[blockIdx.x * offs_per_block] + block_excl_scan_256(__popc(m));
        if (!m)
                return;
        const uint32_t node = (uint32_t)(key >> 32);
        const unsigned long long t = key & 0xffffffffull;
        const uint32_t nm = node_mask[node];
        const uint32_t first = node_first[node];
        while (m) {
                const uint32_t c = __ffs((int)m) - 1;
                m &= m - 1u;
                const uint32_t rank = first + __popc(nm & ((1u << c) - 1u));
                out[pos++] = ((unsigned long long)rank << 32) | t;
                if (leaf_cnt)
                        atomicAdd(&leaf_cnt[rank], 1u);
        }
}

// Counting sort of the last frontier by leaf rank: cursor[leaf] counts DOWN from the leaf's size.
__global__ void k_leaf_scatter(const unsigned long long* __restrict__ keys, uint64_t n,
                               const uint32_t* __restrict__ leaf_start, uint32_t* __restrict__ cursor,
                               uint32_t* __restrict__ refs)
{
        const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        const unsigned long long k = keys[i];
        const uint32_t leaf = (uint32_t)(k >> 32);
        const uint32_t slot = atomicSub(&cursor[leaf], 1u) - 1u;
        refs[leaf_start[leaf] + slot] = (uint32_t)k;
}

constexpr uint32_t kLeafSortSmall = 24;    // up to here: insertion sort by the leaf's thread
constexpr uint32_t kLeafSortBig = 8192;    // up to here: bitonic sort by one block in shared memory

// Ascending triangle index inside every leaf (= the reference's insertion order).  Leaves with more
// than kLeafSortSmall references are queued for k_leaf_sort_big.  big[0] = queue length,
// big[1] = overflow flag (a leaf beyond kLeafSortBig: the caller rebuilds through the sorted path),
// big[2..] = queued leaf ranks.
__global__ void k_leaf_sort_small(const uint32_t* __restrict__ leaf_start, uint32_t num_leaves, uint32_t num_refs,
                                  uint32_t* __restrict__ refs, uint32_t* __restrict__ big, uint32_t big_cap)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= num_leaves)
                return;
        const uint32_t s = leaf_start[i];
        const uint32_t e = (i + 1 < num_leaves) ? leaf_start[i + 1] : num_refs;
        const uint32_t cnt = e - s;
        if (cnt < 2)
                return;
        if (cnt > kLeafSortSmall) {
                if (cnt > kLeafSortBig) {
                        big[1] = 1u;
                        return;
                }
                const uint32_t q = atomicAdd(&big[0], 1u);
                if (q < big_cap)
                        big[2 + q] = i;
                else
                        big[1] = 1u;
                return;
        }
        uint32_t* r = refs + s;
        for (uint32_t a = 1; a < cnt; ++a) {
                const uint32_t v = r[a];
                uint32_t b = a;
                while (b > 0 && r[b - 1] > v) {
                        r[b] = r[b - 1];
                        --b;
                }
                r[b] = v;
        }
}

__global__ void __launch_bounds__(256)
k_leaf_sort_big(const uint32_t* __restrict__ leaf_start, uint32_t num_leaves, uint32_t num_refs,
                uint32_t* __restrict__ refs, const uint32_t* __restrict__ big, uint32_t big_cap)
{
        __shared__ uint32_t sh[kLeafSortBig];
        const uint32_t nq = min(big[0], big_cap);
        for (uint32_t q = blockIdx.x; q < nq; q += gridDim.x) {
                const uint32_t i = big[2 + q];
                const uint32_t s = leaf_start[i];
                const uint32_t e = (i + 1 < num_leaves) ? leaf_start[i + 1] : num_refs;
                const uint32_t cnt = e - s;
                uint32_t p2 = 1;
                while (p2 < cnt)
                        p2 <<= 1;
                for (uint32_t k = threadIdx.x; k < p2; k += blockDim.x)
                        sh[k] = (k < cnt) ? refs[s + k] : 0xffffffffu;
                __syncthreads();
                for (uint32_t size = 2; size <= p2; size <<= 1) {
                        for (uint32_t str = size >> 1; str > 0; str >>= 1) {
                                for (uint32_t k = threadIdx.x; k < p2; k += blockDim.x) {
                                        const uint32_t j = k ^ str;
                                        if (j > k) {
                                                const uint32_t a = sh[k], b = sh[j];
                                                const bool up = (k & size) == 0;
                                                if ((a > b) == up) {
                                                        sh[k] = b;
                                                        sh[j] = a;
                                                }
                                        }
                                }
                                __syncthreads();
                        }
                }
                for (uint32_t k = threadIdx.x; k < cnt; k += blockDim.x)
                        refs[s + k] = sh[k];
                __syncthreads();
        }
}

static int tri_bits_for(uint32_t T)
{
        int tb = 1;
        while ((1ull << tb) < (unsigned long long)T)
                ++tb;
        return tb;
}

static int assemble_blob(vrt_tree* t, int L, uint64_t n, const uint64_t* level_n, const float* d_root6);

// Everything after the keys are known: sort (by Morton bits, or by the full key
// when `sort_full`), leaves, bottom-up levels, blob assembly.
static int finish_from_keys(vrt_tree* t, unsigned long long* keys, uint64_t n, int L, int tb,
                            bool stable_input, const float* d_root6)
{
        cudaStream_t s = t->stream;
        const uint32_t T = t->hdr.num_tris;
        // --- sort -----------------------------------------------------------------
        unsigned long long* sorted = keys;
        if (n > 1) {
                if (t->keys_b.reserve(n * 8))
                        return VRT_ERR_NOMEM;
                uint64_t he = sort_hist_elems(n);
                if (t->hist.reserve(he * 4) || t->tmp_c.reserve(scan_scratch_elems(he) * 4))
                        return VRT_ERR_NOMEM;
                unsigned long long* other = (keys == t->keys_a.as<unsigned long long>())
                                                    ? t->keys_b.as<unsigned long long>()
                                                    : t->keys_a.as<unsigned long long>();
                if (other == nullptr || other == keys) {
                        other = t->keys_b.as<unsigned long long>();
                }
                int lo = stable_input ? tb : 0;
                int hi = tb + 3 * L;
                if (hi > lo)
                        radix_sort_u64(keys, other, n, lo, hi, t->hist.as<uint32_t>(),
                                       t->tmp_c.as<uint32_t>(), s, &sorted);
        }
        // --- leaves ---------------------------------------------------------------
        uint64_t num_leaves = 0;
        if (t->tmp_a.reserve((n + 1) * 4) || t->tmp_b.reserve((n + 1) * 4) ||
            t->tmp_c.reserve(std::max<uint64_t>(scan_scratch_elems(n), 16) * 4))
                return VRT_ERR_NOMEM;
        uint32_t* flag = t->tmp_a.as<uint32_t>();
        uint32_t* pos = t->tmp_b.as<uint32_t>();
        Scratch& refs_s = t->refs_s;  // refs until the blob exists (kept across rebuilds)
        if (n) {
                k_head_flags<<<grid_for(n, 256), 256, 0, s>>>(sorted, n, tb, flag);
                count_launch();
                exclusive_scan_u32(flag, pos, n, t->tmp_c.as<uint32_t>(), s);
                VRT_CUDA(cudaMemcpyAsync(&t->h_counter[0], pos + (n - 1), 4, cudaMemcpyDeviceToHost, s));
                VRT_CUDA(cudaMemcpyAsync(&t->h_counter[1], flag + (n - 1), 4, cudaMemcpyDeviceToHost, s));
                VRT_CUDA(cudaStreamSynchronize(s));
                num_leaves = (uint64_t)t->h_counter[0] + t->h_counter[1];
        }
        if (num_leaves >= 0xfffffff0ull || n >= 0xfffffff0ull) {
                set_error("octree too large for 32-bit node indices (%llu leaves, %llu refs)",
                          (unsigned long long)num_leaves, (unsigned long long)n);
                return VRT_ERR_CAPACITY;
        }
        // level arrays: morton (u64), first (u32), mask (u32).  Level L: first = ref start.
        uint64_t level_n[VRT_MAX_DEPTH + 1] = { 0 };
        level_n[L] = num_leaves;
        if (t->level_morton[L].reserve(std::max<uint64_t>(num_leaves, 1) * 8) ||
            t->level_first[L].reserve(std::max<uint64_t>(num_leaves, 1) * 4))
                return VRT_ERR_NOMEM;
        if (refs_s.reserve(std::max<uint64_t>(n, 1) * 4))
                return VRT_ERR_NOMEM;
        if (n) {
                k_emit_leaves<<<grid_for(n, 256), 256, 0, s>>>(sorted, n, tb, flag, pos,
                                                               t->level_morton[L].as<unsigned long long>(),
                                                               t->level_first[L].as<uint32_t>(),
                                                               refs_s.as<uint32_t>());
                count_launch();
        }
        // --- bottom-up ------------------------------------------------------------
        for (int l = L - 1; l >= 0; --l) {
                const uint64_t nc = level_n[l + 1];
                if (nc == 0) {
                        level_n[l] = 0;
                        continue;
                }
                const unsigned long long* child = t->level_morton[l + 1].as<unsigned long long>();
                k_parent_flags<<<grid_for(nc, 256), 256, 0, s>>>(child, nc, flag);
                count_launch();
                exclusive_scan_u32(flag, pos, nc, t->tmp_c.as<uint32_t>(), s);
                VRT_CUDA(cudaMemcpyAsync(&t->h_counter[0], pos + (nc - 1), 4, cudaMemcpyDeviceToHost, s));
                VRT_CUDA(cudaMemcpyAsync(&t->h_counter[1], flag + (nc - 1), 4, cudaMemcpyDeviceToHost, s));
                VRT_CUDA(cudaStreamSynchronize(s));
                const uint64_t np = (uint64_t)t->h_counter[0] + t->h_counter[1];
                level_n[l] = np;
                if (t->level_morton[l].reserve(np * 8) || t->level_first[l].reserve(np * 4) ||
                    t->level_mask[l].reserve(np * 4))
                        return VRT_ERR_NOMEM;
                k_emit_parents<<<grid_for(nc, 256), 256, 0, s>>>(child, nc, flag, pos,
                                                                 t->level_morton[l].as<unsigned long long>(),
                                                                 t->level_first[l].as<uint32_t>(),
                                                                 t->level_mask[l].as<uint32_t>());
                count_launch();
        }
        return assemble_blob(t, L, n, level_n, d_root6);
}

// Blob assembly from the per-level arrays (level_morton / level_first / level_mask, leaf level L:
// level_first = first ref) and the reference list in refs_s.
static int assemble_blob(vrt_tree* t, int L, uint64_t n, const uint64_t* level_n, const float* d_root6)
{
        cudaStream_t s = t->stream;
        const uint32_t T = t->hdr.num_tris;
        const uint64_t num_leaves = level_n[L];
        Scratch& refs_s = t->refs_s;
        BlobHeader& h = t->hdr;
        h.magic = kBlobMagic;
        h.max_depth = L + 1;
        h.num_leaves = num_leaves;
        h.num_refs = n;
        uint64_t off = 0;
        for (int l = 0; l <= L; ++l) {
                h.level_offset[l] = off;
                off += level_n[l];
        }
        for (int l = L + 1; l <= (int)VRT_MAX_DEPTH; ++l)
                h.level_offset[l] = off;
        h.num_nodes = off;
        if (h.num_nodes >= 0xfffffff0ull) {
                set_error("octree too large for 32-bit node indices");
                return VRT_ERR_CAPACITY;
        }
        h.axis_tab_stride = 2ull << L;
        uint64_t b = kHeaderBytes;
        h.off_nodes = b;
        b = align256(b + std::max<uint64_t>(h.num_nodes, 1) * 8);
        h.off_leaf_morton = b;
        b = align256(b + std::max<uint64_t>(num_leaves, 1) * 8);
        h.off_leaf_refs = b;
        b = align256(b + std::max<uint64_t>(n, 1) * 4);
        h.off_tri4 = b;
        b = align256(b + std::max<uint64_t>(T, 1) * 48);
        h.off_nrm = b;
        b = align256(b + std::max<uint64_t>(T, 1) * 36);
        h.off_axis_tab = b;
        b = align256(b + 3 * h.axis_tab_stride * 8);
        h.bytes = b;
        if (t->blob && t->own_blob && t->blob_bytes < b) {
                cudaFree(t->blob);
                t->blob = nullptr;
        }
        if (!t->blob) {
                if (cudaMalloc(&t->blob, b) != cudaSuccess) {
                        cudaGetLastError();
                        set_error("cudaMalloc(%llu) for the octree blob failed", (unsigned long long)b);
                        return VRT_ERR_NOMEM;
                }
                t->blob_bytes = b;
                t->own_blob = true;
        }
        char* base = static_cast<char*>(t->blob);
        // zero the header's tail and the alignment gaps between the sections: every byte up to h.bytes is then a
        // function of the inputs alone, so a rebuild into a reused blob (vrt_rebuild, vrt_update_*) equals a fresh
        // build byte for byte
        const uint64_t gaps[][2] = { { sizeof h, h.off_nodes },
                                     { h.off_nodes + h.num_nodes * 8, h.off_leaf_morton },
                                     { h.off_leaf_morton + num_leaves * 8, h.off_leaf_refs },
                                     { h.off_leaf_refs + n * 4, h.off_tri4 },
                                     { h.off_tri4 + (uint64_t)T * 48, h.off_nrm },
                                     { h.off_nrm + (uint64_t)T * 36, h.off_axis_tab },
                                     { h.off_axis_tab + 3 * h.axis_tab_stride * 8, h.bytes } };
        for (const auto& g : gaps)
                if (g[1] > g[0])
                        VRT_CUDA(cudaMemsetAsync(base + g[0], 0, g[1] - g[0], s));
        VRT_CUDA(cudaMemcpyAsync(h.root_aabb, d_root6, 24, cudaMemcpyDeviceToHost, s));
        uint2* nodes = reinterpret_cast<uint2*>(base + h.off_nodes);
        for (int l = 0; l < L; ++l) {
                if (!level_n[l])
                        continue;
                k_write_interior<<<grid_for(level_n[l], 256), 256, 0, s>>>(
                        t->level_first[l].as<uint32_t>(), t->level_mask[l].as<uint32_t>(),
                        (uint32_t)level_n[l], (uint32_t)h.level_offset[l + 1], nodes + h.level_offset[l]);
                count_launch();
        }
        if (num_leaves) {
                k_write_leaves<<<grid_for(num_leaves, 256), 256, 0, s>>>(
                        t->level_first[L].as<uint32_t>(), (uint32_t)num_leaves, (uint32_t)n,
                        nodes + h.level_offset[L]);
                count_launch();
                VRT_CUDA(cudaMemcpyAsync(base + h.off_leaf_morton, t->level_morton[L].p, num_leaves * 8,
                                         cudaMemcpyDeviceToDevice, s));
                VRT_CUDA(cudaMemcpyAsync(base + h.off_leaf_refs, refs_s.p, n * 4, cudaMemcpyDeviceToDevice, s));
        }
        if (T) {
                k_pack_tris<<<grid_for(T, 256), 256, 0, s>>>(t->d_tri_in, t->d_nrm_in, T,
                                                             reinterpret_cast<float4*>(base + h.off_tri4),
                                                             reinterpret_cast<float*>(base + h.off_nrm), t->unit_normals ? 1 : 0);
                count_launch();
        }
        k_axis_table<<<1, 1024, 0, s>>>(d_root6, reinterpret_cast<float2*>(base + h.off_axis_tab),
                                        h.axis_tab_stride, L);
        count_launch();
        VRT_CUDA(cudaStreamSynchronize(s));
        VRT_CUDA(cudaMemcpyAsync(base, &h, sizeof h, cudaMemcpyHostToDevice, s));
        VRT_CUDA(cudaStreamSynchronize(s));
        tree_bind_views(t);
        scratch_flush_deferred();  // buffers that had to grow during this build
        return compute_hulls(t);
}

int sort_keys_u64(vrt_tree* t, uint64_t n, int lo, int hi, unsigned long long** sorted)
{
        *sorted = t->keys_a.as<unsigned long long>();
        if (n < 2 || hi <= lo)
                return VRT_OK;
        const uint64_t he = sort_hist_elems(n);
        if (t->keys_b.reserve(n * 8) || t->hist.reserve(he * 4) || t->tmp_c.reserve(scan_scratch_elems(he) * 4))
                return VRT_ERR_NOMEM;
        radix_sort_u64(t->keys_a.as<unsigned long long>(), t->keys_b.as<unsigned long long>(), n, lo, hi,
                       t->hist.as<uint32_t>(), t->tmp_c.as<uint32_t>(), t->stream, sorted);
        return VRT_OK;
}

constexpr int VRT_RANKED_FALLBACK = 1000;  // internal: "use the sorted path" (never leaves this file)

// Removes the dead ends of the ranked build (see k_alive_mask); level_n[0..L-1] are updated.
static int prune_dead_ends(vrt_tree* t, int L, uint64_t* level_n)
{
        cudaStream_t s = t->stream;
        // alive masks, bottom-up, in place (the children of level L-1 are leaves: all stored)
        for (int l = L - 2; l >= 0; --l) {
                k_alive_mask<<<grid_for(level_n[l], 256), 256, 0, s>>>(t->level_mask[l].as<uint32_t>(),
                                                                      t->level_first[l].as<uint32_t>(), (uint32_t)level_n[l],
                                                                      t->level_mask[l + 1].as<uint32_t>());
                count_launch();
        }
        // new ranks per level: idx_buf[off[l] + i], the level's stored-node total at idx_buf[off[l] + n_l]
        uint64_t off[VRT_MAX_DEPTH + 1] = { 0 }, tot = 0, nmax = 0;
        for (int l = 0; l < L; ++l) {
                off[l] = tot;
                tot += level_n[l] + 1;
                nmax = std::max(nmax, level_n[l]);
        }
        if (tot >= 0xfffffff0ull) {
                set_error("octree too large for 32-bit node indices");
                return VRT_ERR_CAPACITY;
        }
        if (t->keys_a.reserve(tot * 4) || t->tmp_b.reserve((nmax + 1) * 4) ||
            t->tmp_c.reserve(std::max<uint64_t>(scan_scratch_elems(nmax + 1), 16) * 4))
                return VRT_ERR_NOMEM;
        uint32_t* idx_buf = t->keys_a.as<uint32_t>();  // (the frontier buffers are free by now)
        uint32_t* flag = t->tmp_b.as<uint32_t>();
        LevelOffsets lo{};
        for (int l = 0; l < L; ++l) {
                const uint64_t nn = level_n[l];
                k_alive_flags<<<grid_for(nn + 1, 256), 256, 0, s>>>(t->level_mask[l].as<uint32_t>(), (uint32_t)nn, flag);
                count_launch();
                exclusive_scan_u32(flag, idx_buf + off[l], nn + 1, t->tmp_c.as<uint32_t>(), s);
                lo.total_at[l] = (uint32_t)(off[l] + nn);
        }
        uint32_t* d_new = t->d_counter + 40;  // L <= 17 values
        k_collect_totals<<<1, 32, 0, s>>>(idx_buf, lo, L, d_new);
        count_launch();
        VRT_CUDA(cudaMemcpyAsync(t->h_counter + 8, d_new, (size_t)L * 4, cudaMemcpyDeviceToHost, s));
        VRT_CUDA(cudaStreamSynchronize(s));
        uint64_t new_n[VRT_MAX_DEPTH + 1];
        for (int l = 0; l < L; ++l)
                new_n[l] = t->h_counter[8 + l];
        // compaction, level by level, through temporaries (an element moves to a lower or equal index,
        // but in parallel that is only safe out of place)
        if (t->keys_b.reserve(nmax * 8) || t->tmp_a.reserve(nmax * 4) || t->tmp_b.reserve((nmax + 1) * 4))
                return VRT_ERR_NOMEM;
        for (int l = 0; l < L; ++l) {
                const uint64_t nn = level_n[l];
                const bool next_changed = (l + 1 < L) && new_n[l + 1] != level_n[l + 1];
                if (new_n[l] == nn && !next_changed)
                        continue;
                k_compact_level<<<grid_for(nn, 256), 256, 0, s>>>(
                        t->level_morton[l].as<unsigned long long>(), t->level_mask[l].as<uint32_t>(),
                        t->level_first[l].as<uint32_t>(), idx_buf + off[l], (l + 1 < L) ? idx_buf + off[l + 1] : nullptr,
                        (uint32_t)nn, t->keys_b.as<unsigned long long>(), t->tmp_a.as<uint32_t>(), t->tmp_b.as<uint32_t>());
                count_launch();
                const uint64_t m = new_n[l];
                if (m) {
                        VRT_CUDA(cudaMemcpyAsync(t->level_morton[l].p, t->keys_b.p, m * 8, cudaMemcpyDeviceToDevice, s));
                        VRT_CUDA(cudaMemcpyAsync(t->level_mask[l].p, t->tmp_a.p, m * 4, cudaMemcpyDeviceToDevice, s));
                        VRT_CUDA(cudaMemcpyAsync(t->level_first[l].p, t->tmp_b.p, m * 4, cudaMemcpyDeviceToDevice, s));
                }
        }
        for (int l = 0; l < L; ++l)
                level_n[l] = new_n[l];
        return VRT_OK;
}

// The ranked top-down build (see the kernels above).  keys_a holds the level-0 frontier
// (key = triangle index, node rank 0), n0 pairs.
static int build_ranked(vrt_tree* t, int L, uint64_t n0, const float* d_root6, const float2* tab, uint64_t stride)
{
        cudaStream_t s = t->stream;
        uint32_t* d_tot = t->d_counter + 32;  // [0] pairs produced, [1] nodes of the next level, [2] dead ends
        VRT_CUDA(cudaMemsetAsync(d_tot, 0, 12, s));
        uint32_t dead_ends = 0;
        uint64_t level_n[VRT_MAX_DEPTH + 1] = { 0 };
        level_n[0] = 1;
        if (t->level_morton[0].reserve(8) || t->level_mask[0].reserve(4) || t->level_first[0].reserve(4))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemsetAsync(t->level_morton[0].p, 0, 8, s));
        Scratch* cur = &t->keys_a;
        Scratch* nxt = &t->keys_b;
        uint64_t n = n0;
        for (int l = 0; l < L; ++l) {
                const uint64_t nn = level_n[l];
                // mask pass: one thread per pair (k_expand_mask_r8, default) or eight lanes per pair
                // (k_expand_mask_r, VRT_BUILD_SAT8=0: a block handles 32 * iters pairs)
                static int sat8 = -1;
                if (sat8 < 0) {
                        const char* e = getenv("VRT_BUILD_SAT8");
                        sat8 = (e && e[0] == '0') ? 0 : 1;
                }
                const int iters = sat8 ? kPairsPerBlock / 32 : ((n < (1ull << 20)) ? 1 : kPairsPerBlock / 32);
                const uint32_t ppb = 32u * (uint32_t)iters;  // pairs per block of the mask pass
                const uint32_t nblk = (uint32_t)((n + ppb - 1) / ppb);
                const uint32_t nblk_emit = (uint32_t)((n + kPairsPerBlock - 1) / kPairsPerBlock);
                if (t->tmp_b.reserve(n) || t->hist.reserve((nblk + 1ull) * 4) || t->tmp_a.reserve((nn + 1) * 4) ||
                    t->refs_s.reserve(nn * 8) ||
                    t->tmp_c.reserve(std::max(scan_scratch_elems(nblk + 1ull), scan_scratch_elems(nn)) * 4))
                        return VRT_ERR_NOMEM;
                uint32_t* bc = t->hist.as<uint32_t>();
                uint32_t* node_mask = t->level_mask[l].as<uint32_t>();
                uint32_t* node_first = t->level_first[l].as<uint32_t>();
                uint32_t* node_cnt = t->tmp_a.as<uint32_t>();
                VRT_CUDA(cudaMemsetAsync(bc + nblk, 0, 4, s));
                uint8_t* child_seen = t->refs_s.as<uint8_t>();  // (the reference list is written after the last level)
                VRT_CUDA(cudaMemsetAsync(child_seen, 0, nn * 8, s));
                const int crowded = (n > 16 * nn && n >= (1ull << 20)) ? 1 : 0;
                if (sat8)
                        k_expand_mask_r8<<<nblk, 256, 0, s>>>(t->d_tri_in, tab, stride, cur->as<unsigned long long>(), (uint32_t)n,
                                                              l, t->level_morton[l].as<unsigned long long>(), child_seen, crowded,
                                                              t->tmp_b.as<uint8_t>(), bc);
                else
                        k_expand_mask_r<<<nblk, 256, 0, s>>>(t->d_tri_in, tab, stride, cur->as<unsigned long long>(), (uint32_t)n,
                                                             l, t->level_morton[l].as<unsigned long long>(), child_seen, crowded,
                                                             iters, t->tmp_b.as<uint8_t>(), bc);
                count_launch();
                if (pair_total_may_wrap(n)) {
                        uint64_t tot64 = 0;
                        int rc64 = sum_u32_as_u64(t, bc, nblk, &tot64);
                        if (rc64)
                                return rc64;
                        if (tot64 >= 0xfffffff0ull) {
                                set_error("more than 2^32 (triangle, cell) pairs at level %d", l + 1);
                                return VRT_ERR_CAPACITY;
                        }
                }
                exclusive_scan_u32(bc, bc, nblk + 1ull, t->tmp_c.as<uint32_t>(), s);
                k_node_counts<<<grid_for(nn, 256), 256, 0, s>>>(t->refs_s.as<unsigned long long>(), (uint32_t)nn, node_mask,
                                                                node_cnt, d_tot + 2);
                count_launch();
                exclusive_scan_u32(node_cnt, node_first, nn, t->tmp_c.as<uint32_t>(), s);
                // totals to the host through the mapped mailbox (h_counter[16..19]; VRT_BUILD_MAILBOX=0: copy + sync)
                static int use_mailbox = -1;
                if (use_mailbox < 0) {
                        const char* e = getenv("VRT_BUILD_MAILBOX");
                        use_mailbox = (e && e[0] == '0') ? 0 : 1;
                }
                volatile uint32_t* mailbox = use_mailbox ? t->h_counter + 16 : nullptr;
                const uint32_t ticket = ++t->mailbox_ticket;
                k_publish_totals<<<1, 1, 0, s>>>(bc + nblk, node_first + (nn - 1), node_cnt + (nn - 1), d_tot, mailbox, ticket);
                count_launch();
                uint64_t produced, nodes_next;
                if (mailbox && wait_mailbox(s, mailbox, ticket)) {
                        produced = mailbox[0];
                        nodes_next = mailbox[1];
                        dead_ends = mailbox[2];
                } else {
                        VRT_CUDA(cudaMemcpyAsync(t->h_counter, d_tot, 12, cudaMemcpyDeviceToHost, s));
                        VRT_CUDA(cudaStreamSynchronize(s));
                        produced = t->h_counter[0];
                        nodes_next = t->h_counter[1];
                        dead_ends = t->h_counter[2];
                }
                if (produced >= 0xfffffff0ull) {
                        set_error("more than 2^32 (triangle, cell) pairs at level %d", l + 1);
                        return VRT_ERR_CAPACITY;
                }
                level_n[l + 1] = nodes_next;
                const bool last = (l + 1 == L);
                if (nxt->reserve(std::max<uint64_t>(produced, 1) * 8) ||
                    t->level_morton[l + 1].reserve(std::max<uint64_t>(nodes_next, 1) * 8) ||
                    t->level_first[l + 1].reserve((nodes_next + 1) * 4) ||
                    (!last && t->level_mask[l + 1].reserve(std::max<uint64_t>(nodes_next, 1) * 4)))
                        return VRT_ERR_NOMEM;
                uint32_t* leaf_cnt = nullptr;
                if (last) {  // per-leaf reference counters (later: the scatter cursors)
                        if (t->tmp_a.reserve((nodes_next + 1) * 4))
                                return VRT_ERR_NOMEM;
                        leaf_cnt = t->tmp_a.as<uint32_t>();
                        VRT_CUDA(cudaMemsetAsync(leaf_cnt, 0, (nodes_next + 1) * 4, s));
                }
                if (nodes_next) {
                        k_children_morton<<<grid_for(nn, 256), 256, 0, s>>>(
                                t->level_morton[l].as<unsigned long long>(), node_mask, node_first, (uint32_t)nn,
                                t->level_morton[l + 1].as<unsigned long long>());
                        count_launch();
                }
                if (produced) {
                        k_expand_emit_r<<<nblk_emit, 256, 0, s>>>(cur->as<unsigned long long>(), (uint32_t)n,
                                                                  t->tmp_b.as<uint8_t>(), bc, node_mask, node_first,
                                                                  nxt->as<unsigned long long>(), leaf_cnt,
                                                                  (uint32_t)(kPairsPerBlock / ppb));
                        count_launch();
                }
                n = produced;
                std::swap(cur, nxt);
                if (!n) {  // nothing below this level (cannot happen for l < L with n > 0 pairs overlapping, kept for safety)
                        for (int k = l + 2; k <= L; ++k)
                                level_n[k] = 0;
                        break;
                }
        }
        const uint64_t num_leaves = level_n[L];
        if (num_leaves >= 0xfffffff0ull || n >= 0xfffffff0ull) {
                set_error("octree too large for 32-bit node indices (%llu leaves, %llu refs)",
                          (unsigned long long)num_leaves, (unsigned long long)n);
                return VRT_ERR_CAPACITY;
        }
        if (!n || !num_leaves)
                return VRT_RANKED_FALLBACK;
        // ---- leaf reference lists: counting sort by leaf rank, then ascending inside every leaf ----
        const uint32_t big_cap = 1u << 16;
        if (t->refs_s.reserve(n * 4) || t->tmp_c.reserve(std::max<uint64_t>(scan_scratch_elems(num_leaves), 16) * 4) ||
            t->hist.reserve((2ull + big_cap) * 4))
                return VRT_ERR_NOMEM;
        uint32_t* leaf_cnt = t->tmp_a.as<uint32_t>();
        uint32_t* leaf_start = t->level_first[L].as<uint32_t>();
        uint32_t* big = t->hist.as<uint32_t>();
        exclusive_scan_u32(leaf_cnt, leaf_start, num_leaves, t->tmp_c.as<uint32_t>(), s);
        VRT_CUDA(cudaMemsetAsync(big, 0, 8, s));
        k_leaf_scatter<<<grid_for(n, 256), 256, 0, s>>>(cur->as<unsigned long long>(), n, leaf_start, leaf_cnt,
                                                         t->refs_s.as<uint32_t>());
        k_leaf_sort_small<<<grid_for(num_leaves, 256), 256, 0, s>>>(leaf_start, (uint32_t)num_leaves, (uint32_t)n,
                                                                    t->refs_s.as<uint32_t>(), big, big_cap);
        k_leaf_sort_big<<<592, 256, 0, s>>>(leaf_start, (uint32_t)num_leaves, (uint32_t)n, t->refs_s.as<uint32_t>(), big,
                                            big_cap);
        count_launch(3);
        VRT_CUDA(cudaMemcpyAsync(t->h_counter, big, 8, cudaMemcpyDeviceToHost, s));
        VRT_CUDA(cudaStreamSynchronize(s));
        if (t->h_counter[1])
                return VRT_RANKED_FALLBACK;
        if (dead_ends) {
                int rc = prune_dead_ends(t, L, level_n);
                if (rc)
                        return rc;
        }
        return assemble_blob(t, L, n, level_n, d_root6);
}

// CUDA loads kernels lazily, one by one, at their first launch (a few ms each for the large ones).
// Which build kernels a scene needs depends on its depth and on the data (sorted or ranked path, dead
// ends, oversize leaves), so the first build on a device loads them all up front: the cost is paid once
// per process, at a predictable place, instead of in the middle of some later build.
static void preload_build_kernels()
{
        static bool done = false;
        if (done)
                return;
        done = true;
        const void* kernels[] = {
                (const void*)k_aabb_final,      (const void*)k_aabb_partial,    (const void*)k_alive_flags,
                (const void*)k_alive_mask,      (const void*)k_axis_table,      (const void*)k_children_morton,
                (const void*)k_collect_totals,  (const void*)k_compact_level,   (const void*)k_emit_leaves,
                (const void*)k_emit_parents,    (const void*)k_expand_emit,     (const void*)k_expand_emit_r,
                (const void*)k_expand_mask,     (const void*)k_expand_mask_r,   (const void*)k_head_flags,
                (const void*)k_expand_mask_r8,
                (const void*)k_leaf_scatter,    (const void*)k_leaf_sort_big,   (const void*)k_leaf_sort_small,
                (const void*)k_node_counts,     (const void*)k_pack_tris,       (const void*)k_parent_flags,
                (const void*)k_publish_totals,  (const void*)k_root_emit,       (const void*)k_root_mask,
                (const void*)k_scan_add,        (const void*)k_scan_tile,       (const void*)k_sort_hist,
                (const void*)k_sort_scatter,    (const void*)k_write_interior,  (const void*)k_write_leaves,
        };
        cudaFuncAttributes a;
        for (const void* k : kernels)
                if (cudaFuncGetAttributes(&a, k) != cudaSuccess)
                        cudaGetLastError();
}

int build_tree(vrt_tree* t, int max_depth)
{
        preload_build_kernels();
        cudaStream_t s = t->stream;
        const uint32_t T = t->hdr.num_tris;
        const int L = max_depth - 1;
        const int tb = tri_bits_for(T);
        if (3 * L + tb > 64) {
                set_error("key does not fit 64 bit: 3*(max_depth-1)=%d Morton bits + %d triangle bits", 3 * L, tb);
                return VRT_ERR_CAPACITY;
        }
        VRT_CUDA(cudaEventRecord(t->ev0, s));
        // root AABB + axis table (scratch copy; the blob gets its own at assembly)
        const int nb = 296;
        if (t->tmp_a.reserve(std::max<uint64_t>((uint64_t)nb * 6 * 8 + 64, 4096)))
                return VRT_ERR_NOMEM;
        float* d_root6 = reinterpret_cast<float*>(t->d_counter + 8);
        k_aabb_partial<<<nb, 256, 0, s>>>(t->d_tri_in, 3u * T, t->tmp_a.as<uint2>());
        k_aabb_final<<<1, 192, 0, s>>>(t->tmp_a.as<uint2>(), nb, d_root6);
        count_launch(2);
        const uint64_t stride = 2ull << L;
        Scratch& tab_s = t->tab_s;
        if (tab_s.reserve(3 * stride * 8))
                return VRT_ERR_NOMEM;
        k_axis_table<<<1, 1024, 0, s>>>(d_root6, tab_s.as<float2>(), stride, L);
        count_launch();
        // level 0
        if (t->keys_a.reserve(std::max<uint64_t>(T, 1) * 8))
                return VRT_ERR_NOMEM;
        uint64_t n = 0;
        if (T) {
                const uint32_t nblk = (T + kPairsPerBlock - 1) / kPairsPerBlock;
                if (t->tmp_b.reserve(T) || t->hist.reserve((nblk + 1ull) * 4) ||
                    t->tmp_c.reserve(scan_scratch_elems(nblk + 1ull) * 4))
                        return VRT_ERR_NOMEM;
                uint32_t* bc = t->hist.as<uint32_t>();
                VRT_CUDA(cudaMemsetAsync(bc + nblk, 0, 4, s));
                k_root_mask<<<nblk, 256, 0, s>>>(t->d_tri_in, T, d_root6, t->tmp_b.as<uint8_t>(), bc);
                count_launch();
                exclusive_scan_u32(bc, bc, nblk + 1ull, t->tmp_c.as<uint32_t>(), s);
                k_root_emit<<<nblk, 256, 0, s>>>(T, t->tmp_b.as<uint8_t>(), bc, t->keys_a.as<unsigned long long>());
                count_launch();
                VRT_CUDA(cudaMemcpyAsync(t->h_counter, bc + nblk, 4, cudaMemcpyDeviceToHost, s));
                VRT_CUDA(cudaStreamSynchronize(s));
                n = t->h_counter[0];
        }
        // the ranked top-down build for everything but shallow trees (whose few leaves hold long
        // reference lists: those keep the sorted path); VRT_BUILD_SORTED=1 forces the sorted path
        const char* env_sorted = getenv("VRT_BUILD_SORTED");
        const bool force_sorted = env_sorted && env_sorted[0] == '1';
        if (L >= 4 && n && !force_sorted) {
                int rc = build_ranked(t, L, n, d_root6, tab_s.as<float2>(), stride);
                if (rc != VRT_RANKED_FALLBACK) {
                        if (rc)
                                return rc;
                        VRT_CUDA(cudaEventRecord(t->ev1, s));
                        VRT_CUDA(cudaEventSynchronize(t->ev1));
                        float ms = 0;
                        VRT_CUDA(cudaEventElapsedTime(&ms, t->ev0, t->ev1));
                        t->build_ms = ms;
                        return VRT_OK;
                }
                // a leaf with more than kLeafSortBig references (or no leaf at all): redo the expansion with
                // Morton keys.  The ranked build has overwritten the level-0 frontier: rebuild it first.
                const uint32_t nblk = (T + kPairsPerBlock - 1) / kPairsPerBlock;
                if (t->keys_a.reserve(std::max<uint64_t>(T, 1) * 8) || t->tmp_b.reserve(T) ||
                    t->hist.reserve((nblk + 1ull) * 4) || t->tmp_c.reserve(scan_scratch_elems(nblk + 1ull) * 4))
                        return VRT_ERR_NOMEM;
                uint32_t* bc = t->hist.as<uint32_t>();
                VRT_CUDA(cudaMemsetAsync(bc + nblk, 0, 4, s));
                k_root_mask<<<nblk, 256, 0, s>>>(t->d_tri_in, T, d_root6, t->tmp_b.as<uint8_t>(), bc);
                exclusive_scan_u32(bc, bc, nblk + 1ull, t->tmp_c.as<uint32_t>(), s);
                k_root_emit<<<nblk, 256, 0, s>>>(T, t->tmp_b.as<uint8_t>(), bc, t->keys_a.as<unsigned long long>());
                count_launch(2);
        }
        Scratch* cur = &t->keys_a;
        Scratch* nxt = &t->keys_b;
        for (int l = 0; l < L && n; ++l) {
                const uint32_t nblk = (uint32_t)((n + kPairsPerBlock - 1) / kPairsPerBlock);
                if (t->tmp_b.reserve(n) || t->hist.reserve((nblk + 1ull) * 4) ||
                    t->tmp_c.reserve(scan_scratch_elems(nblk + 1ull) * 4))
                        return VRT_ERR_NOMEM;
                uint32_t* bc = t->hist.as<uint32_t>();
                VRT_CUDA(cudaMemsetAsync(bc + nblk, 0, 4, s));
                k_expand_mask<<<nblk, 256, 0, s>>>(t->d_tri_in, tab_s.as<float2>(), stride,
                                                   cur->as<unsigned long long>(), (uint32_t)n, l, tb,
                                                   t->tmp_b.as<uint8_t>(), bc);
                count_launch();
                if (pair_total_may_wrap(n)) {
                        uint64_t tot64 = 0;
                        int rc64 = sum_u32_as_u64(t, bc, nblk, &tot64);
                        if (rc64)
                                return rc64;
                        if (tot64 >= 0xfffffff0ull) {
                                set_error("more than 2^32 (triangle, cell) pairs at level %d", l + 1);
                                return VRT_ERR_CAPACITY;
                        }
                }
                exclusive_scan_u32(bc, bc, nblk + 1ull, t->tmp_c.as<uint32_t>(), s);
                VRT_CUDA(cudaMemcpyAsync(t->h_counter, bc + nblk, 4, cudaMemcpyDeviceToHost, s));
                VRT_CUDA(cudaStreamSynchronize(s));
                const uint64_t produced = t->h_counter[0];
                if (produced >= 0xfffffff0ull) {
                        set_error("more than 2^32 (triangle, cell) pairs at level %d", l + 1);
                        return VRT_ERR_CAPACITY;
                }
                if (nxt->reserve(std::max<uint64_t>(produced, 1) * 8))
                        return VRT_ERR_NOMEM;
                if (produced) {
                        k_expand_emit<<<nblk, 256, 0, s>>>(cur->as<unsigned long long>(), (uint32_t)n, tb,
                                                           t->tmp_b.as<uint8_t>(), bc, nxt->as<unsigned long long>());
                        count_launch();
                }
                n = produced;
                std::swap(cur, nxt);
        }
        // keys live in *cur; make sure finish_from_keys ping-pongs with the other one
        if (cur != &t->keys_a)
                std::swap(t->keys_a, t->keys_b);
        int rc = finish_from_keys(t, t->keys_a.as<unsigned long long>(), n, L, tb, /*stable_input=*/true, d_root6);
        if (rc)
                return rc;
        VRT_CUDA(cudaEventRecord(t->ev1, s));
        VRT_CUDA(cudaEventSynchronize(t->ev1));
        float ms = 0;
        VRT_CUDA(cudaEventElapsedTime(&ms, t->ev0, t->ev1));
        t->build_ms = ms;
        return VRT_OK;
}

int import_leaves(vrt_tree* t, int max_depth, const float root_aabb[6], uint64_t num_leaves,
                  const uint32_t* leaf_cell, const uint32_t* leaf_count, const uint32_t* leaf_refs)
{
        const int L = max_depth - 1;
        const uint32_t T = t->hdr.num_tris;
        const int tb = tri_bits_for(T);
        if (3 * L + tb > 64) {
                set_error("key does not fit 64 bit");
                return VRT_ERR_CAPACITY;
        }
        uint64_t n = 0;
        for (uint64_t i = 0; i < num_leaves; ++i)
                n += leaf_count[i];
        // every cell inside the leaf grid, no cell twice (a coordinate >= 2^L would spill into the Morton bits of
        // another cell, a repeated cell would silently merge two reference lists)
        {
                std::vector<unsigned long long> codes(num_leaves);
                for (uint64_t i = 0; i < num_leaves; ++i) {
                        for (int a = 0; a < 3; ++a)
                                if ((uint64_t)leaf_cell[3 * i + a] >> L) {
                                        set_error("leaf_cell[%llu] lies outside the %d-level leaf grid", (unsigned long long)i, L);
                                        return VRT_ERR_ARG;
                                }
                        codes[i] = morton_encode(leaf_cell[3 * i], leaf_cell[3 * i + 1], leaf_cell[3 * i + 2]);
                }
                std::sort(codes.begin(), codes.end());
                if (std::adjacent_find(codes.begin(), codes.end()) != codes.end()) {
                        set_error("leaf_cell lists the same cell twice");
                        return VRT_ERR_ARG;
                }
        }
        std::vector<unsigned long long> keys(n);
        uint64_t k = 0;
        for (uint64_t i = 0; i < num_leaves; ++i) {
                unsigned long long m = morton_encode(leaf_cell[3 * i], leaf_cell[3 * i + 1], leaf_cell[3 * i + 2]);
                for (uint32_t j = 0; j < leaf_count[i]; ++j, ++k) {
                        if (leaf_refs[k] >= T) {
                                set_error("leaf_refs[%llu]=%u out of range", (unsigned long long)k, leaf_refs[k]);
                                return VRT_ERR_ARG;
                        }
                        keys[k] = (m << tb) | leaf_refs[k];
                }
        }
        if (t->keys_a.reserve(std::max<uint64_t>(n, 1) * 8))
                return VRT_ERR_NOMEM;
        cudaStream_t s = t->stream;
        if (n)
                VRT_CUDA(cudaMemcpyAsync(t->keys_a.p, keys.data(), n * 8, cudaMemcpyHostToDevice, s));
        float* d_root6 = reinterpret_cast<float*>(t->d_counter + 8);
        VRT_CUDA(cudaMemcpyAsync(d_root6, root_aabb, 24, cudaMemcpyHostToDevice, s));
        VRT_CUDA(cudaStreamSynchronize(s));
        return finish_from_keys(t, t->keys_a.as<unsigned long long>(), n, L, tb, false, d_root6);
}

// ---------------------------------------------------------------------------
// Content hulls (round 2).  hull[i] of interior node i = per axis the smallest min plane and the
// largest max plane over the node's non-empty LEAF cells, as the very floats of the leaf level of
// the axis table (no arithmetic: min/max of existing values).  Bottom-up, one launch per level;
// the parents of leaves read the leaf cells through leaf_morton, the levels above combine their
// children's hulls.  The ray kernels skip a child whose hull the ray misses: for a tame ray
// t(p) = (p - o) * dinv is monotone in p after rounding, so every leaf cell's per-axis slab
// interval lies inside the hull's and a leaf the reference would accept implies
// max(t0_hull, tmin) <= min(t1_hull, tmax); the contrapositive is the prune.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_hull_level(const uint2* __restrict__ nodes, const unsigned long long* __restrict__ leaf_morton,
             const float2* __restrict__ tab, uint64_t stride, int level /* of the nodes */, int L, uint64_t begin,
             uint64_t count, uint64_t leaf_base, float4* __restrict__ hull, uint8_t* __restrict__ tight8,
             unsigned long long* __restrict__ codes, float sa_max)
{
        const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= count)
                return;
        const uint64_t node = begin + i;
        const uint2 rec = nodes[node];
        const uint32_t mask = rec.y & 0xffu;
        const bool child_is_leaf = (level + 1 == L);
        const uint32_t cbase = 2u << level;  // table offset of the children's level
        const float inf = __int_as_float(0x7f800000);
        float2 hx = make_float2(inf, -inf), hy = hx, hz = hx;
        unsigned long long code = 0;
        uint32_t tight = 0, m = mask;
        uint64_t ch = rec.x;
        while (m) {
                const uint32_t c = __ffs((int)m) - 1;
                m &= m - 1u;
                float2 bx, by, bz;
                const unsigned long long cc = child_is_leaf ? leaf_morton[ch - leaf_base] : codes[ch];
                code = cc >> 3;
                const float2 cx = tab[0 * stride + cbase + compact1by2(cc >> 2)];  // the child's own cell
                const float2 cy = tab[1 * stride + cbase + compact1by2(cc >> 1)];
                const float2 cz = tab[2 * stride + cbase + compact1by2(cc)];
                if (child_is_leaf) {
                        bx = cx;
                        by = cy;
                        bz = cz;
                } else {
                        const float4 ca = hull[2 * ch], cb = hull[2 * ch + 1];
                        bx = make_float2(ca.z, ca.w);
                        by = make_float2(cb.x, cb.y);
                        bz = make_float2(cb.z, cb.w);
                        // "tight": a ray that crosses the child's cell misses the child's content often enough to pay for
                        // the test.  For convex bodies the mean projected area is proportional to the surface area, so
                        // P(a line through the cell also meets the hull) ~ area(hull) / area(cell); the ray kernel only
                        // tests children whose ratio is below `sa_max` (a heuristic: skipping a test never changes a
                        // result, it only gives up a pruning opportunity).
                        const float hx_ = bx.y - bx.x, hy_ = by.y - by.x, hz_ = bz.y - bz.x;
                        const float ex_ = cx.y - cx.x, ey_ = cy.y - cy.x, ez_ = cz.y - cz.x;
                        if (hx_ * hy_ + hy_ * hz_ + hz_ * hx_ <= sa_max * (ex_ * ey_ + ey_ * ez_ + ez_ * ex_))
                                tight |= 1u << c;
                }
                hx.x = fminf(hx.x, bx.x); hx.y = fmaxf(hx.y, bx.y);
                hy.x = fminf(hy.x, by.x); hy.y = fmaxf(hy.y, by.y);
                hz.x = fminf(hz.x, bz.x); hz.y = fmaxf(hz.y, bz.y);
                ++ch;
        }
        codes[node] = code;
        // record: first child, child mask | tight-children mask << 8, then the hull (the tight mask also goes to its
        // own byte array for the statistics / debug readers)
        tight8[node] = (uint8_t)tight;
        hull[2 * node] = make_float4(__uint_as_float(rec.x), __uint_as_float(mask | (tight << 8)), hx.x, hx.y);
        hull[2 * node + 1] = make_float4(hy.x, hy.y, hz.x, hz.y);
}

// v0, e1 = v1 - v0, e2 = v2 - v0 in double: exactly the widening + SUB steps intersect_triangle3 starts with
__global__ void __launch_bounds__(256)
k_tri64(const float4* __restrict__ tri4, uint32_t T, double* __restrict__ out)
{
        const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
        if (t >= T)
                return;
        const float4 a = tri4[3ull * t], b = tri4[3ull * t + 1], c = tri4[3ull * t + 2];
        const double av[3] = { (double)a.x, (double)a.y, (double)a.z };
        const double bv[3] = { (double)b.x, (double)b.y, (double)b.z };
        const double cv[3] = { (double)c.x, (double)c.y, (double)c.z };
        double* o = out + 10ull * t;  // 80-byte records: 16-byte aligned for double2 loads
        o[9] = 0.0;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                o[k] = av[k];
                o[3 + k] = dsub(bv[k], av[k]);
                o[6 + k] = dsub(cv[k], av[k]);
        }
}

int compute_hulls(vrt_tree* t)
{
        const BlobHeader& h = t->hdr;
        const int L = h.max_depth - 1;
        t->dev.hull = nullptr;
        t->dev.tri64 = nullptr;
        if (h.num_tris) {
                if (t->tri64_buf.reserve((uint64_t)h.num_tris * 80))
                        return VRT_ERR_NOMEM;
                k_tri64<<<grid_for(h.num_tris, 256), 256, 0, t->stream>>>(t->dev.tri4, h.num_tris, t->tri64_buf.as<double>());
                count_launch();
                t->dev.tri64 = t->tri64_buf.as<double>();
        }
        static int enabled = -1;
        if (enabled < 0) {
                const char* e = getenv("VRT_HULL");
                enabled = (e && e[0] == '0') ? 0 : 1;
        }
        t->dev.rec_mask = enabled ? 0xffffu : 0x00ffu;  // (VRT_HULL=0: the records are built, the tests are off)
        if (L < 1 || h.num_nodes == 0)
                return VRT_OK;
        const uint64_t interior = h.num_nodes - h.num_leaves;
        if (t->hull_buf.reserve(std::max<uint64_t>(interior, 1) * 33))  // 32-byte records, then one flag byte per node
                return VRT_ERR_NOMEM;
        float4* hull = t->hull_buf.as<float4>();
        static float sa_max = -1.f;  // VRT_HULL_SA: area ratio below which a child's hull is tested (k_hull_level)
        if (sa_max < 0.f) {
                const char* e = getenv("VRT_HULL_SA");
                sa_max = e ? (float)atof(e) : 0.7f;
        }
        // Morton codes of the interior nodes, bottom-up (a node's code = its first child's >> 3): scratch
        if (t->keys_b.reserve(std::max<uint64_t>(interior, 1) * 8))
                return VRT_ERR_NOMEM;
        unsigned long long* codes = t->keys_b.as<unsigned long long>();
        const uint64_t leaf_base = h.level_offset[L];
        for (int l = L - 1; l >= 0; --l) {
                const uint64_t begin = h.level_offset[l], count = h.level_offset[l + 1] - begin;
                if (!count)
                        continue;
                k_hull_level<<<grid_for(count, 256), 256, 0, t->stream>>>(t->dev.nodes, t->dev.leaf_morton, t->dev.tab2[0],
                                                                          h.axis_tab_stride, l, L, begin, count, leaf_base, hull,
                                                                          reinterpret_cast<uint8_t*>(hull + 2ull * interior), codes,
                                                                          sa_max);
                count_launch();
        }
        VRT_CUDA(cudaGetLastError());
        t->dev.hull = hull;
        t->dev.tight8 = reinterpret_cast<const uint8_t*>(hull + 2ull * interior);
        return VRT_OK;
}

}  // namespace vrt
