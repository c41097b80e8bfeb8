// vrt_gi.cu -- the GI rows of SURVEY.md 8(f) on the flat octree:
//   light-map splat      main.cc:75-97     -> gi_splat_camera (ray kernel in OUT_SPLAT mode, radix sort
//                                             by (leaf, ray), ordered per-leaf accumulation)
//   cone_trace_init_filter voxel_octree.cc:190-214 -> gi_filter (one kernel per level, bottom-up)
//   cone_trace           voxel_octree.cc:247-303 -> gi_cone_points (and, fused after the traversal, the
//                                             OUT_GI_FILM mode of the ray kernel in vrt_trace.cu)
// The reference accumulates the light map from pool threads without synchronisation; the result of
// this file is the SEQUENTIAL member of that family (pixel order, samples in order), reproduced
// exactly by summing every leaf's contributions in ray order.
#include <algorithm>
#include <cstdlib>

#include "vrt_gi.cuh"

namespace vrt {

static inline unsigned gi_grid(uint64_t n, unsigned block)
{
        return (unsigned)std::max<uint64_t>(1, (n + block - 1) / block);
}

int gi_init(vrt_tree* t)
{
        const uint64_t n = std::max<uint64_t>(t->hdr.num_nodes, 1);
        if (t->gi_buf.reserve(n * kGiStride * sizeof(float) + 16))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemsetAsync(t->gi_buf.p, 0, n * kGiStride * sizeof(float) + 16, t->stream));
        t->dev.gi = t->gi_buf.as<float>();
        t->dev.gi_ok = reinterpret_cast<const uint32_t*>(t->gi_buf.as<float>() + n * kGiStride);
        return VRT_OK;
}

// One thread per sorted key; the thread that holds the first key of a leaf walks the leaf's
// segment in order (ascending ray index) and adds coeff_i * illum to the six lobes exactly like
// main.cc:88-95: illum = albedo * clamp(dot(normal, -ray.d),0,1) * color(1,1,1)
// (Triangle::get_diffuse voxel_octree.cc:462-469, untextured albedo = material diffuse).
__global__ void k_gi_accumulate(const unsigned long long* __restrict__ keys, uint64_t n,
                                const float4* __restrict__ recs, uint32_t leaf_node0, float* __restrict__ gi)
{
        const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        const unsigned long long k = keys[i];
        if (k == ~0ull)
                return;
        const uint32_t leaf = (uint32_t)(k >> 32);
        if (i > 0 && (uint32_t)(keys[i - 1] >> 32) == leaf)
                return;
        float* g = gi + (size_t)kGiStride * (leaf_node0 + leaf);
        float acc[18];
#pragma unroll
        for (int f = 0; f < 18; ++f)
                acc[f] = g[4 * (f / 3) + f % 3];
        for (uint64_t j = i; j < n; ++j) {
                const unsigned long long kj = keys[j];
                if (kj == ~0ull || (uint32_t)(kj >> 32) != leaf)
                        break;
                const float4 r = __ldg(&recs[2ull * (uint32_t)kj]);  // normal.xyz, illum.x
                const float4 r1 = __ldg(&recs[2ull * (uint32_t)kj + 1]);  // illum.yz
                const float illum[3] = { r.w, r1.x, r1.y };
#pragma unroll
                for (int f = 0; f < 6; ++f) {
                        const float s = (f < 3) ? 1.f : -1.f;
                        const float ax = (f % 3 == 0) ? s : 0.f, ay = (f % 3 == 1) ? s : 0.f, az = (f % 3 == 2) ? s : 0.f;
                        const float coeff = clampf(dot3(ax, ay, az, r.x, r.y, r.z), 0.f, 1.f);
#pragma unroll
                        for (int c = 0; c < 3; ++c)
                                acc[3 * f + c] = fadd(acc[3 * f + c], fmul(coeff, illum[c]));
                }
        }
#pragma unroll
        for (int f = 0; f < 18; ++f)
                g[4 * (f / 3) + f % 3] = acc[f];
}

int gi_splat_camera(vrt_tree* t, const vrt_camera* cam, const float kd[3])
{
        if (!t->dev.gi) {
                set_error("vrt_gi_init has not been called on this tree");
                return VRT_ERR_ARG;
        }
        const uint64_t R = (uint64_t)cam->nx * cam->ny * cam->spp;
        if (R == 0 || t->hdr.num_nodes == 0)
                return VRT_OK;
        if (R >= 0xffffffffull) {
                set_error("light camera has too many rays for 32-bit ray indices");
                return VRT_ERR_ARG;
        }
        if (t->keys_a.reserve(R * 8) || t->gi_recs.reserve(R * 32))
                return VRT_ERR_NOMEM;
        // the light map changes: the filtered levels are stale until the next gi_filter (TreeDev::gi_ok)
        VRT_CUDA(cudaMemsetAsync(const_cast<uint32_t*>(t->dev.gi_ok), 0, 4, t->stream));
        CameraLaunch l{ cam, 0, 0, cam->nx, cam->ny, 0, 0, OUT_SPLAT, t->keys_a.p, t->gi_recs.p };
        for (int c = 0; c < 3; ++c)
                l.kd[c] = kd[c];
        l.stream = t->stream;
        int rc = launch_trace_camera(t, l);
        if (rc)
                return rc;
        int lb = 1;
        while ((1ull << lb) < t->hdr.num_leaves)
                ++lb;
        unsigned long long* sorted = nullptr;
        rc = sort_keys_u64(t, R, 0, 32 + lb, &sorted);
        if (rc)
                return rc;
        k_gi_accumulate<<<gi_grid(R, 128), 128, 0, t->stream>>>(sorted, R, t->gi_recs.as<float4>(),
                                                                (uint32_t)(t->hdr.num_nodes - t->hdr.num_leaves),
                                                                t->gi_buf.as<float>());
        count_launch();
        VRT_CUDA(cudaGetLastError());
        return VRT_OK;
}

// cone_trace_init_filter: a leaf that holds voxels has coverage 1 (its illum is the light map) ...
__global__ void k_gi_leaf_coverage(uint32_t first, uint32_t n, float* __restrict__ gi)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i < n) {
#pragma unroll
                for (int f = 0; f < 6; ++f)
                        gi[(size_t)kGiStride * (first + i) + 4 * f + kGiCoverage] = 1.f;
        }
}

// ... an interior node is the sum over its eight children in child order (absent children are the
// reference's empty leaves: exact zeros), divided by 8.
__global__ void k_gi_filter_level(const uint2* __restrict__ nodes, uint32_t first, uint32_t n, float* __restrict__ gi)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        const uint2 rec = nodes[first + i];
        float acc[19];
#pragma unroll
        for (int f = 0; f < 19; ++f)
                acc[f] = 0.f;
        uint32_t child = rec.x;
        for (uint32_t c = 0; c < 8; ++c) {
                if (!((rec.y >> c) & 1u))
                        continue;
                const float4* g4 = reinterpret_cast<const float4*>(gi + (size_t)kGiStride * child);
                const float4 q0 = g4[0], q1 = g4[1], q2 = g4[2], q3 = g4[3], q4 = g4[4], q5 = g4[5];
                const float v[19] = { q0.x, q0.y, q0.z, q1.x, q1.y, q1.z, q2.x, q2.y, q2.z, q3.x,
                                      q3.y, q3.z, q4.x, q4.y, q4.z, q5.x, q5.y, q5.z, q0.w };
#pragma unroll
                for (int f = 0; f < 19; ++f)
                        acc[f] = fadd(acc[f], v[f]);
                ++child;
        }
        float4* g = reinterpret_cast<float4*>(gi + (size_t)kGiStride * (first + i));
        const float cov = fdiv(acc[18], 8.f);
#pragma unroll
        for (int f = 0; f < 6; ++f)
                g[f] = make_float4(fdiv(acc[3 * f], 8.f), fdiv(acc[3 * f + 1], 8.f), fdiv(acc[3 * f + 2], 8.f), cov);
}

// TreeDev::gi_ok: the filter has run, and the root's values (hence every node's) are finite
__global__ void k_gi_root_finite(const float* __restrict__ gi, uint32_t* __restrict__ ok)
{
        bool fin = true;
        for (int f = 0; f < kGiStride; ++f)
                fin = fin && (fabsf(gi[f]) <= 3.402823466e+38f);
        *ok = fin ? 1u : 0u;
}

int gi_filter(vrt_tree* t)
{
        if (!t->dev.gi) {
                set_error("vrt_gi_init has not been called on this tree");
                return VRT_ERR_ARG;
        }
        const BlobHeader& h = t->hdr;
        if (h.num_nodes == 0)
                return VRT_OK;
        const int L = h.max_depth - 1;
        float* gi = t->gi_buf.as<float>();
        k_gi_leaf_coverage<<<gi_grid(h.num_leaves, 256), 256, 0, t->stream>>>((uint32_t)h.level_offset[L],
                                                                             (uint32_t)h.num_leaves, gi);
        count_launch();
        for (int l = L - 1; l >= 0; --l) {
                const uint64_t n = h.level_offset[l + 1] - h.level_offset[l];
                if (!n)
                        continue;
                k_gi_filter_level<<<gi_grid(n, 128), 128, 0, t->stream>>>(t->dev.nodes, (uint32_t)h.level_offset[l],
                                                                          (uint32_t)n, gi);
                count_launch();
        }
        k_gi_root_finite<<<1, 1, 0, t->stream>>>(gi, const_cast<uint32_t*>(t->dev.gi_ok));
        count_launch();
        VRT_CUDA(cudaGetLastError());
        return VRT_OK;
}

struct GiRoot6 {
        float v[6];
};
__global__ void k_gi_step_table(GiRoot6 root, float res, float4* tab)
{
        gi_step_table_fill(root.v, res, tab);
}

int gi_step_table(const vrt_tree* t, float res, cudaStream_t s, const float4** d_steps)
{
        *d_steps = nullptr;
        static int on = -1;  // VRT_GI_STEPS=0: every cone evaluates the marching arithmetic itself
        if (on < 0) {
                const char* e = getenv("VRT_GI_STEPS");
                on = (e && e[0] == '0') ? 0 : 1;
        }
        if (!on)
                return VRT_OK;
        Scratch& tab = t->gi_steps[(t->alt_stream && s == t->alt_stream) ? 1 : 0];
        if (tab.reserve((size_t)(kGiMaxSteps + 2) * sizeof(float4)))  // (+1: the cone loop reads one entry ahead)
                return VRT_ERR_NOMEM;
        GiRoot6 r;
        for (int k = 0; k < 6; ++k)
                r.v[k] = t->hdr.root_aabb[k];
        k_gi_step_table<<<1, 1, 0, s>>>(r, res, tab.as<float4>());
        count_launch();
        VRT_CUDA(cudaGetLastError());
        *d_steps = tab.as<float4>();
        return VRT_OK;
}

struct GiPointParams {
        TreeDev tree;
        float root[6];
        const float4* steps;
        const float* pos;
        const float* nrm;
        uint64_t n;
        float res;
        float* out;
};

__global__ void __launch_bounds__(128) k_gi_cone_points(GiPointParams p)
{
        const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= p.n)
                return;
        const float pos[3] = { p.pos[3 * i], p.pos[3 * i + 1], p.pos[3 * i + 2] };
        const float nrm[3] = { p.nrm[3 * i], p.nrm[3 * i + 1], p.nrm[3 * i + 2] };
        float out[3];
        extern __shared__ float s_gi_path[];
        gi_cone_trace_point(p.tree, p.root, s_gi_path + threadIdx.x, blockDim.x, pos, nrm, p.res, p.steps, out);
        p.out[3 * i] = out[0];
        p.out[3 * i + 1] = out[1];
        p.out[3 * i + 2] = out[2];
}

int gi_cone_points(const vrt_tree* t, const float* d_pos, const float* d_nrm, uint64_t n, float res, float* d_out)
{
        if (!t->dev.gi) {
                set_error("vrt_gi_init has not been called on this tree");
                return VRT_ERR_ARG;
        }
        if (n == 0)
                return VRT_OK;
        GiPointParams p{};
        p.tree = t->dev;
        for (int k = 0; k < 6; ++k)
                p.root[k] = t->hdr.root_aabb[k];
        p.pos = d_pos;
        p.nrm = d_nrm;
        p.n = n;
        p.res = res;
        p.out = d_out;
        {
                const int rc = gi_step_table(t, res, t->stream, &p.steps);
                if (rc)
                        return rc;
        }
        const size_t smem = (size_t)kGiPathWords * std::max(t->dev.L, 1) * 128 * sizeof(float);
        VRT_CUDA(cudaFuncSetAttribute(k_gi_cone_points, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_gi_cone_points<<<gi_grid(n, 128), 128, smem, t->stream>>>(p);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        return VRT_OK;
}

struct GiAlbedoParams {
        TreeDev tree;
        const uint32_t* tri;
        const float* pos;
        uint64_t n;
        float kd[3];
        float* out;
};

__global__ void k_gi_albedo_points(GiAlbedoParams p)
{
        const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= p.n)
                return;
        const float pos[3] = { p.pos[3 * i], p.pos[3 * i + 1], p.pos[3 * i + 2] };
        float out[3];
        gi_albedo(p.tree, p.tri[i], pos, p.kd, out);
        p.out[3 * i] = out[0];
        p.out[3 * i + 1] = out[1];
        p.out[3 * i + 2] = out[2];
}

int gi_albedo_points(const vrt_tree* t, const uint32_t* d_tri, const float* d_pos, uint64_t n, const float kd[3], float* d_out)
{
        if (n == 0)
                return VRT_OK;
        GiAlbedoParams p{};
        p.tree = t->dev;
        p.tri = d_tri;
        p.pos = d_pos;
        p.n = n;
        p.kd[0] = kd[0];
        p.kd[1] = kd[1];
        p.kd[2] = kd[2];
        p.out = d_out;
        k_gi_albedo_points<<<gi_grid(n, 128), 128, 0, t->stream>>>(p);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        return VRT_OK;
}

}  // namespace vrt
