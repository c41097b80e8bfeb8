// vrt_api.cu -- the extern "C" boundary of libvrt.so (include/vrt.h): handle
// management, error reporting, host<->device staging for the host-pointer entry
// points, and the predicate KAT kernels.  No torch types, no CPU fallback.
#include <algorithm>
#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <mutex>
#include <new>
#include <utility>
#include <vector>
#include <sys/types.h>

#include "vrt_exact.cuh"
#include "vrt_internal.h"

namespace vrt {

static thread_local std::string g_err;
static std::atomic<uint64_t> g_launches{ 0 };

void set_error(const char* fmt, ...)
{
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        g_err = buf;
}

bool cuda_ok(cudaError_t e, const char* what)
{
        if (e == cudaSuccess)
                return true;
        set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
        cudaGetLastError();
        return false;
}

void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

// Scratch buffers come from the device's default stream-ordered pool (kept resident: release threshold
// = max), so the many grow / free steps of a first build and of every new handle do not go back to the
// driver; a buffer that has to grow grows by at least 1.5x.  (Buffers that are shared over CUDA IPC --
// vrt_dev_alloc -- and the octree blob itself stay plain cudaMalloc allocations.)
static void pool_setup_once()
{
        static bool done = false;
        if (done)
                return;
        done = true;
        int dev = 0;
        cudaMemPool_t pool;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
                unsigned long long keep = ~0ull;
                cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
}

// Buffers that are dropped while work may still be reading them (a scratch buffer that has to grow in the middle
// of a build, the buffers of a handle that is being freed) are parked here and freed at the next flush point --
// ONE device synchronisation for all of them instead of one per buffer (a fresh handle's first build used to
// spend most of its wall time in those synchronisations).
struct Parked {
        void* p;
        size_t bytes;
        int device;
};
static std::mutex g_parked_mu;
static std::vector<Parked> g_parked;
static size_t g_parked_bytes = 0;

void scratch_flush_deferred()
{
        std::vector<Parked> v;
        {
                std::lock_guard<std::mutex> lk(g_parked_mu);
                v.swap(g_parked);
                g_parked_bytes = 0;
        }
        if (v.empty())
                return;
        // every buffer is freed on the device it lives on, after that device has drained (single-process
        // multi-GPU hosts park buffers of several devices)
        int cur = 0;
        cudaGetDevice(&cur);
        int synced = -1;
        std::sort(v.begin(), v.end(), [](const Parked& a, const Parked& b) { return a.device < b.device; });
        for (const Parked& e : v) {
                if (e.device != synced) {
                        cudaSetDevice(e.device);
                        cudaDeviceSynchronize();  // nothing may still be using the parked buffers
                        synced = e.device;
                }
                cudaFreeAsync(e.p, cudaStreamPerThread);
        }
        cudaSetDevice(cur);
        cudaGetLastError();
}

int Scratch::reserve(size_t bytes)
{
        if (bytes <= cap && p)
                return 0;
        pool_setup_once();
        size_t want = std::max<size_t>(bytes, 256);
        if (p) {
                want = std::max(want, cap * 2);
                release();
                if (g_parked_bytes > (8ull << 30))
                        scratch_flush_deferred();
        }
        if (cudaMallocAsync(&p, want, cudaStreamPerThread) != cudaSuccess ||
            cudaStreamSynchronize(cudaStreamPerThread) != cudaSuccess) {
                cudaGetLastError();
                scratch_flush_deferred();  // give the parked memory back and try once more
                if (cudaMallocAsync(&p, want, cudaStreamPerThread) != cudaSuccess ||
                    cudaStreamSynchronize(cudaStreamPerThread) != cudaSuccess) {
                        cudaGetLastError();
                        p = nullptr;
                        set_error("cudaMallocAsync(%zu) failed", want);
                        return VRT_ERR_NOMEM;
                }
        }
        cap = want;
        return 0;
}

void Scratch::release()
{
        if (p) {
                int dev = 0;
                cudaGetDevice(&dev);  // (a handle's buffers are only touched with its device current: check_tree)
                std::lock_guard<std::mutex> lk(g_parked_mu);
                g_parked.push_back(Parked{ p, cap, dev });
                g_parked_bytes += cap;
        }
        p = nullptr;
        cap = 0;
}

int tree_alloc(vrt_tree** out)
{
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
                cudaGetLastError();
                set_error("no CUDA device available (libvrt has no CPU fallback)");
                return VRT_ERR_CUDA;
        }
        vrt_tree* t = new (std::nothrow) vrt_tree();
        if (!t)
                return VRT_ERR_NOMEM;
        if (!cuda_ok(cudaGetDevice(&t->device), "cudaGetDevice") ||
            !cuda_ok(cudaMalloc(&t->d_counter, 256), "cudaMalloc(counter)") ||
            !cuda_ok(cudaHostAlloc(&t->h_counter, 256, cudaHostAllocMapped), "cudaHostAlloc(counter)") ||
            !cuda_ok(cudaMemset(t->d_counter, 0, 256), "cudaMemset(counter)") ||
            !cuda_ok(cudaMalloc(&t->d_tile_queues, sizeof(uint32_t) * 8 * vrt_tree::kTileQueues), "cudaMalloc(tile queues)") ||
            !cuda_ok(cudaEventCreate(&t->ev0), "cudaEventCreate") ||
            !cuda_ok(cudaEventCreate(&t->ev1), "cudaEventCreate")) {
                vrt_tree_free(t);
                return VRT_ERR_CUDA;
        }
        memset(t->h_counter, 0, 256);  // (words 16..19: the build's host mailbox, ticket 0 = nothing delivered)
        for (int i = 0; i < vrt_tree::kEvRing; ++i)
                if (!cuda_ok(cudaEventCreate(&t->ring0[i]), "cudaEventCreate") ||
                    !cuda_ok(cudaEventCreate(&t->ring1[i]), "cudaEventCreate")) {
                        vrt_tree_free(t);
                        return VRT_ERR_CUDA;
                }
        *out = t;
        return VRT_OK;
}

void tree_bind_views(vrt_tree* t)
{
        t->n_builds++;  // (tables derived from the blob, e.g. the origin-relative axis tables, are stale now)
        const BlobHeader& h = t->hdr;
        char* base = static_cast<char*>(t->blob);
        TreeDev& d = t->dev;
        d.nodes = reinterpret_cast<const uint2*>(base + h.off_nodes);
        d.leaf_morton = reinterpret_cast<const unsigned long long*>(base + h.off_leaf_morton);
        d.leaf_refs = reinterpret_cast<const uint32_t*>(base + h.off_leaf_refs);
        d.tri4 = reinterpret_cast<const float4*>(base + h.off_tri4);
        d.nrm = reinterpret_cast<const float*>(base + h.off_nrm);
        for (int a = 0; a < 3; ++a) {
                d.tab2[a] = reinterpret_cast<const float2*>(base + h.off_axis_tab) + a * h.axis_tab_stride;
                d.tab4[a] = reinterpret_cast<const float4*>(d.tab2[a]);
        }
        d.gi = nullptr;  // GI state belongs to one node array: vrt_gi_init after every (re)build
        d.gi_ok = nullptr;
        d.hull = nullptr;  // compute_hulls() follows every bind
        d.tight8 = nullptr;
        d.tri64 = nullptr;
        d.num_nodes = (uint32_t)h.num_nodes;
        d.num_leaves = (uint32_t)h.num_leaves;
        d.L = h.max_depth - 1;
        d.tame = 1;
        for (int a = 0; a < 3; ++a) {
                const float mn = h.root_aabb[a], mx = h.root_aabb[3 + a];
                if (!(mn <= mx) || !(fabsf(mn) <= 1e18f) || !(fabsf(mx) <= 1e18f))
                        d.tame = 0;
        }
}

static int check_tree(const vrt_tree* t)
{
        if (!t) {
                set_error("null tree handle");
                return VRT_ERR_ARG;
        }
        if (!t->blob || t->hdr.magic != kBlobMagic) {
                set_error("tree handle holds no built octree");
                return VRT_ERR_STATE;
        }
        int dev = -1;
        if (cudaGetDevice(&dev) != cudaSuccess || dev != t->device) {
                cudaGetLastError();
                set_error("tree lives on device %d but the current device is %d", t->device, dev);
                return VRT_ERR_STATE;
        }
        return VRT_OK;
}

static int upload_inputs(vrt_tree* t, const float* tri, const float* nrm, uint32_t T, bool from_device)
{
        const cudaMemcpyKind kind = from_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        const size_t bytes = (size_t)std::max<uint32_t>(T, 1) * 36;
        if (!cuda_ok(cudaMalloc(&t->d_tri_in, bytes), "cudaMalloc(tri)"))
                return VRT_ERR_NOMEM;
        if (T)
                VRT_CUDA(cudaMemcpyAsync(t->d_tri_in, tri, (size_t)T * 36, kind, t->stream));
        if (nrm) {
                if (!cuda_ok(cudaMalloc(&t->d_nrm_in, bytes), "cudaMalloc(nrm)"))
                        return VRT_ERR_NOMEM;
                if (T)
                        VRT_CUDA(cudaMemcpyAsync(t->d_nrm_in, nrm, (size_t)T * 36, kind, t->stream));
        }
        t->hdr.num_tris = T;
        return VRT_OK;
}

static int build_common(const float* tri, const float* nrm, uint32_t T, int max_depth, bool dev, vrt_tree** out,
                        uint32_t flags = 0)
{
        if (!out || (T && !tri)) {
                set_error("vrt_build: null argument");
                return VRT_ERR_ARG;
        }
        *out = nullptr;
        if (max_depth < 1 || max_depth > (int)VRT_MAX_DEPTH) {
                set_error("vrt_build: max_depth %d out of range [1,%u]", max_depth, VRT_MAX_DEPTH);
                return VRT_ERR_ARG;
        }
        vrt_tree* t = nullptr;
        int rc = tree_alloc(&t);
        if (rc)
                return rc;
        t->unit_normals = (flags & VRT_BUILD_UNIT_NORMALS) != 0;
        rc = upload_inputs(t, tri, nrm, T, dev);
        if (!rc)
                rc = build_tree(t, max_depth);
        if (rc) {
                vrt_tree_free(t);
                return rc;
        }
        *out = t;
        return VRT_OK;
}

// ---- indexed ingest: the arrays tinyobj::LoadObj produces, gathered on the device ------------------
// (obj2voxel voxel_octree.cc:334-366 copies attrib->vertices / normals through mesh.indices into one
// Triangle per face; here that gather is one kernel and no per-triangle host object exists.)
__global__ void k_gather_indexed(const float* __restrict__ vertices, const float* __restrict__ normals,
                                 const int32_t* __restrict__ index3, uint32_t T, float* __restrict__ tri,
                                 float* __restrict__ nrm)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;  // one face vertex
        if (i >= 3u * T)
                return;
        const int32_t vi = index3[3 * i], ni = index3[3 * i + 1];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                tri[3ull * i + k] = vertices[3ull * vi + k];
                if (nrm)
                        nrm[3ull * i + k] = normals[3ull * ni + k];
        }
}

// row r of a row-major 3x4 (w = 4, translation m[3]) or 3x3 (w = 3, no translation) matrix times p, as
// ((m0*x + m1*y) + m2*z) [+ m3] with scalar __fmul_rn / __fadd_rn: these are never contracted, not even into the
// packed FFMA2 that ptxas forms from -fmad=false multiply-add chains (vrt_trace.cu), so a float32 evaluation in this
// order on the host reproduces every coordinate
template <int W>
__device__ __forceinline__ float xf_row(const float* __restrict__ m, float x, float y, float z)
{
        float s = __fadd_rn(__fadd_rn(__fmul_rn(m[0], x), __fmul_rn(m[1], y)), __fmul_rn(m[2], z));
        if (W == 4)
                s = __fadd_rn(s, m[3]);
        return s;
}

// vrt_update_xform: the current pose of triangle i (what the build reads) from its rest pose -- moved by the
// transform whose range holds i, copied when no range does.  xf is sorted by first_tri, its ranges disjoint and
// non-empty (validated on the host), so the range of i is the last one starting at or before i.
__global__ void k_apply_xforms(const float* __restrict__ rest_tri, const float* __restrict__ rest_nrm,
                               const vrt_xform* __restrict__ xf, uint32_t num_xf, uint32_t T, float* __restrict__ tri,
                               float* __restrict__ nrm)
{
        const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;  // one triangle
        if (i >= T)
                return;
        uint32_t lo = 0, hi = num_xf;  // lo = number of ranges starting at or before i
        while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (xf[mid].first_tri <= i)
                        lo = mid + 1;
                else
                        hi = mid;
        }
        const vrt_xform* x = (lo && i - xf[lo - 1].first_tri < xf[lo - 1].num_tris) ? &xf[lo - 1] : nullptr;
        const float* p = rest_tri + 9ull * i;
        float* q = tri + 9ull * i;
#pragma unroll
        for (int v = 0; v < 3; ++v) {
                const float px = p[3 * v], py = p[3 * v + 1], pz = p[3 * v + 2];
#pragma unroll
                for (int r = 0; r < 3; ++r)
                        q[3 * v + r] = x ? xf_row<4>(x->m + 4 * r, px, py, pz) : p[3 * v + r];
        }
        if (!nrm)
                return;
        p = rest_nrm + 9ull * i;
        q = nrm + 9ull * i;
#pragma unroll
        for (int v = 0; v < 3; ++v) {
                const float nx = p[3 * v], ny = p[3 * v + 1], nz = p[3 * v + 2];
#pragma unroll
                for (int r = 0; r < 3; ++r)
                        q[3 * v + r] = x ? xf_row<3>(x->n + 3 * r, nx, ny, nz) : p[3 * v + r];
        }
}

static int build_indexed_impl(const float* vertices, uint64_t num_vertices, const float* normals, uint64_t num_normals,
                              const int32_t* index3, uint32_t num_tris, int max_depth, vrt_tree** out)
{
        if (!out || (num_tris && (!vertices || !index3))) {
                set_error("vrt_build_indexed: null argument");
                return VRT_ERR_ARG;
        }
        *out = nullptr;
        if (max_depth < 1 || max_depth > (int)VRT_MAX_DEPTH) {
                set_error("vrt_build_indexed: max_depth %d out of range [1,%u]", max_depth, VRT_MAX_DEPTH);
                return VRT_ERR_ARG;
        }
        for (uint64_t i = 0; i < 3ull * num_tris; ++i) {
                const int32_t vi = index3[3 * i], ni = index3[3 * i + 1];
                if (vi < 0 || (uint64_t)vi >= num_vertices || (normals && (ni < 0 || (uint64_t)ni >= num_normals))) {
                        set_error("vrt_build_indexed: face vertex %llu has vertex_index %d / normal_index %d out of range",
                                  (unsigned long long)i, vi, ni);  // (the reference asserts normal_index != -1)
                        return VRT_ERR_ARG;
                }
        }
        vrt_tree* t = nullptr;
        int rc = tree_alloc(&t);
        if (rc)
                return rc;
        auto fail = [&](int code) {
                vrt_tree_free(t);
                return code;
        };
        const size_t tb = (size_t)std::max<uint32_t>(num_tris, 1) * 36;
        if (!cuda_ok(cudaMalloc(&t->d_tri_in, tb), "cudaMalloc(tri)") ||
            (normals && !cuda_ok(cudaMalloc(&t->d_nrm_in, tb), "cudaMalloc(nrm)")))
                return fail(VRT_ERR_NOMEM);
        t->hdr.num_tris = num_tris;
        if (num_tris) {
                const size_t vb = (size_t)num_vertices * 12, nb = normals ? (size_t)num_normals * 12 : 0, ib = (size_t)num_tris * 36;
                if (t->io_in.reserve(align256(vb) + align256(nb) + ib))
                        return fail(VRT_ERR_NOMEM);
                char* d = static_cast<char*>(t->io_in.p);
                float* d_v = reinterpret_cast<float*>(d);
                float* d_n = normals ? reinterpret_cast<float*>(d + align256(vb)) : nullptr;
                int32_t* d_i = reinterpret_cast<int32_t*>(d + align256(vb) + align256(nb));
                if (!cuda_ok(cudaMemcpyAsync(d_v, vertices, vb, cudaMemcpyHostToDevice, t->stream), "copy vertices") ||
                    (normals && !cuda_ok(cudaMemcpyAsync(d_n, normals, nb, cudaMemcpyHostToDevice, t->stream), "copy normals")) ||
                    !cuda_ok(cudaMemcpyAsync(d_i, index3, ib, cudaMemcpyHostToDevice, t->stream), "copy indices"))
                        return fail(VRT_ERR_CUDA);
                k_gather_indexed<<<(3u * num_tris + 255u) / 256u, 256, 0, t->stream>>>(d_v, d_n, d_i, num_tris, t->d_tri_in,
                                                                                      t->d_nrm_in);
                count_launch();
                if (!cuda_ok(cudaGetLastError(), "k_gather_indexed"))
                        return fail(VRT_ERR_CUDA);
        }
        rc = build_tree(t, max_depth);
        if (rc)
                return fail(rc);
        *out = t;
        return VRT_OK;
}

// ---------------------------------------------------------------------------
// predicate KAT kernels
// ---------------------------------------------------------------------------
__global__ void k_tribox(const float* __restrict__ c, const float* __restrict__ h, const float* __restrict__ tri,
                         uint64_t n, uint8_t* __restrict__ out)
{
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        float cc[3] = { c[3 * i], c[3 * i + 1], c[3 * i + 2] };
        float hh[3] = { h[3 * i], h[3 * i + 1], h[3 * i + 2] };
        const float* p = tri + 9 * i;
        float v0[3] = { p[0], p[1], p[2] }, v1[3] = { p[3], p[4], p[5] }, v2[3] = { p[6], p[7], p[8] };
        out[i] = tribox_overlap(cc, hh, v0, v1, v2) ? 1 : 0;
}

__global__ void k_tri_aabb(const float* __restrict__ box, const float* __restrict__ tri, uint64_t n,
                           uint8_t* __restrict__ out)
{
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        float mn[3] = { box[6 * i], box[6 * i + 1], box[6 * i + 2] };
        float mx[3] = { box[6 * i + 3], box[6 * i + 4], box[6 * i + 5] };
        const float* p = tri + 9 * i;
        float v0[3] = { p[0], p[1], p[2] }, v1[3] = { p[3], p[4], p[5] }, v2[3] = { p[6], p[7], p[8] };
        out[i] = tri_overlaps_aabb(mn, mx, v0, v1, v2) ? 1 : 0;
}

__global__ void k_raytri(const double* __restrict__ in, uint64_t n, uint8_t* __restrict__ res,
                         double* __restrict__ tuv)
{
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        const double* a = in + 15 * i;
        double o[3] = { a[0], a[1], a[2] }, d[3] = { a[3], a[4], a[5] }, v0[3] = { a[6], a[7], a[8] },
               v1[3] = { a[9], a[10], a[11] }, v2[3] = { a[12], a[13], a[14] };
        double t = 0, u = 0, v = 0;
        int r = ray_triangle3(o, d, v0, v1, v2, t, u, v);
        res[i] = (uint8_t)r;
        // on rejection the reference leaves *t untouched and *u/*v at their
        // intermediate values; only report them for accepted hits
        tuv[3 * i] = r ? t : 0.0;
        tuv[3 * i + 1] = r ? u : 0.0;
        tuv[3 * i + 2] = r ? v : 0.0;
}

__global__ void k_aabb_isect(const float* __restrict__ box, const vrt_ray* __restrict__ rays, uint64_t n,
                             uint8_t* __restrict__ out)
{
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= n)
                return;
        float mn[3] = { box[6 * i], box[6 * i + 1], box[6 * i + 2] };
        float mx[3] = { box[6 * i + 3], box[6 * i + 4], box[6 * i + 5] };
        const vrt_ray r = rays[i];
        float o[3] = { r.o[0], r.o[1], r.o[2] };
        float dinv[3] = { slab_dinv(r.d[0]), slab_dinv(r.d[1]), slab_dinv(r.d[2]) };
        out[i] = aabb_isect(mn, mx, o, dinv, r.tmin, r.tmax) ? 1 : 0;
}

__global__ void k_gen_rays(CameraParams cam, int x0, int y0, int x1, int y1, vrt_ray* __restrict__ out)
{
        const int W = x1 - x0;
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        uint64_t n = (uint64_t)W * (y1 - y0) * cam.spp;
        if (i >= n)
                return;
        const int s = (int)(i % cam.spp);
        const uint64_t pix = i / cam.spp;
        const int px = x0 + (int)(pix % W), py = y0 + (int)(pix / W);
        float o[3], d[3];
        gen_ray(cam, px, py, s, o, d);
        vrt_ray r;
        r.o[0] = o[0]; r.o[1] = o[1]; r.o[2] = o[2];
        r.d[0] = d[0]; r.d[1] = d[1]; r.d[2] = d[2];
        r.tmin = cam.tmin;
        r.tmax = cam.tmax;
        out[i] = r;
}

// small RAII device buffer for the stateless batch entry points
struct DevBuf {
        void* p = nullptr;
        ~DevBuf() { if (p) cudaFree(p); }
        int alloc(size_t bytes)
        {
                if (cudaMalloc(&p, std::max<size_t>(bytes, 16)) != cudaSuccess) {
                        cudaGetLastError();
                        set_error("cudaMalloc(%zu) failed", bytes);
                        p = nullptr;
                        return VRT_ERR_NOMEM;
                }
                return 0;
        }
};

static int need_device()
{
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess || n < 1) {
                cudaGetLastError();
                set_error("no CUDA device available (libvrt has no CPU fallback)");
                return VRT_ERR_CUDA;
        }
        return VRT_OK;
}

static CameraParams to_params(const vrt_camera* c)
{
        CameraParams p;
        for (int k = 0; k < 16; ++k)
                p.C[k] = c->C[k];
        p.z = c->z;
        p.tmin = c->tmin;
        p.tmax = c->tmax;
        p.nx = c->nx;
        p.ny = c->ny;
        p.spp = c->spp;
        return p;
}

static int check_camera(const vrt_camera* cam, int x0, int y0, int x1, int y1)
{
        if (!cam || (cam->spp != 1 && cam->spp != 4) || cam->nx < 1 || cam->ny < 1) {
                set_error("bad camera (spp must be 1 or 4, nx/ny >= 1)");
                return VRT_ERR_ARG;
        }
        // the reference asserts the pixel is inside the film (camera.cc:79,97)
        if (x0 < 0 || y0 < 0 || x1 > cam->nx || y1 > cam->ny || x1 < x0 || y1 < y0) {
                set_error("pixel rectangle [%d,%d)x[%d,%d) outside the %dx%d film", x0, x1, y0, y1, cam->nx, cam->ny);
                return VRT_ERR_ARG;
        }
        return VRT_OK;
}

// cone_trace's min_voxel_size.  The march advances by 0.1 * max(1.414 res, 1.1547 dist): for a normal res every step
// grows dist by at least 11.5 % and the march ends (1,608 steps at res = FLT_MIN even for an infinite root box); for
// 0, a negative or a subnormal res the increment rounds away and every cone would loop forever on the device.  NaN
// and +-inf would end at once (zeros) but are never meant.  The first check of every entry point that takes res, so
// a rejected call has touched neither the handle nor any stream.
static int check_gi_res(float res)
{
        if (!(res >= FLT_MIN) || !(res <= FLT_MAX)) {
                set_error("res %g outside [FLT_MIN, FLT_MAX]: the cone march ends only for a finite res >= FLT_MIN "
                          "(main.cc's Res is 0 for a planar scene: take it from the axes of non-zero size)",
                          (double)res);
                return VRT_ERR_ARG;
        }
        return VRT_OK;
}

}  // namespace vrt

using namespace vrt;

uint64_t vrt_tree::scratch_bytes() const
{
        uint64_t b = keys_a.cap + keys_b.cap + tmp_a.cap + tmp_b.cap + tmp_c.cap + hist.cap + refs_s.cap + tab_s.cap +
                     io_in.cap + io_out.cap + hull_buf.cap + tri64_buf.cap;
        for (unsigned l = 0; l <= VRT_MAX_DEPTH; ++l)
                b += level_morton[l].cap + level_first[l].cap + level_mask[l].cap;
        return b;
}

extern "C" {

int vrt_abi_version(void) { return VRT_ABI_VERSION; }

const char* vrt_last_error(void) { return g_err.c_str(); }

int vrt_device_count(void)
{
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess) {
                cudaGetLastError();
                set_error("cudaGetDeviceCount failed");
                return VRT_ERR_CUDA;
        }
        return n;
}

uint64_t vrt_launch_count(void) { return g_launches.load(); }

int vrt_build(const float* tri_xyz, const float* tri_nrm, uint32_t num_tris, int max_depth, vrt_tree** out)
{
        return build_common(tri_xyz, tri_nrm, num_tris, max_depth, false, out);
}

int vrt_build_ex(const float* tri_xyz, const float* tri_nrm, uint32_t num_tris, int max_depth, uint32_t flags,
                 vrt_tree** out)
{
        if (flags & ~(uint32_t)VRT_BUILD_UNIT_NORMALS) {
                set_error("vrt_build_ex: unknown flags 0x%x", flags);
                return VRT_ERR_ARG;
        }
        return build_common(tri_xyz, tri_nrm, num_tris, max_depth, false, out, flags);
}

int vrt_build_indexed(const float* vertices, uint64_t num_vertices, const float* normals, uint64_t num_normals,
                      const int32_t* index3, uint32_t num_tris, int max_depth, vrt_tree** out)
{
        return build_indexed_impl(vertices, num_vertices, normals, num_normals, index3, num_tris, max_depth, out);
}

int vrt_build_dev(const float* d_tri_xyz, const float* d_tri_nrm, uint32_t num_tris, int max_depth, vrt_tree** out)
{
        return build_common(d_tri_xyz, d_tri_nrm, num_tris, max_depth, true, out);
}

int vrt_rebuild(vrt_tree* tree, int max_depth)
{
        if (!tree || !tree->d_tri_in) {
                set_error("vrt_rebuild: handle holds no input triangles");
                return VRT_ERR_STATE;
        }
        if (max_depth < 1 || max_depth > (int)VRT_MAX_DEPTH) {
                set_error("vrt_rebuild: max_depth %d out of range", max_depth);
                return VRT_ERR_ARG;
        }
        return build_tree(tree, max_depth);
}

void vrt_tree_free(vrt_tree* t)
{
        if (!t)
                return;
        if (t->blob && t->own_blob)
                cudaFree(t->blob);
        if (t->d_tri_in)
                cudaFree(t->d_tri_in);
        if (t->d_nrm_in)
                cudaFree(t->d_nrm_in);
        if (t->d_tri_rest)
                cudaFree(t->d_tri_rest);
        if (t->d_nrm_rest)
                cudaFree(t->d_nrm_rest);
        t->xf_buf.release();
        t->keys_a.release();
        t->keys_b.release();
        t->tmp_a.release();
        t->tmp_b.release();
        t->tmp_c.release();
        t->hist.release();
        t->refs_s.release();
        t->tab_s.release();
        t->io_in.release();
        t->gi_buf.release();
        t->hull_buf.release();
        t->tri64_buf.release();
        t->gi_recs.release();
        t->gi_steps[0].release();
        t->gi_steps[1].release();
        t->tabrel_buf.release();
        for (auto& rs : t->tabrel_slot)
                if (rs.ev) {
                        cudaEventDestroy(rs.ev);
                        cudaEventDestroy(rs.ev_read);
                }
        t->mat_buf.release();
        t->io_out.release();
        t->film_dev[0].release();
        t->film_dev[1].release();
        if (t->copy_stream)
                cudaStreamDestroy(t->copy_stream);
        if (t->alt_stream)
                cudaStreamDestroy(t->alt_stream);
        for (int i = 0; i < 2; ++i) {
                if (t->film_ready[i])
                        cudaEventDestroy(t->film_ready[i]);
                if (t->film_copied[i])
                        cudaEventDestroy(t->film_copied[i]);
        }
        if (t->gi_written)
                cudaEventDestroy(t->gi_written);
        for (unsigned l = 0; l <= VRT_MAX_DEPTH; ++l) {
                t->level_morton[l].release();
                t->level_first[l].release();
                t->level_mask[l].release();
        }
        scratch_flush_deferred();
        if (t->d_counter)
                cudaFree(t->d_counter);
        if (t->d_tile_queues)
                cudaFree(t->d_tile_queues);
        if (t->h_counter)
                cudaFreeHost(t->h_counter);
        if (t->ev0)
                cudaEventDestroy(t->ev0);
        if (t->ev1)
                cudaEventDestroy(t->ev1);
        for (int i = 0; i < vrt_tree::kEvRing; ++i) {
                if (t->ring0[i])
                        cudaEventDestroy(t->ring0[i]);
                if (t->ring1[i])
                        cudaEventDestroy(t->ring1[i]);
        }
        cudaGetLastError();
        delete t;
}

int vrt_tree_get_info(const vrt_tree* t, vrt_tree_info* out)
{
        if (!out) {
                set_error("null out");
                return VRT_ERR_ARG;
        }
        int rc = check_tree(t);
        if (rc)
                return rc;
        memset(out, 0, sizeof *out);
        out->num_tris = t->hdr.num_tris;
        out->max_depth = t->hdr.max_depth;
        memcpy(out->root_aabb, t->hdr.root_aabb, 24);
        out->num_nodes = t->hdr.num_nodes;
        out->num_leaves = t->hdr.num_leaves;
        out->num_refs = t->hdr.num_refs;
        memcpy(out->level_offset, t->hdr.level_offset, sizeof out->level_offset);
        out->device_bytes = t->blob_bytes + t->scratch_bytes() + (t->d_tri_in ? (uint64_t)t->hdr.num_tris * 36 : 0) +
                            (t->d_nrm_in ? (uint64_t)t->hdr.num_tris * 36 : 0) +
                            (t->d_tri_rest ? (uint64_t)t->hdr.num_tris * 36 : 0) +
                            (t->d_nrm_rest ? (uint64_t)t->hdr.num_tris * 36 : 0);
        out->build_ms = t->build_ms;
        return VRT_OK;
}

int vrt_tree_export(const vrt_tree* t, vrt_tree_view* out)
{
        if (!out) {
                set_error("null out");
                return VRT_ERR_ARG;
        }
        int rc = check_tree(t);
        if (rc)
                return rc;
        const BlobHeader& h = t->hdr;
        const char* base = static_cast<const char*>(t->blob);
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        if (out->leaf_refs && h.num_refs)
                VRT_CUDA(cudaMemcpy(out->leaf_refs, base + h.off_leaf_refs, h.num_refs * 4, cudaMemcpyDeviceToHost));
        if (out->nodes && h.num_nodes)
                VRT_CUDA(cudaMemcpy(out->nodes, base + h.off_nodes, h.num_nodes * 8, cudaMemcpyDeviceToHost));
        if ((out->leaf_cell || out->leaf_count) && h.num_leaves) {
                std::vector<unsigned long long> m(h.num_leaves);
                std::vector<uint2> ln(h.num_leaves);
                VRT_CUDA(cudaMemcpy(m.data(), base + h.off_leaf_morton, h.num_leaves * 8, cudaMemcpyDeviceToHost));
                VRT_CUDA(cudaMemcpy(ln.data(), base + h.off_nodes + h.level_offset[h.max_depth - 1] * 8,
                                    h.num_leaves * 8, cudaMemcpyDeviceToHost));
                for (uint64_t i = 0; i < h.num_leaves; ++i) {
                        if (out->leaf_cell) {
                                // de-interleave: x bit2, y bit1, z bit0 of every 3-bit digit
                                uint32_t x = 0, y = 0, z = 0;
                                for (int l = 0; l < h.max_depth - 1; ++l) {
                                        unsigned dgt = (unsigned)((m[i] >> (3 * l)) & 7ull);
                                        x |= ((dgt >> 2) & 1u) << l;
                                        y |= ((dgt >> 1) & 1u) << l;
                                        z |= (dgt & 1u) << l;
                                }
                                out->leaf_cell[3 * i] = x;
                                out->leaf_cell[3 * i + 1] = y;
                                out->leaf_cell[3 * i + 2] = z;
                        }
                        if (out->leaf_count)
                                out->leaf_count[i] = ln[i].y;
                }
        }
        return VRT_OK;
}

int vrt_tree_import(const float* tri_xyz, const float* tri_nrm, uint32_t num_tris, int max_depth,
                    const float root_aabb[6], uint64_t num_leaves, const uint32_t* leaf_cell,
                    const uint32_t* leaf_count, const uint32_t* leaf_refs, vrt_tree** out)
{
        if (!out || (num_tris && !tri_xyz) || !root_aabb || (num_leaves && (!leaf_cell || !leaf_count || !leaf_refs))) {
                set_error("vrt_tree_import: null argument");
                return VRT_ERR_ARG;
        }
        *out = nullptr;
        if (max_depth < 1 || max_depth > (int)VRT_MAX_DEPTH) {
                set_error("vrt_tree_import: max_depth %d out of range", max_depth);
                return VRT_ERR_ARG;
        }
        vrt_tree* t = nullptr;
        int rc = tree_alloc(&t);
        if (rc)
                return rc;
        rc = upload_inputs(t, tri_xyz, tri_nrm, num_tris, false);
        if (!rc)
                rc = import_leaves(t, max_depth, root_aabb, num_leaves, leaf_cell, leaf_count, leaf_refs);
        if (rc) {
                vrt_tree_free(t);
                return rc;
        }
        *out = t;
        return VRT_OK;
}

int vrt_tree_set_stream(vrt_tree* t, void* stream)
{
        if (!t) {
                set_error("null tree handle");
                return VRT_ERR_ARG;
        }
        t->stream = static_cast<cudaStream_t>(stream);
        return VRT_OK;
}

int vrt_tree_blob_dev(const vrt_tree* t, const void** d_blob, uint64_t* bytes)
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        if (!d_blob || !bytes) {
                set_error("null out");
                return VRT_ERR_ARG;
        }
        *d_blob = t->blob;
        *bytes = t->hdr.bytes;
        return VRT_OK;
}

// A blob comes from another process or from a file: every size and offset of its header is checked
// against the blob before a kernel may follow it (a truncated or corrupt checkpoint is VRT_ERR_ARG,
// not an out-of-bounds read on the device).
static bool blob_header_ok(const BlobHeader& h, uint64_t bytes)
{
        if (h.magic != kBlobMagic || h.bytes > bytes || h.bytes < kHeaderBytes)
                return false;
        if (h.max_depth < 1 || h.max_depth > (int)VRT_MAX_DEPTH)
                return false;
        const int L = h.max_depth - 1;
        if (h.num_nodes >= 0xffffffffull || h.num_leaves > h.num_nodes || h.num_refs >= (1ull << 40))
                return false;
        if (h.level_offset[0] != 0)
                return false;
        for (int l = 0; l <= L; ++l)
                if (h.level_offset[l + 1] < h.level_offset[l])
                        return false;
        if (h.level_offset[L + 1] != h.num_nodes || h.level_offset[L + 1] - h.level_offset[L] != h.num_leaves)
                return false;
        if (h.axis_tab_stride != (2ull << L))
                return false;
        auto fits = [&](uint64_t off, uint64_t count, uint64_t elem) {
                return off >= kHeaderBytes && off <= h.bytes && count <= (h.bytes - off) / elem;
        };
        return fits(h.off_nodes, h.num_nodes, 8) && fits(h.off_leaf_morton, h.num_leaves, 8) &&
               fits(h.off_leaf_refs, h.num_refs, 4) && fits(h.off_tri4, 3ull * h.num_tris, 16) &&
               fits(h.off_nrm, 9ull * h.num_tris, 4) && fits(h.off_axis_tab, 3ull * h.axis_tab_stride, 8);
}

int vrt_tree_from_blob_dev(const void* d_blob, uint64_t bytes, vrt_tree** out)
{
        if (!d_blob || !out || bytes < kHeaderBytes) {
                set_error("vrt_tree_from_blob_dev: bad argument");
                return VRT_ERR_ARG;
        }
        *out = nullptr;
        vrt_tree* t = nullptr;
        int rc = tree_alloc(&t);
        if (rc)
                return rc;
        BlobHeader h;
        if (!cuda_ok(cudaMemcpy(&h, d_blob, sizeof h, cudaMemcpyDeviceToHost), "read blob header")) {
                vrt_tree_free(t);
                return VRT_ERR_CUDA;
        }
        if (!blob_header_ok(h, bytes)) {
                set_error("not a valid vrt octree blob (magic, sizes or section offsets inconsistent)");
                vrt_tree_free(t);
                return VRT_ERR_ARG;
        }
        if (!cuda_ok(cudaMalloc(&t->blob, h.bytes), "cudaMalloc(blob)")) {
                vrt_tree_free(t);
                return VRT_ERR_NOMEM;
        }
        t->blob_bytes = h.bytes;
        t->own_blob = true;
        if (!cuda_ok(cudaMemcpy(t->blob, d_blob, h.bytes, cudaMemcpyDeviceToDevice), "copy blob")) {
                vrt_tree_free(t);
                return VRT_ERR_CUDA;
        }
        t->hdr = h;
        tree_bind_views(t);
        rc = compute_hulls(t);
        if (rc) {
                vrt_tree_free(t);
                return rc;
        }
        *out = t;
        return VRT_OK;
}

int vrt_tree_save(const vrt_tree* t, const char* path)
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        if (!path) {
                set_error("null path");
                return VRT_ERR_ARG;
        }
        std::vector<char> host(t->hdr.bytes);
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        VRT_CUDA(cudaMemcpy(host.data(), t->blob, t->hdr.bytes, cudaMemcpyDeviceToHost));
        FILE* f = fopen(path, "wb");
        if (!f) {
                set_error("cannot open %s for writing", path);
                return VRT_ERR_ARG;
        }
        const size_t w = fwrite(host.data(), 1, host.size(), f);
        fclose(f);
        if (w != host.size()) {
                set_error("short write to %s", path);
                return VRT_ERR_ARG;
        }
        return VRT_OK;
}

int vrt_tree_load(const char* path, vrt_tree** out)
{
        if (!path || !out) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        *out = nullptr;
        FILE* f = fopen(path, "rb");
        if (!f) {
                set_error("cannot open %s", path);
                return VRT_ERR_ARG;
        }
        fseeko(f, 0, SEEK_END);
        const off_t sz = ftello(f);
        fseeko(f, 0, SEEK_SET);
        if (sz < (off_t)kHeaderBytes) {
                fclose(f);
                set_error("%s is not a vrt octree checkpoint", path);
                return VRT_ERR_ARG;
        }
        std::vector<char> host((size_t)sz);
        const size_t r = fread(host.data(), 1, host.size(), f);
        fclose(f);
        BlobHeader h;
        memcpy(&h, host.data(), sizeof h);
        if (r != host.size() || !blob_header_ok(h, (uint64_t)sz)) {
                set_error("%s is not a vrt octree checkpoint (magic/size mismatch)", path);
                return VRT_ERR_ARG;
        }
        int rc = need_device();
        if (rc)
                return rc;
        DevBuf d;
        if (d.alloc(h.bytes))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpy(d.p, host.data(), h.bytes, cudaMemcpyHostToDevice));
        return vrt_tree_from_blob_dev(d.p, h.bytes, out);
}

// ---- camera -----------------------------------------------------------------
// Host arithmetic identical to Camera::Camera (camera.cc:65-75): jql::normalize
// = v / sqrtf(((0+x*x)+y*y)+z*z), jql::cross (graphics_math.h:588-592),
// affine_transform (graphics_math.h:1002-1016).  Compiled with -ffp-contract=off.
static void h_normalize(float v[3])
{
        float s = 0.f;
        s += v[0] * v[0];
        s += v[1] * v[1];
        s += v[2] * v[2];
        float l = sqrtf(s);
        v[0] = v[0] / l;
        v[1] = v[1] / l;
        v[2] = v[2] / l;
}

static void h_cross(const float p[3], const float q[3], float o[3])
{
        o[0] = p[1] * q[2] - q[1] * p[2];
        o[1] = p[2] * q[0] - q[2] * p[0];
        o[2] = p[0] * q[1] - q[0] * p[1];
}

int vrt_camera_init(const float cam10[10], float film_h, int nx, int ny, int spp, vrt_camera* out)
{
        if (!cam10 || !out || (spp != 1 && spp != 4) || nx < 1 || ny < 1) {
                set_error("vrt_camera_init: bad argument");
                return VRT_ERR_ARG;
        }
        const float fov = cam10[0];
        const float* eye = cam10 + 1;
        const float* spot = cam10 + 4;
        const float* up = cam10 + 7;
        float f[3] = { spot[0] - eye[0], spot[1] - eye[1], spot[2] - eye[2] };
        h_normalize(f);
        float s[3], u[3];
        h_cross(f, up, s);
        h_normalize(s);
        h_cross(s, f, u);
        h_normalize(u);
        memset(out, 0, sizeof *out);
        for (int r = 0; r < 3; ++r) {
                out->C[r] = s[r];
                out->C[4 + r] = u[r];
                out->C[8 + r] = -f[r];
                out->C[12 + r] = eye[r];
        }
        out->C[15] = 1.f;
        out->z = -(film_h / (2 * tanf(fov / 2)));  // camera.cc:82,100
        out->tmin = 0.f;                           // camera.h:76
        out->tmax = FLT_MAX;                       // camera.h:77
        out->nx = nx;
        out->ny = ny;
        out->spp = spp;
        return VRT_OK;
}

int vrt_gen_rays(const vrt_camera* cam, int x0, int y0, int x1, int y1, vrt_ray* rays_out)
{
        int rc = need_device();
        if (rc)
                return rc;
        rc = check_camera(cam, x0, y0, x1, y1);
        if (rc)
                return rc;
        const uint64_t n = (uint64_t)(x1 - x0) * (y1 - y0) * cam->spp;
        if (!n)
                return VRT_OK;
        if (!rays_out) {
                set_error("null rays_out");
                return VRT_ERR_ARG;
        }
        DevBuf d;
        if (d.alloc(n * sizeof(vrt_ray)))
                return VRT_ERR_NOMEM;
        k_gen_rays<<<(unsigned)((n + 255) / 256), 256>>>(to_params(cam), x0, y0, x1, y1, static_cast<vrt_ray*>(d.p));
        count_launch();
        VRT_CUDA(cudaGetLastError());
        VRT_CUDA(cudaMemcpy(rays_out, d.p, n * sizeof(vrt_ray), cudaMemcpyDeviceToHost));
        return VRT_OK;
}

// ---- trace ------------------------------------------------------------------
int vrt_trace_rays_dev(const vrt_tree* t, const vrt_ray* d_rays, uint64_t n, vrt_hit* d_out)
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        if (n && (!d_rays || !d_out)) {
                set_error("null ray/out pointer");
                return VRT_ERR_ARG;
        }
        return launch_trace_rays(t, d_rays, n, d_out);
}

int vrt_trace_rays(const vrt_tree* tc, const vrt_ray* rays, uint64_t n, vrt_hit* out)
{
        int rc = check_tree(tc);
        if (rc)
                return rc;
        if (!n)
                return VRT_OK;
        if (!rays || !out) {
                set_error("null ray/out pointer");
                return VRT_ERR_ARG;
        }
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        if (t->io_in.reserve(n * sizeof(vrt_ray)) || t->io_out.reserve(n * sizeof(vrt_hit)))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpyAsync(t->io_in.p, rays, n * sizeof(vrt_ray), cudaMemcpyHostToDevice, t->stream));
        rc = launch_trace_rays(t, t->io_in.as<vrt_ray>(), n, t->io_out.as<vrt_hit>());
        if (rc)
                return rc;
        VRT_CUDA(cudaMemcpyAsync(out, t->io_out.p, n * sizeof(vrt_hit), cudaMemcpyDeviceToHost, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        return VRT_OK;
}

static int trace_camera_common(const vrt_tree* tc, const vrt_camera* cam, const vrt_shade* sh, int x0, int y0, int x1,
                               int y1, void* out, OutMode mode, bool dev, const GiArgs* gi = nullptr)
{
        int rc = check_tree(tc);
        if (rc)
                return rc;
        rc = check_camera(cam, x0, y0, x1, y1);
        if (rc)
                return rc;
        const uint64_t npix = (uint64_t)(x1 - x0) * (y1 - y0);
        if (!npix)
                return VRT_OK;
        if (!out || (mode == OUT_FILM && !sh)) {
                set_error("null out/shade pointer");
                return VRT_ERR_ARG;
        }
        if (dev)
                return launch_trace_camera(tc, cam, sh, x0, y0, x1, y1, out, mode, 0, 0, nullptr, 0, gi);
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        const uint64_t bytes = (mode == OUT_FILM || mode == OUT_GI_FILM) ? npix * (uint64_t)vrt_film_pixel_bytes(tc->film_fmt) : npix * cam->spp * (mode == OUT_HIT48 ? 48 : 16);
        if (t->io_out.reserve(bytes))
                return VRT_ERR_NOMEM;
        rc = launch_trace_camera(t, cam, sh, x0, y0, x1, y1, t->io_out.p, mode, 0, 0, nullptr, 0, gi);
        if (rc)
                return rc;
        VRT_CUDA(cudaMemcpyAsync(out, t->io_out.p, bytes, cudaMemcpyDeviceToHost, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        return VRT_OK;
}

int vrt_film_pixel_bytes(int32_t format)
{
        switch (format) {
        case VRT_FILM_F32: return 12;
        case VRT_FILM_RGBE: return 4;
        case VRT_FILM_RGB8: return 3;
        default: set_error("unknown film format %d", (int)format); return VRT_ERR_ARG;
        }
}

int vrt_set_film_format(vrt_tree* t, int32_t format)
{
        if (!t) {
                set_error("null tree");
                return VRT_ERR_ARG;
        }
        if (vrt_film_pixel_bytes(format) < 0)
                return VRT_ERR_ARG;
        t->film_fmt = format;
        return VRT_OK;
}

// Encode an existing float film (host pointers) with the camera kernels' device functions.
int vrt_film_encode(const vrt_tree* tc, const float* film_rgb, uint64_t npix, int32_t format, uint8_t* out)
{
        int rc = check_tree(tc);
        if (rc)
                return rc;
        if (format != VRT_FILM_RGBE && format != VRT_FILM_RGB8) {
                set_error("vrt_film_encode: format must be VRT_FILM_RGBE or VRT_FILM_RGB8");
                return VRT_ERR_ARG;
        }
        if (!npix)
                return VRT_OK;
        if (!film_rgb || !out || npix >= (1ull << 40)) {
                set_error("vrt_film_encode: bad argument");
                return VRT_ERR_ARG;
        }
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        const uint64_t ob = npix * (uint64_t)vrt_film_pixel_bytes(format);
        if (t->io_in.reserve(npix * 12) || t->io_out.reserve(ob))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpyAsync(t->io_in.p, film_rgb, npix * 12, cudaMemcpyHostToDevice, t->stream));
        rc = launch_film_encode(t, t->io_in.as<float>(), npix, format, t->io_out.as<uint8_t>());
        if (rc)
                return rc;
        VRT_CUDA(cudaMemcpyAsync(out, t->io_out.p, ob, cudaMemcpyDeviceToHost, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        return VRT_OK;
}

// stbi_write_hdr's file layout (stb_image_write.h:618-740) over an already encoded RGBE film: the header, then per
// scanline either the flat pixels (nx < 8 or nx >= 32768) or the marker {2, 2, nx >> 8, nx & 255} followed by the
// four components, each run-length encoded on its own: literal dumps of at most 128 bytes up to the next run of
// three equal bytes, runs emitted in pieces of at most 127.
int64_t vrt_hdr_file(const uint8_t* rgbe, int32_t nx, int32_t ny, uint8_t* out, uint64_t cap)
{
        if (!rgbe || nx <= 0 || ny <= 0 || (!out && cap)) {
                set_error("vrt_hdr_file: bad argument");
                return VRT_ERR_ARG;
        }
        uint64_t n = 0;
        auto put = [&](const void* p, size_t len) {
                if (n + len <= cap)
                        memcpy(out + n, p, len);
                n += len;
        };
        static const char header[] = "#?RADIANCE\n# Written by stb_image_write.h\nFORMAT=32-bit_rle_rgbe\n";
        put(header, sizeof(header) - 1);
        char buffer[128];
        const int len = snprintf(buffer, sizeof buffer, "EXPOSURE=          1.0000000000000\n\n-Y %d +X %d\n", (int)ny, (int)nx);
        put(buffer, (size_t)len);
        std::vector<uint8_t> comp((size_t)nx);
        for (int y = 0; y < ny; ++y) {
                const uint8_t* row = rgbe + (size_t)y * nx * 4;
                if (nx < 8 || nx >= 32768) {
                        put(row, (size_t)nx * 4);
                        continue;
                }
                const uint8_t marker[4] = { 2, 2, (uint8_t)((nx & 0xff00) >> 8), (uint8_t)(nx & 0xff) };
                put(marker, 4);
                for (int c = 0; c < 4; ++c) {
                        for (int x = 0; x < nx; ++x)
                                comp[x] = row[4 * (size_t)x + c];
                        int x = 0;
                        while (x < nx) {
                                int r = x;  // first run of three equal bytes at or after x
                                while (r + 2 < nx && !(comp[r] == comp[r + 1] && comp[r] == comp[r + 2]))
                                        ++r;
                                if (r + 2 >= nx)
                                        r = nx;
                                while (x < r) {  // literal bytes up to the run
                                        const int l = std::min(r - x, 128);
                                        const uint8_t lb = (uint8_t)l;
                                        put(&lb, 1);
                                        put(&comp[x], (size_t)l);
                                        x += l;
                                }
                                if (r + 2 < nx) {  // the run itself
                                        while (r < nx && comp[r] == comp[x])
                                                ++r;
                                        while (x < r) {
                                                const int l = std::min(r - x, 127);
                                                const uint8_t rb[2] = { (uint8_t)(l + 128), comp[x] };
                                                put(rb, 2);
                                                x += l;
                                        }
                                }
                        }
                }
        }
        return (int64_t)n;
}

// Streams and events of the pipelined frame loops (vrt_render_camera_async / vrt_render_bands_async): a copy
// stream for the device->host film copies and a second kernel stream, so that consecutive frames alternate
// between two kernel streams (the persistent grid of frame k+1 starts while the last long rays of frame k
// still run) while their copies queue up on the copy stream.
static int async_pipeline_prepare(vrt_tree* t)
{
        if (!t->copy_stream) {
                VRT_CUDA(cudaStreamCreateWithFlags(&t->copy_stream, cudaStreamNonBlocking));
                VRT_CUDA(cudaStreamCreateWithFlags(&t->alt_stream, cudaStreamNonBlocking));
                for (int i = 0; i < 2; ++i) {
                        VRT_CUDA(cudaEventCreateWithFlags(&t->film_ready[i], cudaEventDisableTiming));
                        VRT_CUDA(cudaEventCreateWithFlags(&t->film_copied[i], cudaEventDisableTiming));
                }
                VRT_CUDA(cudaEventCreateWithFlags(&t->gi_written, cudaEventDisableTiming));
        }
        if (t->n_async_frames == 0)  // the alternate stream starts behind everything enqueued so far
                VRT_CUDA(cudaStreamSynchronize(t->stream));
        return VRT_OK;
}
// kernel stream of async frame k: even frames on the handle's stream, odd frames on the alternate one
static cudaStream_t async_kernel_stream(const vrt_tree* t) { return (t->n_async_frames & 1) ? t->alt_stream : t->stream; }

// The writers of the state a GI frame reads (vrt_gi_init, vrt_gi_splat_camera, vrt_gi_filter, vrt_set_materials) work
// on `stream`, while the odd frames of a pipelined sequence run on `alt_stream`.  Between the two calls of this pair
// the writer is ordered after every frame enqueued so far (the even ones are on `stream` already, the last odd one
// recorded film_ready[1]), and every later frame is ordered after the writer (the even ones by stream order, the odd
// ones by the wait of alt_stream).  The frame path itself gains nothing: consecutive frames still overlap.
static int gi_writer_begin(vrt_tree* t)
{
        if (t->n_async_frames >= 2)  // an odd frame of the current sequence exists
                VRT_CUDA(cudaStreamWaitEvent(t->stream, t->film_ready[1], 0));
        return VRT_OK;
}
static int gi_writer_end(vrt_tree* t, int rc)
{
        if (t->alt_stream) {  // (no pipelined frame yet: the first one synchronises with `stream` anyway)
                VRT_CUDA(cudaEventRecord(t->gi_written, t->stream));
                VRT_CUDA(cudaStreamWaitEvent(t->alt_stream, t->gi_written, 0));
        }
        return rc;
}

// Pipelined frame loop: the kernel of frame k+1 runs while frame k's film crosses PCIe.
int vrt_render_camera_async(const vrt_tree* tc, const vrt_camera* cam, const vrt_shade* sh, int x0, int y0, int x1,
                            int y1, float* film_rgb)
{
        int rc = check_tree(tc);
        if (rc)
                return rc;
        rc = check_camera(cam, x0, y0, x1, y1);
        if (rc)
                return rc;
        const uint64_t npix = (uint64_t)(x1 - x0) * (y1 - y0);
        if (!npix)
                return VRT_OK;
        if (!film_rgb || !sh) {
                set_error("null out/shade pointer");
                return VRT_ERR_ARG;
        }
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        rc = async_pipeline_prepare(t);
        if (rc)
                return rc;
        cudaStream_t ks = async_kernel_stream(t);
        const int k = (int)(t->n_async_frames & 1);
        const uint64_t bytes = npix * (uint64_t)vrt_film_pixel_bytes(t->film_fmt);
        if (t->film_dev[k].cap < bytes) {
                VRT_CUDA(cudaStreamSynchronize(t->copy_stream));  // nothing may still read the old buffer
                if (t->film_dev[k].reserve(bytes))
                        return VRT_ERR_NOMEM;
        }
        if (t->n_async_frames >= 2)  // the copy that last read this device film must be done
                VRT_CUDA(cudaStreamWaitEvent(ks, t->film_copied[k], 0));
        t->launch_stream = ks;
        rc = launch_trace_camera(t, cam, sh, x0, y0, x1, y1, t->film_dev[k].p, OUT_FILM);
        t->launch_stream = nullptr;
        if (rc)
                return rc;
        VRT_CUDA(cudaEventRecord(t->film_ready[k], ks));
        VRT_CUDA(cudaStreamWaitEvent(t->copy_stream, t->film_ready[k], 0));
        VRT_CUDA(cudaMemcpyAsync(film_rgb, t->film_dev[k].p, bytes, cudaMemcpyDeviceToHost, t->copy_stream));
        VRT_CUDA(cudaEventRecord(t->film_copied[k], t->copy_stream));
        t->n_async_frames++;
        return VRT_OK;
}

int vrt_trace_camera(const vrt_tree* t, const vrt_camera* cam, int x0, int y0, int x1, int y1, vrt_hit* out)
{
        return trace_camera_common(t, cam, nullptr, x0, y0, x1, y1, out, OUT_HIT48, false);
}
int vrt_trace_camera_dev(const vrt_tree* t, const vrt_camera* cam, int x0, int y0, int x1, int y1, vrt_hit* d_out)
{
        return trace_camera_common(t, cam, nullptr, x0, y0, x1, y1, d_out, OUT_HIT48, true);
}
int vrt_trace_camera16_dev(const vrt_tree* t, const vrt_camera* cam, int x0, int y0, int x1, int y1, vrt_hit16* d_out)
{
        return trace_camera_common(t, cam, nullptr, x0, y0, x1, y1, d_out, OUT_HIT16, true);
}
int vrt_render_camera(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, int x0, int y0, int x1, int y1,
                      float* film_rgb)
{
        return trace_camera_common(t, cam, sh, x0, y0, x1, y1, film_rgb, OUT_FILM, false);
}
int vrt_render_camera_dev(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, int x0, int y0, int x1,
                          int y1, float* d_film_rgb)
{
        return trace_camera_common(t, cam, sh, x0, y0, x1, y1, d_film_rgb, OUT_FILM, true);
}

int vrt_count_camera(const vrt_tree* tc, const vrt_camera* cam, int x0, int y0, int x1, int y1, uint64_t counts[8])
{
        int rc = check_tree(tc);
        if (rc)
                return rc;
        rc = check_camera(cam, x0, y0, x1, y1);
        if (rc)
                return rc;
        if (!counts) {
                set_error("null counts");
                return VRT_ERR_ARG;
        }
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        if (t->io_out.reserve(64))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemsetAsync(t->io_out.p, 0, 64, t->stream));
        memset(counts, 0, 8 * sizeof(uint64_t));
        if (x1 > x0 && y1 > y0) {
                rc = launch_trace_camera(t, cam, nullptr, x0, y0, x1, y1, t->io_out.p, OUT_COUNT);
                if (rc)
                        return rc;
        }
        VRT_CUDA(cudaMemcpyAsync(counts, t->io_out.p, 64, cudaMemcpyDeviceToHost, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        return VRT_OK;
}

int vrt_band_rows(const vrt_camera* cam, const vrt_bands* b)
{
        if (!cam || !b || b->band_h < 1 || b->band_stride < 1 || b->band_first < 0) {
                set_error("bad band description");
                return VRT_ERR_ARG;
        }
        long rows = 0;
        for (long k = b->band_first; k * b->band_h < cam->ny; k += b->band_stride)
                rows += std::min<long>(b->band_h, cam->ny - k * b->band_h);
        return (int)rows;
}

static int bands_common(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, const vrt_bands* b, void* d_out,
                        OutMode mode)
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        rc = check_camera(cam, 0, 0, cam ? cam->nx : 0, cam ? cam->ny : 0);
        if (rc)
                return rc;
        const int rows = vrt_band_rows(cam, b);
        if (rows < 0)
                return rows;
        if (rows == 0)
                return VRT_OK;
        if (!d_out || (mode == OUT_FILM && !sh)) {
                set_error("null out/shade pointer");
                return VRT_ERR_ARG;
        }
        const int y0 = b->band_first * b->band_h;
        return launch_trace_camera(t, cam, sh, 0, y0, cam->nx, y0 + rows, d_out, mode, b->band_h,
                                   b->band_stride * b->band_h);
}

int vrt_render_bands_dev(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, const vrt_bands* b,
                         float* d_film_rgb)
{
        return bands_common(t, cam, sh, b, d_film_rgb, OUT_FILM);
}

// One output's compact band rows (src: this rank's rows, band after band) to their final rows of the full host
// frame dst_full: the full bands by one 2-D copy ("row" = one band of band_h frame rows), then the last, shorter band.
static int copy_bands_to_host(char* dst_full, const char* src, size_t row_bytes, const vrt_bands* b, int rows,
                              cudaStream_t s)
{
        const size_t band_bytes = (size_t)b->band_h * row_bytes;
        const int full_bands = rows / b->band_h, tail_rows = rows % b->band_h;
        char* dst = dst_full + (size_t)b->band_first * band_bytes;
        static int dbg_no_copy = -1;  // VRT_DEBUG_NO_COPY=1: diagnostic only (frames never reach the host)
        if (dbg_no_copy < 0) {
                const char* e = getenv("VRT_DEBUG_NO_COPY");
                dbg_no_copy = (e && e[0] == '1') ? 1 : 0;
        }
        if (full_bands && !dbg_no_copy)
                VRT_CUDA(cudaMemcpy2DAsync(dst, (size_t)b->band_stride * band_bytes, src, band_bytes, band_bytes,
                                           (size_t)full_bands, cudaMemcpyDeviceToHost, s));
        if (tail_rows)
                VRT_CUDA(cudaMemcpyAsync(dst + (size_t)full_bands * b->band_stride * band_bytes,
                                         src + (size_t)full_bands * band_bytes, (size_t)tail_rows * row_bytes,
                                         cudaMemcpyDeviceToHost, s));
        return VRT_OK;
}

// Multi-GPU frame loop to HOST memory: this rank's bands are rendered into one of two device
// band buffers and copied by one strided DMA (cudaMemcpy2DAsync: one row per band) straight to
// their final rows of the full host frame, which every rank of the node maps (shared + pinned),
// so the N ranks use their N PCIe links in parallel and the copy of frame k overlaps the kernel
// of frame k+1 -- the N-GPU counterpart of vrt_render_camera_async.  mode OUT_FILM: the harness
// film (sh); OUT_GI_FILM: the cone-traced GI film (gi->kd, gi->res; the step table is filled on
// the frame's kernel stream); OUT_GI_AOV: the GI film (film_rgb_full may be NULL) plus the planes
// of aov_full (host frames), whose compact band rows share the frame slot's one device buffer.
static int bands_async_common(const vrt_tree* tc, const vrt_camera* cam, const vrt_shade* sh, const GiArgs* gi,
                              const vrt_gi_aov* aov_full, const vrt_bands* b, float* film_rgb_full, OutMode mode)
{
        int rc = check_tree(tc);
        if (rc)
                return rc;
        rc = check_camera(cam, 0, 0, cam ? cam->nx : 0, cam ? cam->ny : 0);
        if (rc)
                return rc;
        const int rows = vrt_band_rows(cam, b);
        if (rows < 0)
                return rows;
        if (rows == 0)
                return VRT_OK;
        if ((mode == OUT_GI_AOV ? !aov_full : !film_rgb_full) || (mode == OUT_FILM ? !sh : !gi)) {
                set_error("null out/shade pointer");
                return VRT_ERR_ARG;
        }
        if (mode != OUT_FILM && !tc->dev.gi) {
                set_error("vrt_gi_init has not been called on this tree");
                return VRT_ERR_ARG;
        }
        // the outputs (film, albedo, direct, indirect, normal, hits): full host frames, and the bytes of one row
        const vrt_gi_aov none = {};
        const vrt_gi_aov& a = mode == OUT_GI_AOV ? *aov_full : none;
        char* const dst[6] = { reinterpret_cast<char*>(film_rgb_full), reinterpret_cast<char*>(a.albedo),
                               reinterpret_cast<char*>(a.direct), reinterpret_cast<char*>(a.indirect),
                               reinterpret_cast<char*>(a.normal), reinterpret_cast<char*>(a.hits) };
        const size_t plane_row = (size_t)cam->nx * 12;
        const size_t row_bytes[6] = { (size_t)cam->nx * (size_t)vrt_film_pixel_bytes(tc->film_fmt), plane_row,
                                      plane_row, plane_row, plane_row, (size_t)cam->nx * cam->spp * sizeof(vrt_hit16) };
        // their compact band rows in the frame slot's one device buffer, each part 256-byte aligned
        uint64_t off[6] = {}, bytes = 0;
        for (int i = 0; i < 6; ++i)
                if (dst[i]) {
                        off[i] = (bytes + 255) & ~255ull;
                        bytes = off[i] + (uint64_t)rows * row_bytes[i];
                }
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        rc = async_pipeline_prepare(t);
        if (rc)
                return rc;
        cudaStream_t ks = async_kernel_stream(t);
        const int k = (int)(t->n_async_frames & 1);
        if (t->film_dev[k].cap < bytes) {
                VRT_CUDA(cudaStreamSynchronize(t->copy_stream));  // nothing may still read the old buffer
                if (t->film_dev[k].reserve(bytes))
                        return VRT_ERR_NOMEM;
        }
        if (t->n_async_frames >= 2)  // the copy that last read this device buffer must be done
                VRT_CUDA(cudaStreamWaitEvent(ks, t->film_copied[k], 0));
        char* const base = static_cast<char*>(t->film_dev[k].p);
        vrt_gi_aov d_aov = {};
        float** const d_planes[4] = { &d_aov.albedo, &d_aov.direct, &d_aov.indirect, &d_aov.normal };
        for (int i = 0; i < 4; ++i)
                if (dst[i + 1])
                        *d_planes[i] = reinterpret_cast<float*>(base + off[i + 1]);
        if (dst[5])
                d_aov.hits = reinterpret_cast<vrt_hit16*>(base + off[5]);
        const int y0 = b->band_first * b->band_h;
        t->launch_stream = ks;
        GiArgs ga{};
        if (mode != OUT_FILM) {
                ga = *gi;
                rc = gi_step_table(t, ga.res, &ga.steps);
        }
        if (!rc)
                rc = launch_trace_camera(t, cam, sh, 0, y0, cam->nx, y0 + rows, dst[0] ? base + off[0] : nullptr, mode,
                                         b->band_h, b->band_stride * b->band_h, nullptr, 0,
                                         mode == OUT_FILM ? nullptr : &ga, mode == OUT_GI_AOV ? &d_aov : nullptr);
        t->launch_stream = nullptr;
        if (rc)
                return rc;
        VRT_CUDA(cudaEventRecord(t->film_ready[k], ks));
        VRT_CUDA(cudaStreamWaitEvent(t->copy_stream, t->film_ready[k], 0));
        for (int i = 0; i < 6 && !rc; ++i)
                if (dst[i])
                        rc = copy_bands_to_host(dst[i], base + off[i], row_bytes[i], b, rows, t->copy_stream);
        if (rc)
                return rc;
        VRT_CUDA(cudaEventRecord(t->film_copied[k], t->copy_stream));
        t->n_async_frames++;
        return VRT_OK;
}

int vrt_render_bands_async(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, const vrt_bands* b,
                           float* film_rgb_full)
{
        return bands_async_common(t, cam, sh, nullptr, nullptr, b, film_rgb_full, OUT_FILM);
}

// The cone-traced GI film (vrt_gi_render_camera) through the same banded, pipelined path.
int vrt_gi_render_bands_async(const vrt_tree* t, const vrt_camera* cam, const float kd[3], float res,
                              const vrt_bands* b, float* film_rgb_full)
{
        if (const int rc = check_gi_res(res))
                return rc;
        if (!kd) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        const GiArgs ga = { { kd[0], kd[1], kd[2] }, res };
        return bands_async_common(t, cam, nullptr, &ga, nullptr, b, film_rgb_full, OUT_GI_FILM);
}

// kd and the planes of a banded plane request: VRT_ERR_ARG for a null pointer or a request without any plane
static int check_gi_aov_request(const float kd[3], const vrt_gi_aov* aov)
{
        if (!kd || !aov) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        if (!aov->albedo && !aov->direct && !aov->indirect && !aov->normal && !aov->hits) {
                set_error("every GI plane is NULL (the film alone is the banded GI film call)");
                return VRT_ERR_ARG;
        }
        return VRT_OK;
}

// The GI film and its planes (vrt_gi_render_aov) through the same banded, pipelined path.
int vrt_gi_render_aov_bands_async(const vrt_tree* t, const vrt_camera* cam, const float kd[3], float res,
                                  const vrt_bands* b, float* film_full_or_null, const vrt_gi_aov* aov_full)
{
        if (const int rc = check_gi_res(res))
                return rc;
        const int rc = check_gi_aov_request(kd, aov_full);
        if (rc)
                return rc;
        const GiArgs ga = { { kd[0], kd[1], kd[2] }, res };
        return bands_async_common(t, cam, nullptr, &ga, aov_full, b, film_full_or_null, OUT_GI_AOV);
}

// ---- animated geometry: new input triangles, then the build of vrt_rebuild ---------------------------------------
// An update writes the pose the build reads (d_tri_in / d_nrm_in) on `stream` and runs build_tree, which rewrites the
// blob, the hulls and tri64 in place.  Frames of the pipelined loops may still read them, on both kernel streams, so
// the update runs between the GI writer pair: after every frame enqueued before it, before every frame after it.
static int check_update(const vrt_tree* t, const char* fn, int max_depth)
{
        if (!t) {
                set_error("%s: null tree handle", fn);
                return VRT_ERR_ARG;
        }
        if (!t->d_tri_in) {
                set_error("%s: handle holds no input triangles (loaded, or made from a blob)", fn);
                return VRT_ERR_STATE;
        }
        int dev = -1;
        if (cudaGetDevice(&dev) != cudaSuccess || dev != t->device) {
                cudaGetLastError();
                set_error("%s: tree lives on device %d but the current device is %d", fn, t->device, dev);
                return VRT_ERR_STATE;
        }
        if (max_depth < 1 || max_depth > (int)VRT_MAX_DEPTH) {
                set_error("%s: max_depth %d out of range [1,%u]", fn, max_depth, VRT_MAX_DEPTH);
                return VRT_ERR_ARG;
        }
        return VRT_OK;
}

static int check_update_triangles(const vrt_tree* t, const char* fn, const float* tri, bool has_nrm, bool nrm_known,
                                  uint32_t num_tris)
{
        if (num_tris != t->hdr.num_tris) {
                set_error("%s: num_tris %u differs from the handle's %u", fn, num_tris, t->hdr.num_tris);
                return VRT_ERR_ARG;
        }
        if (!tri) {
                set_error("%s: null tri_xyz", fn);
                return VRT_ERR_ARG;
        }
        if (nrm_known && has_nrm != (t->d_nrm_in != nullptr)) {
                set_error("%s: tri_nrm must be given exactly when the handle was built with normals", fn);
                return VRT_ERR_ARG;
        }
        return VRT_OK;
}

static int update_triangles(vrt_tree* t, const float* tri, const float* nrm, uint32_t num_tris, int max_depth,
                            bool from_device, const char* fn)
{
        int rc = check_update(t, fn, max_depth);
        if (!rc)
                rc = check_update_triangles(t, fn, tri, nrm != nullptr, true, num_tris);
        if (rc)
                return rc;
        const cudaMemcpyKind kind = from_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        const size_t bytes = (size_t)num_tris * 36;
        rc = gi_writer_begin(t);
        if (!rc && bytes && !cuda_ok(cudaMemcpyAsync(t->d_tri_in, tri, bytes, kind, t->stream), "copy triangles"))
                rc = VRT_ERR_CUDA;
        if (!rc && bytes && nrm && !cuda_ok(cudaMemcpyAsync(t->d_nrm_in, nrm, bytes, kind, t->stream), "copy normals"))
                rc = VRT_ERR_CUDA;
        if (!rc) {
                t->rest_valid = false;  // the new triangles are the rest pose of later transform updates
                rc = build_tree(t, max_depth);  // (synchronises: the caller's arrays are free again on return)
        }
        return gi_writer_end(t, rc);
}

// the table sorted by first_tri; every range non-empty, inside [0, T), disjoint from the others; m and n finite
static int sort_xforms(const vrt_xform* xf, uint32_t num_xf, uint32_t T, const char* fn, std::vector<vrt_xform>* out)
{
        if (!xf || num_xf == 0) {
                set_error("%s: no transforms", fn);
                return VRT_ERR_ARG;
        }
        out->assign(xf, xf + num_xf);
        for (const vrt_xform& x : *out) {
                for (float v : x.m)
                        if (!std::isfinite(v)) {
                                set_error("%s: non-finite matrix entry", fn);
                                return VRT_ERR_ARG;
                        }
                for (float v : x.n)
                        if (!std::isfinite(v)) {
                                set_error("%s: non-finite normal matrix entry", fn);
                                return VRT_ERR_ARG;
                        }
                if (x.num_tris == 0 || (uint64_t)x.first_tri + x.num_tris > T) {
                        set_error("%s: range [%u, +%u) is empty or outside [0, %u)", fn, x.first_tri, x.num_tris, T);
                        return VRT_ERR_ARG;
                }
        }
        std::stable_sort(out->begin(), out->end(),
                         [](const vrt_xform& a, const vrt_xform& b) { return a.first_tri < b.first_tri; });
        for (size_t k = 1; k < out->size(); ++k)
                if ((*out)[k].first_tri < (uint64_t)(*out)[k - 1].first_tri + (*out)[k - 1].num_tris) {
                        set_error("%s: ranges starting at %u and %u overlap", fn, (*out)[k - 1].first_tri,
                                  (*out)[k].first_tri);
                        return VRT_ERR_ARG;
                }
        return VRT_OK;
}

// current pose = rest pose moved by the sorted table, on `stream`; the rest pose is saved from the current one first
// when the inputs were last replaced by a build or a full update
static int apply_xforms(vrt_tree* t, const std::vector<vrt_xform>& xf)
{
        const uint32_t T = t->hdr.num_tris;
        const size_t bytes = (size_t)T * 36;
        if ((!t->d_tri_rest && !cuda_ok(cudaMalloc(&t->d_tri_rest, bytes), "cudaMalloc(rest pose)")) ||
            (t->d_nrm_in && !t->d_nrm_rest && !cuda_ok(cudaMalloc(&t->d_nrm_rest, bytes), "cudaMalloc(rest normals)")))
                return VRT_ERR_NOMEM;
        if (!t->rest_valid) {
                VRT_CUDA(cudaMemcpyAsync(t->d_tri_rest, t->d_tri_in, bytes, cudaMemcpyDeviceToDevice, t->stream));
                if (t->d_nrm_in)
                        VRT_CUDA(cudaMemcpyAsync(t->d_nrm_rest, t->d_nrm_in, bytes, cudaMemcpyDeviceToDevice, t->stream));
                t->rest_valid = true;
        }
        const size_t xb = xf.size() * sizeof(vrt_xform);
        if (t->xf_buf.reserve(xb))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpyAsync(t->xf_buf.p, xf.data(), xb, cudaMemcpyHostToDevice, t->stream));
        k_apply_xforms<<<(T + 255u) / 256u, 256, 0, t->stream>>>(t->d_tri_rest, t->d_nrm_rest, t->xf_buf.as<vrt_xform>(),
                                                                 (uint32_t)xf.size(), T, t->d_tri_in, t->d_nrm_in);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        return VRT_OK;
}

int vrt_update_triangles(vrt_tree* t, const float* tri_xyz, const float* tri_nrm, uint32_t num_tris, int max_depth)
{
        return update_triangles(t, tri_xyz, tri_nrm, num_tris, max_depth, false, "vrt_update_triangles");
}

int vrt_update_triangles_dev(vrt_tree* t, const float* d_tri_xyz, const float* d_tri_nrm, uint32_t num_tris,
                             int max_depth)
{
        return update_triangles(t, d_tri_xyz, d_tri_nrm, num_tris, max_depth, true, "vrt_update_triangles_dev");
}

int vrt_update_xform(vrt_tree* t, const vrt_xform* xf, uint32_t num_xf, int max_depth)
{
        int rc = check_update(t, "vrt_update_xform", max_depth);
        if (rc)
                return rc;
        std::vector<vrt_xform> sorted;
        rc = sort_xforms(xf, num_xf, t->hdr.num_tris, "vrt_update_xform", &sorted);
        if (rc)
                return rc;
        rc = gi_writer_begin(t);
        if (!rc)
                rc = apply_xforms(t, sorted);
        if (!rc)
                rc = build_tree(t, max_depth);
        return gi_writer_end(t, rc);
}

// ---- single-process multi-GPU render (SURVEY.md 8e; replaces render_mt camera.h:41-68 over N devices) -------
// A C / C++ host (main.cc) owns ONE process: vrt_mgpu_create replicates a built octree onto the given devices
// (peer copies of the blob over NVLink), vrt_mgpu_render_async deals the film's 8-row bands round-robin to the
// devices -- each through its own vrt_render_bands_async pipeline, i.e. kernels alternating between two streams and
// the device->host copies of its bands going straight to their final rows of the caller's frame -- and
// vrt_mgpu_sync waits for all of them.  No collective in the data path: the path shards by image rows.
struct vrt_mgpu {
        std::vector<int> devices;
        std::vector<vrt_tree*> trees;  // trees[i] lives on devices[i]; trees[0] is a replica too (the source stays the caller's)
        int band_h = 8;
};

static int set_device_checked(int dev)
{
        VRT_CUDA(cudaSetDevice(dev));
        return VRT_OK;
}

int vrt_mgpu_set_film_format(vrt_mgpu* m, int32_t format)
{
        if (!m) {
                set_error("null handle");
                return VRT_ERR_ARG;
        }
        for (vrt_tree* t : m->trees) {
                const int rc = vrt_set_film_format(t, format);
                if (rc)
                        return rc;
        }
        return VRT_OK;
}

void vrt_mgpu_free(vrt_mgpu* m)
{
        if (!m)
                return;
        int cur = 0;
        cudaGetDevice(&cur);
        for (size_t i = 0; i < m->trees.size(); ++i) {
                cudaSetDevice(m->devices[i]);
                vrt_tree_free(m->trees[i]);
        }
        cudaSetDevice(cur);
        delete m;
}

// the input triangles of `src` (the pose its octree was built from) as the inputs of replica `rep`, whose device is
// current: the rest pose of vrt_mgpu_update_xform, which rebuilds on the first replica
static int copy_inputs(vrt_tree* rep, const vrt_tree* src)
{
        const size_t bytes = (size_t)std::max<uint32_t>(src->hdr.num_tris, 1) * 36;
        if (!cuda_ok(cudaMalloc(&rep->d_tri_in, bytes), "cudaMalloc(tri)") ||
            (src->d_nrm_in && !cuda_ok(cudaMalloc(&rep->d_nrm_in, bytes), "cudaMalloc(nrm)")))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpyPeer(rep->d_tri_in, rep->device, src->d_tri_in, src->device, bytes));
        if (src->d_nrm_in)
                VRT_CUDA(cudaMemcpyPeer(rep->d_nrm_in, rep->device, src->d_nrm_in, src->device, bytes));
        rep->unit_normals = src->unit_normals;
        return VRT_OK;
}

int vrt_mgpu_create(const vrt_tree* tree, int num_devices, const int* devices, vrt_mgpu** out)
{
        int rc = check_tree(tree);
        if (rc)
                return rc;
        if (!out || num_devices < 1) {
                set_error("vrt_mgpu_create: bad argument");
                return VRT_ERR_ARG;
        }
        *out = nullptr;
        int ndev = 0;
        VRT_CUDA(cudaGetDeviceCount(&ndev));
        vrt_mgpu* m = new (std::nothrow) vrt_mgpu();
        if (!m)
                return VRT_ERR_NOMEM;
        for (int i = 0; i < num_devices; ++i) {
                const int d = devices ? devices[i] : i;
                if (d < 0 || d >= ndev) {
                        set_error("vrt_mgpu_create: device %d does not exist (%d visible)", d, ndev);
                        vrt_mgpu_free(m);
                        return VRT_ERR_ARG;
                }
                m->devices.push_back(d);
        }
        const int src_dev = tree->device;
        VRT_CUDA(cudaStreamSynchronize(tree->stream));
        for (int i = 0; i < num_devices && !rc; ++i) {
                const int d = m->devices[i];
                rc = set_device_checked(d);
                if (rc)
                        break;
                vrt_tree* rep = nullptr;
                if (d == src_dev) {
                        rc = vrt_tree_from_blob_dev(tree->blob, tree->hdr.bytes, &rep);
                } else {
                        void* tmp = nullptr;
                        if (cudaMalloc(&tmp, tree->hdr.bytes) != cudaSuccess) {
                                cudaGetLastError();
                                set_error("vrt_mgpu_create: cudaMalloc(%llu) on device %d failed",
                                          (unsigned long long)tree->hdr.bytes, d);
                                rc = VRT_ERR_NOMEM;
                        } else {
                                if (cudaMemcpyPeer(tmp, d, tree->blob, src_dev, tree->hdr.bytes) != cudaSuccess) {
                                        set_error("vrt_mgpu_create: peer copy %d -> %d failed: %s", src_dev, d,
                                                  cudaGetErrorString(cudaGetLastError()));
                                        rc = VRT_ERR_CUDA;
                                } else {
                                        rc = vrt_tree_from_blob_dev(tmp, tree->hdr.bytes, &rep);
                                }
                                cudaFree(tmp);
                        }
                }
                if (!rc && i == 0 && tree->d_tri_in)
                        rc = copy_inputs(rep, tree);
                if (!rc)
                        m->trees.push_back(rep);
                else
                        vrt_tree_free(rep);
        }
        cudaSetDevice(src_dev);
        if (rc) {
                m->devices.resize(m->trees.size());
                vrt_mgpu_free(m);
                return rc;
        }
        *out = m;
        return VRT_OK;
}

int vrt_mgpu_num_devices(const vrt_mgpu* m) { return m ? (int)m->trees.size() : 0; }

// f(i, replica i) for every replica with its device current, up to the first failure; the caller's device is restored
extern "C++" {
namespace {
template <class F>
int mgpu_each(vrt_mgpu* m, F&& f)
{
        if (!m || m->trees.empty()) {
                set_error("null multi-GPU handle");
                return VRT_ERR_ARG;
        }
        int cur = 0;
        VRT_CUDA(cudaGetDevice(&cur));
        int rc = VRT_OK;
        for (int i = 0; i < (int)m->trees.size() && !rc; ++i) {
                rc = set_device_checked(m->devices[i]);
                if (!rc)
                        rc = f(i, m->trees[i]);
        }
        cudaSetDevice(cur);
        return rc;
}
}  // namespace
}  // extern "C++"

// one frame: the 8-row bands dealt round-robin, each replica through its bands_async_common pipeline
static int mgpu_bands_async(vrt_mgpu* m, const vrt_camera* cam, const vrt_shade* sh, const GiArgs* gi,
                            const vrt_gi_aov* aov_full, float* film_rgb_full, OutMode mode)
{
        const int n = m ? (int)m->trees.size() : 0;
        return mgpu_each(m, [&](int i, vrt_tree* t) {
                if (cam && (long)i * m->band_h >= cam->ny)
                        return (int)VRT_OK;  // more devices than bands
                const vrt_bands b = { m->band_h, i, n };
                return bands_async_common(t, cam, sh, gi, aov_full, &b, film_rgb_full, mode);
        });
}

int vrt_mgpu_render_async(vrt_mgpu* m, const vrt_camera* cam, const vrt_shade* sh, float* film_rgb_full)
{
        return mgpu_bands_async(m, cam, sh, nullptr, nullptr, film_rgb_full, OUT_FILM);
}

int vrt_mgpu_sync(vrt_mgpu* m)
{
        if (!m) {
                set_error("null multi-GPU handle");
                return VRT_ERR_ARG;
        }
        int cur = 0;
        VRT_CUDA(cudaGetDevice(&cur));
        int rc = VRT_OK;
        for (size_t i = 0; i < m->trees.size(); ++i) {
                int r2 = set_device_checked(m->devices[i]);
                if (!r2)
                        r2 = vrt_tree_sync(m->trees[i]);
                if (r2 && !rc)
                        rc = r2;
        }
        cudaSetDevice(cur);
        return rc;
}

int vrt_mgpu_render(vrt_mgpu* m, const vrt_camera* cam, const vrt_shade* sh, float* film_rgb_full)
{
        int rc = vrt_mgpu_render_async(m, cam, sh, film_rgb_full);
        const int rs = vrt_mgpu_sync(m);
        return rc ? rc : rs;
}

// ---- GI film on the replicas.  vrt_mgpu_create copies the geometry blob only; materials and the per-node GI state
// are set per replica.  The light pass runs on every replica (the splat accumulates in the sequential loop order, so
// every replica holds the same bits) -- concurrently, since none of the passes waits on the host.
int vrt_mgpu_set_materials(vrt_mgpu* m, const float* tri_uv, const uint32_t* tri_mtl, uint32_t num_mtl,
                           const float* kd, const int32_t* mtl_tex, uint32_t num_tex, const vrt_texture* tex)
{
        return mgpu_each(m, [&](int, vrt_tree* t) {
                return vrt_set_materials(t, tri_uv, tri_mtl, num_mtl, kd, mtl_tex, num_tex, tex);
        });
}

int vrt_mgpu_gi_init(vrt_mgpu* m)
{
        return mgpu_each(m, [](int, vrt_tree* t) { return vrt_gi_init(t); });
}

int vrt_mgpu_gi_splat_camera(vrt_mgpu* m, const vrt_camera* light_cam, const float kd[3])
{
        return mgpu_each(m, [&](int, vrt_tree* t) { return vrt_gi_splat_camera(t, light_cam, kd); });
}

int vrt_mgpu_gi_filter(vrt_mgpu* m)
{
        return mgpu_each(m, [](int, vrt_tree* t) { return vrt_gi_filter(t); });
}

int vrt_mgpu_gi_render_async(vrt_mgpu* m, const vrt_camera* cam, const float kd[3], float res, float* film_rgb_full)
{
        if (const int rc = check_gi_res(res))
                return rc;
        if (!kd) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        const GiArgs ga = { { kd[0], kd[1], kd[2] }, res };
        return mgpu_bands_async(m, cam, nullptr, &ga, nullptr, film_rgb_full, OUT_GI_FILM);
}

int vrt_mgpu_gi_render(vrt_mgpu* m, const vrt_camera* cam, const float kd[3], float res, float* film_rgb_full)
{
        if (const int rc = check_gi_res(res))
                return rc;
        int rc = vrt_mgpu_gi_render_async(m, cam, kd, res, film_rgb_full);
        const int rs = vrt_mgpu_sync(m);
        return rc ? rc : rs;
}

int vrt_mgpu_gi_render_aov_async(vrt_mgpu* m, const vrt_camera* cam, const float kd[3], float res,
                                 float* film_full_or_null, const vrt_gi_aov* aov_full)
{
        if (const int rc = check_gi_res(res))
                return rc;
        const int rc = check_gi_aov_request(kd, aov_full);
        if (rc)
                return rc;
        const GiArgs ga = { { kd[0], kd[1], kd[2] }, res };
        return mgpu_bands_async(m, cam, nullptr, &ga, aov_full, film_full_or_null, OUT_GI_AOV);
}

int vrt_mgpu_gi_render_aov(vrt_mgpu* m, const vrt_camera* cam, const float kd[3], float res, float* film_full_or_null,
                           const vrt_gi_aov* aov_full)
{
        if (const int rc = check_gi_res(res))
                return rc;
        int rc = vrt_mgpu_gi_render_aov_async(m, cam, kd, res, film_full_or_null, aov_full);
        const int rs = vrt_mgpu_sync(m);
        return rc ? rc : rs;
}

// ---- animated geometry on the replicas: the first replica rebuilds (the build synchronises the host at every level,
// so builds on the others would run one after another anyway), then every other replica takes a copy of its blob --
// the path of vrt_mgpu_create: peer copy, bind, compute_hulls -- between its own GI writer pair.
static int replica_take_blob(vrt_tree* t, const vrt_tree* src)
{
        const uint64_t b = src->hdr.bytes;
        VRT_CUDA(cudaStreamSynchronize(t->stream));  // every frame that reads the old blob has finished
        if (t->blob_bytes < b) {
                cudaFree(t->blob);
                t->blob = nullptr;
                if (cudaMalloc(&t->blob, b) != cudaSuccess) {
                        cudaGetLastError();
                        set_error("cudaMalloc(%llu) for a replica's blob failed", (unsigned long long)b);
                        return VRT_ERR_NOMEM;
                }
                t->blob_bytes = b;
        }
        VRT_CUDA(cudaMemcpyPeerAsync(t->blob, t->device, src->blob, src->device, b, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        t->hdr = src->hdr;
        tree_bind_views(t);
        return compute_hulls(t);
}

static int mgpu_replicate(vrt_mgpu* m)
{
        const vrt_tree* src = m->trees[0];
        return mgpu_each(m, [&](int i, vrt_tree* t) {
                if (i == 0)
                        return (int)VRT_OK;
                int rc = gi_writer_begin(t);
                if (!rc)
                        rc = replica_take_blob(t, src);
                return gi_writer_end(t, rc);
        });
}

int vrt_mgpu_update_triangles(vrt_mgpu* m, const float* tri_xyz, const float* tri_nrm, uint32_t num_tris, int max_depth)
{
        const char* fn = "vrt_mgpu_update_triangles";
        if (!m || m->trees.empty()) {
                set_error("null multi-GPU handle");
                return VRT_ERR_ARG;
        }
        vrt_tree* t0 = m->trees[0];
        if (max_depth < 1 || max_depth > (int)VRT_MAX_DEPTH) {
                set_error("%s: max_depth %d out of range [1,%u]", fn, max_depth, VRT_MAX_DEPTH);
                return VRT_ERR_ARG;
        }
        // a replica set made from a tree without input triangles takes its first inputs here, normals or not
        int rc = check_update_triangles(t0, fn, tri_xyz, tri_nrm != nullptr, t0->d_tri_in != nullptr, num_tris);
        if (rc)
                return rc;
        rc = mgpu_each(m, [&](int i, vrt_tree* t) {
                if (i)
                        return (int)VRT_OK;
                const size_t bytes = (size_t)std::max<uint32_t>(num_tris, 1) * 36;
                if (!t->d_tri_in && (!cuda_ok(cudaMalloc(&t->d_tri_in, bytes), "cudaMalloc(tri)") ||
                                     (tri_nrm && !cuda_ok(cudaMalloc(&t->d_nrm_in, bytes), "cudaMalloc(nrm)")))) {
                        cudaFree(t->d_tri_in);
                        t->d_tri_in = nullptr;
                        return (int)VRT_ERR_NOMEM;
                }
                return update_triangles(t, tri_xyz, tri_nrm, num_tris, max_depth, false, fn);
        });
        return rc ? rc : mgpu_replicate(m);
}

int vrt_mgpu_update_xform(vrt_mgpu* m, const vrt_xform* xf, uint32_t num_xf, int max_depth)
{
        if (!m || m->trees.empty()) {
                set_error("null multi-GPU handle");
                return VRT_ERR_ARG;
        }
        const int rc = mgpu_each(m, [&](int i, vrt_tree* t) { return i ? (int)VRT_OK : vrt_update_xform(t, xf, num_xf, max_depth); });
        return rc ? rc : mgpu_replicate(m);
}

double vrt_mgpu_mean_kernel_ms(vrt_mgpu* m, int index, int last_n)
{
        if (!m || index < 0 || index >= (int)m->trees.size())
                return 0;
        double ms = 0;
        int cur = 0;
        if (cudaGetDevice(&cur) != cudaSuccess) {
                cudaGetLastError();
                return 0;
        }
        if (!set_device_checked(m->devices[index]))
                ms = vrt_mean_kernel_ms(m->trees[index], last_n);
        cudaSetDevice(cur);
        return ms;
}

int vrt_trace_bands16_dev(const vrt_tree* t, const vrt_camera* cam, const vrt_bands* b, vrt_hit16* d_out)
{
        return bands_common(t, cam, nullptr, b, d_out, OUT_HIT16);
}

double vrt_last_kernel_ms(const vrt_tree* t)
{
        double ms = 0;
        if (t)
                trace_ms_mean(t, 1, &ms);
        return ms;
}

double vrt_mean_kernel_ms(const vrt_tree* t, int last_n)
{
        double ms = 0;
        if (t)
                trace_ms_mean(t, last_n, &ms);
        return ms;
}

// ---- GI rows (SURVEY.md 8f) -------------------------------------------------------
int vrt_gi_init(vrt_tree* t)
{
        int rc = check_tree(t);
        if (rc || (rc = gi_writer_begin(t)))
                return rc;
        return gi_writer_end(t, gi_init(t));
}

int vrt_gi_splat_camera(vrt_tree* t, const vrt_camera* light_cam, const float kd[3])
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        if (!light_cam || !kd) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        rc = check_camera(light_cam, 0, 0, light_cam->nx, light_cam->ny);
        if (rc || (rc = gi_writer_begin(t)))
                return rc;
        return gi_writer_end(t, gi_splat_camera(t, light_cam, kd));
}

int vrt_gi_filter(vrt_tree* t)
{
        int rc = check_tree(t);
        if (rc || (rc = gi_writer_begin(t)))
                return rc;
        return gi_writer_end(t, gi_filter(t));
}

int vrt_gi_get_level(const vrt_tree* t, int level, float* coverage, float* illum18)
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        if (!t->dev.gi || level < 0 || level > t->hdr.max_depth - 1) {
                set_error("vrt_gi_get_level: no GI state or level out of range");
                return VRT_ERR_ARG;
        }
        const uint64_t first = t->hdr.level_offset[level], n = t->hdr.level_offset[level + 1] - first;
        if (level == t->hdr.max_depth - 1 && n != t->hdr.num_leaves) {
                set_error("inconsistent level table");
                return VRT_ERR_ARG;
        }
        std::vector<float> host(n * kGiStride);
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        if (n)
                VRT_CUDA(cudaMemcpy(host.data(), t->dev.gi + first * kGiStride, n * kGiStride * sizeof(float), cudaMemcpyDeviceToHost));
        for (uint64_t i = 0; i < n; ++i) {
                if (coverage)
                        coverage[i] = host[kGiStride * i + kGiCoverage];
                if (illum18)
                        for (int f = 0; f < 18; ++f)
                                illum18[18 * i + f] = host[kGiStride * i + 4 * (f / 3) + f % 3];
        }
        return VRT_OK;
}

int vrt_gi_cone_trace(const vrt_tree* tc, const float* pos, const float* nrm, uint64_t n, float res, float* out_rgb)
{
        if (const int rc = check_gi_res(res))
                return rc;
        int rc = check_tree(tc);
        if (rc)
                return rc;
        if (n && (!pos || !nrm || !out_rgb)) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        if (n == 0)
                return VRT_OK;
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        if (t->io_in.reserve(n * 24) || t->io_out.reserve(n * 12))
                return VRT_ERR_NOMEM;
        float* d_pos = t->io_in.as<float>();
        float* d_nrm = d_pos + 3 * n;
        VRT_CUDA(cudaMemcpyAsync(d_pos, pos, n * 12, cudaMemcpyHostToDevice, t->stream));
        VRT_CUDA(cudaMemcpyAsync(d_nrm, nrm, n * 12, cudaMemcpyHostToDevice, t->stream));
        rc = gi_cone_points(t, d_pos, d_nrm, n, res, t->io_out.as<float>());
        if (rc)
                return rc;
        VRT_CUDA(cudaMemcpyAsync(out_rgb, t->io_out.p, n * 12, cudaMemcpyDeviceToHost, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        return VRT_OK;
}

// Materials: per-vertex texture coordinates, a material id per triangle, per material a diffuse colour and
// an optional texture (the untextured / textured branches of Triangle::get_albedo).  Host pointers.
int vrt_set_materials(vrt_tree* t, const float* tri_uv, const uint32_t* tri_mtl, uint32_t num_mtl, const float* kd,
                      const int32_t* mtl_tex, uint32_t num_tex, const vrt_texture* tex)
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        const uint64_t T = t->hdr.num_tris;
        if (!tri_uv || !tri_mtl || !num_mtl || !kd || !mtl_tex || (num_tex && !tex)) {
                set_error("vrt_set_materials: null argument");
                return VRT_ERR_ARG;
        }
        for (uint64_t i = 0; i < T; ++i)
                if (tri_mtl[i] >= num_mtl) {
                        set_error("tri_mtl[%llu]=%u out of range", (unsigned long long)i, tri_mtl[i]);
                        return VRT_ERR_ARG;
                }
        std::vector<float> hkd(4 * (size_t)num_mtl);
        for (uint32_t m = 0; m < num_mtl; ++m) {
                if (mtl_tex[m] >= (int32_t)num_tex) {
                        set_error("mtl_tex[%u]=%d out of range", m, mtl_tex[m]);
                        return VRT_ERR_ARG;
                }
                const int32_t tx = mtl_tex[m] < 0 ? -1 : mtl_tex[m];
                memcpy(&hkd[4 * m], kd + 3 * m, 12);
                memcpy(&hkd[4 * m + 3], &tx, 4);
        }
        std::vector<int32_t> htex(4 * (size_t)std::max<uint32_t>(num_tex, 1));
        uint64_t texel_bytes = 0;
        for (uint32_t i = 0; i < num_tex; ++i) {
                if (tex[i].width < 1 || tex[i].height < 1 || tex[i].channels < 1 || tex[i].channels > 4 || !tex[i].data) {
                        set_error("texture %u: bad dimensions or null data", i);
                        return VRT_ERR_ARG;
                }
                if (texel_bytes > 0xfff00000ull) {
                        set_error("textures exceed 4 GB");
                        return VRT_ERR_CAPACITY;
                }
                htex[4 * i] = (int32_t)(uint32_t)texel_bytes;
                htex[4 * i + 1] = tex[i].width;
                htex[4 * i + 2] = tex[i].height;
                htex[4 * i + 3] = tex[i].channels;
                texel_bytes += align256((uint64_t)tex[i].width * tex[i].height * tex[i].channels);
        }
        const uint64_t o_uv = 0, o_tri = align256(o_uv + std::max<uint64_t>(T, 1) * 24);
        const uint64_t o_kd = align256(o_tri + std::max<uint64_t>(T, 1) * 4), o_tex = align256(o_kd + (uint64_t)num_mtl * 16);
        const uint64_t o_px = align256(o_tex + (uint64_t)std::max<uint32_t>(num_tex, 1) * 16);
        rc = gi_writer_begin(t);
        if (rc)
                return rc;
        if (t->mat_buf.reserve(o_px + std::max<uint64_t>(texel_bytes, 256)))
                return gi_writer_end(t, VRT_ERR_NOMEM);
        char* base = static_cast<char*>(t->mat_buf.p);
        // the copies are ordered on the handle's stream (behind every frame that may still read the old materials,
        // gi_writer_begin) and complete before the call returns: the host arrays are borrowed for the call only
        if (T) {
                VRT_CUDA(cudaMemcpyAsync(base + o_uv, tri_uv, T * 24, cudaMemcpyHostToDevice, t->stream));
                VRT_CUDA(cudaMemcpyAsync(base + o_tri, tri_mtl, T * 4, cudaMemcpyHostToDevice, t->stream));
        }
        VRT_CUDA(cudaMemcpyAsync(base + o_kd, hkd.data(), (size_t)num_mtl * 16, cudaMemcpyHostToDevice, t->stream));
        VRT_CUDA(cudaMemcpyAsync(base + o_tex, htex.data(), htex.size() * 4, cudaMemcpyHostToDevice, t->stream));
        for (uint32_t i = 0; i < num_tex; ++i)
                VRT_CUDA(cudaMemcpyAsync(base + o_px + (uint32_t)htex[4 * i], tex[i].data,
                                         (size_t)tex[i].width * tex[i].height * tex[i].channels, cudaMemcpyHostToDevice,
                                         t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        rc = gi_writer_end(t, VRT_OK);
        if (rc)
                return rc;
        t->dev.mat_uv = reinterpret_cast<const float2*>(base + o_uv);
        t->dev.mat_tri = reinterpret_cast<const uint32_t*>(base + o_tri);
        t->dev.mat_kd = reinterpret_cast<const float4*>(base + o_kd);
        t->dev.mat_tex = reinterpret_cast<const int4*>(base + o_tex);
        t->dev.mat_texels = reinterpret_cast<const uint8_t*>(base + o_px);
        return VRT_OK;
}

// Triangle::get_albedo(ISect{hit = pos[i]}) of triangle tri[i]; host pointers.  kd_default is the colour of
// a tree without materials.
int vrt_albedo(const vrt_tree* tc, const uint32_t* tri, const float* pos, uint64_t n, const float kd_default[3],
               float* out_rgb)
{
        int rc = check_tree(tc);
        if (rc)
                return rc;
        if (n && (!tri || !pos || !out_rgb || !kd_default)) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        if (n == 0)
                return VRT_OK;
        for (uint64_t i = 0; i < n; ++i)
                if (tri[i] >= tc->hdr.num_tris) {
                        set_error("tri[%llu]=%u out of range", (unsigned long long)i, tri[i]);
                        return VRT_ERR_ARG;
                }
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        if (t->io_in.reserve(n * 16) || t->io_out.reserve(n * 12))
                return VRT_ERR_NOMEM;
        float* d_pos = t->io_in.as<float>();
        uint32_t* d_tri = reinterpret_cast<uint32_t*>(d_pos + 3 * n);
        VRT_CUDA(cudaMemcpyAsync(d_pos, pos, n * 12, cudaMemcpyHostToDevice, t->stream));
        VRT_CUDA(cudaMemcpyAsync(d_tri, tri, n * 4, cudaMemcpyHostToDevice, t->stream));
        rc = gi_albedo_points(t, d_tri, d_pos, n, kd_default, t->io_out.as<float>());
        if (rc)
                return rc;
        VRT_CUDA(cudaMemcpyAsync(out_rgb, t->io_out.p, n * 12, cudaMemcpyDeviceToHost, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        return VRT_OK;
}

static int gi_render_common(const vrt_tree* tc, const vrt_camera* cam, const float kd[3], float res, int x0, int y0,
                            int x1, int y1, float* film, bool dev)
{
        if (const int rc = check_gi_res(res))
                return rc;
        int rc = check_tree(tc);
        if (rc)
                return rc;
        if (!cam || !kd || !film) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        if (!tc->dev.gi) {
                set_error("vrt_gi_init has not been called on this tree");
                return VRT_ERR_ARG;
        }
        GiArgs ga = { { kd[0], kd[1], kd[2] }, res };
        rc = gi_step_table(tc, res, &ga.steps);
        if (rc)
                return rc;
        return trace_camera_common(tc, cam, nullptr, x0, y0, x1, y1, film, OUT_GI_FILM, dev, &ga);
}

int vrt_gi_render_camera(const vrt_tree* t, const vrt_camera* cam, const float kd[3], float res, int x0, int y0, int x1,
                         int y1, float* film_rgb)
{
        return gi_render_common(t, cam, kd, res, x0, y0, x1, y1, film_rgb, false);
}

int vrt_gi_render_camera_dev(const vrt_tree* t, const vrt_camera* cam, const float kd[3], float res, int x0, int y0,
                             int x1, int y1, float* d_film_rgb)
{
        return gi_render_common(t, cam, kd, res, x0, y0, x1, y1, d_film_rgb, true);
}

// The GI film plus its planes (vrt_gi_aov) in one OUT_GI_AOV launch; host pointers go through one device buffer.
static int gi_render_aov_common(const vrt_tree* tc, const vrt_camera* cam, const float kd[3], float res, int x0,
                                int y0, int x1, int y1, float* film, const vrt_gi_aov* aov, bool dev)
{
        if (const int rc = check_gi_res(res))
                return rc;
        int rc = check_tree(tc);
        if (rc)
                return rc;
        if (!cam || !kd || !aov) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        float* const planes[4] = { aov->albedo, aov->direct, aov->indirect, aov->normal };
        if (!planes[0] && !planes[1] && !planes[2] && !planes[3] && !aov->hits) {
                set_error("vrt_gi_render_aov: every plane is NULL (the film alone is vrt_gi_render_camera)");
                return VRT_ERR_ARG;
        }
        if (!tc->dev.gi) {
                set_error("vrt_gi_init has not been called on this tree");
                return VRT_ERR_ARG;
        }
        rc = check_camera(cam, x0, y0, x1, y1);
        if (rc)
                return rc;
        const uint64_t npix = (uint64_t)(x1 - x0) * (y1 - y0);
        if (!npix)
                return VRT_OK;
        GiArgs ga = { { kd[0], kd[1], kd[2] }, res };
        rc = gi_step_table(tc, res, &ga.steps);
        if (rc)
                return rc;
        if (dev)
                return launch_trace_camera(tc, cam, nullptr, x0, y0, x1, y1, film, OUT_GI_AOV, 0, 0, nullptr, 0, &ga, aov);
        // one device buffer: film, the four float planes, the hit records (each part 256-byte aligned)
        auto up = [](uint64_t b) { return (b + 255) & ~255ull; };
        const uint64_t film_bytes = npix * (uint64_t)vrt_film_pixel_bytes(tc->film_fmt), plane_bytes = npix * 12,
                       hit_bytes = npix * cam->spp * sizeof(vrt_hit16);
        uint64_t off[6] = { 0 };
        off[1] = off[0] + (film ? up(film_bytes) : 0);
        for (int i = 0; i < 4; ++i)
                off[i + 2] = off[i + 1] + (planes[i] ? up(plane_bytes) : 0);
        const uint64_t total = off[5] + (aov->hits ? hit_bytes : 0);
        vrt_tree* t = const_cast<vrt_tree*>(tc);
        if (t->io_out.reserve(total))
                return VRT_ERR_NOMEM;
        char* const base = static_cast<char*>(t->io_out.p);
        vrt_gi_aov d_aov = {};
        float** const d_planes[4] = { &d_aov.albedo, &d_aov.direct, &d_aov.indirect, &d_aov.normal };
        for (int i = 0; i < 4; ++i)
                if (planes[i])
                        *d_planes[i] = reinterpret_cast<float*>(base + off[i + 1]);
        if (aov->hits)
                d_aov.hits = reinterpret_cast<vrt_hit16*>(base + off[5]);
        rc = launch_trace_camera(t, cam, nullptr, x0, y0, x1, y1, film ? base : nullptr, OUT_GI_AOV, 0, 0, nullptr, 0,
                                 &ga, &d_aov);
        if (rc)
                return rc;
        if (film)
                VRT_CUDA(cudaMemcpyAsync(film, base, film_bytes, cudaMemcpyDeviceToHost, t->stream));
        for (int i = 0; i < 4; ++i)
                if (planes[i])
                        VRT_CUDA(cudaMemcpyAsync(planes[i], base + off[i + 1], plane_bytes, cudaMemcpyDeviceToHost,
                                                 t->stream));
        if (aov->hits)
                VRT_CUDA(cudaMemcpyAsync(aov->hits, base + off[5], hit_bytes, cudaMemcpyDeviceToHost, t->stream));
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        return VRT_OK;
}

int vrt_gi_render_aov(const vrt_tree* t, const vrt_camera* cam, const float kd[3], float res, int x0, int y0, int x1,
                      int y1, float* film_or_null, const vrt_gi_aov* aov)
{
        return gi_render_aov_common(t, cam, kd, res, x0, y0, x1, y1, film_or_null, aov, false);
}

int vrt_gi_render_aov_dev(const vrt_tree* t, const vrt_camera* cam, const float kd[3], float res, int x0, int y0,
                          int x1, int y1, float* d_film_or_null, const vrt_gi_aov* d_aov)
{
        return gi_render_aov_common(t, cam, kd, res, x0, y0, x1, y1, d_film_or_null, d_aov, true);
}

int vrt_debug_param_check(uint64_t out[2])
{
        if (!out) {
                set_error("null out");
                return VRT_ERR_ARG;
        }
        unsigned long long v[2] = { 0, 0 };
        int rc = param_check_counts(v);
        out[0] = v[0];
        out[1] = v[1];
        return rc;
}

int vrt_debug_hull_stats(uint64_t out80[80])
{
        unsigned long long v[80];
        int rc = hull_stats(v);
        for (int i = 0; i < 80; ++i)
                out80[i] = v[i];
        return rc;
}

int vrt_debug_set_hull(vrt_tree* t, int on)
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        t->dev.rec_mask = on ? 0xffffu : 0x00ffu;
        return VRT_OK;
}

int vrt_debug_pair_total(const uint32_t* block_counts, uint64_t n, uint64_t* total)
{
        if ((!block_counts && n) || !total) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        vrt_tree* t = nullptr;
        int rc = tree_alloc(&t);
        if (rc)
                return rc;
        DevBuf d;
        rc = d.alloc(n * 4);
        if (!rc && n && cudaMemcpy(d.p, block_counts, n * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
                cudaGetLastError();
                rc = VRT_ERR_CUDA;
        }
        if (!rc)
                rc = sum_u32_as_u64(t, static_cast<const uint32_t*>(d.p), n, total);
        vrt_tree_free(t);
        return rc;
}

uint64_t vrt_debug_general_order_calls(void)
{
        unsigned long long n = 0;
        general_order_calls(&n);
        return n;
}

int vrt_tree_sync(const vrt_tree* t)
{
        if (!t) {
                set_error("null tree handle");
                return VRT_ERR_ARG;
        }
        VRT_CUDA(cudaStreamSynchronize(t->stream));
        // the async frame loops also run kernels on alt_stream and film copies on copy_stream: after this
        // call the films of every enqueued frame are in host memory (include/vrt.h)
        if (t->alt_stream)
                VRT_CUDA(cudaStreamSynchronize(t->alt_stream));
        if (t->copy_stream)
                VRT_CUDA(cudaStreamSynchronize(t->copy_stream));
        // the next async frame starts a new sequence (its stream is ordered behind the handle's stream again)
        const_cast<vrt_tree*>(t)->n_async_frames = 0;
        return VRT_OK;
}

static int frame_common(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, const vrt_bands* b,
                        vrt_hit16* d_hits, float* d_film_rgb, int film_full)
{
        int rc = check_tree(t);
        if (rc)
                return rc;
        rc = check_camera(cam, 0, 0, cam ? cam->nx : 0, cam ? cam->ny : 0);
        if (rc)
                return rc;
        const int rows = vrt_band_rows(cam, b);
        if (rows < 0)
                return rows;
        if (rows == 0)
                return VRT_OK;
        if (!d_hits || !d_film_rgb || !sh) {
                set_error("null out/shade pointer");
                return VRT_ERR_ARG;
        }
        const int y0 = b->band_first * b->band_h;
        return launch_trace_camera(t, cam, sh, 0, y0, cam->nx, y0 + rows, d_hits, OUT_HIT16_FILM, b->band_h,
                                   b->band_stride * b->band_h, d_film_rgb, film_full);
}

int vrt_frame_bands_dev(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, const vrt_bands* b,
                        vrt_hit16* d_hits, float* d_film_rgb)
{
        return frame_common(t, cam, sh, b, d_hits, d_film_rgb, 0);
}

int vrt_frame_bands_peer_dev(const vrt_tree* t, const vrt_camera* cam, const vrt_shade* sh, const vrt_bands* b,
                             vrt_hit16* d_hits, float* d_frame_rgb)
{
        return frame_common(t, cam, sh, b, d_hits, d_frame_rgb, 1);
}

int vrt_dev_alloc(uint64_t bytes, void** d_ptr)
{
        if (!d_ptr || !bytes) {
                set_error("vrt_dev_alloc: bad argument");
                return VRT_ERR_ARG;
        }
        if (cudaMalloc(d_ptr, bytes) != cudaSuccess) {
                cudaGetLastError();
                set_error("cudaMalloc(%llu) failed", (unsigned long long)bytes);
                return VRT_ERR_NOMEM;
        }
        return VRT_OK;
}

int vrt_dev_free(void* d_ptr)
{
        VRT_CUDA(cudaFree(d_ptr));
        return VRT_OK;
}

int vrt_host_register(void* ptr, uint64_t bytes)
{
        if (!ptr || !bytes) {
                set_error("vrt_host_register: bad argument");
                return VRT_ERR_ARG;
        }
        if (cudaHostRegister(ptr, bytes, cudaHostRegisterPortable) != cudaSuccess) {
                cudaGetLastError();
                set_error("cudaHostRegister(%llu bytes) failed", (unsigned long long)bytes);
                return VRT_ERR_CUDA;
        }
        return VRT_OK;
}

int vrt_host_unregister(void* ptr)
{
        VRT_CUDA(cudaHostUnregister(ptr));
        return VRT_OK;
}

int vrt_ipc_export(const void* d_ptr, uint8_t handle[64])
{
        static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle is 64 bytes");
        if (!d_ptr || !handle) {
                set_error("vrt_ipc_export: null argument");
                return VRT_ERR_ARG;
        }
        cudaIpcMemHandle_t h;
        VRT_CUDA(cudaIpcGetMemHandle(&h, const_cast<void*>(d_ptr)));
        memcpy(handle, &h, 64);
        return VRT_OK;
}

int vrt_ipc_open(const uint8_t handle[64], void** d_ptr)
{
        if (!d_ptr || !handle) {
                set_error("vrt_ipc_open: null argument");
                return VRT_ERR_ARG;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, handle, 64);
        VRT_CUDA(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
        return VRT_OK;
}

int vrt_ipc_close(void* d_ptr)
{
        VRT_CUDA(cudaIpcCloseMemHandle(d_ptr));
        return VRT_OK;
}

// ---- predicates ---------------------------------------------------------------
int vrt_tribox_batch(const float* centers, const float* halves, const float* tris, uint64_t n, uint8_t* out)
{
        int rc = need_device();
        if (rc || !n)
                return rc;
        if (!centers || !halves || !tris || !out) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        DevBuf c, h, t, o;
        if (c.alloc(n * 12) || h.alloc(n * 12) || t.alloc(n * 36) || o.alloc(n))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpy(c.p, centers, n * 12, cudaMemcpyHostToDevice));
        VRT_CUDA(cudaMemcpy(h.p, halves, n * 12, cudaMemcpyHostToDevice));
        VRT_CUDA(cudaMemcpy(t.p, tris, n * 36, cudaMemcpyHostToDevice));
        k_tribox<<<(unsigned)((n + 255) / 256), 256>>>((float*)c.p, (float*)h.p, (float*)t.p, n, (uint8_t*)o.p);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        VRT_CUDA(cudaMemcpy(out, o.p, n, cudaMemcpyDeviceToHost));
        return VRT_OK;
}

int vrt_tri_overlap_aabb_batch(const float* aabbs, const float* tris, uint64_t n, uint8_t* out)
{
        int rc = need_device();
        if (rc || !n)
                return rc;
        if (!aabbs || !tris || !out) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        DevBuf b, t, o;
        if (b.alloc(n * 24) || t.alloc(n * 36) || o.alloc(n))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpy(b.p, aabbs, n * 24, cudaMemcpyHostToDevice));
        VRT_CUDA(cudaMemcpy(t.p, tris, n * 36, cudaMemcpyHostToDevice));
        k_tri_aabb<<<(unsigned)((n + 255) / 256), 256>>>((float*)b.p, (float*)t.p, n, (uint8_t*)o.p);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        VRT_CUDA(cudaMemcpy(out, o.p, n, cudaMemcpyDeviceToHost));
        return VRT_OK;
}

int vrt_raytri_batch(const double* in, uint64_t n, uint8_t* result, double* tuv)
{
        int rc = need_device();
        if (rc || !n)
                return rc;
        if (!in || !result || !tuv) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        DevBuf i, r, o;
        if (i.alloc(n * 120) || r.alloc(n) || o.alloc(n * 24))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpy(i.p, in, n * 120, cudaMemcpyHostToDevice));
        k_raytri<<<(unsigned)((n + 255) / 256), 256>>>((double*)i.p, n, (uint8_t*)r.p, (double*)o.p);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        VRT_CUDA(cudaMemcpy(result, r.p, n, cudaMemcpyDeviceToHost));
        VRT_CUDA(cudaMemcpy(tuv, o.p, n * 24, cudaMemcpyDeviceToHost));
        return VRT_OK;
}

int vrt_aabb_isect_batch(const float* aabbs, const vrt_ray* rays, uint64_t n, uint8_t* out)
{
        int rc = need_device();
        if (rc || !n)
                return rc;
        if (!aabbs || !rays || !out) {
                set_error("null argument");
                return VRT_ERR_ARG;
        }
        DevBuf b, r, o;
        if (b.alloc(n * 24) || r.alloc(n * 32) || o.alloc(n))
                return VRT_ERR_NOMEM;
        VRT_CUDA(cudaMemcpy(b.p, aabbs, n * 24, cudaMemcpyHostToDevice));
        VRT_CUDA(cudaMemcpy(r.p, rays, n * 32, cudaMemcpyHostToDevice));
        k_aabb_isect<<<(unsigned)((n + 255) / 256), 256>>>((float*)b.p, (vrt_ray*)r.p, n, (uint8_t*)o.p);
        count_launch();
        VRT_CUDA(cudaGetLastError());
        VRT_CUDA(cudaMemcpy(out, o.p, n, cudaMemcpyDeviceToHost));
        return VRT_OK;
}

}  // extern "C"
