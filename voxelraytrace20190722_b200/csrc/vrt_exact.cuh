// vrt_exact.cuh -- bit-exact device restatements of the reference's scalar
// arithmetic on the hot path.  Everything here must evaluate exactly like the
// reference compiled for x86-64 WITHOUT fused multiply-add
// (VoxelRayTrace20190722.vcxproj:91-120: MSVC /O2 /fp:precise, no /arch), so
//   * every multiply and add is a separately rounded IEEE-754 operation: we use
//     the __f*_rn / __d*_rn intrinsics, which nvcc never contracts into FMA (the
//     translation units are ALSO compiled with -fmad=false as a second guard);
//   * division and sqrt are the IEEE-correct variants (__fdiv_rn, __fsqrt_rn);
//   * denormals are kept (no -ftz), min/max follow std::min/std::max, and
//     first-extremum tie rules follow std::min_element/std::max_element.
// Reference file:line citations are relative to VoxelRayTrace20190722/.
#pragma once

#include <cfloat>
#include <cstdint>
#include <cuda_runtime.h>

namespace vrt {

__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fdiv(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }

// std::min(a,b) = (b<a)?b:a ; std::max(a,b) = (a<b)?b:a  (differs from fminf/fmaxf
// only for NaN operands and for the sign of equal zeros).
__device__ __forceinline__ float std_min(float a, float b) { return (b < a) ? b : a; }
__device__ __forceinline__ float std_max(float a, float b) { return (a < b) ? b : a; }

// jql::dot for Vec3 (graphics_math.h:532-549): value_sum starts at 0 and adds
// the element products left to right.
__device__ __forceinline__ float dot3(float ax, float ay, float az, float bx, float by, float bz)
{
        float s = fadd(0.f, fmul(ax, bx));
        s = fadd(s, fmul(ay, by));
        s = fadd(s, fmul(az, bz));
        return s;
}

// jql::normalize (graphics_math.h:576-586): v / sqrtf(dot(v,v)), true division.
__device__ __forceinline__ void normalize3(float& x, float& y, float& z)
{
        float l = __fsqrt_rn(dot3(x, y, z, x, y, z));
        x = fdiv(x, l);
        y = fdiv(y, l);
        z = fdiv(z, l);
}

// jql::clamp (graphics_math.h:905-909)
__device__ __forceinline__ float clampf(float s, float lo, float hi)
{
        return s > hi ? hi : (s < lo ? lo : s);
}

// ---------------------------------------------------------------------------
// triBoxOverlap (tribox2.cc:112-186) incl. planeBoxOverlap (tribox2.cc:42-63).
// c = box centre, h = box half size, v* = triangle vertices.
// The reference evaluates the 13 axes in a fixed order and returns at the first
// separating one; the result is the conjunction of 13 independent predicates,
// so evaluating them cheapest-and-most-selective first (3 box axes, the plane,
// then the 9 edge axes) does not change it.
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool axis_sep(float pa, float pb, float rad)
{
        // if(pa<pb){min=pa;max=pb;}else{min=pb;max=pa;} if(min>rad||max<-rad) return 0;
        float mn = (pa < pb) ? pa : pb;
        float mx = (pa < pb) ? pb : pa;
        return (mn > rad) || (mx < -rad);
}

__device__ __forceinline__ bool tribox_overlap(const float c[3], const float h[3],
                                               const float t0[3], const float t1[3],
                                               const float t2[3])
{
        float v0[3], v1[3], v2[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                v0[k] = fsub(t0[k], c[k]);
                v1[k] = fsub(t1[k], c[k]);
                v2[k] = fsub(t2[k], c[k]);
        }
        // box axes (tribox2.cc:166-176), strict inequalities
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                float mn = v0[k], mx = v0[k];
                if (v1[k] < mn) mn = v1[k];
                if (v1[k] > mx) mx = v1[k];
                if (v2[k] < mn) mn = v2[k];
                if (v2[k] > mx) mx = v2[k];
                if (mn > h[k] || mx < -h[k])
                        return false;
        }
        float e0[3], e1[3], e2[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                e0[k] = fsub(v1[k], v0[k]);
                e1[k] = fsub(v2[k], v1[k]);
                e2[k] = fsub(v0[k], v2[k]);
        }
        // plane (tribox2.cc:181-183 + 42-63)
        float n[3];
        n[0] = fsub(fmul(e0[1], e1[2]), fmul(e0[2], e1[1]));
        n[1] = fsub(fmul(e0[2], e1[0]), fmul(e0[0], e1[2]));
        n[2] = fsub(fmul(e0[0], e1[1]), fmul(e0[1], e1[0]));
        float d = -fadd(fadd(fmul(n[0], v0[0]), fmul(n[1], v0[1])), fmul(n[2], v0[2]));
        float lo[3], hi[3];
#pragma unroll
        for (int q = 0; q < 3; ++q) {
                if (n[q] > 0.0f) {
                        lo[q] = -h[q];
                        hi[q] = h[q];
                } else {
                        lo[q] = h[q];
                        hi[q] = -h[q];
                }
        }
        float dmin = fadd(fadd(fadd(fmul(n[0], lo[0]), fmul(n[1], lo[1])), fmul(n[2], lo[2])), d);
        if (dmin > 0.0f)
                return false;
        float dmax = fadd(fadd(fadd(fmul(n[0], hi[0]), fmul(n[1], hi[1])), fmul(n[2], hi[2])), d);
        if (!(dmax >= 0.0f))
                return false;
        float fx, fy, fz;
        // edge 0: AXISTEST_X01, Y02, Z12 (tribox2.cc:139-144)
        fx = fabsf(e0[0]); fy = fabsf(e0[1]); fz = fabsf(e0[2]);
        if (axis_sep(fsub(fmul(e0[2], v0[1]), fmul(e0[1], v0[2])),
                     fsub(fmul(e0[2], v2[1]), fmul(e0[1], v2[2])),
                     fadd(fmul(fz, h[1]), fmul(fy, h[2])))) return false;
        if (axis_sep(fadd(fmul(-e0[2], v0[0]), fmul(e0[0], v0[2])),
                     fadd(fmul(-e0[2], v2[0]), fmul(e0[0], v2[2])),
                     fadd(fmul(fz, h[0]), fmul(fx, h[2])))) return false;
        if (axis_sep(fsub(fmul(e0[1], v2[0]), fmul(e0[0], v2[1])),
                     fsub(fmul(e0[1], v1[0]), fmul(e0[0], v1[1])),
                     fadd(fmul(fy, h[0]), fmul(fx, h[1])))) return false;
        // edge 1: X01, Y02, Z0 (tribox2.cc:146-151)
        fx = fabsf(e1[0]); fy = fabsf(e1[1]); fz = fabsf(e1[2]);
        if (axis_sep(fsub(fmul(e1[2], v0[1]), fmul(e1[1], v0[2])),
                     fsub(fmul(e1[2], v2[1]), fmul(e1[1], v2[2])),
                     fadd(fmul(fz, h[1]), fmul(fy, h[2])))) return false;
        if (axis_sep(fadd(fmul(-e1[2], v0[0]), fmul(e1[0], v0[2])),
                     fadd(fmul(-e1[2], v2[0]), fmul(e1[0], v2[2])),
                     fadd(fmul(fz, h[0]), fmul(fx, h[2])))) return false;
        if (axis_sep(fsub(fmul(e1[1], v0[0]), fmul(e1[0], v0[1])),
                     fsub(fmul(e1[1], v1[0]), fmul(e1[0], v1[1])),
                     fadd(fmul(fy, h[0]), fmul(fx, h[1])))) return false;
        // edge 2: X2, Y1, Z12 (tribox2.cc:153-158)
        fx = fabsf(e2[0]); fy = fabsf(e2[1]); fz = fabsf(e2[2]);
        if (axis_sep(fsub(fmul(e2[2], v0[1]), fmul(e2[1], v0[2])),
                     fsub(fmul(e2[2], v1[1]), fmul(e2[1], v1[2])),
                     fadd(fmul(fz, h[1]), fmul(fy, h[2])))) return false;
        if (axis_sep(fadd(fmul(-e2[2], v0[0]), fmul(e2[0], v0[2])),
                     fadd(fmul(-e2[2], v1[0]), fmul(e2[0], v1[2])),
                     fadd(fmul(fz, h[0]), fmul(fx, h[2])))) return false;
        if (axis_sep(fsub(fmul(e2[1], v2[0]), fmul(e2[0], v2[1])),
                     fsub(fmul(e2[1], v1[0]), fmul(e2[0], v1[1])),
                     fadd(fmul(fy, h[0]), fmul(fx, h[1])))) return false;
        return true;
}

// Triangle::is_overlap (voxel_octree.cc:486-492): centre=(min+max)*.5f
// (graphics_math.h:1252-1255), half=(max-min)/2.f.
__device__ __forceinline__ bool tri_overlaps_aabb(const float mn[3], const float mx[3],
                                                  const float t0[3], const float t1[3],
                                                  const float t2[3])
{
        float c[3], h[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                c[k] = fmul(fadd(mn[k], mx[k]), .5f);
                h[k] = fdiv(fsub(mx[k], mn[k]), 2.f);
        }
        return tribox_overlap(c, h, t0, t1, t2);
}

// ---------------------------------------------------------------------------
// The EIGHT Triangle::is_overlap calls of one triangle against the eight children of one cell
// (insert's loop over children, voxel_octree.cc:45-50,61-64), evaluated by ONE thread (round 2).
// Every float operation of the eight triBoxOverlap calls is kept, with the same operands in the same
// order; what is shared are the sub-expressions that are literally identical between children: a
// child's centre/half, the translated vertices and the edges only depend on the child's HALF per axis
// (two values per axis, not eight), an edge-axis test only on two of the three halves (four variants,
// not eight), and the normal's components likewise.  bx/by/bz = (lo.min, lo.max, hi.min, hi.max) of the
// cell's two child intervals per axis.  Returns the 8 verdicts, bit c = child c (x bit 2, y bit 1, z bit 0).
// ---------------------------------------------------------------------------
__device__ __forceinline__ bool axis_sep2(float pa, float pb, float rad)
{
        const float mn = (pa < pb) ? pa : pb;
        const float mx = (pa < pb) ? pb : pa;
        return (mn > rad) || (mx < -rad);
}

__device__ __forceinline__ uint32_t tri_overlaps_children8(const float4 bx, const float4 by, const float4 bz,
                                                           const float t0[3], const float t1[3], const float t2[3])
{
        const float4 bb[3] = { bx, by, bz };
        float h[3][2], v0[3][2], v1[3][2], v2[3][2];
        uint32_t boxok[3];  // bit s: the child half s of this axis passes the box-axis test
#pragma unroll
        for (int a = 0; a < 3; ++a) {
                boxok[a] = 0;
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                        const float mn = s ? bb[a].z : bb[a].x, mx = s ? bb[a].w : bb[a].y;
                        // centre=(min+max)*.5f, half=(max-min)/2.f (x/2.f == x*.5f bit for bit, denormals included)
                        const float c = fmul(fadd(mn, mx), .5f);
                        h[a][s] = fmul(fsub(mx, mn), .5f);
                        v0[a][s] = fsub(t0[a], c);
                        v1[a][s] = fsub(t1[a], c);
                        v2[a][s] = fsub(t2[a], c);
                        float lo = v0[a][s], hi = v0[a][s];
                        if (v1[a][s] < lo) lo = v1[a][s];
                        if (v1[a][s] > hi) hi = v1[a][s];
                        if (v2[a][s] < lo) lo = v2[a][s];
                        if (v2[a][s] > hi) hi = v2[a][s];
                        if (!(lo > h[a][s] || hi < -h[a][s]))
                                boxok[a] |= 1u << s;
                }
        }
        // candidates: children whose three box-axis tests pass
        uint32_t cand = 0;
#pragma unroll
        for (int c = 0; c < 8; ++c)
                if (((boxok[0] >> (c >> 2)) & (boxok[1] >> ((c >> 1) & 1)) & (boxok[2] >> (c & 1)) & 1u) != 0u)
                        cand |= 1u << c;
        if (!cand)
                return 0u;
        float e0[3][2], e1[3][2], e2[3][2];
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                        e0[a][s] = fsub(v1[a][s], v0[a][s]);
                        e1[a][s] = fsub(v2[a][s], v1[a][s]);
                        e2[a][s] = fsub(v0[a][s], v2[a][s]);
                }
        // plane (tribox2.cc:181-183 + 42-63): normal = cross(e0, e1); component q depends on the halves of the
        // two other axes
        float n0[2][2], n1[2][2], n2[2][2];  // n0[sy][sz], n1[sz][sx], n2[sx][sy]
#pragma unroll
        for (int p = 0; p < 2; ++p)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                        n0[p][q] = fsub(fmul(e0[1][p], e1[2][q]), fmul(e0[2][q], e1[1][p]));
                        n1[p][q] = fsub(fmul(e0[2][p], e1[0][q]), fmul(e0[0][q], e1[2][p]));
                        n2[p][q] = fsub(fmul(e0[0][p], e1[1][q]), fmul(e0[1][q], e1[0][p]));
                }
#pragma unroll
        for (int c = 0; c < 8; ++c) {
                if (!((cand >> c) & 1u))
                        continue;
                const int sx = c >> 2, sy = (c >> 1) & 1, sz = c & 1;
                const float nx = n0[sy][sz], ny = n1[sz][sx], nz = n2[sx][sy];
                const float d = -fadd(fadd(fmul(nx, v0[0][sx]), fmul(ny, v0[1][sy])), fmul(nz, v0[2][sz]));
                // vmin[q] = n[q] > 0 ? -h : h ; vmax = -vmin ;  n*(-h) == -(n*h) bit for bit
                const float mx_ = fmul(nx, h[0][sx]), my_ = fmul(ny, h[1][sy]), mz_ = fmul(nz, h[2][sz]);
                const float lx = (nx > 0.0f) ? -mx_ : mx_, ly = (ny > 0.0f) ? -my_ : my_, lz = (nz > 0.0f) ? -mz_ : mz_;
                const float dmin = fadd(fadd(fadd(lx, ly), lz), d);
                const float dmax = fadd(fadd(fadd(-lx, -ly), -lz), d);
                if (dmin > 0.0f || !(dmax >= 0.0f))
                        cand &= ~(1u << c);
        }
        if (!cand)
                return 0u;
        // edge axes.  X-type tests (AXISTEST_X01 / X2) use the y and z halves, Y-type x and z, Z-type x and y.
#pragma unroll
        for (int p = 0; p < 2; ++p)
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                        {  // X-type, halves (sy, sz) = (p, q): children {p*2+q, 4+p*2+q}
                                const uint32_t m = (1u << (p * 2 + q)) | (1u << (4 + p * 2 + q));
                                if (cand & m) {
                                        bool sep;
                                        // edge 0: X01 (v0, v2); edge 1: X01 (v0, v2); edge 2: X2 (v0, v1)
                                        sep = axis_sep2(fsub(fmul(e0[2][q], v0[1][p]), fmul(e0[1][p], v0[2][q])),
                                                        fsub(fmul(e0[2][q], v2[1][p]), fmul(e0[1][p], v2[2][q])),
                                                        fadd(fmul(fabsf(e0[2][q]), h[1][p]), fmul(fabsf(e0[1][p]), h[2][q])));
                                        sep = sep || axis_sep2(fsub(fmul(e1[2][q], v0[1][p]), fmul(e1[1][p], v0[2][q])),
                                                               fsub(fmul(e1[2][q], v2[1][p]), fmul(e1[1][p], v2[2][q])),
                                                               fadd(fmul(fabsf(e1[2][q]), h[1][p]), fmul(fabsf(e1[1][p]), h[2][q])));
                                        sep = sep || axis_sep2(fsub(fmul(e2[2][q], v0[1][p]), fmul(e2[1][p], v0[2][q])),
                                                               fsub(fmul(e2[2][q], v1[1][p]), fmul(e2[1][p], v1[2][q])),
                                                               fadd(fmul(fabsf(e2[2][q]), h[1][p]), fmul(fabsf(e2[1][p]), h[2][q])));
                                        if (sep)
                                                cand &= ~m;
                                }
                        }
                        {  // Y-type, halves (sx, sz) = (p, q): children {p*4+q, p*4+2+q}
                                const uint32_t m = (1u << (p * 4 + q)) | (1u << (p * 4 + 2 + q));
                                if (cand & m) {
                                        bool sep;
                                        // edge 0: Y02 (v0, v2); edge 1: Y02 (v0, v2); edge 2: Y1 (v0, v1)
                                        sep = axis_sep2(fadd(fmul(-e0[2][q], v0[0][p]), fmul(e0[0][p], v0[2][q])),
                                                        fadd(fmul(-e0[2][q], v2[0][p]), fmul(e0[0][p], v2[2][q])),
                                                        fadd(fmul(fabsf(e0[2][q]), h[0][p]), fmul(fabsf(e0[0][p]), h[2][q])));
                                        sep = sep || axis_sep2(fadd(fmul(-e1[2][q], v0[0][p]), fmul(e1[0][p], v0[2][q])),
                                                               fadd(fmul(-e1[2][q], v2[0][p]), fmul(e1[0][p], v2[2][q])),
                                                               fadd(fmul(fabsf(e1[2][q]), h[0][p]), fmul(fabsf(e1[0][p]), h[2][q])));
                                        sep = sep || axis_sep2(fadd(fmul(-e2[2][q], v0[0][p]), fmul(e2[0][p], v0[2][q])),
                                                               fadd(fmul(-e2[2][q], v1[0][p]), fmul(e2[0][p], v1[2][q])),
                                                               fadd(fmul(fabsf(e2[2][q]), h[0][p]), fmul(fabsf(e2[0][p]), h[2][q])));
                                        if (sep)
                                                cand &= ~m;
                                }
                        }
                        {  // Z-type, halves (sx, sy) = (p, q): children {p*4+q*2, p*4+q*2+1}
                                const uint32_t m = (1u << (p * 4 + q * 2)) | (1u << (p * 4 + q * 2 + 1));
                                if (cand & m) {
                                        bool sep;
                                        // edge 0: Z12 (v2, v1); edge 1: Z0 (v0, v1); edge 2: Z12 (v2, v1)
                                        sep = axis_sep2(fsub(fmul(e0[1][q], v2[0][p]), fmul(e0[0][p], v2[1][q])),
                                                        fsub(fmul(e0[1][q], v1[0][p]), fmul(e0[0][p], v1[1][q])),
                                                        fadd(fmul(fabsf(e0[1][q]), h[0][p]), fmul(fabsf(e0[0][p]), h[1][q])));
                                        sep = sep || axis_sep2(fsub(fmul(e1[1][q], v0[0][p]), fmul(e1[0][p], v0[1][q])),
                                                               fsub(fmul(e1[1][q], v1[0][p]), fmul(e1[0][p], v1[1][q])),
                                                               fadd(fmul(fabsf(e1[1][q]), h[0][p]), fmul(fabsf(e1[0][p]), h[1][q])));
                                        sep = sep || axis_sep2(fsub(fmul(e2[1][q], v2[0][p]), fmul(e2[0][p], v2[1][q])),
                                                               fsub(fmul(e2[1][q], v1[0][p]), fmul(e2[0][p], v1[1][q])),
                                                               fadd(fmul(fabsf(e2[1][q]), h[0][p]), fmul(fabsf(e2[0][p]), h[1][q])));
                                        if (sep)
                                                cand &= ~m;
                                }
                        }
                }
        return cand;
}

// ---------------------------------------------------------------------------
// intersect_triangle3 (raytri.cc:197-249): double, two-sided, EPSILON 1e-6
// (raytri.cc:9), inv_det computed before the sign branch, no test on t.
// ---------------------------------------------------------------------------
__device__ __forceinline__ double ddot3(const double a[3], const double b[3])
{
        return dadd(dadd(dmul(a[0], b[0]), dmul(a[1], b[1])), dmul(a[2], b[2]));
}

__device__ __forceinline__ void dcross(double o[3], const double a[3], const double b[3])
{
        o[0] = dsub(dmul(a[1], b[2]), dmul(a[2], b[1]));
        o[1] = dsub(dmul(a[2], b[0]), dmul(a[0], b[2]));
        o[2] = dsub(dmul(a[0], b[1]), dmul(a[1], b[0]));
}

// intersect_triangle3 from the point where edge1 = vert1 - vert0 and edge2 = vert2 - vert0 are known
__device__ __forceinline__ int ray_triangle3_edges(const double o[3], const double dir[3], const double a[3],
                                                   const double e1[3], const double e2[3], double& t, double& u,
                                                   double& v);

__device__ __forceinline__ int ray_triangle3(const double o[3], const double dir[3],
                                             const double a[3], const double b[3],
                                             const double c[3], double& t, double& u,
                                             double& v)
{
        double e1[3], e2[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                e1[k] = dsub(b[k], a[k]);
                e2[k] = dsub(c[k], a[k]);
        }
        return ray_triangle3_edges(o, dir, a, e1, e2, t, u, v);
}

__device__ __forceinline__ int ray_triangle3_edges(const double o[3], const double dir[3], const double a[3],
                                                   const double e1[3], const double e2[3], double& t, double& u,
                                                   double& v)
{
        const double eps = 0.000001;
        double tv[3], pv[3], qv[3];
        dcross(pv, dir, e2);
        double det = ddot3(e1, pv);
#pragma unroll
        for (int k = 0; k < 3; ++k)
                tv[k] = dsub(o[k], a[k]);
        if (det > eps) {
                u = ddot3(tv, pv);
                if (u < 0.0 || u > det)
                        return 0;
                dcross(qv, tv, e1);
                v = ddot3(dir, qv);
                if (v < 0.0 || dadd(u, v) > det)
                        return 0;
        } else if (det < -eps) {
                u = ddot3(tv, pv);
                if (u > 0.0 || u < det)
                        return 0;
                dcross(qv, tv, e1);
                v = ddot3(dir, qv);
                if (v > 0.0 || dadd(u, v) < det)
                        return 0;
        } else {
                return 0;
        }
        double inv = __ddiv_rn(1.0, det);
        t = dmul(ddot3(e2, qv), inv);
        u = dmul(u, inv);
        v = dmul(v, inv);
        return 1;
}

// ray_triangle3_edges for a ray whose origin o is known before the launch: tv = o - a, qv = tv x e1 and tq = e2 . qv
// depend on (o, triangle) only and come precomputed with the same operations (k_tri_eye_rel); branches, the 1/det
// and the results are those of ray_triangle3_edges.
__device__ __forceinline__ int ray_triangle3_eye(const double dir[3], const double e1[3], const double e2[3],
                                                 const double tv[3], const double qv[3], double tq, double& t,
                                                 double& u, double& v)
{
        const double eps = 0.000001;
        double pv[3];
        dcross(pv, dir, e2);
        double det = ddot3(e1, pv);
        if (det > eps) {
                u = ddot3(tv, pv);
                if (u < 0.0 || u > det)
                        return 0;
                v = ddot3(dir, qv);
                if (v < 0.0 || dadd(u, v) > det)
                        return 0;
        } else if (det < -eps) {
                u = ddot3(tv, pv);
                if (u > 0.0 || u < det)
                        return 0;
                v = ddot3(dir, qv);
                if (v > 0.0 || dadd(u, v) < det)
                        return 0;
        } else {
                return 0;
        }
        double inv = __ddiv_rn(1.0, det);
        t = dmul(tq, inv);
        u = dmul(u, inv);
        v = dmul(v, inv);
        return 1;
}

// ---------------------------------------------------------------------------
// AABB<Vec3>::isect(ray, nullptr) (graphics_math.h:1312-1332)
// ---------------------------------------------------------------------------
// d with every 0.f (incl. -0.f) replaced by FLT_MIN, then 1.f/d (true division).
__device__ __forceinline__ float slab_dinv(float d)
{
        float dd = (d == 0.f) ? FLT_MIN : d;
        return fdiv(1.f, dd);
}

// *std::max_element over 3 values: first maximum, '<' only.
__device__ __forceinline__ float max_element3(float a, float b, float c)
{
        float m = a;
        if (m < b) m = b;
        if (m < c) m = c;
        return m;
}
__device__ __forceinline__ float min_element3(float a, float b, float c)
{
        float m = a;
        if (b < m) m = b;
        if (c < m) m = c;
        return m;
}

__device__ __forceinline__ bool slab_accept(float t0, float t1, float tmin, float tmax)
{
        if (t0 > t1)
                return false;
        return (t0 >= tmin && t0 <= tmax) || (t1 >= tmin && t1 <= tmax);
}

__device__ __forceinline__ bool aabb_isect(const float mn[3], const float mx[3],
                                           const float o[3], const float dinv[3],
                                           float tmin, float tmax)
{
        float lo[3], hi[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
                float a = fmul(fsub(mn[k], o[k]), dinv[k]);
                float b = fmul(fsub(mx[k], o[k]), dinv[k]);
                lo[k] = std_min(a, b);
                hi[k] = std_max(a, b);
        }
        float t0 = max_element3(lo[0], lo[1], lo[2]);
        float t1 = min_element3(hi[0], hi[1], hi[2]);
        return slab_accept(t0, t1, tmin, tmax);
}

// ---------------------------------------------------------------------------
// Camera::gen_rays1/gen_rays4 (camera.cc:77-112) for sample s of pixel (px,py)
// ---------------------------------------------------------------------------
struct CameraParams {
        float C[16];
        float z;
        float tmin, tmax;
        int nx, ny, spp;
};

// direction of sample s of pixel (px,py): vector_transform(C, {x_, y_, z}) normalised by the Ray ctor
__device__ __forceinline__ void gen_ray_dir(const CameraParams& cam, int px, int py, int s, float d[3])
{
        // samples: gen_rays1 {4,4}/8 ; gen_rays4 {1,5},{3,1},{7,3},{5,7} /8
        float sx, sy;
        if (cam.spp == 4) {
                sx = (s == 0) ? 0.125f : (s == 1) ? 0.375f : (s == 2) ? 0.875f : 0.625f;
                sy = (s == 0) ? 0.625f : (s == 1) ? 0.125f : (s == 2) ? 0.375f : 0.875f;
        } else {
                sx = 0.5f;
                sy = 0.5f;
        }
        const float x = (float)(px - cam.nx / 2);
        const float y = (float)((cam.ny - 1 - py) - cam.ny / 2);
        const float x_ = fdiv(fadd(x, sx), (float)cam.nx);
        const float y_ = fdiv(fadd(y, sy), (float)cam.ny);
        // vector_transform(C,{x_,y_,z}): graphics_math.h:1063-1077 via dot(Mat4,Vec4) :552-562
#pragma unroll
        for (int r = 0; r < 3; ++r) {
                float b = fadd(0.f, fmul(cam.C[r], x_));
                b = fadd(b, fmul(cam.C[4 + r], y_));
                b = fadd(b, fmul(cam.C[8 + r], cam.z));
                b = fadd(b, fmul(cam.C[12 + r], 0.f));
                d[r] = b;
        }
        normalize3(d[0], d[1], d[2]);  // Ray ctor graphics_math.h:1159-1166
}

// origin of every ray of the camera: point_transform(C, {0,0,0}) -- the same four-term column sums and the
// division by w as the reference, evaluated once per launch (the launcher runs the identical float operations on
// the host, vrt_trace.cu camera_eye_host, and hands the result to the kernel)
__device__ __forceinline__ void gen_ray_origin(const CameraParams& cam, float o[3])
{
        float o4[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
                float a = fadd(0.f, fmul(cam.C[r], 0.f));
                a = fadd(a, fmul(cam.C[4 + r], 0.f));
                a = fadd(a, fmul(cam.C[8 + r], 0.f));
                a = fadd(a, fmul(cam.C[12 + r], 1.f));
                o4[r] = a;
        }
        o[0] = fdiv(o4[0], o4[3]);
        o[1] = fdiv(o4[1], o4[3]);
        o[2] = fdiv(o4[2], o4[3]);
}

__device__ __forceinline__ void gen_ray(const CameraParams& cam, int px, int py, int s,
                                        float o[3], float d[3])
{
        gen_ray_origin(cam, o);
        gen_ray_dir(cam, px, py, s, d);
}

// ---------------------------------------------------------------------------
// Film export encodings (the two formats the reference turns its float film into).
// ---------------------------------------------------------------------------
// float -> unsigned char as x86-64 compiles `(unsigned char)f` / static_cast<std::uint8_t>(f): CVTTSS2SI to a
// 32-bit integer (0x80000000 for NaN and for |f| >= 2^31), then the low byte.  In range ([0,256)) this is the
// plain truncation the C++ standard defines; outside it the standard leaves the result open and this is what the
// reference binary does.
__device__ __forceinline__ uint32_t f2u8_x86(float f)
{
        const int i = (fabsf(f) < 2147483648.f) ? __float2int_rz(f) : (int)0x80000000;
        return (uint32_t)i & 0xffu;
}

// Film::to_byte_array (camera.cc:27-48): v = rawv * 255.9f, every component cast to std::uint8_t.
__device__ __forceinline__ uint32_t film_rgb8(const float c[3])
{
        return f2u8_x86(fmul(c[0], 255.9f)) | (f2u8_x86(fmul(c[1], 255.9f)) << 8) | (f2u8_x86(fmul(c[2], 255.9f)) << 16);
}

// stbiw__linear_to_rgbe (stb_image_write.h:601-616), the pixel encoding of stbi_write_hdr(Film::to_float_array())
// (main.cc:125-126): maxcomp by the `a > b ? a : b` macro, zero below 1e-32f, else
// normalize = (float)frexp(maxcomp, &e) * 256.0f / maxcomp (left to right, single precision) and the three
// components truncated to bytes, e + 128 as the fourth.  maxcomp >= 1e-32f is a normal float, so frexp's mantissa
// and exponent are the float's own fields (finite films; stb's result for Inf/NaN pixels is not defined).
__device__ __forceinline__ uint32_t film_rgbe(const float c[3])
{
        const float m12 = (c[1] > c[2]) ? c[1] : c[2];
        const float mc = (c[0] > m12) ? c[0] : m12;
        if (mc < 1e-32f)
                return 0u;
        const uint32_t b = __float_as_uint(mc);
        const int e = (int)((b >> 23) & 0xffu) - 126;
        const float frac = __uint_as_float((b & 0x807fffffu) | 0x3f000000u);
        const float nrm = fdiv(fmul(frac, 256.0f), mc);
        return f2u8_x86(fmul(c[0], nrm)) | (f2u8_x86(fmul(c[1], nrm)) << 8) | (f2u8_x86(fmul(c[2], nrm)) << 16) |
               (((uint32_t)(e + 128) & 0xffu) << 24);
}

}  // namespace vrt
