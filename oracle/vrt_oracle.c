/* oracle/vrt_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * CPU restatement (plain C99, scalar, FMA-free: compile with
 * -ffp-contract=off) of the reference's hot path, written from the behaviour
 * of jqly/VoxelRayTrace20190722 -- each function cites the reference
 * file:line it follows (paths relative to VoxelRayTrace20190722/).
 *
 * Parity status: PINNED.  The reference ships no golden vectors
 * (SURVEY.md 4), so this restatement is pinned against the reference itself,
 * compiled unmodified into oracle/_ref/libvrt_ref.so (oracle/build_ref.sh):
 * tests/test_oracle_vs_ref.py compares every entry point below with the
 * reference on seeded inputs, and tests/golden/ holds vectors generated from
 * the reference by tests/golden/make_golden.py.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load the library built from this file.  The
 * product (libvrt.so) never links or calls it.
 *
 * Data layout is deliberately NOT the reference's pointer tree: nodes live in
 * one growable pool and are exported as (Morton-sorted leaf list, per-leaf
 * triangle index list) so the GPU result can be compared array-for-array.
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ */
/* Predicates                                                          */
/* ------------------------------------------------------------------ */

/* tribox2.cc:42-63 planeBoxOverlap (2001 variant: normal, d, maxbox). */
static int orc_plane_box(const float n[3], float d, const float hb[3])
{
        float lo[3], hi[3];
        for (int q = 0; q < 3; ++q) {
                if (n[q] > 0.0f) {
                        lo[q] = -hb[q];
                        hi[q] = hb[q];
                } else {
                        lo[q] = hb[q];
                        hi[q] = -hb[q];
                }
        }
        if ((n[0] * lo[0] + n[1] * lo[1] + n[2] * lo[2]) + d > 0.0f)
                return 0;
        if ((n[0] * hi[0] + n[1] * hi[1] + n[2] * hi[2]) + d >= 0.0f)
                return 1;
        return 0;
}

/* One edge-cross-axis SAT test.  pa,pb are the two projected vertices the
 * reference macro evaluates (tribox2.cc:67-110); rad the projected box radius.
 * `first_lt_second` semantics: the macros use  if(pa<pb){min=pa;max=pb;} else
 * {min=pb;max=pa;}  -- for non-NaN inputs that equals plain min/max. */
static int orc_axis_sep(float pa, float pb, float rad)
{
        float mn, mx;
        if (pa < pb) {
                mn = pa;
                mx = pb;
        } else {
                mn = pb;
                mx = pa;
        }
        return (mn > rad || mx < -rad);
}

/* tribox2.cc:112-186 triBoxOverlap.  tri = 9 floats v0,v1,v2. */
int orc_tribox(const float c[3], const float h[3], const float tri[9])
{
        float v0[3], v1[3], v2[3], e0[3], e1[3], e2[3];
        for (int k = 0; k < 3; ++k) {
                v0[k] = tri[k] - c[k];
                v1[k] = tri[3 + k] - c[k];
                v2[k] = tri[6 + k] - c[k];
        }
        for (int k = 0; k < 3; ++k) {
                e0[k] = v1[k] - v0[k];
                e1[k] = v2[k] - v1[k];
                e2[k] = v0[k] - v2[k];
        }
        float fx, fy, fz;
        /* edge 0: X01, Y02, Z12  (tribox2.cc:139-144) */
        fx = fabsf(e0[0]); fy = fabsf(e0[1]); fz = fabsf(e0[2]);
        if (orc_axis_sep(e0[2] * v0[1] - e0[1] * v0[2], e0[2] * v2[1] - e0[1] * v2[2],
                         fz * h[1] + fy * h[2])) return 0;
        if (orc_axis_sep(-e0[2] * v0[0] + e0[0] * v0[2], -e0[2] * v2[0] + e0[0] * v2[2],
                         fz * h[0] + fx * h[2])) return 0;
        /* Z12 compares p2<p1 first; symmetric for min/max of non-NaN */
        if (orc_axis_sep(e0[1] * v2[0] - e0[0] * v2[1], e0[1] * v1[0] - e0[0] * v1[1],
                         fy * h[0] + fx * h[1])) return 0;
        /* edge 1: X01, Y02, Z0  (tribox2.cc:146-151) */
        fx = fabsf(e1[0]); fy = fabsf(e1[1]); fz = fabsf(e1[2]);
        if (orc_axis_sep(e1[2] * v0[1] - e1[1] * v0[2], e1[2] * v2[1] - e1[1] * v2[2],
                         fz * h[1] + fy * h[2])) return 0;
        if (orc_axis_sep(-e1[2] * v0[0] + e1[0] * v0[2], -e1[2] * v2[0] + e1[0] * v2[2],
                         fz * h[0] + fx * h[2])) return 0;
        if (orc_axis_sep(e1[1] * v0[0] - e1[0] * v0[1], e1[1] * v1[0] - e1[0] * v1[1],
                         fy * h[0] + fx * h[1])) return 0;
        /* edge 2: X2, Y1, Z12  (tribox2.cc:153-158) */
        fx = fabsf(e2[0]); fy = fabsf(e2[1]); fz = fabsf(e2[2]);
        if (orc_axis_sep(e2[2] * v0[1] - e2[1] * v0[2], e2[2] * v1[1] - e2[1] * v1[2],
                         fz * h[1] + fy * h[2])) return 0;
        if (orc_axis_sep(-e2[2] * v0[0] + e2[0] * v0[2], -e2[2] * v1[0] + e2[0] * v1[2],
                         fz * h[0] + fx * h[2])) return 0;
        if (orc_axis_sep(e2[1] * v2[0] - e2[0] * v2[1], e2[1] * v1[0] - e2[0] * v1[1],
                         fy * h[0] + fx * h[1])) return 0;
        /* the three box-axis tests, strict inequalities (tribox2.cc:166-176) */
        for (int k = 0; k < 3; ++k) {
                float mn = v0[k], mx = v0[k];
                if (v1[k] < mn) mn = v1[k];
                if (v1[k] > mx) mx = v1[k];
                if (v2[k] < mn) mn = v2[k];
                if (v2[k] > mx) mx = v2[k];
                if (mn > h[k] || mx < -h[k])
                        return 0;
        }
        /* plane test (tribox2.cc:181-183) */
        float n[3];
        n[0] = e0[1] * e1[2] - e0[2] * e1[1];
        n[1] = e0[2] * e1[0] - e0[0] * e1[2];
        n[2] = e0[0] * e1[1] - e0[1] * e1[0];
        float d = -(n[0] * v0[0] + n[1] * v0[1] + n[2] * v0[2]);
        return orc_plane_box(n, d, h) ? 1 : 0;
}

/* voxel_octree.cc:486-492 Triangle::is_overlap: centre=(min+max)*.5f
 * (graphics_math.h:1252-1255), half=(max-min)/2.f. */
int orc_tri_overlaps_aabb(const float mn[3], const float mx[3], const float tri[9])
{
        float c[3], h[3];
        for (int k = 0; k < 3; ++k) {
                c[k] = (mn[k] + mx[k]) * .5f;
                h[k] = (mx[k] - mn[k]) / 2.f;
        }
        return orc_tribox(c, h, tri) == 1;
}

/* raytri.cc:197-249 intersect_triangle3 (double, two-sided, no t test). */
int orc_raytri(const double o[3], const double dir[3], const double a[3],
               const double b[3], const double c[3], double* t, double* u, double* v)
{
        const double eps = 0.000001; /* raytri.cc:9 */
        double e1[3], e2[3], tv[3], pv[3], qv[3];
        for (int k = 0; k < 3; ++k) {
                e1[k] = b[k] - a[k];
                e2[k] = c[k] - a[k];
        }
        pv[0] = dir[1] * e2[2] - dir[2] * e2[1];
        pv[1] = dir[2] * e2[0] - dir[0] * e2[2];
        pv[2] = dir[0] * e2[1] - dir[1] * e2[0];
        double det = e1[0] * pv[0] + e1[1] * pv[1] + e1[2] * pv[2];
        for (int k = 0; k < 3; ++k)
                tv[k] = o[k] - a[k];
        double inv = 1.0 / det;
        qv[0] = tv[1] * e1[2] - tv[2] * e1[1];
        qv[1] = tv[2] * e1[0] - tv[0] * e1[2];
        qv[2] = tv[0] * e1[1] - tv[1] * e1[0];
        if (det > eps) {
                *u = tv[0] * pv[0] + tv[1] * pv[1] + tv[2] * pv[2];
                if (*u < 0.0 || *u > det)
                        return 0;
                *v = dir[0] * qv[0] + dir[1] * qv[1] + dir[2] * qv[2];
                if (*v < 0.0 || *u + *v > det)
                        return 0;
        } else if (det < -eps) {
                *u = tv[0] * pv[0] + tv[1] * pv[1] + tv[2] * pv[2];
                if (*u > 0.0 || *u < det)
                        return 0;
                *v = dir[0] * qv[0] + dir[1] * qv[1] + dir[2] * qv[2];
                if (*v > 0.0 || *u + *v < det)
                        return 0;
        } else {
                return 0;
        }
        *t = (e2[0] * qv[0] + e2[1] * qv[1] + e2[2] * qv[2]) * inv;
        *u *= inv;
        *v *= inv;
        return 1;
}

/* std::min / std::max semantics (matter only for NaN): min(a,b)=(b<a)?b:a,
 * max(a,b)=(a<b)?b:a. */
static float std_minf(float a, float b) { return (b < a) ? b : a; }
static float std_maxf(float a, float b) { return (a < b) ? b : a; }

/* graphics_math.h:1312-1332 AABB<Vec3>::isect(ray, nullptr).
 * ray = o3,d3,tmin,tmax. */
int orc_aabb_isect(const float mn[3], const float mx[3], const float ray[8])
{
        float lo[3], hi[3];
        for (int k = 0; k < 3; ++k) {
                float d = ray[3 + k];
                if (d == 0.f) /* std::replace(...,0.f,FLT_MIN): matches -0.f too */
                        d = FLT_MIN;
                float dinv = 1.f / d;
                float a = (mn[k] - ray[k]) * dinv;
                float b = (mx[k] - ray[k]) * dinv;
                lo[k] = std_minf(a, b);
                hi[k] = std_maxf(a, b);
        }
        /* std::max_element / std::min_element: first extremum, '<' only */
        float t0 = lo[0];
        if (t0 < lo[1]) t0 = lo[1];
        if (t0 < lo[2]) t0 = lo[2];
        float t1 = hi[0];
        if (hi[1] < t1) t1 = hi[1];
        if (hi[2] < t1) t1 = hi[2];
        if (t0 > t1)
                return 0;
        float tmin = ray[6], tmax = ray[7];
        return ((t0 >= tmin && t0 <= tmax) || (t1 >= tmin && t1 <= tmax)) ? 1 : 0;
}

/* ------------------------------------------------------------------ */
/* Camera                                                              */
/* ------------------------------------------------------------------ */

static void v3_normalize(float v[3])
{
        /* graphics_math.h:532-586: dot = ((0+x*x)+y*y)+z*z ; v / sqrtf(dot) */
        float s = 0.f;
        s += v[0] * v[0];
        s += v[1] * v[1];
        s += v[2] * v[2];
        float l = sqrtf(s);
        v[0] = v[0] / l;
        v[1] = v[1] / l;
        v[2] = v[2] / l;
}

static void v3_cross(const float p[3], const float q[3], float out[3])
{
        /* graphics_math.h:588-592 */
        out[0] = p[1] * q[2] - q[1] * p[2];
        out[1] = p[2] * q[0] - q[2] * p[0];
        out[2] = p[0] * q[1] - q[0] * p[1];
}

/* camera.cc:65-75 Camera::Camera -> column-major C_[col][row], 16 floats.
 * cam10 = fov, eye3, spot3, up3. */
void orc_camera_matrix(const float cam10[10], float C[16])
{
        const float* eye = cam10 + 1;
        const float* spot = cam10 + 4;
        const float* up = cam10 + 7;
        float f[3] = { spot[0] - eye[0], spot[1] - eye[1], spot[2] - eye[2] };
        v3_normalize(f);
        float s[3], u[3];
        v3_cross(f, up, s);
        v3_normalize(s);
        v3_cross(s, f, u);
        v3_normalize(u);
        memset(C, 0, 16 * sizeof(float));
        for (int r = 0; r < 3; ++r) {
                C[0 + r] = s[r];
                C[4 + r] = u[r];
                C[8 + r] = -f[r];
                C[12 + r] = eye[r];
        }
        C[15] = 1.f;
}

/* z of camera.cc:82,100:  -(film.h / (2*tanf(fov/2)))  (host libm tanf). */
float orc_camera_z(float fov, float film_h)
{
        return -(film_h / (2 * tanf(fov / 2)));
}

/* camera.cc:77-112 gen_rays1/gen_rays4 for one pixel; out = spp rays x 8. */
void orc_gen_rays_pixel(const float C[16], float z, int nx, int ny, int spp, int px,
                        int py, float* out)
{
        static const float s4[4][2] = { { 1, 5 }, { 3, 1 }, { 7, 3 }, { 5, 7 } };
        const float x = (float)(px - nx / 2);
        const float y = (float)((ny - 1 - py) - ny / 2);
        for (int k = 0; k < spp; ++k) {
                float sx = (spp == 4 ? s4[k][0] : 4.f) / 8.f;
                float sy = (spp == 4 ? s4[k][1] : 4.f) / 8.f;
                float x_ = (x + sx) / (float)nx;
                float y_ = (y + sy) / (float)ny;
                /* point_transform(C,{0,0,0}) graphics_math.h:1063-1070:
                 * acc = 0; acc += C[i]*v[i] for i=0..3 with v=(0,0,0,1); /= w */
                float o4[4], d4[4];
                for (int r = 0; r < 4; ++r) {
                        float a = 0.f;
                        a += C[0 + r] * 0.f;
                        a += C[4 + r] * 0.f;
                        a += C[8 + r] * 0.f;
                        a += C[12 + r] * 1.f;
                        o4[r] = a;
                        float b = 0.f;
                        b += C[0 + r] * x_;
                        b += C[4 + r] * y_;
                        b += C[8 + r] * z;
                        b += C[12 + r] * 0.f;
                        d4[r] = b;
                }
                float* r8 = out + 8 * k;
                r8[0] = o4[0] / o4[3];
                r8[1] = o4[1] / o4[3];
                r8[2] = o4[2] / o4[3];
                float d[3] = { d4[0], d4[1], d4[2] };
                v3_normalize(d); /* Ray ctor graphics_math.h:1159-1166 */
                r8[3] = d[0];
                r8[4] = d[1];
                r8[5] = d[2];
                r8[6] = 0.f;     /* Camera near default camera.h:76 */
                r8[7] = FLT_MAX; /* Camera far default  camera.h:77 */
        }
}

void orc_gen_rays(const float C[16], float z, int nx, int ny, int spp, int x0, int y0,
                  int x1, int y1, float* out)
{
        size_t k = 0;
        for (int py = y0; py < y1; ++py)
                for (int px = x0; px < x1; ++px) {
                        orc_gen_rays_pixel(C, z, nx, ny, spp, px, py, out + 8 * k);
                        k += (size_t)spp;
                }
}

/* ------------------------------------------------------------------ */
/* Octree build (voxel_octree.cc:22-75)                                */
/* ------------------------------------------------------------------ */

typedef struct {
        float mn[3], mx[3];
        int32_t child[8]; /* -1 = this node is a leaf (never split) */
        uint32_t* refs;   /* triangle indices, insertion (= ascending) order */
        uint32_t nrefs, cap;
        /* cone-trace state (voxel_octree.h:66-70): coverage, illum[6] (Vec3 each) */
        float coverage;
        float illum[18];
} orc_node;

typedef struct {
        orc_node* nodes;
        size_t n_nodes, cap_nodes;
        const float* tri; /* borrowed [T][9] */
        float* nrm;       /* owned, NORMALISED per-vertex normals [T][9] */
        float* tri_own;   /* owned copy of the vertices */
        uint32_t T;
        int max_depth;
        /* materials (orc_set_materials): per-vertex uv, material id per triangle, per material kd + texture id */
        float* uv;          /* [T][3][2] */
        uint32_t* tri_mtl;  /* [T] */
        uint32_t n_mtl, n_tex;
        float* mtl_kd;      /* [M][3] */
        int32_t* mtl_tex;   /* [M], -1 = untextured */
        int32_t* tex_whc;   /* [n_tex][3] */
        uint8_t** tex_data;
} orc_tree;

static int32_t orc_new_node(orc_tree* t, const float mn[3], const float mx[3])
{
        if (t->n_nodes == t->cap_nodes) {
                t->cap_nodes = t->cap_nodes ? t->cap_nodes * 2 : 1024;
                t->nodes = (orc_node*)realloc(t->nodes, t->cap_nodes * sizeof(orc_node));
        }
        orc_node* n = &t->nodes[t->n_nodes];
        memcpy(n->mn, mn, sizeof n->mn);
        memcpy(n->mx, mx, sizeof n->mx);
        for (int i = 0; i < 8; ++i)
                n->child[i] = -1;
        n->refs = NULL;
        n->nrefs = n->cap = 0;
        n->coverage = 0.f;
        memset(n->illum, 0, sizeof n->illum);
        return (int32_t)t->n_nodes++;
}

/* voxel_octree.cc:27-39 split: size=(max-min)/2 ; child i: mask=(i&4,i&2,i&1)
 * -> min'=min+mask*size ; max'=min'+size  (float recurrence, NOT closed form). */
static void orc_split(orc_tree* t, int32_t ni)
{
        float mn[3], mx[3], sz[3];
        memcpy(mn, t->nodes[ni].mn, sizeof mn);
        memcpy(mx, t->nodes[ni].mx, sizeof mx);
        for (int k = 0; k < 3; ++k)
                sz[k] = (mx[k] - mn[k]) / 2; /* Vec3 / int -> float division */
        for (int i = 0; i < 8; ++i) {
                float cmn[3], cmx[3];
                int m[3] = { (i & 4) ? 1 : 0, (i & 2) ? 1 : 0, (i & 1) ? 1 : 0 };
                for (int k = 0; k < 3; ++k) {
                        cmn[k] = mn[k] + (float)m[k] * sz[k];
                        cmx[k] = cmn[k] + sz[k];
                }
                int32_t c = orc_new_node(t, cmn, cmx); /* may realloc */
                t->nodes[ni].child[i] = c;
        }
}

/* voxel_octree.cc:41-65 insert */
static void orc_insert(orc_tree* t, int32_t ni, uint32_t tri_idx, int cur, int maxd)
{
        const float* tv = t->tri + 9 * (size_t)tri_idx;
        if (!orc_tri_overlaps_aabb(t->nodes[ni].mn, t->nodes[ni].mx, tv))
                return;
        if (t->nodes[ni].child[0] < 0) {
                if (cur == maxd) {
                        orc_node* n = &t->nodes[ni];
                        if (n->nrefs == n->cap) {
                                n->cap = n->cap ? n->cap * 2 : 4;
                                n->refs = (uint32_t*)realloc(n->refs, n->cap * sizeof(uint32_t));
                        }
                        n->refs[n->nrefs++] = tri_idx;
                        return;
                }
                orc_split(t, ni);
        }
        for (int i = 0; i < 8; ++i)
                orc_insert(t, t->nodes[ni].child[i], tri_idx, cur + 1, maxd);
}

/* voxel_octree.cc:67-75 ray_march_init.  nrm may be NULL (geometric normal
 * cross(p1-p0,p2-p0) is used for all three vertices, as the harness does).
 * Normals are normalised once here like the Triangle ctor (voxel_octree.cc:426). */
orc_tree* orc_build(const float* tri, const float* nrm, uint32_t T, int max_depth)
{
        orc_tree* t = (orc_tree*)calloc(1, sizeof(orc_tree));
        t->T = T;
        t->max_depth = max_depth;
        t->tri_own = (float*)malloc(sizeof(float) * 9 * (size_t)(T ? T : 1));
        memcpy(t->tri_own, tri, sizeof(float) * 9 * (size_t)T);
        t->tri = t->tri_own;
        t->nrm = (float*)malloc(sizeof(float) * 9 * (size_t)(T ? T : 1));
        for (uint32_t i = 0; i < T; ++i) {
                const float* p = tri + 9 * (size_t)i;
                float* n = t->nrm + 9 * (size_t)i;
                if (nrm) {
                        memcpy(n, nrm + 9 * (size_t)i, 9 * sizeof(float));
                } else {
                        float a[3] = { p[3] - p[0], p[4] - p[1], p[5] - p[2] };
                        float b[3] = { p[6] - p[0], p[7] - p[1], p[8] - p[2] };
                        float g[3];
                        v3_cross(a, b, g);
                        for (int v = 0; v < 3; ++v)
                                memcpy(n + 3 * v, g, sizeof g);
                }
                for (int v = 0; v < 3; ++v)
                        v3_normalize(n + 3 * v);
        }
        /* root AABB = merge of triangle AABBs from the empty box
         * (graphics_math.h:1228-1266) */
        float mn[3] = { FLT_MAX, FLT_MAX, FLT_MAX };
        float mx[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
        for (uint32_t i = 0; i < T; ++i) {
                const float* p = tri + 9 * (size_t)i;
                float tmn[3] = { FLT_MAX, FLT_MAX, FLT_MAX };
                float tmx[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
                for (int v = 0; v < 3; ++v)
                        for (int k = 0; k < 3; ++k) {
                                tmn[k] = std_minf(tmn[k], p[3 * v + k]);
                                tmx[k] = std_maxf(tmx[k], p[3 * v + k]);
                        }
                for (int k = 0; k < 3; ++k) {
                        mn[k] = std_minf(mn[k], tmn[k]);
                        mx[k] = std_maxf(mx[k], tmx[k]);
                }
        }
        orc_new_node(t, mn, mx);
        for (uint32_t i = 0; i < T; ++i)
                orc_insert(t, 0, i, 1, max_depth);
        return t;
}

void orc_free(orc_tree* t)
{
        if (!t)
                return;
        for (size_t i = 0; i < t->n_nodes; ++i)
                free(t->nodes[i].refs);
        free(t->nodes);
        free(t->nrm);
        free(t->tri_own);
        free(t->uv);
        free(t->tri_mtl);
        free(t->mtl_kd);
        free(t->mtl_tex);
        free(t->tex_whc);
        for (uint32_t i = 0; i < t->n_tex; ++i)
                free(t->tex_data[i]);
        free(t->tex_data);
        free(t);
}

void orc_root_aabb(const orc_tree* t, float out6[6])
{
        memcpy(out6, t->nodes[0].mn, 12);
        memcpy(out6 + 3, t->nodes[0].mx, 12);
}

/* counts: [0]=nodes (incl. empty leaves) [1]=interior [2]=non-empty leaves
 * [3]=tri refs [4]=max refs/leaf [5]=non-empty nodes (interior+non-empty leaves) */
void orc_stats(const orc_tree* t, uint64_t out[6])
{
        memset(out, 0, 6 * sizeof(uint64_t));
        out[0] = t->n_nodes;
        for (size_t i = 0; i < t->n_nodes; ++i) {
                const orc_node* n = &t->nodes[i];
                if (n->child[0] >= 0)
                        out[1]++;
                else if (n->nrefs) {
                        out[2]++;
                        out[3] += n->nrefs;
                        if (n->nrefs > out[4])
                                out[4] = n->nrefs;
                }
        }
        out[5] = out[1] + out[2];
}

static void orc_dump_walk(const orc_tree* t, int32_t ni, uint32_t x, uint32_t y,
                          uint32_t z, uint32_t* cells, uint32_t* counts,
                          uint32_t* refs, float* boxes, uint64_t* nl, uint64_t* nr)
{
        const orc_node* n = &t->nodes[ni];
        if (n->child[0] < 0) {
                if (!n->nrefs)
                        return;
                uint64_t l = (*nl)++;
                cells[3 * l] = x;
                cells[3 * l + 1] = y;
                cells[3 * l + 2] = z;
                counts[l] = n->nrefs;
                if (boxes) {
                        memcpy(boxes + 6 * l, n->mn, 12);
                        memcpy(boxes + 6 * l + 3, n->mx, 12);
                }
                memcpy(refs + *nr, n->refs, n->nrefs * sizeof(uint32_t));
                *nr += n->nrefs;
                return;
        }
        for (int i = 0; i < 8; ++i)
                orc_dump_walk(t, n->child[i], 2 * x + ((i >> 2) & 1),
                              2 * y + ((i >> 1) & 1), 2 * z + (i & 1), cells, counts,
                              refs, boxes, nl, nr);
}

/* Morton-order (child index order) dump of non-empty leaves. */
void orc_dump_leaves(const orc_tree* t, uint32_t* cells, uint32_t* counts,
                     uint32_t* refs, float* boxes)
{
        uint64_t nl = 0, nr = 0;
        orc_dump_walk(t, 0, 0, 0, 0, cells, counts, refs, boxes, &nl, &nr);
}

/* ------------------------------------------------------------------ */
/* Traversal (voxel_octree.cc:77-188) with work counters               */
/* ------------------------------------------------------------------ */

typedef struct {
        uint64_t n_slab;      /* AABB slab tests                          */
        uint64_t n_int;       /* interior nodes expanded (travorder calls) */
        uint64_t n_leaf_all;  /* leaf visits incl. empty                   */
        uint64_t n_leaf;      /* non-empty leaf visits                     */
        uint64_t n_tri;       /* triangle tests                            */
        uint64_t max_stack;
} orc_counters;

/* voxel_octree.cc:77-97: keys dot(d, centre-o); ascending, stable (libstdc++
 * insertion-sorts 8 elements => ties keep ascending child index). */
static void orc_travorder(const orc_tree* t, const orc_node* n, const float* ray,
                          int ord[8])
{
        float key[8];
        for (int i = 0; i < 8; ++i) {
                const orc_node* c = &t->nodes[n->child[i]];
                float s = 0.f;
                for (int k = 0; k < 3; ++k) {
                        float ctr = (c->mn[k] + c->mx[k]) * .5f;
                        s += ray[3 + k] * (ctr - ray[k]);
                }
                key[i] = s;
                ord[i] = i;
        }
        for (int i = 1; i < 8; ++i) { /* stable insertion sort on '<' */
                int ci = ord[i];
                float kv = key[ci];
                int j = i;
                while (j > 0 && kv < key[ord[j - 1]]) {
                        ord[j] = ord[j - 1];
                        --j;
                }
                ord[j] = ci;
        }
}

/* voxel_octree.cc:438-460 Triangle::isect + :99-129 ray_march_isect. */
static int orc_leaf_isect(const orc_tree* t, const orc_node* leaf, const float* ray,
                          uint32_t* tri_out, float hit_out[3], float nrm_out[3],
                          float* t_out, orc_counters* cn)
{
        int found = 0;
        float best = 0.f;
        for (uint32_t i = 0; i < leaf->nrefs; ++i) {
                uint32_t ti = leaf->refs[i];
                const float* p = t->tri + 9 * (size_t)ti;
                double o[3] = { ray[0], ray[1], ray[2] };
                double d[3] = { ray[3], ray[4], ray[5] };
                double a[3] = { p[0], p[1], p[2] };
                double b[3] = { p[3], p[4], p[5] };
                double c[3] = { p[6], p[7], p[8] };
                double dt = 0, du = 0, dv = 0;
                if (cn)
                        cn->n_tri++;
                if (orc_raytri(o, d, a, b, c, &dt, &du, &dv) != 1)
                        continue;
                float hit[3];
                float tf = (float)dt;
                for (int k = 0; k < 3; ++k)
                        hit[k] = ray[k] + tf * ray[3 + k];
                /* depth = length(hit - o)  voxel_octree.cc:114 */
                float s = 0.f;
                for (int k = 0; k < 3; ++k) {
                        float df = hit[k] - ray[k];
                        s += df * df;
                }
                float depth = sqrtf(s);
                /* std::min_element: first minimum wins (strict '<') */
                if (!found || depth < best) {
                        found = 1;
                        best = depth;
                        *tri_out = ti;
                        *t_out = tf;
                        memcpy(hit_out, hit, sizeof hit);
                        float u = (float)du, v = (float)dv;
                        u = u > 1.f ? 1.f : (u < 0.f ? 0.f : u);
                        v = v > 1.f ? 1.f : (v < 0.f ? 0.f : v);
                        float w = 1 - u - v;
                        w = w > 1.f ? 1.f : (w < 0.f ? 0.f : w);
                        const float* n = t->nrm + 9 * (size_t)ti;
                        float nt[3];
                        for (int k = 0; k < 3; ++k)
                                nt[k] = (n[k] * w + n[3 + k] * u) + n[6 + k] * v;
                        v3_normalize(nt);
                        memcpy(nrm_out, nt, sizeof nt);
                }
        }
        return found;
}

/* voxel_octree.cc:131-188 ray_march.  Returns 1 on hit and fills the hit
 * record (cell xyz at level max_depth-1, triangle index, t, hit, normal). */
static int orc_ray_march_ex(const orc_tree* t, const float ray[8], uint32_t cell[3],
                            uint32_t* tri, float* tt, float hit[3], float nrm[3],
                            orc_counters* cn, int32_t* leaf_node);

int orc_ray_march(const orc_tree* t, const float ray[8], uint32_t cell[3],
                  uint32_t* tri, float* tt, float hit[3], float nrm[3],
                  orc_counters* cn)
{
        int32_t leaf = -1;
        return orc_ray_march_ex(t, ray, cell, tri, tt, hit, nrm, cn, &leaf);
}

/* as above; *leaf_node = pool index of the leaf that produced the hit */
static int orc_ray_march_ex(const orc_tree* t, const float ray[8], uint32_t cell[3],
                            uint32_t* tri, float* tt, float hit[3], float nrm[3],
                            orc_counters* cn, int32_t* leaf_node)
{
        const orc_node* root = &t->nodes[0];
        if (cn)
                cn->n_slab++;
        if (!orc_aabb_isect(root->mn, root->mx, ray))
                return 0;
        if (root->child[0] < 0) {
                if (cn) {
                        cn->n_leaf_all++;
                        if (root->nrefs)
                                cn->n_leaf++;
                }
                if (orc_leaf_isect(t, root, ray, tri, hit, nrm, tt, cn)) {
                        cell[0] = cell[1] = cell[2] = 0;
                        *leaf_node = 0;
                        return 1;
                }
                return 0;
        }
        struct {
                int32_t node;
                int ord[8];
                int cur;
                uint32_t x, y, z;
        } st[40];
        int sp = 0;
        st[0].node = 0;
        st[0].cur = 0;
        st[0].x = st[0].y = st[0].z = 0;
        orc_travorder(t, root, ray, st[0].ord);
        if (cn)
                cn->n_int++;
        sp = 1;
        while (sp > 0) {
                if (cn && (uint64_t)sp > cn->max_stack)
                        cn->max_stack = (uint64_t)sp;
                int top = sp - 1;
                int ci = st[top].ord[st[top].cur++];
                int32_t cidx = t->nodes[st[top].node].child[ci];
                uint32_t cx = 2 * st[top].x + ((ci >> 2) & 1);
                uint32_t cy = 2 * st[top].y + ((ci >> 1) & 1);
                uint32_t cz = 2 * st[top].z + (ci & 1);
                if (st[top].cur == 8)
                        sp--; /* popped before the last child is processed */
                const orc_node* c = &t->nodes[cidx];
                if (cn)
                        cn->n_slab++;
                if (!orc_aabb_isect(c->mn, c->mx, ray))
                        continue;
                if (c->child[0] >= 0) {
                        st[sp].node = cidx;
                        st[sp].cur = 0;
                        st[sp].x = cx;
                        st[sp].y = cy;
                        st[sp].z = cz;
                        orc_travorder(t, c, ray, st[sp].ord);
                        if (cn)
                                cn->n_int++;
                        sp++;
                        continue;
                }
                if (cn) {
                        cn->n_leaf_all++;
                        if (c->nrefs)
                                cn->n_leaf++;
                }
                if (orc_leaf_isect(t, c, ray, tri, hit, nrm, tt, cn)) {
                        cell[0] = cx;
                        cell[1] = cy;
                        cell[2] = cz;
                        *leaf_node = cidx;
                        return 1;
                }
        }
        return 0;
}

/* Batch driver.  Outputs may be NULL except hit.  counters may be NULL. */
void orc_trace_rays(const orc_tree* t, const float* rays, uint64_t R, uint8_t* hit,
                    uint32_t* cell, uint32_t* tri, float* tt, float* pos, float* nrm,
                    uint64_t* counters6)
{
        orc_counters cn;
        memset(&cn, 0, sizeof cn);
        for (uint64_t i = 0; i < R; ++i) {
                uint32_t c[3] = { 0xffffffffu, 0xffffffffu, 0xffffffffu };
                uint32_t ti = 0xffffffffu;
                float t1 = 0.f, h[3] = { 0, 0, 0 }, n[3] = { 0, 0, 0 };
                int r = orc_ray_march(t, rays + 8 * i, c, &ti, &t1, h, n,
                                      counters6 ? &cn : NULL);
                if (!r) {
                        c[0] = c[1] = c[2] = 0xffffffffu;
                        ti = 0xffffffffu;
                        t1 = 0.f;
                        memset(h, 0, sizeof h);
                        memset(n, 0, sizeof n);
                }
                hit[i] = (uint8_t)r;
                if (cell)
                        memcpy(cell + 3 * i, c, sizeof c);
                if (tri)
                        tri[i] = ti;
                if (tt)
                        tt[i] = t1;
                if (pos)
                        memcpy(pos + 3 * i, h, sizeof h);
                if (nrm)
                        memcpy(nrm + 3 * i, n, sizeof n);
        }
        if (counters6) {
                counters6[0] = cn.n_slab;
                counters6[1] = cn.n_int;
                counters6[2] = cn.n_leaf_all;
                counters6[3] = cn.n_leaf;
                counters6[4] = cn.n_tri;
                counters6[5] = cn.max_stack;
        }
}

/* ------------------------------------------------------------------ */
/* GI rows of SURVEY.md 8(f): light-map splat (main.cc:75-97), bottom-up */
/* filter and cone trace (voxel_octree.cc:190-303), final pixel          */
/* (main.cc:10-30,117-123).  One untextured material: kd = material_t    */
/* diffuse (voxel_octree.cc:474-476).                                    */
/* ------------------------------------------------------------------ */
static float orc_clampf(float s, float lo, float hi) /* graphics_math.h:905-909 */
{
        return s > hi ? hi : (s < lo ? lo : s);
}

static float orc_dot3(const float a[3], const float b[3]) /* value_sum starts at 0 */
{
        float s = 0.f;
        s += a[0] * b[0];
        s += a[1] * b[1];
        s += a[2] * b[2];
        return s;
}

static const float orc_illum_d[6][3] = { { 1, 0, 0 },  { 0, 1, 0 },  { 0, 0, 1 },
                                         { -1, 0, 0 }, { 0, -1, 0 }, { 0, 0, -1 } }; /* voxel_octree.cc:19-20 */

void orc_gi_reset(orc_tree* t)
{
        for (size_t i = 0; i < t->n_nodes; ++i) {
                t->nodes[i].coverage = 0.f;
                memset(t->nodes[i].illum, 0, sizeof t->nodes[i].illum);
        }
}

/* ------------------------------------------------------------------ */
/* Materials and textures (SURVEY.md 8f row 3)                          */
/* ------------------------------------------------------------------ */
void orc_set_materials(orc_tree* t, const float* tri_uv, const uint32_t* tri_mtl, uint32_t M, const float* kd,
                       const int32_t* mtl_tex, uint32_t n_tex, const int32_t* tex_whc, const uint8_t* const* tex_data)
{
        t->uv = (float*)malloc(sizeof(float) * 6 * (size_t)(t->T ? t->T : 1));
        memcpy(t->uv, tri_uv, sizeof(float) * 6 * (size_t)t->T);
        t->tri_mtl = (uint32_t*)malloc(sizeof(uint32_t) * (size_t)(t->T ? t->T : 1));
        memcpy(t->tri_mtl, tri_mtl, sizeof(uint32_t) * (size_t)t->T);
        t->n_mtl = M;
        t->mtl_kd = (float*)malloc(sizeof(float) * 3 * (size_t)(M ? M : 1));
        memcpy(t->mtl_kd, kd, sizeof(float) * 3 * (size_t)M);
        t->mtl_tex = (int32_t*)malloc(sizeof(int32_t) * (size_t)(M ? M : 1));
        memcpy(t->mtl_tex, mtl_tex, sizeof(int32_t) * (size_t)M);
        t->n_tex = n_tex;
        t->tex_whc = (int32_t*)malloc(sizeof(int32_t) * 3 * (size_t)(n_tex ? n_tex : 1));
        memcpy(t->tex_whc, tex_whc, sizeof(int32_t) * 3 * (size_t)n_tex);
        t->tex_data = (uint8_t**)malloc(sizeof(uint8_t*) * (size_t)(n_tex ? n_tex : 1));
        for (uint32_t i = 0; i < n_tex; ++i) {
                size_t sz = (size_t)tex_whc[3 * i] * tex_whc[3 * i + 1] * tex_whc[3 * i + 2];
                t->tex_data[i] = (uint8_t*)malloc(sz ? sz : 1);
                memcpy(t->tex_data[i], tex_data[i], sz);
        }
}

static float orc_unit_cycle(float s) /* voxel_octree.cc:392-399 */
{
        while (s > 1.f)
                s -= 1.f;
        while (s < 0.f)
                s += 1.f;
        return s;
}

static int orc_clampi(int s, int lo, int hi)
{
        return s > hi ? hi : (s < lo ? lo : s);
}

/* Triangle::get_albedo voxel_octree.cc:471-484 with barycentric graphics_math.h:1082-1100 and
 * texel_fetch voxel_octree.cc:401-422.  kd_default: the colour used when no materials are set. */
static void orc_albedo_one(const orc_tree* t, uint32_t tri, const float hit[3], const float kd_default[3], float out[3])
{
        if (!t->tri_mtl) {
                memcpy(out, kd_default, 3 * sizeof(float));
                return;
        }
        const uint32_t m = t->tri_mtl[tri];
        const int32_t tx = t->mtl_tex[m];
        if (tx < 0) {
                memcpy(out, t->mtl_kd + 3 * (size_t)m, 3 * sizeof(float));
                return;
        }
        const float* p = t->tri + 9 * (size_t)tri;
        float v0[3], v1[3], v2[3];
        for (int k = 0; k < 3; ++k) {
                v0[k] = p[3 + k] - p[k];
                v1[k] = p[6 + k] - p[k];
                v2[k] = hit[k] - p[k];
        }
        float d00 = orc_dot3(v0, v0), d01 = orc_dot3(v0, v1), d11 = orc_dot3(v1, v1);
        float d20 = orc_dot3(v2, v0), d21 = orc_dot3(v2, v1);
        float denom = d00 * d11 - d01 * d01;
        float bc[3] = { 0.f, 0.f, 0.f };
        if (denom != 0) {
                bc[1] = (d11 * d20 - d01 * d21) / denom;
                bc[2] = (d00 * d21 - d01 * d20) / denom;
                bc[0] = 1.0f - bc[1] - bc[2];
        }
        for (int k = 0; k < 3; ++k)
                bc[k] = orc_clampf(bc[k], 0.f, 1.f);
        const float* uv = t->uv + 6 * (size_t)tri;
        float tc[2];
        for (int k = 0; k < 2; ++k)
                tc[k] = (bc[0] * uv[k] + bc[1] * uv[2 + k]) + bc[2] * uv[4 + k];
        const int w = t->tex_whc[3 * tx], h = t->tex_whc[3 * tx + 1], ch = t->tex_whc[3 * tx + 2];
        int x = orc_clampi((int)(orc_unit_cycle(tc[0]) * w), 0, w - 1);
        int y = orc_clampi((int)(orc_unit_cycle(tc[1]) * h), 0, h - 1);
        y = h - 1 - y;
        const uint8_t* px = t->tex_data[tx] + ((size_t)y * w + x) * ch;
        float pixel[4] = { 0, 0, 0, 0 };
        for (int k = 0; k < ch && k < 4; ++k)
                pixel[k] = (float)px[k];
        for (int k = 0; k < 3; ++k)
                out[k] = pixel[k] / 255.f;
}

void orc_albedo(const orc_tree* t, const uint32_t* tri, const float* pos, uint64_t n, const float kd_default[3], float* out3)
{
        for (uint64_t i = 0; i < n; ++i)
                orc_albedo_one(t, tri[i], pos + 3 * i, kd_default, out3 + 3 * i);
}

/* main.cc:81-96, sequential in pixel order (py outer, px inner, samples in order). */
void orc_gi_splat(orc_tree* t, const float cam10[10], float film_h, int nx, int ny, int spp,
                  const float kd[3])
{
        float C[16];
        orc_camera_matrix(cam10, C);
        const float z = orc_camera_z(cam10[0], film_h);
        for (int py = 0; py < ny; ++py)
                for (int px = 0; px < nx; ++px) {
                        float rays[4 * 8];
                        orc_gen_rays_pixel(C, z, nx, ny, spp, px, py, rays);
                        for (int s = 0; s < spp; ++s) {
                                const float* ray = rays + 8 * s;
                                uint32_t cell[3], tri;
                                float tt, hit[3], n[3];
                                int32_t leaf = -1;
                                if (!orc_ray_march_ex(t, ray, cell, &tri, &tt, hit, n, NULL, &leaf))
                                        continue;
                                /* Triangle::get_diffuse voxel_octree.cc:462-469: albedo * tmp * color(1,1,1) */
                                const float nd[3] = { -ray[3], -ray[4], -ray[5] };
                                float tmp = orc_clampf(orc_dot3(n, nd), 0.f, 1.f);
                                float illum[3], albedo[3];
                                orc_albedo_one(t, tri, hit, kd, albedo);
                                for (int k = 0; k < 3; ++k)
                                        illum[k] = (albedo[k] * tmp) * 1.f;
                                orc_node* ln = &t->nodes[leaf];
                                for (int i = 0; i < 6; ++i) {
                                        float coeff = orc_clampf(orc_dot3(orc_illum_d[i], n), 0.f, 1.f);
                                        for (int k = 0; k < 3; ++k)
                                                ln->illum[3 * i + k] += coeff * illum[k];
                                }
                        }
                }
}

/* voxel_octree.cc:190-214 cone_trace_init_filter */
static void orc_gi_filter_node(orc_tree* t, int32_t ni)
{
        orc_node* n = &t->nodes[ni];
        if (n->child[0] < 0) {
                if (n->nrefs == 0) {
                        n->coverage = 0.f;
                        memset(n->illum, 0, sizeof n->illum);
                        return;
                }
                n->coverage = 1.f;
                return;
        }
        float cov = 0.f, il[18];
        memset(il, 0, sizeof il);
        for (int i = 0; i < 8; ++i) {
                orc_gi_filter_node(t, t->nodes[ni].child[i]);
                const orc_node* c = &t->nodes[t->nodes[ni].child[i]];
                cov += c->coverage;
                for (int f = 0; f < 18; ++f)
                        il[f] += c->illum[f];
        }
        n = &t->nodes[ni];
        for (int f = 0; f < 18; ++f)
                n->illum[f] = il[f] / 8;
        n->coverage = cov / 8.f;
}

void orc_gi_filter(orc_tree* t)
{
        if (t->n_nodes)
                orc_gi_filter_node(t, 0);
}

typedef struct {
        int level;
        uint32_t* cells;
        float* cov;
        float* illum;
        uint64_t cap, n;
} orc_gi_dump;

static void orc_gi_dump_walk(const orc_tree* t, int32_t ni, uint32_t x, uint32_t y, uint32_t z, int level,
                             orc_gi_dump* d)
{
        const orc_node* n = &t->nodes[ni];
        if (level == d->level) {
                if (n->coverage > 0.f) {
                        if (d->n < d->cap) {
                                if (d->cells) {
                                        d->cells[3 * d->n] = x;
                                        d->cells[3 * d->n + 1] = y;
                                        d->cells[3 * d->n + 2] = z;
                                }
                                if (d->cov)
                                        d->cov[d->n] = n->coverage;
                                if (d->illum)
                                        memcpy(d->illum + 18 * d->n, n->illum, sizeof n->illum);
                        }
                        d->n++;
                }
                return;
        }
        if (n->child[0] < 0)
                return;
        for (int i = 0; i < 8; ++i)
                orc_gi_dump_walk(t, n->child[i], 2 * x + ((i >> 2) & 1), 2 * y + ((i >> 1) & 1), 2 * z + (i & 1),
                                 level + 1, d);
}

/* nodes of level `level` with coverage > 0 in Morton order; returns their number */
uint64_t orc_gi_dump_level(const orc_tree* t, int level, uint32_t* cells, float* cov, float* illum18,
                           uint64_t cap)
{
        orc_gi_dump d = { level, cells, cov, illum18, cap, 0 };
        if (t->n_nodes)
                orc_gi_dump_walk(t, 0, 0, 0, 0, 0, &d);
        return d.n;
}

/* VoxelOctree::compute_illum voxel_octree.h:71-81 */
static void orc_compute_illum(const orc_node* n, const float d[3], float out[3])
{
        out[0] = out[1] = out[2] = 0.f;
        for (int i = 0; i < 6; ++i) {
                float coeff = orc_clampf(orc_dot3(orc_illum_d[i], d), 0.f, 1.f);
                for (int k = 0; k < 3; ++k)
                        out[k] += coeff * n->illum[3 * i + k];
        }
}

/* voxel_octree.cc:247-283 cone_trace(root, cone, min_voxel_size); aperture .577350269f, step .1f,
 * litness_decay 1.f (voxel_octree.cc:216-225) */
/* Work counters of the reference's cone trace (bench.py's roofline entry of the GI film): samples taken along the
 * cones, descent steps of their point locations (one node record each), samples that reach their level and read
 * the node's coverage + illum[6] (76 bytes).  Plain globals: the counting run is single-threaded. */
static uint64_t g_cone_counts[3];
void orc_gi_counters_reset(void) { memset(g_cone_counts, 0, sizeof g_cone_counts); }
void orc_gi_counters(uint64_t out[3]) { memcpy(out, g_cone_counts, sizeof g_cone_counts); }

/* split_level = (int)log2f(x) with libm's log2f (the reference's own expression; default), or -- exact mode -- with
 * the correctly rounded log2f, (float)log2((double)x): the definition the device evaluates in closed form
 * (vrt_gi.cuh gi_split_level), so that the GPU's cone trace can be compared bit for bit. */
static int g_exact_log2;
void orc_gi_set_exact_log2(int on) { g_exact_log2 = on != 0; }

static void orc_cone_trace_one(const orc_tree* t, const float o[3], const float d[3], float min_voxel_size,
                               float out[3])
{
        const float aperture = 0.577350269f, step = .1f, decay = 1.f;
        const orc_node* root = &t->nodes[0];
        float mindist = 1.414f * min_voxel_size;
        float sz[3] = { root->mx[0] - root->mn[0], root->mx[1] - root->mn[1], root->mx[2] - root->mn[2] };
        float maxdist = sqrtf(orc_dot3(sz, sz));
        float dist = mindist, opacity = 0.f;
        float diffuse[3] = { 0, 0, 0 };
        const float nd[3] = { -d[0], -d[1], -d[2] };
        while (dist < maxdist && opacity < 1.f) {
                float p[3] = { o[0] + d[0] * dist, o[1] + d[1] * dist, o[2] + d[2] * dist };
                float diam = std_maxf(mindist, aperture * 2.f * dist);
                if (maxdist < diam)
                        break;
                const float ratio = maxdist / diam;
                int split_level = g_exact_log2 ? (int)(float)log2((double)ratio) : (int)log2f(ratio);
                const orc_node* tree = root;
                g_cone_counts[0]++;
                while (tree->child[0] >= 0 && split_level) {
                        g_cone_counts[1]++;
                        int i = 0;
                        i += (p[0] > (tree->mn[0] + tree->mx[0]) * .5f ? 4 : 0);
                        i += (p[1] > (tree->mn[1] + tree->mx[1]) * .5f ? 2 : 0);
                        i += (p[2] > (tree->mn[2] + tree->mx[2]) * .5f ? 1 : 0);
                        tree = &t->nodes[tree->child[i]];
                        split_level--;
                }
                if (split_level == 0) {
                        float illum[3];
                        g_cone_counts[2]++;
                        orc_compute_illum(tree, nd, illum);
                        float transparency = orc_clampf(1.f - opacity, 0.f, 1.f);
                        float a = tree->coverage * step;
                        float w = ((1.f / (1 + decay * dist)) * transparency) * tree->coverage;
                        for (int k = 0; k < 3; ++k)
                                diffuse[k] += w * illum[k];
                        opacity += transparency * a;
                }
                dist += step * diam;
        }
        memcpy(out, diffuse, sizeof diffuse);
}

/* voxel_octree.cc:227-245 HemiCones + orthonormal_basis, :285-303 cone_trace(root, isect, res) */
void orc_gi_cone_trace_point(const orc_tree* t, const float pos[3], const float n[3], float res, float out[3])
{
        static const float hemi[6][4] = {
                { 0.000000f, 0.000000f, 1.0f, 0.25f },   { 0.000000f, 0.866025f, 0.5f, 0.15f },
                { 0.823639f, 0.267617f, 0.5f, 0.15f },   { 0.509037f, -0.700629f, 0.5f, 0.15f },
                { -0.509037f, -0.700629f, 0.5f, 0.15f }, { -0.823639f, 0.267617f, 0.5f, 0.15f },
        };
        float s = (0.0f > n[2]) ? -1.0f : 1.0f;
        float a0 = -1.0f / (s + n[2]);
        float a1 = n[0] * n[1] * a0;
        float tv[3] = { 1.0f + s * n[0] * n[0] * a0, s * a1, -s * n[0] };
        float bv[3] = { a1, s + n[1] * n[1] * a0, -n[1] };
        float diffuse[3] = { 0, 0, 0 };
        for (int i = 0; i < 6; ++i) {
                float d[3];
                for (int k = 0; k < 3; ++k) { /* dot(Mat3{t,b,n}, d): result += column * v[i] */
                        float r = 0.f;
                        r += tv[k] * hemi[i][0];
                        r += bv[k] * hemi[i][1];
                        r += n[k] * hemi[i][2];
                        d[k] = r;
                }
                v3_normalize(d);
                float c[3];
                orc_cone_trace_one(t, pos, d, res, c);
                for (int k = 0; k < 3; ++k)
                        diffuse[k] += hemi[i][3] * c[k];
        }
        memcpy(out, diffuse, sizeof diffuse);
}

void orc_gi_cone_trace(const orc_tree* t, const float* pos, const float* nrm, uint64_t n, float res, float* out3)
{
        for (uint64_t i = 0; i < n; ++i)
                orc_gi_cone_trace_point(t, pos + 3 * i, nrm + 3 * i, res, out3 + 3 * i);
}

/* main.cc:10-30 trace() + :117-123: film[py][px] = sum over samples of colour * (1/spp) */
void orc_gi_render(const orc_tree* t, const float cam10[10], float film_h, int nx, int ny, int spp, float res,
                   const float kd[3], float* film3)
{
        float C[16];
        orc_camera_matrix(cam10, C);
        const float z = orc_camera_z(cam10[0], film_h);
        const float w = (spp == 4) ? .25f : 1.f;
        for (int py = 0; py < ny; ++py)
                for (int px = 0; px < nx; ++px) {
                        float rays[4 * 8];
                        float acc[3] = { 0, 0, 0 };
                        orc_gen_rays_pixel(C, z, nx, ny, spp, px, py, rays);
                        for (int s = 0; s < spp; ++s) {
                                const float* ray = rays + 8 * s;
                                uint32_t cell[3], tri;
                                float tt, hit[3], n[3], c[3];
                                int32_t leaf = -1;
                                if (!orc_ray_march_ex(t, ray, cell, &tri, &tt, hit, n, NULL, &leaf)) {
                                        float tl = (float)(0.5 * ((double)ray[4] + 1.0));
                                        const float v1[3] = { 0.6f, 0.8f, 1.0f };
                                        for (int k = 0; k < 3; ++k)
                                                c[k] = 1.0f + (v1[k] - 1.0f) * tl;
                                } else {
                                        float ind[3], dir[3], albedo[3];
                                        const float nd[3] = { -ray[3], -ray[4], -ray[5] };
                                        orc_gi_cone_trace_point(t, hit, n, res, ind);
                                        orc_compute_illum(&t->nodes[leaf], nd, dir);
                                        orc_albedo_one(t, tri, hit, kd, albedo);
                                        for (int k = 0; k < 3; ++k)
                                                c[k] = albedo[k] * (ind[k] + dir[k]);
                                }
                                for (int k = 0; k < 3; ++k)
                                        acc[k] += c[k] * w;
                        }
                        memcpy(film3 + 3 * ((size_t)py * nx + px), acc, sizeof acc);
                }
}

/* Batch predicate entry points for the KATs. */
void orc_tribox_batch(const float* centers, const float* halves, const float* tris,
                      uint64_t n, uint8_t* out)
{
        for (uint64_t i = 0; i < n; ++i)
                out[i] = (uint8_t)orc_tribox(centers + 3 * i, halves + 3 * i, tris + 9 * i);
}

void orc_tri_overlap_aabb_batch(const float* aabbs6, const float* tris, uint64_t n,
                                uint8_t* out)
{
        for (uint64_t i = 0; i < n; ++i)
                out[i] = (uint8_t)orc_tri_overlaps_aabb(aabbs6 + 6 * i, aabbs6 + 6 * i + 3,
                                                        tris + 9 * i);
}

void orc_raytri_batch(const double* in, uint64_t n, uint8_t* res, double* tuv)
{
        for (uint64_t i = 0; i < n; ++i) {
                const double* a = in + 15 * i;
                double t = 0, u = 0, v = 0;
                res[i] = (uint8_t)orc_raytri(a, a + 3, a + 6, a + 9, a + 12, &t, &u, &v);
                tuv[3 * i] = t;
                tuv[3 * i + 1] = u;
                tuv[3 * i + 2] = v;
        }
}

void orc_aabb_isect_batch(const float* aabbs6, const float* rays8, uint64_t n,
                          uint8_t* out)
{
        for (uint64_t i = 0; i < n; ++i)
                out[i] = (uint8_t)orc_aabb_isect(aabbs6 + 6 * i, aabbs6 + 6 * i + 3,
                                                 rays8 + 8 * i);
}

/* ------------------------------------------------------------------ */
/* Film export (what the reference does with its float film)           */
/* ------------------------------------------------------------------ */

/* `(unsigned char)f` / static_cast<std::uint8_t>(f) as x86-64 compiles it: CVTTSS2SI to int32 (0x80000000 when the
 * value does not fit or is NaN), low byte.  Written out so that the oracle does not depend on what THIS compiler
 * makes of an out-of-range conversion. */
static uint8_t orc_f2u8(float f)
{
        int32_t i = (fabsf(f) < 2147483648.0f) ? (int32_t)f : INT32_MIN;
        return (uint8_t)((uint32_t)i & 0xffu);
}

/* Film::to_byte_array camera.cc:27-48: v = rawv * 255.9f, each component cast to uint8. */
void orc_film_rgb8(const float* rgb, uint64_t npix, uint8_t* out)
{
        for (uint64_t i = 0; i < 3 * npix; ++i)
                out[i] = orc_f2u8(rgb[i] * 255.9f);
}

/* stbiw__linear_to_rgbe stb_image_write.h:601-616 (stbiw__max is the `a > b ? a : b` macro). */
static void orc_linear_to_rgbe(uint8_t rgbe[4], const float linear[3])
{
        float m12 = linear[1] > linear[2] ? linear[1] : linear[2];
        float maxcomp = linear[0] > m12 ? linear[0] : m12;
        if (maxcomp < 1e-32f) {
                rgbe[0] = rgbe[1] = rgbe[2] = rgbe[3] = 0;
        } else {
                int exponent;
                float normalize = (float)frexp(maxcomp, &exponent) * 256.0f / maxcomp;
                rgbe[0] = orc_f2u8(linear[0] * normalize);
                rgbe[1] = orc_f2u8(linear[1] * normalize);
                rgbe[2] = orc_f2u8(linear[2] * normalize);
                rgbe[3] = (uint8_t)(exponent + 128);
        }
}

void orc_film_rgbe(const float* rgb, uint64_t npix, uint8_t* out)
{
        for (uint64_t i = 0; i < npix; ++i)
                orc_linear_to_rgbe(out + 4 * i, rgb + 3 * i);
}
