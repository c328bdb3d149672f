/*
 * daisy_oracle.c -- CPU restatement of the DaisyRiot hot path (see daisy_oracle.h).
 * TEST INFRASTRUCTURE ONLY -- never linked into or called by the product library.
 *
 * Build: gcc -O2 -std=c11 -ffp-contract=off -fno-fast-math -fopenmp -shared -fPIC
 * (FMA contraction must stay off: the reference was built by MSVC 2013 /fp:precise for x64,
 *  i.e. scalar SSE2 mul/add, and the CUDA product mirrors that with __fmul_rn/__fadd_rn.)
 */
#include "daisy_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct { float x, y, z; } v3;

/* ---- glm 0.9.8.4 restatements (R/libraries/glm/glm/detail/func_geometric.inl) ---------- */
static inline v3 ld3(const float *p) { v3 r = { p[0], p[1], p[2] }; return r; }
static inline v3 v_add(v3 a, v3 b) { v3 r = { a.x + b.x, a.y + b.y, a.z + b.z }; return r; }
static inline v3 v_sub(v3 a, v3 b) { v3 r = { a.x - b.x, a.y - b.y, a.z - b.z }; return r; }
static inline v3 v_mul(v3 a, float s) { v3 r = { a.x * s, a.y * s, a.z * s }; return r; }
static inline v3 v_div(v3 a, float s) { v3 r = { a.x / s, a.y / s, a.z / s }; return r; }
/* compute_dot<tvec3>: tmp = x*y; tmp.x + tmp.y + tmp.z           func_geometric.inl:54-61 */
static inline float v_dot(v3 a, v3 b) { float tx = a.x * b.x, ty = a.y * b.y, tz = a.z * b.z; return (tx + ty) + tz; }
/* compute_cross                                                   func_geometric.inl:74-85 */
static inline v3 v_cross(v3 x, v3 y) {
    v3 r = { x.y * y.z - y.y * x.z, x.z * y.x - y.z * x.x, x.x * y.y - y.x * x.y };
    return r;
}
static inline float v_length(v3 a) { return sqrtf(v_dot(a, a)); }
/* normalize = v * inversesqrt(dot(v,v)), inversesqrt = 1/sqrt      func_geometric.inl:88-95 */
static inline v3 v_normalize(v3 a) { float inv = 1.0f / sqrtf(v_dot(a, a)); return v_mul(a, inv); }

static inline void tri_verts(const orc_mesh *m, int tri, v3 *a, v3 *b, v3 *c) {
    const int *t = m->tri + 6 * (int64_t)tri;
    *a = ld3(m->vertices + 3 * (int64_t)t[0]);
    *b = ld3(m->vertices + 3 * (int64_t)t[1]);
    *c = ld3(m->vertices + 3 * (int64_t)t[2]);
}

/* VS/triangle_math.cpp:31-35 / VS/parallellism.cu:209-214: 0.5 is a double literal */
static inline float surface3(v3 a, v3 b, v3 c) {
    v3 ab = v_sub(b, a), ac = v_sub(c, a);
    return (float)(0.5 * (double)v_length(v_cross(ab, ac)));
}
float orc_surface3(const float *a, const float *b, const float *c) { return surface3(ld3(a), ld3(b), ld3(c)); }
float orc_surface_tri(const orc_mesh *m, int tri) { v3 a, b, c; tri_verts(m, tri, &a, &b, &c); return surface3(a, b, c); }

/* VS/triangle_math.cpp:11-21: (p0+p1+p2) then each component / 3 */
static inline v3 centre3(v3 a, v3 b, v3 c) {
    v3 s = v_add(v_add(a, b), c);
    v3 r = { s.x / 3, s.y / 3, s.z / 3 };
    return r;
}
void orc_centre_tri(const orc_mesh *m, int tri, float out[3]) {
    v3 a, b, c; tri_verts(m, tri, &a, &b, &c);
    v3 r = centre3(a, b, c); out[0] = r.x; out[1] = r.y; out[2] = r.z;
}

/* VS/triangle_math.cpp:23-29 */
static inline v3 avg_normal(const orc_mesh *m, int tri) {
    const int *t = m->tri + 6 * (int64_t)tri;
    v3 n0 = ld3(m->normals + 3 * (int64_t)t[3]), n1 = ld3(m->normals + 3 * (int64_t)t[4]), n2 = ld3(m->normals + 3 * (int64_t)t[5]);
    v3 s = v_add(v_add(n0, n1), n2);
    v3 avg = { s.x / 3, s.y / 3, s.z / 3 };
    return v_normalize(avg);
}
void orc_avg_normal(const orc_mesh *m, int tri, float out[3]) { v3 n = avg_normal(m, tri); out[0] = n.x; out[1] = n.y; out[2] = n.z; }

/* VS/triangle_math.cpp:60-74 */
static inline void divide4(const orc_mesh *m, int tri, v3 out[4][3]) {
    v3 a, b, c; tri_verts(m, tri, &a, &b, &c);
    v3 innerA = v_add(v_div(v_sub(b, a), 2.0f), a);
    v3 innerC = v_add(v_div(v_sub(c, a), 2.0f), a);
    v3 innerB = v_add(v_div(v_sub(b, c), 2.0f), c);
    out[0][0] = a;      out[0][1] = innerC; out[0][2] = innerA;
    out[1][0] = innerC; out[1][1] = c;      out[1][2] = innerB;
    out[2][0] = innerA; out[2][1] = innerB; out[2][2] = b;
    out[3][0] = innerA; out[3][1] = innerB; out[3][2] = innerC;
}
void orc_divide4(const orc_mesh *m, int tri, float out[4][3][3]) {
    v3 t[4][3]; divide4(m, tri, t);
    for (int i = 0; i < 4; i++) for (int j = 0; j < 3; j++) { out[i][j][0] = t[i][j].x; out[i][j][1] = t[i][j].y; out[i][j][2] = t[i][j].z; }
}

/* VS/triangle_math.cpp:3-9: a + u*(b-a) + v*(c-a) */
static inline v3 uv2xyz(const orc_mesh *m, int tri, float u, float v) {
    v3 a, b, c; tri_verts(m, tri, &a, &b, &c);
    return v_add(v_add(a, v_mul(v_sub(b, a), u)), v_mul(v_sub(c, a), v));
}
void orc_uv2xyz(const orc_mesh *m, int tri, float u, float v, float out[3]) { v3 p = uv2xyz(m, tri, u, v); out[0] = p.x; out[1] = p.y; out[2] = p.z; }

/* VS/parallellism.cu:197-207 (device: CUDART_PI is double) / VS/triangle_math.cpp:49-58 (host: M_PIf) */
static inline float point_ff(v3 opos, v3 onrm, v3 dpos, v3 dnrm, float surface, int variant) {
    float formfactor = 0;
    float dot1 = v_dot(onrm, v_normalize(v_sub(dpos, opos)));
    float dot2 = v_dot(dnrm, v_normalize(v_sub(opos, dpos)));
    if (dot1 > 0 && dot2 > 0) {
        float length = v_length(v_sub(dpos, opos));
        float len2 = length * length; /* powf(length, 2): nvcc folds to x*x (no lg2/ex2 in the PTX); exact in libm too */
        if (variant == ORC_FF_DEVICE) {
            double den = (double)len2 * 3.14159265358979323846;
            formfactor = (float)((((double)(dot1 * dot2)) / den) * (double)surface);
        } else {
            const float pif = 3.14159265358979323846f;
            formfactor = ((dot1 * dot2) / (len2 * pif)) * surface;
        }
    }
    return formfactor;
}
float orc_point_ff(const float opos[3], const float onrm[3], const float dpos[3], const float dnrm[3], float surface, int variant) {
    return point_ff(ld3(opos), ld3(onrm), ld3(dpos), ld3(dnrm), surface, variant);
}

/* VS/parallellism.cu:113-151 == VS/OptixPrimeFunctionality.cpp:133-161 */
float orc_p2p_ff(const orc_mesh *m, int origin, int dest, int variant) {
    v3 ot[4][3], dt[4][3];
    divide4(m, origin, ot);
    divide4(m, dest, dt);
    v3 on = avg_normal(m, origin), dn = avg_normal(m, dest);
    v3 op[4], dp[4];
    for (int i = 0; i < 4; i++) { op[i] = centre3(ot[i][0], ot[i][1], ot[i][2]); dp[i] = centre3(dt[i][0], dt[i][1], dt[i][2]); }
    float formfactor = 0;
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) {
            float surface = surface3(ot[i][0], ot[i][1], ot[i][2]) * surface3(dt[j][0], dt[j][1], dt[j][2]);
            formfactor = formfactor + point_ff(op[i], on, dp[j], dn, surface, variant);
        }
    formfactor = formfactor / orc_surface_tri(m, origin);
    return formfactor;
}

/* VS/parallellism.cu:91-111: value stored only when > 0, else 0 (NaN on the diagonal -> 0) */
void orc_unoccluded_rows(const orc_mesh *m, int row0, int row1, int variant, float *out) {
    int N = m->ntri;
#pragma omp parallel for schedule(dynamic, 4)
    for (int r = row0; r < row1; r++)
        for (int c = 0; c < N; c++) {
            float f = orc_p2p_ff(m, r, c, variant);
            out[(int64_t)(r - row0) * N + c] = (f > 0.0) ? f : 0.0f;
        }
}

/* VS/OptixPrimeFunctionality.cpp:191-196; optix::normalize = v * (1/sqrtf(dot)), dot = x+y+z order */
void orc_pair_ray(const orc_mesh *m, int origin, int dest, float u, float v, float ray6[6]) {
    v3 o = uv2xyz(m, origin, u, v), d = uv2xyz(m, dest, u, v);
    v3 dir = v_normalize(v_sub(d, o));
    v3 org = v_add(o, v_mul(dir, 0.000001f));
    ray6[0] = org.x; ray6[1] = org.y; ray6[2] = org.z; ray6[3] = dir.x; ray6[4] = dir.y; ray6[5] = dir.z;
}

/* ---- closest hit: PARITY UNPINNED (OptiX Prime is closed source) -------------------------- */
typedef struct { int kx, ky, kz; float Sx, Sy, Sz; v3 o; } wray;

static inline void wray_setup(const float r[6], wray *w) {
    float ax = fabsf(r[3]), ay = fabsf(r[4]), az = fabsf(r[5]);
    int kz = (ax >= ay && ax >= az) ? 0 : ((ay >= az) ? 1 : 2);
    int kx = (kz + 1) % 3, ky = (kx + 1) % 3;
    if (r[3 + kz] < 0.0f) { int t = kx; kx = ky; ky = t; }
    w->kx = kx; w->ky = ky; w->kz = kz;
    w->Sx = r[3 + kx] / r[3 + kz];
    w->Sy = r[3 + ky] / r[3 + kz];
    w->Sz = 1.0f / r[3 + kz];
    w->o = ld3(r);
}

/* Woop, Benthin, Wald: "Watertight Ray/Triangle Intersection", JCGT 2(1) 2013, listing 2,
 * no culling, t computed with an IEEE division.  u,v = weights of vertices 1 and 2. */
static inline int wray_tri(const wray *w, v3 va, v3 vb, v3 vc, float *t, float *u, float *v) {
    v3 A = v_sub(va, w->o), B = v_sub(vb, w->o), C = v_sub(vc, w->o);
    const float *Ap = &A.x, *Bp = &B.x, *Cp = &C.x;
    float Ax = Ap[w->kx] - w->Sx * Ap[w->kz], Ay = Ap[w->ky] - w->Sy * Ap[w->kz];
    float Bx = Bp[w->kx] - w->Sx * Bp[w->kz], By = Bp[w->ky] - w->Sy * Bp[w->kz];
    float Cx = Cp[w->kx] - w->Sx * Cp[w->kz], Cy = Cp[w->ky] - w->Sy * Cp[w->kz];
    float U = Cx * By - Cy * Bx;
    float V = Ax * Cy - Ay * Cx;
    float W = Bx * Ay - By * Ax;
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        double CxBy = (double)Cx * (double)By, CyBx = (double)Cy * (double)Bx;
        U = (float)(CxBy - CyBx);
        double AxCy = (double)Ax * (double)Cy, AyCx = (double)Ay * (double)Cx;
        V = (float)(AxCy - AyCx);
        double BxAy = (double)Bx * (double)Ay, ByAx = (double)By * (double)Ax;
        W = (float)(BxAy - ByAx);
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return 0;
    float det = (U + V) + W;
    if (det == 0.0f) return 0;
    float Az = w->Sz * Ap[w->kz], Bz = w->Sz * Bp[w->kz], Cz = w->Sz * Cp[w->kz];
    float T = (U * Az + V * Bz) + W * Cz;
    float tt = T / det;
    if (!(tt > 0.0f) || isinf(tt)) return 0; /* NaN, <=0, inf -> miss */
    *t = tt; *u = V / det; *v = W / det;
    return 1;
}
int orc_ray_tri(const float ray6[6], const float *a, const float *b, const float *c, float *t, float *u, float *v) {
    wray w; wray_setup(ray6, &w);
    return wray_tri(&w, ld3(a), ld3(b), ld3(c), t, u, v);
}

/* (t, id) lexicographic minimum makes the result independent of the order triangles are visited */
static inline void hit_update(orc_hit *best, float t, int id, float u, float v) {
    if (best->triangleId < 0 || t < best->t || (t == best->t && id < best->triangleId)) {
        best->t = t; best->triangleId = id; best->u = u; best->v = v;
    }
}

void orc_query_closest_brute(const orc_mesh *m, int n, const float *rays6, orc_hit *hits) {
#pragma omp parallel for schedule(dynamic, 16)
    for (int i = 0; i < n; i++) {
        wray w; wray_setup(rays6 + 6 * (int64_t)i, &w);
        orc_hit best = { -1.0f, -1, 0.0f, 0.0f };
        for (int k = 0; k < m->ntri; k++) {
            v3 a, b, c; tri_verts(m, k, &a, &b, &c);
            float t, u, v;
            if (wray_tri(&w, a, b, c, &t, &u, &v)) hit_update(&best, t, k, u, v);
        }
        hits[i] = best;
    }
}

/* ---- a small median-split BVH (any conservative hierarchy gives the same answer) ---------- */
typedef struct { float lo[3], hi[3]; int left, right, first, count; } bnode;
struct orc_bvh { bnode *nodes; int nnodes; int *order; float pad; };

static void tri_box(const orc_mesh *m, int k, float lo[3], float hi[3]) {
    v3 a, b, c; tri_verts(m, k, &a, &b, &c);
    lo[0] = fminf(a.x, fminf(b.x, c.x)); hi[0] = fmaxf(a.x, fmaxf(b.x, c.x));
    lo[1] = fminf(a.y, fminf(b.y, c.y)); hi[1] = fmaxf(a.y, fmaxf(b.y, c.y));
    lo[2] = fminf(a.z, fminf(b.z, c.z)); hi[2] = fmaxf(a.z, fmaxf(b.z, c.z));
}

typedef struct { const orc_mesh *m; float *cent; } sortctx;
static int g_axis; static const float *g_cent;
static int cmp_axis(const void *pa, const void *pb) {
    int a = *(const int *)pa, b = *(const int *)pb;
    float ca = g_cent[3 * (int64_t)a + g_axis], cb = g_cent[3 * (int64_t)b + g_axis];
    return (ca < cb) ? -1 : (ca > cb) ? 1 : (a - b);
}

static int build_rec(orc_bvh *bv, const orc_mesh *m, const float *cent, int first, int count) {
    int id = bv->nnodes++;
    bnode *nd = &bv->nodes[id];
    for (int d = 0; d < 3; d++) { nd->lo[d] = INFINITY; nd->hi[d] = -INFINITY; }
    float clo[3] = { INFINITY, INFINITY, INFINITY }, chi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int i = first; i < first + count; i++) {
        float lo[3], hi[3]; tri_box(m, bv->order[i], lo, hi);
        for (int d = 0; d < 3; d++) {
            nd->lo[d] = fminf(nd->lo[d], lo[d] - bv->pad); nd->hi[d] = fmaxf(nd->hi[d], hi[d] + bv->pad);
            float cc = cent[3 * (int64_t)bv->order[i] + d];
            clo[d] = fminf(clo[d], cc); chi[d] = fmaxf(chi[d], cc);
        }
    }
    nd->first = first; nd->count = count; nd->left = nd->right = -1;
    if (count <= 4) return id;
    int axis = 0; float ext = chi[0] - clo[0];
    if (chi[1] - clo[1] > ext) { axis = 1; ext = chi[1] - clo[1]; }
    if (chi[2] - clo[2] > ext) { axis = 2; ext = chi[2] - clo[2]; }
    g_axis = axis; g_cent = cent;
    qsort(bv->order + first, (size_t)count, sizeof(int), cmp_axis);
    int half = count / 2;
    int l = build_rec(bv, m, cent, first, half);
    int r = build_rec(bv, m, cent, first + half, count - half);
    nd = &bv->nodes[id];
    nd->left = l; nd->right = r; nd->count = 0;
    return id;
}

orc_bvh *orc_bvh_build(const orc_mesh *m) {
    orc_bvh *bv = (orc_bvh *)calloc(1, sizeof(orc_bvh));
    int N = m->ntri;
    bv->nodes = (bnode *)malloc(sizeof(bnode) * (size_t)(2 * N + 1));
    bv->order = (int *)malloc(sizeof(int) * (size_t)(N > 0 ? N : 1));
    float *cent = (float *)malloc(sizeof(float) * 3 * (size_t)(N > 0 ? N : 1));
    float slo[3] = { INFINITY, INFINITY, INFINITY }, shi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int k = 0; k < N; k++) {
        float lo[3], hi[3]; tri_box(m, k, lo, hi);
        for (int d = 0; d < 3; d++) {
            cent[3 * (int64_t)k + d] = 0.5f * (lo[d] + hi[d]);
            slo[d] = fminf(slo[d], lo[d]); shi[d] = fmaxf(shi[d], hi[d]);
        }
        bv->order[k] = k;
    }
    float ext = 0.0f, mag = 0.0f;
    for (int d = 0; d < 3; d++) {
        ext = fmaxf(ext, shi[d] - slo[d]);
        if (N > 0) mag = fmaxf(mag, fmaxf(fabsf(slo[d]), fabsf(shi[d])));
    }
    /* generous conservative padding; results never depend on it (checked vs brute force).  Never below 16 ulp of the largest
     * coordinate: far from the origin 1e-4 x extent rounds away (lo - pad == lo), and a ray lying in a box's face plane then
     * reads 0 * inf = NaN there, which the slab test turns into a miss of a box that holds the hit. */
    bv->pad = fmaxf(1e-4f * ext, 16.0f * (nextafterf(mag, INFINITY) - mag));
    if (N > 0) build_rec(bv, m, cent, 0, N);
    free(cent);
    return bv;
}
void orc_bvh_free(orc_bvh *b) { if (b) { free(b->nodes); free(b->order); free(b); } }

static inline int ray_box(const float o[3], const float inv[3], const float lo[3], const float hi[3], float tmax, float *tnear) {
    float tn = 0.0f, tf = tmax;
    for (int d = 0; d < 3; d++) {
        float t0 = (lo[d] - o[d]) * inv[d], t1 = (hi[d] - o[d]) * inv[d];
        float a = fminf(t0, t1), b = fmaxf(t0, t1); /* fminf/fmaxf drop NaN (0*inf) */
        tn = fmaxf(tn, a); tf = fminf(tf, b);
    }
    *tnear = tn;
    return tn <= tf * 1.00001f + 1e-30f;
}

/* tie bookkeeping for the parity report: tie_t = the largest-so-far t at which two DIFFERENT triangles were accepted with
 * exactly equal t while that t was the running minimum; the ray's closest hit is a tie iff tie_t == best.t at the end */
static inline void hit_update_tie(orc_hit *best, float *tie_t, float t, int id, float u, float v) {
    if (tie_t && best->triangleId >= 0 && t == best->t && id != best->triangleId) *tie_t = t;
    hit_update(best, t, id, u, v);
}

/* seed >= 0: test that triangle first (pure optimisation: the (t,id) minimum is order independent) */
static void closest_one_tie(const orc_mesh *m, const orc_bvh *bv, const float *r, int seed, orc_hit *out, int *tie) {
    wray w; wray_setup(r, &w);
    orc_hit best = { -1.0f, -1, 0.0f, 0.0f };
    float tie_store = -1.0f, *tie_t = tie ? &tie_store : NULL;
    if (seed >= 0) {
        v3 a, b, c; tri_verts(m, seed, &a, &b, &c);
        float t, u, v;
        if (wray_tri(&w, a, b, c, &t, &u, &v)) hit_update(&best, t, seed, u, v);
    }
    if (m->ntri > 0) {
        float inv[3] = { 1.0f / r[3], 1.0f / r[4], 1.0f / r[5] };
        int stack[128], sp = 0; stack[sp++] = 0;
        float tn;
        while (sp > 0) {
            const bnode *nd = &bv->nodes[stack[--sp]];
            float tmax = (best.triangleId >= 0) ? best.t : INFINITY;
            if (!ray_box(r, inv, nd->lo, nd->hi, tmax, &tn)) continue;
            if (nd->left < 0) {
                for (int i = nd->first; i < nd->first + nd->count; i++) {
                    int k = bv->order[i]; v3 a, b, c; tri_verts(m, k, &a, &b, &c);
                    float t, u, v;
                    if (k != seed && wray_tri(&w, a, b, c, &t, &u, &v)) hit_update_tie(&best, tie_t, t, k, u, v);
                }
            } else {
                float tl, tr;
                const bnode *L = &bv->nodes[nd->left], *R = &bv->nodes[nd->right];
                int hl = ray_box(r, inv, L->lo, L->hi, tmax, &tl), hr = ray_box(r, inv, R->lo, R->hi, tmax, &tr);
                if (hl && hr) {
                    if (tl <= tr) { stack[sp++] = nd->right; stack[sp++] = nd->left; }
                    else { stack[sp++] = nd->left; stack[sp++] = nd->right; }
                } else if (hl) stack[sp++] = nd->left;
                else if (hr) stack[sp++] = nd->right;
            }
        }
    }
    *out = best;
    if (tie) *tie = (best.triangleId >= 0 && tie_store == best.t) ? 1 : 0;
}
static void closest_one(const orc_mesh *m, const orc_bvh *bv, const float *r, int seed, orc_hit *out) {
    closest_one_tie(m, bv, r, seed, out, NULL);
}

/* Parity report: over the visibility rays of the listed rows (pairs traced exactly as orc_radmat_rows traces them, direct
 * variant), how many have a closest hit whose t is shared bit for bit by two different triangles -- the cases where the
 * (t, id) tie rule, not geometry, decides the mask bit.  OptiX Prime's own tie-breaking is unpinned (closed source). */
int64_t orc_count_ties(const orc_mesh *m, const orc_bvh *b, const float *uv, int S, const int *rows, int nrows, int variant, int nthreads) {
    int N = m->ntri;
    int64_t ties = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#endif
#pragma omp parallel for schedule(dynamic, 1) num_threads(nthreads) reduction(+ : ties)
    for (int ri = 0; ri < nrows; ri++)
        for (int c = 0; c < N; c++) {
            const int r = rows[ri];
            if (c == r) continue;
            int lo = r < c ? r : c, hi = r < c ? c : r;
            if (!(orc_p2p_ff(m, lo, hi, variant) > 0.0f)) continue;
            for (int i = 0; i < S; i++) {
                float ray[6]; orc_pair_ray(m, lo, hi, uv[2 * i], uv[2 * i + 1], ray);
                orc_hit h; int tie = 0;
                closest_one_tie(m, b, ray, hi, &h, &tie);
                ties += tie;
            }
        }
    return ties;
}

void orc_query_closest(const orc_mesh *m, const orc_bvh *b, int n, const float *rays6, orc_hit *hits) {
#pragma omp parallel for schedule(dynamic, 64)
    for (int i = 0; i < n; i++) closest_one(m, b, rays6 + 6 * (int64_t)i, -1, &hits[i]);
}

/* ---- visibility + assembly: VS/OptixPrimeFunctionality.cpp:169-242 (direct) / 311-366 ----- */
static uint64_t pair_mask(const orc_mesh *m, const orc_bvh *b, const float *uv, int S, int lo, int hi, int brute) {
    uint64_t mask = 0;
    for (int i = 0; i < S; i++) {
        float ray[6]; orc_pair_ray(m, lo, hi, uv[2 * i], uv[2 * i + 1], ray);
        orc_hit h;
        if (brute) {
            wray w; wray_setup(ray, &w);
            h.t = -1.0f; h.triangleId = -1; h.u = h.v = 0.0f;
            for (int k = 0; k < m->ntri; k++) {
                v3 a, bb, c; tri_verts(m, k, &a, &bb, &c);
                float t, u, v;
                if (wray_tri(&w, a, bb, c, &t, &u, &v)) hit_update(&h, t, k, u, v);
            }
        } else closest_one(m, b, ray, hi, &h);
        /* float newT = hits[h].t > 0 && hits[h].triangleId == entries[t].col() ? 1 : 0;   :208 */
        if (h.t > 0 && h.triangleId == hi) mask |= (uint64_t)1 << i;
    }
    return mask;
}

/* one row r of RadMat (and its masks) into F_row / mask_row (each N entries, either may be NULL); returns rays cast */
static int64_t radmat_one_row(const orc_mesh *m, const orc_bvh *b, const float *uv, int S, int r, int variant, int reciprocity, int brute,
                              float *F_row, uint64_t *mask_row) {
    int N = m->ntri;
    int64_t rays = 0;
    for (int c = 0; c < N; c++) {
        float val = 0.0f; uint64_t mask = 0;
        if (c != r) {
            int lo = r < c ? r : c, hi = r < c ? c : r;
            if (!reciprocity) {
                /* tripletlist[row*N+col].m_value > 0 with row<col                          :190 */
                float ff_lohi = orc_p2p_ff(m, lo, hi, variant);
                if (ff_lohi > 0.0f) {
                    mask = pair_mask(m, b, uv, S, lo, hi, brute); rays += S;
                    float visibility = 0;
                    for (int i = 0; i < S; i++) visibility += ((mask >> i) & 1) ? 1.0f : 0.0f;
                    visibility = visibility / S;                                         /* :211 */
                    if (visibility > 0) {
                        float ff_rc = (r == lo) ? ff_lohi : orc_p2p_ff(m, r, c, variant);
                        ff_rc = (ff_rc > 0.0) ? ff_rc : 0.0f;                            /* parallellism.cu:101-107 */
                        /* Tripl(row,col, visibility*m_value): float*double -> double; setFromTriplets casts to float */
                        val = (float)((double)visibility * (double)ff_rc);
                    }
                }
            } else {
                /* calculateRadiosityMatrix: p2pFormfactor(row,col) = formfactor*visibility (float), host pi */
                float ff = orc_p2p_ff(m, lo, hi, ORC_FF_HOST);
                mask = pair_mask(m, b, uv, S, lo, hi, brute); rays += S;
                float visibility = 0;
                for (int i = 0; i < S; i++) visibility += ((mask >> i) & 1) ? 1.0f : 0.0f;
                visibility = visibility / S;
                float ffRC = ff * visibility;
                if (ffRC > 0.0) {
                    if (r == lo) val = ffRC;
                    else val = (orc_surface_tri(m, lo) * ffRC) / orc_surface_tri(m, hi);  /* :343 */
                }
            }
        }
        if (F_row) F_row[c] = val;
        if (mask_row) mask_row[c] = mask;
    }
    return rays;
}

int64_t orc_radmat_rows(const orc_mesh *m, const orc_bvh *b, const float *uv, int S, int row0, int row1,
                        int variant, int reciprocity, int brute, float *F_out, uint64_t *masks_out, int nthreads) {
    int N = m->ntri;
    int64_t rays = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#endif
#pragma omp parallel for schedule(dynamic, 1) num_threads(nthreads) reduction(+ : rays)
    for (int r = row0; r < row1; r++)
        rays += radmat_one_row(m, b, uv, S, r, variant, reciprocity, brute, F_out ? F_out + (int64_t)(r - row0) * N : NULL,
                               masks_out ? masks_out + (int64_t)(r - row0) * N : NULL);
    return rays;
}

/* the same for an arbitrary list of rows (sampled-row parity checks and the bounded CPU baseline sample) */
int64_t orc_radmat_rowlist(const orc_mesh *m, const orc_bvh *b, const float *uv, int S, const int *rows, int nrows,
                           int variant, int reciprocity, int brute, float *F_out, uint64_t *masks_out, int nthreads) {
    int N = m->ntri;
    int64_t rays = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#endif
#pragma omp parallel for schedule(dynamic, 1) num_threads(nthreads) reduction(+ : rays)
    for (int i = 0; i < nrows; i++)
        rays += radmat_one_row(m, b, uv, S, rows[i], variant, reciprocity, brute, F_out ? F_out + (int64_t)i * N : NULL,
                               masks_out ? masks_out + (int64_t)i * N : NULL);
    return rays;
}

/* ---- gather: VS/Lightning.h:196-226 -------------------------------------------------------- */
void orc_gather_pass(const float *F, int64_t ldF, int N, int K, float *res, float *B,
                     const float *M, const int *mat_idx, int accum, double *band_sums, int nthreads) {
    float *bounced = (float *)malloc(sizeof(float) * (size_t)K * (size_t)N);
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#endif
    /* bounced_light[i] = RadMat * residualvector[i]                                          :200-202 */
#pragma omp parallel for schedule(static) num_threads(nthreads)
    for (int p = 0; p < N; p++) {
        const float *row = F + (int64_t)p * ldF;
        for (int k = 0; k < K; k++) {
            const float *x = res + (int64_t)k * N;
            if (accum == 0) {
                float y = 0.0f;
                for (int j = 0; j < N; j++) if (row[j] != 0.0f) y += row[j] * x[j];
                bounced[(int64_t)k * N + p] = y;
            } else {
                double y = 0.0;
                for (int j = 0; j < N; j++) y += (double)row[j] * (double)x[j];
                bounced[(int64_t)k * N + p] = (float)y;
            }
        }
    }
    /* result = reflectionmatrix[i] * patchrowvec; residual[j][i] = result[j]; B += residual   :205-223 */
    for (int k = 0; k < K; k++) band_sums[k] = 0.0;
    for (int p = 0; p < N; p++) {
        const float *Mp = M + (int64_t)mat_idx[p] * K * K;
        for (int k = 0; k < K; k++) {
            float r;
            if (accum == 0) {
                float y = 0.0f;
                for (int j = 0; j < K; j++) y += Mp[(int64_t)j * K + k] * bounced[(int64_t)j * N + p];
                r = y;
            } else {
                double y = 0.0;
                for (int j = 0; j < K; j++) y += (double)Mp[(int64_t)j * K + k] * (double)bounced[(int64_t)j * N + p];
                r = (float)y;
            }
            res[(int64_t)k * N + p] = r;
            B[(int64_t)k * N + p] = B[(int64_t)k * N + p] + r;
            band_sums[k] += (double)r;
        }
    }
    free(bounced);
}

int orc_num_procs(void) {
#ifdef _OPENMP
    return omp_get_num_procs();
#else
    return 1;
#endif
}

/* Upper-triangle form of orc_radmat_rows (direct variant only): for r in [row0,row1) and c > r writes
 * F_rc[(r-row0)*N+c] = RadMat(r,c), F_cr[(r-row0)*N+c] = RadMat(c,r) and the pair's mask; entries with c <= r are 0.
 * Used to generate whole-matrix golden checksums without tracing every pair twice. */
int64_t orc_radmat_upper(const orc_mesh *m, const orc_bvh *b, const float *uv, int S, int row0, int row1,
                         int variant, float *F_rc, float *F_cr, uint64_t *masks_out, int nthreads) {
    int N = m->ntri;
    int64_t rays = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#endif
#pragma omp parallel for schedule(dynamic, 1) num_threads(nthreads) reduction(+ : rays)
    for (int r = row0; r < row1; r++) {
        for (int c = 0; c < N; c++) {
            int64_t o = (int64_t)(r - row0) * N + c;
            float v_rc = 0.0f, v_cr = 0.0f; uint64_t mask = 0;
            if (c > r) {
                float ff_rc = orc_p2p_ff(m, r, c, variant);
                if (ff_rc > 0.0f) {
                    mask = pair_mask(m, b, uv, S, r, c, 0); rays += S;
                    float visibility = 0;
                    for (int i = 0; i < S; i++) visibility += ((mask >> i) & 1) ? 1.0f : 0.0f;
                    visibility = visibility / S;
                    if (visibility > 0) {
                        float ff_cr = orc_p2p_ff(m, c, r, variant);
                        ff_cr = (ff_cr > 0.0) ? ff_cr : 0.0f;
                        v_rc = (float)((double)visibility * (double)ff_rc);
                        v_cr = (float)((double)visibility * (double)ff_cr);
                    }
                }
            }
            if (F_rc) F_rc[o] = v_rc;
            if (F_cr) F_cr[o] = v_cr;
            if (masks_out) masks_out[o] = mask;
        }
    }
    return rays;
}
