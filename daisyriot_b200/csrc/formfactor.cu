// formfactor.cu -- unoccluded 4x4 form-factor rule + 50-sample visibility, fused, writing dense FP32 rows.
//
// Replaces (reference "visual studio/"):
//   parallellism::calculateRow / p2pFormfactor / calcPointFormfactor     parallellism.cu:91-227
//   OptixPrimeFunctionality::calculateAllVisibility                      OptixPrimeFunctionality.cpp:169-242
//   OptixPrimeFunctionality::calculateRadiosityMatrix (cuda_on=false)    OptixPrimeFunctionality.cpp:311-366
// The reference materialises N^2 16-byte triplets on the host, generates 24-byte rays on one CPU thread, ships
// them to OptiX Prime in 4M-ray batches and reduces 16-byte hits on the host.  Here one kernel owns a 64x64 tile
// of the upper triangle: it evaluates the 16 sub-patch terms once (they serve F(r,c) and F(c,r)), generates the
// rays in registers, resolves them against per-pair candidate lists (shaft walk of the LBVH; triangles coplanar with
// one of the two patches are only tested by the few samples near the patch edges, see k_tri_planes) and writes both
// mirrored tiles coalesced through shared memory -- into this rank's matrix or a peer's over NVLink.
#include "daisy_common.cuh"
#include <math.h>
#include <chrono>
#include <stdlib.h>
#include <algorithm>
#include <vector>

#define TILE 64
#define NBR_CAP 32 // ints per triangle in the neighbour table: [0] = count, then up to 31 triangles of its own plane
// CTA shape: 512 threads x 2 CTAs per SM = the same 32 warps per SM at 64 registers as 256 x 4, but half the shared memory
// (two tiles in flight per SM instead of four), which leaves the SM ~124 KB of L1 instead of ~28 KB for the face tables, cell
// lists, vertices and neighbour lists the rays gather from: 537 -> 506 ms at 32K patches, 73 -> 63 / 58 -> 47 ms on the
// reference's scenes (384 x 3: 518 ms; 1024 x 1: 595 ms, the tile barriers bite).
#ifndef FF_THREADS
#define FF_THREADS 512
#endif
#ifndef FF_MINBLOCKS
#define FF_MINBLOCKS 2
#endif
#define PI_D 3.14159265358979323846
#define PI_F 3.14159265358979323846f

// Sample pattern in DEVICE order: samples whose barycentric margin min(u, v, 1-u-v) is at least EDGE_MARGIN come first
// ("inner" samples), the rest ("edge" samples) last; perm maps a device position back to the caller's sample index
// (= bit position in the visibility mask).  Rays of inner samples leave and reach the two patches well inside them, which
// is what lets coplanar neighbours be skipped for them (see k_tri_planes / shaft_candidates).  The pattern travels in the
// kernel's parameters, so every launch carries its own context's pattern: two contexts on one device never see each other's.
#define EDGE_MARGIN 0.02f
#ifdef DAISY_FF_STATS
__device__ unsigned long long g_ffstats[48];
#endif

// fills uv and perm (DAISY_MAX_SAMPLES entries each, zero past S) and returns the number of inner samples
static int samples_device_order(const daisy_ctx *ctx, float *uv, unsigned char *perm) {
    memset(uv, 0, sizeof(float) * 2 * DAISY_MAX_SAMPLES);
    memset(perm, 0, DAISY_MAX_SAMPLES);
    int n = 0, n_inner = 0;
    for (int pass = 0; pass < 2; pass++) {
        for (int i = 0; i < ctx->S; i++) {
            const float u = ctx->h_uv[2 * i], v = ctx->h_uv[2 * i + 1];
            const bool inner = fminf(fminf(u, v), 1.0f - u - v) >= EDGE_MARGIN;
            if (inner == (pass == 0)) { uv[2 * n] = u; uv[2 * n + 1] = v; perm[n] = (unsigned char)i; n++; }
        }
        if (pass == 0) n_inner = n;
    }
    return n_inner;
}

// ---------------------------------------------------------------------------------------------------------
// per-patch precompute: divideInFourTriangles (parallellism.cu:153-172), calculateCentre (:181-186),
// calculateSurface (:209-227), avgNormal (:188-195).  Same operation order as the reference, no FMA.
__global__ void k_patch_geom(const float *__restrict__ vertices, const float *__restrict__ normals, const int *__restrict__ tri,
                             int N, PatchGeom *__restrict__ geom) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N) return;
    const int *t = tri + 6 * (size_t)p;
    f3 a = mk3(vertices[3 * (size_t)t[0]], vertices[3 * (size_t)t[0] + 1], vertices[3 * (size_t)t[0] + 2]);
    f3 b = mk3(vertices[3 * (size_t)t[1]], vertices[3 * (size_t)t[1] + 1], vertices[3 * (size_t)t[1] + 2]);
    f3 c = mk3(vertices[3 * (size_t)t[2]], vertices[3 * (size_t)t[2] + 1], vertices[3 * (size_t)t[2] + 2]);
    f3 n0 = mk3(normals[3 * (size_t)t[3]], normals[3 * (size_t)t[3] + 1], normals[3 * (size_t)t[3] + 2]);
    f3 n1 = mk3(normals[3 * (size_t)t[4]], normals[3 * (size_t)t[4] + 1], normals[3 * (size_t)t[4] + 2]);
    f3 n2 = mk3(normals[3 * (size_t)t[5]], normals[3 * (size_t)t[5] + 1], normals[3 * (size_t)t[5] + 2]);
    // innerA = ((b - a) / 2.0f) + a ; innerC = ((c - a) / 2.0f) + a ; innerB = ((b - c) / 2.0f) + c
    f3 ba = e_sub(b, a), ca = e_sub(c, a), bc = e_sub(b, c);
    f3 iA = e_add(mk3(fd(ba.x, 2.0f), fd(ba.y, 2.0f), fd(ba.z, 2.0f)), a);
    f3 iC = e_add(mk3(fd(ca.x, 2.0f), fd(ca.y, 2.0f), fd(ca.z, 2.0f)), a);
    f3 iB = e_add(mk3(fd(bc.x, 2.0f), fd(bc.y, 2.0f), fd(bc.z, 2.0f)), c);
    f3 T[4][3] = { { a, iC, iA }, { iC, c, iB }, { iA, iB, b }, { iA, iB, iC } };
    PatchGeom g;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        f3 s = e_add(e_add(T[i][0], T[i][1]), T[i][2]);
        g.s[i] = make_float4(fd(s.x, 3.0f), fd(s.y, 3.0f), fd(s.z, 3.0f), e_surface(T[i][0], T[i][1], T[i][2]));
    }
    f3 ns = e_add(e_add(n0, n1), n2);
    f3 nn = e_normalize(mk3(fd(ns.x, 3.0f), fd(ns.y, 3.0f), fd(ns.z, 3.0f)));
    g.n = make_float4(nn.x, nn.y, nn.z, e_surface(a, b, c));
    geom[p] = g;
}


// ---------------------------------------------------------------------------------------------------------
// Per-triangle plane record for coplanar skipping.  A triangle k that lies in the plane of patch t and does not overlap
// t can never be hit by a ray that starts (or ends) inside t by a margin and leaves (reaches) the plane steeply: the ray
// meets the plane once, at a point inside t, so the watertight test's edge functions for k have mixed signs by a margin far
// above rounding.  The shaft walk uses that to drop such k for the inner samples.  This kernel establishes the static
// part of the premise for every t: it is not degenerate or sliver-shaped, and NO coplanar triangle overlaps it (checked
// with a 2-D separating-axis test against every triangle whose padded box meets t's box; coplanar neighbours that are
// slivers or much larger than t also disqualify t, because the rounding bound scales with their size).
// plane[t] = (unit normal, smallest altitude h_t) or w = -1 if t does not qualify.  Double precision: runs once.
struct d3 { double x, y, z; };
__device__ __forceinline__ d3 dsub(d3 a, d3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
__device__ __forceinline__ double ddot(d3 a, d3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ d3 dcross(d3 a, d3 b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }
__device__ __forceinline__ d3 dv(float4 v) { return { (double)v.x, (double)v.y, (double)v.z }; }

// true if the projections of triangles P and Q onto the plane (origin o, axes ux, uy) overlap by more than tol
__device__ bool tri_overlap_2d(const d3 *P, const d3 *Q, d3 o, d3 ux, d3 uy, double tol) {
    double px[6], py[6];
    for (int i = 0; i < 3; i++) {
        d3 a = dsub(P[i], o), b = dsub(Q[i], o);
        px[i] = ddot(a, ux); py[i] = ddot(a, uy);
        px[3 + i] = ddot(b, ux); py[3 + i] = ddot(b, uy);
    }
    for (int t = 0; t < 2; t++)
        for (int e = 0; e < 3; e++) {
            const int i0 = 3 * t + e, i1 = 3 * t + (e + 1) % 3;
            double ax = -(py[i1] - py[i0]), ay = px[i1] - px[i0];
            const double len = sqrt(ax * ax + ay * ay);
            if (len <= 0.0) continue;
            ax /= len; ay /= len;
            double mnP = 1e300, mxP = -1e300, mnQ = 1e300, mxQ = -1e300;
            for (int i = 0; i < 3; i++) {
                const double a = px[i] * ax + py[i] * ay, b = px[3 + i] * ax + py[3 + i] * ay;
                mnP = fmin(mnP, a); mxP = fmax(mxP, a); mnQ = fmin(mnQ, b); mxQ = fmax(mxQ, b);
            }
            if (fmin(mxP, mxQ) - fmax(mnP, mnQ) <= tol) return false; // separated (or only touching) along this axis
        }
    return true;
}

__global__ void k_tri_planes(const TriVerts *__restrict__ tv, const float4 *__restrict__ tribox, const BvhNode *__restrict__ nodes, int root,
                             int N, double tau, double tau2, float grow, const int *__restrict__ pid, float4 *__restrict__ plane, int *__restrict__ nbr) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N) return;
    const TriVerts T = tv[t];
    const int my_pid = pid[t];
    int n_nbr = 0;
    int *my_nbr = nbr + (size_t)t * NBR_CAP;
    my_nbr[0] = 0;
    const d3 P[3] = { dv(T.a), dv(T.b), dv(T.c) };
    const d3 e1 = dsub(P[1], P[0]), e2 = dsub(P[2], P[0]), e3 = dsub(P[2], P[1]);
    d3 n = dcross(e1, e2);
    const double A2 = sqrt(ddot(n, n));
    if (!(A2 > 0.0)) { plane[t] = make_float4(0.f, 0.f, 0.f, -1.f); return; }
    n = { n.x / A2, n.y / A2, n.z / A2 };
    const double maxe = sqrt(fmax(ddot(e1, e1), fmax(ddot(e2, e2), ddot(e3, e3))));
    const double h = A2 / maxe;
    bool safe = h * 8.0 >= maxe;
    const double l1 = sqrt(ddot(e1, e1));
    const d3 ux = { e1.x / l1, e1.y / l1, e1.z / l1 };
    const d3 uy = dcross(n, ux);
    float4 b0 = tribox[2 * (size_t)t], b1 = tribox[2 * (size_t)t + 1];
    b0.x -= grow; b0.y -= grow; b0.z -= grow; b1.x += grow; b1.y += grow; b1.z += grow;
    int stack[64];
    int sp = 0, cur = root;
    while (safe) {
        if (cur < 0) {
            const int k = ~cur;
            if (k != t) {
                const TriVerts K = tv[k];
                const d3 Q[3] = { dv(K.a), dv(K.b), dv(K.c) };
                double dist = 0.0;
                for (int j = 0; j < 3; j++) dist = fmax(dist, fabs(ddot(n, dsub(Q[j], P[0]))));
                const bool same_plane = my_pid != 0 && pid[k] == my_pid;
                if (same_plane) { // goes on this patch's neighbour list: the only triangles of its plane its edge samples have to test
                    if (n_nbr == NBR_CAP - 1) safe = false;
                    else { DZ_ASSERT(1 + n_nbr < NBR_CAP); my_nbr[1 + n_nbr++] = k; }
                }
                if (dist <= 4.0 * tau || same_plane) { // coplanar neighbour
                    const d3 f1 = dsub(Q[1], Q[0]), f2 = dsub(Q[2], Q[0]), f3 = dsub(Q[2], Q[1]);
                    const d3 nk = dcross(f1, f2);
                    const double A2k = sqrt(ddot(nk, nk));
                    const double maxk = sqrt(fmax(ddot(f1, f1), fmax(ddot(f2, f2), ddot(f3, f3))));
                    if (!(A2k > 0.0) || (A2k / maxk) * 8.0 < maxk || maxk > 16.0 * h) safe = false;
                    else if (tri_overlap_2d(P, Q, P[0], ux, uy, tau2)) safe = false;
                }
            }
            if (sp == 0) break;
            cur = stack[--sp];
            continue;
        }
        const BvhNode nd = nodes[cur];
        const bool hl = !(nd.a.x > b1.x || nd.a.w < b0.x || nd.a.y > b1.y || nd.b.x < b0.y || nd.a.z > b1.z || nd.b.y < b0.z);
        const bool hr = !(nd.b.z > b1.x || nd.c.y < b0.x || nd.b.w > b1.y || nd.c.z < b0.y || nd.c.x > b1.z || nd.c.w < b0.z);
        if (hl && hr) { DZ_ASSERT(sp < 64); stack[sp++] = nd.d.y; cur = nd.d.x; }
        else if (hl) cur = nd.d.x;
        else if (hr) cur = nd.d.y;
        else {
            if (sp == 0) break;
            cur = stack[--sp];
        }
    }
    plane[t] = make_float4((float)n.x, (float)n.y, (float)n.z, (safe && my_pid != 0) ? (float)h : -1.f);
    my_nbr[0] = safe ? n_nbr : 0;
}

#define COPLANAR_TAU 3e-7f // x scene extent: a triangle within this distance of a patch's plane counts as coplanar
#define OVERLAP_TAU 2e-6f  // x scene extent: projected overlap below this is "touching", not overlapping
int dz_precompute_geom(daisy_ctx *ctx) {
    if (ctx->N == 0) return DAISY_OK;
    k_patch_geom<<<(ctx->N + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_vertices, ctx->d_normals, ctx->d_tri, ctx->N, ctx->d_geom);
    DZ_CUDA(cudaGetLastError());
    k_tri_planes<<<(ctx->N + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_triverts, ctx->d_tribox, ctx->d_nodes, ctx->root, ctx->N,
                                                             (double)COPLANAR_TAU * ctx->ext, (double)OVERLAP_TAU * ctx->ext, 2.0f * ctx->pad, ctx->d_pid,
                                                             ctx->d_plane, ctx->d_nbr);
    DZ_CUDA(cudaGetLastError());
    return DAISY_OK;
}

// ---------------------------------------------------------------------------------------------------------
// The 16 point-to-point terms of p2pFormfactor for origin patch o and destination patch d.
// term(i,j) is symmetric under swapping the roles of the two patches bit for bit (negation and multiplication
// commute exactly), so one evaluation yields F(o->d) = (sum_i sum_j term)/A_o and F(d->o) = (sum_j sum_i term)/A_d.
template <int VARIANT>
__device__ __forceinline__ void ff_pair(const PatchGeom &o, const PatchGeom &d, float &ff_od, float &ff_do) {
    f3 no = xyz(o.n), nd = xyz(d.n);
    float t[4][4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
#pragma unroll
        for (int j = 0; j < 4; j++) {
            f3 v = e_sub(xyz(d.s[j]), xyz(o.s[i])); // dest.pos - orig.pos
            float l2 = e_dot(v, v);
            float len = fsq(l2);
            float inv = fd(1.0f, len);
            f3 nv = e_scale(v, inv);
            float dot1 = e_dot(no, nv);
            // normalize(orig.pos - dest.pos) is exactly -nv, and dot(n, -x) is exactly -dot(n, x)
            float dot2 = -e_dot(nd, nv);
            float term = 0.0f;
            if (dot1 > 0.0f && dot2 > 0.0f) {
                float surface = fm(o.s[i].w, d.s[j].w);
                float len2 = fm(len, len); // powf(length, 2)
                if (VARIANT == DAISY_FF_DEVICE) {
                    // ((dot1*dot2) / (powf(length,2) * CUDART_PI)) * surface, CUDART_PI double   parallellism.cu:204
                    double den = __dmul_rn((double)len2, PI_D);
                    double q = __ddiv_rn((double)fm(dot1, dot2), den);
                    term = __double2float_rn(__dmul_rn(q, (double)surface));
                } else {
                    // all-float host form with M_PIf                                          triangle_math.cpp:55
                    term = fm(fd(fm(dot1, dot2), fm(len2, PI_F)), surface);
                }
            }
            t[i][j] = term;
        }
    }
    float s_od = 0.0f, s_do = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) s_od = fa(s_od, t[i][j]);
#pragma unroll
    for (int j = 0; j < 4; j++)
#pragma unroll
        for (int i = 0; i < 4; i++) s_do = fa(s_do, t[i][j]);
    ff_od = fd(s_od, o.n.w);
    ff_do = fd(s_do, d.n.w);
}

// dense unoccluded triplets, diagonal included (calculateRow, parallellism.cu:91-111)
template <int VARIANT>
__global__ void k_unoccluded(const PatchGeom *__restrict__ geom, int N, int row0, int nrows, daisy_tripl *__restrict__ out) {
    int c = blockIdx.x * blockDim.x + threadIdx.x;
    int r = row0 + blockIdx.y;
    if (c >= N || r >= row0 + nrows) return;
    PatchGeom o = geom[r], d = geom[c];
    float f_od, f_do;
    ff_pair<VARIANT>(o, d, f_od, f_do);
    daisy_tripl t;
    t.m_row = r; t.m_col = c;
    t.m_value = (f_od > 0.0f) ? (double)f_od : 0.0; // NaN (coincident points) -> 0, as `formfactorRC > 0.0` does
    out[(size_t)(r - row0) * N + c] = t;
}

int dz_unoccluded_rows(daisy_ctx *ctx, int variant, int row0, int nrows, daisy_tripl *d_out) {
    if (nrows <= 0 || ctx->N == 0) return DAISY_OK;
    dim3 grid((ctx->N + 127) / 128, nrows);
    if (variant == DAISY_FF_DEVICE)
        k_unoccluded<DAISY_FF_DEVICE><<<grid, 128, 0, ctx->stream>>>(ctx->d_geom, ctx->N, row0, nrows, d_out);
    else
        k_unoccluded<DAISY_FF_HOST><<<grid, 128, 0, ctx->stream>>>(ctx->d_geom, ctx->N, row0, nrows, d_out);
    DZ_CUDA(cudaGetLastError());
    return DAISY_OK;
}

// ---------------------------------------------------------------------------------------------------------
// One visibility ray of the pair (lo -> hi), sample (u,v): restates OptixPrimeFunctionality.cpp:191-196 and the
// hit test of :208, i.e. "closest hit over ALL triangles has t > 0 and is triangle hi".  Evaluated as an
// occlusion query bounded by the hit on hi itself: the ray sees hi iff the watertight test accepts hi at t_hi and
// no other triangle k is accepted with (t_k, k) < (t_hi, hi) lexicographically -- the same predicate, but the
// traversal can stop at the first occluder and never looks beyond t_hi.
// skip_lo / skip_hi: plane ids whose triangles this ray cannot touch (coplanar skipping, see the kernel; 0 = none): children
// of a node lying entirely in such a plane are not entered.
__device__ __noinline__ bool ray_sees(const BvhNode *__restrict__ nodes, const TriVerts *__restrict__ tv, int root,
                                         const TriVerts &Tlo, const TriVerts &Thi, int lo, int hi, float u, float v, int skip_lo, int skip_hi) {
    // uv2xyz: a + u*(b-a) + v*(c-a)                                                   triangle_math.cpp:3-9
    f3 a0 = xyz(Tlo.a), a1 = xyz(Thi.a);
    f3 org = e_add(e_add(a0, e_scale(e_sub(xyz(Tlo.b), a0), u)), e_scale(e_sub(xyz(Tlo.c), a0), v));
    f3 dst = e_add(e_add(a1, e_scale(e_sub(xyz(Thi.b), a1), u)), e_scale(e_sub(xyz(Thi.c), a1), v));
    f3 dir = e_normalize(e_sub(dst, org));      // optix::normalize(dest - origin)
    f3 o = e_add(org, e_scale(dir, 0.000001f)); // origin + normalize(dest - origin)*0.000001f
    WRay w = wray_setup(o, dir);
    float thi;
    if (!wray_tri_t(w, xyz(Thi.a), xyz(Thi.b), xyz(Thi.c), thi)) return false;
    float tk;
    // the origin patch itself takes part like any other triangle (lo < hi, so a tie on t hides hi)
    if (wray_tri_t(w, xyz(Tlo.a), xyz(Tlo.b), xyz(Tlo.c), tk) && tk <= thi) return false;
    f3 inv = mk3(1.0f / dir.x, 1.0f / dir.y, 1.0f / dir.z);
    int stack[64];
    int sp = 0;
    int cur = root;
    while (true) {
        if (cur < 0) {
            int k = ~cur;
            if (k != lo && k != hi) {
                TriVerts t = tv[k];
                if (wray_tri_t(w, xyz(t.a), xyz(t.b), xyz(t.c), tk) && (tk < thi || (tk == thi && k < hi))) return false;
            }
            if (sp == 0) break;
            cur = stack[--sp];
            continue;
        }
        BvhNode nd = nodes[cur];
        float tl, tr;
        const bool sl = nd.d.z != 0 && (nd.d.z == skip_lo || nd.d.z == skip_hi);
        const bool sr = nd.d.w != 0 && (nd.d.w == skip_lo || nd.d.w == skip_hi);
        bool hl = !sl && ray_box(o, inv, nd.a.x, nd.a.y, nd.a.z, nd.a.w, nd.b.x, nd.b.y, thi, tl);
        bool hr = !sr && ray_box(o, inv, nd.b.z, nd.b.w, nd.c.x, nd.c.y, nd.c.z, nd.c.w, thi, tr);
        if (hl && hr) { DZ_ASSERT(sp < 64); stack[sp++] = nd.d.y; cur = nd.d.x; }
        else if (hl) cur = nd.d.x;
        else if (hr) cur = nd.d.y;
        else {
            if (sp == 0) break;
            cur = stack[--sp];
        }
    }
    return true;
}

// ---------------------------------------------------------------------------------------------------------
// Shaft culling (Haines & Wallace style) per patch pair.  Every visibility ray of the pair (lo -> hi) lies inside
// the convex hull of the two triangles, so a triangle can only be hit by one of those rays if its (padded) box meets
// that hull.  The hull is tested conservatively with six separating axes: x, y, z and D x {x,y,z} with D the
// direction between the two centroids.  Skipping any axis only makes the test say "may intersect" more often, so the
// candidate list is always a superset of the triangles any of the S rays can touch; rays are then tested against the
// list with the very same watertight routine and the same (t, id) rule => identical masks, far fewer node visits.
#define FF_QCAP 6 // pending watertight tests per lane (4 bits each in one register)
#define SHAFT_CAP 256 // ints of global scratch per pair slot; longer lists fall back to per-ray LBVH walks
struct Shaft {
    float lox, loy, loz, hix, hiy, hiz; // hull AABB
    float Dx, Dy, Dz;                   // centroid(hi) - centroid(lo) (scaled by 3, irrelevant)
    float c0min, c0max, c1min, c1max, c2min, c2max; // hull extent along D x e_x, D x e_y, D x e_z
};

__device__ __forceinline__ Shaft make_shaft(const TriVerts &A, const TriVerts &B) {
    Shaft s;
    float4 p[6] = { A.a, A.b, A.c, B.a, B.b, B.c };
    s.lox = s.hix = p[0].x; s.loy = s.hiy = p[0].y; s.loz = s.hiz = p[0].z;
#pragma unroll
    for (int i = 1; i < 6; i++) {
        s.lox = fminf(s.lox, p[i].x); s.hix = fmaxf(s.hix, p[i].x);
        s.loy = fminf(s.loy, p[i].y); s.hiy = fmaxf(s.hiy, p[i].y);
        s.loz = fminf(s.loz, p[i].z); s.hiz = fmaxf(s.hiz, p[i].z);
    }
    s.Dx = (B.a.x + B.b.x + B.c.x) - (A.a.x + A.b.x + A.c.x);
    s.Dy = (B.a.y + B.b.y + B.c.y) - (A.a.y + A.b.y + A.c.y);
    s.Dz = (B.a.z + B.b.z + B.c.z) - (A.a.z + A.b.z + A.c.z);
    s.c0min = s.c1min = s.c2min = INFINITY;
    s.c0max = s.c1max = s.c2max = -INFINITY;
#pragma unroll
    for (int i = 0; i < 6; i++) {
        float q0 = p[i].y * s.Dz - p[i].z * s.Dy;
        float q1 = p[i].z * s.Dx - p[i].x * s.Dz;
        float q2 = p[i].x * s.Dy - p[i].y * s.Dx;
        s.c0min = fminf(s.c0min, q0); s.c0max = fmaxf(s.c0max, q0);
        s.c1min = fminf(s.c1min, q1); s.c1max = fmaxf(s.c1max, q1);
        s.c2min = fminf(s.c2min, q2); s.c2max = fmaxf(s.c2max, q2);
    }
    return s;
}

// conservative: false only if one of the six axes separates the (padded) box from the hull
__device__ __forceinline__ bool shaft_box(const Shaft &s, float lox, float loy, float loz, float hix, float hiy, float hiz) {
    if (lox > s.hix || hix < s.lox || loy > s.hiy || hiy < s.loy || loz > s.hiz || hiz < s.loz) return false;
    float cx = 0.5f * (lox + hix), cy = 0.5f * (loy + hiy), cz = 0.5f * (loz + hiz);
    float hx = 0.5f * (hix - lox), hy = 0.5f * (hiy - loy), hz = 0.5f * (hiz - loz);
    float ax = fabsf(s.Dx), ay = fabsf(s.Dy), az = fabsf(s.Dz);
    // slack: a few ulps of the projected magnitudes, on top of the 1e-4*extent padding the boxes already carry
    float p0 = cy * s.Dz - cz * s.Dy, r0 = hy * az + hz * ay;
    r0 += 1e-5f * (fabsf(p0) + r0);
    if (p0 - r0 > s.c0max || p0 + r0 < s.c0min) return false;
    float p1 = cz * s.Dx - cx * s.Dz, r1 = hz * ax + hx * az;
    r1 += 1e-5f * (fabsf(p1) + r1);
    if (p1 - r1 > s.c1max || p1 + r1 < s.c1min) return false;
    float p2 = cx * s.Dy - cy * s.Dx, r2 = hx * ay + hy * ax;
    r2 += 1e-5f * (fabsf(p2) + r2);
    if (p2 - r2 > s.c2max || p2 + r2 < s.c2min) return false;
    return true;
}

// collect the triangles (other than lo and hi) whose leaf box meets the shaft into the pair's candidate list.  skip_lo /
// skip_hi: plane id of lo / hi when that side's premise of coplanar skipping holds (see k_tri_planes and the kernel), else 0.
// Triangles lying in such a plane are left out altogether -- the only ones a ray of this pair can touch are the patch's
// direct neighbours, which the edge samples test from the precomputed neighbour lists -- and, since every LBVH node
// carries the plane id common to all triangles below it, whole subtrees of a wall the pair starts or ends on are never
// entered.  Returns the number of candidates, or -1 if they do not fit SHAFT_CAP.
//
// Face grids (faces.cu): a child that holds nothing but triangles of gridded faces (plane ids 1..nfaces; the node carries
// the id, or -1 for several faces) is not entered either.  The faces a pair has to consider are found by testing the faces'
// own boxes against the shaft (they are at most DAISY_MAX_FACES); each goes into the pair's face mask and every ray settles
// it on its own (pair_mask_warp: plane crossing + cell lookup, or proof that it stays clear of the plane, or -- for the few
// rays that lie in the plane -- a walk restricted to that face).  In a scene made of planar faces only, the walk ends at the root.
__device__ __forceinline__ int shaft_candidates(const BvhNode *__restrict__ nodes, int root, const Shaft &sh, int skip_lo, int skip_hi, int lo, int hi,
                                                int *__restrict__ cand, const DzFace *__restrict__ faces, int nfaces, unsigned long long &fmask) {
    int n_main = 0;
    int stack[64];
    int sp = 0;
    int cur = root;
    bool overflow = false;
    fmask = 0;
    for (int f = 0; f < nfaces; f++) {
        if (f + 1 == skip_lo || f + 1 == skip_hi) continue;
        DZ_ASSERT(f < DAISY_MAX_FACES);
        const float4 b0 = __ldg(&faces[f].blo), b1 = __ldg(&faces[f].bhi);
        if (shaft_box(sh, b0.x, b0.y, b0.z, b1.x, b1.y, b1.z)) fmask |= 1ull << f;
    }
    if (cur < 0) return 0; // single-triangle hierarchy: no third triangle exists
    while (!overflow) {
        const BvhNode nd = nodes[cur];
        const bool sl = nd.d.z != 0 && (nd.d.z == skip_lo || nd.d.z == skip_hi || nd.d.z == -1 || nd.d.z <= nfaces);
        const bool sr = nd.d.w != 0 && (nd.d.w == skip_lo || nd.d.w == skip_hi || nd.d.w == -1 || nd.d.w <= nfaces);
        bool hl = !sl && shaft_box(sh, nd.a.x, nd.a.y, nd.a.z, nd.a.w, nd.b.x, nd.b.y);
        bool hr = !sr && shaft_box(sh, nd.b.z, nd.b.w, nd.c.x, nd.c.y, nd.c.z, nd.c.w);
        if (hl && nd.d.x < 0) {
            const int k = ~nd.d.x;
            if (k != lo && k != hi) { DZ_ASSERT(k >= 0 && n_main <= SHAFT_CAP); if (n_main == SHAFT_CAP) overflow = true; else cand[n_main++] = k; }
            hl = false;
        }
        if (hr && nd.d.y < 0) {
            const int k = ~nd.d.y;
            if (k != lo && k != hi) { DZ_ASSERT(k >= 0 && n_main <= SHAFT_CAP); if (n_main == SHAFT_CAP) overflow = true; else cand[n_main++] = k; }
            hr = false;
        }
        if (hl && hr) { DZ_ASSERT(sp < 64); stack[sp++] = nd.d.y; cur = nd.d.x; }
        else if (hl) cur = nd.d.x;
        else if (hr) cur = nd.d.y;
        else {
            if (sp == 0) break;
            cur = stack[--sp];
        }
    }
    return overflow ? -1 : n_main;
}

// Premise of coplanar skipping per side of a pair: the patch qualifies (plane.w = its smallest altitude h > 0, k_tri_planes)
// and every ray meets its plane steeply.  The ray directions are convex combinations of the three vertex-to-vertex vectors
// D_i, so n.D_i of one sign bounds cos(theta) >= min|n.D_i| / max|D_i|.  The edge functions of a coplanar triangle near a
// patch are computed from coordinates relative to the ray origin: rounding ~ 8 eps (distance) (its size), against a true
// value >= (margin h)(its edge) cos(theta).  With sizes and aspect ratios bounded by k_tri_planes that gives cos >= 0.02 on
// the origin side (distance ~ size) and margin h cos >= 128 eps (distance) on the destination side.  on_lo / on_hi: the side's
// plane may be skipped by every sample whose barycentric margin is at least m_req (<= EDGE_MARGIN, so by all inner samples).
__device__ __forceinline__ void pair_premise(const TriVerts &A, const TriVerts &B, float4 pl, float4 ph, bool &on_lo, bool &on_hi, float &m_req) {
    const float d0x = B.a.x - A.a.x, d0y = B.a.y - A.a.y, d0z = B.a.z - A.a.z;
    const float d1x = B.b.x - A.b.x, d1y = B.b.y - A.b.y, d1z = B.b.z - A.b.z;
    const float d2x = B.c.x - A.c.x, d2y = B.c.y - A.c.y, d2z = B.c.z - A.c.z;
    const float dmax = sqrtf(fmaxf(d0x * d0x + d0y * d0y + d0z * d0z, fmaxf(d1x * d1x + d1y * d1y + d1z * d1z, d2x * d2x + d2y * d2y + d2z * d2z)));
    const float l0 = pl.x * d0x + pl.y * d0y + pl.z * d0z, l1 = pl.x * d1x + pl.y * d1y + pl.z * d1z, l2 = pl.x * d2x + pl.y * d2y + pl.z * d2z;
    const float h0 = ph.x * d0x + ph.y * d0y + ph.z * d0z, h1 = ph.x * d1x + ph.y * d1y + ph.z * d1z, h2 = ph.x * d2x + ph.y * d2y + ph.z * d2z;
    const float lmin = ((l0 > 0.f) == (l1 > 0.f) && (l1 > 0.f) == (l2 > 0.f)) ? fminf(fabsf(l0), fminf(fabsf(l1), fabsf(l2))) : 0.f;
    const float hmin = ((h0 > 0.f) == (h1 > 0.f) && (h1 > 0.f) == (h2 > 0.f)) ? fminf(fabsf(h0), fminf(fabsf(h1), fabsf(h2))) : 0.f;
    // required margins (fractions of the altitude): m >= 128 eps D / (h cos), D = 32 h on the origin side
    const float mlo = (pl.w > 0.f && lmin > 0.f) ? 2.44e-4f * dmax / lmin : 1.f;
    const float mhi = (ph.w > 0.f && hmin > 0.f) ? 7.63e-6f * (dmax + 64.f * ph.w) * dmax / (hmin * ph.w) : 1.f;
    on_lo = mlo <= EDGE_MARGIN;
    on_hi = mhi <= EDGE_MARGIN;
    m_req = fmaxf(on_lo ? mlo : 0.f, on_hi ? mhi : 0.f);
}

// Visibility mask of one pair with the whole warp: lane = sample (device order), a candidate list is walked in lock step
// (uniform loads), each candidate first meets a cheap conservative slab test against its padded box and only then the
// watertight test.  Same predicate as ray_sees: sample i sees hi iff hi is accepted at t_hi and no other triangle k
// is accepted with (t_k, k) < (t_hi, hi); lo takes part like any other triangle.  The main list is tested by every
// sample, the ring list (coplanar with lo or hi, see shaft_candidates) only by the edge samples.
#define FACE_COS_MIN 0.05f
struct FaceTables {
    const DzFace *faces;
    const int *cells, *lists;
    const BvhNode *nodes;
    int root;
    int64_t ncells, nlist; // table sizes (bounds checks of the checked build)
    float tm;  // margin on the ray parameter: crossings within tm of either end point are resolved by explicit tests
    float eps; // a ray can only touch a triangle of a face where it runs within eps of the face's plane
};

// Is the ray blocked by a triangle of plane id fpid?  LBVH walk that enters only children holding such triangles (their own
// id, or 0 / -1 = mixed) -- the exact test for the few rays that run along a face's plane too flatly for the grid lookup.
__device__ __noinline__ bool face_blocks_ray(const BvhNode *__restrict__ nodes, const TriVerts *__restrict__ tv, int root, const WRay &w, f3 dir, float thi,
                                             int lo, int hi, int fpid) {
    const f3 o = w.o;
    const f3 inv = mk3(1.0f / dir.x, 1.0f / dir.y, 1.0f / dir.z);
    int stack[64];
    int sp = 0, cur = root;
    if (cur < 0) return false;
    while (true) {
        const BvhNode nd = nodes[cur];
        float tl, tr, tk;
        bool hl = (nd.d.z <= 0 || nd.d.z == fpid) && ray_box(o, inv, nd.a.x, nd.a.y, nd.a.z, nd.a.w, nd.b.x, nd.b.y, thi, tl);
        bool hr = (nd.d.w <= 0 || nd.d.w == fpid) && ray_box(o, inv, nd.b.z, nd.b.w, nd.c.x, nd.c.y, nd.c.z, nd.c.w, thi, tr);
        if (hl && nd.d.x < 0) {
            const int k = ~nd.d.x;
            if (nd.d.z == fpid && k != lo && k != hi) {
                const TriVerts t = tv[k];
                if (wray_tri_t(w, xyz(t.a), xyz(t.b), xyz(t.c), tk) && (tk < thi || (tk == thi && k < hi))) return true;
            }
            hl = false;
        }
        if (hr && nd.d.y < 0) {
            const int k = ~nd.d.y;
            if (nd.d.w == fpid && k != lo && k != hi) {
                const TriVerts t = tv[k];
                if (wray_tri_t(w, xyz(t.a), xyz(t.b), xyz(t.c), tk) && (tk < thi || (tk == thi && k < hi))) return true;
            }
            hr = false;
        }
        if (hl && hr) { DZ_ASSERT(sp < 64); stack[sp++] = nd.d.y; cur = nd.d.x; }
        else if (hl) cur = nd.d.x;
        else if (hr) cur = nd.d.y;
        else {
            if (sp == 0) break;
            cur = stack[--sp];
        }
    }
    return false;
}
__device__ __forceinline__ uint64_t pair_mask_warp(const TriVerts *__restrict__ tv, const float4 *__restrict__ tribox,
                                                   const TriVerts &Tlo, const TriVerts &Thi, int lo, int hi, const int *cand,
                                                   int n_main, unsigned long long fmask, const FaceTables &ft, int own_lo, float h_lo, int own_hi, float h_hi, int own_pid_lo, int own_pid_hi,
                                                   const int *nbr_lo, const int *nbr_hi, int n_inner, float m_req, const float *s_uv, const unsigned char *s_perm, int S, int lane, int *wk, float4 *wb) {
    unsigned mask_lo = 0, mask_hi = 0;
    for (int pass = 0; pass * 32 < S; pass++) {
        const int i = pass * 32 + lane;
        const int ii = min(i, S - 1);
        const float u = s_uv[2 * ii], v = s_uv[2 * ii + 1];
        f3 a0 = xyz(Tlo.a), a1 = xyz(Thi.a);
        f3 org = e_add(e_add(a0, e_scale(e_sub(xyz(Tlo.b), a0), u)), e_scale(e_sub(xyz(Tlo.c), a0), v));
        f3 dst = e_add(e_add(a1, e_scale(e_sub(xyz(Thi.b), a1), u)), e_scale(e_sub(xyz(Thi.c), a1), v));
        f3 dir = e_normalize(e_sub(dst, org));
        f3 o = e_add(org, e_scale(dir, 0.000001f));
        WRay w = wray_setup(o, dir);
        float thi = 0.f, tk;
        bool alive = (i < S) && wray_tri_t(w, xyz(Thi.a), xyz(Thi.b), xyz(Thi.c), thi);
        if (alive && wray_tri_t(w, xyz(Tlo.a), xyz(Tlo.b), xyz(Tlo.c), tk) && tk <= thi) alive = false;
        // Face grids first: one plane crossing and one cell lookup per (ray, face).  A covered cell crossed safely between the
        // ray's end points blocks the ray (some triangle of the face accepts it, faces.cu); an empty cell or a crossing beyond
        // the end points cannot; everything else runs the watertight test on the cell's own short list.
        const float mg = fminf(fminf(u, v), 1.0f - u - v);
        if (fmask) {
            unsigned long long fm = fmask;
            bool any = __any_sync(0xffffffffu, alive);
            while (fm && any) {
                const int f = __ffsll((long long)fm) - 1;
                fm &= fm - 1;
                const float4 pl = __ldg(&ft.faces[f].pl);
                const float ndir = pl.x * dir.x + pl.y * dir.y + pl.z * dir.z;
                const float norg = pl.x * o.x + pl.y * o.y + pl.z * o.z;
                const float s0 = norg - pl.w; // signed distance of the origin
                // The face is the plane of lo or hi itself and the pair as a whole did not qualify for coplanar skipping (one ray
                // is too flat, pair_premise): the premise is checked ray by ray instead -- a ray that leaves lo (reaches hi) at
                // |cos| = |ndir| from a sample with barycentric margin mg cannot touch a coplanar neighbour once
                // mg >= 128 eps (32 / cos) on the origin side, mg >= 128 eps (length + 64 h) / (h cos) on the far side
                // (same bounds as pair_premise; h > 0 only for patches k_tri_planes qualified).
                const bool act = alive && !(f == own_lo && mg * fabsf(ndir) >= 2.44e-4f) &&
                                 !(f == own_hi && mg * fabsf(ndir) * h_hi >= 7.63e-6f * (thi + 64.f * h_hi));
                if (act && fabsf(ndir) < FACE_COS_MIN) {
                    // Flat ray: it can only touch triangles of the face where it runs within eps of the plane.  That stretch
                    // [ta, tb] of the ray is usually empty (both end points clear of the plane on one side) or short (the ray
                    // leaves from / arrives on / skims the plane near one end): the lists of the few cells under it are tested.
                    // A long stretch (a ray lying in the plane) searches the face through the LBVH.
                    float ta = 0.f, tb = -1.f;
                    if (fabsf(ndir) > 1e-12f) {
                        const float r = __fdividef(1.0f, ndir), tc = -s0 * r, hw = ft.eps * fabsf(r);
                        ta = fmaxf(tc - hw, 0.f); tb = fminf(tc + hw, thi);
                    } else if (fabsf(s0) <= ft.eps) tb = thi;
                    if (ta <= tb) {
#ifdef DAISY_FF_STATS
                        atomicAdd(&g_ffstats[(f + 1 == own_pid_lo || f + 1 == own_pid_hi) ? 35 : 36], 1ull);
#endif
                        const float4 ex = __ldg(&ft.faces[f].ex), ey = __ldg(&ft.faces[f].ey);
                        const int4 g = __ldg(&ft.faces[f].g);
                        const float Xa = fmaf(ta, dir.x, o.x), Ya = fmaf(ta, dir.y, o.y), Za = fmaf(ta, dir.z, o.z);
                        const float Xb = fmaf(tb, dir.x, o.x), Yb = fmaf(tb, dir.y, o.y), Zb = fmaf(tb, dir.z, o.z);
                        const float a0 = fmaf(Xa, ex.x, fmaf(Ya, ex.y, fmaf(Za, ex.z, ex.w))), b0 = fmaf(Xa, ey.x, fmaf(Ya, ey.y, fmaf(Za, ey.z, ey.w)));
                        const float a1 = fmaf(Xb, ex.x, fmaf(Yb, ex.y, fmaf(Zb, ex.z, ex.w))), b1 = fmaf(Xb, ey.x, fmaf(Yb, ey.y, fmaf(Zb, ey.z, ey.w)));
                        const int ia0 = max(0, (int)floorf(fminf(a0, a1))), ia1 = min(g.x - 1, (int)floorf(fmaxf(a0, a1)));
                        const int ib0 = max(0, (int)floorf(fminf(b0, b1))), ib1 = min(g.y - 1, (int)floorf(fmaxf(b0, b1)));
                        if (ia0 <= ia1 && ib0 <= ib1) {
                            if ((ia1 - ia0) + (ib1 - ib0) <= 1000) {
                                // the cells under the stretch, column by column (the b-range of the stretch inside a column, widened
                                // by a hundredth of a cell); a triangle tested a moment ago is not tested again
                                const float da = a1 - a0, rda = (fabsf(da) > 1e-6f) ? __fdividef(b1 - b0, da) : 0.f;
                                int prev1 = -1, prev2 = -1;
                                for (int ia = ia0; ia <= ia1 && alive; ia++) {
                                    int jb0 = ib0, jb1 = ib1;
                                    if (ia0 != ia1 && fabsf(da) > 1e-6f) {
                                        const float ca0 = fminf(fmaxf((float)ia, fminf(a0, a1)), fmaxf(a0, a1)), ca1 = fminf(fmaxf((float)(ia + 1), fminf(a0, a1)), fmaxf(a0, a1));
                                        const float cb0 = fmaf(ca0 - a0, rda, b0), cb1 = fmaf(ca1 - a0, rda, b0);
                                        jb0 = max(ib0, (int)floorf(fminf(cb0, cb1) - 0.01f)); jb1 = min(ib1, (int)floorf(fmaxf(cb0, cb1) + 0.01f));
                                    }
                                    for (int ib = jb0; ib <= jb1 && alive; ib++) {
                                        DZ_ASSERT(ia >= 0 && ia < g.x && ib >= 0 && ib < g.y && (int64_t)g.z + (int64_t)ib * g.x + ia < ft.ncells);
                                        const int c = __ldg(ft.cells + g.z + ib * g.x + ia);
                                        if (c < 0) continue;
                                        const int *L = ft.lists + (c >> 1);
                                        const int n = __ldg(L);
                                        DZ_ASSERT((int64_t)(c >> 1) + n < ft.nlist && n > 0);
                                        for (int q = 1; q <= n; q++) {
                                            const int k = __ldg(L + q);
                                            if (k == lo || k == hi || k == prev1 || k == prev2) continue;
                                            prev2 = prev1; prev1 = k;
#ifdef DAISY_FF_STATS
                                            atomicAdd(&g_ffstats[23], 1ull);
#endif
                                            const TriVerts tr = tv[k];
                                            if (wray_tri_t(w, xyz(tr.a), xyz(tr.b), xyz(tr.c), tk) && (tk < thi || (tk == thi && k < hi))) { alive = false; break; }
                                        }
                                    }
                                }
                            } else {
#ifdef DAISY_FF_STATS
                                atomicAdd(&g_ffstats[19], 1ull);
#endif
                                if (face_blocks_ray(ft.nodes, tv, ft.root, w, dir, thi, lo, hi, f + 1)) alive = false;
                            }
                        }
                    }
                }
                const float t = __fdividef(-s0, ndir);
                if (act && alive && fabsf(ndir) >= FACE_COS_MIN && t > -ft.tm && t < thi + ft.tm) {
                    const float4 ex = __ldg(&ft.faces[f].ex), ey = __ldg(&ft.faces[f].ey);
                    const int4 g = __ldg(&ft.faces[f].g);
                    const float X = fmaf(t, dir.x, o.x), Y = fmaf(t, dir.y, o.y), Z = fmaf(t, dir.z, o.z);
                    const float ca = fmaf(X, ex.x, fmaf(Y, ex.y, fmaf(Z, ex.z, ex.w)));
                    const float cb = fmaf(X, ey.x, fmaf(Y, ey.y, fmaf(Z, ey.z, ey.w)));
                    if (ca >= 0.f && cb >= 0.f && ca < (float)g.x && cb < (float)g.y) {
                        DZ_ASSERT((int)ca >= 0 && (int)ca < g.x && (int)cb >= 0 && (int)cb < g.y && (int64_t)g.z + (int64_t)(int)cb * g.x + (int)ca < ft.ncells);
                        const int c = __ldg(ft.cells + g.z + (int)cb * g.x + (int)ca);
#ifdef DAISY_FF_STATS
                        atomicAdd(&g_ffstats[15], 1ull);
#endif
#ifdef DAISY_FF_STATS
                        if (c < 0) atomicAdd(&g_ffstats[38], 1ull);
                        else if ((c & 1) && t > ft.tm && t < thi - ft.tm) atomicAdd(&g_ffstats[37], 1ull);
                        else atomicAdd(&g_ffstats[(f + 1 == own_pid_lo || f + 1 == own_pid_hi) ? 32 : ((c & 1) ? 34 : 33)], 1ull);
#endif
                        if (c >= 0) {
                            if ((c & 1) && t > ft.tm && t < thi - ft.tm) alive = false;
                            else {
                                const int *L = ft.lists + (c >> 1);
                                const int n = __ldg(L);
                                DZ_ASSERT(n > 0 && (int64_t)(c >> 1) + n < ft.nlist);
                                for (int q = 1; q <= n; q++) {
                                    const int k = __ldg(L + q);
                                    if (k == lo || k == hi) continue;
#ifdef DAISY_FF_STATS
                                    atomicAdd(&g_ffstats[14], 1ull);
#endif
                                    const TriVerts tr = tv[k];
                                    if (wray_tri_t(w, xyz(tr.a), xyz(tr.b), xyz(tr.c), tk) && (tk < thi || (tk == thi && k < hi))) { alive = false; break; }
                                }
                            }
                        }
                    }
                }
                any = __any_sync(0xffffffffu, alive);
            }
        }
        // neighbour lists are needed by the samples closer to an edge than the pair's required margin (see below)
        unsigned edge = 0;
        if ((nbr_lo || nbr_hi) && pass * 32 + 31 >= n_inner) edge = __ballot_sync(0xffffffffu, alive && i >= n_inner && mg < m_req);
        // reciprocal direction (only the slab tests of the candidate list use it), kept finite: with
        // inv = inf the pre-multiplied form would turn a box that straddles 0 on an axis the ray is parallel to into (-inf, NaN)
        // and reject it
        f3 inv = mk3(0.f, 0.f, 0.f), oi = inv;
        bool neg_x = false, neg_y = false, neg_z = false, sorted = false;
        if (n_main > 0) {
            inv = mk3(1.0f / (fabsf(dir.x) > 1e-30f ? dir.x : copysignf(1e-30f, dir.x)), 1.0f / (fabsf(dir.y) > 1e-30f ? dir.y : copysignf(1e-30f, dir.y)),
                      1.0f / (fabsf(dir.z) > 1e-30f ? dir.z : copysignf(1e-30f, dir.z)));
            oi = mk3(o.x * inv.x, o.y * inv.y, o.z * inv.z);
            // Slab tests run in lock step over the list (uniform box loads); a lane that passes one only QUEUES the
            // triangle.  The expensive watertight tests are then issued for whole queues at a time, so a warp instruction
            // slot is spent on them only when many lanes have one pending, not whenever a single lane does.
            // do all rays of this pass enter every box through the same three planes?  (same signs of the direction components)
            const unsigned act = __ballot_sync(0xffffffffu, i < S);
            const unsigned bx = __ballot_sync(0xffffffffu, i < S && inv.x < 0.f), by = __ballot_sync(0xffffffffu, i < S && inv.y < 0.f),
                           bz = __ballot_sync(0xffffffffu, i < S && inv.z < 0.f);
            neg_x = bx != 0; neg_y = by != 0; neg_z = bz != 0;
            sorted = (bx == 0 || bx == act) && (by == 0 || by == act) && (bz == 0 || bz == act);
        }
        int qlen = 0;
        unsigned qreg = 0; // queued candidates: 4-bit positions inside the staged chunk of 16
        auto flush = [&]() {
#ifdef DAISY_FF_STATS
            {
                const int T = __reduce_add_sync(0xffffffffu, alive ? qlen : 0);
                if (lane == 0 && T) { atomicAdd(&g_ffstats[20], (unsigned long long)((T + 31) / 32)); atomicAdd(&g_ffstats[21], (unsigned long long)T); }
            }
#endif
            for (int t = 0; t < FF_QCAP; t++) {
                if (!__any_sync(0xffffffffu, alive && t < qlen)) break;
#ifdef DAISY_FF_STATS
                if (lane == 0) atomicAdd(&g_ffstats[22], 1ull);
#endif
                if (alive && t < qlen) {
                    const int k = wk[(qreg >> (4 * t)) & 15];
                    DZ_ASSERT(k >= 0 && qlen <= FF_QCAP);
                    TriVerts tr = tv[k];
                    if (wray_tri_t(w, xyz(tr.a), xyz(tr.b), xyz(tr.c), tk) && (tk < thi || (tk == thi && k < hi))) alive = false;
                }
            }
            qlen = 0;
            qreg = 0;
        };
#ifdef DAISY_FF_STATS
        int dbg_iters = 0;
#endif
        {
            bool any_alive = __any_sync(0xffffffffu, alive);
            for (int c0 = 0; c0 < n_main && any_alive; c0 += 16) {
                // stage 16 candidates (id + padded box) in the warp's shared-memory slot: the list was written by another lane
                // of this warp, so it is read through L2 (ld.global.cg); the boxes are then broadcast LDS.128 in the loop
                const int nb = min(16, n_main - c0);
                __syncwarp();
                if (lane < nb) {
                    const int k = __ldcg(cand + c0 + lane);
                    DZ_ASSERT(k >= 0 && c0 + lane < SHAFT_CAP);
                    wk[lane] = k;
                    const float4 lo4 = tribox[2 * (size_t)k], hi4 = tribox[2 * (size_t)k + 1];
                    // rays of one sign pattern (nearly always: they are almost parallel): entry planes first, exit planes second
                    wb[2 * lane] = sorted ? make_float4(neg_x ? hi4.x : lo4.x, neg_y ? hi4.y : lo4.y, neg_z ? hi4.z : lo4.z, 0.f) : lo4;
                    wb[2 * lane + 1] = sorted ? make_float4(neg_x ? lo4.x : hi4.x, neg_y ? lo4.y : hi4.y, neg_z ? lo4.z : hi4.z, 0.f) : hi4;
                }
                __syncwarp();
                for (int j0 = 0; j0 < nb; j0 += FF_QCAP) {
#pragma unroll
                    for (int jj = 0; jj < FF_QCAP; jj++) {
                        const int j = j0 + jj;
                        if (j < nb) {
                            const float4 b0 = wb[2 * j], b1 = wb[2 * j + 1];
                            const bool near_enough = sorted ? ray_box_sorted(oi, inv, b0.x, b0.y, b0.z, b1.x, b1.y, b1.z, thi)
                                                           : ray_box_fma(oi, inv, b0.x, b0.y, b0.z, b1.x, b1.y, b1.z, thi);
                            if (alive && near_enough) { qreg |= (unsigned)j << (4 * qlen); qlen++; }
                        }
                    }
#ifdef DAISY_FF_STATS
                    dbg_iters += min(FF_QCAP, nb - j0);
#endif
                    flush(); // at most FF_QCAP entries were queued since the last flush
                    any_alive = __any_sync(0xffffffffu, alive);
                    if (!any_alive) break;
                }
            }
        }
        // Neighbour lists (triangles in the plane of lo / hi next to the patch, null if that side's premise does not hold):
        // only samples closer to an edge of their triangles than the pair's required margin have to test them.  They are few
        // (usually 0-3 of 50), so the roles flip: the edge sample's ray is broadcast and lane = neighbour.
        {
            edge &= __ballot_sync(0xffffffffu, alive); // the candidate list may have settled some of them meanwhile
            if (edge) {
                // lane < n_lo: neighbour of lo; n_lo <= lane < n_lo + n_hi: neighbour of hi (NBR_CAP - 1 <= 31 each: two rounds at most)
                const int n_lo = nbr_lo ? __ldg(nbr_lo) : 0, n_hi = nbr_hi ? __ldg(nbr_hi) : 0;
                for (int c0 = 0; c0 < n_lo + n_hi; c0 += 32) {
                    const int c = c0 + lane;
                    int k = -1;
                    if (c < n_lo) k = __ldg(nbr_lo + 1 + c);
                    else if (c < n_lo + n_hi) k = __ldg(nbr_hi + 1 + (c - n_lo));
                    float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
                    if (k >= 0) { b0 = tribox[2 * (size_t)k]; b1 = tribox[2 * (size_t)k + 1]; }
                    unsigned todo = edge;
                    while (todo) {
                        const int e = __ffs(todo) - 1;
                        todo &= todo - 1;
                        WRay we;
                        we.o.x = __shfl_sync(0xffffffffu, w.o.x, e); we.o.y = __shfl_sync(0xffffffffu, w.o.y, e); we.o.z = __shfl_sync(0xffffffffu, w.o.z, e);
                        we.perm = __shfl_sync(0xffffffffu, w.perm, e); we.kx = we.ky = we.kz = 0; // the select-based test reads perm only
                        we.Sx = __shfl_sync(0xffffffffu, w.Sx, e); we.Sy = __shfl_sync(0xffffffffu, w.Sy, e); we.Sz = __shfl_sync(0xffffffffu, w.Sz, e);
                        // reciprocal direction of the broadcast ray (a conservative box filter: the fast reciprocal's 2 ulp are far
                        // inside the slab test's 1e-5 slack), kept finite as above
                        const f3 dre = mk3(__shfl_sync(0xffffffffu, dir.x, e), __shfl_sync(0xffffffffu, dir.y, e), __shfl_sync(0xffffffffu, dir.z, e));
                        const f3 inve = mk3(__fdividef(1.0f, fabsf(dre.x) > 1e-30f ? dre.x : copysignf(1e-30f, dre.x)),
                                            __fdividef(1.0f, fabsf(dre.y) > 1e-30f ? dre.y : copysignf(1e-30f, dre.y)),
                                            __fdividef(1.0f, fabsf(dre.z) > 1e-30f ? dre.z : copysignf(1e-30f, dre.z)));
                        const f3 oie = mk3(we.o.x * inve.x, we.o.y * inve.y, we.o.z * inve.z);
                        const float thie = __shfl_sync(0xffffffffu, thi, e);
                        bool hit = false;
                        if (k >= 0 && ray_box_fma(oie, inve, b0.x, b0.y, b0.z, b1.x, b1.y, b1.z, thie)) {
                            const TriVerts tr = tv[k];
                            float t2;
                            if (wray_tri_t(we, xyz(tr.a), xyz(tr.b), xyz(tr.c), t2) && (t2 < thie || (t2 == thie && k < hi))) hit = true;
                        }
                        if (__any_sync(0xffffffffu, hit)) { if (lane == e) alive = false; edge &= ~(1u << e); }
                    }
                }
            }
        }
#ifdef DAISY_FF_STATS
        if (lane == 0) atomicAdd(&g_ffstats[16 + pass], (unsigned long long)dbg_iters);
#endif
        // bit position = the caller's sample index
        const int bit = s_perm[ii];
        const unsigned lo_bit = (alive && bit < 32) ? (1u << bit) : 0u, hi_bit = (alive && bit >= 32) ? (1u << (bit - 32)) : 0u;
        mask_lo |= __reduce_or_sync(0xffffffffu, lo_bit);
        mask_hi |= __reduce_or_sync(0xffffffffu, hi_bit);
    }
    return (uint64_t)mask_lo | ((uint64_t)mask_hi << 32);
}

// ---------------------------------------------------------------------------------------------------------
// Matrix updates after a geometry change (daisy_formfactors_update; DESIGN "Updating the matrix after a geometry change").
// A pair whose two patches did not change keeps its entry unless a ray of the pair can be accepted by a moved triangle in the
// recorded or in the current geometry; by the premise of the shaft culling above that needs the triangle's padded box in that
// geometry to meet the pair's shaft.  The dirty boxes are those padded boxes, grouped into clusters.
#define UPD_CAP 16 // dirty clusters listed per tile; a tile whose shaft meets more treats every pair as dirty

// does the pair's shaft meet one of the dirty boxes listed for its tile?  (list: UPD_CAP + 1 ints, see FFParams::tile_dirty)
__device__ __noinline__ bool pair_meets_dirty(const int *__restrict__ list, const TriVerts *__restrict__ tv, const float4 *__restrict__ cbox,
                                              const int2 *__restrict__ crange, const float4 *__restrict__ leaf, int lo, int hi) {
    const int n = __ldg(list);
    if (n < 0) return true;
    const Shaft sh = make_shaft(tv[lo], tv[hi]);
    for (int i = 0; i < n; i++) {
        const int k = __ldg(list + 1 + i);
        const float4 b0 = __ldg(cbox + 2 * k), b1 = __ldg(cbox + 2 * k + 1);
        if (!shaft_box(sh, b0.x, b0.y, b0.z, b1.x, b1.y, b1.z)) continue;
        const int2 r = __ldg(crange + k);
        for (int j = r.x; j < r.y; j++) {
            const float4 l0 = __ldg(leaf + 2 * j), l1 = __ldg(leaf + 2 * j + 1);
            if (shaft_box(sh, l0.x, l0.y, l0.z, l1.x, l1.y, l1.z)) return true;
        }
    }
    return false;
}

// warp + block reduction of 6 values over the 128 threads of k_ff_classify (op 0 = min, 1 = max, 2 = sum per value)
__device__ __forceinline__ void block_reduce6(float v[6], const int op[6], float (*s_red)[6]) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < 6; q++)
        for (int o = 16; o > 0; o >>= 1) {
            const float x = __shfl_xor_sync(0xffffffffu, v[q], o);
            v[q] = op[q] == 0 ? fminf(v[q], x) : (op[q] == 1 ? fmaxf(v[q], x) : v[q] + x);
        }
    __syncthreads(); // s_red free for reuse
    if (lane == 0)
        for (int q = 0; q < 6; q++) s_red[w][q] = v[q];
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 6; q++) {
        float a = s_red[0][q];
        for (int j = 1; j < 4; j++) a = op[q] == 0 ? fminf(a, s_red[j][q]) : (op[q] == 1 ? fmaxf(a, s_red[j][q]) : a + s_red[j][q]);
        v[q] = a;
    }
}

// One CTA of 128 threads per job (the two slot groups of the tile, one slot per thread).  A tile is kept if a slot holds a
// changed triangle or if the shaft of the whole tile -- the convex hull of all the vertices of both groups, tested like a
// pair's shaft with D = the difference of the two groups' mean vertices -- meets a dirty cluster.  Kept jobs are appended
// (in no particular order: the tile kernel schedules them dynamically anyway) with the clusters their shaft meets.
__global__ void __launch_bounds__(128) k_ff_classify(const int2 *__restrict__ jobs, int njobs, const int *__restrict__ order,
                                                     const TriVerts *__restrict__ tv, const unsigned char *__restrict__ changed,
                                                     const float4 *__restrict__ cbox, int nclusters, int2 *__restrict__ kept_jobs,
                                                     int *__restrict__ kept_lists, int *__restrict__ kept_count) {
    __shared__ float s_red[4][6];
    __shared__ int s_n, s_any, s_slot;
    __shared__ int s_list[UPD_CAP];
    const int tid = threadIdx.x;
    for (int job = blockIdx.x; job < njobs; job += gridDim.x) {
        const int2 jt = jobs[job];
        if (tid == 0) { s_n = 0; s_any = 0; }
        __syncthreads();
        const int t = order[(tid < TILE ? jt.x * TILE : jt.y * TILE - TILE) + tid];
        TriVerts T = {};
        if (t >= 0) T = tv[t];
        if (t >= 0 && changed[t]) s_any = 1; // benign race: every writer stores 1
        const float4 p[3] = { T.a, T.b, T.c };
        float v[6];
        const int mnmx[6] = { 0, 0, 0, 1, 1, 1 }, sums[6] = { 2, 2, 2, 2, 2, 2 };
        v[0] = v[1] = v[2] = INFINITY; v[3] = v[4] = v[5] = -INFINITY;
        if (t >= 0)
            for (int i = 0; i < 3; i++) {
                v[0] = fminf(v[0], p[i].x); v[1] = fminf(v[1], p[i].y); v[2] = fminf(v[2], p[i].z);
                v[3] = fmaxf(v[3], p[i].x); v[4] = fmaxf(v[4], p[i].y); v[5] = fmaxf(v[5], p[i].z);
            }
        block_reduce6(v, mnmx, s_red);
        Shaft sh;
        sh.lox = v[0]; sh.loy = v[1]; sh.loz = v[2]; sh.hix = v[3]; sh.hiy = v[4]; sh.hiz = v[5];
        // group means: sums of vertices (row group in 0..2, column group in 3..5) and counts
        float m[6] = { 0.f, 0.f, 0.f, 0.f, 0.f, 0.f };
        if (t >= 0) {
            const int o = tid < TILE ? 0 : 3;
            m[o] = p[0].x + p[1].x + p[2].x; m[o + 1] = p[0].y + p[1].y + p[2].y; m[o + 2] = p[0].z + p[1].z + p[2].z;
        }
        block_reduce6(m, sums, s_red);
        float cnt[6] = { (t >= 0 && tid < TILE) ? 3.f : 0.f, (t >= 0 && tid >= TILE) ? 3.f : 0.f, 0.f, 0.f, 0.f, 0.f };
        block_reduce6(cnt, sums, s_red);
        // any direction D gives a valid separating axis for the hull; the one between the groups' means separates best
        sh.Dx = cnt[0] > 0.f && cnt[1] > 0.f ? m[3] / cnt[1] - m[0] / cnt[0] : 0.f;
        sh.Dy = cnt[0] > 0.f && cnt[1] > 0.f ? m[4] / cnt[1] - m[1] / cnt[0] : 0.f;
        sh.Dz = cnt[0] > 0.f && cnt[1] > 0.f ? m[5] / cnt[1] - m[2] / cnt[0] : 0.f;
        float c[6] = { INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY };
        const int cmm[6] = { 0, 0, 0, 1, 1, 1 };
        if (t >= 0)
            for (int i = 0; i < 3; i++) {
                const float q0 = p[i].y * sh.Dz - p[i].z * sh.Dy, q1 = p[i].z * sh.Dx - p[i].x * sh.Dz, q2 = p[i].x * sh.Dy - p[i].y * sh.Dx;
                c[0] = fminf(c[0], q0); c[1] = fminf(c[1], q1); c[2] = fminf(c[2], q2);
                c[3] = fmaxf(c[3], q0); c[4] = fmaxf(c[4], q1); c[5] = fmaxf(c[5], q2);
            }
        block_reduce6(c, cmm, s_red);
        sh.c0min = c[0]; sh.c1min = c[1]; sh.c2min = c[2]; sh.c0max = c[3]; sh.c1max = c[4]; sh.c2max = c[5];
        for (int i = tid; i < nclusters; i += blockDim.x) {
            const float4 b0 = __ldg(cbox + 2 * i), b1 = __ldg(cbox + 2 * i + 1);
            if (shaft_box(sh, b0.x, b0.y, b0.z, b1.x, b1.y, b1.z)) {
                const int k = atomicAdd(&s_n, 1);
                if (k < UPD_CAP) s_list[k] = i;
            }
        }
        __syncthreads();
        const int n = s_n;
        if (tid == 0 && (s_any || n > 0)) {
            s_slot = atomicAdd(kept_count, 1);
            kept_jobs[s_slot] = jt;
        }
        __syncthreads();
        if (s_any || n > 0) {
            int *L = kept_lists + (size_t)s_slot * (UPD_CAP + 1);
            if (tid == 0) L[0] = n > UPD_CAP ? -1 : n;
            if (tid < n && tid < UPD_CAP) L[1 + tid] = s_list[tid];
        }
        __syncthreads();
    }
}

struct FFParams {
    const PatchGeom *geom;
    const TriVerts *tv;
    const BvhNode *nodes;
    const float4 *tribox; // padded triangle boxes, 2 float4 per triangle
    const float4 *plane;  // per-triangle plane record (k_tri_planes)
    const int *pid;       // per-triangle plane id (0 = none)
    const int *nbr;       // per-triangle neighbour list in its own plane: NBR_CAP ints, [0] = count (k_tri_planes)
    const DzFace *faces;  // planar face grids (faces.cu): face f = plane id f + 1
    const int *face_cells, *face_lists;
    int nfaces;
    int64_t face_ncells, face_nlist;
    float face_tm;
    const int *order;     // tile composition: slot -> triangle id (-1 = empty slot); tile T holds slots [64 T, 64 T + 64)
    int n_inner;          // samples [0, n_inner) of the device-order pattern are inner samples
    int ring_on;          // coplanar skipping enabled
    int all_heavy;        // the sample pattern leaves the triangle: no culling of any kind, per-ray LBVH walks for every pair
    int *scratch;         // gridDim.x * FF_THREADS * SHAFT_CAP candidate slots
    int root, N, S;
    int row0, row1;      // rows this context owns
    float *F;            // (row1-row0) x ldF, may be null (mask-only run)
    int64_t ldF;
    // peer mode (multi-GPU): every upper-triangle tile is computed by exactly one rank, which stores every entry into the
    // row owner's F -- its own memory or a peer's, mapped through CUDA IPC and written over NVLink
    int peer_mode, n_per_rank;
    float *Fpeer[16];
    uint64_t *masks;     // optional (mrow1-mrow0) x N
    int mrow0, mrow1;
    int ntiles;          // tiles per side
    int *job_counter;    // dynamic tile scheduler
    unsigned long long *pair_counter; // [0] pairs traced by this context, [1] of those, pairs whose lower index it owns, [2] pairs that fell back to per-ray LBVH walks
    int njobs;
    const int2 *jobs;    // (row tile, col tile), col tile >= row tile
    // update runs (PARTIAL, see dz_build_formfactors): the dirty set and, per job, the dirty clusters its tile's shaft meets
    DzUpdate upd;
    const int *tile_dirty; // (UPD_CAP + 1) ints per job: count (-1 = more than UPD_CAP: every pair of the tile is dirty), cluster ids
    float uv[2 * DAISY_MAX_SAMPLES];      // sample pattern in device order (samples_device_order)
    unsigned char perm[DAISY_MAX_SAMPLES]; // device position -> caller's sample index
};

// Tile slots: [0, 64) = the row-tile's patches, [64, 128) = the column-tile's patches.  A listed pair is (rl, cl) plus a
// swap bit: visibility rays always run from the patch with the LOWER triangle id to the one with the higher id
// (OptixPrimeFunctionality.cpp:186-196, row < col), whatever slots the two occupy.
#define PAIR_SWAP 0x1000
#define PAIR_HEAVY 0x2000
struct FFSmem {
    // phase 1 (sub-patch records of the row / column patches) and phase 2 (per-warp candidate staging) never overlap in
    // time, so they share storage: three CTAs fit one SM
    union {
        struct { PatchGeom g[2 * TILE]; } p1;
        struct {
            int wk[FF_THREADS / 32][16];
            float4 wb[FF_THREADS / 32][32];
            TriVerts tv[2 * TILE]; // vertices of the tile's patches (staged after phase 1)
        } p2;
    } u;
    float area[2 * TILE]; // patch areas (needed after phase 1 by the host-variant reciprocity rule)
    float4 pl[2 * TILE];  // plane records
    int pid[2 * TILE];    // exact plane ids
    int id[2 * TILE];     // triangle ids of the slots, -1 = empty
    unsigned char perm[DAISY_MAX_SAMPLES];
    float rc[TILE][TILE + 1]; // F(r->c), indexed [rl][cl]
    float cr[TILE][TILE + 1]; // F(c->r), indexed [cl][rl]
    unsigned short list[TILE * TILE];
    int nlist, next, job, nown, nheavy, hnext;
    float uv[2 * DAISY_MAX_SAMPLES];
};

#ifdef DAISY_FF_STATS
#define FF_CLK(slot)                                                                           \
    do {                                                                                       \
        const long long now_ = clock64();                                                      \
        if (lane == 0) atomicAdd(&g_ffstats[24 + (slot)], (unsigned long long)(now_ - clk_)); \
        clk_ = now_;                                                                           \
    } while (0)
#else
#define FF_CLK(slot) do { } while (0)
#endif

// PARTIAL: an update run -- only the dirty pairs of a tile are traced and stored (pairs with a changed patch, and facing pairs
// whose shaft meets a dirty box listed for the tile); every other entry of F is left as it is.
#define UPD_KEEP 0x7fa5a5a5 // bit pattern of a tile entry an update does not store (a NaN no computation produces)
template <int VARIANT, bool PARTIAL>
__global__ void __launch_bounds__(FF_THREADS, FF_MINBLOCKS) k_ff_tiles(FFParams P) {
    extern __shared__ __align__(16) unsigned char ff_smem_raw[];
    FFSmem &sm = *reinterpret_cast<FFSmem *>(ff_smem_raw);
    PatchGeom *s_g = sm.u.p1.g;
    TriVerts *s_tv = sm.u.p2.tv;
    float(*s_rc)[TILE + 1] = sm.rc;
    float(*s_cr)[TILE + 1] = sm.cr;
    unsigned short *s_list = sm.list;
    int &s_nlist = sm.nlist, &s_next = sm.next, &s_job = sm.job, &s_nown = sm.nown, &s_nheavy = sm.nheavy, &s_hnext = sm.hnext;
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    if (tid < 2 * DAISY_MAX_SAMPLES) sm.uv[tid] = P.uv[tid];
    if (tid < DAISY_MAX_SAMPLES) sm.perm[tid] = P.perm[tid];
    int *my_cand = P.scratch + ((size_t)blockIdx.x * FF_THREADS + tid) * SHAFT_CAP;
    int *warp_cand = P.scratch + ((size_t)blockIdx.x * FF_THREADS + (tid & ~31)) * SHAFT_CAP;
#ifdef DAISY_FF_STATS
    long long clk_ = clock64();
#endif

    while (true) {
        if (tid == 0) s_job = atomicAdd(P.job_counter, 1);
        __syncthreads();
        int job = s_job;
        if (job >= P.njobs) break;
        int2 jt = P.jobs[job];
        const int R0 = jt.x * TILE, C0 = jt.y * TILE;
        const bool diag = (jt.x == jt.y);
        if (tid == 0) { s_nlist = 0; s_next = 0; s_nown = 0; s_nheavy = 0; s_hnext = 0; }
        // stage the two patch groups (float4-granular copies: 5 + 3 float4 per patch); empty slots read triangle 0 and are
        // masked out by id < 0
        if (tid < 2 * TILE) {
            const int t = P.order[(tid < TILE ? R0 : C0 - TILE) + tid];
            DZ_ASSERT(t >= -1 && t < P.N);
            const int tt = max(t, 0);
            sm.id[tid] = t;
            sm.pl[tid] = P.plane[tt];
            sm.area[tid] = P.geom[tt].n.w;
            sm.pid[tid] = P.pid[tt];
        }
        for (int i = tid; i < 2 * TILE * 5; i += FF_THREADS) {
            const int p = i / 5, q = i - p * 5;
            const int t = max(P.order[(p < TILE ? R0 : C0 - TILE) + p], 0);
            ((float4 *)&s_g[p])[q] = ((const float4 *)&P.geom[t])[q];
        }
        __syncthreads();

        // ---- phase 1: unoccluded form factors of every unordered pair of the tile (each once); facing pairs go on the list
        _Pragma("unroll 1") for (int idx = tid; idx < TILE * TILE; idx += FF_THREADS) {
            const int rl = idx >> 6, cl = idx & 63;
            const int r = sm.id[rl], c = sm.id[TILE + cl];
            const bool valid = (r >= 0) && (c >= 0) && (diag ? rl < cl : true) &&
                               (P.peer_mode || (r >= P.row0 && r < P.row1) || (c >= P.row0 && c < P.row1));
            float f_rc = 0.0f, f_cr = 0.0f;
            bool trace = false;
            if (valid) {
                ff_pair<VARIANT>(s_g[rl], s_g[TILE + cl], f_rc, f_cr);
                // calculateRow stores the value only when > 0 (parallellism.cu:101-107)
                f_rc = (f_rc > 0.0f) ? f_rc : 0.0f;
                f_cr = (f_cr > 0.0f) ? f_cr : 0.0f;
                // cuda path: traced iff tripletlist[row*N+col].m_value > 0 with row < col (OptixPrimeFunctionality.cpp:190),
                // i.e. the factor from the lower to the higher triangle id; per-pair path: every pair is traced and tested
                // after the fact (:335-336) -- same matrix, since a zero unoccluded factor gives a zero entry either way
                trace = (r < c ? f_rc : f_cr) > 0.0f;
                if (!trace) { f_rc = 0.0f; f_cr = 0.0f; }
            }
            if (PARTIAL) {
                bool dirty = valid && (P.upd.changed[r] || P.upd.changed[c]);
                if (valid && !dirty && trace)
                    dirty = pair_meets_dirty(P.tile_dirty + (size_t)job * (UPD_CAP + 1), P.tv, P.upd.cbox, P.upd.crange, P.upd.leaf, min(r, c), max(r, c));
                if (!dirty) { trace = false; f_rc = __int_as_float(UPD_KEEP); f_cr = f_rc; }
            }
            s_rc[rl][cl] = f_rc;
            s_cr[cl][rl] = f_cr;
            const int lo_id = min(r, c);
            unsigned m = __ballot_sync(0xffffffffu, trace);
            unsigned mo = __ballot_sync(0xffffffffu, trace && (P.peer_mode || (lo_id >= P.row0 && lo_id < P.row1)));
            if (mo && lane == 0) atomicAdd(&s_nown, __popc(mo));
            if (m) {
                int base = 0;
                int leader = __ffs(m) - 1;
                if (lane == leader) base = atomicAdd(&s_nlist, __popc(m));
                base = __shfl_sync(0xffffffffu, base, leader);
                if (trace) { DZ_ASSERT(base + __popc(m & ((1u << lane) - 1)) < TILE * TILE); s_list[base + __popc(m & ((1u << lane) - 1))] = (unsigned short)(idx | (r > c ? PAIR_SWAP : 0)); }
            }
        }
        __syncthreads();
        const int nlist = s_nlist;
        if (nlist) { // the phase-1 records are dead: their storage now takes the vertices phase 2 works with
            for (int i = tid; i < 2 * TILE * 3; i += FF_THREADS) {
                const int p = i / 3, q = i - p * 3;
                const int t = max(sm.id[p], 0);
                ((float4 *)&s_tv[p])[q] = ((const float4 *)&P.tv[t])[q];
            }
        }
        __syncthreads();
        if (tid == 0 && nlist) { atomicAdd(P.pair_counter, (unsigned long long)nlist); atomicAdd(P.pair_counter + 1, (unsigned long long)s_nown); }
        FF_CLK(0);

        // ---- phase 2: S visibility rays per listed pair; a warp claims 32 pairs at a time, lane = pair, all lanes
        // trace sample i together (neighbouring pairs + same sample => coherent rays).  First every pair gets a
        // shaft candidate list; pairs whose list fits are resolved against it (2a), the rest walk the LBVH per ray (2b).
        auto finish_pair = [&](int rl, int cl, uint64_t mask) {
            const int r = sm.id[rl], c = sm.id[TILE + cl];
            // visibility = (#hits as float) / RAYS_PER_PATCH                 OptixPrimeFunctionality.cpp:206-211
            float visibility = fd((float)__popcll(mask), (float)P.S);
            float f_rc, f_cr;
            if (VARIANT == DAISY_FF_DEVICE) {
                // Tripl(row, col, visibility * m_value): float*double in double; setFromTriplets casts to float
                f_rc = __double2float_rn(__dmul_rn((double)visibility, (double)s_rc[rl][cl]));
                f_cr = __double2float_rn(__dmul_rn((double)visibility, (double)s_cr[cl][rl]));
            } else {
                // p2pFormfactor(lo, hi) returns formfactor*visibility (float); the entry of the higher row follows by
                // reciprocity from the lower one                                                          :165,:343
                if (r < c) {
                    f_rc = fm(s_rc[rl][cl], visibility);
                    f_cr = (f_rc > 0.0f) ? fd(fm(sm.area[rl], f_rc), sm.area[TILE + cl]) : 0.0f;
                } else {
                    f_cr = fm(s_cr[cl][rl], visibility);
                    f_rc = (f_cr > 0.0f) ? fd(fm(sm.area[TILE + cl], f_cr), sm.area[rl]) : 0.0f;
                }
            }
            if (mask == 0) { f_rc = 0.0f; f_cr = 0.0f; }
            s_rc[rl][cl] = f_rc;
            s_cr[cl][rl] = f_cr;
            if (P.masks) {
                if (r >= P.mrow0 && r < P.mrow1) P.masks[(size_t)(r - P.mrow0) * P.N + c] = mask;
                if (c >= P.mrow0 && c < P.mrow1) P.masks[(size_t)(c - P.mrow0) * P.N + r] = mask;
            }
        };
        FaceTables ftab;
        ftab.faces = P.faces; ftab.cells = P.face_cells; ftab.lists = P.face_lists; ftab.tm = P.face_tm;
        ftab.ncells = P.face_ncells; ftab.nlist = P.face_nlist;
        ftab.nodes = P.nodes; ftab.root = P.root; ftab.eps = 0.0625f * P.face_tm;
        while (true) { // 2a
            int q0 = 0;
            if (lane == 0) q0 = atomicAdd(&s_next, 32);
            q0 = __shfl_sync(0xffffffffu, q0, 0);
            if (q0 >= nlist) break;
            // (i) lane = pair: shaft walk, candidates into this lane's global scratch slot
            const int q = q0 + lane;
            int idx = 0, ncand = -2;
            float m_req = 0.f;
            unsigned long long fmask = 0;
            if (q < nlist) {
                idx = s_list[q];
                const int rl = (idx >> 6) & 63, cl = idx & 63;
                const int ilo = (idx & PAIR_SWAP) ? TILE + cl : rl, ihi = (idx & PAIR_SWAP) ? rl : TILE + cl;
                const TriVerts &A = s_tv[ilo], &B = s_tv[ihi];
                Shaft sh = make_shaft(A, B);
                // premise of coplanar skipping per side: the patch qualifies (plane.w = its smallest altitude h > 0) and every
                // ray meets its plane steeply.  The ray directions are convex combinations of the three vertex-to-vertex
                // vectors D_i, so n.D_i of one sign bounds cos(theta) >= min|n.D_i| / max|D_i|.  The edge functions of a
                // coplanar triangle near a patch are computed from coordinates relative to the ray origin: rounding
                // ~ 8 eps (distance) (its size), against a true value >= (EDGE_MARGIN h)(its edge) cos(theta).  With sizes and
                // aspect ratios bounded by k_tri_planes that gives cos >= 0.02 on the origin side (distance ~ size) and
                // EDGE_MARGIN h cos >= 128 eps (distance) on the destination side.
                bool on_lo = false, on_hi = false;
                if (P.ring_on) pair_premise(A, B, sm.pl[ilo], sm.pl[ihi], on_lo, on_hi, m_req);
                // a sample pattern with points outside the triangle (no reference pattern has any): rays may leave the hull of the
                // two patches, so nothing is culled -- every pair takes the per-ray LBVH walk of phase 2b
                ncand = P.all_heavy ? -1 : shaft_candidates(P.nodes, P.root, sh, on_lo ? sm.pid[ilo] : 0, on_hi ? sm.pid[ihi] : 0, sm.id[ilo], sm.id[ihi],
                                                            my_cand, P.faces, P.nfaces, fmask);
                if (ncand >= 0) ncand |= (on_lo ? 0x10000 : 0) | (on_hi ? 0x20000 : 0);
                if (ncand < 0) { // the lists do not fit: flag the pair, phase 2b walks the LBVH per ray
                    s_list[q] = (unsigned short)(idx | PAIR_HEAVY);
                    atomicAdd(&s_nheavy, 1);
                }
            }
            __syncwarp();
            FF_CLK(1);
            // (ii) lane = sample: the warp resolves its 32 pairs one after the other
            uint64_t my_mask = 0;
            for (int j = 0; j < 32; j++) {
                const int nc = __shfl_sync(0xffffffffu, ncand, j);
                if (nc < 0) continue;
                const int idj = __shfl_sync(0xffffffffu, idx, j);
                const float mrq = __shfl_sync(0xffffffffu, m_req, j);
                const unsigned long long fmj = (unsigned long long)__shfl_sync(0xffffffffu, (unsigned)fmask, j) |
                                               ((unsigned long long)__shfl_sync(0xffffffffu, (unsigned)(fmask >> 32), j) << 32);
                const int rl = (idj >> 6) & 63, cl = idj & 63;
                const int ilo = (idj & PAIR_SWAP) ? TILE + cl : rl, ihi = (idj & PAIR_SWAP) ? rl : TILE + cl;
                const TriVerts Tlo = s_tv[ilo], Thi = s_tv[ihi];
                uint64_t mask = pair_mask_warp(P.tv, P.tribox, Tlo, Thi, sm.id[ilo], sm.id[ihi], warp_cand + (size_t)j * SHAFT_CAP, nc & 0xffff, fmj, ftab,
                                               (sm.pl[ilo].w > 0.f) ? sm.pid[ilo] - 1 : -1, sm.pl[ilo].w, (sm.pl[ihi].w > 0.f) ? sm.pid[ihi] - 1 : -1, sm.pl[ihi].w, sm.pid[ilo], sm.pid[ihi],
                                               (nc & 0x10000) ? P.nbr + (size_t)sm.id[ilo] * NBR_CAP : nullptr,
                                               (nc & 0x20000) ? P.nbr + (size_t)sm.id[ihi] * NBR_CAP : nullptr, P.n_inner, mrq,
                                               sm.uv, sm.perm, P.S, lane, sm.u.p2.wk[tid >> 5], sm.u.p2.wb[tid >> 5]);
                if (lane == j) my_mask = mask; // every lane holds the pair's mask: lane j keeps it and finishes its own pair below
#ifdef DAISY_FF_STATS
                if (lane == 0) {
                    const int nm = nc & 0xffff, pc = __popcll(mask);
                    const int cat = nm == 0 ? 0 : (pc == 0 ? 1 : (pc == P.S ? 2 : 3)); // simple / occluded / visible / partial
                    atomicAdd(&g_ffstats[cat], 1ull); atomicAdd(&g_ffstats[4 + cat], (unsigned long long)nm); atomicAdd(&g_ffstats[8 + cat], (unsigned long long)((nc >> 16) & 3));
                    if (nm == 0 && pc == P.S) atomicAdd(&g_ffstats[12], 1ull);
                    atomicAdd(&g_ffstats[13], (unsigned long long)__popcll(fmj));
                    if (nm == 0 && fmj == 0) atomicAdd(&g_ffstats[18], 1ull);
                }
                {
                    const int nm = nc & 0xffff;
                    const long long now_ = clock64();
                    if (lane == 0) atomicAdd(&g_ffstats[nm == 0 ? 26 : 27], (unsigned long long)(now_ - clk_));
                    clk_ = now_;
                }
#endif
            }
            if (ncand >= 0) finish_pair((idx >> 6) & 63, idx & 63, my_mask); // lane = pair again
            __syncwarp();
        }
        __syncthreads();
        FF_CLK(4);
        const int nheavy = s_nheavy;
        if (tid == 0 && s_nheavy) atomicAdd(P.pair_counter + 2, (unsigned long long)s_nheavy);
        // 2b: deferred pairs (flagged in the list), one per warp at a time with lane = sample: the rays of one pair walk the
        // LBVH coherently.  (lane = pair left most of the CTA idle behind one or two busy lanes: a tile defers few pairs.)
        while (nheavy) {
            int q0 = 0;
            if (lane == 0) q0 = atomicAdd(&s_hnext, 8);
            q0 = __shfl_sync(0xffffffffu, q0, 0);
            if (q0 >= nlist) break;
            const int e = (lane < 8 && q0 + lane < nlist) ? s_list[q0 + lane] : 0;
            unsigned hv = __ballot_sync(0xffffffffu, e & PAIR_HEAVY);
            while (hv) {
                const int j = __ffs(hv) - 1;
                hv &= hv - 1;
                const int idx = __shfl_sync(0xffffffffu, e, j);
                const int rl = (idx >> 6) & 63, cl = idx & 63;
                const int ilo = (idx & PAIR_SWAP) ? TILE + cl : rl, ihi = (idx & PAIR_SWAP) ? rl : TILE + cl;
                const TriVerts Tlo = s_tv[ilo], Thi = s_tv[ihi];
                bool on_lo = false, on_hi = false;
                float m_req = 0.f;
                if (P.ring_on) pair_premise(Tlo, Thi, sm.pl[ilo], sm.pl[ihi], on_lo, on_hi, m_req);
                unsigned mask_lo = 0, mask_hi = 0;
                for (int i0 = 0; i0 < P.S; i0 += 32) {
                    const int i = i0 + lane, ii = min(i, P.S - 1);
                    const float su = sm.uv[2 * ii], sv = sm.uv[2 * ii + 1];
                    // the pair's own planes are skipped by the samples far enough from the patch edges; the others walk everything
                    const bool inner = fminf(fminf(su, sv), 1.0f - su - sv) >= m_req;
                    const bool sees = (i < P.S) && ray_sees(P.nodes, P.tv, P.root, Tlo, Thi, sm.id[ilo], sm.id[ihi], su, sv,
                                                            (inner && on_lo) ? sm.pid[ilo] : 0, (inner && on_hi) ? sm.pid[ihi] : 0);
                    const int bit = sm.perm[ii];
                    mask_lo |= __reduce_or_sync(0xffffffffu, (sees && bit < 32) ? (1u << bit) : 0u);
                    mask_hi |= __reduce_or_sync(0xffffffffu, (sees && bit >= 32) ? (1u << (bit - 32)) : 0u);
                }
                if (lane == 0) finish_pair(rl, cl, (uint64_t)mask_lo | ((uint64_t)mask_hi << 32));
            }
        }
        __syncthreads();
        FF_CLK(5);

        // ---- phase 3: tile stores.  Row a of s_rc is row id[a] of F; row a of s_cr is row id[64 + a] of F.  With Morton
        // tiles the columns of one row are short runs of consecutive triangle ids (a few sectors per row), not one segment
        if (P.F) {
            _Pragma("unroll 1") for (int idx = tid; idx < TILE * TILE; idx += FF_THREADS) {
                const int a = idx >> 6, b = idx & 63;
                {
                    const int r = sm.id[a], c = sm.id[TILE + b];
                    const float v = diag ? ((a < b) ? s_rc[a][b] : ((a > b) ? s_cr[a][b] : (PARTIAL ? __int_as_float(UPD_KEEP) : 0.0f))) : s_rc[a][b];
                    if (r >= 0 && c >= 0 && !(PARTIAL && __float_as_int(v) == UPD_KEEP)) {
                        if (P.peer_mode) {
                            const int g = r / P.n_per_rank;
                            DZ_ASSERT(g >= 0 && g < 16 && P.Fpeer[g] != nullptr && c < P.N);
                            P.Fpeer[g][(size_t)(r - g * P.n_per_rank) * P.ldF + c] = v;
                        } else if (r >= P.row0 && r < P.row1) { DZ_ASSERT(c < P.N && (int64_t)c < P.ldF); P.F[(size_t)(r - P.row0) * P.ldF + c] = v; }
                    }
                }
                if (!diag) { // mirrored tile: row = column patch
                    const int r = sm.id[TILE + a], c = sm.id[b];
                    const float v = s_cr[a][b];
                    if (r >= 0 && c >= 0 && !(PARTIAL && __float_as_int(v) == UPD_KEEP)) {
                        if (P.peer_mode) {
                            const int g = r / P.n_per_rank;
                            P.Fpeer[g][(size_t)(r - g * P.n_per_rank) * P.ldF + c] = v;
                        } else if (r >= P.row0 && r < P.row1) P.F[(size_t)(r - P.row0) * P.ldF + c] = v;
                    }
                }
            }
        }
        __syncthreads();
        FF_CLK(6);
    }
}

bool dz_samples_outside(const daisy_ctx *ctx) {
    for (int i = 0; i < ctx->S; i++) {
        const float u = ctx->h_uv[2 * i], v = ctx->h_uv[2 * i + 1];
        if (!(u >= 0.f && v >= 0.f && u + v <= 1.0f + 1e-6f)) return true;
    }
    return false;
}

int dz_build_formfactors(daisy_ctx *ctx, int variant, uint64_t *d_masks, int mrow0, int mrow1, bool write_F, const DzUpdate *upd) {
    const int N = ctx->N;
    if (N == 0) return DAISY_OK;
    cudaStream_t st = ctx->stream;
    const bool timing = getenv("DAISY_TIMING") != nullptr;
    auto tprev = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {
        if (!timing) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "  dz_build_formfactors: %-28s %.3f s\n", what, std::chrono::duration<double>(now - tprev).count());
        tprev = now;
    };
    const int ntiles = (N + TILE - 1) / TILE;
    // row range of interest: the context's rows when writing F, else the mask rows
    int r0 = write_F ? ctx->row0 : mrow0, r1 = write_F ? ctx->row1 : mrow1;
    if (r1 <= r0 && !(write_F && ctx->peers_set)) return DAISY_OK;
    // jobs: upper-triangle tiles (R <= C) of the slot grid.  Local mode: every tile one of whose two patch groups holds a row
    // of the range of interest (off-diagonal blocks are then traced by both owners).  Peer mode: every tile is traced by
    // exactly one rank, chosen by a hash of (R, C) -- any rank can store any entry into its owner's matrix through the IPC
    // mappings, and tile cost varies by orders of magnitude with the geometry (wall-to-wall blocks vs blocks of one plane),
    // so spreading the ~ntiles^2/2 tiles pseudo-randomly is what balances the ranks (owner-based assignment left 8 GPUs at 4.5x).
    const bool peer = write_F && ctx->peers_set && ctx->nranks > 1;
    std::vector<char> has((size_t)ntiles, 0);
    for (int p = 0; p < ctx->nslots; p++) {
        const int t = ctx->h_order[p];
        if (t >= r0 && t < r1) has[(size_t)(p / TILE)] = 1;
    }
    auto mine = [&](int R, int C) -> bool {
        if (!peer) return has[(size_t)R] || has[(size_t)C];
        const uint32_t h = ((uint32_t)R * 0x9E3779B1u) ^ ((uint32_t)C * 0x85EBCA77u);
        return (int)((h >> 12) % (uint32_t)ctx->nranks) == ctx->rank;
    };
    size_t njobs = 0;
    for (int R = 0; R < ntiles; R++)
        for (int C = R; C < ntiles; C++)
            if (mine(R, C)) njobs++;
    int2 *h_jobs = (int2 *)malloc(sizeof(int2) * (njobs ? njobs : 1));
    if (!h_jobs) { daisy_set_error("out of host memory for the tile list"); return DAISY_E_NOMEM; }
    size_t k = 0;
    for (int R = 0; R < ntiles; R++)
        for (int C = R; C < ntiles; C++)
            if (mine(R, C)) h_jobs[k++] = make_int2(R, C);
    lap("tile list (host)");
    int2 *d_jobs = nullptr;
    int *d_counter = nullptr;
    unsigned long long *d_pairs = nullptr;
    DZ_CUDA(cudaMalloc(&d_jobs, sizeof(int2) * (njobs ? njobs : 1)));
    DZ_CUDA(cudaMalloc(&d_counter, sizeof(int)));
    DZ_CUDA(cudaMalloc(&d_pairs, 3 * sizeof(unsigned long long)));
    DZ_CUDA(cudaMemcpyAsync(d_jobs, h_jobs, sizeof(int2) * njobs, cudaMemcpyHostToDevice, st));
    DZ_CUDA(cudaMemsetAsync(d_counter, 0, sizeof(int), st));
    DZ_CUDA(cudaMemsetAsync(d_pairs, 0, 3 * sizeof(unsigned long long), st));
    FFParams P;
    P.geom = ctx->d_geom; P.tv = ctx->d_triverts; P.tribox = ctx->d_tribox; P.scratch = nullptr; P.nodes = ctx->d_nodes; P.root = ctx->root; P.N = N; P.S = ctx->S;
    P.order = ctx->d_order;
    P.plane = ctx->d_plane; P.pid = ctx->d_pid; P.nbr = ctx->d_nbr; P.n_inner = samples_device_order(ctx, P.uv, P.perm);
    P.faces = ctx->d_faces; P.face_cells = ctx->d_face_cells; P.face_lists = ctx->d_face_lists; P.nfaces = ctx->nfaces; P.face_tm = 4.0f * ctx->pad;
    P.face_ncells = ctx->face_cells; P.face_nlist = ctx->face_list_ints;

    { const char *e = getenv("DAISY_FF_RING"); P.ring_on = !(e && e[0] == '0'); }
    P.all_heavy = dz_samples_outside(ctx) ? 1 : 0;
    if (P.all_heavy) P.ring_on = 0;
    P.row0 = r0; P.row1 = r1;
    P.F = write_F ? ctx->d_F : nullptr; P.ldF = ctx->ldF;
    P.peer_mode = peer ? 1 : 0; P.n_per_rank = ctx->rows_per_rank;
    for (int g = 0; g < 16; g++) P.Fpeer[g] = (peer && g < ctx->nranks) ? ctx->peerF[g] : nullptr;
    P.masks = d_masks; P.mrow0 = mrow0; P.mrow1 = mrow1;
    P.upd = DzUpdate{};
    P.ntiles = ntiles; P.job_counter = d_counter; P.pair_counter = d_pairs; P.njobs = (int)njobs; P.jobs = d_jobs;
    cudaEvent_t e0, e1;
    DZ_CUDA(cudaEventCreate(&e0));
    DZ_CUDA(cudaEventCreate(&e1));
    // update run: classify the jobs on the device, keep the tiles the update can reach, each with its dirty clusters
    int2 *d_kept = nullptr;
    int *d_lists = nullptr;
    P.tile_dirty = nullptr;
    if (upd) {
        P.upd = *upd;
        int *d_count = nullptr;
        DZ_CUDA(cudaMalloc(&d_kept, sizeof(int2) * (njobs ? njobs : 1)));
        DZ_CUDA(cudaMalloc(&d_lists, sizeof(int) * (UPD_CAP + 1) * (njobs ? njobs : 1)));
        DZ_CUDA(cudaMalloc(&d_count, sizeof(int)));
        DZ_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int), st));
        DZ_CUDA(cudaEventRecord(e0, st));
        if (njobs)
            k_ff_classify<<<(int)std::min<size_t>(njobs, (size_t)ctx->num_sms * 16), 128, 0, st>>>(d_jobs, (int)njobs, ctx->d_order, ctx->d_triverts, upd->changed,
                                                                                                  upd->cbox, upd->nclusters, d_kept, d_lists, d_count);
        DZ_CUDA(cudaGetLastError());
        DZ_CUDA(cudaEventRecord(e1, st));
        int kept = 0;
        DZ_CUDA(cudaMemcpyAsync(&kept, d_count, sizeof(int), cudaMemcpyDeviceToHost, st));
        DZ_CUDA(cudaStreamSynchronize(st));
        float cms = 0.f;
        DZ_CUDA(cudaEventElapsedTime(&cms, e0, e1));
        cudaFree(d_count);
        ctx->upd_classify_ms = cms;
        njobs = (size_t)kept;
        P.njobs = kept; P.jobs = d_kept; P.tile_dirty = d_lists;
        lap("classification");
    }
    if (write_F) ctx->upd_tiles = (int64_t)njobs;
    int blocks_per_sm = 0;
    const size_t smem = sizeof(FFSmem);
    DZ_CUDA(cudaFuncSetAttribute(k_ff_tiles<DAISY_FF_DEVICE, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DZ_CUDA(cudaFuncSetAttribute(k_ff_tiles<DAISY_FF_HOST, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DZ_CUDA(cudaFuncSetAttribute(k_ff_tiles<DAISY_FF_DEVICE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DZ_CUDA(cudaFuncSetAttribute(k_ff_tiles<DAISY_FF_HOST, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    auto kernel = variant == DAISY_FF_DEVICE ? (upd ? k_ff_tiles<DAISY_FF_DEVICE, true> : k_ff_tiles<DAISY_FF_DEVICE, false>)
                                             : (upd ? k_ff_tiles<DAISY_FF_HOST, true> : k_ff_tiles<DAISY_FF_HOST, false>);
    DZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kernel, FF_THREADS, smem));
    if (blocks_per_sm < 1) blocks_per_sm = 1;
    int grid = ctx->num_sms * blocks_per_sm; // persistent CTAs, a multiple of the SM count
    if ((size_t)grid > njobs) grid = (int)njobs;
    int *d_scratch = nullptr;
    DZ_CUDA(cudaMalloc(&d_scratch, sizeof(int) * (size_t)(grid > 0 ? grid : 1) * FF_THREADS * SHAFT_CAP));
    P.scratch = d_scratch;
    lap("allocations, uploads");
    DZ_CUDA(cudaEventRecord(e0, st));
    if (grid > 0) kernel<<<grid, FF_THREADS, smem, st>>>(P);
    DZ_CUDA(cudaGetLastError());
    DZ_CUDA(cudaEventRecord(e1, st));
    unsigned long long pairs[3] = { 0, 0, 0 };
    DZ_CUDA(cudaMemcpyAsync(pairs, d_pairs, sizeof(pairs), cudaMemcpyDeviceToHost, st));
    DZ_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    DZ_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    lap("kernel");
#ifdef DAISY_FF_STATS
    {
        unsigned long long h[48];
        cudaMemcpyFromSymbolAsync(h, g_ffstats, sizeof(h), 0, cudaMemcpyDeviceToHost, st);
        cudaStreamSynchronize(st);
        const char *nm[4] = { "simple(n_main=0)", "occluded", "visible", "partial" };
        for (int c = 0; c < 4; c++)
            fprintf(stderr, "ffstats %-18s pairs %12llu  mean n_main %7.1f  mean n_ring %6.1f\n", nm[c], h[c], h[c] ? (double)h[4 + c] / h[c] : 0.0, h[c] ? (double)h[8 + c] / h[c] : 0.0);
        fprintf(stderr, "ffstats simple&fully-visible %llu ; slab iterations pass0 %llu pass1 %llu\n", h[12], h[16], h[17]);
        fprintf(stderr, "ffstats faces: %d grids, face entries over all pairs %llu, pairs with neither list nor face %llu, cell lookups %llu, explicit tests in cells %llu, flat-ray tests in cells %llu, rays searching a face %llu\n",
                ctx->nfaces, h[13], h[18], h[15], h[14], h[23], h[19]);
        fprintf(stderr, "ffstats steep lookups: empty %llu, blocked by a covered cell %llu, explicit: own plane %llu, mixed cell %llu, covered but near an end point %llu; flat stretches: own plane %llu, other %llu\n",
                h[38], h[37], h[32], h[33], h[34], h[35], h[36]);
        fprintf(stderr, "ffstats flush: rounds executed %llu, rounds if balanced over lanes %llu, tests queued %llu (%.1f lanes per executed round)\n",
                h[22], h[20], h[21], h[22] ? (double)h[21] / h[22] : 0.0);
        {
            const char *ph[7] = { "stage+phase1", "shaft walk", "samples(simple)", "samples(listed)", "tile barrier wait", "per-ray fallback", "tile store" };
            unsigned long long tot = 0;
            for (int i = 0; i < 7; i++) tot += h[24 + i];
            for (int i = 0; i < 7; i++) fprintf(stderr, "ffstats warp-cycles %-18s %6.2f %%\n", ph[i], tot ? 100.0 * (double)h[24 + i] / (double)tot : 0.0);
        }
        unsigned long long z[48] = { 0 };
        cudaMemcpyToSymbolAsync(g_ffstats, z, sizeof(z), 0, cudaMemcpyHostToDevice, st);
        cudaStreamSynchronize(st);
    }
#endif
    if (write_F) { ctx->ff_ms = ms; ctx->pairs_traced = (int64_t)pairs[0]; ctx->pairs_owned = (int64_t)pairs[1]; ctx->pairs_heavy = (int64_t)pairs[2]; }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d_jobs); cudaFree(d_counter); cudaFree(d_pairs); cudaFree(d_scratch); cudaFree(d_kept); cudaFree(d_lists);
    free(h_jobs);
    lap("clean-up");
    return DAISY_OK;
}
