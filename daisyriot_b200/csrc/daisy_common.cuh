// daisy_common.cuh -- shared device helpers of the sm_100a form-factor / gather library.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>
#include <nvtx3/nvToolsExt.h>
#include "../../include/daisy_b200.h"

// NVTX range over a scope (Nsight Systems / Compute timelines; a no-op function pointer when no tool is attached)
struct DzRange {
    explicit DzRange(const char *name) { nvtxRangePushA(name); }
    ~DzRange() { nvtxRangePop(); }
};

// ---------------------------------------------------------------------------------------------------------
// error plumbing (C-ABI never throws; the C++ shim above it reproduces the reference's print-and-continue)
void daisy_set_error(const char *fmt, ...);
#define DZ_CUDA(call)                                                                                    \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            daisy_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));       \
            return DAISY_E_CUDA;                                                                         \
        }                                                                                                \
    } while (0)
#define DZ_REQUIRE(cond, code, msg)                         \
    do {                                                    \
        if (!(cond)) { daisy_set_error("%s", msg); return code; } \
    } while (0)

// ---------------------------------------------------------------------------------------------------------
// Device-side bounds / invariant checks, compiled in with -DDAISY_BOUNDS_CHECK (`make TAG=check EXTRA=-DDAISY_BOUNDS_CHECK`):
// a violated check prints its location and traps, which the host sees as a launch failure.  This is the memory-safety
// net of this repo: compute-sanitizer is closed on the GPU pool the kernels are developed on, so the checked build is run
// over the small parity cases instead (tools/checked_build.sh), next to the bit-exact comparison with the CPU oracle.
#ifdef DAISY_BOUNDS_CHECK
#define DZ_ASSERT(cond)                                                                                  \
    do {                                                                                                 \
        if (!(cond)) { printf("DZ_ASSERT failed: %s  (%s:%d, block %d thread %d)\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, (int)threadIdx.x); __trap(); } \
    } while (0)
#else
#define DZ_ASSERT(cond) do { } while (0)
#endif

// ---------------------------------------------------------------------------------------------------------
// Exactly-rounded FP32 ops that ptxas may never contract into FMAs.  The reference's host build (MSVC x64,
// /fp:precise) evaluates every glm expression as separate IEEE mul/add; parity with it (and with the CPU oracle)
// is bit-exact only if the device does the same, so every result-defining expression goes through these.
__device__ __forceinline__ float fm(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float fa(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fs(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fd(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float fsq(float a) { return __fsqrt_rn(a); }

struct f3 { float x, y, z; };
__device__ __forceinline__ f3 mk3(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
__device__ __forceinline__ f3 e_sub(f3 a, f3 b) { return mk3(fs(a.x, b.x), fs(a.y, b.y), fs(a.z, b.z)); }
__device__ __forceinline__ f3 e_add(f3 a, f3 b) { return mk3(fa(a.x, b.x), fa(a.y, b.y), fa(a.z, b.z)); }
__device__ __forceinline__ f3 e_scale(f3 a, float s) { return mk3(fm(a.x, s), fm(a.y, s), fm(a.z, s)); }
// glm compute_dot<tvec3>: tmp = x*y; tmp.x + tmp.y + tmp.z          (glm/detail/func_geometric.inl:54-61)
__device__ __forceinline__ float e_dot(f3 a, f3 b) { return fa(fa(fm(a.x, b.x), fm(a.y, b.y)), fm(a.z, b.z)); }
// glm compute_cross                                                  (glm/detail/func_geometric.inl:74-85)
__device__ __forceinline__ f3 e_cross(f3 x, f3 y) {
    return mk3(fs(fm(x.y, y.z), fm(y.y, x.z)), fs(fm(x.z, y.x), fm(y.z, x.x)), fs(fm(x.x, y.y), fm(y.x, x.y)));
}
// glm normalize = v * (1 / sqrt(dot(v,v)))                           (glm/detail/func_geometric.inl:88-95)
__device__ __forceinline__ f3 e_normalize(f3 a) { return e_scale(a, fd(1.0f, fsq(e_dot(a, a)))); }
// calculateSurface: 0.5 * length(cross(b-a, c-a)), 0.5 a double literal (VS/parallellism.cu:209-214); the double
// product rounded to float equals the float product with 0.5f (scaling by a power of two, RN both ways)
__device__ __forceinline__ float e_surface(f3 a, f3 b, f3 c) {
    f3 cr = e_cross(e_sub(b, a), e_sub(c, a));
    return fm(0.5f, fsq(e_dot(cr, cr)));
}

// ---------------------------------------------------------------------------------------------------------
// Watertight ray/triangle test (Woop, Benthin, Wald, JCGT 2013), FP32, no culling, t = T/det by IEEE division.
// Stands in for OptiX Prime's closed-source intersector; the CPU oracle states the same arithmetic.
struct WRay {
    f3 o;           // origin
    int kx, ky, kz; // axis permutation, kz = dominant direction axis
    int perm;       // the same permutation as flags: bit 0 = (kz == 0), bit 1 = (kz == 1), bit 2 = kx and ky swapped (d[kz] < 0)
    float Sx, Sy, Sz;
};
__device__ __forceinline__ float comp(const f3 &v, int k) { return k == 0 ? v.x : (k == 1 ? v.y : v.z); }

__device__ __forceinline__ WRay wray_setup(f3 o, f3 d) {
    WRay w;
    w.o = o;
    float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    int kz = (ax >= ay && ax >= az) ? 0 : ((ay >= az) ? 1 : 2);
    int kx = kz == 2 ? 0 : kz + 1, ky = kx == 2 ? 0 : kx + 1;
    float dz = comp(d, kz);
    w.perm = (kz == 0 ? 1 : 0) | (kz == 1 ? 2 : 0) | (dz < 0.0f ? 4 : 0);
    if (dz < 0.0f) { int t = kx; kx = ky; ky = t; }
    w.kx = kx; w.ky = ky; w.kz = kz;
    w.Sx = fd(comp(d, kx), dz);
    w.Sy = fd(comp(d, ky), dz);
    w.Sz = fd(1.0f, dz);
    return w;
}

// core of the test with the axis permutation resolved at compile time (no per-component selects)
template <int KX, int KY, int KZ>
__device__ __forceinline__ bool wray_tri_k(const WRay &w, f3 va, f3 vb, f3 vc, float &t, float &u, float &v) {
    f3 A = e_sub(va, w.o), B = e_sub(vb, w.o), C = e_sub(vc, w.o);
    const float Akx = KX == 0 ? A.x : (KX == 1 ? A.y : A.z), Aky = KY == 0 ? A.x : (KY == 1 ? A.y : A.z), Akz = KZ == 0 ? A.x : (KZ == 1 ? A.y : A.z);
    const float Bkx = KX == 0 ? B.x : (KX == 1 ? B.y : B.z), Bky = KY == 0 ? B.x : (KY == 1 ? B.y : B.z), Bkz = KZ == 0 ? B.x : (KZ == 1 ? B.y : B.z);
    const float Ckx = KX == 0 ? C.x : (KX == 1 ? C.y : C.z), Cky = KY == 0 ? C.x : (KY == 1 ? C.y : C.z), Ckz = KZ == 0 ? C.x : (KZ == 1 ? C.y : C.z);
    float Ax = fs(Akx, fm(w.Sx, Akz)), Ay = fs(Aky, fm(w.Sy, Akz));
    float Bx = fs(Bkx, fm(w.Sx, Bkz)), By = fs(Bky, fm(w.Sy, Bkz));
    float Cx = fs(Ckx, fm(w.Sx, Ckz)), Cy = fs(Cky, fm(w.Sy, Ckz));
    float U = fs(fm(Cx, By), fm(Cy, Bx));
    float V = fs(fm(Ax, Cy), fm(Ay, Cx));
    float W = fs(fm(Bx, Ay), fm(By, Ax));
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        U = __double2float_rn(__dsub_rn(__dmul_rn((double)Cx, (double)By), __dmul_rn((double)Cy, (double)Bx)));
        V = __double2float_rn(__dsub_rn(__dmul_rn((double)Ax, (double)Cy), __dmul_rn((double)Ay, (double)Cx)));
        W = __double2float_rn(__dsub_rn(__dmul_rn((double)Bx, (double)Ay), __dmul_rn((double)By, (double)Ax)));
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
    float det = fa(fa(U, V), W);
    if (det == 0.0f) return false;
    float Az = fm(w.Sz, Akz), Bz = fm(w.Sz, Bkz), Cz = fm(w.Sz, Ckz);
    float T = fa(fa(fm(U, Az), fm(V, Bz)), fm(W, Cz));
    float tt = fd(T, det);
    if (!(tt > 0.0f) || isinf(tt)) return false;
    t = tt; u = fd(V, det); v = fd(W, det);
    return true;
}

// returns true on a hit with finite t > 0; u,v = barycentric weights of vertices 1 and 2 (HIT_T_TRIID_U_V).
// (kx,ky,kz) is one of six permutations.  wray_tri dispatches to a permutation-specialised body (no per-component
// selects; rays of one patch pair are nearly parallel, so the switch is almost always uniform across a warp) -- six
// copies of the test, used where code size does not matter.  wray_tri_sel resolves the permutation with selects: one
// copy, the form the form-factor kernel uses to stay inside the instruction cache.  Both evaluate the identical
// sequence of IEEE operations on the identical operands, so their results are bit-identical.
__device__ __forceinline__ bool wray_tri(const WRay &w, f3 va, f3 vb, f3 vc, float &t, float &u, float &v) {
    switch (w.kz * 2 + (w.kx == (w.kz == 2 ? 0 : w.kz + 1) ? 0 : 1)) {
    case 0: return wray_tri_k<1, 2, 0>(w, va, vb, vc, t, u, v);
    case 1: return wray_tri_k<2, 1, 0>(w, va, vb, vc, t, u, v);
    case 2: return wray_tri_k<2, 0, 1>(w, va, vb, vc, t, u, v);
    case 3: return wray_tri_k<0, 2, 1>(w, va, vb, vc, t, u, v);
    case 4: return wray_tri_k<0, 1, 2>(w, va, vb, vc, t, u, v);
    default: return wray_tri_k<1, 0, 2>(w, va, vb, vc, t, u, v);
    }
}

__device__ __forceinline__ bool wray_tri_sel(const WRay &w, f3 va, f3 vb, f3 vc, float &t, float &u, float &v) {
    f3 A = e_sub(va, w.o), B = e_sub(vb, w.o), C = e_sub(vc, w.o);
    // (kx, ky, kz) = (kz+1, kz+2, kz) mod 3, kx and ky swapped when the dominant component is negative: a rotation of the
    // components followed by a conditional swap, 8 selects per vertex on three per-ray flags
    const bool r0 = w.perm & 1, r1 = w.perm & 2, sw = w.perm & 4;
    const float A0 = r0 ? A.y : (r1 ? A.z : A.x), A1 = r0 ? A.z : (r1 ? A.x : A.y), Akz = r0 ? A.x : (r1 ? A.y : A.z);
    const float B0 = r0 ? B.y : (r1 ? B.z : B.x), B1 = r0 ? B.z : (r1 ? B.x : B.y), Bkz = r0 ? B.x : (r1 ? B.y : B.z);
    const float C0 = r0 ? C.y : (r1 ? C.z : C.x), C1 = r0 ? C.z : (r1 ? C.x : C.y), Ckz = r0 ? C.x : (r1 ? C.y : C.z);
    const float Akx = sw ? A1 : A0, Aky = sw ? A0 : A1;
    const float Bkx = sw ? B1 : B0, Bky = sw ? B0 : B1;
    const float Ckx = sw ? C1 : C0, Cky = sw ? C0 : C1;
    float Ax = fs(Akx, fm(w.Sx, Akz)), Ay = fs(Aky, fm(w.Sy, Akz));
    float Bx = fs(Bkx, fm(w.Sx, Bkz)), By = fs(Bky, fm(w.Sy, Bkz));
    float Cx = fs(Ckx, fm(w.Sx, Ckz)), Cy = fs(Cky, fm(w.Sy, Ckz));
    float U = fs(fm(Cx, By), fm(Cy, Bx));
    float V = fs(fm(Ax, Cy), fm(Ay, Cx));
    float W = fs(fm(Bx, Ay), fm(By, Ax));
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        U = __double2float_rn(__dsub_rn(__dmul_rn((double)Cx, (double)By), __dmul_rn((double)Cy, (double)Bx)));
        V = __double2float_rn(__dsub_rn(__dmul_rn((double)Ax, (double)Cy), __dmul_rn((double)Ay, (double)Cx)));
        W = __double2float_rn(__dsub_rn(__dmul_rn((double)Bx, (double)Ay), __dmul_rn((double)By, (double)Ax)));
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
    float det = fa(fa(U, V), W);
    if (det == 0.0f) return false;
    float Az = fm(w.Sz, Akz), Bz = fm(w.Sz, Bkz), Cz = fm(w.Sz, Ckz);
    float T = fa(fa(fm(U, Az), fm(V, Bz)), fm(W, Cz));
    float tt = fd(T, det);
    if (!(tt > 0.0f) || isinf(tt)) return false;
    t = tt; u = fd(V, det); v = fd(W, det);
    return true;
}

// The same test for callers that only want the distance (the visibility rays of the form-factor kernel): identical
// operations up to T and det; when their signs already say t <= 0 the IEEE division is skipped (T/det would be negative or a
// signed zero, both rejected), otherwise t is the very same quotient.
__device__ __forceinline__ bool wray_tri_t(const WRay &w, f3 va, f3 vb, f3 vc, float &t) {
    f3 A = e_sub(va, w.o), B = e_sub(vb, w.o), C = e_sub(vc, w.o);
    const bool r0 = w.perm & 1, r1 = w.perm & 2, sw = w.perm & 4;
    const float A0 = r0 ? A.y : (r1 ? A.z : A.x), A1 = r0 ? A.z : (r1 ? A.x : A.y), Akz = r0 ? A.x : (r1 ? A.y : A.z);
    const float B0 = r0 ? B.y : (r1 ? B.z : B.x), B1 = r0 ? B.z : (r1 ? B.x : B.y), Bkz = r0 ? B.x : (r1 ? B.y : B.z);
    const float C0 = r0 ? C.y : (r1 ? C.z : C.x), C1 = r0 ? C.z : (r1 ? C.x : C.y), Ckz = r0 ? C.x : (r1 ? C.y : C.z);
    const float Akx = sw ? A1 : A0, Aky = sw ? A0 : A1;
    const float Bkx = sw ? B1 : B0, Bky = sw ? B0 : B1;
    const float Ckx = sw ? C1 : C0, Cky = sw ? C0 : C1;
    float Ax = fs(Akx, fm(w.Sx, Akz)), Ay = fs(Aky, fm(w.Sy, Akz));
    float Bx = fs(Bkx, fm(w.Sx, Bkz)), By = fs(Bky, fm(w.Sy, Bkz));
    float Cx = fs(Ckx, fm(w.Sx, Ckz)), Cy = fs(Cky, fm(w.Sy, Ckz));
    float U = fs(fm(Cx, By), fm(Cy, Bx));
    float V = fs(fm(Ax, Cy), fm(Ay, Cx));
    float W = fs(fm(Bx, Ay), fm(By, Ax));
    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        U = __double2float_rn(__dsub_rn(__dmul_rn((double)Cx, (double)By), __dmul_rn((double)Cy, (double)Bx)));
        V = __double2float_rn(__dsub_rn(__dmul_rn((double)Ax, (double)Cy), __dmul_rn((double)Ay, (double)Cx)));
        W = __double2float_rn(__dsub_rn(__dmul_rn((double)Bx, (double)Ay), __dmul_rn((double)By, (double)Ax)));
    }
    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
    float det = fa(fa(U, V), W);
    if (det == 0.0f) return false;
    float Az = fm(w.Sz, Akz), Bz = fm(w.Sz, Bkz), Cz = fm(w.Sz, Ckz);
    float T = fa(fa(fm(U, Az), fm(V, Bz)), fm(W, Cz));
    if (T == 0.0f || ((T < 0.0f) != (det < 0.0f))) return false;
    float tt = fd(T, det);
    if (!(tt > 0.0f) || isinf(tt)) return false;
    t = tt;
    return true;
}

// ---------------------------------------------------------------------------------------------------------
// BVH node (64 B): both child boxes live in the parent, so one node fetch decides both descents.
// child < 0 => leaf holding triangle ~child.
struct __align__(16) BvhNode {
    float4 a; // L.lo.x L.lo.y L.lo.z L.hi.x
    float4 b; // L.hi.y L.hi.z R.lo.x R.lo.y
    float4 c; // R.lo.z R.hi.x R.hi.y R.hi.z
    int4 d;   // left, right, plane id shared by every triangle below the left child (0 = mixed / none, -1 = mixed, gridded faces only), same for the right child
};

// conservative slab test against [0, tmax]; boxes are padded at build time, fminf/fmaxf drop the NaN of 0*inf
__device__ __forceinline__ bool ray_box(f3 o, f3 inv, float lox, float loy, float loz, float hix, float hiy, float hiz,
                                        float tmax, float &tnear) {
    float t0x = (lox - o.x) * inv.x, t1x = (hix - o.x) * inv.x;
    float t0y = (loy - o.y) * inv.y, t1y = (hiy - o.y) * inv.y;
    float t0z = (loz - o.z) * inv.z, t1z = (hiz - o.z) * inv.z;
    float tn = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fmaxf(fminf(t0z, t1z), 0.0f));
    float tf = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fminf(fmaxf(t0z, t1z), tmax));
    tnear = tn;
    return tn <= tf * 1.00001f + 1e-30f;
}

// same test with the origin pre-multiplied: t = box*inv - o*inv is one FMA per plane.  inf*0 and inf-inf give NaN, which
// fminf/fmaxf drop, i.e. the plane is ignored: the test can only become more permissive, never cull a real hit.
__device__ __forceinline__ bool ray_box_fma(f3 oi, f3 inv, float lox, float loy, float loz, float hix, float hiy, float hiz, float tmax) {
    float t0x = fmaf(lox, inv.x, -oi.x), t1x = fmaf(hix, inv.x, -oi.x);
    float t0y = fmaf(loy, inv.y, -oi.y), t1y = fmaf(hiy, inv.y, -oi.y);
    float t0z = fmaf(loz, inv.z, -oi.z), t1z = fmaf(hiz, inv.z, -oi.z);
    float tn = fmaxf(fmaxf(fminf(t0x, t1x), fminf(t0y, t1y)), fmaxf(fminf(t0z, t1z), 0.0f));
    float tf = fminf(fminf(fmaxf(t0x, t1x), fmaxf(t0y, t1y)), fminf(fmaxf(t0z, t1z), tmax));
    return tn <= tf * 1.00001f + 1e-30f;
}

// the same for rays whose direction signs are known: (nx, ny, nz) = the box planes the ray enters through, (fx, fy, fz) = the
// ones it leaves through.  For finite operands min(t0, t1) IS the entry-plane value, so the result equals ray_box_fma's; a
// NaN is dropped by the 3-input min / max here as there, which can only make the test more permissive.
__device__ __forceinline__ bool ray_box_sorted(f3 oi, f3 inv, float nx, float ny, float nz, float fx, float fy, float fz, float tmax) {
    const float tn = fmaxf(fmaxf(fmaf(nx, inv.x, -oi.x), fmaf(ny, inv.y, -oi.y)), fmaxf(fmaf(nz, inv.z, -oi.z), 0.0f));
    const float tf = fminf(fminf(fmaf(fx, inv.x, -oi.x), fmaf(fy, inv.y, -oi.y)), fminf(fmaf(fz, inv.z, -oi.z), tmax));
    return tn <= tf * 1.00001f + 1e-30f;
}

// per-triangle vertex record (48 B): float4 a, b, c (w unused)
struct __align__(16) TriVerts { float4 a, b, c; };
// per-patch record for the 4x4 rule (80 B): 4 sub-centroids with sub-areas in w, then normal with area in w
struct __align__(16) PatchGeom { float4 s[4]; float4 n; };

// planar face grid (faces.cu): plane n.X = d, cell coordinates a = dot(X, ex.xyz) + ex.w, b = dot(X, ey.xyz) + ey.w
#define DAISY_MAX_FACES 64
struct __align__(16) DzFace {
    float4 pl; // unit normal, d
    float4 ex; // in-plane axis / cell size, offset
    float4 ey;
    int4 g;    // nx, ny, index of the face's first cell in the cell table, number of triangles
    float4 blo, bhi; // padded bounding box of the face's triangles
};

__device__ __forceinline__ f3 xyz(float4 v) { return mk3(v.x, v.y, v.z); }

// streaming load of 4 floats that are read once: no L1 allocation (F in the gather passes, the tile scan, the CSC count)
__device__ __forceinline__ float4 ldg_stream(const float *p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}

// ---------------------------------------------------------------------------------------------------------
struct daisy_ctx {
    int device = 0;
    cudaStream_t stream = 0;
    int N = 0, nv = 0, nn = 0;
    int rank = 0, nranks = 1, rows_per_rank = 0, row0 = 0, row1 = 0;
    int S = 0;
    float h_uv[2 * DAISY_MAX_SAMPLES];
    // device mesh
    float *d_vertices = nullptr, *d_normals = nullptr;
    int *d_tri = nullptr;
    int *d_vadj_off = nullptr, *d_vadj = nullptr; // MeshS::trianglesPerVertex as CSR: triangles using vertex v, ascending ids
    TriVerts *d_triverts = nullptr;
    float4 *d_tribox = nullptr; // padded per-triangle boxes (2 float4 each), same boxes as the LBVH leaves
    PatchGeom *d_geom = nullptr;
    int *d_order = nullptr;     // tile composition of the form-factor kernel: slot p of the tile grid holds triangle d_order[p]
                                // (Morton order of the LBVH build => 64 consecutive slots are spatially compact); -1 = empty slot
    int *h_order = nullptr;     // host copy (job lists of row-restricted runs)
    int nslots = 0;             // slots = ceil(N / 64) * 64
    int *d_pid = nullptr;       // per triangle: plane id (>= 1; api.cu assign_plane_ids), 0 if it shares its plane with no other triangle
    int *d_nbr = nullptr;       // per triangle: its neighbours in that plane, 32 ints ([0] = count), formfactor.cu k_tri_planes
    float4 *d_plane = nullptr;  // per triangle: unit geometric normal, w = smallest altitude if coplanar skipping is safe for it, else -1
    float ext = 0.f;            // largest scene extent
    // planar face grids (faces.cu): face f = plane id f + 1
    DzFace *d_faces = nullptr;
    int *d_face_cells = nullptr; // per cell: -1 empty, else (offset into d_face_lists << 1) | covered
    int *d_face_lists = nullptr; // per non-empty cell: count, triangle ids
    int nfaces = 0;
    int64_t face_cells = 0, face_list_ints = 0;
    // LBVH
    BvhNode *d_nodes = nullptr;
    int root = 0;
    float scene_lo[3], scene_hi[3], pad = 0.f;
    double lbvh_ms = 0.0;
    // form factors
    float *d_F = nullptr; // (row1-row0) x ldF
    int64_t ldF = 0;
    bool have_F = false;
    uint64_t F_version = 0;         // bumped by every write of F through this library (a solver rescans its tile map when it changes)
    float *peerF[16] = { nullptr }; // every rank's F (own pointer or CUDA-IPC mapping), set by daisy_formfactors_set_peers
    bool peers_set = false;
    bool peers_ipc = false;         // the peer pointers are CUDA-IPC mappings this context has to close (one process per GPU)
    int64_t pairs_traced = 0, pairs_owned = 0, pairs_heavy = 0;
    double ff_ms = 0.0;
    int num_sms = 148;
    // grow-only device buffers of the per-frame entry points (closest-hit queries, traceScreen): a frame loop does not pay a
    // cudaMalloc / cudaFree pair per buffer per call (dz_scratch, api.cu)
    void *scratch[6] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
    size_t scratch_bytes[6] = { 0, 0, 0, 0, 0, 0 };
    // host copies of the mesh: the current geometry (daisy_ctx_create / _update_geometry / _replace_mesh) and the triangle list
    std::vector<float> h_vertices, h_normals;
    std::vector<int> h_tri;
    uint64_t mesh_version = 0; // bumped by daisy_ctx_replace_mesh: solvers created before it are stale (other N, other materials)
    // what F holds (daisy_formfactors_build / _update): the variant, sample pattern and geometry it was computed for, and the
    // box padding of that geometry.  Cleared by daisy_formfactors_write_rows.  Per CURRENT triangle, so that it follows the
    // triangles through daisy_ctx_replace_mesh; triangles removed since the record leave their recorded boxes behind.
    struct {
        bool valid = false;
        int variant = 0, S = 0;
        float uv[2 * DAISY_MAX_SAMPLES];
        std::vector<float> tri;         // 18 floats per triangle: its 3 vertex positions, then its 3 normals, as recorded
        std::vector<unsigned char> has; // per triangle: 1 = recorded, 0 = added since the record
        std::vector<float4> ghost;      // 2 float4 per triangle removed since the record: its recorded padded box
        float pad = 0.f;
    } rec;
    // last daisy_formfactors_update
    int64_t upd_tris_changed = 0, upd_tiles = 0, upd_pairs = 0;
    double upd_classify_ms = 0.0;
    // last daisy_formfactors_write_csc: uploads of the CSC arrays (1: kept resident while validated and scattered, 2: chunks
    // uploaded for the validation, rows only, and again for the scatter)
    int csc_uploads = 0;
};

// The part of F an update has to recompute (formfactor.cu, daisy_formfactors_update): per-triangle changed flags and the
// dirty boxes -- the padded boxes of the moved triangles in the recorded and in the current geometry, as leaves grouped into
// clusters of consecutive Morton order.  Device pointers.
struct DzUpdate {
    const unsigned char *changed; // N flags: a position or a normal of the triangle differs from the record
    const float4 *leaf;           // 2 float4 per dirty box
    const float4 *cbox;           // 2 float4 per cluster: union of its leaves
    const int2 *crange;           // leaves [x, y) of each cluster
    int nclusters;
};
cudaError_t dz_scratch(daisy_ctx *ctx, int slot, size_t bytes, void **out); // api.cu

int dz_build_lbvh(daisy_ctx *ctx);                                   // bvh.cu
int dz_launch_closest(daisy_ctx *ctx, int n, const float *d_rays, daisy_hit *d_hits); // bvh.cu
int dz_precompute_geom(daisy_ctx *ctx);                              // formfactor.cu
int dz_build_faces(daisy_ctx *c, const float *vertices, const int32_t *tri_idx, int ntri, std::vector<int> &pid); // faces.cu
void dz_free_faces(daisy_ctx *c);                                    // faces.cu
int dz_unoccluded_rows(daisy_ctx *ctx, int variant, int row0, int nrows, daisy_tripl *d_out); // formfactor.cu
struct daisy_solver;
// same-process peers (daisy_group): device pointers handed over directly, peer access enabled by the caller
int dz_ctx_set_peer_pointers(daisy_ctx *ctx, float *const *F, int nranks);                                           // api.cu
// daisy_ctx_replace_mesh over ctx[0..n): one context, or every device of a group (rank i of n, F remapped through peer access)  // api.cu
int dz_replace_mesh(daisy_ctx *const *ctx, int n, const float *vertices, int nv, const float *normals, int nn, const int32_t *tri_idx, int ntri,
                    const int32_t *previous, const char *what);
int dz_solver_get_buffers(daisy_solver *s, float **res0, float **res1, unsigned long long **flags);                  // gather.cu
int dz_solver_set_peer_pointers(daisy_solver *s, float *const *res0, float *const *res1, unsigned long long *const *flags, int nranks); // gather.cu
// converge with the stop rule on the device over n solvers issued from one thread (one GPU, or a group's devices)   // gather.cu
int dz_converge_device(daisy_solver *const *ss, int n, double threshold, int per_band, int max_passes);
// the restart pass without reading its band sums back (a group launches it on every device before any waits)   // gather.cu
int dz_solver_restart_launch(daisy_solver *s, const float *B0_local);
// upd != null: only the pairs the update can reach are traced and stored (ctx->upd_tiles, upd_classify_ms report it)
int dz_build_formfactors(daisy_ctx *ctx, int variant, uint64_t *d_masks, int mrow0, int mrow1, bool write_F,
                         const DzUpdate *upd = nullptr);                                                    // formfactor.cu
bool dz_samples_outside(const daisy_ctx *ctx);                                                              // formfactor.cu
int dz_ensure_F(daisy_ctx *ctx); // allocate F (zero-filled) if it does not exist yet                          // api.cu
// the matrix cache on the device (csc.cu): ctx[0..n) hold rows [row0, row1) each, in ascending order, together all N rows
bool dz_csc_host(); // DAISY_CSC_HOST=1: hand F back through the host conversion of dense row read-backs instead
int dz_csc_export(daisy_ctx *const *ctx, int n, int64_t *nnz, float *values, int32_t *inner_idx, int32_t *outer_ptr, const char *what);
int dz_csc_import(daisy_ctx *const *ctx, int n, int64_t nnz, const float *values, const int32_t *inner_idx, const int32_t *outer_ptr, const char *what);
