// bvh.cu -- Morton-code LBVH build (Karras 2012) and the closest-hit query kernel.
//
// Replaces what OptiX Prime did behind OptixPrimeFunctionality's constructor and optixQuery
// (reference visual studio/OptixPrimeFunctionality.cpp:36-47 and :66-81): `model->update()` becomes
// morton -> bitonic sort -> hierarchy -> bottom-up refit -> node packing, all on the device;
// `query->execute()` becomes one thread per ray walking that hierarchy.
#include "daisy_common.cuh"
#include "closest.cuh"
#include <math.h>
#include <stdlib.h>
#include <vector>

// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t expand_bits10(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

__global__ void k_triverts_morton(const float *__restrict__ vertices, const int *__restrict__ tri, int N, int npad,
                                  float3 slo, float3 sinv, TriVerts *__restrict__ tv, uint64_t *__restrict__ keys) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npad) return;
    if (i >= N) { keys[i] = ~0ull; return; }
    const int *t = tri + 6 * (size_t)i;
    float3 a = make_float3(vertices[3 * (size_t)t[0]], vertices[3 * (size_t)t[0] + 1], vertices[3 * (size_t)t[0] + 2]);
    float3 b = make_float3(vertices[3 * (size_t)t[1]], vertices[3 * (size_t)t[1] + 1], vertices[3 * (size_t)t[1] + 2]);
    float3 c = make_float3(vertices[3 * (size_t)t[2]], vertices[3 * (size_t)t[2] + 1], vertices[3 * (size_t)t[2] + 2]);
    TriVerts r;
    r.a = make_float4(a.x, a.y, a.z, 0.f); r.b = make_float4(b.x, b.y, b.z, 0.f); r.c = make_float4(c.x, c.y, c.z, 0.f);
    tv[i] = r;
    float cx = 0.5f * (fminf(a.x, fminf(b.x, c.x)) + fmaxf(a.x, fmaxf(b.x, c.x)));
    float cy = 0.5f * (fminf(a.y, fminf(b.y, c.y)) + fmaxf(a.y, fmaxf(b.y, c.y)));
    float cz = 0.5f * (fminf(a.z, fminf(b.z, c.z)) + fmaxf(a.z, fmaxf(b.z, c.z)));
    uint32_t qx = (uint32_t)fminf(fmaxf((cx - slo.x) * sinv.x * 1024.0f, 0.0f), 1023.0f);
    uint32_t qy = (uint32_t)fminf(fmaxf((cy - slo.y) * sinv.y * 1024.0f, 0.0f), 1023.0f);
    uint32_t qz = (uint32_t)fminf(fmaxf((cz - slo.z) * sinv.z * 1024.0f, 0.0f), 1023.0f);
    uint32_t code = (expand_bits10(qx) << 2) | (expand_bits10(qy) << 1) | expand_bits10(qz);
    keys[i] = ((uint64_t)code << 32) | (uint32_t)i; // the index makes every key unique
}

// bitonic sort of 64-bit keys: strides >= 1024 go through global memory one compare-exchange pass at a time,
// everything below runs inside a 2048-key shared-memory block
__global__ void k_bitonic_global(uint64_t *keys, int j, int k) {
    unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned ixj = i ^ j;
    if (ixj > i) {
        uint64_t a = keys[i], b = keys[ixj];
        bool up = ((i & k) == 0);
        if ((a > b) == up) { keys[i] = b; keys[ixj] = a; }
    }
}
#define BITONIC_BLOCK 2048
__global__ void __launch_bounds__(1024) k_bitonic_shared(uint64_t *keys, int k_start, int k_end, int j_start) {
    // runs the passes (k, j) for k in [k_start..k_end] and j from min(j_start, k/2) down to 1, all with j < BITONIC_BLOCK
    __shared__ uint64_t s[BITONIC_BLOCK];
    unsigned base = blockIdx.x * BITONIC_BLOCK;
    s[threadIdx.x] = keys[base + threadIdx.x];
    s[threadIdx.x + 1024] = keys[base + threadIdx.x + 1024];
    __syncthreads();
    for (int k = k_start; k <= k_end; k <<= 1) {
        int jmax = (k == k_start) ? j_start : (k >> 1);
        for (int j = jmax; j > 0; j >>= 1) {
            for (int q = 0; q < 2; q++) {
                unsigned li = threadIdx.x + q * 1024;
                unsigned lj = li ^ j;
                if (lj > li) {
                    unsigned gi = base + li;
                    uint64_t a = s[li], b = s[lj];
                    bool up = ((gi & k) == 0);
                    if ((a > b) == up) { s[li] = b; s[lj] = a; }
                }
            }
            __syncthreads();
        }
    }
    keys[base + threadIdx.x] = s[threadIdx.x];
    keys[base + threadIdx.x + 1024] = s[threadIdx.x + 1024];
}

static void bitonic_sort(uint64_t *d_keys, int npad, cudaStream_t st) {
    // npad is a power of two >= BITONIC_BLOCK
    int nblk = npad / BITONIC_BLOCK;
    k_bitonic_shared<<<nblk, 1024, 0, st>>>(d_keys, 2, BITONIC_BLOCK, 1);
    for (int k = BITONIC_BLOCK * 2; k <= npad; k <<= 1) {
        int j = k >> 1;
        for (; j >= BITONIC_BLOCK; j >>= 1) k_bitonic_global<<<npad / 256, 256, 0, st>>>(d_keys, j, k);
        k_bitonic_shared<<<nblk, 1024, 0, st>>>(d_keys, k, k, j);
    }
}

// ---------------------------------------------------------------------------------------------------------
// Karras 2012: internal node i covers a key range found from common-prefix lengths; children index >= 0 are
// internal nodes, < 0 leaves (~sorted position).
__device__ __forceinline__ int delta(const uint64_t *keys, int N, int i, int j) {
    if (j < 0 || j >= N) return -1;
    return __clzll(keys[i] ^ keys[j]);
}

__global__ void k_hierarchy(const uint64_t *__restrict__ keys, int N, int2 *__restrict__ children, int *__restrict__ parent) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N - 1) return;
    int d = (delta(keys, N, i, i + 1) - delta(keys, N, i, i - 1)) >= 0 ? 1 : -1;
    int dmin = delta(keys, N, i, i - d);
    int lmax = 2;
    while (delta(keys, N, i, i + lmax * d) > dmin) lmax <<= 1;
    int l = 0;
    for (int t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, N, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta(keys, N, i, j);
    int s = 0;
    int t = l;
    do {
        t = (t + 1) >> 1;
        if (delta(keys, N, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + min(d, 0);
    int left = (min(i, j) == gamma) ? ~gamma : gamma;
    int right = (max(i, j) == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    children[i] = make_int2(left, right);
    // parent slots: internal node n at n, leaf at sorted position p at (N-1)+p
    parent[left >= 0 ? left : (N - 1) + (~left)] = i;
    parent[right >= 0 ? right : (N - 1) + (~right)] = i;
    if (i == 0) parent[0] = -1;
}

// bottom-up refit: the second thread to arrive at a node merges its two children and moves on
__global__ void k_refit(const uint64_t *__restrict__ keys, const TriVerts *__restrict__ tv, int N, float pad,
                        const int2 *__restrict__ children, const int *__restrict__ parent, float *__restrict__ box /* (2N-1) x 6 */,
                        int *__restrict__ flags, float4 *__restrict__ tribox, const int *__restrict__ pid, int *__restrict__ spid /* 2N-1 */, int nfaces) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= N) return;
    int tri = (int)(uint32_t)keys[p];
    TriVerts t = tv[tri];
    float lo[3], hi[3];
    lo[0] = fminf(t.a.x, fminf(t.b.x, t.c.x)) - pad; hi[0] = fmaxf(t.a.x, fmaxf(t.b.x, t.c.x)) + pad;
    lo[1] = fminf(t.a.y, fminf(t.b.y, t.c.y)) - pad; hi[1] = fmaxf(t.a.y, fmaxf(t.b.y, t.c.y)) + pad;
    lo[2] = fminf(t.a.z, fminf(t.b.z, t.c.z)) - pad; hi[2] = fmaxf(t.a.z, fmaxf(t.b.z, t.c.z)) + pad;
    size_t self = (size_t)(N - 1) + p;
    for (int d = 0; d < 3; d++) { box[self * 6 + d] = lo[d]; box[self * 6 + 3 + d] = hi[d]; }
    spid[self] = pid[tri]; // subtree plane id: the id shared by every triangle below a node, 0 if they differ (or have none)
    tribox[2 * (size_t)tri] = make_float4(lo[0], lo[1], lo[2], 0.f);
    tribox[2 * (size_t)tri + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
    if (N == 1) return;
    __threadfence();
    int node = parent[self];
    while (node >= 0) {
        if (atomicAdd(&flags[node], 1) == 0) return; // first arrival: sibling not done yet
        __threadfence();
        int2 ch = children[node];
        size_t l = ch.x >= 0 ? (size_t)ch.x : (size_t)(N - 1) + (~ch.x);
        size_t r = ch.y >= 0 ? (size_t)ch.y : (size_t)(N - 1) + (~ch.y);
        volatile float *vb = box;
        for (int d = 0; d < 3; d++) {
            box[(size_t)node * 6 + d] = fminf(vb[l * 6 + d], vb[r * 6 + d]);
            box[(size_t)node * 6 + 3 + d] = fmaxf(vb[l * 6 + 3 + d], vb[r * 6 + 3 + d]);
        }
        {
            volatile int *vs = spid;
            const int sl = vs[l], sr = vs[r];
            // -1: nothing but triangles of gridded faces below (ids 1..nfaces, several of them): the shaft walk of the
            // form-factor kernel never enters such a subtree, faces are found through their own boxes
            const bool fl = sl == -1 || (sl >= 1 && sl <= nfaces), fr = sr == -1 || (sr >= 1 && sr <= nfaces);
            spid[node] = (sl == sr) ? sl : ((fl && fr) ? -1 : 0);
        }
        __threadfence();
        node = parent[node];
    }
}

__global__ void k_pack_nodes(const uint64_t *__restrict__ keys, int N, const int2 *__restrict__ children,
                             const float *__restrict__ box, const int *__restrict__ spid, BvhNode *__restrict__ nodes) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N - 1) return;
    int2 ch = children[i];
    size_t l = ch.x >= 0 ? (size_t)ch.x : (size_t)(N - 1) + (~ch.x);
    size_t r = ch.y >= 0 ? (size_t)ch.y : (size_t)(N - 1) + (~ch.y);
    const float *L = box + l * 6, *R = box + r * 6;
    BvhNode n;
    n.a = make_float4(L[0], L[1], L[2], L[3]);
    n.b = make_float4(L[4], L[5], R[0], R[1]);
    n.c = make_float4(R[2], R[3], R[4], R[5]);
    // leaves refer to the ORIGINAL triangle id
    int li = ch.x >= 0 ? ch.x : ~(int)(uint32_t)keys[~ch.x];
    int ri = ch.y >= 0 ? ch.y : ~(int)(uint32_t)keys[~ch.y];
    n.d = make_int4(li, ri, spid[l], spid[r]); // plane id common to everything below each child (leaf: the triangle's own), 0 = mixed, -1 = mixed but gridded faces only
    nodes[i] = n;
}

// tile composition for the form-factor kernel: sorted Morton order (spatially compact groups of 64) or the caller's order
__global__ void k_tile_order(const uint64_t *__restrict__ keys, int N, int nslots, int morton, int *__restrict__ order) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nslots) return;
    order[p] = p < N ? (morton ? (int)(uint32_t)keys[p] : p) : -1;
}

int dz_build_lbvh(daisy_ctx *ctx) {
    DzRange range_("lbvh build: morton, sort, hierarchy, refit, pack");
    int N = ctx->N;
    cudaStream_t st = ctx->stream;
    cudaEvent_t e0, e1;
    DZ_CUDA(cudaEventCreate(&e0));
    DZ_CUDA(cudaEventCreate(&e1));
    // a rebuild (daisy_ctx_update_geometry) replaces the previous hierarchy
    cudaFree(ctx->d_triverts); cudaFree(ctx->d_nodes); cudaFree(ctx->d_tribox); cudaFree(ctx->d_order); free(ctx->h_order);
    ctx->d_triverts = nullptr; ctx->d_nodes = nullptr; ctx->d_tribox = nullptr; ctx->d_order = nullptr; ctx->h_order = nullptr;
    DZ_CUDA(cudaEventRecord(e0, st));
    DZ_CUDA(cudaMalloc(&ctx->d_triverts, sizeof(TriVerts) * (size_t)(N > 0 ? N : 1)));
    DZ_CUDA(cudaMalloc(&ctx->d_nodes, sizeof(BvhNode) * (size_t)(N > 1 ? N - 1 : 1)));
    DZ_CUDA(cudaMalloc(&ctx->d_tribox, sizeof(float4) * 2 * (size_t)(N > 0 ? N : 1)));
    ctx->nslots = ((N + 63) / 64) * 64;
    DZ_CUDA(cudaMalloc(&ctx->d_order, sizeof(int) * (size_t)(ctx->nslots > 0 ? ctx->nslots : 1)));
    ctx->h_order = (int *)malloc(sizeof(int) * (size_t)(ctx->nslots > 0 ? ctx->nslots : 1));
    if (!ctx->h_order) { daisy_set_error("out of host memory"); return DAISY_E_NOMEM; }
    if (N == 0) { ctx->root = 0; DZ_CUDA(cudaEventDestroy(e0)); DZ_CUDA(cudaEventDestroy(e1)); return DAISY_OK; }
    int npad = BITONIC_BLOCK;
    while (npad < N) npad <<= 1;
    uint64_t *d_keys = nullptr;
    int2 *d_children = nullptr;
    int *d_parent = nullptr, *d_flags = nullptr;
    float *d_box = nullptr;
    int *d_spid = nullptr;
    DZ_CUDA(cudaMalloc(&d_spid, sizeof(int) * (size_t)(2 * N)));
    DZ_CUDA(cudaMalloc(&d_keys, sizeof(uint64_t) * (size_t)npad));
    DZ_CUDA(cudaMalloc(&d_children, sizeof(int2) * (size_t)N));
    DZ_CUDA(cudaMalloc(&d_parent, sizeof(int) * (size_t)(2 * N)));
    DZ_CUDA(cudaMalloc(&d_flags, sizeof(int) * (size_t)N));
    DZ_CUDA(cudaMalloc(&d_box, sizeof(float) * 6 * (size_t)(2 * N)));
    DZ_CUDA(cudaMemsetAsync(d_flags, 0, sizeof(int) * (size_t)N, st));
    float3 slo = make_float3(ctx->scene_lo[0], ctx->scene_lo[1], ctx->scene_lo[2]);
    float3 sinv;
    float ex = ctx->scene_hi[0] - ctx->scene_lo[0], ey = ctx->scene_hi[1] - ctx->scene_lo[1], ez = ctx->scene_hi[2] - ctx->scene_lo[2];
    sinv.x = ex > 0 ? 1.0f / ex : 0.f; sinv.y = ey > 0 ? 1.0f / ey : 0.f; sinv.z = ez > 0 ? 1.0f / ez : 0.f;
    k_triverts_morton<<<(npad + 255) / 256, 256, 0, st>>>(ctx->d_vertices, ctx->d_tri, N, npad, slo, sinv, ctx->d_triverts, d_keys);
    bitonic_sort(d_keys, npad, st);
    if (N > 1) {
        k_hierarchy<<<(N - 1 + 255) / 256, 256, 0, st>>>(d_keys, N, d_children, d_parent);
    }
    k_refit<<<(N + 255) / 256, 256, 0, st>>>(d_keys, ctx->d_triverts, N, ctx->pad, d_children, d_parent, d_box, d_flags, ctx->d_tribox, ctx->d_pid, d_spid, ctx->nfaces);
    if (N > 1) {
        k_pack_nodes<<<(N - 1 + 255) / 256, 256, 0, st>>>(d_keys, N, d_children, d_box, d_spid, ctx->d_nodes);
        ctx->root = 0;
    } else {
        ctx->root = ~0; // single triangle: the root is the leaf of triangle 0
    }
    {
        const char *e = getenv("DAISY_FF_ORDER"); // "identity": tiles of 64 consecutive caller indices (A/B switch; results are identical)
        const int morton = !(e && e[0] == 'i');
        k_tile_order<<<(ctx->nslots + 255) / 256, 256, 0, st>>>(d_keys, N, ctx->nslots, morton, ctx->d_order);
    }
    DZ_CUDA(cudaGetLastError());
    DZ_CUDA(cudaEventRecord(e1, st));
    DZ_CUDA(cudaMemcpyAsync(ctx->h_order, ctx->d_order, sizeof(int) * (size_t)ctx->nslots, cudaMemcpyDeviceToHost, st));
    DZ_CUDA(cudaStreamSynchronize(st));
    float ms = 0.f;
    DZ_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    ctx->lbvh_ms = ms;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(d_keys); cudaFree(d_children); cudaFree(d_parent); cudaFree(d_flags); cudaFree(d_box); cudaFree(d_spid);
    return DAISY_OK;
}

// ---------------------------------------------------------------------------------------------------------
// closest hit: (t, triangleId) lexicographic minimum over all triangles the watertight test accepts with t > 0
// (device routine in closest.cuh, shared with the traceScreen kernel in trace.cu)
__global__ void __launch_bounds__(128) k_closest(const BvhNode *__restrict__ nodes, const TriVerts *__restrict__ tv, int root,
                                                 int ntri, int n, const float *__restrict__ rays, daisy_hit *__restrict__ hits) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    f3 o = mk3(rays[6 * (size_t)i], rays[6 * (size_t)i + 1], rays[6 * (size_t)i + 2]);
    f3 d = mk3(rays[6 * (size_t)i + 3], rays[6 * (size_t)i + 4], rays[6 * (size_t)i + 5]);
    hits[i] = closest_hit(nodes, tv, root, ntri, o, d);
}

int dz_launch_closest(daisy_ctx *ctx, int n, const float *d_rays, daisy_hit *d_hits) {
    if (n <= 0) return DAISY_OK;
    k_closest<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_nodes, ctx->d_triverts, ctx->root, ctx->N, n, d_rays, d_hits);
    DZ_CUDA(cudaGetLastError());
    return DAISY_OK;
}
