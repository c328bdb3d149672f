// api.cu -- the C-ABI of include/daisy_b200.h for the context (mesh, LBVH, ray query, form factors).
// The solver half of the ABI lives in gather.cu.
#include "daisy_common.cuh"
#include <stdarg.h>
#include <chrono>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <unordered_map>
#include <vector>

static thread_local char g_err[1024] = "";

void daisy_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *daisy_last_error(void) { return g_err; }
extern "C" int daisy_version(void) { return 100; }
extern "C" int daisy_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

cudaError_t dz_scratch(daisy_ctx *ctx, int slot, size_t bytes, void **out) {
    if (bytes == 0) bytes = 16;
    if (ctx->scratch_bytes[slot] < bytes) {
        cudaFree(ctx->scratch[slot]);
        ctx->scratch[slot] = nullptr; ctx->scratch_bytes[slot] = 0;
        const size_t want = bytes + bytes / 4; // some head room: frame sizes creep
        cudaError_t e = cudaMalloc(&ctx->scratch[slot], want);
        if (e != cudaSuccess) { cudaGetLastError(); e = cudaMalloc(&ctx->scratch[slot], bytes); if (e != cudaSuccess) return e; ctx->scratch_bytes[slot] = bytes; }
        else ctx->scratch_bytes[slot] = want;
    }
    *out = ctx->scratch[slot];
    return cudaSuccess;
}

static void free_ctx(daisy_ctx *c) {
    if (!c) return;
    for (int i = 0; i < 6; i++) cudaFree(c->scratch[i]);
    if (c->peers_set && c->peers_ipc)
        for (int g = 0; g < c->nranks && g < 16; g++)
            if (g != c->rank && c->peerF[g]) cudaIpcCloseMemHandle(c->peerF[g]);
    cudaFree(c->d_vertices); cudaFree(c->d_normals); cudaFree(c->d_tri); cudaFree(c->d_triverts); cudaFree(c->d_tribox); cudaFree(c->d_geom); cudaFree(c->d_plane); cudaFree(c->d_pid); cudaFree(c->d_nbr);
    dz_free_faces(c);
    cudaFree(c->d_nodes); cudaFree(c->d_F); cudaFree(c->d_order); free(c->h_order); cudaFree(c->d_vadj_off); cudaFree(c->d_vadj);
    delete c;
}


// ---- plane ids ---------------------------------------------------------------------------------------------------------
// pid[t] >= 1: id of a plane that holds triangle t together with at least one other triangle; 0: none.  Two triangles with
// the same id lie in one plane in the sense coplanar skipping needs (formfactor.cu, k_tri_planes): every vertex of every
// member is within PLANE_TAU x scene extent of ONE plane P, and every member's own normal is within 1e-3 of P's.
//  * axis-aligned planes are recognised exactly (all three vertices carry the very same x, y or z);
//  * other planes (rotated boxes, ramps) are found by seeded fitting in double precision: triangles are bucketed by their
//    rounded plane equation, the largest unassigned triangle of a bucket seeds a plane, members within tolerance are
//    collected, the plane is refitted to the members' vertices (least squares) and members are collected again -- the
//    refits matter because the normal of one small triangle with float-rounded vertices is only good to ~1e-5 rad.
// Whatever ends up alone keeps id 0 and is simply never skipped.
#define PLANE_TAU 3e-7
namespace {
struct V3d { double x, y, z; };
inline V3d vsub(V3d a, V3d b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
inline double vdot(V3d a, V3d b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3d vcross(V3d a, V3d b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }

// least-squares plane through a point set: centroid + eigenvector of the smallest eigenvalue of the covariance (Jacobi)
bool fit_plane(const std::vector<V3d> &pts, V3d &n, V3d &c) {
    if (pts.size() < 3) return false;
    c = { 0, 0, 0 };
    for (const V3d &p : pts) { c.x += p.x; c.y += p.y; c.z += p.z; }
    c.x /= pts.size(); c.y /= pts.size(); c.z /= pts.size();
    double a[3][3] = { { 0 } }, v[3][3] = { { 1, 0, 0 }, { 0, 1, 0 }, { 0, 0, 1 } };
    for (const V3d &p : pts) {
        const double d[3] = { p.x - c.x, p.y - c.y, p.z - c.z };
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) a[i][j] += d[i] * d[j];
    }
    for (int sweep = 0; sweep < 32; sweep++) {
        const double off = fabs(a[0][1]) + fabs(a[0][2]) + fabs(a[1][2]);
        if (off < 1e-300) break;
        for (int p = 0; p < 2; p++)
            for (int q = p + 1; q < 3; q++) {
                if (fabs(a[p][q]) < 1e-300) continue;
                const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double cs = 1.0 / sqrt(t * t + 1.0), sn = t * cs;
                for (int k = 0; k < 3; k++) { const double akp = a[k][p], akq = a[k][q]; a[k][p] = cs * akp - sn * akq; a[k][q] = sn * akp + cs * akq; }
                for (int k = 0; k < 3; k++) { const double apk = a[p][k], aqk = a[q][k]; a[p][k] = cs * apk - sn * aqk; a[q][k] = sn * apk + cs * aqk; }
                for (int k = 0; k < 3; k++) { const double vkp = v[k][p], vkq = v[k][q]; v[k][p] = cs * vkp - sn * vkq; v[k][q] = sn * vkp + cs * vkq; }
            }
    }
    int m = 0;
    if (a[1][1] < a[m][m]) m = 1;
    if (a[2][2] < a[m][m]) m = 2;
    n = { v[0][m], v[1][m], v[2][m] };
    const double l = sqrt(vdot(n, n));
    if (!(l > 0)) return false;
    n = { n.x / l, n.y / l, n.z / l };
    return true;
}
} // namespace

// plain-array form for faces.cu
bool dz_fit_plane(const double *pts_xyz, size_t npts, double n_out[3], double c_out[3]) {
    std::vector<V3d> pts(npts);
    for (size_t i = 0; i < npts; i++) pts[i] = { pts_xyz[3 * i], pts_xyz[3 * i + 1], pts_xyz[3 * i + 2] };
    V3d n, c;
    if (!fit_plane(pts, n, c)) return false;
    n_out[0] = n.x; n_out[1] = n.y; n_out[2] = n.z; c_out[0] = c.x; c_out[1] = c.y; c_out[2] = c.z;
    return true;
}

static void assign_plane_ids(const float *vertices, const int32_t *tri_idx, int ntri, float ext, std::vector<int> &pid) {
    pid.assign((size_t)(ntri > 0 ? ntri : 1), 0);
    int next_id = 1;
    auto vert = [&](int t, int k) -> V3d {
        const float *p = vertices + 3 * (size_t)tri_idx[6 * (size_t)t + k];
        return { (double)p[0], (double)p[1], (double)p[2] };
    };
    // (1) exact axis-aligned planes
    std::unordered_map<uint64_t, int> ids;
    for (int i = 0; i < ntri; i++) {
        const float *a = vertices + 3 * (size_t)tri_idx[6 * (size_t)i], *b = vertices + 3 * (size_t)tri_idx[6 * (size_t)i + 1],
                    *cc = vertices + 3 * (size_t)tri_idx[6 * (size_t)i + 2];
        int axis = -1, count = 0;
        for (int d = 0; d < 3; d++)
            if (a[d] == b[d] && a[d] == cc[d]) { axis = d; count++; }
        if (count != 1) continue; // not axis-aligned, or degenerate (a segment or a point)
        float v = a[axis] + 0.0f; // -0 -> +0
        uint32_t bits;
        memcpy(&bits, &v, 4);
        const uint64_t key = ((uint64_t)axis << 32) | bits;
        auto it = ids.find(key);
        if (it == ids.end()) it = ids.emplace(key, next_id++).first;
        pid[(size_t)i] = it->second;
    }
    // (2) general planes among the rest
    if (!(ext > 0.f)) return;
    const double tau = PLANE_TAU * (double)ext;
    struct TP { V3d n; double d, area2; };
    std::vector<TP> tp((size_t)ntri);
    std::unordered_map<uint64_t, std::vector<int>> buckets;
    const double qn = 2e-3, qd = 2e-3 * (double)ext;
    for (int i = 0; i < ntri; i++) {
        if (pid[(size_t)i]) continue;
        const V3d a = vert(i, 0), b = vert(i, 1), c = vert(i, 2);
        V3d n = vcross(vsub(b, a), vsub(c, a));
        const double l = sqrt(vdot(n, n));
        tp[(size_t)i].area2 = l;
        if (!(l > 0)) continue;
        n = { n.x / l, n.y / l, n.z / l };
        // canonical sign: the component of largest magnitude is positive (a plane has two unit normals)
        const double ax = fabs(n.x), ay = fabs(n.y), az = fabs(n.z);
        const double lead = (ax >= ay && ax >= az) ? n.x : (ay >= az ? n.y : n.z);
        if (lead < 0) n = { -n.x, -n.y, -n.z };
        tp[(size_t)i].n = n;
        tp[(size_t)i].d = vdot(n, a);
        const int64_t k0 = (int64_t)floor(n.x / qn), k1 = (int64_t)floor(n.y / qn), k2 = (int64_t)floor(n.z / qn), k3 = (int64_t)floor(tp[(size_t)i].d / qd);
        const uint64_t key = ((uint64_t)(k0 & 0xffff) << 48) | ((uint64_t)(k1 & 0xffff) << 32) | ((uint64_t)(k2 & 0xffff) << 16) | (uint64_t)(k3 & 0xffff);
        buckets[key].push_back(i);
    }
    std::vector<V3d> pts;
    std::vector<int> members, rest;
    std::vector<char> taken((size_t)ntri, 0);
    for (auto &kv : buckets) {
        rest = kv.second;
        for (int round = 0; round < 8 && rest.size() >= 2; round++) {
            int seed = rest[0];
            for (int t : rest)
                if (tp[(size_t)t].area2 > tp[(size_t)seed].area2) seed = t;
            V3d n = tp[(size_t)seed].n, c0 = vert(seed, 0);
            auto collect = [&]() {
                members.clear();
                for (int t : rest) {
                    if (fabs(vdot(n, tp[(size_t)t].n)) < 1.0 - 5e-7) continue; // own normal within 1e-3 rad of the plane's
                    double dist = 0.0;
                    for (int k = 0; k < 3; k++) dist = fmax(dist, fabs(vdot(n, vsub(vert(t, k), c0))));
                    if (dist <= tau) members.push_back(t);
                }
            };
            collect();
            for (int refit = 0; refit < 3 && members.size() >= 2; refit++) {
                pts.clear();
                for (int t : members)
                    for (int k = 0; k < 3; k++) pts.push_back(vert(t, k));
                V3d nn, cc;
                if (!fit_plane(pts, nn, cc)) break;
                n = nn; c0 = cc;
                const size_t before = members.size();
                collect();
                if (members.size() == before && refit > 0) break;
            }
            bool has_seed = false;
            for (int t : members) has_seed |= (t == seed);
            if (members.size() >= 2 && has_seed) {
                const int id = next_id++;
                for (int t : members) pid[(size_t)t] = id;
            } else {
                members.assign(1, seed); // the seed stays alone (id 0); take it out and try the next largest
            }
            for (int t : members) taken[(size_t)t] = 1;
            std::vector<int> keep;
            for (int t : rest)
                if (!taken[(size_t)t]) keep.push_back(t);
            rest.swap(keep);
        }
    }
}

extern "C" int daisy_plane_ids(const float *vertices, int nv, const int32_t *tri_idx, int ntri, int32_t *pid_out) {
    DZ_REQUIRE(ntri >= 0 && nv >= 0 && (ntri == 0 || (vertices && tri_idx && pid_out)), DAISY_E_INVALID, "daisy_plane_ids: bad argument");
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int i = 0; i < ntri; i++)
        for (int k = 0; k < 3; k++) {
            const int v = tri_idx[6 * (size_t)i + k];
            DZ_REQUIRE(v >= 0 && v < nv, DAISY_E_INVALID, "daisy_plane_ids: triangle index out of range");
            for (int d = 0; d < 3; d++) { lo[d] = fminf(lo[d], vertices[3 * (size_t)v + d]); hi[d] = fmaxf(hi[d], vertices[3 * (size_t)v + d]); }
        }
    float ext = 0.f;
    for (int d = 0; d < 3; d++) if (ntri) ext = fmaxf(ext, hi[d] - lo[d]);
    std::vector<int> pid;
    assign_plane_ids(vertices, tri_idx, ntri, ext, pid);
    for (int i = 0; i < ntri; i++) pid_out[i] = pid[(size_t)i];
    return DAISY_OK;
}

int dz_face_grid_stats(float ext, const float *vertices, const int32_t *tri_idx, int ntri, std::vector<int> &pid, int max_faces, int64_t *out6, int *nfaces_out); // faces.cu
extern "C" int daisy_face_grid_stats(const float *vertices, int nv, const int32_t *tri_idx, int ntri, int max_faces, int64_t *stats6, int32_t *nfaces_out, int32_t *pid_out) {
    DZ_REQUIRE(ntri >= 0 && nv >= 0 && max_faces >= 0 && nfaces_out && (ntri == 0 || (vertices && tri_idx)), DAISY_E_INVALID, "daisy_face_grid_stats: bad argument");
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int i = 0; i < ntri; i++)
        for (int k = 0; k < 3; k++) {
            const int v = tri_idx[6 * (size_t)i + k];
            DZ_REQUIRE(v >= 0 && v < nv, DAISY_E_INVALID, "daisy_face_grid_stats: triangle index out of range");
            for (int d = 0; d < 3; d++) { lo[d] = fminf(lo[d], vertices[3 * (size_t)v + d]); hi[d] = fmaxf(hi[d], vertices[3 * (size_t)v + d]); }
        }
    float ext = 0.f;
    for (int d = 0; d < 3; d++) if (ntri) ext = fmaxf(ext, hi[d] - lo[d]);
    std::vector<int> pid;
    assign_plane_ids(vertices, tri_idx, ntri, ext, pid);
    int nf = 0;
    const int rc = dz_face_grid_stats(ext, vertices, tri_idx, ntri, pid, max_faces, stats6, &nf);
    if (rc) return rc;
    *nfaces_out = nf;
    if (pid_out) for (int i = 0; i < ntri; i++) pid_out[i] = pid[(size_t)i];
    return DAISY_OK;
}

int dz_face_grid_dump(float ext, const float *vertices, const int32_t *tri_idx, int ntri, std::vector<int> &pid, int face, float *frame16, signed char *state,
                      int32_t *count, int64_t cap); // faces.cu
extern "C" int daisy_face_grid_dump(const float *vertices, int nv, const int32_t *tri_idx, int ntri, int face, float *frame16, signed char *state, int32_t *count,
                                    int64_t capacity) {
    DZ_REQUIRE(ntri > 0 && nv > 0 && vertices && tri_idx && frame16, DAISY_E_INVALID, "daisy_face_grid_dump: bad argument");
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int i = 0; i < ntri; i++)
        for (int k = 0; k < 3; k++) {
            const int v = tri_idx[6 * (size_t)i + k];
            DZ_REQUIRE(v >= 0 && v < nv, DAISY_E_INVALID, "daisy_face_grid_dump: triangle index out of range");
            for (int d = 0; d < 3; d++) { lo[d] = fminf(lo[d], vertices[3 * (size_t)v + d]); hi[d] = fmaxf(hi[d], vertices[3 * (size_t)v + d]); }
        }
    float ext = 0.f;
    for (int d = 0; d < 3; d++) ext = fmaxf(ext, hi[d] - lo[d]);
    std::vector<int> pid;
    assign_plane_ids(vertices, tri_idx, ntri, ext, pid);
    return dz_face_grid_dump(ext, vertices, tri_idx, ntri, pid, face, frame16, state, count, capacity);
}

static void set_partition(daisy_ctx *c, int rank, int nranks) {
    c->rank = rank; c->nranks = nranks;
    int n = (c->N + nranks - 1) / nranks;
    // single block: multiple of 4 (16-byte TMA alignment); several blocks: multiple of 256 so that a 256-column
    // TMA tile of the residual never straddles two ranks' blocks
    n = (nranks > 1) ? ((n + 255) / 256) * 256 : ((n + 3) / 4) * 4;
    if (n < 4) n = 4;
    c->rows_per_rank = n;
    c->row0 = (int)fmin((double)c->N, (double)rank * n);
    c->row1 = (int)fmin((double)c->N, (double)(rank + 1) * n);
    int64_t ncols = (int64_t)nranks * n;
    if (ncols < c->N) ncols = c->N;
    c->ldF = ((ncols + 31) / 32) * 32;
}

extern "C" int daisy_ctx_create(const float *vertices, int nv, const float *normals, int nn, const int32_t *tri_idx, int ntri,
                                int device, daisy_ctx **out) {
    DZ_REQUIRE(out, DAISY_E_INVALID, "daisy_ctx_create: null out pointer");
    *out = nullptr;
    DzRange range_("daisy_ctx_create: mesh upload, plane ids, LBVH, patch records");
    DZ_REQUIRE(nv >= 0 && nn >= 0 && ntri >= 0, DAISY_E_INVALID, "daisy_ctx_create: negative count");
    DZ_REQUIRE(ntri == 0 || (vertices && normals && tri_idx), DAISY_E_INVALID, "daisy_ctx_create: null array");
    for (int i = 0; i < ntri; i++)
        for (int k = 0; k < 6; k++) {
            int v = tri_idx[6 * (size_t)i + k];
            DZ_REQUIRE(v >= 0 && v < (k < 3 ? nv : nn), DAISY_E_INVALID, "daisy_ctx_create: triangle index out of range");
        }
    int ndev = 0;
    DZ_CUDA(cudaGetDeviceCount(&ndev));
    DZ_REQUIRE(device >= 0 && device < ndev, DAISY_E_INVALID, "daisy_ctx_create: no such CUDA device");
    DZ_CUDA(cudaSetDevice(device));
    daisy_ctx *c = new daisy_ctx();
    c->device = device; c->N = ntri; c->nv = nv; c->nn = nn;
    cudaDeviceProp prop;
    DZ_CUDA(cudaGetDeviceProperties(&prop, device));
    c->num_sms = prop.multiProcessorCount;
    set_partition(c, 0, 1);
    // scene bounds over the vertices the triangles use (host: the inputs are host arrays anyway)
    for (int d = 0; d < 3; d++) { c->scene_lo[d] = INFINITY; c->scene_hi[d] = -INFINITY; }
    for (int i = 0; i < ntri; i++)
        for (int k = 0; k < 3; k++) {
            const float *p = vertices + 3 * (size_t)tri_idx[6 * (size_t)i + k];
            for (int d = 0; d < 3; d++) { c->scene_lo[d] = fminf(c->scene_lo[d], p[d]); c->scene_hi[d] = fmaxf(c->scene_hi[d], p[d]); }
        }
    float ext = 0.f, mag = 0.f;
    for (int d = 0; d < 3; d++)
        if (ntri) {
            ext = fmaxf(ext, c->scene_hi[d] - c->scene_lo[d]);
            mag = fmaxf(mag, fmaxf(fabsf(c->scene_lo[d]), fabsf(c->scene_hi[d])));
        }
    c->ext = ext;
    // Conservative box padding; results never depend on it (tests compare with brute force).  1e-4 x the extent, but never
    // below 16 ulp of the largest coordinate: far from the origin a smaller pad rounds away (lo - pad == lo), a ray lying in
    // a box's face plane then reads 0 * inf = NaN there and the slab test drops a box that holds its hit.
    const float ulp = nextafterf(mag, INFINITY) - mag;
    c->pad = fmaxf(1e-4f * ext, 16.0f * ulp);
    // The face grids and coplanar skipping rest on margins that are fractions of the extent too, and on ray origins that
    // round by far less than those margins.  When the coordinates round at more than 1/256 of 1e-4 x the extent (a scene
    // many times its own size away from the origin), neither is used: every plane id stays 0, so nothing is skipped.
    const bool far_from_origin = 1e-4f * ext < 256.0f * ulp;
#define CC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { daisy_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); free_ctx(c); return DAISY_E_CUDA; } } while (0)
    CC(cudaMalloc(&c->d_vertices, sizeof(float) * 3 * (size_t)(nv > 0 ? nv : 1)));
    CC(cudaMalloc(&c->d_normals, sizeof(float) * 3 * (size_t)(nn > 0 ? nn : 1)));
    CC(cudaMalloc(&c->d_tri, sizeof(int) * 6 * (size_t)(ntri > 0 ? ntri : 1)));
    CC(cudaMalloc(&c->d_geom, sizeof(PatchGeom) * (size_t)(ntri > 0 ? ntri : 1)));
    CC(cudaMalloc(&c->d_plane, sizeof(float4) * (size_t)(ntri > 0 ? ntri : 1)));
    CC(cudaMalloc(&c->d_nbr, sizeof(int) * 32 * (size_t)(ntri > 0 ? ntri : 1)));
    if (nv) CC(cudaMemcpy(c->d_vertices, vertices, sizeof(float) * 3 * (size_t)nv, cudaMemcpyHostToDevice));
    if (nn) CC(cudaMemcpy(c->d_normals, normals, sizeof(float) * 3 * (size_t)nn, cudaMemcpyHostToDevice));
    if (ntri) CC(cudaMemcpy(c->d_tri, tri_idx, sizeof(int) * 6 * (size_t)ntri, cudaMemcpyHostToDevice));
    {
        std::vector<int> pid;
        if (far_from_origin) pid.assign((size_t)(ntri > 0 ? ntri : 1), 0);
        else assign_plane_ids(vertices, tri_idx, ntri, ext, pid);
        { const int rc_ = dz_build_faces(c, vertices, tri_idx, ntri, pid); if (rc_) { free_ctx(c); return rc_; } } // renumbers pid: face f = id f + 1
        CC(cudaMalloc(&c->d_pid, sizeof(int) * pid.size()));
        CC(cudaMemcpy(c->d_pid, pid.data(), sizeof(int) * pid.size(), cudaMemcpyHostToDevice));
    }
    {
        // MeshS::trianglesPerVertex (MeshS.cpp:107-109) as CSR, lists in ascending triangle order: Drawer::interpolate sums
        // the patch colours of a vertex in exactly that order
        std::vector<int> off((size_t)nv + 1, 0), adj((size_t)3 * (ntri > 0 ? ntri : 1), 0);
        for (int i = 0; i < ntri; i++)
            for (int k = 0; k < 3; k++) off[(size_t)tri_idx[6 * (size_t)i + k] + 1]++;
        for (int v = 0; v < nv; v++) off[(size_t)v + 1] += off[v];
        std::vector<int> fill(off.begin(), off.end() - 1);
        for (int i = 0; i < ntri; i++)
            for (int k = 0; k < 3; k++) adj[(size_t)fill[tri_idx[6 * (size_t)i + k]]++] = i;
        CC(cudaMalloc(&c->d_vadj_off, sizeof(int) * off.size()));
        CC(cudaMalloc(&c->d_vadj, sizeof(int) * adj.size()));
        CC(cudaMemcpy(c->d_vadj_off, off.data(), sizeof(int) * off.size(), cudaMemcpyHostToDevice));
        CC(cudaMemcpy(c->d_vadj, adj.data(), sizeof(int) * adj.size(), cudaMemcpyHostToDevice));
    }
#undef CC
    int rc = dz_build_lbvh(c);
    if (!rc) rc = dz_precompute_geom(c);
    if (!rc && cudaStreamSynchronize(c->stream) != cudaSuccess) { daisy_set_error("daisy_ctx_create: %s", cudaGetErrorString(cudaGetLastError())); rc = DAISY_E_CUDA; }
    if (rc) { free_ctx(c); return rc; }
    *out = c;
    return DAISY_OK;
}

extern "C" void daisy_ctx_destroy(daisy_ctx *ctx) {
    if (ctx) cudaSetDevice(ctx->device);
    free_ctx(ctx);
}

extern "C" int daisy_ctx_set_samples(daisy_ctx *ctx, const float *uv, int S) {
    DZ_REQUIRE(ctx && uv, DAISY_E_INVALID, "daisy_ctx_set_samples: null argument");
    DZ_REQUIRE(S >= 1 && S <= DAISY_MAX_SAMPLES, DAISY_E_INVALID, "daisy_ctx_set_samples: S must be in [1,64]");
    DZ_CUDA(cudaSetDevice(ctx->device));
    memset(ctx->h_uv, 0, sizeof(ctx->h_uv));
    memcpy(ctx->h_uv, uv, sizeof(float) * 2 * (size_t)S);
    ctx->S = S;
    return DAISY_OK;
}

extern "C" int daisy_ctx_set_partition(daisy_ctx *ctx, int rank, int nranks) {
    DZ_REQUIRE(ctx, DAISY_E_INVALID, "daisy_ctx_set_partition: null context");
    DZ_REQUIRE(nranks >= 1 && rank >= 0 && rank < nranks, DAISY_E_INVALID, "daisy_ctx_set_partition: bad rank/nranks");
    // the matrix allocation, its leading dimension and any IPC mapping handed to peers are sized from the row range
    DZ_REQUIRE(!ctx->have_F && !ctx->d_F && !ctx->peers_set, DAISY_E_STATE,
               "daisy_ctx_set_partition: form factors already allocated or built (set the partition before daisy_formfactors_alloc/build/write_rows)");
    set_partition(ctx, rank, nranks);
    return DAISY_OK;
}

extern "C" int daisy_ctx_row_range(daisy_ctx *ctx, int *row0, int *row1, int *rows_per_rank) {
    DZ_REQUIRE(ctx, DAISY_E_INVALID, "daisy_ctx_row_range: null context");
    if (row0) *row0 = ctx->row0;
    if (row1) *row1 = ctx->row1;
    if (rows_per_rank) *rows_per_rank = ctx->rows_per_rank;
    return DAISY_OK;
}

extern "C" int daisy_ctx_set_stream(daisy_ctx *ctx, void *cuda_stream) {
    DZ_REQUIRE(ctx, DAISY_E_INVALID, "daisy_ctx_set_stream: null context");
    DZ_CUDA(cudaSetDevice(ctx->device));
    DZ_CUDA(cudaDeviceSynchronize()); // work enqueued on the previous stream (context set-up) is complete before the new one is used
    ctx->stream = (cudaStream_t)cuda_stream;
    return DAISY_OK;
}

// ---- closest hit -------------------------------------------------------------------------------------------
extern "C" int daisy_query_closest_device(daisy_ctx *ctx, int n, const float *d_rays6, daisy_hit *d_hits) {
    DZ_REQUIRE(ctx && (n == 0 || (d_rays6 && d_hits)), DAISY_E_INVALID, "daisy_query_closest_device: null argument");
    DZ_REQUIRE(n >= 0, DAISY_E_INVALID, "daisy_query_closest_device: negative ray count");
    DZ_CUDA(cudaSetDevice(ctx->device));
    int rc = dz_launch_closest(ctx, n, d_rays6, d_hits);
    if (rc) return rc;
    DZ_CUDA(cudaStreamSynchronize(ctx->stream));
    return DAISY_OK;
}

extern "C" int daisy_query_closest(daisy_ctx *ctx, int n, const float *rays6, daisy_hit *hits) {
    DZ_REQUIRE(ctx && (n == 0 || (rays6 && hits)), DAISY_E_INVALID, "daisy_query_closest: null argument");
    DZ_REQUIRE(n >= 0, DAISY_E_INVALID, "daisy_query_closest: negative ray count");
    if (n == 0) return DAISY_OK;
    DZ_CUDA(cudaSetDevice(ctx->device));
    float *d_r = nullptr;
    daisy_hit *d_h = nullptr;
    cudaError_t e = dz_scratch(ctx, 0, sizeof(float) * 6 * (size_t)n, (void **)&d_r);
    if (e == cudaSuccess) e = dz_scratch(ctx, 1, sizeof(daisy_hit) * (size_t)n, (void **)&d_h);
    if (e != cudaSuccess) { daisy_set_error("daisy_query_closest: %s", cudaGetErrorString(e)); return DAISY_E_CUDA; }
    int rc = DAISY_OK;
    e = cudaMemcpyAsync(d_r, rays6, sizeof(float) * 6 * (size_t)n, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) rc = dz_launch_closest(ctx, n, d_r, d_h);
    if (e == cudaSuccess && !rc) e = cudaMemcpyAsync(hits, d_h, sizeof(daisy_hit) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && !rc) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { daisy_set_error("daisy_query_closest: %s", cudaGetErrorString(e)); return DAISY_E_CUDA; }
    return rc;
}

// ---- form factors --------------------------------------------------------------------------------------------
extern "C" int daisy_unoccluded_rows(daisy_ctx *ctx, int variant, int row0, int nrows, daisy_tripl *out) {
    DZ_REQUIRE(ctx && out, DAISY_E_INVALID, "daisy_unoccluded_rows: null argument");
    DZ_REQUIRE(variant == DAISY_FF_DEVICE || variant == DAISY_FF_HOST, DAISY_E_INVALID, "daisy_unoccluded_rows: bad variant");
    DZ_REQUIRE(row0 >= 0 && nrows >= 0 && row0 + nrows <= ctx->N, DAISY_E_INVALID, "daisy_unoccluded_rows: rows out of range");
    if (nrows == 0 || ctx->N == 0) return DAISY_OK;
    DZ_CUDA(cudaSetDevice(ctx->device));
    const int N = ctx->N;
    int chunk = (int)fmax(1.0, fmin(4096.0, (double)(256u << 20) / (16.0 * N))); // ~256 MB of triplets at a time
    daisy_tripl *d = nullptr;
    DZ_CUDA(cudaMalloc(&d, sizeof(daisy_tripl) * (size_t)chunk * N));
    int rc = DAISY_OK;
    for (int r = row0; r < row0 + nrows && !rc; r += chunk) {
        int nr = (row0 + nrows - r) < chunk ? (row0 + nrows - r) : chunk;
        rc = dz_unoccluded_rows(ctx, variant, r, nr, d);
        if (!rc) {
            cudaError_t e = cudaMemcpyAsync(out + (size_t)(r - row0) * N, d, sizeof(daisy_tripl) * (size_t)nr * N, cudaMemcpyDeviceToHost, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
            if (e != cudaSuccess) { daisy_set_error("daisy_unoccluded_rows: %s", cudaGetErrorString(e)); rc = DAISY_E_CUDA; }
        }
    }
    cudaFree(d);
    return rc;
}

static int ensure_F(daisy_ctx *ctx) {
    if (ctx->d_F) return DAISY_OK;
    size_t rows = (size_t)(ctx->row1 - ctx->row0);
    size_t bytes = sizeof(float) * (rows ? rows : 1) * (size_t)ctx->ldF;
    DZ_CUDA(cudaMalloc(&ctx->d_F, bytes));
    DZ_CUDA(cudaMemsetAsync(ctx->d_F, 0, bytes, ctx->stream)); // padding columns stay zero for the gather
    return DAISY_OK;
}

extern "C" int daisy_formfactors_build(daisy_ctx *ctx, int variant) {
    DZ_REQUIRE(ctx, DAISY_E_INVALID, "daisy_formfactors_build: null context");
    DZ_REQUIRE(variant == DAISY_FF_DEVICE || variant == DAISY_FF_HOST, DAISY_E_INVALID, "daisy_formfactors_build: bad variant");
    DZ_REQUIRE(ctx->S >= 1, DAISY_E_STATE, "daisy_formfactors_build: call daisy_ctx_set_samples first");
    DzRange range_("daisy_formfactors_build: fused form factors + visibility (k_ff_tiles)");
    DZ_CUDA(cudaSetDevice(ctx->device));
    const bool timing = getenv("DAISY_TIMING") != nullptr; // stderr: where the wall time of the call goes
    const auto t0 = std::chrono::steady_clock::now();
    int rc = ensure_F(ctx);
    if (rc) return rc;
    if (timing) { cudaStreamSynchronize(ctx->stream); fprintf(stderr, "daisy_formfactors_build: matrix allocation + zero fill %.3f s\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count()); }
    rc = dz_set_samples_const(ctx);
    if (rc) return rc;
    const auto t1 = std::chrono::steady_clock::now();
    rc = dz_build_formfactors(ctx, variant, nullptr, 0, 0, true);
    if (rc) return rc;
    if (timing) fprintf(stderr, "daisy_formfactors_build: tile list + kernel + clean-up %.3f s (kernel %.3f s)\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count(), ctx->ff_ms * 1e-3);
    ctx->have_F = true;
    ctx->F_version++;
    return DAISY_OK;
}

// ---- multi-GPU: mirrored tiles are written straight into the owning rank's matrix over NVLink -------------------
extern "C" int daisy_formfactors_alloc(daisy_ctx *ctx) {
    DZ_REQUIRE(ctx, DAISY_E_INVALID, "daisy_formfactors_alloc: null context");
    DZ_CUDA(cudaSetDevice(ctx->device));
    int rc = ensure_F(ctx);
    if (rc) return rc;
    DZ_CUDA(cudaStreamSynchronize(ctx->stream)); // the zero fill must be complete before any peer may write
    return DAISY_OK;
}

extern "C" int daisy_formfactors_ipc_handle(daisy_ctx *ctx, void *handle64) {
    DZ_REQUIRE(ctx && handle64, DAISY_E_INVALID, "daisy_formfactors_ipc_handle: null argument");
    DZ_REQUIRE(ctx->d_F, DAISY_E_STATE, "daisy_formfactors_ipc_handle: call daisy_formfactors_alloc first");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DZ_CUDA(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    DZ_CUDA(cudaIpcGetMemHandle(&h, ctx->d_F));
    memcpy(handle64, &h, 64);
    return DAISY_OK;
}

extern "C" int daisy_formfactors_set_peers(daisy_ctx *ctx, const void *handles, int nranks) {
    DZ_REQUIRE(ctx && handles, DAISY_E_INVALID, "daisy_formfactors_set_peers: null argument");
    DZ_REQUIRE(nranks == ctx->nranks && nranks <= 16, DAISY_E_INVALID, "daisy_formfactors_set_peers: nranks must match the partition (<= 16)");
    DZ_REQUIRE(ctx->d_F && !ctx->peers_set, DAISY_E_STATE, "daisy_formfactors_set_peers: allocate first, set once");
    DZ_CUDA(cudaSetDevice(ctx->device));
    for (int g = 0; g < nranks; g++) {
        if (g == ctx->rank) { ctx->peerF[g] = ctx->d_F; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)handles + 64 * (size_t)g, 64);
        void *p = nullptr;
        DZ_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
        ctx->peerF[g] = (float *)p;
    }
    ctx->peers_set = true;
    ctx->peers_ipc = true;
    return DAISY_OK;
}

int dz_ctx_set_peer_pointers(daisy_ctx *ctx, float *const *F, int nranks) {
    DZ_REQUIRE(ctx && F, DAISY_E_INVALID, "set_peer_pointers: null argument");
    DZ_REQUIRE(nranks == ctx->nranks && nranks <= 16, DAISY_E_INVALID, "set_peer_pointers: nranks must match the partition (<= 16)");
    DZ_REQUIRE(ctx->d_F && !ctx->peers_set, DAISY_E_STATE, "set_peer_pointers: allocate first, set once");
    for (int g = 0; g < nranks; g++) ctx->peerF[g] = F[g];
    ctx->peers_set = true;
    ctx->peers_ipc = false;
    return DAISY_OK;
}

extern "C" int daisy_formfactors_ld(daisy_ctx *ctx, int64_t *ld_out) {
    DZ_REQUIRE(ctx && ld_out, DAISY_E_INVALID, "daisy_formfactors_ld: null argument");
    *ld_out = ctx->ldF;
    return DAISY_OK;
}

extern "C" int daisy_formfactors_read_rows(daisy_ctx *ctx, int row0, int nrows, float *out) {
    DZ_REQUIRE(ctx && (nrows == 0 || out), DAISY_E_INVALID, "daisy_formfactors_read_rows: null argument");
    DZ_REQUIRE(ctx->have_F, DAISY_E_STATE, "daisy_formfactors_read_rows: no form factors yet");
    DZ_REQUIRE(nrows >= 0 && row0 >= ctx->row0 && row0 + nrows <= ctx->row1, DAISY_E_INVALID, "daisy_formfactors_read_rows: rows outside this context's range");
    if (nrows == 0) return DAISY_OK;
    DZ_CUDA(cudaSetDevice(ctx->device));
    DZ_CUDA(cudaStreamSynchronize(ctx->stream));
    DZ_CUDA(cudaMemcpy2D(out, sizeof(float) * (size_t)ctx->N, ctx->d_F + (size_t)(row0 - ctx->row0) * ctx->ldF, sizeof(float) * (size_t)ctx->ldF,
                         sizeof(float) * (size_t)ctx->N, (size_t)nrows, cudaMemcpyDeviceToHost));
    return DAISY_OK;
}

extern "C" int daisy_formfactors_write_rows(daisy_ctx *ctx, int row0, int nrows, const float *in) {
    DZ_REQUIRE(ctx && (nrows == 0 || in), DAISY_E_INVALID, "daisy_formfactors_write_rows: null argument");
    DZ_REQUIRE(nrows >= 0 && row0 >= ctx->row0 && row0 + nrows <= ctx->row1, DAISY_E_INVALID, "daisy_formfactors_write_rows: rows outside this context's range");
    DZ_CUDA(cudaSetDevice(ctx->device));
    int rc = ensure_F(ctx);
    if (rc) return rc;
    if (nrows)
        DZ_CUDA(cudaMemcpy2DAsync(ctx->d_F + (size_t)(row0 - ctx->row0) * ctx->ldF, sizeof(float) * (size_t)ctx->ldF, in, sizeof(float) * (size_t)ctx->N,
                                  sizeof(float) * (size_t)ctx->N, (size_t)nrows, cudaMemcpyHostToDevice, ctx->stream));
    DZ_CUDA(cudaStreamSynchronize(ctx->stream));
    ctx->have_F = true;
    ctx->F_version++;
    return DAISY_OK;
}

extern "C" int daisy_formfactors_to_csc(daisy_ctx *ctx, int64_t *nnz, float *values, int32_t *inner_idx, int32_t *outer_ptr) {
    DZ_REQUIRE(ctx && nnz, DAISY_E_INVALID, "daisy_formfactors_to_csc: null argument");
    DZ_REQUIRE(ctx->have_F, DAISY_E_STATE, "daisy_formfactors_to_csc: no form factors yet");
    DZ_REQUIRE(ctx->nranks == 1, DAISY_E_STATE, "daisy_formfactors_to_csc: single-GPU contexts only");
    DZ_CUDA(cudaSetDevice(ctx->device));
    const int N = ctx->N;
    // host-side conversion in row chunks (this is the hand-back path for callers that still want an Eigen SpMat)
    std::vector<int64_t> colcount((size_t)N + 1, 0);
    const int chunk = (int)fmax(1.0, fmin((double)N, (double)(128u << 20) / (4.0 * (N ? N : 1))));
    std::vector<float> rows((size_t)chunk * (N ? N : 1));
    for (int r = 0; r < N; r += chunk) {
        int nr = (N - r) < chunk ? (N - r) : chunk;
        int rc = daisy_formfactors_read_rows(ctx, r, nr, rows.data());
        if (rc) return rc;
        for (int i = 0; i < nr; i++)
            for (int c = 0; c < N; c++)
                if (rows[(size_t)i * N + c] != 0.0f) colcount[(size_t)c + 1]++;
    }
    for (int c = 0; c < N; c++) colcount[(size_t)c + 1] += colcount[c];
    *nnz = colcount[N];
    if (!values) return DAISY_OK;
    DZ_REQUIRE(inner_idx && outer_ptr, DAISY_E_INVALID, "daisy_formfactors_to_csc: null index arrays");
    DZ_REQUIRE(*nnz <= 0x7fffffffLL, DAISY_E_INVALID, "daisy_formfactors_to_csc: more non-zeros than Eigen's int index can hold");
    for (int c = 0; c <= N; c++) outer_ptr[c] = (int32_t)colcount[c];
    std::vector<int64_t> fill(colcount.begin(), colcount.end() - 1);
    for (int r = 0; r < N; r += chunk) {
        int nr = (N - r) < chunk ? (N - r) : chunk;
        int rc = daisy_formfactors_read_rows(ctx, r, nr, rows.data());
        if (rc) return rc;
        for (int i = 0; i < nr; i++)
            for (int c = 0; c < N; c++) {
                float v = rows[(size_t)i * N + c];
                if (v != 0.0f) { int64_t p = fill[c]++; values[p] = v; inner_idx[p] = r + i; } // rows ascend => sorted inner indices
            }
    }
    return DAISY_OK;
}

extern "C" int daisy_visibility_masks(daisy_ctx *ctx, int variant, int row0, int nrows, uint64_t *out) {
    DZ_REQUIRE(ctx && (nrows == 0 || out), DAISY_E_INVALID, "daisy_visibility_masks: null argument");
    DZ_REQUIRE(variant == DAISY_FF_DEVICE || variant == DAISY_FF_HOST, DAISY_E_INVALID, "daisy_visibility_masks: bad variant");
    DZ_REQUIRE(ctx->S >= 1, DAISY_E_STATE, "daisy_visibility_masks: call daisy_ctx_set_samples first");
    DZ_REQUIRE(row0 >= 0 && nrows >= 0 && row0 + nrows <= ctx->N, DAISY_E_INVALID, "daisy_visibility_masks: rows out of range");
    if (nrows == 0 || ctx->N == 0) return DAISY_OK;
    DzRange range_("daisy_visibility_masks");
    DZ_CUDA(cudaSetDevice(ctx->device));
    int rc = dz_set_samples_const(ctx);
    if (rc) return rc;
    uint64_t *d = nullptr;
    size_t bytes = sizeof(uint64_t) * (size_t)nrows * ctx->N;
    DZ_CUDA(cudaMalloc(&d, bytes));
    cudaError_t e = cudaMemsetAsync(d, 0, bytes, ctx->stream);
    if (e == cudaSuccess) rc = dz_build_formfactors(ctx, variant, d, row0, row0 + nrows, false);
    if (e == cudaSuccess && !rc) e = cudaMemcpyAsync(out, d, bytes, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && !rc) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) { daisy_set_error("daisy_visibility_masks: %s", cudaGetErrorString(e)); return DAISY_E_CUDA; }
    return rc;
}

// ---- per-row digests of the resident matrix (parity evidence at sizes whose matrix does not fit the host) ----------
// one warp per row; both digests are exact integer reductions, hence independent of the summation order:
//   xor_out[r]  = XOR over columns of the float bit patterns
//   wsum_out[r] = SUM over columns of bits * (2c + 1) mod 2^64   (position sensitive)
__global__ void k_row_digest(const float *__restrict__ F, int64_t ldF, int N, int nrows, uint32_t *__restrict__ xo, unsigned long long *__restrict__ wo) {
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= nrows) return;
    const float *src = F + (size_t)row * ldF;
    uint32_t x = 0;
    unsigned long long w = 0;
    for (int c = lane; c < N; c += 32) {
        const uint32_t b = __float_as_uint(src[c]);
        x ^= b;
        w += (unsigned long long)b * (unsigned long long)(2 * (long long)c + 1);
    }
    for (int o = 16; o > 0; o >>= 1) {
        x ^= __shfl_xor_sync(0xffffffffu, x, o);
        w += __shfl_xor_sync(0xffffffffu, w, o);
    }
    if (lane == 0) { xo[row] = x; wo[row] = w; }
}

extern "C" int daisy_formfactors_row_digest(daisy_ctx *ctx, int row0, int nrows, uint32_t *xor_out, uint64_t *wsum_out) {
    DZ_REQUIRE(ctx && (nrows == 0 || (xor_out && wsum_out)), DAISY_E_INVALID, "daisy_formfactors_row_digest: null argument");
    DZ_REQUIRE(ctx->have_F, DAISY_E_STATE, "daisy_formfactors_row_digest: no form factors yet");
    DZ_REQUIRE(nrows >= 0 && row0 >= ctx->row0 && row0 + nrows <= ctx->row1, DAISY_E_INVALID, "daisy_formfactors_row_digest: rows outside this context's range");
    if (nrows == 0) return DAISY_OK;
    DZ_CUDA(cudaSetDevice(ctx->device));
    uint32_t *dx = nullptr;
    unsigned long long *dw = nullptr;
    DZ_CUDA(cudaMalloc(&dx, sizeof(uint32_t) * (size_t)nrows));
    cudaError_t e = cudaMalloc(&dw, sizeof(unsigned long long) * (size_t)nrows);
    if (e == cudaSuccess) {
        k_row_digest<<<(nrows + 7) / 8, 256, 0, ctx->stream>>>(ctx->d_F + (size_t)(row0 - ctx->row0) * ctx->ldF, ctx->ldF, ctx->N, nrows, dx, dw);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(xor_out, dx, sizeof(uint32_t) * (size_t)nrows, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(wsum_out, dw, sizeof(uint64_t) * (size_t)nrows, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(dx); cudaFree(dw);
    if (e != cudaSuccess) { daisy_set_error("daisy_formfactors_row_digest: %s", cudaGetErrorString(e)); return DAISY_E_CUDA; }
    return DAISY_OK;
}

extern "C" int daisy_ctx_face_count(daisy_ctx *ctx) { return ctx ? ctx->nfaces : -1; }
extern "C" int64_t daisy_formfactors_pairs_fallback(daisy_ctx *ctx) { return ctx ? ctx->pairs_heavy : -1; }

extern "C" int daisy_formfactors_stats(daisy_ctx *ctx, int64_t *pairs_traced, int64_t *pairs_owned, int64_t *rays, double *lbvh_ms, double *ff_ms) {
    DZ_REQUIRE(ctx, DAISY_E_INVALID, "daisy_formfactors_stats: null context");
    if (pairs_traced) *pairs_traced = ctx->pairs_traced;
    if (pairs_owned) *pairs_owned = ctx->pairs_owned;
    if (rays) *rays = ctx->pairs_traced * (int64_t)ctx->S;
    if (lbvh_ms) *lbvh_ms = ctx->lbvh_ms;
    if (ff_ms) *ff_ms = ctx->ff_ms;
    return DAISY_OK;
}
