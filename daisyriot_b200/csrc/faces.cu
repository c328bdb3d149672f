// faces.cu -- planar face grids: a per-plane acceleration structure for the visibility rays of the form-factor kernel.
//
// Scenes of the kind the reference renders (OptixPrimeFunctionality.cpp:169-242 traces rays between the patches of walls,
// boxes, table tops) consist of large planar faces cut into many small triangles.  A visibility ray that crosses such a face
// well inside it is blocked by SOME triangle of the face, and one that crosses the face's plane away from every triangle of
// the face cannot touch any of them -- which triangle does not matter for "closest hit is the destination patch".  So each
// face (a plane id with at least FACE_MIN_TRIS triangles, at most DAISY_MAX_FACES of them, largest first) gets a uniform 2-D
// grid in its plane.  Per cell:
//   empty    no triangle of the face comes within `delta` of the cell;
//   covered  the cell grown by `delta` lies inside the union of the face's triangles;
//   mixed    anything else (the cell touches the outline of the face, a T-junction, a degenerate triangle ...);
// and every non-empty cell lists the triangles that come within `delta` of it.  The kernel intersects a ray with the plane
// (one division), looks the cell up and only runs the watertight test on the listed triangles of mixed cells or when the
// crossing lies within a margin of the ray's two end points (formfactor.cu, pair_mask_warp).
//
// Why "covered" is exact and not an approximation: the watertight test (daisy_common.cuh) evaluates, with exact signs (the
// float products are monotone, exact zeros are recomputed in double), whether the ray's origin lies in the closed 2-D
// triangle spanned by the sheared, rounded vertices; a vertex is rounded the same way in every triangle that uses it.  The
// sheared image of the face is therefore a planar triangulation with slightly moved vertices, its outline still winds once
// around every point that is more than the rounding error inside it, so at least one of its triangles contains the origin --
// the test accepts it, with t within rounding of the plane crossing.  The outline of the union consists of edges that are NOT
// shared by exactly two triangles of the face lying on opposite sides (shared = bit-identical end points); cells that come
// within `delta` of such an edge are mixed.  `delta` (2.5e-4 x scene extent) exceeds every rounding term involved by more than
// an order of magnitude for rays that meet the plane at |cos| >= FACE_COS_MIN (the kernel checks that per patch pair).
// Everything here runs once per scene on the host in double precision.
#include "daisy_common.cuh"
#include <math.h>
#include <string.h>
#include <algorithm>
#include <atomic>
#include <thread>
#include <unordered_map>
#include <utility>
#include <vector>

#define FACE_MIN_TRIS 32
#define FACE_DELTA 2.5e-4     // x scene extent
#define FACE_CELLS_PER_TRI 16.0
#define FACE_MAX_CELLS (1 << 22)
#define FACE_PLANE_TOL 1.2e-6 // x scene extent: members farther than this from the refitted plane => no grid for the face

bool dz_fit_plane(const double *pts_xyz, size_t npts, double n_out[3], double c_out[3]); // api.cu

namespace {
struct P2 { double a, b; };
struct D3 { double x, y, z; };
inline D3 sub3(D3 a, D3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
inline double dot3(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline D3 cross3(D3 a, D3 b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }
inline double cross2(P2 o, P2 p, P2 q) { return (p.a - o.a) * (q.b - o.b) - (p.b - o.b) * (q.a - o.a); }

struct EdgeKey {
    uint32_t w[6];
    bool operator==(const EdgeKey &o) const { return memcmp(w, o.w, sizeof(w)) == 0; }
};
struct EdgeHash {
    size_t operator()(const EdgeKey &k) const {
        uint64_t h = 0xcbf29ce484222325ull;
        for (int i = 0; i < 6; i++) { h ^= k.w[i]; h *= 0x100000001b3ull; }
        return (size_t)h;
    }
};
struct EdgeInfo { int count; int pos, neg; P2 p, q; };
} // namespace

void dz_free_faces(daisy_ctx *c) {
    cudaFree(c->d_faces); cudaFree(c->d_face_cells); cudaFree(c->d_face_lists);
    c->d_faces = nullptr; c->d_face_cells = nullptr; c->d_face_lists = nullptr; c->nfaces = 0;
}

// Chooses the faces, renumbers `pid` so that face f carries plane id f + 1 (all other groups keep distinct ids above the
// faces'), builds the grids and uploads them.  A face whose grid cannot be built is simply left out (its triangles stay
// ordinary candidates): nothing here can make a result wrong, only slower.
// One face: plane, frame, grid, cell lists and cell classes.  Self-contained (reads the mesh, writes its own vectors), so the
// faces of a scene are built by parallel host threads.  ok = false: no grid for this face (its triangles stay ordinary
// candidates -- never wrong, only slower).
struct FaceBuild {
    bool ok = false;
    DzFace F;
    std::vector<int> cells; // per cell: -1, or (offset into `lists` << 1) | covered, offsets local to this face
    std::vector<int> lists;
};

static void build_one_face(double ext, float pad, const float *vertices, const int32_t *tri_idx, const std::vector<int> &mem, FaceBuild &out) {
    const double delta = FACE_DELTA * ext;
    auto vert = [&](int t, int k) -> D3 {
        const float *p = vertices + 3 * (size_t)tri_idx[6 * (size_t)t + k];
        return { (double)p[0], (double)p[1], (double)p[2] };
    };
    // plane: exact for axis-aligned faces, least squares otherwise
    D3 n = { 0, 0, 0 }, c0 = { 0, 0, 0 };
    {
        int axis = -1;
        for (int d = 0; d < 3 && axis < 0; d++) {
            const float v0 = vertices[3 * (size_t)tri_idx[6 * (size_t)mem[0]] + d];
            bool same = true;
            for (size_t i = 0; i < mem.size() && same; i++)
                for (int k = 0; k < 3 && same; k++) same = vertices[3 * (size_t)tri_idx[6 * (size_t)mem[i] + k] + d] == v0;
            if (same) axis = d;
        }
        if (axis >= 0) {
            n = { axis == 0 ? 1.0 : 0.0, axis == 1 ? 1.0 : 0.0, axis == 2 ? 1.0 : 0.0 };
            c0 = vert(mem[0], 0);
        } else {
            std::vector<double> pts;
            pts.reserve(mem.size() * 9);
            for (int t : mem)
                for (int k = 0; k < 3; k++) { const D3 p = vert(t, k); pts.push_back(p.x); pts.push_back(p.y); pts.push_back(p.z); }
            double nn[3], cc[3];
            if (!dz_fit_plane(pts.data(), pts.size() / 3, nn, cc)) return;
            n = { nn[0], nn[1], nn[2] }; c0 = { cc[0], cc[1], cc[2] };
        }
    }
    double off = 0.0;
    for (int t : mem)
        for (int k = 0; k < 3; k++) off = fmax(off, fabs(dot3(n, sub3(vert(t, k), c0))));
    if (off > FACE_PLANE_TOL * ext) return;
    // in-plane frame: the edge direction of the largest member that gives the smallest bounding rectangle
    int seed = mem[0];
    double seed_a = -1.0, area_sum = 0.0;
    for (int t : mem) {
        const D3 cr = cross3(sub3(vert(t, 1), vert(t, 0)), sub3(vert(t, 2), vert(t, 0)));
        const double a = 0.5 * sqrt(dot3(cr, cr));
        area_sum += a;
        if (a > seed_a) { seed_a = a; seed = t; }
    }
    if (!(seed_a > 0.0)) return;
    D3 ex = { 0, 0, 0 }, ey = { 0, 0, 0 };
    double best = 1e300, amin = 0, bmin = 0, amax = 0, bmax = 0;
    for (int e = 0; e < 3; e++) {
        D3 d = sub3(vert(seed, (e + 1) % 3), vert(seed, e));
        const double dn = dot3(d, n);
        d = { d.x - dn * n.x, d.y - dn * n.y, d.z - dn * n.z };
        const double l = sqrt(dot3(d, d));
        if (!(l > 0.0)) continue;
        const D3 x = { d.x / l, d.y / l, d.z / l }, y = cross3(n, x);
        double a0 = 1e300, a1 = -1e300, b0 = 1e300, b1 = -1e300;
        for (int t : mem)
            for (int k = 0; k < 3; k++) {
                const D3 p = sub3(vert(t, k), c0);
                const double a = dot3(p, x), b = dot3(p, y);
                a0 = fmin(a0, a); a1 = fmax(a1, a); b0 = fmin(b0, b); b1 = fmax(b1, b);
            }
        const double area = (a1 - a0) * (b1 - b0);
        if (area < best) { best = area; ex = x; ey = y; amin = a0; amax = a1; bmin = b0; bmax = b1; }
    }
    if (!(best < 1e300)) return;
    // cell size: FACE_CELLS_PER_TRI cells per average triangle, never below 2 delta, grid bounded
    double cells_per_tri = FACE_CELLS_PER_TRI;
    { const char *e = getenv("DAISY_FACE_CELLS_PER_TRI"); if (e && atof(e) >= 1.0) cells_per_tri = atof(e); } // A/B switch
    double cs = sqrt(area_sum / ((double)mem.size() * cells_per_tri));
    cs = fmax(cs, 2.0 * delta);
    int nx = 0, ny = 0;
    for (int it = 0; it < 64; it++) {
        nx = (int)floor((amax - amin) / cs) + 3; ny = (int)floor((bmax - bmin) / cs) + 3;
        if ((double)nx * (double)ny <= (double)FACE_MAX_CELLS) break;
        cs *= 1.25;
    }
    if ((double)nx * (double)ny > (double)FACE_MAX_CELLS) return;
    const double A0 = amin - cs, B0 = bmin - cs; // one cell of apron (>= 2 delta) on every side
    auto to2 = [&](D3 p) -> P2 { const D3 q = sub3(p, c0); return { dot3(q, ex) - A0, dot3(q, ey) - B0 }; };
    const size_t ncell = (size_t)nx * ny;
    std::vector<char> boundary(ncell, 0);
    // cells whose rectangle, grown by delta, may meet the box [lo, hi]
    auto cell_range = [&](double lo_a, double lo_b, double hi_a, double hi_b, int &i0, int &i1, int &j0, int &j1) {
        i0 = std::max(0, (int)floor((lo_a - delta) / cs)); i1 = std::min(nx - 1, (int)floor((hi_a + delta) / cs));
        j0 = std::max(0, (int)floor((lo_b - delta) / cs)); j1 = std::min(ny - 1, (int)floor((hi_b + delta) / cs));
    };
    // an oriented line f(a, b) = na a + nb b + c against a rectangle: the extremes of f over the rectangle in closed form
    struct Line { double na, nb, c, lo, hi; };
    auto line_misses = [](const Line &l, double a0, double b0, double a1, double b1) -> bool {
        const double mx = l.na * (l.na >= 0 ? a1 : a0) + l.nb * (l.nb >= 0 ? b1 : b0) + l.c;
        const double mn = l.na * (l.na >= 0 ? a0 : a1) + l.nb * (l.nb >= 0 ? b0 : b1) + l.c;
        return mx < l.lo || mn > l.hi;
    };
    // (1) triangles per cell: one rasterisation pass into (cell, triangle) records, then a counting sort by cell
    std::vector<std::pair<int, int>> rec;
    rec.reserve(mem.size() * 24);
    std::unordered_map<EdgeKey, EdgeInfo, EdgeHash> edges;
    edges.reserve(mem.size() * 2);
    for (int t : mem) {
        const P2 T[3] = { to2(vert(t, 0)), to2(vert(t, 1)), to2(vert(t, 2)) };
        Line ln[3];
        for (int e = 0; e < 3; e++) {
            const P2 p = T[e], q = T[(e + 1) % 3], r = T[(e + 2) % 3];
            Line &l = ln[e];
            l.na = -(q.b - p.b); l.nb = q.a - p.a; l.c = -(l.na * p.a + l.nb * p.b);
            const double side = l.na * r.a + l.nb * r.b + l.c, tol = 1e-12 * (fabs(l.na) + fabs(l.nb)) * (fabs(p.a) + fabs(p.b) + cs);
            l.lo = fmin(0.0, side) - tol; l.hi = fmax(0.0, side) + tol; // the triangle spans [0, side] along this normal
        }
        int i0, i1, j0, j1;
        cell_range(fmin(T[0].a, fmin(T[1].a, T[2].a)), fmin(T[0].b, fmin(T[1].b, T[2].b)), fmax(T[0].a, fmax(T[1].a, T[2].a)),
                   fmax(T[0].b, fmax(T[1].b, T[2].b)), i0, i1, j0, j1);
        for (int j = j0; j <= j1; j++)
            for (int i = i0; i <= i1; i++) {
                const double a0 = i * cs - delta, b0 = j * cs - delta, a1 = (i + 1) * cs + delta, b1 = (j + 1) * cs + delta;
                // separating axes of rectangle and triangle: the rectangle's own (the cell range above) and the three edge normals
                if (line_misses(ln[0], a0, b0, a1, b1) || line_misses(ln[1], a0, b0, a1, b1) || line_misses(ln[2], a0, b0, a1, b1)) continue;
                rec.emplace_back(j * nx + i, t);
            }
        for (int e = 0; e < 3; e++) {
            const int v0 = tri_idx[6 * (size_t)t + e], v1 = tri_idx[6 * (size_t)t + (e + 1) % 3];
            uint32_t k0[3], k1[3];
            for (int d = 0; d < 3; d++) {
                float f0 = vertices[3 * (size_t)v0 + d] + 0.0f, f1 = vertices[3 * (size_t)v1 + d] + 0.0f; // -0 -> +0
                memcpy(&k0[d], &f0, 4); memcpy(&k1[d], &f1, 4);
            }
            const bool swap = memcmp(k0, k1, sizeof(k0)) > 0;
            EdgeKey key;
            memcpy(key.w, swap ? k1 : k0, 12); memcpy(key.w + 3, swap ? k0 : k1, 12);
            const P2 p = swap ? T[(e + 1) % 3] : T[e], q = swap ? T[e] : T[(e + 1) % 3], r = T[(e + 2) % 3];
            const double sd = cross2(p, q, r);
            const double scale = (fabs(q.a - p.a) + fabs(q.b - p.b)) * (fabs(r.a - p.a) + fabs(r.b - p.b));
            auto it = edges.find(key);
            if (it == edges.end()) it = edges.emplace(key, EdgeInfo{ 0, 0, 0, p, q }).first;
            it->second.count++;
            if (sd > 1e-9 * scale) it->second.pos++;
            else if (sd < -1e-9 * scale) it->second.neg++;
        }
    }
    std::vector<int> count(ncell, 0), start(ncell, -1);
    for (const auto &r : rec) count[(size_t)r.first]++;
    out.lists.clear();
    size_t total = 0;
    for (size_t q = 0; q < ncell; q++)
        if (count[q]) { start[q] = (int)total; total += 1 + (size_t)count[q]; }
    out.lists.assign(total, -1);
    for (size_t q = 0; q < ncell; q++)
        if (count[q]) { out.lists[(size_t)start[q]] = count[q]; count[q] = 0; }
    for (const auto &r : rec) { const size_t q = (size_t)r.first; out.lists[(size_t)start[q] + 1 + (size_t)count[q]++] = r.second; } // members ascend: so do the lists
    // (2) outline: every edge that is not shared by exactly two members on opposite sides
    for (const auto &kv : edges) {
        const EdgeInfo &e = kv.second;
        if (e.count == 2 && e.pos == 1 && e.neg == 1) continue;
        Line l;
        l.na = -(e.q.b - e.p.b); l.nb = e.q.a - e.p.a; l.c = -(l.na * e.p.a + l.nb * e.p.b);
        const double tol = 1e-12 * (fabs(l.na) + fabs(l.nb)) * (fabs(e.p.a) + fabs(e.p.b) + cs);
        l.lo = -tol; l.hi = tol;
        int i0, i1, j0, j1;
        cell_range(fmin(e.p.a, e.q.a), fmin(e.p.b, e.q.b), fmax(e.p.a, e.q.a), fmax(e.p.b, e.q.b), i0, i1, j0, j1);
        for (int j = j0; j <= j1; j++)
            for (int i = i0; i <= i1; i++)
                if (!line_misses(l, i * cs - delta, j * cs - delta, (i + 1) * cs + delta, (j + 1) * cs + delta)) boundary[(size_t)j * nx + i] = 1;
    }
    out.cells.resize(ncell);
    for (size_t q = 0; q < ncell; q++) out.cells[q] = count[q] ? ((start[q] << 1) | (boundary[q] ? 0 : 1)) : -1;
    DzFace &F = out.F;
    F.pl = make_float4((float)n.x, (float)n.y, (float)n.z, (float)dot3(n, c0));
    // cell coordinate a = (dot(X - c0, ex) - A0) / cs = dot(X, ex / cs) - (dot(c0, ex) + A0) / cs
    F.ex = make_float4((float)(ex.x / cs), (float)(ex.y / cs), (float)(ex.z / cs), (float)(-(dot3(c0, ex) + A0) / cs));
    F.ey = make_float4((float)(ey.x / cs), (float)(ey.y / cs), (float)(ey.z / cs), (float)(-(dot3(c0, ey) + B0) / cs));
    F.g = make_int4(nx, ny, 0, (int)mem.size());
    float blo[3] = { INFINITY, INFINITY, INFINITY }, bhi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int t : mem)
        for (int k = 0; k < 3; k++)
            for (int dd = 0; dd < 3; dd++) {
                const float v = vertices[3 * (size_t)tri_idx[6 * (size_t)t + k] + dd];
                blo[dd] = fminf(blo[dd], v); bhi[dd] = fmaxf(bhi[dd], v);
            }
    F.blo = make_float4(blo[0] - pad, blo[1] - pad, blo[2] - pad, 0.f);
    F.bhi = make_float4(bhi[0] + pad, bhi[1] + pad, bhi[2] + pad, 0.f);
    out.ok = true;
}

// Chooses the faces, builds their grids on parallel host threads, renumbers `pid` so that face f carries plane id f + 1 (all
// other groups keep distinct ids above the faces') and returns the concatenated tables.
static int build_face_tables(float ext_f, float pad, const float *vertices, const int32_t *tri_idx, int ntri, std::vector<int> &pid,
                             std::vector<DzFace> &faces, std::vector<int> &cells, std::vector<int> &lists) {
    faces.clear(); cells.clear(); lists.clear();
    if (ntri == 0 || !(ext_f > 0.f)) return DAISY_OK;
    { const char *e = getenv("DAISY_FF_FACES"); if (e && e[0] == '0') return DAISY_OK; }
    int maxid = 0;
    for (int t = 0; t < ntri; t++) maxid = std::max(maxid, pid[(size_t)t]);
    std::vector<std::vector<int>> members((size_t)maxid + 1);
    for (int t = 0; t < ntri; t++)
        if (pid[(size_t)t] > 0) members[(size_t)pid[(size_t)t]].push_back(t);
    std::vector<int> order;
    for (int g = 1; g <= maxid; g++)
        if ((int)members[(size_t)g].size() >= FACE_MIN_TRIS) order.push_back(g);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return members[(size_t)a].size() > members[(size_t)b].size(); });
    // candidates: a few more than DAISY_MAX_FACES so that faces whose grid cannot be built do not cost a slot
    if (order.size() > (size_t)DAISY_MAX_FACES + 16) order.resize((size_t)DAISY_MAX_FACES + 16);
    std::vector<FaceBuild> built(order.size());
    {
        std::atomic<size_t> next(0);
        auto worker = [&]() {
            for (size_t i = next.fetch_add(1); i < order.size(); i = next.fetch_add(1)) {
                try {
                    build_one_face((double)ext_f, pad, vertices, tri_idx, members[(size_t)order[i]], built[i]);
                } catch (...) { // out of host memory for one face's tables: the face simply gets no grid
                    built[i] = FaceBuild();
                }
            }
        };
        unsigned nthr = std::thread::hardware_concurrency();
        if (nthr == 0) nthr = 1;
        nthr = (unsigned)std::min<size_t>(std::min<size_t>(nthr, 16), order.size());
        std::vector<std::thread> pool;
        for (unsigned i = 1; i < nthr; i++) pool.emplace_back(worker);
        worker();
        for (auto &th : pool) th.join();
    }
    std::vector<int> face_group;
    for (size_t i = 0; i < order.size() && (int)faces.size() < DAISY_MAX_FACES; i++) {
        FaceBuild &b = built[i];
        if (!b.ok) continue;
        if ((double)cells.size() + (double)b.cells.size() > 2.0e8 || (double)lists.size() + (double)b.lists.size() > (double)0x3fffffff) continue;
        const int cell_base = (int)cells.size(), list_base = (int)lists.size();
        for (int c : b.cells) cells.push_back(c < 0 ? -1 : (((c >> 1) + list_base) << 1) | (c & 1));
        lists.insert(lists.end(), b.lists.begin(), b.lists.end());
        b.F.g.z = cell_base;
        faces.push_back(b.F);
        face_group.push_back(order[i]);
        std::vector<int>().swap(b.cells); std::vector<int>().swap(b.lists);
    }
    // renumber the plane ids: face f -> f + 1, every other group -> a distinct id above the faces
    {
        std::vector<int> newid((size_t)maxid + 1, 0);
        for (size_t f = 0; f < face_group.size(); f++) newid[(size_t)face_group[f]] = (int)f + 1;
        int next = (int)face_group.size() + 1;
        for (int g = 1; g <= maxid; g++)
            if (!newid[(size_t)g] && !members[(size_t)g].empty()) newid[(size_t)g] = next++;
        for (int t = 0; t < ntri; t++) pid[(size_t)t] = newid[(size_t)pid[(size_t)t]];
    }
    return DAISY_OK;
}

int dz_build_faces(daisy_ctx *c, const float *vertices, const int32_t *tri_idx, int ntri, std::vector<int> &pid) {
    c->nfaces = 0;
    std::vector<DzFace> faces;
    std::vector<int> cells, lists;
    const int rc = build_face_tables(c->ext, c->pad, vertices, tri_idx, ntri, pid, faces, cells, lists);
    if (rc) return rc;
    if (faces.empty()) return DAISY_OK;
    DZ_CUDA(cudaMalloc(&c->d_faces, sizeof(DzFace) * faces.size()));
    DZ_CUDA(cudaMalloc(&c->d_face_cells, sizeof(int) * cells.size()));
    DZ_CUDA(cudaMalloc(&c->d_face_lists, sizeof(int) * (lists.empty() ? 1 : lists.size())));
    DZ_CUDA(cudaMemcpyAsync(c->d_faces, faces.data(), sizeof(DzFace) * faces.size(), cudaMemcpyHostToDevice, c->stream));
    DZ_CUDA(cudaMemcpyAsync(c->d_face_cells, cells.data(), sizeof(int) * cells.size(), cudaMemcpyHostToDevice, c->stream));
    if (!lists.empty()) DZ_CUDA(cudaMemcpyAsync(c->d_face_lists, lists.data(), sizeof(int) * lists.size(), cudaMemcpyHostToDevice, c->stream));
    DZ_CUDA(cudaStreamSynchronize(c->stream)); // the tables are pageable host memory
    c->nfaces = (int)faces.size();
    c->face_cells = (int64_t)cells.size();
    c->face_list_ints = (int64_t)lists.size();
    return DAISY_OK;
}

// Host-only view of the grids for tests and diagnostics: per face the numbers of triangles, cells, empty / covered / mixed
// cells and list entries (6 int64 each), plus the renumbered plane ids.  No GPU involved.
int dz_face_grid_stats(float ext, const float *vertices, const int32_t *tri_idx, int ntri, std::vector<int> &pid, int max_faces, int64_t *out6, int *nfaces_out) {
    std::vector<DzFace> faces;
    std::vector<int> cells, lists;
    const int rc = build_face_tables(ext, 1e-4f * ext, vertices, tri_idx, ntri, pid, faces, cells, lists);
    if (rc) return rc;
    *nfaces_out = (int)faces.size();
    for (size_t f = 0; f < faces.size() && (int)f < max_faces; f++) {
        const int4 g = faces[f].g;
        int64_t e = 0, cv = 0, mx = 0, le = 0;
        for (int q = 0; q < g.x * g.y; q++) {
            const int c = cells[(size_t)g.z + q];
            if (c < 0) e++;
            else { if (c & 1) cv++; else mx++; le += lists[(size_t)(c >> 1)]; }
        }
        int64_t *o = out6 + 6 * f;
        o[0] = g.w; o[1] = (int64_t)g.x * g.y; o[2] = e; o[3] = cv; o[4] = mx; o[5] = le;
    }
    return DAISY_OK;
}

// Host-only dump of one face's grid for the CPU property tests: frame16 = plane (n, d), ex (xyz / cell size, offset), ey, nx, ny,
// triangle count, 0; state[q] = 0 empty / 1 covered / 2 mixed, count[q] = listed triangles (both nx * ny long, may be NULL).
int dz_face_grid_dump(float ext, const float *vertices, const int32_t *tri_idx, int ntri, std::vector<int> &pid, int face, float *frame16, signed char *state,
                      int32_t *count, int64_t cap) {
    std::vector<DzFace> faces;
    std::vector<int> cells, lists;
    const int rc = build_face_tables(ext, 1e-4f * ext, vertices, tri_idx, ntri, pid, faces, cells, lists);
    if (rc) return rc;
    if (face < 0 || face >= (int)faces.size()) { daisy_set_error("daisy_face_grid_dump: no such face"); return DAISY_E_INVALID; }
    const DzFace &F = faces[(size_t)face];
    const float fr[16] = { F.pl.x, F.pl.y, F.pl.z, F.pl.w, F.ex.x, F.ex.y, F.ex.z, F.ex.w, F.ey.x, F.ey.y, F.ey.z, F.ey.w, (float)F.g.x, (float)F.g.y, (float)F.g.w, 0.f };
    memcpy(frame16, fr, sizeof(fr));
    const int64_t n = (int64_t)F.g.x * F.g.y;
    if ((state || count) && cap < n) { daisy_set_error("daisy_face_grid_dump: buffers too small"); return DAISY_E_INVALID; }
    for (int64_t q = 0; q < n && (state || count); q++) {
        const int c = cells[(size_t)F.g.z + (size_t)q];
        if (state) state[q] = c < 0 ? 0 : ((c & 1) ? 1 : 2);
        if (count) count[q] = c < 0 ? 0 : lists[(size_t)(c >> 1)];
    }
    return DAISY_OK;
}
