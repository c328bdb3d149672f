// group.cu -- several GPUs of one box behind ONE host process (the reference is a single process: main.cpp:97-113).
//
// daisy_group owns one daisy_ctx per device (row block g of the matrix on device g, mesh and LBVH replicated), enables peer
// access between all of them and wires the contexts' peer pointers directly -- no CUDA IPC, no torch.distributed, no NCCL:
//   * form factors: every upper-triangle tile is traced by exactly one device (hash of the tile coordinates) and stored,
//     tile and mirrored tile, into the owners' matrices over NVLink; the devices build concurrently (one host thread each);
//   * gather: daisy_group_solver drives one daisy_solver per device through the fused exchange (the pass kernel stores its
//     new residual block into every device's next buffer and raises flags; the next pass waits for them on the device), so
//     a pass is one asynchronous kernel launch per device and nothing else.
// The multi-process entry points (daisy_ctx_set_partition + *_ipc_handle/_set_peers) remain for hosts that run one process per GPU.
#include "daisy_common.cuh"
#include <string.h>
#include <string>
#include <thread>
#include <vector>

struct daisy_group {
    int ndev = 0;
    int N = 0;
    std::vector<int> devices;
    std::vector<daisy_ctx *> ctx;
};

struct daisy_group_solver {
    daisy_group *g = nullptr;
    uint64_t mesh_version = 0; // device 0's mesh_version at create (daisy_group_replace_mesh moves every device's)
    int K = 0;
    std::vector<daisy_solver *> s;
};

extern "C" void daisy_group_destroy(daisy_group *g) {
    if (!g) return;
    for (daisy_ctx *c : g->ctx) daisy_ctx_destroy(c);
    delete g;
}

extern "C" int daisy_group_create(const float *vertices, int nv, const float *normals, int nn, const int32_t *tri_idx, int ntri,
                                  const int *device_ids, int ndev, daisy_group **out) {
    DZ_REQUIRE(out, DAISY_E_INVALID, "daisy_group_create: null out pointer");
    *out = nullptr;
    DZ_REQUIRE(ndev >= 1 && ndev <= 16, DAISY_E_INVALID, "daisy_group_create: 1 to 16 devices");
    int have = 0;
    DZ_CUDA(cudaGetDeviceCount(&have));
    daisy_group *g = new daisy_group();
    g->ndev = ndev; g->N = ntri;
    for (int i = 0; i < ndev; i++) {
        const int d = device_ids ? device_ids[i] : i;
        if (d < 0 || d >= have) { delete g; daisy_set_error("daisy_group_create: no such CUDA device %d", d); return DAISY_E_INVALID; }
        for (int j = 0; j < i; j++)
            if (g->devices[(size_t)j] == d) { delete g; daisy_set_error("daisy_group_create: device %d listed twice", d); return DAISY_E_INVALID; }
        g->devices.push_back(d);
    }
    // every device must be able to store into every other one's memory
    for (int i = 0; i < ndev; i++)
        for (int j = 0; j < ndev; j++) {
            if (i == j) continue;
            int can = 0;
            cudaError_t e = cudaDeviceCanAccessPeer(&can, g->devices[(size_t)i], g->devices[(size_t)j]);
            if (e != cudaSuccess || !can) {
                delete g;
                daisy_set_error("daisy_group_create: device %d cannot access device %d's memory", i, j);
                return DAISY_E_STATE;
            }
            cudaSetDevice(g->devices[(size_t)i]);
            e = cudaDeviceEnablePeerAccess(g->devices[(size_t)j], 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if (e != cudaSuccess) { delete g; daisy_set_error("daisy_group_create: cudaDeviceEnablePeerAccess -> %s", cudaGetErrorString(e)); return DAISY_E_CUDA; }
        }
    // contexts (mesh upload, LBVH, plane records) are built concurrently: one host thread per device
    g->ctx.assign((size_t)ndev, nullptr);
    std::vector<int> rcs((size_t)ndev, DAISY_OK);
    std::vector<std::string> errs((size_t)ndev);
    std::vector<std::thread> th;
    for (int i = 0; i < ndev; i++)
        th.emplace_back([&, i]() {
            int rc = daisy_ctx_create(vertices, nv, normals, nn, tri_idx, ntri, g->devices[(size_t)i], &g->ctx[(size_t)i]);
            if (!rc && ndev > 1) rc = daisy_ctx_set_partition(g->ctx[(size_t)i], i, ndev);
            rcs[(size_t)i] = rc;
            if (rc) errs[(size_t)i] = daisy_last_error();
        });
    for (auto &t : th) t.join();
    for (int i = 0; i < ndev; i++)
        if (rcs[(size_t)i]) {
            daisy_set_error("daisy_group_create: device %d: %s", g->devices[(size_t)i], errs[(size_t)i].c_str());
            const int rc = rcs[(size_t)i];
            daisy_group_destroy(g);
            return rc;
        }
    *out = g;
    return DAISY_OK;
}

extern "C" int daisy_group_size(daisy_group *g) { return g ? g->ndev : DAISY_E_INVALID; }
extern "C" daisy_ctx *daisy_group_ctx(daisy_group *g, int i) { return (g && i >= 0 && i < g->ndev) ? g->ctx[(size_t)i] : nullptr; }

extern "C" int daisy_group_set_samples(daisy_group *g, const float *uv, int S) {
    DZ_REQUIRE(g, DAISY_E_INVALID, "daisy_group_set_samples: null group");
    for (daisy_ctx *c : g->ctx) {
        int rc = daisy_ctx_set_samples(c, uv, S);
        if (rc) return rc;
    }
    return DAISY_OK;
}

// run fn(i) for every device on its own host thread; first failure wins
template <typename Fn>
static int for_each_device(daisy_group *g, const char *what, Fn fn) {
    std::vector<int> rcs((size_t)g->ndev, DAISY_OK);
    std::vector<std::string> errs((size_t)g->ndev);
    std::vector<std::thread> th;
    for (int i = 0; i < g->ndev; i++)
        th.emplace_back([&, i]() {
            rcs[(size_t)i] = fn(i);
            if (rcs[(size_t)i]) errs[(size_t)i] = daisy_last_error();
        });
    for (auto &t : th) t.join();
    for (int i = 0; i < g->ndev; i++)
        if (rcs[(size_t)i]) { daisy_set_error("%s: device %d: %s", what, g->devices[(size_t)i], errs[(size_t)i].c_str()); return rcs[(size_t)i]; }
    return DAISY_OK;
}

extern "C" int daisy_group_formfactors_build(daisy_group *g, int variant) {
    DZ_REQUIRE(g, DAISY_E_INVALID, "daisy_group_formfactors_build: null group");
    nvtxRangePushA("daisy_group_formfactors_build");
    int rc = DAISY_OK;
    if (g->ndev > 1 && !g->ctx[0]->peers_set) {
        rc = for_each_device(g, "daisy_group_formfactors_build (alloc)", [&](int i) { return daisy_formfactors_alloc(g->ctx[(size_t)i]); });
        if (!rc) {
            float *F[16] = { nullptr };
            for (int i = 0; i < g->ndev; i++) F[i] = g->ctx[(size_t)i]->d_F;
            for (int i = 0; i < g->ndev && !rc; i++) rc = dz_ctx_set_peer_pointers(g->ctx[(size_t)i], F, g->ndev);
        }
    }
    // every device traces its share of the tiles and stores into the owners' rows; the join below is the barrier after
    // which every row block is complete
    if (!rc) rc = for_each_device(g, "daisy_group_formfactors_build", [&](int i) { return daisy_formfactors_build(g->ctx[(size_t)i], variant); });
    // the devices also wrote into each other's rows: every matrix changed after the join, whichever device finished last
    for (int i = 0; i < g->ndev; i++) g->ctx[(size_t)i]->F_version++;
    nvtxRangePop();
    return rc;
}

extern "C" int daisy_group_update_geometry(daisy_group *g, const float *vertices, int nv, const float *normals, int nn) {
    DZ_REQUIRE(g, DAISY_E_INVALID, "daisy_group_update_geometry: null group");
    return for_each_device(g, "daisy_group_update_geometry", [&](int i) { return daisy_ctx_update_geometry(g->ctx[(size_t)i], vertices, nv, normals, nn); });
}

extern "C" int daisy_group_formfactors_update(daisy_group *g, int variant) {
    DZ_REQUIRE(g, DAISY_E_INVALID, "daisy_group_formfactors_update: null group");
    nvtxRangePushA("daisy_group_formfactors_update");
    // the peers are wired by the first build; an update without one traces everything and needs them just the same
    int rc = DAISY_OK;
    if (g->ndev > 1 && !g->ctx[0]->peers_set) {
        rc = for_each_device(g, "daisy_group_formfactors_update (alloc)", [&](int i) { return daisy_formfactors_alloc(g->ctx[(size_t)i]); });
        if (!rc) {
            float *F[16] = { nullptr };
            for (int i = 0; i < g->ndev; i++) F[i] = g->ctx[(size_t)i]->d_F;
            for (int i = 0; i < g->ndev && !rc; i++) rc = dz_ctx_set_peer_pointers(g->ctx[(size_t)i], F, g->ndev);
        }
    }
    if (!rc) rc = for_each_device(g, "daisy_group_formfactors_update", [&](int i) { return daisy_formfactors_update(g->ctx[(size_t)i], variant); });
    // devices store into each other's rows: every matrix may have changed after the join
    for (int i = 0; i < g->ndev; i++) g->ctx[(size_t)i]->F_version++;
    nvtxRangePop();
    return rc;
}

extern "C" int daisy_group_replace_mesh(daisy_group *g, const float *vertices, int nv, const float *normals, int nn, const int32_t *tri_idx, int ntri,
                                        const int32_t *previous) {
    DZ_REQUIRE(g, DAISY_E_INVALID, "daisy_group_replace_mesh: null group");
    DzRange range_("daisy_group_replace_mesh");
    const int rc = dz_replace_mesh(g->ctx.data(), g->ndev, vertices, nv, normals, nn, tri_idx, ntri, previous, "daisy_group_replace_mesh");
    g->N = g->ctx[0]->N;
    return rc;
}

static int owner_of(daisy_group *g, int row) {
    const int n = g->ctx[0]->rows_per_rank;
    int o = n > 0 ? row / n : 0;
    return o < g->ndev ? o : g->ndev - 1;
}

extern "C" int daisy_group_formfactors_read_rows(daisy_group *g, int row0, int nrows, float *out) {
    DZ_REQUIRE(g && (nrows == 0 || out), DAISY_E_INVALID, "daisy_group_formfactors_read_rows: null argument");
    DZ_REQUIRE(row0 >= 0 && nrows >= 0 && row0 + nrows <= g->N, DAISY_E_INVALID, "daisy_group_formfactors_read_rows: rows out of range");
    int r = row0;
    while (r < row0 + nrows) {
        daisy_ctx *c = g->ctx[(size_t)owner_of(g, r)];
        const int r1 = (row0 + nrows < c->row1) ? row0 + nrows : c->row1;
        int rc = daisy_formfactors_read_rows(c, r, r1 - r, out + (size_t)(r - row0) * g->N);
        if (rc) return rc;
        r = r1;
    }
    return DAISY_OK;
}

extern "C" int daisy_group_formfactors_write_rows(daisy_group *g, int row0, int nrows, const float *in) {
    DZ_REQUIRE(g && (nrows == 0 || in), DAISY_E_INVALID, "daisy_group_formfactors_write_rows: null argument");
    DZ_REQUIRE(row0 >= 0 && nrows >= 0 && row0 + nrows <= g->N, DAISY_E_INVALID, "daisy_group_formfactors_write_rows: rows out of range");
    int r = row0;
    while (r < row0 + nrows) {
        daisy_ctx *c = g->ctx[(size_t)owner_of(g, r)];
        const int r1 = (row0 + nrows < c->row1) ? row0 + nrows : c->row1;
        int rc = daisy_formfactors_write_rows(c, r, r1 - r, in + (size_t)(r - row0) * g->N);
        if (rc) return rc;
        r = r1;
    }
    // a device that owns no rows (blocks of rows_per_rank rounded up to 256 can leave the last ones empty) receives none of
    // them above, yet its solver still needs a matrix (the one-row allocation its tensor map points at) and have_F: a write
    // of zero rows gives it both
    for (daisy_ctx *c : g->ctx)
        if (c->row1 == c->row0) {
            int rc = daisy_formfactors_write_rows(c, c->row0, 0, nullptr);
            if (rc) return rc;
        }
    return DAISY_OK;
}

// refill an Eigen::SparseMatrix<float> from the row blocks of all devices (column-major CSC, sorted inner indices, as
// setFromTriplets leaves it, OptixPrimeFunctionality.cpp:25).  values == NULL: nnz only.
extern "C" int daisy_group_formfactors_to_csc(daisy_group *g, int64_t *nnz, float *values, int32_t *inner_idx, int32_t *outer_ptr) {
    DZ_REQUIRE(g && nnz, DAISY_E_INVALID, "daisy_group_formfactors_to_csc: null argument");
    if (g->ndev == 1) return daisy_formfactors_to_csc(g->ctx[0], nnz, values, inner_idx, outer_ptr);
    if (!dz_csc_host()) {
        for (daisy_ctx *c : g->ctx) DZ_REQUIRE(c->have_F, DAISY_E_STATE, "daisy_group_formfactors_to_csc: no form factors yet");
        return dz_csc_export(g->ctx.data(), g->ndev, nnz, values, inner_idx, outer_ptr, "daisy_group_formfactors_to_csc");
    }
    // DAISY_CSC_HOST=1: host-side conversion of dense row read-backs
    const int N = g->N;
    std::vector<int64_t> colcount((size_t)N + 1, 0);
    int chunk = (int)((128u << 20) / (4.0 * (N ? N : 1)));
    if (chunk < 1) chunk = 1;
    if (chunk > N) chunk = N > 0 ? N : 1;
    std::vector<float> rows((size_t)chunk * (N ? N : 1));
    for (int r = 0; r < N; r += chunk) {
        const int nr = (N - r) < chunk ? (N - r) : chunk;
        int rc = daisy_group_formfactors_read_rows(g, r, nr, rows.data());
        if (rc) return rc;
        for (int i = 0; i < nr; i++)
            for (int c = 0; c < N; c++)
                if (rows[(size_t)i * N + c] != 0.0f) colcount[(size_t)c + 1]++;
    }
    for (int c = 0; c < N; c++) colcount[(size_t)c + 1] += colcount[(size_t)c];
    *nnz = colcount[(size_t)N];
    if (!values) return DAISY_OK;
    DZ_REQUIRE(inner_idx && outer_ptr, DAISY_E_INVALID, "daisy_group_formfactors_to_csc: null index arrays");
    DZ_REQUIRE(*nnz <= 0x7fffffffLL, DAISY_E_INVALID, "daisy_group_formfactors_to_csc: more non-zeros than Eigen's int index can hold");
    for (int c = 0; c <= N; c++) outer_ptr[c] = (int32_t)colcount[(size_t)c];
    std::vector<int64_t> fill(colcount.begin(), colcount.end() - 1);
    for (int r = 0; r < N; r += chunk) {
        const int nr = (N - r) < chunk ? (N - r) : chunk;
        int rc = daisy_group_formfactors_read_rows(g, r, nr, rows.data());
        if (rc) return rc;
        for (int i = 0; i < nr; i++)
            for (int c = 0; c < N; c++) {
                const float v = rows[(size_t)i * N + c];
                if (v != 0.0f) { const int64_t q = fill[(size_t)c]++; values[q] = v; inner_idx[q] = r + i; }
            }
    }
    return DAISY_OK;
}

// every device validates the whole matrix before any device stores; each keeps the rows of its block, and a device that owns
// no rows gets have_F as daisy_group_formfactors_write_rows gives it
extern "C" int daisy_group_formfactors_write_csc(daisy_group *g, int64_t nnz, const float *values, const int32_t *inner_idx, const int32_t *outer_ptr) {
    DZ_REQUIRE(g, DAISY_E_INVALID, "daisy_group_formfactors_write_csc: null group");
    DzRange range_("daisy_group_formfactors_write_csc");
    return dz_csc_import(g->ctx.data(), g->ndev, nnz, values, inner_idx, outer_ptr, "daisy_group_formfactors_write_csc");
}

extern "C" int daisy_group_formfactors_stats(daisy_group *g, int64_t *pairs, int64_t *rays, double *lbvh_ms, double *ff_ms) {
    DZ_REQUIRE(g, DAISY_E_INVALID, "daisy_group_formfactors_stats: null group");
    int64_t p = 0, r = 0;
    double a = 0.0, b = 0.0;
    for (daisy_ctx *c : g->ctx) {
        p += c->pairs_owned; r += c->pairs_owned * (int64_t)c->S;
        a = c->lbvh_ms > a ? c->lbvh_ms : a; b = c->ff_ms > b ? c->ff_ms : b;
    }
    if (pairs) *pairs = p;
    if (rays) *rays = r;
    if (lbvh_ms) *lbvh_ms = a;
    if (ff_ms) *ff_ms = b;
    return DAISY_OK;
}

// ---- gather ------------------------------------------------------------------------------------------------------------
extern "C" void daisy_group_solver_destroy(daisy_group_solver *gs) {
    if (!gs) return;
    // no device may still be storing into another one's buffers when they are freed
    for (size_t i = 0; i < gs->s.size(); i++)
        if (gs->s[i]) { cudaSetDevice(gs->g->devices[i]); cudaDeviceSynchronize(); }
    for (daisy_solver *s : gs->s) daisy_solver_destroy(s);
    delete gs;
}

extern "C" int daisy_group_solver_create(daisy_group *g, int K, const float *E, const float *M, int nmat, const int32_t *mat_idx,
                                         daisy_group_solver **out) {
    DZ_REQUIRE(g && out, DAISY_E_INVALID, "daisy_group_solver_create: null argument");
    *out = nullptr;
    daisy_group_solver *gs = new daisy_group_solver();
    gs->g = g; gs->K = K; gs->mesh_version = g->ctx[0]->mesh_version;
    gs->s.assign((size_t)g->ndev, nullptr);
    int rc = for_each_device(g, "daisy_group_solver_create", [&](int i) { return daisy_solver_create(g->ctx[(size_t)i], K, E, M, nmat, mat_idx, &gs->s[(size_t)i]); });
    if (!rc && g->ndev > 1) {
        float *r0[16] = { nullptr }, *r1[16] = { nullptr };
        unsigned long long *fl[16] = { nullptr };
        for (int i = 0; i < g->ndev; i++) dz_solver_get_buffers(gs->s[(size_t)i], &r0[i], &r1[i], &fl[i]);
        for (int i = 0; i < g->ndev && !rc; i++) rc = dz_solver_set_peer_pointers(gs->s[(size_t)i], r0, r1, fl, g->ndev);
    }
    if (rc) { daisy_group_solver_destroy(gs); return rc; }
    *out = gs;
    return DAISY_OK;
}

extern "C" int daisy_group_solver_reset(daisy_group_solver *gs) {
    DZ_REQUIRE(gs, DAISY_E_INVALID, "daisy_group_solver_reset: null solver");
    for (daisy_solver *s : gs->s) {
        int rc = daisy_solver_reset(s);
        if (rc) return rc;
    }
    return DAISY_OK;
}

// one pass on every device: one asynchronous launch each (the devices synchronise among themselves through the exchange
// flags).  band_sums != NULL additionally waits for the pass and returns the per-band totals of the new residual.
extern "C" int daisy_group_solver_step(daisy_group_solver *gs, double *band_sums) {
    DZ_REQUIRE(gs, DAISY_E_INVALID, "daisy_group_solver_step: null solver");
    if (gs->g->ndev == 1) return daisy_solver_step(gs->s[0], band_sums);
    for (daisy_solver *s : gs->s) {
        int rc = daisy_solver_step_fused(s, nullptr);
        if (rc) return rc;
    }
    if (band_sums) return daisy_solver_band_sums(gs->s[0], band_sums); // every device holds every block's sums; device 0 answers
    return DAISY_OK;
}

extern "C" int daisy_group_solver_band_sums(daisy_group_solver *gs, double *band_sums) {
    DZ_REQUIRE(gs && band_sums, DAISY_E_INVALID, "daisy_group_solver_band_sums: null argument");
    return daisy_solver_band_sums(gs->s[0], band_sums);
}

extern "C" int daisy_group_solver_numpasses(daisy_group_solver *gs) { return gs ? daisy_solver_numpasses(gs->s[0]) : DAISY_E_INVALID; }

extern "C" int daisy_group_solver_converge(daisy_group_solver *gs, double threshold, int per_band, int max_passes, int *passes_out) {
    DZ_REQUIRE(gs, DAISY_E_INVALID, "daisy_group_solver_converge: null solver");
    if (gs->g->ndev == 1) return daisy_solver_converge(gs->s[0], threshold, per_band, max_passes, passes_out);
    nvtxRangePushA("daisy_group_solver_converge");
    std::vector<double> sums((size_t)gs->K);
    int rc = daisy_solver_band_sums(gs->s[0], sums.data());
    int done = 0;
    auto unconverged = [&]() {
        double tot = 0.0;
        for (int k = 0; k < gs->K; k++) {
            if (per_band && sums[(size_t)k] > threshold) return true;
            tot += sums[(size_t)k];
        }
        return !per_band && tot > threshold;
    };
    while (!rc && unconverged() && (max_passes <= 0 || done < max_passes)) {
        rc = daisy_group_solver_step(gs, sums.data());
        done++;
    }
    if (passes_out) *passes_out = daisy_solver_numpasses(gs->s[0]);
    nvtxRangePop();
    return rc;
}

// the device converge over every device: the first pass decided from device 0's sums, every device's batches issued from this
// thread; every device takes the same decisions from the same band sums, which the pass counts confirm
extern "C" int daisy_group_solver_converge_device(daisy_group_solver *gs, double threshold, int per_band, int max_passes, int *passes_out) {
    DZ_REQUIRE(gs, DAISY_E_INVALID, "daisy_group_solver_converge_device: null solver");
    if (gs->g->ndev == 1) return daisy_solver_converge_device(gs->s[0], threshold, per_band, max_passes, passes_out);
    nvtxRangePushA("daisy_group_solver_converge_device");
    int rc = dz_converge_device(gs->s.data(), gs->g->ndev, threshold, per_band, max_passes);
    if (!rc && passes_out) *passes_out = daisy_solver_numpasses(gs->s[0]);
    nvtxRangePop();
    return rc;
}

// daisy_solver_restart over every device: B0 (K x N whole scene, or NULL for the current B) is split into the devices' rows, the
// restart pass is launched on every device before any device waits, and device 0 answers the band sums when they are asked for
extern "C" int daisy_group_solver_restart(daisy_group_solver *gs, const float *B0) {
    DZ_REQUIRE(gs, DAISY_E_INVALID, "daisy_group_solver_restart: null solver");
    DZ_REQUIRE(gs->mesh_version == gs->g->ctx[0]->mesh_version, DAISY_E_STATE,
               "daisy_group_solver_restart: the group's mesh was replaced after this solver was created; create a new solver");
    daisy_group *g = gs->g;
    if (g->ndev == 1) return daisy_solver_restart(gs->s[0], B0);
    nvtxRangePushA("daisy_group_solver_restart");
    const int N = g->N, K = gs->K;
    std::vector<float> b;
    int rc = DAISY_OK;
    for (int i = 0; i < g->ndev && !rc; i++) {
        daisy_ctx *c = g->ctx[(size_t)i];
        const int nloc = c->row1 - c->row0;
        if (B0) {
            b.assign((size_t)K * (nloc > 0 ? nloc : 1), 0.f);
            for (int k = 0; k < K && nloc > 0; k++) memcpy(b.data() + (size_t)k * nloc, B0 + (size_t)k * N + c->row0, sizeof(float) * (size_t)nloc);
        }
        rc = dz_solver_restart_launch(gs->s[(size_t)i], B0 ? b.data() : nullptr);
    }
    nvtxRangePop();
    return rc;
}

extern "C" int daisy_group_solver_set_emission(daisy_group_solver *gs, const float *E) {
    DZ_REQUIRE(gs, DAISY_E_INVALID, "daisy_group_solver_set_emission: null solver");
    for (daisy_solver *s : gs->s) { // the same input on every device: the first one refuses invalid input before any changes
        int rc = daisy_solver_set_emission(s, E);
        if (rc) return rc;
    }
    return DAISY_OK;
}

extern "C" int daisy_group_solver_set_materials(daisy_group_solver *gs, const float *M, int nmat, const int32_t *mat_idx) {
    DZ_REQUIRE(gs, DAISY_E_INVALID, "daisy_group_solver_set_materials: null solver");
    for (daisy_solver *s : gs->s) {
        int rc = daisy_solver_set_materials(s, M, nmat, mat_idx);
        if (rc) return rc;
    }
    return DAISY_OK;
}

// lightningvalues and residualvector of the whole scene, K x N band-major, assembled from the devices' row blocks
extern "C" int daisy_group_solver_read(daisy_group_solver *gs, float *B, float *residual) {
    DZ_REQUIRE(gs, DAISY_E_INVALID, "daisy_group_solver_read: null solver");
    DZ_REQUIRE(gs->mesh_version == gs->g->ctx[0]->mesh_version, DAISY_E_STATE,
               "daisy_group_solver_read: the group's mesh was replaced after this solver was created; create a new solver");
    daisy_group *g = gs->g;
    const int N = g->N, K = gs->K;
    std::vector<float> b, r;
    for (int i = 0; i < g->ndev; i++) {
        daisy_ctx *c = g->ctx[(size_t)i];
        const int nloc = c->row1 - c->row0;
        if (nloc <= 0) continue;
        b.resize((size_t)K * nloc); r.resize((size_t)K * nloc);
        int rc = daisy_solver_read(gs->s[(size_t)i], B ? b.data() : nullptr, residual ? r.data() : nullptr);
        if (rc) return rc;
        for (int k = 0; k < K; k++) {
            if (B) memcpy(B + (size_t)k * N + c->row0, b.data() + (size_t)k * nloc, sizeof(float) * (size_t)nloc);
            if (residual) memcpy(residual + (size_t)k * N + c->row0, r.data() + (size_t)k * nloc, sizeof(float) * (size_t)nloc);
        }
    }
    return DAISY_OK;
}

// B and residual of the whole scene from host, K x N band-major: every device receives only its own rows; the residual
// slices reach the other devices over NVLink (daisy_solver_write_slices)
extern "C" int daisy_group_solver_write(daisy_group_solver *gs, const float *B, const float *residual) {
    DZ_REQUIRE(gs && B && residual, DAISY_E_INVALID, "daisy_group_solver_write: null argument");
    DZ_REQUIRE(gs->mesh_version == gs->g->ctx[0]->mesh_version, DAISY_E_STATE,
               "daisy_group_solver_write: the group's mesh was replaced after this solver was created; create a new solver");
    daisy_group *g = gs->g;
    const int N = g->N, K = gs->K;
    if (g->ndev == 1) return daisy_solver_write(gs->s[0], B, residual);
    std::vector<float> b, r;
    for (int i = 0; i < g->ndev; i++) {
        daisy_ctx *c = g->ctx[(size_t)i];
        const int nloc = c->row1 - c->row0;
        b.assign((size_t)K * (nloc > 0 ? nloc : 1), 0.f); r.assign((size_t)K * (nloc > 0 ? nloc : 1), 0.f);
        for (int k = 0; k < K && nloc > 0; k++) {
            memcpy(b.data() + (size_t)k * nloc, B + (size_t)k * N + c->row0, sizeof(float) * (size_t)nloc);
            memcpy(r.data() + (size_t)k * nloc, residual + (size_t)k * N + c->row0, sizeof(float) * (size_t)nloc);
        }
        int rc = daisy_solver_write_slices(gs->s[(size_t)i], b.data(), r.data());
        if (rc) return rc;
    }
    return DAISY_OK;
}
