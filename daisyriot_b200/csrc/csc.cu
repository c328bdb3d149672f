// csc.cu -- the matrix cache on the device: F handed back as a compressed column-major matrix (Eigen::SparseMatrix<float>,
// daisy_formfactors_to_csc / daisy_group_formfactors_to_csc) and such a matrix loaded into F (daisy_formfactors_write_csc /
// daisy_group_formfactors_write_csc).  No dense row crosses PCIe: only the counts per column (N ints per device), the column
// starts and the CSC arrays themselves do.
//
// Export, per device (rows [row0, row1) of the matrix, all rows for a single context):
//   k_csc_count  one streaming read of the rows: cnt[rb][c] = entries of column c in 64-row block rb (<= 64, uint8) and
//                colcnt[c] = entries of column c (integer atomics, order-free);
//   host         outer[c] (int64) from the column totals of all devices; start[g][c] = outer[c] + entries of column c on the
//                devices before g (their rows come first in every column);
//   per chunk of columns [c0, c1), whose CSC segment [outer[c0], outer[c1]) is contiguous in the output:
//     k_csc_base   base[rb][c] = running sum of cnt down the row blocks (one thread per column);
//     k_csc_fill   one thread per (row block, column) walks its 64 rows in ascending order and writes value and row at
//                  start[g][c] + base[rb][c] into the first device's staging buffer (peer stores for the other devices);
//     one cudaMemcpyAsync per array moves the segment into the caller's arrays.  Two staging buffers: the fill of chunk i+1 is
//     enqueued before the copy of chunk i.
// An entry is listed exactly when its bits other than the sign are not all zero (F[r][c] != 0.0f, independent of
// flush-to-zero): +-0 are not listed, NaN, +-inf and denormals are; values are copied bit for bit.  Padding columns
// [N, ldF) are never listed.
//
// Import: the host checks outer (O(N)); values and rows go up in column chunks and k_csc_check (a warp per column) raises a
// flag on a row outside [0, N) or not strictly above its predecessor.  Only when every chunk of every device passed are the
// context's rows of F (padding columns included) zeroed and the entries of its rows scattered by k_csc_scatter (a warp per
// column).  The chunks stay resident when they fit in half the free device memory; otherwise the validation uploads the rows
// alone and the scatter uploads values and rows again (daisy_formfactors_csc_uploads reports which ran).
#include "daisy_common.cuh"
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#define CSC_RB 64 // rows per count block: a block's count of one column fits a uint8

bool dz_csc_host() { // DAISY_CSC_HOST=1: the host conversion through dense row read-backs (A/B switch, reference of the tests)
    const char *e = getenv("DAISY_CSC_HOST");
    return e && e[0] == '1';
}

// bound of the staging buffers (both export buffers together, the import buffer, and a resident import): 256 MB, or
// DAISY_CSC_STAGE_BYTES (small values run the chunked paths at small sizes)
static size_t stage_bytes(bool *set = nullptr) {
    const char *e = getenv("DAISY_CSC_STAGE_BYTES");
    const long long v = e ? atoll(e) : 0;
    if (set) *set = v > 0;
    return v > 0 ? (size_t)std::max(v, 64LL) : ((size_t)256 << 20);
}

// ---- kernels -----------------------------------------------------------------------------------------------------------
// one thread = 4 consecutive columns of one 64-row block (a float4 per row; ldF is a multiple of 32, so a float4 that starts
// below N lies inside the row)
__global__ void __launch_bounds__(256) k_csc_count(const float *__restrict__ F, int64_t ldF, int nloc, int N, int nrb, unsigned char *__restrict__ cnt,
                                                   int *__restrict__ colcnt) {
    const int rb = blockIdx.y;
    DZ_ASSERT(rb < nrb);
    const int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (c >= N) return;
    DZ_ASSERT(c + 3 < ldF);
    const int r0 = rb * CSC_RB, r1 = min(nloc, r0 + CSC_RB);
    int n0 = 0, n1 = 0, n2 = 0, n3 = 0;
#pragma unroll 4
    for (int r = r0; r < r1; r++) {
        const float4 v = ldg_stream(F + (size_t)r * ldF + c);
        n0 += (__float_as_uint(v.x) & 0x7fffffffu) != 0u;
        n1 += (__float_as_uint(v.y) & 0x7fffffffu) != 0u;
        n2 += (__float_as_uint(v.z) & 0x7fffffffu) != 0u;
        n3 += (__float_as_uint(v.w) & 0x7fffffffu) != 0u;
    }
    const int n[4] = { n0, n1, n2, n3 };
    for (int k = 0; k < 4 && c + k < N; k++) {
        DZ_ASSERT(c + k < N && (size_t)rb * N + c + k < (size_t)nrb * N);
        cnt[(size_t)rb * N + c + k] = (unsigned char)n[k];
        if (n[k]) atomicAdd(colcnt + c + k, n[k]);
    }
}

// base[rb * nc + j] = entries of column c0 + j in the row blocks above rb
__global__ void k_csc_base(const unsigned char *__restrict__ cnt, int N, int nrb, int c0, int nc, int *__restrict__ base, int64_t base_cap) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nc) return;
    DZ_ASSERT(c0 + j < N && (int64_t)nrb * nc <= base_cap);
    int s = 0;
#pragma unroll 8
    for (int rb = 0; rb < nrb; rb++) {
        base[(size_t)rb * nc + j] = s;
        s += cnt[(size_t)rb * N + c0 + j];
    }
}

// the entries of column c0 + j in row block rb, rows ascending, at start[c] - seg0 + base of the chunk's staging segment
__global__ void k_csc_fill(const float *__restrict__ F, int64_t ldF, int nloc, int row0, int c0, int nc, const int64_t *__restrict__ start,
                           int64_t seg0, int64_t seglen, const int *__restrict__ base, int64_t base_cap, int N, uint32_t *__restrict__ val,
                           int *__restrict__ row) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, rb = blockIdx.y;
    if (j >= nc) return;
    const int c = c0 + j;
    DZ_ASSERT(c < N && c < ldF && (int64_t)rb * nc + j < base_cap);
    int64_t p = start[c] - seg0 + base[(size_t)rb * nc + j];
    const int r1 = min(nloc, (rb + 1) * CSC_RB);
    for (int r = rb * CSC_RB; r < r1; r++) {
        const uint32_t b = __float_as_uint(__ldcs(F + (size_t)r * ldF + c));
        if (b & 0x7fffffffu) {
            DZ_ASSERT(p >= 0 && p < seglen);
            val[p] = b;
            row[p] = row0 + r;
            p++;
        }
    }
}

// warp per column of [c0, c0 + nc): every row in [0, N) and strictly above the one before it.  Raises *bad, writes nothing else.
__global__ void k_csc_check(const int *__restrict__ outer, int c0, int nc, int64_t seg0, int64_t seglen, const int *__restrict__ row, int N, int *bad) {
    const int w = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= nc) return; // whole warps
    const int c = c0 + w;
    const int64_t s = outer[c] - seg0, e = outer[c + 1] - seg0;
    bool ok = true;
    for (int64_t i = s + lane; i < e; i += 32) {
        DZ_ASSERT(i >= 0 && i < seglen);
        const int r = row[i];
        ok &= r >= 0 && r < N && (i == s || row[i - 1] < r);
    }
    if (__any_sync(0xffffffffu, !ok) && lane == 0) atomicOr(bad, 1);
}

// warp per column: the entries whose row lies in [row0, row1) go into F, bit for bit
__global__ void k_csc_scatter(const int *__restrict__ outer, int c0, int nc, int64_t seg0, int64_t seglen, const uint32_t *__restrict__ val,
                              const int *__restrict__ row, int row0, int row1, uint32_t *__restrict__ F, int64_t ldF, int64_t fcap) {
    const int w = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= nc) return;
    const int c = c0 + w;
    DZ_ASSERT(c < ldF);
    const int64_t s = outer[c] - seg0, e = outer[c + 1] - seg0;
    for (int64_t i = s + lane; i < e; i += 32) {
        DZ_ASSERT(i >= 0 && i < seglen);
        const int r = row[i];
        if (r >= row0 && r < row1) {
            DZ_ASSERT((int64_t)(r - row0) * ldF + c < fcap);
            F[(size_t)(r - row0) * ldF + c] = val[i];
        }
    }
}

// ---- host --------------------------------------------------------------------------------------------------------------
namespace {
struct Chunk { int c0, c1; int64_t e0, e1; }; // columns [c0, c1), entries [e0, e1)

// consecutive column ranges of at most max_entries entries (a column with more gets a chunk of its own) and max_cols columns
template <typename Outer>
std::vector<Chunk> make_chunks(const Outer &outer, int N, int64_t max_entries, int max_cols) {
    std::vector<Chunk> ch;
    int c = 0;
    do {
        Chunk k;
        k.c0 = c; k.e0 = (int64_t)outer[c];
        int c1 = c + 1 <= N ? c + 1 : N;
        while (c1 < N && c1 - c < max_cols && (int64_t)outer[c1 + 1] - k.e0 <= max_entries) c1++;
        k.c1 = c1; k.e1 = (int64_t)outer[c1];
        ch.push_back(k);
        c = c1;
    } while (c < N);
    return ch;
}

// device allocations of one call, freed on every return path
struct DevMem {
    std::vector<std::pair<int, void *>> p;
    cudaError_t alloc(int dev, void **out, size_t bytes) {
        cudaSetDevice(dev);
        cudaError_t e = cudaMalloc(out, bytes ? bytes : 16);
        if (e == cudaSuccess) p.push_back({ dev, *out });
        else { cudaGetLastError(); *out = nullptr; }
        return e;
    }
    ~DevMem() {
        for (auto &q : p) { cudaSetDevice(q.first); cudaFree(q.second); }
    }
};
} // namespace

#define CSC_CUDA(call, what)                                                                                         \
    do {                                                                                                             \
        cudaError_t e_ = (call);                                                                                     \
        if (e_ != cudaSuccess) { daisy_set_error("%s: %s -> %s", what, #call, cudaGetErrorString(e_)); return DAISY_E_CUDA; } \
    } while (0)

// F of the contexts ctx[0..n) -- rows [row0, row1) each, ascending and together all N rows -- as CSC.  values == NULL: nnz only.
int dz_csc_export(daisy_ctx *const *ctx, int n, int64_t *nnz, float *values, int32_t *inner_idx, int32_t *outer_ptr, const char *what) {
    const int N = ctx[0]->N;
    DevMem mem;
    std::vector<unsigned char *> cnt((size_t)n, nullptr);
    std::vector<int *> colcnt((size_t)n, nullptr);
    std::vector<int> nrb((size_t)n, 0);
    // 1. counts, every device at once
    for (int g = 0; g < n; g++) {
        daisy_ctx *c = ctx[g];
        const int nloc = c->row1 - c->row0;
        nrb[(size_t)g] = (nloc + CSC_RB - 1) / CSC_RB;
        CSC_CUDA(mem.alloc(c->device, (void **)&cnt[(size_t)g], (size_t)nrb[(size_t)g] * N), what);
        CSC_CUDA(mem.alloc(c->device, (void **)&colcnt[(size_t)g], sizeof(int) * (size_t)N), what);
        CSC_CUDA(cudaMemsetAsync(colcnt[(size_t)g], 0, sizeof(int) * (size_t)N, c->stream), what);
        if (nrb[(size_t)g] > 0 && N > 0) {
            k_csc_count<<<dim3((unsigned)((N + 1023) / 1024), (unsigned)nrb[(size_t)g]), 256, 0, c->stream>>>(c->d_F, c->ldF, nloc, N, nrb[(size_t)g], cnt[(size_t)g],
                                                                                                           colcnt[(size_t)g]);
            CSC_CUDA(cudaGetLastError(), what);
        }
    }
    std::vector<std::vector<int>> h_cnt((size_t)n, std::vector<int>((size_t)N));
    for (int g = 0; g < n; g++) {
        CSC_CUDA(cudaSetDevice(ctx[g]->device), what);
        if (N) CSC_CUDA(cudaMemcpyAsync(h_cnt[(size_t)g].data(), colcnt[(size_t)g], sizeof(int) * (size_t)N, cudaMemcpyDeviceToHost, ctx[g]->stream), what);
        CSC_CUDA(cudaStreamSynchronize(ctx[g]->stream), what);
    }
    // 2. column starts
    std::vector<int64_t> outer((size_t)N + 1, 0);
    for (int c = 0; c < N; c++) {
        int64_t t = 0;
        for (int g = 0; g < n; g++) t += h_cnt[(size_t)g][(size_t)c];
        outer[(size_t)c + 1] = outer[(size_t)c] + t;
    }
    *nnz = outer[(size_t)N];
    if (!values) return DAISY_OK;
    if (!inner_idx || !outer_ptr) { daisy_set_error("%s: null index arrays", what); return DAISY_E_INVALID; }
    if (*nnz > 0x7fffffffLL) { daisy_set_error("%s: more non-zeros than Eigen's int index can hold", what); return DAISY_E_INVALID; }
    for (int c = 0; c <= N; c++) outer_ptr[c] = (int32_t)outer[(size_t)c];
    if (*nnz == 0) return DAISY_OK;
    std::vector<int64_t *> start((size_t)n, nullptr);
    {
        std::vector<int64_t> s(outer.begin(), outer.end() - 1);
        for (int g = 0; g < n; g++) {
            CSC_CUDA(mem.alloc(ctx[g]->device, (void **)&start[(size_t)g], sizeof(int64_t) * (size_t)N), what);
            CSC_CUDA(cudaSetDevice(ctx[g]->device), what);
            CSC_CUDA(cudaMemcpyAsync(start[(size_t)g], s.data(), sizeof(int64_t) * (size_t)N, cudaMemcpyHostToDevice, ctx[g]->stream), what);
            CSC_CUDA(cudaStreamSynchronize(ctx[g]->stream), what); // `s` is pageable host memory, advanced below
            for (int c = 0; c < N; c++) s[(size_t)c] += h_cnt[(size_t)g][(size_t)c];
        }
    }
    // 3. column chunks through two staging buffers on the first device
    const size_t stage = stage_bytes();
    const int max_nrb = std::max(1, *std::max_element(nrb.begin(), nrb.end()));
    const int max_cols = (int)std::max<size_t>(32, stage / 4 / (sizeof(int) * (size_t)max_nrb)); // base array <= stage / 4
    const std::vector<Chunk> ch = make_chunks(outer, N, std::max<int64_t>(1, (int64_t)(stage / 16)), max_cols);
    int64_t buf_entries = 1;
    int buf_cols = 1;
    for (const Chunk &k : ch) { buf_entries = std::max(buf_entries, k.e1 - k.e0); buf_cols = std::max(buf_cols, k.c1 - k.c0); }
    const int dev0 = ctx[0]->device;
    uint32_t *sval[2] = { nullptr, nullptr };
    int *srow[2] = { nullptr, nullptr };
    for (int b = 0; b < 2; b++) {
        CSC_CUDA(mem.alloc(dev0, (void **)&sval[b], sizeof(uint32_t) * (size_t)buf_entries), what);
        CSC_CUDA(mem.alloc(dev0, (void **)&srow[b], sizeof(int) * (size_t)buf_entries), what);
    }
    std::vector<int *> base((size_t)n, nullptr);
    for (int g = 0; g < n; g++) CSC_CUDA(mem.alloc(ctx[g]->device, (void **)&base[(size_t)g], sizeof(int) * (size_t)nrb[(size_t)g] * buf_cols), what);
    // events and the copy stream (non-blocking: it must not serialise with the legacy default stream the kernels may run on)
    struct Ev {
        std::vector<std::pair<int, cudaEvent_t>> ev;
        cudaStream_t cs = nullptr;
        int cs_dev = 0;
        ~Ev() {
            for (auto &e : ev) { cudaSetDevice(e.first); cudaEventDestroy(e.second); }
            if (cs) { cudaSetDevice(cs_dev); cudaStreamDestroy(cs); }
        }
    } ev;
    auto make_event = [&](int dev, cudaEvent_t *out) {
        cudaSetDevice(dev);
        cudaError_t e = cudaEventCreateWithFlags(out, cudaEventDisableTiming);
        if (e == cudaSuccess) ev.ev.push_back({ dev, *out });
        return e;
    };
    std::vector<cudaEvent_t> filled((size_t)2 * n);
    cudaEvent_t copied[2];
    for (int b = 0; b < 2; b++) {
        for (int g = 0; g < n; g++) CSC_CUDA(make_event(ctx[g]->device, &filled[(size_t)b * n + g]), what);
        CSC_CUDA(make_event(dev0, &copied[b]), what);
    }
    CSC_CUDA(cudaSetDevice(dev0), what);
    CSC_CUDA(cudaStreamCreateWithFlags(&ev.cs, cudaStreamNonBlocking), what);
    ev.cs_dev = dev0;
    auto fill = [&](size_t i) -> int {
        const Chunk &k = ch[i];
        const int b = (int)(i & 1), nc = k.c1 - k.c0;
        for (int g = 0; g < n; g++) {
            daisy_ctx *c = ctx[g];
            CSC_CUDA(cudaSetDevice(c->device), what);
            if (i >= 2) CSC_CUDA(cudaStreamWaitEvent(c->stream, copied[b], 0), what); // the copy of chunk i - 2 has left buffer b
            if (nrb[(size_t)g] > 0 && k.e1 > k.e0) {
                const int64_t base_cap = (int64_t)nrb[(size_t)g] * buf_cols;
                k_csc_base<<<(nc + 255) / 256, 256, 0, c->stream>>>(cnt[(size_t)g], N, nrb[(size_t)g], k.c0, nc, base[(size_t)g], base_cap);
                k_csc_fill<<<dim3((unsigned)((nc + 127) / 128), (unsigned)nrb[(size_t)g]), 128, 0, c->stream>>>(
                    c->d_F, c->ldF, c->row1 - c->row0, c->row0, k.c0, nc, start[(size_t)g], k.e0, k.e1 - k.e0, base[(size_t)g], base_cap, N, sval[b], srow[b]);
                CSC_CUDA(cudaGetLastError(), what);
            }
            CSC_CUDA(cudaEventRecord(filled[(size_t)b * n + g], c->stream), what);
        }
        return DAISY_OK;
    };
    int rc = fill(0);
    for (size_t i = 0; i < ch.size() && !rc; i++) {
        if (i + 1 < ch.size()) rc = fill(i + 1); // enqueued before the copy of chunk i: a copy into pageable memory returns when done
        if (rc) break;
        const Chunk &k = ch[i];
        const int b = (int)(i & 1);
        CSC_CUDA(cudaSetDevice(dev0), what);
        for (int g = 0; g < n; g++) CSC_CUDA(cudaStreamWaitEvent(ev.cs, filled[(size_t)b * n + g], 0), what);
        if (k.e1 > k.e0) {
            CSC_CUDA(cudaMemcpyAsync(values + k.e0, sval[b], sizeof(float) * (size_t)(k.e1 - k.e0), cudaMemcpyDeviceToHost, ev.cs), what);
            CSC_CUDA(cudaMemcpyAsync(inner_idx + k.e0, srow[b], sizeof(int) * (size_t)(k.e1 - k.e0), cudaMemcpyDeviceToHost, ev.cs), what);
        }
        CSC_CUDA(cudaEventRecord(copied[b], ev.cs), what);
    }
    if (rc) return rc;
    CSC_CUDA(cudaStreamSynchronize(ev.cs), what);
    for (int g = 0; g < n; g++) { CSC_CUDA(cudaSetDevice(ctx[g]->device), what); CSC_CUDA(cudaStreamSynchronize(ctx[g]->stream), what); }
    return DAISY_OK;
}

// run fn(g) for every context, on its own host thread when there are several; the first failure's code and message win
template <typename Fn>
static int each_ctx(daisy_ctx *const *ctx, int n, const char *what, Fn fn) {
    if (n == 1) return fn(0);
    std::vector<int> rcs((size_t)n, DAISY_OK);
    std::vector<std::string> errs((size_t)n);
    std::vector<std::thread> th;
    for (int g = 0; g < n; g++)
        th.emplace_back([&, g]() {
            rcs[(size_t)g] = fn(g);
            if (rcs[(size_t)g]) errs[(size_t)g] = daisy_last_error();
        });
    for (auto &t : th) t.join();
    for (int g = 0; g < n; g++)
        if (rcs[(size_t)g]) { daisy_set_error("%s: device %d: %s", what, ctx[g]->device, errs[(size_t)g].c_str()); return rcs[(size_t)g]; }
    return DAISY_OK;
}

// load the CSC matrix into the contexts ctx[0..n) (each keeps the rows of its range).  All of them validate before any stores.
int dz_csc_import(daisy_ctx *const *ctx, int n, int64_t nnz, const float *values, const int32_t *inner_idx, const int32_t *outer_ptr, const char *what) {
    const int N = ctx[0]->N;
    if (!outer_ptr || nnz < 0 || (nnz > 0 && (!values || !inner_idx))) { daisy_set_error("%s: null array or negative nnz", what); return DAISY_E_INVALID; }
    if (nnz > 0x7fffffffLL) { daisy_set_error("%s: more non-zeros than an int index can hold", what); return DAISY_E_INVALID; }
    if (outer_ptr[0] != 0 || (int64_t)outer_ptr[N] != nnz) { daisy_set_error("%s: outer_ptr must start at 0 and end at nnz", what); return DAISY_E_INVALID; }
    for (int c = 0; c < N; c++)
        if (outer_ptr[c + 1] < outer_ptr[c]) { daisy_set_error("%s: outer_ptr decreases at column %d", what, c); return DAISY_E_INVALID; }
    bool limited = false;
    const size_t stage = stage_bytes(&limited);
    const std::vector<Chunk> ch = make_chunks(outer_ptr, N, std::max<int64_t>(1, (int64_t)(stage / 8)), 0x7fffffff);
    int64_t chunk_entries = 1;
    for (const Chunk &k : ch) chunk_entries = std::max(chunk_entries, k.e1 - k.e0);
    struct Dev {
        DevMem mem;
        uint32_t *val = nullptr;
        int *row = nullptr, *outer = nullptr, *bad = nullptr;
        bool resident = false;
    };
    std::vector<Dev> dev((size_t)n);
    // upload chunk k into the device's staging (at its CSC position when resident, at 0 otherwise); the values only when the
    // scatter will read them from there
    auto upload = [&](daisy_ctx *c, Dev &d, const Chunk &k, int64_t *seg0, bool with_values) -> int {
        *seg0 = d.resident ? 0 : k.e0;
        const int64_t at = k.e0 - *seg0;
        if (k.e1 > k.e0) {
            if (with_values) CSC_CUDA(cudaMemcpyAsync(d.val + at, values + k.e0, sizeof(float) * (size_t)(k.e1 - k.e0), cudaMemcpyHostToDevice, c->stream), what);
            CSC_CUDA(cudaMemcpyAsync(d.row + at, inner_idx + k.e0, sizeof(int) * (size_t)(k.e1 - k.e0), cudaMemcpyHostToDevice, c->stream), what);
        }
        return DAISY_OK;
    };
    // 1. validation on every device (each checks the copy it will scatter from)
    int rc = each_ctx(ctx, n, what, [&](int g) -> int {
        daisy_ctx *c = ctx[g];
        Dev &d = dev[(size_t)g];
        CSC_CUDA(cudaSetDevice(c->device), what);
        size_t free_b = 0, total_b = 0;
        CSC_CUDA(cudaMemGetInfo(&free_b, &total_b), what);
        const size_t all = 8 * (size_t)nnz;
        d.resident = all <= free_b / 2 && (!limited || all <= stage);
        const size_t entries = d.resident ? (size_t)std::max<int64_t>(nnz, 1) : (size_t)chunk_entries;
        CSC_CUDA(d.mem.alloc(c->device, (void **)&d.val, sizeof(uint32_t) * entries), what);
        CSC_CUDA(d.mem.alloc(c->device, (void **)&d.row, sizeof(int) * entries), what);
        CSC_CUDA(d.mem.alloc(c->device, (void **)&d.outer, sizeof(int) * ((size_t)N + 1)), what);
        CSC_CUDA(d.mem.alloc(c->device, (void **)&d.bad, sizeof(int)), what);
        CSC_CUDA(cudaMemcpyAsync(d.outer, outer_ptr, sizeof(int) * ((size_t)N + 1), cudaMemcpyHostToDevice, c->stream), what);
        CSC_CUDA(cudaMemsetAsync(d.bad, 0, sizeof(int), c->stream), what);
        for (const Chunk &k : ch) {
            int64_t seg0 = 0;
            int rc_ = upload(c, d, k, &seg0, d.resident); // chunks uploaded again for the scatter: rows only here
            if (rc_) return rc_;
            const int nc = k.c1 - k.c0;
            if (nc > 0 && k.e1 > k.e0) {
                k_csc_check<<<(unsigned)(((int64_t)nc * 32 + 255) / 256), 256, 0, c->stream>>>(d.outer, k.c0, nc, seg0, d.resident ? nnz : chunk_entries, d.row, N, d.bad);
                CSC_CUDA(cudaGetLastError(), what);
            }
        }
        int bad = 0;
        CSC_CUDA(cudaMemcpyAsync(&bad, d.bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream), what);
        CSC_CUDA(cudaStreamSynchronize(c->stream), what);
        if (bad) { daisy_set_error("%s: a row index outside [0, N) or not strictly ascending within its column", what); return DAISY_E_INVALID; }
        return DAISY_OK;
    });
    if (rc) return rc;
    // 2. every device passed: zero the rows and scatter
    return each_ctx(ctx, n, what, [&](int g) -> int {
        daisy_ctx *c = ctx[g];
        Dev &d = dev[(size_t)g];
        CSC_CUDA(cudaSetDevice(c->device), what);
        int rc_ = dz_ensure_F(c);
        if (rc_) return rc_;
        const int nloc = c->row1 - c->row0;
        CSC_CUDA(cudaMemsetAsync(c->d_F, 0, sizeof(float) * (size_t)(nloc > 0 ? nloc : 1) * (size_t)c->ldF, c->stream), what);
        auto scatter = [&](int c0, int nc, int64_t seg0, int64_t seglen) -> int {
            if (nc <= 0 || nloc <= 0) return DAISY_OK;
            k_csc_scatter<<<(unsigned)(((int64_t)nc * 32 + 255) / 256), 256, 0, c->stream>>>(d.outer, c0, nc, seg0, seglen, d.val, d.row, c->row0, c->row1,
                                                                                          (uint32_t *)c->d_F, c->ldF, (int64_t)nloc * c->ldF);
            CSC_CUDA(cudaGetLastError(), what);
            return DAISY_OK;
        };
        if (d.resident) rc_ = scatter(0, N, 0, nnz);
        else
            for (const Chunk &k : ch) {
                int64_t seg0 = 0;
                rc_ = upload(c, d, k, &seg0, true);
                if (!rc_ && k.e1 > k.e0) rc_ = scatter(k.c0, k.c1 - k.c0, seg0, chunk_entries);
                if (rc_) break;
            }
        if (rc_) return rc_;
        CSC_CUDA(cudaStreamSynchronize(c->stream), what);
        c->have_F = true;
        c->F_version++;
        c->rec.valid = false; // F no longer is a matrix this library computed
        c->csc_uploads = d.resident ? 1 : 2;
        return DAISY_OK;
    });
}

extern "C" int daisy_formfactors_write_csc(daisy_ctx *ctx, int64_t nnz, const float *values, const int32_t *inner_idx, const int32_t *outer_ptr) {
    DZ_REQUIRE(ctx, DAISY_E_INVALID, "daisy_formfactors_write_csc: null context");
    DzRange range_("daisy_formfactors_write_csc");
    return dz_csc_import(&ctx, 1, nnz, values, inner_idx, outer_ptr, "daisy_formfactors_write_csc");
}

extern "C" int daisy_formfactors_csc_uploads(daisy_ctx *ctx) { return ctx ? ctx->csc_uploads : DAISY_E_INVALID; }
