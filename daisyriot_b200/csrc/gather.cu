// gather.cu -- the radiosity / fluorescence gather pass: residual <- M (F residual); B += residual.
//
// Replaces the single-threaded Eigen loops of the reference's Lightning family ("visual studio/Lightning.h"):
//   SpectralLightning::increment_light_fluorescent  :196-226  (K SpMVs + N KxK mat-vecs)
//   RGBLightning::increment_lightpass               :342-349  (K=3, M = diag(rho))
//   BWLightning::increment_lightpass                :419-424  (K=1, M = [1])
//   converge_lightning / check_convergence          :145-151, :255-261, :336-340, :410-415
//
// F is dense FP32, row-major, resident in HBM; one pass streams it exactly once.  Three main kernels, all persistent
// with work items (row block) x (column range):
//   k_gather_tma<K>      K <= 9: a producer warp fills a 6-stage shared-memory ring with tiled TMA loads (F tile +
//                        residual band slices), 8 consumer warps do K FMAs per F element; the default
//   k_gather_mma<K>      K = 16 / 32 / 64: tcgen05 3xTF32 tensor-core kernel with the F operand staged in TMEM (gather_mma.cuh);
//                        the only kernel for K > 32
//   k_gather_partial<K>  the first-generation register-prefetch kernel, kept selectable (DAISY_GATHER=ldg) as a reference point
// k_gather_epilogue sums the column-range partials, applies the per-material KxK matrix, accumulates B, writes the new
// residual into this rank's exchange block -- or, with the fused exchange, into every rank's buffer over NVLink -- and
// totals the per-band residual sums.
#include "daisy_common.cuh"
#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <atomic>
#include <cmath>
#include <mutex>
#include <vector>

#define G_WARPS 8
#define G_THREADS (G_WARPS * 32)
#define G_TC 512 // residual tile width (columns)

// a solver is sized by the mesh its context held at daisy_solver_create (N, row blocks, material ids); after
// daisy_ctx_replace_mesh every call but destroy refuses it
#define DZ_SOLVER_CURRENT(s, what)                                                                                           \
    DZ_REQUIRE((s)->mesh_version == (s)->ctx->mesh_version, DAISY_E_STATE,                                                   \
               what ": the context's mesh was replaced (daisy_ctx_replace_mesh) after this solver was created; create a new solver")

struct daisy_solver {
    daisy_ctx *ctx = nullptr;
    uint64_t mesh_version = 0; // the context's mesh_version at create: the mesh N, the row blocks and mat_idx belong to
    int K = 0, Kp = 0; // bands requested / bands the kernel is instantiated for
    int nmat = 0, nmat_cap = 0; // materials in use / material matrices d_M has room for (daisy_solver_set_materials)
    bool abs_sums = false;      // restart mode: the passes total |r| (from daisy_solver_restart to the next reset / write)
    int N = 0, n = 0, G = 1, rank = 0, nloc = 0, row0 = 0;
    int64_t bstride = 0;   // floats per exchange block
    int64_t sums_off = 0;  // float offset of the K doubles inside a block
    float *d_res[2] = { nullptr, nullptr }; // exchange buffers (G blocks each)
    int cur = 0;
    float *d_B = nullptr;  // Kp x n   (band-major, local rows)
    float *d_E = nullptr;  // exchange-layout copy of the emission (reset source)
    float *d_M = nullptr;  // nmat x Kp x Kp column-major
    int *d_mat = nullptr;  // local rows
    float *d_partial = nullptr; // nsplit x nloc x Kp
    double *d_cta_sums = nullptr;
    unsigned int *d_done = nullptr;
    unsigned int *d_rb_arrive = nullptr; // fused epilogue (k_gather_tma): column splits finished per row block
    double *d_rb_sums = nullptr;         // per row block band sums
    int nrb_tma = 0;
    unsigned long long *h_abort = nullptr, *d_abort_host = nullptr; // host-mapped abort marker of the fused exchange
    unsigned long long timeout_ns = 30000000000ull;                  // how long a pass waits for a peer's block (DAISY_EXCHANGE_TIMEOUT_MS)
    int R = 8, nsplit = 1, grid = 148, colw = 0;
    int sk_S = 0, sk_L = 0, sk_total = 0, sk_grid = 0, sk_maxp = 1; // stream-K decomposition of the fused TMA kernel (plan())
    int partial_splits = 0;             // d_partial holds partial_splits x nloc x Kp floats
    // tile skipping (fused K <= 9 kernel, DAISY_GATHER_SKIP=0 turns it off): the stream-K sequence holds only the F tiles with a
    // non-zero entry.  d_sk_list = column step of every entry (-1: the single null entry of a row block without any), d_sk_off =
    // nrb + 1 offsets of the row blocks' entries.  Rebuilt whenever ctx->F_version moves away from scanned_version.
    bool skip = false;
    uint64_t scanned_version = 0;
    int *d_sk_list = nullptr, *d_sk_off = nullptr;
    int64_t sk_list_cap = 0;
    std::vector<unsigned char> occ;     // tile map of the last scan: nrb_tma x sk_S
    int64_t occupied = 0;
    double scan_ms = 0.0;
    bool use_tma = true;
    bool use_mma = false;               // K = 16 / 32 / 64: tcgen05 3xTF32 path (gather_mma.cuh)
    bool fused_epi = false;             // k_gather_tma does the epilogue (and the exchange wait) itself: one launch per pass
    float *d_split = nullptr;           // [Rh; Rl]: 2*Kp x ncolsP, rewritten at the start of every pass
    int ncolsP = 0;
    alignas(64) CUtensorMap tmF;        // F rows of this rank: 2-D (ldF x nloc), box 128 x tile rows
    alignas(64) CUtensorMap tmRes[2];   // exchange buffers: 3-D (n x Kp x G), box 128 x Kp x 1
    alignas(64) CUtensorMap tmFmma;     // F rows, box 32 x 128, SWIZZLE_128B
    alignas(64) CUtensorMap tmSplit;    // d_split, box 32 x 2*Kp, SWIZZLE_128B
    // fused exchange (multi-GPU): the epilogue stores this rank's block straight into every rank's next buffer through
    // CUDA-IPC mappings (NVLink), then raises flag[rank] = pass sequence number in every rank's flag array
    bool fused = false;
    bool peers_ipc = false;                            // peer pointers are CUDA-IPC mappings to be closed (one process per GPU)
    float *peer_res[2][16] = { { nullptr } };          // [buffer][rank] base of that rank's exchange buffer
    unsigned long long *peer_flags[16] = { nullptr };  // [rank] base of that rank's flag array
    unsigned long long *d_flags = nullptr;             // own flag array (16 entries) + [16] = wait timeout marker
    unsigned long long seq = 0;                        // passes launched since creation (never reset)
    int numpasses = 0;
    double last_ms = 0.0;
    std::vector<double> sums;   // band sums of the current residual
    bool sums_valid = true;
    std::vector<double> e_sums; // band sums of the emission
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    int pin16 = 0;                      // sixteenths of the local F rows kept in L2 across passes (plan())
    bool events_recorded = false;       // e0 / e1 bracket the most recent pass
    bool chained = false;               // daisy_solver_set_chained: passes launched back to back without per-pass events
    unsigned int *d_stop = nullptr;     // device converge: {stopped, passes} (DevStop::state), allocated by the first call
    void *h_stop = nullptr;             // pinned: that word, then the G x Kp band sums of the batch's last pass
};

// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    }
}
// 1-D TMA bulk copy global -> shared, completion counted in bytes on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// tiled TMA loads through a tensor map (SASS: UTMALDG); out-of-range parts of the box are zero-filled
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *tm, int c0, int c1, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(dst)), "l"(tm), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}
// the same with an L2 eviction policy (createpolicy): evict_last keeps a tile in the 126 MB L2 from one pass to the next
__device__ __forceinline__ void tma_load_2d_hint(void *dst, const CUtensorMap *tm, int c0, int c1, uint64_t *bar, uint64_t policy) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;"
                 ::"r"(smem_u32(dst)), "l"(tm), "r"(c0), "r"(c1), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void *dst, const CUtensorMap *tm, int c0, int c1, int c2, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_u32(dst)), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)) : "memory");
}

// Device converge (daisy_solver_converge_device, DESIGN 3.3): the passes of one call are launched back to back and every pass
// but the first applies converge_lightning's stop rule to the band sums the previous pass left in the tails of the buffer it
// reads.  state == null: an ordinary pass (one branch on a kernel parameter).
struct DevStop {
    unsigned int *state;   // {stopped, passes}: cleared by the host at the start of the call
    const double *tails;   // rank g's K band sums of the residual this pass reads: tails[g * tstride + k]
    int64_t tstride;
    int G, K;              // ranks, bands that count (not the padded Kp)
    int rule;              // -1: no test (the host decided the first pass), 0: total over bands, 1: per band
    double threshold;
};

// converged(): the host loop's unconverged() negated, on the totals fetch_sums forms -- the same doubles added in the same order
__device__ __forceinline__ bool stop_converged(const DevStop &S) {
    const volatile double *t = S.tails;
    double tot = 0.0;
    bool over = false;
    for (int k = 0; k < S.K; k++) {
        double v = 0.0;
        for (int g = 0; g < S.G; g++) v += t[(size_t)g * S.tstride + k];
        over = over || v > S.threshold;
        tot += v;
    }
    return S.rule ? !over : !(tot > S.threshold);
}
__device__ __forceinline__ bool stop_stopped(const DevStop &S) { return *reinterpret_cast<volatile unsigned int *>(S.state) != 0u; }
// the decision of a pass (every thread that asks gets the same answer): true = do nothing.  A pass that finds the residual
// converged says so in state[0] for the launches behind it, whose buffers are stale and must not be tested.
__device__ __forceinline__ bool stop_decide(const DevStop &S) {
    if (stop_stopped(S)) return true;
    if (S.rule < 0 || !stop_converged(S)) return false;
    *reinterpret_cast<volatile unsigned int *>(S.state) = 1u;
    return true;
}

struct GatherParams {
    const float *F; int64_t ldF;
    int nloc;               // local rows
    int ncols;              // padded column count G*n
    int n;                  // rows per rank (block length)
    const float *res;       // exchange buffer (read)
    int64_t bstride;
    float *partial;         // nsplit x nloc x K
    int nsplit, colw;       // column range width per split (multiple of G_TC)
    int nrb;                // row blocks
    // stream-K decomposition of k_gather_tma (fused epilogue): the (row block, 256-column step) pairs of the whole matrix form
    // one sequence of sk_total steps, row block major; CTA c streams the contiguous range [c sk_L, (c+1) sk_L) -- every SM
    // gets the same number of steps whatever the matrix shape, and a row block is shared by at most a few CTAs ("pieces")
    int sk;                 // 1: stream-K pieces, 0: (row block, column split) items
    int sk_S, sk_L, sk_total; // steps per row block, steps per CTA, steps in total
    // tile skipping (sk_off != null): the sequence is the list of occupied tiles instead, sk_total entries, row block rb owning
    // entries [sk_off[rb], sk_off[rb+1]) whose column steps are sk_list[]; CTA c streams the entries [c T / grid, (c+1) T / grid)
    const int *sk_list, *sk_off;
    // L2 residency: the F tiles whose step number s has (s * 11 + rb * 5) % 16 < pin16 are loaded evict_last, the others
    // evict_first -- a fixed subset of the matrix, spread evenly over the CTAs, that stays in L2 from pass to pass when the
    // matrix is not much larger than L2 (the reference's own scenes: 164 / 238 MB against 126 MB of L2)
    int pin16;
    DevStop stop;
};

// one unit of work of k_gather_tma: steps [s0, s1) of row block rb (tile skipping: entries [s0, s1) of sk_list); idx / np =
// this piece's ordinal among / number of the pieces that make up the row block (their partial sums are added in idx order)
struct Piece { int rb, s0, s1, idx, np; };

// stage the K bands of columns [j0, j0+w) of the exchange buffer into tile[k][0..w)
template <int K>
__device__ __forceinline__ void issue_tile(const GatherParams &P, float *tile, uint64_t *bar, int j0, int w) {
    mbar_expect_tx(bar, (uint32_t)(K * w * 4));
    int g = j0 / P.n, jl = j0 - g * P.n;
    int w1 = min(w, P.n - jl); // part inside block g; the rest (if any) continues in block g+1
#pragma unroll 1
    for (int k = 0; k < K; k++) {
        bulk_g2s(tile + k * G_TC, P.res + (size_t)g * P.bstride + (size_t)k * P.n + jl, (uint32_t)(w1 * 4), bar);
        if (w1 < w) bulk_g2s(tile + k * G_TC + w1, P.res + (size_t)(g + 1) * P.bstride + (size_t)k * P.n, (uint32_t)((w - w1) * 4), bar);
    }
}

template <int K, int R>
__global__ void __launch_bounds__(G_THREADS, 1) k_gather_partial(GatherParams P) {
    extern __shared__ __align__(128) unsigned char g_smem[];
    float *tiles = reinterpret_cast<float *>(g_smem);                 // 2 x K x G_TC
    uint64_t *bars = reinterpret_cast<uint64_t *>(g_smem + 2 * K * G_TC * sizeof(float));
    int *s_stop = reinterpret_cast<int *>(bars + 2);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) {
        mbar_init(&bars[0], 1);
        mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (P.stop.state) *s_stop = stop_decide(P.stop);
    }
    __syncthreads();
    if (P.stop.state && *s_stop) return; // device converge: no load has been issued yet
    uint32_t phase[2] = { 0, 0 };
    const int nitems = P.nrb * P.nsplit;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int rb = item / P.nsplit, split = item - rb * P.nsplit;
        const int c_begin = split * P.colw;
        const int c_end = min(P.ncols, c_begin + P.colw);
        const int ntile = (c_end - c_begin + G_TC - 1) / G_TC;
        const int row_base = rb * (G_WARPS * R) + warp * R;
        const float *Frow[R];
#pragma unroll
        for (int r = 0; r < R; r++) Frow[r] = P.F + (size_t)min(row_base + r, P.nloc - 1) * P.ldF + c_begin + lane * 4;
        float acc[R][K];
#pragma unroll
        for (int r = 0; r < R; r++)
#pragma unroll
            for (int k = 0; k < K; k++) acc[r][k] = 0.0f;
        if (tid == 0) {
            issue_tile<K>(P, tiles, &bars[0], c_begin, min(G_TC, c_end - c_begin));
            if (ntile > 1) issue_tile<K>(P, tiles + K * G_TC, &bars[1], c_begin + G_TC, min(G_TC, c_end - c_begin - G_TC));
        }
        const int nstep = (c_end - c_begin + 127) / 128;
        float4 fcur[R], fnxt[R];
        {
            bool in = (lane * 4) < (c_end - c_begin);
#pragma unroll
            for (int r = 0; r < R; r++) fcur[r] = in ? ldg_stream(Frow[r]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        for (int s = 0; s < nstep; s++) {
            const int t = s >> 2, buf = t & 1;
            if (s + 1 < nstep) {
                bool in = ((s + 1) * 128 + lane * 4) < (c_end - c_begin);
#pragma unroll
                for (int r = 0; r < R; r++) fnxt[r] = in ? ldg_stream(Frow[r] + (size_t)(s + 1) * 128) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            if ((s & 3) == 0) { mbar_wait(&bars[buf], phase[buf]); phase[buf] ^= 1; }
            const int col = (s & 3) * 128 + lane * 4; // tile-local column
            if (t * G_TC + col < c_end - c_begin) {
                const float *tile = tiles + buf * K * G_TC + col;
#pragma unroll
                for (int k = 0; k < K; k++) {
                    float4 x = *reinterpret_cast<const float4 *>(tile + k * G_TC);
#pragma unroll
                    for (int r = 0; r < R; r++) {
                        acc[r][k] = fmaf(fcur[r].x, x.x, acc[r][k]);
                        acc[r][k] = fmaf(fcur[r].y, x.y, acc[r][k]);
                        acc[r][k] = fmaf(fcur[r].z, x.z, acc[r][k]);
                        acc[r][k] = fmaf(fcur[r].w, x.w, acc[r][k]);
                    }
                }
            }
            if ((s & 3) == 3 || s == nstep - 1) {
                __syncthreads(); // every warp is done with tile t
                if (tid == 0 && t + 2 < ntile) {
                    int j0 = c_begin + (t + 2) * G_TC;
                    issue_tile<K>(P, tiles + buf * K * G_TC, &bars[buf], j0, min(G_TC, c_end - j0));
                }
            }
#pragma unroll
            for (int r = 0; r < R; r++) fcur[r] = fnxt[r];
        }
        // lane reduction (fixed xor tree => deterministic), lane 0 stores the column-range partial
#pragma unroll
        for (int r = 0; r < R; r++)
#pragma unroll
            for (int k = 0; k < K; k++) {
                float v = acc[r][k];
                v += __shfl_xor_sync(0xffffffffu, v, 16);
                v += __shfl_xor_sync(0xffffffffu, v, 8);
                v += __shfl_xor_sync(0xffffffffu, v, 4);
                v += __shfl_xor_sync(0xffffffffu, v, 2);
                v += __shfl_xor_sync(0xffffffffu, v, 1);
                acc[r][k] = v;
            }
        if (lane == 0) {
#pragma unroll
            for (int r = 0; r < R; r++) {
                int row = row_base + r;
                if (row < P.nloc) {
                    float *dst = P.partial + ((size_t)split * P.nloc + row) * K;
#pragma unroll
                    for (int k = 0; k < K; k++) dst[k] = acc[r][k];
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// k_gather_tma: the same work decomposition with a register-free load pipeline.  Warp 8 is the producer: for every
// 128-column step it fills one shared-memory stage -- the 64x128 F tile as 64 row segments plus the K residual band
// slices -- with 1-D TMA bulk copies that complete on the stage's "full" mbarrier.  Warps 0-7 consume: LDS.128 of their
// 8 F rows and the K band slices, K FMAs per F element, then one arrive on the stage's "empty" mbarrier.  Up to
// NSTAGE x (64+K) x 512 B (~219 KB for K=9) are in flight per SM without holding a single register, and there is no
// CTA-wide barrier in the loop.
// The F tile of the K <= 9 kernel is 64 rows x 256 columns: 1 KB of every row per TMA box, three 73 KB stages.  With 64 x 128
// tiles (512 B per row, six stages -- the first version) the same kernel reached 6.9 TB/s at 131072 columns; 1 KB segments
// give 7.1 TB/s (DRAM page locality).  32 x 256 tiles (five stages) are as fast on one GPU but lose on row-sharded matrices,
// where the residual tile (K x 256 per box, from L2) is a larger share of the traffic (measured on 2 GPUs: 0.371 / 0.357 /
// 0.345 ms per pass for 32x256 / 64x128 / 64x256 at 32768 patches).
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// rows per consumer warp / consumer warps per CTA: the K accumulators of RW rows must fit the register file
template <int K> struct TmaCfg { static constexpr int RW = 8, NCW = 8, COLS = 256; };   // K <= 9 : 64 x 256 tiles, 9 warps
template <> struct TmaCfg<16> { static constexpr int RW = 4, NCW = 16, COLS = 128; };   // 64 x 128 tiles, 17 warps
template <> struct TmaCfg<32> { static constexpr int RW = 4, NCW = 8, COLS = 128; };    // 32 x 128 tiles, 9 warps (FP32-pipe bound anyway)
template <int K>
__host__ __device__ constexpr int tma_rows() { return TmaCfg<K>::RW * TmaCfg<K>::NCW; }
template <int K>
__host__ __device__ constexpr int tma_stage_bytes() { return (tma_rows<K>() + K) * TmaCfg<K>::COLS * 4; }
// shared memory kept back for the fused epilogue: the block's K sums per row (single column split: they never leave the SM)
// and the scratch of the ordered band-sum reductions
template <int K>
__host__ __device__ constexpr int tma_epi_bytes() { return 2 * tma_rows<K>() * K * 4 + 2048 + 64; }
template <int K>
__host__ __device__ constexpr int tma_nstage() {
    return (227 * 1024 - 256 - tma_epi_bytes<K>()) / tma_stage_bytes<K>() > 8 ? 8 : (227 * 1024 - 256 - tma_epi_bytes<K>()) / tma_stage_bytes<K>();
}

// What used to be a second kernel (k_gather_epilogue) and, multi-GPU, a third one in front (k_wait_flags), folded into the
// streaming kernel:
//  * the CTA that completes the LAST column split of a row block (per-block arrival counter) sums the splits in split order,
//    applies the material matrices, accumulates B, stores the block's new residual -- into this rank's exchange block or,
//    fused exchange, into every rank's buffer over NVLink -- and leaves the block's band sums in rb_sums;
//  * the CTA that completes the last row block of the pass totals the band sums in block order and publishes them (and,
//    fused exchange, raises flag[rank] = seq in every rank's flag array);
//  * fused exchange: the producer lane polls flag[g] >= wait_seq only right before the first residual tile of rank g's block,
//    so the stream starts on the blocks that have already arrived (the F tile of that step is already in flight).
// A peer that does not show up within timeout_ns sets the abort markers (device flag word 16 and a host-mapped word): this
// pass then publishes nothing, every later pass returns at once, and the host reports the error at its next call.
struct FusedEpi {
    int enabled;
    unsigned int *rb_arrive;  // per row block: column splits finished (returns to 0 by the end of the pass)
    double *rb_sums;          // nrb x K
    unsigned int *done;       // row blocks finished
    const float *M; const int *mat; float *B;
    float *res_out_block;     // this rank's block of the next exchange buffer (npeers == 0)
    double *block_sums;
    int npeers;
    float *peer_out[16];
    double *peer_sums[16];
    unsigned long long *peer_flag[16];
    unsigned long long seq;
    unsigned long long *flags;       // own flag array; [16] = abort marker
    unsigned long long *host_abort;  // host-mapped copy of the abort marker (may be null)
    int G;
    unsigned long long wait_seq;     // 0: nothing to wait for
    unsigned long long timeout_ns;
    // restart pass (read only by the ABS instantiation): the pass reads B_old, and the epilogue forms B_new = y + E and
    // r = B_new - B_old from this rank's emission block instead of B += y
    int restart;
    const float *E_block;
};

// acquire flag[g] >= wait_seq: rank g's block of the previous pass has landed here and rank g has finished reading the buffer
// this pass writes into.  A peer that does not show up within timeout_ns sets the abort markers instead.
__device__ __forceinline__ void wait_flag(const FusedEpi &E, int g) {
    unsigned long long t0, t1, v;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    while (true) {
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(E.flags + g) : "memory");
        if (v >= E.wait_seq) break;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
        if (t1 - t0 > E.timeout_ns) {
            E.flags[16] = E.seq;
            if (E.host_abort) *reinterpret_cast<volatile unsigned long long *>(E.host_abort) = E.seq;
            __threadfence_system();
            break;
        }
        __nanosleep(100);
    }
}

// the device-converge decision of k_gather_tma.  Fused exchange: the test needs every rank's sums of the previous pass, so
// all G flags are awaited first (a pass that stops raises no flag, so a stopped launch must not wait for any)
__device__ __forceinline__ bool tma_stop_decide(const DevStop &S, const FusedEpi &E) {
    if (stop_stopped(S)) return true;
    if (S.rule < 0) return false;
    if (E.enabled && E.npeers > 0 && E.wait_seq != 0ull) {
        for (int g = 0; g < E.G; g++) wait_flag(E, g);
        if (*reinterpret_cast<volatile unsigned long long *>(E.flags + 16) != 0ull) return true; // gave up on a peer: the host reports it
    }
    return stop_decide(S);
}


#ifdef __CUDA_ARCH__
#define DZ_ASSERT_HD(cond) DZ_ASSERT(cond)
#define DZ_LDG(p) __ldg(p)
#else
#define DZ_ASSERT_HD(cond) do { } while (0)
#define DZ_LDG(p) (*(p))
#endif
// tile skipping: CTA c of ncta streams the entries [sk_bound(c), sk_bound(c+1)) -- lengths differ by at most one; sk_owner(e) is
// the CTA whose range holds entry e
__host__ __device__ __forceinline__ int sk_bound(int c, int T, int ncta) { return (int)((long long)c * T / ncta); }
__host__ __device__ __forceinline__ int sk_owner(int e, int T, int ncta) { return (int)((((long long)e + 1) * ncta - 1) / T); }
// column step of position e of a piece's range
__device__ __forceinline__ int piece_step(const GatherParams &P, int e) {
    const int s = P.sk_list ? __ldg(P.sk_list + e) : e;
    DZ_ASSERT(s >= 0 && s < P.sk_S && (!P.sk_list || e < P.sk_total));
    return s;
}

// the i-th piece of CTA `cta` (cursor: running position, start at 0; p: the piece the previous call returned); false when the
// CTA has no more work.  Host-callable for daisy_gather_plan_dump.
template <int T_COLS>
__host__ __device__ __forceinline__ bool next_piece(const GatherParams &P, int cta, int ncta, int &cursor, Piece &p) {
    if (P.sk_off) {
        const int c1 = sk_bound(cta + 1, P.sk_total, ncta), g0 = sk_bound(cta, P.sk_total, ncta) + cursor;
        if (g0 >= c1) return false;
        int rb;
        if (cursor == 0) { // largest rb with sk_off[rb] <= g0
            int lo = 0, hi = P.nrb - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (DZ_LDG(P.sk_off + mid) <= g0) lo = mid; else hi = mid - 1;
            }
            rb = lo;
        } else {
            rb = p.rb + 1; // a CTA's range is contiguous and every row block owns at least one entry
        }
        const int e0 = DZ_LDG(P.sk_off + rb), e1 = DZ_LDG(P.sk_off + rb + 1);
        DZ_ASSERT_HD(rb >= 0 && rb < P.nrb && e0 <= g0 && g0 < e1 && e1 <= P.sk_total);
        p.rb = rb;
        p.s0 = g0;
        p.s1 = e1 < c1 ? e1 : c1;
        const int first = sk_owner(e0, P.sk_total, ncta);
        p.idx = cta - first;
        p.np = sk_owner(e1 - 1, P.sk_total, ncta) - first + 1;
        cursor += p.s1 - p.s0;
        if (DZ_LDG(P.sk_list + e0) < 0) p.s1 = p.s0; // the null entry of a row block without an occupied tile: nothing to stream
        return true;
    }
    if (P.sk) {
        const int g0 = cta * P.sk_L + cursor, g1 = min(P.sk_total, (cta + 1) * P.sk_L);
        if (g0 >= g1) return false;
        p.rb = g0 / P.sk_S;
        p.s0 = g0 - p.rb * P.sk_S;
        p.s1 = min(P.sk_S, p.s0 + (g1 - g0));
        const int first = (p.rb * P.sk_S) / P.sk_L, lastc = ((p.rb + 1) * P.sk_S - 1) / P.sk_L;
        p.idx = cta - first;
        p.np = lastc - first + 1;
        cursor += p.s1 - p.s0;
        return true;
    }
    const int item = cta + cursor * ncta;
    if (item >= P.nrb * P.nsplit) return false;
    p.rb = item / P.nsplit;
    p.idx = item - p.rb * P.nsplit;
    p.np = P.nsplit;
    const int c_begin = p.idx * P.colw, c_end = min(P.ncols, c_begin + P.colw);
    p.s0 = c_begin / T_COLS;
    p.s1 = p.s0 + (c_end - c_begin + T_COLS - 1) / T_COLS;
    cursor++;
    return true;
}

// ABS (restart mode, DESIGN 3.3b): the band sums total |r| instead of r, and E.restart selects the restart epilogue.  A template
// parameter rather than a flag, so that the kernel of an ordinary pass is the one it always was.
template <int K, bool ABS = false>
__global__ void __launch_bounds__((TmaCfg<K>::NCW + 3) * 32, 1)
k_gather_tma(GatherParams P, const __grid_constant__ CUtensorMap tmF, const __grid_constant__ CUtensorMap tmRes, const __grid_constant__ FusedEpi E) {
    constexpr int NST = tma_nstage<K>();
    constexpr int STAGE_F = tma_stage_bytes<K>() / 4; // floats per stage
    constexpr int RW = TmaCfg<K>::RW, NCW = TmaCfg<K>::NCW, T_ROWS = RW * NCW, T_COLS = TmaCfg<K>::COLS;
    extern __shared__ __align__(128) unsigned char g_smem[];
    float *stages = reinterpret_cast<float *>(g_smem);
    uint64_t *full = reinterpret_cast<uint64_t *>(g_smem + (size_t)NST * tma_stage_bytes<K>());
    uint64_t *empty = full + NST;
    float *s_out = reinterpret_cast<float *>(empty + NST + 2);              // 2 x T_ROWS x K sums of a block (single split), double-buffered
    double *s_red = reinterpret_cast<double *>(s_out + 2 * tma_rows<K>() * K); // 2 KB: ordered reductions
    int *s_flag = reinterpret_cast<int *>(empty + NST);
    int *s_stop = s_flag + 1;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (E.enabled && *reinterpret_cast<volatile unsigned long long *>(E.flags + 16) != 0ull) return; // an earlier pass gave up on a peer
    if (tid == 0) {
        for (int i = 0; i < NST; i++) { mbar_init(&full[i], 1); mbar_init(&empty[i], NCW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // Programmatic dependent launch (chained passes, launch_pass_K): the next pass's grid may be scheduled onto SMs as this one
    // leaves them.  Its producer starts streaming F -- which no pass ever writes -- and only then waits for this grid to
    // complete before touching the residual; everything else in the kernel is downstream of the producer's loads, and the
    // other warps wait as well before they read or write global memory.  Without the launch attribute both are no-ops.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    uint32_t it = 0; // global step counter: stage = it % NST, phase = (it / NST) & 1
    int cursor = 0;
    Piece pc;
    // producer lane: the F tiles of the first NST steps go out before the previous pass is known to be complete; returns how many
    uint32_t pre = 0;
    auto issue_first_tiles = [&]() {
        uint64_t pl, pf;
        asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pl));
        asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pf));
        uint32_t n = 0;
        int cur2 = 0;
        Piece p2;
        while (n < (uint32_t)NST && next_piece<T_COLS>(P, blockIdx.x, gridDim.x, cur2, p2))
            for (int e = p2.s0; e < p2.s1 && n < (uint32_t)NST; e++, n++) {
                const int s = piece_step(P, e);
                mbar_expect_tx(&full[n], (uint32_t)tma_stage_bytes<K>());
                tma_load_2d_hint(stages + (size_t)n * STAGE_F, &tmF, s * T_COLS, p2.rb * T_ROWS, &full[n],
                                 (((s * 11 + p2.rb * 5) & 15) < P.pin16) ? pl : pf);
            }
        return n;
    };
    if (P.stop.state) {
        // device converge: the whole CTA takes the stop decision once the previous pass is complete.  A pass that does not run
        // leaves when the F tiles already in flight have landed: their stages expected the residual bytes too, which are
        // completed here instead of loaded.
        if (warp == NCW && lane == 0) pre = issue_first_tiles();
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (tid == 0) *s_stop = tma_stop_decide(P.stop, E);
        __syncthreads();
        if (*s_stop) {
            if (warp == NCW && lane == 0)
                for (uint32_t i = 0; i < pre; i++) {
                    asm volatile("mbarrier.complete_tx.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(&full[i])), "r"((uint32_t)(K * T_COLS * 4)) : "memory");
                    mbar_wait(&full[i], 0);
                }
            return;
        }
        if (warp == NCW && lane == 0) asm volatile("fence.proxy.async;" ::: "memory"); // the peers' blocks seen by tid 0, before the TMA reads
    }
    if (warp != NCW) asm volatile("griddepcontrol.wait;" ::: "memory");
    if (warp > NCW) {
        // ------------------------------- epilogue warps (64 threads) -------------------------------
        // They take over each finished item from the consumers (named barriers 2/3: "item done", 4/5: "buffer free"), so
        // the streaming never waits for an epilogue; only the last epilogue of a CTA is exposed.
        if (!E.enabled) return;
        const int et = tid - (NCW + 1) * 32, ewarp = et >> 5;
        auto esync = [&]() { asm volatile("bar.sync 1, 64;" ::: "memory"); };
        unsigned nitem_done = 0;
        // fused exchange: the stores below go into the buffer every peer read in the previous pass.  The pieces of a row block
        // need not have streamed a tile of every rank's block (tile skipping), so before its first peer store the CTA observes
        // every rank's flag itself
        bool flags_seen = E.npeers == 0 || E.wait_seq == 0ull;
        for (; next_piece<T_COLS>(P, blockIdx.x, gridDim.x, cursor, pc); nitem_done++) {
            const int rb = pc.rb;
            const int buf = (int)(nitem_done & 1u);
            DZ_ASSERT(rb >= 0 && rb < P.nrb && pc.idx >= 0 && pc.idx < pc.np);
            if (!flags_seen) {
                if (et == 0)
                    for (int g = 0; g < E.G; g++) wait_flag(E, g);
                esync();
                flags_seen = true;
            }
            asm volatile("bar.sync %0, %1;" ::"r"(2 + buf), "n"(NCW * 32 + 64) : "memory"); // the consumers have written this item's sums
            bool last = true;
            if (pc.np > 1) {
                if (et == 0) {
                    // release: the consumers' partial rows (ordered before this thread by the named barrier) become visible
                    // device-wide before the arrival is counted -- barrier + one fence + atomic, the usual semaphore pattern
                    __threadfence();
                    const unsigned old = atomicAdd(&E.rb_arrive[rb], 1u);
                    const int l = (old == (unsigned)pc.np - 1u);
                    if (l) E.rb_arrive[rb] = 0u;
                    *s_flag = l;
                }
                esync();
                last = *s_flag != 0;
                esync();
                if (last) __threadfence();
            }
            if (last) {
                double loc[K];
#pragma unroll
                for (int k = 0; k < K; k++) loc[k] = 0.0;
                const int row = rb * T_ROWS + et;
                if (et < T_ROWS && row < P.nloc) {
                    float b[K], Bv[K];
#pragma unroll
                    for (int k = 0; k < K; k++) Bv[k] = E.B[(size_t)k * P.n + row]; // issued first: independent of everything below
                    DZ_ASSERT(E.mat[row] >= 0 && row < P.n);
                    const float *Mp = E.M + (size_t)E.mat[row] * K * K;
                    if (pc.np == 1) {
#pragma unroll
                        for (int k = 0; k < K; k++) b[k] = s_out[buf * (T_ROWS * K) + et * K + k];
                    } else {
#pragma unroll
                        for (int k = 0; k < K; k++) b[k] = 0.0f;
                        for (int sp = 0; sp < pc.np; sp++) { // fixed order: the result does not depend on which CTA came last
                            const float *src = P.partial + ((size_t)sp * P.nloc + row) * K;
#pragma unroll
                            for (int k = 0; k < K; k++) b[k] += __ldcg(src + k);
                        }
                    }
                    float y[K];
#pragma unroll
                    for (int k = 0; k < K; k++) {
                        // result = reflectionmatrix[i] * patchrowvec  (column-major K x K)            Lightning.h:212
                        float v = 0.0f;
#pragma unroll
                        for (int j = 0; j < K; j++) v = fmaf(__ldg(Mp + j * K + k), b[j], v);
                        y[k] = v;
                        if constexpr (!ABS) loc[k] = (double)v;
                    }
                    if constexpr (ABS) {
                        // y = M (F B_old): B_new = y + E, r = B_new - B_old (restart pass); otherwise B += r, r = y
#pragma unroll
                        for (int k = 0; k < K; k++) {
                            float bn;
                            if (E.restart) {
                                bn = __fadd_rn(y[k], __ldg(E.E_block + (size_t)k * P.n + row));
                                y[k] = __fsub_rn(bn, Bv[k]);
                            } else {
                                bn = __fadd_rn(Bv[k], y[k]);
                            }
                            Bv[k] = bn;
                            loc[k] = fabs((double)y[k]);
                        }
#pragma unroll
                        for (int k = 0; k < K; k++) {
                            if (E.npeers > 0) {
                                for (int g = 0; g < E.npeers; g++) E.peer_out[g][(size_t)k * P.n + row] = y[k];
                            } else {
                                E.res_out_block[(size_t)k * P.n + row] = y[k];
                            }
                            E.B[(size_t)k * P.n + row] = Bv[k];
                        }
                    } else {
#pragma unroll
                        for (int k = 0; k < K; k++) {
                            if (E.npeers > 0) {
                                for (int g = 0; g < E.npeers; g++) E.peer_out[g][(size_t)k * P.n + row] = y[k]; // NVLink stores into every rank's buffer
                            } else {
                                E.res_out_block[(size_t)k * P.n + row] = y[k];                   // residualvector[j][i] = result[j]
                            }
                            E.B[(size_t)k * P.n + row] = Bv[k] + y[k];                           // lightningvalues += residual   :221-223
                        }
                    }
                    if (E.npeers > 0) __threadfence_system(); else __threadfence();
                }
                // band sums of the block: lanes -> warps -> block, always in index order
#pragma unroll
                for (int k = 0; k < K; k++) {
                    double v = loc[k];
                    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
                    if (lane == 0) s_red[ewarp * K + k] = v;
                }
                esync();
                if (et < K) {
                    E.rb_sums[(size_t)rb * K + et] = s_red[et] + s_red[K + et];
                    __threadfence();
                }
                esync();
                if (et == 0) *s_flag = (atomicAdd(E.done, 1u) == (unsigned)P.nrb - 1u);
                esync();
                const bool final_block = *s_flag != 0;
                esync();
                if (final_block) {
                    // the pass's last row block: total the band sums in block order (a fixed two-level order) and publish
                    __threadfence();
                    constexpr int NCH = (256 / K) < 32 ? (256 / K) : 32; // chunks of consecutive row blocks per band (NCH x K doubles fit s_red)
                    const int per = (P.nrb + NCH - 1) / NCH;
                    for (int t = et; t < NCH * K; t += 64) {
                        const int k = t % K, c = t / K;
                        double v = 0.0;
                        const volatile double *rs = E.rb_sums;
                        for (int b2 = c * per; b2 < min(P.nrb, (c + 1) * per); b2++) v += rs[(size_t)b2 * K + k];
                        s_red[c * K + k] = v;
                    }
                    esync();
                    const bool aborted = *reinterpret_cast<volatile unsigned long long *>(E.flags + 16) != 0ull;
                    if (et < K) {
                        double v = 0.0;
                        for (int c = 0; c < NCH; c++) v += s_red[c * K + et];
                        if (E.npeers > 0) { for (int g = 0; g < E.npeers; g++) E.peer_sums[g][et] = v; }
                        else E.block_sums[et] = v;
                    }
                    if (et == 0) {
                        *E.done = 0u;
                        if (P.stop.state) P.stop.state[1]++; // device converge: this pass ran
                    }
                    if (E.npeers > 0) {
                        __threadfence_system();
                        esync();
                        if (et < E.npeers && !aborted) {
                            // release: every store of this pass (fenced by its CTA before it arrived on `done`) precedes the flag
                            asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(E.peer_flag[et]), "l"(E.seq) : "memory");
                        }
                    }
                    esync();
                }
            }
            asm volatile("bar.arrive %0, %1;" ::"r"(4 + buf), "n"(NCW * 32 + 64) : "memory"); // this buffer may be refilled
        }
    } else if (warp == NCW) {
        // ------------------------------- producer -------------------------------
        // one elected lane issues two tiled TMA loads per stage: the T_ROWS x 128 block of F and the K x 128 block
        // of the residual bands (tiles never straddle an exchange block: n is a multiple of 256 when G > 1, and a
        // single block's tail beyond n is zero-filled by the TMA unit)
        if (lane == 0) {
            // ranks whose block of the previous pass is known to be here (a tested device-converge pass has awaited them all)
            unsigned ready = (E.enabled && E.wait_seq != 0ull && !(P.stop.state && P.stop.rule >= 0)) ? 0u : 0xffffffffu;
            uint64_t pol_last, pol_first;
            asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_last));
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));
            auto pol = [&](int rb, int s) -> uint64_t { return (((s * 11 + rb * 5) & 15) < P.pin16) ? pol_last : pol_first; };
            if (!P.stop.state) pre = issue_first_tiles();
            asm volatile("griddepcontrol.wait;" ::: "memory");
            while (next_piece<T_COLS>(P, blockIdx.x, gridDim.x, cursor, pc)) {
                const int row0 = pc.rb * T_ROWS;
                for (int e = pc.s0; e < pc.s1; e++, it++) {
                    const int st = it % NST;
                    const int s = piece_step(P, e);
                    const int col0 = s * T_COLS;
                    float *sf = stages + (size_t)st * STAGE_F;
                    if (it >= pre) {
                        mbar_wait(&empty[st], ((it / NST) & 1) ^ 1);
                        mbar_expect_tx(&full[st], (uint32_t)tma_stage_bytes<K>());
                        tma_load_2d_hint(sf, &tmF, col0, row0, &full[st], pol(pc.rb, s));
                    }
                    const int g = col0 / P.n, jl = col0 - g * P.n;
                    DZ_ASSERT(g >= 0 && g < 32 && col0 < P.ncols && row0 < P.nloc + T_ROWS);
                    if (!((ready >> g) & 1u)) {
                        wait_flag(E, g);
                        ready |= 1u << g;
                        asm volatile("fence.proxy.async;" ::: "memory"); // the peer's stores, seen by the acquire above, before the TMA reads below
                    }
                    tma_load_3d(sf + T_ROWS * T_COLS, &tmRes, jl, 0, g, &full[st]);
                }
            }
        }
    } else {
        // ------------------------------- consumers ------------------------------
        unsigned nitem_done = 0;
        while (next_piece<T_COLS>(P, blockIdx.x, gridDim.x, cursor, pc)) {
            const int split = pc.idx;
            const int row_base = pc.rb * T_ROWS + warp * RW;
            float acc[RW][K];
#pragma unroll
            for (int r = 0; r < RW; r++)
#pragma unroll
                for (int k = 0; k < K; k++) acc[r][k] = 0.0f;
            for (int s = pc.s0; s < pc.s1; s++, it++) {
                const int st = it % NST;
                mbar_wait(&full[st], (it / NST) & 1);
#pragma unroll
                for (int hcol = 0; hcol < T_COLS; hcol += 128) { // a lane covers 4 columns of every 128
                    const float *sf = stages + (size_t)st * STAGE_F + lane * 4 + hcol;
                    float4 f[RW];
#pragma unroll
                    for (int r = 0; r < RW; r++) f[r] = *reinterpret_cast<const float4 *>(sf + (warp * RW + r) * T_COLS);
#pragma unroll
                    for (int k = 0; k < K; k++) {
                        float4 x = *reinterpret_cast<const float4 *>(sf + (T_ROWS + k) * T_COLS);
#pragma unroll
                        for (int r = 0; r < RW; r++) {
                            acc[r][k] = fmaf(f[r].x, x.x, acc[r][k]);
                            acc[r][k] = fmaf(f[r].y, x.y, acc[r][k]);
                            acc[r][k] = fmaf(f[r].z, x.z, acc[r][k]);
                            acc[r][k] = fmaf(f[r].w, x.w, acc[r][k]);
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[st]);
            }
#pragma unroll
            for (int r = 0; r < RW; r++)
#pragma unroll
                for (int k = 0; k < K; k++) {
                    float v = acc[r][k];
                    v += __shfl_xor_sync(0xffffffffu, v, 16);
                    v += __shfl_xor_sync(0xffffffffu, v, 8);
                    v += __shfl_xor_sync(0xffffffffu, v, 4);
                    v += __shfl_xor_sync(0xffffffffu, v, 2);
                    v += __shfl_xor_sync(0xffffffffu, v, 1);
                    acc[r][k] = v;
                }
            // hand the block's sums to the epilogue warps (double-buffered: the consumers go straight on to the next item)
            const int buf = (int)(nitem_done & 1u);
            if (E.enabled && nitem_done >= 2u) asm volatile("bar.sync %0, %1;" ::"r"(4 + buf), "n"(NCW * 32 + 64) : "memory"); // epilogue of item - 2 has let go of this buffer
            if (lane == 0) {
#pragma unroll
                for (int r = 0; r < RW; r++) {
                    int row = row_base + r;
                    if (E.enabled && pc.np == 1) {
                        float *dst = s_out + buf * (T_ROWS * K) + (warp * RW + r) * K;
#pragma unroll
                        for (int k = 0; k < K; k++) dst[k] = acc[r][k];
                    } else if (row < P.nloc) {
                        float *dst = P.partial + ((size_t)split * P.nloc + row) * K;
#pragma unroll
                        for (int k = 0; k < K; k++) dst[k] = acc[r][k];
                    }
                }
            }
            if (E.enabled) asm volatile("bar.arrive %0, %1;" ::"r"(2 + buf), "n"(NCW * 32 + 64) : "memory");
            nitem_done++;
        }
    }
}

#include "gather_mma.cuh"

struct EpiParams {
    const float *partial; int nsplit, nloc, n;
    const float *M; const int *mat;
    float *res_out_block; // this rank's block of the next exchange buffer: K x n floats
    float *B;             // K x n
    double *cta_sums;     // gridDim x K
    double *block_sums;   // K doubles in the tail of this rank's block
    unsigned int *done;
    // fused exchange: npeers > 0 => the block (and its band sums) go to peer_out[g] / peer_sums[g] of every rank g
    // (own rank included) and, once every CTA's stores are fenced, flag[rank] of every rank is set to seq
    int npeers;
    float *peer_out[16];
    double *peer_sums[16];
    unsigned long long *peer_flag[16];
    unsigned long long seq;
    const unsigned long long *abort_marker; // flag word 16 of this rank (null: single GPU)
    unsigned int *stop_state;               // device converge: {stopped, passes} (the streaming kernel decided), else null
    int restart;                            // restart pass (ABS instantiation only): B_new = y + E_block, r = B_new - B_old
    const float *E_block;
};

// ABS: restart mode, band sums of |r| (see k_gather_tma)
template <int K, bool ABS = false>
__global__ void __launch_bounds__(256) k_gather_epilogue(EpiParams P) {
    __shared__ double s_sum[8][K];
    __shared__ bool s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (P.stop_state && *reinterpret_cast<volatile unsigned int *>(P.stop_state) != 0u) return;
    double loc[K];
#pragma unroll
    for (int k = 0; k < K; k++) loc[k] = 0.0;
    for (int row = blockIdx.x * blockDim.x + tid; row < P.nloc; row += gridDim.x * blockDim.x) {
        float b[K];
#pragma unroll
        for (int k = 0; k < K; k++) b[k] = 0.0f;
        for (int s = 0; s < P.nsplit; s++) {
            const float *src = P.partial + ((size_t)s * P.nloc + row) * K;
#pragma unroll
            for (int k = 0; k < K; k++) b[k] += src[k];
        }
        const float *Mp = P.M + (size_t)P.mat[row] * K * K;
#pragma unroll
        for (int k = 0; k < K; k++) {
            // result = reflectionmatrix[i] * patchrowvec  (column-major K x K)            Lightning.h:212
            float y = 0.0f;
#pragma unroll
            for (int j = 0; j < K; j++) y = fmaf(Mp[j * K + k], b[j], y);
            if constexpr (ABS) {
                const float bo = P.B[(size_t)k * P.n + row];
                float bn;
                if (P.restart) {
                    bn = __fadd_rn(y, P.E_block[(size_t)k * P.n + row]);
                    y = __fsub_rn(bn, bo);
                } else {
                    bn = __fadd_rn(bo, y);
                }
                if (P.npeers > 0) {
                    for (int g = 0; g < P.npeers; g++) P.peer_out[g][(size_t)k * P.n + row] = y;
                } else {
                    P.res_out_block[(size_t)k * P.n + row] = y;
                }
                P.B[(size_t)k * P.n + row] = bn;
                loc[k] += fabs((double)y);
                continue;
            }
            if (P.npeers > 0) {
                for (int g = 0; g < P.npeers; g++) P.peer_out[g][(size_t)k * P.n + row] = y; // NVLink stores into every rank's buffer
            } else {
                P.res_out_block[(size_t)k * P.n + row] = y;                      // residualvector[j][i] = result[j]
            }
            P.B[(size_t)k * P.n + row] = P.B[(size_t)k * P.n + row] + y;         // lightningvalues += residual   :221-223
            loc[k] += (double)y;
        }
    }
    // deterministic totals: lanes -> warps -> CTA -> (last CTA) grid, always in index order
#pragma unroll
    for (int k = 0; k < K; k++) {
        double v = loc[k];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) s_sum[warp][k] = v;
    }
    __syncthreads();
    if (tid < K) {
        double v = 0.0;
        for (int w = 0; w < 8; w++) v += s_sum[w][tid];
        P.cta_sums[(size_t)blockIdx.x * K + tid] = v;
    }
    if (P.npeers > 0) __threadfence_system(); else __threadfence(); // peer stores must be visible before the flag below
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(P.done, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
        __threadfence();
        if (tid < K) {
            double v = 0.0;
            volatile const double *cs = P.cta_sums;
            for (unsigned b = 0; b < gridDim.x; b++) v += cs[(size_t)b * K + tid];
            if (P.npeers > 0) { for (int g = 0; g < P.npeers; g++) P.peer_sums[g][tid] = v; }
            else P.block_sums[tid] = v;
        }
        if (tid == 0) {
            *P.done = 0;
            if (P.stop_state) P.stop_state[1]++; // device converge: this pass ran
        }
        if (P.npeers > 0) {
            __threadfence_system();
            __syncthreads();
            const bool aborted = P.abort_marker && *reinterpret_cast<const volatile unsigned long long *>(P.abort_marker) != 0ull;
            if (tid < P.npeers && !aborted) {
                // release: every store of this kernel (fenced by each CTA before it arrived on `done`) precedes the flag
                asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(P.peer_flag[tid]), "l"(P.seq) : "memory");
            }
        }
    }
}

// waits until every rank's block of pass `seq` has arrived in this rank's buffer (flag[g] >= seq for all g).  A peer that does
// not show up within timeout_ns turns into an error instead of a hung GPU: the abort markers are set (flag word 16 and the
// host-mapped word), the kernels of later passes return at once and nothing more is published to the peers.
// stopped != null (device converge): a launch behind the pass that found convergence waits for nothing, since no flag follows
__global__ void k_wait_flags(unsigned long long *flags, int G, unsigned long long seq, unsigned long long timeout_ns, unsigned long long *host_abort,
                             const unsigned int *stopped = nullptr) {
    const int g = threadIdx.x;
    if (g >= G) return;
    if (stopped && *reinterpret_cast<const volatile unsigned int *>(stopped) != 0u) return;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    while (true) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(flags + g) : "memory");
        if (v >= seq) break;
        if (*reinterpret_cast<volatile unsigned long long *>(flags + 16) != 0ull) break;
        unsigned long long t1;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
        if (t1 - t0 > timeout_ns) {
            flags[16] = seq;
            if (host_abort) *reinterpret_cast<volatile unsigned long long *>(host_abort) = seq;
            __threadfence_system();
            break;
        }
        __nanosleep(200);
    }
}

// ---------------------------------------------------------------------------------------------------------
template <int K, int R>
static int launch_partial(daisy_solver *s, const GatherParams &P) {
    size_t smem = 2 * K * G_TC * sizeof(float) + 64;
    // per device: a function attribute belongs to the device's context.  Solvers may run from several host threads; setting
    // the attribute twice is harmless, a torn flag is not.
    static std::atomic<bool> attr_done[64];
    if (!attr_done[s->ctx->device & 63].load()) {
        DZ_CUDA(cudaFuncSetAttribute(k_gather_partial<K, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_done[s->ctx->device & 63].store(true);
    }
    k_gather_partial<K, R><<<s->grid, G_THREADS, smem, s->ctx->stream>>>(P);
    DZ_CUDA(cudaGetLastError());
    return DAISY_OK;
}

// wait_seq != 0 (fused exchange): the blocks of pass wait_seq must have arrived before the residual is read.  The fused TMA
// kernel waits by itself, block by block; the other kernels get a k_wait_flags launch in front.
// stop != null: a pass of a device converge (state, rule and threshold set by the caller; the tails are filled in here)
// restart: the restart pass (daisy_solver_restart); s->abs_sums selects the epilogues that total |r|
template <int K>
static int launch_pass_K(daisy_solver *s, unsigned long long wait_seq, const DevStop *stop, bool restart) {
    daisy_ctx *c = s->ctx;
    if (wait_seq != 0ull && !s->fused_epi) {
        k_wait_flags<<<1, 32, 0, c->stream>>>(s->d_flags, s->G, wait_seq, s->timeout_ns, s->d_abort_host, stop ? stop->state : nullptr);
        DZ_CUDA(cudaGetLastError());
    }
    GatherParams P;
    P.F = c->d_F; P.ldF = c->ldF; P.nloc = s->nloc; P.ncols = s->G * s->n; P.n = s->n;
    P.res = s->d_res[s->cur]; P.bstride = s->bstride; P.partial = s->d_partial;
    P.nsplit = s->nsplit; P.colw = s->colw; P.nrb = (s->nloc + G_WARPS * s->R - 1) / (G_WARPS * s->R);
    P.sk = 0; P.sk_S = P.sk_L = P.sk_total = 0; P.pin16 = 0;
    P.sk_list = P.sk_off = nullptr;
    memset(&P.stop, 0, sizeof(P.stop));
    if (stop) {
        P.stop = *stop;
        P.stop.tails = reinterpret_cast<const double *>(s->d_res[s->cur] + s->sums_off);
        P.stop.tstride = s->bstride / 2; // bstride is a multiple of 4 floats
        P.stop.G = s->G; P.stop.K = s->K;
    }
    int rc;
    if (s->use_mma && (K == 16 || K == 32 || K == 64)) {
        if constexpr (K == 16 || K == 32 || K == 64) {
            constexpr size_t smem = mm_smem_bytes<K>();
            static std::atomic<bool> attr_done[64]; // per device
            if (!attr_done[c->device & 63].load()) {
                DZ_CUDA(cudaFuncSetAttribute(k_gather_mma<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                attr_done[c->device & 63].store(true);
            }
            k_split_residual<K><<<(s->ncolsP + 255) / 256, 256, 0, c->stream>>>(s->d_res[s->cur], s->bstride, s->n, s->G * s->n, s->ncolsP, s->d_split, P.stop);
            DZ_CUDA(cudaGetLastError());
            P.nrb = (s->nloc + MM_ROWS - 1) / MM_ROWS;
            k_gather_mma<K><<<s->grid, MM_THREADS, smem, c->stream>>>(P, s->tmFmma, s->tmSplit);
            DZ_CUDA(cudaGetLastError());
        }
        rc = DAISY_OK;
    } else if constexpr (K > 32) {
        daisy_set_error("%d bands run only on the tensor-core kernel", K); // daisy_solver_create refuses the other paths
        return DAISY_E_INVALID;
    } else if (s->use_tma) {
        constexpr int NST = tma_nstage<K>();
        size_t smem = (size_t)NST * tma_stage_bytes<K>() + 2 * NST * sizeof(uint64_t) + tma_epi_bytes<K>();
        // restart mode runs the ABS instantiation; only the fused epilogue reads it (otherwise the epilogue warps return at once)
        const bool abs_kernel = s->abs_sums && s->fused_epi;
        auto kern = abs_kernel ? k_gather_tma<K, true> : k_gather_tma<K, false>;
        static std::atomic<bool> attr_done[2][64]; // per instantiation and device
        if (!attr_done[abs_kernel][c->device & 63].load()) {
            DZ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            attr_done[abs_kernel][c->device & 63].store(true);
        }
        P.nrb = s->nrb_tma; // (nloc + tma_rows<K>() - 1) / tma_rows<K>(), and 1 for a rank without rows (plan())
        P.sk = s->fused_epi ? 1 : 0; P.sk_S = s->sk_S; P.sk_L = s->sk_L; P.sk_total = s->sk_total;
        if (s->skip) { P.sk_list = s->d_sk_list; P.sk_off = s->d_sk_off; }
        P.pin16 = s->pin16;
        const int grid = s->fused_epi ? s->sk_grid : s->grid;
        FusedEpi F;
        memset(&F, 0, sizeof(F));
        F.enabled = s->fused_epi ? 1 : 0;
        if (s->fused_epi) {
            float *next = s->d_res[s->cur ^ 1] + (size_t)s->rank * s->bstride;
            F.rb_arrive = s->d_rb_arrive; F.rb_sums = s->d_rb_sums; F.done = s->d_done;
            F.M = s->d_M; F.mat = s->d_mat; F.B = s->d_B;
            F.res_out_block = next; F.block_sums = reinterpret_cast<double *>(next + s->sums_off);
            F.seq = s->seq; F.flags = s->d_flags; F.host_abort = s->d_abort_host; F.G = s->G;
            F.wait_seq = wait_seq; F.timeout_ns = s->timeout_ns;
            F.restart = restart ? 1 : 0; F.E_block = s->d_E + (size_t)s->rank * s->bstride;
            if (s->fused) {
                F.npeers = s->G;
                for (int g = 0; g < s->G; g++) {
                    float *blk = s->peer_res[s->cur ^ 1][g] + (size_t)s->rank * s->bstride;
                    F.peer_out[g] = blk;
                    F.peer_sums[g] = reinterpret_cast<double *>(blk + s->sums_off);
                    F.peer_flag[g] = s->peer_flags[g] + s->rank;
                }
            }
        }
        {
            // chained single-GPU passes: programmatic dependent launch lets this grid move onto SMs as the previous pass leaves
            // them and stream its first F tiles meanwhile (the kernel waits for the previous grid before it touches anything
            // a pass writes).  Multi-GPU passes keep plain stream order (their abort marker is read at kernel start).  A device
            // converge always chains on one GPU.
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((TmaCfg<K>::NCW + 3) * 32); cfg.dynamicSmemBytes = smem; cfg.stream = c->stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = at;
            cfg.numAttrs = (s->fused_epi && (s->chained || stop) && s->G == 1) ? 1 : 0;
            DZ_CUDA(cudaLaunchKernelEx(&cfg, kern, P, s->tmF, s->tmRes[s->cur], F));
        }
        DZ_CUDA(cudaGetLastError());
        if (s->fused_epi) return DAISY_OK; // the whole pass was that one launch
        rc = DAISY_OK;
    } else if constexpr (K <= 9) {
        rc = (s->R == 8) ? launch_partial<K, 8>(s, P) : launch_partial<K, 4>(s, P);
    } else {
        rc = (s->R == 4) ? launch_partial<K, 4>(s, P) : launch_partial<K, 2>(s, P);
    }
    if (rc) return rc;
    EpiParams E;
    float *next = s->d_res[s->cur ^ 1] + (size_t)s->rank * s->bstride;
    E.partial = s->d_partial; E.nsplit = s->nsplit; E.nloc = s->nloc; E.n = s->n;
    E.M = s->d_M; E.mat = s->d_mat; E.res_out_block = next; E.B = s->d_B;
    E.cta_sums = s->d_cta_sums; E.block_sums = reinterpret_cast<double *>(next + s->sums_off); E.done = s->d_done;
    E.npeers = 0; E.seq = s->seq; E.abort_marker = s->fused ? s->d_flags + 16 : nullptr;
    E.stop_state = P.stop.state;
    E.restart = restart ? 1 : 0; E.E_block = s->d_E + (size_t)s->rank * s->bstride;
    if (s->fused) {
        E.npeers = s->G;
        for (int g = 0; g < s->G; g++) {
            float *blk = s->peer_res[s->cur ^ 1][g] + (size_t)s->rank * s->bstride;
            E.peer_out[g] = blk;
            E.peer_sums[g] = reinterpret_cast<double *>(blk + s->sums_off);
            E.peer_flag[g] = s->peer_flags[g] + s->rank;
        }
    }
    int egrid = (s->nloc + 255) / 256;
    if (egrid > 148) egrid = 148;
    if (egrid < 1) egrid = 1;
    if (s->abs_sums) k_gather_epilogue<K, true><<<egrid, 256, 0, c->stream>>>(E);
    else k_gather_epilogue<K, false><<<egrid, 256, 0, c->stream>>>(E);
    DZ_CUDA(cudaGetLastError());
    return DAISY_OK;
}

static int scan_and_plan(daisy_solver *s);

static int launch_pass(daisy_solver *s, unsigned long long wait_seq = 0ull, const DevStop *stop = nullptr, bool restart = false) {
    if (s->skip && s->scanned_version != s->ctx->F_version) { // F was written since the last scan (a host integer compare per pass)
        int rc = scan_and_plan(s);
        if (rc) return rc;
    }
    switch (s->Kp) {
    case 1: return launch_pass_K<1>(s, wait_seq, stop, restart);
    case 3: return launch_pass_K<3>(s, wait_seq, stop, restart);
    case 9: return launch_pass_K<9>(s, wait_seq, stop, restart);
    case 16: return launch_pass_K<16>(s, wait_seq, stop, restart);
    case 32: return launch_pass_K<32>(s, wait_seq, stop, restart);
    case 64: return launch_pass_K<64>(s, wait_seq, stop, restart);
    }
    daisy_set_error("unsupported padded band count %d", s->Kp);
    return DAISY_E_INVALID;
}

// ---- tensor maps (driver entry point fetched through the runtime; no libcuda link dependency) ------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                    const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled get_encode() {
    static std::once_flag once; // solvers may be created from several host threads
    static PFN_encodeTiled fn = nullptr;
    std::call_once(once, [] {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    });
    return fn;
}

static int make_maps(daisy_solver *s) {
    PFN_encodeTiled enc = get_encode();
    if (!enc) { daisy_set_error("cuTensorMapEncodeTiled is not available from this driver"); return DAISY_E_CUDA; }
    daisy_ctx *c = s->ctx;
    const int trows = (s->Kp == 32) ? 32 : 64, tcols = (s->Kp <= 9) ? 256 : 128; // = tma_rows<Kp>() x TmaCfg<Kp>::COLS
    {
        cuuint64_t dims[2] = { (cuuint64_t)c->ldF, (cuuint64_t)(s->nloc > 0 ? s->nloc : 1) };
        cuuint64_t strides[1] = { (cuuint64_t)c->ldF * 4 };
        cuuint32_t box[2] = { (cuuint32_t)tcols, (cuuint32_t)trows };
        cuuint32_t es[2] = { 1, 1 };
        CUresult r = enc(&s->tmF, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, c->d_F, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { daisy_set_error("cuTensorMapEncodeTiled(F) failed: %d", (int)r); return DAISY_E_CUDA; }
    }
    for (int b = 0; b < 2; b++) {
        cuuint64_t dims[3] = { (cuuint64_t)s->n, (cuuint64_t)s->Kp, (cuuint64_t)s->G };
        cuuint64_t strides[2] = { (cuuint64_t)s->n * 4, (cuuint64_t)s->bstride * 4 };
        cuuint32_t box[3] = { (cuuint32_t)tcols, (cuuint32_t)s->Kp, 1 };
        cuuint32_t es[3] = { 1, 1, 1 };
        CUresult r = enc(&s->tmRes[b], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, s->d_res[b], dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { daisy_set_error("cuTensorMapEncodeTiled(residual) failed: %d", (int)r); return DAISY_E_CUDA; }
    }
    if (s->use_mma) {
        {
            cuuint64_t dims[2] = { (cuuint64_t)c->ldF, (cuuint64_t)(s->nloc > 0 ? s->nloc : 1) };
            cuuint64_t strides[1] = { (cuuint64_t)c->ldF * 4 };
            cuuint32_t box[2] = { MM_SUB, MM_ROWS };
            cuuint32_t es[2] = { 1, 1 };
            CUresult r = enc(&s->tmFmma, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, c->d_F, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) { daisy_set_error("cuTensorMapEncodeTiled(F, swizzled) failed: %d", (int)r); return DAISY_E_CUDA; }
        }
        {
            cuuint64_t dims[2] = { (cuuint64_t)s->ncolsP, (cuuint64_t)(2 * s->Kp) };
            cuuint64_t strides[1] = { (cuuint64_t)s->ncolsP * 4 };
            cuuint32_t box[2] = { MM_SUB, (cuuint32_t)(2 * s->Kp) };
            cuuint32_t es[2] = { 1, 1 };
            CUresult r = enc(&s->tmSplit, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, s->d_split, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) { daisy_set_error("cuTensorMapEncodeTiled(split residual) failed: %d", (int)r); return DAISY_E_CUDA; }
        }
    }
    return DAISY_OK;
}

// L2 residency (GatherParams::pin16) for a pass that streams fbytes of F: keep ~45 % of the L2 filled with F tiles that are read
// again next pass; the rest of the matrix streams through evict_first (which by itself is worth 9 % on the 164 MB matrix: the
// stream no longer pushes the residual vectors out).  Measured on the reference's scenes (164 / 238 MB): best at 61 / 45 MB
// pinned, worse from ~70 MB on (the two L2 halves mirror lines read from both dies).  DAISY_GATHER_PIN16 = 0..16 overrides.
static int pin16_for(const daisy_solver *s, double fbytes) {
    int l2 = 0;
    cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, s->ctx->device);
    int p16 = fbytes > 0.0 ? (int)floor(16.0 * 0.45 * (double)l2 / fbytes) : 0;
    if (p16 > 16) p16 = 16;
    if (p16 < 0) p16 = 0;
    const char *e3 = getenv("DAISY_GATHER_PIN16");
    if (e3) { p16 = atoi(e3); if (p16 < 0) p16 = 0; if (p16 > 16) p16 = 16; }
    return p16;
}

// choose rows-per-warp and the column split so that (row blocks x splits) fills the persistent grid evenly
static void plan(daisy_solver *s) {
    int sms = s->ctx->num_sms;
    s->grid = sms;
    const char *env = getenv("DAISY_GATHER");
    s->use_tma = !(env && strcmp(env, "ldg") == 0);
    // wide band counts run on the tensor cores unless DAISY_GATHER=fp32 (or ldg) asks for the CUDA-core kernels (K <= 32 only:
    // daisy_solver_create refuses those for more bands)
    s->use_mma = s->use_tma && s->Kp >= 16 && !(env && strcmp(env, "fp32") == 0);
    {
        const char *e2 = getenv("DAISY_GATHER_EPI"); // "split": keep the separate epilogue kernel (A/B switch)
        s->fused_epi = s->use_tma && !s->use_mma && !(e2 && strcmp(e2, "split") == 0);
        const char *e4 = getenv("DAISY_GATHER_SKIP"); // "0": stream every tile of F (the dense plan, A/B switch)
        s->skip = s->fused_epi && s->Kp <= 9 && !(e4 && strcmp(e4, "0") == 0);
    }
    int Rs[2];
    if (s->use_mma) { Rs[0] = Rs[1] = MM_ROWS / G_WARPS; } // 128-row tiles
    else if (s->use_tma) { Rs[0] = Rs[1] = (s->Kp == 32 ? 4 : 8); } // rows per block / G_WARPS: 64-row tiles, 32-row for K=32
    else if (s->Kp <= 9) { Rs[0] = 8; Rs[1] = 4; } else { Rs[0] = 2; Rs[1] = 4; }
    int ncols = s->G * s->n;
    // keep at least 2048 columns per item -- 1024 with the fused epilogue, where a split costs one partial row per block and no
    // extra launch: small matrices (the reference's own scenes: ~120 row blocks) then fill the 148 SMs evenly
    const int mincols = s->fused_epi ? 2 * G_TC : 4 * G_TC;
    int maxsplit = (ncols + mincols - 1) / mincols;
    if (maxsplit < 1) maxsplit = 1;
    if (maxsplit > 32) maxsplit = 32;
    double best = -1.0;
    for (int ri = 0; ri < 2; ri++) {
        int R = Rs[ri];
        int nrb = (s->nloc + G_WARPS * R - 1) / (G_WARPS * R);
        for (int sp = 1; sp <= maxsplit; sp++) {
            long items = (long)nrb * sp;
            long rounds = (items + sms - 1) / sms;
            double eff = (double)items / (double)(rounds * sms);
            eff -= 0.004 * (sp - 1) + (ri == 1 ? 0.02 : 0.0); // prefer fewer splits and the first R on ties
            if (eff > best) { best = eff; s->R = R; s->nsplit = sp; }
        }
    }
    int colw = (ncols + s->nsplit - 1) / s->nsplit;
    s->colw = ((colw + G_TC - 1) / G_TC) * G_TC; // multiple of 512 columns (and of the 128-column TMA step)
    s->nsplit = (ncols + s->colw - 1) / s->colw;
    // column steps of a row block of k_gather_tma, whatever the plan: every step a piece streams lies below it (piece_step)
    const int tcols = (s->Kp <= 9) ? 256 : 128; // = TmaCfg<Kp>::COLS
    s->sk_S = (ncols + tcols - 1) / tcols;
    if (s->fused_epi) {
        // stream-K: the (row block, column step) sequence cut into one contiguous, equally long range per SM
        const int trows = (s->Kp == 32) ? 32 : 64; // = tma_rows<Kp>()
        // a rank that owns no rows (the last ranks of a partition whose blocks are rounded up to 256) still gets one row block
        // over zero rows: only the epilogue of a pass's last row block publishes the rank's band sums and raises its flag,
        // which every peer's next pass waits for
        const int nrb = s->nloc > 0 ? (s->nloc + trows - 1) / trows : 1;
        s->sk_total = nrb * s->sk_S;
        s->sk_grid = s->sk_total < sms ? (s->sk_total > 0 ? s->sk_total : 1) : sms;
        s->sk_L = (s->sk_total + s->sk_grid - 1) / s->sk_grid;
        if (s->sk_L < 1) s->sk_L = 1;
        s->sk_maxp = s->sk_S / s->sk_L + 2;
        s->pin16 = pin16_for(s, (double)s->nloc * (double)ncols * 4.0); // tile skipping rebases it on the occupied tiles
    }
}

// ---- tile skipping ------------------------------------------------------------------------------------------------
// occ[rb * S + s] = 1 iff tile (rb, s) -- rows [rb T_ROWS, +T_ROWS) x columns [s T_COLS, +T_COLS), clipped to the nloc x ldF
// extent the F tensor map covers, i.e. exactly what the producer would load -- holds an entry whose bits other than the sign
// are not all zero (NaN and Inf tiles are kept).  One CTA per tile, 4 rows x 256 columns per load.
__global__ void __launch_bounds__(256) k_tile_scan(const float *F, int64_t ldF, int nloc, int trows, int tcols, int S, unsigned char *occ) {
    const int s = blockIdx.x, rb = blockIdx.y, lanes = tcols / 4;
    const int64_t col = (int64_t)s * tcols + (threadIdx.x % lanes) * 4;
    const int r1 = min(nloc, (rb + 1) * trows);
    unsigned any = 0u;
    if (col < ldF) // ldF is a multiple of 32: a float4 is either inside or outside
        for (int r = rb * trows + (int)threadIdx.x / lanes; r < r1; r += 256 / lanes) {
            const float4 v = ldg_stream(F + (size_t)r * ldF + col);
            any |= (__float_as_uint(v.x) | __float_as_uint(v.y) | __float_as_uint(v.z) | __float_as_uint(v.w)) & 0x7fffffffu;
        }
    any = __syncthreads_or(any != 0u);
    if (threadIdx.x == 0) occ[(size_t)rb * S + s] = any ? 1 : 0;
}

// the compacted stream-K plan over the occupied tiles of an nrb x S map: the entries of every row block in column order, a
// row block without an occupied tile gets one null entry (-1: nothing streamed, its epilogue still runs)
struct SkipPlan {
    std::vector<int> list, off;
    int total = 0, grid = 1, L = 0, maxp = 1;
    int64_t occupied = 0;
};
static void build_skip_plan(const unsigned char *occ, int nrb, int S, int sms, SkipPlan &sp) {
    sp.list.clear();
    sp.off.assign((size_t)nrb + 1, 0);
    sp.occupied = 0;
    for (int rb = 0; rb < nrb; rb++) {
        sp.off[(size_t)rb] = (int)sp.list.size();
        for (int st = 0; st < S; st++)
            if (occ[(size_t)rb * S + st]) sp.list.push_back(st);
        sp.occupied += (int64_t)sp.list.size() - sp.off[(size_t)rb];
        if ((int)sp.list.size() == sp.off[(size_t)rb]) sp.list.push_back(-1);
    }
    sp.off[(size_t)nrb] = (int)sp.list.size();
    sp.total = (int)sp.list.size();
    sp.grid = sp.total < sms ? (sp.total > 0 ? sp.total : 1) : sms;
    sp.L = sp.total > 0 ? (sp.total + sp.grid - 1) / sp.grid : 1;
    sp.maxp = 1;
    for (int rb = 0; rb < nrb; rb++) {
        const int np = sk_owner(sp.off[(size_t)rb + 1] - 1, sp.total, sp.grid) - sk_owner(sp.off[(size_t)rb], sp.total, sp.grid) + 1;
        if (np > sp.maxp) sp.maxp = np;
    }
}

// scan F, rebuild the plan and upload it.  Runs at solver creation and before the first pass after F changed.
static int scan_and_plan(daisy_solver *s) {
    daisy_ctx *c = s->ctx;
    const int trows = 64, tcols = 256; // = tma_rows<K>() x TmaCfg<K>::COLS for K <= 9
    const int nrb = s->nrb_tma, S = s->sk_S; // a rank without rows: one row block, whose null entry runs the epilogue (plan())
    cudaStream_t st = c->stream;
    s->occ.assign((size_t)nrb * S, 0);
    if (s->nloc > 0 && S > 0) {
        unsigned char *d_occ = nullptr;
        cudaEvent_t t0 = nullptr, t1 = nullptr;
        int rc = DAISY_OK;
        auto ok = [&](cudaError_t e, const char *what) {
            if (e != cudaSuccess && !rc) { daisy_set_error("tile scan: %s -> %s", what, cudaGetErrorString(e)); rc = DAISY_E_CUDA; }
            return rc == DAISY_OK;
        };
        if (ok(cudaMalloc(&d_occ, s->occ.size()), "cudaMalloc") && ok(cudaEventCreate(&t0), "cudaEventCreate") && ok(cudaEventCreate(&t1), "cudaEventCreate") &&
            ok(cudaEventRecord(t0, st), "cudaEventRecord")) {
            k_tile_scan<<<dim3((unsigned)S, (unsigned)nrb), 256, 0, st>>>(c->d_F, c->ldF, s->nloc, trows, tcols, S, d_occ);
            if (ok(cudaGetLastError(), "k_tile_scan") && ok(cudaEventRecord(t1, st), "cudaEventRecord") &&
                ok(cudaMemcpyAsync(s->occ.data(), d_occ, s->occ.size(), cudaMemcpyDeviceToHost, st), "cudaMemcpyAsync") &&
                ok(cudaStreamSynchronize(st), "cudaStreamSynchronize")) {
                float ms = 0.f;
                if (ok(cudaEventElapsedTime(&ms, t0, t1), "cudaEventElapsedTime")) s->scan_ms = ms;
            }
        }
        if (t0) cudaEventDestroy(t0);
        if (t1) cudaEventDestroy(t1);
        cudaFree(d_occ);
        if (rc) return rc;
    }
    SkipPlan sp;
    build_skip_plan(s->occ.data(), nrb, S, c->num_sms, sp);
    // the stream is idle here (synchronised above): no pass can still read the arrays about to be replaced
    if ((int64_t)sp.list.size() > s->sk_list_cap) {
        cudaFree(s->d_sk_list); s->d_sk_list = nullptr; s->sk_list_cap = 0;
        DZ_CUDA(cudaMalloc(&s->d_sk_list, sizeof(int) * sp.list.size()));
        s->sk_list_cap = (int64_t)sp.list.size();
    }
    if (!s->d_sk_off) DZ_CUDA(cudaMalloc(&s->d_sk_off, sizeof(int) * ((size_t)nrb + 1)));
    if (sp.maxp > s->partial_splits) {
        cudaFree(s->d_partial); s->d_partial = nullptr; s->partial_splits = 0;
        DZ_CUDA(cudaMalloc(&s->d_partial, sizeof(float) * (size_t)sp.maxp * (s->nloc > 0 ? s->nloc : 1) * s->Kp));
        s->partial_splits = sp.maxp;
    }
    DZ_CUDA(cudaMemcpyAsync(s->d_sk_list, sp.list.data(), sizeof(int) * sp.list.size(), cudaMemcpyHostToDevice, st));
    DZ_CUDA(cudaMemcpyAsync(s->d_sk_off, sp.off.data(), sizeof(int) * sp.off.size(), cudaMemcpyHostToDevice, st));
    DZ_CUDA(cudaStreamSynchronize(st)); // `sp` is pageable host memory
    s->sk_total = sp.total; s->sk_grid = sp.grid; s->sk_L = sp.L; s->sk_maxp = sp.maxp;
    s->occupied = sp.occupied;
    s->pin16 = pin16_for(s, (double)sp.occupied * trows * tcols * 4.0); // the bytes a pass actually streams
    s->scanned_version = c->F_version;
    return DAISY_OK;
}

// ---------------------------------------------------------------------------------------------------------
static int padded_K(int K) { return K <= 1 ? 1 : K <= 3 ? 3 : K <= 9 ? 9 : K <= 16 ? 16 : K <= 32 ? 32 : 64; }

static void free_solver(daisy_solver *s) {
    if (!s) return;
    if (s->fused && s->peers_ipc)
        for (int g = 0; g < s->G; g++) {
            if (g == s->rank) continue;
            if (s->peer_res[0][g]) cudaIpcCloseMemHandle(s->peer_res[0][g]);
            if (s->peer_res[1][g]) cudaIpcCloseMemHandle(s->peer_res[1][g]);
            if (s->peer_flags[g]) cudaIpcCloseMemHandle(s->peer_flags[g]);
        }
    cudaFree(s->d_flags);
    cudaFree(s->d_res[0]); cudaFree(s->d_res[1]); cudaFree(s->d_B); cudaFree(s->d_E); cudaFree(s->d_M); cudaFree(s->d_mat);
    cudaFree(s->d_partial); cudaFree(s->d_cta_sums); cudaFree(s->d_done); cudaFree(s->d_split);
    cudaFree(s->d_rb_arrive); cudaFree(s->d_rb_sums);
    cudaFree(s->d_sk_list); cudaFree(s->d_sk_off);
    cudaFree(s->d_stop);
    if (s->h_stop) cudaFreeHost(s->h_stop);
    if (s->h_abort) cudaFreeHost(s->h_abort);
    if (s->e0) cudaEventDestroy(s->e0);
    if (s->e1) cudaEventDestroy(s->e1);
    delete s;
}

// host (K x N band-major) -> exchange layout (G blocks of [Kp x n] + tail)
static void to_exchange(const daisy_solver *s, const float *src, std::vector<float> &dst) {
    dst.assign((size_t)s->G * s->bstride, 0.0f);
    for (int k = 0; k < s->K; k++)
        for (int p = 0; p < s->N; p++) {
            int g = p / s->n, jl = p - g * s->n;
            dst[(size_t)g * s->bstride + (size_t)k * s->n + jl] = src[(size_t)k * s->N + p];
        }
}

// FP64 sum of n floats with eight independent partial sums (fixed order, so deterministic): a single dependent chain costs
// 1 ns per element, which was 1.2 of the 1.5 ms a host-buffer step spent outside the pass at 131072 patches x 9 bands
static double host_sum(const float *x, size_t n) {
    double a[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
    size_t i = 0;
    for (; i + 8 <= n; i += 8)
        for (int j = 0; j < 8; j++) a[j] += (double)x[i + j];
    for (int j = 0; i < n; i++, j++) a[j] += (double)x[i];
    return ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
}

// M (nmat x K x K column-major) padded to Kp x Kp: the extra bands are inert (zero rows and columns)
static void pad_materials(const daisy_solver *s, const float *M, int nmat, std::vector<float> &Mp) {
    Mp.assign((size_t)nmat * s->Kp * s->Kp, 0.0f);
    for (int m = 0; m < nmat; m++)
        for (int j = 0; j < s->K; j++)
            for (int i = 0; i < s->K; i++) Mp[((size_t)m * s->Kp + j) * s->Kp + i] = M[((size_t)m * s->K + j) * s->K + i];
}

static int compute_sums_from_host(daisy_solver *s, const float *res /* K x N */) {
    // band sums of a residual supplied by the host (reset / write): same quantity the kernels total on device
    s->sums.assign(s->K, 0.0);
    for (int k = 0; k < s->K; k++) s->sums[k] = host_sum(res + (size_t)k * s->N, (size_t)s->N);
    return DAISY_OK;
}

extern "C" int daisy_solver_create(daisy_ctx *ctx, int K, const float *E, const float *M, int nmat, const int32_t *mat_idx,
                                   daisy_solver **out) {
    DZ_REQUIRE(ctx && out && E && M && mat_idx, DAISY_E_INVALID, "daisy_solver_create: null argument");
    DZ_REQUIRE(K >= 1 && K <= DAISY_MAX_BANDS, DAISY_E_INVALID,
               "daisy_solver_create: K must be in [1,64] (kernels for 1, 3, 9, 16, 32 and 64 bands, K padded up to the next)");
    {
        const char *env = getenv("DAISY_GATHER");
        DZ_REQUIRE(K <= 32 || !(env && (strcmp(env, "fp32") == 0 || strcmp(env, "ldg") == 0)), DAISY_E_INVALID,
                   "daisy_solver_create: K > 32 runs only on the tensor-core kernel; DAISY_GATHER=fp32 / ldg has no kernel for it");
    }
    DZ_REQUIRE(nmat >= 1, DAISY_E_INVALID, "daisy_solver_create: need at least one material");
    DZ_REQUIRE(ctx->have_F, DAISY_E_STATE, "daisy_solver_create: build or load the form factors first");
    DZ_REQUIRE(ctx->N > 0, DAISY_E_INVALID, "daisy_solver_create: empty mesh");
    for (int p = 0; p < ctx->N; p++)
        DZ_REQUIRE(mat_idx[p] >= 0 && mat_idx[p] < nmat, DAISY_E_INVALID, "daisy_solver_create: material index out of range");
    DZ_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    daisy_solver *s = new daisy_solver();
    s->ctx = ctx; s->mesh_version = ctx->mesh_version; s->K = K; s->Kp = padded_K(K); s->nmat = s->nmat_cap = nmat;
    s->N = ctx->N; s->n = ctx->rows_per_rank; s->G = ctx->nranks; s->rank = ctx->rank;
    s->row0 = ctx->row0; s->nloc = ctx->row1 - ctx->row0;
    int64_t body = (int64_t)s->Kp * s->n;
    s->sums_off = body;
    s->bstride = ((body + 2 * s->Kp + 3) / 4) * 4; // K doubles = 2K floats, block padded to 16 B
    plan(s);
    size_t exb = sizeof(float) * (size_t)s->G * s->bstride;
    int rc = DAISY_OK;
#define SC(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { daisy_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); free_solver(s); return DAISY_E_CUDA; } } while (0)
    SC(cudaMalloc(&s->d_res[0], exb));
    SC(cudaMalloc(&s->d_res[1], exb));
    SC(cudaMalloc(&s->d_E, exb));
    SC(cudaMalloc(&s->d_B, sizeof(float) * (size_t)s->Kp * s->n));
    SC(cudaMalloc(&s->d_M, sizeof(float) * (size_t)nmat * s->Kp * s->Kp));
    SC(cudaMalloc(&s->d_mat, sizeof(int) * (size_t)(s->nloc > 0 ? s->nloc : 1)));
    s->partial_splits = s->nsplit > s->sk_maxp ? s->nsplit : s->sk_maxp;
    SC(cudaMalloc(&s->d_partial, sizeof(float) * (size_t)s->partial_splits * (s->nloc > 0 ? s->nloc : 1) * s->Kp));
    SC(cudaMalloc(&s->d_cta_sums, sizeof(double) * 148 * s->Kp));
    SC(cudaMalloc(&s->d_done, sizeof(unsigned int)));
    SC(cudaMemsetAsync(s->d_done, 0, sizeof(unsigned int), st));
    {
        const int trows = (s->Kp == 32) ? 32 : 64; // = tma_rows<Kp>()
        s->nrb_tma = (s->nloc + trows - 1) / trows;
        if (s->nrb_tma < 1) s->nrb_tma = 1; // a rank without rows runs one row block over zero rows (plan())
        SC(cudaMalloc(&s->d_rb_arrive, sizeof(unsigned int) * (size_t)s->nrb_tma));
        SC(cudaMemsetAsync(s->d_rb_arrive, 0, sizeof(unsigned int) * (size_t)s->nrb_tma, st));
        SC(cudaMalloc(&s->d_rb_sums, sizeof(double) * (size_t)s->nrb_tma * s->Kp));
        SC(cudaHostAlloc(reinterpret_cast<void **>(&s->h_abort), sizeof(unsigned long long), cudaHostAllocMapped));
        *s->h_abort = 0ull;
        SC(cudaHostGetDevicePointer(reinterpret_cast<void **>(&s->d_abort_host), s->h_abort, 0));
        const char *e = getenv("DAISY_EXCHANGE_TIMEOUT_MS");
        if (e && atof(e) > 0.0) s->timeout_ns = (unsigned long long)(atof(e) * 1e6);
    }
    SC(cudaMalloc(&s->d_flags, sizeof(unsigned long long) * 17));
    SC(cudaMemsetAsync(s->d_flags, 0, sizeof(unsigned long long) * 17, st));
    SC(cudaMemsetAsync(s->d_res[0], 0, exb, st));
    SC(cudaMemsetAsync(s->d_res[1], 0, exb, st));
    SC(cudaEventCreate(&s->e0));
    SC(cudaEventCreate(&s->e1));
    if (s->use_mma) {
        s->ncolsP = ((s->G * s->n + 63) / 64) * 64;
        SC(cudaMalloc(&s->d_split, sizeof(float) * (size_t)2 * s->Kp * s->ncolsP));
    }
    if (s->use_tma) { int mrc = make_maps(s); if (mrc) { free_solver(s); return mrc; } }
    {
        std::vector<float> ex, Mp;
        to_exchange(s, E, ex);
        SC(cudaMemcpyAsync(s->d_E, ex.data(), exb, cudaMemcpyHostToDevice, st));
        pad_materials(s, M, nmat, Mp);
        SC(cudaMemcpyAsync(s->d_M, Mp.data(), sizeof(float) * Mp.size(), cudaMemcpyHostToDevice, st));
        if (s->nloc > 0) SC(cudaMemcpyAsync(s->d_mat, mat_idx + s->row0, sizeof(int) * (size_t)s->nloc, cudaMemcpyHostToDevice, st));
        SC(cudaStreamSynchronize(st)); // `ex` and `Mp` are pageable host memory
    }
#undef SC
    if (s->skip) { rc = scan_and_plan(s); if (rc) { free_solver(s); return rc; } }
    compute_sums_from_host(s, E);
    s->e_sums = s->sums;
    *out = s;
    rc = daisy_solver_reset(s);
    if (rc) { free_solver(s); *out = nullptr; }
    return rc;
}

extern "C" void daisy_solver_destroy(daisy_solver *s) {
    if (s && s->ctx) cudaSetDevice(s->ctx->device);
    free_solver(s);
}

extern "C" int daisy_solver_reset(daisy_solver *s) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_reset: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_reset");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    size_t exb = sizeof(float) * (size_t)s->G * s->bstride;
    // fused exchange: a slower rank may still be storing its block of the last pass into this rank's buffers
    if (s->fused && s->seq > 0) {
        k_wait_flags<<<1, 32, 0, st>>>(s->d_flags, s->G, s->seq, s->timeout_ns, s->d_abort_host);
        DZ_CUDA(cudaGetLastError());
    }
    // a pass that gave up on a peer leaves its counters half way and the abort markers set: start clean
    DZ_CUDA(cudaMemsetAsync(s->d_done, 0, sizeof(unsigned int), st));
    DZ_CUDA(cudaMemsetAsync(s->d_rb_arrive, 0, sizeof(unsigned int) * (size_t)s->nrb_tma, st));
    DZ_CUDA(cudaMemsetAsync(s->d_flags + 16, 0, sizeof(unsigned long long), st));
    if (s->h_abort) *s->h_abort = 0ull;
    // residualvector = emission; lightningvalues = emission                                 Lightning.h:159-165
    s->cur = 0;
    DZ_CUDA(cudaMemcpyAsync(s->d_res[0], s->d_E, exb, cudaMemcpyDeviceToDevice, st));
    DZ_CUDA(cudaMemcpyAsync(s->d_B, s->d_E + (size_t)s->rank * s->bstride, sizeof(float) * (size_t)s->Kp * s->n, cudaMemcpyDeviceToDevice, st));
    DZ_CUDA(cudaStreamSynchronize(st));
    s->numpasses = 0;
    s->sums = s->e_sums; // band sums of E (totalled at create and by daisy_solver_set_emission)
    s->sums_valid = true;
    s->abs_sums = false;
    return DAISY_OK;
}

// the passes of daisy_solver_step_local / _step_finish; daisy_solver_step and _step_fused check the solver once per pass
static int step_local(daisy_solver *s) {
    DzRange range_("gather pass");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    if (!s->chained) DZ_CUDA(cudaEventRecord(s->e0, st)); // an event between two passes would keep them from overlapping
    int rc = launch_pass(s);
    if (rc) return rc;
    if (!s->chained) DZ_CUDA(cudaEventRecord(s->e1, st));
    s->events_recorded = !s->chained;
    return DAISY_OK;
}

extern "C" int daisy_solver_set_chained(daisy_solver *s, int on) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_set_chained: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_set_chained");
    s->chained = on != 0;
    return DAISY_OK;
}

extern "C" int daisy_solver_exchange_info(daisy_solver *s, void **d_next_buffer, int64_t *block_bytes, int64_t *total_bytes) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_exchange_info: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_exchange_info");
    if (d_next_buffer) *d_next_buffer = s->d_res[s->cur ^ 1];
    if (block_bytes) *block_bytes = (int64_t)sizeof(float) * s->bstride;
    if (total_bytes) *total_bytes = (int64_t)sizeof(float) * s->bstride * s->G;
    return DAISY_OK;
}

static int fetch_sums(daisy_solver *s) {
    // per-rank partial band sums sit in the tail of every block of the current buffer
    cudaStream_t st = s->ctx->stream;
    unsigned long long timed_out = 0;
    if (s->fused) {
        k_wait_flags<<<1, 32, 0, st>>>(s->d_flags, s->G, s->seq, s->timeout_ns, s->d_abort_host); // every rank's block of the last pass has landed
        DZ_CUDA(cudaGetLastError());
        DZ_CUDA(cudaMemcpyAsync(&timed_out, s->d_flags + 16, sizeof(timed_out), cudaMemcpyDeviceToHost, st));
    }
    std::vector<double> tails((size_t)s->G * s->Kp);
    for (int g = 0; g < s->G; g++)
        DZ_CUDA(cudaMemcpyAsync(&tails[(size_t)g * s->Kp], s->d_res[s->cur] + (size_t)g * s->bstride + s->sums_off,
                                sizeof(double) * s->Kp, cudaMemcpyDeviceToHost, st));
    DZ_CUDA(cudaStreamSynchronize(st));
    if (timed_out) {
        daisy_set_error("fused exchange: a peer's block of pass %llu did not arrive within %.1f s; the solver is stopped until daisy_solver_reset",
                        timed_out, (double)s->timeout_ns * 1e-9);
        return DAISY_E_STATE;
    }
    float ms = 0.f;
    if (s->events_recorded) {
        if (cudaEventElapsedTime(&ms, s->e0, s->e1) == cudaSuccess) s->last_ms = ms;
        else cudaGetLastError(); // not an error of this call's work: do not leave it for the next cudaGetLastError()
    }
    s->sums.assign(s->K, 0.0);
    for (int k = 0; k < s->K; k++) {
        double v = 0.0;
        for (int g = 0; g < s->G; g++) v += tails[(size_t)g * s->Kp + k];
        s->sums[k] = v;
    }
    s->sums_valid = true;
    return DAISY_OK;
}

// band_sums == NULL: nothing is read back and the call does not wait for the device (back-to-back passes);
// the sums are fetched lazily by daisy_solver_band_sums / daisy_solver_converge.
static int step_finish(daisy_solver *s, double *band_sums) {
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    s->cur ^= 1;
    s->numpasses++;
    s->sums_valid = false;
    if (!band_sums) return DAISY_OK;
    int rc = fetch_sums(s);
    if (rc) return rc;
    memcpy(band_sums, s->sums.data(), sizeof(double) * s->K);
    return DAISY_OK;
}

extern "C" int daisy_solver_step_local(daisy_solver *s) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_step_local: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_step_local");
    return step_local(s);
}

extern "C" int daisy_solver_step_finish(daisy_solver *s, double *band_sums) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_step_finish: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_step_finish");
    return step_finish(s, band_sums);
}

extern "C" int daisy_solver_step(daisy_solver *s, double *band_sums) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_step: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_step");
    DZ_REQUIRE(s->G == 1, DAISY_E_STATE, "daisy_solver_step: partitioned solver needs step_local / exchange / step_finish");
    int rc = step_local(s);
    if (rc) return rc;
    return step_finish(s, band_sums);
}

// ---- fused exchange over peer memory (multi-GPU, one process per GPU) ------------------------------------------
extern "C" int daisy_solver_ipc_handles(daisy_solver *s, void *handles192) {
    DZ_REQUIRE(s && handles192, DAISY_E_INVALID, "daisy_solver_ipc_handles: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_ipc_handles");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaIpcMemHandle_t h[3];
    DZ_CUDA(cudaIpcGetMemHandle(&h[0], s->d_res[0]));
    DZ_CUDA(cudaIpcGetMemHandle(&h[1], s->d_res[1]));
    DZ_CUDA(cudaIpcGetMemHandle(&h[2], s->d_flags));
    memcpy(handles192, h, sizeof(h));
    return DAISY_OK;
}

extern "C" int daisy_solver_set_peers(daisy_solver *s, const void *handles, int nranks) {
    DZ_REQUIRE(s && handles, DAISY_E_INVALID, "daisy_solver_set_peers: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_set_peers");
    DZ_REQUIRE(nranks == s->G && nranks <= 16, DAISY_E_INVALID, "daisy_solver_set_peers: nranks must match the partition (<= 16)");
    DZ_REQUIRE(!s->fused, DAISY_E_STATE, "daisy_solver_set_peers: peers already set");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    for (int g = 0; g < nranks; g++) {
        if (g == s->rank) { s->peer_res[0][g] = s->d_res[0]; s->peer_res[1][g] = s->d_res[1]; s->peer_flags[g] = s->d_flags; continue; }
        cudaIpcMemHandle_t h[3];
        memcpy(h, (const char *)handles + (size_t)g * sizeof(h), sizeof(h));
        void *p0 = nullptr, *p1 = nullptr, *p2 = nullptr;
        DZ_CUDA(cudaIpcOpenMemHandle(&p0, h[0], cudaIpcMemLazyEnablePeerAccess));
        DZ_CUDA(cudaIpcOpenMemHandle(&p1, h[1], cudaIpcMemLazyEnablePeerAccess));
        DZ_CUDA(cudaIpcOpenMemHandle(&p2, h[2], cudaIpcMemLazyEnablePeerAccess));
        s->peer_res[0][g] = (float *)p0; s->peer_res[1][g] = (float *)p1; s->peer_flags[g] = (unsigned long long *)p2;
    }
    s->fused = true;
    s->peers_ipc = true;
    return DAISY_OK;
}

int dz_solver_get_buffers(daisy_solver *s, float **res0, float **res1, unsigned long long **flags) {
    *res0 = s->d_res[0]; *res1 = s->d_res[1]; *flags = s->d_flags;
    return DAISY_OK;
}

int dz_solver_set_peer_pointers(daisy_solver *s, float *const *res0, float *const *res1, unsigned long long *const *flags, int nranks) {
    DZ_REQUIRE(s && res0 && res1 && flags, DAISY_E_INVALID, "solver_set_peer_pointers: null argument");
    DZ_REQUIRE(nranks == s->G && nranks <= 16, DAISY_E_INVALID, "solver_set_peer_pointers: nranks must match the partition (<= 16)");
    DZ_REQUIRE(!s->fused, DAISY_E_STATE, "solver_set_peer_pointers: peers already set");
    for (int g = 0; g < nranks; g++) { s->peer_res[0][g] = res0[g]; s->peer_res[1][g] = res1[g]; s->peer_flags[g] = flags[g]; }
    s->fused = true;
    s->peers_ipc = false;
    return DAISY_OK;
}

// ---- slice upload for the fused exchange: every rank uploads ONLY its own rows of B and of the residual; the residual slice
// (with its band sums) is then handed to every rank over NVLink exactly like the output of a pass -- block `rank` of every
// rank's next buffer, flag[rank] = new pass number -- so the next pass finds the whole vector in place.
__global__ void k_raise_flags(int npeers, unsigned long long seq, const unsigned long long *abort_marker, unsigned long long *f0, unsigned long long *f1,
                              unsigned long long *f2, unsigned long long *f3, unsigned long long *f4, unsigned long long *f5, unsigned long long *f6,
                              unsigned long long *f7, unsigned long long *f8, unsigned long long *f9, unsigned long long *f10, unsigned long long *f11,
                              unsigned long long *f12, unsigned long long *f13, unsigned long long *f14, unsigned long long *f15) {
    unsigned long long *f[16] = { f0, f1, f2, f3, f4, f5, f6, f7, f8, f9, f10, f11, f12, f13, f14, f15 };
    const int g = threadIdx.x;
    if (g >= npeers || *reinterpret_cast<const volatile unsigned long long *>(abort_marker) != 0ull) return;
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(f[g]), "l"(seq) : "memory");
}

extern "C" int daisy_solver_write_slices(daisy_solver *s, const float *B_local, const float *residual_local) {
    DZ_REQUIRE(s && B_local && residual_local, DAISY_E_INVALID, "daisy_solver_write_slices: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_write_slices");
    DZ_REQUIRE(s->G == 1 || s->fused, DAISY_E_STATE, "daisy_solver_write_slices: a partitioned solver needs the fused exchange (daisy_solver_set_peers)");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    if (s->G == 1) return daisy_solver_write(s, B_local, residual_local);
    // every rank has finished the last pass (and with it all reads of the buffer about to be overwritten)
    if (s->seq > 0) {
        k_wait_flags<<<1, 32, 0, st>>>(s->d_flags, s->G, s->seq, s->timeout_ns, s->d_abort_host);
        DZ_CUDA(cudaGetLastError());
    }
    const int nxt = s->cur ^ 1;
    float *own = s->d_res[nxt] + (size_t)s->rank * s->bstride;
    if (s->nloc > 0) {
        DZ_CUDA(cudaMemcpy2DAsync(s->d_B, sizeof(float) * s->n, B_local, sizeof(float) * s->nloc, sizeof(float) * s->nloc, s->K, cudaMemcpyHostToDevice, st));
        DZ_CUDA(cudaMemcpy2DAsync(own, sizeof(float) * s->n, residual_local, sizeof(float) * s->nloc, sizeof(float) * s->nloc, s->K, cudaMemcpyHostToDevice, st));
    }
    std::vector<double> tail((size_t)s->Kp, 0.0);
    for (int k = 0; k < s->K; k++) tail[(size_t)k] = host_sum(residual_local + (size_t)k * s->nloc, (size_t)s->nloc);
    DZ_CUDA(cudaMemcpyAsync(own + s->sums_off, tail.data(), sizeof(double) * s->Kp, cudaMemcpyHostToDevice, st));
    DZ_CUDA(cudaStreamSynchronize(st)); // `tail` is pageable host memory
    for (int g = 0; g < s->G; g++) {
        if (g == s->rank) continue;
        DZ_CUDA(cudaMemcpyAsync(s->peer_res[nxt][g] + (size_t)s->rank * s->bstride, own, sizeof(float) * (size_t)s->bstride, cudaMemcpyDeviceToDevice, st));
    }
    s->seq++;
    unsigned long long *f[16];
    for (int g = 0; g < 16; g++) f[g] = (g < s->G) ? s->peer_flags[g] + s->rank : nullptr;
    k_raise_flags<<<1, 32, 0, st>>>(s->G, s->seq, s->d_flags + 16, f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7], f[8], f[9], f[10], f[11], f[12],
                                    f[13], f[14], f[15]);
    DZ_CUDA(cudaGetLastError());
    s->cur = nxt;
    s->sums_valid = false;
    s->abs_sums = false;
    return DAISY_OK;
}

// one pass with the exchange fused into the epilogue kernel: wait for the blocks of the previous pass, gather, store
// this rank's new block into every rank's next buffer and raise the flags.  No host synchronisation, no NCCL call.
extern "C" int daisy_solver_step_fused(daisy_solver *s, double *band_sums) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_step_fused: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_step_fused");
    DZ_REQUIRE(s->fused, DAISY_E_STATE, "daisy_solver_step_fused: call daisy_solver_set_peers first");
    DzRange range_("gather pass + fused exchange");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    if (s->h_abort && *reinterpret_cast<volatile unsigned long long *>(s->h_abort) != 0ull) {
        daisy_set_error("fused exchange: a peer's block of pass %llu did not arrive within %.1f s; the solver is stopped until daisy_solver_reset",
                        *s->h_abort, (double)s->timeout_ns * 1e-9);
        return DAISY_E_STATE;
    }
    DZ_CUDA(cudaEventRecord(s->e0, st));
    const unsigned long long wait_seq = s->seq; // the blocks of the previous pass (0: first pass, nothing to wait for)
    s->seq++;
    int rc = launch_pass(s, wait_seq);
    if (rc) return rc;
    DZ_CUDA(cudaEventRecord(s->e1, st));
    s->events_recorded = true;
    return step_finish(s, band_sums);
}

static bool unconverged(const daisy_solver *s, double threshold, int per_band) {
    if (per_band) {
        for (int k = 0; k < s->K; k++) if (s->sums[k] > threshold) return true;
        return false;
    }
    double tot = 0.0;
    for (int k = 0; k < s->K; k++) tot += s->sums[k];
    return tot > threshold;
}

extern "C" int daisy_solver_converge(daisy_solver *s, double threshold, int per_band, int max_passes, int *passes_out) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_converge: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_converge");
    DZ_REQUIRE(s->G == 1, DAISY_E_STATE, "daisy_solver_converge: partitioned solver is driven by the host exchange loop (or daisy_group_solver_converge)");
    DzRange range_("daisy_solver_converge");
    int done = 0;
    std::vector<double> tmp(s->K);
    if (!s->sums_valid) { int rc = fetch_sums(s); if (rc) return rc; }
    while (unconverged(s, threshold, per_band) && (max_passes <= 0 || done < max_passes)) {
        int rc = step_local(s);
        if (!rc) rc = step_finish(s, tmp.data());
        if (rc) return rc;
        done++;
    }
    if (passes_out) *passes_out = s->numpasses;
    return DAISY_OK;
}

// ---- converge with the stop rule on the device ------------------------------------------------------------------------------
// The passes of a call are launched back to back in batches; every pass but the first tests the band sums the previous pass left
// (DevStop) and the pass that finds the residual converged stops the launches behind it.  Between batches the host reads
// {stopped, passes} and the band sums of the last pass through one pinned copy and sizes the next batch so that it most likely
// holds the deciding pass: the criterion (largest band total for per_band, total over bands otherwise) is extrapolated
// geometrically from its ratio over the last batch, plus two launches -- the one that decides and one of margin, since a launch
// that finds `stopped` costs a few microseconds and another batch a host round trip.  The first batch is 4 launches, a batch
// without a contraction to extrapolate doubles, and no batch exceeds 64.
static int ensure_stop_buffers(daisy_solver *s) {
    if (s->d_stop) return DAISY_OK;
    DZ_CUDA(cudaMalloc(&s->d_stop, 2 * sizeof(unsigned int)));
    DZ_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&s->h_stop), sizeof(double) * (1 + (size_t)s->G * s->Kp), cudaHostAllocDefault));
    return DAISY_OK;
}

static double stop_metric(const double *v, int K, int per_band) {
    double m = per_band ? v[0] : 0.0;
    for (int k = 0; k < K; k++) m = per_band ? (v[k] > m ? v[k] : m) : m + v[k];
    return m;
}

static int abort_error(const daisy_solver *s) {
    daisy_set_error("fused exchange: a peer's block of pass %llu did not arrive within %.1f s; the solver is stopped until daisy_solver_reset",
                    *s->h_abort, (double)s->timeout_ns * 1e-9);
    return DAISY_E_STATE;
}

// ss[0 .. n): one solver, or every device's solver of a group (fused exchange), all issued from this thread.  The first pass is
// decided on the host from ss[0]'s sums, as the host loop does.
int dz_converge_device(daisy_solver *const *ss, int n, double threshold, int per_band, int max_passes) {
    daisy_solver *s0 = ss[0];
    for (int i = 0; i < n; i++) {
        daisy_solver *s = ss[i];
        DZ_SOLVER_CURRENT(s, "daisy_solver_converge_device");
        DZ_CUDA(cudaSetDevice(s->ctx->device));
        if (s->fused && s->h_abort && *reinterpret_cast<volatile unsigned long long *>(s->h_abort) != 0ull) return abort_error(s);
        int rc = ensure_stop_buffers(s);
        if (rc) return rc;
    }
    DZ_CUDA(cudaSetDevice(s0->ctx->device));
    if (!s0->sums_valid) { int rc = fetch_sums(s0); if (rc) return rc; }
    if (!unconverged(s0, threshold, per_band)) return DAISY_OK; // nothing launched
    std::vector<int> cur0((size_t)n);
    std::vector<unsigned long long> seq0((size_t)n);
    for (int i = 0; i < n; i++) {
        daisy_solver *s = ss[i];
        DZ_CUDA(cudaSetDevice(s->ctx->device));
        DZ_CUDA(cudaMemsetAsync(s->d_stop, 0, 2 * sizeof(unsigned int), s->ctx->stream));
        cur0[(size_t)i] = s->cur; seq0[(size_t)i] = s->seq;
    }
    const long long budget = max_passes > 0 ? max_passes : (1ll << 62);
    long long issued = 0;
    int batch = 4;
    double m_prev = stop_metric(s0->sums.data(), s0->K, per_band);
    std::vector<double> tot((size_t)s0->K);
    while (true) {
        const int nb = (int)std::min<long long>(batch, budget - issued);
        for (int i = 0; i < n; i++) {
            daisy_solver *s = ss[i];
            cudaStream_t st = s->ctx->stream;
            DZ_CUDA(cudaSetDevice(s->ctx->device));
            for (int j = 0; j < nb; j++) {
                DevStop ds;
                memset(&ds, 0, sizeof(ds));
                ds.state = s->d_stop; ds.rule = (issued + j == 0) ? -1 : (per_band ? 1 : 0); ds.threshold = threshold;
                const unsigned long long wait_seq = s->fused ? s->seq : 0ull;
                if (s->fused) s->seq++;
                int rc = launch_pass(s, wait_seq, &ds);
                if (rc) return rc;
                s->cur ^= 1;
            }
            DZ_CUDA(cudaMemcpyAsync(s->h_stop, s->d_stop, 2 * sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
            if (i == 0) // band sums of the last pass (meaningful only if every pass of the batch ran): the next batch's size
                for (int g = 0; g < s->G; g++)
                    DZ_CUDA(cudaMemcpyAsync(reinterpret_cast<double *>(s->h_stop) + 1 + (size_t)g * s->Kp, s->d_res[s->cur] + (size_t)g * s->bstride + s->sums_off,
                                            sizeof(double) * s->Kp, cudaMemcpyDeviceToHost, st));
        }
        issued += nb;
        for (int i = 0; i < n; i++) {
            DZ_CUDA(cudaSetDevice(ss[i]->ctx->device));
            DZ_CUDA(cudaStreamSynchronize(ss[i]->ctx->stream));
        }
        for (int i = 0; i < n; i++)
            if (ss[i]->fused && *reinterpret_cast<volatile unsigned long long *>(ss[i]->h_abort) != 0ull) return abort_error(ss[i]);
        const unsigned int *state = reinterpret_cast<const unsigned int *>(s0->h_stop);
        if (state[0] || issued >= budget) break;
        const double *tails = reinterpret_cast<const double *>(s0->h_stop) + 1;
        for (int k = 0; k < s0->K; k++) {
            double v = 0.0;
            for (int g = 0; g < s0->G; g++) v += tails[(size_t)g * s0->Kp + k];
            tot[(size_t)k] = v;
        }
        const double m = stop_metric(tot.data(), s0->K, per_band);
        const double r = pow(m / m_prev, 1.0 / nb); // contraction per pass over the last batch
        double est = -1.0;
        if (m > threshold && r > 0.0 && r < 1.0 && std::isfinite(r)) est = ceil(log(threshold / m) / log(r));
        batch = (est >= 0.0 && est < 64.0) ? (int)est + 2 : (est >= 64.0 ? 64 : std::min(2 * nb, 64));
        m_prev = m;
    }
    std::vector<unsigned int> passes((size_t)n);
    for (int i = 0; i < n; i++) passes[(size_t)i] = reinterpret_cast<const unsigned int *>(ss[i]->h_stop)[1];
    for (int i = 0; i < n; i++) {
        daisy_solver *s = ss[i];
        const unsigned int p = passes[(size_t)i];
        s->cur = cur0[(size_t)i] ^ (int)(p & 1u);
        s->numpasses += (int)p;
        if (s->fused) s->seq = seq0[(size_t)i] + p;
        s->sums_valid = false;
        s->events_recorded = false; // no per-pass events: daisy_solver_last_step_ms keeps its value
    }
    for (int i = 1; i < n; i++)
        if (passes[(size_t)i] != passes[0]) {
            daisy_set_error("device converge: device %d ran %u passes, device 0 ran %u", i, passes[(size_t)i], passes[0]);
            return DAISY_E_STATE;
        }
    return DAISY_OK;
}

extern "C" int daisy_solver_converge_device(daisy_solver *s, double threshold, int per_band, int max_passes, int *passes_out) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_converge_device: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_converge_device");
    DZ_REQUIRE(s->G == 1 || s->fused, DAISY_E_STATE, "daisy_solver_converge_device: a partitioned solver needs the fused exchange (daisy_solver_set_peers)");
    DzRange range_("daisy_solver_converge_device");
    int rc = dz_converge_device(&s, 1, threshold, per_band, max_passes);
    if (rc) return rc;
    if (passes_out) *passes_out = s->numpasses;
    return DAISY_OK;
}

extern "C" int daisy_solver_numpasses(daisy_solver *s) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_numpasses: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_numpasses");
    return s->numpasses;
}

extern "C" int daisy_solver_band_sums(daisy_solver *s, double *band_sums) {
    DZ_REQUIRE(s && band_sums, DAISY_E_INVALID, "daisy_solver_band_sums: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_band_sums");
    if (!s->sums_valid) { DZ_CUDA(cudaSetDevice(s->ctx->device)); int rc = fetch_sums(s); if (rc) return rc; }
    memcpy(band_sums, s->sums.data(), sizeof(double) * s->K);
    return DAISY_OK;
}

extern "C" int daisy_solver_read(daisy_solver *s, float *B, float *residual) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_read: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_read");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    // local rows only: out[k*nloc + pl]; both copies ride the solver's stream behind the passes, one synchronisation at the end
    cudaStream_t st = s->ctx->stream;
    if (B)
        DZ_CUDA(cudaMemcpy2DAsync(B, sizeof(float) * s->nloc, s->d_B, sizeof(float) * s->n, sizeof(float) * s->nloc, s->K, cudaMemcpyDeviceToHost, st));
    if (residual)
        DZ_CUDA(cudaMemcpy2DAsync(residual, sizeof(float) * s->nloc, s->d_res[s->cur] + (size_t)s->rank * s->bstride, sizeof(float) * s->n,
                                  sizeof(float) * s->nloc, s->K, cudaMemcpyDeviceToHost, st));
    DZ_CUDA(cudaStreamSynchronize(st));
    return DAISY_OK;
}

extern "C" int daisy_solver_write(daisy_solver *s, const float *B, const float *residual) {
    DZ_REQUIRE(s && B && residual, DAISY_E_INVALID, "daisy_solver_write: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_write");
    DZ_REQUIRE(s->G == 1, DAISY_E_STATE, "daisy_solver_write: single-GPU solvers only");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    DZ_CUDA(cudaMemcpy2DAsync(s->d_B, sizeof(float) * s->n, B, sizeof(float) * s->N, sizeof(float) * s->N, s->K, cudaMemcpyHostToDevice, st));
    DZ_CUDA(cudaMemcpy2DAsync(s->d_res[s->cur], sizeof(float) * s->n, residual, sizeof(float) * s->N, sizeof(float) * s->N, s->K,
                              cudaMemcpyHostToDevice, st));
    compute_sums_from_host(s, residual); // while the copies are in flight
    DZ_CUDA(cudaStreamSynchronize(st));
    s->sums_valid = true;
    s->abs_sums = false;
    return DAISY_OK;
}

// partitioned counterpart of daisy_solver_write: B_local is K x nloc (this rank's rows), residual_full is K x N (every
// rank holds the whole residual vector, as after an exchange)
extern "C" int daisy_solver_write_partitioned(daisy_solver *s, const float *B_local, const float *residual_full) {
    DZ_REQUIRE(s && B_local && residual_full, DAISY_E_INVALID, "daisy_solver_write_partitioned: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_write_partitioned");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    if (s->fused && s->seq > 0) { // peers' stores of the last pass have landed
        k_wait_flags<<<1, 32, 0, st>>>(s->d_flags, s->G, s->seq, s->timeout_ns, s->d_abort_host);
        DZ_CUDA(cudaGetLastError());
    }
    if (s->nloc > 0)
        DZ_CUDA(cudaMemcpy2DAsync(s->d_B, sizeof(float) * s->n, B_local, sizeof(float) * s->nloc, sizeof(float) * s->nloc, s->K, cudaMemcpyHostToDevice, st));
    for (int g = 0; g < s->G; g++) {
        const int c0 = g * s->n, w = (c0 < s->N) ? ((s->N - c0 < s->n) ? s->N - c0 : s->n) : 0;
        if (w > 0)
            DZ_CUDA(cudaMemcpy2DAsync(s->d_res[s->cur] + (size_t)g * s->bstride, sizeof(float) * s->n, residual_full + c0, sizeof(float) * s->N,
                                      sizeof(float) * w, s->K, cudaMemcpyHostToDevice, st));
    }
    compute_sums_from_host(s, residual_full); // while the copies are in flight
    DZ_CUDA(cudaStreamSynchronize(st));
    s->sums_valid = true;
    s->abs_sums = false;
    return DAISY_OK;
}

// ---- warm restart (DESIGN 3.3b) ----------------------------------------------------------------------------------------
// The restart pass streams F once with B_old as the input vector: y = M (F B_old) with the arithmetic of an ordinary pass,
// B_new = y + E, r = B_new - B_old.  B_old (this rank's K x nloc rows, or the solver's own B when B0_local is NULL) goes into
// d_B and, as the pass's input, into this rank's block of the buffer the pass reads -- with the fused exchange also into every
// peer's copy of that buffer, published with flag[rank] the way daisy_solver_write_slices publishes a residual, so the pass's
// own flag waits cover it.  From here on the solver is in restart mode: every pass totals |r|.
int dz_solver_restart_launch(daisy_solver *s, const float *B0_local) {
    DZ_SOLVER_CURRENT(s, "daisy_solver_restart");
    DZ_REQUIRE(s->G == 1 || s->fused, DAISY_E_STATE,
               "daisy_solver_restart: a partitioned solver needs the fused exchange (daisy_solver_set_peers); a partition exchanged by the host cannot restart");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    if (s->fused && s->h_abort && *reinterpret_cast<volatile unsigned long long *>(s->h_abort) != 0ull) return abort_error(s);
    cudaStream_t st = s->ctx->stream;
    // fused exchange: every rank has finished the last pass, and with it every read of the buffer about to be overwritten
    if (s->fused && s->seq > 0) {
        k_wait_flags<<<1, 32, 0, st>>>(s->d_flags, s->G, s->seq, s->timeout_ns, s->d_abort_host);
        DZ_CUDA(cudaGetLastError());
    }
    if (B0_local && s->nloc > 0) {
        DZ_CUDA(cudaMemcpy2DAsync(s->d_B, sizeof(float) * s->n, B0_local, sizeof(float) * s->nloc, sizeof(float) * s->nloc, s->K, cudaMemcpyHostToDevice, st));
        DZ_CUDA(cudaStreamSynchronize(st)); // B0_local is pageable host memory the caller may reuse at once
    }
    // the padded bands and the columns nloc..n-1 of d_B are zero (reset copies the zero-padded emission block; no pass writes them)
    const int in = s->fused ? (s->cur ^ 1) : s->cur;
    float *own = s->d_res[in] + (size_t)s->rank * s->bstride;
    DZ_CUDA(cudaMemcpyAsync(own, s->d_B, sizeof(float) * (size_t)s->Kp * s->n, cudaMemcpyDeviceToDevice, st));
    if (s->fused) {
        for (int g = 0; g < s->G; g++) {
            if (g == s->rank) continue;
            DZ_CUDA(cudaMemcpyAsync(s->peer_res[in][g] + (size_t)s->rank * s->bstride, own, sizeof(float) * (size_t)s->Kp * s->n, cudaMemcpyDeviceToDevice, st));
        }
        s->seq++;
        unsigned long long *f[16];
        for (int g = 0; g < 16; g++) f[g] = (g < s->G) ? s->peer_flags[g] + s->rank : nullptr;
        k_raise_flags<<<1, 32, 0, st>>>(s->G, s->seq, s->d_flags + 16, f[0], f[1], f[2], f[3], f[4], f[5], f[6], f[7], f[8], f[9], f[10], f[11], f[12],
                                        f[13], f[14], f[15]);
        DZ_CUDA(cudaGetLastError());
        s->cur = in;
    }
    if (!s->chained) DZ_CUDA(cudaEventRecord(s->e0, st));
    const unsigned long long wait_seq = s->fused ? s->seq : 0ull; // the B_old blocks just published
    if (s->fused) s->seq++;
    s->abs_sums = true;
    int rc = launch_pass(s, wait_seq, nullptr, true);
    if (rc) return rc;
    if (!s->chained) DZ_CUDA(cudaEventRecord(s->e1, st));
    s->events_recorded = !s->chained;
    s->numpasses = 0; // the restart pass counts as the first pass of the new solve
    return step_finish(s, nullptr);
}

extern "C" int daisy_solver_restart(daisy_solver *s, const float *B0) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_restart: null solver");
    DzRange range_("daisy_solver_restart");
    int rc = dz_solver_restart_launch(s, B0);
    if (rc) return rc;
    return fetch_sums(s); // the band sums of the restart pass: sum |r|
}

extern "C" int daisy_solver_set_emission(daisy_solver *s, const float *E) {
    DZ_REQUIRE(s && E, DAISY_E_INVALID, "daisy_solver_set_emission: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_set_emission");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    std::vector<float> ex;
    to_exchange(s, E, ex);
    DZ_CUDA(cudaStreamSynchronize(st)); // a restart pass enqueued earlier may still read the old emission
    DZ_CUDA(cudaMemcpyAsync(s->d_E, ex.data(), sizeof(float) * ex.size(), cudaMemcpyHostToDevice, st));
    std::vector<double> es((size_t)s->K);
    for (int k = 0; k < s->K; k++) es[(size_t)k] = host_sum(E + (size_t)k * s->N, (size_t)s->N);
    DZ_CUDA(cudaStreamSynchronize(st)); // `ex` is pageable host memory
    s->e_sums = es;
    return DAISY_OK;
}

extern "C" int daisy_solver_set_materials(daisy_solver *s, const float *M, int nmat, const int32_t *mat_idx) {
    DZ_REQUIRE(s && M && mat_idx, DAISY_E_INVALID, "daisy_solver_set_materials: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_set_materials");
    DZ_REQUIRE(nmat >= 1, DAISY_E_INVALID, "daisy_solver_set_materials: need at least one material");
    for (int p = 0; p < s->N; p++)
        DZ_REQUIRE(mat_idx[p] >= 0 && mat_idx[p] < nmat, DAISY_E_INVALID, "daisy_solver_set_materials: material index out of range");
    DZ_CUDA(cudaSetDevice(s->ctx->device));
    cudaStream_t st = s->ctx->stream;
    DZ_CUDA(cudaStreamSynchronize(st)); // no pass in flight reads d_M or d_mat below
    if (nmat > s->nmat_cap) {
        float *d = nullptr;
        DZ_CUDA(cudaMalloc(&d, sizeof(float) * (size_t)nmat * s->Kp * s->Kp)); // on failure the solver keeps its old matrices
        cudaFree(s->d_M);
        s->d_M = d;
        s->nmat_cap = nmat;
    }
    std::vector<float> Mp;
    pad_materials(s, M, nmat, Mp);
    DZ_CUDA(cudaMemcpyAsync(s->d_M, Mp.data(), sizeof(float) * Mp.size(), cudaMemcpyHostToDevice, st));
    if (s->nloc > 0) DZ_CUDA(cudaMemcpyAsync(s->d_mat, mat_idx + s->row0, sizeof(int) * (size_t)s->nloc, cudaMemcpyHostToDevice, st));
    DZ_CUDA(cudaStreamSynchronize(st)); // `Mp` is pageable host memory
    s->nmat = nmat;
    return DAISY_OK;
}

// kernels one pass launches in this solver's configuration (the benchmark reports it)
extern "C" int daisy_solver_launches_per_pass(daisy_solver *s) {
    DZ_REQUIRE(s, DAISY_E_INVALID, "daisy_solver_launches_per_pass: null solver");
    DZ_SOLVER_CURRENT(s, "daisy_solver_launches_per_pass");
    if (s->fused_epi) return 1;                         // k_gather_tma with the epilogue and the exchange wait inside
    int n = 2;                                          // streaming kernel + k_gather_epilogue
    if (s->use_mma) n += 1;                             // k_split_residual
    if (s->fused) n += 1;                               // k_wait_flags
    return n;
}

extern "C" int daisy_solver_last_step_ms(daisy_solver *s, double *ms) {
    DZ_REQUIRE(s && ms, DAISY_E_INVALID, "daisy_solver_last_step_ms: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_last_step_ms");
    *ms = s->last_ms;
    return DAISY_OK;
}

// tile map of the last scan (tile skipping): dims2 = row blocks, column steps (0, 0 when the solver streams the dense plan);
// occ (may be NULL) receives the nrb x S map if capacity allows; occupied = tiles with a non-zero entry; scan_ms = device time
// of the scan kernel
extern "C" int daisy_solver_tile_map(daisy_solver *s, int32_t *dims2, uint8_t *occ, int64_t capacity, int64_t *occupied, double *scan_ms) {
    DZ_REQUIRE(s && dims2, DAISY_E_INVALID, "daisy_solver_tile_map: null argument");
    DZ_SOLVER_CURRENT(s, "daisy_solver_tile_map");
    const bool have = s->skip && !s->occ.empty();
    dims2[0] = have ? (int32_t)(s->occ.size() / (size_t)s->sk_S) : 0;
    dims2[1] = have ? s->sk_S : 0;
    if (occ && have) {
        DZ_REQUIRE(capacity >= (int64_t)s->occ.size(), DAISY_E_INVALID, "daisy_solver_tile_map: buffer too small");
        memcpy(occ, s->occ.data(), s->occ.size());
    }
    if (occupied) *occupied = have ? s->occupied : 0;
    if (scan_ms) *scan_ms = have ? s->scan_ms : 0.0;
    return DAISY_OK;
}

// diagnostic, host only: the compacted stream-K plan k_gather_tma runs for an nrb x S tile map on `sms` SMs, with the pieces every
// CTA takes as the kernel's own next_piece computes them
extern "C" int daisy_gather_plan_dump(const uint8_t *occ, int nrb, int S, int sms, int32_t *info5, int32_t *list, int32_t *off, int32_t *pieces6,
                                      int64_t capacity) {
    DZ_REQUIRE(occ && info5 && nrb >= 0 && S >= 0 && sms >= 1, DAISY_E_INVALID, "daisy_gather_plan_dump: bad argument");
    SkipPlan sp;
    build_skip_plan(occ, nrb, S, sms, sp);
    GatherParams P;
    memset(&P, 0, sizeof(P));
    P.nrb = nrb; P.sk = 1; P.sk_S = S; P.sk_L = sp.L; P.sk_total = sp.total;
    P.sk_list = sp.list.data(); P.sk_off = sp.off.data();
    std::vector<int32_t> pcs;
    for (int c = 0; c < sp.grid && sp.total > 0; c++) {
        int cursor = 0;
        Piece p;
        memset(&p, 0, sizeof(p));
        while (next_piece<256>(P, c, sp.grid, cursor, p)) {
            const int32_t rec[6] = { c, p.rb, p.s0, p.s1, p.idx, p.np };
            pcs.insert(pcs.end(), rec, rec + 6);
        }
    }
    info5[0] = sp.total; info5[1] = sp.grid; info5[2] = sp.L; info5[3] = sp.maxp; info5[4] = (int32_t)(pcs.size() / 6);
    if (list || off || pieces6)
        DZ_REQUIRE(capacity >= (int64_t)pcs.size() && capacity >= (int64_t)sp.total && capacity >= (int64_t)nrb + 1, DAISY_E_INVALID,
                   "daisy_gather_plan_dump: buffers too small");
    if (list) memcpy(list, sp.list.data(), sizeof(int32_t) * sp.list.size());
    if (off) memcpy(off, sp.off.data(), sizeof(int32_t) * sp.off.size());
    if (pieces6) memcpy(pieces6, pcs.data(), sizeof(int32_t) * pcs.size());
    return DAISY_OK;
}
