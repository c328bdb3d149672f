// gather_mma.cuh -- the gather pass for wide band counts (K = 16 / 32 / 64) on the 5th-generation tensor cores.
//
// With K bands every F element feeds K FMAs; at K = 32 that is 16 flop per HBM byte, beyond what the FP32 pipe can
// sustain at HBM speed (128 FMA/clk/SM against 5.8 F elements/clk/SM x 32).  The contraction
//     out[r, k] = sum_c F[r, c] * R[k, c]          (SpectralLightning::increment_light_fluorescent, Lightning.h:203-206)
// is a real dense GEMM there (M = rows, N = K, reduction over the N columns), so it runs as tcgen05.mma kind::tf32.
// TF32 alone (10-bit mantissa) would miss the 1e-5 parity bar, so both operands are split into two TF32 terms
// (3xTF32):  F = Fh + Fl,  R = Rh + Rl,  F*R ~= Fh*Rh + Fh*Rl + Fl*Rh, every term rounded to nearest (cvt.rna), so the
// split error is unbiased and < 2^-21 relative.  The tensor core adds into its FP32 accumulator with truncation; over
// thousands of k-steps that is a systematic bias (measured 4.5e-6 after 2048 columns), so the TMEM accumulator only
// ever holds ONE 64-column stage (16 MMAs, 24 at K = 64) and the stage sums are added up in FP32 round-to-nearest by the epilogue
// warps (tcgen05.ld moves 64 B/clk, which is why the accumulator is not drained more often than that).
//
// Per CTA (one per SM, persistent over (128-row block) x (column range) items):
//   warp 0      TMA producer: per stage two F sub-tiles 128 x 32 (SWIZZLE_128B) + two band sub-tiles [Rh;Rl] 2K x 32,
//               4-stage ring (3 stages at K = 64)
//   warps 4-11  converters (two sets alternating stages): LDS their row of the F tile, Fh = tf32(F) (round to nearest),
//               Fl = F - Fh, tcgen05.st both into a TMEM operand ring -- the A operand is read from TMEM, so the F
//               bytes cross shared memory exactly once on the way in and once to registers
//   warp 1      MMA issuer (one elected lane): per 8-column k-step  D[:, 0:2K] += Fh x [Rh;Rl]^T  and  D[:, 0:K] += Fl x Rh^T,
//               at K = 64 D[:, 0:K] += Fh x Rh^T, Fh x Rl^T and Fl x Rh^T (three MMAs of N = 64 into the same columns),
//               one tcgen05.commit per stage on the mma_done ring (frees the smem slot and the operand slot, signals the
//               epilogue); this thread is the kernel's critical path
//   warps 12-15 epilogue: per stage tcgen05.ld the 2K accumulator columns, acc[k] += D[:, k] + D[:, K+k] (K = 64: the K
//               columns, acc[k] += D[:, k], in two 32-column chunks); at the end
//               of the item the column-range partials go to global memory
//   warp 2      TMEM allocation
// TMEM: 4 accumulator buffers (2K columns each) + 2 operand stages (128 columns each) = 512 columns for K = 32; K = 64:
// 3 accumulator buffers of 64 columns, the operand stages at columns 256-511 (MmaCfg).
#pragma once

#define MM_ROWS 128
#define MM_SUB 32   // columns per SWIZZLE_128B sub-tile (128 bytes)
#define MM_COLS 64  // columns per stage: two sub-tiles, i.e. 256 contiguous bytes of every F row per stage
#define MM_NS 4     // shared-memory stages (K = 16 / 32)
#define MM_NA 2     // TMEM operand stages (128 columns each: 64 of Fh, 64 of Fl)
#define MM_ND 4     // TMEM accumulator buffers (one stage each; K = 16 / 32)
#define MM_THREADS 512

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{ .reg .pred p; elect.sync _|p, 0xffffffff; selp.u32 %0, 1, 0, p; }" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[tmem] x B[smem]^T, TF32 inputs, FP32 accumulate; issued by one thread
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
// shared-memory matrix descriptor: K-major rows of 128 B, SWIZZLE_128B, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t tc_smem_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);       // start address, 16-byte units
    d |= (uint64_t)1 << 16;                        // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset: 8 rows x 128 B
    d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)
    d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
    return d;
}
// instruction descriptor, kind::tf32: D = F32, A = B = TF32, both K-major, M x N
__host__ __device__ constexpr uint32_t tc_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// 32 registers -> 32 TMEM columns of this warp's 32 lanes
__device__ __forceinline__ void tc_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]),
        "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]),
        "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31]) : "memory");
}
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// 32 TMEM columns of this warp's 32 lanes -> 32 registers
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}

// residual bands of the current exchange buffer -> [Rh (K rows); Rl (K rows)] x ncolsP, Rh = R rounded to TF32,
// Rl = (R - Rh) rounded to TF32.  Device converge (stop.state != null): the first kernel of the pass takes the stop decision;
// every CTA reaches the same one, and k_gather_mma and the epilogue only read `stopped`.
template <int K>
__global__ void k_split_residual(const float *__restrict__ res, int64_t bstride, int n, int ncols, int ncolsP, float *__restrict__ split,
                                 DevStop stop) {
    if (stop.state) {
        __shared__ int s_stop;
        if (threadIdx.x == 0) s_stop = stop_decide(stop);
        __syncthreads();
        if (s_stop) return;
    }
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncolsP) return;
    const int g = c / n, jl = c - g * n;
#pragma unroll 4
    for (int k = 0; k < K; k++) {
        float x = (c < ncols) ? res[(size_t)g * bstride + (size_t)k * n + jl] : 0.0f;
        uint32_t hb;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(x));
        float h = __uint_as_float(hb);
        split[(size_t)k * ncolsP + c] = h;
        uint32_t lb;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(lb) : "f"(x - h));
        split[(size_t)(K + k) * ncolsP + c] = __uint_as_float(lb);
    }
}

// Ring depths and TMEM layout per band count.  K = 16 / 32: 4 shared-memory stages, 4 accumulator buffers of 2K columns
// (Fh x Rh and Fh x Rl side by side, Fl x Rh added into the first K).  K = 64: a stage is 64 KB (32 KB of F + 32 KB of
// [Rh;Rl]), so 3 stages fill the 227 KB; all three products go into the same K columns (24 MMAs of N = 64 per stage instead
// of 16), which keeps the drain at 64 columns per stage (512 of the 1424-cycle HBM budget, as at K = 32) and lets 3
// accumulator buffers of 64 columns sit below the operand ring at column 256.  ND <= NS and NA < NS: no mma_done slot can
// complete a second phase before every role has observed the first (see k_gather_mma).
template <int K> struct MmaCfg {
    static constexpr int NS = MM_NS, ND = MM_ND, DCOLS = 2 * K, A_COL0 = MM_ND * 2 * K;
};
template <> struct MmaCfg<64> { static constexpr int NS = 3, ND = 3, DCOLS = 64, A_COL0 = 256; };

template <int K>
__host__ __device__ constexpr int mm_stage_bytes() { return 2 * (MM_ROWS * MM_SUB * 4 + 2 * K * MM_SUB * 4); }
template <int K>
__host__ __device__ constexpr int mm_smem_bytes() { return MmaCfg<K>::NS * mm_stage_bytes<K>() + 1024 + 512; }

template <int K>
__global__ void __launch_bounds__(MM_THREADS, 1)
k_gather_mma(GatherParams P, const __grid_constant__ CUtensorMap tmF, const __grid_constant__ CUtensorMap tmR) {
    constexpr int STAGE = mm_stage_bytes<K>();
    constexpr int F_SUB = MM_ROWS * MM_SUB * 4;  // one F sub-tile
    constexpr int B_SUB = 2 * K * MM_SUB * 4;    // one band sub-tile
    constexpr int B_OFF = 2 * F_SUB;             // band sub-tiles follow the two F sub-tiles
    constexpr int NS = MmaCfg<K>::NS, ND = MmaCfg<K>::ND;
    constexpr int DCOLS = MmaCfg<K>::DCOLS;      // accumulator columns per buffer
    constexpr int A_COL0 = MmaCfg<K>::A_COL0;    // operand ring starts after the accumulator buffers
    constexpr int A_COLS = 2 * MM_COLS;          // Fh columns then Fl columns
    constexpr uint32_t IDESC_2K = tc_idesc_tf32(MM_ROWS, 2 * K), IDESC_K = tc_idesc_tf32(MM_ROWS, K);
    static_assert(ND * DCOLS <= A_COL0 && A_COL0 + MM_NA * A_COLS <= 512, "TMEM budget");
    static_assert(NS * STAGE + 1024 + 512 <= 227 * 1024, "shared-memory budget");
    extern __shared__ unsigned char mm_smem_raw[];
    const uint32_t raw = smem_u32(mm_smem_raw);
    unsigned char *base = mm_smem_raw + (((raw + 1023u) & ~1023u) - raw); // SWIZZLE_128B tiles need 1024-byte alignment
    uint64_t *bars = reinterpret_cast<uint64_t *>(base + (size_t)NS * STAGE);
    // full barriers: the two converter sets take alternate stages, so with an odd ring depth a slot's consecutive stages
    // belong to different sets, and the set of stage it + NS could wait for the slot's next phase before the current one has
    // completed -- which a parity wait cannot tell from a completed phase.  NF = 2 NS barriers then give every barrier to one set.
    constexpr int NF = (NS % 2 == 0) ? NS : 2 * NS;
    uint64_t *full = bars, *empty = bars + NF, *a_full = bars + NF + NS;
    static_assert((NF + 2 * NS + MM_NA + ND) * 8 + 4 <= 512, "barrier space");
    uint64_t *mma_done = a_full + MM_NA, *d_empty = mma_done + NS;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(d_empty + ND);
    // mma_done[it % NS] completes once per stage, and every waiter must see a phase before the slot completes again: the
    // epilogue releases stage it before the MMAs of stage it + NS may start (ND <= NS), and the converters wait on stage
    // it - NA before they hand over stage it, which the MMAs of every later stage follow (NA < NS)
    static_assert(MM_NA == 2 && ND <= NS && MM_NA < NS, "mma_done ring indexing below assumes these depths");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (P.stop.state && stop_stopped(P.stop)) return; // device converge: before any TMEM is allocated
    if (tid == 0) {
        for (int i = 0; i < NS; i++) { mbar_init(&full[i], 1); mbar_init(&empty[i], 4); mbar_init(&mma_done[i], 1); }  // empty: 4 converter warps
        for (int i = NS; i < NF; i++) mbar_init(&full[i], 1);
        for (int i = 0; i < MM_NA; i++) mbar_init(&a_full[i], 4);
        for (int i = 0; i < ND; i++) mbar_init(&d_empty[i], 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const int nitems = P.nrb * P.nsplit;
    uint32_t it = 0; // global stage counter, identical in every role

    if (warp == 0) {
        // ------------------------------- TMA producer -------------------------------
        if (lane == 0) {
            uint64_t pol_first;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_first));
            for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
                const int rb = item / P.nsplit, split = item - rb * P.nsplit;
                const int c_begin = split * P.colw, c_end = min(P.ncols, c_begin + P.colw);
                const int nstep = (c_end - c_begin + MM_COLS - 1) / MM_COLS;
                for (int s = 0; s < nstep; s++, it++) {
                    const int st = it % NS;
                    mbar_wait(&empty[st], ((it / NS) & 1) ^ 1);      // converters have read the F tiles of stage it-NS
                    mbar_wait(&mma_done[st], ((it / NS) & 1) ^ 1);   // the MMAs of stage it-NS have read its band tiles
                    unsigned char *sf = base + (size_t)st * STAGE;
                    const int c0 = c_begin + s * MM_COLS;
                    uint64_t *fb = &full[it % NF];
                    mbar_expect_tx(fb, (uint32_t)STAGE);
                    // F streams through L2 evict_first: it is read once per pass and must not push the split residual out
                    tma_load_2d_hint(sf, &tmF, c0, rb * MM_ROWS, fb, pol_first);
                    tma_load_2d_hint(sf + F_SUB, &tmF, c0 + MM_SUB, rb * MM_ROWS, fb, pol_first);
                    tma_load_2d(sf + B_OFF, &tmR, c0, 0, fb);
                    tma_load_2d(sf + B_OFF + B_SUB, &tmR, c0 + MM_SUB, 0, fb);
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------- MMA issuer ---------------------------------
        // The whole warp runs the loop (uniform control flow keeps descriptors in uniform registers); one elected lane
        // issues.  The issuing thread is the critical path of this kernel (per-MMA issue ~40 clk plus the barrier
        // round trips), so it waits on two barriers per stage and signals one: a_full[a] implies the stage's full barrier (the
        // converters waited on it), and a single commit per stage serves the producer (smem slot), the converters
        // (operand slot) and the epilogue (accumulator ready).
        const bool leader = elect_one();
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
            const int split = item % P.nsplit;
            const int c_begin = split * P.colw, c_end = min(P.ncols, c_begin + P.colw);
            const int nstep = (c_end - c_begin + MM_COLS - 1) / MM_COLS;
            for (int s = 0; s < nstep; s++, it++) {
                const int st = it % NS, a = it % MM_NA, b = it % ND;
                mbar_wait(&a_full[a], (it / MM_NA) & 1);
                mbar_wait(&d_empty[b], ((it / ND) & 1) ^ 1);
                tc_fence_after();
                const uint32_t b_addr = smem_u32(base + (size_t)st * STAGE + B_OFF);
                const uint32_t a_tmem = tmem + A_COL0 + a * A_COLS;
                const uint32_t d_tmem = tmem + b * DCOLS;
                if (leader) {
#pragma unroll
                    for (int k = 0; k < MM_COLS / 8; k++) {
                        const uint64_t bdesc = tc_smem_desc_sw128(b_addr + (k >> 2) * B_SUB + (k & 3) * 32);
                        if constexpr (K == 64) {
                            // Rl starts K rows = 8 KB into the band sub-tile: a whole number of 1024-byte swizzle atoms
                            const uint64_t bdesc_l = tc_smem_desc_sw128(b_addr + (k >> 2) * B_SUB + K * 128 + (k & 3) * 32);
                            tc_mma_tf32_ts(d_tmem, a_tmem + k * 8, bdesc, IDESC_K, k > 0 ? 1u : 0u);     // Fh x Rh
                            tc_mma_tf32_ts(d_tmem, a_tmem + k * 8, bdesc_l, IDESC_K, 1u);                // Fh x Rl
                        } else {
                            tc_mma_tf32_ts(d_tmem, a_tmem + k * 8, bdesc, IDESC_2K, k > 0 ? 1u : 0u);    // Fh x [Rh;Rl]
                        }
                        tc_mma_tf32_ts(d_tmem, a_tmem + MM_COLS + k * 8, bdesc, IDESC_K, 1u);          // Fl x Rh
                    }
                    tc_commit(&mma_done[it % NS]);
                }
                __syncwarp();
            }
        }
    } else if (warp >= 4 && warp < 12) {
        // ------------------------------- converters ---------------------------------
        const uint32_t set = (warp - 4) >> 2;              // stages with (it & 1) == set
        const int row = (warp & 3) * 32 + lane;            // tile row = TMEM lane
        const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
            const int split = item % P.nsplit;
            const int c_begin = split * P.colw, c_end = min(P.ncols, c_begin + P.colw);
            const int nstep = (c_end - c_begin + MM_COLS - 1) / MM_COLS;
            for (int s = 0; s < nstep; s++, it++) {
                if ((it & 1) != set) continue;
                const int st = it % NS, a = it % MM_NA;
                mbar_wait(&full[it % NF], (it / NF) & 1);
                const uint32_t a_tmem = tmem + lane_off + A_COL0 + a * A_COLS;
#pragma unroll
                for (int sub = 0; sub < 2; sub++) {
                    const unsigned char *srow = base + (size_t)st * STAGE + sub * F_SUB + row * 128;
                    uint32_t hi[32], lo[32];
#pragma unroll
                    for (int q = 0; q < 8; q++) {
                        const float4 v = *reinterpret_cast<const float4 *>(srow + ((q ^ (row & 7)) << 4));
                        const float f[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            // Fh = F rounded to TF32 (nearest, ties away: add half an ulp of the 10-bit mantissa, clear the rest);
                            // Fl = F - Fh is exact, symmetric around 0, and the tensor core keeps its top 11 bits
                            const uint32_t h = (__float_as_uint(f[e]) + 0x1000u) & 0xFFFFE000u;
                            hi[q * 4 + e] = h;
                            lo[q * 4 + e] = __float_as_uint(f[e] - __uint_as_float(h));
                        }
                    }
                    if (sub == 1) {
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&empty[st]);     // both F sub-tiles are in registers
                    }
                    if (sub == 0) {
                        if (it >= MM_NA) mbar_wait(&mma_done[(it - MM_NA) % NS], ((it - MM_NA) / NS) & 1); // MMAs of stage it-2 are done with this operand slot
                        tc_fence_after();
                    }
                    tc_st32(a_tmem + sub * MM_SUB, hi);
                    tc_st32(a_tmem + MM_COLS + sub * MM_SUB, lo);
                }
                tc_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[a]);
            }
        }
    } else if (warp >= 12) {
        // ------------------------------- epilogue -----------------------------------
        const int row_in = (warp & 3) * 32 + lane;
        const uint32_t lane_off = (uint32_t)((warp & 3) * 32) << 16;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
            const int rb = item / P.nsplit, split = item - rb * P.nsplit;
            const int c_begin = split * P.colw, c_end = min(P.ncols, c_begin + P.colw);
            const int nstep = (c_end - c_begin + MM_COLS - 1) / MM_COLS;
            float out[K];
#pragma unroll
            for (int k = 0; k < K; k++) out[k] = 0.0f;
            for (int s = 0; s < nstep; s++, it++) {
                const int b = it % ND;
                mbar_wait(&mma_done[it % NS], (it / NS) & 1);
                tc_fence_after();
                if constexpr (K == 64) {
                    // one 32-column chunk in registers at a time: out[64] and 64 loaded columns would not fit 128 registers
                    uint32_t r[32];
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        tc_ld32(tmem + lane_off + b * DCOLS + h * 32, r);
                        tc_wait_ld();
#pragma unroll
                        for (int k = 0; k < 32; k++) out[h * 32 + k] += __uint_as_float(r[k]);
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&d_empty[b]);
                } else if constexpr (K == 32) {
                    uint32_t r0[32], r1[32];
                    tc_ld32(tmem + lane_off + b * DCOLS, r0);
                    tc_ld32(tmem + lane_off + b * DCOLS + 32, r1);
                    tc_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&d_empty[b]);
#pragma unroll
                    for (int k = 0; k < 32; k++) out[k] += __uint_as_float(r0[k]) + __uint_as_float(r1[k]);
                } else {
                    uint32_t r0[16], r1[16];
                    tc_ld16(tmem + lane_off + b * DCOLS, r0);
                    tc_ld16(tmem + lane_off + b * DCOLS + 16, r1);
                    tc_wait_ld();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&d_empty[b]);
#pragma unroll
                    for (int k = 0; k < 16; k++) out[k] += __uint_as_float(r0[k]) + __uint_as_float(r1[k]);
                }
            }
            const int row = rb * MM_ROWS + row_in;
            if (row < P.nloc) {
                float4 *dst = reinterpret_cast<float4 *>(P.partial + ((size_t)split * P.nloc + row) * K);
#pragma unroll
                for (int q = 0; q < K / 4; q++) dst[q] = make_float4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}
