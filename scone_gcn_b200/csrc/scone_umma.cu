// scone_umma.cu — the dense fused Hodge-Laplacian layer (width 32 -> 32) on the 5th-generation tensor cores (tcgen05 / TMEM):
//
//   Hout = act(Hin W0 + (S0 Hin) W1 + (S1 Hin) W2)                           trajectory_experiments.py:145-149,163-167
//
// Same gather as the slab kernel (scone_slab.cu: one pass over the merged operator row, warp-wide 128-bit loads, packed FFMA2
// sums whose registers are mma A fragments), but the product runs as M = 128 tcgen05.mma tiles instead of per-warp mma.sync:
//   * a GROUP of 8 warps owns a tile of 128 rows (8 consecutive edges x 16 trajectories); warp w of the group writes its 16 gathered
//     rows, split hi / lo for 3xTF32, with tcgen05.st.16x128b.x2 into TMEM lanes 32 (w % 4) + 16 (w / 4) .. + 15 — the fragment
//     registers {a0, a1, a2, a3} of a k-step ARE that instruction's register layout, so the gathered rows go registers -> TMEM,
//     never through shared memory;
//   * one elected thread issues 36 tcgen05.mma.kind::tf32 (A from TMEM, B = the 96 x 32 weight stack hi / lo in shared memory,
//     no-swizzle K-major canonical layout, staged once per CTA): D[128][32] (fp32, TMEM) = A_lo B_hi + A_hi B_lo + A_hi B_hi;
//     tcgen05.commit arrives on an mbarrier;
//   * every warp reads its 16 rows of D back with tcgen05.ld.16x256b.x4 (the mma C-fragment layout), applies the activation and
//     stores 64-bit pairs exactly as the slab kernel does.
// Two groups per CTA (16 warps, one persistent CTA per SM) with private TMEM regions (2 x (96 + 96 + 32) = 448 of 512 columns) and
// private barriers: while one group's tile is in the tensor core the other group gathers.  Weights are read once per 128 rows
// (mma.sync: once per 16 rows) and the tensor instruction stream is one thread's, not every warp's.
// Every wait is bounded: a protocol error sets *err and the kernel runs on (wrong results, reported by the host) instead of hanging.
#include "common.cuh"

namespace {

#include "slab_common.cuh"

constexpr int kGatherWarps = 16, kGroupWarps = 8, kUmmaThreads = kGatherWarps * 32;
// (no dedicated MMA warp: a 17th warp would put 5 warps on one SM sub-partition and cap every thread at 96 registers)
constexpr int kC = 32;
constexpr int kGatherDepth = 4;            // neighbour rows in flight per warp: the gather is bound by load latency at 17 warps per SM
// Forward tile order: chunks of kTileChunk consecutive tiles dealt round-robin to the CTAs.  Inside a chunk the neighbour rows of
// consecutive edges are L1 hits; with small chunks all CTAs sweep the same region of the tensor and an L1 miss is an L2 hit instead
// of a DRAM read.  Measured on the 1M-edge complex: 9.34 ms at 8, 9.62 ms with one contiguous range per CTA, 10.86 ms at 1.
constexpr int kTileChunk = 8;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kColsAhi = 0, kColsAlo = 96, kColsD = 192, kColsGroup = 224;
// f32 accumulate, tf32 x tf32, A / B K-major, N = 32, M = 128 (UMMA instruction descriptor, cute/arch/mma_sm100_desc.hpp)
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((32u >> 3) << 17) | ((128u >> 4) << 24);
constexpr uint32_t kLbo = 512, kSbo = 128;               // bytes: K-direction / N-direction stride between 8 x 16 B core matrices
constexpr int kSpinLimit = 4000000;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_st_16x128b_x2(uint32_t taddr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
    asm volatile("tcgen05.st.sync.aligned.16x128b.x2.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
__device__ __forceinline__ void tc_ld_16x256b_x4(uint32_t taddr, float (&d)[4][4]) {
    uint32_t r[16];
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
        for (int q = 0; q < 4; ++q) d[nt][q] = __uint_as_float(r[4 * nt + q]);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
    return ok != 0;
}
// bounded wait: a protocol error sets *err and lets the kernel run on instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int* err) {
    int spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        if (++spins > kSpinLimit) {
            *err = 1;
            break;
        }
    }
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(kIdesc), "r"(accumulate), "r"(0u)
        : "memory");
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {       // no-swizzle K-major descriptor, version 1 (Blackwell)
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((kLbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((kSbo >> 4) & 0x3FFF) << 32) |
           ((uint64_t)1 << 46);
}

// Pipeline.  16 warps in two groups of 8 (group = one 128-row MMA tile = 8 consecutive edges x 16 trajectories).
//   per warp and iteration:   [gather slab i+1 into registers]  while the tensor core works on tile i
//                             wait D_full(i) -> tcgen05.ld -> activation -> store           (its 16 rows of tile i)
//                             split + tcgen05.st slab i+1 into TMEM -> count itself in       (the 8th arrival issues the tile's
//                                                                                             36 tcgen05.mma + tcgen05.commit -> D_full)
// D may be overwritten by tile i+1 only after all 8 warps read tile i: each counts itself in for tile i+1 after its tcgen05.ld completed.
// A may be overwritten by slab i+1 only after the MMAs of tile i finished: the warp waited on D_full(i) first.
template <int ACT>
__global__ void __launch_bounds__(kUmmaThreads, 1) layer_fwd_umma_kernel(const float* __restrict__ Hin, float* __restrict__ Hout,
                                                                        const float* __restrict__ W0, const float* __restrict__ W1,
                                                                        const float* __restrict__ W2, const int32_t* __restrict__ mptr,
                                                                        const int2* __restrict__ ment, int E, int b, int* __restrict__ err) {
    constexpr int TS = 16;
    using G = SlabGeom<kC, TS>;
    constexpr int NT = kC / 8;
    // B operand: [hi | lo][k-chunk 24][n-group 4][8 rows][4 floats]; element (n, k) of the stacked weights, k = 32 term + 8 s + kappa
    // <-> input channel chan(s, kappa) of W_term (the k order of the gather's fragments)
    __shared__ __align__(128) float Bs[2][24 * 4 * 32];
    __shared__ __align__(8) uint64_t s_dfull[2];
    __shared__ unsigned s_arrived[2];                     // warps of the group whose rows of the current tile are in TMEM
    __shared__ uint32_t s_tmem;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tig = lane & 3;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (threadIdx.x == 0) {
        s_arrived[0] = s_arrived[1] = 0u;
        mbar_init(&s_dfull[0], 1);
        mbar_init(&s_dfull[1], 1);
    }
    for (int i = threadIdx.x; i < 96 * kC; i += kUmmaThreads) {
        const int k = i / kC, n = i % kC;
        const int term = k / 32, s = (k % 32) / 8, kappa = k % 8;
        const float* W = term == 0 ? W0 : (term == 1 ? W1 : W2);
        const float w = W[G::chan(s, kappa) * kC + n];
        const uint32_t hi = to_tf32(w), lo = to_tf32(w - __uint_as_float(hi));
        const int off = (k / 4) * 128 + (n / 8) * 32 + (n % 8) * 4 + (k % 4);
        Bs[0][off] = __uint_as_float(hi);
        Bs[1][off] = __uint_as_float(lo);
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");       // generic-proxy writes of Bs -> the tensor core's async proxy
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const int n_ts = (b + TS - 1) / TS;
    const int tiles_per_ts = (E + kGatherWarps - 1) / kGatherWarps;      // a CTA tile = 16 consecutive edges x one slab of 16 trajectories
    const long long n_tiles = (long long)n_ts * tiles_per_ts;

    {
        // ---- gather warps ----
        const int group = warp / kGroupWarps, gw = warp % kGroupWarps;
        const uint32_t tbase = s_tmem + (uint32_t)group * kColsGroup;
        const uint32_t lane_base = (uint32_t)(32 * (gw & 3) + 16 * (gw >> 2)) << 16;   // this warp's 16 TMEM lanes of the tile
        const unsigned rowbytes_in = (unsigned)b * kC * 4u;
        const size_t rowlen_out = (size_t)b * kC;
        uint32_t phase = 0;
        int pe0 = 0, pt0 = 0;                              // slab whose product is in flight
        bool pending = false, plive = false;
        for (long long k = 0;; ++k) {
            const long long tile = ((k / kTileChunk) * gridDim.x + blockIdx.x) * kTileChunk + k % kTileChunk;
            const bool have = tile < n_tiles;
            int e0 = 0, t0 = 0;
            bool live = false;
            u64 acc[3][G::NL][2];
            if (have) {
                const int ts = (int)(tile / tiles_per_ts);
                e0 = (int)(tile - (long long)ts * tiles_per_ts) * kGatherWarps + warp;
                t0 = ts * TS;
                live = e0 < E;                             // (a dead slab still takes part in the barriers; its rows are never stored)
                if (live) {
                    slab_gather<kC, TS, kGatherDepth>(Hin, rowbytes_in, mptr, ment, E, b, e0, t0, acc);
                } else {
#pragma unroll
                    for (int k = 0; k < 3; ++k)
#pragma unroll
                        for (int i = 0; i < G::NL; ++i) acc[k][i][0] = acc[k][i][1] = 0ull;
                }
            }
            if (pending) {                                 // epilogue of the previous slab: its tile has been in the tensor core meanwhile
                mbar_wait(&s_dfull[group], phase, err);
                phase ^= 1u;
                tc_fence_after();
                float d[NT][4];
                tc_ld_16x256b_x4(tbase + kColsD + lane_base, d);
                if (plive) {
                    slab_activate<ACT, NT>(d);
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        int e, t;
                        slab_row<kC, TS>(r, pe0, pt0, e, t);
                        if (e < E && t < b) {
                            float* dst = Hout + (size_t)e * rowlen_out + (size_t)t * kC + 2 * tig;
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
                                *reinterpret_cast<float2*>(dst + nt * 8) = make_float2(d[nt][2 * r], d[nt][2 * r + 1]);
                        }
                    }
                }
            }
            if (have) {
                // fragments of every (term, k-step), split for 3xTF32, straight into TMEM: columns 32 term + 8 s .. + 7 of A_hi / A_lo
#pragma unroll
                for (int term = 0; term < 3; ++term) {
                    float fr[G::KS][4];
                    slab_fragments<kC, TS>(acc[term], fr);
#pragma unroll
                    for (int s = 0; s < G::KS; ++s) {
                        uint32_t ah[4], al[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) split_tf32(fr[s][q], ah[q], al[q]);
                        const uint32_t col = (uint32_t)(32 * term + 8 * s);
                        tc_st_16x128b_x2(tbase + kColsAhi + col + lane_base, ah[0], ah[1], ah[2], ah[3]);
                        tc_st_16x128b_x2(tbase + kColsAlo + col + lane_base, al[0], al[1], al[2], al[3]);
                    }
                }
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                tc_fence_before();
                __syncwarp();
                // the LAST of the group's 8 warps to get here issues the tile's MMAs (acq_rel counter: the other warps' TMEM stores
                // happen-before its tcgen05.mma); nobody waits for anybody
                unsigned last_one = 0u;
                if (lane == 0) {
                    unsigned old;
                    asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(&s_arrived[group])) : "memory");
                    last_one = (old % kGroupWarps) == (unsigned)(kGroupWarps - 1) ? 1u : 0u;     // (the counter runs on: no reset to order)
                    if (last_one) {
                        tc_fence_after();
                        const uint32_t bhi = smem_u32(&Bs[0][0]), blo = smem_u32(&Bs[1][0]);
#pragma unroll
                        for (int j = 0; j < 12; ++j) {     // K = 96 in steps of 8: two 16-byte k-chunks of B per step
                            const uint64_t dh = umma_desc(bhi + (uint32_t)j * 2 * kLbo), dl = umma_desc(blo + (uint32_t)j * 2 * kLbo);
                            umma_tf32_ts(tbase + kColsD, tbase + kColsAlo + 8 * j, dh, j > 0 ? 1u : 0u);
                            umma_tf32_ts(tbase + kColsD, tbase + kColsAhi + 8 * j, dl, 1u);
                            umma_tf32_ts(tbase + kColsD, tbase + kColsAhi + 8 * j, dh, 1u);
                        }
                        umma_commit(&s_dfull[group]);
                    }
                }
                __syncwarp();
                pending = true;
                plive = live;
                pe0 = e0;
                pt0 = t0;
            } else {
                break;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s_tmem), "r"(kTmemCols));
}

int* g_umma_err = nullptr;

// =================================================================================================================
// Backward of the same layer (32 -> 32, dense [E][b][32] tensors):
//
//   AG      = [G | S0 G | S1 G]                          (the forward's gather, on G = dL/dZ; S0, S1 are symmetric)
//   Gprev   = (AG [W0^T; W1^T; W2^T]) * act'(Hin)        per row
//   dW_term = Hin^T AG_term                              summed over all E * b rows              scone_trajectory_model.py:307
//
// A warp owns a slab of 16 rows as in the forward kernels.  The row product AG W^T contracts over channels — the gathered
// registers are its mma A fragments (3xTF32 mma.sync, the slab kernel's product with transposed weight fragments).  The weight
// gradient contracts over ROWS, which no register fragment layout offers: the warp writes its slab of AG (96 columns) and of Hin
// (32 columns), split hi / lo, into its private shared-memory buffers in the K-major canonical (no-swizzle) UMMA layout with
// K = the 16 rows, and one lane issues 6 tcgen05.mma.kind::tf32 (M = 128: AG column, 96 used; N = 32: Hin channel; K = 8 rows
// each; A_lo B_hi + A_hi B_lo + A_hi B_hi) that ACCUMULATE into the warp's own 32 TMEM columns for the whole kernel — the weight
// gradient never touches registers or shared memory until the end, when warps 0..2 read term 0..2 (TMEM lanes 32 term .. + 31)
// of every warp's accumulator, add them in warp order and write the CTA's partial; a second kernel folds the CTA partials in
// CTA order.  Static slab -> warp -> CTA assignment: deterministic.  No CTA barrier in the slab loop: a warp only waits for its
// own previous commit (one gather earlier) before it overwrites its buffers.
// Buffer strides are padded (core-matrix pitch 144 B, k-chunk pitch = 8 words mod 32) so that the fragment-layout stores of a
// warp hit 32 different banks.
// =================================================================================================================
constexpr int kBwdWarps = 12;              // warps per CTA: their operand buffers (BwdBuf) fill the shared memory
constexpr int kBwdGatherDepth = 4;         // neighbour rows in flight per warp (measured faster than 6 or 8)
constexpr int kFlushTiles = 32;            // slabs per warp between two flushes of the TMEM accumulators
constexpr int kDW = 3 * kC * kC;

// Accumulator row m (TMEM lane) <-> AG column: m = 32 term + 8 s + 4 h + tig holds column co = 16 h + 4 tig + s of term `term` (the
// fragment value a lane keeps for k-step s, half h): the four lanes of a quad write four consecutive rows of ONE core matrix, so
// with the k-chunk pitch at 16 banks mod 32 every fragment store of a warp hits 32 different banks at the canonical 128-byte
// core-matrix pitch (16.6 KB per warp: 12 warps + 24 KB of weight fragments fill the 227 KB of shared memory)
struct BwdBuf {
    static constexpr uint32_t SBO_A = 128u;                         // bytes between core matrices adjacent in M (8 accumulator rows)
    static constexpr uint32_t LBO_A = 1600u;                        // ... adjacent in K (row / 4): 12 core matrices of M + 64 B (16 banks)
    static constexpr uint32_t A_BYTES = 4u * LBO_A;                 // 16 rows = 4 k-chunks  (M rows 96..127 of the MMA read on into
    static constexpr uint32_t SBO_B = 128u;                         //  the next buffer of the same warp: their D lanes are never read)
    static constexpr uint32_t LBO_B = 528u;
    static constexpr uint32_t B_BYTES = 4u * LBO_B;
    static constexpr uint32_t WARP_BYTES = 2u * A_BYTES + 2u * B_BYTES;      // [A_hi | A_lo | B_hi | B_lo]
};
constexpr uint32_t kBwdBfBytes = 3u * 4u * 4u * 32u * 16u;          // weight fragments of the transposed product: [3][KS][NT][32] uint4

__device__ __forceinline__ uint64_t umma_desc2(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
           ((uint64_t)1 << 46);
}
__device__ __forceinline__ void umma_tf32_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(kIdesc), "r"(accumulate), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void tc_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {      // thread i <- TMEM lane base + i, 32 columns
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, "
        "%19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

template <int ACT>
__device__ __forceinline__ float umma_dact(float h) {               // derivative through the OUTPUT h = act(z)
    if (ACT == SCONE_ACT_TANH) return 1.f - h * h;
    if (ACT == SCONE_ACT_LEAKY_RELU) return h >= 0.f ? 1.f : 0.01f;
    return h > 0.f ? 1.f : 0.f;
}

template <int ACT, bool WG>
__global__ void __launch_bounds__(kBwdWarps * 32, 1) layer_bwd_umma_kernel(const float* __restrict__ Gd, const float* Hin, float* Gprev,
                                                                           const float* __restrict__ W0, const float* __restrict__ W1,
                                                                           const float* __restrict__ W2, float* __restrict__ ws,
                                                                           const int32_t* __restrict__ mptr, const int2* __restrict__ ment,
                                                                           int E, int b, int* __restrict__ err) {
    constexpr int TS = 16, NW = kBwdWarps;
    using G = SlabGeom<kC, TS>;
    using L = BwdBuf;
    constexpr int NT = kC / 8;
    extern __shared__ __align__(128) unsigned char bw_smem[];
    __shared__ __align__(8) uint64_t s_bar[NW];
    __shared__ int s_used[NW];
    __shared__ uint32_t s_tmem;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tig = lane & 3, g = lane >> 2;
    uint4* Bf = reinterpret_cast<uint4*>(bw_smem);

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (threadIdx.x < NW) {
        mbar_init(&s_bar[threadIdx.x], 1);
        s_used[threadIdx.x] = 0;
    }
    if (WG) stage_weight_fragments<kC, kC, TS, true>(Bf, W0, W1, W2);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const uint32_t a_hi = smem_u32(bw_smem) + kBwdBfBytes + (uint32_t)warp * L::WARP_BYTES, a_lo = a_hi + L::A_BYTES;
    const uint32_t b_hi = a_lo + L::A_BYTES, b_lo = b_hi + L::B_BYTES;
    // fragment value (row g + 8 r, AG column 16 h + 4 tig + s of term) -> k-chunk (g >> 2) + 2 r, core matrix 4 term + s, row 4 h + tig of
    // the core matrix, word g & 3;   Hin value (row g + 8 r, channel 8 nt + 2 tig + j) -> core matrix nt, row 2 tig + j
    const uint32_t lane_a = (uint32_t)(g >> 2) * L::LBO_A + (uint32_t)tig * 16u + (uint32_t)(g & 3) * 4u;
    const uint32_t lane_b = (uint32_t)(g >> 2) * L::LBO_B + (uint32_t)tig * 32u + (uint32_t)(g & 3) * 4u;
    const uint32_t tmem_d = s_tmem + (uint32_t)warp * 32u;
    // the stores go through generic shared-memory pointers (one base register per buffer, immediate offsets)
    unsigned char* const wbuf = bw_smem + kBwdBfBytes + (size_t)warp * L::WARP_BYTES;
    unsigned char* const pa_hi = wbuf + lane_a;
    unsigned char* const pa_lo = pa_hi + L::A_BYTES;
    unsigned char* const pb_hi = wbuf + 2u * L::A_BYTES + lane_b;
    unsigned char* const pb_lo = pb_hi + L::B_BYTES;

    const unsigned rowbytes = (unsigned)b * kC * 4u;
    const size_t rowlen = (size_t)b * kC;
    const int n_ts = b / TS;
    const int tiles_per_ts = (E + NW - 1) / NW;                          // a CTA tile = NW consecutive edges x one slab of 16 trajectories
    const long long n_tiles = (long long)n_ts * tiles_per_ts;
    // Tile -> CTA, static and interleaved: CTA i takes tiles i, i + grid, ...: at any time the CTAs work on ~grid x NW consecutive edges
    // of one trajectory slab, every neighbour row comes from DRAM once and is an L2 hit for its other ~13 uses (the operand buffers
    // leave ~16 KB of L1: contiguous tile ranges per CTA, which live on L1 reuse, gave L1 14 % / L2 54 % hits and 1.97 x the
    // compulsory DRAM reads here).
    const long long lo = blockIdx.x, hi = n_tiles, step = gridDim.x;
    // this warp's share of the flushes: TMEM lane quarter q = warp & 3 (term q of the stacked gradient) of the accumulators
    // j = warp >> 2, + nq, ... (nq = warps of this quarter); its running fp32 sums live in ws[cta][warp >> 2][term q][ci][co = lane]
    const int fq = warp & 3, fidx = warp >> 2, fnq = (NW - fq + 3) / 4;
    // TMEM lane 32 fq + lane = accumulator row 8 s + 4 h + tig (s = lane >> 3, h = (lane >> 2) & 1, tig = lane & 3) of term fq
    float* fdst = ws + ((size_t)blockIdx.x * 3 + fidx) * kDW + fq * kC * kC + (16 * ((lane >> 2) & 1) + 4 * (lane & 3) + (lane >> 3));
    for (int i = threadIdx.x; i < 3 * kDW; i += NW * 32) ws[(size_t)blockIdx.x * 3 * kDW + i] = 0.f;      // (visible after the flush's barrier)
    uint32_t phase = 0;
    bool pending = false, fresh = true;                                  // MMAs not yet waited for / accumulator holds nothing
    int it = 0;
    for (long long tile = lo; tile < hi; tile += step, ++it) {
        const int ts = (int)(tile / tiles_per_ts);
        const int e0 = (int)(tile - (long long)ts * tiles_per_ts) * NW + warp, t0 = ts * TS;
        if (e0 < E) {
        float2 hv[2][NT];                                                // own rows of Hin in the mma C-fragment layout
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            int e, t;
            slab_row<kC, TS>(r, e0, t0, e, t);
            const float* src = Hin + (size_t)e * rowlen + (size_t)t * kC + 2 * tig;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) hv[r][nt] = *reinterpret_cast<const float2*>(src + nt * 8);
        }
        u64 acc[3][G::NL][2];
        slab_gather<kC, TS, kBwdGatherDepth>(Gd, rowbytes, mptr, ment, E, b, e0, t0, acc);
        if (pending) {                                                   // the MMAs of the previous slab have read the buffers
            mbar_wait(&s_bar[warp], phase, err);
            phase ^= 1u;
        }
        float d[NT][4];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) d[nt][0] = d[nt][1] = d[nt][2] = d[nt][3] = 0.f;
#pragma unroll
        for (int term = 0; term < 3; ++term) {
            float fr[G::KS][4];
            slab_fragments<kC, TS>(acc[term], fr);
            if (WG) slab_mma_term<G::KS, NT>(d, fr, Bf + term * G::KS * NT * 32);
#pragma unroll
            for (int s = 0; s < G::KS; ++s)
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    uint32_t vh, vl;
                    split_tf32(fr[s][q], vh, vl);
                    const uint32_t off = (uint32_t)(q & 1) * 2u * L::LBO_A + (uint32_t)(4 * term + s) * L::SBO_A + (uint32_t)(q >> 1) * 64u;
                    *reinterpret_cast<uint32_t*>(pa_hi + off) = vh;
                    *reinterpret_cast<uint32_t*>(pa_lo + off) = vl;
                }
        }
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                uint32_t xh, xl, yh, yl;
                split_tf32(hv[r][nt].x, xh, xl);
                split_tf32(hv[r][nt].y, yh, yl);
                const uint32_t off = (uint32_t)r * 2u * L::LBO_B + (uint32_t)nt * L::SBO_B;
                *reinterpret_cast<uint32_t*>(pb_hi + off) = xh;
                *reinterpret_cast<uint32_t*>(pb_lo + off) = xl;
                *reinterpret_cast<uint32_t*>(pb_hi + off + 16u) = yh;
                *reinterpret_cast<uint32_t*>(pb_lo + off + 16u) = yl;
            }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy stores -> the tensor core's async proxy
        __syncwarp();
        if (lane == 0) {
            tc_fence_after();
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {                             // K = 16 rows in two steps of 8 (two 16-byte k-chunks each)
                const uint64_t dah = umma_desc2(a_hi + (uint32_t)ks * 2u * L::LBO_A, L::LBO_A, L::SBO_A);
                const uint64_t dal = umma_desc2(a_lo + (uint32_t)ks * 2u * L::LBO_A, L::LBO_A, L::SBO_A);
                const uint64_t dbh = umma_desc2(b_hi + (uint32_t)ks * 2u * L::LBO_B, L::LBO_B, L::SBO_B);
                const uint64_t dbl = umma_desc2(b_lo + (uint32_t)ks * 2u * L::LBO_B, L::LBO_B, L::SBO_B);
                umma_tf32_ss(tmem_d, dal, dbh, (!fresh || ks > 0) ? 1u : 0u);
                umma_tf32_ss(tmem_d, dah, dbl, 1u);
                umma_tf32_ss(tmem_d, dah, dbh, 1u);
            }
            umma_commit(&s_bar[warp]);
        }
        __syncwarp();
        pending = true;
        fresh = false;
        if (WG) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                int e, t;
                slab_row<kC, TS>(r, e0, t0, e, t);
                float* dst = Gprev + (size_t)e * rowlen + (size_t)t * kC + 2 * tig;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
                    *reinterpret_cast<float2*>(dst + nt * 8) =
                        make_float2(d[nt][2 * r] * umma_dact<ACT>(hv[r][nt].x), d[nt][2 * r + 1] * umma_dact<ACT>(hv[r][nt].y));
            }
        }
        }
        // Flush every kFlushTiles slabs: the tensor core's fp32 accumulation rounds towards zero, so a chain of n accumulations drifts
        // by ~n ulp (measured: 6.6e-5 of max |dW| after 3600 accumulations, 4.6e-6 for the fp32 SIMT kernel); chains of 6 kFlushTiles
        // accumulations are folded into fp32 sums with round-to-nearest adds.  CTA-uniform condition.
        if (it % kFlushTiles == kFlushTiles - 1 || tile + step >= hi) {
            if (pending) {
                mbar_wait(&s_bar[warp], phase, err);
                phase ^= 1u;
                pending = false;
            }
            if (lane == 0) s_used[warp] = fresh ? 0 : 1;
            tc_fence_before();
            __syncthreads();
            tc_fence_after();
            if (fq < 3) {
                float sum[kC];
#pragma unroll
                for (int j = 0; j < kC; ++j) sum[j] = 0.f;
                for (int w = fidx; w < NW; w += fnq) {
                    if (!s_used[w]) continue;                            // (warp-uniform)
                    uint32_t r[32];
                    tc_ld_32x32b_x32(s_tmem + (uint32_t)w * 32u + ((uint32_t)(32 * fq) << 16), r);
#pragma unroll
                    for (int j = 0; j < kC; ++j) sum[j] += __uint_as_float(r[j]);
                }
#pragma unroll
                for (int j = 0; j < kC; ++j) fdst[j * kC] += sum[j];     // dW[term][ci = j][co of this lane]; this thread's own running sum
            }
            tc_fence_before();
            __syncthreads();
            tc_fence_after();
            fresh = true;
        }
    }
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(s_tmem), "r"(kTmemCols));
}

// CTA partials -> dW in CTA order (8 slices of ascending parts, combined in slice order: a fixed tree)
__global__ void __launch_bounds__(256) umma_reduce_partials_kernel(const float* __restrict__ partial, int nparts, int n,
                                                                  float* __restrict__ out, int accumulate) {
    __shared__ float red[8][32];
    const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;
    const int per = (nparts + 7) / 8;
    const int p0 = slice * per, p1 = min(nparts, p0 + per);
    float s = 0.f;
    if (i < n)
        for (int p = p0; p < p1; ++p) s += partial[(size_t)p * n + i];
    red[slice][lane] = s;
    __syncthreads();
    if (slice == 0 && i < n) {
        float t = red[0][lane];
#pragma unroll
        for (int k = 1; k < 8; ++k) t += red[k][lane];
        out[i] = accumulate ? out[i] + t : t;
    }
}

template <int ACT, bool WG>
int launch_bwd_umma(const scone_complex* cx, int b, const float* G, const float* Hin, const float* W0, const float* W1, const float* W2,
                    float* Gprev, float* ws, int* grid_out, cudaStream_t st) {
    const size_t smem = (size_t)kBwdBfBytes + (size_t)kBwdWarps * BwdBuf::WARP_BYTES;
    auto kern = layer_bwd_umma_kernel<ACT, WG>;
    static bool configured = false;
    if (!configured) {
        SCONE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    const long long n_tiles = (long long)(b / 16) * ((cx->E + kBwdWarps - 1) / kBwdWarps);
    const int grid = (int)(n_tiles < cx->num_sms ? n_tiles : cx->num_sms);
    *grid_out = grid;
    kern<<<grid, kBwdWarps * 32, smem, st>>>(G, Hin, Gprev, W0, W1, W2, ws, cx->d_mptr, cx->d_ment, cx->E, b, g_umma_err);
    SCONE_LAUNCHED();
    return 0;
}

}  // namespace

bool scone_umma_supported(const scone_complex* cx, int cin, int cout, int b) {
    return cx->d_mptr != nullptr && cin == 32 && cout == 32 && b % 16 == 0;
}

// Hout = act(Hin W0 + (S0 Hin) W1 + (S1 Hin) W2) over dense [E][b][32] tensors.  Returns 3 if the kernel reported a tcgen05 protocol
// time-out on an earlier launch (checked lazily: the flag of the PREVIOUS launch is read, so the call itself stays asynchronous).
int scone_umma_forward(const scone_complex* cx, int act, int b, const float* Hin, const float* W0, const float* W1, const float* W2,
                       float* Hout, cudaStream_t st) {
    if (!g_umma_err) {
        SCONE_CUDA(cudaMalloc((void**)&g_umma_err, sizeof(int)));
        SCONE_CUDA(cudaMemset(g_umma_err, 0, sizeof(int)));
    }
    const int n_ts = (b + 15) / 16;
    const long long n_tiles = (long long)n_ts * ((cx->E + kGatherWarps - 1) / kGatherWarps);
    const int grid = (int)(n_tiles < cx->num_sms ? n_tiles : cx->num_sms);
    switch (act) {
        case SCONE_ACT_TANH:
            layer_fwd_umma_kernel<SCONE_ACT_TANH><<<grid, kUmmaThreads, 0, st>>>(Hin, Hout, W0, W1, W2, cx->d_mptr, cx->d_ment, cx->E, b, g_umma_err);
            break;
        case SCONE_ACT_LEAKY_RELU:
            layer_fwd_umma_kernel<SCONE_ACT_LEAKY_RELU><<<grid, kUmmaThreads, 0, st>>>(Hin, Hout, W0, W1, W2, cx->d_mptr, cx->d_ment, cx->E, b, g_umma_err);
            break;
        case SCONE_ACT_RELU:
            layer_fwd_umma_kernel<SCONE_ACT_RELU><<<grid, kUmmaThreads, 0, st>>>(Hin, Hout, W0, W1, W2, cx->d_mptr, cx->d_ment, cx->E, b, g_umma_err);
            break;
        default:
            scone_set_error("unknown activation %d", act);
            return 2;
    }
    SCONE_LAUNCHED();
    return 0;
}

// Gprev = (AG W^T) * act'(Hin) (skipped when Gprev == NULL), dW [3][32][32] (+)= Hin^T AG over dense [E][b][32] tensors; workspace:
// 3 x grid x 3072 floats.  Asynchronous; a tcgen05 protocol time-out is reported by scone_umma_check like the forward kernel's.
int scone_umma_backward(const scone_complex* cx, int act, int b, const float* G, const float* Hin, const float* W0, const float* W1,
                        const float* W2, float* Gprev, float* dW, int accumulate, float* ws, cudaStream_t st) {
    if (!g_umma_err) {
        SCONE_CUDA(cudaMalloc((void**)&g_umma_err, sizeof(int)));
        SCONE_CUDA(cudaMemset(g_umma_err, 0, sizeof(int)));
    }
    int rc = 2, grid = 0;
#define SCONE_UMMA_BWD(A)                                                                                                      \
    case A:                                                                                                                    \
        rc = Gprev ? launch_bwd_umma<A, true>(cx, b, G, Hin, W0, W1, W2, Gprev, ws, &grid, st)                                  \
                   : launch_bwd_umma<A, false>(cx, b, G, Hin, W0, W1, W2, Gprev, ws, &grid, st);                                \
        break;
    switch (act) {
        SCONE_UMMA_BWD(SCONE_ACT_TANH)
        SCONE_UMMA_BWD(SCONE_ACT_LEAKY_RELU)
        SCONE_UMMA_BWD(SCONE_ACT_RELU)
        default:
            scone_set_error("unknown activation %d", act);
            return 2;
    }
#undef SCONE_UMMA_BWD
    if (rc) return rc;
    umma_reduce_partials_kernel<<<(kDW + 31) / 32, 256, 0, st>>>(ws, 3 * grid, kDW, dW, accumulate);
    SCONE_LAUNCHED();
    return 0;
}

int scone_umma_check(cudaStream_t st) {
    if (!g_umma_err) return 0;
    int e = 0;
    SCONE_CUDA(cudaMemcpyAsync(&e, g_umma_err, sizeof(int), cudaMemcpyDeviceToHost, st));
    SCONE_CUDA(cudaStreamSynchronize(st));
    if (e) {
        cudaMemset(g_umma_err, 0, sizeof(int));
        scone_set_error("layer_fwd_umma_kernel: an mbarrier wait timed out (tcgen05 protocol error); results of that launch are invalid");
        return 3;
    }
    return 0;
}
