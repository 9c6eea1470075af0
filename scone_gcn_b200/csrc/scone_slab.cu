// scone_slab.cu — "slab" kernels: the dense fused Hodge-Laplacian layer for widths 16 / 32 on sm_100a.
//
//   Hout = act(Hin W0 + (S0 Hin) W1 + (S1 Hin) W2)                           trajectory_experiments.py:145-149,163-167
//
// A warp owns a slab of 16 (edge, trajectory) rows = EPS edges x TS trajectories and runs gather -> product -> activation
// -> store on its own (no CTA barrier in the tile loop):
//   * gather: one pass over the MERGED operator row (S0 and S1 share their pattern: the off-diagonals of B2 B2^T are a
//     subset of those of B1^T B1, so one neighbour row load feeds both sums and the own row); every load is a warp-wide
//     512-byte contiguous 128-bit load; sums are accumulated with packed fma.rn.f32x2 (FFMA2) in ascending column order
//     (same order, same roundings as the scalar kernels: bit-identical gathers, no atomics);
//   * the accumulators ARE the mma.sync m16n8k8 A fragments: the lane <-> (row, channel) assignment of the loads is
//     chosen so that (width 16) no data movement at all, (width 32) one lane^4 exchange of half the registers puts every
//     lane's two fragment rows in place — the gathered rows never go through shared memory;
//   * product on the tensor cores with the 3xTF32 split (a = a_hi + a_lo, w = w_hi + w_lo; a_lo w_hi + a_hi w_lo +
//     a_hi w_hi, fp32 accumulate): fp32-grade accuracy (plain TF32 would break the 1e-5 tolerance); the weight fragments
//     (hi, lo) sit in shared memory in fragment order, one conflict-free 128-bit load per (term, k-step, n-tile);
//   * activation in registers, 64-bit stores that fill whole 32-byte sectors.
// CTAs are persistent (one per SM, 16 warps) and walk CONTIGUOUS ranges of tiles along the locality edge order inside one
// trajectory slab, so the neighbour rows of consecutive edges are served by the SM's L1.
#include <cstdlib>
#include "common.cuh"

namespace {

#include "slab_common.cuh"

template <int CIN, int COUT, int ACT, int TS>
__global__ void __launch_bounds__(kSlabThreads, 1) layer_fwd_slab_kernel(const float* __restrict__ Hin, float* __restrict__ Hout,
                                                                        const float* __restrict__ W0, const float* __restrict__ W1,
                                                                        const float* __restrict__ W2, const int32_t* __restrict__ mptr,
                                                                        const int2* __restrict__ ment, int E, int b) {
    using G = SlabGeom<CIN, TS>;
    constexpr int NT = COUT / 8;
    extern __shared__ __align__(16) uint4 Bf[];           // [3][KS][NT][32]
    stage_weight_fragments<CIN, COUT, TS, false>(Bf, W0, W1, W2);
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tig = lane & 3;
    const unsigned rowbytes_in = (unsigned)b * CIN * 4u;
    const size_t rowlen_out = (size_t)b * COUT;
    const int n_ts = (b + TS - 1) / TS;
    const int n_eg = (E + G::EPS - 1) / G::EPS;                          // edge groups (slabs per trajectory slab)
    const int tiles_per_ts = (n_eg + kSlabWarps - 1) / kSlabWarps;       // a tile = kSlabWarps consecutive edge groups
    const long long n_tiles = (long long)n_ts * tiles_per_ts;
    const long long per = (n_tiles + gridDim.x - 1) / gridDim.x;
    const long long lo = (long long)blockIdx.x * per, hi = lo + per < n_tiles ? lo + per : n_tiles;
    for (long long tile = lo; tile < hi; ++tile) {
        const int ts = (int)(tile / tiles_per_ts);
        const int eg = (int)(tile - (long long)ts * tiles_per_ts) * kSlabWarps + warp;
        if (eg >= n_eg) continue;
        const int e0 = eg * G::EPS, t0 = ts * TS;
        u64 acc[3][G::NL][2];
        slab_gather<CIN, TS>(Hin, rowbytes_in, mptr, ment, E, b, e0, t0, acc);
        float d[NT][4];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) d[nt][0] = d[nt][1] = d[nt][2] = d[nt][3] = 0.f;
#pragma unroll
        for (int term = 0; term < 3; ++term) {
            float fr[G::KS][4];
            slab_fragments<CIN, TS>(acc[term], fr);
            slab_mma_term<G::KS, NT>(d, fr, Bf + term * G::KS * NT * 32);
        }
        slab_activate<ACT, NT>(d);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            int e, t;
            slab_row<CIN, TS>(r, e0, t0, e, t);
            if (e < E && t < b) {
                float* dst = Hout + (size_t)e * rowlen_out + (size_t)t * COUT + 2 * tig;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
                    *reinterpret_cast<float2*>(dst + nt * 8) = make_float2(d[nt][2 * r], d[nt][2 * r + 1]);
            }
        }
    }
}

template <int CIN, int COUT, int ACT, int TS>
int launch_fwd_slab(const scone_complex* cx, int b, const float* Hin, const float* W0, const float* W1, const float* W2, float* Hout,
                    cudaStream_t st) {
    using G = SlabGeom<CIN, TS>;
    constexpr int NT = COUT / 8;
    const size_t smem = (size_t)3 * G::KS * NT * 32 * sizeof(uint4);
    auto kern = layer_fwd_slab_kernel<CIN, COUT, ACT, TS>;
    static bool configured = false;
    if (!configured) {
        SCONE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    const int n_ts = (b + TS - 1) / TS, n_eg = (cx->E + G::EPS - 1) / G::EPS;
    const long long n_tiles = (long long)n_ts * ((n_eg + kSlabWarps - 1) / kSlabWarps);
    const int grid = (int)(n_tiles < cx->num_sms ? n_tiles : cx->num_sms);
    kern<<<grid, kSlabThreads, smem, st>>>(Hin, Hout, W0, W1, W2, cx->d_mptr, cx->d_ment, cx->E, b);
    SCONE_LAUNCHED();
    return 0;
}

template <int CIN, int COUT, int ACT>
int dispatch_fwd_ts(const scone_complex* cx, int ts, int b, const float* Hin, const float* W0, const float* W1, const float* W2,
                    float* Hout, cudaStream_t st) {
    if (ts == 8) return launch_fwd_slab<CIN, COUT, ACT, 8>(cx, b, Hin, W0, W1, W2, Hout, st);
    return launch_fwd_slab<CIN, COUT, ACT, 16>(cx, b, Hin, W0, W1, W2, Hout, st);
}

template <int CIN, int COUT>
int dispatch_fwd_act(const scone_complex* cx, int act, int ts, int b, const float* Hin, const float* W0, const float* W1,
                     const float* W2, float* Hout, cudaStream_t st) {
    switch (act) {
        case SCONE_ACT_TANH: return dispatch_fwd_ts<CIN, COUT, SCONE_ACT_TANH>(cx, ts, b, Hin, W0, W1, W2, Hout, st);
        case SCONE_ACT_LEAKY_RELU: return dispatch_fwd_ts<CIN, COUT, SCONE_ACT_LEAKY_RELU>(cx, ts, b, Hin, W0, W1, W2, Hout, st);
        case SCONE_ACT_RELU: return dispatch_fwd_ts<CIN, COUT, SCONE_ACT_RELU>(cx, ts, b, Hin, W0, W1, W2, Hout, st);
    }
    scone_set_error("unknown activation %d", act);
    return 2;
}

// =================================================================================================================
// Row-list forward (occupancy flags given): the same gather -> fragments -> 3xTF32 product pipeline on a COMPACTED list of
// candidate rows.  rows[] holds the ids e*b + t of the rows of Hout that can be non-zero (ascending: the output's row
// bitmap compacted by compact_bitmap_kernel); a warp takes 16 consecutive list entries.  Lane group q (the LPR = C/4 lanes
// that cover one row) walks the merged operator row of ITS row; a neighbour row is loaded only if its flag byte in occ_in
// (or, in the bitmap pipeline, its bit in bm_in) is set (unflagged rows are exact zeros and, in the model-level
// pipelines, may never have been written).  All 16 rows' k-th
// neighbours are in flight together.  Each row's result is independent of the other rows in its slab and uses the same
// summation order and mma sequence as the dense slab kernel: bit-identical to it.
// =================================================================================================================
// COMPACT (with BITS): tensors are stored compactly — row r of Hin at index rank(r) in (bm_in, pref_in), row rows[i] of Hout at
// index i — so memory and traffic follow the support and a micro-batch can hold thousands of trajectories.
template <int CIN, int COUT, int ACT, bool BITS, bool COMPACT>
__global__ void __launch_bounds__(kRowsThreads, 1) layer_fwd_rows_kernel(const float* __restrict__ Hin, float* __restrict__ Hout,
                                                                        const float* __restrict__ W0, const float* __restrict__ W1,
                                                                        const float* __restrict__ W2, const int32_t* __restrict__ mptr,
                                                                        const int2* __restrict__ ment, const uint8_t* __restrict__ occ_in,
                                                                        const uint32_t* __restrict__ rows, const int* __restrict__ n_ptr,
                                                                        int b, unsigned long long* __restrict__ row_counter,
                                                                        const uint32_t* __restrict__ bm_in,
                                                                        const uint32_t* __restrict__ pref_in, int out_cap,
                                                                        int* __restrict__ overflow, int E) {
    static_assert(!COMPACT || BITS, "compact storage is addressed through the row bitmaps");
    using G = SlabGeom<CIN, 16>;
    constexpr int NT = COUT / 8, NL = G::NL, Q = G::Q, LPR = CIN / 4;      // Q rows per warp-wide load, LPR lanes per row
    extern __shared__ __align__(16) uint4 Bf[];
    stage_weight_fragments<CIN, COUT, 16, false>(Bf, W0, W1, W2);
    __syncthreads();
    const int lane = threadIdx.x & 31, tig = lane & 3, g = lane >> 2;
    const int gq = lane / LPR, cq = lane % LPR;
    const unsigned rowbytes = COMPACT ? CIN * 4u : (unsigned)b * CIN * 4u;    // stride of the gather index (compact row / edge row)
    const char* Hb = reinterpret_cast<const char*>(Hin);
    int n = *n_ptr;
    if (COMPACT && n > out_cap) {                          // the compact output cannot hold this many rows: flag it (host raises)
        if (blockIdx.x == 0 && threadIdx.x == 0) *overflow = 1;
        n = out_cap;
    }
    const int n_slabs = (n + 15) / 16;
    const int n_minis = (n_slabs + kRowsMini - 1) / kRowsMini;
    if (row_counter != nullptr && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(row_counter, (unsigned long long)n);
    // every WARP takes kRowsMini consecutive slabs at a time from a global counter (n_ptr[1], zeroed by the compaction kernel): slab
    // cost varies (longest merged row of its 16 rows, cache misses); a static split left SMs idle for a third of the kernel and
    // CTA-wide tiles made 15 warps wait for the slowest at every tile.  Consecutive slabs stay in one warp: their rows are
    // neighbours (same trajectory, nearby edges) and share gathered rows through L1.
    int* tile_counter = const_cast<int*>(n_ptr) + 1;
    for (;;) {
        int mini = 0;
        if (lane == 0) mini = atomicAdd(tile_counter, 1);
        mini = __shfl_sync(0xffffffffu, mini, 0);
        if (mini >= n_minis) break;
        const int slab_end = min(n_slabs, (mini + 1) * kRowsMini);
        for (int slab = mini * kRowsMini; slab < slab_end; ++slab) {
        // this lane's row in each load slot
        uint32_t rid[NL];
        unsigned oidx[NL];                                 // index of the own row in Hin's storage
        int len[NL], p0[NL], tq[NL];
        const char* P[NL];
        bool own[NL];
        int maxlen = 0;
#pragma unroll
        for (int i = 0; i < NL; ++i) {
            const int li = slab * 16 + i * Q + gq;
            const bool valid = li < n;
            rid[i] = valid ? __ldg(rows + li) : 0u;
            const RowIds<COMPACT> ids(rid[i], b, E);
            const int e = (int)ids.e;
            tq[i] = (int)ids.toff;                         // e-major: t; trajectory-major (compact): t * E
            const int cpos = (CIN == 32 && i >= 2) ? (cq ^ 4) : cq;
            P[i] = Hb + (size_t)((unsigned)((COMPACT ? 0 : tq[i] * CIN) + 4 * cpos) * 4u);
            asm volatile("" : "+l"(P[i]));                 // keep base + lane offset folded: one IMAD.WIDE per load address
            p0[i] = valid ? __ldg(mptr + e) : 0;
            len[i] = valid ? __ldg(mptr + e + 1) - p0[i] : 0;
            if (COMPACT) {
                own[i] = rank_lookup(bm_in, pref_in, rid[i], oidx[i]) && valid;
            } else {
                oidx[i] = (unsigned)e;
                own[i] = valid && (BITS ? bit_test(bm_in, rid[i]) : __ldg(occ_in + rid[i]) != 0);
            }
            maxlen = max(maxlen, len[i]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) maxlen = max(maxlen, __shfl_xor_sync(0xffffffffu, maxlen, o));
        u64 acc[3][NL][2];
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int i = 0; i < NL; ++i) acc[k][i][0] = acc[k][i][1] = 0ull;
#pragma unroll
        for (int i = 0; i < NL; ++i)
            if (own[i]) ldg128(reinterpret_cast<const float*>(P[i] + (size_t)oidx[i] * rowbytes), acc[0][i][0], acc[0][i][1]);
#pragma unroll 2
        for (int k = 0; k < maxlen; ++k) {
            int2 ent[NL];
            bool on[NL];
#pragma unroll
            for (int i = 0; i < NL; ++i) {
                on[i] = k < len[i];
                ent[i] = on[i] ? __ldg(ment + p0[i] + k) : make_int2(0, 0);
            }
            unsigned gidx[NL];                             // gather index of the neighbour row: its edge, or its compact rank
#pragma unroll
            for (int i = 0; i < NL; ++i) {                 // branch-free flag test (entry {0,0} of an idle lane tests row tq: in range)
                const unsigned nrow = RowIds<COMPACT>::row_of((unsigned)ent[i].x, (unsigned)tq[i], b);       // E*b < 2^32
                if (COMPACT) {
                    on[i] = rank_lookup(bm_in, pref_in, nrow, gidx[i]) && on[i];
                } else {
                    const unsigned f = BITS ? (__ldg(bm_in + (nrow >> 5)) >> (nrow & 31)) & 1u : (unsigned)__ldg(occ_in + nrow);
                    on[i] = on[i] && f != 0u;
                    gidx[i] = (unsigned)ent[i].x;
                }
            }
            u64 v[NL][2];
#pragma unroll
            for (int i = 0; i < NL; ++i) {
                v[i][0] = v[i][1] = 0ull;
                if (on[i]) ldg128(reinterpret_cast<const float*>(P[i] + (size_t)gidx[i] * rowbytes), v[i][0], v[i][1]);
            }
#pragma unroll
            for (int i = 0; i < NL; ++i) {
                const float c0 = (float)(short)(ent[i].y & 0xffff), c1 = (float)(ent[i].y >> 16);
                const u64 q0 = bcast2(c0), q1 = bcast2(c1);
                ffma2(acc[1][i][0], q0, v[i][0]);
                ffma2(acc[1][i][1], q0, v[i][1]);
                ffma2(acc[2][i][0], q1, v[i][0]);
                ffma2(acc[2][i][1], q1, v[i][1]);
            }
        }
        float d[NT][4];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) d[nt][0] = d[nt][1] = d[nt][2] = d[nt][3] = 0.f;
#pragma unroll
        for (int term = 0; term < 3; ++term) {
            float fr[G::KS][4];
            slab_fragments<CIN, 16>(acc[term], fr);
            slab_mma_term<G::KS, NT>(d, fr, Bf + term * G::KS * NT * 32);
        }
        slab_activate<ACT, NT>(d);
        // fragment row r (0: row g, 1: row g + 8) is this lane's own row of slot 2*(g&1) + r (width 32) / slot r (width 16)
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            uint32_t orow;
            int oli;
            if (CIN == 32) {
                const bool odd = g & 1;
                orow = odd ? rid[2 + r] : rid[r];
                oli = slab * 16 + (odd ? 2 + r : r) * Q + gq;
            } else {
                orow = rid[r];
                oli = slab * 16 + r * Q + gq;
            }
            if (oli < n) {
                float* dst = Hout + (size_t)(COMPACT ? (uint32_t)oli : orow) * COUT + 2 * tig;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) *reinterpret_cast<float2*>(dst + nt * 8) = make_float2(d[nt][2 * r], d[nt][2 * r + 1]);
            }
        }
        }
    }
}

template <int CIN, int COUT, int ACT>
int launch_fwd_rows(const scone_complex* cx, int b, const float* Hin, const float* W0, const float* W1, const float* W2, float* Hout,
                    const uint8_t* occ_in, const uint32_t* rows, const int* n_ptr, unsigned long long* row_counter,
                    const uint32_t* bm_in, const uint32_t* pref_in, int out_cap, int* overflow, cudaStream_t st) {
    using G = SlabGeom<CIN, 16>;
    constexpr int NT = COUT / 8;
    const size_t smem = (size_t)3 * G::KS * NT * 32 * sizeof(uint4);
    static bool configured = false;
    if (!configured) {
        SCONE_CUDA(cudaFuncSetAttribute(layer_fwd_rows_kernel<CIN, COUT, ACT, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SCONE_CUDA(cudaFuncSetAttribute(layer_fwd_rows_kernel<CIN, COUT, ACT, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SCONE_CUDA(cudaFuncSetAttribute(layer_fwd_rows_kernel<CIN, COUT, ACT, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
#define SCONE_ROWS_LAUNCH(BITS_, COMPACT_)                                                                                          \
    layer_fwd_rows_kernel<CIN, COUT, ACT, BITS_, COMPACT_><<<cx->num_sms, kRowsThreads, smem, st>>>(                                \
        Hin, Hout, W0, W1, W2, cx->d_mptr, cx->d_ment, occ_in, rows, n_ptr, b, row_counter, bm_in, pref_in, out_cap, overflow, cx->E)
    if (bm_in != nullptr && pref_in != nullptr) SCONE_ROWS_LAUNCH(true, true);
    else if (bm_in != nullptr) SCONE_ROWS_LAUNCH(true, false);
    else SCONE_ROWS_LAUNCH(false, false);
#undef SCONE_ROWS_LAUNCH
    SCONE_LAUNCHED();
    return 0;
}

template <int CIN, int COUT>
int dispatch_rows_act(const scone_complex* cx, int act, int b, const float* Hin, const float* W0, const float* W1, const float* W2,
                      float* Hout, const uint8_t* occ_in, const uint32_t* rows, const int* n_ptr, unsigned long long* rc,
                      const uint32_t* bm_in, const uint32_t* pref_in, int out_cap, int* overflow, cudaStream_t st) {
    switch (act) {
        case SCONE_ACT_TANH: return launch_fwd_rows<CIN, COUT, SCONE_ACT_TANH>(cx, b, Hin, W0, W1, W2, Hout, occ_in, rows, n_ptr, rc, bm_in, pref_in, out_cap, overflow, st);
        case SCONE_ACT_LEAKY_RELU: return launch_fwd_rows<CIN, COUT, SCONE_ACT_LEAKY_RELU>(cx, b, Hin, W0, W1, W2, Hout, occ_in, rows, n_ptr, rc, bm_in, pref_in, out_cap, overflow, st);
        case SCONE_ACT_RELU: return launch_fwd_rows<CIN, COUT, SCONE_ACT_RELU>(cx, b, Hin, W0, W1, W2, Hout, occ_in, rows, n_ptr, rc, bm_in, pref_in, out_cap, overflow, st);
    }
    scone_set_error("unknown activation %d", act);
    return 2;
}

}  // namespace

// Flagged fused layer forward over a compacted row list (see layer_fwd_rows_kernel); the caller checked scone_slab_supported.
int scone_slab_forward_rows(const scone_complex* cx, int act, int b, int cin, int cout, const float* Hin, const float* W0,
                            const float* W1, const float* W2, float* Hout, const uint8_t* occ_in, const uint32_t* rows,
                            const int* n_rows_dev, unsigned long long* row_counter, const uint32_t* bm_in, const uint32_t* pref_in,
                            int out_cap, int* overflow_dev, cudaStream_t st) {
#define SCONE_ROWS_CASE(CI, CO)                                                                                                 \
    if (cin == CI && cout == CO)                                                                                                \
        return dispatch_rows_act<CI, CO>(cx, act, b, Hin, W0, W1, W2, Hout, occ_in, rows, n_rows_dev, row_counter, bm_in, pref_in, out_cap, overflow_dev, st);
    SCONE_ROWS_CASE(16, 16)
    SCONE_ROWS_CASE(16, 32)
    SCONE_ROWS_CASE(32, 16)
    SCONE_ROWS_CASE(32, 32)
#undef SCONE_ROWS_CASE
    scone_set_error("scone_slab_forward_rows: unsupported widths %d -> %d", cin, cout);
    return 2;
}

int g_scone_dense_kernel = 3;   // 0: fp32 SIMT tile kernels; 1: slab kernels, 16 trajectories x 1 edge per slab; 2: slab, 8 x 2;
                                // 3: tcgen05 tiles of 128 rows for 32 -> 32 with b % 16 == 0 (scone_umma.cu), slab 16 x 1 elsewhere

bool scone_slab_supported(const scone_complex* cx, int cin, int cout) {
    return g_scone_dense_kernel != 0 && cx->d_mptr != nullptr && (cin == 16 || cin == 32) && (cout == 16 || cout == 32);
}

static int slab_ts() { return g_scone_dense_kernel == 2 ? 8 : 16; }

// Dense fused layer forward on the slab kernels; the caller checked scone_slab_supported.
int scone_slab_forward(const scone_complex* cx, int act, int b, int cin, int cout, const float* Hin, const float* W0, const float* W1,
                       const float* W2, float* Hout, cudaStream_t st) {
    if (g_scone_dense_kernel == 3 && scone_umma_supported(cx, cin, cout, b))      // tcgen05 / TMEM product (scone_umma.cu)
        return scone_umma_forward(cx, act, b, Hin, W0, W1, W2, Hout, st);
    const int ts = slab_ts();
    if (cin == 16 && cout == 16) return dispatch_fwd_act<16, 16>(cx, act, ts, b, Hin, W0, W1, W2, Hout, st);
    if (cin == 16 && cout == 32) return dispatch_fwd_act<16, 32>(cx, act, ts, b, Hin, W0, W1, W2, Hout, st);
    if (cin == 32 && cout == 16) return dispatch_fwd_act<32, 16>(cx, act, ts, b, Hin, W0, W1, W2, Hout, st);
    if (cin == 32 && cout == 32) return dispatch_fwd_act<32, 32>(cx, act, ts, b, Hin, W0, W1, W2, Hout, st);
    scone_set_error("scone_slab_forward: unsupported widths %d -> %d", cin, cout);
    return 2;
}

extern "C" int scone_set_dense_kernel(int32_t which) {
    SCONE_REQUIRE(which >= 0 && which <= 3, "scone_set_dense_kernel: 0 (fp32 SIMT tiles), 1 (slab 16x1), 2 (slab 8x2) or 3 (tcgen05 tiles)");
    g_scone_dense_kernel = which;
    return 0;
}
extern "C" int scone_get_dense_kernel(void) { return g_scone_dense_kernel; }
