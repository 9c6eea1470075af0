// scone_kernels.cu — hand-written sm_100a kernels of the SCoNe hot path.
//
//   Hout = act(Hin W0 + (S0 Hin) W1 + (S1 Hin) W2)                           trajectory_experiments.py:145-149,163-167
//   backward of the same (what jax.grad derives, scone_trajectory_model.py:307):
//       A_k = S_k G,  Gprev = (sum_k A_k W_k^T) * act'(Hin),  dW_k = Hin^T A_k      (S_k symmetric)
//   readout Bcond(last) @ H_L @ w_out, padded log-softmax, NLL + gradient       trajectory_experiments.py:151-152,298-303
//   JAX adam update                                                             scone_trajectory_model.py:300,310
//
// Layout: activations H[E][b][C] fp32 (e = internal edge row), one edge row = b*C contiguous floats.  Two kernel
// families implement the fused layer (DESIGN.md):
//   * DENSE tile kernels (no occupancy information): a CTA owns 128 (edge, trajectory) rows; every warp gathers whole
//     edge rows (1 + nnz(S0 row) + nnz(S1 row) neighbour rows, 128-bit coalesced loads, CSR order = fixed summation
//     order, no atomics) into shared memory, then the 3C x C weight products + sum + activation run as a
//     register-tiled contraction and are stored with 128-bit coalesced stores.
//   * UNIT kernels (occupancy flags given): there is no bias and act(0) = 0, so activations are exactly zero outside the
//     l-hop neighbourhood of a trajectory.  The flagged (edge, trajectory-chunk) units of the input are compacted into a
//     worklist (deterministic order), their support is scattered one hop into the output's flags, those are compacted
//     again, and one warp per candidate unit does a flag-aware gather + per-row contraction.  Skipping a zero row is exact.
// Weight gradients are accumulated in registers in a data-independent thread mapping and a fixed row order, written
// as per-CTA partials and reduced in CTA order: bit-reproducible run to run.
#include <math_constants.h>
#include <cstdlib>
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kTileRows = 128;      // (edge, trajectory) rows per dense tile
constexpr int kTileCols = 128;      // gathered columns per edge per warp pass (32 lanes x float4)

template <int ACT>
__device__ __forceinline__ float act_fn(float z) {
    if (ACT == SCONE_ACT_TANH) return tanhf(z);
    if (ACT == SCONE_ACT_LEAKY_RELU) return z >= 0.f ? z : 0.01f * z;
    return fmaxf(z, 0.f);
}
// derivative expressed through the OUTPUT h = act(z) (sign(z) == sign(h) for leaky-relu / relu)
template <int ACT>
__device__ __forceinline__ float dact_fn(float h) {
    if (ACT == SCONE_ACT_TANH) return 1.f - h * h;
    if (ACT == SCONE_ACT_LEAKY_RELU) return h >= 0.f ? 1.f : 0.01f;
    return h > 0.f ? 1.f : 0.f;
}
__device__ __forceinline__ float dact_rt(int act, float h) {
    if (act == SCONE_ACT_TANH) return 1.f - h * h;
    if (act == SCONE_ACT_LEAKY_RELU) return h >= 0.f ? 1.f : 0.01f;
    return h > 0.f ? 1.f : 0.f;
}

__device__ __forceinline__ void fma4(float4& a, float s, const float4& v) {
    a.x = fmaf(s, v.x, a.x);
    a.y = fmaf(s, v.y, a.y);
    a.z = fmaf(s, v.z, a.z);
    a.w = fmaf(s, v.w, a.w);
}
__device__ __forceinline__ bool nz4(const float4& v) { return v.x != 0.f || v.y != 0.f || v.z != 0.f || v.w != 0.f; }
__device__ __forceinline__ float4 zero4() { return make_float4(0.f, 0.f, 0.f, 0.f); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---------------------------------------------------------------------------------------------------------------
// Row gathers: sum_p coef_p * H[col_p][colofs .. colofs+3] over one CSR row, ascending column order.
// ---------------------------------------------------------------------------------------------------------------
// Dense flavour: every neighbour row is loaded; 4 independent 128-bit loads in flight.
__device__ __forceinline__ float4 gather_row4_dense(const float* __restrict__ H, size_t rowlen, int colofs, DevCsr S, int e) {
    float4 acc = zero4();
    int p = __ldg(S.rowptr + e);
    const int end = __ldg(S.rowptr + e + 1);
    for (; p + 4 <= end; p += 4) {
        int2 c0 = __ldg(S.ent + p), c1 = __ldg(S.ent + p + 1), c2 = __ldg(S.ent + p + 2), c3 = __ldg(S.ent + p + 3);
        float4 v0 = __ldg(reinterpret_cast<const float4*>(H + (size_t)c0.x * rowlen + colofs));
        float4 v1 = __ldg(reinterpret_cast<const float4*>(H + (size_t)c1.x * rowlen + colofs));
        float4 v2 = __ldg(reinterpret_cast<const float4*>(H + (size_t)c2.x * rowlen + colofs));
        float4 v3 = __ldg(reinterpret_cast<const float4*>(H + (size_t)c3.x * rowlen + colofs));
        fma4(acc, __int_as_float(c0.y), v0);
        fma4(acc, __int_as_float(c1.y), v1);
        fma4(acc, __int_as_float(c2.y), v2);
        fma4(acc, __int_as_float(c3.y), v3);
    }
    for (; p < end; ++p) {
        int2 c0 = __ldg(S.ent + p);
        float4 v0 = __ldg(reinterpret_cast<const float4*>(H + (size_t)c0.x * rowlen + colofs));
        fma4(acc, __int_as_float(c0.y), v0);
    }
    return acc;
}

// Flag-aware flavour: lanes fetch the row's (column, coefficient) entries in parallel and test whether neighbour row i
// has a non-zero among this unit's TT trajectories; the warp then loads only the flagged neighbour rows.
template <int TT>
__device__ __forceinline__ float4 gather_row4_flagged(const float* __restrict__ H, size_t rowlen, int colofs, bool colok, DevCsr S,
                                                      int e, const uint8_t* __restrict__ occ, int b, int t0, int jl) {
    float4 acc = zero4();
    const int lane = threadIdx.x & 31;
    const int p0 = __ldg(S.rowptr + e), p1 = __ldg(S.rowptr + e + 1);
    for (int base = p0; base < p1; base += 32) {
        const int idx = base + lane;
        int2 ent = make_int2(e, 0);
        unsigned fm = 0;                                  // bit k: trajectory t0+k of neighbour row `idx` is flagged
        if (idx < p1) {
            ent = __ldg(S.ent + idx);
            const uint8_t* f = occ + (size_t)ent.x * b + t0;
#pragma unroll
            for (int k = 0; k < TT; ++k)
                if (t0 + k < b && __ldg(f + k) != 0) fm |= 1u << k;
        }
        unsigned mask = __ballot_sync(0xffffffffu, fm != 0u);
        while (mask) {
            const int n = min(4, __popc(mask));          // warp-uniform
            float c[4];
            int col[4];
            bool mine[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (u < n) {
                    const int src = __ffs(mask) - 1;
                    mask &= mask - 1;
                    col[u] = __shfl_sync(0xffffffffu, ent.x, src);
                    c[u] = __int_as_float(__shfl_sync(0xffffffffu, ent.y, src));
                    const unsigned nfm = __shfl_sync(0xffffffffu, fm, src);      // (all lanes take part in the shuffle)
                    mine[u] = colok && ((nfm >> jl) & 1u);                       // unflagged rows are never read
                }
            }
            float4 v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (u < n && mine[u]) v[u] = __ldg(reinterpret_cast<const float4*>(H + (size_t)col[u] * rowlen + colofs));
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (u < n && mine[u]) fma4(acc, c[u], v[u]);
        }
    }
    return acc;
}

// scalar flavour for the flows X[E][b]
__device__ __forceinline__ float gather_row1(const float* __restrict__ X, int b, int t, DevCsr S, int e) {
    float acc = 0.f;
    int p = __ldg(S.rowptr + e);
    const int end = __ldg(S.rowptr + e + 1);
    for (; p < end; ++p) {
        int2 c0 = __ldg(S.ent + p);
        acc = fmaf(__int_as_float(c0.y), __ldg(X + (size_t)c0.x * b + t), acc);
    }
    return acc;
}

// ---------------------------------------------------------------------------------------------------------------
// Register-tiled contraction out[128][NOUT] = T[128][KD] * Wm[KD][NOUT] from shared memory (dense tile kernels).
// Thread (tx, ty): columns 4*tx .. 4*tx+3, rows ty + i*NRT (i < RT).
// ---------------------------------------------------------------------------------------------------------------
template <int KD, int NOUT, int LDT>
struct TileGemm {
    static constexpr int NTX = NOUT / 4;
    static constexpr int NRT = kThreads / NTX;
    static constexpr int RT = kTileRows / NRT;
    static_assert(NOUT % 4 == 0 && kThreads % NTX == 0 && kTileRows % NRT == 0, "tile shape");
    __device__ __forceinline__ static void run(const float* __restrict__ Ts, const float* __restrict__ Ws, float4 (&acc)[RT]) {
        const int tx = threadIdx.x % NTX, ty = threadIdx.x / NTX;
#pragma unroll
        for (int i = 0; i < RT; ++i) acc[i] = zero4();
#pragma unroll 2
        for (int kq = 0; kq < KD / 4; ++kq) {
            float4 w[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) w[q] = *reinterpret_cast<const float4*>(Ws + (4 * kq + q) * NOUT + 4 * tx);
#pragma unroll
            for (int i = 0; i < RT; ++i) {
                const float4 a = *reinterpret_cast<const float4*>(Ts + (ty + i * NRT) * LDT + 4 * kq);
                fma4(acc[i], a.x, w[0]);
                fma4(acc[i], a.y, w[1]);
                fma4(acc[i], a.z, w[2]);
                fma4(acc[i], a.w, w[3]);
            }
        }
    }
};

// One output row x 4 columns: out[rho][4tx..4tx+3] = T[rho][:] * Wm[:][4tx..4tx+3]   (unit kernels)
template <int KD, int NOUT, int LDT>
__device__ __forceinline__ float4 row_gemm(const float* __restrict__ Ts, const float* __restrict__ Ws, int rho, int tx) {
    float4 acc = zero4();
#pragma unroll 4
    for (int kq = 0; kq < KD / 4; ++kq) {
        const float4 a = *reinterpret_cast<const float4*>(Ts + rho * LDT + 4 * kq);
        const float4 w0 = *reinterpret_cast<const float4*>(Ws + (4 * kq + 0) * NOUT + 4 * tx);
        const float4 w1 = *reinterpret_cast<const float4*>(Ws + (4 * kq + 1) * NOUT + 4 * tx);
        const float4 w2 = *reinterpret_cast<const float4*>(Ws + (4 * kq + 2) * NOUT + 4 * tx);
        const float4 w3 = *reinterpret_cast<const float4*>(Ws + (4 * kq + 3) * NOUT + 4 * tx);
        fma4(acc, a.x, w0);
        fma4(acc, a.y, w1);
        fma4(acc, a.z, w2);
        fma4(acc, a.w, w3);
    }
    return acc;
}

// lanes [g*NTX, (g+1)*NTX) of a warp hold one row's outputs; the group's first lane stores the row's flag.
template <int NTX>
__device__ __forceinline__ void store_row_flag(uint8_t* __restrict__ occ_out, size_t pos, bool valid, bool nz) {
    const unsigned bal = __ballot_sync(0xffffffffu, nz);
    const int lane = threadIdx.x & 31;
    if (occ_out != nullptr && valid && (lane % NTX) == 0) {
        const unsigned grp = (bal >> (lane - lane % NTX)) & ((NTX >= 32) ? 0xffffffffu : ((1u << NTX) - 1u));
        occ_out[pos] = grp ? 1 : 0;
    }
}

// =================================================================================================================
// DENSE tile kernels
// =================================================================================================================
template <int CIN, int COUT, int ACT>
__global__ void __launch_bounds__(kThreads) layer_fwd_dense_kernel(const float* __restrict__ Hin, float* __restrict__ Hout,
                                                                  const float* __restrict__ W0, const float* __restrict__ W1,
                                                                  const float* __restrict__ W2, DevCsr S0, DevCsr S1, int E, int b) {
    constexpr int TT = kTileCols / CIN;      // trajectories per tile
    constexpr int TE = kTileRows / TT;       // edges per tile
    constexpr int KD = 3 * CIN, LDT = KD + 4;
    using Gemm = TileGemm<KD, COUT, LDT>;
    extern __shared__ __align__(16) float smem[];
    float* Ts = smem;                        // [128][LDT]
    float* Ws = smem + kTileRows * LDT;      // [KD][COUT]
    for (int i = threadIdx.x; i < CIN * COUT; i += kThreads) {
        Ws[i] = W0[i];
        Ws[CIN * COUT + i] = W1[i];
        Ws[2 * CIN * COUT + i] = W2[i];
    }
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const size_t rowlen_in = (size_t)b * CIN, rowlen_out = (size_t)b * COUT;
    const int n_tb = (b + TT - 1) / TT, n_eb = (E + TE - 1) / TE;
    const int jl = (4 * lane) / CIN, cil = (4 * lane) % CIN;
    const int tx = threadIdx.x % Gemm::NTX, ty = threadIdx.x / Gemm::NTX;
    for (int tile = blockIdx.x; tile < n_tb * n_eb; tile += gridDim.x) {
        const int tb = tile % n_tb, eb = tile / n_tb;
        const int e0 = eb * TE, t0 = tb * TT;
        const int colofs = tb * kTileCols + 4 * lane;
        const bool colok = colofs < (int)rowlen_in;
        __syncthreads();                      // previous tile's contraction done (and Ws visible)
        for (int r = warp; r < TE; r += kWarps) {
            const int e = e0 + r;
            float4 a0 = zero4(), a1 = a0, a2 = a0;
            if (e < E && colok) {
                a0 = __ldg(reinterpret_cast<const float4*>(Hin + (size_t)e * rowlen_in + colofs));
                a1 = gather_row4_dense(Hin, rowlen_in, colofs, S0, e);
                a2 = gather_row4_dense(Hin, rowlen_in, colofs, S1, e);
            }
            float* dst = Ts + (r * TT + jl) * LDT + cil;
            *reinterpret_cast<float4*>(dst) = a0;
            *reinterpret_cast<float4*>(dst + CIN) = a1;
            *reinterpret_cast<float4*>(dst + 2 * CIN) = a2;
        }
        __syncthreads();
        float4 acc[Gemm::RT];
        Gemm::run(Ts, Ws, acc);
#pragma unroll
        for (int i = 0; i < Gemm::RT; ++i) {
            const int rho = ty + i * Gemm::NRT;
            const int e = e0 + rho / TT, t = t0 + rho % TT;
            if (e < E && t < b) {
                float4 o;
                o.x = act_fn<ACT>(acc[i].x);
                o.y = act_fn<ACT>(acc[i].y);
                o.z = act_fn<ACT>(acc[i].z);
                o.w = act_fn<ACT>(acc[i].w);
                *reinterpret_cast<float4*>(Hout + (size_t)e * rowlen_out + (size_t)t * COUT + 4 * tx) = o;
            }
        }
    }
}

template <int CIN, int COUT>
struct BwdShape {
    static constexpr int TT = kTileCols / COUT, TE = kTileRows / TT;
    static constexpr int KD = 3 * COUT, LDA = KD + 4, LDH = CIN + 4;
    static constexpr int UNITS = COUT * CIN / 4;                          // (co, ci-quad) pairs
    static constexpr int UPT = UNITS >= kThreads ? UNITS / kThreads : 1;  // pairs per thread
    static constexpr int RS = UNITS >= kThreads ? 1 : kThreads / UNITS;   // row split
    static constexpr int DW = 3 * CIN * COUT;
};

// dw[u][k][q] += H[rho][4ciq+q] * A_k[rho][co] for one row; thread -> (co, ciq) mapping is data independent
#define SCONE_DW_ROW(Hs_, As_, rho_)                                                                                      \
    do {                                                                                                                  \
        const float4 h_ = *reinterpret_cast<const float4*>((Hs_) + (rho_) * LDH + 4 * ciq);                               \
        const float a0_ = (As_)[(rho_) * LDA + co], a1_ = (As_)[(rho_) * LDA + COUT + co],                                \
                    a2_ = (As_)[(rho_) * LDA + 2 * COUT + co];                                                            \
        dw[u][0][0] = fmaf(h_.x, a0_, dw[u][0][0]); dw[u][0][1] = fmaf(h_.y, a0_, dw[u][0][1]);                           \
        dw[u][0][2] = fmaf(h_.z, a0_, dw[u][0][2]); dw[u][0][3] = fmaf(h_.w, a0_, dw[u][0][3]);                           \
        dw[u][1][0] = fmaf(h_.x, a1_, dw[u][1][0]); dw[u][1][1] = fmaf(h_.y, a1_, dw[u][1][1]);                           \
        dw[u][1][2] = fmaf(h_.z, a1_, dw[u][1][2]); dw[u][1][3] = fmaf(h_.w, a1_, dw[u][1][3]);                           \
        dw[u][2][0] = fmaf(h_.x, a2_, dw[u][2][0]); dw[u][2][1] = fmaf(h_.y, a2_, dw[u][2][1]);                           \
        dw[u][2][2] = fmaf(h_.z, a2_, dw[u][2][2]); dw[u][2][3] = fmaf(h_.w, a2_, dw[u][2][3]);                           \
    } while (0)

// per-CTA partial dw_partial[cta][k][ci][co]; row splits are combined in split order through shared memory
template <int CIN, int COUT>
__device__ __forceinline__ void write_dw_partial(float (&dw)[BwdShape<CIN, COUT>::UPT][3][4], float* __restrict__ red,
                                                 float* __restrict__ dw_partial) {
    using Sh = BwdShape<CIN, COUT>;
    __syncthreads();
    float* outp = dw_partial + (size_t)blockIdx.x * Sh::DW;
#pragma unroll
    for (int u = 0; u < Sh::UPT; ++u) {
        const int unit = (Sh::UNITS >= kThreads) ? (int)threadIdx.x + u * kThreads : (int)threadIdx.x % Sh::UNITS;
        const int split = (Sh::UNITS >= kThreads) ? 0 : (int)threadIdx.x / Sh::UNITS;
        const int co = unit % COUT, ciq = unit / COUT;
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int o = (k * CIN + 4 * ciq + q) * COUT + co;
                if (Sh::RS == 1) outp[o] = dw[u][k][q];
                else red[split * Sh::DW + o] = dw[u][k][q];
            }
    }
    if (Sh::RS > 1) {
        __syncthreads();
        for (int o = threadIdx.x; o < Sh::DW; o += kThreads) {
            float s = 0.f;
            for (int sp = 0; sp < Sh::RS; ++sp) s += red[sp * Sh::DW + o];
            outp[o] = s;
        }
    }
}

template <int CIN, int COUT, int ACT, bool WRITE_GPREV>
__global__ void __launch_bounds__(kThreads) layer_bwd_dense_kernel(const float* __restrict__ G, const float* __restrict__ Hin,
                                                                  float* __restrict__ Gprev, const float* __restrict__ W0,
                                                                  const float* __restrict__ W1, const float* __restrict__ W2,
                                                                  float* __restrict__ dw_partial, DevCsr S0, DevCsr S1, int E, int b) {
    using Sh = BwdShape<CIN, COUT>;
    constexpr int TT = Sh::TT, TE = Sh::TE, KD = Sh::KD, LDA = Sh::LDA, LDH = Sh::LDH;
    using Gemm = TileGemm<KD, CIN, LDA>;
    extern __shared__ __align__(16) float smem[];
    float* As = smem;                          // [128][LDA]   rows = (edge, traj), cols = k*COUT + co
    float* Hs = As + kTileRows * LDA;          // [128][LDH]
    float* Wt = Hs + kTileRows * LDH;          // [KD][CIN]    Wt[k*COUT+co][ci] = W_k[ci][co]
    for (int i = threadIdx.x; i < CIN * COUT; i += kThreads) {
        const int ci = i / COUT, co = i % COUT;
        Wt[(co)*CIN + ci] = W0[i];
        Wt[(COUT + co) * CIN + ci] = W1[i];
        Wt[(2 * COUT + co) * CIN + ci] = W2[i];
    }
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const size_t rowlen_g = (size_t)b * COUT, rowlen_h = (size_t)b * CIN;
    const int n_tb = (b + TT - 1) / TT, n_eb = (E + TE - 1) / TE;
    const int jl = (4 * lane) / COUT, col = (4 * lane) % COUT;
    float dw[Sh::UPT][3][4];
#pragma unroll
    for (int u = 0; u < Sh::UPT; ++u)
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int q = 0; q < 4; ++q) dw[u][k][q] = 0.f;

    for (int tile = blockIdx.x; tile < n_tb * n_eb; tile += gridDim.x) {
        const int tb = tile % n_tb, eb = tile / n_tb;
        const int e0 = eb * TE, t0 = tb * TT;
        const int colofs = tb * kTileCols + 4 * lane;
        const bool colok = colofs < (int)rowlen_g;
        __syncthreads();
        for (int r = warp; r < TE; r += kWarps) {
            const int e = e0 + r;
            float4 a0 = zero4(), a1 = a0, a2 = a0;
            if (e < E && colok) {
                a0 = __ldg(reinterpret_cast<const float4*>(G + (size_t)e * rowlen_g + colofs));
                a1 = gather_row4_dense(G, rowlen_g, colofs, S0, e);
                a2 = gather_row4_dense(G, rowlen_g, colofs, S1, e);
            }
            float* dst = As + (r * TT + jl) * LDA + col;
            *reinterpret_cast<float4*>(dst) = a0;
            *reinterpret_cast<float4*>(dst + COUT) = a1;
            *reinterpret_cast<float4*>(dst + 2 * COUT) = a2;
        }
        for (int idx = threadIdx.x; idx < kTileRows * (CIN / 4); idx += kThreads) {
            const int rho = idx / (CIN / 4), c4 = idx % (CIN / 4);
            const int e = e0 + rho / TT, t = t0 + rho % TT;
            float4 h = zero4();
            if (e < E && t < b) h = __ldg(reinterpret_cast<const float4*>(Hin + (size_t)e * rowlen_h + (size_t)t * CIN + 4 * c4));
            *reinterpret_cast<float4*>(Hs + rho * LDH + 4 * c4) = h;
        }
        __syncthreads();
        if (WRITE_GPREV) {
            float4 acc[Gemm::RT];
            Gemm::run(As, Wt, acc);
            const int tx = threadIdx.x % Gemm::NTX, ty = threadIdx.x / Gemm::NTX;
#pragma unroll
            for (int i = 0; i < Gemm::RT; ++i) {
                const int rho = ty + i * Gemm::NRT;
                const int e = e0 + rho / TT, t = t0 + rho % TT;
                if (e < E && t < b) {
                    const float4 h = *reinterpret_cast<const float4*>(Hs + rho * LDH + 4 * tx);
                    float4 o;
                    o.x = acc[i].x * dact_fn<ACT>(h.x);
                    o.y = acc[i].y * dact_fn<ACT>(h.y);
                    o.z = acc[i].z * dact_fn<ACT>(h.z);
                    o.w = acc[i].w * dact_fn<ACT>(h.w);
                    *reinterpret_cast<float4*>(Gprev + (size_t)e * rowlen_h + (size_t)t * CIN + 4 * tx) = o;
                }
            }
        }
#pragma unroll
        for (int u = 0; u < Sh::UPT; ++u) {
            const int unit = (Sh::UNITS >= kThreads) ? (int)threadIdx.x + u * kThreads : (int)threadIdx.x % Sh::UNITS;
            const int split = (Sh::UNITS >= kThreads) ? 0 : (int)threadIdx.x / Sh::UNITS;
            const int co = unit % COUT, ciq = unit / COUT;
#pragma unroll 4
            for (int rho = split; rho < kTileRows; rho += Sh::RS) SCONE_DW_ROW(Hs, As, rho);
        }
    }
    write_dw_partial<CIN, COUT>(dw, smem, dw_partial);
}

// =================================================================================================================
// UNIT kernels (occupancy flags)
//
// occ[e][t] (one byte) == 0 promises that row (e, t) of a tensor is entirely zero (structural support, a superset of
// the non-zero rows).  A unit is (edge e, chunk of TT = 128 / C consecutive trajectories) = 128 contiguous columns.
// Per flagged launch:   worklist(in) = compaction of occ_in            (deterministic, ascending unit id)
//                       occ_out      = one-hop scatter from worklist(in)   (idempotent byte stores of 1: no atomics)
//                       worklist(out)= compaction of occ_out
//                       one warp per worklist(out) entry does gather + contraction + store.
// =================================================================================================================
constexpr int kCompactBlock = 1024;           // units per compaction CTA (4 per thread)

template <int TT>
__device__ __forceinline__ unsigned unit_row_mask(const uint8_t* __restrict__ flags, int e, int t0, int b) {
    unsigned m = 0;
    const uint8_t* f = flags + (size_t)e * b + t0;
    if (TT == 4 && (b & 3) == 0) {             // aligned fast path: one 32-bit load
        const uint32_t w = __ldg(reinterpret_cast<const uint32_t*>(f));
        m = ((w & 0xffu) ? 1u : 0u) | ((w & 0xff00u) ? 2u : 0u) | ((w & 0xff0000u) ? 4u : 0u) | ((w & 0xff000000u) ? 8u : 0u);
    } else {
#pragma unroll
        for (int k = 0; k < TT; ++k)
            if (t0 + k < b && __ldg(f + k) != 0) m |= 1u << k;
    }
    return m;
}

// pass 1 / pass 3 of the compaction: WRITE = false counts the flagged units of each 1024-unit block,
// WRITE = true writes their ids at the block's offset (ascending order).
template <int TT, bool WRITE>
__global__ void __launch_bounds__(kThreads) compact_units_kernel(const uint8_t* __restrict__ flags, long long n_units, int nchunk, int b,
                                                                int* __restrict__ block_counts, uint32_t* __restrict__ list) {
    __shared__ int wcount[4 * kWarps];
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const long long unit0 = (long long)blockIdx.x * kCompactBlock;
    unsigned bal[4];
    bool on[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long u = unit0 + k * kThreads + threadIdx.x;
        bool a = false;
        if (u < n_units) {
            const int e = (int)(u / nchunk);
            a = unit_row_mask<TT>(flags, e, (int)(u - (long long)e * nchunk) * TT, b) != 0u;
        }
        on[k] = a;
        bal[k] = __ballot_sync(0xffffffffu, a);
        if (lane == 0) wcount[k * kWarps + warp] = __popc(bal[k]);
    }
    __syncthreads();
    if (!WRITE) {
        if (threadIdx.x == 0) {
            int total = 0;
            for (int j = 0; j < 4 * kWarps; ++j) total += wcount[j];
            block_counts[blockIdx.x] = total;
        }
        return;
    }
    const int off = block_counts[blockIdx.x];          // exclusive prefix after the scan
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (on[k]) {
            int base = off;
            for (int j = 0; j < k * kWarps + warp; ++j) base += wcount[j];
            list[base + __popc(bal[k] & ((1u << lane) - 1u))] = (uint32_t)(unit0 + k * kThreads + threadIdx.x);
        }
    }
}

// in-place exclusive scan of block_counts[0..n) by one CTA; *total = sum
__global__ void __launch_bounds__(1024) scan_counts_kernel(int* __restrict__ counts, int n, int* __restrict__ total) {
    __shared__ int part[1024];
    const int per = (n + 1023) / 1024;
    const int lo = threadIdx.x * per, hi = min(n, lo + per);
    int s = 0;
    for (int i = lo; i < hi; ++i) s += counts[i];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0;
        for (int i = 0; i < 1024; ++i) { const int v = part[i]; part[i] = run; run += v; }
        *total = run;
    }
    __syncthreads();
    int run = part[threadIdx.x];
    for (int i = lo; i < hi; ++i) { const int v = counts[i]; counts[i] = run; run += v; }
}

// occ_out[e'][t] = 1 for every flagged row (e, t) of the input worklist and every e' in {e} + S0 row + S1 row.
// row bitmap: bit e*b + t mirrors the flag byte of row (e, t).  Setting bits is idempotent (atomicOr), so the bitmap — like
// the flags — does not depend on the order of the writers.  A unit's tt <= 16 rows start at a multiple of tt (b % tt == 0),
// so they sit in one 32-bit word.
__device__ __forceinline__ bool bitmap_test_row(const uint32_t* __restrict__ bm, size_t row) { return (bm[row >> 5] >> (row & 31)) & 1u; }
__device__ __forceinline__ void bitmap_set_rows(uint32_t* __restrict__ bm, size_t row0, unsigned m) {
    const uint32_t bits = m << (row0 & 31);
    uint32_t* w = bm + (row0 >> 5);
    if ((*w & bits) != bits) atomicOr(w, bits);
}

template <int TT>
__global__ void __launch_bounds__(kThreads) scatter_support_kernel(const uint32_t* __restrict__ wl, const int* __restrict__ n_ptr,
                                                                  const uint8_t* __restrict__ occ_in, uint8_t* __restrict__ occ_out,
                                                                  uint32_t* __restrict__ bm_out, DevCsr S0, DevCsr S1, int nchunk, int b) {
    const int n = *n_ptr, lane = threadIdx.x % 32;
    const long long nw = (long long)gridDim.x * kWarps;
    for (long long i = (long long)blockIdx.x * kWarps + threadIdx.x / 32; i < n; i += nw) {
        const uint32_t u = wl[i];
        const int e = (int)(u / (uint32_t)nchunk), t0 = (int)(u - (uint32_t)e * (uint32_t)nchunk) * TT;
        const unsigned m = unit_row_mask<TT>(occ_in, e, t0, b);
        if (lane < TT && ((m >> lane) & 1u)) occ_out[(size_t)e * b + t0 + lane] = 1;
        if (bm_out != nullptr && lane == 0) bitmap_set_rows(bm_out, (size_t)e * b + t0, m);
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const DevCsr S = s == 0 ? S0 : S1;
            const int p0 = __ldg(S.rowptr + e), p1 = __ldg(S.rowptr + e + 1);
            for (int p = p0 + lane; p < p1; p += 32) {
                const size_t row0 = (size_t)__ldg(S.ent + p).x * b + t0;
                uint8_t* dst = occ_out + row0;
#pragma unroll
                for (int k = 0; k < TT; ++k)
                    if ((m >> k) & 1u) dst[k] = 1;
                if (bm_out != nullptr) bitmap_set_rows(bm_out, row0, m);
            }
        }
    }
}

// Worklist of the flagged units (or rows, G = 1) from the row bitmap, ascending id, in ONE launch: CTA c owns a contiguous
// slice of bitmap words; it counts, publishes its total (ticket = ready bit | count), sums the tickets of the CTAs before it
// (decoupled look-back; lower block indices are dispatched first), then writes its ids.  A unit is G = TT adjacent rows
// (b % TT == 0, TT in {4, 8, 16}).  tickets[] must be zero at launch.
template <int G>
__device__ __forceinline__ uint32_t collapse_quads(uint32_t w) {
    if (G == 1) return w;
    w = (w | (w >> 1) | (w >> 2) | (w >> 3)) & 0x11111111u;
    if (G == 4) return w;
    w = (w | (w >> 4)) & 0x01010101u;
    if (G == 8) return w;
    return (w | (w >> 8)) & 0x00010001u;
}

template <int R>
__global__ void __launch_bounds__(kThreads) compact_bitmap_kernel(const uint32_t* __restrict__ bm, long long n_words,
                                                                 uint32_t* __restrict__ list, int* __restrict__ n_out,
                                                                 unsigned long long* __restrict__ tickets,
                                                                 uint32_t* __restrict__ pref_out, long long list_cap) {
    // pref_out (optional, R == 1): pref_out[w] = number of set bits before word w = list index of word w's first set bit; the
    // rank of row r is then pref_out[r >> 5] + popc(bm[r >> 5] & ((1 << (r & 31)) - 1)).  Only words with a set bit are written
    // (the rank of a row whose bit is clear is never used).
    constexpr int WPT = 16;                               // words per thread and chunk: four 128-bit loads in flight
    constexpr int kChunk = WPT * kThreads;
    __shared__ int s_warp[kWarps];
    __shared__ long long s_prefix;
    __shared__ int s_total;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long per_cta = ((n_words + gridDim.x - 1) / gridDim.x + kChunk - 1) / kChunk * kChunk;   // whole chunks
    const long long lo = (long long)blockIdx.x * per_cta, hi = lo + per_cta < n_words ? lo + per_cta : n_words;
    auto load16 = [&](long long w, uint32_t (&c)[WPT]) {  // words w .. w+15 (w % 16 == 0), zero beyond hi; the bitmap is padded
#pragma unroll
        for (int v4 = 0; v4 < WPT / 4; ++v4) {
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (w + 4 * v4 < hi) v = __ldg(reinterpret_cast<const uint4*>(bm + w + 4 * v4));
            c[4 * v4 + 0] = collapse_quads<R>(v.x);
            c[4 * v4 + 1] = w + 4 * v4 + 1 < hi ? collapse_quads<R>(v.y) : 0u;
            c[4 * v4 + 2] = w + 4 * v4 + 2 < hi ? collapse_quads<R>(v.z) : 0u;
            c[4 * v4 + 3] = w + 4 * v4 + 3 < hi ? collapse_quads<R>(v.w) : 0u;
        }
    };
    // pass 1: count
    int cnt = 0;
    for (long long w = lo + (long long)WPT * threadIdx.x; w < hi; w += kChunk) {
        uint32_t c[WPT];
        load16(w, c);
#pragma unroll
        for (int q = 0; q < WPT; ++q) cnt += __popc(c[q]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) s_warp[warp] = cnt;
    if (threadIdx.x == 0) s_prefix = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        int total = 0;
        for (int k = 0; k < kWarps; ++k) total += s_warp[k];
        s_total = total;
        atomicExch(tickets + blockIdx.x, (1ull << 63) | (unsigned long long)(unsigned)total);
    }
    long long part = 0;
    for (int c = threadIdx.x; c < (int)blockIdx.x; c += kThreads) {
        unsigned long long t;
        do { t = atomicAdd(tickets + c, 0ull); } while (!(t >> 63));
        part += (long long)(t & 0xffffffffull);
    }
    if (part) atomicAdd((unsigned long long*)&s_prefix, (unsigned long long)part);
    __syncthreads();
    long long base = s_prefix;
    const int total = s_total;
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
        n_out[0] = (int)(base + total);
        n_out[1] = 0;                                     // tile counter of the row-list kernel that consumes this list
    }
    if (total == 0) return;                               // (uniform) nothing flagged in this slice
    // pass 2: block-exclusive scan of the per-thread counts of a chunk, ids written in ascending order
    for (long long w0 = lo; w0 < hi; w0 += kChunk) {
        const long long w = w0 + (long long)WPT * threadIdx.x;
        uint32_t c[WPT];
        load16(w, c);
        int n = 0;
#pragma unroll
        for (int q = 0; q < WPT; ++q) n += __popc(c[q]);
        int incl = n;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        __syncthreads();                                  // s_warp of the previous chunk fully consumed
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        int woff = 0, ctot = 0;
#pragma unroll
        for (int k = 0; k < kWarps; ++k) {
            const int v = s_warp[k];
            if (k < warp) woff += v;
            ctot += v;
        }
        long long off = base + woff + incl - n;
        if (n) {
#pragma unroll
            for (int q = 0; q < WPT; ++q) {
                uint32_t cc = c[q];
                if (cc == 0u) continue;
                if (pref_out != nullptr) pref_out[w + q] = (uint32_t)off;
                while (cc) {
                    const int pbit = __ffs(cc) - 1;
                    cc &= cc - 1;
                    if (off < list_cap) list[off] = (uint32_t)(((w + q) * 32 + pbit) / R);     // (*n_out still reports the full count)
                    ++off;
                }
            }
        }
        base += ctot;
    }
}

// (own row, S0 row, S1 row) of unit (e, t0..t0+TT) into Ts rows [slot0 + j]; returns the ballot of non-zero lanes.
template <int C, int LD>
__device__ __forceinline__ unsigned gather_unit(const float* __restrict__ H, size_t rowlen, DevCsr S0, DevCsr S1, int b, int e,
                                                int chunk, const uint8_t* __restrict__ occ, float* __restrict__ Ts, int slot0) {
    constexpr int TT = kTileCols / C;
    const int lane = threadIdx.x & 31;
    const int jl = (4 * lane) / C, cl = (4 * lane) % C, t0 = chunk * TT;
    const int colofs = chunk * kTileCols + 4 * lane;
    const bool colok = colofs < (int)rowlen;
    float4 a0 = zero4();
    if (colok && __ldg(occ + (size_t)e * b + t0 + jl) != 0) a0 = __ldg(reinterpret_cast<const float4*>(H + (size_t)e * rowlen + colofs));
    const float4 a1 = gather_row4_flagged<TT>(H, rowlen, colofs, colok, S0, e, occ, b, t0, jl);
    const float4 a2 = gather_row4_flagged<TT>(H, rowlen, colofs, colok, S1, e, occ, b, t0, jl);
    float* dst = Ts + (slot0 + jl) * LD + cl;
    *reinterpret_cast<float4*>(dst) = a0;
    *reinterpret_cast<float4*>(dst + C) = a1;
    *reinterpret_cast<float4*>(dst + 2 * C) = a2;
    return __ballot_sync(0xffffffffu, nz4(a0) || nz4(a1) || nz4(a2));
}

// Forward: one warp per worklist unit.  Every flagged row of the unit is written (zeros when the gathered rows are
// numerically zero), so that the output's flags (occ_out == the candidates) never point at unwritten memory.
template <int CIN, int COUT, int ACT>
__global__ void __launch_bounds__(kThreads, 3) layer_fwd_units_kernel(const float* __restrict__ Hin, float* __restrict__ Hout,
                                                                  const float* __restrict__ W0, const float* __restrict__ W1,
                                                                  const float* __restrict__ W2, DevCsr S0, DevCsr S1, int E, int b,
                                                                  const uint8_t* __restrict__ occ_in, const uint8_t* __restrict__ occ_out,
                                                                  const uint32_t* __restrict__ wl, const int* __restrict__ n_ptr,
                                                                  unsigned long long* __restrict__ row_counter) {
    constexpr int TT = kTileCols / CIN, KD = 3 * CIN, LDT = KD + 4, NTX = COUT / 4, NG = CIN / 4, ITEMS = TT * NTX;
    unsigned rows_done = 0;
    extern __shared__ __align__(16) float smem[];
    float* Ws = smem;                              // [KD][COUT]
    float* Tw = smem + KD * COUT;                  // [kWarps][TT][LDT]
    for (int i = threadIdx.x; i < CIN * COUT; i += kThreads) {
        Ws[i] = W0[i];
        Ws[CIN * COUT + i] = W1[i];
        Ws[2 * CIN * COUT + i] = W2[i];
    }
    __syncthreads();
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const size_t rowlen_in = (size_t)b * CIN, rowlen_out = (size_t)b * COUT;
    const int nchunk = (b + TT - 1) / TT;
    const int n = *n_ptr;
    const long long nw = (long long)gridDim.x * kWarps;
    float* T = Tw + warp * TT * LDT;
    for (long long i = (long long)blockIdx.x * kWarps + warp; i < n; i += nw) {
        const uint32_t u = wl[i];
        const int e = (int)(u / (uint32_t)nchunk), chunk = (int)(u - (uint32_t)e * (uint32_t)nchunk), t0 = chunk * TT;
        const unsigned cm = unit_row_mask<TT>(occ_out, e, t0, b);          // candidate rows of this unit
        rows_done += __popc(cm);
        const unsigned bal = gather_unit<CIN, LDT>(Hin, rowlen_in, S0, S1, b, e, chunk, occ_in, T, 0);
        __syncwarp();
#pragma unroll
        for (int p = 0; p < (ITEMS + 31) / 32; ++p) {
            const int it = p * 32 + lane;
            const int j = it / NTX, tx = it % NTX;
            if (it < ITEMS && ((cm >> j) & 1u)) {
                float4 o = zero4();
                if (((bal >> (j * NG)) & ((NG >= 32) ? 0xffffffffu : ((1u << NG) - 1u))) != 0u) {
                    o = row_gemm<KD, COUT, LDT>(T, Ws, j, tx);
                    o.x = act_fn<ACT>(o.x);
                    o.y = act_fn<ACT>(o.y);
                    o.z = act_fn<ACT>(o.z);
                    o.w = act_fn<ACT>(o.w);
                }
                *reinterpret_cast<float4*>(Hout + (size_t)e * rowlen_out + (size_t)(t0 + j) * COUT + 4 * tx) = o;
            }
        }
        __syncwarp();                              // T is reused by this warp's next unit
    }
    if (row_counter != nullptr && lane == 0 && rows_done) atomicAdd(row_counter, (unsigned long long)rows_done);
}

template <int CIN, int COUT>
struct BwdUnitShape {
    static constexpr int TT = kTileCols / COUT;
    static constexpr int UC = 16;                        // units staged per dW round
    static constexpr int RC = UC * TT;                   // staged rows
    static constexpr int KD = 3 * COUT, LDA = KD + 4, LDH = CIN + 4;
    static constexpr size_t smem_floats_layout = (size_t)KD * CIN + (size_t)RC * LDA + (size_t)RC * LDH;
    static constexpr size_t red_floats = (size_t)BwdShape<CIN, COUT>::RS * BwdShape<CIN, COUT>::DW;
    static constexpr size_t smem_floats = smem_floats_layout > red_floats ? smem_floats_layout : red_floats;
};

// Backward: CTA c owns the contiguous worklist slice [c*per, (c+1)*per); rounds of UC units are staged by the warps
// (A rows = G / S0 G / S1 G, Hin rows) and then all threads accumulate the weight gradients over the staged rows.
template <int CIN, int COUT, int ACT, bool WRITE_GPREV>
__global__ void __launch_bounds__(kThreads, 3) layer_bwd_units_kernel(const float* __restrict__ G, const float* __restrict__ Hin,
                                                                  float* __restrict__ Gprev, const float* __restrict__ W0,
                                                                  const float* __restrict__ W1, const float* __restrict__ W2,
                                                                  float* __restrict__ dw_partial, DevCsr S0, DevCsr S1, int E, int b,
                                                                  const uint8_t* __restrict__ occ_g, const uint8_t* __restrict__ occ_h,
                                                                  const uint8_t* __restrict__ occ_prev, const uint32_t* __restrict__ wl,
                                                                  const int* __restrict__ n_ptr, unsigned long long* __restrict__ row_counter) {
    using Sh = BwdShape<CIN, COUT>;
    using Us = BwdUnitShape<CIN, COUT>;
    unsigned rows_done = 0;
    constexpr int TT = Us::TT, UC = Us::UC, RC = Us::RC, KD = Us::KD, LDA = Us::LDA, LDH = Us::LDH;
    constexpr int NTX = CIN / 4, NG = COUT / 4, ITEMS = TT * NTX;
    extern __shared__ __align__(16) float smem[];
    float* Wt = smem;                              // [KD][CIN]    Wt[k*COUT+co][ci] = W_k[ci][co]
    float* Ar = Wt + KD * CIN;                     // [RC][LDA]
    float* Hr = Ar + RC * LDA;                     // [RC][LDH]
    __shared__ uint8_t rowact[RC];
    for (int i = threadIdx.x; i < CIN * COUT; i += kThreads) {
        const int ci = i / COUT, co = i % COUT;
        Wt[(co)*CIN + ci] = W0[i];
        Wt[(COUT + co) * CIN + ci] = W1[i];
        Wt[(2 * COUT + co) * CIN + ci] = W2[i];
    }
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const size_t rowlen_g = (size_t)b * COUT, rowlen_h = (size_t)b * CIN;
    const int nchunk = (b + TT - 1) / TT;
    float dw[Sh::UPT][3][4];
#pragma unroll
    for (int u = 0; u < Sh::UPT; ++u)
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int q = 0; q < 4; ++q) dw[u][k][q] = 0.f;
    const int n = *n_ptr;
    const int per = (n + (int)gridDim.x - 1) / (int)gridDim.x;
    const int lo = min(n, (int)blockIdx.x * per), hi = min(n, lo + per);
    __syncthreads();
    for (int c0 = lo; c0 < hi; c0 += UC) {
        const int nu = min(UC, hi - c0);
        for (int i = warp; i < nu; i += kWarps) {
            const uint32_t u = wl[c0 + i];
            const int e = (int)(u / (uint32_t)nchunk), chunk = (int)(u - (uint32_t)e * (uint32_t)nchunk), t0 = chunk * TT;
            const int slot0 = i * TT;
            const unsigned cm = WRITE_GPREV ? unit_row_mask<TT>(occ_prev, e, t0, b) : 0u;
            const unsigned bal = gather_unit<COUT, LDA>(G, rowlen_g, S0, S1, b, e, chunk, occ_g, Ar, slot0);
            rows_done += __popc(unit_row_mask<TT>(WRITE_GPREV ? occ_prev : occ_g, e, t0, b));
#pragma unroll
            for (int p = 0; p < (ITEMS + 31) / 32; ++p) {
                const int it = p * 32 + lane;
                const int j = it / NTX, hx = it % NTX;
                if (it < ITEMS) {
                    const bool ra = t0 + j < b && ((bal >> (j * NG)) & ((NG >= 32) ? 0xffffffffu : ((1u << NG) - 1u))) != 0u;
                    float4 h = zero4();
                    if (ra && (occ_h == nullptr || __ldg(occ_h + (size_t)e * b + t0 + j) != 0))
                        h = __ldg(reinterpret_cast<const float4*>(Hin + (size_t)e * rowlen_h + (size_t)(t0 + j) * CIN + 4 * hx));
                    *reinterpret_cast<float4*>(Hr + (slot0 + j) * LDH + 4 * hx) = h;
                    if (hx == 0) rowact[slot0 + j] = ra ? 1 : 0;
                }
            }
            __syncwarp();
            if (WRITE_GPREV) {
#pragma unroll
                for (int p = 0; p < (ITEMS + 31) / 32; ++p) {
                    const int it = p * 32 + lane;
                    const int j = it / NTX, tx = it % NTX;
                    if (it < ITEMS && ((cm >> j) & 1u)) {
                        float4 o = zero4();
                        if (rowact[slot0 + j]) {
                            o = row_gemm<KD, CIN, LDA>(Ar, Wt, slot0 + j, tx);
                            const float4 h = *reinterpret_cast<const float4*>(Hr + (slot0 + j) * LDH + 4 * tx);
                            o.x *= dact_fn<ACT>(h.x);
                            o.y *= dact_fn<ACT>(h.y);
                            o.z *= dact_fn<ACT>(h.z);
                            o.w *= dact_fn<ACT>(h.w);
                        }
                        *reinterpret_cast<float4*>(Gprev + (size_t)e * rowlen_h + (size_t)(t0 + j) * CIN + 4 * tx) = o;
                    }
                }
            }
        }
        __syncthreads();
        const int n_rows = nu * TT;
#pragma unroll
        for (int u = 0; u < Sh::UPT; ++u) {
            const int unit = (Sh::UNITS >= kThreads) ? (int)threadIdx.x + u * kThreads : (int)threadIdx.x % Sh::UNITS;
            const int split = (Sh::UNITS >= kThreads) ? 0 : (int)threadIdx.x / Sh::UNITS;
            const int co = unit % COUT, ciq = unit / COUT;
            for (int rho = split; rho < n_rows; rho += Sh::RS)
                if (rowact[rho]) SCONE_DW_ROW(Hr, Ar, rho);
        }
        __syncthreads();
    }
    if (row_counter != nullptr && lane == 0 && rows_done) atomicAdd(row_counter, (unsigned long long)rows_done);
    write_dw_partial<CIN, COUT>(dw, smem, dw_partial);
}

// First layer on units: lanes (row j, channel quad c4); the scalar gathers of X are repeated by the COUT/4 lanes of a row
// (broadcast loads).  Forward writes every candidate row; backward accumulates dW_k[0][co] over flagged rows of G0.
template <int COUT>
__device__ __forceinline__ void layer0_unit_rows(const float* __restrict__ X, DevCsr S0, DevCsr S1, int b, int e, int t, bool ok,
                                                 float& a0, float& a1, float& a2) {
    a0 = a1 = a2 = 0.f;
    if (ok) {
        a0 = __ldg(X + (size_t)e * b + t);
        a1 = gather_row1(X, b, t, S0, e);
        a2 = gather_row1(X, b, t, S1, e);
    }
}

template <int COUT, int ACT>
__global__ void __launch_bounds__(kThreads) layer0_fwd_units_kernel(const float* __restrict__ X, float* __restrict__ Hout,
                                                                   const float* __restrict__ W0, const float* __restrict__ W1,
                                                                   const float* __restrict__ W2, DevCsr S0, DevCsr S1, int E, int b,
                                                                   const uint8_t* __restrict__ occ_out, const uint32_t* __restrict__ wl,
                                                                   const int* __restrict__ n_ptr) {
    constexpr int TT = kTileCols / COUT, C4 = COUT / 4;
    __shared__ __align__(16) float ws[3 * COUT];
    for (int i = threadIdx.x; i < COUT; i += kThreads) {
        ws[i] = W0[i];
        ws[COUT + i] = W1[i];
        ws[2 * COUT + i] = W2[i];
    }
    __syncthreads();
    const int lane = threadIdx.x % 32, j = lane / C4, c4 = lane % C4;
    const int nchunk = (b + TT - 1) / TT, n = *n_ptr;
    const long long nw = (long long)gridDim.x * kWarps;
    const float4 w0 = *reinterpret_cast<const float4*>(ws + 4 * c4);
    const float4 w1 = *reinterpret_cast<const float4*>(ws + COUT + 4 * c4);
    const float4 w2 = *reinterpret_cast<const float4*>(ws + 2 * COUT + 4 * c4);
    for (long long i = (long long)blockIdx.x * kWarps + threadIdx.x / 32; i < n; i += nw) {
        const uint32_t u = wl[i];
        const int e = (int)(u / (uint32_t)nchunk), t = (int)(u - (uint32_t)e * (uint32_t)nchunk) * TT + j;
        const bool ok = t < b && __ldg(occ_out + (size_t)e * b + t) != 0;
        float a0, a1, a2;
        layer0_unit_rows<COUT>(X, S0, S1, b, e, t, ok, a0, a1, a2);
        if (ok) {
            float4 o = zero4();
            if (a0 != 0.f || a1 != 0.f || a2 != 0.f) {
                o.x = act_fn<ACT>(fmaf(a2, w2.x, fmaf(a1, w1.x, a0 * w0.x)));
                o.y = act_fn<ACT>(fmaf(a2, w2.y, fmaf(a1, w1.y, a0 * w0.y)));
                o.z = act_fn<ACT>(fmaf(a2, w2.z, fmaf(a1, w1.z, a0 * w0.z)));
                o.w = act_fn<ACT>(fmaf(a2, w2.w, fmaf(a1, w1.w, a0 * w0.w)));
            }
            *reinterpret_cast<float4*>(Hout + ((size_t)e * b + t) * COUT + 4 * c4) = o;
        }
    }
}

template <int COUT>
__global__ void __launch_bounds__(kThreads) layer0_bwd_units_kernel(const float* __restrict__ X, const float* __restrict__ G0,
                                                                   float* __restrict__ dw_partial, DevCsr S0, DevCsr S1, int E, int b,
                                                                   const uint8_t* __restrict__ occ_g, const uint32_t* __restrict__ wl,
                                                                   const int* __restrict__ n_ptr) {
    constexpr int TT = kTileCols / COUT, C4 = COUT / 4;
    __shared__ float red[kThreads * 12];
    const int lane = threadIdx.x % 32, j = lane / C4, c4 = lane % C4;
    const int nchunk = (b + TT - 1) / TT, n = *n_ptr;
    const long long nw = (long long)gridDim.x * kWarps;
    float acc[3][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    for (long long i = (long long)blockIdx.x * kWarps + threadIdx.x / 32; i < n; i += nw) {
        const uint32_t u = wl[i];
        const int e = (int)(u / (uint32_t)nchunk), t = (int)(u - (uint32_t)e * (uint32_t)nchunk) * TT + j;
        const bool ok = t < b && __ldg(occ_g + (size_t)e * b + t) != 0;
        float a[3];
        layer0_unit_rows<COUT>(X, S0, S1, b, e, t, ok, a[0], a[1], a[2]);
        if (ok) {
            const float4 g = __ldg(reinterpret_cast<const float4*>(G0 + ((size_t)e * b + t) * COUT + 4 * c4));
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                acc[k][0] = fmaf(a[k], g.x, acc[k][0]);
                acc[k][1] = fmaf(a[k], g.y, acc[k][1]);
                acc[k][2] = fmaf(a[k], g.z, acc[k][2]);
                acc[k][3] = fmaf(a[k], g.w, acc[k][3]);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int q = 0; q < 4; ++q) red[threadIdx.x * 12 + k * 4 + q] = acc[k][q];
    __syncthreads();
    // thread o < 3*COUT sums its (k, co) over the threads that own channel quad co/4 (lane % C4 == co/4), ascending
    for (int o = threadIdx.x; o < 3 * COUT; o += kThreads) {
        const int k = o / COUT, co = o % COUT, q4 = co / 4, q = co % 4;
        float s = 0.f;
        for (int th = q4; th < kThreads; th += C4) s += red[th * 12 + k * 4 + q];
        dw_partial[(size_t)blockIdx.x * 3 * COUT + o] = s;
    }
}

// Dense zero-fill of an output tensor (128-bit streaming stores, grid-stride).  In the default (zero-fill ON) mode this is
// where the HBM time of a step goes: every dense [E][b][C] tensor is written once per micro-batch.
// One short-lived CTA per 32 KB chunk: SM slots turn over every few microseconds, so the (higher-priority) flag / unit
// kernels of the main stream are scheduled in between instead of queueing behind a persistent fill.
__global__ void __launch_bounds__(kThreads) zero_fill_kernel(float4* __restrict__ p, size_t n16) {
    const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
    const size_t base = (size_t)blockIdx.x * ((size_t)kThreads * 8);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const size_t i = base + (size_t)k * kThreads + threadIdx.x;
        if (i < n16) __stcs(p + i, z);
    }
}

// out[i] (+)= sum over parts p (ascending) of partial[p][i]
// 256 threads = 32 outputs x 8 slices of the parts; slice sums (ascending p inside a slice) are combined in slice order:
// a fixed summation tree, independent of the launch shape of the producer only through nparts.
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ partial, int nparts, int n,
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

// =================================================================================================================
// First layer (C_in = 1): input X[E][b].
// =================================================================================================================
constexpr int kL0Edges = 32;     // edges per tile; 32 trajectories per tile (lane = trajectory)

__device__ __forceinline__ void layer0_gather(const float* __restrict__ X, DevCsr S0, DevCsr S1, int E, int b, int e0, int t0,
                                              float* ts /* [3][kL0Edges][32] */) {
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int t = t0 + lane;
    for (int r = warp; r < kL0Edges; r += kWarps) {
        const int e = e0 + r;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        if (e < E && t < b) {
            a0 = __ldg(X + (size_t)e * b + t);
            a1 = gather_row1(X, b, t, S0, e);
            a2 = gather_row1(X, b, t, S1, e);
        }
        ts[(0 * kL0Edges + r) * 32 + lane] = a0;
        ts[(1 * kL0Edges + r) * 32 + lane] = a1;
        ts[(2 * kL0Edges + r) * 32 + lane] = a2;
    }
}

// write_zero_rows: false when the caller pre-zeroed Hout (or runs in sparse mode): only live rows are stored.
template <int COUT, int ACT>
__global__ void __launch_bounds__(kThreads) layer0_fwd_kernel(const float* __restrict__ X, float* __restrict__ Hout,
                                                             const float* __restrict__ W0, const float* __restrict__ W1,
                                                             const float* __restrict__ W2, DevCsr S0, DevCsr S1, int E, int b,
                                                             uint8_t* __restrict__ occ_out, int write_zero_rows) {
    __shared__ float ts[3 * kL0Edges * 32];
    __shared__ __align__(16) float ws[3 * COUT];
    for (int i = threadIdx.x; i < COUT; i += kThreads) {
        ws[i] = W0[i];
        ws[COUT + i] = W1[i];
        ws[2 * COUT + i] = W2[i];
    }
    constexpr int C4 = COUT / 4;
    const int n_tb = (b + 31) / 32, n_eb = (E + kL0Edges - 1) / kL0Edges;
    for (int tile = blockIdx.x; tile < n_tb * n_eb; tile += gridDim.x) {
        const int tb = tile % n_tb, eb = tile / n_tb;
        const int e0 = eb * kL0Edges, t0 = tb * 32;
        __syncthreads();
        layer0_gather(X, S0, S1, E, b, e0, t0, ts);
        __syncthreads();
        for (int idx = threadIdx.x; idx < kL0Edges * 32 * C4; idx += kThreads) {
            const int c4 = idx % C4, j = (idx / C4) % 32, r = idx / (C4 * 32);
            const int e = e0 + r, t = t0 + j;
            if (e < E && t < b) {
                const float a0 = ts[(0 * kL0Edges + r) * 32 + j], a1 = ts[(1 * kL0Edges + r) * 32 + j],
                            a2 = ts[(2 * kL0Edges + r) * 32 + j];
                const bool live = a0 != 0.f || a1 != 0.f || a2 != 0.f;      // act(0) == 0: zero rows need no math
                if (live) {
                    const float4 w0 = *reinterpret_cast<const float4*>(ws + 4 * c4);
                    const float4 w1 = *reinterpret_cast<const float4*>(ws + COUT + 4 * c4);
                    const float4 w2 = *reinterpret_cast<const float4*>(ws + 2 * COUT + 4 * c4);
                    float4 o;
                    o.x = act_fn<ACT>(fmaf(a2, w2.x, fmaf(a1, w1.x, a0 * w0.x)));
                    o.y = act_fn<ACT>(fmaf(a2, w2.y, fmaf(a1, w1.y, a0 * w0.y)));
                    o.z = act_fn<ACT>(fmaf(a2, w2.z, fmaf(a1, w1.z, a0 * w0.z)));
                    o.w = act_fn<ACT>(fmaf(a2, w2.w, fmaf(a1, w1.w, a0 * w0.w)));
                    *reinterpret_cast<float4*>(Hout + ((size_t)e * b + t) * COUT + 4 * c4) = o;
                } else if (write_zero_rows) {
                    *reinterpret_cast<float4*>(Hout + ((size_t)e * b + t) * COUT + 4 * c4) = zero4();
                }
                if (occ_out != nullptr && c4 == 0 && (live || write_zero_rows)) occ_out[(size_t)e * b + t] = live ? 1 : 0;
            }
        }
    }
}

// dense: dW_k[0][co] = sum_{e,t} (S_k X)[e][t] * G0[e][t][co]
template <int COUT>
__global__ void __launch_bounds__(kThreads) layer0_bwd_dense_kernel(const float* __restrict__ X, const float* __restrict__ G0,
                                                                   float* __restrict__ dw_partial, DevCsr S0, DevCsr S1, int E, int b) {
    __shared__ float ts[3 * kL0Edges * 32];
    __shared__ float red[kThreads * 12];
    constexpr int C4 = COUT / 4;
    static_assert(kThreads % C4 == 0, "thread->channel-quad mapping must be tile independent");
    float acc[3][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    const int n_tb = (b + 31) / 32, n_eb = (E + kL0Edges - 1) / kL0Edges;
    for (int tile = blockIdx.x; tile < n_tb * n_eb; tile += gridDim.x) {
        const int tb = tile % n_tb, eb = tile / n_tb;
        const int e0 = eb * kL0Edges, t0 = tb * 32;
        __syncthreads();
        layer0_gather(X, S0, S1, E, b, e0, t0, ts);
        __syncthreads();
        for (int idx = threadIdx.x; idx < kL0Edges * 32 * C4; idx += kThreads) {
            const int c4 = idx % C4, j = (idx / C4) % 32, r = idx / (C4 * 32);
            const int e = e0 + r, t = t0 + j;
            if (e < E && t < b) {
                const float4 g = __ldg(reinterpret_cast<const float4*>(G0 + ((size_t)e * b + t) * COUT + 4 * c4));
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float a = ts[(k * kL0Edges + r) * 32 + j];
                    acc[k][0] = fmaf(a, g.x, acc[k][0]);
                    acc[k][1] = fmaf(a, g.y, acc[k][1]);
                    acc[k][2] = fmaf(a, g.z, acc[k][2]);
                    acc[k][3] = fmaf(a, g.w, acc[k][3]);
                }
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int q = 0; q < 4; ++q) red[threadIdx.x * 12 + k * 4 + q] = acc[k][q];
    __syncthreads();
    for (int o = threadIdx.x; o < 3 * COUT; o += kThreads) {
        const int k = o / COUT, co = o % COUT, c4 = co / 4, q = co % 4;
        float s = 0.f;
        for (int th = c4; th < kThreads; th += C4) s += red[th * 12 + k * 4 + q];
        dw_partial[(size_t)blockIdx.x * 3 * COUT + o] = s;
    }
}

// X[E][b] from sparse flows; one warp per trajectory (X pre-zeroed).
__global__ void flows_to_dense_kernel(const int32_t* __restrict__ traj_ptr, const int32_t* __restrict__ flow_edge,
                                      const float* __restrict__ flow_val, const int32_t* __restrict__ rank,
                                      float* __restrict__ X, uint8_t* __restrict__ occX, uint32_t* __restrict__ bm, int E, int b) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) / 32, lane = threadIdx.x % 32;
    if (t >= b) return;
    for (int p = traj_ptr[t] + lane; p < traj_ptr[t + 1]; p += 32) {
        const int e = flow_edge[p];
        if (e >= 0 && e < E) {
            const size_t row = (size_t)rank[e] * b + t;
            X[row] = flow_val[p];
            if (occX != nullptr) occX[row] = 1;
            if (bm != nullptr) atomicOr(bm + (row >> 5), 1u << (row & 31));
        }
    }
}

// =================================================================================================================
// Readout: one CTA per trajectory.
// =================================================================================================================
constexpr int kReadoutMaxD = SCONE_MAX_DEGREE, kReadoutMaxCper = 4;   // D <= 128, C <= 128

// One CTA (4 warps) per trajectory; warp w owns the neighbour slots j = w, w + 4, ...  A row of GL receives at most two
// contributions (an edge has two end nodes), added with atomicAdd onto a zeroed row: a + b == b + a, so the result does not
// depend on the order (deterministic without serialising the warps).
constexpr int kReadoutWarps = 4;
__global__ void __launch_bounds__(32 * kReadoutWarps) readout_kernel(const float* __restrict__ HL, const float* __restrict__ wout,
                                                     const int32_t* __restrict__ last_nodes, const int32_t* __restrict__ nbrhoods,
                                                     const int32_t* __restrict__ inc_ptr, const int2* __restrict__ inc_ent,
                                                     float* __restrict__ logprobs, const int32_t* __restrict__ target_idx,
                                                     const float* __restrict__ mask, float scale, float* __restrict__ GL,
                                                     float* __restrict__ partial /* [b][C+2] */, const uint8_t* __restrict__ occ_HL,
                                                     uint8_t* __restrict__ occ_GL, uint32_t* __restrict__ bm_GL, int act, int N, int D,
                                                     int b, int C, const uint32_t* __restrict__ bm_HL, uint32_t* __restrict__ bm_cand,
                                                     const int32_t* __restrict__ mptr, const int2* __restrict__ ment) {
    // bm_HL != NULL: the row bitmap of H_L replaces the flag bytes; bm_cand != NULL: every row of G_L this trajectory touches
    // also marks the candidate rows one hop further (its merged operator row) for the first backward layer
    __shared__ float logit[kReadoutMaxD];
    __shared__ float s_dw[kReadoutWarps][32 * kReadoutMaxCper];
    __shared__ float s_lse;
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int t = blockIdx.x;
    const int last = last_nodes[t];
    const bool last_ok = last >= 0 && last < N;
    float w[kReadoutMaxCper];
#pragma unroll
    for (int q = 0; q < kReadoutMaxCper; ++q) w[q] = (lane + 32 * q < C) ? wout[lane + 32 * q] : 0.f;

    for (int j = warp; j < D; j += kReadoutWarps) {
        const int nbr = last_ok ? nbrhoods[(size_t)last * D + j] : -1;
        float l = 0.f;                                     // padded slot: row -1 of B1_jax = zeros -> logit 0
        if (nbr >= 0) {
            float part = 0.f;
            float z[kReadoutMaxCper] = {0.f, 0.f, 0.f, 0.f};
            for (int p = inc_ptr[nbr]; p < inc_ptr[nbr + 1]; ++p) {
                const int2 es = inc_ent[p];
                if (bm_HL != nullptr ? !bitmap_test_row(bm_HL, (size_t)es.x * b + t)
                                     : (occ_HL != nullptr && occ_HL[(size_t)es.x * b + t] == 0)) continue;      // row is exactly zero
                const float* row = HL + ((size_t)es.x * b + t) * C;
#pragma unroll
                for (int q = 0; q < kReadoutMaxCper; ++q)
                    if (lane + 32 * q < C) z[q] = fmaf(__int_as_float(es.y), row[lane + 32 * q], z[q]);
            }
#pragma unroll
            for (int q = 0; q < kReadoutMaxCper; ++q) part = fmaf(z[q], w[q], part);
            l = warp_sum(part);
        }
        if (lane == 0) logit[j] = l;
    }
    __syncthreads();
    if (warp == 0) {
        float mx = -CUDART_INF_F;
        for (int j = lane; j < D; j += 32) mx = fmaxf(mx, logit[j]);
        mx = warp_max(mx);
        float se = 0.f;
        for (int j = lane; j < D; j += 32) se += expf(logit[j] - mx);
        se = warp_sum(se);
        const float lse_ = mx + logf(se);
        for (int j = lane; j < D; j += 32) logprobs[(size_t)t * D + j] = logit[j] - lse_;
        if (lane == 0) s_lse = lse_;
    }
    if (GL == nullptr) return;
    // gradient: the rows of GL this trajectory touches are zeroed and flagged first ...
    for (int j = warp; j < D; j += kReadoutWarps) {
        const int nbr = last_ok ? nbrhoods[(size_t)last * D + j] : -1;
        if (nbr < 0) continue;
        for (int p = inc_ptr[nbr]; p < inc_ptr[nbr + 1]; ++p) {
            const size_t row = (size_t)inc_ent[p].x * b + t;
#pragma unroll
            for (int q = 0; q < kReadoutMaxCper; ++q)
                if (lane + 32 * q < C) GL[row * C + lane + 32 * q] = 0.f;
            if (occ_GL != nullptr && lane == 0) occ_GL[row] = 1;
            if (bm_GL != nullptr && lane == 0) atomicOr(bm_GL + (row >> 5), 1u << (row & 31));
            if (bm_cand != nullptr) {
                const int e = inc_ent[p].x;
                for (int q = mptr[e] + lane; q < mptr[e + 1]; q += 32) {
                    const size_t crow = (size_t)(unsigned)ment[q].x * b + t;
                    atomicOr(bm_cand + (crow >> 5), 1u << (crow & 31));
                }
            }
        }
    }
    __syncthreads();                                       // ... (also publishes s_lse) then accumulated
    const float lse = s_lse;
    const float mk = mask[t];
    const int y = target_idx[t];
    float dwl[kReadoutMaxCper] = {0.f, 0.f, 0.f, 0.f};
    for (int j = warp; j < D; j += kReadoutWarps) {
        const int nbr = last_ok ? nbrhoods[(size_t)last * D + j] : -1;
        if (nbr < 0) continue;
        const float dl = mk * scale * (expf(logit[j] - lse) - (j == y ? 1.f : 0.f));
        for (int p = inc_ptr[nbr]; p < inc_ptr[nbr + 1]; ++p) {
            const int2 es = inc_ent[p];
            const size_t base = ((size_t)es.x * b + t) * C;
            const float sdl = __int_as_float(es.y) * dl;
            const bool hz = bm_HL != nullptr ? !bitmap_test_row(bm_HL, (size_t)es.x * b + t)
                                             : (occ_HL != nullptr && occ_HL[(size_t)es.x * b + t] == 0);
#pragma unroll
            for (int q = 0; q < kReadoutMaxCper; ++q)
                if (lane + 32 * q < C) {
                    const float h = hz ? 0.f : HL[base + lane + 32 * q];
                    dwl[q] = fmaf(sdl, h, dwl[q]);                                // z[j][c] * dlogit[j]
                    atomicAdd(GL + base + lane + 32 * q, sdl * w[q] * dact_rt(act, h));
                }
        }
    }
#pragma unroll
    for (int q = 0; q < kReadoutMaxCper; ++q) s_dw[warp][lane + 32 * q] = dwl[q];
    __syncthreads();
    if (warp == 0) {
        float* pt = partial + (size_t)t * (C + 2);
#pragma unroll
        for (int q = 0; q < kReadoutMaxCper; ++q)
            if (lane + 32 * q < C) {
                float sacc = s_dw[0][lane + 32 * q];
                for (int k = 1; k < kReadoutWarps; ++k) sacc += s_dw[k][lane + 32 * q];
                pt[lane + 32 * q] = sacc;
            }
        if (lane == 0) {
            pt[C] = (y >= 0 && y < D) ? -mk * (logit[y] - lse) : 0.f;
            pt[C + 1] = mk;
        }
    }
}

// dwout[c] (+)= sum_t partial[t][c]; nll (+)= sum_t partial[t][C]; count (+)= sum_t partial[t][C+1]  (t ascending)
__global__ void readout_reduce_kernel(const float* __restrict__ partial, int b, int C, float* __restrict__ dwout,
                                      float* __restrict__ nll, float* __restrict__ count, int accumulate) {
    const int c = threadIdx.x;
    if (c >= C + 2) return;
    float s = 0.f;
    for (int t = 0; t < b; ++t) s += partial[(size_t)t * (C + 2) + c];
    float* dst = c < C ? dwout + c : (c == C ? nll : count);
    if (dst) *dst = accumulate ? *dst + s : s;
}

__global__ void adam_kernel(float* __restrict__ W, float* __restrict__ m, float* __restrict__ v, const float* __restrict__ gradbuf,
                            long long n, float lr, float wd, float b1, float b2, float eps, float c1, float c2,
                            const int* __restrict__ overflow) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    // a micro-batch exceeded a row-list capacity: the accumulated gradients are truncated -> leave weights and Adam state alone
    // (the flag stays set; scone_model_check_overflow / read_grads / forward_host report it as error code 4)
    if (overflow != nullptr && *overflow != 0) return;
    const float count = gradbuf[n + 1];
    const float g = gradbuf[i] / count + 2.f * wd * W[i];
    const float mi = (1.f - b1) * g + b1 * m[i];
    const float vi = (1.f - b2) * g * g + b2 * v[i];
    m[i] = mi;
    v[i] = vi;
    W[i] = W[i] - lr * (mi / c1) / (sqrtf(vi / c2) + eps);
}

}  // namespace

bool g_scone_zero_fill = true;

namespace {

// =================================================================================================================
// launchers
// =================================================================================================================
int grid_for(const scone_complex* cx, long long n_work, int ctas_per_sm) {
    long long g = (long long)cx->num_sms * ctas_per_sm;
    if (n_work < g) g = n_work > 0 ? n_work : 1;
    return (int)g;
}

template <typename K>
int occupancy_of(K kern, size_t smem, int* out) {
    int occ = 1;
    SCONE_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SCONE_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kThreads, smem));
    *out = occ > 0 ? occ : 1;
    return 0;
}

// scratch carved from the caller's occ_scratch buffer (scone_occ_scratch_bytes): two worklists (ping-pong), counters
struct UnitScratch {
    uint32_t* wl[2];
    int* n[2];
    int* counts;
    uint32_t* bm;                       // row bitmap of the flags a call produces (scatter -> compaction)
    unsigned long long* tickets;        // look-back tickets of compact_bitmap_kernel
    uint8_t* occ_tmp;
};
constexpr int kTicketSlots = 1024;
size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }
size_t max_units(const scone_complex* cx, int b) { return (size_t)cx->E * (size_t)b; }   // a worklist may also hold row ids
UnitScratch carve_scratch(const scone_complex* cx, int b, uint8_t* base) {
    UnitScratch sc;
    const size_t nu = max_units(cx, b);
    size_t off = 0;
    sc.wl[0] = reinterpret_cast<uint32_t*>(base + off); off += align256(nu * 4);
    sc.wl[1] = reinterpret_cast<uint32_t*>(base + off); off += align256(nu * 4);
    sc.counts = reinterpret_cast<int*>(base + off); off += align256((nu / kCompactBlock + 2) * 4);
    sc.n[0] = reinterpret_cast<int*>(base + off); off += 256;
    sc.n[1] = reinterpret_cast<int*>(base + off); off += 256;
    sc.bm = reinterpret_cast<uint32_t*>(base + off); off += align256(scone_bitmap_words(cx->E, b) * 4);
    sc.tickets = reinterpret_cast<unsigned long long*>(base + off); off += align256(kTicketSlots * 8);
    sc.occ_tmp = base + off;
    return sc;
}

template <int TT>
int compact_units(const scone_complex* cx, int b, const uint8_t* flags, uint32_t* list, int* counts, int* n_ptr, cudaStream_t st) {
    const int nchunk = (b + TT - 1) / TT;
    const long long n_units = (long long)cx->E * nchunk;
    const int nblk = (int)((n_units + kCompactBlock - 1) / kCompactBlock);
    compact_units_kernel<TT, false><<<nblk, kThreads, 0, st>>>(flags, n_units, nchunk, b, counts, nullptr);
    SCONE_LAUNCHED();
    scan_counts_kernel<<<1, 1024, 0, st>>>(counts, nblk, n_ptr);
    SCONE_LAUNCHED();
    compact_units_kernel<TT, true><<<nblk, kThreads, 0, st>>>(flags, n_units, nchunk, b, counts, list);
    SCONE_LAUNCHED();
    return 0;
}

// The same worklist from the quad bitmap of the flags (TT in {4, 8, 16}, b % TT == 0): one launch over E*b/32 bytes.
bool bitmap_ok(int tt, int b) { return (tt == 4 || tt == 8 || tt == 16) && b % tt == 0; }

template <int TT>
int compact_bitmap(const scone_complex* cx, int b, const uint32_t* bm, uint32_t* list, int* n_ptr, unsigned long long* tickets,
                   cudaStream_t st, uint32_t* pref_out = nullptr, long long list_cap = (1ll << 62)) {
    constexpr int R = TT;                // TT = 1: row list
    const long long n_words = ((long long)cx->E * b + 31) / 32;
    int grid = cx->num_sms * 4 < kTicketSlots ? cx->num_sms * 4 : kTicketSlots;
    if (n_words < (long long)grid * 16 * kThreads) grid = (int)((n_words + 16 * kThreads - 1) / (16 * kThreads));
    if (grid < 1) grid = 1;
    SCONE_CUDA(cudaMemsetAsync(tickets, 0, (size_t)grid * 8, st));
    compact_bitmap_kernel<R><<<grid, kThreads, 0, st>>>(bm, n_words, list, n_ptr, tickets, pref_out, list_cap);
    SCONE_LAUNCHED();
    return 0;
}

// Input worklist: the caller's hint (the previous launch's output worklist, same flags, same TT) or a fresh compaction.
template <int TT>
int input_worklist(const scone_complex* cx, int b, const uint8_t* occ_in, const UnitScratch& sc, cudaStream_t st,
                   const SconeLaunchHints* h, int* in) {
    if (h && h->in_wl >= 0 && h->in_tt == TT) {
        *in = h->in_wl;
        return 0;
    }
    *in = 0;
    if (h && h->in_bm != nullptr && bitmap_ok(TT, b)) return compact_bitmap<TT>(cx, b, h->in_bm, sc.wl[0], sc.n[0], sc.tickets, st);
    return compact_units<TT>(cx, b, occ_in, sc.wl[0], sc.counts, sc.n[0], st);
}

// worklist(occ_in) -> one-hop scatter into occ_out -> worklist(occ_out); *out = index of that worklist in sc (also h->out_wl)
template <int TT>
int prepare_units(const scone_complex* cx, int b, const uint8_t* occ_in, uint8_t* occ_out, const UnitScratch& sc, cudaStream_t st,
                  SconeLaunchHints* h, int* out) {
    int in = 0;
    if (input_worklist<TT>(cx, b, occ_in, sc, st, h, &in)) return 1;
    SCONE_CUDA(cudaMemsetAsync(occ_out, 0, (size_t)cx->E * b, st));
    uint32_t* bm = bitmap_ok(TT, b) ? sc.bm : nullptr;
    if (bm) SCONE_CUDA(cudaMemsetAsync(bm, 0, scone_bitmap_words(cx->E, b) * 4, st));
    scatter_support_kernel<TT><<<cx->num_sms * 8, kThreads, 0, st>>>(sc.wl[in], sc.n[in], occ_in, occ_out, bm, cx->S(0), cx->S(1),
                                                                     (b + TT - 1) / TT, b);
    SCONE_LAUNCHED();
    *out = 1 - in;
    if (h) {
        h->out_wl = *out;
        h->out_tt = TT;
    }
    if (bm) return compact_bitmap<TT>(cx, b, bm, sc.wl[*out], sc.n[*out], sc.tickets, st);
    return compact_units<TT>(cx, b, occ_out, sc.wl[*out], sc.counts, sc.n[*out], st);
}

bool zero_fill_here(const SconeLaunchHints* h) { return g_scone_zero_fill && !(h && h->skip_fill); }

template <int CIN, int COUT, int ACT>
int launch_fwd(const scone_complex* cx, int b, const float* Hin, const float* W0, const float* W1, const float* W2, float* Hout,
               const uint8_t* occ_in, uint8_t* occ_out, uint8_t* scratch, cudaStream_t st, SconeLaunchHints* h) {
    constexpr int TT = kTileCols / CIN, TE = kTileRows / TT, KD = 3 * CIN, LDT = KD + 4;
    ScopedProf prof(SCONE_K_LAYER_FWD, st);
    if (occ_in == nullptr) {                                  // dense path
        if (scone_slab_supported(cx, CIN, COUT)) {            // slab kernel: merged-row gather into mma fragments, 3xTF32 product
            if (scone_slab_forward(cx, ACT, b, CIN, COUT, Hin, W0, W1, W2, Hout, st)) return 1;
            if (occ_out) SCONE_CUDA(cudaMemsetAsync(occ_out, 1, (size_t)cx->E * b, st));
            return 0;
        }
        const long long n_tiles = (long long)((b + TT - 1) / TT) * ((cx->E + TE - 1) / TE);
        {                                                     // fp32 SIMT register-tiled product
            const size_t smem = ((size_t)kTileRows * LDT + (size_t)KD * COUT) * sizeof(float);
            auto kern = layer_fwd_dense_kernel<CIN, COUT, ACT>;
            static int occ = 0;
            if (!occ && occupancy_of(kern, smem, &occ)) return 1;
            kern<<<grid_for(cx, n_tiles, occ), kThreads, smem, st>>>(Hin, Hout, W0, W1, W2, cx->S(0), cx->S(1), cx->E, b);
        }
        SCONE_LAUNCHED();
        if (occ_out) SCONE_CUDA(cudaMemsetAsync(occ_out, 1, (size_t)cx->E * b, st));   // no information: everything may be non-zero
        return 0;
    }
    SCONE_REQUIRE(occ_out != nullptr && scratch != nullptr, "scone_layer_forward: occ_in needs occ_out and occ_scratch");
    const UnitScratch sc = carve_scratch(cx, b, scratch);
    int wo = 0;
    if (prepare_units<TT>(cx, b, occ_in, occ_out, sc, st, h, &wo)) return 1;
    if (zero_fill_here(h) && scone_zero_fill(cx, Hout, (size_t)cx->E * b * COUT * sizeof(float), st)) return 1;
    if (scone_slab_supported(cx, CIN, COUT) && bitmap_ok(TT, b)) {
        // candidate ROWS of the output (row bitmap of occ_out, still in the scratch) -> compacted list -> row-list kernel.  The
        // list goes where the consumed input worklist was; the output unit worklist (hint for the next call) stays intact.
        const int wi = 1 - wo;
        if (compact_bitmap<1>(cx, b, sc.bm, sc.wl[wi], sc.n[wi], sc.tickets, st)) return 1;
        return scone_slab_forward_rows(cx, ACT, b, CIN, COUT, Hin, W0, W1, W2, Hout, occ_in, sc.wl[wi], sc.n[wi],
                                       scone_prof_row_counter(SCONE_K_LAYER_FWD), nullptr, nullptr, 0, nullptr, st);
    }
    const size_t smem = ((size_t)KD * COUT + (size_t)kWarps * TT * LDT) * sizeof(float);
    auto kern = layer_fwd_units_kernel<CIN, COUT, ACT>;
    static int occ = 0;
    if (!occ && occupancy_of(kern, smem, &occ)) return 1;
    kern<<<cx->num_sms * occ, kThreads, smem, st>>>(Hin, Hout, W0, W1, W2, cx->S(0), cx->S(1), cx->E, b, occ_in, occ_out, sc.wl[wo],
                                                  sc.n[wo], scone_prof_row_counter(SCONE_K_LAYER_FWD));
    SCONE_LAUNCHED();
    return 0;
}

template <int CIN, int COUT>
int dispatch_fwd_act(const scone_complex* cx, int act, int b, const float* Hin, const float* W0, const float* W1, const float* W2,
                     float* Hout, const uint8_t* occ_in, uint8_t* occ_out, uint8_t* scratch, cudaStream_t st, SconeLaunchHints* h) {
    switch (act) {
        case SCONE_ACT_TANH: return launch_fwd<CIN, COUT, SCONE_ACT_TANH>(cx, b, Hin, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, h);
        case SCONE_ACT_LEAKY_RELU: return launch_fwd<CIN, COUT, SCONE_ACT_LEAKY_RELU>(cx, b, Hin, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, h);
        case SCONE_ACT_RELU: return launch_fwd<CIN, COUT, SCONE_ACT_RELU>(cx, b, Hin, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, h);
    }
    scone_set_error("unknown activation %d", act);
    return 2;
}

constexpr int kBwdMaxCtas = 148 * 8;     // upper bound on persistent CTAs (workspace sizing)

template <int CIN, int COUT, int ACT, bool WG>
int launch_bwd(const scone_complex* cx, int b, const float* G, const float* Hin, const float* W0, const float* W1, const float* W2,
               float* Gprev, float* dW, int accumulate, float* ws, const uint8_t* occ_g, const uint8_t* occ_h, uint8_t* occ_prev,
               uint8_t* scratch, cudaStream_t st, SconeLaunchHints* h) {
    using Sh = BwdShape<CIN, COUT>;
    ScopedProf prof(SCONE_K_LAYER_BWD, st);
    int grid = 1;
    if (occ_g == nullptr) {                                   // dense path
        size_t smem_f = (size_t)kTileRows * Sh::LDA + (size_t)kTileRows * Sh::LDH + (size_t)Sh::KD * CIN;
        if ((size_t)Sh::RS * Sh::DW > smem_f) smem_f = (size_t)Sh::RS * Sh::DW;
        const size_t smem = smem_f * sizeof(float);
        auto kern = layer_bwd_dense_kernel<CIN, COUT, ACT, WG>;
        static int occ = 0;
        if (!occ && occupancy_of(kern, smem, &occ)) return 1;
        const long long n_tiles = (long long)((b + Sh::TT - 1) / Sh::TT) * ((cx->E + Sh::TE - 1) / Sh::TE);
        grid = grid_for(cx, n_tiles, occ);
        if (grid > kBwdMaxCtas) grid = kBwdMaxCtas;
        kern<<<grid, kThreads, smem, st>>>(G, Hin, Gprev, W0, W1, W2, ws, cx->S(0), cx->S(1), cx->E, b);
        SCONE_LAUNCHED();
        if (WG && occ_prev) SCONE_CUDA(cudaMemsetAsync(occ_prev, 1, (size_t)cx->E * b, st));
    } else {
        using Us = BwdUnitShape<CIN, COUT>;
        SCONE_REQUIRE(scratch != nullptr && (!WG || occ_prev != nullptr), "scone_layer_backward: occ_g needs occ_gprev and occ_scratch");
        const UnitScratch sc = carve_scratch(cx, b, scratch);
        uint8_t* cand = WG ? occ_prev : sc.occ_tmp;           // rows whose (G, S0 G, S1 G) can be non-zero
        int wo = 0;
        if (prepare_units<Us::TT>(cx, b, occ_g, cand, sc, st, h, &wo)) return 1;
        if (WG && zero_fill_here(h) && scone_zero_fill(cx, Gprev, (size_t)cx->E * b * CIN * sizeof(float), st)) return 1;
        const size_t smem = Us::smem_floats * sizeof(float);
        auto kern = layer_bwd_units_kernel<CIN, COUT, ACT, WG>;
        static int occ = 0;
        if (!occ && occupancy_of(kern, smem, &occ)) return 1;
        grid = cx->num_sms * occ;
        if (grid > kBwdMaxCtas) grid = kBwdMaxCtas;
        kern<<<grid, kThreads, smem, st>>>(G, Hin, Gprev, W0, W1, W2, ws, cx->S(0), cx->S(1), cx->E, b, occ_g, occ_h, cand, sc.wl[wo],
                                          sc.n[wo], scone_prof_row_counter(SCONE_K_LAYER_BWD));
        SCONE_LAUNCHED();
    }
    reduce_partials_kernel<<<(Sh::DW + 31) / 32, 256, 0, st>>>(ws, grid, Sh::DW, dW, accumulate);
    SCONE_LAUNCHED();
    return 0;
}

template <int CIN, int COUT>
int dispatch_bwd_act(const scone_complex* cx, int act, int b, const float* G, const float* Hin, const float* W0, const float* W1,
                     const float* W2, float* Gprev, float* dW, int accumulate, float* ws, const uint8_t* occ_g, const uint8_t* occ_h,
                     uint8_t* occ_prev, uint8_t* scratch, cudaStream_t st, SconeLaunchHints* h) {
#define SCONE_BWD_CASE(A)                                                                                                          \
    case A:                                                                                                                        \
        return Gprev ? launch_bwd<CIN, COUT, A, true>(cx, b, G, Hin, W0, W1, W2, Gprev, dW, accumulate, ws, occ_g, occ_h, occ_prev, \
                                                      scratch, st, h)                                                              \
                     : launch_bwd<CIN, COUT, A, false>(cx, b, G, Hin, W0, W1, W2, Gprev, dW, accumulate, ws, occ_g, occ_h, occ_prev, \
                                                       scratch, st, h);
    switch (act) {
        SCONE_BWD_CASE(SCONE_ACT_TANH)
        SCONE_BWD_CASE(SCONE_ACT_LEAKY_RELU)
        SCONE_BWD_CASE(SCONE_ACT_RELU)
    }
#undef SCONE_BWD_CASE
    scone_set_error("unknown activation %d", act);
    return 2;
}

bool width_ok(int c) { return c == 8 || c == 16 || c == 32 || c == 64; }

}  // namespace

// ascending list of the set bits of a row bitmap (ids e*b + t) and their count, both on the device; tickets: kTicketSlots * 8 bytes
int scone_compact_rows(const scone_complex* cx, int b, const uint32_t* bm, uint32_t* list, int* n_dev, unsigned long long* tickets,
                       cudaStream_t st, uint32_t* pref_out, long long list_cap) {
    return compact_bitmap<1>(cx, b, bm, list, n_dev, tickets, st, pref_out, list_cap);
}
size_t scone_ticket_bytes() { return (size_t)kTicketSlots * 8; }

// zero-fill `bytes` (multiple of 16) at p on stream st with the library's own kernel
int scone_zero_fill(const scone_complex* cx, void* p, size_t bytes, cudaStream_t st) {
    if (bytes == 0) return 0;
    if ((bytes & 15) || ((uintptr_t)p & 15)) {
        SCONE_CUDA(cudaMemsetAsync(p, 0, bytes, st));
        return 0;
    }
    ScopedProf prof(SCONE_K_FILL, st);
    const size_t n16 = bytes / 16;
    // the (unused) dynamic shared memory caps residency at ~4 fill CTAs per SM, leaving slots for the concurrent kernels
    static bool configured = false;
    const int fill_smem = getenv("SCONE_FILL_SMEM") ? atoi(getenv("SCONE_FILL_SMEM")) : 56 * 1024;
    if (!configured) {
        SCONE_CUDA(cudaFuncSetAttribute(zero_fill_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        configured = true;
    }
    zero_fill_kernel<<<(unsigned)((n16 + (size_t)kThreads * 8 - 1) / ((size_t)kThreads * 8)), kThreads, fill_smem, st>>>(reinterpret_cast<float4*>(p), n16);
    SCONE_LAUNCHED();
    return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------------------------
extern "C" int scone_set_zero_fill(int32_t on) {
    g_scone_zero_fill = on != 0;
    return 0;
}
extern "C" int scone_get_zero_fill(void) { return g_scone_zero_fill ? 1 : 0; }

#define SCONE_DISPATCH_WIDTHS(FN, ...)                                              \
    do {                                                                            \
        const int key_ = cin * 1000 + cout;                                         \
        switch (key_) {                                                             \
            case 8008: return FN<8, 8>(__VA_ARGS__);                                \
            case 8016: return FN<8, 16>(__VA_ARGS__);                               \
            case 16008: return FN<16, 8>(__VA_ARGS__);                              \
            case 16016: return FN<16, 16>(__VA_ARGS__);                             \
            case 16032: return FN<16, 32>(__VA_ARGS__);                             \
            case 32016: return FN<32, 16>(__VA_ARGS__);                             \
            case 32032: return FN<32, 32>(__VA_ARGS__);                             \
            case 32064: return FN<32, 64>(__VA_ARGS__);                             \
            case 64032: return FN<64, 32>(__VA_ARGS__);                             \
            case 64064: return FN<64, 64>(__VA_ARGS__);                             \
        }                                                                           \
    } while (0)

extern "C" int64_t scone_occ_scratch_bytes(const scone_complex* cx, int32_t b) {
    if (!cx || b <= 0) return 0;
    const size_t nu = max_units(cx, b);
    return (int64_t)(2 * align256(nu * 4) + align256((nu / kCompactBlock + 2) * 4) + 512 + align256(scone_bitmap_words(cx->E, b) * 4) +
                     align256(kTicketSlots * 8) + align256((size_t)cx->E * b));
}

int scone_layer_forward_hinted(const scone_complex* cx, int32_t act, int32_t b, int32_t cin, int32_t cout, const float* Hin,
                               const float* W0, const float* W1, const float* W2, float* Hout, const uint8_t* occ_in,
                               uint8_t* occ_out, uint8_t* occ_scratch, void* stream, SconeLaunchHints* hints) {
    SCONE_REQUIRE(cx && Hin && W0 && W1 && W2 && Hout, "scone_layer_forward: NULL argument");
    SCONE_REQUIRE(!cx->host_only, "scone_layer_forward: index-only complex has no device arrays");
    SCONE_REQUIRE(b > 0, "scone_layer_forward: b must be positive");
    if (cin == 1) return scone_layer0_forward(cx, act, b, cout, Hin, W0, W1, W2, Hout, occ_in, occ_out, occ_scratch, stream, hints);
    SCONE_REQUIRE(width_ok(cin) && width_ok(cout),
                  "scone_layer_forward: hidden widths must be in {8,16,32,64} with |log2 ratio| <= 1 (got %d -> %d)", cin, cout);
    SCONE_DISPATCH_WIDTHS(dispatch_fwd_act, cx, act, b, Hin, W0, W1, W2, Hout, occ_in, occ_out, occ_scratch, as_stream(stream), hints);
    scone_set_error("scone_layer_forward: unsupported width pair %d -> %d", cin, cout);
    return 2;
}

extern "C" int scone_layer_forward(const scone_complex* cx, int32_t act, int32_t b, int32_t cin, int32_t cout, const float* Hin,
                                   const float* W0, const float* W1, const float* W2, float* Hout, const uint8_t* occ_in,
                                   uint8_t* occ_out, uint8_t* occ_scratch, void* stream) {
    return scone_layer_forward_hinted(cx, act, b, cin, cout, Hin, W0, W1, W2, Hout, occ_in, occ_out, occ_scratch, stream, nullptr);
}

extern "C" int64_t scone_layer_backward_workspace_bytes(int32_t cin, int32_t cout) {
    if (cin == 1) return scone_layer0_backward_workspace_bytes(cout);
    return (int64_t)kBwdMaxCtas * 3 * cin * cout * sizeof(float);
}

int scone_layer_backward_hinted(const scone_complex* cx, int32_t act, int32_t b, int32_t cin, int32_t cout, const float* G,
                                const float* Hin, const float* W0, const float* W1, const float* W2, float* Gprev, float* dW,
                                int32_t accumulate, void* workspace, const uint8_t* occ_g, const uint8_t* occ_hin,
                                uint8_t* occ_prev, uint8_t* occ_scratch, void* stream, SconeLaunchHints* hints) {
    SCONE_REQUIRE(cx && G && Hin && dW && workspace, "scone_layer_backward: NULL argument");
    SCONE_REQUIRE(!cx->host_only, "scone_layer_backward: index-only complex has no device arrays");
    SCONE_REQUIRE(b > 0, "scone_layer_backward: b must be positive");
    if (cin == 1) return scone_layer0_backward(cx, b, cout, G, Hin, dW, accumulate, workspace, occ_g, occ_scratch, stream, hints);
    SCONE_REQUIRE(W0 && W1 && W2, "scone_layer_backward: NULL weights");
    SCONE_REQUIRE(width_ok(cin) && width_ok(cout),
                  "scone_layer_backward: hidden widths must be in {8,16,32,64} with |log2 ratio| <= 1 (got %d -> %d)", cin, cout);
    if (g_scone_dense_kernel == 3 && occ_g == nullptr && scone_umma_supported(cx, cin, cout, b)) {      // tcgen05 / TMEM (scone_umma.cu)
        ScopedProf prof(SCONE_K_LAYER_BWD, as_stream(stream));
        if (Gprev && occ_prev) SCONE_CUDA(cudaMemsetAsync(occ_prev, 1, (size_t)cx->E * b, as_stream(stream)));
        return scone_umma_backward(cx, act, b, G, Hin, W0, W1, W2, Gprev, dW, accumulate, (float*)workspace, as_stream(stream));
    }
    SCONE_DISPATCH_WIDTHS(dispatch_bwd_act, cx, act, b, G, Hin, W0, W1, W2, Gprev, dW, accumulate, (float*)workspace, occ_g, occ_hin,
                          occ_prev, occ_scratch, as_stream(stream), hints);
    scone_set_error("scone_layer_backward: unsupported width pair %d -> %d", cin, cout);
    return 2;
}

extern "C" int scone_layer_backward(const scone_complex* cx, int32_t act, int32_t b, int32_t cin, int32_t cout, const float* G,
                                    const float* Hin, const float* W0, const float* W1, const float* W2, float* Gprev, float* dW,
                                    int32_t accumulate, void* workspace, const uint8_t* occ_g, const uint8_t* occ_hin,
                                    uint8_t* occ_prev, uint8_t* occ_scratch, void* stream) {
    return scone_layer_backward_hinted(cx, act, b, cin, cout, G, Hin, W0, W1, W2, Gprev, dW, accumulate, workspace, occ_g, occ_hin,
                                       occ_prev, occ_scratch, stream, nullptr);
}

template <int COUT, int ACT>
static int launch_l0_fwd_act(const scone_complex* cx, int b, const float* X, const float* W0, const float* W1, const float* W2,
                             float* Hout, const uint8_t* occ_in, uint8_t* occ_out, uint8_t* scratch, cudaStream_t st,
                             SconeLaunchHints* h) {
    ScopedProf prof(SCONE_K_LAYER0_FWD, st);
    if (occ_in == nullptr) {               // dense: every row is computed; flags (if wanted) are value based
        const long long n_tiles = (long long)((b + 31) / 32) * ((cx->E + kL0Edges - 1) / kL0Edges);
        layer0_fwd_kernel<COUT, ACT><<<grid_for(cx, n_tiles, 6), kThreads, 0, st>>>(X, Hout, W0, W1, W2, cx->S(0), cx->S(1), cx->E, b,
                                                                                   occ_out, 1);
        SCONE_LAUNCHED();
        return 0;
    }
    SCONE_REQUIRE(occ_out != nullptr && scratch != nullptr, "scone_layer_forward: occ_in needs occ_out and occ_scratch");
    constexpr int TT = kTileCols / COUT;
    const UnitScratch sc = carve_scratch(cx, b, scratch);
    int wo = 0;
    if (prepare_units<TT>(cx, b, occ_in, occ_out, sc, st, h, &wo)) return 1;
    if (zero_fill_here(h) && scone_zero_fill(cx, Hout, (size_t)cx->E * b * COUT * sizeof(float), st)) return 1;
    layer0_fwd_units_kernel<COUT, ACT><<<cx->num_sms * 8, kThreads, 0, st>>>(X, Hout, W0, W1, W2, cx->S(0), cx->S(1), cx->E, b, occ_out,
                                                                            sc.wl[wo], sc.n[wo]);
    SCONE_LAUNCHED();
    return 0;
}

template <int COUT>
static int launch_l0_fwd(const scone_complex* cx, int act, int b, const float* X, const float* W0, const float* W1, const float* W2,
                         float* Hout, const uint8_t* occ_in, uint8_t* occ_out, uint8_t* scratch, cudaStream_t st, SconeLaunchHints* h) {
    switch (act) {
        case SCONE_ACT_TANH: return launch_l0_fwd_act<COUT, SCONE_ACT_TANH>(cx, b, X, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, h);
        case SCONE_ACT_LEAKY_RELU: return launch_l0_fwd_act<COUT, SCONE_ACT_LEAKY_RELU>(cx, b, X, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, h);
        case SCONE_ACT_RELU: return launch_l0_fwd_act<COUT, SCONE_ACT_RELU>(cx, b, X, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, h);
    }
    scone_set_error("unknown activation %d", act);
    return 2;
}

int scone_layer0_forward(const scone_complex* cx, int32_t act, int32_t b, int32_t cout, const float* X, const float* W0,
                         const float* W1, const float* W2, float* Hout, const uint8_t* occ_in, uint8_t* occ_out, uint8_t* scratch,
                         void* stream, SconeLaunchHints* hints) {
    cudaStream_t st = as_stream(stream);
    switch (cout) {
        case 8: return launch_l0_fwd<8>(cx, act, b, X, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, hints);
        case 16: return launch_l0_fwd<16>(cx, act, b, X, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, hints);
        case 32: return launch_l0_fwd<32>(cx, act, b, X, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, hints);
        case 64: return launch_l0_fwd<64>(cx, act, b, X, W0, W1, W2, Hout, occ_in, occ_out, scratch, st, hints);
    }
    scone_set_error("scone_layer_forward: first-layer width must be in {8,16,32,64} (got %d)", cout);
    return 2;
}

constexpr int kL0BwdCtas = 148 * 8;
int64_t scone_layer0_backward_workspace_bytes(int32_t cout) { return (int64_t)kL0BwdCtas * 3 * cout * sizeof(float); }

template <int COUT>
static int launch_l0_bwd(const scone_complex* cx, int b, const float* G, const float* X, float* dW, int accumulate, float* ws,
                         const uint8_t* occ_g, uint8_t* scratch, cudaStream_t st, const SconeLaunchHints* h) {
    ScopedProf prof(SCONE_K_LAYER0_BWD, st);
    int grid;
    if (occ_g == nullptr) {
        const long long n_tiles = (long long)((b + 31) / 32) * ((cx->E + kL0Edges - 1) / kL0Edges);
        grid = grid_for(cx, n_tiles, 4);
        if (grid > kL0BwdCtas) grid = kL0BwdCtas;
        layer0_bwd_dense_kernel<COUT><<<grid, kThreads, 0, st>>>(X, G, ws, cx->S(0), cx->S(1), cx->E, b);
    } else {
        SCONE_REQUIRE(scratch != nullptr, "scone_layer_backward: occ_g needs occ_scratch");
        constexpr int TT = kTileCols / COUT;
        const UnitScratch sc = carve_scratch(cx, b, scratch);
        int wi = 0;
        if (input_worklist<TT>(cx, b, occ_g, sc, st, h, &wi)) return 1;
        grid = cx->num_sms * 4;
        if (grid > kL0BwdCtas) grid = kL0BwdCtas;
        layer0_bwd_units_kernel<COUT><<<grid, kThreads, 0, st>>>(X, G, ws, cx->S(0), cx->S(1), cx->E, b, occ_g, sc.wl[wi], sc.n[wi]);
    }
    SCONE_LAUNCHED();
    reduce_partials_kernel<<<(3 * COUT + 31) / 32, 256, 0, st>>>(ws, grid, 3 * COUT, dW, accumulate);
    SCONE_LAUNCHED();
    return 0;
}

int scone_layer0_backward(const scone_complex* cx, int32_t b, int32_t cout, const float* G, const float* X, float* dW,
                          int32_t accumulate, void* workspace, const uint8_t* occ_g, uint8_t* scratch, void* stream,
                          const SconeLaunchHints* hints) {
    cudaStream_t st = as_stream(stream);
    float* ws = (float*)workspace;
    switch (cout) {
        case 8: return launch_l0_bwd<8>(cx, b, G, X, dW, accumulate, ws, occ_g, scratch, st, hints);
        case 16: return launch_l0_bwd<16>(cx, b, G, X, dW, accumulate, ws, occ_g, scratch, st, hints);
        case 32: return launch_l0_bwd<32>(cx, b, G, X, dW, accumulate, ws, occ_g, scratch, st, hints);
        case 64: return launch_l0_bwd<64>(cx, b, G, X, dW, accumulate, ws, occ_g, scratch, st, hints);
    }
    scone_set_error("scone_layer_backward: first-layer width must be in {8,16,32,64} (got %d)", cout);
    return 2;
}

int scone_flows_to_dense_hinted(const scone_complex* cx, int32_t b, const int32_t* traj_ptr, const int32_t* flow_edge,
                                const float* flow_val, float* X, uint8_t* occX, void* stream, const SconeLaunchHints* hints) {
    SCONE_REQUIRE(cx && traj_ptr && X && b > 0, "scone_flows_to_dense: bad argument");
    SCONE_REQUIRE(!cx->host_only, "scone_flows_to_dense: index-only complex has no device arrays");
    cudaStream_t st = as_stream(stream);
    ScopedProf prof(SCONE_K_OTHER, st);
    SCONE_CUDA(cudaMemsetAsync(X, 0, (size_t)cx->E * b * sizeof(float), st));
    if (occX) SCONE_CUDA(cudaMemsetAsync(occX, 0, (size_t)cx->E * b, st));
    uint32_t* bm = (hints && occX != nullptr && b % 4 == 0) ? hints->out_bm : nullptr;
    if (bm) SCONE_CUDA(cudaMemsetAsync(bm, 0, scone_bitmap_words(cx->E, b) * 4, st));
    flows_to_dense_kernel<<<(b * 32 + 255) / 256, 256, 0, st>>>(traj_ptr, flow_edge, flow_val, cx->d_rank, X, occX, bm, cx->E, b);
    SCONE_LAUNCHED();
    return 0;
}

extern "C" int scone_flows_to_dense(const scone_complex* cx, int32_t b, const int32_t* traj_ptr, const int32_t* flow_edge,
                                    const float* flow_val, float* X, uint8_t* occX, void* stream) {
    return scone_flows_to_dense_hinted(cx, b, traj_ptr, flow_edge, flow_val, X, occX, stream, nullptr);
}

int64_t scone_readout_workspace_bytes(int32_t b, int32_t C) { return (int64_t)b * (C + 2) * sizeof(float); }

int scone_readout_ws(const scone_complex* cx, int32_t act, int32_t b, int32_t C, const float* HL, const float* wout,
                     const int32_t* last_nodes, float* logprobs, const int32_t* target_idx, const float* mask, float scale,
                     float* GL, float* dwout, float* nll_sum, float* count, int32_t accumulate, void* workspace,
                     const uint8_t* occ_HL, uint8_t* occ_GL, void* stream, const SconeLaunchHints* hints) {
    SCONE_REQUIRE(cx && HL && wout && last_nodes && logprobs, "scone_readout: NULL argument");
    SCONE_REQUIRE(!cx->host_only, "scone_readout: index-only complex has no device arrays");
    SCONE_REQUIRE(C >= 1 && C <= 32 * kReadoutMaxCper, "scone_readout: C must be in [1,%d]", 32 * kReadoutMaxCper);
    SCONE_REQUIRE(cx->D <= kReadoutMaxD, "scone_readout: max degree %d exceeds %d", cx->D, kReadoutMaxD);
    cudaStream_t st = as_stream(stream);
    ScopedProf prof(SCONE_K_READOUT, st);
    const SconeLaunchHints h = hints ? *hints : SconeLaunchHints{};
    if (GL) {
        SCONE_REQUIRE(target_idx && mask && workspace, "scone_readout: gradient mode needs target_idx, mask, workspace");
        // without flags the consumer reads every row of GL: it must be dense zeros; with flags only when zero-fill is on
        const bool flagged = occ_GL != nullptr || h.out_bm != nullptr;
        if ((!flagged || zero_fill_here(&h)) && scone_zero_fill(cx, GL, (size_t)cx->E * b * C * sizeof(float), st)) return 1;
        if (occ_GL) SCONE_CUDA(cudaMemsetAsync(occ_GL, 0, (size_t)cx->E * b, st));
    }
    const uint32_t* bm_HL = h.in_bm;                       // row-bitmap pipeline: bits instead of flag bytes
    uint32_t* bm_cand = GL ? h.cand_bm : nullptr;
    uint32_t* bm = (GL && (occ_GL || bm_HL)) ? h.out_bm : nullptr;
    if (bm) SCONE_CUDA(cudaMemsetAsync(bm, 0, scone_bitmap_words(cx->E, b) * 4, st));
    if (bm_cand) SCONE_CUDA(cudaMemsetAsync(bm_cand, 0, scone_bitmap_words(cx->E, b) * 4, st));
    readout_kernel<<<b, 32 * kReadoutWarps, 0, st>>>(HL, wout, last_nodes, cx->d_nbrhoods, cx->d_inc_ptr, cx->d_inc_ent, logprobs,
                                              target_idx, mask, scale, GL, (float*)workspace, occ_HL, GL ? occ_GL : nullptr, bm, act,
                                              cx->N, cx->D, b, C, bm_HL, bm_cand, cx->d_mptr, cx->d_ment);
    SCONE_LAUNCHED();
    if (GL) {
        readout_reduce_kernel<<<1, ((C + 2 + 31) / 32) * 32, 0, st>>>((const float*)workspace, b, C, dwout, nll_sum, count, accumulate);
        SCONE_LAUNCHED();
    }
    return 0;
}

extern "C" int64_t scone_readout_workspace(int32_t b, int32_t C) { return scone_readout_workspace_bytes(b, C); }

extern "C" int scone_readout(const scone_complex* cx, int32_t act, int32_t b, int32_t C, const float* HL, const float* wout,
                             const int32_t* last_nodes, float* logprobs, const int32_t* target_idx, const float* mask, float scale,
                             float* GL, float* dwout, float* nll_sum, float* count, int32_t accumulate, void* workspace,
                             const uint8_t* occ_HL, uint8_t* occ_GL, void* stream) {
    return scone_readout_ws(cx, act, b, C, HL, wout, last_nodes, logprobs, target_idx, mask, scale, GL, dwout, nll_sum, count,
                            accumulate, workspace, occ_HL, occ_GL, stream, nullptr);
}

int scone_adam_launch(float* W, float* m, float* v, const float* gradbuf, int64_t n, int32_t step, float lr, float wd, void* stream,
                      const int* overflow_dev) {
    const float b1 = 0.9f, b2 = 0.999f, eps = 1e-8f;
    const float c1 = 1.f - powf(b1, (float)(step + 1)), c2 = 1.f - powf(b2, (float)(step + 1));
    adam_kernel<<<(int)((n + 255) / 256), 256, 0, as_stream(stream)>>>(W, m, v, gradbuf, (long long)n, lr, wd, b1, b2, eps, c1, c2, overflow_dev);
    SCONE_LAUNCHED();
    return 0;
}
