// scone_bunch.cu — SCCONV / "bunch" model (trajectory_experiments.py:173-203, bunch_model_matrices.py:118-135).
//
// Three-level message passing (nodes V, edges H, triangles T) with seven weighted shift operators S_00 .. S_22 per
// layer and relu after every layer; readout = node values at the (padded, -1 wraps to node N-1: quirk Q2) neighbours of
// the last node, log-softmax, NLL.  The operators are diagonal rescalings of incidence products (non-integer values,
// non-square), so this path uses generic float CSR operators and simple deterministic kernels (CSR x dense, small dense
// products, fixed-tree reductions); it is meant for the reference's complex sizes (config 3), not for the 1M-edge runs.
#include <cstring>
#include <vector>
#include "common.cuh"

struct scone_csr {
    int32_t rows = 0, cols = 0;
    int64_t nnz = 0;
    int32_t *d_rowptr = nullptr, *d_col = nullptr;
    float* d_val = nullptr;
    int32_t *d_t_rowptr = nullptr, *d_t_col = nullptr;     // transpose (cols x rows), for the input gradients
    float* d_t_val = nullptr;
};

namespace {

constexpr int kBT = 256;

// Y[r][j] (+)= sum_p val_p * X[col_p][j],  j < width (flat [b*c] columns); one thread per (r, j), CSR order
__global__ void csr_spmm_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const float* __restrict__ val,
                                const float* __restrict__ X, float* __restrict__ Y, int rows, int width, int accumulate) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)rows * width) return;
    const int r = (int)(idx / width), j = (int)(idx % width);
    float acc = 0.f;
    for (int p = rowptr[r]; p < rowptr[r + 1]; ++p) acc = fmaf(val[p], X[(size_t)col[p] * width + j], acc);
    Y[idx] = accumulate ? Y[idx] + acc : acc;
}

// Z[m][co] (+)= sum_ci U[m][ci] * W[ci][co]
__global__ void rows_times_w_kernel(const float* __restrict__ U, const float* __restrict__ W, float* __restrict__ Z, long long M,
                                    int cin, int cout, int accumulate) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * cout) return;
    const long long m = idx / cout;
    const int co = (int)(idx % cout);
    float acc = 0.f;
    for (int ci = 0; ci < cin; ++ci) acc = fmaf(U[m * cin + ci], W[ci * cout + co], acc);
    Z[idx] = accumulate ? Z[idx] + acc : acc;
}

// dU[m][ci] = sum_co G[m][co] * W[ci][co]
__global__ void rows_times_wt_kernel(const float* __restrict__ G, const float* __restrict__ W, float* __restrict__ dU, long long M,
                                     int cin, int cout) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= M * cin) return;
    const long long m = idx / cin;
    const int ci = (int)(idx % cin);
    float acc = 0.f;
    for (int co = 0; co < cout; ++co) acc = fmaf(G[m * cout + co], W[ci * cout + co], acc);
    dU[idx] = acc;
}

// dW[ci][co] += sum_m U[m][ci] * G[m][co]; one block per (ci, co), strided partial sums + fixed shared-memory tree
__global__ void __launch_bounds__(kBT) outer_reduce_kernel(const float* __restrict__ U, const float* __restrict__ G, float* __restrict__ dW,
                                                          long long M, int cin, int cout) {
    __shared__ float red[kBT];
    const int ci = blockIdx.x / cout, co = blockIdx.x % cout;
    float acc = 0.f;
    for (long long m = threadIdx.x; m < M; m += kBT) acc = fmaf(U[m * cin + ci], G[m * cout + co], acc);
    red[threadIdx.x] = acc;
    __syncthreads();
    for (int s = kBT / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) dW[ci * cout + co] += red[0];
}

// The same product for the common small widths, coalesced and with every row read once: a thread keeps an 8 x 8 tile of dW in
// registers, walks rows m = global thread, + grid threads, ... (its 8 U and 8 G values are contiguous: two 32-byte loads), the
// block folds its threads' tiles in a fixed order (shuffle tree, then warps in order) into partial[blockIdx.x][tile]; blockIdx.y
// selects the tile of (ci, co).  outer_fold_kernel adds the blocks' partials in block order.  Deterministic.
constexpr int kOT = 8;
constexpr int kOuterBlocks = 296;
constexpr int kOuterTilesMax = 16;         // widths up to 32 x 32
__global__ void __launch_bounds__(kBT) outer_tile_kernel(const float* __restrict__ U, const float* __restrict__ G, float* __restrict__ partial,
                                                        long long M, int cin, int cout) {
    __shared__ float red[kBT / 32][kOT * kOT];
    const int tiles_co = (cout + kOT - 1) / kOT;
    const int ci0 = (blockIdx.y / tiles_co) * kOT, co0 = (blockIdx.y % tiles_co) * kOT;
    float acc[kOT][kOT];
#pragma unroll
    for (int i = 0; i < kOT; ++i)
#pragma unroll
        for (int j = 0; j < kOT; ++j) acc[i][j] = 0.f;
    const long long stride = (long long)gridDim.x * kBT;
    for (long long m = (long long)blockIdx.x * kBT + threadIdx.x; m < M; m += stride) {
        float u[kOT], g[kOT];
#pragma unroll
        for (int i = 0; i < kOT; ++i) u[i] = ci0 + i < cin ? U[m * cin + ci0 + i] : 0.f;
#pragma unroll
        for (int j = 0; j < kOT; ++j) g[j] = co0 + j < cout ? G[m * cout + co0 + j] : 0.f;
#pragma unroll
        for (int i = 0; i < kOT; ++i)
#pragma unroll
            for (int j = 0; j < kOT; ++j) acc[i][j] = fmaf(u[i], g[j], acc[i][j]);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < kOT; ++i)
#pragma unroll
        for (int j = 0; j < kOT; ++j) {
            float v = acc[i][j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red[warp][i * kOT + j] = v;
        }
    __syncthreads();
    if (threadIdx.x < kOT * kOT) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < kBT / 32; ++w) v += red[w][threadIdx.x];
        partial[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (kOT * kOT) + threadIdx.x] = v;
    }
}

__global__ void outer_fold_kernel(const float* __restrict__ partial, int n_blocks, float* __restrict__ dW, int cin, int cout) {
    const int tiles_co = (cout + kOT - 1) / kOT;
    const int tile = blockIdx.x, e = threadIdx.x;          // one block of 64 threads per tile
    const int ci = (tile / tiles_co) * kOT + e / kOT, co = (tile % tiles_co) * kOT + e % kOT;
    if (ci >= cin || co >= cout) return;
    float v = 0.f;
    for (int b = 0; b < n_blocks; ++b) v += partial[((size_t)tile * n_blocks + b) * (kOT * kOT) + e];
    dW[ci * cout + co] += v;
}

// ---- fused layer kernels (widths 1 / 8 / 16): one launch per simplex level instead of spmm + product (+ accumulate) per operator ----
// The operators that write (forward) / read (input gradient) one level, at most three.
struct BunchOps {
    int n;
    const int32_t* rowptr[3];
    const int32_t* col[3];
    const float* val[3];
    const float* X[3];                  // forward: state of the operator's input level [cols][b][CI]; backward: G of its output level [rows][b][CO]
    const float* W[3];                  // [CI][CO]
};

// u[0..C) += v * x[0..C): 128-bit loads when the row has them (C = 8 / 16: rows are 32 / 64 bytes, aligned)
template <int C>
__device__ __forceinline__ void axpy_row(float (&u)[C], float v, const float* __restrict__ x) {
    if (C % 4 == 0) {
#pragma unroll
        for (int q = 0; q < C / 4; ++q) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(x) + q);
            u[4 * q + 0] = fmaf(v, w.x, u[4 * q + 0]);
            u[4 * q + 1] = fmaf(v, w.y, u[4 * q + 1]);
            u[4 * q + 2] = fmaf(v, w.z, u[4 * q + 2]);
            u[4 * q + 3] = fmaf(v, w.w, u[4 * q + 3]);
        }
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) u[i] = fmaf(v, __ldg(x + i), u[i]);
    }
}
template <int C>
__device__ __forceinline__ void store_row(float* __restrict__ dst, const float (&z)[C]) {
    if (C % 4 == 0) {
#pragma unroll
        for (int q = 0; q < C / 4; ++q) reinterpret_cast<float4*>(dst)[q] = make_float4(z[4 * q], z[4 * q + 1], z[4 * q + 2], z[4 * q + 3]);
    } else {
#pragma unroll
        for (int i = 0; i < C; ++i) dst[i] = z[i];
    }
}

// forward of one level: Z[r][t][:] = relu( sum_k (sum_p val_p X_k[col_p][t][:]) W_k ); one thread per (r, t)
template <int CI, int CO>
__global__ void __launch_bounds__(kBT) bunch_level_fwd_kernel(const BunchOps o, float* __restrict__ Z, int rows, int b) {
    const long long idx = (long long)blockIdx.x * kBT + threadIdx.x;
    if (idx >= (long long)rows * b) return;
    const int r = (int)(idx / b), t = (int)(idx % b);
    float z[CO];
#pragma unroll
    for (int j = 0; j < CO; ++j) z[j] = 0.f;
    for (int k = 0; k < o.n; ++k) {
        float u[CI];
#pragma unroll
        for (int i = 0; i < CI; ++i) u[i] = 0.f;
        const int p1 = o.rowptr[k][r + 1];
        for (int p = o.rowptr[k][r]; p < p1; ++p) {
            axpy_row<CI>(u, o.val[k][p], o.X[k] + ((size_t)o.col[k][p] * b + t) * CI);
        }
        const float* W = o.W[k];
#pragma unroll
        for (int j = 0; j < CO; ++j) {
            float acc = 0.f;
#pragma unroll
            for (int i = 0; i < CI; ++i) acc = fmaf(u[i], W[i * CO + j], acc);
            z[j] += acc;
        }
    }
#pragma unroll
    for (int j = 0; j < CO; ++j) z[j] = fmaxf(z[j], 0.f);
    store_row<CO>(Z + (size_t)idx * CO, z);
}

// input gradient of one level: dX[c][t][:] = sum_k (sum_p val_p G_k[row_p][t][:]) W_k^T over the transposed operators; one thread per (c, t)
template <int CI, int CO>
__global__ void __launch_bounds__(kBT) bunch_level_bwd_kernel(const BunchOps o, float* __restrict__ dX, int cols, int b) {
    const long long idx = (long long)blockIdx.x * kBT + threadIdx.x;
    if (idx >= (long long)cols * b) return;
    const int c = (int)(idx / b), t = (int)(idx % b);
    float dx[CI];
#pragma unroll
    for (int i = 0; i < CI; ++i) dx[i] = 0.f;
    for (int k = 0; k < o.n; ++k) {
        float v[CO];
#pragma unroll
        for (int j = 0; j < CO; ++j) v[j] = 0.f;
        const int p1 = o.rowptr[k][c + 1];
        for (int p = o.rowptr[k][c]; p < p1; ++p) {
            axpy_row<CO>(v, o.val[k][p], o.X[k] + ((size_t)o.col[k][p] * b + t) * CO);
        }
        const float* W = o.W[k];
#pragma unroll
        for (int i = 0; i < CI; ++i) {
            float acc = 0.f;
#pragma unroll
            for (int j = 0; j < CO; ++j) acc = fmaf(v[j], W[i * CO + j], acc);
            dx[i] += acc;
        }
    }
    store_row<CI>(dX + (size_t)idx * CI, dx);
}

// weight gradient of one operator with U = S X computed on the fly (outer_tile_kernel without the U round trip)
__global__ void __launch_bounds__(kBT) outer_tile_spmm_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                             const float* __restrict__ val, const float* __restrict__ X,
                                                             const float* __restrict__ G, float* __restrict__ partial, int rows, int b, int cin,
                                                             int cout) {
    __shared__ float red[kBT / 32][kOT * kOT];
    const int tiles_co = (cout + kOT - 1) / kOT;
    const int ci0 = (blockIdx.y / tiles_co) * kOT, co0 = (blockIdx.y % tiles_co) * kOT;
    float acc[kOT][kOT];
#pragma unroll
    for (int i = 0; i < kOT; ++i)
#pragma unroll
        for (int j = 0; j < kOT; ++j) acc[i][j] = 0.f;
    const long long M = (long long)rows * b, stride = (long long)gridDim.x * kBT;
    for (long long m = (long long)blockIdx.x * kBT + threadIdx.x; m < M; m += stride) {
        const int r = (int)(m / b), t = (int)(m % b);
        float u[kOT], g[kOT];
#pragma unroll
        for (int i = 0; i < kOT; ++i) u[i] = 0.f;
        const int p1 = rowptr[r + 1];
        for (int p = rowptr[r]; p < p1; ++p) {
            const float v = val[p];
            const float* x = X + ((size_t)col[p] * b + t) * cin + ci0;
            if (cin % kOT == 0) {                          // (uniform) the tile is a whole, aligned 32-byte piece of the row
                axpy_row<kOT>(u, v, x);
            } else {
#pragma unroll
                for (int i = 0; i < kOT; ++i)
                    if (ci0 + i < cin) u[i] = fmaf(v, x[i], u[i]);
            }
        }
        if (cout % kOT == 0) {
#pragma unroll
            for (int q = 0; q < kOT / 4; ++q) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(G + m * cout + co0) + q);
                g[4 * q] = w.x; g[4 * q + 1] = w.y; g[4 * q + 2] = w.z; g[4 * q + 3] = w.w;
            }
        } else {
#pragma unroll
            for (int j = 0; j < kOT; ++j) g[j] = co0 + j < cout ? G[m * cout + co0 + j] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < kOT; ++i)
#pragma unroll
            for (int j = 0; j < kOT; ++j) acc[i][j] = fmaf(u[i], g[j], acc[i][j]);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < kOT; ++i)
#pragma unroll
        for (int j = 0; j < kOT; ++j) {
            float v = acc[i][j];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red[warp][i * kOT + j] = v;
        }
    __syncthreads();
    if (threadIdx.x < kOT * kOT) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < kBT / 32; ++w) v += red[w][threadIdx.x];
        partial[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * (kOT * kOT) + threadIdx.x] = v;
    }
}

__global__ void relu_kernel(float* __restrict__ Z, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) Z[i] = fmaxf(Z[i], 0.f);
}
// G = dX * relu'(z) expressed through h = relu(z): 1 where h > 0, else 0.  (jnp.maximum splits the tie z == 0 evenly, but an
// exact zero pre-activation only occurs at structurally zero rows, whose gradient never reaches a weight: SURVEY App. A.)
__global__ void relu_bwd_kernel(const float* __restrict__ dX, const float* __restrict__ h, float* __restrict__ G, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) G[i] = h[i] > 0.f ? dX[i] : 0.f;
}

// readout: one thread per trajectory.  COT (cotangent seed, scone_bunch_vjp_host): dlogit_j = cot_j - p_j * sum_k cot_k over all D
// slots, added to the node slot j reads (a padded slot reads node N - 1); partial = {sum_j cot_j * logp_j, 0}; tgt / mask unused.
template <bool COT>
__global__ void bunch_readout_kernel(const float* __restrict__ VL /* [N][b] */, const int32_t* __restrict__ nbrhoods,
                                     const int32_t* __restrict__ last_nodes, float* __restrict__ logprobs, const int32_t* __restrict__ tgt,
                                     const float* __restrict__ mask, float* __restrict__ dVL /* [N][b], pre-zeroed or NULL */,
                                     float* __restrict__ partial /* [b][2] */, int N, int D, int b, const float* __restrict__ cot /* [b][D] */) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= b) return;
    const int last = last_nodes[t];
    float mx = -3.4e38f;
    for (int j = 0; j < D; ++j) {
        int idx = nbrhoods[(size_t)last * D + j];
        if (idx < 0) idx += N;                                  // -1 -> node N-1 (negative indexing)
        mx = fmaxf(mx, VL[(size_t)idx * b + t]);
    }
    float se = 0.f;
    for (int j = 0; j < D; ++j) {
        int idx = nbrhoods[(size_t)last * D + j];
        if (idx < 0) idx += N;
        se += expf(VL[(size_t)idx * b + t] - mx);
    }
    const float lse = mx + logf(se);
    for (int j = 0; j < D; ++j) {
        int idx = nbrhoods[(size_t)last * D + j];
        if (idx < 0) idx += N;
        logprobs[(size_t)t * D + j] = VL[(size_t)idx * b + t] - lse;
    }
    if (dVL == nullptr) return;
    if (COT) {
        const float* c = cot + (size_t)t * D;
        float cs = 0.f, el = 0.f;
        for (int j = 0; j < D; ++j) cs += c[j];
        for (int j = 0; j < D; ++j) {
            int idx = nbrhoods[(size_t)last * D + j];
            if (idx < 0) idx += N;
            const float lp = VL[(size_t)idx * b + t] - lse;
            dVL[(size_t)idx * b + t] += c[j] - expf(lp) * cs;                          // same thread: sequential
            el = fmaf(c[j], lp, el);
        }
        partial[2 * t] = el;
        partial[2 * t + 1] = 0.f;
        return;
    }
    const float mk = mask[t];
    const int y = tgt[t];
    for (int j = 0; j < D; ++j) {
        int idx = nbrhoods[(size_t)last * D + j];
        if (idx < 0) idx += N;
        dVL[(size_t)idx * b + t] += mk * (expf(VL[(size_t)idx * b + t] - lse) - (j == y ? 1.f : 0.f));   // same thread: sequential
    }
    int yi = nbrhoods[(size_t)last * D + y];
    if (yi < 0) yi += N;
    partial[2 * t] = -mk * (VL[(size_t)yi * b + t] - lse);
    partial[2 * t + 1] = mk;
}
__global__ void bunch_readout_reduce_kernel(const float* __restrict__ partial, int b, float* __restrict__ nll, float* __restrict__ count) {
    if (threadIdx.x < 2) {
        float s = 0.f;
        for (int t = 0; t < b; ++t) s += partial[2 * t + threadIdx.x];
        float* dst = threadIdx.x == 0 ? nll : count;
        *dst += s;
    }
}

inline int nblk(long long n) { return (int)((n + kBT - 1) / kBT); }

template <typename T>
int up(T** dst, const T* src, size_t n) {
    SCONE_CUDA(cudaMalloc((void**)dst, (n ? n : 1) * sizeof(T)));
    if (n) SCONE_CUDA(cudaMemcpy(*dst, src, n * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

}  // namespace

extern "C" int scone_csr_create(int32_t rows, int32_t cols, const int32_t* rowptr, const int32_t* col, const float* val, scone_csr** out) {
    // rows / cols may be 0: a complex without triangles has F = 0, so S_21 is E x 0, S_12 is 0 x E and S_22 is 0 x 0
    SCONE_REQUIRE(out && rowptr && rows >= 0 && cols >= 0, "scone_csr_create: bad arguments");
    *out = nullptr;
    const int64_t nnz = rowptr[rows];
    SCONE_REQUIRE(nnz == 0 || (col && val), "scone_csr_create: NULL col/val");
    for (int64_t p = 0; p < nnz; ++p) SCONE_REQUIRE(col[p] >= 0 && col[p] < cols, "scone_csr_create: column %d out of range", col[p]);
    scone_csr* S = new scone_csr();
    S->rows = rows; S->cols = cols; S->nnz = nnz;
    // transpose (counting sort keeps rows ascending inside each column: deterministic order)
    std::vector<int32_t> tp(cols + 1, 0), tc(nnz);
    std::vector<float> tv(nnz);
    for (int64_t p = 0; p < nnz; ++p) tp[col[p] + 1]++;
    for (int32_t c = 0; c < cols; ++c) tp[c + 1] += tp[c];
    std::vector<int32_t> fill(tp.begin(), tp.end() - 1);
    for (int32_t r = 0; r < rows; ++r)
        for (int32_t p = rowptr[r]; p < rowptr[r + 1]; ++p) {
            const int32_t q = fill[col[p]]++;
            tc[q] = r;
            tv[q] = val[p];
        }
    int rc = up(&S->d_rowptr, rowptr, (size_t)rows + 1) | up(&S->d_col, col, (size_t)nnz) | up(&S->d_val, val, (size_t)nnz) |
             up(&S->d_t_rowptr, tp.data(), (size_t)cols + 1) | up(&S->d_t_col, tc.data(), (size_t)nnz) | up(&S->d_t_val, tv.data(), (size_t)nnz);
    if (rc) { scone_csr_destroy(S); return rc; }
    *out = S;
    return 0;
}

extern "C" int scone_csr_destroy(scone_csr* S) {
    if (!S) return 0;
    cudaFree(S->d_rowptr); cudaFree(S->d_col); cudaFree(S->d_val);
    cudaFree(S->d_t_rowptr); cudaFree(S->d_t_col); cudaFree(S->d_t_val);
    delete S;
    return 0;
}

// term k: output level, input level (0 nodes, 1 edges, 2 triangles) — trajectory_experiments.py:184-192
static const int kOutLevel[7] = {0, 0, 1, 1, 1, 2, 2};
static const int kInLevel[7] = {0, 1, 0, 1, 2, 1, 2};

struct scone_bunch {
    const scone_csr* S[7];
    int32_t n[3];                             // N, E, F
    int32_t D = 0, L = 0, mb = 0;
    std::vector<int32_t> width;               // width[i] = channels of the state entering layer i; width[L] = 1
    std::vector<int64_t> w_off;               // 7 per layer
    int64_t n_params = 0;
    float *d_w = nullptr, *d_m = nullptr, *d_v = nullptr, *d_grad = nullptr;
    int32_t* d_nbr = nullptr;
    int32_t* d_rank_identity = nullptr;       // flows arrive in the caller's edge order; this path keeps it
    std::vector<float*> act[3];               // act[level][i], i = 0..L : state entering layer i (i = L: final output)
    float *d_U = nullptr, *d_dU = nullptr;    // [max rows][mb][cmax]
    float* d_G[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};   // dL/dZ ping-pong per level
    float* d_dX[3] = {nullptr, nullptr, nullptr};
    float *d_logp = nullptr, *d_partial = nullptr;
    float* d_outer = nullptr;                 // [tiles][blocks][64] partial weight-gradient tiles
    int32_t *d_ptr = nullptr, *d_edge = nullptr, *d_last = nullptr, *d_tgt = nullptr;
    float *d_val = nullptr, *d_mask = nullptr, *d_logp_all = nullptr, *d_cot = nullptr;
    int64_t cap_B = 0, cap_nnz = 0;
};

extern "C" int scone_bunch_destroy(scone_bunch* m) {
    if (!m) return 0;
    cudaFree(m->d_w); cudaFree(m->d_m); cudaFree(m->d_v); cudaFree(m->d_grad); cudaFree(m->d_nbr);
    for (int lv = 0; lv < 3; ++lv) {
        for (float* p : m->act[lv]) cudaFree(p);
        cudaFree(m->d_G[0][lv]); cudaFree(m->d_G[1][lv]); cudaFree(m->d_dX[lv]);
    }
    cudaFree(m->d_U); cudaFree(m->d_dU); cudaFree(m->d_logp); cudaFree(m->d_partial); cudaFree(m->d_outer);
    cudaFree(m->d_ptr); cudaFree(m->d_edge); cudaFree(m->d_last); cudaFree(m->d_tgt); cudaFree(m->d_val); cudaFree(m->d_mask);
    cudaFree(m->d_logp_all); cudaFree(m->d_cot);
    delete m;
    return 0;
}

extern "C" int scone_bunch_create(const scone_csr* const* S7, int32_t N, int32_t E, int32_t F, int32_t D, const int32_t* nbrhoods,
                                  int32_t n_hidden, const int32_t* hidden, int32_t micro_batch, scone_bunch** out) {
    SCONE_REQUIRE(out && S7 && nbrhoods && hidden && n_hidden >= 1 && micro_batch >= 1 && D >= 1, "scone_bunch_create: bad arguments");
    *out = nullptr;
    for (int i = 0; i < n_hidden; ++i) SCONE_REQUIRE(hidden[i] >= 1, "scone_bunch_create: hidden width %d of layer %d is below 1", hidden[i], i);
    // the readout gathers node rows through this table: an entry outside [-1, N) would read outside the node state
    for (int64_t p = 0; p < (int64_t)N * D; ++p)
        SCONE_REQUIRE(nbrhoods[p] >= -1 && nbrhoods[p] < N, "scone_bunch_create: nbrhoods[%lld][%lld] = %d is outside [-1, %d)",
                      (long long)(p / D), (long long)(p % D), nbrhoods[p], N);
    const int32_t rows_of[3] = {N, E, F};
    for (int k = 0; k < 7; ++k) {
        SCONE_REQUIRE(S7[k] != nullptr, "scone_bunch_create: shift %d is NULL", k);
        SCONE_REQUIRE(S7[k]->rows == rows_of[kOutLevel[k]] && S7[k]->cols == rows_of[kInLevel[k]],
                      "scone_bunch_create: shift %d has shape %d x %d", k, S7[k]->rows, S7[k]->cols);
    }
    scone_bunch* m = new scone_bunch();
    for (int k = 0; k < 7; ++k) m->S[k] = S7[k];
    m->n[0] = N; m->n[1] = E; m->n[2] = F;
    m->D = D; m->mb = micro_batch;
    m->L = n_hidden + 1;                       // generate_weights appends one more group of 7 mapping to out_channels = 1
    m->width.push_back(1);
    for (int i = 0; i < n_hidden; ++i) m->width.push_back(hidden[i]);
    m->width.push_back(1);
    int64_t off = 0;
    int cmax = 1;
    for (int i = 0; i < m->L; ++i) {
        for (int k = 0; k < 7; ++k) { m->w_off.push_back(off); off += (int64_t)m->width[i] * m->width[i + 1]; }
        cmax = std::max(cmax, std::max(m->width[i], m->width[i + 1]));
    }
    m->n_params = off;
    int rc = 0;
    auto alloc = [&](void** p, size_t bytes) {
        if (!rc && cudaMalloc(p, bytes ? bytes : 4) != cudaSuccess) { scone_set_error("scone_bunch_create: cudaMalloc(%zu) failed", bytes); rc = 1; }
    };
    const size_t mb = micro_batch, rmax = std::max(N, std::max(E, F));
    alloc((void**)&m->d_w, off * 4); alloc((void**)&m->d_m, off * 4); alloc((void**)&m->d_v, off * 4); alloc((void**)&m->d_grad, (off + 2) * 4);
    alloc((void**)&m->d_nbr, (size_t)N * D * 4);
    for (int lv = 0; lv < 3; ++lv) {
        m->act[lv].assign(m->L + 1, nullptr);
        for (int i = 0; i <= m->L; ++i) alloc((void**)&m->act[lv][i], (size_t)rows_of[lv] * mb * m->width[i] * 4);
        for (int q = 0; q < 2; ++q) alloc((void**)&m->d_G[q][lv], (size_t)rows_of[lv] * mb * cmax * 4);
        alloc((void**)&m->d_dX[lv], (size_t)rows_of[lv] * mb * cmax * 4);
    }
    alloc((void**)&m->d_U, rmax * mb * cmax * 4); alloc((void**)&m->d_dU, rmax * mb * cmax * 4);
    alloc((void**)&m->d_outer, (size_t)kOuterTilesMax * kOuterBlocks * kOT * kOT * 4);
    alloc((void**)&m->d_logp, mb * D * 4); alloc((void**)&m->d_partial, mb * 2 * 4);
    if (!rc) {
        cudaMemcpy(m->d_nbr, nbrhoods, (size_t)N * D * 4, cudaMemcpyHostToDevice);
        cudaMemset(m->d_w, 0, off * 4); cudaMemset(m->d_m, 0, off * 4); cudaMemset(m->d_v, 0, off * 4); cudaMemset(m->d_grad, 0, (off + 2) * 4);
    } else {
        scone_bunch_destroy(m);
        return rc;
    }
    *out = m;
    return 0;
}

extern "C" int64_t scone_bunch_num_params(const scone_bunch* m) { return m ? m->n_params : -1; }
extern "C" float* scone_bunch_grads_dev(scone_bunch* m) { return m ? m->d_grad : nullptr; }
extern "C" int scone_bunch_set_weights(scone_bunch* m, const float* w, int32_t reset_adam) {
    SCONE_REQUIRE(m && w, "scone_bunch_set_weights: NULL argument");
    SCONE_CUDA(cudaMemcpy(m->d_w, w, m->n_params * 4, cudaMemcpyHostToDevice));
    if (reset_adam) { SCONE_CUDA(cudaMemset(m->d_m, 0, m->n_params * 4)); SCONE_CUDA(cudaMemset(m->d_v, 0, m->n_params * 4)); }
    return 0;
}
extern "C" int scone_bunch_get_weights(const scone_bunch* m, float* w) {
    SCONE_REQUIRE(m && w, "scone_bunch_get_weights: NULL argument");
    SCONE_CUDA(cudaMemcpy(w, m->d_w, m->n_params * 4, cudaMemcpyDeviceToHost));
    return 0;
}

namespace {

__global__ void flows_to_edges_kernel(const int32_t* __restrict__ ptr, const int32_t* __restrict__ edge, const float* __restrict__ val,
                                      float* __restrict__ H0, int E, int b) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= b) return;
    for (int p = ptr[t]; p < ptr[t + 1]; ++p)
        if (edge[p] >= 0 && edge[p] < E) H0[(size_t)edge[p] * b + t] = val[p];
}

int ensure_staging(scone_bunch* m, int64_t B, int64_t nnz) {
    if (B > m->cap_B) {
        cudaFree(m->d_ptr); cudaFree(m->d_last); cudaFree(m->d_tgt); cudaFree(m->d_mask); cudaFree(m->d_logp_all); cudaFree(m->d_cot);
        const int64_t cap = B + B / 4 + 16;
        SCONE_CUDA(cudaMalloc((void**)&m->d_ptr, (cap + 1) * 4)); SCONE_CUDA(cudaMalloc((void**)&m->d_last, cap * 4));
        SCONE_CUDA(cudaMalloc((void**)&m->d_tgt, cap * 4)); SCONE_CUDA(cudaMalloc((void**)&m->d_mask, cap * 4));
        SCONE_CUDA(cudaMalloc((void**)&m->d_logp_all, cap * (size_t)m->D * 4));
        SCONE_CUDA(cudaMalloc((void**)&m->d_cot, cap * (size_t)m->D * 4));
        m->cap_B = cap;
    }
    if (nnz > m->cap_nnz) {
        cudaFree(m->d_edge); cudaFree(m->d_val);
        const int64_t cap = nnz + nnz / 4 + 16;
        SCONE_CUDA(cudaMalloc((void**)&m->d_edge, cap * 4)); SCONE_CUDA(cudaMalloc((void**)&m->d_val, cap * 4));
        m->cap_nnz = cap;
    }
    return 0;
}

// The readout uses both arrays as device indices: every last node must be a node, every target a slot of the neighbour table.
int check_readout_indices(const char* fn, const scone_bunch* m, int32_t B, const int32_t* last, const int32_t* tgt) {
    for (int32_t t = 0; t < B; ++t) {
        SCONE_REQUIRE(last[t] >= 0 && last[t] < m->n[0], "%s: last_nodes[%d] = %d is outside [0, %d)", fn, t, last[t], m->n[0]);
        if (tgt) SCONE_REQUIRE(tgt[t] >= 0 && tgt[t] < m->D, "%s: target_idx[%d] = %d is outside [0, %d)", fn, t, tgt[t], m->D);
    }
    return 0;
}

bool fused_width(int c) { return c == 1 || c == 8 || c == 16; }

template <bool FWD>
int launch_level(const BunchOps& o, float* out, int rows, int b, int cin, int cout, cudaStream_t st) {
    if (rows == 0) return 0;                                  // an empty level (F = 0): nothing to write
    const unsigned grid = (unsigned)(((long long)rows * b + kBT - 1) / kBT);
#define SCONE_BUNCH_CASE(CI, CO)                                                                          \
    if (cin == CI && cout == CO) {                                                                       \
        if (FWD) bunch_level_fwd_kernel<CI, CO><<<grid, kBT, 0, st>>>(o, out, rows, b);                   \
        else bunch_level_bwd_kernel<CI, CO><<<grid, kBT, 0, st>>>(o, out, rows, b);                       \
        SCONE_LAUNCHED();                                                                                \
        return 0;                                                                                        \
    }
    SCONE_BUNCH_CASE(1, 8) SCONE_BUNCH_CASE(1, 16) SCONE_BUNCH_CASE(8, 8) SCONE_BUNCH_CASE(16, 16) SCONE_BUNCH_CASE(8, 16)
    SCONE_BUNCH_CASE(16, 8) SCONE_BUNCH_CASE(8, 1) SCONE_BUNCH_CASE(16, 1) SCONE_BUNCH_CASE(1, 1)
#undef SCONE_BUNCH_CASE
    scone_set_error("scone_bunch: no fused layer kernel for widths %d -> %d", cin, cout);
    return 1;
}

// forward of one micro-batch; states kept in m->act
int bunch_forward_mb(scone_bunch* m, int b, const int32_t* ptr, const int32_t* edge, const float* val, cudaStream_t st) {
    for (int lv = 0; lv < 3; ++lv) SCONE_CUDA(cudaMemsetAsync(m->act[lv][0], 0, (size_t)m->n[lv] * b * 4, st));   // V_0 = T_0 = 0
    flows_to_edges_kernel<<<nblk(b), kBT, 0, st>>>(ptr, edge, val, m->act[1][0], m->n[1], b);
    SCONE_LAUNCHED();
    for (int i = 0; i < m->L; ++i) {
        const int cin = m->width[i], cout = m->width[i + 1];
        if (fused_width(cin) && fused_width(cout)) {       // one launch per level: gather, products, relu
            for (int lv = 0; lv < 3; ++lv) {
                BunchOps o{};
                for (int k = 0; k < 7; ++k)
                    if (kOutLevel[k] == lv) {
                        const scone_csr* S = m->S[k];
                        o.rowptr[o.n] = S->d_rowptr; o.col[o.n] = S->d_col; o.val[o.n] = S->d_val;
                        o.X[o.n] = m->act[kInLevel[k]][i]; o.W[o.n] = m->d_w + m->w_off[7 * i + k];
                        ++o.n;
                    }
                if (launch_level<true>(o, m->act[lv][i + 1], m->n[lv], b, cin, cout, st)) return 1;
            }
            continue;
        }
        bool first[3] = {true, true, true};
        for (int k = 0; k < 7; ++k) {
            const scone_csr* S = m->S[k];
            if (S->rows == 0) continue;                       // writes an empty level (F = 0)
            const int ol = kOutLevel[k], il = kInLevel[k];
            const int wdt = b * cin;
            csr_spmm_kernel<<<nblk((long long)S->rows * wdt), kBT, 0, st>>>(S->d_rowptr, S->d_col, S->d_val, m->act[il][i], m->d_U, S->rows,
                                                                           wdt, 0);
            SCONE_LAUNCHED();
            const long long M = (long long)S->rows * b;
            rows_times_w_kernel<<<nblk(M * cout), kBT, 0, st>>>(m->d_U, m->d_w + m->w_off[7 * i + k], m->act[ol][i + 1], M, cin, cout,
                                                              first[ol] ? 0 : 1);
            SCONE_LAUNCHED();
            first[ol] = false;
        }
        for (int lv = 0; lv < 3; ++lv) {
            const long long n = (long long)m->n[lv] * b * cout;
            if (n == 0) continue;
            relu_kernel<<<nblk(n), kBT, 0, st>>>(m->act[lv][i + 1], n);
            SCONE_LAUNCHED();
        }
    }
    return 0;
}

}  // namespace

extern "C" int scone_bunch_forward_host(scone_bunch* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                        const int32_t* last, float* logprobs_out, void* stream) {
    SCONE_REQUIRE(m && ptr && last && logprobs_out && B >= 0, "scone_bunch_forward_host: bad arguments");
    if (check_readout_indices("scone_bunch_forward_host", m, B, last, nullptr)) return 2;
    if (B == 0) return 0;
    cudaStream_t st = as_stream(stream);
    const int64_t nnz = ptr[B];
    if (ensure_staging(m, B, nnz)) return 1;
    SCONE_CUDA(cudaMemcpyAsync(m->d_ptr, ptr, (B + 1) * 4, cudaMemcpyHostToDevice, st));
    if (nnz) {
        SCONE_CUDA(cudaMemcpyAsync(m->d_edge, edge, nnz * 4, cudaMemcpyHostToDevice, st));
        SCONE_CUDA(cudaMemcpyAsync(m->d_val, val, nnz * 4, cudaMemcpyHostToDevice, st));
    }
    SCONE_CUDA(cudaMemcpyAsync(m->d_last, last, B * 4, cudaMemcpyHostToDevice, st));
    for (int32_t off = 0; off < B; off += m->mb) {
        const int b = B - off < m->mb ? B - off : m->mb;
        if (bunch_forward_mb(m, b, m->d_ptr + off, m->d_edge, m->d_val, st)) return 1;
        bunch_readout_kernel<false><<<nblk(b), kBT, 0, st>>>(m->act[0][m->L], m->d_nbr, m->d_last + off, m->d_logp_all + (size_t)off * m->D,
                                                            nullptr, nullptr, nullptr, nullptr, m->n[0], m->D, b, nullptr);
        SCONE_LAUNCHED();
    }
    SCONE_CUDA(cudaMemcpyAsync(logprobs_out, m->d_logp_all, (size_t)B * m->D * 4, cudaMemcpyDeviceToHost, st));
    SCONE_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// loss + gradient (tgt / mask) or VJP (cot [B][D], count_add) over B trajectories from HOST buffers
static int bunch_grad_host(scone_bunch* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                           const int32_t* tgt, const float* mask, const float* cot, float count_add, int32_t zero_first, cudaStream_t st) {
    if (zero_first) SCONE_CUDA(cudaMemsetAsync(m->d_grad, 0, (m->n_params + 2) * 4, st));
    if (cot && count_add != 0.f && scone_add_scalar_launch(m->d_grad + m->n_params + 1, count_add, st)) return 1;
    if (B == 0) return 0;                                     // nothing to add: the buffer is cleared (zero_first) or left as it is
    const int64_t nnz = ptr[B];
    if (ensure_staging(m, B, nnz)) return 1;
    SCONE_CUDA(cudaMemcpyAsync(m->d_ptr, ptr, (B + 1) * 4, cudaMemcpyHostToDevice, st));
    if (nnz) {
        SCONE_CUDA(cudaMemcpyAsync(m->d_edge, edge, nnz * 4, cudaMemcpyHostToDevice, st));
        SCONE_CUDA(cudaMemcpyAsync(m->d_val, val, nnz * 4, cudaMemcpyHostToDevice, st));
    }
    SCONE_CUDA(cudaMemcpyAsync(m->d_last, last, B * 4, cudaMemcpyHostToDevice, st));
    if (cot) {
        SCONE_CUDA(cudaMemcpyAsync(m->d_cot, cot, (size_t)B * m->D * 4, cudaMemcpyHostToDevice, st));
    } else {
        SCONE_CUDA(cudaMemcpyAsync(m->d_tgt, tgt, B * 4, cudaMemcpyHostToDevice, st));
        SCONE_CUDA(cudaMemcpyAsync(m->d_mask, mask, B * 4, cudaMemcpyHostToDevice, st));
    }
    const int L = m->L;
    for (int32_t off = 0; off < B; off += m->mb) {
        const int b = B - off < m->mb ? B - off : m->mb;
        if (bunch_forward_mb(m, b, m->d_ptr + off, m->d_edge, m->d_val, st)) return 1;
        // dL/d(output of the last layer): only the node level is read by the readout
        int cur = 0;
        for (int lv = 0; lv < 3; ++lv) SCONE_CUDA(cudaMemsetAsync(m->d_dX[lv], 0, (size_t)m->n[lv] * b * m->width[L] * 4, st));
        if (cot)
            bunch_readout_kernel<true><<<nblk(b), kBT, 0, st>>>(m->act[0][L], m->d_nbr, m->d_last + off, m->d_logp, nullptr, nullptr, m->d_dX[0],
                                                               m->d_partial, m->n[0], m->D, b, m->d_cot + (size_t)off * m->D);
        else
            bunch_readout_kernel<false><<<nblk(b), kBT, 0, st>>>(m->act[0][L], m->d_nbr, m->d_last + off, m->d_logp, m->d_tgt + off,
                                                                m->d_mask + off, m->d_dX[0], m->d_partial, m->n[0], m->D, b, nullptr);
        SCONE_LAUNCHED();
        bunch_readout_reduce_kernel<<<1, 32, 0, st>>>(m->d_partial, b, m->d_grad + m->n_params, m->d_grad + m->n_params + 1);
        SCONE_LAUNCHED();
        for (int i = L - 1; i >= 0; --i) {
            const int cin = m->width[i], cout = m->width[i + 1];
            // G = dX * relu'(output of layer i)
            for (int lv = 0; lv < 3; ++lv) {
                const long long n = (long long)m->n[lv] * b * cout;
                if (n == 0) continue;
                relu_bwd_kernel<<<nblk(n), kBT, 0, st>>>(m->d_dX[lv], m->act[lv][i + 1], m->d_G[cur][lv], n);
                SCONE_LAUNCHED();
            }
            if (fused_width(cin) && fused_width(cout)) {
                // weight gradients: U = S X on the fly; input gradients: one launch per level over the transposed operators
                for (int k = 0; k < 7; ++k) {
                    const scone_csr* S = m->S[k];
                    const int ol = kOutLevel[k], il = kInLevel[k];
                    const long long M = (long long)S->rows * b;
                    if (M == 0) continue;                     // an operator into an empty level: its weight gradient stays 0
                    const int tiles = ((cin + kOT - 1) / kOT) * ((cout + kOT - 1) / kOT);
                    const int nb = (int)std::min<long long>(kOuterBlocks, (M + kBT - 1) / kBT);
                    outer_tile_spmm_kernel<<<dim3(nb, tiles), kBT, 0, st>>>(S->d_rowptr, S->d_col, S->d_val, m->act[il][i], m->d_G[cur][ol],
                                                                            m->d_outer, S->rows, b, cin, cout);
                    SCONE_LAUNCHED();
                    outer_fold_kernel<<<tiles, kOT * kOT, 0, st>>>(m->d_outer, nb, m->d_grad + m->w_off[7 * i + k], cin, cout);
                    SCONE_LAUNCHED();
                }
                if (i > 0)
                    for (int lv = 0; lv < 3; ++lv) {
                        BunchOps o{};
                        for (int k = 0; k < 7; ++k)
                            if (kInLevel[k] == lv) {
                                const scone_csr* S = m->S[k];
                                o.rowptr[o.n] = S->d_t_rowptr; o.col[o.n] = S->d_t_col; o.val[o.n] = S->d_t_val;
                                o.X[o.n] = m->d_G[cur][kOutLevel[k]]; o.W[o.n] = m->d_w + m->w_off[7 * i + k];
                                ++o.n;
                            }
                        if (launch_level<false>(o, m->d_dX[lv], m->n[lv], b, cin, cout, st)) return 1;
                    }
                cur ^= 1;
                continue;
            }
            if (i > 0)
                for (int lv = 0; lv < 3; ++lv) SCONE_CUDA(cudaMemsetAsync(m->d_dX[lv], 0, (size_t)m->n[lv] * b * cin * 4, st));
            for (int k = 0; k < 7; ++k) {
                const scone_csr* S = m->S[k];
                if (S->rows == 0) continue;                   // an operator into an empty level: no weight or input gradient
                const int ol = kOutLevel[k], il = kInLevel[k];
                const int wdt = b * cin;
                const long long M = (long long)S->rows * b;
                csr_spmm_kernel<<<nblk((long long)S->rows * wdt), kBT, 0, st>>>(S->d_rowptr, S->d_col, S->d_val, m->act[il][i], m->d_U, S->rows,
                                                                               wdt, 0);
                SCONE_LAUNCHED();
                {
                    // dW_k += U^T G over the M = rows x b stacked rows
                    const int tiles = ((cin + kOT - 1) / kOT) * ((cout + kOT - 1) / kOT);
                    const int nb = (int)std::min<long long>(kOuterBlocks, (M + kBT - 1) / kBT);
                    if (tiles <= kOuterTilesMax) {
                        outer_tile_kernel<<<dim3(nb, tiles), kBT, 0, st>>>(m->d_U, m->d_G[cur][ol], m->d_outer, M, cin, cout);
                        SCONE_LAUNCHED();
                        outer_fold_kernel<<<tiles, kOT * kOT, 0, st>>>(m->d_outer, nb, m->d_grad + m->w_off[7 * i + k], cin, cout);
                        SCONE_LAUNCHED();
                    } else {
                        outer_reduce_kernel<<<cin * cout, kBT, 0, st>>>(m->d_U, m->d_G[cur][ol], m->d_grad + m->w_off[7 * i + k], M, cin, cout);
                        SCONE_LAUNCHED();
                    }
                }
                if (i > 0 && S->cols > 0) {
                    rows_times_wt_kernel<<<nblk(M * cin), kBT, 0, st>>>(m->d_G[cur][ol], m->d_w + m->w_off[7 * i + k], m->d_dU, M, cin, cout);
                    SCONE_LAUNCHED();
                    csr_spmm_kernel<<<nblk((long long)S->cols * wdt), kBT, 0, st>>>(S->d_t_rowptr, S->d_t_col, S->d_t_val, m->d_dU,
                                                                                   m->d_dX[il], S->cols, wdt, 1);
                    SCONE_LAUNCHED();
                }
            }
            cur ^= 1;
        }
    }
    return 0;
}

extern "C" int scone_bunch_loss_grad_host(scone_bunch* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                          const int32_t* last, const int32_t* tgt, const float* mask, int32_t zero_first, void* stream) {
    SCONE_REQUIRE(m && ptr && last && tgt && mask && B >= 0, "scone_bunch_loss_grad_host: bad arguments");
    if (check_readout_indices("scone_bunch_loss_grad_host", m, B, last, tgt)) return 2;
    return bunch_grad_host(m, B, ptr, edge, val, last, tgt, mask, nullptr, 0.f, zero_first, as_stream(stream));
}

extern "C" int scone_bunch_vjp_host(scone_bunch* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                                    const float* cot, float count_add, int32_t zero_first, void* stream) {
    SCONE_REQUIRE(m && ptr && last && B >= 0, "scone_bunch_vjp_host: bad arguments");
    SCONE_REQUIRE(cot || B == 0, "scone_bunch_vjp_host: cot is NULL");
    if (check_readout_indices("scone_bunch_vjp_host", m, B, last, nullptr)) return 2;
    return bunch_grad_host(m, B, ptr, edge, val, last, nullptr, nullptr, cot, count_add, zero_first, as_stream(stream));
}

extern "C" int scone_bunch_read_grads(scone_bunch* m, float* out, void* stream) {
    SCONE_REQUIRE(m && out, "scone_bunch_read_grads: NULL argument");
    cudaStream_t st = as_stream(stream);
    SCONE_CUDA(cudaMemcpyAsync(out, m->d_grad, (m->n_params + 2) * 4, cudaMemcpyDeviceToHost, st));
    SCONE_CUDA(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int scone_bunch_adam_step(scone_bunch* m, int32_t step, float lr, float wd, void* stream) {
    SCONE_REQUIRE(m && step >= 0, "scone_bunch_adam_step: bad arguments");
    return scone_adam_launch(m->d_w, m->d_m, m->d_v, m->d_grad, m->n_params, step, lr, wd, stream);
}
