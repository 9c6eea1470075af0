// common.cuh — shared declarations for libscone_b200.so (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include <vector>
#include "scone_b200.h"

void scone_set_error(const char* fmt, ...);
extern std::atomic<long long> g_scone_launches;

#define SCONE_CUDA(x)                                                                                   \
    do {                                                                                                \
        cudaError_t e_ = (x);                                                                           \
        if (e_ != cudaSuccess) {                                                                        \
            scone_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #x, cudaGetErrorString(e_));         \
            return 1;                                                                                   \
        }                                                                                               \
    } while (0)

#define SCONE_REQUIRE(cond, ...)                                                                        \
    do {                                                                                                \
        if (!(cond)) {                                                                                  \
            scone_set_error(__VA_ARGS__);                                                               \
            return 2;                                                                                   \
        }                                                                                               \
    } while (0)

#define SCONE_LAUNCHED()                                                                                \
    do {                                                                                                \
        g_scone_launches.fetch_add(1, std::memory_order_relaxed);                                       \
        SCONE_CUDA(cudaGetLastError());                                                                 \
    } while (0)

// Optional per-kernel timing (CUDA events on the launching stream), off by default; bench.py's roofline uses it.
enum { SCONE_K_LAYER_FWD = 0, SCONE_K_LAYER_BWD = 1, SCONE_K_LAYER0_FWD = 2, SCONE_K_LAYER0_BWD = 3, SCONE_K_READOUT = 4,
       SCONE_K_OTHER = 5, SCONE_K_FILL = 6, SCONE_K_CONE = 7, SCONE_K_COUNT = 8 };
extern bool g_scone_prof;
void scone_prof_begin_impl(int kind, cudaStream_t st);
void scone_prof_end_impl(int kind, cudaStream_t st);
// device counter of the (edge, trajectory) rows a unit kernel family produced while profiling is on (NULL when off)
unsigned long long* scone_prof_row_counter(int kind);
struct ScopedProf {
    int kind; cudaStream_t st;
    ScopedProf(int k, cudaStream_t s) : kind(k), st(s) { if (g_scone_prof) scone_prof_begin_impl(kind, st); }
    ~ScopedProf() { if (g_scone_prof) scone_prof_end_impl(kind, st); }
};

// Hints the model-level code passes to one flagged kernel-level call (the *_hinted functions and scone_readout_ws below; nullptr =
// none, which is what the public C entry points pass):
//   in_wl/in_tt   the previous call's output worklist (index in the scratch, unit width) describes occ_in -> no re-compaction
//   skip_fill     the caller reads only the flagged rows of the output: no zero-fill, unflagged rows stay unwritten
// out_wl/out_tt are written back by the call (out_wl stays -1 when it built no output worklist).
//   in_bm         row bitmap of occ_in (bit e*b + t set <=> flag byte set): compaction reads it instead of the E*b flag bytes
//   out_bm        row bitmap the producer call (scone_flows_to_dense, scone_readout) should set next to the flags it writes
struct SconeLaunchHints {
    int in_wl = -1, in_tt = 0, out_wl = -1, out_tt = 0;
    bool skip_fill = false;
    const uint32_t* in_bm = nullptr;
    uint32_t* out_bm = nullptr;
    uint32_t* cand_bm = nullptr;     // readout: also mark the candidate rows one hop beyond the rows of G_L it writes
};
static inline size_t scone_bitmap_words(size_t E, size_t b) { return ((E * b + 31) / 32 + 31) / 16 * 16; }   // padded to whole 64-byte groups

// Integer-valued shift operator in CSR form.  ent[p] = {column, float bits of the coefficient};
// columns ascending inside a row (fixed, deterministic summation order).
struct DevCsr {
    const int32_t* rowptr;
    const int2* ent;
};

struct HostCsr {
    std::vector<int32_t> rowptr;
    std::vector<int32_t> col;
    std::vector<float> val;
};

struct scone_complex {
    int32_t N = 0, E = 0, F = 0, D = 0, model = 0;
    int num_sms = 148;
    bool host_only = false;                    // built by scone_complex_create_index_only: no device arrays
    HostCsr hS[2];
    std::vector<int32_t> h_nbrhoods;           // [N][D], pad -1
    std::vector<int32_t> h_rank;               // [E] caller's edge id -> internal edge row
    // device
    int32_t* d_rowptr[2] = {nullptr, nullptr};
    int2* d_ent[2] = {nullptr, nullptr};
    int32_t* d_nbrhoods = nullptr;             // [N][D]
    int32_t* d_inc_ptr = nullptr;              // [N+1]   B1 rows: node -> incident edges
    int2* d_inc_ent = nullptr;                 // [2E]    {internal edge id, float bits of sign}, ascending
    int32_t* d_rank = nullptr;                 // [E]     caller's edge id -> internal (locality-ordered) edge row
    // merged operator rows (slab kernels): union of the S0 / S1 patterns (+ the diagonal), columns ascending,
    // ent = {internal column, (c1 << 16) | (c0 & 0xffff)} with both integer coefficients as int16
    int32_t* d_mptr = nullptr;                 // [E+1]
    int2* d_ment = nullptr;
    DevCsr S(int k) const { return DevCsr{d_rowptr[k], d_ent[k]}; }
};

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
int scone_zero_fill(const scone_complex* cx, void* p, size_t bytes, cudaStream_t st);

// internal kernels-level helpers implemented in scone_kernels.cu
int scone_layer0_forward(const scone_complex* cx, int32_t act, int32_t b, int32_t cout, const float* X_dev,
                         const float* W0, const float* W1, const float* W2, float* Hout, const uint8_t* occ_in, uint8_t* occ_out,
                         uint8_t* scratch, void* stream, SconeLaunchHints* hints);
int64_t scone_layer0_backward_workspace_bytes(int32_t cout);
int scone_layer0_backward(const scone_complex* cx, int32_t b, int32_t cout, const float* G_dev, const float* X_dev,
                          float* dW_dev, int32_t accumulate, void* workspace, const uint8_t* occ_g, uint8_t* scratch,
                          void* stream, const SconeLaunchHints* hints);
int64_t scone_readout_workspace_bytes(int32_t b, int32_t C);
// scone_flows_to_dense, scone_layer_forward, scone_layer_backward and scone_readout of scone_b200.h, with launch hints
int scone_flows_to_dense_hinted(const scone_complex* cx, int32_t b, const int32_t* traj_ptr, const int32_t* flow_edge,
                                const float* flow_val, float* X, uint8_t* occX, void* stream, const SconeLaunchHints* hints);
int scone_layer_forward_hinted(const scone_complex* cx, int32_t act, int32_t b, int32_t cin, int32_t cout, const float* Hin,
                               const float* W0, const float* W1, const float* W2, float* Hout, const uint8_t* occ_in,
                               uint8_t* occ_out, uint8_t* occ_scratch, void* stream, SconeLaunchHints* hints);
int scone_layer_backward_hinted(const scone_complex* cx, int32_t act, int32_t b, int32_t cin, int32_t cout, const float* G,
                                const float* Hin, const float* W0, const float* W1, const float* W2, float* Gprev, float* dW,
                                int32_t accumulate, void* workspace, const uint8_t* occ_g, const uint8_t* occ_hin,
                                uint8_t* occ_prev, uint8_t* occ_scratch, void* stream, SconeLaunchHints* hints);
int scone_readout_ws(const scone_complex* cx, int32_t act, int32_t b, int32_t C, const float* HL, const float* wout,
                     const int32_t* last_nodes, float* logprobs, const int32_t* target_idx, const float* mask,
                     float scale, float* GL, float* dwout, float* nll_sum, float* count, int32_t accumulate,
                     void* workspace, const uint8_t* occ_HL, uint8_t* occ_GL, void* stream, const SconeLaunchHints* hints,
                     const float* cot = nullptr);   // cot [b][D]: cotangent seed instead of target_idx / mask (readout_kernel)
// data-parallel exchange fused with Adam (scone_dp.cu)
struct scone_dp;
int scone_dp_allreduce_adam(scone_dp* d, float* W, float* m, float* v, float* grad, int64_t n_params, const int* overflow_dev,
                            int32_t step, float lr, float wd, cudaStream_t st);
// tcgen05 dense layer (scone_umma.cu)
bool scone_umma_supported(const scone_complex* cx, int cin, int cout, int b);
int scone_umma_forward(const scone_complex* cx, int act, int b, const float* Hin, const float* W0, const float* W1, const float* W2,
                       float* Hout, cudaStream_t st);
int scone_umma_backward(const scone_complex* cx, int act, int b, const float* G, const float* Hin, const float* W0, const float* W1,
                        const float* W2, float* Gprev, float* dW, int accumulate, float* ws, cudaStream_t st);
int scone_umma_check(cudaStream_t st);
// slab kernels (scone_slab.cu): dense fused layer for widths 16 / 32, tensor-core product
extern int g_scone_dense_kernel;
bool scone_slab_supported(const scone_complex* cx, int cin, int cout);
int scone_slab_forward(const scone_complex* cx, int act, int b, int cin, int cout, const float* Hin, const float* W0, const float* W1,
                       const float* W2, float* Hout, cudaStream_t st);
int scone_slab_forward_rows(const scone_complex* cx, int act, int b, int cin, int cout, const float* Hin, const float* W0,
                            const float* W1, const float* W2, float* Hout, const uint8_t* occ_in, const uint32_t* rows,
                            const int* n_rows_dev, unsigned long long* row_counter, const uint32_t* bm_in, const uint32_t* pref_in,
                            int out_cap, int* overflow_dev, cudaStream_t st);
int scone_rows_mark(const scone_complex* cx, int b, const uint32_t* rows, const int* n_dev, uint32_t* bm_next, int list_cap,
                    cudaStream_t st, bool tmaj, size_t sum_off = 0, const uint32_t* bm_filter = nullptr);
// cone pipeline: two-level bitmaps (summary words at bm + sum_off, sum_off = 0: none)
int scone_rows_cone(const scone_complex* cx, int b, const int32_t* last_nodes, uint32_t* const* bm_levels, int n_levels, size_t sum_off,
                    int* overflow_dev, cudaStream_t st);
int scone_compact_rows_summary(const scone_complex* cx, int b, const uint32_t* bm, size_t sum_off, uint32_t* list, int* n_dev,
                               unsigned long long* tickets, cudaStream_t st, uint32_t* pref_out, long long list_cap);
int scone_clear_summary(const scone_complex* cx, int b, uint32_t* const* bms, int count, int master, size_t sum_off, cudaStream_t st);
// bitmap-native row-list pipeline (scone_rows.cu, scone_slab.cu)
bool scone_rows_supported(const scone_complex* cx, int n_layers, const int32_t* hidden);
int64_t scone_rows_dw_workspace_bytes(int cin, int cout);
size_t scone_ticket_bytes();
int scone_compact_rows(const scone_complex* cx, int b, const uint32_t* bm, uint32_t* list, int* n_dev, unsigned long long* tickets,
                       cudaStream_t st, uint32_t* pref_out = nullptr, long long list_cap = (1ll << 62));
int scone_rows_flows(const scone_complex* cx, int b, const int32_t* traj_ptr, const int32_t* flow_edge, const float* flow_val, float* X,
                     uint32_t* bmX, uint32_t* bm_next, bool clear, bool tmaj, cudaStream_t st, const uint32_t* bm_filter = nullptr,
                     size_t sum_off = 0);
int scone_rows_layer0_forward(const scone_complex* cx, int act, int b, int cout, const float* X, const float* W0, const float* W1,
                              const float* W2, float* Hout, const uint32_t* rows, const int* n_dev, uint32_t* bm_next, int out_cap,
                              int* overflow_dev, cudaStream_t st);
int scone_rows_layer0_backward(const scone_complex* cx, int b, int cout, const float* X, const float* G, const uint32_t* rows,
                               const int* n_dev, float* dW, int accumulate, float* ws, int g_cap, cudaStream_t st);
// dL/dx at the flow entries from G_1 = G (dense rows with byte flags occ, dense rows with bitmap bm, or compact rows through bm + pref)
int scone_rows_flow_grad(const scone_complex* cx, int b, const int32_t* traj_ptr, const int32_t* flow_edge, int C, const float* G,
                         const uint8_t* occ, const uint32_t* bm, const uint32_t* pref, int cap, const float* w0, const float* w1,
                         const float* w2, float* dflow, cudaStream_t st);
int scone_rows_backward(const scone_complex* cx, int act, int b, int cin, int cout, const float* G, const float* Hin, float* Gprev,
                        float* Abuf, const float* W0, const float* W1, const float* W2, const uint32_t* rows, const int* n_dev,
                        const uint32_t* bmG, const uint32_t* bmH, int a_cap, int* overflow_dev, float* dW, int accumulate, float* ws,
                        const uint32_t* prefG, const uint32_t* prefH, bool hin_by_list, cudaStream_t st);
int scone_rows_readout_forward(const scone_complex* cx, int b, int C, const float* HL, const float* wout, const int32_t* last_nodes,
                               float* logprobs, const uint32_t* bmH, const uint32_t* prefH, uint32_t* bmG, uint32_t* bm_cand,
                               cudaStream_t st);
int scone_rows_readout_backward(const scone_complex* cx, int act, int b, int C, const float* HL, const float* wout,
                                const int32_t* last_nodes, const float* logprobs, const int32_t* target_idx, const float* mask,
                                float scale, float* GL, const int* n_dev, int g_cap, int* overflow_dev, float* dwout, float* nll_sum,
                                float* count, int accumulate, float* ws, const uint32_t* bmH, const uint32_t* prefH, const uint32_t* bmG,
                                const uint32_t* prefG, cudaStream_t st, const float* cot = nullptr);
int scone_accuracy_launch(int B, int D, const float* logprobs, const int32_t* n_nbrs, const int32_t* target_idx, const float* mask,
                          int32_t* out, cudaStream_t st);
int scone_predict_launch(int B, int D, const float* logprobs, const int32_t* n_nbrs, int32_t* choice, cudaStream_t st);
int scone_two_target_launch(int B, int D, const float* logprobs, const int32_t* n_nbrs, const int32_t* true_idx, const int32_t* rand_idx,
                            const float* mask, int32_t* out, cudaStream_t st);
int scone_nll_launch(int B, int D, const float* logprobs, const int32_t* target_idx, const float* mask, float* out, cudaStream_t st);
int scone_add_scalar_launch(float* dst, float v, cudaStream_t st);      // *dst += v on the stream (the count of a VJP call)
int scone_adam_launch(float* W, float* m, float* v, const float* gradbuf, int64_t n, int32_t step, float lr,
                      float wd, void* stream, const int* overflow_dev = nullptr);
