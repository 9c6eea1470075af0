// scone_model.cu — model-level entry points: micro-batched forward / loss+grad / Adam.
//
// Replaces, for -model scone / ebli, the reference's
//   Scone_GCN.setup + generate_weights shapes   scone_trajectory_model.py:215-262
//   self.model(weights, *shifts, *inputs)       scone_trajectory_model.py:46,64   (vmap of scone_func / ebli_func)
//   grad(self.loss) + adam update               scone_trajectory_model.py:300-326
// Trajectories are processed in micro-batches of `micro_batch` so that the [E][b][C] activations of all
// layers stay resident in HBM (SURVEY.md §7 H2); weight gradients accumulate across micro-batches in one
// flat device buffer [grads | nll_sum | count] that is the single all-reduce payload of a data-parallel step.
#include <algorithm>
#include <cstring>
#include "common.cuh"
#include "fused.cuh"

struct scone_model {
    const scone_complex* cx = nullptr;
    int32_t L = 0, mb = 0, act = 0, cmax = 0;
    std::vector<int32_t> hidden;              // channel count per conv layer
    std::vector<int64_t> w_off;               // offsets of W[0..3L] in the flat buffer
    int64_t n_params = 0;
    float *d_w = nullptr, *d_m = nullptr, *d_v = nullptr, *d_grad = nullptr;     // d_grad: [n_params + 2]
    float* d_X = nullptr;                     // [E][mb]
    std::vector<float*> d_H;                  // H_1..H_L, [E][mb][C_l]
    std::vector<float*> d_G;                  // dL/dZ of layer l, [E][mb][C_l]
    std::vector<uint8_t*> d_occH;             // occupancy flags of H_1..H_L, [E][mb]
    std::vector<uint8_t*> d_occG;             // occupancy flags of the dL/dZ buffers
    cudaStream_t compute = nullptr;           // all kernels of a model-level call (highest priority), forked from / joined to the caller's stream
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaStream_t copy = nullptr;              // pipeline 4, *_host entry points: the flow arrays arrive in parts under the plan kernels
    cudaEvent_t ev_copy0 = nullptr, ev_part[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_plan_done = nullptr;       // the plan kernels of the last overlapped *_host call have read the flow staging buffers
    long long staging_epoch = 0, plan_done_epoch = -1;      // ensure_staging calls so far / value when ev_plan_done was recorded
    uint8_t* d_occS = nullptr;                // worklists / counters scratch (scone_occ_scratch_bytes)
    uint8_t* d_occX = nullptr;                // flags of the flows X
    uint32_t *d_bmX = nullptr, *d_bmG = nullptr;   // quad bitmaps of the flags of X and of G_L (compaction reads these)
    // bitmap-native row-list pipeline (scone_rows.cu): row bitmaps per tensor, one row list, compact A rows for the dW GEMM
    // pipeline: 0 unit kernels + byte flags (dense [E][mb][C] tensors), 1 row lists over the dense tensors, 2 row lists over
    // COMPACT tensors (row r of a tensor at index rank(r) of its bitmap = its position in the compacted row list), 3 the same
    // kernels over the READOUT CONE only: H_l and G_l share one row set per layer, the rows that can reach the log-probs
    bool rows_ok = false, x_clean = false, dense_ready = false, rows_ready = false, compact_ready = false;
    bool cone_clean = false;                  // pipeline 3: the two-level bitmaps d_bmGr are all-zero between micro-batches
    size_t sum_off = 0, bmg_bytes = 0;        // summary words of d_bmGr[l] start at word sum_off; bytes of one d_bmGr allocation
    int pipeline = 0;
    FusedState* fused = nullptr;              // pipeline 4: trajectory-fused kernels (scone_fused.cu); nullptr = not available for this model
    std::vector<uint32_t*> d_bmH, d_bmGr, d_prefH, d_prefG;
    std::vector<uint32_t*> d_bmC;             // pipeline 3: geometric cone per layer (d_bmGr[l] then holds the LIVE rows: cone & support)
    std::vector<float*> d_cH, d_cG;           // compact tensors [row_cap][C_l]
    int row_cap = 0;                          // rows a compact tensor / the row list can hold
    size_t rows_list_cap = 0;
    uint32_t* d_rows = nullptr;
    std::vector<uint32_t*> d_rowsC;           // pipeline 3: the cone's row list per layer (forward and backward walk the same list)
    int* d_nrows = nullptr;                   // {count, tile counter} pairs: [0] the shared list, [1 + l] the cone list of layer l
    int* d_overflow = nullptr;
    unsigned long long* d_tickets = nullptr;
    float* d_Abuf = nullptr;
    int a_cap = 0;
    void* d_ws = nullptr;                     // backward / readout workspace
    float* d_logp = nullptr;                  // [mb][D]
    // staging for the *_host entry points
    int32_t *d_ptr = nullptr, *d_edge = nullptr, *d_last = nullptr, *d_tgt = nullptr, *d_nn = nullptr, *d_acc = nullptr;
    float *d_val = nullptr, *d_mask = nullptr, *d_logp_all = nullptr;
    float* d_cot = nullptr;                   // [cap_B][D] cotangents of the *_vjp_*_host entry points (allocated on first use)
    float* d_dflow = nullptr;                 // [cap_dflow] flow gradients of scone_model_vjp_flows_host (allocated on first use)
    int64_t cap_B = 0, cap_nnz = 0, cap_cot = 0, cap_dflow = 0;
    int32_t *d_choice = nullptr, *d_rand = nullptr;   // evaluation: predictions, random other targets
    float* d_evalf = nullptr;
    int64_t cap_choice = 0;
    int32_t eval_B = 0;                        // trajectories whose log-probs scone_model_eval_host left in d_logp_all
};

namespace {

int ensure_staging(scone_model* m, int64_t B, int64_t nnz) {
    m->staging_epoch += 1;
    if (nnz > m->cap_nnz) m->plan_done_epoch = -1;       // (the buffers are about to be reallocated)
    if (B > m->cap_B) {
        cudaFree(m->d_ptr); cudaFree(m->d_last); cudaFree(m->d_tgt); cudaFree(m->d_mask); cudaFree(m->d_logp_all); cudaFree(m->d_nn);
        int64_t cap = B + B / 4 + 16;
        SCONE_CUDA(cudaMalloc((void**)&m->d_ptr, (cap + 1) * sizeof(int32_t)));
        SCONE_CUDA(cudaMalloc((void**)&m->d_last, cap * sizeof(int32_t)));
        SCONE_CUDA(cudaMalloc((void**)&m->d_tgt, cap * sizeof(int32_t)));
        SCONE_CUDA(cudaMalloc((void**)&m->d_nn, cap * sizeof(int32_t)));
        if (!m->d_acc) SCONE_CUDA(cudaMalloc((void**)&m->d_acc, 2 * sizeof(int32_t)));
        SCONE_CUDA(cudaMalloc((void**)&m->d_mask, cap * sizeof(float)));
        SCONE_CUDA(cudaMalloc((void**)&m->d_logp_all, cap * (size_t)(m->cx->D > 0 ? m->cx->D : 1) * sizeof(float)));
        m->cap_B = cap;
    }
    if (nnz > m->cap_nnz) {
        cudaFree(m->d_edge); cudaFree(m->d_val);
        int64_t cap = nnz + nnz / 4 + 16;
        SCONE_CUDA(cudaMalloc((void**)&m->d_edge, cap * sizeof(int32_t)));
        SCONE_CUDA(cudaMalloc((void**)&m->d_val, cap * sizeof(float)));
        m->cap_nnz = cap;
    }
    return 0;
}

// Copies the [B][D] cotangents of a *_vjp_*_host entry point to the device staging buffer on s.
int stage_cot(scone_model* m, int32_t B, const float* cot, cudaStream_t s) {
    const size_t n = (size_t)B * m->cx->D;
    if ((int64_t)n > m->cap_cot) {
        cudaFree(m->d_cot);
        m->d_cot = nullptr;
        m->cap_cot = 0;
        const size_t cap = n + n / 4 + 16;
        SCONE_CUDA(cudaMalloc((void**)&m->d_cot, cap * sizeof(float)));
        m->cap_cot = (int64_t)cap;
    }
    if (n) SCONE_CUDA(cudaMemcpyAsync(m->d_cot, cot, n * sizeof(float), cudaMemcpyHostToDevice, s));
    return 0;
}

// Stages the HOST inputs of a *_host entry point on s: ptr [B+1] always; last / n_nbrs / tgt / mask [B] when B > 0 and given; the
// flow arrays edge / val [ptr[B]] when `flows` (the overlapped fused path copies them itself, on its copy stream).
int stage_host_inputs(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* last, const int32_t* n_nbrs, const int32_t* tgt,
                      const float* mask, const int32_t* edge, const float* val, bool flows, cudaStream_t s) {
    const int64_t nnz = B > 0 ? ptr[B] : 0;
    if (ensure_staging(m, B, nnz)) return 1;
    SCONE_CUDA(cudaMemcpyAsync(m->d_ptr, ptr, (B + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    if (B > 0) {
        if (last) SCONE_CUDA(cudaMemcpyAsync(m->d_last, last, B * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        if (n_nbrs) SCONE_CUDA(cudaMemcpyAsync(m->d_nn, n_nbrs, B * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        if (tgt) SCONE_CUDA(cudaMemcpyAsync(m->d_tgt, tgt, B * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        if (mask) SCONE_CUDA(cudaMemcpyAsync(m->d_mask, mask, B * sizeof(float), cudaMemcpyHostToDevice, s));
    }
    if (flows && nnz > 0) {
        SCONE_CUDA(cudaMemcpyAsync(m->d_edge, edge, nnz * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        SCONE_CUDA(cudaMemcpyAsync(m->d_val, val, nnz * sizeof(float), cudaMemcpyHostToDevice, s));
    }
    return 0;
}

// Reports a row-list capacity overflow of the work enqueued on s so far (error code 4): copies the device flag, synchronises s and,
// if it is set, clears it.  `what` names the entry point.
int report_overflow(scone_model* m, cudaStream_t s, const char* what) {
    int overflow = 0;
    if (m->d_overflow) SCONE_CUDA(cudaMemcpyAsync(&overflow, m->d_overflow, sizeof(int), cudaMemcpyDeviceToHost, s));
    SCONE_CUDA(cudaStreamSynchronize(s));
    if (!overflow) return 0;
    cudaMemset(m->d_overflow, 0, sizeof(int));
    m->cone_clean = false;                                 // a truncated cone list: the clearing may have missed bits
    scone_set_error("%s: a micro-batch exceeded a row-list capacity (%d rows per compact tensor, %d rows of the backward's A buffer, 2048 "
                    "cone edges per trajectory and layer); results since the last check are incomplete and any Adam step since then was "
                    "skipped — use a smaller micro-batch or another pipeline (scone_model_set_pipeline)", what, m->row_cap, m->a_cap);
    return 4;
}

// forward over one micro-batch [off, off+b): X -> H_1 .. H_L (kept) ; returns 0 on success
int forward_mb(scone_model* m, int32_t b, const int32_t* ptr, const int32_t* edge, const float* val, void* st) {
    const scone_complex* cx = m->cx;
    SconeLaunchHints xh;
    xh.out_bm = m->d_bmX;
    int rc = scone_flows_to_dense_hinted(cx, b, ptr, edge, val, m->d_X, m->d_occX, st, &xh);
    if (rc) return rc;
    const float* in = m->d_X;
    int cin = 1, wl = -1, tt = 0;
    for (int l = 0; l < m->L; ++l) {
        const int cout = m->hidden[l];
        SconeLaunchHints h;                  // the previous layer's output worklist; layer 0 compacts from the bitmap of X
        h.in_wl = wl;
        h.in_tt = tt;
        h.skip_fill = true;
        if (l == 0) h.in_bm = m->d_bmX;
        rc = scone_layer_forward_hinted(cx, m->act, b, cin, cout, in, m->d_w + m->w_off[3 * l], m->d_w + m->w_off[3 * l + 1],
                                        m->d_w + m->w_off[3 * l + 2], m->d_H[l], l > 0 ? m->d_occH[l - 1] : m->d_occX, m->d_occH[l],
                                        m->d_occS, st, &h);
        if (rc) return rc;
        wl = h.out_wl;
        tt = h.out_tt;
        in = m->d_H[l];
        cin = cout;
    }
    return 0;
}

// backward over one micro-batch whose readout has written G_L: G_L -> G_{L-1} .. G_1, weight gradients accumulated into d_grad
int backward_mb(scone_model* m, int32_t b, void* st) {
    const int L = m->L;
    int wl = -1, tt = 0;
    for (int l = L - 1; l >= 0; --l) {
        const int cout = m->hidden[l], cin = l > 0 ? m->hidden[l - 1] : 1;
        const float* Hin = l > 0 ? m->d_H[l - 1] : m->d_X;
        SconeLaunchHints h;                  // the previous layer's output worklist; layer L - 1 compacts from the bitmap of G_L
        h.in_wl = wl;
        h.in_tt = tt;
        h.skip_fill = l > 0;                 // layer 0 writes no G_{l-1}
        if (l == L - 1) h.in_bm = m->d_bmG;
        int rc = scone_layer_backward_hinted(m->cx, m->act, b, cin, cout, m->d_G[l], Hin, m->d_w + m->w_off[3 * l], m->d_w + m->w_off[3 * l + 1],
                                             m->d_w + m->w_off[3 * l + 2], l > 0 ? m->d_G[l - 1] : nullptr, m->d_grad + m->w_off[3 * l], 1,
                                             m->d_ws, m->d_occG[l], l > 0 ? m->d_occH[l - 1] : nullptr, l > 0 ? m->d_occG[l - 1] : nullptr,
                                             m->d_occS, st, &h);
        if (rc) return rc;
        wl = h.out_wl;
        tt = h.out_tt;
    }
    return 0;
}

// dL/dx at the flow entries of a micro-batch from G_1 (after the backward; see rows_flow_grad_kernel for the three addressings)
int flow_grad_mb(scone_model* m, int32_t b, const int32_t* ptr, const int32_t* edge, const float* G, const uint8_t* occ,
                 const uint32_t* bm, const uint32_t* pref, float* dflow, cudaStream_t s) {
    ScopedProf prof(SCONE_K_LAYER0_BWD, s);
    return scone_rows_flow_grad(m->cx, b, ptr, edge, m->hidden[0], G, occ, bm, pref, m->row_cap, m->d_w + m->w_off[0], m->d_w + m->w_off[1],
                                m->d_w + m->w_off[2], dflow, s);
}

// pipeline 0 over one micro-batch [off, off+b) (ptr / last / tgt / mask / cot: at off); grad = false: log-probs only; cot != NULL:
// the gradient is seeded with the cotangent rows instead of tgt / mask; dflow != NULL (with cot): dL/dx at the flow entries too
int unit_mb(scone_model* m, int32_t b, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last, float* logprobs,
            const int32_t* tgt, const float* mask, const float* cot, float* dflow, bool grad, cudaStream_t s) {
    const int L = m->L, CL = m->hidden[L - 1];
    const float* wout = m->d_w + m->w_off[3 * L];
    m->x_clean = false;
    int rc = forward_mb(m, b, ptr, edge, val, s);
    if (rc) return rc;
    if (!grad)
        return scone_readout_ws(m->cx, m->act, b, CL, m->d_H[L - 1], wout, last, logprobs, nullptr, nullptr, 0.f, nullptr, nullptr, nullptr,
                                nullptr, 0, nullptr, m->d_occH[L - 1], nullptr, s, nullptr);
    SconeLaunchHints h;                      // G_L's flags also go to the bitmap d_bmG
    h.skip_fill = true;
    h.out_bm = m->d_bmG;
    rc = scone_readout_ws(m->cx, m->act, b, CL, m->d_H[L - 1], wout, last, logprobs, tgt, mask, 1.f, m->d_G[L - 1], m->d_grad + m->w_off[3 * L],
                          m->d_grad + m->n_params, m->d_grad + m->n_params + 1, 1, m->d_ws, m->d_occH[L - 1], m->d_occG[L - 1], s, &h, cot);
    if (!rc) rc = backward_mb(m, b, s);
    if (!rc && dflow) rc = flow_grad_mb(m, b, ptr, edge, m->d_G[0], m->d_occG[0], nullptr, nullptr, dflow, s);
    return rc;
}

// ---- buffers of the active pipeline, allocated on first use ----------------------------------------------------------
int dev_alloc(void** p, size_t bytes, const char* what) {
    if (*p) return 0;
    cudaError_t e = cudaMalloc(p, bytes ? bytes : 4);
    if (e != cudaSuccess) {
        scone_set_error("scone_model: cudaMalloc(%zu bytes) for %s failed: %s", bytes, what, cudaGetErrorString(e));
        *p = nullptr;
        return 1;
    }
    return 0;
}
#define SCONE_ALLOC(p, bytes, what)                      \
    do {                                                 \
        if (dev_alloc((void**)&(p), (bytes), (what))) return 1; \
    } while (0)

int ensure_buffers(scone_model* m) {
    const scone_complex* cx = m->cx;
    const size_t E = cx->E, mb = m->mb;
    const int L = m->L;
    const int pl = m->pipeline;
    if (!m->d_overflow) {
        SCONE_ALLOC(m->d_overflow, 256, "counters");
        SCONE_CUDA(cudaMemset(m->d_overflow, 0, 256));
    }
    if (pl == 4) return 0;                                 // the fused pipeline owns its buffers (FusedState); no dense X, no bitmaps
    SCONE_ALLOC(m->d_X, E * mb * sizeof(float), "dense flows X");
    if (pl <= 1 && !m->dense_ready) {                      // dense [E][mb][C] tensors (+ byte flags for the unit kernels)
        for (int l = 0; l < L; ++l) {
            SCONE_ALLOC(m->d_H[l], E * mb * m->hidden[l] * sizeof(float), "dense activations");
            SCONE_ALLOC(m->d_G[l], E * mb * m->hidden[l] * sizeof(float), "dense gradients");
            SCONE_ALLOC(m->d_occH[l], E * mb, "flags");
            SCONE_ALLOC(m->d_occG[l], E * mb, "flags");
        }
        SCONE_ALLOC(m->d_occS, (size_t)scone_occ_scratch_bytes(cx, m->mb), "worklist scratch");
        SCONE_ALLOC(m->d_occX, E * mb, "flags");
        SCONE_ALLOC(m->d_bmX, scone_bitmap_words(E, mb) * 4, "bitmap");
        SCONE_ALLOC(m->d_bmG, scone_bitmap_words(E, mb) * 4, "bitmap");
        m->dense_ready = true;
    }
    if (pl >= 1 && !m->rows_ready) {                       // row bitmaps, the row list, the compact A buffer
        const size_t bm_bytes = scone_bitmap_words(E, mb) * 4;
        m->d_bmH.resize(L, nullptr);
        m->d_bmGr.resize(L, nullptr);
        m->sum_off = scone_bitmap_words(E, mb);             // + one summary bit per bitmap word (cone pipeline)
        m->bmg_bytes = bm_bytes + ((m->sum_off + 31) / 32 + 16) * 4;
        for (int l = 0; l < L; ++l) SCONE_ALLOC(m->d_bmGr[l], m->bmg_bytes, "bitmap");
        SCONE_ALLOC(m->d_nrows, 8 * (size_t)(L + 1), "counters");
        SCONE_ALLOC(m->d_tickets, scone_ticket_bytes(), "tickets");
        const size_t acap = E * mb < (size_t)6000000 ? E * mb : (size_t)6000000;    // rows of the compact A buffer (backward)
        m->a_cap = (int)acap;
        SCONE_ALLOC(m->d_Abuf, acap * 3 * (size_t)m->cmax * sizeof(float), "A buffer");
        const size_t rcap = E * mb < (size_t)32000000 ? E * mb : (size_t)32000000;   // rows of a compact tensor
        m->row_cap = (int)rcap;
        m->rows_ready = true;
    }
    if (pl == 1 || pl == 2) {                              // bitmaps of X and the activations (the cone pipeline has none)
        const size_t bm_bytes = scone_bitmap_words(E, mb) * 4;
        SCONE_ALLOC(m->d_bmX, bm_bytes, "bitmap");
        for (int l = 0; l < L; ++l) SCONE_ALLOC(m->d_bmH[l], bm_bytes, "bitmap");
    }
    if (pl == 1 || pl == 2) {                              // the row list: every row under pipeline 1, row_cap rows under 2
        const size_t need = pl == 1 ? E * mb : (size_t)m->row_cap;
        if (need > m->rows_list_cap) {
            cudaFree(m->d_rows);
            m->d_rows = nullptr;
            SCONE_ALLOC(m->d_rows, need * sizeof(uint32_t), "row list");
            m->rows_list_cap = need;
        }
    }
    if (pl >= 2) {                                         // compact tensors + rank prefixes (allocated once, shared by 2 and 3)
        const size_t bm_bytes = scone_bitmap_words(E, mb) * 4;
        m->d_prefH.resize(L, nullptr);
        m->d_prefG.resize(L, nullptr);
        m->d_cH.resize(L, nullptr);
        m->d_cG.resize(L, nullptr);
        m->d_rowsC.resize(L, nullptr);
        for (int l = 0; l < L; ++l) {
            if (pl == 2) SCONE_ALLOC(m->d_prefH[l], bm_bytes, "rank prefix");
            SCONE_ALLOC(m->d_prefG[l], bm_bytes, "rank prefix");
            SCONE_ALLOC(m->d_cH[l], (size_t)m->row_cap * m->hidden[l] * sizeof(float), "compact activations");
            SCONE_ALLOC(m->d_cG[l], (size_t)m->row_cap * m->hidden[l] * sizeof(float), "compact gradients");
            if (pl == 3) SCONE_ALLOC(m->d_rowsC[l], (size_t)m->row_cap * sizeof(uint32_t), "cone row list");
            if (pl == 3) {
                m->d_bmC.resize(L, nullptr);
                SCONE_ALLOC(m->d_bmC[l], m->bmg_bytes, "cone bitmap");
            }
        }
    }
    return 0;
}

// ---- row-list pipeline -------------------------------------------------------------------------------------------
int rows_forward_mb(scone_model* m, int32_t b, const int32_t* ptr, const int32_t* edge, const float* val, cudaStream_t s) {
    const scone_complex* cx = m->cx;
    const bool compact = m->pipeline == 2;
    const size_t bm_bytes = scone_bitmap_words(cx->E, b) * 4;
    const long long list_cap = compact ? (long long)m->row_cap : (1ll << 62);
    m->cone_clean = false;                                 // pipelines 1 / 2 use d_bmGr as plain bitmaps
    if (!m->x_clean) {                                     // X must be all-zero outside the flows (no flag test in the first layer)
        SCONE_CUDA(cudaMemsetAsync(m->d_X, 0, (size_t)cx->E * m->mb * sizeof(float), s));
        m->x_clean = true;
    }
    {
        ScopedProf prof(SCONE_K_OTHER, s);
        SCONE_CUDA(cudaMemsetAsync(m->d_bmX, 0, bm_bytes, s));
        SCONE_CUDA(cudaMemsetAsync(m->d_bmH[0], 0, bm_bytes, s));
        if (scone_rows_flows(cx, b, ptr, edge, val, m->d_X, m->d_bmX, m->d_bmH[0], false, compact, s)) return 1;
    }
    int cin = 1;
    for (int l = 0; l < m->L; ++l) {
        const int cout = m->hidden[l];
        ScopedProf prof(l == 0 ? SCONE_K_LAYER0_FWD : SCONE_K_LAYER_FWD, s);
        if (scone_compact_rows(cx, b, m->d_bmH[l], m->d_rows, m->d_nrows, m->d_tickets, s, compact ? m->d_prefH[l] : nullptr, list_cap))
            return 1;
        uint32_t* next = l + 1 < m->L ? m->d_bmH[l + 1] : nullptr;
        if (next) {
            SCONE_CUDA(cudaMemsetAsync(next, 0, bm_bytes, s));
            if (scone_rows_mark(cx, b, m->d_rows, m->d_nrows, next, compact ? m->row_cap : 0x7fffffff, s, compact)) return 1;
        }
        const float *W0 = m->d_w + m->w_off[3 * l], *W1 = m->d_w + m->w_off[3 * l + 1], *W2 = m->d_w + m->w_off[3 * l + 2];
        float* Hout = compact ? m->d_cH[l] : m->d_H[l];
        int rc;
        if (l == 0)
            rc = scone_rows_layer0_forward(cx, m->act, b, cout, m->d_X, W0, W1, W2, Hout, m->d_rows, m->d_nrows, nullptr,
                                           compact ? m->row_cap : 0, m->d_overflow, s);
        else
            rc = scone_slab_forward_rows(cx, m->act, b, cin, cout, compact ? m->d_cH[l - 1] : m->d_H[l - 1], W0, W1, W2, Hout, nullptr,
                                         m->d_rows, m->d_nrows, scone_prof_row_counter(SCONE_K_LAYER_FWD), m->d_bmH[l - 1],
                                         compact ? m->d_prefH[l - 1] : nullptr, m->row_cap, m->d_overflow, s);
        if (rc) return rc;
        cin = cout;
    }
    return 0;
}

int rows_clear_x(scone_model* m, int32_t b, const int32_t* ptr, const int32_t* edge, const float* val, cudaStream_t s) {
    ScopedProf prof(SCONE_K_OTHER, s);
    return scone_rows_flows(m->cx, b, ptr, edge, val, m->d_X, nullptr, nullptr, true, m->pipeline >= 2, s);
}

// readout on the row-list pipelines; grad = false: log-probs only
int rows_readout(scone_model* m, int32_t b, const int32_t* last, float* logprobs, bool grad, const int32_t* tgt, const float* mask,
                 const float* cot, cudaStream_t s) {
    const scone_complex* cx = m->cx;
    const int L = m->L, CL = m->hidden[L - 1];
    const float* wout = m->d_w + m->w_off[3 * L];
    ScopedProf prof(SCONE_K_READOUT, s);
    if (m->pipeline == 1) {
        SconeLaunchHints h;                  // row bitmaps instead of flag bytes; G_L is read only at the rows its bitmap marks: no fill
        h.skip_fill = true;
        h.in_bm = m->d_bmH[L - 1];
        if (grad) {
            h.out_bm = m->d_bmGr[L - 1];
            h.cand_bm = L >= 2 ? m->d_bmGr[L - 2] : nullptr;
            return scone_readout_ws(cx, m->act, b, CL, m->d_H[L - 1], wout, last, logprobs, tgt, mask, 1.f, m->d_G[L - 1],
                                    m->d_grad + m->w_off[3 * L], m->d_grad + m->n_params, m->d_grad + m->n_params + 1, 1, m->d_ws, nullptr,
                                    nullptr, s, &h, cot);
        }
        return scone_readout_ws(cx, m->act, b, CL, m->d_H[L - 1], wout, last, logprobs, nullptr, nullptr, 0.f, nullptr, nullptr, nullptr,
                                nullptr, 0, nullptr, nullptr, nullptr, s, &h);
    }
    const size_t bm_bytes = scone_bitmap_words(cx->E, b) * 4;
    uint32_t *bmG = nullptr, *cand = nullptr;
    if (grad) {
        bmG = m->d_bmGr[L - 1];
        SCONE_CUDA(cudaMemsetAsync(bmG, 0, bm_bytes, s));
        if (L >= 2) {
            cand = m->d_bmGr[L - 2];
            SCONE_CUDA(cudaMemsetAsync(cand, 0, bm_bytes, s));
        }
    }
    if (scone_rows_readout_forward(cx, b, CL, m->d_cH[L - 1], wout, last, logprobs, m->d_bmH[L - 1], m->d_prefH[L - 1], bmG, cand, s)) return 1;
    if (!grad) return 0;
    if (scone_compact_rows(cx, b, bmG, m->d_rows, m->d_nrows, m->d_tickets, s, m->d_prefG[L - 1], m->row_cap)) return 1;
    return scone_rows_readout_backward(cx, m->act, b, CL, m->d_cH[L - 1], wout, last, logprobs, tgt, mask, 1.f, m->d_cG[L - 1], m->d_nrows,
                                       m->row_cap, m->d_overflow, m->d_grad + m->w_off[3 * L], m->d_grad + m->n_params,
                                       m->d_grad + m->n_params + 1, 1, (float*)m->d_ws, m->d_bmH[L - 1], m->d_prefH[L - 1], bmG,
                                       m->d_prefG[L - 1], s, cot);
}

int rows_backward_mb(scone_model* m, int32_t b, cudaStream_t s) {
    const scone_complex* cx = m->cx;
    const int L = m->L;
    const bool compact = m->pipeline == 2;
    const size_t bm_bytes = scone_bitmap_words(cx->E, b) * 4;
    const long long list_cap = compact ? (long long)m->row_cap : (1ll << 62);
    const int a_cap = compact && m->row_cap < m->a_cap ? m->row_cap : m->a_cap;
    for (int l = L - 1; l >= 1; --l) {
        ScopedProf prof(SCONE_K_LAYER_BWD, s);
        if (scone_compact_rows(cx, b, m->d_bmGr[l - 1], m->d_rows, m->d_nrows, m->d_tickets, s, compact ? m->d_prefG[l - 1] : nullptr, list_cap))
            return 1;
        uint32_t* next = l >= 2 ? m->d_bmGr[l - 2] : nullptr;
        if (next) {
            SCONE_CUDA(cudaMemsetAsync(next, 0, bm_bytes, s));
            if (scone_rows_mark(cx, b, m->d_rows, m->d_nrows, next, compact ? m->row_cap : 0x7fffffff, s, compact)) return 1;
        }
        int rc = scone_rows_backward(cx, m->act, b, m->hidden[l - 1], m->hidden[l], compact ? m->d_cG[l] : m->d_G[l],
                                     compact ? m->d_cH[l - 1] : m->d_H[l - 1], compact ? m->d_cG[l - 1] : m->d_G[l - 1], m->d_Abuf,
                                     m->d_w + m->w_off[3 * l], m->d_w + m->w_off[3 * l + 1], m->d_w + m->w_off[3 * l + 2], m->d_rows,
                                     m->d_nrows, m->d_bmGr[l], m->d_bmH[l - 1], a_cap, m->d_overflow, m->d_grad + m->w_off[3 * l], 1,
                                     (float*)m->d_ws, compact ? m->d_prefG[l] : nullptr, compact ? m->d_prefH[l - 1] : nullptr, false, s);
        if (rc) return rc;
    }
    ScopedProf prof(SCONE_K_LAYER0_BWD, s);
    if (L == 1 && !compact && scone_compact_rows(cx, b, m->d_bmGr[0], m->d_rows, m->d_nrows, m->d_tickets, s)) return 1;
    // (compact, L == 1: the list of G_0's rows is still the one the readout compacted)
    return scone_rows_layer0_backward(cx, b, m->hidden[0], m->d_X, compact ? m->d_cG[0] : m->d_G[0], m->d_rows, m->d_nrows,
                                      m->d_grad + m->w_off[0], 1, (float*)m->d_ws, compact ? m->row_cap : 0, s);
}

// pipelines 1 / 2 over one micro-batch (arguments as unit_mb)
int rows_mb(scone_model* m, int32_t b, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last, float* logprobs,
            const int32_t* tgt, const float* mask, const float* cot, float* dflow, bool grad, cudaStream_t s) {
    const bool compact = m->pipeline == 2;
    int rc = rows_forward_mb(m, b, ptr, edge, val, s);
    if (!rc) rc = rows_readout(m, b, last, logprobs, grad, tgt, mask, cot, s);
    if (!rc && grad) rc = rows_backward_mb(m, b, s);
    if (!rc && grad && dflow)                              // G_1's rows: d_bmGr[0] (+ its rank prefix when compact)
        rc = flow_grad_mb(m, b, ptr, edge, compact ? m->d_cG[0] : m->d_G[0], nullptr, m->d_bmGr[0], compact ? m->d_prefG[0] : nullptr,
                          dflow, s);
    if (!rc) rc = rows_clear_x(m, b, ptr, edge, val, s);
    return rc;
}

// ---- cone-pruned row-list pipeline (3) -----------------------------------------------------------------------------
// The log-probs of trajectory t read H_L only at the edges incident to the neighbours of its last node; H_{L-1} is needed one
// hop around those rows, and so on: the receptive cone (geometry only: d_bmC[l], built from last_nodes).  Inside the cone only
// the rows in the structural support of the flows can be non-zero; the LIVE rows of layer l (d_bmGr[l]) are the cone rows with a
// live neighbour one layer below (layer 0: a flow entry in their merged operator row) — marked layer by layer, each list
// compacted once.  A live row is computed exactly as in pipeline 2 (its live neighbours are pipeline 2's present neighbours
// inside the cone; everything it reads outside is an exact zero there too), so the log-probs are bit-identical.  The backward
// walks the same lists: G_l outside the cone is never needed, and G_l on a cone row outside the support multiplies exact zeros
// in every weight gradient and only feeds such rows further down — dropping it leaves every sum's non-zero terms unchanged.
// Each layer has ONE bitmap / rank prefix / row list for H_l and G_l.
int* cone_n(scone_model* m, int l) { return m->d_nrows + 2 * (1 + l); }

int cone_build_mb(scone_model* m, int32_t b, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                  cudaStream_t s) {
    const scone_complex* cx = m->cx;
    const int L = m->L;
    if (!m->x_clean) {
        SCONE_CUDA(cudaMemsetAsync(m->d_X, 0, (size_t)cx->E * m->mb * sizeof(float), s));
        m->x_clean = true;
    }
    ScopedProf prof(SCONE_K_CONE, s);
    if (!m->cone_clean) {                                  // once: afterwards every micro-batch clears exactly what it set
        for (int l = 0; l < L; ++l) {
            SCONE_CUDA(cudaMemsetAsync(m->d_bmGr[l], 0, m->bmg_bytes, s));
            SCONE_CUDA(cudaMemsetAsync(m->d_bmC[l], 0, m->bmg_bytes, s));
        }
    }
    m->cone_clean = false;                                 // until cone_clear_mb has run (an error return in between leaves bits set)
    if (scone_rows_cone(cx, b, last, m->d_bmC.data(), L, m->sum_off, m->d_overflow, s)) return 1;
    // flows -> X, live rows of H_1
    if (scone_rows_flows(cx, b, ptr, edge, val, m->d_X, nullptr, m->d_bmGr[0], false, true, s, m->d_bmC[0], m->sum_off)) return 1;
    for (int l = 0; l < L; ++l) {
        if (scone_compact_rows_summary(cx, b, m->d_bmGr[l], m->sum_off, m->d_rowsC[l], cone_n(m, l), m->d_tickets, s, m->d_prefG[l],
                                       m->row_cap))
            return 1;
        if (l + 1 < L)
            if (scone_rows_mark(cx, b, m->d_rowsC[l], cone_n(m, l), m->d_bmGr[l + 1], m->row_cap, s, true, m->sum_off, m->d_bmC[l + 1]))
                return 1;
    }
    return 0;
}

// end of a micro-batch: the bitmaps go back to all-zero (cost follows the cone, not E*b)
int cone_clear_mb(scone_model* m, int32_t b, cudaStream_t s) {
    ScopedProf prof(SCONE_K_CONE, s);
    std::vector<uint32_t*> bms(m->d_bmC);                 // [0] = the lowest cone level: contains every other bitmap of the step
    bms.insert(bms.end(), m->d_bmGr.begin(), m->d_bmGr.end());
    if (scone_clear_summary(m->cx, b, bms.data(), (int)bms.size(), 0, m->sum_off, s)) return 1;
    m->cone_clean = true;
    return 0;
}

int cone_forward_mb(scone_model* m, int32_t b, cudaStream_t s) {
    const scone_complex* cx = m->cx;
    int cin = 1;
    for (int l = 0; l < m->L; ++l) {
        const int cout = m->hidden[l];
        ScopedProf prof(l == 0 ? SCONE_K_LAYER0_FWD : SCONE_K_LAYER_FWD, s);
        const float *W0 = m->d_w + m->w_off[3 * l], *W1 = m->d_w + m->w_off[3 * l + 1], *W2 = m->d_w + m->w_off[3 * l + 2];
        int rc;
        if (l == 0)
            rc = scone_rows_layer0_forward(cx, m->act, b, cout, m->d_X, W0, W1, W2, m->d_cH[0], m->d_rowsC[0], cone_n(m, 0), nullptr,
                                           m->row_cap, m->d_overflow, s);
        else
            rc = scone_slab_forward_rows(cx, m->act, b, cin, cout, m->d_cH[l - 1], W0, W1, W2, m->d_cH[l], nullptr, m->d_rowsC[l],
                                         cone_n(m, l), scone_prof_row_counter(SCONE_K_LAYER_FWD), m->d_bmGr[l - 1], m->d_prefG[l - 1],
                                         m->row_cap, m->d_overflow, s);
        if (rc) return rc;
        cin = cout;
    }
    return 0;
}

int cone_readout(scone_model* m, int32_t b, const int32_t* last, float* logprobs, bool grad, const int32_t* tgt, const float* mask,
                 const float* cot, cudaStream_t s) {
    const scone_complex* cx = m->cx;
    const int L = m->L, CL = m->hidden[L - 1];
    const float* wout = m->d_w + m->w_off[3 * L];
    ScopedProf prof(SCONE_K_READOUT, s);
    if (scone_rows_readout_forward(cx, b, CL, m->d_cH[L - 1], wout, last, logprobs, m->d_bmGr[L - 1], m->d_prefG[L - 1], nullptr, nullptr, s))
        return 1;
    if (!grad) return 0;
    return scone_rows_readout_backward(cx, m->act, b, CL, m->d_cH[L - 1], wout, last, logprobs, tgt, mask, 1.f, m->d_cG[L - 1],
                                       cone_n(m, L - 1), m->row_cap, m->d_overflow, m->d_grad + m->w_off[3 * L], m->d_grad + m->n_params,
                                       m->d_grad + m->n_params + 1, 1, (float*)m->d_ws, m->d_bmGr[L - 1], m->d_prefG[L - 1],
                                       m->d_bmGr[L - 1], m->d_prefG[L - 1], s, cot);
}

int cone_backward_mb(scone_model* m, int32_t b, cudaStream_t s) {
    const scone_complex* cx = m->cx;
    const int L = m->L;
    const int a_cap = m->row_cap < m->a_cap ? m->row_cap : m->a_cap;
    // the forward consumed the tile counters of the lists it walked: zero the counter of every list again
    SCONE_CUDA(cudaMemset2DAsync(m->d_nrows + 1, 2 * sizeof(int), 0, sizeof(int), (size_t)(L + 1), s));
    for (int l = L - 1; l >= 1; --l) {
        ScopedProf prof(SCONE_K_LAYER_BWD, s);
        int rc = scone_rows_backward(cx, m->act, b, m->hidden[l - 1], m->hidden[l], m->d_cG[l], m->d_cH[l - 1], m->d_cG[l - 1], m->d_Abuf,
                                     m->d_w + m->w_off[3 * l], m->d_w + m->w_off[3 * l + 1], m->d_w + m->w_off[3 * l + 2], m->d_rowsC[l - 1],
                                     cone_n(m, l - 1), m->d_bmGr[l], m->d_bmGr[l - 1], a_cap, m->d_overflow, m->d_grad + m->w_off[3 * l], 1,
                                     (float*)m->d_ws, m->d_prefG[l], m->d_prefG[l - 1], true, s);
        if (rc) return rc;
    }
    ScopedProf prof(SCONE_K_LAYER0_BWD, s);
    return scone_rows_layer0_backward(cx, b, m->hidden[0], m->d_X, m->d_cG[0], m->d_rowsC[0], cone_n(m, 0), m->d_grad + m->w_off[0], 1,
                                      (float*)m->d_ws, m->row_cap, s);
}

// pipeline 3 over one micro-batch (arguments as unit_mb)
int cone_mb(scone_model* m, int32_t b, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last, float* logprobs,
            const int32_t* tgt, const float* mask, const float* cot, float* dflow, bool grad, cudaStream_t s) {
    int rc = cone_build_mb(m, b, ptr, edge, val, last, s);
    if (!rc) rc = cone_forward_mb(m, b, s);
    if (!rc) rc = cone_readout(m, b, last, logprobs, grad, tgt, mask, cot, s);
    if (!rc && grad) rc = cone_backward_mb(m, b, s);
    if (!rc && grad && dflow)                              // the live rows of layer 1 (cone & support), before the bitmaps are cleared
        rc = flow_grad_mb(m, b, ptr, edge, m->d_cG[0], nullptr, m->d_bmGr[0], m->d_prefG[0], dflow, s);
    if (!rc) rc = rows_clear_x(m, b, ptr, edge, val, s);
    if (!rc) rc = cone_clear_mb(m, b, s);
    return rc;
}

}  // namespace

extern "C" int scone_model_create(const scone_complex* cx, int32_t n_layers, const int32_t* hidden, int32_t micro_batch,
                                  scone_model** out) {
    SCONE_REQUIRE(out != nullptr, "scone_model_create: out is NULL");
    *out = nullptr;
    SCONE_REQUIRE(cx && hidden && n_layers >= 1 && micro_batch >= 1, "scone_model_create: bad arguments");
    SCONE_REQUIRE(!cx->host_only, "scone_model_create: index-only complex has no device arrays");
    SCONE_REQUIRE(cx->D <= SCONE_MAX_DEGREE, "scone_model_create: max node degree %d exceeds the supported maximum of %d", cx->D,
                  SCONE_MAX_DEGREE);
    scone_model* m = new scone_model();
    m->cx = cx;
    m->L = n_layers;
    m->mb = micro_batch;
    m->act = cx->model == SCONE_MODEL_EBLI ? SCONE_ACT_LEAKY_RELU : SCONE_ACT_TANH;
    m->hidden.assign(hidden, hidden + n_layers);
    int64_t off = 0;
    int cin = 1;
    for (int l = 0; l < n_layers; ++l) {
        const int c = hidden[l];
        if (!(c == 8 || c == 16 || c == 32 || c == 64)) {
            scone_set_error("scone_model_create: hidden width %d of layer %d unsupported (8, 16, 32 or 64)", c, l);
            delete m;
            return 2;
        }
        if (l > 0 && !(c == cin || c == 2 * cin || 2 * c == cin)) {
            scone_set_error("scone_model_create: consecutive widths %d -> %d unsupported (ratio must be 1/2, 1 or 2)", cin, c);
            delete m;
            return 2;
        }
        for (int k = 0; k < 3; ++k) {
            m->w_off.push_back(off);
            off += (int64_t)cin * c;
        }
        m->cmax = c > m->cmax ? c : m->cmax;
        cin = c;
    }
    m->w_off.push_back(off);
    off += cin;                               // W[-1]: [C_L][1]
    m->n_params = off;
    const size_t E = cx->E, mb = micro_batch;
    int rc = 0;
    auto alloc = [&](void** p, size_t bytes) {
        if (rc) return;
        cudaError_t e = cudaMalloc(p, bytes ? bytes : 4);
        if (e != cudaSuccess) {
            scone_set_error("scone_model_create: cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
            rc = 1;
        }
    };
    alloc((void**)&m->d_w, off * sizeof(float));
    alloc((void**)&m->d_m, off * sizeof(float));
    alloc((void**)&m->d_v, off * sizeof(float));
    alloc((void**)&m->d_grad, (off + 2) * sizeof(float));
    m->d_H.assign(n_layers, nullptr);
    m->d_G.assign(n_layers, nullptr);
    m->d_occH.assign(n_layers, nullptr);
    m->d_occG.assign(n_layers, nullptr);
    // row ids are 32-bit: unsigned (E * mb < 2^32) in the compact trajectory-major pipelines, E * mb < 2^31 elsewhere
    m->rows_ok = scone_rows_supported(cx, n_layers, hidden) && E * mb < ((size_t)1 << 32);
    // the cone kernel stages at most 2048 edges per trajectory and level in shared memory: the top level alone has up to D * D
    // edges, so complexes with very high degrees start on the whole-support pipeline (the cone would report an overflow)
    m->pipeline = m->rows_ok ? ((cx->D <= 32 || E * mb >= ((size_t)1 << 31)) ? 3 : 2) : 0;
    if (scone_fused_supported(cx, n_layers, hidden)) {     // measured static bounds decide; nullptr = cones too large for the tables
        if (scone_fused_create(cx, n_layers, hidden[0], micro_batch, m->n_params, &m->fused)) {
            delete m;
            return 1;
        }
        if (m->fused) m->pipeline = 4;
    }
    if (m->pipeline != 4 && !m->rows_ok && E * mb >= ((size_t)1 << 31)) {
        scone_set_error("scone_model_create: E * micro_batch = %zu needs the row-list pipeline (widths 16 / 32, E * micro_batch < 2^32)", E * mb);
        delete m;
        return 2;
    }
    int64_t ws = scone_readout_workspace_bytes(micro_batch, m->cmax);
    if (scone_rows_dw_workspace_bytes(m->cmax, m->cmax) > ws) ws = scone_rows_dw_workspace_bytes(m->cmax, m->cmax);
    cin = 1;
    for (int l = 0; l < n_layers; ++l) {
        int64_t w = scone_layer_backward_workspace_bytes(cin, hidden[l]);
        ws = w > ws ? w : ws;
        cin = hidden[l];
    }
    alloc(&m->d_ws, ws);
    alloc((void**)&m->d_logp, mb * (size_t)(cx->D > 0 ? cx->D : 1) * sizeof(float));
    if (!rc) {
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        cudaStreamCreateWithPriority(&m->compute, cudaStreamNonBlocking, prio_hi);
        cudaEventCreateWithFlags(&m->ev_fork, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&m->ev_join, cudaEventDisableTiming);
        cudaMemset(m->d_w, 0, off * sizeof(float));
        cudaMemset(m->d_m, 0, off * sizeof(float));
        cudaMemset(m->d_v, 0, off * sizeof(float));
        cudaMemset(m->d_grad, 0, (off + 2) * sizeof(float));
    }
    if (!rc) rc = ensure_buffers(m);
    if (rc) {
        scone_model_destroy(m);
        return rc;
    }
    *out = m;
    return 0;
}

extern "C" int scone_model_destroy(scone_model* m) {
    if (!m) return 0;
    cudaFree(m->d_w); cudaFree(m->d_m); cudaFree(m->d_v); cudaFree(m->d_grad); cudaFree(m->d_X);
    for (float* p : m->d_H) cudaFree(p);
    for (uint8_t* p : m->d_occH) cudaFree(p);
    for (uint8_t* p : m->d_occG) cudaFree(p);
    cudaFree(m->d_occS); cudaFree(m->d_occX); cudaFree(m->d_bmX); cudaFree(m->d_bmG);
    for (uint32_t* p : m->d_bmH) cudaFree(p);
    for (uint32_t* p : m->d_bmGr) cudaFree(p);
    for (uint32_t* p : m->d_prefH) cudaFree(p);
    for (uint32_t* p : m->d_prefG) cudaFree(p);
    for (float* p : m->d_cH) cudaFree(p);
    for (float* p : m->d_cG) cudaFree(p);
    for (uint32_t* p : m->d_rowsC) cudaFree(p);
    for (uint32_t* p : m->d_bmC) cudaFree(p);
    cudaFree(m->d_rows); cudaFree(m->d_nrows); cudaFree(m->d_overflow); cudaFree(m->d_tickets); cudaFree(m->d_Abuf);
    for (float* p : m->d_G) cudaFree(p);
    cudaFree(m->d_ws); cudaFree(m->d_logp);
    scone_fused_destroy(m->fused);
    if (m->compute) cudaStreamDestroy(m->compute);
    if (m->ev_fork) cudaEventDestroy(m->ev_fork);
    if (m->ev_join) cudaEventDestroy(m->ev_join);
    if (m->copy) cudaStreamDestroy(m->copy);
    if (m->ev_copy0) cudaEventDestroy(m->ev_copy0);
    if (m->ev_plan_done) cudaEventDestroy(m->ev_plan_done);
    for (auto e : m->ev_part) if (e) cudaEventDestroy(e);
    cudaFree(m->d_ptr); cudaFree(m->d_edge); cudaFree(m->d_last); cudaFree(m->d_tgt); cudaFree(m->d_val);
    cudaFree(m->d_mask); cudaFree(m->d_logp_all); cudaFree(m->d_nn); cudaFree(m->d_acc); cudaFree(m->d_cot); cudaFree(m->d_dflow);
    cudaFree(m->d_choice); cudaFree(m->d_rand); cudaFree(m->d_evalf);
    delete m;
    return 0;
}

extern "C" int64_t scone_model_num_params(const scone_model* m) { return m ? m->n_params : -1; }
extern "C" int scone_model_set_pipeline(scone_model* m, int32_t which) {
    SCONE_REQUIRE(m != nullptr && which >= 0 && which <= 4,
                  "scone_model_set_pipeline: 0 (unit kernels, byte flags), 1 (row lists, dense tensors), 2 (row lists, compact tensors), "
                  "3 (compact row lists over the readout cone) or 4 (trajectory-fused kernels)");
    SCONE_REQUIRE(which != 4 || m->fused != nullptr,
                  "scone_model_set_pipeline: the fused pipeline needs one uniform hidden width of 16 or 32, at most 3 layers, and cones that fit "
                  "its shared-memory tables");
    SCONE_REQUIRE(which == 0 || which == 4 || m->rows_ok, "scone_model_set_pipeline: the row-list pipelines need hidden widths in {16, 32}");
    SCONE_REQUIRE(which >= 3 || (size_t)m->cx->E * m->mb < ((size_t)1 << 31),
                  "scone_model_set_pipeline: E * micro_batch >= 2^31 runs on pipelines 3 / 4 only");
    SCONE_REQUIRE(which != 3 || (size_t)m->cx->E * m->mb < ((size_t)1 << 32), "scone_model_set_pipeline: pipeline 3 needs E * micro_batch < 2^32");
    const int old = m->pipeline;
    m->pipeline = which;
    if (ensure_buffers(m)) {
        m->pipeline = old;
        return 1;
    }
    return 0;
}
extern "C" int scone_model_get_pipeline(const scone_model* m) { return m ? m->pipeline : -1; }
extern "C" float* scone_model_weights_dev(scone_model* m) { return m ? m->d_w : nullptr; }
extern "C" float* scone_model_grads_dev(scone_model* m) { return m ? m->d_grad : nullptr; }

extern "C" int scone_model_set_weights(scone_model* m, const float* w) {
    SCONE_REQUIRE(m && w, "scone_model_set_weights: NULL argument");
    SCONE_CUDA(cudaMemcpy(m->d_w, w, m->n_params * sizeof(float), cudaMemcpyHostToDevice));
    SCONE_CUDA(cudaMemset(m->d_m, 0, m->n_params * sizeof(float)));
    SCONE_CUDA(cudaMemset(m->d_v, 0, m->n_params * sizeof(float)));
    return 0;
}

extern "C" int scone_model_get_weights(const scone_model* m, float* w) {
    SCONE_REQUIRE(m && w, "scone_model_get_weights: NULL argument");
    SCONE_CUDA(cudaMemcpy(w, m->d_w, m->n_params * sizeof(float), cudaMemcpyDeviceToHost));
    return 0;
}

// The caller's stream is forked into the model's highest-priority compute stream (and joined back): block scheduling then
// prefers the library's kernels over work that other streams of the process have queued.
static int fork_to_compute(scone_model* m, void* user_st) {
    SCONE_CUDA(cudaEventRecord(m->ev_fork, as_stream(user_st)));
    SCONE_CUDA(cudaStreamWaitEvent(m->compute, m->ev_fork, 0));
    return 0;
}
static int join_from_compute(scone_model* m, void* user_st) {
    SCONE_CUDA(cudaEventRecord(m->ev_join, m->compute));
    SCONE_CUDA(cudaStreamWaitEvent(as_stream(user_st), m->ev_join, 0));
    return 0;
}

// A failed launch inside a micro-batch leaves X / the cone bitmaps dirty: every model-level call leaves through this exit, which
// marks them so (the next call re-clears) and still joins the caller's stream to the compute stream.
static int finish_call(scone_model* m, int rc, void* user_st) {
    if (rc) {
        m->x_clean = false;
        m->cone_clean = false;
    }
    const int jr = join_from_compute(m, user_st);
    return rc ? rc : jr;
}

// pipeline 4: the micro-batch is walked in chunks the program arena was sized for (scone_fused_create)
static int fused_call(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                      float* logprobs, const int32_t* tgt, const float* mask, const float* cot, float* dflow, bool grad, cudaStream_t s) {
    const int step = m->fused->chunk < m->mb ? m->fused->chunk : m->mb;
    for (int32_t off = 0; off < B; off += step) {
        const int32_t b = B - off < step ? B - off : step;
        int rc = scone_fused_run(m->cx, m->fused, m->act, b, ptr + off, edge, val, last + off, m->d_w, m->w_off.data(),
                                 logprobs ? logprobs + (size_t)off * m->cx->D : nullptr, grad && !cot ? tgt + off : nullptr,
                                 grad && !cot ? mask + off : nullptr, grad ? m->d_grad : nullptr, m->d_overflow, g_scone_prof, s,
                                 grad && cot ? cot + (size_t)off * m->cx->D : nullptr, grad && cot ? dflow : nullptr);
        if (rc) return rc;
    }
    return 0;
}

// pipeline 4 behind a *_host entry point, batch within one arena chunk: the flow arrays (all but a few hundred KB of the H2D bytes)
// are copied in four parts on a copy stream and every part is planned as soon as it has landed — the copy of part k + 1 runs under the
// plan kernels of part k; one compute launch over the whole batch at the end.  ptr / last / tgt / mask: already enqueued on s.
static bool fused_host_overlap_ok(const scone_model* m, int32_t B, int64_t nnz) {
    return m->pipeline == 4 && m->fused && B >= 512 && B <= m->fused->chunk && B <= m->mb && nnz >= (1 << 13);
}

// cot_dev != NULL (grad): the VJP seeded with these staged cotangents; count_add is added to the count slot.
static int fused_host_overlapped(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, float* logprobs_dev,
                                 bool grad, int32_t zero_first, cudaStream_t s, const float* cot_dev = nullptr, float count_add = 0.f) {
    // parts of >= 4096 trajectories, at most 4: a part's first plan tier runs as soon as its flows have landed; the later tiers (a few
    // heavy trajectories, each launch as long as its slowest one) run once over all parts.  Small batches are planned in one piece
    // (their copy is short, and steps enqueued back to back copy under the previous compute)
    constexpr int kMaxParts = 4;
    const int kParts = B >= 4 * 4096 ? 4 : (B >= 2 * 4096 ? 2 : 1);
    if (!m->copy) {
        SCONE_CUDA(cudaStreamCreateWithFlags(&m->copy, cudaStreamNonBlocking));
        SCONE_CUDA(cudaEventCreateWithFlags(&m->ev_copy0, cudaEventDisableTiming));
        SCONE_CUDA(cudaEventCreateWithFlags(&m->ev_plan_done, cudaEventDisableTiming));
        for (auto& e : m->ev_part) SCONE_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    // The flow staging buffers are read by the plan kernels only.  If their last user was the previous overlapped call (exactly one
    // ensure_staging since: this call's), they are free as soon as ITS plan kernels are done — the copy of this batch then runs
    // under that call's compute kernel when the caller enqueues steps back to back.  Otherwise: once everything enqueued on s so
    // far has run (every call joins its kernels into s).
    if (m->plan_done_epoch >= 0 && m->plan_done_epoch == m->staging_epoch - 1) {
        SCONE_CUDA(cudaStreamWaitEvent(m->copy, m->ev_plan_done, 0));
    } else {
        SCONE_CUDA(cudaEventRecord(m->ev_copy0, s));
        SCONE_CUDA(cudaStreamWaitEvent(m->copy, m->ev_copy0, 0));
    }
    int32_t b0[kMaxParts + 1];
    for (int k = 0; k <= kParts; ++k) b0[k] = (int32_t)((int64_t)B * k / kParts);
    for (int k = 0; k < kParts; ++k) {
        const int64_t q0 = ptr[b0[k]], q1 = ptr[b0[k + 1]];
        if (q1 > q0) {
            SCONE_CUDA(cudaMemcpyAsync(m->d_edge + q0, edge + q0, (q1 - q0) * sizeof(int32_t), cudaMemcpyHostToDevice, m->copy));
            SCONE_CUDA(cudaMemcpyAsync(m->d_val + q0, val + q0, (q1 - q0) * sizeof(float), cudaMemcpyHostToDevice, m->copy));
        }
        SCONE_CUDA(cudaEventRecord(m->ev_part[k], m->copy));
    }
    if (fork_to_compute(m, (void*)s)) return 1;
    cudaStream_t c = m->compute;
    if (grad && zero_first) SCONE_CUDA(cudaMemsetAsync(m->d_grad, 0, (m->n_params + 2) * sizeof(float), c));
    if (grad && cot_dev && count_add != 0.f && scone_add_scalar_launch(m->d_grad + m->n_params + 1, count_add, c)) return finish_call(m, 1, (void*)s);
    int rc = scone_fused_begin(m->fused, c);
    for (int k = 0; k < kParts && !rc; ++k) {
        SCONE_CUDA(cudaStreamWaitEvent(c, m->ev_part[k], 0));
        rc = scone_fused_plan_part(m->cx, m->fused, b0[k], b0[k + 1] - b0[k], m->d_ptr, m->d_edge, m->d_val, m->d_last, m->d_overflow, c,
                                   kParts > 1);
    }
    if (!rc && kParts > 1) rc = scone_fused_plan_finish(m->cx, m->fused, B, m->d_ptr, m->d_edge, m->d_val, m->d_last, m->d_overflow, c);
    if (!rc) {
        SCONE_CUDA(cudaEventRecord(m->ev_plan_done, c));
        m->plan_done_epoch = m->staging_epoch;
    } else {
        m->plan_done_epoch = -1;
    }
    if (!rc)
        rc = scone_fused_compute(m->cx, m->fused, m->act, B, m->d_w, m->w_off.data(), logprobs_dev, grad && !cot_dev ? m->d_tgt : nullptr,
                                 grad && !cot_dev ? m->d_mask : nullptr, grad ? m->d_grad : nullptr, g_scone_prof, c, grad ? cot_dev : nullptr);
    return finish_call(m, rc, (void*)s);
}

// Forward (grad = false: log-probs to logprobs [B][D]) or loss + gradient (grad = true: into d_grad, cleared first if zero_first).
// cot != NULL (grad): the VJP — the gradient is seeded with the cotangent rows [B][D] instead of tgt / mask, and count_add is added to
// the count slot; dflow != NULL (with cot): dL/dx at the flow entries [ptr[0], ptr[B]) too, indexed like val.
static int run_batch(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                     float* logprobs, const int32_t* tgt, const float* mask, bool grad, int32_t zero_first, void* user_st,
                     const float* cot = nullptr, float count_add = 0.f, float* dflow = nullptr) {
    if (fork_to_compute(m, user_st)) return 1;
    cudaStream_t s = m->compute;
    if (grad && zero_first) SCONE_CUDA(cudaMemsetAsync(m->d_grad, 0, (m->n_params + 2) * sizeof(float), s));
    if (grad && cot && count_add != 0.f && scone_add_scalar_launch(m->d_grad + m->n_params + 1, count_add, s)) return finish_call(m, 1, user_st);
    const int pl = m->pipeline;
    if (pl == 4) return finish_call(m, fused_call(m, B, ptr, edge, val, last, logprobs, tgt, mask, cot, dflow, grad, s), user_st);
    auto step = pl == 3 ? cone_mb : pl >= 1 ? rows_mb : unit_mb;
    int rc = 0;
    for (int32_t off = 0; off < B && !rc; off += m->mb) {
        const int32_t b = B - off < m->mb ? B - off : m->mb;
        rc = step(m, b, ptr + off, edge, val, last + off, grad ? m->d_logp : logprobs + (size_t)off * m->cx->D,
                  grad && !cot ? tgt + off : nullptr, grad && !cot ? mask + off : nullptr, grad && cot ? cot + (size_t)off * m->cx->D : nullptr,
                  grad && cot ? dflow : nullptr, grad, s);
    }
    return finish_call(m, rc, user_st);
}

extern "C" int scone_model_forward_dev(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                       const int32_t* last, float* logprobs, void* user_st) {
    SCONE_REQUIRE(m && ptr && last && logprobs && B >= 0, "scone_model_forward_dev: bad arguments");
    return run_batch(m, B, ptr, edge, val, last, logprobs, nullptr, nullptr, false, 0, user_st);
}

extern "C" int scone_model_loss_grad_dev(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                         const int32_t* last, const int32_t* tgt, const float* mask, int32_t zero_first,
                                         void* user_st) {
    SCONE_REQUIRE(m && ptr && last && tgt && mask && B >= 0, "scone_model_loss_grad_dev: bad arguments");
    return run_batch(m, B, ptr, edge, val, last, nullptr, tgt, mask, true, zero_first, user_st);
}

extern "C" int scone_model_forward_host(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                        const int32_t* last, float* logprobs_out, void* st) {
    SCONE_REQUIRE(m && ptr && last && logprobs_out && B >= 0, "scone_model_forward_host: bad arguments");
    if (B == 0) return 0;
    cudaStream_t s = as_stream(st);
    const bool overlap = fused_host_overlap_ok(m, B, ptr[B]);
    int rc = stage_host_inputs(m, B, ptr, last, nullptr, nullptr, nullptr, edge, val, !overlap, s);
    if (rc) return rc;
    if (overlap) rc = fused_host_overlapped(m, B, ptr, edge, val, m->d_logp_all, false, 0, s);
    else rc = scone_model_forward_dev(m, B, m->d_ptr, m->d_edge, m->d_val, m->d_last, m->d_logp_all, st);
    if (rc) return rc;
    SCONE_CUDA(cudaMemcpyAsync(logprobs_out, m->d_logp_all, (size_t)B * m->cx->D * sizeof(float), cudaMemcpyDeviceToHost, s));
    return report_overflow(m, s, "scone_model_forward_host");
}

extern "C" int scone_accuracy_dev(int32_t B, int32_t D, const float* logprobs, const int32_t* n_nbrs, const int32_t* target_idx,
                                  const float* mask, int32_t* out, void* st) {
    SCONE_REQUIRE(B >= 0 && D >= 1 && out && (B == 0 || (logprobs && n_nbrs && target_idx && mask)), "scone_accuracy_dev: bad arguments");
    return scone_accuracy_launch(B, D, logprobs, n_nbrs, target_idx, mask, out, as_stream(st));
}

extern "C" int scone_model_accuracy_host(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                         const int32_t* last, const int32_t* n_nbrs, const int32_t* tgt, const float* mask,
                                         int32_t* out_host, void* st) {
    SCONE_REQUIRE(m && out_host && B >= 0 && (B == 0 || (ptr && last && n_nbrs && tgt && mask)), "scone_model_accuracy_host: bad arguments");
    out_host[0] = out_host[1] = 0;
    if (B == 0) return 0;
    cudaStream_t s = as_stream(st);
    int rc = stage_host_inputs(m, B, ptr, last, n_nbrs, tgt, mask, edge, val, true, s);
    if (rc) return rc;
    rc = scone_model_forward_dev(m, B, m->d_ptr, m->d_edge, m->d_val, m->d_last, m->d_logp_all, st);
    if (rc) return rc;
    rc = scone_accuracy_launch(B, m->cx->D, m->d_logp_all, m->d_nn, m->d_tgt, m->d_mask, m->d_acc, s);
    if (rc) return rc;
    SCONE_CUDA(cudaMemcpyAsync(out_host, m->d_acc, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    return report_overflow(m, s, "scone_model_accuracy_host");
}

// ---- evaluation without the log-probs leaving the device (scone_trajectory_model.py:42-56, 59-71, 73-108) --------------------
// scone_model_eval_host: forward over B trajectories from HOST buffers; the log-probs stay in the model's device buffer (valid until
// the next model-level call).  Optional outputs, each computed on the device:
//   choice_out [B]     argmax prediction per trajectory (n_nbrs masking, first maximum)            (needs n_nbrs)
//   acc_out [2]        correct predictions, masked trajectories                                      (needs n_nbrs, target_idx, mask)
//   nll_out [2]        sum of -mask * logprob[target], sum of mask                                   (needs target_idx, mask)
extern "C" int scone_model_eval_host(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                     const int32_t* last, const int32_t* n_nbrs, const int32_t* tgt, const float* mask,
                                     int32_t* choice_out, int32_t* acc_out, float* nll_out, void* st) {
    SCONE_REQUIRE(m && B >= 0 && (B == 0 || (ptr && last)), "scone_model_eval_host: bad arguments");
    SCONE_REQUIRE(!choice_out || n_nbrs, "scone_model_eval_host: choice_out needs n_nbrs");
    SCONE_REQUIRE(!acc_out || (n_nbrs && tgt && mask), "scone_model_eval_host: acc_out needs n_nbrs, target_idx and mask");
    SCONE_REQUIRE(!nll_out || (tgt && mask), "scone_model_eval_host: nll_out needs target_idx and mask");
    if (acc_out) acc_out[0] = acc_out[1] = 0;
    if (nll_out) nll_out[0] = nll_out[1] = 0.f;
    m->eval_B = 0;
    if (B == 0) return 0;
    cudaStream_t s = as_stream(st);
    int rc = stage_host_inputs(m, B, ptr, last, n_nbrs, tgt, mask, edge, val, true, s);
    if (rc) return rc;
    if (!m->d_choice || m->cap_choice < B) {
        cudaFree(m->d_choice); cudaFree(m->d_rand);
        m->d_choice = m->d_rand = nullptr;
        SCONE_CUDA(cudaMalloc((void**)&m->d_choice, (size_t)m->cap_B * sizeof(int32_t)));
        SCONE_CUDA(cudaMalloc((void**)&m->d_rand, (size_t)m->cap_B * sizeof(int32_t)));
        m->cap_choice = m->cap_B;
    }
    if (!m->d_evalf) SCONE_CUDA(cudaMalloc((void**)&m->d_evalf, 4 * sizeof(float)));
    rc = scone_model_forward_dev(m, B, m->d_ptr, m->d_edge, m->d_val, m->d_last, m->d_logp_all, st);
    if (rc) return rc;
    const int D = m->cx->D;
    if (choice_out) {
        if (scone_predict_launch(B, D, m->d_logp_all, m->d_nn, m->d_choice, s)) return 1;
        SCONE_CUDA(cudaMemcpyAsync(choice_out, m->d_choice, B * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    }
    if (acc_out) {
        if (scone_accuracy_launch(B, D, m->d_logp_all, m->d_nn, m->d_tgt, m->d_mask, m->d_acc, s)) return 1;
        SCONE_CUDA(cudaMemcpyAsync(acc_out, m->d_acc, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    }
    if (nll_out) {
        if (scone_nll_launch(B, D, m->d_logp_all, m->d_tgt, m->d_mask, m->d_evalf, s)) return 1;
        SCONE_CUDA(cudaMemcpyAsync(nll_out, m->d_evalf, 2 * sizeof(float), cudaMemcpyDeviceToHost, s));
    }
    rc = report_overflow(m, s, "scone_model_eval_host");
    if (rc) return rc;
    m->eval_B = B;
    return 0;
}

// Two-target comparison (scone_trajectory_model.py:95-108) on the log-probs the last scone_model_eval_host left on the device (same B,
// n_nbrs and mask as that call): out[0] = rows with true > random, out[1] = rows with true == random, over mask != 0.
extern "C" int scone_model_two_target_host(scone_model* m, int32_t B, const int32_t* true_idx, const int32_t* rand_idx, int32_t* out, void* st) {
    SCONE_REQUIRE(m && out && B >= 0 && (B == 0 || (true_idx && rand_idx)), "scone_model_two_target_host: bad arguments");
    SCONE_REQUIRE(B == m->eval_B, "scone_model_two_target_host: call scone_model_eval_host (with n_nbrs and mask) on the same %d trajectories first", B);
    out[0] = out[1] = 0;
    if (B == 0) return 0;
    cudaStream_t s = as_stream(st);
    SCONE_CUDA(cudaMemcpyAsync(m->d_tgt, true_idx, B * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    SCONE_CUDA(cudaMemcpyAsync(m->d_rand, rand_idx, B * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    if (scone_two_target_launch(B, m->cx->D, m->d_logp_all, m->d_nn, m->d_tgt, m->d_rand, m->d_mask, m->d_acc, s)) return 1;
    SCONE_CUDA(cudaMemcpyAsync(out, m->d_acc, 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    SCONE_CUDA(cudaStreamSynchronize(s));
    return 0;
}

extern "C" int scone_model_loss_grad_host(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                          const int32_t* last, const int32_t* tgt, const float* mask, int32_t zero_first,
                                          void* st) {
    SCONE_REQUIRE(m && ptr && last && tgt && mask && B >= 0, "scone_model_loss_grad_host: bad arguments");
    cudaStream_t s = as_stream(st);
    const bool overlap = fused_host_overlap_ok(m, B, B > 0 ? ptr[B] : 0);
    int rc = stage_host_inputs(m, B, ptr, last, nullptr, tgt, mask, edge, val, !overlap, s);
    if (rc) return rc;
    if (overlap) return fused_host_overlapped(m, B, ptr, edge, val, nullptr, true, zero_first, s);
    // (B == 0: only ptr was staged; the call still clears the gradient buffer when zero_first is set)
    return scone_model_loss_grad_dev(m, B, m->d_ptr, m->d_edge, m->d_val, m->d_last, m->d_tgt, m->d_mask, zero_first, st);
}

extern "C" int scone_model_vjp_dev(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                                   const float* cot, float count_add, int32_t zero_first, void* user_st) {
    SCONE_REQUIRE(m && ptr && last && B >= 0, "scone_model_vjp_dev: bad arguments");
    SCONE_REQUIRE(cot || B == 0, "scone_model_vjp_dev: cot is NULL");
    return run_batch(m, B, ptr, edge, val, last, nullptr, nullptr, nullptr, true, zero_first, user_st, cot, count_add);
}

extern "C" int scone_model_vjp_host(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                                    const float* cot, float count_add, int32_t zero_first, void* st) {
    SCONE_REQUIRE(m && ptr && last && B >= 0, "scone_model_vjp_host: bad arguments");
    SCONE_REQUIRE(cot || B == 0, "scone_model_vjp_host: cot is NULL");
    cudaStream_t s = as_stream(st);
    const bool overlap = fused_host_overlap_ok(m, B, B > 0 ? ptr[B] : 0);
    int rc = stage_host_inputs(m, B, ptr, last, nullptr, nullptr, nullptr, edge, val, !overlap, s);
    if (!rc) rc = stage_cot(m, B, cot, s);
    if (rc) return rc;
    if (overlap) return fused_host_overlapped(m, B, ptr, edge, val, nullptr, true, zero_first, s, m->d_cot, count_add);
    return scone_model_vjp_dev(m, B, m->d_ptr, m->d_edge, m->d_val, m->d_last, B > 0 ? m->d_cot : nullptr, count_add, zero_first, st);
}

extern "C" int scone_model_vjp_flows_dev(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                         const int32_t* last, const float* cot, float count_add, int32_t zero_first, float* dflow,
                                         void* user_st) {
    SCONE_REQUIRE(m && ptr && last && B >= 0, "scone_model_vjp_flows_dev: bad arguments");
    SCONE_REQUIRE((cot && dflow) || B == 0, "scone_model_vjp_flows_dev: cot or dflow is NULL");
    return run_batch(m, B, ptr, edge, val, last, nullptr, nullptr, nullptr, true, zero_first, user_st, cot, count_add, dflow);
}

// the plain staged path (no part-wise copy overlap): dflow is a host output, so the call ends with a stream synchronise anyway
extern "C" int scone_model_vjp_flows_host(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val,
                                          const int32_t* last, const float* cot, float count_add, int32_t zero_first, float* dflow,
                                          void* st) {
    SCONE_REQUIRE(m && ptr && last && B >= 0, "scone_model_vjp_flows_host: bad arguments");
    SCONE_REQUIRE((cot && dflow) || B == 0, "scone_model_vjp_flows_host: cot or dflow is NULL");
    cudaStream_t s = as_stream(st);
    const int64_t p0 = B > 0 ? ptr[0] : 0, nnz = B > 0 ? ptr[B] : 0;
    int rc = stage_host_inputs(m, B, ptr, last, nullptr, nullptr, nullptr, edge, val, true, s);
    if (!rc) rc = stage_cot(m, B, cot, s);
    if (rc) return rc;
    if (nnz > m->cap_dflow) {
        cudaFree(m->d_dflow);
        m->d_dflow = nullptr;
        m->cap_dflow = 0;
        const int64_t cap = nnz + nnz / 4 + 16;
        SCONE_CUDA(cudaMalloc((void**)&m->d_dflow, cap * sizeof(float)));
        m->cap_dflow = cap;
    }
    rc = scone_model_vjp_flows_dev(m, B, m->d_ptr, m->d_edge, m->d_val, m->d_last, B > 0 ? m->d_cot : nullptr, count_add, zero_first,
                                   m->d_dflow, st);
    if (rc) return rc;
    if (nnz > p0) SCONE_CUDA(cudaMemcpyAsync(dflow + p0, m->d_dflow + p0, (size_t)(nnz - p0) * sizeof(float), cudaMemcpyDeviceToHost, s));
    SCONE_CUDA(cudaStreamSynchronize(s));
    return 0;
}

extern "C" int scone_model_read_grads_async(scone_model* m, float* out_pinned, void* st) {
    SCONE_REQUIRE(m && out_pinned, "scone_model_read_grads_async: NULL argument");
    SCONE_CUDA(cudaMemcpyAsync(out_pinned, m->d_grad, (m->n_params + 2) * sizeof(float), cudaMemcpyDeviceToHost, as_stream(st)));
    return 0;
}

extern "C" int scone_model_read_grads(scone_model* m, float* out, void* st) {
    SCONE_REQUIRE(m && out, "scone_model_read_grads: NULL argument");
    cudaStream_t s = as_stream(st);
    SCONE_CUDA(cudaMemcpyAsync(out, m->d_grad, (m->n_params + 2) * sizeof(float), cudaMemcpyDeviceToHost, s));
    return report_overflow(m, s, "scone_model_read_grads");
}

// ---- planned sets (pipeline 4): plan a dataset once, run only the compute kernel on rows of it every step ----------------------
extern "C" int scone_model_plan_dev(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                                    void* user_st) {
    SCONE_REQUIRE(m && B >= 0 && (B == 0 || (ptr && last)), "scone_model_plan_dev: bad arguments");
    SCONE_REQUIRE(m->fused != nullptr, "scone_model_plan_dev: planned sets need the fused pipeline (uniform width 16 / 32, <= 3 layers)");
    if (fork_to_compute(m, user_st)) return 1;
    const int rc = scone_fused_plan_set(m->cx, m->fused, B, ptr, edge, val, last, m->d_overflow, m->compute);
    return finish_call(m, rc, user_st);
}

extern "C" int scone_model_plan_host(scone_model* m, int32_t B, const int32_t* ptr, const int32_t* edge, const float* val, const int32_t* last,
                                     void* st) {
    SCONE_REQUIRE(m && B >= 0 && (B == 0 || (ptr && last)), "scone_model_plan_host: bad arguments");
    SCONE_REQUIRE(m->fused != nullptr, "scone_model_plan_host: planned sets need the fused pipeline (uniform width 16 / 32, <= 3 layers)");
    // the plan reads its inputs only while it is built: the staging buffers of the *_host entry points serve
    int rc = stage_host_inputs(m, B, ptr, last, nullptr, nullptr, nullptr, edge, val, true, as_stream(st));
    if (rc) return rc;
    rc = scone_model_plan_dev(m, B, m->d_ptr, m->d_edge, m->d_val, m->d_last, st);
    if (rc) return rc;
    return scone_model_check_overflow(m, st);
}

extern "C" int scone_model_loss_grad_planned_dev(scone_model* m, int32_t n, const int32_t* rows_dev, const int32_t* tgt_dev, const float* mask_dev,
                                                 int32_t zero_first, void* user_st) {
    SCONE_REQUIRE(m && n >= 0 && (n == 0 || (tgt_dev && mask_dev)), "scone_model_loss_grad_planned_dev: bad arguments");
    SCONE_REQUIRE(m->fused != nullptr, "scone_model_loss_grad_planned_dev: no fused pipeline");
    if (fork_to_compute(m, user_st)) return 1;
    cudaStream_t s = m->compute;
    if (zero_first) SCONE_CUDA(cudaMemsetAsync(m->d_grad, 0, (m->n_params + 2) * sizeof(float), s));
    const int rc = scone_fused_run_planned(m->cx, m->fused, m->act, n, rows_dev, m->d_w, m->w_off.data(), nullptr, tgt_dev, mask_dev, m->d_grad,
                                           g_scone_prof, s);
    return finish_call(m, rc, user_st);
}

extern "C" int scone_model_loss_grad_planned_host(scone_model* m, int32_t n, const int32_t* rows, const int32_t* tgt, const float* mask,
                                                  int32_t zero_first, void* st) {
    SCONE_REQUIRE(m && n >= 0 && (n == 0 || (tgt && mask)), "scone_model_loss_grad_planned_host: bad arguments");
    cudaStream_t s = as_stream(st);
    int rc = ensure_staging(m, n, 0);
    if (rc) return rc;
    if (n) {
        if (rows) SCONE_CUDA(cudaMemcpyAsync(m->d_nn, rows, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        SCONE_CUDA(cudaMemcpyAsync(m->d_tgt, tgt, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        SCONE_CUDA(cudaMemcpyAsync(m->d_mask, mask, n * sizeof(float), cudaMemcpyHostToDevice, s));
    }
    return scone_model_loss_grad_planned_dev(m, n, rows ? m->d_nn : nullptr, m->d_tgt, m->d_mask, zero_first, st);
}

extern "C" int scone_model_vjp_planned_dev(scone_model* m, int32_t n, const int32_t* rows_dev, const float* cot_dev, float count_add,
                                           int32_t zero_first, void* user_st) {
    SCONE_REQUIRE(m && n >= 0, "scone_model_vjp_planned_dev: bad arguments");
    SCONE_REQUIRE(cot_dev || n == 0, "scone_model_vjp_planned_dev: cot is NULL");
    SCONE_REQUIRE(m->fused != nullptr, "scone_model_vjp_planned_dev: no fused pipeline");
    if (fork_to_compute(m, user_st)) return 1;
    cudaStream_t s = m->compute;
    if (zero_first) SCONE_CUDA(cudaMemsetAsync(m->d_grad, 0, (m->n_params + 2) * sizeof(float), s));
    int rc = count_add != 0.f ? scone_add_scalar_launch(m->d_grad + m->n_params + 1, count_add, s) : 0;
    if (!rc)
        rc = scone_fused_run_planned(m->cx, m->fused, m->act, n, rows_dev, m->d_w, m->w_off.data(), nullptr, nullptr, nullptr, m->d_grad,
                                     g_scone_prof, s, cot_dev);
    return finish_call(m, rc, user_st);
}

extern "C" int scone_model_vjp_planned_host(scone_model* m, int32_t n, const int32_t* rows, const float* cot, float count_add,
                                            int32_t zero_first, void* st) {
    SCONE_REQUIRE(m && n >= 0, "scone_model_vjp_planned_host: bad arguments");
    SCONE_REQUIRE(cot || n == 0, "scone_model_vjp_planned_host: cot is NULL");
    SCONE_REQUIRE(m->fused != nullptr, "scone_model_vjp_planned_host: no fused pipeline");
    cudaStream_t s = as_stream(st);
    int rc = ensure_staging(m, n, 0);
    if (!rc) rc = stage_cot(m, n, cot, s);
    if (rc) return rc;
    if (n && rows) SCONE_CUDA(cudaMemcpyAsync(m->d_nn, rows, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    return scone_model_vjp_planned_dev(m, n, rows ? m->d_nn : nullptr, n ? m->d_cot : nullptr, count_add, zero_first, st);
}

extern "C" int scone_model_forward_planned_host(scone_model* m, int32_t n, const int32_t* rows, float* logprobs_out, void* st) {
    SCONE_REQUIRE(m && n >= 0 && (n == 0 || logprobs_out), "scone_model_forward_planned_host: bad arguments");
    SCONE_REQUIRE(m->fused != nullptr, "scone_model_forward_planned_host: no fused pipeline");
    if (n == 0) return 0;
    cudaStream_t s = as_stream(st);
    int rc = ensure_staging(m, n, 0);
    if (rc) return rc;
    if (rows) SCONE_CUDA(cudaMemcpyAsync(m->d_nn, rows, n * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    if (fork_to_compute(m, st)) return 1;
    rc = scone_fused_run_planned(m->cx, m->fused, m->act, n, rows ? m->d_nn : nullptr, m->d_w, m->w_off.data(), m->d_logp_all, nullptr, nullptr,
                                 nullptr, false, m->compute);
    rc = finish_call(m, rc, st);
    if (rc) return rc;
    SCONE_CUDA(cudaMemcpyAsync(logprobs_out, m->d_logp_all, (size_t)n * m->cx->D * sizeof(float), cudaMemcpyDeviceToHost, s));
    SCONE_CUDA(cudaStreamSynchronize(s));
    return 0;
}

extern "C" int scone_model_check_overflow(scone_model* m, void* st) {
    SCONE_REQUIRE(m != nullptr, "scone_model_check_overflow: NULL model");
    return report_overflow(m, as_stream(st), "scone_model_check_overflow");
}

extern "C" int scone_model_set_weights_keep_state(scone_model* m, const float* w, void* st) {
    SCONE_REQUIRE(m && w, "scone_model_set_weights_keep_state: NULL argument");
    SCONE_CUDA(cudaMemcpyAsync(m->d_w, w, m->n_params * sizeof(float), cudaMemcpyHostToDevice, as_stream(st)));
    return 0;
}

extern "C" int scone_model_fused_info(const scone_model* m, int32_t* out /* [16] */) {
    SCONE_REQUIRE(m && out, "scone_model_fused_info: NULL argument");
    for (int i = 0; i < 16; ++i) out[i] = 0;
    if (!m->fused) return 0;
    const FusedState* f = m->fused;
    out[0] = 1; out[1] = f->bound_cone; out[2] = f->bound_list; out[3] = f->HS; out[4] = f->chunk; out[5] = f->cap_rows;
    out[6] = (int32_t)(f->plan_smem / 1024); out[7] = (int32_t)(f->traj_smem_small / 1024);
    out[8] = f->HS0; out[9] = f->LV0; out[10] = (int32_t)(f->plan_smem0 / 1024); out[11] = f->two_tiers ? 1 : 0;
    out[12] = f->tb_rows ? (int32_t)std::max<unsigned long long>(1, f->tb_bytes >> 20) : 0; out[13] = (int32_t)(f->arena_words >> 20);
    out[14] = (int32_t)std::min<unsigned long long>(f->cone_entries >> 10, 0x7fffffffull); out[15] = scone_fused_last_retries(m->fused);
    return 0;
}

extern "C" int scone_model_fused_read(scone_model* m, int32_t t, int32_t* hdr_out, uint32_t off, int32_t words, uint32_t* arena_out) {
    SCONE_REQUIRE(m && m->fused, "scone_model_fused_read: the model has no fused pipeline");
    SCONE_REQUIRE(t >= 0 && t < m->fused->chunk && (uint64_t)off + (uint64_t)(words > 0 ? words : 0) <= m->fused->arena_words,
                  "scone_model_fused_read: out of range");
    return scone_fused_read(m->fused, t, hdr_out, off, words, arena_out);
}

extern "C" int scone_model_read_rows_done(scone_model* m, int64_t* out /* [2] */) {
    SCONE_REQUIRE(m && out, "scone_model_read_rows_done: NULL argument");
    out[0] = out[1] = 0;
    if (!m->fused) return 0;
    unsigned long long v[2];
    SCONE_CUDA(cudaMemcpy(v, m->fused->d_rows_done, sizeof(v), cudaMemcpyDeviceToHost));
    SCONE_CUDA(cudaMemset(m->fused->d_rows_done, 0, sizeof(v)));
    out[0] = (int64_t)v[0];
    out[1] = (int64_t)v[1];
    return 0;
}

extern "C" int scone_umma_status(void* st) { return scone_umma_check(as_stream(st)); }

extern "C" int scone_model_dp_adam_step(scone_model* m, scone_dp* dp, int32_t step, float lr, float wd, void* st) {
    SCONE_REQUIRE(m && dp && step >= 0, "scone_model_dp_adam_step: bad arguments");
    return scone_dp_allreduce_adam(dp, m->d_w, m->d_m, m->d_v, m->d_grad, m->n_params, m->d_overflow, step, lr, wd, as_stream(st));
}

extern "C" int scone_model_adam_step(scone_model* m, int32_t step, float lr, float wd, void* st) {
    SCONE_REQUIRE(m && step >= 0, "scone_model_adam_step: bad arguments");
    return scone_adam_launch(m->d_w, m->d_m, m->d_v, m->d_grad, m->n_params, step, lr, wd, st, m->d_overflow);
}
