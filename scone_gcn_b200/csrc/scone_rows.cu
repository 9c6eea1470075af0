// scone_rows.cu — the bitmap-native row-list pipelines behind the model-level entry points (widths 16 / 32).
//
// A tensor is a ROW BITMAP (bit set <=> the row may be non-zero and has been written), an ascending row list, a rank prefix per
// bitmap word and a compact array [rows][C]; row ids are trajectory-major (t*E + e) for compact tensors, edge-major (e*b + t)
// over dense tensors (RowIds, slab_common.cuh).  Two orchestrations (scone_model.cu) use the kernels below:
//   pipeline 3 (default)  one row set per layer shared by H_l and G_l: the LIVE rows = receptive cone of the readout (geometry,
//                         rows_cone_kernel) & structural support of the flows (marked layer by layer); two-level bitmaps
//                         (summary bit per word) so that compaction and clearing never scan E*b bits
//   pipelines 2 / 1       every tensor has its own bitmap over its whole support; producers mark the candidate rows of the next
//                         tensor one hop further; per layer: clear, compact (scone_kernels.cu), run one row-list kernel
// Marking is an idempotent atomicOr (the bitmap does not depend on the order of the writers); lists are ascending: deterministic.
//
//   cone           rows of H_L the log-probs read, one hop down per layer   trajectory_experiments.py:151,298-303 (Bconds_func)
//   flows          X rows (+ live / candidate bits of H_1)                    synthetic_data_gen.py:327-344 (path_to_flow)
//   first layer    H_1 = act(X w0 + (S0 X) w1 + (S1 X) w2)                    trajectory_experiments.py:145-149 (i = 0)
//   conv layers    layer_fwd_rows_kernel (scone_slab.cu)                      trajectory_experiments.py:145-149
//   readout        logits, padded log-softmax, NLL gradient                   trajectory_experiments.py:151-152
//   backward       A_k = S_k G, Gprev = (sum_k A_k W_k^T) * act'(Hin); dW_k = Hin^T A_k     (jax.grad, scone_trajectory_model.py:307)
//   first layer bwd  dW_k[0][:] = sum_rows (S_k X)[row] * G_1[row][:]
//   accuracy       mask-to--100 + argmax + compare                            scone_trajectory_model.py:59-71
#include <cstdlib>
#include "common.cuh"

namespace {

#include "slab_common.cuh"

constexpr int kRoWarps = 8, kRoMaxD = SCONE_MAX_DEGREE, kRoMaxCper = 4;     // readout / cone kernels: max degree, channels per lane
constexpr int kRoItems = 1024;                                  // (neighbour, incident edge) pairs of a trajectory staged in shared memory

template <int ACT>
__device__ __forceinline__ float act_scalar(float z) {
    if (ACT == SCONE_ACT_TANH) return scone_tanh(z);
    if (ACT == SCONE_ACT_LEAKY_RELU) return z >= 0.f ? z : 0.01f * z;
    return fmaxf(z, 0.f);
}
template <int ACT>
__device__ __forceinline__ float dact_out(float h) {       // derivative through the OUTPUT h = act(z)
    if (ACT == SCONE_ACT_TANH) return 1.f - h * h;
    if (ACT == SCONE_ACT_LEAKY_RELU) return h >= 0.f ? 1.f : 0.01f;
    return h > 0.f ? 1.f : 0.f;
}

// ---------------------------------------------------------------------------------------------------------------
// flows: one CTA per trajectory.  X[row] = value, bit of X, and the candidate bits of H_1 (the row itself is in its own
// merged operator row).  CLEAR = true undoes the X writes after the step (X stays all-zero between micro-batches, so the
// first-layer gathers need no flag test and X needs no E*b memset).
// ---------------------------------------------------------------------------------------------------------------
template <bool CLEAR>
__global__ void __launch_bounds__(256) rows_flows_kernel(const int32_t* __restrict__ traj_ptr, const int32_t* __restrict__ flow_edge,
                                                        const float* __restrict__ flow_val, const int32_t* __restrict__ rank,
                                                        float* __restrict__ X, uint32_t* __restrict__ bmX, uint32_t* __restrict__ bm_next,
                                                        const int32_t* __restrict__ mptr, const int2* __restrict__ ment, int E, int b,
                                                        bool tmaj, const uint32_t* __restrict__ bm_filter, size_t sum_off) {
    // a quad of threads per flow entry: lane 0 of the quad writes X, the four lanes split the entry's merged operator row
    const int t = blockIdx.x, ql = threadIdx.x & 3;
    const size_t se = tmaj ? 1 : (size_t)b, toff = tmaj ? (size_t)t * E : (size_t)t;     // row id = e * se + toff (see RowIds)
    uint32_t* next1 = sum_off && bm_next != nullptr ? bm_next + sum_off : nullptr;
    for (int p = traj_ptr[t] + (threadIdx.x >> 2); p < traj_ptr[t + 1]; p += blockDim.x >> 2) {
        const int eo = flow_edge[p];
        if (eo < 0 || eo >= E) continue;
        const int e = rank[eo];
        const size_t row = (size_t)e * se + toff;
        if (CLEAR) {
            if (ql == 0) X[row] = 0.f;
            continue;
        }
        if (ql == 0) {
            X[row] = flow_val[p];
            if (bmX != nullptr) bit_set(bmX, row);
        }
        if (bm_next != nullptr) {
            const int q1 = mptr[e + 1];
            for (int q = mptr[e] + ql; q < q1; q += 4) {         // candidate rows of H_1; with a filter only those inside it (the cone)
                const size_t nrow = (size_t)(unsigned)ment[q].x * se + toff;
                if (bm_filter == nullptr || bit_test(bm_filter, nrow)) bit_set2(bm_next, next1, nrow);
            }
        }
    }
}

// candidate rows one hop further: a quad of threads per row of the list splits its merged operator row; every entry marks
// (column, t) in bm_next — with a filter only inside it (idempotent atomicOr: the bitmap does not depend on the order)
__global__ void __launch_bounds__(256) rows_mark_kernel(const uint32_t* __restrict__ rows, const int* __restrict__ n_ptr,
                                                       const int32_t* __restrict__ mptr, const int2* __restrict__ ment, int b,
                                                       uint32_t* __restrict__ bm_next, int list_cap, size_t sum_off, int E, bool tmaj,
                                                       const uint32_t* __restrict__ bm_filter) {
    const int n = min(*n_ptr, list_cap);
    const unsigned dv = tmaj ? (unsigned)E : (unsigned)b, se = tmaj ? 1u : (unsigned)b;
    uint32_t* bm1 = sum_off ? bm_next + sum_off : nullptr;
    const int ql = threadIdx.x & 3;
    for (int li = (blockIdx.x * blockDim.x + threadIdx.x) >> 2; li < n; li += (gridDim.x * blockDim.x) >> 2) {
        const uint32_t rid = __ldg(rows + li);
        const unsigned q = rid / dv, r = rid - q * dv;
        const unsigned e = tmaj ? r : q, toff = tmaj ? rid - r : r;
        const int p1 = __ldg(mptr + e + 1);
        for (int p = __ldg(mptr + e) + ql; p < p1; p += 4) {
            const unsigned nrow = (unsigned)__ldg(ment + p).x * se + toff;
            if (bm_filter == nullptr || bit_test(bm_filter, nrow)) bit_set2(bm_next, bm1, nrow);
        }
    }
}

// Compaction of a SPARSE two-level bitmap (see bit_set2): same contract as compact_bitmap_kernel (ascending row list, count, rank
// prefix per non-empty word, one launch, per-CTA totals + decoupled look-back over tickets, deterministic) but the CTAs scan the
// summary words and touch only the bitmap words whose summary bit is set.  tickets[] must be zero at launch.
constexpr int kSumMaxChunks = 64;       // chunks (WPT * 256 summary words) per CTA
// A warp walks its 32 * WPT summary words of a chunk (WPT per lane, ascending = lane-major) COOPERATIVELY: for every non-empty summary
// word the 32 lanes load the 32 bitmap words under it (one 128-byte line) at once.  With trajectory-major row ids the set bits
// of a sparse bitmap sit in a few dense clusters; a thread-per-word walk left all the work to a handful of threads.
// WRITE = false: returns this lane's share of the count (sum over the warp = rows under the warp's words).
// WRITE = true: rows are written from list index `off` on (ascending), prefixes for the non-empty bitmap words.
template <bool WRITE, int WPT>
__device__ __forceinline__ long long summary_walk(const uint32_t* __restrict__ bm, long long w1_lane, const uint32_t (&sm)[WPT],
                                                  long long off, uint32_t* __restrict__ list, uint32_t* __restrict__ pref_out,
                                                  long long list_cap) {
    const int lane = threadIdx.x & 31;
    long long cnt = 0;
    uint32_t any = 0u;
#pragma unroll
    for (int k = 0; k < WPT; ++k) any |= sm[k];
    unsigned mask = __ballot_sync(0xffffffffu, any != 0u);
    while (mask) {
        const int src = __ffs(mask) - 1;
        mask &= mask - 1;
        const long long w1s = __shfl_sync(0xffffffffu, w1_lane, src);
#pragma unroll
        for (int k = 0; k < WPT; ++k) {
            const uint32_t word = __shfl_sync(0xffffffffu, sm[k], src);
            if (word == 0u) continue;                     // (uniform)
            const long long w = (w1s + k) * 32 + lane;    // this lane's bitmap word
            uint32_t cc = (word >> lane) & 1u ? __ldg(bm + w) : 0u;
            const int c = __popc(cc);
            if (!WRITE) {
                cnt += c;
            } else {
                int incl = c;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += v;
                }
                long long o2 = off + incl - c;
                if (c) {
                    if (pref_out != nullptr) pref_out[w] = (uint32_t)o2;
                    while (cc) {
                        const int pbit = __ffs(cc) - 1;
                        cc &= cc - 1;
                        if (o2 < list_cap) list[o2] = (uint32_t)(w * 32 + pbit);
                        ++o2;
                    }
                }
                off += __shfl_sync(0xffffffffu, incl, 31);
            }
        }
    }
    return WRITE ? off : cnt;
}

// WPT (summary words per thread: 16, 4 or 1) is chosen by the launcher so that small bitmaps still spread over warps / CTAs.
template <int WPT>
__global__ void __launch_bounds__(256) compact_summary_kernel(const uint32_t* __restrict__ bm, const uint32_t* __restrict__ bm1,
                                                             long long n1_words, uint32_t* __restrict__ list, int* __restrict__ n_out,
                                                             unsigned long long* __restrict__ tickets, uint32_t* __restrict__ pref_out,
                                                             long long list_cap) {
    constexpr int kSumWpt = WPT, kSumChunk = WPT * 256;
    __shared__ int s_cnt[kSumMaxChunks * 8];              // rows under (chunk, warp), chunk-major = ascending
    __shared__ long long s_prefix;
    __shared__ int s_total;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long per_cta = ((n1_words + gridDim.x - 1) / gridDim.x + kSumChunk - 1) / kSumChunk * kSumChunk;     // whole chunks
    const long long lo = (long long)blockIdx.x * per_cta, hi = lo + per_cta < n1_words ? lo + per_cta : n1_words;
    const int n_chunks = hi > lo ? (int)((hi - lo + kSumChunk - 1) / kSumChunk) : 0;
    auto load4 = [&](long long w1, uint32_t (&sm)[kSumWpt]) {   // summary words w1 .. w1+WPT-1 (w1 % WPT == 0; the summary is padded), zero beyond hi
        if (WPT == 1) {
            sm[0] = w1 < hi ? __ldg(bm1 + w1) : 0u;
        } else {
#pragma unroll
            for (int v4 = 0; v4 < (WPT + 3) / 4; ++v4) {
                uint4 v = make_uint4(0u, 0u, 0u, 0u);
                if (w1 + 4 * v4 < hi) v = __ldg(reinterpret_cast<const uint4*>(bm1 + w1 + 4 * v4));
                sm[(4 * v4 + 0) % WPT] = v.x;
                sm[(4 * v4 + 1) % WPT] = w1 + 4 * v4 + 1 < hi ? v.y : 0u;
                sm[(4 * v4 + 2) % WPT] = w1 + 4 * v4 + 2 < hi ? v.z : 0u;
                sm[(4 * v4 + 3) % WPT] = w1 + 4 * v4 + 3 < hi ? v.w : 0u;
            }
        }
    };
    uint32_t sm[kSumWpt];                                  // (one chunk per CTA — the usual case — is loaded once for both passes)
    for (int c = 0; c < n_chunks; ++c) {
        const long long w1 = lo + (long long)c * kSumChunk + (long long)kSumWpt * threadIdx.x;
        load4(w1, sm);
        int cnt = (int)summary_walk<false, WPT>(bm, w1, sm, 0, nullptr, nullptr, 0);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if (lane == 0) s_cnt[c * 8 + warp] = cnt;
    }
    if (threadIdx.x == 0) s_prefix = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        int total = 0;
        for (int k = 0; k < n_chunks * 8; ++k) total += s_cnt[k];
        s_total = total;
        atomicExch(tickets + blockIdx.x, (1ull << 63) | (unsigned long long)(unsigned)total);
    }
    long long part = 0;
    for (int c = threadIdx.x; c < (int)blockIdx.x; c += 256) {
        unsigned long long t;
        do { t = *reinterpret_cast<volatile unsigned long long*>(tickets + c); } while (!(t >> 63));
        part += (long long)(t & 0xffffffffull);
    }
    if (part) atomicAdd((unsigned long long*)&s_prefix, (unsigned long long)part);
    __syncthreads();
    const long long base = s_prefix;
    const int total = s_total;
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
        n_out[0] = (int)(base + total);
        n_out[1] = 0;                                     // tile counter of the row-list kernel that consumes this list
    }
    if (total == 0) return;                               // (uniform) nothing set in this slice
    for (int c = 0; c < n_chunks; ++c) {
        if (s_cnt[c * 8 + warp] == 0) continue;           // (warp-uniform)
        int before = 0;                                   // rows of this CTA before (c, warp)
        for (int k = lane; k < c * 8 + warp; k += 32) before += s_cnt[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
        const long long w1 = lo + (long long)c * kSumChunk + (long long)kSumWpt * threadIdx.x;
        if (n_chunks > 1) load4(w1, sm);
        summary_walk<true, WPT>(bm, w1, sm, base + before, list, pref_out, list_cap);
    }
}

// back to all-zero.  `master` is the summary of a bitmap that contains every bit set in any bitmap of the list (the lowest cone
// level): for each of its set bits the word is zeroed in ALL bitmaps, then the summary word in all of them.  One scan of one
// summary instead of one per bitmap.
constexpr int kClearMax = 16;
struct ClearList {
    uint32_t* bm[kClearMax];
};
__global__ void __launch_bounds__(256) clear_summary_kernel(ClearList list, int count, uint32_t* __restrict__ master, size_t sum_off,
                                                           long long n1_words) {
    const long long n4 = (n1_words + 3) / 4;              // summaries are 64-byte aligned and padded to whole 16-byte groups
    for (long long g4 = (long long)blockIdx.x * blockDim.x + threadIdx.x; g4 < n4; g4 += (long long)gridDim.x * blockDim.x) {
        const uint4 v = *reinterpret_cast<const uint4*>(master + 4 * g4);
        if ((v.x | v.y | v.z | v.w) == 0u) continue;
        const uint32_t sm4[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t sm = sm4[k];
            while (sm) {
                const int q = __ffs(sm) - 1;
                sm &= sm - 1;
                for (int i = 0; i < count; ++i) list.bm[i][(4 * g4 + k) * 32 + q] = 0u;
            }
        }
        for (int i = 0; i < count; ++i) *reinterpret_cast<uint4*>(list.bm[i] + sum_off + 4 * g4) = make_uint4(0u, 0u, 0u, 0u);
    }
}

// Receptive cone of the readout (pure geometry: last node + complex).  The log-probs of trajectory t depend on H_L only at the
// edges incident to the neighbours of its last node (trajectory_experiments.py:151,298-303): the top of the cone.  H_{L-1} has to
// provide the rows one hop around those, and so on down.  Rows outside the cone reach neither the log-probs nor any weight
// gradient; the cone pipeline never computes them.  One CTA per trajectory builds the bitmaps of ALL levels: the edges that
// turned a bit on at level l (atomicOr reports it: an exact, duplicate-free list in shared memory) are expanded into level
// l - 1.  A (neighbour, edge) or (edge, merged row) expansion is split over a quad of threads.  bm[l]: bitmap of level l
// (tensor H_{l+1}), trajectory-major ids, summary words at + sum_off.
constexpr int kConeCap = 2048;           // edges per level and trajectory staged in shared memory (2 lists)
constexpr int kConeHash = 4096;          // open-addressing set of the edges of the level being built (power of two > kConeCap)
constexpr int kConeMaxLevels = 8;
struct ConeBitmaps {
    uint32_t* bm[kConeMaxLevels];
};
__global__ void __launch_bounds__(256) rows_cone_kernel(const int32_t* __restrict__ last_nodes, const int32_t* __restrict__ nbrhoods,
                                                       const int32_t* __restrict__ inc_ptr, const int2* __restrict__ inc_ent,
                                                       ConeBitmaps cone, int n_levels, const int32_t* __restrict__ mptr,
                                                       const int2* __restrict__ ment, int N, int D, int E, size_t sum_off,
                                                       int* __restrict__ overflow) {
    // Duplicates are removed in SHARED memory (a hash set per level): an edge new to the level is appended to the level's list
    // and its bitmap / summary bits are set with fire-and-forget atomics — no thread ever waits on a global atomic or re-reads
    // the bitmap; the only global latency on the path is the merged-row load.
    __shared__ int s_ptr[kRoMaxD], s_off[kRoMaxD + 1];
    __shared__ int s_list[2][kConeCap];
    __shared__ int s_hash[kConeHash];
    __shared__ int s_n[2];
    const int t = blockIdx.x;
    const int last = last_nodes[t];
    if (last < 0 || last >= N) return;
    for (int j = threadIdx.x; j < D; j += blockDim.x) {
        const int nbr = nbrhoods[(size_t)last * D + j];
        s_ptr[j] = nbr >= 0 ? inc_ptr[nbr] : 0;
        s_off[j + 1] = nbr >= 0 ? inc_ptr[nbr + 1] - inc_ptr[nbr] : 0;
    }
    for (int i = threadIdx.x; i < kConeHash; i += blockDim.x) s_hash[i] = -1;
    if (threadIdx.x == 0) s_n[0] = s_n[1] = 0;
    __syncthreads();
    if (threadIdx.x == 0) {
        s_off[0] = 0;
        for (int j = 0; j < D; ++j) s_off[j + 1] += s_off[j];
    }
    __syncthreads();
    const size_t tbase = (size_t)t * (size_t)E;
    // adds edge e to level lv: true if it was not there yet (then its bits are set and, above the last level, it is listed)
    auto add = [&](int lv, int which, int e) {
        unsigned h = ((unsigned)e * 2654435761u) >> 20;   // kConeHash = 2^12 slots
        for (int probes = 0; probes < kConeHash; ++probes) {
            const int old = atomicCAS(&s_hash[h], -1, e);
            if (old == e) return;
            if (old == -1) {
                uint32_t* bm = cone.bm[lv];
                const size_t row = tbase + (unsigned)e, widx = row >> 5;
                atomicOr(bm + widx, 1u << (row & 31));
                // only the lowest level keeps summary bits: it contains every level above it (a merged operator row holds its own
                // diagonal) and every live row, so its summary is the one the clearing kernel scans
                if (lv == 0) atomicOr(bm + sum_off + (widx >> 5), 1u << (widx & 31));
                if (lv > 0) {
                    const int pos = atomicAdd(&s_n[which], 1);
                    if (pos < kConeCap) s_list[which][pos] = e;
                    else *overflow = 1;                   // (host: scone_model_read_grads / forward_host report it)
                }
                return;
            }
            h = (h + 1) & (kConeHash - 1);
        }
        *overflow = 1;
    };
    // top level: edges incident to the neighbours of the last node
    int lv = n_levels - 1, cur = 0;
    for (int i = threadIdx.x; i < s_off[D]; i += blockDim.x) {
        int j = 0;
        while (s_off[j + 1] <= i) ++j;
        add(lv, cur, inc_ent[s_ptr[j] + (i - s_off[j])].x);
    }
    // one hop down per level
    const int ql = threadIdx.x & 3;
    for (--lv; lv >= 0; --lv) {
        __syncthreads();
        const int n_cur = min(s_n[cur], kConeCap);
        for (int i = threadIdx.x; i < kConeHash; i += blockDim.x) s_hash[i] = -1;
        if (threadIdx.x == 0) s_n[1 - cur] = 0;
        __syncthreads();
        for (int i = threadIdx.x >> 2; i < n_cur; i += blockDim.x >> 2) {
            const int e = s_list[cur][i];
            const int p1 = mptr[e + 1];
            for (int q = mptr[e] + ql; q < p1; q += 4) add(lv, 1 - cur, ment[q].x);
        }
        cur = 1 - cur;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// first layer forward over a row list: lane = row for the scalar gathers of X (no flag test: X is zero off its support), then
// the 32 rows of the warp are written one after the other with lane = channel (coalesced).  Gather order = merged row order
// = ascending columns for both sums, same as the unit kernels.
// ---------------------------------------------------------------------------------------------------------------
template <int COUT, int ACT, bool COMPACT>
__global__ void __launch_bounds__(256) rows_layer0_fwd_kernel(const float* __restrict__ X, float* __restrict__ Hout,
                                                             const float* __restrict__ W0, const float* __restrict__ W1,
                                                             const float* __restrict__ W2, const int32_t* __restrict__ mptr,
                                                             const int2* __restrict__ ment, const uint32_t* __restrict__ rows,
                                                             const int* __restrict__ n_ptr, int b, uint32_t* __restrict__ bm_next,
                                                             int out_cap, int* __restrict__ overflow, int E) {
    static_assert(COUT == 16 || COUT == 32, "first-layer row kernel: widths 16 / 32");
    constexpr int RPI = 32 / COUT;                        // rows written per iteration of the store loop
    const int lane = threadIdx.x & 31;
    int n = *n_ptr;
    if (COMPACT && n > out_cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) *overflow = 1;
        n = out_cap;
    }
    const int c = lane % COUT;
    const float w0 = W0[c], w1 = W1[c], w2 = W2[c];
    const int n_groups = (n + 31) / 32;
    const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    for (int grp = gw; grp < n_groups; grp += nw) {
        const int li = grp * 32 + lane;
        uint32_t rid = 0;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        if (li < n) {
            rid = __ldg(rows + li);
            const RowIds<COMPACT> ids(rid, b, E);
            const int e = (int)ids.e;
            a0 = __ldg(X + rid);
            const int p1 = __ldg(mptr + e + 1);
            for (int p = __ldg(mptr + e); p < p1; ++p) {
                const int2 en = __ldg(ment + p);
                const size_t nrow = ids.row((unsigned)en.x);
                const float x = __ldg(X + nrow);
                a1 = fmaf((float)(short)(en.y & 0xffff), x, a1);
                a2 = fmaf((float)(en.y >> 16), x, a2);
                if (bm_next != nullptr) bit_set(bm_next, nrow);
            }
        }
        const int cnt = min(32, n - grp * 32);
        for (int r0 = 0; r0 < cnt; r0 += RPI) {
            const int r = r0 + lane / COUT;
            const float s0 = __shfl_sync(0xffffffffu, a0, r & 31), s1 = __shfl_sync(0xffffffffu, a1, r & 31),
                        s2 = __shfl_sync(0xffffffffu, a2, r & 31);
            const uint32_t orow = __shfl_sync(0xffffffffu, rid, r & 31);
            if (r < cnt) Hout[(size_t)(COMPACT ? (uint32_t)(grp * 32 + r) : orow) * COUT + c] = act_scalar<ACT>(fmaf(s2, w2, fmaf(s1, w1, s0 * w0)));
        }
    }
}

// first layer backward: dW_k[0][c] = sum_rows a_k[row] * G_1[row][c] with a_0 = X[row], a_1 = (S0 X)[row], a_2 = (S1 X)[row].  A warp
// takes 32 consecutive list rows: lane = row for the scalar gathers of X (exact small integers), then lane = channel walks the 32
// rows (coalesced G rows, a_k by shuffle).  Fixed row -> warp mapping and order; per-CTA partials [3][COUT] (reduced by
// rows_reduce_kernel): deterministic.
constexpr int kL0bWarps = 32;      // the gathers are latency-bound: full occupancy (2 CTAs x 32 warps per SM)
template <int COUT, bool COMPACT>
__global__ void __launch_bounds__(32 * kL0bWarps) rows_layer0_bwd_kernel(const float* __restrict__ X, const float* __restrict__ G,
                                                             const int32_t* __restrict__ mptr, const int2* __restrict__ ment,
                                                             const uint32_t* __restrict__ rows, const int* __restrict__ n_ptr, int b,
                                                             float* __restrict__ partial /* [grid][3*COUT] */, int cap, int E) {
    static_assert(COUT == 16 || COUT == 32, "first-layer row kernel: widths 16 / 32");
    constexpr int RPI = 32 / COUT;                             // rows per iteration of the channel loop
    __shared__ float red[kL0bWarps][3 * 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int n = *n_ptr;
    if (COMPACT && n > cap) n = cap;
    const int n_groups = (n + 31) / 32;
    const int per = (n_groups + gridDim.x - 1) / gridDim.x;   // contiguous slice of 32-row groups per CTA, strided over its warps
    const int lo = min(n_groups, (int)blockIdx.x * per), hi = min(n_groups, lo + per);
    const int c = lane % COUT, sub = lane / COUT;
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f;
    for (int grp = lo + warp; grp < hi; grp += kL0bWarps) {
        const int li = grp * 32 + lane;
        uint32_t rid = 0;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        if (li < n) {
            rid = __ldg(rows + li);
            const RowIds<COMPACT> ids(rid, b, E);
            const int e = (int)ids.e;
            a0 = __ldg(X + rid);
            const int p1 = __ldg(mptr + e + 1);
            for (int p = __ldg(mptr + e); p < p1; ++p) {
                const int2 en = __ldg(ment + p);
                const float x = __ldg(X + ids.row((unsigned)en.x));
                a1 = fmaf((float)(short)(en.y & 0xffff), x, a1);
                a2 = fmaf((float)(en.y >> 16), x, a2);
            }
        }
        const int cnt = min(32, n - grp * 32);
#pragma unroll 4
        for (int r0 = 0; r0 < cnt; r0 += RPI) {
            const int r = r0 + sub;
            const float s0 = __shfl_sync(0xffffffffu, a0, r & 31), s1 = __shfl_sync(0xffffffffu, a1, r & 31),
                        s2 = __shfl_sync(0xffffffffu, a2, r & 31);
            const uint32_t orow = __shfl_sync(0xffffffffu, rid, r & 31);
            if (r < cnt) {
                const float gv = __ldg(G + (size_t)(COMPACT ? (uint32_t)(grp * 32 + r) : orow) * COUT + c);
                acc0 = fmaf(s0, gv, acc0);
                acc1 = fmaf(s1, gv, acc1);
                acc2 = fmaf(s2, gv, acc2);
            }
        }
    }
    if (RPI == 2) {                                            // the two half-warps hold alternate rows of the same channels
        acc0 += __shfl_down_sync(0xffffffffu, acc0, 16);
        acc1 += __shfl_down_sync(0xffffffffu, acc1, 16);
        acc2 += __shfl_down_sync(0xffffffffu, acc2, 16);
    }
    red[warp][lane] = acc0;
    red[warp][32 + lane] = acc1;
    red[warp][64 + lane] = acc2;
    __syncthreads();
    for (int o = threadIdx.x; o < 3 * COUT; o += blockDim.x) {
        const int k = o / COUT, cc = o % COUT;
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kL0bWarps; ++w) s += red[w][k * 32 + cc];
        partial[(size_t)blockIdx.x * 3 * COUT + o] = s;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Backward over a row list (the candidate rows of Gprev = rows where S G can be non-zero): same gather as the forward row
// kernel on G (flag test = row bitmap of G), the three gathered terms A_k are (1) stored compactly, row i of the list at
// Abuf[i][3*COUT], for the weight-gradient GEMM, (2) contracted with W^T on the tensor cores (3xTF32) into
// Gprev = (sum_k A_k W_k^T) * act'(Hin) with Hin rows read through the row bitmap of H_{l-1} (an unflagged row is an exact
// zero: act'(0)).
// ---------------------------------------------------------------------------------------------------------------
template <int CIN, int COUT, int ACT, bool COMPACT>
__global__ void __launch_bounds__(kRowsThreads, 1) rows_bwd_kernel(const float* __restrict__ Gin, const float* __restrict__ Hin,
                                                                  float* __restrict__ Gprev, float* __restrict__ Abuf,
                                                                  const float* __restrict__ W0, const float* __restrict__ W1,
                                                                  const float* __restrict__ W2, const int32_t* __restrict__ mptr,
                                                                  const int2* __restrict__ ment, const uint32_t* __restrict__ rows,
                                                                  const int* __restrict__ n_ptr, int b, const uint32_t* __restrict__ bmG,
                                                                  const uint32_t* __restrict__ bmH, int a_cap, int* __restrict__ overflow,
                                                                  unsigned long long* __restrict__ row_counter,
                                                                  const uint32_t* __restrict__ prefG, const uint32_t* __restrict__ prefH, int E) {
    using G = SlabGeom<COUT, 16>;                          // the gathered tensor has COUT channels
    constexpr int NT = CIN / 8, NL = G::NL, Q = G::Q, LPR = COUT / 4;
    extern __shared__ __align__(16) uint4 Bf[];
    stage_weight_fragments<COUT, CIN, 16, true>(Bf, W0, W1, W2);
    __syncthreads();
    const int lane = threadIdx.x & 31, tig = lane & 3, g = lane >> 2;
    const int gq = lane / LPR, cq = lane % LPR;
    const unsigned rowbytes = COMPACT ? COUT * 4u : (unsigned)b * COUT * 4u;
    const char* Gb = reinterpret_cast<const char*>(Gin);
    int n = *n_ptr;
    if (n > a_cap) {                                       // the compact A buffer cannot hold this many rows: flag it (host raises)
        if (blockIdx.x == 0 && threadIdx.x == 0) *overflow = 1;
        n = a_cap;
    }
    const int n_slabs = (n + 15) / 16;
    const int n_minis = (n_slabs + kRowsMini - 1) / kRowsMini;
    if (row_counter != nullptr && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(row_counter, (unsigned long long)n);
    int* tile_counter = const_cast<int*>(n_ptr) + 1;       // per-warp dynamic mini-tiles, see layer_fwd_rows_kernel
    for (;;) {
        int mini = 0;
        if (lane == 0) mini = atomicAdd(tile_counter, 1);
        mini = __shfl_sync(0xffffffffu, mini, 0);
        if (mini >= n_minis) break;
        const int slab_end = min(n_slabs, (mini + 1) * kRowsMini);
        for (int slab = mini * kRowsMini; slab < slab_end; ++slab) {
        uint32_t rid[NL];
        unsigned oidx[NL];
        int len[NL], p0[NL], tq[NL], cpos[NL];
        const char* P[NL];
        bool own[NL], valid[NL];
        int maxlen = 0;
#pragma unroll
        for (int i = 0; i < NL; ++i) {
            const int li = slab * 16 + i * Q + gq;
            valid[i] = li < n;
            rid[i] = valid[i] ? __ldg(rows + li) : 0u;
            const RowIds<COMPACT> ids(rid[i], b, E);
            const int e = (int)ids.e;
            tq[i] = (int)ids.toff;                         // e-major: t; trajectory-major: t * E
            cpos[i] = (COUT == 32 && i >= 2) ? (cq ^ 4) : cq;
            P[i] = Gb + (size_t)((unsigned)((COMPACT ? 0 : tq[i] * COUT) + 4 * cpos[i]) * 4u);
            asm volatile("" : "+l"(P[i]));
            p0[i] = valid[i] ? __ldg(mptr + e) : 0;
            len[i] = valid[i] ? __ldg(mptr + e + 1) - p0[i] : 0;
            if (COMPACT) {
                own[i] = rank_lookup(bmG, prefG, rid[i], oidx[i]) && valid[i];
            } else {
                oidx[i] = (unsigned)e;
                own[i] = valid[i] && bit_test(bmG, rid[i]);
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
            unsigned gidx[NL];
#pragma unroll
            for (int i = 0; i < NL; ++i) {                 // branch-free bit test (entry {0,0} of an idle lane tests row tq: in range)
                const unsigned nrow = RowIds<COMPACT>::row_of((unsigned)ent[i].x, (unsigned)tq[i], b);
                if (COMPACT) {
                    on[i] = rank_lookup(bmG, prefG, nrow, gidx[i]) && on[i];
                } else {
                    on[i] = on[i] && ((__ldg(bmG + (nrow >> 5)) >> (nrow & 31)) & 1u) != 0u;
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
        // (1) the gathered terms, row li of the list -> Abuf[li][term * COUT + channel]
#pragma unroll
        for (int i = 0; i < NL; ++i)
            if (valid[i]) {
                float* dst = Abuf + (size_t)(slab * 16 + i * Q + gq) * (3 * COUT) + 4 * cpos[i];
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    float4 o;
                    unpack2(acc[k][i][0], o.x, o.y);
                    unpack2(acc[k][i][1], o.z, o.w);
                    *reinterpret_cast<float4*>(dst + k * COUT) = o;
                }
            }
        // (2) Gprev
        float d[NT][4];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) d[nt][0] = d[nt][1] = d[nt][2] = d[nt][3] = 0.f;
#pragma unroll
        for (int term = 0; term < 3; ++term) {
            float fr[G::KS][4];
            slab_fragments<COUT, 16>(acc[term], fr);
            slab_mma_term<G::KS, NT>(d, fr, Bf + term * G::KS * NT * 32);
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            uint32_t orow;
            bool ok;
            int oslot;
            if (COUT == 32) {
                const bool odd = g & 1;
                oslot = odd ? 2 + r : r;
                orow = odd ? rid[2 + r] : rid[r];
                ok = odd ? valid[2 + r] : valid[r];
            } else {
                oslot = r;
                orow = rid[r];
                ok = valid[r];
            }
            if (ok) {
                unsigned hidx = orow;
                const bool hset = COMPACT ? rank_lookup(bmH, prefH, orow, hidx) : bit_test(bmH, orow);
                const float* hsrc = Hin + (size_t)hidx * CIN + 2 * tig;
                float* dst = Gprev + (size_t)(COMPACT ? (uint32_t)(slab * 16 + oslot * Q + gq) : orow) * CIN + 2 * tig;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    float2 h = make_float2(0.f, 0.f);
                    if (hset) h = __ldg(reinterpret_cast<const float2*>(hsrc + nt * 8));
                    *reinterpret_cast<float2*>(dst + nt * 8) =
                        make_float2(d[nt][2 * r] * dact_out<ACT>(h.x), d[nt][2 * r + 1] * dact_out<ACT>(h.y));
                }
            }
        }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Weight gradients dW_k[ci][co] = sum_i Hin[rows[i]][ci] * A_k[i][co]: a tall-skinny GEMM (M = CIN, N = 3*COUT, K = rows)
// on mma.sync with the 3xTF32 split of both operands.  CTA c owns a contiguous slice of the list; its 8 warps own disjoint
// (m-tile, n-tile) sets and all walk the slice in k-steps of 8 rows (fixed order), operands fetched straight from global
// memory in fragment layout (each 32-bit load fills whole 32-byte sectors; the 8 warps share the rows through L1).
// Per-CTA partials, reduced over CTAs in a fixed tree: deterministic.
// ---------------------------------------------------------------------------------------------------------------
// IDENT: Hin is stored in the order of this very list (cone pipeline: row rows[i] of Hin at index i) — no rank lookup.
// The k-loop is software-pipelined UNR steps deep: all operand loads of UNR consecutive k-steps are issued before the first
// product (the loop was bound by the rows -> bitmap / prefix -> operand load chain, one chain per step); the mma order is the
// plain ascending k order either way.
template <int CIN, int COUT, bool COMPACT, bool IDENT>
__global__ void __launch_bounds__(256) rows_dw_kernel(const float* __restrict__ Hin, const uint32_t* __restrict__ bmH,
                                                     const float* __restrict__ Abuf, const uint32_t* __restrict__ rows,
                                                     const int* __restrict__ n_ptr, int a_cap, float* __restrict__ partial /* [grid][3*CIN*COUT] */,
                                                     const uint32_t* __restrict__ prefH) {
    constexpr int MT = CIN / 16, NTT = 3 * COUT / 8;       // m-tiles, n-tiles
    constexpr int TILES = MT * NTT;
    constexpr int TPW = TILES >= 24 ? 3 : (TILES >= 12 ? 2 : 1);   // (m, n) tiles per warp; TILES / TPW <= 8 warps work
    constexpr int UNR = 4;
    static_assert(TILES % TPW == 0 && TILES / TPW <= 8, "tile count must split over at most 8 warps");
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tig = lane & 3, g = lane >> 2;
    if (warp >= TILES / TPW) return;                       // (no CTA barrier below)
    int n = *n_ptr;
    if (n > a_cap) n = a_cap;
    const int n_steps = (n + 7) / 8;
    const int per = (n_steps + gridDim.x - 1) / gridDim.x;
    const int lo = min(n_steps, (int)blockIdx.x * per), hi = min(n_steps, lo + per);
    // this warp's tiles: consecutive n-tiles of one m-tile
    const int t0 = warp * TPW;
    const int mt = t0 / NTT, nt0 = t0 % NTT;
    static_assert(NTT % TPW == 0, "a warp's tiles must share one m-tile");
    float acc[TPW][4];
#pragma unroll
    for (int j = 0; j < TPW; ++j) acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
    const float* Hc = Hin + mt * 16 + g;
    const float* Ac = Abuf + nt0 * 8 + g;
    for (int s0 = lo; s0 < hi; s0 += UNR) {
        float a[UNR][4], bv[UNR][TPW][2];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int i0 = (s0 + u) * 8 + tig, i1 = i0 + 4;           // list positions of this lane's two k rows
            const bool ok0 = s0 + u < hi && i0 < n, ok1 = s0 + u < hi && i1 < n;
            a[u][0] = a[u][1] = a[u][2] = a[u][3] = 0.f;
            unsigned r0 = (unsigned)i0, r1 = (unsigned)i1;
            bool h0 = ok0, h1 = ok1;
            if (!IDENT) {
                if (ok0) {
                    r0 = __ldg(rows + i0);
                    h0 = COMPACT ? rank_lookup(bmH, prefH, r0, r0) : bit_test(bmH, r0);
                }
                if (ok1) {
                    r1 = __ldg(rows + i1);
                    h1 = COMPACT ? rank_lookup(bmH, prefH, r1, r1) : bit_test(bmH, r1);
                }
            }
            if (h0) {
                a[u][0] = __ldg(Hc + (size_t)r0 * CIN);
                a[u][1] = __ldg(Hc + (size_t)r0 * CIN + 8);
            }
            if (h1) {
                a[u][2] = __ldg(Hc + (size_t)r1 * CIN);
                a[u][3] = __ldg(Hc + (size_t)r1 * CIN + 8);
            }
#pragma unroll
            for (int j = 0; j < TPW; ++j) {
                bv[u][j][0] = ok0 ? __ldg(Ac + (size_t)i0 * (3 * COUT) + j * 8) : 0.f;
                bv[u][j][1] = ok1 ? __ldg(Ac + (size_t)i1 * (3 * COUT) + j * 8) : 0.f;
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            uint32_t ahi[4], alo[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) split_tf32(a[u][q], ahi[q], alo[q]);
#pragma unroll
            for (int j = 0; j < TPW; ++j) {
                uint32_t bh0, bl0, bh1, bl1;
                split_tf32(bv[u][j][0], bh0, bl0);
                split_tf32(bv[u][j][1], bh1, bl1);
                mma_tf32(acc[j], alo, bh0, bh1);
                mma_tf32(acc[j], ahi, bl0, bl1);
                mma_tf32(acc[j], ahi, bh0, bh1);
            }
        }
    }
    // D fragment (m = ci, n = k*COUT + co): c0,c1 -> (ci = g, n = 2*tig, +1); c2,c3 -> (ci = g + 8, ...)
    float* outp = partial + (size_t)blockIdx.x * (3 * CIN * COUT);
#pragma unroll
    for (int j = 0; j < TPW; ++j) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int ci = mt * 16 + g + (q >> 1) * 8;
            const int ncol = (nt0 + j) * 8 + 2 * tig + (q & 1);
            const int k = ncol / COUT, co = ncol % COUT;
            outp[(k * CIN + ci) * COUT + co] = acc[j][q];
        }
    }
}

// out[i] (+)= sum over parts (fixed tree): 256 threads = 32 outputs x 8 slices
__global__ void __launch_bounds__(256) rows_reduce_kernel(const float* __restrict__ partial, int nparts, int n, float* __restrict__ out,
                                                         int accumulate) {
    __shared__ float red[8][32];
    const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;
    const int per = (nparts + 7) / 8;
    const int p0 = slice * per, p1 = min(nparts, p0 + per);
    float s = 0.f;
    if (i < n) {
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;     // four loads in flight; fixed grouping
        int p = p0;
        for (; p + 3 < p1; p += 4) {
            s0 += partial[(size_t)p * n + i];
            s1 += partial[(size_t)(p + 1) * n + i];
            s2 += partial[(size_t)(p + 2) * n + i];
            s3 += partial[(size_t)(p + 3) * n + i];
        }
        for (; p < p1; ++p) s0 += partial[(size_t)p * n + i];
        s = (s0 + s1) + (s2 + s3);
    }
    red[slice][lane] = s;
    __syncthreads();
    if (slice == 0 && i < n) {
        float t = red[0][lane];
#pragma unroll
        for (int k = 1; k < 8; ++k) t += red[k][lane];
        out[i] = accumulate ? out[i] + t : t;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Readout for compact storage, in two kernels around the compaction of G_L's bitmap:
//   rows_readout_fwd_kernel   logits -> padded log-softmax (trajectory_experiments.py:151-152,298-303); with `grad` also the bits
//                             of the rows of G_L this trajectory touches and the candidate bits one hop further
//   rows_readout_bwd_kernel   dl_j = mask * scale * (exp(logp_j) - [j == y]); adds s(e, nbr_j) * dl_j * w * act'(h) onto row rank(e, t)
//                             of the zeroed compact G_L (at most two contributions per row: a + b == b + a, deterministic), the
//                             w_out gradient partials, the NLL term and the mask count.
// One CTA (4 warps) per trajectory, warps split the neighbour slots (same arithmetic as readout_kernel).
// ---------------------------------------------------------------------------------------------------------------

// The (neighbour slot j, incident edge) pairs of a trajectory are flattened: a first phase resolves every pair's row (sign, rank
// in H_L's storage, rank in G_L's) with one thread per pair — all lookups in flight at once — into shared memory; the second
// phase (warp per neighbour slot, rows in ascending pair order: the summation order of the sequential version) then issues its
// row loads four deep.  Pairs beyond kRoItems are resolved on the fly.
struct RoItem {
    int hidx;        // rank of the row in H_L's storage, -1: the row is exactly zero
    int gidx;        // rank in G_L's storage (backward)
    float sign;
};
struct RoPairs {
    int s_ptr[kRoMaxD], s_off[kRoMaxD + 1];
    __device__ __forceinline__ int setup(const int32_t* __restrict__ nbrhoods, const int32_t* __restrict__ inc_ptr, int last, bool last_ok, int D) {
        for (int j = threadIdx.x; j < D; j += blockDim.x) {
            const int nbr = last_ok ? nbrhoods[(size_t)last * D + j] : -1;
            s_ptr[j] = nbr >= 0 ? inc_ptr[nbr] : -1;
            s_off[j + 1] = nbr >= 0 ? inc_ptr[nbr + 1] - inc_ptr[nbr] : 0;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            s_off[0] = 0;
            for (int j = 0; j < D; ++j) s_off[j + 1] += s_off[j];
        }
        __syncthreads();
        return s_off[D];
    }
    __device__ __forceinline__ int slot_of(int i) const {
        int j = 0;
        while (s_off[j + 1] <= i) ++j;
        return j;
    }
};

__global__ void __launch_bounds__(32 * kRoWarps) rows_readout_fwd_kernel(const float* __restrict__ HL, const float* __restrict__ wout,
                                                                        const int32_t* __restrict__ last_nodes, const int32_t* __restrict__ nbrhoods,
                                                                        const int32_t* __restrict__ inc_ptr, const int2* __restrict__ inc_ent,
                                                                        float* __restrict__ logprobs, const uint32_t* __restrict__ bmH,
                                                                        const uint32_t* __restrict__ prefH, uint32_t* __restrict__ bmG,
                                                                        uint32_t* __restrict__ bm_cand, const int32_t* __restrict__ mptr,
                                                                        const int2* __restrict__ ment, int N, int D, int E, int C) {
    __shared__ float logit[kRoMaxD];
    __shared__ RoPairs pairs;
    __shared__ RoItem items[kRoItems];
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int t = blockIdx.x;
    const int last = last_nodes[t];
    const bool last_ok = last >= 0 && last < N;
    const unsigned tbase = (unsigned)t * (unsigned)E;      // compact tensors: trajectory-major row ids
    const int total = pairs.setup(nbrhoods, inc_ptr, last, last_ok, D);
    auto resolve = [&](int i, int j) {
        const int2 es = inc_ent[pairs.s_ptr[j] + (i - pairs.s_off[j])];
        RoItem it;
        unsigned idx;
        it.hidx = rank_lookup(bmH, prefH, tbase + (unsigned)es.x, idx) ? (int)idx : -1;
        it.gidx = es.x;
        it.sign = __int_as_float(es.y);
        return it;
    };
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const RoItem it = resolve(i, pairs.slot_of(i));
        if (i < kRoItems) items[i] = it;
        if (bmG != nullptr) {                              // gradient wanted (pipeline 2): this row of G_L will be written
            bit_set(bmG, tbase + (unsigned)it.gidx);
            if (bm_cand != nullptr)
                for (int q = mptr[it.gidx]; q < mptr[it.gidx + 1]; ++q) bit_set(bm_cand, tbase + (unsigned)ment[q].x);
        }
    }
    __syncthreads();
    float w[kRoMaxCper];
#pragma unroll
    for (int q = 0; q < kRoMaxCper; ++q) w[q] = (lane + 32 * q < C) ? wout[lane + 32 * q] : 0.f;
    for (int j = warp; j < D; j += kRoWarps) {
        float l = 0.f;
        if (pairs.s_ptr[j] >= 0) {
            float z[kRoMaxCper] = {0.f, 0.f, 0.f, 0.f};
            const int i1 = pairs.s_off[j + 1];
            for (int i0 = pairs.s_off[j]; i0 < i1; i0 += 4) {
                RoItem it[4];
                float hv[4][kRoMaxCper];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    it[u].hidx = -1;
                    it[u].sign = 0.f;
                    if (i0 + u < i1) it[u] = i0 + u < kRoItems ? items[i0 + u] : resolve(i0 + u, j);
#pragma unroll
                    for (int q = 0; q < kRoMaxCper; ++q)
                        hv[u][q] = (it[u].hidx >= 0 && lane + 32 * q < C) ? __ldg(HL + (size_t)it[u].hidx * C + lane + 32 * q) : 0.f;
                }
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (it[u].hidx >= 0) {                 // (an absent row is skipped, not added as 0: same sums as before)
#pragma unroll
                        for (int q = 0; q < kRoMaxCper; ++q) z[q] = fmaf(it[u].sign, hv[u][q], z[q]);
                    }
            }
            float part = 0.f;
#pragma unroll
            for (int q = 0; q < kRoMaxCper; ++q) part = fmaf(z[q], w[q], part);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            l = part;
        }
        if (lane == 0) logit[j] = l;
    }
    __syncthreads();
    if (warp == 0) {
        float mx = -3.4e38f;
        for (int j = lane; j < D; j += 32) mx = fmaxf(mx, logit[j]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        float se = 0.f;
        for (int j = lane; j < D; j += 32) se += expf(logit[j] - mx);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
        const float lse = mx + logf(se);
        for (int j = lane; j < D; j += 32) logprobs[(size_t)t * D + j] = logit[j] - lse;
    }
}

// zero the first min(*n, cap) rows of a compact tensor (row = C floats)
__global__ void __launch_bounds__(256) rows_zero_kernel(float4* __restrict__ T, const int* __restrict__ n_ptr, int cap, int c4,
                                                       int* __restrict__ overflow) {
    int n = *n_ptr;
    if (n > cap) {
        if (blockIdx.x == 0 && threadIdx.x == 0) *overflow = 1;
        n = cap;
    }
    const size_t total = (size_t)n * c4;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
        T[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void __launch_bounds__(32 * kRoWarps) rows_readout_bwd_kernel(const float* __restrict__ HL, const float* __restrict__ wout,
                                                                        const int32_t* __restrict__ last_nodes, const int32_t* __restrict__ nbrhoods,
                                                                        const int32_t* __restrict__ inc_ptr, const int2* __restrict__ inc_ent,
                                                                        const float* __restrict__ logprobs, const int32_t* __restrict__ target_idx,
                                                                        const float* __restrict__ mask, float scale, float* __restrict__ GL,
                                                                        float* __restrict__ partial /* [b][C+2] */, const uint32_t* __restrict__ bmH,
                                                                        const uint32_t* __restrict__ prefH, const uint32_t* __restrict__ bmG,
                                                                        const uint32_t* __restrict__ prefG, int g_cap, int act, int N, int D, int E, int C) {
    __shared__ float s_dw[kRoWarps][32 * kRoMaxCper];
    __shared__ RoPairs pairs;
    __shared__ RoItem items[kRoItems];
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int t = blockIdx.x;
    const int last = last_nodes[t];
    const bool last_ok = last >= 0 && last < N;
    const unsigned tbase = (unsigned)t * (unsigned)E;
    const int total = pairs.setup(nbrhoods, inc_ptr, last, last_ok, D);
    auto resolve = [&](int i, int j) {
        const int2 es = inc_ent[pairs.s_ptr[j] + (i - pairs.s_off[j])];
        const unsigned row = tbase + (unsigned)es.x;
        RoItem it;
        unsigned hidx, gidx;
        it.hidx = rank_lookup(bmH, prefH, row, hidx) ? (int)hidx : -1;
        if (bmG == bmH && prefG == prefH) {                // cone pipeline: G_L and H_L share their (live) row set; an absent row
            it.gidx = it.hidx >= 0 ? it.hidx : g_cap;      // is outside the flows' support: its gradient reaches no weight — skipped
        } else {
            rank_lookup(bmG, prefG, row, gidx);
            it.gidx = (int)gidx;
        }
        it.sign = __int_as_float(es.y);
        return it;
    };
    for (int i = threadIdx.x; i < total && i < kRoItems; i += blockDim.x) items[i] = resolve(i, pairs.slot_of(i));
    __syncthreads();
    float w[kRoMaxCper];
#pragma unroll
    for (int q = 0; q < kRoMaxCper; ++q) w[q] = (lane + 32 * q < C) ? wout[lane + 32 * q] : 0.f;
    const float mk = mask[t];
    const int y = target_idx[t];
    float dwl[kRoMaxCper] = {0.f, 0.f, 0.f, 0.f};
    for (int j = warp; j < D; j += kRoWarps) {
        if (pairs.s_ptr[j] < 0) continue;
        const float dl = mk * scale * (expf(logprobs[(size_t)t * D + j]) - (j == y ? 1.f : 0.f));
        const int i1 = pairs.s_off[j + 1];
        for (int i0 = pairs.s_off[j]; i0 < i1; i0 += 4) {
            RoItem it[4];
            float hv[4][kRoMaxCper];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                it[u].hidx = -1;
                it[u].gidx = g_cap;                        // (skipped below)
                it[u].sign = 0.f;
                if (i0 + u < i1) it[u] = i0 + u < kRoItems ? items[i0 + u] : resolve(i0 + u, j);
#pragma unroll
                for (int q = 0; q < kRoMaxCper; ++q)
                    hv[u][q] = (it[u].hidx >= 0 && lane + 32 * q < C) ? __ldg(HL + (size_t)it[u].hidx * C + lane + 32 * q) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (i0 + u >= i1 || it[u].gidx >= g_cap) continue;      // overflow already flagged by rows_zero_kernel
                const float sdl = it[u].sign * dl;
#pragma unroll
                for (int q = 0; q < kRoMaxCper; ++q)
                    if (lane + 32 * q < C) {
                        const float h = hv[u][q];
                        dwl[q] = fmaf(sdl, h, dwl[q]);
                        const float da = act == SCONE_ACT_TANH ? 1.f - h * h : (act == SCONE_ACT_LEAKY_RELU ? (h >= 0.f ? 1.f : 0.01f) : (h > 0.f ? 1.f : 0.f));
                        atomicAdd(GL + (size_t)it[u].gidx * C + lane + 32 * q, sdl * w[q] * da);
                    }
            }
        }
    }
#pragma unroll
    for (int q = 0; q < kRoMaxCper; ++q) s_dw[warp][lane + 32 * q] = dwl[q];
    __syncthreads();
    if (warp == 0) {
        float* pt = partial + (size_t)t * (C + 2);
#pragma unroll
        for (int q = 0; q < kRoMaxCper; ++q)
            if (lane + 32 * q < C) {
                float sacc = s_dw[0][lane + 32 * q];
                for (int k = 1; k < kRoWarps; ++k) sacc += s_dw[k][lane + 32 * q];
                pt[lane + 32 * q] = sacc;
            }
        if (lane == 0) {
            pt[C] = (y >= 0 && y < D) ? -mk * logprobs[(size_t)t * D + y] : 0.f;
            pt[C + 1] = mk;
        }
    }
}

// dwout[c] (+)= sum_t partial[t][c]; nll (+)= sum_t partial[t][C]; count (+)= sum_t partial[t][C+1]: one warp per output, lane l sums
// t = l, l + 32, ... in ascending order, then a fixed butterfly — deterministic
__global__ void __launch_bounds__(256) rows_readout_reduce_kernel(const float* __restrict__ partial, int b, int C, float* __restrict__ dwout,
                                                                 float* __restrict__ nll, float* __restrict__ count, int accumulate) {
    const int lane = threadIdx.x & 31;
    const int cc = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (cc >= C + 2) return;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    int t = lane;
    for (; t + 96 < b; t += 128) {
        s0 += partial[(size_t)t * (C + 2) + cc];
        s1 += partial[(size_t)(t + 32) * (C + 2) + cc];
        s2 += partial[(size_t)(t + 64) * (C + 2) + cc];
        s3 += partial[(size_t)(t + 96) * (C + 2) + cc];
    }
    for (; t < b; t += 32) s0 += partial[(size_t)t * (C + 2) + cc];
    float s = (s0 + s1) + (s2 + s3);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) {
        float* dst = cc < C ? dwout + cc : (cc == C ? nll : count);
        *dst = accumulate ? *dst + s : s;
    }
}

// Next-node accuracy (scone_trajectory_model.py:59-71): thread = trajectory.  preds[t][n_nbrs[t]:] = -100, argmax over all D slots
// (first maximum; a NaN beats numbers, as NumPy), compared with the target; integer counts (atomicAdd on ints is exact).
__global__ void __launch_bounds__(256) accuracy_kernel(const float* __restrict__ logprobs, const int32_t* __restrict__ n_nbrs,
                                                      const int32_t* __restrict__ target_idx, const float* __restrict__ mask, int B, int D,
                                                      int32_t* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    int correct = 0, counted = 0;
    if (t < B && mask[t] != 0.f) {
        const int n = n_nbrs[t];
        float best = 0.f;
        int arg = 0;
        for (int j = 0; j < D; ++j) {
            const float v = j < n ? logprobs[(size_t)t * D + j] : -100.f;
            if (j == 0 || v > best || (v != v && best == best)) {
                best = v;
                arg = j;
            }
        }
        counted = 1;
        correct = arg == target_idx[t] ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        correct += __shfl_xor_sync(0xffffffffu, correct, o);
        counted += __shfl_xor_sync(0xffffffffu, counted, o);
    }
    if ((threadIdx.x & 31) == 0 && counted) {
        atomicAdd(out, correct);
        atomicAdd(out + 1, counted);
    }
}

// Device halves of the host-side metrics (scone_trajectory_model.py:73-108, 42-56): the log-probs never leave the GPU.
//   predict      choice[t] = argmax_j (j < n_nbrs[t] ? logprobs[t][j] : -100), first maximum, NaN beats numbers (as accuracy_kernel)
//   two_target   out[0] += [true > random], out[1] += [true == random] over the masked rows, where true / random are the log-probs
//                of the true target and of the (host-drawn) random other target — exact integer counts
//   nll          out[0] = sum_t -mask_t * logprobs[t][target_t] (one CTA, fixed lane-strided order + fixed tree: deterministic),
//                out[1] = sum_t mask_t
__global__ void __launch_bounds__(256) predict_kernel(const float* __restrict__ logprobs, const int32_t* __restrict__ n_nbrs, int B, int D,
                                                     int32_t* __restrict__ choice) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B) return;
    const int n = n_nbrs[t];
    float best = 0.f;
    int arg = 0;
    for (int j = 0; j < D; ++j) {
        const float v = j < n ? logprobs[(size_t)t * D + j] : -100.f;
        if (j == 0 || v > best || (v != v && best == best)) {
            best = v;
            arg = j;
        }
    }
    choice[t] = arg;
}

__global__ void __launch_bounds__(256) two_target_kernel(const float* __restrict__ logprobs, const int32_t* __restrict__ n_nbrs,
                                                        const int32_t* __restrict__ true_idx, const int32_t* __restrict__ rand_idx,
                                                        const float* __restrict__ mask, int B, int D, int32_t* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    int gt = 0, eq = 0;
    if (t < B && mask[t] != 0.f) {
        const int n = n_nbrs[t], a = true_idx[t], r = rand_idx[t];
        const float tv = (a >= 0 && a < n) ? logprobs[(size_t)t * D + a] : -100.f;     // preds[i, n_nbrs[i]:] = -100 (:84-85)
        const float rv = (r >= 0 && r < n) ? logprobs[(size_t)t * D + r] : -100.f;
        gt = tv > rv ? 1 : 0;
        eq = tv == rv ? 1 : 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        gt += __shfl_xor_sync(0xffffffffu, gt, o);
        eq += __shfl_xor_sync(0xffffffffu, eq, o);
    }
    if ((threadIdx.x & 31) == 0 && (gt | eq)) {
        atomicAdd(out, gt);
        atomicAdd(out + 1, eq);
    }
}

__global__ void __launch_bounds__(1024) nll_kernel(const float* __restrict__ logprobs, const int32_t* __restrict__ target_idx,
                                                  const float* __restrict__ mask, int B, int D, float* __restrict__ out) {
    __shared__ float s_n[32], s_c[32];
    float nll = 0.f, cnt = 0.f;
    for (int t = threadIdx.x; t < B; t += blockDim.x) {
        const float mk = mask[t];
        const int y = target_idx[t];
        if (mk != 0.f && y >= 0 && y < D) nll += -mk * logprobs[(size_t)t * D + y];
        cnt += mk;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        nll += __shfl_xor_sync(0xffffffffu, nll, o);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if ((threadIdx.x & 31) == 0) {
        s_n[threadIdx.x >> 5] = nll;
        s_c[threadIdx.x >> 5] = cnt;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
        nll = s_n[threadIdx.x];
        cnt = s_c[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            nll += __shfl_xor_sync(0xffffffffu, nll, o);
            cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        }
        if (threadIdx.x == 0) {
            out[0] = nll;
            out[1] = cnt;
        }
    }
}

constexpr int kDwCtas = 148 * 2;

template <int CIN, int COUT, int ACT>
int launch_rows_bwd(const scone_complex* cx, int b, const float* G, const float* Hin, float* Gprev, float* Abuf, const float* W0,
                    const float* W1, const float* W2, const uint32_t* rows, const int* n_ptr, const uint32_t* bmG, const uint32_t* bmH,
                    int a_cap, int* overflow, const uint32_t* prefG, const uint32_t* prefH, cudaStream_t st) {
    using Gm = SlabGeom<COUT, 16>;
    constexpr int NT = CIN / 8;
    const size_t smem = (size_t)3 * Gm::KS * NT * 32 * sizeof(uint4);
    static bool configured = false;
    if (!configured) {
        SCONE_CUDA(cudaFuncSetAttribute(rows_bwd_kernel<CIN, COUT, ACT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SCONE_CUDA(cudaFuncSetAttribute(rows_bwd_kernel<CIN, COUT, ACT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    if (prefG != nullptr)
        rows_bwd_kernel<CIN, COUT, ACT, true><<<cx->num_sms, kRowsThreads, smem, st>>>(G, Hin, Gprev, Abuf, W0, W1, W2, cx->d_mptr, cx->d_ment, rows,
                                                                                     n_ptr, b, bmG, bmH, a_cap, overflow,
                                                                                     scone_prof_row_counter(SCONE_K_LAYER_BWD), prefG, prefH, cx->E);
    else
        rows_bwd_kernel<CIN, COUT, ACT, false><<<cx->num_sms, kRowsThreads, smem, st>>>(G, Hin, Gprev, Abuf, W0, W1, W2, cx->d_mptr, cx->d_ment, rows,
                                                                                      n_ptr, b, bmG, bmH, a_cap, overflow,
                                                                                      scone_prof_row_counter(SCONE_K_LAYER_BWD), prefG, prefH, cx->E);
    SCONE_LAUNCHED();
    return 0;
}

template <int CIN, int COUT>
int dispatch_rows_bwd(const scone_complex* cx, int act, int b, const float* G, const float* Hin, float* Gprev, float* Abuf,
                      const float* W0, const float* W1, const float* W2, const uint32_t* rows, const int* n_ptr, const uint32_t* bmG,
                      const uint32_t* bmH, int a_cap, int* overflow, const uint32_t* prefG, const uint32_t* prefH, cudaStream_t st) {
    switch (act) {
        case SCONE_ACT_TANH:
            return launch_rows_bwd<CIN, COUT, SCONE_ACT_TANH>(cx, b, G, Hin, Gprev, Abuf, W0, W1, W2, rows, n_ptr, bmG, bmH, a_cap, overflow, prefG, prefH, st);
        case SCONE_ACT_LEAKY_RELU:
            return launch_rows_bwd<CIN, COUT, SCONE_ACT_LEAKY_RELU>(cx, b, G, Hin, Gprev, Abuf, W0, W1, W2, rows, n_ptr, bmG, bmH, a_cap, overflow, prefG, prefH, st);
        case SCONE_ACT_RELU:
            return launch_rows_bwd<CIN, COUT, SCONE_ACT_RELU>(cx, b, G, Hin, Gprev, Abuf, W0, W1, W2, rows, n_ptr, bmG, bmH, a_cap, overflow, prefG, prefH, st);
    }
    scone_set_error("unknown activation %d", act);
    return 2;
}

template <int CIN, int COUT>
int launch_rows_dw(const scone_complex* cx, const float* Hin, const uint32_t* bmH, const float* Abuf, const uint32_t* rows,
                   const int* n_ptr, int a_cap, float* dW, int accumulate, float* ws, const uint32_t* prefH, bool hin_by_list,
                   cudaStream_t st) {
    if (hin_by_list)
        rows_dw_kernel<CIN, COUT, true, true><<<kDwCtas, 256, 0, st>>>(Hin, bmH, Abuf, rows, n_ptr, a_cap, ws, prefH);
    else if (prefH != nullptr)
        rows_dw_kernel<CIN, COUT, true, false><<<kDwCtas, 256, 0, st>>>(Hin, bmH, Abuf, rows, n_ptr, a_cap, ws, prefH);
    else
        rows_dw_kernel<CIN, COUT, false, false><<<kDwCtas, 256, 0, st>>>(Hin, bmH, Abuf, rows, n_ptr, a_cap, ws, prefH);
    SCONE_LAUNCHED();
    constexpr int DW = 3 * CIN * COUT;
    rows_reduce_kernel<<<(DW + 31) / 32, 256, 0, st>>>(ws, kDwCtas, DW, dW, accumulate);
    SCONE_LAUNCHED();
    return 0;
}

template <int COUT, int ACT>
int launch_rows_l0_fwd_act(const scone_complex* cx, int b, const float* X, const float* W0, const float* W1, const float* W2, float* Hout,
                           const uint32_t* rows, const int* n_ptr, uint32_t* bm_next, int out_cap, int* overflow, cudaStream_t st) {
    const int grid = cx->num_sms * 8;
    if (out_cap > 0)
        rows_layer0_fwd_kernel<COUT, ACT, true><<<grid, 256, 0, st>>>(X, Hout, W0, W1, W2, cx->d_mptr, cx->d_ment, rows, n_ptr, b, bm_next, out_cap, overflow, cx->E);
    else
        rows_layer0_fwd_kernel<COUT, ACT, false><<<grid, 256, 0, st>>>(X, Hout, W0, W1, W2, cx->d_mptr, cx->d_ment, rows, n_ptr, b, bm_next, out_cap, overflow, cx->E);
    SCONE_LAUNCHED();
    return 0;
}

template <int COUT>
int launch_rows_l0_fwd(const scone_complex* cx, int act, int b, const float* X, const float* W0, const float* W1, const float* W2,
                       float* Hout, const uint32_t* rows, const int* n_ptr, uint32_t* bm_next, int out_cap, int* overflow, cudaStream_t st) {
    switch (act) {
        case SCONE_ACT_TANH: return launch_rows_l0_fwd_act<COUT, SCONE_ACT_TANH>(cx, b, X, W0, W1, W2, Hout, rows, n_ptr, bm_next, out_cap, overflow, st);
        case SCONE_ACT_LEAKY_RELU: return launch_rows_l0_fwd_act<COUT, SCONE_ACT_LEAKY_RELU>(cx, b, X, W0, W1, W2, Hout, rows, n_ptr, bm_next, out_cap, overflow, st);
        case SCONE_ACT_RELU: return launch_rows_l0_fwd_act<COUT, SCONE_ACT_RELU>(cx, b, X, W0, W1, W2, Hout, rows, n_ptr, bm_next, out_cap, overflow, st);
    }
    scone_set_error("unknown activation %d", act);
    return 2;
}

}  // namespace

int scone_accuracy_launch(int B, int D, const float* logprobs, const int32_t* n_nbrs, const int32_t* target_idx, const float* mask,
                          int32_t* out, cudaStream_t st) {
    SCONE_CUDA(cudaMemsetAsync(out, 0, 2 * sizeof(int32_t), st));
    if (B > 0) {
        accuracy_kernel<<<(B + 255) / 256, 256, 0, st>>>(logprobs, n_nbrs, target_idx, mask, B, D, out);
        SCONE_LAUNCHED();
    }
    return 0;
}

int scone_predict_launch(int B, int D, const float* logprobs, const int32_t* n_nbrs, int32_t* choice, cudaStream_t st) {
    if (B > 0) {
        predict_kernel<<<(B + 255) / 256, 256, 0, st>>>(logprobs, n_nbrs, B, D, choice);
        SCONE_LAUNCHED();
    }
    return 0;
}

int scone_two_target_launch(int B, int D, const float* logprobs, const int32_t* n_nbrs, const int32_t* true_idx, const int32_t* rand_idx,
                            const float* mask, int32_t* out, cudaStream_t st) {
    SCONE_CUDA(cudaMemsetAsync(out, 0, 2 * sizeof(int32_t), st));
    if (B > 0) {
        two_target_kernel<<<(B + 255) / 256, 256, 0, st>>>(logprobs, n_nbrs, true_idx, rand_idx, mask, B, D, out);
        SCONE_LAUNCHED();
    }
    return 0;
}

int scone_nll_launch(int B, int D, const float* logprobs, const int32_t* target_idx, const float* mask, float* out, cudaStream_t st) {
    nll_kernel<<<1, 1024, 0, st>>>(logprobs, target_idx, mask, B, D, out);
    SCONE_LAUNCHED();
    return 0;
}

bool scone_rows_supported(const scone_complex* cx, int n_layers, const int32_t* hidden) {
    if (g_scone_dense_kernel == 0 || cx->d_mptr == nullptr || cx->D > kRoMaxD) return false;   // (readout / cone kernels: degree <= kRoMaxD)
    for (int l = 0; l < n_layers; ++l)
        if (hidden[l] != 16 && hidden[l] != 32) return false;
    return true;
}
int64_t scone_rows_dw_workspace_bytes(int cin, int cout) { return (int64_t)kDwCtas * 3 * (cin > 1 ? cin : 1) * cout * sizeof(float); }

int scone_rows_flows(const scone_complex* cx, int b, const int32_t* traj_ptr, const int32_t* flow_edge, const float* flow_val, float* X,
                     uint32_t* bmX, uint32_t* bm_next, bool clear, bool tmaj, cudaStream_t st, const uint32_t* bm_filter, size_t sum_off) {
    if (clear)
        rows_flows_kernel<true><<<b, 256, 0, st>>>(traj_ptr, flow_edge, flow_val, cx->d_rank, X, bmX, bm_next, cx->d_mptr, cx->d_ment, cx->E, b, tmaj,
                                                   bm_filter, sum_off);
    else
        rows_flows_kernel<false><<<b, 256, 0, st>>>(traj_ptr, flow_edge, flow_val, cx->d_rank, X, bmX, bm_next, cx->d_mptr, cx->d_ment, cx->E, b, tmaj,
                                                    bm_filter, sum_off);
    SCONE_LAUNCHED();
    return 0;
}

int scone_rows_mark(const scone_complex* cx, int b, const uint32_t* rows, const int* n_dev, uint32_t* bm_next, int list_cap,
                    cudaStream_t st, bool tmaj, size_t sum_off, const uint32_t* bm_filter) {
    rows_mark_kernel<<<cx->num_sms * 8, 256, 0, st>>>(rows, n_dev, cx->d_mptr, cx->d_ment, b, bm_next, list_cap, sum_off, cx->E, tmaj, bm_filter);
    SCONE_LAUNCHED();
    return 0;
}

int scone_rows_cone(const scone_complex* cx, int b, const int32_t* last_nodes, uint32_t* const* bm_levels, int n_levels, size_t sum_off,
                    int* overflow_dev, cudaStream_t st) {
    SCONE_REQUIRE(cx->D <= kRoMaxD, "scone_rows_cone: max degree <= %d", kRoMaxD);
    SCONE_REQUIRE(n_levels >= 1 && n_levels <= kConeMaxLevels && sum_off > 0, "scone_rows_cone: 1..%d levels, two-level bitmaps", kConeMaxLevels);
    ConeBitmaps cone;
    for (int l = 0; l < kConeMaxLevels; ++l) cone.bm[l] = l < n_levels ? bm_levels[l] : nullptr;
    rows_cone_kernel<<<b, 256, 0, st>>>(last_nodes, cx->d_nbrhoods, cx->d_inc_ptr, cx->d_inc_ent, cone, n_levels, cx->d_mptr, cx->d_ment, cx->N,
                                       cx->D, cx->E, sum_off, overflow_dev);
    SCONE_LAUNCHED();
    return 0;
}

// two-level bitmaps: the summary words of bm start at bm + sum_off
static long long summary_words(const scone_complex* cx, int b) { return (((long long)cx->E * b + 31) / 32 + 31) / 32; }

int scone_compact_rows_summary(const scone_complex* cx, int b, const uint32_t* bm, size_t sum_off, uint32_t* list, int* n_dev,
                               unsigned long long* tickets, cudaStream_t st, uint32_t* pref_out, long long list_cap) {
    const long long n1 = summary_words(cx, b);
    const int max_grid = cx->num_sms * 4 < 1024 ? cx->num_sms * 4 : 1024;     // (1024 single-chunk CTAs measured slower: 48 vs 34 us)
    // summary words per thread: 16 when that still fills the GPU, else 4, else 1 (a small / dense bitmap must not end up in one warp)
    const int wpt = n1 >= (long long)16 * 256 * cx->num_sms ? 16 : (n1 >= (long long)4 * 256 * cx->num_sms ? 4 : 1);
    const long long chunk = (long long)wpt * 256;
    int grid = max_grid;
    if (n1 < (long long)grid * chunk) grid = (int)((n1 + chunk - 1) / chunk);
    if (grid < 1) grid = 1;
    SCONE_REQUIRE((n1 + grid - 1) / grid <= (long long)kSumMaxChunks * chunk, "scone_compact_rows_summary: bitmap too large for %d CTAs", grid);
    SCONE_CUDA(cudaMemsetAsync(tickets, 0, (size_t)grid * 8, st));
    if (wpt == 16) compact_summary_kernel<16><<<grid, 256, 0, st>>>(bm, bm + sum_off, n1, list, n_dev, tickets, pref_out, list_cap);
    else if (wpt == 4) compact_summary_kernel<4><<<grid, 256, 0, st>>>(bm, bm + sum_off, n1, list, n_dev, tickets, pref_out, list_cap);
    else compact_summary_kernel<1><<<grid, 256, 0, st>>>(bm, bm + sum_off, n1, list, n_dev, tickets, pref_out, list_cap);
    SCONE_LAUNCHED();
    return 0;
}

// bms[0 .. count): two-level bitmaps to clear; bms[master] must contain every bit set in any of them and carry the summary bits
int scone_clear_summary(const scone_complex* cx, int b, uint32_t* const* bms, int count, int master, size_t sum_off, cudaStream_t st) {
    SCONE_REQUIRE(count >= 1 && count <= kClearMax && master >= 0 && master < count, "scone_clear_summary: 1..%d bitmaps", kClearMax);
    const long long n1 = summary_words(cx, b);
    long long grid = ((n1 + 3) / 4 + 255) / 256;
    if (grid > cx->num_sms * 8) grid = cx->num_sms * 8;
    if (grid < 1) grid = 1;
    ClearList list;
    for (int i = 0; i < kClearMax; ++i) list.bm[i] = i < count ? bms[i] : nullptr;
    clear_summary_kernel<<<(unsigned)grid, 256, 0, st>>>(list, count, bms[master] + sum_off, sum_off, n1);
    SCONE_LAUNCHED();
    return 0;
}

// out_cap > 0: compact storage (row rows[i] of Hout at index i, at most out_cap rows)
int scone_rows_layer0_forward(const scone_complex* cx, int act, int b, int cout, const float* X, const float* W0, const float* W1,
                              const float* W2, float* Hout, const uint32_t* rows, const int* n_dev, uint32_t* bm_next, int out_cap,
                              int* overflow_dev, cudaStream_t st) {
    if (cout == 16) return launch_rows_l0_fwd<16>(cx, act, b, X, W0, W1, W2, Hout, rows, n_dev, bm_next, out_cap, overflow_dev, st);
    if (cout == 32) return launch_rows_l0_fwd<32>(cx, act, b, X, W0, W1, W2, Hout, rows, n_dev, bm_next, out_cap, overflow_dev, st);
    scone_set_error("scone_rows_layer0_forward: unsupported width %d", cout);
    return 2;
}

// g_cap > 0: G is compact (row rows[i] at index i)
int scone_rows_layer0_backward(const scone_complex* cx, int b, int cout, const float* X, const float* G, const uint32_t* rows,
                               const int* n_dev, float* dW, int accumulate, float* ws, int g_cap, cudaStream_t st) {
#define SCONE_L0B(CO)                                                                                                         \
    if (g_cap > 0) rows_layer0_bwd_kernel<CO, true><<<kDwCtas, 32 * kL0bWarps, 0, st>>>(X, G, cx->d_mptr, cx->d_ment, rows, n_dev, b, ws, g_cap, cx->E); \
    else rows_layer0_bwd_kernel<CO, false><<<kDwCtas, 32 * kL0bWarps, 0, st>>>(X, G, cx->d_mptr, cx->d_ment, rows, n_dev, b, ws, g_cap, cx->E);
    if (cout == 16) { SCONE_L0B(16) }
    else if (cout == 32) { SCONE_L0B(32) }
    else {
        scone_set_error("scone_rows_layer0_backward: unsupported width %d", cout);
        return 2;
    }
#undef SCONE_L0B
    SCONE_LAUNCHED();
    rows_reduce_kernel<<<(3 * cout + 31) / 32, 256, 0, st>>>(ws, kDwCtas, 3 * cout, dW, accumulate);
    SCONE_LAUNCHED();
    return 0;
}

// prefG / prefH != NULL: compact storage of G, Hin, Gprev (a_cap then also bounds the rows of Gprev); hin_by_list: Hin's row set
// IS this list (cone pipeline), row rows[i] at index i
int scone_rows_backward(const scone_complex* cx, int act, int b, int cin, int cout, const float* G, const float* Hin, float* Gprev,
                        float* Abuf, const float* W0, const float* W1, const float* W2, const uint32_t* rows, const int* n_dev,
                        const uint32_t* bmG, const uint32_t* bmH, int a_cap, int* overflow_dev, float* dW, int accumulate, float* ws,
                        const uint32_t* prefG, const uint32_t* prefH, bool hin_by_list, cudaStream_t st) {
#define SCONE_RB_CASE(CI, CO)                                                                                                     \
    if (cin == CI && cout == CO) {                                                                                                \
        if (dispatch_rows_bwd<CI, CO>(cx, act, b, G, Hin, Gprev, Abuf, W0, W1, W2, rows, n_dev, bmG, bmH, a_cap, overflow_dev,      \
                                      prefG, prefH, st))                                                                          \
            return 1;                                                                                                             \
        return launch_rows_dw<CI, CO>(cx, Hin, bmH, Abuf, rows, n_dev, a_cap, dW, accumulate, ws, prefH, hin_by_list, st);          \
    }
    SCONE_RB_CASE(16, 16)
    SCONE_RB_CASE(16, 32)
    SCONE_RB_CASE(32, 16)
    SCONE_RB_CASE(32, 32)
#undef SCONE_RB_CASE
    scone_set_error("scone_rows_backward: unsupported widths %d -> %d", cin, cout);
    return 2;
}

// Readout over compact storage (see rows_readout_*_kernel).  Forward: log-probs; with bmG != NULL also the bits of G_L's rows and
// (bm_cand != NULL) the candidate bits one hop further — the caller cleared both bitmaps.
int scone_rows_readout_forward(const scone_complex* cx, int b, int C, const float* HL, const float* wout, const int32_t* last_nodes,
                               float* logprobs, const uint32_t* bmH, const uint32_t* prefH, uint32_t* bmG, uint32_t* bm_cand,
                               cudaStream_t st) {
    SCONE_REQUIRE(C >= 1 && C <= 32 * kRoMaxCper && cx->D <= kRoMaxD, "scone_rows_readout: C <= %d and max degree <= %d", 32 * kRoMaxCper, kRoMaxD);
    rows_readout_fwd_kernel<<<b, 32 * kRoWarps, 0, st>>>(HL, wout, last_nodes, cx->d_nbrhoods, cx->d_inc_ptr, cx->d_inc_ent, logprobs, bmH,
                                                        prefH, bmG, bm_cand, cx->d_mptr, cx->d_ment, cx->N, cx->D, cx->E, C);
    SCONE_LAUNCHED();
    return 0;
}

// Gradient part, after bmG was compacted (prefG, n_dev = number of rows of G_L): zero the rows, accumulate, reduce the partials.
int scone_rows_readout_backward(const scone_complex* cx, int act, int b, int C, const float* HL, const float* wout,
                                const int32_t* last_nodes, const float* logprobs, const int32_t* target_idx, const float* mask,
                                float scale, float* GL, const int* n_dev, int g_cap, int* overflow_dev, float* dwout, float* nll_sum,
                                float* count, int accumulate, float* ws, const uint32_t* bmH, const uint32_t* prefH, const uint32_t* bmG,
                                const uint32_t* prefG, cudaStream_t st) {
    rows_zero_kernel<<<cx->num_sms * 4, 256, 0, st>>>(reinterpret_cast<float4*>(GL), n_dev, g_cap, C / 4, overflow_dev);
    SCONE_LAUNCHED();
    rows_readout_bwd_kernel<<<b, 32 * kRoWarps, 0, st>>>(HL, wout, last_nodes, cx->d_nbrhoods, cx->d_inc_ptr, cx->d_inc_ent, logprobs, target_idx,
                                                        mask, scale, GL, ws, bmH, prefH, bmG, prefG, g_cap, act, cx->N, cx->D, cx->E, C);
    SCONE_LAUNCHED();
    rows_readout_reduce_kernel<<<(C + 2 + 7) / 8, 256, 0, st>>>(ws, b, C, dwout, nll_sum, count, accumulate);
    SCONE_LAUNCHED();
    return 0;
}
