// scone_fused.cu — pipeline 4: the TRAJECTORY-FUSED path behind the model-level entry points (uniform hidden width 16 / 32,
// at most 3 conv layers).  Two kernels per micro-batch instead of the ~25 launches of the bitmap pipeline:
//
//   fused_plan_kernel   (weight-independent integer work, one CTA per trajectory; the HASH plan — the fallback of the table plan in
//                        scone_plan_table.cu, which produces the same headers and programs from per-node operator rows)
//        receptive cone of the readout (trajectory_experiments.py:151,298-303: the log-probs read H_L only at the edges incident
//        to the neighbours of the last node; one merged-operator hop further down per layer), intersected layer by layer with the
//        structural support of the flows (no bias, act(0) = 0: a row with no live neighbour below is exactly zero) -> per layer
//        the LIVE rows in ascending edge order, and for every live row its GATHER PROGRAM: {index of the live neighbour row one
//        layer below, both integer operator coefficients}, plus the transposed programs the backward walks and the readout
//        pairs.  Everything lives in a shared-memory hash set (edge -> slot); nothing is proportional to E * batch: no bitmaps,
//        no dense X, no compaction, no clearing.
//   fused_traj_kernel   (persistent CTAs, trajectories assigned statically = deterministic)
//        layer 1 from the three exact scalars of each live row; conv layers l >= 2 as gather (shared memory) -> 3xTF32 mma.sync
//        product against the weights staged once per CTA -> activation; readout + padded log-softmax + NLL
//        (trajectory_experiments.py:151-152, scone_trajectory_model.py:46-54); backward through the transposed programs with
//        the weight gradients accumulated in mma accumulator REGISTERS across all trajectories of the CTA; one partial vector
//        per CTA, reduced in CTA order by fused_reduce_kernel.  Activations and gradients of a trajectory never leave the SM.
//
// All capacities are STATIC bounds measured once per complex (scone_table_build: the cone of every possible last node), so a
// micro-batch cannot overflow: the hash set holds |T_0| <= bound entries, a layer has at most |T_1| <= bound rows, the program
// arena is sized for the worst case.  A trajectory whose rows do not fit the shared-memory row store runs in the BIG variant of
// the same kernel (rows in a per-CTA global scratch).
#include <algorithm>
#include <cub/device/device_radix_sort.cuh>
#include "common.cuh"
#include "fused.cuh"

namespace {

#include "slab_common.cuh"

constexpr int kTrajThreads = 256;
constexpr int kFuMaxD = SCONE_MAX_DEGREE;
constexpr uint32_t kNoRow = 0xFFFFu;
constexpr uint32_t kFlaggedKey = 0xFFFFFFu;   // sort key of a trajectory the plan kernel flagged (overflow): belongs to no launch

template <int ACT>
__device__ __forceinline__ float fu_act(float z) {
    if (ACT == SCONE_ACT_TANH) return scone_tanh(z);
    if (ACT == SCONE_ACT_LEAKY_RELU) return z >= 0.f ? z : 0.01f * z;
    return fmaxf(z, 0.f);
}
template <int ACT>
__device__ __forceinline__ float fu_dact(float h) {        // derivative through the OUTPUT h = act(z)
    if (ACT == SCONE_ACT_TANH) return 1.f - h * h;
    if (ACT == SCONE_ACT_LEAKY_RELU) return h >= 0.f ? 1.f : 0.01f;
    return h > 0.f ? 1.f : 0.f;
}

__device__ __forceinline__ int align2(int x) { return (x + 1) & ~1; }

// ---------------------------------------------------------------------------------------------------------------------
// shared-memory hash set of internal edge ids (open addressing, linear probing; the table can never fill: HS > static bound)
// ---------------------------------------------------------------------------------------------------------------------
struct EdgeSet {
    int* keys;
    int mask, shift;
    __device__ __forceinline__ unsigned home(int e) const { return ((unsigned)e * 2654435761u) >> shift; }
    // returns the slot; is_new = this call created the entry
    __device__ __forceinline__ int insert(int e, bool& is_new) {
        unsigned h = home(e);
        is_new = false;
        for (int probes = 0; probes <= mask; ++probes) {
            const int old = atomicCAS(&keys[h], -1, e);
            if (old == -1) {
                is_new = true;
                return (int)h;
            }
            if (old == e) return (int)h;
            h = (h + 1) & mask;
        }
        return -1;                                        // full (only possible in bound mode)
    }
    __device__ __forceinline__ int find(int e) const {    // (the table always has empty slots: load <= 3/4)
        unsigned h = home(e);
        int k = keys[h];
        while (k != e) {
            if (k == -1) return -1;
            h = (h + 1) & mask;
            k = keys[h];
        }
        return (int)h;
    }
};

// (neighbour slot j, incident edge) pairs of the last node, flattened (same enumeration as the row-list readout kernels)
struct FuPairs {
    int s_ptr[kFuMaxD], s_off[kFuMaxD + 1];
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
    __device__ __forceinline__ int slot_of(int i, int D) const {
        int j = 0;
        while (j + 1 < D && s_off[j + 1] <= i) ++j;
        return j;
    }
};

// ---------------------------------------------------------------------------------------------------------------------
// the plan of one trajectory (one CTA of THREADS threads)
//
//   hash set      T_0 of the last node, loaded from the cone table (level = highest cone level of the edge; level 0 = the ring whose
//                 flow values can reach a row of T_1); the flow entries of the trajectory that fall into it get their value x —
//                 the rest of the path is too far from the last node to matter and is never touched again
//   live rows     PUSHED from below: a row of layer 1 is live iff it is in T_1 and a flow edge sits in its merged operator row,
//                 i.e. iff it is in the merged row of a flow edge (the operators are symmetric); a row of layer l iff it is in T_l
//                 and in the merged row of a live row of layer l - 1.  Cost follows the flows and the live rows, not the cone.
//   rank          live rows of a layer are numbered by ascending edge id: the deterministic row order of every list
//   one scan      the merged rows of the live rows of a layer are walked ONCE (global loads + hash lookups); the hash slot of every
//                 entry is kept in shared memory (ebuf) and serves the layer's forward program (or the layer-1 scalars), the marking
//                 of the next layer's live rows and the next layer's transposed program
//   FG            flow-gradient plan (scone_model_vjp_flows_*): every flow entry of T_0 seeds layer-1 liveness whatever its value (dL/dx
//                 at an entry whose value is 0 reads the rows a non-zero value would make live; they hold exact zeros in the forward),
//                 and the layer-0 transposed program goes to a.fg_off[t] (fused_flow_program)
// ---------------------------------------------------------------------------------------------------------------------
template <int THREADS, bool FG>
__device__ __forceinline__ void plan_trajectory(const PlanArgs& a, const int t, unsigned char* sm) {
    constexpr int QUADS = THREADS / 4;
    const int HS = a.HS, LV = a.LV, EC = a.EC, L = a.L, D = a.D;
    int* keys = reinterpret_cast<int*>(sm);                          // [HS] internal edge id, -1 = empty
    float* xv = reinterpret_cast<float*>(keys + HS);                 // [HS] flow value of the edge
    int* lvl = reinterpret_cast<int*>(xv + HS);                      // [HS] bits 0-7: cone level (0 = flow edge outside the cone); bit 8 + l: marked live in layer l
    uint16_t* idx0 = reinterpret_cast<uint16_t*>(lvl + HS);          // [3][HS] row index of the edge in the live list of layer l: idx0 + (l % 3) * HS
    int* rowcnt = reinterpret_cast<int*>(idx0 + 3 * HS);             // [LV + 4] entries per ranked row -> exclusive scan
    int* erow = rowcnt + LV + 4;                                     // [LV + 4] start of the row's entries in ebuf
    int* live_edge = erow + LV + 4;                                  // [LV] edge id of the k-th live row (unordered)
    uint16_t* live = reinterpret_cast<uint16_t*>(live_edge + LV);    // [LV] hash slot of the k-th live row (unordered)
    uint16_t* rankA = live + LV;                                     // [LV] hash slot of the row with rank r (ping)
    uint16_t* rankB = rankA + LV;                                    // [LV] (pong)
    uint16_t* ebuf = rankB + LV;                                      // [EC] hash slot of every merged-row entry of the scanned rows
    __shared__ FuPairs pairs;
    __shared__ int s_nhash, s_nlive, s_ovf, s_warp[THREADS / 32];
    __shared__ unsigned s_piece;

    const int tid = threadIdx.x, lane = tid & 31, ql = tid & 3;
    const unsigned qmask = 0xFu << (lane & ~3);
    int* hdr = a.hdr + (size_t)t * kFusedHdrW;
    // a table of this tier overflowed: tier 0 hands the trajectory to tier 1 (tables sized by the measured bounds)
    auto give_up = [&]() {
        if (tid == 0) {
            if (a.retry != nullptr) {
                hdr[0] = kFusedFlagRetry;
                a.retry[atomicAdd(a.n_retry, 1)] = t;
            } else {
                hdr[0] = kFusedFlagOverflow;
                *a.overflow = 1;
            }
        }
    };
    for (int i = tid; i < HS; i += THREADS) {
        keys[i] = -1;
        xv[i] = 0.f;
        lvl[i] = 0;
    }
    for (int i = tid; i < 3 * HS; i += THREADS) idx0[i] = (uint16_t)kNoRow;
    if (tid == 0) s_nhash = s_ovf = s_nlive = 0;
    const int last = a.last_nodes[t];
    const bool last_ok = last >= 0 && last < a.N;
    const int total_pairs = pairs.setup(a.nbrhoods, a.inc_ptr, last, last_ok, D);     // (barriers inside: the tables are initialised)
    EdgeSet set{keys, HS - 1, a.hshift};
    const int hash_cap = (HS * 3) / 4;
    // arena allocation for one piece (thread 0 allocates, everybody gets the word offset)
    auto alloc = [&](int words) -> unsigned {
        __syncthreads();
        if (tid == 0) {
            const unsigned long long w = (unsigned long long)align2(words);
            const unsigned long long o = atomicAdd(a.bump, w);
            if (o + w > a.arena_words) {
                s_ovf = 2;
                s_piece = 0u;
            } else {
                s_piece = (unsigned)o;
            }
        }
        __syncthreads();
        return s_piece;
    };
    const int fp0 = a.traj_ptr[t], fp1 = a.traj_ptr[t + 1];

    // ---- the cone of the last node, from the table ----
    {
        const unsigned c0 = last_ok ? a.cone_ptr[last] : 0u, c1 = last_ok ? a.cone_ptr[last + 1] : 0u;
        const int n_cone = (int)(c1 - c0);
        if (n_cone > hash_cap) {                           // (uniform) this tier's table is too small
            give_up();
            return;
        }
        for (int i = tid; i < n_cone; i += THREADS) {
            const uint32_t en = a.cone_ent[c0 + i];
            bool is_new;
            const int s = set.insert((int)(en & 0x3FFFFFFFu), is_new);
            lvl[s] = (int)(en >> 30);
        }
        if (tid == 0) s_nhash = n_cone;
    }
    __syncthreads();
    // ---- flows: only edges of T_0 can reach a cone row ----
    for (int p = fp0 + tid; p < fp1; p += THREADS) {
        const int eo = a.flow_edge[p];
        if (eo < 0 || eo >= a.E) continue;
        const int s = set.find(a.rank[eo]);
        if (s >= 0) xv[s] = a.flow_val[p];
    }
    __syncthreads();
    // marks (once) the cone edge in slot s2 as a live row of layer l
    auto mark = [&](int s2, int l) {
        const int bit = 1 << (8 + l);
        const int old = atomicOr(&lvl[s2], bit);
        if (!(old & bit)) {
            const int k = atomicAdd(&s_nlive, 1);
            if (k < LV) {
                live[k] = (uint16_t)s2;
                live_edge[k] = keys[s2];
            } else {
                s_ovf = 1;
            }
        }
    };
    // ranks the s_nlive live rows by edge id: idx[slot] = rank, byrank[rank] = slot; returns the count
    auto rank_live = [&](uint16_t* idx, uint16_t* byrank) -> int {
        __syncthreads();
        const int n = min(s_nlive, LV);
        for (int k = tid; k < n; k += THREADS) {
            const int e = live_edge[k];
            int r = 0;
            for (int m = 0; m < n; ++m) r += live_edge[m] < e ? 1 : 0;
            idx[live[k]] = (uint16_t)r;
            byrank[r] = live[k];
        }
        __syncthreads();
        return n;
    };

    // ---- layer 1: live rows = cone edges in the merged row of a flow edge with a non-zero value (FG: any value) ----
    for (int p = fp0 + (tid >> 2); p < fp1; p += QUADS) {
        const int eo = a.flow_edge[p];
        if (eo < 0 || eo >= a.E) continue;                 // (same decision on the four lanes of the quad)
        const int e = a.rank[eo];
        const int s = set.find(e);
        if (s < 0 || (!FG && xv[s] == 0.f)) continue;
        const int p1 = a.mptr[e + 1];
        for (int q = a.mptr[e] + ql; q < p1; q += 4) {
            const int s2 = set.find(a.ment[q].x);
            if (s2 >= 0 && (lvl[s2] & 0xFF) >= 1) mark(s2, 1);
        }
    }
    uint16_t *rcur = rankA, *rnext = rankB;
    int n_cur = rank_live(idx0 + 1 * HS, rcur);
    if (s_ovf) {
        give_up();
        return;
    }
    int n_l[kFusedMaxL + 1] = {0, 0, 0, 0};
    unsigned off_l1 = 0, off_f[kFusedMaxL + 1] = {0, 0, 0, 0}, off_b[kFusedMaxL + 1] = {0, 0, 0, 0};
    int tot_f[kFusedMaxL + 1] = {0, 0, 0, 0}, tot_b[kFusedMaxL + 1] = {0, 0, 0, 0};

    // program of the n_cur scanned rows against the row indices `idx`: rowptr + entries {row | own << 31, coefficients} into the
    // arena, entries in column order (count pass, scan, fill pass — all over the shared-memory slot buffer)
    auto emit_program = [&](const uint16_t* byrank, int n_rows, const uint16_t* idx, int& total_out) -> unsigned {
        for (int r = tid >> 2; r < n_rows; r += QUADS) {
            const int b0 = erow[r], b1 = erow[r + 1];
            int c = 0;
            for (int i = b0 + ql; i < b1; i += 4) {
                const uint32_t s2 = ebuf[i];
                if (s2 != kNoRow && idx[s2] != (uint16_t)kNoRow) ++c;
            }
            c += __shfl_xor_sync(qmask, c, 1);
            c += __shfl_xor_sync(qmask, c, 2);
            if (ql == 0) rowcnt[r] = c;
        }
        __syncthreads();
        const int total = fused_block_scan_excl<THREADS>(rowcnt, n_rows, s_warp);
        total_out = total;
        const unsigned off = alloc(align2(n_rows + 1) + 2 * total);
        if (!s_ovf) {
            int* pdst = reinterpret_cast<int*>(a.arena + off);
            int2* edst = reinterpret_cast<int2*>(a.arena + off + align2(n_rows + 1));
            for (int r = tid; r <= n_rows; r += THREADS) pdst[r] = rowcnt[r];
            for (int r = tid >> 2; r < n_rows; r += QUADS) {
                const int e = keys[byrank[r]];
                const int p0 = a.mptr[e], b0 = erow[r], b1 = erow[r + 1];
                int base = rowcnt[r];
                for (int i0 = b0; i0 < b1; i0 += 4) {     // (uniform inside the quad)
                    const int i = i0 + ql;
                    uint32_t rr = kNoRow;
                    if (i < b1) {
                        const uint32_t s2 = ebuf[i];
                        if (s2 != kNoRow) rr = idx[s2];
                    }
                    const bool valid = rr != kNoRow;
                    const unsigned bits = (__ballot_sync(qmask, valid) >> (lane & ~3)) & 0xFu;
                    if (valid) {
                        const int2 en = a.ment[p0 + (i - b0)];
                        edst[base + __popc(bits & ((1u << ql) - 1u))] = make_int2((int)(rr | (en.x == e ? 0x80000000u : 0u)), en.y);
                    }
                    base += __popc(bits);
                }
            }
        }
        __syncthreads();
        return off;
    };

    for (int l = 1; l <= L; ++l) {
        uint16_t* idx_prev = idx0 + ((l + 2) % 3) * HS;   // layer l - 1
        uint16_t* idx_next = idx0 + ((l + 1) % 3) * HS;   // layer l + 1
        n_l[l] = n_cur;
        // ---- the one scan of the live rows of layer l: slot of every merged-row entry -> ebuf ----
        for (int r = tid; r < n_cur; r += THREADS) {
            const int e = keys[rcur[r]];
            rowcnt[r] = a.mptr[e + 1] - a.mptr[e];
        }
        __syncthreads();
        const int n_ent = fused_block_scan_excl<THREADS>(rowcnt, n_cur, s_warp);
        if (n_ent > EC) {                                  // (uniform) this tier's entry buffer is too small
            if (tid == 0) s_ovf = 1;
            __syncthreads();
            break;
        }
        for (int r = tid; r <= n_cur; r += THREADS) erow[r] = rowcnt[r];
        __syncthreads();
        for (int r = tid >> 2; r < n_cur; r += QUADS) {
            const int e = keys[rcur[r]];
            const int p0 = a.mptr[e], b0 = erow[r], len = erow[r + 1] - b0;
            for (int i = ql; i < len; i += 4) {
                const int s2 = set.find(a.ment[p0 + i].x);
                ebuf[b0 + i] = s2 >= 0 ? (uint16_t)s2 : (uint16_t)kNoRow;
            }
        }
        __syncthreads();
        if (l == 1) {
            // the three exact scalars of each live row: x, (S0 x), (S1 x)
            off_l1 = alloc(3 * n_cur);
            if (!s_ovf) {
                float* dst = reinterpret_cast<float*>(a.arena + off_l1);
                for (int r = tid >> 2; r < n_cur; r += QUADS) {
                    const int slot = rcur[r];
                    const int e = keys[slot];
                    const int p0 = a.mptr[e], b0 = erow[r], len = erow[r + 1] - b0;
                    float a1 = 0.f, a2 = 0.f;
                    for (int i = ql; i < len; i += 4) {
                        const uint32_t s2 = ebuf[b0 + i];
                        const float x = s2 != kNoRow ? xv[s2] : 0.f;
                        if (x != 0.f) {
                            const int pk = a.ment[p0 + i].y;
                            a1 = fmaf((float)(short)(pk & 0xffff), x, a1);
                            a2 = fmaf((float)(pk >> 16), x, a2);
                        }
                    }
#pragma unroll
                    for (int o = 1; o < 4; o <<= 1) {
                        a1 += __shfl_xor_sync(qmask, a1, o);
                        a2 += __shfl_xor_sync(qmask, a2, o);
                    }
                    if (ql == 0) {
                        dst[3 * r + 0] = xv[slot];
                        dst[3 * r + 1] = a1;
                        dst[3 * r + 2] = a2;
                    }
                }
            }
            __syncthreads();
        } else {
            off_f[l] = emit_program(rcur, n_cur, idx_prev, tot_f[l]);       // forward: rows of layer l, entries = live rows of layer l - 1
        }
        if (l == L) break;
        // ---- live rows of layer l + 1: cone edges of level >= l + 1 among the scanned entries ----
        if (tid == 0) s_nlive = 0;
        for (int i = tid; i < HS; i += THREADS) idx_next[i] = (uint16_t)kNoRow;
        __syncthreads();
        for (int i = tid; i < n_ent; i += THREADS) {
            const uint32_t s2 = ebuf[i];
            if (s2 != kNoRow && (lvl[s2] & 0xFF) >= l + 1) mark((int)s2, l + 1);
        }
        const int n_next = rank_live(idx_next, rnext);
        if (s_ovf) break;
        off_b[l + 1] = emit_program(rcur, n_cur, idx_next, tot_b[l + 1]);       // transposed program of layer l + 1: rows of layer l
        uint16_t* tmp = rcur; rcur = rnext; rnext = tmp;
        n_cur = n_next;
    }
    __syncthreads();
    if (s_ovf == 1) {                                      // (uniform: s_ovf is only read after barriers)
        give_up();
        return;
    }
    // ---- readout pairs: {row of H_L | neighbour slot << 16, sign bits}; a pair whose edge has no live row keeps kNoRow ----
    const uint16_t* idxL = idx0 + (L % 3) * HS;
    const unsigned off_ro = alloc(align2(D + 1) + 2 * total_pairs);
    if (!s_ovf) {
        int* pdst = reinterpret_cast<int*>(a.arena + off_ro);
        int2* edst = reinterpret_cast<int2*>(a.arena + off_ro + align2(D + 1));
        for (int j = tid; j <= D; j += THREADS) pdst[j] = pairs.s_off[j];
        for (int i = tid; i < total_pairs; i += THREADS) {
            const int j = pairs.slot_of(i, D);
            const int2 es = a.inc_ent[pairs.s_ptr[j] + (i - pairs.s_off[j])];
            const int s = set.find(es.x);
            const uint32_t r = s >= 0 ? (uint32_t)idxL[s] : kNoRow;
            edst[i] = make_int2((int)(r | ((uint32_t)j << 16)), es.y);
        }
    }
    __syncthreads();
    if (FG && !s_ovf) {                                    // layer-0 transposed program: the merged row of each flow edge of T_0
        const uint16_t* idx1 = idx0 + 1 * HS;
        const unsigned off_fg = fused_flow_program<THREADS>(a, fp1 - fp0, s_warp, [&](int i, auto&& emit) {
            const int eo = a.flow_edge[fp0 + i];
            if (eo < 0 || eo >= a.E) return;
            const int e = a.rank[eo];
            if (set.find(e) < 0) return;
            const int q1 = a.mptr[e + 1];
            for (int q = a.mptr[e]; q < q1; ++q) {
                const int2 en = a.ment[q];
                const int s2 = set.find(en.x);
                if (s2 >= 0 && idx1[s2] != (uint16_t)kNoRow) emit(make_int2((int)(idx1[s2] | (en.x == e ? 0x80000000u : 0u)), en.y));
            }
        });
        if (tid == 0) {
            if (off_fg == ~0u) s_ovf = 2;
            else a.fg_off[t] = off_fg;
        }
        __syncthreads();
    }
    if (s_ovf) {                                           // the arena is exhausted (the average program exceeds its share)
        if (tid == 0) {
            hdr[0] = kFusedFlagOverflow;
            *a.overflow = 1;
        }
        return;
    }
    if (tid == 0) {
        hdr[0] = 0;
        for (int l = 1; l <= kFusedMaxL; ++l) hdr[l] = l <= L ? n_l[l] : 0;
        hdr[4] = (int)off_l1;
        for (int l = 2; l <= kFusedMaxL; ++l) {
            hdr[5 + (l - 2)] = (int)off_f[l];
            hdr[7 + (l - 2)] = (int)off_b[l];
        }
        hdr[9] = (int)off_ro;
        hdr[10] = total_pairs;
        hdr[11] = s_nhash;
        hdr[12] = tot_f[2];
        hdr[13] = fp1 - fp0;
        hdr[14] = tot_f[3];
        hdr[15] = min(tot_b[2], 0xFFFF) | (min(tot_b[3], 0xFFFF) << 16);
    }
}

template <int THREADS, bool FG = false>
__global__ void __launch_bounds__(THREADS) fused_plan_kernel(const PlanArgs a) {
    extern __shared__ __align__(16) unsigned char sm[];
    const int n_work = a.tier == 0 ? a.n_work : *a.n_in;
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
        plan_trajectory<THREADS, FG>(a, a.tier == 0 ? w : a.in_list[w], sm);
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// the compute kernel
// ---------------------------------------------------------------------------------------------------------------------
struct TrajArgs {
    const int* hdr;
    const uint32_t* arena;
    const int32_t* rows;                   // planned set: trajectory t of the batch is entry rows[t] of the set (NULL: t itself)
    const uint32_t* okeys;                 // live rows of the batch's trajectories in descending order (0: flagged by the plan kernel)
    const int32_t* order;                  //   and the trajectory each key belongs to (ties: ascending trajectory)
    const float* W;                        // flat weights
    int w_off[3 * kFusedMaxL + 1];
    int L, b, D, n_params;
    float* logprobs;                       // [b][D] or NULL
    const int32_t* target_idx;
    const float* mask;
    float* partial;                        // [gridDim.x][n_params + 2]
    float* scratch;                        // BIG: per-CTA row store
    size_t scratch_stride;                 // floats per CTA
    int cap_rows;                          // rows of the shared-memory row store (small variant)
    int big_rows;                          // rows of the per-CTA global row store
    unsigned long long* rows_done;         // optional device counters: [0] forward rows, [1] backward rows produced
    const float* cot;                      // [b][D] cotangent seed of the COT variant (target_idx / mask unused), else NULL
    const unsigned* fg_off;                // FG variant: layer-0 transposed program of trajectory t (flow-gradient plan)
    const int32_t* traj_ptr;               //   flow entries of trajectory t: [traj_ptr[t], traj_ptr[t + 1])
    float* dflow;                          //   dL/dx at the flow entries, indexed like flow_val
};

template <int C>
struct FuGeom {
    static constexpr int LDH = C + 8;       // row store stride: (tig * LDH + g) hits 32 distinct banks
    static constexpr int LDA = 3 * C + 4;   // gathered tile stride: (g * LDA + tig) hits 32 distinct banks
    static constexpr int LDW = C + 8;
    static constexpr int CH = 80;           // rows gathered per chunk (5 m-tiles)
    static constexpr int SE = 1024;         // program entries staged in shared memory per chunk
    static constexpr int SP = 200;          // staged row pointers (a whole program of the small variant: <= 192 rows; D + 1 for the readout pairs)
    static constexpr int SL1 = 384;         // staged layer-1 scalars (3 per row: 128 rows)
    static constexpr int LPR = C / 4;       // lanes per row in the gather (one float4 each)
    static constexpr int NP = C / 16;       // pairs of n-tiles per row tile
    static constexpr int NMT = C / 16;      // dW: m-tiles (input channels)
    static constexpr int NNT = 3 * C / 8;   // dW: n-tiles (term, output channel)
    static constexpr int WPM = 8 / NMT;     // dW: warps per m-tile
    static constexpr int TPW = (NNT + WPM - 1) / WPM;   // dW tiles per warp
};

// gather of nr rows (program rows r0 .. r0 + nr) from the row store `src` into the tile: [own | S0 sum | S1 sum]; rows up to
// the next multiple of 16 are zero-filled.  ptr[r] = row pointer of program row r0 + r; entry p lives at ent[p - pbase] (STAGED:
// both in shared memory — a dependent global load per entry is what this kernel cannot afford)
template <int C>
__device__ __forceinline__ void fu_gather(float* __restrict__ tile, const float* src, const int* ptr, const int2* ent, int pbase, int nr) {
    using G = FuGeom<C>;
    const int lr = threadIdx.x % G::LPR, rr = threadIdx.x / G::LPR;
    const int npad = (nr + 15) & ~15;
    for (int r = rr; r < npad; r += kTrajThreads / G::LPR) {
        u64 s0a = 0ull, s0b = 0ull, s1a = 0ull, s1b = 0ull;       // packed pairs: (x, y) and (z, w) of the row's float4 chunk
        int own = -1;
        if (r < nr) {
            const int p1 = ptr[r + 1] - pbase;
            for (int p = ptr[r] - pbase; p < p1; ++p) {
                const int2 en = ent[p];
                const float c0 = (float)(short)(en.y & 0xffff), c1 = (float)(en.y >> 16);
                const float* vp = src + (size_t)(en.x & 0xFFFF) * G::LDH + 4 * lr;
                const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(vp);
                const u64 q0 = bcast2(c0), q1 = bcast2(c1);
                ffma2(s0a, q0, v.x);
                ffma2(s0b, q0, v.y);
                ffma2(s1a, q1, v.x);
                ffma2(s1b, q1, v.y);
                own = en.x < 0 ? (en.x & 0xFFFF) : own;
            }
        }
        float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
        if (own >= 0) o = *reinterpret_cast<const float4*>(src + (size_t)own * G::LDH + 4 * lr);
        float* d = tile + (size_t)r * G::LDA + 4 * lr;
        *reinterpret_cast<float4*>(d) = o;
        *reinterpret_cast<ulonglong2*>(d + C) = make_ulonglong2(s0a, s0b);
        *reinterpret_cast<ulonglong2*>(d + 2 * C) = make_ulonglong2(s1a, s1b);
    }
}

__device__ __forceinline__ void cp_async_4(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_8(void* dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Asynchronous copy of a WHOLE program (row pointers + entries; also the readout pair list: D rows) into the staging buffers, issued
// while the previous phase still computes (the staged loads were the top stall of this kernel).  false (nothing issued): the program
// does not fit — the caller stages it chunk by chunk (fu_stage).  Completion: cp_async_wait_all() + barrier.
template <int C>
__device__ __forceinline__ bool fu_prefetch(const uint32_t* __restrict__ arena, unsigned off, int n_rows, int tot, int* sptr, int2* sent) {
    using G = FuGeom<C>;
    if (n_rows + 1 > G::SP || tot > G::SE) return false;   // (block-uniform)
    const int* gptr = reinterpret_cast<const int*>(arena + off);
    const int2* gent = reinterpret_cast<const int2*>(gptr + align2(n_rows + 1));
    for (int i = threadIdx.x; i <= n_rows; i += kTrajThreads) cp_async_4(sptr + i, gptr + i);
    for (int i = threadIdx.x; i < tot; i += kTrajThreads) cp_async_8(sent + i, gent + i);
    return true;
}

// Stages the next chunk of a program (rows r0 ...) into shared memory: row pointers into sptr, entries into sent.  Returns the rows
// of the chunk (<= CH, shrunk in steps of 16 until the entries fit; a chunk that still does not fit is gathered from global memory:
// *staged = false).  Two barriers inside; every thread gets the same answer.
template <int C>
__device__ __forceinline__ int fu_stage(const int* __restrict__ gptr, const int2* __restrict__ gent, int r0, int n_rows, int* sptr,
                                        int2* sent, bool* staged) {
    using G = FuGeom<C>;
    int nr = min(G::CH, n_rows - r0);
    for (int i = threadIdx.x; i <= nr; i += kTrajThreads) sptr[i] = __ldg(gptr + r0 + i);
    __syncthreads();
    const int pbase = sptr[0];
    while (nr > 16 && sptr[nr] - pbase > G::SE) nr -= 16;
    const int cnt = sptr[nr] - pbase;
    *staged = cnt <= G::SE;
    if (*staged)
        for (int i = threadIdx.x; i < cnt; i += kTrajThreads) sent[i] = __ldg(gent + pbase + i);
    __syncthreads();
    return nr;
}

// (3xTF32 splits: slab_common.cuh's round-to-nearest split_tf32.  A two-instruction split — hi = the value as is, truncated by the tensor
// core, lo = a - trunc(a) — was measured: 3 % faster, but its one-sided truncations add up along K: 1.1e-5 on log-probs of magnitude
// 12 and 1.1e-4 relative on the smallest weight gradients, both past the tolerances.  Not used.)
// row tile product: D[nr x C] = tile[nr x 3C] * B, B = [W0; W1; W2] (forward) or [W0^T; W1^T; W2^T] (TRANSPOSED: the backward
// data product); 3xTF32, fp32 accumulate.  A warp owns (m-tile, pair of n-tiles); epi(row, col, v0, v1) receives two adjacent columns.
template <int C, bool TRANSPOSED, typename Epi>
__device__ __forceinline__ void fu_product(const float* __restrict__ tile, const float* __restrict__ Wsm, int nr, Epi epi) {
    using G = FuGeom<C>;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, tig = lane & 3;
    const int n_mt = (nr + 15) >> 4;
    for (int tl = warp; tl < n_mt * G::NP; tl += kTrajThreads / 32) {
        const int mt = tl / G::NP, np = tl % G::NP;
        float d[2][4], dx[2][4];                          // dx: the two small cross terms (a_lo w_hi + a_hi w_lo): an independent mma chain
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int q = 0; q < 4; ++q) d[j][q] = dx[j][q] = 0.f;
        const float* arow0 = tile + (size_t)(16 * mt + g) * G::LDA + tig;
        const float* arow1 = arow0 + 8 * G::LDA;
#pragma unroll 4
        for (int ks = 0; ks < 3 * C / 8; ++ks) {
            const int k0 = 8 * ks;
            uint32_t ahi[4], alo[4];
            split_tf32(arow0[k0], ahi[0], alo[0]);
            split_tf32(arow1[k0], ahi[1], alo[1]);
            split_tf32(arow0[k0 + 4], ahi[2], alo[2]);
            split_tf32(arow1[k0 + 4], ahi[3], alo[3]);
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int n0 = (2 * np + j) * 8;
                float b0, b1;
                if (!TRANSPOSED) {
                    b0 = Wsm[(k0 + tig) * G::LDW + n0 + g];
                    b1 = Wsm[(k0 + tig + 4) * G::LDW + n0 + g];
                } else {                                   // k = term * C + co, n = ci: W_term[ci][co]
                    const int term = k0 / C, co = k0 % C + tig;
                    b0 = Wsm[(term * C + n0 + g) * G::LDW + co];
                    b1 = Wsm[(term * C + n0 + g) * G::LDW + co + 4];
                }
                uint32_t bh0, bl0, bh1, bl1;
                split_tf32(b0, bh0, bl0);
                split_tf32(b1, bh1, bl1);
                mma_tf32(dx[j], alo, bh0, bh1);
                mma_tf32(dx[j], ahi, bl0, bl1);
                mma_tf32(d[j], ahi, bh0, bh1);
            }
        }
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int q = 0; q < 4; ++q) d[j][q] += dx[j][q];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int col = (2 * np + j) * 8 + 2 * tig;
            const int r0 = 16 * mt + g, r1 = r0 + 8;
            if (r0 < nr) epi(r0, col, d[j][0], d[j][1]);
            if (r1 < nr) epi(r1, col, d[j][2], d[j][3]);
        }
    }
}

// weight-gradient tiles: acc += Hprev[rows]^T * tile[rows][3C] (K = the nr rows of the chunk); a warp owns one m-tile of input
// channels and TPW n-tiles of (term, output channel); both operands split for 3xTF32
template <int C>
__device__ __forceinline__ void fu_dw(float (&acc)[FuGeom<C>::TPW][4], const float* hprev, const float* __restrict__ tile, int nr) {
    using G = FuGeom<C>;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, tig = lane & 3;
    const int mt = warp % G::NMT, ntg = warp / G::NMT;
    for (int k0 = 0; k0 < nr; k0 += 8) {
        const int ra = k0 + tig, rb = ra + 4;
        const float* ha = hprev + (size_t)ra * G::LDH + 16 * mt + g;
        const float* hb = hprev + (size_t)rb * G::LDH + 16 * mt + g;
        uint32_t ahi[4], alo[4];
        split_tf32(ra < nr ? ha[0] : 0.f, ahi[0], alo[0]);
        split_tf32(ra < nr ? ha[8] : 0.f, ahi[1], alo[1]);
        split_tf32(rb < nr ? hb[0] : 0.f, ahi[2], alo[2]);
        split_tf32(rb < nr ? hb[8] : 0.f, ahi[3], alo[3]);
#pragma unroll
        for (int s = 0; s < G::TPW; ++s) {
            const int nt = ntg + G::WPM * s;
            if (nt < G::NNT) {                             // (warp-uniform)
                uint32_t bh0, bl0, bh1, bl1;
                split_tf32(tile[(size_t)ra * G::LDA + 8 * nt + g], bh0, bl0);     // rows >= nr of the tile are zero
                split_tf32(tile[(size_t)rb * G::LDA + 8 * nt + g], bh1, bl1);
                mma_tf32(acc[s], alo, bh0, bh1);
                mma_tf32(acc[s], ahi, bl0, bl1);
                mma_tf32(acc[s], ahi, bh0, bh1);
            }
        }
    }
}

// COT (with GRAD; scone_model_vjp_*): the readout's dlogit seed is dl_j = cot_j - p_j * sum_k cot_k over ALL D slots (padded slots
// included: quirk Q1), the NLL slot takes sum_j cot_j * logp_j and the count slot 0.  Everything after the seed is shared.
// FG (with COT; scone_model_vjp_flows_*, flow-gradient plans): after the first layer's weight gradient, one transposed operator hop
// without activation gives dL/dx = G_1 w0^T + S0 (G_1 w1^T) + S1 (G_1 w2^T) at the flow entries (the layer-0 program).
template <int C, int ACT, bool GRAD, bool BIG, bool COT = false, bool FG = false>
__global__ void __launch_bounds__(kTrajThreads, 2) fused_traj_kernel(const TrajArgs a) {
    using G = FuGeom<C>;
    extern __shared__ __align__(16) unsigned char sm[];
    const int L = a.L, D = a.D;
    float* Wsm = reinterpret_cast<float*>(sm);                        // [(L-1)][3C][LDW]
    float* w1s = Wsm + (size_t)(kFusedMaxL - 1) * 3 * C * G::LDW;    // [3][C] first-layer weights
    float* wos = w1s + 3 * C;                                        // [C] w_out
    float* tile = wos + C;                                           // [CH][LDA]
    float* zs = tile + (size_t)G::CH * G::LDA;                       // [D][C] readout sums
    float* lg = zs + (size_t)D * C;                                  // [D] logits -> log-probs
    float* dl = lg + ((D + 3) & ~3);                                 // [D] dlogits
    int2* sent = reinterpret_cast<int2*>(dl + ((D + 3) & ~3));       // [SE] staged program entries of the current chunk
    int* sptr = reinterpret_cast<int*>(sent + G::SE);                // [SP] staged row pointers
    float* l1s = reinterpret_cast<float*>(sptr + G::SP);             // [2][SL1] staged layer-1 scalars of this / the next trajectory
    float* rows_sm = l1s + 2 * G::SL1;                                   // [cap_rows][LDH]  (small variant)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int l = 2; l <= L; ++l)
        for (int i = tid; i < 3 * C * C; i += kTrajThreads) {
            const int term = i / (C * C), rem = i % (C * C);
            Wsm[(size_t)(l - 2) * 3 * C * G::LDW + (term * C + rem / C) * G::LDW + rem % C] = a.W[a.w_off[3 * (l - 1) + term] + rem];
        }
    for (int i = tid; i < 3 * C; i += kTrajThreads) w1s[i] = a.W[a.w_off[i / C] + i % C];
    for (int i = tid; i < C; i += kTrajThreads) wos[i] = a.W[a.w_off[3 * L] + i];
    __syncthreads();

    float acc[kFusedMaxL - 1][G::TPW][4];
#pragma unroll
    for (int l = 0; l < kFusedMaxL - 1; ++l)
#pragma unroll
        for (int s = 0; s < G::TPW; ++s)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[l][s][q] = 0.f;
    float acc1 = 0.f, acc_out = 0.f, acc_nll = 0.f, acc_cnt = 0.f;
    unsigned long long n_fwd = 0, n_bwd = 0;

    float* rows = BIG ? a.scratch + (size_t)blockIdx.x * a.scratch_stride : rows_sm;

    // The launch's trajectories: the range of the cost-sorted batch whose live rows fit this launch's row store and no smaller one
    // (keys descending: BIG = the head, small = the tail).  They are dealt to the CTAs in snake order — heaviest first, every CTA gets
    // one of each round — so that the CTAs finish together; the order depends on the data only: deterministic.
    // Trajectories are software-pipelined: while trajectory k computes, the header of trajectory k + 1 (order -> set row -> header: three
    // dependent loads) is fetched in steps, and once the staging buffers are free its layer-1 scalars and first program follow.
    __shared__ int s_range[2];
    __shared__ int s_hdr[2][kFusedHdrW];
    if (tid == 0) {
        // keys descending; plan-flagged trajectories carry the largest key: they head the list and belong to no launch
        int f = 0, hi = a.b;
        while (f < hi) {                                   // first position with key < kFlaggedKey
            const int mid = (f + hi) >> 1;
            if (a.okeys[mid] >= kFlaggedKey) f = mid + 1;
            else hi = mid;
        }
        int lo = f;
        hi = a.b;
        while (lo < hi) {                                  // first position with key <= cap_rows
            const int mid = (lo + hi) >> 1;
            if ((int)a.okeys[mid] > a.cap_rows) lo = mid + 1;
            else hi = mid;
        }
        s_range[0] = BIG ? f : lo;
        s_range[1] = BIG ? lo : a.b;
    }
    __syncthreads();
    const int i_lo = s_range[0], i_hi = s_range[1];
    auto index_of = [&](int kk) { return i_lo + kk * (int)gridDim.x + ((kk & 1) ? (int)gridDim.x - 1 - (int)blockIdx.x : (int)blockIdx.x); };
    // asynchronous staging of the layer-1 scalars (read twice) and the first program of the trajectory whose header is hn
    auto issue_first = [&](const int* hn, float* l1buf) -> bool {
        const int n1 = hn[1];
        if (3 * n1 <= G::SL1) {                            // (block-uniform)
            const float* l1g = reinterpret_cast<const float*>(a.arena + (unsigned)hn[4]);
            for (int i = tid; i < 3 * n1; i += kTrajThreads) cp_async_4(l1buf + i, l1g + i);
        }
        return L >= 2 ? fu_prefetch<C>(a.arena, (unsigned)hn[5], hn[2], hn[12], sptr, sent)
                      : fu_prefetch<C>(a.arena, (unsigned)hn[9], D, hn[10], sptr, sent);
    };
    bool have = index_of(0) < i_hi, pf_first = false;
    int t = 0;
    if (have) {                                            // prologue: the first trajectory's header, synchronously
        t = a.order[index_of(0)];
        const int rid = a.rows != nullptr ? a.rows[t] : t;
        if (tid < kFusedHdrW) s_hdr[0][tid] = a.hdr[(size_t)rid * kFusedHdrW + tid];
        __syncthreads();
        pf_first = issue_first(s_hdr[0], l1s);
    }
    for (int k = 0; have; ++k) {
        const int* h = s_hdr[k & 1];
        float* l1buf = l1s + (k & 1) * G::SL1;
        const bool have_next = index_of(k + 1) < i_hi;
        const int t_next = have_next ? a.order[index_of(k + 1)] : 0;      // (consumed after layer 1: the load flies meanwhile)
        bool issued_next = false, pf_first_next = false;
        cp_async_wait_all();
        __syncthreads();
        int n[kFusedMaxL + 1], hb[kFusedMaxL + 2];
        int tot = 0;
        n[0] = 0;
        hb[0] = hb[1] = 0;
#pragma unroll
        for (int l = 1; l <= kFusedMaxL; ++l) {
            n[l] = l <= L ? h[l] : 0;
            hb[l] = tot;
            tot += n[l];
        }
        const float* l1 = reinterpret_cast<const float*>(a.arena + (unsigned)h[4]);
        n_fwd += (unsigned long long)tot;
        // entries of the programs (header): forward of layers 2 / 3, transposed of layers 2 / 3 (saturated at 0xFFFF: never fits then)
        const int tot_f[kFusedMaxL + 1] = {0, 0, h[12], h[14]};
        const int tot_b[kFusedMaxL + 1] = {0, 0, h[15] & 0xFFFF, (int)((unsigned)h[15] >> 16)};
        bool pf = pf_first;
        if (3 * n[1] <= G::SL1) l1 = l1buf;                // (block-uniform) staged by issue_first

        // ---- layer 1 ----
        for (int i = tid; i < n[1] * C; i += kTrajThreads) {
            const int r = i / C, c = i % C;
            const float z = fmaf(l1[3 * r + 2], w1s[2 * C + c], fmaf(l1[3 * r + 1], w1s[C + c], l1[3 * r] * w1s[c]));
            rows[(size_t)r * G::LDH + c] = fu_act<ACT>(z);
        }
        const int rid_next = have_next ? (a.rows != nullptr ? a.rows[t_next] : t_next) : 0;   // (consumed after the conv layers)
        __syncthreads();
        // ---- conv layers ----
#pragma unroll
        for (int l = 2; l <= kFusedMaxL; ++l) {
            if (l > L) break;
            const int nl = n[l];
            const int* ptr = reinterpret_cast<const int*>(a.arena + (unsigned)h[5 + (l - 2)]);
            const int2* ent = reinterpret_cast<const int2*>(ptr + align2(nl + 1));
            const float* hprev = rows + (size_t)hb[l - 1] * G::LDH;
            float* hout = rows + (size_t)hb[l] * G::LDH;
            const float* Wl = Wsm + (size_t)(l - 2) * 3 * C * G::LDW;
            bool pf_next = false;
            if (nl == 0)                                   // (no chunk below issues the next program's copy)
                pf_next = l < L ? fu_prefetch<C>(a.arena, (unsigned)h[5 + (l - 1)], n[l + 1], tot_f[l < kFusedMaxL ? l + 1 : l], sptr, sent)
                                : fu_prefetch<C>(a.arena, (unsigned)h[9], D, h[10], sptr, sent);
            for (int r0 = 0; r0 < nl;) {
                int nr;
                if (pf) {                                  // the whole program is in the staging buffers
                    nr = min(G::CH, nl - r0);
                    fu_gather<C>(tile, hprev, sptr + r0, sent, 0, nr);
                } else {
                    bool staged;
                    nr = fu_stage<C>(ptr, ent, r0, nl, sptr, sent, &staged);
                    if (staged) fu_gather<C>(tile, hprev, sptr, sent, sptr[0], nr);
                    else fu_gather<C>(tile, hprev, sptr, ent, 0, nr);
                }
                __syncthreads();
                if (r0 + nr >= nl)                         // the staging buffers are free: the next program flies under the product
                    pf_next = l < L ? fu_prefetch<C>(a.arena, (unsigned)h[5 + (l - 1)], n[l + 1], tot_f[l < kFusedMaxL ? l + 1 : l], sptr, sent)
                                    : fu_prefetch<C>(a.arena, (unsigned)h[9], D, h[10], sptr, sent);
                fu_product<C, false>(tile, Wl, nr, [&](int r, int col, float v0, float v1) {
                    float* o = hout + (size_t)(r0 + r) * G::LDH + col;
                    *reinterpret_cast<float2*>(o) = make_float2(fu_act<ACT>(v0), fu_act<ACT>(v1));
                });
                cp_async_wait_all();
                __syncthreads();
                r0 += nr;
            }
            if (nl == 0) {
                cp_async_wait_all();
                __syncthreads();
            }
            pf = pf_next;
        }
        if (have_next && tid < kFusedHdrW) cp_async_4(&s_hdr[(k + 1) & 1][tid], a.hdr + (size_t)rid_next * kFusedHdrW + tid);
        // ---- readout: z_j = sum over the edges incident to neighbour j of sign * H_L[row]; logit_j = z_j . w_out ----
        const int* rptr = reinterpret_cast<const int*>(a.arena + (unsigned)h[9]);
        const int2* rent = reinterpret_cast<const int2*>(rptr + align2(D + 1));
        if (pf) {
            rptr = sptr;
            rent = sent;
        } else if (h[10] <= G::SE) {                       // (block-uniform) stage the pair list: read by the logits and by dq
            for (int i = tid; i <= D; i += kTrajThreads) sptr[i] = __ldg(rptr + i);
            for (int i = tid; i < h[10]; i += kTrajThreads) sent[i] = __ldg(rent + i);
            __syncthreads();
            rptr = sptr;
            rent = sent;
        }
        const float* hL = rows + (size_t)hb[L] * G::LDH;
        for (int j = warp; j < D; j += kTrajThreads / 32) {
            float z = 0.f;
            const int p1 = rptr[j + 1];
            for (int p = rptr[j]; p < p1; ++p) {
                const int2 en = rent[p];
                const uint32_t r = (uint32_t)en.x & 0xFFFFu;
                if (r != kNoRow && lane < C) z = fmaf(__int_as_float(en.y), hL[(size_t)r * G::LDH + lane], z);
            }
            if (lane < C) zs[j * C + lane] = z;
            float part = lane < C ? z * wos[lane] : 0.f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            if (lane == 0) lg[j] = part;
        }
        __syncthreads();
        if (warp == 0) {                                   // padded slots (logit exactly 0) take part in the normaliser: quirk Q1
            float mx = -3.4e38f;
            for (int j = lane; j < D; j += 32) mx = fmaxf(mx, lg[j]);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
            float se = 0.f;
            for (int j = lane; j < D; j += 32) se += expf(lg[j] - mx);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
            const float lse = mx + logf(se);
            const float mk = GRAD && !COT ? a.mask[t] : 0.f;
            const int y = GRAD && !COT ? a.target_idx[t] : -1;
            float cs = 0.f;                                // COT: sum_k cot_k (lane-strided, fixed butterfly); dl holds the row meanwhile
            if (COT) {
                for (int j = lane; j < D; j += 32) {
                    const float c = a.cot[(size_t)t * D + j];
                    dl[j] = c;
                    cs += c;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) cs += __shfl_xor_sync(0xffffffffu, cs, o);
            }
            for (int j = lane; j < D; j += 32) {
                const float lp = lg[j] - lse;
                if (a.logprobs != nullptr) a.logprobs[(size_t)t * D + j] = lp;
                if (COT) {
                    const float c = dl[j];
                    dl[j] = c - expf(lp) * cs;
                    acc_nll = fmaf(c, lp, acc_nll);        // (summed over lanes at the end)
                } else if (GRAD) {
                    dl[j] = mk * (expf(lp) - (j == y ? 1.f : 0.f));
                    if (j == y) acc_nll += -mk * lp;       // (lane y % 32 of warp 0 owns the term; summed over lanes at the end)
                }
            }
            if (GRAD && !COT && lane == 0) acc_cnt += mk;
        }
        if (!GRAD) {
            cp_async_wait_all();
            __syncthreads();                               // the next header has landed, the pair list is done with
            if (have_next) pf_first = issue_first(s_hdr[(k + 1) & 1], l1s + ((k + 1) & 1) * G::SL1);
            t = t_next;
            have = have_next;
            continue;
        }
        // ---- backward of the readout: dq[row] = sum of sign * dl_j over its (at most two) pairs; G_L = dq w_out act'(H_L) ----
        // dq[r] lives in the first padding column of row r of G_L (columns C .. C+7 of a stored row are never read as data)
        const int nL = n[L];
        // G_l takes the place of H_l: once dH_l is known, H_l is only needed for act'(H_l) (same element, same thread) — the weight
        // gradient of layer l + 1, the other reader of H_l, is accumulated BEFORE the rows are overwritten (barrier in the loop below)
        float* gL = rows + (size_t)hb[L] * G::LDH;
        for (int r = tid; r < nL; r += kTrajThreads) gL[(size_t)r * G::LDH + C] = 0.f;
        __syncthreads();
        if (tid < C) {
            float s = acc_out;
            for (int j = 0; j < D; ++j) s = fmaf(dl[j], zs[j * C + tid], s);
            acc_out = s;
        }
        {
            const int npairs = rptr[D];
            for (int p = tid; p < npairs; p += kTrajThreads) {
                const int2 en = rent[p];
                const uint32_t r = (uint32_t)en.x & 0xFFFFu;
                if (r != kNoRow) atomicAdd(&gL[(size_t)r * G::LDH + C], __int_as_float(en.y) * dl[((uint32_t)en.x >> 16) & 0x7FFFu]);   // a + b == b + a
            }
        }
        __syncthreads();
        // the pair list is done with: the transposed program of layer L flies under the elementwise pass
        pf = L >= 2 ? fu_prefetch<C>(a.arena, (unsigned)h[7 + (L - 2)], n[L - 1], tot_b[L], sptr, sent) : false;
        for (int i = tid; i < nL * C; i += kTrajThreads) {
            const int r = i / C, c = i % C;
            gL[(size_t)r * G::LDH + c] = gL[(size_t)r * G::LDH + C] * wos[c] * fu_dact<ACT>(hL[(size_t)r * G::LDH + c]);
        }
        cp_async_wait_all();
        __syncthreads();
        // ---- conv layers backward: AG = [G_l | S0 G_l | S1 G_l] on the live rows of layer l - 1 ----
#pragma unroll
        for (int l = kFusedMaxL; l >= 2; --l) {
            if (l > L) continue;
            const int np_ = n[l - 1];
            const int* ptr = reinterpret_cast<const int*>(a.arena + (unsigned)h[7 + (l - 2)]);
            const int2* ent = reinterpret_cast<const int2*>(ptr + align2(np_ + 1));
            const float* gl = rows + (size_t)hb[l] * G::LDH;
            float* hprev = rows + (size_t)hb[l - 1] * G::LDH;
            float* gprev = hprev;
            const float* Wl = Wsm + (size_t)(l - 2) * 3 * C * G::LDW;
            n_bwd += (unsigned long long)np_;
            bool pf_next = false;
            if (np_ == 0 && l > 2) pf_next = fu_prefetch<C>(a.arena, (unsigned)h[7 + (l - 3)], n[l - 2], tot_b[l - 1], sptr, sent);
            for (int r0 = 0; r0 < np_;) {
                int nr;
                if (pf) {
                    nr = min(G::CH, np_ - r0);
                    fu_gather<C>(tile, gl, sptr + r0, sent, 0, nr);
                } else {
                    bool staged;
                    nr = fu_stage<C>(ptr, ent, r0, np_, sptr, sent, &staged);
                    if (staged) fu_gather<C>(tile, gl, sptr, sent, sptr[0], nr);
                    else fu_gather<C>(tile, gl, sptr, ent, 0, nr);
                }
                __syncthreads();
                if (r0 + nr >= np_) {                      // the staging buffers are free
                    if (l > 2) {
                        pf_next = fu_prefetch<C>(a.arena, (unsigned)h[7 + (l - 3)], n[l - 2], tot_b[l - 1], sptr, sent);
                    } else if (have_next) {                // last gather of this trajectory: the next one's first pieces
                        pf_first_next = issue_first(s_hdr[(k + 1) & 1], l1s + ((k + 1) & 1) * G::SL1);
                        issued_next = true;
                    }
                }
                fu_dw<C>(acc[l - 2], hprev + (size_t)r0 * G::LDH, tile, nr);
                __syncthreads();                           // every warp has read H_{l-1} of this chunk: G_{l-1} may overwrite it
                fu_product<C, true>(tile, Wl, nr, [&](int r, int col, float v0, float v1) {
                    const float2 hv = *reinterpret_cast<const float2*>(hprev + (size_t)(r0 + r) * G::LDH + col);
                    *reinterpret_cast<float2*>(gprev + (size_t)(r0 + r) * G::LDH + col) =
                        make_float2(v0 * fu_dact<ACT>(hv.x), v1 * fu_dact<ACT>(hv.y));
                });
                cp_async_wait_all();
                __syncthreads();
                r0 += nr;
            }
            if (np_ == 0) {
                cp_async_wait_all();
                __syncthreads();
            }
            pf = pf_next;
        }
        // ---- first layer: dW_k[0][c] += sum_rows a_k[row] G_1[row][c] ----
        if (tid < 3 * C) {
            const int k = tid / C, c = tid % C;
            const float* g1 = rows;
            float s = acc1;
            for (int r = 0; r < n[1]; ++r) s = fmaf(l1[3 * r + k], g1[(size_t)r * G::LDH + c], s);
            acc1 = s;
        }
        if constexpr (FG) {                                // (discarded from every other instantiation: their SASS is unchanged)
            // u_k[r] = G_1[r] . w_k in the padding columns C .. C + 2 of the live layer-1 rows (the loop above reads columns < C) ...
            for (int i = tid; i < 3 * n[1]; i += kTrajThreads) {
                const int r = i / 3, k = i - 3 * r;
                const float* g = rows + (size_t)r * G::LDH;
                float s = 0.f;
#pragma unroll 8
                for (int c = 0; c < C; ++c) s = fmaf(g[c], w1s[k * C + c], s);
                rows[(size_t)r * G::LDH + C + k] = s;
            }
            __syncthreads();
            // ... then a thread per flow entry walks its row of the layer-0 program: dL/dx = sum (own ? u0 : 0) + c0 u1 + c1 u2.  The
            // trajectory owns its output range: no atomics.  (The staging buffers may hold the next trajectory's first pieces by now:
            // the program is read from the arena.)
            const int nf = h[13];
            const int* fptr = reinterpret_cast<const int*>(a.arena + a.fg_off[t]);
            const int2* fent = reinterpret_cast<const int2*>(fptr + align2(nf + 1));
            float* out = a.dflow + a.traj_ptr[t];
            for (int i = tid; i < nf; i += kTrajThreads) {
                float s = 0.f;
                const int p1 = fptr[i + 1];
                for (int p = fptr[i]; p < p1; ++p) {
                    const int2 en = fent[p];
                    const float* u = rows + (size_t)(en.x & 0xFFFF) * G::LDH + C;
                    if (en.x < 0) s += u[0];
                    s = fmaf((float)(short)(en.y & 0xffff), u[1], s);
                    s = fmaf((float)(en.y >> 16), u[2], s);
                }
                out[i] = s;
            }
        }
        if (have_next && !issued_next) {                   // (no conv layer / no live row in layer 1: nothing above issued it)
            cp_async_wait_all();
            __syncthreads();
            pf_first_next = issue_first(s_hdr[(k + 1) & 1], l1s + ((k + 1) & 1) * G::SL1);
        }
        pf_first = pf_first_next;
        t = t_next;
        have = have_next;
    }

    if (a.rows_done != nullptr && tid == 0 && (n_fwd | n_bwd)) {
        atomicAdd(a.rows_done, n_fwd);
        atomicAdd(a.rows_done + 1, n_bwd);
    }
    if (!GRAD) return;
    // ---- the CTA's partial gradient vector ----
    float* P = a.partial + (size_t)blockIdx.x * (a.n_params + 2);
    if (tid < 3 * C) P[a.w_off[tid / C] + tid % C] = acc1;
    {
        const int g = lane >> 2, tig = lane & 3;
        const int mt = warp % G::NMT, ntg = warp / G::NMT;
#pragma unroll
        for (int l = 2; l <= kFusedMaxL; ++l) {
            if (l > L) break;
#pragma unroll
            for (int s = 0; s < G::TPW; ++s) {
                const int nt = ntg + G::WPM * s;
                if (nt >= G::NNT) continue;
                const int nn = 8 * nt + 2 * tig, term = nn / C, co = nn % C;
                float* dst = P + a.w_off[3 * (l - 1) + term];
                const int ci = 16 * mt + g;
                dst[ci * C + co] = acc[l - 2][s][0];
                dst[ci * C + co + 1] = acc[l - 2][s][1];
                dst[(ci + 8) * C + co] = acc[l - 2][s][2];
                dst[(ci + 8) * C + co + 1] = acc[l - 2][s][3];
            }
        }
    }
    if (tid < C) P[a.w_off[3 * L] + tid] = acc_out;
    if (warp == 0) {
        float s = acc_nll;                                 // fixed butterfly over the lanes of warp 0
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) {
            P[a.n_params] = s;
            P[a.n_params + 1] = acc_cnt;
        }
    }
}

// sort keys of a batch: live rows of trajectory t (0 when the plan kernel flagged it), value t
__global__ void __launch_bounds__(256) fused_cost_kernel(const int* __restrict__ hdr, const int32_t* __restrict__ rows, int b, int L,
                                                         uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= b) return;
    const int* h = hdr + (size_t)(rows != nullptr ? rows[t] : t) * kFusedHdrW;
    int tot = 0;
    for (int l = 1; l <= L; ++l) tot += h[l];
    keys[t] = h[0] != 0 ? kFlaggedKey : min((uint32_t)tot, kFlaggedKey - 1u);
    vals[t] = t;
}

// out[i] += sum over the CTAs' partial vectors in a fixed order (deterministic): a block owns 32 consecutive elements (lane = element:
// 128-byte reads), its 8 warps take the partials p = warp, warp + 8, ... and are folded in a fixed tree
__global__ void __launch_bounds__(256) fused_reduce_kernel(const float* __restrict__ partial, int nparts, int n, float* __restrict__ out) {
    __shared__ float red[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;
    float s = 0.f;
    if (i < n)
        for (int p = warp; p < nparts; p += 8) s += partial[(size_t)p * n + i];
    red[warp][lane] = s;
    __syncthreads();
    if (warp == 0 && i < n)
        out[i] += ((red[0][lane] + red[1][lane]) + (red[2][lane] + red[3][lane])) + ((red[4][lane] + red[5][lane]) + (red[6][lane] + red[7][lane]));
}

size_t plan_smem_bytes(int HS, int LV, int EC) {
    return (size_t)HS * 18 + (size_t)(LV + 4) * 8 + (size_t)LV * 10 + (size_t)EC * 2 + 16;
}

template <int C>
size_t traj_smem_bytes(int D, int cap_rows) {
    using G = FuGeom<C>;
    size_t fl = (size_t)(kFusedMaxL - 1) * 3 * C * G::LDW + 3 * C + C + (size_t)G::CH * G::LDA + (size_t)D * C + 2 * ((D + 3) & ~3) +
                2 * (size_t)G::SE + G::SP + 2 * G::SL1 + (size_t)cap_rows * G::LDH;
    return fl * sizeof(float);
}

template <int C, int ACT, bool GRAD, bool COT, bool FG>
int launch_traj(const TrajArgs& base, int grid_small, int grid_big, size_t smem_small, size_t smem_big, cudaStream_t st) {
    static bool configured = false;
    if (!configured) {
        SCONE_CUDA(cudaFuncSetAttribute(fused_traj_kernel<C, ACT, GRAD, false, COT, FG>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 1024));
        SCONE_CUDA(cudaFuncSetAttribute(fused_traj_kernel<C, ACT, GRAD, true, COT, FG>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 1024));
        configured = true;
    }
    TrajArgs a = base;
    fused_traj_kernel<C, ACT, GRAD, false, COT, FG><<<grid_small, kTrajThreads, smem_small, st>>>(a);
    SCONE_LAUNCHED();
    if (grid_big > 0) {
        if (GRAD) a.partial = base.partial + (size_t)grid_small * (base.n_params + 2);
        fused_traj_kernel<C, ACT, GRAD, true, COT, FG><<<grid_big, kTrajThreads, smem_big, st>>>(a);
        SCONE_LAUNCHED();
    }
    return 0;
}

template <int C, bool GRAD, bool COT = false, bool FG = false>
int dispatch_traj(int act, const TrajArgs& a, int gs, int gb, size_t ss, size_t sb, cudaStream_t st) {
    switch (act) {
        case SCONE_ACT_TANH: return launch_traj<C, SCONE_ACT_TANH, GRAD, COT, FG>(a, gs, gb, ss, sb, st);
        case SCONE_ACT_LEAKY_RELU: return launch_traj<C, SCONE_ACT_LEAKY_RELU, GRAD, COT, FG>(a, gs, gb, ss, sb, st);
        case SCONE_ACT_RELU: return launch_traj<C, SCONE_ACT_RELU, GRAD, COT, FG>(a, gs, gb, ss, sb, st);
    }
    scone_set_error("unknown activation %d", act);
    return 2;
}

// Compute kernels over the plans t.hdr / t.arena describe (+ the fixed-order reduce of the CTAs' partial vectors into grad).  The
// batch is first sorted by live rows (stable radix sort: the order depends on the data only).
int run_traj(FusedState* f, int act, TrajArgs& t, float* grad, cudaStream_t st) {
    const bool want_grad = grad != nullptr;
    const int n = t.b;
    if (n > f->sort_cap) {
        cudaFree(f->d_sort);
        cudaFree(f->d_sort_tmp);
        f->d_sort = nullptr;
        f->d_sort_tmp = nullptr;
        f->sort_cap = 0;
        uint32_t* k = nullptr;
        int32_t* v = nullptr;
        size_t bytes = 0;
        SCONE_CUDA(cub::DeviceRadixSort::SortPairsDescending(nullptr, bytes, k, k, v, v, n, 0, 24, st));
        SCONE_CUDA(cudaMalloc((void**)&f->d_sort, 4 * (size_t)n * sizeof(uint32_t)));
        SCONE_CUDA(cudaMalloc((void**)&f->d_sort_tmp, bytes ? bytes : 16));
        f->sort_tmp_bytes = bytes;
        f->sort_cap = n;
    }
    uint32_t* k_in = f->d_sort;
    uint32_t* k_out = k_in + f->sort_cap;
    int32_t* v_in = reinterpret_cast<int32_t*>(k_out + f->sort_cap);
    int32_t* v_out = v_in + f->sort_cap;
    ScopedProf prof(want_grad ? SCONE_K_LAYER_BWD : SCONE_K_LAYER_FWD, st);
    fused_cost_kernel<<<(n + 255) / 256, 256, 0, st>>>(t.hdr, t.rows, n, f->L, k_in, v_in);
    SCONE_LAUNCHED();
    size_t bytes = f->sort_tmp_bytes;
    SCONE_CUDA(cub::DeviceRadixSort::SortPairsDescending(f->d_sort_tmp, bytes, k_in, k_out, v_in, v_out, n, 0, 24, st));
    t.okeys = k_out;
    t.order = v_out;
    int rc;
    const int gs = f->grid_small, gb = f->grid_big;
    const size_t ss = f->traj_smem_small, sb = f->traj_smem_big;
    if (want_grad && t.cot && t.dflow)
        rc = f->C == 32 ? dispatch_traj<32, true, true, true>(act, t, gs, gb, ss, sb, st) : dispatch_traj<16, true, true, true>(act, t, gs, gb, ss, sb, st);
    else if (f->C == 32)
        rc = !want_grad ? dispatch_traj<32, false>(act, t, gs, gb, ss, sb, st)
                        : (t.cot ? dispatch_traj<32, true, true>(act, t, gs, gb, ss, sb, st) : dispatch_traj<32, true>(act, t, gs, gb, ss, sb, st));
    else
        rc = !want_grad ? dispatch_traj<16, false>(act, t, gs, gb, ss, sb, st)
                        : (t.cot ? dispatch_traj<16, true, true>(act, t, gs, gb, ss, sb, st) : dispatch_traj<16, true>(act, t, gs, gb, ss, sb, st));
    if (rc) return rc;
    if (want_grad) {
        const int np = (int)f->n_params + 2;
        fused_reduce_kernel<<<(np + 31) / 32, 256, 0, st>>>(f->d_partial, f->grid_small + f->grid_big, np, grad);
        SCONE_LAUNCHED();
    }
    return 0;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------------
bool scone_fused_supported(const scone_complex* cx, int n_layers, const int32_t* hidden) {
    if (cx->d_mptr == nullptr || cx->D > kFuMaxD || cx->D < 1 || n_layers < 1 || n_layers > kFusedMaxL) return false;
    for (int l = 0; l < n_layers; ++l)
        if (hidden[l] != hidden[0] || (hidden[l] != 16 && hidden[l] != 32)) return false;
    return true;
}

void scone_fused_destroy(FusedState* f) {
    if (!f) return;
    cudaFree(f->d_hdr); cudaFree(f->d_retry); cudaFree(f->d_arena); cudaFree(f->d_set_hdr); cudaFree(f->d_set_arena); cudaFree(f->d_set_bump); cudaFree(f->d_bump); cudaFree(f->d_partial); cudaFree(f->d_scratch); cudaFree(f->d_stats);
    cudaFree(f->d_rows_done); cudaFree(f->d_sort); cudaFree(f->d_sort_tmp); cudaFree(f->d_fg_off);
    scone_table_destroy(f);
    delete f;
}

// Measures the static bounds of the complex and sizes every buffer of the fused pipeline for micro-batches of `mb` trajectories.
// Returns 0 and *out = nullptr when the complex does not fit the pipeline's shared-memory tables (caller keeps pipeline 3 / 2).
static void table_shape(int entries, int* HS, int* hshift) {
    int hs = 256;
    while (hs * 3 / 4 < entries + 1) hs *= 2;
    *HS = hs;
    *hshift = 32;
    for (int v = hs; v > 1; v >>= 1) --*hshift;
}

int scone_fused_create(const scone_complex* cx, int L, int C, int mb, int64_t n_params, FusedState** out) {
    *out = nullptr;
    if ((unsigned)cx->E >= (1u << 30)) return 0;           // cone table entries carry the level in their top two bits
    FusedState* f = new FusedState();
    f->L = L;
    f->C = C;
    f->n_params = n_params;
    // ---- the node table: cone entries of every node (and, memory permitting, the operator rows of the cone in local indices: the
    // table plan); weight- and data-independent geometry of the complex.  Its sizes are the static bounds of the pipeline ----
    {
        bool ok = false;
        const int rc = scone_table_build(cx, f, L, &ok);
        if (rc || !ok) {                                   // cones larger than any table: not this pipeline's regime
            scone_fused_destroy(f);
            return rc;
        }
    }
    int max_row = 1;
    {
        std::vector<int32_t> mp((size_t)cx->E + 1);
        SCONE_CUDA(cudaMemcpy(mp.data(), cx->d_mptr, mp.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
        for (int e = 0; e < cx->E; ++e) max_row = std::max(max_row, mp[e + 1] - mp[e]);
    }
    // tier 1 (cannot overflow its tables; 1024 threads per trajectory): hash for the largest T_0, live rows up to the largest T_1.
    // tier 0 (256 threads): tables that hold T_0 of 99 % of the nodes (a few hull / hole boundary nodes of a Delaunay complex have
    // cones ten times the typical size; sizing every CTA for them costs the occupancy the plan kernel lives on)
    constexpr int kMaxPlanSmem = 225 * 1024;
    f->LV = (f->bound_list + 63) & ~63;
    table_shape(f->bound_cone, &f->HS, &f->hshift);
    // slot buffer: every merged-row entry of the live rows of one layer.  The worst case (every cone edge live, every row of maximum
    // length) rarely fits next to the tables; the buffer then takes what is left of the shared-memory budget (tens of thousands of
    // entries against a few thousand for the largest trajectories seen) and a layer beyond it is reported through the overflow flag
    f->EC = (int)std::min<long long>((long long)f->bound_list * max_row, 1ll << 30);
    f->EC = (f->EC + 63) & ~63;
    {
        const size_t fixed = plan_smem_bytes(f->HS, f->LV, 0);
        if (fixed + 2 * (size_t)f->EC > (size_t)kMaxPlanSmem && fixed + 2 * 8192 <= (size_t)kMaxPlanSmem)
            f->EC = (int)(((size_t)kMaxPlanSmem - fixed) / 2) & ~63;
    }
    f->plan_smem = plan_smem_bytes(f->HS, f->LV, f->EC);
    if (!f->tb_rows && (f->plan_smem > (size_t)kMaxPlanSmem || f->bound_list >= 0xFFFF || f->HS > 32768)) {   // neither plan kernel fits
        scone_fused_destroy(f);
        return 0;
    }
    {
        // (measured on the 1M-edge bench complex: 1024 slots / 27 KB per CTA beat 2048 / 45 KB although twice as
        // many trajectories go to the second tier — occupancy is what the first tier lives on; 192 live rows / 3072 entries per
        // layer hold all but the trajectories the compute kernel sends to its big variant anyway)
        table_shape(f->quantile_cone, &f->HS0, &f->hshift0);
        f->LV0 = std::min(192, f->LV);
        f->EC0 = std::min(3072, f->EC);
        f->two_tiers = f->HS0 < f->HS || f->LV0 < f->LV || f->EC0 < f->EC;
        if (!f->two_tiers) {
            f->HS0 = f->HS;
            f->hshift0 = f->hshift;
        }
        f->plan_smem0 = plan_smem_bytes(f->HS0, f->LV0, f->EC0);
    }
    SCONE_CUDA(cudaFuncSetAttribute(fused_plan_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPlanSmem));
    SCONE_CUDA(cudaFuncSetAttribute(fused_plan_kernel<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPlanSmem));
    SCONE_CUDA(cudaFuncSetAttribute(fused_plan_kernel<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPlanSmem));
    SCONE_CUDA(cudaFuncSetAttribute(fused_plan_kernel<1024, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxPlanSmem));
    // ---- compute kernel: shared-memory row store of the small variant, per-CTA global row store of the big one ----
    const int ldh = C + 8;
    f->cap_rows = C == 32 ? 192 : 384;
    f->big_rows = L * f->bound_list;
    f->traj_smem_small = C == 32 ? traj_smem_bytes<32>(cx->D, f->cap_rows) : traj_smem_bytes<16>(cx->D, f->cap_rows);
    f->traj_smem_big = C == 32 ? traj_smem_bytes<32>(cx->D, 0) : traj_smem_bytes<16>(cx->D, 0);
    if (f->traj_smem_small > 113 * 1024) {                 // very high degrees: shrink the row store, keep two CTAs per SM
        const size_t over = f->traj_smem_small - 113 * 1024;
        const int less = (int)((over + ldh * 4 - 1) / (ldh * 4));
        f->cap_rows = f->cap_rows > less + 32 ? f->cap_rows - less : 32;
        f->traj_smem_small = C == 32 ? traj_smem_bytes<32>(cx->D, f->cap_rows) : traj_smem_bytes<16>(cx->D, f->cap_rows);
    }
    f->grid_small = 2 * cx->num_sms;
    f->grid_big = f->big_rows > f->cap_rows ? 2 * cx->num_sms : 0;   // (every trajectory fits the shared-memory store otherwise)
    if (f->grid_big) {
        f->scratch_stride = (size_t)f->big_rows * ldh;
        SCONE_CUDA(cudaMalloc((void**)&f->d_scratch, (size_t)f->grid_big * f->scratch_stride * sizeof(float)));
    }
    SCONE_CUDA(cudaMalloc((void**)&f->d_partial, (size_t)(f->grid_small + f->grid_big) * (n_params + 2) * sizeof(float)));
    // ---- program arena.  Worst case per trajectory from the bounds (every row of every layer live, every merged-row entry kept).
    // The arena holds min(worst * chunk, 4 GB): when the worst case fits, it cannot overflow; otherwise it is exhausted only if the
    // AVERAGE program of a chunk exceeds 64 KB (typical: 5 - 10 KB), which the plan kernel reports through the overflow flag. ----
    const unsigned long long bl = (unsigned long long)f->bound_list;
    unsigned long long worst = 3 * bl + 2 + (unsigned long long)(cx->D + 3) + 2ull * cx->D * cx->D + 16;   // (a neighbour has at most D incident edges)
    for (int l = 2; l <= L; ++l)                            // layer l: n_l <= |T_1| rows; the two programs hold the same entries
        worst += 2 * (bl + 3) + 4 * bl * (unsigned long long)max_row;
    const unsigned long long budget_words = (1ull << 30) - 1024;                 // 4 GB of 32-bit words; offsets are 32-bit
    const unsigned long long share_words = 16 * 1024;                            // 64 KB per trajectory
    f->worst_words = worst;
    if (worst * (unsigned long long)mb <= budget_words) {
        f->chunk = mb;
        f->arena_words = worst * (unsigned long long)mb;
    } else {
        f->chunk = (int)std::min<unsigned long long>((unsigned long long)mb, std::max<unsigned long long>(1, budget_words / std::min(worst, share_words)));
        f->arena_words = std::min(budget_words, worst * (unsigned long long)f->chunk);
    }
    SCONE_CUDA(cudaMalloc((void**)&f->d_arena, f->arena_words * sizeof(uint32_t)));
    SCONE_CUDA(cudaMalloc((void**)&f->d_hdr, (size_t)f->chunk * kFusedHdrW * sizeof(int)));
    SCONE_CUDA(cudaMalloc((void**)&f->d_retry, 2 * (size_t)f->chunk * sizeof(int)));
    SCONE_CUDA(cudaMalloc((void**)&f->d_bump, 2 * sizeof(unsigned long long)));  // [0] arena bump pointer, [1] retry counter (int)
    SCONE_CUDA(cudaMalloc((void**)&f->d_rows_done, 4 * sizeof(unsigned long long)));
    SCONE_CUDA(cudaMemset(f->d_rows_done, 0, 4 * sizeof(unsigned long long)));
    *out = f;
    return 0;
}

// Plan kernels over b trajectories (p: trajectories, outputs and the retry list set by the caller): the table plan when the node table
// holds rows, else the hash plan; first tier, then the retry list.
static int launch_plans(const scone_complex* cx, const FusedState* f, PlanArgs p, int b, cudaStream_t st) {
    if (f->tb_rows) return scone_table_plan_launch(f, p, b, cx->num_sms, st);
    p.tier = 0; p.n_work = b;
    p.HS = f->HS0; p.LV = f->LV0; p.EC = f->EC0; p.hshift = f->hshift0;
    int* retry = p.retry;
    if (!f->two_tiers) p.retry = nullptr;
    if (p.fg_off) fused_plan_kernel<256, true><<<b, 256, f->plan_smem0, st>>>(p);
    else fused_plan_kernel<256><<<b, 256, f->plan_smem0, st>>>(p);
    SCONE_LAUNCHED();
    if (f->two_tiers) {                                    // the few trajectories whose cone overflowed the first tier's tables: 1024 threads each
        p.tier = 1; p.HS = f->HS; p.LV = f->LV; p.EC = f->EC; p.hshift = f->hshift; p.n_in = p.n_retry; p.in_list = retry; p.retry = nullptr;
        if (p.fg_off) fused_plan_kernel<1024, true><<<std::min(b, cx->num_sms), 1024, f->plan_smem, st>>>(p);
        else fused_plan_kernel<1024><<<std::min(b, cx->num_sms), 1024, f->plan_smem, st>>>(p);
        SCONE_LAUNCHED();
    }
    return 0;
}

// One chunk (<= f->chunk trajectories) in three steps, so that a caller can plan the parts of a chunk as their inputs arrive
// (scone_model_*_host: the H2D copy of part k + 1 runs under the plan kernels of part k):
//   scone_fused_begin      rearms the chunk's program arena
//   scone_fused_plan_part  plans trajectories off .. off + b of the chunk (traj_ptr / last_nodes: the CHUNK's arrays)
//   scone_fused_compute    compute kernels over the b planned trajectories of the chunk (+ partial reduce into grad)
int scone_fused_begin(FusedState* f, cudaStream_t st) {
    SCONE_CUDA(cudaMemsetAsync(f->d_bump, 0, 2 * sizeof(unsigned long long), st));
    return 0;
}

static PlanArgs plan_args(const scone_complex* cx, FusedState* f, int off, const int32_t* traj_ptr, const int32_t* flow_edge,
                          const float* flow_val, const int32_t* last_nodes, int* overflow) {
    PlanArgs p{};
    p.traj_ptr = traj_ptr + off; p.flow_edge = flow_edge; p.flow_val = flow_val; p.last_nodes = last_nodes + off;
    p.rank = cx->d_rank; p.nbrhoods = cx->d_nbrhoods; p.inc_ptr = cx->d_inc_ptr; p.inc_ent = cx->d_inc_ent;
    p.mptr = cx->d_mptr; p.ment = cx->d_ment; p.cone_ptr = f->d_cone_ptr; p.cone_ent = f->d_cone_ent;
    p.N = cx->N; p.D = cx->D; p.E = cx->E; p.L = f->L;
    p.hdr = f->d_hdr + (size_t)off * kFusedHdrW; p.arena = f->d_arena; p.bump = f->d_bump; p.arena_words = f->arena_words; p.overflow = overflow;
    p.n_retry = reinterpret_cast<int*>(f->d_bump + 1); p.retry = f->d_retry;
    return p;
}

// defer_tiers (table plan only): run the first tier over this part and leave its give-ups on the chunk's work list; the later tiers
// run once over all parts (scone_fused_plan_finish) instead of once per part — each of their launches lasts as long as its slowest
// trajectory, whatever the number of trajectories.
// flow_grad: a flow-gradient plan (PlanArgs::fg_off) for scone_fused_compute with dflow.
int scone_fused_plan_part(const scone_complex* cx, FusedState* f, int off, int b, const int32_t* traj_ptr, const int32_t* flow_edge,
                          const float* flow_val, const int32_t* last_nodes, int* overflow, cudaStream_t st, bool defer_tiers, bool flow_grad) {
    if (b <= 0) return 0;
    SCONE_REQUIRE(off >= 0 && off + b <= f->chunk, "scone_fused_plan_part: trajectories %d .. %d exceed the planned chunk of %d", off, off + b, f->chunk);
    if (flow_grad && !f->d_fg_off) SCONE_CUDA(cudaMalloc((void**)&f->d_fg_off, (size_t)f->chunk * sizeof(unsigned)));
    ScopedProf prof(SCONE_K_CONE, st);
    if (defer_tiers && f->tb_rows) {
        PlanArgs p = plan_args(cx, f, 0, traj_ptr, flow_edge, flow_val, last_nodes, overflow);      // absolute trajectory numbers
        p.t0 = off;
        p.fg_off = flow_grad ? f->d_fg_off : nullptr;
        return scone_table_plan_launch(f, p, b, cx->num_sms, st, 0);
    }
    if (off > 0) SCONE_CUDA(cudaMemsetAsync(f->d_bump + 1, 0, sizeof(unsigned long long), st));   // retry counter only: the arena keeps growing
    PlanArgs p = plan_args(cx, f, off, traj_ptr, flow_edge, flow_val, last_nodes, overflow);
    p.fg_off = flow_grad ? f->d_fg_off + off : nullptr;
    return launch_plans(cx, f, p, b, st);
}

// The later tiers of the parts planned with defer_tiers (no-op for the hash plan, which runs its tiers per part).
int scone_fused_plan_finish(const scone_complex* cx, FusedState* f, int B, const int32_t* traj_ptr, const int32_t* flow_edge,
                            const float* flow_val, const int32_t* last_nodes, int* overflow, cudaStream_t st) {
    if (B <= 0 || !f->tb_rows) return 0;
    ScopedProf prof(SCONE_K_CONE, st);
    return scone_table_plan_launch(f, plan_args(cx, f, 0, traj_ptr, flow_edge, flow_val, last_nodes, overflow), B, cx->num_sms, st, 1);
}

// Arguments of the compute kernels over b trajectories planned into hdr / arena (rows: see TrajArgs)
static TrajArgs traj_args(const scone_complex* cx, const FusedState* f, const int* hdr, const uint32_t* arena, const int32_t* rows, int b,
                          const float* W, const int64_t* w_off, float* logprobs, const int32_t* target_idx, const float* mask, const float* cot,
                          bool count_rows) {
    TrajArgs t;
    t.hdr = hdr; t.arena = arena; t.rows = rows; t.W = W;
    for (int i = 0; i <= 3 * kFusedMaxL; ++i) t.w_off[i] = i <= 3 * f->L ? (int)w_off[i] : 0;
    t.L = f->L; t.b = b; t.D = cx->D; t.n_params = (int)f->n_params;
    t.logprobs = logprobs; t.target_idx = target_idx; t.mask = mask; t.cot = cot;
    t.partial = f->d_partial; t.scratch = f->d_scratch; t.scratch_stride = f->scratch_stride;
    t.cap_rows = f->cap_rows; t.big_rows = f->big_rows;
    t.rows_done = count_rows ? f->d_rows_done : nullptr;
    t.fg_off = nullptr; t.traj_ptr = nullptr; t.dflow = nullptr;
    return t;
}

int scone_fused_compute(const scone_complex* cx, FusedState* f, int act, int b, const float* W, const int64_t* w_off, float* logprobs,
                        const int32_t* target_idx, const float* mask, float* grad, bool count_rows, cudaStream_t st, const float* cot,
                        float* dflow, const int32_t* traj_ptr) {
    if (b <= 0) return 0;
    SCONE_REQUIRE(dflow == nullptr || (cot && grad && traj_ptr && f->d_fg_off), "scone_fused_compute: dflow needs cot, grad, traj_ptr and a flow-gradient plan");
    TrajArgs t = traj_args(cx, f, f->d_hdr, f->d_arena, nullptr, b, W, w_off, logprobs, target_idx, mask, cot, count_rows);
    if (dflow) {
        t.fg_off = f->d_fg_off; t.traj_ptr = traj_ptr; t.dflow = dflow;
    }
    return run_traj(f, act, t, grad, st);
}

int scone_fused_run(const scone_complex* cx, FusedState* f, int act, int b, const int32_t* traj_ptr, const int32_t* flow_edge,
                    const float* flow_val, const int32_t* last_nodes, const float* W, const int64_t* w_off, float* logprobs,
                    const int32_t* target_idx, const float* mask, float* grad, int* overflow, bool count_rows, cudaStream_t st,
                    const float* cot, float* dflow) {
    if (b <= 0) return 0;
    SCONE_REQUIRE(b <= f->chunk, "scone_fused_run: chunk of %d trajectories exceeds the planned %d", b, f->chunk);
    int rc = scone_fused_begin(f, st);
    if (!rc) rc = scone_fused_plan_part(cx, f, 0, b, traj_ptr, flow_edge, flow_val, last_nodes, overflow, st, false, dflow != nullptr);
    if (!rc) rc = scone_fused_compute(cx, f, act, b, W, w_off, logprobs, target_idx, mask, grad, count_rows, st, cot, dflow, traj_ptr);
    return rc;
}

// ---- planned sets: the plan is weight-independent, so a dataset that is revisited every epoch is planned ONCE --------------------
// Plans B trajectories into the set's own arena (kept until the next scone_fused_plan_set / destroy).
int scone_fused_plan_set(const scone_complex* cx, FusedState* f, int B, const int32_t* traj_ptr, const int32_t* flow_edge,
                         const float* flow_val, const int32_t* last_nodes, int* overflow, cudaStream_t st) {
    if (B > f->set_cap) {
        cudaFree(f->d_set_hdr);
        cudaFree(f->d_set_arena);
        f->d_set_hdr = nullptr;
        f->d_set_arena = nullptr;
        f->set_cap = 0;
        const unsigned long long budget_words = (1ull << 30) - 1024;
        f->set_arena_words = std::min(budget_words, f->worst_words * (unsigned long long)B);
        SCONE_CUDA(cudaMalloc((void**)&f->d_set_hdr, (size_t)B * kFusedHdrW * sizeof(int)));
        SCONE_CUDA(cudaMalloc((void**)&f->d_set_arena, f->set_arena_words * sizeof(uint32_t)));
        if (!f->d_set_bump) SCONE_CUDA(cudaMalloc((void**)&f->d_set_bump, 2 * sizeof(unsigned long long)));
        f->set_cap = B;
    }
    f->set_n = 0;
    SCONE_CUDA(cudaMemsetAsync(f->d_set_bump, 0, 2 * sizeof(unsigned long long), st));
    PlanArgs p = plan_args(cx, f, 0, traj_ptr, flow_edge, flow_val, last_nodes, overflow);
    p.arena = f->d_set_arena; p.bump = f->d_set_bump; p.arena_words = f->set_arena_words;     // the set's own arena; hdr: per chunk
    p.n_retry = reinterpret_cast<int*>(f->d_set_bump + 1);
    ScopedProf prof(SCONE_K_CONE, st);
    for (int off = 0; off < B; off += f->chunk) {
        const int b = std::min(f->chunk, B - off);
        SCONE_CUDA(cudaMemsetAsync(f->d_set_bump + 1, 0, sizeof(unsigned long long), st));       // retry counter only: the arena keeps growing
        p.traj_ptr = traj_ptr + off; p.last_nodes = last_nodes + off; p.hdr = f->d_set_hdr + (size_t)off * kFusedHdrW;
        const int rc = launch_plans(cx, f, p, b, st);
        if (rc) return rc;
    }
    f->set_n = B;
    return 0;
}

// Compute kernel over n trajectories of the planned set (rows_dev[t] = index into the set; NULL = the first n of the set).
int scone_fused_run_planned(const scone_complex* cx, FusedState* f, int act, int n, const int32_t* rows_dev, const float* W, const int64_t* w_off,
                            float* logprobs, const int32_t* target_idx, const float* mask, float* grad, bool count_rows, cudaStream_t st,
                            const float* cot) {
    if (n <= 0) return 0;
    SCONE_REQUIRE(f->set_n > 0, "scone_fused_run_planned: no planned set (call scone_model_plan_* first)");
    SCONE_REQUIRE(rows_dev != nullptr || n <= f->set_n, "scone_fused_run_planned: %d trajectories requested, the planned set holds %d", n, f->set_n);
    TrajArgs t = traj_args(cx, f, f->d_set_hdr, f->d_set_arena, rows_dev, n, W, w_off, logprobs, target_idx, mask, cot, count_rows);
    return run_traj(f, act, t, grad, st);
}

// debug / test access: header of trajectory t of the last chunk and `words` arena words from word offset `off`
int scone_fused_last_retries(FusedState* f) {
    unsigned long long v[2] = {0, 0};
    if (cudaDeviceSynchronize() != cudaSuccess) return -1;
    if (cudaMemcpy(v, f->d_bump, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    return (int)(v[1] & 0xffffffffull);
}

int scone_fused_read(FusedState* f, int t, int* hdr_out, unsigned off, int words, uint32_t* arena_out) {
    SCONE_CUDA(cudaDeviceSynchronize());
    if (hdr_out) SCONE_CUDA(cudaMemcpy(hdr_out, f->d_hdr + (size_t)t * kFusedHdrW, kFusedHdrW * sizeof(int), cudaMemcpyDeviceToHost));
    if (arena_out && words > 0) SCONE_CUDA(cudaMemcpy(arena_out, f->d_arena + off, (size_t)words * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return 0;
}
