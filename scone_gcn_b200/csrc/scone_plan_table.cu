// scone_plan_table.cu — the NODE TABLE of the fused pipeline and the plan kernel that reads it.
//
// The receptive cone of the readout (trajectory_experiments.py:151,298-303: the log-probs read H_L only at the edges incident to the
// neighbours of the last node, one operator hop further down per layer) depends on the complex and the last node only.  It is built
// ONCE per complex for every node, together with everything a plan needs from the operators:
//
//   cone entries   T_0 of the node in ascending edge order, each tagged with the highest cone level it belongs to (edge | level << 30).
//                  The position of an edge in this list is its LOCAL INDEX.
//   rows           the merged operator rows of the cone in local indices: for a member of T_1 the complete row (all its columns lie in
//                  T_0), for a level-0 member only its columns in T_1 (what a flow value on it can reach); entries
//                  {local column | own << 31, (c1 << 16) | c0} in ascending column order
//   readout pairs  (neighbour slot, incident edge) pairs of the node with the edge as local index
//
// table_plan_kernel then plans a trajectory with plain arrays indexed by local index — no hash set, no lookups, no operator rows of the
// complex: flows are placed by binary search in the cone entries, live rows are bit sets ranked by popcount (ascending edge id, the
// deterministic row order of every list), programs are the table rows filtered by the live sets.  Its output (headers + program
// arena) is exactly the hash plan's (scone_fused.cu), bit for bit, so the compute kernel and the planned sets do not care which
// plan kernel ran.
#include <algorithm>
#include <cstdlib>
#include <vector>
#include "common.cuh"
#include "fused.cuh"

namespace {

constexpr int kTbThreads = 256;
constexpr int kTbHS = 32768;             // hash slots of one build CTA
constexpr int kTbLC = 16384;             // cone entries one build CTA can hold / sort
constexpr uint32_t kEdgeMask = 0x3FFFFFFFu;
constexpr uint32_t kEmpty = 0xFFFFFFFFu;
constexpr uint32_t kNoRow = 0xFFFFu;
constexpr int kTbMaxD = SCONE_MAX_DEGREE;
constexpr int kTbBuckets = 1024;

__device__ __forceinline__ int align2(int x) { return (x + 1) & ~1; }

struct BuildArgs {
    const int32_t* nbrhoods;
    const int32_t* inc_ptr;
    const int2* inc_ent;
    const int32_t* mptr;
    const int2* ment;
    int N, D, L;
    int* stats;                          // [0] max |T_0|  [1] max |T_1|  [2] error (1 overflow, 2 count mismatch)  [3] max pairs  [4..] histogram of |T_0| / 32
    // pass 1 (keys == NULL): counts per node
    int* cnt_m;
    unsigned* cnt_e;
    int* cnt_p;
    // pass 2
    const unsigned* cone_ptr;
    uint32_t* keys;
    int with_rows;
    const unsigned long long* node_off;
    unsigned* rowptr;
    int2* ent;
    const unsigned* pair_ptr;
    int2* pairs;
    int* pair_off;
};

// position of edge e in the ascending list s[0..m) (entries edge | level << 30), or -1
__device__ __forceinline__ int find_sorted(const uint32_t* s, int m, uint32_t e) {
    int lo = 0, hi = m;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((s[mid] & kEdgeMask) < e) lo = mid + 1;
        else hi = mid;
    }
    return lo < m && (s[lo] & kEdgeMask) == e ? lo : -1;
}

// One CTA per node.  Cone: level L = edges incident to the node's neighbours, one merged-row hop further down per level, down to level
// 0 (T_0 = the edges whose flow value can reach a row of T_1); an edge keeps the HIGHEST level it is reached at (levels are expanded in
// descending order, so the first insertion wins).
__global__ void __launch_bounds__(kTbThreads) table_build_kernel(const BuildArgs a) {
    extern __shared__ __align__(16) unsigned char sm[];
    uint32_t* hk = reinterpret_cast<uint32_t*>(sm);       // [kTbHS] hash: edge | level << 30; later: unsorted entries / row counts
    uint32_t* list = hk + kTbHS;                           // [kTbLC] level >= 1 edges in arrival order; later: the sorted entries
    __shared__ int s_ptr[kTbMaxD], s_off[kTbMaxD + 1];
    __shared__ int s_nlist, s_m, s_n1, s_ovf, s_nat[kFusedMaxL + 2], s_warp[kTbThreads / 32];
    __shared__ unsigned s_etot;
    const int tid = threadIdx.x, lane = tid & 31, ql = tid & 3;
    const unsigned qmask = 0xFu << (lane & ~3);
    const int node = blockIdx.x, D = a.D, L = a.L;
    const bool fill = a.keys != nullptr;
    for (int i = tid; i < kTbHS; i += kTbThreads) hk[i] = kEmpty;
    if (tid == 0) {
        s_nlist = s_m = s_n1 = s_ovf = 0;
        s_etot = 0u;
    }
    for (int j = tid; j < D; j += kTbThreads) {
        const int nbr = a.nbrhoods[(size_t)node * D + j];
        s_ptr[j] = nbr >= 0 ? a.inc_ptr[nbr] : -1;
        s_off[j + 1] = nbr >= 0 ? a.inc_ptr[nbr + 1] - a.inc_ptr[nbr] : 0;
    }
    __syncthreads();
    if (tid == 0) {
        s_off[0] = 0;
        for (int j = 0; j < D; ++j) s_off[j + 1] += s_off[j];
    }
    __syncthreads();
    const int total_pairs = s_off[D];
    auto slot_of = [&](int i) {
        int j = 0;
        while (j + 1 < D && s_off[j + 1] <= i) ++j;
        return j;
    };
    const unsigned c0 = fill ? a.cone_ptr[node] : 0u;
    const int cap = fill ? (int)(a.cone_ptr[node + 1] - c0) : kTbLC;
    uint32_t* kout = fill ? a.keys + c0 : nullptr;
    auto home = [](uint32_t e) { return (e * 2654435761u) >> 17; };      // 15 bits: kTbHS slots
    auto level_of = [&](uint32_t e) -> int {                              // -1: not in the cone
        unsigned h = home(e);
        for (;;) {
            const uint32_t k = hk[h];
            if (k == kEmpty) return -1;
            if ((k & kEdgeMask) == e) return (int)(k >> 30);
            h = (h + 1) & (kTbHS - 1);
        }
    };
    auto add = [&](uint32_t e, int lv) {
        unsigned h = home(e);
        const uint32_t val = e | ((uint32_t)lv << 30);
        for (int probes = 0; probes < kTbHS; ++probes) {
            const uint32_t old = atomicCAS(&hk[h], kEmpty, val);
            if (old == kEmpty) {
                const int k = atomicAdd(&s_m, 1);
                if (k >= cap) s_ovf = 1;
                else if (kout != nullptr) kout[k] = val;
                if (lv >= 1) {                              // level 0 edges are not expanded
                    atomicAdd(&s_n1, 1);
                    const int pos = atomicAdd(&s_nlist, 1);
                    if (pos < kTbLC) list[pos] = e;
                    else s_ovf = 1;
                }
                return;
            }
            if ((old & kEdgeMask) == e) return;
            h = (h + 1) & (kTbHS - 1);
        }
        s_ovf = 1;
    };
    for (int i = tid; i < total_pairs; i += kTbThreads) {
        const int j = slot_of(i);
        add((uint32_t)a.inc_ent[s_ptr[j] + (i - s_off[j])].x, L);
    }
    __syncthreads();
    if (tid == 0) s_nat[L] = min(s_nlist, kTbLC);
    __syncthreads();
    int f0 = 0;
    for (int lv = L - 1; lv >= 0; --lv) {
        const int f1 = s_nat[lv + 1];
        if (!s_ovf)
            for (int i = f0 + (tid >> 2); i < f1; i += kTbThreads / 4) {
                const int e = (int)list[i];
                const int p1 = a.mptr[e + 1];
                for (int q = a.mptr[e] + ql; q < p1; q += 4) add((uint32_t)a.ment[q].x, lv);
            }
        __syncthreads();
        if (tid == 0) s_nat[lv] = min(s_nlist, kTbLC);
        __syncthreads();
        f0 = f1;
    }
    const int m = s_m;
    const bool bad = s_ovf != 0 || m > cap;
    if (!fill) {
        // ---- pass 1: counts.  Row entries: every entry of the rows of T_1 counts once for its own row and, if its column is a level-0
        // member, once more for the mirrored entry of that member's row (the operators are symmetric) ----
        if (!bad) {
            unsigned c = 0;
            const int n1 = s_nlist;
            for (int i = tid >> 2; i < n1; i += kTbThreads / 4) {
                const int e = (int)list[i];
                const int p1 = a.mptr[e + 1];
                for (int q = a.mptr[e] + ql; q < p1; q += 4) c += level_of((uint32_t)a.ment[q].x) == 0 ? 2u : 1u;
            }
            if (c) atomicAdd(&s_etot, c);
        }
        __syncthreads();
        if (tid == 0) {
            a.cnt_m[node] = bad ? 0 : m;
            a.cnt_e[node] = bad ? 0u : s_etot;
            a.cnt_p[node] = total_pairs;
            if (bad) a.stats[2] = 1;
            else {
                atomicMax(&a.stats[0], m);
                atomicMax(&a.stats[1], s_n1);
                atomicMax(&a.stats[3], total_pairs);
                atomicAdd(&a.stats[4 + min(kTbBuckets - 1, m / 32)], 1);
            }
        }
        return;
    }
    if (bad) {                                             // (cannot happen after a clean pass 1)
        if (tid == 0) a.stats[2] = 1;
        return;
    }
    // ---- pass 2: sort the entries by edge id (rank by counting over a shared-memory copy) ----
    __syncthreads();
    uint32_t* tmp = hk;                                    // the hash is no longer needed: lookups go through the sorted list
    for (int i = tid; i < m; i += kTbThreads) tmp[i] = kout[i];
    __syncthreads();
    uint32_t* sorted = list;
    for (int k = tid; k < m; k += kTbThreads) {
        const uint32_t v = tmp[k], e = v & kEdgeMask;
        int r = 0;
        for (int q = 0; q < m; ++q) r += (tmp[q] & kEdgeMask) < e ? 1 : 0;
        sorted[r] = v;
    }
    __syncthreads();
    for (int i = tid; i < m; i += kTbThreads) kout[i] = sorted[i];
    // readout pairs in local indices
    if (a.with_rows) {
        for (int i = tid; i < total_pairs; i += kTbThreads) {
            const int j = slot_of(i);
            const int2 es = a.inc_ent[s_ptr[j] + (i - s_off[j])];
            const int li = find_sorted(sorted, m, (uint32_t)es.x);
            a.pairs[a.pair_ptr[node] + i] = make_int2((int)((li >= 0 ? (uint32_t)li : kNoRow) | ((uint32_t)j << 16)), es.y);
        }
        for (int j = tid; j <= D; j += kTbThreads) a.pair_off[(size_t)node * (D + 1) + j] = s_off[j];
    }
    if (!a.with_rows) return;
    // ---- rows in local indices: count, scan, fill ----
    int* cnt = reinterpret_cast<int*>(hk);                 // [m + 1]
    for (int i = tid >> 2; i < m; i += kTbThreads / 4) {
        const uint32_t v = sorted[i];
        const int e = (int)(v & kEdgeMask);
        const bool full = (v >> 30) >= 1;
        const int p1 = a.mptr[e + 1];
        int c = 0;
        for (int q = a.mptr[e] + ql; q < p1; q += 4) {
            const int li = find_sorted(sorted, m, (uint32_t)a.ment[q].x);
            if (li >= 0 && (full || (sorted[li] >> 30) >= 1)) ++c;
        }
        c += __shfl_xor_sync(qmask, c, 1);
        c += __shfl_xor_sync(qmask, c, 2);
        if (ql == 0) cnt[i] = c;
    }
    __syncthreads();
    const int total = fused_block_scan_excl<kTbThreads>(cnt, m, s_warp);
    const unsigned long long nb = a.node_off[node];
    if ((unsigned long long)total != a.node_off[node + 1] - nb) {        // (uniform) pass 1 promised another size: write nothing
        if (tid == 0) a.stats[2] = 2;
        return;
    }
    unsigned* rp = a.rowptr + c0 + node;
    for (int i = tid; i <= m; i += kTbThreads) rp[i] = (unsigned)cnt[i];
    int2* ent = a.ent + nb;
    for (int i = tid >> 2; i < m; i += kTbThreads / 4) {
        const uint32_t v = sorted[i];
        const int e = (int)(v & kEdgeMask);
        const bool full = (v >> 30) >= 1;
        const int p0 = a.mptr[e], p1 = a.mptr[e + 1];
        int base = cnt[i];
        for (int q0 = p0; q0 < p1; q0 += 4) {             // (uniform inside the quad)
            const int q = q0 + ql;
            int li = -1;
            int2 en = make_int2(0, 0);
            if (q < p1) {
                en = a.ment[q];
                li = find_sorted(sorted, m, (uint32_t)en.x);
                if (li >= 0 && !(full || (sorted[li] >> 30) >= 1)) li = -1;
            }
            const bool valid = li >= 0;
            const unsigned bits = (__ballot_sync(qmask, valid) >> (lane & ~3)) & 0xFu;
            if (valid) ent[base + __popc(bits & ((1u << ql) - 1u))] = make_int2((int)((uint32_t)li | (li == i ? 0x80000000u : 0u)), en.y);
            base += __popc(bits);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// the plan of one trajectory from the node table (one CTA of THREADS threads)
// ---------------------------------------------------------------------------------------------------------------------
__host__ __device__ inline size_t table_plan_smem(int M, int LV) {
    const size_t W = (size_t)M / 32;
    return (size_t)M * 8 + (3 * W + W + 2) * 4 + (4 * (size_t)LV + 8) * 4 + 3 * (size_t)M * 2 + 3 * (size_t)LV * 2 + (size_t)M + 16;
}

// Phases (barriers are what this kernel pays for — about 17 per trajectory):
//   1  cone entries of the last node -> keys / levels; flow values placed by binary search; a non-zero value marks the level >= 1
//      members of its row live in layer 1
//   2  per layer: rank the marks (popcount prefix over the bit set), walk the live rows and mark the next layer
//   3  one pass over the live rows of all layers counts the entries of every program row; ONE scan gives every row pointer and the
//      size of the trajectory's piece of the arena (allocated inside the scan)
//   4  one pass writes everything: layer-1 scalars, forward and transposed programs (entries in column order), readout pairs
template <int THREADS>
__device__ __forceinline__ void table_plan_trajectory(const PlanArgs& a, const int t, unsigned char* sm) {
    constexpr int QUADS = THREADS / 4;
    const int M = a.M, LV = a.LV, L = a.L, D = a.D, W = M >> 5;
    uint32_t* keys = reinterpret_cast<uint32_t*>(sm);                // [M] edge ids of the cone, ascending
    float* x = reinterpret_cast<float*>(keys + M);                   // [M] flow value
    unsigned* bits = reinterpret_cast<unsigned*>(x + M);             // [3][W] live marks of layer l at (l - 1) * W
    int* wpre = reinterpret_cast<int*>(bits + 3 * W);                // [W + 2] live rows before each word
    int* cnt = wpre + W + 2;                                         // [4 LV + 8] entries per program row, programs back to back -> exclusive scan
    uint16_t* idx = reinterpret_cast<uint16_t*>(cnt + 4 * LV + 8);   // [3][M] rank of the edge among the live rows of layer l at (l - 1) * M
    uint16_t* byr = idx + 3 * M;                                     // [3][LV] local index of the row with rank r of layer l at (l - 1) * LV
    uint8_t* lv = reinterpret_cast<uint8_t*>(byr + 3 * LV);          // [M] cone level
    __shared__ int s_n, s_ovf, s_warp[THREADS / 32];
    __shared__ unsigned s_piece;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, ql = tid & 3;
    const unsigned qmask = 0xFu << (lane & ~3);
    int* hdr = a.hdr + (size_t)t * kFusedHdrW;
    auto give_up = [&]() {                                  // a table of this tier is too small: tier 0 hands the trajectory to tier 1
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
    const int last = a.last_nodes[t];
    const bool last_ok = last >= 0 && last < a.N;
    const unsigned c0 = last_ok ? a.cone_ptr[last] : 0u;
    const int m = last_ok ? (int)(a.cone_ptr[last + 1] - c0) : 0;
    if (m > M) {                                           // (uniform)
        give_up();
        return;
    }
    const int Wm = (m + 31) >> 5;
    for (int i = tid; i < m; i += THREADS) {
        const uint32_t k = a.cone_ent[c0 + i];
        keys[i] = k & kEdgeMask;
        lv[i] = (uint8_t)(k >> 30);
        x[i] = 0.f;
        idx[i] = idx[M + i] = idx[2 * M + i] = (uint16_t)kNoRow;
    }
    for (int w = tid; w < Wm; w += THREADS) bits[w] = bits[W + w] = bits[2 * W + w] = 0u;
    if (tid == 0) s_ovf = 0;
    const unsigned* rp = a.tb_rowptr + c0 + (last_ok ? last : 0);
    const int2* ent = a.tb_ent + (last_ok ? a.node_off[last] : 0ull);
    const int fp0 = a.traj_ptr[t], fp1 = a.traj_ptr[t + 1];
    __syncthreads();
    // ranks the marked rows of layer l by local index (= by edge id): idx_l[j] = rank, byr_l[rank] = j; returns the count
    auto rank_live = [&](int l) -> int {
        __syncthreads();
        const unsigned* bl = bits + (l - 1) * W;
        uint16_t* il = idx + (l - 1) * M;
        uint16_t* byrank = byr + (l - 1) * LV;
        if (warp == 0) {
            int run = 0;
            for (int base = 0; base < Wm; base += 32) {
                const int w = base + lane < Wm ? __popc(bl[base + lane]) : 0;
                int inc = w;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += v;
                }
                if (base + lane < Wm) wpre[base + lane] = run + inc - w;
                run += __shfl_sync(0xffffffffu, inc, 31);
            }
            if (lane == 0) {
                s_n = run;
                if (run > LV) s_ovf = 1;
            }
        }
        __syncthreads();
        const int n = s_n;
        if (n <= LV)
            for (int j = tid; j < m; j += THREADS) {
                const unsigned wd = bl[j >> 5];
                if ((wd >> (j & 31)) & 1u) {
                    const int r = wpre[j >> 5] + __popc(wd & ((1u << (j & 31)) - 1u));
                    il[j] = (uint16_t)r;
                    byrank[r] = (uint16_t)j;
                }
            }
        return n;                                          // (the next phase starts with a barrier)
    };

    // ---- 1: flows (a thread per entry).  Only edges of T_0 can reach a cone row; a non-zero value marks the level >= 1 members of
    // its row live in layer 1 ----
    for (int p = fp0 + tid; p < fp1; p += THREADS) {
        const int eo = a.flow_edge[p];
        if (eo < 0 || eo >= a.E) continue;
        const uint32_t e = (uint32_t)a.rank[eo];
        int lo = 0, hi = m;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (keys[mid] < e) lo = mid + 1;
            else hi = mid;
        }
        if (lo >= m || keys[lo] != e) continue;
        const float v = a.flow_val[p];
        x[lo] = v;
        if (v == 0.f) continue;
        const unsigned q1 = rp[lo + 1];
        for (unsigned q = rp[lo]; q < q1; ++q) {
            const int j = ent[q].x & 0xFFFF;
            if (lv[j] >= 1) atomicOr(&bits[j >> 5], 1u << (j & 31));
        }
    }
    // ---- 2: live rows layer by layer, and the entries per program row on the way.  Programs back to back in cnt: for s = 1 .. L the
    // forward program of layer s (s >= 2), then the transposed program of layer s + 1 (s < L); both have the live rows of layer s as
    // rows.  An entry of a live row of layer s belongs to the transposed program iff its column is live in layer s + 1, and that is
    // the case iff the column lies in T_{s+1} (it has a live neighbour below: this row) — known before layer s + 1 is ranked. ----
    int n_l[kFusedMaxL + 2] = {0, 0, 0, 0, 0};
    int pbF[kFusedMaxL + 2] = {0, 0, 0, 0, 0}, pbT[kFusedMaxL + 2] = {0, 0, 0, 0, 0}, rbase[kFusedMaxL + 2] = {0, 0, 0, 0, 0};
    int n_prog_rows = 0, n_rows = 0, ptr_words = 0;
    n_l[1] = rank_live(1);
    for (int s = 1; s <= L && !s_ovf; ++s) {               // (s_ovf: uniform, written before a barrier inside rank_live)
        __syncthreads();
        const int ns = n_l[s];
        rbase[s] = n_rows;
        n_rows += ns;
        if (s >= 2) {
            pbF[s] = n_prog_rows;
            n_prog_rows += ns;
            ptr_words += align2(ns + 1);
        }
        if (s < L) {
            pbT[s] = n_prog_rows;
            n_prog_rows += ns;
            ptr_words += align2(ns + 1);
        }
        if (s == 1 && L == 1) break;                       // (no program has the rows of layer 1 as rows, nothing to mark)
        const uint16_t* brow = byr + (s - 1) * LV;
        const uint16_t* idx_prev = idx + (s >= 2 ? s - 2 : 0) * M;
        unsigned* bn = bits + (s < L ? s : 0) * W;
        int* cF = cnt + pbF[s];
        int* cT = cnt + pbT[s];
        const int lnext = s + 1;
        for (int r = tid >> 2; r < ns; r += QUADS) {
            const int i = brow[r];
            const unsigned q1 = rp[i + 1];
            int f = 0, tr = 0;
            for (unsigned q = rp[i] + ql; q < q1; q += 4) {
                const int j = ent[q].x & 0xFFFF;
                if (s >= 2 && idx_prev[j] != (uint16_t)kNoRow) ++f;
                if (s < L && lv[j] >= lnext) {
                    ++tr;
                    atomicOr(&bn[j >> 5], 1u << (j & 31));
                }
            }
            f += __shfl_xor_sync(qmask, f, 1);
            f += __shfl_xor_sync(qmask, f, 2);
            tr += __shfl_xor_sync(qmask, tr, 1);
            tr += __shfl_xor_sync(qmask, tr, 2);
            if (ql == 0) {
                if (s >= 2) cF[r] = f;
                if (s < L) cT[r] = tr;
            }
        }
        if (s < L) n_l[s + 1] = rank_live(s + 1);
    }
    __syncthreads();
    if (s_ovf) {
        give_up();
        return;
    }
    for (int s = L + 1; s <= kFusedMaxL + 1; ++s) rbase[s] = n_rows;
    auto layer_of = [&](int row) { return row < rbase[2] ? 1 : (row < rbase[3] ? 2 : 3); };
    const unsigned pp0 = last_ok ? a.pair_ptr[last] : 0u;
    const int total_pairs = last_ok ? (int)(a.pair_ptr[last + 1] - pp0) : 0;
    const int fixed_words = align2(3 * n_l[1]) + align2(D + 1) + 2 * total_pairs + ptr_words;
    // exclusive scan of cnt[0 .. n_prog_rows) in place with the arena allocation inside (thread 0, between the scan's barriers)
    int total_ent;
    {
        const int n = n_prog_rows;
        const int per = (n + THREADS - 1) / THREADS;
        const int lo = min(n, tid * per), hi = min(n, lo + per);
        int sum = 0;
        for (int i = lo; i < hi; ++i) sum += cnt[i];
        int inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        int base = 0, total = 0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) {
            const int v = s_warp[w];
            if (w < warp) base += v;
            total += v;
        }
        int run = base + inc - sum;
        for (int i = lo; i < hi; ++i) {
            const int v = cnt[i];
            cnt[i] = run;
            run += v;
        }
        if (tid == 0) {
            cnt[n] = total;
            const unsigned long long w = (unsigned long long)(fixed_words + 2 * total);
            const unsigned long long o = atomicAdd(a.bump, w);
            if (o + w > a.arena_words) {
                s_ovf = 2;
                s_piece = 0u;
            } else {
                s_piece = (unsigned)o;
            }
        }
        __syncthreads();
        total_ent = total;
    }
    if (s_ovf) {                                           // (uniform) the arena is exhausted (the average program exceeds its share)
        if (tid == 0) {
            hdr[0] = kFusedFlagOverflow;
            *a.overflow = 1;
        }
        return;
    }
    // ---- 4: the piece: [layer-1 scalars | readout | programs in cnt order: row pointers then entries] ----
    const unsigned off_l1 = s_piece;
    const unsigned off_ro = off_l1 + (unsigned)align2(3 * n_l[1]);
    unsigned off_f[kFusedMaxL + 2] = {0, 0, 0, 0, 0}, off_b[kFusedMaxL + 2] = {0, 0, 0, 0, 0};
    int tot_f[kFusedMaxL + 2] = {0, 0, 0, 0, 0}, tot_b[kFusedMaxL + 2] = {0, 0, 0, 0, 0};
    {
        unsigned o = off_ro + (unsigned)(align2(D + 1) + 2 * total_pairs);
        for (int s = 1; s <= L; ++s) {
            if (s >= 2) {
                off_f[s] = o;
                tot_f[s] = cnt[pbF[s] + n_l[s]] - cnt[pbF[s]];
                o += (unsigned)(align2(n_l[s] + 1) + 2 * tot_f[s]);
            }
            if (s < L) {
                off_b[s + 1] = o;
                tot_b[s + 1] = cnt[pbT[s] + n_l[s]] - cnt[pbT[s]];
                o += (unsigned)(align2(n_l[s] + 1) + 2 * tot_b[s + 1]);
            }
        }
    }
    (void)total_ent;
    // row pointers (relative to the program's first entry)
    for (int s = 1; s <= L; ++s) {
        const int ns = n_l[s];
        if (s >= 2) {
            int* pF = reinterpret_cast<int*>(a.arena + off_f[s]);
            const int b0 = cnt[pbF[s]];
            for (int r = tid; r <= ns; r += THREADS) pF[r] = cnt[pbF[s] + r] - b0;
        }
        if (s < L) {
            int* pT = reinterpret_cast<int*>(a.arena + off_b[s + 1]);
            const int b0 = cnt[pbT[s]];
            for (int r = tid; r <= ns; r += THREADS) pT[r] = cnt[pbT[s] + r] - b0;
        }
    }
    {
        float* l1dst = reinterpret_cast<float*>(a.arena + off_l1);
        for (int row = tid >> 2; row < n_rows; row += QUADS) {
            const int s = layer_of(row), r = row - rbase[s];
            const int i = byr[(s - 1) * LV + r];
            const uint16_t* idx_prev = idx + (s >= 2 ? s - 2 : 0) * M;
            const uint16_t* idx_next = idx + (s < L ? s : 0) * M;
            int2* eF = reinterpret_cast<int2*>(a.arena + off_f[s] + align2(n_l[s] + 1));
            int2* eT = reinterpret_cast<int2*>(a.arena + off_b[s < L ? s + 1 : 0] + align2(n_l[s] + 1));
            int baseF = s >= 2 ? cnt[pbF[s] + r] - cnt[pbF[s]] : 0, baseT = s < L ? cnt[pbT[s] + r] - cnt[pbT[s]] : 0;
            const unsigned q0r = rp[i], q1 = rp[i + 1];
            float a1 = 0.f, a2 = 0.f;
            for (unsigned q0 = q0r; q0 < q1; q0 += 4) {      // (uniform inside the quad)
                const unsigned q = q0 + ql;
                uint32_t rf = kNoRow, rt = kNoRow;
                int2 en = make_int2(0, 0);
                if (q < q1) {
                    en = ent[q];
                    const int j = en.x & 0xFFFF;
                    if (s >= 2) rf = idx_prev[j];
                    if (s < L) rt = idx_next[j];
                    if (s == 1) {                          // the three exact scalars of a layer-1 row: x, (S0 x), (S1 x)
                        const float xj = x[j];
                        if (xj != 0.f) {
                            a1 = fmaf((float)(short)(en.y & 0xffff), xj, a1);
                            a2 = fmaf((float)(en.y >> 16), xj, a2);
                        }
                    }
                }
                const uint32_t own = (uint32_t)en.x & 0x80000000u;
                if (s >= 2) {
                    const unsigned b = (__ballot_sync(qmask, rf != kNoRow) >> (lane & ~3)) & 0xFu;
                    if (rf != kNoRow) eF[baseF + __popc(b & ((1u << ql) - 1u))] = make_int2((int)(rf | own), en.y);
                    baseF += __popc(b);
                }
                if (s < L) {
                    const unsigned b = (__ballot_sync(qmask, rt != kNoRow) >> (lane & ~3)) & 0xFu;
                    if (rt != kNoRow) eT[baseT + __popc(b & ((1u << ql) - 1u))] = make_int2((int)(rt | own), en.y);
                    baseT += __popc(b);
                }
            }
            if (s == 1) {
#pragma unroll
                for (int o = 1; o < 4; o <<= 1) {
                    a1 += __shfl_xor_sync(qmask, a1, o);
                    a2 += __shfl_xor_sync(qmask, a2, o);
                }
                if (ql == 0) {
                    l1dst[3 * r + 0] = x[i];
                    l1dst[3 * r + 1] = a1;
                    l1dst[3 * r + 2] = a2;
                }
            }
        }
    }
    // readout pairs: {row of H_L | neighbour slot << 16, sign bits}; a pair whose edge has no live row keeps kNoRow
    {
        const uint16_t* idxL = idx + (L - 1) * M;
        int* pdst = reinterpret_cast<int*>(a.arena + off_ro);
        int2* edst = reinterpret_cast<int2*>(a.arena + off_ro + align2(D + 1));
        for (int j = tid; j <= D; j += THREADS) pdst[j] = last_ok ? a.pair_off[(size_t)last * (D + 1) + j] : 0;
        for (int i = tid; i < total_pairs; i += THREADS) {
            const int2 pr = a.tb_pairs[pp0 + i];
            const uint32_t li = (uint32_t)pr.x & 0xFFFFu;
            const uint32_t r = li != kNoRow ? (uint32_t)idxL[li] : kNoRow;
            edst[i] = make_int2((int)(r | ((uint32_t)pr.x & 0xFFFF0000u)), pr.y);
        }
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
        hdr[11] = m;
        hdr[12] = tot_f[2];
        hdr[13] = fp1 - fp0;
        hdr[14] = tot_f[3];
        hdr[15] = min(tot_b[2], 0xFFFF) | (min(tot_b[3], 0xFFFF) << 16);
    }
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS) table_plan_kernel(const PlanArgs a) {
    extern __shared__ __align__(16) unsigned char sm[];
    const int n_work = a.tier == 0 ? a.n_work : *a.n_in;
    for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
        table_plan_trajectory<THREADS>(a, a.tier == 0 ? a.t0 + w : a.in_list[w], sm);
        __syncthreads();
    }
}

constexpr int kTier1Threads = 512;
constexpr size_t kMaxTablePlanSmem = 220 * 1024;

}  // namespace

void scone_table_destroy(FusedState* f) {
    cudaFree(f->d_cone_ptr); cudaFree(f->d_cone_ent); cudaFree(f->d_node_off); cudaFree(f->d_tb_rowptr); cudaFree(f->d_tb_ent);
    cudaFree(f->d_pair_ptr); cudaFree(f->d_tb_pairs); cudaFree(f->d_pair_off);
    f->d_cone_ptr = nullptr; f->d_cone_ent = nullptr; f->d_node_off = nullptr; f->d_tb_rowptr = nullptr; f->d_tb_ent = nullptr;
    f->d_pair_ptr = nullptr; f->d_tb_pairs = nullptr; f->d_pair_off = nullptr;
    f->tb_rows = false;
}

// Builds the cone table of the complex (always) and, memory permitting, the rows / pairs in local indices (tb_rows).  *ok = false: a
// cone exceeds what one build CTA holds — not the fused pipeline's regime.  Fills bound_cone / bound_list / quantile_cone.
int scone_table_build(const scone_complex* cx, FusedState* f, int L, bool* ok) {
    *ok = false;
    const int N = cx->N, D = cx->D;
    if (D > kTbMaxD || N < 1) return 0;
    const int n_stats = 4 + kTbBuckets;
    SCONE_CUDA(cudaMalloc((void**)&f->d_stats, n_stats * sizeof(int)));
    SCONE_CUDA(cudaMemset(f->d_stats, 0, n_stats * sizeof(int)));
    const size_t smem = (size_t)kTbHS * 4 + (size_t)kTbLC * 4;
    SCONE_CUDA(cudaFuncSetAttribute(table_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int* d_cnt_m = nullptr;
    unsigned* d_cnt_e = nullptr;
    int* d_cnt_p = nullptr;
    SCONE_CUDA(cudaMalloc((void**)&d_cnt_m, (size_t)N * sizeof(int)));
    SCONE_CUDA(cudaMalloc((void**)&d_cnt_e, (size_t)N * sizeof(unsigned)));
    SCONE_CUDA(cudaMalloc((void**)&d_cnt_p, (size_t)N * sizeof(int)));
    BuildArgs a{};
    a.nbrhoods = cx->d_nbrhoods; a.inc_ptr = cx->d_inc_ptr; a.inc_ent = cx->d_inc_ent; a.mptr = cx->d_mptr; a.ment = cx->d_ment;
    a.N = N; a.D = D; a.L = L; a.stats = f->d_stats;
    a.cnt_m = d_cnt_m; a.cnt_e = d_cnt_e; a.cnt_p = d_cnt_p;
    table_build_kernel<<<N, kTbThreads, smem>>>(a);
    SCONE_LAUNCHED();
    std::vector<int> st(n_stats), cm((size_t)N), cp((size_t)N);
    std::vector<unsigned> ce((size_t)N);
    SCONE_CUDA(cudaMemcpy(st.data(), f->d_stats, n_stats * sizeof(int), cudaMemcpyDeviceToHost));
    SCONE_CUDA(cudaMemcpy(cm.data(), d_cnt_m, (size_t)N * sizeof(int), cudaMemcpyDeviceToHost));
    SCONE_CUDA(cudaMemcpy(ce.data(), d_cnt_e, (size_t)N * sizeof(unsigned), cudaMemcpyDeviceToHost));
    SCONE_CUDA(cudaMemcpy(cp.data(), d_cnt_p, (size_t)N * sizeof(int), cudaMemcpyDeviceToHost));
    cudaFree(d_cnt_m); cudaFree(d_cnt_e); cudaFree(d_cnt_p);
    std::vector<unsigned> cone_ptr((size_t)N + 1), pair_ptr((size_t)N + 1);
    std::vector<unsigned long long> node_off((size_t)N + 1);
    unsigned long long tm = 0, te = 0, tp = 0;
    for (int n = 0; n < N; ++n) {
        cone_ptr[n] = (unsigned)tm; node_off[n] = te; pair_ptr[n] = (unsigned)tp;
        tm += (unsigned long long)cm[n]; te += ce[n]; tp += (unsigned long long)cp[n];
    }
    if (st[2] || tm + (unsigned long long)N + 1 >= (1ull << 32) || tp >= (1ull << 32)) return 0;
    cone_ptr[N] = (unsigned)tm; node_off[N] = te; pair_ptr[N] = (unsigned)tp;
    f->cone_entries = tm;
    int quantile999 = 0;
    f->bound_cone = st[0] > 0 ? st[0] : 1;
    f->bound_list = st[1] > 0 ? st[1] : 1;
    {
        long long acc = 0, want = ((long long)N * 99 + 99) / 100;
        int q0 = 32 * kTbBuckets;
        for (int b = 0; b < kTbBuckets; ++b) {
            acc += st[4 + b];
            if (acc >= want) {
                q0 = 32 * (b + 1);
                break;
            }
        }
        f->quantile_cone = std::min(q0, f->bound_cone);
        acc = 0;
        want = ((long long)N * 999 + 999) / 1000;
        quantile999 = f->bound_cone;
        for (int b = 0; b < kTbBuckets; ++b) {
            acc += st[4 + b];
            if (acc >= want) {
                quantile999 = std::min(32 * (b + 1), f->bound_cone);
                break;
            }
        }
    }
    // rows in local indices: only if they fit comfortably (the hash plan needs none of it)
    const unsigned long long bytes = te * 8 + (tm + (unsigned long long)N + 1) * 4 + tp * 8 + (unsigned long long)N * (D + 1) * 4 + ((unsigned long long)N + 1) * 16;
    bool want_rows = true;
    {
        const char* v = getenv("SCONE_FUSED_TABLE");
        if (v && *v == '0') want_rows = false;
        size_t free_b = 0, total_b = 0;
        SCONE_CUDA(cudaMemGetInfo(&free_b, &total_b));
        if (bytes > free_b / 3) want_rows = false;
        f->tbM = (f->bound_cone + 63) & ~63;
        f->tbLV = (f->bound_list + 63) & ~63;
        f->tb_smem = table_plan_smem(f->tbM, f->tbLV);
        if (f->tb_smem > kMaxTablePlanSmem || f->bound_cone >= 0xFFFF || f->bound_list >= 0xFFFF) want_rows = false;
    }
    SCONE_CUDA(cudaMalloc((void**)&f->d_cone_ptr, cone_ptr.size() * sizeof(unsigned)));
    SCONE_CUDA(cudaMalloc((void**)&f->d_cone_ent, (size_t)(tm ? tm : 1) * sizeof(uint32_t)));
    SCONE_CUDA(cudaMemcpy(f->d_cone_ptr, cone_ptr.data(), cone_ptr.size() * sizeof(unsigned), cudaMemcpyHostToDevice));
    a.cnt_m = nullptr; a.cnt_e = nullptr; a.cnt_p = nullptr;
    a.cone_ptr = f->d_cone_ptr; a.keys = f->d_cone_ent; a.with_rows = want_rows ? 1 : 0;
    if (want_rows) {
        SCONE_CUDA(cudaMalloc((void**)&f->d_node_off, node_off.size() * sizeof(unsigned long long)));
        SCONE_CUDA(cudaMalloc((void**)&f->d_tb_rowptr, (size_t)(tm + N + 1) * sizeof(unsigned)));
        SCONE_CUDA(cudaMalloc((void**)&f->d_tb_ent, (size_t)(te ? te : 1) * sizeof(int2)));
        SCONE_CUDA(cudaMalloc((void**)&f->d_pair_ptr, pair_ptr.size() * sizeof(unsigned)));
        SCONE_CUDA(cudaMalloc((void**)&f->d_tb_pairs, (size_t)(tp ? tp : 1) * sizeof(int2)));
        SCONE_CUDA(cudaMalloc((void**)&f->d_pair_off, (size_t)N * (D + 1) * sizeof(int)));
        SCONE_CUDA(cudaMemcpy(f->d_node_off, node_off.data(), node_off.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice));
        SCONE_CUDA(cudaMemcpy(f->d_pair_ptr, pair_ptr.data(), pair_ptr.size() * sizeof(unsigned), cudaMemcpyHostToDevice));
        a.node_off = f->d_node_off; a.rowptr = f->d_tb_rowptr; a.ent = f->d_tb_ent;
        a.pair_ptr = f->d_pair_ptr; a.pairs = f->d_tb_pairs; a.pair_off = f->d_pair_off;
    }
    table_build_kernel<<<N, kTbThreads, smem>>>(a);
    SCONE_LAUNCHED();
    SCONE_CUDA(cudaDeviceSynchronize());
    SCONE_CUDA(cudaMemcpy(st.data(), f->d_stats, 4 * sizeof(int), cudaMemcpyDeviceToHost));
    if (st[2] == 1) return 0;
    if (st[2] == 2) {                                      // the two passes disagree on a row count: keep the cone entries, drop the rows
        want_rows = false;
        SCONE_CUDA(cudaMemset(f->d_stats + 2, 0, sizeof(int)));
        cudaFree(f->d_node_off); cudaFree(f->d_tb_rowptr); cudaFree(f->d_tb_ent); cudaFree(f->d_pair_ptr); cudaFree(f->d_tb_pairs); cudaFree(f->d_pair_off);
        f->d_node_off = nullptr; f->d_tb_rowptr = nullptr; f->d_tb_ent = nullptr; f->d_pair_ptr = nullptr; f->d_tb_pairs = nullptr; f->d_pair_off = nullptr;
    }
    f->tb_rows = want_rows;
    if (want_rows) {
        f->tb_entries = te;
        f->tb_bytes = bytes;
        auto env_int = [](const char* name, int dflt) {    // tuning overrides (profiling experiments)
            const char* v = getenv(name);
            return v && *v ? atoi(v) : dflt;
        };
        // first tier: tables for the cones of ~99 % of the nodes and the live rows of all but the heaviest trajectories
        f->tbM0 = std::min(f->tbM, (env_int("SCONE_TABLE_M0", f->quantile_cone) + 63) & ~63);
        f->tbLV0 = std::min(f->tbLV, (env_int("SCONE_TABLE_LV0", 192) + 63) & ~63);
        f->tb_two_tiers = f->tbM0 < f->tbM || f->tbLV0 < f->tbLV;
        f->tb_smem0 = table_plan_smem(f->tbM0, f->tbLV0);
        // middle tier: the cones of ~99.9 % of the nodes, 512 live rows per layer — a fraction of the last tier's shared memory
        f->tbM1 = std::min(f->tbM, (env_int("SCONE_TABLE_M1", std::max(quantile999, 2 * f->tbM0)) + 63) & ~63);
        f->tbLV1 = std::min(f->tbLV, (env_int("SCONE_TABLE_LV1", 512) + 63) & ~63);
        f->tb_smem1 = table_plan_smem(f->tbM1, f->tbLV1);
        f->tb_mid_tier = f->tb_two_tiers && (f->tbM1 > f->tbM0 || f->tbLV1 > f->tbLV0) && 2 * f->tb_smem1 <= f->tb_smem;
        SCONE_CUDA(cudaFuncSetAttribute(table_plan_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxTablePlanSmem));
        SCONE_CUDA(cudaFuncSetAttribute(table_plan_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxTablePlanSmem));
        SCONE_CUDA(cudaFuncSetAttribute(table_plan_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxTablePlanSmem));
        SCONE_CUDA(cudaFuncSetAttribute(table_plan_kernel<kTier1Threads>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxTablePlanSmem));
    }
    *ok = true;
    return 0;
}

// Plans b trajectories (p: trajectories, outputs, retry list already set) with the table plan: first tier, then the retry list.
// phase 0: the first tier only, over trajectories p.t0 .. p.t0 + b (its give-ups are APPENDED to the work list: the counters are not
// reset between launches); phase 1: the later tiers over the accumulated work list (b = trajectories of the whole chunk); 2: both.
int scone_table_plan_launch(const FusedState* f, PlanArgs p, int b, int num_sms, cudaStream_t st, int phase) {
    const int f_chunk = f->chunk;
    p.cone_ptr = f->d_cone_ptr; p.cone_ent = f->d_cone_ent; p.node_off = f->d_node_off; p.tb_rowptr = f->d_tb_rowptr; p.tb_ent = f->d_tb_ent;
    p.pair_ptr = f->d_pair_ptr; p.tb_pairs = f->d_tb_pairs; p.pair_off = f->d_pair_off;
    p.tier = 0; p.n_work = b;
    p.M = f->tbM0; p.LV = f->tbLV0;
    // up to three tiers; a tier hands the trajectories its tables cannot hold to the next one through a work list
    int* list0 = p.retry;                                  // [2][chunk]
    int* list1 = p.retry + f_chunk;
    int* cnt0 = p.n_retry;                                 // two int counters (zeroed by the caller)
    int* cnt1 = p.n_retry + 1;
    p.retry = f->tb_two_tiers ? list0 : nullptr;
    p.n_retry = cnt0;
    if (phase != 1) {
        static const int t0 = [] { const char* v = getenv("SCONE_TABLE_T0"); return v && *v ? atoi(v) : 128; }();
        if (t0 == 64) table_plan_kernel<64><<<b, 64, f->tb_smem0, st>>>(p);
        else if (t0 == 256) table_plan_kernel<256><<<b, 256, f->tb_smem0, st>>>(p);
        else table_plan_kernel<128><<<b, 128, f->tb_smem0, st>>>(p);
        SCONE_LAUNCHED();
    }
    if (!f->tb_two_tiers || phase == 0) return 0;
    const int* n_in = cnt0;
    const int* in_list = list0;
    if (f->tb_mid_tier) {                                  // tables for all but the largest cones: 256 threads, several CTAs per SM
        p.tier = 1; p.M = f->tbM1; p.LV = f->tbLV1; p.n_in = n_in; p.in_list = in_list; p.retry = list1; p.n_retry = cnt1;
        const int per_sm = std::max(1, std::min(8, (int)((size_t)220 * 1024 / (f->tb_smem1 + 1024))));
        table_plan_kernel<256><<<std::min(b, per_sm * num_sms), 256, f->tb_smem1, st>>>(p);
        SCONE_LAUNCHED();
        n_in = cnt1;
        in_list = list1;
    }
    p.tier = 2; p.M = f->tbM; p.LV = f->tbLV; p.n_in = n_in; p.in_list = in_list; p.retry = nullptr; p.n_retry = cnt0;
    const int per_sm = std::max(1, std::min(4, (int)((size_t)220 * 1024 / (f->tb_smem + 1024))));
    table_plan_kernel<512><<<std::min(b, per_sm * num_sms), 512, f->tb_smem, st>>>(p);
    SCONE_LAUNCHED();
    return 0;
}
