// fused.cuh — state and entry points of the trajectory-fused pipeline (scone_fused.cu), used by scone_model.cu.
#pragma once
#include "common.cuh"

constexpr int kFusedMaxL = 3;             // conv layers the fused compute kernel keeps weight-gradient tiles in registers for
constexpr int kFusedHdrW = 16;            // ints per trajectory header
constexpr int kFusedFlagOverflow = 1;
constexpr int kFusedFlagRetry = 2;        // tier 0 of the plan kernel overflowed its tables: tier 1 redoes the trajectory

// Per-trajectory header written by fused_plan_kernel (word offsets into the program arena):
//   [0] flags   [1..3] live rows of layers 1..3   [4] layer-1 scalars {x, S0 x, S1 x} per row
//   [5],[6] forward programs of layers 2, 3: rowptr[n_l + 1] then int2 entries {row below | own << 31, (c1 << 16) | c0}
//   [7],[8] transposed programs of layers 2, 3 (rows = live rows of layer l - 1, entries = rows of layer l)
//   [9] readout: rowptr[D + 1] then int2 {row of H_L | slot << 16, sign bits}   [10] pairs   [11] hash entries (flows + cone)
//   [12] / [14] entries of the forward programs of layers 2 / 3   [13] flow entries
//   [15] entries of the transposed programs of layers 2 (low half) and 3 (high half), saturated at 0xFFFF
// Arguments of the plan kernels (both flavours: the hash plan of scone_fused.cu and the table plan of scone_plan_table.cu)
struct PlanArgs {
    const int32_t* traj_ptr;
    const int32_t* flow_edge;
    const float* flow_val;
    const int32_t* last_nodes;
    const int32_t* rank;
    const int32_t* nbrhoods;
    const int32_t* inc_ptr;
    const int2* inc_ent;
    const int32_t* mptr;
    const int2* ment;
    int N, D, E, L;
    int HS, hshift;            // hash plan: hash slots (power of two): the flow edges and the cone T_0 of the trajectory
    const unsigned* cone_ptr;  // cone table: entries of node n at cone_ent[cone_ptr[n] .. cone_ptr[n + 1]), ascending edge id
    const uint32_t* cone_ent;  //   edge | level << 30
    int LV;                    // live rows per layer
    int EC;                    // hash plan: merged-row entries of the live rows of one layer (slot buffer)
    // node table (table plan): the operator rows of the cone in LOCAL indices (position of the edge in the node's cone entries)
    int M;                     // cone entries this tier's tables hold
    const unsigned long long* node_off;   // [N + 1] first row entry of node n
    const unsigned* tb_rowptr;            // m + 1 local offsets per node, at cone_ptr[n] + n
    const int2* tb_ent;                   // {local column | own << 31, (c1 << 16) | c0}, ascending column
    const unsigned* pair_ptr;             // [N + 1] readout pairs of node n
    const int2* tb_pairs;                 // {local index | neighbour slot << 16, sign bits}
    const int* pair_off;                  // [N][D + 1] first pair of every neighbour slot
    int* hdr;
    uint32_t* arena;
    unsigned long long* bump;
    unsigned long long arena_words;
    int* overflow;
    int tier;                  // 0: trajectory = work item, tables sized for ~99 % of the nodes; >= 1: the work list of the tier before
    int n_work;                // tier 0: trajectories of the chunk
    int t0;                    // tier 0: first trajectory of this launch (work item w = trajectory t0 + w)
    const int* n_in;           // tier >= 1: work list = the trajectories the tier before gave up on (device counter + list)
    const int* in_list;
    int* n_retry;              // trajectories this tier gives up on (tables too small): device counter + list; retry == NULL: last tier,
    int* retry;                //   giving up = the overflow flag
    unsigned* fg_off;          // flow-gradient plan (NULL: none): word offset of trajectory t's layer-0 transposed program (below)
};

#ifdef __CUDACC__
// exclusive scan of a[0..n) in place (a[n] = total); every thread of the THREADS-thread CTA calls it
template <int THREADS>
__device__ inline int fused_block_scan_excl(int* a, int n, int* s_warp) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + THREADS - 1) / THREADS;
    const int lo = min(n, tid * per), hi = min(n, lo + per);
    int sum = 0;
    for (int i = lo; i < hi; ++i) sum += a[i];
    int inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    __syncthreads();                                      // (s_warp may still be read from a previous call)
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
        const int v = a[i];
        a[i] = run;
        run += v;
    }
    if (tid == 0) a[n] = total;
    __syncthreads();
    return total;
}

// Layer-0 transposed program of a flow-gradient plan (both plan kernels; written at PlanArgs::fg_off[t]): row pointers [n_f + 1]
// (relative to the first entry) then int2 entries {live layer-1 row | own << 31, (c1 << 16) | c0} in column order, the format of the
// transposed programs of layers 2 / 3.  One row per flow entry of the trajectory in CSR order; an entry outside T_0 or with an edge id
// out of range has an empty row.  row(i, emit) calls emit(entry) for the entries of flow entry i in column order.  The rows go
// kFlowChunk at a time: one pass counts (the size of the arena piece), a second scans each chunk and writes it.  Returns the piece's
// word offset, or ~0u when the arena is exhausted (block-uniform; every thread of the THREADS-thread CTA calls it).
constexpr int kFlowChunk = 128;
template <int THREADS, typename Row>
__device__ unsigned fused_flow_program(const PlanArgs& a, int n_f, int* s_warp, Row row) {
    static_assert(THREADS >= kFlowChunk, "a thread per row of a chunk");
    __shared__ int s_c[kFlowChunk + 1];
    __shared__ unsigned s_off;
    const int tid = threadIdx.x;
    auto count = [&](int i) {
        int c = 0;
        if (tid < kFlowChunk && i < n_f) row(i, [&](int2) { ++c; });
        if (tid < kFlowChunk) s_c[tid] = c;
    };
    int total = 0;
    for (int base = 0; base < n_f; base += kFlowChunk) {
        count(base + tid);
        total += fused_block_scan_excl<THREADS>(s_c, kFlowChunk, s_warp);
    }
    const int ptr_words = (n_f + 2) & ~1;
    if (tid == 0) {
        const unsigned long long w = (unsigned long long)ptr_words + 2ull * (unsigned long long)total;
        const unsigned long long o = atomicAdd(a.bump, w);
        s_off = o + w > a.arena_words ? ~0u : (unsigned)o;
    }
    __syncthreads();
    const unsigned off = s_off;
    if (off == ~0u) return off;
    int* ptr = reinterpret_cast<int*>(a.arena + off);
    int2* ent = reinterpret_cast<int2*>(a.arena + off + ptr_words);
    int run = 0;
    for (int base = 0; base < n_f; base += kFlowChunk) {
        const int i = base + tid;
        count(i);
        const int chunk_total = fused_block_scan_excl<THREADS>(s_c, kFlowChunk, s_warp);
        if (tid < kFlowChunk && i < n_f) {
            int k = run + s_c[tid];
            ptr[i] = k;
            row(i, [&](int2 en) { ent[k++] = en; });
        }
        run += chunk_total;
    }
    if (tid == 0) ptr[n_f] = run;
    return off;
}
#endif

struct FusedState {
    int L = 0, C = 0;
    int64_t n_params = 0;
    int bound_cone = 0, bound_list = 0;   // static bounds of the complex: |T_0| (hash entries) / |T_1| (rows of a layer) of any last node
    unsigned* d_cone_ptr = nullptr;       // cone table: T_0 of every node, entries edge | level << 30
    uint32_t* d_cone_ent = nullptr;
    unsigned long long cone_entries = 0;
    // node table (scone_plan_table.cu): operator rows of every node's cone in local indices + its readout pairs
    bool tb_rows = false;                 // the table holds rows: plans come from table_plan_kernel (else: the hash plan)
    unsigned long long* d_node_off = nullptr;
    unsigned* d_tb_rowptr = nullptr;
    int2* d_tb_ent = nullptr;
    unsigned* d_pair_ptr = nullptr;
    int2* d_tb_pairs = nullptr;
    int* d_pair_off = nullptr;
    unsigned long long tb_entries = 0, tb_bytes = 0;
    int tbM0 = 0, tbLV0 = 0, tbM1 = 0, tbLV1 = 0, tbM = 0, tbLV = 0;   // table plan tiers: cone entries / live rows per layer the tables hold
    size_t tb_smem0 = 0, tb_smem1 = 0, tb_smem = 0;
    bool tb_two_tiers = false, tb_mid_tier = false;
    int quantile_cone = 0;                // |T_0| of ~99 % of the nodes
    int HS = 0, LV = 0, EC = 0, hshift = 0;        // plan tables, tier 1: sized by the bounds
    int HS0 = 0, LV0 = 0, EC0 = 0, hshift0 = 0;   // tier 0: sized for the cones of 99 % of the nodes
    bool two_tiers = false;
    int flow_room = 0;
    size_t plan_smem0 = 0;
    unsigned long long worst_words = 0;
    int* d_retry = nullptr;               // [2][chunk] work lists handed from tier to tier
    size_t plan_smem = 0, traj_smem_small = 0, traj_smem_big = 0;
    int cap_rows = 0, big_rows = 0, grid_small = 0, grid_big = 0, chunk = 0;
    size_t scratch_stride = 0;
    unsigned long long arena_words = 0;
    int* d_hdr = nullptr;
    uint32_t* d_arena = nullptr;
    unsigned long long* d_bump = nullptr;
    float* d_partial = nullptr;
    float* d_scratch = nullptr;
    int* d_stats = nullptr;
    unsigned long long* d_rows_done = nullptr;
    uint32_t* d_sort = nullptr;           // cost-sorted batch: keys in / out, trajectories in / out
    void* d_sort_tmp = nullptr;
    size_t sort_tmp_bytes = 0;
    int sort_cap = 0;
    // planned set (scone_fused_plan_set): headers + programs of a whole dataset, kept across calls
    unsigned* d_fg_off = nullptr;         // [chunk] layer-0 transposed programs of a flow-gradient plan (allocated on first use)
    int* d_set_hdr = nullptr;
    uint32_t* d_set_arena = nullptr;
    unsigned long long* d_set_bump = nullptr;
    unsigned long long set_arena_words = 0;
    int set_cap = 0, set_n = 0;
};

// scone_plan_table.cu
int scone_table_build(const scone_complex* cx, FusedState* f, int L, bool* ok);
int scone_table_plan_launch(const FusedState* f, PlanArgs p, int b, int num_sms, cudaStream_t st, int phase = 2);
void scone_table_destroy(FusedState* f);

bool scone_fused_supported(const scone_complex* cx, int n_layers, const int32_t* hidden);
int scone_fused_create(const scone_complex* cx, int L, int C, int mb, int64_t n_params, FusedState** out);
void scone_fused_destroy(FusedState* f);
int scone_fused_run(const scone_complex* cx, FusedState* f, int act, int b, const int32_t* traj_ptr, const int32_t* flow_edge,
                    const float* flow_val, const int32_t* last_nodes, const float* W, const int64_t* w_off, float* logprobs,
                    const int32_t* target_idx, const float* mask, float* grad, int* overflow, bool count_rows, cudaStream_t st,
                    const float* cot = nullptr,    // cot [b][D] (with grad): cotangent seed instead of target_idx / mask
                    float* dflow = nullptr);       // (with cot) d(sum cot * logprob) / d flow_val, indexed like flow_val
int scone_fused_begin(FusedState* f, cudaStream_t st);
int scone_fused_plan_part(const scone_complex* cx, FusedState* f, int off, int b, const int32_t* traj_ptr, const int32_t* flow_edge,
                          const float* flow_val, const int32_t* last_nodes, int* overflow, cudaStream_t st,
                          bool defer_tiers = false, bool flow_grad = false);
int scone_fused_plan_finish(const scone_complex* cx, FusedState* f, int B, const int32_t* traj_ptr, const int32_t* flow_edge,
                            const float* flow_val, const int32_t* last_nodes, int* overflow, cudaStream_t st);
int scone_fused_compute(const scone_complex* cx, FusedState* f, int act, int b, const float* W, const int64_t* w_off, float* logprobs,
                        const int32_t* target_idx, const float* mask, float* grad, bool count_rows, cudaStream_t st,
                        const float* cot = nullptr, float* dflow = nullptr, const int32_t* traj_ptr = nullptr);
int scone_fused_plan_set(const scone_complex* cx, FusedState* f, int B, const int32_t* traj_ptr, const int32_t* flow_edge,
                         const float* flow_val, const int32_t* last_nodes, int* overflow, cudaStream_t st);
int scone_fused_run_planned(const scone_complex* cx, FusedState* f, int act, int n, const int32_t* rows_dev, const float* W, const int64_t* w_off,
                            float* logprobs, const int32_t* target_idx, const float* mask, float* grad, bool count_rows, cudaStream_t st,
                            const float* cot = nullptr);
int scone_fused_last_retries(FusedState* f);
int scone_fused_read(FusedState* f, int t, int* hdr_out, unsigned off, int words, uint32_t* arena_out);
