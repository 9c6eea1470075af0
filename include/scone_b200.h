/*
 * scone_b200.h — C ABI of the B200-native SCoNe hot path (libscone_b200.so).
 *
 * The reference (nglaze00/SCoNe_GCN) is pure Python/JAX and has no FFI; the seam this library sits
 * behind is the per-sample model function that Scone_GCN.setup vmaps
 * (trajectory_analysis/scone_trajectory_model.py:256) and that Scone_GCN.loss / accuracy / train call
 * (:46, :64, :307).  Each entry point below names the reference code it replaces.  All functions
 *   - return 0 on success, non-zero on error (message: scone_last_error(), thread-local),
 *   - never throw across the ABI, never allocate behind the caller's back except inside the opaque
 *     handles (scone_complex, scone_model), and launch only on the stream they are given
 *     (`stream` is a cudaStream_t passed as void*; NULL = legacy default stream),
 *   - take plain pointers and sizes.  "dev" = device pointer, "host" = host pointer.
 *
 * Device layouts (fp32, row-major; e = INTERNAL edge row, see scone_complex_get_edge_rank):
 *   activations  H[e][t][c]  -> ((e * b) + t) * C + c      e < E edges, t < b trajectories, c < C channels
 *   flows        X[e][t]     -> e * b + t                  (layer-0 input, C = 1)
 *   weights      flat concatenation of the reference's weight list, each [C_in][C_out] row-major, in
 *                list order W[0], W[1], ... (scone_trajectory_model.py:222-237).
 */
#ifndef SCONE_B200_H
#define SCONE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCONE_B200_VERSION 100
/* Largest maximum node degree D (width of the neighbour table) the model entry points support: the readout, cone and plan kernels
 * keep per-slot arrays of this size in shared memory.  scone_model_create rejects a complex with a larger D (error code 2). */
#define SCONE_MAX_DEGREE 128

typedef struct scone_complex scone_complex;   /* simplicial complex: device-resident index arrays */
typedef struct scone_model scone_model;       /* weights + Adam state + activation workspace     */

enum { SCONE_MODEL_SCONE = 0, SCONE_MODEL_EBLI = 1, SCONE_MODEL_BUNCH = 2 };
enum { SCONE_ACT_TANH = 0, SCONE_ACT_LEAKY_RELU = 1, SCONE_ACT_RELU = 2 };

int scone_version(void);
const char* scone_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * Complex construction — replaces the dense operator assembly
 *   L1_lower = B1.T @ B1 ; L1_upper = B2 @ B2.T ; ebli: L1, L1 @ L1      trajectory_experiments.py:239-253
 *   nbrhoods / n_nbrs / B1_jax / Bconds_func                               trajectory_experiments.py:262-303
 * Input is the signed incidence structure itself (what B1.npy / B2.npy encode,
 * synthetic_data_gen.py:139-161): per edge its two end nodes and their B1 signs, per triangle its three
 * edges and their B2 signs.  edge_signs == NULL means (-1,+1) (tail, head); `-flip_edges 1`
 * (trajectory_experiments.py:214-219,242-244,290) is expressed by passing the flipped signs.
 * All integer work is exact.  model selects which shift pair is built: scone -> (L_lower, L_upper),
 * ebli -> (L1, L1^2).
 * ------------------------------------------------------------------------------------------- */
int scone_complex_create(int32_t n_nodes, int32_t n_edges, int32_t n_tris,
                         const int32_t* edge_nodes /* host [E][2] */, const int8_t* edge_signs /* host [E][2] or NULL */,
                         const int32_t* tri_edges /* host [F][3] */, const int8_t* tri_signs /* host [F][3] */,
                         int32_t model, scone_complex** out);
/* Same exact index construction, but WITHOUT touching a GPU: the handle only serves the copy-out getters
 * below (bit-exact index parity tests on a CPU-only machine); every compute entry point refuses it. */
int scone_complex_create_index_only(int32_t n_nodes, int32_t n_edges, int32_t n_tris,
                                    const int32_t* edge_nodes, const int8_t* edge_signs,
                                    const int32_t* tri_edges, const int8_t* tri_signs,
                                    int32_t model, scone_complex** out);
int scone_complex_destroy(scone_complex* cx);
/* dims: N, E, F, D (max degree), nnz of shift 0, nnz of shift 1 */
int scone_complex_dims(const scone_complex* cx, int32_t* n_nodes, int32_t* n_edges, int32_t* n_tris,
                       int32_t* max_degree, int64_t* nnz0, int64_t* nnz1);
/* copy-out (host buffers) for bit-exact parity tests */
int scone_complex_get_shift_csr(const scone_complex* cx, int32_t which, int32_t* rowptr /* [E+1] */,
                                int32_t* col /* [nnz] */, float* val /* [nnz] */);
int scone_complex_get_nbrhoods(const scone_complex* cx, int32_t* nbrhoods /* [N][D], pad -1 */);
/* Device tensors H[E][b][C], X[E][b] and the occupancy flags are stored in an INTERNAL edge order chosen for memory
 * locality (Hilbert curve over two BFS distance fields); rank[e] is the internal row of the caller's edge e.  The
 * model-level entry points and scone_flows_to_dense translate for the caller; only code that fills H directly
 * (kernel-level tests, the jax.ffi layer ops) needs this map. */
int scone_complex_get_edge_rank(const scone_complex* cx, int32_t* rank /* host [E] */);

/* ---------------------------------------------------------------------------------------------
 * Kernel-level entry points (device pointers).  These are what a jax.ffi handler binds, one per
 * custom call; INTEGRATION.md shows the shim.
 * ------------------------------------------------------------------------------------------- */

/* path_to_flow output (synthetic_data_gen.py:327-344) in sparse form -> dense X[E][b].
 * Trajectory t owns entries [traj_ptr[t], traj_ptr[t+1]) of (flow_edge, flow_val). */
int scone_flows_to_dense(const scone_complex* cx, int32_t b, const int32_t* traj_ptr_dev /* [b+1] */,
                         const int32_t* flow_edge_dev, const float* flow_val_dev, float* X_dev /* [E][b] */,
                         uint8_t* occ_X_dev /* [E][b] flags of X, or NULL */, void* stream);

/* One fused Hodge-Laplacian convolution layer, forward:
 *   Hout = act(Hin W0 + (S0 Hin) W1 + (S1 Hin) W2)                       trajectory_experiments.py:145-149,163-167
 * Hin [E][b][cin], Hout [E][b][cout], W* [cin][cout] (device).
 * Occupancy flags (optional, NULL = none): occ[e*b + t] == 0 promises that row (e, t) of the tensor is entirely
 * zero (a superset of the non-zero rows is fine).  There is no bias and act(0) == 0, so activations are structurally
 * zero outside the l-hop neighbourhood of a trajectory (SURVEY.md §7).  With occ_in the call (1) compacts the flagged
 * units of the input into a worklist, (2) scatters the support one hop into occ_out, (3) compacts occ_out, and (4) runs
 * one warp per candidate unit; unflagged neighbour rows are never read.  Results are bit-identical to the dense
 * kernel.  occ_scratch: scone_occ_scratch_bytes(cx, b) bytes.  Without occ_in the dense tile kernel runs and occ_out
 * (if given) is set to all ones. */
int64_t scone_occ_scratch_bytes(const scone_complex* cx, int32_t b);
int scone_layer_forward(const scone_complex* cx, int32_t act, int32_t b, int32_t cin, int32_t cout,
                        const float* Hin_dev, const float* W0_dev, const float* W1_dev, const float* W2_dev,
                        float* Hout_dev, const uint8_t* occ_in_dev, uint8_t* occ_out_dev, uint8_t* occ_scratch_dev,
                        void* stream);

/* Backward of the same layer (what jax.grad derives from the lines above, scone_trajectory_model.py:307).
 * G_dev = dL/dZ of this layer ( = dL/dHout * act'(Hout), already multiplied) [E][b][cout].
 * Outputs:  Gprev_dev [E][b][cin] = dL/dZ of the previous layer = (dL/dHin) * act'(Hin)
 *           (pass NULL for the first layer: the reference never differentiates w.r.t. the flows);
 *           dW_dev [3][cin][cout] += sum over rows, reduced in a fixed order (deterministic, no atomics).
 * workspace: scone_layer_backward_workspace_bytes(cin, cout) bytes, device. */
int64_t scone_layer_backward_workspace_bytes(int32_t cin, int32_t cout);
int scone_layer_backward(const scone_complex* cx, int32_t act, int32_t b, int32_t cin, int32_t cout,
                         const float* G_dev, const float* Hin_dev,
                         const float* W0_dev, const float* W1_dev, const float* W2_dev,
                         float* Gprev_dev, float* dW_dev, int32_t accumulate, void* workspace_dev,
                         const uint8_t* occ_g_dev, const uint8_t* occ_hin_dev, uint8_t* occ_gprev_dev,
                         uint8_t* occ_scratch_dev, void* stream);

/* Readout + padded log-softmax (+ NLL and its gradient):
 *   logits = Bcond(last_node) @ H_L @ w_out ; logits - logsumexp(logits)   trajectory_experiments.py:151-152,298-303
 *   loss term  -sum(preds * y) over masked rows                            scone_trajectory_model.py:46,54
 * logprobs_dev [b][D].  If GL_dev != NULL also writes GL = dL/dZ of the last conv layer
 * [E][b][C] (zero except on edges incident to the neighbours of last_node), the w_out gradient
 * (dwout_dev [C]), the masked NLL sum (*nll_sum_dev) and the mask count (*count_dev) — each reduced over
 * trajectories in ascending order and added to the destination when accumulate != 0.
 * workspace_dev: scone_readout_workspace(b, C) bytes (gradient mode only).
 * target_idx_dev[t] = argmax of the one-hot target row; mask_dev[t] in {0,1}; scale multiplies the
 * upstream gradient (1 / number of masked rows in the whole batch). */
int64_t scone_readout_workspace(int32_t b, int32_t C);
int scone_readout(const scone_complex* cx, int32_t act, int32_t b, int32_t C,
                  const float* HL_dev, const float* wout_dev, const int32_t* last_nodes_dev,
                  float* logprobs_dev,
                  const int32_t* target_idx_dev, const float* mask_dev, float scale,
                  float* GL_dev, float* dwout_dev, float* nll_sum_dev, float* count_dev, int32_t accumulate,
                  void* workspace_dev, const uint8_t* occ_HL_dev, uint8_t* occ_GL_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Model-level entry points — replace Scone_GCN.{setup, loss, accuracy, train's adam_step}
 * (scone_trajectory_model.py:42-71,215-262,300-326) for -model scone / ebli.
 * hidden[l] = channel count of layer l (the reference's hidden_layers[l][1]); micro_batch = number of
 * trajectories resident per pass (activations are [E][micro_batch][C] per layer).
 * ------------------------------------------------------------------------------------------- */
int scone_model_create(const scone_complex* cx, int32_t n_layers, const int32_t* hidden, int32_t micro_batch,
                       scone_model** out);
int scone_model_destroy(scone_model* m);
int64_t scone_model_num_params(const scone_model* m);
/* The model-level calls keep their activation / gradient tensors private, so by default (0) unflagged rows are never written
 * and traffic follows the support of the trajectories; 1 = bulk zero-fill every tensor once per micro-batch (complete dense
 * [E][b][C] arrays, the dense-streaming formulation).  Results are bit-identical either way. */
int scone_model_set_zero_fill(scone_model* m, int32_t on);
int scone_model_get_zero_fill(const scone_model* m);
/* Model-level pipeline (same results within fp32 rounding; buffers of a pipeline are allocated on first use):
 *   3 (default when every hidden width is 16 or 32) = pipeline 2's kernels restricted to the READOUT CONE: the log-probs of a
 *     trajectory read H_L only at the edges incident to the neighbours of its last node (trajectory_experiments.py:151,298-303),
 *     H_{L-1} one hop around those, and so on; the cone of layer l is both the rows of H_l the forward must produce and the rows
 *     of G_l the backward produces, so each layer has one bitmap / rank prefix / row list, built from last_nodes before the
 *     forward; inside the cone only the rows in the structural support of the flows (LIVE rows) are computed.  Log-probs are
 *     bit-identical to pipeline 2, gradients equal up to the grouping of the fp32 sums (tests).  Row ids are 32-bit unsigned:
 *     E * micro_batch < 2^32 (2^31 for the other pipelines).  Capacities per micro-batch: 32 M rows per compact tensor, 6 M rows
 *     of the backward's A buffer, 2048 cone edges per trajectory and layer; beyond them scone_model_read_grads /
 *     scone_model_forward_host report an error (complexes with max degree > 32 therefore start on pipeline 2).
 *   2 = row lists over COMPACT tensors, whole support: each tensor carries a row bitmap, row r is
 *     stored at index rank(r) = its position in the compacted row list, producers mark the candidate rows of the next tensor,
 *     per layer one bitmap compaction + one row-list kernel (tensor-core product).  Memory and traffic follow the support of
 *     the trajectories, so micro_batch can be thousands (E * micro_batch < 2^31).  A compact tensor holds at most 32 M rows and
 *     the backward's A buffer 6 M rows per micro-batch; beyond that scone_model_read_grads reports an error.
 *   1 = the same row-list kernels over dense [E][micro_batch][C] tensors.
 *   0 = unit kernels over byte flags and dense tensors (every width; fp32 SIMT).  zero_fill = 1 always uses 0. */
/*   4 (default when all hidden widths are equal, 16 or 32, with at most 3 layers, and the cones of the complex fit the shared-memory
 *     tables) = TRAJECTORY-FUSED kernels (csrc/scone_fused.cu): one plan kernel (cone & support -> per-trajectory live rows in ascending
 *     edge order + gather programs; weight-independent integer work) and one compute kernel that keeps all activations and
 *     gradients of a trajectory in shared memory (gather -> 3xTF32 mma.sync product -> activation per layer, readout, log-softmax,
 *     NLL, backward, weight-gradient tiles in registers across trajectories) + one fixed-order reduce of the per-CTA partials.
 *     Same live rows as pipeline 3, each computed from the same neighbours in the same (ascending column) order.  No capacity can
 *     overflow: every table is sized from bounds measured on the complex at scone_model_create (the cone of every node).
 *     Nothing is proportional to E * micro_batch (no dense X, no bitmaps), so E * micro_batch is unbounded. */
int scone_model_set_pipeline(scone_model* m, int32_t which);
int scone_model_get_pipeline(const scone_model* m);
int scone_model_set_weights(scone_model* m, const float* weights_host);     /* also resets Adam state */
int scone_model_get_weights(const scone_model* m, float* weights_host);
float* scone_model_weights_dev(scone_model* m);                              /* flat device weights      */
float* scone_model_grads_dev(scone_model* m);                                /* flat [n_params + 2]: grads, nll_sum, count */

/* Batched forward: log-probs for B trajectories given as sparse flows (HOST buffers; copies inside).
 * Replaces self.model(weights, *shifts, *inputs) (scone_trajectory_model.py:46,64). */
int scone_model_forward_host(scone_model* m, int32_t B, const int32_t* traj_ptr /* [B+1] */,
                             const int32_t* flow_edge, const float* flow_val, const int32_t* last_nodes,
                             float* logprobs_out /* [B][D] */, void* stream);
/* Same with DEVICE buffers (inputs already resident). */
int scone_model_forward_dev(scone_model* m, int32_t B, const int32_t* traj_ptr_dev, const int32_t* flow_edge_dev,
                            const float* flow_val_dev, const int32_t* last_nodes_dev, float* logprobs_dev, void* stream);

/* Loss + weight gradients over B trajectories (forward + backward, micro-batched), accumulating the
 * UNNORMALISED sums into the model's flat gradient buffer [grads | nll_sum | count]:
 *   grads += sum_t mask_t * d(-log p_t[target_t])/dW ;  nll_sum += ... ; count += sum(mask).
 * Replaces grad(self.loss) minus the ridge term and the 1/sum(mask) factor, which scone_model_adam_step
 * applies after the (optional) cross-GPU all-reduce of that buffer.  zero_first != 0 clears the buffer. */
int scone_model_loss_grad_dev(scone_model* m, int32_t B, const int32_t* traj_ptr_dev, const int32_t* flow_edge_dev,
                              const float* flow_val_dev, const int32_t* last_nodes_dev,
                              const int32_t* target_idx_dev, const float* mask_dev, int32_t zero_first, void* stream);
int scone_model_loss_grad_host(scone_model* m, int32_t B, const int32_t* traj_ptr, const int32_t* flow_edge,
                               const float* flow_val, const int32_t* last_nodes,
                               const int32_t* target_idx, const float* mask, int32_t zero_first, void* stream);
/* Next-node accuracy on the device (scone_trajectory_model.py:59-71): for every trajectory with mask != 0 the prediction is
 * argmax_j of (j < n_nbrs[t] ? logprobs[t][j] : -100) over ALL D slots — the first maximum wins, a NaN wins over numbers, as
 * NumPy / JAX argmax — compared with target_idx[t].  out[0] = correct predictions, out[1] = masked trajectories (integers:
 * accuracy = out[0] / out[1], identical to np.mean(pred_choice == target_choice)).  out_dev is overwritten. */
int scone_accuracy_dev(int32_t B, int32_t D, const float* logprobs_dev, const int32_t* n_nbrs_dev,
                       const int32_t* target_idx_dev, const float* mask_dev, int32_t* out_dev /* [2] */, void* stream);
/* Forward + accuracy from HOST buffers (micro-batched forward, the log-probs never leave the device); out_host[2] as above. */
int scone_model_accuracy_host(scone_model* m, int32_t B, const int32_t* traj_ptr, const int32_t* flow_edge,
                              const float* flow_val, const int32_t* last_nodes, const int32_t* n_nbrs,
                              const int32_t* target_idx, const float* mask, int32_t* out_host /* [2] */, void* stream);
/* Evaluation with the log-probs staying on the device (the host-side metric loops of scone_trajectory_model.py:42-56 loss,
 * :59-71 accuracy, :73-108 two_target_accuracy): forward over B trajectories from HOST buffers, then on the device, each optional
 * (NULL = skip):  choice_out [B] = argmax_j (j < n_nbrs[t] ? logprob : -100), first maximum, as NumPy / JAX (needs n_nbrs);
 * acc_out [2] = correct predictions, masked trajectories (needs n_nbrs, target_idx, mask);  nll_out [2] = sum of -mask *
 * logprob[target] (fixed summation order), sum of mask (needs target_idx, mask).  Synchronises the stream. */
int scone_model_eval_host(scone_model* m, int32_t B, const int32_t* traj_ptr, const int32_t* flow_edge, const float* flow_val,
                          const int32_t* last_nodes, const int32_t* n_nbrs, const int32_t* target_idx, const float* mask,
                          int32_t* choice_out, int32_t* acc_out, float* nll_out, void* stream);
/* Two-target comparison (scone_trajectory_model.py:95-108) on the log-probs the last scone_model_eval_host left on the device (same
 * B; its n_nbrs and mask are reused): true_idx / rand_idx [B] = slot of the true target / of the host-drawn random other target
 * (the redraw loop :89-91 consumes the host RNG stream and stays on the host, fed by choice_out).  out[0] = rows with true > random,
 * out[1] = rows with true == random, over mask != 0: the reference's score is (out[0] + 0.5 * out[1]) / sum(mask). */
int scone_model_two_target_host(scone_model* m, int32_t B, const int32_t* true_idx, const int32_t* rand_idx, int32_t* out /* [2] */,
                                void* stream);
/* Read back [grads | nll_sum | count] (host, n_params + 2 floats); synchronises the stream. */
int scone_model_read_grads(scone_model* m, float* out_host, void* stream);
/* The same copy enqueued on the stream without synchronising (out_pinned: page-locked host memory, valid once the caller has
 * synchronised with the stream, e.g. through an event recorded after this call).  Lets a caller enqueue step k + 1 before it looks at
 * the loss of step k: the *_host entry points of the fused pipeline then copy the flow arrays of step k + 1 under the compute kernel
 * of step k (their staging buffers are free once the plan kernels of step k are done).  Capacity overflow is not reported here:
 * scone_model_check_overflow. */
int scone_model_read_grads_async(scone_model* m, float* out_pinned, void* stream);

/* Adam step on the accumulated buffer (upstream JAX `adam`, used at scone_trajectory_model.py:300,310):
 *   g = grads / count + 2 * weight_decay * W ;  m,v update ;  W -= lr * mhat / (sqrt(vhat) + eps)
 * step = 0-based iteration index i. */
int scone_model_adam_step(scone_model* m, int32_t step, float lr, float weight_decay, void* stream);

/* Data-parallel optimizer step over NVLink peer memory (one process per GPU of one node, <= 8 ranks): ONE kernel per rank pushes the
 * rank's [grads | nll_sum | count] buffer into every peer's exchange buffer (CUDA IPC mappings), waits for the peers' pushes, sums
 * the `world` vectors in rank order (bit-identical weights on every rank), writes the sums back into the gradient buffer and applies
 * the Adam update — what `dist.all_reduce(scone_model_grads_dev)` + scone_model_adam_step do in two launches and an NCCL call
 * (SURVEY.md 8e; the update is scone_trajectory_model.py:264-357's).  If any rank's micro-batch overflowed a capacity, no rank updates.
 *   scone_dp_create(rank, world, n_params + 2, &dp); scone_dp_get_handle -> all-gather the scone_dp_handle_bytes()-byte handles ->
 *   scone_dp_open(dp, handles); then scone_model_dp_adam_step every step.  scone_dp_status synchronises the stream and returns 3 if
 *   a peer did not arrive within ~10 s. */
typedef struct scone_dp scone_dp;
int scone_dp_create(int32_t rank, int32_t world, int64_t n_floats, scone_dp** out);
int32_t scone_dp_handle_bytes(void);
int scone_dp_get_handle(scone_dp* dp, void* handle_out);
int scone_dp_open(scone_dp* dp, const void* handles_rank_major);
int scone_model_dp_adam_step(scone_model* m, scone_dp* dp, int32_t step, float lr, float wd, void* stream);
int scone_dp_status(scone_dp* dp, void* stream);
void scone_dp_destroy(scone_dp* dp);
/* Planned sets (pipeline 4).  The plan of a trajectory — receptive cone, live rows, gather programs — depends on the complex, the
 * flows and the last node, not on the weights: a dataset that is revisited every epoch (Scone_GCN.train samples its batches from the
 * same N trajectories for `epochs` epochs, scone_trajectory_model.py:318-322) is planned ONCE and every step runs only the compute
 * kernel on the rows of its batch.  scone_model_plan_* builds and keeps the plan of B trajectories (replacing the previous set);
 * *_planned_* take rows[n] = indices into that set (NULL = its first n trajectories), target_idx / mask / logprobs indexed by batch
 * position.  Same results as the unplanned entry points, bit for bit (the same kernels on the same programs). */
int scone_model_plan_host(scone_model* m, int32_t B, const int32_t* traj_ptr, const int32_t* flow_edge, const float* flow_val,
                          const int32_t* last_nodes, void* stream);
int scone_model_plan_dev(scone_model* m, int32_t B, const int32_t* traj_ptr_dev, const int32_t* flow_edge_dev, const float* flow_val_dev,
                         const int32_t* last_nodes_dev, void* stream);
int scone_model_loss_grad_planned_host(scone_model* m, int32_t n, const int32_t* rows, const int32_t* target_idx, const float* mask,
                                       int32_t zero_first, void* stream);
int scone_model_loss_grad_planned_dev(scone_model* m, int32_t n, const int32_t* rows_dev, const int32_t* target_idx_dev, const float* mask_dev,
                                      int32_t zero_first, void* stream);
int scone_model_forward_planned_host(scone_model* m, int32_t n, const int32_t* rows, float* logprobs_out /* [n][D] */, void* stream);
/* Capacity overflow (pipelines 2 / 3 only; pipeline 4 and the dense pipelines cannot overflow): a micro-batch whose row lists exceed
 * their capacity sets a device flag.  While the flag is set scone_model_adam_step leaves the weights and the Adam state untouched (the
 * gradients are truncated).  The flag is REPORTED (error code 4) and cleared by scone_model_read_grads, scone_model_forward_host,
 * scone_model_accuracy_host and by this call, which synchronises the stream; the *_dev entry points and scone_model_adam_step
 * themselves never synchronise and never report it. */
int scone_model_check_overflow(scone_model* m, void* stream);
/* Weights only (Adam state kept), asynchronous on the caller's stream; weights_host must stay valid until the copy has run. */
int scone_model_set_weights_keep_state(scone_model* m, const float* weights_host, void* stream);
/* Fused pipeline introspection (tests / bench): out[0] = available, [1] bound on |T_0| (hash entries: the cone of any node down to the
 * ring whose flows can reach it), [2] bound on |T_1| (rows a layer can have), [3] hash slots of tier 1, [4] trajectories per arena
 * chunk, [5] rows of the shared-memory row store, [6] / [7] KB of dynamic shared memory of the tier-1 plan / the compute kernel,
 * [8] / [9] hash slots / live rows per layer of tier 0 (tables that hold the cone of ~99 % of the nodes), [10] its KB, [11] two tiers in
 * use, [12] MB of the node table's operator rows (plans come from the table plan kernel; 0 = the hash plan: SCONE_FUSED_TABLE=0 or not enough memory), [13] arena Mwords, [14] K entries of the per-complex cone table,
 * [15] trajectories of the last chunk the first tier handed to the second (synchronises the device). */
int scone_model_fused_info(const scone_model* m, int32_t* out /* [16] */);
/* Plan of trajectory t of the LAST chunk run (synchronises the device): header (16 ints, layout in csrc/fused.cuh) and `words` 32-bit
 * words of the program arena from word offset `off` (either output may be NULL). */
int scone_model_fused_read(scone_model* m, int32_t t, int32_t* hdr_out /* [16] */, uint32_t off, int32_t words, uint32_t* arena_out);
/* (edge, trajectory) rows the fused compute kernel produced since the last call, counted while scone_profile_enable(1): out[0] forward
 * rows (all layers), out[1] backward rows.  bench.py's byte accounting. */
int scone_model_read_rows_done(scone_model* m, int64_t* out /* [2] */);

/* ---------------------------------------------------------------------------------------------
 * SCCONV / "bunch" model (-model bunch): bunch_func (trajectory_experiments.py:173-203) over the seven weighted shift
 * operators of compute_shift_matrices (bunch_model_matrices.py:118-135), given as generic float CSR matrices in the
 * reference order S_00, S_10, S_01, S_11, S_21, S_12, S_22.  Edge rows keep the CALLER's order on this path.
 * hidden[i] = width of hidden layer i; the model has n_hidden + 1 layers of 7 weights (the last maps to 1 channel),
 * weights flat in list order.  Same [grads | nll_sum | count] / Adam contract as scone_model.
 * Operators may have zero rows or columns: a complex without triangles (F = 0) has S_21 E x 0, S_12 0 x E and S_22 0 x 0, and
 * runs like any other (the weights of those operators get a zero gradient).  There is no degree limit on this path.
 * Checked (error code 2, nothing copied or launched): every hidden width >= 1 and every nbrhoods entry in [-1, N) at creation;
 * every last_nodes entry in [0, N) and every target_idx entry in [0, D) in the host entry points (an O(B) loop over host arrays).
 * B = 0: forward writes nothing; loss_grad only clears the buffer when zero_first != 0 and otherwise leaves it as it is.
 * ------------------------------------------------------------------------------------------- */
typedef struct scone_csr scone_csr;
typedef struct scone_bunch scone_bunch;
int scone_csr_create(int32_t rows, int32_t cols, const int32_t* rowptr /* host */, const int32_t* col, const float* val,
                     scone_csr** out);
int scone_csr_destroy(scone_csr* S);
int scone_bunch_create(const scone_csr* const* S7, int32_t n_nodes, int32_t n_edges, int32_t n_tris, int32_t max_degree,
                       const int32_t* nbrhoods /* host [N][D], pad -1 */, int32_t n_hidden, const int32_t* hidden,
                       int32_t micro_batch, scone_bunch** out);
int scone_bunch_destroy(scone_bunch* m);
int64_t scone_bunch_num_params(const scone_bunch* m);
float* scone_bunch_grads_dev(scone_bunch* m);
int scone_bunch_set_weights(scone_bunch* m, const float* weights_host, int32_t reset_adam);
int scone_bunch_get_weights(const scone_bunch* m, float* weights_host);
int scone_bunch_forward_host(scone_bunch* m, int32_t B, const int32_t* traj_ptr, const int32_t* flow_edge, const float* flow_val,
                             const int32_t* last_nodes, float* logprobs_out /* [B][D] */, void* stream);
int scone_bunch_loss_grad_host(scone_bunch* m, int32_t B, const int32_t* traj_ptr, const int32_t* flow_edge, const float* flow_val,
                               const int32_t* last_nodes, const int32_t* target_idx, const float* mask, int32_t zero_first,
                               void* stream);
int scone_bunch_read_grads(scone_bunch* m, float* out_host, void* stream);
int scone_bunch_adam_step(scone_bunch* m, int32_t step, float lr, float weight_decay, void* stream);

/* KERNEL-LEVEL calls: flagged kernels write only the rows that can be non-zero.  With zero-fill ON (default) every output tensor is first
 * bulk-zeroed, so it is a complete dense [E][b][C] array (the dense-streaming contract: each output byte written).
 * With zero-fill OFF unflagged rows are left unwritten and every consumer must honour the flags (all kernels of this
 * library do): traffic then scales with the support of the trajectories instead of E.  Results are identical. */
int scone_set_zero_fill(int32_t on);
int scone_get_zero_fill(void);

/* Dense (no occupancy flags) fused layer kernels: 3 (default, see below) = tcgen05 / TMEM; 1 = slab kernels for widths 16 / 32 (merged-row gather straight
 * into mma.sync fragments, 3xTF32 tensor-core product, fp32-grade accuracy), a warp owning 16 trajectories of one edge;
 * 2 = the same with 8 trajectories of two edges per warp; 0 = the fp32 SIMT tile kernels for every width (bit-identical to
 * the flagged unit kernels; used by the tests that assert that identity). */
int scone_set_dense_kernel(int32_t which);
/* 3 = tcgen05 / TMEM tiles (csrc/scone_umma.cu) for 32 -> 32 layers with b % 16 == 0: the slab gather feeds 128-row tcgen05.mma.kind::tf32
 * tiles (A written to TMEM with tcgen05.st straight from the gather's registers, weights in shared memory, D read back with tcgen05.ld);
 * other shapes fall back to 1.  With 3, scone_layer_backward (no occupancy flags, 32 -> 32, b % 16 == 0) also runs on tcgen05: the gather
 * of G, the row product (AG W^T) * act'(Hin) on mma.sync, and the weight gradient Hin^T AG as tcgen05.mma over K = rows with both
 * operands in shared memory, accumulated in TMEM and folded into fp32 sums every 32 slabs (deterministic; Gprev may alias Hin).
 * scone_umma_status synchronises the stream and returns 3 if a launch reported an mbarrier time-out. */
int scone_umma_status(void* stream);
/* Tile order of the tcgen05 forward kernel: tiles (16 edges x 16 trajectories) are dealt to the CTAs in chunks of `tiles` consecutive
 * tiles, round-robin; 0 = one contiguous range per CTA.  Also read from SCONE_DENSE_CHUNK when the first dense layer runs. */
int scone_set_dense_chunk(int32_t tiles);
int scone_get_dense_kernel(void);

/* Optional per-kernel-family device timing (CUDA events recorded on the launching stream around each launch);
 * off by default.  kind: 0 fused conv layer fwd, 1 fused conv layer bwd (+ its partial reduce), 2 first layer fwd,
 * 3 first layer bwd, 4 readout (+reduce), 5 flows->dense, 6 dense zero-fill of output tensors (on the model's side
 * stream in the model-level calls).  Used by bench.py for the roofline figures. */
int scone_profile_enable(int32_t on);
int scone_profile_reset(void);
int scone_profile_read(int32_t kind, int64_t* launches, double* total_ms);
/* (edge, trajectory) rows the flagged unit kernels of kind 0 (layer fwd) / 1 (layer bwd) produced since the last reset, counted
 * on the device while profiling is on: the support-aware work behind bench.py's byte accounting. */
int scone_profile_read_rows(int32_t kind, int64_t* rows);

/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
int64_t scone_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SCONE_B200_H */
