/* rrnco_b200_train.h - C ABI of librrnco_b200_train.so: the training hand-off of the construction rollout.
 *
 * Upstream's training step (rrnco/models/rl.py:99-130) back-propagates log pi(a_t | s_t) of the sampled rollouts through
 * RRNetDecoder (rrnco/models/decoder.py:151-206, 281-326).  With the actions known, every decode step of every rollout is
 * one ROW of a batched problem (rrnco_b200/training.py); the entry points below are the hand-written sm_100a kernels of
 * its heavy parts, forward and backward, in the same fp32-faithful fp16 hi|lo operand split as the rollout kernels
 * (three tcgen05 kind::f16 MMAs per product, fp32 accumulation in TMEM):
 *
 *   rrnco_train_ffn         residual FFN  y = W2 relu(W1 x + b1) + b2 + x      (decoder.py:272-277, 296), forward, and its
 *                           data gradient  dx = W1^T (relu' . W2^T dy) + dy     (the same kernel on the transposed weights,
 *                           the activation replaced by the relu bit mask the forward call wrote)
 *   rrnco_train_xty         C += X^T Y over millions of rows (weight gradients dW1 = dH^T x, dW2^T = H^T dy), with the
 *                           column sums of X and Y (bias gradients) from the same pass
 *   rrnco_train_attention   masked 8-head attention of one query row per (rollout, step) over the instance's keys
 *                           (decoder.py:281-293), forward and backward; _tiled: the same for up to 1024 nodes
 *   rrnco_train_context_query  the context projection as a table gather + rank-k update (context.py:18-70), forward / backward
 *   rrnco_train_inst_gemm / _xty  the pointer scores g . Lk^T and their gradients, one weight tile per instance (decoder.py:298-301);
 *                           rrnco_train_inst_tiled_*: the same with ceil(N / 128) key tiles per instance, up to 1024 nodes
 *   rrnco_train_logits_tail edge bias, log(exp(.) + 1e-6), tanh clip, mask, temperature, log-softmax and the log-prob of
 *                           the given action with its Jacobian, in one pass (decoder.py:183-198, decoding.py:311-399)
 *   rrnco_train_nab_backward the parameter gradients of the encoder's gating neural adaptive bias (attn_freenet.py:242-289)
 *   rrnco_train_nab_dur_backward  the same for the rcvrptw three-way (duration) gate
 *
 * Conventions as in rrnco_b200.h: plain pointers and sizes, device pointers unless noted, return 0 = RRNCO_OK or a negative
 * error, `stream` = cudaStream_t (NULL = default stream), `status` = sticky device word (RRNCO_DEV_NAN_LOGITS when an fp16
 * operand overflowed: the result is then not to be trusted).  All matrices are row-major fp32.
 */
#ifndef RRNCO_B200_TRAIN_H
#define RRNCO_B200_TRAIN_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* bytes of the packed weight stream of rrnco_train_ffn (fp16 hi|lo slices in tensor-pipe order) */
int64_t rrnco_train_ffn_packed_bytes(void);

/* Packs `wa` [512, 128] and `wb` [128, 512] for rrnco_train_ffn: forward (wa, wb) = (W1, W2) of pointer.ffn (decoder.py:272-277);
 * backward-data (wa, wb) = (W2^T, W1^T).  |w| < 255. */
int rrnco_train_ffn_pack(const float* wa, const float* wb, void* packed, uint32_t* status, void* stream);

/* mode 0 (forward):        hidden = relu(x wa^T + b1),  y = hidden wb^T + b2 + x;  `mask` (out, optional) = relu bit mask
 * mode 1 (backward-data):  hidden = (x wa^T) . mask,    y = hidden wb^T + x;        `mask` (in, required); b1 / b2 unused
 *   rows:       number of rows of x / y ([rows, 128]); tiles of 128 rows, any remainder
 *   a_scale:    optional device scalar (power of two): x and hidden are multiplied by it before the fp16 hi|lo split
 *               (gradients are tiny: pick 2^k with max|x| a_scale ~ 512); NULL = 16, the rollout kernels' activation scale
 *   mask:       [rows, 16] uint32: bit (j & 31) of word j >> 5 = hidden unit j active
 *   hidden_out: optional fp32 copy of `hidden`, the X operand of rrnco_train_xty, TILE-BLOCKED AND TRANSPOSED:
 *               [ceil(rows / 128)][512][128], element (row r, unit j) at (r / 128) * 65536 + j * 128 + r % 128 (coalesced for the
 *               thread-per-row epilogue that writes it; rows beyond `rows` are not written)
 *   y:          optional [rows, 128] */
int rrnco_train_ffn(int32_t mode, int64_t rows, const float* x, const void* packed, const float* b1, const float* b2,
                    const float* a_scale, uint32_t* mask, float* hidden_out, float* y, uint32_t* status, void* stream);

/* C[512, 128] += X^T Y,  xsum[512] += column sums of X,  ysum[128] += column sums of Y  (xsum / ysum optional).
 *   x: [rows, 512] row-major (x_tiled == 0) or the tile-blocked layout of rrnco_train_ffn's hidden_out (x_tiled != 0), y: [rows, 128];
 *   sx / sy: optional device scalars (powers of two) applied before the split, NULL = 16.
 * C / xsum / ysum are accumulated with fp32 atomics (the order of the partial sums is not fixed run to run). */
int rrnco_train_xty(int64_t rows, const float* x, int32_t x_tiled, const float* y, const float* sx, const float* sy, float* c,
                    float* xsum, float* ysum, uint32_t* status, void* stream);

/* Masked multi-head attention of decoder.py:281-293 for the batched replay: instance b owns rows [b L, (b + 1) L) of q.
 *   q [n_inst L, 128], k / v [n_inst, n_nodes, 128] (head h = columns 16 h .. 16 h + 15), mask [n_inst L, n_nodes] bytes
 *   (non-zero = feasible; a row with no feasible node is an error upstream and yields zeros here), n_nodes <= 128.
 * forward:   out = softmax(q_h k_h^T / 4 + mask) v_h (+ q when add_residual != 0);  lse [n_inst L, 8] = log2-sum-exp2 of the scaled
 *            masked scores (opaque: saved for the backward pass)
 * backward:  given d_out (gradient of `out`) and the forward call's `out` / `lse` / `add_residual`: dq [n_inst L, 128] (the residual
 *            path d_out included when add_residual != 0), dk / dv [n_inst, n_nodes, 128]
 *            (zeroed, then accumulated with fp32 atomics); n_nodes <= 102 (K, V, dK, dV tiles in shared memory) */
int rrnco_train_attention_fwd(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* q, const float* k, const float* v,
                              const uint8_t* mask, int32_t add_residual, float* out, float* lse, void* stream);
int rrnco_train_attention_bwd(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* q, const float* k, const float* v,
                              const uint8_t* mask, const float* out, int32_t add_residual, const float* lse, const float* d_out,
                              float* dq, float* dk, float* dv, void* stream);

/* The attention above (decoder.py:281-293) for n_nodes <= 1024: the same arguments, math and lse convention, with the keys streamed
 * through shared memory in tiles of 32 (online softmax across the tiles; CUDA cores, fp32 FMAs).  The forward visits the keys in the
 * order and with the arithmetic of rrnco_train_attention_fwd (bitwise equal outputs measured at 101 nodes).
 * backward:  dq from row groups that loop over the key tiles; dk / dv from (instance, key tile, row split) work items whose
 *            partials are added in a fixed order (no float atomics: bitwise reproducible run to run on one device); dk / dv are
 *            written, not accumulated.  workspace: rrnco_train_attention_tiled_workspace_bytes(n_inst, rows_per_inst, n_nodes)
 *            bytes (depends on the current device's SM count), 16-byte aligned: D = dO . attn [rows, 8] and the split partials. */
int64_t rrnco_train_attention_tiled_workspace_bytes(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes);
int rrnco_train_attention_tiled_fwd(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* q, const float* k,
                                    const float* v, const uint8_t* mask, int32_t add_residual, float* out, float* lse, void* stream);
int rrnco_train_attention_tiled_bwd(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* q, const float* k,
                                    const float* v, const uint8_t* mask, const float* out, int32_t add_residual, const float* lse,
                                    const float* d_out, void* workspace, float* dq, float* dk, float* dv, void* stream);

/* Tail of the pointer for the batched replay (decoder.py:183-198 edge bias + log(exp(.) + 1e-6); decoding.py:311-361 tanh clip,
 * mask, temperature; :386-399 log-prob of the given action), one pass:
 *   z [rows, ldz] (in / out; row stride ldz >= n_nodes, <= 1024): raw pointer scores g . Lk^T on entry, J = d logp / d z on return
 *   (backward: dz = g_row J; padding columns are zeroed)
 *   distance / duration [n_inst, n_nodes, n_nodes] (duration NULL except rcvrptw), instance of a row = row / rows_per_inst
 *   current_node / action [rows] int64, mask [rows, n_nodes] bytes, alpha / beta device scalars (decoder.alpha / .beta)
 *   logp [rows] = log pi(action | state);  dlogp_dalpha / dlogp_dbeta [rows] (beta: NULL without duration);  n_nodes <= 1024 */
int rrnco_train_logits_tail(int64_t rows, int64_t rows_per_inst, int32_t n_nodes, int32_t ldz, float* z, const float* distance,
                            const float* duration, const int64_t* current_node, const uint8_t* mask, const int64_t* action,
                            const float* alpha, const float* beta, float inv_sqrt_e, float tanh_clipping, float temperature,
                            float* logp, float* dlogp_dalpha, float* dlogp_dbeta, void* stream);

/* Context query of the pointer (rrnco/models/env_embeddings/context.py:18-70, decoder.py:151-170) for the batched replay:
 *     q[row] = table_a[b, index_a[row]] (+ table_b[b, index_b[row]]) + sum_s state[row, s] state_w[s]        b = row / rows_per_inst
 *   table_a / table_b [n_inst, n_nodes, 128] = row_emb W_t^T (the node part of project_context; table_b / index_b NULL except
 *   atsp: [first node, current node]); state [rows, n_state] (n_state <= 8), state_w [n_state, 128] = the state columns of W.
 * backward: d_table_a / d_table_b / d_state_w are ACCUMULATED (fp32 vector atomics): the caller zeroes them. */
int rrnco_train_context_query_fwd(int64_t rows, int64_t rows_per_inst, int32_t n_nodes, const float* table_a, const int64_t* index_a,
                                  const float* table_b, const int64_t* index_b, const float* state, int32_t n_state,
                                  const float* state_w, float* q, void* stream);
int rrnco_train_context_query_bwd(int64_t rows, int64_t rows_per_inst, int32_t n_nodes, const float* dq, const int64_t* index_a,
                                  const int64_t* index_b, const float* state, int32_t n_state, float* d_table_a, float* d_table_b,
                                  float* d_state_w, void* stream);

/* Pointer scores (decoder.py:298-301) on tcgen05, one zero-padded 128 x 128 weight tile per instance:
 *   rrnco_train_inst_pack   w [n_inst, n_nodes, 128] -> packed (rrnco_train_inst_packed_bytes(n_inst) bytes); transpose == 0 packs
 *                           B[node][e] (z = g w^T), transpose == 1 packs B[e][node] (dg = dz w); |w| < 4094
 *   rrnco_train_inst_gemm   y [n_inst L, 128] = x [n_inst L, 128] B_b   (a_scale: optional device power of two for gradient operands)
 *   rrnco_train_inst_xty    c [n_inst, n_nodes, 128] += x_b^T y_b over the rows of instance b (x, y [n_inst L, 128]; fp32 atomics)
 *   row_scale (optional, [n_inst L]): x is used as diag(row_scale) x -- the upstream gradient of a row times the Jacobian that
 *   rrnco_train_logits_tail left in z, without materialising the product */
int64_t rrnco_train_inst_packed_bytes(int64_t n_inst);
int rrnco_train_inst_pack(int64_t n_inst, int32_t n_nodes, const float* w, int32_t transpose, void* packed, uint32_t* status,
                          void* stream);
int rrnco_train_inst_gemm(int64_t n_inst, int64_t rows_per_inst, const float* x, const void* packed, const float* a_scale,
                          const float* row_scale, float* y, uint32_t* status, void* stream);
int rrnco_train_inst_xty(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* x, const float* y, const float* sx,
                         const float* sy, const float* row_scale, float* c, uint32_t* status, void* stream);

/* Pointer scores (decoder.py:298-301) for n_nodes <= 1024, with n_kt = ceil(n_nodes / 128) zero-padded 128 x 128 weight tiles per
 * instance and score rows ldz = 128 n_kt wide (padding columns are zero); operand scales, row_scale and status as above:
 *   rrnco_train_inst_tiled_pack   w [n_inst, n_nodes, 128] -> packed (rrnco_train_inst_tiled_packed_bytes(n_inst, n_nodes) bytes),
 *                                 transpose as for rrnco_train_inst_pack, per key tile
 *   rrnco_train_inst_tiled_gemm   transpose == 0: y [n_inst L, ldz] = x [n_inst L, 128] B_b    (z = g Lk^T, one column block per tile)
 *                                 transpose == 1: y [n_inst L, 128] = x [n_inst L, ldz] B_b    (dg = dz Lk, the key tiles summed in TMEM)
 *                                 (`packed` packed with the same transpose)
 *   rrnco_train_inst_tiled_xty    c [n_inst, n_nodes, 128] += x_b^T y_b, x [n_inst L, ldz], y [n_inst L, 128], per (instance, key
 *                                 tile) (dLk_b = dz_b^T g_b; fp32 atomics) */
int64_t rrnco_train_inst_tiled_packed_bytes(int64_t n_inst, int32_t n_nodes);
int rrnco_train_inst_tiled_pack(int64_t n_inst, int32_t n_nodes, const float* w, int32_t transpose, void* packed, uint32_t* status,
                                void* stream);
int rrnco_train_inst_tiled_gemm(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, int32_t transpose, const float* x,
                                const void* packed, const float* a_scale, const float* row_scale, float* y, uint32_t* status,
                                void* stream);
int rrnco_train_inst_tiled_xty(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* x, const float* y, const float* sx,
                               const float* sy, const float* row_scale, float* c, uint32_t* status, void* stream);

/* Backward of the encoder's gating neural adaptive bias (DistAngleFusion.forward, rrnco/models/nn/attn_freenet.py:242-289,
 * the two-way gate of ATSP / RCVRP), the forward of which is rrnco_nab_gating (rrnco_b200.h):
 *   coords [n_inst, n_nodes, 2], cost [n_inst, n_nodes, n_nodes] (read as its transpose when transpose_cost != 0), `packed` and
 *   `scale` exactly as the forward call got them; grad_out [n_inst, n_nodes, n_nodes] = dL/d out.
 *   params / grads: the module's 12 tensors in nn.Linear layouts, concatenated (rrnco_train_nab_grad_floats() floats):
 *   dist_emb.0.weight [E,1], dist_emb.0.bias [E], dist_emb.2.weight [E,E], dist_emb.2.bias [E], the same four of angle_emb,
 *   gate.0.weight [1,2E], gate.0.bias [1], out_lin.weight [1,E], out_lin.bias [1]  (E = 128).  grads are written, not accumulated.
 *   workspace: rrnco_train_nab_workspace_bytes(n_inst, n_nodes) bytes (depends on the current device), 8-byte aligned.
 * One pass over the pairs (the forward's per-pair work and a per-segment histogram), nothing of size [n_inst, N, N, E];
 * no atomics: the gradients are bitwise identical run to run on one device.  No gradients for coords / cost.
 * rrnco_train_nab_packed_floats() = the size of `packed` this library expects (= rrnco_nab_packed_floats()). */
int64_t rrnco_train_nab_packed_floats(void);
int64_t rrnco_train_nab_grad_floats(void);
int64_t rrnco_train_nab_workspace_bytes(int64_t n_inst, int32_t n_nodes);
int rrnco_train_nab_backward(int64_t n_inst, int32_t n_nodes, const float* coords, const float* cost, int32_t transpose_cost,
                             const float* packed, const float* params, float scale, const float* grad_out, void* workspace,
                             float* grads, void* stream);

/* Backward of the rcvrptw three-way (duration) gate of the neural adaptive bias (DistAngleFusion.forward with
 * use_duration_matrix), the forward of which is rrnco_nab_dur_gating (rrnco_b200.h):
 *   coords, cost, duration, transpose, `packed` and `scale` exactly as the forward call got them; grad_out [n_inst, N, N].
 *   params / grads: the 19 tensors in the pointer order of rrnco_nab_dur_pack (dist / angle / dur emb.0.weight, emb.0.bias,
 *   emb.2.weight, emb.2.bias, gate.0.weight [E,3E], gate.0.bias, gate.2.weight [3,E], gate.2.bias, gate_temperature,
 *   out_lin.weight, out_lin.bias), concatenated (rrnco_train_nab_dur_grad_floats() floats); grads are written, not accumulated.
 *   workspace: rrnco_train_nab_dur_workspace_bytes(n_inst, n_nodes) bytes (depends on the SM count, not on n_inst), 16-byte
 *   aligned.  status: RRNCO_DEV_NAN_LOGITS is or-ed in when an fp16 operand overflows or a value is not finite.
 * Two tcgen05 passes over the pairs (each recomputes the forward), nothing of size [n_inst, N, N, E]; no float atomics: the
 * gradients are bitwise identical run to run on one device.  No gradients for coords / cost / duration.
 * rrnco_train_nab_dur_packed_bytes() = the size of `packed` this library expects (= rrnco_nab_dur_packed_bytes()). */
int64_t rrnco_train_nab_dur_packed_bytes(void);
int64_t rrnco_train_nab_dur_grad_floats(void);
int64_t rrnco_train_nab_dur_workspace_bytes(int64_t n_inst, int32_t n_nodes);
int rrnco_train_nab_dur_backward(int64_t n_inst, int32_t n_nodes, const float* coords, const float* cost, const float* duration,
                                 int32_t transpose, const void* packed, const float* params, float scale, const float* grad_out,
                                 void* workspace, float* grads, uint32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif
