/*
 * rrnco_b200.h -- C ABI of librrnco_b200.so: the B200-native (sm_100a) construction-rollout hot path of
 * ai4co/real-routing-nco (RRNCO).
 *
 * The reference has NO FFI / plugin / operator registry (SURVEY.md section 8b): its boundary is the Python
 * class API of rl4co-style envs and of RRNetDecoder / RRNetPolicy.  Each entry point below is therefore
 * what a binding for ONE reference method would call; the reference interface it replaces is cited as
 * file:line (paths relative to the upstream repo root).  `rrnco_b200/` (Python) mirrors the reference
 * classes on top of this ABI via ctypes; INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *  - extern "C", C99 types only; every pointer is a DEVICE pointer unless its name starts with `h_`.
 *  - The library never allocates or frees caller-visible memory.  Its only process-wide state are the three
 *    development knobs below (rrnco_set_precision / rrnco_set_ffn_engine / rrnco_set_step_tiling / rrnco_set_start_split: defaults are the
 *    product configuration, set them before the first launch and never concurrently with one) and per-device
 *    launch-configuration caches (shared-memory attributes, SM count), which are idempotent.
 *  - All work is enqueued on `stream` (a cudaStream_t passed as void*); no call synchronises.
 *  - Return value: 0 = RRNCO_OK, negative = error (see rrnco_strerror).  Device-side conditions the
 *    reference raises as Python exceptions (NaN logits, infeasible action) are OR-ed into a caller-owned
 *    sticky `status` word (RRNCO_DEV_*), read back by the host once per rollout.
 *  - "Reference layout": flat rollout index r = s * n_inst + b (repeat-major batchify,
 *    rrnco/models/decoding.py:189, rrnco/models/decoder.py:203), int64 nodes/actions, bool/uint8 masks,
 *    fp32 everything else -- exactly the td tensors of SURVEY.md App. B, passed by data_ptr().
 *  - `data_rows`: instance data (demand, matrices, time windows ...) may be given un-replicated; rollout r
 *    uses row r % data_rows.  The reference's batchified td has data_rows == R.
 */
#ifndef RRNCO_B200_H
#define RRNCO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RRNCO_ABI_VERSION 1

/* status codes */
#define RRNCO_OK 0
#define RRNCO_ERR_BAD_ARG (-1)        /* null pointer / non-positive size / misaligned pointer */
#define RRNCO_ERR_UNSUPPORTED (-2)    /* variant or size not supported by this build (e.g. N > RRNCO_MAX_NODES_FUSED) */
#define RRNCO_ERR_CUDA (-3)           /* a CUDA runtime call failed (launch error) */

/* bits of the device-side sticky status word */
#define RRNCO_DEV_NAN_LOGITS 1u       /* "Logits contain NaNs"           rrnco/models/decoder.py:303-304 */
#define RRNCO_DEV_INFEASIBLE 2u       /* "infeasible action selected"    rrnco/models/decoding.py:278-280 */
#define RRNCO_DEV_NO_FEASIBLE 4u      /* fully-masked row (never happens upstream: depot always feasible) */
#define RRNCO_DEV_TRUNCATED 8u        /* rollout cut at t_cap with unfinished tours ("Exceeded maximum number of steps",
                                         rrnco/models/policy.py:222-226: upstream logs an error and breaks) */
#define RRNCO_DEV_SOFTMAX_RANGE 16u   /* key-tiled fused kernel (N > RRNCO_MAX_NODES_TILE) only: an attention head's scores
                                         exceed the range its fixed softmax shift covers (|q_h| max|k_h| / 4 > 4.85); the
                                         rollout's outputs must be discarded and the per-step entry points used instead */
#define RRNCO_DEV_BAD_PARENT 32u      /* rrnco_beam_backtrack: a parent row outside [0, n_rows) (corrupted beam records) */

#define RRNCO_ENV_ATSP 0
#define RRNCO_ENV_RCVRP 1
#define RRNCO_ENV_RCVRPTW 2

#define RRNCO_DECODE_GREEDY 0         /* argmax, ties -> lowest index     rrnco/models/decoding.py:272-282 */
#define RRNCO_DECODE_SAMPLING 1       /* Gumbel-max sample of softmax     rrnco/models/decoding.py:284-298 */
#define RRNCO_DECODE_EVALUATE 2       /* actions given, log-probs out     rrnco/models/decoding.py:386-399 */

#define RRNCO_EMBED_DIM 128           /* experiment/rrnet.yaml: embed_dim 128, 8 heads */
#define RRNCO_NUM_HEADS 8
#define RRNCO_MAX_NODES_TILE 128      /* one key tile: rrnco_decoder_logits and the single-tile fused kernels */
#define RRNCO_MAX_NODES_FUSED 1024    /* rrnco_rollout: up to 8 key tiles of 128 (key-tiled kernel above RRNCO_MAX_NODES_TILE);
                                         larger N -> RRNCO_ERR_UNSUPPORTED (use the per-step entry points) */

int rrnco_abi_version(void);
const char* rrnco_strerror(int code);

/* Host twin of the device mapping from a 32-bit Philox word to a uniform in the OPEN interval (0, 1) used by the
 * Gumbel-max sampler (rrnco/models/decoding.py:284-298 samples with torch.multinomial; see rrnco_rollout):
 * u = ((x >> 9) + 0.5) / 2^23, exact in fp32, never 0 or 1 -- so -log(-log(u)) is always finite. */
float rrnco_u01(uint32_t x);

/* Precision of the in-kernel contractions of the fused decoder kernels (process-wide, set before use):
 *   3 = error-compensated tensor-core contractions, fp32-faithful (default; the reference's CPU / fp32 path):
 *       three-term fp16 operand split on tcgen05 (engine 1) / 3xTF32 on mma.sync (engine 0)
 *   1 = one reduced-precision pass (analogue of the reference's `torch.autocast("cuda")` inference path, test.py:182-185)
 * The key-tiled kernel (n_nodes > RRNCO_MAX_NODES_TILE) is built fp32-faithful only and ignores the setting. */
int rrnco_set_precision(int32_t passes);

/* FFN engine of the fused rollout kernel (process-wide, set before use):
 *   1 = tcgen05.mma kind::f16 for attention, FFN and logits, TMEM accumulators, TMA-streamed operands (default)
 *   0 = mma.sync tensor-core path (also what rrnco_decoder_logits uses) */
int rrnco_set_ffn_engine(int32_t engine);

/* Key sharing of the any-N per-step decoder (rrnco_decoder_logits_large; process-wide, set before use):
 *   1 = one CTA per (instance, group of starts): key / value / logit-key rows staged once per CTA in shared memory; the
 *       pointer logits (starts x keys contraction) on mma.sync 3xTF32 tensor-core tiles (default)
 *   2 = same tiling, logits as FFMA dot products in the accumulation order of mode 0
 *   0 = one warp per rollout streaming its own copy of the rows from L2 (first version; kept as the cross-check) */
int rrnco_set_step_tiling(int32_t mode);

/* ------------------------------------------------------------------------------------------------
 * env.reset: per-instance min-max normalisation of the distance matrix
 *   replaces RCVRPEnv._reset rrnco/envs/rcvrp/env.py:138-145 (same lines in atsp/env.py:113-120,
 *   rmtvrp/env.py:271-280):  out = (d - min) / (max - min + 1e-6), min/max over the whole [N,N] matrix.
 * ---------------------------------------------------------------------------------------------- */
int rrnco_minmax_normalize(int64_t n_mat, int32_t n_nodes, const float* dist_in, float* dist_out,
                           float* min_out, float* max_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Instance sub-sampling gather: out[b,i,j] = (float) M[idx[b,i], idx[b,j]]
 *   replaces Real_World_Sampler.sample rrnco/envs/rcvrp/sampler.py:84-90 (+ the fp32 cast of
 *   rrnco/envs/rcvrp/generator_lazy.py:300).  M is the float64 city matrix [L,L]
 *   (data_generation/utilities/create_dataset.py:169-174); idx is int32 [batch, n].
 *   normalize == 1 fuses the min-max normalisation of env.reset, (d - min) / (max - min + 1e-6);
 *   normalize == 2 fuses the generators' duration law, (d - min) / (max - min) with a zero range replaced by 1
 *   (rrnco/envs/rmtvrp/generator_lazy.py:365-369); min_out / max_out are filled in both cases and may be NULL
 *   when normalize == 0.
 * ---------------------------------------------------------------------------------------------- */
int rrnco_gather_submatrix(const double* city_matrix, int32_t city_len, const int32_t* idx, int64_t batch,
                           int32_t n, float* out, int32_t normalize, float* min_out, float* max_out,
                           void* stream);

/* Same gather from an fp32 copy of the city matrix (the cast of generator_lazy.py:300 commutes with the gather, so the
 * results are bit-identical): 8 instead of 4 elements per 32-byte L2 sector.  rrnco_city_matrix_to_f32 makes the copy,
 * once per city (n_elems = L*L; also usable for `points`). */
int rrnco_gather_submatrix_f32(const float* city_matrix_f32, int32_t city_len, const int32_t* idx, int64_t batch,
                               int32_t n, float* out, int32_t normalize, float* min_out, float* max_out,
                               void* stream);
int rrnco_city_matrix_to_f32(const double* city_matrix, int64_t n_elems, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * ATSPEnv._step  rrnco/envs/atsp/env.py:79-105   (reference layout, R rollouts)
 *   mask_out = mask_in with action cleared; done = no node left; first_node latched when *step_i == 0
 *   (step_i: DEVICE pointer to td["i"]; upstream reads it with a blocking .item(), atsp/env.py:82).
 *   In/out pointers may alias.
 * ---------------------------------------------------------------------------------------------- */
int rrnco_atsp_step(int64_t R, int32_t n_nodes, const int64_t* action, const int64_t* step_i,
                    const uint8_t* mask_in, const int64_t* first_in, uint8_t* mask_out, int64_t* first_out,
                    int64_t* current_out, uint8_t* done_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * RCVRPEnv._step + get_action_mask  rrnco/envs/rcvrp/env.py:90-122, 183-195
 *   demand [data_rows, N-1] (customers only, already / capacity), capacity [data_rows_cap] broadcast by
 *   r % cap_rows.  If action == NULL only the mask is recomputed from (visited_in, used_in, current_in)
 *   (= the static get_action_mask).  visited is uint8 [R,N], mask bool [R,N].
 * ---------------------------------------------------------------------------------------------- */
int rrnco_rcvrp_step(int64_t R, int32_t n_nodes, int64_t data_rows, const int64_t* action,
                     const float* demand, const float* capacity, int64_t cap_rows, const float* used_in,
                     const uint8_t* visited_in, const int64_t* current_in, float* used_out,
                     uint8_t* visited_out, int64_t* current_out, uint8_t* done_out, uint8_t* mask_out,
                     void* stream);

/* ------------------------------------------------------------------------------------------------
 * Residual FFN of RRNet_PointerAttention  rrnco/models/decoder.py:272-277,296  (rl4co MLP E -> 4E -> E, ReLU)
 *   g_out = W2 relu(W1 g_in + b1) + b2 + g_in     g: [n_rows, E] fp32
 *   tcgen05 (kind::f16, three-term fp16 operand split, TMEM accumulators) form of the FFN phase of the fused kernel.
 *   workspace >= rrnco_pointer_ffn_workspace_bytes() bytes (holds the hi/lo split of W1, W2).
 * ---------------------------------------------------------------------------------------------- */
int64_t rrnco_pointer_ffn_workspace_bytes(void);
int rrnco_pointer_ffn(int64_t n_rows, const float* g_in, const float* w1, const float* b1, const float* w2,
                      const float* b2, float* g_out, void* workspace, void* stream);

/* Instance data shared by the RCVRPTW step and the fused kernels (row = index % data_rows). Unused members NULL. */
typedef struct rrnco_instance_data {
  int64_t data_rows;
  const float* distance;        /* [rows,N,N] normalised (env.reset output) */
  const float* duration;        /* [rows,N,N] rcvrptw */
  const float* demand;          /* rcvrp: [rows,N-1]; rcvrptw: demand_linehaul [rows,N] depot-padded */
  const float* demand_backhaul; /* rcvrptw [rows,N] */
  const float* time_windows;    /* rcvrptw [rows,N,2] */
  const float* service_time;    /* rcvrptw [rows,N] */
  const float* vehicle_capacity;/* [rows] */
  const float* distance_limit;  /* rcvrptw [rows] */
  const uint8_t* open_route;    /* rcvrptw [rows] */
  const float* backhaul_class;  /* rcvrptw [rows] */
  const float* min_distance;    /* [rows] for the de-normalised reward (may be NULL) */
  const float* max_distance;    /* [rows] */
} rrnco_instance_data_t;

/* ------------------------------------------------------------------------------------------------
 * RMTVRPEnv._step + get_action_mask  rrnco/envs/rmtvrp/env.py:155-215, 343-428  (all O/B/L/MB/TW branches)
 *   data->demand is demand_linehaul [rows,N]; every rcvrptw member of `data` must be set.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rrnco_rmtvrp_state {
  int64_t* current_node;        /* [R] */
  float* current_time;          /* [R] */
  float* current_route_length;  /* [R] */
  float* used_capacity_linehaul;/* [R] */
  float* used_capacity_backhaul;/* [R] */
  uint8_t* visited;             /* [R,N] bool */
} rrnco_rmtvrp_state_t;

/* action == NULL -> mask only (static get_action_mask on state_in). state_in / state_out may alias. */
int rrnco_rmtvrp_step(int64_t R, int32_t n_nodes, const rrnco_instance_data_t* data, const int64_t* action,
                      const rrnco_rmtvrp_state_t* state_in, const rrnco_rmtvrp_state_t* state_out,
                      uint8_t* done_out, uint8_t* mask_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * env._get_reward: negative tour length over the (normalised) matrix + de-normalised "real" value
 *   ATSP    rrnco/envs/atsp/env.py:192-211     closed tour a_0..a_{T-1}->a_0              (prepend_depot 0)
 *   RCVRP   rrnco/envs/rcvrp/env.py:197-219    depot, a_0..a_{T-1}, back to depot         (prepend_depot 1)
 *   RCVRPTW rrnco/envs/rmtvrp/env.py:430-455   same, legs INTO the depot cost 0 if open_route[row]
 *   real = norm * (max - min + 1e-6) + min   (min_d/max_d [data_rows]; pass NULL to skip `real_out`).
 * ---------------------------------------------------------------------------------------------- */
int rrnco_tour_reward(int64_t R, int32_t T, int32_t n_nodes, int64_t data_rows, const int64_t* actions,
                      const float* distance, int32_t prepend_depot, const uint8_t* open_route,
                      const float* min_d, const float* max_d, float* norm_out, float* real_out,
                      void* stream);

/* ------------------------------------------------------------------------------------------------
 * Decoder weights + per-batch cache (RRNetDecoder.state_dict(), SURVEY.md App. C)
 * ---------------------------------------------------------------------------------------------- */
typedef struct rrnco_decoder_weights {
  const float* ffn_w1;   /* pointer.ffn.lins.0.weight [4E, E]   rrnco/models/decoder.py:272-277 */
  const float* ffn_b1;   /* pointer.ffn.lins.0.bias   [4E] */
  const float* ffn_w2;   /* pointer.ffn.lins.1.weight [E, 4E] */
  const float* ffn_b2;   /* pointer.ffn.lins.1.bias   [E] */
  const float* ctx_state_w; /* [n_state, E]: transposed state columns of context_embedding.project_context.weight
                               (rcvrp: 1 row; rcvrptw: 4 rows; atsp: NULL)  rrnco/models/env_embeddings/context.py:27-31 */
  const float* ctx_placeholder_q; /* [E] = W_ctx . W_placeholder (atsp, only used when multistart == 0), else NULL */
  float alpha;           /* distance-bias scale  rrnco/models/decoder.py:121,189-193 */
  float beta;            /* duration-bias scale (rcvrptw) rrnco/models/decoder.py:97-98 */
  float tanh_clipping;   /* 10.0  rrnco/models/policy.py:83 */
  float temperature;     /* 1.0 */
} rrnco_decoder_weights_t;

typedef struct rrnco_decoder_cache {
  /* all [n_inst, N, E] fp32, contiguous; K/V/Lk = project_node_embeddings(col_emb).chunk(3)
     rrnco/models/decoder.py:214-232 */
  const float* glimpse_key;
  const float* glimpse_val;
  const float* logit_key;
  const float* ctx_node_proj;   /* row_emb . W_ctx[:, :E]^T  (atsp: first-node half W_ctx[:, :E]) */
  const float* ctx_node_proj2;  /* atsp only: row_emb . W_ctx[:, E:2E]^T (current-node half), else NULL */
} rrnco_decoder_cache_t;

/* Fills K/V/Lk/ctx projections from the encoder output with the library's own GEMM kernel:
 *   RRNetDecoder._precompute_cache rrnco/models/decoder.py:214-232 + the node half of EnvContext.forward
 *   rrnco/models/env_embeddings/context.py:27-31.  w_node [3E,E], w_ctx [E, ctx_in] as in state_dict. */
int rrnco_precompute_cache(int32_t env, int64_t n_inst, int32_t n_nodes, const float* row_emb,
                           const float* col_emb, const float* w_node, const float* w_ctx, int32_t ctx_in,
                           float* glimpse_key, float* glimpse_val, float* logit_key, float* ctx_node_proj,
                           float* ctx_node_proj2, void* stream);


/* ------------------------------------------------------------------------------------------------
 * RRNetDecoder.forward  rrnco/models/decoder.py:151-206  (one decode step, logits only)
 *   state in reference layout: current [R] int64, first [R] int64 (atsp, else NULL), mask bool [R,N],
 *   ctx_state fp32 [R, n_state] (rcvrp: capacity-used; rcvrptw: avail_load, time, open, remaining_dist;
 *   atsp: NULL).  logits_out fp32 [R,N] = log(exp(pointer_logits - bias) + 1e-6), rows in (s b) order.
 *   use_placeholder != 0: atsp step 0 without multistart (TSPContext placeholder query).
 * ---------------------------------------------------------------------------------------------- */
int rrnco_decoder_logits(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts,
                         const rrnco_decoder_weights_t* w, const rrnco_decoder_cache_t* cache,
                         const rrnco_instance_data_t* data, const int64_t* current, const int64_t* first,
                         const uint8_t* mask, const float* ctx_state, int32_t use_placeholder,
                         float* logits_out, uint32_t* status, void* stream);

/* Key-streaming variant of rrnco_decoder_logits for ANY number of nodes (e.g. the n=1000 generalisation
 * configs): online-softmax attention over streamed keys, the tcgen05 pointer FFN, streamed logit keys.
 * Same arguments plus a workspace of >= rrnco_decoder_logits_large_workspace_bytes(n_inst * n_starts) bytes. */
int64_t rrnco_decoder_logits_large_workspace_bytes(int64_t n_rollouts);
int rrnco_decoder_logits_large(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts,
                               const rrnco_decoder_weights_t* w, const rrnco_decoder_cache_t* cache,
                               const rrnco_instance_data_t* data, const int64_t* current, const int64_t* first,
                               const uint8_t* mask, const float* ctx_state, int32_t use_placeholder,
                               float* logits_out, uint32_t* status, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------
 * DecodingStrategy.step  rrnco/models/decoding.py:219-298 with process_logits :311-361
 *   logits fp32 [R,N] (decoder output), mask bool [R,N]  ->  action int64 [R], log-prob of the action fp32 [R]
 *   greedy: argmax of the log-softmax, lowest index on ties; sampling: Gumbel-max with noise
 *   Philox(seed; (r, step, n >> 2))[n & 3]; evaluate: forced_action [R].
 *   rrnco_select_action = rrnco_select_action_filtered with top_k = 0, top_p = 0 (no filter).
 *
 * Logit filters (rrnco_select_action_filtered, rrnco_rollout_filtered), applied after tanh clipping, the mask and the
 * temperature, before the log-softmax, for every decode mode:
 *   top_k > 0      keep the entries >= the k-th largest value (ties kept; masked entries take part, so a row with fewer
 *                  than k feasible nodes is unchanged).  top_k = 0: off.
 *   0 < top_p < 1  then keep entry j iff the softmax mass of the entries strictly greater than it is < top_p (a tie group
 *                  is kept or dropped whole; the top entry is always kept).  top_p = 0 or 1: off.
 *   The log-probs are renormalised over the kept entries; a forced (evaluate) action that is feasible but filtered out
 *   gets log-prob -inf and is not reported as infeasible.  Sampling draws the same Gumbel noise as without a filter and
 *   skips the dropped entries.  top_k < 0 or top_p outside [0, 1] (or NaN): RRNCO_ERR_BAD_ARG, nothing launched.
 * ---------------------------------------------------------------------------------------------- */
int rrnco_select_action(int64_t n_rollouts, int32_t n_nodes, const float* logits, const uint8_t* mask,
                        int32_t decode_mode, float tanh_clipping, float temperature, uint64_t seed, int32_t step,
                        const int64_t* forced_action, int64_t* action_out, float* logprob_out, uint32_t* status,
                        void* stream);
int rrnco_select_action_filtered(int64_t n_rollouts, int32_t n_nodes, const float* logits, const uint8_t* mask,
                                 int32_t decode_mode, float tanh_clipping, float temperature, uint64_t seed, int32_t step,
                                 const int64_t* forced_action, int64_t* action_out, float* logprob_out, uint32_t* status,
                                 int32_t top_k, float top_p, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Beam search (rl4co BeamSearch._make_beam_step / _backtrack, decoding.py:402-542), one decode step per call.
 *   Rows r = w * n_inst + b (beam w of instance b, the (w b) order of batchify).  Beam w's log-probs lp[r, n] are the
 *   per-row math of rrnco_select_action (tanh clipping, mask, temperature, log-softmax); the candidates of instance b are
 *   score_in[r] + lp[r, n] with flat index w * n_nodes + n.  The beam_width largest, ranked by (value descending, flat
 *   index ascending: lower index first among equal values), become the new beams: rank w' writes row w' * n_inst + b with
 *   action_out = n, parent_out = the parent's ROW (w * n_inst + b), logprob_out = lp[parent, n], score_out = the candidate
 *   value (fp32, score + lp).  When fewer than beam_width candidates are finite, ranks from #finite upward copy rank 0
 *   (no finite candidate at all sets RRNCO_DEV_NO_FEASIBLE).  score_out may alias score_in.
 *   beam_width < 2: RRNCO_ERR_BAD_ARG; > RRNCO_MAX_BEAM_WIDTH: RRNCO_ERR_UNSUPPORTED; both before any CUDA call.
 *
 * rrnco_beam_backtrack: actions / parents int64 and logprobs fp32, step-major [n_steps, n_rows] (row t = what step t
 *   wrote; parents of step 0 are never read) -> actions_out int64 [n_rows, n_steps], logprob_out fp32 [n_rows, n_steps]
 *   (may be NULL) aligned along the path of final beam r, loglik_out fp32 [n_rows] = their fp64 sum.  A parent row
 *   outside [0, n_rows) sets RRNCO_DEV_BAD_PARENT in `status`; that row's earlier steps come out as action 0 with
 *   log-prob NaN and its log-likelihood is NaN.
 * ---------------------------------------------------------------------------------------------- */
#define RRNCO_MAX_BEAM_WIDTH 1024
int rrnco_beam_select(int64_t n_inst, int32_t beam_width, int32_t n_nodes, const float* logits, const uint8_t* mask,
                      const float* score_in, float tanh_clipping, float temperature, int64_t* action_out, int64_t* parent_out,
                      float* logprob_out, float* score_out, uint32_t* status, void* stream);
int rrnco_beam_backtrack(int64_t n_rows, int32_t n_steps, const int64_t* actions, const int64_t* parents,
                         const float* logprobs, int64_t* actions_out, float* logprob_out, float* loglik_out,
                         uint32_t* status, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused construction rollout = RRNetPolicy.forward decode loop  rrnco/models/policy.py:203-243
 *   (multistart pre-hook decoding.py:157-205, decoder.py:151-206, process_logits decoding.py:311-361,
 *    greedy / sampling / evaluate decoding.py:272-298,386-399, env._step, _get_reward, get_log_likelihood)
 *   One launch decodes all R = n_inst * n_starts rollouts to completion without host round-trips.
 *
 *   multistart != 0: rollout (b, s) is forced to start node (s % num_loc) + has_depot
 *                    (rl4co select_start_nodes; rrnco/envs/rmtvrp/selectstartnodes.py:42-50); that action is
 *                    written as actions[:,0] with log-prob 0.   multistart == 0 requires n_starts == 1.
 *   forced_actions  (mode EVALUATE): int64 [R, forced_T] in reference layout, the decisions AFTER the forced
 *                    start (policy.py:214-218 indexes actions[..., step]).
 *   actions_out     int64 [R, t_cap]; unused tail filled with 0 (= depot, what upstream emits for finished
 *                    rollouts).  t_cap must be >= the longest rollout; *max_steps_out (device int32) receives
 *                    the longest length = the T upstream would have produced.
 *   logprob_out     fp32 [R, t_cap] per-step log-probs (may be NULL); loglik_out fp32 [R] their sum.
 *   norm_reward_out fp32 [R] = -(tour length on the normalised matrix); real_reward_out de-normalised
 *                    (NULL if data->min_distance is NULL).  Padding legs 0->0 are accounted like upstream.
 *   workspace       >= rrnco_rollout_workspace_bytes(...) bytes, 16-byte aligned: fp64 accumulators (16 B per rollout),
 *                    tile step counts, the packed FFN weights (512 KB) and 256 per-SM slots of 192 KB holding the fp16
 *                    tiles of the resident instance's keys / values / logit keys.  Scratch only: nothing in it
 *                    survives the call, but two concurrent rollouts (different streams) need two workspaces.
 * ---------------------------------------------------------------------------------------------- */
int64_t rrnco_rollout_workspace_bytes(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts);

/* POMO starts per CTA tile of rrnco_rollout for this shape on the current device: 128, unless rrnco_set_start_split(1)
 * (process-wide development knob, default 0; 2 = default tiling but without the key-tiled kernel's CTA pairs, i.e. one
 * CTA per tile even when that leaves most SMs idle) lets the key-tiled kernel (n_nodes > RRNCO_MAX_NODES_TILE, one CTA per SM)
 * split the starts of an instance over several CTAs, in whole warps of 32 rows, when the instances alone would not fill
 * the SMs (config C4: 64 instances x 100 starts -> 2 tiles of 64 / 36; measured gain 5 %: the passes are bound per SM
 * sub-partition, so it is off).  The workspace holds one int32 step count per (instance, tile):
 * n_inst * ceil(n_starts / tile_rows) of them, instance-major, at byte offset 16 * n_inst * n_starts. */
int32_t rrnco_rollout_tile_rows(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts);
int rrnco_set_start_split(int32_t mode);

int rrnco_rollout(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts, int32_t multistart,
                  int32_t decode_mode, uint64_t seed, const rrnco_decoder_weights_t* w,
                  const rrnco_decoder_cache_t* cache, const rrnco_instance_data_t* data,
                  const int64_t* forced_actions, int32_t forced_T, int32_t t_cap, int64_t* actions_out,
                  float* logprob_out, float* loglik_out, float* norm_reward_out, float* real_reward_out,
                  int32_t* max_steps_out, uint32_t* status, void* workspace, void* stream);
/* rrnco_rollout with the logit filters described at rrnco_select_action_filtered (rrnco_rollout = top_k 0, top_p 0).  A
 * filter runs on the single-tile tcgen05 engines (n_nodes <= RRNCO_MAX_NODES_TILE, engines 1 and 2); the key-tiled
 * kernel (n_nodes > RRNCO_MAX_NODES_TILE) and the mma.sync engine 0 return RRNCO_ERR_UNSUPPORTED for an active filter:
 * decode such calls with the per-step entry points (rrnco_decoder_logits_large + rrnco_select_action_filtered). */
int rrnco_rollout_filtered(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts, int32_t multistart,
                           int32_t decode_mode, uint64_t seed, const rrnco_decoder_weights_t* w,
                           const rrnco_decoder_cache_t* cache, const rrnco_instance_data_t* data,
                           const int64_t* forced_actions, int32_t forced_T, int32_t t_cap, int64_t* actions_out,
                           float* logprob_out, float* loglik_out, float* norm_reward_out, float* real_reward_out,
                           int32_t* max_steps_out, uint32_t* status, void* workspace, int32_t top_k, float top_p,
                           void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused beam search: the whole BeamSearch decode (rl4co decoding.py:402-542) in one launch of the lean rollout kernel,
 * one CTA per instance whose beam_width rows are the beams.  Same semantics as a loop of rrnco_beam_select steps:
 *   Rows r = w * n_inst + b.  The beams start at select_start_nodes (start w % num_loc + has_depot, log-prob 0, score 0).
 *   Each step computes every beam row's log-probs as rrnco_rollout does (tanh clipping, mask, temperature, log-softmax),
 *   ranks the candidates score + lp (fp32) of an instance by (value descending, flat index w * n_nodes + n ascending),
 *   keeps the beam_width largest (ranks from #finite upward copy rank 0; none finite sets RRNCO_DEV_NO_FEASIBLE), moves
 *   each new beam's rollout state to its parent row and steps the env with its action.  Scores: score_t = score_{t-1} + lp_t.
 *   An instance whose beams are all done keeps them: parent = the row itself, action 0, log-prob 0, as a further
 *   rrnco_beam_select step on its depot-only masks would.
 *   step_actions / step_parents int64, step_logprobs fp32: step-major [t_cap, R], the inputs of rrnco_beam_backtrack
 *   (rows 0 .. *n_steps_out - 1 are written; step 0 holds the starts).  *n_steps_out (device int32) = the number of
 *   steps of the longest instance, the T of the per-step loop.  t_cap: 2 * n_nodes + 3 for the VRPs, n_nodes for ATSP
 *   (the per-step loop's bound); an instance still running at t_cap sets RRNCO_DEV_TRUNCATED.
 *   workspace: >= rrnco_beam_rollout_workspace_bytes(...) bytes, 16-byte aligned, scratch only.
 *   Built for the default engine and precision only (fp32-faithful operands: rrnco_set_ffn_engine(2),
 *   rrnco_set_precision(3)).  beam_width < 2: RRNCO_ERR_BAD_ARG; beam_width > RRNCO_MAX_BEAM_WIDTH_FUSED,
 *   n_nodes > 112, another engine or precision: RRNCO_ERR_UNSUPPORTED; all before any CUDA call (the per-step entry
 *   points serve those calls).
 * rrnco_beam_rollout_workspace_bytes: the workspace size, or 0 when rrnco_beam_rollout does not serve the call (the
 *   same width, size, engine and precision rule): callers route on it.
 * ---------------------------------------------------------------------------------------------- */
#define RRNCO_MAX_BEAM_WIDTH_FUSED 128
int64_t rrnco_beam_rollout_workspace_bytes(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t beam_width);
int rrnco_beam_rollout(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t beam_width, const rrnco_decoder_weights_t* w,
                       const rrnco_decoder_cache_t* cache, const rrnco_instance_data_t* data, int32_t t_cap,
                       int64_t* step_actions, int64_t* step_parents, float* step_logprobs, int32_t* n_steps_out,
                       uint32_t* status, void* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Encoder hot spot (SURVEY.md 8(f) rank 4): gating neural adaptive bias of an attention-free block, variant without the
 * duration channel -- DistAngleFusion.forward, rrnco/models/nn/attn_freenet.py:242-289 (ATSP / RCVRP encoders,
 * rrnco/models/encoder.py:63-66), times the block's `alpha` (attn_freenet.py:424-430).
 *   adapt_bias[b,i,j] = scale * out_lin( g * dist_emb(c) + (1 - g) * angle_emb(theta) ),  g = sigmoid(gate([dist_emb, angle_emb]))
 *   c = cost[b,i,j] (cost[b,j,i] when transpose_cost != 0: the col-encoding block sees the transposed matrix with the
 *   same coords, attn_freenet.py:480-486), theta = atan2(y_i - y_j, x_i - x_j).
 * Upstream materialises the two [B,N,N,E] embeddings; here the module is collapsed once per call into four E-vectors
 * (rrnco_nab_pack, fp64 accumulation: the second Linear of each MLP, the gate and out_lin are linear in the hidden
 * vectors) and evaluated per pair on the CUDA cores: 4 B read + 4 B written per pair, nothing materialised.
 *   rrnco_nab_pack: the module's parameters in nn.Linear layout (dist_emb.0 / .2, angle_emb.0 / .2: weight [E,1] / [E,E],
 *                   bias [E]; gate.0: weight [1,2E], bias [1]; out_lin: weight [1,E], bias [1]) -> packed fp32
 *                   [rrnco_nab_packed_floats()], 16-byte aligned.
 *   rrnco_nab_gating: coords fp32 [B,N,2] (8-byte aligned), cost fp32 [B,N,N], out fp32 [B,N,N].
 *                   variant 0 (default): each collapsed function is piecewise linear in its scalar with <= E breakpoints;
 *                   the pack holds them sorted with per-segment slope / intercept (fp64 sums), the kernel does two
 *                   8-probe segment searches + 4 FMAs per pair.  variant 1: the sum over the E hidden units (cross-check).
 * Forward only (test.py / validation path). ---------------------------------------------------- */
int64_t rrnco_nab_packed_floats(void);
int rrnco_nab_pack(const float* dist_w1, const float* dist_b1, const float* dist_w2, const float* dist_b2,
                   const float* angle_w1, const float* angle_b1, const float* angle_w2, const float* angle_b2,
                   const float* gate_w, const float* gate_b, const float* out_w, const float* out_b, float* packed,
                   void* stream);
int rrnco_nab_gating(int64_t n_inst, int32_t n_nodes, const float* coords, const float* cost, int32_t transpose_cost,
                     const float* packed, float scale, int32_t variant, float* out, void* stream);

/* Duration-channel variant (rcvrptw encoder, use_duration_matrix = True): three MLPs (cost, angle, duration) and the gate
 * Linear(3E,E) - SiLU - Linear(E,3) - softmax(. / exp(temperature)); attn_freenet.py:226-238,268-281.  The layers that are
 * linear in the hidden vectors are collapsed at pack time (fp64); the remaining [pairs x 3E] . [3E x E] contraction runs on
 * tcgen05 (three-term fp16 split, fp32-faithful) over tiles of 128 pairs, the A operand generated on the fly from the
 * pair's scalars, the weight slices streamed by TMA; SiLU / E -> 3 / softmax / blend in the epilogue.
 *   d_params: DEVICE array of 19 device pointers, nn.Linear layouts: dist_emb.0.weight, .0.bias, .2.weight, .2.bias, the same
 *             four of angle_emb and of dur_emb, gate.0.weight [E,3E], gate.0.bias, gate.2.weight [3,E], gate.2.bias,
 *             gate_temperature [1], out_lin.weight [1,E], out_lin.bias [1]
 *   packed:   rrnco_nab_dur_packed_bytes() bytes, 16-byte aligned; status: sticky device word (RRNCO_DEV_NAN_LOGITS on an
 *             fp16 operand overflow: |weights| >= 255 or hidden activations >= 4094)
 *   transpose != 0: cost AND duration are read transposed (col-encoding block, attn_freenet.py:476-486). */
int64_t rrnco_nab_dur_packed_bytes(void);
int rrnco_nab_dur_pack(const float* const* d_params, void* packed, uint32_t* status, void* stream);
int rrnco_nab_dur_gating(int64_t n_inst, int32_t n_nodes, const float* coords, const float* cost, const float* duration,
                         int32_t transpose, const void* packed, float scale, float* out, uint32_t* status, void* stream);

/* The O(N^2) part of one attention-free block fused (attn_freenet.py:424-432 + AFTFull.forward :309-327, n_nodes <= 128):
 *   out[b,i,:] = sigmoid(q[b,i,:]) * (sum_j a_ij E2[j,:]) / (sum_j a_ij E1[j,:]),   a_ij = exp(softmax_j(scale * adapt_bias[b,i,j])),
 *   E1 = exp(softmax over the tokens of k[b]), E2 = E1 * v[b]   -- i.e. AFTFull without its four Linear layers (q / k / v are
 *   to_q(x) / to_k(y) / to_v(y), the caller applies `project`).  adapt_bias comes from the segment tables of rrnco_nab_pack
 *   and never reaches memory; E1 / E2 of the instance stay in shared memory.  q, k, v, out fp32 [B,N,128] (16-byte aligned).
 *   packed == NULL: `cost` holds adapt_bias [B,N,N] itself (e.g. the output of rrnco_nab_dur_gating), coords is unused. */
int rrnco_aft_nab(int64_t n_inst, int32_t n_nodes, const float* q, const float* k, const float* v, const float* coords,
                  const float* cost, int32_t transpose_cost, const float* packed, float scale, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RRNCO_B200_H */
