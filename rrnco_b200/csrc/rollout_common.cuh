// Definitions shared by the fused rollout kernels (rollout_kernel.cu: one CTA per SM, 512 TMEM columns, and the mma.sync
// engine; rollout_lean.cu: two CTAs per SM, 256 TMEM columns each).
#pragma once
#include "common.cuh"

namespace rrnco {

constexpr int kRows = 128;   // rollouts per CTA tile
constexpr int kMaxState = 4;

struct RolloutParams {
  int N, NT, S, n_tiles, n_state;
  int tile_rows;                    // POMO starts per CTA tile (<= kRows); tile t holds starts [t tile_rows, (t + 1) tile_rows)
  int64_t n_inst;
  int multistart, mode, logits_only, use_placeholder, t_cap, forced_T, max_steps;
  uint64_t seed;
  rrnco_decoder_weights_t w;
  rrnco_decoder_cache_t c;
  rrnco_instance_data_t d;
  const int64_t* in_cur;
  const int64_t* in_first;
  const uint8_t* in_mask;
  const float* in_state;
  float* logits_out;
  const int64_t* forced;
  int64_t* actions;
  float* logprob;
  double* ws_len;
  double* ws_lp;
  int32_t* ws_tile_steps;
  int32_t* max_steps_out;
  uint32_t* status;
  const unsigned char* ffn_packed;  // tcgen05 variant: W1 / W2 packed fp16 hi | lo slices (ffn_pack.cuh)
  const float* ffn_bias_scaled;     // lean engine: kAScale * b1 [512] | kAScale * b2 [128] (written by its weight-pack kernel)
  unsigned char* kv_pack;           // tcgen05 variant: kKvSlots per-SM slots of packed fp16 K | V tiles (kKvSlotBytes each)
  int32_t top_k;                    // logit filters (filter_cut, common.cuh): read by the filtered instantiations only
  float top_p;
};
// The lean kernel's beam search (rrnco_beam_rollout): actions / logprob are step-major [t_cap, R] there, with the parent
// rows beside them.  (A derived struct: the parameter layout of every other kernel stays as it is.)
struct BeamParams : RolloutParams {
  int64_t* beam_parent;
};

// Transcendentals of the softmax / bias / clip chain on the SFU (ex2 / lg2 / rcp .approx): absolute error
// <~ 1e-6 on the ranges that occur here, i.e. below the 3xTF32 noise of the logits themselves (~3e-6).
// The .ftz forms skip the denormal pre/post-scaling sequences of __expf / __logf (never needed here: the arguments
// of lg2 are >= 1e-6, and the softmax sums never need a denormal term: see kMaxFixedShift).
__device__ __forceinline__ float ex2a(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2a(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcpa(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fexp(float x) { return ex2a(x * 1.4426950408889634f); }
__device__ __forceinline__ float flog(float x) { return lg2a(x) * 0.6931471805599453f; }
__device__ __forceinline__ float ftanh(float x) { return fmaf(-2.0f, rcpa(ex2a(x * 2.8853900817779268f) + 1.0f), 1.0f); }

// Single-pass selects (rollout_lean.cu, rollout_tiled.cu) sum exp(v - shift) with ex2a, which flushes every term below
// 2^-126 (v - shift < -87.3) to 0.  Clipped values lie in [-clip / T, clip / T], so the bound clip / T can serve as a
// fixed shift (no maximum pass) only while 2 clip / T stays inside that range: up to clip / T = 32 every term is
// >= e^-64, so no term flushes.  Beyond it (T < clip / 32: low temperatures, large clips) a row whose
// values all sit far below the bound would sum to 0 and return +inf log-probs, so the passes keep a running maximum,
// as they do without clipping.  The row's sum against its maximum is >= 1, against which a flushed term is negligible.
constexpr float kMaxFixedShift = 32.f;

// One (shift m, sum s) partial of a row's sum of exp, rescaled to the merged shift mx >= m.  A partial that saw no
// unmasked column (s = 0; m = -inf under a running maximum) adds 0, also when every partial is empty (mx = -inf).
__device__ __forceinline__ float rescaled_sum(float s, float m, float mx) { return s == 0.f ? 0.f : s * fexp(m - mx); }

// Gumbel noise of four consecutive columns (canonical mapping, see the select epilogue).  Deliberately not inlined:
// sixteen inlined copies of Philox + 8 accurate logarithms were 80 KB of code that the greedy path had to jump over.
static __device__ __noinline__ float4 gumbel4(uint4 ctr, uint2 key) {
  const uint4 r = philox4x32(ctr, key);
  return make_float4(-logf(-logf(u01(r.x))), -logf(-logf(u01(r.y))), -logf(-logf(u01(r.z))), -logf(-logf(u01(r.w))));
}


}  // namespace rrnco
