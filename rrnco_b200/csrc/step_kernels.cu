// Per-step decoder kernels for ANY number of nodes (the key-streaming variant used when N exceeds the
// 128-key tile of the fused kernel, e.g. BASELINE config "ATSP n=1000 generalisation rollout"):
//   rrnco_decoder_logits_large  = RRNetDecoder.forward            rrnco/models/decoder.py:151-206
//       attention_stream_kernel : context query + 8-head masked attention, online softmax over streamed keys
//       pointer FFN             : the tcgen05 kernel of ffn_tc_kernel.cu (rows = rollouts)
//       logits_stream_kernel    : g'.Lk^T / sqrt(E), scale-adaptive bias, log(exp(.) + 1e-6)
//   rrnco_select_action         = DecodingStrategy.step           rrnco/models/decoding.py:219-298,311-361
// One warp per rollout; keys / values / logit keys are streamed from L2 with coalesced 128-bit loads (a key row is
// 512 contiguous bytes = one float4 per lane); infeasible keys are skipped.  Instance data is never replicated:
// rollout r = s * n_inst + b reads the cache / matrices of instance b.
#include "common.cuh"
#include "ffn_pack.cuh"

namespace rrnco {

constexpr int kStepWarps = 4;

__device__ __forceinline__ float sfexp(float x) { return __expf(x); }

struct StepArgs {
  int env, N, n_state, use_placeholder;
  int64_t R, n_inst, data_rows;
  const float *K, *V, *Lk, *P1, *P2;           // [n_inst, N, 128]
  const float *wstate, *placeholder;            // [n_state, 128], [128]
  const float *dist, *dur;                      // [data_rows, N, N]
  float alpha, beta;
  const int64_t *cur, *first;                   // [R]
  const uint8_t* mask;                          // [R, N] bool
  const float* state;                           // [R, n_state]
  float* G;                                     // [R, 128] glimpse (attention out) / g' (FFN out)
  float* logits;                                // [R, N]
  uint32_t* status;
};

// query: node half of the context projection (precomputed) + state scalars . state weights; lane l gets dims 4l..4l+3
__device__ __forceinline__ float4 step_query(const StepArgs& a, int64_t r, int64_t b, int cur, int lane) {
  const int N = a.N;
  float4 q;
  if (a.env == RRNCO_ENV_ATSP) {
    if (a.use_placeholder) {
      q = __ldg(reinterpret_cast<const float4*>(a.placeholder) + lane);
    } else {
      const float4 f4 = __ldg(reinterpret_cast<const float4*>(a.P1 + (b * N + (int)a.first[r]) * (int64_t)kE) + lane);
      const float4 c4 = __ldg(reinterpret_cast<const float4*>(a.P2 + (b * N + cur) * (int64_t)kE) + lane);
      q = make_float4(f4.x + c4.x, f4.y + c4.y, f4.z + c4.z, f4.w + c4.w);
    }
  } else {
    q = __ldg(reinterpret_cast<const float4*>(a.P1 + (b * N + cur) * (int64_t)kE) + lane);
    for (int k = 0; k < a.n_state; ++k) {
      const float st = a.state[r * a.n_state + k];
      const float4 w4 = __ldg(reinterpret_cast<const float4*>(a.wstate + k * kE) + lane);
      q.x = fmaf(st, w4.x, q.x); q.y = fmaf(st, w4.y, q.y); q.z = fmaf(st, w4.z, q.z); q.w = fmaf(st, w4.w, q.w);
    }
  }
  return q;
}

// one key of the online softmax of a head, for the lane that owns dims 4l..4l+3 (explicit fma / rn ops: the streaming and
// the tiled kernel must round identically)
__device__ __forceinline__ void attn_key(const float4& q, const float4& k4, const float4& v4, float& m, float& l, float4& acc) {
  float s = fmaf(q.w, k4.w, fmaf(q.z, k4.z, fmaf(q.y, k4.y, __fmul_rn(q.x, k4.x))));
  s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, 1));
  s = __fadd_rn(s, __shfl_xor_sync(0xffffffffu, s, 2));
  s = __fmul_rn(s, 0.25f);  // 1 / sqrt(head dim 16)
  const float mn = fmaxf(m, s);
  const float corr = sfexp(__fsub_rn(m, mn)), p = sfexp(__fsub_rn(s, mn));
  l = fmaf(l, corr, p);
  acc.x = fmaf(acc.x, corr, __fmul_rn(p, v4.x)); acc.y = fmaf(acc.y, corr, __fmul_rn(p, v4.y));
  acc.z = fmaf(acc.z, corr, __fmul_rn(p, v4.z)); acc.w = fmaf(acc.w, corr, __fmul_rn(p, v4.w));
  m = mn;
}
__device__ __forceinline__ float4 attn_finish(const float4& q, const float4& acc, float l) {
  const float inv = l > 0.f ? __frcp_rn(l) : 0.f;
  return make_float4(fmaf(acc.x, inv, q.x), fmaf(acc.y, inv, q.y), fmaf(acc.z, inv, q.z), fmaf(acc.w, inv, q.w));
}

__global__ void __launch_bounds__(kStepWarps * 32) attention_stream_kernel(const StepArgs a) {
  const int64_t r = (int64_t)blockIdx.x * kStepWarps + (threadIdx.x >> 5);
  if (r >= a.R) return;
  const int lane = threadIdx.x & 31;
  const int64_t b = r % a.n_inst;
  const int N = a.N;
  const float4* Kb = reinterpret_cast<const float4*>(a.K + b * (int64_t)N * kE);
  const float4* Vb = reinterpret_cast<const float4*>(a.V + b * (int64_t)N * kE);
  const int cur = (int)a.cur[r];
  const float4 q = step_query(a, r, b, cur, lane);
  // lane l owns dims 4l..4l+3 of head l >> 2; online softmax state is replicated over the 4 lanes of a head
  float m = -INFINITY, l = 0.f;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const uint8_t* mrow = a.mask + r * (int64_t)N;
  for (int n0 = 0; n0 < N; n0 += 32) {
    const int nn = n0 + lane;
    uint32_t feas = __ballot_sync(0xffffffffu, nn < N && mrow[nn] != 0);
    while (feas) {
      const int j = __ffs(feas) - 1;
      feas &= feas - 1;
      const int n = n0 + j;
      attn_key(q, __ldg(Kb + (size_t)n * 32 + lane), __ldg(Vb + (size_t)n * 32 + lane), m, l, acc);
    }
  }
  if (l <= 0.f && lane == 0) atomicOr(a.status, RRNCO_DEV_NO_FEASIBLE);
  reinterpret_cast<float4*>(a.G + r * (int64_t)kE)[lane] = attn_finish(q, acc, l);  // glimpse = heads + q (decoder.py:292-293)
}

// Tiled variant of attention_stream_kernel: one CTA = one instance x blockDim / 32 consecutive starts (one warp per rollout, same
// lane -> dims mapping and the same key order, so the glimpses are bit-identical).  Key / value rows are staged once per
// CTA in double-buffered shared-memory tiles of 32 keys (cp.async) and shared by the CTA's rollouts; each warp walks
// its own feasible keys of the tile.
constexpr int kAtGMax = 16, kAtKeys = 32;  // up to 16 warps per CTA, 64 KB of tiles: 3 CTAs per SM
__global__ void __launch_bounds__(kAtGMax * 32) attention_tile_kernel(const StepArgs a, int n_starts) {
  extern __shared__ __align__(16) float asm_[];  // [2][K tile | V tile], each kAtKeys x kE
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = blockIdx.x % a.n_inst;
  const int s = (int)(blockIdx.x / a.n_inst) * (int)(blockDim.x >> 5) + w;
  const bool live = s < n_starts;
  const int64_t r = live ? (int64_t)s * a.n_inst + b : 0;
  const int N = a.N;
  const float* Kb = a.K + b * (int64_t)N * kE;
  const float* Vb = a.V + b * (int64_t)N * kE;
  auto stage = [&](int t, int buf) {
    float* dk = asm_ + buf * 2 * kAtKeys * kE;
    float* dv = dk + kAtKeys * kE;
    const int n0 = t * kAtKeys;
    for (int i = threadIdx.x; i < kAtKeys * (kE / 4); i += blockDim.x) {
      const int k = i / (kE / 4);
      const bool ok = n0 + k < N;
      const size_t src = (size_t)min(n0 + k, N - 1) * kE + (i % (kE / 4)) * 4;
      cp_async16_zfill(dk + i * 4, Kb + src, ok);
      cp_async16_zfill(dv + i * 4, Vb + src, ok);
    }
  };
  const int n_tiles = (N + kAtKeys - 1) / kAtKeys;
  stage(0, 0);
  cp_async_commit();
  const int cur = (int)a.cur[r];
  const float4 q = step_query(a, r, b, cur, lane);
  float m = -INFINITY, l = 0.f;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  const uint8_t* mrow = a.mask + r * (int64_t)N;
  for (int t = 0; t < n_tiles; ++t) {
    if (t + 1 < n_tiles) stage(t + 1, (t + 1) & 1);
    cp_async_commit();
    const int nn = t * kAtKeys + lane;
    uint32_t feas = __ballot_sync(0xffffffffu, live && nn < N && mrow[nn] != 0);
    cp_async_wait<1>();
    __syncthreads();
    const float4* Kt = reinterpret_cast<const float4*>(asm_ + (t & 1) * 2 * kAtKeys * kE);
    const float4* Vt = Kt + kAtKeys * (kE / 4);
    while (feas) {
      const int j = __ffs(feas) - 1;
      feas &= feas - 1;
      attn_key(q, Kt[j * 32 + lane], Vt[j * 32 + lane], m, l, acc);
    }
    __syncthreads();  // every warp is done with buffer t & 1 before it is re-staged
  }
  cp_async_wait<0>();
  if (!live) return;
  if (l <= 0.f && lane == 0) atomicOr(a.status, RRNCO_DEV_NO_FEASIBLE);
  reinterpret_cast<float4*>(a.G + r * (int64_t)kE)[lane] = attn_finish(q, acc, l);  // glimpse = heads + q (decoder.py:292-293)
}

__global__ void __launch_bounds__(kStepWarps * 32) logits_stream_kernel(const StepArgs a) {
  __shared__ float4 sg[kStepWarps][32];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * kStepWarps + w;
  if (r >= a.R) return;
  const int64_t b = r % a.n_inst, drow = b % a.data_rows;
  const int N = a.N;
  sg[w][lane] = reinterpret_cast<const float4*>(a.G + r * (int64_t)kE)[lane];
  __syncwarp();
  const int cur = (int)a.cur[r];
  const float* Lkb = a.Lk + b * (int64_t)N * kE;
  const float* Drow = a.dist + (drow * N + cur) * (int64_t)N;
  const float* Urow = a.env == RRNCO_ENV_RCVRPTW ? a.dur + (drow * N + cur) * (int64_t)N : nullptr;
  bool nan_seen = false;
  for (int n0 = 0; n0 < N; n0 += 32) {
    const int n = n0 + lane;  // one key per lane, its 512-byte row streamed as 32 float4
    if (n < N) {
      const float4* krow = reinterpret_cast<const float4*>(Lkb + (size_t)n * kE);
      float acc = 0.f;
#pragma unroll 8
      for (int d4 = 0; d4 < 32; ++d4) {
        const float4 k4 = __ldg(krow + d4);
        const float4 g4 = sg[w][d4];
        acc = fmaf(g4.x, k4.x, acc); acc = fmaf(g4.y, k4.y, acc); acc = fmaf(g4.z, k4.z, acc); acc = fmaf(g4.w, k4.w, acc);
      }
      float lg = acc * 0.08838834764831845f;  // 1 / sqrt(128)
      nan_seen |= lg != lg;
      float bias = __fmul_rn(a.alpha, Drow[n]);
      if (Urow) bias = __fadd_rn(bias, __fmul_rn(a.beta, Urow[n]));
      lg = __logf(__fadd_rn(sfexp(__fsub_rn(lg, bias)), 1e-6f));  // decoder.py:198
      a.logits[r * (int64_t)N + n] = lg;
    }
  }
  if (__any_sync(0xffffffffu, nan_seen) && lane == 0) atomicOr(a.status, RRNCO_DEV_NAN_LOGITS);
}

// Tiled variant of logits_stream_kernel: one CTA = one instance x kLtG consecutive starts.  The logit-key rows are staged
// once per CTA through a double-buffered shared-memory tile of 32 keys (cp.async, rows padded to 132 floats so that the
// lane = key float4 reads are conflict-free) and shared by the CTA's rollouts, instead of every rollout streaming all
// N x 512 B from L2 with 16-byte accesses at a 512-byte lane stride (ncu launch list, ATSP n=1000: 800 us of a 1.2 ms
// decode step).  A warp owns 4 rollouts, lane = key; g' rows sit in shared memory and are read as broadcasts.  The
// accumulation order per (rollout, key) is the same as in logits_stream_kernel, so the logits are bit-identical.
constexpr int kLtWarps = 8, kLtPerWarp = 4, kLtG = kLtWarps * kLtPerWarp, kLtKeys = 32, kLtStride = kE + 4;
__global__ void __launch_bounds__(kLtWarps * 32) logits_tile_kernel(const StepArgs a, int n_starts) {
  extern __shared__ __align__(16) float lsm[];
  float* sg = lsm;                                  // [kLtG][kE]
  float* tiles = lsm + kLtG * kE;                   // [2][kLtKeys][kLtStride]
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = blockIdx.x % a.n_inst;
  const int s0 = (int)(blockIdx.x / a.n_inst) * kLtG;
  const int n_here = min(kLtG, n_starts - s0);
  const int N = a.N;
  const int64_t drow = b % a.data_rows;
  for (int i = threadIdx.x; i < kLtG * (kE / 4); i += blockDim.x) {
    const int j = i / (kE / 4), c = i % (kE / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j < n_here) v = reinterpret_cast<const float4*>(a.G + ((int64_t)(s0 + j) * a.n_inst + b) * kE)[c];
    reinterpret_cast<float4*>(sg + j * kE)[c] = v;
  }
  const float* Lkb = a.Lk + b * (int64_t)N * kE;
  auto stage = [&](int t, int buf) {
    float* dst = tiles + buf * kLtKeys * kLtStride;
    const int n0 = t * kLtKeys;
    for (int i = threadIdx.x; i < kLtKeys * (kE / 4); i += blockDim.x) {
      const int k = i / (kE / 4), c = i % (kE / 4);
      cp_async16_zfill(dst + k * kLtStride + c * 4, Lkb + (size_t)min(n0 + k, N - 1) * kE + c * 4, n0 + k < N);
    }
  };
  // blockIdx.y = chunk of key tiles (more CTAs than (instance, start group) pairs when those are few)
  const int tiles_all = (N + kLtKeys - 1) / kLtKeys;
  const int per_chunk = (tiles_all + gridDim.y - 1) / gridDim.y;
  const int t_begin = blockIdx.y * per_chunk, t_end = min(tiles_all, t_begin + per_chunk);
  if (t_begin >= t_end) return;
  stage(t_begin, 0);
  cp_async_commit();
  int64_t rr[kLtPerWarp];
  const float* Drow[kLtPerWarp];
  const float* Urow[kLtPerWarp];
#pragma unroll
  for (int j = 0; j < kLtPerWarp; ++j) {
    const int sj = s0 + w * kLtPerWarp + j;
    rr[j] = sj < n_starts ? (int64_t)sj * a.n_inst + b : -1;
    const int cur = rr[j] >= 0 ? (int)a.cur[rr[j]] : 0;
    Drow[j] = a.dist + (drow * N + cur) * (int64_t)N;
    Urow[j] = a.env == RRNCO_ENV_RCVRPTW ? a.dur + (drow * N + cur) * (int64_t)N : nullptr;
  }
  bool nan_seen = false;
  for (int t = t_begin; t < t_end; ++t) {
    const int buf = (t - t_begin) & 1;
    if (t + 1 < t_end) stage(t + 1, buf ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();  // tile t (and, at the first one, the g' rows) visible to every warp
    const float4* krow = reinterpret_cast<const float4*>(tiles + buf * kLtKeys * kLtStride + lane * kLtStride);
    float acc[kLtPerWarp];
#pragma unroll
    for (int j = 0; j < kLtPerWarp; ++j) acc[j] = 0.f;
#pragma unroll 8
    for (int d4 = 0; d4 < kE / 4; ++d4) {
      const float4 k4 = krow[d4];
#pragma unroll
      for (int j = 0; j < kLtPerWarp; ++j) {
        const float4 g4 = reinterpret_cast<const float4*>(sg + (w * kLtPerWarp + j) * kE)[d4];
        acc[j] = fmaf(g4.x, k4.x, acc[j]); acc[j] = fmaf(g4.y, k4.y, acc[j]);
        acc[j] = fmaf(g4.z, k4.z, acc[j]); acc[j] = fmaf(g4.w, k4.w, acc[j]);
      }
    }
    const int n = t * kLtKeys + lane;
    if (n < N) {
#pragma unroll
      for (int j = 0; j < kLtPerWarp; ++j) {
        if (rr[j] < 0) continue;
        float lg = acc[j] * 0.08838834764831845f;  // 1 / sqrt(128)
        nan_seen |= lg != lg;
        float bias = __fmul_rn(a.alpha, Drow[j][n]);
        if (Urow[j]) bias = __fadd_rn(bias, __fmul_rn(a.beta, Urow[j][n]));
        lg = __logf(__fadd_rn(sfexp(__fsub_rn(lg, bias)), 1e-6f));  // decoder.py:198
        a.logits[rr[j] * (int64_t)N + n] = lg;
      }
    }
    __syncthreads();  // every warp is done with this buffer before it is re-staged (the next iteration stages t + 2)
  }
  cp_async_wait<0>();
  if (__any_sync(0xffffffffu, nan_seen) && lane == 0) atomicOr(a.status, RRNCO_DEV_NAN_LOGITS);
}

// Tensor-core form of logits_tile_kernel: the logits of one instance are the dense contraction
// [starts x 128] . [128 x keys] that the POMO starts share, so it runs on mma.sync m16n8k8 with the 3xTF32 split
// (fp32-faithful, same helpers as the cache GEMM) instead of 128 FFMAs per (rollout, key).  One CTA = one instance x 32
// starts x a chunk of key tiles; 8 warps = 2 (rollout halves) x 4 (16-key slices of a 64-key tile).  The warp's A
// fragments (its 16 g' rows, hi | lo) are split once and stay in registers for every key tile; B fragments are split on
// the fly from the cp.async-staged, 132-float-padded key tile (conflict-free: bank = 4 g + t).
constexpr int kMmG = 32, kMmKeys = 64, kMmLd = kE + 4;
__global__ void __launch_bounds__(256) logits_mma_kernel(const StepArgs a, int n_starts) {
  extern __shared__ __align__(16) float msm[];
  float* sg = msm;                       // [kMmG][kMmLd]
  float* tiles = msm + kMmG * kMmLd;     // [2][kMmKeys][kMmLd]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int wm = warp >> 2, wn = warp & 3;
  const int64_t b = blockIdx.x % a.n_inst;
  const int s0 = (int)(blockIdx.x / a.n_inst) * kMmG;
  const int N = a.N;
  const int64_t drow = b % a.data_rows;
  const int tiles_all = (N + kMmKeys - 1) / kMmKeys;
  const int per_chunk = (tiles_all + gridDim.y - 1) / gridDim.y;
  const int t_begin = blockIdx.y * per_chunk, t_end = min(tiles_all, t_begin + per_chunk);
  if (t_begin >= t_end) return;
  for (int i = threadIdx.x; i < kMmG * (kE / 4); i += blockDim.x) {
    const int j = i / (kE / 4), c = i % (kE / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s0 + j < n_starts) v = reinterpret_cast<const float4*>(a.G + ((int64_t)(s0 + j) * a.n_inst + b) * kE)[c];
    *reinterpret_cast<float4*>(sg + j * kMmLd + c * 4) = v;
  }
  const float* Lkb = a.Lk + b * (int64_t)N * kE;
  auto stage = [&](int tt, int buf) {
    float* dst = tiles + buf * kMmKeys * kMmLd;
    const int n0 = tt * kMmKeys;
    for (int i = threadIdx.x; i < kMmKeys * (kE / 4); i += blockDim.x) {
      const int k = i / (kE / 4), c = i % (kE / 4);
      cp_async16_zfill(dst + k * kMmLd + c * 4, Lkb + (size_t)min(n0 + k, N - 1) * kE + c * 4, n0 + k < N);
    }
  };
  stage(t_begin, 0);
  cp_async_commit();
  // the two rollout rows this lane owns in the accumulator fragments: wm * 16 + g and + 8
  int64_t rr[2];
  const float* Drow[2];
  const float* Urow[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int sj = s0 + wm * 16 + g + 8 * h;
    rr[h] = sj < n_starts ? (int64_t)sj * a.n_inst + b : -1;
    const int cur = rr[h] >= 0 ? (int)a.cur[rr[h]] : 0;
    Drow[h] = a.dist + (drow * N + cur) * (int64_t)N;
    Urow[h] = a.env == RRNCO_ENV_RCVRPTW ? a.dur + (drow * N + cur) * (int64_t)N : nullptr;
  }
  __syncthreads();  // g' rows visible
  uint32_t ah[16][4], al[16][4];
#pragma unroll
  for (int ks = 0; ks < 16; ++ks) {
    const float* ap = sg + (wm * 16 + g) * kMmLd + ks * 8 + t;
    split_tf32(ap[0], ah[ks][0], al[ks][0]);
    split_tf32(ap[8 * kMmLd], ah[ks][1], al[ks][1]);
    split_tf32(ap[4], ah[ks][2], al[ks][2]);
    split_tf32(ap[8 * kMmLd + 4], ah[ks][3], al[ks][3]);
  }
  bool nan_seen = false;
  for (int tt = t_begin; tt < t_end; ++tt) {
    const int buf = (tt - t_begin) & 1;
    if (tt + 1 < t_end) stage(tt + 1, buf ^ 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    const float* tile = tiles + buf * kMmKeys * kMmLd;
    float acc[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 16; ++ks) {
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const float* bp = tile + (wn * 16 + nt * 8 + g) * kMmLd + ks * 8 + t;
        uint32_t bh[2], bl[2];
        split_tf32(bp[0], bh[0], bl[0]);
        split_tf32(bp[4], bh[1], bl[1]);
        mma_x<3>(acc[nt], ah[ks], al[ks], bh, bl);
      }
    }
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int n = tt * kMmKeys + wn * 16 + nt * 8 + 2 * t + e;
          if (n >= N || rr[h] < 0) continue;
          float lg = acc[nt][2 * h + e] * 0.08838834764831845f;  // 1 / sqrt(128)
          nan_seen |= lg != lg;
          float bias = __fmul_rn(a.alpha, Drow[h][n]);
          if (Urow[h]) bias = __fadd_rn(bias, __fmul_rn(a.beta, Urow[h][n]));
          lg = __logf(__fadd_rn(sfexp(__fsub_rn(lg, bias)), 1e-6f));  // decoder.py:198
          a.logits[rr[h] * (int64_t)N + n] = lg;
        }
    __syncthreads();  // every warp is done with this buffer before it is re-staged
  }
  cp_async_wait<0>();
  if (__any_sync(0xffffffffu, nan_seen) && lane == 0) atomicOr(a.status, RRNCO_DEV_NAN_LOGITS);
}

// a row of select_action_kernel for filter_cut: one warp, lane l owns the columns l, l + 32, ...
template <class Clipped>
struct FilterRowWarp {
  const Clipped& clipped;
  int N, lane;
  template <class F>
  __device__ __forceinline__ void for_each(F&& f) const {
    for (int n = lane; n < N; n += 32) f(clipped(n));
  }
  __device__ __forceinline__ float sum(float x) const {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
  }
  __device__ __forceinline__ int count(int c) const { return __reduce_add_sync(0xffffffffu, c); }
};

// DecodingStrategy.step: process_logits (tanh clip, mask, temperature, [top-k, top-p,] log-softmax) + greedy / Gumbel-max /
// forced.  kFilter: entries below the cut of filter_cut are dropped like masked ones (a forced action among them gets
// log p = -inf and is not reported as infeasible); every column draws the same Gumbel noise as without a filter.
template <bool kFilter>
__global__ void __launch_bounds__(kStepWarps * 32) select_action_kernel(int64_t R, int N, const float* __restrict__ logits,
                                                                       const uint8_t* __restrict__ mask, int mode,
                                                                       float tanh_clip, float temperature, uint64_t seed,
                                                                       int step, const int64_t* __restrict__ forced,
                                                                       int64_t* __restrict__ action_out,
                                                                       float* __restrict__ logp_out, uint32_t* status,
                                                                       int top_k, float top_p) {
  const int64_t r = (int64_t)blockIdx.x * kStepWarps + (threadIdx.x >> 5);
  if (r >= R) return;
  const int lane = threadIdx.x & 31;
  const float* lrow = logits + r * (int64_t)N;
  const uint8_t* mrow = mask + r * (int64_t)N;
  auto clipped = [&](int n) -> float {
    float l = lrow[n];
    if (tanh_clip > 0.f) l = __fmul_rn(1.0f - __fdividef(2.0f, __expf(2.0f * l) + 1.0f), tanh_clip);
    return mrow[n] ? __fdiv_rn(l, temperature) : -INFINITY;
  };
  float mx = -INFINITY;
  for (int n = lane; n < N; n += 32) mx = fmaxf(mx, clipped(n));
  mx = warp_max(mx);
  float cut = -INFINITY;
  if constexpr (kFilter) cut = filter_cut(FilterRowWarp<decltype(clipped)>{clipped, N, lane}, top_k, top_p, mx);
  auto kept = [&](int n) -> float {  // clipped(n), or -inf when the filter drops it
    const float v = clipped(n);
    if constexpr (kFilter) return v < cut ? -INFINITY : v;
    return v;
  };
  float se = 0.f;
  for (int n = lane; n < N; n += 32) se += sfexp((kFilter ? kept(n) : clipped(n)) - mx);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
  se = __logf(se);
  float best = -INFINITY;
  int besti = 0x7fffffff;
  const uint2 key2 = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  for (int n = lane; n < N; n += 32) {
    const float lp = __fsub_rn(__fsub_rn(kFilter ? kept(n) : clipped(n), mx), se);
    float key = lp;
    if (mode == RRNCO_DECODE_SAMPLING) {  // same stream as the fused kernel: Philox(seed; (r, step, n >> 2))[n & 3]
      const uint4 rnd = philox4x32(make_uint4((uint32_t)r, (uint32_t)(r >> 32), (uint32_t)step, (uint32_t)(n >> 2)), key2);
      const int c = n & 3;
      const uint32_t x = c == 0 ? rnd.x : c == 1 ? rnd.y : c == 2 ? rnd.z : rnd.w;
      key = lp + (-logf(-logf(u01(x))));
    }
    if (key > best) { best = key; besti = n; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, besti, o);
    if (ov > best || (ov == best && oi < besti)) { best = ov; besti = oi; }
  }
  int act = besti == 0x7fffffff ? 0 : besti;
  if (mode == RRNCO_DECODE_EVALUATE) act = min(max((int)forced[r], 0), N - 1);
  if (lane == 0) {
    if (!mrow[act]) atomicOr(status, besti == 0x7fffffff ? RRNCO_DEV_NO_FEASIBLE : RRNCO_DEV_INFEASIBLE);
    action_out[r] = act;
    logp_out[r] = __fsub_rn(__fsub_rn(kFilter ? kept(act) : clipped(act), mx), se);
  }
}

// rl4co BeamSearch._make_beam_step for one instance b per CTA: the W beam rows r = w * n_inst + b, candidate (w, n) of value
// score[r] + lp[r, n] and flat index w * N + n.  The W largest candidates are found with a 4-pass 8-bit radix select on the
// order-preserving key of filter_key (every pass recomputes the candidates from the L1/L2-resident logits: nothing of size
// W x N is stored), ranked by (value desc, flat index asc), and ranks from #finite upward copy rank 0 (_fill_up_beams).
// lp is select_action_kernel's per-row math (same operations, same order), so both give the same log-probs bit for bit.
constexpr int kBeamThreads = 512;
__global__ void __launch_bounds__(kBeamThreads) beam_select_kernel(int64_t n_inst, int W, int N, const float* __restrict__ logits,
                                                                   const uint8_t* __restrict__ mask, const float* score_in,
                                                                   float tanh_clip, float temperature,
                                                                   int64_t* __restrict__ action_out,
                                                                   int64_t* __restrict__ parent_out,
                                                                   float* __restrict__ logp_out, float* score_out,
                                                                   uint32_t* status) {
  extern __shared__ float bsm[];
  float* rmx = bsm;                                          // [W] row max of the processed logits
  float* rse = rmx + W;                                      // [W] row log-sum-exp
  float* rsc = rse + W;                                      // [W] beam scores (read before any is written: may alias)
  uint32_t* ckey = reinterpret_cast<uint32_t*>(rsc + W);     // [W] selected keys, unordered
  int* cidx = reinterpret_cast<int*>(ckey + W);              // [W] their flat indices
  int* sidx = cidx + W;                                      // [W] flat index of rank w
  float* sval = reinterpret_cast<float*>(sidx + W);          // [W] value of rank w
  __shared__ int hist[256];
  __shared__ int wsum[kBeamThreads / 32];
  __shared__ int s_digit, s_need, s_gt, s_eq;
  const int64_t b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  const int M = W * N;
  auto clipped = [&](const float* lrow, int n) -> float {
    float l = lrow[n];
    if (tanh_clip > 0.f) l = __fmul_rn(1.0f - __fdividef(2.0f, __expf(2.0f * l) + 1.0f), tanh_clip);
    return __fdiv_rn(l, temperature);
  };
  for (int w = warp; w < W; w += nw) {
    const int64_t r = (int64_t)w * n_inst + b;
    const float* lrow = logits + r * (int64_t)N;
    const uint8_t* mrow = mask + r * (int64_t)N;
    float mx = -INFINITY;
    for (int n = lane; n < N; n += 32) mx = fmaxf(mx, mrow[n] ? clipped(lrow, n) : -INFINITY);
    mx = warp_max(mx);
    float se = 0.f;
    for (int n = lane; n < N; n += 32) se += sfexp((mrow[n] ? clipped(lrow, n) : -INFINITY) - mx);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
    if (lane == 0) {
      rmx[w] = mx;
      rse[w] = __logf(se);
      rsc[w] = score_in[r];
    }
  }
  __syncthreads();
  // log-prob of node n in beam w's row (-inf when masked) and the candidate value score + lp
  auto logp = [&](int w, int n) -> float {
    const int64_t r = (int64_t)w * n_inst + b;
    if (!mask[r * (int64_t)N + n]) return -INFINITY;
    return __fsub_rn(__fsub_rn(clipped(logits + r * (int64_t)N, n), rmx[w]), rse[w]);
  };
  auto cand_key = [&](int f) -> uint32_t {
    const int w = f / N;
    return filter_key(__fadd_rn(rsc[w], logp(w, f - w * N)));
  };
  // radix select: K = the W-th largest key; `need` = how many candidates of key K rank among the W
  uint32_t prefix = 0u, pmask = 0u;
  int need = W;
#pragma unroll 1
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int f = tid; f < M; f += blockDim.x) {
      const uint32_t k = cand_key(f);
      if ((k & pmask) == prefix) atomicAdd(&hist[(k >> shift) & 255u], 1);
    }
    __syncthreads();
    if (tid == 0) {
      int acc = 0, d = 255;
      for (; d > 0; --d) {
        if (acc + hist[d] >= need) break;
        acc += hist[d];
      }
      s_digit = d;
      s_need = need - acc;
    }
    __syncthreads();
    prefix |= (uint32_t)s_digit << shift;
    pmask |= 255u << shift;
    need = s_need;
  }
  const uint32_t K = prefix;
  const int n_gt = W - need;
  // collect: every key > K, and the `need` lowest flat indices of key K (block-wide prefix count, in flat order)
  if (tid == 0) { s_gt = 0; s_eq = 0; }
  __syncthreads();
  for (int f0 = 0; f0 < M; f0 += blockDim.x) {
    const int f = f0 + tid;
    const uint32_t k = f < M ? cand_key(f) : 0u;
    const bool eq = f < M && k == K, gt = f < M && k > K;
    if (gt) {
      const int slot = atomicAdd(&s_gt, 1);
      ckey[slot] = k;
      cidx[slot] = f;
    }
    const unsigned bal = __ballot_sync(0xffffffffu, eq);
    if (lane == 0) wsum[warp] = __popc(bal);
    __syncthreads();
    int off = s_eq;
    for (int i = 0; i < warp; ++i) off += wsum[i];
    const int rank = off + __popc(bal & ((1u << lane) - 1u));
    if (eq && rank < need) {
      ckey[n_gt + rank] = k;
      cidx[n_gt + rank] = f;
    }
    __syncthreads();
    if (tid == 0) {
      int t = 0;
      for (int i = 0; i < nw; ++i) t += wsum[i];
      s_eq += t;
    }
    __syncthreads();
  }
  // order the W selected by (value desc, flat index asc); count the finite ones
  int fin = 0;
  for (int i = tid; i < W; i += blockDim.x) {
    const uint32_t ki = ckey[i];
    const int fi = cidx[i];
    int rk = 0;
    for (int j = 0; j < W; ++j) rk += (ckey[j] > ki || (ckey[j] == ki && cidx[j] < fi)) ? 1 : 0;
    sidx[rk] = fi;
    fin += ki > filter_key(-INFINITY) ? 1 : 0;
  }
  if (tid == 0) s_gt = 0;
  __syncthreads();
  if (fin) atomicAdd(&s_gt, fin);
  __syncthreads();
  const int finite = s_gt;
  for (int w = tid; w < W; w += blockDim.x) {
    const int f = sidx[w < finite ? w : 0];
    const int pw = f / N, n = f - pw * N;
    const float lp = logp(pw, n);
    sval[w] = __fadd_rn(rsc[pw], lp);
    const int64_t r = (int64_t)w * n_inst + b;
    action_out[r] = n;
    parent_out[r] = (int64_t)pw * n_inst + b;
    logp_out[r] = lp;
  }
  __syncthreads();  // every parent score has been read: score_out may alias score_in
  for (int w = tid; w < W; w += blockDim.x) score_out[(int64_t)w * n_inst + b] = sval[w];
  if (tid == 0 && finite == 0) atomicOr(status, RRNCO_DEV_NO_FEASIBLE);
}

// BeamSearch._backtrack: row r of the output is the path of the final beam r, followed back through the parent rows.
// Step-major inputs [T, R] (row t = what step t wrote; the parents of step 0 are never read); outputs [R, T], log-likelihood =
// fp64 sum of the aligned log-probs.  A parent row outside [0, R) sets RRNCO_DEV_BAD_PARENT; that row's earlier steps are
// written as action 0 with log-prob NaN, and its log-likelihood is NaN.
__global__ void beam_backtrack_kernel(int64_t R, int T, const int64_t* __restrict__ actions,
                                      const int64_t* __restrict__ parents, const float* __restrict__ logprobs,
                                      int64_t* __restrict__ actions_out, float* __restrict__ logprob_out,
                                      float* __restrict__ loglik_out, uint32_t* status) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  int64_t cur = r;
  double s = 0.0;
  int t = T - 1;
  for (; t >= 0; --t) {
    const int64_t i = (int64_t)t * R + cur;
    const float lp = logprobs[i];
    actions_out[r * T + t] = actions[i];
    if (logprob_out) logprob_out[r * T + t] = lp;
    s += (double)lp;
    if (t == 0) break;
    cur = parents[i];
    if (cur < 0 || cur >= R) {
      atomicOr(status, RRNCO_DEV_BAD_PARENT);
      s = NAN;
      break;
    }
  }
  for (--t; t >= 0; --t) {  // only after a bad parent
    actions_out[r * T + t] = 0;
    if (logprob_out) logprob_out[r * T + t] = NAN;
  }
  loglik_out[r] = (float)s;
}

}  // namespace rrnco

using namespace rrnco;

static int g_step_tiling = 1;  // rrnco_set_step_tiling (process-wide, read-only on the hot path)

extern "C" {

int rrnco_set_step_tiling(int32_t mode) {
  if (mode < 0 || mode > 2) return RRNCO_ERR_BAD_ARG;
  g_step_tiling = mode;
  return RRNCO_OK;
}

int64_t rrnco_decoder_logits_large_workspace_bytes(int64_t n_rollouts) {
  if (n_rollouts <= 0) return 0;
  return 2 * n_rollouts * (int64_t)kE * (int64_t)sizeof(float) + rrnco_pointer_ffn_workspace_bytes();
}

int rrnco_decoder_logits_large(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts,
                               const rrnco_decoder_weights_t* w, const rrnco_decoder_cache_t* cache,
                               const rrnco_instance_data_t* data, const int64_t* current, const int64_t* first,
                               const uint8_t* mask, const float* ctx_state, int32_t use_placeholder, float* logits_out,
                               uint32_t* status, void* workspace, void* stream) {
  RRNCO_CHECK_ARG(w && cache && data && n_inst > 0 && n_starts > 0 && n_nodes > 1 && env >= 0 && env <= 2);
  RRNCO_CHECK_ARG(w->ffn_w1 && w->ffn_b1 && w->ffn_w2 && w->ffn_b2);
  RRNCO_CHECK_ARG(cache->glimpse_key && cache->glimpse_val && cache->logit_key && cache->ctx_node_proj);
  RRNCO_CHECK_ARG(data->data_rows > 0 && data->distance && current && mask && logits_out && status && workspace);
  RRNCO_CHECK_ARG(((uintptr_t)workspace & 15) == 0);
  RRNCO_CHECK_ARG(env == RRNCO_ENV_ATSP ? (first && cache->ctx_node_proj2) : (ctx_state && w->ctx_state_w));
  RRNCO_CHECK_ARG(env != RRNCO_ENV_RCVRPTW || data->duration);
  RRNCO_CHECK_ARG(!use_placeholder || w->ctx_placeholder_q);
  cudaStream_t st = (cudaStream_t)stream;
  StepArgs a{};
  a.env = env; a.N = n_nodes; a.n_state = env == RRNCO_ENV_ATSP ? 0 : env == RRNCO_ENV_RCVRP ? 1 : 4;
  a.use_placeholder = use_placeholder;
  a.R = n_inst * n_starts; a.n_inst = n_inst; a.data_rows = data->data_rows;
  a.K = cache->glimpse_key; a.V = cache->glimpse_val; a.Lk = cache->logit_key;
  a.P1 = cache->ctx_node_proj; a.P2 = cache->ctx_node_proj2;
  a.wstate = w->ctx_state_w; a.placeholder = w->ctx_placeholder_q;
  a.dist = data->distance; a.dur = data->duration; a.alpha = w->alpha; a.beta = w->beta;
  a.cur = current; a.first = first; a.mask = mask; a.state = ctx_state;
  float* g0 = reinterpret_cast<float*>(workspace);
  float* g1 = g0 + a.R * kE;
  void* ffn_ws = g1 + a.R * kE;
  a.logits = logits_out; a.status = status;
  const unsigned grid = (unsigned)((a.R + kStepWarps - 1) / kStepWarps);
  a.G = g0;
  if (g_step_tiling && n_starts >= 4) {  // rollouts of one instance share the staged key / value tiles
    const size_t smem = (size_t)4 * kAtKeys * kE * sizeof(float);
    static PerDeviceOnce once;  // per device ordinal; idempotent, benign if raced
    if (once.first()) {
      if (cudaFuncSetAttribute(attention_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        once.undo();
        return RRNCO_ERR_CUDA;
      }
    }
    // 16 warps per CTA, the last group of an instance ragged.  Measured on BASELINE's ATSP n=1000 case (100 starts): 7
    // groups of 16 (the last one 4 warps) 303 us per step; 7 even groups of 15 warps 330-345 us; 5 groups of 20 warps
    // (one wave) 342 us - the CTA barriers per key tile cost more with wider / more uniform CTAs than the partial wave.
    const int64_t groups = (n_starts + kAtGMax - 1) / kAtGMax;
    const int warps = n_starts < kAtGMax ? n_starts : kAtGMax;
    attention_tile_kernel<<<(unsigned)(n_inst * groups), warps * 32, smem, st>>>(a, n_starts);
  } else {
    attention_stream_kernel<<<grid, kStepWarps * 32, 0, st>>>(a);
  }
  int rc = rrnco_launch_status();
  if (rc != RRNCO_OK) return rc;
  rc = rrnco_pointer_ffn(a.R, g0, w->ffn_w1, w->ffn_b1, w->ffn_w2, w->ffn_b2, g1, ffn_ws, stream);
  if (rc != RRNCO_OK) return rc;
  a.G = g1;
  if (g_step_tiling == 1 && n_starts >= 8) {  // the starts of one instance share the staged logit keys: tensor-core tiles
    const size_t smem = (size_t)(kMmG * kMmLd + 2 * kMmKeys * kMmLd) * sizeof(float);
    static PerDeviceOnce once;  // per device ordinal; idempotent, benign if raced
    if (once.first()) {
      if (cudaFuncSetAttribute(logits_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        once.undo();
        return RRNCO_ERR_CUDA;
      }
    }
    const int64_t groups = (n_starts + kMmG - 1) / kMmG;
    const int64_t tiles_all = (n_nodes + kMmKeys - 1) / kMmKeys;
    // 174 registers: one CTA per SM; aim at >= 6 waves so that the last, partial one costs little
    int64_t chunks = (6 * 148 + n_inst * groups - 1) / (n_inst * groups);
    chunks = chunks < 1 ? 1 : chunks > tiles_all ? tiles_all : chunks;
    logits_mma_kernel<<<dim3((unsigned)(n_inst * groups), (unsigned)chunks), 256, smem, st>>>(a, n_starts);
  } else if (g_step_tiling && n_starts >= kLtPerWarp) {  // FFMA form of the same tiling (rrnco_set_step_tiling(2))
    const size_t smem = (size_t)(kLtG * kE + 2 * kLtKeys * kLtStride) * sizeof(float);
    static PerDeviceOnce once;  // per device ordinal; idempotent, benign if raced
    if (once.first()) {
      if (cudaFuncSetAttribute(logits_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        once.undo();
        return RRNCO_ERR_CUDA;
      }
    }
    const int64_t groups = (n_starts + kLtG - 1) / kLtG;
    const int64_t tiles_all = (n_nodes + kLtKeys - 1) / kLtKeys;
    int64_t chunks = 4 * 148 / (n_inst * groups);  // fill, but do not exceed, one wave of 4 CTAs per SM when CTAs are few
    chunks = chunks < 1 ? 1 : chunks > tiles_all ? tiles_all : chunks;
    logits_tile_kernel<<<dim3((unsigned)(n_inst * groups), (unsigned)chunks), kLtWarps * 32, smem, st>>>(a, n_starts);
  } else {
    logits_stream_kernel<<<grid, kStepWarps * 32, 0, st>>>(a);
  }
  return rrnco_launch_status();
}

int rrnco_select_action_filtered(int64_t n_rollouts, int32_t n_nodes, const float* logits, const uint8_t* mask,
                                 int32_t decode_mode, float tanh_clipping, float temperature, uint64_t seed, int32_t step,
                                 const int64_t* forced_action, int64_t* action_out, float* logprob_out, uint32_t* status,
                                 int32_t top_k, float top_p, void* stream) {
  RRNCO_CHECK_ARG(top_k >= 0 && top_p >= 0.f && top_p <= 1.f);  // (a NaN top_p fails both comparisons)
  if (n_rollouts == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_rollouts > 0 && n_nodes > 0 && logits && mask && action_out && logprob_out && status);
  RRNCO_CHECK_ARG(decode_mode >= 0 && decode_mode <= 2 && temperature > 0.f);
  RRNCO_CHECK_ARG(decode_mode != RRNCO_DECODE_EVALUATE || forced_action);
  const unsigned grid = (unsigned)((n_rollouts + kStepWarps - 1) / kStepWarps);
  auto kern = rrnco_filter_active(top_k, top_p) ? select_action_kernel<true> : select_action_kernel<false>;
  kern<<<grid, kStepWarps * 32, 0, (cudaStream_t)stream>>>(n_rollouts, n_nodes, logits, mask, decode_mode, tanh_clipping,
                                                           temperature, seed, step, forced_action, action_out, logprob_out,
                                                           status, top_k, top_p);
  return rrnco_launch_status();
}

int rrnco_beam_select(int64_t n_inst, int32_t beam_width, int32_t n_nodes, const float* logits, const uint8_t* mask,
                      const float* score_in, float tanh_clipping, float temperature, int64_t* action_out, int64_t* parent_out,
                      float* logprob_out, float* score_out, uint32_t* status, void* stream) {
  RRNCO_CHECK_ARG(beam_width >= 2);
  if (beam_width > RRNCO_MAX_BEAM_WIDTH) return RRNCO_ERR_UNSUPPORTED;
  if (n_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && n_inst <= INT32_MAX && n_nodes > 0 && (int64_t)beam_width * n_nodes <= INT32_MAX);
  RRNCO_CHECK_ARG(logits && mask && score_in && action_out && parent_out && logprob_out && score_out && status);
  RRNCO_CHECK_ARG(temperature > 0.f);
  const size_t smem = (size_t)7 * beam_width * sizeof(float);  // <= 28 KB: no opt-in needed
  beam_select_kernel<<<(unsigned)n_inst, kBeamThreads, smem, (cudaStream_t)stream>>>(
      n_inst, beam_width, n_nodes, logits, mask, score_in, tanh_clipping, temperature, action_out, parent_out, logprob_out,
      score_out, status);
  return rrnco_launch_status();
}

int rrnco_beam_backtrack(int64_t n_rows, int32_t n_steps, const int64_t* actions, const int64_t* parents,
                         const float* logprobs, int64_t* actions_out, float* logprob_out, float* loglik_out,
                         uint32_t* status, void* stream) {
  if (n_rows == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_rows > 0 && n_steps > 0 && actions && parents && logprobs && actions_out && loglik_out && status);
  const unsigned grid = (unsigned)((n_rows + 127) / 128);
  beam_backtrack_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(n_rows, n_steps, actions, parents, logprobs, actions_out,
                                                                 logprob_out, loglik_out, status);
  return rrnco_launch_status();
}

int rrnco_select_action(int64_t n_rollouts, int32_t n_nodes, const float* logits, const uint8_t* mask, int32_t decode_mode,
                        float tanh_clipping, float temperature, uint64_t seed, int32_t step, const int64_t* forced_action,
                        int64_t* action_out, float* logprob_out, uint32_t* status, void* stream) {
  return rrnco_select_action_filtered(n_rollouts, n_nodes, logits, mask, decode_mode, tanh_clipping, temperature, seed, step,
                                      forced_action, action_out, logprob_out, status, 0, 0.f, stream);
}

}  // extern "C"
