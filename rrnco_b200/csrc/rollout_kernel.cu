// Fused construction-rollout kernel (RRNetPolicy.forward decode loop, rrnco/models/policy.py:203-243).
//
// One CTA = one problem instance x one tile of up to 128 POMO starts, persistent over ALL decode steps:
// rollout state (current node, visited bitset, load / time / route length, running tour length and
// log-likelihood) never leaves shared memory, so HBM only sees the per-instance key cache, the matrix
// rows the bias / mask need, and the int64 action stream that the reference API returns.
//
// Per step (all 128 rollouts of the tile together, weights shared => real GEMMs on the tensor pipe):
//   A. action mask (env.get_action_mask) as 128-bit row bitsets; query q = ctx_node_proj[cur] + state.w
//   C. 8-head masked attention: S = Q_h K_h^T, masked softmax, P V_h, + q
//   E. FFN 128 -> 512 -> 128 with residual
//   G. pointer logits g.Lk^T / sqrt(E), scale-adaptive bias log(exp(l - a.D[cur,:] - b.Dur[cur,:]) + 1e-6),
//      10.tanh, mask, log-softmax, greedy argmax / Gumbel-max sample / forced action, state transition.
//
// Two engines (template parameter kTc, rrnco_set_ffn_engine):
//   kTc = true  (default): every contraction on tcgen05.mma kind::f16 with the two-term fp16 operand split of
//       ffn_pack.cuh (three MMAs per K step = fp32-faithful; kPasses == 1 keeps only hi*hi), accumulators and the A
//       operands of the second GEMMs in tensor memory, K / V / logit keys pre-packed per CTA and TMA-loaded each step,
//       FFN weights TMA-streamed through a 4-stage ring; warps 0-7 run the element-wise passes thread-per-rollout,
//       warp 8 is the TMA producer, warps 9-11 issue the MMAs.  See DESIGN.md section 4.2 for the memory maps.
//   kTc = false: the first working version, everything on mma.sync.m16n8k8 3xTF32 with flash-style attention in
//       registers and a cp.async weight ring; also serves the logits-only mode (rrnco_decoder_logits).
#include <cstdio>
#include "common.cuh"
#include "tc05.cuh"
#include "ffn_pack.cuh"
#include "rollout_common.cuh"

namespace rrnco {

constexpr int kThreads = 256;      // compute threads (8 warps)
constexpr int kThreadsTc = 320;    // tcgen05 variant: + warp 8 (TMA producer) + warp 9 (MMA issue: one elected thread)
constexpr int kLdA = 132;    // fp32 row stride of the activation tiles (bank-conflict-free fragments)
constexpr int kLdB = 36;     // fp32 row stride of a streamed weight slice (32 k + 4 pad)
constexpr int kSliceK = 32;
constexpr int kStages = 3;
constexpr int kStageFloats = kRows * kLdB;
constexpr int kTileFloats = kRows * kLdA;
constexpr int kNumSlices = 36;  // 4 chunks x (4 W1 + 4 W2) + 4 Lk

// per-phase cycle accumulator of CTA 0 (debug / profiling aid, read back with rrnco_debug_phase_cycles)
__device__ long long g_phase_cycles[16];
#ifdef RRNCO_PHASE_STAMPS
#define PHASE_STAMP(i)                                   \
  do {                                                   \
    if (blockIdx.x == 0 && tid == 0) {                   \
      const long long now_ = clock64();                  \
      g_phase_cycles[i] += now_ - phase_t0;              \
      phase_t0 = now_;                                   \
    }                                                    \
  } while (0)
#else  // each stamp is a global read-modify-write on the critical warp: compiled out of the product build
#define PHASE_STAMP(i) do { } while (0)
#endif

#ifdef RRNCO_PHASE_STAMPS
// event timeline of CTA 0 at decode step kTlStep (development aid): (tag, clock64) pairs
__device__ long long g_tl[512];
__device__ int g_tl_n;
constexpr int kTlStep = 6;
#define TL(stepvar, tag)                                           \
  do {                                                             \
    if (blockIdx.x == 0 && ((stepvar) == kTlStep || (stepvar) == kTlStep + 1)) { \
      const int i_ = atomicAdd(&g_tl_n, 1);                        \
      if (i_ < 256) { g_tl[2 * i_] = (tag); g_tl[2 * i_ + 1] = clock64(); } \
    }                                                              \
  } while (0)
#else
#define TL(stepvar, tag) do { } while (0)
#endif

struct Smem {
  float A[kTileFloats];   // q -> glimpse -> glimpse'
  float Hb[kTileFloats];  // K tile (attention) / FFN hidden chunk
  float Bs[kTileFloats];  // V tile (attention) / 3-stage weight-slice ring
  float b1[kF];
  float b2[kE];
  float wstate[kMaxState][kE];
  float placeholder[kE];
  // per-instance node data
  float dem[kRows], demb[kRows], tw0[kRows], tw1[kRows], svc[kRows], dj0[kRows], uj0[kRows];
  // per-rollout state
  int cur[kRows], first[kRows], active[kRows], done[kRows];
  float f[kMaxState][kRows];  // rcvrp: used | rcvrptw: time, route, used_l, used_b | logits_only: ctx state
  uint32_t vis[kRows][4];
  uint32_t mask[kRows][4];
  double len[kRows];
  double lp[kRows];
  // thread-per-row select epilogue of the tcgen05 variant: the two column halves of a row exchange here
  float xf[3][2][kRows];
  int xi[2][kRows];
  float xchosen[kRows];
  uint32_t lhmask[4];     // rcvrptw: nodes with linehaul demand (bitset)
  float xsum[kH][kRows];  // tcgen05 attention: softmax denominators (written and read by the same thread)
  // tcgen05 FFN pipeline
  uint64_t bar_full[kFStages];
  uint64_t bar_empty[kFStages];
  uint64_t bar_go;      // compute -> producer: K / V tiles are dead, stream this step's weights (256 arrivals; or exit)
  uint64_t bar_kvgo;    // compute -> producer: the ring memory is free, load the packed K / V tiles of the next step
  uint64_t bar_kv;      // TMA -> issuers: packed K / V tiles landed
  uint64_t bar_q;       // compute -> issuers: query tiles written (256 arrivals; also the exit signal)
  uint64_t bar_qkdone;  // issuers -> producer: every Q K^T of the step complete, the K tiles are dead (8 commits)
  uint64_t bar_s[kH];   // issuers -> compute: scores of head h in TMEM
  uint64_t bar_p[kH];   // compute -> issuers: probabilities of head h written in place (128 arrivals)
  uint64_t bar_o[kH];   // issuers -> compute: P V of head h complete
  uint64_t bar_gready;  // compute -> issuers: glimpse tiles (A operand of GEMM1) written (256 arrivals)
  uint64_t bar_h[2];    // issuers -> compute: GEMM1 into hidden accumulator b complete
  uint64_t bar_epi;     // compute -> issuers: epilogue 1 done (A operand of GEMM2 in TMEM, accumulator re-zeroed)
  uint64_t bar_g2;      // issuers -> compute: GEMM2 of a chunk complete (its A operand may be overwritten)
  uint64_t bar_lk;      // compute -> issuers: g' (A operand of the logits GEMM) written to TMEM
  uint64_t bar_lkfull;  // TMA -> issuers: packed logit-key tiles landed
  uint64_t bar_acc;     // issuers -> compute: logits complete
  uint32_t tmem_base;
  volatile int exit_flag;
};

__device__ __forceinline__ bool bit_of(const uint32_t (&w)[4], int j, int e8) {
  // column c = 8 j + e8 (e8 < 8): word j >> 2, bit 8 (j & 3) + e8
  return (w[j >> 2] >> (8 * (j & 3) + e8)) & 1u;
}

// ---- env transition on the shared-memory state (one lane per row) -----------------------------------
template <int kEnv>
__device__ __forceinline__ void transition(Smem& sm, const RolloutParams& p, int row, int a, const float* D,
                                           const float* U, float cap, float closed, bool count_leg) {
  const int prev = sm.cur[row];
  const int N = p.N;
  if (kEnv == RRNCO_ENV_ATSP) {
    if (count_leg) sm.len[row] += (double)D[prev * N + a];
  } else if (kEnv == RRNCO_ENV_RCVRP) {
    sm.len[row] += (double)D[prev * N + a];
    const int di = min(max(a - 1, 0), N - 2) + 1;  // clamp(a-1, 0, n_loc-1), dem[] is depot-shifted
    sm.f[0][row] = __fmul_rn(__fadd_rn(sm.f[0][row], sm.dem[di]), a != 0 ? 1.0f : 0.0f);
  } else {
    const float away = a != 0 ? 1.0f : 0.0f;
    float leg = D[prev * N + a];
    if (a == 0) leg = __fmul_rn(leg, closed);
    sm.len[row] += (double)leg;
    const float dist = D[prev * N + a], dur = U[prev * N + a];
    sm.f[0][row] = __fmul_rn(away, __fadd_rn(fmaxf(__fadd_rn(sm.f[0][row], dur), sm.tw0[a]), sm.svc[a]));
    sm.f[1][row] = __fmul_rn(away, __fadd_rn(sm.f[1][row], dist));
    sm.f[2][row] = __fmul_rn(away, __fadd_rn(sm.f[2][row], sm.dem[a]));
    sm.f[3][row] = __fmul_rn(away, __fadd_rn(sm.f[3][row], sm.demb[a]));
  }
  sm.vis[row][a >> 5] |= 1u << (a & 31);
  sm.cur[row] = a;
  const int cnt = __popc(sm.vis[row][0]) + __popc(sm.vis[row][1]) + __popc(sm.vis[row][2]) + __popc(sm.vis[row][3]);
  sm.done[row] = cnt == N;
}

// ---- weight / logit-key slice stream ---------------------------------------------------------------
__device__ __forceinline__ void issue_slice(int s, Smem& sm, const RolloutParams& p, const float* Lk, int tid) {
  if (s < kNumSlices) {
    float* dst = sm.Bs + (s % kStages) * kStageFloats;
    const float* src;
    int ld, nrows;
    if (s < 32) {
      const int c = s >> 3, ks = s & 3;
      if (((s >> 2) & 1) == 0) {
        src = p.w.ffn_w1 + (size_t)c * kRows * kE + ks * kSliceK;  // rows: hidden units of chunk c
        ld = kE;
      } else {
        src = p.w.ffn_w2 + c * kRows + ks * kSliceK;  // rows: output dims, cols: hidden units of chunk c
        ld = kF;
      }
      nrows = kRows;
    } else {
      src = Lk + (s - 32) * kSliceK;
      ld = kE;
      nrows = p.N;
    }
#pragma unroll
    for (int i = 0; i < (kRows * 8) / kThreads; ++i) {
      const int idx = tid + i * kThreads, row = idx >> 3, c4 = idx & 7;
      cp_async16_zfill(dst + row * kLdB + c4 * 4, src + (size_t)(row < nrows ? row : 0) * ld + c4 * 4, row < nrows);
    }
  }
  cp_async_commit();  // always commit (possibly empty) so that wait_group counting stays uniform
}

// CTA-wide barriers over the 256 compute threads (the producer warp of the tcgen05 variant never joins them)
template <bool kTc>
__device__ __forceinline__ void cta_sync() {
  if (kTc) asm volatile("bar.sync 1, 256;\n" ::: "memory");
  else __syncthreads();
}
template <bool kTc>
__device__ __forceinline__ int cta_sync_and(int pred) {
  if (!kTc) return __syncthreads_and(pred);
  uint32_t r;
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.u32 q, %1, 0;\n\t"
      "bar.red.and.pred p, 1, 256, q;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(r)
      : "r"((uint32_t)pred)
      : "memory");
  return (int)r;
}

template <int kEnv, int kNTMax, int kPasses, bool kTc, bool kFilter>
__global__ void __launch_bounds__(kTc ? kThreadsTc : kThreads, 1) rollout_kernel(const RolloutParams p) {
  static_assert(kTc || !kFilter, "the top-k / top-p filters are built for the tcgen05 engine");
  extern __shared__ __align__(16) unsigned char smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>(smem_raw);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int N = p.N, NT = p.NT;
  const int tile = blockIdx.x % p.n_tiles;
  const int64_t b = blockIdx.x / p.n_tiles;
  const int64_t drow = b % p.d.data_rows;
  const float* D = p.d.distance + drow * (int64_t)N * N;
  const float* U = kEnv == RRNCO_ENV_RCVRPTW ? p.d.duration + drow * (int64_t)N * N : nullptr;
  const float* Kc = p.c.glimpse_key + b * (int64_t)N * kE;
  const float* Vc = p.c.glimpse_val + b * (int64_t)N * kE;
  const float* Lk = p.c.logit_key + b * (int64_t)N * kE;
  const float* P1 = p.c.ctx_node_proj + b * (int64_t)N * kE;
  const float* P2 = kEnv == RRNCO_ENV_ATSP ? p.c.ctx_node_proj2 + b * (int64_t)N * kE : nullptr;
  const float cap = (kEnv == RRNCO_ENV_ATSP || p.logits_only) ? 0.f : p.d.vehicle_capacity[drow];
  float closed = 1.f, limit = INFINITY, bclass = 1.f;
  if (kEnv == RRNCO_ENV_RCVRPTW && !p.logits_only) {
    closed = p.d.open_route[drow] ? 0.f : 1.f;
    limit = p.d.distance_limit[drow];
    bclass = p.d.backhaul_class[drow];
  }

  if (tid == 0) TL(kTlStep, 200);  // kernel start
  // ---------------- one-time staging ----------------
  if (kTc) {
    if (warp == 0) tc05::tmem_alloc(&sm.tmem_base, 512);
    if (tid == 32) {
      for (int i = 0; i < kFStages; ++i) {
        tc05::mbar_init(&sm.bar_full[i], 1);
        tc05::mbar_init(&sm.bar_empty[i], 1);
      }
      tc05::mbar_init(&sm.bar_go, kThreads);
      tc05::mbar_init(&sm.bar_kvgo, 1);
      tc05::mbar_init(&sm.bar_kv, 1);
      tc05::mbar_init(&sm.bar_q, kThreads);
      tc05::mbar_init(&sm.bar_qkdone, kH);
      for (int i = 0; i < kH; ++i) {
        tc05::mbar_init(&sm.bar_s[i], 1);
        tc05::mbar_init(&sm.bar_p[i], kThreads / 2);
        tc05::mbar_init(&sm.bar_o[i], 1);
      }
      tc05::mbar_init(&sm.bar_gready, kThreads);
      tc05::mbar_init(&sm.bar_h[0], 1);
      tc05::mbar_init(&sm.bar_h[1], 1);
      tc05::mbar_init(&sm.bar_epi, kThreads);
      tc05::mbar_init(&sm.bar_g2, 1);
      tc05::mbar_init(&sm.bar_lk, kThreads);
      tc05::mbar_init(&sm.bar_lkfull, 1);
      tc05::mbar_init(&sm.bar_acc, 1);
      tc05::fence_mbar_init();
      sm.exit_flag = 0;
    }
  }
  for (int i = tid; i < kF; i += kTc ? kThreadsTc : kThreads) sm.b1[i] = p.w.ffn_b1[i];
  if (tid < kE) {
    sm.b2[tid] = p.w.ffn_b2[tid];
    sm.placeholder[tid] = p.w.ctx_placeholder_q ? p.w.ctx_placeholder_q[tid] : 0.f;
#pragma unroll
    for (int k = 0; k < kMaxState; ++k) sm.wstate[k][tid] = k < p.n_state ? p.w.ctx_state_w[k * kE + tid] : 0.f;
  }
  if (tid < kRows && !p.logits_only) {
    const int n = tid;
    float dem = 0.f, demb = 0.f, tw0 = 0.f, tw1 = 0.f, svc = 0.f, dj0 = 0.f, uj0 = 0.f;
    if (n < N) {
      if (kEnv == RRNCO_ENV_RCVRP) dem = n >= 1 ? p.d.demand[drow * (N - 1) + n - 1] : 0.f;
      if (kEnv == RRNCO_ENV_RCVRPTW) {
        dem = p.d.demand[drow * N + n];
        demb = p.d.demand_backhaul[drow * N + n];
        tw0 = p.d.time_windows[(drow * N + n) * 2];
        tw1 = p.d.time_windows[(drow * N + n) * 2 + 1];
        svc = p.d.service_time[drow * N + n];
        dj0 = D[n * N];
        uj0 = U[n * N];
      }
    }
    sm.dem[n] = dem; sm.demb[n] = demb; sm.tw0[n] = tw0; sm.tw1[n] = tw1; sm.svc[n] = svc;
    sm.dj0[n] = dj0; sm.uj0[n] = uj0;
    const uint32_t lh = __ballot_sync(0xffffffffu, kEnv == RRNCO_ENV_RCVRPTW && dem > 0.f);
    if (lane == 0) sm.lhmask[warp] = lh;
  }
  __syncthreads();

  if (tid == 0) TL(kTlStep, 201);  // staging done
  // ---------------- rollout state init ----------------
  const int num_loc = kEnv == RRNCO_ENV_ATSP ? N : N - 1;
  if (tid < kRows) {
    const int row = tid;
    const int s_real = tile * kRows + row;
    const int active = s_real < p.S;
    const int s = active ? s_real : tile * kRows;  // padded rows shadow the tile's first rollout
    const int64_t r = (int64_t)s * p.n_inst + b;
    sm.active[row] = active;
    sm.len[row] = 0.0;
    sm.lp[row] = 0.0;
    sm.first[row] = 0;
#pragma unroll
    for (int k = 0; k < kMaxState; ++k) sm.f[k][row] = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) { sm.vis[row][k] = 0u; sm.mask[row][k] = 0u; }
    sm.done[row] = 0;
    sm.cur[row] = 0;
    if (p.logits_only) {
      sm.cur[row] = (int)p.in_cur[r];
      if (kEnv == RRNCO_ENV_ATSP) sm.first[row] = (int)p.in_first[r];
      for (int k = 0; k < p.n_state; ++k) sm.f[k][row] = p.in_state[r * p.n_state + k];
      const uint8_t* m = p.in_mask + r * (int64_t)N;
      for (int n = 0; n < N; ++n)
        if (m[n]) sm.mask[row][n >> 5] |= 1u << (n & 31);
    } else if (p.multistart) {
      const int a0 = s % num_loc + (kEnv == RRNCO_ENV_ATSP ? 0 : 1);  // select_start_nodes
      transition<kEnv>(sm, p, row, a0, D, U, cap, closed, /*count_leg=*/false);
      sm.first[row] = a0;
      if (active) {
        p.actions[r * p.t_cap] = a0;
        if (p.logprob) p.logprob[r * p.t_cap] = 0.f;
      }
    }
  }
  __syncthreads();

  if (kTc) {
    // ---- one-time: K / V of this instance -> fp16 hi | lo tiles in the shared-memory layouts of the attention MMAs,
    // parked in this SM's workspace slot (L2-resident; exactly one CTA lives on an SM at a time) and re-loaded by TMA
    // every decode step, because the FFN weight ring needs the same shared memory in between.
    //   K: [hi | lo][16-byte K chunk c8 (16)][key (R16)][8 halves]            B operand of Q K^T, head h = chunks 2h, 2h+1
    //   V: [hi | lo][head (8)][key chunk (R16 / 8)][dim (16)][8 halves]       B operand (V_h^T, K-major) of P V
    if (tid == 0) TL(kTlStep, 202);  // state init done
    const int R16p = ((N + 15) >> 4) << 4;
    uint32_t smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    if (smid >= (uint32_t)kKvSlots) __trap();
    unsigned char* slot = p.kv_pack + (size_t)smid * kKvSlotBytes;
    if (tid < kThreads) {
      uint4* v_hi = reinterpret_cast<uint4*>(slot + kKvOffV);
      const int var16 = R16p * 16;  // uint4 elements per variant
#pragma unroll 1
      for (int which = 0; which < 2; ++which) {  // glimpse keys, then logit keys: same row-major -> chunk-major repack
        const float* src = which ? Lk : Kc;
        const float scale = which ? kLkScale : kKvScale;
        uint4* k_hi = reinterpret_cast<uint4*>(slot + (which ? kKvOffLk : 0));
        for (int idx = tid; idx < R16p * 16; idx += kThreads) {
          const int r = idx >> 4, c8 = idx & 15;
          float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
          if (r < N) {
            v0 = __ldg(reinterpret_cast<const float4*>(src + (size_t)r * kE) + c8 * 2);
            v1 = __ldg(reinterpret_cast<const float4*>(src + (size_t)r * kE) + c8 * 2 + 1);
          }
          uint32_t h[4], l[4];
          f16s_split2(v0.x, v0.y, scale, h[0], l[0]); f16s_split2(v0.z, v0.w, scale, h[1], l[1]);
          f16s_split2(v1.x, v1.y, scale, h[2], l[2]); f16s_split2(v1.z, v1.w, scale, h[3], l[3]);
          k_hi[c8 * R16p + r] = make_uint4(h[0], h[1], h[2], h[3]);
          k_hi[var16 + c8 * R16p + r] = make_uint4(l[0], l[1], l[2], l[3]);
        }
      }
      const int nkc = R16p >> 3;
      for (int idx = tid; idx < R16p * 16; idx += kThreads) {
        const int d = idx & 15, kc = (idx >> 4) % nkc, hh = (idx >> 4) / nkc;
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int key = kc * 8 + j;
          x[j] = key < N ? __ldg(Vc + (size_t)key * kE + hh * kDh + d) : 0.f;
        }
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) f16s_split2(x[2 * j], x[2 * j + 1], kKvScale, h[j], l[j]);
        v_hi[(hh * nkc + kc) * 16 + d] = make_uint4(h[0], h[1], h[2], h[3]);
        v_hi[var16 + (hh * nkc + kc) * 16 + d] = make_uint4(l[0], l[1], l[2], l[3]);
      }
      tc05::fence_proxy_async_all();
    }
    tc05::fence_before_sync();
    __syncthreads();
    tc05::fence_after_sync();
    if (tid == 0) tc05::mbar_arrive(&sm.bar_kvgo);
    if (tid == 0) TL(kTlStep, 203);  // K / V / Lk packed
    // warp index as a value the compiler knows to be warp-uniform (threadIdx.x >> 5 is not, to its analysis)
    const int uwarp = __shfl_sync(0xffffffffu, warp, 0);
    if (uwarp == 8) {
      // ===== TMA producer warp.  Per decode step: the packed K / V tiles (as soon as the previous step's logits have
      // released the Hb | Bs regions), then -- once the attention is done with them -- the 16 packed 32 KB FFN weight
      // slices through the same memory used as a 4-stage ring.  One elected thread (tc05::elect_one) =====
      if (tc05::elect_one()) {
        uint32_t go_phase = 0;
        uint32_t sl = 0;
        unsigned char* ring = reinterpret_cast<unsigned char*>(sm.Hb);
        const uint32_t kv_bytes = (uint32_t)R16p * 512u;  // hi | lo tiles of K (same for V)
        while (true) {
          tc05::mbar_wait(&sm.bar_kvgo, go_phase, 64);
          tc05::mbar_arrive_expect_tx(&sm.bar_kv, 2 * kv_bytes);
          tc05::bulk_g2s(ring, slot, kv_bytes, &sm.bar_kv);
          tc05::bulk_g2s(ring + kKvOffV, slot + kKvOffV, kv_bytes, &sm.bar_kv);
          // Weight slices 0 and 1 land in ring stages that overlap only the K tiles: they start as soon as the last
          // Q K^T has completed, i.e. under the softmax / P V of the last heads.  The rest waits for the V tiles to die.
          tc05::mbar_wait(&sm.bar_qkdone, go_phase, 64);
          if (sm.exit_flag) break;
#pragma unroll 1
          for (int s = 0; s < kFSlices; ++s, ++sl) {
            if (s == 2) tc05::mbar_wait(&sm.bar_go, go_phase, 64);
            const int st = sl & (kFStages - 1);
            if (sl >= kFStages) tc05::mbar_wait(&sm.bar_empty[st], ((sl / kFStages) - 1) & 1);
            tc05::mbar_arrive_expect_tx(&sm.bar_full[st], kFSliceBytes);
            tc05::bulk_g2s(ring + (size_t)st * kFSliceBytes, p.ffn_packed + (size_t)s * kFSliceBytes, kFSliceBytes,
                           &sm.bar_full[st]);
          }
          go_phase ^= 1u;
          // logit keys -> ring start (stages 0 and 1) as soon as the weight slices 12 and 13 held there are consumed
          tc05::mbar_wait(&sm.bar_empty[(sl - 4) & (kFStages - 1)], (((sl - 4) / kFStages)) & 1);
          tc05::mbar_wait(&sm.bar_empty[(sl - 3) & (kFStages - 1)], (((sl - 3) / kFStages)) & 1);
          tc05::mbar_arrive_expect_tx(&sm.bar_lkfull, kv_bytes);
          tc05::bulk_g2s(ring, slot + kKvOffLk, kv_bytes, &sm.bar_lkfull);
        }
      }
      return;
    }
    if (uwarp == 9) {
      // ===== MMA issue warp: ONE elected thread issues every tcgen05.mma of the CTA, in a fixed program order.  The
      // tensor pipe executes MMAs in issue order, so the accumulation order into every TMEM accumulator is fixed and the
      // rollout is bitwise reproducible run to run.  (Issue costs ~10 cycles per MMA from waterfall-free code, against
      // 21 / 67 / 75 / 107 cycles of tensor time for TS N=16 / TS N=112 / TS N=128 / SS N=128: one thread is enough.)
      //  attention: heads in the sequence 0 4 1 5 2 6 3 7 (the two compute-warp groups take alternate positions), score
      //    buffer k % 3.  Q K^T of positions 0-2 at once; then per position k: wait for P(k), issue P V(k) (R16 / 16 K
      //    steps x split terms into the pre-zeroed O tile) and, behind it on the in-order pipe, Q K^T(k + 3) into the
      //    score buffer P V(k) has just finished reading.
      //  FFN / logits: per K step the split terms (A_hi B_hi, A_lo B_hi, A_hi B_lo; single-pass mode: the first only), all
      //    into pre-zeroed TMEM tiles.  Tensor-pipe order  G1(0) G1(1) G2(0) G1(2) G2(1) G1(3) G2(2) G2(3) logits: GEMM1
      //    alternates between two accumulators, so epilogue 1 of chunk c runs under GEMM1 of chunk c + 1. =====
      if (tc05::elect_one()) {
        const uint32_t tb = sm.tmem_base;
        const uint32_t t_hacc0 = tb, t_oacc = tb + 256, t_ahi = tb + 384, t_alo = tb + 448;
        const uint32_t idesc = tc05::make_idesc_f16(128, 128);
        const uint32_t q_addr = tc05::smem_u32(sm.A);                // Q_hi | Q_lo, then G_hi | G_lo
        const uint32_t a_lo_off = kRows * kE * 2;
        const uint32_t ring_addr = tc05::smem_u32(sm.Hb);
        const uint32_t b_lo_off = kFVariantHalves * 2;
        const int R16i = R16p;
        const uint32_t idesc_l = tc05::make_idesc_f16(128, R16i);
        const uint32_t idesc_pv = tc05::make_idesc_f16(128, 16);
        const uint32_t lbo_l = (uint32_t)R16i * 16u;
        const uint32_t kv_var = (uint32_t)R16i * 256u;  // bytes of one hi / lo variant of the K (or V) tiles
        uint32_t step_par = 0, epi_phase = 0, sl = 0;
        int istep = -1;
        auto issue_qk = [&](int k) {
          const int h = (k & 1) * 4 + (k >> 1);
          const uint32_t t_s = tb + (uint32_t)(k % 3) * 128u;
          const uint32_t qh = q_addr + 2 * h * kLboTile, kh = ring_addr + 2 * h * lbo_l;
          const uint64_t q_hi = tc05::make_desc(qh, kLboTile, kSbo), k_hi = tc05::make_desc(kh, lbo_l, kSbo);
          tc05::mma_ss_f16(t_s, q_hi, k_hi, idesc_l, 0u);
          if (kPasses == 3) {
            tc05::mma_ss_f16(t_s, tc05::make_desc(qh + a_lo_off, kLboTile, kSbo), k_hi, idesc_l, 1u);
            tc05::mma_ss_f16(t_s, q_hi, tc05::make_desc(kh + kv_var, lbo_l, kSbo), idesc_l, 1u);
          }
          tc05::commit(&sm.bar_s[h]);
          tc05::commit(&sm.bar_qkdone);
          TL(istep, 110 + h);  // QK(h) issued
        };
        while (true) {
          tc05::mbar_wait(&sm.bar_q, step_par, 32);
          if (sm.exit_flag) break;
          ++istep;
          TL(istep, 100);  // Q ready seen
          tc05::mbar_wait(&sm.bar_kv, step_par, 32);
          tc05::fence_after_sync();
          issue_qk(0);
          issue_qk(1);
          issue_qk(2);
#pragma unroll 1
          for (int k = 0; k < kH; ++k) {
            const int h = (k & 1) * 4 + (k >> 1);
            const uint32_t t_s = tb + (uint32_t)(k % 3) * 128u;
            tc05::mbar_wait(&sm.bar_p[h], step_par, 32);
            tc05::fence_after_sync();
            TL(istep, 120 + h);  // P(h) seen
            // V_h^T tile: 16 dims x keys, K-major: 256 B between 16-byte key chunks, 128 B between 8-dim groups;
            // P_hi at columns 16 j, P_lo at 16 j + 8 of the score buffer
            const uint32_t vh = ring_addr + kKvOffV + h * (R16i * 32);
#pragma unroll 1
            for (int j = 0; j < (R16i >> 4); ++j) {
              const uint64_t v_hi = tc05::make_desc(vh + j * 512, 256, kSbo);
              tc05::mma_ts_f16(tb + 384 + 16 * h, t_s + 16 * j, v_hi, idesc_pv, 1u);
              if (kPasses == 3) {
                tc05::mma_ts_f16(tb + 384 + 16 * h, t_s + 16 * j + 8, v_hi, idesc_pv, 1u);
                tc05::mma_ts_f16(tb + 384 + 16 * h, t_s + 16 * j, tc05::make_desc(vh + kv_var + j * 512, 256, kSbo), idesc_pv, 1u);
              }
            }
            tc05::commit(&sm.bar_o[h]);
            TL(istep, 130 + h);  // PV(h) issued
            if (k + 3 < kH) issue_qk(k + 3);
          }
          tc05::mbar_wait(&sm.bar_gready, step_par, 32);
          tc05::fence_after_sync();
          TL(istep, 140);  // glimpse seen
#pragma unroll 1
          for (int j = 0; j < 8; ++j) {
            const int c = ffn_job_chunk(j), half = ffn_job_half(j);
            if (half == 1) {  // A operand of GEMM2(c) written (and, one job later, accumulator c & 1 re-zeroed)
              tc05::mbar_wait(&sm.bar_epi, epi_phase, 32);
              epi_phase ^= 1u;
              tc05::fence_after_sync();
            }
#pragma unroll 1
            for (int sj = 0; sj < kFSlicesPerJob; ++sj, ++sl) {
              const int st = sl & (kFStages - 1);
              tc05::mbar_wait(&sm.bar_full[st], (sl / kFStages) & 1);
              tc05::fence_after_sync();
              const uint32_t b_addr = ring_addr + st * kFSliceBytes;
#pragma unroll
              for (int kk = 0; kk < kFKSteps; ++kk) {
                const int ks = sj * kFKSteps + kk;  // K step (16 values) of the job
                const uint64_t b_hi = tc05::make_desc(b_addr + kk * 2 * kLboTile, kLboTile, kSbo);
                const uint64_t b_lo = tc05::make_desc(b_addr + b_lo_off + kk * 2 * kLboTile, kLboTile, kSbo);
                if (half == 0) {
                  const uint32_t t_h = t_hacc0 + (c & 1) * 128;
                  const uint64_t a_hi = tc05::make_desc(q_addr + ks * 2 * kLboTile, kLboTile, kSbo);
                  tc05::mma_ss_f16(t_h, a_hi, b_hi, idesc, 1u);
                  if (kPasses == 3) {
                    tc05::mma_ss_f16(t_h, tc05::make_desc(q_addr + a_lo_off + ks * 2 * kLboTile, kLboTile, kSbo), b_hi, idesc, 1u);
                    tc05::mma_ss_f16(t_h, a_hi, b_lo, idesc, 1u);
                  }
                } else {
                  tc05::mma_ts_f16(t_oacc, t_ahi + ks * 8, b_hi, idesc, 1u);
                  if (kPasses == 3) {
                    tc05::mma_ts_f16(t_oacc, t_alo + ks * 8, b_hi, idesc, 1u);
                    tc05::mma_ts_f16(t_oacc, t_ahi + ks * 8, b_lo, idesc, 1u);
                  }
                }
              }
              tc05::commit(&sm.bar_empty[st]);
            }
            tc05::commit(half == 0 ? &sm.bar_h[c & 1] : &sm.bar_g2);
            TL(istep, 150 + j);  // FFN job j issued
          }
          // pointer logits: D[128 x R16] = g'(hi | lo, TMEM) . Lk(hi | lo, shared memory)^T, 8 K steps
          tc05::mbar_wait(&sm.bar_lk, step_par, 32);
          tc05::mbar_wait(&sm.bar_lkfull, step_par, 32);
          tc05::fence_after_sync();
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            const uint64_t l_hi = tc05::make_desc(ring_addr + ks * 2 * lbo_l, lbo_l, kSbo);
            tc05::mma_ts_f16(t_hacc0, t_ahi + ks * 8, l_hi, idesc_l, 1u);
            if (kPasses == 3) {
              tc05::mma_ts_f16(t_hacc0, t_alo + ks * 8, l_hi, idesc_l, 1u);
              tc05::mma_ts_f16(t_hacc0, t_ahi + ks * 8, tc05::make_desc(ring_addr + kv_var + ks * 2 * lbo_l, lbo_l, kSbo), idesc_l, 1u);
            }
          }
          tc05::commit(&sm.bar_acc);
          TL(istep, 160);  // logits issued
          step_par ^= 1u;
        }
      }
      return;
    }
  }
  uint32_t tc_step_par = 0;  // parity of the once-per-step barriers (bar_acc)
  if (kTc) {  // every MMA accumulates: zero the two hidden-chunk accumulators and the output accumulator once
    uint32_t z[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) z[i] = 0u;
    const uint32_t lb = (uint32_t)((warp & 3) * 32) << 16;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      tc05::tmem_st16(sm.tmem_base + lb + (warp >> 2) * 64 + q * 16, z);
      tc05::tmem_st16(sm.tmem_base + 128 + lb + (warp >> 2) * 64 + q * 16, z);
      tc05::tmem_st16(sm.tmem_base + 256 + lb + (warp >> 2) * 64 + q * 16, z);
      tc05::tmem_st16(sm.tmem_base + 384 + lb + (warp >> 2) * 64 + q * 16, z);  // O tile of the attention
    }
    tc05::tmem_wait_st();
    tc05::fence_before_sync();
    cta_sync<kTc>();
    tc05::fence_after_sync();
  }
  if (tid == 0) TL(kTlStep, 204);  // TMEM zeroed, entering the step loop
  long long phase_t0 = clock64();
  const int r0 = warp * 16 + g, r1 = r0 + 8;  // rows owned by this quad in the row-owner phases
  const int wm = warp >> 1, wn = warp & 1;    // FFN warp grid 4 (M) x 2 (N): 32 x 64 warp tiles
  int step = 0;
  int t_out = p.multistart ? 1 : 0;
  const int NPAD = NT * 8;
  bool kv_prefetched = false;

  while (true) {
    if (!p.logits_only) {
      const int all_done = cta_sync_and<kTc>(tid < kRows ? (sm.done[tid] || !sm.active[tid]) : 1);
      if (all_done) break;
      if (step >= p.max_steps) {  // policy.py:222-226: cut, but never silently
        if (tid == 0) atomicOr(p.status, RRNCO_DEV_TRUNCATED);
        break;
      }
    }
    // ---- B (issued first so that the copies overlap phase A): K -> Hb, V -> Bs -----------------
    // (the tcgen05 variant prefetches them for step t+1 right after the logits MMAs of step t)
    if (!kTc && !kv_prefetched) {
      for (int idx = tid; idx < NPAD * 32; idx += kThreads) {
        const int row = idx >> 5, c4 = idx & 31;
        const bool ok = row < N;
        const size_t off = (size_t)(ok ? row : 0) * kE + c4 * 4;
        cp_async16_zfill(sm.Hb + row * kLdA + c4 * 4, Kc + off, ok);
        cp_async16_zfill(sm.Bs + row * kLdA + c4 * 4, Vc + off, ok);
      }
      cp_async_commit();
    }
    kv_prefetched = false;

    // ---- A1: action mask bitsets (row-owner quads; the tcgen05 variant computes them in its phase A below) ----
    if (!kTc && !p.logits_only) {
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const int row = rr ? r1 : r0;
        const int cur = sm.cur[row];
        uint32_t vis[4], bits[4] = {0u, 0u, 0u, 0u};
        *reinterpret_cast<uint4*>(vis) = *reinterpret_cast<const uint4*>(sm.vis[row]);
        float f0 = sm.f[0][row], f1 = sm.f[1][row], f2 = sm.f[2][row], f3 = sm.f[3][row];
        bool missing = false, carrying_b = false;
        if (kEnv == RRNCO_ENV_RCVRPTW) {
          // linehauls_missing: any unvisited node with linehaul demand (lane-strided scan of 128 nodes)
          for (int n = t; n < N; n += 4)
            missing |= sm.dem[n] > 0.f && !((vis[n >> 5] >> (n & 31)) & 1u);
          missing = __any_sync(0xfu << (lane & ~3), missing);
          carrying_b = sm.demb[cur] > 0.f;
        }
#pragma unroll
        for (int j = 0; j < kNTMax; ++j) {
          if (j < NT) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int c = 8 * j + 2 * t + e;
              bool ok = false;
              if (c < N) {
                const bool v = bit_of(vis, j, 2 * t + e);
                if (kEnv == RRNCO_ENV_ATSP) {
                  ok = !v;
                } else if (kEnv == RRNCO_ENV_RCVRP) {
                  ok = c >= 1 && !v && !(__fadd_rn(sm.dem[c], f0) > cap);
                } else if (c >= 1) {
                  const float dist_ij = D[cur * N + c], dur_ij = U[cur * N + c];
                  const float arrival = __fadd_rn(f0, dur_ij);
                  const bool reach_c = arrival < sm.tw1[c];
                  const bool reach_d =
                      __fmul_rn(__fadd_rn(__fadd_rn(fmaxf(arrival, sm.tw0[c]), sm.svc[c]), sm.uj0[c]), closed) <
                      sm.tw1[0];
                  const bool exc_lim = __fadd_rn(__fadd_rn(f1, dist_ij), __fmul_rn(sm.dj0[c], closed)) > limit;
                  const bool exc_l = __fadd_rn(sm.dem[c], f2) > cap;
                  const bool exc_b = __fadd_rn(sm.demb[c], f3) > cap;
                  const bool ok1 = (missing && !exc_l && !carrying_b && sm.dem[c] > 0.f) ||
                                   (!exc_b && sm.demb[c] > 0.f);
                  const bool cannot_l = sm.dem[c] > __fsub_rn(cap, f3);
                  const bool ok2 = !exc_l && !exc_b && !cannot_l;
                  const bool okc = (bclass == 1.0f && ok1) || (bclass == 2.0f && ok2);
                  ok = reach_c && reach_d && okc && !exc_lim && !v;
                }
              }
              if (ok) bits[j >> 2] |= 1u << (8 * (j & 3) + 2 * t + e);
            }
          }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          bits[k] |= __shfl_xor_sync(0xffffffffu, bits[k], 1);
          bits[k] |= __shfl_xor_sync(0xffffffffu, bits[k], 2);
        }
        if (kEnv != RRNCO_ENV_ATSP) {
          const bool any_cust = ((bits[0] & ~1u) | bits[1] | bits[2] | bits[3]) != 0u;
          if (!(cur == 0 && any_cust)) bits[0] |= 1u;
        }
        if ((bits[0] | bits[1] | bits[2] | bits[3]) == 0u) {  // cannot happen upstream; keep the math finite
          if (t == 0 && sm.active[row] && !sm.done[row]) atomicOr(p.status, RRNCO_DEV_NO_FEASIBLE);
          bits[0] |= 1u;
        }
        sm.mask[row][t] = t == 0 ? bits[0] : t == 1 ? bits[1] : t == 2 ? bits[2] : bits[3];
      }
    }
    if (kTc) {
      if (tid == 0) TL(step, 1);  // step start (after the all-done vote)
      // ---- A (tcgen05): lane = (rollout of the warp's 16, 64-wide half of the columns): the action-mask words of
      // that half, then the query rows -> fp16 hi | lo core-matrix tiles (A operand of Q K^T) in the A region with
      // conflict-free 16-byte tile stores.  The query source rows are requested first: their L2 latency hides under the mask.
      {
        uint16_t* q_hi = reinterpret_cast<uint16_t*>(sm.A);
        uint16_t* q_lo = q_hi + kRows * kE;
        const int row = warp * 16 + (lane & 15), dh = lane >> 4;
        const int cur = sm.cur[row];
        float st[kMaxState] = {0.f, 0.f, 0.f, 0.f};
        const float f0 = sm.f[0][row], f1 = sm.f[1][row], f2 = sm.f[2][row], f3 = sm.f[3][row];
        const float* src1;
        const float* src2 = nullptr;
        if (kEnv == RRNCO_ENV_ATSP) {
          if (p.use_placeholder && step == 0) {
            src1 = sm.placeholder;
          } else {
            src1 = P1 + (size_t)sm.first[row] * kE;
            src2 = P2 + (size_t)cur * kE;
          }
        } else {
          src1 = P1 + (size_t)cur * kE;
          if (kEnv == RRNCO_ENV_RCVRP) {
            st[0] = __fsub_rn(cap, f0);
          } else {
            const float used = f3 == 0.f ? f2 : f3;
            st[0] = __fsub_rn(cap, used);
            st[1] = f0;
            st[2] = closed == 0.f ? 1.f : 0.f;
            float rem = __fsub_rn(limit, f1);  // nan_to_num(limit - route, posinf=10)
            rem = rem == INFINITY ? 10.f : (rem != rem ? 0.f : (rem == -INFINITY ? -3.4028234663852886e38f : rem));
            st[3] = rem;
          }
        }
        // action mask (rcvrp/env.py:183-195, rmtvrp/env.py:343-428, atsp/env.py:107-111): words 2 dh, 2 dh + 1
        uint32_t bits2[2];
        float4 pq[16];
        {
          const uint2 visw = *reinterpret_cast<const uint2*>(&sm.vis[row][2 * dh]);
          bool missing = false, carrying_b = false;
          if (kEnv == RRNCO_ENV_RCVRPTW) {
            uint32_t m = (sm.lhmask[2 * dh] & ~visw.x) | (sm.lhmask[2 * dh + 1] & ~visw.y);
            m |= __shfl_xor_sync(0xffffffffu, m, 16);
            missing = m != 0u;  // linehauls_missing
            carrying_b = sm.demb[cur] > 0.f;
          }
            // query source rows: requested after every shared-memory read above has been consumed, so that the mask loop
            // below does not wait on their scoreboard
  #pragma unroll
          for (int cc = 0; cc < 16; ++cc) {
            pq[cc] = *reinterpret_cast<const float4*>(src1 + dh * 64 + cc * 4);
            if (kEnv == RRNCO_ENV_ATSP && src2) {
              const float4 w = __ldg(reinterpret_cast<const float4*>(src2 + dh * 64 + cc * 4));
              pq[cc] = make_float4(pq[cc].x + w.x, pq[cc].y + w.y, pq[cc].z + w.z, pq[cc].w + w.w);
            }
          }
#pragma unroll 1
          for (int k = 0; k < 2; ++k) {
            const int c0 = 64 * dh + 32 * k;
            const uint32_t valid = N >= c0 + 32 ? 0xffffffffu : (N > c0 ? (1u << (N - c0)) - 1u : 0u);
            uint32_t ok = ~(k ? visw.y : visw.x) & valid;
            if (kEnv == RRNCO_ENV_RCVRP) {
              uint32_t bad = 0u;
#pragma unroll 8
              for (int i = 0; i < 32; ++i) bad |= (__fadd_rn(sm.dem[c0 + i], f0) > cap ? 1u : 0u) << i;
              ok &= ~bad;
            } else if (kEnv == RRNCO_ENV_RCVRPTW) {
              uint32_t good = 0u;
#pragma unroll 2
              for (int i = 0; i < 32; ++i) {
                const int c = c0 + i;
                if (c < N) {
                  const float dist_ij = D[cur * N + c], dur_ij = U[cur * N + c];
                  const float arrival = __fadd_rn(f0, dur_ij);
                  const bool reach_c = arrival < sm.tw1[c];
                  const bool reach_d =
                      __fmul_rn(__fadd_rn(__fadd_rn(fmaxf(arrival, sm.tw0[c]), sm.svc[c]), sm.uj0[c]), closed) < sm.tw1[0];
                  const bool exc_lim = __fadd_rn(__fadd_rn(f1, dist_ij), __fmul_rn(sm.dj0[c], closed)) > limit;
                  const bool exc_l = __fadd_rn(sm.dem[c], f2) > cap;
                  const bool exc_b = __fadd_rn(sm.demb[c], f3) > cap;
                  const bool ok1 = (missing && !exc_l && !carrying_b && sm.dem[c] > 0.f) || (!exc_b && sm.demb[c] > 0.f);
                  const bool cannot_l = sm.dem[c] > __fsub_rn(cap, f3);
                  const bool ok2 = !exc_l && !exc_b && !cannot_l;
                  const bool okc = (bclass == 1.0f && ok1) || (bclass == 2.0f && ok2);
                  good |= (reach_c && reach_d && okc && !exc_lim ? 1u : 0u) << i;
                }
              }
              ok &= good;
            }
            if (kEnv != RRNCO_ENV_ATSP && c0 == 0) ok &= ~1u;  // the depot bit is decided below
            bits2[k] = ok;
          }
          if (kEnv != RRNCO_ENV_ATSP) {
            uint32_t any_cust = bits2[0] | bits2[1];
            any_cust |= __shfl_xor_sync(0xffffffffu, any_cust, 16);
            if (dh == 0 && !(cur == 0 && any_cust != 0u)) bits2[0] |= 1u;
          }
          uint32_t tot = bits2[0] | bits2[1];
          tot |= __shfl_xor_sync(0xffffffffu, tot, 16);
          if (tot == 0u && dh == 0) {  // cannot happen upstream; keep the math finite
            if (sm.active[row] && !sm.done[row]) atomicOr(p.status, RRNCO_DEV_NO_FEASIBLE);
            bits2[0] |= 1u;
          }
          *reinterpret_cast<uint2*>(&sm.mask[row][2 * dh]) = make_uint2(bits2[0], bits2[1]);
        }
        PHASE_STAMP(15);
        if (tid == 0) TL(step, 3);  // mask words written
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) {
          const int c8 = dh * 8 + cc;
          float4 v0 = pq[2 * cc], v1 = pq[2 * cc + 1];
          if (kEnv != RRNCO_ENV_ATSP) {
#pragma unroll
            for (int k = 0; k < kMaxState; ++k) {
              if (k < p.n_state) {
                const float4 w0 = *reinterpret_cast<const float4*>(&sm.wstate[k][c8 * 8]);
                const float4 w1 = *reinterpret_cast<const float4*>(&sm.wstate[k][c8 * 8 + 4]);
                v0.x = fmaf(st[k], w0.x, v0.x); v0.y = fmaf(st[k], w0.y, v0.y);
                v0.z = fmaf(st[k], w0.z, v0.z); v0.w = fmaf(st[k], w0.w, v0.w);
                v1.x = fmaf(st[k], w1.x, v1.x); v1.y = fmaf(st[k], w1.y, v1.y);
                v1.z = fmaf(st[k], w1.z, v1.z); v1.w = fmaf(st[k], w1.w, v1.w);
              }
            }
          }
          uint32_t h[4], l[4];
          f16s_split2(v0.x, v0.y, kAScale, h[0], l[0]); f16s_split2(v0.z, v0.w, kAScale, h[1], l[1]);
          f16s_split2(v1.x, v1.y, kAScale, h[2], l[2]); f16s_split2(v1.z, v1.w, kAScale, h[3], l[3]);
          const int dst = c8 * (kRows * 8) + row * 8;
          *reinterpret_cast<uint4*>(&q_hi[dst]) = make_uint4(h[0], h[1], h[2], h[3]);
          *reinterpret_cast<uint4*>(&q_lo[dst]) = make_uint4(l[0], l[1], l[2], l[3]);
        }
      }
      tc05::fence_proxy_async();
      tc05::fence_before_sync();
      tc05::mbar_arrive(&sm.bar_q);
      if (tid == 0) TL(step, 2);  // mask + query done
      cta_sync<kTc>();  // action-mask bitsets visible to the row-owner threads
      PHASE_STAMP(0);

      // ---- C (tcgen05): attention.  Scores of head h arrive in a TMEM buffer (lane = rollout); the thread that owns
      // (rollout, head group) runs the masked softmax on its row and writes the unnormalised probabilities back IN
      // PLACE as the fp16 hi | lo A operand of P V (columns 16 j .. 16 j + 7 | 16 j + 8 .. 16 j + 15 of key block j).
      // Warps 0-3 take heads 0-3, warps 4-7 heads 4-7, so a thread later normalises exactly the columns it summed.
      {
        const int row = (warp & 3) * 32 + lane, grp = warp >> 2;
        const uint32_t tb = sm.tmem_base, lane_b = (uint32_t)((warp & 3) * 32) << 16;
        const int R16a = ((N + 15) >> 4) << 4;
        // s = q . k / 4; the operands carry kAScale kKvScale.  exp(s - m) = ex2(c1 v - c1 vmax); + 4 = log2(kAScale)
        const float c1 = 0.25f * 1.4426950408889634f / (kAScale * kKvScale);
        const int nblk = (R16a + 31) >> 5;  // 32-column blocks; columns past R16 hold stale data that the mask zeroes
        // Rolled loops on purpose: the decode-step body is far larger than the instruction cache, and every unrolled
        // copy of this code is fetched from L2 once per step (stall_no_inst was > 50 % of this phase when unrolled).
#pragma unroll 1
        for (int j = 0; j < 4; ++j) {
          const int h = 4 * grp + j, k = 2 * j + grp;
          const uint32_t t_s = tb + (uint32_t)(k % 3) * 128u + lane_b;
          if ((tid & 127) == 0) TL(step, 10 + h);  // group waits for scores h
          tc05::mbar_wait(&sm.bar_s[h], tc_step_par, 20);
          tc05::fence_after_sync();
          if ((tid & 127) == 0) TL(step, 20 + h);  // scores h seen
          PHASE_STAMP(11);
          // pass 1: row maximum over the feasible keys (four independent partial maxima).  A TMEM load costs ~230
          // cycles round trip: 64 columns per wait (columns past R16 hold stale data that the mask ignores).
          float vm[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll 1
          for (int gb = 0; gb < nblk; gb += 2) {
            uint32_t v[4][16];
#pragma unroll
            for (int u = 0; u < 4; ++u) tc05::tmem_ld16(t_s + gb * 32 + u * 16, v[u]);
            const uint2 mw2 = *reinterpret_cast<const uint2*>(&sm.mask[row][gb]);
            tc05::tmem_wait_ld();
#pragma unroll
            for (int i = 0; i < 64; ++i)
              vm[i & 3] = fmaxf(vm[i & 3], (((i < 32 ? mw2.x : mw2.y) >> (i & 31)) & 1u) ? __uint_as_float(v[i >> 4][i & 15]) : -INFINITY);
          }
          const float off = fmaf(-c1, fmaxf(fmaxf(vm[0], vm[1]), fmaxf(vm[2], vm[3])), 4.0f);
          PHASE_STAMP(12);
          // pass 2: p = exp(s - max) (x kAScale), row sum, fp16 hi | lo split written back in place.  Software
          // pipelined over 32-column blocks: the load of block gb + 1 is in flight while block gb is processed.
          float sum0 = 0.f, sum1 = 0.f;
          auto exp_block = [&](const uint32_t (&v)[2][16], int gb) {
            const uint32_t mw = sm.mask[row][gb];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              uint32_t w[16];  // [hi (8 words) | lo (8 words)] of key block 2 gb + u
#pragma unroll
              for (int i = 0; i < 16; i += 2) {
                const float e0 = ex2a(fmaf(c1, __uint_as_float(v[u][i]), off));
                const float e1 = ex2a(fmaf(c1, __uint_as_float(v[u][i + 1]), off));
                const float p0 = ((mw >> (16 * u + i)) & 1u) ? e0 : 0.f;
                const float p1 = ((mw >> (16 * u + i + 1)) & 1u) ? e1 : 0.f;
                sum0 += p0;
                sum1 += p1;
                f16s_split2(p0, p1, 1.0f, w[i >> 1], w[8 + (i >> 1)]);
              }
              tc05::tmem_st16(t_s + gb * 32 + u * 16, w);
            }
          };
          uint32_t va[2][16], vb[2][16];
          tc05::tmem_ld16(t_s, va[0]);
          tc05::tmem_ld16(t_s + 16, va[1]);
#pragma unroll 1
          for (int gb = 0; gb < nblk; gb += 2) {
            tc05::tmem_wait_ld();
            if (gb + 1 < nblk) {
              tc05::tmem_ld16(t_s + (gb + 1) * 32, vb[0]);
              tc05::tmem_ld16(t_s + (gb + 1) * 32 + 16, vb[1]);
            }
            exp_block(va, gb);
            if (gb + 1 < nblk) {
              tc05::tmem_wait_ld();
              if (gb + 2 < nblk) {
                tc05::tmem_ld16(t_s + (gb + 2) * 32, va[0]);
                tc05::tmem_ld16(t_s + (gb + 2) * 32 + 16, va[1]);
              }
              exp_block(vb, gb + 1);
            }
          }
          sm.xsum[h][row] = sum0 + sum1;
          tc05::tmem_wait_st();
          tc05::fence_before_sync();
          tc05::mbar_arrive(&sm.bar_p[h]);
          if ((tid & 127) == 0) TL(step, 30 + h);  // P(h) written
          PHASE_STAMP(13);
        }
        // every P V complete (all eight: the score buffers are zeroed and the K / V memory handed over below)
#pragma unroll 1
        for (int h = 0; h < kH; ++h) tc05::mbar_wait(&sm.bar_o[h], tc_step_par, 20);
        tc05::fence_after_sync();
        if ((tid & 127) == 0) TL(step, 40 + grp);  // all PV seen
        PHASE_STAMP(14);
        // glimpse = heads / sum + q (decoder.py:292-293) -> fp16 hi | lo tiles of the FFN, in place over the query tiles
        uint16_t* g_hi = reinterpret_cast<uint16_t*>(sm.A);
        uint16_t* g_lo = g_hi + kRows * kE;
#pragma unroll 1
        for (int j = 0; j < 4; ++j) {
          const int h = 4 * grp + j;
          uint32_t o[16];
          tc05::tmem_ld16(tb + 384 + 16 * h + lane_b, o);
          const float inv = __fdividef(1.0f, kKvScale * sm.xsum[h][row]);
          tc05::tmem_wait_ld();
#pragma unroll
          for (int cc = 0; cc < 2; ++cc) {
            const int offq = (2 * h + cc) * (kRows * 8) + row * 8;
            const uint4 qh = *reinterpret_cast<const uint4*>(&g_hi[offq]);
            const uint4 ql = *reinterpret_cast<const uint4*>(&g_lo[offq]);
            const uint32_t qhw[4] = {qh.x, qh.y, qh.z, qh.w}, qlw[4] = {ql.x, ql.y, ql.z, ql.w};
            uint32_t hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&qhw[e]));
              const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&qlw[e]));
              const float g0 = fmaf(__uint_as_float(o[cc * 8 + 2 * e]), inv, (fh.x + fl.x) * (1.0f / kAScale));
              const float g1 = fmaf(__uint_as_float(o[cc * 8 + 2 * e + 1]), inv, (fh.y + fl.y) * (1.0f / kAScale));
              f16s_split2(g0, g1, kAScale, hi[e], lo[e]);
            }
            *reinterpret_cast<uint4*>(&g_hi[offq]) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(&g_lo[offq]) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          }
        }
        {  // the three score buffers become the (pre-zeroed) accumulators of the FFN
          uint32_t z[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) z[i] = 0u;
#pragma unroll
          for (int q = 0; q < 12; ++q) tc05::tmem_st16(tb + lane_b + (q >> 2) * 128 + grp * 64 + (q & 3) * 16, z);
          tc05::tmem_wait_st();
        }
      }
      tc05::fence_proxy_async();
      tc05::fence_before_sync();
      tc05::mbar_arrive(&sm.bar_go);      // K / V tiles are dead: the producer starts this step's weight stream
      tc05::mbar_arrive(&sm.bar_gready);  // glimpse tiles written: GEMM1 may start
      if ((tid & 127) == 0) TL(step, 42 + (warp >> 2));  // glimpse written
      PHASE_STAMP(1);
    } else {
      // ---- A2: query rows q = ctx_node_proj[cur] (+ proj2[...]) + sum_k state_k * wstate[k] ------
  #pragma unroll 4
      for (int i = 0; i < 16; ++i) {
        const int row = warp * 16 + i;
        const int cur = sm.cur[row];
        float4 q;
        if (kEnv == RRNCO_ENV_ATSP) {
          if (p.use_placeholder && step == 0) {
            q = *reinterpret_cast<const float4*>(&sm.placeholder[lane * 4]);
          } else {
            const float4 a4 = __ldg(reinterpret_cast<const float4*>(P1 + (size_t)sm.first[row] * kE) + lane);
            const float4 c4 = __ldg(reinterpret_cast<const float4*>(P2 + (size_t)cur * kE) + lane);
            q = make_float4(a4.x + c4.x, a4.y + c4.y, a4.z + c4.z, a4.w + c4.w);
          }
        } else {
          q = __ldg(reinterpret_cast<const float4*>(P1 + (size_t)cur * kE) + lane);
          float st[kMaxState];
          if (p.logits_only) {
  #pragma unroll
            for (int k = 0; k < kMaxState; ++k) st[k] = sm.f[k][row];
          } else if (kEnv == RRNCO_ENV_RCVRP) {
            st[0] = __fsub_rn(cap, sm.f[0][row]);
            st[1] = st[2] = st[3] = 0.f;
          } else {
            const float used = sm.f[3][row] == 0.f ? sm.f[2][row] : sm.f[3][row];
            st[0] = __fsub_rn(cap, used);
            st[1] = sm.f[0][row];
            st[2] = closed == 0.f ? 1.f : 0.f;
            float rem = __fsub_rn(limit, sm.f[1][row]);  // nan_to_num(limit - route, posinf=10)
            rem = rem == INFINITY ? 10.f : (rem != rem ? 0.f : (rem == -INFINITY ? -3.4028234663852886e38f : rem));
            st[3] = rem;
          }
  #pragma unroll
          for (int k = 0; k < kMaxState; ++k) {
            if (k < p.n_state) {
              const float4 w4 = *reinterpret_cast<const float4*>(&sm.wstate[k][lane * 4]);
              q.x = fmaf(st[k], w4.x, q.x); q.y = fmaf(st[k], w4.y, q.y);
              q.z = fmaf(st[k], w4.z, q.z); q.w = fmaf(st[k], w4.w, q.w);
            }
          }
        }
        *reinterpret_cast<float4*>(&sm.A[row * kLdA + lane * 4]) = q;
      }
      cp_async_wait<0>();
      cta_sync<kTc>();
      PHASE_STAMP(0);

      // ---- C: attention, 16 rows x 8 heads per warp ----------------------------------------------
      {
        uint32_t m0[4], m1[4];
        *reinterpret_cast<uint4*>(m0) = *reinterpret_cast<const uint4*>(sm.mask[r0]);
        *reinterpret_cast<uint4*>(m1) = *reinterpret_cast<const uint4*>(sm.mask[r1]);
        const float* sK = sm.Hb;
        const float* sV = sm.Bs;
  #pragma unroll 1
        for (int h = 0; h < kH; ++h) {
          uint32_t ah[2][4], al[2][4];
  #pragma unroll
          for (int ks = 0; ks < 2; ++ks) {
            const int k0 = h * kDh + ks * 8 + t;
            split_tf32(sm.A[r0 * kLdA + k0], ah[ks][0], al[ks][0]);
            split_tf32(sm.A[r1 * kLdA + k0], ah[ks][1], al[ks][1]);
            split_tf32(sm.A[r0 * kLdA + k0 + 4], ah[ks][2], al[ks][2]);
            split_tf32(sm.A[r1 * kLdA + k0 + 4], ah[ks][3], al[ks][3]);
          }
          float sc[kNTMax][4];
  #pragma unroll
          for (int j = 0; j < kNTMax; ++j) {
            sc[j][0] = sc[j][1] = sc[j][2] = sc[j][3] = 0.f;
            if (j < NT) {
  #pragma unroll
              for (int ks = 0; ks < 2; ++ks) {
                const float* kp = sK + (8 * j + g) * kLdA + h * kDh + ks * 8 + t;
                uint32_t bh[2], bl[2];
                split_tf32(kp[0], bh[0], bl[0]);
                split_tf32(kp[4], bh[1], bl[1]);
                mma_x<kPasses>(sc[j], ah[ks], al[ks], bh, bl);
              }
            }
          }
          // masked softmax over the keys (scale 1/sqrt(16) is a power of two: exact)
          float mx0 = -INFINITY, mx1 = -INFINITY;
  #pragma unroll
          for (int j = 0; j < kNTMax; ++j) {
            if (j < NT) {
  #pragma unroll
              for (int e = 0; e < 2; ++e) {
                sc[j][e] = bit_of(m0, j, 2 * t + e) ? sc[j][e] * 0.25f : -INFINITY;
                sc[j][2 + e] = bit_of(m1, j, 2 * t + e) ? sc[j][2 + e] * 0.25f : -INFINITY;
                mx0 = fmaxf(mx0, sc[j][e]);
                mx1 = fmaxf(mx1, sc[j][2 + e]);
              }
            }
          }
          mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
          mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
          mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
          mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
          float sum0 = 0.f, sum1 = 0.f;
  #pragma unroll
          for (int j = 0; j < kNTMax; ++j) {
            if (j < NT) {
  #pragma unroll
              for (int e = 0; e < 2; ++e) {
                sc[j][e] = fexp(sc[j][e] - mx0);
                sc[j][2 + e] = fexp(sc[j][2 + e] - mx1);
                sum0 += sc[j][e];
                sum1 += sc[j][2 + e];
              }
            }
          }
          sum0 += __shfl_xor_sync(0xffffffffu, sum0, 1);
          sum0 += __shfl_xor_sync(0xffffffffu, sum0, 2);
          sum1 += __shfl_xor_sync(0xffffffffu, sum1, 1);
          sum1 += __shfl_xor_sync(0xffffffffu, sum1, 2);
          // heads = P V_h: the accumulator tile j IS the A fragment of k-step j under the key permutation
          // k = t -> key 8j + 2t, k = t + 4 -> key 8j + 2t + 1 (applied to the V rows below).
          float o[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  #pragma unroll
          for (int j = 0; j < kNTMax; ++j) {
            if (j < NT) {
              uint32_t ph[4], pl[4];
              split_tf32(sc[j][0], ph[0], pl[0]);
              split_tf32(sc[j][2], ph[1], pl[1]);
              split_tf32(sc[j][1], ph[2], pl[2]);
              split_tf32(sc[j][3], ph[3], pl[3]);
  #pragma unroll
              for (int dd = 0; dd < 2; ++dd) {
                const float* vp = sV + (8 * j + 2 * t) * kLdA + h * kDh + dd * 8 + g;
                uint32_t bh[2], bl[2];
                split_tf32(vp[0], bh[0], bl[0]);
                split_tf32(vp[kLdA], bh[1], bl[1]);
                mma_x<kPasses>(o[dd], ph, pl, bh, bl);
              }
            }
          }
          const float inv0 = 1.0f / sum0, inv1 = 1.0f / sum1;
  #pragma unroll
          for (int dd = 0; dd < 2; ++dd) {
            const int col = h * kDh + dd * 8 + 2 * t;
            float2* g0 = reinterpret_cast<float2*>(&sm.A[r0 * kLdA + col]);
            float2* g1 = reinterpret_cast<float2*>(&sm.A[r1 * kLdA + col]);
            float2 q0 = *g0, q1 = *g1;
            q0.x += o[dd][0] * inv0; q0.y += o[dd][1] * inv0;
            q1.x += o[dd][2] * inv1; q1.y += o[dd][3] * inv1;
            *g0 = q0;  // glimpse = heads + q  (decoder.py:292-293), in place: these columns are only read
            *g1 = q1;  // by head h of this warp, whose A fragments are already in registers
          }
          __syncwarp();
        }
      }
      if (kTc) tc05::fence_proxy_async();  // generic-proxy reads of the V tile precede the TMA writes into the same memory
      cta_sync<kTc>();  // all warps done with the K / V tiles; glimpse complete in A
      PHASE_STAMP(1);

    }

    // ---- E: FFN  g' = W2 relu(W1 g + b1) + b2 + g ---------------------------------------------
    int sl = 0;
    if (kTc) {
      // tcgen05 path (see ffn_tc_kernel.cu for the standalone form): glimpse = fp16 hi | lo K-major core-matrix
      // tiles in the A region, weights streamed by the TMA producer warp through the Hb | Bs regions, accumulators and
      // the hidden activations (A operand of GEMM2) in tensor memory, MMAs issued by warps 9-11.  The compute warps
      // only run the epilogues.
      uint16_t* g_hi = reinterpret_cast<uint16_t*>(sm.A);  // [16-byte K chunk (16)][row (128)][8 halves], written by
      uint16_t* g_lo = g_hi + kRows * kE;                   // the attention epilogue (each thread re-reads its own part)
      const int R16 = ((N + 15) >> 4) << 4;  // rows of the logit-key tile = N of the logits MMA (multiple of 16)
      const uint32_t tbase = sm.tmem_base;
      const uint32_t t_hacc = tbase, t_oacc = tbase + 256, t_hhi = tbase + 384, t_hlo = tbase + 448;
      const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
      const int colhalf = warp >> 2;
      constexpr float kUnscaleW = 1.0f / (kAScale * kWScale), kUnscaleL = 1.0f / (kAScale * kLkScale);
      float nonfinite = 0.f;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        // hidden chunk c: + b1, relu, split -> A operand (hi | lo, fp16) of GEMM2 in tensor memory
        tc05::mbar_wait(&sm.bar_h[c & 1], (c >> 1) & 1, 32);
        if (tid == 0) TL(step, 50 + c);  // hidden chunk c seen
        if (c > 0) tc05::mbar_wait(&sm.bar_g2, (c - 1) & 1, 32);  // GEMM2(c - 1) has consumed the previous A operand
        tc05::fence_after_sync();
        const uint32_t t_h = t_hacc + (c & 1) * 128;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int col0 = colhalf * 64 + q * 16;
          uint32_t v[16], hi[8], lo[8];
          tc05::tmem_ld16(t_h + lane_base + col0, v);
          tc05::tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            const float h0 = fmaxf(fmaf(__uint_as_float(v[i]), kUnscaleW, sm.b1[c * kFRows + col0 + i]), 0.f);
            const float h1 = fmaxf(fmaf(__uint_as_float(v[i + 1]), kUnscaleW, sm.b1[c * kFRows + col0 + i + 1]), 0.f);
            // the ReLU would swallow a NaN (fp16 operand overflow upstream of here, ffn_pack.cuh): x * 0 keeps it
            nonfinite = fmaf(__uint_as_float(v[i]), 0.0f, fmaf(__uint_as_float(v[i + 1]), 0.0f, nonfinite));
            f16s_split2(h0, h1, kAScale, hi[i >> 1], lo[i >> 1]);
          }
          tc05::tmem_st8(t_hhi + lane_base + (col0 >> 1), hi);
          tc05::tmem_st8(t_hlo + lane_base + (col0 >> 1), lo);
          if (c < 3) {  // re-zero the chunk accumulator for GEMM1(c + 2) / the logits (c == 2)
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = 0u;
            tc05::tmem_st16(t_h + lane_base + col0, v);
          }
        }
        tc05::tmem_wait_st();
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_epi);
        if (tid == 0) TL(step, 54 + c);  // epilogue 1 of chunk c done
      }
      if (nonfinite != 0.f) atomicOr(p.status, RRNCO_DEV_NAN_LOGITS);  // NaN != 0
      tc05::mbar_wait(&sm.bar_g2, 1, 32);  // GEMM2(3): FFN output complete, ring memory idle
      tc05::fence_after_sync();
      if (tid == 0) TL(step, 58);  // FFN output seen
      PHASE_STAMP(3);
      // ---- output epilogue (thread per row): g' = acc + b2 + g  ->  split -> TMEM as the A operand of the logits GEMM
      {
        const int row = (warp & 3) * 32 + lane;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int col0 = colhalf * 64 + q * 16;
          uint32_t v[16], hi[8], lo[8];
          tc05::tmem_ld16(t_oacc + lane_base + col0, v);
          tc05::tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 16; i += 8) {
            const int off = ((col0 + i) >> 3) * (kRows * 8) + row * 8;  // residual g = (hi + lo) / kAScale, exact to 2^-24
            const uint4 gh = *reinterpret_cast<const uint4*>(&g_hi[off]);
            const uint4 gl = *reinterpret_cast<const uint4*>(&g_lo[off]);
            const uint32_t ghw[4] = {gh.x, gh.y, gh.z, gh.w}, glw[4] = {gl.x, gl.y, gl.z, gl.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&ghw[e]));
              const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&glw[e]));
              const float o0 = fmaf(__uint_as_float(v[i + 2 * e]), kUnscaleW, sm.b2[col0 + i + 2 * e]) +
                               (fh.x + fl.x) * (1.0f / kAScale);
              const float o1 = fmaf(__uint_as_float(v[i + 2 * e + 1]), kUnscaleW, sm.b2[col0 + i + 2 * e + 1]) +
                               (fh.y + fl.y) * (1.0f / kAScale);
              f16s_split2(o0, o1, kAScale, hi[(i >> 1) + e], lo[(i >> 1) + e]);
            }
          }
          tc05::tmem_st8(t_hhi + lane_base + (col0 >> 1), hi);
          tc05::tmem_st8(t_hlo + lane_base + (col0 >> 1), lo);
        }
      }
      tc05::tmem_wait_st();
      tc05::fence_before_sync();
      tc05::mbar_arrive(&sm.bar_lk);
      if (tid == 0) TL(step, 59);  // g' written
      PHASE_STAMP(4);

      // bias rows of the rollouts (alpha . D[cur,:] + beta . Dur[cur,:]) -> fp32 tile in the Bs region (idle: the weight
      // ring is drained, the logit keys sit in Hb) while the logits MMAs run: coalesced, one warp per 16 rollouts.
      {
        float* btile = sm.Bs;
#pragma unroll 4
        for (int i = 0; i < 16; ++i) {
          const int row_s = warp * 16 + i;
          const int cur_s = sm.cur[row_s];
#pragma unroll
          for (int cq = 0; cq < 4; ++cq) {
            const int c = cq * 32 + lane;
            float bias = 0.f;
            if (c < N) {
              bias = __fmul_rn(p.w.alpha, D[cur_s * N + c]);
              if (kEnv == RRNCO_ENV_RCVRPTW) bias = __fadd_rn(bias, __fmul_rn(p.w.beta, U[cur_s * N + c]));
            }
            btile[row_s * kLdA + c] = bias;
          }
        }
      }
      cta_sync<kTc>();
      tc05::mbar_wait(&sm.bar_acc, tc_step_par, 32);
      tc_step_par ^= 1u;
      tc05::fence_after_sync();
      if (tid == 0) TL(step, 60);  // logits seen
      PHASE_STAMP(5);

      // ---- select epilogue, thread per row: two threads own one rollout, 16-column groups dealt round-robin ----
      // Three rolled passes over the logits, which stay in TMEM (pass A rewrites them in place): the decode-step body is
      // several times the instruction cache, so code size costs more than the extra TMEM round trips.
      {
        const int row = (warp & 3) * 32 + lane;
        const int64_t rg = (int64_t)(tile * kRows + (sm.active[row] ? row : 0)) * p.n_inst + b;
        const float inv_sqrt_e = 0.08838834764831845f * kUnscaleL;  // 1 / sqrt(128), and the operand scales undone
        const float clip = p.w.tanh_clipping;
        const int hsh = 16 * colhalf;  // this thread's columns: 32 q + hsh + i
        const uint32_t t_l = t_hacc + lane_base + hsh;
        const int nq = (R16 - hsh + 31) >> 5;  // 16-column groups of this thread (warp-uniform)
        const float* brow = sm.Bs + row * kLdA + hsh;
        // pass A: bias, clip, mask (decoder.py:198-204) -> TMEM, running maximum
        float mxl = -INFINITY;
        bool nan_seen = false;
#pragma unroll 1
        for (int q = 0; q < nq; ++q) {
          uint32_t v[16];
          tc05::tmem_ld16(t_l + 32 * q, v);
          float bv[16];
#pragma unroll
          for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(&bv[i]) = *reinterpret_cast<const float4*>(brow + 32 * q + i);
          const uint32_t mq = sm.mask[row][q] >> hsh;  // mask bits of columns >= N are never set
          tc05::tmem_wait_ld();
          if (clip > 0.f) {
            // clip * tanh(log u), u = exp(l - bias) + 1e-6 (decoder.py:198-201), as clip * (1 - 2 / (u^2 + 1)):
            // two SFU operations per element instead of four (this pass is SFU-bound)
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float l = __uint_as_float(v[i]) * inv_sqrt_e;
              nan_seen |= !(fabsf(l) <= 3.0e38f);  // NaN, or an fp16 operand overflow (ffn_pack.cuh)
              const float u = __fadd_rn(fexp(__fsub_rn(l, bv[i])), 1e-6f);
              const float th = fmaf(-2.0f, rcpa(fmaf(u, u, 1.0f)), 1.0f);
              v[i] = __float_as_uint(((mq >> i) & 1u) ? __fmul_rn(th, clip) : -INFINITY);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              float l = __uint_as_float(v[i]) * inv_sqrt_e;
              nan_seen |= !(fabsf(l) <= 3.0e38f);
              l = flog(__fadd_rn(fexp(__fsub_rn(l, bv[i])), 1e-6f));
              v[i] = __float_as_uint(((mq >> i) & 1u) ? l : -INFINITY);
            }
          }
          if (p.w.temperature != 1.0f) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __float_as_uint(__fdiv_rn(__uint_as_float(v[i]), p.w.temperature));
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) mxl = fmaxf(mxl, __uint_as_float(v[i]));
          tc05::tmem_st16(t_l + 32 * q, v);
          if (kFilter) {  // the values also overwrite this thread's own columns of the bias tile (read by filter_cut below)
#pragma unroll
            for (int i = 0; i < 16; i += 4)
              *reinterpret_cast<uint4*>(const_cast<float*>(brow) + 32 * q + i) = make_uint4(v[i], v[i + 1], v[i + 2], v[i + 3]);
          }
        }
        {  // the O tile of the next step's attention accumulates: zero it
          uint32_t z[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) z[i] = 0u;
#pragma unroll
          for (int q = 0; q < 4; ++q) tc05::tmem_st16(tbase + 384 + lane_base + colhalf * 64 + q * 16, z);
        }
        tc05::tmem_wait_st();
        PHASE_STAMP(7);
        if (nan_seen) atomicOr(p.status, RRNCO_DEV_NAN_LOGITS);
        sm.xf[0][colhalf][row] = mxl;
        cta_sync<kTc>();
        float cut = -INFINITY;  // top-k / top-p: both threads of the row find the same cut over the row's values
        if (kFilter) {
          cut = filter_cut(FilterRowLocal{sm.Bs + row * kLdA, R16}, p.top_k, p.top_p,
                           fmaxf(sm.xf[0][0][row], sm.xf[0][1][row]));
          cta_sync<kTc>();
        }
        // bias tile and logit-key tiles are dead: the producer may load the packed K / V tiles of the next decode step
        if (tid == 0) tc05::mbar_arrive(&sm.bar_kvgo);
        const float mx = fmaxf(sm.xf[0][0][row], sm.xf[0][1][row]);
        // pass B: softmax denominator
        float sel = 0.f;
#pragma unroll 1
        for (int q = 0; q < nq; ++q) {
          uint32_t v[16];
          tc05::tmem_ld16(t_l + 32 * q, v);
          tc05::tmem_wait_ld();
          if (kFilter) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(v[i]) < cut ? __float_as_uint(-INFINITY) : v[i];
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) sel += fexp(__uint_as_float(v[i]) - mx);
        }
        sm.xf[1][colhalf][row] = sel;
        cta_sync<kTc>();
        PHASE_STAMP(8);
        const float se = flog(sm.xf[1][0][row] + sm.xf[1][1][row]);
        // pass C: log-softmax in the reference's order; argmax of log p (greedy) or of log p + Gumbel noise (sampling);
        // evaluate: log p of the forced action
        int forced = -1;
        if (p.mode == RRNCO_DECODE_EVALUATE) {
          forced = step < p.forced_T ? (int)p.forced[rg * p.forced_T + step] : 0;
          forced = min(max(forced, 0), N - 1);
        }
        float best = -INFINITY, bestlp = -INFINITY;
        int besti = 0x7fffffff;
        const uint2 key2 = make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32));
#pragma unroll 1
        for (int q = 0; q < nq; ++q) {
          uint32_t v[16];
          tc05::tmem_ld16(t_l + 32 * q, v);
          tc05::tmem_wait_ld();
          if (kFilter) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(v[i]) < cut ? __float_as_uint(-INFINITY) : v[i];
          }
          const int cbase = 32 * q + hsh;
          if (p.mode == RRNCO_DECODE_SAMPLING) {
#pragma unroll 1
            for (int i4 = 0; i4 < 16; i4 += 4) {
              const float4 gn = gumbel4(make_uint4((uint32_t)rg, (uint32_t)(rg >> 32), (uint32_t)step, (uint32_t)((cbase + i4) >> 2)), key2);
              const float gv[4] = {gn.x, gn.y, gn.z, gn.w};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                // v[] is indexed dynamically here only through the unrolled selects below
                const uint32_t raw = i4 == 0 ? v[e] : i4 == 4 ? v[4 + e] : i4 == 8 ? v[8 + e] : v[12 + e];
                const float lpv = __fsub_rn(__fsub_rn(__uint_as_float(raw), mx), se);
                const float key = lpv + gv[e];
                const bool better = key > best;
                best = better ? key : best;
                bestlp = better ? lpv : bestlp;
                besti = better ? cbase + i4 + e : besti;
              }
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float lpv = __fsub_rn(__fsub_rn(__uint_as_float(v[i]), mx), se);
              const bool better = lpv > best;
              best = better ? lpv : best;
              besti = better ? cbase + i : besti;
              if (cbase + i == forced) bestlp = lpv;
            }
          }
        }
        if (p.mode == RRNCO_DECODE_GREEDY) bestlp = best;
        sm.xf[2][colhalf][row] = best;
        sm.xf[0][colhalf][row] = bestlp;  // xf[0] (row maxima) was last read before the previous barrier
        sm.xi[colhalf][row] = besti;
        cta_sync<kTc>();
        if (tid == 0) TL(step, 63);  // select passes done
        PHASE_STAMP(9);
        int act = sm.xi[0][row];  // larger key wins, ties -> lower index
        int win = 0;
        if (sm.xf[2][1][row] > sm.xf[2][0][row] || (sm.xf[2][1][row] == sm.xf[2][0][row] && sm.xi[1][row] < act)) win = 1;
        act = sm.xi[win][row];
        if (act == 0x7fffffff) act = 0;
        if (p.mode == RRNCO_DECODE_EVALUATE) {
          act = forced;
          win = (act >> 4) & 1;  // the half that owns the forced column recorded its log p
        }
        const float chosen = sm.xf[0][win][row];
        uint32_t mrow[4];
        *reinterpret_cast<uint4*>(mrow) = *reinterpret_cast<const uint4*>(sm.mask[row]);
        PHASE_STAMP(10);
        if (colhalf == 0) {
          const bool feasible = (mrow[act >> 5] >> (act & 31)) & 1u;
          if (!feasible && sm.active[row]) atomicOr(p.status, RRNCO_DEV_INFEASIBLE);
          const bool count_leg = kEnv != RRNCO_ENV_ATSP || t_out > 0;
          transition<kEnv>(sm, p, row, act, D, U, cap, closed, count_leg);
          if (kEnv == RRNCO_ENV_ATSP && t_out == 0) sm.first[row] = act;
          if (tid == 0) TL(step, 64);  // transition done
          sm.lp[row] += (double)chosen;
          if (sm.active[row] && t_out < p.t_cap) {
            p.actions[rg * p.t_cap + t_out] = act;
            if (p.logprob) p.logprob[rg * p.t_cap + t_out] = chosen;
          }
#ifdef RRNCO_DEBUG_PRINT
          if (blockIdx.x == 0 && row < 2 && step < 3)
            printf("dbg row %d step %d t_out %d act %d rg %lld t_cap %d active %d chosen %f ptr %p\n", row, step, t_out, act,
                   (long long)rg, p.t_cap, sm.active[row], chosen, (void*)p.actions);
#endif
        }
      }
    } else {
      issue_slice(0, sm, p, Lk, tid);
      issue_slice(1, sm, p, Lk, tid);
      sl = 0;
      float acc2[2][8][4];
  #pragma unroll
      for (int mt = 0; mt < 2; ++mt)
  #pragma unroll
        for (int nt = 0; nt < 8; ++nt) acc2[mt][nt][0] = acc2[mt][nt][1] = acc2[mt][nt][2] = acc2[mt][nt][3] = 0.f;

  #pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        float acc1[2][8][4];
  #pragma unroll
        for (int mt = 0; mt < 2; ++mt)
  #pragma unroll
          for (int nt = 0; nt < 8; ++nt) acc1[mt][nt][0] = acc1[mt][nt][1] = acc1[mt][nt][2] = acc1[mt][nt][3] = 0.f;
  #pragma unroll 1
        for (int half = 0; half < 2; ++half) {
          const float* Asrc = half == 0 ? sm.A : sm.Hb;
  #pragma unroll 1
          for (int ks4 = 0; ks4 < 4; ++ks4, ++sl) {
            cp_async_wait<1>();
            cta_sync<kTc>();
            issue_slice(sl + 2, sm, p, Lk, tid);
            const float* sB = sm.Bs + (sl % kStages) * kStageFloats;
  #pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
              uint32_t ah[2][4], al[2][4];
  #pragma unroll
              for (int mt = 0; mt < 2; ++mt) {
                const float* ap = Asrc + (wm * 32 + mt * 16 + g) * kLdA + ks4 * kSliceK + kk * 8 + t;
                split_tf32(ap[0], ah[mt][0], al[mt][0]);
                split_tf32(ap[8 * kLdA], ah[mt][1], al[mt][1]);
                split_tf32(ap[4], ah[mt][2], al[mt][2]);
                split_tf32(ap[8 * kLdA + 4], ah[mt][3], al[mt][3]);
              }
  #pragma unroll
              for (int nt = 0; nt < 8; ++nt) {
                const float* bp = sB + (wn * 64 + nt * 8 + g) * kLdB + kk * 8 + t;
                uint32_t bh[2], bl[2];
                split_tf32(bp[0], bh[0], bl[0]);
                split_tf32(bp[4], bh[1], bl[1]);
                if (half == 0) {
                  mma_x<kPasses>(acc1[0][nt], ah[0], al[0], bh, bl);
                  mma_x<kPasses>(acc1[1][nt], ah[1], al[1], bh, bl);
                } else {
                  mma_x<kPasses>(acc2[0][nt], ah[0], al[0], bh, bl);
                  mma_x<kPasses>(acc2[1][nt], ah[1], al[1], bh, bl);
                }
              }
            }
          }
          if (half == 0) {
            // hidden chunk c: relu(acc1 + b1) -> Hb.  Every warp passed >= 1 barrier since it last read Hb
            // (GEMM2 of chunk c-1 / the K tile), and the next slice barrier publishes these writes.
  #pragma unroll
            for (int mt = 0; mt < 2; ++mt)
  #pragma unroll
              for (int nt = 0; nt < 8; ++nt) {
                const int col = wn * 64 + nt * 8 + 2 * t;
                const int row = wm * 32 + mt * 16 + g;
                const float bb0 = sm.b1[c * kRows + col], bb1 = sm.b1[c * kRows + col + 1];
                *reinterpret_cast<float2*>(&sm.Hb[row * kLdA + col]) =
                    make_float2(fmaxf(acc1[mt][nt][0] + bb0, 0.f), fmaxf(acc1[mt][nt][1] + bb1, 0.f));
                *reinterpret_cast<float2*>(&sm.Hb[(row + 8) * kLdA + col]) =
                    make_float2(fmaxf(acc1[mt][nt][2] + bb0, 0.f), fmaxf(acc1[mt][nt][3] + bb1, 0.f));
              }
          }
        }
      }
      // residual epilogue: g' = acc2 + b2 + g, in place (each element is read and written by one thread)
  #pragma unroll
      for (int mt = 0; mt < 2; ++mt)
  #pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          const int col = wn * 64 + nt * 8 + 2 * t;
          const int row = wm * 32 + mt * 16 + g;
          float2* g0 = reinterpret_cast<float2*>(&sm.A[row * kLdA + col]);
          float2* g1 = reinterpret_cast<float2*>(&sm.A[(row + 8) * kLdA + col]);
          float2 v0 = *g0, v1 = *g1;
          v0.x += acc2[mt][nt][0] + sm.b2[col]; v0.y += acc2[mt][nt][1] + sm.b2[col + 1];
          v1.x += acc2[mt][nt][2] + sm.b2[col]; v1.y += acc2[mt][nt][3] + sm.b2[col + 1];
          *g0 = v0;
          *g1 = v1;
        }
    }

    if (!kTc) {
      PHASE_STAMP(3);
      // ---- G: pointer logits, row-owner layout (warp = 16 rows x all keys) ------------------------
      float lg[kNTMax][4];
  #pragma unroll
      for (int j = 0; j < kNTMax; ++j) lg[j][0] = lg[j][1] = lg[j][2] = lg[j][3] = 0.f;
  #pragma unroll 1
      for (int ks4 = 0; ks4 < 4; ++ks4, ++sl) {
        cp_async_wait<1>();
        cta_sync<kTc>();  // first iteration also publishes the residual epilogue
        issue_slice(sl + 2, sm, p, Lk, tid);
        const float* sB = sm.Bs + (sl % kStages) * kStageFloats;
  #pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          uint32_t ah[4], al[4];
          const float* ap = sm.A + r0 * kLdA + ks4 * kSliceK + kk * 8 + t;
          split_tf32(ap[0], ah[0], al[0]);
          split_tf32(ap[8 * kLdA], ah[1], al[1]);
          split_tf32(ap[4], ah[2], al[2]);
          split_tf32(ap[8 * kLdA + 4], ah[3], al[3]);
  #pragma unroll
          for (int j = 0; j < kNTMax; ++j) {
            if (j < NT) {
              const float* bp = sB + (8 * j + g) * kLdB + kk * 8 + t;
              uint32_t bh[2], bl[2];
              split_tf32(bp[0], bh[0], bl[0]);
              split_tf32(bp[4], bh[1], bl[1]);
              mma_x<kPasses>(lg[j], ah, al, bh, bl);
            }
          }
        }
      }
      cp_async_wait<0>();
      PHASE_STAMP(5);

      // ---- epilogue: bias, clip, mask, log-softmax, selection, transition --------------------------
      const float inv_sqrt_e = 0.08838834764831845f;  // 1 / sqrt(128)
      const int cur0 = sm.cur[r0], cur1 = sm.cur[r1];
      bool nan_seen = false;
  #pragma unroll
      for (int j = 0; j < kNTMax; ++j) {
        if (j < NT) {
  #pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int c = 8 * j + 2 * t + (e & 1);
            const int cur = e < 2 ? cur0 : cur1;
            float l = lg[j][e] * inv_sqrt_e;
            if (c < N) {
              nan_seen |= l != l;
              float bias = __fmul_rn(p.w.alpha, D[cur * N + c]);
              if (kEnv == RRNCO_ENV_RCVRPTW) bias = __fadd_rn(bias, __fmul_rn(p.w.beta, U[cur * N + c]));
              l = flog(__fadd_rn(fexp(__fsub_rn(l, bias)), 1e-6f));  // decoder.py:198
            }
            lg[j][e] = l;
          }
        }
      }
      if (nan_seen) atomicOr(p.status, RRNCO_DEV_NAN_LOGITS);

      if (p.logits_only) {
  #pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
          const int row = rr ? r1 : r0;
          const int s = tile * kRows + row;
          if (s < p.S) {
            float* dst = p.logits_out + ((int64_t)s * p.n_inst + b) * N;
  #pragma unroll
            for (int j = 0; j < kNTMax; ++j)
              if (j < NT) {
                const int c = 8 * j + 2 * t;
                if (c < N) dst[c] = lg[j][2 * rr];
                if (c + 1 < N) dst[c + 1] = lg[j][2 * rr + 1];
              }
          }
        }
        break;
      }

      uint32_t m0[4], m1[4];
      *reinterpret_cast<uint4*>(m0) = *reinterpret_cast<const uint4*>(sm.mask[r0]);
      *reinterpret_cast<uint4*>(m1) = *reinterpret_cast<const uint4*>(sm.mask[r1]);
      float mx[2] = {-INFINITY, -INFINITY};
  #pragma unroll
      for (int j = 0; j < kNTMax; ++j) {
        if (j < NT) {
  #pragma unroll
          for (int e = 0; e < 4; ++e) {
            const bool ok = bit_of(e < 2 ? m0 : m1, j, 2 * t + (e & 1));
            float l = lg[j][e];
            if (p.w.tanh_clipping > 0.f) l = __fmul_rn(ftanh(l), p.w.tanh_clipping);  // decoding.py:342-343
            l = ok ? __fdiv_rn(l, p.w.temperature) : -INFINITY;                       // decoding.py:348-351
            lg[j][e] = l;
            mx[e >> 1] = fmaxf(mx[e >> 1], l);
          }
        }
      }
  #pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        mx[rr] = fmaxf(mx[rr], __shfl_xor_sync(0xffffffffu, mx[rr], 1));
        mx[rr] = fmaxf(mx[rr], __shfl_xor_sync(0xffffffffu, mx[rr], 2));
      }
      float se[2] = {0.f, 0.f};
  #pragma unroll
      for (int j = 0; j < kNTMax; ++j)
        if (j < NT) {
  #pragma unroll
          for (int e = 0; e < 4; ++e) se[e >> 1] += fexp(lg[j][e] - mx[e >> 1]);
        }
  #pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        se[rr] += __shfl_xor_sync(0xffffffffu, se[rr], 1);
        se[rr] += __shfl_xor_sync(0xffffffffu, se[rr], 2);
        se[rr] = flog(se[rr]);
      }
      // log-probs (x - max) - log(sum) in the reference's order; selection on them
      float best[2] = {-INFINITY, -INFINITY};
      int besti[2] = {0x7fffffff, 0x7fffffff};
      // reference-layout rollout ids (padded rows shadow the tile's first rollout)
      const int64_t rg0 = (int64_t)(tile * kRows + (sm.active[r0] ? r0 : 0)) * p.n_inst + b;
      const int64_t rg1 = (int64_t)(tile * kRows + (sm.active[r1] ? r1 : 0)) * p.n_inst + b;
  #pragma unroll
      for (int j = 0; j < kNTMax; ++j) {
        if (j < NT) {
          // Gumbel noise of (rollout r, step, column c) = Philox(key = seed; ctr = (r, step, c >> 2))[c & 3]
          uint4 rnd0 = make_uint4(0, 0, 0, 0), rnd1 = rnd0;
          if (p.mode == RRNCO_DECODE_SAMPLING) {
            const uint2 key2 = make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32));
            rnd0 = philox4x32(make_uint4((uint32_t)rg0, (uint32_t)(rg0 >> 32), (uint32_t)step, (uint32_t)(2 * j + (t >> 1))), key2);
            rnd1 = philox4x32(make_uint4((uint32_t)rg1, (uint32_t)(rg1 >> 32), (uint32_t)step, (uint32_t)(2 * j + (t >> 1))), key2);
          }
  #pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int c = 8 * j + 2 * t + (e & 1);
            const float lpv = __fsub_rn(__fsub_rn(lg[j][e], mx[e >> 1]), se[e >> 1]);
            lg[j][e] = lpv;
            float key = lpv;
            if (p.mode == RRNCO_DECODE_SAMPLING) {
              const uint4 rnd = e < 2 ? rnd0 : rnd1;
              const int comp = 2 * (t & 1) + (e & 1);
              const uint32_t x = comp == 0 ? rnd.x : comp == 1 ? rnd.y : comp == 2 ? rnd.z : rnd.w;
              key = lpv + (-logf(-logf(u01(x))));  // Gumbel-max
            }
            if (key > best[e >> 1]) {  // strict: lowest index wins ties (ascending c within a lane)
              best[e >> 1] = key;
              besti[e >> 1] = c;
            }
          }
        }
      }
  #pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
  #pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, best[rr], o);
          const int oi = __shfl_xor_sync(0xffffffffu, besti[rr], o);
          if (ov > best[rr] || (ov == best[rr] && oi < besti[rr])) {
            best[rr] = ov;
            besti[rr] = oi;
          }
        }
      }
      int act[2] = {besti[0] == 0x7fffffff ? 0 : besti[0], besti[1] == 0x7fffffff ? 0 : besti[1]};
      if (p.mode == RRNCO_DECODE_EVALUATE) {
        const bool have = step < p.forced_T;
        act[0] = have && sm.active[r0] ? (int)p.forced[rg0 * p.forced_T + step] : act[0];
        act[1] = have && sm.active[r1] ? (int)p.forced[rg1 * p.forced_T + step] : act[1];
        act[0] = min(max(act[0], 0), N - 1);
        act[1] = min(max(act[1], 0), N - 1);
      }
      // chosen log-prob: owner lane contributes, quad-sum
      float chosen[2] = {0.f, 0.f};
  #pragma unroll
      for (int j = 0; j < kNTMax; ++j)
        if (j < NT) {
  #pragma unroll
          for (int e = 0; e < 4; ++e)
            if (8 * j + 2 * t + (e & 1) == act[e >> 1]) chosen[e >> 1] = lg[j][e];
        }
  #pragma unroll
      for (int rr = 0; rr < 2; ++rr) {  // only the owner lane matched: quad-sum broadcasts its value
        chosen[rr] += __shfl_xor_sync(0xffffffffu, chosen[rr], 1);
        chosen[rr] += __shfl_xor_sync(0xffffffffu, chosen[rr], 2);
      }
      // one lane per row applies the transition and emits the outputs
      if (t < 2) {
        const int rr = t;
        const int row = rr ? r1 : r0;
        const int a = act[rr];
        const int64_t rg = rr ? rg1 : rg0;
        const bool feasible = (sm.mask[row][a >> 5] >> (a & 31)) & 1u;
        if (!feasible && sm.active[row]) atomicOr(p.status, RRNCO_DEV_INFEASIBLE);
        const bool count_leg = kEnv != RRNCO_ENV_ATSP || t_out > 0;
        transition<kEnv>(sm, p, row, a, D, U, cap, closed, count_leg);
        if (kEnv == RRNCO_ENV_ATSP && t_out == 0) sm.first[row] = a;
        sm.lp[row] += (double)chosen[rr];
        if (sm.active[row] && t_out < p.t_cap) {
          p.actions[rg * p.t_cap + t_out] = a;
          if (p.logprob) p.logprob[rg * p.t_cap + t_out] = chosen[rr];
        }
      }
    }
    ++step;
    ++t_out;
    PHASE_STAMP(6);
  }

  cp_async_wait<0>();  // a prefetch of the tcgen05 variant may still be in flight
  if (p.logits_only) return;
  // ---------------- exit: close the tours, publish per-rollout sums ----------------
  cta_sync<kTc>();
  if (tid < kRows && sm.active[tid]) {
    const int row = tid;
    const int64_t r = (int64_t)(tile * kRows + row) * p.n_inst + b;
    const int last = sm.cur[row];
    float leg;
    if (kEnv == RRNCO_ENV_ATSP) {
      leg = D[last * N + sm.first[row]];
    } else {
      leg = D[last * N];  // back to the depot (go_to = roll(go_from, -1), rcvrp/env.py:203)
      if (kEnv == RRNCO_ENV_RCVRPTW) leg = __fmul_rn(leg, closed);
    }
    p.ws_len[r] = sm.len[row] + (double)leg;
    p.ws_lp[r] = sm.lp[row];
  }
  if (tid == 0) {
    p.ws_tile_steps[blockIdx.x] = t_out;
    atomicMax(p.max_steps_out, t_out);
  }
  if (kTc) {
    if (tid == 0) {
      sm.exit_flag = 1;
      tc05::mbar_wait(&sm.bar_kv, tc_step_par);  // the K / V load for the step that will not happen must have landed
    }
    tc05::fence_before_sync();
    cta_sync<kTc>();
    if (tid < kH) tc05::mbar_arrive(&sm.bar_qkdone);  // releases the producer warp ...
    tc05::mbar_arrive(&sm.bar_q);                     // ... and the MMA-issue warps (both see exit_flag)
    if (warp == 0) tc05::tmem_dealloc(sm.tmem_base, 512);
  }
}

// After the rollout: pad legs (0 -> 0) up to the global length, de-normalised reward, zero action tails.
template <int kEnv>
__global__ void __launch_bounds__(256) finalize_kernel(RolloutParams p, float* loglik, float* norm_out, float* real_out) {
  const int64_t R = p.n_inst * (int64_t)p.S;
  const int t_glob = *p.max_steps_out;
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = r % p.n_inst;
    const int s = (int)(r / p.n_inst);
    const int64_t drow = b % p.d.data_rows;
    const int t_own = p.ws_tile_steps[b * p.n_tiles + s / p.tile_rows];
    double len = p.ws_len[r];
    if (kEnv != RRNCO_ENV_ATSP && t_glob > t_own) {
      float d00 = p.d.distance[drow * (int64_t)p.N * p.N];
      if (kEnv == RRNCO_ENV_RCVRPTW && p.d.open_route[drow]) d00 = __fmul_rn(d00, 0.f);
      len += (double)(t_glob - t_own) * (double)d00;
    }
    const float neg = -(float)len;
    if (norm_out) norm_out[r] = neg;
    if (real_out) {
      const float mn = p.d.min_distance[drow], mx = p.d.max_distance[drow];
      real_out[r] = __fadd_rn(__fmul_rn(neg, __fadd_rn(__fsub_rn(mx, mn), 1e-6f)), mn);
    }
    if (loglik) loglik[r] = (float)p.ws_lp[r];
    for (int tt = t_own; tt < t_glob && tt < p.t_cap; ++tt) {
      p.actions[r * p.t_cap + tt] = 0;
      if (p.logprob) p.logprob[r * p.t_cap + tt] = 0.f;
    }
  }
}

// The kernel template is instantiated in two translation units so that they compile in parallel:
// this file (mma.sync FFN, also the logits-only mode) and rollout_kernel_tc.cu (RRNCO_BUILD_TC: tcgen05 FFN).
template <int kEnv, int kNTMax, int kPasses, bool kTc, bool kFilter = false>
int launch_rollout(const RolloutParams& p, cudaStream_t st) {
  auto kern = rollout_kernel<kEnv, kNTMax, kPasses, kTc, kFilter>;
  static PerDeviceOnce once;  // per device ordinal; idempotent attribute, benign if raced
  if (once.first()) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(Smem)) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  const int64_t grid = p.n_inst * p.n_tiles;
  if (grid <= 0 || grid > 0x7fffffffLL) return RRNCO_ERR_UNSUPPORTED;
  kern<<<(unsigned)grid, kTc ? kThreadsTc : kThreads, sizeof(Smem), st>>>(p);
  return rrnco_launch_status();
}

template <int kEnv, bool kTc>
int dispatch_rollout(const RolloutParams& p, int passes, cudaStream_t st) {
  if constexpr (kTc) {
    if (rrnco_filter_active(p.top_k, p.top_p))  // filtered: the NT <= 16 form only (it serves every N <= 128)
      return passes == 1 ? launch_rollout<kEnv, 16, 1, true, true>(p, st) : launch_rollout<kEnv, 16, 3, true, true>(p, st);
  }
  if (p.NT <= 13)
    return passes == 1 ? launch_rollout<kEnv, 13, 1, kTc>(p, st) : launch_rollout<kEnv, 13, 3, kTc>(p, st);
  return passes == 1 ? launch_rollout<kEnv, 16, 1, kTc>(p, st) : launch_rollout<kEnv, 16, 3, kTc>(p, st);
}

static int phase_cycles_local(long long* h_out, int reset) {
  if (h_out && cudaMemcpyFromSymbol(h_out, g_phase_cycles, sizeof(long long) * 16) != cudaSuccess) return RRNCO_ERR_CUDA;
  if (reset) {
    long long z[16] = {0};
    if (cudaMemcpyToSymbol(g_phase_cycles, z, sizeof(z)) != cudaSuccess) return RRNCO_ERR_CUDA;
  }
  return RRNCO_OK;
}

#ifdef RRNCO_BUILD_TC
int phase_cycles_tc(long long* h_out, int reset) { return phase_cycles_local(h_out, reset); }
// development aid: (tag, clock) event pairs of CTA 0 at decode step kTlStep (RRNCO_PHASE_STAMPS builds only)
int timeline_tc(long long* h_out, int* n_out) {
#ifdef RRNCO_PHASE_STAMPS
  int zero = 0;
  if (cudaMemcpyFromSymbol(h_out, g_tl, sizeof(long long) * 512) != cudaSuccess) return RRNCO_ERR_CUDA;
  if (cudaMemcpyFromSymbol(n_out, g_tl_n, sizeof(int)) != cudaSuccess) return RRNCO_ERR_CUDA;
  if (cudaMemcpyToSymbol(g_tl_n, &zero, sizeof(int)) != cudaSuccess) return RRNCO_ERR_CUDA;
  return RRNCO_OK;
#else
  (void)h_out;
  *n_out = 0;
  return RRNCO_ERR_UNSUPPORTED;
#endif
}
int dispatch_env_tc(const RolloutParams& p, int env, int passes, cudaStream_t st) {
  switch (env) {
    case RRNCO_ENV_ATSP: return dispatch_rollout<RRNCO_ENV_ATSP, true>(p, passes, st);
    case RRNCO_ENV_RCVRP: return dispatch_rollout<RRNCO_ENV_RCVRP, true>(p, passes, st);
    case RRNCO_ENV_RCVRPTW: return dispatch_rollout<RRNCO_ENV_RCVRPTW, true>(p, passes, st);
    default: return RRNCO_ERR_BAD_ARG;
  }
}
}  // namespace rrnco
#else
int dispatch_env_tc(const RolloutParams& p, int env, int passes, cudaStream_t st);  // rollout_kernel_tc.cu
int dispatch_env_lean(const RolloutParams& p, int env, int passes, cudaStream_t st);  // rollout_lean.cu
int pack_ffn_lean(const float* w1, const float* w2, const float* b1, const float* b2, void* packed, uint32_t* status,
                  cudaStream_t st);
constexpr int64_t kLeanBiasBytes = 4096;  // scaled biases behind the packed weight slices
int64_t lean_kv_bytes(int32_t n_nodes, int64_t n_tiles_total);
int phase_cycles_lean(long long* h_out, int reset);
constexpr int kLeanMaxNodes = 112;  // two score buffers + two P V slots in 256 TMEM columns
int dispatch_env_tiled(const RolloutParams& p, int env, int passes, cudaStream_t st);  // rollout_tiled.cu (N > 128)
int pack_kv_tiled(const RolloutParams& p, cudaStream_t st);
int64_t tiled_kv_bytes(int32_t n_nodes, int64_t n_inst);
int phase_cycles_tiled(long long* h_out, int reset);
extern int g_tiled_pairs;
int phase_cycles_tc(long long* h_out, int reset);
int timeline_tc(long long* h_out, int* n_out);

int dispatch_env(const RolloutParams& p, int env, int passes, cudaStream_t st) {
  switch (env) {
    case RRNCO_ENV_ATSP: return dispatch_rollout<RRNCO_ENV_ATSP, false>(p, passes, st);
    case RRNCO_ENV_RCVRP: return dispatch_rollout<RRNCO_ENV_RCVRP, false>(p, passes, st);
    case RRNCO_ENV_RCVRPTW: return dispatch_rollout<RRNCO_ENV_RCVRPTW, false>(p, passes, st);
    default: return RRNCO_ERR_BAD_ARG;
  }
}
}  // namespace rrnco

using namespace rrnco;

namespace {

inline bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0; }

int check_common(int32_t env, int32_t N, int64_t n_inst, int32_t S, const rrnco_decoder_weights_t* w,
                 const rrnco_decoder_cache_t* c, const rrnco_instance_data_t* d) {
  RRNCO_CHECK_ARG(w && c && d && n_inst > 0 && S > 0 && N > 1);
  RRNCO_CHECK_ARG(env >= 0 && env <= 2);
  if (N > RRNCO_MAX_NODES_FUSED) return RRNCO_ERR_UNSUPPORTED;
  RRNCO_CHECK_ARG(w->ffn_w1 && w->ffn_b1 && w->ffn_w2 && w->ffn_b2 && w->temperature > 0.f);
  RRNCO_CHECK_ARG(c->glimpse_key && c->glimpse_val && c->logit_key && c->ctx_node_proj);
  RRNCO_CHECK_ARG(aligned16(w->ffn_w1) && aligned16(w->ffn_w2) && aligned16(c->glimpse_key) &&
                  aligned16(c->glimpse_val) && aligned16(c->logit_key) && aligned16(c->ctx_node_proj));
  RRNCO_CHECK_ARG(d->data_rows > 0 && d->distance);
  if (env == RRNCO_ENV_ATSP) RRNCO_CHECK_ARG(c->ctx_node_proj2 && aligned16(c->ctx_node_proj2));
  if (env != RRNCO_ENV_ATSP) RRNCO_CHECK_ARG(w->ctx_state_w != nullptr);
  if (env == RRNCO_ENV_RCVRPTW) RRNCO_CHECK_ARG(d->duration != nullptr);
  return RRNCO_OK;
}

int g_passes = 3;  // set through rrnco_set_precision (process-wide default, read-only on the hot path)
int g_start_split = 0;  // key-tiled kernel: split the starts of an instance over several CTAs when the SMs would idle.  Off: the
                        // per-element passes are bound per SM SUB-PARTITION (rows <-> TMEM lane quarter <-> warp % 4), so a
                        // tile of 32 or 64 rows takes as long as one of 128 (measured: 132.9 vs 139.8 ms at config C4)
// POMO starts per CTA tile and tiles per instance (see rrnco_rollout_tile_rows in the header)
void rollout_tiling(int32_t n_nodes, int64_t n_inst, int32_t n_starts, int* tile_rows, int* n_tiles) {
  int tr = kRows;
  if (n_nodes > RRNCO_MAX_NODES_TILE && g_start_split) {
    const int sms = device_sm_count();
    int64_t k = sms > 0 ? sms / n_inst : 1;
    const int64_t kmax = (n_starts + 31) / 32;
    k = k > kmax ? kmax : k;
    k = k < 1 ? 1 : k;
    tr = (int)(((n_starts + k - 1) / k + 31) / 32 * 32);
    tr = tr > kRows ? kRows : tr;
  }
  *tile_rows = tr;
  *n_tiles = (n_starts + tr - 1) / tr;
}
bool g_last_tiled = false;  // the last rrnco_rollout call ran the key-tiled kernel (which counters rrnco_debug_phase_cycles reads)
int g_engine = 2;  // engine of the fused rollout: 2 = tcgen05, two lean CTAs per SM (N <= 112; else 1), 1 = tcgen05, one CTA
                   // per SM, 0 = mma.sync

}  // namespace

extern "C" {

// debug: per-phase cycle totals of CTA 0 since the last reset (host buffer of 16 int64); reset != 0 clears them
int rrnco_debug_phase_cycles(long long* h_out, int reset) {
  if (g_last_tiled) return phase_cycles_tiled(h_out, reset);  // 32 counters
  if (g_engine == 2) return phase_cycles_lean(h_out, reset);  // 32 counters
  return g_engine == 1 ? phase_cycles_tc(h_out, reset) : phase_cycles_local(h_out, reset);
}

// debug: event timeline of the tcgen05 variant (512 int64 = 256 (tag, clock) pairs); development builds only
int rrnco_debug_timeline(long long* h_out, int* n_out) { return timeline_tc(h_out, n_out); }

// precision of the in-kernel contractions: 3 = 3xTF32 (fp32-faithful, default), 1 = single TF32 pass
int rrnco_set_precision(int32_t passes) {
  if (passes != 1 && passes != 3) return RRNCO_ERR_BAD_ARG;
  g_passes = passes;
  return RRNCO_OK;
}

// Engine of the fused rollout kernel: 2 = the lean kernel (two CTAs per SM) for N <= 112, else 1 (default); 1 = one CTA
// per SM, tcgen05.mma + TMEM + TMA weight stream; 0 = the mma.sync FFN
int rrnco_set_ffn_engine(int32_t engine) {
  if (engine < 0 || engine > 2) return RRNCO_ERR_BAD_ARG;
  g_engine = engine;
  return RRNCO_OK;
}

int32_t rrnco_rollout_tile_rows(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts) {
  (void)env;
  if (n_inst <= 0 || n_starts <= 0) return kRows;
  int tr, nt;
  rollout_tiling(n_nodes, n_inst, n_starts, &tr, &nt);
  return tr;
}

int rrnco_set_start_split(int32_t mode) {  // 0 = product configuration; 1 = split the starts over CTAs; 2 = no CTA pairs
  if (mode < 0 || mode > 2) return RRNCO_ERR_BAD_ARG;
  g_start_split = mode == 1 ? 1 : 0;
  g_tiled_pairs = mode == 2 ? 0 : 1;
  return RRNCO_OK;
}

int64_t rrnco_rollout_workspace_bytes(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts) {
  (void)env;
  if (n_inst <= 0 || n_starts <= 0) return 0;
  const int64_t R = n_inst * n_starts;
  int tile_rows, n_tiles;
  rollout_tiling(n_nodes, n_inst, n_starts, &tile_rows, &n_tiles);
  const int64_t tiles = n_inst * n_tiles;
  // packed K / V / logit-key tiles: one region per CTA (lean engine) or one slot per SM (one-CTA engine)
  int64_t kv = (int64_t)kKvSlots * kKvSlotBytes;
  if (n_nodes <= kLeanMaxNodes && lean_kv_bytes(n_nodes, tiles) > kv) kv = lean_kv_bytes(n_nodes, tiles);
  if (n_nodes > RRNCO_MAX_NODES_TILE) kv = tiled_kv_bytes(n_nodes, n_inst);  // one pack per instance, shared by its start tiles
  return 2 * R * (int64_t)sizeof(double) + ((tiles * (int64_t)sizeof(int32_t) + 15) & ~15LL) + kFfnPackedBytes + kLeanBiasBytes + kv;
}

int rrnco_decoder_logits(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts,
                         const rrnco_decoder_weights_t* w, const rrnco_decoder_cache_t* cache,
                         const rrnco_instance_data_t* data, const int64_t* current, const int64_t* first,
                         const uint8_t* mask, const float* ctx_state, int32_t use_placeholder, float* logits_out,
                         uint32_t* status, void* stream) {
  int rc = check_common(env, n_nodes, n_inst, n_starts, w, cache, data);
  if (rc != RRNCO_OK) return rc;
  if (n_nodes > RRNCO_MAX_NODES_TILE) return RRNCO_ERR_UNSUPPORTED;  // rrnco_decoder_logits_large serves any N
  RRNCO_CHECK_ARG(current && mask && logits_out && status);
  RRNCO_CHECK_ARG(env == RRNCO_ENV_ATSP ? first != nullptr : ctx_state != nullptr);
  RRNCO_CHECK_ARG(!use_placeholder || w->ctx_placeholder_q);
  RolloutParams p{};
  p.N = n_nodes; p.NT = (n_nodes + 7) / 8; p.S = n_starts; p.n_tiles = (n_starts + kRows - 1) / kRows;
  p.n_state = env == RRNCO_ENV_ATSP ? 0 : env == RRNCO_ENV_RCVRP ? 1 : 4;
  p.tile_rows = kRows;
  p.n_inst = n_inst; p.logits_only = 1; p.use_placeholder = use_placeholder; p.max_steps = 1;
  p.w = *w; p.c = *cache; p.d = *data;
  p.in_cur = current; p.in_first = first; p.in_mask = mask; p.in_state = ctx_state; p.logits_out = logits_out;
  p.status = status;
  return dispatch_env(p, env, g_passes, (cudaStream_t)stream);
}

int rrnco_rollout_filtered(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts, int32_t multistart,
                           int32_t decode_mode, uint64_t seed, const rrnco_decoder_weights_t* w,
                           const rrnco_decoder_cache_t* cache, const rrnco_instance_data_t* data,
                           const int64_t* forced_actions, int32_t forced_T, int32_t t_cap, int64_t* actions_out,
                           float* logprob_out, float* loglik_out, float* norm_reward_out, float* real_reward_out,
                           int32_t* max_steps_out, uint32_t* status, void* workspace, int32_t top_k, float top_p,
                           void* stream) {
  RRNCO_CHECK_ARG(top_k >= 0 && top_p >= 0.f && top_p <= 1.f);  // (a NaN top_p fails both comparisons)
  int rc = check_common(env, n_nodes, n_inst, n_starts, w, cache, data);
  if (rc != RRNCO_OK) return rc;
  const bool filtered = rrnco_filter_active(top_k, top_p);
  // a filter needs a row's values at once: the key-tiled kernel never holds them; the mma.sync engine is not built for it
  if (filtered && (n_nodes > RRNCO_MAX_NODES_TILE || g_engine == 0)) return RRNCO_ERR_UNSUPPORTED;
  RRNCO_CHECK_ARG(actions_out && max_steps_out && status && workspace && aligned16(workspace) && t_cap > 0);
  RRNCO_CHECK_ARG(decode_mode >= 0 && decode_mode <= 2);
  RRNCO_CHECK_ARG(multistart || n_starts == 1);
  RRNCO_CHECK_ARG(decode_mode != RRNCO_DECODE_EVALUATE || (forced_actions && forced_T > 0));
  RRNCO_CHECK_ARG(real_reward_out == nullptr || (data->min_distance && data->max_distance));
  if (env == RRNCO_ENV_RCVRP) RRNCO_CHECK_ARG(data->demand && data->vehicle_capacity);
  if (env == RRNCO_ENV_RCVRPTW)
    RRNCO_CHECK_ARG(data->demand && data->demand_backhaul && data->time_windows && data->service_time &&
                    data->vehicle_capacity && data->distance_limit && data->open_route && data->backhaul_class);
  if (env == RRNCO_ENV_ATSP && !multistart) RRNCO_CHECK_ARG(w->ctx_placeholder_q != nullptr);
  cudaStream_t st = (cudaStream_t)stream;
  RolloutParams p{};
  p.N = n_nodes; p.NT = (n_nodes + 7) / 8; p.S = n_starts;
  rollout_tiling(n_nodes, n_inst, n_starts, &p.tile_rows, &p.n_tiles);
  p.n_state = env == RRNCO_ENV_ATSP ? 0 : env == RRNCO_ENV_RCVRP ? 1 : 4;
  p.n_inst = n_inst; p.multistart = multistart; p.mode = decode_mode; p.use_placeholder = !multistart;
  p.t_cap = t_cap; p.forced_T = forced_T; p.max_steps = t_cap - (multistart ? 1 : 0); p.seed = seed;
  p.w = *w; p.c = *cache; p.d = *data;
  p.forced = forced_actions; p.actions = actions_out; p.logprob = logprob_out;
  const int64_t R = n_inst * n_starts;
  p.ws_len = reinterpret_cast<double*>(workspace);
  p.ws_lp = p.ws_len + R;
  p.ws_tile_steps = reinterpret_cast<int32_t*>(p.ws_lp + R);
  const int64_t tiles = n_inst * p.n_tiles;
  unsigned char* packed = reinterpret_cast<unsigned char*>(p.ws_tile_steps) + ((tiles * (int64_t)sizeof(int32_t) + 15) & ~15LL);
  p.ffn_packed = packed;
  p.ffn_bias_scaled = reinterpret_cast<const float*>(packed + kFfnPackedBytes);
  p.kv_pack = packed + kFfnPackedBytes + kLeanBiasBytes;  // 16-byte aligned: every part above is a multiple of 16 bytes
  p.max_steps_out = max_steps_out; p.status = status;
  p.top_k = filtered ? top_k : 0; p.top_p = filtered ? top_p : 0.f;
  if (cudaMemsetAsync(max_steps_out, 0, sizeof(int32_t), st) != cudaSuccess) return RRNCO_ERR_CUDA;
  g_last_tiled = n_nodes > RRNCO_MAX_NODES_TILE;
  if (n_nodes > RRNCO_MAX_NODES_TILE) {  // key-tiled tcgen05 kernel (the only fused engine for more than one key tile)
    rc = pack_ffn_lean(w->ffn_w1, w->ffn_w2, w->ffn_b1, w->ffn_b2, packed, status, st);
    if (rc != RRNCO_OK) return rc;
    rc = pack_kv_tiled(p, st);
    if (rc != RRNCO_OK) return rc;
    rc = dispatch_env_tiled(p, env, g_passes, st);
  } else if (g_engine == 2 && n_nodes <= kLeanMaxNodes) {
    rc = pack_ffn_lean(w->ffn_w1, w->ffn_w2, w->ffn_b1, w->ffn_b2, packed, status, st);
    if (rc != RRNCO_OK) return rc;
    rc = dispatch_env_lean(p, env, g_passes, st);
  } else if (g_engine >= 1) {
    rc = pack_ffn_weights(w->ffn_w1, w->ffn_w2, packed, st);
    if (rc != RRNCO_OK) return rc;
    rc = dispatch_env_tc(p, env, g_passes, st);
  } else {
    rc = dispatch_env(p, env, g_passes, st);
  }
  if (rc != RRNCO_OK) return rc;
  const unsigned fgrid = (unsigned)((R + 255) / 256 > 4096 ? 4096 : (R + 255) / 256);
  switch (env) {
    case RRNCO_ENV_ATSP: finalize_kernel<RRNCO_ENV_ATSP><<<fgrid, 256, 0, st>>>(p, loglik_out, norm_reward_out, real_reward_out); break;
    case RRNCO_ENV_RCVRP: finalize_kernel<RRNCO_ENV_RCVRP><<<fgrid, 256, 0, st>>>(p, loglik_out, norm_reward_out, real_reward_out); break;
    default: finalize_kernel<RRNCO_ENV_RCVRPTW><<<fgrid, 256, 0, st>>>(p, loglik_out, norm_reward_out, real_reward_out); break;
  }
  return rrnco_launch_status();
}

int rrnco_rollout(int32_t env, int32_t n_nodes, int64_t n_inst, int32_t n_starts, int32_t multistart,
                  int32_t decode_mode, uint64_t seed, const rrnco_decoder_weights_t* w,
                  const rrnco_decoder_cache_t* cache, const rrnco_instance_data_t* data,
                  const int64_t* forced_actions, int32_t forced_T, int32_t t_cap, int64_t* actions_out,
                  float* logprob_out, float* loglik_out, float* norm_reward_out, float* real_reward_out,
                  int32_t* max_steps_out, uint32_t* status, void* workspace, void* stream) {
  return rrnco_rollout_filtered(env, n_nodes, n_inst, n_starts, multistart, decode_mode, seed, w, cache, data, forced_actions,
                                forced_T, t_cap, actions_out, logprob_out, loglik_out, norm_reward_out, real_reward_out,
                                max_steps_out, status, workspace, 0, 0.f, stream);
}

}  // extern "C"
#endif  // RRNCO_BUILD_TC
