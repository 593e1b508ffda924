// Fused construction-rollout kernel, lean form: TWO resident CTAs per SM (RRNetPolicy.forward decode loop,
// rrnco/models/policy.py:203-243; per-step math as in rollout_kernel.cu, whose header describes phases A-S).
//
// Why: inside one tile the phases of a decode step are serial (each step needs the previous action) and they load
// different units -- the softmax / select passes are bound by instruction issue with the tensor pipe idle, the FFN by the
// tensor pipe / the weight stream with the CUDA cores idle.  With two independent tiles resident on an SM the hardware
// interleaves them: one tile's FFN runs under the other tile's softmax.  That needs half the footprint per tile:
//   * <= 113 KB of shared memory: the 64 KB activation tiles (Q -> glimpse, fp16 hi | lo, A operands of the SS MMAs) plus a
//     4-5 x 8 KB ring through which EVERY B operand streams by TMA (cp.async.bulk) in the fixed order the tensor pipe
//     consumes it: per step 16 K_h / V_h head tiles, 64 FFN weight K-step slices, 8 logit-key K-step slices, all
//     <= 8 KB, all pre-packed fp16 hi | lo core-matrix tiles that stay L2-resident.  Nothing is resident but the
//     activations; the fp32 bias tile alpha.D[cur,:] (+ beta.Dur[cur,:]) borrows the activation region while it is dead
//     (logits MMAs + select).
//   * 256 TMEM columns: two score buffers (one per compute-warp group) with a 16-column P V accumulator each; the FFN
//     hidden accumulator is converted IN PLACE to the fp16 hi | lo A operand of GEMM2 (16 fp32 columns -> 8 + 8 packed
//     columns at the same address), the FFN output accumulator likewise to the A operand of the logits GEMM.
//   * <= 96 registers per thread: every per-element pass works on 16 or 32 TMEM columns at a time.
// One elected thread of warp 9 issues every tcgen05.mma in program order (first MMA of each accumulation overwrites: no
// zeroing passes), one elected thread of warp 8 issues every bulk copy; warps 0-7 run the element-wise passes
// thread-per-rollout.  Results are bitwise reproducible and identical in value to rollout_kernel<..., kTc = true>.
#include <cstdio>
#include "common.cuh"
#include "tc05.cuh"
#include "ffn_pack.cuh"
#include "rollout_common.cuh"

namespace rrnco {

constexpr int kLThreads = 320;            // warps 0-7 compute, 8 TMA producer, 9 MMA issue
constexpr int kLCompute = 256;
constexpr uint32_t kLStageBytes = 8192;
constexpr int kLBiasLd = 116;             // fp32 row stride of the bias tile (conflict-free float4 rows, 16-byte aligned)
constexpr int kLBiasBytes = kRows * kLBiasLd * 4;  // 59 392: the select exchange arrays live behind it in the A region
constexpr int kLJobs = 8;                 // G1(0) G2(0) G1(1) G2(1) G1(2) G2(2) G1(3) G2(3): one hidden accumulator
constexpr int kLWSlices = kLJobs * 8;     // one 8 KB slice per K step (16 k values) of a 128 x 128 x 128 job
constexpr int64_t kLeanFfnPackedBytes = (int64_t)kLWSlices * kLStageBytes;  // 512 KB

// per-phase cycle accumulator of thread 0 of CTA 0 (development builds: RRNCO_PHASE_STAMPS), read with rrnco_debug_phase_cycles
__device__ long long g_lean_cycles[32];
#ifdef RRNCO_PHASE_STAMPS
#define LSTAMP(i)                                   \
  do {                                              \
    if (blockIdx.x == 0 && tid == 0) {              \
      const long long now_ = clock64();             \
      g_lean_cycles[i] += now_ - stamp_t0;          \
      stamp_t0 = now_;                              \
    }                                               \
  } while (0)
#else
#define LSTAMP(i) do { } while (0)
#endif

template <int kEnv>
struct LeanSmem {
  // ring depth: as many 8 KB stages as fit beside the activation tiles in 113 KB (the time-window env needs 7 per-node
  // arrays and 4 state words per rollout: one stage less)
  static constexpr int kStages = 4;  // (a fifth stage where it fits was measured neutral; the space holds the FFN biases)
  static constexpr int kNodeArrays = kEnv == RRNCO_ENV_RCVRPTW ? 7 : 1;
  static constexpr int kStateArrays = kEnv == RRNCO_ENV_RCVRPTW ? 4 : 1;
  unsigned char A[kRows * kE * 4];         // Q -> glimpse (fp16 hi | lo tiles) | fp32 bias tile during logits + select
  unsigned char ring[kStages][kLStageBytes];
  float ffn_bias[kF + kE];                 // kAScale b1 | kAScale b2: read by every epilogue block (from L1 / L2 they were the
                                           // top stall of the FFN epilogues: 17.8 % of the kernel's stall samples)
  float wstate[kStateArrays][kE];          // context state weights; ATSP: row 0 = placeholder query
  float node[kNodeArrays][kRows];          // dem | demb tw0 tw1 svc dj0 uj0 (rcvrptw)
  float f[kStateArrays][kRows];            // rcvrp: used | rcvrptw: time, route, used_l, used_b
  uint32_t vis[kRows][4];
  uint32_t mask[kRows][4];
  unsigned char cur[kRows], first[kRows], active[kRows], done[kRows];
  uint32_t lhmask[4];
  uint32_t kmax2[kH];                      // max over the keys of |K_h row|^2 (fp32 bits; non-negative floats order as integers)
  // rcvrp: the capacity mask {c : fl(demand_c + used) > cap} is an upper set in demand order (fl(x + u) is monotone in x), so a
  // rollout finds it with a 8-probe search over the instance's sorted demands and one precomputed 128-bit suffix mask
  // instead of 112 add-compare-shift steps per decode step -- bit-exact, the predicate is evaluated as upstream writes it
  static constexpr int kSorted = kEnv == RRNCO_ENV_RCVRP ? kRows : 1;
  float sdem[kSorted];                     // demands ascending (ties by node index)
  uint32_t sufmask[kSorted + 1][4];        // sufmask[K] = nodes of rank >= K
  uint64_t bar_full[kStages], bar_empty[kStages];
  uint64_t bar_step;     // compute -> producer: another decode step follows (or exit)
  uint64_t bar_q;        // compute -> issuer: query tiles written (256 arrivals; also the exit signal)
  uint64_t bar_s[kH];    // issuer -> compute: scores of head h in TMEM
  uint64_t bar_p[kH];    // compute -> issuer: probabilities of head h written in place (128 arrivals)
  uint64_t bar_o[kH];    // issuer -> compute: P V of head h complete
  uint64_t bar_gready;   // compute -> issuer: glimpse tiles written, O slots read (256 arrivals)
  uint64_t bar_h;        // issuer -> compute: GEMM1 of a chunk complete
  uint64_t bar_epi;      // compute -> issuer: hidden chunk converted in place to the A operand of GEMM2 (256 arrivals)
  uint64_t bar_g2;       // issuer -> compute: FFN output complete
  uint64_t bar_lk;       // compute -> issuer: g' converted in place to the A operand of the logits GEMM (256 arrivals)
  uint64_t bar_acc;      // issuer -> compute: logits complete
  uint32_t tmem_base;
  volatile int exit_flag;
};

__device__ __forceinline__ void lean_sync() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }
// Waits of many warps for one mbarrier: a single warp watches the mbarrier, the others sleep in a hardware barrier that
// costs no issue slots (eight warps polling one mbarrier through the FFN were ~20 % of the executed instructions).
__device__ __forceinline__ void lean_wait_all(uint64_t* bar, uint32_t parity, int warp) {
  if (warp == 0) tc05::mbar_wait(bar, parity);
  asm volatile("bar.sync 4, 256;\n" ::: "memory");
}
__device__ __forceinline__ void lean_wait_group(uint64_t* bar, uint32_t parity, int warp) {  // the 4 warps of a head group
  if ((warp & 3) == 0) tc05::mbar_wait(bar, parity);
  if (warp < 4) asm volatile("bar.sync 2, 128;\n" ::: "memory");
  else asm volatile("bar.sync 3, 128;\n" ::: "memory");
}
__device__ __forceinline__ int lean_sync_and(int pred) {
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

// Pack W1 / W2 into 64 slices of 8 KB in tensor-pipe order: slice (job j, K step ks), job j = chunk j >> 1, half j & 1
// (0: W1 rows of the chunk, k = input dims; 1: W2 rows = output dims, k = hidden units of the chunk);
// layout [hi | lo][16-byte K chunk (2)][row (128)][8 halves].  One thread per (slice, row, k pair).
// Also writes the biases pre-scaled by kAScale behind the slices (b1 [512] | b2 [128]): the epilogues then produce the
// scaled fp16 operands directly.  A weight outside the fp16 range of its scaled hi part is reported, never silent.
__global__ void pack_ffn_lean_kernel(const float* __restrict__ w1, const float* __restrict__ w2, const float* __restrict__ b1,
                                     const float* __restrict__ b2, uint32_t* __restrict__ packed, uint32_t* status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kF + kE) {
    float* bs = reinterpret_cast<float*>(packed + kLWSlices * (kLStageBytes / 4));
    bs[i] = kAScale * (i < kF ? b1[i] : b2[i - kF]);
  }
  if (i >= kLWSlices * kRows * 8) return;
  const int kp = i & 7, row = (i >> 3) & 127, s = i >> 10;
  const int j = s >> 3, ks = s & 7, c = j >> 1, half = j & 1;
  const int k = ks * 16 + kp * 2;
  float v0, v1;
  if (half == 0) {
    v0 = w1[(size_t)(c * kRows + row) * kE + k];
    v1 = w1[(size_t)(c * kRows + row) * kE + k + 1];
  } else {
    v0 = w2[(size_t)row * kF + c * kRows + k];
    v1 = w2[(size_t)row * kF + c * kRows + k + 1];
  }
  if (!(fabsf(v0) * kWScale < 65504.f) || !(fabsf(v1) * kWScale < 65504.f)) atomicOr(status, RRNCO_DEV_NAN_LOGITS);
  uint32_t hi, lo;
  f16s_split2(v0, v1, kWScale, hi, lo);
  uint32_t* dst = packed + (size_t)s * (kLStageBytes / 4) + (kp >> 2) * (kRows * 4) + row * 4 + (kp & 3);
  dst[0] = hi;
  dst[kLStageBytes / 8] = lo;
}

// ---- env transition on the shared-memory state (one thread per row); returns the leg to add to the tour length ----
template <int kEnv>
__device__ __forceinline__ float lean_transition(LeanSmem<kEnv>& sm, int N, int row, int a, const float* D, const float* U,
                                                 float closed, bool count_leg) {
  const int prev = sm.cur[row];
  float leg = 0.f;
  if (kEnv == RRNCO_ENV_ATSP) {
    if (count_leg) leg = D[prev * N + a];
  } else if (kEnv == RRNCO_ENV_RCVRP) {
    leg = D[prev * N + a];
    const int di = min(max(a - 1, 0), N - 2) + 1;  // clamp(a-1, 0, n_loc-1), dem[] is depot-shifted
    sm.f[0][row] = __fmul_rn(__fadd_rn(sm.f[0][row], sm.node[0][di]), a != 0 ? 1.0f : 0.0f);
  } else {
    const float away = a != 0 ? 1.0f : 0.0f;
    const float dist = D[prev * N + a], dur = U[prev * N + a];
    leg = a == 0 ? __fmul_rn(dist, closed) : dist;
    const int kN = LeanSmem<kEnv>::kNodeArrays - 1;  // (index clamp keeps the non-rcvrptw instantiations in bounds)
    sm.f[0][row] = __fmul_rn(away, __fadd_rn(fmaxf(__fadd_rn(sm.f[0][row], dur), sm.node[min(2, kN)][a]), sm.node[min(4, kN)][a]));
    const int kS = LeanSmem<kEnv>::kStateArrays - 1;
    sm.f[min(1, kS)][row] = __fmul_rn(away, __fadd_rn(sm.f[min(1, kS)][row], dist));
    sm.f[min(2, kS)][row] = __fmul_rn(away, __fadd_rn(sm.f[min(2, kS)][row], sm.node[0][a]));
    sm.f[min(3, kS)][row] = __fmul_rn(away, __fadd_rn(sm.f[min(3, kS)][row], sm.node[min(1, kN)][a]));
  }
  sm.vis[row][a >> 5] |= 1u << (a & 31);
  sm.cur[row] = (unsigned char)a;
  const int cnt = __popc(sm.vis[row][0]) + __popc(sm.vis[row][1]) + __popc(sm.vis[row][2]) + __popc(sm.vis[row][3]);
  sm.done[row] = cnt == N;
  return leg;
}

// kFilter: decode with the top-k / top-p filters of p (single-pass select only)
template <int kEnv, int kPasses, bool kFilter>
__global__ void __launch_bounds__(kLThreads, 2) rollout_lean_kernel(const RolloutParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  using SmemT = LeanSmem<kEnv>;
  SmemT& sm = *reinterpret_cast<SmemT*>(smem_raw);
  constexpr int kNA = SmemT::kNodeArrays - 1, kSA = SmemT::kStateArrays - 1;
  // node-array / state-array indices, clamped so that every instantiation stays in bounds
  constexpr int iDem = 0, iDemb = kNA < 1 ? kNA : 1, iTw0 = kNA < 2 ? kNA : 2, iTw1 = kNA < 3 ? kNA : 3, iSvc = kNA < 4 ? kNA : 4,
                iDj0 = kNA < 5 ? kNA : 5, iUj0 = kNA < 6 ? kNA : 6;
  constexpr int f1i = kSA < 1 ? kSA : 1, f2i = kSA < 2 ? kSA : 2, f3i = kSA < 3 ? kSA : 3;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N;
  const int R16 = ((N + 15) >> 4) << 4;
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
  const float cap = kEnv == RRNCO_ENV_ATSP ? 0.f : p.d.vehicle_capacity[drow];
  float closed = 1.f, limit = INFINITY, bclass = 1.f;
  if (kEnv == RRNCO_ENV_RCVRPTW) {
    closed = p.d.open_route[drow] ? 0.f : 1.f;
    limit = p.d.distance_limit[drow];
    bclass = p.d.backhaul_class[drow];
  }
  // this CTA's packed K / V / logit-key tiles (24 slices of R16 x 64 bytes), L2-resident for the whole rollout
  const uint32_t kv_slice = (uint32_t)R16 * 64u;
  unsigned char* slot = p.kv_pack + (size_t)blockIdx.x * (24u * kv_slice);

  // ---------------- one-time staging ----------------
  if (warp == 0) tc05::tmem_alloc(&sm.tmem_base, 256);
  if (tid == 32) {
    for (int i = 0; i < SmemT::kStages; ++i) {
      tc05::mbar_init(&sm.bar_full[i], 1);
      tc05::mbar_init(&sm.bar_empty[i], 1);
    }
    tc05::mbar_init(&sm.bar_step, 1);
    tc05::mbar_init(&sm.bar_q, kLCompute);
    for (int i = 0; i < kH; ++i) {
      tc05::mbar_init(&sm.bar_s[i], 1);
      tc05::mbar_init(&sm.bar_p[i], kLCompute / 2);
      tc05::mbar_init(&sm.bar_o[i], 1);
    }
    tc05::mbar_init(&sm.bar_gready, kLCompute);
    tc05::mbar_init(&sm.bar_h, 1);
    tc05::mbar_init(&sm.bar_epi, kLCompute);
    tc05::mbar_init(&sm.bar_g2, 1);
    tc05::mbar_init(&sm.bar_lk, kLCompute);
    tc05::mbar_init(&sm.bar_acc, 1);
    tc05::fence_mbar_init();
    sm.exit_flag = 0;
    for (int i = 0; i < kH; ++i) sm.kmax2[i] = 0u;
  }
  for (int i = tid; i < kF + kE; i += kLThreads) sm.ffn_bias[i] = p.ffn_bias_scaled[i];
  if (tid < kE) {
#pragma unroll
    for (int k = 0; k < SmemT::kStateArrays; ++k) {
      float w = 0.f;
      if (kEnv == RRNCO_ENV_ATSP) w = p.w.ctx_placeholder_q ? p.w.ctx_placeholder_q[tid] : 0.f;
      else if (k < p.n_state) w = p.w.ctx_state_w[k * kE + tid];
      sm.wstate[k][tid] = w;
    }
  }
  if (tid < kRows) {
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
    sm.node[iDem][n] = dem;
    if (kEnv == RRNCO_ENV_RCVRPTW) {
      sm.node[iDemb][n] = demb; sm.node[iTw0][n] = tw0; sm.node[iTw1][n] = tw1; sm.node[iSvc][n] = svc;
      sm.node[iDj0][n] = dj0; sm.node[iUj0][n] = uj0;
    }
    const uint32_t lh = __ballot_sync(0xffffffffu, kEnv == RRNCO_ENV_RCVRPTW && dem > 0.f);
    if (lane == 0) sm.lhmask[warp] = lh;
  }
  __syncthreads();

  if (kEnv == RRNCO_ENV_RCVRP) {
    unsigned char* s_rank = sm.A;  // (scratch: the activation region is not in use yet)
    if (tid < kRows) {
      const float dk = sm.node[iDem][tid];
      int r = 0;
      for (int j = 0; j < kRows; ++j) {
        const float dj = sm.node[iDem][j];
        r += (dj < dk || (dj == dk && j < tid)) ? 1 : 0;
      }
      s_rank[tid] = (unsigned char)r;
      sm.sdem[r % SmemT::kSorted] = dk;
    }
    __syncthreads();
    if (tid <= kRows) {  // suffix masks: nodes of rank >= tid
      uint32_t w[4] = {0u, 0u, 0u, 0u};
      for (int c = 0; c < kRows; ++c)
        if ((int)s_rank[c] >= tid) w[c >> 5] |= 1u << (c & 31);
#pragma unroll
      for (int k = 0; k < 4; ++k) sm.sufmask[tid % (SmemT::kSorted + 1)][k] = w[k];
    }
    __syncthreads();
  }

  // ---------------- rollout state init ----------------
  const int num_loc = kEnv == RRNCO_ENV_ATSP ? N : N - 1;
  double len_acc = 0.0, lp_acc = 0.0;  // running tour length / log-likelihood of the row this thread transitions
  if (tid < kRows) {
    const int row = tid;
    const int s_real = tile * kRows + row;
    const int active = s_real < p.S;
    const int s = active ? s_real : tile * kRows;  // padded rows shadow the tile's first rollout
    const int64_t r = (int64_t)s * p.n_inst + b;
    sm.active[row] = (unsigned char)active;
    sm.first[row] = 0;
#pragma unroll
    for (int k = 0; k < SmemT::kStateArrays; ++k) sm.f[k][row] = 0.f;
#pragma unroll
    for (int k = 0; k < 4; ++k) { sm.vis[row][k] = 0u; sm.mask[row][k] = 0u; }
    sm.done[row] = 0;
    sm.cur[row] = 0;
    if (p.multistart) {
      const int a0 = s % num_loc + (kEnv == RRNCO_ENV_ATSP ? 0 : 1);  // select_start_nodes
      len_acc += (double)lean_transition<kEnv>(sm, N, row, a0, D, U, closed, /*count_leg=*/false);  // depot -> a0 (VRPs)
      sm.first[row] = (unsigned char)a0;
      if (active) {
        p.actions[r * p.t_cap] = a0;
        if (p.logprob) p.logprob[r * p.t_cap] = 0.f;
      }
    }
  }
  __syncthreads();

  // ---- one-time: K / V / Lk of this instance -> fp16 hi | lo tiles in the shared-memory layouts of the MMAs (B operands),
  // one contiguous slice per head / K step so that ONE bulk copy moves it:
  //   K_h, Lk_ks : [hi | lo][16-byte K chunk (2)][key (R16)][8 halves]
  //   V_h        : [hi | lo][key chunk (R16 / 8)][dim (16)][8 halves]      (V_h^T, K-major over the keys)
  // slices 0-7 K heads, 8-15 V heads, 16-23 logit-key K steps.
  if (tid < kLCompute) {
#pragma unroll 1
    for (int which = 0; which < 2; ++which) {
      const float* src = which ? Lk : Kc;
      const float scale = which ? kLkScale : kKvScale;
      uint4* base = reinterpret_cast<uint4*>(slot + (size_t)(which ? 16 : 0) * kv_slice);
      for (int idx = tid; idx < R16 * 16; idx += kLCompute) {
        const int r = idx >> 4, c8 = idx & 15;
        float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
        if (r < N) {
          v0 = __ldg(reinterpret_cast<const float4*>(src + (size_t)r * kE) + c8 * 2);
          v1 = __ldg(reinterpret_cast<const float4*>(src + (size_t)r * kE) + c8 * 2 + 1);
        }
        if (which == 0) {  // |K_h row|^2 (lanes 2i, 2i+1 hold the two halves of a head) -> per-head maximum over the keys
          float n2 = v0.x * v0.x + v0.y * v0.y + v0.z * v0.z + v0.w * v0.w + v1.x * v1.x + v1.y * v1.y + v1.z * v1.z + v1.w * v1.w;
          n2 += __shfl_xor_sync(0xffffffffu, n2, 1);
          if ((c8 & 1) == 0) atomicMax(&sm.kmax2[c8 >> 1], __float_as_uint(n2));
        }
        uint32_t h[4], l[4];
        f16s_split2(v0.x, v0.y, scale, h[0], l[0]); f16s_split2(v0.z, v0.w, scale, h[1], l[1]);
        f16s_split2(v1.x, v1.y, scale, h[2], l[2]); f16s_split2(v1.z, v1.w, scale, h[3], l[3]);
        uint4* sl = base + (size_t)(c8 >> 1) * (R16 * 4);  // slice of head c8 >> 1: R16 x 64 bytes = R16 x 4 uint4
        sl[(c8 & 1) * R16 + r] = make_uint4(h[0], h[1], h[2], h[3]);
        sl[2 * R16 + (c8 & 1) * R16 + r] = make_uint4(l[0], l[1], l[2], l[3]);
      }
    }
    const int nkc = R16 >> 3;
    uint4* vbase = reinterpret_cast<uint4*>(slot + (size_t)8 * kv_slice);
    for (int idx = tid; idx < R16 * 16; idx += kLCompute) {
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
      uint4* sl = vbase + (size_t)hh * (R16 * 4);
      sl[kc * 16 + d] = make_uint4(h[0], h[1], h[2], h[3]);
      sl[2 * R16 + kc * 16 + d] = make_uint4(l[0], l[1], l[2], l[3]);
    }
    tc05::fence_proxy_async_all();  // generic-proxy global writes -> visible to the TMA reads below
  }
  tc05::fence_before_sync();
  __syncthreads();
  tc05::fence_after_sync();

  const int uwarp = __shfl_sync(0xffffffffu, warp, 0);  // warp index as a value the compiler knows to be warp-uniform
  if (uwarp == 8) {
    // ===== TMA producer: per decode step 88 slices through the ring, in the order the issuer consumes them =====
    if (tc05::elect_one()) {
      uint32_t st = 0, round = 0, step_par = 0;  // ring stage, number of completed passes over the ring
      auto push = [&](const unsigned char* src, uint32_t bytes) {
        if (round > 0) tc05::mbar_wait(&sm.bar_empty[st], (round - 1) & 1, 32);
        tc05::mbar_arrive_expect_tx(&sm.bar_full[st], bytes);
        tc05::bulk_g2s(sm.ring[st], src, bytes, &sm.bar_full[st]);
        if (++st == (uint32_t)SmemT::kStages) { st = 0; ++round; }
      };
      while (true) {
        tc05::mbar_wait(&sm.bar_step, step_par, 64);
        step_par ^= 1u;
        if (sm.exit_flag) break;
        // attention: K of positions 0, 1, then V(k), K(k + 2); position k -> head (k & 1) * 4 + (k >> 1)
        push(slot + (size_t)0 * kv_slice, kv_slice);  // K, position 0 = head 0
        push(slot + (size_t)4 * kv_slice, kv_slice);  // K, position 1 = head 4
#pragma unroll 1
        for (int k = 0; k < kH; ++k) {
          const int h = (k & 1) * 4 + (k >> 1);
          push(slot + (size_t)(8 + h) * kv_slice, kv_slice);
          if (k + 2 < kH) {
            const int h2 = ((k + 2) & 1) * 4 + ((k + 2) >> 1);
            push(slot + (size_t)h2 * kv_slice, kv_slice);
          }
        }
#pragma unroll 1
        for (int s = 0; s < kLWSlices; ++s) push(p.ffn_packed + (size_t)s * kLStageBytes, kLStageBytes);
#pragma unroll 1
        for (int ks = 0; ks < 8; ++ks) push(slot + (size_t)(16 + ks) * kv_slice, kv_slice);
      }
    }
    return;
  }
  if (uwarp == 9) {
    // ===== MMA issue: one elected thread, fixed program order (bitwise reproducible accumulation) =====
    if (tc05::elect_one()) {
      const uint32_t tb = sm.tmem_base;
      const uint32_t t_hacc = tb, t_oacc = tb + 128;
      const uint32_t idesc = tc05::make_idesc_f16(128, 128);
      const uint32_t idesc_l = tc05::make_idesc_f16(128, R16);
      const uint32_t idesc_pv = tc05::make_idesc_f16(128, 16);
      const uint32_t q_addr = tc05::smem_u32(sm.A);
      const uint32_t a_lo_off = kRows * kE * 2;
      const uint32_t ring_addr = tc05::smem_u32(sm.ring[0]);
      const uint32_t lbo_l = (uint32_t)R16 * 16u;   // bytes between the two K chunks of a K_h / Lk slice
      const uint32_t var_l = (uint32_t)R16 * 32u;   // hi -> lo variant of a K_h / V_h / Lk slice
      uint32_t st = 0, round = 0, step_par = 0;  // ring stage, number of completed passes over the ring
      auto stage_wait = [&]() -> uint32_t {
        tc05::mbar_wait(&sm.bar_full[st], round & 1);
        tc05::fence_after_sync();
        return ring_addr + st * kLStageBytes;
      };
      auto stage_release = [&]() {
        tc05::commit(&sm.bar_empty[st]);
        if (++st == (uint32_t)SmemT::kStages) { st = 0; ++round; }
      };
      auto issue_qk = [&](int k) {
        const int h = (k & 1) * 4 + (k >> 1);
        const uint32_t t_s = tb + (uint32_t)(k & 1) * 128u;
        const uint32_t kh = stage_wait();
        const uint32_t qh = q_addr + 2 * h * kLboTile;
        const uint64_t q_hi = tc05::make_desc(qh, kLboTile, kSbo), k_hi = tc05::make_desc(kh, lbo_l, kSbo);
        tc05::mma_ss_f16(t_s, q_hi, k_hi, idesc_l, 0u);
        if (kPasses == 3) {
          tc05::mma_ss_f16(t_s, tc05::make_desc(qh + a_lo_off, kLboTile, kSbo), k_hi, idesc_l, 1u);
          tc05::mma_ss_f16(t_s, q_hi, tc05::make_desc(kh + var_l, lbo_l, kSbo), idesc_l, 1u);
        }
        tc05::commit(&sm.bar_s[h]);
        stage_release();
      };
      while (true) {
        tc05::mbar_wait(&sm.bar_q, step_par, 32);
        if (sm.exit_flag) break;
        tc05::fence_after_sync();
        issue_qk(0);
        issue_qk(1);
#pragma unroll 1
        for (int k = 0; k < kH; ++k) {
          const int h = (k & 1) * 4 + (k >> 1);
          const uint32_t t_s = tb + (uint32_t)(k & 1) * 128u, t_o = t_s + 112u;
          tc05::mbar_wait(&sm.bar_p[h], step_par, 32);
          tc05::fence_after_sync();
          const uint32_t vh = stage_wait();
          // V_h^T slice: 16 dims x keys, K-major: 256 B between 16-byte key chunks, 128 B between 8-dim groups;
          // P_hi at columns 16 j, P_lo at 16 j + 8 of the score buffer
#pragma unroll 1
          for (int j = 0; j < (R16 >> 4); ++j) {
            const uint64_t v_hi = tc05::make_desc(vh + j * 512, 256, kSbo);
            tc05::mma_ts_f16(t_o, t_s + 16 * j, v_hi, idesc_pv, j > 0 ? 1u : 0u);
            if (kPasses == 3) {
              tc05::mma_ts_f16(t_o, t_s + 16 * j + 8, v_hi, idesc_pv, 1u);
              tc05::mma_ts_f16(t_o, t_s + 16 * j, tc05::make_desc(vh + var_l + j * 512, 256, kSbo), idesc_pv, 1u);
            }
          }
          tc05::commit(&sm.bar_o[h]);
          stage_release();
          if (k + 2 < kH) issue_qk(k + 2);
        }
        tc05::mbar_wait(&sm.bar_gready, step_par, 32);
        tc05::fence_after_sync();
#pragma unroll 1
        for (int j = 0; j < kLJobs; ++j) {
          const int c = j >> 1, half = j & 1;
          if (half == 1) {  // hidden chunk c converted in place to the A operand of GEMM2(c)
            tc05::mbar_wait(&sm.bar_epi, c & 1, 32);
            tc05::fence_after_sync();
          }
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) {
            const uint32_t b_addr = stage_wait();
            const uint64_t b_hi = tc05::make_desc(b_addr, kLboTile, kSbo);
            const uint64_t b_lo = tc05::make_desc(b_addr + kLStageBytes / 2, kLboTile, kSbo);
            if (half == 0) {
              const uint64_t a_hi = tc05::make_desc(q_addr + ks * 2 * kLboTile, kLboTile, kSbo);
              tc05::mma_ss_f16(t_hacc, a_hi, b_hi, idesc, ks > 0 ? 1u : 0u);
              if (kPasses == 3) {
                tc05::mma_ss_f16(t_hacc, tc05::make_desc(q_addr + a_lo_off + ks * 2 * kLboTile, kLboTile, kSbo), b_hi, idesc, 1u);
                tc05::mma_ss_f16(t_hacc, a_hi, b_lo, idesc, 1u);
              }
            } else {
              tc05::mma_ts_f16(t_oacc, t_hacc + 16 * ks, b_hi, idesc, (c > 0 || ks > 0) ? 1u : 0u);
              if (kPasses == 3) {
                tc05::mma_ts_f16(t_oacc, t_hacc + 16 * ks + 8, b_hi, idesc, 1u);
                tc05::mma_ts_f16(t_oacc, t_hacc + 16 * ks, b_lo, idesc, 1u);
              }
            }
            stage_release();
          }
          if (half == 0) tc05::commit(&sm.bar_h);
        }
        tc05::commit(&sm.bar_g2);
        // pointer logits: D[128 x R16] = g'(hi | lo in place over the output accumulator) . Lk^T, 8 K steps
        tc05::mbar_wait(&sm.bar_lk, step_par, 32);
        tc05::fence_after_sync();
#pragma unroll 1
        for (int ks = 0; ks < 8; ++ks) {
          const uint32_t lk = stage_wait();
          const uint64_t l_hi = tc05::make_desc(lk, lbo_l, kSbo);
          tc05::mma_ts_f16(t_hacc, t_oacc + 16 * ks, l_hi, idesc_l, ks > 0 ? 1u : 0u);
          if (kPasses == 3) {
            tc05::mma_ts_f16(t_hacc, t_oacc + 16 * ks + 8, l_hi, idesc_l, 1u);
            tc05::mma_ts_f16(t_hacc, t_oacc + 16 * ks, tc05::make_desc(lk + var_l, lbo_l, kSbo), idesc_l, 1u);
          }
          stage_release();
        }
        tc05::commit(&sm.bar_acc);
        step_par ^= 1u;
      }
    }
    return;
  }

  // ================= compute warps 0-7 =================
  const uint32_t tb = sm.tmem_base;
  const int lq = warp & 3, grp = warp >> 2;               // TMEM lane quarter, head group / column half
  const int trow = lq * 32 + lane;                        // the row this thread owns in the thread-per-row passes
  const uint32_t lane_b = (uint32_t)(lq * 32) << 16;
  uint32_t step_par = 0;
  int step = 0;
  int t_out = p.multistart ? 1 : 0;
#ifdef RRNCO_PHASE_STAMPS
  long long stamp_t0 = clock64();
#endif
  uint16_t* a_hi = reinterpret_cast<uint16_t*>(sm.A);     // [16-byte K chunk (16)][row (128)][8 halves]
  uint16_t* a_lo = a_hi + kRows * kE;
  constexpr float kUnscaleW = 1.0f / (kAScale * kWScale), kUnscaleL = 1.0f / (kAScale * kLkScale);

  while (true) {
    LSTAMP(24);
    const int all_done = lean_sync_and(tid < kRows ? (sm.done[tid] || !sm.active[tid]) : 1);  // own rows only: no race
    if (all_done) break;
    if (step >= p.max_steps) {  // policy.py:222-226: cut, but never silently
      if (tid == 0) atomicOr(p.status, RRNCO_DEV_TRUNCATED);
      break;
    }
    if (tid == 0) tc05::mbar_arrive(&sm.bar_step);
    LSTAMP(0);

    // ---- A: lane = (rollout of the warp's 16, 64-wide half of the columns): action-mask words of that half, then the
    // query rows q = ctx_proj[cur] + sum_k state_k w_k -> fp16 hi | lo core-matrix tiles (A operand of Q K^T) ----
    {
      const int row = warp * 16 + (lane & 15), dh = lane >> 4;
      const int cur = sm.cur[row];
      float st[kMaxState] = {0.f, 0.f, 0.f, 0.f};
      const float f0 = sm.f[0][row], f1 = sm.f[f1i][row], f2 = sm.f[f2i][row], f3 = sm.f[f3i][row];
      const float* src1;
      const float* src2 = nullptr;
      if (kEnv == RRNCO_ENV_ATSP) {
        if (p.use_placeholder && step == 0) {
          src1 = sm.wstate[0];
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
      float4 pq0[8];  // first half of the query row: in flight while the mask words are computed
#pragma unroll
      for (int cc = 0; cc < 8; ++cc) {
        pq0[cc] = *reinterpret_cast<const float4*>(src1 + dh * 64 + cc * 4);
        if (kEnv == RRNCO_ENV_ATSP && src2) {
          const float4 w = __ldg(reinterpret_cast<const float4*>(src2 + dh * 64 + cc * 4));
          pq0[cc] = make_float4(pq0[cc].x + w.x, pq0[cc].y + w.y, pq0[cc].z + w.z, pq0[cc].w + w.w);
        }
      }
      // action mask (rcvrp/env.py:183-195, rmtvrp/env.py:343-428, atsp/env.py:107-111): words 2 dh, 2 dh + 1
      {
        uint32_t bits2[2];
        const uint2 visw = *reinterpret_cast<const uint2*>(&sm.vis[row][2 * dh]);
        bool missing = false, carrying_b = false;
        uint32_t over2[2] = {0u, 0u};  // rcvrp: capacity-mask words 2 dh, 2 dh + 1
        if (kEnv == RRNCO_ENV_RCVRP) {
          int pos = 0;  // number of nodes, in demand order, that still fit: lower bound of the (monotone) predicate
#pragma unroll
          for (int stp = kRows / 2; stp >= 1; stp >>= 1)
            pos += __fadd_rn(sm.sdem[(pos + stp - 1) % SmemT::kSorted], f0) > cap ? 0 : stp;
          pos += __fadd_rn(sm.sdem[pos % SmemT::kSorted], f0) > cap ? 0 : 1;
          const uint2 sw = *reinterpret_cast<const uint2*>(&sm.sufmask[pos % (SmemT::kSorted + 1)][2 * dh]);
          over2[0] = sw.x;
          over2[1] = sw.y;
        }
        if (kEnv == RRNCO_ENV_RCVRPTW) {
          uint32_t m = (sm.lhmask[2 * dh] & ~visw.x) | (sm.lhmask[2 * dh + 1] & ~visw.y);
          m |= __shfl_xor_sync(0xffffffffu, m, 16);
          missing = m != 0u;  // linehauls_missing
          carrying_b = sm.node[iDemb][cur] > 0.f;
        }
#pragma unroll 1
        for (int k = 0; k < 2; ++k) {
          const int c0 = 64 * dh + 32 * k;
          const uint32_t valid = N >= c0 + 32 ? 0xffffffffu : (N > c0 ? (1u << (N - c0)) - 1u : 0u);
          uint32_t ok = ~(k ? visw.y : visw.x) & valid;
          if (kEnv == RRNCO_ENV_RCVRP) {
            ok &= ~over2[k];
          } else if (kEnv == RRNCO_ENV_RCVRPTW) {
            uint32_t good = 0u;
#pragma unroll 2
            for (int i = 0; i < 32; ++i) {
              const int c = c0 + i;
              if (c < N) {
                const float dist_ij = D[cur * N + c], dur_ij = U[cur * N + c];
                const float dem_c = sm.node[iDem][c], demb_c = sm.node[iDemb][c];
                const float arrival = __fadd_rn(f0, dur_ij);
                const bool reach_c = arrival < sm.node[iTw1][c];
                const bool reach_d =
                    __fmul_rn(__fadd_rn(__fadd_rn(fmaxf(arrival, sm.node[iTw0][c]), sm.node[iSvc][c]), sm.node[iUj0][c]), closed) <
                    sm.node[iTw1][0];
                const bool exc_lim = __fadd_rn(__fadd_rn(f1, dist_ij), __fmul_rn(sm.node[iDj0][c], closed)) > limit;
                const bool exc_l = __fadd_rn(dem_c, f2) > cap;
                const bool exc_b = __fadd_rn(demb_c, f3) > cap;
                const bool ok1 = (missing && !exc_l && !carrying_b && dem_c > 0.f) || (!exc_b && demb_c > 0.f);
                const bool cannot_l = dem_c > __fsub_rn(cap, f3);
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
      // query rows, 4 chunks of 8 dims at a time.  The 8 float4 loads of the first half were issued BEFORE the mask words were
      // computed (pq0: their L2 latency hides under the mask code), those of the second half before the first is processed.
      auto load_q = [&](int half, float4 (&pq)[8]) {
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) {
          pq[cc] = *reinterpret_cast<const float4*>(src1 + dh * 64 + half * 32 + cc * 4);
          if (kEnv == RRNCO_ENV_ATSP && src2) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(src2 + dh * 64 + half * 32 + cc * 4));
            pq[cc] = make_float4(pq[cc].x + w.x, pq[cc].y + w.y, pq[cc].z + w.z, pq[cc].w + w.w);
          }
        }
      };
      auto write_q = [&](int half, const float4 (&pq)[8]) {
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          const int c8 = dh * 8 + half * 4 + cc;
          float4 v0 = pq[2 * cc], v1 = pq[2 * cc + 1];
          if (kEnv != RRNCO_ENV_ATSP) {
#pragma unroll
            for (int k = 0; k < SmemT::kStateArrays; ++k) {
              const float4 w0 = *reinterpret_cast<const float4*>(&sm.wstate[k][c8 * 8]);
              const float4 w1 = *reinterpret_cast<const float4*>(&sm.wstate[k][c8 * 8 + 4]);
              v0.x = fmaf(st[k], w0.x, v0.x); v0.y = fmaf(st[k], w0.y, v0.y);
              v0.z = fmaf(st[k], w0.z, v0.z); v0.w = fmaf(st[k], w0.w, v0.w);
              v1.x = fmaf(st[k], w1.x, v1.x); v1.y = fmaf(st[k], w1.y, v1.y);
              v1.z = fmaf(st[k], w1.z, v1.z); v1.w = fmaf(st[k], w1.w, v1.w);
            }
          }
          uint32_t h[4], l[4];
          f16s_split2(v0.x, v0.y, kAScale, h[0], l[0]); f16s_split2(v0.z, v0.w, kAScale, h[1], l[1]);
          f16s_split2(v1.x, v1.y, kAScale, h[2], l[2]); f16s_split2(v1.z, v1.w, kAScale, h[3], l[3]);
          const int dst = c8 * (kRows * 8) + row * 8;
          *reinterpret_cast<uint4*>(&a_hi[dst]) = make_uint4(h[0], h[1], h[2], h[3]);
          *reinterpret_cast<uint4*>(&a_lo[dst]) = make_uint4(l[0], l[1], l[2], l[3]);
        }
      };
      {
        float4 pq1[8];
        load_q(1, pq1);
        write_q(0, pq0);
        write_q(1, pq1);
      }
    }
    tc05::fence_proxy_async();
    tc05::fence_before_sync();
    tc05::mbar_arrive(&sm.bar_q);
    LSTAMP(1);
    lean_sync();  // action-mask bitsets visible to the row-owner threads
    LSTAMP(2);

    // ---- C: attention.  Group g (warps 4g .. 4g+3) owns score buffer g and heads 4g .. 4g+3: masked softmax of the
    // thread's row, probabilities written back IN PLACE as the fp16 hi | lo A operand of P V; then, once P V(h) has
    // completed, glimpse_h = O_h / sum + q_h -> fp16 hi | lo tiles in place over the query tiles of head h ----
    {
      const int row = trow;
      const uint32_t t_s = tb + (uint32_t)grp * 128u + lane_b, t_o = t_s + 112u;
      // s = q . k / 4; the operands carry kAScale kKvScale.  exp(s - m) = ex2(c1 v - c1 vmax); + 4 = log2(kAScale)
      const float c1 = 0.25f * 1.4426950408889634f / (kAScale * kKvScale);
      uint32_t mrow[4];
      *reinterpret_cast<uint4*>(mrow) = *reinterpret_cast<const uint4*>(sm.mask[row]);
      bool bad_operand = false;
#pragma unroll 1
      for (int j = 0; j < 4; ++j) {
        const int h = 4 * grp + j;
        // Softmax shift.  Any shift m' >= max gives the same probabilities; the exact row maximum costs a pass over the
        // scores (a quarter of the softmax instructions), the Cauchy-Schwarz bound |q_h| max_k |k_h| costs ~30.  The fp16
        // hi | lo operands of P V resolve 2^-24 absolute, so the largest p must stay >= 1 after scaling: with p scaled by
        // 2^14 the bound may exceed the true maximum by 14 (log2 units), which holds whenever c1 vB <= 7 (scores within
        // +-4.8: every random-init and moderately peaked head).  Otherwise: the exact maximum, p scaled by 2^4 as before.
        // The bound needs the query tile only: it is computed BEFORE waiting for the scores of the head.
        float off, vB;
        {
          const uint4 q0 = *reinterpret_cast<const uint4*>(&a_hi[(2 * h) * (kRows * 8) + row * 8]);
          const uint4 q1 = *reinterpret_cast<const uint4*>(&a_hi[(2 * h + 1) * (kRows * 8) + row * 8]);
          const uint32_t qw[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
          float qn2 = 0.f;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&qw[e]));
            qn2 = fmaf(f.x, f.x, fmaf(f.y, f.y, qn2));
          }
          // v = sum (kAScale q)(kKvScale k) <= |Q_hi| (1 + 2^-10) kKvScale max|k_h|
          vB = sqrtf(qn2 * __uint_as_float(sm.kmax2[h])) * (kKvScale * 1.004f);
          off = fmaf(-c1, vB, 14.0f);
        }
        lean_wait_group(&sm.bar_s[h], step_par, warp);
        tc05::fence_after_sync();
        LSTAMP(3);
        // Both passes walk the row in 16-column blocks with the TMEM load of block k + 1 in flight while block k is
        // processed (a TMEM round trip is a few hundred cycles; two resident tiles do not hide it by themselves).
        const int nb16 = R16 >> 4;
        uint32_t va[16], vb[16];
        {
          // (warp-uniform decision: the TMEM loads below are warp-collective)
          if (__any_sync(0xffffffffu, !(c1 * vB <= 7.0f))) {
            // exact row maximum over the feasible keys
            float vm0 = -INFINITY, vm1 = -INFINITY;
            auto max_block = [&](const uint32_t (&v)[16], int kb) {
              const uint32_t mw = mrow[kb >> 1] >> (16 * (kb & 1));
#pragma unroll
              for (int i = 0; i < 16; i += 2) {
                vm0 = fmaxf(vm0, ((mw >> i) & 1u) ? __uint_as_float(v[i]) : -INFINITY);
                vm1 = fmaxf(vm1, ((mw >> (i + 1)) & 1u) ? __uint_as_float(v[i + 1]) : -INFINITY);
              }
            };
#pragma unroll 1
            for (int kb = 0; kb < nb16; ++kb) {
              tc05::tmem_ld16(t_s + kb * 16, va);
              tc05::tmem_wait_ld();
              max_block(va, kb);
            }
            off = fmaf(-c1, fmaxf(vm0, vm1), 4.0f);
          }
        }
        LSTAMP(4);
        // p = exp(s - m') (x 2^14 or 2^4), row sum, fp16 hi | lo split written back in place
        float2 sum01 = make_float2(0.f, 0.f);
        const float2 c1c1 = make_float2(c1, c1), offoff = make_float2(off, off);
        auto exp_block = [&](const uint32_t (&v)[16], int kb) {
          const uint32_t mw = mrow[kb >> 1] >> (16 * (kb & 1));
          uint32_t w[16];  // [hi (8 words) | lo (8 words)] of key block kb
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            const float2 a = ffma2(c1c1, make_float2(__uint_as_float(v[i]), __uint_as_float(v[i + 1])), offoff);
            const float e0 = ex2a(a.x), e1 = ex2a(a.y);
            const float2 pp = make_float2(((mw >> i) & 1u) ? e0 : 0.f, ((mw >> (i + 1)) & 1u) ? e1 : 0.f);
            sum01 = fadd2(sum01, pp);
            f16s_split_pair(pp, w[i >> 1], w[8 + (i >> 1)]);
          }
          tc05::tmem_st16(t_s + kb * 16, w);
        };
        tc05::tmem_ld16(t_s, va);
#pragma unroll 1
        for (int kb = 0; kb < nb16; kb += 2) {
          tc05::tmem_wait_ld();
          if (kb + 1 < nb16) tc05::tmem_ld16(t_s + (kb + 1) * 16, vb);
          exp_block(va, kb);
          if (kb + 1 < nb16) {
            tc05::tmem_wait_ld();
            if (kb + 2 < nb16) tc05::tmem_ld16(t_s + (kb + 2) * 16, va);
            exp_block(vb, kb + 1);
          }
        }
        tc05::tmem_wait_st();
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_p[h]);
        LSTAMP(5);
        // glimpse of head h (decoder.py:292-293)
        const float inv = __fdividef(kAScale, kKvScale * (sum01.x + sum01.y));  // glimpse scaled by kAScale, like the query tiles
        lean_wait_group(&sm.bar_o[h], step_par, warp);
        tc05::fence_after_sync();
        LSTAMP(6);
        uint32_t o[16];
        tc05::tmem_ld16(t_o, o);
        tc05::tmem_wait_ld();
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
          const int offq = (2 * h + cc) * (kRows * 8) + row * 8;
          const uint4 qh = *reinterpret_cast<const uint4*>(&a_hi[offq]);
          const uint4 ql = *reinterpret_cast<const uint4*>(&a_lo[offq]);
          const uint32_t qhw[4] = {qh.x, qh.y, qh.z, qh.w}, qlw[4] = {ql.x, ql.y, ql.z, ql.w};
          uint32_t hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&qhw[e]));
            const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&qlw[e]));
            const float2 gg = ffma2(make_float2(__uint_as_float(o[cc * 8 + 2 * e]), __uint_as_float(o[cc * 8 + 2 * e + 1])),
                                    make_float2(inv, inv), fadd2(fh, fl));
            const float g0 = gg.x, g1 = gg.y;
            // every operand overflow / NaN upstream of the FFN ends up here (a ReLU would swallow it later): keep it loud
            bad_operand |= !(fabsf(g0) < 65504.f) | !(fabsf(g1) < 65504.f);
            f16s_split_pair(gg, hi[e], lo[e]);
          }
          *reinterpret_cast<uint4*>(&a_hi[offq]) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<uint4*>(&a_lo[offq]) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
      }
      if (bad_operand) atomicOr(p.status, RRNCO_DEV_NAN_LOGITS);
      LSTAMP(7);
    }
    tc05::fence_proxy_async();
    tc05::fence_before_sync();
    tc05::mbar_arrive(&sm.bar_gready);  // glimpse tiles written, both O slots read: GEMM1 may start

    // ---- E: FFN epilogues.  Hidden chunk c (fp32, 128 columns): + b1, relu, fp16 hi | lo split written back IN PLACE
    // (16 fp32 columns of K step ks -> hi at 16 ks .. +7, lo at 16 ks + 8 .. +15) = the A operand of GEMM2(c) ----
    {
      const uint32_t t_h = tb + lane_b;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        lean_wait_all(&sm.bar_h, c & 1, warp);
        tc05::fence_after_sync();
        LSTAMP(9);
        uint32_t va[16], vb[16];
        auto epi_block = [&](const uint32_t (&v)[16], int q) {
          const int col0 = grp * 64 + q * 16;
          uint32_t w[16];
          float bb[16];
#pragma unroll
          for (int i = 0; i < 16; i += 4)
            *reinterpret_cast<float4*>(&bb[i]) = *reinterpret_cast<const float4*>(&sm.ffn_bias[c * kRows + col0 + i]);
#pragma unroll
          for (int i = 0; i < 16; i += 2) {
            // kAScale relu(acc / (kAScale kWScale) + b1): the scaled operand directly (b1 pre-scaled; powers of two: exact).
            // Non-finite accumulators cannot arise here: the operands of GEMM1 were checked where they were written.
            const float2 a = ffma2(make_float2(__uint_as_float(v[i]), __uint_as_float(v[i + 1])),
                                   make_float2(kAScale * kUnscaleW, kAScale * kUnscaleW), make_float2(bb[i], bb[i + 1]));
            f16s_split_pair(make_float2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f)), w[i >> 1], w[8 + (i >> 1)]);
          }
          tc05::tmem_st16(t_h + col0, w);
        };
        tc05::tmem_ld16(t_h + grp * 64, va);
        tc05::tmem_wait_ld();
        tc05::tmem_ld16(t_h + grp * 64 + 16, vb);
        epi_block(va, 0);
        tc05::tmem_wait_ld();
        tc05::tmem_ld16(t_h + grp * 64 + 32, va);
        epi_block(vb, 1);
        tc05::tmem_wait_ld();
        tc05::tmem_ld16(t_h + grp * 64 + 48, vb);
        epi_block(va, 2);
        tc05::tmem_wait_ld();
        epi_block(vb, 3);
        tc05::tmem_wait_st();
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_epi);
        LSTAMP(10);
      }
      lean_wait_all(&sm.bar_g2, step_par, warp);
      tc05::fence_after_sync();
      LSTAMP(11);
      // output epilogue: g' = acc + b2 + g -> fp16 hi | lo in place over the output accumulator (A operand of the logits)
      const uint32_t t_oa = tb + 128u + lane_b;
      const int row = trow;
#pragma unroll 1
      for (int q = 0; q < 4; ++q) {
        const int col0 = grp * 64 + q * 16;
        uint32_t v[16], w[16];
        tc05::tmem_ld16(t_oa + col0, v);
        float bb[16];
#pragma unroll
        for (int i = 0; i < 16; i += 4)
          *reinterpret_cast<float4*>(&bb[i]) = *reinterpret_cast<const float4*>(&sm.ffn_bias[kF + col0 + i]);
        tc05::tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; i += 8) {
          const int off = ((col0 + i) >> 3) * (kRows * 8) + row * 8;  // residual kAScale g = hi + lo, exact to 2^-24
          const uint4 gh = *reinterpret_cast<const uint4*>(&a_hi[off]);
          const uint4 gl = *reinterpret_cast<const uint4*>(&a_lo[off]);
          const uint32_t ghw[4] = {gh.x, gh.y, gh.z, gh.w}, glw[4] = {gl.x, gl.y, gl.z, gl.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&ghw[e]));
            const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&glw[e]));
            const float2 acc = ffma2(make_float2(__uint_as_float(v[i + 2 * e]), __uint_as_float(v[i + 2 * e + 1])),
                                     make_float2(kAScale * kUnscaleW, kAScale * kUnscaleW), make_float2(bb[i + 2 * e], bb[i + 2 * e + 1]));
            f16s_split_pair(fadd2(acc, fadd2(fh, fl)), w[(i >> 1) + e], w[8 + (i >> 1) + e]);
          }
        }
        tc05::tmem_st16(t_oa + col0, w);
      }
      tc05::tmem_wait_st();
      tc05::fence_before_sync();
      tc05::mbar_arrive(&sm.bar_lk);
      LSTAMP(12);
    }
    // bias rows of the rollouts (alpha . D[cur,:] + beta . Dur[cur,:]) -> fp32 tile in the (dead) activation region while
    // the logits MMAs run: coalesced, one warp per 16 rollouts, 8 rollouts at a time (up to 32 / 64 independent L2 loads in
    // flight per lane before the first store).  The loads of the first 8 are issued BEFORE the barrier that frees the
    // activation region (only the stores need it).
    {
      float* btile = reinterpret_cast<float*>(sm.A);
      float bias[8][4];
      auto load_rows = [&](int i0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int cur_s = sm.cur[warp * 16 + i0 + i];
#pragma unroll
          for (int cq = 0; cq < 4; ++cq) {
            const int c = cq * 32 + lane;
            float bv = 0.f;
            if (c < N) {
              bv = __fmul_rn(p.w.alpha, D[cur_s * N + c]);
              if (kEnv == RRNCO_ENV_RCVRPTW) bv = __fadd_rn(bv, __fmul_rn(p.w.beta, U[cur_s * N + c]));
#ifndef RRNCO_LEAN_SELECT3
              bv *= 1.4426950408889634f;  // the single-pass select works in log2 units
#endif
            }
            bias[i][cq] = bv;
          }
        }
      };
      auto store_rows = [&](int i0) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int cq = 0; cq < 4; ++cq) {
            const int c = cq * 32 + lane;
            if (c < R16) btile[(warp * 16 + i0 + i) * kLBiasLd + c] = bias[i][cq];
          }
      };
      load_rows(0);
      lean_sync();
      LSTAMP(13);  // every thread has read its residual: the activation region may be overwritten by the bias tile
      store_rows(0);
      load_rows(8);
      store_rows(8);
    }
    LSTAMP(14);
    lean_sync();
    LSTAMP(15);
    lean_wait_all(&sm.bar_acc, step_par, warp);
    tc05::fence_after_sync();
    LSTAMP(16);

#ifndef RRNCO_LEAN_SELECT3
    // ---- S: select, thread per row, SINGLE pass: two threads own one rollout, 16-column groups dealt round-robin.  Per
    // element: u = 2^(acc k1 - bias log2 e) + 1e-6 (decoder.py:198-201), v = clip (1 - 2 / (u^2 + 1)) (= clip tanh(log u)),
    // mask; sum of exp(v - shift) with the fixed shift clip / temperature while that bound is within kMaxFixedShift (no
    // maximum pass), else (low temperatures, large or no clipping) against a running maximum;
    // arg-max by a tree maximum per block + an index search only when the block improves it.  log p(chosen) =
    // (v - max) - log sum.  Greedy = arg-max v (lowest index on ties), sampling = arg-max v + Gumbel, evaluate = the forced
    // column.  (The three-pass form -- values rewritten to TMEM, sum pass, log-softmax pass -- is kept behind
    // RRNCO_LEAN_SELECT3: two TMEM round trips and two CTA barriers more per step.) ----
    {
      const int row = trow, colhalf = grp;
      const int64_t rg = (int64_t)(tile * kRows + (sm.active[row] ? row : 0)) * p.n_inst + b;
      const float k1 = 0.08838834764831845f * kUnscaleL * 1.4426950408889634f;  // raw accumulator -> logit in log2 units
      const float clip = p.w.tanh_clipping, temperature = p.w.temperature;
      const int hsh = 16 * colhalf;  // this thread's columns: 32 q + hsh + i
      const uint32_t t_l = tb + lane_b + hsh;
      const int nq = (R16 - hsh + 31) >> 5;  // 16-column groups of this thread (warp-uniform)
      const float* brow = reinterpret_cast<const float*>(sm.A) + row * kLBiasLd + hsh;  // bias in log2 units (gather above)
      // exchange between the two column halves of a row: behind the bias tile in the (dead) activation region
      float (*xf)[2][kRows] = reinterpret_cast<float (*)[2][kRows]>(sm.A + kLBiasBytes);            // [4][2][kRows]
      unsigned char (*xi)[kRows] = reinterpret_cast<unsigned char (*)[kRows]>(sm.A + kLBiasBytes + 4 * 2 * kRows * 4);
      uint32_t mrow[4];
      *reinterpret_cast<uint4*>(mrow) = *reinterpret_cast<const uint4*>(sm.mask[row]);
      int forced = -1;
      if (p.mode == RRNCO_DECODE_EVALUATE) {
        forced = step < p.forced_T ? (int)p.forced[rg * p.forced_T + step] : 0;
        forced = min(max(forced, 0), N - 1);
      }
      const uint2 key2 = make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32));
      const float mfix = clip > 0.f ? __fdiv_rn(clip, temperature) : INFINITY;
      const bool fixed_shift = mfix <= kMaxFixedShift;
      float m = fixed_shift ? mfix : -INFINITY;
      float ssum = 0.f, best = -INFINITY, bestv = -INFINITY, chk = 0.f;
      int besti = 255;
      float cut = -INFINITY;
      if constexpr (kFilter) {
        // top-k / top-p: the processed values (as computed below) go to TMEM in place and over this thread's own columns
        // of the bias tile; after the barrier both threads of the row find the same cut over the whole row, and the pass
        // below reads the values back and drops those under the cut like masked ones
        float* vrow = reinterpret_cast<float*>(sm.A) + row * kLBiasLd;
#pragma unroll 1
        for (int q = 0; q < nq; ++q) {
          uint32_t v[16];
          tc05::tmem_ld16(t_l + 32 * q, v);
          float bv[16];
#pragma unroll
          for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(&bv[i]) = *reinterpret_cast<const float4*>(brow + 32 * q + i);
          const uint32_t mq = mrow[q] >> hsh;
          tc05::tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            chk = fmaf(__uint_as_float(v[i]), 0.f, chk);
            const float u = __fadd_rn(ex2a(fmaf(__uint_as_float(v[i]), k1, -bv[i])), 1e-6f);
            float x;
            if (clip > 0.f) x = __fmul_rn(fmaf(-2.0f, rcpa(fmaf(u, u, 1.0f)), 1.0f), clip);
            else x = flog(u);
            x = ((mq >> i) & 1u) ? x : -INFINITY;
            if (temperature != 1.0f) x = __fdiv_rn(x, temperature);
            v[i] = __float_as_uint(x);
          }
          tc05::tmem_st16(t_l + 32 * q, v);
#pragma unroll
          for (int i = 0; i < 16; i += 4)
            *reinterpret_cast<uint4*>(vrow + hsh + 32 * q + i) = make_uint4(v[i], v[i + 1], v[i + 2], v[i + 3]);
        }
        tc05::tmem_wait_st();
        lean_sync();
        float vmax = -INFINITY;
        for (int c = 0; c < R16; ++c) vmax = fmaxf(vmax, vrow[c]);
        cut = filter_cut(FilterRowLocal{vrow, R16}, p.top_k, p.top_p, vmax);
      }
#pragma unroll 1
      for (int q = 0; q < nq; ++q) {
        uint32_t v[16];
        tc05::tmem_ld16(t_l + 32 * q, v);
        float bv[16];
#pragma unroll
        for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4*>(&bv[i]) = *reinterpret_cast<const float4*>(brow + 32 * q + i);
        const uint32_t mq = mrow[q] >> hsh;  // mask bits of columns >= N are never set
        const int cbase = 32 * q + hsh;
        tc05::tmem_wait_ld();
        float val[16];
        if constexpr (kFilter) {
#pragma unroll
          for (int i = 0; i < 16; ++i) val[i] = __uint_as_float(v[i]) < cut ? -INFINITY : __uint_as_float(v[i]);
        } else {
        if (clip > 0.f) {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            chk = fmaf(__uint_as_float(v[i]), 0.f, chk);  // NaN / Inf accumulators (fp16 operand overflow) -> NaN, masked columns too
            const float u = __fadd_rn(ex2a(fmaf(__uint_as_float(v[i]), k1, -bv[i])), 1e-6f);
            const float th = fmaf(-2.0f, rcpa(fmaf(u, u, 1.0f)), 1.0f);
            val[i] = ((mq >> i) & 1u) ? __fmul_rn(th, clip) : -INFINITY;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            chk = fmaf(__uint_as_float(v[i]), 0.f, chk);
            const float l = flog(__fadd_rn(ex2a(fmaf(__uint_as_float(v[i]), k1, -bv[i])), 1e-6f));
            val[i] = ((mq >> i) & 1u) ? l : -INFINITY;
          }
        }
        if (temperature != 1.0f) {
#pragma unroll
          for (int i = 0; i < 16; ++i) val[i] = __fdiv_rn(val[i], temperature);
        }
        }
        float bm = fmaxf(fmaxf(fmaxf(val[0], val[1]), fmaxf(val[2], val[3])), fmaxf(fmaxf(val[4], val[5]), fmaxf(val[6], val[7])));
        bm = fmaxf(bm, fmaxf(fmaxf(fmaxf(val[8], val[9]), fmaxf(val[10], val[11])), fmaxf(fmaxf(val[12], val[13]), fmaxf(val[14], val[15]))));
        if (!fixed_shift && bm > m) {  // running maximum
          ssum *= fexp(m - bm);
          m = bm;
        }
        const float ms2 = (m == -INFINITY ? 0.f : m) * 1.4426950408889634f;
#pragma unroll
        for (int i = 0; i < 16; ++i) ssum += ex2a(fmaf(val[i], 1.4426950408889634f, -ms2));
        if (p.mode == RRNCO_DECODE_SAMPLING) {
#pragma unroll 1
          for (int i4 = 0; i4 < 16; i4 += 4) {
            const float4 gn = gumbel4(make_uint4((uint32_t)rg, (uint32_t)(rg >> 32), (uint32_t)step, (uint32_t)((cbase + i4) >> 2)), key2);
            const float gv[4] = {gn.x, gn.y, gn.z, gn.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float x = i4 == 0 ? val[e] : i4 == 4 ? val[4 + e] : i4 == 8 ? val[8 + e] : val[12 + e];
              const float key = x + gv[e];
              const bool better = key > best;
              best = better ? key : best;
              bestv = better ? x : bestv;
              besti = better ? cbase + i4 + e : besti;
            }
          }
        } else {
          if (bm > best) {  // a new maximum: its first column (the groups come in increasing column order)
            best = bm;
            int idx = 15;
#pragma unroll
            for (int i = 14; i >= 0; --i) idx = val[i] == bm ? i : idx;
            besti = cbase + idx;
          }
          if (p.mode == RRNCO_DECODE_EVALUATE && (unsigned)(forced - cbase) < 16u) {
#pragma unroll
            for (int i = 0; i < 16; ++i) bestv = cbase + i == forced ? val[i] : bestv;
          }
        }
      }
      if (!(chk == 0.f)) atomicOr(p.status, RRNCO_DEV_NAN_LOGITS);
      if (p.mode == RRNCO_DECODE_GREEDY) bestv = best;
      xf[0][colhalf][row] = m;
      xf[1][colhalf][row] = ssum;
      xf[2][colhalf][row] = best;
      xf[3][colhalf][row] = bestv;
      xi[colhalf][row] = (unsigned char)besti;
      LSTAMP(17);
      lean_sync();
      LSTAMP(18);
      if (colhalf == 0) {
        const float m0 = xf[0][0][row], m1 = xf[0][1][row];
        const float mx = fmaxf(m0, m1);
        const float se = flog(xf[1][0][row] * fexp(m0 - mx) + xf[1][1][row] * fexp(m1 - mx));
        int win = 0;  // larger key wins, ties -> lower index
        if (xf[2][1][row] > xf[2][0][row] || (xf[2][1][row] == xf[2][0][row] && xi[1][row] < xi[0][row])) win = 1;
        int act = xi[win][row];
        if (act == 255) act = 0;
        if (p.mode == RRNCO_DECODE_EVALUATE) {
          act = forced;
          win = (act >> 4) & 1;  // the half that owns the forced column recorded its value
        }
        const float chosen = __fsub_rn(__fsub_rn(xf[3][win][row], mx), se);
        const bool feasible = (mrow[act >> 5] >> (act & 31)) & 1u;
        if (!feasible && sm.active[row]) atomicOr(p.status, RRNCO_DEV_INFEASIBLE);
        const bool count_leg = kEnv != RRNCO_ENV_ATSP || t_out > 0;
        len_acc += (double)lean_transition<kEnv>(sm, N, row, act, D, U, closed, count_leg);
        if (kEnv == RRNCO_ENV_ATSP && t_out == 0) sm.first[row] = (unsigned char)act;
        lp_acc += (double)chosen;
        if (sm.active[row] && t_out < p.t_cap) {
          p.actions[rg * p.t_cap + t_out] = act;
          if (p.logprob) p.logprob[rg * p.t_cap + t_out] = chosen;
        }
      }
    }
#else
    // ---- S: select, thread per row: two threads own one rollout, 16-column groups dealt round-robin; three rolled
    // passes over the logits, which stay in TMEM (pass A rewrites them in place) ----
    {
      const int row = trow, colhalf = grp;
      const int64_t rg = (int64_t)(tile * kRows + (sm.active[row] ? row : 0)) * p.n_inst + b;
      const float inv_sqrt_e = 0.08838834764831845f * kUnscaleL;  // 1 / sqrt(128), and the operand scales undone
      const float clip = p.w.tanh_clipping;
      const int hsh = 16 * colhalf;  // this thread's columns: 32 q + hsh + i
      const uint32_t t_l = tb + lane_b + hsh;
      const int nq = (R16 - hsh + 31) >> 5;  // 16-column groups of this thread (warp-uniform)
      const float* brow = reinterpret_cast<const float*>(sm.A) + row * kLBiasLd + hsh;
      // exchange between the two column halves of a row: behind the bias tile in the (dead) activation region
      float (*xf)[2][kRows] = reinterpret_cast<float (*)[2][kRows]>(sm.A + kLBiasBytes);            // [3][2][kRows]
      unsigned char (*xi)[kRows] = reinterpret_cast<unsigned char (*)[kRows]>(sm.A + kLBiasBytes + 3 * 2 * kRows * 4);
      uint32_t mrow[4];
      *reinterpret_cast<uint4*>(mrow) = *reinterpret_cast<const uint4*>(sm.mask[row]);
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
        const uint32_t mq = mrow[q] >> hsh;  // mask bits of columns >= N are never set
        tc05::tmem_wait_ld();
        if (clip > 0.f) {
          // clip * tanh(log u), u = exp(l - bias) + 1e-6 (decoder.py:198-201), as clip * (1 - 2 / (u^2 + 1))
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
      }
      tc05::tmem_wait_st();
      if (nan_seen) atomicOr(p.status, RRNCO_DEV_NAN_LOGITS);
      xf[0][colhalf][row] = mxl;
      LSTAMP(17);
      lean_sync();
      LSTAMP(18);
      const float mx = fmaxf(xf[0][0][row], xf[0][1][row]);
      // pass B: softmax denominator
      float sel = 0.f;
#pragma unroll 1
      for (int q = 0; q < nq; ++q) {
        uint32_t v[16];
        tc05::tmem_ld16(t_l + 32 * q, v);
        tc05::tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) sel += fexp(__uint_as_float(v[i]) - mx);
      }
      xf[1][colhalf][row] = sel;
      LSTAMP(19);
      lean_sync();
      LSTAMP(20);
      const float se = flog(xf[1][0][row] + xf[1][1][row]);
      // pass C: log-softmax in the reference's order; argmax of log p (greedy) or of log p + Gumbel noise (sampling);
      // evaluate: log p of the forced action
      int forced = -1;
      if (p.mode == RRNCO_DECODE_EVALUATE) {
        forced = step < p.forced_T ? (int)p.forced[rg * p.forced_T + step] : 0;
        forced = min(max(forced, 0), N - 1);
      }
      float best = -INFINITY, bestlp = -INFINITY;
      int besti = 255;
      const uint2 key2 = make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32));
#pragma unroll 1
      for (int q = 0; q < nq; ++q) {
        uint32_t v[16];
        tc05::tmem_ld16(t_l + 32 * q, v);
        tc05::tmem_wait_ld();
        const int cbase = 32 * q + hsh;
        if (p.mode == RRNCO_DECODE_SAMPLING) {
#pragma unroll 1
          for (int i4 = 0; i4 < 16; i4 += 4) {
            const float4 gn = gumbel4(make_uint4((uint32_t)rg, (uint32_t)(rg >> 32), (uint32_t)step, (uint32_t)((cbase + i4) >> 2)), key2);
            const float gv[4] = {gn.x, gn.y, gn.z, gn.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
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
      xf[2][colhalf][row] = best;
      xf[0][colhalf][row] = bestlp;  // xf[0] (row maxima) was last read before the previous barrier
      xi[colhalf][row] = (unsigned char)besti;
      LSTAMP(21);
      lean_sync();
      LSTAMP(22);
      int act = xi[0][row];  // larger key wins, ties -> lower index
      int win = 0;
      if (xf[2][1][row] > xf[2][0][row] || (xf[2][1][row] == xf[2][0][row] && xi[1][row] < act)) win = 1;
      act = xi[win][row];
      if (act == 255) act = 0;
      if (p.mode == RRNCO_DECODE_EVALUATE) {
        act = forced;
        win = (act >> 4) & 1;  // the half that owns the forced column recorded its log p
      }
      const float chosen = xf[0][win][row];
      if (colhalf == 0) {
        const bool feasible = (mrow[act >> 5] >> (act & 31)) & 1u;
        if (!feasible && sm.active[row]) atomicOr(p.status, RRNCO_DEV_INFEASIBLE);
        const bool count_leg = kEnv != RRNCO_ENV_ATSP || t_out > 0;
        len_acc += (double)lean_transition<kEnv>(sm, N, row, act, D, U, closed, count_leg);
        if (kEnv == RRNCO_ENV_ATSP && t_out == 0) sm.first[row] = (unsigned char)act;
        lp_acc += (double)chosen;
        if (sm.active[row] && t_out < p.t_cap) {
          p.actions[rg * p.t_cap + t_out] = act;
          if (p.logprob) p.logprob[rg * p.t_cap + t_out] = chosen;
        }
      }
    }
#endif
    LSTAMP(23);
    ++step;
    ++t_out;
    step_par ^= 1u;
  }

  // ---------------- exit: close the tours, publish per-rollout sums ----------------
  if (tid < kRows && sm.active[tid]) {  // tid < 128 = warps 0-3 = column half 0: the threads that own len_acc / lp_acc
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
    p.ws_len[r] = len_acc + (double)leg;
    p.ws_lp[r] = lp_acc;
  }
  if (tid == 0) {
    p.ws_tile_steps[blockIdx.x] = t_out;
    atomicMax(p.max_steps_out, t_out);
    sm.exit_flag = 1;
  }
  tc05::fence_before_sync();
  lean_sync();
  if (tid == 0) tc05::mbar_arrive(&sm.bar_step);  // releases the producer ...
  tc05::mbar_arrive(&sm.bar_q);                   // ... and the issuer (both see exit_flag)
  if (warp == 0) tc05::tmem_dealloc(sm.tmem_base, 256);
}

template <int kEnv, int kPasses, bool kFilter>
static int launch_lean(const RolloutParams& p, cudaStream_t st) {
  auto kern = rollout_lean_kernel<kEnv, kPasses, kFilter>;
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(LeanSmem<kEnv>)) != cudaSuccess ||
        cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  const int64_t grid = p.n_inst * p.n_tiles;
  if (grid <= 0 || grid > 0x7fffffffLL) return RRNCO_ERR_UNSUPPORTED;
  kern<<<(unsigned)grid, kLThreads, sizeof(LeanSmem<kEnv>), st>>>(p);
  return rrnco_launch_status();
}

// entry points used by rrnco_rollout (rollout_kernel.cu)
int64_t lean_kv_bytes(int32_t n_nodes, int64_t n_tiles_total) {
  const int64_t R16 = ((n_nodes + 15) >> 4) << 4;
  return n_tiles_total * 24 * R16 * 64;
}
int pack_ffn_lean(const float* w1, const float* w2, const float* b1, const float* b2, void* packed, uint32_t* status,
                  cudaStream_t st) {
  const int n = kLWSlices * kRows * 8;
  pack_ffn_lean_kernel<<<(n + 255) / 256, 256, 0, st>>>(w1, w2, b1, b2, reinterpret_cast<uint32_t*>(packed), status);
  return rrnco_launch_status();
}
int phase_cycles_lean(long long* h_out, int reset) {
  if (h_out && cudaMemcpyFromSymbol(h_out, g_lean_cycles, sizeof(long long) * 32) != cudaSuccess) return RRNCO_ERR_CUDA;
  if (reset) {
    long long z[32] = {0};
    if (cudaMemcpyToSymbol(g_lean_cycles, z, sizeof(z)) != cudaSuccess) return RRNCO_ERR_CUDA;
  }
  return RRNCO_OK;
}
int dispatch_env_lean(const RolloutParams& p, int env, int passes, cudaStream_t st) {
  static_assert(sizeof(LeanSmem<RRNCO_ENV_RCVRPTW>) <= 115712 && sizeof(LeanSmem<RRNCO_ENV_RCVRP>) <= 115712 &&
                    sizeof(LeanSmem<RRNCO_ENV_ATSP>) <= 115712, "two CTAs per SM need <= 113 KB of shared memory each");
  static_assert(kLBiasBytes + 4 * 2 * kRows * 4 + 2 * kRows <= kRows * kE * 4, "bias tile + exchange arrays fit the A region");
  if (rrnco_filter_active(p.top_k, p.top_p)) {
#ifdef RRNCO_LEAN_SELECT3
    return RRNCO_ERR_UNSUPPORTED;  // the filtered select is built on the single-pass form
#else
    switch (env) {
      case RRNCO_ENV_ATSP: return passes == 1 ? launch_lean<RRNCO_ENV_ATSP, 1, true>(p, st) : launch_lean<RRNCO_ENV_ATSP, 3, true>(p, st);
      case RRNCO_ENV_RCVRP: return passes == 1 ? launch_lean<RRNCO_ENV_RCVRP, 1, true>(p, st) : launch_lean<RRNCO_ENV_RCVRP, 3, true>(p, st);
      case RRNCO_ENV_RCVRPTW:
        return passes == 1 ? launch_lean<RRNCO_ENV_RCVRPTW, 1, true>(p, st) : launch_lean<RRNCO_ENV_RCVRPTW, 3, true>(p, st);
      default: return RRNCO_ERR_BAD_ARG;
    }
#endif
  }
  switch (env) {
    case RRNCO_ENV_ATSP: return passes == 1 ? launch_lean<RRNCO_ENV_ATSP, 1, false>(p, st) : launch_lean<RRNCO_ENV_ATSP, 3, false>(p, st);
    case RRNCO_ENV_RCVRP: return passes == 1 ? launch_lean<RRNCO_ENV_RCVRP, 1, false>(p, st) : launch_lean<RRNCO_ENV_RCVRP, 3, false>(p, st);
    case RRNCO_ENV_RCVRPTW:
      return passes == 1 ? launch_lean<RRNCO_ENV_RCVRPTW, 1, false>(p, st) : launch_lean<RRNCO_ENV_RCVRPTW, 3, false>(p, st);
    default: return RRNCO_ERR_BAD_ARG;
  }
}

}  // namespace rrnco
