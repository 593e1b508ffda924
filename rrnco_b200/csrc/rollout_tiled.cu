// Fused construction-rollout kernel for MORE THAN ONE KEY TILE (128 < N <= 1024 nodes; BASELINE config C4: ATSP n = 1000):
// the decode loop of RRNetPolicy.forward (rrnco/models/policy.py:203-243; decoder.py:281-306 per step) as one persistent
// launch, every contraction on tcgen05.mma.  Same building blocks as rollout_lean.cu (fp16 hi | lo three-term operands, ONE
// elected issuing thread in a fixed program order => bitwise reproducible, every B operand streamed through one TMA ring
// of 8 KB slices), with the key dimension tiled by 128:
//   * attention: pairs i = (head h, key tile t), i = h nT + t.  S_i = Q_h K_{h,t}^T (3 SS MMAs, N = 128) lands in one of
//     THREE score buffers (uses are numbered across sweeps and steps: use u -> buffer u % 3, so the scores of pair i + 2
//     are ready when a group finishes pair i); compute-warp group i & 1 turns it IN PLACE into unnormalised
//     probabilities (fp16 hi | lo) with a FIXED per-(row, head) softmax shift, so P V accumulates over the key tiles
//     without rescaling; O_h += P_i V_{h,t} (3 x 8 TS MMAs, N = 16) into the head's own 16 TMEM columns; row sums are
//     exchanged through shared memory; the glimpse epilogue runs once per step for all heads.
//     The shift: the Cauchy-Schwarz bound |q_h| max_k |k_h| when it is tight enough for the fp16 operand range
//     (CTA-uniform decision per step); otherwise a first sweep over all pairs with SINGLE-term scores (Q_hi K_hi^T, error
//     2^-10 of the bound) takes the masked row maxima, and the second sweep shifts by them.
//   * FFN 128 -> 512 -> 128: exactly the lean kernel's (one hidden accumulator converted in place to the A operand of GEMM2).
//   * pointer logits: one 128-key tile at a time into two TMEM buffers; the select pass is SINGLE-pass over each tile
//     (bias alpha.D[cur,:] (+ beta.Dur[cur,:]) read straight from L2, clip, mask; running maximum / sum / arg-max per
//     thread), merged across the two groups at the end: log p(chosen) = (v - max) - log sum exp(v - max).
//     Greedy = arg-max of v (lowest index on ties); sampling = arg-max of v + Gumbel noise (same Philox counters as the
//     other kernels); evaluate = the forced column.
// K / V / logit keys are packed once per INSTANCE (pack_kv_tiled_kernel) into 24 slices per key tile; all start tiles of an
// instance stream the same L2-resident pack.  TMEM (512 columns): scores 0 / 128 / 256, O of the 8 heads at 384 + 16 h;
// FFN hidden 0, output 128; logits 256 / 384.  One CTA per SM (~185 KB of shared memory).
// The bias rows are staged by cp.async (coalesced 16-byte pieces, XOR-swizzled) into per-group double buffers of 32
// columns inside the activation region (dead between the output epilogue and the next step): a thread-per-row read straight from global memory costs one L1 wavefront per element and bounded the select.
// A tile holds p.tile_rows <= 128 POMO starts (the launcher splits the starts of an instance over several CTAs when the
// grid would not fill the SMs); warps whose 32 rows are all padding skip every per-element pass.
// CTA PAIRS (kPair, a thread-block cluster of 2): when the tiles alone leave more than half of the SMs idle (config C4: 64
// tiles on 148 SMs) two CTAs share a tile.  Both hold the full rollout state and run the FFN redundantly; rank r computes
// the attention of heads 4 r .. 4 r + 3 only and writes its half of the glimpse tile into BOTH CTAs' activation tiles
// (st.shared::cluster), and it computes the logits / select pass of half of the key tiles only; the per-row partial
// results (maximum, sum, best key) are exchanged the same way and merged in rank order, so both CTAs take the same
// transition.  Cross-CTA ordering: remote mbarrier arrivals with release / acquire at cluster scope.
// Scores beyond the single-term sweep's reach (|q_h| max|k_h| / 4 > 350) raise RRNCO_DEV_SOFTMAX_RANGE:
// the host then runs the per-step pipeline (step_kernels.cu) instead -- loud, never silently inaccurate.
#include <cstdio>
#include "common.cuh"
#include "tc05.cuh"
#include "ffn_pack.cuh"
#include "rollout_common.cuh"

namespace rrnco {

constexpr int kGThreads = 320;             // warps 0-7 compute, 8 TMA producer, 9 MMA issue
constexpr int kGCompute = 256;
constexpr uint32_t kGStage = 8192;
constexpr int kGMaxNodes = RRNCO_MAX_NODES_FUSED;   // 1024
constexpr int kGWords = kGMaxNodes / 32;   // 32 mask words per rollout
constexpr int kGWordLd = kGWords + 1;      // padded row stride: thread-per-row accesses are conflict-free
constexpr int kGSlicesPerTile = 24;        // K heads 0-7 | V heads 8-15 | logit-key K steps 16-23
constexpr int kGJobs = 8, kGWSlices = kGJobs * 8;
int g_tiled_pairs = 1;  // rrnco_set_start_split(2) turns the CTA pairs off (development knob)

// per-phase cycle accumulator of thread 0 of CTA 0 (development builds: RRNCO_PHASE_STAMPS), read with rrnco_debug_phase_cycles
__device__ long long g_tiled_cycles[32];
#ifdef RRNCO_PHASE_STAMPS
#define GSTAMP(i)                                   \
  do {                                              \
    if (blockIdx.x == 0 && tid == 0) {              \
      const long long now_ = clock64();             \
      g_tiled_cycles[i] += now_ - stamp_t0;         \
      stamp_t0 = now_;                              \
    }                                               \
  } while (0)
#else
#define GSTAMP(i) do { } while (0)
#endif

template <int kEnv>
struct TiledSmem {
  static constexpr int kStages = kEnv == RRNCO_ENV_RCVRPTW ? 6 : 8;
  static constexpr int kNodeArrays = kEnv == RRNCO_ENV_RCVRPTW ? 7 : 1;
  static constexpr int kStateArrays = kEnv == RRNCO_ENV_RCVRPTW ? 4 : 1;
  static constexpr int kNodeLen = kEnv == RRNCO_ENV_ATSP ? 4 : kGMaxNodes;
  unsigned char A[kRows * kE * 4];         // Q -> glimpse (fp16 hi | lo tiles)
  unsigned char ring[kStages][kGStage];
  float ffn_bias[kF + kE];                 // kAScale b1 | kAScale b2 (shared-memory broadcast reads in the FFN epilogues)
  float wstate[kStateArrays][kE];          // context state weights; ATSP: row 0 = placeholder query
  float node[kNodeArrays][kNodeLen];       // dem | demb tw0 tw1 svc dj0 uj0 (rcvrptw)
  float f[kStateArrays][kRows];            // rcvrp: used | rcvrptw: time, route, used_l, used_b
  uint32_t vis[kRows][kGWordLd];
  uint32_t mask[kRows][kGWordLd];
  float psum[2][kH][kRows];                // softmax row sums of the two groups
  float pmax[2][kH][kRows];                // masked row maxima of the single-term scores (exact-shift sweep)
  float xf[4][2][kRows];                   // select exchange: running max, sum, best key, value at the best / forced column
  int xi[2][kRows];
  float xpf[4][kRows];                     // CTA pair: the peer's per-row partial of the select pass (written remotely)
  int xpi[kRows];
  uint16_t cur[kRows], first[kRows], cnt[kRows];
  unsigned char active[kRows], done[kRows];
  uint32_t lhmask[kGWords];
  uint32_t kmax2[kH];
  uint64_t bar_full[kStages], bar_empty[kStages];
  uint64_t bar_step;      // compute -> producer: another decode step follows (or exit)
  uint64_t bar_q;         // compute -> issuer: query tiles written (256 arrivals; also the exit signal)
  uint64_t bar_mode;      // compute -> producer: sm.need_max of this step is valid
  uint64_t bar_s[3];      // issuer -> compute: scores of a pair in buffer b
  uint64_t bar_p[3];      // compute -> issuer: buffer b consumed (sweep 1) / probabilities written in place (128 arrivals)
  uint64_t bar_o;         // issuer -> compute: every P V of the step complete
  uint64_t bar_gready;    // compute -> issuer: glimpse tiles written (256 arrivals)
  uint64_t bar_h, bar_epi, bar_g2, bar_lk;  // FFN chain, as in rollout_lean.cu
  uint64_t bar_l[2];      // issuer -> group b: logits of a key tile in buffer b
  uint64_t bar_lfree[2];  // group b -> issuer: logits buffer b consumed (128 arrivals)
  uint64_t bar_xg;        // CTA pair: the peer's half of the glimpse tile has been written into this CTA's A (256 remote arrivals)
  uint64_t bar_xs;        // CTA pair: the peer's select partials have been written into xpf / xpi (128 remote arrivals)
  uint32_t tmem_base;
  volatile int exit_flag;
  volatile int need_max;  // this step runs the exact-shift sweep first (CTA-uniform)
};

// ---- thread-block cluster helpers (CTA pair) ----
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {  // every thread of both CTAs (used once, before any thread exits)
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_rank(const void* local_smem, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(r) : "r"(tc05::smem_u32(local_smem)), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_cluster_b32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared::cluster.b32 [%0], %1;\n" ::"r"(addr), "r"(v) : "memory");
}
// arrive on an mbarrier of the peer CTA; release at cluster scope: this thread's earlier (remote) stores are visible to
// whoever observes the phase completion with an acquire at cluster scope
__device__ __forceinline__ void mbar_arrive_remote(uint32_t remote_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];\n" ::"r"(remote_bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = tc05::smem_u32(bar);
  uint32_t ok = 0, polls = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(addr), "r"(parity), "r"(1000000u)
        : "memory");
    if (ok) break;
    if (++polls > (1u << 24)) __trap();
  }
}

__device__ __forceinline__ void tiled_sync() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }
__device__ __forceinline__ void tiled_wait_all(uint64_t* bar, uint32_t parity, int warp) {
  if (warp == 0) tc05::mbar_wait(bar, parity);
  asm volatile("bar.sync 4, 256;\n" ::: "memory");
}
__device__ __forceinline__ void tiled_wait_group(uint64_t* bar, uint32_t parity, int warp) {
  if ((warp & 3) == 0) tc05::mbar_wait(bar, parity);
  if (warp < 4) asm volatile("bar.sync 2, 128;\n" ::: "memory");
  else asm volatile("bar.sync 3, 128;\n" ::: "memory");
}
__device__ __forceinline__ void tiled_group_sync(int warp) {
  if (warp < 4) asm volatile("bar.sync 2, 128;\n" ::: "memory");
  else asm volatile("bar.sync 3, 128;\n" ::: "memory");
}
__device__ __forceinline__ int tiled_sync_or(int pred) {
  uint32_t r;
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t"
      "setp.ne.u32 q, %1, 0;\n\t"
      "bar.red.or.pred p, 1, 256, q;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(r)
      : "r"((uint32_t)pred)
      : "memory");
  return (int)r;
}
__device__ __forceinline__ int tiled_sync_and(int pred) {
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

// ---- once per rollout call: K / V / Lk of every instance -> fp16 hi | lo slices in the shared-memory layouts of the MMAs.
// One block per (instance, key tile of 128); slices of a tile (8 KB each, keys beyond N zero):
//   K_h (0-7), Lk_ks (16-23): [hi | lo][16-byte K chunk (2)][key (128)][8 halves]
//   V_h (8-15)              : [hi | lo][key chunk (16)][dim (16)][8 halves]        (V_h^T, K-major over the keys)
// kmax2[b][h] = max over the keys of |K_h row|^2 (fp32 bits; zero-initialised by the caller).
__global__ void __launch_bounds__(256) pack_kv_tiled_kernel(const float* __restrict__ Kc, const float* __restrict__ Vc,
                                                            const float* __restrict__ Lk, int N, int nT,
                                                            unsigned char* __restrict__ pack, uint32_t* __restrict__ kmax2) {
  __shared__ uint32_t s_max[kH];
  const int tid = threadIdx.x;
  const int64_t b = blockIdx.x / nT;
  const int t = blockIdx.x % nT;
  if (tid < kH) s_max[tid] = 0u;
  __syncthreads();
  uint4* slot = reinterpret_cast<uint4*>(pack + (size_t)blockIdx.x * (kGSlicesPerTile * kGStage));
  constexpr int kSliceU4 = kGStage / 16;  // 512
#pragma unroll 1
  for (int which = 0; which < 2; ++which) {
    const float* src = (which ? Lk : Kc) + b * (int64_t)N * kE;
    const float scale = which ? kLkScale : kKvScale;
    uint4* base = slot + (size_t)(which ? 16 : 0) * kSliceU4;
    for (int idx = tid; idx < kRows * 16; idx += 256) {
      const int r = idx >> 4, c8 = idx & 15, key = t * kRows + r;
      float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
      if (key < N) {
        v0 = __ldg(reinterpret_cast<const float4*>(src + (size_t)key * kE) + c8 * 2);
        v1 = __ldg(reinterpret_cast<const float4*>(src + (size_t)key * kE) + c8 * 2 + 1);
      }
      if (which == 0) {
        float n2 = v0.x * v0.x + v0.y * v0.y + v0.z * v0.z + v0.w * v0.w + v1.x * v1.x + v1.y * v1.y + v1.z * v1.z + v1.w * v1.w;
        n2 += __shfl_xor_sync(0xffffffffu, n2, 1);
        if ((c8 & 1) == 0) atomicMax(&s_max[c8 >> 1], __float_as_uint(n2));
      }
      uint32_t h[4], l[4];
      f16s_split2(v0.x, v0.y, scale, h[0], l[0]); f16s_split2(v0.z, v0.w, scale, h[1], l[1]);
      f16s_split2(v1.x, v1.y, scale, h[2], l[2]); f16s_split2(v1.z, v1.w, scale, h[3], l[3]);
      uint4* sl = base + (size_t)(c8 >> 1) * kSliceU4;
      sl[(c8 & 1) * kRows + r] = make_uint4(h[0], h[1], h[2], h[3]);
      sl[2 * kRows + (c8 & 1) * kRows + r] = make_uint4(l[0], l[1], l[2], l[3]);
    }
  }
  const float* vsrc = Vc + b * (int64_t)N * kE;
  uint4* vbase = slot + (size_t)8 * kSliceU4;
  for (int idx = tid; idx < kH * 16 * 16; idx += 256) {
    const int d = idx & 15, kc = (idx >> 4) & 15, hh = idx >> 8;
    float x[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int key = t * kRows + kc * 8 + j;
      x[j] = key < N ? __ldg(vsrc + (size_t)key * kE + hh * kDh + d) : 0.f;
    }
    uint32_t h[4], l[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) f16s_split2(x[2 * j], x[2 * j + 1], kKvScale, h[j], l[j]);
    uint4* sl = vbase + (size_t)hh * kSliceU4;
    sl[kc * 16 + d] = make_uint4(h[0], h[1], h[2], h[3]);
    sl[2 * kRows + kc * 16 + d] = make_uint4(l[0], l[1], l[2], l[3]);
  }
  __syncthreads();
  if (tid < kH) atomicMax(&kmax2[b * kH + tid], s_max[tid]);
}

// ---- env transition on the shared-memory state (one thread per row); returns the leg to add to the tour length ----
template <int kEnv>
__device__ __forceinline__ float tiled_transition(TiledSmem<kEnv>& sm, int N, int row, int a, const float* D, const float* U,
                                                  float closed, bool count_leg) {
  const int prev = sm.cur[row];
  float leg = 0.f;
  constexpr int kN = TiledSmem<kEnv>::kNodeArrays - 1, kS = TiledSmem<kEnv>::kStateArrays - 1;
  if (kEnv == RRNCO_ENV_ATSP) {
    if (count_leg) leg = D[(size_t)prev * N + a];
  } else if (kEnv == RRNCO_ENV_RCVRP) {
    leg = D[(size_t)prev * N + a];
    const int di = min(max(a - 1, 0), N - 2) + 1;  // clamp(a-1, 0, n_loc-1), dem[] is depot-shifted
    sm.f[0][row] = __fmul_rn(__fadd_rn(sm.f[0][row], sm.node[0][di]), a != 0 ? 1.0f : 0.0f);
  } else {
    const float away = a != 0 ? 1.0f : 0.0f;
    const float dist = D[(size_t)prev * N + a], dur = U[(size_t)prev * N + a];
    leg = a == 0 ? __fmul_rn(dist, closed) : dist;
    sm.f[0][row] = __fmul_rn(away, __fadd_rn(fmaxf(__fadd_rn(sm.f[0][row], dur), sm.node[min(2, kN)][a]), sm.node[min(4, kN)][a]));
    sm.f[min(1, kS)][row] = __fmul_rn(away, __fadd_rn(sm.f[min(1, kS)][row], dist));
    sm.f[min(2, kS)][row] = __fmul_rn(away, __fadd_rn(sm.f[min(2, kS)][row], sm.node[0][a]));
    sm.f[min(3, kS)][row] = __fmul_rn(away, __fadd_rn(sm.f[min(3, kS)][row], sm.node[min(1, kN)][a]));
  }
  const uint32_t bit = 1u << (a & 31), old = sm.vis[row][a >> 5];
  sm.vis[row][a >> 5] = old | bit;
  const int cnt = sm.cnt[row] + ((old & bit) ? 0 : 1);
  sm.cnt[row] = (uint16_t)cnt;
  sm.cur[row] = (uint16_t)a;
  sm.done[row] = cnt == N;
  return leg;
}

template <int kEnv, int kPasses, bool kPair>
__global__ void __launch_bounds__(kGThreads, 1) rollout_tiled_kernel(const RolloutParams p) {  // (168 registers: 3 of the 10 warps share one 16 K-register sub-partition)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  using SmemT = TiledSmem<kEnv>;
  SmemT& sm = *reinterpret_cast<SmemT*>(smem_raw);
  constexpr int kNA = SmemT::kNodeArrays - 1, kSA = SmemT::kStateArrays - 1;
  constexpr int iDem = 0, iDemb = kNA < 1 ? kNA : 1, iTw0 = kNA < 2 ? kNA : 2, iTw1 = kNA < 3 ? kNA : 3, iSvc = kNA < 4 ? kNA : 4,
                iDj0 = kNA < 5 ? kNA : 5, iUj0 = kNA < 6 ? kNA : 6;
  constexpr int f1i = kSA < 1 ? kSA : 1, f2i = kSA < 2 ? kSA : 2, f3i = kSA < 3 ? kSA : 3;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = p.N;
  const int nT = (N + kRows - 1) / kRows;              // key tiles
  const int W = (N + 31) >> 5;                         // mask words in use
  const int nb_last = ((N - (nT - 1) * kRows) + 15) >> 4;  // 16-key blocks of the last key tile
  const uint32_t rank = kPair ? cluster_rank() : 0u;           // CTA pair: which half of the heads / key tiles is mine
  const int tile_id = kPair ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile = tile_id % p.n_tiles;
  const int64_t b = tile_id / p.n_tiles;
  const int h_lo = kPair ? 4 * (int)rank : 0;                  // my attention heads [h_lo, h_lo + n_heads)
  constexpr int n_heads = kPair ? kH / 2 : kH;
  const int t_lo = kPair && rank ? (nT + 1) / 2 : 0;           // my logits key tiles [t_lo, t_hi)
  const int t_hi = kPair && !rank ? (nT + 1) / 2 : nT;
  const int rows_here = min(p.tile_rows, p.S - tile * p.tile_rows);  // real rollouts of this tile (rows beyond are padding)
  const int rows_on = min(kRows, (rows_here + 31) & ~31);            // rows of the warps that compute (padding rows among
                                                                     // them shadow the tile's first rollout)
  const int64_t drow = b % p.d.data_rows;
  const float* D = p.d.distance + drow * (int64_t)N * N;
  const float* U = kEnv == RRNCO_ENV_RCVRPTW ? p.d.duration + drow * (int64_t)N * N : nullptr;
  const float* P1 = p.c.ctx_node_proj + b * (int64_t)N * kE;
  const float* P2 = kEnv == RRNCO_ENV_ATSP ? p.c.ctx_node_proj2 + b * (int64_t)N * kE : nullptr;
  const float cap = kEnv == RRNCO_ENV_ATSP ? 0.f : p.d.vehicle_capacity[drow];
  float closed = 1.f, limit = INFINITY, bclass = 1.f;
  if (kEnv == RRNCO_ENV_RCVRPTW) {
    closed = p.d.open_route[drow] ? 0.f : 1.f;
    limit = p.d.distance_limit[drow];
    bclass = p.d.backhaul_class[drow];
  }
  // this instance's packed K / V / logit-key slices (24 per key tile), L2-resident for the whole rollout
  const unsigned char* pack = p.kv_pack + (size_t)b * ((size_t)nT * kGSlicesPerTile * kGStage);

  // ---------------- one-time staging ----------------
  if (warp == 0) tc05::tmem_alloc(&sm.tmem_base, 512);
  if (tid == 32) {
    for (int i = 0; i < SmemT::kStages; ++i) {
      tc05::mbar_init(&sm.bar_full[i], 1);
      tc05::mbar_init(&sm.bar_empty[i], 1);
    }
    tc05::mbar_init(&sm.bar_step, 1);
    tc05::mbar_init(&sm.bar_mode, 1);
    tc05::mbar_init(&sm.bar_q, kGCompute);
    for (int i = 0; i < 3; ++i) {
      tc05::mbar_init(&sm.bar_s[i], 1);
      tc05::mbar_init(&sm.bar_p[i], kGCompute / 2);
    }
    for (int i = 0; i < 2; ++i) {
      tc05::mbar_init(&sm.bar_l[i], 1);
      tc05::mbar_init(&sm.bar_lfree[i], kGCompute / 2);
    }
    tc05::mbar_init(&sm.bar_o, 1);
    tc05::mbar_init(&sm.bar_gready, kGCompute);
    tc05::mbar_init(&sm.bar_h, 1);
    tc05::mbar_init(&sm.bar_epi, kGCompute);
    tc05::mbar_init(&sm.bar_g2, 1);
    tc05::mbar_init(&sm.bar_lk, kGCompute);
    tc05::mbar_init(&sm.bar_xg, kGCompute);
    tc05::mbar_init(&sm.bar_xs, kGCompute / 2);
    tc05::fence_mbar_init();
    sm.exit_flag = 0;
    sm.need_max = 0;
    // max |K_h row|^2 over the keys, written by the pack kernel (kmax2 sits behind the slices of all instances)
    const uint32_t* km = reinterpret_cast<const uint32_t*>(p.kv_pack + (size_t)p.n_inst * ((size_t)nT * kGSlicesPerTile * kGStage));
    for (int i = 0; i < kH; ++i) sm.kmax2[i] = km[b * kH + i];
  }
  for (int i = tid; i < kF + kE; i += kGThreads) sm.ffn_bias[i] = p.ffn_bias_scaled[i];
  if (tid < kE) {
#pragma unroll
    for (int k = 0; k < SmemT::kStateArrays; ++k) {
      float w = 0.f;
      if (kEnv == RRNCO_ENV_ATSP) w = p.w.ctx_placeholder_q ? p.w.ctx_placeholder_q[tid] : 0.f;
      else if (k < p.n_state) w = p.w.ctx_state_w[k * kE + tid];
      sm.wstate[k][tid] = w;
    }
  }
  if (kEnv != RRNCO_ENV_ATSP) {
    for (int n = tid; n < kGMaxNodes; n += kGThreads) {
      float dem = 0.f, demb = 0.f, tw0 = 0.f, tw1 = 0.f, svc = 0.f, dj0 = 0.f, uj0 = 0.f;
      if (n < N) {
        if (kEnv == RRNCO_ENV_RCVRP) dem = n >= 1 ? p.d.demand[drow * (N - 1) + n - 1] : 0.f;
        if (kEnv == RRNCO_ENV_RCVRPTW) {
          dem = p.d.demand[drow * N + n];
          demb = p.d.demand_backhaul[drow * N + n];
          tw0 = p.d.time_windows[(drow * N + n) * 2];
          tw1 = p.d.time_windows[(drow * N + n) * 2 + 1];
          svc = p.d.service_time[drow * N + n];
          dj0 = D[(size_t)n * N];
          uj0 = U[(size_t)n * N];
        }
      }
      sm.node[iDem][n] = dem;
      if (kEnv == RRNCO_ENV_RCVRPTW) {
        sm.node[iDemb][n] = demb; sm.node[iTw0][n] = tw0; sm.node[iTw1][n] = tw1; sm.node[iSvc][n] = svc;
        sm.node[iDj0][n] = dj0; sm.node[iUj0][n] = uj0;
      }
    }
  }
  __syncthreads();
  if (tid < kGWords) {  // linehaul customers as a bitset (rmtvrp/env.py:381-383)
    uint32_t lh = 0u;
    if (kEnv == RRNCO_ENV_RCVRPTW)
      for (int i = 0; i < 32; ++i) lh |= (sm.node[iDem][tid * 32 + i] > 0.f ? 1u : 0u) << i;
    sm.lhmask[tid] = lh;
  }

  // ---------------- rollout state init ----------------
  const int num_loc = kEnv == RRNCO_ENV_ATSP ? N : N - 1;
  double len_acc = 0.0, lp_acc = 0.0;  // running tour length / log-likelihood of the row this thread transitions
  if (tid < kRows) {
    const int row = tid;
    const int s_real = tile * p.tile_rows + row;
    const int active = row < p.tile_rows && s_real < p.S;
    const int s = active ? s_real : tile * p.tile_rows;  // padded rows shadow the tile's first rollout
    const int64_t r = (int64_t)s * p.n_inst + b;
    sm.active[row] = (unsigned char)active;
    sm.first[row] = 0;
#pragma unroll
    for (int k = 0; k < SmemT::kStateArrays; ++k) sm.f[k][row] = 0.f;
    for (int k = 0; k < kGWordLd; ++k) { sm.vis[row][k] = 0u; sm.mask[row][k] = 0u; }
    sm.done[row] = 0;
    sm.cur[row] = 0;
    sm.cnt[row] = 0;
    if (p.multistart) {
      const int a0 = s % num_loc + (kEnv == RRNCO_ENV_ATSP ? 0 : 1);  // select_start_nodes
      len_acc += (double)tiled_transition<kEnv>(sm, N, row, a0, D, U, closed, /*count_leg=*/false);  // depot -> a0 (VRPs)
      sm.first[row] = (uint16_t)a0;
      if (active && rank == 0u) {
        p.actions[r * p.t_cap] = a0;
        if (p.logprob) p.logprob[r * p.t_cap] = 0.f;
      }
    }
  }
  tc05::fence_before_sync();
  __syncthreads();
  tc05::fence_after_sync();
  if (kPair) cluster_sync_all();  // the peer CTA has started and initialised its barriers: its shared memory may be written

  const int uwarp = __shfl_sync(0xffffffffu, warp, 0);  // warp index as a value the compiler knows to be warp-uniform
  const int n_pairs = n_heads * nT;
  if (uwarp == 8) {
    // ===== TMA producer: the slices of a decode step in the order the issuer consumes them =====
    if (tc05::elect_one()) {
      uint32_t st = 0, round = 0, step_par = 0;
      auto push = [&](const unsigned char* src) {
        if (round > 0) tc05::mbar_wait(&sm.bar_empty[st], (round - 1) & 1, 32);
        tc05::mbar_arrive_expect_tx(&sm.bar_full[st], kGStage);
        tc05::bulk_g2s(sm.ring[st], src, kGStage, &sm.bar_full[st]);
        if (++st == (uint32_t)SmemT::kStages) { st = 0; ++round; }
      };
      auto slice = [&](int t, int s) { return pack + ((size_t)t * kGSlicesPerTile + s) * kGStage; };
      while (true) {
        tc05::mbar_wait(&sm.bar_step, step_par, 64);
        step_par ^= 1u;
        if (sm.exit_flag) break;
        // attention: K(0), K(1), K(2) [both modes start with them], then -- once the mode of this step is known -- the
        // rest of the exact-shift sweep (K of every pair, then K(0..2) again), then V(i), K(i + 3);
        // pair i = (head i / nT, key tile i % nT)
        const int npre = min(3, n_pairs);
        for (int i = 0; i < npre; ++i) push(slice(i % nT, h_lo + i / nT));
        tc05::mbar_wait(&sm.bar_mode, step_par ^ 1u, 32);  // (step_par was flipped above: this step's phase)
        if (sm.need_max) {
          int h = h_lo + npre / nT, t = npre % nT;
#pragma unroll 1
          for (int i = npre; i < n_pairs; ++i) {
            push(slice(t, h));
            if (++t == nT) { t = 0; ++h; }
          }
          for (int i = 0; i < npre; ++i) push(slice(i % nT, h_lo + i / nT));
        }
        int h = h_lo, t = 0, h2 = h_lo + 3 / nT, t2 = 3 % nT;
#pragma unroll 1
        for (int i = 0; i < n_pairs; ++i) {
          push(slice(t, 8 + h));
          if (i + 3 < n_pairs) push(slice(t2, h2));
          if (++t == nT) { t = 0; ++h; }
          if (++t2 == nT) { t2 = 0; ++h2; }
        }
#pragma unroll 1
        for (int s = 0; s < kGWSlices; ++s) push(p.ffn_packed + (size_t)s * kGStage);
#pragma unroll 1
        for (int tt = t_lo; tt < t_hi; ++tt)
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) push(slice(tt, 16 + ks));
      }
    }
    return;
  }
  if (uwarp == 9) {
    // ===== MMA issue: one elected thread, fixed program order (bitwise reproducible accumulation) =====
    if (tc05::elect_one()) {
      const uint32_t tb = sm.tmem_base;
      const uint32_t t_hacc = tb, t_oacc = tb + 128, t_o = tb + 384, t_l = tb + 256;
      const uint32_t idesc = tc05::make_idesc_f16(128, 128);
      const uint32_t idesc_pv = tc05::make_idesc_f16(128, 16);
      const uint32_t q_addr = tc05::smem_u32(sm.A);
      const uint32_t a_lo_off = kRows * kE * 2;
      const uint32_t ring_addr = tc05::smem_u32(sm.ring[0]);
      constexpr uint32_t var_l = kGStage / 2;   // hi -> lo variant of a slice
      uint32_t st = 0, round = 0, step_par = 0;
      uint32_t u0 = 0u;                 // uses of the score buffers before the current sweep (use u -> buffer u % 3, phase u / 3)
      uint32_t n_l[2] = {0u, 0u};       // uses of the logits buffers so far (mbarrier phases)
      auto stage_wait = [&]() -> uint32_t {
        tc05::mbar_wait(&sm.bar_full[st], round & 1);
        tc05::fence_after_sync();
        return ring_addr + st * kGStage;
      };
      auto stage_release = [&]() {
        tc05::commit(&sm.bar_empty[st]);
        if (++st == (uint32_t)SmemT::kStages) { st = 0; ++round; }
      };
      // scores of pair i (head h) of the current sweep; `terms` = 1: Q_hi K_hi^T only (exact-shift sweep)
      auto issue_qk = [&](int i, int h, int terms) {
        const uint32_t bsel = (u0 + (uint32_t)i) % 3u;
        const uint32_t t_s = tb + bsel * 128u;
        const uint32_t kh = stage_wait();
        const uint32_t qh = q_addr + 2 * h * kLboTile;
        const uint64_t q_hi = tc05::make_desc(qh, kLboTile, kSbo), k_hi = tc05::make_desc(kh, kLboTile, kSbo);
        tc05::mma_ss_f16(t_s, q_hi, k_hi, idesc, 0u);
        if (terms == 3) {
          tc05::mma_ss_f16(t_s, tc05::make_desc(qh + a_lo_off, kLboTile, kSbo), k_hi, idesc, 1u);
          tc05::mma_ss_f16(t_s, q_hi, tc05::make_desc(kh + var_l, kLboTile, kSbo), idesc, 1u);
        }
        tc05::commit(&sm.bar_s[bsel]);
        stage_release();
      };
      auto wait_consumed = [&](int i) -> uint32_t {  // the compute group has finished with the buffer of pair i
        const uint32_t u = u0 + (uint32_t)i, bsel = u % 3u;
        tc05::mbar_wait(&sm.bar_p[bsel], (u / 3u) & 1u, 32);
        tc05::fence_after_sync();
        return bsel;
      };
      const int npre = min(3, n_pairs);
      while (true) {
        tc05::mbar_wait(&sm.bar_q, step_par, 32);
        if (sm.exit_flag) break;
        tc05::fence_after_sync();
        if (sm.need_max) {
          // sweep 1: single-term scores of every pair, consumed by the row-maximum pass
          for (int i = 0; i < npre; ++i) issue_qk(i, h_lo + i / nT, 1);
          int h2 = h_lo + 3 / nT, t2 = 3 % nT;
#pragma unroll 1
          for (int i = 0; i < n_pairs; ++i) {
            wait_consumed(i);
            if (i + 3 < n_pairs) issue_qk(i + 3, h2, 1);
            if (++t2 == nT) { t2 = 0; ++h2; }
          }
          u0 += (uint32_t)n_pairs;
        }
        for (int i = 0; i < npre; ++i) issue_qk(i, h_lo + i / nT, kPasses);
        int h = h_lo, t = 0, h2 = h_lo + 3 / nT, t2 = 3 % nT;
#pragma unroll 1
        for (int i = 0; i < n_pairs; ++i) {
          const uint32_t t_s = tb + wait_consumed(i) * 128u;
          const uint32_t vh = stage_wait();
          // V_h^T slice: 16 dims x keys, K-major: 256 B between 16-byte key chunks, 128 B between 8-dim groups;
          // P_hi at columns 16 j, P_lo at 16 j + 8 of the score buffer
          const int nks = t == nT - 1 ? nb_last : 8;
#pragma unroll 1
          for (int j = 0; j < nks; ++j) {
            const uint64_t v_hi = tc05::make_desc(vh + j * 512, 256, kSbo);
            tc05::mma_ts_f16(t_o + 16 * h, t_s + 16 * j, v_hi, idesc_pv, (t > 0 || j > 0) ? 1u : 0u);
            if (kPasses == 3) {
              tc05::mma_ts_f16(t_o + 16 * h, t_s + 16 * j + 8, v_hi, idesc_pv, 1u);
              tc05::mma_ts_f16(t_o + 16 * h, t_s + 16 * j, tc05::make_desc(vh + var_l + j * 512, 256, kSbo), idesc_pv, 1u);
            }
          }
          stage_release();
          if (i + 3 < n_pairs) issue_qk(i + 3, h2, kPasses);
          if (++t == nT) { t = 0; ++h; }
          if (++t2 == nT) { t2 = 0; ++h2; }
        }
        u0 += (uint32_t)n_pairs;
        tc05::commit(&sm.bar_o);
        tc05::mbar_wait(&sm.bar_gready, step_par, 32);
        tc05::fence_after_sync();
#pragma unroll 1
        for (int j = 0; j < kGJobs; ++j) {
          const int c = j >> 1, half = j & 1;
          if (half == 1) {  // hidden chunk c converted in place to the A operand of GEMM2(c)
            tc05::mbar_wait(&sm.bar_epi, c & 1, 32);
            tc05::fence_after_sync();
          }
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) {
            const uint32_t b_addr = stage_wait();
            const uint64_t b_hi = tc05::make_desc(b_addr, kLboTile, kSbo);
            const uint64_t b_lo = tc05::make_desc(b_addr + var_l, kLboTile, kSbo);
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
        // pointer logits, one key tile at a time: D[128 x 128] = g'(hi | lo in place over the output accumulator) . Lk_t^T
        tc05::mbar_wait(&sm.bar_lk, step_par, 32);
        tc05::fence_after_sync();
#pragma unroll 1
        for (int tt = t_lo; tt < t_hi; ++tt) {
          const int bsel = (tt - t_lo) & 1;
          if (n_l[bsel] > 0u) {  // the previous tile in this buffer has been consumed
            tc05::mbar_wait(&sm.bar_lfree[bsel], (n_l[bsel] - 1u) & 1u, 32);
            tc05::fence_after_sync();
          }
          ++n_l[bsel];
          const uint32_t t_lb = t_l + (uint32_t)bsel * 128u;
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) {
            const uint32_t lk = stage_wait();
            const uint64_t l_hi = tc05::make_desc(lk, kLboTile, kSbo);
            tc05::mma_ts_f16(t_lb, t_oacc + 16 * ks, l_hi, idesc, ks > 0 ? 1u : 0u);
            if (kPasses == 3) {
              tc05::mma_ts_f16(t_lb, t_oacc + 16 * ks + 8, l_hi, idesc, 1u);
              tc05::mma_ts_f16(t_lb, t_oacc + 16 * ks, tc05::make_desc(lk + var_l, kLboTile, kSbo), idesc, 1u);
            }
            stage_release();
          }
          tc05::commit(&sm.bar_l[bsel]);
        }
        step_par ^= 1u;
      }
    }
    return;
  }

  // ================= compute warps 0-7 =================
  const uint32_t tb = sm.tmem_base;
  const int lq = warp & 3, grp = warp >> 2;               // TMEM lane quarter, group (score / logits buffer)
  const int trow = lq * 32 + lane;                        // the row this thread owns in the thread-per-row passes
  const uint32_t lane_b = (uint32_t)(lq * 32) << 16;
  const bool warp_on = lq * 32 < rows_here;               // some of this warp's 32 rows are real rollouts
  uint32_t step_par = 0, u0 = 0u, n_lt = 0;               // uses of the score buffers before the current sweep / of this
                                                          // group's logits buffer so far
  int step = 0;
  int t_out = p.multistart ? 1 : 0;
  uint16_t* a_hi = reinterpret_cast<uint16_t*>(sm.A);     // [16-byte K chunk (16)][row (128)][8 halves]
  uint16_t* a_lo = a_hi + kRows * kE;
  constexpr float kUnscaleW = 1.0f / (kAScale * kWScale), kUnscaleL = 1.0f / (kAScale * kLkScale);
#ifdef RRNCO_PHASE_STAMPS
  long long stamp_t0 = clock64();
#endif

  while (true) {
    GSTAMP(15);
    const int all_done = tiled_sync_and(tid < kRows ? (sm.done[tid] || !sm.active[tid]) : 1);  // own rows only: no race
    if (all_done) break;
    if (step >= p.max_steps) {  // policy.py:222-226: cut, but never silently
      if (tid == 0) atomicOr(p.status, RRNCO_DEV_TRUNCATED);
      break;
    }
    if (tid == 0) tc05::mbar_arrive(&sm.bar_step);
    GSTAMP(0);

    // ---- A: lane = (rollout of the warp's 16, half of the mask words / of the query columns) ----
    int loose_bound = 0;
    if (warp * 16 < rows_on) {
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
      {
        const int colb = kPair ? 64 * (int)rank + 32 * dh : 64 * dh;
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) {
          pq0[cc] = *reinterpret_cast<const float4*>(src1 + colb + cc * 4);
          if (kEnv == RRNCO_ENV_ATSP && src2) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(src2 + colb + cc * 4));
            pq0[cc] = make_float4(pq0[cc].x + w.x, pq0[cc].y + w.y, pq0[cc].z + w.z, pq0[cc].w + w.w);
          }
        }
      }
      // action mask (rcvrp/env.py:183-195, rmtvrp/env.py:343-428, atsp/env.py:107-111): words [16 dh, 16 dh + 16)
      {
        const int w_lo = dh * (kGWords / 2), w_hi = min(W, w_lo + kGWords / 2);
        bool missing = false, carrying_b = false;
        if (kEnv == RRNCO_ENV_RCVRPTW) {
          uint32_t m = 0u;
          for (int w = w_lo; w < w_hi; ++w) m |= sm.lhmask[w] & ~sm.vis[row][w];
          m |= __shfl_xor_sync(0xffffffffu, m, 16);
          missing = m != 0u;  // linehauls_missing
          carrying_b = sm.node[iDemb][cur] > 0.f;
        }
        uint32_t any_ok = 0u, word0 = 0u;
#pragma unroll 1
        for (int w = w_lo; w < w_hi; ++w) {
          const int c0 = 32 * w;
          const uint32_t valid = N >= c0 + 32 ? 0xffffffffu : (1u << (N - c0)) - 1u;
          uint32_t ok = ~sm.vis[row][w] & valid;
          if (kEnv == RRNCO_ENV_RCVRP) {
            uint32_t bad = 0u;
#pragma unroll 8
            for (int i = 0; i < 32; ++i) bad |= (__fadd_rn(sm.node[iDem][c0 + i], f0) > cap ? 1u : 0u) << i;
            ok &= ~bad;
          } else if (kEnv == RRNCO_ENV_RCVRPTW) {
            uint32_t good = 0u;
#pragma unroll 2
            for (int i = 0; i < 32; ++i) {
              const int c = c0 + i;
              if (c < N) {
                const float dist_ij = D[(size_t)cur * N + c], dur_ij = U[(size_t)cur * N + c];
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
          if (kEnv != RRNCO_ENV_ATSP && w == 0) ok &= ~1u;  // the depot bit is decided below
          any_ok |= ok;
          if (w == 0) word0 = ok;
          else sm.mask[row][w] = ok;
        }
        any_ok |= __shfl_xor_sync(0xffffffffu, any_ok, 16);
        if (dh == 0) {
          if (kEnv != RRNCO_ENV_ATSP && !(cur == 0 && any_ok != 0u)) { word0 |= 1u; any_ok |= 1u; }
          if (any_ok == 0u) {  // cannot happen upstream for an unfinished rollout; keep the math finite
            if (sm.active[row] && !sm.done[row]) atomicOr(p.status, RRNCO_DEV_NO_FEASIBLE);
            word0 |= 1u;
          }
          sm.mask[row][0] = word0;
        }
      }
      // query rows, 4 chunks of 8 dims at a time.  A CTA of a pair needs the columns of its own heads only (the peer writes
      // the other half of the glimpse tile): 32 columns per lane instead of 64.  The 8 float4 loads of the first (only)
      // half were issued before the mask words were computed (pq0): their L2 latency hides under the mask code.
      auto load_q = [&](int half, float4 (&pq)[8]) {
        const int colb = kPair ? 64 * (int)rank + 32 * dh : 64 * dh + 32 * half;
#pragma unroll
        for (int cc = 0; cc < 8; ++cc) {
          pq[cc] = *reinterpret_cast<const float4*>(src1 + colb + cc * 4);
          if (kEnv == RRNCO_ENV_ATSP && src2) {
            const float4 w = __ldg(reinterpret_cast<const float4*>(src2 + colb + cc * 4));
            pq[cc] = make_float4(pq[cc].x + w.x, pq[cc].y + w.y, pq[cc].z + w.z, pq[cc].w + w.w);
          }
        }
      };
      auto write_q = [&](int half, const float4 (&pq)[8]) {
        const int colb = kPair ? 64 * (int)rank + 32 * dh : 64 * dh + 32 * half;
        float qn2 = 0.f;
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
          const int c8 = (colb >> 3) + cc;
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
          // |q_h|^2 over the two chunks of head c8 >> 1: is |q_h| max_k |k_h| / 4 (in log2 units) within the range the
          // Cauchy-Schwarz shift covers?  (same test as the shift computation of the attention sweep, with its margin)
          if ((cc & 1) == 0) qn2 = 0.f;
          qn2 += v0.x * v0.x + v0.y * v0.y + v0.z * v0.z + v0.w * v0.w + v1.x * v1.x + v1.y * v1.y + v1.z * v1.z + v1.w * v1.w;
          if (cc & 1)
            loose_bound |= !(sqrtf(qn2 * __uint_as_float(sm.kmax2[c8 >> 1])) * (0.25f * 1.4426950408889634f * 1.01f) <= 7.0f);
          uint32_t h[4], l[4];
          f16s_split2(v0.x, v0.y, kAScale, h[0], l[0]); f16s_split2(v0.z, v0.w, kAScale, h[1], l[1]);
          f16s_split2(v1.x, v1.y, kAScale, h[2], l[2]); f16s_split2(v1.z, v1.w, kAScale, h[3], l[3]);
          const int dst = c8 * (kRows * 8) + row * 8;
          *reinterpret_cast<uint4*>(&a_hi[dst]) = make_uint4(h[0], h[1], h[2], h[3]);
          *reinterpret_cast<uint4*>(&a_lo[dst]) = make_uint4(l[0], l[1], l[2], l[3]);
        }
      };
      if (kPair) {
        write_q(0, pq0);
      } else {
        float4 pq1[8];
        load_q(1, pq1);
        write_q(0, pq0);
        write_q(1, pq1);
      }
    }
    {  // row sums of the softmax start from zero
      float* ps = &sm.psum[0][0][0];
#pragma unroll
      for (int k = 0; k < (2 * kH * kRows) / kGCompute; ++k) ps[tid + k * kGCompute] = 0.f;
    }
    tc05::fence_proxy_async();
    GSTAMP(1);
    // action-mask bitsets / zeroed row sums visible to the row-owner threads; and the CTA-uniform mode of this step: is the
    // Cauchy-Schwarz bound of every (row, head) tight enough to serve as the softmax shift?
    const int need_max = tiled_sync_or(loose_bound);
    if (tid == 0) {
      sm.need_max = need_max;
      tc05::mbar_arrive(&sm.bar_mode);
    }
    tc05::fence_before_sync();
    tc05::mbar_arrive(&sm.bar_q);
    GSTAMP(2);

    // ---- C: attention.  Pair i of a sweep is use u0 + i of the score buffers (buffer u % 3, mbarrier phase u / 3) and
    // belongs to group i & 1.  s = q . k / 4; the operands carry kAScale kKvScale: exp(s - m) = ex2(c1 v + off) ----
    const float c1 = 0.25f * 1.4426950408889634f / (kAScale * kKvScale);
    if (need_max) {
      // sweep 1: masked row maxima of the single-term scores, per head
      const int row = trow;
      float mx0 = -INFINITY, mx1 = -INFINITY;
      int h = h_lo + grp / nT, t = grp % nT, hprev = h;
#pragma unroll 1
      for (int i = grp; i < n_pairs; i += 2) {
        if (h != hprev) {
          sm.pmax[grp][hprev][row] = fmaxf(mx0, mx1);
          mx0 = -INFINITY;
          mx1 = -INFINITY;
          hprev = h;
        }
        const uint32_t u = u0 + (uint32_t)i, bsel = u % 3u;
        tiled_wait_group(&sm.bar_s[bsel], (u / 3u) & 1u, warp);
        tc05::fence_after_sync();
        if (warp_on) {
          const uint32_t t_s = tb + bsel * 128u + lane_b;
          const int nb16 = t == nT - 1 ? nb_last : 8;
          uint32_t mrow[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) mrow[k] = sm.mask[row][min(4 * t + k, kGWords - 1)];
          uint32_t va[16], vb[16];
          auto max_block = [&](const uint32_t (&v)[16], int kb) {
            const uint32_t mw = mrow[kb >> 1] >> (16 * (kb & 1));
#pragma unroll
            for (int e = 0; e < 16; e += 2) {
              mx0 = fmaxf(mx0, ((mw >> e) & 1u) ? __uint_as_float(v[e]) : -INFINITY);
              mx1 = fmaxf(mx1, ((mw >> (e + 1)) & 1u) ? __uint_as_float(v[e + 1]) : -INFINITY);
            }
          };
          tc05::tmem_ld16(t_s, va);
#pragma unroll 1
          for (int kb = 0; kb < nb16; kb += 2) {
            tc05::tmem_wait_ld();
            if (kb + 1 < nb16) tc05::tmem_ld16(t_s + (kb + 1) * 16, vb);
            max_block(va, kb);
            if (kb + 1 < nb16) {
              tc05::tmem_wait_ld();
              if (kb + 2 < nb16) tc05::tmem_ld16(t_s + (kb + 2) * 16, va);
              max_block(vb, kb + 1);
            }
          }
        }
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_p[bsel]);
        t += 2;
        while (t >= nT) { t -= nT; ++h; }
      }
      sm.pmax[grp][hprev][row] = fmaxf(mx0, mx1);
      u0 += (uint32_t)n_pairs;
      GSTAMP(18);
      tiled_sync();  // both groups' maxima written
    }
    {
      // sweep 2: masked exp of the thread's row with the fixed shift, probabilities written back IN PLACE as the fp16
      // hi | lo A operand of P V
      const int row = trow;
      float off = 0.f, sum0 = 0.f, sum1 = 0.f;
      bool range_bad = false;
      int h = h_lo + grp / nT, t = grp % nT, hprev = -1;
#pragma unroll 1
      for (int i = grp; i < n_pairs; i += 2) {
        if (h != hprev) {
          hprev = h;
          sum0 = 0.f;
          sum1 = 0.f;
          // softmax shift of head h.  Cauchy-Schwarz bound (see rollout_lean.cu): p = 2^(c1 v - c1 vB + 14) <= 2^14; the
          // largest p of the row stays >= 1 (fp16 hi | lo resolves 2^-24 absolute) whenever c1 vB <= 7.  Otherwise the
          // masked row maximum of the single-term scores, which is within 2^-10 c1 vB of the true one: p <= 2^13.5.
          const uint4 q0 = *reinterpret_cast<const uint4*>(&a_hi[(2 * h) * (kRows * 8) + row * 8]);
          const uint4 q1 = *reinterpret_cast<const uint4*>(&a_hi[(2 * h + 1) * (kRows * 8) + row * 8]);
          const uint32_t qw[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
          float qn2 = 0.f;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&qw[e]));
            qn2 = fmaf(f.x, f.x, fmaf(f.y, f.y, qn2));
          }
          const float vB = sqrtf(qn2 * __uint_as_float(sm.kmax2[h])) * (kKvScale * 1.004f);
          if (need_max) {
            const float m = fmaxf(sm.pmax[0][h][row], sm.pmax[1][h][row]);
            off = m == -INFINITY ? 0.f : fmaf(-c1, m, 13.0f);
            range_bad |= warp_on && !(c1 * vB <= 512.0f);
          } else {
            off = fmaf(-c1, vB, 14.0f);
          }
        }
        GSTAMP(5);
        const uint32_t u = u0 + (uint32_t)i, bsel = u % 3u;
        tiled_wait_group(&sm.bar_s[bsel], (u / 3u) & 1u, warp);
        tc05::fence_after_sync();
        GSTAMP(3);
        if (warp_on) {
          const uint32_t t_s = tb + bsel * 128u + lane_b;
          const int nb16 = t == nT - 1 ? nb_last : 8;
          uint32_t mrow[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) mrow[k] = sm.mask[row][min(4 * t + k, kGWords - 1)];
          uint32_t va[16], vb[16];
          const float2 c1c1 = make_float2(c1, c1), offoff = make_float2(off, off);
          float2 sum01 = make_float2(sum0, sum1);
          auto exp_block = [&](const uint32_t (&v)[16], int kb) {
            const uint32_t mw = mrow[kb >> 1] >> (16 * (kb & 1));
            uint32_t w[16];  // [hi (8 words) | lo (8 words)] of key block kb
#pragma unroll
            for (int e = 0; e < 16; e += 2) {
              const float2 a = ffma2(c1c1, make_float2(__uint_as_float(v[e]), __uint_as_float(v[e + 1])), offoff);
              const float e0 = ex2a(a.x), e1 = ex2a(a.y);
              const float2 pp = make_float2(((mw >> e) & 1u) ? e0 : 0.f, ((mw >> (e + 1)) & 1u) ? e1 : 0.f);
              sum01 = fadd2(sum01, pp);
              f16s_split_pair(pp, w[e >> 1], w[8 + (e >> 1)]);
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
          sum0 = sum01.x;
          sum1 = sum01.y;
          sm.psum[grp][h][row] = sum0 + sum1;  // running sum of this group's tiles of head h
          tc05::tmem_wait_st();
        }
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_p[bsel]);
        GSTAMP(4);
        t += 2;
        while (t >= nT) { t -= nT; ++h; }
      }
      u0 += (uint32_t)n_pairs;
      if (range_bad) atomicOr(p.status, RRNCO_DEV_SOFTMAX_RANGE);
    }
    GSTAMP(5);
    tiled_sync();  // both groups' row sums written
    tiled_wait_all(&sm.bar_o, step_par, warp);
    tc05::fence_after_sync();
    GSTAMP(6);
    // glimpse of heads 4 grp .. 4 grp + 3 (decoder.py:292-293): O_h / sum + q_h -> fp16 hi | lo tiles in place over the query
    // (CTA pair: heads h_lo + 2 grp, + 1, written into the peer's tile as well)
    const uint32_t peer_a_hi = kPair ? map_to_rank(sm.A, rank ^ 1u) : 0u;
    if (warp_on) {
      const int row = trow;
      bool bad_operand = false;
#pragma unroll 1
      for (int j = 0; j < (kPair ? 2 : 4); ++j) {
        const int h = kPair ? h_lo + 2 * grp + j : 4 * grp + j;
        const float inv = __fdividef(kAScale, kKvScale * (sm.psum[0][h][row] + sm.psum[1][h][row]));
        uint32_t o[16];
        tc05::tmem_ld16(tb + 384u + 16u * h + lane_b, o);
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
            bad_operand |= !(fabsf(g0) < 65504.f) | !(fabsf(g1) < 65504.f);
            f16s_split_pair(gg, hi[e], lo[e]);
          }
          const uint4 whi = make_uint4(hi[0], hi[1], hi[2], hi[3]), wlo = make_uint4(lo[0], lo[1], lo[2], lo[3]);
          *reinterpret_cast<uint4*>(&a_hi[offq]) = whi;
          *reinterpret_cast<uint4*>(&a_lo[offq]) = wlo;
          if (kPair) {
            st_cluster_v4(peer_a_hi + 2u * offq, whi);
            st_cluster_v4(peer_a_hi + 2u * (offq + kRows * kE), wlo);
          }
        }
      }
      if (bad_operand) atomicOr(p.status, RRNCO_DEV_NAN_LOGITS);
    }
    if (kPair) {
      // my half of the glimpse tile is in the peer's A; wait for the peer's half in mine
      mbar_arrive_remote(map_to_rank(&sm.bar_xg, rank ^ 1u));
      if ((warp & 3) == 0) mbar_wait_cluster(&sm.bar_xg, step_par);
      tiled_group_sync(warp);
    }
    tc05::fence_proxy_async();
    tc05::fence_before_sync();
    tc05::mbar_arrive(&sm.bar_gready);  // glimpse tiles written, O slots read: GEMM1 may start
    GSTAMP(7);

    // ---- E: FFN epilogues (as in rollout_lean.cu) ----
    {
      const uint32_t t_h = tb + lane_b;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        tiled_wait_all(&sm.bar_h, c & 1, warp);
        tc05::fence_after_sync();
        GSTAMP(8);
        if (warp_on) {
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
        }
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_epi);
        GSTAMP(9);
      }
      tiled_wait_all(&sm.bar_g2, step_par, warp);
      tc05::fence_after_sync();
      GSTAMP(10);
      // output epilogue: g' = acc + b2 + g -> fp16 hi | lo in place over the output accumulator (A operand of the logits)
      const uint32_t t_oa = tb + 128u + lane_b;
      const int row = trow;
#pragma unroll 1
      for (int q = 0; q < (warp_on ? 4 : 0); ++q) {
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
          const int offg = ((col0 + i) >> 3) * (kRows * 8) + row * 8;  // residual kAScale g = hi + lo, exact to 2^-24
          const uint4 gh = *reinterpret_cast<const uint4*>(&a_hi[offg]);
          const uint4 gl = *reinterpret_cast<const uint4*>(&a_lo[offg]);
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
      GSTAMP(11);
    }

    // ---- S: select, single pass.  Group g owns logits buffer g and the key tiles t = g, g + 2, ...; thread per row ----
    {
      const int row = trow;
      const int cur = sm.cur[row];
      const int64_t rg = (int64_t)(tile * p.tile_rows + (sm.active[row] ? row : 0)) * p.n_inst + b;
      const float inv_sqrt_e = 0.08838834764831845f * kUnscaleL;  // 1 / sqrt(128), and the operand scales undone
      const float clip = p.w.tanh_clipping;
      const float temperature = p.w.temperature;
      const uint32_t t_l = tb + 256u + (uint32_t)grp * 128u + lane_b;
      const float* drow_p = D + (size_t)cur * N;
      const float* urow_p = kEnv == RRNCO_ENV_RCVRPTW ? U + (size_t)cur * N : nullptr;
      int forced = -1;
      if (p.mode == RRNCO_DECODE_EVALUATE) {
        forced = step < p.forced_T ? (int)p.forced[rg * p.forced_T + step] : 0;
        forced = min(max(forced, 0), N - 1);
      }
      const uint2 key2 = make_uint2((uint32_t)p.seed, (uint32_t)(p.seed >> 32));
      const float k1 = inv_sqrt_e * 1.4426950408889634f;  // raw accumulator -> logit in log2 units
      const float alpha2 = p.w.alpha * 1.4426950408889634f, beta2 = p.w.beta * 1.4426950408889634f;
      // with clipping every value is <= clip / temperature: a fixed shift for the sum of exp (no running maximum) while
      // that bound is within kMaxFixedShift
      const float mfix = clip > 0.f ? __fdiv_rn(clip, temperature) : INFINITY;
      const bool fixed_shift = mfix <= kMaxFixedShift;
      float m = fixed_shift ? mfix : -INFINITY;
      float ssum = 0.f, best = -INFINITY, bestv = -INFINITY, chk = 0.f;
      int besti = 0x7fffffff;
      // Bias rows alpha . D[cur, :]: a thread-per-row read from global memory is one L1 wavefront per ELEMENT (32 lanes, 32
      // rows), which bounded this pass.  Instead the group's 128 threads copy 32 columns of every row at a time with
      // cp.async: 16-byte pieces, eight consecutive lanes per row (coalesced), XOR-swizzled by the row so that the
      // thread-per-row float4 reads are conflict-free, into a double buffer in the (dead) activation region: group g owns
      // the bytes of chunks 8g .. 8g + 7 of the hi and of the lo tile, which only ITS threads read in the output epilogue --
      // so one group barrier after that epilogue frees them.  (The time-window env would need two matrices staged: it
      // keeps the direct loads.)
      constexpr bool kStage = kEnv != RRNCO_ENV_RCVRPTW;
      const int gt = tid & 127;
      const bool vec16 = (N & 3) == 0 && (reinterpret_cast<uintptr_t>(D) & 15u) == 0;
      auto bias_buf = [&](int buf) { return reinterpret_cast<float*>(sm.A + buf * (kRows * kE * 2) + grp * (kRows * 32 * 4)); };
      auto stage_chunk = [&](int c_lo, int buf) {  // columns [c_lo, c_lo + 32) of the rows that compute
        float* dstb = bias_buf(buf);
#pragma unroll 2
        for (int k = 0; k < 8; ++k) {
          const int q = gt + 128 * k, r = q >> 3, piece = q & 7;
          if (r < rows_on) {
            const int col = c_lo + piece * 4;
            const float* src = D + (size_t)sm.cur[r] * N + col;
            const uint32_t dst = tc05::smem_u32(dstb + r * 32 + ((piece ^ (r & 7)) << 2));
            if (vec16) {
              const int nbytes = max(0, min(16, (N - col) * 4));
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(nbytes > 0 ? src : D), "r"(nbytes));
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int nbytes = col + e < N ? 4 : 0;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(dst + 4 * e), "l"(nbytes ? src + e : D), "r"(nbytes));
              }
            }
          }
        }
        cp_async_commit();
      };
      int kchunk = 0;
      if (kStage) {
        tiled_group_sync(warp);  // every thread of the group has read its residual: the group's share of A is free
        if (t_lo + grp < t_hi) stage_chunk((t_lo + grp) * kRows, 0);
      }
#pragma unroll 1
      for (int t = t_lo + grp; t < t_hi; t += 2) {
        const int nb16 = t == nT - 1 ? nb_last : 8;
        const int nch = (nb16 + 1) >> 1;
        uint32_t mrow[4];
#pragma unroll 1
        for (int c = 0; c < nch; ++c) {
          if (kStage) {
            cp_async_wait<0>();
            tiled_group_sync(warp);  // chunk `kchunk` landed for every thread; everyone is done reading the other buffer
            if (c + 1 < nch) stage_chunk(t * kRows + (c + 1) * 32, (kchunk + 1) & 1);
            else if (t + 2 < t_hi) stage_chunk((t + 2) * kRows, (kchunk + 1) & 1);
          }
          if (c == 0) {
            GSTAMP(14);
            tiled_wait_group(&sm.bar_l[grp], n_lt & 1u, warp);
            ++n_lt;
            tc05::fence_after_sync();
            GSTAMP(12);
#pragma unroll
            for (int k = 0; k < 4; ++k) mrow[k] = sm.mask[row][min(4 * t + k, kGWords - 1)];
          }
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int kb = 2 * c + half;
            if (kb < nb16 && warp_on) {
            const int c0 = t * kRows + kb * 16;
            uint32_t v[16];
            tc05::tmem_ld16(t_l + kb * 16, v);
            float bv[16];
            if (kStage) {
              const float* srcb = bias_buf(kchunk & 1) + row * 32;
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 x = *reinterpret_cast<const float4*>(srcb + (((4 * half + j) ^ (row & 7)) << 2));
                bv[4 * j] = alpha2 * x.x; bv[4 * j + 1] = alpha2 * x.y;
                bv[4 * j + 2] = alpha2 * x.z; bv[4 * j + 3] = alpha2 * x.w;
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                float x = 0.f;
                if (c0 + i < N) {
                  x = alpha2 * __ldg(drow_p + c0 + i);
                  if (kEnv == RRNCO_ENV_RCVRPTW) x = fmaf(beta2, __ldg(urow_p + c0 + i), x);
                }
                bv[i] = x;
              }
            }
            const uint32_t mq = mrow[kb >> 1] >> (16 * (kb & 1));  // mask bits of columns >= N are never set
            tc05::tmem_wait_ld();
            float val[16];
            // l = acc / sqrt(128) (operand scales undone), u = exp(l - bias) + 1e-6 (decoder.py:198-201) in the log2 domain:
            // one FFMA per element (bv holds bias . log2 e); chk turns NaN / Inf accumulators (fp16 operand overflow,
            // ffn_pack.cuh) into NaN with one FFMA per element, masked columns included, like upstream's assert on the raw logits
            if (clip > 0.f) {
              // clip * tanh(log u) as clip * (1 - 2 / (u^2 + 1))
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                chk = fmaf(__uint_as_float(v[i]), 0.f, chk);
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
            float bm = fmaxf(fmaxf(fmaxf(val[0], val[1]), fmaxf(val[2], val[3])), fmaxf(fmaxf(val[4], val[5]), fmaxf(val[6], val[7])));
            bm = fmaxf(bm, fmaxf(fmaxf(fmaxf(val[8], val[9]), fmaxf(val[10], val[11])), fmaxf(fmaxf(val[12], val[13]), fmaxf(val[14], val[15]))));
            // sum of exp against a shift (masked columns contribute exp(-inf) = 0): the fixed bound clip / temperature
            // (kMaxFixedShift), otherwise the running maximum
            if (!fixed_shift && bm > m) {
              ssum *= fexp(m - bm);  // m = -inf: 0 (ssum is 0 then anyway)
              m = bm;
            }
            const float ms2 = (m == -INFINITY ? 0.f : m) * 1.4426950408889634f;
#pragma unroll
            for (int i = 0; i < 16; ++i) ssum += ex2a(fmaf(val[i], 1.4426950408889634f, -ms2));
            if (p.mode == RRNCO_DECODE_SAMPLING) {
#pragma unroll 1
              for (int i4 = 0; i4 < 16; i4 += 4) {
                const float4 gn = gumbel4(make_uint4((uint32_t)rg, (uint32_t)(rg >> 32), (uint32_t)step, (uint32_t)((c0 + i4) >> 2)), key2);
                const float gv[4] = {gn.x, gn.y, gn.z, gn.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float x = i4 == 0 ? val[e] : i4 == 4 ? val[4 + e] : i4 == 8 ? val[8 + e] : val[12 + e];
                  const float key = x + gv[e];
                  const bool better = key > best;
                  best = better ? key : best;
                  bestv = better ? x : bestv;
                  besti = better ? c0 + i4 + e : besti;
                }
              }
            } else {
              if (bm > best) {  // a new maximum: its first column (the blocks come in increasing column order)
                best = bm;
                int idx = 15;
#pragma unroll
                for (int i = 14; i >= 0; --i) idx = val[i] == bm ? i : idx;
                besti = c0 + idx;
              }
              if (p.mode == RRNCO_DECODE_EVALUATE && (unsigned)(forced - c0) < 16u) {
#pragma unroll
                for (int i = 0; i < 16; ++i) bestv = c0 + i == forced ? val[i] : bestv;
              }
            }
            }
          }
          ++kchunk;
        }
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_lfree[grp]);
        GSTAMP(13);
      }
      if (!(chk == 0.f)) atomicOr(p.status, RRNCO_DEV_NAN_LOGITS);
      if (p.mode == RRNCO_DECODE_GREEDY) bestv = best;
      sm.xf[0][grp][row] = m;
      sm.xf[1][grp][row] = ssum;
      sm.xf[2][grp][row] = best;
      sm.xf[3][grp][row] = bestv;
      sm.xi[grp][row] = besti;
      GSTAMP(14);
      tiled_sync();
      GSTAMP(16);
      if (grp == 0) {
        // this CTA's partial over its key tiles: the two groups merged (larger key wins, ties -> lower index)
        float m0 = sm.xf[0][0][row], m1 = sm.xf[0][1][row];
        float mx = fmaxf(m0, m1);
        // (under a running maximum a group whose key tiles are all masked for this row has m = -inf, s = 0)
        float tot = rescaled_sum(sm.xf[1][0][row], m0, mx) + rescaled_sum(sm.xf[1][1][row], m1, mx);
        int win = 0;
        if (sm.xf[2][1][row] > sm.xf[2][0][row] || (sm.xf[2][1][row] == sm.xf[2][0][row] && sm.xi[1][row] < sm.xi[0][row])) win = 1;
        float bkey = sm.xf[2][win][row], bval = sm.xf[3][win][row];
        int act = sm.xi[win][row];
        // evaluate: only the group that owns the forced column recorded its value (-inf elsewhere)
        if (p.mode == RRNCO_DECODE_EVALUATE) bval = fmaxf(sm.xf[3][0][row], sm.xf[3][1][row]);
        if (kPair) {
          // exchange the partial with the peer CTA and merge in RANK order: both CTAs compute bit-identical results
          const uint32_t peer = rank ^ 1u;
          st_cluster_b32(map_to_rank(&sm.xpf[0][row], peer), __float_as_uint(mx));
          st_cluster_b32(map_to_rank(&sm.xpf[1][row], peer), __float_as_uint(tot));
          st_cluster_b32(map_to_rank(&sm.xpf[2][row], peer), __float_as_uint(bkey));
          st_cluster_b32(map_to_rank(&sm.xpf[3][row], peer), __float_as_uint(bval));
          st_cluster_b32(map_to_rank(&sm.xpi[row], peer), (uint32_t)act);
          mbar_arrive_remote(map_to_rank(&sm.bar_xs, peer));
          mbar_wait_cluster(&sm.bar_xs, step_par);
          const float mp = sm.xpf[0][row], sp = sm.xpf[1][row], kp = sm.xpf[2][row], vp = sm.xpf[3][row];
          const int ip = sm.xpi[row];
          const float ma = rank ? mp : mx, mb = rank ? mx : mp;      // a = rank 0 (lower key tiles), b = rank 1
          const float sa = rank ? sp : tot, sb = rank ? tot : sp;
          const float ka = rank ? kp : bkey, kb2 = rank ? bkey : kp;
          const float va = rank ? vp : bval, vb2 = rank ? bval : vp;
          const int ia = rank ? ip : act, ib = rank ? act : ip;
          mx = fmaxf(ma, mb);
          tot = rescaled_sum(sa, ma, mx) + rescaled_sum(sb, mb, mx);
          const bool second = kb2 > ka || (kb2 == ka && ib < ia);
          bkey = second ? kb2 : ka;
          bval = p.mode == RRNCO_DECODE_EVALUATE ? fmaxf(va, vb2) : (second ? vb2 : va);
          act = second ? ib : ia;
        }
        if (warp_on) {
          const float se = flog(tot);
          if (act == 0x7fffffff) act = 0;
          if (p.mode == RRNCO_DECODE_EVALUATE) act = forced;
          const float chosen = __fsub_rn(__fsub_rn(bval, mx), se);
          const bool feasible = (sm.mask[row][act >> 5] >> (act & 31)) & 1u;
          if (!feasible && sm.active[row]) atomicOr(p.status, RRNCO_DEV_INFEASIBLE);
          const bool count_leg = kEnv != RRNCO_ENV_ATSP || t_out > 0;
          len_acc += (double)tiled_transition<kEnv>(sm, N, row, act, D, U, closed, count_leg);
          if (kEnv == RRNCO_ENV_ATSP && t_out == 0) sm.first[row] = (uint16_t)act;
          lp_acc += (double)chosen;
          if (sm.active[row] && t_out < p.t_cap && rank == 0u) {
            p.actions[rg * p.t_cap + t_out] = act;
            if (p.logprob) p.logprob[rg * p.t_cap + t_out] = chosen;
          }
        }
      }
    }
    GSTAMP(17);
    ++step;
    ++t_out;
    step_par ^= 1u;
  }

  // ---------------- exit: close the tours, publish per-rollout sums ----------------
  if (tid < kRows && sm.active[tid] && rank == 0u) {  // tid < 128 = group 0: the threads that own len_acc / lp_acc
    const int row = tid;
    const int64_t r = (int64_t)(tile * p.tile_rows + row) * p.n_inst + b;
    const int last = sm.cur[row];
    float leg;
    if (kEnv == RRNCO_ENV_ATSP) {
      leg = D[(size_t)last * N + sm.first[row]];
    } else {
      leg = D[(size_t)last * N];  // back to the depot (go_to = roll(go_from, -1), rcvrp/env.py:203)
      if (kEnv == RRNCO_ENV_RCVRPTW) leg = __fmul_rn(leg, closed);
    }
    p.ws_len[r] = len_acc + (double)leg;
    p.ws_lp[r] = lp_acc;
  }
  if (tid == 0) {
    if (rank == 0u) {
      p.ws_tile_steps[tile_id] = t_out;
      atomicMax(p.max_steps_out, t_out);
    }
    sm.exit_flag = 1;
  }
  tc05::fence_before_sync();
  tiled_sync();
  if (tid == 0) tc05::mbar_arrive(&sm.bar_step);  // releases the producer ...
  tc05::mbar_arrive(&sm.bar_q);                   // ... and the issuer (both see exit_flag)
  // CTA pair: neither CTA leaves while the other could still touch its shared memory.  (The step protocol already implies
  // it -- the last remote accesses precede the partner's last wait -- this makes it explicit; exited threads of the
  // producer / issuer warps count as arrived.)
  if (kPair) cluster_sync_all();
  if (warp == 0) tc05::tmem_dealloc(sm.tmem_base, 512);
}

template <int kEnv, int kPasses, bool kPair>
static int launch_tiled(const RolloutParams& p, cudaStream_t st) {
  auto kern = rollout_tiled_kernel<kEnv, kPasses, kPair>;
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TiledSmem<kEnv>)) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  const int64_t grid = p.n_inst * p.n_tiles * (kPair ? 2 : 1);
  if (grid <= 0 || grid > 0x7fffffffLL) return RRNCO_ERR_UNSUPPORTED;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kGThreads);
  cfg.dynamicSmemBytes = sizeof(TiledSmem<kEnv>);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kPair ? 2 : 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (cudaLaunchKernelEx(&cfg, kern, p) != cudaSuccess) return RRNCO_ERR_CUDA;
  return rrnco_launch_status();
}

// entry points used by rrnco_rollout (rollout_kernel.cu)
int64_t tiled_kv_bytes(int32_t n_nodes, int64_t n_inst) {
  const int64_t nT = (n_nodes + kRows - 1) / kRows;
  return n_inst * nT * kGSlicesPerTile * (int64_t)kGStage + ((n_inst * kH * 4 + 15) & ~15LL);
}
int pack_kv_tiled(const RolloutParams& p, cudaStream_t st) {
  const int nT = (p.N + kRows - 1) / kRows;
  const int64_t blocks = p.n_inst * nT;
  if (blocks <= 0 || blocks > 0x7fffffffLL) return RRNCO_ERR_UNSUPPORTED;
  uint32_t* kmax2 = reinterpret_cast<uint32_t*>(p.kv_pack + (size_t)blocks * (kGSlicesPerTile * kGStage));
  if (cudaMemsetAsync(kmax2, 0, (size_t)p.n_inst * kH * 4, st) != cudaSuccess) return RRNCO_ERR_CUDA;
  pack_kv_tiled_kernel<<<(unsigned)blocks, 256, 0, st>>>(p.c.glimpse_key, p.c.glimpse_val, p.c.logit_key, p.N, nT, p.kv_pack, kmax2);
  return rrnco_launch_status();
}
int phase_cycles_tiled(long long* h_out, int reset) {
  if (h_out && cudaMemcpyFromSymbol(h_out, g_tiled_cycles, sizeof(long long) * 32) != cudaSuccess) return RRNCO_ERR_CUDA;
  if (reset) {
    long long z[32] = {0};
    if (cudaMemcpyToSymbol(g_tiled_cycles, z, sizeof(z)) != cudaSuccess) return RRNCO_ERR_CUDA;
  }
  return RRNCO_OK;
}
// CTA pairs when the tiles leave more than half of the SMs idle
bool tiled_use_pairs(int64_t n_tiles_total) {
  const int sms = device_sm_count();
  return g_tiled_pairs && sms > 0 && 2 * n_tiles_total <= sms;
}
int dispatch_env_tiled(const RolloutParams& p, int env, int passes, cudaStream_t st) {
  static_assert(sizeof(TiledSmem<RRNCO_ENV_RCVRPTW>) <= 232448, "one CTA per SM: at most 227 KB of shared memory");
  static_assert(sizeof(TiledSmem<RRNCO_ENV_ATSP>) <= 232448 && sizeof(TiledSmem<RRNCO_ENV_RCVRP>) <= 232448, "shared memory");
  (void)passes;  // the key-tiled kernel is built fp32-faithful only (three-term products)
  auto launch = [&](bool pairs) -> int {
    switch (env) {
      case RRNCO_ENV_ATSP: return pairs ? launch_tiled<RRNCO_ENV_ATSP, 3, true>(p, st) : launch_tiled<RRNCO_ENV_ATSP, 3, false>(p, st);
      case RRNCO_ENV_RCVRP: return pairs ? launch_tiled<RRNCO_ENV_RCVRP, 3, true>(p, st) : launch_tiled<RRNCO_ENV_RCVRP, 3, false>(p, st);
      case RRNCO_ENV_RCVRPTW: return pairs ? launch_tiled<RRNCO_ENV_RCVRPTW, 3, true>(p, st) : launch_tiled<RRNCO_ENV_RCVRPTW, 3, false>(p, st);
      default: return RRNCO_ERR_BAD_ARG;
    }
  };
  if (tiled_use_pairs(p.n_inst * p.n_tiles)) {
    // a device partition that cannot co-schedule a 2-CTA cluster of this footprint refuses the launch: one CTA per tile then
    if (launch(true) == RRNCO_OK) return RRNCO_OK;
    (void)cudaGetLastError();
  }
  return launch(false);
}

}  // namespace rrnco
