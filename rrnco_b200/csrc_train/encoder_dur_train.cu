// Training hand-off of the encoder, rcvrptw: backward of the three-way (duration) gate of the neural adaptive bias
// (DistAngleFusion.forward with use_duration_matrix, rrnco/models/nn/attn_freenet.py:242-289), the forward of which is
// csrc/encoder_dur_kernel.cu (notation: that file's header).  Per pair, with gamma = scale dL/d out:
//     dO_x = gamma g_x,   dz_c = gamma g_c (O_c - sum_x g_x O_x),   r = tau (dz^T Wg2) . SiLU'(hp)      (r: an E-vector)
// and every one of the 19 parameter gradients needs only sums over the pairs:
//     A_x = sum r (on_x s_x)^T,  B_x = sum r on_x^T        (E x E, on_x = [w1_x s_x + b1_x > 0]: K = pairs, tcgen05)
//     rho = sum r,  sum dz sigma^T (3 x E),  sum dz,  sum dz.z,  sum gamma,  sum dO_x,
//     a1_x[k] = sum_{on_k} dO_x s_x,  a0_x[k] = sum_{on_k} dO_x
// which a few fp64 kernels turn into the nn.Linear layouts (nab_dur_fin*_kernel).  Nothing of size [B, N, N, E] exists.
//
// nab_dur_bwd_kernel<pass>: persistent, one CTA per SM (512 TMEM columns: the forward's 128-column accumulator plus three
// 128 x 128 fp32 weight-gradient accumulators; six would need 896, hence two passes over the pairs, each of which recomputes
// the forward).  Pass 0 accumulates A_0..A_2 (three fp16 hi|lo split terms), pass 1 B_0..B_2 (two terms: on_x is exact in
// fp16) and the small sums.  Per 128-pair tile:
//   1. the forward, operation for operation (same generation, same 72 MMAs in the same order against the same TMA-streamed
//      slices of `packed`): the g the backward sees is the forward's g;
//   2. epilogue, thread per pair: the logits as the forward forms them, then dz, dO and r.  r (times a power-of-two scale
//      that brings a bound on max |r| to [1024, 2048): gradients are tiny; nab_dur_bound_kernel) is staged in fp32
//      [unit][pair], then converted to the
//      K-major fp16 hi|lo operand [pair chunk][unit][8 pairs] -- the transposition the K = pairs contraction needs;
//   3. per source x the compute warps write the second operand (on_x s_x, or on_x) in the same layout and the issuer adds
//      8 K-steps into accumulator x.
// The phases are serial within a CTA (one operand buffer each); nothing overlaps but the TMA stream.
//
// Determinism: tiles are dealt to CTAs statically; each CTA's TMEM accumulators are fp32 sums in a fixed MMA order; the
// small sums are per-thread (fixed pair order) fp32 per tile, fp64 across tiles; the per-CTA partials are reduced in a fixed
// order in fp64.  No float atomics (the one integer atomicMax finds the bound on |r|, an order-free quantity): the
// gradients are bitwise identical run to run on one device.
#include "../csrc/common.cuh"
#include "../csrc/tc05.cuh"
#include "../csrc/ffn_pack.cuh"
#include "../../include/rrnco_b200_train.h"

namespace rrnco {

// layout of the forward's `packed` buffer (csrc/encoder_dur_kernel.cu, rrnco_nab_dur_pack); rrnco_train_nab_dur_packed_bytes()
// lets the host check it against rrnco_nab_dur_packed_bytes() of the rollout library
constexpr int kDbRows = 128;
constexpr uint32_t kDbStage = 8192;
constexpr int kDbStages = 4;
constexpr int kDbSlices = 24;
constexpr int kDbVec = 3 * kE * 3 + kE + 3 * kE;
constexpr int kDbConsts = 8;
constexpr int64_t kDbPackedBytes = (int64_t)kDbSlices * kDbStage + (kDbVec + kDbConsts) * 4;
constexpr int kDbThreads = 320;   // warps 0-7 compute, 8 TMA producer, 9 MMA issue
constexpr float kDbF16Max = 65504.f;
constexpr float kDbSScale = kAScale;  // pair scalars in the pass-0 operand: |s| < 4094 representable

// `params` / `grads`: the 19 tensors in the pointer order of rrnco_nab_dur_pack, concatenated
constexpr int kDbMlp = 3 * kE + kE * kE;     // emb.0.weight [E,1], emb.0.bias [E], emb.2.weight [E,E], emb.2.bias [E]
constexpr int kDbWg1 = 3 * kDbMlp;           // gate.0.weight [E, 3E]
constexpr int kDbBg1 = kDbWg1 + 3 * kE * kE; // gate.0.bias [E]
constexpr int kDbWg2 = kDbBg1 + kE;          // gate.2.weight [3, E]
constexpr int kDbBg2 = kDbWg2 + 3 * kE;      // gate.2.bias [3]
constexpr int kDbT = kDbBg2 + 3;             // gate_temperature [1]
constexpr int kDbWo = kDbT + 1;              // out_lin.weight [1, E]
constexpr int kDbBo = kDbWo + kE;            // out_lin.bias [1]
constexpr int kDbGrads = kDbBo + 1;

// per-CTA partials: the three accumulators of a pass (fp32, as TMEM holds them) | the small sums (fp64, pass 1), per
// column half h of the conversion threads: rho[2][E], dzs[2][3][E], a1[2][3][E], a0[2][3][E], then 8 scalars
// (sum dz_c (3), sum dz.z, sum gamma, sum dO_x (3))
constexpr int kDbAcc = 3 * kE * kE;
constexpr int kDbOffRho = 0, kDbOffDzs = 2 * kE, kDbOffA1 = 8 * kE, kDbOffA0 = 14 * kE, kDbOffSc = 20 * kE;
constexpr int kDbSmall = kDbOffSc + 8;

struct DurBwdSmem {
  unsigned char A[kDbRows * kE * 4];  // forward h_x operand | fp32 staging of r | second backward operand (on_x s_x or on_x)
  unsigned char R[kDbRows * kE * 4];  // r operand, hi | lo [pair chunk (16)][unit (128)][8 pairs] | pass 1: fp32 staging of sigma
  unsigned char ring[kDbStages][kDbStage];
  float vec[kDbVec + kDbConsts];
  float od[3][kDbRows];
  float xl[3][2][kDbRows];
  float s[3][kDbRows];     // the tile's pair scalars (cost, angle, duration)
  float dO[3][kDbRows];
  float dz[3][kDbRows];
  uint64_t bar_full[kDbStages], bar_empty[kDbStages];
  uint64_t bar_a;    // compute -> issuer: an operand tile written (256 arrivals)
  uint64_t bar_mma;  // issuer -> compute: the MMAs of one operand tile complete
  uint32_t tmem_base;
};
static_assert(sizeof(DurBwdSmem) <= 227 * 1024, "shared memory");

// fp32 staging [unit j][pair p], 16-pair chunks XOR-swizzled by the unit: the epilogue's stores (32 pairs of one unit) and the
// conversion's loads (8 pairs of consecutive units) stay (nearly) free of bank conflicts
__device__ __forceinline__ int stg(int j, int p) { return j * kDbRows + ((((p >> 3) ^ (j & 15))) << 3) + (p & 7); }

__device__ __forceinline__ void dsync() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }

// Bound on |r| before the passes, so that one power-of-two scale fits every tile: per pair
//     |r_j| <= tau (sum_c |wg2[c][j]|) 1.1 max_c |dz_c|,   |dz_c| <= |gamma| (max_x O_x - min_x O_x)      (SiLU' <= 1.0999)
// and the O_x need only the hidden vectors (no GEMM).  This kernel takes max over the pairs of |gamma| (max O - min O) as float
// bits (non-negative floats order like their bit patterns: an integer max, order-free; NaN counts as infinite).
__global__ void __launch_bounds__(256) nab_dur_bound_kernel(int N, int64_t n_pairs, const float* __restrict__ coords,
                                                            const float* __restrict__ cost, const float* __restrict__ dur,
                                                            int transpose, const unsigned char* __restrict__ packed, float scale,
                                                            const float* __restrict__ grad_out, uint32_t* __restrict__ out) {
  __shared__ float v[9 * kE];  // w1[3][E] b1[3][E] uo[3][E]
  __shared__ float co[3];
  const float* vsrc = reinterpret_cast<const float*>(packed + (size_t)kDbSlices * kDbStage);
  for (int i = threadIdx.x; i < 9 * kE; i += blockDim.x) v[i] = vsrc[i];
  if (threadIdx.x < 3) co[threadIdx.x] = vsrc[kDbVec + 3 + threadIdx.x];
  __syncthreads();
  const int64_t NN = (int64_t)N * N;
  uint32_t m = 0u;
  for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < n_pairs; p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = p / NN;
    const int r = (int)(p - b * NN), i = r / N, j = r - i * N;
    const int64_t src = transpose ? b * NN + (int64_t)j * N + i : p;
    const float2 pi = __ldg(reinterpret_cast<const float2*>(coords) + b * N + i);
    const float2 pj = __ldg(reinterpret_cast<const float2*>(coords) + b * N + j);
    const float sx[3] = {__ldg(cost + src), atan2f(pi.y - pj.y, pi.x - pj.x), __ldg(dur + src)};
    float omax = -INFINITY, omin = INFINITY;
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      float o = co[x];
      for (int k = 0; k < kE; ++k) o = fmaf(v[6 * kE + x * kE + k], fmaxf(fmaf(v[x * kE + k], sx[x], v[3 * kE + x * kE + k]), 0.f), o);
      omax = fmaxf(omax, o);
      omin = fminf(omin, o);
    }
    const float a = fabsf(scale * __ldg(grad_out + p)) * (omax - omin);
    m = max(m, a == a ? __float_as_uint(a) : 0x7f800000u);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, m);
}

// power of two bringing the bound on |r| to [1024, 2048) (vec: the forward's vectors, wg2 at 10 E, 1/exp(T) at kDbVec + 7);
// a non-finite bound: status
__device__ __forceinline__ float nab_dur_rscale(const uint32_t* bound_bits, const float* vec, uint32_t* status) {
  float w = 0.f;
  for (int j = 0; j < kE; ++j) w = fmaxf(w, fabsf(vec[10 * kE + j]) + fabsf(vec[11 * kE + j]) + fabsf(vec[12 * kE + j]));
  const float bound = __uint_as_float(*bound_bits) * vec[kDbVec + 7] * w * 1.1f;
  if (!(bound < INFINITY)) {
    atomicOr(status, RRNCO_DEV_NAN_LOGITS);
    return 1.f;
  }
  if (bound == 0.f) return 1.f;
  int e = 10 - ilogbf(bound);
  e = e > 120 ? 120 : (e < -120 ? -120 : e);
  return exp2f((float)e);
}

template <int kPass>
__global__ void __launch_bounds__(kDbThreads, 1) nab_dur_bwd_kernel(
    int N, int64_t n_pairs, const float* __restrict__ coords, const float* __restrict__ cost, const float* __restrict__ dur,
    int transpose, const unsigned char* __restrict__ packed, float scale, const float* __restrict__ grad_out,
    const uint32_t* __restrict__ gmax_bits, float* __restrict__ part_acc, double* __restrict__ part_small,
    uint32_t* __restrict__ status) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  DurBwdSmem& sm = *reinterpret_cast<DurBwdSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t n_tiles = (n_pairs + kDbRows - 1) / kDbRows;
  if (warp == 0) tc05::tmem_alloc(&sm.tmem_base, 512);
  if (tid == 32) {
    for (int i = 0; i < kDbStages; ++i) {
      tc05::mbar_init(&sm.bar_full[i], 1);
      tc05::mbar_init(&sm.bar_empty[i], 1);
    }
    tc05::mbar_init(&sm.bar_a, 256);
    tc05::mbar_init(&sm.bar_mma, 1);
    tc05::fence_mbar_init();
  }
  {
    const float* vsrc = reinterpret_cast<const float*>(packed + (size_t)kDbSlices * kDbStage);
    for (int i = tid; i < kDbVec + kDbConsts; i += kDbThreads) sm.vec[i] = vsrc[i];
  }
  tc05::fence_before_sync();
  __syncthreads();
  tc05::fence_after_sync();

  const int uwarp = __shfl_sync(0xffffffffu, warp, 0);
  if (uwarp == 8) {
    // ===== TMA producer: the forward's 24 weight slices per tile, source-major =====
    if (tc05::elect_one()) {
      uint32_t st = 0, round = 0;
      for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
#pragma unroll 1
        for (int s = 0; s < kDbSlices; ++s) {
          if (round > 0) tc05::mbar_wait(&sm.bar_empty[st], (round - 1) & 1);
          tc05::mbar_arrive_expect_tx(&sm.bar_full[st], kDbStage);
          tc05::bulk_g2s(sm.ring[st], packed + (size_t)s * kDbStage, kDbStage, &sm.bar_full[st]);
          if (++st == (uint32_t)kDbStages) { st = 0; ++round; }
        }
      }
    }
    return;
  }
  if (uwarp == 9) {
    // ===== MMA issue: one elected thread, fixed order =====
    if (tc05::elect_one()) {
      const uint32_t tb = sm.tmem_base;
      const uint32_t idesc = tc05::make_idesc_f16(128, 128);
      const uint32_t a_addr = tc05::smem_u32(sm.A), r_addr = tc05::smem_u32(sm.R), lo_off = kDbRows * kE * 2;
      const uint32_t ring_addr = tc05::smem_u32(sm.ring[0]);
      uint32_t st = 0, round = 0, n_a = 0, acc = 0;
      for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        // the forward (encoder_dur_kernel.cu, nab_dur_kernel): hp accumulator = columns [0, 128)
#pragma unroll 1
        for (int x = 0; x < 3; ++x) {
          tc05::mbar_wait(&sm.bar_a, n_a & 1u);
          ++n_a;
          tc05::fence_after_sync();
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) {
            tc05::mbar_wait(&sm.bar_full[st], round & 1);
            tc05::fence_after_sync();
            const uint32_t b_addr = ring_addr + st * kDbStage;
            const uint64_t b_hi = tc05::make_desc(b_addr, kLboTile, kSbo);
            const uint64_t b_lo = tc05::make_desc(b_addr + kDbStage / 2, kLboTile, kSbo);
            const uint64_t a_hi = tc05::make_desc(a_addr + ks * 2 * kLboTile, kLboTile, kSbo);
            tc05::mma_ss_f16(tb, a_hi, b_hi, idesc, (x > 0 || ks > 0) ? 1u : 0u);
            tc05::mma_ss_f16(tb, tc05::make_desc(a_addr + lo_off + ks * 2 * kLboTile, kLboTile, kSbo), b_hi, idesc, 1u);
            tc05::mma_ss_f16(tb, a_hi, b_lo, idesc, 1u);
            tc05::commit(&sm.bar_empty[st]);
            if (++st == (uint32_t)kDbStages) { st = 0; ++round; }
          }
          tc05::commit(&sm.bar_mma);
        }
        // the contractions over the tile's pairs: D_x[j, k] += sum_p r[p, j] b_x[p, k], accumulator x = columns 128 (x + 1)
#pragma unroll 1
        for (int x = 0; x < 3; ++x) {
          tc05::mbar_wait(&sm.bar_a, n_a & 1u);
          ++n_a;
          tc05::fence_after_sync();
          const uint32_t d = tb + 128u * (uint32_t)(x + 1);
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) {
            const uint64_t r_hi = tc05::make_desc(r_addr + ks * 2 * kLboTile, kLboTile, kSbo);
            const uint64_t r_lo = tc05::make_desc(r_addr + lo_off + ks * 2 * kLboTile, kLboTile, kSbo);
            const uint64_t b_hi = tc05::make_desc(a_addr + ks * 2 * kLboTile, kLboTile, kSbo);
            tc05::mma_ss_f16(d, r_hi, b_hi, idesc, (acc || ks > 0) ? 1u : 0u);
            tc05::mma_ss_f16(d, r_lo, b_hi, idesc, 1u);
            if (kPass == 0) tc05::mma_ss_f16(d, r_hi, tc05::make_desc(a_addr + lo_off + ks * 2 * kLboTile, kLboTile, kSbo), idesc, 1u);
          }
          tc05::commit(&sm.bar_mma);
        }
        acc = 1;
      }
    }
    return;
  }

  // ================= compute warps 0-7 =================
  const uint32_t tb = sm.tmem_base;
  const int lq = warp & 3, grp = warp >> 2;
  const int trow = lq * 32 + lane;
  const uint32_t lane_b = (uint32_t)(lq * 32) << 16;
  uint16_t* a_hi = reinterpret_cast<uint16_t*>(sm.A);
  uint16_t* a_lo = a_hi + kDbRows * kE;
  uint16_t* r_hi = reinterpret_cast<uint16_t*>(sm.R);
  uint16_t* r_lo = r_hi + kDbRows * kE;
  float* stage_r = reinterpret_cast<float*>(sm.A);
  float* stage_sig = reinterpret_cast<float*>(sm.R);
  const float* w1 = sm.vec;
  const float* b1 = sm.vec + 3 * kE;
  const float* uo = sm.vec + 6 * kE;
  const float* c0 = sm.vec + 9 * kE;
  const float* wg2 = sm.vec + 10 * kE;
  const float* cs = sm.vec + kDbVec;  // bg2[3] co[3] bo inv_temp
  constexpr float kUnscale = 1.0f / (kAScale * kWScale);
  const float rscale = nab_dur_rscale(gmax_bits, sm.vec, status), runscale = 1.0f / rscale;
  uint32_t n_m = 0;  // completed waits on bar_mma
  const int64_t NN = (int64_t)N * N;
  // conversion threads: unit (or output column) u, pair chunks hc, hc + 2, ..., hc + 14
  const int u = tid & 127, hc = tid >> 7;
  bool bad = false;  // an operand outside the fp16 range, or not finite
  double s_rho = 0.0, s_dzs[3] = {0.0, 0.0, 0.0}, s_a1[3] = {0.0, 0.0, 0.0}, s_a0[3] = {0.0, 0.0, 0.0};
  double s_sc[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};  // epilogue threads of column half 0: the per-pair scalar sums

  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    // ---- 1. the forward's generation (nab_dur_kernel), operation for operation ----
    const int grow = warp * 16 + (lane & 15), dh = lane >> 4;
    {
      const int64_t p = t * kDbRows + grow;
      float c = 0.f, th = 0.f, uu = 0.f;
      if (p < n_pairs) {
        const int64_t b = p / NN;
        const int r = (int)(p - b * NN), i = r / N, j = r - i * N;
        const int64_t src = transpose ? b * NN + (int64_t)j * N + i : p;
        c = __ldg(cost + src);
        uu = __ldg(dur + src);
        const float2 pi = __ldg(reinterpret_cast<const float2*>(coords) + b * N + i);
        const float2 pj = __ldg(reinterpret_cast<const float2*>(coords) + b * N + j);
        th = atan2f(pi.y - pj.y, pi.x - pj.x);
      }
      if (dh == 0) {
        sm.s[0][grow] = c;
        sm.s[1][grow] = th;
        sm.s[2][grow] = uu;
      }
#pragma unroll 1
      for (int x = 0; x < 3; ++x) {
        const float s = x == 0 ? c : (x == 1 ? th : uu);
        if (x > 0) {  // the MMAs that read the previous A tile have completed (x == 0: the end of the previous tile waited)
          if ((warp & 3) == 0) tc05::mbar_wait(&sm.bar_mma, n_m & 1u);
          dsync();
          ++n_m;
        }
        float od = 0.f, hmax = 0.f;
#pragma unroll 2
        for (int cc = 0; cc < 8; ++cc) {
          const int c8 = dh * 8 + cc, k0 = c8 * 8;
          float h[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            h[e] = fmaxf(fmaf(w1[x * kE + k0 + e], s, b1[x * kE + k0 + e]), 0.f);
            od = fmaf(uo[x * kE + k0 + e], h[e], od);
            hmax = fmaxf(hmax, h[e]);
          }
          uint32_t hh[4], ll[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) f16s_split2(h[2 * e], h[2 * e + 1], kAScale, hh[e], ll[e]);
          const int dst = c8 * (kDbRows * 8) + grow * 8;
          *reinterpret_cast<uint4*>(&a_hi[dst]) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
          *reinterpret_cast<uint4*>(&a_lo[dst]) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
        }
        if (!(hmax * kAScale < kDbF16Max)) atomicOr(status, RRNCO_DEV_NAN_LOGITS);
        od += __shfl_xor_sync(0xffffffffu, od, 16);
        if (dh == 0) sm.od[x][grow] = od;
        tc05::fence_proxy_async();
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_a);
      }
    }
    // ---- 2. epilogue: the forward's logits, then dz, dO and r (thread = pair `row`, column half `grp`) ----
    if ((warp & 3) == 0) tc05::mbar_wait(&sm.bar_mma, n_m & 1u);
    dsync();
    ++n_m;
    tc05::fence_after_sync();
    {
      const int row = trow;
      const int64_t p = t * kDbRows + row;
      float l0 = 0.f, l1 = 0.f, l2 = 0.f;
#pragma unroll 1
      for (int q = 0; q < 4; ++q) {
        const int col0 = grp * 64 + q * 16;
        uint32_t v[16];
        tc05::tmem_ld16(tb + lane_b + col0, v);
        tc05::tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float hp = fmaf(__uint_as_float(v[i]), kUnscale, c0[col0 + i]);
          const float si = hp / (1.0f + expf(-hp));
          l0 = fmaf(wg2[col0 + i], si, l0);
          l1 = fmaf(wg2[kE + col0 + i], si, l1);
          l2 = fmaf(wg2[2 * kE + col0 + i], si, l2);
        }
      }
      sm.xl[0][grp][row] = l0;
      sm.xl[1][grp][row] = l1;
      sm.xl[2][grp][row] = l2;
      dsync();
      const float z0 = (sm.xl[0][0][row] + sm.xl[0][1][row] + cs[0]) * cs[7];
      const float z1 = (sm.xl[1][0][row] + sm.xl[1][1][row] + cs[1]) * cs[7];
      const float z2 = (sm.xl[2][0][row] + sm.xl[2][1][row] + cs[2]) * cs[7];
      const float zm = fmaxf(z0, fmaxf(z1, z2));
      const float e0 = expf(z0 - zm), e1 = expf(z1 - zm), e2 = expf(z2 - zm);
      const float inv = 1.0f / (e0 + e1 + e2);
      const float O0 = sm.od[0][row] + cs[3], O1 = sm.od[1][row] + cs[4], O2 = sm.od[2][row] + cs[5];
      const float ob = (e0 * O0 + e1 * O1 + e2 * O2) * inv;
      const float gam = p < n_pairs ? scale * __ldg(grad_out + p) : 0.f;
      const float g0 = e0 * inv, g1 = e1 * inv, g2 = e2 * inv;
      const float dz0 = gam * g0 * (O0 - ob), dz1 = gam * g1 * (O1 - ob), dz2 = gam * g2 * (O2 - ob);
      if (kPass == 1 && grp == 0) {
        sm.dO[0][row] = gam * g0;
        sm.dO[1][row] = gam * g1;
        sm.dO[2][row] = gam * g2;
        sm.dz[0][row] = dz0;
        sm.dz[1][row] = dz1;
        sm.dz[2][row] = dz2;
        s_sc[0] += dz0;
        s_sc[1] += dz1;
        s_sc[2] += dz2;
        s_sc[3] += (double)dz0 * z0 + (double)dz1 * z1 + (double)dz2 * z2;
        s_sc[4] += gam;
        s_sc[5] += gam * g0;
        s_sc[6] += gam * g1;
        s_sc[7] += gam * g2;
      }
      // r_j = tau (sum_c dz_c wg2[c][j]) SiLU'(hp_j), times rscale, staged [j][pair]
      const float q0 = dz0 * cs[7] * rscale, q1 = dz1 * cs[7] * rscale, q2 = dz2 * cs[7] * rscale;
#pragma unroll 1
      for (int q = 0; q < 4; ++q) {
        const int col0 = grp * 64 + q * 16;
        uint32_t v[16];
        tc05::tmem_ld16(tb + lane_b + col0, v);
        tc05::tmem_wait_ld();
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int j = col0 + i;
          const float hp = fmaf(__uint_as_float(v[i]), kUnscale, c0[j]);
          const float sg = 1.0f / (1.0f + expf(-hp));
          stage_r[stg(j, row)] = fmaf(q0, wg2[j], fmaf(q1, wg2[kE + j], q2 * wg2[2 * kE + j])) * (sg * fmaf(hp, 1.0f - sg, 1.0f));
          if (kPass == 1) stage_sig[stg(j, row)] = hp / (1.0f + expf(-hp));
        }
      }
      tc05::fence_before_sync();
      dsync();
    }
    // ---- conversion: r -> the K-major fp16 hi|lo operand [pair chunk][unit][8 pairs]; pass 1: rho, sum dz sigma^T ----
    {
      if (kPass == 1) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll 2
        for (int i = 0; i < 8; ++i) {
          const int ch = hc + 2 * i;
          const float4* src = reinterpret_cast<const float4*>(stage_sig + stg(u, ch * 8));
          const float4 v0 = src[0], v1 = src[1];
          const float sv[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            a0 = fmaf(sm.dz[0][ch * 8 + e], sv[e], a0);
            a1 = fmaf(sm.dz[1][ch * 8 + e], sv[e], a1);
            a2 = fmaf(sm.dz[2][ch * 8 + e], sv[e], a2);
          }
        }
        s_dzs[0] += a0;
        s_dzs[1] += a1;
        s_dzs[2] += a2;
        dsync();  // sigma staging (in R) read by everyone before R is overwritten
      }
      float rs = 0.f;
#pragma unroll 2
      for (int i = 0; i < 8; ++i) {
        const int ch = hc + 2 * i;
        const float4* src = reinterpret_cast<const float4*>(stage_r + stg(u, ch * 8));
        const float4 v0 = src[0], v1 = src[1];
        const float rv[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
        uint32_t hh[4], ll[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          bad |= !(fabsf(rv[2 * e]) < kDbF16Max) || !(fabsf(rv[2 * e + 1]) < kDbF16Max);
          rs += rv[2 * e] + rv[2 * e + 1];
          f16s_split2(rv[2 * e], rv[2 * e + 1], 1.0f, hh[e], ll[e]);
        }
        const int dst = ch * (kDbRows * 8) + u * 8;
        *reinterpret_cast<uint4*>(&r_hi[dst]) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
        *reinterpret_cast<uint4*>(&r_lo[dst]) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
      }
      if (kPass == 1) s_rho += (double)(rs * runscale);
      dsync();  // r staging (in A) read by everyone before A is overwritten
    }
    // ---- 3. per source: the second operand [pair chunk][unit k][8 pairs], then 8 K-steps into accumulator x ----
#pragma unroll 1
    for (int x = 0; x < 3; ++x) {
      if (x > 0) {  // the MMAs that read the previous operand have completed
        if ((warp & 3) == 0) tc05::mbar_wait(&sm.bar_mma, n_m & 1u);
        dsync();
        ++n_m;
      }
      const float wk = w1[x * kE + u], bk = b1[x * kE + u];
      float sa1 = 0.f, sa0 = 0.f;
#pragma unroll 2
      for (int i = 0; i < 8; ++i) {
        const int ch = hc + 2 * i;
        float bv[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float s = sm.s[x][ch * 8 + e];
          const bool on = fmaf(wk, s, bk) > 0.f;  // the forward's relu(w1 s + b1) > 0
          if (kPass == 0) {
            bv[e] = on ? s : 0.f;
            bad |= !(fabsf(bv[e]) * kDbSScale < kDbF16Max);
          } else {
            bv[e] = on ? 1.f : 0.f;
            const float d = on ? sm.dO[x][ch * 8 + e] : 0.f;
            sa1 = fmaf(d, s, sa1);
            sa0 += d;
          }
        }
        uint32_t hh[4], ll[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) f16s_split2(bv[2 * e], bv[2 * e + 1], kPass == 0 ? kDbSScale : 1.0f, hh[e], ll[e]);
        const int dst = ch * (kDbRows * 8) + u * 8;
        *reinterpret_cast<uint4*>(&a_hi[dst]) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
        if (kPass == 0) *reinterpret_cast<uint4*>(&a_lo[dst]) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
      }
      if (kPass == 1) {
#pragma unroll
        for (int y = 0; y < 3; ++y)  // (register arrays: compile-time indices only)
          if (y == x) {
            s_a1[y] += sa1;
            s_a0[y] += sa0;
          }
      }
      tc05::fence_proxy_async();
      tc05::fence_before_sync();
      tc05::mbar_arrive(&sm.bar_a);
    }
    // the tile's last contraction has completed: every buffer may be rewritten by the next tile
    if ((warp & 3) == 0) tc05::mbar_wait(&sm.bar_mma, n_m & 1u);
    dsync();
    ++n_m;
  }
  if (bad) atomicOr(status, RRNCO_DEV_NAN_LOGITS);  // fp16 operand overflow or non-finite value: loud
  tc05::fence_after_sync();

  // ---- the CTA's partials ----
  {
    float* pa = part_acc + (size_t)blockIdx.x * kDbAcc;
#pragma unroll 1
    for (int x = 0; x < 3; ++x) {
#pragma unroll 1
      for (int q = 0; q < 4; ++q) {
        const int col0 = grp * 64 + q * 16;
        uint32_t v[16];
        tc05::tmem_ld16(tb + lane_b + 128u * (uint32_t)(x + 1) + col0, v);
        tc05::tmem_wait_ld();
        float* dst = pa + (size_t)x * kE * kE + (size_t)trow * kE + col0;
#pragma unroll
        for (int i = 0; i < 16; i += 4)
          *reinterpret_cast<float4*>(dst + i) = make_float4(__uint_as_float(v[i]), __uint_as_float(v[i + 1]),
                                                            __uint_as_float(v[i + 2]), __uint_as_float(v[i + 3]));
      }
    }
  }
  if (kPass == 1) {
    double* ps = part_small + (size_t)blockIdx.x * kDbSmall;
    ps[kDbOffRho + hc * kE + u] = s_rho;
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      ps[kDbOffDzs + (hc * 3 + x) * kE + u] = s_dzs[x];
      ps[kDbOffA1 + (hc * 3 + x) * kE + u] = s_a1[x];
      ps[kDbOffA0 + (hc * 3 + x) * kE + u] = s_a0[x];
    }
    // the per-pair scalars of the 128 column-half-0 threads, summed in thread order (A is free: every MMA has completed)
    double* red = reinterpret_cast<double*>(sm.A);
    if (grp == 0)
#pragma unroll
      for (int k = 0; k < 8; ++k) red[k * kDbRows + trow] = s_sc[k];
    dsync();
    if (tid < 8) {
      double a = 0.0;
      for (int r = 0; r < kDbRows; ++r) a += red[tid * kDbRows + r];
      ps[kDbOffSc + tid] = a;
    }
  }
  tc05::fence_before_sync();
  dsync();
  if (warp == 0) tc05::tmem_dealloc(tb, 512);
}

// totals[i] = sum over the CTA partials in a fixed order: block = 32 entries, warp w sums partials w, w + 8, ...
template <typename T>
__global__ void __launch_bounds__(256) nab_dur_reduce_kernel(int n_parts, int n, const T* __restrict__ partials,
                                                             double* __restrict__ totals) {
  __shared__ double red[8][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 32 + lane;
  double a = 0.0;
  if (i < n)
    for (int c = warp; c < n_parts; c += 8) a += (double)partials[(size_t)c * n + i];
  red[warp][lane] = a;
  __syncthreads();
  if (warp == 0 && i < n) {
    double t = red[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) t += red[w][lane];
    totals[i] = t;
  }
}

// totals (fp64): A[3][E][E] | B[3][E][E] | small sums (kDbSmall), the accumulators still scaled
struct DurTotals {
  const double* A;
  const double* B;
  const double* sm;
  double ua, ub;  // unscale of A / B
  __device__ double a(int x, int j, int k) const { return A[(x * kE + j) * kE + k] * ua; }
  __device__ double b(int x, int j, int k) const { return B[(x * kE + j) * kE + k] * ub; }
  __device__ double half2(int off, int x, int k) const { return sm[off + x * kE + k] + sm[off + (3 + x) * kE + k]; }
  __device__ double a1(int x, int k) const { return half2(kDbOffA1, x, k); }
  __device__ double a0(int x, int k) const { return half2(kDbOffA0, x, k); }
  __device__ double rho(int j) const { return sm[kDbOffRho + j] + sm[kDbOffRho + kE + j]; }
};

__device__ inline DurTotals dur_totals(const double* totals, const uint32_t* gmax_bits, const unsigned char* packed,
                                      uint32_t* status) {
  DurTotals T;
  T.A = totals;
  T.B = totals + kDbAcc;
  T.sm = totals + 2 * kDbAcc;
  const double rs = (double)nab_dur_rscale(gmax_bits, reinterpret_cast<const float*>(packed + (size_t)kDbSlices * kDbStage), status);
  T.ua = 1.0 / (rs * (double)kDbSScale);
  T.ub = 1.0 / rs;
  return T;
}

// block (e, x), thread k:  PA = Wg1_x^T A_x, PB = Wg1_x^T B_x (row e);  dW2_x[e, k] = PA w1_k + PB b1_k + wo_e eta_k;
// prod[x][e][k] = (W2_x[e,k] PA, W2_x[e,k] PB) for dw1 / db1 (summed over e in nab_dur_fin3_kernel)
__global__ void __launch_bounds__(kE) nab_dur_fin1_kernel(const double* __restrict__ totals, const uint32_t* __restrict__ gmax_bits,
    const unsigned char* __restrict__ packed,
                                                          const float* __restrict__ params, double* __restrict__ prod,
                                                          float* __restrict__ grads, uint32_t* __restrict__ status) {
  const int e = blockIdx.x, x = blockIdx.y, k = threadIdx.x;
  const DurTotals T = dur_totals(totals, gmax_bits, packed, status);
  const float* P = params + x * kDbMlp;
  const float* wg1 = params + kDbWg1;
  double pa = 0.0, pb = 0.0;
  for (int j = 0; j < kE; ++j) {
    const double g = wg1[j * 3 * kE + x * kE + e];
    pa += g * T.a(x, j, k);
    pb += g * T.b(x, j, k);
  }
  const double w = P[k], bb = P[kE + k];
  const double eta = w * T.a1(x, k) + bb * T.a0(x, k);
  grads[x * kDbMlp + 2 * kE + e * kE + k] = (float)(pa * w + pb * bb + (double)params[kDbWo + e] * eta);
  const double w2 = P[2 * kE + e * kE + k];
  prod[((size_t)(x * kE + e) * kE + k) * 2] = w2 * pa;
  prod[((size_t)(x * kE + e) * kE + k) * 2 + 1] = w2 * pb;
}

// block (j, x), thread e:  dWg1[j, x E + e] = sum_k R_x[j, k] W2_x[e, k] + rho_j b2_x[e],  R_x = A_x diag(w1_x) + B_x diag(b1_x)
__global__ void __launch_bounds__(kE) nab_dur_fin2_kernel(const double* __restrict__ totals, const uint32_t* __restrict__ gmax_bits,
    const unsigned char* __restrict__ packed,
                                                          const float* __restrict__ params, float* __restrict__ grads,
                                                          uint32_t* __restrict__ status) {
  __shared__ double rrow[kE];
  const int j = blockIdx.x, x = blockIdx.y, e = threadIdx.x;
  const DurTotals T = dur_totals(totals, gmax_bits, packed, status);
  const float* P = params + x * kDbMlp;
  rrow[e] = T.a(x, j, e) * (double)P[e] + T.b(x, j, e) * (double)P[kE + e];
  __syncthreads();
  const float* W2 = P + 2 * kE;
  double a = 0.0;
  for (int k = 0; k < kE; ++k) a += rrow[k] * (double)W2[e * kE + k];
  grads[kDbWg1 + j * 3 * kE + x * kE + e] = (float)(a + T.rho(j) * (double)P[2 * kE + kE * kE + e]);
}

// one block, thread n: the remaining vectors and scalars
__global__ void __launch_bounds__(kE) nab_dur_fin3_kernel(const double* __restrict__ totals, const uint32_t* __restrict__ gmax_bits,
    const unsigned char* __restrict__ packed,
                                                          const float* __restrict__ params, const double* __restrict__ prod,
                                                          float* __restrict__ grads, uint32_t* __restrict__ status) {
  __shared__ double eta[3][kE];
  const int n = threadIdx.x;
  const DurTotals T = dur_totals(totals, gmax_bits, packed, status);
  const float* wo = params + kDbWo;
  const float* wg1 = params + kDbWg1;
  const double* sc = T.sm + kDbOffSc;
  const double tau = exp(-(double)params[kDbT]);
  for (int x = 0; x < 3; ++x) {
    const float* P = params + x * kDbMlp;
    const float* W2 = P + 2 * kE;
    double uo = 0.0, pa = 0.0, pb = 0.0;
    for (int e = 0; e < kE; ++e) {
      uo += (double)wo[e] * W2[e * kE + n];
      pa += prod[((size_t)(x * kE + e) * kE + n) * 2];
      pb += prod[((size_t)(x * kE + e) * kE + n) * 2 + 1];
    }
    grads[x * kDbMlp + n] = (float)(pa + uo * T.a1(x, n));       // emb.0.weight
    grads[x * kDbMlp + kE + n] = (float)(pb + uo * T.a0(x, n));  // emb.0.bias
    eta[x][n] = (double)P[n] * T.a1(x, n) + (double)P[kE + n] * T.a0(x, n);
    double g = 0.0;
    for (int j = 0; j < kE; ++j) g += (double)wg1[j * 3 * kE + x * kE + n] * T.rho(j);
    grads[x * kDbMlp + 2 * kE + kE * kE + n] = (float)(g + (double)wo[n] * sc[5 + x]);  // emb.2.bias
  }
  grads[kDbBg1 + n] = (float)T.rho(n);  // gate.0.bias
  for (int c = 0; c < 3; ++c) grads[kDbWg2 + c * kE + n] = (float)(tau * T.half2(kDbOffDzs, c, n));  // gate.2.weight
  __syncthreads();
  double dwo = 0.0;
  for (int x = 0; x < 3; ++x) {
    const float* P = params + x * kDbMlp;
    double a = 0.0;
    for (int k = 0; k < kE; ++k) a += (double)P[2 * kE + n * kE + k] * eta[x][k];
    dwo += a + (double)P[2 * kE + kE * kE + n] * sc[5 + x];
  }
  grads[kDbWo + n] = (float)dwo;  // out_lin.weight
  if (n < 3) grads[kDbBg2 + n] = (float)(tau * sc[n]);  // gate.2.bias
  if (n == 0) {
    grads[kDbT] = (float)(-sc[3]);  // gate_temperature
    grads[kDbBo] = (float)sc[4];    // out_lin.bias
  }
}

inline int64_t nab_dur_bwd_grid(int64_t n_inst, int n_nodes) {
  const int64_t n_tiles = (n_inst * (int64_t)n_nodes * n_nodes + kDbRows - 1) / kDbRows;
  const int64_t sms = device_sm_count();
  return n_tiles < sms ? n_tiles : sms;
}

// workspace: gmax bits (16 B) | partial accumulators (float, grid x kDbAcc) | small partials (double, grid x kDbSmall) |
//            totals (double, 2 kDbAcc + kDbSmall) | prod (double, 3 E E 2)
inline int64_t nab_dur_ws_bytes(int64_t grid) {
  return 16 + grid * kDbAcc * 4 + grid * kDbSmall * 8 + (2 * (int64_t)kDbAcc + kDbSmall) * 8 + 3LL * kE * kE * 2 * 8;
}

}  // namespace rrnco

using namespace rrnco;

extern "C" {

int64_t rrnco_train_nab_dur_packed_bytes(void) { return kDbPackedBytes; }

int64_t rrnco_train_nab_dur_grad_floats(void) { return kDbGrads; }

int64_t rrnco_train_nab_dur_workspace_bytes(int64_t n_inst, int32_t n_nodes) {
  if (n_inst <= 0 || n_nodes <= 0) return RRNCO_ERR_BAD_ARG;
  const int64_t grid = nab_dur_bwd_grid(n_inst, n_nodes);
  if (grid <= 0) return RRNCO_ERR_CUDA;
  return nab_dur_ws_bytes(grid);
}

int rrnco_train_nab_dur_backward(int64_t n_inst, int32_t n_nodes, const float* coords, const float* cost, const float* duration,
                                 int32_t transpose, const void* packed, const float* params, float scale, const float* grad_out,
                                 void* workspace, float* grads, uint32_t* status, void* stream) {
  RRNCO_CHECK_ARG(n_inst > 0 && n_nodes > 0 && coords && cost && duration && packed && params && grad_out && workspace && grads &&
                  status);
  RRNCO_CHECK_ARG((reinterpret_cast<uintptr_t>(coords) & 7u) == 0 && (reinterpret_cast<uintptr_t>(packed) & 15u) == 0 &&
                  (reinterpret_cast<uintptr_t>(workspace) & 15u) == 0);
  const int64_t grid = nab_dur_bwd_grid(n_inst, n_nodes);
  if (grid <= 0) return RRNCO_ERR_CUDA;
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(nab_dur_bwd_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DurBwdSmem)) != cudaSuccess ||
        cudaFuncSetAttribute(nab_dur_bwd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DurBwdSmem)) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  uint32_t* gmax = reinterpret_cast<uint32_t*>(ws);
  float* part_acc = reinterpret_cast<float*>(ws + 16);
  double* part_small = reinterpret_cast<double*>(ws + 16 + grid * kDbAcc * 4);
  double* totals = part_small + grid * kDbSmall;
  double* prod = totals + 2 * kDbAcc + kDbSmall;
  const int64_t n_pairs = n_inst * (int64_t)n_nodes * n_nodes;
  const cudaStream_t s = (cudaStream_t)stream;
  const unsigned char* pk = reinterpret_cast<const unsigned char*>(packed);
  if (cudaMemsetAsync(gmax, 0, 4, s) != cudaSuccess) return RRNCO_ERR_CUDA;
  nab_dur_bound_kernel<<<(unsigned)(4 * device_sm_count()), 256, 0, s>>>(n_nodes, n_pairs, coords, cost, duration, transpose, pk,
                                                                          scale, grad_out, gmax);
  nab_dur_bwd_kernel<0><<<(unsigned)grid, kDbThreads, sizeof(DurBwdSmem), s>>>(
      n_nodes, n_pairs, coords, cost, duration, transpose, pk, scale, grad_out, gmax, part_acc, part_small, status);
  nab_dur_reduce_kernel<float><<<(kDbAcc + 31) / 32, 256, 0, s>>>((int)grid, kDbAcc, part_acc, totals);
  nab_dur_bwd_kernel<1><<<(unsigned)grid, kDbThreads, sizeof(DurBwdSmem), s>>>(
      n_nodes, n_pairs, coords, cost, duration, transpose, pk, scale, grad_out, gmax, part_acc, part_small, status);
  nab_dur_reduce_kernel<float><<<(kDbAcc + 31) / 32, 256, 0, s>>>((int)grid, kDbAcc, part_acc, totals + kDbAcc);
  nab_dur_reduce_kernel<double><<<(kDbSmall + 31) / 32, 256, 0, s>>>((int)grid, kDbSmall, part_small, totals + 2 * kDbAcc);
  nab_dur_fin1_kernel<<<dim3(kE, 3), kE, 0, s>>>(totals, gmax, pk, params, prod, grads, status);
  nab_dur_fin2_kernel<<<dim3(kE, 3), kE, 0, s>>>(totals, gmax, pk, params, grads, status);
  nab_dur_fin3_kernel<<<1, kE, 0, s>>>(totals, gmax, pk, params, prod, grads, status);
  return rrnco_launch_status();
}

}  // extern "C"
