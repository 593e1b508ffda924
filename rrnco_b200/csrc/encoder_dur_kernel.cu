// Encoder hot spot, duration-channel variant (rcvrptw): DistAngleFusion.forward with the three-way gate,
// rrnco/models/nn/attn_freenet.py:242-289 (use_duration_matrix = True, encoder.py:63-66):
//     d = MLP_d(cost), a = MLP_a(angle), u = MLP_u(duration)                       three Linear(1,E)-ReLU-Linear(E,E)
//     g = softmax( Linear(E,3)( SiLU( Linear(3E,E)([d, a, u]) ) ) / exp(temperature) )
//     adapt_bias = out_lin( g_0 d + g_1 a + g_2 u )
// Upstream materialises three [B,N,N,E] embeddings and a [B,N,N,3E] concatenation per block.  As in the two-way variant
// (encoder_kernels.cu) everything that is linear in the hidden vectors h_x = relu(w_x s_x + b_x) is collapsed at pack time
// (fp64): the gate's first layer becomes  hidden_pre = M_d h_d + M_a h_a + M_u h_u + c0  with M_x = Wg1[:, x] W2_x, and
// out_lin(x-embedding) = uo_x . h_x + co_x.  What remains per pair IS GEMM-shaped -- [pairs x 3E] . [3E x E] -- and runs on
// tcgen05 with the rollout kernels' machinery: tiles of 128 pairs; per source the compute warps generate the A operand
// (h_x as fp16 hi | lo core-matrix tiles, 64 KB) straight from the pair's scalar, one elected thread issues 8 K-steps x 3
// split terms against the weight slices streamed through a TMA ring (same 8 KB slice layout as the FFN weights), the
// accumulator (128 TMEM columns) collects the three sources; the epilogue applies SiLU, the E -> 3 layer, the tempered
// softmax and the blend, thread per pair.  Two CTAs per SM (109 KB of shared memory, 128 TMEM columns each) overlap one
// tile's generation / epilogue with the other's MMAs.  Nothing of size [B,N,N,E] exists.
#include "common.cuh"
#include "tc05.cuh"
#include "ffn_pack.cuh"

namespace rrnco {

constexpr int kDThreads = 320;   // warps 0-7 compute, 8 TMA producer, 9 MMA issue
constexpr int kDRows = 128;      // pairs per tile
constexpr uint32_t kDStage = 8192;
constexpr int kDStages = 4;
constexpr int kDSlices = 24;     // 3 sources x 8 K-steps
// fp32 vectors behind the packed slices: w1[3][E] b1[3][E] uo[3][E] c0[E] wg2[3][E] | consts: bg2[3] co[3] bo inv_temp
constexpr int kDVec = 3 * kE * 3 + kE + 3 * kE;
constexpr int kDConsts = 8;
constexpr int64_t kDPackedBytes = (int64_t)kDSlices * kDStage + (kDVec + kDConsts) * 4;

struct DurSmem {
  unsigned char A[kDRows * kE * 4];
  unsigned char ring[kDStages][kDStage];
  float vec[kDVec + kDConsts];
  float od[3][kDRows];            // uo_x . h_x per pair
  float xl[3][2][kDRows];         // epilogue exchange: partial gate logits of the two column halves
  uint64_t bar_full[kDStages], bar_empty[kDStages];
  uint64_t bar_a;                 // compute -> issuer: A tile of a source written (256 arrivals)
  uint64_t bar_mma;               // issuer -> compute: MMAs of a source complete (A free; after the third: accumulator ready)
  uint32_t tmem_base;
};

// one block; thread n collapses row n of the gate's first layer / column n of the second layers (fp64)
__global__ void __launch_bounds__(kE) nab_dur_pack_kernel(const float* const* __restrict__ prm, unsigned char* __restrict__ packed,
                                                          uint32_t* __restrict__ status) {
  // prm: [0..3] dist w1 b1 W2 b2, [4..7] angle, [8..11] dur, [12] gate.0.weight [E,3E], [13] gate.0.bias [E],
  //      [14] gate.2.weight [3,E], [15] gate.2.bias [3], [16] gate_temperature [1], [17] out_lin.weight [1,E], [18] out_lin.bias [1]
  const int n = threadIdx.x;
  float* vec = reinterpret_cast<float*>(packed + (size_t)kDSlices * kDStage);
  const float* wg1 = prm[12];
  const float* wo = prm[17];
  double c0 = prm[13][n];
  for (int x = 0; x < 3; ++x) {
    const float* w1 = prm[4 * x];
    const float* b1 = prm[4 * x + 1];
    const float* W2 = prm[4 * x + 2];
    const float* b2 = prm[4 * x + 3];
    vec[x * kE + n] = w1[n];
    vec[3 * kE + x * kE + n] = b1[n];
    double uo = 0.0;
    for (int e = 0; e < kE; ++e) {
      uo += (double)wo[e] * W2[e * kE + n];             // column n of W2_x
      c0 += (double)wg1[n * 3 * kE + x * kE + e] * b2[e];
    }
    vec[6 * kE + x * kE + n] = (float)uo;
    // row n of M_x = Wg1[:, x] W2_x, written into the 8 K-step slices of source x:
    // [hi | lo][16-byte K chunk (2)][row n (128)][8 halves]
    for (int k = 0; k < kE; k += 2) {
      double m0 = 0.0, m1 = 0.0;
      for (int e = 0; e < kE; ++e) {
        const double g = wg1[n * 3 * kE + x * kE + e];
        m0 += g * W2[e * kE + k];
        m1 += g * W2[e * kE + k + 1];
      }
      if (!(fabs(m0) * kWScale < 65504.0) || !(fabs(m1) * kWScale < 65504.0)) atomicOr(status, RRNCO_DEV_NAN_LOGITS);
      uint32_t hi, lo;
      f16s_split2((float)m0, (float)m1, kWScale, hi, lo);
      const int ks = k >> 4, kp = (k & 15) >> 1;  // K step, pair index within the 16 k values of the step
      uint32_t* dst = reinterpret_cast<uint32_t*>(packed + (size_t)(x * 8 + ks) * kDStage) + (kp >> 2) * (kDRows * 4) + n * 4 + (kp & 3);
      dst[0] = hi;
      dst[kDStage / 8] = lo;
    }
    if (n == 0) {
      double co = 0.0;
      for (int e = 0; e < kE; ++e) co += (double)wo[e] * b2[e];
      vec[kDVec + 3 + x] = (float)co;
    }
  }
  vec[9 * kE + n] = (float)c0;
  for (int c = 0; c < 3; ++c) vec[10 * kE + c * kE + n] = prm[14][c * kE + n];
  if (n == 0) {
    for (int c = 0; c < 3; ++c) vec[kDVec + c] = prm[15][c];
    vec[kDVec + 6] = prm[18][0];
    vec[kDVec + 7] = expf(-prm[16][0]);  // logits / exp(temperature)
  }
}

__global__ void __launch_bounds__(kDThreads, 2) nab_dur_kernel(int N, int64_t n_pairs, const float* __restrict__ coords,
                                                               const float* __restrict__ cost, const float* __restrict__ dur,
                                                               int transpose, const unsigned char* __restrict__ packed,
                                                               float scale, float* __restrict__ out, uint32_t* __restrict__ status) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  DurSmem& sm = *reinterpret_cast<DurSmem*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t n_tiles = (n_pairs + kDRows - 1) / kDRows;
  if (warp == 0) tc05::tmem_alloc(&sm.tmem_base, 128);
  if (tid == 32) {
    for (int i = 0; i < kDStages; ++i) {
      tc05::mbar_init(&sm.bar_full[i], 1);
      tc05::mbar_init(&sm.bar_empty[i], 1);
    }
    tc05::mbar_init(&sm.bar_a, 256);
    tc05::mbar_init(&sm.bar_mma, 1);
    tc05::fence_mbar_init();
  }
  {
    const float* vsrc = reinterpret_cast<const float*>(packed + (size_t)kDSlices * kDStage);
    for (int i = tid; i < kDVec + kDConsts; i += kDThreads) sm.vec[i] = vsrc[i];
  }
  tc05::fence_before_sync();
  __syncthreads();
  tc05::fence_after_sync();

  const int uwarp = __shfl_sync(0xffffffffu, warp, 0);
  if (uwarp == 8) {
    // ===== TMA producer: the 24 weight slices of a tile, source-major =====
    if (tc05::elect_one()) {
      uint32_t st = 0, round = 0;
      for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
#pragma unroll 1
        for (int s = 0; s < kDSlices; ++s) {
          if (round > 0) tc05::mbar_wait(&sm.bar_empty[st], (round - 1) & 1, 32);
          tc05::mbar_arrive_expect_tx(&sm.bar_full[st], kDStage);
          tc05::bulk_g2s(sm.ring[st], packed + (size_t)s * kDStage, kDStage, &sm.bar_full[st]);
          if (++st == (uint32_t)kDStages) { st = 0; ++round; }
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
      const uint32_t a_addr = tc05::smem_u32(sm.A), a_lo_off = kDRows * kE * 2;
      const uint32_t ring_addr = tc05::smem_u32(sm.ring[0]);
      uint32_t st = 0, round = 0, n_a = 0;
      for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
#pragma unroll 1
        for (int x = 0; x < 3; ++x) {
          tc05::mbar_wait(&sm.bar_a, n_a & 1u, 32);
          ++n_a;
          tc05::fence_after_sync();
#pragma unroll 1
          for (int ks = 0; ks < 8; ++ks) {
            tc05::mbar_wait(&sm.bar_full[st], round & 1);
            tc05::fence_after_sync();
            const uint32_t b_addr = ring_addr + st * kDStage;
            const uint64_t b_hi = tc05::make_desc(b_addr, kLboTile, kSbo);
            const uint64_t b_lo = tc05::make_desc(b_addr + kDStage / 2, kLboTile, kSbo);
            const uint64_t a_hi = tc05::make_desc(a_addr + ks * 2 * kLboTile, kLboTile, kSbo);
            tc05::mma_ss_f16(tb, a_hi, b_hi, idesc, (x > 0 || ks > 0) ? 1u : 0u);
            tc05::mma_ss_f16(tb, tc05::make_desc(a_addr + a_lo_off + ks * 2 * kLboTile, kLboTile, kSbo), b_hi, idesc, 1u);
            tc05::mma_ss_f16(tb, a_hi, b_lo, idesc, 1u);
            tc05::commit(&sm.bar_empty[st]);
            if (++st == (uint32_t)kDStages) { st = 0; ++round; }
          }
          tc05::commit(&sm.bar_mma);
        }
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
  uint16_t* a_lo = a_hi + kDRows * kE;
  const float* w1 = sm.vec;
  const float* b1 = sm.vec + 3 * kE;
  const float* uo = sm.vec + 6 * kE;
  const float* c0 = sm.vec + 9 * kE;
  const float* wg2 = sm.vec + 10 * kE;
  const float* cs = sm.vec + kDVec;  // bg2[3] co[3] bo inv_temp
  constexpr float kUnscale = 1.0f / (kAScale * kWScale);
  uint32_t n_m = 0;  // completed waits on bar_mma
  const int64_t NN = (int64_t)N * N;

  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    // the pair of this thread's generation row and its three scalars (both column halves compute them)
    const int grow = warp * 16 + (lane & 15), dh = lane >> 4;
    {
      const int64_t p = t * kDRows + grow;
      float c = 0.f, th = 0.f, u = 0.f;
      if (p < n_pairs) {
        const int64_t b = p / NN;
        const int r = (int)(p - b * NN), i = r / N, j = r - i * N;
        const int64_t src = transpose ? b * NN + (int64_t)j * N + i : p;
        c = __ldg(cost + src);
        u = __ldg(dur + src);
        const float2 pi = __ldg(reinterpret_cast<const float2*>(coords) + b * N + i);
        const float2 pj = __ldg(reinterpret_cast<const float2*>(coords) + b * N + j);
        th = atan2f(pi.y - pj.y, pi.x - pj.x);
      }
      // (each lane keeps the pair's three scalars in registers for the generation below)
#pragma unroll 1
      for (int x = 0; x < 3; ++x) {
        const float s = x == 0 ? c : (x == 1 ? th : u);
        if (x > 0) {  // the MMAs that read the previous A tile have completed (x == 0: the epilogue below waited for them)
          if ((warp & 3) == 0) tc05::mbar_wait(&sm.bar_mma, n_m & 1u);
          asm volatile("bar.sync 1, 256;\n" ::: "memory");
          ++n_m;
        }
        float od = 0.f, hmax = 0.f;
#pragma unroll 2
        for (int cc = 0; cc < 8; ++cc) {
          const int c8 = dh * 8 + cc, k0 = c8 * 8;
          float h[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            h[e] = fmax_nan(fmaf(w1[x * kE + k0 + e], s, b1[x * kE + k0 + e]), 0.f);  // a NaN scalar: NaN (upstream's relu)
            od = fmaf(uo[x * kE + k0 + e], h[e], od);
            hmax = fmax_nan(hmax, h[e]);
          }
          uint32_t hh[4], ll[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) f16s_split2(h[2 * e], h[2 * e + 1], kAScale, hh[e], ll[e]);
          const int dst = c8 * (kDRows * 8) + grow * 8;
          *reinterpret_cast<uint4*>(&a_hi[dst]) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
          *reinterpret_cast<uint4*>(&a_lo[dst]) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
        }
        if (!(hmax * kAScale < 65504.f)) atomicOr(status, RRNCO_DEV_NAN_LOGITS);  // fp16 operand overflow or non-finite input: loud
        od += __shfl_xor_sync(0xffffffffu, od, 16);
        if (dh == 0) sm.od[x][grow] = od;
        tc05::fence_proxy_async();
        tc05::fence_before_sync();
        tc05::mbar_arrive(&sm.bar_a);
      }
    }
    // ---- epilogue: accumulator complete ----
    if ((warp & 3) == 0) tc05::mbar_wait(&sm.bar_mma, n_m & 1u);
    asm volatile("bar.sync 1, 256;\n" ::: "memory");
    ++n_m;
    tc05::fence_after_sync();
    {
      const int row = trow;
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
          const float si = hp / (1.0f + expf(-hp));  // SiLU
          l0 = fmaf(wg2[col0 + i], si, l0);
          l1 = fmaf(wg2[kE + col0 + i], si, l1);
          l2 = fmaf(wg2[2 * kE + col0 + i], si, l2);
        }
      }
      sm.xl[0][grp][row] = l0;
      sm.xl[1][grp][row] = l1;
      sm.xl[2][grp][row] = l2;
      tc05::fence_before_sync();
      asm volatile("bar.sync 1, 256;\n" ::: "memory");
      if (grp == 0) {
        const int64_t p = t * kDRows + row;
        if (p < n_pairs) {
          const float z0 = (sm.xl[0][0][row] + sm.xl[0][1][row] + cs[0]) * cs[7];
          const float z1 = (sm.xl[1][0][row] + sm.xl[1][1][row] + cs[1]) * cs[7];
          const float z2 = (sm.xl[2][0][row] + sm.xl[2][1][row] + cs[2]) * cs[7];
          const float zm = fmaxf(z0, fmaxf(z1, z2));
          const float e0 = expf(z0 - zm), e1 = expf(z1 - zm), e2 = expf(z2 - zm);
          const float inv = 1.0f / (e0 + e1 + e2);
          const float y = (e0 * (sm.od[0][row] + cs[3]) + e1 * (sm.od[1][row] + cs[4]) + e2 * (sm.od[2][row] + cs[5])) * inv + cs[6];
          out[p] = y * scale;
        }
      }
      asm volatile("bar.sync 1, 256;\n" ::: "memory");  // od / xl are rewritten by the next tile's generation
    }
  }
  tc05::fence_before_sync();
  asm volatile("bar.sync 1, 256;\n" ::: "memory");
  if (warp == 0) tc05::tmem_dealloc(sm.tmem_base, 128);
}

}  // namespace rrnco

using namespace rrnco;

extern "C" {

int64_t rrnco_nab_dur_packed_bytes(void) { return kDPackedBytes; }

int rrnco_nab_dur_pack(const float* const* d_params, void* packed, uint32_t* status, void* stream) {
  RRNCO_CHECK_ARG(d_params && packed && status && (reinterpret_cast<uintptr_t>(packed) & 15u) == 0);
  nab_dur_pack_kernel<<<1, kE, 0, (cudaStream_t)stream>>>(d_params, reinterpret_cast<unsigned char*>(packed), status);
  return rrnco_launch_status();
}

int rrnco_nab_dur_gating(int64_t n_inst, int32_t n_nodes, const float* coords, const float* cost, const float* duration,
                         int32_t transpose, const void* packed, float scale, float* out, uint32_t* status, void* stream) {
  RRNCO_CHECK_ARG(n_inst > 0 && n_nodes > 0 && coords && cost && duration && packed && out && status);
  RRNCO_CHECK_ARG((reinterpret_cast<uintptr_t>(coords) & 7u) == 0 && (reinterpret_cast<uintptr_t>(packed) & 15u) == 0);
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(nab_dur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DurSmem)) != cudaSuccess ||
        cudaFuncSetAttribute(nab_dur_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  static_assert(sizeof(DurSmem) <= 115712, "two CTAs per SM");
  const int64_t n_pairs = n_inst * (int64_t)n_nodes * n_nodes;
  const int64_t n_tiles = (n_pairs + kDRows - 1) / kDRows;
  const int sms = device_sm_count();
  const int64_t grid = n_tiles < 2LL * sms ? n_tiles : 2LL * sms;
  nab_dur_kernel<<<(unsigned)grid, kDThreads, sizeof(DurSmem), (cudaStream_t)stream>>>(
      n_nodes, n_pairs, coords, cost, duration, transpose, reinterpret_cast<const unsigned char*>(packed), scale, out, status);
  return rrnco_launch_status();
}

}  // extern "C"
