// Training hand-off, pointer scores of RRNet_PointerAttention (rrnco/models/decoder.py:298-301: g . logit_key^T) for the rows of
// the batched replay, forward and backward, on tcgen05 in the fp32-faithful fp16 hi|lo split (the fp32 SIMT batched GEMMs of
// torch.bmm were 12 ms of the 128 ms training step):
//   inst_gemm_kernel   Y[rows, 128] = X[rows, 128] W_b            one 128 x 128 weight tile per INSTANCE b (zero-padded)
//                      forward:  z  = g  Lk_b^T  (columns >= n_nodes are zero)        backward:  dg = dz Lk_b
//   xty_inst_kernel    C_b[n_nodes, 128] = X_b^T Y_b over the rows of instance b    (dLk_b = dz_b^T g_b)
// Scores / their gradients are kept 128 wide (row stride 128 floats): thread-per-row epilogues then store whole sectors.
// Instances of more than 128 nodes (the rrnco_train_inst_tiled_* entry points) use ceil(N / 128) weight tiles per instance, and
// scores rows ldz = 128 ceil(N / 128) wide: the forward writes one 128-column block per tile (grid z), dg accumulates the key tiles
// in TMEM (the weight tile is reloaded per key tile), and dLk_b is computed per (instance, key tile) (grid z).
#include "../csrc/common.cuh"
#include "../csrc/tc05.cuh"
#include "../csrc/ffn_pack.cuh"
#include "../../include/rrnco_b200_train.h"

namespace rrnco {

constexpr int kPtThreads = 288;
constexpr uint32_t kPtTileBytes = kFRows * kE * 2;  // one fp16 variant of a 128 x 128 tile: 32 KB
constexpr float kPtMax = 65504.f;
constexpr int kPtMaxNodes = 1024;   // the rrnco_train_inst_tiled_* entry points: up to 8 key tiles

// [n_inst, N, 128] -> per (instance, key tile) [hi | lo][16-byte K chunk (16)][row n (128)][8 halves], key tile = grid z;
// transpose == 0: B[n = node][k = e] (z = g Lk^T), transpose == 1: B[n = e][k = node] (dg = dz Lk); nodes beyond N are zero
__global__ void pack_inst_weights_kernel(const float* __restrict__ src, int N, int transpose, uint32_t* __restrict__ packed,
                                         uint32_t* __restrict__ status) {
  const int64_t b = blockIdx.y;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // (row n, k pair)
  if (i >= kFRows * (kE / 2)) return;
  const int n = i >> 6, kp = i & 63, k = kp * 2, j0 = blockIdx.z * kFRows;
  const float* s = src + (b * N + j0) * kE;
  const int nj = N - j0;   // nodes of this key tile (> 128: the tile is full)
  float v0 = 0.f, v1 = 0.f;
  if (!transpose) {
    if (n < nj) { v0 = s[n * kE + k]; v1 = s[n * kE + k + 1]; }
  } else {
    if (k < nj) v0 = s[k * kE + n];
    if (k + 1 < nj) v1 = s[(k + 1) * kE + n];
  }
  if (!(fabsf(v0) * kLkScale < kPtMax) || !(fabsf(v1) * kLkScale < kPtMax)) atomicOr(status, RRNCO_DEV_NAN_LOGITS);
  uint32_t hi, lo;
  f16s_split2(v0, v1, kLkScale, hi, lo);
  uint32_t* dst = packed + (b * gridDim.z + blockIdx.z) * (2 * kPtTileBytes / 4) + (kp >> 2) * (kFRows * 4) + n * 4 + (kp & 3);
  dst[0] = hi;
  dst[kPtTileBytes / 4] = lo;
}

struct InstGemmSmem {
  uint16_t a_hi[kFRows * kE];
  uint16_t a_lo[kFRows * kE];
  uint16_t b_hi[kFRows * kE];
  uint16_t b_lo[kFRows * kE];
  float stage[kFRows * 132];   // output tile, row stride 132 floats: thread-per-row float4 writes and row-contiguous reads are conflict-free
  uint64_t bar_b, bar_a, bar_mma;
  uint32_t tmem_base;
};

// Y[rows, grid z tiles of 128 columns] (row stride ldy) = sum over nk key tiles of X[rows, key tile] (row stride ldx) B_(b, z, kt):
// nk == 1, one column block: the 128-node form; weight tile (b, z, kt) at packed index (b gridDim.z + z) nk + kt
__global__ void __launch_bounds__(kPtThreads, 1) inst_gemm_kernel(int64_t L, int rows_per_cta, int ldx, int nk, int ldy,
                                                                 const float* __restrict__ X,
                                                                 const unsigned char* __restrict__ packed,
                                                                 const float* __restrict__ a_scale_ptr,
                                                                 const float* __restrict__ row_scale, float* __restrict__ Y,
                                                                 uint32_t* __restrict__ status) {
  extern __shared__ __align__(128) unsigned char pt_smem_raw[];
  InstGemmSmem& sm = *reinterpret_cast<InstGemmSmem*>(pt_smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t b = blockIdx.y;
  const int64_t row_lo = b * L + (int64_t)blockIdx.x * rows_per_cta;
  const int64_t row_hi = min(row_lo + rows_per_cta, (b + 1) * L);
  const int n_tiles = (int)((row_hi - row_lo + kFRows - 1) / kFRows);
  if (warp == 0) tc05::tmem_alloc(&sm.tmem_base, 128);
  if (tid == 32) {
    tc05::mbar_init(&sm.bar_b, 1);
    tc05::mbar_init(&sm.bar_a, 256);
    tc05::mbar_init(&sm.bar_mma, 1);
    tc05::fence_mbar_init();
  }
  tc05::fence_before_sync();
  __syncthreads();
  tc05::fence_after_sync();
  const uint32_t tb = sm.tmem_base;

  const int uwarp = __shfl_sync(0xffffffffu, warp, 0);
  if (uwarp == 8) {
    if (tc05::elect_one()) {
      const unsigned char* pb = packed + (b * gridDim.z + blockIdx.z) * (size_t)nk * (2 * (size_t)kPtTileBytes);
      auto load_b = [&](int kt, uint32_t parity) {
        tc05::mbar_arrive_expect_tx(&sm.bar_b, 2 * kPtTileBytes);
        tc05::bulk_g2s(sm.b_hi, pb + kt * (2 * (size_t)kPtTileBytes), kPtTileBytes, &sm.bar_b);
        tc05::bulk_g2s(sm.b_lo, pb + kt * (2 * (size_t)kPtTileBytes) + kPtTileBytes, kPtTileBytes, &sm.bar_b);
        tc05::mbar_wait(&sm.bar_b, parity);
      };
      if (nk == 1) load_b(0, 0u);   // the instance's weight tile, once per CTA
      const uint32_t idesc = tc05::make_idesc_f16(128, 128);
      const uint32_t a_hi = tc05::smem_u32(sm.a_hi), a_lo = tc05::smem_u32(sm.a_lo);
      const uint32_t b_hi = tc05::smem_u32(sm.b_hi), b_lo = tc05::smem_u32(sm.b_lo);
      for (int i = 0; i < n_tiles; ++i) {
        for (int kt = 0; kt < nk; ++kt) {
          const int c = i * nk + kt;   // MMA step: bar_a / bar_mma phase c
          if (nk > 1) {                // key tile kt replaces the previous one once the MMAs that read it have completed
            if (c > 0) tc05::mbar_wait(&sm.bar_mma, (c - 1) & 1);
            load_b(kt, c & 1);
          }
          tc05::mbar_wait(&sm.bar_a, c & 1);
          tc05::fence_after_sync();
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            const uint32_t o = ks * 2 * kLboTile;
            const uint64_t dah = tc05::make_desc(a_hi + o, kLboTile, kSbo), dal = tc05::make_desc(a_lo + o, kLboTile, kSbo);
            const uint64_t dbh = tc05::make_desc(b_hi + o, kLboTile, kSbo), dbl = tc05::make_desc(b_lo + o, kLboTile, kSbo);
            tc05::mma_ss_f16(tb, dah, dbh, idesc, (kt > 0 || ks > 0) ? 1u : 0u);
            tc05::mma_ss_f16(tb, dal, dbh, idesc, 1u);
            tc05::mma_ss_f16(tb, dah, dbl, idesc, 1u);
          }
          tc05::commit(&sm.bar_mma);
        }
      }
    }
    return;
  }

  const int row = (warp & 3) * 32 + lane;
  const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
  const int colhalf = warp >> 2;
  const float a_scale = a_scale_ptr ? __ldg(a_scale_ptr) : kAScale;
  const float unscale = 1.0f / (a_scale * kLkScale);
  float amax = 0.f;
  float4 buf[16];   // this thread's 8 (row, 8-column chunk) items of a tile, raw: the next tile is in flight while the current one is consumed
  auto load_tile = [&](int64_t m0, int kt) {
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int idx = tid + it * 256, r = idx & 127, c8 = idx >> 7;
      float4 v0 = make_float4(0.f, 0.f, 0.f, 0.f), v1 = v0;
      if (m0 + r < row_hi) {
        const float4* src = reinterpret_cast<const float4*>(X + (m0 + r) * ldx + kt * kFRows) + c8 * 2;
        v0 = __ldg(src);
        v1 = __ldg(src + 1);
        if (row_scale != nullptr) {  // x = diag(row_scale) X: the upstream gradient of a row times its saved Jacobian
          const float rs = __ldg(row_scale + m0 + r);
          v0.x *= rs; v0.y *= rs; v0.z *= rs; v0.w *= rs;
          v1.x *= rs; v1.y *= rs; v1.z *= rs; v1.w *= rs;
        }
      }
      buf[2 * it] = v0;
      buf[2 * it + 1] = v1;
    }
  };
  if (n_tiles > 0) load_tile(row_lo, 0);
  for (int c = 0; c < n_tiles * nk; ++c) {
    const int i = c / nk, kt = c - i * nk;
    const int64_t m0 = row_lo + (int64_t)i * kFRows;
    // x tile -> fp16 hi | lo core-matrix tiles (the previous tile's MMAs have completed: its epilogue waited for them)
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int idx = tid + it * 256, r = idx & 127, c8 = idx >> 7;
      const float4 v0 = buf[2 * it], v1 = buf[2 * it + 1];
      amax = fmaxf(amax, fmaxf(fmaxf(fabsf(v0.x), fabsf(v0.y)), fmaxf(fabsf(v0.z), fabsf(v0.w))) * a_scale);
      amax = fmaxf(amax, fmaxf(fmaxf(fabsf(v1.x), fabsf(v1.y)), fmaxf(fabsf(v1.z), fabsf(v1.w))) * a_scale);
      uint32_t h[4], l[4];
      f16s_split2(v0.x, v0.y, a_scale, h[0], l[0]);
      f16s_split2(v0.z, v0.w, a_scale, h[1], l[1]);
      f16s_split2(v1.x, v1.y, a_scale, h[2], l[2]);
      f16s_split2(v1.z, v1.w, a_scale, h[3], l[3]);
      const int dst = c8 * (kFRows * 8) + r * 8;
      *reinterpret_cast<uint4*>(&sm.a_hi[dst]) = make_uint4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<uint4*>(&sm.a_lo[dst]) = make_uint4(l[0], l[1], l[2], l[3]);
    }
    if (kt + 1 < nk) load_tile(m0, kt + 1);
    else if (i + 1 < n_tiles) load_tile(m0 + kFRows, 0);
    tc05::fence_proxy_async();
    tc05::mbar_arrive(&sm.bar_a);
    tc05::mbar_wait(&sm.bar_mma, c & 1);
    tc05::fence_after_sync();
    if (kt + 1 < nk) continue;   // the accumulator sums the remaining key tiles first
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int col0 = colhalf * 64 + q * 16;
      uint32_t v[16];
      tc05::tmem_ld16(tb + lane_base + col0, v);
      tc05::tmem_wait_ld();
      // through shared memory: a thread-per-row store to global memory is 32 half-filled sectors per instruction, a staged warp
      // writes one whole 512-byte row per instruction
      float4* dst = reinterpret_cast<float4*>(&sm.stage[row * 132 + col0]);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        dst[j] = make_float4(__uint_as_float(v[4 * j]) * unscale, __uint_as_float(v[4 * j + 1]) * unscale,
                             __uint_as_float(v[4 * j + 2]) * unscale, __uint_as_float(v[4 * j + 3]) * unscale);
    }
    tc05::fence_before_sync();
    asm volatile("bar.sync 1, 256;\n" ::: "memory");  // tile staged (and every accumulator read has completed)
#pragma unroll 4
    for (int k = tid; k < kFRows * (kE / 4); k += 256) {
      const int r = k >> 5, c4 = k & 31;
      if (m0 + r < row_hi)
        reinterpret_cast<float4*>(Y + (m0 + r) * ldy + blockIdx.z * kFRows)[c4] = *reinterpret_cast<const float4*>(&sm.stage[r * 132 + c4 * 4]);
    }
    // (the next tile's epilogue writes `stage` only after bar_mma, i.e. after every thread has arrived on bar_a behind this loop)
  }
  if (!(amax < kPtMax)) atomicOr(status, RRNCO_DEV_NAN_LOGITS);
  tc05::fence_before_sync();
  asm volatile("bar.sync 1, 256;\n" ::: "memory");
  if (warp == 0) tc05::tmem_dealloc(tb, 128);
}

// C_b[n_nodes, 128] += X_b^T Y_b over a slab of the rows of instance b (X: [rows, ldx], Y: [rows, 128]); as xty_kernel of ffn_train.cu
// with one 128-feature block: 32-row tiles, two-stage operand buffer, 8 conversion warps (thread = one column of X or of Y) + issuer.
// Grid z = key tile: columns [128 z, 128 z + 128) of X give rows [128 z, ..) of C_b.
constexpr int kXiRows = 32;
struct XtyInstSmem {
  uint16_t x_hi[2][kE * kXiRows];   // [8-row K chunk (4)][feature (128)][8 halves]
  uint16_t x_lo[2][kE * kXiRows];
  uint16_t y_hi[2][kE * kXiRows];
  uint16_t y_lo[2][kE * kXiRows];
  uint64_t bar_full[2], bar_free[2], bar_done;
  uint32_t tmem_base;
};

__global__ void __launch_bounds__(kPtThreads, 2) xty_inst_kernel(int64_t L, int rows_per_cta, int N, int ldx, const float* __restrict__ X,
                                                                const float* __restrict__ Y, const float* __restrict__ sx_ptr,
                                                                const float* __restrict__ sy_ptr,
                                                                const float* __restrict__ row_scale, float* __restrict__ C,
                                                                uint32_t* __restrict__ status) {
  extern __shared__ __align__(128) unsigned char pt_smem_raw[];
  XtyInstSmem& sm = *reinterpret_cast<XtyInstSmem*>(pt_smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t b = blockIdx.y;
  const int64_t row_lo = b * L + (int64_t)blockIdx.x * rows_per_cta;
  const int64_t row_hi = min(row_lo + rows_per_cta, (b + 1) * L);
  const int n_tiles = (int)((row_hi - row_lo + kXiRows - 1) / kXiRows);
  if (warp == 0) tc05::tmem_alloc(&sm.tmem_base, 128);
  if (tid == 32) {
    for (int i = 0; i < 2; ++i) {
      tc05::mbar_init(&sm.bar_full[i], 256);
      tc05::mbar_init(&sm.bar_free[i], 1);
    }
    tc05::mbar_init(&sm.bar_done, 1);
    tc05::fence_mbar_init();
  }
  tc05::fence_before_sync();
  __syncthreads();
  tc05::fence_after_sync();
  const uint32_t tb = sm.tmem_base;

  const int uwarp = __shfl_sync(0xffffffffu, warp, 0);
  if (uwarp == 8) {
    if (tc05::elect_one()) {
      const uint32_t idesc = tc05::make_idesc_f16(128, 128);
      for (int it = 0; it < n_tiles; ++it) {
        const uint32_t st = it & 1;
        tc05::mbar_wait(&sm.bar_full[st], (it >> 1) & 1);
        tc05::fence_after_sync();
        const uint32_t xh = tc05::smem_u32(sm.x_hi[st]), xl = tc05::smem_u32(sm.x_lo[st]);
        const uint32_t yh = tc05::smem_u32(sm.y_hi[st]), yl = tc05::smem_u32(sm.y_lo[st]);
#pragma unroll
        for (int ks = 0; ks < kXiRows / 16; ++ks) {
          const uint32_t o = ks * 2 * kLboTile;
          const uint64_t a_hi = tc05::make_desc(xh + o, kLboTile, kSbo), a_lo = tc05::make_desc(xl + o, kLboTile, kSbo);
          const uint64_t b_hi = tc05::make_desc(yh + o, kLboTile, kSbo), b_lo = tc05::make_desc(yl + o, kLboTile, kSbo);
          tc05::mma_ss_f16(tb, a_hi, b_hi, idesc, (it > 0 || ks > 0) ? 1u : 0u);
          tc05::mma_ss_f16(tb, a_lo, b_hi, idesc, 1u);
          tc05::mma_ss_f16(tb, a_hi, b_lo, idesc, 1u);
        }
        tc05::commit(&sm.bar_free[st]);
      }
      tc05::commit(&sm.bar_done);
    }
    return;
  }

  const float sx = sx_ptr ? __ldg(sx_ptr) : kAScale, sy = sy_ptr ? __ldg(sy_ptr) : kAScale;
  const bool is_x = tid < 128;
  const int f = tid & 127;
  const int n0 = blockIdx.z * kFRows;
  const float* src = is_x ? X + n0 + f : Y + f;
  const int64_t lds = is_x ? ldx : kE;
  const float sc = is_x ? sx : sy;
  float amax = 0.f;
  for (int it = 0; it < n_tiles; ++it) {
    const uint32_t st = it & 1;
    const int64_t r0 = row_lo + (int64_t)it * kXiRows;
    float xv[kXiRows];
#pragma unroll
    for (int r = 0; r < kXiRows; ++r) xv[r] = (r0 + r < row_hi) ? __ldg(src + (r0 + r) * lds) : 0.f;
    if (is_x && row_scale != nullptr) {
#pragma unroll
      for (int r = 0; r < kXiRows; ++r) xv[r] *= (r0 + r < row_hi) ? __ldg(row_scale + r0 + r) : 0.f;
    }
    if (it >= 2) tc05::mbar_wait(&sm.bar_free[st], ((it >> 1) - 1) & 1);
    uint16_t* dh = is_x ? sm.x_hi[st] : sm.y_hi[st];
    uint16_t* dl = is_x ? sm.x_lo[st] : sm.y_lo[st];
#pragma unroll
    for (int kc = 0; kc < 4; ++kc) {
      uint32_t h[4], l[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float a = xv[kc * 8 + 2 * i], c = xv[kc * 8 + 2 * i + 1];
        amax = fmaxf(amax, fmaxf(fabsf(a), fabsf(c)) * sc);
        f16s_split2(a, c, sc, h[i], l[i]);
      }
      const int dst = kc * (kFRows * 8) + f * 8;
      *reinterpret_cast<uint4*>(&dh[dst]) = make_uint4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<uint4*>(&dl[dst]) = make_uint4(l[0], l[1], l[2], l[3]);
    }
    tc05::fence_proxy_async();
    tc05::mbar_arrive(&sm.bar_full[st]);
  }
  tc05::mbar_wait(&sm.bar_done, 0u);
  tc05::fence_after_sync();
  {
    const int m = (warp & 3) * 32 + lane, colhalf = warp >> 2;
    const uint32_t lane_b = (uint32_t)((warp & 3) * 32) << 16;
    const float unscale = 1.0f / (sx * sy);
#pragma unroll 1
    for (int q = 0; q < 4; ++q) {
      uint32_t v[16];
      tc05::tmem_ld16(tb + lane_b + colhalf * 64 + q * 16, v);
      tc05::tmem_wait_ld();
      if (n0 + m < N) {
        float* crow = C + (b * N + n0 + m) * kE + colhalf * 64 + q * 16;
#pragma unroll
        for (int i = 0; i < 16; ++i) atomicAdd(crow + i, __uint_as_float(v[i]) * unscale);
      }
    }
  }
  if (!(amax < kPtMax)) atomicOr(status, RRNCO_DEV_NAN_LOGITS);
  tc05::fence_before_sync();
  asm volatile("bar.sync 1, 256;\n" ::: "memory");
  if (warp == 0) tc05::tmem_dealloc(tb, 128);
}

static int pt_rows_per_cta(int64_t L, int64_t n_inst, int* ctas_per_inst) {
  int64_t per = 1;   // as few CTAs per instance as keep >= 4 waves on the device (the weight tile / the C tile is per CTA)
  const int sms = device_sm_count();
  while (per * n_inst < 4LL * sms && per * 256 < L) ++per;
  int64_t rows = (L + per - 1) / per;
  rows = (rows + kFRows - 1) / kFRows * kFRows;
  *ctas_per_inst = (int)((L + rows - 1) / rows);
  return (int)rows;
}

static int pt_pack(int64_t n_inst, int32_t n_nodes, const float* w, int32_t transpose, void* packed, uint32_t* status, void* stream) {
  pack_inst_weights_kernel<<<dim3(kFRows * (kE / 2) / 256, (unsigned)n_inst, (unsigned)((n_nodes + kFRows - 1) / kFRows)), 256, 0,
                             (cudaStream_t)stream>>>(w, n_nodes, transpose, reinterpret_cast<uint32_t*>(packed), status);
  return rrnco_launch_status();
}

// n_out column blocks of 128 (grid z), nk key tiles summed per block
static int pt_gemm(int64_t n_inst, int64_t rows_per_inst, int ldx, int nk, int ldy, int n_out, const float* x, const void* packed,
                   const float* a_scale, const float* row_scale, float* y, uint32_t* status, void* stream) {
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(inst_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(InstGemmSmem)) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  int per = 1;
  const int rows = pt_rows_per_cta(rows_per_inst, n_inst * n_out, &per);
  inst_gemm_kernel<<<dim3((unsigned)per, (unsigned)n_inst, (unsigned)n_out), kPtThreads, sizeof(InstGemmSmem), (cudaStream_t)stream>>>(
      rows_per_inst, rows, ldx, nk, ldy, x, reinterpret_cast<const unsigned char*>(packed), a_scale, row_scale, y, status);
  return rrnco_launch_status();
}

static int pt_xty(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, int ldx, const float* x, const float* y, const float* sx,
                  const float* sy, const float* row_scale, float* c, uint32_t* status, void* stream) {
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(xty_inst_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(XtyInstSmem)) != cudaSuccess ||
        cudaFuncSetAttribute(xty_inst_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  const int n_kt = (n_nodes + kFRows - 1) / kFRows;
  int per = 1;
  const int rows = pt_rows_per_cta(rows_per_inst, n_inst * n_kt, &per);
  xty_inst_kernel<<<dim3((unsigned)per, (unsigned)n_inst, (unsigned)n_kt), kPtThreads, sizeof(XtyInstSmem), (cudaStream_t)stream>>>(
      rows_per_inst, rows, n_nodes, ldx, x, y, sx, sy, row_scale, c, status);
  return rrnco_launch_status();
}

}  // namespace rrnco

using namespace rrnco;

extern "C" {

int64_t rrnco_train_inst_packed_bytes(int64_t n_inst) { return n_inst * 2 * (int64_t)kPtTileBytes; }

int rrnco_train_inst_pack(int64_t n_inst, int32_t n_nodes, const float* w, int32_t transpose, void* packed, uint32_t* status,
                          void* stream) {
  if (n_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && n_nodes > 0 && w && packed && status && (reinterpret_cast<uintptr_t>(packed) & 15u) == 0);
  if (n_nodes > 128 || n_inst > 65535) return RRNCO_ERR_UNSUPPORTED;
  return pt_pack(n_inst, n_nodes, w, transpose, packed, status, stream);
}

int rrnco_train_inst_gemm(int64_t n_inst, int64_t rows_per_inst, const float* x, const void* packed, const float* a_scale,
                          const float* row_scale, float* y, uint32_t* status, void* stream) {
  if (n_inst == 0 || rows_per_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && rows_per_inst > 0 && x && packed && y && status);
  RRNCO_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(packed) | reinterpret_cast<uintptr_t>(y)) & 15u) == 0);
  if (n_inst > 65535) return RRNCO_ERR_UNSUPPORTED;
  return pt_gemm(n_inst, rows_per_inst, kE, 1, kE, 1, x, packed, a_scale, row_scale, y, status, stream);
}

int rrnco_train_inst_xty(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* x, const float* y, const float* sx,
                         const float* sy, const float* row_scale, float* c, uint32_t* status, void* stream) {
  if (n_inst == 0 || rows_per_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && rows_per_inst > 0 && n_nodes > 0 && x && y && c && status);
  if (n_nodes > 128 || n_inst > 65535) return RRNCO_ERR_UNSUPPORTED;
  return pt_xty(n_inst, rows_per_inst, n_nodes, kE, x, y, sx, sy, row_scale, c, status, stream);
}

int64_t rrnco_train_inst_tiled_packed_bytes(int64_t n_inst, int32_t n_nodes) {
  if (n_inst <= 0 || n_nodes <= 0 || n_nodes > kPtMaxNodes) return 0;
  return n_inst * ((n_nodes + kFRows - 1) / kFRows) * 2 * (int64_t)kPtTileBytes;
}

int rrnco_train_inst_tiled_pack(int64_t n_inst, int32_t n_nodes, const float* w, int32_t transpose, void* packed, uint32_t* status,
                                void* stream) {
  if (n_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && n_nodes > 0 && w && packed && status && (reinterpret_cast<uintptr_t>(packed) & 15u) == 0);
  if (n_nodes > kPtMaxNodes || n_inst > 65535) return RRNCO_ERR_UNSUPPORTED;
  return pt_pack(n_inst, n_nodes, w, transpose, packed, status, stream);
}

int rrnco_train_inst_tiled_gemm(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, int32_t transpose, const float* x,
                                const void* packed, const float* a_scale, const float* row_scale, float* y, uint32_t* status,
                                void* stream) {
  if (n_inst == 0 || rows_per_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && rows_per_inst > 0 && n_nodes > 0 && x && packed && y && status);
  RRNCO_CHECK_ARG(((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(packed) | reinterpret_cast<uintptr_t>(y)) & 15u) == 0);
  if (n_nodes > kPtMaxNodes || n_inst > 65535) return RRNCO_ERR_UNSUPPORTED;
  const int n_kt = (n_nodes + kFRows - 1) / kFRows, ldz = n_kt * kFRows;
  return transpose ? pt_gemm(n_inst, rows_per_inst, ldz, n_kt, kE, 1, x, packed, a_scale, row_scale, y, status, stream)
                   : pt_gemm(n_inst, rows_per_inst, kE, 1, ldz, n_kt, x, packed, a_scale, row_scale, y, status, stream);
}

int rrnco_train_inst_tiled_xty(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* x, const float* y, const float* sx,
                               const float* sy, const float* row_scale, float* c, uint32_t* status, void* stream) {
  if (n_inst == 0 || rows_per_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && rows_per_inst > 0 && n_nodes > 0 && x && y && c && status);
  if (n_nodes > kPtMaxNodes || n_inst > 65535) return RRNCO_ERR_UNSUPPORTED;
  return pt_xty(n_inst, rows_per_inst, n_nodes, (n_nodes + kFRows - 1) / kFRows * kFRows, x, y, sx, sy, row_scale, c, status, stream);
}

}  // extern "C"
