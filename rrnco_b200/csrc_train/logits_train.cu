// Training hand-off, tail of the pointer (rrnco/models/decoder.py:183-198 scale-adaptive edge bias + log(exp(.) + 1e-6),
// rrnco/models/utils/decoding.py:311-361 tanh clip / mask / temperature, :386-399 log-prob of the given action) for the rows
// of the batched replay.  One pass over the raw pointer scores z = g . Lk^T (one warp per row) produces
//   logp[row]            = log pi(a | s)
//   z[row, :]  (in place) <- J = d logp / d z        (the backward pass is then  dz = g_row J, one multiply)
//   a_out[row], b_out[row] = d logp / d alpha, d logp / d beta
// instead of ~25 element-wise ATen passes over [rows, N] tensors (forward + autograd), none of which is saved.
// EPL = elements per lane: 4 for rows of up to 128 scores, 32 for up to 1024 (the key-tiled pointer scores of larger instances).
#include "../csrc/common.cuh"
#include "../../include/rrnco_b200_train.h"

namespace rrnco {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int EPL>
__global__ void __launch_bounds__(256) logits_tail_kernel(int64_t rows, int64_t L, int N, int ldz, float* __restrict__ z,
                                                         const float* __restrict__ dist, const float* __restrict__ dur,
                                                         const int64_t* __restrict__ cur, const uint8_t* __restrict__ mask,
                                                         const int64_t* __restrict__ act, const float* __restrict__ alpha_p,
                                                         const float* __restrict__ beta_p, float inv_sqrt_e, float clip,
                                                         float inv_temp, float* __restrict__ logp, float* __restrict__ a_out,
                                                         float* __restrict__ b_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5), nwarps = (int64_t)gridDim.x * 8;
  const float alpha = __ldg(alpha_p), beta = dur != nullptr ? __ldg(beta_p) : 0.f;
  for (int64_t row = warp0; row < rows; row += nwarps) {
    const int64_t b = row / L;
    const int64_t c = __ldg(cur + row);
    const int a = (int)__ldg(act + row);
    const float* drow = dist + (b * N + c) * N;
    const float* urow = dur != nullptr ? dur + (b * N + c) * N : nullptr;
    float* zrow = z + row * ldz;
    const uint8_t* mrow = mask + row * N;
    float lj[EPL], dj[EPL], uj[EPL], fac[EPL];  // clipped logit / T, distance, duration, d l / d x
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < EPL; ++i) {
      const int j = lane + 32 * i;
      lj[i] = -INFINITY;
      dj[i] = uj[i] = fac[i] = 0.f;
      if (j < N && __ldg(mrow + j) != 0) {
        dj[i] = __ldg(drow + j);
        float bias = alpha * dj[i];
        if (urow != nullptr) {
          uj[i] = __ldg(urow + j);
          bias += beta * uj[i];
        }
        const float x = zrow[j] * inv_sqrt_e - bias;
        const float ex = expf(x);
        const float y = ex + 1e-6f;                     // decoder.py:198: u = log(y)
        const float sig = 1.0f - 1e-6f / y;             // d u / d x = ex / (ex + 1e-6), finite for ex = 0 and ex = inf
        if (clip > 0.f) {                               // decoding.py:332-333
          // tanh(log y) = (y^2 - 1) / (y^2 + 1) = 1 - w,  1 - tanh^2 = w (2 - w),  w = 2 / (y^2 + 1): no log, no tanh, finite for y = inf
          const float w = 2.0f / fmaf(y, y, 1.0f);
          lj[i] = (1.0f - w) * clip * inv_temp;
          fac[i] = clip * w * (2.0f - w) * sig * inv_temp;
        } else {
          lj[i] = logf(y) * inv_temp;
          fac[i] = sig * inv_temp;
        }
        mx = fmaxf(mx, lj[i]);
      }
    }
    mx = warp_max(mx);
    float se = 0.f, ej[EPL];
#pragma unroll
    for (int i = 0; i < EPL; ++i) {
      ej[i] = lj[i] > -INFINITY ? expf(lj[i] - mx) : 0.f;
      se += ej[i];
    }
    se = warp_sum(se);
    const float lse = mx + logf(se), inv_se = 1.0f / se;
    float la = lj[0];
#pragma unroll
    for (int i = 1; i < EPL; ++i) la = (a >> 5) >= i ? lj[i] : la;   // a < N: lj[a >> 5]
    la = __shfl_sync(0xffffffffu, la, a & 31);
    float sa = 0.f, sb = 0.f;
#pragma unroll
    for (int i = 0; i < EPL; ++i) {
      const int j = lane + 32 * i;
      if (j < N) {
        float dx = 0.f;  // d logp / d x_j
        if (lj[i] > -INFINITY) dx = ((j == a ? 1.0f : 0.f) - ej[i] * inv_se) * fac[i];
        zrow[j] = dx * inv_sqrt_e;
        sa = fmaf(-dx, dj[i], sa);
        sb = fmaf(-dx, uj[i], sb);
      } else if (j < ldz) {
        zrow[j] = 0.f;   // padding columns of a 128 ceil(N / 128)-wide score row
      }
    }
    sa = warp_sum(sa);
    sb = warp_sum(sb);
    if (lane == 0) {
      logp[row] = la - lse;
      a_out[row] = sa;
      if (b_out != nullptr) b_out[row] = sb;
    }
  }
}

}  // namespace rrnco

using namespace rrnco;

extern "C" {

int rrnco_train_logits_tail(int64_t rows, int64_t rows_per_inst, int32_t n_nodes, int32_t ldz, float* z, const float* distance,
                            const float* duration, const int64_t* current_node, const uint8_t* mask, const int64_t* action,
                            const float* alpha, const float* beta, float inv_sqrt_e, float tanh_clipping, float temperature,
                            float* logp, float* dlogp_dalpha, float* dlogp_dbeta, void* stream) {
  if (rows == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(rows > 0 && rows_per_inst > 0 && n_nodes > 0 && z && distance && current_node && mask && action && alpha && logp &&
                  dlogp_dalpha && temperature > 0.f);
  RRNCO_CHECK_ARG(duration == nullptr || (beta != nullptr && dlogp_dbeta != nullptr));
  RRNCO_CHECK_ARG(ldz >= n_nodes);
  if (n_nodes > 1024 || ldz > 1024) return RRNCO_ERR_UNSUPPORTED;
  const int sms = device_sm_count();
  int64_t grid = (rows + 7) / 8;
  if (grid > 16LL * sms) grid = 16LL * sms;
  auto kernel = ldz <= 128 ? logits_tail_kernel<4> : logits_tail_kernel<32>;
  kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(rows, rows_per_inst, n_nodes, ldz, z, distance, duration, current_node, mask,
                                                          action, alpha, beta, inv_sqrt_e, tanh_clipping, 1.0f / temperature, logp,
                                                          dlogp_dalpha, dlogp_dbeta);
  return rrnco_launch_status();
}

}  // extern "C"
