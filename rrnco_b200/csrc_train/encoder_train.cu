// Training hand-off of the encoder: backward of the gating neural adaptive bias of an attention-free block
// (DistAngleFusion.forward, rrnco/models/nn/attn_freenet.py:242-289, ATSP / RCVRP two-way gate), the forward of which is
// csrc/encoder_kernels.cu (notation and the collapse to four E-vectors: that file's header).
//
// Per pair p = (i, j) with cost c and angle theta the forward evaluates, from the piecewise-linear segment tables,
//     z = f_gd(c) + f_ga(theta) + cg,  g = sigmoid(z),  Od = f_od(c) + wo.b2d,  Oa = f_oa(theta) + wo.b2a,
//     out = scale (g Od + (1 - g) Oa + bo).
// With the upstream gradient G:  s = scale G,  alpha_d = s g,  alpha_a = s (1 - g),  t = dL/dz = s (Od - Oa) g (1 - g).
// d L / d d = alpha_d wo + t wg_d per pair, so every parameter gradient is a rank-2 expression in the per-unit sums
//     sum alpha h_k = w1_k sum_on alpha x + b1_k sum_on alpha,    sum t h_k = w1_k sum_on t x + b1_k sum_on t
// ("on": unit k active, x = c or theta), and dW1 / db1 need the same four on-sums.  Whether unit k is active depends only
// on the segment of x in the sorted breakpoints (rule of rrnco_nab_pack), so a pass over the pairs only has to histogram
// (alpha x, alpha, t x, t) over the E + 1 segments of each MLP; prefix / suffix sums in rank order give every unit's sums.
// Nothing of size [B, N, N, E] exists; the pass reads 12 B per pair (cost, G, and the coordinates of the instance).
//
// Determinism: the pairs are dealt to CTAs / warps statically; a warp merges the lanes that share a segment in lane order
// (__match_any_sync, fp32, at most 32 terms) and its leader adds the sum to the warp's own fp32 histogram in shared memory
// (at most 128 pairs of one tile); after each tile the CTA adds the warp histograms, in warp order, to its fp64 histogram;
// each CTA writes that as its partial; the partials are reduced in a fixed order.  No atomics: bitwise identical run to
// run on the same device.  (fp32 warp histograms: 54 KB of shared memory per CTA, four CTAs per SM -- the pass is
// latency-bound, and fp64 ones would allow two.)
#include "../csrc/common.cuh"
#include "../../include/rrnco_b200_train.h"

namespace rrnco {

// layout of the forward's `packed` buffer (csrc/encoder_kernels.cu, rrnco_nab_pack); rrnco_train_nab_packed_floats() lets
// the host check it against rrnco_nab_packed_floats() of the rollout library
constexpr int kNabBrute = kE * 8 + 4;
constexpr int kNabTable = kE + (kE + 1) * 4;
constexpr int kNabPacked = kNabBrute + 2 * kNabTable;

constexpr int kNbThreads = 256;
constexpr int kNbWarps = kNbThreads / 32;
constexpr int kNbPairs = 4;                        // pairs per thread and tile (coalesced: pair t + 256 m of the tile)
constexpr int kNbTile = kNbThreads * kNbPairs;
constexpr int kNbSegs = kE + 1;
constexpr int kNbBins = 2 * kNbSegs * 4;           // (mlp, segment, {alpha x, alpha, t x, t})
constexpr int kNbCtasPerSm = 4;
constexpr size_t kNbSmem = (size_t)kNbBins * sizeof(double) + (size_t)kNbWarps * kNbBins * sizeof(float) +
                           (size_t)kNbWarps * 64 * sizeof(float4) + (size_t)(2 * kNabTable + 4) * sizeof(float);
// `params` / `grads`: the 12 tensors of the module in nn.Linear layouts, concatenated
constexpr int kNbMlp = 3 * kE + kE * kE;           // emb.0.weight [E,1], emb.0.bias [E], emb.2.weight [E,E], emb.2.bias [E]
constexpr int kNbGateW = 2 * kNbMlp;               // gate.0.weight [1, 2E]
constexpr int kNbGateB = kNbGateW + 2 * kE;        // gate.0.bias [1]
constexpr int kNbOutW = kNbGateB + 1;              // out_lin.weight [1, E]
constexpr int kNbOutB = kNbOutW + kE;              // out_lin.bias [1]
constexpr int kNbGrads = kNbOutB + 1;

// number of sorted breakpoints strictly below x: the forward's segment search (csrc/encoder_kernels.cu, nab_segment)
__device__ __forceinline__ int nab_segment(const float* __restrict__ t, float x) {
  int pos = 0;
#pragma unroll
  for (int step = kE / 2; step >= 1; step >>= 1) pos += t[pos + step - 1] < x ? step : 0;
  return pos + (t[pos] < x ? 1 : 0);
}

// Adds the four values the lanes staged in `ws` into bin `seg` of the warp histogram `h`: lanes with the same segment are
// summed in lane order by the lowest of them (seg < 0: no pair).
__device__ __forceinline__ void nab_bin(const float4* ws, float* h, int seg, int lane) {
  const unsigned grp = __match_any_sync(0xffffffffu, seg);
  if (seg >= 0 && __ffs(grp) - 1 == lane) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (unsigned m = grp; m; m &= m - 1) {
      const float4 v = ws[__ffs(m) - 1];
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    float* q = h + seg * 4;
    q[0] += a.x; q[1] += a.y; q[2] += a.z; q[3] += a.w;
  }
}

// Persistent grid: CTA c takes the tiles (instance, chunk of kNbTile pairs) c, c + gridDim.x, ...
__global__ void __launch_bounds__(kNbThreads, kNbCtasPerSm) nab_bwd_pairs_kernel(
    int64_t n_inst, int N, const float* __restrict__ coords, const float* __restrict__ cost, int transpose_cost,
    const float* __restrict__ packed, float scale, const float* __restrict__ grad_out, double* __restrict__ partials) {
  extern __shared__ __align__(16) unsigned char smem_nb[];
  double* hcta = reinterpret_cast<double*>(smem_nb);                         // [kNbBins] fp64, the CTA's partial
  float* hist = reinterpret_cast<float*>(hcta + kNbBins);                     // [warps][kNbBins] fp32, one tile
  float4* stage = reinterpret_cast<float4*>(hist + kNbWarps * kNbBins);      // [warps][2][32]
  float* st = reinterpret_cast<float*>(stage + kNbWarps * 64);               // segment tables + 4 constants
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < kNbBins; i += kNbThreads) hcta[i] = 0.0;
  for (int i = tid; i < kNbWarps * kNbBins; i += kNbThreads) hist[i] = 0.f;
  for (int i = tid; i < 2 * kNabTable; i += kNbThreads) st[i] = packed[kNabBrute + i];
  if (tid < 4) st[2 * kNabTable + tid] = packed[kE * 8 + tid];
  __syncthreads();
  const float* td = st;
  const float* ta = st + kNabTable;
  const float cg = st[2 * kNabTable], cod = st[2 * kNabTable + 1], coa = st[2 * kNabTable + 2];
  float* wh = hist + warp * kNbBins;
  float4* ws = stage + warp * 64;
  const int NN = N * N;
  const int chunks = (NN + kNbTile - 1) / kNbTile;
  const int64_t tiles = n_inst * chunks;
  for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const int64_t b = tile / chunks;
    const int p0 = (int)(tile - b * chunks) * kNbTile;
    const float* cb = cost + b * (int64_t)NN;
    const float* gb = grad_out + b * (int64_t)NN;
    const float2* xy = reinterpret_cast<const float2*>(coords + b * (int64_t)N * 2);
    float c[kNbPairs], th[kNbPairs], gr[kNbPairs];
#pragma unroll
    for (int m = 0; m < kNbPairs; ++m) {
      const int p = p0 + m * kNbThreads + tid;
      c[m] = th[m] = gr[m] = 0.f;
      if (p < NN) {
        const int i = p / N, j = p - i * N;
        c[m] = transpose_cost ? __ldg(cb + (size_t)j * N + i) : __ldg(cb + p);
        gr[m] = __ldg(gb + p);
        const float2 pi = __ldg(xy + i), pj = __ldg(xy + j);
        th[m] = atan2f(pi.y - pj.y, pi.x - pj.x);  // attn_freenet.py:254-262
      }
    }
    // all four pairs first (independent segment searches), then the warp-wide binning
    int sd[kNbPairs], sa[kNbPairs];
    float ad[kNbPairs], aa[kNbPairs], t[kNbPairs];
#pragma unroll
    for (int m = 0; m < kNbPairs; ++m) {
      sd[m] = sa[m] = -1;
      ad[m] = aa[m] = t[m] = 0.f;
      if (p0 + m * kNbThreads + tid < NN) {  // the forward's arithmetic (nab_gating_table_kernel), operation for operation
        sd[m] = nab_segment(td, c[m]);
        sa[m] = nab_segment(ta, th[m]);
        const float4 qd = *reinterpret_cast<const float4*>(td + kE + 4 * sd[m]);
        const float4 qa = *reinterpret_cast<const float4*>(ta + kE + 4 * sa[m]);
        const float z = fmaf(qd.x, c[m], qd.y) + fmaf(qa.x, th[m], qa.y) + cg;
        const float g = 1.0f / (1.0f + expf(-z));
        const float od = fmaf(qd.z, c[m], qd.w) + cod, oa = fmaf(qa.z, th[m], qa.w) + coa;
        const float s = scale * gr[m];
        ad[m] = s * g;
        aa[m] = s * (1.0f - g);
        t[m] = s * (od - oa) * (g * (1.0f - g));
      }
    }
#pragma unroll
    for (int m = 0; m < kNbPairs; ++m) {
      ws[lane] = make_float4(ad[m] * c[m], ad[m], t[m] * c[m], t[m]);
      ws[32 + lane] = make_float4(aa[m] * th[m], aa[m], t[m] * th[m], t[m]);
      __syncwarp();
      nab_bin(ws, wh, sd[m], lane);
      nab_bin(ws + 32, wh + kNbSegs * 4, sa[m], lane);
      __syncwarp();
    }
    __syncthreads();  // the tile's warp histograms -> the CTA's fp64 histogram, in warp order
    for (int i = tid; i < kNbBins; i += kNbThreads) {
      float a[kNbWarps];
#pragma unroll
      for (int w = 0; w < kNbWarps; ++w) {
        a[w] = hist[w * kNbBins + i];
        hist[w * kNbBins + i] = 0.f;
      }
      double acc = hcta[i];
#pragma unroll
      for (int w = 0; w < kNbWarps; ++w) acc += a[w];
      hcta[i] = acc;
    }
    __syncthreads();
  }
  for (int i = tid; i < kNbBins; i += kNbThreads) partials[(size_t)blockIdx.x * kNbBins + i] = hcta[i];
}

// totals[bin] = sum of the CTA partials in a fixed order: block = 32 bins, warp w sums partials w, w + 8, ...
__global__ void __launch_bounds__(256) nab_bwd_reduce_kernel(int n_parts, const double* __restrict__ partials,
                                                             double* __restrict__ totals) {
  __shared__ double red[8][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int bin = blockIdx.x * 32 + lane;
  double a = 0.0;
  if (bin < kNbBins)
    for (int c = warp; c < n_parts; c += 8) a += partials[(size_t)c * kNbBins + bin];
  red[warp][lane] = a;
  __syncthreads();
  if (warp == 0 && bin < kNbBins) {
    double t = red[0][lane];
#pragma unroll
    for (int w = 1; w < 8; ++w) t += red[w][lane];
    totals[bin] = t;
  }
}

// One block, fp64: thread (m, k) = hidden unit k of MLP m (0 = dist, 1 = angle).  Recomputes the collapsed vectors and the
// unit ranks exactly as nab_pack_kernel does, turns the segment histogram into the 12 gradients.
__global__ void __launch_bounds__(2 * kE) nab_bwd_finalize_kernel(const double* __restrict__ totals,
                                                                  const float* __restrict__ params, float* __restrict__ grads) {
  __shared__ double s_t[2][kE];
  __shared__ double s_pre[2][kNbSegs][4];  // inclusive prefix sums over the segments
  __shared__ double s_ah[2][kE], s_th[2][kE];  // sum alpha h_k, sum t h_k
  __shared__ double s_dwo[kE];
  const int tid = threadIdx.x, m = tid / kE, k = tid % kE;
  const float* P = params + m * kNbMlp;
  const float* W2 = P + 2 * kE;
  const float* b2 = P + 2 * kE + kE * kE;
  const float* wg = params + kNbGateW + m * kE;  // this MLP's half of the gate weights
  const float* wo = params + kNbOutW;
  const double w = P[k], bb = P[kE + k];
  double ug = 0.0, uo = 0.0;
  for (int e = 0; e < kE; ++e) {
    const double v = W2[e * kE + k];
    ug += v * (double)wg[e];
    uo += v * (double)wo[e];
  }
  s_t[m][k] = w != 0.0 ? -bb / w : INFINITY;
  if (tid < 8) {
    const int mm = tid >> 2, comp = tid & 3;
    double a = 0.0;
    for (int sg = 0; sg < kNbSegs; ++sg) {
      a += totals[(mm * kNbSegs + sg) * 4 + comp];
      s_pre[mm][sg][comp] = a;
    }
  }
  __syncthreads();
  int r = 0;
  for (int j = 0; j < kE; ++j) r += (s_t[m][j] < s_t[m][k] || (s_t[m][j] == s_t[m][k] && j < k)) ? 1 : 0;
  // active segments of unit k: w > 0: rank < s (suffix after r); w < 0: rank >= s (prefix through r); w == 0: all iff b > 0
  const double* tot = s_pre[m][kE];
  double on[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) on[q] = w > 0.0 ? tot[q] - s_pre[m][r][q] : (w < 0.0 ? s_pre[m][r][q] : (bb > 0.0 ? tot[q] : 0.0));
  grads[m * kNbMlp + k] = (float)(uo * on[0] + ug * on[2]);       // emb.0.weight
  grads[m * kNbMlp + kE + k] = (float)(uo * on[1] + ug * on[3]);  // emb.0.bias
  s_ah[m][k] = w * on[0] + bb * on[1];
  s_th[m][k] = w * on[2] + bb * on[3];
  __syncthreads();
  const double sum_t = s_pre[0][kE][3], sum_a = s_pre[m][kE][1];
  // emb.2.weight[e, k] = wo_e sum alpha h_k + wg_e sum t h_k (rank 2)
  for (int i = tid; i < 2 * kE * kE; i += 2 * kE) {
    const int mm = i / (kE * kE), e = (i / kE) % kE, kk = i % kE;
    grads[mm * kNbMlp + 2 * kE + e * kE + kk] =
        (float)((double)wo[e] * s_ah[mm][kk] + (double)params[kNbGateW + mm * kE + e] * s_th[mm][kk]);
  }
  const int e = k;
  double dot_t = 0.0, dot_a = 0.0;
  for (int kk = 0; kk < kE; ++kk) {
    const double v = W2[e * kE + kk];
    dot_t += v * s_th[m][kk];
    dot_a += v * s_ah[m][kk];
  }
  grads[m * kNbMlp + 2 * kE + kE * kE + e] = (float)((double)wo[e] * sum_a + (double)wg[e] * sum_t);  // emb.2.bias
  grads[kNbGateW + m * kE + e] = (float)(dot_t + (double)b2[e] * sum_t);                              // gate.0.weight
  const double dwo = dot_a + (double)b2[e] * sum_a;
  if (m == 1) s_dwo[e] = dwo;
  __syncthreads();
  if (m == 0) grads[kNbOutW + e] = (float)(dwo + s_dwo[e]);  // out_lin.weight
  if (tid == 0) {
    grads[kNbGateB] = (float)sum_t;                                  // gate.0.bias
    grads[kNbOutB] = (float)(s_pre[0][kE][1] + s_pre[1][kE][1]);    // out_lin.bias: sum s
  }
}

inline int64_t nab_bwd_grid(int64_t n_inst, int n_nodes) {
  const int64_t NN = (int64_t)n_nodes * n_nodes;
  const int64_t tiles = n_inst * ((NN + kNbTile - 1) / kNbTile);
  const int64_t cap = (int64_t)kNbCtasPerSm * device_sm_count();
  return tiles < cap ? tiles : cap;
}

}  // namespace rrnco

using namespace rrnco;

extern "C" {

int64_t rrnco_train_nab_packed_floats(void) { return kNabPacked; }

int64_t rrnco_train_nab_grad_floats(void) { return kNbGrads; }

int64_t rrnco_train_nab_workspace_bytes(int64_t n_inst, int32_t n_nodes) {
  if (n_inst <= 0 || n_nodes <= 0) return RRNCO_ERR_BAD_ARG;
  const int64_t grid = nab_bwd_grid(n_inst, n_nodes);
  if (grid <= 0) return RRNCO_ERR_CUDA;
  return (grid + 1) * kNbBins * (int64_t)sizeof(double);
}

int rrnco_train_nab_backward(int64_t n_inst, int32_t n_nodes, const float* coords, const float* cost, int32_t transpose_cost,
                             const float* packed, const float* params, float scale, const float* grad_out, void* workspace,
                             float* grads, void* stream) {
  RRNCO_CHECK_ARG(n_inst > 0 && n_nodes > 0 && coords && cost && packed && params && grad_out && workspace && grads);
  RRNCO_CHECK_ARG((reinterpret_cast<uintptr_t>(coords) & 7u) == 0 && (reinterpret_cast<uintptr_t>(packed) & 15u) == 0 &&
                  (reinterpret_cast<uintptr_t>(workspace) & 7u) == 0);
  // the forward's limits (rrnco_nab_gating): at most 65535 chunks of 1024 pairs per instance
  if ((int64_t)n_nodes * n_nodes > 65535LL * kNbTile) return RRNCO_ERR_UNSUPPORTED;
  const int64_t grid = nab_bwd_grid(n_inst, n_nodes);
  if (grid <= 0) return RRNCO_ERR_CUDA;
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(nab_bwd_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kNbSmem) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  double* partials = static_cast<double*>(workspace);
  double* totals = partials + grid * kNbBins;
  const cudaStream_t s = (cudaStream_t)stream;
  nab_bwd_pairs_kernel<<<(unsigned)grid, kNbThreads, kNbSmem, s>>>(n_inst, n_nodes, coords, cost, transpose_cost, packed, scale,
                                                                  grad_out, partials);
  nab_bwd_reduce_kernel<<<(kNbBins + 31) / 32, 256, 0, s>>>((int)grid, partials, totals);
  nab_bwd_finalize_kernel<<<1, 2 * kE, 0, s>>>(totals, params, grads);
  return rrnco_launch_status();
}

}  // extern "C"
