// Encoder hot spot (SURVEY.md 8(f) rank 4): the gating neural adaptive bias of an attention-free block without the
// duration channel -- DistAngleFusion.forward, rrnco/models/nn/attn_freenet.py:242-289, the variant the encoder builds for
// ATSP and RCVRP (rrnco/models/encoder.py:63-66); one module per block, 2 blocks per layer, 6 layers.
//
// Upstream materialises dist_emb = MLP(cost) and angle_emb = MLP(angle) as [B, N, N, E] tensors (two Linear(E, E) per
// ordered node pair: 65.5 kFLOP and 1 KB of activations per pair and module; 43 GB per block at B' = 8192, N = 101) and
// then keeps four scalar products of them: the gate logit  wg_d . d + wg_a . a + bg  and, because the output layer is
// linear,  wo . (g d + (1 - g) a) + bo = g (wo . d) + (1 - g)(wo . a) + bo.   The second Linear of each MLP is linear too:
//     d = W2d h_d + b2d,  h_d = relu(w1d c + b1d)   =>   wg_d . d = (W2d^T wg_d) . h_d + wg_d . b2d
// so the whole module collapses, exactly in real arithmetic, to four E-vectors u and a few constants per module
// (rrnco_nab_pack, fp64 accumulation), and a pair costs 2 x E relu-FMAs + 4 x E FMAs on the CUDA cores: nothing is
// materialised, the kernel reads the cost entry (4 B) and writes the bias (4 B).  This is NOT GEMM-shaped work (four output
// columns per pair, an A operand that would have to be generated element by element): no tensor cores.
//
// Each of the four collapsed functions  f(x) = sum_k u_k relu(w_k x + b_k)  is PIECEWISE LINEAR in its scalar argument with
// at most E breakpoints t_k = -b_k / w_k.  rrnco_nab_pack therefore also sorts the breakpoints of the two MLPs and tabulates
// slope and intercept of the gate and output functions on each of the E + 1 segments (fp64 prefix sums): the default
// variant of the kernel finds the segment of the cost entry and of the angle by binary search in shared memory and
// evaluates four FMAs -- ~100 instructions per pair instead of ~1000, which moves the kernel from the fp32 pipes toward
// the HBM bound (4 B read + 4 B written per pair).  The brute-force sum over the hidden units (variant 1) is the cross-check.
//
// Layout of `packed` (fp32): [E][8] = (w1d, b1d, ug_d, uo_d, w1a, b1a, ug_a, uo_a) per hidden unit k, 4 constants
// (gate constant, wo . b2d, wo . b2a, bo); then per MLP (dist, angle): E sorted breakpoints, (E + 1) x 4 segment
// coefficients (gate slope, gate intercept, out slope, out intercept).
#include "common.cuh"
#include "ffn_pack.cuh"  // ffma2: packed fp32 pairs

namespace rrnco {

constexpr int kNabThreads = 256;
constexpr int kNabPairs = 4;                                  // pairs per thread: every parameter load serves four pairs
constexpr int kNabBrute = kE * 8 + 4;
constexpr int kNabTable = kE + (kE + 1) * 4;                  // sorted breakpoints + segment coefficients of one MLP
constexpr int kNabPacked = kNabBrute + 2 * kNabTable;

// one block of kE threads: thread k collapses hidden unit k
__global__ void __launch_bounds__(kE) nab_pack_kernel(const float* __restrict__ w1d, const float* __restrict__ b1d,
                                                      const float* __restrict__ W2d, const float* __restrict__ b2d,
                                                      const float* __restrict__ w1a, const float* __restrict__ b1a,
                                                      const float* __restrict__ W2a, const float* __restrict__ b2a,
                                                      const float* __restrict__ wg, const float* __restrict__ bg,
                                                      const float* __restrict__ wo, const float* __restrict__ bo,
                                                      float* __restrict__ packed) {
  const int k = threadIdx.x;
  double ugd = 0.0, uod = 0.0, uga = 0.0, uoa = 0.0;
  for (int e = 0; e < kE; ++e) {  // column k of the second-layer weights (nn.Linear stores [out, in])
    const double vd = W2d[e * kE + k], va = W2a[e * kE + k];
    ugd += vd * (double)wg[e];
    uod += vd * (double)wo[e];
    uga += va * (double)wg[kE + e];
    uoa += va * (double)wo[e];
  }
  float* q = packed + k * 8;
  q[0] = w1d[k]; q[1] = b1d[k]; q[2] = (float)ugd; q[3] = (float)uod;
  q[4] = w1a[k]; q[5] = b1a[k]; q[6] = (float)uga; q[7] = (float)uoa;
  if (k == 0) {
    double cg = bg[0], cod = 0.0, coa = 0.0;
    for (int e = 0; e < kE; ++e) {
      cg += (double)wg[e] * b2d[e] + (double)wg[kE + e] * b2a[e];
      cod += (double)wo[e] * b2d[e];
      coa += (double)wo[e] * b2a[e];
    }
    float* c = packed + kE * 8;
    c[0] = (float)cg; c[1] = (float)cod; c[2] = (float)coa; c[3] = bo[0];
  }
  // ---- piecewise-linear tables of the two MLPs ----
  __shared__ double s_t[kE], s_w[kE], s_b[kE], s_ug[kE], s_uo[kE];
  __shared__ int s_rank[kE];
#pragma unroll 1
  for (int mlp = 0; mlp < 2; ++mlp) {
    const double w = mlp ? (double)w1a[k] : (double)w1d[k], bb = mlp ? (double)b1a[k] : (double)b1d[k];
    __syncthreads();
    s_w[k] = w; s_b[k] = bb; s_ug[k] = mlp ? uga : ugd; s_uo[k] = mlp ? uoa : uod;
    s_t[k] = w != 0.0 ? -bb / w : INFINITY;  // a unit with zero slope never switches: no breakpoint
    __syncthreads();
    int r = 0;
    for (int j = 0; j < kE; ++j) r += (s_t[j] < s_t[k] || (s_t[j] == s_t[k] && j < k)) ? 1 : 0;
    s_rank[k] = r;
    float* tab = packed + kNabBrute + mlp * kNabTable;
    tab[r] = (float)s_t[k];
    __syncthreads();
    // segment s = arguments with exactly s breakpoints strictly below them; unit j is active there iff
    // (w_j > 0 and rank_j < s) or (w_j < 0 and rank_j >= s) or (w_j == 0 and b_j > 0)
    for (int sgm = k; sgm <= kE; sgm += kE) {
      double sg = 0.0, tg = 0.0, so = 0.0, to = 0.0;
      for (int j = 0; j < kE; ++j) {
        const bool on = s_w[j] > 0.0 ? s_rank[j] < sgm : (s_w[j] < 0.0 ? s_rank[j] >= sgm : s_b[j] > 0.0);
        if (on) {
          sg += s_ug[j] * s_w[j]; tg += s_ug[j] * s_b[j];
          so += s_uo[j] * s_w[j]; to += s_uo[j] * s_b[j];
        }
      }
      float* q4 = tab + kE + sgm * 4;
      q4[0] = (float)sg; q4[1] = (float)tg; q4[2] = (float)so; q4[3] = (float)to;
    }
  }
}

// grid (instances, chunks of kNabThreads * kNabPairs pairs); thread t of a chunk owns pairs t, t + 256, t + 512, t + 768 of
// the chunk (pair p = i N + j): loads and stores are coalesced across the warp.
__global__ void __launch_bounds__(kNabThreads) nab_gating_kernel(int N, const float* __restrict__ coords,
                                                                 const float* __restrict__ cost, int transpose_cost,
                                                                 const float* __restrict__ packed, float scale,
                                                                 float* __restrict__ out) {
  __shared__ __align__(16) float sp[kNabBrute];
  const int tid = threadIdx.x;
  for (int i = tid; i < kNabBrute; i += kNabThreads) sp[i] = packed[i];
  __syncthreads();
  const int64_t b = blockIdx.x;
  const int NN = N * N;
  const float* cb = cost + b * (int64_t)NN;
  const float* xy = coords + b * (int64_t)N * 2;
  float c[kNabPairs], th[kNabPairs];
  int pidx[kNabPairs];
#pragma unroll
  for (int m = 0; m < kNabPairs; ++m) {
    const int p = blockIdx.y * (kNabThreads * kNabPairs) + m * kNabThreads + tid;
    pidx[m] = p;
    c[m] = 0.f;
    th[m] = 0.f;
    if (p < NN) {
      const int i = p / N, j = p - i * N;
      c[m] = transpose_cost ? __ldg(cb + (size_t)j * N + i) : __ldg(cb + p);
      const float2 pi = __ldg(reinterpret_cast<const float2*>(xy) + i), pj = __ldg(reinterpret_cast<const float2*>(xy) + j);
      th[m] = atan2f(pi.y - pj.y, pi.x - pj.x);  // attn_freenet.py:254-262
    }
  }
  float gd[kNabPairs] = {0.f, 0.f, 0.f, 0.f}, od[kNabPairs] = {0.f, 0.f, 0.f, 0.f};
  float ga[kNabPairs] = {0.f, 0.f, 0.f, 0.f}, oa[kNabPairs] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
  for (int k = 0; k < kE; ++k) {
    const float4 pd = *reinterpret_cast<const float4*>(&sp[k * 8]);      // w1d, b1d, ug_d, uo_d (shared-memory broadcast)
    const float4 pa = *reinterpret_cast<const float4*>(&sp[k * 8 + 4]);  // w1a, b1a, ug_a, uo_a
#pragma unroll
    for (int m = 0; m < kNabPairs; ++m) {
      const float hd = fmax_nan(fmaf(pd.x, c[m], pd.y), 0.f);  // a NaN scalar stays NaN, as in the table variant
      gd[m] = fmaf(pd.z, hd, gd[m]);
      od[m] = fmaf(pd.w, hd, od[m]);
      const float ha = fmax_nan(fmaf(pa.x, th[m], pa.y), 0.f);
      ga[m] = fmaf(pa.z, ha, ga[m]);
      oa[m] = fmaf(pa.w, ha, oa[m]);
    }
  }
  const float cg = sp[kE * 8], cod = sp[kE * 8 + 1], coa = sp[kE * 8 + 2], bo = sp[kE * 8 + 3];
#pragma unroll
  for (int m = 0; m < kNabPairs; ++m) {
    if (pidx[m] < NN) {
      const float z = gd[m] + ga[m] + cg;
      const float g = 1.0f / (1.0f + expf(-z));  // nn.Sigmoid (attn_freenet.py:239)
      const float y = g * (od[m] + cod) + (1.0f - g) * (oa[m] + coa) + bo;
      out[b * (int64_t)NN + pidx[m]] = y * scale;
    }
  }
}

// number of sorted breakpoints strictly below x (lower bound over kE = 128 entries, 8 shared-memory probes)
__device__ __forceinline__ int nab_segment(const float* __restrict__ t, float x) {
  int pos = 0;
#pragma unroll
  for (int step = kE / 2; step >= 1; step >>= 1) pos += t[pos + step - 1] < x ? step : 0;
  return pos + (t[pos] < x ? 1 : 0);
}

// Table variant: thread t of a chunk owns pairs t, t + 256, ... (coalesced loads / stores), one segment search per scalar.
__global__ void __launch_bounds__(kNabThreads) nab_gating_table_kernel(int N, const float* __restrict__ coords,
                                                                       const float* __restrict__ cost, int transpose_cost,
                                                                       const float* __restrict__ packed, float scale,
                                                                       float* __restrict__ out) {
  __shared__ __align__(16) float st[2 * kNabTable + 4];
  const int tid = threadIdx.x;
  for (int i = tid; i < 2 * kNabTable; i += kNabThreads) st[i] = packed[kNabBrute + i];
  if (tid < 4) st[2 * kNabTable + tid] = packed[kE * 8 + tid];
  __syncthreads();
  const float* td = st;                      // dist: breakpoints, then coefficients
  const float* ta = st + kNabTable;          // angle
  const float cg = st[2 * kNabTable], cod = st[2 * kNabTable + 1], coa = st[2 * kNabTable + 2], bo = st[2 * kNabTable + 3];
  const int64_t b = blockIdx.x;
  const int NN = N * N;
  const float* cb = cost + b * (int64_t)NN;
  const float2* xy = reinterpret_cast<const float2*>(coords + b * (int64_t)N * 2);
#pragma unroll
  for (int m = 0; m < kNabPairs; ++m) {
    const int p = blockIdx.y * (kNabThreads * kNabPairs) + m * kNabThreads + tid;
    if (p < NN) {
      const int i = p / N, j = p - i * N;
      const float c = transpose_cost ? __ldg(cb + (size_t)j * N + i) : __ldg(cb + p);
      const float2 pi = __ldg(xy + i), pj = __ldg(xy + j);
      const float th = atan2f(pi.y - pj.y, pi.x - pj.x);  // attn_freenet.py:254-262
      const float4 qd = *reinterpret_cast<const float4*>(td + kE + 4 * nab_segment(td, c));
      const float4 qa = *reinterpret_cast<const float4*>(ta + kE + 4 * nab_segment(ta, th));
      const float z = fmaf(qd.x, c, qd.y) + fmaf(qa.x, th, qa.y) + cg;
      const float g = 1.0f / (1.0f + expf(-z));
      const float y = g * (fmaf(qd.z, c, qd.w) + cod) + (1.0f - g) * (fmaf(qa.z, th, qa.w) + coa) + bo;
      out[b * (int64_t)NN + p] = y * scale;
    }
  }
}


// ---------------------------------------------------------------------------------------------------------------------
// Fused neural-adaptive-bias + AFT-full of one attention-free block (attn_freenet.py:424-432 + AFTFull.forward :309-327):
//     Y[i,:] = sigmoid(Q[i,:]) * (sum_j a_ij E2[j,:]) / (sum_j a_ij E1[j,:]),
//     a_ij = exp(softmax_j(alpha * adapt_bias[i,j])),  E1 = exp(softmax over the tokens of K),  E2 = E1 * V
// One CTA per instance.  Upstream writes adapt_bias [B,N,N], its softmax, its exp and two [B,N,N] x [B,N,E] products
// through HBM; here the bias row of a node is produced in registers by the segment tables (above), normalised with
// warp shuffles and consumed at once, and E1 / E2 of the instance stay in shared memory: HBM sees Q, K, V, the cost
// matrix once and Y.  Four rows per warp at a time, so that every shared-memory read of an E1 / E2 row serves four rows
// (the products are bound by shared-memory wavefronts otherwise); a_ij travels by shuffle.  fp32 FMAs: the two products are
// 2 x N x N x E = 2.6 MFLOP per instance, far too small and too oddly shaped (N = 101) for a tcgen05 tile.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kAftThreads = 256;
constexpr int kAftRows = 4;            // rows per warp per pass
constexpr int kAftMaxNodes = 128;      // four key slots per lane

template <bool kGiven>  // kGiven: `cost` holds the adapt_bias itself (any gate variant, e.g. from rrnco_nab_dur_gating)
__global__ void __launch_bounds__(kAftThreads, 2) aft_nab_kernel(int N, const float* __restrict__ Q, const float* __restrict__ K,
                                                                 const float* __restrict__ V, const float* __restrict__ coords,
                                                                 const float* __restrict__ cost, int transpose_cost,
                                                                 const float* __restrict__ packed, float scale,
                                                                 float* __restrict__ Y) {
  extern __shared__ __align__(16) float smem_aft[];
  float* E1 = smem_aft;                        // [N][kE]
  float* E2 = E1 + (size_t)N * kE;             // [N][kE]
  float* st = E2 + (size_t)N * kE;             // segment tables (2 * kNabTable + 4)
  float2* xy = reinterpret_cast<float2*>(st + 2 * kNabTable + 4);  // [N]
  float* red = reinterpret_cast<float*>(xy + kAftMaxNodes);        // [2][kE] column-softmax exchange
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t b = blockIdx.x;
  const float* Kb = K + b * (int64_t)N * kE;
  const float* Vb = V + b * (int64_t)N * kE;
  const float* Qb = Q + b * (int64_t)N * kE;
  if (!kGiven) {
    for (int i = tid; i < 2 * kNabTable; i += kAftThreads) st[i] = packed[kNabBrute + i];
    if (tid < 4) st[2 * kNabTable + tid] = packed[kE * 8 + tid];
    if (tid < N) xy[tid] = __ldg(reinterpret_cast<const float2*>(coords + b * (int64_t)N * 2) + tid);
  }
  // ---- E1 = exp(softmax over the tokens (dim = 1) of K), E2 = E1 * V (attn_freenet.py:320-322): thread = (column, row half) ----
  {
    const int d = tid & (kE - 1), half = tid >> 7;
    const int j0 = half ? N / 2 : 0, j1 = half ? N : N / 2;
    float mx = -INFINITY;
#pragma unroll 8
    for (int j = j0; j < j1; ++j) mx = fmaxf(mx, __ldg(Kb + (size_t)j * kE + d));
    red[half * kE + d] = mx;
    __syncthreads();
    mx = fmaxf(red[d], red[kE + d]);
    float sum = 0.f;
#pragma unroll 8
    for (int j = j0; j < j1; ++j) sum += expf(__ldg(Kb + (size_t)j * kE + d) - mx);
    __syncthreads();
    red[half * kE + d] = sum;
    __syncthreads();
    sum = red[d] + red[kE + d];
    const float inv_sum = 1.0f / sum;
#pragma unroll 4
    for (int j = j0; j < j1; ++j) {
      const float e = expf(expf(__ldg(Kb + (size_t)j * kE + d) - mx) * inv_sum);
      E1[(size_t)j * kE + d] = e;
      E2[(size_t)j * kE + d] = e * __ldg(Vb + (size_t)j * kE + d);
    }
  }
  __syncthreads();
  const float* td = st;
  const float* ta = st + kNabTable;
  const float cg = st[2 * kNabTable], cod = st[2 * kNabTable + 1], coa = st[2 * kNabTable + 2], bo = st[2 * kNabTable + 3];
  const float* cb = cost + b * (int64_t)N * N;
  // ---- rows: warp w owns rows 4 (w + 8 t) .. + 3 ----
  for (int i0 = warp * kAftRows; i0 < N; i0 += (kAftThreads / 32) * kAftRows) {
    float a[kAftRows][4];  // a_ij of row i0 + r, key j = lane + 32 m
#pragma unroll
    for (int r = 0; r < kAftRows; ++r) {
      const int i = min(i0 + r, N - 1);  // (rows beyond N repeat the last one; they are not stored)
      const float2 pi = kGiven ? make_float2(0.f, 0.f) : xy[i];
      float bias[4];
      float mx = -INFINITY;
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        const int j = lane + 32 * m;
        bias[m] = -INFINITY;
        if (j < N) {
          const float c = transpose_cost ? __ldg(cb + (size_t)j * N + i) : __ldg(cb + (size_t)i * N + j);
          if (kGiven) {
            bias[m] = c * scale;
          } else {
            const float2 pj = xy[j];
            const float th = atan2f(pi.y - pj.y, pi.x - pj.x);
            const float4 qd = *reinterpret_cast<const float4*>(td + kE + 4 * nab_segment(td, c));
            const float4 qa = *reinterpret_cast<const float4*>(ta + kE + 4 * nab_segment(ta, th));
            const float z = fmaf(qd.x, c, qd.y) + fmaf(qa.x, th, qa.y) + cg;
            const float g = 1.0f / (1.0f + expf(-z));
            bias[m] = (g * (fmaf(qd.z, c, qd.w) + cod) + (1.0f - g) * (fmaf(qa.z, th, qa.w) + coa) + bo) * scale;
          }
        }
        mx = fmaxf(mx, bias[m]);
      }
      mx = warp_max(mx);
      float sum = 0.f;
#pragma unroll
      for (int m = 0; m < 4; ++m) {
        bias[m] = expf(bias[m] - mx);  // exp(-inf) = 0 for the slots beyond N
        sum += bias[m];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
#pragma unroll
      for (int m = 0; m < 4; ++m) a[r][m] = lane + 32 * m < N ? expf(bias[m] / sum) : 0.f;  // exp(softmax) (attn_freenet.py:319-321)
    }
    // num / den over the keys; lane owns output dims 4 lane .. 4 lane + 3 (packed fp32 pairs: two FMAs per issue slot)
    float2 num[kAftRows][2], den[kAftRows][2];
#pragma unroll
    for (int r = 0; r < kAftRows; ++r) num[r][0] = num[r][1] = den[r][0] = den[r][1] = make_float2(0.f, 0.f);
#pragma unroll
    for (int m = 0; m < 4; ++m) {
      const int jn = min(32, N - 32 * m);
#pragma unroll 4
      for (int jj = 0; jj < jn; ++jj) {
        const int j = 32 * m + jj;
        const float4 e2 = *reinterpret_cast<const float4*>(E2 + (size_t)j * kE + 4 * lane);
        const float4 e1 = *reinterpret_cast<const float4*>(E1 + (size_t)j * kE + 4 * lane);
#pragma unroll
        for (int r = 0; r < kAftRows; ++r) {
          const float w = __shfl_sync(0xffffffffu, a[r][m], jj);
          const float2 ww = make_float2(w, w);
          num[r][0] = ffma2(ww, make_float2(e2.x, e2.y), num[r][0]);
          num[r][1] = ffma2(ww, make_float2(e2.z, e2.w), num[r][1]);
          den[r][0] = ffma2(ww, make_float2(e1.x, e1.y), den[r][0]);
          den[r][1] = ffma2(ww, make_float2(e1.z, e1.w), den[r][1]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < kAftRows; ++r) {
      const int i = i0 + r;
      if (i < N) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(Qb + (size_t)i * kE) + lane);
        float4 y;
        y.x = num[r][0].x / den[r][0].x / (1.0f + expf(-q.x)); y.y = num[r][0].y / den[r][0].y / (1.0f + expf(-q.y));
        y.z = num[r][1].x / den[r][1].x / (1.0f + expf(-q.z)); y.w = num[r][1].y / den[r][1].y / (1.0f + expf(-q.w));
        reinterpret_cast<float4*>(Y + (b * (int64_t)N + i) * kE)[lane] = y;
      }
    }
  }
}

}  // namespace rrnco

using namespace rrnco;

extern "C" {

int64_t rrnco_nab_packed_floats(void) { return kNabPacked; }

int rrnco_nab_pack(const float* dist_w1, const float* dist_b1, const float* dist_w2, const float* dist_b2,
                   const float* angle_w1, const float* angle_b1, const float* angle_w2, const float* angle_b2,
                   const float* gate_w, const float* gate_b, const float* out_w, const float* out_b, float* packed,
                   void* stream) {
  RRNCO_CHECK_ARG(dist_w1 && dist_b1 && dist_w2 && dist_b2 && angle_w1 && angle_b1 && angle_w2 && angle_b2 && gate_w &&
                  gate_b && out_w && out_b && packed);
  nab_pack_kernel<<<1, kE, 0, (cudaStream_t)stream>>>(dist_w1, dist_b1, dist_w2, dist_b2, angle_w1, angle_b1, angle_w2, angle_b2,
                                                      gate_w, gate_b, out_w, out_b, packed);
  return rrnco_launch_status();
}

int rrnco_nab_gating(int64_t n_inst, int32_t n_nodes, const float* coords, const float* cost, int32_t transpose_cost,
                     const float* packed, float scale, int32_t variant, float* out, void* stream) {
  RRNCO_CHECK_ARG(n_inst > 0 && n_nodes > 0 && coords && cost && packed && out);
  RRNCO_CHECK_ARG((reinterpret_cast<uintptr_t>(coords) & 7u) == 0 && (reinterpret_cast<uintptr_t>(packed) & 15u) == 0);
  const int per_cta = kNabThreads * kNabPairs;
  const int64_t chunks = ((int64_t)n_nodes * n_nodes + per_cta - 1) / per_cta;
  if (n_inst > 0x7fffffffLL || chunks > 65535) return RRNCO_ERR_UNSUPPORTED;
  const dim3 grid((unsigned)n_inst, (unsigned)chunks);
  RRNCO_CHECK_ARG(variant == 0 || variant == 1);
  if (variant == 0)
    nab_gating_table_kernel<<<grid, kNabThreads, 0, (cudaStream_t)stream>>>(n_nodes, coords, cost, transpose_cost, packed, scale, out);
  else
    nab_gating_kernel<<<grid, kNabThreads, 0, (cudaStream_t)stream>>>(n_nodes, coords, cost, transpose_cost, packed, scale, out);
  return rrnco_launch_status();
}


int rrnco_aft_nab(int64_t n_inst, int32_t n_nodes, const float* q, const float* k, const float* v, const float* coords,
                  const float* cost, int32_t transpose_cost, const float* packed, float scale, float* out, void* stream) {
  // packed == NULL: `cost` is the adapt_bias [B,N,N] itself (times `scale`), coords unused
  RRNCO_CHECK_ARG(n_inst > 0 && n_nodes > 0 && q && k && v && cost && out && (packed == nullptr || coords != nullptr));
  RRNCO_CHECK_ARG(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(out)) & 15u) == 0 &&
                  (reinterpret_cast<uintptr_t>(coords) & 7u) == 0);
  if (n_nodes > kAftMaxNodes || n_inst > 0x7fffffffLL) return RRNCO_ERR_UNSUPPORTED;
  const size_t smem = ((size_t)2 * n_nodes * kE + 2 * kNabTable + 4 + 2 * kAftMaxNodes + 2 * kE) * sizeof(float);
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(aft_nab_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(aft_nab_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess ||
        cudaFuncSetAttribute(aft_nab_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024) != cudaSuccess ||
        cudaFuncSetAttribute(aft_nab_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) != cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  if (packed)
    aft_nab_kernel<false><<<(unsigned)n_inst, kAftThreads, smem, (cudaStream_t)stream>>>(n_nodes, q, k, v, coords, cost, transpose_cost,
                                                                                        packed, scale, out);
  else
    aft_nab_kernel<true><<<(unsigned)n_inst, kAftThreads, smem, (cudaStream_t)stream>>>(n_nodes, q, k, v, coords, cost, transpose_cost,
                                                                                       packed, scale, out);
  return rrnco_launch_status();
}

}  // extern "C"
