// Training hand-off, masked 8-head attention of RRNet_PointerAttention (rrnco/models/decoder.py:281-293) for instances of up to
// 1024 nodes: the same math and conventions as attention_train.cu (which keeps K, V, dK and dV of one instance in shared memory
// and so stops at 102 nodes), with the keys streamed through shared memory in tiles of 32.  CUDA cores, fp32 FMAs throughout.
//   forward:  warp = head, lane = two rows of a 64-row group (one CTA); the K / V tiles are double-buffered (cp.async) and the
//             online softmax runs across them in the log2 domain with the lazy rescale of attention_train.cu.  Keys are visited in
//             the same order with the same arithmetic as rrnco_train_attention_fwd (bitwise equal outputs measured at 101 nodes).
//   backward: dq from 32-row groups (lane = row) that loop over the key tiles and recompute p / ds from the saved log-sum-exp
//             (flash-attention identity D = dO . O; D is written to the workspace); dK / dV from (instance, 32-key tile, row
//             split) work items, lane = key, that loop over the rows of their split staged in shared memory.  Splits write
//             partials that one more kernel adds in a fixed order: no float atomics, the gradients are bitwise reproducible.
#include "../csrc/common.cuh"
#include "../csrc/ffn_pack.cuh"   // ffma2: packed fp32 pairs (two IEEE FMAs per issue slot, same bits as the scalar forms)
#include "../../include/rrnco_b200_train.h"

namespace rrnco {

constexpr int kTaThreads = 256;
constexpr int kTaKeys = 32;        // keys per tile: one mask word per row and tile
constexpr int kTaMaxNodes = 1024;
constexpr float kTaQScale = 0.25f * 1.4426950408889634f;  // 1 / sqrt(16) and log2(e): scores in the log2 domain
constexpr int kTaDkvRows = 32;     // rows staged per step of the dK / dV kernel

__device__ __forceinline__ void load_kv_tile(float* Ks, float* Vs, const float* __restrict__ kb, const float* __restrict__ vb, int j0,
                                             int N, int tid) {
  const int n4 = min(kTaKeys, N - j0) * (kE / 4);
  for (int i = tid; i < n4; i += kTaThreads) {
    cp_async16(Ks + 4 * i, kb + (size_t)j0 * kE + 4 * i);
    cp_async16(Vs + 4 * i, vb + (size_t)j0 * kE + 4 * i);
  }
  cp_async_commit();
}

// mask bytes of rows [g0, g0 + n_rows) -> one 32-key word per (row, tile) in shared memory, a warp per (row, tile): one coalesced
// 32-byte read and a ballot
__device__ __forceinline__ void stage_mask_words(uint32_t* mb, int mstride, const uint8_t* __restrict__ mask, int64_t g0,
                                                 int64_t row_hi, int N, int nt, int n_rows, int warp, int lane) {
  for (int p = warp; p < n_rows * nt; p += kTaThreads / 32) {
    const int r = p / nt, w = p - r * nt, j = w * kTaKeys + lane;
    const bool bit = g0 + r < row_hi && j < N && __ldg(mask + (g0 + r) * N + j) != 0;
    const uint32_t word = __ballot_sync(0xffffffffu, bit);
    if (lane == 0) mb[r * mstride + w] = word;
  }
}

__host__ __device__ constexpr int ta_kv_floats() { return 2 * 2 * kTaKeys * kE; }   // [2 buffers][K | V][32 keys][128]

__global__ void __launch_bounds__(kTaThreads, 2) attn_tiled_fwd_kernel(int64_t L, int N, const float* __restrict__ q,
                                                                      const float* __restrict__ k, const float* __restrict__ v,
                                                                      const uint8_t* __restrict__ mask, int add_res,
                                                                      float* __restrict__ out, float* __restrict__ lse2) {
  extern __shared__ __align__(16) float ta_smem[];
  const int nt = (N + kTaKeys - 1) / kTaKeys, mstride = nt | 1;   // odd word stride: lane-per-row reads are conflict-free
  uint32_t* mb = reinterpret_cast<uint32_t*>(ta_smem + ta_kv_floats());   // [64 rows][mstride]
  const int tid = threadIdx.x, h = tid >> 5, lane = tid & 31;
  const int64_t b = blockIdx.y;
  const int64_t g0 = b * L + (int64_t)blockIdx.x * 64;
  const int64_t row_hi = min(g0 + 64, (b + 1) * L);
  const float* kb = k + b * N * kE;
  const float* vb = v + b * N * kE;
  load_kv_tile(ta_smem, ta_smem + kTaKeys * kE, kb, vb, 0, N, tid);
  stage_mask_words(mb, mstride, mask, g0, row_hi, N, nt, 64, h, lane);
  const int64_t rowa = g0 + lane, rowb = g0 + 32 + lane;
  const bool va = rowa < row_hi, vb_ = rowb < row_hi;
  float qa[16], qb[16], oa[16], ob[16];
  {
    const float4* sa = reinterpret_cast<const float4*>(q + rowa * kE + h * 16);
    const float4* sb = reinterpret_cast<const float4*>(q + rowb * kE + h * 16);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 ta = va ? __ldg(sa + i) : z, tb = vb_ ? __ldg(sb + i) : z;
      qa[4 * i] = ta.x * kTaQScale; qa[4 * i + 1] = ta.y * kTaQScale; qa[4 * i + 2] = ta.z * kTaQScale; qa[4 * i + 3] = ta.w * kTaQScale;
      qb[4 * i] = tb.x * kTaQScale; qb[4 * i + 1] = tb.y * kTaQScale; qb[4 * i + 2] = tb.z * kTaQScale; qb[4 * i + 3] = tb.w * kTaQScale;
    }
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) oa[i] = ob[i] = 0.f;
  float ma = -1e30f, la = 0.f, mbx = -1e30f, lb = 0.f;
#pragma unroll 1
  for (int t = 0; t < nt; ++t) {
    if (t + 1 < nt) {
      float* nxt = ta_smem + ((t + 1) & 1) * 2 * kTaKeys * kE;
      load_kv_tile(nxt, nxt + kTaKeys * kE, kb, vb, (t + 1) * kTaKeys, N, tid);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();   // tile t (and, at t = 0, the mask words) visible to every warp
    const float* Ks = ta_smem + (t & 1) * 2 * kTaKeys * kE;
    const float* Vs = Ks + kTaKeys * kE;
    const uint32_t worda = mb[lane * mstride + t], wordb = mb[(32 + lane) * mstride + t];
    if (__any_sync(0xffffffffu, (worda | wordb) != 0u)) {
      const int jn = min(kTaKeys, N - t * kTaKeys);
#pragma unroll 1
      for (int jj = 0; jj < jn; ++jj) {
        const bool bita = (worda >> jj) & 1u, bitb = (wordb >> jj) & 1u;
        if (!__any_sync(0xffffffffu, bita || bitb)) continue;
        const float4* kp = reinterpret_cast<const float4*>(Ks + jj * kE + h * 16);
        float2 a0 = make_float2(0.f, 0.f), a1 = a0, b0 = a0, b1 = a0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 tk = kp[i];
          a0 = ffma2(make_float2(qa[4 * i], qa[4 * i + 1]), make_float2(tk.x, tk.y), a0);
          a1 = ffma2(make_float2(qa[4 * i + 2], qa[4 * i + 3]), make_float2(tk.z, tk.w), a1);
          b0 = ffma2(make_float2(qb[4 * i], qb[4 * i + 1]), make_float2(tk.x, tk.y), b0);
          b1 = ffma2(make_float2(qb[4 * i + 2], qb[4 * i + 3]), make_float2(tk.z, tk.w), b1);
        }
        const float sa = (a0.x + a0.y) + (a1.x + a1.y), sb = (b0.x + b0.y) + (b1.x + b1.y);
        if (bita && sa > ma + 8.f) {  // lazy rescale, as in attention_train.cu: also across tiles
          const float corr = exp2f(ma - sa);
          la *= corr;
#pragma unroll
          for (int i = 0; i < 16; ++i) oa[i] *= corr;
          ma = sa;
        }
        if (bitb && sb > mbx + 8.f) {
          const float corr = exp2f(mbx - sb);
          lb *= corr;
#pragma unroll
          for (int i = 0; i < 16; ++i) ob[i] *= corr;
          mbx = sb;
        }
        const float wa = bita ? exp2f(sa - ma) : 0.f, wb = bitb ? exp2f(sb - mbx) : 0.f;
        la += wa;
        lb += wb;
        const float4* vp = reinterpret_cast<const float4*>(Vs + jj * kE + h * 16);
        const float2 wa2 = make_float2(wa, wa), wb2 = make_float2(wb, wb);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 tv = vp[i];
          const float2 x0 = ffma2(wa2, make_float2(tv.x, tv.y), make_float2(oa[4 * i], oa[4 * i + 1]));
          const float2 x1 = ffma2(wa2, make_float2(tv.z, tv.w), make_float2(oa[4 * i + 2], oa[4 * i + 3]));
          const float2 y0 = ffma2(wb2, make_float2(tv.x, tv.y), make_float2(ob[4 * i], ob[4 * i + 1]));
          const float2 y1 = ffma2(wb2, make_float2(tv.z, tv.w), make_float2(ob[4 * i + 2], ob[4 * i + 3]));
          oa[4 * i] = x0.x; oa[4 * i + 1] = x0.y; oa[4 * i + 2] = x1.x; oa[4 * i + 3] = x1.y;
          ob[4 * i] = y0.x; ob[4 * i + 1] = y0.y; ob[4 * i + 2] = y1.x; ob[4 * i + 3] = y1.y;
        }
      }
    }
    __syncthreads();   // buffer t & 1 is refilled with tile t + 2 next
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int64_t row = r == 0 ? rowa : rowb;
    if (row < row_hi) {
      const float l = r == 0 ? la : lb, m = r == 0 ? ma : mbx;
      const float inv = l > 0.f ? 1.0f / l : 0.f;
      float4* dst = reinterpret_cast<float4*>(out + row * kE + h * 16);
      const float4* src = reinterpret_cast<const float4*>(q + row * kE + h * 16);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float* o = r == 0 ? oa : ob;
        float4 tt = make_float4(o[4 * i] * inv, o[4 * i + 1] * inv, o[4 * i + 2] * inv, o[4 * i + 3] * inv);
        if (add_res) {
          const float4 u = __ldg(src + i);
          tt.x += u.x; tt.y += u.y; tt.z += u.z; tt.w += u.w;
        }
        dst[i] = tt;
      }
      lse2[row * kH + h] = l > 0.f ? m + log2f(l) : 1e30f;
    }
  }
}

// dq of a 32-row group (lane = row, warp = head) over the streamed key tiles; also writes D = dO . attn [rows, 8] for the dK / dV kernel
__global__ void __launch_bounds__(kTaThreads, 2) attn_tiled_dq_kernel(int64_t L, int N, const float* __restrict__ q,
                                                                     const float* __restrict__ k, const float* __restrict__ v,
                                                                     const uint8_t* __restrict__ mask, const float* __restrict__ out,
                                                                     int add_res, const float* __restrict__ lse2,
                                                                     const float* __restrict__ d_out, float* __restrict__ dq,
                                                                     float* __restrict__ Dw) {
  extern __shared__ __align__(16) float ta_smem[];
  const int nt = (N + kTaKeys - 1) / kTaKeys, mstride = nt | 1;
  uint32_t* mb = reinterpret_cast<uint32_t*>(ta_smem + ta_kv_floats());   // [32 rows][mstride]
  const int tid = threadIdx.x, h = tid >> 5, lane = tid & 31;
  const int64_t b = blockIdx.y;
  const int64_t g0 = b * L + (int64_t)blockIdx.x * 32;
  const int64_t row_hi = min(g0 + 32, (b + 1) * L);
  const float* kb = k + b * N * kE;
  const float* vb = v + b * N * kE;
  load_kv_tile(ta_smem, ta_smem + kTaKeys * kE, kb, vb, 0, N, tid);
  stage_mask_words(mb, mstride, mask, g0, row_hi, N, nt, 32, h, lane);
  const int64_t row = g0 + lane;
  const bool valid = row < row_hi;
  float qs[16], go[16], gq[16];
  float D = 0.f;
  {
    const float4* qsrc = reinterpret_cast<const float4*>(q + row * kE + h * 16);
    const float4* gsrc = reinterpret_cast<const float4*>(d_out + row * kE + h * 16);
    const float4* osrc = reinterpret_cast<const float4*>(out + row * kE + h * 16);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 tq = valid ? __ldg(qsrc + i) : z, tg = valid ? __ldg(gsrc + i) : z;
      float4 to = valid ? __ldg(osrc + i) : z;
      if (add_res) { to.x -= tq.x; to.y -= tq.y; to.z -= tq.z; to.w -= tq.w; }
      qs[4 * i] = tq.x * kTaQScale; qs[4 * i + 1] = tq.y * kTaQScale; qs[4 * i + 2] = tq.z * kTaQScale; qs[4 * i + 3] = tq.w * kTaQScale;
      go[4 * i] = tg.x; go[4 * i + 1] = tg.y; go[4 * i + 2] = tg.z; go[4 * i + 3] = tg.w;
      D = fmaf(tg.x, to.x, D); D = fmaf(tg.y, to.y, D); D = fmaf(tg.z, to.z, D); D = fmaf(tg.w, to.w, D);
    }
  }
  const float lse = valid ? __ldg(lse2 + row * kH + h) : 1e30f;
#pragma unroll
  for (int i = 0; i < 16; ++i) gq[i] = 0.f;
#pragma unroll 1
  for (int t = 0; t < nt; ++t) {
    if (t + 1 < nt) {
      float* nxt = ta_smem + ((t + 1) & 1) * 2 * kTaKeys * kE;
      load_kv_tile(nxt, nxt + kTaKeys * kE, kb, vb, (t + 1) * kTaKeys, N, tid);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* Ks = ta_smem + (t & 1) * 2 * kTaKeys * kE;
    const float* Vs = Ks + kTaKeys * kE;
    const uint32_t word = mb[lane * mstride + t];
    if (__any_sync(0xffffffffu, word != 0u)) {
      const int jn = min(kTaKeys, N - t * kTaKeys);
#pragma unroll 1
      for (int jj = 0; jj < jn; ++jj) {
        const bool bit = (word >> jj) & 1u;
        if (!__any_sync(0xffffffffu, bit)) continue;
        const float4* kp = reinterpret_cast<const float4*>(Ks + jj * kE + h * 16);
        const float4* vp = reinterpret_cast<const float4*>(Vs + jj * kE + h * 16);
        float kr[16], sp[4], dpp[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 a = kp[i], u = vp[i];
          kr[4 * i] = a.x; kr[4 * i + 1] = a.y; kr[4 * i + 2] = a.z; kr[4 * i + 3] = a.w;
          sp[i] = fmaf(qs[4 * i + 3], a.w, fmaf(qs[4 * i + 2], a.z, fmaf(qs[4 * i + 1], a.y, qs[4 * i] * a.x)));
          dpp[i] = fmaf(go[4 * i + 3], u.w, fmaf(go[4 * i + 2], u.z, fmaf(go[4 * i + 1], u.y, go[4 * i] * u.x)));
        }
        const float s = (sp[0] + sp[1]) + (sp[2] + sp[3]), dp = (dpp[0] + dpp[1]) + (dpp[2] + dpp[3]);
        const float p = bit ? exp2f(s - lse) : 0.f;
        const float ds = p * (dp - D);  // gradient of the natural-log-domain score q . k / 4
#pragma unroll
        for (int i = 0; i < 16; ++i) gq[i] = fmaf(ds, kr[i], gq[i]);
      }
    }
    __syncthreads();
  }
  if (valid) {
    float4* dst = reinterpret_cast<float4*>(dq + row * kE + h * 16);
#pragma unroll
    for (int i = 0; i < 4; ++i)
      dst[i] = add_res ? make_float4(fmaf(gq[4 * i], 0.25f, go[4 * i]), fmaf(gq[4 * i + 1], 0.25f, go[4 * i + 1]),
                                     fmaf(gq[4 * i + 2], 0.25f, go[4 * i + 2]), fmaf(gq[4 * i + 3], 0.25f, go[4 * i + 3]))
                       : make_float4(gq[4 * i] * 0.25f, gq[4 * i + 1] * 0.25f, gq[4 * i + 2] * 0.25f, gq[4 * i + 3] * 0.25f);
    Dw[row * kH + h] = D;
  }
}

// dK / dV of one (32-key tile, instance, row split): warp = head, lane = key; the split's rows are staged 32 at a time (scaled q for
// the scores, raw q for dK, dO, log-sum-exp, D and the mask bytes), every read of them is a broadcast.
struct DkvSmem {
  float qs[kTaDkvRows][kE];
  float qr[kTaDkvRows][kE];
  float go[kTaDkvRows][kE];
  float lse[kTaDkvRows][kH];
  float D[kTaDkvRows][kH];
  uint8_t m[kTaDkvRows][kTaKeys];
};

__global__ void __launch_bounds__(kTaThreads, 2) attn_tiled_dkv_kernel(int64_t L, int N, int rows_per_split,
                                                                      const float* __restrict__ q, const float* __restrict__ k,
                                                                      const float* __restrict__ v, const uint8_t* __restrict__ mask,
                                                                      const float* __restrict__ lse2, const float* __restrict__ Dw,
                                                                      const float* __restrict__ d_out, float* __restrict__ dk,
                                                                      float* __restrict__ dv) {
  extern __shared__ __align__(16) float ta_smem[];
  DkvSmem& sm = *reinterpret_cast<DkvSmem*>(ta_smem);
  const int tid = threadIdx.x, h = tid >> 5, lane = tid & 31;
  const int64_t b = blockIdx.y;
  const int j = blockIdx.x * kTaKeys + lane;
  const bool jvalid = j < N;
  const int64_t r_lo = b * L + (int64_t)blockIdx.z * rows_per_split;
  const int64_t r_hi = min(r_lo + rows_per_split, (b + 1) * L);
  float kr[16], vr[16], ak[16], av[16];
  {
    const float4* ks = reinterpret_cast<const float4*>(k + (b * N + (jvalid ? j : 0)) * kE + h * 16);
    const float4* vs = reinterpret_cast<const float4*>(v + (b * N + (jvalid ? j : 0)) * kE + h * 16);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 a = __ldg(ks + i), u = __ldg(vs + i);
      kr[4 * i] = a.x; kr[4 * i + 1] = a.y; kr[4 * i + 2] = a.z; kr[4 * i + 3] = a.w;
      vr[4 * i] = u.x; vr[4 * i + 1] = u.y; vr[4 * i + 2] = u.z; vr[4 * i + 3] = u.w;
    }
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) ak[i] = av[i] = 0.f;
#pragma unroll 1
  for (int64_t g0 = r_lo; g0 < r_hi; g0 += kTaDkvRows) {
    __syncthreads();   // the previous rows are consumed
    for (int i = tid; i < kTaDkvRows * (kE / 4); i += kTaThreads) {
      const int r = i >> 5, c4 = i & 31;
      float4 tq = make_float4(0.f, 0.f, 0.f, 0.f), tg = tq;
      if (g0 + r < r_hi) {
        tq = __ldg(reinterpret_cast<const float4*>(q + (g0 + r) * kE) + c4);
        tg = __ldg(reinterpret_cast<const float4*>(d_out + (g0 + r) * kE) + c4);
      }
      reinterpret_cast<float4*>(sm.qr[r])[c4] = tq;
      reinterpret_cast<float4*>(sm.qs[r])[c4] = make_float4(tq.x * kTaQScale, tq.y * kTaQScale, tq.z * kTaQScale, tq.w * kTaQScale);
      reinterpret_cast<float4*>(sm.go[r])[c4] = tg;
    }
    {
      const int r = tid >> 3, c = tid & 7;   // 32 rows x 8 heads
      const bool ok = g0 + r < r_hi;
      sm.lse[r][c] = ok ? __ldg(lse2 + (g0 + r) * kH + c) : 1e30f;
      sm.D[r][c] = ok ? __ldg(Dw + (g0 + r) * kH + c) : 0.f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int jj = blockIdx.x * kTaKeys + c * 4 + i;
        sm.m[r][c * 4 + i] = (ok && jj < N) ? __ldg(mask + (g0 + r) * N + jj) : (uint8_t)0;
      }
    }
    __syncthreads();
    const int nr = (int)min((int64_t)kTaDkvRows, r_hi - g0);
#pragma unroll 1
    for (int r = 0; r < nr; ++r) {
      const bool bit = sm.m[r][lane] != 0;
      if (!__any_sync(0xffffffffu, bit)) continue;
      const float4* qp = reinterpret_cast<const float4*>(&sm.qs[r][h * 16]);
      const float4* gp = reinterpret_cast<const float4*>(&sm.go[r][h * 16]);
      float sp[4], dpp[4], g[16];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 a = qp[i], u = gp[i];
        g[4 * i] = u.x; g[4 * i + 1] = u.y; g[4 * i + 2] = u.z; g[4 * i + 3] = u.w;
        sp[i] = fmaf(a.w, kr[4 * i + 3], fmaf(a.z, kr[4 * i + 2], fmaf(a.y, kr[4 * i + 1], a.x * kr[4 * i])));
        dpp[i] = fmaf(u.w, vr[4 * i + 3], fmaf(u.z, vr[4 * i + 2], fmaf(u.y, vr[4 * i + 1], u.x * vr[4 * i])));
      }
      const float s = (sp[0] + sp[1]) + (sp[2] + sp[3]), dp = (dpp[0] + dpp[1]) + (dpp[2] + dpp[3]);
      const float p = bit ? exp2f(s - sm.lse[r][h]) : 0.f;
      const float ds = p * (dp - sm.D[r][h]);
      const float4* qq = reinterpret_cast<const float4*>(&sm.qr[r][h * 16]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 a = qq[i];
        ak[4 * i] = fmaf(ds, a.x, ak[4 * i]); ak[4 * i + 1] = fmaf(ds, a.y, ak[4 * i + 1]);
        ak[4 * i + 2] = fmaf(ds, a.z, ak[4 * i + 2]); ak[4 * i + 3] = fmaf(ds, a.w, ak[4 * i + 3]);
      }
#pragma unroll
      for (int i = 0; i < 16; ++i) av[i] = fmaf(p, g[i], av[i]);
    }
  }
  if (jvalid) {   // dk / dv: the output, or the partial of this split ([split][n_inst][N][128])
    const size_t off = ((size_t)blockIdx.z * gridDim.y + b) * N * kE + (size_t)j * kE + h * 16;
    float4* dkp = reinterpret_cast<float4*>(dk + off);
    float4* dvp = reinterpret_cast<float4*>(dv + off);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      dkp[i] = make_float4(ak[4 * i] * 0.25f, ak[4 * i + 1] * 0.25f, ak[4 * i + 2] * 0.25f, ak[4 * i + 3] * 0.25f);
      dvp[i] = make_float4(av[4 * i], av[4 * i + 1], av[4 * i + 2], av[4 * i + 3]);
    }
  }
}

// out[i] = sum over the splits of part[s][i], in split order (float4 i)
__global__ void sum_splits_kernel(int64_t n4, int n_split, const float4* __restrict__ part, float4* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 acc = __ldg(part + i);
    for (int s = 1; s < n_split; ++s) {
      const float4 t = __ldg(part + s * n4 + i);
      acc.x += t.x; acc.y += t.y; acc.z += t.z; acc.w += t.w;
    }
    out[i] = acc;
  }
}

static size_t ta_fwd_smem(int N, int rows) {
  const int nt = (N + kTaKeys - 1) / kTaKeys;
  return (size_t)ta_kv_floats() * sizeof(float) + (size_t)rows * (nt | 1) * sizeof(uint32_t);
}

// row splits of the dK / dV work: enough (key tile, instance, split) items for ~2 waves of 2 CTAs per SM, at least 8 row steps each
static int ta_splits(int64_t n_inst, int64_t L, int N, int* rows_per_split) {
  const int64_t items = (int64_t)((N + kTaKeys - 1) / kTaKeys) * n_inst;
  const int64_t want = 4LL * device_sm_count();
  int64_t s = 1;
  while (s < 64 && s * items < want && (s + 1) * 8 * kTaDkvRows <= L) ++s;
  int64_t rows = (L + s - 1) / s;
  rows = (rows + kTaDkvRows - 1) / kTaDkvRows * kTaDkvRows;
  *rows_per_split = (int)rows;
  return (int)((L + rows - 1) / rows);
}

}  // namespace rrnco

using namespace rrnco;

extern "C" {

int64_t rrnco_train_attention_tiled_workspace_bytes(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes) {
  if (n_inst <= 0 || rows_per_inst <= 0 || n_nodes <= 0 || n_nodes > kTaMaxNodes) return 0;
  int rps = 0;
  const int splits = ta_splits(n_inst, rows_per_inst, n_nodes, &rps);
  const int64_t d = n_inst * rows_per_inst * kH * (int64_t)sizeof(float);
  return d + (splits > 1 ? 2LL * splits * n_inst * n_nodes * kE * (int64_t)sizeof(float) : 0);
}

int rrnco_train_attention_tiled_fwd(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* q, const float* k,
                                    const float* v, const uint8_t* mask, int32_t add_residual, float* out, float* lse, void* stream) {
  if (n_inst == 0 || rows_per_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && rows_per_inst > 0 && n_nodes > 0 && q && k && v && mask && out && lse);
  RRNCO_CHECK_ARG(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
                    reinterpret_cast<uintptr_t>(out)) & 15u) == 0);
  if (n_nodes > kTaMaxNodes || n_inst > 65535) return RRNCO_ERR_UNSUPPORTED;
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(attn_tiled_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ta_fwd_smem(kTaMaxNodes, 64)) !=
            cudaSuccess ||
        cudaFuncSetAttribute(attn_tiled_fwd_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) !=
            cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  attn_tiled_fwd_kernel<<<dim3((unsigned)((rows_per_inst + 63) / 64), (unsigned)n_inst), kTaThreads, ta_fwd_smem(n_nodes, 64),
                          (cudaStream_t)stream>>>(rows_per_inst, n_nodes, q, k, v, mask, add_residual, out, lse);
  return rrnco_launch_status();
}

int rrnco_train_attention_tiled_bwd(int64_t n_inst, int64_t rows_per_inst, int32_t n_nodes, const float* q, const float* k,
                                    const float* v, const uint8_t* mask, const float* out, int32_t add_residual, const float* lse,
                                    const float* d_out, void* workspace, float* dq, float* dk, float* dv, void* stream) {
  if (n_inst == 0 || rows_per_inst == 0) return RRNCO_OK;
  RRNCO_CHECK_ARG(n_inst > 0 && rows_per_inst > 0 && n_nodes > 0 && q && k && v && mask && out && lse && d_out && workspace && dq &&
                  dk && dv);
  RRNCO_CHECK_ARG(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
                    reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(d_out) | reinterpret_cast<uintptr_t>(dq) |
                    reinterpret_cast<uintptr_t>(dk) | reinterpret_cast<uintptr_t>(dv) | reinterpret_cast<uintptr_t>(workspace)) &
                   15u) == 0);
  if (n_nodes > kTaMaxNodes || n_inst > 65535) return RRNCO_ERR_UNSUPPORTED;
  static PerDeviceOnce once;
  if (once.first()) {
    if (cudaFuncSetAttribute(attn_tiled_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ta_fwd_smem(kTaMaxNodes, 32)) !=
            cudaSuccess ||
        cudaFuncSetAttribute(attn_tiled_dq_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) !=
            cudaSuccess ||
        cudaFuncSetAttribute(attn_tiled_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DkvSmem)) != cudaSuccess ||
        cudaFuncSetAttribute(attn_tiled_dkv_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared) !=
            cudaSuccess) {
      once.undo();
      return RRNCO_ERR_CUDA;
    }
  }
  cudaStream_t st = (cudaStream_t)stream;
  float* Dw = reinterpret_cast<float*>(workspace);
  attn_tiled_dq_kernel<<<dim3((unsigned)((rows_per_inst + 31) / 32), (unsigned)n_inst), kTaThreads, ta_fwd_smem(n_nodes, 32), st>>>(
      rows_per_inst, n_nodes, q, k, v, mask, out, add_residual, lse, d_out, dq, Dw);
  int rps = 0;
  const int splits = ta_splits(n_inst, rows_per_inst, n_nodes, &rps);
  const int64_t n = n_inst * n_nodes * kE;
  float* pk = splits > 1 ? Dw + n_inst * rows_per_inst * kH : dk;
  float* pv = splits > 1 ? pk + splits * n : dv;
  attn_tiled_dkv_kernel<<<dim3((unsigned)((n_nodes + kTaKeys - 1) / kTaKeys), (unsigned)n_inst, (unsigned)splits), kTaThreads,
                          sizeof(DkvSmem), st>>>(rows_per_inst, n_nodes, rps, q, k, v, mask, lse, Dw, d_out, pk, pv);
  if (splits > 1) {
    const int64_t n4 = n / 4;
    const int grid = (int)std::min<int64_t>((n4 + 255) / 256, 8LL * device_sm_count());
    sum_splits_kernel<<<grid, 256, 0, st>>>(n4, splits, reinterpret_cast<const float4*>(pk), reinterpret_cast<float4*>(dk));
    sum_splits_kernel<<<grid, 256, 0, st>>>(n4, splits, reinterpret_cast<const float4*>(pv), reinterpret_cast<float4*>(dv));
  }
  return rrnco_launch_status();
}

}  // extern "C"
