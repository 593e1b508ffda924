// Shared device helpers for librrnco_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rrnco_b200.h"

#define RRNCO_CHECK_ARG(cond) \
  do {                        \
    if (!(cond)) return RRNCO_ERR_BAD_ARG; \
  } while (0)

// a top-k / top-p pair that can drop an entry (top_k > 0, or 0 < top_p < 1): those calls run the filtered kernels
static inline bool rrnco_filter_active(int32_t top_k, float top_p) { return top_k > 0 || (top_p > 0.f && top_p < 1.f); }

static inline int rrnco_launch_status() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? RRNCO_OK : RRNCO_ERR_CUDA;
}

namespace rrnco {

constexpr int kE = RRNCO_EMBED_DIM;   // 128
constexpr int kH = RRNCO_NUM_HEADS;   // 8
constexpr int kDh = kE / kH;          // 16
constexpr int kF = 4 * kE;            // 512 FFN hidden

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// max / min that return NaN when either operand is NaN (fmaxf / fminf return the other operand): relu(x) = fmax_nan(x, 0)
// keeps a NaN input visible, at the cost of fmaxf (one FMNMX)
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float fmin_nan(float a, float b) {
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- cp.async (LDGSTS) 16-byte copies, L2-only caching for streamed operands -------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gmem_src, bool valid) {
  uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst));
  int n = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem_src), "r"(n));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N));
}

// ---- 3xTF32 tensor-core MMA (fp32-faithful: a*b ~= ah*bh + al*bh + ah*bl) ----------------------
// Round-to-nearest (ties away from zero) to the 10-bit TF32 mantissa = cvt.rna.tf32.f32, but done with two
// integer ops on the full-rate ALU pipe: the conversion instruction issues at quarter rate and was the single most
// executed instruction of the fused kernel (31 % of all instructions, profiles/r1_ncu_source_hotspots.txt).
__device__ __forceinline__ uint32_t f2tf32(float x) { return (__float_as_uint(x) + 0x1000u) & 0xffffe000u; }
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = f2tf32(x);
#ifdef RRNCO_SPLIT_LO_RAW
  lo = __float_as_uint(x - __uint_as_float(hi));  // experiment: let the tensor core truncate the low part
#else
  lo = f2tf32(x - __uint_as_float(hi));
#endif
}
// D(16x8) += A(16x8, row) * B(8x8, col); fragment layouts per PTX ISA mma.m16n8k8.tf32.
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
      "{%0,%1,%2,%3};\n"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// kPasses == 3: 3xTF32 (fp32-faithful); kPasses == 1: single TF32 pass (autocast-like fast mode)
template <int kPasses>
__device__ __forceinline__ void mma_x(float (&d)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4],
                                      const uint32_t (&bh)[2], const uint32_t (&bl)[2]) {
  if (kPasses == 3) {
    mma_tf32(d, al, bh);
    mma_tf32(d, ah, bl);
  }
  mma_tf32(d, ah, bh);
}

// ---- Philox-4x32-10 counter RNG (Gumbel-max sampling) -----------------------------------------
__device__ __forceinline__ uint4 philox4x32(uint4 ctr, uint2 key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
// uniform in the OPEN interval (0,1), 23 bits: (k + 0.5) / 2^23 for k < 2^23 is exact in fp32 (24 significant bits),
// so the largest value is 1 - 2^-24 < 1 and -log(-log(u)) stays finite.  (A 24-bit k would round 16777215.5 up to
// 2^24 and return exactly 1.0 -> +inf Gumbel noise once per 2^24 draws.)
__host__ __device__ __forceinline__ float u01(uint32_t x) { return ((float)(x >> 9) + 0.5f) * (1.0f / 8388608.0f); }

// ---- decode-time logit filters: top-k / top-p (rl4co process_logits, decoding.py:311-361) --------------------------
// A filter keeps the set {j : v_j >= cut} of a row's processed values v (after tanh clipping, the mask as -inf and the
// temperature), so a decoder only needs the cut value and then treats v < cut like a masked entry.
//   top-k (k > 0, at most the row length): cut = the k-th largest v; ties with it are kept, -inf entries take part.
//   top-p (0 < p < 1), applied to the top-k survivors: keep j iff the softmax mass of the entries strictly greater than
//   v_j is < p.  That keeps or drops a tie group as a whole; the top entry is always kept.
// Both cuts are the largest key K with W(K) >= target, W(K) = sum over the entries with key >= K of a weight (1 for
// top-k, exp(v - shift) for top-p), found bit by bit on the order-preserving uint32 key of the float.
__device__ __forceinline__ uint32_t filter_key(float x) {
  const uint32_t u = __float_as_uint(x + 0.f);  // -0 -> +0: key order = float order for every non-NaN value
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
// Row is how the threads that decode one row hold it: row.for_each(f) calls f(v) on each value this thread owns,
// row.sum(x) / row.count(c) reduce over the threads that share the row.  Every one of them returns the same cut.
template <class Row>
__device__ __forceinline__ float filter_cut(const Row& row, int top_k, float top_p, float shift) {
  uint32_t kcut = 0u;  // 0: keep everything
  if (top_k > 0) {
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t cand = kcut | (1u << bit);
      int c = 0;
      row.for_each([&](float v) { c += filter_key(v) >= cand ? 1 : 0; });
      if (row.count(c) >= top_k) kcut = cand;
    }
  }
  if (top_p > 0.f && top_p < 1.f) {
    if (shift == -INFINITY) shift = 0.f;  // no feasible entry (reported by the caller): keep the sums free of NaN
    float tot = 0.f;
    row.for_each([&](float v) { tot += filter_key(v) >= kcut ? __expf(v - shift) : 0.f; });
    const float target = top_p * row.sum(tot);
    uint32_t pcut = 0u;
#pragma unroll 1
    for (int bit = 31; bit >= 0; --bit) {
      const uint32_t cand = pcut | (1u << bit);
      const uint32_t lo = cand > kcut ? cand : kcut;
      float s = 0.f;
      row.for_each([&](float v) { s += filter_key(v) >= lo ? __expf(v - shift) : 0.f; });
      if (row.sum(s) >= target) pcut = cand;
    }
    kcut = pcut > kcut ? pcut : kcut;
  }
  if (kcut <= filter_key(-INFINITY)) return -INFINITY;
  return __uint_as_float((kcut & 0x80000000u) ? (kcut & 0x7fffffffu) : ~kcut);
}
// the whole row in this thread's own memory (no reduction)
struct FilterRowLocal {
  const float* v;
  int n;
  template <class F>
  __device__ __forceinline__ void for_each(F&& f) const {
    for (int i = 0; i < n; ++i) f(v[i]);
  }
  __device__ __forceinline__ float sum(float x) const { return x; }
  __device__ __forceinline__ int count(int c) const { return c; }
};

// ---- per-device launch configuration ----------------------------------------------------------
// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) and the SM count belong to a DEVICE, not to the process: launchers
// remember them per device ordinal (a process may hold tensors on several GPUs).  Races are benign (idempotent).
struct PerDeviceOnce {
  unsigned long long done[4] = {0, 0, 0, 0};  // one bit per device ordinal (< 256)
  // true exactly when the current device has not been configured yet through this object (sets the bit)
  bool first(int* dev_out = nullptr) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    if (dev_out) *dev_out = dev;
    const unsigned long long bit = 1ull << (dev & 63);
    unsigned long long& w = done[(dev >> 6) & 3];
    if (w & bit) return false;
    w |= bit;
    return true;
  }
  void undo() {  // configuration failed: try again on the next call
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
    done[(dev >> 6) & 3] &= ~(1ull << (dev & 63));
  }
};
inline int device_sm_count() {
  static int cache[256] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  int& c = cache[dev & 255];
  if (c == 0) {
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    c = sms;
  }
  return c;
}

}  // namespace rrnco
