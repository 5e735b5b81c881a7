// common.cuh -- shared device helpers for librbm_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/rbm.h"

#define RBM_NUM_SMS 148  // B200: 2 dies x 74 SMs; persistent / capped grids are sized in multiples of this

void rbm_set_error(const char* fmt, ...);

#define RBM_REQUIRE(cond, ...)        \
  do {                                \
    if (!(cond)) {                    \
      rbm_set_error(__VA_ARGS__);     \
      return -1;                      \
    }                                 \
  } while (0)

#define RBM_LAUNCH_CHECK(name)                                              \
  do {                                                                      \
    cudaError_t _e = cudaGetLastError();                                    \
    if (_e != cudaSuccess) {                                                \
      rbm_set_error("%s: launch failed: %s", name, cudaGetErrorString(_e)); \
      return (int)_e;                                                       \
    }                                                                       \
  } while (0)

static inline bool rbm_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static inline int64_t rbm_cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------------------------
// Philox4x32 counter-based RNG.  One call yields 4 x u32 for 4 consecutive logical elements.
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t rbm_mulhi(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
  return __umulhi(a, b);
#else
  return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32);
#endif
}

template <int ROUNDS>
__host__ __device__ __forceinline__ uint4 rbm_philox_rounds(uint64_t seed, uint64_t site, uint64_t idx4) {
  uint32_t c0 = (uint32_t)idx4, c1 = (uint32_t)(idx4 >> 32), c2 = (uint32_t)site, c3 = (uint32_t)(site >> 32);
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < ROUNDS; ++r) {
    uint32_t hi0 = rbm_mulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = rbm_mulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0;
    c1 = lo1;
    c2 = hi0 ^ c3 ^ k1;
    c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
// Philox4x32-10: batch construction and negative sampling (bit-exact against oracle/batches.py and its goldens)
__host__ __device__ __forceinline__ uint4 rbm_philox(uint64_t seed, uint64_t site, uint64_t idx4) {
  return rbm_philox_rounds<10>(seed, site, idx4);
}
// Philox4x32-7 for the dropout sites (element-wise and attention): seven rounds are the fewest that pass BigCrush (Salmon et al.,
// SC'11, table 2; ten is the library default for margin).  Dropout needs independent-looking keep bits, not cryptographic
// margin, and the rounds are a visible share of the softmax / epilogue instruction streams (~100 of them per call).
__host__ __device__ __forceinline__ uint4 rbm_philox_drop(uint64_t seed, uint64_t site, uint64_t idx4) {
  return rbm_philox_rounds<7>(seed, site, idx4);
}

// dropout threshold: an element is KEPT iff its u32 >= thr, i.e. dropped with probability thr / 2^32.
__host__ __device__ __forceinline__ uint32_t rbm_drop_threshold(float p) {
  double t = (double)p * 4294967296.0;
  if (t <= 0.0) return 0u;
  if (t >= 4294967295.0) return 4294967295u;
  return (uint32_t)t;
}

// keep-scale of the 4 elements [4*idx4, 4*idx4+4) of an elementwise site: 0 or 1/(1-p)
__device__ __forceinline__ float4 rbm_drop4(uint64_t seed, uint64_t site, uint64_t idx4, uint32_t thr, float inv_keep) {
  uint4 r = rbm_philox_drop(seed, site, idx4);
  return make_float4(r.x >= thr ? inv_keep : 0.f, r.y >= thr ? inv_keep : 0.f, r.z >= thr ? inv_keep : 0.f,
                     r.w >= thr ? inv_keep : 0.f);
}

// ---------------------------------------------------------------------------------------------
// Step counter for CUDA-graph replay.  Dropout sites are step*64 + local id, with the step baked into the launch
// arguments -- a captured graph would replay the same masks for ever.  rbm_set_step_counter(ptr) installs a device-side
// counter instead: every kernel adds 64 * (*ptr) to its sites (and Adam adds *ptr to its step), the captured graph
// increments the counter itself.  Eager launches (ptr = null) are unchanged, and eager step s equals replay number s of
// a graph captured at step 0, bit for bit.  The pointer lives in one __device__ variable per translation unit.
// ---------------------------------------------------------------------------------------------
static __device__ const unsigned long long* rbm_step_ptr_dev = nullptr;
__device__ __forceinline__ uint64_t rbm_step_offset() {
  const unsigned long long* p = rbm_step_ptr_dev;
  return p ? (uint64_t)*p : 0ull;
}
__device__ __forceinline__ uint64_t rbm_site(uint64_t site) { return site + 64ull * rbm_step_offset(); }
#define RBM_DEFINE_STEP_PTR_SETTER(name) \
  int name(const unsigned long long* p) { return (int)cudaMemcpyToSymbol(rbm_step_ptr_dev, &p, sizeof(p)); }

// Attention-probability sites (L <= 256).  Element (sequence-head bh, query i, key j) takes one 16-bit field of a
// Philox call; it is kept iff field >= p*65536.  The 8 fields of a call are laid out so that both the row-major
// consumers (forward / dQ pass: an mma lane owns rows {g, g+8} x cols {2t, 2t+1} of two adjacent 8-key tiles) and
// the transposed consumer (dK/dV pass) amortise calls:
//   tile = i >> 4, g = i & 7, rh = (i >> 3) & 1;   n = j >> 3, t = (j & 7) >> 1, e = j & 1
//   call  = ((((bh*16 + tile)*8 + g)*4 + t)*16 + (n >> 1));      field = rh*4 + e*2 + (n & 1)
__host__ __device__ __forceinline__ uint64_t rbm_attn_call(uint64_t bh, int tile, int g, int t, int npair) {
  return ((((bh * 16 + (uint64_t)tile) * 8 + (uint64_t)g) * 4 + (uint64_t)t) * 16 + (uint64_t)npair);
}
__host__ __device__ __forceinline__ uint32_t rbm_attn_field(const uint4& r, int f) {
  uint32_t w = (f >> 1) == 0 ? r.x : ((f >> 1) == 1 ? r.y : ((f >> 1) == 2 ? r.z : r.w));
  return (f & 1) ? (w >> 16) : (w & 0xffffu);
}
__host__ __device__ __forceinline__ uint32_t rbm_drop_threshold16(float p) {
  double t = (double)p * 65536.0 + 0.5;
  if (t <= 0.5) return 0u;
  if (t >= 65535.0) return 65535u;
  return (uint32_t)t;
}
// reference implementation of the per-element rule (debug mask kernel, tests)
__host__ __device__ __forceinline__ bool rbm_attn_keep(uint64_t seed, uint64_t site, uint64_t bh, int i, int j, uint32_t thr16) {
  uint4 r = rbm_philox_drop(seed, site, rbm_attn_call(bh, i >> 4, i & 7, (j & 7) >> 1, j >> 4));
  return rbm_attn_field(r, ((i >> 3) & 1) * 4 + (j & 1) * 2 + ((j >> 3) & 1)) >= thr16;
}

// cuTensorMapEncodeTiled is a driver-API call: it needs the primary context current on the CALLING thread.  A thread that
// has not made a context-binding runtime call yet (an autograd worker whose allocations all came from the cache) fails it
// with CUDA_ERROR_INVALID_CONTEXT, so every host thread binds once before its first encode.
inline void rbm_bind_context() {
  static thread_local bool bound = false;
  if (!bound) {
    cudaFree(0);
    bound = true;
  }
}

// raises a kernel's dynamic shared-memory limit; false, with the error recorded under `name`, when the runtime refuses
template <typename K>
inline bool set_smem(K kern, size_t bytes, const char* name) {
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) {
    rbm_set_error("%s: cudaFuncSetAttribute: %s", name, cudaGetErrorString(e));
    return false;
  }
  return true;
}

// ---------------------------------------------------------------------------------------------
// warp helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// TF32 residual of the 3xTF32 products: x minus x with its low 13 mantissa bits cleared (the part the tensor core drops)
__device__ __forceinline__ float tf32_lo(float x) { return x - __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
// dst = tf32_lo(src), elementwise over n4 float4 (layout-agnostic: a swizzled tile stays swizzled)
__device__ __forceinline__ void split_lo(const float* src, float* dst, int n4, int tid, int nthr) {
  for (int i = tid; i < n4; i += nthr) {
    const float4 v = ld4(src + i * 4);
    st4(dst + i * 4, make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w)));
  }
}

// 0.5*x*(1+tanh(u)), u = sqrt(2/pi)*(x+0.044715*x^3)   NN/models/bert_modules/utils/gelu.py:12
// evaluated through the identity 0.5*(1+tanh(u)) = sigmoid(2u) = 1/(1+2^(-2u*log2e)): no 1+tanh cancellation for negative x
// (a few ulp relative error everywhere) and ~8 instructions (ex2 + rcp) instead of libdevice tanhf's ~25 with branches
__device__ __forceinline__ float gelu_sigmoid_2u(float x, float x2) {
  const float c2 = -2.f * 0.7978845608028654f * 1.4426950408889634f;  // -2*sqrt(2/pi)*log2(e)
  const float w = c2 * (x + 0.044715f * x * x2);                      // -2u*log2e
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(w));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));  // 2^w = inf for very negative u: 1/inf = 0
  return r;
}
__device__ __forceinline__ float gelu_tanh_f(float x) { return x * gelu_sigmoid_2u(x, x * x); }
__device__ __forceinline__ float gelu_tanh_grad_f(float x) {
  const float c = 0.7978845608028654f;
  const float x2 = x * x;
  const float s = gelu_sigmoid_2u(x, x2);
  const float du = c * (1.f + 3.f * 0.044715f * x2);
  return s + 2.f * x * s * (1.f - s) * du;  // d/dx [x*sigmoid(2u)]
}
