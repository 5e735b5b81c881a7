// split16.cuh -- the split-fp16 operand arithmetic shared by the kind::f16 tensor kernels (ce_wide.cu, attention_pair.cu,
// attention_seq.cu, tc_gemm16.cu, tc_dw16.cu, tc_topk.cu): every fp32 operand x is scaled by a power of two that brings its
// maximum magnitude just under the top of the fp16 range and split into hi = fp16(x), lo = fp16(x - hi) (22 significant bits);
// a product is then three kind::f16 passes, hi.hi + hi.lo + lo.hi.  Device helpers here, pre-pass kernels in split16.cu.
#pragma once
#include <cuda_fp16.h>
#include "common.cuh"

namespace rbm_tc {

// power of two that brings a maximum magnitude m into [2^(top_exp - 1), 2^top_exp); 0, inf and nan give 2^top_exp (the products
// of an all-zero operand stay zero, a non-finite operand poisons them)
__host__ __device__ __forceinline__ float pow2_scale(float m, int top_exp) {
  int e = 0;
  if (m > 0.f && m < INFINITY) frexpf(m, &e);  // m = f * 2^e, f in [0.5, 1)
  e = e < -100 ? -100 : (e > 100 ? 100 : e);
  return ldexpf(1.f, top_exp - e);
}

// (x0, x1) -> hi / lo words: fp16 of x0 in the low half, of x1 in the high half
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
  const __half l0 = __float2half_rn(x0 - __half2float(h0)), l1 = __float2half_rn(x1 - __half2float(h1));
  hi = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
  lo = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
}
// 16 values -> 8 packed words each (element 2j in the low half of word j: the order a 16-bit A operand in tensor memory is
// read in)
__device__ __forceinline__ void split_pack16(const float (&g)[16], uint32_t (&hi)[8], uint32_t (&lo)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) split2(g[2 * j], g[2 * j + 1], hi[j], lo[j]);
}
// four values times s -> four fp16 hi + four fp16 lo (8 bytes each)
__device__ __forceinline__ void split4(float4 v, float s, uint2& hi, uint2& lo) {
  const float x[4] = {v.x * s, v.y * s, v.z * s, v.w * s};
  split2(x[0], x[1], hi.x, lo.x);
  split2(x[2], x[3], hi.y, lo.y);
}

// Pre-pass kernels (split16.cu).  Every launch goes to stream st; a launch error is left for the caller's RBM_LAUNCH_CHECK.
// max |x| over a strided [rows, cols] fp32 matrix (cols % 4 == 0, 16-byte aligned rows), atomically max-ed into *out_bits as the
// bit pattern of a non-negative float: order-independent, so the result is deterministic.  *out_bits must start at 0.
void maxabs_launch(const float* src, int64_t ld, int64_t rows, int cols, unsigned* out_bits, int grid, cudaStream_t st);
// scales[i] = pow2_scale(max bits[i], 15) for i = 0, 1: max |x| -> [2^14, 2^15)
void scales_launch(const unsigned* bits, float* scales, cudaStream_t st);
// hi / lo fp16 copies of w[0, 4 n4) * *scale (hi, lo: n4 uint2 each)
void split_w_launch(const float* w, const float* scale, uint2* hi, uint2* lo, int64_t n4, cudaStream_t st);

}  // namespace rbm_tc
