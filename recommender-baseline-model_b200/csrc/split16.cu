// split16.cu -- pre-pass kernels of the split-fp16 tensor path (split16.cuh): per-tensor max-abs, the power-of-two range
// scales, and the hi / lo fp16 copy of a weight.
#include "split16.cuh"

namespace {

using namespace rbm_tc;

// four independent 16-byte loads per thread and iteration: a one-load grid-stride loop is latency bound (measured 1.2 TB/s)
__global__ void __launch_bounds__(256) maxabs_kernel(const float* __restrict__ src, int64_t ld, int64_t rows, int c4, unsigned* __restrict__ out_bits) {
  float m = 0.f;
  const int64_t n = rows * c4, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < n; i0 += 4 * stride) {
    float4 v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t i = i0 + j * stride;
      v[j] = i < n ? ld4(src + (i / c4) * ld + (i % c4) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) m = fmaxf(fmaxf(m, fmaxf(fabsf(v[j].x), fabsf(v[j].y))), fmaxf(fabsf(v[j].z), fabsf(v[j].w)));
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out_bits, __float_as_uint(m));
}
__global__ void scales_kernel(const unsigned* __restrict__ bits, float* __restrict__ scales) {
  const int i = threadIdx.x;
  if (i >= 2) return;
  scales[i] = pow2_scale(__uint_as_float(bits[i]), 15);
}
__global__ void __launch_bounds__(256) split_w_kernel(const float* __restrict__ w, const float* __restrict__ scale, uint2* __restrict__ hi,
                                                      uint2* __restrict__ lo, int64_t n4) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  uint2 a, b;
  split4(ld4(w + i * 4), *scale, a, b);
  hi[i] = a;
  lo[i] = b;
}

}  // namespace

namespace rbm_tc {

void maxabs_launch(const float* src, int64_t ld, int64_t rows, int cols, unsigned* out_bits, int grid, cudaStream_t st) {
  maxabs_kernel<<<grid, 256, 0, st>>>(src, ld, rows, cols / 4, out_bits);
}
void scales_launch(const unsigned* bits, float* scales, cudaStream_t st) { scales_kernel<<<1, 32, 0, st>>>(bits, scales); }
void split_w_launch(const float* w, const float* scale, uint2* hi, uint2* lo, int64_t n4, cudaStream_t st) {
  split_w_kernel<<<(unsigned)rbm_cdiv(n4, 256), 256, 0, st>>>(w, scale, hi, lo, n4);
}

}  // namespace rbm_tc
