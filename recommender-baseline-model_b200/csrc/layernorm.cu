// layernorm.cu -- both LayerNorm flavours of the reference, forward and backward.
//   RBM_LN_TORCH: y = (x-mu)/sqrt(var_biased+eps)*g+b      NN/models/sas_model/sas.py:39,42,50 (eps 1e-8)
//   RBM_LN_BERT : y = g*(x-mu)/(std_unbiased+eps)+b        NN/models/bert_modules/utils/layer_norm.py:14-17
// One warp per row, row cached in registers (d <= 1024), two-pass moments, warp-shuffle reductions.
// HBM-bound: fwd reads x once / writes y once; bwd reads x, dy once / writes dx once.
#include "common.cuh"

#define LN_MAXD 1024
// A row is owned by a group of GW lanes (GW in {8,16,32}), each caching NV float4: d/4 <= GW*NV.

template <int GW>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = GW / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int NV, int GW>
__device__ __forceinline__ void ln_load_row(const float* __restrict__ p, int d4, int lane, float4 (&v)[NV]) {
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    int c4 = lane + GW * t;
    v[t] = c4 < d4 ? ld4(p + c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

template <int NV, int GW>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float* __restrict__ y,
                                                            float* __restrict__ stats, int64_t rows, int d, float eps,
                                                            int flavour) {
  int lane = threadIdx.x % GW;
  int64_t row = (int64_t)blockIdx.x * (blockDim.x / GW) + (threadIdx.x / GW);
  if (row >= rows) row = rows - 1;  // keep whole warps alive for the shuffles; duplicates rewrite identical values
  int d4 = d >> 2;
  float4 v[NV];
  ln_load_row<NV, GW>(x + row * d, d4, lane, v);
  float s = 0.f;
#pragma unroll
  for (int t = 0; t < NV; ++t) s += (v[t].x + v[t].y) + (v[t].z + v[t].w);
  float mean = group_sum<GW>(s) / (float)d;
  float q = 0.f;
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    if (lane + GW * t < d4) {
      float a = v[t].x - mean, b = v[t].y - mean, c = v[t].z - mean, e = v[t].w - mean;
      q += (a * a + b * b) + (c * c + e * e);
    }
  }
  q = group_sum<GW>(q);
  float rstd;
  if (flavour == RBM_LN_TORCH) rstd = 1.f / sqrtf(q / (float)d + eps);
  else rstd = 1.f / (sqrtf(q / (float)(d - 1)) + eps);
  if (lane == 0 && stats) {
    stats[row * 2] = mean;
    stats[row * 2 + 1] = rstd;
  }
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    int c4 = lane + GW * t;
    if (c4 < d4) {
      float4 g = ld4(gamma + c4 * 4), b = ld4(beta + c4 * 4), o;
      if (flavour == RBM_LN_TORCH) {
        o.x = (v[t].x - mean) * rstd * g.x + b.x; o.y = (v[t].y - mean) * rstd * g.y + b.y;
        o.z = (v[t].z - mean) * rstd * g.z + b.z; o.w = (v[t].w - mean) * rstd * g.w + b.w;
      } else {
        o.x = g.x * (v[t].x - mean) * rstd + b.x; o.y = g.y * (v[t].y - mean) * rstd + b.y;
        o.z = g.z * (v[t].z - mean) * rstd + b.z; o.w = g.w * (v[t].w - mean) * rstd + b.w;
      }
      st4(y + row * d + c4 * 4, o);
    }
  }
}

// Each block owns a contiguous slab of rows; its warps stride over the slab.  Per-lane column accumulators
// for dgamma/dbeta are combined across the block's warps in fixed order and written to partial[block].
#define LN_BWD_WARPS 8
template <int NV, int GW>
__global__ void __launch_bounds__(32 * LN_BWD_WARPS) layernorm_bwd_kernel(
    const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ dy,
    const float* __restrict__ dy2, const float* __restrict__ dres, const float* __restrict__ stats, float* __restrict__ dx,
    float* __restrict__ partial, int64_t rows, int d, int64_t rows_per_block, float eps, int flavour) {
  extern __shared__ float sm[];  // [NG][2][d]
  constexpr int NG = 32 * LN_BWD_WARPS / GW;  // row groups per block
  int lane = threadIdx.x % GW, warp = threadIdx.x / GW;
  int d4 = d >> 2;
  int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  int64_t r1 = r0 + rows_per_block < rows ? r0 + rows_per_block : rows;
  float4 gm[NV], ag[NV], ab[NV];
  ln_load_row<NV, GW>(gamma, d4, lane, gm);
#pragma unroll
  for (int t = 0; t < NV; ++t) ag[t] = ab[t] = make_float4(0.f, 0.f, 0.f, 0.f);
  // all groups of a warp run the same trip count (shuffles need full warps); out-of-range groups are masked
  int64_t span = r1 - r0;
  int64_t trips = (span + NG - 1) / NG;
  for (int64_t it = 0; it < trips; ++it) {
    int64_t row = r0 + it * NG + warp;
    bool live = row < r1;
    if (!live) row = r1 - 1;
    float4 xv[NV], gy[NV];
    ln_load_row<NV, GW>(x + row * d, d4, lane, xv);
    ln_load_row<NV, GW>(dy + row * d, d4, lane, gy);
    if (dy2 != nullptr) {  // the normalised output feeds two consumers: their gradients are summed on the way in
      float4 g2[NV];
      ln_load_row<NV, GW>(dy2 + row * d, d4, lane, g2);
#pragma unroll
      for (int t = 0; t < NV; ++t) {
        gy[t].x += g2[t].x; gy[t].y += g2[t].y; gy[t].z += g2[t].z; gy[t].w += g2[t].w;
      }
    }
    if (!live) {
#pragma unroll
      for (int t = 0; t < NV; ++t) gy[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float mean = stats[row * 2], rstd = stats[row * 2 + 1];
    float sg = 0.f, sgx = 0.f;
#pragma unroll
    for (int t = 0; t < NV; ++t) {
      if (lane + GW * t < d4) {
        float4 xh = make_float4((xv[t].x - mean) * rstd, (xv[t].y - mean) * rstd, (xv[t].z - mean) * rstd, (xv[t].w - mean) * rstd);
        ag[t].x += gy[t].x * xh.x; ag[t].y += gy[t].y * xh.y; ag[t].z += gy[t].z * xh.z; ag[t].w += gy[t].w * xh.w;
        ab[t].x += gy[t].x; ab[t].y += gy[t].y; ab[t].z += gy[t].z; ab[t].w += gy[t].w;
        float4 g = make_float4(gy[t].x * gm[t].x, gy[t].y * gm[t].y, gy[t].z * gm[t].z, gy[t].w * gm[t].w);
        sg += (g.x + g.y) + (g.z + g.w);
        sgx += (g.x * xh.x + g.y * xh.y) + (g.z * xh.z + g.w * xh.w);
        xv[t] = xh;
        gy[t] = g;
      }
    }
    sg = group_sum<GW>(sg);
    sgx = group_sum<GW>(sgx);
    float mg = sg / (float)d;
    float coef;
    if (flavour == RBM_LN_TORCH) coef = rstd / (float)d;
    else {
      float s = 1.f / rstd - eps;
      coef = s > 0.f ? 1.f / ((float)(d - 1) * s) : 0.f;
    }
    float k = coef * sgx;
#pragma unroll
    for (int t = 0; t < NV; ++t) {
      int c4 = lane + GW * t;
      if (c4 < d4 && live) {
        float4 o = make_float4(rstd * (gy[t].x - mg) - xv[t].x * k, rstd * (gy[t].y - mg) - xv[t].y * k,
                               rstd * (gy[t].z - mg) - xv[t].z * k, rstd * (gy[t].w - mg) - xv[t].w * k);
        if (dres != nullptr) {  // gradient of the residual branch that shares this input (x -> LN and x -> + ...)
          const float4 r = ld4(dres + row * d + c4 * 4);
          o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
        }
        st4(dx + row * d + c4 * 4, o);
      }
    }
  }
#pragma unroll
  for (int t = 0; t < NV; ++t) {
    int c4 = lane + GW * t;
    if (c4 < d4) {
      st4(sm + (warp * 2 + 0) * d + c4 * 4, ag[t]);
      st4(sm + (warp * 2 + 1) * d + c4 * 4, ab[t]);
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < 2 * d; c += blockDim.x) {
    int which = c / d, col = c - which * d;
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < NG; ++w) s += sm[(w * 2 + which) * d + col];
    partial[(int64_t)blockIdx.x * 2 * d + c] = s;
  }
}

// out[c] = sum_b partial[b][c] in a fixed order: 32 interleaved groups (b = g, g+32, ... ascending), then the groups
// ascending.  One block = 32 columns x 32 groups (the per-block partials are a few hundred rows: fewer, longer per-thread
// chains were latency-bound -- 18 us for 592 x 128 floats with 8 groups).
__global__ void __launch_bounds__(1024) colsum_partials_kernel(const float* __restrict__ partial, float* __restrict__ out0,
                                                               float* __restrict__ out1, int nblk, int d) {
  __shared__ float acc[32][33];
  const int o = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + o;
  float s = 0.f;
  if (c < 2 * d)
    for (int b = g; b < nblk; b += 32) s += partial[(int64_t)b * 2 * d + c];
  acc[g][o] = s;
  __syncthreads();
  if (g == 0 && c < 2 * d) {
#pragma unroll
    for (int k = 1; k < 32; ++k) s += acc[k][o];
    if (c < d) out0[c] = s;
    else out1[c - d] = s;
  }
}

static int ln_bwd_blocks(int64_t rows) {
  int64_t nb = rbm_cdiv(rows, LN_BWD_WARPS * 16);
  int64_t cap = RBM_NUM_SMS * 4;
  return (int)(nb < cap ? (nb < 1 ? 1 : nb) : cap);
}

extern "C" size_t rbm_layernorm_ws_bytes(int64_t rows, int d) { return (size_t)ln_bwd_blocks(rows) * 2 * d * sizeof(float); }

extern "C" int rbm_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* stats,
                                 int64_t rows, int d, float eps, int flavour, rbm_stream_t stream) {
  RBM_REQUIRE(x && gamma && beta && y, "rbm_layernorm_fwd: null pointer");
  RBM_REQUIRE(d >= 4 && d % 4 == 0 && d <= LN_MAXD, "rbm_layernorm_fwd: unsupported d=%d (need d%%4==0, d<=1024)", d);
  RBM_REQUIRE(flavour == RBM_LN_TORCH || flavour == RBM_LN_BERT, "rbm_layernorm_fwd: bad flavour %d", flavour);
  RBM_REQUIRE(rbm_aligned16(x) && rbm_aligned16(y) && rbm_aligned16(gamma) && rbm_aligned16(beta), "rbm_layernorm_fwd: pointers must be 16B aligned");
  if (rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  int d4 = d / 4;
#define LN_FWD(NV, GW) layernorm_fwd_kernel<NV, GW><<<(unsigned)rbm_cdiv(rows, 256 / GW), 256, 0, st>>>(x, gamma, beta, y, stats, rows, d, eps, flavour)
  if (d4 <= 8) LN_FWD(1, 8);
  else if (d4 <= 16) LN_FWD(1, 16);
  else if (d4 <= 32) LN_FWD(1, 32);
  else if (d4 <= 64) LN_FWD(2, 32);
  else if (d4 <= 128) LN_FWD(4, 32);
  else LN_FWD(8, 32);
#undef LN_FWD
  RBM_LAUNCH_CHECK("rbm_layernorm_fwd");
  return 0;
}

extern "C" int rbm_layernorm_bwd_residual(const float* x, const float* gamma, const float* dy, const float* dres, const float* stats,
                                          float* dx, float* dgamma, float* dbeta, int64_t rows, int d, float eps, int flavour,
                                          void* ws, size_t ws_bytes, rbm_stream_t stream);

extern "C" int rbm_layernorm_bwd(const float* x, const float* gamma, const float* dy, const float* stats, float* dx,
                                 float* dgamma, float* dbeta, int64_t rows, int d, float eps, int flavour, void* ws,
                                 size_t ws_bytes, rbm_stream_t stream) {
  return rbm_layernorm_bwd_residual(x, gamma, dy, nullptr, stats, dx, dgamma, dbeta, rows, d, eps, flavour, ws, ws_bytes, stream);
}

extern "C" int rbm_layernorm_bwd_fanout(const float* x, const float* gamma, const float* dy, const float* dy2, const float* dres,
                                        const float* stats, float* dx, float* dgamma, float* dbeta, int64_t rows, int d, float eps,
                                        int flavour, void* ws, size_t ws_bytes, rbm_stream_t stream);

extern "C" int rbm_layernorm_bwd_residual(const float* x, const float* gamma, const float* dy, const float* dres, const float* stats,
                                          float* dx, float* dgamma, float* dbeta, int64_t rows, int d, float eps, int flavour,
                                          void* ws, size_t ws_bytes, rbm_stream_t stream) {
  return rbm_layernorm_bwd_fanout(x, gamma, dy, nullptr, dres, stats, dx, dgamma, dbeta, rows, d, eps, flavour, ws, ws_bytes, stream);
}

extern "C" int rbm_layernorm_bwd_fanout(const float* x, const float* gamma, const float* dy, const float* dy2, const float* dres,
                                        const float* stats, float* dx, float* dgamma, float* dbeta, int64_t rows, int d, float eps,
                                        int flavour, void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(x && gamma && dy && stats && dx && dgamma && dbeta && ws, "rbm_layernorm_bwd: null pointer");
  RBM_REQUIRE(!dy2 || rbm_aligned16(dy2), "rbm_layernorm_bwd: dy2 must be 16B aligned");
  RBM_REQUIRE(!dres || rbm_aligned16(dres), "rbm_layernorm_bwd: dres must be 16B aligned");
  RBM_REQUIRE(d >= 4 && d % 4 == 0 && d <= LN_MAXD, "rbm_layernorm_bwd: unsupported d=%d", d);
  RBM_REQUIRE(rows > 0, "rbm_layernorm_bwd: rows must be > 0");
  RBM_REQUIRE(ws_bytes >= rbm_layernorm_ws_bytes(rows, d), "rbm_layernorm_bwd: workspace too small");
  RBM_REQUIRE(rbm_aligned16(x) && rbm_aligned16(dy) && rbm_aligned16(dx) && rbm_aligned16(gamma) && rbm_aligned16(ws), "rbm_layernorm_bwd: pointers must be 16B aligned");
  int nblk = ln_bwd_blocks(rows);
  int64_t rpb = rbm_cdiv(rows, nblk);
  cudaStream_t st = (cudaStream_t)stream;
  int d4 = d / 4;
#define LN_BWD(NV, GW)                                                                                              \
  do {                                                                                                              \
    size_t smem = (size_t)(32 * LN_BWD_WARPS / GW) * 2 * d * sizeof(float);                                         \
    if (smem > 48 * 1024 && !set_smem(layernorm_bwd_kernel<NV, GW>, smem, "rbm_layernorm_bwd")) return -1;         \
    layernorm_bwd_kernel<NV, GW><<<nblk, 32 * LN_BWD_WARPS, smem, st>>>(x, gamma, dy, dy2, dres, stats, dx, (float*)ws,  \
                                                                        rows, d, rpb, eps, flavour);                \
  } while (0)
  if (d4 <= 8) LN_BWD(1, 8);
  else if (d4 <= 16) LN_BWD(1, 16);
  else if (d4 <= 32) LN_BWD(1, 32);
  else if (d4 <= 64) LN_BWD(2, 32);
  else if (d4 <= 128) LN_BWD(4, 32);
  else LN_BWD(8, 32);
#undef LN_BWD
  RBM_LAUNCH_CHECK("rbm_layernorm_bwd");
  colsum_partials_kernel<<<(unsigned)rbm_cdiv(2 * d, 32), 1024, 0, (cudaStream_t)stream>>>((const float*)ws, dgamma, dbeta, nblk, d);
  RBM_LAUNCH_CHECK("rbm_layernorm_bwd(colsum)");
  return 0;
}
