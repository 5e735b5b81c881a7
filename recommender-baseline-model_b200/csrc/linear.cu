// linear.cu -- fp32 Linear layers with fused epilogues (bias, activation, two dropouts, residual, pad-row
// zeroing) and their backward GEMMs.  Replaces the nn.Linear / Conv1d(k=1) + Dropout + activation + residual
// chains of NN/models/bert_modules/{attention/multi_head.py:29-40, utils/feed_forward.py:16, utils/sublayer.py:18,
// transformer.py:32} and NN/models/sas_model/sas.py:16-19,75,79,84.
//
// Round-1 implementation: register-tiled SIMT fp32 GEMM (exact fp32 parity with the reference).  The tcgen05 /
// TMEM path for these shapes is tracked in DESIGN.md ("next").
#include "common.cuh"
#include "tc_gemm.cuh"
#include "tc_dw16.cuh"
#include "tc_gemm16.cuh"

namespace {

constexpr int BK = 16;
constexpr int PAD = 4;

struct Epilogue {
  const float* bias;
  float* pre;
  const float* residual;
  int64_t ldres;
  const int64_t* row_tok;
  int act;
  uint32_t thrA, thrB;
  float invA, invB;
  uint64_t siteA, siteB, seed;
};

__device__ __forceinline__ float act_apply(float v, int act) {
  if (act == RBM_ACT_RELU) return fmaxf(v, 0.f);
  if (act == RBM_ACT_GELU_TANH) return gelu_tanh_f(v);
  return v;
}

// ---------------------------------------------------------------------------------------------------------
// C[M,N] = A[M,K] . B^T   (B_NK: B is [N,K] row-major)     -- forward
// C[M,N] = A[M,K] . B     (!B_NK: B is [K,N] row-major)    -- backward-data
// 128x64 tile, 256 threads, 8x4 register micro-tile, BK=16, register-prefetch double buffering.
// ---------------------------------------------------------------------------------------------------------
template <bool B_NK, bool HAS_EPI>
__global__ void __launch_bounds__(256) gemm_rowmajor_kernel(const float* __restrict__ A, int64_t lda,
                                                            const float* __restrict__ B, int64_t ldb,
                                                            float* __restrict__ C, int64_t ldc, int64_t M, int N, int K,
                                                            Epilogue ep) {
  constexpr int BM = 128, BN = 64, TM = 8, TN = 4;
  __shared__ __align__(16) float As[2][BK][BM + PAD];
  __shared__ __align__(16) float Bs[2][BK][BN + PAD];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  float4 ra[2], rb;
  auto gload = [&](int k0) {
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      int li = tid + t * 256, m = li >> 2, kq = li & 3;
      int64_t gm = m0 + m;
      int gk = k0 + kq * 4;
      ra[t] = (gm < M && gk < K) ? ld4(A + gm * lda + gk) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (B_NK) {
      int n = tid >> 2, kq = tid & 3;
      int gn = n0 + n, gk = k0 + kq * 4;
      rb = (gn < N && gk < K) ? ld4(B + (int64_t)gn * ldb + gk) : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
      int kk = tid >> 4, nq = tid & 15;
      int gk = k0 + kk, gn = n0 + nq * 4;
      rb = (gk < K && gn < N) ? ld4(B + (int64_t)gk * ldb + gn) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      int li = tid + t * 256, m = li >> 2, kq = li & 3;
      As[buf][kq * 4 + 0][m] = ra[t].x;
      As[buf][kq * 4 + 1][m] = ra[t].y;
      As[buf][kq * 4 + 2][m] = ra[t].z;
      As[buf][kq * 4 + 3][m] = ra[t].w;
    }
    if (B_NK) {
      int n = tid >> 2, kq = tid & 3;
      Bs[buf][kq * 4 + 0][n] = rb.x;
      Bs[buf][kq * 4 + 1][n] = rb.y;
      Bs[buf][kq * 4 + 2][n] = rb.z;
      Bs[buf][kq * 4 + 3][n] = rb.w;
    } else {
      int kk = tid >> 4, nq = tid & 15;
      st4(&Bs[buf][kk][nq * 4], rb);
    }
  };

  const int nk = (K + BK - 1) / BK;
  gload(0);
  sstore(0);
  __syncthreads();
  for (int kt = 0; kt < nk; ++kt) {
    int buf = kt & 1;
    if (kt + 1 < nk) gload((kt + 1) * BK);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a0 = ld4(&As[buf][kk][ty * TM]), a1 = ld4(&As[buf][kk][ty * TM + 4]);
      float4 b = ld4(&Bs[buf][kk][tx * TN]);
      float a[TM] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      float bb[TN] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    if (kt + 1 < nk) {
      sstore(buf ^ 1);
      __syncthreads();
    }
  }

  const int col = n0 + tx * TN;
  if (col >= N) return;
  float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (HAS_EPI && ep.bias) bias4 = ld4(ep.bias + col);
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int64_t row = m0 + ty * TM + i;
    if (row >= M) break;
    float4 v = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    if (HAS_EPI) {
      v.x += bias4.x; v.y += bias4.y; v.z += bias4.z; v.w += bias4.w;
      if (ep.pre) st4(ep.pre + row * N + col, v);
      v.x = act_apply(v.x, ep.act); v.y = act_apply(v.y, ep.act); v.z = act_apply(v.z, ep.act); v.w = act_apply(v.w, ep.act);
      uint64_t e4 = (uint64_t)(row * N + col) >> 2;
      if (ep.thrA) {
        float4 m = rbm_drop4(ep.seed, rbm_site(ep.siteA), e4, ep.thrA, ep.invA);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      if (ep.residual) {
        float4 r = ld4(ep.residual + row * ep.ldres + col);
        v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
      }
      if (ep.thrB) {
        float4 m = rbm_drop4(ep.seed, rbm_site(ep.siteB), e4, ep.thrB, ep.invB);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      if (ep.row_tok && ep.row_tok[row] == 0) v = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    st4(C + row * ldc + col, v);
  }
}

// ---------------------------------------------------------------------------------------------------------
// dW partial[s][N,K] = sum over token rows of split s of  dpre[r, n] * x[r, k]   (reduction over rows)
// 64x64 tile, 256 threads, 4x4 micro-tile.  Column sums of dpre (bias grad) by the k-tile-0 blocks.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gemm_tn_split_kernel(const float* __restrict__ A, int64_t lda,
                                                            const float* __restrict__ B, int64_t ldb,
                                                            float* __restrict__ part, float* __restrict__ part_b,
                                                            int64_t M, int N, int K, int64_t rows_per_split) {
  constexpr int BT = 64, T = 4;
  __shared__ __align__(16) float As[2][BK][BT + PAD];
  __shared__ __align__(16) float Bs[2][BK][BT + PAD];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n0 = blockIdx.x * BT;  // output row tile (N: columns of dpre)
  const int k0 = blockIdx.y * BT;  // output col tile (K: columns of x)
  const int64_t r_begin = (int64_t)blockIdx.z * rows_per_split;
  const int64_t r_end = r_begin + rows_per_split < M ? r_begin + rows_per_split : M;

  float acc[T][T];
  float bsum[T] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < T; ++i)
#pragma unroll
    for (int j = 0; j < T; ++j) acc[i][j] = 0.f;

  float4 ra, rb;
  const int lr = tid >> 4, lq = tid & 15;
  auto gload = [&](int64_t r0) {
    int64_t gr = r0 + lr;
    int gn = n0 + lq * 4, gk = k0 + lq * 4;
    ra = (gr < r_end && gn < N) ? ld4(A + gr * lda + gn) : make_float4(0.f, 0.f, 0.f, 0.f);
    rb = (gr < r_end && gk < K) ? ld4(B + gr * ldb + gk) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  auto sstore = [&](int buf) {
    st4(&As[buf][lr][lq * 4], ra);
    st4(&Bs[buf][lr][lq * 4], rb);
  };
  const int64_t nt = (r_end - r_begin + BK - 1) / BK;
  if (nt > 0) {
    gload(r_begin);
    sstore(0);
  }
  __syncthreads();
  for (int64_t it = 0; it < nt; ++it) {
    int buf = (int)(it & 1);
    if (it + 1 < nt) gload(r_begin + (it + 1) * BK);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float4 a = ld4(&As[buf][kk][ty * T]);
      float4 b = ld4(&Bs[buf][kk][tx * T]);
      float av[T] = {a.x, a.y, a.z, a.w}, bv[T] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < T; ++i) {
#pragma unroll
        for (int j = 0; j < T; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        bsum[i] += av[i];
      }
    }
    if (it + 1 < nt) {
      sstore(buf ^ 1);
      __syncthreads();
    }
  }
  float* out = part + (int64_t)blockIdx.z * N * K;
  const int col = k0 + tx * T;
#pragma unroll
  for (int i = 0; i < T; ++i) {
    int row = n0 + ty * T + i;
    if (row < N && col < K) st4(out + (int64_t)row * K + col, make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]));
    if (part_b && blockIdx.y == 0 && tx == 0 && row < N) part_b[(int64_t)blockIdx.z * N + row] = bsum[i];
  }
}

// out[i] = sum_s part[s][i] in a fixed order: eight interleaved groups (s = g, g+8, ... ascending), then the groups
// ascending.  One block = 32 float4 outputs x 8 groups; blocks [0, nblk_w) reduce the weight partials, the rest the bias
// partials (part_b may be null).  n and nb are multiples of 4.
__global__ void __launch_bounds__(256) reduce_splits_kernel(const float* __restrict__ part, float* __restrict__ out, int64_t n, int nblk_w,
                                                            const float* __restrict__ part_b, float* __restrict__ out_b, int64_t nb,
                                                            int S) {
  __shared__ float4 acc[8][32];
  const int o = threadIdx.x & 31, g = threadIdx.x >> 5;
  const bool is_b = (int)blockIdx.x >= nblk_w;
  const float* src = is_b ? part_b : part;
  float* dst = is_b ? out_b : out;
  const int64_t len = is_b ? nb : n;
  const int64_t i4 = (int64_t)(is_b ? blockIdx.x - nblk_w : blockIdx.x) * 32 + o;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i4 * 4 < len)
    for (int s = g; s < S; s += 8) {
      const float4 v = ld4(src + (int64_t)s * len + i4 * 4);
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
  acc[g][o] = a;
  __syncthreads();
  if (g == 0 && i4 * 4 < len) {
#pragma unroll
    for (int k = 1; k < 8; ++k) {
      const float4 v = acc[k][o];
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
    if (is_b) {  // the bias gradient pointer is only required to be 4-byte aligned
      dst[i4 * 4] = a.x; dst[i4 * 4 + 1] = a.y; dst[i4 * 4 + 2] = a.z; dst[i4 * 4 + 3] = a.w;
    } else {
      st4(dst + i4 * 4, a);
    }
  }
}

static void launch_reduce_splits(const float* part, float* dw, int64_t n, const float* part_b, float* db, int64_t nb, int S, cudaStream_t st) {
  const int nblk_w = (int)rbm_cdiv(n, 128), nblk_b = part_b ? (int)rbm_cdiv(nb, 128) : 0;
  reduce_splits_kernel<<<nblk_w + nblk_b, 256, 0, st>>>(part, dw, n, nblk_w, part_b, db, nb, S);
}

__global__ void __launch_bounds__(256) epilogue_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ pre,
                                                           float* __restrict__ dpre, float* __restrict__ dres,
                                                           int64_t total4, int N4, int act, const int64_t* __restrict__ row_tok,
                                                           uint32_t thrA, float invA, uint64_t siteA, uint32_t thrB,
                                                           float invB, uint64_t siteB, uint64_t seed) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  float4 g = ld4(dout + i * 4);
  if (row_tok && row_tok[i / N4] == 0) g = make_float4(0.f, 0.f, 0.f, 0.f);
  if (thrB) {
    float4 m = rbm_drop4(seed, rbm_site(siteB), (uint64_t)i, thrB, invB);
    g.x *= m.x; g.y *= m.y; g.z *= m.z; g.w *= m.w;
  }
  if (dres) st4(dres + i * 4, g);
  if (thrA) {
    float4 m = rbm_drop4(seed, rbm_site(siteA), (uint64_t)i, thrA, invA);
    g.x *= m.x; g.y *= m.y; g.z *= m.z; g.w *= m.w;
  }
  if (act == RBM_ACT_RELU) {
    float4 u = ld4(pre + i * 4);
    g.x = u.x > 0.f ? g.x : 0.f; g.y = u.y > 0.f ? g.y : 0.f; g.z = u.z > 0.f ? g.z : 0.f; g.w = u.w > 0.f ? g.w : 0.f;
  } else if (act == RBM_ACT_GELU_TANH) {
    float4 u = ld4(pre + i * 4);
    g.x *= gelu_tanh_grad_f(u.x); g.y *= gelu_tanh_grad_f(u.y); g.z *= gelu_tanh_grad_f(u.z); g.w *= gelu_tanh_grad_f(u.w);
  }
  st4(dpre + i * 4, g);
}

__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, int rows, int cols) {
  __shared__ float tile[32][33];
  int c = blockIdx.x * 32 + threadIdx.x, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8)
    if (r0 + i < rows && c < cols) tile[i][threadIdx.x] = src[(int64_t)(r0 + i) * cols + c];
  __syncthreads();
  int r = r0 + threadIdx.x, c0 = blockIdx.x * 32;
  for (int i = threadIdx.y; i < 32; i += 8)
    if (c0 + i < cols && r < rows) dst[(int64_t)(c0 + i) * rows + r] = tile[threadIdx.x][i];
}

// column sums of dpre (bias gradient) for the tcgen05 dW path: block b sums rows [b*rpb, ...) -> part_b[b][N]
__global__ void __launch_bounds__(256) colsum_split_kernel(const float* __restrict__ a, int64_t lda, float* __restrict__ part_b, int64_t M, int N,
                                                           int64_t rows_per_block) {
  __shared__ float4 red[256];
  const int n4 = N >> 2;                 // <= 64 float4 columns
  const int groups = 256 / n4;           // row groups working in parallel
  const int c4 = threadIdx.x % n4, rg = threadIdx.x / n4;
  int64_t r0 = (int64_t)blockIdx.x * rows_per_block, r1 = r0 + rows_per_block < M ? r0 + rows_per_block : M;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (rg < groups)
    for (int64_t r = r0 + rg; r < r1; r += groups) {
      float4 v = ld4(a + r * lda + c4 * 4);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  red[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x < n4) {
    float4 t = red[threadIdx.x];
    for (int gq = 1; gq < groups; ++gq) {
      float4 v = red[gq * n4 + threadIdx.x];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    st4(part_b + (int64_t)blockIdx.x * N + threadIdx.x * 4, t);
  }
}

int tn_splits(int64_t M, int N, int K) {
  int64_t tiles = rbm_cdiv(N, 64) * rbm_cdiv(K, 64);
  int64_t want = rbm_cdiv((int64_t)RBM_NUM_SMS * 4, tiles);
  int64_t max_by_rows = rbm_cdiv(M, 256);
  int64_t s = want < max_by_rows ? want : max_by_rows;
  return (int)(s < 1 ? 1 : s);
}

}  // namespace

// wide layers with enough rows to fill the machine go to the split-fp16 tiled kernel (tc_gemm16.cu); N = output columns, K = contraction
// length.  Measured at M = 102400 / 204800: 1.5x .. 2.5x the 3xTF32 kernel from K = 256 up, slower at K = 128
// (two MMA k-blocks per unit cannot cover the epilogue)
static bool gemm16_wanted(int64_t M, int N, int K) { return M >= 512 && N >= 128 && K >= 256; }

extern "C" size_t rbm_linear_fwd_ws_bytes(int64_t M, int N, int K) {
  return gemm16_wanted(M, N, K) && N % 128 == 0 && K % 64 == 0 ? rbm_gemm16_ws_bytes(N, K) : 0;
}

extern "C" int rbm_linear_fwd(const float* x, int64_t ldx, const float* w, const float* bias, float* y, int64_t ldy,
                              float* pre, int64_t M, int N, int K, int act, const float* residual, int64_t ldres,
                              const int64_t* row_tok, float pA, uint64_t siteA, float pB, uint64_t siteB, uint64_t seed,
                              rbm_stream_t stream) {
  return rbm_linear_fwd_ws(x, ldx, w, bias, y, ldy, pre, M, N, K, act, residual, ldres, row_tok, pA, siteA, pB, siteB, seed, nullptr, 0,
                           stream);
}

extern "C" int rbm_linear_fwd_ws(const float* x, int64_t ldx, const float* w, const float* bias, float* y, int64_t ldy,
                                 float* pre, int64_t M, int N, int K, int act, const float* residual, int64_t ldres,
                                 const int64_t* row_tok, float pA, uint64_t siteA, float pB, uint64_t siteB, uint64_t seed,
                                 void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(x && w && y, "rbm_linear_fwd: null pointer");
  RBM_REQUIRE(M >= 0 && N > 0 && K > 0 && N % 4 == 0 && K % 4 == 0, "rbm_linear_fwd: need N%%4==0 and K%%4==0 (N=%d K=%d)", N, K);
  RBM_REQUIRE(ldx % 4 == 0 && ldy % 4 == 0 && ldx >= K && ldy >= N, "rbm_linear_fwd: bad leading dimensions");
  RBM_REQUIRE(!residual || (ldres % 4 == 0 && ldres >= N), "rbm_linear_fwd: bad residual stride");
  RBM_REQUIRE(act >= 0 && act <= 2, "rbm_linear_fwd: bad activation %d", act);
  RBM_REQUIRE(pA >= 0.f && pA < 1.f && pB >= 0.f && pB < 1.f, "rbm_linear_fwd: dropout p out of [0,1)");
  RBM_REQUIRE(rbm_aligned16(x) && rbm_aligned16(w) && rbm_aligned16(y) && rbm_aligned16(bias) && rbm_aligned16(pre) && rbm_aligned16(residual),
              "rbm_linear_fwd: pointers must be 16B aligned");
  if (M == 0) return 0;
  if (gemm16_wanted(M, N, K) && ws && rbm_aligned16(ws) && ws_bytes >= rbm_gemm16_ws_bytes(N, K) &&
      rbm_gemm16_supported(M, N, K, ldx, x, w)) {
    RbmTcEpilogue te{y, ldy, pre, bias, residual, ldres, row_tok, act, rbm_drop_threshold(pA), rbm_drop_threshold(pB),
                     1.f / (1.f - pA), 1.f / (1.f - pB), siteA, siteB, seed};
    return rbm_gemm16_launch(x, ldx, w, M, N, K, te, ws, (cudaStream_t)stream);
  }
  if (ldy % 4 == 0 && rbm_tc_linear_supported(M, N, K, ldx, x, w)) {
    RbmTcEpilogue te{y, ldy, pre, bias, residual, ldres, row_tok, act, rbm_drop_threshold(pA), rbm_drop_threshold(pB),
                     1.f / (1.f - pA), 1.f / (1.f - pB), siteA, siteB, seed};
    return rbm_tc_linear_launch(x, ldx, w, M, N, K, te, (cudaStream_t)stream);
  }
  Epilogue ep{bias, pre, residual, ldres, row_tok, act, rbm_drop_threshold(pA), rbm_drop_threshold(pB),
              1.f / (1.f - pA), 1.f / (1.f - pB), siteA, siteB, seed};
  dim3 grid((unsigned)rbm_cdiv(M, 128), (unsigned)rbm_cdiv(N, 64));
  gemm_rowmajor_kernel<true, true><<<grid, 256, 0, (cudaStream_t)stream>>>(x, ldx, w, K, y, ldy, M, N, K, ep);
  RBM_LAUNCH_CHECK("rbm_linear_fwd");
  return 0;
}

extern "C" int rbm_linear_epilogue_bwd(const float* dout, const float* pre, float* dpre, float* dres, int64_t M, int N,
                                       int act, const int64_t* row_tok, float pA, uint64_t siteA, float pB,
                                       uint64_t siteB, uint64_t seed, rbm_stream_t stream) {
  RBM_REQUIRE(dout && dpre, "rbm_linear_epilogue_bwd: null pointer");
  RBM_REQUIRE(N > 0 && N % 4 == 0, "rbm_linear_epilogue_bwd: N=%d must be a multiple of 4", N);
  RBM_REQUIRE(act == RBM_ACT_NONE || pre, "rbm_linear_epilogue_bwd: activation needs the saved pre-activation");
  RBM_REQUIRE(pA >= 0.f && pA < 1.f && pB >= 0.f && pB < 1.f, "rbm_linear_epilogue_bwd: dropout p out of [0,1)");
  RBM_REQUIRE(rbm_aligned16(dout) && rbm_aligned16(pre) && rbm_aligned16(dpre) && rbm_aligned16(dres), "rbm_linear_epilogue_bwd: pointers must be 16B aligned");
  if (M == 0) return 0;
  int64_t total4 = M * (N / 4);
  epilogue_bwd_kernel<<<(unsigned)rbm_cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(
      dout, pre, dpre, dres, total4, N / 4, act, row_tok, rbm_drop_threshold(pA), 1.f / (1.f - pA), siteA,
      rbm_drop_threshold(pB), 1.f / (1.f - pB), siteB, seed);
  RBM_LAUNCH_CHECK("rbm_linear_epilogue_bwd");
  return 0;
}

// transposed weight (fp32) | its fp16 hi / lo copies + scales for the split-fp16 kernel
extern "C" size_t rbm_linear_bwd_data_ws_bytes(int N, int K) { return (size_t)N * K * sizeof(float) + 256 + rbm_gemm16_ws_bytes(K, N); }

extern "C" int rbm_linear_bwd_data(const float* dpre, int64_t lddpre, const float* w, float* dx, int64_t lddx, int64_t M,
                                   int N, int K, void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(dpre && w && dx, "rbm_linear_bwd_data: null pointer");
  RBM_REQUIRE(N > 0 && K > 0 && N % 4 == 0 && K % 4 == 0, "rbm_linear_bwd_data: need N%%4==0 and K%%4==0");
  RBM_REQUIRE(lddpre % 4 == 0 && lddx % 4 == 0 && lddpre >= N && lddx >= K, "rbm_linear_bwd_data: bad leading dimensions");
  RBM_REQUIRE(rbm_aligned16(dpre) && rbm_aligned16(w) && rbm_aligned16(dx), "rbm_linear_bwd_data: pointers must be 16B aligned");
  if (M == 0) return 0;
  // dx = dpre . w  ==  dpre[M,N] . (w^T)[K,N]^T : the tcgen05 kernel wants both operands contraction-major, so the
  // (small) weight is transposed into the workspace first
  if (ws && ws_bytes >= rbm_linear_bwd_data_ws_bytes(N, K) && rbm_aligned16(ws) &&
      rbm_tc_linear_supported(M, K, N, lddpre, dpre, ws)) {
    float* wt = (float*)ws;
    dim3 tg((unsigned)rbm_cdiv(K, 32), (unsigned)rbm_cdiv(N, 32)), tb(32, 8);
    transpose_kernel<<<tg, tb, 0, (cudaStream_t)stream>>>(w, wt, N, K);
    RBM_LAUNCH_CHECK("rbm_linear_bwd_data(transpose)");
    RbmTcEpilogue te{};
    te.y = dx;
    te.ldy = lddx;
    te.invA = te.invB = 1.f;
    if (gemm16_wanted(M, K, N) && rbm_gemm16_supported(M, K, N, lddpre, dpre, wt))
      return rbm_gemm16_launch(dpre, lddpre, wt, M, K, N, te, (uint8_t*)ws + (size_t)N * K * sizeof(float) + 256, (cudaStream_t)stream);
    return rbm_tc_linear_launch(dpre, lddpre, wt, M, K, N, te, (cudaStream_t)stream);
  }
  Epilogue ep{};
  dim3 grid((unsigned)rbm_cdiv(M, 128), (unsigned)rbm_cdiv(K, 64));
  // C[M,K] = dpre[M,N] . w[N,K]  -> reduction length N, B = w as [Kred=N, Nout=K]
  gemm_rowmajor_kernel<false, false><<<grid, 256, 0, (cudaStream_t)stream>>>(dpre, lddpre, w, K, dx, lddx, M, K, N, ep);
  RBM_LAUNCH_CHECK("rbm_linear_bwd_data");
  return 0;
}

extern "C" size_t rbm_linear_bwd_weight_ws_bytes(int64_t M, int N, int K) {
  int S = tn_splits(M, N, K);
  int S2 = rbm_tc_dw_splits(M);
  if (S2 > S) S = S2;
  if (N % 128 == 0 && K % 128 == 0) {
    int S3 = rbm_dw16_splits(M, N, K);
    if (S3 > S) S = S3;
  }
  return (size_t)S * ((size_t)N * K + N) * sizeof(float) + rbm_dw16_extra_bytes();
}

extern "C" int rbm_linear_bwd_weight(const float* dpre, int64_t lddpre, const float* x, int64_t ldx, float* dw, float* db,
                                     int64_t M, int N, int K, void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(dpre && x && dw && ws, "rbm_linear_bwd_weight: null pointer");
  RBM_REQUIRE(M > 0 && N > 0 && K > 0 && N % 4 == 0 && K % 4 == 0, "rbm_linear_bwd_weight: need M>0, N%%4==0, K%%4==0");
  RBM_REQUIRE(lddpre % 4 == 0 && ldx % 4 == 0 && lddpre >= N && ldx >= K, "rbm_linear_bwd_weight: bad leading dimensions");
  RBM_REQUIRE(ws_bytes >= rbm_linear_bwd_weight_ws_bytes(M, N, K), "rbm_linear_bwd_weight: workspace too small");
  RBM_REQUIRE(rbm_aligned16(dpre) && rbm_aligned16(x) && rbm_aligned16(dw) && rbm_aligned16(ws), "rbm_linear_bwd_weight: pointers must be 16B aligned");
  if (rbm_dw16_supported(M, N, K, lddpre, ldx, dpre, x)) {  // wide layers: split-fp16 tcgen05 kernel (tc_dw16.cu)
    const int S = rbm_dw16_splits(M, N, K);
    float* part = (float*)ws;
    float* part_b = part + (size_t)S * N * K;
    void* aux = (uint8_t*)ws + rbm_linear_bwd_weight_ws_bytes(M, N, K) - rbm_dw16_extra_bytes();
    int rc = rbm_dw16_launch(dpre, lddpre, x, ldx, part, db ? part_b : nullptr, aux, M, N, K, (cudaStream_t)stream);  // db rides along
    if (rc) return rc;
    launch_reduce_splits(part, dw, (int64_t)N * K, db ? part_b : nullptr, db, N, S, (cudaStream_t)stream);
    RBM_LAUNCH_CHECK("rbm_linear_bwd_weight(reduce)");
    return 0;
  }
  if (rbm_tc_dw_supported(M, N, K, lddpre, ldx, dpre, x)) {
    const int S = rbm_tc_dw_splits(M);
    float* part = (float*)ws;
    float* part_b = part + (size_t)S * N * K;
    const bool fused_b = db && rbm_tc_dw_bias_fused(N, K);
    int rc = rbm_tc_dw_launch(dpre, lddpre, x, ldx, part, fused_b ? part_b : nullptr, M, N, K, (cudaStream_t)stream);
    if (rc) return rc;
    if (db && !fused_b) {
      int64_t rpb = rbm_cdiv(M, S);
      colsum_split_kernel<<<S, 256, 0, (cudaStream_t)stream>>>(dpre, lddpre, part_b, M, N, rpb);
      RBM_LAUNCH_CHECK("rbm_linear_bwd_weight(bias)");
    }
    launch_reduce_splits(part, dw, (int64_t)N * K, db ? part_b : nullptr, db, N, S, (cudaStream_t)stream);
    RBM_LAUNCH_CHECK("rbm_linear_bwd_weight(reduce)");
    return 0;
  }
  int S = tn_splits(M, N, K);
  int64_t rps = rbm_cdiv(rbm_cdiv(M, S), BK) * BK;
  float* part = (float*)ws;
  float* part_b = part + (size_t)S * N * K;
  dim3 grid((unsigned)rbm_cdiv(N, 64), (unsigned)rbm_cdiv(K, 64), S);
  gemm_tn_split_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(dpre, lddpre, x, ldx, part, db ? part_b : nullptr, M, N, K, rps);
  RBM_LAUNCH_CHECK("rbm_linear_bwd_weight");
  launch_reduce_splits(part, dw, (int64_t)N * K, db ? part_b : nullptr, db, N, S, (cudaStream_t)stream);
  RBM_LAUNCH_CHECK("rbm_linear_bwd_weight(reduce)");
  return 0;
}

RBM_DEFINE_STEP_PTR_SETTER(rbm_step_ptr_set_linear)
