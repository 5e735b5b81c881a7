// tc_dw16.cu -- weight gradient of the wide Linear layers (d >= 256):  dW[N, K] = dpre[M, N]^T . x[M, K], contraction over the
// M tokens, on the Blackwell tensor path in SPLIT fp16 (split16.cuh).  Replaces, for N > 256 or K > 256
// (shapes the TF32 kernel tc_dw_kernel cannot hold in tensor memory; they ran the fp32 SIMT kernel at 24 TFLOP/s), the
// autograd of nn.Linear's weight (NN/models/bert_modules/utils/feed_forward.py:10-11, attention/multi_head.py:18-19).
//   * both operands are token-major in HBM, i.e. MN-major for the tensor core: eight converter warps read fp32 rows
//     (512 B of dpre, 1 KB of x per token: whole cache lines), scale by the per-tensor power of two from a max-abs pre-pass,
//     split into fp16 hi/lo and write 128-byte-swizzled [64 tokens x 64 columns] blocks -- the layout an MN-major descriptor
//     reads -- into a two-stage ring;
//   * one elected thread issues tcgen05.mma kind::f16 with a_major = b_major = MN: D[128 x KT] += A[128 n x 16 tokens] .
//     B[16 tokens x KT], three passes (hi.hi + hi.lo + lo.hi), KT = 256 (N = 256 instructions run at the tensor floor);
//   * a CTA owns one [128 x KT] tile of dW and one slab of tokens; partial tiles are summed in fixed order by the caller
//     (linear.cu, launch_reduce_splits): bit-deterministic, no atomics.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "split16.cuh"
#include "tc_dw16.cuh"

namespace {

using namespace rbm_tc;

constexpr int TOKB = 64;                 // tokens per stage
constexpr uint32_t BLK = TOKB * 128;     // one [64 tokens x 64 columns] fp16 block = 8 KB
constexpr int NCONV = 8;                 // converter / epilogue warps

struct Dw16Args {
  const float *dpre, *x;
  const float* scales;  // [0] dpre, [1] x
  float* part;          // [S][N][K]
  float* part_b;        // [S][N] partial column sums of dpre (bias gradient), or nullptr
  int64_t lda, ldb, M;
  int N, K, KT, tiles_k;
};

// 8 consecutive fp32 values (two float4) x scale -> 8 fp16 hi + 8 fp16 lo (16 bytes each)
__device__ __forceinline__ void split8(const float4& a, const float4& b, float s, uint4& hi, uint4& lo) {
  const float v[8] = {a.x * s, a.y * s, a.z * s, a.w * s, b.x * s, b.y * s, b.z * s, b.w * s};
  uint32_t h[4], l[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) split2(v[2 * e], v[2 * e + 1], h[e], l[e]);
  hi = make_uint4(h[0], h[1], h[2], h[3]);
  lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// stage: A hi (2 blocks) | A lo (2 blocks) | B hi (KT/64 blocks) | B lo (KT/64 blocks)
__global__ void __launch_bounds__(32 * (NCONV + 1), 1) dw16_kernel(const Dw16Args a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[2], empty_bar[2], done_bar;
  __shared__ uint32_t tmem_base_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KT = a.KT, KBK = KT / 64;
  const int tn = blockIdx.x / a.tiles_k, tk = blockIdx.x % a.tiles_k;
  const int n0 = tn * 128, k0 = tk * KT;
  const int S = gridDim.y, sp = blockIdx.y;
  const int64_t nblk_all = (a.M + TOKB - 1) / TOKB, bps = (nblk_all + S - 1) / S;
  const int64_t blk0 = (int64_t)sp * bps;
  const int nblk = (int)(blk0 >= nblk_all ? 0 : (blk0 + bps <= nblk_all ? bps : nblk_all - blk0));
  const uint32_t a_bytes = 2 * BLK, b_bytes = (uint32_t)KBK * BLK, stage_bytes = 2 * a_bytes + 2 * b_bytes;
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sb = smem_u32(sm);
  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(smem_u32(&full_bar[s]), NCONV);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    mbar_init(smem_u32(&done_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == NCONV) tmem_alloc(smem_u32(&tmem_base_slot), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tD = tmem_base_slot;
  if (warp == NCONV) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      const uint32_t idesc = make_idesc_f16(128, KT, 1, 1);
      uint32_t acc = 0;
      for (int j = 0; j < nblk; ++j) {
        const int s = j & 1;
        mbar_wait(smem_u32(&full_bar[s]), (j >> 1) & 1);
        tc_fence_after();
        const uint32_t st = sb + s * stage_bytes, sAh = st, sAl = st + a_bytes, sBh = st + 2 * a_bytes, sBl = sBh + b_bytes;
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t pa = pass == 2 ? sAl : sAh, pb = pass == 1 ? sBl : sBh;
#pragma unroll
          for (int ks = 0; ks < TOKB / 16; ++ks) {
            umma_f16(tD, make_sw128_desc_mn16(pa + ks * 2048, BLK), make_sw128_desc_mn16(pb + ks * 2048, BLK), idesc, acc);
            acc = 1;
          }
        }
        umma_commit(smem_u32(&empty_bar[s]));
      }
      umma_commit(smem_u32(&done_bar));
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------------ converters, then the epilogue
    const int tid = threadIdx.x;  // 0 .. 255
    const float sA = a.scales[0], sB = a.scales[1];
    const bool want_b = a.part_b != nullptr && tk == 0;
    float bsum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // this thread's 8 dpre columns (chunk tid & 15) over its tokens, exact fp32
    for (int j = 0; j < nblk; ++j) {
      const int s = j & 1;
      if (j >= 2) mbar_wait(smem_u32(&empty_bar[s]), ((j >> 1) - 1) & 1);
      uint8_t* st = sm + (size_t)s * stage_bytes;
      const int64_t m0 = (blk0 + j) * TOKB;
      // A: 64 tokens x 16 chunks of 8 columns (128 columns of dpre)
      {
        float4 va[4][2];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int task = it * 256 + tid, tok = task >> 4, ch = task & 15;
          const int64_t m = m0 + tok;
          va[it][0] = va[it][1] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (m < a.M) {
            const float* p = a.dpre + m * a.lda + n0 + ch * 8;
            va[it][0] = ld4(p);
            va[it][1] = ld4(p + 4);
          }
        }
        if (want_b) {
#pragma unroll
          for (int it = 0; it < 4; ++it) {
            bsum[0] += va[it][0].x; bsum[1] += va[it][0].y; bsum[2] += va[it][0].z; bsum[3] += va[it][0].w;
            bsum[4] += va[it][1].x; bsum[5] += va[it][1].y; bsum[6] += va[it][1].z; bsum[7] += va[it][1].w;
          }
        }
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int task = it * 256 + tid, tok = task >> 4, ch = task & 15;
          uint4 hi, lo;
          split8(va[it][0], va[it][1], sA, hi, lo);
          const uint32_t off = (uint32_t)(ch >> 3) * BLK + (uint32_t)tok * 128u + (uint32_t)(((ch & 7) ^ (tok & 7)) << 4);
          *reinterpret_cast<uint4*>(st + off) = hi;
          *reinterpret_cast<uint4*>(st + a_bytes + off) = lo;
        }
      }
      // B: 64 tokens x KT/8 chunks (KT columns of x), four tasks at a time
      const int chunks = KT / 8, tasks = TOKB * chunks;  // KT = 256: 2048 tasks, 8 per thread
      for (int base = 0; base < tasks; base += 4 * 256) {
        float4 vb[4][2];
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int task = base + it * 256 + tid, tok = task / chunks, ch = task - tok * chunks;
          const int64_t m = m0 + tok;
          vb[it][0] = vb[it][1] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (task < tasks && m < a.M) {
            const float* p = a.x + m * a.ldb + k0 + ch * 8;
            vb[it][0] = ld4(p);
            vb[it][1] = ld4(p + 4);
          }
        }
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const int task = base + it * 256 + tid, tok = task / chunks, ch = task - tok * chunks;
          if (task < tasks) {
            uint4 hi, lo;
            split8(vb[it][0], vb[it][1], sB, hi, lo);
            const uint32_t off = (uint32_t)(ch >> 3) * BLK + (uint32_t)tok * 128u + (uint32_t)(((ch & 7) ^ (tok & 7)) << 4);
            *reinterpret_cast<uint4*>(st + 2 * a_bytes + off) = hi;
            *reinterpret_cast<uint4*>(st + 2 * a_bytes + b_bytes + off) = lo;
          }
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&full_bar[s]));
    }
    // epilogue: thread = dW row n0 + (32 q + lane), the two warps of a lane quarter split the KT columns
    mbar_wait(smem_u32(&done_bar), 0);
    tc_fence_after();
    if (want_b) {  // bias gradient: the 16 threads of a column chunk meet in the (now idle) first stage, fixed order
      float* red = reinterpret_cast<float*>(sm);
      named_bar_sync(1, 32 * NCONV);  // every converter is past its last stage write and every MMA has completed
#pragma unroll
      for (int e = 0; e < 8; ++e) red[tid * 8 + e] = bsum[e];
      named_bar_sync(1, 32 * NCONV);
      if (tid < 128) {
        const int ch = tid >> 3, e = tid & 7;
        float t = 0.f;
        for (int g = 0; g < 16; ++g) t += red[((g << 4) | ch) * 8 + e];
        a.part_b[(int64_t)sp * a.N + n0 + tid] = t;
      }
    }
    const int q = warp & 3, half = warp >> 2;
    const int row = n0 + q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const float mul = 1.f / (sA * sB);
    float* dst = a.part + ((int64_t)sp * a.N + row) * a.K + k0;
    for (int c0 = half * (KT / 2); c0 < (half + 1) * (KT / 2); c0 += 16) {
      float o[16];
      if (nblk > 0) {
        tmem_ld16(tD + lane_sel + (uint32_t)c0, o);
      } else {
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) o[jj] = 0.f;
      }
      if (row < a.N) {
#pragma unroll
        for (int jj = 0; jj < 16; jj += 4) st4(dst + c0 + jj, make_float4(o[jj] * mul, o[jj + 1] * mul, o[jj + 2] * mul, o[jj + 3] * mul));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == NCONV) {
    tc_fence_after();
    tmem_dealloc(tD, 256);
  }
}

int tile_k(int K) { return K % 256 == 0 ? 256 : 128; }

}  // namespace

bool rbm_dw16_supported(int64_t M, int N, int K, int64_t lda, int64_t ldb, const void* a, const void* b) {
  if (M < 1 || N % 128 != 0 || K % 128 != 0) return false;
  if (!(N > 256 || K > 256 || (N == 256 && K == 256))) return false;  // smaller layers: tc_dw_kernel (one pass over the operands)
  if (lda % 4 != 0 || ldb % 4 != 0 || ((uintptr_t)a & 15) || ((uintptr_t)b & 15)) return false;
  return true;
}

int rbm_dw16_splits(int64_t M, int N, int K) {
  const int64_t tiles = (int64_t)(N / 128) * (K / tile_k(K)), blocks = rbm_cdiv(M, TOKB);
  int64_t s = (2 * RBM_NUM_SMS) / tiles;  // about two waves of (tile, slab) units
  if (s > blocks / 4) s = blocks / 4;     // at least four stages of work per CTA
  if (s > 64) s = 64;
  return (int)(s < 1 ? 1 : s);
}

size_t rbm_dw16_extra_bytes() { return 64; }  // max-abs bits + scales, behind the partials

// part: [rbm_dw16_splits][N][K] partial sums (every slot is written); part_b: [splits][N] partial column sums of dpre or nullptr;
// aux: rbm_dw16_extra_bytes() of scratch
int rbm_dw16_launch(const float* dpre, int64_t lda, const float* x, int64_t ldb, float* part, float* part_b, void* aux, int64_t M, int N, int K,
                    cudaStream_t st) {
  unsigned* bits = (unsigned*)aux;
  float* scales = (float*)((uint8_t*)aux + 16);
  cudaMemsetAsync(aux, 0, 16, st);
  maxabs_launch(dpre, lda, M, N, bits, 2 * RBM_NUM_SMS, st);
  maxabs_launch(x, ldb, M, K, bits + 1, 2 * RBM_NUM_SMS, st);
  scales_launch(bits, scales, st);
  Dw16Args a{};
  a.dpre = dpre; a.x = x; a.scales = scales; a.part = part; a.part_b = part_b; a.lda = lda; a.ldb = ldb; a.M = M; a.N = N; a.K = K;
  a.KT = tile_k(K);
  a.tiles_k = K / a.KT;
  const size_t smem = 2 * (size_t)(4 * BLK + 2 * (a.KT / 64) * BLK) + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    if (!set_smem(dw16_kernel, 2 * (4 * BLK + 8 * BLK) + 1024, "rbm_linear_bwd_weight(dw16)")) return -1;
    attr_set = true;
  }
  dim3 grid((unsigned)((N / 128) * a.tiles_k), (unsigned)rbm_dw16_splits(M, N, K));
  dw16_kernel<<<grid, 32 * (NCONV + 1), smem, st>>>(a);
  RBM_LAUNCH_CHECK("rbm_linear_bwd_weight(dw16)");
  return 0;
}
