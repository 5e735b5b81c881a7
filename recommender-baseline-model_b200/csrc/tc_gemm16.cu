// tc_gemm16.cu -- Linear forward / backward-data for WIDE layers (N, K >= 128: d >= 128 models) on the Blackwell tensor path
// in SPLIT fp16:  y[M, N] = epilogue(x[M, K] . w[N, K]^T).  Replaces nn.Linear / Conv1d(k = 1) + bias + GELU / ReLU + dropout(s) +
// residual + pad-row zeroing (NN/models/bert_modules/utils/feed_forward.py:15-16, sublayer.py:16-18, attention/multi_head.py:
// 29-40, NN/models/sas_model/sas.py:16-20,75-79) where the 3xTF32 kernel of tc_gemm.cu -- which keeps the whole-K weight block
// resident in shared memory -- is left with 16..64-column blocks, i.e. N = 16..64 instructions at the fixed ~70-cycle cost.
//   * classic tiled GEMM: persistent CTAs walk (128-row tile, 128-column tile) units (column tiles of a row tile back to back:
//     the x tile comes out of L2 after its first reader), K in 64-wide blocks through a 2-stage ring;
//   * B (weight) blocks: TMA from the hi / lo fp16 copies a small pre-pass writes once per call (range-scaled by a power of two);
//     A (activation) blocks: TMA brings the fp32 block into a staging ring (rows past M arrive as zeros), eight converter warps
//     scale it, split it into fp16 hi / lo and write the 128-byte-swizzled K-major tiles -- loads issued from registers could not
//     keep enough bytes in flight (one block per L2 round trip: measured 9 us per 128 x 128 x 256 unit);
//   * one elected thread issues 128 x 128 x 16 kind::f16 instructions (64 cycles: the tensor floor), three passes per K step,
//     into one of two TMEM accumulators; eight epilogue warps (thread per row, two per lane) apply the epilogue of unit n while
//     the MMAs of unit n + 1 run.  The epilogue is the arithmetic of tc_gemm.cu's (same Philox element indexing: the
//     backward regenerates the masks).
#include <cuda_fp16.h>
#include "common.cuh"
#include "tc_ptx.cuh"
#include "split16.cuh"
#include "tc_gemm.cuh"
#include "tc_gemm16.cuh"

namespace {

using namespace rbm_tc;

constexpr int NSTG = 2;
constexpr uint32_t BLK16 = 128 * 128;        // [128 rows x 64 fp16] = 16 KB
constexpr uint32_t STAGE = 4 * BLK16;        // A hi | A lo | B hi | B lo
constexpr uint32_t A32 = 2 * BLK16;          // fp32 staging of one A block: two [128 rows x 32 fp32] boxes
constexpr int NCONV = 8;                      // converter warps (warps 2..9); epilogue warps 10..17
constexpr int THREADS = 32 * (2 + NCONV + 8);
constexpr uint32_t STG_BYTES = 8 * 4096;     // per epilogue warp: [32 rows x 32 fp32] transposition buffer

struct G16Params {
  const float* a;
  int64_t lda;
  const float* scales;  // [0] activation, [1] weight
  float* y;
  int64_t ldy;
  float* pre;
  const float* bias;
  const float* residual;
  int64_t ldres;
  const int64_t* row_tok;
  int64_t M;
  int N, K, act;
  uint32_t thrA, thrB;
  float invA, invB;
  uint64_t siteA, siteB, seed;
};

// shared memory: operand ring NSTG x 64 KB | fp32 A staging NSTG x 32 KB | epilogue transposition buffers 32 KB
__global__ void __launch_bounds__(THREADS, 1) gemm16_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapBh,
                                                           const __grid_constant__ CUtensorMap mapBl, const G16Params p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t fullA[NSTG], fullB[NSTG], empty_bar[NSTG], a32_full[NSTG], a32_empty[NSTG], tfull[2], tempty[2];
  __shared__ uint32_t tmem_base_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KB = p.K / 64, NCT = p.N / 128;
  const int n_units = (int)((p.M + 127) / 128) * NCT;
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sb = smem_u32(sm);
  if (threadIdx.x == 0) {
    for (int s = 0; s < NSTG; ++s) {
      mbar_init(smem_u32(&fullA[s]), NCONV);
      mbar_init(smem_u32(&fullB[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
      mbar_init(smem_u32(&a32_full[s]), 1);
      mbar_init(smem_u32(&a32_empty[s]), NCONV);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tfull[b]), 1);
      mbar_init(smem_u32(&tempty[b]), 8);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------------------ TMA: weight blocks (hi, lo)
    if (elect_one()) {
      int g = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int ct = u % NCT, rt = u / NCT;
        for (int kb = 0; kb < KB; ++kb, ++g) {
          const int s = g % NSTG;
          if (g >= NSTG) mbar_wait(smem_u32(&a32_empty[s]), ((g / NSTG) - 1) & 1);
          const uint32_t abar = smem_u32(&a32_full[s]), ast = sb + NSTG * STAGE + s * A32;
          mbar_expect_tx(abar, A32);
          tma_load_2d(ast, &mapA, abar, kb * 64, rt * 128);
          tma_load_2d(ast + BLK16, &mapA, abar, kb * 64 + 32, rt * 128);
          if (g >= NSTG) mbar_wait(smem_u32(&empty_bar[s]), ((g / NSTG) - 1) & 1);
          const uint32_t bar = smem_u32(&fullB[s]), st = sb + s * STAGE;
          mbar_expect_tx(bar, 2 * BLK16);
          tma_load_2d(st + 2 * BLK16, &mapBh, bar, kb * 64, ct * 128);
          tma_load_2d(st + 3 * BLK16, &mapBl, bar, kb * 64, ct * 128);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------- MMA issuer
    if (elect_one()) {
      const uint32_t idesc = make_idesc_f16(128, 128, 0, 0);
      int g = 0, it = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++it) {
        const int buf = it & 1;
        if (it >= 2) {
          mbar_wait(smem_u32(&tempty[buf]), ((it >> 1) - 1) & 1);
          tc_fence_after();
        }
        const uint32_t d = tmem + (uint32_t)(buf * 128);
        uint32_t acc = 0;
        for (int kb = 0; kb < KB; ++kb, ++g) {
          const int s = g % NSTG;
          mbar_wait(smem_u32(&fullA[s]), (g / NSTG) & 1);
          mbar_wait(smem_u32(&fullB[s]), (g / NSTG) & 1);
          tc_fence_after();
          const uint32_t st = sb + s * STAGE;
#pragma unroll
          for (int pass = 0; pass < 3; ++pass) {
            const uint64_t ad = make_sw128_desc(st + (pass == 2 ? BLK16 : 0)), bd = make_sw128_desc(st + 2 * BLK16 + (pass == 1 ? BLK16 : 0));
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              umma_f16(d, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc, acc);
              acc = 1;
            }
          }
          umma_commit(smem_u32(&empty_bar[s]));
        }
        umma_commit(smem_u32(&tfull[buf]));
      }
    }
    __syncwarp();
  } else if (warp < 2 + NCONV) {
    // ------------------------------------------------------------------ converters: activation rows -> fp16 hi / lo tiles
    // warp cw owns rows [16 cw, 16 cw + 16) of the staged block
    const int cw = warp - 2, rsub = lane >> 3, c = lane & 7;
    const float sA = p.scales[0];
    const int my_units = (int)blockIdx.x < n_units ? (n_units - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int total = my_units * KB;
    for (int g = 0; g < total; ++g) {
      const int s = g % NSTG;
      mbar_wait(smem_u32(&a32_full[s]), (g / NSTG) & 1);
      if (g >= NSTG) mbar_wait(smem_u32(&empty_bar[s]), ((g / NSTG) - 1) & 1);
      const uint8_t* src = sm + (size_t)NSTG * STAGE + (size_t)s * A32;
      uint8_t* st = sm + (size_t)s * STAGE;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int r = cw * 16 + i + 4 * rsub;  // rows r, r + 4, r + 8, r + 12 of one instruction: no bank conflicts either way
          const float4 v = *reinterpret_cast<const float4*>(src + j * BLK16 + r * 128 + ((c ^ (r & 7)) << 4));
          const __half2 h01 = __floats2half2_rn(v.x * sA, v.y * sA), h23 = __floats2half2_rn(v.z * sA, v.w * sA);
          const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
          const __half2 l01 = __floats2half2_rn(fmaf(v.x, sA, -f01.x), fmaf(v.y, sA, -f01.y));
          const __half2 l23 = __floats2half2_rn(fmaf(v.z, sA, -f23.x), fmaf(v.w, sA, -f23.y));
          const uint32_t off = (uint32_t)r * 128u + (uint32_t)(((4 * j + (c >> 1)) ^ (r & 7)) << 4) + (uint32_t)((c & 1) << 3);
          *reinterpret_cast<uint2*>(st + off) = make_uint2(*reinterpret_cast<const uint32_t*>(&h01), *reinterpret_cast<const uint32_t*>(&h23));
          *reinterpret_cast<uint2*>(st + BLK16 + off) = make_uint2(*reinterpret_cast<const uint32_t*>(&l01), *reinterpret_cast<const uint32_t*>(&l23));
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(smem_u32(&a32_empty[s]));
        mbar_arrive(smem_u32(&fullA[s]));
      }
    }
  } else {
    // ---------------------------------------------------------------------------------------------- epilogue
    // warp ew reads its TMEM lane quarter (thread = row), transposes 32 x 32 pieces through shared memory and applies the epilogue
    // with a row's 128 bytes on eight adjacent lanes: bias / residual / pre / y accesses are whole cache lines
    const int ew = warp - 2 - NCONV, q = warp & 3, half = ew >> 2;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    uint8_t* stg = sm + (size_t)NSTG * (STAGE + A32) + (size_t)ew * 4096;
    const float inv = 1.f / (p.scales[0] * p.scales[1]);
    const uint64_t siteA_e = rbm_site(p.siteA), siteB_e = rbm_site(p.siteB);
    const int rsub = lane >> 3, ch = lane & 7;
    int it = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++it) {
      const int buf = it & 1;
      const int64_t rbase = (int64_t)(u / NCT) * 128 + q * 32;
      const int n0 = (u % NCT) * 128 + half * 64;
      mbar_wait(smem_u32(&tfull[buf]), (it >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 32) {
        {
          float v[32];
          tmem_ld32(tmem + lane_sel + (uint32_t)(buf * 128 + half * 64 + c0), v);
          if (c0 == 32) {  // last read of this accumulator by this warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&tempty[buf]));
          }
#pragma unroll
          for (int c = 0; c < 8; ++c)
            *reinterpret_cast<float4*>(stg + lane * 128 + ((c ^ (lane & 7)) << 4)) = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
        }
        __syncwarp();
        const int col = n0 + c0 + ch * 4;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) b4 = ld4(p.bias + col);
#pragma unroll 2
        for (int i = 0; i < 8; ++i) {
          const int rl = 4 * i + rsub;
          const int64_t row = rbase + rl;
          if (row >= p.M) continue;
          const float4 a4 = *reinterpret_cast<const float4*>(stg + rl * 128 + ((ch ^ (rl & 7)) << 4));
          float4 x = make_float4(fmaf(a4.x, inv, b4.x), fmaf(a4.y, inv, b4.y), fmaf(a4.z, inv, b4.z), fmaf(a4.w, inv, b4.w));
          if (p.act != 0 || p.pre) {
            if (p.pre) st4(p.pre + row * p.N + col, x);
            if (p.act == RBM_ACT_RELU) {
              x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f);
            } else if (p.act == RBM_ACT_GELU_TANH) {
              x.x = gelu_tanh_f(x.x); x.y = gelu_tanh_f(x.y); x.z = gelu_tanh_f(x.z); x.w = gelu_tanh_f(x.w);
            }
          }
          const uint64_t e4 = (uint64_t)(row * p.N + col) >> 2;
          if (p.thrA) {
            const float4 m = rbm_drop4(p.seed, siteA_e, e4, p.thrA, p.invA);
            x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
          }
          if (p.residual) {
            const float4 r4 = ld4(p.residual + row * p.ldres + col);
            x.x += r4.x; x.y += r4.y; x.z += r4.z; x.w += r4.w;
          }
          if (p.thrB) {
            const float4 m = rbm_drop4(p.seed, siteB_e, e4, p.thrB, p.invB);
            x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
          }
          if (p.row_tok && p.row_tok[row] == 0) x = make_float4(0.f, 0.f, 0.f, 0.f);
          st4(p.y + row * p.ldy + col, x);
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 256);
  }
}

}  // namespace

bool rbm_gemm16_supported(int64_t M, int N, int K, int64_t lda, const void* a, const void* b) {
  if (M < 1 || N < 128 || K < 128 || N % 128 != 0 || K % 64 != 0) return false;
  if (lda % 4 != 0 || ((uintptr_t)a & 15) || ((uintptr_t)b & 15)) return false;
  return get_encode() != nullptr;
}

size_t rbm_gemm16_ws_bytes(int N, int K) { return (size_t)N * K * 4 + 256; }  // weight hi + lo (2 B each) + max-abs bits + scales

// y = epilogue(a[M, K] . b[N, K]^T); ws: rbm_gemm16_ws_bytes(N, K)
int rbm_gemm16_launch(const float* a, int64_t lda, const float* b, int64_t M, int N, int K, const RbmTcEpilogue& ep, void* ws, cudaStream_t st) {
  uint8_t* w8 = (uint8_t*)ws;
  void* b_hi = w8;
  void* b_lo = w8 + (size_t)N * K * 2;
  unsigned* bits = (unsigned*)(w8 + (size_t)N * K * 4);
  float* scales = (float*)(w8 + (size_t)N * K * 4 + 16);
  cudaMemsetAsync(bits, 0, 16, st);
  maxabs_launch(a, lda, M, K, bits, 8 * RBM_NUM_SMS, st);
  maxabs_launch(b, K, N, K, bits + 1, RBM_NUM_SMS, st);
  scales_launch(bits, scales, st);
  split_w_launch(b, scales + 1, (uint2*)b_hi, (uint2*)b_lo, (int64_t)N * K / 4, st);
  CUtensorMap mA, mBh, mBl;
  if (!encode_f16_rows(&mBh, b_hi, N, K, 128) || !encode_f16_rows(&mBl, b_lo, N, K, 128) || !encode_f32_rows(&mA, a, M, K, lda, 128, false)) {
    rbm_set_error("rbm_linear(gemm16): cuTensorMapEncodeTiled failed");
    return -1;
  }
  G16Params p{};
  p.a = a; p.lda = lda; p.scales = scales; p.y = ep.y; p.ldy = ep.ldy; p.pre = ep.pre; p.bias = ep.bias; p.residual = ep.residual;
  p.ldres = ep.ldres; p.row_tok = ep.row_tok; p.M = M; p.N = N; p.K = K; p.act = ep.act;
  p.thrA = ep.thrA; p.thrB = ep.thrB; p.invA = ep.invA; p.invB = ep.invB; p.siteA = ep.siteA; p.siteB = ep.siteB; p.seed = ep.seed;
  const size_t smem = (size_t)NSTG * (STAGE + A32) + STG_BYTES + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    if (!set_smem(gemm16_kernel, smem, "rbm_linear(gemm16)")) return -1;
    attr_set = true;
  }
  const int64_t units = rbm_cdiv(M, 128) * (N / 128);
  const int grid = (int)(units < RBM_NUM_SMS ? units : RBM_NUM_SMS);
  gemm16_kernel<<<grid, THREADS, smem, st>>>(mA, mBh, mBl, p);
  RBM_LAUNCH_CHECK("rbm_linear(gemm16)");
  return 0;
}

RBM_DEFINE_STEP_PTR_SETTER(rbm_step_ptr_set_gemm16)
