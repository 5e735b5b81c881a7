// tc_gemm.cu -- Blackwell-native GEMM for the Linear layers:  D[M,N] = A[M,K] . B[N,K]^T  (+ fused epilogue), and the weight
// gradient dW = dpre^T . x.  Operands stay fp32 in HBM; TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) stages them into shared
// memory and tcgen05.mma consumes them as TF32 (kind::tf32, fp32 accumulation in TMEM), with the TF32 residuals of the operands
// as extra products (3xTF32) for fp32-level accuracy.  The forward kernel serves rbm_linear_fwd and rbm_linear_bwd_data (with the weight transposed by the
// caller); shapes that do not meet the TMA/UMMA constraints take the SIMT kernels of linear.cu.
#include "common.cuh"
#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace rbm_tc;

constexpr int BM = 128;      // UMMA_M (cta_group::1)
constexpr int BKE = 32;      // K elements per stage = one 128-byte swizzle row of fp32/tf32
constexpr int UMMA_K = 8;    // tf32

struct TcParams {
  float* y;
  int64_t ldy;
  const float* acc_in;  // split-K: partial sums of the earlier K chunks (same layout as y; y itself is the accumulator)
  float* pre;
  const float* bias;
  const float* residual;
  int64_t ldres;
  const int64_t* row_tok;
  int64_t M;
  int N, K, BN, nstage, act;
  int ngroups;  // persistent kernel: column groups of BN = N / ngroups output columns
  uint32_t thrA, thrB;
  float invA, invB;
  uint64_t siteA, siteB, seed;
  uint32_t tmem_cols;
};

// =====================================================================================================
// Forward: persistent, weight-resident, 3xTF32.
//   * one persistent CTA per SM walks M tiles (tile = blockIdx.x + i*gridDim.x);
//   * the whole weight B[N<=256, K] is TMA-loaded ONCE per CTA and stays in shared memory (raw + lo copy);
//   * A streams through a ring of 32-wide K-block stages; two "split" warps derive A_lo = A - trunc_tf32(A) next to
//     each raw stage, so that  D = A_raw.B_lo + A_lo.B_raw + A_raw.B_raw  (three tcgen05.mma per K step) carries
//     fp32-level accuracy while the tensor core only ever sees TF32 operands;
//   * accumulators are double-buffered in TMEM: the epilogue of tile i overlaps TMA + MMA of tile i+1;
//   * the epilogue transposes 32x32 accumulator chunks through a per-warp staging tile so that every global load
//     (residual) and store (y, pre-activation) is a fully coalesced 128-byte row segment.
// warps: 0 = TMA producer, 1 = TMEM alloc + MMA issuer, 2-3 = operand split, 4-11 = epilogue (two per TMEM quarter,
// alternating 32-column chunks).
// =====================================================================================================
constexpr int STG_LD = 32;  // staging tile: 32x32 floats per warp, 16-byte chunks XOR-swizzled by (row & 7): conflict-free both ways

constexpr int EPI_WARPS = 8;
// ACT: 0 none, 1 ReLU, 2 tanh-GELU, 3 none but the pre-activation is stored; DROPA / DROPB: the Philox dropout sites.  The
// variant is a compile-time property so that the unrolled epilogue rows are straight-line code (uniform runtime branches
// around every activation / Philox block kept the compiler from interleaving the eight independent rows).  The
// epilogue loop is fully unrolled, so leaving the unused branches out keeps its body inside the instruction cache.
template <int ACT, bool DROPA, bool DROPB>
__global__ void __launch_bounds__(128 + 32 * EPI_WARPS, 1) tc_linear_persistent_kernel(const __grid_constant__ CUtensorMap mapA,
                                                                      const __grid_constant__ CUtensorMap mapB, const TcParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[8], split_bar[8], empty_bar[8], tfull_bar[2], tempty_bar[2], bfull_bar, bsplit_bar;
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KB = p.K / BKE, BN = p.BN, ns = p.nstage;
  const int tiles = (int)((p.M + BM - 1) / BM);
  // column groups: CTA c serves the output columns [n0, n0 + BN) of the row tiles cta, cta + stride, ...; the groups walk
  // the same row tiles side by side, so every A tile after its first reader comes out of L2
  const int cta = (int)blockIdx.x / p.ngroups, stride = (int)gridDim.x / p.ngroups;
  const int n0 = ((int)blockIdx.x % p.ngroups) * BN;
  const uint32_t a_bytes = BM * BKE * 4, bk_bytes = (uint32_t)BN * BKE * 4, b_bytes = bk_bytes * KB;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen_base = smem_raw + (smem_base - smem_u32(smem_raw));  // generic pointer to the aligned base
  const uint32_t off_blo = b_bytes, off_stage = 2 * b_bytes, off_stg = off_stage + (uint32_t)ns * 2 * a_bytes;

  if (threadIdx.x == 0) {
    for (int s = 0; s < ns; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&split_bar[s]), 2);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tfull_bar[b]), 1);
      mbar_init(smem_u32(&tempty_bar[b]), EPI_WARPS);
    }
    mbar_init(smem_u32(&bfull_bar), 1);
    mbar_init(smem_u32(&bsplit_bar), 2);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_slot;

  if (warp == 0) {
    if (elect_one()) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
      const uint32_t bb = smem_u32(&bfull_bar);
      mbar_expect_tx(bb, b_bytes);
      for (int kb = 0; kb < KB; ++kb) tma_load_2d(smem_base + kb * bk_bytes, &mapB, bb, kb * BKE, n0);
      int g = 0;
      for (int tile = cta; tile < tiles; tile += stride)
        for (int kb = 0; kb < KB; ++kb, ++g) {
          const int s = g % ns;
          if (g >= ns) mbar_wait(smem_u32(&empty_bar[s]), ((g / ns) - 1) & 1);
          const uint32_t bar = smem_u32(&full_bar[s]);
          mbar_expect_tx(bar, a_bytes);
          tma_load_2d(smem_base + off_stage + s * 2 * a_bytes, &mapA, bar, kb * BKE, tile * BM);
        }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc_tf32(BM, BN, 0, 0);
      mbar_wait(smem_u32(&bsplit_bar), 0);
      tc_fence_after();
      int g = 0, it = 0;
      for (int tile = cta; tile < tiles; tile += stride, ++it) {
        const int buf = it & 1;
        if (it >= 2) {
          mbar_wait(smem_u32(&tempty_bar[buf]), ((it >> 1) - 1) & 1);
          tc_fence_after();
        }
        const uint32_t d = tmem_d + (uint32_t)(buf * BN);
        for (int kb = 0; kb < KB; ++kb, ++g) {
          const int s = g % ns;
          mbar_wait(smem_u32(&full_bar[s]), (g / ns) & 1);
          mbar_wait(smem_u32(&split_bar[s]), (g / ns) & 1);
          tc_fence_after();
          const uint32_t sa = smem_base + off_stage + s * 2 * a_bytes;
          const uint64_t a_raw = make_sw128_desc(sa), a_lo = make_sw128_desc(sa + a_bytes);
          const uint64_t b_raw = make_sw128_desc(smem_base + kb * bk_bytes), b_lo = make_sw128_desc(smem_base + off_blo + kb * bk_bytes);
#pragma unroll
          for (int k = 0; k < BKE / UMMA_K; ++k) {
            const uint64_t o = (uint64_t)(k * 2);
            umma_tf32(d, a_raw + o, b_lo + o, idesc, (kb | k) != 0);
            umma_tf32(d, a_lo + o, b_raw + o, idesc, 1);
            umma_tf32(d, a_raw + o, b_raw + o, idesc, 1);
          }
          umma_commit(smem_u32(&empty_bar[s]));
        }
        umma_commit(smem_u32(&tfull_bar[buf]));
      }
    }
    __syncwarp();
  } else if (warp < 4) {
    const int tid = threadIdx.x - 64;
    mbar_wait(smem_u32(&bfull_bar), 0);
    split_lo(reinterpret_cast<const float*>(gen_base), reinterpret_cast<float*>(gen_base + off_blo), (int)(b_bytes / 16), tid, 64);
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&bsplit_bar));
    int g = 0;
    for (int tile = cta; tile < tiles; tile += stride)
      for (int kb = 0; kb < KB; ++kb, ++g) {
        const int s = g % ns;
        mbar_wait(smem_u32(&full_bar[s]), (g / ns) & 1);
        uint8_t* st = gen_base + off_stage + (size_t)s * 2 * a_bytes;
        split_lo(reinterpret_cast<const float*>(st), reinterpret_cast<float*>(st + a_bytes), (int)(a_bytes / 16), tid, 64);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&split_bar[s]));
      }
  } else {
    const int q = warp & 3, half = (warp - 4) >> 2;
    float* stg = reinterpret_cast<float*>(gen_base + off_stg) + (warp - 4) * 32 * STG_LD;
    const int rsub = lane >> 3, cg = (lane & 7) * 4;
    const float* __restrict__ resid = p.residual;
    const float* __restrict__ biasp = p.bias;
    float* __restrict__ yout = p.y;
    float* __restrict__ preout = p.pre;
    const int last_c0 = ((BN / 32 - 1 - half) / 2) * 64 + half * 32;  // this warp's last chunk
    const uint64_t siteA_e = rbm_site(p.siteA), siteB_e = rbm_site(p.siteB);
    int it = 0;
    for (int tile = cta; tile < tiles; tile += stride, ++it) {
      const int buf = it & 1;
      mbar_wait(smem_u32(&tfull_bar[buf]), (it >> 1) & 1);
      tc_fence_after();
      const int64_t rbase = (int64_t)tile * BM + q * 32;
      if (half * 32 >= BN) {  // BN == 16/32: the second warp of the pair has no chunk, it only releases the buffer
        if (lane == 0) mbar_arrive(smem_u32(&tempty_bar[buf]));
        continue;
      }
      for (int c0 = half * 32; c0 < BN; c0 += 64) {
        float v[32];
        tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + c0), v);
        if (c0 == last_c0) {  // last read of this accumulator by this warp: hand the TMEM buffer back
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(&tempty_bar[buf]));
        }
        const int col = n0 + c0 + cg;
        const bool col_ok = c0 + cg < BN && col < p.N;  // (a 32-column chunk may reach past a BN = 16 / 48 / ... block)
        // all residual loads of the chunk are issued before anything depends on them
        float4 res[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int64_t row = rbase + i * 4 + rsub;
          res[i] = (resid && col_ok && row < p.M) ? ld4(resid + row * p.ldres + col) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        uint32_t zero_rows = 0;  // bit i: row i*4+rsub is a padding token whose output is forced to zero
        if (p.row_tok) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int64_t row = rbase + i * 4 + rsub;
            if (row < p.M && p.row_tok[row] == 0) zero_rows |= 1u << i;
          }
        }
#pragma unroll
        for (int j = 0; j < 32; j += 4) st4(stg + lane * STG_LD + (((j >> 2) ^ (lane & 7)) << 2), make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
        __syncwarp();
        if (col_ok) {
          float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (biasp) bias4 = ld4(biasp + col);
          auto row_out = [&](int i) {
            const int rl = i * 4 + rsub;
            const int64_t row = rbase + rl;
            float4 x = ld4(stg + rl * STG_LD + (((cg >> 2) ^ (rl & 7)) << 2));
            if (p.acc_in) {  // this thread reads exactly the elements it overwrites below: y may be the accumulator
              const float4 t = ld4(p.acc_in + row * p.ldy + col);
              x.x += t.x; x.y += t.y; x.z += t.z; x.w += t.w;
            }
            x.x += bias4.x; x.y += bias4.y; x.z += bias4.z; x.w += bias4.w;
            if constexpr (ACT != 0) {
              if (preout) st4(preout + row * p.N + col, x);
            }
            if constexpr (ACT == RBM_ACT_RELU) {
              x.x = fmaxf(x.x, 0.f); x.y = fmaxf(x.y, 0.f); x.z = fmaxf(x.z, 0.f); x.w = fmaxf(x.w, 0.f);
            } else if constexpr (ACT == RBM_ACT_GELU_TANH) {
              x.x = gelu_tanh_f(x.x); x.y = gelu_tanh_f(x.y); x.z = gelu_tanh_f(x.z); x.w = gelu_tanh_f(x.w);
            }
            const uint64_t e4 = (uint64_t)(row * p.N + col) >> 2;
            if constexpr (DROPA) {
              const float4 m = rbm_drop4(p.seed, siteA_e, e4, p.thrA, p.invA);
              x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
            }
            x.x += res[i].x; x.y += res[i].y; x.z += res[i].z; x.w += res[i].w;
            if constexpr (DROPB) {
              const float4 m = rbm_drop4(p.seed, siteB_e, e4, p.thrB, p.invB);
              x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
            }
            if ((zero_rows >> i) & 1u) x = make_float4(0.f, 0.f, 0.f, 0.f);
            st4(yout + row * p.ldy + col, x);
          };
          if (rbase + 32 <= p.M) {  // whole 32-row slice inside the matrix: eight independent straight-line rows
#pragma unroll
            for (int i = 0; i < 8; ++i) row_out(i);
          } else {
#pragma unroll
            for (int i = 0; i < 8; ++i)  // (unrolled too: a dynamic index would push res[] into local memory)
              if (rbase + i * 4 + rsub < p.M) row_out(i);
          }
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_d, p.tmem_cols);
  }
}

// =====================================================================================================
// Weight gradient:  dW[N, K] = dpre[M, N]^T . x[M, K]   (contraction over the M tokens)
// Both operands are token-major in HBM, i.e. MN-major for the tensor core: TMA (128-byte swizzle with 32-byte atoms,
// the only MN-major layout for 32-bit operands) stages [32 tokens x 32 columns] blocks, tcgen05.mma runs with
// a_major = b_major = MN.  Each persistent CTA owns a contiguous slab of tokens and accumulates its partial dW in
// TMEM (one or two 128-row M tiles x K columns); partials are summed in fixed order by reduce_splits (linear.cu).
// 3xTF32: split warps derive the TF32 residual of every staged block.
// warps: 0 = TMA, 1 = MMA, 2-5 = split, then all of 2-5 read the accumulators out at the end.
// =====================================================================================================
constexpr int DW_TOK = 32;                 // tokens per stage
constexpr int DW_BLK = DW_TOK * 128;       // bytes of one [32 tokens x 32 columns] block

struct DwParams {
  float* part;     // [S][N][K]
  float* part_b;   // [S][N] column sums of A (the bias gradient), or nullptr
  int64_t M, tok_per_cta;
  int N, K, nblkA, nblkB, mtiles, nstage;
  int wide;        // 1: one instruction per operand half against [B | B_lo | ones] (N = 2K + 32); 0: three products + bias pair
  uint32_t tmem_cols;
};
constexpr int DW_BIAS_N = 16;  // narrow mode: width of the all-ones B operand that turns the bias gradient into an accumulator

// A tcgen05.mma costs its issuer ~40 cycles and the pipe max(N/2, ~16) cycles, so fewer and wider instructions win.  In
// wide mode the B side of a stage is laid out as consecutive MN blocks  [x raw | x residual | all-ones]  and every 8-token
// step needs two instructions per 128-row tile:  D += A.[x | x_lo | 1]  and  D += A_lo.[x | x_lo | 1]  (the A_lo.x_lo
// product that comes along is below fp32 resolution).  dW = D[:, 0:K] + D[:, K:2K], db = D[:, 2K].
__global__ void __launch_bounds__(192, 1) tc_dw_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                                                       const DwParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[8], split_bar[8], empty_bar[8], done_bar;
  __shared__ uint32_t tmem_base_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (smem_base - smem_u32(smem_raw));
  // No padding of A up to a multiple of 128 dW rows: the last M tile's descriptor simply runs on into the blocks that
  // follow (A residual, B ...), which hold finite staged data; the accumulator rows they produce (n >= N) are never read.
  // B raw + B residual + ones are >= 3 blocks, enough for the <= 3 blocks the last residual tile overruns.
  const uint32_t a_bytes = (uint32_t)p.nblkA * DW_BLK, b_bytes = (uint32_t)p.nblkB * DW_BLK;
  // stage: A raw | A residual | B raw | B residual | all-ones block
  const uint32_t oAl = a_bytes, oB = 2 * a_bytes, oBl = 2 * a_bytes + b_bytes, oOnes = 2 * (a_bytes + b_bytes);
  const uint32_t stage_bytes = oOnes + DW_BLK;
  const int64_t t0 = (int64_t)blockIdx.x * p.tok_per_cta;
  int64_t t1 = t0 + p.tok_per_cta;
  if (t1 > p.M) t1 = p.M;
  const int nst = t1 > t0 ? (int)((t1 - t0 + DW_TOK - 1) / DW_TOK) : 0;
  const int NB = p.wide ? 2 * p.K + (p.part_b ? 32 : 0) : p.K;  // accumulator columns per M tile (narrow: + bias columns behind)
  const uint32_t bias_col = (uint32_t)(p.mtiles * p.K);         // narrow mode

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.nstage; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&split_bar[s]), 4);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    mbar_init(smem_u32(&done_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), p.tmem_cols);
  for (int s = 0; s < p.nstage; ++s) {
    uint8_t* st = gen + (size_t)s * stage_bytes;
    // the all-ones block (swizzle-invariant) turns the bias gradient db = A^T . 1 into accumulator columns
    for (int i = threadIdx.x; i < (int)(DW_BLK / 4); i += blockDim.x) reinterpret_cast<float*>(st + oOnes)[i] = 1.f;
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_d = tmem_base_slot;

  if (warp == 0) {
    if (elect_one()) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
      for (int g = 0; g < nst; ++g) {
        const int s = g % p.nstage;
        if (g >= p.nstage) mbar_wait(smem_u32(&empty_bar[s]), ((g / p.nstage) - 1) & 1);
        const uint32_t bar = smem_u32(&full_bar[s]);
        const uint32_t sa = smem_base + s * stage_bytes;
        mbar_expect_tx(bar, (uint32_t)(p.nblkA + p.nblkB) * DW_BLK);
        const int tok = (int)(t0 + (int64_t)g * DW_TOK);
        for (int j = 0; j < p.nblkA; ++j) tma_load_2d(sa + j * DW_BLK, &mapA, bar, j * 32, tok);
        for (int j = 0; j < p.nblkB; ++j) tma_load_2d(sa + oB + j * DW_BLK, &mapB, bar, j * 32, tok);
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc_tf32(BM, p.wide ? NB : p.K, 1, 1);
      const uint32_t idesc_b = make_idesc_tf32(BM, DW_BIAS_N, 1, 1);
      for (int g = 0; g < nst; ++g) {
        const int s = g % p.nstage;
        mbar_wait(smem_u32(&full_bar[s]), (g / p.nstage) & 1);
        mbar_wait(smem_u32(&split_bar[s]), (g / p.nstage) & 1);
        tc_fence_after();
        const uint32_t sa = smem_base + s * stage_bytes;
        for (int mt = 0; mt < p.mtiles; ++mt) {
#pragma unroll
          for (int k = 0; k < DW_TOK / UMMA_K; ++k) {  // 8 tokens = 1024 bytes inside every block
            const uint64_t a_raw = make_sw128_desc_mn(sa + mt * 4 * DW_BLK + k * 1024, DW_BLK);
            const uint64_t a_lo = make_sw128_desc_mn(sa + oAl + mt * 4 * DW_BLK + k * 1024, DW_BLK);
            const uint64_t b_raw = make_sw128_desc_mn(sa + oB + k * 1024, DW_BLK);  // wide: runs on into B residual and ones
            if (p.wide) {
              const uint32_t d = tmem_d + (uint32_t)(mt * NB);
              umma_tf32(d, a_raw, b_raw, idesc, (g | k) != 0);
              umma_tf32(d, a_lo, b_raw, idesc, 1);
            } else {
              const uint32_t d = tmem_d + (uint32_t)(mt * p.K);
              const uint64_t b_lo = make_sw128_desc_mn(sa + oBl + k * 1024, DW_BLK);
              umma_tf32(d, a_raw, b_lo, idesc, (g | k) != 0);
              umma_tf32(d, a_lo, b_raw, idesc, 1);
              umma_tf32(d, a_raw, b_raw, idesc, 1);
              if (p.part_b) {
                const uint64_t ones = make_sw128_desc_mn(sa + oOnes + k * 1024, DW_BLK);
                const uint32_t dbias = tmem_d + bias_col + (uint32_t)(mt * DW_BIAS_N);
                umma_tf32(dbias, a_lo, ones, idesc_b, (g | k) != 0);
                umma_tf32(dbias, a_raw, ones, idesc_b, 1);
              }
            }
          }
        }
        umma_commit(smem_u32(&empty_bar[s]));
      }
      umma_commit(smem_u32(&done_bar));
    }
    __syncwarp();
  } else {
    const int tid = threadIdx.x - 64;
    for (int g = 0; g < nst; ++g) {
      const int s = g % p.nstage;
      mbar_wait(smem_u32(&full_bar[s]), (g / p.nstage) & 1);
      uint8_t* st = gen + (size_t)s * stage_bytes;
      // residuals of the blocks TMA wrote (A valid blocks, then B)
      split_lo(reinterpret_cast<const float*>(st), reinterpret_cast<float*>(st + oAl), p.nblkA * DW_BLK / 16, tid, 128);
      split_lo(reinterpret_cast<const float*>(st + oB), reinterpret_cast<float*>(st + oBl), (int)(b_bytes / 16), tid, 128);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&split_bar[s]));
    }
    // ---- read the partial dW out: warp w owns TMEM lanes [32*(w%4), +32)
    mbar_wait(smem_u32(&done_bar), 0);
    tc_fence_after();
    const int q = warp & 3;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    float* part = p.part + (int64_t)blockIdx.x * p.N * p.K;
    for (int mt = 0; mt < p.mtiles; ++mt) {
      const int n = mt * BM + q * 32 + lane;
      const uint32_t dcol = tmem_d + lane_sel + (uint32_t)(mt * (p.wide ? NB : p.K));
      for (int c0 = 0; c0 < p.K; c0 += 32) {
        float v[32];
        if (nst > 0) {
          tmem_ld32(dcol + (uint32_t)c0, v);
          if (p.wide) {
            float v2[32];
            tmem_ld32(dcol + (uint32_t)(p.K + c0), v2);
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += v2[j];
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0.f;
        }
        if (n < p.N) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) st4(part + (int64_t)n * p.K + c0 + j, make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]));
        }
      }
      if (p.part_b) {
        float v[16];
        if (nst > 0) tmem_ld16(p.wide ? dcol + (uint32_t)(2 * p.K) : tmem_d + lane_sel + bias_col + (uint32_t)(mt * DW_BIAS_N), v);
        else v[0] = 0.f;
        if (n < p.N) p.part_b[(int64_t)blockIdx.x * p.N + n] = v[0];
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_d, p.tmem_cols);
  }
}

}  // namespace

static bool weight_fits(int N, int K, int* nstage_out) {
  if (N > 256) return false;
  const size_t b_bytes = (size_t)N * K * 4, a_stage = (size_t)2 * BM * BKE * 4, stg = (size_t)EPI_WARPS * 32 * STG_LD * 4;
  const size_t budget = (size_t)231424 - 1024;  // 227 KB per block minus static barriers and alignment slack
  if (2 * b_bytes + stg + 2 * a_stage > budget) return false;
  int ns = (int)((budget - 2 * b_bytes - stg) / a_stage);
  if (ns > 8) ns = 8;
  *nstage_out = ns;
  return ns >= 2;
}

// Column groups of the persistent kernel: the fewest equal blocks of output columns whose weight block (raw + TF32
// residual) stays resident in shared memory next to at least two A stages.  0 = no such split.
static int pick_groups(int N, int K, int* nstage_out) {
  // (measured and dropped: preferring >= 64-column blocks that leave room for the A stages of two row tiles -- N = 256, K = 64 then
  //  runs as two groups with four stages instead of one group with two -- changed nothing: 138 vs 134 us, tools/time_linear_cfg2.py)
  for (int ng = 1; ng <= 32; ++ng) {
    if (N % ng != 0 || (N / ng) % 16 != 0) continue;
    if (weight_fits(N / ng, K, nstage_out)) return ng;
  }
  return 0;
}

bool rbm_tc_linear_supported(int64_t M, int N, int K, int64_t lda, const void* a, const void* b) {
  if (M < 1 || N % 16 != 0 || K % BKE != 0 || K < BKE || N < 16) return false;
  if (lda % 4 != 0 || ((uintptr_t)a & 15) || ((uintptr_t)b & 15)) return false;
  if (get_encode() == nullptr) return false;
  int ns;
  return pick_groups(N, K, &ns) != 0;
}

static int launch_single(const float* a, int64_t lda, const float* b, int64_t ldb, int64_t M, int N, int K, const RbmTcEpilogue& ep,
                         const float* acc_in, cudaStream_t st);

// Split-K: when the whole-K weight block that fits shared memory is narrower than 64 columns (K = 1024 at d = 256: 16-column
// blocks, i.e. N = 16 instructions at the fixed ~70-cycle cost), the contraction is cut into 256-wide chunks whose weight blocks
// are >= 64 columns wide; chunk c adds its product to the partial sums of the chunks before it, with y itself as the accumulator
// (every epilogue thread reads exactly the elements it overwrites), and the last chunk applies the real epilogue.
int rbm_tc_linear_launch(const float* a, int64_t lda, const float* b, int64_t M, int N, int K, const RbmTcEpilogue& ep,
                         cudaStream_t st) {
  constexpr int KC = 256;
  if (K > KC && K % KC == 0) {
    int ns, ns2;
    const int ng = pick_groups(N, K, &ns), ng2 = pick_groups(N, KC, &ns2);
    if (ng > 0 && ng2 > 0 && N / ng < 64 && N / ng2 >= 64) {
      RbmTcEpilogue plain{};
      plain.y = ep.y;
      plain.ldy = ep.ldy;
      for (int c = 0; c < K / KC; ++c) {
        const bool last = c == K / KC - 1;
        int rc = launch_single(a + (size_t)c * KC, lda, b + (size_t)c * KC, K, M, N, KC, last ? ep : plain, c > 0 ? ep.y : nullptr, st);
        if (rc) return rc;
      }
      return 0;
    }
  }
  return launch_single(a, lda, b, K, M, N, K, ep, nullptr, st);
}

static int launch_single(const float* a, int64_t lda, const float* b, int64_t ldb, int64_t M, int N, int K, const RbmTcEpilogue& ep,
                         const float* acc_in, cudaStream_t st) {
  int ns;
  const int NG = pick_groups(N, K, &ns);
  if (NG <= 0) {
    rbm_set_error("rbm_linear(tcgen05): no resident-weight split for N=%d K=%d", N, K);
    return -1;
  }
  const int BN = N / NG;
  CUtensorMap mapA, mapB;
  if (!encode_f32_rows(&mapA, a, M, K, lda, BM, false) || !encode_f32_rows(&mapB, b, N, K, ldb, BN, false)) {
    rbm_set_error("rbm_linear(tcgen05): cuTensorMapEncodeTiled failed (M=%lld N=%d K=%d lda=%lld)", (long long)M, N, K, (long long)lda);
    return -1;
  }
  TcParams p{};
  p.y = ep.y; p.ldy = ep.ldy; p.acc_in = acc_in; p.pre = ep.pre; p.bias = ep.bias; p.residual = ep.residual; p.ldres = ep.ldres; p.row_tok = ep.row_tok;
  p.M = M; p.N = N; p.K = K; p.BN = BN; p.ngroups = NG; p.act = ep.act;
  p.thrA = ep.thrA; p.thrB = ep.thrB; p.invA = ep.invA; p.invB = ep.invB; p.siteA = ep.siteA; p.siteB = ep.siteB; p.seed = ep.seed;
  static bool attr_set = false;
  if (!attr_set) {
    // every (activation, dropout A, dropout B) variant of the persistent kernel
#define RBM_TC_ATTR(A, DA, DB) set_smem(tc_linear_persistent_kernel<A, DA, DB>, 231424, "rbm_linear(tcgen05)")
#define RBM_TC_ATTR4(A) RBM_TC_ATTR(A, false, false) && RBM_TC_ATTR(A, true, false) && RBM_TC_ATTR(A, false, true) && RBM_TC_ATTR(A, true, true)
    const bool ok = RBM_TC_ATTR4(0) && RBM_TC_ATTR4(1) && RBM_TC_ATTR4(2) && RBM_TC_ATTR4(3);
#undef RBM_TC_ATTR4
#undef RBM_TC_ATTR
    if (!ok) return -1;
    attr_set = true;
  }
  p.nstage = ns;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * BN) || cols < (uint32_t)(BN + ((BN + 31) & ~31))) cols <<= 1;  // the epilogue reads whole 32-column chunks
  p.tmem_cols = cols;
  size_t smem = (size_t)2 * BN * K * 4 + (size_t)ns * 2 * BM * BKE * 4 + (size_t)EPI_WARPS * 32 * STG_LD * 4 + 1024;
  int tiles = (int)rbm_cdiv(M, BM);
  int per_group = RBM_NUM_SMS / NG;  // CTAs per column group (one CTA per SM in total)
  if (per_group > tiles) per_group = tiles;
  int grid = per_group * NG;
  const int act = p.act != 0 ? p.act : (p.pre != nullptr ? 3 : 0);  // 3: no activation, pre-activation still stored
  const bool da = p.thrA != 0, db = p.thrB != 0;
  const int nthr = 128 + 32 * EPI_WARPS;
#define RBM_TC_GO(A, DA, DB) tc_linear_persistent_kernel<A, DA, DB><<<grid, nthr, smem, st>>>(mapA, mapB, p)
#define RBM_TC_GO4(A)                       \
  do {                                      \
    if (da && db) RBM_TC_GO(A, true, true); \
    else if (da) RBM_TC_GO(A, true, false); \
    else if (db) RBM_TC_GO(A, false, true); \
    else RBM_TC_GO(A, false, false);        \
  } while (0)
  if (act == 0) RBM_TC_GO4(0);
  else if (act == RBM_ACT_RELU) RBM_TC_GO4(1);
  else if (act == RBM_ACT_GELU_TANH) RBM_TC_GO4(2);
  else RBM_TC_GO4(3);
#undef RBM_TC_GO4
#undef RBM_TC_GO
  RBM_LAUNCH_CHECK("rbm_linear(tcgen05 persistent)");
  return 0;
}

// ------------------------------------------------------------------------------------------ weight gradient launch
namespace {
int dw_stages(int N, int K, int* mtiles_out) {
  int mtiles = (N + BM - 1) / BM;
  size_t stage = (size_t)2 * ((size_t)N / 32 + K / 32) * DW_BLK + DW_BLK;  // + the all-ones block
  int ns = (int)(((size_t)231424 - 1024) / stage);
  if (ns > 8) ns = 8;
  *mtiles_out = mtiles;
  return ns;
}
// wide mode: accumulators [x | x_lo | ones] per 128-row tile must fit the 512 TMEM columns and one instruction (N <= 256)
bool dw_wide(int N, int K, bool bias) {
  const int nb = 2 * K + (bias ? 32 : 0);
  return nb <= 256 && ((N + BM - 1) / BM) * nb <= 512;
}
}  // namespace

int rbm_tc_dw_splits(int64_t M) {
  int64_t s = rbm_cdiv(M, 4 * DW_TOK);  // at least 4 stages of work per CTA
  return (int)(s < 1 ? 1 : (s > RBM_NUM_SMS ? RBM_NUM_SMS : s));
}

// the bias gradient rides along when its accumulator columns fit in TMEM next to dW
bool rbm_tc_dw_bias_fused(int N, int K) { return dw_wide(N, K, true) || ((N + BM - 1) / BM) * (K + DW_BIAS_N) <= 512; }

bool rbm_tc_dw_supported(int64_t M, int N, int K, int64_t lda, int64_t ldb, const void* a, const void* b) {
  if (M < 1 || N % 32 != 0 || K % 32 != 0 || N > 256 || K > 256 || K < 32 || N < 32) return false;
  if (lda % 4 != 0 || ldb % 4 != 0 || ((uintptr_t)a & 15) || ((uintptr_t)b & 15)) return false;
  int mt;
  if (dw_stages(N, K, &mt) < 2 || mt * K > 512) return false;
  return get_encode() != nullptr;
}

// part: [rbm_tc_dw_splits(M)][N][K] partial sums (every slot is written)
// part_b: [rbm_tc_dw_splits(M)][N] partial column sums of dpre, or nullptr (requires rbm_tc_dw_bias_fused(N, K))
int rbm_tc_dw_launch(const float* dpre, int64_t lda, const float* x, int64_t ldb, float* part, float* part_b, int64_t M, int N, int K,
                     cudaStream_t st) {
  CUtensorMap mapA, mapB;
  if (!encode_f32_rows(&mapA, dpre, M, N, lda, DW_TOK, true) || !encode_f32_rows(&mapB, x, M, K, ldb, DW_TOK, true)) {
    rbm_set_error("rbm_linear_bwd_weight(tcgen05): cuTensorMapEncodeTiled failed");
    return -1;
  }
  DwParams p{};
  p.part = part; p.part_b = part_b; p.M = M; p.N = N; p.K = K; p.nblkA = N / 32; p.nblkB = K / 32;
  p.nstage = dw_stages(N, K, &p.mtiles);
  const int S = rbm_tc_dw_splits(M);
  p.tok_per_cta = rbm_cdiv(rbm_cdiv(M, S), DW_TOK) * DW_TOK;
  p.wide = dw_wide(N, K, part_b != nullptr) ? 1 : 0;
  const int per_tile = p.wide ? 2 * K + (part_b ? 32 : 0) : K + (part_b ? DW_BIAS_N : 0);
  uint32_t cols = 32;
  while (cols < (uint32_t)(p.mtiles * per_tile)) cols <<= 1;
  p.tmem_cols = cols;
  size_t smem = (size_t)p.nstage * (2 * ((size_t)p.nblkA + p.nblkB) + 1) * DW_BLK + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    if (!set_smem(tc_dw_kernel, 231424, "rbm_linear_bwd_weight(tcgen05)")) return -1;
    attr_set = true;
  }
  tc_dw_kernel<<<S, 192, smem, st>>>(mapA, mapB, p);
  RBM_LAUNCH_CHECK("rbm_linear_bwd_weight(tcgen05)");
  return 0;
}

RBM_DEFINE_STEP_PTR_SETTER(rbm_step_ptr_set_tc_gemm)
