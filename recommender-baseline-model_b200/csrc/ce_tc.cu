// ce_tc.cu -- BERT4Rec output scoring fused with masked cross-entropy on the Blackwell tensor path (d in {32,64}).
// Logits only ever exist as [128 x 64] tiles in tensor memory.  3xTF32 everywhere (fp32-level accuracy): the weight and
// the compacted hidden rows are pre-split once per call into (raw, TF32 residual) pairs in global memory so TMA streams
// both copies; per-CTA resident operands (hidden rows / weight rows) sit in TMEM as A operands with their residuals.
//   ce_fwd_tc     rows = 128 masked positions; vocab streams in 64-row K-major chunks; S = H.W^T into double-buffered
//                 TMEM; 8 softmax warps (thread per row) keep an online (max, sum-exp) in the log2 domain + target logit.
//   ce_bwd_dh_tc  same streaming; G = (softmax - onehot)*g and its residual overwrite S in TMEM and feed
//                 dH += G.W[chunk]  (A from TMEM, W chunk MN-major).
//   ce_bwd_dw_tc  rows = 128 vocab entries (W rows in TMEM); compacted hidden rows stream in 64-row chunks (K-major for
//                 S^T = W.H^T, MN-major for dW += G^T.H); db = row sums of G^T; row chunks split over blockIdx.y with
//                 a fixed-order reduction.
#include "common.cuh"
#include "mma_tiles.cuh"  // ex2, RBM_LOG2E, RBM_LN2
#include "tc_ptx.cuh"
#include "ce_tc.cuh"

namespace {

using namespace rbm_tc;
using rbm_mma::ex2;

constexpr int NSW = 8;
constexpr int CW = 64;                 // streamed rows (vocab or masked rows) per chunk
constexpr uint32_t BLK = CW * 128;     // one [64 x 32] fp32 block = 8 KB

struct CeTcArgs {
  const float* h;        // [n, d] hidden states
  const float* w;        // [V1, d]
  const int32_t* rows;   // compacted row ids
  const int64_t* tgt;
  const int32_t* count;
  const float* bias;
  const float* lse_in;
  const float* dloss;
  float *lse_out, *partial, *dh_full, *part_w, *part_b;
  int V1, d, KB, nstage;
  uint32_t tmem_cols;  // power of two >= the kernel's column need (256 lets two CTAs share an SM)
  int bias_vec;        // bias pointer is 16-byte aligned: whole-chunk float4 loads
};

// thread-owned row (d floats, global) -> TMEM raw / lo regions, scaled
__device__ __forceinline__ void row_to_tmem(const float* __restrict__ src, bool valid, float mul, int d, uint32_t t_raw, uint32_t t_lo) {
  for (int c0 = 0; c0 < d; c0 += 16) {
    float v[16], lo[16];
#pragma unroll
    for (int c = 0; c < 16; c += 4) {
      float4 x = valid ? ld4(src + c0 + c) : make_float4(0.f, 0.f, 0.f, 0.f);
      v[c] = x.x * mul; v[c + 1] = x.y * mul; v[c + 2] = x.z * mul; v[c + 3] = x.w * mul;
    }
#pragma unroll
    for (int c = 0; c < 16; ++c) lo[c] = tf32_lo(v[c]);
    tmem_st16(t_raw + c0, v);
    tmem_st16(t_lo + c0, lo);
  }
  tmem_st_wait();
}

// 3xTF32: D[tmem] (+)= A[tmem raw/lo, KB*32 columns] . B[chunk K-major raw/lo]^T
__device__ __forceinline__ void mma_scores(uint32_t d_t, uint32_t a_raw, uint32_t a_lo, uint32_t b_raw, uint32_t b_lo, int KB, uint32_t idesc) {
  for (int kb = 0; kb < KB; ++kb) {
    const uint64_t br = make_sw128_desc(b_raw + kb * BLK), bl = make_sw128_desc(b_lo + kb * BLK);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint64_t o = (uint64_t)(k * 2);
      const uint32_t ac = (uint32_t)(kb * 32 + k * 8);
      umma_tf32_ts(d_t, a_raw + ac, bl + o, idesc, (kb | k) != 0);
      umma_tf32_ts(d_t, a_lo + ac, br + o, idesc, 1);
      umma_tf32_ts(d_t, a_raw + ac, br + o, idesc, 1);
    }
  }
}
// --------------------------------------------------------------------------------------------------- forward
// TMEM: H raw [0,d) | H lo [d,2d) | S buffers [2d, 2d+128)
__global__ void __launch_bounds__(64 + 32 * NSW, 1) ce_fwd_tc_kernel(const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapWl,
                                                                     const CeTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[8], empty_bar[8], tfull[2], tempty[2], h_bar;
  __shared__ uint32_t tmem_base_slot;
  __shared__ float xm[2][128], xl[2][128], xt[2][128];
  __shared__ float contrib[128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int count = *a.count;
  const int r0 = blockIdx.x * 128;
  if (r0 >= count) {
    if (threadIdx.x == 0) a.partial[blockIdx.x] = 0.f;
    return;
  }
  const int d = a.d, KB = a.KB, ns = a.nstage, V1 = a.V1;
  const int NC = (V1 + CW - 1) / CW;
  const uint32_t stage_bytes = 2 * KB * BLK;  // raw blocks then lo blocks
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (threadIdx.x == 0) {
    for (int s = 0; s < ns; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&tfull[i]), 1);
      mbar_init(smem_u32(&tempty[i]), NSW);
    }
    mbar_init(smem_u32(&h_bar), NSW);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), a.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tH = tmem, tHl = tmem + d, tS = tmem + 2 * d;

  if (warp == 0) {
    if (elect_one()) {
      for (int c = 0; c < NC; ++c) {
        const int s = c % ns;
        if (c >= ns) mbar_wait(smem_u32(&empty_bar[s]), ((c / ns) - 1) & 1);
        const uint32_t bar = smem_u32(&full_bar[s]), sa = smem_base + s * stage_bytes;
        mbar_expect_tx(bar, stage_bytes);
        for (int kb = 0; kb < KB; ++kb) {
          tma_load_2d(sa + kb * BLK, &mapW, bar, kb * 32, c * CW);
          tma_load_2d(sa + (KB + kb) * BLK, &mapWl, bar, kb * 32, c * CW);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idS = make_idesc_tf32(128, CW, 0, 0);
      mbar_wait(smem_u32(&h_bar), 0);
      tc_fence_after();
      for (int c = 0; c < NC; ++c) {
        const int s = c % ns, buf = c & 1;
        if (c >= 2) {
          mbar_wait(smem_u32(&tempty[buf]), ((c >> 1) - 1) & 1);
          tc_fence_after();
        }
        mbar_wait(smem_u32(&full_bar[s]), (c / ns) & 1);
        tc_fence_after();
        const uint32_t sa = smem_base + s * stage_bytes;
        mma_scores(tS + buf * CW, tH, tHl, sa, sa + KB * BLK, KB, idS);
        umma_commit(smem_u32(&empty_bar[s]));
        umma_commit(smem_u32(&tfull[buf]));
      }
    }
    __syncwarp();
  } else {
    const int sw = warp - 2, q = warp & 3, half = sw >> 2;
    const int rl = q * 32 + lane, r = r0 + rl;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const bool valid = r < count;
    if (half == 0) row_to_tmem(a.h + (int64_t)(valid ? a.rows[r] : 0) * d, valid, RBM_LOG2E, d, tH + lane_sel, tHl + lane_sel);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(smem_u32(&h_bar));
    int64_t tg = valid ? a.tgt[r] : -1;
    if (tg < 0 || tg >= V1) tg = -1;  // a target outside this (shard of the) vocabulary matches no column
    float m = -INFINITY, l = 0.f, tl = 0.f;
    for (int c = 0; c < NC; ++c) {
      const int buf = c & 1;
      const int v0 = c * CW + half * 32;
      // bias of this warp's 32 columns in the log2 domain, -inf beyond the vocabulary; fetched ahead of the wait
      float bb[32];
      if (v0 + 32 <= V1 && (a.bias == nullptr || a.bias_vec)) {
        if (a.bias) {
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const float4 t = ld4(a.bias + v0 + j);
            bb[j] = t.x * RBM_LOG2E; bb[j + 1] = t.y * RBM_LOG2E; bb[j + 2] = t.z * RBM_LOG2E; bb[j + 3] = t.w * RBM_LOG2E;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) bb[j] = 0.f;
        }
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) bb[j] = v0 + j < V1 ? (a.bias ? a.bias[v0 + j] * RBM_LOG2E : 0.f) : -INFINITY;
      }
      mbar_wait(smem_u32(&tfull[buf]), (c >> 1) & 1);
      tc_fence_after();
      float v[32];
      tmem_ld32(tS + lane_sel + (uint32_t)(buf * CW + half * 32), v);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&tempty[buf]));
      float cm = -INFINITY;
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        v[j] += bb[j];
        cm = fmaxf(cm, v[j]);
      }
      const uint32_t ts = (uint32_t)(tg - (int64_t)v0);  // this row's target column inside the slice, if < 32
      if (__any_sync(0xffffffffu, ts < 32u)) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (ts == (uint32_t)j) tl = v[j];
      }
      const float mn = fmaxf(m, cm);
      if (mn > -INFINITY) {
        float ps = 0.f;
#pragma unroll
        for (int j = 0; j < 32; ++j) ps += ex2(v[j] - mn);
        l = l * (m == -INFINITY ? 0.f : ex2(m - mn)) + ps;
        m = mn;
      }
    }
    xm[half][rl] = m; xl[half][rl] = l; xt[half][rl] = tl;
    named_bar_sync(2 + q, 64);
    if (half == 0) {
      const float m0 = xm[0][rl], m1 = xm[1][rl];
      const float mm = fmaxf(m0, m1);
      const float ll = xl[0][rl] * (m0 == -INFINITY ? 0.f : ex2(m0 - mm)) + xl[1][rl] * (m1 == -INFINITY ? 0.f : ex2(m1 - mm));
      const float lse = (mm + log2f(ll)) * RBM_LN2;
      const float tsum = (xt[0][rl] + xt[1][rl]) * RBM_LN2;
      if (valid) a.lse_out[r] = lse;
      contrib[rl] = valid ? lse - tsum : 0.f;
    }
    named_bar_sync(1, NSW * 32);
    if (warp == 2 && lane == 0) {
      float sacc = 0.f;
      for (int i = 0; i < 128; ++i) sacc += contrib[i];
      a.partial[blockIdx.x] = sacc;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, a.tmem_cols);
  }
}

// ------------------------------------------------------------------------------------------------ backward
// Both backward kernels keep 128 "resident" rows as TMEM A operands (masked hidden rows for dH, weight rows for dW/db)
// and stream the other side in 64-row chunks, each chunk as K-major tiles (scores) and MN-major tiles (update).  Two
// groups of four warps (one warp per TMEM lane quarter, one thread per resident row) take the chunks alternately, each
// with its own S/G column block, so the tensor core works on one group's chunk while the other group turns scores into
// G = (softmax - onehot) * dloss/count.  The update runs as  D[:, 0:2d] += G.[B | B_lo]  (one N = 2d instruction: raw
// and residual MN-major blocks are adjacent in the stage)  and  D[:, 0:d] += G_lo.B;  the halves are added on the way out.
//   TMEM: R raw [0,d) | R lo [d,2d) | group g at 2d + 128g: S/G raw [+0,64) G lo [+64,128) | D [2d+256, 4d+256)   (d <= 64)
//   stage: chunk K-major raw | lo | MN-major raw | lo   (KB blocks each)
__device__ __forceinline__ void mma_accum2(uint32_t d_t, uint32_t g_raw, uint32_t g_lo, uint32_t b_mn_raw, uint32_t id2, uint32_t id1, bool first) {
#pragma unroll
  for (int kk = 0; kk < CW / 8; ++kk) {
    const uint64_t b2 = make_sw128_desc_mn(b_mn_raw + kk * 1024, BLK);  // 2*KB blocks: raw then residual
    umma_tf32_ts(d_t, g_raw + kk * 8, b2, id2, !(first && kk == 0));
    umma_tf32_ts(d_t, g_lo + kk * 8, b2, id1, 1);                      // first KB blocks only (N = d)
  }
}

__global__ void __launch_bounds__(64 + 32 * NSW, 1) ce_bwd_dh_tc_kernel(const __grid_constant__ CUtensorMap mapW, const __grid_constant__ CUtensorMap mapWl,
                                                                        const __grid_constant__ CUtensorMap mapWm,
                                                                        const __grid_constant__ CUtensorMap mapWml, const CeTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[4], empty_bar[4], s_full[2], g_full[2], h_bar, done_bar;
  __shared__ uint32_t tmem_base_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int count = *a.count;
  const int r0 = blockIdx.x * 128;
  if (r0 >= count) return;
  const int d = a.d, KB = a.KB, ns = a.nstage, V1 = a.V1;
  const int NC = (V1 + CW - 1) / CW;
  const uint32_t stage_bytes = 4 * KB * BLK;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (threadIdx.x == 0) {
    for (int s = 0; s < ns; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&g_full[i]), NSW / 2);
    }
    mbar_init(smem_u32(&h_bar), NSW / 2);
    mbar_init(smem_u32(&done_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tH = tmem, tHl = tmem + d, tG0 = tmem + 2 * d, tD = tG0 + 4 * CW;

  if (warp == 0) {
    if (elect_one()) {
      for (int c = 0; c < NC; ++c) {
        const int s = c % ns;
        if (c >= ns) mbar_wait(smem_u32(&empty_bar[s]), ((c / ns) - 1) & 1);
        const uint32_t bar = smem_u32(&full_bar[s]), sa = smem_base + s * stage_bytes;
        mbar_expect_tx(bar, stage_bytes);
        for (int kb = 0; kb < KB; ++kb) {
          tma_load_2d(sa + kb * BLK, &mapW, bar, kb * 32, c * CW);
          tma_load_2d(sa + (KB + kb) * BLK, &mapWl, bar, kb * 32, c * CW);
          tma_load_2d(sa + (2 * KB + kb) * BLK, &mapWm, bar, kb * 32, c * CW);
          tma_load_2d(sa + (3 * KB + kb) * BLK, &mapWml, bar, kb * 32, c * CW);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idS = make_idesc_tf32(128, CW, 0, 0), id2 = make_idesc_tf32(128, 2 * d, 0, 1), id1 = make_idesc_tf32(128, d, 0, 1);
      mbar_wait(smem_u32(&h_bar), 0);
      tc_fence_after();
      int pend[2] = {-1, -1};
      auto accum = [&](int grp) {
        const int c = pend[grp], s = c % ns;
        const uint32_t tS = tG0 + (uint32_t)grp * 2 * CW;
        mbar_wait(smem_u32(&g_full[grp]), (c >> 1) & 1);
        tc_fence_after();
        mma_accum2(tD, tS, tS + CW, smem_base + s * stage_bytes + 2 * KB * BLK, id2, id1, c == 0);
        umma_commit(smem_u32(&empty_bar[s]));
        pend[grp] = -1;
      };
      for (int c = 0; c < NC; ++c) {
        const int s = c % ns, grp = c & 1;
        if (pend[grp] >= 0) accum(grp);  // frees the group's column block (the tensor pipe runs in order)
        mbar_wait(smem_u32(&full_bar[s]), (c / ns) & 1);
        tc_fence_after();
        const uint32_t sa = smem_base + s * stage_bytes;
        mma_scores(tG0 + (uint32_t)grp * 2 * CW, tH, tHl, sa, sa + KB * BLK, KB, idS);
        umma_commit(smem_u32(&s_full[grp]));
        pend[grp] = c;
      }
      if (pend[0] >= 0 && pend[1] >= 0) {
        const int f = pend[0] < pend[1] ? 0 : 1;
        accum(f);
        accum(f ^ 1);
      } else if (pend[0] >= 0) {
        accum(0);
      } else if (pend[1] >= 0) {
        accum(1);
      }
      umma_commit(smem_u32(&done_bar));
    }
    __syncwarp();
  } else {
    const int q = warp & 3, grp = (warp - 2) >> 2;
    const int rl = q * 32 + lane, r = r0 + rl;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const bool valid = r < count;
    if (grp == 0) {
      row_to_tmem(a.h + (int64_t)(valid ? a.rows[r] : 0) * d, valid, RBM_LOG2E, d, tH + lane_sel, tHl + lane_sel);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&h_bar));
    }
    int64_t tg = valid ? a.tgt[r] : -1;
    if (tg < 0 || tg >= V1) tg = -1;  // a target outside this (shard of the) vocabulary matches no column
    const float lse2 = valid ? a.lse_in[r] * RBM_LOG2E : INFINITY;  // rows beyond the count: 2^(-inf) = 0
    const float gscale = *a.dloss / (float)count;
    const uint32_t tS = tG0 + lane_sel + (uint32_t)grp * 2 * CW, tGl = tS + CW;
    for (int c = grp; c < NC; c += 2) {
      mbar_wait(smem_u32(&s_full[grp]), (c >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int part = 0; part < CW / 16; ++part) {
        const int v0 = c * CW + part * 16;
        float bb[16];  // bias in the log2 domain minus the row's log-sum-exp; -inf beyond the vocabulary
        if (v0 + 16 <= V1 && (a.bias == nullptr || a.bias_vec)) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 t = a.bias ? ld4(a.bias + v0 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
            bb[j] = fmaf(t.x, RBM_LOG2E, -lse2); bb[j + 1] = fmaf(t.y, RBM_LOG2E, -lse2);
            bb[j + 2] = fmaf(t.z, RBM_LOG2E, -lse2); bb[j + 3] = fmaf(t.w, RBM_LOG2E, -lse2);
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) bb[j] = v0 + j < V1 ? fmaf(a.bias ? a.bias[v0 + j] : 0.f, RBM_LOG2E, -lse2) : -INFINITY;
        }
        float v[16], lo[16];
        tmem_ld16(tS + (uint32_t)(part * 16), v);
        const uint32_t ts = (uint32_t)(tg - (int64_t)v0);  // this row's target column inside the slice, if < 16
        const bool hit = __any_sync(0xffffffffu, ts < 16u);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float p = ex2(v[j] + bb[j]);
          if (hit && ts == (uint32_t)j) p -= 1.f;
          const float gg = p * gscale;
          v[j] = gg;
          lo[j] = tf32_lo(gg);
        }
        tmem_st16(tS + (uint32_t)(part * 16), v);
        tmem_st16(tGl + (uint32_t)(part * 16), lo);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&g_full[grp]));
    }
    mbar_wait(smem_u32(&done_bar), 0);
    tc_fence_after();
    // dH row = D[:, 0:d] + D[:, d:2d]; the two groups split the d columns
    const int dc = d / 2;
    for (int c0 = grp * dc; c0 < (grp + 1) * dc; c0 += 16) {
      float o[16], o2[16];
      tmem_ld16(tD + lane_sel + (uint32_t)c0, o);
      tmem_ld16(tD + lane_sel + (uint32_t)(d + c0), o2);
      if (valid) {
        float* dst = a.dh_full + (int64_t)a.rows[r] * d + c0;
#pragma unroll
        for (int j = 0; j < 16; j += 4) st4(dst + j, make_float4(o[j] + o2[j], o[j + 1] + o2[j + 1], o[j + 2] + o2[j + 2], o[j + 3] + o2[j + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// dW and db: rows = vocab entries (W rows resident), the compacted hidden rows stream; row chunks are split over
// blockIdx.y with a fixed-order reduction afterwards.
__global__ void __launch_bounds__(64 + 32 * NSW, 1) ce_bwd_dw_tc_kernel(const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapHl,
                                                                        const __grid_constant__ CUtensorMap mapHm,
                                                                        const __grid_constant__ CUtensorMap mapHml, const CeTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[4], empty_bar[4], s_full[2], g_full[2], w_bar, done_bar;
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float lse_s[2][CW], tgt_s[2][CW];  // per group: statistics of the chunk's masked rows
  __shared__ float xb[2][128];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int count = *a.count;
  const int d = a.d, KB = a.KB, ns = a.nstage, V1 = a.V1;
  const int S = gridDim.y, sp = blockIdx.y;
  const int NC = (count + CW - 1) / CW;
  const int NL = NC > sp ? (NC - sp + S - 1) / S : 0;  // chunks of this split: sp, sp + S, ...
  const int v0 = blockIdx.x * 128;
  const uint32_t stage_bytes = 4 * KB * BLK;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (threadIdx.x == 0) {
    for (int s = 0; s < ns; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&g_full[i]), NSW / 2);
    }
    mbar_init(smem_u32(&w_bar), NSW / 2);
    mbar_init(smem_u32(&done_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tW = tmem, tWl = tmem + d, tG0 = tmem + 2 * d, tD = tG0 + 4 * CW;

  if (warp == 0) {
    if (elect_one()) {
      for (int n = 0; n < NL; ++n) {
        const int c = sp + n * S, s = n % ns;
        if (n >= ns) mbar_wait(smem_u32(&empty_bar[s]), ((n / ns) - 1) & 1);
        const uint32_t bar = smem_u32(&full_bar[s]), sa = smem_base + s * stage_bytes;
        mbar_expect_tx(bar, stage_bytes);
        for (int kb = 0; kb < KB; ++kb) {
          tma_load_2d(sa + kb * BLK, &mapH, bar, kb * 32, c * CW);
          tma_load_2d(sa + (KB + kb) * BLK, &mapHl, bar, kb * 32, c * CW);
          tma_load_2d(sa + (2 * KB + kb) * BLK, &mapHm, bar, kb * 32, c * CW);
          tma_load_2d(sa + (3 * KB + kb) * BLK, &mapHml, bar, kb * 32, c * CW);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idS = make_idesc_tf32(128, CW, 0, 0), id2 = make_idesc_tf32(128, 2 * d, 0, 1), id1 = make_idesc_tf32(128, d, 0, 1);
      mbar_wait(smem_u32(&w_bar), 0);
      tc_fence_after();
      int pend[2] = {-1, -1};
      auto accum = [&](int grp) {
        const int n = pend[grp], s = n % ns;
        const uint32_t tS = tG0 + (uint32_t)grp * 2 * CW;
        mbar_wait(smem_u32(&g_full[grp]), (n >> 1) & 1);
        tc_fence_after();
        mma_accum2(tD, tS, tS + CW, smem_base + s * stage_bytes + 2 * KB * BLK, id2, id1, n == 0);
        umma_commit(smem_u32(&empty_bar[s]));
        pend[grp] = -1;
      };
      for (int n = 0; n < NL; ++n) {
        const int s = n % ns, grp = n & 1;
        if (pend[grp] >= 0) accum(grp);
        mbar_wait(smem_u32(&full_bar[s]), (n / ns) & 1);
        tc_fence_after();
        const uint32_t sa = smem_base + s * stage_bytes;
        mma_scores(tG0 + (uint32_t)grp * 2 * CW, tW, tWl, sa, sa + KB * BLK, KB, idS);
        umma_commit(smem_u32(&s_full[grp]));
        pend[grp] = n;
      }
      if (pend[0] >= 0 && pend[1] >= 0) {
        const int f = pend[0] < pend[1] ? 0 : 1;
        accum(f);
        accum(f ^ 1);
      } else if (pend[0] >= 0) {
        accum(0);
      } else if (pend[1] >= 0) {
        accum(1);
      }
      umma_commit(smem_u32(&done_bar));
    }
    __syncwarp();
  } else {
    const int q = warp & 3, grp = (warp - 2) >> 2;
    const int gt = q * 32 + lane;  // thread index inside the group (lane quarters arrive in warp order 2,3,0,1 -- any bijection works)
    const int rl = q * 32 + lane, vrow = v0 + rl;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const bool valid = vrow < V1;
    if (grp == 0) {
      row_to_tmem(a.w + (int64_t)(valid ? vrow : 0) * d, valid, RBM_LOG2E, d, tW + lane_sel, tWl + lane_sel);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&w_bar));
    }
    const float b2 = valid ? (a.bias ? a.bias[vrow] * RBM_LOG2E : 0.f) : -INFINITY;  // rows beyond the vocabulary: p = 0
    const float gscale = *a.dloss / (float)count;
    const float frow = valid ? (float)vrow : -2.f;
    const uint32_t tS = tG0 + lane_sel + (uint32_t)grp * 2 * CW, tGl = tS + CW;
    float bsum = 0.f;
    for (int n = grp; n < NL; n += 2) {
      const int c = sp + n * S;
      // statistics of the chunk's 64 masked rows (the group's previous chunk has been consumed: its g_full arrival
      // came after the last read of these arrays)
      named_bar_sync(1 + grp, 128);
      if (gt < CW) {
        const int r = c * CW + gt;
        lse_s[grp][gt] = r < count ? a.lse_in[r] * RBM_LOG2E : INFINITY;  // columns beyond the count: p = 0
        tgt_s[grp][gt] = (r < count && a.tgt[r] >= 0 && a.tgt[r] < V1) ? (float)a.tgt[r] : -1.f;
      }
      named_bar_sync(1 + grp, 128);
      mbar_wait(smem_u32(&s_full[grp]), (n >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int part = 0; part < CW / 16; ++part) {
        float v[16], lo[16], ls[16], tc[16];
#pragma unroll
        for (int j = 0; j < 16; j += 4) {
          const float4 x = ld4(&lse_s[grp][part * 16 + j]), y = ld4(&tgt_s[grp][part * 16 + j]);
          ls[j] = x.x; ls[j + 1] = x.y; ls[j + 2] = x.z; ls[j + 3] = x.w;
          tc[j] = y.x; tc[j + 1] = y.y; tc[j + 2] = y.z; tc[j + 3] = y.w;
        }
        tmem_ld16(tS + (uint32_t)(part * 16), v);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          float p = ex2(v[j] + b2 - ls[j]);
          if (tc[j] == frow) p -= 1.f;
          const float gg = p * gscale;
          bsum += gg;
          v[j] = gg;
          lo[j] = tf32_lo(gg);
        }
        tmem_st16(tS + (uint32_t)(part * 16), v);
        tmem_st16(tGl + (uint32_t)(part * 16), lo);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&g_full[grp]));
    }
    xb[grp][rl] = bsum;
    mbar_wait(smem_u32(&done_bar), 0);
    tc_fence_after();
    named_bar_sync(3, NSW * 32);
    float* pw = a.part_w + ((int64_t)sp * V1 + vrow) * d;
    const int dc = d / 2;
    for (int c0 = grp * dc; c0 < (grp + 1) * dc; c0 += 16) {
      float o[16], o2[16];
      if (NL > 0) {
        tmem_ld16(tD + lane_sel + (uint32_t)c0, o);
        tmem_ld16(tD + lane_sel + (uint32_t)(d + c0), o2);
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) o[j] = o2[j] = 0.f;
      }
      if (valid) {
#pragma unroll
        for (int j = 0; j < 16; j += 4) st4(pw + c0 + j, make_float4(o[j] + o2[j], o[j + 1] + o2[j + 1], o[j + 2] + o2[j + 2], o[j + 3] + o2[j + 3]));
      }
    }
    if (grp == 0 && valid) a.part_b[(int64_t)sp * V1 + vrow] = xb[0][rl] + xb[1][rl];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// ---------------------------------------------------------------------------------------------- helper kernels
// dst_lo = src - trunc_tf32(src)
__global__ void __launch_bounds__(256) lo_copy_kernel(const float* __restrict__ src, float* __restrict__ lo, int64_t n4) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float4 v = ld4(src + i * 4);
  st4(lo + i * 4, make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w)));
}
// Hc[r] = h[rows[r]] (r < count), zeros up to the next multiple of 128; plus its TF32 residual
__global__ void __launch_bounds__(256) gather_split_kernel(const float* __restrict__ h, const int32_t* __restrict__ rows,
                                                           const int32_t* __restrict__ count_p, float* __restrict__ hc, float* __restrict__ hcl,
                                                           int64_t cap, int d4) {
  const int count = *count_p;
  int64_t lim = ((int64_t)count + 127) / 128 * 128;
  if (lim > cap) lim = cap;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= lim * d4) return;
  int64_t r = i / d4;
  int c4 = (int)(i - r * d4);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (r < count) v = ld4(h + ((int64_t)rows[r] * d4 + c4) * 4);
  st4(hc + i * 4, v);
  st4(hcl + i * 4, make_float4(tf32_lo(v.x), tf32_lo(v.y), tf32_lo(v.z), tf32_lo(v.w)));
}

}  // namespace

bool rbm_ce_tc_supported(int V1, int d, const void* h, const void* w) {
  if ((d != 32 && d != 64) || V1 < CW) return false;  // backward: 4d + 256 TMEM columns
  if (((uintptr_t)h | (uintptr_t)w) & 15) return false;
  return get_encode() != nullptr;
}

// extra workspace (floats): W_lo [V1*d] + Hc [cap128*d] + Hc_lo [cap128*d]
size_t rbm_ce_tc_ws_floats(int64_t cap, int V1, int d) {
  int64_t cap128 = (cap + 127) / 128 * 128;
  return (size_t)V1 * d + 2 * (size_t)cap128 * d + 64;
}

int rbm_ce_tc_dw_splits(int64_t cap, int V1) {
  int64_t vt = rbm_cdiv(V1, 128), chunks = rbm_cdiv(cap, CW);
  int64_t s = (int64_t)RBM_NUM_SMS / vt;  // one wave: vt * s <= #SMs (27 vocabulary tiles x 6 splits was 162 CTAs = two waves)
  if (s > chunks) s = chunks;
  if (s > 32) s = 32;
  return (int)(s < 1 ? 1 : s);
}

int rbm_ce_tc_fwd(const float* h, const int32_t* rows, const int64_t* tgt, const int32_t* count, const float* w, const float* bias,
                  float* lse, float* partial, int64_t cap, int V1, int d, float* extra_ws, int* nblk_out, cudaStream_t st) {
  float* w_lo = extra_ws;
  const int64_t nw4 = (int64_t)V1 * d / 4;
  lo_copy_kernel<<<(unsigned)rbm_cdiv(nw4, 256), 256, 0, st>>>(w, w_lo, nw4);
  CUtensorMap mW, mWl;
  if (!encode_f32_rows(&mW, w, V1, d, d, CW, false) || !encode_f32_rows(&mWl, w_lo, V1, d, d, CW, false)) {
    rbm_set_error("rbm_ce_fwd(tcgen05): cuTensorMapEncodeTiled failed");
    return -1;
  }
  CeTcArgs a{};
  a.h = h; a.w = w; a.rows = rows; a.tgt = tgt; a.count = count; a.bias = bias; a.lse_out = lse; a.partial = partial; a.V1 = V1; a.d = d;
  a.KB = d / 32;
  const size_t stage = (size_t)2 * a.KB * BLK;
  a.tmem_cols = 2 * d + 2 * CW <= 256 ? 256 : 512;
  a.bias_vec = bias != nullptr && ((uintptr_t)bias & 15) == 0;
  // d <= 64 needs 256 TMEM columns: three 32 KB stages keep the CTA under half an SM so that two CTAs co-reside (one
  // wave for the cfg2 row count, and each CTA's waits are covered by the other)
  int ns = a.tmem_cols == 256 ? (int)((108 * 1024) / stage) : (int)((180 * 1024) / stage);
  a.nstage = ns > 8 ? 8 : ns;
  const size_t smem = (size_t)a.nstage * stage + 1024;
  if (!set_smem(ce_fwd_tc_kernel, smem, "rbm_ce_fwd(tcgen05)")) return -1;
  const int nblk = (int)rbm_cdiv(cap, 128);
  *nblk_out = nblk;
  ce_fwd_tc_kernel<<<nblk, 64 + 32 * NSW, smem, st>>>(mW, mWl, a);
  RBM_LAUNCH_CHECK("rbm_ce_fwd(tcgen05)");
  return 0;
}

int rbm_ce_tc_bwd(const float* h, const int32_t* rows, const int64_t* tgt, const int32_t* count, const float* w, const float* bias,
                  const float* lse, const float* dloss, float* dh_full, float* part_w, float* part_b, int S, int64_t cap, int V1, int d,
                  float* extra_ws, cudaStream_t st) {
  const int64_t cap128 = (cap + 127) / 128 * 128;
  float* w_lo = extra_ws;
  float* hc = w_lo + (size_t)V1 * d;
  float* hcl = hc + (size_t)cap128 * d;
  const int64_t nw4 = (int64_t)V1 * d / 4;
  lo_copy_kernel<<<(unsigned)rbm_cdiv(nw4, 256), 256, 0, st>>>(w, w_lo, nw4);
  gather_split_kernel<<<(unsigned)rbm_cdiv(cap128 * (d / 4), 256), 256, 0, st>>>(h, rows, count, hc, hcl, cap128, d / 4);
  CUtensorMap mW, mWl, mWm, mWml, mH, mHl, mHm, mHml;
  // 64-row chunks of [rows, d]: K-major maps for the score products, MN-major ones for the accumulations
  if (!encode_f32_rows(&mW, w, V1, d, d, CW, false) || !encode_f32_rows(&mWl, w_lo, V1, d, d, CW, false) ||
      !encode_f32_rows(&mWm, w, V1, d, d, CW, true) || !encode_f32_rows(&mWml, w_lo, V1, d, d, CW, true) ||
      !encode_f32_rows(&mH, hc, cap128, d, d, CW, false) || !encode_f32_rows(&mHl, hcl, cap128, d, d, CW, false) ||
      !encode_f32_rows(&mHm, hc, cap128, d, d, CW, true) || !encode_f32_rows(&mHml, hcl, cap128, d, d, CW, true)) {
    rbm_set_error("rbm_ce_bwd(tcgen05): cuTensorMapEncodeTiled failed");
    return -1;
  }
  CeTcArgs a{};
  a.h = h; a.w = w; a.rows = rows; a.tgt = tgt; a.count = count; a.bias = bias; a.lse_in = lse; a.dloss = dloss;
  a.dh_full = dh_full; a.part_w = part_w; a.part_b = part_b; a.V1 = V1; a.d = d; a.KB = d / 32;
  a.bias_vec = bias != nullptr && ((uintptr_t)bias & 15) == 0;
  const size_t stage = (size_t)4 * a.KB * BLK;
  int ns = (int)((192 * 1024) / stage);
  a.nstage = ns > 4 ? 4 : ns;
  const size_t smem = (size_t)a.nstage * stage + 1024;
  if (!set_smem(ce_bwd_dh_tc_kernel, smem, "rbm_ce_bwd(tcgen05 dh)") || !set_smem(ce_bwd_dw_tc_kernel, smem, "rbm_ce_bwd(tcgen05 dw)")) return -1;
  ce_bwd_dh_tc_kernel<<<(unsigned)rbm_cdiv(cap, 128), 64 + 32 * NSW, smem, st>>>(mW, mWl, mWm, mWml, a);
  RBM_LAUNCH_CHECK("rbm_ce_bwd(tcgen05 dh)");
  dim3 gdw((unsigned)rbm_cdiv(V1, 128), S);
  ce_bwd_dw_tc_kernel<<<gdw, 64 + 32 * NSW, smem, st>>>(mH, mHl, mHm, mHml, a);
  RBM_LAUNCH_CHECK("rbm_ce_bwd(tcgen05 dw)");
  return 0;
}
