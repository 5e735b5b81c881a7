// ce_wide.cu -- BERT4Rec output scoring fused with masked cross-entropy on the Blackwell tensor path for WIDE hidden
// sizes (d = 128, 256) and catalogue-scale vocabularies (BASELINE configs[3]: d = 256, 10^6 items).  Replaces
// self.out(h) + CrossEntropyLoss(ignore_index=0) (NN/models/bert.py:16, NN/trainers/bert.py:11,36-40) and their autograd;
// logits only ever exist as [128 x NV] tiles in tensor memory.
//
// Arithmetic: SPLIT fp16.  Every fp32 operand x is range-scaled by a per-tensor power of two (max |x| -> [2^14, 2^15),
// found by a max-abs pass, so no magnitude overflows or underflows fp16) and split once per call into hi = fp16(x),
// lo = fp16(x - hi): 22 significant bits, the precision of 3xTF32.  A product is three tcgen05.mma kind::f16 passes
// (hi.hi + hi.lo + lo.hi, fp32 accumulate in TMEM) at twice the TF32 rate with half the operand bytes, which is what
// lets a 128-row operand of d = 256 stay resident in shared memory (128 KB) next to a ring of streamed tiles: at d > 64
// the TF32 design of ce_tc.cu (resident operand + residual in TMEM) no longer fits TMEM, and streaming both operands
// would be L2-bound.  16-bit operands also need no second (MN-major) copy of the streamed tile: the 128-byte-swizzled
// K-major tile TMA writes is, read with an MN-major descriptor, exactly the B operand of the update product.
//
// A CTA owns 128 "resident" rows (TMEM lanes, one epilogue thread per row) and streams the other side in chunks:
//   FWD  (ce_wide_fwd128_kernel) resident = 128 compacted hidden rows, stream = vocabulary range of the unit in 128-row tiles:
//        S = R.W^T into TMEM, two groups of four warps alternate chunks keeping an online (max, sum-exp) in the log2 domain +
//        the target logit.
//   The backward is one kernel template with two modes, streaming NV-row chunks (NV = 48 at d = 256, 64 at d = 128):
//   DH   resident = 128 compacted hidden rows, stream = vocabulary range of the unit: S = R.W^T, then G = (softmax - onehot) as
//        split fp16 pairs overwrites TMEM columns and feeds D[128 x d] += G . W[chunk]   (A from TMEM, B = the same streamed
//        tile read MN-major).
//   DW   resident = 128 vocabulary rows, stream = compacted hidden rows: S^T, G^T, D[128 x d] += G^T . H[chunk],
//        db = row sums of G^T; hidden-row chunks split over blockIdx.y.
// Units: FWD / DH = (row tile, vocabulary split); the split count is derived ON THE DEVICE from the live row count (the
// number of labelled rows is only known there) so that small batches still fill 148 SMs; partial (max, sum-exp, target)
// statistics / dH blocks per unit are combined in fixed order by small kernels (no atomics: bit-deterministic).
#include <cuda_fp16.h>
#include <stdlib.h>
#include "common.cuh"
#include "mma_tiles.cuh"  // ex2, RBM_LOG2E, RBM_LN2
#include "tc_ptx.cuh"
#include "split16.cuh"
#include "ce_wide.cuh"

namespace {

using namespace rbm_tc;
using rbm_mma::ex2;

constexpr int NSW = 8;                   // epilogue warps (two groups of four)
constexpr int RBLK = 128 * 128;          // one resident K-block: 128 rows x 64 fp16 = 16 KB
constexpr int UMAX = 8 * RBM_NUM_SMS;    // most (row tile, vocabulary split) units the device-side decomposition creates
constexpr float GSCALE = 16384.f;        // softmax - onehot in [-1, 1] -> fp16 range with 2^-14 * 2^-24 absolute resolution

enum { MODE_DH = 1, MODE_DW = 2 };

struct WideArgs {
  const int32_t* rows;
  const int64_t* tgt;
  const int32_t* count;
  const float* bias;
  const float* lse_in;
  const float* dloss;
  const float* scales;   // [0] = power-of-two scale of the hidden rows, [1] = of the weight
  float *st_m, *st_l, *st_t;  // FWD: per unit and resident row: running max, sum-exp (log2 domain), target logit
  float* dpart;               // DH: [unit][128][d] unscaled partial dH;  DW: part_w [S][V1][d]
  float* part_b;              // DW: [S][V1]
  const __half *r_hi, *r_lo;  // pre-split resident matrix ([r_rows, d] fp16): hidden rows (FWD / DH) or the weight (DW)
  int64_t r_rows;
  int V1, d, KB, NV, nstage, npass, S, bias_vec;
};

// vocabulary splits per row tile: the split count that fills whole waves of 148 SMs best with at most UMAX units
__host__ __device__ inline int pick_vs(int RT) {
  if (RT <= 0) return 1;
  int best = 1;
  float best_eff = -1.f;
  for (int vs = 1; vs <= 64; ++vs) {
    const int u = RT * vs;
    if (u > UMAX) break;
    const float eff = (float)u / (float)(RBM_NUM_SMS * ((u + RBM_NUM_SMS - 1) / RBM_NUM_SMS));
    if (eff > best_eff + 1e-6f) {
      best_eff = eff;
      best = vs;
    }
  }
  return best;
}

// --------------------------------------------------------------------------------------------- the backward kernel
// The resident operand's hi half lives in TENSOR MEMORY (16-bit A operand: two K elements per 32-bit column), written once
// per unit by the epilogue threads from the pre-split global copy, so the score products read only the streamed tile from
// shared memory: with both operands in shared memory a 128 x NV x 16 instruction fetches 4 KB of A + 32 NV bytes of B and
// measured ~70 cycles whatever NV (~80 B/cycle of operand fetch), three times the tensor floor of NV/2 cycles.  The lo
// half follows into TMEM where columns are left (d = 128); at d = 256 it stays in shared memory (64 KB, K-major) and only the
// third pass pays the shared-memory fetch.
//   TMEM columns: R hi [0, d/2) | group g at 128 + 64 g: S [+0, +NV) fp32, overwritten by G hi [+0, +NV/2) | G lo
//                 [+NV/2, +NV) | D [256, 256 + d)   (d = 128: R lo [384, 448))
//   SMEM: { resident lo: KB blocks of 16 KB, unless it is in TMEM } | nstage x { streamed hi (KB blocks of NV x 128 B) | lo }
template <int MODE>
__global__ void __launch_bounds__(64 + 32 * NSW, 1)
ce_wide_kernel(const __grid_constant__ CUtensorMap mapRl, const __grid_constant__ CUtensorMap mapSh, const __grid_constant__ CUtensorMap mapSl,
               const WideArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[4], empty_bar[4], s_full[2], g_full[2], r_bar, rt_bar, done_bar;
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float lse_s[2][64], tgt_s[2][64];  // DW: statistics of the chunk's streamed (hidden) rows, per group
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int count = *a.count;
  const int d = a.d, KB = a.KB, NV = a.NV, ns = a.nstage, V1 = a.V1;
  const bool lo_tmem = d <= 128;
  // ---- unit: resident tile + chunk range [c_begin, c_end) step c_step of the streamed side
  int r_tile, c_begin, c_end, c_step, unit;
  if (MODE == MODE_DW) {
    r_tile = blockIdx.x;
    unit = 0;
    c_begin = blockIdx.y;
    c_step = a.S;
    c_end = (count + NV - 1) / NV;
  } else {
    const int RT = (count + 127) / 128, VS = pick_vs(RT);
    unit = blockIdx.x;
    if (unit >= RT * VS) return;
    // vocabulary split fastest.  (Measured the other order too -- all concurrently running CTAs walking the SAME vocabulary range,
    // which cuts the DRAM reads of the streamed operand from 4x to 1x its size -- and it was SLOWER: forward 24 -> 35 ms at
    // B = 512; a hundred CTAs requesting the same L2 lines at the same moment serialise on them.  The kernel is not DRAM-bound.)
    r_tile = unit / VS;
    const int NCall = (V1 + NV - 1) / NV, cps = (NCall + VS - 1) / VS;
    c_begin = (unit % VS) * cps;
    c_end = c_begin + cps < NCall ? c_begin + cps : NCall;
    c_step = 1;
  }
  const int NL = c_end > c_begin ? (c_end - c_begin + c_step - 1) / c_step : 0;
  const uint32_t sblk = (uint32_t)NV * 128u;              // one streamed K-block
  const uint32_t stage_bytes = 2u * KB * sblk;            // hi blocks then lo blocks
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sRl = smem_base, sSt = smem_base + (lo_tmem ? 0u : (uint32_t)KB * RBLK);
  if (threadIdx.x == 0) {
    for (int s = 0; s < ns; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&g_full[i]), NSW / 2);
    }
    mbar_init(smem_u32(&r_bar), 1);
    mbar_init(smem_u32(&rt_bar), lo_tmem ? NSW : NSW / 2);
    mbar_init(smem_u32(&done_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tRh = tmem, tG0 = tmem + 128, tD = tmem + 256, tRl = tmem + 384;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      if (!lo_tmem) {
        mbar_expect_tx(smem_u32(&r_bar), (uint32_t)KB * RBLK);
        for (int kb = 0; kb < KB; ++kb) tma_load_2d(sRl + kb * RBLK, &mapRl, smem_u32(&r_bar), kb * 64, r_tile * 128);
      }
      for (int n = 0; n < NL; ++n) {
        const int c = c_begin + n * c_step, s = n % ns;
        if (n >= ns) mbar_wait(smem_u32(&empty_bar[s]), ((n / ns) - 1) & 1);
        const uint32_t bar = smem_u32(&full_bar[s]), sa = sSt + s * stage_bytes;
        mbar_expect_tx(bar, stage_bytes);
        for (int kb = 0; kb < KB; ++kb) {
          tma_load_2d(sa + kb * sblk, &mapSh, bar, kb * 64, c * NV);
          tma_load_2d(sa + (KB + kb) * sblk, &mapSl, bar, kb * 64, c * NV);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------- MMA issuer
    if (elect_one()) {
      const uint32_t idS = make_idesc_f16(128, NV, 0, 0), idU = make_idesc_f16(128, d, 0, 1);
      mbar_wait(smem_u32(&rt_bar), 0);
      if (!lo_tmem) mbar_wait(smem_u32(&r_bar), 0);
      tc_fence_after();
      // S[grp] = R . chunk^T : passes (R hi, C hi), (R hi, C lo), (R lo, C hi)
      auto scores = [&](int n) {
        const uint32_t sa = sSt + (n % ns) * stage_bytes, tS = tG0 + (uint32_t)(n & 1) * 64;
        uint32_t acc = 0;
        for (int pass = 0; pass < a.npass; ++pass) {
          const uint32_t cb = pass == 1 ? sa + KB * sblk : sa;
          for (int kb = 0; kb < KB; ++kb) {
            const uint64_t bd = make_sw128_desc(cb + kb * sblk);
            if (pass == 2 && !lo_tmem) {
              const uint64_t ad = make_sw128_desc(sRl + kb * RBLK);
#pragma unroll
              for (int k = 0; k < 4; ++k) umma_f16(tS, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idS, 1);
            } else {
              const uint32_t ta = (pass == 2 ? tRl : tRh) + (uint32_t)(kb * 32);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                umma_f16_ts(tS, ta + (uint32_t)(k * 8), bd + (uint64_t)(k * 2), idS, acc);
                acc = 1;
              }
            }
          }
        }
      };
      int pend[2] = {-1, -1};
      bool d_started = false;
      // D += G[grp] . chunk : passes (G hi, C hi), (G hi, C lo), (G lo, C hi); K = the chunk's NV rows, 16 per instruction
      auto accum = [&](int grp) {
        const int n = pend[grp], s = n % ns;
        mbar_wait(smem_u32(&g_full[grp]), (n >> 1) & 1);
        tc_fence_after();
        const uint32_t sa = sSt + s * stage_bytes, tGh = tG0 + (uint32_t)grp * 64, tGl = tGh + (uint32_t)(NV / 2);
        for (int pass = 0; pass < a.npass; ++pass) {
          const uint32_t ga = pass == 2 ? tGl : tGh, cb = pass == 1 ? sa + KB * sblk : sa;
          for (int ks = 0; ks < NV / 16; ++ks) {
            umma_f16_ts(tD, ga + (uint32_t)(ks * 8), make_sw128_desc_mn16(cb + ks * 2048, sblk), idU, d_started ? 1u : 0u);
            d_started = true;
          }
        }
        umma_commit(smem_u32(&empty_bar[s]));
        pend[grp] = -1;
      };
      for (int n = 0; n < NL; ++n) {
        const int s = n % ns, grp = n & 1;
        if (pend[grp] >= 0) accum(grp);  // frees the group's column block (the tensor pipe runs in order)
        mbar_wait(smem_u32(&full_bar[s]), (n / ns) & 1);
        tc_fence_after();
        scores(n);
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
    // ----------------------------------------------------------------------------------- epilogue / softmax warps
    const int q = warp & 3, grp = (warp - 2) >> 2;
    const int gt = q * 32 + lane;  // thread index inside the group (= resident row; lane quarters in warp order 2,3,0,1)
    const int rl = gt;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const uint32_t tS = tG0 + lane_sel + (uint32_t)grp * 64, tGl = tS + (uint32_t)(NV / 2);
    const float sh = a.scales[0], sw = a.scales[1];
    const float c1 = RBM_LOG2E / (sh * sw);  // accumulator -> logit in the log2 domain
    float* xch = reinterpret_cast<float*>(smem_raw + (sSt - smem_u32(smem_raw)));  // first stage, reused after the MMAs
    // ---- resident rows -> tensor memory (group 0: hi half; group 1: lo half where it lives there)
    if (grp == 0 || lo_tmem) {
      const int64_t grow = (int64_t)r_tile * 128 + rl;
      const uint4* src = reinterpret_cast<const uint4*>((grp == 0 ? a.r_hi : a.r_lo) + grow * d);
      const bool inb = grow < a.r_rows;
      const uint32_t dstc = (grp == 0 ? tRh : tRl) + lane_sel;
      for (int c0 = 0; c0 < d / 2; c0 += 8) {  // 8 words = 16 fp16 = two 16-byte loads
        uint32_t w8[8];
        const uint4 x = inb ? src[c0 / 4] : make_uint4(0, 0, 0, 0), y = inb ? src[c0 / 4 + 1] : make_uint4(0, 0, 0, 0);
        w8[0] = x.x; w8[1] = x.y; w8[2] = x.z; w8[3] = x.w; w8[4] = y.x; w8[5] = y.y; w8[6] = y.z; w8[7] = y.w;
        tmem_st8(dstc + (uint32_t)c0, w8);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&rt_bar));
    }
    if (MODE == MODE_DH) {
      const int r = r_tile * 128 + rl;
      const bool valid = r < count;
      int64_t tg = valid ? a.tgt[r] : -1;
      if (tg < 0 || tg >= V1) tg = -1;  // a target outside this (shard of the) vocabulary matches no column
      const float lse2 = valid ? a.lse_in[r] * RBM_LOG2E : INFINITY;  // rows beyond the count: p = 0
      for (int n = grp; n < NL; n += 2) {
        const int c = c_begin + n;
        mbar_wait(smem_u32(&s_full[grp]), (n >> 1) & 1);
        tc_fence_after();
        float sv[64];  // the chunk's scores of this row (all of them are read before G overwrites the columns)
#pragma unroll
        for (int part = 0; part < 4; ++part)
          if (part * 16 < NV) tmem_ld16(tS + (uint32_t)(part * 16), *reinterpret_cast<float(*)[16]>(&sv[part * 16]));
#pragma unroll
        for (int part = 0; part < 4; ++part) {
          if (part * 16 < NV) {
            const int v0 = c * NV + part * 16;
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
            float(&v)[16] = *reinterpret_cast<float(*)[16]>(&sv[part * 16]);
            const uint32_t ts = (uint32_t)(tg - (int64_t)v0);  // this row's target column inside the slice, if < 16
            const bool hit = __any_sync(0xffffffffu, ts < 16u);
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float p = ex2(fmaf(v[j], c1, bb[j]));
              if (hit && ts == (uint32_t)j) p -= 1.f;
              v[j] = p * GSCALE;
            }
            split_pack16(v, hi, lo);
            tmem_st8(tS + (uint32_t)(part * 8), hi);
            tmem_st8(tGl + (uint32_t)(part * 8), lo);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&g_full[grp]));
      }
      mbar_wait(smem_u32(&done_bar), 0);
      tc_fence_after();
      // unscaled partial dH block of this unit; the two groups split the d columns
      float* dst = a.dpart + ((int64_t)unit * 128 + rl) * d;
      const int dc = d / 2;
      for (int c0 = grp * dc; c0 < (grp + 1) * dc; c0 += 16) {
        float o[16];
        if (NL > 0) {
          tmem_ld16(tD + lane_sel + (uint32_t)c0, o);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) o[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < 16; j += 4) st4(dst + c0 + j, make_float4(o[j], o[j + 1], o[j + 2], o[j + 3]));
      }
    } else {
      // ------------------------------------------------------------------------------------------ DW: rows = vocabulary
      const int vrow = r_tile * 128 + rl;
      const bool valid = vrow < V1;
      const float b2 = valid ? (a.bias ? a.bias[vrow] * RBM_LOG2E : 0.f) : -INFINITY;  // rows beyond the vocabulary: p = 0
      const float frow = valid ? (float)vrow : -2.f;
      float bsum = 0.f;
      for (int n = grp; n < NL; n += 2) {
        const int c = c_begin + n * c_step;
        // statistics of the chunk's NV hidden rows (the group's previous chunk has been consumed: its g_full arrival came
        // after the last read of these arrays)
        named_bar_sync(1 + grp, 128);
        if (gt < NV) {
          const int r = c * NV + gt;
          lse_s[grp][gt] = r < count ? a.lse_in[r] * RBM_LOG2E : INFINITY;  // columns beyond the count: p = 0
          tgt_s[grp][gt] = (r < count && a.tgt[r] >= 0 && a.tgt[r] < V1) ? (float)a.tgt[r] : -1.f;
        }
        named_bar_sync(1 + grp, 128);
        mbar_wait(smem_u32(&s_full[grp]), (n >> 1) & 1);
        tc_fence_after();
        float sv[64];
#pragma unroll
        for (int part = 0; part < 4; ++part)
          if (part * 16 < NV) tmem_ld16(tS + (uint32_t)(part * 16), *reinterpret_cast<float(*)[16]>(&sv[part * 16]));
#pragma unroll
        for (int part = 0; part < 4; ++part) {
          if (part * 16 < NV) {
            float(&v)[16] = *reinterpret_cast<float(*)[16]>(&sv[part * 16]);
            float ls[16], tc[16];
#pragma unroll
            for (int j = 0; j < 16; j += 4) {
              const float4 x = ld4(&lse_s[grp][part * 16 + j]), y = ld4(&tgt_s[grp][part * 16 + j]);
              ls[j] = x.x; ls[j + 1] = x.y; ls[j + 2] = x.z; ls[j + 3] = x.w;
              tc[j] = y.x; tc[j + 1] = y.y; tc[j + 2] = y.z; tc[j + 3] = y.w;
            }
            uint32_t hi[8], lo[8];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float p = ls[j] == INFINITY ? 0.f : ex2(fmaf(v[j], c1, b2) - ls[j]);  // columns beyond the count: exactly zero
              if (tc[j] == frow) p -= 1.f;
              bsum += p;
              v[j] = p * GSCALE;
            }
            split_pack16(v, hi, lo);
            tmem_st8(tS + (uint32_t)(part * 8), hi);
            tmem_st8(tGl + (uint32_t)(part * 8), lo);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&g_full[grp]));
      }
      mbar_wait(smem_u32(&done_bar), 0);
      tc_fence_after();
      named_bar_sync(7, NSW * 32);
      xch[grp * 128 + rl] = bsum;
      named_bar_sync(7, NSW * 32);
      // no labelled row: zero, not 0 x (dloss / 0) = NaN (test_ce_no_labelled_row)
      const float gscale = count > 0 ? *a.dloss / (float)count : 0.f;
      const float wmul = gscale / (GSCALE * sh);  // D = sum (2^14 G) . (s_h H)
      float* pw = a.dpart + ((int64_t)blockIdx.y * V1 + vrow) * d;
      const int dc = d / 2;
      for (int c0 = grp * dc; c0 < (grp + 1) * dc; c0 += 16) {
        float o[16];
        if (NL > 0) {
          tmem_ld16(tD + lane_sel + (uint32_t)c0, o);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) o[j] = 0.f;
        }
        if (valid) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) st4(pw + c0 + j, make_float4(o[j] * wmul, o[j + 1] * wmul, o[j + 2] * wmul, o[j + 3] * wmul));
        }
      }
      if (grp == 0 && valid) a.part_b[(int64_t)blockIdx.y * V1 + vrow] = (xch[rl] + xch[128 + rl]) * gscale;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// ------------------------------------------------------------------------------------------ forward, 128-row tiles
// The forward has no accumulator to keep, so tensor memory holds BOTH resident halves (2 x d/2 columns) and two score blocks
// of 128 columns: the score products become 128 x 128 x 16 instructions, the smallest that run at the tensor floor (64 cycles;
// the 64-column instructions of the template above cost ~70).  A 128-row vocabulary tile is 128 KB of hi + lo operand, too big
// for whole-tile stages, so the ring is made of 16 KB K-block PIECES [128 rows x 64 columns], consumed in the order
// hi[0] (x R hi, x R lo), lo[0] (x R hi), hi[1], ...: thirteen pieces (208 KB) are in flight.
//   TMEM columns: R hi [0, d/2) | S0 [128, 256) | S1 [256, 384) | R lo [384, 384 + d/2)
constexpr int NPIECE = 13;
__global__ void __launch_bounds__(64 + 32 * NSW, 1)
ce_wide_fwd128_kernel(const __grid_constant__ CUtensorMap mapSh, const __grid_constant__ CUtensorMap mapSl, const WideArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t pfull[NPIECE], pempty[NPIECE], s_full[2], g_full[2], rt_bar;
  __shared__ uint32_t tmem_base_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int count = *a.count;
  const int d = a.d, KB = a.KB, V1 = a.V1;
  constexpr int NV = 128;
  const int RT = (count + 127) / 128, VS = pick_vs(RT);
  const int unit = blockIdx.x;
  if (unit >= RT * VS) return;
  const int r_tile = unit / VS;
  const int NCall = (V1 + NV - 1) / NV, cps = (NCall + VS - 1) / VS;
  const int c_begin = (unit % VS) * cps;
  const int c_end = c_begin + cps < NCall ? c_begin + cps : NCall;
  const int NL = c_end > c_begin ? c_end - c_begin : 0;
  const int ppc = (a.npass == 1 ? 1 : 2) * KB;  // pieces per chunk
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  if (threadIdx.x == 0) {
    for (int s = 0; s < NPIECE; ++s) {
      mbar_init(smem_u32(&pfull[s]), 1);
      mbar_init(smem_u32(&pempty[s]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&g_full[i]), NSW / 2);
    }
    mbar_init(smem_u32(&rt_bar), NSW);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;
  const uint32_t tRh = tmem, tS0 = tmem + 128, tRl = tmem + 384;

  if (warp == 0) {
    if (elect_one()) {
      int q = 0;
      for (int n = 0; n < NL; ++n) {
        const int c = c_begin + n;
        for (int pp = 0; pp < ppc; ++pp, ++q) {
          const int slot = q % NPIECE, kb = a.npass == 1 ? pp : pp >> 1, lo = a.npass == 1 ? 0 : pp & 1;
          if (q >= NPIECE) mbar_wait(smem_u32(&pempty[slot]), ((q / NPIECE) - 1) & 1);
          const uint32_t bar = smem_u32(&pfull[slot]);
          mbar_expect_tx(bar, RBLK);
          tma_load_2d(smem_base + slot * RBLK, lo ? &mapSl : &mapSh, bar, kb * 64, c * NV);
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idS = make_idesc_f16(128, NV, 0, 0);
      mbar_wait(smem_u32(&rt_bar), 0);
      tc_fence_after();
      int q = 0;
      for (int n = 0; n < NL; ++n) {
        const int grp = n & 1;
        const uint32_t tS = tS0 + (uint32_t)grp * 128;
        if (n >= 2) {
          mbar_wait(smem_u32(&g_full[grp]), ((n >> 1) - 1) & 1);
          tc_fence_after();
        }
        uint32_t acc = 0;
        for (int pp = 0; pp < ppc; ++pp, ++q) {
          const int slot = q % NPIECE, kb = a.npass == 1 ? pp : pp >> 1, lo = a.npass == 1 ? 0 : pp & 1;
          mbar_wait(smem_u32(&pfull[slot]), (q / NPIECE) & 1);
          tc_fence_after();
          const uint64_t bd = make_sw128_desc(smem_base + slot * RBLK);
#pragma unroll
          for (int k = 0; k < 4; ++k) {  // this piece x R hi
            umma_f16_ts(tS, tRh + (uint32_t)(kb * 32 + k * 8), bd + (uint64_t)(k * 2), idS, acc);
            acc = 1;
          }
          if (!lo && a.npass != 1) {
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16_ts(tS, tRl + (uint32_t)(kb * 32 + k * 8), bd + (uint64_t)(k * 2), idS, 1);  // hi piece x R lo
          }
          umma_commit(smem_u32(&pempty[slot]));
        }
        umma_commit(smem_u32(&s_full[grp]));
      }
    }
    __syncwarp();
  } else {
    const int q4 = warp & 3, grp = (warp - 2) >> 2;
    const int rl = q4 * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q4 * 32) << 16;
    const uint32_t tS = tS0 + lane_sel + (uint32_t)grp * 128;
    const float c1 = RBM_LOG2E / (a.scales[0] * a.scales[1]);
    float* xch = reinterpret_cast<float*>(smem_raw + (smem_base - smem_u32(smem_raw)));
    {  // resident rows -> tensor memory (group 0: hi half, group 1: lo half)
      const int64_t grow = (int64_t)r_tile * 128 + rl;
      const uint4* src = reinterpret_cast<const uint4*>((grp == 0 ? a.r_hi : a.r_lo) + grow * d);
      const bool inb = grow < a.r_rows;
      const uint32_t dstc = (grp == 0 ? tRh : tRl) + lane_sel;
      for (int c0 = 0; c0 < d / 2; c0 += 8) {
        uint32_t w8[8];
        const uint4 x = inb ? src[c0 / 4] : make_uint4(0, 0, 0, 0), y = inb ? src[c0 / 4 + 1] : make_uint4(0, 0, 0, 0);
        w8[0] = x.x; w8[1] = x.y; w8[2] = x.z; w8[3] = x.w; w8[4] = y.x; w8[5] = y.y; w8[6] = y.z; w8[7] = y.w;
        tmem_st8(dstc + (uint32_t)c0, w8);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&rt_bar));
    }
    const int r = r_tile * 128 + rl;
    const bool valid = r < count;
    int64_t tg = valid ? a.tgt[r] : -1;
    if (tg < 0 || tg >= V1) tg = -1;
    float m = -INFINITY, l = 0.f, tl = 0.f;
    for (int n = grp; n < NL; n += 2) {
      const int c = c_begin + n;
      mbar_wait(smem_u32(&s_full[grp]), (n >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int part = 0; part < NV / 16; ++part) {
        const int v0 = c * NV + part * 16;
        float bb[16];
        if (v0 + 16 <= V1 && (a.bias == nullptr || a.bias_vec)) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {
            const float4 t = a.bias ? ld4(a.bias + v0 + j) : make_float4(0.f, 0.f, 0.f, 0.f);
            bb[j] = t.x * RBM_LOG2E; bb[j + 1] = t.y * RBM_LOG2E; bb[j + 2] = t.z * RBM_LOG2E; bb[j + 3] = t.w * RBM_LOG2E;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) bb[j] = v0 + j < V1 ? (a.bias ? a.bias[v0 + j] * RBM_LOG2E : 0.f) : -INFINITY;
        }
        float v[16];
        tmem_ld16(tS + (uint32_t)(part * 16), v);
        if (part == NV / 16 - 1) {  // last read of this chunk's score block
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(smem_u32(&g_full[grp]));
        }
        const uint32_t ts = (uint32_t)(tg - (int64_t)v0);
        const bool hit = __any_sync(0xffffffffu, ts < 16u);
        float cm = -INFINITY;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          v[j] = fmaf(v[j], c1, bb[j]);
          cm = fmaxf(cm, v[j]);
        }
        if (hit) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (ts == (uint32_t)j) tl = v[j];
        }
        const float mn = fmaxf(m, cm);
        if (mn > -INFINITY) {
          float ps = 0.f;
#pragma unroll
          for (int j = 0; j < 16; ++j) ps += ex2(v[j] - mn);
          l = l * (m == -INFINITY ? 0.f : ex2(m - mn)) + ps;
          m = mn;
        }
      }
    }
    // every chunk's scores have been read, hence every MMA has completed and every piece is free
    named_bar_sync(7, NSW * 32);
    xch[(grp * 3 + 0) * 128 + rl] = m;
    xch[(grp * 3 + 1) * 128 + rl] = l;
    xch[(grp * 3 + 2) * 128 + rl] = tl;
    named_bar_sync(7, NSW * 32);
    if (grp == 0) {
      const float m0 = xch[rl], m1 = xch[3 * 128 + rl];
      const float mm = fmaxf(m0, m1);
      const float ll = xch[128 + rl] * (m0 == -INFINITY ? 0.f : ex2(m0 - mm)) + xch[4 * 128 + rl] * (m1 == -INFINITY ? 0.f : ex2(m1 - mm));
      a.st_m[(int64_t)unit * 128 + rl] = mm;
      a.st_l[(int64_t)unit * 128 + rl] = ll;
      a.st_t[(int64_t)unit * 128 + rl] = xch[2 * 128 + rl] + xch[5 * 128 + rl];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// ---------------------------------------------------------------------------------------------- helper kernels
// Hc[r] = h[rows[r]] * scales[0] (r < count) as hi/lo fp16; zeros up to the next multiple of 128 PLUS one more tile: the DW
// kernel streams these rows in NV-row chunks, and the last chunk may reach past the 128-row boundary into what would
// otherwise be stale workspace (0 x NaN = NaN inside the tensor core)
__global__ void __launch_bounds__(256) gather_split_h_kernel(const float* __restrict__ h, const int32_t* __restrict__ rows,
                                                             const int32_t* __restrict__ count_p, const float* __restrict__ scales,
                                                             uint2* __restrict__ hi, uint2* __restrict__ lo, int64_t cap128, int d4) {
  const int count = *count_p;
  int64_t lim = ((int64_t)count + 127) / 128 * 128 + 128;
  if (lim > cap128) lim = cap128;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= lim * d4) return;
  const int64_t r = i / d4;
  const int c4 = (int)(i - r * d4);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (r < count) v = ld4(h + ((int64_t)rows[r] * d4 + c4) * 4);
  uint2 a, b;
  split4(v, scales[0], a, b);
  hi[i] = a;
  lo[i] = b;
}
// FWD: per row, combine the vocabulary splits' (max, sum-exp, target logit) -> lse[r]; per 128-row block the sum of
// (lse - target logit) in fixed order -> partial[block]
__global__ void __launch_bounds__(128) fwd_combine_kernel(const float* __restrict__ st_m, const float* __restrict__ st_l, const float* __restrict__ st_t,
                                                          const int32_t* __restrict__ count_p, float* __restrict__ lse_out, float* __restrict__ partial) {
  __shared__ float contrib[128];
  const int count = *count_p, RT = (count + 127) / 128, VS = pick_vs(RT);
  const int b = blockIdx.x, t = threadIdx.x, r = b * 128 + t;
  if (b >= RT) {
    if (t == 0) partial[b] = 0.f;
    return;
  }
  float M = -INFINITY;
  for (int vs = 0; vs < VS; ++vs) M = fmaxf(M, st_m[((int64_t)b * VS + vs) * 128 + t]);
  float L = 0.f, TL = 0.f;
  for (int vs = 0; vs < VS; ++vs) {
    const int64_t o = ((int64_t)b * VS + vs) * 128 + t;
    const float m = st_m[o];
    if (m > -INFINITY) L += st_l[o] * ex2(m - M);
    TL += st_t[o];
  }
  const float lse = (M + log2f(L)) * RBM_LN2;
  const bool valid = r < count;
  if (valid) lse_out[r] = lse;
  contrib[t] = valid ? lse - TL * RBM_LN2 : 0.f;
  __syncthreads();
  if (t == 0) {
    float s = 0.f;
    for (int i = 0; i < 128; ++i) s += contrib[i];
    partial[b] = s;
  }
}
// DH: dh_full[rows[r]] = (sum over the row tile's vocabulary splits, in order) * dloss / (count * 2^14 * s_w)
__global__ void __launch_bounds__(256) dh_reduce_kernel(const float* __restrict__ dpart, const int32_t* __restrict__ rows,
                                                        const int32_t* __restrict__ count_p, const float* __restrict__ scales,
                                                        const float* __restrict__ dloss, float* __restrict__ dh_full, int d4) {
  const int count = *count_p, RT = (count + 127) / 128, VS = pick_vs(RT);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t r = i / d4;
  if (r >= count) return;
  const int c4 = (int)(i - r * d4);
  const int rt = (int)(r >> 7), rl = (int)(r & 127);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int vs = 0; vs < VS; ++vs) {
    const float4 v = ld4(dpart + ((((int64_t)rt * VS + vs) * 128 + rl) * d4 + c4) * 4);
    s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
  }
  const float mul = *dloss / ((float)count * GSCALE * scales[1]);
  st4(dh_full + ((int64_t)rows[r] * d4 + c4) * 4, make_float4(s.x * mul, s.y * mul, s.z * mul, s.w * mul));
}

// fp16 passes per product: 3 (hi.hi + hi.lo + lo.hi), or 1 (hi.hi) under RBM_CE_WIDE_PASSES=1, the reduced-precision line.
// Read on every call, never cached: bench.py's labelled reduced-precision line and test_score_ce_wide_million_items set and
// unset the variable inside one process, and a cached value would time or test the three-pass kernels under the wrong label.
int wide_passes() {
  const char* e = getenv("RBM_CE_WIDE_PASSES");
  return e && atoi(e) == 1 ? 1 : 3;
}
struct Shape {
  int NV, ns, npass;
  size_t smem;
};
// streamed rows per chunk, ring depth, shared memory of the backward kernels: at d = 128 both resident halves are in tensor
// memory -> all shared memory is ring; at d = 256 the resident lo half (64 KB) stays in shared memory
Shape pick_shape(int d) {
  Shape s;
  const bool lo_tmem = d <= 128;
  s.NV = lo_tmem ? 64 : 48;
  const size_t res = lo_tmem ? 0 : (size_t)(d / 64) * RBLK, stage = (size_t)2 * (d / 64) * s.NV * 128;
  int ns = (int)(((size_t)231000 - 1024 - res) / stage);
  s.ns = ns > 4 ? 4 : ns;
  s.npass = wide_passes();
  s.smem = res + (size_t)s.ns * stage + 1024;
  return s;
}
int64_t grid_units(int64_t cap128) { return cap128 / 128 > UMAX ? cap128 / 128 : UMAX; }

// workspace carve-up (floats): scales + bits (16) | W hi | W lo | Hc hi | Hc lo | fwd stats 3 x UG x 128 | dH partial UG x 128 x d
struct WideWs {
  unsigned* bits;
  float* scales;
  void *w_hi, *w_lo, *h_hi, *h_lo;
  float *st_m, *st_l, *st_t, *dpart;
  size_t total;
};
WideWs carve(float* base, int64_t cap, int V1, int d) {
  const int64_t cap128 = (cap + 127) / 128 * 128, UG = grid_units(cap128);
  WideWs w;
  size_t o = 0;
  w.bits = (unsigned*)(base + o);
  w.scales = base + o + 4;
  o += 16;
  const size_t wh = ((size_t)V1 * d / 2 + 3) & ~(size_t)3, hh = (size_t)cap128 * d / 2;
  w.w_hi = base + o; o += wh;
  w.w_lo = base + o; o += wh;
  w.h_hi = base + o; o += hh;
  w.h_lo = base + o; o += hh;
  w.st_m = base + o; o += (size_t)UG * 128;
  w.st_l = base + o; o += (size_t)UG * 128;
  w.st_t = base + o; o += (size_t)UG * 128;
  w.dpart = base + o; o += (size_t)UG * 128 * d;
  w.total = o;
  return w;
}

// range scales + split copies of both operands (recomputed by the backward: the workspace is shared scratch)
int prepare(const float* h, const int32_t* rows, const int32_t* count, const float* w, int64_t cap, int V1, int d, const WideWs& ws,
            cudaStream_t st) {
  const int64_t cap128 = (cap + 127) / 128 * 128;
  cudaMemsetAsync(ws.bits, 0, 16, st);
  const int64_t nh4 = cap * d / 4, nw4 = (int64_t)V1 * d / 4;
  maxabs_launch(h, d, cap, d, ws.bits, (int)(rbm_cdiv(nh4, 256) < 4 * RBM_NUM_SMS ? rbm_cdiv(nh4, 256) : 4 * RBM_NUM_SMS), st);
  maxabs_launch(w, d, V1, d, ws.bits + 1, (int)(rbm_cdiv(nw4, 256) < 4 * RBM_NUM_SMS ? rbm_cdiv(nw4, 256) : 4 * RBM_NUM_SMS), st);
  scales_launch(ws.bits, ws.scales, st);
  split_w_launch(w, ws.scales + 1, (uint2*)ws.w_hi, (uint2*)ws.w_lo, nw4, st);
  gather_split_h_kernel<<<(unsigned)rbm_cdiv(cap128 * (d / 4), 256), 256, 0, st>>>(h, rows, count, ws.scales, (uint2*)ws.h_hi, (uint2*)ws.h_lo,
                                                                                  cap128, d / 4);
  RBM_LAUNCH_CHECK("rbm_ce(wide prepare)");
  return 0;
}

}  // namespace

static bool wide_dim(int d) { return d == 128 || d == 256; }

bool rbm_ce_wide_supported(int V1, int d, const void* h, const void* w) {
  if (!wide_dim(d) || V1 < 64) return false;
  if (((uintptr_t)h | (uintptr_t)w) & 15) return false;
  return get_encode() != nullptr;
}

size_t rbm_ce_wide_ws_floats(int64_t cap, int V1, int d) {
  if (!wide_dim(d)) return 0;
  return carve(nullptr, cap, V1, d).total + 64;
}

// hidden-row splits of the dW / db kernel: enough (vocabulary tile, split) units for about four waves of SMs
int rbm_ce_wide_dw_splits(int64_t cap, int V1) {
  int64_t vt = rbm_cdiv(V1, 128), chunks = rbm_cdiv(cap, 64);
  int64_t s = rbm_cdiv((int64_t)4 * RBM_NUM_SMS, vt);
  if (s > chunks) s = chunks;
  if (s > 64) s = 64;
  return (int)(s < 1 ? 1 : s);
}

int rbm_ce_wide_fwd(const float* h, const int32_t* rows, const int64_t* tgt, const int32_t* count, const float* w, const float* bias,
                    float* lse, float* partial, int64_t cap, int V1, int d, float* extra_ws, int* nblk_out, cudaStream_t st) {
  const int64_t cap128 = (cap + 127) / 128 * 128;
  const WideWs ws = carve(extra_ws, cap, V1, d);
  if (int rc = prepare(h, rows, count, w, cap, V1, d, ws, st)) return rc;
  // 128-row vocabulary tiles through a ring of K-block pieces (N = 128 instructions)
  CUtensorMap mSh, mSl;
  if (!encode_f16_rows(&mSh, ws.w_hi, V1, d, 128) || !encode_f16_rows(&mSl, ws.w_lo, V1, d, 128)) {
    rbm_set_error("rbm_ce_fwd(wide): cuTensorMapEncodeTiled failed");
    return -1;
  }
  WideArgs a{};
  a.rows = rows; a.tgt = tgt; a.count = count; a.bias = bias; a.scales = ws.scales; a.st_m = ws.st_m; a.st_l = ws.st_l; a.st_t = ws.st_t;
  a.r_hi = (const __half*)ws.h_hi; a.r_lo = (const __half*)ws.h_lo; a.r_rows = cap128;
  a.V1 = V1; a.d = d; a.KB = d / 64; a.npass = wide_passes();
  a.bias_vec = bias != nullptr && ((uintptr_t)bias & 15) == 0;
  const size_t smem = (size_t)NPIECE * RBLK + 1024;
  if (!set_smem(ce_wide_fwd128_kernel, smem, "rbm_ce_fwd(wide 128)")) return -1;
  ce_wide_fwd128_kernel<<<(unsigned)grid_units(cap128), 64 + 32 * NSW, smem, st>>>(mSh, mSl, a);
  RBM_LAUNCH_CHECK("rbm_ce_fwd(wide)");
  const int nblk = (int)(cap128 / 128);
  fwd_combine_kernel<<<nblk, 128, 0, st>>>(ws.st_m, ws.st_l, ws.st_t, count, lse, partial);
  RBM_LAUNCH_CHECK("rbm_ce_fwd(wide combine)");
  *nblk_out = nblk;
  return 0;
}

int rbm_ce_wide_bwd(const float* h, const int32_t* rows, const int64_t* tgt, const int32_t* count, const float* w, const float* bias,
                    const float* lse, const float* dloss, float* dh_full, float* part_w, float* part_b, int S, int64_t cap, int V1, int d,
                    float* extra_ws, cudaStream_t st) {
  const int64_t cap128 = (cap + 127) / 128 * 128;
  const WideWs ws = carve(extra_ws, cap, V1, d);
  if (int rc = prepare(h, rows, count, w, cap, V1, d, ws, st)) return rc;
  const Shape sh = pick_shape(d);
  CUtensorMap mHlr, mWs, mWls, mWlr, mHs, mHls;
  if (!encode_f16_rows(&mHlr, ws.h_lo, cap128, d, 128) || !encode_f16_rows(&mWs, ws.w_hi, V1, d, sh.NV) ||
      !encode_f16_rows(&mWls, ws.w_lo, V1, d, sh.NV) || !encode_f16_rows(&mWlr, ws.w_lo, V1, d, 128) ||
      !encode_f16_rows(&mHs, ws.h_hi, cap128, d, sh.NV) || !encode_f16_rows(&mHls, ws.h_lo, cap128, d, sh.NV)) {
    rbm_set_error("rbm_ce_bwd(wide): cuTensorMapEncodeTiled failed");
    return -1;
  }
  WideArgs a{};
  a.rows = rows; a.tgt = tgt; a.count = count; a.bias = bias; a.lse_in = lse; a.dloss = dloss; a.scales = ws.scales;
  a.V1 = V1; a.d = d; a.KB = d / 64; a.NV = sh.NV; a.nstage = sh.ns; a.npass = sh.npass; a.S = S;
  a.bias_vec = bias != nullptr && ((uintptr_t)bias & 15) == 0;
  if (!set_smem(ce_wide_kernel<MODE_DH>, sh.smem, "rbm_ce_bwd(wide dh)") || !set_smem(ce_wide_kernel<MODE_DW>, sh.smem, "rbm_ce_bwd(wide dw)"))
    return -1;
  a.dpart = ws.dpart;
  a.r_hi = (const __half*)ws.h_hi; a.r_lo = (const __half*)ws.h_lo; a.r_rows = cap128;
  ce_wide_kernel<MODE_DH><<<(unsigned)grid_units(cap128), 64 + 32 * NSW, sh.smem, st>>>(mHlr, mWs, mWls, a);
  RBM_LAUNCH_CHECK("rbm_ce_bwd(wide dh)");
  dh_reduce_kernel<<<(unsigned)rbm_cdiv(cap * (d / 4), 256), 256, 0, st>>>(ws.dpart, rows, count, ws.scales, dloss, dh_full, d / 4);
  RBM_LAUNCH_CHECK("rbm_ce_bwd(wide dh reduce)");
  a.dpart = part_w;
  a.part_b = part_b;
  a.r_hi = (const __half*)ws.w_hi; a.r_lo = (const __half*)ws.w_lo; a.r_rows = V1;
  dim3 gdw((unsigned)rbm_cdiv(V1, 128), S);
  ce_wide_kernel<MODE_DW><<<gdw, 64 + 32 * NSW, sh.smem, st>>>(mWlr, mHs, mHls, a);
  RBM_LAUNCH_CHECK("rbm_ce_bwd(wide dw)");
  return 0;
}
