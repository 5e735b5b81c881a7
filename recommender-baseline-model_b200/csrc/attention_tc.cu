// attention_tc.cu -- attention forward and backward on the Blackwell tensor path for d_k = 32, L <= 256 (the cfg2
// BERT4Rec shape).  Three persistent, warp-specialised kernels (forward, backward pass A: dQ, backward pass B: dK/dV),
// one CTA per SM walking (sequence, head, 128-row tile) work items; see the comment block in front of each kernel.
// Common ground: TMA (3-D maps over [B, L, cols]) streams token rows as 128-byte-swizzled tiles -- K-major tiles for
// products that contract along d_k, MN-major (32-byte-atom swizzle) tiles for products that contract along tokens;
// the 128 resident rows of a tile are TMEM A operands; scores / probabilities / score gradients only ever exist in
// TMEM; every product is 3xTF32-compensated (operand = TF32 part + TF32 residual), i.e. fp32-level accuracy.
// Shapes outside (d_k == 32, L <= 256) use the mma.sync kernels (attention.cu).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "common.cuh"
#include "mma_tiles.cuh"  // ex2, RBM_LOG2E, RBM_PADFILL
#include "tc_ptx.cuh"
#include "attention_tc.cuh"

namespace {

using namespace rbm_tc;
using rbm_mma::ex2;

constexpr int DK = 32;
constexpr int ROWB = DK * 4;     // 128 bytes per token row

// =====================================================================================================
// Dropout words of one query row for the 16 keys [16*npair, 16*npair + 16).  Rows i and i^8 (lanes l, l^8 of a warp
// whose lanes hold consecutive rows) share their four Philox calls: each lane computes two and trades the words the
// other row needs.  w[2*t + e] holds the fields of keys jj with ((jj & 7) >> 1) == t, (jj & 1) == e: low half for
// jj < 8, high half for jj >= 8 (common.cuh, rbm_attn_call / rbm_attn_field).
// =====================================================================================================
struct KeepWords {
  uint32_t w[8];
};
__device__ __forceinline__ KeepWords attn_keep_words(uint64_t seed, uint64_t site, uint64_t bh, int i, int npair) {
  const int tile = i >> 4, g = i & 7, rh = (i >> 3) & 1;
  const uint4 ca = rbm_philox_drop(seed, site, rbm_attn_call(bh, tile, g, rh * 2 + 0, npair));
  const uint4 cb = rbm_philox_drop(seed, site, rbm_attn_call(bh, tile, g, rh * 2 + 1, npair));
  // mine: words rh*2 + e; the partner row (rh ^ 1) wants the other pair
  const uint32_t ma0 = rh ? ca.z : ca.x, ma1 = rh ? ca.w : ca.y, mb0 = rh ? cb.z : cb.x, mb1 = rh ? cb.w : cb.y;
  const uint32_t sa0 = rh ? ca.x : ca.z, sa1 = rh ? ca.y : ca.w, sb0 = rh ? cb.x : cb.z, sb1 = rh ? cb.y : cb.w;
  const uint32_t pa0 = __shfl_xor_sync(0xffffffffu, sa0, 8), pa1 = __shfl_xor_sync(0xffffffffu, sa1, 8);
  const uint32_t pb0 = __shfl_xor_sync(0xffffffffu, sb0, 8), pb1 = __shfl_xor_sync(0xffffffffu, sb1, 8);
  KeepWords k;  // my calls are t = rh*2, rh*2 + 1; the partner's are t = (rh^1)*2, (rh^1)*2 + 1
  k.w[0] = rh ? pa0 : ma0; k.w[1] = rh ? pa1 : ma1; k.w[2] = rh ? pb0 : mb0; k.w[3] = rh ? pb1 : mb1;
  k.w[4] = rh ? ma0 : pa0; k.w[5] = rh ? ma1 : pa1; k.w[6] = rh ? mb0 : pb0; k.w[7] = rh ? mb1 : pb1;
  return k;
}
// keep decision of key jj (compile-time after unrolling); thr_hi = thr16 << 16
__device__ __forceinline__ bool attn_keep_bit(const KeepWords& k, int jj, uint32_t thr_hi) {
  const uint32_t w = k.w[((jj & 7) >> 1) * 2 + (jj & 1)];
  return (jj & 8) ? (w >= thr_hi) : ((w << 16) >= thr_hi);
}

// =====================================================================================================
// Forward on the tensor path: persistent, one CTA per SM walking the work items (sequence, head, 128-query tile).
//   warp 0      TMA: the item's Q rows (one 128-row tile) and the key stream in chunks of <= 64 -- K chunks (K-major, for
//               S = Q.K^T) and V chunks (MN-major, for O += P.V) through two 4-stage rings, issued in consumption order
//   warps 14-15 TF32 residual copy of every staged tile
//   warp 1      tcgen05.mma issue.  The whole score tile S [128 x Lp] lives in TMEM (exact row maxima need every key
//               before the first exponential); the chunks of item n+1 are computed into the columns that item n's
//               P.V products have just consumed, so the softmax warps never wait for scores at an item boundary.
//   warps 2-9   two softmax groups (one warp per TMEM lane quarter, one thread per query row) taking chunks alternately:
//               pass 1 row maximum over their chunks (exchanged through shared memory), pass 2 probabilities, dropout,
//               P written over S in place and its TF32 residual into the group's own column block
//   warps 10-13 per item: Q rows (pre-scaled to the log2 domain, raw + residual) into TMEM as the A operand, key classes
//               (valid / padded / beyond the sequence) into shared memory; finished O scaled by 1/rowsum and written out
//               through a swizzled staging tile (coalesced)
//   TMEM columns: S/P [0,256) | P_lo of group g [256 + 64g, +64) | O [384,448): [P.V + P_lo.V | P.V_lo] | Q raw,lo [448,512)
// =====================================================================================================
constexpr int F_NSTG = 4;
constexpr uint32_t F_TILE = 64 * ROWB;       // 8 KB: one [64 x 32] fp32 tile
constexpr uint32_t F_STAGE = 2 * F_TILE;     // raw | residual
constexpr uint32_t F_ROWS = 128 * ROWB;      // 16 KB: the Q rows of one tile
constexpr uint32_t F_OUT = 32 * ROWB;        // 4 KB per operand warp: staging tile for coalesced O stores
constexpr uint32_t F_S = 0, F_PL = 256, F_O = 384, F_Q = 448, F_QL = 480;
constexpr int F_THREADS = 512;

struct TcAttnArgs {
  const int64_t* tok;
  float* out;
  float* stats;
  int64_t ldo;
  int L, LPK, h, NT, mask_mode, items;
  int Lq;  // query rows per sequence (== L unless the queries are a compacted subset: rbm_attn_fwd_lq / rbm_attn_bwd_lq)
  float scale_log2;
  uint32_t thr16;
  float inv_keep;
  uint64_t seed, site;
};

template <bool CAUSAL, bool DROP>
__global__ void __launch_bounds__(F_THREADS, 1) attn_fwd_tc_kernel(const __grid_constant__ CUtensorMap mapQ,
                                                                   const __grid_constant__ CUtensorMap mapK,
                                                                   const __grid_constant__ CUtensorMap mapV, const TcAttnArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t kfull[F_NSTG], ksplit[F_NSTG], kempty[F_NSTG], vfull[F_NSTG], vsplit[F_NSTG], vempty[F_NSTG], s_full[4],
      p_full[2], pl_free[2], q_full, q_free, o_full, o_free, inv_full[2], rows_full, rows_free;
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float kuse[2][256], kfill[2][256];  // per key: 1 = score used as is / the value that replaces it
  __shared__ float xmax[2][128], xsum[2][128], xinv[2][128];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = a.L, LPK = a.LPK;
  const int NU = LPK >> 4, NCH = (NU + 3) >> 2;  // 16-key units; chunks of <= 4 units, sizes as even as possible
  const int n_items = a.items > (int)blockIdx.x ? (a.items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t off_v = F_NSTG * F_STAGE, off_rows = 2 * F_NSTG * F_STAGE, off_out = off_rows + F_ROWS;

  if (threadIdx.x == 0) {
    for (int i = 0; i < F_NSTG; ++i) {
      mbar_init(smem_u32(&kfull[i]), 1);
      mbar_init(smem_u32(&ksplit[i]), 2);
      mbar_init(smem_u32(&kempty[i]), 1);
      mbar_init(smem_u32(&vfull[i]), 1);
      mbar_init(smem_u32(&vsplit[i]), 2);
      mbar_init(smem_u32(&vempty[i]), 1);
      mbar_init(smem_u32(&s_full[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&p_full[i]), 4);
      mbar_init(smem_u32(&pl_free[i]), 1);
      mbar_init(smem_u32(&inv_full[i]), 4);
    }
    mbar_init(smem_u32(&q_full), 4);
    mbar_init(smem_u32(&q_free), 1);
    mbar_init(smem_u32(&o_full), 1);
    mbar_init(smem_u32(&o_free), 4);
    mbar_init(smem_u32(&rows_full), 1);
    mbar_init(smem_u32(&rows_free), 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;
  // Work order shared by producer, split warps and issuer:  K(0,*);  then per item n, per chunk c:  V(n,c), K(n+1,c).
  // Ring slots follow the global chunk counter g = n*NCH + c of each stream.

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapQ) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapK) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapV) : "memory");
      auto item_of = [&](int n, int& b, int& hh, int& mt) {
        const int item = (int)blockIdx.x + n * (int)gridDim.x;
        const int bh = item / a.NT;
        mt = item - bh * a.NT; b = bh / a.h; hh = bh - b * a.h;
      };
      auto issue_rows = [&](int n) {
        int b, hh, mt;
        item_of(n, b, hh, mt);
        if (n >= 1) mbar_wait(smem_u32(&rows_free), (n - 1) & 1);
        mbar_expect_tx(smem_u32(&rows_full), F_ROWS);
        tma_load_3d(smem_base + off_rows, &mapQ, smem_u32(&rows_full), hh * DK, mt * 128, b);
      };
      auto issue_k = [&](int n, int c) {
        int b, hh, mt;
        item_of(n, b, hh, mt);
        const int g = n * NCH + c, s = g % F_NSTG, k0 = ((c * NU) / NCH) << 4;
        if (g >= F_NSTG) mbar_wait(smem_u32(&kempty[s]), ((g / F_NSTG) - 1) & 1);
        mbar_expect_tx(smem_u32(&kfull[s]), F_TILE);
        tma_load_3d(smem_base + s * F_STAGE, &mapK, smem_u32(&kfull[s]), hh * DK, k0, b);
      };
      auto issue_v = [&](int n, int c) {
        int b, hh, mt;
        item_of(n, b, hh, mt);
        const int g = n * NCH + c, s = g % F_NSTG, k0 = ((c * NU) / NCH) << 4;
        if (g >= F_NSTG) mbar_wait(smem_u32(&vempty[s]), ((g / F_NSTG) - 1) & 1);
        mbar_expect_tx(smem_u32(&vfull[s]), F_TILE);
        tma_load_3d(smem_base + off_v + s * F_STAGE, &mapV, smem_u32(&vfull[s]), hh * DK, k0, b);
      };
      if (n_items > 0) {
        issue_rows(0);
        for (int c = 0; c < NCH; ++c) issue_k(0, c);
      }
      for (int n = 0; n < n_items; ++n) {
        if (n + 1 < n_items) issue_rows(n + 1);
        for (int c = 0; c < NCH; ++c) {
          issue_v(n, c);
          if (n + 1 < n_items) issue_k(n + 1, c);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    if (tmem != 0) __trap();  // the CTA owns all 512 columns: literal addresses keep the issue loop on the uniform datapath
    if (elect_one()) {
      constexpr uint32_t tmem = 0;
      const uint32_t idO2 = make_idesc_tf32(128, 2 * DK, 0, 1);  // A from TMEM, [V | V_lo] MN-major, N = 64
      const uint32_t idO1 = make_idesc_tf32(128, DK, 0, 1);
      auto issue_s = [&](int n, int c) {
        const int g = n * NCH + c, s = g % F_NSTG;
        const int k0 = ((c * NU) / NCH) << 4, nh = ((((c + 1) * NU) / NCH) << 4) - k0;
        if (c == 0) mbar_wait(smem_u32(&q_full), n & 1);
        mbar_wait(smem_u32(&kfull[s]), (g / F_NSTG) & 1);
        mbar_wait(smem_u32(&ksplit[s]), (g / F_NSTG) & 1);
        tc_fence_after();
        const uint32_t idS = make_idesc_tf32(128, nh, 0, 0);
        const uint32_t sa = smem_base + s * F_STAGE;
        const uint64_t dK = make_sw128_desc(sa), dKl = make_sw128_desc(sa + F_TILE);
        const uint32_t tS = tmem + F_S + (uint32_t)k0;
#pragma unroll
        for (int k = 0; k < DK / 8; ++k) {
          const uint64_t o = (uint64_t)(k * 2);
          umma_tf32_ts(tS, tmem + F_Q + k * 8, dKl + o, idS, k != 0);
          umma_tf32_ts(tS, tmem + F_QL + k * 8, dK + o, idS, 1);
          umma_tf32_ts(tS, tmem + F_Q + k * 8, dK + o, idS, 1);
        }
        umma_commit(smem_u32(&kempty[s]));
        umma_commit(smem_u32(&s_full[c]));
        if (c == NCH - 1) umma_commit(smem_u32(&q_free));  // Q of this item has been consumed
      };
      auto issue_pv = [&](int n, int c) {
        const int g = n * NCH + c, s = g % F_NSTG, grp = g & 1;
        const int k0 = ((c * NU) / NCH) << 4, nh = ((((c + 1) * NU) / NCH) << 4) - k0;
        mbar_wait(smem_u32(&p_full[grp]), (g >> 1) & 1);
        if (c == 0 && n >= 1) mbar_wait(smem_u32(&o_free), (n - 1) & 1);
        mbar_wait(smem_u32(&vfull[s]), (g / F_NSTG) & 1);
        mbar_wait(smem_u32(&vsplit[s]), (g / F_NSTG) & 1);
        tc_fence_after();
        const uint32_t sa = smem_base + off_v + s * F_STAGE;
        const uint32_t tP = tmem + F_S + (uint32_t)k0, tPl = tmem + F_PL + (uint32_t)grp * 64;
        for (int kk = 0; kk < nh / 8; ++kk) {
          const uint64_t dV2 = make_sw128_desc_mn(sa + kk * 1024, F_TILE);  // second MN block = the residual tile
          const uint64_t dV1 = make_sw128_desc_mn(sa + kk * 1024, 0);
          umma_tf32_ts(tmem + F_O, tP + kk * 8, dV2, idO2, (c | kk) != 0);  // [P.V | P.V_lo]
          umma_tf32_ts(tmem + F_O, tPl + kk * 8, dV1, idO1, 1);             // P_lo.V
        }
        umma_commit(smem_u32(&vempty[s]));
        umma_commit(smem_u32(&pl_free[grp]));
        if (c == NCH - 1) umma_commit(smem_u32(&o_full));
      };
      if (n_items > 0)
        for (int c = 0; c < NCH; ++c) issue_s(0, c);
      for (int n = 0; n < n_items; ++n)
        for (int c = 0; c < NCH; ++c) {
          issue_pv(n, c);
          if (n + 1 < n_items) issue_s(n + 1, c);
        }
    }
    __syncwarp();
  } else if (warp < 10) {
    // ------------------------------------------------------------------------------------------ softmax groups
    const int q = warp & 3, grp = (warp - 2) >> 2;
    const int rl = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const uint32_t thr_hi = a.thr16 << 16;
    const uint64_t site_e = rbm_site(a.site);
    const uint32_t tS = tmem + lane_sel + F_S, tPl = tmem + lane_sel + F_PL + (uint32_t)grp * 64;
    for (int n = 0; n < n_items; ++n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      const int bh = item / a.NT, mt = item - bh * a.NT;
      const int i = mt * 128 + rl;
      const bool warp_live = mt * 128 + q * 32 < a.Lq;  // a warp whose 32 rows all lie beyond the sequence only keeps the hand-shakes going
      const float* ku = kuse[n & 1];
      const float* kf = kfill[n & 1];
      // ---- pass 1: row maximum (log2 domain) over this group's chunks
      float mx = -INFINITY;
      for (int c = 0; c < NCH; ++c) {
        if (((n * NCH + c) & 1) != grp) continue;
        const int k0 = ((c * NU) / NCH) << 4, nh = ((((c + 1) * NU) / NCH) << 4) - k0;
        mbar_wait(smem_u32(&s_full[c]), n & 1);
        tc_fence_after();
        if (warp_live) {
          for (int c0 = 0; c0 < nh; c0 += 16) {
            const int j0 = k0 + c0;
            float v[16];
            tmem_ld16(tS + (uint32_t)j0, v);
#pragma unroll
            for (int jj = 0; jj < 16; jj += 4) {
              const float4 u = ld4(ku + j0 + jj), f = ld4(kf + j0 + jj);
              float x0 = u.x != 0.f ? v[jj] : f.x, x1 = u.y != 0.f ? v[jj + 1] : f.y, x2 = u.z != 0.f ? v[jj + 2] : f.z,
                    x3 = u.w != 0.f ? v[jj + 3] : f.w;
              if (CAUSAL) {
                if (j0 + jj > i) x0 = -INFINITY;
                if (j0 + jj + 1 > i) x1 = -INFINITY;
                if (j0 + jj + 2 > i) x2 = -INFINITY;
                if (j0 + jj + 3 > i) x3 = -INFINITY;
              }
              mx = fmaxf(mx, fmaxf(fmaxf(x0, x1), fmaxf(x2, x3)));
            }
          }
        }
      }
      xmax[grp][rl] = mx;
      named_bar_sync(2 + q, 64);
      mx = fmaxf(xmax[0][rl], xmax[1][rl]);
      const float base = mx == -INFINITY ? 0.f : mx;
      // ---- pass 2: probabilities, dropout, P (raw in place, residual into the group's block)
      float sum = 0.f;
      for (int c = 0; c < NCH; ++c) {
        const int g = n * NCH + c;
        if ((g & 1) != grp) continue;
        const int k0 = ((c * NU) / NCH) << 4, nh = ((((c + 1) * NU) / NCH) << 4) - k0;
        if (g >= 2) {  // the group's previous chunk has been multiplied into O: its residual block is free again
          mbar_wait(smem_u32(&pl_free[grp]), ((g >> 1) - 1) & 1);
          tc_fence_after();
        }
        if (warp_live) {
          for (int c0 = 0; c0 < nh; c0 += 16) {
            const int j0 = k0 + c0;
            uint32_t rs[16];
            tmem_ld16_issue(tS + (uint32_t)j0, rs);
            KeepWords kw;
            if (DROP) kw = attn_keep_words(a.seed, site_e, (uint64_t)bh, i, j0 >> 4);  // overlaps the TMEM read
            float us[16], fs[16];
#pragma unroll
            for (int jj = 0; jj < 16; jj += 4) {
              const float4 u = ld4(ku + j0 + jj), f = ld4(kf + j0 + jj);
              us[jj] = u.x; us[jj + 1] = u.y; us[jj + 2] = u.z; us[jj + 3] = u.w;
              fs[jj] = f.x; fs[jj + 1] = f.y; fs[jj + 2] = f.z; fs[jj + 3] = f.w;
            }
            tmem_ld_wait16(rs);
            float v[16], lo[16];
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              float x = us[jj] != 0.f ? __uint_as_float(rs[jj]) : fs[jj];
              if (CAUSAL && j0 + jj > i) x = -INFINITY;
              float p = ex2(x - base);
              sum += p;
              if (DROP) p = attn_keep_bit(kw, jj, thr_hi) ? p * a.inv_keep : 0.f;
              v[jj] = p;
              lo[jj] = tf32_lo(p);
            }
            tmem_st16(tS + (uint32_t)j0, v);
            tmem_st16(tPl + (uint32_t)c0, lo);
          }
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&p_full[grp]));
      }
      xsum[grp][rl] = sum;
      named_bar_sync(2 + q, 64);
      if (grp == 0) {
        const float inv = 1.f / (xsum[0][rl] + xsum[1][rl]);
        xinv[n & 1][rl] = inv;
        if (i < a.Lq && a.stats) {
          const int64_t sr = ((int64_t)bh * a.Lq + i) * 2;
          a.stats[sr] = mx;
          a.stats[sr + 1] = inv;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&inv_full[n & 1]));
      }
      named_bar_sync(2 + q, 64);  // xmax / xsum are free for the next item
    }
  } else if (warp < 14) {
    // ------------------------------------------------------------------------------------------ operand / output warps
    const int q = warp & 3, rl = q * 32 + lane, t128 = (warp - 10) * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    float* stage = reinterpret_cast<float*>(gen + off_out + (warp - 10) * F_OUT);
    float qv[32];
    float u0 = 0.f, f0 = 0.f, u1 = 0.f, f1 = 0.f;  // classes of keys t128 and t128 + 128 of the item being staged
    auto key_class = [&](int b, int j, float& u, float& f) {
      if (j >= L) { u = 0.f; f = -INFINITY; }                                                  // beyond the sequence
      else if (a.mask_mode == RBM_MASK_KEYPAD && a.tok[(int64_t)b * L + j] == 0) { u = 0.f; f = RBM_PADFILL; }  // padding token: -1e9
      else { u = 1.f; f = 0.f; }
    };
    auto load_item = [&](int n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      const int b = (item / a.NT) / a.h;
      key_class(b, t128, u0, f0);
      key_class(b, t128 + 128, u1, f1);
      mbar_wait(smem_u32(&rows_full), n & 1);
      const float* qs = reinterpret_cast<const float*>(gen + off_rows) + rl * DK;
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        const int sc = ((c >> 2) ^ (rl & 7)) << 2;  // 128-byte swizzle: 16-byte chunk c of row r sits at c ^ (r & 7)
        const float4 x = ld4(qs + sc);
        qv[c] = x.x * a.scale_log2; qv[c + 1] = x.y * a.scale_log2; qv[c + 2] = x.z * a.scale_log2; qv[c + 3] = x.w * a.scale_log2;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&rows_free));
    };
    auto store_o = [&](int n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      const int bh = item / a.NT, mt = item - bh * a.NT, b = bh / a.h, hh = bh - b * a.h;
      mbar_wait(smem_u32(&inv_full[n & 1]), (n >> 1) & 1);
      const float inv = xinv[n & 1][rl];
      mbar_wait(smem_u32(&o_full), n & 1);
      tc_fence_after();
      float* dst = stage + lane * DK;
#pragma unroll
      for (int part = 0; part < 2; ++part) {
        float x[16], y[16];
        tmem_ld16(tmem + lane_sel + F_O + part * 16, x);
        tmem_ld16(tmem + lane_sel + F_O + DK + part * 16, y);
#pragma unroll
        for (int c = 0; c < 16; c += 4) {
          const int ch = part * 4 + (c >> 2);
          st4(dst + ((ch ^ (lane & 7)) << 2), make_float4((x[c] + y[c]) * inv, (x[c + 1] + y[c + 1]) * inv, (x[c + 2] + y[c + 2]) * inv,
                                                          (x[c + 3] + y[c + 3]) * inv));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&o_free));
      const int64_t row0 = (int64_t)b * a.Lq + mt * 128 + q * 32;
      const int rows_ok = a.Lq - (mt * 128 + q * 32);
      float* base = a.out + row0 * a.ldo + hh * DK;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int r = it * 4 + (lane >> 3), ch = lane & 7;
        if (r < rows_ok) st4(base + r * a.ldo + ch * 4, ld4(stage + r * DK + ((ch ^ (r & 7)) << 2)));
      }
      __syncwarp();
    };
    if (n_items > 0) load_item(0);
    for (int n = 0; n < n_items; ++n) {
      kuse[n & 1][t128] = u0; kfill[n & 1][t128] = f0;
      kuse[n & 1][t128 + 128] = u1; kfill[n & 1][t128 + 128] = f1;
      if (n >= 1) {
        mbar_wait(smem_u32(&q_free), (n - 1) & 1);  // every S chunk of the previous item has read its Q
        tc_fence_after();
      }
      {
        float t16[16];
#pragma unroll
        for (int part = 0; part < 2; ++part) {
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = qv[part * 16 + c];
          tmem_st16(tmem + lane_sel + F_Q + part * 16, t16);
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = tf32_lo(t16[c]);
          tmem_st16(tmem + lane_sel + F_QL + part * 16, t16);
        }
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&q_full));
      // O is single-buffered: the previous item's result has to leave before this item's first P.V
      if (n >= 1) store_o(n - 1);
      if (n + 1 < n_items) load_item(n + 1);
    }
    if (n_items > 0) store_o(n_items - 1);
  } else {
    // ------------------------------------------------------------------------------------------ TF32 residual copies
    const int tid = (warp - 14) * 32 + lane;
    auto split = [&](uint64_t* full, uint64_t* done, uint32_t off, int g) {
      const int s = g % F_NSTG;
      mbar_wait(smem_u32(&full[s]), (g / F_NSTG) & 1);
      float* st = reinterpret_cast<float*>(gen + off + (size_t)s * F_STAGE);
      split_lo(st, st + F_TILE / 4, (int)(F_TILE / 16), tid, 64);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&done[s]));
    };
    if (n_items > 0)
      for (int c = 0; c < NCH; ++c) split(kfull, ksplit, 0, c);
    for (int n = 0; n < n_items; ++n)
      for (int c = 0; c < NCH; ++c) {
        split(vfull, vsplit, off_v, n * NCH + c);
        if (n + 1 < n_items) split(kfull, ksplit, 0, (n + 1) * NCH + c);
      }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// =====================================================================================================
// Backward pass A (dQ and delta) on the tensor path: a persistent kernel, one CTA per SM walking the work items
// (sequence, head, 128-query tile).  Every stage of the pipeline belongs to its own warps, and all of them run ahead
// across item boundaries, so TMA latency, operand staging, tensor work, softmax arithmetic and the dQ write-back of
// neighbouring items overlap:
//   warp 0      TMA: keys stream in chunks of <= 64 (multiples of 16) through a 4-stage ring; a stage holds the chunk's
//               K rows twice (K-major for S = Q.K^T, MN-major / 32-byte-atom swizzle for dQ += dS.K) and its V rows
//   warps 14-15 derive the TF32 residual copy of every staged tile (3xTF32)
//   warp 1      issues tcgen05.mma: S and dP of a chunk into the accumulator pair of the chunk's softmax group, then --
//               once that group has replaced them by dS (raw + residual) -- dQ += dS.K with dS as the TMEM A operand
//   warps 2-9   two softmax groups (one warp per TMEM lane quarter, one thread per query row) taking chunks alternately
//   warps 10-13 per item: Q and dO rows (raw + residual) into TMEM as A operands, delta_i = <dO_i, O_i>, key validity;
//               and the finished dQ accumulator (double-buffered) out to HBM
//   TMEM columns: group g: S [128g, +64) | dP [128g + 64, +64);  Q raw,lo [256,320) | dO raw,lo [320,384) |
//                 dQ [384 + 64*(item & 1), +64): columns [0,32) dS.K + dS_lo.K, [32,64) dS.K_lo, added on the way out
// =====================================================================================================
constexpr int CW = 64;        // columns of one chunk accumulator / key rows of one staged tile
constexpr int A_NSTG = 3;
constexpr uint32_t A_TILE = CW * ROWB;      // 8 KB
constexpr uint32_t A_STAGE = 6 * A_TILE;    // Kk | Vk | Km raw, then the three residual copies
constexpr uint32_t A_GRP = 128, A_DP = 64, A_Q = 256, A_QL = 288, A_DO = 320, A_DOL = 352, A_DQ = 384;
constexpr int A_THREADS = 512;
constexpr uint32_t A_ROWS = 128 * ROWB;     // 16 KB: the Q / dO / O rows of one 128-query tile

struct TcBwdArgs {
  const float *q, *o, *dout, *stats;
  float *dq, *delta;
  int64_t ldq, ldo, lddo, lddq;
  const int64_t* tok;
  int L, LPK, h, NT, mask_mode, items;
  int Lq;  // query rows per sequence (== L unless the queries are a compacted subset: rbm_attn_fwd_lq / rbm_attn_bwd_lq)
  float scale, scale_log2;
  uint32_t thr16;
  float inv_keep;
  uint64_t seed, site;
};

template <bool CAUSAL, bool DROP>
__global__ void __launch_bounds__(A_THREADS, 1) attn_bwd_dq_tc_kernel(const __grid_constant__ CUtensorMap mapKk,
                                                                      const __grid_constant__ CUtensorMap mapKm,
                                                                      const __grid_constant__ CUtensorMap mapVk,
                                                                      const __grid_constant__ CUtensorMap mapQ,
                                                                      const __grid_constant__ CUtensorMap mapDO,
                                                                      const __grid_constant__ CUtensorMap mapO, const TcBwdArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[A_NSTG], split_bar[A_NSTG], empty_bar[A_NSTG], s_full[2], ds_full[2], ops_free, ops_full,
      dq_full[2], dq_free[2], rows_full, rows_free;
  __shared__ uint32_t tmem_base_slot;
  __shared__ __align__(16) float kvalid[2][256];  // 1 = key takes part (inside the sequence and not a padding token)
  __shared__ float xdelta[2][128];

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = a.L, LPK = a.LPK;
  const int NU = LPK >> 4, NCH = (NU + 3) >> 2;  // 16-key units; chunks of <= 4 units, sizes as even as possible
  const int n_items = a.items > (int)blockIdx.x ? (a.items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const int n_chunks = n_items * NCH;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (smem_base - smem_u32(smem_raw));

  if (threadIdx.x == 0) {
    for (int i = 0; i < A_NSTG; ++i) {
      mbar_init(smem_u32(&full_bar[i]), 1);
      mbar_init(smem_u32(&split_bar[i]), 2);
      mbar_init(smem_u32(&empty_bar[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&ds_full[i]), 4);
      mbar_init(smem_u32(&dq_full[i]), 1);
      mbar_init(smem_u32(&dq_free[i]), 4);
    }
    mbar_init(smem_u32(&ops_free), 1);
    mbar_init(smem_u32(&ops_full), 4);
    mbar_init(smem_u32(&rows_full), 1);
    mbar_init(smem_u32(&rows_free), 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapKk) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapKm) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapVk) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapQ) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapDO) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapO) : "memory");
      // the Q / dO / O rows of an item land in one single-buffered 48 KB area (the operand warps copy them to registers
      // as soon as they arrive); a tile's rows beyond the sequence are zero-filled by TMA
      auto issue_rows = [&](int n) {
        const int item = (int)blockIdx.x + n * (int)gridDim.x;
        const int bh = item / a.NT, mt = item - bh * a.NT, b = bh / a.h, hh = bh % a.h;
        if (n >= 1) mbar_wait(smem_u32(&rows_free), (n - 1) & 1);
        const uint32_t bar = smem_u32(&rows_full), dst = smem_base + A_NSTG * A_STAGE;
        mbar_expect_tx(bar, 3 * A_ROWS);
        tma_load_3d(dst, &mapQ, bar, hh * DK, mt * 128, b);
        tma_load_3d(dst + A_ROWS, &mapDO, bar, hh * DK, mt * 128, b);
        tma_load_3d(dst + 2 * A_ROWS, &mapO, bar, hh * DK, mt * 128, b);
      };
      if (n_items > 0) issue_rows(0);
      int g = 0;
      for (int n = 0; n < n_items; ++n) {
        const int item = (int)blockIdx.x + n * (int)gridDim.x;
        const int bh = item / a.NT, b = bh / a.h, hh = bh % a.h;
        for (int c = 0; c < NCH; ++c, ++g) {
          const int s = g % A_NSTG, k0 = ((c * NU) / NCH) << 4;
          if (g >= A_NSTG) mbar_wait(smem_u32(&empty_bar[s]), ((g / A_NSTG) - 1) & 1);
          const uint32_t bar = smem_u32(&full_bar[s]), sa = smem_base + s * A_STAGE;
          mbar_expect_tx(bar, 3 * A_TILE);
          tma_load_3d(sa, &mapKk, bar, hh * DK, k0, b);
          tma_load_3d(sa + A_TILE, &mapVk, bar, hh * DK, k0, b);
          tma_load_3d(sa + 2 * A_TILE, &mapKm, bar, hh * DK, k0, b);
        }
        if (n + 1 < n_items) issue_rows(n + 1);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    // The CTA owns all 512 TMEM columns, so the allocation starts at column 0, lane 0: using the literal keeps every
    // operand of the issue loop on the uniform datapath (a value read back from shared memory would not be).
    if (tmem != 0) __trap();
    if (elect_one()) {
    constexpr uint32_t tmem = 0;
    // All 32 lanes run the loop in lockstep; one elected lane issues each tcgen05 instruction.  A tcgen05.mma of this
    // size costs the issuing warp (and the pipe) ~64 cycles whatever its N <= 128, so the count of instructions is what
    // matters: the two products that share the A operand dS_raw run as one N = 64 instruction against [K_raw | K_lo].
    const uint32_t idQ2 = make_idesc_tf32(128, 2 * DK, 0, 1);  // dQ: A from TMEM, [K | K_lo] MN-major, N = 64
    const uint32_t idQ1 = make_idesc_tf32(128, DK, 0, 1);
    auto issue_dq = [&](int g) {
      const int n = g / NCH, c = g - n * NCH, s = g % A_NSTG;
      const int k0 = ((c * NU) / NCH) << 4, nh = ((((c + 1) * NU) / NCH) << 4) - k0;
      const uint32_t tS = tmem + (uint32_t)(g & 1) * A_GRP, tP = tS + A_DP, tD = tmem + A_DQ + (uint32_t)(n & 1) * (2 * DK);
      const uint32_t sa = smem_base + s * A_STAGE;
      mbar_wait(smem_u32(&ds_full[g & 1]), (g >> 1) & 1);
      if (c == 0 && n >= 2) mbar_wait(smem_u32(&dq_free[n & 1]), ((n >> 1) - 1) & 1);
      tc_fence_after();
      for (int kk = 0; kk < nh / 8; ++kk) {
        const uint64_t dKm2 = make_sw128_desc_mn(sa + 2 * A_TILE + kk * 1024, 3 * A_TILE);  // second MN block = the residual tile
        const uint64_t dKm = make_sw128_desc_mn(sa + 2 * A_TILE + kk * 1024, 0);
        umma_tf32_ts(tD, tS + kk * 8, dKm2, idQ2, (c | kk) != 0);  // [dS.K | dS.K_lo]
        umma_tf32_ts(tD, tP + kk * 8, dKm, idQ1, 1);               // dS_lo.K
      }
      umma_commit(smem_u32(&empty_bar[s]));
      if (c == NCH - 1) umma_commit(smem_u32(&dq_full[n & 1]));
    };
    int g = 0;
    for (int n = 0; n < n_items; ++n) {
      for (int c = 0; c < NCH; ++c, ++g) {
        if (g >= 2) issue_dq(g - 2);  // frees this group's accumulators (the tensor pipe runs in order)
        const int s = g % A_NSTG;
        const int k0 = ((c * NU) / NCH) << 4, nh = ((((c + 1) * NU) / NCH) << 4) - k0;
        if (c == 0) mbar_wait(smem_u32(&ops_full), n & 1);
        mbar_wait(smem_u32(&full_bar[s]), (g / A_NSTG) & 1);
        mbar_wait(smem_u32(&split_bar[s]), (g / A_NSTG) & 1);
        tc_fence_after();
        const uint32_t tS = tmem + (uint32_t)(g & 1) * A_GRP, tP = tS + A_DP;
        const uint32_t idS = make_idesc_tf32(128, nh, 0, 0);
        const uint32_t sa = smem_base + s * A_STAGE;
        const uint64_t dK = make_sw128_desc(sa), dKl = make_sw128_desc(sa + 3 * A_TILE);
        const uint64_t dV = make_sw128_desc(sa + A_TILE), dVl = make_sw128_desc(sa + 4 * A_TILE);
#pragma unroll
        for (int k = 0; k < DK / 8; ++k) {
          const uint64_t o = (uint64_t)(k * 2);
          umma_tf32_ts(tS, tmem + A_Q + k * 8, dKl + o, idS, k != 0);
          umma_tf32_ts(tS, tmem + A_QL + k * 8, dK + o, idS, 1);
          umma_tf32_ts(tS, tmem + A_Q + k * 8, dK + o, idS, 1);
        }
#pragma unroll
        for (int k = 0; k < DK / 8; ++k) {
          const uint64_t o = (uint64_t)(k * 2);
          umma_tf32_ts(tP, tmem + A_DO + k * 8, dVl + o, idS, k != 0);
          umma_tf32_ts(tP, tmem + A_DOL + k * 8, dV + o, idS, 1);
          umma_tf32_ts(tP, tmem + A_DO + k * 8, dV + o, idS, 1);
        }
        umma_commit(smem_u32(&s_full[g & 1]));
        if (c == NCH - 1) umma_commit(smem_u32(&ops_free));  // Q / dO of this item have been consumed
      }
    }
    for (int gg = n_chunks >= 2 ? n_chunks - 2 : 0; gg < n_chunks; ++gg) issue_dq(gg);
    }
    __syncwarp();
  } else if (warp < 10) {
    // ------------------------------------------------------------------------------------------ softmax groups
    const int q = warp & 3, grp = (warp - 2) >> 2;
    const int rl = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const uint32_t thr_hi = a.thr16 << 16;
    const uint64_t site_e = rbm_site(a.site);
    const uint32_t tS = tmem + lane_sel + (uint32_t)grp * A_GRP, tP = tS + A_DP;
    int cur_n = -1, bh = 0, i = 0;
    bool warp_live = false;
    float mx = 0.f, inv = 0.f, ndelta = 0.f;
    for (int g = grp; g < n_chunks; g += 2) {
      const int n = g / NCH, c = g - n * NCH;
      const int k0 = ((c * NU) / NCH) << 4, nh = ((((c + 1) * NU) / NCH) << 4) - k0;
      const bool new_item = n != cur_n;
      if (new_item) {  // the row statistics do not depend on the barrier: fetch them ahead of the wait
        cur_n = n;
        const int item = (int)blockIdx.x + n * (int)gridDim.x;
        bh = item / a.NT;
        const int mt = item - bh * a.NT;
        i = mt * 128 + rl;
        warp_live = mt * 128 + q * 32 < a.Lq;  // a warp whose 32 rows all lie beyond the sequence has nothing to do
        // rows beyond the sequence hold zero operands: mx = 0, inv = 0 makes every dS of theirs an exact zero
        mx = 0.f; inv = 0.f;
        if (i < a.Lq) {
          const int64_t sr = ((int64_t)bh * a.Lq + i) * 2;
          mx = a.stats[sr];
          inv = a.stats[sr + 1];
        }
      }
      mbar_wait(smem_u32(&s_full[grp]), (g >> 1) & 1);
      tc_fence_after();
      if (new_item) ndelta = -xdelta[n & 1][rl];
      if (warp_live) {
        const float* kvp = kvalid[n & 1];
        for (int c0 = 0; c0 < nh; c0 += 16) {
          uint32_t rs[16], rd[16];
          tmem_ld16_issue(tS + (uint32_t)c0, rs);
          tmem_ld16_issue(tP + (uint32_t)c0, rd);
          const int j0 = k0 + c0;
          KeepWords kw;
          if (DROP) kw = attn_keep_words(a.seed, site_e, (uint64_t)bh, i, j0 >> 4);  // overlaps the TMEM reads
          float kv[16];
#pragma unroll
          for (int jj = 0; jj < 16; jj += 4) {
            const float4 t = ld4(kvp + j0 + jj);
            kv[jj] = t.x; kv[jj + 1] = t.y; kv[jj + 2] = t.z; kv[jj + 3] = t.w;
          }
          tmem_ld_wait16(rs);
          tmem_ld_wait16(rd);
          float sv[16], lo[16];
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) {
            const float p = ex2(__uint_as_float(rs[jj]) - mx) * inv;
            const float dpv = __uint_as_float(rd[jj]);
            float t;
            if (DROP) t = attn_keep_bit(kw, jj, thr_hi) ? fmaf(dpv, a.inv_keep, ndelta) : ndelta;
            else t = dpv + ndelta;
            bool live = kv[jj] != 0.f;  // no score gradient through a padded key (its probability is an exact zero)
            if (CAUSAL) live = live && (j0 + jj <= i);
            const float ds = live ? p * t : 0.f;
            sv[jj] = ds;
            lo[jj] = tf32_lo(ds);
          }
          tmem_st16(tS + (uint32_t)c0, sv);
          tmem_st16(tP + (uint32_t)c0, lo);
        }
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&ds_full[grp]));
    }
  } else if (warp < 14) {
    // ------------------------------------------------------------------------------------------ operand / dQ warps
    const int q = warp & 3, rl = q * 32 + lane, t128 = (warp - 10) * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    float qv[32], dv[32];
    float dl = 0.f;
    bool kval0 = false, kval1 = false;  // validity of keys t128 and t128 + 128 of the item being staged
    // this thread's Q, dO, O rows out of the TMA tiles (128-byte swizzle: 16-byte chunk c of row r sits at c ^ (r & 7))
    auto load_rows = [&](int n) {
      {
        const int item = (int)blockIdx.x + n * (int)gridDim.x;
        const int b = (item / a.NT) / a.h;
        const bool keypad = a.mask_mode == RBM_MASK_KEYPAD;
        kval0 = t128 < L && !(keypad && a.tok[(int64_t)b * L + t128] == 0);
        kval1 = t128 + 128 < L && !(keypad && a.tok[(int64_t)b * L + t128 + 128] == 0);
      }
      mbar_wait(smem_u32(&rows_full), n & 1);
      const float* qs = reinterpret_cast<const float*>(gen + A_NSTG * A_STAGE) + rl * DK;
      const float* ds = qs + A_ROWS / 4;
      const float* os = ds + A_ROWS / 4;
      dl = 0.f;
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        const int sc = ((c >> 2) ^ (rl & 7)) << 2;
        const float4 x = ld4(qs + sc), y = ld4(ds + sc), z = ld4(os + sc);
        qv[c] = x.x * a.scale_log2; qv[c + 1] = x.y * a.scale_log2; qv[c + 2] = x.z * a.scale_log2; qv[c + 3] = x.w * a.scale_log2;
        dv[c] = y.x; dv[c + 1] = y.y; dv[c + 2] = y.z; dv[c + 3] = y.w;
        dl = fmaf(y.x, z.x, dl); dl = fmaf(y.y, z.y, dl); dl = fmaf(y.z, z.z, dl); dl = fmaf(y.w, z.w, dl);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&rows_free));
    };
    auto store_dq = [&](int n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      const int bh = item / a.NT, mt = item - bh * a.NT, b = bh / a.h, hh = bh - b * a.h;
      const int i = mt * 128 + rl;
      mbar_wait(smem_u32(&dq_full[n & 1]), (n >> 1) & 1);
      tc_fence_after();
      float o[32];
      {  // dQ = [dS.K + dS_lo.K] + [dS.K_lo]
        float o1[32];
        tmem_ld32(tmem + lane_sel + A_DQ + (uint32_t)(n & 1) * (2 * DK), o);
        tmem_ld32(tmem + lane_sel + A_DQ + (uint32_t)(n & 1) * (2 * DK) + DK, o1);
#pragma unroll
        for (int jj = 0; jj < 32; ++jj) o[jj] += o1[jj];
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&dq_free[n & 1]));
      if (i < a.Lq) {
        float* dst = a.dq + ((int64_t)b * a.Lq + i) * a.lddq + hh * DK;
#pragma unroll
        for (int jj = 0; jj < 32; jj += 4)
          st4(dst + jj, make_float4(o[jj] * a.scale, o[jj + 1] * a.scale, o[jj + 2] * a.scale, o[jj + 3] * a.scale));
      }
    };
    if (n_items > 0) load_rows(0);
    for (int n = 0; n < n_items; ++n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      const int bh = item / a.NT, mt = item - bh * a.NT;
      const int i = mt * 128 + rl;
      // key validity of this item's sequence, delta of its rows
      kvalid[n & 1][t128] = kval0 ? 1.f : 0.f;
      kvalid[n & 1][t128 + 128] = kval1 ? 1.f : 0.f;
      xdelta[n & 1][rl] = dl;
      if (i < a.Lq) a.delta[(int64_t)bh * a.Lq + i] = dl;
      if (n >= 1) {
        mbar_wait(smem_u32(&ops_free), (n - 1) & 1);  // every S / dP of the previous item has read its Q / dO
        tc_fence_after();
      }
      {
        float t16[16];
#pragma unroll
        for (int part = 0; part < 2; ++part) {
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = qv[part * 16 + c];
          tmem_st16(tmem + lane_sel + A_Q + part * 16, t16);
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = tf32_lo(t16[c]);
          tmem_st16(tmem + lane_sel + A_QL + part * 16, t16);
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = dv[part * 16 + c];
          tmem_st16(tmem + lane_sel + A_DO + part * 16, t16);
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = tf32_lo(t16[c]);
          tmem_st16(tmem + lane_sel + A_DOL + part * 16, t16);
        }
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&ops_full));
      if (n + 1 < n_items) load_rows(n + 1);  // in flight while this item is being worked on
      if (n >= 1) store_dq(n - 1);
    }
    if (n_items > 0) store_dq(n_items - 1);
  } else {
    // ------------------------------------------------------------------------------------------ TF32 residual copies
    const int tid = (warp - 14) * 32 + lane;  // warps 14, 15
    for (int g = 0; g < n_chunks; ++g) {
      const int s = g % A_NSTG;
      mbar_wait(smem_u32(&full_bar[s]), (g / A_NSTG) & 1);
      float* st = reinterpret_cast<float*>(gen + (size_t)s * A_STAGE);
      split_lo(st, st + 3 * A_TILE / 4, (int)(3 * A_TILE / 16), tid, 64);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&split_bar[s]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// =====================================================================================================
// Backward pass B (dK, dV) on the tensor path: persistent, one CTA per SM walking the work items (sequence, head,
// 128-key tile); accumulator rows = keys.  Same division of labour as pass A:
//   warp 0      TMA: the item's K and V rows (one 128-row tile each) and the query stream -- sub-chunks of 32 queries
//               through a 4-stage ring, every sub-chunk twice: Q and dO as K-major tiles (B operands of S^T = K.Q^T and
//               dP^T = V.dO^T) and as MN-major tiles (B operands of dK += dS^T.Q and dV += P~^T.dO)
//   warps 14-15 TF32 residual copy of every staged tile
//   warp 1      tcgen05.mma issue (K and V rows are the TMEM A operands of S^T / dP^T; dS^T and P~^T, written back by
//               the softmax warps, are the TMEM A operands of the dK / dV updates)
//   warps 2-9   two softmax groups (one warp per TMEM lane quarter, one thread per key) taking sub-chunks alternately,
//               each with its own S^T / dP^T / P~^T column block
//   warps 10-13 per item: K and V rows (raw + residual) into TMEM, the row statistics (max, 1/sum, delta) of the
//               sequence into shared memory; finished dK / dV out to HBM through a swizzled staging tile (coalesced)
//   TMEM columns: K raw,lo [0,64) | V raw,lo [64,128) | group g at 128 + 128g: S^T [+0,32) dP^T [+32,64) P~ [+64,96)
//                 P~_lo [+96,128) | dK [384,448) | dV [448,512); dK / dV hold [x.B + x_lo.B | x.B_lo], added on the way out
// =====================================================================================================
constexpr int SQ = 32;                      // queries per sub-chunk / ring stage
constexpr int B_NSTG = 4;
constexpr uint32_t B_TILE = SQ * ROWB;      // 4 KB: one [32 x 32] fp32 tile
constexpr uint32_t B_STAGE = 8 * B_TILE;    // Qk, Qm, dOk, dOm (raw) + the same four (residual)
constexpr uint32_t B_ROWS = 128 * ROWB;     // 16 KB: the K (or V) rows of one 128-key tile
constexpr uint32_t B_OUT = 32 * ROWB;       // 4 KB: staging tile for coalesced stores (two per operand warp: dK, dV)
constexpr uint32_t B_K = 0, B_KL = 32, B_V = 64, B_VL = 96, B_GRP0 = 128, B_GRP = 128, B_DPT = 32, B_P = 64, B_PL = 96, B_DK = 384,
                   B_DV = 448;
constexpr int B_THREADS = 512;

struct TcBwdKvArgs {
  const float *stats, *delta;
  float *dk, *dv;
  int64_t lddk, lddv;
  const int64_t* tok;
  int L, LPK, h, NT, mask_mode, items;
  int Lq;  // query rows per sequence (== L unless the queries are a compacted subset: rbm_attn_fwd_lq / rbm_attn_bwd_lq)
  float scale, scale_log2;
  uint32_t thr16;
  float inv_keep;
  uint64_t seed, site;
};

template <bool CAUSAL, bool DROP>
__global__ void __launch_bounds__(B_THREADS, 1) attn_bwd_dkv_tc_kernel(const __grid_constant__ CUtensorMap mapQk,
                                                                       const __grid_constant__ CUtensorMap mapQm,
                                                                       const __grid_constant__ CUtensorMap mapOk,
                                                                       const __grid_constant__ CUtensorMap mapOm,
                                                                       const __grid_constant__ CUtensorMap mapK,
                                                                       const __grid_constant__ CUtensorMap mapV, const TcBwdKvArgs a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[B_NSTG], split_bar[B_NSTG], empty_bar[B_NSTG], s_full[2], ds_full[2], ops_free, ops_full,
      dkv_full, dkv_free, rows_full, rows_free;
  __shared__ uint32_t tmem_base_slot;
  __shared__ float st_m[2][256], st_i[2][256], st_d[2][256];  // per query: row max (log2 domain), 1/rowsum, delta

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = a.L, LPK = a.LPK;
  const int NSC = (LPK + SQ - 1) / SQ;  // sub-chunks per sequence
  const int n_items = a.items > (int)blockIdx.x ? (a.items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t off_rows = B_NSTG * B_STAGE, off_out = off_rows + 2 * B_ROWS;
  // causal: queries before a key tile never attend to it
  auto first_chunk = [&](int kt) { return CAUSAL ? (kt * 128) / SQ : 0; };

  if (threadIdx.x == 0) {
    for (int i = 0; i < B_NSTG; ++i) {
      mbar_init(smem_u32(&full_bar[i]), 1);
      mbar_init(smem_u32(&split_bar[i]), 2);
      mbar_init(smem_u32(&empty_bar[i]), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(smem_u32(&s_full[i]), 1);
      mbar_init(smem_u32(&ds_full[i]), 4);
    }
    mbar_init(smem_u32(&ops_free), 1);
    mbar_init(smem_u32(&ops_full), 4);
    mbar_init(smem_u32(&dkv_full), 1);
    mbar_init(smem_u32(&dkv_free), 4);
    mbar_init(smem_u32(&rows_full), 1);
    mbar_init(smem_u32(&rows_free), 4);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapQk) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapQm) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapOk) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapOm) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapK) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&mapV) : "memory");
      auto issue_rows = [&](int n) {
        const int item = (int)blockIdx.x + n * (int)gridDim.x;
        const int bh = item / a.NT, kt = item - bh * a.NT, b = bh / a.h, hh = bh % a.h;
        if (n >= 1) mbar_wait(smem_u32(&rows_free), (n - 1) & 1);
        const uint32_t bar = smem_u32(&rows_full), dst = smem_base + off_rows;
        mbar_expect_tx(bar, 2 * B_ROWS);
        tma_load_3d(dst, &mapK, bar, hh * DK, kt * 128, b);
        tma_load_3d(dst + B_ROWS, &mapV, bar, hh * DK, kt * 128, b);
      };
      if (n_items > 0) issue_rows(0);
      int g = 0;
      for (int n = 0; n < n_items; ++n) {
        const int item = (int)blockIdx.x + n * (int)gridDim.x;
        const int bh = item / a.NT, kt = item - bh * a.NT, b = bh / a.h, hh = bh % a.h;
        for (int c = first_chunk(kt); c < NSC; ++c, ++g) {
          const int s = g % B_NSTG;
          if (g >= B_NSTG) mbar_wait(smem_u32(&empty_bar[s]), ((g / B_NSTG) - 1) & 1);
          const uint32_t bar = smem_u32(&full_bar[s]), sa = smem_base + s * B_STAGE;
          mbar_expect_tx(bar, 4 * B_TILE);
          tma_load_3d(sa + 0 * B_TILE, &mapQk, bar, hh * DK, c * SQ, b);
          tma_load_3d(sa + 1 * B_TILE, &mapQm, bar, hh * DK, c * SQ, b);
          tma_load_3d(sa + 2 * B_TILE, &mapOk, bar, hh * DK, c * SQ, b);
          tma_load_3d(sa + 3 * B_TILE, &mapOm, bar, hh * DK, c * SQ, b);
        }
        if (n + 1 < n_items) issue_rows(n + 1);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------------------------------ MMA issuer
    if (tmem != 0) __trap();  // the CTA owns all 512 columns: literal addresses keep the issue loop on the uniform datapath
    if (elect_one()) {
      constexpr uint32_t tmem = 0;
      const uint32_t idA2 = make_idesc_tf32(128, 2 * DK, 0, 1);  // A from TMEM, [B | B_lo] MN-major, N = 64
      const uint32_t idA1 = make_idesc_tf32(128, DK, 0, 1);
      // the two most recent sub-chunks (one per group) whose dK / dV update is still to be issued
      int p_g[2] = {-1, -1}, p_nq[2] = {0, 0}, p_n[2] = {0, 0};
      bool p_first[2] = {false, false}, p_last[2] = {false, false};
      auto issue_dkv = [&](int grp) {
        const int g = p_g[grp], nq = p_nq[grp], n = p_n[grp], s = g % B_NSTG;
        const uint32_t tG = tmem + B_GRP0 + (uint32_t)grp * B_GRP;
        const uint32_t sa = smem_base + s * B_STAGE;
        mbar_wait(smem_u32(&ds_full[grp]), (g >> 1) & 1);
        if (p_first[grp] && n >= 1) mbar_wait(smem_u32(&dkv_free), (n - 1) & 1);
        tc_fence_after();
        for (int kk = 0; kk < nq / 8; ++kk) {
          const uint64_t dQ2 = make_sw128_desc_mn(sa + 1 * B_TILE + kk * 1024, 4 * B_TILE);  // second MN block = the residual tile
          const uint64_t dQ1 = make_sw128_desc_mn(sa + 1 * B_TILE + kk * 1024, 0);
          const uint64_t dO2 = make_sw128_desc_mn(sa + 3 * B_TILE + kk * 1024, 4 * B_TILE);
          const uint64_t dO1 = make_sw128_desc_mn(sa + 3 * B_TILE + kk * 1024, 0);
          const uint32_t acc = !(p_first[grp] && kk == 0);
          umma_tf32_ts(tmem + B_DK, tG + kk * 8, dQ2, idA2, acc);          // [dS^T.Q | dS^T.Q_lo]
          umma_tf32_ts(tmem + B_DK, tG + B_DPT + kk * 8, dQ1, idA1, 1);    // dS^T_lo.Q
          umma_tf32_ts(tmem + B_DV, tG + B_P + kk * 8, dO2, idA2, acc);    // [P~^T.dO | P~^T.dO_lo]
          umma_tf32_ts(tmem + B_DV, tG + B_PL + kk * 8, dO1, idA1, 1);     // P~^T_lo.dO
        }
        umma_commit(smem_u32(&empty_bar[s]));
        if (p_last[grp]) umma_commit(smem_u32(&dkv_full));
        p_g[grp] = -1;
      };
      int g = 0;
      for (int n = 0; n < n_items; ++n) {
        const int item = (int)blockIdx.x + n * (int)gridDim.x;
        const int kt = item % a.NT;
        const int c0 = first_chunk(kt);
        for (int c = c0; c < NSC; ++c, ++g) {
          const int grp = g & 1, s = g % B_NSTG;
          if (p_g[grp] >= 0) issue_dkv(grp);  // frees this group's column block (the tensor pipe runs in order)
          const int nq = LPK - c * SQ < SQ ? LPK - c * SQ : SQ;  // valid (16-multiple) queries of this sub-chunk
          if (c == c0) mbar_wait(smem_u32(&ops_full), n & 1);
          mbar_wait(smem_u32(&full_bar[s]), (g / B_NSTG) & 1);
          mbar_wait(smem_u32(&split_bar[s]), (g / B_NSTG) & 1);
          tc_fence_after();
          const uint32_t tG = tmem + B_GRP0 + (uint32_t)grp * B_GRP;
          const uint32_t idS = make_idesc_tf32(128, nq, 0, 0);
          const uint32_t sa = smem_base + s * B_STAGE, sl = sa + 4 * B_TILE;
          const uint64_t dQk = make_sw128_desc(sa + 0 * B_TILE), dQkl = make_sw128_desc(sl + 0 * B_TILE);
          const uint64_t dOk = make_sw128_desc(sa + 2 * B_TILE), dOkl = make_sw128_desc(sl + 2 * B_TILE);
#pragma unroll
          for (int k = 0; k < DK / 8; ++k) {
            const uint64_t o = (uint64_t)(k * 2);
            umma_tf32_ts(tG, tmem + B_K + k * 8, dQkl + o, idS, k != 0);
            umma_tf32_ts(tG, tmem + B_KL + k * 8, dQk + o, idS, 1);
            umma_tf32_ts(tG, tmem + B_K + k * 8, dQk + o, idS, 1);
          }
#pragma unroll
          for (int k = 0; k < DK / 8; ++k) {
            const uint64_t o = (uint64_t)(k * 2);
            umma_tf32_ts(tG + B_DPT, tmem + B_V + k * 8, dOkl + o, idS, k != 0);
            umma_tf32_ts(tG + B_DPT, tmem + B_VL + k * 8, dOk + o, idS, 1);
            umma_tf32_ts(tG + B_DPT, tmem + B_V + k * 8, dOk + o, idS, 1);
          }
          umma_commit(smem_u32(&s_full[grp]));
          if (c == NSC - 1) umma_commit(smem_u32(&ops_free));  // K / V of this item have been consumed
          p_g[grp] = g; p_nq[grp] = nq; p_n[grp] = n; p_first[grp] = false; p_last[grp] = false;
          if (c == c0) p_first[grp] = true;
          if (c == NSC - 1) p_last[grp] = true;
        }
      }
      // drain in issue order
      if (p_g[0] >= 0 && p_g[1] >= 0) {
        const int firstg = p_g[0] < p_g[1] ? 0 : 1;
        issue_dkv(firstg);
        issue_dkv(firstg ^ 1);
      } else if (p_g[0] >= 0) {
        issue_dkv(0);
      } else if (p_g[1] >= 0) {
        issue_dkv(1);
      }
    }
    __syncwarp();
  } else if (warp < 10) {
    // ------------------------------------------------------------------------------------------ softmax groups
    const int q = warp & 3, grp = (warp - 2) >> 2;
    const int rl = q * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    const uint32_t tG = tmem + lane_sel + B_GRP0 + (uint32_t)grp * B_GRP;
    // dropout: lanes {l, l^1, l^8, l^9} hold keys that share their Philox calls; each computes two of the eight
    const int wq = (lane & 1) | (((lane >> 3) & 1) << 1);
    const uint64_t site_e = rbm_site(a.site);
    int g = 0;
    for (int n = 0; n < n_items; ++n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      const int bh = item / a.NT, kt = item - bh * a.NT, b = bh / a.h;
      const int j = kt * 128 + rl;  // this thread's key
      const bool warp_live = kt * 128 + q * 32 < L;
      // a padded key keeps the reference's score of -1e9: probability 0, unless the whole row is padding (then the
      // row is uniform and still feeds dV); no score gradient flows through it either way
      const bool jpad = j < L && a.mask_mode == RBM_MASK_KEYPAD && a.tok[(int64_t)b * L + j] == 0;
      const bool jin = j < L;
      const int e_j = j & 1, nb_j = (j >> 3) & 1, t_j = (j & 7) >> 1, np_j = j >> 4;
      const float* sm = st_m[n & 1];
      const float* si = st_i[n & 1];
      const float* sd = st_d[n & 1];
      for (int c = first_chunk(kt); c < NSC; ++c, ++g) {
        if ((g & 1) != grp) continue;
        const int nq = LPK - c * SQ < SQ ? LPK - c * SQ : SQ;
        mbar_wait(smem_u32(&s_full[grp]), (g >> 1) & 1);
        tc_fence_after();
        if (warp_live) {
          for (int c0 = 0; c0 < nq; c0 += 16) {
            uint32_t rs[16], rd[16];
            tmem_ld16_issue(tG + (uint32_t)c0, rs);
            tmem_ld16_issue(tG + B_DPT + (uint32_t)c0, rd);
            const int i0 = c * SQ + c0;  // 16 consecutive queries, one Philox "tile"
            uint32_t w0[8], w1[8];       // per query-in-octet g: the two words (rh = 0, 1) that hold this key's fields
            if (DROP) {
              uint4 ca = rbm_philox_drop(a.seed, site_e, rbm_attn_call((uint64_t)bh, i0 >> 4, 2 * wq + 0, t_j, np_j));
              uint4 cb = rbm_philox_drop(a.seed, site_e, rbm_attn_call((uint64_t)bh, i0 >> 4, 2 * wq + 1, t_j, np_j));
#pragma unroll
              for (int gq = 0; gq < 8; ++gq) {
                // call of query-octet position gq is owned by the lane whose (bit0, bit3) = ((gq>>1)&1, (gq>>2)&1); the
                // requester picks the words of ITS key parity e: word index = rh*2 + e
                const int src = (lane & ~9) | ((gq >> 1) & 1) | (((gq >> 2) & 1) << 3);
                const uint4 cc = (gq & 1) ? cb : ca;
                const uint32_t rx = __shfl_sync(0xffffffffu, cc.x, src), ry = __shfl_sync(0xffffffffu, cc.y, src);
                const uint32_t rz = __shfl_sync(0xffffffffu, cc.z, src), rw = __shfl_sync(0xffffffffu, cc.w, src);
                w0[gq] = e_j ? ry : rx;
                w1[gq] = e_j ? rw : rz;
              }
            }
            tmem_ld_wait16(rs);
            tmem_ld_wait16(rd);
            float sv[16], dlo[16], t16[16];
#pragma unroll
            for (int ii = 0; ii < 16; ++ii) {
              const int i = i0 + ii;
              bool live = jin;
              if (CAUSAL) live = live && (j <= i);
              // queries beyond the sequence hold zero rows and zero statistics: p = 2^0 * 0
              const float x = jpad ? RBM_PADFILL : __uint_as_float(rs[ii]);
              const float p = live ? ex2(x - sm[i]) * si[i] : 0.f;
              float mk = 1.f;
              if (DROP) {
                const uint32_t word = (ii & 8) ? w1[ii & 7] : w0[ii & 7];  // rh = (i >> 3) & 1
                const uint32_t fld = nb_j ? (word >> 16) : (word & 0xffffu);
                mk = fld >= a.thr16 ? a.inv_keep : 0.f;
              }
              const float ds = jpad ? 0.f : p * (mk * __uint_as_float(rd[ii]) - sd[i]);
              sv[ii] = ds;
              dlo[ii] = tf32_lo(ds);
              t16[ii] = p * mk;
            }
            tmem_st16(tG + (uint32_t)c0, sv);
            tmem_st16(tG + B_DPT + (uint32_t)c0, dlo);
            tmem_st16(tG + B_P + (uint32_t)c0, t16);
#pragma unroll
            for (int ii = 0; ii < 16; ++ii) t16[ii] = tf32_lo(t16[ii]);
            tmem_st16(tG + B_PL + (uint32_t)c0, t16);
          }
          tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&ds_full[grp]));
      }
    }
  } else if (warp < 14) {
    // ------------------------------------------------------------------------------------------ operand / output warps
    const int q = warp & 3, rl = q * 32 + lane, t128 = (warp - 10) * 32 + lane;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    float* stage = reinterpret_cast<float*>(gen + off_out + (warp - 10) * 2 * B_OUT);
    float kv[32], vv[32];
    float m0 = 0.f, i0 = 0.f, d0 = 0.f, m1 = 0.f, i1 = 0.f, d1 = 0.f;  // statistics of queries t128 and t128 + 128
    auto load_item = [&](int n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      const int bh = item / a.NT;
      m0 = i0 = d0 = m1 = i1 = d1 = 0.f;
      if (t128 < a.Lq) {
        const int64_t r = (int64_t)bh * a.Lq + t128;
        m0 = a.stats[r * 2]; i0 = a.stats[r * 2 + 1]; d0 = a.delta[r];
      }
      if (t128 + 128 < a.Lq) {
        const int64_t r = (int64_t)bh * a.Lq + t128 + 128;
        m1 = a.stats[r * 2]; i1 = a.stats[r * 2 + 1]; d1 = a.delta[r];
      }
      mbar_wait(smem_u32(&rows_full), n & 1);
      const float* ks = reinterpret_cast<const float*>(gen + off_rows) + rl * DK;
      const float* vs = ks + B_ROWS / 4;
#pragma unroll
      for (int c = 0; c < 32; c += 4) {
        const int sc = ((c >> 2) ^ (rl & 7)) << 2;  // 128-byte swizzle: 16-byte chunk c of row r sits at c ^ (r & 7)
        const float4 x = ld4(ks + sc), y = ld4(vs + sc);
        kv[c] = x.x * a.scale_log2; kv[c + 1] = x.y * a.scale_log2; kv[c + 2] = x.z * a.scale_log2; kv[c + 3] = x.w * a.scale_log2;
        vv[c] = y.x; vv[c + 1] = y.y; vv[c + 2] = y.z; vv[c + 3] = y.w;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&rows_free));
    };
    auto store_dkv = [&](int n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      const int bh = item / a.NT, kt = item - bh * a.NT, b = bh / a.h, hh = bh - b * a.h;
      mbar_wait(smem_u32(&dkv_full), n & 1);
      tc_fence_after();
      // [x.B + x_lo.B | x.B_lo] halves added, dK scaled, into the warp's staging tiles (16-byte chunks XOR-swizzled by
      // row) so that every global store below is a full 128-byte row
#pragma unroll
      for (int which = 0; which < 2; ++which) {
        const uint32_t tcol = tmem + lane_sel + (which == 0 ? B_DK : B_DV);
        const float mul = which == 0 ? a.scale : 1.f;
        float* dst = stage + which * (B_OUT / 4) + lane * DK;
#pragma unroll
        for (int part = 0; part < 2; ++part) {
          float x[16], y[16];
          tmem_ld16(tcol + part * 16, x);
          tmem_ld16(tcol + DK + part * 16, y);
#pragma unroll
          for (int c = 0; c < 16; c += 4) {
            const int ch = part * 4 + (c >> 2);
            st4(dst + ((ch ^ (lane & 7)) << 2), make_float4((x[c] + y[c]) * mul, (x[c + 1] + y[c + 1]) * mul, (x[c + 2] + y[c + 2]) * mul,
                                                            (x[c + 3] + y[c + 3]) * mul));
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&dkv_free));
      const int64_t row0 = (int64_t)b * L + kt * 128 + q * 32;
      const int rows_ok = L - (kt * 128 + q * 32);  // rows of this warp inside the sequence
#pragma unroll
      for (int which = 0; which < 2; ++which) {
        const float* src = stage + which * (B_OUT / 4);
        float* base = which == 0 ? a.dk + row0 * a.lddk + hh * DK : a.dv + row0 * a.lddv + hh * DK;
        const int64_t ld = which == 0 ? a.lddk : a.lddv;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int r = it * 4 + (lane >> 3), ch = lane & 7;
          if (r < rows_ok) st4(base + r * ld + ch * 4, ld4(src + r * DK + ((ch ^ (r & 7)) << 2)));
        }
      }
      __syncwarp();
    };
    if (n_items > 0) load_item(0);
    for (int n = 0; n < n_items; ++n) {
      st_m[n & 1][t128] = m0; st_i[n & 1][t128] = i0; st_d[n & 1][t128] = d0;
      st_m[n & 1][t128 + 128] = m1; st_i[n & 1][t128 + 128] = i1; st_d[n & 1][t128 + 128] = d1;
      if (n >= 1) {
        mbar_wait(smem_u32(&ops_free), (n - 1) & 1);  // every S^T / dP^T of the previous item has read its K / V
        tc_fence_after();
      }
      {
        float t16[16];
#pragma unroll
        for (int part = 0; part < 2; ++part) {
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = kv[part * 16 + c];
          tmem_st16(tmem + lane_sel + B_K + part * 16, t16);
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = tf32_lo(t16[c]);
          tmem_st16(tmem + lane_sel + B_KL + part * 16, t16);
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = vv[part * 16 + c];
          tmem_st16(tmem + lane_sel + B_V + part * 16, t16);
#pragma unroll
          for (int c = 0; c < 16; ++c) t16[c] = tf32_lo(t16[c]);
          tmem_st16(tmem + lane_sel + B_VL + part * 16, t16);
        }
        tmem_st_wait();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&ops_full));
      // dK / dV are single-buffered: the previous item's result must leave before this item's first update, and the
      // producer only reaches the next item's K / V rows once this item's query stream has drained -- so this order
      if (n >= 1) store_dkv(n - 1);
      if (n + 1 < n_items) load_item(n + 1);
    }
    if (n_items > 0) store_dkv(n_items - 1);
  } else {
    // ------------------------------------------------------------------------------------------ TF32 residual copies
    const int tid = (warp - 14) * 32 + lane;
    int g = 0;
    for (int n = 0; n < n_items; ++n) {
      const int item = (int)blockIdx.x + n * (int)gridDim.x;
      for (int c = first_chunk(item % a.NT); c < NSC; ++c, ++g) {
        const int s = g % B_NSTG;
        mbar_wait(smem_u32(&full_bar[s]), (g / B_NSTG) & 1);
        float* st = reinterpret_cast<float*>(gen + (size_t)s * B_STAGE);
        split_lo(st, st + 4 * B_TILE / 4, (int)(4 * B_TILE / 16), tid, 64);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&split_bar[s]));
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

// [B, L, width] fp32 view of a token-major buffer with row stride ld; box = [1, box_rows, 32], 128-byte swizzle
bool encode_map3(CUtensorMap* map, const float* base, int B, int L, int width, int64_t ld, int box_rows, bool mn_major) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t gdim[3] = {(cuuint64_t)width, (cuuint64_t)L, (cuuint64_t)B};
  cuuint64_t gstride[2] = {(cuuint64_t)ld * sizeof(float), (cuuint64_t)L * ld * sizeof(float)};
  cuuint32_t box[3] = {(cuuint32_t)DK, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  // K-major consumers read the classic 128-byte swizzle; MN-major TF32 consumers need the 32-byte-atom variant
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    fprintf(stderr, "librbm_b200: cuTensorMapEncodeTiled rc=%d base=%p dims=(%d,%d,%d) ld=%lld box_rows=%d mn=%d\n", (int)r, (const void*)base,
            width, L, B, (long long)ld, box_rows, (int)mn_major);
  return r == CUDA_SUCCESS;
}

}  // namespace

// RBM_ATTN_IMPL=mma sends every dense attention call to the SIMT kernels of attention.cu: tests/test_attention_gpu.py and
// tools/run_env_matrix.sh use it to run those kernels at d_k = 32 and 64, where the shape rules pick the tensor-core ones.  Read
// once per process: the tests set it before the library is loaded.
bool rbm_attn_tc_enabled() {
  static const bool v = [] {
    const char* e = getenv("RBM_ATTN_IMPL");
    return !(e && strcmp(e, "mma") == 0);
  }();
  return v;
}

bool rbm_attn_fwd_tc_supported(int L, int dk, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, const void* q, const void* k,
                               const void* v, const void* out) {
  if (!rbm_attn_tc_enabled() || dk != DK || L < 1 || L > 256) return false;  // the score tile is one TMEM region of Lp <= 256 columns
  if (ldq % 4 || ldk % 4 || ldv % 4 || ldo % 4) return false;
  if (((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)out) & 15) return false;
  return get_encode() != nullptr;
}

int rbm_attn_fwd_tc_launch(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const int64_t* tok,
                           float* out, int64_t ldo, float* stats, int B, int L, int Lq, int h, int mask_mode, float scale, float p,
                           uint64_t seed, uint64_t site, cudaStream_t st) {
  const int LPK = (L + 15) & ~15, NT = (Lq + 127) / 128;  // query tiles over Lq rows, keys over L
  CUtensorMap mapQ, mapK, mapV;
  if (!encode_map3(&mapQ, q, B, Lq, h * DK, ldq, 128, false) || !encode_map3(&mapK, k, B, L, h * DK, ldk, 64, false) ||
      !encode_map3(&mapV, v, B, L, h * DK, ldv, 64, true)) {
    rbm_set_error("rbm_attn_fwd(tcgen05): cuTensorMapEncodeTiled failed");
    return -1;
  }
  TcAttnArgs a{};
  a.tok = tok; a.out = out; a.stats = stats; a.ldo = ldo; a.L = L; a.Lq = Lq; a.LPK = LPK; a.h = h; a.NT = NT; a.mask_mode = mask_mode;
  a.scale_log2 = scale * RBM_LOG2E;
  a.thr16 = rbm_drop_threshold16(p); a.inv_keep = 1.f / (1.f - p); a.seed = seed; a.site = site;
  a.items = B * h * NT;
  const size_t smem = (size_t)2 * F_NSTG * F_STAGE + F_ROWS + 4 * F_OUT + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    if (!set_smem(attn_fwd_tc_kernel<false, false>, smem, "rbm_attn_fwd(tcgen05)") ||
        !set_smem(attn_fwd_tc_kernel<false, true>, smem, "rbm_attn_fwd(tcgen05)") ||
        !set_smem(attn_fwd_tc_kernel<true, false>, smem, "rbm_attn_fwd(tcgen05)") ||
        !set_smem(attn_fwd_tc_kernel<true, true>, smem, "rbm_attn_fwd(tcgen05)"))
      return -1;
    attr_set = true;
  }
  const bool causal = mask_mode == RBM_MASK_CAUSAL, drop = a.thr16 != 0;
  const int grid = a.items < RBM_NUM_SMS ? a.items : RBM_NUM_SMS;
  if (causal && drop) attn_fwd_tc_kernel<true, true><<<grid, F_THREADS, smem, st>>>(mapQ, mapK, mapV, a);
  else if (causal) attn_fwd_tc_kernel<true, false><<<grid, F_THREADS, smem, st>>>(mapQ, mapK, mapV, a);
  else if (drop) attn_fwd_tc_kernel<false, true><<<grid, F_THREADS, smem, st>>>(mapQ, mapK, mapV, a);
  else attn_fwd_tc_kernel<false, false><<<grid, F_THREADS, smem, st>>>(mapQ, mapK, mapV, a);
  RBM_LAUNCH_CHECK("rbm_attn_fwd(tcgen05)");
  return 0;
}

bool rbm_attn_bwd_dq_tc_supported(int L, int dk, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, int64_t lddo, int64_t lddq,
                                  const void* q, const void* k, const void* v, const void* o, const void* dout, const void* dq) {
  if (!rbm_attn_tc_enabled() || dk != DK || L < 1 || L > 256) return false;
  if (ldq % 4 || ldk % 4 || ldv % 4 || ldo % 4 || lddo % 4 || lddq % 4) return false;
  if (((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)o | (uintptr_t)dout | (uintptr_t)dq) & 15) return false;
  return get_encode() != nullptr;
}

int rbm_attn_bwd_dq_tc_launch(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const int64_t* tok,
                              const float* o, int64_t ldo, const float* dout, int64_t lddo, const float* stats, float* dq, int64_t lddq,
                              float* delta, int B, int L, int Lq, int h, int mask_mode, float scale, float p, uint64_t seed,
                              uint64_t site, cudaStream_t st) {
  const int LPK = (L + 15) & ~15, NT = (Lq + 127) / 128;
  CUtensorMap mapKk, mapKm, mapVk, mapQ, mapDO, mapO;
  if (!encode_map3(&mapKk, k, B, L, h * DK, ldk, CW, false) || !encode_map3(&mapKm, k, B, L, h * DK, ldk, CW, true) ||
      !encode_map3(&mapVk, v, B, L, h * DK, ldv, CW, false) || !encode_map3(&mapQ, q, B, Lq, h * DK, ldq, 128, false) ||
      !encode_map3(&mapDO, dout, B, Lq, h * DK, lddo, 128, false) || !encode_map3(&mapO, o, B, Lq, h * DK, ldo, 128, false)) {
    rbm_set_error("rbm_attn_bwd(tcgen05): cuTensorMapEncodeTiled failed");
    return -1;
  }
  TcBwdArgs a{};
  a.q = q; a.o = o; a.dout = dout; a.stats = stats; a.dq = dq; a.delta = delta; a.ldq = ldq; a.ldo = ldo; a.lddo = lddo; a.lddq = lddq;
  a.tok = tok; a.L = L; a.Lq = Lq; a.LPK = LPK; a.h = h; a.NT = NT; a.mask_mode = mask_mode; a.scale = scale; a.scale_log2 = scale * RBM_LOG2E;
  a.thr16 = rbm_drop_threshold16(p); a.inv_keep = 1.f / (1.f - p); a.seed = seed; a.site = site;
  a.items = B * h * NT;
  const size_t smem = (size_t)A_NSTG * A_STAGE + 3 * A_ROWS + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    if (!set_smem(attn_bwd_dq_tc_kernel<false, false>, smem, "rbm_attn_bwd(tcgen05)") ||
        !set_smem(attn_bwd_dq_tc_kernel<false, true>, smem, "rbm_attn_bwd(tcgen05)") ||
        !set_smem(attn_bwd_dq_tc_kernel<true, false>, smem, "rbm_attn_bwd(tcgen05)") ||
        !set_smem(attn_bwd_dq_tc_kernel<true, true>, smem, "rbm_attn_bwd(tcgen05)"))
      return -1;
    attr_set = true;
  }
  const bool causal = mask_mode == RBM_MASK_CAUSAL, drop = a.thr16 != 0;
  const int grid = a.items < RBM_NUM_SMS ? a.items : RBM_NUM_SMS;
  if (causal && drop) attn_bwd_dq_tc_kernel<true, true><<<grid, A_THREADS, smem, st>>>(mapKk, mapKm, mapVk, mapQ, mapDO, mapO, a);
  else if (causal) attn_bwd_dq_tc_kernel<true, false><<<grid, A_THREADS, smem, st>>>(mapKk, mapKm, mapVk, mapQ, mapDO, mapO, a);
  else if (drop) attn_bwd_dq_tc_kernel<false, true><<<grid, A_THREADS, smem, st>>>(mapKk, mapKm, mapVk, mapQ, mapDO, mapO, a);
  else attn_bwd_dq_tc_kernel<false, false><<<grid, A_THREADS, smem, st>>>(mapKk, mapKm, mapVk, mapQ, mapDO, mapO, a);
  RBM_LAUNCH_CHECK("rbm_attn_bwd(tcgen05 dq)");
  return 0;
}

bool rbm_attn_bwd_dkv_tc_supported(int L, int dk, int64_t ldq, int64_t ldk, int64_t ldv, int64_t lddo, int64_t lddk, int64_t lddv,
                                   const void* q, const void* k, const void* v, const void* dout, const void* dk_, const void* dv) {
  if (!rbm_attn_tc_enabled() || dk != DK || L < 1 || L > 256) return false;
  if (ldq % 4 || ldk % 4 || ldv % 4 || lddo % 4 || lddk % 4 || lddv % 4) return false;
  if (((uintptr_t)q | (uintptr_t)k | (uintptr_t)v | (uintptr_t)dout | (uintptr_t)dk_ | (uintptr_t)dv) & 15) return false;
  return get_encode() != nullptr;
}

int rbm_attn_bwd_dkv_tc_launch(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const int64_t* tok,
                               const float* dout, int64_t lddo, const float* stats, const float* delta, float* dk_, int64_t lddk,
                               float* dv, int64_t lddv, int B, int L, int Lq, int h, int mask_mode, float scale, float p, uint64_t seed,
                               uint64_t site, cudaStream_t st) {
  const int LPK = (Lq + 15) & ~15, NT = (L + 127) / 128;  // this kernel tiles the KEYS (L) and streams the queries (Lq, padded to 16)
  CUtensorMap mQk, mQm, mOk, mOm, mK, mV;
  if (!encode_map3(&mQk, q, B, Lq, h * DK, ldq, SQ, false) || !encode_map3(&mQm, q, B, Lq, h * DK, ldq, SQ, true) ||
      !encode_map3(&mOk, dout, B, Lq, h * DK, lddo, SQ, false) || !encode_map3(&mOm, dout, B, Lq, h * DK, lddo, SQ, true) ||
      !encode_map3(&mK, k, B, L, h * DK, ldk, 128, false) || !encode_map3(&mV, v, B, L, h * DK, ldv, 128, false)) {
    rbm_set_error("rbm_attn_bwd(tcgen05 dkv): cuTensorMapEncodeTiled failed");
    return -1;
  }
  TcBwdKvArgs a{};
  a.stats = stats; a.delta = delta; a.dk = dk_; a.dv = dv; a.lddk = lddk; a.lddv = lddv;
  a.tok = tok; a.L = L; a.Lq = Lq; a.LPK = LPK; a.h = h; a.NT = NT; a.mask_mode = mask_mode; a.scale = scale; a.scale_log2 = scale * RBM_LOG2E;
  a.thr16 = rbm_drop_threshold16(p); a.inv_keep = 1.f / (1.f - p); a.seed = seed; a.site = site;
  a.items = B * h * NT;
  const size_t smem = (size_t)B_NSTG * B_STAGE + 2 * B_ROWS + 8 * B_OUT + 1024;
  static bool attr_set = false;
  if (!attr_set) {
    if (!set_smem(attn_bwd_dkv_tc_kernel<false, false>, smem, "rbm_attn_bwd(tcgen05 dkv)") ||
        !set_smem(attn_bwd_dkv_tc_kernel<false, true>, smem, "rbm_attn_bwd(tcgen05 dkv)") ||
        !set_smem(attn_bwd_dkv_tc_kernel<true, false>, smem, "rbm_attn_bwd(tcgen05 dkv)") ||
        !set_smem(attn_bwd_dkv_tc_kernel<true, true>, smem, "rbm_attn_bwd(tcgen05 dkv)"))
      return -1;
    attr_set = true;
  }
  const bool causal = mask_mode == RBM_MASK_CAUSAL, drop = a.thr16 != 0;
  const int grid = a.items < RBM_NUM_SMS ? a.items : RBM_NUM_SMS;
  if (causal && drop) attn_bwd_dkv_tc_kernel<true, true><<<grid, B_THREADS, smem, st>>>(mQk, mQm, mOk, mOm, mK, mV, a);
  else if (causal) attn_bwd_dkv_tc_kernel<true, false><<<grid, B_THREADS, smem, st>>>(mQk, mQm, mOk, mOm, mK, mV, a);
  else if (drop) attn_bwd_dkv_tc_kernel<false, true><<<grid, B_THREADS, smem, st>>>(mQk, mQm, mOk, mOm, mK, mV, a);
  else attn_bwd_dkv_tc_kernel<false, false><<<grid, B_THREADS, smem, st>>>(mQk, mQm, mOk, mOm, mK, mV, a);
  RBM_LAUNCH_CHECK("rbm_attn_bwd(tcgen05 dkv)");
  return 0;
}

RBM_DEFINE_STEP_PTR_SETTER(rbm_step_ptr_set_attention_tc)
