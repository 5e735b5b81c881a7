// attention_seq.cu -- attention forward and backward on the Blackwell tensor path for d_k = 64 and 64 < L <= 256 (any mask
// mode): BERT4Rec at BASELINE configs[3] (d = 256, 4 heads, max_len = 200; NN/models/bert_modules/attention/single.py:13-35,
// multi_head.py:24-40) and its autograd.  Replaces the mma.sync kernels of attention.cu for these shapes; the companion of
// attention_pair.cu (d_k = 64, L <= 64), same arithmetic: SPLIT fp16 -- every fp32 operand tile is scaled by a power of two
// (per item and tensor: max -> [2^13, 2^14)) and split into hi = fp16(x), lo = fp16(x - hi); a product is three tcgen05.mma
// kind::f16 passes (hi.hi + hi.lo + lo.hi, fp32 accumulation in tensor memory): 22 significant bits, as 3xTF32.  A staged
// 128-byte-swizzled K-major tile doubles as the MN-major operand of the products that contract along tokens.
//
// One persistent CTA per SM walks the (sequence, head) items; 256 threads stage the tiles (global fp32 -> split fp16) and
// share the row work: two threads per tensor-memory lane, each with half of the row's columns; one elected thread issues
// the MMAs.  Blocks are [128 queries x 128 keys]; an item has up to 2 x 2 of them.
//   forward  (per 128-query tile): S [128 x 256] = Q.K^T -> exact row max (first read), probabilities + dropout written back as
//            packed fp16 pairs over the score columns (second read) -> O = P~.V
//   dQ       (per query tile, per key tile): S, dP~ = dO.V^T -> dS (over the scores) -> dQ += dS.K
//   dK, dV   (per key tile, per query tile): S^T = K.Q^T, dP~^T = V.dO^T -> P~^T, dS^T -> dV += P~^T.dO, dK += dS^T.Q
// Reference semantics kept: padded keys score -1e9 (masked_fill: a fully padded row gets the uniform softmax) and pass no
// score gradient; causal / beyond-L keys are excluded; dropout per the library's Philox contract (common.cuh).
#include <cuda_fp16.h>
#include "common.cuh"
#include "mma_tiles.cuh"  // ex2, RBM_LOG2E, RBM_PADFILL
#include "tc_ptx.cuh"
#include "split16.cuh"
#include "attention_f16.cuh"
#include "attention_seq.cuh"
#include "attention_tc.cuh"  // rbm_attn_tc_enabled

namespace {

using namespace rbm_tc;
using namespace rbm_attn16;
using rbm_mma::ex2;

constexpr int DK = 64;
constexpr uint32_t T128 = 128 * 128;  // [128 rows x 64 fp16] = 16 KB

struct SeqArgs {
  const float *q, *k, *v, *o, *dout, *stats_in;
  const int64_t* tok;
  float *out, *stats, *dq, *dk_, *dv;
  int64_t ldq, ldk, ldv, ldo, lddo, lddq, lddk, lddv;
  int L, h, n_items, mask_mode;
  float scale, inv_keep, pscale, keep_pow2;  // pscale: P~ (<= inv_keep) -> fp16 range; keep_pow2: power of two >= inv_keep
  uint32_t thr16;
  uint64_t seed, site;
};

// ------------------------------------------------------------------------------------------------ tile staging
// 128 tokens [t0, t0 + 128) of item (b, hh), 64 columns: thread task (row r, 16-byte output chunk c) = 8 consecutive columns.
__device__ __forceinline__ float tile_fetch(float (&v)[4][8], const float* __restrict__ src, int64_t ld, float mul, int b, int hh, int t0, int L) {
  float mx = 0.f;
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int task = it * THREADS + (int)threadIdx.x, r = task >> 3, c = task & 7;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f), y = x;
    if (t0 + r < L) {
      const float* p = src + ((int64_t)b * L + t0 + r) * ld + hh * DK + c * 8;
      x = ld4(p);
      y = ld4(p + 4);
    }
    v[it][0] = x.x * mul; v[it][1] = x.y * mul; v[it][2] = x.z * mul; v[it][3] = x.w * mul;
    v[it][4] = y.x * mul; v[it][5] = y.y * mul; v[it][6] = y.z * mul; v[it][7] = y.w * mul;
#pragma unroll
    for (int e = 0; e < 8; ++e) mx = fmaxf(mx, fabsf(v[it][e]));
  }
  return mx;
}
// all rows of one tensor of the item (up to 256 tokens, two 128-row halves sharing ONE scale) -> hi / lo tiles of 256 rows.
// Must be called by all THREADS threads; *maxbits must be zero on entry (and is consumed).  Returns the scale.
__device__ __forceinline__ float stage_rows256(const float* __restrict__ src, int64_t ld, float mul, int b, int hh, int L, uint8_t* hi, uint8_t* lo,
                                               unsigned* maxbits) {
  float va[4][8], vb[4][8];
  tile_max(tile_fetch(va, src, ld, mul, b, hh, 0, L), maxbits);
  tile_max(tile_fetch(vb, src, ld, mul, b, hh, 128, L), maxbits);
  __syncthreads();
  const float sc = pow2_scale(__uint_as_float(*maxbits), 14);
  tile_store(va, sc, hi, lo);
  tile_store(vb, sc, hi + T128, lo + T128);
  return sc;
}
__device__ __forceinline__ float stage_rows128(const float* __restrict__ src, int64_t ld, float mul, int b, int hh, int t0, int L, uint8_t* hi,
                                               uint8_t* lo, unsigned* maxbits) {
  float va[4][8];
  tile_max(tile_fetch(va, src, ld, mul, b, hh, t0, L), maxbits);
  __syncthreads();
  const float sc = pow2_scale(__uint_as_float(*maxbits), 14);
  tile_store(va, sc, hi, lo);
  return sc;
}

// D[128 x 64] (+)= A (tensor memory, 128 tokens as two thread-halves: tokens [64 hf, 64 hf + 64) have their hi words at
// a_t + 64 hf, lo words at a_t + 64 hf + 32) . B_tile rows [0, 128) (MN-major view: one 64-element MN block, so its leading
// offset is never applied); three passes
__device__ __forceinline__ void mma_ts3_128(uint32_t d_t, uint32_t a_t, uint32_t b_hi, uint32_t b_lo, uint32_t idesc, uint32_t& acc) {
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t bt = pass == 1 ? b_lo : b_hi;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint32_t at = a_t + (uint32_t)((ks >> 2) * 64 + (pass == 2 ? 32 : 0) + (ks & 3) * 8);
      umma_f16_ts(d_t, at, make_sw128_desc_mn16(bt + ks * 2048, 1024), idesc, acc);
      acc = 1;
    }
  }
}

// shared prologue of the three kernels
#define SEQ_PROLOGUE(TMEM_COLS)                                                              \
  extern __shared__ uint8_t smem_raw[];                                                      \
  __shared__ __align__(8) uint64_t mma_bar;                                                  \
  __shared__ uint32_t tmem_base_slot;                                                        \
  __shared__ unsigned maxbits[4];                                                            \
  __shared__ uint8_t kpad[256];                                                              \
  const uint64_t site_e = rbm_site(a.site);                                                  \
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;                                \
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);                 \
  const uint32_t sb = smem_u32(sm);                                                          \
  if (threadIdx.x == 0) {                                                                    \
    mbar_init(smem_u32(&mma_bar), 1);                                                        \
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");                       \
  }                                                                                          \
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), TMEM_COLS);                           \
  tc_fence_before();                                                                         \
  __syncthreads();                                                                           \
  tc_fence_after();                                                                          \
  const uint32_t tmem = tmem_base_slot;                                                      \
  const int q4 = warp & 3, hf = warp >> 2;                                                   \
  const int r = q4 * 32 + lane;                                                              \
  const uint32_t lane_sel = (uint32_t)(q4 * 32) << 16;                                       \
  const int L = a.L, nt = (L + 127) / 128;                                                   \
  const bool causal = a.mask_mode == RBM_MASK_CAUSAL, keypad = a.mask_mode == RBM_MASK_KEYPAD; \
  uint32_t ph = 0;                                                                           \
  (void)site_e; (void)lane_sel; (void)hf; (void)r

#define SEQ_EPILOGUE(TMEM_COLS)   \
  tc_fence_before();              \
  __syncthreads();                \
  if (warp == 0) {                \
    tc_fence_after();             \
    tmem_dealloc(tmem, TMEM_COLS); \
  }

// SMEM tile map (bytes from the aligned base): every [256 x 64] tensor = hi (32 KB) | lo (32 KB)
constexpr uint32_t OFF_K = 0, OFF_V = 4 * T128, OFF_Q = 8 * T128, OFF_G = 10 * T128;          // fwd / dQ: K, V whole; Q, dO one tile
constexpr uint32_t OFB_Q = 0, OFB_G = 4 * T128, OFB_K = 8 * T128, OFB_V = 10 * T128;          // dKV: Q, dO whole; K, V one tile

// =================================================================================================== forward
// TMEM: S [0,256) -> P~ (per thread-half: hi words [128 hf, +64), lo words [128 hf + 64, +64));  O [256,320)
__global__ void __launch_bounds__(THREADS, 1) attn_seq_fwd_kernel(const SeqArgs a) {
  SEQ_PROLOGUE(512);
  __shared__ float xmax[2][128], xsum[2][128];
  const uint32_t tS = tmem, tO = tmem + 256;
  const uint32_t idS = make_idesc_f16(128, nt == 2 ? 256 : 128, 0, 0), idO = make_idesc_f16(128, DK, 0, 1);
  for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
    const int b = item / a.h, hh = item - b * a.h;
    if (threadIdx.x < 4) maxbits[threadIdx.x] = 0u;
    kpad[threadIdx.x] = (keypad && (int)threadIdx.x < L && a.tok[(int64_t)b * L + threadIdx.x] == 0) ? 1 : 0;
    __syncthreads();
    const float sK = stage_rows256(a.k, a.ldk, 1.f, b, hh, L, sm + OFF_K, sm + OFF_K + 2 * T128, &maxbits[0]);
    const float sV = stage_rows256(a.v, a.ldv, 1.f, b, hh, L, sm + OFF_V, sm + OFF_V + 2 * T128, &maxbits[1]);
    for (int qt = 0; qt < nt; ++qt) {
      if (threadIdx.x == 0) maxbits[2] = 0u;
      __syncthreads();  // (also: the previous tile's MMAs have completed and its O has been read)
      const float sQ = stage_rows128(a.q, a.ldq, a.scale * RBM_LOG2E, b, hh, qt * 128, L, sm + OFF_Q, sm + OFF_Q + T128, &maxbits[2]);
      fence_proxy_async();
      __syncthreads();
      if (warp == 0 && elect_one()) {
        tc_fence_after();
        mma_ss3(tS, sb + OFF_Q, sb + OFF_Q + T128, sb + OFF_K, sb + OFF_K + 2 * T128, idS);
        umma_commit(smem_u32(&mma_bar));
      }
      __syncwarp();
      const int i = qt * 128 + r;
      const bool row_ok = i < L;
      const bool act = hf < nt;  // this thread-half has key columns at all (L <= 128: only the first half)
      const float us = 1.f / (sQ * sK);
      mbar_wait(smem_u32(&mma_bar), ph);
      ph ^= 1;
      tc_fence_after();
      // pass 1: exact row maximum
      float m = -INFINITY;
      if (act) {
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
          float v[16];
          tmem_ld16(tS + lane_sel + (uint32_t)(hf * 128 + c * 16), v);
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) {
            const int j = hf * 128 + c * 16 + jj;
            float x = kpad[j] ? RBM_PADFILL : v[jj] * us;
            if (j >= L || (causal && j > i)) x = -INFINITY;
            m = fmaxf(m, x);
          }
        }
      }
      xmax[hf][r] = m;
      __syncthreads();
      m = row_ok ? fmaxf(xmax[0][r], xmax[1][r]) : 0.f;
      // pass 2: probabilities, dropout, packed fp16 pairs over the thread's own score columns (lo words after all reads)
      float l = 0.f;
      if (act) {
        uint32_t lo_all[8][8];
        const float keep = a.thr16 ? a.inv_keep * a.pscale : a.pscale;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          float v[16];
          tmem_ld16(tS + lane_sel + (uint32_t)(hf * 128 + c * 16), v);
          uint32_t bits = 0xffffu;
          if (a.thr16) bits = keep_bits_row(a.seed, site_e, (uint64_t)item, i, hf * 8 + c, a.thr16);
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) {
            const int j = hf * 128 + c * 16 + jj;
            float x = kpad[j] ? RBM_PADFILL : v[jj] * us;
            const bool ok = row_ok && j < L && !(causal && j > i);
            const float p = ok ? ex2(x - m) : 0.f;
            l += p;
            v[jj] = ((bits >> jj) & 1u) ? p * keep : 0.f;
          }
          uint32_t hi[8];
          split_pack16(v, hi, lo_all[c]);
          tmem_st8(tS + lane_sel + (uint32_t)(hf * 128 + c * 8), hi);
        }
#pragma unroll
        for (int c = 0; c < 8; ++c) tmem_st8(tS + lane_sel + (uint32_t)(hf * 128 + 64 + c * 8), lo_all[c]);
      }
      xsum[hf][r] = l;
      tmem_st_wait();
      tc_fence_before();
      __syncthreads();
      if (warp == 0 && elect_one()) {
        tc_fence_after();
        uint32_t acc = 0;
#pragma unroll 1
        for (int pass = 0; pass < 3; ++pass) {
          const uint32_t vt = sb + OFF_V + (pass == 1 ? 2 * T128 : 0);
          for (int kh = 0; kh < nt; ++kh)
#pragma unroll
            for (int ks = 0; ks < 8; ++ks) {
              umma_f16_ts(tO, tS + (uint32_t)(kh * 128 + (pass == 2 ? 64 : 0) + ks * 8), make_sw128_desc_mn16(vt + (kh * 128 + ks * 16) * 128, 1024),
                          idO, acc);
              acc = 1;
            }
        }
        umma_commit(smem_u32(&mma_bar));
      }
      __syncwarp();
      const float lsum = xsum[0][r] + xsum[1][r];
      const float inv_l = row_ok ? 1.f / lsum : 0.f;
      if (row_ok && hf == 0 && a.stats) {
        const int64_t sr = ((int64_t)item * L + i) * 2;
        a.stats[sr] = m;
        a.stats[sr + 1] = inv_l;
      }
      mbar_wait(smem_u32(&mma_bar), ph);
      ph ^= 1;
      tc_fence_after();
      {
        const float mul = inv_l / (a.pscale * sV);
        float* dst = a.out + ((int64_t)b * L + i) * a.ldo + hh * DK + hf * 32;
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 16) {
          float o[16];
          tmem_ld16(tO + lane_sel + (uint32_t)(hf * 32 + c0), o);
          if (row_ok) {
#pragma unroll
            for (int jj = 0; jj < 16; jj += 2) *reinterpret_cast<float2*>(dst + c0 + jj) = make_float2(o[jj] * mul, o[jj + 1] * mul);
          }
        }
      }
      tc_fence_before();
    }
    __syncthreads();
  }
  SEQ_EPILOGUE(512);
}

// shared by the two backward kernels: probability and score gradient of element (query i, key j) from the raw accumulators
struct BwdCoef {
  float us, up, keep, sd;
};

// ============================================================================================ backward: dQ
// TMEM: S [0,128) -> dS (per thread-half: hi words [64 hf, +32), lo words [64 hf + 32, +32));  dP~ [128,256);  dQ [256,320)
__global__ void __launch_bounds__(THREADS, 1) attn_seq_dq_kernel(const SeqArgs a) {
  SEQ_PROLOGUE(512);
  __shared__ float row_m[128], row_inv[128], row_delta[128];
  const uint32_t tS = tmem, tP = tmem + 128, tDQ = tmem + 256;
  const uint32_t idS = make_idesc_f16(128, 128, 0, 0), idO = make_idesc_f16(128, DK, 0, 1);
  for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
    const int b = item / a.h, hh = item - b * a.h;
    if (threadIdx.x < 4) maxbits[threadIdx.x] = 0u;
    kpad[threadIdx.x] = (keypad && (int)threadIdx.x < L && a.tok[(int64_t)b * L + threadIdx.x] == 0) ? 1 : 0;
    __syncthreads();
    const float sK = stage_rows256(a.k, a.ldk, 1.f, b, hh, L, sm + OFF_K, sm + OFF_K + 2 * T128, &maxbits[0]);
    const float sV = stage_rows256(a.v, a.ldv, 1.f, b, hh, L, sm + OFF_V, sm + OFF_V + 2 * T128, &maxbits[1]);
    for (int qt = 0; qt < nt; ++qt) {
      if (threadIdx.x < 2) maxbits[2 + threadIdx.x] = 0u;
      __syncthreads();  // (also: the previous tile's MMAs have completed and its dQ has been read)
      const int i = qt * 128 + r;
      const bool row_ok = i < L;
      if (hf == 0) {  // row statistics and delta_i = <dO_i, O_i> (fp32, from HBM)
        float m = 0.f, inv = 0.f, delta = 0.f;
        if (row_ok) {
          const int64_t sr = ((int64_t)item * L + i) * 2;
          m = a.stats_in[sr];
          inv = a.stats_in[sr + 1];
          const float* po = a.o + ((int64_t)b * L + i) * a.ldo + hh * DK;
          const float* pg = a.dout + ((int64_t)b * L + i) * a.lddo + hh * DK;
#pragma unroll
          for (int c = 0; c < DK; c += 4) {
            const float4 x = ld4(pg + c);
            const float2 y0 = *reinterpret_cast<const float2*>(po + c), y1 = *reinterpret_cast<const float2*>(po + c + 2);
            delta = fmaf(x.x, y0.x, delta); delta = fmaf(x.y, y0.y, delta); delta = fmaf(x.z, y1.x, delta); delta = fmaf(x.w, y1.y, delta);
          }
        }
        row_m[r] = m; row_inv[r] = inv; row_delta[r] = delta;
      }
      float sQ, sG;
      {
        float va[4][8], vb[4][8];
        tile_max(tile_fetch(va, a.q, a.ldq, a.scale * RBM_LOG2E, b, hh, qt * 128, L), &maxbits[2]);
        tile_max(tile_fetch(vb, a.dout, a.lddo, 1.f, b, hh, qt * 128, L), &maxbits[3]);
        __syncthreads();
        sQ = pow2_scale(__uint_as_float(maxbits[2]), 14);
        sG = pow2_scale(__uint_as_float(maxbits[3]), 14);
        tile_store(va, sQ, sm + OFF_Q, sm + OFF_Q + T128);
        tile_store(vb, sG, sm + OFF_G, sm + OFF_G + T128);
      }
      fence_proxy_async();
      __syncthreads();
      const float m = row_m[r], inv = row_inv[r], delta = row_delta[r];
      const float us = 1.f / (sQ * sK), up = 1.f / (sG * sV), keep = a.thr16 ? a.inv_keep : 1.f;
      // |dS| <= P (keep |dP~| + |delta|) <= 2 keep max|dP~| and |dP~ accumulator| <= 64 * 2^14 * 2^14: this power of two keeps dS in fp16 range
      const float sd = sG * sV * (1.f / 2097152.f) / a.keep_pow2;
      uint32_t dq_acc = 0;
      for (int kt = 0; kt < nt; ++kt) {
        if (warp == 0 && elect_one()) {
          tc_fence_after();
          mma_ss3(tS, sb + OFF_Q, sb + OFF_Q + T128, sb + OFF_K + kt * T128, sb + OFF_K + 2 * T128 + kt * T128, idS);  // S = Q.K^T
          mma_ss3(tP, sb + OFF_G, sb + OFF_G + T128, sb + OFF_V + kt * T128, sb + OFF_V + 2 * T128 + kt * T128, idS);  // dP~ = dO.V^T
          umma_commit(smem_u32(&mma_bar));
        }
        __syncwarp();
        mbar_wait(smem_u32(&mma_bar), ph);
        ph ^= 1;
        tc_fence_after();
        float ds[64];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float(&v)[16] = *reinterpret_cast<float(*)[16]>(&ds[c * 16]);
          float dp[16];
          tmem_ld16(tS + lane_sel + (uint32_t)(hf * 64 + c * 16), v);
          tmem_ld16(tP + lane_sel + (uint32_t)(hf * 64 + c * 16), dp);
          uint32_t bits = 0xffffu;
          if (a.thr16) bits = keep_bits_row(a.seed, site_e, (uint64_t)item, i, kt * 8 + hf * 4 + c, a.thr16);
#pragma unroll
          for (int jj = 0; jj < 16; ++jj) {
            const int j = kt * 128 + hf * 64 + c * 16 + jj;
            const bool pad = kpad[j & 255] != 0;
            const bool ok = row_ok && j < L && !(causal && j > i);
            const float x = pad ? RBM_PADFILL : v[jj] * us;
            const float p = ok ? ex2(x - m) * inv : 0.f;
            const float mk = ((bits >> jj) & 1u) ? keep : 0.f;
            v[jj] = pad ? 0.f : p * (mk * dp[jj] * up - delta) * sd;  // no score gradient through a padded key
          }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t hi[8], lo[8];
          split_pack16(*reinterpret_cast<float(*)[16]>(&ds[c * 16]), hi, lo);
          tmem_st8(tS + lane_sel + (uint32_t)(hf * 64 + c * 8), hi);
          tmem_st8(tS + lane_sel + (uint32_t)(hf * 64 + 32 + c * 8), lo);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncthreads();
        if (warp == 0 && elect_one()) {
          tc_fence_after();
          mma_ts3_128(tDQ, tS, sb + OFF_K + kt * T128, sb + OFF_K + 2 * T128 + kt * T128, idO, dq_acc);  // dQ += dS.K
          if (kt == nt - 1) umma_commit(smem_u32(&mma_bar));
        }
        dq_acc = 1;
        __syncwarp();
      }
      mbar_wait(smem_u32(&mma_bar), ph);
      ph ^= 1;
      tc_fence_after();
      {
        const float mul = a.scale / (sd * sK);
        float* dst = a.dq + ((int64_t)b * L + i) * a.lddq + hh * DK + hf * 32;
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 16) {
          float o[16];
          tmem_ld16(tDQ + lane_sel + (uint32_t)(hf * 32 + c0), o);
          if (row_ok) {
#pragma unroll
            for (int jj = 0; jj < 16; jj += 2) *reinterpret_cast<float2*>(dst + c0 + jj) = make_float2(o[jj] * mul, o[jj + 1] * mul);
          }
        }
      }
      tc_fence_before();
    }
    __syncthreads();
  }
  SEQ_EPILOGUE(512);
}

// ========================================================================================= backward: dK, dV
// TMEM: S^T [0,128) -> P~^T;  dP~^T [128,256) -> dS^T (per thread-half: hi words [64 hf, +32), lo words [64 hf + 32, +32) of each
// block);  dV [256,320);  dK [320,384)
__global__ void __launch_bounds__(THREADS, 1) attn_seq_dkv_kernel(const SeqArgs a) {
  SEQ_PROLOGUE(512);
  __shared__ float row_m[256], row_inv[256], row_delta[256];
  const uint32_t tS = tmem, tP = tmem + 128, tDV = tmem + 256, tDK = tmem + 320;
  const uint32_t idS = make_idesc_f16(128, 128, 0, 0), idO = make_idesc_f16(128, DK, 0, 1);
  for (int item = blockIdx.x; item < a.n_items; item += gridDim.x) {
    const int b = item / a.h, hh = item - b * a.h;
    if (threadIdx.x < 4) maxbits[threadIdx.x] = 0u;
    kpad[threadIdx.x] = (keypad && (int)threadIdx.x < L && a.tok[(int64_t)b * L + threadIdx.x] == 0) ? 1 : 0;
    {  // statistics of all queries of the item: one thread per query
      const int i = threadIdx.x;
      float m = 0.f, inv = 0.f, delta = 0.f;
      if (i < L) {
        const int64_t sr = ((int64_t)item * L + i) * 2;
        m = a.stats_in[sr];
        inv = a.stats_in[sr + 1];
        const float* po = a.o + ((int64_t)b * L + i) * a.ldo + hh * DK;
        const float* pg = a.dout + ((int64_t)b * L + i) * a.lddo + hh * DK;
#pragma unroll
        for (int c = 0; c < DK; c += 4) {
          const float4 x = ld4(pg + c);
          const float2 y0 = *reinterpret_cast<const float2*>(po + c), y1 = *reinterpret_cast<const float2*>(po + c + 2);
          delta = fmaf(x.x, y0.x, delta); delta = fmaf(x.y, y0.y, delta); delta = fmaf(x.z, y1.x, delta); delta = fmaf(x.w, y1.y, delta);
        }
      }
      row_m[i] = m; row_inv[i] = inv; row_delta[i] = delta;
    }
    __syncthreads();
    const float sQ = stage_rows256(a.q, a.ldq, a.scale * RBM_LOG2E, b, hh, L, sm + OFB_Q, sm + OFB_Q + 2 * T128, &maxbits[0]);
    const float sG = stage_rows256(a.dout, a.lddo, 1.f, b, hh, L, sm + OFB_G, sm + OFB_G + 2 * T128, &maxbits[1]);
    for (int kt = 0; kt < nt; ++kt) {
      if (threadIdx.x < 2) maxbits[2 + threadIdx.x] = 0u;
      __syncthreads();  // (also: the previous tile's MMAs have completed and its dK / dV have been read)
      float sK, sV;
      {
        float va[4][8], vb[4][8];
        tile_max(tile_fetch(va, a.k, a.ldk, 1.f, b, hh, kt * 128, L), &maxbits[2]);
        tile_max(tile_fetch(vb, a.v, a.ldv, 1.f, b, hh, kt * 128, L), &maxbits[3]);
        __syncthreads();
        sK = pow2_scale(__uint_as_float(maxbits[2]), 14);
        sV = pow2_scale(__uint_as_float(maxbits[3]), 14);
        tile_store(va, sK, sm + OFB_K, sm + OFB_K + T128);
        tile_store(vb, sV, sm + OFB_V, sm + OFB_V + T128);
      }
      fence_proxy_async();
      __syncthreads();
      const int j = kt * 128 + r;  // this lane's key
      const bool key_ok = j < L;
      const bool pad = kpad[j & 255] != 0;
      const float us = 1.f / (sQ * sK), up = 1.f / (sG * sV), keep = a.thr16 ? a.inv_keep : 1.f;
      const float sd = sG * sV * (1.f / 2097152.f) / a.keep_pow2;
      uint32_t acc_v = 0, acc_k = 0;
      for (int qt = 0; qt < nt; ++qt) {
        if (warp == 0 && elect_one()) {
          tc_fence_after();
          mma_ss3(tS, sb + OFB_K, sb + OFB_K + T128, sb + OFB_Q + qt * T128, sb + OFB_Q + 2 * T128 + qt * T128, idS);  // S^T = K.Q^T
          mma_ss3(tP, sb + OFB_V, sb + OFB_V + T128, sb + OFB_G + qt * T128, sb + OFB_G + 2 * T128 + qt * T128, idS);  // dP~^T = V.dO^T
          umma_commit(smem_u32(&mma_bar));
        }
        __syncwarp();
        mbar_wait(smem_u32(&mma_bar), ph);
        ph ^= 1;
        tc_fence_after();
        float ds[64], pt[64];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float(&v)[16] = *reinterpret_cast<float(*)[16]>(&ds[c * 16]);
          float(&pv)[16] = *reinterpret_cast<float(*)[16]>(&pt[c * 16]);
          float dp[16];
          tmem_ld16(tS + lane_sel + (uint32_t)(hf * 64 + c * 16), v);
          tmem_ld16(tP + lane_sel + (uint32_t)(hf * 64 + c * 16), dp);
          const int T = qt * 8 + hf * 4 + c;  // this chunk's 16 queries [16 T, 16 T + 16)
          uint32_t bits = 0xffffu;
          if (a.thr16) bits = keep_bits_col(a.seed, site_e, (uint64_t)item, j, T, a.thr16);
#pragma unroll
          for (int ii = 0; ii < 16; ++ii) {
            const int qi = T * 16 + ii;
            const bool ok = key_ok && qi < L && !(causal && j > qi);
            const float x = pad ? RBM_PADFILL : v[ii] * us;
            const float p = ok ? ex2(x - row_m[qi & 255]) * row_inv[qi & 255] : 0.f;
            const float mk = ((bits >> ii) & 1u) ? keep : 0.f;
            pv[ii] = p * mk * a.pscale;
            v[ii] = pad ? 0.f : p * (mk * dp[ii] * up - row_delta[qi & 255]) * sd;
          }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t hi[8], lo[8];
          split_pack16(*reinterpret_cast<float(*)[16]>(&pt[c * 16]), hi, lo);
          tmem_st8(tS + lane_sel + (uint32_t)(hf * 64 + c * 8), hi);
          tmem_st8(tS + lane_sel + (uint32_t)(hf * 64 + 32 + c * 8), lo);
          split_pack16(*reinterpret_cast<float(*)[16]>(&ds[c * 16]), hi, lo);
          tmem_st8(tP + lane_sel + (uint32_t)(hf * 64 + c * 8), hi);
          tmem_st8(tP + lane_sel + (uint32_t)(hf * 64 + 32 + c * 8), lo);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncthreads();
        if (warp == 0 && elect_one()) {
          tc_fence_after();
          mma_ts3_128(tDV, tS, sb + OFB_G + qt * T128, sb + OFB_G + 2 * T128 + qt * T128, idO, acc_v);  // dV += P~^T.dO
          mma_ts3_128(tDK, tP, sb + OFB_Q + qt * T128, sb + OFB_Q + 2 * T128 + qt * T128, idO, acc_k);  // dK += dS^T.Q
          if (qt == nt - 1) umma_commit(smem_u32(&mma_bar));
        }
        acc_v = acc_k = 1;
        __syncwarp();
      }
      mbar_wait(smem_u32(&mma_bar), ph);
      ph ^= 1;
      tc_fence_after();
      {
        const float mv = 1.f / (a.pscale * sG), mkk = 1.f / (sd * sQ * RBM_LOG2E);  // the q tiles hold q * scale * log2(e)
        float* dstv = a.dv + ((int64_t)b * L + j) * a.lddv + hh * DK + hf * 32;
        float* dstk = a.dk_ + ((int64_t)b * L + j) * a.lddk + hh * DK + hf * 32;
#pragma unroll
        for (int c0 = 0; c0 < 32; c0 += 16) {
          float o[16], o2[16];
          tmem_ld16(tDV + lane_sel + (uint32_t)(hf * 32 + c0), o);
          tmem_ld16(tDK + lane_sel + (uint32_t)(hf * 32 + c0), o2);
          if (key_ok) {
#pragma unroll
            for (int jj = 0; jj < 16; jj += 2) {
              *reinterpret_cast<float2*>(dstv + c0 + jj) = make_float2(o[jj] * mv, o[jj + 1] * mv);
              *reinterpret_cast<float2*>(dstk + c0 + jj) = make_float2(o2[jj] * mkk, o2[jj + 1] * mkk);
            }
          }
        }
      }
      tc_fence_before();
    }
    __syncthreads();
  }
  SEQ_EPILOGUE(512);
}

void fill_common(SeqArgs& a, int B, int L, int h, int mask_mode, float scale, float p, uint64_t seed, uint64_t site, const int64_t* tok) {
  a.L = L; a.h = h; a.n_items = B * h; a.mask_mode = mask_mode; a.scale = scale; a.tok = tok;
  a.thr16 = rbm_drop_threshold16(p);
  a.inv_keep = 1.f / (1.f - p);
  int e = 0;
  frexpf(a.inv_keep, &e);  // inv_keep <= 2^e
  a.keep_pow2 = ldexpf(1.f, e);
  a.pscale = pow2_scale(a.inv_keep, 14);
  a.seed = seed; a.site = site;
}

}  // namespace

bool rbm_attn_seq_supported(int L, int dk, int mask_mode) { return rbm_attn_tc_enabled() && dk == DK && L > 64 && L <= 256 && mask_mode >= 0 && mask_mode <= 2; }

int rbm_attn_seq_fwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const int64_t* tok, float* out,
                     int64_t ldo, float* stats, int B, int L, int h, int mask_mode, float scale, float p, uint64_t seed, uint64_t site,
                     cudaStream_t st) {
  SeqArgs a{};
  a.q = q; a.k = k; a.v = v; a.out = out; a.stats = stats; a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo;
  fill_common(a, B, L, h, mask_mode, scale, p, seed, site, tok);
  const size_t smem = 10 * T128 + 1024;
  if (!set_smem(attn_seq_fwd_kernel, smem, "rbm_attn_fwd(seq)")) return -1;
  const int grid = a.n_items < RBM_NUM_SMS ? a.n_items : RBM_NUM_SMS;
  attn_seq_fwd_kernel<<<grid, THREADS, smem, st>>>(a);
  RBM_LAUNCH_CHECK("rbm_attn_fwd(seq)");
  return 0;
}

int rbm_attn_seq_bwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const int64_t* tok, const float* out,
                     int64_t ldo, const float* dout, int64_t lddo, const float* stats, float* dq, int64_t lddq, float* dk_, int64_t lddk,
                     float* dv, int64_t lddv, int B, int L, int h, int mask_mode, float scale, float p, uint64_t seed, uint64_t site,
                     cudaStream_t st) {
  SeqArgs a{};
  a.q = q; a.k = k; a.v = v; a.o = out; a.dout = dout; a.stats_in = stats; a.dq = dq; a.dk_ = dk_; a.dv = dv;
  a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo; a.lddo = lddo; a.lddq = lddq; a.lddk = lddk; a.lddv = lddv;
  fill_common(a, B, L, h, mask_mode, scale, p, seed, site, tok);
  const size_t smem = 12 * T128 + 1024;
  if (!set_smem(attn_seq_dq_kernel, smem, "rbm_attn_bwd(seq dq)") || !set_smem(attn_seq_dkv_kernel, smem, "rbm_attn_bwd(seq dkv)")) return -1;
  const int grid = a.n_items < RBM_NUM_SMS ? a.n_items : RBM_NUM_SMS;
  attn_seq_dq_kernel<<<grid, THREADS, smem, st>>>(a);
  RBM_LAUNCH_CHECK("rbm_attn_bwd(seq dq)");
  attn_seq_dkv_kernel<<<grid, THREADS, smem, st>>>(a);
  RBM_LAUNCH_CHECK("rbm_attn_bwd(seq dkv)");
  return 0;
}

RBM_DEFINE_STEP_PTR_SETTER(rbm_step_ptr_set_attention_seq)
