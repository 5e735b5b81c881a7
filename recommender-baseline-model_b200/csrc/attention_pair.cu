// attention_pair.cu -- attention forward and backward on the Blackwell tensor path for SHORT sequences with d_k = 64
// (L <= 64; no mask or causal mask): the SASRec shapes (NN/models/sas_model/sas.py:75-76, nn.MultiheadAttention with
// d = 64, h = 1 or d = 128, h = 2 at max_len = 50).  Replaces the mma.sync kernels of attention.cu for these shapes.
//
// Two (sequence, head) items share one 128-lane tensor-memory tile: item 2w in rows / columns [0, 64), item 2w + 1 in
// [64, 128); score products are [128 x 128] with the two off-diagonal blocks ignored (a tcgen05.mma with M = 128 costs
// ~64 cycles whatever N <= 128 is, so the wasted half is free).  Arithmetic: SPLIT fp16 -- every fp32 tile (q, k, v, dO)
// is scaled by its own power of two (tile max -> [2^13, 2^14)) and written to shared memory as hi = fp16(x),
// lo = fp16(x - hi) in the 128-byte-swizzled K-major layout; a product is three kind::f16 passes (hi.hi + hi.lo + lo.hi):
// 22 significant bits, the accuracy of 3xTF32.  The same tile serves as K-major operand (contraction along d_k) and,
// read through an MN-major descriptor, as the operand of the products that contract along tokens.  Probabilities and score
// gradients are written back to tensor memory as packed fp16 pairs (A operands).
//   forward : S = Q.K^T -> softmax (thread per query row, exact row max), dropout -> O = P~.V
//   backward: phase 1 (lanes = queries): S, dP~ = dO.V^T -> dS -> dQ = dS.K
//             phase 2 (lanes = keys)   : S^T = K.Q^T, dP~^T = V.dO^T -> P~^T, dS^T -> dV = P~^T.dO, dK = dS^T.Q
// Persistent CTAs (one per SM) walk the item pairs; 256 threads: all eight warps stage the tiles (global fp32 -> split fp16, two
// tiles in flight) and share the softmax work -- two threads per tensor-memory lane, each with half of the row's columns; one
// elected thread of warp 0 issues the MMAs.  Dropout follows the library's Philox
// contract (common.cuh, rbm_attn_keep), atomics-free and bit-deterministic.
#include <cuda_fp16.h>
#include "common.cuh"
#include "mma_tiles.cuh"  // ex2, RBM_LOG2E
#include "tc_ptx.cuh"
#include "split16.cuh"
#include "attention_f16.cuh"
#include "attention_pair.cuh"
#include "attention_tc.cuh"  // rbm_attn_tc_enabled

namespace {

using namespace rbm_tc;
using namespace rbm_attn16;
using rbm_mma::ex2;

constexpr int DK = 64;
constexpr uint32_t TILE = 128 * 128;  // [128 rows x 64 fp16] = 16 KB
enum { T_QH = 0, T_QL, T_KH, T_KL, T_VH, T_VL, T_GH, T_GL };

struct PairArgs {
  const float *q, *k, *v, *o, *dout, *stats_in;
  float *out, *stats, *dq, *dk_, *dv;
  int64_t ldq, ldk, ldv, ldo, lddo, lddq, lddk, lddv;
  int L, h, n_items, causal;
  float scale, inv_keep, pscale;  // pscale: power of two that brings P~ (<= inv_keep) into fp16 range
  uint32_t thr16;
  uint64_t seed, site;
};

// ------------------------------------------------------------------------------------------------ tile staging
// One [128 x 64] tile = the rows of both items of the pair (item s in rows [64 s, 64 s + L); the rest zero).  Thread task
// (row r, 16-byte output chunk c) covers 8 consecutive columns.  Returns the values in registers and the thread's max |x|.
__device__ __forceinline__ float tile_fetch(float (&v)[4][8], const float* __restrict__ src, int64_t ld, float mul, int pair, const PairArgs& a) {
  float mx = 0.f;
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int task = it * THREADS + (int)threadIdx.x, r = task >> 3, c = task & 7;
    const int s = r >> 6, i = r & 63, item = 2 * pair + s;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f), y = x;
    if (item < a.n_items && i < a.L) {
      const int b = item / a.h, hh = item - b * a.h;
      const float* p = src + ((int64_t)b * a.L + i) * ld + hh * DK + c * 8;
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
__device__ __forceinline__ float tile_scale_of(const unsigned* maxbits) { return pow2_scale(__uint_as_float(*maxbits), 14); }

// D[128 x 64] = A (tensor memory, K = 128 tokens: hi words at a_t, lo words at a_t + 64) . B_tile (MN-major view: one 64-element
// MN block, so its leading offset is never applied); three passes
__device__ __forceinline__ void mma_ts3(uint32_t d_t, uint32_t a_t, uint32_t b_hi, uint32_t b_lo, uint32_t idesc) {
  uint32_t acc = 0;
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint32_t at = pass == 2 ? a_t + 64 : a_t, bt = pass == 1 ? b_lo : b_hi;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      umma_f16_ts(d_t, at + (uint32_t)(ks * 8), make_sw128_desc_mn16(bt + ks * 2048, 1024), idesc, acc);
      acc = 1;
    }
  }
}

// Packed A operands (K = 128 tokens): hi words [0, 64), lo words [64, 128); word w = tokens (2 w, 2 w + 1); slot s owns words
// [32 s, 32 s + 32), the other slot's words are zero.  A thread covers the 16-token parts {2 hf, 2 hf + 1} of its row.
__device__ __forceinline__ void store_packed_part(uint32_t t_hi, int slot, int part, const uint32_t (&hi)[8], const uint32_t (&lo)[8]) {
  tmem_st8(t_hi + (uint32_t)(slot * 32 + part * 8), hi);
  tmem_st8(t_hi + 64 + (uint32_t)(slot * 32 + part * 8), lo);
}
__device__ __forceinline__ void store_zero_parts(uint32_t t_hi, int slot, int hf) {
  const uint32_t z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
  for (int pp = 0; pp < 2; ++pp) {
    tmem_st8(t_hi + (uint32_t)((1 - slot) * 32 + (2 * hf + pp) * 8), z);
    tmem_st8(t_hi + 64 + (uint32_t)((1 - slot) * 32 + (2 * hf + pp) * 8), z);
  }
}

// Thread layout of both kernels: 8 warps; warp w owns tensor-memory lanes [32 (w & 3), +32) (row r = 32 (w & 3) + lane: slot
// r >> 6, token i = r & 63) and the column half hf = w >> 2 of its row: tokens [32 hf, 32 hf + 32) of the row's own block,
// columns [32 hf, 32 hf + 32) of the 64-wide outputs.  The two threads of a row meet through shared memory.

// =================================================================================================== forward
// TMEM columns: S [0,128) -> P~ hi [0,64) | lo [64,128);  O [128,192)
__global__ void __launch_bounds__(THREADS, 2) attn_pair_fwd_kernel(const PairArgs a, int n_pairs) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t mma_bar;
  __shared__ uint32_t tmem_base_slot;
  __shared__ unsigned maxbits[4];
  __shared__ float xmax[2][128], xsum[2][128];
  const uint64_t site_e = rbm_site(a.site);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sb = smem_u32(sm);
  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&mma_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot, tS = tmem, tO = tmem + 128;
  const uint32_t idS = make_idesc_f16(128, 128, 0, 0), idO = make_idesc_f16(128, DK, 0, 1);
  const int q4 = warp & 3, hf = warp >> 2;
  const int r = q4 * 32 + lane, slot = r >> 6, i = r & 63;
  const uint32_t lane_sel = (uint32_t)(q4 * 32) << 16;
  uint32_t ph = 0;  // parity of the next mma_bar completion
  for (int pair = blockIdx.x; pair < n_pairs; pair += gridDim.x) {
    if (threadIdx.x < 4) maxbits[threadIdx.x] = 0u;
    __syncthreads();
    float sQ, sK, sV;
    {  // global fp32 -> split fp16 tiles, two tiles in flight
      float va[4][8], vb[4][8];
      tile_max(tile_fetch(va, a.q, a.ldq, a.scale * RBM_LOG2E, pair, a), &maxbits[0]);
      tile_max(tile_fetch(vb, a.k, a.ldk, 1.f, pair, a), &maxbits[1]);
      __syncthreads();
      sQ = tile_scale_of(&maxbits[0]);
      sK = tile_scale_of(&maxbits[1]);
      tile_store(va, sQ, sm + T_QH * TILE, sm + T_QL * TILE);
      tile_max(tile_fetch(va, a.v, a.ldv, 1.f, pair, a), &maxbits[2]);
      tile_store(vb, sK, sm + T_KH * TILE, sm + T_KL * TILE);
      __syncthreads();
      sV = tile_scale_of(&maxbits[2]);
      tile_store(va, sV, sm + T_VH * TILE, sm + T_VL * TILE);
    }
    fence_proxy_async();
    __syncthreads();
    if (warp == 0 && elect_one()) {
      tc_fence_after();
      mma_ss3(tS, sb + T_QH * TILE, sb + T_QL * TILE, sb + T_KH * TILE, sb + T_KL * TILE, idS);
      umma_commit(smem_u32(&mma_bar));
    }
    __syncwarp();
    const int item = 2 * pair + slot;
    const bool row_ok = item < a.n_items && i < a.L;
    mbar_wait(smem_u32(&mma_bar), ph);
    ph ^= 1;
    tc_fence_after();
    float sv[32];
#pragma unroll
    for (int pp = 0; pp < 2; ++pp)
      tmem_ld16(tS + lane_sel + (uint32_t)(slot * 64 + hf * 32 + pp * 16), *reinterpret_cast<float(*)[16]>(&sv[pp * 16]));
    const float us = 1.f / (sQ * sK);
    float m = -INFINITY;
#pragma unroll
    for (int jj = 0; jj < 32; ++jj) {
      const int j = hf * 32 + jj;
      const bool ok = j < a.L && (!a.causal || j <= i);
      sv[jj] = ok ? sv[jj] * us : -INFINITY;
      m = fmaxf(m, sv[jj]);
    }
    xmax[hf][r] = m;
    __syncthreads();  // both halves of every row have read their scores: the score columns may be overwritten from here on
    m = row_ok ? fmaxf(xmax[0][r], xmax[1][r]) : 0.f;
    float l = 0.f;
#pragma unroll
    for (int jj = 0; jj < 32; ++jj) {
      sv[jj] = row_ok ? ex2(sv[jj] - m) : 0.f;
      l += sv[jj];
    }
    xsum[hf][r] = l;
#pragma unroll
    for (int pp = 0; pp < 2; ++pp) {
      const int part = 2 * hf + pp;
      float(&v)[16] = *reinterpret_cast<float(*)[16]>(&sv[pp * 16]);
      uint32_t bits = 0xffffu;
      if (a.thr16) bits = keep_bits_row(a.seed, site_e, (uint64_t)(item < a.n_items ? item : 0), i, part, a.thr16);
      const float keep = a.thr16 ? a.inv_keep * a.pscale : a.pscale;
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) v[jj] = ((bits >> jj) & 1u) ? v[jj] * keep : 0.f;
      uint32_t hi[8], lo[8];
      split_pack16(v, hi, lo);
      store_packed_part(tS + lane_sel, slot, part, hi, lo);
    }
    store_zero_parts(tS + lane_sel, slot, hf);
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    if (warp == 0 && elect_one()) {
      tc_fence_after();
      mma_ts3(tO, tS, sb + T_VH * TILE, sb + T_VL * TILE, idO);
      umma_commit(smem_u32(&mma_bar));
    }
    __syncwarp();
    const float lsum = xsum[0][r] + xsum[1][r];
    const float inv_l = row_ok ? 1.f / lsum : 0.f;
    if (row_ok && hf == 0 && a.stats) {
      const int64_t sr = ((int64_t)item * a.L + i) * 2;
      a.stats[sr] = m;
      a.stats[sr + 1] = inv_l;
    }
    mbar_wait(smem_u32(&mma_bar), ph);
    ph ^= 1;
    tc_fence_after();
    {
      const float mul = inv_l / (a.pscale * sV);
      const int b = item / a.h, hh = item - b * a.h;
      float* dst = a.out + ((int64_t)b * a.L + i) * a.ldo + hh * DK + hf * 32;
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
    __syncthreads();  // tensor memory and the tiles are free for the next pair
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, 256);
  }
}

// =================================================================================================== backward
// TMEM columns: phase 1: S [0,128) -> dS hi [0,64) | lo [64,128);  dP~ [128,256);  dQ [256,320)
//               phase 2: S^T [0,128) -> P~^T hi | lo;  dP~^T [128,256) -> dS^T hi | lo;  dV [320,384);  dK [384,448)
__global__ void __launch_bounds__(THREADS, 1) attn_pair_bwd_kernel(const PairArgs a, int n_pairs) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t mma_bar;
  __shared__ uint32_t tmem_base_slot;
  __shared__ unsigned maxbits[5];   // tiles q, k, v, dO; [4] = max |dS|
  __shared__ float row_m[128], row_inv[128], row_delta[128];
  const uint64_t site_e = rbm_site(a.site);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* sm = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t sb = smem_u32(sm);
  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&mma_bar), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) tmem_alloc(smem_u32(&tmem_base_slot), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_slot, tS = tmem, tP = tmem + 128, tDQ = tmem + 256, tDV = tmem + 320, tDK = tmem + 384;
  const uint32_t idS = make_idesc_f16(128, 128, 0, 0), idO = make_idesc_f16(128, DK, 0, 1);
  const int q4 = warp & 3, hf = warp >> 2;
  const int r = q4 * 32 + lane, slot = r >> 6, i = r & 63;
  const uint32_t lane_sel = (uint32_t)(q4 * 32) << 16;
  uint32_t ph = 0;
  for (int pair = blockIdx.x; pair < n_pairs; pair += gridDim.x) {
    if (threadIdx.x < 5) maxbits[threadIdx.x] = 0u;
    __syncthreads();
    const int item = 2 * pair + slot;
    const bool it_ok = item < a.n_items, row_ok = it_ok && i < a.L;
    const int b = it_ok ? item / a.h : 0, hh = it_ok ? item - b * a.h : 0;
    float sQ, sK, sV, sG;
    {  // global fp32 -> split fp16 tiles, two tiles in flight
      float va[4][8], vb[4][8];
      tile_max(tile_fetch(va, a.q, a.ldq, a.scale * RBM_LOG2E, pair, a), &maxbits[0]);
      tile_max(tile_fetch(vb, a.k, a.ldk, 1.f, pair, a), &maxbits[1]);
      __syncthreads();
      sQ = tile_scale_of(&maxbits[0]);
      sK = tile_scale_of(&maxbits[1]);
      tile_store(va, sQ, sm + T_QH * TILE, sm + T_QL * TILE);
      tile_max(tile_fetch(va, a.v, a.ldv, 1.f, pair, a), &maxbits[2]);
      tile_store(vb, sK, sm + T_KH * TILE, sm + T_KL * TILE);
      tile_max(tile_fetch(vb, a.dout, a.lddo, 1.f, pair, a), &maxbits[3]);
      __syncthreads();
      sV = tile_scale_of(&maxbits[2]);
      sG = tile_scale_of(&maxbits[3]);
      tile_store(va, sV, sm + T_VH * TILE, sm + T_VL * TILE);
      tile_store(vb, sG, sm + T_GH * TILE, sm + T_GL * TILE);
    }
    fence_proxy_async();
    __syncthreads();
    // ---------------------------------------------------------------------------------- phase 1: lanes = queries
    if (warp == 0 && elect_one()) {
      tc_fence_after();
      mma_ss3(tS, sb + T_QH * TILE, sb + T_QL * TILE, sb + T_KH * TILE, sb + T_KL * TILE, idS);  // S = Q.K^T
      mma_ss3(tP, sb + T_GH * TILE, sb + T_GL * TILE, sb + T_VH * TILE, sb + T_VL * TILE, idS);  // dP~ = dO.V^T
      umma_commit(smem_u32(&mma_bar));
    }
    __syncwarp();
    const float us = 1.f / (sQ * sK), up = 1.f / (sG * sV);
    const float keep = a.thr16 ? a.inv_keep : 1.f;
    if (hf == 0) {  // row statistics and delta_i = <dO_i, O_i> (from HBM, fp32) while the tensor core works
      float m = 0.f, inv = 0.f, delta = 0.f;
      if (row_ok) {
        const int64_t sr = ((int64_t)item * a.L + i) * 2;
        m = a.stats_in[sr];
        inv = a.stats_in[sr + 1];
        const float* po = a.o + ((int64_t)b * a.L + i) * a.ldo + hh * DK;
        const float* pg = a.dout + ((int64_t)b * a.L + i) * a.lddo + hh * DK;
#pragma unroll
        for (int c = 0; c < DK; c += 4) {
          const float4 x = ld4(pg + c);
          const float2 y0 = *reinterpret_cast<const float2*>(po + c), y1 = *reinterpret_cast<const float2*>(po + c + 2);
          delta = fmaf(x.x, y0.x, delta); delta = fmaf(x.y, y0.y, delta); delta = fmaf(x.z, y1.x, delta); delta = fmaf(x.w, y1.y, delta);
        }
      }
      row_m[r] = m; row_inv[r] = inv; row_delta[r] = delta;
    }
    __syncthreads();
    float ds[32];
    {
      const float m = row_m[r], inv = row_inv[r], delta = row_delta[r];
      mbar_wait(smem_u32(&mma_bar), ph);
      ph ^= 1;
      tc_fence_after();
      float mx = 0.f;
#pragma unroll
      for (int pp = 0; pp < 2; ++pp) {
        const int part = 2 * hf + pp;
        float(&v)[16] = *reinterpret_cast<float(*)[16]>(&ds[pp * 16]);
        float dp[16];
        tmem_ld16(tS + lane_sel + (uint32_t)(slot * 64 + part * 16), v);
        tmem_ld16(tP + lane_sel + (uint32_t)(slot * 64 + part * 16), dp);
        uint32_t bits = 0xffffu;
        if (a.thr16) bits = keep_bits_row(a.seed, site_e, (uint64_t)(it_ok ? item : 0), i, part, a.thr16);
#pragma unroll
        for (int jj = 0; jj < 16; ++jj) {
          const int j = part * 16 + jj;
          const bool ok = row_ok && j < a.L && (!a.causal || j <= i);
          const float p = ok ? ex2(v[jj] * us - m) * inv : 0.f;
          const float mk = ((bits >> jj) & 1u) ? keep : 0.f;
          v[jj] = p * (mk * dp[jj] * up - delta);
          mx = fmaxf(mx, fabsf(v[jj]));
        }
      }
      mx = warp_max(mx);
      if (lane == 0 && mx > 0.f) atomicMax(&maxbits[4], __float_as_uint(mx));
    }
    __syncthreads();  // max |dS| is known; every score / dP~ column has been read and may be overwritten
    const float sd = pow2_scale(__uint_as_float(maxbits[4]), 14);
#pragma unroll
    for (int pp = 0; pp < 2; ++pp) {
      float(&v)[16] = *reinterpret_cast<float(*)[16]>(&ds[pp * 16]);
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) v[jj] *= sd;
      uint32_t hi[8], lo[8];
      split_pack16(v, hi, lo);
      store_packed_part(tS + lane_sel, slot, 2 * hf + pp, hi, lo);
    }
    store_zero_parts(tS + lane_sel, slot, hf);
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    if (warp == 0 && elect_one()) {
      tc_fence_after();
      mma_ts3(tDQ, tS, sb + T_KH * TILE, sb + T_KL * TILE, idO);  // dQ = dS.K
      umma_commit(smem_u32(&mma_bar));
    }
    __syncwarp();
    mbar_wait(smem_u32(&mma_bar), ph);
    ph ^= 1;
    tc_fence_after();
    {
      const float mul = a.scale / (sd * sK);
      float* dst = a.dq + ((int64_t)b * a.L + i) * a.lddq + hh * DK + hf * 32;
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
    __syncthreads();
    // ------------------------------------------------------------------------------------- phase 2: lanes = keys
    if (warp == 0 && elect_one()) {
      tc_fence_after();
      mma_ss3(tS, sb + T_KH * TILE, sb + T_KL * TILE, sb + T_QH * TILE, sb + T_QL * TILE, idS);  // S^T = K.Q^T
      mma_ss3(tP, sb + T_VH * TILE, sb + T_VL * TILE, sb + T_GH * TILE, sb + T_GL * TILE, idS);  // dP~^T = V.dO^T
      umma_commit(smem_u32(&mma_bar));
    }
    __syncwarp();
    float pt[32];  // P~^T of this key for the queries [32 hf, 32 hf + 32) (scaled); ds[] is reused for dS^T
    {
      const int j = i;  // this lane's key
      const bool key_ok = it_ok && j < a.L;
      mbar_wait(smem_u32(&mma_bar), ph);
      ph ^= 1;
      tc_fence_after();
#pragma unroll
      for (int pp = 0; pp < 2; ++pp) {
        const int T = 2 * hf + pp;
        float(&v)[16] = *reinterpret_cast<float(*)[16]>(&ds[pp * 16]);
        float(&pv)[16] = *reinterpret_cast<float(*)[16]>(&pt[pp * 16]);
        float dp[16];
        tmem_ld16(tS + lane_sel + (uint32_t)(slot * 64 + T * 16), v);
        tmem_ld16(tP + lane_sel + (uint32_t)(slot * 64 + T * 16), dp);
        uint32_t bits = 0xffffu;
        if (a.thr16) bits = keep_bits_col(a.seed, site_e, (uint64_t)(it_ok ? item : 0), j, T, a.thr16);
#pragma unroll
        for (int ii = 0; ii < 16; ++ii) {
          const int qi = T * 16 + ii, qr = slot * 64 + qi;
          const bool ok = key_ok && qi < a.L && (!a.causal || j <= qi);
          const float p = ok ? ex2(v[ii] * us - row_m[qr]) * row_inv[qr] : 0.f;
          const float mk = ((bits >> ii) & 1u) ? keep : 0.f;
          pv[ii] = p * mk * a.pscale;
          v[ii] = p * (mk * dp[ii] * up - row_delta[qr]) * sd;
        }
      }
    }
    __syncthreads();  // every S^T / dP~^T column has been read
#pragma unroll
    for (int pp = 0; pp < 2; ++pp) {
      uint32_t hi[8], lo[8];
      split_pack16(*reinterpret_cast<float(*)[16]>(&pt[pp * 16]), hi, lo);
      store_packed_part(tS + lane_sel, slot, 2 * hf + pp, hi, lo);
      split_pack16(*reinterpret_cast<float(*)[16]>(&ds[pp * 16]), hi, lo);
      store_packed_part(tP + lane_sel, slot, 2 * hf + pp, hi, lo);
    }
    store_zero_parts(tS + lane_sel, slot, hf);
    store_zero_parts(tP + lane_sel, slot, hf);
    tmem_st_wait();
    tc_fence_before();
    __syncthreads();
    if (warp == 0 && elect_one()) {
      tc_fence_after();
      mma_ts3(tDV, tS, sb + T_GH * TILE, sb + T_GL * TILE, idO);  // dV = P~^T.dO
      mma_ts3(tDK, tP, sb + T_QH * TILE, sb + T_QL * TILE, idO);  // dK = dS^T.Q
      umma_commit(smem_u32(&mma_bar));
    }
    __syncwarp();
    mbar_wait(smem_u32(&mma_bar), ph);
    ph ^= 1;
    tc_fence_after();
    {
      const bool key_ok = it_ok && i < a.L;
      const float mv = 1.f / (a.pscale * sG), mkk = 1.f / (sd * sQ * RBM_LOG2E);  // the q tile holds q * scale * log2(e)
      float* dstv = a.dv + ((int64_t)b * a.L + i) * a.lddv + hh * DK + hf * 32;
      float* dstk = a.dk_ + ((int64_t)b * a.L + i) * a.lddk + hh * DK + hf * 32;
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
    __syncthreads();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

float pscale_for(float inv_keep) { return pow2_scale(inv_keep, 14); }  // P~ <= inv_keep, so P~ * pscale < 2^14

}  // namespace

bool rbm_attn_pair_supported(int L, int dk, int mask_mode) {
  return rbm_attn_tc_enabled() && dk == DK && L >= 1 && L <= 64 && (mask_mode == RBM_MASK_NONE || mask_mode == RBM_MASK_CAUSAL);
}

int rbm_attn_pair_fwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, float* out, int64_t ldo,
                      float* stats, int B, int L, int h, int mask_mode, float scale, float p, uint64_t seed, uint64_t site, cudaStream_t st) {
  PairArgs a{};
  a.q = q; a.k = k; a.v = v; a.out = out; a.stats = stats; a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo;
  a.L = L; a.h = h; a.n_items = B * h; a.causal = mask_mode == RBM_MASK_CAUSAL; a.scale = scale;
  a.thr16 = rbm_drop_threshold16(p); a.inv_keep = 1.f / (1.f - p); a.pscale = pscale_for(a.inv_keep); a.seed = seed; a.site = site;
  const int n_pairs = (a.n_items + 1) / 2;
  const size_t smem = 6 * TILE + 1024;
  if (!set_smem(attn_pair_fwd_kernel, smem, "rbm_attn_fwd(pair)")) return -1;
  const int grid = n_pairs < 2 * RBM_NUM_SMS ? n_pairs : 2 * RBM_NUM_SMS;  // two CTAs per SM: one stages while the other computes
  attn_pair_fwd_kernel<<<grid, THREADS, smem, st>>>(a, n_pairs);
  RBM_LAUNCH_CHECK("rbm_attn_fwd(pair)");
  return 0;
}

int rbm_attn_pair_bwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const float* out, int64_t ldo,
                      const float* dout, int64_t lddo, const float* stats, float* dq, int64_t lddq, float* dk_, int64_t lddk, float* dv,
                      int64_t lddv, int B, int L, int h, int mask_mode, float scale, float p, uint64_t seed, uint64_t site, cudaStream_t st) {
  PairArgs a{};
  a.q = q; a.k = k; a.v = v; a.o = out; a.dout = dout; a.stats_in = stats; a.dq = dq; a.dk_ = dk_; a.dv = dv;
  a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo; a.lddo = lddo; a.lddq = lddq; a.lddk = lddk; a.lddv = lddv;
  a.L = L; a.h = h; a.n_items = B * h; a.causal = mask_mode == RBM_MASK_CAUSAL; a.scale = scale;
  a.thr16 = rbm_drop_threshold16(p); a.inv_keep = 1.f / (1.f - p); a.pscale = pscale_for(a.inv_keep); a.seed = seed; a.site = site;
  const int n_pairs = (a.n_items + 1) / 2;
  const size_t smem = 8 * TILE + 1024;
  if (!set_smem(attn_pair_bwd_kernel, smem, "rbm_attn_bwd(pair)")) return -1;
  const int grid = n_pairs < RBM_NUM_SMS ? n_pairs : RBM_NUM_SMS;
  attn_pair_bwd_kernel<<<grid, THREADS, smem, st>>>(a, n_pairs);
  RBM_LAUNCH_CHECK("rbm_attn_bwd(pair)");
  return 0;
}

RBM_DEFINE_STEP_PTR_SETTER(rbm_step_ptr_set_attention_pair)
