// attention_f16.cuh -- pieces shared by the split-fp16 tcgen05 attention kernels of attention_pair.cu and attention_seq.cu:
// staging of 128 x 64 operand tiles, the three-pass product of two staged tiles, and the dropout keep bits in the layout of
// the library's attention Philox contract (common.cuh, rbm_attn_keep).
#pragma once
#include "common.cuh"
#include "tc_ptx.cuh"
#include "split16.cuh"

namespace rbm_attn16 {

constexpr int THREADS = 256;  // block size of every kernel; tile_store's thread tasks assume it

// scale, split and store into the hi / lo tiles [128 rows x 64 columns] (128-byte swizzle: 16-byte chunk c of row r lands at
// chunk c ^ (r & 7)).  Thread task (row r, chunk c) covers 8 consecutive columns.
__device__ __forceinline__ void tile_store(const float (&v)[4][8], float sc, uint8_t* hi, uint8_t* lo) {
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int task = it * THREADS + (int)threadIdx.x, r = task >> 3, c = task & 7;
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) rbm_tc::split2(v[it][2 * e] * sc, v[it][2 * e + 1] * sc, h[e], l[e]);
    const uint32_t off = (uint32_t)r * 128u + (uint32_t)((c ^ (r & 7)) << 4);
    *reinterpret_cast<uint4*>(hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}
// this thread's share of the tile maximum -> block maximum (shared-memory atomicMax on the bit pattern: order-independent)
__device__ __forceinline__ void tile_max(float mx, unsigned* maxbits) {
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(maxbits, __float_as_uint(mx));
}

// D[128 x N] = A_tile (K-major, 128 rows) . B_tile^T (K-major, N rows), contraction over d_k = 64 (four k-steps of 16); three
// passes
__device__ __forceinline__ void mma_ss3(uint32_t d_t, uint32_t a_hi, uint32_t a_lo, uint32_t b_hi, uint32_t b_lo, uint32_t idesc) {
  uint32_t acc = 0;
#pragma unroll
  for (int pass = 0; pass < 3; ++pass) {
    const uint64_t ad = rbm_tc::make_sw128_desc(pass == 2 ? a_lo : a_hi), bd = rbm_tc::make_sw128_desc(pass == 1 ? b_lo : b_hi);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      rbm_tc::umma_f16(d_t, ad + (uint64_t)(k * 2), bd + (uint64_t)(k * 2), idesc, acc);
      acc = 1;
    }
  }
}

// keep decisions of query row i for the 16 keys [16 np, 16 np + 16): bit (8 n1 + 2 t + e) of the result.  Rows i and i ^ 8
// (lanes l and l ^ 8) share their four Philox calls: the rh = 0 lane computes t = 0, 1, the rh = 1 lane t = 2, 3, and they
// trade the two words the other row's fields live in.  Must be called by both lanes together.
__device__ __forceinline__ uint32_t keep_bits_row(uint64_t seed, uint64_t site, uint64_t bh, int i, int np, uint32_t thr16) {
  const int rh = (i >> 3) & 1, g = i & 7, tile = i >> 4;
  uint32_t own[2][2], got[2][2];  // [tt][e]: words holding MY fields (low half n1 = 0, high half n1 = 1) of call t = 2 rh + tt (own)
                                  // and of my partner's call t = 2 (1 - rh) + tt (got)
#pragma unroll
  for (int tt = 0; tt < 2; ++tt) {
    const uint4 r = rbm_philox_drop(seed, site, rbm_attn_call(bh, tile, g, 2 * rh + tt, np));
    own[tt][0] = rh ? r.z : r.x;
    own[tt][1] = rh ? r.w : r.y;
    got[tt][0] = __shfl_xor_sync(0xffffffffu, rh ? r.x : r.z, 8);  // my partner's words of my call <-> mine of theirs
    got[tt][1] = __shfl_xor_sync(0xffffffffu, rh ? r.y : r.w, 8);
  }
  uint32_t bits = 0;
#pragma unroll
  for (int t = 0; t < 4; ++t)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const uint32_t w = ((t >> 1) == rh) ? own[t & 1][e] : got[t & 1][e];
#pragma unroll
      for (int n1 = 0; n1 < 2; ++n1)
        if (((w >> (16 * n1)) & 0xffffu) >= thr16) bits |= 1u << (8 * n1 + 2 * t + e);
    }
  return bits;
}
// keep decisions of key j for the 16 queries [16 T, 16 T + 16): bit (g + 8 rh) of the result
__device__ __forceinline__ uint32_t keep_bits_col(uint64_t seed, uint64_t site, uint64_t bh, int j, int T, uint32_t thr16) {
  const int t = (j & 7) >> 1, e = j & 1, n1 = (j >> 3) & 1, np = j >> 4;
  uint32_t bits = 0;
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    const uint4 r = rbm_philox_drop(seed, site, rbm_attn_call(bh, T, g, t, np));
    const uint32_t w0 = e ? r.y : r.x, w1 = e ? r.w : r.z;  // rh = 0 / rh = 1
    if (((w0 >> (16 * n1)) & 0xffffu) >= thr16) bits |= 1u << g;
    if (((w1 >> (16 * n1)) & 0xffffu) >= thr16) bits |= 1u << (g + 8);
  }
  return bits;
}

}  // namespace rbm_attn16
