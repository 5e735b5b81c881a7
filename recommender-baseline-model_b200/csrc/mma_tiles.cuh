// mma_tiles.cuh -- warp-level tensor-core tile primitives shared by the attention and scoring kernels.
//   * mma.sync m16n8k8 TF32 with 3xTF32 error compensation (fp32-level accuracy; -DRBM_ATTN_TF32X1: single pass);
//   * XOR-swizzled shared-memory "panels" [rows][LD] that serve both B-fragment access patterns conflict-free:
//       load_b_nk : contraction along the panel's columns  (scores = tile . panel^T)
//       load_b_kn : contraction along the panel's rows     (out    = weights . panel)
//   * per-warp row-major tiles [16][ld] as A operands.
#pragma once
#include "common.cuh"

namespace rbm_mma {

constexpr int CH = 64;         // columns per chunk = 8 mma n-tiles
constexpr int PB_LD = CH + 4;  // per-warp weight/probability tile row stride (== 4*odd mod 32: conflict-free A fragments)

__device__ __forceinline__ int swz(int r) { return (((r & 3) << 1) | ((r >> 2) & 1)) << 2; }

// 3xTF32 operand split.  The tensor core reads only the upper 19 bits of a tf32 operand, so hi = x with the low 13
// mantissa bits cleared (one LOP3; cvt.rna.tf32 is emulated with ~10 integer instructions on sm_100) and lo = x - hi,
// which is exact in fp32 and is itself truncated by the hardware to its top 11 significant bits: the dropped part is
// O(2^-22 |x|), the same order as the lo*lo term 3xTF32 neglects anyway.
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(tf32_lo(x));
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
struct FragA {
  uint32_t hi[4], lo[4];
};
struct FragB {
  uint32_t hi[2], lo[2];
};
__device__ __forceinline__ void mma3(float (&d)[4], const FragA& a, const FragB& b) {
#ifndef RBM_ATTN_TF32X1
  mma_tf32(d, a.lo, b.hi);
  mma_tf32(d, a.hi, b.lo);
#endif
  mma_tf32(d, a.hi, b.hi);
}

// A fragment (16 x 8) of a row-major per-warp tile [16][ld] at column k0
__device__ __forceinline__ FragA load_a(const float* tile, int ld, int k0, int g, int t) {
  FragA f;
  split_tf32(tile[g * ld + k0 + t], f.hi[0], f.lo[0]);
  split_tf32(tile[(g + 8) * ld + k0 + t], f.hi[1], f.lo[1]);
  split_tf32(tile[g * ld + k0 + t + 4], f.hi[2], f.lo[2]);
  split_tf32(tile[(g + 8) * ld + k0 + t + 4], f.hi[3], f.lo[3]);
  return f;
}
// B fragment, contraction along the panel's COLUMNS: B[k][n] = panel[n0 + n][k0 + k]
__device__ __forceinline__ FragB load_b_nk(const float* panel, int LD, int n0, int k0, int g, int t) {
  const float* row = panel + (n0 + g) * LD;
  int c0 = (k0 ^ swz(g)) + t;  // == (k0 + t) ^ swz(g): k0 is a multiple of 8, the swizzle touches bits 2..4 only
  FragB f;
  split_tf32(row[c0], f.hi[0], f.lo[0]);
  split_tf32(row[c0 ^ 4], f.hi[1], f.lo[1]);
  return f;
}
// B fragment, contraction along the panel's ROWS: B[k][n] = panel[k0 + k][n0 + n]
__device__ __forceinline__ FragB load_b_kn(const float* panel, int LD, int k0, int n0, int g, int t) {
  FragB f;
  split_tf32(panel[(k0 + t) * LD + ((n0 + g) ^ swz(t))], f.hi[0], f.lo[0]);
  split_tf32(panel[(k0 + t + 4) * LD + ((n0 + g) ^ swz(t + 4))], f.hi[1], f.lo[1]);
  return f;
}

// panel[LP8][LD] (swizzled) <- rows (row0 + r) of src, columns [col0, col0 + dk), times mul; rows >= L are zero
__device__ __forceinline__ void load_panel(float* dst, const float* __restrict__ src, int64_t ld, int64_t row0, int col0, int L,
                                           int LP8, int dk, int LD, float mul) {
  int dk4 = dk >> 2;
  for (int idx = threadIdx.x; idx < LP8 * dk4; idx += blockDim.x) {
    int r = idx / dk4, c4 = idx - r * dk4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < L) v = ld4(src + (row0 + r) * ld + col0 + c4 * 4);
    st4(dst + r * LD + ((c4 * 4) ^ swz(r)), make_float4(v.x * mul, v.y * mul, v.z * mul, v.w * mul));
  }
}
// per-warp tile[16][ldt] <- rows (row0 + i0 + r), r < 16
__device__ __forceinline__ void stage_tile(float* dst, int ldt, const float* __restrict__ src, int64_t ld, int64_t row0, int col0,
                                           int i0, int L, int dk, float mul, int lane) {
  int dk4 = dk >> 2;
  for (int idx = lane; idx < 16 * dk4; idx += 32) {
    int r = idx / dk4, c4 = idx - r * dk4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i0 + r < L) v = ld4(src + (row0 + i0 + r) * ld + col0 + c4 * 4);
    st4(dst + r * ldt + c4 * 4, make_float4(v.x * mul, v.y * mul, v.z * mul, v.w * mul));
  }
}

__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}
__device__ __forceinline__ bool masked_inf(int mode, int i, int j, int L) { return j >= L || (mode == RBM_MASK_CAUSAL && j > i); }
// Scores are kept in the log2 domain (q is pre-multiplied by scale*log2(e)): softmax needs one ex2.approx per element.
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
#define RBM_LOG2E 1.4426950408889634f
#define RBM_LN2 0.6931471805599453f
#define RBM_PADFILL (-1.0e9f * RBM_LOG2E)  // masked_fill(mask == 0, -1e9) expressed in the log2 domain

// acc[nt] (+)= Atile(16 x dk) . panel[jb + nt*8 .. +8][0..dk)^T  for nt < 8
__device__ __forceinline__ void tile_dot_panel(float (&acc)[8][4], const float* atile, int lda, const float* panel, int LD, int jb,
                                               int LP8, int dk, int g, int t) {
  for (int k0 = 0; k0 < dk; k0 += 8) {
    FragA a = load_a(atile, lda, k0, g, t);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      if (jb + nt * 8 < LP8) {
        FragB b = load_b_nk(panel, LD, jb + nt * 8, k0, g, t);
        mma3(acc[nt], a, b);
      }
    }
  }
}
// acc[dt] += Ptile(16 x 64 chunk) . panel[jb .. jb+64][dt*8 .. +8]   for dt*8 < dk
template <int DT>
__device__ __forceinline__ void ptile_times_panel(float (&acc)[DT][4], const float* ptile, const float* panel, int LD, int jb, int LP8,
                                                  int dk, int g, int t) {
#pragma unroll
  for (int ks = 0; ks < 8; ++ks) {
    if (jb + ks * 8 < LP8) {
      FragA a = load_a(ptile, PB_LD, ks * 8, g, t);
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        if (dt * 8 < dk) {
          FragB b = load_b_kn(panel, LD, jb + ks * 8, dt * 8, g, t);
          mma3(acc[dt], a, b);
        }
      }
    }
  }
}


}  // namespace rbm_mma
