// tc_topk.cu -- full-catalogue scoring fused with candidate selection on the Blackwell tensor path, plus the exact
// fp32 re-scoring of the survivors.  Replaces, at catalogue scale, SAS.predict's gather+matvec / BERT's last-position
// logits followed by argsort(-scores)[:, :k] (NN/models/sas_model/sas.py:110-114, NN/trainers/bert.py:47-49,
// NN/trainers/utils.py:36-38): the [U, V] score matrix never exists anywhere but in tensor memory.
//
//   stage 0 (d % 64 == 0): one pass over the item range finds max |x| and the largest row norm, a second writes a range-scaled
//     fp16 copy of the rows (per-tensor power of two: max |x| -> [2^14, 2^15)); the user rows likewise.  fp16 rounds to 11
//     significant bits (TF32 operands are TRUNCATED to 11), the tensor core runs kind::f16 at twice the TF32 rate with
//     K = 16 per instruction, and the streamed tiles are half the bytes.  (d = 32: kind::tf32 on the fp32 data, as before.)
//   stage 1 (tc_topk_kernel): persistent CTAs walk (user tile, item split) units; for d <= 64 a user tile is two 128-row
//     sub-tiles that share every streamed item tile.  The user tile is TMA-loaded once
//     per unit and stays in shared memory; item-table tiles ([BN items x d], K-major, 128-byte swizzle) stream through
//     a TMA ring; one tcgen05.mma pass (this stage only has to be right about WHO is near the top)
//     writes [128 x BN] score tiles into double-buffered TMEM; 8 epilogue warps (one thread per user row, tcgen05.ld)
//     compare every score with the thread's running KC-th best (one FMNMX per score) and insert the rare survivors into
//     a register-resident sorted list of KC = 16 (approx score, item id) candidates per (item split, column half).
//   stage 2 (topk_rescore_kernel): one warp per user recomputes the EXACT fp32 score of every candidate (sequential
//     fp32 FMA over d) and selects the final top-k under the canonical order (score desc, id asc).
//   certificate: stage 1 ranks by single-pass reduced-precision scores: |approximate - fp32 score| <= eps(u) =
//     c * ||f_u|| * max_v ||table_v|| by Cauchy-Schwarz over the per-product operand error, c = 1.05e-3 for fp16 operands
//     (rounded: 2^-11 each) and 2.1e-3 for TF32 (truncated: 2^-10 each), both including the fp32 accumulation slack.  An item a list dropped has an approximate score <= tau = that list's final
//     KC-th entry, hence an exact score <= tau + eps.  Stage 2 therefore PROVES its answer for user u when
//     max_lists(tau) + eps(u) < (exact k-th best score); every other user is appended to a device-side list and
//     re-ranked by the exact fp32 scan kernel of topk.cu (stage 3, no host synchronisation; its grid exits at once
//     when the list is empty).  The result always equals the canonical (fp32 score desc, id asc) top-k, where the fp32
//     score is the sequential FMA over the hidden dimension (the arithmetic of stage 2 and of the scan kernel).
#include <cuda_fp16.h>
#include <stdlib.h>
#include <type_traits>
#include "common.cuh"
#include "tc_ptx.cuh"
#include "split16.cuh"
#include "tc_topk.cuh"

namespace {

using namespace rbm_tc;

constexpr int BM = 128;
constexpr int KC = 16;       // candidates kept per (user, item split, column half)
constexpr int EPI = 8;       // epilogue warps

struct TopkParams {
  const float* bias;
  const float* scales;  // F16 path: [0] = scale of the item rows, [1] = of the user rows (scores and lists are in scaled units)
  float* cand_s;     // [S*2][U][KC]
  int64_t* cand_i;   // [S*2][U][KC]
  int64_t U, v_begin, v_end, id_offset, tiles_per_split, row_base;  // row_base: table row of the kernel's row 0
  int d, BN, nstage, S, n_utiles;
  int nst;  // 128-row user sub-tiles per unit: 2 (d <= 64: 256 users share every streamed item tile) or 1
  uint32_t tmem_cols;
};
// the exclusion path's parameters extend the struct instead of growing it: the kernels without exclusion keep their code
struct TopkExclParams : TopkParams {
  const int64_t* excl;  // row u = user u's excluded output ids, ascending (row stride ld_excl, n_excl entries)
  int64_t ld_excl;
  int n_excl;
};

// first index of the ascending row ex[0 .. n) whose id is >= key (n when none)
__device__ __forceinline__ int excl_lower_bound(const int64_t* __restrict__ ex, int n, int64_t key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (ex[mid] < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

// F16: operands are the range-scaled fp16 copies (64 elements per 128-byte row, K = 16 per instruction, kind::f16);
// otherwise the fp32 data itself (32 elements per row, K = 8, kind::tf32).
// EX: items of the user's exclusion row never enter a candidate list.  The filter sits on the rare insertion path only: a
// thread meets its item ids in ascending order within a unit, so a cursor into the sorted row (next excluded id in a
// register) advances monotonically and reads each entry at most once per unit.
template <bool F16, bool EX>
__global__ void __launch_bounds__(64 + 32 * EPI, 1) tc_topk_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                                                                   const std::conditional_t<EX, TopkExclParams, TopkParams> p) {
  constexpr int BKE = F16 ? 64 : 32;      // elements per 128-byte K block
  constexpr int ESZ = F16 ? 2 : 4;
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t a_full, a_empty, full_bar[4], empty_bar[4], tfull[2], tempty[2];
  __shared__ uint32_t tmem_base_slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int KB = p.d / BKE, BN = p.BN, ns = p.nstage;
  const int NST = p.nst;
  const uint32_t a_sub = (uint32_t)KB * BM * BKE * ESZ, a_bytes = a_sub * NST, kb_bytes = (uint32_t)BN * BKE * ESZ, stage_bytes = kb_bytes * KB;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int64_t n_items = p.v_end - p.v_begin;
  const int64_t n_tiles = (n_items + BN - 1) / BN;
  const int n_units = p.n_utiles * p.S;

  if (threadIdx.x == 0) {
    mbar_init(smem_u32(&a_full), 1);
    mbar_init(smem_u32(&a_empty), 1);
    for (int s = 0; s < ns; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tfull[b]), 1);
      mbar_init(smem_u32(&tempty[b]), EPI);
    }
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
      int g = 0, un = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++un) {
        const int ut = u / p.S, sp = u % p.S;
        if (un > 0) mbar_wait(smem_u32(&a_empty), (un - 1) & 1);  // the previous unit's MMAs no longer read the user tile
        mbar_expect_tx(smem_u32(&a_full), a_bytes);
        for (int st = 0; st < NST; ++st)
          for (int kb = 0; kb < KB; ++kb)
            tma_load_2d(smem_base + st * a_sub + kb * BM * BKE * ESZ, &mapA, smem_u32(&a_full), kb * BKE, (ut * NST + st) * BM);
        const int64_t tb = (int64_t)sp * p.tiles_per_split;
        const int64_t te = tb + p.tiles_per_split < n_tiles ? tb + p.tiles_per_split : n_tiles;
        for (int64_t t = tb; t < te; ++t, ++g) {
          const int s = g % ns;
          if (g >= ns) mbar_wait(smem_u32(&empty_bar[s]), ((g / ns) - 1) & 1);
          const uint32_t bar = smem_u32(&full_bar[s]);
          mbar_expect_tx(bar, stage_bytes);
          for (int kb = 0; kb < KB; ++kb)
            tma_load_2d(smem_base + a_bytes + s * stage_bytes + kb * kb_bytes, &mapB, bar, kb * BKE, (int)(p.v_begin + t * BN));
        }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      const uint32_t idesc = F16 ? make_idesc_f16(BM, BN, 0, 0) : make_idesc_tf32(BM, BN, 0, 0);
      int g = 0, it = 0, un = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x, ++un) {
        const int sp = u % p.S;
        mbar_wait(smem_u32(&a_full), un & 1);
        const int64_t tb = (int64_t)sp * p.tiles_per_split;
        const int64_t te = tb + p.tiles_per_split < n_tiles ? tb + p.tiles_per_split : n_tiles;
        for (int64_t t = tb; t < te; ++t, ++g, ++it) {
          const int s = g % ns, buf = it & 1;
          if (it >= 2) {
            mbar_wait(smem_u32(&tempty[buf]), ((it >> 1) - 1) & 1);
            tc_fence_after();
          }
          mbar_wait(smem_u32(&full_bar[s]), (g / ns) & 1);
          tc_fence_after();
          for (int st = 0; st < NST; ++st) {  // every user sub-tile against the same streamed item tile
            const uint32_t d = tmem_d + (uint32_t)((buf * NST + st) * BN);
            for (int kb = 0; kb < KB; ++kb) {
              const uint64_t adesc = make_sw128_desc(smem_base + st * a_sub + kb * BM * BKE * ESZ);
              const uint64_t bdesc = make_sw128_desc(smem_base + a_bytes + s * stage_bytes + kb * kb_bytes);
#pragma unroll
              for (int k = 0; k < 4; ++k) {  // four 32-byte K steps per 128-byte row
                if (F16) umma_f16(d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
                else umma_tf32(d, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) != 0);
              }
            }
          }
          umma_commit(smem_u32(&empty_bar[s]));
          umma_commit(smem_u32(&tfull[buf]));
        }
        umma_commit(smem_u32(&a_empty));
      }
    }
    __syncwarp();
  } else {
    const int q = warp & 3, half = (warp - 2) >> 2;
    // two user sub-tiles: the second group of four warps owns sub-tile 1 and every thread scans all BN columns;
    // one sub-tile: the two groups split the columns
    const int st = NST == 2 ? half : 0, chalf = NST == 2 ? 0 : half;
    const int hw = NST == 2 ? BN : BN / 2;  // columns per thread and tile
    const float bscale = F16 ? p.scales[0] * p.scales[1] : 1.f;  // the bias joins the scores in their (scaled) units
    int it = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int ut = u / p.S, sp = u % p.S;
      const int64_t user = ((int64_t)ut * NST + st) * BM + q * 32 + lane;
      float ls[KC];
      int li[KC];
#pragma unroll
      for (int t = 0; t < KC; ++t) {
        ls[t] = -INFINITY;
        li[t] = -1;
      }
      const int64_t tb = (int64_t)sp * p.tiles_per_split;
      const int64_t te = tb + p.tiles_per_split < n_tiles ? tb + p.tiles_per_split : n_tiles;
      // EX cursor: ex_row[ex_pos] = ex_next is the first excluded id >= every id this thread has offered so far in the unit
      // (rows past U read nothing: n = 0, next = +inf)
      const int64_t* ex_row = nullptr;
      int ex_n = 0, ex_pos = 0;
      int64_t ex_next = INT64_MAX;
      if constexpr (EX) {
        if (user < p.U) {
          ex_row = p.excl + user * p.ld_excl;
          ex_n = p.n_excl;
          ex_pos = excl_lower_bound(ex_row, ex_n, p.v_begin + tb * BN + p.row_base + p.id_offset);
          ex_next = ex_pos < ex_n ? ex_row[ex_pos] : INT64_MAX;
        }
      }
      for (int64_t t = tb; t < te; ++t, ++it) {
        const int buf = it & 1;
        mbar_wait(smem_u32(&tfull[buf]), (it >> 1) & 1);
        tc_fence_after();
        const int64_t item0 = p.v_begin + t * BN + chalf * hw;  // table row of this thread's first column
        for (int c0 = 0; c0 < hw; c0 += 32) {
          float v[32];
          tmem_ld32(tmem_d + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * NST + st) * BN + chalf * hw + c0), v);
          if (c0 + 32 >= hw) {  // this warp's last read of the buffer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&tempty[buf]));
          }
          const int64_t r0 = item0 + c0;
          if (p.bias) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              if (r0 + j + 3 < p.v_end) {
                float4 b4 = make_float4(p.bias[r0 + j], p.bias[r0 + j + 1], p.bias[r0 + j + 2], p.bias[r0 + j + 3]);
                v[j] = fmaf(b4.x, bscale, v[j]); v[j + 1] = fmaf(b4.y, bscale, v[j + 1]);
                v[j + 2] = fmaf(b4.z, bscale, v[j + 2]); v[j + 3] = fmaf(b4.w, bscale, v[j + 3]);
              } else {
                for (int e = 0; e < 4; ++e)
                  if (r0 + j + e < p.v_end) v[j + e] = fmaf(p.bias[r0 + j + e], bscale, v[j + e]);
              }
            }
          }
          if (r0 + 32 > p.v_end) {  // ragged end of the item range: rows beyond it must never win
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (r0 + j >= p.v_end) v[j] = -INFINITY;
          }
          float mx = v[0];
#pragma unroll
          for (int j = 1; j < 32; ++j) mx = fmaxf(mx, v[j]);
          if (mx > ls[KC - 1]) {  // rare: some score of this chunk beats the running 32nd best
            float loc[32];        // dynamically indexed -> local memory, only touched on this path
            unsigned m = 0;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              loc[j] = v[j];
              m |= (v[j] > ls[KC - 1] ? 1u : 0u) << j;
            }
            for (; m; m &= m - 1) {
              const int j = __ffs(m) - 1;
              const float x = loc[j];
              if (x > ls[KC - 1]) {
                const int id = (int)(r0 + j + p.row_base);
                if constexpr (EX) {
                  const int64_t key = (int64_t)id + p.id_offset;
                  while (ex_next < key) ex_next = ++ex_pos < ex_n ? ex_row[ex_pos] : INT64_MAX;
                  if (ex_next == key) continue;
                }
                bool placed = false;
#pragma unroll
                for (int tt = KC - 1; tt > 0; --tt) {
                  if (!placed) {
                    if (ls[tt - 1] < x) {
                      ls[tt] = ls[tt - 1];
                      li[tt] = li[tt - 1];
                    } else {
                      ls[tt] = x;
                      li[tt] = id;
                      placed = true;
                    }
                  }
                }
                if (!placed) {
                  ls[0] = x;
                  li[0] = id;
                }
              }
            }
          }
        }
      }
      if (user < p.U) {
        const int64_t base = ((int64_t)(NST == 2 ? sp : sp * 2 + half) * p.U + user) * KC;
#pragma unroll
        for (int t = 0; t < KC; ++t) {
          p.cand_s[base + t] = ls[t];
          p.cand_i[base + t] = li[t] < 0 ? -1 : (int64_t)li[t];
        }
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

// ----------------------------------------------------------------------------- exact re-score + final top-k
__device__ __forceinline__ bool better(float s, int64_t id, float ts, int64_t tid) { return s > ts || (s == ts && id < tid); }

__global__ void __launch_bounds__(256) topk_rescore_kernel(const float* __restrict__ f, int64_t ldf, const float* __restrict__ table,
                                                           const float* __restrict__ bias, const int64_t* __restrict__ cand_i,
                                                           const float* __restrict__ cand_s, int n_lists, int64_t id_offset,
                                                           float* __restrict__ out_s, int64_t* __restrict__ out_i, int64_t U, int d, int k,
                                                           const unsigned* __restrict__ emax2_bits, float eps_mul, const float* __restrict__ scales,
                                                           int32_t* __restrict__ flag_list, int32_t* __restrict__ flag_count) {
  extern __shared__ float fs[];  // [8 warps][d]
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t u = (int64_t)blockIdx.x * 8 + wib;
  if (u >= U) return;
  float* fu = fs + wib * d;
  for (int c = lane; c < d; c += 32) fu[c] = f[u * ldf + c];
  __syncwarp();
  float ms = -INFINITY;       // lane t holds the t-th best (t < k)
  int64_t mi = INT64_MAX;
  const int NC = n_lists * KC;
  for (int c0 = 0; c0 < NC; c0 += 32) {
    const int c = c0 + lane;
    int64_t row = -1;
    if (c < NC) row = cand_i[((int64_t)(c / KC) * U + u) * KC + (c % KC)];
    float s = 0.f;
    if (row >= 0) {
      const float* tr = table + row * d;
      for (int kk = 0; kk < d; kk += 4) {
        float4 t4 = ld4(tr + kk);
        s = fmaf(fu[kk], t4.x, s); s = fmaf(fu[kk + 1], t4.y, s); s = fmaf(fu[kk + 2], t4.z, s); s = fmaf(fu[kk + 3], t4.w, s);
      }
      if (bias) s += bias[row];
    }
    const int64_t id = row + id_offset;
    // offer every valid candidate to the warp-distributed sorted list
    const float ts = __shfl_sync(0xffffffffu, ms, k - 1);
    const int64_t tid = __shfl_sync(0xffffffffu, mi, k - 1);
    unsigned m = __ballot_sync(0xffffffffu, row >= 0 && better(s, id, ts, tid));
    while (m) {
      const int src = __ffs(m) - 1;
      m &= m - 1;
      const float cs = __shfl_sync(0xffffffffu, s, src);
      const int64_t cid = __shfl_sync(0xffffffffu, id, src);
      const bool beats_me = better(cs, cid, ms, mi);
      const int pos = __popc(__ballot_sync(0xffffffffu, lane < k && !beats_me));
      const float up_s = __shfl_up_sync(0xffffffffu, ms, 1);
      const int64_t up_i = __shfl_up_sync(0xffffffffu, mi, 1);
      if (lane < k) {
        if (lane == pos) {
          ms = cs;
          mi = cid;
        } else if (lane > pos) {
          ms = up_s;
          mi = up_i;
        }
      }
    }
  }
  if (lane < k) {
    out_s[u * k + lane] = mi == INT64_MAX ? -INFINITY : ms;
    out_i[u * k + lane] = mi == INT64_MAX ? -1 : mi;
  }
  // certificate (see the file header): a dropped item's exact score is <= tau + eps
  float tau = -INFINITY;
  for (int l = lane; l < n_lists; l += 32) tau = fmaxf(tau, cand_s[((int64_t)l * U + u) * KC + (KC - 1)]);
  tau = warp_max(tau);
  if (scales) tau = tau / (scales[0] * scales[1]);  // the lists of the fp16 path are in scaled units (powers of two: exact)
  float hn2 = 0.f;
  for (int c = lane; c < d; c += 32) hn2 = fmaf(fu[c], fu[c], hn2);
  hn2 = warp_sum(hn2);
  const float sk = __shfl_sync(0xffffffffu, ms, k - 1);
  const bool full = __shfl_sync(0xffffffffu, mi, k - 1) != INT64_MAX;
  if (lane == 0 && tau > -INFINITY) {
    const float eps = eps_mul * sqrtf(hn2) * sqrtf(__uint_as_float(*emax2_bits)) + 1e-6f * (fabsf(sk) + fabsf(tau));
    if (!full || !(tau + eps < sk)) flag_list[atomicAdd(flag_count, 1)] = (int32_t)u;
  }
}

// max over table rows [v_begin, v_end) of the squared row norm, as the bit pattern of a non-negative float (atomicMax on
// unsigned: order-independent, hence deterministic).  LPR lanes per row, float4 per lane and step.
// out_bits[1] (when asked for) = max |x| over the same rows, for the range scaling of the fp16 copy.
__global__ void __launch_bounds__(256) row_norm_max_kernel(const float* __restrict__ table, int64_t v_begin, int64_t v_end, int d, int lpr,
                                                           unsigned* __restrict__ out_bits, int want_maxabs) {
  const int lane = threadIdx.x & 31;
  const int rpw = 32 / lpr, sub = lane / lpr, li = lane % lpr;
  const int64_t warp_g = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), n_warps = (int64_t)gridDim.x * (blockDim.x >> 5);
  float best = 0.f, amax = 0.f;
  for (int64_t r0 = v_begin + warp_g * rpw; r0 < v_end; r0 += n_warps * rpw) {
    const int64_t r = r0 + sub;
    float s = 0.f;
    if (r < v_end)
      for (int c = li * 4; c < d; c += lpr * 4) {
        const float4 t = ld4(table + r * d + c);
        s = fmaf(t.x, t.x, s); s = fmaf(t.y, t.y, s); s = fmaf(t.z, t.z, s); s = fmaf(t.w, t.w, s);
        amax = fmaxf(fmaxf(amax, fmaxf(fabsf(t.x), fabsf(t.y))), fmaxf(fabsf(t.z), fabsf(t.w)));
      }
    for (int o = lpr >> 1; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    best = fmaxf(best, s);
  }
  best = warp_max(best);
  if (lane == 0) atomicMax(out_bits, __float_as_uint(best));
  if (want_maxabs) {
    amax = warp_max(amax);
    if (lane == 0) atomicMax(out_bits + 1, __float_as_uint(amax));
  }
}
// fp16 copy of rows [r_begin, r_end) of src (row stride ld) times *scale -> dst rows [r_begin, r_end) (dense, d columns)
__global__ void __launch_bounds__(256) to_half_kernel(const float* __restrict__ src, int64_t ld, int64_t r_begin, int64_t r_end, int d4,
                                                      const float* __restrict__ scale, uint2* __restrict__ dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (r_end - r_begin) * d4) return;
  const int64_t r = r_begin + i / d4;
  const int c4 = (int)(i % d4);
  const float4 v = ld4(src + r * ld + c4 * 4);
  const float s = *scale;
  const __half2 a = __floats2half2_rn(v.x * s, v.y * s), b = __floats2half2_rn(v.z * s, v.w * s);
  dst[r * d4 + c4] = make_uint2(*reinterpret_cast<const uint32_t*>(&a), *reinterpret_cast<const uint32_t*>(&b));
}

bool encode_map(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool f16) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * (f16 ? 2 : 4)};
  cuuint32_t box[2] = {(cuuint32_t)(f16 ? 64 : 32), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// d <= 64: two 128-user sub-tiles per unit against 128-item tiles (every streamed tile is used by 256 users: the kernel is
// L2-bandwidth bound, and this halves the item-table traffic); larger d: one sub-tile
int pick_nst(int d) { return d <= 64 ? 2 : 1; }
int pick_bn(int d) { return d <= 128 ? 128 : 64; }

}  // namespace

// Item splits per user tile.  Every (user tile, split) unit warms its candidate lists up from scratch, and while a list
// has seen fewer than ~16 k items nearly every 32-score chunk takes the divergent insertion path -- so as FEW splits as
// still fill the machine, and never more units than one wave of SMs (measured at 16384 x 10^6, d = 64: 2 splits 5.2 ms,
// 4 splits 6.2 ms, 7 splits 8.4 ms).
int rbm_tc_topk_splits(int64_t U, int64_t n_items, int d) {
  int64_t ut = rbm_cdiv(U, BM * pick_nst(d)), tiles = rbm_cdiv(n_items, pick_bn(d));
  // Units = user tiles x splits run in waves of one CTA per SM: pick the split count with the best (wave fill) x (1 - list
  // warm-up cost), the warm-up cost of a split being ~10^5 items' worth of slow-path insertions (fitted to the measurements
  // above: 16384 users x 10^7 items -> 9 splits, 576 units = 3.9 waves; x 10^6 items -> 2 splits)
  int best = 1;
  double best_score = -1.0;
  for (int s = 1; s <= 32; ++s) {
    if (s > 1 && s > tiles / 8) break;  // at least 8 item tiles per unit
    const int64_t units = ut * s, waves = rbm_cdiv(units, RBM_NUM_SMS);
    double pen = (double)s * 1.0e5 / (double)n_items;
    if (pen > 0.9) pen = 0.9;
    const double score = (double)units / (double)(waves * RBM_NUM_SMS) * (1.0 - pen);
    if (score > best_score + 1e-9) {
      best_score = score;
      best = s;
    }
  }
  return best;
}

// item splits of the exact re-scan of uncertified users: as many as keep its partial lists under 128 MB
int rbm_tc_topk_fb_splits(int64_t U, int64_t n_items, int k) {
  int64_t s = ((int64_t)128 << 20) / (U * k * 12);
  int64_t tiles = rbm_cdiv(n_items, 64);
  if (s > tiles) s = tiles;
  if (s > 64) s = 64;
  return (int)(s < 1 ? 1 : s);
}
static size_t cand_bytes(int64_t U, int64_t n_items, int d) {
  size_t S = (size_t)rbm_tc_topk_splits(U, n_items, d);
  return S * 2 * (size_t)U * KC * (sizeof(float) + sizeof(int64_t));
}
static bool use_f16(int d) { return d % 64 == 0; }
static size_t half_bytes(int64_t U, int64_t n_items, int d) {  // fp16 copies: item rows [n_items, d], user rows [U padded to 128, d]
  if (!use_f16(d)) return 0;
  return (((size_t)n_items * d * 2 + 255) & ~(size_t)255) + (size_t)rbm_cdiv(U, 128) * 128 * d * 2 + 256;
}
// [candidate ids | candidate scores | bits + flag count + scales (48 B) | flag list U int32 (padded to 16 B) | re-scan partial lists |
//  fp16 copy of the item rows | fp16 copy of the user rows]
size_t rbm_tc_topk_ws_bytes(int64_t U, int64_t n_items, int d, int k) {
  size_t fb = (size_t)rbm_tc_topk_fb_splits(U, n_items, k) * (size_t)U * k * (sizeof(float) + sizeof(int64_t));
  return cand_bytes(U, n_items, d) + 48 + (((size_t)U * 4 + 15) & ~(size_t)15) + ((fb + 255) & ~(size_t)255) + half_bytes(U, n_items, d) + 256;
}

bool rbm_tc_topk_supported(int64_t U, int64_t n_items, int d, int k, int64_t ldf, const void* f, const void* table) {
  if (d % 32 != 0 || d < 32 || d > 256 || k > KC - 6 || U < 1) return false;  // k <= 10: six spare list slots (larger k: exact fp32 scan kernel)
  if (n_items < 8192) return false;  // small catalogues: the fp32 tile kernel is already latency-bound
  if (ldf % 4 != 0 || ((uintptr_t)f & 15) || ((uintptr_t)table & 15)) return false;
  return get_encode() != nullptr;
}

int rbm_tc_topk_launch(const float* f, int64_t ldf, const float* table, const float* bias, int64_t v_begin, int64_t v_end,
                       int64_t id_offset, const int64_t* excl, int64_t ld_excl, int n_excl, float* top_scores, int64_t* top_ids, int64_t U,
                       int d, int k, void* ws, cudaStream_t st) {
  const int BN = pick_bn(d);
  const int64_t n_items = v_end - v_begin;
  const bool f16 = use_f16(d);
  // workspace carve-up (see rbm_tc_topk_ws_bytes)
  uint8_t* aux = (uint8_t*)ws + cand_bytes(U, n_items, d);
  unsigned* bits = (unsigned*)aux;              // [0] max squared item-row norm, [1] max |item element|, [2] max |user element|
  int32_t* flag_count = (int32_t*)(aux + 12);
  float* scales = (float*)(aux + 16);           // [0] item rows, [1] user rows
  int32_t* flag_list = (int32_t*)(aux + 48);
  uint8_t* fb_ws = aux + 48 + (((size_t)U * 4 + 15) & ~(size_t)15);
  const size_t fb = (size_t)rbm_tc_topk_fb_splits(U, n_items, k) * (size_t)U * k * (sizeof(float) + sizeof(int64_t));
  uint8_t* th = fb_ws + ((fb + 255) & ~(size_t)255);                         // fp16 item rows, indexed like the table from v_begin
  uint8_t* uh = th + (((size_t)n_items * d * 2 + 255) & ~(size_t)255);       // fp16 user rows
  cudaMemsetAsync(aux, 0, 48, st);
  // stage 0: row norms (certificate) and, for the fp16 path, the range scales and the scaled fp16 copies of both operands
  const int lpr = d / 4 < 32 ? d / 4 : 32;
  row_norm_max_kernel<<<RBM_NUM_SMS * 4, 256, 0, st>>>(table, v_begin, v_end, d, lpr, bits, f16 ? 1 : 0);
  RBM_LAUNCH_CHECK("rbm_score_topk(row norms)");
  if (f16) {
    maxabs_launch(f, ldf, U, d, bits + 2, RBM_NUM_SMS, st);
    scales_launch(bits + 1, scales, st);  // scales[0] / [1]: item rows (bits[1]) / user rows (bits[2])
    to_half_kernel<<<(unsigned)rbm_cdiv(n_items * (d / 4), 256), 256, 0, st>>>(table + v_begin * d, d, 0, n_items, d / 4, scales, (uint2*)th);
    to_half_kernel<<<(unsigned)rbm_cdiv(U * (d / 4), 256), 256, 0, st>>>(f, ldf, 0, U, d / 4, scales + 1, (uint2*)uh);
    RBM_LAUNCH_CHECK("rbm_score_topk(fp16 copies)");
  }
  CUtensorMap mapA, mapB;
  const bool ok = f16 ? (encode_map(&mapA, uh, U, d, d, BM, true) && encode_map(&mapB, th, n_items, d, d, BN, true))
                      : (encode_map(&mapA, f, U, d, ldf, BM, false) && encode_map(&mapB, table, v_end, d, d, BN, false));
  if (!ok) {
    rbm_set_error("rbm_score_topk(tcgen05): cuTensorMapEncodeTiled failed");
    return -1;
  }
  TopkParams p{};
  p.bias = bias; p.scales = scales; p.U = U; p.v_begin = v_begin; p.v_end = v_end; p.id_offset = id_offset; p.d = d; p.BN = BN;
  const bool ex = excl != nullptr && n_excl > 0;
  p.S = rbm_tc_topk_splits(U, n_items, d);
  p.nst = pick_nst(d);
  p.n_utiles = (int)rbm_cdiv(U, (int64_t)BM * p.nst);
  p.tiles_per_split = rbm_cdiv(rbm_cdiv(n_items, BN), p.S);
  p.cand_i = (int64_t*)ws;
  p.cand_s = (float*)(p.cand_i + (size_t)p.S * 2 * U * KC);
  const int esz = f16 ? 2 : 4;
  const size_t a_bytes = (size_t)BM * pick_nst(d) * d * esz, stage = (size_t)BN * d * esz;
  int ns = (int)(((size_t)231424 - 1024 - a_bytes) / stage);
  if (ns > 4) ns = 4;
  if (ns < 2) {
    rbm_set_error("rbm_score_topk(tcgen05): d=%d leaves no room for a 2-stage ring", d);
    return -1;
  }
  p.nstage = ns;
  uint32_t cols = 32;
  while (cols < (uint32_t)(2 * BN * pick_nst(d))) cols <<= 1;
  p.tmem_cols = cols;
  static bool attr_set = false;
  if (!attr_set) {
    if (!set_smem(tc_topk_kernel<false, false>, 231424, "rbm_score_topk(tcgen05)") || !set_smem(tc_topk_kernel<true, false>, 231424, "rbm_score_topk(tcgen05)") ||
        !set_smem(tc_topk_kernel<false, true>, 231424, "rbm_score_topk(tcgen05)") || !set_smem(tc_topk_kernel<true, true>, 231424, "rbm_score_topk(tcgen05)"))
      return -1;
    attr_set = true;
  }
  size_t smem = a_bytes + (size_t)ns * stage + 1024;
  int units = p.n_utiles * p.S;
  int grid = units < RBM_NUM_SMS ? units : RBM_NUM_SMS;
  if (f16) {
    // the fp16 copy holds the item range from row 0: the kernel's row coordinates become relative to v_begin, ids stay absolute
    TopkParams ph = p;
    ph.bias = bias ? bias + v_begin : nullptr;
    ph.v_begin = 0;
    ph.v_end = n_items;
    ph.row_base = v_begin;
    if (ex) tc_topk_kernel<true, true><<<grid, 64 + 32 * EPI, smem, st>>>(mapA, mapB, TopkExclParams{ph, excl, ld_excl, n_excl});
    else tc_topk_kernel<true, false><<<grid, 64 + 32 * EPI, smem, st>>>(mapA, mapB, ph);
  } else {
    if (ex) tc_topk_kernel<false, true><<<grid, 64 + 32 * EPI, smem, st>>>(mapA, mapB, TopkExclParams{p, excl, ld_excl, n_excl});
    else tc_topk_kernel<false, false><<<grid, 64 + 32 * EPI, smem, st>>>(mapA, mapB, p);
  }
  RBM_LAUNCH_CHECK("rbm_score_topk(tcgen05)");
  // 2^-10 (two rounded fp16 operands) resp. 2^-9 (two truncated TF32 operands) per product, plus the fp32 accumulation slack
  float eps_mul = f16 ? 1.05e-3f : 2.1e-3f;
  // RBM_TOPK_EPS overrides the bound: test_score_topk_fused sets a huge value to send every user through the exact re-scan.  Read on
  // every call, never cached, because the test sets and unsets it inside one process.
  if (const char* e = getenv("RBM_TOPK_EPS")) eps_mul = (float)atof(e);
  topk_rescore_kernel<<<(unsigned)rbm_cdiv(U, 8), 256, 8 * d * sizeof(float), st>>>(f, ldf, table, bias, p.cand_i, p.cand_s, p.nst == 2 ? p.S : p.S * 2,
                                                                                   id_offset, top_scores, top_ids, U, d, k, bits, eps_mul,
                                                                                   f16 ? scales : nullptr, flag_list, flag_count);
  RBM_LAUNCH_CHECK("rbm_score_topk(rescore)");
  // stage 3: users whose answer the certificate does not cover are re-ranked by the exact fp32 scan (grid exits when none).
  // Stage 2 needs no exclusion filter: the lists hold non-excluded items only, and an excluded item is no candidate of the
  // certificate either (every non-excluded item a list dropped still has approximate score <= tau)
  return rbm_simt_topk_listed(f, ldf, table, bias, v_begin, v_end, id_offset, ex ? excl : nullptr, ld_excl, ex ? n_excl : 0, top_scores, top_ids,
                              U, d, k, flag_list, flag_count, fb_ws, rbm_tc_topk_fb_splits(U, n_items, k), st);
}
