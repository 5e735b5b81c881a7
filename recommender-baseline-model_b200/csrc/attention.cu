// attention.cu -- short-sequence (L <= 256) multi-head attention, forward and backward, on tensor cores.
//
// One CTA per (sequence, head).  The K/V (or Q/dO) panel of the head sits in shared memory, XOR-swizzled so that both
// mma B-fragment access patterns (contraction along the panel's columns, as in q.k^T, and along its rows, as in P.v)
// are bank-conflict free.  Each warp owns 16-row query (or key) tiles and walks the other dimension in 64-wide
// chunks, flash-attention style: scores live in mma accumulator registers, the masked softmax runs on them with
// quad shuffles, dropout is regenerated from Philox, probabilities go through a small per-warp shared tile back into
// the tensor cores.  The [B,h,L,L] probability tensor the reference materialises (NN/models/bert_modules/attention/
// single.py:14-33; torch MHA inside NN/models/sas_model/sas.py:75-76) never exists in HBM.
//
// Math: mma.sync m16n8k8 TF32 with fp32 accumulation and 3xTF32 error compensation (a = a_hi + a_lo, three MMAs per
// product), i.e. fp32-level accuracy on the legacy tensor path; -DRBM_ATTN_TF32X1 selects single-pass TF32.  The
// backward is recompute-based and atomics-free (pass A: dQ by query tiles; pass B: dK, dV by key tiles), so results
// are bit-deterministic.  A tcgen05/TMEM formulation of these L<=256 tiles is tracked in DESIGN.md ("next").
#include "common.cuh"
#include "attention_pair.cuh"
#include "attention_seq.cuh"
#include "mma_tiles.cuh"
#include "attention_tc.cuh"

namespace {

using namespace rbm_mma;
constexpr int MAX_WARPS = 8;

struct AttnArgs {
  const float *q, *k, *v, *o, *dout, *stats_in;
  float *out, *stats, *dq, *dk_, *dv, *delta;
  int64_t ldq, ldk, ldv, ldo, lddo, lddq, lddk, lddv;
  const int64_t* tok;
  int L, h, dk, mask_mode;
  float scale;
  uint32_t thr16;
  float inv_keep;
  uint64_t seed, site;
};

// ---------------------------------------------------------------------------------------------------- forward
template <int DT>
__global__ void __launch_bounds__(32 * MAX_WARPS) attn_fwd_kernel(AttnArgs a) {
  const uint64_t site_e = rbm_site(a.site);
  extern __shared__ __align__(16) float sm[];
  const int L = a.L, dk = a.dk, LP8 = (L + 7) & ~7, LPC = (L + CH - 1) / CH * CH, LD = (dk + 31) & ~31, QLD = dk + 4;
  const int b = blockIdx.x / a.h, hh = blockIdx.x % a.h;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t row0 = (int64_t)b * L;
  const int col0 = hh * dk;
  float* Kp = sm;
  float* Vp = Kp + LP8 * LD;
  float* padk = Vp + LP8 * LD;  // [LPC]
  float* chunk_pad = padk + LPC;  // [4]: chunk contains a padded key
  // L <= CH: one key chunk per query tile, the q tile is dead once the scores exist -> the probability tile reuses its
  // shared memory (per-warp footprint halves: 3 -> 4 resident CTAs at L=50, d_k=64)
  const bool single = L <= CH;
  const int QPW = single ? 16 * (QLD > PB_LD ? QLD : PB_LD) : 16 * QLD;
  float* wbase = chunk_pad + 4 + (size_t)warp * (single ? QPW : 16 * QLD + 16 * PB_LD);
  float* Qs = wbase;                          // [16][QLD] scaled q tile
  float* Pb = single ? wbase : wbase + 16 * QLD;  // [16][PB_LD]

  load_panel(Kp, a.k, a.ldk, row0, col0, L, LP8, dk, LD, 1.f);
  load_panel(Vp, a.v, a.ldv, row0, col0, L, LP8, dk, LD, 1.f);
  for (int j = threadIdx.x; j < LPC; j += blockDim.x)
    padk[j] = (a.mask_mode == RBM_MASK_KEYPAD && j < L && a.tok[row0 + j] == 0) ? 1.f : 0.f;
  __syncthreads();
  if (threadIdx.x < 4) {
    float any = 0.f;
    for (int j = threadIdx.x * CH; j < (threadIdx.x + 1) * CH && j < LPC; ++j) any += padk[j];
    chunk_pad[threadIdx.x] = any;
  }
  __syncthreads();

  for (int i0 = warp * 16; i0 < L; i0 += nwarps * 16) {
    stage_tile(Qs, QLD, a.q, a.ldq, row0, col0, i0, L, dk, a.scale * RBM_LOG2E, lane);
    __syncwarp();
    float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
    float o[DT][4];
#pragma unroll
    for (int dt = 0; dt < DT; ++dt) o[dt][0] = o[dt][1] = o[dt][2] = o[dt][3] = 0.f;
    const int kend = a.mask_mode == RBM_MASK_CAUSAL ? (i0 + 16 < L ? i0 + 16 : L) : L;
    for (int jb = 0; jb < kend; jb += CH) {
      float s[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
      tile_dot_panel(s, Qs, QLD, Kp, LD, jb, LP8, dk, g, t);
      float cm[2] = {-INFINITY, -INFINITY};
      // masking only where it can bite: padded keys (chunk flag), the causal diagonal chunk, the ragged last chunk
      const bool need_mask = chunk_pad[jb / CH] != 0.f || jb + CH > L || (a.mask_mode == RBM_MASK_CAUSAL && jb + CH > i0);
      if (need_mask) {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
          float2 pk = *reinterpret_cast<const float2*>(padk + jb + nt * 8 + 2 * t);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            int hrow = c >> 1, j = jb + nt * 8 + 2 * t + (c & 1), i = i0 + g + 8 * hrow;
            float v = s[nt][c];
            if (((c & 1) ? pk.y : pk.x) != 0.f) v = RBM_PADFILL;
            if (masked_inf(a.mask_mode, i, j, L)) v = -INFINITY;
            s[nt][c] = v;
          }
        }
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        cm[0] = fmaxf(cm[0], fmaxf(s[nt][0], s[nt][1]));
        cm[1] = fmaxf(cm[1], fmaxf(s[nt][2], s[nt][3]));
      }
      float base[2], alpha[2], ps[2] = {0.f, 0.f};
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) {
        float mn = fmaxf(m[hrow], quad_max(cm[hrow]));
        alpha[hrow] = m[hrow] == -INFINITY ? 0.f : ex2(m[hrow] - mn);
        base[hrow] = mn == -INFINITY ? 0.f : mn;
        m[hrow] = mn;
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float p = ex2(s[nt][c] - base[c >> 1]);
          s[nt][c] = p;
          ps[c >> 1] += p;
        }
#pragma unroll
      for (int hrow = 0; hrow < 2; ++hrow) l[hrow] = l[hrow] * alpha[hrow] + quad_sum(ps[hrow]);
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        o[dt][0] *= alpha[0]; o[dt][1] *= alpha[0]; o[dt][2] *= alpha[1]; o[dt][3] *= alpha[1];
      }
      if (a.thr16) {
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {
          if (jb + qd * 16 < LP8) {
            uint4 rnd = rbm_philox_drop(a.seed, site_e, rbm_attn_call((uint64_t)blockIdx.x, i0 >> 4, g, t, (jb >> 4) + qd));
#pragma unroll
            for (int bb = 0; bb < 2; ++bb)
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                int f = (c >> 1) * 4 + (c & 1) * 2 + bb;
                s[qd * 2 + bb][c] = rbm_attn_field(rnd, f) >= a.thr16 ? s[qd * 2 + bb][c] * a.inv_keep : 0.f;
              }
          }
        }
      }
      if (single) __syncwarp();  // every lane is done reading the q tile that Pb overlays
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        *reinterpret_cast<float2*>(Pb + g * PB_LD + nt * 8 + 2 * t) = make_float2(s[nt][0], s[nt][1]);
        *reinterpret_cast<float2*>(Pb + (g + 8) * PB_LD + nt * 8 + 2 * t) = make_float2(s[nt][2], s[nt][3]);
      }
      __syncwarp();
      ptile_times_panel<DT>(o, Pb, Vp, LD, jb, LP8, dk, g, t);
      __syncwarp();
    }
    float inv[2] = {1.f / l[0], 1.f / l[1]};
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      int i = i0 + g + 8 * hrow;
      if (i < L) {
        if (t == 0 && a.stats) {
          int64_t sr = ((int64_t)blockIdx.x * L + i) * 2;
          a.stats[sr] = m[hrow];
          a.stats[sr + 1] = inv[hrow];
        }
#pragma unroll
        for (int dt = 0; dt < DT; ++dt)
          if (dt * 8 < dk)
            *reinterpret_cast<float2*>(a.out + (row0 + i) * a.ldo + col0 + dt * 8 + 2 * t) =
                make_float2(o[dt][2 * hrow] * inv[hrow], o[dt][2 * hrow + 1] * inv[hrow]);
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------- backward pass A: dQ and delta
template <int DT>
__global__ void __launch_bounds__(32 * MAX_WARPS) attn_bwd_dq_kernel(AttnArgs a) {
  const uint64_t site_e = rbm_site(a.site);
  extern __shared__ __align__(16) float sm[];
  const int L = a.L, dk = a.dk, LP8 = (L + 7) & ~7, LPC = (L + CH - 1) / CH * CH, LD = (dk + 31) & ~31, QLD = dk + 4;
  const int b = blockIdx.x / a.h, hh = blockIdx.x % a.h;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t row0 = (int64_t)b * L;
  const int col0 = hh * dk;
  float* Kp = sm;
  float* Vp = Kp + LP8 * LD;
  float* padk = Vp + LP8 * LD;
  float* chunk_pad = padk + LPC;
  const bool single = L <= CH;  // one key chunk: the dS tile reuses the q tile's shared memory (see attn_fwd_kernel)
  const int QPW = single ? 16 * (QLD > PB_LD ? QLD : PB_LD) : 16 * QLD;
  float* wbase = chunk_pad + 4 + (size_t)warp * (single ? QPW + 16 * QLD : 32 * QLD + 16 * PB_LD);
  float* Qs = wbase;                            // [16][QLD] scaled q
  float* dOs = wbase + QPW;                     // [16][QLD]
  float* Pb = single ? wbase : dOs + 16 * QLD;  // [16][PB_LD] dS chunk

  load_panel(Kp, a.k, a.ldk, row0, col0, L, LP8, dk, LD, 1.f);
  load_panel(Vp, a.v, a.ldv, row0, col0, L, LP8, dk, LD, 1.f);
  for (int j = threadIdx.x; j < LPC; j += blockDim.x)
    padk[j] = (a.mask_mode == RBM_MASK_KEYPAD && j < L && a.tok[row0 + j] == 0) ? 1.f : 0.f;
  __syncthreads();
  if (threadIdx.x < 4) {
    float any = 0.f;
    for (int j = threadIdx.x * CH; j < (threadIdx.x + 1) * CH && j < LPC; ++j) any += padk[j];
    chunk_pad[threadIdx.x] = any;
  }
  __syncthreads();

  for (int i0 = warp * 16; i0 < L; i0 += nwarps * 16) {
    stage_tile(Qs, QLD, a.q, a.ldq, row0, col0, i0, L, dk, a.scale * RBM_LOG2E, lane);
    stage_tile(dOs, QLD, a.dout, a.lddo, row0, col0, i0, L, dk, 1.f, lane);
    float delta[2] = {0.f, 0.f}, mx[2] = {0.f, 0.f}, inv[2] = {0.f, 0.f};
    {
      // delta[i] = <dO[i], O[i]>: all sixteen rows' loads are issued before the first reduction (the row-by-row loop was a
      // chain of sixteen global-load latencies per tile)
      float part[16];
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        const int i = i0 + r;
        float acc = 0.f;
        if (i < L)
          for (int c = lane; c < dk; c += 32)
            acc = fmaf(__ldg(a.dout + (row0 + i) * a.lddo + col0 + c), __ldg(a.o + (row0 + i) * a.ldo + col0 + c), acc);
        part[r] = acc;
      }
#pragma unroll
      for (int r = 0; r < 16; ++r) {
        const float tot = warp_sum(part[r]);
        if (lane == 0 && i0 + r < L) a.delta[(int64_t)blockIdx.x * L + i0 + r] = tot;
        if (r == g) delta[0] = tot;
        if (r == g + 8) delta[1] = tot;
      }
    }
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      int i = i0 + g + 8 * hrow;
      if (i < L) {
        int64_t sr = ((int64_t)blockIdx.x * L + i) * 2;
        mx[hrow] = a.stats_in[sr];
        inv[hrow] = a.stats_in[sr + 1];
      }
    }
    __syncwarp();
    float dq[DT][4];
#pragma unroll
    for (int dt = 0; dt < DT; ++dt) dq[dt][0] = dq[dt][1] = dq[dt][2] = dq[dt][3] = 0.f;
    const int kend = a.mask_mode == RBM_MASK_CAUSAL ? (i0 + 16 < L ? i0 + 16 : L) : L;
    for (int jb = 0; jb < kend; jb += CH) {
      float s[8][4], dp[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
      }
      tile_dot_panel(s, Qs, QLD, Kp, LD, jb, LP8, dk, g, t);
      tile_dot_panel(dp, dOs, QLD, Vp, LD, jb, LP8, dk, g, t);
#pragma unroll
      for (int qd = 0; qd < 4; ++qd) {
        uint4 rnd = make_uint4(~0u, ~0u, ~0u, ~0u);
        if (a.thr16 && jb + qd * 16 < LP8)
          rnd = rbm_philox_drop(a.seed, site_e, rbm_attn_call((uint64_t)blockIdx.x, i0 >> 4, g, t, (jb >> 4) + qd));
#pragma unroll
        for (int bb = 0; bb < 2; ++bb) {
          const int nt = qd * 2 + bb;
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            int hrow = c >> 1, j = jb + nt * 8 + 2 * t + (c & 1), i = i0 + g + 8 * hrow;
            bool pad = padk[j] != 0.f;
            float v = pad ? RBM_PADFILL : s[nt][c];
            float p = (i >= L || masked_inf(a.mask_mode, i, j, L)) ? 0.f : ex2(v - mx[hrow]) * inv[hrow];
            float mk = 1.f;
            if (a.thr16) mk = rbm_attn_field(rnd, hrow * 4 + (c & 1) * 2 + bb) >= a.thr16 ? a.inv_keep : 0.f;
            // masked_fill(-1e9) replaces the score by a constant: no gradient reaches q.k through a padded key
            s[nt][c] = pad ? 0.f : p * (mk * dp[nt][c] - delta[hrow]);
          }
        }
      }
      if (single) __syncwarp();
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        *reinterpret_cast<float2*>(Pb + g * PB_LD + nt * 8 + 2 * t) = make_float2(s[nt][0], s[nt][1]);
        *reinterpret_cast<float2*>(Pb + (g + 8) * PB_LD + nt * 8 + 2 * t) = make_float2(s[nt][2], s[nt][3]);
      }
      __syncwarp();
      ptile_times_panel<DT>(dq, Pb, Kp, LD, jb, LP8, dk, g, t);
      __syncwarp();
    }
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      int i = i0 + g + 8 * hrow;
      if (i < L) {
#pragma unroll
        for (int dt = 0; dt < DT; ++dt)
          if (dt * 8 < dk)
            *reinterpret_cast<float2*>(a.dq + (row0 + i) * a.lddq + col0 + dt * 8 + 2 * t) =
                make_float2(dq[dt][2 * hrow] * a.scale, dq[dt][2 * hrow + 1] * a.scale);
      }
    }
    __syncwarp();
  }
}

// ------------------------------------------------------------------------------- backward pass B: dK and dV
// MAXW = 4: the variant for CTAs of at most four warps (L <= 64); three resident CTAs are asked for, which holds ptxas to
// 168 registers (it takes 244 when allowed to, without needing them: 12 bytes of spill) -> 2 -> 3 CTAs per SM
template <int DT, int MAXW = MAX_WARPS>
__global__ void __launch_bounds__(32 * MAXW, MAXW <= 4 ? 3 : 1) attn_bwd_dkv_kernel(AttnArgs a) {
  const uint64_t site_e = rbm_site(a.site);
  extern __shared__ __align__(16) float sm[];
  const int L = a.L, dk = a.dk, LP8 = (L + 7) & ~7, LPC = (L + CH - 1) / CH * CH, LD = (dk + 31) & ~31, QLD = dk + 4;
  const int b = blockIdx.x / a.h, hh = blockIdx.x % a.h;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t row0 = (int64_t)b * L;
  const int col0 = hh * dk;
  float* Qp = sm;               // [LP8][LD] scaled q panel
  float* dOp = Qp + LP8 * LD;   // [LP8][LD]
  float* st_m = dOp + LP8 * LD; // [LPC]
  float* st_i = st_m + LPC;
  float* st_d = st_i + LPC;
  const bool single = L <= CH;  // one query chunk: dS^T / P~^T reuse the key / value tiles' shared memory (see attn_fwd_kernel)
  const int QPW = single ? 16 * (QLD > PB_LD ? QLD : PB_LD) : 16 * QLD;
  float* wbase = st_d + LPC + (size_t)warp * (single ? 2 * QPW : 32 * QLD + 32 * PB_LD);
  float* Ks = wbase;                                // [16][QLD] key tile
  float* Vs = Ks + QPW;                             // [16][QLD] value tile
  float* P1 = single ? Ks : Vs + 16 * QLD;          // [16][PB_LD] dS^T chunk
  float* P2 = single ? Vs : P1 + 16 * PB_LD;        // [16][PB_LD] P~^T chunk

  load_panel(Qp, a.q, a.ldq, row0, col0, L, LP8, dk, LD, a.scale * RBM_LOG2E);
  load_panel(dOp, a.dout, a.lddo, row0, col0, L, LP8, dk, LD, 1.f);
  for (int i = threadIdx.x; i < LPC; i += blockDim.x) {
    bool in = i < L;
    int64_t sr = ((int64_t)blockIdx.x * L + i) * 2;
    st_m[i] = in ? a.stats_in[sr] : 0.f;
    st_i[i] = in ? a.stats_in[sr + 1] : 0.f;
    st_d[i] = in ? a.delta[(int64_t)blockIdx.x * L + i] : 0.f;
  }
  __syncthreads();

  for (int j0 = warp * 16; j0 < L; j0 += nwarps * 16) {
    stage_tile(Ks, QLD, a.k, a.ldk, row0, col0, j0, L, dk, 1.f, lane);
    stage_tile(Vs, QLD, a.v, a.ldv, row0, col0, j0, L, dk, 1.f, lane);
    bool jpad[2];
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      int j = j0 + g + 8 * hrow;
      jpad[hrow] = a.mask_mode == RBM_MASK_KEYPAD && j < L && a.tok[row0 + j] == 0;
    }
    __syncwarp();
    float dkacc[DT][4], dvacc[DT][4];
#pragma unroll
    for (int dt = 0; dt < DT; ++dt) {
      dkacc[dt][0] = dkacc[dt][1] = dkacc[dt][2] = dkacc[dt][3] = 0.f;
      dvacc[dt][0] = dvacc[dt][1] = dvacc[dt][2] = dvacc[dt][3] = 0.f;
    }
    const int ib0 = a.mask_mode == RBM_MASK_CAUSAL ? (j0 / CH) * CH : 0;  // queries before j0 never see these keys
    for (int ib = ib0; ib < L; ib += CH) {
      float s[8][4], dp[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
        dp[nt][0] = dp[nt][1] = dp[nt][2] = dp[nt][3] = 0.f;
      }
      tile_dot_panel(s, Ks, QLD, Qp, LD, ib, LP8, dk, g, t);    // S^T chunk: rows = keys, cols = queries
      tile_dot_panel(dp, Vs, QLD, dOp, LD, ib, LP8, dk, g, t);  // dP~^T chunk
#pragma unroll
      for (int qd = 0; qd < 4; ++qd) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          uint4 rnd = make_uint4(~0u, ~0u, ~0u, ~0u);
          if (a.thr16 && ib + qd * 16 < LP8)
            rnd = rbm_philox_drop(a.seed, site_e, rbm_attn_call((uint64_t)blockIdx.x, (ib >> 4) + qd, 2 * t + e, g >> 1, j0 >> 4));
#pragma unroll
          for (int bb = 0; bb < 2; ++bb) {
            const int nt = qd * 2 + bb;
            const int i = ib + nt * 8 + 2 * t + e;
            const float mi = st_m[i], ii = st_i[i], di = st_d[i];
#pragma unroll
            for (int hrow = 0; hrow < 2; ++hrow) {
              const int c = hrow * 2 + e, j = j0 + g + 8 * hrow;
              float v = jpad[hrow] ? RBM_PADFILL : s[nt][c];
              float p = (i >= L || j >= L || masked_inf(a.mask_mode, i, j, L)) ? 0.f : ex2(v - mi) * ii;
              float mk = 1.f;
              if (a.thr16) mk = rbm_attn_field(rnd, bb * 4 + (g & 1) * 2 + hrow) >= a.thr16 ? a.inv_keep : 0.f;
              s[nt][c] = jpad[hrow] ? 0.f : p * (mk * dp[nt][c] - di);  // dS^T (no score gradient through a padded key)
              dp[nt][c] = p * mk;                                      // P~^T
            }
          }
        }
      }
      if (single) __syncwarp();
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        *reinterpret_cast<float2*>(P1 + g * PB_LD + nt * 8 + 2 * t) = make_float2(s[nt][0], s[nt][1]);
        *reinterpret_cast<float2*>(P1 + (g + 8) * PB_LD + nt * 8 + 2 * t) = make_float2(s[nt][2], s[nt][3]);
        *reinterpret_cast<float2*>(P2 + g * PB_LD + nt * 8 + 2 * t) = make_float2(dp[nt][0], dp[nt][1]);
        *reinterpret_cast<float2*>(P2 + (g + 8) * PB_LD + nt * 8 + 2 * t) = make_float2(dp[nt][2], dp[nt][3]);
      }
      __syncwarp();
      ptile_times_panel<DT>(dkacc, P1, Qp, LD, ib, LP8, dk, g, t);   // Qp carries scale*log2(e); ln2 applied at the store
      ptile_times_panel<DT>(dvacc, P2, dOp, LD, ib, LP8, dk, g, t);
      __syncwarp();
    }
#pragma unroll
    for (int hrow = 0; hrow < 2; ++hrow) {
      int j = j0 + g + 8 * hrow;
      if (j < L) {
#pragma unroll
        for (int dt = 0; dt < DT; ++dt)
          if (dt * 8 < dk) {
            *reinterpret_cast<float2*>(a.dk_ + (row0 + j) * a.lddk + col0 + dt * 8 + 2 * t) =
                make_float2(dkacc[dt][2 * hrow] * RBM_LN2, dkacc[dt][2 * hrow + 1] * RBM_LN2);
            *reinterpret_cast<float2*>(a.dv + (row0 + j) * a.lddv + col0 + dt * 8 + 2 * t) = make_float2(dvacc[dt][2 * hrow], dvacc[dt][2 * hrow + 1]);
          }
      }
    }
    __syncwarp();
  }
}

int pick_warps(int L) {
  int ntile = (L + 15) / 16, rounds = (ntile + MAX_WARPS - 1) / MAX_WARPS;
  return (ntile + rounds - 1) / rounds;
}
size_t panel_floats(int L, int dk) { return (size_t)2 * ((L + 7) & ~7) * ((dk + 31) & ~31); }
// per-warp staging: with one chunk (L <= CH) the probability tiles overlay the q / k / v tiles (see the kernels)
size_t qpw(int L, int dk) { return L <= CH ? (size_t)16 * ((dk + 4) > PB_LD ? (dk + 4) : PB_LD) : (size_t)16 * (dk + 4); }
size_t smem_fwd(int L, int dk, int w) {
  const size_t per = L <= CH ? qpw(L, dk) : (size_t)16 * (dk + 4) + 16 * PB_LD;
  return sizeof(float) * (panel_floats(L, dk) + (L + CH - 1) / CH * CH + 4 + (size_t)w * per);
}
size_t smem_dq(int L, int dk, int w) {
  const size_t per = L <= CH ? qpw(L, dk) + (size_t)16 * (dk + 4) : (size_t)32 * (dk + 4) + 16 * PB_LD;
  return sizeof(float) * (panel_floats(L, dk) + (L + CH - 1) / CH * CH + 4 + (size_t)w * per);
}
size_t smem_dkv(int L, int dk, int w) {
  const size_t per = L <= CH ? 2 * qpw(L, dk) : (size_t)32 * (dk + 4) + 32 * PB_LD;
  return sizeof(float) * (panel_floats(L, dk) + 3 * ((L + CH - 1) / CH * CH) + (size_t)w * per);
}

template <typename Kern>
int launch(Kern kern, const AttnArgs& a, int B, int warps, size_t (*smem_fn)(int, int, int), cudaStream_t st, const char* name) {
  while (warps > 1 && smem_fn(a.L, a.dk, warps) > 227 * 1024) --warps;  // fewer warps per CTA when the tiles are wide
  size_t smem = smem_fn(a.L, a.dk, warps);
  if (smem > 227 * 1024) {
    rbm_set_error("%s: L=%d dk=%d needs %zu B of shared memory (> 227 KB): unsupported shape", name, a.L, a.dk, smem);
    return -1;
  }
  if (!set_smem(kern, smem, name)) return -1;
  kern<<<B * a.h, 32 * warps, smem, st>>>(a);
  RBM_LAUNCH_CHECK(name);
  return 0;
}

int check_common(const char* name, int B, int L, int h, int dk, int mask_mode, float p, const int64_t* tok) {
  RBM_REQUIRE(B > 0 && L > 0 && L <= 256 && h > 0, "%s: need B>0, 0<L<=256, h>0 (B=%d L=%d h=%d)", name, B, L, h);
  RBM_REQUIRE(dk >= 8 && dk % 8 == 0 && dk <= 128, "%s: unsupported head dim %d (need dk%%8==0, 8<=dk<=128)", name, dk);
  RBM_REQUIRE(mask_mode >= 0 && mask_mode <= 2, "%s: bad mask_mode %d", name, mask_mode);
  RBM_REQUIRE(mask_mode != RBM_MASK_KEYPAD || tok, "%s: key-padding mask needs tok", name);
  RBM_REQUIRE(p >= 0.f && p < 1.f, "%s: dropout p out of [0,1)", name);
  return 0;
}

}  // namespace

#define ATTN_DISPATCH(KERNEL, SMEM, NAME)                                              \
  do {                                                                                 \
    if (dk <= 32) rc = launch(KERNEL<4>, a, B, warps, SMEM, st, NAME);                 \
    else if (dk <= 64) rc = launch(KERNEL<8>, a, B, warps, SMEM, st, NAME);            \
    else rc = launch(KERNEL<16>, a, B, warps, SMEM, st, NAME);                         \
  } while (0)

extern "C" int rbm_attn_fwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                            const int64_t* tok, float* out, int64_t ldo, float* stats, int B, int L, int h, int dk,
                            int mask_mode, float scale, float p, uint64_t seed, uint64_t site, rbm_stream_t stream) {
  RBM_REQUIRE(q && k && v && out, "rbm_attn_fwd: null pointer");
  if (check_common("rbm_attn_fwd", B, L, h, dk, mask_mode, p, tok)) return -1;
  RBM_REQUIRE(ldq % 4 == 0 && ldk % 4 == 0 && ldv % 4 == 0 && ldo % 2 == 0 && rbm_aligned16(q) && rbm_aligned16(k) && rbm_aligned16(v) &&
                  ((uintptr_t)out & 7) == 0,
              "rbm_attn_fwd: q/k/v must be 16B aligned with strides %% 4 == 0 (out: 8B, stride %% 2)");
  if (rbm_attn_fwd_tc_supported(L, dk, ldq, ldk, ldv, ldo, q, k, v, out))  // Blackwell tensor path (d_k == 32)
    return rbm_attn_fwd_tc_launch(q, ldq, k, ldk, v, ldv, tok, out, ldo, stats, B, L, L, h, mask_mode, scale, p, seed, site,
                                  (cudaStream_t)stream);
  if (rbm_attn_pair_supported(L, dk, mask_mode) && stats && ldo % 2 == 0)  // d_k = 64, L <= 64: split-fp16 tcgen05 path (attention_pair.cu)
    return rbm_attn_pair_fwd(q, ldq, k, ldk, v, ldv, out, ldo, stats, B, L, h, mask_mode, scale, p, seed, site, (cudaStream_t)stream);
  if (rbm_attn_seq_supported(L, dk, mask_mode) && stats && ldo % 2 == 0)  // d_k = 64, 64 < L <= 256: split-fp16 tcgen05 path (attention_seq.cu)
    return rbm_attn_seq_fwd(q, ldq, k, ldk, v, ldv, tok, out, ldo, stats, B, L, h, mask_mode, scale, p, seed, site, (cudaStream_t)stream);
  AttnArgs a{};
  a.q = q; a.k = k; a.v = v; a.out = out; a.stats = stats; a.tok = tok;
  a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo;
  a.L = L; a.h = h; a.dk = dk; a.mask_mode = mask_mode; a.scale = scale;
  a.thr16 = rbm_drop_threshold16(p); a.inv_keep = 1.f / (1.f - p); a.seed = seed; a.site = site;
  cudaStream_t st = (cudaStream_t)stream;
  int warps = pick_warps(L), rc;
  ATTN_DISPATCH(attn_fwd_kernel, smem_fwd, "rbm_attn_fwd");
  return rc;
}

extern "C" size_t rbm_attn_bwd_ws_bytes(int B, int L, int h) { return (size_t)B * L * h * sizeof(float); }

extern "C" int rbm_attn_bwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                            const int64_t* tok, const float* out, int64_t ldo, const float* dout, int64_t lddo,
                            const float* stats, float* dq, int64_t lddq, float* dk_, int64_t lddk, float* dv,
                            int64_t lddv, int B, int L, int h, int dk, int mask_mode, float scale, float p, uint64_t seed,
                            uint64_t site, void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(q && k && v && out && dout && stats && dq && dk_ && dv && ws, "rbm_attn_bwd: null pointer");
  if (check_common("rbm_attn_bwd", B, L, h, dk, mask_mode, p, tok)) return -1;
  RBM_REQUIRE(ws_bytes >= rbm_attn_bwd_ws_bytes(B, L, h), "rbm_attn_bwd: workspace too small");
  RBM_REQUIRE(ldq % 4 == 0 && ldk % 4 == 0 && ldv % 4 == 0 && lddo % 4 == 0 && rbm_aligned16(q) && rbm_aligned16(k) &&
                  rbm_aligned16(v) && rbm_aligned16(dout),
              "rbm_attn_bwd: q/k/v/dout must be 16B aligned with strides %% 4 == 0");
  RBM_REQUIRE(lddq % 2 == 0 && lddk % 2 == 0 && lddv % 2 == 0 && (((uintptr_t)dq | (uintptr_t)dk_ | (uintptr_t)dv) & 7) == 0,
              "rbm_attn_bwd: dq/dk/dv must be 8B aligned with even strides");
  if (rbm_attn_pair_supported(L, dk, mask_mode) && ldo % 2 == 0)  // d_k = 64, L <= 64: split-fp16 tcgen05 path (attention_pair.cu)
    return rbm_attn_pair_bwd(q, ldq, k, ldk, v, ldv, out, ldo, dout, lddo, stats, dq, lddq, dk_, lddk, dv, lddv, B, L, h, mask_mode, scale, p,
                             seed, site, (cudaStream_t)stream);
  if (rbm_attn_seq_supported(L, dk, mask_mode) && ldo % 2 == 0)  // d_k = 64, 64 < L <= 256: split-fp16 tcgen05 path (attention_seq.cu)
    return rbm_attn_seq_bwd(q, ldq, k, ldk, v, ldv, tok, out, ldo, dout, lddo, stats, dq, lddq, dk_, lddk, dv, lddv, B, L, h, mask_mode, scale,
                            p, seed, site, (cudaStream_t)stream);
  AttnArgs a{};
  a.q = q; a.k = k; a.v = v; a.o = out; a.dout = dout; a.stats_in = stats; a.tok = tok;
  a.dq = dq; a.dk_ = dk_; a.dv = dv; a.delta = (float*)ws;
  a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo; a.lddo = lddo; a.lddq = lddq; a.lddk = lddk; a.lddv = lddv;
  a.L = L; a.h = h; a.dk = dk; a.mask_mode = mask_mode; a.scale = scale;
  a.thr16 = rbm_drop_threshold16(p); a.inv_keep = 1.f / (1.f - p); a.seed = seed; a.site = site;
  cudaStream_t st = (cudaStream_t)stream;
  int warps = pick_warps(L), rc;
  if (rbm_attn_bwd_dq_tc_supported(L, dk, ldq, ldk, ldv, ldo, lddo, lddq, q, k, v, out, dout, dq)) {
    rc = rbm_attn_bwd_dq_tc_launch(q, ldq, k, ldk, v, ldv, tok, out, ldo, dout, lddo, stats, dq, lddq, (float*)ws, B, L, L, h, mask_mode,
                                   scale, p, seed, site, st);
  } else {
    ATTN_DISPATCH(attn_bwd_dq_kernel, smem_dq, "rbm_attn_bwd(dq)");
  }
  if (rc) return rc;
  if (rbm_attn_bwd_dkv_tc_supported(L, dk, ldq, ldk, ldv, lddo, lddk, lddv, q, k, v, dout, dk_, dv))
    return rbm_attn_bwd_dkv_tc_launch(q, ldq, k, ldk, v, ldv, tok, dout, lddo, stats, (const float*)ws, dk_, lddk, dv, lddv, B, L, L, h,
                                      mask_mode, scale, p, seed, site, st);
  if (warps <= 4 && dk <= 64) {  // (the d_k = 128 accumulators do not fit 168 registers: 2 KB of spills)
    if (dk <= 32) rc = launch(attn_bwd_dkv_kernel<4, 4>, a, B, warps, smem_dkv, st, "rbm_attn_bwd(dkv)");
    else rc = launch(attn_bwd_dkv_kernel<8, 4>, a, B, warps, smem_dkv, st, "rbm_attn_bwd(dkv)");
  } else {
    ATTN_DISPATCH(attn_bwd_dkv_kernel, smem_dkv, "rbm_attn_bwd(dkv)");
  }
  return rc;
}

// ---- queries are a per-sequence compacted subset (Lq rows per sequence, zero rows after the real ones), keys / values all L positions.
// Tensor path only (d_k = 32, L <= 256), no causal mask (a compacted query has lost its position); dropout fields are indexed by
// (sequence-head, compact query ordinal, key position).
extern "C" int rbm_attn_lq_supported(int L, int Lq, int dk, int mask_mode) {
  return dk == 32 && L >= 1 && L <= 256 && Lq >= 1 && Lq <= L && mask_mode != RBM_MASK_CAUSAL ? 1 : 0;
}

extern "C" int rbm_attn_fwd_lq(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                               const int64_t* tok, float* out, int64_t ldo, float* stats, int B, int L, int Lq, int h, int dk,
                               int mask_mode, float scale, float p, uint64_t seed, uint64_t site, rbm_stream_t stream) {
  RBM_REQUIRE(q && k && v && out && stats, "rbm_attn_fwd_lq: null pointer");
  if (check_common("rbm_attn_fwd_lq", B, L, h, dk, mask_mode, p, tok)) return -1;
  RBM_REQUIRE(rbm_attn_lq_supported(L, Lq, dk, mask_mode), "rbm_attn_fwd_lq: need d_k = 32, Lq <= L <= 256, no causal mask (L=%d Lq=%d d_k=%d)", L,
              Lq, dk);
  RBM_REQUIRE(rbm_attn_fwd_tc_supported(L, dk, ldq, ldk, ldv, ldo, q, k, v, out), "rbm_attn_fwd_lq: operands not laid out for the tensor path");
  return rbm_attn_fwd_tc_launch(q, ldq, k, ldk, v, ldv, tok, out, ldo, stats, B, L, Lq, h, mask_mode, scale, p, seed, site, (cudaStream_t)stream);
}

extern "C" size_t rbm_attn_bwd_lq_ws_bytes(int B, int Lq, int h) { return (size_t)B * Lq * h * sizeof(float); }

extern "C" int rbm_attn_bwd_lq(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                               const int64_t* tok, const float* out, int64_t ldo, const float* dout, int64_t lddo,
                               const float* stats, float* dq, int64_t lddq, float* dk_, int64_t lddk, float* dv, int64_t lddv, int B,
                               int L, int Lq, int h, int dk, int mask_mode, float scale, float p, uint64_t seed, uint64_t site, void* ws,
                               size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(q && k && v && out && dout && stats && dq && dk_ && dv && ws, "rbm_attn_bwd_lq: null pointer");
  if (check_common("rbm_attn_bwd_lq", B, L, h, dk, mask_mode, p, tok)) return -1;
  RBM_REQUIRE(rbm_attn_lq_supported(L, Lq, dk, mask_mode), "rbm_attn_bwd_lq: need d_k = 32, Lq <= L <= 256, no causal mask (L=%d Lq=%d d_k=%d)", L,
              Lq, dk);
  RBM_REQUIRE(ws_bytes >= rbm_attn_bwd_lq_ws_bytes(B, Lq, h), "rbm_attn_bwd_lq: workspace too small");
  RBM_REQUIRE(rbm_attn_bwd_dq_tc_supported(L, dk, ldq, ldk, ldv, ldo, lddo, lddq, q, k, v, out, dout, dq) &&
                  rbm_attn_bwd_dkv_tc_supported(L, dk, ldq, ldk, ldv, lddo, lddk, lddv, q, k, v, dout, dk_, dv),
              "rbm_attn_bwd_lq: operands not laid out for the tensor path");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = rbm_attn_bwd_dq_tc_launch(q, ldq, k, ldk, v, ldv, tok, out, ldo, dout, lddo, stats, dq, lddq, (float*)ws, B, L, Lq, h, mask_mode, scale,
                                     p, seed, site, st);
  if (rc) return rc;
  return rbm_attn_bwd_dkv_tc_launch(q, ldq, k, ldk, v, ldv, tok, dout, lddo, stats, (const float*)ws, dk_, lddk, dv, lddv, B, L, Lq, h,
                                    mask_mode, scale, p, seed, site, st);
}

RBM_DEFINE_STEP_PTR_SETTER(rbm_step_ptr_set_attention)
