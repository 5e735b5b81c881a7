// score_ce.cu -- BERT4Rec output scoring fused with masked cross-entropy; logits are never written to HBM.
// Replaces  logits = self.out(h)  (NN/models/bert.py:16, materialises [B,L,V+1]) followed by
// CrossEntropyLoss(ignore_index=0) (NN/trainers/bert.py:11,36-40) and their autograd.
//   fwd : rows with labels != 0 are compacted; each warp owns 16 of them, the [V+1, d] weight streams through shared
//         memory in 64-row swizzled panels (cp.async double buffer); 16x64 logit tiles are produced on tensor cores
//         (mma.sync TF32, 3xTF32 compensated), an online (max, sum-exp) in the log2 domain and the target logit are
//         kept in registers.
//   bwd : logits are recomputed tile-wise;  dH = G.W  (warp per 16 rows, the same panel serves both MMAs),
//         dW = G^T.H, db = colsum(G)  (warp per 16 vocab rows, gathered H panels stream, row chunks split over
//         blockIdx.y with a fixed-order reduction), G = (softmax - onehot) * dloss / count.
#include "common.cuh"
#include "mma_tiles.cuh"
#include "ce_tc.cuh"
#include "ce_wide.cuh"

namespace {

using namespace rbm_mma;

// ---------------------------------------------------------------------------------------------- compaction
__global__ void __launch_bounds__(256) compact_count_kernel(const int64_t* __restrict__ labels, int64_t n, int32_t* __restrict__ blk_cnt) {
  __shared__ int wc[8];
  int64_t base = (int64_t)blockIdx.x * 1024;
  int c = 0;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    int64_t i = base + t * 256 + threadIdx.x;
    c += (i < n && labels[i] != 0) ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < 8; ++w) s += wc[w];
    blk_cnt[blockIdx.x] = s;
  }
}

__global__ void compact_scan_kernel(int32_t* blk_cnt, int nblk, int32_t* count_out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int run = 0;
    for (int b = 0; b < nblk; ++b) {
      int c = blk_cnt[b];
      blk_cnt[b] = run;
      run += c;
    }
    *count_out = run;
  }
}

__global__ void __launch_bounds__(256) compact_write_kernel(const int64_t* __restrict__ labels, int64_t n, const int32_t* __restrict__ blk_off,
                                                            int32_t* __restrict__ rows_out, int64_t* __restrict__ tgt_out) {
  __shared__ int wc[8];
  int64_t base = (int64_t)blockIdx.x * 1024;
  int run = blk_off[blockIdx.x];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int t = 0; t < 4; ++t) {
    int64_t i = base + t * 256 + threadIdx.x;
    int64_t lab = i < n ? labels[i] : 0;
    bool f = lab != 0;
    unsigned bal = __ballot_sync(0xffffffffu, f);
    if (lane == 0) wc[warp] = __popc(bal);
    __syncthreads();
    int woff = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      int c = wc[w];
      if (w < warp) woff += c;
      tot += c;
    }
    if (f) {
      int pos = run + woff + __popc(bal & ((1u << lane) - 1u));
      rows_out[pos] = (int32_t)i;
      tgt_out[pos] = lab;
    }
    run += tot;
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------ async panel loads
__device__ __forceinline__ void cp_async16(float* dst, const float* src, bool valid) {
  uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
  int sz = valid ? 16 : 0;  // src-size 0: zero-fill
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// panel[64][LD] (swizzled) <- rows r0.. of src; row index through `rows` when given; rows >= limit zero-filled
__device__ __forceinline__ void panel_load_async(float* panel, const float* __restrict__ src, const int32_t* __restrict__ rows,
                                                 int64_t r0, int64_t limit, int d, int LD) {
  int d4 = d >> 2;
  for (int idx = threadIdx.x; idx < CH * d4; idx += blockDim.x) {
    int r = idx / d4, c4 = idx - r * d4;
    bool ok = r0 + r < limit;
    int64_t gr = ok ? (rows ? (int64_t)rows[r0 + r] : (r0 + r)) : 0;
    cp_async16(panel + r * LD + ((c4 * 4) ^ swz(r)), src + gr * d + c4 * 4, ok);
  }
}
// per-warp tile[16][ldt] <- rows (r0 + r) of src (through `rows` when given) times mul; rows >= limit zero
__device__ __forceinline__ void stage_rows(float* dst, int ldt, const float* __restrict__ src, const int32_t* __restrict__ rows,
                                           int64_t r0, int64_t limit, int d, float mul, int lane) {
  int d4 = d >> 2;
  for (int idx = lane; idx < 16 * d4; idx += 32) {
    int r = idx / d4, c4 = idx - r * d4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r0 + r < limit) {
      int64_t gr = rows ? (int64_t)rows[r0 + r] : (r0 + r);
      v = ld4(src + gr * d + c4 * 4);
    }
    st4(dst + r * ldt + c4 * 4, make_float4(v.x * mul, v.y * mul, v.z * mul, v.w * mul));
  }
}

struct CeArgs {
  const float* h;
  const int32_t* rows;
  const int64_t* tgt;
  const int32_t* count;
  const float* w;
  const float* bias;
  const float* lse_in;
  const float* dloss;
  float *lse_out, *partial, *dh_full, *part_w, *part_b;
  int V1, d;
};

// ------------------------------------------------------------------------------------------------ forward
__global__ void __launch_bounds__(256) ce_fwd_kernel(CeArgs a) {
  extern __shared__ __align__(16) float sm[];
  const int d = a.d, V1 = a.V1, LD = (d + 31) & ~31, QLD = d + 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int count = *a.count;
  const int r0cta = blockIdx.x * nwarps * 16;
  if (r0cta >= count) {
    if (threadIdx.x == 0) a.partial[blockIdx.x] = 0.f;
    return;
  }
  float* panel = sm;                      // [2][64][LD]
  float* bias_s = panel + 2 * CH * LD;    // [2][64]
  float* contrib = bias_s + 2 * CH;       // [nwarps*16]
  float* Hs = contrib + nwarps * 16 + (size_t)warp * 16 * QLD;
  const int r0 = r0cta + warp * 16;
  stage_rows(Hs, QLD, a.h, a.rows, r0, count, d, RBM_LOG2E, lane);
  int64_t tg[2];
  float m[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f}, tl[2] = {0.f, 0.f};
#pragma unroll
  for (int hr = 0; hr < 2; ++hr) {
    int r = r0 + g + 8 * hr;
    tg[hr] = (r < count && a.tgt[r] >= 0 && a.tgt[r] < a.V1) ? a.tgt[r] : -1;  // outside the (shard of the) vocabulary: no column
  }
  const int NC = (V1 + CH - 1) / CH;
  auto issue = [&](int c) {
    panel_load_async(panel + (c & 1) * CH * LD, a.w, nullptr, (int64_t)c * CH, V1, d, LD);
    for (int j = threadIdx.x; j < CH; j += blockDim.x) {
      int v = c * CH + j;
      bias_s[(c & 1) * CH + j] = (a.bias && v < V1) ? a.bias[v] * RBM_LOG2E : 0.f;
    }
    cp_async_commit();
  };
  issue(0);
  for (int c = 0; c < NC; ++c) {
    if (c + 1 < NC) {
      issue(c + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* pn = panel + (c & 1) * CH * LD;
    const float* bs = bias_s + (c & 1) * CH;
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    tile_dot_panel(s, Hs, QLD, pn, LD, 0, CH, d, g, t);
    float cm[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      float2 b2 = *reinterpret_cast<const float2*>(bs + nt * 8 + 2 * t);
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        int v = c * CH + nt * 8 + 2 * t + (cc & 1);
        float x = v < V1 ? s[nt][cc] + ((cc & 1) ? b2.y : b2.x) : -INFINITY;
        if ((int64_t)v == tg[cc >> 1]) tl[cc >> 1] += x;
        s[nt][cc] = x;
        cm[cc >> 1] = fmaxf(cm[cc >> 1], x);
      }
    }
    float base[2], ps[2] = {0.f, 0.f};
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) {
      float mn = fmaxf(m[hr], quad_max(cm[hr]));
      l[hr] *= (m[hr] == -INFINITY ? 0.f : ex2(m[hr] - mn));
      base[hr] = mn;
      m[hr] = mn;
    }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) ps[cc >> 1] += ex2(s[nt][cc] - base[cc >> 1]);
#pragma unroll
    for (int hr = 0; hr < 2; ++hr) l[hr] += quad_sum(ps[hr]);
    __syncthreads();
  }
#pragma unroll
  for (int hr = 0; hr < 2; ++hr) {
    int r = r0 + g + 8 * hr;
    float tsum = quad_sum(tl[hr]);
    float lse = (m[hr] + log2f(l[hr])) * RBM_LN2;
    if (t == 0) {
      if (r < count) a.lse_out[r] = lse;
      contrib[warp * 16 + g + 8 * hr] = r < count ? lse - tsum * RBM_LN2 : 0.f;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float sacc = 0.f;
    for (int r = 0; r < nwarps * 16; ++r) sacc += contrib[r];
    a.partial[blockIdx.x] = sacc;
  }
}

__global__ void __launch_bounds__(256) ce_loss_finalize_kernel(const float* __restrict__ partial, int nblk,
                                                               const int32_t* __restrict__ count_p, float* __restrict__ loss) {
  __shared__ float red[256];
  float s = 0.f;
  for (int b = threadIdx.x; b < nblk; b += 256) s += partial[b];
  red[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 256; ++i) t += red[i];
    *loss = t / (float)(*count_p);
  }
}

// ---------------------------------------------------------------------------------------- backward: dH
template <int DT>
__global__ void __launch_bounds__(256) ce_bwd_dh_kernel(CeArgs a) {
  extern __shared__ __align__(16) float sm[];
  const int d = a.d, V1 = a.V1, LD = (d + 31) & ~31, QLD = d + 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int count = *a.count;
  const int r0cta = blockIdx.x * nwarps * 16;
  if (r0cta >= count) return;
  float* panel = sm;
  float* bias_s = panel + 2 * CH * LD;
  float* wbase = bias_s + 2 * CH + (size_t)warp * (16 * QLD + 16 * PB_LD);
  float* Hs = wbase;
  float* Pb = wbase + 16 * QLD;
  const int r0 = r0cta + warp * 16;
  const float gscale = *a.dloss / (float)count;
  stage_rows(Hs, QLD, a.h, a.rows, r0, count, d, RBM_LOG2E, lane);
  int64_t tg[2];
  float lse2[2];
  bool live[2];
#pragma unroll
  for (int hr = 0; hr < 2; ++hr) {
    int r = r0 + g + 8 * hr;
    live[hr] = r < count;
    tg[hr] = (r < count && a.tgt[r] >= 0 && a.tgt[r] < a.V1) ? a.tgt[r] : -1;  // outside the (shard of the) vocabulary: no column
    lse2[hr] = r < count ? a.lse_in[r] * RBM_LOG2E : 0.f;
  }
  float acc[DT][4];
#pragma unroll
  for (int dt = 0; dt < DT; ++dt) acc[dt][0] = acc[dt][1] = acc[dt][2] = acc[dt][3] = 0.f;
  const int NC = (V1 + CH - 1) / CH;
  auto issue = [&](int c) {
    panel_load_async(panel + (c & 1) * CH * LD, a.w, nullptr, (int64_t)c * CH, V1, d, LD);
    for (int j = threadIdx.x; j < CH; j += blockDim.x) {
      int v = c * CH + j;
      bias_s[(c & 1) * CH + j] = (a.bias && v < V1) ? a.bias[v] * RBM_LOG2E : 0.f;
    }
    cp_async_commit();
  };
  issue(0);
  for (int c = 0; c < NC; ++c) {
    if (c + 1 < NC) {
      issue(c + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* pn = panel + (c & 1) * CH * LD;
    const float* bs = bias_s + (c & 1) * CH;
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    tile_dot_panel(s, Hs, QLD, pn, LD, 0, CH, d, g, t);
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      float2 b2 = *reinterpret_cast<const float2*>(bs + nt * 8 + 2 * t);
      float gg[4];
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        int v = c * CH + nt * 8 + 2 * t + (cc & 1), hr = cc >> 1;
        // a live row whose target lies in another vocabulary shard (tg = -1) still has its softmax here: test_ce_vocab_shards
        // (simt_d48_S3) caught this guard once testing tg >= 0 instead of the row being live
        float p = (v < V1 && live[hr]) ? ex2(s[nt][cc] + ((cc & 1) ? b2.y : b2.x) - lse2[hr]) : 0.f;
        if ((int64_t)v == tg[hr]) p -= 1.f;
        gg[cc] = p * gscale;
      }
      *reinterpret_cast<float2*>(Pb + g * PB_LD + nt * 8 + 2 * t) = make_float2(gg[0], gg[1]);
      *reinterpret_cast<float2*>(Pb + (g + 8) * PB_LD + nt * 8 + 2 * t) = make_float2(gg[2], gg[3]);
    }
    __syncwarp();
    ptile_times_panel<DT>(acc, Pb, pn, LD, 0, CH, d, g, t);  // dH += G . W[chunk]
    __syncthreads();
  }
#pragma unroll
  for (int hr = 0; hr < 2; ++hr) {
    int r = r0 + g + 8 * hr;
    if (r < count) {
      float* dst = a.dh_full + (int64_t)a.rows[r] * d;
#pragma unroll
      for (int dt = 0; dt < DT; ++dt)
        if (dt * 8 < d) *reinterpret_cast<float2*>(dst + dt * 8 + 2 * t) = make_float2(acc[dt][2 * hr], acc[dt][2 * hr + 1]);
    }
  }
}

// ------------------------------------------------------------------------------------ backward: dW and db
// grid (vocab tiles of 16*nwarps rows, S): row chunks {s, s+S, ...} of 64 compacted rows each
template <int DT>
__global__ void __launch_bounds__(256) ce_bwd_dw_kernel(CeArgs a) {
  extern __shared__ __align__(16) float sm[];
  const int d = a.d, V1 = a.V1, LD = (d + 31) & ~31, QLD = d + 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int count = *a.count;
  const int S = gridDim.y, sp = blockIdx.y;
  float* panel = sm;                       // [2][64][LD] gathered H rows
  float* lse_s = panel + 2 * CH * LD;      // [2][64] lse (log2 domain)
  float* tgt_s = lse_s + 2 * CH;           // [2][64] target id as float (exact below 2^24) or -1
  float* wbase = tgt_s + 2 * CH + (size_t)warp * (16 * QLD + 16 * PB_LD);
  float* Ws = wbase;
  float* Pb = wbase + 16 * QLD;
  const int v0 = (blockIdx.x * nwarps + warp) * 16;
  const float gscale = *a.dloss / (float)count;
  stage_rows(Ws, QLD, a.w, nullptr, v0, V1, d, RBM_LOG2E, lane);
  float b2[2];
  int vrow[2];
#pragma unroll
  for (int hr = 0; hr < 2; ++hr) {
    vrow[hr] = v0 + g + 8 * hr;
    b2[hr] = (a.bias && vrow[hr] < V1) ? a.bias[vrow[hr]] * RBM_LOG2E : 0.f;
  }
  float acc[DT][4], bsum[2] = {0.f, 0.f};
#pragma unroll
  for (int dt = 0; dt < DT; ++dt) acc[dt][0] = acc[dt][1] = acc[dt][2] = acc[dt][3] = 0.f;
  const int NC = (count + CH - 1) / CH;
  auto issue = [&](int c, int buf) {
    panel_load_async(panel + buf * CH * LD, a.h, a.rows, (int64_t)c * CH, count, d, LD);
    for (int j = threadIdx.x; j < CH; j += blockDim.x) {
      int r = c * CH + j;
      lse_s[buf * CH + j] = r < count ? a.lse_in[r] * RBM_LOG2E : INFINITY;  // columns beyond the count: p = 0
      tgt_s[buf * CH + j] = (r < count && a.tgt[r] >= 0 && a.tgt[r] < a.V1) ? (float)a.tgt[r] : -1.f;
    }
    cp_async_commit();
  };
  int it = 0;
  if (sp < NC) issue(sp, 0);
  for (int c = sp; c < NC; c += S, ++it) {
    const int buf = it & 1;
    if (c + S < NC) {
      issue(c + S, buf ^ 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* pn = panel + buf * CH * LD;
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
    tile_dot_panel(s, Ws, QLD, pn, LD, 0, CH, d, g, t);  // S^T: rows = vocab, cols = compacted rows
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      float2 ls = *reinterpret_cast<const float2*>(lse_s + buf * CH + nt * 8 + 2 * t);
      float2 ts = *reinterpret_cast<const float2*>(tgt_s + buf * CH + nt * 8 + 2 * t);
      float gg[4];
#pragma unroll
      for (int cc = 0; cc < 4; ++cc) {
        int hr = cc >> 1;
        float tcol = (cc & 1) ? ts.y : ts.x, lcol = (cc & 1) ? ls.y : ls.x;
        // the column of a live row whose target lies in another vocabulary shard (tcol = -1) is not zero: test_ce_vocab_shards
        // (simt_d48_S3) caught this guard once testing tcol >= 0 instead of the row being live
        float p = (vrow[hr] < V1 && lcol != INFINITY) ? ex2(s[nt][cc] + b2[hr] - lcol) : 0.f;
        if (tcol == (float)vrow[hr]) p -= 1.f;
        gg[cc] = p * gscale;
        bsum[hr] += gg[cc];
      }
      *reinterpret_cast<float2*>(Pb + g * PB_LD + nt * 8 + 2 * t) = make_float2(gg[0], gg[1]);
      *reinterpret_cast<float2*>(Pb + (g + 8) * PB_LD + nt * 8 + 2 * t) = make_float2(gg[2], gg[3]);
    }
    __syncwarp();
    ptile_times_panel<DT>(acc, Pb, pn, LD, 0, CH, d, g, t);  // dW += G^T . H[chunk]
    __syncthreads();
  }
#pragma unroll
  for (int hr = 0; hr < 2; ++hr) {
    float bs = quad_sum(bsum[hr]);
    if (vrow[hr] < V1) {
      float* dst = a.part_w + ((int64_t)sp * V1 + vrow[hr]) * d;
#pragma unroll
      for (int dt = 0; dt < DT; ++dt)
        if (dt * 8 < d) *reinterpret_cast<float2*>(dst + dt * 8 + 2 * t) = make_float2(acc[dt][2 * hr], acc[dt][2 * hr + 1]);
      if (t == 0) a.part_b[(int64_t)sp * V1 + vrow[hr]] = bs;
    }
  }
}

__global__ void ce_reduce_splits_kernel(const float* __restrict__ part, float* __restrict__ out, int64_t n, int S) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int k = 0; k < S; ++k) s += part[(int64_t)k * n + i];
  out[i] = s;
}

// warps per CTA so that the tiles fit in shared memory (fewer warps for wide hidden sizes)
size_t ce_smem(int d, int warps, bool with_pb) {
  int LD = (d + 31) & ~31;
  return sizeof(float) * ((size_t)2 * CH * LD + 4 * CH + warps * 16 + (size_t)warps * (16 * (d + 4) + (with_pb ? 16 * PB_LD : 0)));
}
int ce_warps(int d, bool with_pb) {
  int w = 8;
  while (w > 1 && ce_smem(d, w, with_pb) > 100 * 1024) w >>= 1;  // <= 100 KB: two CTAs per SM
  while (w > 1 && ce_smem(d, w, with_pb) > 227 * 1024) w >>= 1;
  return w;
}
int dw_splits(int64_t cap, int V1, int warps) {
  int64_t vt = rbm_cdiv(V1, 16 * warps), chunks = rbm_cdiv(cap, CH);
  int64_t s = rbm_cdiv((int64_t)RBM_NUM_SMS * 4, vt);
  if (s > chunks) s = chunks;
  if (s > 64) s = 64;
  return (int)(s < 1 ? 1 : s);
}

}  // namespace

extern "C" size_t rbm_compact_ws_bytes(int64_t n) { return (size_t)rbm_cdiv(n, 1024) * sizeof(int32_t) + 16; }

extern "C" int rbm_compact_labels(const int64_t* labels, int64_t n, int32_t* rows_out, int64_t* tgt_out, int32_t* count_out,
                                  void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(labels && rows_out && tgt_out && count_out && ws, "rbm_compact_labels: null pointer");
  RBM_REQUIRE(n > 0 && n < (int64_t)1 << 31, "rbm_compact_labels: n=%lld out of range", (long long)n);
  RBM_REQUIRE(ws_bytes >= rbm_compact_ws_bytes(n), "rbm_compact_labels: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  int nblk = (int)rbm_cdiv(n, 1024);
  int32_t* blk = (int32_t*)ws;
  compact_count_kernel<<<nblk, 256, 0, st>>>(labels, n, blk);
  compact_scan_kernel<<<1, 32, 0, st>>>(blk, nblk, count_out);
  compact_write_kernel<<<nblk, 256, 0, st>>>(labels, n, blk, rows_out, tgt_out);
  RBM_LAUNCH_CHECK("rbm_compact_labels");
  return 0;
}

// workspace layout (floats): [partial: cdiv(cap,16)] [part_w: Smax*V1*d] [part_b: Smax*V1] [tcgen05 extras]
static size_t ce_smax(int64_t cap, int V1) {
  size_t S = (size_t)dw_splits(cap, V1, 1);
  if (S < (size_t)dw_splits(cap, V1, 8)) S = (size_t)dw_splits(cap, V1, 8);
  if (S < (size_t)rbm_ce_tc_dw_splits(cap, V1)) S = (size_t)rbm_ce_tc_dw_splits(cap, V1);
  if (S < (size_t)rbm_ce_wide_dw_splits(cap, V1)) S = (size_t)rbm_ce_wide_dw_splits(cap, V1);
  return S;
}
static size_t ce_off_partw(int64_t cap) { return ((size_t)rbm_cdiv(cap, 16) + 3) & ~(size_t)3; }
static size_t ce_off_extra(int64_t cap, int V1, int d) { return (ce_off_partw(cap) + ce_smax(cap, V1) * ((size_t)V1 * d + V1) + 3) & ~(size_t)3; }

extern "C" size_t rbm_ce_ws_bytes(int64_t cap, int V1, int d) {
  size_t extra = rbm_ce_tc_ws_floats(cap, V1, d), wide = rbm_ce_wide_ws_floats(cap, V1, d);
  return (ce_off_extra(cap, V1, d) + (extra > wide ? extra : wide)) * sizeof(float) + 64;
}

static int ce_check(const char* name, int64_t cap, int V1, int d) {
  RBM_REQUIRE(cap > 0 && cap < (int64_t)1 << 31 && V1 > 0 && V1 < (1 << 24), "%s: bad sizes cap=%lld V1=%d (V1 < 2^24)", name, (long long)cap, V1);
  RBM_REQUIRE(d >= 8 && d % 8 == 0 && d <= 256, "%s: unsupported hidden size d=%d (need d%%8==0, d<=256)", name, d);
  return 0;
}

extern "C" int rbm_ce_fwd(const float* h, const int32_t* rows, const int64_t* tgt, const int32_t* count, const float* w,
                          const float* bias, float* lse, float* loss, int64_t cap, int V1, int d, void* ws, size_t ws_bytes,
                          rbm_stream_t stream) {
  RBM_REQUIRE(h && rows && tgt && count && w && lse && loss && ws, "rbm_ce_fwd: null pointer");
  if (ce_check("rbm_ce_fwd", cap, V1, d)) return -1;
  RBM_REQUIRE(ws_bytes >= rbm_ce_ws_bytes(cap, V1, d), "rbm_ce_fwd: workspace too small");
  RBM_REQUIRE(rbm_aligned16(h) && rbm_aligned16(w) && rbm_aligned16(ws), "rbm_ce_fwd: pointers must be 16B aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (rbm_ce_tc_supported(V1, d, h, w)) {  // Blackwell tensor path
    int nblk_tc = 0;
    int rc = rbm_ce_tc_fwd(h, rows, tgt, count, w, bias, lse, (float*)ws, cap, V1, d, (float*)ws + ce_off_extra(cap, V1, d), &nblk_tc, st);
    if (rc) return rc;
    ce_loss_finalize_kernel<<<1, 256, 0, st>>>((const float*)ws, nblk_tc, count, loss);
    RBM_LAUNCH_CHECK("rbm_ce_fwd(finalize)");
    return 0;
  }
  if (rbm_ce_wide_supported(V1, d, h, w)) {  // d = 128 / 256: split-fp16 tensor path (ce_wide.cu)
    int nblk_w = 0;
    int rc = rbm_ce_wide_fwd(h, rows, tgt, count, w, bias, lse, (float*)ws, cap, V1, d, (float*)ws + ce_off_extra(cap, V1, d), &nblk_w, st);
    if (rc) return rc;
    ce_loss_finalize_kernel<<<1, 256, 0, st>>>((const float*)ws, nblk_w, count, loss);
    RBM_LAUNCH_CHECK("rbm_ce_fwd(finalize)");
    return 0;
  }
  int warps = ce_warps(d, false);
  int nblk = (int)rbm_cdiv(cap, 16 * warps);
  size_t smem = ce_smem(d, warps, false);
  if (!set_smem(ce_fwd_kernel, smem, "rbm_ce_fwd")) return -1;
  CeArgs a{};
  a.h = h; a.rows = rows; a.tgt = tgt; a.count = count; a.w = w; a.bias = bias; a.lse_out = lse; a.partial = (float*)ws; a.V1 = V1; a.d = d;
  ce_fwd_kernel<<<nblk, 32 * warps, smem, st>>>(a);
  RBM_LAUNCH_CHECK("rbm_ce_fwd");
  ce_loss_finalize_kernel<<<1, 256, 0, st>>>((const float*)ws, nblk, count, loss);
  RBM_LAUNCH_CHECK("rbm_ce_fwd(finalize)");
  return 0;
}

extern "C" int rbm_ce_bwd(const float* h, const int32_t* rows, const int64_t* tgt, const int32_t* count, const float* w,
                          const float* bias, const float* lse, const float* dloss, float* dh_full, float* dw, float* db,
                          int64_t cap, int V1, int d, void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(h && rows && tgt && count && w && lse && dloss && dh_full && dw && db && ws, "rbm_ce_bwd: null pointer");
  if (ce_check("rbm_ce_bwd", cap, V1, d)) return -1;
  RBM_REQUIRE(ws_bytes >= rbm_ce_ws_bytes(cap, V1, d), "rbm_ce_bwd: workspace too small");
  RBM_REQUIRE(rbm_aligned16(h) && rbm_aligned16(w) && rbm_aligned16(ws) && rbm_aligned16(dh_full) && rbm_aligned16(dw),
              "rbm_ce_bwd: pointers must be 16B aligned");
  cudaStream_t st = (cudaStream_t)stream;
  float* part_w = (float*)ws + ce_off_partw(cap);
  if (rbm_ce_tc_supported(V1, d, h, w)) {  // Blackwell tensor path
    const int S = rbm_ce_tc_dw_splits(cap, V1);
    float* part_b = part_w + (size_t)S * V1 * d;
    int rc = rbm_ce_tc_bwd(h, rows, tgt, count, w, bias, lse, dloss, dh_full, part_w, part_b, S, cap, V1, d,
                           (float*)ws + ce_off_extra(cap, V1, d), st);
    if (rc) return rc;
    int64_t n = (int64_t)V1 * d;
    ce_reduce_splits_kernel<<<(unsigned)rbm_cdiv(n, 256), 256, 0, st>>>(part_w, dw, n, S);
    ce_reduce_splits_kernel<<<(unsigned)rbm_cdiv(V1, 256), 256, 0, st>>>(part_b, db, V1, S);
    RBM_LAUNCH_CHECK("rbm_ce_bwd(reduce)");
    return 0;
  }
  if (rbm_ce_wide_supported(V1, d, h, w)) {  // d = 128 / 256: split-fp16 tensor path (ce_wide.cu)
    const int S = rbm_ce_wide_dw_splits(cap, V1);
    float* part_b = part_w + (size_t)S * V1 * d;
    int rc = rbm_ce_wide_bwd(h, rows, tgt, count, w, bias, lse, dloss, dh_full, part_w, part_b, S, cap, V1, d,
                             (float*)ws + ce_off_extra(cap, V1, d), st);
    if (rc) return rc;
    int64_t n = (int64_t)V1 * d;
    ce_reduce_splits_kernel<<<(unsigned)rbm_cdiv(n, 256), 256, 0, st>>>(part_w, dw, n, S);
    ce_reduce_splits_kernel<<<(unsigned)rbm_cdiv(V1, 256), 256, 0, st>>>(part_b, db, V1, S);
    RBM_LAUNCH_CHECK("rbm_ce_bwd(reduce)");
    return 0;
  }
  int warps = ce_warps(d, true);
  int nblk = (int)rbm_cdiv(cap, 16 * warps);
  int S = dw_splits(cap, V1, warps);
  size_t smem = ce_smem(d, warps, true);
  float* part_b = part_w + (size_t)S * V1 * d;
  CeArgs a{};
  a.h = h; a.rows = rows; a.tgt = tgt; a.count = count; a.w = w; a.bias = bias; a.lse_in = lse; a.dloss = dloss;
  a.dh_full = dh_full; a.part_w = part_w; a.part_b = part_b; a.V1 = V1; a.d = d;
  dim3 gdw((unsigned)rbm_cdiv(V1, 16 * warps), S);
#define CE_BWD(DT)                                                                                          \
  do {                                                                                                      \
    if (!set_smem(ce_bwd_dh_kernel<DT>, smem, "rbm_ce_bwd(dh)")) return -1;                               \
    ce_bwd_dh_kernel<DT><<<nblk, 32 * warps, smem, st>>>(a);                                                \
    if (!set_smem(ce_bwd_dw_kernel<DT>, smem, "rbm_ce_bwd(dw)")) return -1;                               \
    ce_bwd_dw_kernel<DT><<<gdw, 32 * warps, smem, st>>>(a);                                                 \
  } while (0)
  if (d <= 32) CE_BWD(4);
  else if (d <= 64) CE_BWD(8);
  else if (d <= 128) CE_BWD(16);
  else CE_BWD(32);
#undef CE_BWD
  RBM_LAUNCH_CHECK("rbm_ce_bwd");
  int64_t n = (int64_t)V1 * d;
  ce_reduce_splits_kernel<<<(unsigned)rbm_cdiv(n, 256), 256, 0, st>>>(part_w, dw, n, S);
  ce_reduce_splits_kernel<<<(unsigned)rbm_cdiv(V1, 256), 256, 0, st>>>(part_b, db, V1, S);
  RBM_LAUNCH_CHECK("rbm_ce_bwd(reduce)");
  return 0;
}
