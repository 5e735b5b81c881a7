// topk.cu -- full-catalogue scoring fused with top-k, standalone top-k, shard merge, ranking metrics.
// Replaces, for evaluation: SAS.predict's gather+matvec (NN/models/sas_model/sas.py:110-114) / BERT's last-position
// logits (NN/trainers/bert.py:47-49) followed by (-scores).argsort(dim=1)[:, :k] and the HR/NDCG/MRR arithmetic
// (NN/trainers/utils.py:36-55).  Scores of the full catalogue never reach HBM: a 64-user x 64-item score tile is
// produced in registers/shared memory, filtered against each user's running k-th best (one compare per score), and
// the rare survivors are inserted into a per-user sorted list that lives in the registers of one warp.
// Order rule everywhere: score descending, item id ascending  (canonical form of the reference's argsort).
#include "common.cuh"
#include "tc_topk.cuh"

namespace {

constexpr int T = 64;
constexpr int LDT = T + 4;
constexpr int KC = 16;
constexpr int64_t ID_NONE = INT64_MAX;

struct Entry {
  float s;
  int64_t id;
};
__device__ __forceinline__ bool better(float s, int64_t id, float ts, int64_t tid) { return s > ts || (s == ts && id < tid); }

// warp-collective insert of candidate (cs, cid) into the sorted list whose t-th entry lives in lane t (t < k)
__device__ __forceinline__ void list_insert(Entry& mine, float cs, int64_t cid, int k, int lane) {
  bool beats_me = better(cs, cid, mine.s, mine.id);
  unsigned keep = __ballot_sync(0xffffffffu, lane < k && !beats_me);  // prefix of entries that stay ahead of cand
  int pos = __popc(keep);
  float up_s = __shfl_up_sync(0xffffffffu, mine.s, 1);
  int64_t up_id = __shfl_up_sync(0xffffffffu, mine.id, 1);
  if (lane < k) {
    if (lane == pos) {
      mine.s = cs;
      mine.id = cid;
    } else if (lane > pos) {
      mine.s = up_s;
      mine.id = up_id;
    }
  }
}

// consider one candidate per lane (valid flag), against the list's current k-th entry
__device__ __forceinline__ void list_offer(Entry& mine, float s, int64_t id, bool valid, int k, int lane) {
  float ts = __shfl_sync(0xffffffffu, mine.s, k - 1);
  int64_t tid = __shfl_sync(0xffffffffu, mine.id, k - 1);
  unsigned m = __ballot_sync(0xffffffffu, valid && better(s, id, ts, tid));
  while (m) {
    int src = __ffs(m) - 1;
    m &= m - 1;
    float cs = __shfl_sync(0xffffffffu, s, src);
    int64_t cid = __shfl_sync(0xffffffffu, id, src);
    list_insert(mine, cs, cid, k, lane);
  }
}

// lane's candidate id is in the ascending row ex[0 .. n) (binary search; only asked of lanes that would enter the list)
__device__ __forceinline__ bool excluded(const int64_t* __restrict__ ex, int n, int64_t id) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (ex[mid] < id) lo = mid + 1;
    else hi = mid;
  }
  return lo < n && ex[lo] == id;
}

// list_offer for a user with an exclusion row (ex, n): the filter runs after the cheap compare, on the rare survivors only
__device__ __forceinline__ void list_offer_excl(Entry& mine, float s, int64_t id, bool valid, int k, int lane, const int64_t* ex, int n) {
  float ts = __shfl_sync(0xffffffffu, mine.s, k - 1);
  int64_t tid = __shfl_sync(0xffffffffu, mine.id, k - 1);
  bool pass = valid && better(s, id, ts, tid);
  if (pass) pass = !excluded(ex, n, id);
  unsigned m = __ballot_sync(0xffffffffu, pass);
  while (m) {
    int src = __ffs(m) - 1;
    m &= m - 1;
    float cs = __shfl_sync(0xffffffffu, s, src);
    int64_t cid = __shfl_sync(0xffffffffu, id, src);
    list_insert(mine, cs, cid, k, lane);
  }
}

__device__ __forceinline__ void list_store(const Entry& mine, float* out_s, int64_t* out_i, int64_t u, int k, int lane) {
  if (lane < k) {
    out_s[u * k + lane] = mine.id == ID_NONE ? -INFINITY : mine.s;
    out_i[u * k + lane] = mine.id == ID_NONE ? -1 : mine.id;
  }
}

// -------------------------------------------------------------------------------- fused scoring + top-k
// EX: row u of excl (stride ld_excl, n_excl ascending output ids) lists what user u must not be offered
template <bool EX>
__global__ void __launch_bounds__(256) score_topk_kernel(const float* __restrict__ f, int64_t ldf, const float* __restrict__ table,
                                                         const float* __restrict__ bias, int64_t v_begin, int64_t v_end, int64_t id_offset,
                                                         float* __restrict__ out_s, int64_t* __restrict__ out_i, int64_t U, int d, int k,
                                                         int64_t tiles_per_split, const int32_t* __restrict__ ulist,
                                                         const int32_t* __restrict__ ucount, const int64_t* __restrict__ excl, int64_t ld_excl,
                                                         int n_excl) {
  // listed mode (ulist != null): row slot j of the launch is user ulist[j], j < *ucount (device-side count); results go
  // to slot j of the partial lists (stride U)
  const int64_t U_eff = ulist ? (int64_t)*ucount : U;
  if ((int64_t)blockIdx.x * T >= U_eff) return;
  extern __shared__ __align__(16) float sm[];
  float* Hst = sm;               // [d][LDT]  users transposed
  float* Wc = Hst + d * LDT;     // [KC][LDT] item chunk transposed
  float* Ss = Wc + KC * LDT;     // [T users][LDT]
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t u0 = (int64_t)blockIdx.x * T;
  {
    int d4 = d >> 2;
    for (int idx = threadIdx.x; idx < T * d4; idx += blockDim.x) {
      int r = idx / d4, c4 = idx - r * d4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (u0 + r < U_eff) v = ld4(f + (ulist ? (int64_t)ulist[u0 + r] : u0 + r) * ldf + c4 * 4);
      Hst[(c4 * 4 + 0) * LDT + r] = v.x;
      Hst[(c4 * 4 + 1) * LDT + r] = v.y;
      Hst[(c4 * 4 + 2) * LDT + r] = v.z;
      Hst[(c4 * 4 + 3) * LDT + r] = v.w;
    }
  }
  Entry lists[8];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    lists[q].s = -INFINITY;
    lists[q].id = ID_NONE;
  }
  int ex_user[8];  // EX: the user (not the slot) of list q; -1 past the last user
  if (EX) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int64_t slot = u0 + warp * 8 + q;
      ex_user[q] = slot < U_eff ? (ulist ? ulist[slot] : (int)slot) : -1;
    }
  }
  const int64_t t_begin = (int64_t)blockIdx.y * tiles_per_split;
  const int64_t n_tiles = (v_end - v_begin + T - 1) / T;
  int64_t t_end = t_begin + tiles_per_split < n_tiles ? t_begin + tiles_per_split : n_tiles;
  for (int64_t it = t_begin; it < t_end; ++it) {
    const int64_t v0 = v_begin + it * T;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < d; k0 += KC) {
      __syncthreads();
      {
        int c = threadIdx.x >> 2, kq = threadIdx.x & 3;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (v0 + c < v_end && k0 + kq * 4 < d) v = ld4(table + (v0 + c) * d + k0 + kq * 4);
        Wc[(kq * 4 + 0) * LDT + c] = v.x;
        Wc[(kq * 4 + 1) * LDT + c] = v.y;
        Wc[(kq * 4 + 2) * LDT + c] = v.z;
        Wc[(kq * 4 + 3) * LDT + c] = v.w;
      }
      __syncthreads();
      int kmax = d - k0 < KC ? d - k0 : KC;
      for (int kk = 0; kk < kmax; ++kk) {
        float4 a = ld4(Hst + (k0 + kk) * LDT + ty * 4);
        float4 b = ld4(Wc + kk * LDT + tx * 4);
        float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      }
    }
    {
      int64_t cb = v0 + tx * 4;
      float4 bb = make_float4(0.f, 0.f, 0.f, 0.f);
      if (bias) {
        bb.x = cb + 0 < v_end ? bias[cb + 0] : 0.f;
        bb.y = cb + 1 < v_end ? bias[cb + 1] : 0.f;
        bb.z = cb + 2 < v_end ? bias[cb + 2] : 0.f;
        bb.w = cb + 3 < v_end ? bias[cb + 3] : 0.f;
      }
#pragma unroll
      for (int i = 0; i < 4; ++i)
        st4(Ss + (ty * 4 + i) * LDT + tx * 4, make_float4(acc[i][0] + bb.x, acc[i][1] + bb.y, acc[i][2] + bb.z, acc[i][3] + bb.w));
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float* row = Ss + (warp * 8 + q) * LDT;
#pragma unroll
      for (int hlf = 0; hlf < 2; ++hlf) {
        int c = lane + 32 * hlf;
        int64_t v = v0 + c;
        if (EX) list_offer_excl(lists[q], row[c], v + id_offset, v < v_end, k, lane, excl + (int64_t)ex_user[q] * ld_excl, ex_user[q] < 0 ? 0 : n_excl);
        else list_offer(lists[q], row[c], v + id_offset, v < v_end, k, lane);
      }
    }
  }
  float* ps = out_s + (int64_t)blockIdx.y * U * k;
  int64_t* pi = out_i + (int64_t)blockIdx.y * U * k;
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    int64_t u = u0 + warp * 8 + q;
    if (u < U_eff) list_store(lists[q], ps, pi, u, k, lane);
  }
}

// ---------------------------------------------------------------------- top-k of materialised score rows
__global__ void __launch_bounds__(256) topk_rows_kernel(const float* __restrict__ scores, int64_t ld, float* __restrict__ out_s,
                                                        int64_t* __restrict__ out_i, int64_t U, int64_t C, int k, int64_t id_offset) {
  int lane = threadIdx.x & 31;
  int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= U) return;
  Entry mine{-INFINITY, ID_NONE};
  const float* row = scores + u * ld;
  for (int64_t c0 = 0; c0 < C; c0 += 32) {
    int64_t c = c0 + lane;
    float s = c < C ? row[c] : 0.f;
    list_offer(mine, s, c + id_offset, c < C, k, lane);
  }
  list_store(mine, out_s, out_i, u, k, lane);
}

__global__ void __launch_bounds__(256) topk_merge_kernel(const float* __restrict__ in_s, const int64_t* __restrict__ in_i,
                                                         float* __restrict__ out_s, int64_t* __restrict__ out_i, int S, int64_t U, int k,
                                                         const int32_t* __restrict__ ulist, const int32_t* __restrict__ ucount) {
  int lane = threadIdx.x & 31;
  int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (u >= (ulist ? (int64_t)*ucount : U)) return;
  Entry mine{-INFINITY, ID_NONE};
  for (int s = 0; s < S; ++s) {
    const float* ps = in_s + ((int64_t)s * U + u) * k;
    const int64_t* pi = in_i + ((int64_t)s * U + u) * k;
    float cs = lane < k ? ps[lane] : 0.f;
    int64_t cid = lane < k ? pi[lane] : -1;
    list_offer(mine, cs, cid, lane < k && cid >= 0, k, lane);
  }
  list_store(mine, out_s, out_i, ulist ? (int64_t)ulist[u] : u, k, lane);  // listed mode: slot u holds user ulist[u]
}

// ------------------------------------------------------------------------------------- ranking metrics
#define MAX_KS 8
struct KsArg {
  int32_t ks[MAX_KS];
  int nk;
};

__global__ void __launch_bounds__(128) rank_metrics_kernel(const int64_t* __restrict__ top_ids, const int64_t* __restrict__ labels,
                                                           const int64_t* __restrict__ positives, const float* __restrict__ w_ndcg,
                                                           const float* __restrict__ w_mrr, KsArg ka, float* __restrict__ per_user,
                                                           int64_t U, int K, int64_t C, int64_t id_offset) {
  int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= U) return;
  int64_t n_pos = 1;
  if (labels) {
    n_pos = 0;
    for (int64_t c = 0; c < C; ++c) n_pos += labels[u * C + c];
  }
  for (int j = 0; j < ka.nk; ++j) {
    int k = ka.ks[j];
    float hits = 0.f, dcg = 0.f, mrr = 0.f;
    for (int t = 0; t < k; ++t) {
      int64_t id = top_ids[u * K + t];
      float hit;
      if (labels) {
        int64_t c = id - id_offset;
        hit = (id >= 0 && c >= 0 && c < C) ? (float)labels[u * C + c] : 0.f;
      } else {
        hit = id == positives[u] ? 1.f : 0.f;
      }
      hits += hit;
      dcg += hit * w_ndcg[t];
      mrr += hit * w_mrr[t];
    }
    float idcg = 0.f;
    int lim = n_pos < k ? (int)n_pos : k;
    for (int t = 0; t < lim; ++t) idcg += w_ndcg[t];
    float* o = per_user + (u * ka.nk + j) * 3;
    o[0] = hits / (float)n_pos;
    o[1] = dcg / idcg;
    o[2] = mrr;
  }
}

// two-stage column mean in double, fixed order
__global__ void __launch_bounds__(256) colmean_partial_kernel(const float* __restrict__ x, double* __restrict__ partial, int64_t U, int cols,
                                                              int64_t rows_per_block) {
  int c = threadIdx.x;
  if (c >= cols) return;
  int64_t r0 = (int64_t)blockIdx.x * rows_per_block, r1 = r0 + rows_per_block < U ? r0 + rows_per_block : U;
  double s = 0.0;
  for (int64_t r = r0; r < r1; ++r) s += (double)x[r * cols + c];
  partial[(int64_t)blockIdx.x * cols + c] = s;
}
__global__ void colmean_final_kernel(const double* __restrict__ partial, float* __restrict__ out, int nblk, int cols, int64_t U) {
  int c = threadIdx.x;
  if (c >= cols) return;
  double s = 0.0;
  for (int b = 0; b < nblk; ++b) s += partial[(int64_t)b * cols + c];
  out[c] = (float)(s / (double)U);
}

int topk_splits(int64_t U, int64_t n_items) {
  int64_t ut = rbm_cdiv(U, T), it = rbm_cdiv(n_items, T);
  int64_t s = rbm_cdiv((int64_t)RBM_NUM_SMS * 2, ut);
  if (s > it) s = it;
  if (s > 64) s = 64;
  return (int)(s < 1 ? 1 : s);
}

}  // namespace

extern "C" size_t rbm_score_topk_ws_bytes_d(int64_t U, int64_t n_items, int d, int k) {
  size_t S = (size_t)topk_splits(U, n_items);
  size_t simt = S * (size_t)U * k * (sizeof(float) + sizeof(int64_t)) + 256;
  size_t tc = rbm_tc_topk_ws_bytes(U, n_items, d, k);
  return simt > tc ? simt : tc;
}

extern "C" size_t rbm_score_topk_ws_bytes(int64_t U, int64_t n_items, int k) {
  size_t best = 0;
  for (int d = 32; d <= 256; d *= 2) {  // d is not part of this query: cover every hidden size the tcgen05 path takes
    size_t b = rbm_score_topk_ws_bytes_d(U, n_items, d, k);
    if (b > best) best = b;
  }
  return best;
}

static size_t simt_smem(int d) { return sizeof(float) * ((size_t)d * LDT + KC * LDT + T * LDT); }

// one launch of the fp32 scan kernel: EX instantiation exactly when there is something to exclude
static void launch_score_topk(dim3 grid, size_t smem, cudaStream_t st, const float* f, int64_t ldf, const float* table, const float* bias,
                              int64_t v_begin, int64_t v_end, int64_t id_offset, float* out_s, int64_t* out_i, int64_t U, int d, int k,
                              int64_t tps, const int32_t* ulist, const int32_t* ucount, const int64_t* excl, int64_t ld_excl, int n_excl) {
  if (excl && n_excl > 0)
    score_topk_kernel<true><<<grid, 256, smem, st>>>(f, ldf, table, bias, v_begin, v_end, id_offset, out_s, out_i, U, d, k, tps, ulist, ucount,
                                                     excl, ld_excl, n_excl);
  else
    score_topk_kernel<false><<<grid, 256, smem, st>>>(f, ldf, table, bias, v_begin, v_end, id_offset, out_s, out_i, U, d, k, tps, ulist, ucount,
                                                      nullptr, 0, 0);
}

static bool set_simt_smem(size_t smem, const char* name) {
  return set_smem(score_topk_kernel<false>, smem, name) && set_smem(score_topk_kernel<true>, smem, name);
}

extern "C" int rbm_score_topk(const float* f, int64_t ldf, const float* table, const float* bias, int64_t v_begin, int64_t v_end,
                              int64_t id_offset, float* top_scores, int64_t* top_ids, int64_t U, int d, int k, void* ws,
                              size_t ws_bytes, rbm_stream_t stream) {
  return rbm_score_topk_excl(f, ldf, table, bias, v_begin, v_end, id_offset, nullptr, 0, 0, top_scores, top_ids, U, d, k, ws, ws_bytes, stream);
}

extern "C" int rbm_score_topk_excl(const float* f, int64_t ldf, const float* table, const float* bias, int64_t v_begin, int64_t v_end,
                                   int64_t id_offset, const int64_t* excl, int64_t ld_excl, int n_excl, float* top_scores,
                                   int64_t* top_ids, int64_t U, int d, int k, void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(f && table && top_scores && top_ids && ws, "rbm_score_topk: null pointer");
  RBM_REQUIRE(n_excl >= 0 && (n_excl == 0 || (excl && ld_excl >= n_excl)), "rbm_score_topk_excl: bad exclusion matrix (n_excl=%d, ld_excl=%lld)",
              n_excl, (long long)ld_excl);
  RBM_REQUIRE(U > 0 && v_begin >= 0 && v_end > v_begin, "rbm_score_topk: empty user or item range");
  RBM_REQUIRE(k >= 1 && k <= 32, "rbm_score_topk: k=%d out of [1,32]", k);
  RBM_REQUIRE(d >= 4 && d % 4 == 0 && d <= 256 && ldf % 4 == 0 && ldf >= d, "rbm_score_topk: unsupported d=%d (need d%%4==0, d<=256)", d);
  RBM_REQUIRE(ws_bytes >= rbm_score_topk_ws_bytes_d(U, v_end - v_begin, d, k), "rbm_score_topk: workspace too small");
  RBM_REQUIRE(rbm_aligned16(f) && rbm_aligned16(table) && rbm_aligned16(ws), "rbm_score_topk: pointers must be 16B aligned");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t n_items = v_end - v_begin;
  // catalogue-scale path: tcgen05 candidate selection + exact fp32 re-score (tc_topk.cu)
  if (rbm_tc_topk_supported(U, n_items, d, k, ldf, f, table))
    return rbm_tc_topk_launch(f, ldf, table, bias, v_begin, v_end, id_offset, excl, ld_excl, n_excl, top_scores, top_ids, U, d, k, ws, st);
  int S = topk_splits(U, n_items);
  int64_t tps = rbm_cdiv(rbm_cdiv(n_items, T), S);
  size_t smem = simt_smem(d);
  if (!set_simt_smem(smem, "rbm_score_topk")) return -1;
  int64_t* part_i = (int64_t*)ws;
  float* part_s = (float*)(part_i + (size_t)S * U * k);
  dim3 grid((unsigned)rbm_cdiv(U, T), S);
  if (S == 1) {
    launch_score_topk(grid, smem, st, f, ldf, table, bias, v_begin, v_end, id_offset, top_scores, top_ids, U, d, k, tps, nullptr, nullptr, excl,
                      ld_excl, n_excl);
    RBM_LAUNCH_CHECK("rbm_score_topk");
  } else {
    launch_score_topk(grid, smem, st, f, ldf, table, bias, v_begin, v_end, id_offset, part_s, part_i, U, d, k, tps, nullptr, nullptr, excl, ld_excl,
                      n_excl);
    RBM_LAUNCH_CHECK("rbm_score_topk");
    topk_merge_kernel<<<(unsigned)rbm_cdiv(U, 8), 256, 0, st>>>(part_s, part_i, top_scores, top_ids, S, U, k, nullptr, nullptr);
    RBM_LAUNCH_CHECK("rbm_score_topk(merge)");
  }
  return 0;
}

// exact fp32 scan + top-k of the users ulist[0 .. *ucount) (tc_topk.cu stage 3): partial lists per item split, then merge
int rbm_simt_topk_listed(const float* f, int64_t ldf, const float* table, const float* bias, int64_t v_begin, int64_t v_end,
                         int64_t id_offset, const int64_t* excl, int64_t ld_excl, int n_excl, float* top_scores, int64_t* top_ids, int64_t U,
                         int d, int k, const int32_t* ulist, const int32_t* ucount, void* part_ws, int S, cudaStream_t st) {
  int64_t tps = rbm_cdiv(rbm_cdiv(v_end - v_begin, T), S);
  size_t smem = simt_smem(d);
  if (!set_simt_smem(smem, "rbm_score_topk(exact re-scan)")) return -1;
  int64_t* part_i = (int64_t*)part_ws;
  float* part_s = (float*)(part_i + (size_t)S * U * k);
  dim3 grid((unsigned)rbm_cdiv(U, T), S);
  launch_score_topk(grid, smem, st, f, ldf, table, bias, v_begin, v_end, id_offset, part_s, part_i, U, d, k, tps, ulist, ucount, excl, ld_excl,
                    n_excl);
  RBM_LAUNCH_CHECK("rbm_score_topk(exact re-scan)");
  topk_merge_kernel<<<(unsigned)rbm_cdiv(U, 8), 256, 0, st>>>(part_s, part_i, top_scores, top_ids, S, U, k, ulist, ucount);
  RBM_LAUNCH_CHECK("rbm_score_topk(exact re-scan merge)");
  return 0;
}

extern "C" int rbm_topk_rows(const float* scores, int64_t ld, float* top_scores, int64_t* top_ids, int64_t U, int64_t C, int k,
                             int64_t id_offset, rbm_stream_t stream) {
  RBM_REQUIRE(scores && top_scores && top_ids, "rbm_topk_rows: null pointer");
  RBM_REQUIRE(U > 0 && C > 0 && ld >= C && k >= 1 && k <= 32, "rbm_topk_rows: bad sizes (k must be in [1,32])");
  topk_rows_kernel<<<(unsigned)rbm_cdiv(U, 8), 256, 0, (cudaStream_t)stream>>>(scores, ld, top_scores, top_ids, U, C, k, id_offset);
  RBM_LAUNCH_CHECK("rbm_topk_rows");
  return 0;
}

extern "C" int rbm_topk_merge(const float* scores, const int64_t* ids, float* out_scores, int64_t* out_ids, int S, int64_t U, int k,
                              rbm_stream_t stream) {
  RBM_REQUIRE(scores && ids && out_scores && out_ids, "rbm_topk_merge: null pointer");
  RBM_REQUIRE(S >= 1 && U > 0 && k >= 1 && k <= 32, "rbm_topk_merge: bad sizes");
  topk_merge_kernel<<<(unsigned)rbm_cdiv(U, 8), 256, 0, (cudaStream_t)stream>>>(scores, ids, out_scores, out_ids, S, U, k, nullptr, nullptr);
  RBM_LAUNCH_CHECK("rbm_topk_merge");
  return 0;
}

extern "C" int rbm_rank_metrics(const int64_t* top_ids, const int64_t* labels, const int64_t* positives, const float* w_ndcg,
                                const float* w_mrr, const int32_t* ks_host, int nk, float* per_user, int64_t U, int K, int64_t C,
                                int64_t id_offset, rbm_stream_t stream) {
  RBM_REQUIRE(top_ids && (labels || positives) && w_ndcg && w_mrr && ks_host && per_user, "rbm_rank_metrics: null pointer");
  RBM_REQUIRE(nk >= 1 && nk <= MAX_KS && U > 0 && K >= 1, "rbm_rank_metrics: bad sizes (at most %d cut-offs)", MAX_KS);
  KsArg ka{};
  ka.nk = nk;
  for (int j = 0; j < nk; ++j) {
    RBM_REQUIRE(ks_host[j] >= 1 && ks_host[j] <= K, "rbm_rank_metrics: cut-off %d outside [1,%d]", ks_host[j], K);
    ka.ks[j] = ks_host[j];
  }
  rank_metrics_kernel<<<(unsigned)rbm_cdiv(U, 128), 128, 0, (cudaStream_t)stream>>>(top_ids, labels, positives, w_ndcg, w_mrr, ka, per_user, U, K, C, id_offset);
  RBM_LAUNCH_CHECK("rbm_rank_metrics");
  return 0;
}

static int colmean_blocks(int64_t U) {
  int64_t nb = rbm_cdiv(U, 4096);
  return (int)(nb < 1 ? 1 : (nb > 1024 ? 1024 : nb));
}
extern "C" size_t rbm_column_mean_ws_bytes(int64_t U, int cols) { return (size_t)colmean_blocks(U) * cols * sizeof(double); }

extern "C" int rbm_column_mean(const float* x, float* out, int64_t U, int cols, void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(x && out && ws && U > 0 && cols >= 1 && cols <= 256, "rbm_column_mean: bad arguments (cols <= 256)");
  RBM_REQUIRE(ws_bytes >= rbm_column_mean_ws_bytes(U, cols), "rbm_column_mean: workspace too small");
  int nblk = colmean_blocks(U);
  int64_t rpb = rbm_cdiv(U, nblk);
  colmean_partial_kernel<<<nblk, 256, 0, (cudaStream_t)stream>>>(x, (double*)ws, U, cols, rpb);
  colmean_final_kernel<<<1, 256, 0, (cudaStream_t)stream>>>((const double*)ws, out, nblk, cols, U);
  RBM_LAUNCH_CHECK("rbm_column_mean");
  return 0;
}
