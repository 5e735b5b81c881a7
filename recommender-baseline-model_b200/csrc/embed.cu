// embed.cu -- embedding stage: row gather (+scale) + positional add + dropout + pad-row zeroing, fwd/bwd.
// Replaces NN/models/sas_model/sas.py:60-67 and NN/models/bert_modules/embedding/bert.py:29-31.
// HBM-bound: one 16-byte load per thread from the table row, one from the positional row, one 16-byte store.
#include "common.cuh"

__global__ void __launch_bounds__(256) embed_fwd_kernel(const int64_t* __restrict__ tok, const float* __restrict__ table,
                                                        const float* __restrict__ pos, float* __restrict__ out,
                                                        int64_t total4, int L, int d4, int64_t vocab, int64_t v_begin,
                                                        int64_t v_end, float scale, int zero_pad, uint32_t thr,
                                                        float inv_keep, uint64_t seed, uint64_t site) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  int64_t r = i / d4;
  int c4 = (int)(i - r * d4);
  int64_t t = tok[r];
  float4 o;
  if (zero_pad && t == 0) {
    o = make_float4(0.f, 0.f, 0.f, 0.f);
  } else if (t < 0 || t >= vocab) {
    float n = __int_as_float(0x7fc00000);  // out-of-range index: poison the row so it cannot go unnoticed
    o = make_float4(n, n, n, n);
  } else if (t < v_begin || t >= v_end) {
    o = make_float4(0.f, 0.f, 0.f, 0.f);  // row held by another shard: its owner writes the value, the exchange adds zeros
  } else {
    float4 e = ld4(table + (t - v_begin) * (int64_t)d4 * 4 + c4 * 4);
    float4 pe = ld4(pos + (int64_t)(r % L) * d4 * 4 + c4 * 4);
    o = make_float4(e.x * scale + pe.x, e.y * scale + pe.y, e.z * scale + pe.z, e.w * scale + pe.w);
    if (thr) {
      float4 m = rbm_drop4(seed, rbm_site(site), (uint64_t)i, thr, inv_keep);
      o.x *= m.x; o.y *= m.y; o.z *= m.z; o.w *= m.w;
    }
  }
  st4(out + i * 4, o);
}

// block (16,16): x = float4 column inside a 16-column group, y = batch lane; one block per (position l, group)
__global__ void __launch_bounds__(256) embed_bwd_kernel(const int64_t* __restrict__ tok, const float* __restrict__ dout,
                                                        float* __restrict__ g, float* __restrict__ dpos, int B, int L,
                                                        int d4, int zero_pad, uint32_t thr, float inv_keep,
                                                        uint64_t seed, uint64_t site, uint64_t elem_offset4) {
  __shared__ float4 red[16][16];
  int l = blockIdx.x;
  int c4 = blockIdx.y * 16 + threadIdx.x;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c4 < d4) {
    for (int b = threadIdx.y; b < B; b += 16) {
      int64_t r = (int64_t)b * L + l;
      int64_t i = r * d4 + c4;
      float4 v = ld4(dout + i * 4);
      if (zero_pad && tok[r] == 0) {
        v = make_float4(0.f, 0.f, 0.f, 0.f);
      } else if (thr) {
        float4 m = rbm_drop4(seed, rbm_site(site), (uint64_t)i + elem_offset4, thr, inv_keep);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      st4(g + i * 4, v);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c4 < d4) {
    float4 s = red[0][threadIdx.x];
#pragma unroll
    for (int y = 1; y < 16; ++y) {
      float4 t = red[y][threadIdx.x];
      s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
    }
    st4(dpos + ((int64_t)l * d4 + c4) * 4, s);
  }
}

// ---- the same backward on the live (token != 0) rows only (csrc/rows.cu): dout_c / g_c are [cap, d] compact tensors, row r is row
// rows[r] of the [B, L] batch.  The dropout stream is still indexed by the element's place in the full batch.
__global__ void __launch_bounds__(256) embed_bwd_rows_kernel(const int64_t* __restrict__ tok, const int32_t* __restrict__ rows,
                                                             const int32_t* __restrict__ count, int64_t cap, const float* __restrict__ dout_c,
                                                             float* __restrict__ g_c, int64_t* __restrict__ idx_c, int d4, uint32_t thr,
                                                             float inv_keep, uint64_t seed, uint64_t site) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cap * d4) return;
  const int64_t r = i / d4;
  const int c4 = (int)(i - r * d4);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  int64_t t = 0;
  if (r < *count) {
    const int64_t row = rows[r];
    t = tok[row];
    v = ld4(dout_c + i * 4);
    if (thr) {
      const float4 m = rbm_drop4(seed, rbm_site(site), (uint64_t)(row * d4 + c4), thr, inv_keep);
      v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
    }
  }
  st4(g_c + i * 4, v);
  if (c4 == 0) idx_c[r] = t;
}
// positional-table gradient, stage 1: block b walks its contiguous range of compact rows in ascending order and adds each into a
// private [L, d] image in shared memory (thread = float4 column: no two threads touch one cell); stage 2 adds the images in block order
constexpr int EPOS_BLOCKS = RBM_NUM_SMS;
__global__ void embed_dpos_partial_kernel(const int32_t* __restrict__ rows, const int32_t* __restrict__ count, const float* __restrict__ g_c,
                                          int L, int d4, float* __restrict__ part) {
  extern __shared__ float4 img[];
  for (int e = threadIdx.x; e < L * d4; e += blockDim.x) img[e] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  const int64_t n = *count, per = (n + gridDim.x - 1) / gridDim.x, r0 = blockIdx.x * per, r1 = r0 + per < n ? r0 + per : n;
  for (int c4 = threadIdx.x; c4 < d4; c4 += blockDim.x)
    for (int64_t r = r0; r < r1; ++r) {
      const int l = rows[r] % L;
      const float4 v = ld4(g_c + (r * d4 + c4) * 4);
      float4& a = img[l * d4 + c4];
      a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
    }
  __syncthreads();
  float4* out = reinterpret_cast<float4*>(part) + (int64_t)blockIdx.x * L * d4;
  for (int e = threadIdx.x; e < L * d4; e += blockDim.x) out[e] = img[e];
}
__global__ void __launch_bounds__(256) embed_dpos_final_kernel(const float* __restrict__ part, int nb, int64_t n4, float* __restrict__ dpos) {
  const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n4) return;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int b0 = 0; b0 < nb; b0 += 4) {  // four loads in flight, added in block order
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = b0 + u < nb ? ld4(part + ((int64_t)(b0 + u) * n4 + e) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int u = 0; u < 4; ++u) { s.x += v[u].x; s.y += v[u].y; s.z += v[u].z; s.w += v[u].w; }
  }
  st4(dpos + e * 4, s);
}

__global__ void dropout_mask_kernel(uint8_t* out, int64_t n, uint32_t thr, uint64_t seed, uint64_t site) {
  int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 * 4 >= n) return;
  uint4 r = rbm_philox_drop(seed, site, (uint64_t)i4);
  uint32_t v[4] = {r.x, r.y, r.z, r.w};
  for (int c = 0; c < 4; ++c)
    if (i4 * 4 + c < n) out[i4 * 4 + c] = v[c] >= thr ? 1 : 0;
}

__global__ void dropout_mask_attn_kernel(uint8_t* out, int64_t rows, int L, uint32_t thr16, uint64_t seed, uint64_t site) {
  int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= rows * L) return;
  int64_t R = e / L;  // R = bh * L + i
  int j = (int)(e - R * L);
  out[e] = rbm_attn_keep(seed, site, (uint64_t)(R / L), (int)(R % L), j, thr16) ? 1 : 0;
}

extern "C" int rbm_embed_fwd_shard(const int64_t* tok, const float* table_shard, const float* pos, float* out, int64_t rows, int L,
                                   int d, int64_t vocab, int64_t v_begin, int64_t v_end, float scale, int zero_pad, float p,
                                   uint64_t seed, uint64_t site, rbm_stream_t stream);

extern "C" int rbm_embed_fwd(const int64_t* tok, const float* table, const float* pos, float* out, int64_t rows, int L,
                             int d, int64_t vocab, float scale, int zero_pad, float p, uint64_t seed, uint64_t site,
                             rbm_stream_t stream) {
  return rbm_embed_fwd_shard(tok, table, pos, out, rows, L, d, vocab, 0, vocab, scale, zero_pad, p, seed, site, stream);
}

extern "C" int rbm_embed_fwd_shard(const int64_t* tok, const float* table, const float* pos, float* out, int64_t rows, int L,
                                   int d, int64_t vocab, int64_t v_begin, int64_t v_end, float scale, int zero_pad, float p,
                                   uint64_t seed, uint64_t site, rbm_stream_t stream) {
  // an empty shard (v_begin == v_end) is never read: its table may be NULL, which is what a zero-row tensor hands over
  RBM_REQUIRE(tok && (table || v_begin == v_end) && pos && out, "rbm_embed_fwd: null pointer");
  RBM_REQUIRE(v_begin >= 0 && v_begin <= v_end && v_end <= vocab, "rbm_embed_fwd: bad shard range [%lld, %lld) of %lld rows",
              (long long)v_begin, (long long)v_end, (long long)vocab);
  RBM_REQUIRE(d > 0 && d % 4 == 0, "rbm_embed_fwd: d=%d must be a positive multiple of 4", d);
  RBM_REQUIRE(L > 0 && rows >= 0 && rows % L == 0, "rbm_embed_fwd: rows=%lld not a multiple of L=%d", (long long)rows, L);
  RBM_REQUIRE(p >= 0.f && p < 1.f, "rbm_embed_fwd: dropout p=%f out of [0,1)", p);
  RBM_REQUIRE(rbm_aligned16(table) && rbm_aligned16(pos) && rbm_aligned16(out), "rbm_embed_fwd: pointers must be 16B aligned");
  if (rows == 0) return 0;
  int64_t total4 = rows * (d / 4);
  uint32_t thr = rbm_drop_threshold(p);
  embed_fwd_kernel<<<(unsigned)rbm_cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(
      tok, table, pos, out, total4, L, d / 4, vocab, v_begin, v_end, scale, zero_pad, thr, 1.f / (1.f - p), seed, site);
  RBM_LAUNCH_CHECK("rbm_embed_fwd");
  return 0;
}

extern "C" int rbm_embed_bwd_offset(const int64_t* tok, const float* dout, float* g, float* dpos, int64_t rows, int L, int d,
                                    int zero_pad, float p, uint64_t seed, uint64_t site, uint64_t row_offset, rbm_stream_t stream);

extern "C" int rbm_embed_bwd(const int64_t* tok, const float* dout, float* g, float* dpos, int64_t rows, int L, int d,
                             int zero_pad, float p, uint64_t seed, uint64_t site, rbm_stream_t stream) {
  return rbm_embed_bwd_offset(tok, dout, g, dpos, rows, L, d, zero_pad, p, seed, site, 0, stream);
}

extern "C" int rbm_embed_bwd_offset(const int64_t* tok, const float* dout, float* g, float* dpos, int64_t rows, int L, int d,
                                    int zero_pad, float p, uint64_t seed, uint64_t site, uint64_t row_offset, rbm_stream_t stream) {
  RBM_REQUIRE(tok && dout && g && dpos, "rbm_embed_bwd: null pointer");
  RBM_REQUIRE(d > 0 && d % 4 == 0, "rbm_embed_bwd: d=%d must be a positive multiple of 4", d);
  RBM_REQUIRE(L > 0 && rows > 0 && rows % L == 0, "rbm_embed_bwd: rows=%lld not a positive multiple of L=%d", (long long)rows, L);
  RBM_REQUIRE(p >= 0.f && p < 1.f, "rbm_embed_bwd: dropout p=%f out of [0,1)", p);
  RBM_REQUIRE(rbm_aligned16(dout) && rbm_aligned16(g) && rbm_aligned16(dpos), "rbm_embed_bwd: pointers must be 16B aligned");
  int d4 = d / 4;
  dim3 grid(L, (unsigned)rbm_cdiv(d4, 16)), block(16, 16);
  embed_bwd_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(tok, dout, g, dpos, (int)(rows / L), L, d4, zero_pad,
                                                             rbm_drop_threshold(p), 1.f / (1.f - p), seed, site, row_offset * (uint64_t)d4);
  RBM_LAUNCH_CHECK("rbm_embed_bwd");
  return 0;
}

extern "C" size_t rbm_embed_bwd_rows_ws_bytes(int L, int d) { return (size_t)EPOS_BLOCKS * L * d * sizeof(float); }

extern "C" int rbm_embed_bwd_rows(const int64_t* tok, const int32_t* rows, const int32_t* count, int64_t cap, const float* dout_c,
                                  float* g_c, int64_t* idx_c, float* dpos, int L, int d, float p, uint64_t seed, uint64_t site,
                                  void* ws, size_t ws_bytes, rbm_stream_t stream) {
  RBM_REQUIRE(tok && rows && count && dout_c && g_c && idx_c && dpos && ws, "rbm_embed_bwd_rows: null pointer");
  RBM_REQUIRE(d > 0 && d % 4 == 0 && L > 0 && cap > 0, "rbm_embed_bwd_rows: bad shape (d=%d L=%d)", d, L);
  RBM_REQUIRE(p >= 0.f && p < 1.f, "rbm_embed_bwd_rows: dropout p=%f out of [0,1)", p);
  RBM_REQUIRE((size_t)L * d * sizeof(float) <= 96 * 1024, "rbm_embed_bwd_rows: L*d*4 = %zu B exceeds the 96 KB shared-memory image",
              (size_t)L * d * sizeof(float));
  RBM_REQUIRE(ws_bytes >= rbm_embed_bwd_rows_ws_bytes(L, d), "rbm_embed_bwd_rows: workspace too small");
  RBM_REQUIRE(rbm_aligned16(dout_c) && rbm_aligned16(g_c) && rbm_aligned16(dpos) && rbm_aligned16(ws), "rbm_embed_bwd_rows: pointers must be 16B aligned");
  const int d4 = d / 4;
  embed_bwd_rows_kernel<<<(unsigned)rbm_cdiv(cap * d4, 256), 256, 0, (cudaStream_t)stream>>>(tok, rows, count, cap, dout_c, g_c, idx_c, d4,
                                                                                           rbm_drop_threshold(p), 1.f / (1.f - p), seed, site);
  RBM_LAUNCH_CHECK("rbm_embed_bwd_rows");
  const size_t smem = (size_t)L * d * sizeof(float);
  static size_t smem_set = 0;
  if (smem > 48 * 1024 && smem > smem_set) {
    if (!set_smem(embed_dpos_partial_kernel, smem, "rbm_embed_bwd_rows")) return -1;
    smem_set = smem;
  }
  const int threads = d4 <= 32 ? 32 : (d4 <= 64 ? 64 : 128);
  embed_dpos_partial_kernel<<<EPOS_BLOCKS, threads, smem, (cudaStream_t)stream>>>(rows, count, g_c, L, d4, (float*)ws);
  RBM_LAUNCH_CHECK("rbm_embed_bwd_rows(dpos partial)");
  const int64_t n4 = (int64_t)L * d4;
  embed_dpos_final_kernel<<<(unsigned)rbm_cdiv(n4, 256), 256, 0, (cudaStream_t)stream>>>((const float*)ws, EPOS_BLOCKS, n4, dpos);
  RBM_LAUNCH_CHECK("rbm_embed_bwd_rows(dpos)");
  return 0;
}

extern "C" int rbm_dropout_mask(uint8_t* out, int64_t n, float p, uint64_t seed, uint64_t site, rbm_stream_t stream) {
  RBM_REQUIRE(out && n >= 0 && p >= 0.f && p < 1.f, "rbm_dropout_mask: bad argument");
  if (n == 0) return 0;
  dropout_mask_kernel<<<(unsigned)rbm_cdiv(rbm_cdiv(n, 4), 256), 256, 0, (cudaStream_t)stream>>>(out, n, rbm_drop_threshold(p), seed, site);
  RBM_LAUNCH_CHECK("rbm_dropout_mask");
  return 0;
}

extern "C" int rbm_dropout_mask_attn(uint8_t* out, int64_t rows, int L, float p, uint64_t seed, uint64_t site,
                                     rbm_stream_t stream) {
  RBM_REQUIRE(out && rows >= 0 && L > 0 && L <= 256 && p >= 0.f && p < 1.f, "rbm_dropout_mask_attn: bad argument");
  if (rows == 0) return 0;
  dropout_mask_attn_kernel<<<(unsigned)rbm_cdiv(rows * L, 256), 256, 0, (cudaStream_t)stream>>>(out, rows, L, rbm_drop_threshold16(p), seed, site);
  RBM_LAUNCH_CHECK("rbm_dropout_mask_attn");
  return 0;
}

RBM_DEFINE_STEP_PTR_SETTER(rbm_step_ptr_set_embed)
