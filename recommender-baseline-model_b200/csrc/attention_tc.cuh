// (L = keys per sequence, Lq = query rows per sequence: equal except for rbm_attn_fwd_lq / rbm_attn_bwd_lq)
// attention_tc.cuh -- internal interface of the tcgen05 attention forward (attention_tc.cu), dispatched from attention.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// false under RBM_ATTN_IMPL=mma; gates the tcgen05 kernels of attention_tc.cu, attention_pair.cu and attention_seq.cu
bool rbm_attn_tc_enabled();

bool rbm_attn_fwd_tc_supported(int L, int dk, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, const void* q, const void* k,
                               const void* v, const void* out);
int rbm_attn_fwd_tc_launch(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const int64_t* tok,
                           float* out, int64_t ldo, float* stats, int B, int L, int Lq, int h, int mask_mode, float scale, float p,
                           uint64_t seed, uint64_t site, cudaStream_t st);

// backward pass A (dQ + delta) on the tensor path
bool rbm_attn_bwd_dq_tc_supported(int L, int dk, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, int64_t lddo, int64_t lddq,
                                  const void* q, const void* k, const void* v, const void* o, const void* dout, const void* dq);
int rbm_attn_bwd_dq_tc_launch(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const int64_t* tok,
                              const float* o, int64_t ldo, const float* dout, int64_t lddo, const float* stats, float* dq, int64_t lddq,
                              float* delta, int B, int L, int Lq, int h, int mask_mode, float scale, float p, uint64_t seed,
                              uint64_t site, cudaStream_t st);

// backward pass B (dK, dV) on the tensor path; needs the delta written by pass A
bool rbm_attn_bwd_dkv_tc_supported(int L, int dk, int64_t ldq, int64_t ldk, int64_t ldv, int64_t lddo, int64_t lddk, int64_t lddv,
                                   const void* q, const void* k, const void* v, const void* dout, const void* dk_, const void* dv);
int rbm_attn_bwd_dkv_tc_launch(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv, const int64_t* tok,
                               const float* dout, int64_t lddo, const float* stats, const float* delta, float* dk_, int64_t lddk,
                               float* dv, int64_t lddv, int B, int L, int Lq, int h, int mask_mode, float scale, float p, uint64_t seed,
                               uint64_t site, cudaStream_t st);
