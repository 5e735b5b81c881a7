// tc_topk.cuh -- internal interface of the tcgen05 full-catalogue scoring + candidate selection (tc_topk.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

int rbm_tc_topk_splits(int64_t U, int64_t n_items, int d);
size_t rbm_tc_topk_ws_bytes(int64_t U, int64_t n_items, int d, int k);
int rbm_tc_topk_fb_splits(int64_t U, int64_t n_items, int k);
bool rbm_tc_topk_supported(int64_t U, int64_t n_items, int d, int k, int64_t ldf, const void* f, const void* table);
// excl: NULL or row u = user u's excluded output ids, ascending (row stride ld_excl, n_excl entries); see rbm_score_topk_excl
int rbm_tc_topk_launch(const float* f, int64_t ldf, const float* table, const float* bias, int64_t v_begin, int64_t v_end,
                       int64_t id_offset, const int64_t* excl, int64_t ld_excl, int n_excl, float* top_scores, int64_t* top_ids, int64_t U,
                       int d, int k, void* ws, cudaStream_t st);
// topk.cu: exact fp32 scan + top-k of the users named by ulist[0 .. *ucount) (device-side list and count; no host sync);
// their rows of top_scores / top_ids are overwritten.  part_ws >= S * U * k * 12 bytes.  excl (NULL: none) is indexed by the
// user, not by the slot of the list.
int rbm_simt_topk_listed(const float* f, int64_t ldf, const float* table, const float* bias, int64_t v_begin, int64_t v_end,
                         int64_t id_offset, const int64_t* excl, int64_t ld_excl, int n_excl, float* top_scores, int64_t* top_ids, int64_t U, int d, int k, const int32_t* ulist,
                         const int32_t* ucount, void* part_ws, int S, cudaStream_t st);
