// tc_encode.cu -- the host-side lookup of cuTensorMapEncodeTiled shared by every TMA-fed kernel family, the fp32 row-tile tensor
// map of the 3xTF32 kernels (tc_gemm.cu, ce_tc.cu, and the fp32 A operand of tc_gemm16.cu) and the fp16 row-tile tensor map of
// the split-fp16 kernels (ce_wide.cu, tc_gemm16.cu).
#include "tc_ptx.cuh"

namespace rbm_tc {

EncodeTiledFn get_encode() {
  rbm_bind_context();
  static const EncodeTiledFn fn = [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      return (EncodeTiledFn)sym;
    return (EncodeTiledFn) nullptr;
  }();
  return fn;
}

bool encode_f32_rows(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows, bool mn_major) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool encode_f16_rows(CUtensorMap* map, const void* base, int64_t rows, int cols, int box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace rbm_tc
