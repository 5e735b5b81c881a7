// tc_encode.cu -- the host-side lookup of cuTensorMapEncodeTiled shared by every TMA-fed kernel family.
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

}  // namespace rbm_tc
