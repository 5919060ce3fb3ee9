// fp16-operand build of the implicit-GEMM kernel (see the LS_HALF_FP16 note in ptx.cuh).
#ifndef LS_NO_FP16_BUILD
#define LS_HALF_FP16 1
#include "conv_gemm.cu"
#else  // development aid: a library without the fp16-operand kernels
#include "kernels.h"
namespace ls {
cudaError_t launch_conv_gemm_fp16(const CUtensorMap&, const CUtensorMap&, const CUtensorMap&, const ConvGemmParams&, int, cudaStream_t, int*) {
  return cudaErrorNotSupported;
}
}  // namespace ls
#endif
