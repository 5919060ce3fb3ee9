// fp16-operand build of the fused transformer-block kernel (see the LS_HALF_FP16 note in ptx.cuh).
#ifndef LS_NO_FP16_BUILD
#define LS_HALF_FP16 1
#include "tblock.cu"
#else  // development aid: a library without the fp16-operand kernels
#include "kernels.h"
namespace ls {
cudaError_t launch_tblock_fp16(const TBlockMaps&, const TBlockParams&, int, cudaStream_t, int*) { return cudaErrorNotSupported; }
}  // namespace ls
#endif
