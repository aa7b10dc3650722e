// G2 fused kernels with 8-bit input and bf16 output planes (see march_out16.cuh).
#include "march_out16.cuh"

namespace cvs {
template cudaError_t launch_march_g2_out16<__nv_bfloat16, unsigned char>(const FamilyTaps&, const BatchGeom&, const MarchArgs&, cudaStream_t, LaunchInfo*);
}  // namespace cvs
