// G4 fused basis and steer@map kernels with 8-bit input and f16 output planes (see march_out16.cuh).
#include "march_out16.cuh"

namespace cvs {
template cudaError_t launch_march_g4_out16<__half, unsigned char>(const FamilyTaps&, const BatchGeom&, const MarchArgs&, cudaStream_t, LaunchInfo*);
}  // namespace cvs
