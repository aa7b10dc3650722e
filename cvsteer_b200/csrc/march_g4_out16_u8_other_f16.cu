// G4 fused steer kernels at a scalar angle and at theta_d with 8-bit input and f16 output planes (see march_out16.cuh).
#include "march_out16.cuh"

namespace cvs {
template cudaError_t launch_march_g4_out16_other<__half, unsigned char>(const BatchGeom&, const MarchArgs&, const TapTable<G4Fam::NSETS, G4Fam::R>&, dim3,
                                                                    cudaStream_t, LaunchInfo*);
}  // namespace cvs
