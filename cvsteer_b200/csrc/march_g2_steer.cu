// G2/H2 fused kernels with fp32 planes: steer(theta, g2, h2, e, magnitude, phase) at a scalar angle and at an angle
// map (reference cvsteer/SteerableFiltersG2.cpp:157-177 fused with the basis stage; entries 6-7).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM_F32(G2Fam, 6)
CVS_FORM_F32(G2Fam, 7)
}  // namespace cvs
