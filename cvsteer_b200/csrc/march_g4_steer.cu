// G4/H4 fused kernels with fp32 planes: steering at one scalar angle (reference SteerableFiltersG4.cpp:114-122) and at
// this library's G4 theta_d (entries 3-4).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM_F32(G4Fam, 3)
CVS_FORM_F32(G4Fam, 4)
}  // namespace cvs
