// G4/H4 fused kernels with fp32 planes (reference cvsteer/SteerableFiltersG4.cpp:67-122 fused): the run-time-mask
// kernel, the basis and steering at an angle map (march_launch.cuh's G4 table, entries 0-2).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM_F32(G4Fam, 0)
CVS_FORM_F32(G4Fam, 1)
CVS_FORM_F32(G4Fam, 2)
}  // namespace cvs
