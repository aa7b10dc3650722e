// G2/H2 fused kernels with fp32 planes (reference cvsteer/SteerableFiltersG2.cpp:60-177 fused): the run-time-mask
// kernel, M0, M1 and M2 (march_launch.cuh's G2 table, entries 0-3).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM_F32(G2Fam, 0)
CVS_FORM_F32(G2Fam, 1)
CVS_FORM_F32(G2Fam, 2)
CVS_FORM_F32(G2Fam, 3)
}  // namespace cvs
