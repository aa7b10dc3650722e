// G2/H2 fused kernels with fp32 planes: edges / dark lines / bright lines at theta_d, without and with the fused
// min / max statistics (reference example/steer.cpp:73-90; entries 4-5).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM_F32(G2Fam, 4)
CVS_FORM_F32(G2Fam, 5)
}  // namespace cvs
