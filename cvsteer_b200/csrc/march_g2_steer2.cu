// G2/H2 fused kernels with fp32 planes: the M2 and `lines` masks steered at a scalar angle and at an angle map instead
// of theta_d (entries 8-11).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM_F32(G2Fam, 8)
CVS_FORM_F32(G2Fam, 9)
CVS_FORM_F32(G2Fam, 10)
CVS_FORM_F32(G2Fam, 11)
}  // namespace cvs
