// G4/H4 fused steering kernels at a scalar angle and at theta_d with bf16 planes from 8-bit frames (G4 entries 3-4).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM(G4Fam, 3, __nv_bfloat16, unsigned char)
CVS_FORM(G4Fam, 4, __nv_bfloat16, unsigned char)
}  // namespace cvs
