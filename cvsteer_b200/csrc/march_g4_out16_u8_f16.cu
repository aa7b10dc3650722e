// G4/H4 fused basis and steer@map kernels with f16 planes from 8-bit frames (G4 entries 0-2).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM(G4Fam, 0, __half, unsigned char)
CVS_FORM(G4Fam, 1, __half, unsigned char)
CVS_FORM(G4Fam, 2, __half, unsigned char)
}  // namespace cvs
