// G2/H2 fused kernels with f16 planes from fp32 frames (every G2 entry; those without a 16-bit twin compile to no
// kernel).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM(G2Fam, 0, __half, float)
CVS_FORM(G2Fam, 1, __half, float)
CVS_FORM(G2Fam, 2, __half, float)
CVS_FORM(G2Fam, 3, __half, float)
CVS_FORM(G2Fam, 4, __half, float)
CVS_FORM(G2Fam, 5, __half, float)
CVS_FORM(G2Fam, 6, __half, float)
CVS_FORM(G2Fam, 7, __half, float)
CVS_FORM(G2Fam, 8, __half, float)
CVS_FORM(G2Fam, 9, __half, float)
CVS_FORM(G2Fam, 10, __half, float)
CVS_FORM(G2Fam, 11, __half, float)
}  // namespace cvs
