// G2/H2 fused kernels with f16 planes from 8-bit frames (every G2 entry; those without a 16-bit twin compile to no
// kernel).
#include "march_forms.cuh"

namespace cvs {
CVS_FORM(G2Fam, 0, __half, unsigned char)
CVS_FORM(G2Fam, 1, __half, unsigned char)
CVS_FORM(G2Fam, 2, __half, unsigned char)
CVS_FORM(G2Fam, 3, __half, unsigned char)
CVS_FORM(G2Fam, 4, __half, unsigned char)
CVS_FORM(G2Fam, 5, __half, unsigned char)
CVS_FORM(G2Fam, 6, __half, unsigned char)
CVS_FORM(G2Fam, 7, __half, unsigned char)
CVS_FORM(G2Fam, 8, __half, unsigned char)
CVS_FORM(G2Fam, 9, __half, unsigned char)
CVS_FORM(G2Fam, 10, __half, unsigned char)
CVS_FORM(G2Fam, 11, __half, unsigned char)
}  // namespace cvs
