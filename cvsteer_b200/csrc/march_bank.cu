// Fused G2 steering-bank kernels (march_bank.cuh): fp32 / 8-bit frames x fp32 / fp16 / bf16 planes, and their launcher.
#include "march_bank.cuh"

namespace cvs {

static_assert(sizeof(BankSpec::cos_t) / sizeof(float) == CVS_BANK_MAX_ANGLES && sizeof(BankSpec::outs) / sizeof(void*) == sizeof(BankArgs::out) / sizeof(char*),
              "BankSpec mirrors cvsteer_c.h");

cudaError_t launch_g2_bank(int fmt, const FamilyTaps& taps, const BatchGeom& g, const BankSpec& bk, cudaStream_t stream, LaunchInfo* info,
                           bool* taken)
{
    return launch_bank_fam<G2BankFam>(fmt, taps, g, bk, stream, info, taken);
}

}  // namespace cvs
