// Fused G4 steering-bank kernels (march_bank.cuh): fp32 / 8-bit frames x fp32 / fp16 / bf16 planes, and their launcher.
#include "march_bank.cuh"

namespace cvs {

cudaError_t launch_g4_bank(int fmt, const FamilyTaps& taps, const BatchGeom& g, const BankSpec& bk, cudaStream_t stream, LaunchInfo* info,
                           bool* taken)
{
    return launch_bank_fam<G4BankFam>(fmt, taps, g, bk, stream, info, taken);
}

}  // namespace cvs
