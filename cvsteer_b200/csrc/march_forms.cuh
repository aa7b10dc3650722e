// The launcher of each fused kernel form (march_launch.cuh's table): included only by the translation units that instantiate
// it, CVS_FORM(Fam, I, TOut, TIn) once per form.
#pragma once
#include "march_launch.cuh"

namespace cvs {

template <class Fam, int I, bool TMA, typename TIn, bool BAKED, int PX, typename TOut>
static cudaError_t launch_k_march(const CUtensorMap& tm, const BatchGeom& g, const MarchArgs& a, const TapTable<Fam::NSETS, Fam::R>& tt,
                                  cudaStream_t stream, LaunchInfo* info, const char* loader)
{
    constexpr MarchForm F = MarchForms<Fam>::form[I];
    char nm[96];
    snprintf(nm, sizeof(nm), "%s<%s>/%s", MarchForms<Fam>::family, F.name, loader);
    return launch_kernel<k_march<Fam, F.key, TMA, TIn, BAKED, PX, TOut>>(march_grid<Fam>(g), MARCH_TW / PX,
                                                                         march_smem_bytes(Fam::R, Fam::BH, TMA && sizeof(TIn) == 1), stream,
                                                                         info, nm, tm, a, tt);
}

template <class Fam, int I, typename TOut, typename TIn>
cudaError_t launch_form(const BatchGeom& g, const MarchArgs& a, const TapTable<Fam::NSETS, Fam::R>& tt, int fast_px, cudaStream_t stream,
                        LaunchInfo* info)
{
    constexpr MarchForm F = MarchForms<Fam>::form[I];
    constexpr bool U8 = sizeof(TIn) == 1;
    CUtensorMap tm{};
    if constexpr (!std::is_same_v<TOut, float>) {
        if constexpr (F.out16) {
            constexpr int PX = U8 ? 1 : F.px;
            char loader[48];
            snprintf(loader, sizeof(loader), "%s/imm-taps%s/%s", U8 ? "tma-u8" : "tma", PX == 2 ? "/2px" : "",
                     std::is_same_v<TOut, __half> ? "f16" : "bf16");
            if (make_tmap<Fam>(&tm, g)) return launch_k_march<Fam, I, true, TIn, true, PX, TOut>(tm, g, a, tt, stream, info, loader);
        }
        return cudaErrorInvalidValue;
    } else {
        const bool tma = tma_eligible(g, Fam::R) && make_tmap<Fam>(&tm, g);
        if constexpr (U8) {
            if (tma) return launch_k_march<Fam, I, true, TIn, false, 1, float>(tm, g, a, tt, stream, info, "tma-u8");
            return launch_k_march<Fam, I, false, TIn, false, 1, float>(tm, g, a, tt, stream, info, "ldg-u8");
        } else {
            if (tma) {
                if constexpr (F.px == 2)
                    if (fast_px == 2) return launch_k_march<Fam, I, true, float, true, 2, float>(tm, g, a, tt, stream, info, "tma/imm-taps/2px");
                if constexpr (F.key != 0)
                    if (fast_px) return launch_k_march<Fam, I, true, float, true, 1, float>(tm, g, a, tt, stream, info, "tma/imm-taps");
                return launch_k_march<Fam, I, true, float, false, 1, float>(tm, g, a, tt, stream, info, "tma");
            }
            return launch_k_march<Fam, I, false, float, false, 1, float>(tm, g, a, tt, stream, info, "ldg");
        }
    }
}

#define CVS_FORM(Fam, I, TOut, TIn)                                                                                                   \
    template cudaError_t launch_form<Fam, I, TOut, TIn>(const BatchGeom&, const MarchArgs&, const TapTable<Fam::NSETS, Fam::R>&, int, \
                                                        cudaStream_t, LaunchInfo*);
// fp32 planes from fp32 and from 8-bit frames
#define CVS_FORM_F32(Fam, I) CVS_FORM(Fam, I, float, float) CVS_FORM(Fam, I, float, unsigned char)

}  // namespace cvs
