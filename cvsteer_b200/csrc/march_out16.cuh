// Fused 16-bit (fp16 / bf16) instantiations of the marching kernel: the same static kernels as the fp32 ones, with the
// output planes rounded to nearest even at the store (OutCursor<..., TOut>).  Only the fast form exists -- TMA-staged tile,
// baked default taps, two pixels per thread where the fp32 twin has them; march_out16.cu decides eligibility and runs
// every other launch as fp32 into scratch + k_narrow.
// TIn = unsigned char: the 8-bit-input twins.  The bytes are staged by TMA and expanded to the fp32 tile in shared memory (as
// the fp32-output `.../tma-u8` kernels do), always one pixel per thread: the expansion gives each thread two tile columns,
// which a 64-thread CTA cannot cover, and a two-pixel 8-bit form measured no faster in fp32 (DESIGN.md section 4, item 8).
// Separate translation units per family, input type, format and (G4) kernel pair so that `make -j` compiles them in parallel.
#pragma once
#include <type_traits>

#include "march_launch.cuh"

namespace cvs {

// pixels per thread of the fused 16-bit kernel for (family, mask, steering source, input type); 0 = no fused kernel (take the
// fallback).  Mirrors the static fp32 dispatch of march_g2*.cu / march_g4*.cu; 8-bit input is one pixel per thread throughout.
inline int out16_kernel_px(int family, unsigned mask, int source, bool in_u8 = false)
{
    const int PX = CVS_MARCH_PX2 > 0 && !in_u8 ? 2 : 1, PX_M1 = CVS_MARCH_PX2 > 1 && !in_u8 ? 2 : 1;
    if (family == 4) return (mask == CVS_G4_MASK_BASIS || mask == CVS_G4_MASK_STEER) ? 1 : 0;
    if (mask == CVS_G2_MASK_STATE) return 1;  // no steered plane: the source is irrelevant
    if (source == CVS_STEER_DOMINANT) return mask == CVS_G2_MASK_ORIENT ? PX_M1 : (mask == CVS_G2_MASK_FULL || mask == CVS_G2_MASK_LINES) ? PX : 0;
    if (mask == CVS_G2_MASK_FULL || mask == CVS_G2_MASK_STEER5) return PX;
    if (mask == CVS_G2_MASK_LINES) return source == CVS_STEER_SCALAR ? PX : 1;  // lines@map: one pixel, as its fp32 twin
    return 0;
}

template <typename TOut>
constexpr const char* out16_suffix() { return std::is_same_v<TOut, __half> ? "f16" : "bf16"; }

template <class Fam, unsigned MASK, int PX, typename TOut, typename TIn>
static cudaError_t launch_march16(const BatchGeom& g, const MarchArgs& a, const TapTable<Fam::NSETS, Fam::R>& tt, dim3 grid, cudaStream_t stream,
                                  LaunchInfo* info, const char* name)
{
    constexpr bool U8 = sizeof(TIn) == 1;
    static_assert(!U8 || PX == 1, "8-bit input: one pixel per thread");
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));
    if (!make_tmap(&tm, g, U8 ? (int)MARCH_U8_TW : march_tile_width(Fam::R), Fam::BH + 2 * Fam::R)) return cudaErrorInvalidValue;
    char nm[96];
    snprintf(nm, sizeof(nm), "%s/%s/imm-taps%s/%s", name, U8 ? "tma-u8" : "tma", PX == 2 ? "/2px" : "", out16_suffix<TOut>());
    return launch_march_one<Fam, MASK, true, TIn, true, PX, TOut>(tm, a, tt, grid, stream, info, nm);
}

template <typename TOut, typename TIn = float>
cudaError_t launch_march_g2_out16(const FamilyTaps& taps, const BatchGeom& g, const MarchArgs& a, cudaStream_t stream, LaunchInfo* info)
{
    TapTable<G2Fam::NSETS, G2Fam::R> tt;
    fill_tap_table<G2Fam>(taps, tt);
    const dim3 grid((g.cols + MARCH_TW - 1) / MARCH_TW, (g.out_row_end - g.out_row_begin + G2Fam::BH - 1) / G2Fam::BH, g.n);
    constexpr bool U8 = sizeof(TIn) == 1;
    constexpr int PX = CVS_MARCH_PX2 > 0 && !U8 ? 2 : 1, PX_M1 = CVS_MARCH_PX2 > 1 && !U8 ? 2 : 1;
    constexpr unsigned SC = CVS_STEER_SCALAR, MP = CVS_STEER_MAP;
    const unsigned m = a.mask;
    if (m == CVS_G2_MASK_STATE) return launch_march16<G2Fam, CVS_G2_MASK_STATE, 1, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<M0>");
    if (a.steer_source == CVS_STEER_DOMINANT) {
        if (m == CVS_G2_MASK_ORIENT) return launch_march16<G2Fam, CVS_G2_MASK_ORIENT, PX_M1, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<M1>");
        if (m == CVS_G2_MASK_FULL) return launch_march16<G2Fam, CVS_G2_MASK_FULL, PX, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<M2>");
        if (m == CVS_G2_MASK_LINES) return launch_march16<G2Fam, CVS_G2_MASK_LINES, PX, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<lines>");
    } else if (a.steer_source == CVS_STEER_SCALAR) {
        if (m == CVS_G2_MASK_FULL) return launch_march16<G2Fam, march_key(CVS_G2_MASK_FULL, SC), PX, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<M2@scalar>");
        if (m == CVS_G2_MASK_LINES)
            return launch_march16<G2Fam, march_key(CVS_G2_MASK_LINES, SC), PX, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<lines@scalar>");
        if (m == CVS_G2_MASK_STEER5)
            return launch_march16<G2Fam, march_key(CVS_G2_MASK_STEER5, SC), PX, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<steer5@scalar>");
    } else {
        if (m == CVS_G2_MASK_FULL) return launch_march16<G2Fam, march_key(CVS_G2_MASK_FULL, MP), PX, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<M2@map>");
        if (m == CVS_G2_MASK_LINES) return launch_march16<G2Fam, march_key(CVS_G2_MASK_LINES, MP), 1, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<lines@map>");
        if (m == CVS_G2_MASK_STEER5)
            return launch_march16<G2Fam, march_key(CVS_G2_MASK_STEER5, MP), PX, TOut, TIn>(g, a, tt, grid, stream, info, "g2_march<steer5@map>");
    }
    return cudaErrorInvalidValue;  // out16_kernel_px() said there is no fused kernel for this launch
}

// the steer mask at a scalar angle and at theta_d (own translation units: march_g4_out16_other_*.cu)
template <typename TOut, typename TIn = float>
cudaError_t launch_march_g4_out16_other(const BatchGeom& g, const MarchArgs& a, const TapTable<G4Fam::NSETS, G4Fam::R>& tt, dim3 grid,
                                        cudaStream_t stream, LaunchInfo* info)
{
    if (a.steer_source == CVS_STEER_SCALAR)
        return launch_march16<G4Fam, march_key(CVS_G4_MASK_STEER, CVS_STEER_SCALAR), 1, TOut, TIn>(g, a, tt, grid, stream, info, "g4_march<steer@scalar>");
    return launch_march16<G4Fam, march_key(CVS_G4_MASK_STEER, CVS_STEER_DOMINANT), 1, TOut, TIn>(g, a, tt, grid, stream, info, "g4_march<steer@theta_d>");
}

template <typename TOut, typename TIn = float>
cudaError_t launch_march_g4_out16(const FamilyTaps& taps, const BatchGeom& g, const MarchArgs& a, cudaStream_t stream, LaunchInfo* info)
{
    TapTable<G4Fam::NSETS, G4Fam::R> tt;
    fill_tap_table<G4Fam>(taps, tt);
    const dim3 grid((g.cols + MARCH_TW - 1) / MARCH_TW, (g.out_row_end - g.out_row_begin + G4Fam::BH - 1) / G4Fam::BH, g.n);
    if (a.mask == CVS_G4_MASK_BASIS) return launch_march16<G4Fam, CVS_G4_MASK_BASIS, 1, TOut, TIn>(g, a, tt, grid, stream, info, "g4_march<basis>");
    if (a.mask != CVS_G4_MASK_STEER) return cudaErrorInvalidValue;
    if (a.steer_source == CVS_STEER_MAP)
        return launch_march16<G4Fam, march_key(CVS_G4_MASK_STEER, CVS_STEER_MAP), 1, TOut, TIn>(g, a, tt, grid, stream, info, "g4_march<steer@map>");
    return launch_march_g4_out16_other<TOut, TIn>(g, a, tt, grid, stream, info);
}

// each instantiation lives in exactly one translation unit (march_g{2,4}_out16*_{f16,bf16}.cu)
#define CVS_OUT16_EXTERN(T, TIN)                                                                                                  \
    extern template cudaError_t launch_march_g2_out16<T, TIN>(const FamilyTaps&, const BatchGeom&, const MarchArgs&, cudaStream_t, LaunchInfo*); \
    extern template cudaError_t launch_march_g4_out16<T, TIN>(const FamilyTaps&, const BatchGeom&, const MarchArgs&, cudaStream_t, LaunchInfo*); \
    extern template cudaError_t launch_march_g4_out16_other<T, TIN>(const BatchGeom&, const MarchArgs&, const TapTable<G4Fam::NSETS, G4Fam::R>&, \
                                                                    dim3, cudaStream_t, LaunchInfo*);
CVS_OUT16_EXTERN(__half, float)
CVS_OUT16_EXTERN(__nv_bfloat16, float)
CVS_OUT16_EXTERN(__half, unsigned char)
CVS_OUT16_EXTERN(__nv_bfloat16, unsigned char)
#undef CVS_OUT16_EXTERN

}  // namespace cvs
