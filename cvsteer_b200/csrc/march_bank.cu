// Fused steering-bank kernels (march_bank.cuh): fp32 / 8-bit frames x fp32 / fp16 / bf16 planes, and their launcher.
#include <type_traits>

#include "march_bank.cuh"

namespace cvs {

static_assert(sizeof(BankSpec::cos_t) / sizeof(float) == CVS_BANK_MAX_ANGLES && sizeof(BankSpec::outs) / sizeof(void*) == CVS_G2_NPLANES,
              "BankSpec mirrors cvsteer_c.h");

template <typename TIn, typename TOut>
static cudaError_t launch_bank(const BatchGeom& g, const MarchArgs& a, const TapTable<G2Fam::NSETS, G2Fam::R>& tt, const BankArgs& bk,
                               cudaStream_t stream, LaunchInfo* info)
{
    constexpr bool U8 = sizeof(TIn) == 1;
    CUtensorMap tm{};
    if (!make_tmap<G2Fam>(&tm, g)) return cudaErrorInvalidValue;
    char nm[96];
    snprintf(nm, sizeof(nm), "g2_bank/%s/imm-taps%s", U8 ? "tma-u8" : "tma",
             std::is_same_v<TOut, float> ? "" : std::is_same_v<TOut, __half> ? "/f16" : "/bf16");
    return launch_kernel<k_bank<TIn, TOut>>(march_grid<G2Fam>(g), MARCH_TW, march_smem_bytes(G2Fam::R, G2Fam::BH, U8), stream, info, nm, tm, a,
                                            tt, bk);
}

cudaError_t launch_g2_bank(int fmt, const FamilyTaps& taps, const BatchGeom& g, const BankSpec& bk, cudaStream_t stream, LaunchInfo* info,
                           bool* taken)
{
    *taken = false;
    if (!uses_march_path(2, taps.width) || !tma_eligible(g, G2Fam::R)) return cudaSuccess;
    TapTable<G2Fam::NSETS, G2Fam::R> tt;
    fill_tap_table<G2Fam>(taps, tt);
    if (!taps_are_baked<G2Fam>(tt)) return cudaSuccess;
    // one-pixel stores: every plane, the pitch and both strides multiples of the element size
    const size_t esz = fmt == CVS_OUT_F32 ? 4 : 2;
    if ((g.out_pitch | g.out_frame_stride | bk.angle_stride) & (esz - 1)) return cudaSuccess;
    for (int q = 0; q < CVS_G2_NPLANES; ++q)
        if ((bk.mask >> q & 1u) && ((uintptr_t)bk.outs[q] & (esz - 1))) return cudaSuccess;
    if (g.out_row_end <= g.out_row_begin || g.cols <= 0 || g.n <= 0) return cudaErrorInvalidValue;
    *taken = true;
    SteerSpec st{};
    st.source = CVS_STEER_SCALAR;
    const MarchArgs a = make_args(g, 0u, st, nullptr, 0);
    BankArgs ba;
    memset(&ba, 0, sizeof(ba));
    ba.n_angles = bk.n_angles;
    ba.mask = bk.mask;
    for (int j = 0; j < bk.n_angles; ++j) ba.cos_t[j] = bk.cos_t[j], ba.sin_t[j] = bk.sin_t[j];
    ba.angle_stride = (long long)bk.angle_stride;
    ba.out_pitch = (long long)g.out_pitch;
    return for_each_frame_chunk(g, a, esz, [&](const BatchGeom& gc, const MarchArgs& ac, size_t out_off) {
        BankArgs bc = ba;
        for (int q = 0; q < CVS_G2_NPLANES; ++q)
            if (bk.mask >> q & 1u) bc.out[q] = static_cast<char*>(bk.outs[q]) + out_off;
        if (g.in_u8)
            return fmt == CVS_OUT_F32  ? launch_bank<unsigned char, float>(gc, ac, tt, bc, stream, info)
                   : fmt == CVS_OUT_F16 ? launch_bank<unsigned char, __half>(gc, ac, tt, bc, stream, info)
                                        : launch_bank<unsigned char, __nv_bfloat16>(gc, ac, tt, bc, stream, info);
        return fmt == CVS_OUT_F32  ? launch_bank<float, float>(gc, ac, tt, bc, stream, info)
               : fmt == CVS_OUT_F16 ? launch_bank<float, __half>(gc, ac, tt, bc, stream, info)
                                    : launch_bank<float, __nv_bfloat16>(gc, ac, tt, bc, stream, info);
    });
}

}  // namespace cvs
