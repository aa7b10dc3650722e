// Fused steering-bank kernels (march_bank.cuh): fp32 / 8-bit frames x fp32 / fp16 / bf16 planes, and their launcher.
#include <type_traits>

#include "march_bank.cuh"

namespace cvs {

static_assert(sizeof(BankSpec::cos_t) / sizeof(float) == CVS_BANK_MAX_ANGLES && sizeof(BankSpec::outs) / sizeof(void*) == CVS_G2_NPLANES,
              "BankSpec mirrors cvsteer_c.h");

template <typename TIn, typename TOut>
static cudaError_t launch_bank_one(const BatchGeom& g, const MarchArgs& a, const TapTable<G2Fam::NSETS, G2Fam::R>& tt, const BankArgs& bk,
                                   cudaStream_t stream, LaunchInfo* info)
{
    constexpr bool U8 = sizeof(TIn) == 1;
    constexpr int smem = march_smem_bytes(G2Fam::R, G2Fam::BH, U8);
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));
    if (!make_tmap(&tm, g, U8 ? (int)MARCH_U8_TW : march_tile_width(G2Fam::R), G2Fam::BH + 2 * G2Fam::R)) return cudaErrorInvalidValue;
    auto kfn = k_bank<TIn, TOut>;
    static std::atomic<unsigned long long> done[4];  // per device, as launch_march_one
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev); e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    std::atomic<unsigned long long>& word = done[(dev >> 6) & 3];
    if (!(word.load(std::memory_order_acquire) & bit)) {
        cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kfn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        word.fetch_or(bit, std::memory_order_release);
    }
    const dim3 grid((g.cols + MARCH_TW - 1) / MARCH_TW, (g.out_row_end - g.out_row_begin + G2Fam::BH - 1) / G2Fam::BH, g.n);
    kfn<<<grid, MARCH_TW, smem, stream>>>(tm, a, tt, bk);
    g_launches.fetch_add(1);
    if (info) {
        info->grid[0] = grid.x, info->grid[1] = grid.y, info->grid[2] = grid.z;
        info->block = MARCH_TW;
        info->smem = smem;
        const char* fmt = std::is_same_v<TOut, float> ? "" : std::is_same_v<TOut, __half> ? "/f16" : "/bf16";
        snprintf(info->name, sizeof(info->name), "g2_bank/%s/imm-taps%s", U8 ? "tma-u8" : "tma", fmt);
    }
    return cudaGetLastError();
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
    MarchArgs a = make_args(g, 0u, st, nullptr, 0);
    BankArgs ba;
    memset(&ba, 0, sizeof(ba));
    ba.n_angles = bk.n_angles;
    ba.mask = bk.mask;
    for (int j = 0; j < bk.n_angles; ++j) ba.cos_t[j] = bk.cos_t[j], ba.sin_t[j] = bk.sin_t[j];
    ba.angle_stride = (long long)bk.angle_stride;
    ba.out_pitch = (long long)g.out_pitch;
    // gridDim.z carries the frame index: batches beyond 65535 frames go out as several launches (as launch_basis_fused)
    for (int f0 = 0; f0 < g.n; f0 += 65535) {
        BatchGeom gc = g;
        MarchArgs ac = a;
        BankArgs bc = ba;
        gc.n = g.n - f0 < 65535 ? g.n - f0 : 65535;
        gc.in = static_cast<const char*>(g.in) + (size_t)f0 * g.in_frame_stride;
        ac.in = gc.in;
        for (int q = 0; q < CVS_G2_NPLANES; ++q)
            if (bk.mask >> q & 1u) bc.out[q] = static_cast<char*>(bk.outs[q]) + (size_t)f0 * g.out_frame_stride;
        if (ac.pyr_out) ac.pyr_out = reinterpret_cast<float*>(reinterpret_cast<char*>(a.pyr_out) + (size_t)f0 * g.next_frame_stride);
        cudaError_t e;
        if (g.in_u8)
            e = fmt == CVS_OUT_F32  ? launch_bank_one<unsigned char, float>(gc, ac, tt, bc, stream, info)
                : fmt == CVS_OUT_F16 ? launch_bank_one<unsigned char, __half>(gc, ac, tt, bc, stream, info)
                                     : launch_bank_one<unsigned char, __nv_bfloat16>(gc, ac, tt, bc, stream, info);
        else
            e = fmt == CVS_OUT_F32  ? launch_bank_one<float, float>(gc, ac, tt, bc, stream, info)
                : fmt == CVS_OUT_F16 ? launch_bank_one<float, __half>(gc, ac, tt, bc, stream, info)
                                     : launch_bank_one<float, __nv_bfloat16>(gc, ac, tt, bc, stream, info);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

}  // namespace cvs
