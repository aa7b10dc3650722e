// Steering banks: one march of a family's basis, then the steered quantities at up to CVS_BANK_MAX_ANGLES scalar angles,
// written from registers.  The tile staging, row and column passes and loops are march_body's (march.cuh); only the
// epilogue and the output cursor differ from k_march.  Every per-angle value is computed by the same device functions, in
// the same order, as the family's epilogue at a scalar angle (the `steer5@scalar` / `steer@scalar` kernels), and G2's
// theta_d / strength by the same orientation_g2<true> as the M1 kernels, so each plane is bit for bit the one those kernels
// store.
// Only the fast forms exist: TMA-staged tile (fp32 or 8-bit frames), baked default taps, one pixel per thread.
#pragma once
#include <type_traits>

#include "march_launch.cuh"

namespace cvs {

struct BankArgs {
    int n_angles;
    unsigned mask;                         // bits of CVS_G2_BANK_PLANES / CVS_G4_BANK_PLANES
    float cos_t[CVS_BANK_MAX_ANGLES], sin_t[CVS_BANK_MAX_ANGLES];  // host-evaluated, as the single-angle calls do
    long long angle_stride;                // bytes between angle k and k + 1 of a per-angle plane
    long long out_pitch;                   // bytes
    char* out[(int)CVS_G2_NPLANES > (int)CVS_G4_NPLANES ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES];  // indexed by the family's plane enum; band origin of frame 0
};

// Where this thread's pixel of the current row lives: one byte offset shared by every plane and angle.
template <typename TOut>
struct BankCursor {
    const BankArgs& k;
    long long off;
    __device__ __forceinline__ BankCursor(const BankArgs& bk, long long band_off, int x) : k(bk), off(band_off + (long long)sizeof(TOut) * x) {}
    __device__ __forceinline__ void put(int q, long long angle_off, float v) const
    {
        char* p = k.out[q] + angle_off + off;
        if constexpr (sizeof(TOut) == 4) __stcs(reinterpret_cast<float*>(p), v);
        else __stcs(reinterpret_cast<unsigned short*>(p), to_out16<TOut>(v));
    }
    // (march_body asks for a steering-angle map only when the family reads one; the bank never does)
    __device__ __forceinline__ float theta(const MarchArgs&, int = 0) const { return 0.f; }
    __device__ __forceinline__ void next_row() { off += k.out_pitch; }
};

struct G2BankFam : G2Fam {
    static constexpr int family = 2;
    static constexpr const char* name = "g2_bank";
    static constexpr unsigned kKey = march_key(CVS_G2_BANK_PLANES, CVS_STEER_SCALAR);

    template <unsigned MASK>
    __device__ __forceinline__ static bool reads_theta_map(const MarchArgs&) { return false; }

    template <unsigned MASK, bool PRESCALED = false, bool PRECS = false, class Cursor>
    __device__ __forceinline__ static void epilogue(const float (&b)[NBASIS], const MarchArgs&, const Cursor& cur, float, float = 0.f,
                                                    float = 0.f)
    {
        const BankArgs& k = cur.k;
        const unsigned m = k.mask;
        const dev::Orientation o = dev::orientation_g2<true>(b[0], b[1], b[2], b[3], b[4], b[5], b[6]);
        if (m & CVS_BIT(CVS_THETA)) cur.put(CVS_THETA, 0, o.theta);
        if (m & CVS_BIT(CVS_STRENGTH)) cur.put(CVS_STRENGTH, 0, o.strength);
        // rolled: the body stays small enough for the instruction cache whatever the number of angles (DESIGN.md section 9)
        long long ao = 0;
#pragma unroll 1
        for (int j = 0; j < k.n_angles; ++j, ao += k.angle_stride) {
            const float ct = k.cos_t[j], st = k.sin_t[j];
            // G2Fam::epilogue at CVS_STEER_SCALAR, expression for expression
            if (m & CVS_BIT(CVS_E)) cur.put(CVS_E, ao, fmaf(o.c2, fmaf(ct, ct, -st * st), fmaf(o.c3, 2.f * ct * st, o.c1)));
            if (!(m & (CVS_BIT(CVS_G2T) | CVS_BIT(CVS_H2T) | CVS_BIT(CVS_MAG) | CVS_BIT(CVS_PHASE)))) continue;
            float g2, h2;
            dev::steer_g2(ct, st, b[0], b[1], b[2], b[3], b[4], b[5], b[6], g2, h2);
            if (m & CVS_BIT(CVS_G2T)) cur.put(CVS_G2T, ao, g2);
            if (m & CVS_BIT(CVS_H2T)) cur.put(CVS_H2T, ao, h2);
            if (m & (CVS_BIT(CVS_MAG) | CVS_BIT(CVS_PHASE))) {
                float mag, ph;
                dev::magnitude_phase<true>(g2, h2, mag, ph);
                if (m & CVS_BIT(CVS_MAG)) cur.put(CVS_MAG, ao, mag);
                if (m & CVS_BIT(CVS_PHASE)) cur.put(CVS_PHASE, ao, ph);
            }
        }
    }
};

// G4: the steer@scalar epilogue per angle.  The bank's static key is steer@scalar's, so march_body folds the binomial
// steering factors into the baked column taps exactly as it does there (G4Fam::prescaled), and the basis values arrive
// pre-multiplied -- which is why the bank has no theta_d / strength: G4Fam::orientation needs the plain values.
struct G4BankFam : G4Fam {
    static constexpr int family = 4;
    static constexpr const char* name = "g4_bank";
    static constexpr unsigned kKey = march_key(CVS_G4_MASK_STEER, CVS_STEER_SCALAR);

    template <unsigned MASK>
    __device__ __forceinline__ static bool reads_theta_map(const MarchArgs&) { return false; }

    // (PRECS / ct_pre / st_pre: the pipelined loop's cos / sin of a map angle, never computed for a scalar key; ignored)
    template <unsigned MASK, bool PRESCALED = false, bool PRECS = false, class Cursor>
    __device__ __forceinline__ static void epilogue(const float (&b)[NBASIS], const MarchArgs&, const Cursor& cur, float, float = 0.f,
                                                    float = 0.f)
    {
        static_assert(PRESCALED, "the G4 bank steers prescaled basis values, as steer@scalar does");
        const BankArgs& k = cur.k;
        const unsigned m = k.mask;
        // rolled, as in G2BankFam: the pipelined loop runs the epilogue once per row, outside its slot dispatch, so the loop
        // adds its code once
        long long ao = 0;
#pragma unroll 1
        for (int j = 0; j < k.n_angles; ++j, ao += k.angle_stride) {
            const float ct = k.cos_t[j], st = k.sin_t[j];
            // G4Fam::epilogue at CVS_STEER_SCALAR with PRESCALED and FAST, expression for expression
            float g4, h4;
            dev::steer_g4_prescaled(ct, st, &b[0], &b[5], g4, h4);
            if (m & CVS_BIT(CVS_G4T)) cur.put(CVS_G4T, ao, g4);
            if (m & CVS_BIT(CVS_H4T)) cur.put(CVS_H4T, ao, h4);
            if (m & (CVS_BIT(CVS_MAG4) | CVS_BIT(CVS_PHASE4))) {
                float mag, ph;
                dev::magnitude_phase<true>(g4, h4, mag, ph);
                if (m & CVS_BIT(CVS_MAG4)) cur.put(CVS_MAG4, ao, mag);
                if (m & CVS_BIT(CVS_PHASE4)) cur.put(CVS_PHASE4, ao, ph);
            }
        }
    }
};

// BFam::kKey is march_body's static key: any non-zero key without the min/max flag selects the static-mask loops; the planes
// themselves are chosen at run time (BankArgs::mask).  For G4 the key also decides the prescaled column taps.
template <class BFam, typename TIn, typename TOut>
__global__ void __launch_bounds__(MARCH_TW, BFam::MIN_CTAS)
k_bank(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ MarchArgs a, const __grid_constant__ TapTable<BFam::NSETS, BFam::R> taps,
       const __grid_constant__ BankArgs bk)
{
    march_body<BFam, BFam::kKey, true, TIn, true, 1, TOut, BankCursor<TOut>>(tmap, a, taps, bk);
}

template <class BFam, typename TIn, typename TOut>
static cudaError_t launch_bank(const BatchGeom& g, const MarchArgs& a, const TapTable<BFam::NSETS, BFam::R>& tt, const BankArgs& bk,
                               cudaStream_t stream, LaunchInfo* info)
{
    constexpr bool U8 = sizeof(TIn) == 1;
    CUtensorMap tm{};
    if (!make_tmap<BFam>(&tm, g)) return cudaErrorInvalidValue;
    char nm[96];
    snprintf(nm, sizeof(nm), "%s/%s/imm-taps%s", BFam::name, U8 ? "tma-u8" : "tma",
             std::is_same_v<TOut, float> ? "" : std::is_same_v<TOut, __half> ? "/f16" : "/bf16");
    return launch_kernel<k_bank<BFam, TIn, TOut>>(march_grid<BFam>(g), MARCH_TW, march_smem_bytes(BFam::R, BFam::BH, U8), stream, info, nm, tm,
                                                  a, tt, bk);
}

// The fused bank of family BFam when its forms apply (default width and taps, TMA-eligible frames, planes, pitch and strides
// multiples of the element size); otherwise nothing is launched and *taken stays false.  Each family's kernels are
// instantiated in its own translation unit (march_bank.cu, march_bank_g4.cu).
template <class BFam>
static cudaError_t launch_bank_fam(int fmt, const FamilyTaps& taps, const BatchGeom& g, const BankSpec& bk, cudaStream_t stream, LaunchInfo* info,
                                   bool* taken)
{
    *taken = false;
    if (!uses_march_path(BFam::family, taps.width) || !tma_eligible(g, BFam::R)) return cudaSuccess;
    TapTable<BFam::NSETS, BFam::R> tt;
    fill_tap_table<BFam>(taps, tt);
    if (!taps_are_baked<BFam>(tt)) return cudaSuccess;
    // one-pixel stores: every plane, the pitch and both strides multiples of the element size
    const size_t esz = fmt == CVS_OUT_F32 ? 4 : 2;
    if ((g.out_pitch | g.out_frame_stride | bk.angle_stride) & (esz - 1)) return cudaSuccess;
    for (int q = 0; q < BFam::NPLANES; ++q)
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
        for (int q = 0; q < BFam::NPLANES; ++q)
            if (bk.mask >> q & 1u) bc.out[q] = static_cast<char*>(bk.outs[q]) + out_off;
        if (g.in_u8)
            return fmt == CVS_OUT_F32  ? launch_bank<BFam, unsigned char, float>(gc, ac, tt, bc, stream, info)
                   : fmt == CVS_OUT_F16 ? launch_bank<BFam, unsigned char, __half>(gc, ac, tt, bc, stream, info)
                                        : launch_bank<BFam, unsigned char, __nv_bfloat16>(gc, ac, tt, bc, stream, info);
        return fmt == CVS_OUT_F32  ? launch_bank<BFam, float, float>(gc, ac, tt, bc, stream, info)
               : fmt == CVS_OUT_F16 ? launch_bank<BFam, float, __half>(gc, ac, tt, bc, stream, info)
                                    : launch_bank<BFam, float, __nv_bfloat16>(gc, ac, tt, bc, stream, info);
    });
}

}  // namespace cvs
