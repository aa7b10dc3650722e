// Steering banks: one march of the G2/H2 basis, then the steered quantities at up to CVS_BANK_MAX_ANGLES scalar angles,
// written from registers.  The tile staging, row and column passes and loops are march_body's (march.cuh); only the
// epilogue and the output cursor differ from k_march.  Every per-angle value is computed by the same device functions, in
// the same order, as G2Fam::epilogue at a scalar angle (the `steer5@scalar` kernels), and theta_d / strength by the same
// orientation_g2<true> as the M1 kernels, so each plane is bit for bit the one those kernels store.
// Only the fast forms exist: TMA-staged tile (fp32 or 8-bit frames), baked default taps, one pixel per thread.
#pragma once
#include "march_launch.cuh"

namespace cvs {

struct BankArgs {
    int n_angles;
    unsigned mask;                         // bits of CVS_G2_BANK_PLANES
    float cos_t[CVS_BANK_MAX_ANGLES], sin_t[CVS_BANK_MAX_ANGLES];  // host-evaluated, as the single-angle calls do
    long long angle_stride;                // bytes between angle k and k + 1 of a per-angle plane
    long long out_pitch;                   // bytes
    char* out[CVS_G2_NPLANES];             // indexed by cvs_g2_plane; band origin of frame 0
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

// march_body's static key: any non-zero key without the min/max flag selects the static-mask loops; the planes themselves
// are chosen at run time (BankArgs::mask)
inline constexpr unsigned kBankKey = march_key(CVS_G2_BANK_PLANES, CVS_STEER_SCALAR);

template <typename TIn, typename TOut>
__global__ void __launch_bounds__(MARCH_TW, G2Fam::MIN_CTAS)
k_bank(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ MarchArgs a, const __grid_constant__ TapTable<G2Fam::NSETS, G2Fam::R> taps,
       const __grid_constant__ BankArgs bk)
{
    march_body<G2BankFam, kBankKey, true, TIn, true, 1, TOut, BankCursor<TOut>>(tmap, a, taps, bk);
}

}  // namespace cvs
