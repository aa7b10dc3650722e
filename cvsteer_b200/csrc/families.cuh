// Filter families for the marching kernel: which unique 1-D tap sets exist, which (row set, column set)
// pair makes each basis plane, and the fused point-wise epilogue.
//
// G2/H2 pairs: reference cvsteer/SteerableFiltersG2.cpp:62-68; G4/H4 pairs: SteerableFiltersG4.cpp:69-80.
// cv::sepFilter2D(image, dst, CV_32F, kernelX, kernelY): kernelX runs along x (the row pass), kernelY along y
// (the column pass); correlation, no flip.  g2 == h2 == exp(-x^2) in both families, so one row pass is shared.
#pragma once
#include "../../include/cvsteer_c.h"
#include "march.cuh"
#include "taps_baked.inc"

namespace cvs {

#ifndef CVS_G2_SHARED_ROW
#define CVS_G2_SHARED_ROW false
#endif
#ifndef CVS_G4_SHARED_ROW
#define CVS_G4_SHARED_ROW true
#endif
#ifndef CVS_G2_BH
#define CVS_G2_BH 64
#endif
#ifndef CVS_G2_MIN_CTAS
#define CVS_G2_MIN_CTAS 4
#endif
struct G2Fam {
    static constexpr int R = 4, NSETS = 6, NROW = 5, NBASIS = 7, NPLANES = CVS_G2_NPLANES, BH = CVS_G2_BH, MIN_CTAS = CVS_G2_MIN_CTAS;
    static constexpr bool SHARED_ROW_PASS = CVS_G2_SHARED_ROW;
    // unique tap sets: 0 g1, 1 g2(=h2), 2 g3, 3 h1, 4 h3, 5 h4   (index into TapTable::t)
    // map from the API's 7 tap sets (g1,g2,g3,h1,h2,h3,h4) to unique sets
    __host__ __device__ static constexpr int unique_of(int api) { constexpr int t[7] = {0, 1, 2, 3, 1, 4, 5}; return t[api]; }
    __host__ __device__ static constexpr bool set_odd(int s) { return s == 2 || s == 3 || s == 4; }
    // Row-filtered planes kept in the register window: g1, g2(=h2), h1, h3, h4.  There is no g3 plane: g3(x) =
    // sqrt(1.843) x exp(-x^2) is h3(x) = x exp(-x^2) times a constant, so G2b = (g3 row)(g3 col) is computed from the h3
    // row plane with the column taps pre-scaled by that constant (TapTable set 2, see fill_tap_table).  One row
    // pass and nine window registers less; the result moves by <= 1 ulp of the taps (1e-7 of range).
    __host__ __device__ static constexpr int row_set(int p) { constexpr int t[5] = {0, 1, 3, 4, 5}; return t[p]; }
    __host__ __device__ static constexpr bool row_odd(int p) { return set_odd(row_set(p)); }
    // basis planes (CVS_G2A..CVS_H2D):  row(kernelX) plane, column(kernelY) set
    //   G2a (g1,g2)  G2b (g3~h3,g3')  G2c (g2,g1)  H2a (h1,h2)  H2b (h4,h3)  H2c (h3,h4)  H2d (h2,h1)
    __host__ __device__ static constexpr int basis_row(int q) { constexpr int t[7] = {0, 3, 1, 2, 4, 3, 1}; return t[q]; }
    __host__ __device__ static constexpr int basis_set(int q) { constexpr int t[7] = {1, 2, 0, 1, 4, 5, 3}; return t[q]; }
    __host__ __device__ static constexpr bool basis_odd(int q) { return set_odd(basis_set(q)); }
    // TapTable row kScaledSet = taps of API set kScaledFromApi times the ratio (API set kScaleNumApi / API set kScaleDenApi):
    // here g3 * (g3/h3), overwriting g3's own row (plain g3 is no longer used anywhere).
    static constexpr int kScaledSet = 2, kScaledFromApi = 2, kScaleNumApi = 2, kScaleDenApi = 5;
    // reference-default taps (width 4, spacing 0.67f) as compile-time constants -> FFMA immediates
    static constexpr int kBakedWidth = CVS_BAKED_G2_WIDTH;
    __host__ __device__ static constexpr float baked(int set, int i) { constexpr float t[NSETS][R + 1] = CVS_BAKED_G2_TAPS; return t[set][i]; }

    // (no steering factors folded into the column taps for this family)
    template <unsigned MASK, bool BAKED>
    __host__ __device__ static constexpr bool prescaled() { return false; }
    __host__ __device__ static constexpr float steer_coeff(int) { return 1.f; }

    // does this launch read the per-pixel steering-angle map?
    template <unsigned MASK>
    __device__ __forceinline__ static bool reads_theta_map(const MarchArgs& a)
    {
        if (MASK) return (MASK >> MARCH_SRC_SHIFT) == CVS_STEER_MAP && (MASK & (kNeedsSteer | CVS_BIT(CVS_E)));
        return a.steer_source == CVS_STEER_MAP && (a.mask & (kNeedsSteer | CVS_BIT(CVS_E)));
    }

    static constexpr unsigned kNeedsOrient = 0x000FFF80u;   // anything beyond the 7 basis planes
    static constexpr unsigned kNeedsSteer = CVS_BIT(CVS_G2T) | CVS_BIT(CVS_H2T) | CVS_BIT(CVS_MAG) | CVS_BIT(CVS_PHASE) |
                                            CVS_BIT(CVS_EDGES) | CVS_BIT(CVS_DARK) | CVS_BIT(CVS_BRIGHT);

    // Fused epilogue on the 7 basis values of one pixel.  MASK != 0: compile-time plane set and steering source (see
    // march_key), SFU approximations for 1/x, sqrt and sin/cos (all far inside the 1e-4-of-range / 1e-3 rad parity
    // budget).  MASK == 0: run-time mask and steer source, accurate sincosf for arbitrary angles.
    // Nothing in here diverges: there is no bounds predicate (out-of-range threads are clamped onto a valid column).
    template <unsigned MASK, bool PRESCALED = false, bool PRECS = false, class Cursor>
    __device__ __forceinline__ static void epilogue(const float (&b)[NBASIS], const MarchArgs& a, const Cursor& cur, float theta_px, float = 0.f,
                                                    float = 0.f)
    {
        // The class state (M0: what setup() leaves behind and the getters return) takes the exact cv::cartToPolar sequence
        // (IEEE division and sqrt, NaNs propagate): that kernel is HBM-bound, the extra ~20 instructions are free.
        constexpr bool FAST = MASK != 0 && MASK != CVS_G2_MASK_STATE;
        const unsigned m = MASK ? (MASK & MARCH_PLANE_BITS) : a.mask;
        auto put = [&](int p, float v) { cur.put(a, p, v); };
#pragma unroll
        for (int q = 0; q < NBASIS; ++q)
            if (m & (1u << q)) put(q, b[q]);
        if (!(m & kNeedsOrient)) return;

        const int src = MASK ? (int)(MASK >> MARCH_SRC_SHIFT) : a.steer_source;
        dev::Orientation o{};
        const bool need_orient = (m & (CVS_BIT(CVS_C1) | CVS_BIT(CVS_C2) | CVS_BIT(CVS_C3) | CVS_BIT(CVS_THETA) |
                                       CVS_BIT(CVS_STRENGTH) | CVS_BIT(CVS_E))) || src == CVS_STEER_DOMINANT;
        if (need_orient) {
            o = dev::orientation_g2<FAST>(b[0], b[1], b[2], b[3], b[4], b[5], b[6]);
            if (m & CVS_BIT(CVS_C1)) put(CVS_C1, o.c1);
            if (m & CVS_BIT(CVS_C2)) put(CVS_C2, o.c2);
            if (m & CVS_BIT(CVS_C3)) put(CVS_C3, o.c3);
            if (m & CVS_BIT(CVS_THETA)) put(CVS_THETA, o.theta);
            if (m & CVS_BIT(CVS_STRENGTH)) put(CVS_STRENGTH, o.strength);
        }
        if (!(m & (kNeedsSteer | CVS_BIT(CVS_E)))) return;

        float ct, st;
        if (src == CVS_STEER_DOMINANT) {
            // E(theta_d) = c1 + c2 cos(2 theta_d) + c3 sin(2 theta_d) = c1 + strength  (G2.cpp:174-176 at theta_d)
            if (m & CVS_BIT(CVS_E)) put(CVS_E, o.c1 + o.strength);
            if (!(m & kNeedsSteer)) return;
            if (FAST) __sincosf(o.theta, &st, &ct);  // |theta_d| <= pi/2: MUFU.SIN/COS abs error < 5e-7
            else sincosf(o.theta, &st, &ct);
        } else {
            if (src == CVS_STEER_SCALAR) {
                ct = a.cos_t;
                st = a.sin_t;
            } else if (FAST) {
                __sincosf(theta_px, &st, &ct);  // MUFU works on theta / 2 pi mod 1: abs error < 3.6e-7 (+ 1.6e-7 |theta| beyond pi)
            } else {
                dev::sincos_steer(theta_px, &st, &ct);
            }
            // cos 2t = c^2 - s^2, sin 2t = 2cs  (reference: polarToCart(2*theta), G2.cpp:175)
            if (m & CVS_BIT(CVS_E)) put(CVS_E, fmaf(o.c2, fmaf(ct, ct, -st * st), fmaf(o.c3, 2.f * ct * st, o.c1)));
            if (!(m & kNeedsSteer)) return;
        }
        float g2, h2;
        dev::steer_g2(ct, st, b[0], b[1], b[2], b[3], b[4], b[5], b[6], g2, h2);
        if (m & CVS_BIT(CVS_G2T)) put(CVS_G2T, g2);
        if (m & CVS_BIT(CVS_H2T)) put(CVS_H2T, h2);
        if (m & (kNeedsSteer & ~(CVS_BIT(CVS_G2T) | CVS_BIT(CVS_H2T)))) {
            float mag, ph;
            dev::magnitude_phase<FAST>(g2, h2, mag, ph);
            if (m & CVS_BIT(CVS_MAG)) put(CVS_MAG, mag);
            if (m & CVS_BIT(CVS_PHASE)) put(CVS_PHASE, ph);
            // find*(magnitude, phase): both reference callers feed magnitude (example/steer.cpp:88-90)
            constexpr bool TRACK = (MASK & MARCH_MINMAX_FLAG) != 0;  // fused NORM_MINMAX statistics of the three maps
            if (m & CVS_BIT(CVS_EDGES)) {
                const float v = mag * dev::phase_weight<FAST>(ph, 1.57079637050628662f, false);
                put(CVS_EDGES, v);
                if (TRACK) cur.track(0, v);
            }
            if (m & CVS_BIT(CVS_DARK)) {
                const float v = mag * dev::phase_weight<FAST>(ph, 0.f, true);
                put(CVS_DARK, v);
                if (TRACK) cur.track(1, v);
            }
            if (m & CVS_BIT(CVS_BRIGHT)) {
                const float v = mag * dev::phase_weight<FAST>(ph, 3.14159274101257324f, true);
                put(CVS_BRIGHT, v);
                if (TRACK) cur.track(2, v);
            }
        }
    }
};

// 90 rows per CTA: the 12-row window fill is paid once per 102 tile rows instead of once per 76 (measured +2-3 % on every G4
// kernel), 1080 = 12 x 90 and 2160 = 24 x 90 leave no ragged last band, and three (90 + 12) x 144 fp32 tiles (176 KB) still fit
// the SM beside the three CTAs the register file allows.  108 would fit too but leaves fewer, longer CTAs per wave.
#ifndef CVS_G4_BH
#define CVS_G4_BH 90
#endif
// 3 CTAs (12 warps) per SM: the pipelined loop with its 2R-slot window needs 144-156 registers (round 1: 167 with MIN_CTAS 2)
#ifndef CVS_G4_MIN_CTAS
#define CVS_G4_MIN_CTAS 3
#endif
struct G4Fam {
    static constexpr int R = 6, NSETS = 11, NROW = 9, NBASIS = 11, NPLANES = CVS_G4_NPLANES, BH = CVS_G4_BH, MIN_CTAS = CVS_G4_MIN_CTAS;
    static constexpr bool SHARED_ROW_PASS = CVS_G4_SHARED_ROW;
    // tap table rows: 0 g1, 1 g2(=h2), 2 g3, 3 g4, 4 g5, 5 h1, 6 h3, 7 h4, 8 h5, 9 h6, 10 g3 * (g4/h4)
    // API order g1..g5,h1..h6
    __host__ __device__ static constexpr int unique_of(int api) { constexpr int t[11] = {0, 1, 2, 3, 4, 5, 1, 6, 7, 8, 9}; return t[api]; }
    __host__ __device__ static constexpr bool set_odd(int s) { return s == 2 || s == 3 || s == 5 || s == 7 || s == 8 || s == 10; }
    // Row planes in the window: g1, g2(=h2), g3, g5, h1, h3, h4, h5, h6.  No g4 plane: g4(x) = 1.246 x exp(-x^2) is h4(x)
    // times a constant, so G4d = (g4 row)(g3 col) comes from the h4 row plane with g3's column taps pre-scaled by that
    // constant (table row 10).  Plain g3 (row pass of G4b) and plain g4 (column pass of G4b) stay in rows 2 and 3.
    __host__ __device__ static constexpr int row_set(int p) { constexpr int t[9] = {0, 1, 2, 4, 5, 6, 7, 8, 9}; return t[p]; }
    __host__ __device__ static constexpr bool row_odd(int p) { return set_odd(row_set(p)); }
    //   G4a (g1,g2) G4b (g3,g4) G4c (g5,g5) G4d (g4~h4,g3') G4e (g2,g1)
    //   H4a (h1,h2) H4b (h3,h4) H4c (h5,h6) H4d (h6,h5) H4e (h4,h3) H4f (h2,h1)
    // row planes:      g1=0 g2=1 g3=2 g5=3 h1=4 h3=5 h4=6 h5=7 h6=8
    __host__ __device__ static constexpr int basis_row(int q) { constexpr int t[11] = {0, 2, 3, 6, 1, 4, 5, 7, 8, 6, 1}; return t[q]; }
    __host__ __device__ static constexpr int basis_set(int q) { constexpr int t[11] = {1, 3, 4, 10, 0, 1, 7, 9, 8, 6, 5}; return t[q]; }
    __host__ __device__ static constexpr bool basis_odd(int q) { return set_odd(basis_set(q)); }
    static constexpr int kScaledSet = 10, kScaledFromApi = 2, kScaleNumApi = 3, kScaleDenApi = 8;  // g3 * (g4/h4)
    static constexpr int kBakedWidth = CVS_BAKED_G4_WIDTH;
    __host__ __device__ static constexpr float baked(int set, int i) { constexpr float t[NSETS][R + 1] = CVS_BAKED_G4_TAPS; return t[set][i]; }

    static constexpr unsigned kNeedsSteer = CVS_G4_MASK_STEER;
    static constexpr unsigned kNeedsOrient = CVS_BIT(CVS_G4_THETA) | CVS_BIT(CVS_G4_STRENGTH);

    // C1, C2, C3 of E(theta) = G4(theta)^2 + H4(theta)^2 as quadratic forms of the 11 basis values (coefficients generated
    // by gen_baked_taps.cpp; zero entries vanish at compile time), then theta_d / strength exactly as the G2 class does.
    template <bool FAST>
    __device__ __forceinline__ static dev::Orientation orientation(const float (&b)[NBASIS])
    {
        constexpr float Q[3][36] = CVS_G4_ORIENT_FORMS;
        float c[3] = {0.f, 0.f, 0.f};
        int e = 0;
#pragma unroll
        for (int blk = 0; blk < 2; ++blk) {
            const int n = blk == 0 ? 5 : 6, o = blk == 0 ? 0 : 5;
#pragma unroll
            for (int i = 0; i < n; ++i)
#pragma unroll
                for (int j = i; j < n; ++j, ++e) {
                    const float p = b[o + i] * b[o + j];
#pragma unroll
                    for (int k = 0; k < 3; ++k)
                        if (Q[k][e] != 0.f) c[k] = fmaf(Q[k][e], p, c[k]);
                }
        }
        dev::Orientation r;
        r.c1 = c[0], r.c2 = c[1], r.c3 = c[2];
        r.strength = dev::cv_magnitude<FAST>(c[1], c[2]);
        if (FAST) r.theta = dev::cv_atan2_wrapped_fast<true>(c[2], c[1]);
        else r.theta = 0.5f * dev::wrap_pi(dev::cv_atan2<false, true>(c[2], c[1]));
        return r;
    }
    // Steer-only static kernels with baked taps fold the binomial steering factors into the column taps at compile time
    // (every basis value arrives pre-multiplied: G4 1 -4 6 -4 1, H4 1 -5 10 -10 5 -1), which shortens the epilogue by 8
    // instructions; the scaled tap is rounded once (<= 1 ulp of the tap: 6e-8 relative).  Not when basis planes or the
    // orientation forms are wanted as well -- those need the plain values.
    template <unsigned MASK, bool BAKED>
    __host__ __device__ static constexpr bool prescaled()
    {
        return BAKED && MASK != 0 && ((MASK & MARCH_PLANE_BITS) & (CVS_G4_MASK_BASIS | kNeedsOrient)) == 0 &&
               (MASK >> MARCH_SRC_SHIFT) != CVS_STEER_DOMINANT;
    }
    __host__ __device__ static constexpr float steer_coeff(int q) { constexpr float t[11] = {1.f, -4.f, 6.f, -4.f, 1.f, 1.f, -5.f, 10.f, -10.f, 5.f, -1.f}; return t[q]; }

    template <unsigned MASK>
    __device__ __forceinline__ static bool reads_theta_map(const MarchArgs& a)
    {
        if (MASK) return (MASK >> MARCH_SRC_SHIFT) == CVS_STEER_MAP && (MASK & kNeedsSteer) != 0;
        return a.steer_source == CVS_STEER_MAP && (a.mask & kNeedsSteer);
    }

    // MASK != 0: compile-time plane set and steering source (march_key; config 4 = steer mask at a per-pixel angle map),
    // SFU approximations.  MASK == 0: run-time mask; steering at a scalar angle, an angle map, or the in-kernel dominant angle.
    // PRECS: cos / sin of this pixel's steering angle were computed by the caller one row ahead (ct_pre, st_pre), which takes
    // the angle load and the MUFU latency off the head of the epilogue's dependent chain.
    template <unsigned MASK, bool PRESCALED = false, bool PRECS = false, class Cursor>
    __device__ __forceinline__ static void epilogue(const float (&b)[NBASIS], const MarchArgs& a, const Cursor& cur, float theta_px,
                                                    float ct_pre = 0.f, float st_pre = 0.f)
    {
        constexpr bool FAST = MASK != 0;
        const unsigned m = MASK ? (MASK & MARCH_PLANE_BITS) : a.mask;
        const int src = MASK ? (int)(MASK >> MARCH_SRC_SHIFT) : a.steer_source;
        auto put = [&](int p, float v) { cur.put(a, p, v); };
#pragma unroll
        for (int q = 0; q < NBASIS; ++q)
            if (m & (1u << q)) put(q, b[q]);
        if (!(m & (kNeedsSteer | kNeedsOrient))) return;
        const bool dominant = src == CVS_STEER_DOMINANT;
        if ((m & kNeedsOrient) || (dominant && (m & kNeedsSteer))) {
            const dev::Orientation o = orientation<FAST>(b);
            if (m & CVS_BIT(CVS_G4_THETA)) put(CVS_G4_THETA, o.theta);
            if (m & CVS_BIT(CVS_G4_STRENGTH)) put(CVS_G4_STRENGTH, o.strength);
            if (dominant) theta_px = o.theta;
        }
        if (!(m & kNeedsSteer)) return;
        float ct, st;
        if (src == CVS_STEER_SCALAR) {
            ct = a.cos_t;
            st = a.sin_t;
        } else if (PRECS && !dominant) {
            ct = ct_pre;
            st = st_pre;
        } else if (FAST) {
            // MUFU.SIN/COS work on theta / 2 pi modulo 1: no range branch, abs error < 3.6e-7 for |theta| <= pi and up to
            // 1.6e-7 * |theta| more beyond (theta * float(1 / 2 pi) rounds toward zero: < 2u, plus the constant's 0.68u)
            __sincosf(theta_px, &st, &ct);
        } else {
            dev::sincos_steer(theta_px, &st, &ct);
        }
        float g4, h4;
        if (PRESCALED) dev::steer_g4_prescaled(ct, st, &b[0], &b[5], g4, h4);
        else dev::steer_g4(ct, st, &b[0], &b[5], g4, h4);
        if (m & CVS_BIT(CVS_G4T)) put(CVS_G4T, g4);
        if (m & CVS_BIT(CVS_H4T)) put(CVS_H4T, h4);
        if (m & (CVS_BIT(CVS_MAG4) | CVS_BIT(CVS_PHASE4))) {
            float mag, ph;
            dev::magnitude_phase<FAST>(g4, h4, mag, ph);
            if (m & CVS_BIT(CVS_MAG4)) put(CVS_MAG4, mag);
            if (m & CVS_BIT(CVS_PHASE4)) put(CVS_PHASE4, ph);
        }
    }
};

}  // namespace cvs
