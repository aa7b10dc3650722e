// Host-side launch helpers for the marching kernel (tensor-map creation, variant selection).
// Included by march_g2.cu / march_g4.cu (one translation unit per family so they compile in parallel).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "families.cuh"
#include "launch.h"

namespace cvs {

extern std::atomic<unsigned long long> g_launches;

// ------------------------------------------------------------------------------------------------
// TMA tensor map (driver entry point fetched through the runtime: no link-time libcuda dependency)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline PFN_encodeTiled get_encode_fn()
{
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    });
    return fn;
}

// 3-D fp32 (or 8-bit) tensor (x = cols, y = buffer rows, z = frames); box = (box_w, box_h, 1) elements; OOB -> zeros.
static inline bool make_tmap(CUtensorMap* m, const BatchGeom& g, int box_w, int box_h)
{
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return false;
    cuuint64_t dims[3] = {(cuuint64_t)g.cols, (cuuint64_t)g.buf_rows, (cuuint64_t)g.n};
    cuuint64_t strides[2] = {(cuuint64_t)g.in_pitch, (cuuint64_t)(g.n > 1 ? g.in_frame_stride : g.in_pitch * (size_t)g.buf_rows)};
    cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, g.in_u8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(g.in), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

static inline bool tma_eligible(const BatchGeom& g, int R)
{
    static const bool force_ldg = getenv("CVS_FORCE_LDG") != nullptr;  // A/B switch for profiling the two loaders
    if (force_ldg) return false;
    if (((uintptr_t)g.in & 15) || (g.in_pitch & 15) || (g.in_frame_stride & 15)) return false;
    if (g.cols < R + 1 || g.full_rows < R + 1) return false;  // one reflect fold must land inside the tile
    if (g.n > 1 && g.in_frame_stride < g.in_pitch * (size_t)g.buf_rows) return false;
    return true;
}

// ------------------------------------------------------------------------------------------------
// Marching-kernel dispatch
// ------------------------------------------------------------------------------------------------
template <class Fam>
static void fill_tap_table(const FamilyTaps& ft, TapTable<Fam::NSETS, Fam::R>& tt)
{
    for (int api = 0; api < ft.nsets; ++api) {
        const int u = Fam::unique_of(api);
        for (int i = 0; i <= Fam::R; ++i) tt.t[u][i] = ft.t[api][Fam::R + i];
    }
    float scaled[MAX_TAPS];
    scale_taps_by_ratio(ft.t[Fam::kScaledFromApi], ft.t[Fam::kScaleNumApi], ft.t[Fam::kScaleDenApi], 2 * Fam::R + 1, scaled);
    for (int i = 0; i <= Fam::R; ++i) tt.t[Fam::kScaledSet][i] = scaled[Fam::R + i];
}

template <class Fam, unsigned MASK, bool TMA, typename TIn, bool BAKED, int PX = 1, typename TOut = float>
static cudaError_t launch_march_one(const CUtensorMap& tm, const MarchArgs& a, const TapTable<Fam::NSETS, Fam::R>& tt, dim3 grid,
                                    cudaStream_t stream, LaunchInfo* info, const char* name)
{
    constexpr int smem = march_smem_bytes(Fam::R, Fam::BH, TMA && sizeof(TIn) == 1);
    auto kfn = k_march<Fam, MASK, TMA, TIn, BAKED, PX, TOut>;
    // Function attributes are per DEVICE (context): one flag per (instantiation, device).  The 8-bit TMA variants ask for
    // more than the 48 KB default, so a process that drives several GPUs must set them on each one.
    static std::atomic<unsigned long long> done[4];  // 256 devices
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev); e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    std::atomic<unsigned long long>& word = done[(dev >> 6) & 3];
    if (!(word.load(std::memory_order_acquire) & bit)) {
        cudaError_t e = cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kfn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        word.fetch_or(bit, std::memory_order_release);  // idempotent: a racing thread at worst sets the attributes twice
    }
    kfn<<<grid, MARCH_TW / PX, smem, stream>>>(tm, a, tt);
    g_launches.fetch_add(1);
    if (info) {
        info->grid[0] = grid.x, info->grid[1] = grid.y, info->grid[2] = grid.z;
        info->block = MARCH_TW / PX;
        info->smem = smem;
        snprintf(info->name, sizeof(info->name), "%s", name);
    }
    return cudaGetLastError();
}

// true when the handle's taps are bit-identical to the baked reference defaults of the family
template <class Fam>
static bool taps_are_baked(const TapTable<Fam::NSETS, Fam::R>& tt)
{
    static const bool disabled = getenv("CVS_NO_BAKED") != nullptr;  // A/B switch: constant-bank taps everywhere
    if (disabled) return false;
    for (int s = 0; s < Fam::NSETS; ++s)
        for (int i = 0; i <= Fam::R; ++i) {
            const float bk = Fam::baked(s, i);
            if (memcmp(&bk, &tt.t[s][i], sizeof(float)) != 0) return false;
        }
    return true;
}

// BAKED_OK: whether a baked-tap instantiation exists for this mask (kept to the hot static-mask variants to bound
// compile time and binary size).
// Two-pixel threads store 8 bytes per plane: every selected plane, the pitch and the frame stride must be multiples of 8
// and the width even (the clamped last pair stays aligned).
static inline bool pair_store_ok(const BatchGeom& g, const MarchArgs& a)
{
    static const bool disabled = getenv("CVS_PX1") != nullptr;  // A/B switch: one pixel per thread everywhere
    if (disabled || (g.cols & 1) || (g.out_pitch & 7) || (g.out_frame_stride & 7)) return false;
    for (int p = 0; p < MARCH_MAX_OUT; ++p)
        if (a.out[p] && ((uintptr_t)a.out[p] & 7)) return false;
    if (a.steer_source == CVS_STEER_MAP && ((uintptr_t)a.theta_map & 7)) return false;  // angle pairs are 8-byte loads as well
    return true;
}

// PX2_OK: whether a two-pixels-per-thread instantiation exists for this mask (issue-bound static masks only).
template <class Fam, unsigned MASK, bool BAKED_OK = false, bool PX2_OK = false>
static cudaError_t launch_march_mask(const BatchGeom& g, const MarchArgs& a, const TapTable<Fam::NSETS, Fam::R>& tt, dim3 grid,
                                     cudaStream_t stream, LaunchInfo* info, const char* name)
{
    CUtensorMap tm;
    memset(&tm, 0, sizeof(tm));
    constexpr int TROWS = Fam::BH + 2 * Fam::R, TWH = march_tile_width(Fam::R);
    char nm[96];
    if (g.in_u8 && tma_eligible(g, Fam::R) && make_tmap(&tm, g, MARCH_U8_TW, TROWS)) {
        snprintf(nm, sizeof(nm), "%s/tma-u8", name);
        return launch_march_one<Fam, MASK, true, unsigned char, false>(tm, a, tt, grid, stream, info, nm);
    }
    if (!g.in_u8 && tma_eligible(g, Fam::R) && make_tmap(&tm, g, TWH, TROWS)) {
        if constexpr (BAKED_OK) {
            if (taps_are_baked<Fam>(tt)) {
                if constexpr (PX2_OK) {
                    if (pair_store_ok(g, a)) {
                        snprintf(nm, sizeof(nm), "%s/tma/imm-taps/2px", name);
                        return launch_march_one<Fam, MASK, true, float, true, 2>(tm, a, tt, grid, stream, info, nm);
                    }
                }
                snprintf(nm, sizeof(nm), "%s/tma/imm-taps", name);
                return launch_march_one<Fam, MASK, true, float, true>(tm, a, tt, grid, stream, info, nm);
            }
        }
        snprintf(nm, sizeof(nm), "%s/tma", name);
        return launch_march_one<Fam, MASK, true, float, false>(tm, a, tt, grid, stream, info, nm);
    }
    if (g.in_u8) {
        snprintf(nm, sizeof(nm), "%s/ldg-u8", name);
        return launch_march_one<Fam, MASK, false, unsigned char, false>(tm, a, tt, grid, stream, info, nm);
    }
    snprintf(nm, sizeof(nm), "%s/ldg", name);
    return launch_march_one<Fam, MASK, false, float, false>(tm, a, tt, grid, stream, info, nm);
}

static inline MarchArgs make_args(const BatchGeom& g, unsigned mask, const SteerSpec& st, float* const* outs, int nplanes)
{
    MarchArgs a;
    memset(&a, 0, sizeof(a));
    a.in = g.in;
    a.in_pitch = (long long)g.in_pitch;
    a.in_frame_stride = (long long)g.in_frame_stride;
    a.cols = g.cols;
    a.full_rows = g.full_rows;
    a.buf_rows = g.buf_rows;
    a.y_origin = g.y_origin;
    a.out_row_begin = g.out_row_begin;
    a.out_row_end = g.out_row_end;
    a.out_row_origin = g.out_row_origin;
    a.out_pitch = (long long)g.out_pitch;
    a.out_frame_stride = (long long)g.out_frame_stride;
    a.mask = mask;
    a.steer_source = st.source;
    a.cos_t = st.cos_t;
    a.sin_t = st.sin_t;
    a.theta_map = st.theta_map;
    a.pyr_out = g.next_level;
    a.pyr_pitch = (long long)g.next_pitch;
    a.pyr_frame_stride = (long long)g.next_frame_stride;
    a.minmax = g.minmax;
    a.minmax_frames = g.minmax_frames;
    for (int p = 0; p < nplanes && p < MARCH_MAX_OUT; ++p) a.out[p] = (mask >> p & 1u) ? outs[p] : nullptr;
    return a;
}


}  // namespace cvs
