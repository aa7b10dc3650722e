// Host-side launch helpers for the marching kernels: tensor-map creation, launch plumbing shared with the bank kernel, the
// table of fused kernel forms of each family and the dispatcher that picks a form for a launch.  The forms' launchers
// (launch_form, march_forms.cuh) are instantiated in their own translation units so that `make -j` compiles them in parallel.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdio>
#include <cstring>
#include <iterator>
#include <mutex>
#include <type_traits>
#include <utility>

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

// The tile of family Fam's TMA-staged kernels: a 3-D fp32 (or 8-bit) tensor (x = cols, y = buffer rows, z = frames), box =
// one tile row band with its halos (the raw byte rows for 8-bit frames); OOB -> zeros.
template <class Fam>
static bool make_tmap(CUtensorMap* m, const BatchGeom& g)
{
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) return false;
    cuuint64_t dims[3] = {(cuuint64_t)g.cols, (cuuint64_t)g.buf_rows, (cuuint64_t)g.n};
    cuuint64_t strides[2] = {(cuuint64_t)g.in_pitch, (cuuint64_t)(g.n > 1 ? g.in_frame_stride : g.in_pitch * (size_t)g.buf_rows)};
    cuuint32_t box[3] = {(cuuint32_t)(g.in_u8 ? (int)MARCH_U8_TW : march_tile_width(Fam::R)), (cuuint32_t)(Fam::BH + 2 * Fam::R), 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(m, g.in_u8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(g.in), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

static inline bool tma_eligible(const BatchGeom& g, int R)
{
    if (((uintptr_t)g.in & 15) || (g.in_pitch & 15) || (g.in_frame_stride & 15)) return false;
    if (g.cols < R + 1 || g.full_rows < R + 1) return false;  // one reflect fold must land inside the tile
    if (g.n > 1 && g.in_frame_stride < g.in_pitch * (size_t)g.buf_rows) return false;
    return true;
}

// ------------------------------------------------------------------------------------------------
// Launch plumbing shared by the marching and bank kernels
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

// true when the handle's taps are bit-identical to the baked reference defaults of the family
template <class Fam>
static bool taps_are_baked(const TapTable<Fam::NSETS, Fam::R>& tt)
{
    for (int s = 0; s < Fam::NSETS; ++s)
        for (int i = 0; i <= Fam::R; ++i) {
            const float bk = Fam::baked(s, i);
            if (memcmp(&bk, &tt.t[s][i], sizeof(float)) != 0) return false;
        }
    return true;
}

// Two-pixel threads store both pixels of a plane as one store of 2 * esz bytes (esz = output element size): every selected
// plane, the pitch and the frame stride must be multiples of it and the width even (the clamped last pair stays aligned).
// The angle pairs are 8-byte loads whatever the output type (the map keeps fp32 elements).
static inline bool pair_store_ok(const BatchGeom& g, const MarchArgs& a, size_t esz)
{
    const size_t m = 2 * esz - 1;
    if ((g.cols & 1) || (g.out_pitch & m) || (g.out_frame_stride & m)) return false;
    for (int p = 0; p < MARCH_MAX_OUT; ++p)
        if (a.out[p] && ((uintptr_t)a.out[p] & m)) return false;
    return !(a.steer_source == CVS_STEER_MAP && ((uintptr_t)a.theta_map & 7));
}

template <class Fam>
static dim3 march_grid(const BatchGeom& g)
{
    return dim3((g.cols + MARCH_TW - 1) / MARCH_TW, (g.out_row_end - g.out_row_begin + Fam::BH - 1) / Fam::BH, g.n);
}

// KFN<<<grid, block, smem, stream>>>(args...), counted in g_launches and described in *info.  Function attributes are per
// DEVICE (context): one flag per (kernel, device).  The 8-bit TMA kernels ask for more than the 48 KB default, so a process
// that drives several GPUs must set them on each one.
template <auto KFN, class... Args>
static cudaError_t launch_kernel(dim3 grid, int block, int smem, cudaStream_t stream, LaunchInfo* info, const char* name, const Args&... args)
{
    static std::atomic<unsigned long long> done[4];  // 256 devices
    int dev = 0;
    if (cudaError_t e = cudaGetDevice(&dev); e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    std::atomic<unsigned long long>& word = done[(dev >> 6) & 3];
    if (!(word.load(std::memory_order_acquire) & bit)) {
        cudaError_t e = cudaFuncSetAttribute(KFN, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(KFN, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        if (e != cudaSuccess) return e;
        word.fetch_or(bit, std::memory_order_release);  // idempotent: a racing thread at worst sets the attributes twice
    }
    KFN<<<grid, block, smem, stream>>>(args...);
    g_launches.fetch_add(1);
    if (info) {
        info->grid[0] = grid.x, info->grid[1] = grid.y, info->grid[2] = grid.z;
        info->block = block;
        info->smem = smem;
        snprintf(info->name, sizeof(info->name), "%s", name);
    }
    return cudaGetLastError();
}

// gridDim.z carries the frame index: batches beyond 65535 frames go out as several launches.  launch(gc, ac, out_off) runs
// one chunk; out_off is the byte offset of its first frame in planes of out_esz-byte elements.  The angle map keeps 4-byte
// elements in the outputs' element layout, so its offset scales by 4 / out_esz.
template <class F>
static cudaError_t for_each_frame_chunk(const BatchGeom& g, const MarchArgs& a, size_t out_esz, F&& launch)
{
    for (int f0 = 0; f0 < g.n; f0 += 65535) {
        BatchGeom gc = g;
        MarchArgs ac = a;
        const size_t out_off = (size_t)f0 * g.out_frame_stride;
        gc.n = g.n - f0 < 65535 ? g.n - f0 : 65535;
        gc.in = static_cast<const char*>(g.in) + (size_t)f0 * g.in_frame_stride;
        ac.in = gc.in;
        for (int p = 0; p < MARCH_MAX_OUT; ++p)
            if (ac.out[p]) ac.out[p] = reinterpret_cast<float*>(reinterpret_cast<char*>(a.out[p]) + out_off);
        if (ac.theta_map) ac.theta_map = reinterpret_cast<const float*>(reinterpret_cast<const char*>(a.theta_map) + 4 / out_esz * out_off);
        if (ac.pyr_out) ac.pyr_out = reinterpret_cast<float*>(reinterpret_cast<char*>(a.pyr_out) + (size_t)f0 * g.next_frame_stride);
        if (ac.minmax) ac.minmax = a.minmax + 2 * (size_t)f0;
        if (cudaError_t e = launch(static_cast<const BatchGeom&>(gc), static_cast<const MarchArgs&>(ac), out_off); e != cudaSuccess) return e;
    }
    return cudaSuccess;
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

// ------------------------------------------------------------------------------------------------
// Fused kernel forms
// ------------------------------------------------------------------------------------------------
// One entry per static kernel key of a family; entry 0, key 0, is the run-time-mask kernel (`<dyn>`) that takes every launch
// no other entry matches.  Each entry has these kernels (march_forms.cuh):
//   fp32 planes, fp32 frames: /tma/imm-taps[/2px] (default taps, static keys only), /tma, /ldg;
//   fp32 planes, 8-bit frames: /tma-u8, /ldg-u8 (constant-bank taps; see capi.cu's `widen` for where that matters);
//   16-bit planes (out16 entries): /tma[-u8]/imm-taps[/2px]/{f16,bf16} only -- other launches narrow an fp32 launch.
struct MarchForm {
    unsigned key;     // march_key(mask, source), | MARCH_MINMAX_FLAG for the fused `lines` statistics
    const char* name;
    int px;           // pixels per thread of the baked-tap forms on fp32 frames (8-bit frames: always 1)
    bool out16;       // has fused fp16 / bf16 twins
    bool any_source;  // no steered plane: the key's mask runs at every steering source
};

template <class Fam>
struct MarchForms;

// Two pixels per thread: 198 instead of 217 instructions per pixel-row, but with the K-fold unrolled body the loop grows to
// 57 KB and falls out of the instruction cache (M2 138.9 -> 118.6 Gpix/s); it pays together with the shift loop
// (CVS_MARCH_SHIFT_U, 27 KB body, 209 instructions per pixel-row): M2 138.9 -> 143.2 Gpix/s at 1080p, 134.7 -> 139.7 at 4K.
// So the issue-bound masks take two pixels.  M1 (short epilogue) loses 1-2 % that way and keeps the unrolled one-pixel
// kernel; lines@map measured 152-155 Gpix/s at one pixel against 142-149 at two.  8-bit frames take one pixel throughout: the
// byte expansion gives each thread two tile columns, which a 64-thread CTA cannot cover, and a two-pixel 8-bit form measured
// no faster (DESIGN.md section 4, item 8).
template <>
struct MarchForms<G2Fam> {
    static constexpr const char* family = "g2_march";
    static constexpr MarchForm form[] = {
        {0u, "dyn", 1, false, false},
        {CVS_G2_MASK_STATE, "M0", 1, true, true},
        {CVS_G2_MASK_ORIENT, "M1", 1, true, false},
        {CVS_G2_MASK_FULL, "M2", 2, true, false},
        {CVS_G2_MASK_LINES, "lines", 2, true, false},
        // min / max exist for `lines` at theta_d only: any other mask with them is cudaErrorNotSupported
        {CVS_G2_MASK_LINES | MARCH_MINMAX_FLAG, "lines+minmax", 2, false, false},
        {march_key(CVS_G2_MASK_STEER5, CVS_STEER_SCALAR), "steer5@scalar", 2, true, false},
        {march_key(CVS_G2_MASK_STEER5, CVS_STEER_MAP), "steer5@map", 2, true, false},
        {march_key(CVS_G2_MASK_FULL, CVS_STEER_SCALAR), "M2@scalar", 2, true, false},
        {march_key(CVS_G2_MASK_FULL, CVS_STEER_MAP), "M2@map", 2, true, false},
        {march_key(CVS_G2_MASK_LINES, CVS_STEER_SCALAR), "lines@scalar", 2, true, false},
        {march_key(CVS_G2_MASK_LINES, CVS_STEER_MAP), "lines@map", 1, true, false},
    };
};

// G4: one pixel per thread throughout (two-pixel forms exist for the issue-bound G2 masks only)
template <>
struct MarchForms<G4Fam> {
    static constexpr const char* family = "g4_march";
    static constexpr MarchForm form[] = {
        {0u, "dyn", 1, false, false},
        {CVS_G4_MASK_BASIS, "basis", 1, true, true},
        {march_key(CVS_G4_MASK_STEER, CVS_STEER_MAP), "steer@map", 1, true, false},
        {march_key(CVS_G4_MASK_STEER, CVS_STEER_SCALAR), "steer@scalar", 1, true, false},
        {march_key(CVS_G4_MASK_STEER, CVS_STEER_DOMINANT), "steer@theta_d", 1, true, false},
    };
};

// Entry of Fam's table for (mask, source, min/max statistics?): 0 (the run-time-mask kernel) when no static key matches, -1
// when none can run it (statistics without their kernel).
template <class Fam>
static int find_form(unsigned mask, int source, bool minmax)
{
    const unsigned key = march_key(mask, source) | (minmax ? (unsigned)MARCH_MINMAX_FLAG : 0u);
    const auto& forms = MarchForms<Fam>::form;
    for (int i = 1; i < (int)std::size(forms); ++i)
        if (forms[i].key == key || (forms[i].any_source && !minmax && forms[i].key == mask)) return i;
    return minmax ? -1 : 0;
}

// Launches entry I of Fam's table with TOut planes from TIn frames (march_forms.cuh; each instantiated explicitly in exactly
// one translation unit, march_g{2,4}*.cu).  fast_px: the baked-tap form to take on fp32 frames (0 = none, 1 or 2 pixels per thread); 16-bit planes
// always take their fast form.
template <class Fam, int I, typename TOut, typename TIn>
cudaError_t launch_form(const BatchGeom& g, const MarchArgs& a, const TapTable<Fam::NSETS, Fam::R>& tt, int fast_px, cudaStream_t stream,
                        LaunchInfo* info);

template <class Fam, typename TOut, typename TIn, size_t... I>
static cudaError_t launch_form_at(int i, const BatchGeom& g, const MarchArgs& a, const TapTable<Fam::NSETS, Fam::R>& tt, int fast_px,
                                  cudaStream_t stream, LaunchInfo* info, std::index_sequence<I...>)
{
    static constexpr decltype(&launch_form<Fam, 0, TOut, TIn>) fn[] = {&launch_form<Fam, (int)I, TOut, TIn>...};
    return fn[i](g, a, tt, fast_px, stream, info);
}

// One fused march of family Fam into TOut planes.  fp32 planes always take a kernel (the loader ladder of launch_form);
// 16-bit planes take the fast form -- a twin of the entry, TMA-eligible frames, the default taps, pair-aligned planes where
// the form has two pixels -- or nothing, and *taken says which (the caller narrows an fp32 launch otherwise).
template <class Fam, typename TOut>
static cudaError_t launch_march(const FamilyTaps& taps, const BatchGeom& g, const MarchArgs& a, cudaStream_t stream, LaunchInfo* info, bool* taken)
{
    *taken = false;
    const int i = find_form<Fam>(a.mask, a.steer_source, a.minmax != nullptr);
    if (i < 0) return cudaErrorNotSupported;
    const MarchForm& f = MarchForms<Fam>::form[i];
    TapTable<Fam::NSETS, Fam::R> tt;
    fill_tap_table<Fam>(taps, tt);
    const bool baked = f.key != 0 && taps_are_baked<Fam>(tt);
    const bool px2 = f.px == 2 && !g.in_u8 && pair_store_ok(g, a, sizeof(TOut));
    if constexpr (!std::is_same_v<TOut, float>)
        if (!f.out16 || !baked || !tma_eligible(g, Fam::R) || (f.px == 2 && !g.in_u8 && !px2)) return cudaSuccess;
    if (g.out_row_end <= g.out_row_begin || g.cols <= 0 || g.n <= 0) return cudaErrorInvalidValue;
    *taken = true;
    const int fast_px = baked ? (px2 ? 2 : 1) : 0;
    constexpr auto all = std::make_index_sequence<std::size(MarchForms<Fam>::form)>{};
    return for_each_frame_chunk(g, a, sizeof(TOut), [&](const BatchGeom& gc, const MarchArgs& ac, size_t) {
        return g.in_u8 ? launch_form_at<Fam, TOut, unsigned char>(i, gc, ac, tt, fast_px, stream, info, all)
                       : launch_form_at<Fam, TOut, float>(i, gc, ac, tt, fast_px, stream, info, all);
    });
}

}  // namespace cvs
