// Fused separable-basis "marching" kernel for sm_100a.
//
// One CTA owns a strip of TW image columns and a band of BH image rows of one frame.
//   1. The input tile (band + R halo rows/cols each side) is staged ONCE into shared memory: a single
//      TMA tensor copy (cp.async.bulk.tensor.3d + mbarrier) for tiles the tensor map can describe, with
//      BORDER_REFLECT_101 halos patched in shared memory afterwards (TMA can only zero-fill), or a
//      cooperative reflect-indexed load for unaligned / tiny / 8-bit inputs.
//   2. Each thread owns one column and marches down the band.  Per row it runs ALL unique row passes from
//      2R+1 shared-memory reads (even/odd tap symmetry: R adds + R subs shared by every filter), pushes
//      the results into a (2R+1)-row register window per row-filtered plane, then runs ALL column passes
//      from registers.  No intermediate ever touches shared or global memory.
//   3. The family's epilogue (orientation analysis, steering, energy, magnitude, phase ...) runs on the
//      basis values still in registers and stores only the selected planes, one coalesced 128 B line
//      per warp per plane.
//
// This replaces the reference's 7 (G2) / 11 (G4) full-image cv::sepFilter2D passes plus ~40 full-image
// Mat temporaries (cvsteer/SteerableFiltersG2.cpp:62-99, SteerableFiltersG4.cpp:69-80) by one pass that
// reads each input pixel from HBM once and writes each selected output once.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

#include <type_traits>
#include <utility>

#include "device_math.cuh"

// 1: static-mask kernels of families without a shared row pass replicate the whole row body per window slot (no slot
// dispatch in the loop).  Measured on B200: M1 155 -> 180 Gpix/s, M2 122 -> 132 Gpix/s versus the switch-based loop.
#ifndef CVS_MARCH_UNROLL_EPILOGUE
#define CVS_MARCH_UNROLL_EPILOGUE 1
#endif
// The slot dispatch of the rolled loops is a balanced compare tree, not a switch (which nvcc lowers to a constant-memory
// jump table: LDC + BRX on the critical path of every row; measured 9-15 % slower).
// masks with at most this many planes keep a 64-bit base per plane in registers (2 registers each)
// With two-pixel threads (the forms that march_launch.cuh's table gives two pixels): replace the K-fold unrolled body by a
// "shift" loop -- U row bodies on a LINEAR register window (2R old rows + U new ones), then 2R x NROW x PX register moves
// shift the window down by U.  Body = U x 2 x ~200 instructions (U = 4: 27 KB, inside the instruction cache) at the price
// of 2R*NROW/U moves per pixel-row.  0 = off.
#ifndef CVS_MARCH_SHIFT_U
#define CVS_MARCH_SHIFT_U 4
#endif
// Static-mask kernels of families WITH a shared row pass (G4: 13 slot bodies) run a software-pipelined loop: the row pass of
// tile row rt+1 is issued in the same basic block as the point-wise epilogue of output row rt, so its 59 independent FMAs
// and 13 shared-memory loads fill the issue slots the epilogue's long dependent chain (sincos -> weights -> steer ->
// rcp -> atan polynomial) leaves empty at 3 warps per scheduler.  0 = the plain rolled loop.
#ifndef CVS_MARCH_PIPE
#define CVS_MARCH_PIPE 1
#endif
// two-pixel kernels (64 threads): minimum CTAs per SM for the register cap.  6 -> 168 registers (ptxas settles at 155-164 without
// spills instead of 167-189), so shared memory (5 CTAs) and not the register file (4) bounds the occupancy: 10 warps per SM
// instead of 8, measured +1.0-1.5 % on M2 and +2.5 % on steer5@scalar.  0 = the family's MIN_CTAS (no cap at 64 threads).
#ifndef CVS_PX2_MIN_CTAS
#define CVS_PX2_MIN_CTAS 6
#endif
#ifndef CVS_CURSOR_MAX_PLANES
#define CVS_CURSOR_MAX_PLANES 8
#endif

namespace cvs {

// ------------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA (no CUTLASS dependency)
// ------------------------------------------------------------------------------------------------
namespace ptx {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int x, int y, int z, uint64_t* bar)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
        : "memory");
}
// contiguous bytes -> L2 (no shared-memory destination, no completion to wait for); 16-byte aligned address and size
__device__ __forceinline__ void bulk_prefetch_l2(const void* gptr, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
}  // namespace ptx

// ------------------------------------------------------------------------------------------------
// Kernel arguments
// ------------------------------------------------------------------------------------------------
enum { MARCH_TW = 128, MARCH_MAX_OUT = 20 };
// Static specialisations are keyed by the plane mask AND the steering source: key = planes | source << 28 (source 0 =
// the in-kernel dominant angle, so a bare plane mask keeps meaning "steer at theta_d").  Key 0 = everything at run time.
// Bit 27 of a key: also reduce min / max of the three `lines` maps per frame (fused cv::normalize NORM_MINMAX statistics).
enum : unsigned { MARCH_PLANE_BITS = 0x07FFFFFFu, MARCH_MINMAX_FLAG = 0x08000000u, MARCH_SRC_SHIFT = 28 };
__host__ __device__ constexpr unsigned march_key(unsigned planes, int steer_source) { return planes | ((unsigned)steer_source << MARCH_SRC_SHIFT); }
// TMA needs every box row to START on a 16-byte boundary of global memory, i.e. the innermost start coordinate must be
// a multiple of 4 floats (x0 - 6 faults with "illegal instruction"; x0 - 4 and x0 - 8 are fine).  So the tile's left
// halo is the radius rounded up to 4 floats, and the row pitch follows.
__host__ __device__ constexpr int march_halo_left(int R) { return (R + 3) & ~3; }
__host__ __device__ constexpr int march_tile_width(int R) { return MARCH_TW + 2 * march_halo_left(R); }
// 8-bit input staged by TMA: the box starts 16 BYTES left of the strip (start coordinates must be multiples of 16 bytes),
// so a raw tile row is 128 + 2 * 16 bytes; it is expanded to the fp32 tile in shared memory before the march.
enum { MARCH_U8_HALO = 16, MARCH_U8_TW = MARCH_TW + 2 * MARCH_U8_HALO };
__host__ __device__ constexpr int march_smem_bytes(int R, int BH, bool tma_u8)
{
    const int f32 = (BH + 2 * R) * march_tile_width(R) * 4 + 16;  // fp32 tile + mbarrier
    return tma_u8 ? ((f32 + 127) & ~127) + (BH + 2 * R) * MARCH_U8_TW : f32;
}

struct MarchArgs {
    // input: n frames, rows are buffer rows; element (f, r, c) at in + f*in_frame_stride + r*in_pitch + c (bytes for
    // pitch/stride).  The buffer holds image rows [y_origin, y_origin + buf_rows) of an image full_rows tall.
    const void* in;
    long long in_pitch, in_frame_stride;   // bytes
    int cols, full_rows, buf_rows, y_origin;
    int out_row_begin, out_row_end, out_row_origin;  // image rows to produce; output buffer row = y - out_row_origin
    long long out_pitch, out_frame_stride;           // bytes
    unsigned mask;
    int steer_source;          // cvs_steer_source
    float cos_t, sin_t;        // scalar steering angle
    const float* theta_map;    // per-pixel angle map in output layout (steer_source == MAP)
    float* out[MARCH_MAX_OUT];
    // optional fused pyramid emission (whole frames only): next level = cv::pyrDown(input), written from the staged tile
    float* pyr_out;
    long long pyr_pitch, pyr_frame_stride;  // bytes
    // optional fused min/max of the tracked maps (keys with MARCH_MINMAX_FLAG): ordered-uint32 pairs, map m of frame f at
    // minmax[2 * (m * minmax_frames + f)] (min) and [.. + 1] (max); initialised to (0xffffffff, 0) by the caller
    unsigned* minmax;
    int minmax_frames;
};

// Tap tables passed BY VALUE as a kernel parameter: they live in the constant bank, so every FFMA takes
// its tap as a constant-bank operand (no register, no global state shared between handles).
// t[s][i] = tap i (i = 0..R) of unique tap set s; odd sets have t[s][0] == 0.
template <int NSETS, int R>
struct TapTable {
    float t[NSETS][R + 1];
};

// Balanced compare tree over [LO, HI): calls f(integral_constant<int, slot>) for the run-time `slot`.
template <int LO, int HI, class F>
__device__ __forceinline__ void dispatch_tree(int slot, F&& f)
{
    if constexpr (HI - LO == 1) {
        f(std::integral_constant<int, LO>{});
    } else {
        constexpr int MID = (LO + HI) / 2;
        if (slot < MID) dispatch_tree<LO, MID>(slot, f);
        else dispatch_tree<MID, HI>(slot, f);
    }
}

// ------------------------------------------------------------------------------------------------
// Output cursor: where this thread's pixel of the current row lives in every output plane.
// ------------------------------------------------------------------------------------------------
// Static masks: every selected plane keeps a loop-invariant 64-bit base (band origin of this CTA) in a vector register
// pair, and ONE 32-bit element index per thread walks down the band.  A store is then IMAD.WIDE.U32 (idx*4 + base) +
// STG: 2 issue slots instead of the 4 a 64-bit add pair per plane costs.  The bases are laundered through an opaque
// `mov` so that ptxas keeps them in vector registers (as a uniform-register value they could not be the addend of
// IMAD.WIDE); the index stays far below 2^32 because it is relative to the CTA's own band (<= BH rows).
__device__ __forceinline__ unsigned long long opaque64(unsigned long long v)
{
    unsigned long long r;
    asm volatile("mov.b64 %0, %1;" : "=l"(r) : "l"(v));
    return r;
}

// 16-bit output planes (TOut = __half / __nv_bfloat16): the fp32 value the epilogue computed, rounded to nearest even at the
// store -- bit for bit what torch.Tensor.to(float16 / bfloat16) makes of the fp32 plane (NaN stays NaN, fp16 overflow is +-inf)
template <typename TOut>
__device__ __forceinline__ unsigned short to_out16(float v)
{
    unsigned short h;
    if constexpr (std::is_same_v<TOut, __half>) asm("cvt.rn.f16.f32 %0, %1;" : "=h"(h) : "f"(v));
    else asm("cvt.rn.bf16.f32 %0, %1;" : "=h"(h) : "f"(v));
    return h;
}
// two adjacent pixels packed by one instruction: v0 in the low half (lower address), v1 in the high half
template <typename TOut>
__device__ __forceinline__ unsigned to_out16x2(float v0, float v1)
{
    unsigned r;
    if constexpr (std::is_same_v<TOut, __half>) asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(v1), "f"(v0));
    else asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(v1), "f"(v0));
    return r;
}

// The steering-angle map stays fp32 in the outputs' ELEMENT layout: with 16-bit outputs its byte offsets and row step are
// twice the outputs' (kThetaScale), with fp32 outputs they are the same.
template <typename TOut>
inline constexpr long long kThetaScale = 4 / (long long)sizeof(TOut);

template <unsigned MASK, int NPLANES, typename TOut = float>
struct OutCursor {
    static constexpr bool F32 = sizeof(TOut) == 4;
    unsigned long long base[NPLANES];
    unsigned long long th_base;  // steering-angle map (same element layout as the outputs); dead unless theta() is used
    unsigned idx;                // element index of this thread's pixel relative to the bases
    unsigned pitch_elems;
    mutable float pend[NPLANES];  // two-pixel threads: the left pixel's value waits here for its neighbour (registers)
    mutable float mn[3], mx[3];  // running min / max of up to three tracked maps (dead unless used)
    __device__ __forceinline__ void track(int k, float v) const { mn[k] = fminf(mn[k], v), mx[k] = fmaxf(mx[k], v); }  // fmin/fmax skip NaNs
    __device__ __forceinline__ OutCursor(const MarchArgs& a, long long band_off, int x)
    {
#pragma unroll
        for (int q = 0; q < NPLANES; ++q)
            base[q] = (MASK >> q & 1u) ? opaque64((unsigned long long)(reinterpret_cast<char*>(a.out[q]) + band_off)) : 0ull;
        th_base = (MASK >> MARCH_SRC_SHIFT) == 2u /* CVS_STEER_MAP */
                      ? opaque64((unsigned long long)(reinterpret_cast<const char*>(a.theta_map) + kThetaScale<TOut> * band_off))
                      : 0ull;
        idx = (unsigned)x;
        pitch_elems = (unsigned)(a.out_pitch >> (F32 ? 2 : 1));
#pragma unroll
        for (int k = 0; k < 3; ++k) mn[k] = __int_as_float(0x7f800000), mx[k] = __int_as_float(0xff800000);  // +inf / -inf
    }
    // No predicate: threads past the right image edge are clamped onto the last valid column (see k_march), so they
    // recompute that pixel and store the identical value to the identical address.
    __device__ __forceinline__ void put(const MarchArgs&, int q, float v) const
    {
        if constexpr (F32)
            asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %1, 4, %0;\n\tst.global.cs.f32 [a], %2;\n\t}" ::"l"(base[q]), "r"(idx), "f"(v) : "memory");
        else
            asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %1, 2, %0;\n\tst.global.cs.b16 [a], %2;\n\t}" ::"l"(base[q]), "r"(idx), "h"(to_out16<TOut>(v))
                         : "memory");
    }
    // two adjacent pixels of one thread as one 8-byte (fp32) or 4-byte (16-bit) store (x even, bases and pitch multiples of the
    // store width: host-checked)
    __device__ __forceinline__ void put2(const MarchArgs&, int q, float v0, float v1) const
    {
        if constexpr (F32)
            asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %1, 4, %0;\n\tst.global.cs.v2.f32 [a], {%2, %3};\n\t}" ::"l"(base[q]), "r"(idx), "f"(v0),
                         "f"(v1)
                         : "memory");
        else
            asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %1, 2, %0;\n\tst.global.cs.b32 [a], %2;\n\t}" ::"l"(base[q]), "r"(idx),
                         "r"(to_out16x2<TOut>(v0, v1))
                         : "memory");
    }
    // steering angle of this thread's pixel `rows_ahead` output rows below the current one
    __device__ __forceinline__ float theta(const MarchArgs&, int rows_ahead = 0) const
    {
        float v;
        asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %2, 4, %1;\n\tld.global.nc.f32 %0, [a];\n\t}"
                     : "=f"(v)
                     : "l"(th_base), "r"(idx + (unsigned)rows_ahead * pitch_elems));
        return v;
    }
    // ... of the two adjacent pixels of a two-pixel thread (8-byte aligned: x even, map base and pitch multiples of 8, host-checked)
    __device__ __forceinline__ float2 theta2(const MarchArgs&, int rows_ahead = 0) const
    {
        float2 v;
        asm volatile("{\n\t.reg .u64 a;\n\tmad.wide.u32 a, %3, 4, %2;\n\tld.global.nc.v2.f32 {%0, %1}, [a];\n\t}"
                     : "=f"(v.x), "=f"(v.y)
                     : "l"(th_base), "r"(idx + (unsigned)rows_ahead * pitch_elems));
        return v;
    }
    __device__ __forceinline__ void next_row() { idx += pitch_elems; }
};

template <int NPLANES, typename TOut>
struct OutCursor<0u, NPLANES, TOut> {  // run-time mask: one shared byte offset, 64-bit add per plane at the store
    static constexpr bool F32 = sizeof(TOut) == 4;
    long long off, pitch;
    mutable float pend[NPLANES];
    mutable float mn[3], mx[3];
    __device__ __forceinline__ void track(int k, float v) const { mn[k] = fminf(mn[k], v), mx[k] = fmaxf(mx[k], v); }
    __device__ __forceinline__ OutCursor(const MarchArgs& a, long long band_off, int x)
        : off(band_off + (long long)sizeof(TOut) * x), pitch(a.out_pitch)
    {
#pragma unroll
        for (int k = 0; k < 3; ++k) mn[k] = __int_as_float(0x7f800000), mx[k] = __int_as_float(0xff800000);
    }
    __device__ __forceinline__ void put(const MarchArgs& a, int q, float v) const
    {
        if constexpr (F32) __stcs(reinterpret_cast<float*>(reinterpret_cast<char*>(a.out[q]) + off), v);
        else __stcs(reinterpret_cast<unsigned short*>(reinterpret_cast<char*>(a.out[q]) + off), to_out16<TOut>(v));
    }
    __device__ __forceinline__ void put2(const MarchArgs& a, int q, float v0, float v1) const
    {
        if constexpr (F32) __stcs(reinterpret_cast<float2*>(reinterpret_cast<char*>(a.out[q]) + off), make_float2(v0, v1));
        else __stcs(reinterpret_cast<unsigned*>(reinterpret_cast<char*>(a.out[q]) + off), to_out16x2<TOut>(v0, v1));
    }
    __device__ __forceinline__ float theta(const MarchArgs& a, int rows_ahead = 0) const
    {
        return *reinterpret_cast<const float*>(reinterpret_cast<const char*>(a.theta_map) + kThetaScale<TOut> * (off + rows_ahead * pitch));
    }
    __device__ __forceinline__ float2 theta2(const MarchArgs& a, int rows_ahead = 0) const
    {
        return *reinterpret_cast<const float2*>(reinterpret_cast<const char*>(a.theta_map) + kThetaScale<TOut> * (off + rows_ahead * pitch));
    }
    __device__ __forceinline__ void next_row() { off += pitch; }
};

// Views of a cursor for threads that own two adjacent pixels: the epilogue of the left pixel parks its values, the
// epilogue of the right pixel stores both as one 8-byte access per plane.
template <class Cur>
struct PairLeft {
    const Cur& c;
    __device__ __forceinline__ void put(const MarchArgs&, int q, float v) const { c.pend[q] = v; }
    __device__ __forceinline__ void track(int k, float v) const { c.track(k, v); }
};
template <class Cur>
struct PairRight {
    const Cur& c;
    __device__ __forceinline__ void put(const MarchArgs& a, int q, float v) const { c.put2(a, q, c.pend[q], v); }
    __device__ __forceinline__ void track(int k, float v) const { c.track(k, v); }
};

// ------------------------------------------------------------------------------------------------
// Tile loaders
// ------------------------------------------------------------------------------------------------
// Patch BORDER_REFLECT_101 halos of a TMA-loaded (zero-filled) tile in place.  Requires cols >= R+1 and
// full_rows >= R+1 so that one fold lands inside the tile (host guarantees; smaller images take the manual path).
template <int R, int TWH, int TROWS>
__device__ __forceinline__ void patch_reflect(float* tile, int x0, int ytop, int cols, int full_rows, int nthreads)
{
    constexpr int HL = march_halo_left(R);  // tile column 0 is image column x0 - HL
    const bool fix_l = (x0 - R) < 0, fix_r = (x0 + MARCH_TW + R) > cols;
    const bool fix_t = ytop < 0, fix_b = (ytop + TROWS) > full_rows;
    if (!(fix_l || fix_r || fix_t || fix_b)) return;  // CTA-uniform
    if (fix_l || fix_r) {
        for (int i = threadIdx.x; i < TROWS * 2 * R; i += nthreads) {
            const int rt = i / (2 * R), k = i % (2 * R);
            const int gx = (k < R) ? (k - R) : (cols + (k - R));  // -R..-1, cols..cols+R-1
            const int ct = gx - (x0 - HL);
            const bool need = (k < R) ? fix_l : (fix_r && ct < TWH);
            if (need && ct >= 0) {
                const int sx = (gx < 0 ? -gx : 2 * (cols - 1) - gx) - (x0 - HL);
                tile[rt * TWH + ct] = tile[rt * TWH + sx];
            }
        }
        __syncthreads();
    }
    if (fix_t || fix_b) {
        for (int i = threadIdx.x; i < 2 * R * TWH; i += nthreads) {
            const int k = i / TWH, ct = i % TWH;
            const int gy = (k < R) ? (k - R) : (full_rows + (k - R));
            const int rt = gy - ytop;
            const bool need = (k < R) ? fix_t : fix_b;
            if (need && rt >= 0 && rt < TROWS) {
                const int sy = (gy < 0 ? -gy : 2 * (full_rows - 1) - gy) - ytop;
                tile[rt * TWH + ct] = tile[sy * TWH + ct];
            }
        }
        __syncthreads();
    }
}

// Cooperative reflect-indexed load: any size (iterated folding), any alignment, fp32 or u8 input.
// Row-oriented: a thread owns tile columns t and t + nthreads for every tile row, so the column fold is done once per
// thread and a warp's load is one contiguous 128-byte (32-byte for u8) segment; the row fold is warp-uniform and a
// single select unless the image is shorter than the tile, so the row loop is unrolled to keep 8 loads in flight.
template <int R, int TWH, int TROWS, typename TIn>
__device__ __forceinline__ void load_tile_manual(float* tile, const MarchArgs& a, int frame, int x0, int ytop,
                                                 int nthreads)
{
    const char* base = (const char*)a.in + (long long)frame * a.in_frame_stride;
    const int c0 = threadIdx.x, c1 = threadIdx.x + nthreads;  // TWH <= 2 * nthreads
    const bool two = c1 < TWH;
    const int gx0 = dev::reflect101(x0 - march_halo_left(R) + c0, a.cols);
    const int gx1 = two ? dev::reflect101(x0 - march_halo_left(R) + c1, a.cols) : gx0;
    const int n = a.full_rows;
    if (ytop >= -(n - 1) && ytop + TROWS - 1 <= 2 * (n - 1)) {
        // one fold reaches every row of this tile (always, unless the image is shorter than the tile): branch-free rows
#pragma unroll 8
        for (int rt = 0; rt < TROWS; ++rt) {
            const int p = ytop + rt;
            const int gy = (p < 0 ? -p : (p >= n ? 2 * (n - 1) - p : p)) - a.y_origin;
            const bool ok = gy >= 0 && gy < a.buf_rows;  // band mode: rows outside the resident band are never used
            const TIn* rp = (const TIn*)(base + (long long)(ok ? gy : 0) * a.in_pitch);
            const float v0 = (float)rp[gx0], v1 = (float)rp[gx1];
            tile[rt * TWH + c0] = ok ? v0 : 0.f;
            if (two) tile[rt * TWH + c1] = ok ? v1 : 0.f;
        }
    } else {
        for (int rt = 0; rt < TROWS; ++rt) {
            const int gy = dev::reflect101(ytop + rt, n) - a.y_origin;
            float v0 = 0.f, v1 = 0.f;
            if (gy >= 0 && gy < a.buf_rows) {
                const TIn* rp = (const TIn*)(base + (long long)gy * a.in_pitch);
                v0 = (float)rp[gx0], v1 = (float)rp[gx1];
            }
            tile[rt * TWH + c0] = v0;
            if (two) tile[rt * TWH + c1] = v1;
        }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------------
// The marching kernel.  Fam supplies:
//   R, NSETS, NROW, NBASIS, BH, MIN_CTAS
//   row_set[NROW], row_odd[NROW]                  tap set / parity of each row-filtered plane
//   basis_row[NBASIS], basis_set[NBASIS], basis_odd[NBASIS]   row plane / column tap set / parity per basis plane
//   static void epilogue<MASK>(const float (&b)[NBASIS], const MarchArgs&, long long out_off, long long th_off)
// ------------------------------------------------------------------------------------------------
// Fused pyramid emission: the next pyramid level (cv::pyrDown of the input: [1 4 6 4 1]^2/256, reflect-101, even samples)
// for the part of the image this CTA has staged anyway.  The tile's halo (R >= 2) already holds the reflected border, so
// this costs shared-memory reads and ~4 % more arithmetic instead of a second pass over the input in HBM.
// CTA region: output rows [yb/2, ceil((yb+nrows)/2)) x output columns [x0/2, x0/2 + 64); thread t takes column t & 63 and
// the first / second half of the rows (t >> 6), marching with a 5-row window of horizontal sums.
template <int R, int BH, int NT>
__device__ __forceinline__ void emit_next_level(const float* tile, const MarchArgs& a, int frame, int x0, int yb)
{
    static_assert(NT == 64 || NT == 128, "64 output columns x 1 or 2 row halves");
    constexpr int TWH = march_tile_width(R), HL = march_halo_left(R);
    int nrows = a.out_row_end - yb;
    nrows = nrows < BH ? nrows : BH;
    const int ocols = (a.cols + 1) >> 1;
    const int xl = threadIdx.x & 63, half = threadIdx.x >> 6;
    const int xo = (x0 >> 1) + xl;
    const int nout = (nrows + 1) >> 1;                 // output rows of this CTA (yb is even)
    const int per = NT == 128 ? (nout + 1) >> 1 : nout;
    const int ly0 = half * per, ly1 = min(nout, ly0 + per);
    if (xo >= ocols || ly0 >= ly1) return;
    const float* tc = tile + 2 * xl + HL;              // tile column of input column 2*xo
    auto H = [&](int lr) {                             // horizontal 5-tap of input row yb + lr (tile row lr + R)
        const float* p = tc + (lr + R) * TWH;
        return dev::pyr_tap5(p[-2], p[-1], p[0], p[1], p[2]);
    };
    float* dst = reinterpret_cast<float*>(reinterpret_cast<char*>(a.pyr_out) + (long long)frame * a.pyr_frame_stride +
                                          (long long)((yb >> 1) + ly0) * a.pyr_pitch) + xo;
    const long long op = a.pyr_pitch >> 2;
    int lr = 2 * ly0;
    float h0 = H(lr - 2), h1 = H(lr - 1), h2 = H(lr);
    for (int ly = ly0; ly < ly1; ++ly) {
        const float h3 = H(lr + 1), h4 = H(lr + 2);
        *dst = dev::pyr_tap5(h0, h1, h2, h3, h4) * (1.f / 256.f);
        dst += op;
        h0 = h2, h1 = h3, h2 = h4;
        lr += 2;
    }
}

// PX = pixels (adjacent columns) per thread.  PX = 2 halves the per-pixel cost of everything that is per THREAD and row:
// shared-memory loads (K + 1 values as 8-byte loads feed two pixels instead of K values feeding one), store instructions
// and their 64-bit address arithmetic (one 8-byte store per plane for two pixels), loop control.
// TOut: element type of the output planes (float, or __half / __nv_bfloat16 rounded at the store; see OutCursor).
// march_body is the whole kernel; the epilogue stores through a Cursor(out, band_off, x) (k_march: an OutCursor on a.out[], with
// out = a; k_bank in march_bank.cuh: the bank's per-angle planes).
template <class Fam, unsigned MASK, bool USE_TMA, typename TIn, bool BAKED, int PX, typename TOut, class Cursor, class OutArgs>
__device__ __forceinline__ void march_body(const CUtensorMap& tmap, const MarchArgs& a, const TapTable<Fam::NSETS, Fam::R>& taps,
                                           const OutArgs& out)
{
    constexpr int R = Fam::R, K = 2 * R + 1, TW = MARCH_TW, TWH = march_tile_width(R), BH = Fam::BH, TROWS = BH + 2 * R;
    constexpr int NROW = Fam::NROW, NB = Fam::NBASIS, NT = TW / PX;
    static_assert(K <= 13, "extend the slot switch");
    static_assert(PX == 1 || (PX == 2 && USE_TMA && MASK != 0 && (march_halo_left(R) - R) % 2 == 0),
                  "two-pixel threads: TMA-staged tile, static mask, 8-byte aligned tap window");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* tile = reinterpret_cast<float*>(smem_raw);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + sizeof(float) * TROWS * TWH);

    const int frame = blockIdx.z;
    const int x0 = blockIdx.x * TW;
    const int yb = a.out_row_begin + blockIdx.y * BH;  // first image row this CTA produces
    const int ytop = yb - R;                           // image row of tile row 0

    if (USE_TMA) {
        constexpr bool U8 = sizeof(TIn) == 1;
        unsigned char* raw = smem_raw + ((sizeof(float) * TROWS * TWH + 16 + 127) & ~size_t(127));  // 8-bit staging area (U8 only)
        if (threadIdx.x == 0) {
            ptx::prefetch_tmap(&tmap);
            ptx::mbar_init(bar, 1);
            ptx::fence_mbar_init();
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            if constexpr (U8) {
                ptx::mbar_arrive_expect_tx(bar, TROWS * MARCH_U8_TW);
                ptx::tma_load_3d(raw, &tmap, x0 - MARCH_U8_HALO, ytop - a.y_origin, frame, bar);
            } else {
                ptx::mbar_arrive_expect_tx(bar, TROWS * TWH * sizeof(float));
                ptx::tma_load_3d(tile, &tmap, x0 - march_halo_left(R), ytop - a.y_origin, frame, bar);
            }
        }
        ptx::mbar_wait(bar, 0);
        if constexpr (U8) {
            // expand bytes -> fp32 tile: a thread owns tile columns t and t + NT for every row (TMA zero-filled the
            // out-of-image part, which patch_reflect overwrites below exactly as for fp32 input)
            static_assert(TWH <= 2 * NT, "two tile columns per thread");
            const int c0 = threadIdx.x, c1 = threadIdx.x + NT;
            const unsigned char* rp = raw + (MARCH_U8_HALO - march_halo_left(R));
#pragma unroll 8
            for (int rt = 0; rt < TROWS; ++rt, rp += MARCH_U8_TW) {
                tile[rt * TWH + c0] = (float)rp[c0];
                if (c1 < TWH) tile[rt * TWH + c1] = (float)rp[c1];
            }
            __syncthreads();
        }
        patch_reflect<R, TWH, TROWS>(tile, x0, ytop, a.cols, a.full_rows, NT);
    } else {
        load_tile_manual<R, TWH, TROWS, TIn>(tile, a, frame, x0, ytop, NT);
    }

    // Steering-angle map of this CTA's band -> L2, one 512-byte row segment per thread, issued before the march starts.
    // The in-loop load (one row ahead) then costs an L2 hit instead of a DRAM round trip: with one 128-byte line in flight
    // per warp and 12 warps per SM, Little's law capped the map read at ~290 GB/s -- exactly what the G4 steer kernel
    // needed, and 11 % of its warp samples sat on that load (profiles/r02_ncu_g4_steer_before.txt).
    if constexpr (MASK != 0) {
        if (Fam::template reads_theta_map<MASK>(a)) {
            const int rows_here = min(BH, a.out_row_end - yb);
            const int seg = (min(TW, a.cols - x0) * 4) & ~15;
            constexpr long long TS = kThetaScale<TOut>;  // map offsets in bytes of 4-byte elements
            const long long th_pitch = TS * a.out_pitch;
            const char* tp = reinterpret_cast<const char*>(a.theta_map) + TS * ((long long)frame * a.out_frame_stride) +
                             TS * ((long long)(yb - a.out_row_origin) * a.out_pitch) + 4ll * x0;
            if (seg > 0 && ((reinterpret_cast<uintptr_t>(tp) | (uintptr_t)th_pitch) & 15) == 0)
                for (int r = threadIdx.x; r < rows_here; r += NT) ptx::bulk_prefetch_l2(tp + (long long)r * th_pitch, (uint32_t)seg);
        }
    }

    // Threads past the right image edge (ragged last strip) are clamped onto the last valid column: they redo that pixel
    // and store the same value to the same address, so the loop needs no bounds predicate at all.
    // (PX = 2: cols is even, host-checked, so the clamped pair stays aligned)
    const int x = min(x0 + PX * (int)threadIdx.x, a.cols - PX);
    const float* tcol = tile + (x - x0) + (march_halo_left(R) - R);  // leftmost tap of this thread's column
    int nrows = a.out_row_end - yb;
    nrows = nrows < BH ? nrows : BH;

    // Taps: FFMA immediates when the handle's taps are the baked reference defaults, else constant-bank operands
    // straight out of the kernel parameter block.
    auto tap = [&](int set, int i) -> float {
        if constexpr (BAKED) return Fam::baked(set, i);
        else return taps.t[set][i];
    };

    // column-pass tap of basis plane q: the family may fold a per-plane constant (steering factor) into it
    constexpr bool PRESC = Fam::template prescaled<MASK, BAKED>();
    auto ctap = [&](int q, int set, int i) -> float { return PRESC ? tap(set, i) * Fam::steer_coeff(q) : tap(set, i); };

    float win[NROW][K][PX];  // (2R+1)-row register window per row-filtered plane; slot indices are compile-time
    float b[PX][NB];

    // One tile row: all unique row passes (even/odd symmetry: R sums + R differences are shared by every filter of the
    // pass), results in r[].
    float r[NROW][PX];
    auto row_pass = [&](int rt) {
        const float* src = tcol + rt * TWH;
        float v[K + PX - 1];
        if constexpr (PX == 2) {  // K + 1 values, 8-byte aligned (x, the halo offset and the tile pitch are even)
            const float2* src2 = reinterpret_cast<const float2*>(src);
#pragma unroll
            for (int k = 0; k < (K + 1) / 2; ++k) {
                const float2 t = src2[k];
                v[2 * k] = t.x, v[2 * k + 1] = t.y;
            }
        } else {
#pragma unroll
            for (int k = 0; k < K; ++k) v[k] = src[k];
        }
#pragma unroll
        for (int px = 0; px < PX; ++px) {
            float s[R + 1], d[R + 1];
            s[0] = v[px + R];
            d[0] = 0.f;
#pragma unroll
            for (int i = 1; i <= R; ++i) {
                s[i] = v[px + R + i] + v[px + R - i];
                d[i] = v[px + R + i] - v[px + R - i];
            }
#pragma unroll
            for (int p = 0; p < NROW; ++p) {
                const int set = Fam::row_set(p);
                float acc;
                if (Fam::row_odd(p)) {
                    acc = tap(set, 1) * d[1];
#pragma unroll
                    for (int i = 2; i <= R; ++i) acc = fmaf(tap(set, i), d[i], acc);
                } else {
                    acc = tap(set, 0) * s[0];
#pragma unroll
                    for (int i = 1; i <= R; ++i) acc = fmaf(tap(set, i), s[i], acc);
                }
                r[p][px] = acc;
            }
        }
    };
    // Column passes for the window whose NEWEST row is r[] (not yet stored) and whose oldest row still sits in `slot`;
    // afterwards r[] takes the oldest row's place.  Row offset k in [-R, R] around the centre row lives in slot
    // (slot + 1 + R + k) mod K for k < R, and in r[] for k == R.
    auto col_pass = [&](bool emit, auto slot_c) {
        constexpr int slot = decltype(slot_c)::value;
        if (emit) {  // CTA-uniform: the first 2R rows only feed the window
#pragma unroll
            for (int px = 0; px < PX; ++px) {
#pragma unroll
                for (int q = 0; q < NB; ++q) {
                    const int rp = Fam::basis_row(q), set = Fam::basis_set(q);
                    auto w = [&](int k) -> float { return k == R ? r[rp][px] : win[rp][(slot + 1 + R + k + K) % K][px]; };
                    float acc;
                    if (Fam::basis_odd(q)) {
                        acc = ctap(q, set, 1) * (w(1) - w(-1));
#pragma unroll
                        for (int i = 2; i <= R; ++i) acc = fmaf(ctap(q, set, i), w(i) - w(-i), acc);
                    } else {
                        acc = ctap(q, set, 0) * w(0);
#pragma unroll
                        for (int i = 1; i <= R; ++i) acc = fmaf(ctap(q, set, i), w(i) + w(-i), acc);
                    }
                    b[px][q] = acc;
                }
            }
        }
#pragma unroll
        for (int p = 0; p < NROW; ++p)
#pragma unroll
            for (int px = 0; px < PX; ++px) win[p][slot][px] = r[p][px];
    };

    // The window rotates by one slot per row.  Register files cannot be indexed dynamically, so the slot-dependent code
    // exists once per slot behind a K-way switch.  Everything that does not depend on the slot follows the switch ONCE
    // (the whole point-wise epilogue) or, for families with Fam::SHARED_ROW_PASS, precedes it once (the row pass, at
    // the price of NROW register moves per row): this is what keeps the loop body inside the instruction cache.
    // Output addressing: see OutCursor.
    const long long band_off = (long long)frame * a.out_frame_stride + (long long)(yb - a.out_row_origin) * a.out_pitch;
    Cursor cur(out, band_off, x);
    // point-wise epilogue of the row just finished by col_pass (+ the stores), then on to the next output row
    auto emit_row = [&](float th, float th_right = 0.f) {  // th_right: the right pixel's steering angle (two-pixel @map kernels)
        if constexpr (PX == 1) {
            Fam::template epilogue<MASK, PRESC, false>(b[0], a, cur, th);
        } else {
            Fam::template epilogue<MASK, PRESC, false>(b[0], a, PairLeft<Cursor>{cur}, th);
            Fam::template epilogue<MASK, PRESC, false>(b[1], a, PairRight<Cursor>{cur}, th_right);
        }
        cur.next_row();
    };
    int rt_done = 0;  // tile rows already consumed by the unrolled path below (always a multiple of K)
    constexpr bool SHIFT = CVS_MARCH_SHIFT_U > 0 && PX == 2 && MASK != 0 && !Fam::SHARED_ROW_PASS;
    if constexpr (SHIFT) {
        constexpr int U = CVS_MARCH_SHIFT_U > 0 ? CVS_MARCH_SHIFT_U : 1, W2 = 2 * R;
        float lw[NROW][W2 + U][PX];  // linear window: [0, 2R) = the 2R rows above the newest ones, oldest first; [2R, 2R+U) = new rows
        const int total = nrows + W2;
        auto push = [&](auto pos_c) {
            constexpr int pos = decltype(pos_c)::value;
#pragma unroll
            for (int p = 0; p < NROW; ++p)
#pragma unroll
                for (int px = 0; px < PX; ++px) lw[p][pos][px] = r[p][px];
        };
        auto col_lin = [&](auto u_c) {  // the output row whose newest window row sits at position 2R + u
            constexpr int u = decltype(u_c)::value;
#pragma unroll
            for (int px = 0; px < PX; ++px) {
#pragma unroll
                for (int q = 0; q < NB; ++q) {
                    const int rp = Fam::basis_row(q), set = Fam::basis_set(q);
                    auto w = [&](int k) -> float { return lw[rp][u + R + k][px]; };
                    float acc;
                    if (Fam::basis_odd(q)) {
                        acc = ctap(q, set, 1) * (w(1) - w(-1));
#pragma unroll
                        for (int i = 2; i <= R; ++i) acc = fmaf(ctap(q, set, i), w(i) - w(-i), acc);
                    } else {
                        acc = ctap(q, set, 0) * w(0);
#pragma unroll
                        for (int i = 1; i <= R; ++i) acc = fmaf(ctap(q, set, i), w(i) + w(-i), acc);
                    }
                    b[px][q] = acc;
                }
            }
        };
        auto shift = [&](auto by_c) {
            constexpr int by = decltype(by_c)::value;
#pragma unroll
            for (int p = 0; p < NROW; ++p)
#pragma unroll
                for (int i = 0; i < W2; ++i)
#pragma unroll
                    for (int px = 0; px < PX; ++px) lw[p][i][px] = lw[p][i + by][px];
        };
        [&]<int... I>(std::integer_sequence<int, I...>) {
            ((row_pass(I), push(std::integral_constant<int, I>{})), ...);
        }(std::make_integer_sequence<int, W2>{});
        int rt = W2;
        // @map kernels: the angle pair of an output row is loaded ONE ROW AHEAD (an L2 hit after the bulk prefetch above), so the
        // load is in flight during the previous row's arithmetic; the last row of the band re-reads its own angles
        const bool maps = Fam::template reads_theta_map<MASK>(a);
        float2 thp = maps ? cur.theta2(a) : make_float2(0.f, 0.f);
        auto one_row = [&](int tile_row, auto pos_c, auto u_c) {
            const float2 thn = maps ? cur.theta2(a, tile_row + 1 < total ? 1 : 0) : thp;
            row_pass(tile_row);
            push(pos_c);
            col_lin(u_c);
            emit_row(thp.x, thp.y);
            thp = thn;
        };
#pragma unroll 1
        for (; rt + U <= total; rt += U) {  // unchecked groups of U output rows: one basic block
            [&]<int... I>(std::integer_sequence<int, I...>) {
                (one_row(rt + I, std::integral_constant<int, W2 + I>{}, std::integral_constant<int, I>{}), ...);
            }(std::make_integer_sequence<int, U>{});
            shift(std::integral_constant<int, U>{});
        }
#pragma unroll 1
        for (; rt < total; ++rt) {  // fewer than U rows left (last band of an image): one row per iteration
            one_row(rt, std::integral_constant<int, W2>{}, std::integral_constant<int, 0>{});
            shift(std::integral_constant<int, 1>{});
        }
        rt_done = total;
    }
    if constexpr (CVS_MARCH_UNROLL_EPILOGUE && MASK != 0 && !Fam::SHARED_ROW_PASS && !SHIFT) {
        // Variant for short epilogues: the whole row body (row pass, column pass, epilogue) is replicated per slot, so the
        // loop needs no slot dispatch at all.  Only worth it while K x (body) still fits the instruction cache.
        // Groups of K rows run WITHOUT per-row bounds checks, i.e. as one basic block that the scheduler can overlap
        // across rows (next row's shared-memory loads under the previous row's epilogue).  BH + 2R is a multiple of K for
        // the G2 family (64 + 8 = 8 x 9), so a full band is exactly group 0 (2R window-filling rows + the first output row)
        // plus whole groups; only the last band of an image leaves a remainder for the rolled loop below.
        static_assert(2 * R == K - 1, "group 0 = 2R pre-roll rows + 1 output row");
        const int total = nrows + 2 * R;
        if (total >= K) {
            [&]<int... I>(std::integer_sequence<int, I...>) {
                ((row_pass(I), col_pass(false, std::integral_constant<int, I>{})), ...);
            }(std::make_integer_sequence<int, 2 * R>{});
            // (the steering-angle load, if this family reads a map, is issued ahead of the row's arithmetic)
            float th0 = Fam::template reads_theta_map<MASK>(a) ? cur.theta(a) : 0.f;
            row_pass(2 * R);
            col_pass(true, std::integral_constant<int, 2 * R>{});
            emit_row(th0);
            rt_done = K;
#pragma unroll 1
            for (; rt_done + K <= total; rt_done += K) {
                [&]<int... I>(std::integer_sequence<int, I...>) {
                    ((th0 = Fam::template reads_theta_map<MASK>(a) ? cur.theta(a) : 0.f, row_pass(rt_done + I),
                      col_pass(true, std::integral_constant<int, I>{}), emit_row(th0)),
                     ...);
                }(std::make_integer_sequence<int, K>{});
            }
        }
    }
    // What bounds this loop: instruction FETCH.  One row walks the slot-independent code (2.7 KB) and one of 2R slot bodies
    // (2.3 KB each for G4), 30 KB per window rotation against a per-scheduler L0 instruction cache of a few KB.  Measured
    // (profiles/experiments/r02_g4_icache_diagnostics.md): with the rows cycling through 1 / 2 / 4 / 12 bodies -- same
    // instructions, branches and memory traffic -- g4 steer@map runs at 112 / 105 / 94 / 88 Gpix/s.  Shifting the window
    // (fewer bodies), phase-locking the warps of a scheduler (three strips per CTA) and straight-line groups of 2R rows
    // were all measured slower; do not expect ALU-side micro-optimisations to show (+-3 instructions per row: no effect).
    constexpr bool PIPE = CVS_MARCH_PIPE && Fam::SHARED_ROW_PASS && MASK != 0 && PX == 1 && !SHIFT;
    if constexpr (PIPE) {
        // 2R-slot window: when the newest row arrives in r[], the rows at offsets -R .. R-1 sit in slots
        // (slot + R + k) mod 2R and the oldest one (k = -R, slot `slot`) is replaced by r[] after the column passes --
        // one row of registers (NROW) and one slot body less than the K-slot window of the other loops.
        constexpr int W = 2 * R;
        float pw[NROW][W];
        auto col_pipe = [&](bool emit, auto slot_c) {
            constexpr int slot = decltype(slot_c)::value;
            if (emit) {
#pragma unroll
                for (int q = 0; q < NB; ++q) {
                    const int rp = Fam::basis_row(q), set = Fam::basis_set(q);
                    auto w = [&](int k) -> float { return k == R ? r[rp][0] : pw[rp][(slot + R + k) % W]; };
                    float acc;
                    if (Fam::basis_odd(q)) {
                        acc = ctap(q, set, 1) * (w(1) - w(-1));
#pragma unroll
                        for (int i = 2; i <= R; ++i) acc = fmaf(ctap(q, set, i), w(i) - w(-i), acc);
                    } else {
                        acc = ctap(q, set, 0) * w(0);
#pragma unroll
                        for (int i = 1; i <= R; ++i) acc = fmaf(ctap(q, set, i), w(i) + w(-i), acc);
                    }
                    b[0][q] = acc;
                }
            }
#pragma unroll
            for (int p = 0; p < NROW; ++p) pw[p][slot] = r[p][0];
        };
        const int total = nrows + 2 * R;  // tile rows to consume; >= 2R + 1
        const bool maps = Fam::template reads_theta_map<MASK>(a);
        // Window-filling rows (nothing to emit): PRE rows at a time go straight-line into the LAST PRE slots, and the window is
        // shifted down by PRE at the top of every trip, so after W / PRE trips tile row j sits in slot j.  No dispatch (a
        // second dispatch tree made ptxas spill the window), and 4 row bodies of code instead of 12: straight-line code
        // that runs once per CTA is always cold in the instruction cache (15 % no_instructions samples with 12 bodies).
        constexpr int PRE = 4;
        static_assert(W % PRE == 0, "pre-roll trips");
#pragma unroll 1
        for (int it = 0; it < W / PRE; ++it) {
#pragma unroll
            for (int p = 0; p < NROW; ++p)
#pragma unroll
                for (int i = 0; i < W - PRE; ++i) pw[p][i] = pw[p][i + PRE];  // (first trip: moves don't-care values)
            [&]<int... I>(std::integer_sequence<int, I...>) {
                ((row_pass(it * PRE + I), col_pipe(false, std::integral_constant<int, W - PRE + I>{})), ...);
            }(std::make_integer_sequence<int, PRE>{});
        }
        int slot = 0;
        float th = maps ? cur.theta(a) : 0.f;
        // cos / sin of the steering angle are computed ONE ROW AHEAD (static map kernels): the angle load and the MUFU latency
        // leave the head of the epilogue's dependent chain (sincos -> weights -> 6-deep FMA chain -> rcp -> atan polynomial)
        float ct = 1.f, st = 0.f;
        if (maps) __sincosf(th, &st, &ct);
        row_pass(W);
#pragma unroll 1
        for (int rt = W; rt < total; ++rt) {
            const bool more = rt + 1 < total;  // CTA-uniform
            // the angle of the NEXT output row (an L2 hit after the prefetch above), in flight during this row's arithmetic
            const float th_next = maps ? cur.theta(a, more ? 1 : 0) : 0.f;
            dispatch_tree<0, W>(slot, [&](auto slot_c) { col_pipe(true, slot_c); });
            slot = (slot + 1 == W) ? 0 : slot + 1;
            // one basic block: epilogue of this output row + row pass of the next tile row (the last iteration recomputes
            // the final row instead of branching around it)
            Fam::template epilogue<MASK, PRESC, true>(b[0], a, cur, th, ct, st);
            cur.next_row();
            row_pass(more ? rt + 1 : rt);
            th = th_next;
            if (maps) __sincosf(th_next, &st, &ct);
        }
        rt_done = total;
    }
    if constexpr (!SHIFT && !PIPE) {
    int slot = 0;  // rt_done is a multiple of K, so the window slot of tile row rt_done is 0 again
    float theta_next = 0.f;
    if (Fam::template reads_theta_map<MASK>(a) && rt_done >= 2 * R && rt_done < nrows + 2 * R) theta_next = cur.theta(a);
#pragma unroll 1
    for (int rt = rt_done; rt < nrows + 2 * R; ++rt) {
        // steering-angle map: the load for an output row is issued ONE ROW AHEAD (during the previous row's arithmetic):
        // measured on G4 steer, issuing it at the top of its own row still left 25 % of warp samples waiting on it
        const float theta_px = theta_next;
        if (Fam::template reads_theta_map<MASK>(a) && rt + 1 >= 2 * R && rt + 1 < nrows + 2 * R)
            theta_next = cur.theta(a, rt >= 2 * R ? 1 : 0);
        if constexpr (Fam::SHARED_ROW_PASS) row_pass(rt);
        dispatch_tree<0, K>(slot, [&](auto slot_c) {
            if constexpr (!Fam::SHARED_ROW_PASS) row_pass(rt);
            col_pass(rt >= 2 * R, slot_c);
        });
        slot = (slot + 1 == K) ? 0 : slot + 1;
        if (rt >= 2 * R) emit_row(theta_px);
    }
    }  // !SHIFT && !PIPE
    if constexpr ((MASK & MARCH_MINMAX_FLAG) != 0) {
        // CTA-wide min / max of the tracked maps: warp reduce on the order-preserving integer image of the floats, combine the
        // warps through shared memory, then ONE atomic pair per map per CTA (same-address atomics serialise in L2).  NaNs
        // never entered (fminf / fmaxf drop them), and a map without any finite value leaves the caller's (0xffffffff, 0)
        // initial pair alone, exactly like k_minmax.
        __shared__ unsigned s_mm[NT / 32][6];
        auto ord = [](float f) { const unsigned u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); };
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const bool any = cur.mn[k] <= cur.mx[k];
            const unsigned lo = __reduce_min_sync(0xffffffffu, any ? ord(cur.mn[k]) : 0xffffffffu);
            const unsigned hi = __reduce_max_sync(0xffffffffu, any ? ord(cur.mx[k]) : 0u);
            if ((threadIdx.x & 31) == 0) s_mm[threadIdx.x >> 5][2 * k] = lo, s_mm[threadIdx.x >> 5][2 * k + 1] = hi;
        }
        __syncthreads();
        if (threadIdx.x < 6) {
            const int k = threadIdx.x >> 1;
            const bool is_max = threadIdx.x & 1;
            unsigned v = s_mm[0][threadIdx.x];
#pragma unroll
            for (int w = 1; w < NT / 32; ++w) v = is_max ? max(v, s_mm[w][threadIdx.x]) : min(v, s_mm[w][threadIdx.x]);
            unsigned* mm = a.minmax + 2 * ((long long)k * a.minmax_frames + frame) + (is_max ? 1 : 0);
            if (is_max) {
                if (v != 0u) atomicMax(mm, v);
            } else if (v != 0xffffffffu) {
                atomicMin(mm, v);
            }
        }
    }
    if (a.pyr_out) emit_next_level<R, BH, NT>(tile, a, frame, x0, yb);  // CTA-uniform; the tile is read-only after staging
}

template <class Fam, unsigned MASK /* 0 = use a.mask at run time */, bool USE_TMA, typename TIn, bool BAKED, int PX = 1, typename TOut = float>
__global__ void __launch_bounds__(MARCH_TW / PX, (PX == 2 && CVS_PX2_MIN_CTAS > 0) ? CVS_PX2_MIN_CTAS : Fam::MIN_CTAS)
k_march(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ MarchArgs a,
        const __grid_constant__ TapTable<Fam::NSETS, Fam::R> taps)
{
    // per-plane base registers only pay off while there are few planes (2 registers each); wide masks share one offset
    // (the same goes for the families whose nine 13-row windows leave no registers to spare: G4)
    using Cursor = OutCursor<((__builtin_popcount(MASK & MARCH_PLANE_BITS) <= CVS_CURSOR_MAX_PLANES && !Fam::SHARED_ROW_PASS) ? MASK : 0u), Fam::NPLANES, TOut>;
    march_body<Fam, MASK, USE_TMA, TIn, BAKED, PX, TOut, Cursor>(tmap, a, taps, a);
}

}  // namespace cvs
