// 16-bit output planes: choice between the fused 16-bit kernels (march_out16.cuh) and the narrowing kernel the fallback
// (capi.cu: fp32 kernel into scratch, then k_narrow) ends with.
#include "march_out16.cuh"

namespace cvs {

// Two 16-bit pixels per thread are one 4-byte store per plane: planes, pitch and frame stride multiples of 4, even width (the
// clamped last pair stays aligned); the fp32 angle pairs stay 8-byte loads (map pitch = 2 x out_pitch).
static bool pair_store16_ok(const BatchGeom& g, const MarchArgs& a)
{
    if ((g.cols & 1) || (g.out_pitch & 3) || (g.out_frame_stride & 3)) return false;
    for (int p = 0; p < MARCH_MAX_OUT; ++p)
        if (a.out[p] && ((uintptr_t)a.out[p] & 3)) return false;
    return !(a.steer_source == CVS_STEER_MAP && ((uintptr_t)a.theta_map & 7));
}

template <class Fam>
static bool default_taps(const FamilyTaps& taps)
{
    TapTable<Fam::NSETS, Fam::R> tt;
    fill_tap_table<Fam>(taps, tt);
    return taps_are_baked<Fam>(tt);
}

cudaError_t launch_basis_fused16(int family, int fmt, const FamilyTaps& taps, const BatchGeom& g, unsigned mask, const SteerSpec& st,
                                 void* const* outs, cudaStream_t stream, LaunchInfo* info, bool* taken)
{
    *taken = false;
    if (fmt != 1 && fmt != 2) return cudaErrorInvalidValue;
    // 8-bit frames take the fused kernels where the fp32-output launch would stage them by TMA (march_launch.cuh); the
    // cooperative `ldg-u8` loader stays on the fallback
    const int px = uses_march_path(family, taps.width) ? out16_kernel_px(family, mask, st.source, g.in_u8) : 0;
    if (!px || !tma_eligible(g, family == 2 ? G2Fam::R : G4Fam::R)) return cudaSuccess;
    if (!(family == 2 ? default_taps<G2Fam>(taps) : default_taps<G4Fam>(taps))) return cudaSuccess;
    const int nplanes = family == 2 ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES;
    const MarchArgs a = make_args(g, mask, st, reinterpret_cast<float* const*>(outs), nplanes);
    if (px == 2 && !pair_store16_ok(g, a)) return cudaSuccess;
    if (g.out_row_end <= g.out_row_begin || g.cols <= 0 || g.n <= 0) return cudaErrorInvalidValue;
    *taken = true;
    // gridDim.z carries the frame index: batches beyond 65535 frames go out as several launches (as launch_basis_fused)
    for (int f0 = 0; f0 < g.n; f0 += 65535) {
        BatchGeom gc = g;
        MarchArgs ac = a;
        gc.n = g.n - f0 < 65535 ? g.n - f0 : 65535;
        gc.in = static_cast<const char*>(g.in) + (size_t)f0 * g.in_frame_stride;
        ac.in = gc.in;
        for (int p = 0; p < MARCH_MAX_OUT; ++p)
            if (ac.out[p]) ac.out[p] = reinterpret_cast<float*>(reinterpret_cast<char*>(a.out[p]) + (size_t)f0 * g.out_frame_stride);
        if (ac.theta_map)  // 4-byte elements in the outputs' element layout
            ac.theta_map = reinterpret_cast<const float*>(reinterpret_cast<const char*>(a.theta_map) + 2 * (size_t)f0 * g.out_frame_stride);
        if (ac.pyr_out) ac.pyr_out = reinterpret_cast<float*>(reinterpret_cast<char*>(a.pyr_out) + (size_t)f0 * g.next_frame_stride);
        cudaError_t e;
        if (family == 2 && g.in_u8)
            e = fmt == 1 ? launch_march_g2_out16<__half, unsigned char>(taps, gc, ac, stream, info)
                         : launch_march_g2_out16<__nv_bfloat16, unsigned char>(taps, gc, ac, stream, info);
        else if (family == 2)
            e = fmt == 1 ? launch_march_g2_out16<__half>(taps, gc, ac, stream, info) : launch_march_g2_out16<__nv_bfloat16>(taps, gc, ac, stream, info);
        else if (g.in_u8)
            e = fmt == 1 ? launch_march_g4_out16<__half, unsigned char>(taps, gc, ac, stream, info)
                         : launch_march_g4_out16<__nv_bfloat16, unsigned char>(taps, gc, ac, stream, info);
        else
            e = fmt == 1 ? launch_march_g4_out16<__half>(taps, gc, ac, stream, info) : launch_march_g4_out16<__nv_bfloat16>(taps, gc, ac, stream, info);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

struct NarrowArgs {
    const float* src[MARCH_MAX_OUT];
    void* dst[MARCH_MAX_OUT];
    long long src_pitch, src_frame_stride, dst_pitch, dst_frame_stride;
    int nplanes, rows, cols;
};

// One fp32 -> 16-bit element per thread and row: 4 bytes read, 2 written, both streaming (HBM-bound).  blockIdx.z = frame x
// plane; rows are grid-strided so that any height fits gridDim.y.
template <typename TOut>
__global__ void __launch_bounds__(256) k_narrow(const __grid_constant__ NarrowArgs a)
{
    const int x = blockIdx.x * 256 + threadIdx.x;
    if (x >= a.cols) return;
    const int p = blockIdx.z % a.nplanes, f = blockIdx.z / a.nplanes;
    const char* s = reinterpret_cast<const char*>(a.src[p]) + f * a.src_frame_stride + 4ll * x;
    char* d = reinterpret_cast<char*>(a.dst[p]) + f * a.dst_frame_stride + 2ll * x;
    for (int y = blockIdx.y; y < a.rows; y += gridDim.y)
        __stcs(reinterpret_cast<unsigned short*>(d + y * a.dst_pitch), to_out16<TOut>(__ldcs(reinterpret_cast<const float*>(s + y * a.src_pitch))));
}

cudaError_t launch_narrow(int fmt, int nplanes, const float* const* src, size_t src_pitch, size_t src_frame_stride, void* const* dst,
                          size_t dst_pitch, size_t dst_frame_stride, int n, int rows, int cols, cudaStream_t stream)
{
    if (nplanes <= 0 || nplanes > MARCH_MAX_OUT || n <= 0 || rows <= 0 || cols <= 0 || (long long)n * nplanes > 65535 || (fmt != 1 && fmt != 2))
        return cudaErrorInvalidValue;
    NarrowArgs a;
    memset(&a, 0, sizeof(a));
    for (int i = 0; i < nplanes; ++i) a.src[i] = src[i], a.dst[i] = dst[i];
    a.src_pitch = (long long)src_pitch, a.src_frame_stride = (long long)src_frame_stride;
    a.dst_pitch = (long long)dst_pitch, a.dst_frame_stride = (long long)dst_frame_stride;
    a.nplanes = nplanes, a.rows = rows, a.cols = cols;
    const dim3 grid((cols + 255) / 256, rows < 65535 ? rows : 65535, n * nplanes);
    if (fmt == 1) k_narrow<__half><<<grid, 256, 0, stream>>>(a);
    else k_narrow<__nv_bfloat16><<<grid, 256, 0, stream>>>(a);
    g_launches.fetch_add(1);
    return cudaGetLastError();
}

// One byte -> fp32 per thread and row (the host-buffer path's 8-bit frames where it must run the fp32-frame kernel).  blockIdx.z
// and the rows are grid-strided so that any batch fits the grid.
__global__ void __launch_bounds__(256) k_widen(const unsigned char* src, long long src_pitch, long long src_frame_stride, float* dst,
                                               long long dst_pitch, long long dst_frame_stride, int n, int rows, int cols)
{
    const int x = blockIdx.x * 256 + threadIdx.x;
    if (x >= cols) return;
    for (int f = blockIdx.z; f < n; f += gridDim.z)
        for (int y = blockIdx.y; y < rows; y += gridDim.y)
            *reinterpret_cast<float*>(reinterpret_cast<char*>(dst) + f * dst_frame_stride + y * dst_pitch + 4ll * x) =
                (float)src[f * src_frame_stride + y * src_pitch + x];
}

cudaError_t launch_widen(const unsigned char* src, size_t src_pitch, size_t src_frame_stride, float* dst, size_t dst_pitch,
                         size_t dst_frame_stride, int n, int rows, int cols, cudaStream_t stream)
{
    if (n <= 0 || rows <= 0 || cols <= 0) return cudaErrorInvalidValue;
    const dim3 grid((cols + 255) / 256, rows < 65535 ? rows : 65535, n < 65535 ? n : 65535);
    k_widen<<<grid, 256, 0, stream>>>(src, (long long)src_pitch, (long long)src_frame_stride, dst, (long long)dst_pitch,
                                      (long long)dst_frame_stride, n, rows, cols);
    g_launches.fetch_add(1);
    return cudaGetLastError();
}

}  // namespace cvs
