// 16-bit output planes without a fused 16-bit kernel (capi.cu: fp32 kernel into scratch, then k_narrow), and 8-bit frames
// widened to fp32 for the host-buffer path.
#include "march_launch.cuh"

namespace cvs {

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
