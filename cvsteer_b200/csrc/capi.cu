// C ABI of libcvsteer_b200.so (include/cvsteer_c.h).  Host-side state lives here: tap tables, the resident
// class state of a set-up image, streams, staging.  All arithmetic on pixels happens in CUDA kernels; there
// is no CPU fallback anywhere in this file.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <new>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "../../include/cvsteer_c.h"
#include "internal.h"
#include "launch.h"
#include "taps.h"

using namespace cvs;
using namespace cvsi;

#define MARCH_MAX_OUT_HOST 32

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int cvsi::fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
using cvsi::fail;

extern "C" const char* cvs_version(void) { return "cvsteer_b200 0.2.0 (sm_100a)"; }
extern "C" const char* cvs_last_error(void) { return g_err; }

extern "C" int cvs_device_count(int* count)
{
    if (!count) return fail(CVS_ERR_INVALID_ARG, "count is null");
    CU_TRY(cudaGetDeviceCount(count));
    return CVS_OK;
}

extern "C" int cvs_enable_peer_access(int device, int peer_device)
{
    if (device == peer_device) return CVS_OK;
    int can = 0;
    CU_TRY(cudaDeviceCanAccessPeer(&can, device, peer_device));
    if (!can) return fail(CVS_ERR_CUDA, "device %d has no peer path to device %d", device, peer_device);
    CU_TRY(cudaSetDevice(device));
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer_device, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();  // not an error: someone (torch, NCCL, an earlier call) enabled it already
        return CVS_OK;
    }
    CU_TRY(e);
    return CVS_OK;
}

static_assert(sizeof(cudaIpcMemHandle_t) == CVS_IPC_HANDLE_BYTES, "IPC handle size");
extern "C" int cvs_shared_alloc(int device, size_t bytes, void** ptr, unsigned char handle[CVS_IPC_HANDLE_BYTES])
{
    if (!ptr || !handle || !bytes) return fail(CVS_ERR_INVALID_ARG, "null argument");
    CU_TRY(cudaSetDevice(device));
    void* p = nullptr;
    CU_TRY(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    const cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        CU_TRY(e);
    }
    memcpy(handle, &h, sizeof(h));
    *ptr = p;
    return CVS_OK;
}
extern "C" int cvs_shared_open(int device, const unsigned char handle[CVS_IPC_HANDLE_BYTES], void** ptr)
{
    if (!ptr || !handle) return fail(CVS_ERR_INVALID_ARG, "null argument");
    CU_TRY(cudaSetDevice(device));  // the IMPORTER's GPU: the mapping (and the peer path to the owner) is made for it
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    CU_TRY(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return CVS_OK;
}
extern "C" int cvs_shared_close(int device, void* ptr)
{
    if (!ptr) return CVS_OK;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaIpcCloseMemHandle(ptr));
    return CVS_OK;
}
extern "C" int cvs_shared_free(int device, void* ptr)
{
    if (!ptr) return CVS_OK;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(cudaFree(ptr));
    return CVS_OK;
}

extern "C" int cvs_g2_make_taps(int which, int width, float spacing, float* dst)
{
    if (which < 0 || which >= G2_NUM_TAPSETS || width < 1 || width > MAX_WIDTH || !dst)
        return fail(CVS_ERR_INVALID_ARG, "cvs_g2_make_taps: which=%d width=%d", which, width);
    make_taps_g2(which, width, spacing, dst);
    return CVS_OK;
}

extern "C" int cvs_g4_make_taps(int which, int width, float spacing, float* dst)
{
    if (which < 0 || which >= G4_NUM_TAPSETS || width < 1 || width > MAX_WIDTH || !dst)
        return fail(CVS_ERR_INVALID_ARG, "cvs_g4_make_taps: which=%d width=%d", which, width);
    make_taps_g4(which, width, spacing, dst);
    return CVS_OK;
}

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
namespace cvsi {


int filter_create(Filter** out, int family, int device, int width, float spacing)
{
    if (!out) return fail(CVS_ERR_INVALID_ARG, "out is null");
    *out = nullptr;
    if (width < 1 || width > MAX_WIDTH) return fail(CVS_ERR_INVALID_ARG, "width %d outside [1, %d]", width, (int)MAX_WIDTH);
    int ndev = 0;
    CU_TRY(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) return fail(CVS_ERR_INVALID_ARG, "device %d of %d", device, ndev);
    Filter* f = new (std::nothrow) Filter();
    if (!f) return fail(CVS_ERR_CUDA, "out of host memory");
    f->family = family;
    f->device = device;
    f->taps.width = width;
    f->taps.nsets = family == 2 ? (int)G2_NUM_TAPSETS : (int)G4_NUM_TAPSETS;
    memset(f->taps.t, 0, sizeof(f->taps.t));
    for (int s = 0; s < f->taps.nsets; ++s) {
        if (family == 2) make_taps_g2(s, width, spacing, f->taps.t[s]);
        else make_taps_g4(s, width, spacing, f->taps.t[s]);
    }
    f->nstate = family == 2 ? 12 : 13;  // G4: 11 basis planes + lazily computed theta_d / strength
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&f->stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete f;
        return fail(CVS_ERR_CUDA, "stream create: %s", cudaGetErrorString(e));
    }
    *out = f;
    return CVS_OK;
}

int filter_destroy(Filter* f)
{
    if (!f) return CVS_OK;
    cudaSetDevice(f->device);
    if (f->stream) {
        cudaStreamSynchronize(f->stream);
        cudaStreamDestroy(f->stream);
    }
    for (cudaStream_t& s : f->pipe)
        if (s) {
            cudaStreamSynchronize(s);
            cudaStreamDestroy(s);
            s = nullptr;
        }
    if (f->scratch_ev) cudaEventDestroy(f->scratch_ev);
    f->in.release();
    f->state.release();
    f->work.release();
    f->scratch.release();
    delete f;
    return CVS_OK;
}

BatchGeom whole_frame_geom(const void* in, bool u8, int n, int rows, int cols, size_t in_pitch, size_t in_fs, size_t out_pitch,
                           size_t out_fs)
{
    BatchGeom g{};
    g.in = in;
    g.in_u8 = u8;
    g.n = n;
    g.cols = cols;
    g.buf_rows = rows;
    g.full_rows = rows;
    g.y_origin = 0;
    g.out_row_begin = 0;
    g.out_row_end = rows;
    g.out_row_origin = 0;
    g.in_pitch = in_pitch;
    g.in_frame_stride = in_fs;
    g.out_pitch = out_pitch;
    g.out_frame_stride = out_fs;
    return g;
}

// out_esz: bytes per output element (4 = fp32 planes, 2 = 16-bit planes)
int geom_from_batch(const cvs_batch* b, BatchGeom* g, size_t out_esz = 4)
{
    if (!b || !b->in) return fail(CVS_ERR_INVALID_ARG, "batch or batch->in is null");
    if (b->n <= 0 || b->rows <= 0 || b->cols <= 0) return fail(CVS_ERR_INVALID_ARG, "batch n/rows/cols must be positive");
    const size_t esz = b->in_is_u8 ? 1 : 4;
    if (b->in_pitch < (size_t)b->cols * esz) return fail(CVS_ERR_INVALID_ARG, "in_pitch %zu < cols*%zu", b->in_pitch, esz);
    if (b->out_pitch < (size_t)b->cols * 4 / 2) return fail(CVS_ERR_INVALID_ARG, "out_pitch too small");
    if ((b->out_pitch & (out_esz - 1)) || (b->out_frame_stride & (out_esz - 1)) ||
        (!b->in_is_u8 && ((b->in_pitch & 3) || (b->in_frame_stride & 3) || ((uintptr_t)b->in & 3))))
        return fail(CVS_ERR_INVALID_ARG, out_esz == 4 ? "fp32 planes need 4-byte aligned base, pitch and frame stride"
                                                      : "16-bit output planes need an even pitch and frame stride, fp32 input 4-byte alignment");
    *g = whole_frame_geom(b->in, b->in_is_u8 != 0, b->n, b->rows, b->cols, b->in_pitch, b->in_frame_stride, b->out_pitch,
                          b->out_frame_stride);
    if (b->next_level) {
        if (b->full_rows > 0) return fail(CVS_ERR_UNSUPPORTED, "next_level fusion is for whole frames; bands use cvs_pyr_down_dev");
        if (b->next_pitch < (size_t)((b->cols + 1) / 2) * 4) return fail(CVS_ERR_INVALID_ARG, "next_pitch too small");
        g->next_level = b->next_level;
        g->next_pitch = b->next_pitch;
        g->next_frame_stride = b->next_frame_stride;
    }
    if (b->full_rows > 0) {
        g->full_rows = b->full_rows;
        g->y_origin = b->y_origin;
        g->out_row_begin = b->out_row_begin;
        g->out_row_end = b->out_row_end;
        g->out_row_origin = b->out_row_origin;
        if (g->y_origin < 0 || g->y_origin + g->buf_rows > g->full_rows)
            return fail(CVS_ERR_INVALID_ARG, "band buffer rows [%d,%d) outside image of %d rows", g->y_origin, g->y_origin + g->buf_rows,
                        g->full_rows);
    }
    return CVS_OK;
}

// The band contract: the buffer must hold every image row the requested output rows read, i.e. rows
// [need_lo, need_hi) = the filter footprint of [out_row_begin, out_row_end) clipped to the image (reflect-101 only ever
// folds back INTO that clipped interval).  stride = 1: a (2*radius+1)-tap filter at the same level; stride = 2: pyr_down,
// whose output row y reads input rows 2y-2 .. 2y+2.  A violation would not fault (the loaders clamp) but silently
// filter zeros, so it is an argument error.
int check_band(const BatchGeom& g, int radius, int full_rows_out_level, int stride = 1)
{
    if (g.out_row_begin < 0 || g.out_row_end > full_rows_out_level || g.out_row_begin >= g.out_row_end)
        return fail(CVS_ERR_INVALID_ARG, "output rows [%d,%d) invalid", g.out_row_begin, g.out_row_end);
    const long long lo = (long long)stride * g.out_row_begin - radius, hi = (long long)stride * (g.out_row_end - 1) + radius + 1;
    const long long need_lo = lo < 0 ? 0 : lo, need_hi = hi > g.full_rows ? g.full_rows : hi;
    if (g.y_origin > need_lo || (long long)g.y_origin + g.buf_rows < need_hi)
        return fail(CVS_ERR_INVALID_ARG, "band buffer holds image rows [%d,%d) but output rows [%d,%d) need [%lld,%lld)", g.y_origin,
                    g.y_origin + g.buf_rows, g.out_row_begin, g.out_row_end, need_lo, need_hi);
    return CVS_OK;
}

// `slot` of `nslots`: callers that keep several launches in flight on different streams (the host-batch pipelines) give
// each stream its own slice of the generic-width scratch; the per-frame scratch size does not depend on the chunk.
int run_fused(Filter* f, const BatchGeom& g, unsigned mask, const SteerSpec& st, float* const* outs, cudaStream_t stream, int slot, int nslots)
{
    CU_TRY(cudaSetDevice(f->device));
    float* scratch = nullptr;
    if (!uses_march_path(f->family, f->taps.width)) {
        const size_t per = align_up(scratch_bytes_generic(f->family, g), 256);
        CU_TRY(f->scratch.reserve(per * (size_t)nslots));  // growing frees the old block: cudaFree waits for kernels still using it
        scratch = reinterpret_cast<float*>(static_cast<char*>(f->scratch.p) + per * (size_t)slot);
        // the same slice used from another stream than last time: order the two streams (device-side, no host wait)
        if (slot < 3 && f->scratch_used[slot] && f->scratch_stream[slot] != stream) {
            if (!f->scratch_ev) CU_TRY(cudaEventCreateWithFlags(&f->scratch_ev, cudaEventDisableTiming));
            cudaError_t e = cudaEventRecord(f->scratch_ev, f->scratch_stream[slot]);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, f->scratch_ev, 0);
            if (e != cudaSuccess) {  // e.g. the caller destroyed the earlier stream: fall back to a full device sync
                cudaGetLastError();
                CU_TRY(cudaDeviceSynchronize());
            }
        }
        if (slot < 3) f->scratch_used[slot] = true, f->scratch_stream[slot] = stream;
    }
    CU_TRY(launch_basis_fused(f->family, f->taps, g, mask, st, outs, scratch, stream, &f->last));
    return CVS_OK;
}

// run_fused with output planes in `fmt` (cvs_out_format; g.out_pitch / g.out_frame_stride in bytes of them).  The fused 16-bit
// kernel when one exists for this launch; otherwise the fp32 kernel writes stream-ordered scratch in the angle map's layout
// (4-byte elements, twice the outputs' pitch and frame stride, so CVS_STEER_MAP works unchanged), chunked by frames to bound
// its size, and k_narrow rounds it into the caller's planes: the same bits either way.
int run_fused_fmt(Filter* f, const BatchGeom& g, unsigned mask, const SteerSpec& st, void* const* outs, int fmt, cudaStream_t stream, int slot = 0,
                  int nslots = 1)
{
    if (fmt == CVS_OUT_F32) return run_fused(f, g, mask, st, reinterpret_cast<float* const*>(outs), stream, slot, nslots);
    CU_TRY(cudaSetDevice(f->device));
    bool taken = false;
    CU_TRY(launch_basis_fused16(f->family, fmt, f->taps, g, mask, st, outs, stream, &f->last, &taken));
    if (taken) return CVS_OK;
    const int nplanes = f->family == 2 ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES;
    int sel[MARCH_MAX_OUT_HOST], np = 0;
    for (int p = 0; p < nplanes; ++p)
        if (mask >> p & 1u) sel[np++] = p;
    const int rows = g.out_row_end - g.out_row_begin;
    if (np == 0 || rows <= 0) return fail(CVS_ERR_INVALID_ARG, "empty launch");
    const size_t s_pitch = 2 * g.out_pitch, s_fs = g.n > 1 ? 2 * g.out_frame_stride : s_pitch * rows;
    const size_t budget = 512ull << 20;  // scratch bytes per call (at least one frame)
    int chunk = (int)std::min<size_t>((size_t)g.n, std::max<size_t>(1, budget / (s_fs * np)));
    chunk = std::min(chunk, 65535 / np);  // k_narrow: frames x planes in gridDim.z
    const size_t plane_bytes = (size_t)(chunk - 1) * s_fs + s_pitch * rows;
    void* scratch = nullptr;
    CU_TRY(cudaMallocAsync(&scratch, plane_bytes * np, stream));
    int rc = CVS_OK;
    for (int f0 = 0; f0 < g.n && rc == CVS_OK; f0 += chunk) {
        const int nf = std::min(chunk, g.n - f0);
        BatchGeom gc = g;
        gc.n = nf;
        gc.in = static_cast<const char*>(g.in) + (size_t)f0 * g.in_frame_stride;
        gc.out_pitch = s_pitch, gc.out_frame_stride = s_fs;
        if (g.next_level) gc.next_level = reinterpret_cast<float*>(reinterpret_cast<char*>(g.next_level) + (size_t)f0 * g.next_frame_stride);
        SteerSpec sc = st;
        if (sc.theta_map) sc.theta_map = reinterpret_cast<const float*>(reinterpret_cast<const char*>(st.theta_map) + (size_t)f0 * s_fs);
        float* souts[MARCH_MAX_OUT_HOST] = {nullptr};
        const float* src[MARCH_MAX_OUT_HOST];
        void* dst[MARCH_MAX_OUT_HOST];
        for (int i = 0; i < np; ++i) {
            souts[sel[i]] = reinterpret_cast<float*>(static_cast<char*>(scratch) + (size_t)i * plane_bytes);
            src[i] = souts[sel[i]];
            dst[i] = static_cast<char*>(outs[sel[i]]) + (size_t)f0 * g.out_frame_stride;
        }
        rc = run_fused(f, gc, mask, sc, souts, stream, slot, nslots);
        if (rc == CVS_OK) {
            const cudaError_t e = launch_narrow(fmt, np, src, s_pitch, s_fs, dst, g.out_pitch, g.out_frame_stride, nf, rows, g.cols, stream);
            if (e != cudaSuccess) rc = fail(CVS_ERR_CUDA, "narrow: %s", cudaGetErrorString(e));
        }
    }
    const cudaError_t e = cudaFreeAsync(scratch, stream);
    if (rc != CVS_OK) return rc;
    CU_TRY(e);
    const size_t len = strlen(f->last.name);
    snprintf(f->last.name + len, sizeof(f->last.name) - len, "+narrow-%s", fmt == CVS_OUT_F16 ? "f16" : "bf16");
    return CVS_OK;
}

// Steering bank (cvs_g2_steer_bank_dev / cvs_g4_steer_bank_dev): the family's fused bank kernel when its forms apply, otherwise
// the calls the contract names, with the planes they write but the caller did not select in stream-ordered scratch of the
// caller's layout.  Both give the same bits.
//   G2: one STEER5 launch per scalar angle and one ORIENT launch at theta_d when theta_d or strength is wanted.
//   G4: one STEER launch per scalar angle, on the frames widened to fp32 when they are 8-bit (the contract's reference: the
//       8-bit single-angle kernels with fp32 planes do not prescale their taps, see run_batch_host's `widen`).
int run_bank(Filter* f, const BatchGeom& g, const BankSpec& bk, int fmt, cudaStream_t stream, int slot = 0, int nslots = 1)
{
    CU_TRY(cudaSetDevice(f->device));
    const bool g4 = f->family == 4;
    bool taken = false;
    CU_TRY((g4 ? launch_g4_bank : launch_g2_bank)(fmt, f->taps, g, bk, stream, &f->last, &taken));
    if (taken) return CVS_OK;
    const unsigned per_angle = g4 ? (unsigned)CVS_G4_MASK_STEER : (unsigned)CVS_G2_MASK_STEER5;
    const unsigned orient_bits = g4 ? 0u : CVS_BIT(CVS_THETA) | CVS_BIT(CVS_STRENGTH);
    const bool steer = (bk.mask & per_angle) != 0, orient = (bk.mask & orient_bits) != 0;
    unsigned scr = 0;  // planes written to scratch: G2's E of the ORIENT launch always (the caller's E planes hold E(theta_k))
    if (steer) scr |= per_angle & ~bk.mask;
    if (orient) scr |= CVS_G2_MASK_ORIENT & ~(bk.mask & orient_bits);
    const size_t set_bytes = (size_t)(g.n - 1) * g.out_frame_stride + (size_t)(g.out_row_end - g.out_row_begin) * g.out_pitch;
    void* scratch = nullptr;
    if (scr) CU_TRY(cudaMallocAsync(&scratch, set_bytes * __builtin_popcount(scr), stream));
    void* so[CVS_G2_NPLANES] = {nullptr};
    for (int q = 0, i = 0; q < CVS_G2_NPLANES; ++q)
        if (scr >> q & 1u) so[q] = static_cast<char*>(scratch) + (size_t)(i++) * set_bytes;
    auto pick = [&](int q, size_t off) -> void* { return (bk.mask >> q & 1u) ? static_cast<char*>(bk.outs[q]) + off : so[q]; };
    char first[sizeof(f->last.name)] = "";
    BatchGeom gk = g;
    int rc = CVS_OK;
    void* wide = nullptr;  // G4, 8-bit frames: the buffer rows widened to dense fp32 frames (the layout of x.float())
    if (g4 && g.in_u8) {
        const size_t wpitch = (size_t)g.cols * 4, wfs = wpitch * (size_t)g.buf_rows;
        if (cudaError_t e = cudaMallocAsync(&wide, wfs * (size_t)g.n, stream); e != cudaSuccess) {
            if (scr) cudaFreeAsync(scratch, stream);
            CU_TRY(e);
        }
        const cudaError_t e = launch_widen(static_cast<const unsigned char*>(g.in), g.in_pitch, g.in_frame_stride, static_cast<float*>(wide), wpitch,
                                           wfs, g.n, g.buf_rows, g.cols, stream);
        if (e != cudaSuccess) rc = fail(CVS_ERR_CUDA, "widen: %s", cudaGetErrorString(e));
        gk.in = wide, gk.in_u8 = false, gk.in_pitch = wpitch, gk.in_frame_stride = wfs;
    }
    for (int k = 0; steer && k < bk.n_angles && rc == CVS_OK; ++k) {
        void* outs[CVS_G2_NPLANES] = {nullptr};
        for (int q = 0; q < CVS_G2_NPLANES; ++q)
            if (per_angle >> q & 1u) outs[q] = pick(q, (size_t)k * bk.angle_stride);
        SteerSpec st{};
        st.source = CVS_STEER_SCALAR;
        st.cos_t = bk.cos_t[k];
        st.sin_t = bk.sin_t[k];
        rc = run_fused_fmt(f, gk, per_angle, st, outs, fmt, stream, slot, nslots);
        if (!first[0]) snprintf(first, sizeof(first), "%s", f->last.name);
        gk.next_level = nullptr;  // the first launch emitted it
    }
    if (orient && rc == CVS_OK) {
        void* outs[CVS_G2_NPLANES] = {nullptr};
        outs[CVS_THETA] = pick(CVS_THETA, 0), outs[CVS_STRENGTH] = pick(CVS_STRENGTH, 0), outs[CVS_E] = so[CVS_E];
        SteerSpec st{};
        st.source = CVS_STEER_DOMINANT;
        rc = run_fused_fmt(f, gk, CVS_G2_MASK_ORIENT, st, outs, fmt, stream, slot, nslots);
        if (!first[0]) snprintf(first, sizeof(first), "%s", f->last.name);
    }
    const cudaError_t ew = wide ? cudaFreeAsync(wide, stream) : cudaSuccess;
    const cudaError_t e = scr ? cudaFreeAsync(scratch, stream) : cudaSuccess;
    if (rc != CVS_OK) return rc;
    CU_TRY(ew);
    CU_TRY(e);
    snprintf(f->last.name, sizeof(f->last.name), "bank-fallback:%s", first);
    return CVS_OK;
}

int filter_setup(Filter* f, const void* image, bool u8, int rows, int cols, size_t step)
{
    if (!f) return fail(CVS_ERR_INVALID_ARG, "handle is null");
    if (!image || rows <= 0 || cols <= 0) return fail(CVS_ERR_INVALID_ARG, "empty image (%p, %dx%d)", image, rows, cols);
    const size_t esz = u8 ? 1 : 4;
    if (step < (size_t)cols * esz) return fail(CVS_ERR_INVALID_ARG, "step %zu < cols*%zu", step, esz);
    CU_TRY(cudaSetDevice(f->device));
    f->ready = false;
    f->g4_orient_ready = false;
    f->rows = rows;
    f->cols = cols;
    f->pitch = align_up((size_t)cols * 4, 128);
    const size_t in_pitch = u8 ? align_up((size_t)cols, 128) : f->pitch;
    CU_TRY(f->in.reserve(in_pitch * rows));
    CU_TRY(f->state.reserve(f->pitch * rows * (size_t)f->nstate));
    CU_TRY(cudaMemcpy2DAsync(f->in.p, in_pitch, image, step, (size_t)cols * esz, rows, cudaMemcpyHostToDevice, f->stream));
    BatchGeom g = whole_frame_geom(f->in.p, u8, 1, rows, cols, in_pitch, in_pitch * rows, f->pitch, f->pitch * rows);
    float* outs[MAX_TAPS] = {nullptr};
    for (int i = 0; i < (f->family == 2 ? 12 : 11); ++i) outs[i] = f->state_plane(i);
    SteerSpec st{};
    st.source = CVS_STEER_DOMINANT;
    const unsigned mask = f->family == 2 ? CVS_G2_MASK_STATE : CVS_G4_MASK_BASIS;
    int rc = run_fused(f, g, mask, st, outs, f->stream);
    if (rc) return rc;
    CU_TRY(cudaStreamSynchronize(f->stream));  // the caller may free `image` as soon as setup() returns
    f->ready = true;
    return CVS_OK;
}

int download(Filter* f, const float* dplane, float* dst, size_t step)
{
    if (!dst) return CVS_OK;
    if (step < (size_t)f->cols * 4) return fail(CVS_ERR_INVALID_ARG, "dst step %zu < cols*4", step);
    CU_TRY(cudaMemcpy2DAsync(dst, step, dplane, f->pitch, (size_t)f->cols * 4, f->rows, cudaMemcpyDeviceToHost, f->stream));
    return CVS_OK;
}

// G4 only: theta_d / strength are not part of the reference's setup(); computed on first use from the resident basis
int ensure_g4_orientation(Filter* f)
{
    if (f->family != 4 || f->g4_orient_ready) return CVS_OK;
    PlaneSet ps{};
    for (int i = 0; i < 11; ++i) ps.p[i] = f->state_plane(i);
    ps.pitch = f->pitch;
    CU_TRY(launch_g4_orient_planes(ps, f->rows, f->cols, f->state_plane(11), f->state_plane(12), f->pitch, f->stream));
    f->g4_orient_ready = true;
    return CVS_OK;
}

int filter_get_plane(Filter* f, int plane, float* dst, size_t step)
{
    if (!f || !dst) return fail(CVS_ERR_INVALID_ARG, "null argument");
    if (!f->ready) return fail(CVS_ERR_NOT_SETUP, "get_plane before setup");
    CU_TRY(cudaSetDevice(f->device));
    if (f->family == 4 && (plane == CVS_G4_THETA || plane == CVS_G4_STRENGTH)) {
        int rc = ensure_g4_orientation(f);
        if (rc) return rc;
        plane = plane == CVS_G4_THETA ? 11 : 12;
    } else if (f->family == 4 && plane >= 11) {
        return fail(CVS_ERR_INVALID_ARG, "plane %d not part of the class state", plane);
    }
    if (plane < 0 || plane >= f->nstate) return fail(CVS_ERR_INVALID_ARG, "plane %d not part of the class state", plane);
    int rc = download(f, f->state_plane(plane), dst, step);
    if (rc) return rc;
    CU_TRY(cudaStreamSynchronize(f->stream));
    return CVS_OK;
}

// steer on the stored planes.  outs_host indexed by family plane id; theta host map optional.
int filter_steer(Filter* f, int source, float theta, const float* theta_host, size_t theta_step, unsigned mask, float* const* outs_host,
                 size_t step)
{
    if (!f) return fail(CVS_ERR_INVALID_ARG, "handle is null");
    if (!f->ready) return fail(CVS_ERR_NOT_SETUP, "steer before setup");
    CU_TRY(cudaSetDevice(f->device));
    const int nplanes = f->family == 2 ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES;
    const size_t plane_bytes = f->pitch * f->rows;
    CU_TRY(f->work.reserve(plane_bytes * 6));  // 5 outputs + an uploaded theta map
    SteerSpec st{};
    st.source = source;
    float c2t = 0.f, s2t = 0.f;
    size_t th_pitch = f->pitch;
    if (source == CVS_STEER_SCALAR) {
        // the reference evaluates std::cos/std::sin on the float angle on the host (G2.cpp:140, G4.cpp:116) and
        // cos/sin of (theta * 2.0) in double (G2.cpp:163)
        st.cos_t = std::cos(theta);
        st.sin_t = std::sin(theta);
        c2t = (float)std::cos(theta * 2.0);
        s2t = (float)std::sin(theta * 2.0);
    } else if (theta_host) {
        if (theta_step < (size_t)f->cols * 4) return fail(CVS_ERR_SIZE_MISMATCH, "theta step %zu < cols*4", theta_step);
        CU_TRY(cudaMemcpy2DAsync(f->work_plane(5), f->pitch, theta_host, theta_step, (size_t)f->cols * 4, f->rows, cudaMemcpyHostToDevice,
                                 f->stream));
        st.theta_map = f->work_plane(5);
    } else {
        if (f->family == 4) {  // extension: the reference never assigns G4's m_theta (G4.h:40-41); see CVS_G4_THETA
            int rc = ensure_g4_orientation(f);
            if (rc) return rc;
        }
        st.theta_map = f->state_plane(f->family == 2 ? (int)CVS_THETA : 11);  // steer(getDominantOrientationAngle(), ...) without a round trip
    }
    float* outs_dev[MARCH_MAX_OUT_HOST] = {nullptr};
    int slot = 0;
    for (int p = 0; p < nplanes; ++p)
        if (mask >> p & 1u) outs_dev[p] = f->work_plane(slot++);
    if (slot > 5) return fail(CVS_ERR_INVALID_ARG, "too many steer outputs");
    PlaneSet ps{};
    for (int i = 0; i < (f->family == 2 ? 12 : 11); ++i) ps.p[i] = f->state_plane(i);
    ps.pitch = f->pitch;
    if (f->family == 2)
        CU_TRY(launch_g2_steer_planes(ps, f->rows, f->cols, st, c2t, s2t, th_pitch, mask, outs_dev, f->pitch, f->stream));
    else
        CU_TRY(launch_g4_steer_planes(ps, f->rows, f->cols, st, th_pitch, mask, outs_dev, f->pitch, f->stream));
    for (int p = 0; p < nplanes; ++p)
        if (mask >> p & 1u) {
            int rc = download(f, outs_dev[p], outs_host[p], step);
            if (rc) return rc;
        }
    CU_TRY(cudaStreamSynchronize(f->stream));
    return CVS_OK;
}

}  // namespace cvsi

// cvs_g2 / cvs_g4 are opaque to callers; both are a Filter underneath.

// ================================ G2 ================================
extern "C" int cvs_g2_create(cvs_g2** out, int device, int width, float spacing)
{
    return filter_create(reinterpret_cast<Filter**>(out), 2, device, width, spacing);
}
extern "C" int cvs_g2_destroy(cvs_g2* h) { return filter_destroy(reinterpret_cast<Filter*>(h)); }
extern "C" int cvs_g2_setup_host(cvs_g2* h, const float* image, int rows, int cols, size_t step)
{
    return filter_setup(reinterpret_cast<Filter*>(h), image, false, rows, cols, step);
}
extern "C" int cvs_g2_setup_host_u8(cvs_g2* h, const uint8_t* image, int rows, int cols, size_t step)
{
    return filter_setup(reinterpret_cast<Filter*>(h), image, true, rows, cols, step);
}
extern "C" int cvs_g2_size(const cvs_g2* h, int* rows, int* cols)
{
    if (!h) return fail(CVS_ERR_INVALID_ARG, "handle is null");
    const Filter* f = reinterpret_cast<const Filter*>(h);
    if (rows) *rows = f->ready ? f->rows : 0;
    if (cols) *cols = f->ready ? f->cols : 0;
    return CVS_OK;
}
extern "C" int cvs_g2_get_plane_host(cvs_g2* h, int plane, float* dst, size_t step)
{
    return filter_get_plane(reinterpret_cast<Filter*>(h), plane, dst, step);
}

static unsigned g2_steer_mask(float* g2, float* h2, float* e, float* mag, float* phase)
{
    return (g2 ? CVS_BIT(CVS_G2T) : 0u) | (h2 ? CVS_BIT(CVS_H2T) : 0u) | (e ? CVS_BIT(CVS_E) : 0u) | (mag ? CVS_BIT(CVS_MAG) : 0u) |
           (phase ? CVS_BIT(CVS_PHASE) : 0u);
}

extern "C" int cvs_g2_steer_scalar_host(cvs_g2* h, float theta, float* g2, float* h2, float* e, float* magnitude, float* phase, size_t step)
{
    float* outs[CVS_G2_NPLANES] = {nullptr};
    outs[CVS_G2T] = g2, outs[CVS_H2T] = h2, outs[CVS_E] = e, outs[CVS_MAG] = magnitude, outs[CVS_PHASE] = phase;
    return filter_steer(reinterpret_cast<Filter*>(h), CVS_STEER_SCALAR, theta, nullptr, 0, g2_steer_mask(g2, h2, e, magnitude, phase), outs, step);
}

extern "C" int cvs_g2_steer_map_host(cvs_g2* h, const float* theta, size_t theta_step, float* g2, float* h2, float* e, float* magnitude,
                                     float* phase, size_t step)
{
    float* outs[CVS_G2_NPLANES] = {nullptr};
    outs[CVS_G2T] = g2, outs[CVS_H2T] = h2, outs[CVS_E] = e, outs[CVS_MAG] = magnitude, outs[CVS_PHASE] = phase;
    return filter_steer(reinterpret_cast<Filter*>(h), CVS_STEER_MAP, 0.f, theta, theta_step, g2_steer_mask(g2, h2, e, magnitude, phase), outs,
                        step);
}

extern "C" int cvs_g2_steer_point(cvs_g2* h, int x, int y, float theta, float out[5])
{
    Filter* f = reinterpret_cast<Filter*>(h);
    if (!f || !out) return fail(CVS_ERR_INVALID_ARG, "null argument");
    if (!f->ready) return fail(CVS_ERR_NOT_SETUP, "steer before setup");
    if (x < 0 || y < 0 || x >= f->cols || y >= f->rows) return fail(CVS_ERR_INVALID_ARG, "point (%d,%d) outside %dx%d", x, y, f->cols, f->rows);
    CU_TRY(cudaSetDevice(f->device));
    // Fetch the 10 state values of this pixel (7 basis, c1..c3): element (y,x) of 10 consecutive planes = one strided copy.
    float v[10];
    const char* src = reinterpret_cast<const char*>(f->state.p) + (size_t)y * f->pitch + (size_t)x * 4;
    const size_t plane_bytes = f->pitch * f->rows;
    if (plane_bytes < (1ull << 31)) {  // cudaMemcpy2D pitches are limited to 2 GiB (cudaDeviceProp::memPitch)
        CU_TRY(cudaMemcpy2DAsync(v, 4, src, plane_bytes, 4, 10, cudaMemcpyDeviceToHost, f->stream));
    } else {
        for (int i = 0; i < 10; ++i) CU_TRY(cudaMemcpyAsync(&v[i], src + (size_t)i * plane_bytes, 4, cudaMemcpyDeviceToHost, f->stream));
    }
    CU_TRY(cudaStreamSynchronize(f->stream));
    // The per-point overloads are host code in the reference as well (G2.cpp:115-134): a handful of scalar flops on
    // values read from the Mats.  Same expressions, same types.
    float ct(std::cos(theta)), ct2(ct * ct), ct3(ct2 * ct), st(std::sin(theta)), st2(st * st), st3(st2 * st);
    float ga(ct2), gb(-2.0 * ct * st), gc(st2);
    float ha(ct3), hb(-3.0 * ct2 * st), hc(3.0 * ct * st2), hd(-st3);
    const float g2 = ga * v[0] + gb * v[1] + gc * v[2];
    const float h2 = ha * v[3] + hb * v[4] + hc * v[5] + hd * v[6];
    float c2t(std::cos(theta * 2.0)), s2t(std::sin(theta * 2.0));
    out[0] = g2;
    out[1] = h2;
    out[2] = v[7] + (c2t * v[8]) + (s2t * v[9]);
    out[3] = std::sqrt(h2 * h2 + g2 * g2);
    out[4] = std::atan2(h2, g2);
    return CVS_OK;
}

// ================================ stateless point-wise ops ================================
namespace {
struct TempDev {  // small RAII helper for the stateless host entry points
    void* p = nullptr;
    ~TempDev()
    {
        if (p) cudaFree(p);
    }
};
}  // namespace

static int pointwise_host(int device, int op, int kind, const float* a, const float* b, size_t in_step, float* o1, float* o2, size_t out_step,
                          int rows, int cols, float phi, int signum)
{
    if (rows <= 0 || cols <= 0) return fail(CVS_ERR_INVALID_ARG, "empty image");
    if (in_step < (size_t)cols * 4 || out_step < (size_t)cols * 4) return fail(CVS_ERR_INVALID_ARG, "step < cols*4");
    CU_TRY(cudaSetDevice(device));
    const size_t pitch = align_up((size_t)cols * 4, 128), plane = pitch * rows;
    TempDev t;
    CU_TRY(cudaMalloc(&t.p, plane * 4));
    float* da = static_cast<float*>(t.p);
    float* db = reinterpret_cast<float*>(static_cast<char*>(t.p) + plane);
    float* d1 = reinterpret_cast<float*>(static_cast<char*>(t.p) + 2 * plane);
    float* d2 = reinterpret_cast<float*>(static_cast<char*>(t.p) + 3 * plane);
    cudaStream_t s = nullptr;  // legacy default stream: these calls are synchronous by contract
    if (a) CU_TRY(cudaMemcpy2DAsync(da, pitch, a, in_step, (size_t)cols * 4, rows, cudaMemcpyHostToDevice, s));
    if (b) CU_TRY(cudaMemcpy2DAsync(db, pitch, b, in_step, (size_t)cols * 4, rows, cudaMemcpyHostToDevice, s));
    if (op == 0)
        CU_TRY(launch_mag_phase(da, db, pitch, o1 ? d1 : nullptr, o2 ? d2 : nullptr, pitch, rows, cols, s));
    else
        CU_TRY(launch_phase_maps(kind, da, db, pitch, d1, pitch, rows, cols, phi, signum, s));
    if (o1) CU_TRY(cudaMemcpy2DAsync(o1, out_step, d1, pitch, (size_t)cols * 4, rows, cudaMemcpyDeviceToHost, s));
    if (o2) CU_TRY(cudaMemcpy2DAsync(o2, out_step, d2, pitch, (size_t)cols * 4, rows, cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    return CVS_OK;
}

extern "C" int cvs_magnitude_phase_host(int device, const float* g, const float* h, size_t in_step, float* magnitude, float* phase,
                                        size_t out_step, int rows, int cols)
{
    if (!g || !h || (!magnitude && !phase)) return fail(CVS_ERR_INVALID_ARG, "null argument");
    return pointwise_host(device, 0, 0, g, h, in_step, magnitude, phase, out_step, rows, cols, 0.f, 0);
}

extern "C" int cvs_phase_weights_host(int device, const float* phase, size_t in_step, float* lambda, size_t out_step, int rows, int cols,
                                      float phi, int signum, float k)
{
    (void)k;  // unused in the reference too (G2.cpp:179-186)
    if (!phase || !lambda) return fail(CVS_ERR_INVALID_ARG, "null argument");
    return pointwise_host(device, 1, 0, nullptr, phase, in_step, lambda, nullptr, out_step, rows, cols, phi, signum);
}

extern "C" int cvs_find_host(int device, int kind, const float* e, const float* phase, size_t in_step, float* out, size_t out_step, int rows,
                             int cols, float k)
{
    (void)k;
    if (!e || !phase || !out || kind < 0 || kind > 2) return fail(CVS_ERR_INVALID_ARG, "bad argument");
    return pointwise_host(device, 1, kind + 1, e, phase, in_step, out, nullptr, out_step, rows, cols, 0.f, 0);
}

// ================================ G4 ================================
extern "C" int cvs_g4_create(cvs_g4** out, int device, int width, float spacing)
{
    return filter_create(reinterpret_cast<Filter**>(out), 4, device, width, spacing);
}
extern "C" int cvs_g4_destroy(cvs_g4* h) { return filter_destroy(reinterpret_cast<Filter*>(h)); }
extern "C" int cvs_g4_setup_host(cvs_g4* h, const float* image, int rows, int cols, size_t step)
{
    return filter_setup(reinterpret_cast<Filter*>(h), image, false, rows, cols, step);
}
extern "C" int cvs_g4_size(const cvs_g4* h, int* rows, int* cols)
{
    if (!h) return fail(CVS_ERR_INVALID_ARG, "handle is null");
    const Filter* f = reinterpret_cast<const Filter*>(h);
    if (rows) *rows = f->ready ? f->rows : 0;
    if (cols) *cols = f->ready ? f->cols : 0;
    return CVS_OK;
}
extern "C" int cvs_g4_get_plane_host(cvs_g4* h, int plane, float* dst, size_t step)
{
    return filter_get_plane(reinterpret_cast<Filter*>(h), plane, dst, step);
}
static unsigned g4_steer_mask(float* g4, float* h4, float* mag, float* phase)
{
    return (g4 ? CVS_BIT(CVS_G4T) : 0u) | (h4 ? CVS_BIT(CVS_H4T) : 0u) | (mag ? CVS_BIT(CVS_MAG4) : 0u) | (phase ? CVS_BIT(CVS_PHASE4) : 0u);
}
extern "C" int cvs_g4_steer_scalar_host(cvs_g4* h, float theta, float* g4, float* h4, float* magnitude, float* phase, size_t step)
{
    float* outs[CVS_G4_NPLANES] = {nullptr};
    outs[CVS_G4T] = g4, outs[CVS_H4T] = h4, outs[CVS_MAG4] = magnitude, outs[CVS_PHASE4] = phase;
    return filter_steer(reinterpret_cast<Filter*>(h), CVS_STEER_SCALAR, theta, nullptr, 0, g4_steer_mask(g4, h4, magnitude, phase), outs, step);
}
extern "C" int cvs_g4_steer_map_host(cvs_g4* h, const float* theta, size_t theta_step, float* g4, float* h4, float* magnitude, float* phase,
                                     size_t step)
{
    /* theta == NULL: steer at the handle's own dominant-orientation map (extension, see CVS_G4_THETA) */
    float* outs[CVS_G4_NPLANES] = {nullptr};
    outs[CVS_G4T] = g4, outs[CVS_H4T] = h4, outs[CVS_MAG4] = magnitude, outs[CVS_PHASE4] = phase;
    return filter_steer(reinterpret_cast<Filter*>(h), CVS_STEER_MAP, 0.f, theta, theta_step, g4_steer_mask(g4, h4, magnitude, phase), outs, step);
}

// ================================ device-resident batch path ================================
// 16-bit output layout (fmt != CVS_OUT_F32): checked before anything else, the handle included, and before any CUDA call
// (nplanes: entries of `outs` that may be read)
static int check_out16(int fmt, int cols, size_t out_pitch, unsigned mask, int nplanes, void* const* outs)
{
    if (fmt != CVS_OUT_F16 && fmt != CVS_OUT_BF16) return fail(CVS_ERR_INVALID_ARG, "out_format %d is not a cvs_out_format", fmt);
    if (out_pitch < (size_t)cols * 2) return fail(CVS_ERR_INVALID_ARG, "out_pitch %zu < cols*2", out_pitch);
    if (out_pitch & 1) return fail(CVS_ERR_INVALID_ARG, "16-bit planes need an even out_pitch (%zu)", out_pitch);
    for (int p = 0; outs && p < nplanes; ++p)
        if ((mask >> p & 1u) && ((uintptr_t)outs[p] & 1)) return fail(CVS_ERR_INVALID_ARG, "outs[%d] is not 2-byte aligned", p);
    return CVS_OK;
}

static int run_batch_dev(Filter* f, const cvs_batch* b, unsigned mask, int steer_source, float theta, const float* theta_map,
                         void* const* outs, void* stream, int fmt = CVS_OUT_F32)
{
    const size_t esz = fmt == CVS_OUT_F32 ? 4 : 2;
    if (fmt != CVS_OUT_F32) {
        if (!b) return fail(CVS_ERR_INVALID_ARG, "batch is null");
        const int nplanes = f && f->family == 2 ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES;  // no handle: the smaller family
        if (int rc = check_out16(fmt, b->cols, b->out_pitch, mask, nplanes, outs)) return rc;
    }
    if (!f) return fail(CVS_ERR_INVALID_ARG, "handle is null");
    BatchGeom g;
    int rc = geom_from_batch(b, &g, esz);
    if (rc) return rc;
    rc = check_band(g, f->taps.width, g.full_rows);
    if (rc) return rc;
    const int nplanes = f->family == 2 ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES;
    if (!mask || (mask >> nplanes)) return fail(CVS_ERR_INVALID_ARG, "mask 0x%x selects no / unknown planes", mask);
    if (!outs) return fail(CVS_ERR_INVALID_ARG, "outs is null");
    for (int p = 0; p < nplanes; ++p)
        if ((mask >> p & 1u) && !outs[p]) return fail(CVS_ERR_INVALID_ARG, "outs[%d] is null but selected by mask", p);
    if (b->out_pitch < (size_t)b->cols * esz) return fail(CVS_ERR_INVALID_ARG, "out_pitch %zu < cols*%zu", b->out_pitch, esz);
    if (steer_source < CVS_STEER_DOMINANT || steer_source > CVS_STEER_MAP) return fail(CVS_ERR_INVALID_ARG, "steer_source %d", steer_source);
    if (steer_source == CVS_STEER_MAP && !theta_map) return fail(CVS_ERR_INVALID_ARG, "theta_map is null");
    SteerSpec st{};
    st.source = steer_source;
    st.cos_t = std::cos(theta);
    st.sin_t = std::sin(theta);
    st.theta_map = theta_map;
    return run_fused_fmt(f, g, mask, st, outs, fmt, static_cast<cudaStream_t>(stream));
}

extern "C" int cvs_g2_run_batch_dev(cvs_g2* h, const cvs_batch* b, unsigned mask, int steer_source, float theta_scalar,
                                    const float* theta_map, float* const* outs, void* stream)
{
    return run_batch_dev(reinterpret_cast<Filter*>(h), b, mask, steer_source, theta_scalar, theta_map, reinterpret_cast<void* const*>(outs), stream);
}
extern "C" int cvs_g4_run_batch_dev(cvs_g4* h, const cvs_batch* b, unsigned mask, int steer_source, float theta_scalar,
                                    const float* theta_map, float* const* outs, void* stream)
{
    return run_batch_dev(reinterpret_cast<Filter*>(h), b, mask, steer_source, theta_scalar, theta_map, reinterpret_cast<void* const*>(outs), stream);
}
extern "C" int cvs_g2_run_batch_dev_fmt(cvs_g2* h, const cvs_batch* b, unsigned mask, int steer_source, float theta_scalar,
                                        const float* theta_map, void* const* outs, void* stream, int out_format)
{
    return run_batch_dev(reinterpret_cast<Filter*>(h), b, mask, steer_source, theta_scalar, theta_map, outs, stream, out_format);
}
extern "C" int cvs_g4_run_batch_dev_fmt(cvs_g4* h, const cvs_batch* b, unsigned mask, int steer_source, float theta_scalar,
                                        const float* theta_map, void* const* outs, void* stream, int out_format)
{
    return run_batch_dev(reinterpret_cast<Filter*>(h), b, mask, steer_source, theta_scalar, theta_map, outs, stream, out_format);
}

// Steering-bank arguments, checked before the handle is looked at and before any CUDA call.  out_rows: rows of one output plane.
// family: 2 or 4 -- its bank planes, the per-angle ones among them and its plane count.
static int check_bank(int family, const float* thetas, int n_angles, unsigned mask, void* const* outs, int fmt, int cols, int n, int out_rows,
                      size_t out_pitch, size_t out_frame_stride, size_t angle_stride)
{
    const unsigned planes = family == 2 ? (unsigned)CVS_G2_BANK_PLANES : (unsigned)CVS_G4_BANK_PLANES;
    const unsigned per_angle = family == 2 ? (unsigned)CVS_G2_MASK_STEER5 : (unsigned)CVS_G4_MASK_STEER;
    const int nplanes = family == 2 ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES;
    if (n_angles < 1 || n_angles > CVS_BANK_MAX_ANGLES) return fail(CVS_ERR_INVALID_ARG, "n_angles %d outside [1, %d]", n_angles, CVS_BANK_MAX_ANGLES);
    if (!thetas) return fail(CVS_ERR_INVALID_ARG, "thetas is null");
    if (!mask || (mask & ~planes)) return fail(CVS_ERR_INVALID_ARG, "mask 0x%x: bank planes are 0x%x", mask, planes);
    if (!outs) return fail(CVS_ERR_INVALID_ARG, "outs is null");
    for (int p = 0; p < nplanes; ++p)
        if ((mask >> p & 1u) && !outs[p]) return fail(CVS_ERR_INVALID_ARG, "outs[%d] is null but selected by mask", p);
    if (fmt != CVS_OUT_F32)
        if (int rc = check_out16(fmt, cols, out_pitch, mask, nplanes, outs)) return rc;
    const size_t esz = fmt == CVS_OUT_F32 ? 4 : 2;
    if (out_pitch < (size_t)cols * esz) return fail(CVS_ERR_INVALID_ARG, "out_pitch %zu < cols*%zu", out_pitch, esz);
    if ((out_frame_stride | angle_stride) & (esz - 1))
        return fail(CVS_ERR_INVALID_ARG, "out_frame_stride %zu / angle_stride %zu not multiples of %zu bytes", out_frame_stride, angle_stride, esz);
    // no two (angle, frame) planes of one quantity overlap: sort the strides of the dimensions that have more than one plane
    struct Dim { long long count; size_t stride; } d[2];
    int nd = 0;
    if ((mask & per_angle) && n_angles > 1) d[nd++] = {n_angles, angle_stride};
    if (n > 1) d[nd++] = {n, out_frame_stride};
    if (nd == 2 && d[1].stride < d[0].stride) std::swap(d[0], d[1]);
    const size_t extent = (size_t)std::max(out_rows, 0) * out_pitch;
    if ((nd >= 1 && d[0].stride < extent) || (nd == 2 && d[1].stride / (size_t)d[0].count < d[0].stride))
        return fail(CVS_ERR_INVALID_ARG, "angle_stride %zu and out_frame_stride %zu overlap planes of %zu bytes (%d angles, %d frames)", angle_stride,
                    out_frame_stride, extent, n_angles, n);
    return CVS_OK;
}

static BankSpec make_bank(const float* thetas, int n_angles, unsigned mask, void* const* outs, size_t angle_stride)
{
    BankSpec bk{};
    bk.n_angles = n_angles;
    bk.mask = mask;
    for (int k = 0; k < n_angles; ++k) bk.cos_t[k] = std::cos(thetas[k]), bk.sin_t[k] = std::sin(thetas[k]);  // as run_batch_dev
    for (int p = 0; p < CVS_G2_NPLANES; ++p) bk.outs[p] = (mask >> p & 1u) ? outs[p] : nullptr;
    bk.angle_stride = angle_stride;
    return bk;
}

static int steer_bank_dev(int family, Filter* f, const cvs_batch* b, const float* thetas, int n_angles, unsigned mask, void* const* outs,
                          size_t angle_stride, void* stream, int out_format)
{
    if (!b) return fail(CVS_ERR_INVALID_ARG, "batch is null");
    const int out_rows = b->full_rows > 0 ? b->out_row_end - b->out_row_begin : b->rows;
    if (int rc = check_bank(family, thetas, n_angles, mask, outs, out_format, b->cols, b->n, out_rows, b->out_pitch, b->out_frame_stride,
                            angle_stride))
        return rc;
    if (!f || f->family != family) return fail(CVS_ERR_INVALID_ARG, "handle is null or not a G%d handle", family);
    BatchGeom g;
    int rc = geom_from_batch(b, &g, out_format == CVS_OUT_F32 ? 4 : 2);
    if (rc) return rc;
    rc = check_band(g, f->taps.width, g.full_rows);
    if (rc) return rc;
    return run_bank(f, g, make_bank(thetas, n_angles, mask, outs, angle_stride), out_format, static_cast<cudaStream_t>(stream));
}

extern "C" int cvs_g2_steer_bank_dev(cvs_g2* h, const cvs_batch* b, const float* thetas, int n_angles, unsigned mask, void* const* outs,
                                     size_t angle_stride, void* stream, int out_format)
{
    return steer_bank_dev(2, reinterpret_cast<Filter*>(h), b, thetas, n_angles, mask, outs, angle_stride, stream, out_format);
}
extern "C" int cvs_g4_steer_bank_dev(cvs_g4* h, const cvs_batch* b, const float* thetas, int n_angles, unsigned mask, void* const* outs,
                                     size_t angle_stride, void* stream, int out_format)
{
    return steer_bank_dev(4, reinterpret_cast<Filter*>(h), b, thetas, n_angles, mask, outs, angle_stride, stream, out_format);
}

extern "C" int cvs_pyr_down_dev(int device, const cvs_batch* b, float* out, void* stream)
{
    BatchGeom g;
    int rc = geom_from_batch(b, &g);
    if (rc) return rc;
    if (!out) return fail(CVS_ERR_INVALID_ARG, "out is null");
    if (b->full_rows <= 0) {  // whole frames: all rows of the output level
        g.out_row_begin = 0;
        g.out_row_end = (g.full_rows + 1) / 2;
        g.out_row_origin = 0;
    }
    rc = check_band(g, 2, (g.full_rows + 1) / 2, 2);
    if (rc) return rc;
    CU_TRY(cudaSetDevice(device));
    CU_TRY(launch_pyr_down(g, out, static_cast<cudaStream_t>(stream)));
    return CVS_OK;
}

// Host-buffer batch: frames are processed in chunks on two streams so that the upload of chunk i+1, the kernel of
// chunk i and the download of chunk i-1 overlap.
namespace {
// The input layout of the 8-bit entry points, checked before anything else (the handle included) and before any CUDA call, as
// the 16-bit output layout is (check_out16)
int check_in_u8(const void* in, int cols, size_t in_step)
{
    if (!in) return fail(CVS_ERR_INVALID_ARG, "in is null");
    if (in_step < (size_t)cols) return fail(CVS_ERR_INVALID_ARG, "in_step %zu < cols", in_step);
    return CVS_OK;
}

// in_u8: 8-bit frames (in_step / in_frame_stride in bytes of them), else fp32; the device holds them in the same element type.
// fmt: cvs_out_format of the host output planes (out_step / out_frame_stride in bytes of them)
// bank: a steering bank instead of one launch of `mask` -- its mask and host planes are `mask` / `outs`, per-angle plane p of
// angle k at outs[p] + k * bank->angle_stride; each (plane, angle) pair is one more device plane per chunk and one more download
int run_batch_host(Filter* f, int family, const void* in, bool in_u8, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                   unsigned mask, int steer_source, float theta, void* const* outs, size_t out_step, size_t out_frame_stride, int fmt = CVS_OUT_F32,
                   const BankSpec* bank = nullptr)
{
    const size_t esz = fmt == CVS_OUT_F32 ? 4 : 2, in_esz = in_u8 ? 1 : 4;
    if (in_u8)
        if (int rc = check_in_u8(in, cols, in_step)) return rc;
    if (fmt != CVS_OUT_F32) {
        if (int rc = check_out16(fmt, cols, out_step, mask, family == 2 ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES, outs)) return rc;
        if (out_frame_stride & 1) return fail(CVS_ERR_INVALID_ARG, "16-bit planes need an even out_frame_stride (%zu)", out_frame_stride);
    }
    if (!f || f->family != family || !in || !outs) return fail(CVS_ERR_INVALID_ARG, "null argument or wrong handle family");
    const int NPLANES = family == 2 ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES;
    if (steer_source != CVS_STEER_DOMINANT && steer_source != CVS_STEER_SCALAR)
        return fail(CVS_ERR_INVALID_ARG, "host batches steer at theta_d or at one scalar angle (steer_source %d)", steer_source);
    if (n <= 0 || rows <= 0 || cols <= 0) return fail(CVS_ERR_INVALID_ARG, "n/rows/cols must be positive");
    if (in_step < (size_t)cols * in_esz) return fail(CVS_ERR_INVALID_ARG, "in_step < cols*%zu", in_esz);
    if (out_step < (size_t)cols * esz) return fail(CVS_ERR_INVALID_ARG, "step < cols*%zu", esz);
    if (!mask || (mask >> NPLANES)) return fail(CVS_ERR_INVALID_ARG, "mask 0x%x", mask);
    // device planes per frame: one per selected plane, or one per angle for a bank's per-angle planes
    const unsigned per_angle = family == 2 ? (unsigned)CVS_G2_MASK_STEER5 : (unsigned)CVS_G4_MASK_STEER;
    auto copies = [&](int p) { return bank && (per_angle >> p & 1u) ? bank->n_angles : 1; };
    int nout = 0;
    for (int p = 0; p < NPLANES; ++p)
        if (mask >> p & 1u) {
            if (!outs[p]) return fail(CVS_ERR_INVALID_ARG, "outs[%d] is null but selected by mask", p);
            nout += copies(p);
        }
    CU_TRY(cudaSetDevice(f->device));
    const size_t in_row = (size_t)cols * in_esz, pitch = align_up(in_row, 128), fbytes = pitch * rows;  // device input frames
    const size_t opitch = align_up((size_t)cols * esz, 128), obytes = opitch * rows;  // device output planes
    // G4 steering at a scalar angle into fp32 planes: with the default taps the fp32-frame launch folds the steering factors
    // into the baked column taps (G4Fam::prescaled), which the fp32-output 8-bit kernel does not, so the two differ in the
    // last bits.  There the 8-bit chunk is widened on the device and runs the fp32-frame launch, which keeps the contract
    // (the planes of the widened frames).  Every 16-bit format has fused 8-bit kernels with the same taps as the fp32 ones.  A G4
    // bank keeps the contract on 8-bit frames itself (run_bank), so its chunks stay 8-bit.
    const bool widen = in_u8 && fmt == CVS_OUT_F32 && family == 4 && steer_source == CVS_STEER_SCALAR && !bank;
    const size_t wpitch = align_up((size_t)cols * 4, 128), wbytes = widen ? wpitch * rows : 0;  // fp32 frames; widened ones
    // chunk so that >= 4 chunks exist (pipeline depth) but each is large enough to amortise launch + copy latency: 64 MB of
    // fp32 frames.  8-bit frames count as the fp32 frames they stand for, so 1-byte input does not make chunks four times
    // larger and the pipeline shorter (sizing by input + output bytes instead made the chunks of narrow outputs larger as well,
    // measured 3-7 % slower end to end; DESIGN.md section 11)
    int chunk = (int)((64ull << 20) / (wpitch * rows));
    if (chunk < 1) chunk = 1;
    if (chunk > (n + 3) / 4) chunk = (n + 3) / 4;
    if (chunk < 1) chunk = 1;
    const int NBUF = 3;
    const size_t slot_bytes = (size_t)chunk * (fbytes + wbytes + nout * obytes);
    CU_TRY(f->work.reserve(NBUF * slot_bytes));
    cudaStream_t* streams = f->pipe;  // owned by the handle: they live on the handle's device
    for (int i = 0; i < NBUF; ++i)
        if (!streams[i]) CU_TRY(cudaStreamCreateWithFlags(&streams[i], cudaStreamNonBlocking));
    SteerSpec st{};
    st.source = steer_source;
    st.cos_t = std::cos(theta);
    st.sin_t = std::sin(theta);
    int ci = 0;
    for (int f0 = 0; f0 < n; f0 += chunk, ++ci) {
        const int nf = (n - f0 < chunk) ? (n - f0) : chunk;
        const int b = ci % NBUF;
        cudaStream_t s = streams[b];
        char* base = static_cast<char*>(f->work.p) + (size_t)b * slot_bytes;
        char* din = base;
        // 3-D copy: frames x rows x row-bytes
        cudaMemcpy3DParms cp{};
        cp.srcPtr = make_cudaPitchedPtr(const_cast<char*>(static_cast<const char*>(in)) + (size_t)f0 * in_frame_stride, in_step, in_row,
                                        in_frame_stride / in_step);
        cp.dstPtr = make_cudaPitchedPtr(din, pitch, in_row, rows);
        cp.extent = make_cudaExtent(in_row, rows, nf);
        cp.kind = cudaMemcpyHostToDevice;
        // fully contiguous on both sides (the common case: dense frames whose row is a multiple of 128 bytes): one linear copy,
        // which the copy engine streams a little faster than the equivalent pitched 3-D copy
        const bool in_dense = pitch == in_row && in_step == pitch && in_frame_stride == fbytes;
        if (in_dense) {
            CU_TRY(cudaMemcpyAsync(din, static_cast<const char*>(in) + (size_t)f0 * in_frame_stride, (size_t)nf * fbytes, cudaMemcpyHostToDevice, s));
        } else if (in_frame_stride % in_step == 0) {
            CU_TRY(cudaMemcpy3DAsync(&cp, s));
        } else {
            for (int k = 0; k < nf; ++k)
                CU_TRY(cudaMemcpy2DAsync(din + (size_t)k * fbytes, pitch, static_cast<const char*>(in) + (size_t)(f0 + k) * in_frame_stride, in_step,
                                         in_row, rows, cudaMemcpyHostToDevice, s));
        }
        void* douts[(int)CVS_G2_NPLANES > (int)CVS_G4_NPLANES ? (int)CVS_G2_NPLANES : (int)CVS_G4_NPLANES] = {nullptr};
        int slot = 0;
        for (int p = 0; p < NPLANES; ++p)
            if (mask >> p & 1u) douts[p] = base + (size_t)chunk * fbytes + (size_t)slot * chunk * obytes, slot += copies(p);
        BatchGeom g = whole_frame_geom(din, in_u8, nf, rows, cols, pitch, fbytes, opitch, obytes);
        if (widen) {
            float* dw = reinterpret_cast<float*>(base + (size_t)chunk * (fbytes + nout * obytes));
            CU_TRY(launch_widen(reinterpret_cast<const unsigned char*>(din), pitch, fbytes, dw, wpitch, wbytes, nf, rows, cols, s));
            g = whole_frame_geom(dw, false, nf, rows, cols, wpitch, wbytes, opitch, obytes);
        }
        int rc;
        if (bank) {  // on the device, angle k of a per-angle plane follows the chunk's frames of angle k - 1
            BankSpec bd = *bank;
            for (int p = 0; p < NPLANES; ++p) bd.outs[p] = douts[p];
            bd.angle_stride = (size_t)chunk * obytes;
            rc = run_bank(f, g, bd, fmt, s, b, NBUF);
        } else {
            rc = run_fused_fmt(f, g, mask, st, douts, fmt, s, b, NBUF);
        }
        if (rc) return rc;
        const size_t row_bytes = (size_t)cols * esz;
        for (int p = 0; p < NPLANES; ++p)
            for (int a = 0; (mask >> p & 1u) && a < copies(p); ++a) {
                char* dst = static_cast<char*>(outs[p]) + (size_t)f0 * out_frame_stride + (size_t)a * (bank ? bank->angle_stride : 0);
                char* src = static_cast<char*>(douts[p]) + (size_t)a * chunk * obytes;
                if (opitch == row_bytes && out_step == opitch && out_frame_stride == obytes) {
                    CU_TRY(cudaMemcpyAsync(dst, src, (size_t)nf * obytes, cudaMemcpyDeviceToHost, s));
                } else if (out_frame_stride % out_step == 0) {
                    cudaMemcpy3DParms cq{};
                    cq.srcPtr = make_cudaPitchedPtr(src, opitch, row_bytes, rows);
                    cq.dstPtr = make_cudaPitchedPtr(dst, out_step, row_bytes, out_frame_stride / out_step);
                    cq.extent = make_cudaExtent(row_bytes, rows, nf);
                    cq.kind = cudaMemcpyDeviceToHost;
                    CU_TRY(cudaMemcpy3DAsync(&cq, s));
                } else {
                    for (int k = 0; k < nf; ++k)
                        CU_TRY(cudaMemcpy2DAsync(dst + (size_t)k * out_frame_stride, out_step, src + (size_t)k * obytes, opitch, row_bytes, rows,
                                                 cudaMemcpyDeviceToHost, s));
                }
            }
    }
    for (int i = 0; i < NBUF; ++i) CU_TRY(cudaStreamSynchronize(streams[i]));
    return CVS_OK;
}
}  // namespace

extern "C" int cvs_g2_run_batch_host(cvs_g2* h, const float* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                     unsigned mask, float* const* outs, size_t out_step, size_t out_frame_stride)
{
    return run_batch_host(reinterpret_cast<Filter*>(h), 2, in, false, n, rows, cols, in_step, in_frame_stride, mask, CVS_STEER_DOMINANT, 0.f,
                          reinterpret_cast<void* const*>(outs), out_step, out_frame_stride);
}
extern "C" int cvs_g4_run_batch_host(cvs_g4* h, const float* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                     unsigned mask, int steer_source, float theta_scalar, float* const* outs, size_t out_step,
                                     size_t out_frame_stride)
{
    return run_batch_host(reinterpret_cast<Filter*>(h), 4, in, false, n, rows, cols, in_step, in_frame_stride, mask, steer_source, theta_scalar,
                          reinterpret_cast<void* const*>(outs), out_step, out_frame_stride);
}
extern "C" int cvs_g2_run_batch_host_fmt(cvs_g2* h, const float* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                         unsigned mask, void* const* outs, size_t out_step, size_t out_frame_stride, int out_format)
{
    return run_batch_host(reinterpret_cast<Filter*>(h), 2, in, false, n, rows, cols, in_step, in_frame_stride, mask, CVS_STEER_DOMINANT, 0.f, outs,
                          out_step, out_frame_stride, out_format);
}
extern "C" int cvs_g4_run_batch_host_fmt(cvs_g4* h, const float* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                         unsigned mask, int steer_source, float theta_scalar, void* const* outs, size_t out_step,
                                         size_t out_frame_stride, int out_format)
{
    return run_batch_host(reinterpret_cast<Filter*>(h), 4, in, false, n, rows, cols, in_step, in_frame_stride, mask, steer_source, theta_scalar, outs,
                          out_step, out_frame_stride, out_format);
}
extern "C" int cvs_g2_run_batch_host_u8(cvs_g2* h, const uint8_t* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                        unsigned mask, void* const* outs, size_t out_step, size_t out_frame_stride, int out_format)
{
    return run_batch_host(reinterpret_cast<Filter*>(h), 2, in, true, n, rows, cols, in_step, in_frame_stride, mask, CVS_STEER_DOMINANT, 0.f, outs,
                          out_step, out_frame_stride, out_format);
}
extern "C" int cvs_g4_run_batch_host_u8(cvs_g4* h, const uint8_t* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                        unsigned mask, int steer_source, float theta_scalar, void* const* outs, size_t out_step,
                                        size_t out_frame_stride, int out_format)
{
    return run_batch_host(reinterpret_cast<Filter*>(h), 4, in, true, n, rows, cols, in_step, in_frame_stride, mask, steer_source, theta_scalar, outs,
                          out_step, out_frame_stride, out_format);
}

static int steer_bank_host(int family, Filter* f, const void* in, int in_is_u8, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                           const float* thetas, int n_angles, unsigned mask, void* const* outs, size_t out_step, size_t out_frame_stride,
                           size_t angle_stride, int out_format)
{
    if (int rc = check_bank(family, thetas, n_angles, mask, outs, out_format, cols, n, rows, out_step, out_frame_stride, angle_stride)) return rc;
    if (!in) return fail(CVS_ERR_INVALID_ARG, "in is null");
    const size_t in_esz = in_is_u8 ? 1 : 4;
    if (in_step < (size_t)cols * in_esz) return fail(CVS_ERR_INVALID_ARG, "in_step %zu < cols*%zu", in_step, in_esz);
    const BankSpec bk = make_bank(thetas, n_angles, mask, outs, angle_stride);
    return run_batch_host(f, family, in, in_is_u8 != 0, n, rows, cols, in_step, in_frame_stride, mask, CVS_STEER_SCALAR, 0.f, outs, out_step,
                          out_frame_stride, out_format, &bk);
}

extern "C" int cvs_g2_steer_bank_host(cvs_g2* h, const void* in, int in_is_u8, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                      const float* thetas, int n_angles, unsigned mask, void* const* outs, size_t out_step, size_t out_frame_stride,
                                      size_t angle_stride, int out_format)
{
    return steer_bank_host(2, reinterpret_cast<Filter*>(h), in, in_is_u8, n, rows, cols, in_step, in_frame_stride, thetas, n_angles, mask, outs,
                           out_step, out_frame_stride, angle_stride, out_format);
}
extern "C" int cvs_g4_steer_bank_host(cvs_g4* h, const void* in, int in_is_u8, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                      const float* thetas, int n_angles, unsigned mask, void* const* outs, size_t out_step, size_t out_frame_stride,
                                      size_t angle_stride, int out_format)
{
    return steer_bank_host(4, reinterpret_cast<Filter*>(h), in, in_is_u8, n, rows, cols, in_step, in_frame_stride, thetas, n_angles, mask, outs,
                           out_step, out_frame_stride, angle_stride, out_format);
}

extern "C" int cvs_to_u8_dev(int device, const float* src, int n, int rows, int cols, size_t pitch, size_t frame_stride, float gain, uint8_t* dst,
                             size_t dst_pitch, size_t dst_frame_stride, void* stream)
{
    if (!src || !dst || n <= 0 || rows <= 0 || cols <= 0) return fail(CVS_ERR_INVALID_ARG, "bad argument");
    if (pitch < (size_t)cols * 4 || dst_pitch < (size_t)cols) return fail(CVS_ERR_INVALID_ARG, "pitch too small");
    CU_TRY(cudaSetDevice(device));
    unsigned* mm = nullptr;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!(gain > 0.f)) CU_TRY(cudaMallocAsync(reinterpret_cast<void**>(&mm), sizeof(unsigned) * 2 * n, s));
    cudaError_t e = launch_to_u8(src, pitch, frame_stride, n, rows, cols, gain, mm, dst, dst_pitch, dst_frame_stride, s);
    if (mm) cudaFreeAsync(mm, s);
    CU_TRY(e);
    return CVS_OK;
}

extern "C" int cvs_g2_lines_u8_host(cvs_g2* h, const uint8_t* gray, int n, int rows, int cols, size_t step, size_t frame_stride, float gain,
                                    uint8_t* edges, uint8_t* lines_dark, uint8_t* lines_bright, size_t out_step, size_t out_frame_stride)
{
    Filter* f = reinterpret_cast<Filter*>(h);
    if (!f || f->family != 2 || !gray) return fail(CVS_ERR_INVALID_ARG, "null argument");
    if (n <= 0 || rows <= 0 || cols <= 0) return fail(CVS_ERR_INVALID_ARG, "n/rows/cols must be positive");
    if (step < (size_t)cols || out_step < (size_t)cols) return fail(CVS_ERR_INVALID_ARG, "step < cols");
    uint8_t* outs8[3] = {edges, lines_dark, lines_bright};
    const int planes[3] = {CVS_EDGES, CVS_DARK, CVS_BRIGHT};
    unsigned mask = 0;
    for (int i = 0; i < 3; ++i)
        if (outs8[i]) mask |= CVS_BIT(planes[i]);
    if (!mask) return fail(CVS_ERR_INVALID_ARG, "no output requested");
    CU_TRY(cudaSetDevice(f->device));
    const size_t pin = align_up((size_t)cols, 128), pf = align_up((size_t)cols * 4, 128), p8 = pin;
    // Frames are independent (the min-max normalisation is per frame): process them in chunks round-robin on the handle's
    // pipeline streams so that upload, kernels and download of neighbouring chunks overlap.
    const size_t per_frame = pin * rows + 3 * pf * rows + 3 * p8 * rows;  // [u8 in][3 float maps][3 u8 maps]
    int chunk = (int)std::min<size_t>(16384, std::max<size_t>(1, (256ull << 20) / per_frame));
    if (chunk > (n + 3) / 4) chunk = std::max(1, (n + 3) / 4);
    const int NBUF = 3;
    const int nbuf = std::min(NBUF, (n + chunk - 1) / chunk);
    const size_t slot_bytes = align_up(per_frame * chunk, 256) + align_up(sizeof(unsigned) * 6 * chunk, 256);
    CU_TRY(f->work.reserve(slot_bytes * nbuf));
    cudaStream_t* streams = f->pipe;
    for (int i = 0; i < nbuf; ++i)
        if (!streams[i]) CU_TRY(cudaStreamCreateWithFlags(&streams[i], cudaStreamNonBlocking));
    SteerSpec st{};
    st.source = CVS_STEER_DOMINANT;
    // strided <-> pitched copies of `nf` frames; one flat copy when both sides are dense (2-D DMA of short rows is slow)
    auto copy_frames = [&](void* dst, size_t dpitch, size_t dframe, const void* src, size_t spitch, size_t sframe, int nf, cudaMemcpyKind kind,
                           cudaStream_t s) -> cudaError_t {
        if (dpitch == spitch && dframe == sframe && dframe == dpitch * rows) return cudaMemcpyAsync(dst, src, dframe * nf, kind, s);
        if (nf == 1 || (dframe % dpitch == 0 && sframe % spitch == 0)) {
            cudaMemcpy3DParms cp{};
            cp.srcPtr = make_cudaPitchedPtr(const_cast<void*>(src), spitch, cols, nf == 1 ? rows : sframe / spitch);
            cp.dstPtr = make_cudaPitchedPtr(dst, dpitch, cols, nf == 1 ? rows : dframe / dpitch);
            cp.extent = make_cudaExtent(cols, rows, nf);
            cp.kind = kind;
            return cudaMemcpy3DAsync(&cp, s);
        }
        for (int k = 0; k < nf; ++k) {
            cudaError_t e = cudaMemcpy2DAsync(static_cast<char*>(dst) + (size_t)k * dframe, dpitch, static_cast<const char*>(src) + (size_t)k * sframe,
                                              spitch, cols, rows, kind, s);
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    };
    int ci = 0;
    for (int f0 = 0; f0 < n; f0 += chunk, ++ci) {
        const int nf = std::min(chunk, n - f0);
        cudaStream_t s = streams[ci % nbuf];
        char* w = static_cast<char*>(f->work.p) + (size_t)(ci % nbuf) * slot_bytes;
        const size_t in_bytes = pin * rows * chunk, f_bytes = pf * rows * nf, o_bytes = p8 * rows * nf;  // maps: 3*nf dense frames
        uint8_t* din = reinterpret_cast<uint8_t*>(w);
        unsigned* mm = reinterpret_cast<unsigned*>(w + align_up(per_frame * chunk, 256));
        CU_TRY(copy_frames(din, pin, pin * rows, gray + (size_t)f0 * frame_stride, step, frame_stride, nf, cudaMemcpyHostToDevice, s));
        BatchGeom g = whole_frame_geom(din, true, nf, rows, cols, pin, pin * rows, pf, pf * rows);
        float* outs[CVS_G2_NPLANES] = {nullptr};
        for (int i = 0; i < 3; ++i) outs[planes[i]] = reinterpret_cast<float*>(w + in_bytes + i * f_bytes);
        const bool all3 = outs8[0] && outs8[1] && outs8[2];
        // all three maps + min-max normalisation on the tuned path: the fused kernel reduces the statistics itself (one atomic
        // pair per map per warp), so the float maps are read back once (conversion) instead of twice (min/max + conversion)
        const bool fused_mm = all3 && !(gain > 0.f) && uses_march_path(2, f->taps.width);
        if (fused_mm) {
            CU_TRY(launch_minmax_init(mm, 3 * nf, s));
            g.minmax = mm;
            g.minmax_frames = nf;
        }
        int rc = run_fused(f, g, mask, st, outs, s, ci % nbuf, nbuf);
        if (rc) return rc;
        uint8_t* dout0 = reinterpret_cast<uint8_t*>(w + in_bytes + 3 * f_bytes);
        if (all3)  // the three maps are 3*nf consecutive frames: one conversion launch for all of them
            CU_TRY(launch_to_u8(outs[planes[0]], pf, pf * rows, 3 * nf, rows, cols, gain, mm, dout0, p8, p8 * rows, s, fused_mm));
        for (int i = 0; i < 3; ++i) {
            if (!outs8[i]) continue;
            uint8_t* dout = dout0 + i * o_bytes;
            if (!all3) CU_TRY(launch_to_u8(outs[planes[i]], pf, pf * rows, nf, rows, cols, gain, mm + 2 * (size_t)i * nf, dout, p8, p8 * rows, s));
            CU_TRY(copy_frames(outs8[i] + (size_t)f0 * out_frame_stride, out_step, out_frame_stride, dout, p8, p8 * rows, nf, cudaMemcpyDeviceToHost, s));
        }
    }
    for (int i = 0; i < nbuf; ++i) CU_TRY(cudaStreamSynchronize(streams[i]));
    return CVS_OK;
}

static int run_batch_host_multi(int n_devices, const int* devices, int width, float spacing, const void* in, bool in_u8, int n, int rows,
                                int cols, size_t in_step, size_t in_frame_stride, unsigned mask, void* const* outs, size_t out_step,
                                size_t out_frame_stride, int fmt)
{
    if (in_u8)
        if (int rc = check_in_u8(in, cols, in_step)) return rc;
    if (fmt != CVS_OUT_F32) {
        if (int rc = check_out16(fmt, cols, out_step, mask, CVS_G2_NPLANES, outs)) return rc;
        if (out_frame_stride & 1) return fail(CVS_ERR_INVALID_ARG, "16-bit planes need an even out_frame_stride (%zu)", out_frame_stride);
    }
    if (n_devices <= 0 || n_devices > 64 || !in || !outs || n <= 0) return fail(CVS_ERR_INVALID_ARG, "bad argument");
    const int per = (n + n_devices - 1) / n_devices;
    std::vector<std::thread> threads;
    std::vector<int> rc(n_devices, CVS_OK);
    std::vector<std::string> msg(n_devices);
    for (int d = 0; d < n_devices; ++d) {
        const int f0 = d * per, nf = std::min(per, n - f0);
        if (nf <= 0) break;
        threads.emplace_back([&, d, f0, nf] {
            cvs_g2* h = nullptr;
            int r = cvs_g2_create(&h, devices ? devices[d] : d, width, spacing);
            if (r == CVS_OK) {
                void* o[CVS_G2_NPLANES];
                for (int p = 0; p < CVS_G2_NPLANES; ++p) o[p] = outs[p] ? static_cast<char*>(outs[p]) + (size_t)f0 * out_frame_stride : nullptr;
                r = run_batch_host(reinterpret_cast<Filter*>(h), 2, static_cast<const char*>(in) + (size_t)f0 * in_frame_stride, in_u8, nf, rows, cols,
                                   in_step, in_frame_stride, mask, CVS_STEER_DOMINANT, 0.f, o, out_step, out_frame_stride, fmt);
            }
            if (r != CVS_OK) msg[d] = cvs_last_error();  // thread-local text: carry it back to the caller's thread
            rc[d] = r;
            cvs_g2_destroy(h);
        });
    }
    for (auto& t : threads) t.join();
    for (int d = 0; d < n_devices; ++d)
        if (rc[d] != CVS_OK) return fail(rc[d], "device %d: %s", devices ? devices[d] : d, msg[d].c_str());
    return CVS_OK;
}

extern "C" int cvs_g2_run_batch_host_multi(int n_devices, const int* devices, int width, float spacing, const float* in, int n, int rows,
                                           int cols, size_t in_step, size_t in_frame_stride, unsigned mask, float* const* outs,
                                           size_t out_step, size_t out_frame_stride)
{
    return run_batch_host_multi(n_devices, devices, width, spacing, in, false, n, rows, cols, in_step, in_frame_stride, mask,
                                reinterpret_cast<void* const*>(outs), out_step, out_frame_stride, CVS_OUT_F32);
}
extern "C" int cvs_g2_run_batch_host_multi_fmt(int n_devices, const int* devices, int width, float spacing, const float* in, int n, int rows,
                                               int cols, size_t in_step, size_t in_frame_stride, unsigned mask, void* const* outs,
                                               size_t out_step, size_t out_frame_stride, int out_format)
{
    return run_batch_host_multi(n_devices, devices, width, spacing, in, false, n, rows, cols, in_step, in_frame_stride, mask, outs, out_step,
                                out_frame_stride, out_format);
}
extern "C" int cvs_g2_run_batch_host_multi_u8(int n_devices, const int* devices, int width, float spacing, const uint8_t* in, int n, int rows,
                                              int cols, size_t in_step, size_t in_frame_stride, unsigned mask, void* const* outs,
                                              size_t out_step, size_t out_frame_stride, int out_format)
{
    return run_batch_host_multi(n_devices, devices, width, spacing, in, true, n, rows, cols, in_step, in_frame_stride, mask, outs, out_step,
                                out_frame_stride, out_format);
}

// ---- row bands of one very large image over several GPUs of this process -------------------------------------------
namespace cvsi {

// Same rule as cvsteer_b200/multi.py::plan_bands: band edges on multiples of 2^(levels-1) rows, so that the even-sample
// pyramid of a band coincides with the pyramid of the whole image; `have` adds the filter halo and the pyr_down support.
std::vector<BandPlanC> plan_bands_c(int rows, int world, int levels, int radius)
{
    const int align = 1 << (levels - 1);
    std::vector<int> hl(levels);
    hl[0] = rows;
    for (int l = 1; l < levels; ++l) hl[l] = (hl[l - 1] + 1) / 2;
    const int units = (rows + align - 1) / align, per = (units + world - 1) / world;
    std::vector<int> edges(world + 1);
    for (int r = 0; r <= world; ++r) edges[r] = std::min<long long>(rows, (long long)r * per * align);
    edges[world] = rows;
    std::vector<BandPlanC> plans(world);
    for (int r = 0; r < world; ++r) {
        BandPlanC& p = plans[r];
        p.rows = hl;
        p.out.resize(levels);
        p.have.resize(levels);
        for (int l = 0; l < levels; ++l) {
            if (edges[r] >= rows) {
                p.out[l] = {hl[l], hl[l]};
                continue;
            }
            const int lo = std::min(hl[l], edges[r] >> l);
            const int hi = edges[r + 1] >= rows ? hl[l] : std::min(hl[l], edges[r + 1] >> l);
            p.out[l] = {lo, std::max(lo, hi)};
        }
        for (int l = levels - 1; l >= 0; --l) {
            std::pair<int, int> need = p.out[l];
            if (need.first < need.second) need = {std::max(0, need.first - radius), std::min(hl[l], need.second + radius)};
            if (l + 1 < levels && p.have[l + 1].first < p.have[l + 1].second) {
                const std::pair<int, int> src = {std::max(0, 2 * p.have[l + 1].first - 2), std::min(hl[l], 2 * (p.have[l + 1].second - 1) + 3)};
                need = need.first < need.second ? std::make_pair(std::min(need.first, src.first), std::max(need.second, src.second)) : src;
            }
            p.have[l] = need;
        }
    }
    return plans;
}

int run_band_on_device(int device, int width, float spacing, const BandPlanC& plan, const float* image, int cols, size_t step, int levels,
                       unsigned mask, float* const* const* outs, const size_t* out_steps)
{
    if (plan.empty()) return CVS_OK;
    cvs_g2* hh = nullptr;
    int rc = cvs_g2_create(&hh, device, width, spacing);
    if (rc) return rc;
    Filter* f = reinterpret_cast<Filter*>(hh);
    auto done = [&](int r) {
        cvs_g2_destroy(hh);
        return r;
    };
    int nsel = 0;
    for (int p = 0; p < CVS_G2_NPLANES; ++p) nsel += (mask >> p) & 1u;
    std::vector<int> lc(levels);
    lc[0] = cols;
    for (int l = 1; l < levels; ++l) lc[l] = (lc[l - 1] + 1) / 2;
    // resident level buffers (rows plan.have[l]) + one output staging area sized for level 0
    std::vector<DevBuf> lv(levels);
    std::vector<size_t> pitch(levels);
    for (int l = 0; l < levels; ++l) {
        pitch[l] = align_up((size_t)lc[l] * 4, 128);
        if (cudaError_t e = lv[l].reserve(pitch[l] * (size_t)(plan.have[l].second - plan.have[l].first)); e != cudaSuccess)
            return done(fail(CVS_ERR_CUDA, "band level %d: %s", l, cudaGetErrorString(e)));
    }
    DevBuf stage;
    if (cudaError_t e = stage.reserve(pitch[0] * (size_t)(plan.out[0].second - plan.out[0].first) * nsel); e != cudaSuccess)
        return done(fail(CVS_ERR_CUDA, "band outputs: %s", cudaGetErrorString(e)));
    cudaStream_t s = f->stream;
    auto cu = [&](cudaError_t e, const char* what) { return e == cudaSuccess ? CVS_OK : fail(CVS_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e)); };
    rc = cu(cudaMemcpy2DAsync(lv[0].p, pitch[0], reinterpret_cast<const char*>(image) + (size_t)plan.have[0].first * step, step, (size_t)cols * 4,
                              plan.have[0].second - plan.have[0].first, cudaMemcpyHostToDevice, s),
            "band upload");
    for (int l = 0; l < levels && rc == CVS_OK; ++l) {
        const int lo = plan.out[l].first, hi = plan.out[l].second;
        if (lo < hi) {
            BatchGeom g = whole_frame_geom(lv[l].p, false, 1, plan.have[l].second - plan.have[l].first, lc[l], pitch[l], 0, pitch[l], 0);
            g.full_rows = plan.rows[l];
            g.y_origin = plan.have[l].first;
            g.out_row_begin = lo, g.out_row_end = hi, g.out_row_origin = lo;
            float* d_out[CVS_G2_NPLANES] = {nullptr};
            int slot = 0;
            for (int p = 0; p < CVS_G2_NPLANES; ++p)
                if (mask >> p & 1u) d_out[p] = reinterpret_cast<float*>(static_cast<char*>(stage.p) + (size_t)(slot++) * pitch[l] * (hi - lo));
            SteerSpec st{};
            st.source = CVS_STEER_DOMINANT;
            rc = run_fused(f, g, mask, st, d_out, s);
            for (int p = 0; p < CVS_G2_NPLANES && rc == CVS_OK; ++p)
                if (mask >> p & 1u)   // the "gather": each band lands directly in its rows of the caller's full-size plane
                    rc = cu(cudaMemcpy2DAsync(reinterpret_cast<char*>(outs[l][p]) + (size_t)lo * out_steps[l], out_steps[l], d_out[p], pitch[l],
                                              (size_t)lc[l] * 4, hi - lo, cudaMemcpyDeviceToHost, s),
                            "band download");
        }
        if (rc == CVS_OK && l + 1 < levels && plan.have[l + 1].first < plan.have[l + 1].second) {
            BatchGeom g = whole_frame_geom(lv[l].p, false, 1, plan.have[l].second - plan.have[l].first, lc[l], pitch[l], 0, pitch[l + 1], 0);
            g.full_rows = plan.rows[l];
            g.y_origin = plan.have[l].first;
            g.out_row_begin = plan.have[l + 1].first, g.out_row_end = plan.have[l + 1].second, g.out_row_origin = plan.have[l + 1].first;
            rc = cu(launch_pyr_down(g, static_cast<float*>(lv[l + 1].p), s), "band pyr_down");
        }
        // the staging area is reused by the next level: its downloads are ordered on the same stream
    }
    if (rc == CVS_OK) rc = cu(cudaStreamSynchronize(s), "band sync");
    for (auto& b : lv) b.release();
    stage.release();
    return done(rc);
}
}  // namespace cvsi

extern "C" int cvs_plan_bands(int rows, int world, int levels, int radius, int* plan, int* rows_per_level)
{
    if (rows <= 0 || world <= 0 || levels <= 0 || levels > 30 || radius < 0 || !plan) return fail(CVS_ERR_INVALID_ARG, "cvs_plan_bands: bad argument");
    const std::vector<BandPlanC> plans = plan_bands_c(rows, world, levels, radius);
    for (int r = 0; r < world; ++r)
        for (int l = 0; l < levels; ++l) {
            int* q = plan + ((size_t)r * levels + l) * 4;
            q[0] = plans[r].out[l].first, q[1] = plans[r].out[l].second;
            q[2] = plans[r].have[l].first, q[3] = plans[r].have[l].second;
        }
    if (rows_per_level)
        for (int l = 0; l < levels; ++l) rows_per_level[l] = plans[0].rows[l];
    return CVS_OK;
}

extern "C" int cvs_g2_run_bands_host_multi(int n_devices, const int* devices, int width, float spacing, const float* image, int rows, int cols,
                                           size_t step, int levels, unsigned mask, float* const* const* outs, const size_t* out_steps)
{
    if (n_devices <= 0 || n_devices > 64 || !image || !outs || !out_steps || rows <= 0 || cols <= 0) return fail(CVS_ERR_INVALID_ARG, "bad argument");
    if (levels < 1 || levels > 16 || step < (size_t)cols * 4) return fail(CVS_ERR_INVALID_ARG, "levels / step out of range");
    if (!mask || (mask >> CVS_G2_NPLANES)) return fail(CVS_ERR_INVALID_ARG, "mask 0x%x", mask);
    for (int l = 0, c = cols; l < levels; ++l, c = (c + 1) / 2) {
        if (!outs[l] || out_steps[l] < (size_t)c * 4) return fail(CVS_ERR_INVALID_ARG, "outs[%d] / out_steps[%d]", l, l);
        for (int p = 0; p < CVS_G2_NPLANES; ++p)
            if ((mask >> p & 1u) && !outs[l][p]) return fail(CVS_ERR_INVALID_ARG, "outs[%d][%d] is null but selected by mask", l, p);
    }
    const std::vector<BandPlanC> plans = plan_bands_c(rows, n_devices, levels, width);
    std::vector<std::thread> threads;
    std::vector<int> rc(n_devices, CVS_OK);
    std::vector<std::string> msg(n_devices);
    for (int d = 0; d < n_devices; ++d)
        threads.emplace_back([&, d] {
            rc[d] = run_band_on_device(devices ? devices[d] : d, width, spacing, plans[d], image, cols, step, levels, mask, outs, out_steps);
            if (rc[d] != CVS_OK) msg[d] = cvs_last_error();
        });
    for (auto& t : threads) t.join();
    for (int d = 0; d < n_devices; ++d)
        if (rc[d] != CVS_OK) return fail(rc[d], "device %d: %s", devices ? devices[d] : d, msg[d].c_str());
    return CVS_OK;
}

// ================================ measurement helpers ================================
extern "C" int cvs_bench_ffma(int device, int form, int iters, double* instr_per_s, float* elapsed_ms)
{
    if (form < 0 || form > 5 || iters <= 0 || !instr_per_s) return fail(CVS_ERR_INVALID_ARG, "bad argument");
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    const int threads = 256, blocks = prop.multiProcessorCount * 8;
    float* sink = nullptr;
    CU_TRY(cudaMalloc(&sink, 4));
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    CU_TRY(launch_ffma_bench(form, iters / 8 + 1, blocks, threads, sink, nullptr));  // warm-up
    CU_TRY(cudaEventRecord(e0, nullptr));
    CU_TRY(launch_ffma_bench(form, iters, blocks, threads, sink, nullptr));
    CU_TRY(cudaEventRecord(e1, nullptr));
    CU_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(sink);
    // 64 FMA instructions per `iters` unit per thread (the scalar forms run them 512 to a loop trip: iters rounds up to a
    // multiple of 8); the packed forms (3, 4) do two lane-FMAs per instruction
    const double units = form <= 2 ? (double)((iters + 7) / 8 * 8) : (double)iters;
    const double n = (double)blocks * threads * units * 64.0 * ((form == 3 || form == 4) ? 2.0 : 1.0);
    *instr_per_s = n / (ms * 1e-3);
    if (elapsed_ms) *elapsed_ms = ms;
    return CVS_OK;
}

extern "C" int cvs_g2_last_launch(const cvs_g2* h, int* grid_xyz, int* block, int* smem, char* name, int name_len)
{
    if (!h) return fail(CVS_ERR_INVALID_ARG, "handle is null");
    const Filter* f = reinterpret_cast<const Filter*>(h);
    if (grid_xyz) memcpy(grid_xyz, f->last.grid, sizeof(int) * 3);
    if (block) *block = f->last.block;
    if (smem) *smem = f->last.smem;
    if (name && name_len > 0) snprintf(name, (size_t)name_len, "%s", f->last.name);
    return CVS_OK;
}

extern "C" unsigned long long cvs_launch_count(void) { return launch_count(); }
