/*
 * cvsteer_c.h -- C ABI of libcvsteer_b200.so: the B200 (sm_100a) implementation of cvsteer's hot path.
 *
 * This is the drop-in boundary.  Plain pointers and sizes only; no C++/torch/OpenCV types.  Every entry
 * point cites the reference interface it replaces (paths relative to the reference tree,
 * headupinclouds/cvsteer).  The C++ classes in include/cvsteer/SteerableFiltersG{2,4}.h keep the
 * reference's class surface and forward here; INTEGRATION.md shows the binding a maintainer adds.
 *
 * Conventions
 *   - All images are single-channel fp32, row-major; `step`/`pitch` arguments are BYTES per row
 *     (cv::Mat::step), `rows`/`cols` as in cv::Mat.
 *   - Every function returns 0 on success or a negative cvs_status; cvs_last_error() gives text for the
 *     calling thread.  Nothing throws across this boundary.  There is NO CPU fallback: without a CUDA
 *     device every compute entry point fails with CVS_ERR_CUDA.
 *   - A handle is single-threaded; distinct handles may be used concurrently from different threads
 *     (each owns its stream), mirroring the reference where each cv::parallel_for_ iteration builds
 *     its own filter object (example/steer.cpp:69-90,169).
 *   - The library never allocates caller memory: outputs are caller-provided (wrapper does Mat::create).
 */
#ifndef CVSTEER_C_H_
#define CVSTEER_C_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define CVS_API __declspec(dllexport)
#else
#define CVS_API __attribute__((visibility("default")))
#endif

typedef enum cvs_status {
    CVS_OK = 0,
    CVS_ERR_INVALID_ARG = -1,   /* null pointer, rows/cols <= 0, width out of range, step < cols*4 ... */
    CVS_ERR_CUDA = -2,          /* any CUDA runtime/driver failure (incl. no device) */
    CVS_ERR_NOT_SETUP = -3,     /* steer/get before setup (reference: empty Mats -> cv::Exception) */
    CVS_ERR_SIZE_MISMATCH = -4, /* theta map / input planes not the size of the set-up image */
    CVS_ERR_UNSUPPORTED = -5
} cvs_status;

/* Output planes.  Bit i of a `mask` selects plane i.  Names follow the reference's members
 * (cvsteer/SteerableFiltersG2.h:62-66) and steer() outputs (SteerableFiltersG2.cpp:157-177). */
typedef enum cvs_g2_plane {
    CVS_G2A = 0, CVS_G2B, CVS_G2C, CVS_H2A, CVS_H2B, CVS_H2C, CVS_H2D, /* 7 basis planes  G2.cpp:62-68 */
    CVS_C1 = 7, CVS_C2, CVS_C3,                                         /* G2.cpp:93-95 */
    CVS_THETA = 10,      /* dominant orientation angle, (-pi/2, pi/2]      G2.cpp:97-99 */
    CVS_STRENGTH = 11,   /* dominant orientation strength sqrt(c2^2+c3^2)  G2.cpp:97 */
    CVS_G2T = 12,        /* G2 steered to the chosen angle                 G2.cpp:153 */
    CVS_H2T = 13,        /* H2 steered                                     G2.cpp:154 */
    CVS_E = 14,          /* oriented energy c1 + c2 cos2t + c3 sin2t       G2.cpp:174-176 */
    CVS_MAG = 15,        /* sqrt(g2^2+h2^2)                                G2.cpp:109 */
    CVS_PHASE = 16,      /* wrap(atan2(h2,g2)) in (-pi,pi], NaN->0         G2.cpp:109-111 */
    CVS_EDGES = 17,      /* findEdges(magnitude, phase)      G2.cpp:201-204, fed as callers do */
    CVS_DARK = 18,       /* findDarkLines(magnitude, phase)  G2.cpp:205-208 */
    CVS_BRIGHT = 19,     /* findBrightLines(magnitude,phase) G2.cpp:209-212 */
    CVS_G2_NPLANES = 20
} cvs_g2_plane;

#define CVS_BIT(p) (1u << (p))
/* M0: the class state setup() leaves behind (7 basis + c1..c3 + theta + strength) */
#define CVS_G2_MASK_STATE 0x00000FFFu
/* M1: orientation analysis only: theta_d, strength, energy at theta_d */
#define CVS_G2_MASK_ORIENT (CVS_BIT(CVS_THETA) | CVS_BIT(CVS_STRENGTH) | CVS_BIT(CVS_E))
/* M2: full fused basis+steer+orientation: theta_d, strength, g2, h2, e, magnitude, phase */
#define CVS_G2_MASK_FULL (CVS_G2_MASK_ORIENT | CVS_BIT(CVS_G2T) | CVS_BIT(CVS_H2T) | CVS_BIT(CVS_MAG) | CVS_BIT(CVS_PHASE))
/* the five outputs of steer(theta, g2, h2, e, magnitude, phase) (G2.cpp:157-177) at a GIVEN angle: with CVS_STEER_SCALAR or
 * CVS_STEER_MAP this mask has its own fused specialisation, like the masks above have for CVS_STEER_DOMINANT */
#define CVS_G2_MASK_STEER5 (CVS_BIT(CVS_G2T) | CVS_BIT(CVS_H2T) | CVS_BIT(CVS_E) | CVS_BIT(CVS_MAG) | CVS_BIT(CVS_PHASE))
/* the cvsteer-run per-file outputs (example/steer.cpp:88-90): findEdges / findDarkLines / findBrightLines at theta_d */
#define CVS_G2_MASK_LINES (CVS_BIT(CVS_EDGES) | CVS_BIT(CVS_DARK) | CVS_BIT(CVS_BRIGHT))

typedef enum cvs_g4_plane {
    CVS_G4A = 0, CVS_G4B, CVS_G4C, CVS_G4D, CVS_G4E,                /* G4.cpp:69-73 */
    CVS_H4A = 5, CVS_H4B, CVS_H4C, CVS_H4D, CVS_H4E, CVS_H4F,        /* G4.cpp:75-80 */
    CVS_G4T = 11,      /* G4 steered  G4.cpp:110 / :120 */
    CVS_H4T = 12,      /* H4 steered  G4.cpp:111 / :121 */
    CVS_MAG4 = 13,     /* sqrt(g4^2+h4^2): the reference's G4 computeMagnitudeAndPhase is empty */
    CVS_PHASE4 = 14,   /* (G4.cpp:88-90); defined as the G2 class's (G2.cpp:107-112) on (g4,h4) */
    /* G4 orientation analysis -- NOT in the reference (m_theta / m_orientationStrength are declared but never assigned,
     * G4.h:40-41,55).  Defined here exactly as the reference defines it for G2: the lowest-order Fourier terms of the
     * oriented energy E(theta) = G4(theta)^2 + H4(theta)^2 ~ C1 + C2 cos 2theta + C3 sin 2theta, theta_d = atan2(C3,C2)/2,
     * strength = |(C2,C3)|; the same derivation reproduces the G2 constants of G2.cpp:93-95 exactly. */
    CVS_G4_THETA = 15,
    CVS_G4_STRENGTH = 16,
    CVS_G4_NPLANES = 17
} cvs_g4_plane;
#define CVS_G4_MASK_BASIS 0x000007FFu
#define CVS_G4_MASK_STEER (CVS_BIT(CVS_G4T) | CVS_BIT(CVS_H4T) | CVS_BIT(CVS_MAG4) | CVS_BIT(CVS_PHASE4))

/* Which angle the fused kernels steer to.
 * Performance: every mask NAMED above has a fused, fully specialised kernel for every source it is meaningful with (G2: STATE,
 * ORIENT, FULL, LINES at theta_d; FULL, LINES, STEER5 at a scalar angle or an angle map; G4: BASIS, STEER at a map, a scalar or
 * theta_d).  Any other combination of planes runs the run-time-mask kernel: same results, exact cv-compatible math (IEEE
 * division / sqrt, NaNs propagate into theta_d), about half the speed.  The specialised steer kernels use the SFU
 * approximations (<= 1e-6 rad / 1e-6 of range; NaN inputs give phase 0 as cv::patchNaNs does, but a finite theta_d). */
typedef enum cvs_steer_source {
    CVS_STEER_DOMINANT = 0, /* per-pixel theta_d computed in the same kernel (what both reference callers do:
                               example/steer.cpp:87, test/test.cpp:86); for G4 see CVS_G4_THETA. */
    CVS_STEER_SCALAR = 1,   /* one angle for the image   steer(float theta, ...)  G2.cpp:137, G4.cpp:114 */
    CVS_STEER_MAP = 2       /* per-pixel angle map       steer(const Mat1f& theta, ...) G2.cpp:147, G4.cpp:92 */
} cvs_steer_source;

typedef struct cvs_g2 cvs_g2;   /* replaces fa::SteerableFiltersG2  (cvsteer/SteerableFiltersG2.h:35) */
typedef struct cvs_g4 cvs_g4;   /* replaces fa::SteerableFiltersG4  (cvsteer/SteerableFiltersG4.h:35) */

CVS_API const char* cvs_version(void);
CVS_API const char* cvs_last_error(void);     /* thread-local text of the last failure */
CVS_API int cvs_device_count(int* count);
/* Let kernels running on `device` load/store memory that lives on `peer_device` (NVLink / NVSwitch peer memory), e.g.
 * output planes of another GPU mapped through CUDA IPC: the row-band mode then stores each band straight into the root
 * GPU's planes from inside the fused kernel.  Idempotent; CVS_ERR_CUDA when the two GPUs have no peer path. */
CVS_API int cvs_enable_peer_access(int device, int peer_device);
/* Device memory that other PROCESSES on this node can map (one process per GPU): the owner allocates and exports a
 * 64-byte CUDA IPC handle; every other rank opens it WITH ITS OWN GPU CURRENT, which also sets up the NVLink peer
 * mapping, and gets a pointer its kernels can store through.  cvs_shared_close unmaps (importers), cvs_shared_free
 * releases (owner, after every importer has closed). */
#define CVS_IPC_HANDLE_BYTES 64
CVS_API int cvs_shared_alloc(int device, size_t bytes, void** ptr, unsigned char handle[CVS_IPC_HANDLE_BYTES]);
CVS_API int cvs_shared_open(int device, const unsigned char handle[CVS_IPC_HANDLE_BYTES], void** ptr);
CVS_API int cvs_shared_close(int device, void* ptr);
CVS_API int cvs_shared_free(int device, void* ptr);

/* ---- taps: SteerableFilters::create (cvsteer/SteerableFilters.cpp:33-42) with the reference's tap
 *      functions G21..G23,H21..H24 (G2.cpp:35-42) / G41..G45,H41..H46 (G4.cpp:34-45).  Host-only.
 *      `which`: G2 family 0..6 = g1,g2,g3,h1,h2,h3,h4;  G4 family 0..10 = g1..g5,h1..h6.
 *      Writes 2*width+1 floats. */
CVS_API int cvs_g2_make_taps(int which, int width, float spacing, float* dst);
CVS_API int cvs_g4_make_taps(int which, int width, float spacing, float* dst);

/* ================================ G2/H2 handle (class semantics) ================================ */
/* ctor part 1 (taps) -- SteerableFiltersG2::SteerableFiltersG2 G2.cpp:44-56.  1 <= width <= 32. */
CVS_API int cvs_g2_create(cvs_g2** out, int device, int width, float spacing);
CVS_API int cvs_g2_destroy(cvs_g2* h);
/* setup(const Mat1f&) G2.cpp:60-100: upload, fused basis + C1..C3 + theta_d + strength, results stay
 * resident on the device.  Re-callable (re-uses taps), any size >= 1x1. */
CVS_API int cvs_g2_setup_host(cvs_g2* h, const float* image, int rows, int cols, size_t step);
/* same, from 8-bit gray (what both callers pass: the implicit Mat(8UC1)->Mat1f conversion of
 * example/steer.cpp:86 / test/test.cpp:85 is done on the device; values 0..255, no scaling). */
CVS_API int cvs_g2_setup_host_u8(cvs_g2* h, const uint8_t* image, int rows, int cols, size_t step);
CVS_API int cvs_g2_size(const cvs_g2* h, int* rows, int* cols);
/* protected members / getters (G2.h:40-41,62-66): download one plane of the class state
 * (CVS_G2A..CVS_STRENGTH). */
CVS_API int cvs_g2_get_plane_host(cvs_g2* h, int plane, float* dst, size_t step);
/* steer(float theta, g2,h2[,e,magnitude,phase]) G2.cpp:137-145,157-165.  Any output may be NULL. */
CVS_API int cvs_g2_steer_scalar_host(cvs_g2* h, float theta, float* g2, float* h2, float* e,
                                     float* magnitude, float* phase, size_t step);
/* steer(const Mat1f& theta, g2,h2[,e,magnitude,phase]) G2.cpp:147-155,167-177.
 * theta == NULL means "the handle's own dominant-orientation map" without a host round trip
 * (the callers' steer(getDominantOrientationAngle(), ...) idiom). */
CVS_API int cvs_g2_steer_map_host(cvs_g2* h, const float* theta, size_t theta_step, float* g2, float* h2,
                                  float* e, float* magnitude, float* phase, size_t step);
/* steer(const Point&, float, ...) G2.cpp:115-134: out = {g2, h2, e, magnitude, phase}; phase here is the
 * reference's plain atan2 (no wrap, no NaN patch), as in G2.cpp:128. */
CVS_API int cvs_g2_steer_point(cvs_g2* h, int x, int y, float theta, float out[5]);

/* ---- stateless point-wise ops on host images (static / non-member-like in the reference) ---- */
/* computeMagnitudeAndPhase G2.cpp:107-112 */
CVS_API int cvs_magnitude_phase_host(int device, const float* g, const float* h, size_t in_step,
                                     float* magnitude, float* phase, size_t out_step, int rows, int cols);
/* phaseWeights G2.cpp:179-186 (k unused in the reference; accepted and ignored) */
CVS_API int cvs_phase_weights_host(int device, const float* phase, size_t in_step, float* lambda,
                                   size_t out_step, int rows, int cols, float phi, int signum, float k);
/* findEdges / findDarkLines / findBrightLines G2.cpp:201-212: kind = 0 edges, 1 dark, 2 bright */
CVS_API int cvs_find_host(int device, int kind, const float* e, const float* phase, size_t in_step,
                          float* out, size_t out_step, int rows, int cols, float k);

/* ================================ G4/H4 handle ================================ */
CVS_API int cvs_g4_create(cvs_g4** out, int device, int width, float spacing);   /* G4.cpp:47-65 */
CVS_API int cvs_g4_destroy(cvs_g4* h);
CVS_API int cvs_g4_setup_host(cvs_g4* h, const float* image, int rows, int cols, size_t step); /* G4.cpp:67-81 */
CVS_API int cvs_g4_size(const cvs_g4* h, int* rows, int* cols);
CVS_API int cvs_g4_get_plane_host(cvs_g4* h, int plane, float* dst, size_t step);  /* CVS_G4A..CVS_H4F, CVS_G4_THETA, CVS_G4_STRENGTH */
/* steer(float theta, g4, h4) G4.cpp:114-122; magnitude/phase optional (see CVS_MAG4) */
CVS_API int cvs_g4_steer_scalar_host(cvs_g4* h, float theta, float* g4, float* h4, float* magnitude,
                                     float* phase, size_t step);
/* steer(const Mat1f& theta, g4, h4) G4.cpp:92-112 */
CVS_API int cvs_g4_steer_map_host(cvs_g4* h, const float* theta, size_t theta_step, float* g4, float* h4,
                                  float* magnitude, float* phase, size_t step);

/* ================================ device-resident batch path ================================
 * The throughput path: frames already in HBM, outputs written to HBM, one fused launch per pyramid
 * level, nothing else touches memory.  The reference has no batch API; this is its per-file loop
 * (example/steer.cpp:69-124) with the file I/O removed.
 *
 * A batch is `n` frames of rows x cols, frame f at  base + f*frame_stride  bytes, row r at + r*pitch.
 * outs[p] (device pointer, same n/pitch/frame_stride convention via out_pitch/out_frame_stride) is
 * written for every p set in `mask`; other entries are ignored and may be NULL.
 * `stream` is a cudaStream_t (0 = default stream); the call is asynchronous on it.
 */
typedef struct cvs_batch {
    const void* in;          /* device pointer: fp32, or u8 when in_is_u8 != 0 */
    int in_is_u8;
    int n, rows, cols;
    size_t in_pitch, in_frame_stride;
    size_t out_pitch, out_frame_stride;
    /* Row-band support (one huge image split across GPUs, SURVEY section 8e): the buffer holds image
     * rows [y_origin, y_origin+rows) of an image that is `full_rows` tall; outputs are produced for
     * image rows [out_row_begin, out_row_end) only and written at buffer-relative row
     * (y - out_row_origin) of the output planes.  Vertical reflect-101 applies at image rows <0 and
     * >= full_rows only.  For whole frames set full_rows = 0 (=> y_origin 0, all rows). */
    int full_rows, y_origin, out_row_begin, out_row_end, out_row_origin;
    /* Optional pyramid fusion (whole frames only, i.e. full_rows == 0): when next_level != NULL the SAME launch also
     * writes the next pyramid level, cv::pyrDown of the input ((cols+1)/2 x (rows+1)/2 per frame, fp32), from the tile it
     * has staged anyway -- the level never costs a second pass over the input.  Identical bits to cvs_pyr_down_dev. */
    float* next_level;
    size_t next_pitch, next_frame_stride;
} cvs_batch;

/* Layout and speed (results never depend on it): the fast kernels stage tiles by TMA, which needs `in` and in_pitch /
 * in_frame_stride to be multiples of 16 bytes and the default tap width; the two-pixel kernels (FULL, LINES, STEER5) also need
 * an even `cols`, output planes / out_pitch / out_frame_stride -- and theta_map for CVS_STEER_MAP -- that are multiples of 8
 * bytes.  Dense 1920- or 3840-column fp32 frames from cudaMalloc satisfy all of it; anything else silently takes the
 * one-pixel or the cooperative-loader form of the same kernel (bit-identical planes, 5-40 % slower).  cvs_g2_last_launch
 * names the kernel that ran. */
CVS_API int cvs_g2_run_batch_dev(cvs_g2* h, const cvs_batch* b, unsigned mask, int steer_source,
                                 float theta_scalar, const float* theta_map /* device, out_pitch layout */,
                                 float* const* outs, void* stream);
CVS_API int cvs_g4_run_batch_dev(cvs_g4* h, const cvs_batch* b, unsigned mask, int steer_source,
                                 float theta_scalar, const float* theta_map, float* const* outs, void* stream);

/* ---- 16-bit output planes ----
 * The *_fmt entry points below take the same arguments as their fp32 counterparts plus `out_format`; one format applies to
 * every output plane of a call.  Contract: a 16-bit plane is, bit for bit, the fp32 plane the same call writes with
 * CVS_OUT_F32, rounded to nearest even into the chosen format (what torch.Tensor.to(torch.float16 / torch.bfloat16) does
 * to that fp32 plane): NaN stays NaN, and fp16 overflow gives +-inf as IEEE specifies.
 *   - CVS_OUT_F16: 11 significant bits, finite up to 65504.  The quadratic planes (c1..c3, strength, E) of 8-bit-range
 *     images reach 1e5 and overflow; scale such inputs so those planes stay below 65504, e.g. to [0,1].
 *   - CVS_OUT_BF16: any fp32 range at 8 significant bits (about 3 significant digits; half an ulp of an angle near pi is
 *     8e-3 rad, against 9.8e-4 rad in fp16).
 * Layout: out_pitch / out_frame_stride are bytes of the 16-bit planes (out_pitch >= cols*2; out_pitch and every plane
 * 2-byte aligned).  The CVS_STEER_MAP angle map stays fp32 in the outputs' ELEMENT layout, so its byte pitch and frame
 * stride are twice the outputs'.  `next_level` stays fp32 and is unchanged (it is the next level's input).
 * Speed: every mask/source pair with a fused kernel above has a fused 16-bit twin (it stores 2 bytes per pixel and plane;
 * two-pixel kernels need 4-byte aligned planes / out_pitch / out_frame_stride), for fp32 and for 8-bit input (in_is_u8; one
 * pixel per thread, TMA-staged: 16-byte aligned `in`, in_pitch and in_frame_stride).  Everything else -- the cooperative
 * loader, other taps, other masks, a layout misaligned for the store width -- runs the fp32 kernel into stream-ordered
 * scratch on the call's stream and narrows it, with the same bits.  CVS_OUT_F32 is exactly the fp32 call. */
typedef enum cvs_out_format { CVS_OUT_F32 = 0, CVS_OUT_F16 = 1, CVS_OUT_BF16 = 2 } cvs_out_format;
CVS_API int cvs_g2_run_batch_dev_fmt(cvs_g2* h, const cvs_batch* b, unsigned mask, int steer_source, float theta_scalar,
                                     const float* theta_map, void* const* outs, void* stream, int out_format);
CVS_API int cvs_g4_run_batch_dev_fmt(cvs_g4* h, const cvs_batch* b, unsigned mask, int steer_source, float theta_scalar,
                                     const float* theta_map, void* const* outs, void* stream, int out_format);

/* Pyramid level l -> l+1 on the device.  No reference counterpart; defined as cv::pyrDown:
 * [1 4 6 4 1]^2/256, BORDER_REFLECT_101, even samples, out size ((cols+1)/2, (rows+1)/2).
 * Band fields of `b` apply to the INPUT level; outputs rows [out_row_begin,out_row_end) are in the
 * coordinates of the OUTPUT level. */
CVS_API int cvs_pyr_down_dev(int device, const cvs_batch* b, float* out, void* stream);

/* Host-buffer batch (the end-to-end call a user with frames in host memory makes): uploads in chunks,
 * runs the fused kernel, downloads the selected planes; copies and kernels overlap on internal
 * streams.  Host buffers should be pinned for full PCIe rate; frames whose rows are dense multiples of 128 bytes (in_step ==
 * cols * 4 == a multiple of 128, in_frame_stride == rows * in_step, likewise for the outputs) move as one linear copy per
 * plane and chunk, which reaches the plain-memcpy PCIe rate (bench.py: 0.98 of it).  steer source = dominant. */
CVS_API int cvs_g2_run_batch_host(cvs_g2* h, const float* in, int n, int rows, int cols, size_t in_step,
                                  size_t in_frame_stride, unsigned mask, float* const* outs,
                                  size_t out_step, size_t out_frame_stride);
/* G4/H4 twin (config 4 with frames in host memory).  steer_source: CVS_STEER_DOMINANT (the G4 theta_d of this
 * library's extension) or CVS_STEER_SCALAR with theta_scalar; a host theta map is not taken here. */
CVS_API int cvs_g4_run_batch_host(cvs_g4* h, const float* in, int n, int rows, int cols, size_t in_step,
                                  size_t in_frame_stride, unsigned mask, int steer_source, float theta_scalar,
                                  float* const* outs, size_t out_step, size_t out_frame_stride);

/* 16-bit host-buffer batches (see cvs_out_format): outs are host planes of the chosen format, out_step / out_frame_stride
 * in bytes of them; downloads move 2 bytes per pixel and plane, dense rows (out_step == cols*2 == a multiple of 128) still
 * as one linear copy per plane and chunk. */
CVS_API int cvs_g2_run_batch_host_fmt(cvs_g2* h, const float* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                      unsigned mask, void* const* outs, size_t out_step, size_t out_frame_stride, int out_format);
CVS_API int cvs_g4_run_batch_host_fmt(cvs_g4* h, const float* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                      unsigned mask, int steer_source, float theta_scalar, void* const* outs, size_t out_step,
                                      size_t out_frame_stride, int out_format);

/* 8-bit host-buffer batches: the arguments of the _fmt calls above, with 8-bit gray frames (`in`, in_step >= cols and
 * in_frame_stride in bytes of 8-bit rows).  Contract: every plane is, bit for bit, what the fp32-frame call with the same
 * out_format writes for the same frames widened to float (values 0..255, no scaling); CVS_OUT_F32 is allowed.  A null `in`,
 * in_step < cols and the 16-bit output layout errors of the _fmt calls are CVS_ERR_INVALID_ARG before the handle is looked at
 * and before any CUDA call.  Uploads move 1 byte per pixel instead of 4 and the frames stay 8-bit on the device, where the
 * fused kernels stage them by TMA and widen them in shared memory; dense rows (in_step == cols == a multiple of 128, as
 * 1920 and 3840 are, in_frame_stride == rows * cols) move as one linear copy per chunk.  With 16-bit planes a caller that
 * holds 8-bit frames sends 15 bytes per pixel over PCIe for M2 (7 planes) instead of 18, and 7 instead of 10 for M1. */
CVS_API int cvs_g2_run_batch_host_u8(cvs_g2* h, const uint8_t* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                     unsigned mask, void* const* outs, size_t out_step, size_t out_frame_stride, int out_format);
CVS_API int cvs_g4_run_batch_host_u8(cvs_g4* h, const uint8_t* in, int n, int rows, int cols, size_t in_step, size_t in_frame_stride,
                                     unsigned mask, int steer_source, float theta_scalar, void* const* outs, size_t out_step,
                                     size_t out_frame_stride, int out_format);

/* ---- steering banks: one filtering pass, the steered planes at up to 16 angles ----
 * The basis is filtered once per pixel and steered to each of `n_angles` scalar angles thetas[k] (a host array) in the same
 * launch: an oriented-energy or texture feature bank, or one level of a steerable pyramid, without re-reading the frames.
 * Bits of `mask`: per angle any of CVS_G2T, CVS_H2T, CVS_E, CVS_MAG, CVS_PHASE; once per pixel CVS_THETA, CVS_STRENGTH.
 * Layout (bytes): angle k of frame f of per-angle plane p at  outs[p] + k*angle_stride + f*out_frame_stride + row*out_pitch;
 * theta_d and strength at  outs[p] + f*out_frame_stride + row*out_pitch.  angle_stride and out_frame_stride may come in
 * either order ([N, n, rows, cols] or [n, N, rows, cols] tensors), but no two (angle, frame) planes of one quantity may
 * overlap: the smaller stride must be at least one plane (output rows x out_pitch) and the larger must span all the
 * planes of the smaller.  A count of 1 (one frame, one angle, or no per-angle plane) puts no condition on its stride.
 * Contract, for fp32 and 8-bit frames and every out_format:
 *   - for every k, each selected per-angle plane equals, bit for bit, that plane of
 *     cvs_g2_run_batch_dev_fmt(h, b, CVS_G2_MASK_STEER5, CVS_STEER_SCALAR, thetas[k], ..., out_format);
 *   - theta_d and strength equal, bit for bit, those of CVS_G2_MASK_ORIENT at CVS_STEER_DOMINANT.
 * The band fields of `b` and next_level are honoured as in cvs_g2_run_batch_dev.  Argument errors are CVS_ERR_INVALID_ARG
 * before the handle is looked at and before any CUDA call: n_angles outside [1, CVS_BANK_MAX_ANGLES] or null thetas, mask
 * bits outside CVS_G2_BANK_PLANES or none, a null selected plane, an unknown out_format and the 16-bit layout rules of the
 * _fmt calls (angle_stride included), overlapping planes, and (host call) in_step below cols times the element size.
 * Speed: with the default width and taps, TMA-eligible frames (see cvs_g2_run_batch_dev) and planes, pitch and strides
 * aligned to the element size, the whole batch is one fused launch (cvs_g2_last_launch: g2_bank/...).  Anything else runs
 * the calls the contract names, one per angle plus one CVS_G2_MASK_ORIENT launch for theta_d / strength, with unselected
 * quantities in stream-ordered scratch (bank-fallback:<the per-angle kernel>).  More than 16 angles: split the list. */
#define CVS_BANK_MAX_ANGLES 16
#define CVS_G2_BANK_PLANES (CVS_G2_MASK_STEER5 | CVS_BIT(CVS_THETA) | CVS_BIT(CVS_STRENGTH))
CVS_API int cvs_g2_steer_bank_dev(cvs_g2* h, const cvs_batch* b, const float* thetas /* host, n_angles */, int n_angles, unsigned mask,
                                  void* const* outs, size_t angle_stride, void* stream, int out_format);
/* Host-buffer twin (pinned host frames and planes; the chunked upload / kernel / download pipeline of
 * cvs_g2_run_batch_host_fmt).  in_is_u8: 8-bit frames (in_step / in_frame_stride in bytes of them), else fp32.
 * Per-angle plane p of angle k, frame f at  outs[p] + k*angle_stride + f*out_frame_stride + row*out_step. */
CVS_API int cvs_g2_steer_bank_host(cvs_g2* h, const void* in, int in_is_u8, int n, int rows, int cols, size_t in_step,
                                   size_t in_frame_stride, const float* thetas, int n_angles, unsigned mask,
                                   void* const* outs, size_t out_step, size_t out_frame_stride, size_t angle_stride,
                                   int out_format);
/* G4/H4 steering bank: the 11-plane basis is filtered once per pixel and steered to each of `n_angles` scalar angles in the
 * same launch -- G4 orientation feature banks and steerable-pyramid levels without re-reading the frames or re-running the
 * basis march, which is the larger part of the work.  Bits of `mask`: per angle any of CVS_G4T, CVS_H4T, CVS_MAG4,
 * CVS_PHASE4.  Layout as for cvs_g2_steer_bank_dev: angle k of frame f of plane p at
 * outs[p] + k*angle_stride + f*out_frame_stride + row*out_pitch, either stride order, no two (angle, frame) planes of one
 * quantity overlapping.
 * Contract, for fp32 and 8-bit frames and every out_format: for every k, each selected plane equals, bit for bit (NaN
 * positions included), that plane of
 *     cvs_g4_run_batch_dev_fmt(h, b', CVS_G4_MASK_STEER, CVS_STEER_SCALAR, thetas[k], ..., out_format)
 * where b' is the batch with its frames as fp32: b itself for fp32 frames, the 8-bit frames widened to float (values 0..255,
 * no scaling) for 8-bit frames.  (With fp32 planes the single-angle call on 8-bit frames itself runs a kernel whose taps are
 * not prescaled, so its last bits differ from the widened-frames call; the bank follows the widened frames, as the host-buffer
 * 8-bit calls do.)
 * No theta_d / strength: the steer@scalar kernels fold the binomial steering factors into the column taps, so the basis
 * values they steer are not the plain ones the G4 orientation forms need.  Callers who want CVS_G4_THETA / CVS_G4_STRENGTH
 * make one cvs_g4_run_batch_dev_fmt call for them.
 * The band fields of `b` and next_level are honoured as in cvs_g4_run_batch_dev.  Argument errors are CVS_ERR_INVALID_ARG
 * before the handle is looked at and before any CUDA call: n_angles outside [1, CVS_BANK_MAX_ANGLES] or null thetas, mask
 * bits outside CVS_G4_BANK_PLANES or none, a null selected plane, an unknown out_format and the 16-bit layout rules of the
 * _fmt calls (angle_stride included), overlapping planes, and (host call) in_step below cols times the element size; so is a
 * G2 handle.
 * Speed: with the default width and taps, TMA-eligible frames and planes, pitch and strides aligned to the element size, the
 * whole batch is one fused launch (cvs_g2_last_launch on the G4 handle: g4_bank/...).  Anything else widens 8-bit frames into
 * stream-ordered scratch and runs the calls the contract names, one per angle, with unselected quantities in stream-ordered
 * scratch (bank-fallback:<the per-angle kernel>). */
#define CVS_G4_BANK_PLANES CVS_G4_MASK_STEER /* per angle: G4T, H4T, MAG4, PHASE4 */
CVS_API int cvs_g4_steer_bank_dev(cvs_g4* h, const cvs_batch* b, const float* thetas /* host, n_angles */, int n_angles, unsigned mask,
                                  void* const* outs, size_t angle_stride, void* stream, int out_format);
/* Host-buffer twin (the pipeline of cvs_g2_steer_bank_host): in_is_u8 selects 8-bit frames, else fp32. */
CVS_API int cvs_g4_steer_bank_host(cvs_g4* h, const void* in, int in_is_u8, int n, int rows, int cols, size_t in_step,
                                   size_t in_frame_stride, const float* thetas, int n_angles, unsigned mask,
                                   void* const* outs, size_t out_step, size_t out_frame_stride, size_t angle_stride,
                                   int out_format);

/* ---- the callers' 8-bit post-processing (reference example/steer.cpp:92-104, test/test.cpp:93-95), on the device ----
 * gain > 0: Mat::convertTo(CV_8UC1, gain); gain <= 0: cv::normalize(src, dst, 0, 255, NORM_MINMAX, CV_8UC1), per frame. */
CVS_API int cvs_to_u8_dev(int device, const float* src, int n, int rows, int cols, size_t pitch, size_t frame_stride, float gain,
                          uint8_t* dst, size_t dst_pitch, size_t dst_frame_stride, void* stream);
/* The whole per-file body of cvsteer-run (example/steer.cpp:73-104) for a batch of 8-bit gray frames in host memory:
 * SteerableFiltersG2(gray) -> steer(theta_d, ...) -> findEdges / findDarkLines / findBrightLines(magnitude, phase) ->
 * 8-bit maps.  One fused launch + the conversion kernels per batch; any of the three outputs may be NULL. */
CVS_API int cvs_g2_lines_u8_host(cvs_g2* h, const uint8_t* gray, int n, int rows, int cols, size_t step, size_t frame_stride,
                                 float gain, uint8_t* edges, uint8_t* lines_dark, uint8_t* lines_bright, size_t out_step,
                                 size_t out_frame_stride);

/* Same call sharded by frame over `n_devices` GPUs of this process (devices[i], or 0..n-1 when devices == NULL):
 * contiguous blocks of ceil(n/n_devices) frames, one host thread + one handle + its own streams per GPU, NO collective
 * (frames are independent units, as the reference's cv::parallel_for_ over files is: example/steer.cpp:169).
 * For one-process-per-GPU deployments use the per-rank calls above; cvsteer_b200/multi.py does that over
 * torch.distributed, including the row-band mode with its NCCL gather. */
CVS_API int cvs_g2_run_batch_host_multi(int n_devices, const int* devices, int width, float spacing, const float* in, int n,
                                        int rows, int cols, size_t in_step, size_t in_frame_stride, unsigned mask,
                                        float* const* outs, size_t out_step, size_t out_frame_stride);

/* 16-bit twin of cvs_g2_run_batch_host_multi (see cvs_out_format) */
CVS_API int cvs_g2_run_batch_host_multi_fmt(int n_devices, const int* devices, int width, float spacing, const float* in, int n,
                                            int rows, int cols, size_t in_step, size_t in_frame_stride, unsigned mask,
                                            void* const* outs, size_t out_step, size_t out_frame_stride, int out_format);
/* 8-bit-frame twin of cvs_g2_run_batch_host_multi_fmt (see cvs_g2_run_batch_host_u8) */
CVS_API int cvs_g2_run_batch_host_multi_u8(int n_devices, const int* devices, int width, float spacing, const uint8_t* in, int n,
                                           int rows, int cols, size_t in_step, size_t in_frame_stride, unsigned mask,
                                           void* const* outs, size_t out_step, size_t out_frame_stride, int out_format);

/* The row-band plan both band paths use (this library's multi-GPU entry point below and cvsteer_b200/multi.py), for
 * callers that shard one huge image over one process per GPU themselves.  Band edges sit on multiples of 2^(levels-1)
 * rows; per rank r and pyramid level l, plan[(r*levels + l)*4 + {0,1,2,3}] = out_lo, out_hi (rows of level l the rank
 * PRODUCES) and have_lo, have_hi (rows of level l it must hold: outputs + filter halo `radius` + what pyr_down of the
 * next level reads).  rows_per_level[l] = image height at level l.  Ranks past the end of the image get empty ranges. */
CVS_API int cvs_plan_bands(int rows, int world, int levels, int radius, int* plan, int* rows_per_level);

/* One very large image split into ROW BANDS over `n_devices` GPUs of this process (SURVEY section 8e, config 5).  Band
 * edges sit on multiples of 2^(levels-1) rows; every GPU uploads its band plus the halo its coarsest level needs straight
 * from the host image (no halo exchange), builds its slice of the `levels`-level pyramid in band mode, runs the fused
 * kernel per level and downloads its rows directly into the caller's full-size planes outs[level][plane] (row pitch
 * out_steps[level]) -- the gather IS the download.  Bit-identical to the single-GPU whole-image pyramid.  The
 * device-resident variants (outputs gathered in a root GPU's memory over NVLink) are cvs_bands_* / cvs_g2_run_bands_dev_multi below. */
CVS_API int cvs_g2_run_bands_host_multi(int n_devices, const int* devices, int width, float spacing, const float* image,
                                        int rows, int cols, size_t step, int levels, unsigned mask,
                                        float* const* const* outs, const size_t* out_steps);

/* ================================ row bands, device-resident (config 5) ================================
 * ONE very large image split into ROW BANDS over several GPUs with the outputs gathered in the ROOT GPU's memory.  A
 * cvs_bands context is one rank (= one GPU; one process per GPU, or one host thread per GPU) of such a run.  It owns the
 * rank's slice of every pyramid level (band + halo, planned as cvs_plan_bands does), runs band-mode pyr_down + the fused
 * kernel level by level, and delivers its rows to the root's full-size planes:
 *   CVS_GATHER_NONE        results stay in this rank's local planes (cvs_bands_local_plane);
 *   CVS_GATHER_NCCL        grouped ncclSend/ncclRecv per level on a second stream, level l travelling while level l+1 computes;
 *   CVS_GATHER_PEER_STORE  the fused kernel stores straight into the root's planes over NVLink peer memory (compute and
 *                          gather are ONE kernel; no local planes, no second pass);
 *   CVS_GATHER_PEER_COPY   local planes + one copy-engine transfer per level into the root's planes, overlapped like NCCL.
 * Bit-identical to the single-GPU whole-image pyramid in every mode.  No reference counterpart (one image, one thread:
 * example/steer.cpp:69-124).  NCCL is bound at run time (the libnccl already loaded in the process, else the system one). */
typedef struct cvs_bands cvs_bands;
typedef enum cvs_band_gather { CVS_GATHER_NONE = 0, CVS_GATHER_NCCL = 1, CVS_GATHER_PEER_STORE = 2, CVS_GATHER_PEER_COPY = 3 } cvs_band_gather;
#define CVS_NCCL_ID_BYTES 128

CVS_API int cvs_bands_create(cvs_bands** out, int device, int rank, int world, int root, int rows, int cols, int levels,
                             unsigned mask, int width, float spacing);
CVS_API int cvs_bands_destroy(cvs_bands* b);
/* Orderly teardown with one process per rank: EVERY rank calls cvs_bands_detach (destroys the library-owned NCCL communicator,
 * unmaps an imported root block; may wait for the peers' calls, so do not serialise the ranks), the caller's barrier, then
 * cvs_bands_destroy (the root frees its block only now). */
CVS_API int cvs_bands_detach(cvs_bands* b);
/* geometry of `rank` (-1 = this context's own) at `level`: image size of the level, rows produced [out_lo, out_hi), rows held
 * [have_lo, have_hi), row pitch (bytes) of the context's level buffers / local planes / own root planes.  Any out may be NULL. */
CVS_API int cvs_bands_geometry(const cvs_bands* b, int rank, int level, int* level_rows, int* level_cols, int* out_lo, int* out_hi,
                               int* have_lo, int* have_hi, size_t* pitch);
/* level-0 input of this rank: device buffer holding image rows [have_lo, have_hi) (fill it in place), or upload from a host image */
CVS_API int cvs_bands_input_dev(cvs_bands* b, float** ptr, size_t* pitch);
CVS_API int cvs_bands_upload_host(cvs_bands* b, const float* image /* row 0 of the WHOLE image */, size_t step, void* stream);
/* the root's planes: the root allocates one block (cvs_bands_root_bytes) and exports a CUDA IPC handle; other processes import
 * it with their own GPU current; threads of the root's process attach the block pointer (after cvs_enable_peer_access) or
 * caller-owned planes[level][plane] with per-level pitches */
CVS_API int cvs_bands_root_bytes(const cvs_bands* b, size_t* bytes);
CVS_API int cvs_bands_root_export(cvs_bands* b, unsigned char handle[CVS_IPC_HANDLE_BYTES], void** base);
CVS_API int cvs_bands_root_import(cvs_bands* b, const unsigned char handle[CVS_IPC_HANDLE_BYTES]);
CVS_API int cvs_bands_root_attach(cvs_bands* b, void* base);
CVS_API int cvs_bands_root_attach_planes(cvs_bands* b, float* const* const* planes, const size_t* pitches);
CVS_API int cvs_bands_root_plane(cvs_bands* b, int level, int plane, float** ptr, size_t* pitch);
CVS_API int cvs_bands_local_plane(cvs_bands* b, int level, int plane, float** ptr, size_t* pitch);
/* NCCL communicator over the band ranks: created here from a unique id (rank 0 makes it, the caller's control plane carries
 * it to the others; collective), or a caller-owned ncclComm_t */
CVS_API int cvs_nccl_unique_id(unsigned char id[CVS_NCCL_ID_BYTES]);
CVS_API int cvs_bands_nccl_init(cvs_bands* b, const unsigned char id[CVS_NCCL_ID_BYTES]);
CVS_API int cvs_bands_nccl_attach(cvs_bands* b, void* nccl_comm);
/* One step (all levels), asynchronous on `stream`: when the stream has drained, this rank's kernels, copies and sends (root:
 * receives) are complete.  With the peer modes the root additionally needs every OTHER rank's stream to have drained:
 * cvs_bands_barrier enqueues a 1-element ncclAllReduce on the stream for that (or use your own barrier). */
CVS_API int cvs_bands_run(cvs_bands* b, int gather, void* stream);
CVS_API int cvs_bands_barrier(cvs_bands* b, void* stream);
/* The same from ONE process over n_devices GPUs (a host thread per GPU, peer access to devices[0]): image in host memory,
 * outputs device-resident in caller-owned planes root_planes[level][plane] on devices[0] (row pitch root_pitches[level]).
 * gather = CVS_GATHER_PEER_STORE or CVS_GATHER_PEER_COPY.  Synchronous; it runs on the library's own non-blocking streams, so
 * work the caller still has in flight on the output planes (e.g. a fill) must have completed before the call. */
CVS_API int cvs_g2_run_bands_dev_multi(int n_devices, const int* devices, int width, float spacing, const float* image, int rows,
                                       int cols, size_t step, int levels, unsigned mask, int gather,
                                       float* const* const* root_planes, const size_t* root_pitches);

/* ---- measurement helpers (used by bench.py; not part of the reference surface) ---- */
/* Saturating FFMA loop: returns achieved fp32 instructions/s (1 FFMA = 1 instr = 2 flop).
 * form: 0 = immediate-operand FFMA, 1 = register-operand, 2 = constant-bank operand; 3 = packed FFMA2 (counted as 2 per
 * instruction), 4 = FFMA2 interleaved 1:1 with integer ALU work, 5 = scalar FFMA interleaved 1:1 with the same ALU work. */
CVS_API int cvs_bench_ffma(int device, int form, int iters, double* instr_per_s, float* elapsed_ms);
/* Last kernel launch configuration of a handle, for reporting (grid, block, dynamic smem bytes, kernel name). */
CVS_API int cvs_g2_last_launch(const cvs_g2* h, int* grid_xyz, int* block, int* smem, char* name, int name_len);
CVS_API unsigned long long cvs_launch_count(void);  /* kernels launched by this library so far (process-wide) */

#ifdef __cplusplus
}
#endif
#endif /* CVSTEER_C_H_ */
