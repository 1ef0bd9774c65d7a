/*
 * srcnn_b200.h -- C ABI of the B200-native SRCNN inference hot path (libsrcnn_b200.so).
 *
 * This is the drop-in boundary for shuwang127/SRCNN_Cpp's hot path.  The reference has no FFI or
 * plugin layer; what its own host code binds for this path is (citations into /root/reference):
 *   (1) the timed body of pthreadcall(), src/srcnn.cpp:505-659  -> srcnn_process_host()/_device()
 *   (2) the conv entry points declared at src/srcnn.cpp:60-73    -> srcnn_stage_cnn_device()
 *   (3) the OpenCV stage calls at src/srcnn.cpp:509,540,577-582  -> srcnn_stage_color_bicubic_device()
 *       and at src/srcnn.cpp:637-639,657                         -> srcnn_stage_merge_device()
 *   (4) the implied library call ProcessSRCNN(), src/test.cpp:347-353 -> include/libsrcnn.h (C++)
 * INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Plain C: pointers, sizes, ints.  No C++/torch/OpenCV types.  Every function returns an int status
 * (0 = OK, negative = error) and never throws.  There is NO CPU fallback: without a usable CUDA
 * device srcnn_create() fails with SRCNN_E_NODEVICE.
 *
 * Pixel formats: 8-bit, row stride in BYTES.  `order` says whether memory order is B,G,R (OpenCV /
 * bin/srcnn, src/srcnn.cpp:462) or R,G,B (ProcessSRCNN, src/test.cpp:334) -- 3 interleaved channels (HWC)
 * -- or SRCNN_ORDER_GRAY: one channel, 1 byte per pixel in and out (src_stride >= w, dst_stride >= ow).
 * A grey call returns the CNN's Y' of resize(grey) and never computes chroma; it is bit-identical to any
 * channel of the colour path on the grey image replicated to 3 channels (a grey pixel has Y = v and
 * Cr = Cb = 128, which convert back to B = G = R = Y').
 * SRCNN_ORDER_BGRA / SRCNN_ORDER_RGBA: 4 interleaved bytes per pixel in and out (src_stride >= 4*w, dst_stride >= 4*ow), straight
 * (not premultiplied) alpha in byte 3.  Bytes 0..2 of every output pixel equal, byte for byte, the 3-channel call with the
 * matching order (BGRA -> BGR, RGBA -> RGB) on bytes 0..2 of the source; alpha has no influence on them.  Byte 3 is the alpha
 * plane through the one-plane resize (srcnn_stage_resize_plane_device: resize(alpha, INTER_CUBIC), no CNN) -- what the
 * reference does to its planes after `split` (src/srcnn.cpp:540,577-582) and what ProcessSRCNN returns for d = 4.  It is NOT
 * always channel 3 of cv::resize on a CV_8UC4 image: with 4 channels OpenCV splits its float body and integer tail at another
 * column, and the two differ by 1 LSB on some geometries.
 * SRCNN_ORDER_NV12 / SRCNN_ORDER_I420: a packed 4:2:0 video frame in one buffer -- what (h*3/2) x w arrays are to FFmpeg raw
 * video and OpenCV's COLOR_YUV2BGR_NV12 / _I420.  `stride` is in bytes.  NV12: rows 0 .. h-1 are Y (w bytes each, `stride`
 * apart), rows h .. h + h/2 - 1 the interleaved chroma pairs (w bytes = w/2 pairs each, also `stride` apart).  I420: Y as in
 * NV12; U at base + h*stride, h/2 rows of w/2 bytes, stride/2 apart; V follows at U + (h/2)*(stride/2) with the same geometry.
 * The output has the same layout with ow, oh, dst_stride.  w, h, ow and oh must all be even (ow / oh are still the truncation
 * below, so a scale may give an odd size: SRCNN_E_ARG), stride >= w, dst_stride >= ow, I420 strides even, and batch frame
 * strides >= stride*h*3/2 (dst_stride*oh*3/2).  The chroma planes are treated independently, so NV21 (pairs V, U) and YV12
 * (V plane first) are the same two orders.  Byte for byte: the output's Y plane is the SRCNN_ORDER_GRAY call on the source's
 * Y plane; each output chroma plane is resize(plane, Size(ow/2, oh/2), INTER_CUBIC) of the matching source plane -- exactly
 * srcnn_stage_resize_plane_device on it, no CNN.  NV12's interleaved plane is resized as two planes, not as one CV_8UC2 image
 * (whose float body / integer tail split differs, as for alpha above).  No colour matrix is applied anywhere: the network sees
 * the Y plane as it is (limited or full range), and chroma takes cv::resize's centre-aligned grid, so left-sited (MPEG-2 /
 * H.264) chroma gets the quarter-pixel horizontal shift any centre-aligned resize gives -- not compensated.  Whole-frame calls
 * only: the band calls (srcnn_process_band_*, srcnn_mgpu_process_banded_*) return SRCNN_E_ARG for these orders.
 * SRCNN_ORDER_YUY2 / SRCNN_ORDER_UYVY: packed 4:2:2 -- what V4L2 (YUYV), DeckLink (2vuy), Media Foundation (YUY2 / UYVY),
 * FFmpeg (yuyv422 / uyvy422) and OpenCV's CV_8UC2 frames for COLOR_YUV2BGR_YUY2 / _UYVY hold.  A frame of w x h pixels is h rows
 * of 2*w bytes, `stride` bytes apart: w/2 four-byte macropixels Y0 U Y1 V (YUY2) or U Y0 V Y1 (UYVY) per row.  The output has
 * the same layout with ow, oh, dst_stride.  w and ow must be even (h and oh need not be), stride >= 2*w, dst_stride >= 2*ow,
 * batch frame strides >= stride*h (dst_stride*oh); any alignment (unaligned buffers may take slower kernels).  Byte for byte:
 * the output's Y plane is the SRCNN_ORDER_GRAY call on the source's Y plane; each output chroma plane (ow/2 x oh) is
 * resize(plane, Size(ow/2, oh), INTER_CUBIC) of the matching source plane (w/2 x h) -- exactly srcnn_stage_resize_plane_device
 * on it, no CNN.  U and V are resized as two planes, not as one CV_8UC2 image (see NV12 above).  No colour matrix is applied: the
 * network sees Y as it is (limited or full range).  Chroma takes cv::resize's centre-aligned grid; 4:2:2 chroma is co-sited
 * with the even luma samples, so it gets the quarter-pixel horizontal shift any centre-aligned resize gives -- not compensated.
 * The planes are treated independently, so YVYU and VYUY (V before U) are the same two orders.  Chroma has the full vertical
 * resolution, so every whole-path call takes these orders, the band calls and srcnn_mgpu_process_banded_* included.
 * SRCNN_ORDER_GRAYA: grey + alpha, 2 interleaved bytes per pixel in and out -- PNG colour type 4, FFmpeg's ya8, two-channel
 * luminance-alpha textures, ProcessSRCNN's d = 2.  Grey in byte 0, straight (not premultiplied) alpha in byte 1.  stride >= 2*w,
 * dst_stride >= 2*ow, batch frame strides >= stride*h (dst_stride*oh); any w, h and scale (no evenness rule) and any alignment
 * (unaligned buffers may take slower kernels).  Byte for byte: byte 0 of every output pixel is the SRCNN_ORDER_GRAY call on the
 * source's grey plane (alpha has no influence on it); byte 1 is the alpha plane through the one-plane resize
 * (srcnn_stage_resize_plane_device: resize(alpha, INTER_CUBIC), no CNN).  It is NOT always channel 1 of cv::resize on a CV_8UC2
 * image, whose float body / integer tail split differs (see the four-channel orders above).  Alpha has the full vertical
 * resolution, so every whole-path call takes this order, the band calls and srcnn_mgpu_process_banded_* included.
 * Output size is ow=(int)((float)w*scale), oh=(int)((float)h*scale) -- the reference's truncation (src/srcnn.cpp:573-575,
 * src/test.cpp:357-358).
 */
#ifndef SRCNN_B200_H
#define SRCNN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRCNN_B200_ABI_VERSION 2

#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

typedef struct srcnn_ctx srcnn_ctx;

/* Arithmetic variant of the CNN stage (Convolution99x11 + Convolution55). */
enum {
    SRCNN_VARIANT_TC = 0,   /* fused tcgen05/TMEM kernel, FP16 operands, FP32 accumulate (<=1 LSB on >=99.9% px, max 2) */
    SRCNN_VARIANT_FP32 = 1  /* strict FP32 CUDA-core kernels in the reference's summation order (bit-exact) */
};

/* 5 is not assigned: it has been rejected as an unknown order since the four-channel orders were added, and stays so. */
enum { SRCNN_ORDER_BGR = 0, SRCNN_ORDER_RGB = 1, SRCNN_ORDER_GRAY = 2, SRCNN_ORDER_BGRA = 3, SRCNN_ORDER_RGBA = 4,
       SRCNN_ORDER_NV12 = 6, SRCNN_ORDER_I420 = 7, SRCNN_ORDER_YUY2 = 8, SRCNN_ORDER_UYVY = 9, SRCNN_ORDER_GRAYA = 10 };

/* Status codes.  -1 / -2 / -3 / -10 keep the reference CLI's meanings (src/srcnn.cpp:479,493,526,555,684). */
enum {
    SRCNN_OK = 0,
    SRCNN_E_RATIO = -1,     /* scale makes an empty image ("ratio too small", src/srcnn.cpp:485-495) */
    SRCNN_E_ARG = -20,      /* null pointer, non-positive size, stride too small, unknown enum */
    SRCNN_E_NODEVICE = -30, /* no CUDA device / device is not sm_100 */
    SRCNN_E_CUDA = -31,     /* a CUDA runtime call or kernel failed; see srcnn_last_error() */
    SRCNN_E_NOMEM = -32,    /* device or pinned-host allocation failed */
    SRCNN_E_KERNEL = -33    /* a device-side guard tripped (pipeline watchdog) */
};

/* Stage of the whole path in which the last failed call died (srcnn_last_failed_stage): lets the CLI keep the
 * reference's distinct exit codes -2 (colour conversion, src/srcnn.cpp:526) and -3 (split, :555). */
enum {
    SRCNN_STAGE_NONE = 0,
    SRCNN_STAGE_COLOR_BICUBIC = 1, /* cvtColor + resize, src/srcnn.cpp:509,570-583 */
    SRCNN_STAGE_PLANES = 2,        /* the plane set `split` produces, src/srcnn.cpp:539-540 */
    SRCNN_STAGE_CNN = 3,           /* Convolution99x11 + Convolution55, src/srcnn.cpp:609,627 */
    SRCNN_STAGE_MERGE = 4          /* merge + cvtColor back, src/srcnn.cpp:637-657 */
};

int srcnn_abi_version(void);
const char* srcnn_strerror(int status);

/* Context = one device + one stream + workspace + packed weights.  Re-entrant: one context per host
 * thread (or serialise calls); may be created and used from a non-main thread like the reference's
 * worker pthread (src/srcnn.cpp:717-724).  Every call runs on the context's device and restores the
 * calling thread's current CUDA device before it returns. */
int srcnn_create(srcnn_ctx** out, int device, int variant);
int srcnn_destroy(srcnn_ctx* ctx);
const char* srcnn_last_error(srcnn_ctx* ctx);
int srcnn_last_failed_stage(srcnn_ctx* ctx);
int srcnn_get_device(srcnn_ctx* ctx);
int srcnn_set_variant(srcnn_ctx* ctx, int variant);
int srcnn_get_variant(srcnn_ctx* ctx);
/* Use an existing CUDA stream (cudaStream_t as void*) for all work of this context; NULL = own stream. */
int srcnn_set_stream(srcnn_ctx* ctx, void* cuda_stream);
void* srcnn_get_stream(srcnn_ctx* ctx);
int srcnn_sync(srcnn_ctx* ctx);
/* Number of kernels this context has launched since creation (for bench.py's gpu_launches). */
long long srcnn_launch_count(srcnn_ctx* ctx);
int srcnn_device_sm_count(srcnn_ctx* ctx);
/* Optional per-stage device timing with CUDA events on the context stream (used by bench.py for the
 * roofline numbers).  srcnn_profile_read synchronises, returns the summed milliseconds of
 * [0] colour+bicubic, [1] fused SRCNN, [2] merge+colour-back over everything processed since the
 * previous read, and the number of whole-path API calls that work came from (a batch or a banded
 * call counts once, however many frames or bands it ran). */
/* on = 1: events around all three stages (the stages of consecutive calls then run strictly one after another);
 * on = 2: events around the CNN stage only, so that the merge kernel of one call and the colour+bicubic kernel of the next stay
 *         adjacent in the stream and may overlap (DESIGN.md "Cross-call overlap"): srcnn_profile_read then returns
 *         [0] the summed time BETWEEN consecutive CNN launches, [1] the CNN stage, [2] 0. */
int srcnn_profile_enable(srcnn_ctx* ctx, int on);
int srcnn_profile_read(srcnn_ctx* ctx, double* ms3, int* calls);

int srcnn_out_dims(int w, int h, float scale, int* ow, int* oh);

/* Pinned host memory for callers that want true async DMA (bench e2e, CLI): allocated page-locked, or the
 * caller's own buffer page-locked in place.  Both are valid for every device of the process. */
int srcnn_host_alloc(void** p, size_t bytes);
int srcnn_host_free(void* p);
int srcnn_host_register(void* p, size_t bytes);
int srcnn_host_unregister(void* p);

/* ---- whole path: replaces src/srcnn.cpp:505-659 -------------------------------------------------- */
/* Host buffers in, host buffers out; H2D and D2H copies are part of the call; returns when dst is ready. */
int srcnn_process_host(srcnn_ctx* ctx, const uint8_t* src, int w, int h, size_t src_stride, int order,
                       float scale, uint8_t* dst, size_t dst_stride);
/* Device buffers; enqueued on the context stream, returns without synchronising.  Ordinary stream semantics: ordered after
 * everything the caller enqueued before the call, complete when the stream reaches the point after it.  (Between two whole-path
 * calls that follow each other directly the library may run the second call's first kernel beside the first call's last one --
 * never when the second call's source overlaps the first call's result; SRCNN_OVERLAP=0 switches that off.) */
int srcnn_process_device(srcnn_ctx* ctx, const uint8_t* d_src, int w, int h, size_t src_stride, int order,
                         float scale, uint8_t* d_dst, size_t dst_stride);
/* n same-sized frames, frame f at base + f*frame_stride (bytes).  Device or host variants. */
int srcnn_process_batch_device(srcnn_ctx* ctx, const uint8_t* d_src, int n, int w, int h, size_t src_stride,
                               size_t src_frame_stride, int order, float scale, uint8_t* d_dst,
                               size_t dst_stride, size_t dst_frame_stride);
int srcnn_process_batch_host(srcnn_ctx* ctx, const uint8_t* src, int n, int w, int h, size_t src_stride,
                             size_t src_frame_stride, int order, float scale, uint8_t* dst,
                             size_t dst_stride, size_t dst_frame_stride);

/* ---- row bands (gigapixel images, multi-GPU sharding; SURVEY 8e) -------------------------------- */
/* Source rows [*s0,*s1) that output rows [r0,r1) of the full (w x h)*scale image depend on (6-px halo
 * in the upscaled-Y domain: 4 for conv1 + 2 for conv3, src/srcnn.cpp:273,279,203,209). */
int srcnn_band_src_rows(int h, float scale, int r0, int r1, int* s0, int* s1);
/* Computes output rows [r0,r1).  d_src points at source row s0 (as returned above) and holds rows
 * [s0,s1); d_dst points at output row r0.  All coordinates, taps and border clamps are those of the
 * full image, so the union of bands is bit-identical to the unsplit result. */
int srcnn_process_band_device(srcnn_ctx* ctx, const uint8_t* d_src, int w, int h, size_t src_stride, int s0,
                              int s1, int order, float scale, int r0, int r1, uint8_t* d_dst,
                              size_t dst_stride);

/* Host-buffer form: `src` is the WHOLE source image (row 0), `dst_rows` points at output row r0.  Copies in only
 * the source rows the band needs, pipelines sub-bands over three streams, returns when dst_rows is ready. */
int srcnn_process_band_host(srcnn_ctx* ctx, const uint8_t* src, int w, int h, size_t src_stride, int order,
                            float scale, int r0, int r1, uint8_t* dst_rows, size_t dst_stride);

/* ---- all GPUs of one box behind one call (SURVEY 8b "device list", 8e) ----------------------------
 * The reference's unit of parallelism is the OpenMP row loop inside one call from one worker thread
 * (src/srcnn.cpp:283,213,717-724).  Its drop-in equivalent: ONE call that fans frames (frame f -> device
 * f mod n) or output-row bands (6-px halo, srcnn_band_src_rows) out over a list of devices.  One host
 * thread, one srcnn_ctx and one stream set per device, disjoint outputs, no inter-GPU traffic, no NCCL.
 * Calls block until every device has finished.  A device may be listed more than once (several contexts
 * on one GPU). */
typedef struct srcnn_mgpu srcnn_mgpu;
/* devices == NULL: devices 0..n-1; n <= 0: every visible device. */
int srcnn_mgpu_create(srcnn_mgpu** out, const int* devices, int n, int variant);
int srcnn_mgpu_destroy(srcnn_mgpu* m);
int srcnn_mgpu_device_count(srcnn_mgpu* m);
srcnn_ctx* srcnn_mgpu_context(srcnn_mgpu* m, int i);       /* worker i's context (variant, profiling, error text) */
const char* srcnn_mgpu_last_error(srcnn_mgpu* m);
/* Worker i's share of a banded image: output rows [*r0,*r1) and the source rows [*s0,*s1) they need.  Pure
 * host arithmetic (callable without a GPU). */
int srcnn_mgpu_band_plan(int n_workers, int h, float scale, int i, int* r0, int* r1, int* s0, int* s1);
/* Frames: frame f is processed by worker f mod n.  Host buffers (H2D / kernels / D2H pipelined per device). */
int srcnn_mgpu_process_batch_host(srcnn_mgpu* m, const uint8_t* src, int nframes, int w, int h, size_t src_stride,
                                  size_t src_frame_stride, int order, float scale, uint8_t* dst, size_t dst_stride,
                                  size_t dst_frame_stride);
/* One image cut into n row bands, worker i computes band i straight into dst.  Host buffers. */
int srcnn_mgpu_process_banded_host(srcnn_mgpu* m, const uint8_t* src, int w, int h, size_t src_stride, int order,
                                   float scale, uint8_t* dst, size_t dst_stride);
/* Device-resident forms: d_src[i] / d_dst[i] live on worker i's device.  Batch: worker i owns counts[i]
 * frames.  Banded: d_src[i] holds source rows [s0_i, s1_i) of srcnn_mgpu_band_plan, d_dst[i] points at
 * output row r0_i. */
int srcnn_mgpu_process_batch_device(srcnn_mgpu* m, const uint8_t* const* d_src, const int* counts, int w, int h,
                                    size_t src_stride, size_t src_frame_stride, int order, float scale,
                                    uint8_t* const* d_dst, size_t dst_stride, size_t dst_frame_stride);
int srcnn_mgpu_process_banded_device(srcnn_mgpu* m, const uint8_t* const* d_src, int w, int h, size_t src_stride,
                                     int order, float scale, uint8_t* const* d_dst, size_t dst_stride);
/* Timing of the last call: per-worker device time (CUDA events on each worker's stream around its share;
 * host-buffer calls: the worker's wall time, copies included) and the call's wall time.  ms has room for
 * srcnn_mgpu_device_count() doubles. */
int srcnn_mgpu_last_timing(srcnn_mgpu* m, double* ms_per_worker, double* wall_ms);

/* ---- stream ingest (SURVEY 8f, N4): JPEG frames in, JPEG frames out ----------------------------------
 * The reference decodes one file before and encodes one after its timed region (cv::imread / cv::imwrite,
 * src/srcnn.cpp:462,670).  For a stream of same-sized frames: nvJPEG decode of frame i+1, the kernels of frame i
 * and the nvJPEG encode of frame i-1 overlap on three streams; pixels never visit host memory.  out[i] is
 * allocated by the library (release with srcnn_jpeg_free); quality 95 + 4:2:0 = cv::imwrite's defaults.  File
 * codecs are outside the parity contract. */
typedef struct srcnn_jpeg_stream srcnn_jpeg_stream;
int srcnn_jpeg_stream_create(srcnn_jpeg_stream** out, srcnn_ctx* ctx, int quality);
int srcnn_jpeg_stream_destroy(srcnn_jpeg_stream* s);
const char* srcnn_jpeg_stream_last_error(srcnn_jpeg_stream* s);
int srcnn_jpeg_stream_process(srcnn_jpeg_stream* s, const uint8_t* const* jpegs, const size_t* sizes, int n, float scale,
                              uint8_t** out, size_t* out_sizes, int* out_w, int* out_h);
void srcnn_jpeg_free(uint8_t* p);

/* ---- stages (device pointers; enqueued on the context stream) ------------------------------------ */
/* cvtColor + split + 3x resize (src/srcnn.cpp:509,540,570-583): BGR8 -> three u8 planes of ow x oh.  Colour orders only
 * (SRCNN_ORDER_GRAY, _BGRA, _RGBA, _GRAYA, the 4:2:0 and 4:2:2 orders: SRCNN_E_ARG; srcnn_stage_resize_plane_device is the
 * one-plane stage). */
int srcnn_stage_color_bicubic_device(srcnn_ctx* ctx, const uint8_t* d_src, int w, int h, size_t src_stride,
                                     int order, float scale, uint8_t* d_y, uint8_t* d_cr, uint8_t* d_cb,
                                     size_t plane_pitch);
/* One 8-bit plane through resize(..., CV_INTER_CUBIC) (src/srcnn.cpp:577-582), host buffers. */
int srcnn_resize_plane_host(srcnn_ctx* ctx, const uint8_t* src, int w, int h, size_t src_stride, float scale,
                            uint8_t* dst, size_t dst_stride);
/* The same on device buffers, enqueued on the context stream: one u8 plane through resize(..., CV_INTER_CUBIC).  Any
 * stride >= the row and any alignment (an unaligned destination costs one extra device copy). */
int srcnn_stage_resize_plane_device(srcnn_ctx* ctx, const uint8_t* d_src, int w, int h, size_t src_stride, float scale,
                                    uint8_t* d_dst, size_t dst_stride);
/* Convolution99x11 + Convolution55 (src/srcnn.cpp:609,627): Y plane -> Y' plane, `variant` as above. */
int srcnn_stage_cnn_device(srcnn_ctx* ctx, int variant, const uint8_t* d_y, int w, int h, size_t pitch,
                           uint8_t* d_out, size_t out_pitch);
/* FP32 variant only: also returns conv2's activations, 32 planes of h*w float (src/srcnn.cpp:602-607). */
int srcnn_stage_conv99x11_fp32_device(srcnn_ctx* ctx, const uint8_t* d_y, int w, int h, size_t pitch,
                                      float* d_act2);
/* merge + cvtColor back (src/srcnn.cpp:637-639,657): three planes -> BGR8 HWC.  Colour orders only (BGR, RGB). */
int srcnn_stage_merge_device(srcnn_ctx* ctx, const uint8_t* d_y, const uint8_t* d_cr, const uint8_t* d_cb,
                             int w, int h, size_t plane_pitch, int order, uint8_t* d_dst, size_t dst_stride);

/* ---- optional: frawscale-compatible float-plane resize (SURVEY 8f, N3) --------------------------- */
/* FRAWResizeEngine::scale (src/frawscale.h:160-161, src/frawscale.cpp:162-286) on device float planes (tight
 * rows).  filter: 0 = Box, 1 = Bilinear, 2 = Bicubic (Mitchell B = C = 1/3, the reference default).  Not used by
 * the bin/srcnn path (the reference never calls frawscale either); bit-identical to the compiled reference: every
 * non-NaN output has the reference's bits, and NaN appears where it does.  Only NaN-ness is promised: on a B200 a NaN
 * input kept its sign and payload and Inf - Inf gave x86's NaN in every case measured, but which payload survives a sum
 * of several NaNs is the hardware's choice.  The claim rests on the golden vectors and on a float64 restatement
 * (oracle/fraw.py) that equals them, checked against the stage on planes built to show FMA contraction, another tap
 * order, a float accumulator and off-by-an-ulp table weights (tests/test_fraw_precision.py).  A plane of equal size is
 * copied whole.  Source and destination must not overlap (SRCNN_E_ARG): a one-axis resize reads the source while it
 * writes the destination.  At most 65535 rows on either side. */
enum { SRCNN_FRAW_BOX = 0, SRCNN_FRAW_BILINEAR = 1, SRCNN_FRAW_BICUBIC = 2 };
int srcnn_fraw_scale_device(srcnn_ctx* ctx, const float* d_src, unsigned src_w, unsigned src_h, unsigned dst_w,
                            unsigned dst_h, float* d_dst, int filter);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* SRCNN_B200_H */
