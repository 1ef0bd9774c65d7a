// common.h -- internal declarations shared by the translation units of libsrcnn_b200.so.
// Nothing here is part of the C ABI (include/srcnn_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../include/srcnn_b200.h"
#include "weights.h"

namespace srcnn {

// ---- error plumbing: every CUDA call is checked and turned into a status + message ---------------
struct Ctx;
int fail(Ctx* c, int status, const char* fmt, ...);

#define SRCNN_CUDA(ctx, expr)                                                                       \
    do {                                                                                            \
        cudaError_t e__ = (expr);                                                                   \
        if (e__ != cudaSuccess)                                                                     \
            return srcnn::fail((ctx), e__ == cudaErrorMemoryAllocation ? SRCNN_E_NOMEM : SRCNN_E_CUDA, \
                               "%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
    } while (0)

// ---- the calling thread's current device is put back when an entry point returns ------------------
struct DeviceScope {
    int prev = -1;
    bool ok = true;
    explicit DeviceScope(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; }
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
        else prev = -1;   // nothing to restore
    }
    ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;
};

// ---- a grow-only device buffer --------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
};

// ---- bicubic tap tables for one (src -> dst) axis pair, resident on the device --------------------
// ofs[d]  = floor(source coordinate of destination sample d)       (may be -1 .. src-1; taps ofs-1..ofs+2)
// coef[d] = the four 11-bit fixed-point Keys-cubic taps (A=-0.75), exactly as cv::resize builds them.
struct TapTable {
    int src = 0, dst = 0;
    int* d_ofs = nullptr;
    short4* d_coef = nullptr;
    std::vector<int> h_ofs;      // host copies (band planning, footprint bounds)
    std::vector<short4> h_coef;
    unsigned long long stamp = 0;
    int int_scale = 0;           // 2 or 4 when dst = int_scale * src and the table is the periodic one the integer-scale kernel assumes
};

// ---- plane set produced by the colour+bicubic kernel and consumed by the CNN / merge kernels ------
// Planes are u8, `pitch` bytes per row (multiple of 128), `rows` rows starting at output row `row0`.
struct Planes {
    uint8_t* y = nullptr;
    // FP16 copy of the Y plane for the tcgen05 kernel's TMA staging: element (row, x) at index x + kY16Pad of its row, columns
    // -kY16Pad..-1 and W..W+7 hold the replicated edge pixels, rows are `pitch16` BYTES apart (a multiple of 16)
    uint8_t* y16 = nullptr;
    size_t pitch16 = 0;
    uint8_t* cr = nullptr;
    uint8_t* cb = nullptr;
    uint8_t* a = nullptr;       // alpha plane of a four-channel call (SRCNN_ORDER_BGRA / _RGBA), same pitch / frame stride as cr
    uint8_t* yout = nullptr;
    size_t pitch = 0;
    int row0 = 0, rows = 0;
    // a batch of frames: frame f's planes start f * frame_stride (u8 planes) / f * frame_stride16 (FP16 plane) bytes further
    size_t frame_stride = 0, frame_stride16 = 0;
};

// row-walking kernel: the cached cut of a launch's row steps over its pipelines (srcnn_tc2.cu, tc2_partition)
constexpr int kY16Pad = 8;
inline size_t y16_pitch_bytes(int w) { return ((size_t)w + 144 + 7) / 8 * 8 * 2; }   // the last strip's 144-column copy stays inside the row

struct Tc2Partition {
    int nstrips = 0, hb = 0, nworkers = 0, ovh = -1;
    std::vector<long long> bounds;
};

// host-buffer pipeline as a CUDA graph: everything a replay depends on
struct PipeKey {
    const void* src;
    void* dst;
    int n, w, h;
    size_t src_stride, src_frame_stride;
    int order;
    float scale;
    int R0, R1;
    size_t dst_stride, dst_frame_stride;
    int variant, fuse, host_bands, seg_ovh;
    void* stream;
    bool operator==(const PipeKey& o) const {   // field by field: the struct has padding
        return src == o.src && dst == o.dst && n == o.n && w == o.w && h == o.h && src_stride == o.src_stride &&
               src_frame_stride == o.src_frame_stride && order == o.order && scale == o.scale && R0 == o.R0 && R1 == o.R1 &&
               dst_stride == o.dst_stride && dst_frame_stride == o.dst_frame_stride && variant == o.variant && fuse == o.fuse &&
               host_bands == o.host_bands && seg_ovh == o.seg_ovh && stream == o.stream;
    }
};
struct PipeGraph {
    PipeKey key;
    cudaGraphExec_t exec = nullptr;
    bool failed = false;
    long long kernel_launches = 0;      // kernels one replay launches (for srcnn_launch_count)
    unsigned long long stamp = 0;
};

struct Ctx {
    int device = 0;
    int variant = SRCNN_VARIANT_TC;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    cudaStream_t own = nullptr;
    long long launches = 0;
    char err[1536] = {0};

    float* d_params = nullptr;       // the 8129 fp32 parameters (FP32 variant reads these)
    float b3 = 0.f;                  // conv3 bias, handed to the fused kernel as a launch parameter
    void* d_tc2_weights = nullptr;   // packed FP16 operand images for the row-walking tcgen05 kernel (srcnn_tc2.cu)
    bool fuse_merge = false;         // row-walking kernel: merge + YCrCb->BGR in its last epilogue instead of the K-C launch
                                     // (SRCNN_FUSE_MERGE=1; byte-identical, but 0.236 vs 0.214 ms per 4K frame: off by default)
    Tc2Partition tc2_part;
    bool batch_launch = true;        // device-resident batches: one launch per stage and chunk of frames (SRCNN_BATCH_LAUNCH=0: frame by frame)
    int band_first = 0;              // host-buffer pipeline: rows of a single frame's first sub-band (0 = rows / host_bands, >= 256) ...
    double band_growth = 1.3;        // ... and how much longer each following sub-band is (tools/e2e_sweep.py: flat optimum 1.3-1.5)
    int host_bands = 8;              // host-buffer pipeline: most sub-bands a single frame is cut into (SRCNN_HOST_BANDS)
    int ka_int_isr = 0;              // ... tile height in source rows, 0 = chosen per launch (SRCNN_KA_ISR, A/B aid)
    bool ka_int = true;              // colour+bicubic: the integer-scale kernel for x2 / x4 (SRCNN_KA_INT=0: always the generic tiled kernel)
    int tc2_seg_ovh = 12;            // cost of opening a segment, in row steps (SRCNN_TC2_SEG_OVH; 0 = cut into equal row counts)
    int* d_guard = nullptr;          // device-side watchdog flag (mapped pinned)
    int* h_guard = nullptr;

    DevBuf plane_buf;   // Y, Cr, Cb, Y' planes (+ the FP16 Y plane)
    DevBuf plane_buf2;  // a second Cr/Cb pair: consecutive device-resident whole-path calls alternate between the two, so that the
                        // colour+bicubic kernel of call i+1 may run beside the merge kernel of call i (api.cu, carve_planes)
    int plane_sel = 0;               // Cr/Cb pair of the call being enqueued (0 / 1)
    bool overlap = true;             // SRCNN_OVERLAP=0: one plane set, every kernel fully serialised (A/B aid)
    int merge_ctas_per_sm = 0;       // merge kernel: 0 = one 16-pixel group per thread (fastest: 12.5 us per 4K frame, 6.4 TB/s on a 16K frame);
                                     // n = at most n CTAs per SM, threads walk several groups (SRCNN_MERGE_CTAS, A/B aid: 14.0-14.5 us / 5.5-5.7 TB/s)
    bool host_path = false;          // inside the host-buffer pipeline (its sub-bands share one plane set; may be under graph capture)
    // the last merge kernel this context enqueued: the plane set it reads (-1: not a whole-path call's), the stream, and the
    // bytes it writes -- what the next colour+bicubic launch must not touch if it is to start before that merge has finished
    int merge_sel = -1;
    size_t plane_layout[3] = {0, 0, 0}, merge_layout[3] = {0, 0, 0};   // (pitch, rows, frames) of the current carve / of that merge's
    long long early_launches = 0;    // colour+bicubic launches that were allowed to start early (srcnn_debug_overlap)
    cudaStream_t merge_stream = nullptr;
    const uint8_t* merge_lo = nullptr;
    const uint8_t* merge_hi = nullptr;
    DevBuf y16_buf;     // stage API: FP16 copy of a caller's u8 Y plane
    DevBuf act2_buf;    // FP32 variant: conv2 activations (32 float planes) of one row chunk
    DevBuf src_buf;     // device copy of a host source image / batch
    DevBuf dst_buf;     // device copy of the result before D2H
    DevBuf work_buf;    // debug timeline of the fused kernel (SRCNN_TC_DEBUG=1)

    TapTable taps[8];
    unsigned long long tap_clock = 0;
    void* fraw_cache = nullptr;      // fraw_resize.cu: contribution tables kept on the device per (filter, dst, src)

    // host-buffer pipeline (srcnn_process_batch_host): copy-in / copy-out streams and their events
    cudaStream_t s_in = nullptr, s_out = nullptr;
    std::vector<cudaEvent_t> pipe_events;

    // CUDA-graph replay of repeated host-buffer calls (api.cu, host_pipeline)
    std::vector<PipeGraph> graphs;
    unsigned long long graph_clock = 0;
    bool use_graphs = true;          // SRCNN_GRAPHS=0 switches it off
    bool capturing = false;

    // optional per-stage device timing (srcnn_profile_*): 4 events per band processed (mode 1), or 2 -- around the CNN stage
    // only -- in mode 2, which leaves merge(i) and colour+bicubic(i+1) adjacent in the stream (cross-call overlap stays on);
    // prof_calls counts the API calls
    int profiling = 0;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    int prof_calls = 0;
    int fail_stage = 0;              // which stage the last failed whole-path call died in (srcnn_last_failed_stage)
};
int prof_mark(Ctx* c, int which);   // records the next event of the pool on c->stream when profiling is on (api.cu)

int ensure(Ctx* c, DevBuf& b, size_t bytes);
void drop_graphs(Ctx* c);
int get_taps(Ctx* c, int src, int dst, TapTable** out);
void build_cubic_taps(int src, int dst, int* ofs, short4* coef);

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- kernel launchers (each enqueues on c->stream and bumps c->launches) ---------------------------
inline bool yuv420(int order) { return order == SRCNN_ORDER_NV12 || order == SRCNN_ORDER_I420; }
inline bool yuv422(int order) { return order == SRCNN_ORDER_YUY2 || order == SRCNN_ORDER_UYVY; }
// internal order of the resize kernels: two interleaved one-byte planes (NV12's chroma pairs), resized plane by plane into pl.y,
// written interleaved
constexpr int kOrderUV = 100;
// ... and for packed 4:2:2 frames on the generic path: the Y plane as every second byte of the rows (src at the first Y byte),
// and U, V as the bytes 0 and 2 of each 4-byte macropixel (src at the first U byte), resized into pl.y and pl.cr
constexpr int kOrderY422 = 101, kOrderUV422 = 102;

// The chroma planes of 4:2:0 frames (SRCNN_ORDER_NV12 / _I420): resized, no CNN, straight into the caller's output.
// Packed 4:2:2 frames (SRCNN_ORDER_YUY2 / _UYVY) use the same description: `src` is row 0 of the packed frame (src_pitch its
// stride, src_v = 0: the order says where U and V sit in a macropixel), `dst` / `dst + dst_v` are the workspace's Cr / Cb planes
// (U', V'), `dst` shifted so that chroma output row r is at dst + r * dst_pitch; sizes w/2 x h -> ow/2 x oh, rows [r0, r1).
// Grey + alpha frames (SRCNN_ORDER_GRAYA) describe their alpha plane the same way: `src` is row 0 of the frame (alpha is byte 1 of
// each pixel), `dst` the workspace's Cr plane (A'); sizes w x h -> ow x oh, rows [r0, r1).
struct Chroma420 {
    const uint8_t* src = nullptr;   // chroma row 0 of frame 0 (NV12: the interleaved pairs, I420: the U plane)
    size_t src_pitch = 0;           // bytes between chroma rows
    size_t src_v = 0;               // I420: V plane - U plane
    uint8_t* dst = nullptr;         // the same in the output
    size_t dst_pitch = 0, dst_v = 0;
    size_t dst_frame = 0;           // output frame stride (the source's is ResizeArgs::src_frame_stride)
    int sw = 0, sh = 0, ow = 0, oh = 0;   // chroma plane sizes: w/2, h/2, ow/2, oh/2
    int row_begin = 0, row_end = 0;       // chroma output rows to produce: [r0/2, r1/2) of the luma rows [r0, r1)
    const TapTable* tx = nullptr;
    const TapTable* ty = nullptr;
};

struct ResizeArgs {
    const uint8_t* src;   // points at source row `src_row0`
    size_t src_stride;
    int sw, sh;           // full source image size
    int src_row0, src_row1;  // source rows present at src: [src_row0, src_row1)
    int order;
    int ow, oh;           // full output image size
    int row_begin, row_end;  // output rows to produce
    Planes pl;            // destination planes (pl.row0 = output row stored at plane row 0)
    const TapTable* tx;
    const TapTable* ty;
    int nframes = 1;      // same-sized frames in one launch, src_frame_stride / pl.frame_stride apart
    size_t src_frame_stride = 0;
    bool early = false;   // may start while the previous kernel of the stream (a merge kernel of ours) is still running
    Chroma420 ch;         // SRCNN_ORDER_NV12 / _I420 / _YUY2 / _UYVY: the chroma planes (the Y plane is `src`, as for a grey call);
                          // SRCNN_ORDER_GRAYA: the alpha plane
};
int launch_color_bicubic(Ctx* c, const ResizeArgs& a);   // order SRCNN_ORDER_GRAY: the one plane, into pl.y / pl.y16;
                                                         // SRCNN_ORDER_BGRA / _RGBA: pl.a as well;
                                                         // SRCNN_ORDER_NV12 / _I420 / _YUY2 / _UYVY / _GRAYA: Y into pl.y /
                                                         // pl.y16, chroma or alpha per `ch`
inline bool four_channel(int order) { return order == SRCNN_ORDER_BGRA || order == SRCNN_ORDER_RGBA; }

struct MergeArgs {
    const uint8_t* y;
    const uint8_t* cr;
    const uint8_t* cb;
    size_t pitch;
    int w, rows;
    int order;
    uint8_t* dst;
    size_t dst_stride;
    const uint8_t* a = nullptr;   // four-channel orders: the alpha plane (same pitch), written as byte 3 of every pixel
};
int launch_merge(Ctx* c, const MergeArgs& a);
// packed 4:2:2 (a.order SRCNN_ORDER_YUY2 / _UYVY): Y' (a.y) and U', V' (a.cr, a.cb: a.w/2 columns, same pitch) interleaved into
// macropixels; grey + alpha (SRCNN_ORDER_GRAYA): Y' (a.y) and A' (a.cr) interleaved into byte pairs.  In place of the merge, and
// like it the last kernel of the call (releases its dependents on entry)
int launch_pack(Ctx* c, const MergeArgs& a);
void note_merge(Ctx* c);   // api.cu: this context has just put a merge kernel (which releases its dependents early) on its stream
// u8 Y plane -> FP16 plane in the Planes::y16 layout (replicated edge columns included)
int launch_y8_to_y16(Ctx* c, const uint8_t* y, size_t pitch, int w, int rows, uint8_t* y16, size_t pitch16);

// CNN on a plane band.  y points at plane row 0 which is image row `row0`; the plane holds image rows
// [row0, row0+rows).  Produces image rows [out_begin, out_end) into `out`, whose row 0 is image row `out_row0`.
// Border clamps use the FULL image height H / width W (true borders only; band seams read real halo).
struct CnnArgs {
    const uint8_t* y;
    size_t pitch;
    const uint8_t* y16 = nullptr;   // FP16 Y plane (Planes::y16 layout), same row0 convention; tcgen05 variant: built from y when null
    size_t pitch16 = 0;
    int W, H;
    int row0, rows;
    int out_begin, out_end;
    uint8_t* out;
    size_t out_pitch;
    int out_row0 = 0;   // the planes' row0 for the Y' plane; r0 when a grey call writes straight into the caller's band
    // optional fused merge + YCrCb->BGR (row-walking tcgen05 kernel only): when `bgr` is set the kernel reads the Cr/Cb planes
    // (same pitch / row0 convention as y) and writes interleaved pixels for output rows [out_begin, out_end) to `bgr`
    // (which points at row out_begin) instead of the Y' plane
    const uint8_t* cr = nullptr;
    const uint8_t* cb = nullptr;
    uint8_t* bgr = nullptr;
    size_t bgr_stride = 0;
    int order = 0;
    // a batch of frames in one launch (row-walking tcgen05 kernel; not with the fused merge): frames are more strips
    int nframes = 1;
    size_t y16_frame_stride = 0, out_frame_stride = 0;
};
int launch_cnn_fp32(Ctx* c, const CnnArgs& a, float* act2_out /* optional full act2 dump, may be null */);
int fp32_prepare(Ctx* c);    // uploads the parameters to the device's constant bank (once per device and process)
void fraw_release(Ctx* c);   // frees the cached frawscale contribution tables
int launch_cnn_tc2(Ctx* c, const CnnArgs& a);
void tc2_pack_weights(const float* params, uint8_t* img);   // host only: img = tc2_weight_bytes() bytes
size_t tc2_weight_bytes();
int tc2_prepare_weights(Ctx* c, const float* params);
void tc2_release(Ctx* c);
void tc2_partition(int nstrips, int hb, int nworkers, int ovh, long long* bounds);

}  // namespace srcnn

struct srcnn_ctx : public srcnn::Ctx {};
