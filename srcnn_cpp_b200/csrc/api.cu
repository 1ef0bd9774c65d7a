// api.cu -- the C ABI of libsrcnn_b200.so (include/srcnn_b200.h): context, workspace, and the
// host-side orchestration that replaces the timed body of the reference's pthreadcall()
// (src/srcnn.cpp:505-659) with three kernel stages on one CUDA stream:
//   K-A colour+bicubic  ->  K-B fused SRCNN (tcgen05 or strict FP32)  ->  K-C merge+colour back.
// No CPU fallback exists anywhere in this file: every path ends in a kernel launch or an error.
#include <cstdarg>
#include <cstdlib>
#include <iterator>
#include <mutex>
#include <new>
#include <unordered_map>

#include "common.h"

namespace srcnn {

int fail(Ctx* c, int status, const char* fmt, ...) {
    if (c) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(c->err, sizeof(c->err), fmt, ap);
        va_end(ap);
        if (c->h_guard && *c->h_guard != 0) {   // a kernel watchdog tripped before the CUDA error surfaced: say which
            size_t n = strlen(c->err);
            n += snprintf(c->err + n, sizeof(c->err) - n, " [device watchdog code %d;", *c->h_guard);
            for (int i = 1; i < 65 && n + 24 < sizeof(c->err); i++)   // who else was waiting, and at which row
                if (c->h_guard[i]) n += snprintf(c->err + n, sizeof(c->err) - n, " p%d:%d@%d", (i - 1) / 32, c->h_guard[i] & 255, (c->h_guard[i] >> 8) - 1);
            snprintf(c->err + n, sizeof(c->err) - n, "]");
        }
    }
    return status;
}

int ensure(Ctx* c, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap) return SRCNN_OK;
    drop_graphs(c);   // captured pipelines hold the old device addresses
    if (b.p) {
        SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
        SRCNN_CUDA(c, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    const size_t want = align_up(bytes + bytes / 8, 1 << 20);  // slack so slightly larger frames do not realloc
    SRCNN_CUDA(c, cudaMalloc(&b.p, want));
    b.cap = want;
    return SRCNN_OK;
}

// `which`: 0 before colour+bicubic, 1 after it, 2 after the CNN stage, 3 after the merge.  Mode 2 keeps only the pair around
// the CNN stage: an event between the merge of one call and the colour+bicubic of the next would separate the two kernels
// in the stream and switch their overlap off.
int prof_mark(Ctx* c, int which) {
    if (!c->profiling) return SRCNN_OK;
    if (c->profiling == 2 && which != 1 && which != 2) return SRCNN_OK;
    if (c->ev_used == c->ev_pool.size()) {
        cudaEvent_t e;
        SRCNN_CUDA(c, cudaEventCreate(&e));
        c->ev_pool.push_back(e);
    }
    SRCNN_CUDA(c, cudaEventRecord(c->ev_pool[c->ev_used++], c->stream));
    return SRCNN_OK;
}

static int scaled_dim(int n, float scale) {
    // `newsz.width *= image_multiply` (src/srcnn.cpp:574-575): int -> float multiply -> truncation
    return (int)((float)n * scale);
}

// bytes per pixel of a row (4:2:0: of a Y row; a chroma row of NV12 has as many, an I420 chroma row half as many; packed 4:2:2: 2)
static size_t bytes_per_pixel(int order) {
    return order == SRCNN_ORDER_GRAY || yuv420(order) ? 1 : (yuv422(order) ? 2 : (four_channel(order) ? 4 : 3));
}
// rows of one frame in memory (4:2:0: h rows of Y, then h/2 rows of NV12 pairs or of I420 U and V)
static size_t frame_rows(int order, int h) { return yuv420(order) ? (size_t)h / 2 * 3 : (size_t)h; }

static int check_image(Ctx* c, const void* src, int w, int h, size_t stride, int order, float scale, const void* dst,
                       size_t dst_stride, int* ow, int* oh) {
    if (!c) return SRCNN_E_ARG;
    if (!src || !dst) return fail(c, SRCNN_E_ARG, "null image pointer");
    if (w <= 0 || h <= 0) return fail(c, SRCNN_E_ARG, "non-positive image size %dx%d", w, h);
    if (order != SRCNN_ORDER_BGR && order != SRCNN_ORDER_RGB && order != SRCNN_ORDER_GRAY && !four_channel(order) && !yuv420(order) &&
        !yuv422(order))
        return fail(c, SRCNN_E_ARG, "unknown pixel order %d", order);
    const size_t bpp = bytes_per_pixel(order);
    if (stride < (size_t)w * bpp) return fail(c, SRCNN_E_ARG, "source stride %zu < %zu*w", stride, bpp);
    if (yuv420(order) && ((w | h) & 1)) return fail(c, SRCNN_E_ARG, "4:2:0 frames need an even width and height, got %dx%d", w, h);
    if (yuv422(order) && (w & 1)) return fail(c, SRCNN_E_ARG, "4:2:2 frames need an even width (whole macropixels), got %d", w);
    if (order == SRCNN_ORDER_I420 && ((stride | dst_stride) & 1))
        return fail(c, SRCNN_E_ARG, "I420 strides must be even (chroma rows are stride/2 apart), got %zu / %zu", stride, dst_stride);
    // src/srcnn.cpp:485-495 "ratio too small"
    if (!(((float)w * scale) > 0.f) || !(((float)h * scale) > 0.f)) return fail(c, SRCNN_E_RATIO, "scale %g gives an empty image", scale);
    *ow = scaled_dim(w, scale);
    *oh = scaled_dim(h, scale);
    if (*ow <= 0 || *oh <= 0) return fail(c, SRCNN_E_RATIO, "scale %g gives an empty image", scale);
    if (yuv420(order) && ((*ow | *oh) & 1))
        return fail(c, SRCNN_E_ARG, "scale %g gives an odd 4:2:0 output size %dx%d (width and height must be even)", scale, *ow, *oh);
    if (yuv422(order) && (*ow & 1))
        return fail(c, SRCNN_E_ARG, "scale %g gives an odd 4:2:2 output width %d (whole macropixels: it must be even)", scale, *ow);
    if (dst_stride < (size_t)*ow * bpp) return fail(c, SRCNN_E_ARG, "destination stride %zu < %zu*ow", dst_stride, bpp);
    return SRCNN_OK;
}

// The chroma planes of 4:2:0 frames whose Y rows start at `src` / `dst` (frame 0), for the luma output rows [r0, r1): chroma output
// rows [r0/2, r1/2).  A chroma row is resized without the CNN, so it needs no halo.
static int chroma_planes(Ctx* c, int order, const uint8_t* src, int w, int h, size_t src_stride, uint8_t* dst, int ow, int oh,
                         size_t dst_stride, size_t dst_frame_stride, int r0, int r1, Chroma420* ch) {
    TapTable *tx, *ty;
    int rc = get_taps(c, w / 2, ow / 2, &tx);
    if (rc) return rc;
    if ((rc = get_taps(c, h / 2, oh / 2, &ty))) return rc;
    const bool i420 = order == SRCNN_ORDER_I420;
    ch->src = src + (size_t)h * src_stride;
    ch->src_pitch = i420 ? src_stride / 2 : src_stride;
    ch->src_v = i420 ? (size_t)(h / 2) * (src_stride / 2) : 0;
    ch->dst = dst + (size_t)oh * dst_stride;
    ch->dst_pitch = i420 ? dst_stride / 2 : dst_stride;
    ch->dst_v = i420 ? (size_t)(oh / 2) * (dst_stride / 2) : 0;
    ch->dst_frame = dst_frame_stride;
    ch->sw = w / 2; ch->sh = h / 2; ch->ow = ow / 2; ch->oh = oh / 2;
    ch->row_begin = r0 / 2; ch->row_end = r1 / 2;
    ch->tx = tx; ch->ty = ty;
    return SRCNN_OK;
}

// The chroma planes of packed 4:2:2 frames whose row 0 is at `src` (frame 0), for the output rows [r0, r1): U' and V' go into the
// Cr / Cb planes of `pl` (its first ow/2 columns), which the pack kernel reads for the same rows.  No halo: chroma has no CNN.
static int chroma_planes422(Ctx* c, const uint8_t* src, int w, int h, size_t src_stride, const Planes& pl, int ow, int oh, int r0,
                            int r1, Chroma420* ch) {
    TapTable *tx, *ty;
    int rc = get_taps(c, w / 2, ow / 2, &tx);
    if (rc) return rc;
    if ((rc = get_taps(c, h, oh, &ty))) return rc;
    ch->src = src; ch->src_pitch = src_stride; ch->src_v = 0;
    ch->dst = pl.cr - (ptrdiff_t)pl.row0 * (ptrdiff_t)pl.pitch;   // chroma output row r at dst + r * pitch
    ch->dst_pitch = pl.pitch;
    ch->dst_v = (size_t)(pl.cb - pl.cr);
    ch->dst_frame = pl.frame_stride;
    ch->sw = w / 2; ch->sh = h; ch->ow = ow / 2; ch->oh = oh;
    ch->row_begin = r0; ch->row_end = r1;
    ch->tx = tx; ch->ty = ty;
    return SRCNN_OK;
}

// planes of `nframes` same-sized frames: [Y frames][Cr frames][Cb frames][Y' frames][FP16 Y frames], and for a four-channel
// call [A frames] after them (so the colour and grey layouts do not depend on it)
// Cross-call overlap: the only planes the colour+bicubic kernel of call i+1 writes AND the merge kernel of call i reads are Cr and
// Cb (and A, for four-channel calls), so device-resident whole-path calls alternate between two sets of them (the second in
// plane_buf2, when a set is at most 4 GiB: Cr, Cb and A of a four-channel call); Y, Y' and the FP16 Y plane are shared (the merge
// never reads Y / FP16 Y, and Y' is written by the next CNN launch, which waits for everything before it).  c->plane_sel says which
// set this call got.  Keeping the rest single also keeps the planes L2-resident from step to step: two whole plane sets (116 MB
// at 4K) measured 3 us slower in the colour+bicubic kernel.
// The host-buffer pipeline keeps to set 0 (its sub-bands are separated by copies and events anyway).  A grey or 4:2:0 call has no
// Cr/Cb planes: it leaves the set selection alone (and ends the early-start chain, end_merge_chain).  A packed 4:2:2 call keeps its
// U' / V' planes in the Cr / Cb slots and so takes part like a colour call.
static int carve_planes(Ctx* c, int ow, int rows, int row0, Planes* pl, int nframes = 1, int order = SRCNN_ORDER_BGR) {
    const bool gray = order == SRCNN_ORDER_GRAY || yuv420(order), four = four_channel(order);
    const size_t pitch = align_up((size_t)ow, 128);
    const size_t plane = pitch * (size_t)rows;
    const size_t pitch16 = y16_pitch_bytes(ow);
    const size_t plane16 = align_up(pitch16 * (size_t)rows, 256);
    const size_t nf = (size_t)nframes;
    const size_t nalt = four ? 3 : 2;                         // planes of the alternating set: Cr, Cb (, A)
    // slack: the last row's last strip copy may run past the row
    const size_t bytes = (plane * 4 + plane16) * nf + (four ? plane * nf : 0) + 512;
    const bool two = c->overlap && !c->host_path && !c->capturing && plane * nalt * nf <= ((size_t)4 << 30);
    if (!gray) c->plane_sel = two ? (c->plane_sel ^ 1) : 0;
    int rc = ensure(c, c->plane_buf, bytes);
    if (rc) return rc;
    if (!gray && c->plane_sel && (rc = ensure(c, c->plane_buf2, plane * nalt * nf))) return rc;
    c->plane_layout[0] = pitch; c->plane_layout[1] = (size_t)rows; c->plane_layout[2] = nf;
    uint8_t* base = (uint8_t*)c->plane_buf.p;
    pl->y = base;
    pl->cr = gray ? nullptr : c->plane_sel ? (uint8_t*)c->plane_buf2.p : base + plane * nf;
    pl->cb = gray ? nullptr : c->plane_sel ? (uint8_t*)c->plane_buf2.p + plane * nf : base + 2 * plane * nf;
    pl->a = !four ? nullptr : c->plane_sel ? (uint8_t*)c->plane_buf2.p + 2 * plane * nf : base + (4 * plane + plane16) * nf;
    pl->yout = base + 3 * plane * nf;
    pl->y16 = base + 4 * plane * nf;
    pl->frame_stride = plane;
    pl->frame_stride16 = plane16;
    pl->pitch16 = pitch16;
    pl->pitch = pitch;
    pl->row0 = row0;
    pl->rows = rows;
    return SRCNN_OK;
}

// Which context enqueued the most recent merge kernel on a stream (process-wide: a caller may run several contexts on one stream
// and feed one's result to the other).
static std::mutex g_merge_mu;
static std::unordered_map<cudaStream_t, Ctx*> g_last_merge;
void note_merge(Ctx* c) {
    std::lock_guard<std::mutex> lk(g_merge_mu);
    g_last_merge[c->stream] = c;
}
static Ctx* last_merge_on(cudaStream_t s) {
    std::lock_guard<std::mutex> lk(g_merge_mu);
    auto it = g_last_merge.find(s);
    return it == g_last_merge.end() ? nullptr : it->second;
}
// A grey or 4:2:0 call launches no merge: the kernel that ends up last on the stream does not release its dependents, so neither this
// context's next colour call nor any other context's on this stream may start early.
static void end_merge_chain(Ctx* c) {
    c->merge_sel = -1;
    std::lock_guard<std::mutex> lk(g_merge_mu);
    g_last_merge.erase(c->stream);
}
static void forget_merges_of(Ctx* c) {
    std::lock_guard<std::mutex> lk(g_merge_mu);
    for (auto it = g_last_merge.begin(); it != g_last_merge.end();)
        it = it->second == c ? g_last_merge.erase(it) : std::next(it);
}

// May the colour+bicubic kernel about to be enqueued start while the stream's previous kernel is still running?  Only when that
// kernel is a merge of ours (launch_merge lets its dependents go at once) which reads the OTHER Cr/Cb pair and writes nothing
// this call's source overlaps (a caller may feed one call's result to the next).  Anything the caller put on the stream in
// between simply keeps the usual order: the early start is a property of two adjacent kernels (programmatic dependent launch).
static bool may_start_early(Ctx* c, const uint8_t* src, size_t src_bytes) {
    if (!c->overlap || c->host_path || c->capturing || c->profiling == 1) return false;
    if (c->merge_sel < 0 || c->merge_sel == c->plane_sel || c->merge_stream != c->stream) return false;
    if (last_merge_on(c->stream) != c) return false;   // another context of the process has put a merge on this stream since: its result is unknown here
    // same plane geometry as that call: Y, Y' and the FP16 Y plane are shared, and another layout of the same buffer could put this
    // call's Y where that merge still reads its Y'
    if (c->merge_layout[0] != c->plane_layout[0] || c->merge_layout[1] != c->plane_layout[1] || c->merge_layout[2] != c->plane_layout[2]) return false;
    return src + src_bytes <= c->merge_lo || src >= c->merge_hi;
}
static void merged_into(Ctx* c, const uint8_t* dst, size_t bytes) {   // after the whole-path call's (last) launch_merge
    c->merge_sel = c->plane_sel;
    for (int i = 0; i < 3; i++) c->merge_layout[i] = c->plane_layout[i];
    c->merge_stream = c->stream;
    c->merge_lo = dst;
    c->merge_hi = dst + bytes;
}

static int run_cnn(Ctx* c, int variant, const CnnArgs& a) {
    if (variant == SRCNN_VARIANT_FP32) return launch_cnn_fp32(c, a, nullptr);
    if (variant == SRCNN_VARIANT_TC) return launch_cnn_tc2(c, a);
    return fail(c, SRCNN_E_ARG, "unknown variant %d", variant);
}

// rows [r0,r1) of the full output; d_src holds source rows [s0,s1); d_dst points at output row r0
static int process_rows_impl(Ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int s0, int s1, int order,
                             float scale, int ow, int oh, int r0, int r1, uint8_t* d_dst, size_t dst_stride) {
    TapTable *tx, *ty;
    c->fail_stage = SRCNN_STAGE_COLOR_BICUBIC;
    int rc = get_taps(c, w, ow, &tx);
    if (rc) return rc;
    rc = get_taps(c, h, oh, &ty);
    if (rc) return rc;
    const int p0 = std::max(r0 - 6, 0), p1 = std::min(r1 + 6, oh);  // 6-px halo: 4 (conv1) + 2 (conv3)
    // grey: one-plane resize, then the CNN straight into the caller's rows; no chroma, no merge.  4:2:0: the same for Y, and the
    // resize launch also writes the chroma rows [r0/2, r1/2) straight into the caller's frame (d_dst is its row r0)
    const bool gray = order == SRCNN_ORDER_GRAY || yuv420(order);
    if (gray) end_merge_chain(c);
    Planes pl;
    c->fail_stage = SRCNN_STAGE_PLANES;
    rc = carve_planes(c, ow, p1 - p0, p0, &pl, 1, order);
    if (rc) return rc;
    c->fail_stage = SRCNN_STAGE_COLOR_BICUBIC;
    // the band must bring every source row its taps touch
    const int need0 = std::min(std::max(ty->h_ofs[p0] - 1, 0), h - 1);
    const int need1 = std::min(std::max(ty->h_ofs[p1 - 1] + 2, 0), h - 1) + 1;
    if (s0 > need0 || s1 < need1)
        return fail(c, SRCNN_E_ARG, "band rows [%d,%d) need source rows [%d,%d), got [%d,%d)", r0, r1, need0, need1, s0, s1);

    ResizeArgs ra;
    ra.src = d_src; ra.src_stride = src_stride;
    ra.sw = w; ra.sh = h; ra.src_row0 = s0; ra.src_row1 = s1;
    ra.order = order;
    ra.ow = ow; ra.oh = oh;
    ra.row_begin = p0; ra.row_end = p1;
    ra.pl = pl; ra.tx = tx; ra.ty = ty;
    if (yuv420(order) && (rc = chroma_planes(c, order, d_src - (size_t)s0 * src_stride, w, h, src_stride, d_dst - (size_t)r0 * dst_stride,
                                             ow, oh, dst_stride, 0, r0, r1, &ra.ch)))
        return rc;
    // 4:2:2: chroma rows [r0, r1) only (the pack kernel's); the luma halo rows [p0, r0) and [r1, p1) are the CNN's
    if (yuv422(order) && (rc = chroma_planes422(c, d_src - (size_t)s0 * src_stride, w, h, src_stride, pl, ow, oh, r0, r1, &ra.ch)))
        return rc;
    if (c->variant != SRCNN_VARIANT_TC) ra.pl.y16 = nullptr;      // the strict FP32 kernels read the u8 plane
    ra.early = !gray && may_start_early(c, d_src, (size_t)(s1 - s0) * src_stride);
    c->early_launches += ra.early;
    if ((rc = prof_mark(c, 0))) return rc;
    rc = launch_color_bicubic(c, ra);
    if (rc) return rc;
    if ((rc = prof_mark(c, 1))) return rc;

    c->fail_stage = SRCNN_STAGE_CNN;
    CnnArgs ca;
    ca.y = pl.y; ca.pitch = pl.pitch;
    ca.y16 = pl.y16; ca.pitch16 = pl.pitch16;
    ca.W = ow; ca.H = oh;
    ca.row0 = p0; ca.rows = p1 - p0;
    ca.out_begin = r0; ca.out_end = r1;
    if (gray) { ca.out = d_dst; ca.out_pitch = dst_stride; ca.out_row0 = r0; }
    else { ca.out = pl.yout; ca.out_pitch = pl.pitch; ca.out_row0 = p0; }
    // optionally the row-walking tcgen05 kernel merges Cr/Cb and converts back to BGR in its last epilogue (no Y' plane, no
    // K-C launch); measured slower than the separate launch (byte stores from one-thread-per-column lanes), so off by default
    // (colour orders only: a four-channel call takes the separate merge, which writes alpha too; a 4:2:2 call its pack kernel)
    const bool fused = (order == SRCNN_ORDER_BGR || order == SRCNN_ORDER_RGB) && c->variant == SRCNN_VARIANT_TC && c->fuse_merge;
    if (fused) {
        ca.cr = pl.cr; ca.cb = pl.cb;
        ca.bgr = d_dst; ca.bgr_stride = dst_stride; ca.order = order;
    }
    rc = run_cnn(c, c->variant, ca);
    if (rc) return rc;
    if ((rc = prof_mark(c, 2))) return rc;
    if (fused || gray) return prof_mark(c, 3);

    c->fail_stage = SRCNN_STAGE_MERGE;
    MergeArgs ma;
    const size_t off = (size_t)(r0 - p0) * pl.pitch;
    ma.y = pl.yout + off; ma.cr = pl.cr + off; ma.cb = pl.cb + off;
    if (pl.a) ma.a = pl.a + off;
    ma.pitch = pl.pitch; ma.w = ow; ma.rows = r1 - r0;
    ma.order = order;
    ma.dst = d_dst; ma.dst_stride = dst_stride;
    rc = yuv422(order) ? launch_pack422(c, ma) : launch_merge(c, ma);
    if (rc) return rc;
    merged_into(c, d_dst, (size_t)(r1 - r0) * dst_stride);
    return prof_mark(c, 3);
}

static int process_rows(Ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int s0, int s1, int order,
                        float scale, int ow, int oh, int r0, int r1, uint8_t* d_dst, size_t dst_stride) {
    const size_t ev0 = c->ev_used;
    const int rc = process_rows_impl(c, d_src, w, h, src_stride, s0, s1, order, scale, ow, oh, r0, r1, d_dst, dst_stride);
    if (rc) c->ev_used = ev0;        // a failed band leaves no half-recorded event group behind (srcnn_profile_read pairs by 4)
    else c->fail_stage = SRCNN_STAGE_NONE;
    return rc;
}

// `n` whole frames resident on the device, in chunks whose planes stay below ~1 GB: per chunk ONE launch of each stage -- the
// colour+bicubic grid gets a frame dimension, the row-walking kernel sees the frames as more strips of one work list (no
// per-frame pipeline fill / drain), the merge kernel sees the chunk's planes as one tall image.
static int process_frames_impl(Ctx* c, const uint8_t* d_src, int n, int w, int h, size_t src_stride, size_t src_frame_stride, int order,
                               float scale, int ow, int oh, uint8_t* d_dst, size_t dst_stride, size_t dst_frame_stride) {
    TapTable *tx, *ty;
    c->fail_stage = SRCNN_STAGE_COLOR_BICUBIC;
    int rc = get_taps(c, w, ow, &tx);
    if (rc) return rc;
    if ((rc = get_taps(c, h, oh, &ty))) return rc;
    const size_t per_frame = align_up((size_t)ow, 128) * (size_t)oh * (four_channel(order) ? 5 : 4) + y16_pitch_bytes(ow) * (size_t)oh;
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n, ((size_t)1 << 30) / per_frame));
    const bool gray = order == SRCNN_ORDER_GRAY || yuv420(order);   // the CNN writes into the caller's frames, no merge
    if (gray) end_merge_chain(c);
    for (int f0 = 0; f0 < n; f0 += chunk) {
        const int m = std::min(chunk, n - f0);
        Planes pl;
        c->fail_stage = SRCNN_STAGE_PLANES;
        if ((rc = carve_planes(c, ow, oh, 0, &pl, m, order))) return rc;
        c->fail_stage = SRCNN_STAGE_COLOR_BICUBIC;
        ResizeArgs ra;
        ra.src = d_src + (size_t)f0 * src_frame_stride; ra.src_stride = src_stride;
        ra.sw = w; ra.sh = h; ra.src_row0 = 0; ra.src_row1 = h;
        ra.order = order;
        ra.ow = ow; ra.oh = oh;
        ra.row_begin = 0; ra.row_end = oh;
        ra.pl = pl; ra.tx = tx; ra.ty = ty;
        ra.nframes = m; ra.src_frame_stride = src_frame_stride;
        if (yuv420(order) && (rc = chroma_planes(c, order, ra.src, w, h, src_stride, d_dst + (size_t)f0 * dst_frame_stride, ow, oh, dst_stride,
                                                 dst_frame_stride, 0, oh, &ra.ch)))
            return rc;
        if (yuv422(order) && (rc = chroma_planes422(c, ra.src, w, h, src_stride, pl, ow, oh, 0, oh, &ra.ch))) return rc;
        ra.early = !gray && may_start_early(c, ra.src, (size_t)(m - 1) * src_frame_stride + (size_t)h * src_stride);
        c->early_launches += ra.early;
        if ((rc = prof_mark(c, 0))) return rc;
        if ((rc = launch_color_bicubic(c, ra))) return rc;
        if ((rc = prof_mark(c, 1))) return rc;
        c->fail_stage = SRCNN_STAGE_CNN;
        CnnArgs ca;
        ca.y = pl.y; ca.pitch = pl.pitch;
        ca.y16 = pl.y16; ca.pitch16 = pl.pitch16;
        ca.W = ow; ca.H = oh;
        ca.row0 = 0; ca.rows = oh;
        ca.out_begin = 0; ca.out_end = oh;
        ca.out = pl.yout; ca.out_pitch = pl.pitch;
        ca.nframes = m; ca.y16_frame_stride = pl.frame_stride16; ca.out_frame_stride = pl.frame_stride;
        uint8_t* dst0 = d_dst + (size_t)f0 * dst_frame_stride;
        if (gray) { ca.out = dst0; ca.out_pitch = dst_stride; ca.out_frame_stride = dst_frame_stride; }
        if ((rc = launch_cnn_tc2(c, ca))) return rc;
        if ((rc = prof_mark(c, 2))) return rc;
        if (gray) {
            if ((rc = prof_mark(c, 3))) return rc;
            continue;
        }
        c->fail_stage = SRCNN_STAGE_MERGE;
        MergeArgs ma;
        ma.y = pl.yout; ma.cr = pl.cr; ma.cb = pl.cb; ma.a = pl.a;
        ma.pitch = pl.pitch; ma.w = ow;
        ma.order = order;
        auto merge = [&]() { return yuv422(order) ? launch_pack422(c, ma) : launch_merge(c, ma); };   // 4:2:2: the pack kernel
        if (m == 1 || dst_frame_stride == dst_stride * (size_t)oh) {   // the chunk's results are one tall image too
            ma.rows = oh * m; ma.dst = dst0; ma.dst_stride = dst_stride;
            if ((rc = merge())) return rc;
        } else {
            for (int f = 0; f < m; f++) {
                ma.y = pl.yout + (size_t)f * pl.frame_stride; ma.cr = pl.cr + (size_t)f * pl.frame_stride; ma.cb = pl.cb + (size_t)f * pl.frame_stride;
                if (pl.a) ma.a = pl.a + (size_t)f * pl.frame_stride;
                ma.rows = oh; ma.dst = dst0 + (size_t)f * dst_frame_stride; ma.dst_stride = dst_stride;
                if ((rc = merge())) return rc;
            }
        }
        merged_into(c, dst0, (size_t)(m - 1) * dst_frame_stride + (size_t)oh * dst_stride);
        if ((rc = prof_mark(c, 3))) return rc;
    }
    return SRCNN_OK;
}

static int process_frames(Ctx* c, const uint8_t* d_src, int n, int w, int h, size_t src_stride, size_t src_frame_stride, int order,
                          float scale, int ow, int oh, uint8_t* d_dst, size_t dst_stride, size_t dst_frame_stride) {
    // one launch per stage and chunk needs the row-walking kernel with a separate merge; everything else goes frame by frame
    // (the fused merge only takes the colour orders: grey and four-channel batches stay batched with it switched on)
    const bool fuses = c->fuse_merge && (order == SRCNN_ORDER_BGR || order == SRCNN_ORDER_RGB);
    if (n == 1 || c->variant != SRCNN_VARIANT_TC || fuses || !c->batch_launch) {
        for (int f = 0; f < n; f++) {
            int rc = process_rows(c, d_src + (size_t)f * src_frame_stride, w, h, src_stride, 0, h, order, scale, ow, oh, 0, oh,
                                  d_dst + (size_t)f * dst_frame_stride, dst_stride);
            if (rc) return rc;
        }
        return SRCNN_OK;
    }
    const size_t ev0 = c->ev_used;
    const int rc = process_frames_impl(c, d_src, n, w, h, src_stride, src_frame_stride, order, scale, ow, oh, d_dst, dst_stride, dst_frame_stride);
    if (rc) c->ev_used = ev0;
    else c->fail_stage = SRCNN_STAGE_NONE;
    return rc;
}

static int check_guard(Ctx* c) {
    if (c->h_guard && *c->h_guard != 0) {
        int v = *c->h_guard;
        *c->h_guard = 0;
        return fail(c, SRCNN_E_KERNEL, "device-side pipeline watchdog tripped (code %d)", v);
    }
    return SRCNN_OK;
}


// ---- host-buffer pipeline -------------------------------------------------------------------------
// Output rows [R0, R1) of n same-sized frames: host buffers in, host buffers out.  `src` points at row 0 of frame 0 (the
// whole source image must be addressable: a band reads the source rows its taps touch), `dst` at output row R0 of frame 0.
// Three streams: copy-in (H2D), compute (the context stream), copy-out (D2H).  A unit is one row band of one frame: a
// single frame (or a single band of a gigapixel image) is cut into sub-bands so that its D2H -- 4x the H2D bytes at x2 --
// overlaps the kernels of the next sub-band; frames of a batch overlap the same way.
struct StreamDrain {   // on every exit path: no async copy may still reference the caller's buffers
    Ctx* c;
    ~StreamDrain() {
        if (c->capturing) return;   // a capture is ended (and thrown away) by its owner; nothing has run yet
        if (c->s_in) cudaStreamSynchronize(c->s_in);
        if (c->s_out) cudaStreamSynchronize(c->s_out);
        cudaStreamSynchronize(c->stream);
    }
};

static bool is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

void drop_graphs(Ctx* c) {
    for (auto& g : c->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    c->graphs.clear();
}

// Luma rows [y0, y1) and chroma rows [c0, c1) of one 4:2:0 frame between two buffers whose Y rows are `ds` / `ss` bytes apart
// (w x h: the frame's size).  NV12's chroma rows follow the Y rows with the same stride; I420's U and V rows are half as long.
static int copy_420(Ctx* c, bool i420, uint8_t* dst, size_t ds, const uint8_t* src, size_t ss, int w, int h, int y0, int y1, int c0,
                    int c1, cudaMemcpyKind kind, cudaStream_t st) {
    if (y1 > y0)
        SRCNN_CUDA(c, cudaMemcpy2DAsync(dst + (size_t)y0 * ds, ds, src + (size_t)y0 * ss, ss, (size_t)w, y1 - y0, kind, st));
    if (c1 <= c0) return SRCNN_OK;
    dst += (size_t)h * ds;
    src += (size_t)h * ss;
    if (!i420) {
        SRCNN_CUDA(c, cudaMemcpy2DAsync(dst + (size_t)c0 * ds, ds, src + (size_t)c0 * ss, ss, (size_t)w, c1 - c0, kind, st));
        return SRCNN_OK;
    }
    ds /= 2;
    ss /= 2;
    for (int pl = 0; pl < 2; pl++) {   // U, then V h/2 rows further
        const size_t r = (size_t)(pl * (h / 2) + c0);
        SRCNN_CUDA(c, cudaMemcpy2DAsync(dst + r * ds, ds, src + r * ss, ss, (size_t)w / 2, c1 - c0, kind, st));
    }
    return SRCNN_OK;
}

// Enqueues the whole pipeline of one chunk of frames (f0 .. f0+m) on the three streams and joins the copy streams back
// into the compute stream; does not wait.  Identical whether the streams are live or being captured into a CUDA graph.
static int enqueue_chunk(Ctx* c, const uint8_t* src, int f0, int m, int w, int h, size_t src_stride, size_t src_frame_stride, int order,
                         float scale, int ow, int oh, int R0, int R1, uint8_t* dst, size_t dst_stride, size_t dst_frame_stride,
                         const TapTable* ty, const TapTable* cty, int S0, int S1, const std::vector<int>& edges, int group, size_t s_row, size_t d_row, size_t s_frame,
                         size_t d_frame) {
    const int bands = (int)edges.size() - 1;
    const size_t bpp = bytes_per_pixel(order), w_bytes = (size_t)w * bpp, ow_bytes = (size_t)ow * bpp;
    // 4:2:0: frames are staged whole (S0 = 0, R0 = 0), every row at its place in the frame; a sub-band copies the chroma rows its
    // chroma output rows [r0/2, r1/2) read (chroma tap table cty) along with its Y rows
    const bool yuv = yuv420(order), i420 = order == SRCNN_ORDER_I420;
    const size_t in_rows = yuv ? frame_rows(order, h) : (size_t)(S1 - S0), out_rows = yuv ? frame_rows(order, oh) : (size_t)(R1 - R0);
    int rc;
    uint8_t* ds = (uint8_t*)c->src_buf.p;
    uint8_t* dd = (uint8_t*)c->dst_buf.p;
    auto event_at = [&](size_t i, cudaEvent_t* e) -> int {
        while (c->pipe_events.size() <= i) {
            cudaEvent_t ev;
            SRCNN_CUDA(c, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            c->pipe_events.push_back(ev);
        }
        *e = c->pipe_events[i];
        return SRCNN_OK;
    };
    auto src_hi = [&](int r1) {   // one past the last source row output rows < r1 touch (6-px halo in the output)
        const int p1 = std::min(r1 + 6, oh);
        return std::min(std::max(ty->h_ofs[p1 - 1] + 2, 0), h - 1) + 1;
    };
    const int rows = R1 - R0;
    cudaEvent_t ev_start;
    if ((rc = event_at(0, &ev_start))) return rc;
    size_t ei = 1;
    // everything queued earlier on the compute stream (previous calls, tap-table uploads) precedes the copies
    SRCNN_CUDA(c, cudaEventRecord(ev_start, c->stream));
    SRCNN_CUDA(c, cudaStreamWaitEvent(c->s_in, ev_start, 0));
    SRCNN_CUDA(c, cudaStreamWaitEvent(c->s_out, ev_start, 0));
    if (bands == 1 && m > 1) {
        // A batch of whole frames: groups of frames travel together -- one copy in, ONE launch per stage (process_frames: no
        // per-frame pipeline fill / drain in the fused kernel), one copy out -- sized so that a group's result is >= 64 MB:
        // large copies keep the PCIe link busy, and the next group's kernels still hide behind this group's D2H.
        const bool rows_tight_in = src_stride == w_bytes && s_row == w_bytes;      // a frame is one contiguous run of bytes
        const bool rows_tight_out = dst_stride == ow_bytes && d_row == ow_bytes;
        for (int g0 = 0; g0 < m; g0 += group) {
            const int g = std::min(group, m - g0);
            const uint8_t* hsrc = src + (size_t)(f0 + g0) * src_frame_stride;
            uint8_t* hdst = dst + (size_t)(f0 + g0) * dst_frame_stride;
            cudaEvent_t ev_in, ev_done;
            if ((rc = event_at(ei++, &ev_in))) return rc;
            if (rows_tight_in) {   // frames are the "rows" of one 2-D copy
                SRCNN_CUDA(c, cudaMemcpy2DAsync(ds + (size_t)g0 * s_frame, s_frame, hsrc + (size_t)S0 * src_stride, src_frame_stride,
                                                in_rows * s_row, g, cudaMemcpyHostToDevice, c->s_in));
            } else if (yuv) {
                for (int f = 0; f < g; f++)
                    if ((rc = copy_420(c, i420, ds + (size_t)(g0 + f) * s_frame, s_row, hsrc + (size_t)f * src_frame_stride, src_stride, w, h,
                                       0, h, 0, h / 2, cudaMemcpyHostToDevice, c->s_in)))
                        return rc;
            } else {
                for (int f = 0; f < g; f++)
                    SRCNN_CUDA(c, cudaMemcpy2DAsync(ds + (size_t)(g0 + f) * s_frame, s_row, hsrc + (size_t)f * src_frame_stride + (size_t)S0 * src_stride,
                                                    src_stride, w_bytes, S1 - S0, cudaMemcpyHostToDevice, c->s_in));
            }
            SRCNN_CUDA(c, cudaEventRecord(ev_in, c->s_in));
            SRCNN_CUDA(c, cudaStreamWaitEvent(c->stream, ev_in, 0));
            if (R0 == 0 && R1 == oh) {
                rc = process_frames(c, ds + (size_t)g0 * s_frame, g, w, h, s_row, s_frame, order, scale, ow, oh, dd + (size_t)g0 * d_frame, d_row, d_frame);
                if (rc) return rc;
            } else {
                for (int f = 0; f < g; f++) {
                    rc = process_rows(c, ds + (size_t)(g0 + f) * s_frame, w, h, s_row, S0, S1, order, scale, ow, oh, R0, R1, dd + (size_t)(g0 + f) * d_frame, d_row);
                    if (rc) return rc;
                }
            }
            if ((rc = event_at(ei++, &ev_done))) return rc;
            SRCNN_CUDA(c, cudaEventRecord(ev_done, c->stream));
            SRCNN_CUDA(c, cudaStreamWaitEvent(c->s_out, ev_done, 0));
            if (rows_tight_out) {
                SRCNN_CUDA(c, cudaMemcpy2DAsync(hdst, dst_frame_stride, dd + (size_t)g0 * d_frame, d_frame, out_rows * d_row, g,
                                                cudaMemcpyDeviceToHost, c->s_out));
            } else if (yuv) {
                for (int f = 0; f < g; f++)
                    if ((rc = copy_420(c, i420, hdst + (size_t)f * dst_frame_stride, dst_stride, dd + (size_t)(g0 + f) * d_frame, d_row, ow, oh,
                                       0, oh, 0, oh / 2, cudaMemcpyDeviceToHost, c->s_out)))
                        return rc;
            } else {
                for (int f = 0; f < g; f++)
                    SRCNN_CUDA(c, cudaMemcpy2DAsync(hdst + (size_t)f * dst_frame_stride, dst_stride, dd + (size_t)(g0 + f) * d_frame, d_row, ow_bytes, rows,
                                                    cudaMemcpyDeviceToHost, c->s_out));
            }
        }
    } else
    for (int f = 0; f < m; f++) {
        const uint8_t* hsrc = src + (size_t)(f0 + f) * src_frame_stride;
        uint8_t* hdst = dst + (size_t)(f0 + f) * dst_frame_stride;
        int copied = S0;   // source rows [S0, copied) of this frame are on their way to the device
        int c_copied = 0;  // 4:2:0: chroma source rows [0, c_copied) likewise
        for (int bi = 0; bi < bands; bi++) {
            const int r0 = edges[bi], r1 = edges[bi + 1];
            const int s_hi = bi + 1 < bands ? src_hi(r1) : S1;
            const int c_hi = !yuv ? 0 : bi + 1 < bands ? std::min(std::max(cty->h_ofs[r1 / 2 - 1] + 2, 0), h / 2 - 1) + 1 : h / 2;
            if (s_hi > copied || c_hi > c_copied) {
                cudaEvent_t ev_in;
                if ((rc = event_at(ei++, &ev_in))) return rc;
                if (yuv) {
                    if ((rc = copy_420(c, i420, ds + f * s_frame, s_row, hsrc, src_stride, w, h, copied, s_hi, c_copied, c_hi,
                                       cudaMemcpyHostToDevice, c->s_in)))
                        return rc;
                } else {
                    SRCNN_CUDA(c, cudaMemcpy2DAsync(ds + f * s_frame + (size_t)(copied - S0) * s_row, s_row, hsrc + (size_t)copied * src_stride,
                                                    src_stride, w_bytes, s_hi - copied, cudaMemcpyHostToDevice, c->s_in));
                }
                SRCNN_CUDA(c, cudaEventRecord(ev_in, c->s_in));
                SRCNN_CUDA(c, cudaStreamWaitEvent(c->stream, ev_in, 0));
                copied = std::max(copied, s_hi);
                c_copied = std::max(c_copied, c_hi);
            }
            rc = process_rows(c, ds + f * s_frame, w, h, s_row, S0, S1, order, scale, ow, oh, r0, r1,
                              dd + f * d_frame + (size_t)(r0 - R0) * d_row, d_row);
            if (rc) return rc;
            cudaEvent_t ev_done;
            if ((rc = event_at(ei++, &ev_done))) return rc;
            SRCNN_CUDA(c, cudaEventRecord(ev_done, c->stream));
            SRCNN_CUDA(c, cudaStreamWaitEvent(c->s_out, ev_done, 0));
            if (yuv) {
                if ((rc = copy_420(c, i420, hdst, dst_stride, dd + f * d_frame, d_row, ow, oh, r0, r1, r0 / 2, r1 / 2, cudaMemcpyDeviceToHost,
                                   c->s_out)))
                    return rc;
                continue;
            }
            SRCNN_CUDA(c, cudaMemcpy2DAsync(hdst + (size_t)(r0 - R0) * dst_stride, dst_stride,
                                            dd + f * d_frame + (size_t)(r0 - R0) * d_row, d_row, ow_bytes, r1 - r0,
                                            cudaMemcpyDeviceToHost, c->s_out));
        }
    }
    // join: the compute stream ends after the last copy in either direction
    cudaEvent_t ev_j1, ev_j2;
    if ((rc = event_at(ei++, &ev_j1))) return rc;
    if ((rc = event_at(ei++, &ev_j2))) return rc;
    SRCNN_CUDA(c, cudaEventRecord(ev_j1, c->s_in));
    SRCNN_CUDA(c, cudaEventRecord(ev_j2, c->s_out));
    SRCNN_CUDA(c, cudaStreamWaitEvent(c->stream, ev_j1, 0));
    SRCNN_CUDA(c, cudaStreamWaitEvent(c->stream, ev_j2, 0));
    return SRCNN_OK;
}

int host_pipeline(Ctx* c, const uint8_t* src, int n, int w, int h, size_t src_stride, size_t src_frame_stride, int order,
                  float scale, int ow, int oh, int R0, int R1, uint8_t* dst, size_t dst_stride, size_t dst_frame_stride) {
    int rc;
    struct HostPath {   // the pipeline's sub-bands and groups share Cr/Cb pair 0 (carve_planes) and never start early
        Ctx* c;
        explicit HostPath(Ctx* c_) : c(c_) { c->host_path = true; c->merge_sel = -1; }
        ~HostPath() { c->host_path = false; c->merge_sel = -1; }
    } host_path{c};
    TapTable *ty = nullptr, *tx = nullptr, *cty = nullptr, *ctx_ = nullptr;
    if ((rc = get_taps(c, h, oh, &ty))) return rc;
    if ((rc = get_taps(c, w, ow, &tx))) return rc;      // uploaded here, not inside a graph capture
    const bool yuv = yuv420(order);
    if (yuv && ((rc = get_taps(c, h / 2, oh / 2, &cty)) || (rc = get_taps(c, w / 2, ow / 2, &ctx_)))) return rc;   // chroma
    if (yuv422(order) && (rc = get_taps(c, w / 2, ow / 2, &ctx_))) return rc;   // 4:2:2 chroma (its vertical table is ty)
    auto src_hi = [&](int r1) {
        const int p1 = std::min(r1 + 6, oh);
        return std::min(std::max(ty->h_ofs[p1 - 1] + 2, 0), h - 1) + 1;
    };
    // 4:2:0 frames are staged whole (whole-frame calls only: R0 = 0, R1 = oh), every row at its place in the frame
    const int S0 = yuv ? 0 : std::min(std::max(ty->h_ofs[std::max(R0 - 6, 0)] - 1, 0), h - 1), S1 = yuv ? h : src_hi(R1);
    // device staging: tight rows (4:2:0: 16-byte multiples, so that I420's half-length chroma rows stay 8-byte aligned), 256-byte
    // aligned frames; only the rows this call needs
    const size_t bpp = bytes_per_pixel(order), row_align = yuv ? 16 : 4;
    const size_t s_row = align_up((size_t)w * bpp, row_align), d_row = align_up((size_t)ow * bpp, row_align);
    const size_t s_frame = align_up(s_row * (yuv ? frame_rows(order, h) : (size_t)(S1 - S0)), 256);
    const size_t d_frame = align_up(d_row * (yuv ? frame_rows(order, oh) : (size_t)(R1 - R0)), 256);
    // frames in flight are bounded so staging stays modest (<= 4 GiB of output; one frame may be larger).  Chunks are separated by
    // a full drain of the pipeline, so the bound is generous: 180 GB of HBM is not the scarce resource here.
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n, ((size_t)4 << 30) / d_frame));
    if ((rc = ensure(c, c->src_buf, s_frame * chunk))) return rc;
    if ((rc = ensure(c, c->dst_buf, d_frame * chunk))) return rc;
    if (!c->s_in) {
        SRCNN_CUDA(c, cudaStreamCreateWithFlags(&c->s_in, cudaStreamNonBlocking));
        SRCNN_CUDA(c, cudaStreamCreateWithFlags(&c->s_out, cudaStreamNonBlocking));
    }
    // A single large frame is cut into sub-bands; each sub-band's source rows are copied in separately, so the first one computes
    // after a fraction of the H2D and the D2H stream (the PCIe-bound leg: 4x the H2D bytes at x2) starts early and never idles.
    // The bands GROW: a band's kernels (~25 us of launches and pipeline fill + ~0.09 us per 4K row) only have to finish before
    // the previous band's D2H (~0.21 us per row) does, so a short first band starts the D2H early and longer later bands
    // keep the per-band overhead of the persistent kernel small (equal bands: 8 x 47 us of fused kernel for a frame that takes
    // 147 us whole).  Very tall bands (a gigapixel image) are cut into equal pieces whose planes stay below ~256 MB.
    const int rows = R1 - R0;
    std::vector<int> edges{R0};
    if (n == 1 && rows >= 1024) {
        const long long by_mem = ((long long)rows * (long long)ow * (four_channel(order) ? 5 : 4) + (256ll << 20) - 1) / (256ll << 20);
        if (by_mem > c->host_bands) {
            const int nb = (int)std::min<long long>(by_mem, rows / 64);
            for (int bi = 1; bi < nb; bi++) edges.push_back((R0 + (int)((long long)rows * bi / nb)) & (yuv ? ~1 : ~0));   // 4:2:0: even
        } else if (c->host_bands > 1) {
            double len = c->band_first > 0 ? (double)c->band_first : std::max(256.0, (double)rows / c->host_bands);
            int pos = R0;
            while ((int)edges.size() < c->host_bands) {
                const int take = (int)len & (yuv ? ~1 : ~0);
                if (R1 - (pos + take) < take / 2) break;      // the rest joins the last band
                pos += take;
                edges.push_back(pos);
                len *= c->band_growth;
            }
        }
    }
    edges.push_back(R1);
    const int bands = (int)edges.size() - 1;
    int tallest = 0;
    for (int bi = 0; bi < bands; bi++) tallest = std::max(tallest, edges[bi + 1] - edges[bi]);
    // frames of a batch travel in groups whose result is >= 64 MB (see enqueue_chunk)
    const int group = (int)std::max<size_t>(1, std::min<size_t>(16, ((size_t)64 << 20) / std::max<size_t>(1, (size_t)ow * bpp * (size_t)rows) + 1));
    {   // the planes of the tallest sub-band / of a group of frames, allocated before anything is enqueued or captured
        Planes pl;
        if ((rc = carve_planes(c, ow, std::min(tallest + 12, oh), 0, &pl, (bands == 1 && n > 1) ? std::min(group, n) : 1, order)))
            return rc;
    }

    // ---- CUDA-graph replay.  A call that repeats an earlier one exactly (same buffers, same geometry: a stream of frames through
    // a pair of pinned buffers) is ~50 API calls of host work for ~0.5 ms of device work; the second time a call is seen its
    // pipeline is captured into a graph, from then on it is one cudaGraphLaunch.  One-off calls never pay for instantiation.
    PipeGraph* hit = nullptr;
    const bool graphable = c->use_graphs && !c->profiling && chunk >= n && bands * n <= 256;
    if (graphable) {
        PipeKey key{src, dst, n, w, h, src_stride, src_frame_stride, order, scale, R0, R1, dst_stride, dst_frame_stride, c->variant,
                    (int)c->fuse_merge, c->host_bands * 4096 + c->band_first, c->tc2_seg_ovh + (int)(c->band_growth * 1000.0) * 256, (void*)c->stream};
        for (auto& g : c->graphs)
            if (g.key == key) hit = &g;
        if (!hit) {
            if (c->graphs.size() >= 8) {   // forget the least recently used
                size_t v = 0;
                for (size_t i = 1; i < c->graphs.size(); i++)
                    if (c->graphs[i].stamp < c->graphs[v].stamp) v = i;
                if (c->graphs[v].exec) cudaGraphExecDestroy(c->graphs[v].exec);
                c->graphs.erase(c->graphs.begin() + v);
            }
            PipeGraph g;
            g.key = key;
            c->graphs.push_back(g);          // first sighting: run it live below
            hit = nullptr;
        } else {
            hit->stamp = ++c->graph_clock;
        }
    }
    if (hit && !hit->exec && !hit->failed && is_pinned(src) && is_pinned(dst)) {
        // second sighting: capture.  Nothing below allocates, uploads or synchronises (tables, staging and planes exist).
        cudaGraph_t graph = nullptr;
        const long long launches_before = c->launches;   // capturing enqueues nothing: the launch counter must not move
        cudaError_t e = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal);
        if (e == cudaSuccess) {
            c->capturing = true;
            rc = enqueue_chunk(c, src, 0, n, w, h, src_stride, src_frame_stride, order, scale, ow, oh, R0, R1, dst, dst_stride,
                               dst_frame_stride, ty, cty, S0, S1, edges, group, s_row, d_row, s_frame, d_frame);
            e = cudaStreamEndCapture(c->stream, &graph);
            c->capturing = false;
            if (rc == SRCNN_OK && e == cudaSuccess && graph && cudaGraphInstantiate(&hit->exec, graph, 0) != cudaSuccess) hit->exec = nullptr;
            if (graph) cudaGraphDestroy(graph);
        }
        cudaGetLastError();
        c->launches = launches_before;
        if (!hit->exec) hit->failed = true;   // run live from now on
    }
    StreamDrain drain{c};
    if (hit && hit->exec) {
        SRCNN_CUDA(c, cudaGraphLaunch(hit->exec, c->stream));
        c->launches += hit->kernel_launches;
        SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
        return check_guard(c);
    }
    for (int f0 = 0; f0 < n; f0 += chunk) {
        const int m = std::min(chunk, n - f0);
        const long long l0 = c->launches;
        rc = enqueue_chunk(c, src, f0, m, w, h, src_stride, src_frame_stride, order, scale, ow, oh, R0, R1, dst, dst_stride,
                           dst_frame_stride, ty, cty, S0, S1, edges, group, s_row, d_row, s_frame, d_frame);
        if (rc) return rc;
        if (graphable && f0 == 0)
            for (auto& g : c->graphs)
                if (!g.exec && g.kernel_launches == 0) g.kernel_launches = c->launches - l0;   // what a replay of this call launches
        SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
        rc = check_guard(c);
        if (rc) return rc;
    }
    return SRCNN_OK;
}

}  // namespace srcnn

using namespace srcnn;

// Every entry point runs on the context's device and puts the caller's current device back on return (a host
// application -- PyTorch, for one -- keeps its own notion of the current device).
#define ENTER(ctx)                                                                                              \
    if (!(ctx)) return SRCNN_E_ARG;                                                                             \
    srcnn::DeviceScope dev_scope__((ctx)->device);                                                              \
    if (!dev_scope__.ok) return fail((ctx), SRCNN_E_CUDA, "cudaSetDevice(%d) failed", (ctx)->device)
// the whole-path calls also report a watchdog trip of an EARLIER launch (callers that synchronise through their own
// stream never pass srcnn_sync)
#define ENTER_PROCESS(ctx)                                                                                      \
    ENTER(ctx);                                                                                                 \
    do {                                                                                                        \
        int g__ = check_guard(ctx);                                                                             \
        if (g__) return g__;                                                                                    \
        if ((ctx)->profiling) (ctx)->prof_calls++;                                                              \
    } while (0)

extern "C" {

int srcnn_abi_version(void) { return SRCNN_B200_ABI_VERSION; }

const char* srcnn_strerror(int s) {
    switch (s) {
        case SRCNN_OK: return "ok";
        case SRCNN_E_RATIO: return "image scale error: ratio too small";
        case SRCNN_E_ARG: return "invalid argument";
        case SRCNN_E_NODEVICE: return "no usable CUDA device (sm_100 required; there is no CPU fallback)";
        case SRCNN_E_CUDA: return "CUDA error";
        case SRCNN_E_NOMEM: return "out of device or pinned memory";
        case SRCNN_E_KERNEL: return "device-side guard tripped";
        default: return "unknown status";
    }
}

int srcnn_create(srcnn_ctx** out, int device, int variant) {
    if (!out) return SRCNN_E_ARG;
    *out = nullptr;
    if (variant != SRCNN_VARIANT_TC && variant != SRCNN_VARIANT_FP32) return SRCNN_E_ARG;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
        cudaGetLastError();
        return SRCNN_E_NODEVICE;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return SRCNN_E_NODEVICE;
    if (prop.major != 10) return SRCNN_E_NODEVICE;  // the only code in this library is sm_100a SASS
    srcnn::DeviceScope scope(device);
    if (!scope.ok) return SRCNN_E_NODEVICE;
    srcnn_ctx* c = new (std::nothrow) srcnn_ctx();
    if (!c) return SRCNN_E_NOMEM;
    c->device = device;
    c->variant = variant;
    c->sm_count = prop.multiProcessorCount;
    c->cc_major = prop.major;
    c->cc_minor = prop.minor;
    auto bail = [&](int rc) { srcnn_destroy(c); return rc; };
    if (cudaStreamCreateWithFlags(&c->own, cudaStreamNonBlocking) != cudaSuccess) return bail(SRCNN_E_CUDA);
    c->stream = c->own;
    c->own_stream = true;
    if (srcnn_weights_blob_size != sizeof(float) * kNumParams) return bail(SRCNN_E_ARG);
    if (cudaMalloc(&c->d_params, sizeof(float) * kNumParams) != cudaSuccess) return bail(SRCNN_E_NOMEM);
    if (cudaMemcpyAsync(c->d_params, srcnn_weights_blob, sizeof(float) * kNumParams, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) return bail(SRCNN_E_CUDA);
    if (cudaHostAlloc((void**)&c->h_guard, 128 * sizeof(int), cudaHostAllocMapped) != cudaSuccess) return bail(SRCNN_E_NOMEM);
    memset(c->h_guard, 0, 128 * sizeof(int));
    if (cudaHostGetDevicePointer((void**)&c->d_guard, c->h_guard, 0) != cudaSuccess) return bail(SRCNN_E_CUDA);
    int rc = fp32_prepare(c);
    if (rc) return bail(rc);
    rc = tc2_prepare_weights(c, (const float*)srcnn_weights_blob);
    if (rc) return bail(rc);
    // every upload above came from pageable memory (the embedded blob, a std::vector): such a copy may return before its
    // DMA has landed, and the context's non-blocking stream is not ordered against the legacy stream.  One device-wide
    // synchronisation here and the first launch -- on whatever stream -- sees the parameters.
    if (cudaDeviceSynchronize() != cudaSuccess) return bail(SRCNN_E_CUDA);
    if (const char* k = getenv("SRCNN_FUSE_MERGE")) c->fuse_merge = atoi(k) != 0;
    if (const char* k = getenv("SRCNN_TC2_SEG_OVH")) c->tc2_seg_ovh = std::max(0, std::min(64, atoi(k)));   // tuning aid
    if (const char* k = getenv("SRCNN_BATCH_LAUNCH")) c->batch_launch = atoi(k) != 0;                        // A/B aid
    if (const char* k = getenv("SRCNN_KA_INT")) c->ka_int = atoi(k) != 0;                                    // A/B aid
    if (const char* k = getenv("SRCNN_KA_ISR")) c->ka_int_isr = atoi(k);                                     // A/B aid
    if (const char* k = getenv("SRCNN_GRAPHS")) c->use_graphs = atoi(k) != 0;                                // A/B aid
    if (const char* k = getenv("SRCNN_OVERLAP")) c->overlap = atoi(k) != 0;                                  // A/B aid
    if (const char* k = getenv("SRCNN_MERGE_CTAS")) c->merge_ctas_per_sm = std::max(0, std::min(64, atoi(k))); // tuning aid
    if (const char* k = getenv("SRCNN_BAND_FIRST")) c->band_first = std::max(0, atoi(k));                       // tuning aids: rows of the first
    if (const char* k = getenv("SRCNN_BAND_GROWTH")) c->band_growth = std::max(1.0, std::min(4.0, atof(k)));   // sub-band, growth per band
    if (const char* k = getenv("SRCNN_HOST_BANDS")) c->host_bands = std::max(1, std::min(64, atoi(k)));     // tuning aid
    *out = c;
    return SRCNN_OK;
}

int srcnn_destroy(srcnn_ctx* c) {
    if (!c) return SRCNN_E_ARG;
    srcnn::DeviceScope scope(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    forget_merges_of(c);
    drop_graphs(c);
    tc2_release(c);
    fraw_release(c);
    for (auto& t : c->taps) {
        if (t.d_ofs) cudaFree(t.d_ofs);
        if (t.d_coef) cudaFree(t.d_coef);
    }
    for (DevBuf* b : {&c->plane_buf, &c->plane_buf2, &c->y16_buf, &c->act2_buf, &c->src_buf, &c->dst_buf, &c->work_buf})
        if (b->p) cudaFree(b->p);
    for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
    for (cudaEvent_t e : c->pipe_events) cudaEventDestroy(e);
    if (c->s_in) cudaStreamDestroy(c->s_in);
    if (c->s_out) cudaStreamDestroy(c->s_out);
    if (c->d_params) cudaFree(c->d_params);
    if (c->h_guard) cudaFreeHost(c->h_guard);
    if (c->own) cudaStreamDestroy(c->own);
    cudaGetLastError();
    delete c;
    return SRCNN_OK;
}

const char* srcnn_last_error(srcnn_ctx* c) { return c ? c->err : "null context"; }
int srcnn_last_failed_stage(srcnn_ctx* c) { return c ? c->fail_stage : SRCNN_E_ARG; }

int srcnn_set_variant(srcnn_ctx* c, int variant) {
    if (!c || (variant != SRCNN_VARIANT_TC && variant != SRCNN_VARIANT_FP32)) return SRCNN_E_ARG;
    c->variant = variant;
    return SRCNN_OK;
}
int srcnn_get_variant(srcnn_ctx* c) { return c ? c->variant : SRCNN_E_ARG; }
int srcnn_get_device(srcnn_ctx* c) { return c ? c->device : SRCNN_E_ARG; }

// test hook: 1 = merge + colour-back fused into the tcgen05 kernel, 0 = separate K-C launch (default)
extern "C" __attribute__((visibility("default"))) int srcnn_debug_set_fuse_merge(srcnn_ctx* c, int on) {
    if (!c) return SRCNN_E_ARG;
    c->fuse_merge = on != 0;
    return SRCNN_OK;
}

// test hooks: the row-walking kernel's work cut (pure host arithmetic, callable without a GPU) and its segment-cost knob
extern "C" __attribute__((visibility("default"))) int srcnn_debug_tc2_partition(int nstrips, int hb, int nworkers, int ovh, long long* bounds) {
    if (nstrips <= 0 || hb <= 0 || nworkers <= 0 || !bounds) return SRCNN_E_ARG;
    srcnn::tc2_partition(nstrips, hb, nworkers, ovh, bounds);
    return SRCNN_OK;
}
// the row-walking kernel's packed FP16 operand image (host code only, no device needed): `bytes` must be tc2_weight_bytes()
extern "C" __attribute__((visibility("default"))) int srcnn_debug_tc2_weights(uint8_t* img, size_t bytes) {
    if (!img || bytes != srcnn::tc2_weight_bytes()) return SRCNN_E_ARG;
    srcnn::tc2_pack_weights((const float*)srcnn_weights_blob, img);
    return SRCNN_OK;
}
// the colour+bicubic kernels' tap table for one axis (build_cubic_taps, host code only): ofs[dst], coef[4 * dst]
extern "C" __attribute__((visibility("default"))) int srcnn_debug_cubic_taps(int src, int dst, int* ofs, int16_t* coef) {
    if (src <= 0 || dst <= 0 || !ofs || !coef) return SRCNN_E_ARG;
    std::vector<short4> c((size_t)dst);
    srcnn::build_cubic_taps(src, dst, ofs, c.data());
    for (int d = 0; d < dst; d++) {
        coef[4 * d] = c[d].x; coef[4 * d + 1] = c[d].y; coef[4 * d + 2] = c[d].z; coef[4 * d + 3] = c[d].w;
    }
    return SRCNN_OK;
}
extern "C" __attribute__((visibility("default"))) int srcnn_debug_set_tc2_seg_ovh(srcnn_ctx* c, int ovh) {
    if (!c || ovh < 0 || ovh > 64) return SRCNN_E_ARG;
    c->tc2_seg_ovh = ovh;
    return SRCNN_OK;
}
extern "C" __attribute__((visibility("default"))) int srcnn_debug_set_host_bands(srcnn_ctx* c, int bands) {
    if (!c || bands < 1 || bands > 64) return SRCNN_E_ARG;
    c->host_bands = bands;
    return SRCNN_OK;
}
// tuning hook: rows of the first sub-band of a single host frame (0 = rows / host_bands, at least 256) and the growth per band
extern "C" __attribute__((visibility("default"))) int srcnn_debug_set_band_schedule(srcnn_ctx* c, int first_rows, double growth) {
    if (!c || first_rows < 0 || !(growth >= 1.0 && growth <= 4.0)) return SRCNN_E_ARG;
    c->band_first = first_rows;
    c->band_growth = growth;
    return SRCNN_OK;
}
// test hook: a device-resident batch as one launch per stage and chunk (default) or frame by frame
extern "C" __attribute__((visibility("default"))) int srcnn_debug_set_batch_launch(srcnn_ctx* c, int on) {
    if (!c) return SRCNN_E_ARG;
    c->batch_launch = on != 0;
    return SRCNN_OK;
}
// test hook: cross-call overlap (two Cr/Cb pairs; colour+bicubic of call i+1 beside the merge of call i) on / off; returns
// how many colour+bicubic launches so far were allowed to start early
extern "C" __attribute__((visibility("default"))) long long srcnn_debug_overlap(srcnn_ctx* c, int on) {
    if (!c) return SRCNN_E_ARG;
    if (on >= 0) { c->overlap = on != 0; c->merge_sel = -1; }
    return c->early_launches;
}
// test hook: CUDA-graph replay of repeated host-buffer calls on / off; returns the number of instantiated graphs
extern "C" __attribute__((visibility("default"))) int srcnn_debug_graphs(srcnn_ctx* c, int on) {
    if (!c) return SRCNN_E_ARG;
    if (on >= 0) c->use_graphs = on != 0;
    int n = 0;
    for (auto& g : c->graphs) n += g.exec != nullptr;
    return n;
}

int srcnn_set_stream(srcnn_ctx* c, void* s) {
    ENTER(c);
    SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
    drop_graphs(c);
    if (s) { c->stream = (cudaStream_t)s; c->own_stream = false; }
    else { c->stream = c->own; c->own_stream = true; }
    return SRCNN_OK;
}
void* srcnn_get_stream(srcnn_ctx* c) { return c ? (void*)c->stream : nullptr; }

int srcnn_sync(srcnn_ctx* c) {
    ENTER(c);
    SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_guard(c);
}

long long srcnn_launch_count(srcnn_ctx* c) { return c ? c->launches : -1; }
int srcnn_device_sm_count(srcnn_ctx* c) { return c ? c->sm_count : SRCNN_E_ARG; }

int srcnn_profile_enable(srcnn_ctx* c, int on) {
    ENTER(c);
    SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
    c->profiling = on == 2 ? 2 : (on != 0);
    c->ev_used = 0;
    c->prof_calls = 0;
    return SRCNN_OK;
}

// Sums the device time of the three stages over every band processed since the last read:
// ms[0] colour+bicubic, ms[1] fused SRCNN, ms[2] merge+colour-back; *calls = number of whole-path API calls.
// Mode 2 (events around the CNN stage only): ms[1] as above; ms[0] = the time BETWEEN consecutive CNN launches, i.e. the merge
// of one call and the colour+bicubic of the next running side by side (n - 1 intervals for n launches); ms[2] = 0.
int srcnn_profile_read(srcnn_ctx* c, double* ms, int* calls) {
    ENTER(c);
    if (!ms || !calls) return fail(c, SRCNN_E_ARG, "null pointer");
    SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
    ms[0] = ms[1] = ms[2] = 0.0;
    if (c->profiling == 2) {
        const size_t n = c->ev_used / 2;
        for (size_t i = 0; i < n; i++) {
            float t = 0.f;
            SRCNN_CUDA(c, cudaEventElapsedTime(&t, c->ev_pool[2 * i], c->ev_pool[2 * i + 1]));
            ms[1] += t;
            if (i + 1 < n) {
                SRCNN_CUDA(c, cudaEventElapsedTime(&t, c->ev_pool[2 * i + 1], c->ev_pool[2 * i + 2]));
                ms[0] += t;
            }
        }
    } else {
        const size_t n = c->ev_used / 4;
        for (size_t i = 0; i < n; i++)
            for (int k = 0; k < 3; k++) {
                float t = 0.f;
                SRCNN_CUDA(c, cudaEventElapsedTime(&t, c->ev_pool[4 * i + k], c->ev_pool[4 * i + k + 1]));
                ms[k] += t;
            }
    }
    *calls = c->prof_calls;
    c->ev_used = 0;
    c->prof_calls = 0;
    return SRCNN_OK;
}

int srcnn_out_dims(int w, int h, float scale, int* ow, int* oh) {
    if (!ow || !oh || w <= 0 || h <= 0) return SRCNN_E_ARG;
    if (!(((float)w * scale) > 0.f) || !(((float)h * scale) > 0.f)) return SRCNN_E_RATIO;
    *ow = scaled_dim(w, scale);
    *oh = scaled_dim(h, scale);
    return (*ow > 0 && *oh > 0) ? SRCNN_OK : SRCNN_E_RATIO;
}

int srcnn_host_alloc(void** p, size_t bytes) {
    if (!p) return SRCNN_E_ARG;
    // portable: page-locked for every device of the process (the multi-GPU driver copies from one buffer to all of them)
    cudaError_t e = cudaHostAlloc(p, bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) { cudaGetLastError(); *p = nullptr; return SRCNN_E_NOMEM; }
    return SRCNN_OK;
}
int srcnn_host_free(void* p) {
    if (!p) return SRCNN_OK;
    return cudaFreeHost(p) == cudaSuccess ? SRCNN_OK : SRCNN_E_CUDA;
}
int srcnn_host_register(void* p, size_t bytes) {
    if (!p || !bytes) return SRCNN_E_ARG;
    cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) { cudaGetLastError(); return e == cudaErrorMemoryAllocation ? SRCNN_E_NOMEM : SRCNN_E_CUDA; }
    return SRCNN_OK;
}
int srcnn_host_unregister(void* p) {
    if (!p) return SRCNN_OK;
    if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return SRCNN_E_CUDA; }
    return SRCNN_OK;
}

int srcnn_process_device(srcnn_ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int order, float scale,
                         uint8_t* d_dst, size_t dst_stride) {
    ENTER_PROCESS(c);
    int ow, oh;
    int rc = check_image(c, d_src, w, h, src_stride, order, scale, d_dst, dst_stride, &ow, &oh);
    if (rc) return rc;
    return process_rows(c, d_src, w, h, src_stride, 0, h, order, scale, ow, oh, 0, oh, d_dst, dst_stride);
}

int srcnn_process_batch_device(srcnn_ctx* c, const uint8_t* d_src, int n, int w, int h, size_t src_stride,
                               size_t src_frame_stride, int order, float scale, uint8_t* d_dst, size_t dst_stride,
                               size_t dst_frame_stride) {
    ENTER_PROCESS(c);
    if (n < 0) return fail(c, SRCNN_E_ARG, "negative frame count");
    if (n == 0) return SRCNN_OK;
    int ow, oh;
    int rc = check_image(c, d_src, w, h, src_stride, order, scale, d_dst, dst_stride, &ow, &oh);
    if (rc) return rc;
    if (n > 1 && (src_frame_stride < src_stride * frame_rows(order, h) || dst_frame_stride < dst_stride * frame_rows(order, oh)))
        return fail(c, SRCNN_E_ARG, "frame stride smaller than one frame");
    return process_frames(c, d_src, n, w, h, src_stride, src_frame_stride, order, scale, ow, oh, d_dst, dst_stride, dst_frame_stride);
}

int srcnn_process_batch_host(srcnn_ctx* c, const uint8_t* src, int n, int w, int h, size_t src_stride,
                             size_t src_frame_stride, int order, float scale, uint8_t* dst, size_t dst_stride,
                             size_t dst_frame_stride) {
    ENTER_PROCESS(c);
    if (n < 0) return fail(c, SRCNN_E_ARG, "negative frame count");
    if (n == 0) return SRCNN_OK;
    int ow, oh;
    int rc = check_image(c, src, w, h, src_stride, order, scale, dst, dst_stride, &ow, &oh);
    if (rc) return rc;
    if (n > 1 && (src_frame_stride < src_stride * frame_rows(order, h) || dst_frame_stride < dst_stride * frame_rows(order, oh)))
        return fail(c, SRCNN_E_ARG, "frame stride smaller than one frame");
    return host_pipeline(c, src, n, w, h, src_stride, src_frame_stride, order, scale, ow, oh, 0, oh, dst, dst_stride, dst_frame_stride);
}

int srcnn_process_host(srcnn_ctx* c, const uint8_t* src, int w, int h, size_t src_stride, int order, float scale,
                       uint8_t* dst, size_t dst_stride) {
    return srcnn_process_batch_host(c, src, 1, w, h, src_stride, 0, order, scale, dst, dst_stride, 0);
}

int srcnn_band_src_rows(int h, float scale, int r0, int r1, int* s0, int* s1) {
    if (!s0 || !s1 || h <= 0) return SRCNN_E_ARG;
    if (!(((float)h * scale) > 0.f)) return SRCNN_E_RATIO;
    const int oh = scaled_dim(h, scale);
    if (oh <= 0) return SRCNN_E_RATIO;
    if (r0 < 0 || r1 > oh || r0 >= r1) return SRCNN_E_ARG;
    const int p0 = std::max(r0 - 6, 0), p1 = std::min(r1 + 6, oh);
    std::vector<int> ofs(oh);
    std::vector<short4> coef(oh);
    build_cubic_taps(h, oh, ofs.data(), coef.data());
    *s0 = std::min(std::max(ofs[p0] - 1, 0), h - 1);
    *s1 = std::min(std::max(ofs[p1 - 1] + 2, 0), h - 1) + 1;
    return SRCNN_OK;
}

int srcnn_process_band_device(srcnn_ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int s0, int s1,
                              int order, float scale, int r0, int r1, uint8_t* d_dst, size_t dst_stride) {
    ENTER_PROCESS(c);
    int ow, oh;
    int rc = check_image(c, d_src, w, h, src_stride, order, scale, d_dst, dst_stride, &ow, &oh);
    if (rc) return rc;
    if (yuv420(order)) return fail(c, SRCNN_E_ARG, "4:2:0 frames are whole-frame calls only (no band calls)");
    if (r0 < 0 || r1 > oh || r0 >= r1) return fail(c, SRCNN_E_ARG, "bad output band [%d,%d) of %d rows", r0, r1, oh);
    if (s0 < 0 || s1 > h || s0 >= s1) return fail(c, SRCNN_E_ARG, "bad source band [%d,%d) of %d rows", s0, s1, h);
    return process_rows(c, d_src, w, h, src_stride, s0, s1, order, scale, ow, oh, r0, r1, d_dst, dst_stride);
}

int srcnn_process_band_host(srcnn_ctx* c, const uint8_t* src, int w, int h, size_t src_stride, int order, float scale,
                            int r0, int r1, uint8_t* dst_rows, size_t dst_stride) {
    ENTER_PROCESS(c);
    int ow, oh;
    int rc = check_image(c, src, w, h, src_stride, order, scale, dst_rows, dst_stride, &ow, &oh);
    if (rc) return rc;
    if (yuv420(order)) return fail(c, SRCNN_E_ARG, "4:2:0 frames are whole-frame calls only (no band calls)");
    if (r0 < 0 || r1 > oh || r0 >= r1) return fail(c, SRCNN_E_ARG, "bad output band [%d,%d) of %d rows", r0, r1, oh);
    return host_pipeline(c, src, 1, w, h, src_stride, 0, order, scale, ow, oh, r0, r1, dst_rows, dst_stride, 0);
}

int srcnn_stage_color_bicubic_device(srcnn_ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int order,
                                     float scale, uint8_t* d_y, uint8_t* d_cr, uint8_t* d_cb, size_t plane_pitch) {
    ENTER(c);
    if (!d_src || !d_y || !d_cr || !d_cb) return fail(c, SRCNN_E_ARG, "null pointer");
    if (order != SRCNN_ORDER_BGR && order != SRCNN_ORDER_RGB) return fail(c, SRCNN_E_ARG, "colour order expected, got %d", order);
    if (w <= 0 || h <= 0 || src_stride < (size_t)w * 3) return fail(c, SRCNN_E_ARG, "bad source geometry");
    if (!(((float)w * scale) > 0.f) || !(((float)h * scale) > 0.f)) return fail(c, SRCNN_E_RATIO, "ratio too small");
    const int ow = scaled_dim(w, scale), oh = scaled_dim(h, scale);
    if (ow <= 0 || oh <= 0) return fail(c, SRCNN_E_RATIO, "ratio too small");
    if (plane_pitch < align_up((size_t)ow, 4) || (plane_pitch & 3) || (((uintptr_t)d_y | (uintptr_t)d_cr | (uintptr_t)d_cb) & 3))
        return fail(c, SRCNN_E_ARG, "planes must be 4-byte aligned with pitch a multiple of 4 and >= ow rounded up to 4");
    TapTable *tx, *ty;
    int rc = get_taps(c, w, ow, &tx);
    if (rc) return rc;
    rc = get_taps(c, h, oh, &ty);
    if (rc) return rc;
    ResizeArgs ra;
    ra.src = d_src; ra.src_stride = src_stride;
    ra.sw = w; ra.sh = h; ra.src_row0 = 0; ra.src_row1 = h;
    ra.order = order; ra.ow = ow; ra.oh = oh;
    ra.row_begin = 0; ra.row_end = oh;
    ra.pl.y = d_y; ra.pl.cr = d_cr; ra.pl.cb = d_cb; ra.pl.yout = nullptr; ra.pl.y16 = nullptr;
    ra.pl.pitch = plane_pitch; ra.pl.row0 = 0; ra.pl.rows = oh;
    ra.tx = tx; ra.ty = ty;
    return launch_color_bicubic(c, ra);
}

// One 8-bit plane through cv::resize(..., INTER_CUBIC) (src/srcnn.cpp:577-582): the one-plane resize kernels.  Device buffers,
// enqueued; d_dst must be 4-byte aligned with a pitch that is a multiple of 4 (the tiled kernel's word stores).
static int resize_plane(Ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int ow, int oh, uint8_t* d_dst,
                        size_t dst_stride) {
    TapTable *tx, *ty;
    int rc = get_taps(c, w, ow, &tx);
    if (rc) return rc;
    if ((rc = get_taps(c, h, oh, &ty))) return rc;
    ResizeArgs ra;
    ra.src = d_src; ra.src_stride = src_stride;
    ra.sw = w; ra.sh = h; ra.src_row0 = 0; ra.src_row1 = h;
    ra.order = SRCNN_ORDER_GRAY; ra.ow = ow; ra.oh = oh;
    ra.row_begin = 0; ra.row_end = oh;
    ra.pl.y = d_dst; ra.pl.pitch = dst_stride; ra.pl.row0 = 0; ra.pl.rows = oh;
    ra.tx = tx; ra.ty = ty;
    return launch_color_bicubic(c, ra);
}

static int check_plane(Ctx* c, const void* src, int w, int h, size_t src_stride, float scale, const void* dst, size_t dst_stride,
                       int* ow, int* oh) {
    if (!src || !dst) return fail(c, SRCNN_E_ARG, "null pointer");
    if (w <= 0 || h <= 0 || src_stride < (size_t)w) return fail(c, SRCNN_E_ARG, "bad source geometry");
    if (!(((float)w * scale) > 0.f) || !(((float)h * scale) > 0.f)) return fail(c, SRCNN_E_RATIO, "ratio too small");
    *ow = scaled_dim(w, scale);
    *oh = scaled_dim(h, scale);
    if (*ow <= 0 || *oh <= 0) return fail(c, SRCNN_E_RATIO, "ratio too small");
    if (dst_stride < (size_t)*ow) return fail(c, SRCNN_E_ARG, "destination stride %zu < ow", dst_stride);
    return SRCNN_OK;
}

int srcnn_stage_resize_plane_device(srcnn_ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, float scale,
                                    uint8_t* d_dst, size_t dst_stride) {
    ENTER(c);
    int ow, oh;
    int rc = check_plane(c, d_src, w, h, src_stride, scale, d_dst, dst_stride, &ow, &oh);
    if (rc) return rc;
    if ((((uintptr_t)d_dst | dst_stride) & 3) == 0) return resize_plane(c, d_src, w, h, src_stride, ow, oh, d_dst, dst_stride);
    // a destination the word stores cannot take: resize into the staging buffer, then one device copy
    const size_t pitch = align_up((size_t)ow, 128);
    if ((rc = ensure(c, c->dst_buf, pitch * (size_t)oh))) return rc;
    if ((rc = resize_plane(c, d_src, w, h, src_stride, ow, oh, (uint8_t*)c->dst_buf.p, pitch))) return rc;
    SRCNN_CUDA(c, cudaMemcpy2DAsync(d_dst, dst_stride, c->dst_buf.p, pitch, (size_t)ow, oh, cudaMemcpyDeviceToDevice, c->stream));
    return SRCNN_OK;
}

// Host buffers (ProcessSRCNN's alpha): copy the plane in, resize, copy the result out.
int srcnn_resize_plane_host(srcnn_ctx* c, const uint8_t* src, int w, int h, size_t src_stride, float scale, uint8_t* dst,
                            size_t dst_stride) {
    ENTER(c);
    int ow, oh;
    int rc = check_plane(c, src, w, h, src_stride, scale, dst, dst_stride, &ow, &oh);
    if (rc) return rc;
    const size_t s_pitch = align_up((size_t)w, 4), d_pitch = align_up((size_t)ow, 128);
    if ((rc = ensure(c, c->src_buf, s_pitch * (size_t)h))) return rc;
    if ((rc = ensure(c, c->dst_buf, d_pitch * (size_t)oh))) return rc;
    StreamDrain drain{c};   // no copy may still reference the caller's buffers when this returns
    SRCNN_CUDA(c, cudaMemcpy2DAsync(c->src_buf.p, s_pitch, src, src_stride, (size_t)w, h, cudaMemcpyHostToDevice, c->stream));
    if ((rc = resize_plane(c, (const uint8_t*)c->src_buf.p, w, h, s_pitch, ow, oh, (uint8_t*)c->dst_buf.p, d_pitch))) return rc;
    SRCNN_CUDA(c, cudaMemcpy2DAsync(dst, dst_stride, c->dst_buf.p, d_pitch, (size_t)ow, oh, cudaMemcpyDeviceToHost, c->stream));
    SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
    return SRCNN_OK;
}

int srcnn_stage_cnn_device(srcnn_ctx* c, int variant, const uint8_t* d_y, int w, int h, size_t pitch, uint8_t* d_out,
                           size_t out_pitch) {
    ENTER(c);
    if (!d_y || !d_out) return fail(c, SRCNN_E_ARG, "null pointer");
    if (w <= 0 || h <= 0 || pitch < (size_t)w || out_pitch < (size_t)w) return fail(c, SRCNN_E_ARG, "bad plane geometry");
    CnnArgs ca;
    ca.y = d_y; ca.pitch = pitch; ca.W = w; ca.H = h;
    ca.row0 = 0; ca.rows = h; ca.out_begin = 0; ca.out_end = h;
    ca.out = d_out; ca.out_pitch = out_pitch;
    return run_cnn(c, variant, ca);
}

int srcnn_stage_conv99x11_fp32_device(srcnn_ctx* c, const uint8_t* d_y, int w, int h, size_t pitch, float* d_act2) {
    ENTER(c);
    if (!d_y || !d_act2) return fail(c, SRCNN_E_ARG, "null pointer");
    if (w <= 0 || h <= 0 || pitch < (size_t)w) return fail(c, SRCNN_E_ARG, "bad plane geometry");
    CnnArgs ca;
    ca.y = d_y; ca.pitch = pitch; ca.W = w; ca.H = h;
    ca.row0 = 0; ca.rows = h; ca.out_begin = 0; ca.out_end = h;
    ca.out = nullptr; ca.out_pitch = 0;
    return launch_cnn_fp32(c, ca, d_act2);
}

int srcnn_stage_merge_device(srcnn_ctx* c, const uint8_t* d_y, const uint8_t* d_cr, const uint8_t* d_cb, int w, int h,
                             size_t plane_pitch, int order, uint8_t* d_dst, size_t dst_stride) {
    ENTER(c);
    if (!d_y || !d_cr || !d_cb || !d_dst) return fail(c, SRCNN_E_ARG, "null pointer");
    if (order != SRCNN_ORDER_BGR && order != SRCNN_ORDER_RGB) return fail(c, SRCNN_E_ARG, "colour order expected, got %d", order);
    if (w <= 0 || h <= 0 || dst_stride < (size_t)w * 3) return fail(c, SRCNN_E_ARG, "bad geometry");
    if (plane_pitch < align_up((size_t)w, 4) || (plane_pitch & 3) || (((uintptr_t)d_y | (uintptr_t)d_cr | (uintptr_t)d_cb) & 3))
        return fail(c, SRCNN_E_ARG, "planes must be 4-byte aligned with pitch a multiple of 4 and >= w rounded up to 4");
    MergeArgs ma;
    ma.y = d_y; ma.cr = d_cr; ma.cb = d_cb; ma.pitch = plane_pitch;
    ma.w = w; ma.rows = h; ma.order = order; ma.dst = d_dst; ma.dst_stride = dst_stride;
    return launch_merge(c, ma);
}

}  // extern "C"
