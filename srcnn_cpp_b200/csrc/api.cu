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
#include <utility>

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

// What the host path needs to know about a pixel order, from layout_of: no other function of the whole path asks for the order.
struct Layout {
    enum Finish { kCnnOut, kMerge, kPack };   // the last kernel: the CNN into the caller's frame, the merge, the pack kernel
                                              // (4:2:2, grey + alpha)
    enum Chroma { kNone, k420, k422, kAlpha };   // planes resized without the CNN: none, chroma w/2 x h/2, w/2 x h, alpha w x h
    int order = -1;                           // -1: not an order of the whole path
    size_t bpp = 0;          // bytes per pixel of a row (4:2:0: of a Y row; NV12's chroma rows have as many, I420's half as many)
    size_t row_align = 4;    // device staging rows (4:2:0: 16-byte multiples, so that I420's half-length rows stay 8-byte aligned)
    Finish finish = kMerge;
    Chroma chroma = kNone;
    bool i420 = false;       // chroma rows half as long, stride/2 apart: even strides
    bool alpha = false;      // four-channel: an A plane beside Cr / Cb
    bool fuses = false;      // the fused merge takes it (a four-channel call needs the merge for alpha, 4:2:2 and GRAYA their pack kernel)
    // 4:2:0: h rows of Y, then h/2 rows of NV12 pairs or of I420 U and V: even sizes, frames staged whole, no band calls
    bool whole() const { return chroma == k420; }
    int csub() const { return chroma == kAlpha ? 1 : 2; }   // Y columns per column of the planes resized without the CNN
    // the workspace has Cr / Cb planes (4:2:2: U' / V'; GRAYA: A' in the Cr slot, Cb unused), so the call merges
    bool cbcr() const { return finish != kCnnOut; }
    int planes() const { return alpha ? 5 : 4; }    // u8 workspace planes per frame
    size_t rows(int n) const { return whole() ? (size_t)n / 2 * 3 : (size_t)n; }   // rows in memory of a frame of n Y rows
};

static Layout layout_of(int order) {
    Layout L;
    switch (order) {
        case SRCNN_ORDER_BGR: case SRCNN_ORDER_RGB: L.bpp = 3; L.fuses = true; break;
        case SRCNN_ORDER_BGRA: case SRCNN_ORDER_RGBA: L.bpp = 4; L.alpha = true; break;
        case SRCNN_ORDER_GRAY: L.bpp = 1; L.finish = Layout::kCnnOut; break;
        case SRCNN_ORDER_NV12: case SRCNN_ORDER_I420:
            L.bpp = 1; L.row_align = 16; L.finish = Layout::kCnnOut; L.chroma = Layout::k420; L.i420 = order == SRCNN_ORDER_I420; break;
        case SRCNN_ORDER_YUY2: case SRCNN_ORDER_UYVY: L.bpp = 2; L.finish = Layout::kPack; L.chroma = Layout::k422; break;
        case SRCNN_ORDER_GRAYA: L.bpp = 2; L.finish = Layout::kPack; L.chroma = Layout::kAlpha; break;
        default: return L;
    }
    L.order = order;
    return L;
}

// One whole-path call: frames of w x h -> ow x oh.  `src` / `dst` are at frame 0 (a band's: at its first source / output row),
// the frames src_frame / dst_frame bytes apart; both are 0 for a single frame, whose kernels then take no frame strides.
struct Image {
    const uint8_t* src = nullptr;
    size_t src_stride = 0, src_frame = 0;
    uint8_t* dst = nullptr;
    size_t dst_stride = 0, dst_frame = 0;
    int w = 0, h = 0, ow = 0, oh = 0;
    float scale = 0.f;
    Layout L;
    Image frame(int f) const {   // frame f as a call of its own
        return Image{src + (size_t)f * src_frame, src_stride, 0, dst + (size_t)f * dst_frame, dst_stride, 0, w, h, ow, oh, scale, L};
    }
};

static int check_image(Ctx* c, const uint8_t* src, int w, int h, size_t stride, int order, float scale, uint8_t* dst,
                       size_t dst_stride, Image* im) {
    if (!c) return SRCNN_E_ARG;
    if (!src || !dst) return fail(c, SRCNN_E_ARG, "null image pointer");
    if (w <= 0 || h <= 0) return fail(c, SRCNN_E_ARG, "non-positive image size %dx%d", w, h);
    const Layout L = layout_of(order);
    if (L.order < 0) return fail(c, SRCNN_E_ARG, "unknown pixel order %d", order);
    if (stride < (size_t)w * L.bpp) return fail(c, SRCNN_E_ARG, "source stride %zu < %zu*w", stride, L.bpp);
    if (L.whole() && ((w | h) & 1)) return fail(c, SRCNN_E_ARG, "4:2:0 frames need an even width and height, got %dx%d", w, h);
    if (L.chroma == Layout::k422 && (w & 1)) return fail(c, SRCNN_E_ARG, "4:2:2 frames need an even width (whole macropixels), got %d", w);
    if (L.i420 && ((stride | dst_stride) & 1))
        return fail(c, SRCNN_E_ARG, "I420 strides must be even (chroma rows are stride/2 apart), got %zu / %zu", stride, dst_stride);
    int ow, oh;   // src/srcnn.cpp:485-495 "ratio too small"
    if (srcnn_out_dims(w, h, scale, &ow, &oh)) return fail(c, SRCNN_E_RATIO, "scale %g gives an empty image", scale);
    if (L.whole() && ((ow | oh) & 1))
        return fail(c, SRCNN_E_ARG, "scale %g gives an odd 4:2:0 output size %dx%d (width and height must be even)", scale, ow, oh);
    if (L.chroma == Layout::k422 && (ow & 1))
        return fail(c, SRCNN_E_ARG, "scale %g gives an odd 4:2:2 output width %d (whole macropixels: it must be even)", scale, ow);
    if (dst_stride < (size_t)ow * L.bpp) return fail(c, SRCNN_E_ARG, "destination stride %zu < %zu*ow", dst_stride, L.bpp);
    *im = Image{src, stride, 0, dst, dst_stride, 0, w, h, ow, oh, scale, L};
    return SRCNN_OK;
}

// check_image for a batch of n frames, and its frame strides.  n = 0 passes with nothing filled in.
static int check_batch(Ctx* c, int n, const uint8_t* src, int w, int h, size_t stride, size_t src_frame, int order, float scale,
                       uint8_t* dst, size_t dst_stride, size_t dst_frame, Image* im) {
    if (n < 0) return fail(c, SRCNN_E_ARG, "negative frame count");
    if (n == 0) return SRCNN_OK;
    int rc = check_image(c, src, w, h, stride, order, scale, dst, dst_stride, im);
    if (rc) return rc;
    if (n > 1 && (src_frame < stride * im->L.rows(h) || dst_frame < dst_stride * im->L.rows(im->oh)))
        return fail(c, SRCNN_E_ARG, "frame stride smaller than one frame");
    im->src_frame = src_frame; im->dst_frame = dst_frame;
    return SRCNN_OK;
}

constexpr int kHalo = 6;   // output rows the CNN reads around a band: 4 (conv1) + 2 (conv3)

// The source rows that output rows [r0, r1) and `halo` output rows either side of them touch, from the tap table `ofs` (h -> oh)
static std::pair<int, int> src_rows(const int* ofs, int h, int oh, int r0, int r1, int halo = kHalo) {
    const int p0 = std::max(r0 - halo, 0), p1 = std::min(r1 + halo, oh);
    return {std::min(std::max(ofs[p0] - 1, 0), h - 1), std::min(std::max(ofs[p1 - 1] + 2, 0), h - 1) + 1};
}

// The chroma descriptor of the luma output rows [r0, r1) of frames whose row 0 is at `src` / `dst` (frame 0).  No halo: a chroma
// row is resized without the CNN.  4:2:0: the chroma rows after the Y rows, resized straight into the caller's frames (chroma
// output rows [r0/2, r1/2)).  4:2:2: U' and V' of the packed rows go into the Cr / Cb planes of `pl` (their first ow/2 columns),
// which the pack kernel reads for the same rows.  GRAYA: the alpha plane (w x h -> ow x oh) likewise, into the Cr plane.
static int chroma_planes(Ctx* c, const Image& im, const uint8_t* src, uint8_t* dst, const Planes& pl, int r0, int r1, Chroma420* ch) {
    const int v = im.L.whole() ? 2 : 1, u = im.L.csub();   // Y rows per chroma row, Y columns per chroma column
    TapTable *tx, *ty;
    int rc = get_taps(c, im.w / u, im.ow / u, &tx);
    if (rc) return rc;
    if ((rc = get_taps(c, im.h / v, im.oh / v, &ty))) return rc;
    ch->sw = im.w / u; ch->sh = im.h / v; ch->ow = im.ow / u; ch->oh = im.oh / v;
    ch->row_begin = r0 / v; ch->row_end = r1 / v;
    ch->tx = tx; ch->ty = ty;
    if (!im.L.whole()) {
        ch->src = src; ch->src_pitch = im.src_stride; ch->src_v = 0;
        ch->dst = pl.cr - (ptrdiff_t)pl.row0 * (ptrdiff_t)pl.pitch;   // chroma output row r at dst + r * pitch
        ch->dst_pitch = pl.pitch;
        ch->dst_v = (size_t)(pl.cb - pl.cr);
        ch->dst_frame = pl.frame_stride;
        return SRCNN_OK;
    }
    const bool i420 = im.L.i420;
    ch->src = src + (size_t)im.h * im.src_stride;
    ch->src_pitch = i420 ? im.src_stride / 2 : im.src_stride;
    ch->src_v = i420 ? (size_t)(im.h / 2) * (im.src_stride / 2) : 0;
    ch->dst = dst + (size_t)im.oh * im.dst_stride;
    ch->dst_pitch = i420 ? im.dst_stride / 2 : im.dst_stride;
    ch->dst_v = i420 ? (size_t)(im.oh / 2) * (im.dst_stride / 2) : 0;
    ch->dst_frame = im.dst_frame;
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
// U' / V' planes in the Cr / Cb slots, a GRAYA call its A' plane in the Cr slot, and so they take part like a colour call.
static int carve_planes(Ctx* c, int ow, int rows, int row0, Planes* pl, int nframes, const Layout& L) {
    const bool gray = !L.cbcr(), four = L.alpha;
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

// The three stages over frames [f0, f0 + m) of `im`, output rows [r0, r1) from source rows [s0, s1) (im.src is at source row s0,
// im.dst at output row r0).  A band or a single frame is m = 1.  A batch chunk is whole frames, ONE launch of each stage: the
// colour+bicubic grid gets a frame dimension, the row-walking kernel sees the frames as more strips of one work list (no
// per-frame pipeline fill / drain), the merge kernel sees the chunk's planes as one tall image.
static int run_stages(Ctx* c, const Image& im, int f0, int m, int s0, int s1, int r0, int r1) {
    const Layout& L = im.L;
    const uint8_t* src = im.src + (size_t)f0 * im.src_frame;
    uint8_t* dst = im.dst + (size_t)f0 * im.dst_frame;
    TapTable *tx, *ty;
    c->fail_stage = SRCNN_STAGE_COLOR_BICUBIC;
    int rc = get_taps(c, im.w, im.ow, &tx);
    if (rc) return rc;
    if ((rc = get_taps(c, im.h, im.oh, &ty))) return rc;
    const int p0 = std::max(r0 - kHalo, 0), p1 = std::min(r1 + kHalo, im.oh);
    // grey: one-plane resize, then the CNN straight into the caller's rows; no chroma, no merge.  4:2:0: the same for Y, and the
    // resize launch also writes the chroma rows [r0/2, r1/2) straight into the caller's frame
    if (!L.cbcr()) end_merge_chain(c);
    Planes pl;
    c->fail_stage = SRCNN_STAGE_PLANES;
    if ((rc = carve_planes(c, im.ow, p1 - p0, p0, &pl, m, L))) return rc;
    c->fail_stage = SRCNN_STAGE_COLOR_BICUBIC;
    // the band must bring every source row its taps touch
    const auto need = src_rows(ty->h_ofs.data(), im.h, im.oh, r0, r1);
    if (s0 > need.first || s1 < need.second)
        return fail(c, SRCNN_E_ARG, "band rows [%d,%d) need source rows [%d,%d), got [%d,%d)", r0, r1, need.first, need.second, s0, s1);

    ResizeArgs ra;
    ra.src = src; ra.src_stride = im.src_stride;
    ra.sw = im.w; ra.sh = im.h; ra.src_row0 = s0; ra.src_row1 = s1;
    ra.order = L.order;
    ra.ow = im.ow; ra.oh = im.oh;
    ra.row_begin = p0; ra.row_end = p1;
    ra.pl = pl; ra.tx = tx; ra.ty = ty;
    ra.nframes = m; ra.src_frame_stride = im.src_frame;
    // chroma for the rows [r0, r1) only: the luma halo rows [p0, r0) and [r1, p1) are the CNN's
    if (L.chroma != Layout::kNone &&
        (rc = chroma_planes(c, im, src - (size_t)s0 * im.src_stride, dst - (size_t)r0 * im.dst_stride, pl, r0, r1, &ra.ch)))
        return rc;
    if (c->variant != SRCNN_VARIANT_TC) ra.pl.y16 = nullptr;      // the strict FP32 kernels read the u8 plane
    ra.early = L.cbcr() && may_start_early(c, src, (size_t)(m - 1) * im.src_frame + (size_t)(s1 - s0) * im.src_stride);
    c->early_launches += ra.early;
    if ((rc = prof_mark(c, 0))) return rc;
    if ((rc = launch_color_bicubic(c, ra))) return rc;
    if ((rc = prof_mark(c, 1))) return rc;

    c->fail_stage = SRCNN_STAGE_CNN;
    CnnArgs ca;
    ca.y = pl.y; ca.pitch = pl.pitch;
    ca.y16 = pl.y16; ca.pitch16 = pl.pitch16;
    ca.W = im.ow; ca.H = im.oh;
    ca.row0 = p0; ca.rows = p1 - p0;
    ca.out_begin = r0; ca.out_end = r1;
    ca.nframes = m;
    if (im.dst_frame) { ca.y16_frame_stride = pl.frame_stride16; ca.out_frame_stride = pl.frame_stride; }
    if (!L.cbcr()) { ca.out = dst; ca.out_pitch = im.dst_stride; ca.out_row0 = r0; ca.out_frame_stride = im.dst_frame; }
    else { ca.out = pl.yout; ca.out_pitch = pl.pitch; ca.out_row0 = p0; }
    // optionally the row-walking tcgen05 kernel merges Cr/Cb and converts back to BGR in its last epilogue (no Y' plane, no
    // K-C launch); measured slower than the separate launch (byte stores from one-thread-per-column lanes), so off by default
    const bool fused = L.fuses && c->variant == SRCNN_VARIANT_TC && c->fuse_merge;
    if (fused) {
        ca.cr = pl.cr; ca.cb = pl.cb;
        ca.bgr = dst; ca.bgr_stride = im.dst_stride; ca.order = L.order;
    }
    if ((rc = run_cnn(c, c->variant, ca))) return rc;
    if ((rc = prof_mark(c, 2))) return rc;
    if (fused || !L.cbcr()) return prof_mark(c, 3);

    c->fail_stage = SRCNN_STAGE_MERGE;
    MergeArgs ma;
    ma.pitch = pl.pitch; ma.w = im.ow;
    ma.order = L.order;
    ma.dst_stride = im.dst_stride;
    const bool tall = m == 1 || im.dst_frame == im.dst_stride * (size_t)im.oh;   // the chunk's results are one tall image
    for (int f = 0; f < (tall ? 1 : m); f++) {
        const size_t off = (size_t)(r0 - p0) * pl.pitch + (size_t)f * pl.frame_stride;
        ma.y = pl.yout + off; ma.cr = pl.cr + off; ma.cb = pl.cb + off;
        if (pl.a) ma.a = pl.a + off;
        ma.rows = tall ? (r1 - r0) * m : r1 - r0;
        ma.dst = dst + (size_t)f * im.dst_frame;
        if ((rc = L.finish == Layout::kPack ? launch_pack(c, ma) : launch_merge(c, ma))) return rc;
    }
    merged_into(c, dst, (size_t)(m - 1) * im.dst_frame + (size_t)(r1 - r0) * im.dst_stride);
    return prof_mark(c, 3);
}

// n frames of `im` resident on the device (n > 1: whole frames).  A batch goes in chunks whose planes stay below ~1 GB, one
// launch per stage and chunk; that needs the row-walking kernel with a separate merge, everything else goes frame by frame (the
// fused merge only takes the colour orders: grey and four-channel batches stay batched with it switched on).
static int process(Ctx* c, const Image& im, int n, int s0, int s1, int r0, int r1) {
    if (n > 1 && (c->variant != SRCNN_VARIANT_TC || (c->fuse_merge && im.L.fuses) || !c->batch_launch)) {
        for (int f = 0; f < n; f++)
            if (int rc = process(c, im.frame(f), 1, s0, s1, r0, r1)) return rc;
        return SRCNN_OK;
    }
    const Image frames = n == 1 ? im.frame(0) : im;
    const size_t per_frame = align_up((size_t)im.ow, 128) * (size_t)im.oh * im.L.planes() + y16_pitch_bytes(im.ow) * (size_t)im.oh;
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n, ((size_t)1 << 30) / per_frame));
    const size_t ev0 = c->ev_used;
    int rc = SRCNN_OK;
    for (int f0 = 0; f0 < n && !rc; f0 += chunk) rc = run_stages(c, frames, f0, std::min(chunk, n - f0), s0, s1, r0, r1);
    if (rc) c->ev_used = ev0;        // a failed call leaves no half-recorded event group behind (srcnn_profile_read pairs by 4)
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

// What host_pipeline works out once for enqueue_chunk, which enqueues it live or under graph capture
struct HostPlan {
    int S0 = 0, S1 = 0;                      // source rows staged per frame (4:2:0: the whole frame)
    std::vector<int> edges;                  // the sub-bands' output rows: R0, ..., R1
    int group = 1;                           // frames of a batch per copy and launch
    size_t s_row = 0, d_row = 0, s_frame = 0, d_frame = 0;   // device staging
    TapTable *ty = nullptr, *cty = nullptr;  // vertical taps of Y and of 4:2:0 chroma
};

// Rows [y0, y1) of one w x h frame, and for 4:2:0 its chroma rows [c0, c1), between two buffers whose rows are `ds` / `ss`
// bytes apart and which point at the same row (4:2:0: row 0).  NV12's chroma rows follow the Y rows with the same stride;
// I420's U and V rows are half as long.
static int copy_rows(Ctx* c, const Layout& L, uint8_t* dst, size_t ds, const uint8_t* src, size_t ss, int w, int h, int y0, int y1,
                     int c0, int c1, cudaMemcpyKind kind, cudaStream_t st) {
    if (y1 > y0)
        SRCNN_CUDA(c, cudaMemcpy2DAsync(dst + (size_t)y0 * ds, ds, src + (size_t)y0 * ss, ss, (size_t)w * L.bpp, y1 - y0, kind, st));
    if (!L.whole() || c1 <= c0) return SRCNN_OK;
    dst += (size_t)h * ds;
    src += (size_t)h * ss;
    const int np = L.i420 ? 2 : 1;   // NV12: one plane of pairs; I420: U, then V h/2 rows further
    ds /= np;
    ss /= np;
    for (int pl = 0; pl < np; pl++) {
        const size_t r = (size_t)(pl * (h / 2) + c0);
        SRCNN_CUDA(c, cudaMemcpy2DAsync(dst + r * ds, ds, src + r * ss, ss, (size_t)w / np, c1 - c0, kind, st));
    }
    return SRCNN_OK;
}

// Enqueues the whole pipeline of frames [f0, f0 + m) of `im` on the three streams and joins the copy streams back into the
// compute stream; does not wait.  Identical whether the streams are live or being captured into a CUDA graph.
static int enqueue_chunk(Ctx* c, const Image& im, int f0, int m, const HostPlan& p) {
    const Layout& L = im.L;
    const int R0 = p.edges.front(), R1 = p.edges.back(), bands = (int)p.edges.size() - 1;
    const size_t w_bytes = (size_t)im.w * L.bpp, ow_bytes = (size_t)im.ow * L.bpp;
    int rc;
    uint8_t* ds = (uint8_t*)c->src_buf.p;
    uint8_t* dd = (uint8_t*)c->dst_buf.p;
    auto staged = [&](int f) {   // the device staging from frame f on, as a call of its own
        return Image{ds + (size_t)f * p.s_frame, p.s_row, p.s_frame, dd + (size_t)f * p.d_frame, p.d_row, p.d_frame,
                     im.w, im.h, im.ow, im.oh, im.scale, L};
    };
    size_t ei = 0;
    auto join = [&](cudaStream_t from, cudaStream_t to) -> int {   // `to` waits for what `from` has been given so far
        if (ei == c->pipe_events.size()) {
            cudaEvent_t ev;
            SRCNN_CUDA(c, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            c->pipe_events.push_back(ev);
        }
        SRCNN_CUDA(c, cudaEventRecord(c->pipe_events[ei], from));
        SRCNN_CUDA(c, cudaStreamWaitEvent(to, c->pipe_events[ei++], 0));
        return SRCNN_OK;
    };
    // everything queued earlier on the compute stream (previous calls, tap-table uploads) precedes the copies
    if ((rc = join(c->stream, c->s_in))) return rc;
    SRCNN_CUDA(c, cudaStreamWaitEvent(c->s_out, c->pipe_events[0], 0));
    if (bands == 1 && m > 1) {
        // A batch of whole frames: groups of frames travel together -- one copy in, ONE launch per stage (process: no
        // per-frame pipeline fill / drain in the fused kernel), one copy out -- sized so that a group's result is >= 64 MB:
        // large copies keep the PCIe link busy, and the next group's kernels still hide behind this group's D2H.
        const bool rows_tight_in = im.src_stride == w_bytes && p.s_row == w_bytes;      // a frame is one contiguous run of bytes
        const bool rows_tight_out = im.dst_stride == ow_bytes && p.d_row == ow_bytes;
        for (int g0 = 0; g0 < m; g0 += p.group) {
            const int g = std::min(p.group, m - g0);
            const uint8_t* hsrc = im.src + (size_t)(f0 + g0) * im.src_frame + (size_t)p.S0 * im.src_stride;
            uint8_t* hdst = im.dst + (size_t)(f0 + g0) * im.dst_frame;
            if (rows_tight_in)   // frames are the "rows" of one 2-D copy
                SRCNN_CUDA(c, cudaMemcpy2DAsync(ds + (size_t)g0 * p.s_frame, p.s_frame, hsrc, im.src_frame, L.rows(p.S1 - p.S0) * p.s_row, g,
                                                cudaMemcpyHostToDevice, c->s_in));
            else
                for (int f = 0; f < g; f++)
                    if ((rc = copy_rows(c, L, ds + (size_t)(g0 + f) * p.s_frame, p.s_row, hsrc + (size_t)f * im.src_frame, im.src_stride,
                                        im.w, im.h, 0, p.S1 - p.S0, 0, im.h / 2, cudaMemcpyHostToDevice, c->s_in)))
                        return rc;
            if ((rc = join(c->s_in, c->stream))) return rc;
            if ((rc = process(c, staged(g0), g, 0, im.h, 0, im.oh)) || (rc = join(c->stream, c->s_out))) return rc;   // whole frames
            if (rows_tight_out)
                SRCNN_CUDA(c, cudaMemcpy2DAsync(hdst, im.dst_frame, dd + (size_t)g0 * p.d_frame, p.d_frame, L.rows(R1 - R0) * p.d_row, g,
                                                cudaMemcpyDeviceToHost, c->s_out));
            else
                for (int f = 0; f < g; f++)
                    if ((rc = copy_rows(c, L, hdst + (size_t)f * im.dst_frame, im.dst_stride, dd + (size_t)(g0 + f) * p.d_frame, p.d_row,
                                        im.ow, im.oh, 0, R1 - R0, 0, im.oh / 2, cudaMemcpyDeviceToHost, c->s_out)))
                        return rc;
        }
    } else
    for (int f = 0; f < m; f++) {
        const uint8_t* hsrc = im.src + (size_t)(f0 + f) * im.src_frame + (size_t)p.S0 * im.src_stride;
        uint8_t* hdst = im.dst + (size_t)(f0 + f) * im.dst_frame;
        int copied = p.S0;   // source rows [S0, copied) of this frame are on their way to the device
        int c_copied = 0;    // 4:2:0: chroma source rows [0, c_copied) likewise
        for (int bi = 0; bi < bands; bi++) {
            const int r0 = p.edges[bi], r1 = p.edges[bi + 1];
            const int s_hi = bi + 1 < bands ? src_rows(p.ty->h_ofs.data(), im.h, im.oh, r0, r1).second : p.S1;
            // 4:2:0: a sub-band also copies the chroma rows its chroma output rows [r0/2, r1/2) read
            const int c_hi = !L.whole() ? 0 : bi + 1 < bands ? src_rows(p.cty->h_ofs.data(), im.h / 2, im.oh / 2, r0 / 2, r1 / 2, 0).second
                                                            : im.h / 2;
            if (s_hi > copied || c_hi > c_copied) {
                if ((rc = copy_rows(c, L, ds + (size_t)f * p.s_frame, p.s_row, hsrc, im.src_stride, im.w, im.h, copied - p.S0, s_hi - p.S0,
                                    c_copied, c_hi, cudaMemcpyHostToDevice, c->s_in)))
                    return rc;
                if ((rc = join(c->s_in, c->stream))) return rc;
                copied = std::max(copied, s_hi);
                c_copied = std::max(c_copied, c_hi);
            }
            Image band = staged(f);
            band.dst += (size_t)(r0 - R0) * p.d_row;
            if ((rc = process(c, band, 1, p.S0, p.S1, r0, r1)) || (rc = join(c->stream, c->s_out))) return rc;
            if ((rc = copy_rows(c, L, hdst, im.dst_stride, dd + (size_t)f * p.d_frame, p.d_row, im.ow, im.oh, r0 - R0, r1 - R0, r0 / 2, r1 / 2,
                                cudaMemcpyDeviceToHost, c->s_out)))
                return rc;
        }
    }
    // the compute stream ends after the last copy in either direction
    if ((rc = join(c->s_in, c->stream))) return rc;
    return join(c->s_out, c->stream);
}

static int host_pipeline(Ctx* c, const Image& im, int n, int R0, int R1) {
    const Layout& L = im.L;
    int rc;
    struct HostPath {   // the pipeline's sub-bands and groups share Cr/Cb pair 0 (carve_planes) and never start early
        Ctx* c;
        explicit HostPath(Ctx* c_) : c(c_) { c->host_path = true; c->merge_sel = -1; }
        ~HostPath() { c->host_path = false; c->merge_sel = -1; }
    } host_path{c};
    HostPlan p;
    TapTable *tx, *ctx_;
    if ((rc = get_taps(c, im.h, im.oh, &p.ty))) return rc;
    if ((rc = get_taps(c, im.w, im.ow, &tx))) return rc;      // uploaded here, not inside a graph capture
    if (L.whole() && (rc = get_taps(c, im.h / 2, im.oh / 2, &p.cty))) return rc;                      // chroma (4:2:2: its vertical
    if (L.chroma != Layout::kNone && (rc = get_taps(c, im.w / L.csub(), im.ow / L.csub(), &ctx_))) return rc;   // table is ty)
    // 4:2:0 frames are staged whole (whole-frame calls only: R0 = 0, R1 = oh), every row at its place in the frame
    const auto need = src_rows(p.ty->h_ofs.data(), im.h, im.oh, R0, R1);
    p.S0 = L.whole() ? 0 : need.first;
    p.S1 = L.whole() ? im.h : need.second;
    // device staging: tight rows, 256-byte aligned frames; only the rows this call needs
    p.s_row = align_up((size_t)im.w * L.bpp, L.row_align);
    p.d_row = align_up((size_t)im.ow * L.bpp, L.row_align);
    p.s_frame = align_up(p.s_row * L.rows(p.S1 - p.S0), 256);
    p.d_frame = align_up(p.d_row * L.rows(R1 - R0), 256);
    // frames in flight are bounded so staging stays modest (<= 4 GiB of output; one frame may be larger).  Chunks are separated by
    // a full drain of the pipeline, so the bound is generous: 180 GB of HBM is not the scarce resource here.
    const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)n, ((size_t)4 << 30) / p.d_frame));
    if ((rc = ensure(c, c->src_buf, p.s_frame * chunk))) return rc;
    if ((rc = ensure(c, c->dst_buf, p.d_frame * chunk))) return rc;
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
    const int rows = R1 - R0, even = L.whole() ? ~1 : ~0;   // 4:2:0: even band edges
    p.edges.push_back(R0);
    if (n == 1 && rows >= 1024) {
        const long long by_mem = ((long long)rows * (long long)im.ow * L.planes() + (256ll << 20) - 1) / (256ll << 20);
        if (by_mem > c->host_bands) {
            const int nb = (int)std::min<long long>(by_mem, rows / 64);
            for (int bi = 1; bi < nb; bi++) p.edges.push_back((R0 + (int)((long long)rows * bi / nb)) & even);
        } else if (c->host_bands > 1) {
            double len = c->band_first > 0 ? (double)c->band_first : std::max(256.0, (double)rows / c->host_bands);
            int pos = R0;
            while ((int)p.edges.size() < c->host_bands) {
                const int take = (int)len & even;
                if (R1 - (pos + take) < take / 2) break;      // the rest joins the last band
                pos += take;
                p.edges.push_back(pos);
                len *= c->band_growth;
            }
        }
    }
    p.edges.push_back(R1);
    const int bands = (int)p.edges.size() - 1;
    int tallest = 0;
    for (int bi = 0; bi < bands; bi++) tallest = std::max(tallest, p.edges[bi + 1] - p.edges[bi]);
    // frames of a batch travel in groups whose result is >= 64 MB (see enqueue_chunk)
    p.group = (int)std::max<size_t>(1, std::min<size_t>(16, ((size_t)64 << 20) / std::max<size_t>(1, (size_t)im.ow * L.bpp * (size_t)rows) + 1));
    {   // the planes of the tallest sub-band / of a group of frames, allocated before anything is enqueued or captured
        Planes pl;
        if ((rc = carve_planes(c, im.ow, std::min(tallest + 12, im.oh), 0, &pl, (bands == 1 && n > 1) ? std::min(p.group, n) : 1, L)))
            return rc;
    }

    // ---- CUDA-graph replay.  A call that repeats an earlier one exactly (same buffers, same geometry: a stream of frames through
    // a pair of pinned buffers) is ~50 API calls of host work for ~0.5 ms of device work; the second time a call is seen its
    // pipeline is captured into a graph, from then on it is one cudaGraphLaunch.  One-off calls never pay for instantiation.
    PipeGraph* hit = nullptr;
    const bool graphable = c->use_graphs && !c->profiling && chunk >= n && bands * n <= 256;
    if (graphable) {
        PipeKey key{im.src, im.dst, n, im.w, im.h, im.src_stride, im.src_frame, L.order, im.scale, R0, R1, im.dst_stride, im.dst_frame,
                    c->variant, (int)c->fuse_merge, c->host_bands * 4096 + c->band_first, c->tc2_seg_ovh + (int)(c->band_growth * 1000.0) * 256,
                    (void*)c->stream};
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
    if (hit && !hit->exec && !hit->failed && is_pinned(im.src) && is_pinned(im.dst)) {
        // second sighting: capture.  Nothing below allocates, uploads or synchronises (tables, staging and planes exist).
        cudaGraph_t graph = nullptr;
        const long long launches_before = c->launches;   // capturing enqueues nothing: the launch counter must not move
        cudaError_t e = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal);
        if (e == cudaSuccess) {
            c->capturing = true;
            rc = enqueue_chunk(c, im, 0, n, p);
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
        if ((rc = enqueue_chunk(c, im, f0, m, p))) return rc;
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
    return srcnn_process_batch_device(c, d_src, 1, w, h, src_stride, 0, order, scale, d_dst, dst_stride, 0);
}

int srcnn_process_batch_device(srcnn_ctx* c, const uint8_t* d_src, int n, int w, int h, size_t src_stride,
                               size_t src_frame_stride, int order, float scale, uint8_t* d_dst, size_t dst_stride,
                               size_t dst_frame_stride) {
    ENTER_PROCESS(c);
    Image im;
    int rc = check_batch(c, n, d_src, w, h, src_stride, src_frame_stride, order, scale, d_dst, dst_stride, dst_frame_stride, &im);
    if (rc || n == 0) return rc;
    return process(c, im, n, 0, h, 0, im.oh);
}

int srcnn_process_batch_host(srcnn_ctx* c, const uint8_t* src, int n, int w, int h, size_t src_stride,
                             size_t src_frame_stride, int order, float scale, uint8_t* dst, size_t dst_stride,
                             size_t dst_frame_stride) {
    ENTER_PROCESS(c);
    Image im;
    int rc = check_batch(c, n, src, w, h, src_stride, src_frame_stride, order, scale, dst, dst_stride, dst_frame_stride, &im);
    if (rc || n == 0) return rc;
    return host_pipeline(c, im, n, 0, im.oh);
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
    std::vector<int> ofs(oh);
    std::vector<short4> coef(oh);
    build_cubic_taps(h, oh, ofs.data(), coef.data());
    std::tie(*s0, *s1) = src_rows(ofs.data(), h, oh, r0, r1);
    return SRCNN_OK;
}

// the output band of a band call, after check_image
static int check_band(Ctx* c, const Image& im, int r0, int r1) {
    if (im.L.whole()) return fail(c, SRCNN_E_ARG, "4:2:0 frames are whole-frame calls only (no band calls)");
    if (r0 < 0 || r1 > im.oh || r0 >= r1) return fail(c, SRCNN_E_ARG, "bad output band [%d,%d) of %d rows", r0, r1, im.oh);
    return SRCNN_OK;
}

int srcnn_process_band_device(srcnn_ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int s0, int s1,
                              int order, float scale, int r0, int r1, uint8_t* d_dst, size_t dst_stride) {
    ENTER_PROCESS(c);
    Image im;
    int rc = check_image(c, d_src, w, h, src_stride, order, scale, d_dst, dst_stride, &im);
    if (rc || (rc = check_band(c, im, r0, r1))) return rc;
    if (s0 < 0 || s1 > h || s0 >= s1) return fail(c, SRCNN_E_ARG, "bad source band [%d,%d) of %d rows", s0, s1, h);
    return process(c, im, 1, s0, s1, r0, r1);
}

int srcnn_process_band_host(srcnn_ctx* c, const uint8_t* src, int w, int h, size_t src_stride, int order, float scale,
                            int r0, int r1, uint8_t* dst_rows, size_t dst_stride) {
    ENTER_PROCESS(c);
    Image im;
    int rc = check_image(c, src, w, h, src_stride, order, scale, dst_rows, dst_stride, &im);
    if (rc || (rc = check_band(c, im, r0, r1))) return rc;
    return host_pipeline(c, im, 1, r0, r1);
}

// Rows [0, oh) of a whole image through the colour+bicubic kernels into `pl` (the stage entry points)
static int resize_image(Ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int order, int ow, int oh, const Planes& pl) {
    TapTable *tx, *ty;
    int rc = get_taps(c, w, ow, &tx);
    if (rc) return rc;
    if ((rc = get_taps(c, h, oh, &ty))) return rc;
    ResizeArgs ra;
    ra.src = d_src; ra.src_stride = src_stride;
    ra.sw = w; ra.sh = h; ra.src_row0 = 0; ra.src_row1 = h;
    ra.order = order; ra.ow = ow; ra.oh = oh;
    ra.row_begin = 0; ra.row_end = oh;
    ra.pl = pl; ra.pl.row0 = 0; ra.pl.rows = oh;
    ra.tx = tx; ra.ty = ty;
    return launch_color_bicubic(c, ra);
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
    Planes pl;
    pl.y = d_y; pl.cr = d_cr; pl.cb = d_cb; pl.pitch = plane_pitch;
    return resize_image(c, d_src, w, h, src_stride, order, ow, oh, pl);
}

// One 8-bit plane through cv::resize(..., INTER_CUBIC) (src/srcnn.cpp:577-582): the one-plane resize kernels.  Device buffers,
// enqueued; d_dst must be 4-byte aligned with a pitch that is a multiple of 4 (the tiled kernel's word stores).
static int resize_plane(Ctx* c, const uint8_t* d_src, int w, int h, size_t src_stride, int ow, int oh, uint8_t* d_dst,
                        size_t dst_stride) {
    Planes pl;
    pl.y = d_dst; pl.pitch = dst_stride;
    return resize_image(c, d_src, w, h, src_stride, SRCNN_ORDER_GRAY, ow, oh, pl);
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

// Host buffers: copy the plane in, resize, copy the result out.
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
