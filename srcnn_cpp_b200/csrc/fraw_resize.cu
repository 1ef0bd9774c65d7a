// fraw_resize.cu -- optional frawscale-compatible resize stage (SURVEY 8f row N3).
//
// The reference ships a separable float resampler, FRAWResizeEngine (src/frawscale.h:150-170,
// src/frawscale.cpp:162-385), that bin/srcnn never calls (SURVEY fact 2) but BASELINE.json's north_star
// names.  This is its B200 counterpart on float planes, for callers that want that resampler's numbers:
//   * per-output-sample contribution tables {Left, Right, Weights[]} built on the host in double, following
//     FRawScaleWeightsTable's constructor (src/frawscale.cpp:8-112): window = 2*ceil(width)+1, centre
//     u/scale + (0.5/scale - 0.5), borders TRUNCATED (not replicated) and the weights renormalised,
//     trailing zero weights trimmed;
//   * filters: Box (width 0.5), Bilinear (width 1), Bicubic = Mitchell with B = C = 1/3 (width 2)
//     (src/frawscale.h:57-118);
//   * pass order like scale(): vertical then horizontal when dst_width > src_width, else horizontal then
//     vertical (src/frawscale.cpp:195-278);
//   * every output sample = (float) of a double sum accumulated in tap order with separate multiply and
//     add (__dmul_rn/__dadd_rn), as the -O0 x86-64 reference objects do (src/frawscale.cpp:316-325, 369-378).
// Bit-identical to the compiled reference (tests/test_fraw.py) and to a float64 restatement of it on planes built to
// expose FMA, tap order and last-bit table changes (tests/test_fraw_precision.py); NaN only as NaN.  HBM-bound: 4 B
// read + 4 B written per sample and pass.  One documented deviation: for equal source and destination size the
// reference copies only sizeof(unsigned short) bytes per sample (src/frawscale.cpp:189) and leaves the rest
// uninitialised; this stage copies the whole plane.
#include <cmath>

#include "common.h"

namespace srcnn {
namespace {

struct FrawFilter {
    int kind;  // 0 box, 1 bilinear, 2 bicubic (Mitchell B=C=1/3)
    double width;
    double p0, p2, p3, q0, q1, q2, q3;
    explicit FrawFilter(int k) : kind(k), width(k == 0 ? 0.5 : (k == 1 ? 1.0 : 2.0)) {
        const double b = 1 / (double)3, c = 1 / (double)3;      // src/frawscale.h:93
        p0 = (6 - 2 * b) / 6;
        p2 = (-18 + 12 * b + 6 * c) / 6;
        p3 = (12 - 9 * b - 6 * c) / 6;
        q0 = (8 * b + 24 * c) / 6;
        q1 = (-12 * b - 48 * c) / 6;
        q2 = (6 * b + 30 * c) / 6;
        q3 = (-b - 6 * c) / 6;
    }
    double eval(double v) const {
        v = fabs(v);
        if (kind == 0) return v <= width ? 1.0 : 0.0;            // :66
        if (kind == 1) return v < width ? width - v : 0.0;       // :76-80
        if (v < 1) return p0 + v * v * (p2 + v * p3);            // :110-111
        if (v < 2) return q0 + v * (q1 + v * (q2 + v * q3));     // :113-114
        return 0;
    }
};

// Contribution table of one axis: for every destination sample the first source index, the number of taps and the
// (renormalised) weights.  Same numbers, computed in the same order in double, as FRawScaleWeightsTable's constructor
// (src/frawscale.cpp:8-112) -- bit-identical tables are what makes the resize bit-identical.
struct FrawTable {
    int window = 0;
    std::vector<int> left, count;     // first source index and number of taps per destination sample
    std::vector<double> w;            // [dst][window + 1]
    FrawTable(const FrawFilter& f, unsigned dst, unsigned src) {
        const double ratio = double(dst) / double(src);
        // down-scaling stretches the filter's support by 1/ratio and scales its argument by ratio (:21-33)
        const double support = ratio < 1.0 ? f.width / ratio : f.width;
        const double arg_scale = ratio < 1.0 ? ratio : 1.0;
        window = 2 * (int)ceil(support) + 1;
        const int stride = window + 1;
        left.resize(dst); count.resize(dst); w.assign((size_t)dst * stride, 0.0);
        const double shift = (0.5 / ratio) - 0.5;                        // centre of destination sample 0 in source units
        const int last_src = int(src) - 1;
        for (unsigned u = 0; u < dst; u++) {
            const double centre = (double)u / ratio + shift;
            int first = std::max(0, (int)floor(centre - support));      // borders are TRUNCATED, not replicated
            int last = std::min((int)ceil(centre + support), last_src);
            if (last - first + 1 > window) {
                // the reference compares against `int(uSrcSize) - 1 / 2`, i.e. src - 0 (integer division), at :57:
                // always true for a valid index, so it is always the left end that gives way
                if (first < int(src) - 1 / 2) first++; else last--;
            }
            double* wt = &w[(size_t)u * stride];
            double total = 0;
            for (int i = first; i <= last; i++) {
                const double weight = arg_scale * f.eval(arg_scale * (centre - (double)i));
                wt[i - first] = weight;
                total += weight;
            }
            int kept_last = last;
            if (total > 0 && total != 1) {
                for (int i = first; i <= last; i++) wt[i - first] /= total;
                for (int k = last - first; wt[k] == 0; k--) {           // :97-106 drops trailing zero taps
                    kept_last--;
                    if (kept_last == first) break;
                }
            }
            left[u] = first;
            count[u] = kept_last - first + 1;
        }
    }
};

// dst[y][x] = (float) sum_i w[y][i] * (double)src[(left[y] + i)][x]     (verticalFilter, :335-385)
__global__ void __launch_bounds__(256) k_fraw_vertical(const float* __restrict__ src, unsigned width, float* __restrict__ dst,
                                                       unsigned dst_h, const int* __restrict__ left, const int* __restrict__ count,
                                                       const double* __restrict__ w, int stride) {
    const unsigned x = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned y = blockIdx.y;
    if (x >= width || y >= dst_h) return;
    const int l = left[y], n = count[y];
    const double* wt = w + (size_t)y * stride;
    double gray = 0.0;
    for (int i = 0; i < n; i++) gray = __dadd_rn(gray, __dmul_rn(wt[i], (double)src[(size_t)(l + i) * width + x]));
    dst[(size_t)y * width + x] = (float)gray;
}

// dst[y][x] = (float) sum_i w[x][i] * (double)src[y][left[x] + i]        (horizontalFilter, :288-332)
__global__ void __launch_bounds__(256) k_fraw_horizontal(const float* __restrict__ src, unsigned src_w, float* __restrict__ dst,
                                                         unsigned dst_w, unsigned height, const int* __restrict__ left,
                                                         const int* __restrict__ count, const double* __restrict__ w, int stride) {
    const unsigned x = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned y = blockIdx.y;
    if (x >= dst_w || y >= height) return;
    const int l = left[x], n = count[x];
    const double* wt = w + (size_t)x * stride;
    const float* row = src + (size_t)y * src_w + l;
    double gray = 0.0;
    for (int i = 0; i < n; i++) gray = __dadd_rn(gray, __dmul_rn(wt[i], (double)row[i]));
    dst[(size_t)y * dst_w + x] = (float)gray;
}

// Device copies of the tables, kept per context and (filter, dst, src): a stream of same-sized frames builds and uploads
// them once, and no pass waits for the stream (an evicted entry is freed only after the stream has drained).
struct DevTable {
    int filter = -1;
    unsigned dst = 0, src = 0;
    int* left = nullptr;
    int* count = nullptr;
    double* w = nullptr;
    int stride = 0;
    unsigned long long stamp = 0;
    void release() { cudaFree(left); cudaFree(count); cudaFree(w); left = count = nullptr; w = nullptr; filter = -1; }
};
struct FrawCache {
    DevTable slot[8];
    unsigned long long clock = 0;
};

int get_table(Ctx* c, const FrawFilter& f, unsigned dst, unsigned src, DevTable** out) {
    if (!c->fraw_cache) c->fraw_cache = new FrawCache();
    FrawCache* fc = (FrawCache*)c->fraw_cache;
    DevTable* victim = &fc->slot[0];
    for (auto& d : fc->slot) {
        if (d.filter == f.kind && d.dst == dst && d.src == src) { d.stamp = ++fc->clock; *out = &d; return SRCNN_OK; }
        if (d.stamp < victim->stamp) victim = &d;
    }
    DevTable* d = victim;
    if (d->filter >= 0) {   // in-flight kernels may still read it
        SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
        d->release();
    }
    const FrawTable t(f, dst, src);
    d->stride = t.window + 1;
    SRCNN_CUDA(c, cudaMalloc(&d->left, sizeof(int) * t.left.size()));
    SRCNN_CUDA(c, cudaMalloc(&d->count, sizeof(int) * t.count.size()));
    SRCNN_CUDA(c, cudaMalloc(&d->w, sizeof(double) * t.w.size()));
    // pageable sources: the runtime has staged them when the calls return, the vectors may go out of scope
    SRCNN_CUDA(c, cudaMemcpyAsync(d->left, t.left.data(), sizeof(int) * t.left.size(), cudaMemcpyHostToDevice, c->stream));
    SRCNN_CUDA(c, cudaMemcpyAsync(d->count, t.count.data(), sizeof(int) * t.count.size(), cudaMemcpyHostToDevice, c->stream));
    SRCNN_CUDA(c, cudaMemcpyAsync(d->w, t.w.data(), sizeof(double) * t.w.size(), cudaMemcpyHostToDevice, c->stream));
    d->filter = f.kind; d->dst = dst; d->src = src;
    d->stamp = ++fc->clock;
    *out = d;
    return SRCNN_OK;
}

int run_vertical(Ctx* c, const FrawFilter& f, const float* src, unsigned width, unsigned sh, float* dst, unsigned dh) {
    DevTable* d;
    int rc = get_table(c, f, dh, sh, &d);
    if (rc) return rc;
    dim3 grid((width + 255) / 256, dh);
    k_fraw_vertical<<<grid, 256, 0, c->stream>>>(src, width, dst, dh, d->left, d->count, d->w, d->stride);
    c->launches++;
    SRCNN_CUDA(c, cudaGetLastError());
    return SRCNN_OK;
}

int run_horizontal(Ctx* c, const FrawFilter& f, const float* src, unsigned sw, unsigned height, float* dst, unsigned dw) {
    DevTable* d;
    int rc = get_table(c, f, dw, sw, &d);
    if (rc) return rc;
    dim3 grid((dw + 255) / 256, height);
    k_fraw_horizontal<<<grid, 256, 0, c->stream>>>(src, sw, dst, dw, height, d->left, d->count, d->w, d->stride);
    c->launches++;
    SRCNN_CUDA(c, cudaGetLastError());
    return SRCNN_OK;
}

}  // namespace

void fraw_release(Ctx* c) {
    FrawCache* fc = (FrawCache*)c->fraw_cache;
    if (!fc) return;
    for (auto& d : fc->slot)
        if (d.filter >= 0) d.release();
    delete fc;
    c->fraw_cache = nullptr;
}

}  // namespace srcnn

using namespace srcnn;

// FrawTable of one axis (host code only, no device needed).  With left, count and w all null only *window is written;
// otherwise left[dst], count[dst] and w[dst * (window + 1)] receive the table as the passes read it.
extern "C" __attribute__((visibility("default"))) int srcnn_debug_fraw_table(int filter, unsigned dst, unsigned src, int* left,
                                                                             int* count, double* w, int* window) {
    if (filter < 0 || filter > 2 || dst == 0 || src == 0 || !window) return SRCNN_E_ARG;
    const bool query = !left && !count && !w;
    if (!query && (!left || !count || !w)) return SRCNN_E_ARG;
    const FrawTable t(FrawFilter(filter), dst, src);
    *window = t.window;
    if (query) return SRCNN_OK;
    std::copy(t.left.begin(), t.left.end(), left);
    std::copy(t.count.begin(), t.count.end(), count);
    std::copy(t.w.begin(), t.w.end(), w);
    return SRCNN_OK;
}

extern "C" int srcnn_fraw_scale_device(srcnn_ctx* c, const float* d_src, unsigned sw, unsigned sh, unsigned dw, unsigned dh,
                                       float* d_dst, int filter) {
    if (!c) return SRCNN_E_ARG;
    srcnn::DeviceScope scope(c->device);
    if (!scope.ok) return fail(c, SRCNN_E_CUDA, "cudaSetDevice failed");
    if (!d_src || !d_dst) return fail(c, SRCNN_E_ARG, "null pointer");
    if (sw == 0 || sh == 0 || dw == 0 || dh == 0) return fail(c, SRCNN_E_ARG, "empty plane");      // :168-169
    if (filter < 0 || filter > 2) return fail(c, SRCNN_E_ARG, "unknown filter %d", filter);
    if (dh > 65535u || sh > 65535u) return fail(c, SRCNN_E_ARG, "plane taller than 65535 rows: split it into bands");
    // a one-pass resize reads d_src while it writes d_dst (and a copy of overlapping ranges is undefined): no overlap
    const uintptr_t s0 = (uintptr_t)d_src, s1 = s0 + sizeof(float) * (size_t)sw * sh;
    const uintptr_t d0 = (uintptr_t)d_dst, d1 = d0 + sizeof(float) * (size_t)dw * dh;
    if (s0 < d1 && d0 < s1) return fail(c, SRCNN_E_ARG, "source and destination planes overlap");
    const FrawFilter f(filter);
    if (sw == dw && sh == dh) {
        SRCNN_CUDA(c, cudaMemcpyAsync(d_dst, d_src, sizeof(float) * (size_t)sw * sh, cudaMemcpyDeviceToDevice, c->stream));
        return SRCNN_OK;
    }
    int rc = SRCNN_OK;
    if (dw <= sw) {   // horizontal first, then vertical (:195-237)
        const float* mid = d_src;
        if (sw != dw) {
            float* tmp = d_dst;
            if (sh != dh) {
                rc = ensure(c, c->act2_buf, sizeof(float) * (size_t)dw * sh);
                if (rc) return rc;
                tmp = (float*)c->act2_buf.p;
            }
            rc = run_horizontal(c, f, d_src, sw, sh, tmp, dw);
            if (rc) return rc;
            mid = tmp;
        }
        if (sh != dh) rc = run_vertical(c, f, mid, dw, sh, d_dst, dh);
    } else {          // vertical first, then horizontal (:238-278)
        const float* mid = d_src;
        if (sh != dh) {
            rc = ensure(c, c->act2_buf, sizeof(float) * (size_t)sw * dh);
            if (rc) return rc;
            float* tmp = (float*)c->act2_buf.p;
            rc = run_vertical(c, f, d_src, sw, sh, tmp, dh);
            if (rc) return rc;
            mid = tmp;
        }
        rc = run_horizontal(c, f, mid, sw, dh, d_dst, dw);
    }
    return rc;
}
