// color_bicubic.cu -- kernels A and C of the hot path (HBM-bound stages).
//
//   K-A  colour + split + bicubic:  BGR8 HWC  ->  Y, Cr, Cb u8 planes of the upscaled size.
//        Replaces cvtColor(BGR2YCrCb) src/srcnn.cpp:509, split :540 and the three
//        resize(..., CV_INTER_CUBIC) calls :570-583 of the reference with ONE pass over the source.
//   K-C  merge + colour back:       Y', Cr, Cb planes -> BGR8 HWC.
//        Replaces `pImg[0] = pImgConv3; merge` src/srcnn.cpp:637-639 and cvtColor(YCrCb2BGR) :657.
//
// Arithmetic is OpenCV's 8-bit path restated from its published algorithm (SURVEY.md Appendix A):
// 14-bit fixed-point BT.601 colour; Keys cubic A=-0.75 with 11-bit integer taps, integer horizontal
// pass, float vertical pass `H0*b0 + (H1*b1 + (H2*b2 + H3*b3))` with separate multiplies and adds
// (hence __fmul_rn/__fadd_rn: no FMA contraction), round-half-even, and the integer form on the
// last (ow mod 8) columns.  Results are bit-identical to the oracle (tests/test_stage_parity.py).
//
// A grey source (SRCNN_ORDER_GRAY) takes the same kernels with one plane and no colour conversion: the plain
// resize(..., CV_INTER_CUBIC) of that plane.
//
// A four-channel source (SRCNN_ORDER_BGRA / _RGBA) takes them with a fourth plane: the raw alpha byte, resized like the others
// (not colour-converted), and K-C writes it back as byte 3 of every pixel.
//
// Algorithmic HBM bytes per output pixel: 3/s^2 (BGR read) + 3 (planes written); K-C: 3 + 3.  Grey: 1/s^2 + 1.  Four-channel:
// 4/s^2 + 4; K-C: 4 + 4.
#include <cuda_fp16.h>

#include <cmath>
#include <cstdarg>

#include "common.h"
#include "color_bicubic.h"

namespace srcnn {

// ------------------------------------------------------------------------------------------------
// Host: tap tables.  Same float32/double sequence as cv::resize's table builder; nvcc host flags in
// the Makefile forbid FMA contraction.
// ------------------------------------------------------------------------------------------------
void build_cubic_taps(int src, int dst, int* ofs, short4* coef) {
    const float A = -0.75f;
    const double inv = (double)dst / (double)src;
    const double sc = 1.0 / inv;
    for (int d = 0; d < dst; d++) {
        float f = (float)((d + 0.5) * sc - 0.5);
        int s = (int)floorf(f);
        float x = f - (float)s;
        float x1 = x + 1.f;
        float c0 = ((A * x1 - 5 * A) * x1 + 8 * A) * x1 - 4 * A;
        float c1 = ((A + 2) * x - (A + 3)) * x * x + 1;
        float y = 1.f - x;
        float c2 = ((A + 2) * y - (A + 3)) * y * y + 1;
        float c3 = 1.f - c0 - c1 - c2;
        float cf[4] = {c0, c1, c2, c3};
        short q[4];
        for (int k = 0; k < 4; k++) {
            long r = lrintf(cf[k] * 2048.f);
            r = r > 32767 ? 32767 : (r < -32768 ? -32768 : r);
            q[k] = (short)r;
        }
        ofs[d] = s;
        coef[d] = make_short4(q[0], q[1], q[2], q[3]);
    }
}

int get_taps(Ctx* c, int src, int dst, TapTable** out) {
    TapTable* victim = &c->taps[0];
    for (auto& t : c->taps) {
        if (t.src == src && t.dst == dst && t.d_ofs) {
            t.stamp = ++c->tap_clock;
            *out = &t;
            return SRCNN_OK;
        }
        if (t.stamp < victim->stamp) victim = &t;
    }
    TapTable& t = *victim;
    if (t.d_ofs) {  // evict: in-flight kernels may still read it, captured pipelines hold its addresses
        drop_graphs(c);
        SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
        cudaFree(t.d_ofs);
        cudaFree(t.d_coef);
        t.d_ofs = nullptr;
        t.d_coef = nullptr;
    }
    t.src = src;
    t.dst = dst;
    t.h_ofs.resize(dst);
    t.h_coef.resize(dst);
    build_cubic_taps(src, dst, t.h_ofs.data(), t.h_coef.data());
    // integer up-scale: sample d = S*j + k reads source columns j-2+(k >= S/2) .. +3 with the taps of phase k, whatever j is.
    // Checked, not assumed: the integer-scale kernel (color_bicubic_int.cu) is only chosen for a table that really is periodic.
    t.int_scale = 0;
    if (dst % src == 0 && (dst / src == 2 || dst / src == 4)) {
        const int S = dst / src;
        bool periodic = true;
        for (int d = 0; d < dst && periodic; d++) {
            const short4 a = t.h_coef[d], b = t.h_coef[d % S];
            periodic = t.h_ofs[d] == d / S - 1 + ((d % S) >= S / 2 ? 1 : 0) && a.x == b.x && a.y == b.y && a.z == b.z && a.w == b.w;
        }
        if (periodic) t.int_scale = S;
    }
    SRCNN_CUDA(c, cudaMalloc(&t.d_ofs, sizeof(int) * (size_t)dst));
    SRCNN_CUDA(c, cudaMalloc(&t.d_coef, sizeof(short4) * (size_t)dst));

    // pageable source: the runtime stages it before returning, so the vectors may be reused freely
    SRCNN_CUDA(c, cudaMemcpyAsync(t.d_ofs, t.h_ofs.data(), sizeof(int) * (size_t)dst, cudaMemcpyHostToDevice, c->stream));
    SRCNN_CUDA(c, cudaMemcpyAsync(t.d_coef, t.h_coef.data(), sizeof(short4) * (size_t)dst, cudaMemcpyHostToDevice, c->stream));
    t.stamp = ++c->tap_clock;
    *out = &t;
    return SRCNN_OK;
}

// ------------------------------------------------------------------------------------------------
// K-A, direct form: one thread per output pixel, everything from global memory.  Used for any
// geometry the tiled kernel's shared-memory footprint cannot hold (strong down-scales) and as the
// in-library cross-check of the tiled kernel.
// ------------------------------------------------------------------------------------------------
// planes: 3 = Y, Cr, Cb of a colour source, 4 = Y, Cr, Cb and the raw alpha byte of a four-channel source (into pa)
template <int NP>
__global__ void __launch_bounds__(256) k_color_bicubic_direct(ResizeDev p, uint8_t* pa) {
    const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
    const int dy = p.row_begin + blockIdx.y * 8 + (threadIdx.x >> 5);
    if (dx >= p.ow || dy >= p.row_end) return;
    const int sx = p.xofs[dx], sy = p.yofs[dy];
    const short4 cx = p.xcoef[dx], cy = p.ycoef[dy];
    const int cxs[4] = {cx.x, cx.y, cx.z, cx.w};
    int hY[4], hCr[4], hCb[4], hA[4];
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const int gy = clampi(sy - 1 + r, 0, p.sh - 1) - p.src_row0;
        const uint8_t* row = p.src + (size_t)gy * p.src_stride;
        int aY = 0, aCr = 0, aCb = 0, aA = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int gx = clampi(sx - 1 + k, 0, p.sw - 1);
            int c0 = row[NP * gx], c1 = row[NP * gx + 1], c2 = row[NP * gx + 2];
            if (NP == 4) aA += (int)row[NP * gx + 3] * cxs[k];
            int B = p.swapRB ? c2 : c0, R = p.swapRB ? c0 : c2;
            int Y, Cr, Cb;
            bgr_to_ycc(B, c1, R, Y, Cr, Cb);
            aY += Y * cxs[k];
            aCr += Cr * cxs[k];
            aCb += Cb * cxs[k];
        }
        hY[r] = aY; hCr[r] = aCr; hCb[r] = aCb; hA[r] = aA;
    }
    const bool fpath = dx < p.simd_w;
    const size_t o = (size_t)(dy - p.plane_row0) * p.pitch + dx;
    p.y[o] = (uint8_t)vertical_tap(hY[0], hY[1], hY[2], hY[3], cy, fpath);
    p.cr[o] = (uint8_t)vertical_tap(hCr[0], hCr[1], hCr[2], hCr[3], cy, fpath);
    p.cb[o] = (uint8_t)vertical_tap(hCb[0], hCb[1], hCb[2], hCb[3], cy, fpath);
    if (NP == 4) pa[o] = (uint8_t)vertical_tap(hA[0], hA[1], hA[2], hA[3], cy, fpath);
}

// The same for NPL planes of raw bytes (no colour conversion; byte loads and stores: any alignment).  Plane k's sample x of a
// row is byte k * sv + x * sstep past the row's start in the source, k * dv + x * dstep past it in p.y.  A grey plane: one plane,
// steps 1; the Y bytes of packed 4:2:2 rows: sstep 2; their U and V bytes: sv 2, sstep 4, dv the distance of the V output plane
// from the U one; NV12's chroma pairs: sv = dv = 1, steps 2; I420's U and V planes: sv / dv = V's distance from U, steps 1.
template <int NPL>
__global__ void __launch_bounds__(256) k_planes_bicubic_direct(ResizeDev p, size_t sv, int sstep, size_t dv, int dstep) {
    const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
    const int dy = p.row_begin + blockIdx.y * 8 + (threadIdx.x >> 5);
    if (dx >= p.ow || dy >= p.row_end) return;
    const int sx = p.xofs[dx], sy = p.yofs[dy];
    const short4 cx = p.xcoef[dx], cy = p.ycoef[dy];
    const int cxs[4] = {cx.x, cx.y, cx.z, cx.w};
    int h[NPL][4];
#pragma unroll
    for (int r = 0; r < 4; r++) {
        const uint8_t* row = p.src + (size_t)(clampi(sy - 1 + r, 0, p.sh - 1) - p.src_row0) * p.src_stride;
        int acc[NPL] = {};
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const size_t x = (size_t)clampi(sx - 1 + k, 0, p.sw - 1) * sstep;
#pragma unroll
            for (int pl = 0; pl < NPL; pl++) acc[pl] += (int)row[pl * sv + x] * cxs[k];
        }
#pragma unroll
        for (int pl = 0; pl < NPL; pl++) h[pl][r] = acc[pl];
    }
    const bool fpath = dx < p.simd_w;
    uint8_t* d = p.y + (size_t)(dy - p.plane_row0) * p.pitch + (size_t)dx * dstep;
#pragma unroll
    for (int pl = 0; pl < NPL; pl++) d[pl * dv] = (uint8_t)vertical_tap(h[pl][0], h[pl][1], h[pl][2], h[pl][3], cy, fpath);
}

// ------------------------------------------------------------------------------------------------
// K-A, tiled form (the fast path for up-scaling).  One CTA produces a TW x TH tile of all NP
// planes: (1) the source footprint is colour-converted ONCE into shared memory (three u8 planes,
// replicate border applied at load; a grey source, NP = 1, is copied as it is), (2) the integer
// horizontal pass runs once per footprint row, (3) the vertical pass reads four shared-memory sums
// per sample and writes 4 pixels per store.
// ------------------------------------------------------------------------------------------------
constexpr int kTW = 64;                 // output tile width; the height is a template parameter (64 or 32 rows)
constexpr int kMaxSC = 72, kMaxSR = 40; // footprint capacity (source cols / rows incl. the 3-tap apron)
constexpr int kMaxSR4 = 35;             // ... rows with four planes (the static shared memory of one CTA stays within 48 KB)
__host__ __device__ constexpr int tiled_max_rows(int np) { return np == 4 ? kMaxSR4 : kMaxSR; }

// NP = 4: the planes of a four-channel source, plane 3 (alpha, the raw byte 3 of each pixel) into pa.  NP = 2: the two bytes of an
// interleaved pair (NV12 chroma) as two planes, written back interleaved into p.y (4-byte aligned rows).  NP = 5 / 6: packed 4:2:2
// rows as in k_planes_bicubic_direct (one / two planes, NPL below), written like a grey call's plane / into p.y and p.cr.
template <int kTH, int NP>
__global__ void __launch_bounds__(256, 5) k_color_bicubic_tiled(ResizeDev p, uint8_t* pa) {   // 5 CTAs per SM: 48 registers (4 CTAs measured 6 % slower)
    constexpr int SR = tiled_max_rows(NP);
    constexpr int NPL = NP == 5 ? 1 : (NP == 6 ? 2 : NP);    // planes
    __shared__ __align__(16) uint8_t sP[NPL][SR][kMaxSC + 8];   // +8: the 3-word window read of the last quad may run past a row
    // horizontal sums kept as float: they are integers below 2^24, so the conversion is exact and is done
    // once per sum instead of once per use in the vertical pass
    __shared__ __align__(16) float sH[NPL][SR][kTW];
    // per tile row: the four vertical taps as floats (b_k = coef_k * 2^-22, exact) and the first tap's row in sH -- computed once
    // per tile instead of once per (thread, row) in the vertical pass
    __shared__ __align__(16) float4 sB[kTH];
    __shared__ int sSr[kTH];

    const size_t fz = blockIdx.z;                       // frame of a batch
    const uint8_t* const fsrc = p.src + fz * p.src_frame;
    const size_t fplane = fz * p.plane_frame, fy16 = fz * p.y16_frame;
    const int dx0 = blockIdx.x * kTW;
    const int dy0 = p.row_begin + blockIdx.y * kTH;
    const int dx1 = min(dx0 + kTW, p.ow), dy1 = min(dy0 + kTH, p.row_end);
    const int sx_lo = p.xofs[dx0] - 1, sx_hi = p.xofs[dx1 - 1] + 2;
    const int sy_lo = p.yofs[dy0] - 1, sy_hi = p.yofs[dy1 - 1] + 2;
    const int nsc = sx_hi - sx_lo + 1, nsr = sy_hi - sy_lo + 1;
    const int tid = threadIdx.x;

    if (tid < kTH && dy0 + tid < dy1) {
        const short4 cy = p.ycoef[dy0 + tid];
        const float sc = 1.0f / 4194304.0f;  // 2^-22, exact
        sB[tid] = make_float4(__fmul_rn((float)cy.x, sc), __fmul_rn((float)cy.y, sc), __fmul_rn((float)cy.z, sc), __fmul_rn((float)cy.w, sc));
        sSr[tid] = p.yofs[dy0 + tid] - 1 - sy_lo;
    }
    // (1) colour-convert the footprint (replicate border applied here); i / nsc by multiply-shift (exact for i < 2^12).
    //     The B and R bytes are picked by pointer offset, the chroma clamps are one saturating conversion each.
    const unsigned rcp20 = ((1u << 20) + (unsigned)nsc - 1u) / (unsigned)nsc;
    const int oB = p.swapRB ? 2 : 0, oR = 2 - oB;
    for (int i = tid; i < nsr * nsc; i += 256) {
        const int r = (int)(((unsigned)i * rcp20) >> 20), c = i - r * nsc;
        const int gy = clampi(sy_lo + r, 0, p.sh - 1) - p.src_row0;
        const int gx = clampi(sx_lo + c, 0, p.sw - 1);
        if (NP == 1) {
            sP[0][r][c] = fsrc[(size_t)gy * p.src_stride + gx];
            continue;
        }
        if (NP == 5) {
            sP[0][r][c] = fsrc[(size_t)gy * p.src_stride + 2 * (size_t)gx];
            continue;
        }
        if (NP == 6) {
            const uint8_t* px = fsrc + (size_t)gy * p.src_stride + 4 * (size_t)gx;
            sP[0][r][c] = px[0];
            sP[NPL - 1][r][c] = px[2];
            continue;
        }
        if (NP == 2) {
            const uint8_t* px = fsrc + (size_t)gy * p.src_stride + 2 * (size_t)gx;
            sP[0][r][c] = px[0];
            sP[NP - 1][r][c] = px[1];
            continue;
        }
        const uint8_t* px = fsrc + (size_t)gy * p.src_stride + (NP == 4 ? 4 : 3) * (size_t)gx;
        const int B = px[oB], G = px[1], R = px[oR];
        if (NP == 4) sP[NP - 1][r][c] = px[3];
        const int Y = (1868 * B + 9617 * G + 4899 * R + 8192) >> 14;          // OpenCV RGB2YCrCb_i<uchar>, yuv_shift 14
        uint32_t Cr, Cb;
        asm("cvt.sat.u8.s32 %0, %1;" : "=r"(Cr) : "r"(((R - Y) * 11682 + (128 << 14) + 8192) >> 14));
        asm("cvt.sat.u8.s32 %0, %1;" : "=r"(Cb) : "r"(((B - Y) * 9241 + (128 << 14) + 8192) >> 14));
        sP[0][r][c] = (uint8_t)Y;
        sP[NP > 1 ? 1 : 0][r][c] = (uint8_t)Cr;
        sP[NP > 1 ? 2 : 0][r][c] = (uint8_t)Cb;
    }
    __syncthreads();

    // (2) integer horizontal pass.  Fast form (any up-scale): a thread owns 4 adjacent output columns; their taps lie
    //     in one 8-byte window of the converted row, fetched as three aligned words + funnel shifts, and each sum is
    //     two dp2a (signed 16-bit taps x unsigned 8-bit pixels).  Slow form: one column per thread, byte loads.
    if (p.quad_ok) {
        const int q = tid & 15, col = q * 4, dx = dx0 + col;
        if (dx < dx1) {
            const int s0 = p.xofs[dx] - 1 - sx_lo;
            int off[4];
            uint32_t k01[4], k23[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int dxj = min(dx + j, dx1 - 1);           // columns past the tile edge repeat the last one (never stored)
                off[j] = 8 * (p.xofs[dxj] - p.xofs[dx]);
                const short4 cx = p.xcoef[dxj];
                k01[j] = ((uint32_t)(unsigned short)cx.x) | ((uint32_t)(unsigned short)cx.y << 16);
                k23[j] = ((uint32_t)(unsigned short)cx.z) | ((uint32_t)(unsigned short)cx.w << 16);
            }
            const int wsh = 8 * (s0 & 3);
            for (int r = tid >> 4; r < nsr; r += 16) {
#pragma unroll
                for (int pl = 0; pl < NPL; pl++) {
                    const uint32_t* w = reinterpret_cast<const uint32_t*>(&sP[pl][r][s0 & ~3]);
                    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
                    const uint32_t lo = __funnelshift_r(w0, w1, wsh), hi = __funnelshift_r(w1, w2, wsh);
                    float h[4];
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const uint32_t px4 = __funnelshift_rc(lo, hi, off[j]);
                        int acc;
                        asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(acc) : "r"(k01[j]), "r"(px4), "r"(0));
                        asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(acc) : "r"(k23[j]), "r"(px4), "r"(acc));
                        h[j] = (float)acc;
                    }
                    *reinterpret_cast<float4*>(&sH[pl][r][col]) = make_float4(h[0], h[1], h[2], h[3]);
                }
            }
        }
    } else {
        const int col = tid & (kTW - 1);
        const int dx = dx0 + col;
        if (dx < dx1) {
            const int s = p.xofs[dx] - 1 - sx_lo;
            const short4 cx = p.xcoef[dx];
            const int k0 = cx.x, k1 = cx.y, k2 = cx.z, k3 = cx.w;
            for (int r = tid >> 6; r < nsr; r += 256 / kTW) {
#pragma unroll
                for (int pl = 0; pl < NPL; pl++) {
                    const uint8_t* q = &sP[pl][r][s];
                    sH[pl][r][col] = (float)((int)q[0] * k0 + (int)q[1] * k1 + (int)q[2] * k2 + (int)q[3] * k3);
                }
            }
        }
    }
    __syncthreads();

    // (3) vertical pass: thread owns 4 consecutive columns (one 128-bit shared load per tap row) and
    //     walks the tile rows; v = H0*b0 + (H1*b1 + (H2*b2 + H3*b3)), separate multiplies and adds
    // Interior tiles (whole, on cv::resize's float path, not touching the first / last image column) take a form of the pass
    // without per-sample edge cases and with running output pointers: address arithmetic and branches were 40 % of the pass's
    // instructions (ncu source page), the 42 packed FP32 operations, 12 loads, 12 conversions and 3 stores per task are not.
    if (dx0 > 0 && dx0 + kTW < p.ow && dx0 + kTW <= p.simd_w && dy0 + kTH <= p.row_end) {
        const int col = (tid & 15) * 4, ty0 = tid >> 4;
        const unsigned long long nz = p.negzero2;
        const size_t o = fplane + (size_t)(dy0 + ty0 - p.plane_row0) * p.pitch + (size_t)(dx0 + col) * (NP == 2 ? 2 : 1);
        uint8_t* pcr = NP == 3 || NP == 4 || NP == 6 ? p.cr + o : nullptr;
        uint8_t* pcb = NP == 3 || NP == 4 ? p.cb + o : nullptr;
        uint8_t* ppa = NP == 4 ? pa + o : nullptr;
        uint8_t* py = p.y16 ? p.y16 + fy16 + (size_t)(dy0 + ty0 - p.plane_row0) * p.pitch16 + 2 * (size_t)(dx0 + col + kY16Pad) : p.y + o;
        const size_t step = 16 * p.pitch, ystep = p.y16 ? 16 * p.pitch16 : step;
        const bool y16 = p.y16 != nullptr;
#pragma unroll
        for (int k = 0; k < kTH / 16; k++) {
            const int ty = ty0 + 16 * k;
            const float4 bq = sB[ty];
            const float* hrow = &sH[0][sSr[ty]][col];
            uint32_t packed[NPL > 3 ? NPL : 3];
#pragma unroll
            for (int pl = 0; pl < NPL; pl++) {
                const float* h = hrow + pl * (SR * kTW);
                const ulonglong2 g0 = *reinterpret_cast<const ulonglong2*>(h);
                const ulonglong2 g1 = *reinterpret_cast<const ulonglong2*>(h + kTW);
                const ulonglong2 g2 = *reinterpret_cast<const ulonglong2*>(h + 2 * kTW);
                const ulonglong2 g3 = *reinterpret_cast<const ulonglong2*>(h + 3 * kTW);
                const unsigned long long bb0 = f2_pack(bq.x, bq.x), bb1 = f2_pack(bq.y, bq.y), bb2 = f2_pack(bq.z, bq.z), bb3 = f2_pack(bq.w, bq.w);
                unsigned long long va = f2_mul_rn(g3.x, bb3, nz), vb = f2_mul_rn(g3.y, bb3, nz);
                va = f2_add_rn(f2_mul_rn(g2.x, bb2, nz), va);
                vb = f2_add_rn(f2_mul_rn(g2.y, bb2, nz), vb);
                va = f2_add_rn(f2_mul_rn(g1.x, bb1, nz), va);
                vb = f2_add_rn(f2_mul_rn(g1.y, bb1, nz), vb);
                va = f2_add_rn(f2_mul_rn(g0.x, bb0, nz), va);
                vb = f2_add_rn(f2_mul_rn(g0.y, bb0, nz), vb);
                float v0, v1, v2, v3;
                f2_unpack(va, v0, v1);
                f2_unpack(vb, v2, v3);
                const uint32_t r0 = sat_u8_rn(v0), r1 = sat_u8_rn(v1), r2 = sat_u8_rn(v2), r3 = sat_u8_rn(v3);
                if (pl == 0 && y16) {   // exact u8 -> FP16: 0x6400 | v is 1024 + v, minus 1024
                    const __half2 k1024 = __float2half2_rn(1024.f);
                    uint32_t a01 = (r0 | (r1 << 16)) | 0x64006400u, a23 = (r2 | (r3 << 16)) | 0x64006400u;
                    __half2 h01 = __hsub2(*reinterpret_cast<__half2*>(&a01), k1024), h23 = __hsub2(*reinterpret_cast<__half2*>(&a23), k1024);
                    *reinterpret_cast<uint2*>(py) = make_uint2(*reinterpret_cast<uint32_t*>(&h01), *reinterpret_cast<uint32_t*>(&h23));
                } else {
                    packed[pl] = r0 | (r1 << 8) | (r2 << 16) | (r3 << 24);
                }
            }
            if (NP == 2) {   // U0 V0 U1 V1 | U2 V2 U3 V3
                reinterpret_cast<uint32_t*>(py)[0] = __byte_perm(packed[0], packed[1], 0x5140);
                reinterpret_cast<uint32_t*>(py)[1] = __byte_perm(packed[0], packed[1], 0x7362);
            } else if (!y16) {
                *reinterpret_cast<uint32_t*>(py) = packed[0];
            }
            py += ystep;
            if (NP == 6) {
                *reinterpret_cast<uint32_t*>(pcr) = packed[1];
                pcr += step;
            }
            if (NP == 3 || NP == 4) {
                *reinterpret_cast<uint32_t*>(pcr) = packed[1];
                *reinterpret_cast<uint32_t*>(pcb) = packed[2];
                pcr += step; pcb += step;
            }
            if (NP == 4) {
                *reinterpret_cast<uint32_t*>(ppa) = packed[NP - 1];
                ppa += step;
            }
        }
        return;
    }
    {
        const int q = tid & 15, col = q * 4, dx = dx0 + col;
        if (dx < dx1) {
            const bool all_float = dx + 3 < p.simd_w && dx + 3 < dx1;
            const unsigned long long nz = p.negzero2;
            for (int ty = tid >> 4; ty < kTH; ty += 16) {
                const int dy = dy0 + ty;
                if (dy >= dy1) break;
                const int sr = sSr[ty];
                const float4 bq = sB[ty];
                const float b0 = bq.x, b1 = bq.y, b2 = bq.z, b3 = bq.w;
                const size_t o = fplane + (size_t)(dy - p.plane_row0) * p.pitch + dx;
                const unsigned long long bb0 = f2_pack(b0, b0), bb1 = f2_pack(b1, b1), bb2 = f2_pack(b2, b2), bb3 = f2_pack(b3, b3);
#pragma unroll
                for (int pl = 0; pl < NPL; pl++) {
                    if (all_float) {   // two samples per instruction: v = H0*b0 + (H1*b1 + (H2*b2 + H3*b3)), each op rounded
                        const ulonglong2 g0 = *reinterpret_cast<const ulonglong2*>(&sH[pl][sr][col]);
                        const ulonglong2 g1 = *reinterpret_cast<const ulonglong2*>(&sH[pl][sr + 1][col]);
                        const ulonglong2 g2 = *reinterpret_cast<const ulonglong2*>(&sH[pl][sr + 2][col]);
                        const ulonglong2 g3 = *reinterpret_cast<const ulonglong2*>(&sH[pl][sr + 3][col]);
                        unsigned long long va = f2_mul_rn(g3.x, bb3, nz), vb = f2_mul_rn(g3.y, bb3, nz);
                        va = f2_add_rn(f2_mul_rn(g2.x, bb2, nz), va);
                        vb = f2_add_rn(f2_mul_rn(g2.y, bb2, nz), vb);
                        va = f2_add_rn(f2_mul_rn(g1.x, bb1, nz), va);
                        vb = f2_add_rn(f2_mul_rn(g1.y, bb1, nz), vb);
                        va = f2_add_rn(f2_mul_rn(g0.x, bb0, nz), va);
                        vb = f2_add_rn(f2_mul_rn(g0.y, bb0, nz), vb);
                        float v0, v1, v2, v3;
                        f2_unpack(va, v0, v1);
                        f2_unpack(vb, v2, v3);
                        const uint32_t r0 = sat_u8_rn(v0), r1 = sat_u8_rn(v1), r2 = sat_u8_rn(v2), r3 = sat_u8_rn(v3);
                        if (pl == 0 && p.y16) {   // Y as FP16 for the tcgen05 kernel's TMA staging; exact: 0x6400 | v is 1024 + v, minus 1024
                            const __half2 k1024 = __float2half2_rn(1024.f);
                            uint32_t a01 = (r0 | (r1 << 16)) | 0x64006400u, a23 = (r2 | (r3 << 16)) | 0x64006400u;
                            __half2 h01 = __hsub2(*reinterpret_cast<__half2*>(&a01), k1024), h23 = __hsub2(*reinterpret_cast<__half2*>(&a23), k1024);
                            const uint32_t w01 = *reinterpret_cast<uint32_t*>(&h01), w23 = *reinterpret_cast<uint32_t*>(&h23);
                            uint8_t* o16 = p.y16 + fy16 + (size_t)(dy - p.plane_row0) * p.pitch16 + 2 * (size_t)(dx + kY16Pad);
                            *reinterpret_cast<uint2*>(o16) = make_uint2(w01, w23);
                            if (dx == 0) {            // replicated columns -8..-1 (conv1 reads Y[clamp(c-4)], src/srcnn.cpp:279)
                                const uint32_t e = __byte_perm(w01, 0, 0x1010);
                                *reinterpret_cast<uint4*>(o16 - 2 * kY16Pad) = make_uint4(e, e, e, e);
                            }
                            if (dx + 4 >= p.ow) {     // this thread holds the last column: replicate it into W..W+7
                                const unsigned short e = (unsigned short)(w23 >> 16);
                                unsigned short* q16 = reinterpret_cast<unsigned short*>(o16) + 4;
#pragma unroll
                                for (int k = 0; k < 8; k++) q16[k] = e;
                            }
                            continue;
                        }
                        if (NP == 2) {
                            uint8_t* d = p.y + o + dx + pl;
                            d[0] = (uint8_t)r0; d[2] = (uint8_t)r1; d[4] = (uint8_t)r2; d[6] = (uint8_t)r3;
                            continue;
                        }
                        uint8_t* outp = (pl == 0 ? p.y : (pl == 1 ? p.cr : (NP == 4 && pl == 3 ? pa : p.cb))) + o;
                        *reinterpret_cast<uint32_t*>(outp) = r0 | (r1 << 8) | (r2 << 16) | (r3 << 24);
                        continue;
                    }
                    const float4 h0 = *reinterpret_cast<const float4*>(&sH[pl][sr][col]);
                    const float4 h1 = *reinterpret_cast<const float4*>(&sH[pl][sr + 1][col]);
                    const float4 h2 = *reinterpret_cast<const float4*>(&sH[pl][sr + 2][col]);
                    const float4 h3 = *reinterpret_cast<const float4*>(&sH[pl][sr + 3][col]);
                    uint8_t* out = (pl == 0 ? p.y : (pl == 1 ? p.cr : (NP == 4 && pl == 3 ? pa : p.cb))) + o;
                    {  // tile edge and/or cv::resize's integer scalar tail (last ow mod 8 columns)
                        const float hh[4][4] = {{h0.x, h0.y, h0.z, h0.w}, {h1.x, h1.y, h1.z, h1.w}, {h2.x, h2.y, h2.z, h2.w}, {h3.x, h3.y, h3.z, h3.w}};
                        for (int j = 0; j < 4 && dx + j < dx1; j++) {
                            const int r = vertical_tap(__float2int_rn(hh[0][j]), __float2int_rn(hh[1][j]), __float2int_rn(hh[2][j]),
                                                       __float2int_rn(hh[3][j]), p.ycoef[dy], (dx + j) < p.simd_w);
                            if (pl == 0 && p.y16) {
                                const unsigned short e = __half_as_ushort(__ushort2half_rn((unsigned short)r));
                                unsigned short* q16 = reinterpret_cast<unsigned short*>(p.y16 + fy16 + (size_t)(dy - p.plane_row0) * p.pitch16) + kY16Pad + dx + j;
                                q16[0] = e;
                                if (dx + j == 0)
                                    for (int k = 1; k <= kY16Pad; k++) q16[-k] = e;
                                if (dx + j == p.ow - 1)
                                    for (int k = 1; k <= 8; k++) q16[k] = e;
                            } else if (NP == 2) {
                                p.y[o + dx + 2 * j + pl] = (uint8_t)r;
                            } else {
                                out[j] = (uint8_t)r;
                            }
                        }
                    }
                }
            }
        }
    }
}


static ResizeDev resize_dev(const ResizeArgs& a) {
    ResizeDev p;
    p.src = a.src;
    p.src_stride = a.src_stride;
    p.sw = a.sw; p.sh = a.sh; p.src_row0 = a.src_row0;
    p.swapRB = a.order == SRCNN_ORDER_RGB || a.order == SRCNN_ORDER_RGBA;
    p.ow = a.ow; p.oh = a.oh;
    p.row_begin = a.row_begin; p.row_end = a.row_end;
    p.y = a.pl.y; p.cr = a.pl.cr; p.cb = a.pl.cb;
    p.pitch = a.pl.pitch;
    p.y16 = a.pl.y16; p.pitch16 = a.pl.pitch16;       // tiled kernel: the tcgen05 path's Y goes straight to the padded FP16 plane
    p.src_frame = a.src_frame_stride; p.plane_frame = a.pl.frame_stride; p.y16_frame = a.pl.frame_stride16;
    p.plane_row0 = a.pl.row0;
    p.xofs = a.tx->d_ofs; p.xcoef = a.tx->d_coef;
    p.yofs = a.ty->d_ofs; p.ycoef = a.ty->d_coef;
    p.simd_w = (a.ow / 8) * 8;
    p.negzero2 = 0x8000000080000000ull;
    p.quad_ok = 1;
    return p;
}

static int launch_yuv420(Ctx* c, const ResizeArgs& a);
static int launch_yuv422(Ctx* c, const ResizeArgs& a);
static int launch_graya(Ctx* c, const ResizeArgs& a);

int launch_color_bicubic(Ctx* c, const ResizeArgs& a) {
    if (a.order == SRCNN_ORDER_GRAYA) return launch_graya(c, a);
    if (yuv420(a.order) || yuv422(a.order)) {
        if (c->ka_int) {   // x2 / x4: luma and chroma in one launch of the integer-scale kernel
            ResizeArgs y = a;
            y.order = SRCNN_ORDER_GRAY;
            bool done = false;
            const int rc = launch_yuv_int(c, resize_dev(y), a, &done);
            if (rc || done) return rc;
        }
        return yuv420(a.order) ? launch_yuv420(c, a) : launch_yuv422(c, a);
    }
    ResizeDev p = resize_dev(a);
    const int nframes = std::max(1, a.nframes);
    const int rows = a.row_end - a.row_begin;
    if (rows <= 0) return SRCNN_OK;

    // does every tile's source footprint fit the tiled kernel's shared memory?  (64-row tiles amortise the 3-row apron and
    // fill the horizontal pass better: 33 vs 38 us at 1080p -> 4K; 32-row tiles cover smaller up-scales such as x1.5)
    bool fits_x = true;
    for (int dx0 = 0; dx0 < a.ow && fits_x; dx0 += kTW) {
        int dx1 = std::min(dx0 + kTW, a.ow);
        if (a.tx->h_ofs[dx1 - 1] - a.tx->h_ofs[dx0] + 4 > kMaxSC) fits_x = false;
    }
    const bool gray = a.order == SRCNN_ORDER_GRAY, four = four_channel(a.order), uv = a.order == kOrderUV;
    const bool y422 = a.order == kOrderY422, uv422 = a.order == kOrderUV422;
    uint8_t* const pa = four ? a.pl.a : nullptr;
    const int max_rows = tiled_max_rows(four ? 4 : 3);
    auto fits_rows = [&](int th) {
        for (int dy0 = a.row_begin; dy0 < a.row_end; dy0 += th) {
            int dy1 = std::min(dy0 + th, a.row_end);
            if (a.ty->h_ofs[dy1 - 1] - a.ty->h_ofs[dy0] + 4 > max_rows) return false;
        }
        return true;
    };
    const int th = !fits_x ? 0 : (fits_rows(64) ? 64 : (fits_rows(32) ? 32 : 0));
    for (int dx = 0; dx + 3 < a.ow && p.quad_ok; dx += 4)
        if (a.tx->h_ofs[dx + 3] - a.tx->h_ofs[dx] > 4) p.quad_ok = 0;
    if (c->ka_int && !uv && !y422 && !uv422) {                           // x2 / x4: the integer-scale kernel (constant tap phases, no tables)
        bool done = false;
        const int rc = launch_color_bicubic_int(c, p, a, &done);
        if (rc || done) return rc;
    }
    if (th) {
        dim3 grid((a.ow + kTW - 1) / kTW, (rows + th - 1) / th, nframes);   // a batch of frames is one launch
        if (th == 64) (gray ? k_color_bicubic_tiled<64, 1> : uv ? k_color_bicubic_tiled<64, 2> : four ? k_color_bicubic_tiled<64, 4> : y422 ? k_color_bicubic_tiled<64, 5>
                       : uv422 ? k_color_bicubic_tiled<64, 6> : k_color_bicubic_tiled<64, 3>)<<<grid, 256, 0, c->stream>>>(p, pa);
        else (gray ? k_color_bicubic_tiled<32, 1> : uv ? k_color_bicubic_tiled<32, 2> : four ? k_color_bicubic_tiled<32, 4> : y422 ? k_color_bicubic_tiled<32, 5>
              : uv422 ? k_color_bicubic_tiled<32, 6> : k_color_bicubic_tiled<32, 3>)<<<grid, 256, 0, c->stream>>>(p, pa);
        c->launches++;
        SRCNN_CUDA(c, cudaGetLastError());
        return SRCNN_OK;
    }
    // the direct kernel (strong down-scales, rare): frame by frame; it writes the u8 plane, the FP16 copy is a pass of its own
    for (int f = 0; f < nframes; f++) {
        ResizeDev q = p;
        q.src += (size_t)f * p.src_frame;
        q.y += (size_t)f * p.plane_frame;
        dim3 grid((a.ow + 31) / 32, (rows + 7) / 8);
        if (gray || y422) {
            k_planes_bicubic_direct<1><<<grid, 256, 0, c->stream>>>(q, 0, y422 ? 2 : 1, 0, 1);
        } else if (uv) {
            k_planes_bicubic_direct<2><<<grid, 256, 0, c->stream>>>(q, 1, 2, 1, 2);
        } else if (uv422) {
            k_planes_bicubic_direct<2><<<grid, 256, 0, c->stream>>>(q, 2, 4, (size_t)(p.cr - p.y), 1);
        } else {
            q.cr += (size_t)f * p.plane_frame;
            q.cb += (size_t)f * p.plane_frame;
            uint8_t* const qa = four ? pa + (size_t)f * p.plane_frame : nullptr;
            (four ? k_color_bicubic_direct<4> : k_color_bicubic_direct<3>)<<<grid, 256, 0, c->stream>>>(q, qa);
        }
        c->launches++;
        SRCNN_CUDA(c, cudaGetLastError());
        if (a.pl.y16) {
            int rc = launch_y8_to_y16(c, q.y, a.pl.pitch, a.ow, rows, a.pl.y16 + (size_t)f * a.pl.frame_stride16, a.pl.pitch16);
            if (rc) return rc;
        }
    }
    return SRCNN_OK;
}

// A 4:2:0 frame (SRCNN_ORDER_NV12 / _I420).  x2 / x4 with ow/2 % 8 == 0 and 8-byte aligned chroma rows: one launch for luma and
// chroma (color_bicubic_int.cu).  Otherwise the Y plane takes the grey instances and the chroma planes the generic ones, resized as
// an image of their own straight into the caller's output: NV12's pairs as two interleaved planes (NP = 2), I420's U and V planes
// as two frames of a one-plane launch (one launch for a single frame, one per plane for a batch).  Chroma rows of the output that
// are not 4-byte aligned (the tiled kernel stores words) take k_planes_bicubic_direct, one launch per frame for both planes.
static int launch_yuv420(Ctx* c, const ResizeArgs& a) {
    ResizeArgs y = a;
    y.order = SRCNN_ORDER_GRAY;
    int rc = launch_color_bicubic(c, y);
    if (rc) return rc;
    const Chroma420& ch = a.ch;
    const bool words = (((uintptr_t)ch.dst | ch.dst_pitch | ch.dst_v | ch.dst_frame) & 3) == 0;
    ResizeArgs u;
    u.src = ch.src; u.src_stride = ch.src_pitch;
    u.sw = ch.sw; u.sh = ch.sh; u.src_row0 = 0; u.src_row1 = ch.sh;
    u.ow = ch.ow; u.oh = ch.oh;
    u.row_begin = ch.row_begin; u.row_end = ch.row_end;
    u.pl.y = ch.dst; u.pl.pitch = ch.dst_pitch; u.pl.row0 = 0; u.pl.rows = ch.oh; u.pl.frame_stride = ch.dst_frame;
    u.tx = ch.tx; u.ty = ch.ty;
    u.nframes = a.nframes; u.src_frame_stride = a.src_frame_stride;
    if (!words) {
        if (ch.row_end <= ch.row_begin) return SRCNN_OK;
        const bool nv12 = a.order == SRCNN_ORDER_NV12;
        u.order = SRCNN_ORDER_GRAY;
        for (int f = 0; f < std::max(1, a.nframes); f++) {
            ResizeDev q = resize_dev(u);
            q.src += (size_t)f * a.src_frame_stride;
            q.y += (size_t)f * ch.dst_frame;
            dim3 grid((ch.ow + 31) / 32, (ch.row_end - ch.row_begin + 7) / 8);
            k_planes_bicubic_direct<2><<<grid, 256, 0, c->stream>>>(q, nv12 ? 1 : ch.src_v, nv12 ? 2 : 1, nv12 ? 1 : ch.dst_v, nv12 ? 2 : 1);
            c->launches++;
            SRCNN_CUDA(c, cudaGetLastError());
        }
        return SRCNN_OK;
    }
    if (a.order == SRCNN_ORDER_NV12) {
        u.order = kOrderUV;
        return launch_color_bicubic(c, u);
    }
    u.order = SRCNN_ORDER_GRAY;
    if (std::max(1, a.nframes) == 1) {   // V is U's second frame
        u.nframes = 2; u.src_frame_stride = ch.src_v; u.pl.frame_stride = ch.dst_v;
        return launch_color_bicubic(c, u);
    }
    if ((rc = launch_color_bicubic(c, u))) return rc;
    u.src += ch.src_v; u.pl.y += ch.dst_v;
    return launch_color_bicubic(c, u);
}

// A packed 4:2:2 frame (SRCNN_ORDER_YUY2 / _UYVY).  x2 / x4 with ow % 16 == 0: one launch for luma and chroma (color_bicubic_int.cu).
// Otherwise two launches of the generic kernels: the Y plane as every second byte of the rows (kOrderY422, into pl.y / pl.y16 as a
// grey call's), then U and V as bytes 0 and 2 of each macropixel (kOrderUV422) into the workspace's Cr / Cb planes.  The two
// variants differ only in where the first Y / U byte of a row is.  (The direct kernels, for strong down-scales, go frame by frame.)
static int launch_yuv422(Ctx* c, const ResizeArgs& a) {
    const bool uyvy = a.order == SRCNN_ORDER_UYVY;
    ResizeArgs y = a;
    y.order = kOrderY422;
    y.src = a.src + (uyvy ? 1 : 0);
    int rc = launch_color_bicubic(c, y);
    if (rc) return rc;
    const Chroma420& ch = a.ch;
    ResizeArgs u;
    u.order = kOrderUV422;
    u.src = ch.src + (uyvy ? 0 : 1); u.src_stride = ch.src_pitch;
    u.sw = ch.sw; u.sh = ch.sh; u.src_row0 = 0; u.src_row1 = ch.sh;
    u.ow = ch.ow; u.oh = ch.oh;
    u.row_begin = ch.row_begin; u.row_end = ch.row_end;
    u.pl.y = ch.dst; u.pl.cr = ch.dst + ch.dst_v; u.pl.pitch = ch.dst_pitch; u.pl.row0 = 0; u.pl.rows = ch.oh;
    u.pl.frame_stride = ch.dst_frame;
    u.tx = ch.tx; u.ty = ch.ty;
    u.nframes = a.nframes; u.src_frame_stride = a.src_frame_stride;
    return launch_color_bicubic(c, u);
}

// A grey + alpha frame (SRCNN_ORDER_GRAYA).  x2 / x4 with ow % 8 == 0: one launch for grey and alpha (color_bicubic_int.cu).
// Otherwise two launches of the generic kernels, both on every second byte of the rows (kOrderY422, as a YUY2 / UYVY Y plane):
// grey from byte 0 into pl.y / pl.y16 as a grey call's, then alpha from byte 1 into the workspace's Cr plane, for the output rows
// [r0, r1) of `ch` only (the halo rows around them are the CNN's).  (The direct kernels, for strong down-scales, go frame by frame.)
static int launch_graya(Ctx* c, const ResizeArgs& a) {
    ResizeArgs y = a;
    if (c->ka_int) {
        y.order = SRCNN_ORDER_GRAY;
        bool done = false;
        const int rc = launch_graya_int(c, resize_dev(y), a, &done);
        if (rc || done) return rc;
    }
    y.order = kOrderY422;
    int rc = launch_color_bicubic(c, y);
    if (rc) return rc;
    const Chroma420& ch = a.ch;
    ResizeArgs al;
    al.order = kOrderY422;
    al.src = ch.src + 1; al.src_stride = ch.src_pitch;
    al.sw = ch.sw; al.sh = ch.sh; al.src_row0 = 0; al.src_row1 = ch.sh;
    al.ow = ch.ow; al.oh = ch.oh;
    al.row_begin = ch.row_begin; al.row_end = ch.row_end;
    al.pl.y = ch.dst; al.pl.pitch = ch.dst_pitch; al.pl.row0 = 0; al.pl.rows = ch.oh; al.pl.frame_stride = ch.dst_frame;
    al.tx = ch.tx; al.ty = ch.ty;
    al.nframes = a.nframes; al.src_frame_stride = a.src_frame_stride;
    return launch_color_bicubic(c, al);
}

// u8 Y plane -> padded FP16 plane (Planes::y16): 8 pixels per thread; the first / last group of a row also writes the
// replicated edge columns.  Off the hot path (the tiled kernel writes FP16 itself): stage API and fallback geometries.
__global__ void __launch_bounds__(256) k_y8_to_y16(const uint8_t* __restrict__ y, size_t pitch, int w, int rows, uint8_t* __restrict__ y16,
                                                   size_t pitch16, int groups) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(gid / groups), g = (int)(gid - (long long)row * groups);
    if (row >= rows) return;
    const uint8_t* src = y + (size_t)row * pitch;
    unsigned short* dst = reinterpret_cast<unsigned short*>(y16 + (size_t)row * pitch16) + kY16Pad;
    const int x0 = g * 8;
    for (int j = 0; j < 8 && x0 + j < w; j++) dst[x0 + j] = __half_as_ushort(__ushort2half_rn((unsigned short)src[x0 + j]));
    if (g == 0) {
        const unsigned short e = __half_as_ushort(__ushort2half_rn((unsigned short)src[0]));
        for (int k = 1; k <= kY16Pad; k++) dst[-k] = e;
    }
    if (x0 <= w - 1 && w - 1 < x0 + 8) {
        const unsigned short e = __half_as_ushort(__ushort2half_rn((unsigned short)src[w - 1]));
        for (int k = 0; k < 8; k++) dst[w + k] = e;
    }
}

int launch_y8_to_y16(Ctx* c, const uint8_t* y, size_t pitch, int w, int rows, uint8_t* y16, size_t pitch16) {
    if (rows <= 0 || w <= 0) return SRCNN_OK;
    const int groups = (w + 7) / 8;
    const long long total = (long long)groups * rows;
    k_y8_to_y16<<<(unsigned)((total + 255) / 256), 256, 0, c->stream>>>(y, pitch, w, rows, y16, pitch16, groups);
    c->launches++;
    SRCNN_CUDA(c, cudaGetLastError());
    return SRCNN_OK;
}

// test hook: force the direct form (exported through the C ABI as a stage option is overkill; the
// tiled/direct agreement is covered by running geometries on both sides of the footprint limit)

// ------------------------------------------------------------------------------------------------
// K-C: merge + YCrCb -> BGR.  4 pixels per thread: three aligned 32-bit plane loads, 12 output bytes.  NC = 4 (BGRA / RGBA):
// a fourth plane `a` becomes byte 3 of every pixel, 16 output bytes.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void ycc_to_bgr(int Y, int Cr, int Cb, int& B, int& G, int& R) {
    const int cr = Cr - 128, cb = Cb - 128;
    B = clampi(Y + ((cb * 29049 + 8192) >> 14), 0, 255);
    G = clampi(Y + ((cb * -5636 + cr * -11698 + 8192) >> 14), 0, 255);
    R = clampi(Y + ((cr * 22987 + 8192) >> 14), 0, 255);
}

template <int NC>
__global__ void __launch_bounds__(256) k_merge_ycc2bgr(const uint8_t* __restrict__ y, const uint8_t* __restrict__ cr,
                                                       const uint8_t* __restrict__ cb, size_t pitch, int w, int rows,
                                                       int swapRB, uint8_t* __restrict__ dst, size_t dst_stride,
                                                       int dst_aligned, int blocks_per_row, const uint8_t* __restrict__ a) {
    // 1-D grid (rows can exceed the 65535 limit of gridDim.y): blocks_per_row blocks per image row
    const int row = blockIdx.x / blocks_per_row;
    const int q = (blockIdx.x - row * blocks_per_row) * blockDim.x + threadIdx.x;  // 4-pixel group
    const int x = q * 4;
    if (x >= w || row >= rows) return;
    const size_t o = (size_t)row * pitch + x;
    const uint32_t vy = *reinterpret_cast<const uint32_t*>(y + o);
    const uint32_t vr = *reinterpret_cast<const uint32_t*>(cr + o);
    const uint32_t vb = *reinterpret_cast<const uint32_t*>(cb + o);
    const uint32_t va = NC == 4 ? *reinterpret_cast<const uint32_t*>(a + o) : 0u;
    uint8_t px[4 * NC];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        int B, G, R;
        ycc_to_bgr((vy >> (8 * j)) & 255, (vr >> (8 * j)) & 255, (vb >> (8 * j)) & 255, B, G, R);
        px[NC * j] = (uint8_t)(swapRB ? R : B);
        px[NC * j + 1] = (uint8_t)G;
        px[NC * j + 2] = (uint8_t)(swapRB ? B : R);
        if (NC == 4) px[NC * j + 3] = (uint8_t)(va >> (8 * j));
    }
    uint8_t* d = dst + (size_t)row * dst_stride + NC * (size_t)x;
    if (dst_aligned && x + 3 < w) {
        uint32_t* d32 = reinterpret_cast<uint32_t*>(d);
#pragma unroll
        for (int k = 0; k < NC; k++)
            d32[k] = px[4 * k] | (px[4 * k + 1] << 8) | (px[4 * k + 2] << 16) | ((uint32_t)px[4 * k + 3] << 24);
    } else {
        const int n = min(4, w - x) * NC;
        for (int j = 0; j < n; j++) d[j] = px[j];
    }
}

// 16 pixels per thread: three 128-bit plane loads, three 128-bit stores (needs 16-byte aligned rows).  Arithmetic per pixel
// (bit-identical to ycc_to_bgr above): with t = Y * 2^14 + 8192, every channel is (t + chroma term) >> 14 -- adding a
// multiple of 2^14 before the shift is adding Y after it -- and each chroma term is ONE dp2a: (Cb-128, Cr-128) as a pair of
// signed bytes (x ^ 0x80) times a pair of 16-bit coefficients.  Saturation and byte packing are cvt.pack.sat.u8.s32 (two
// channels per instruction).  ~10 instructions per pixel instead of ~25; R/B order is a choice of coefficient pairs.
__device__ __forceinline__ int dp2a_lo_ss(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp2a.lo.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi_ss(uint32_t a, uint32_t b, int c) {
    int d;
    asm("dp2a.hi.s32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
// d = sat_u8(lo) | sat_u8(hi) << 8 | (upper & 0xFFFF) << 16
__device__ __forceinline__ uint32_t pack_sat_u8(int lo, int hi, uint32_t upper) {
    uint32_t d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(hi), "r"(lo), "r"(upper));
    return d;
}

// Every CTA lets the kernel's dependents go on entry (griddepcontrol.launch_dependents): once the last CTA has started, the
// colour+bicubic kernel of the NEXT whole-path call -- when api.cu launched it with programmatic stream serialisation -- fills the
// SMs' free warp slots while this kernel, which is bound by L2 / HBM and leaves the issue slots idle, is still running.  A kernel
// launched the ordinary way waits for this one to finish as always.  Threads walk the 16-pixel groups row-major with a grid stride
// (one group per thread unless the grid is capped).  NC = 4: a fourth 128-bit load of the alpha plane `a`, whose bytes join the
// colour bytes with one byte permutation per pixel, and four 128-bit stores (64 bytes per 16 pixels).
template <int NC>
__global__ void __launch_bounds__(256) k_merge_ycc2bgr_v16(const uint8_t* __restrict__ y, const uint8_t* __restrict__ cr,
                                                           const uint8_t* __restrict__ cb, size_t pitch, int w, int rows,
                                                           int swapRB, uint8_t* __restrict__ dst, size_t dst_stride,
                                                           int groups_per_row, const uint8_t* __restrict__ a) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // 16-bit coefficient pairs (low half x Cb-128, high half x Cr-128): B = 29049 cb, G = -5636 cb - 11698 cr, R = 22987 cr
    const uint32_t kB = 29049u, kG = (uint32_t)(unsigned short)(-5636) | ((uint32_t)(unsigned short)(-11698) << 16), kR = 22987u << 16;
    const uint32_t k0 = swapRB ? kR : kB, k2 = swapRB ? kB : kR;      // first and third byte of a pixel
    // (row, group) of this thread's items without a division per item: one step of the grid-stride walk is `srow` rows and `sgrp`
    // groups further, with a carry into the next row.  The next item's three 16-byte loads are in flight while this one is
    // converted and stored.
    const unsigned stride = gridDim.x * blockDim.x;
    const unsigned first = blockIdx.x * blockDim.x + threadIdx.x;
    const int srow = (int)(stride / (unsigned)groups_per_row), sgrp = (int)(stride % (unsigned)groups_per_row);
    int row = (int)(first / (unsigned)groups_per_row), grp = (int)(first % (unsigned)groups_per_row);
    if (row >= rows) return;
    uint4 vy, vr, vb, va;
    {
        const size_t o = (size_t)row * pitch + grp * 16;
        vy = *reinterpret_cast<const uint4*>(y + o);
        vr = *reinterpret_cast<const uint4*>(cr + o);
        vb = *reinterpret_cast<const uint4*>(cb + o);
        if (NC == 4) va = *reinterpret_cast<const uint4*>(a + o);
    }
    for (;;) {
        const int x = grp * 16, crow = row;
        const uint32_t wy[4] = {vy.x, vy.y, vy.z, vy.w}, wr[4] = {vr.x, vr.y, vr.z, vr.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
        uint32_t wa[4];
        if (NC == 4) { wa[0] = va.x; wa[1] = va.y; wa[2] = va.z; wa[3] = va.w; }
        row += srow; grp += sgrp;
        if (grp >= groups_per_row) { grp -= groups_per_row; row++; }
        const bool more = row < rows;
        if (more) {
            const size_t o = (size_t)row * pitch + grp * 16;
            vy = *reinterpret_cast<const uint4*>(y + o);
            vr = *reinterpret_cast<const uint4*>(cr + o);
            vb = *reinterpret_cast<const uint4*>(cb + o);
            if (NC == 4) va = *reinterpret_cast<const uint4*>(a + o);
        }
        uint32_t outw[4 * NC];
#pragma unroll
        for (int k = 0; k < 4; k++) {   // 4 pixels -> 12 bytes -> 3 words
            const uint32_t sb = wb[k] ^ 0x80808080u, sr = wr[k] ^ 0x80808080u;     // Cb-128, Cr-128 as signed bytes
            const uint32_t c01 = __byte_perm(sb, sr, 0x5140), c23 = __byte_perm(sb, sr, 0x7362);   // (cb0,cr0,cb1,cr1), (cb2,cr2,cb3,cr3)
            int v[4][3];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int t = (int)((wy[k] >> (8 * j)) & 255u) * 16384 + 8192;
                const uint32_t cc = j < 2 ? c01 : c23;
                if (j & 1) {
                    v[j][0] = dp2a_hi_ss(k0, cc, t) >> 14;
                    v[j][1] = dp2a_hi_ss(kG, cc, t) >> 14;
                    v[j][2] = dp2a_hi_ss(k2, cc, t) >> 14;
                } else {
                    v[j][0] = dp2a_lo_ss(k0, cc, t) >> 14;
                    v[j][1] = dp2a_lo_ss(kG, cc, t) >> 14;
                    v[j][2] = dp2a_lo_ss(k2, cc, t) >> 14;
                }
            }
            if (NC == 4) {
                // pixel j: c0 c1 c2 from the conversion, byte 3 = byte j of the alpha word
#pragma unroll
                for (int j = 0; j < 4; j++)
                    outw[4 * k + j] = __byte_perm(pack_sat_u8(v[j][0], v[j][1], pack_sat_u8(v[j][2], 0, 0u)), wa[k], 0x0210 | ((4 + j) << 12));
                continue;
            }
            // bytes: p0c0 p0c1 p0c2 p1c0 | p1c1 p1c2 p2c0 p2c1 | p2c2 p3c0 p3c1 p3c2
            outw[3 * k] = pack_sat_u8(v[0][0], v[0][1], pack_sat_u8(v[0][2], v[1][0], 0u));
            outw[3 * k + 1] = pack_sat_u8(v[1][1], v[1][2], pack_sat_u8(v[2][0], v[2][1], 0u));
            outw[3 * k + 2] = pack_sat_u8(v[2][2], v[3][0], pack_sat_u8(v[3][1], v[3][2], 0u));
        }
        uint8_t* d = dst + (size_t)crow * dst_stride + NC * (size_t)x;
        if (x + 15 < w) {
            uint4* d4 = reinterpret_cast<uint4*>(d);
#pragma unroll
            for (int k = 0; k < NC; k++) d4[k] = make_uint4(outw[4 * k], outw[4 * k + 1], outw[4 * k + 2], outw[4 * k + 3]);
        } else if (NC == 4) {   // a pixel is one aligned word (static indices keep outw in registers)
#pragma unroll
            for (int j = 0; j < 16; j++)
                if (x + j < w) reinterpret_cast<uint32_t*>(d)[j] = outw[j];
        } else {
            const int n = (w - x) * NC;
            for (int j = 0; j < n; j++) d[j] = (uint8_t)(outw[j >> 2] >> (8 * (j & 3)));
        }
        if (!more) break;
    }
}

// ------------------------------------------------------------------------------------------------
// K-C for packed 4:2:2 (SRCNN_ORDER_YUY2 / _UYVY): Y' and the resized U', V' planes interleaved into macropixels -- no colour
// conversion, so none of the merge's arithmetic.  16 pixels per thread: one 128-bit load of Y', 64 bits each of U' and V', four
// byte permutations for the (U V U V) words and eight for the output, two 128-bit stores (needs 16-byte aligned rows).  Releases
// its dependents on entry like k_merge_ycc2bgr_v16, so the next call's K-A may fill the SMs beside it.
// ------------------------------------------------------------------------------------------------
template <bool kUYVY>
__global__ void __launch_bounds__(256) k_pack_yuv422_v16(const uint8_t* __restrict__ y, const uint8_t* __restrict__ u,
                                                         const uint8_t* __restrict__ v, size_t pitch, int w, int rows,
                                                         uint8_t* __restrict__ dst, size_t dst_stride, int groups_per_row) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(gid / groups_per_row), x = 16 * (int)(gid - (long long)row * groups_per_row);
    if (row >= rows) return;
    const size_t o = (size_t)row * pitch;
    const uint4 vy = *reinterpret_cast<const uint4*>(y + o + x);
    const uint2 vu = *reinterpret_cast<const uint2*>(u + o + x / 2), vv = *reinterpret_cast<const uint2*>(v + o + x / 2);
    const uint32_t wy[4] = {vy.x, vy.y, vy.z, vy.w};
    // (U0 V0 U1 V1) for the first four Y, (U2 V2 U3 V3) for the next four, ...
    const uint32_t wuv[4] = {__byte_perm(vu.x, vv.x, 0x5140), __byte_perm(vu.x, vv.x, 0x7362), __byte_perm(vu.y, vv.y, 0x5140),
                             __byte_perm(vu.y, vv.y, 0x7362)};
    uint32_t out[8];
#pragma unroll
    for (int k = 0; k < 4; k++) {   // Y0 U0 Y1 V0 | Y2 U1 Y3 V1  or  U0 Y0 V0 Y1 | U1 Y2 V1 Y3
        out[2 * k] = __byte_perm(wy[k], wuv[k], kUYVY ? 0x1504 : 0x5140);
        out[2 * k + 1] = __byte_perm(wy[k], wuv[k], kUYVY ? 0x3726 : 0x7362);
    }
    uint8_t* d = dst + (size_t)row * dst_stride + 2 * (size_t)x;
    if (x + 15 < w) {
        reinterpret_cast<uint4*>(d)[0] = make_uint4(out[0], out[1], out[2], out[3]);
        reinterpret_cast<uint4*>(d)[1] = make_uint4(out[4], out[5], out[6], out[7]);
    } else {   // the row's last, partial group: one aligned word per macropixel (w is even; static indices keep out in registers)
#pragma unroll
        for (int j = 0; j < 8; j++)
            if (x + 2 * j < w) reinterpret_cast<uint32_t*>(d)[j] = out[j];
    }
}

// The same for destinations the 128-bit stores cannot take: one macropixel (two pixels) per thread, byte stores.
template <bool kUYVY>
__global__ void __launch_bounds__(256) k_pack_yuv422(const uint8_t* __restrict__ y, const uint8_t* __restrict__ u,
                                                     const uint8_t* __restrict__ v, size_t pitch, int w, int rows,
                                                     uint8_t* __restrict__ dst, size_t dst_stride) {
    const int mpr = w / 2;
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(gid / mpr), m = (int)(gid - (long long)row * mpr);
    if (row >= rows) return;
    const size_t o = (size_t)row * pitch;
    const uint8_t y0 = y[o + 2 * m], y1 = y[o + 2 * m + 1], cu = u[o + m], cv = v[o + m];
    uint8_t* d = dst + (size_t)row * dst_stride + 4 * (size_t)m;
    d[0] = kUYVY ? cu : y0;
    d[1] = kUYVY ? y0 : cu;
    d[2] = kUYVY ? cv : y1;
    d[3] = kUYVY ? y1 : cv;
}

// ------------------------------------------------------------------------------------------------
// K-C for grey + alpha (SRCNN_ORDER_GRAYA): Y' and the resized A' plane (the Cr slot) interleaved into byte pairs.  16 pixels per
// thread: one 128-bit load of each plane, eight byte permutations, two 128-bit stores (needs 16-byte aligned rows).  Releases its
// dependents on entry like k_pack_yuv422_v16.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pack_ya_v16(const uint8_t* __restrict__ y, const uint8_t* __restrict__ a, size_t pitch, int w,
                                                     int rows, uint8_t* __restrict__ dst, size_t dst_stride, int groups_per_row) {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(gid / groups_per_row), x = 16 * (int)(gid - (long long)row * groups_per_row);
    if (row >= rows) return;
    const size_t o = (size_t)row * pitch + x;
    const uint4 vy = *reinterpret_cast<const uint4*>(y + o), va = *reinterpret_cast<const uint4*>(a + o);
    const uint32_t wy[4] = {vy.x, vy.y, vy.z, vy.w}, wa[4] = {va.x, va.y, va.z, va.w};
    uint32_t out[8];
#pragma unroll
    for (int k = 0; k < 4; k++) {   // Y0 A0 Y1 A1 | Y2 A2 Y3 A3
        out[2 * k] = __byte_perm(wy[k], wa[k], 0x5140);
        out[2 * k + 1] = __byte_perm(wy[k], wa[k], 0x7362);
    }
    uint8_t* d = dst + (size_t)row * dst_stride + 2 * (size_t)x;
    if (x + 15 < w) {
        reinterpret_cast<uint4*>(d)[0] = make_uint4(out[0], out[1], out[2], out[3]);
        reinterpret_cast<uint4*>(d)[1] = make_uint4(out[4], out[5], out[6], out[7]);
    } else {   // the row's last, partial group: one aligned 16-bit store per pixel (static indices keep out in registers)
#pragma unroll
        for (int j = 0; j < 16; j++)
            if (x + j < w) reinterpret_cast<uint16_t*>(d)[j] = (uint16_t)(out[j >> 1] >> (16 * (j & 1)));
    }
}

// The same for destinations the 128-bit stores cannot take: one pixel per thread, byte stores.
__global__ void __launch_bounds__(256) k_pack_ya(const uint8_t* __restrict__ y, const uint8_t* __restrict__ a, size_t pitch, int w, int rows,
                                                 uint8_t* __restrict__ dst, size_t dst_stride) {
    const long long gid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int row = (int)(gid / w), x = (int)(gid - (long long)row * w);
    if (row >= rows) return;
    const size_t o = (size_t)row * pitch + x;
    uint8_t* d = dst + (size_t)row * dst_stride + 2 * (size_t)x;
    d[0] = y[o];
    d[1] = a[o];
}

int launch_pack(Ctx* c, const MergeArgs& a) {
    if (a.rows <= 0 || a.w <= 0) return SRCNN_OK;
    const bool ya = a.order == SRCNN_ORDER_GRAYA, uyvy = a.order == SRCNN_ORDER_UYVY;
    const bool wide = ((((uintptr_t)a.dst) | a.dst_stride | (uintptr_t)a.y | (uintptr_t)a.cr | (uintptr_t)a.cb | a.pitch) & 15) == 0 &&
                      a.pitch >= align_up((size_t)a.w, 16);
    c->merge_sel = -1;   // as for a merge: the whole-path caller says afterwards which Cr/Cb pair this launch reads
    note_merge(c);
    if (wide) {
        const int groups16 = (a.w + 15) / 16;
        const long long blocks = ((long long)groups16 * a.rows + 255) / 256;
        if (ya)
            k_pack_ya_v16<<<(unsigned)blocks, 256, 0, c->stream>>>(a.y, a.cr, a.pitch, a.w, a.rows, a.dst, a.dst_stride, groups16);
        else
            (uyvy ? k_pack_yuv422_v16<true> : k_pack_yuv422_v16<false>)<<<(unsigned)blocks, 256, 0, c->stream>>>(a.y, a.cr, a.cb, a.pitch, a.w,
                                                                                                                a.rows, a.dst, a.dst_stride, groups16);
    } else if (ya) {
        const long long blocks = ((long long)a.w * a.rows + 255) / 256;
        k_pack_ya<<<(unsigned)blocks, 256, 0, c->stream>>>(a.y, a.cr, a.pitch, a.w, a.rows, a.dst, a.dst_stride);
    } else {
        const long long blocks = ((long long)(a.w / 2) * a.rows + 255) / 256;
        (uyvy ? k_pack_yuv422<true> : k_pack_yuv422<false>)<<<(unsigned)blocks, 256, 0, c->stream>>>(a.y, a.cr, a.cb, a.pitch, a.w, a.rows,
                                                                                                    a.dst, a.dst_stride);
    }
    c->launches++;
    SRCNN_CUDA(c, cudaGetLastError());
    return SRCNN_OK;
}

int launch_merge(Ctx* c, const MergeArgs& a) {
    if (a.rows <= 0 || a.w <= 0) return SRCNN_OK;
    const bool four = four_channel(a.order), swap = a.order == SRCNN_ORDER_RGB || a.order == SRCNN_ORDER_RGBA;
    const bool wide = ((((uintptr_t)a.dst) | a.dst_stride | (uintptr_t)a.y | (uintptr_t)a.cr | (uintptr_t)a.cb | (uintptr_t)a.a | a.pitch) & 15) == 0 &&
                      a.pitch >= align_up((size_t)a.w, 16);
    c->merge_sel = -1;   // a whole-path caller says afterwards which Cr/Cb pair this launch reads (api.cu, merged_into)
    note_merge(c);
    if (wide) {
        const int groups16 = (a.w + 15) / 16;
        const long long ngroups = (long long)groups16 * a.rows;
        // one group per thread by default (a thread that walks several groups is slower: common.h, merge_ctas_per_sm); the
        // dependents are then released when the last CTA has started, roughly half-way through a 4K frame
        const long long want = (ngroups + 255) / 256, cap = c->merge_ctas_per_sm > 0 ? (long long)c->merge_ctas_per_sm * std::max(1, c->sm_count) : want;
        const long long k = (want + cap - 1) / cap;
        const int grid = (int)((want + k - 1) / k);
        (four ? k_merge_ycc2bgr_v16<4> : k_merge_ycc2bgr_v16<3>)<<<grid, 256, 0, c->stream>>>(a.y, a.cr, a.cb, a.pitch, a.w, a.rows, swap, a.dst,
                                                                                           a.dst_stride, groups16, a.a);
        c->launches++;
        SRCNN_CUDA(c, cudaGetLastError());
        return SRCNN_OK;
    }
    const int groups = (a.w + 3) / 4;
    const int bpr = (groups + 255) / 256;
    const unsigned grid = (unsigned)bpr * (unsigned)a.rows;
    const int aligned = (((uintptr_t)a.dst & 3) == 0) && ((a.dst_stride & 3) == 0);
    (four ? k_merge_ycc2bgr<4> : k_merge_ycc2bgr<3>)<<<grid, 256, 0, c->stream>>>(a.y, a.cr, a.cb, a.pitch, a.w, a.rows, swap, a.dst,
                                                                               a.dst_stride, aligned, bpr, a.a);
    c->launches++;
    SRCNN_CUDA(c, cudaGetLastError());
    return SRCNN_OK;
}

}  // namespace srcnn
