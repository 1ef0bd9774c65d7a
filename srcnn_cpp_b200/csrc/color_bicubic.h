// color_bicubic.h -- device helpers and the launch parameters shared by the colour+bicubic kernels
// (color_bicubic.cu: generic scales; color_bicubic_int.cu: integer up-scales x2 / x4).  Internal, not part of the C ABI.
#pragma once
#include <cuda_fp16.h>

#include "common.h"

namespace srcnn {

// ------------------------------------------------------------------------------------------------
// Device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int clampi(int v, int lo, int hi) { return min(max(v, lo), hi); }

// BGR -> Y,Cr,Cb  (OpenCV RGB2YCrCb_i<uchar>: yuv_shift 14)
__device__ __forceinline__ void bgr_to_ycc(int B, int G, int R, int& Y, int& Cr, int& Cb) {
    Y = (1868 * B + 9617 * G + 4899 * R + 8192) >> 14;
    Cr = clampi(((R - Y) * 11682 + (128 << 14) + 8192) >> 14, 0, 255);
    Cb = clampi(((B - Y) * 9241 + (128 << 14) + 8192) >> 14, 0, 255);
}

// Vertical cubic pass on four horizontal sums.  `fpath`: column belongs to cv::resize's 8-lane float
// body (dx < (ow/8)*8), else to its integer scalar tail.
__device__ __forceinline__ int vertical_tap(int h0, int h1, int h2, int h3, short4 c, bool fpath) {
    int r;
    if (fpath) {
        const float s = 1.0f / 4194304.0f;  // 2^-22, exact
        const float b0 = __fmul_rn((float)c.x, s), b1 = __fmul_rn((float)c.y, s);
        const float b2 = __fmul_rn((float)c.z, s), b3 = __fmul_rn((float)c.w, s);
        float v = __fmul_rn((float)h3, b3);
        v = __fadd_rn(__fmul_rn((float)h2, b2), v);
        v = __fadd_rn(__fmul_rn((float)h1, b1), v);
        v = __fadd_rn(__fmul_rn((float)h0, b0), v);
        r = __float2int_rn(v);
    } else {
        r = (h0 * (int)c.x + h1 * (int)c.y + h2 * (int)c.z + h3 * (int)c.w + (1 << 21)) >> 22;
    }
    return clampi(r, 0, 255);
}

struct ResizeDev {
    const uint8_t* src;
    size_t src_stride;
    int sw, sh, src_row0;
    int swapRB;
    int ow, oh;
    int row_begin, row_end;
    uint8_t* y;
    uint8_t* cr;
    uint8_t* cb;
    size_t pitch;
    uint8_t* y16;      // tiled kernel: when set, Y goes to the padded FP16 plane (Planes::y16) INSTEAD of the u8 plane
    size_t pitch16;
    // a batch of same-sized frames in one launch (blockIdx.z = frame): byte distance between consecutive frames
    size_t src_frame, plane_frame, y16_frame;
    int plane_row0;
    const int* xofs;
    const short4* xcoef;
    const int* yofs;
    const short4* ycoef;
    int simd_w;
    unsigned long long negzero2;   // the pair (-0.0f, -0.0f), opaque to the compiler (see f2_mul_rn)
    int quad_ok;   // every aligned group of 4 output columns spans <= 4 source columns (true for any up-scale)
};

// round-half-even + saturate to 0..255 in one instruction (what v_round + v_pack_u do in cv::resize)
__device__ __forceinline__ uint32_t sat_u8_rn(float v) {
    uint32_t r;
    asm("cvt.rni.sat.u8.f32 %0, %1;" : "=r"(r) : "f"(v));
    return r;
}

// Packed FP32 pairs (sm_100 FMUL2 / FADD2 / FFMA2: two IEEE single-precision operations per issue slot).  The vertical pass
// needs every product and every sum rounded on its own (cv::resize's SIMD body has no FMA), and ptxas contracts a
// mul.rn.f32x2 feeding an add.rn.f32x2 into FFMA2 even though both carry an explicit rounding mode.  So a product is written
// as fma(a, b, -0.0) -- exactly round(a*b), signed zeros included -- with the -0.0 pair coming from a kernel parameter the
// compiler cannot see through; an FFMA2 feeding an FADD2 cannot be contracted any further.
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(unsigned long long v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ unsigned long long f2_mul_rn(unsigned long long a, unsigned long long b, unsigned long long negzero) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(negzero));
    return r;
}
__device__ __forceinline__ unsigned long long f2_add_rn(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
// the vertical pass on a pair of columns: H0*b0 + (H1*b1 + (H2*b2 + H3*b3)), every product and sum rounded on its own
__device__ __forceinline__ unsigned long long f2_vtap(unsigned long long h0, unsigned long long h1, unsigned long long h2, unsigned long long h3,
                                                      unsigned long long b0, unsigned long long b1, unsigned long long b2, unsigned long long b3,
                                                      unsigned long long negzero) {
    unsigned long long v = f2_mul_rn(h3, b3, negzero);
    v = f2_add_rn(f2_mul_rn(h2, b2, negzero), v);
    v = f2_add_rn(f2_mul_rn(h1, b1, negzero), v);
    return f2_add_rn(f2_mul_rn(h0, b0, negzero), v);
}

// two u8 values (the low bytes of `lo` and `hi`) -> an FP16 pair, exactly: 0x6400 | v is 1024 + v, minus 1024
__device__ __forceinline__ uint32_t u8x2_to_h2(uint32_t lo, uint32_t hi) {
    uint32_t u = __byte_perm(lo, hi, 0x5410) | 0x64006400u;
    const __half2 h = __hsub2(*reinterpret_cast<__half2*>(&u), __float2half2_rn(1024.f));
    return *reinterpret_cast<const uint32_t*>(&h);
}

// A walk down `nit` output-row groups with a window of four rows of horizontal sums in registers: hsum(r, h) fills h with the sums
// of footprint row r, emit(h0, h1, h2, h3) produces the output rows of one window.  The window rotates by unrolling, not by
// register moves.
template <typename H, typename HSum, typename Emit>
__device__ __forceinline__ void walk_window(int nit, HSum&& hsum, Emit&& emit) {
    H hA, hB, hC, hD;
    hsum(0, hA);
    hsum(1, hB);
    hsum(2, hC);
    for (int tt = 0; tt < nit; tt += 4) {
        hsum(tt + 3, hD);
        emit(hA, hB, hC, hD);
        if (tt + 1 >= nit) break;
        hsum(tt + 4, hA);
        emit(hB, hC, hD, hA);
        if (tt + 2 >= nit) break;
        hsum(tt + 5, hB);
        emit(hC, hD, hA, hB);
        if (tt + 3 >= nit) break;
        hsum(tt + 6, hC);
        emit(hD, hA, hB, hC);
    }
}


// integer up-scales (color_bicubic_int.cu); returns SRCNN_OK with *done = false when the geometry is not eligible
int launch_color_bicubic_int(Ctx* c, const ResizeDev& p, const ResizeArgs& a, bool* done);
// the same for a 4:2:0 or packed 4:2:2 frame (a.order NV12 / I420 / YUY2 / UYVY; p describes its Y plane as a grey call's, a.ch
// its chroma): luma and chroma in one launch
int launch_yuv_int(Ctx* c, const ResizeDev& p, const ResizeArgs& a, bool* done);
// the same for a grey + alpha frame (a.order SRCNN_ORDER_GRAYA; p describes its grey plane as a grey call's, a.ch its alpha plane)
int launch_graya_int(Ctx* c, const ResizeDev& p, const ResizeArgs& a, bool* done);

}  // namespace srcnn
