/*
 * oracle/srcnn_oracle.c -- CPU restatement of the SRCNN_Cpp inference hot path.
 *
 * THIS IS TEST INFRASTRUCTURE, NOT PRODUCT CODE.  Only tests/, __graft_entry__.smoke() and the
 * cpu_baseline / --impl reference legs of bench.py may load this library, and only as the checker.
 * The product (srcnn_cpp_b200/csrc, libsrcnn_b200.so) never links, loads or calls anything here and
 * has no CPU fallback.
 *
 * What it restates (reference file:line are into /root/reference):
 *   orc_bgr2ycrcb   cv::cvtColor(BGR->YCrCb) call at src/srcnn.cpp:509       (OpenCV 8U fixed point)
 *   orc_resize_cubic cv::resize(..., INTER_CUBIC) call at src/srcnn.cpp:577-582 (OpenCV 8U, native path)
 *   orc_conv99x11   Convolution99x11, src/srcnn.cpp:254-325 (+ IntTrim :77-81)
 *   orc_conv55      Convolution55,    src/srcnn.cpp:189-243
 *   orc_ycrcb2bgr   cv::cvtColor(YCrCb->BGR) call at src/srcnn.cpp:657
 *   orc_pipeline    the timed region of pthreadcall, src/srcnn.cpp:505-659
 *   orc_cnn_at      orc_cnn at listed pixels, exactly or with one near miss of its arithmetic (tests only)
 *
 * The OpenCV arithmetic lives in a third-party dependency that is NOT vendored in the reference
 * (Makefile:8-9, pkg-config opencv4, no version pin).  It is restated from OpenCV's published
 * algorithm (imgproc color_yuv / resize, INTER_RESIZE_COEF_BITS = 11, cubic A = -0.75) and PINNED
 * against (a) python cv2 4.13.0 with IPP disabled, stage by stage, and (b) the reference's only
 * golden vector Pictures/butterfly.png -> Pictures/butterfly-srcnn.png at --scale=1.5, which the
 * whole chain reproduces byte for byte (tests/test_oracle.py).  The conv functions are additionally
 * pinned against the reference's own unmodified srcnn.cpp compiled into oracle/_ref/libref.so.
 *
 * Build: see oracle/Makefile.  Must be compiled WITHOUT -ffast-math and WITHOUT FMA contraction
 * (-ffp-contract=off, no -march=native): the reference objects are plain x86-64 SSE2 code.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_API __attribute__((visibility("default")))

/* ---- weights blob layout (srcnn_cpp_b200/data/srcnn_weights.bin, tools/pack_weights.cpp) ---- */
enum {
    ORC_W1 = 0,                    /* [64][9][9]  convdata.h:32-674  */
    ORC_B1 = ORC_W1 + 64 * 81,     /* [64]        convdata.h:19-29   */
    ORC_W2 = ORC_B1 + 64,          /* [32][64]    convdata.h:686-976 */
    ORC_B2 = ORC_W2 + 32 * 64,     /* [32]        convdata.h:677-683 */
    ORC_W3 = ORC_B2 + 32,          /* [32][5][5]  convdata.h:982-1176 */
    ORC_B3 = ORC_W3 + 32 * 25,     /* scalar      convdata.h:979     */
    ORC_NPARAM = ORC_B3 + 1        /* 8129 */
};

ORC_API int orc_num_params(void) { return ORC_NPARAM; }

ORC_API int orc_max_threads(void) {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* IntTrim(a,b,c): clamp c into [a,b]  (src/srcnn.cpp:77-81) */
static inline int int_trim(int a, int b, int c) { return c <= a ? a : (c <= b ? c : b); }

static inline uint8_t sat_u8(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

/* ------------------------------------------------------------------------------------------------
 * cv::cvtColor 8U, BT.601 full range, 14-bit fixed point (OpenCV imgproc/color_yuv, yuv_shift = 14,
 * coefficients B2Y 1868, G2Y 9617, R2Y 4899, YCrI 11682, YCbI 9241; inverse 22987, -11698, -5636,
 * 29049).  Memory order B,G,R <-> Y,Cr,Cb.  call sites src/srcnn.cpp:509 and :657.
 * ---------------------------------------------------------------------------------------------- */
ORC_API void orc_bgr2ycrcb(const uint8_t* bgr, size_t stride, int w, int h, uint8_t* ycc, size_t ostride) {
    for (int y = 0; y < h; y++) {
        const uint8_t* s = bgr + (size_t)y * stride;
        uint8_t* d = ycc + (size_t)y * ostride;
        for (int x = 0; x < w; x++) {
            int B = s[3 * x], G = s[3 * x + 1], R = s[3 * x + 2];
            int Y = (1868 * B + 9617 * G + 4899 * R + 8192) >> 14;
            int Cr = ((R - Y) * 11682 + (128 << 14) + 8192) >> 14;
            int Cb = ((B - Y) * 9241 + (128 << 14) + 8192) >> 14;
            d[3 * x] = sat_u8(Y);
            d[3 * x + 1] = sat_u8(Cr);
            d[3 * x + 2] = sat_u8(Cb);
        }
    }
}

ORC_API void orc_ycrcb2bgr(const uint8_t* ycc, size_t stride, int w, int h, uint8_t* bgr, size_t ostride) {
    for (int y = 0; y < h; y++) {
        const uint8_t* s = ycc + (size_t)y * stride;
        uint8_t* d = bgr + (size_t)y * ostride;
        for (int x = 0; x < w; x++) {
            int Y = s[3 * x], cr = s[3 * x + 1] - 128, cb = s[3 * x + 2] - 128;
            int b = Y + ((cb * 29049 + 8192) >> 14);
            int g = Y + ((cb * -5636 + cr * -11698 + 8192) >> 14);
            int r = Y + ((cr * 22987 + 8192) >> 14);
            d[3 * x] = sat_u8(b);
            d[3 * x + 1] = sat_u8(g);
            d[3 * x + 2] = sat_u8(r);
        }
    }
}

/* split / merge (src/srcnn.cpp:540, :639): HWC <-> planes */
ORC_API void orc_split3(const uint8_t* hwc, size_t stride, int w, int h, uint8_t* p0, uint8_t* p1, uint8_t* p2) {
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            const uint8_t* s = hwc + (size_t)y * stride + 3 * (size_t)x;
            size_t o = (size_t)y * w + x;
            p0[o] = s[0]; p1[o] = s[1]; p2[o] = s[2];
        }
}

ORC_API void orc_merge3(const uint8_t* p0, const uint8_t* p1, const uint8_t* p2, int w, int h, uint8_t* hwc, size_t stride) {
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) {
            uint8_t* d = hwc + (size_t)y * stride + 3 * (size_t)x;
            size_t o = (size_t)y * w + x;
            d[0] = p0[o]; d[1] = p1[o]; d[2] = p2[o];
        }
}

/* ------------------------------------------------------------------------------------------------
 * cv::resize INTER_CUBIC, CV_8U, one channel (call site src/srcnn.cpp:570-583).
 * Published algorithm (OpenCV imgproc/resize.cpp, resizeGeneric_ + HResizeCubic<uchar,int,short> +
 * VResizeCubic<uchar,int,short,FixedPtCast<..,22>, VResizeCubicVec_32s8u>):
 *   src coord  f = (float)((d + 0.5) * (1.0 / ((double)dst / src)) - 0.5),  s = floor(f), x = f - s
 *   coefficients: Keys cubic A = -0.75 in float32, then short = round-half-even(c * 2048)
 *   taps s-1..s+2, replicate border
 *   horizontal pass -> int32;  vertical pass:
 *     columns below (dw/8)*8 : float, v = H0*b0 + (H1*b1 + (H2*b2 + H3*b3)), b_k = coef_k * 2^-22,
 *                              separate mul/add, round-half-even, saturate        (8-lane SIMD body)
 *     remaining tail columns : integer (sum + 2^21) >> 22, saturate                 (scalar tail)
 * ---------------------------------------------------------------------------------------------- */
ORC_API int orc_scaled_dim(int n, float scale) {
    /* `newsz.width *= image_multiply` on an int: int -> float multiply -> truncating int (srcnn.cpp:573-575) */
    return (int)((float)n * scale);
}

/* tap table for one axis: ofs[d] = floor(src coord); coef[4*d..] = 11-bit fixed-point taps */
ORC_API void orc_cubic_taps(int src, int dst, int* ofs, int16_t* coef) {
    const float A = -0.75f;
    double inv = (double)dst / (double)src;
    double sc = 1.0 / inv;
    for (int d = 0; d < dst; d++) {
        float f = (float)((d + 0.5) * sc - 0.5);
        int s = (int)floorf(f);
        float x = f - (float)s;
        float c0, c1, c2, c3; /* float32 every step: build flags forbid contraction/x87 */
        float x1 = x + 1.f;
        c0 = ((A * x1 - 5 * A) * x1 + 8 * A) * x1 - 4 * A;
        c1 = ((A + 2) * x - (A + 3)) * x * x + 1;
        float y = 1.f - x;
        c2 = ((A + 2) * y - (A + 3)) * y * y + 1;
        c3 = 1.f - c0 - c1 - c2;
        float c[4] = {c0, c1, c2, c3};
        ofs[d] = s;
        for (int k = 0; k < 4; k++) {
            long r = lrintf(c[k] * 2048.f); /* default FP env: round-half-even, like cvRound */
            if (r > 32767) r = 32767;
            if (r < -32768) r = -32768;
            coef[4 * d + k] = (int16_t)r;
        }
    }
}

ORC_API void orc_resize_cubic(const uint8_t* src, size_t stride, int sw, int sh, uint8_t* dst, size_t ostride, int dw, int dh) {
    int* xofs = (int*)malloc(sizeof(int) * (size_t)dw);
    int* yofs = (int*)malloc(sizeof(int) * (size_t)dh);
    int16_t* xc = (int16_t*)malloc(sizeof(int16_t) * 4 * (size_t)dw);
    int16_t* yc = (int16_t*)malloc(sizeof(int16_t) * 4 * (size_t)dh);
    orc_cubic_taps(sw, dw, xofs, xc);
    orc_cubic_taps(sh, dh, yofs, yc);
    /* horizontal pass of every source row (int32) */
    int32_t* hbuf = (int32_t*)malloc(sizeof(int32_t) * (size_t)sh * (size_t)dw);
#pragma omp parallel for schedule(static)
    for (int y = 0; y < sh; y++) {
        const uint8_t* s = src + (size_t)y * stride;
        int32_t* hrow = hbuf + (size_t)y * dw;
        for (int dx = 0; dx < dw; dx++) {
            int32_t acc = 0;
            for (int k = 0; k < 4; k++) {
                int sx = int_trim(0, sw - 1, xofs[dx] - 1 + k);
                acc += (int32_t)s[sx] * xc[4 * dx + k];
            }
            hrow[dx] = acc;
        }
    }
    const int simd_w = (dw / 8) * 8;
    const float inv22 = 1.0f / 4194304.0f;
#pragma omp parallel for schedule(static)
    for (int dy = 0; dy < dh; dy++) {
        const int32_t* S[4];
        for (int k = 0; k < 4; k++) S[k] = hbuf + (size_t)int_trim(0, sh - 1, yofs[dy] - 1 + k) * dw;
        const int16_t* b = yc + 4 * dy;
        float b0 = (float)b[0] * inv22, b1 = (float)b[1] * inv22, b2 = (float)b[2] * inv22, b3 = (float)b[3] * inv22;
        uint8_t* d = dst + (size_t)dy * ostride;
        for (int dx = 0; dx < simd_w; dx++) {
            float t3 = (float)S[3][dx] * b3;
            float t2 = (float)S[2][dx] * b2;
            float a2 = t2 + t3;
            float t1 = (float)S[1][dx] * b1;
            float a1 = t1 + a2;
            float t0 = (float)S[0][dx] * b0;
            float a0 = t0 + a1;
            d[dx] = sat_u8((int)lrintf(a0));
        }
        for (int dx = simd_w; dx < dw; dx++) {
            int32_t v = S[0][dx] * b[0] + S[1][dx] * b[1] + S[2][dx] * b[2] + S[3][dx] * b[3];
            d[dx] = sat_u8((v + (1 << 21)) >> 22);
        }
    }
    free(hbuf); free(xofs); free(yofs); free(xc); free(yc);
}

/* ------------------------------------------------------------------------------------------------
 * Convolution99x11 (src/srcnn.cpp:254-325): conv1 9x9 1->64 + b1 + ReLU, conv2 1x1 64->32 + b2 +
 * ReLU, fused per pixel.  float32, strictly sequential accumulation in (i,j) then k order, product
 * float * (float)(int)uint8, bias added after the sum (:301, :316).  dst: 32 planes of h*w float
 * (plane k at dst + k*h*w), like the reference's vector<Mat> of CV_32F planes (:602-607).
 * ---------------------------------------------------------------------------------------------- */
ORC_API void orc_conv99x11(const float* params, const uint8_t* y, int w, int h, float* dst) {
    const float* w1 = params + ORC_W1;
    const float* b1 = params + ORC_B1;
    const float* w2 = params + ORC_W2;
    const float* b2 = params + ORC_B2;
    int* rowf = (int*)malloc(sizeof(int) * ((size_t)h + 8));
    int* colf = (int*)malloc(sizeof(int) * ((size_t)w + 8));
    for (int r = 0; r < h + 8; r++) rowf[r] = int_trim(0, h - 1, r - 4); /* :271-274 */
    for (int c = 0; c < w + 8; c++) colf[c] = int_trim(0, w - 1, c - 4); /* :277-280 */
    const size_t plane = (size_t)w * h;
#pragma omp parallel for schedule(static)
    for (int row = 0; row < h; row++) {
        for (int col = 0; col < w; col++) {
            float temp[64];
            for (int k = 0; k < 64; k++) {
                float acc = 0.0f; /* one float32 rounding per product and per add (no FMA: see Makefile) */
                for (int i = 0; i < 9; i++)
                    for (int j = 0; j < 9; j++) {
                        float p = w1[(k * 9 + i) * 9 + j] * (float)(int)y[(size_t)rowf[row + i] * w + colf[col + j]];
                        acc = acc + p; /* :297 */
                    }
                acc = acc + b1[k];                 /* :301 */
                temp[k] = (acc < 0) ? 0 : acc;     /* :304 */
            }
            for (int k = 0; k < 32; k++) {
                float res = 0.0f;
                for (int i = 0; i < 64; i++) {
                    float p = temp[i] * w2[k * 64 + i];
                    res = res + p;                 /* :314 */
                }
                res = res + b2[k];                 /* :316 */
                dst[k * plane + (size_t)row * w + col] = (res < 0) ? 0 : res; /* :319-321 */
            }
        }
    }
    free(rowf); free(colf);
}

/* ------------------------------------------------------------------------------------------------
 * Convolution55 (src/srcnn.cpp:189-243): conv3 5x5 32->1.  Products float32*float32 -> float32,
 * inner 25-term sum in double (:222-230), `temp += temppixel` = (float)((double)temp + temppixel)
 * (:232), + bias in float (:235), IntTrim(0,255,temp) with the implicit float->int TRUNCATION (:238),
 * store u8 (:240).
 * ---------------------------------------------------------------------------------------------- */
ORC_API void orc_conv55(const float* params, const float* src, int w, int h, uint8_t* dst) {
    const float* w3 = params + ORC_W3;
    const float b3 = params[ORC_B3];
    int* rowf = (int*)malloc(sizeof(int) * ((size_t)h + 4));
    int* colf = (int*)malloc(sizeof(int) * ((size_t)w + 4));
    for (int r = 0; r < h + 4; r++) rowf[r] = int_trim(0, h - 1, r - 2); /* :201-204 */
    for (int c = 0; c < w + 4; c++) colf[c] = int_trim(0, w - 1, c - 2); /* :207-210 */
    const size_t plane = (size_t)w * h;
#pragma omp parallel for schedule(static)
    for (int row = 0; row < h; row++) {
        for (int col = 0; col < w; col++) {
            float temp = 0;
            for (int i = 0; i < 32; i++) {
                double temppixel = 0;
                for (int m = 0; m < 5; m++)
                    for (int n = 0; n < 5; n++) {
                        float p = w3[(i * 5 + m) * 5 + n] * src[i * plane + (size_t)rowf[row + m] * w + colf[col + n]];
                        temppixel = temppixel + (double)p; /* :227-228 */
                    }
                temp = (float)((double)temp + temppixel);   /* :232 */
            }
            temp = temp + b3;                               /* :235 */
            int t = int_trim(0, 255, (int)temp);            /* :238 (float -> int truncates toward zero) */
            dst[(size_t)row * w + col] = (uint8_t)t;        /* :240 */
        }
    }
    free(rowf); free(colf);
}

/* Y plane -> CNN -> Y' plane (the calls at src/srcnn.cpp:609 and :627).  act2 may be NULL. */
ORC_API int orc_cnn(const float* params, const uint8_t* y, int w, int h, uint8_t* out, float* act2) {
    float* tmp = act2;
    if (!tmp) {
        tmp = (float*)malloc(sizeof(float) * 32 * (size_t)w * h);
        if (!tmp) return -1;
    }
    orc_conv99x11(params, y, w, h, tmp);
    orc_conv55(params, tmp, w, h, out);
    if (!act2) free(tmp);
    return 0;
}

/* ------------------------------------------------------------------------------------------------
 * The CNN at listed pixels only, exactly (mode 0) or with one near miss of its arithmetic (modes 1-12).
 * Mode 0 is orc_conv99x11 + orc_conv55 restricted to the pixels asked for: the same clamped 13x13 field,
 * the same roundings in the same order.  The near misses are what a kernel that claims bit-identity
 * could plausibly do instead; tests/test_fp32_cnn_witnesses.py builds planes on which they show.
 * fma / fmaf round once (C99 7.12.13.1); nothing else here contracts (SAFE_FP in the Makefile).
 * ---------------------------------------------------------------------------------------------- */
enum {
    ORC_AT_EXACT = 0,
    ORC_AT_TEMP_DOUBLE = 1,        /* M1 conv3: `temp` accumulated in double, one float rounding at the end */
    ORC_AT_INNER_FLOAT = 2,        /* M2 conv3: the inner 25-term sum in float */
    ORC_AT_EXACT_PRODUCTS = 3,     /* M3 conv3: products formed exactly in double (no float rounding) */
    ORC_AT_CHANNELS_REVERSED = 4,  /* M4 conv3: channels summed 31 .. 0 */
    ORC_AT_FMA_DOUBLE = 5,         /* M5 conv3: fma(w, a, tp) into the double sum */
    ORC_AT_TAPS_NM = 6,            /* conv3: (n,m) tap order instead of (m,n) */
    ORC_AT_B3_DOUBLE = 7,          /* conv3: b3 added in double, then rounded to float */
    ORC_AT_CONV1_FMA = 8,          /* conv1: acc = fmaf(w, y, acc) */
    ORC_AT_CONV1_BIAS_FIRST = 9,   /* conv1: accumulator starts at b1 instead of adding it last */
    ORC_AT_CONV1_JI = 10,          /* conv1: (j,i) tap order */
    ORC_AT_CONV2_FMA = 11,         /* conv2: res = fmaf(act1, w, res) */
    ORC_AT_CONV2_REVERSED = 12,    /* conv2: inputs summed 63 .. 0 */
    ORC_AT_NMODES = 13
};

ORC_API int orc_at_modes(void) { return ORC_AT_NMODES; }

/* conv1 + ReLU + conv2 + ReLU at image pixel (row, col) (src/srcnn.cpp:283-321), modes 0 and 8-12 */
static void act2_px(const float* params, const uint8_t* y, int w, int h, int row, int col, int mode, float out[32]) {
    const float* w1 = params + ORC_W1;
    const float* b1 = params + ORC_B1;
    const float* w2 = params + ORC_W2;
    const float* b2 = params + ORC_B2;
    float temp[64];
    for (int k = 0; k < 64; k++) {
        float acc = mode == ORC_AT_CONV1_BIAS_FIRST ? b1[k] : 0.0f;
        for (int a = 0; a < 9; a++)
            for (int b = 0; b < 9; b++) {
                const int i = mode == ORC_AT_CONV1_JI ? b : a, j = mode == ORC_AT_CONV1_JI ? a : b;
                const float wv = w1[(k * 9 + i) * 9 + j];
                const float x = (float)(int)y[(size_t)int_trim(0, h - 1, row + i - 4) * w + int_trim(0, w - 1, col + j - 4)];
                if (mode == ORC_AT_CONV1_FMA) acc = fmaf(wv, x, acc);
                else { float p = wv * x; acc = acc + p; }
            }
        if (mode != ORC_AT_CONV1_BIAS_FIRST) acc = acc + b1[k];
        temp[k] = (acc < 0) ? 0 : acc;
    }
    for (int k = 0; k < 32; k++) {
        float res = 0.0f;
        for (int t = 0; t < 64; t++) {
            const int i = mode == ORC_AT_CONV2_REVERSED ? 63 - t : t;
            if (mode == ORC_AT_CONV2_FMA) res = fmaf(temp[i], w2[k * 64 + i], res);
            else { float p = temp[i] * w2[k * 64 + i]; res = res + p; }
        }
        res = res + b2[k];
        out[k] = (res < 0) ? 0 : res;
    }
}

/* conv3 at (row, col) over the 25 clamped act2 positions (src/srcnn.cpp:213-240), modes 0-7; returns temp + b3 */
static float conv55_px(const float* params, const float a2[25][32], int mode) {
    const float* w3 = params + ORC_W3;
    const float b3 = params[ORC_B3];
    float temp = 0;
    double td = 0;
    for (int t = 0; t < 32; t++) {
        const int i = mode == ORC_AT_CHANNELS_REVERSED ? 31 - t : t;
        double tp = 0;
        float tf = 0;
        for (int a = 0; a < 5; a++)
            for (int b = 0; b < 5; b++) {
                const int m = mode == ORC_AT_TAPS_NM ? b : a, n = mode == ORC_AT_TAPS_NM ? a : b;
                const float wv = w3[(i * 5 + m) * 5 + n], sv = a2[m * 5 + n][i];
                if (mode == ORC_AT_INNER_FLOAT) { float p = wv * sv; tf = tf + p; }
                else if (mode == ORC_AT_EXACT_PRODUCTS) tp = tp + (double)wv * (double)sv;
                else if (mode == ORC_AT_FMA_DOUBLE) tp = fma((double)wv, (double)sv, tp);
                else { float p = wv * sv; tp = tp + (double)p; }
            }
        if (mode == ORC_AT_INNER_FLOAT) tp = (double)tf;
        if (mode == ORC_AT_TEMP_DOUBLE) td = td + tp;
        else temp = (float)((double)temp + tp);
    }
    if (mode == ORC_AT_TEMP_DOUBLE) temp = (float)td;
    return mode == ORC_AT_B3_DOUBLE ? (float)((double)temp + (double)b3) : temp + b3;
}

/* pixels (rows[p], cols[p]), p < n: out_v[p] = temp + b3 (float, before truncation), out_byte[p] = the byte.
 * Returns -1 for a bad mode or a pixel outside the plane. */
ORC_API int orc_cnn_at(const float* params, const uint8_t* y, int w, int h, const int* rows, const int* cols, int n,
                       int mode, float* out_v, uint8_t* out_byte) {
    if (mode < 0 || mode >= ORC_AT_NMODES) return -1;
    for (int p = 0; p < n; p++)
        if (rows[p] < 0 || rows[p] >= h || cols[p] < 0 || cols[p] >= w) return -1;
    const int mode12 = mode >= ORC_AT_CONV1_FMA ? mode : ORC_AT_EXACT;
    const int mode3 = mode >= ORC_AT_CONV1_FMA ? ORC_AT_EXACT : mode;
#pragma omp parallel for schedule(dynamic, 16)
    for (int p = 0; p < n; p++) {
        float a2[25][32];
        for (int m = 0; m < 5; m++)
            for (int q = 0; q < 5; q++)
                act2_px(params, y, w, h, int_trim(0, h - 1, rows[p] + m - 2), int_trim(0, w - 1, cols[p] + q - 2), mode12,
                        a2[m * 5 + q]);
        const float v = conv55_px(params, (const float(*)[32])a2, mode3);
        if (out_v) out_v[p] = v;
        if (out_byte) out_byte[p] = (uint8_t)int_trim(0, 255, (int)v);
    }
    return 0;
}

/* conv2's 32 activations at the listed pixels (out: [n][32]), exactly (mode 0) or under a conv1 / conv2 near miss (8-12) */
ORC_API int orc_act2_at(const float* params, const uint8_t* y, int w, int h, const int* rows, const int* cols, int n,
                        int mode, float* out) {
    if (mode != ORC_AT_EXACT && (mode < ORC_AT_CONV1_FMA || mode >= ORC_AT_NMODES)) return -1;
    for (int p = 0; p < n; p++)
        if (rows[p] < 0 || rows[p] >= h || cols[p] < 0 || cols[p] >= w) return -1;
#pragma omp parallel for schedule(static)
    for (int p = 0; p < n; p++) act2_px(params, y, w, h, rows[p], cols[p], mode, out + (size_t)p * 32);
    return 0;
}

/* ------------------------------------------------------------------------------------------------
 * The whole timed region of pthreadcall (src/srcnn.cpp:505-659): BGR8 HWC in, BGR8 HWC out.
 * Optional stage taps (any may be NULL): up_y/up_cr/up_cb = the three bicubic planes (pImg[0..2]),
 * cnn_y = Convolution55's output plane.  Returns 0, or -1 for a bad ratio (src/srcnn.cpp:485-495).
 * ---------------------------------------------------------------------------------------------- */
ORC_API int orc_pipeline(const float* params, const uint8_t* bgr, size_t stride, int w, int h, float scale,
                         uint8_t* out, size_t ostride, uint8_t* up_y, uint8_t* up_cr, uint8_t* up_cb, uint8_t* cnn_y) {
    if (((float)w * scale) <= 0.f || ((float)h * scale) <= 0.f) return -1;
    const int ow = orc_scaled_dim(w, scale), oh = orc_scaled_dim(h, scale);
    if (ow <= 0 || oh <= 0) return -1;
    const size_t sn = (size_t)w * h, dn = (size_t)ow * oh;
    uint8_t* ycc = (uint8_t*)malloc(3 * sn);
    uint8_t* sp = (uint8_t*)malloc(3 * sn);
    uint8_t* dp = (uint8_t*)malloc(4 * dn);
    uint8_t* merged = (uint8_t*)malloc(3 * dn);
    orc_bgr2ycrcb(bgr, stride, w, h, ycc, 3 * (size_t)w);               /* :509 */
    orc_split3(ycc, 3 * (size_t)w, w, h, sp, sp + sn, sp + 2 * sn);     /* :540 */
    for (int i = 0; i < 3; i++)                                         /* :570-583 */
        orc_resize_cubic(sp + i * sn, (size_t)w, w, h, dp + i * dn, (size_t)ow, ow, oh);
    int rc = orc_cnn(params, dp, ow, oh, dp + 3 * dn, NULL);            /* :609, :627 */
    if (rc == 0) {
        orc_merge3(dp + 3 * dn, dp + dn, dp + 2 * dn, ow, oh, merged, 3 * (size_t)ow); /* :638-639 */
        orc_ycrcb2bgr(merged, 3 * (size_t)ow, ow, oh, out, ostride);    /* :657 */
        if (up_y) memcpy(up_y, dp, dn);
        if (up_cr) memcpy(up_cr, dp + dn, dn);
        if (up_cb) memcpy(up_cb, dp + 2 * dn, dn);
        if (cnn_y) memcpy(cnn_y, dp + 3 * dn, dn);
    }
    free(ycc); free(sp); free(dp); free(merged);
    return rc;
}
