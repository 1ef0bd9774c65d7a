// srcnn_fp32.cu -- K-B-fp32: the strict FP32 CUDA-core validation variant of the SRCNN stage.
//
// Same arithmetic, in the same order, as the reference's CPU code, so the result is bit-identical:
//   k_conv99x11_strict  = Convolution99x11, src/srcnn.cpp:254-325: per pixel 64 x (81 float32
//       multiply, then float32 add, sequential (i,j) order, product float * (float)(int)uint8),
//       + bias, ReLU; then 32 x (64 multiply/add in i order) + bias, ReLU.  __fmul_rn/__fadd_rn keep
//       every rounding step (the reference objects are -O0 x86-64: no FMA).
//   k_conv55_strict     = Convolution55, src/srcnn.cpp:189-243: float32 products, inner 25-term sum
//       in double, `temp += temppixel` as (float)((double)temp + temppixel), + bias, (int) truncation,
//       clamp 0..255.
// Border handling = the reference's two clamps (IntTrim, src/srcnn.cpp:77-81): conv1 reads
// Y[clamp(r+i-4)][clamp(c+j-4)], conv3 reads act2[clamp(r+m-2)][clamp(c+n-2)].
//
// This variant is the parity yardstick for the tcgen05 kernel; it is CUDA-core bound (~14.5 k
// non-fused FP32 ops per pixel) and materialises conv2's activations (128 B/px) in HBM in row chunks.
#include <mutex>

#include "common.h"

namespace srcnn {

__constant__ float c_params[kNumParams];

__device__ __forceinline__ int clampi32(int v, int lo, int hi) { return min(max(v, lo), hi); }

constexpr int kBX = 32, kBY = 8;  // pixels per CTA

// act2 plane k, image row r, col c  ->  act2[k * plane_stride + (r - arow0) * W + c]
__global__ void __launch_bounds__(kBX * kBY) k_conv99x11_strict(const uint8_t* __restrict__ y, size_t pitch, int W, int H,
                                                                int yrow0, int yrows, int rb, int re, float* __restrict__ act2,
                                                                size_t plane_stride, int arow0) {
    __shared__ uint8_t tile[kBY + 8][kBX + 8];
    const int col0 = blockIdx.x * kBX, row0 = rb + blockIdx.y * kBY;
    for (int i = threadIdx.x; i < (kBY + 8) * (kBX + 8); i += kBX * kBY) {
        const int tr = i / (kBX + 8), tc = i - tr * (kBX + 8);
        int gr = clampi32(row0 + tr - 4, 0, H - 1);
        const int gc = clampi32(col0 + tc - 4, 0, W - 1);
        gr = clampi32(gr - yrow0, 0, yrows - 1);  // rows past the band are never consumed; keep the load in bounds
        tile[tr][tc] = y[(size_t)gr * pitch + gc];
    }
    __syncthreads();
    const int tx = threadIdx.x & (kBX - 1), ty = threadIdx.x / kBX;
    const int col = col0 + tx, row = row0 + ty;
    if (col >= W || row >= re) return;

    float px[81];
#pragma unroll
    for (int i = 0; i < 9; i++)
#pragma unroll
        for (int j = 0; j < 9; j++) px[i * 9 + j] = (float)(int)tile[ty + i][tx + j];

    float res[kC2];
#pragma unroll
    for (int m = 0; m < kC2; m++) res[m] = 0.0f;

#pragma unroll 1
    for (int k = 0; k < kC1; k++) {
        const float* wk = c_params + kOffW1 + k * 81;
        float acc = 0.0f;
#pragma unroll
        for (int t = 0; t < 81; t++) acc = __fadd_rn(acc, __fmul_rn(wk[t], px[t]));  // :297
        acc = __fadd_rn(acc, c_params[kOffB1 + k]);                                  // :301
        acc = (acc < 0) ? 0 : acc;                                                   // :304
        // conv2 accumulates in i (= k here) order for every output m, exactly like :312-315
#pragma unroll
        for (int m = 0; m < kC2; m++) res[m] = __fadd_rn(res[m], __fmul_rn(acc, c_params[kOffW2 + m * kC1 + k]));
    }
    const size_t o = (size_t)(row - arow0) * W + col;
#pragma unroll
    for (int m = 0; m < kC2; m++) {
        float r = __fadd_rn(res[m], c_params[kOffB2 + m]);  // :316
        act2[m * plane_stride + o] = (r < 0) ? 0 : r;       // :319-321
    }
}

__global__ void __launch_bounds__(256) k_conv55_strict(const float* __restrict__ act2, size_t plane_stride, int arow0,
                                                       int W, int H, int rb, int re, uint8_t* __restrict__ out,
                                                       size_t out_pitch, int orow0) {
    const int col = blockIdx.x * 32 + (threadIdx.x & 31);
    const int row = rb + blockIdx.y * 8 + (threadIdx.x >> 5);
    if (col >= W || row >= re) return;
    int rr[5], cc[5];
#pragma unroll
    for (int t = 0; t < 5; t++) {
        rr[t] = clampi32(row + t - 2, 0, H - 1) - arow0;
        cc[t] = clampi32(col + t - 2, 0, W - 1);
    }
    float temp = 0.0f;
#pragma unroll 1
    for (int i = 0; i < kC2; i++) {
        const float* pl = act2 + i * plane_stride;
        const float* wk = c_params + kOffW3 + i * 25;
        double tp = 0.0;
#pragma unroll
        for (int m = 0; m < 5; m++)
#pragma unroll
            for (int n = 0; n < 5; n++) {
                const float p = __fmul_rn(wk[m * 5 + n], pl[(size_t)rr[m] * W + cc[n]]);
                tp = __dadd_rn(tp, (double)p);                 // :227-228
            }
        temp = (float)__dadd_rn((double)temp, tp);             // :232
    }
    temp = __fadd_rn(temp, c_params[kOffB3]);                  // :235
    int t = (int)temp;                                         // :238 truncation toward zero
    t = clampi32(t, 0, 255);
    out[(size_t)(row - orow0) * out_pitch + col] = (uint8_t)t; // :240
}

// The parameters live in the constant bank of each DEVICE (one copy per device and process, shared by every context on it).
// Called from srcnn_create with the context's device current; srcnn_create synchronises the device afterwards, so no
// launch -- from this context or from one created later by another thread -- can run ahead of the upload.
int fp32_prepare(Ctx* c) {
    static std::mutex mu;
    static bool loaded[64] = {false};
    std::lock_guard<std::mutex> lock(mu);
    if (c->device < 64 && loaded[c->device]) return SRCNN_OK;
    SRCNN_CUDA(c, cudaMemcpyToSymbolAsync(c_params, srcnn_weights_blob, sizeof(float) * kNumParams, 0, cudaMemcpyHostToDevice, c->stream));
    SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
    if (c->device < 64) loaded[c->device] = true;
    return SRCNN_OK;
}

int launch_cnn_fp32(Ctx* c, const CnnArgs& a, float* act2_out) {
    int rc;
    const int W = a.W, H = a.H;
    if (act2_out) {  // full-image activations dump (stage API): plane stride H*W, row 0 = image row 0
        dim3 g1((W + kBX - 1) / kBX, (H + kBY - 1) / kBY);
        k_conv99x11_strict<<<g1, kBX * kBY, 0, c->stream>>>(a.y, a.pitch, W, H, a.row0, a.rows, 0, H, act2_out,
                                                            (size_t)W * H, 0);
        c->launches++;
        SRCNN_CUDA(c, cudaGetLastError());
        return SRCNN_OK;
    }
    // row chunks: conv2 activations of rows [cb-2, ce+2) live in the scratch buffer (<= ~512 MB)
    const size_t row_bytes = (size_t)W * sizeof(float) * kC2;
    long long max_rows = (long long)((512ull << 20) / row_bytes) - 4;
    if (max_rows < 8) max_rows = 8;
    for (int cb = a.out_begin; cb < a.out_end; cb += (int)max_rows) {
        const int ce = std::min<long long>(a.out_end, cb + max_rows);
        const int ab = std::max(cb - 2, 0), ae = std::min(ce + 2, H);
        const size_t plane_stride = (size_t)(ae - ab) * W;
        rc = ensure(c, c->act2_buf, plane_stride * kC2 * sizeof(float));
        if (rc) return rc;
        float* act2 = (float*)c->act2_buf.p;
        dim3 g1((W + kBX - 1) / kBX, (ae - ab + kBY - 1) / kBY);
        k_conv99x11_strict<<<g1, kBX * kBY, 0, c->stream>>>(a.y, a.pitch, W, H, a.row0, a.rows, ab, ae, act2, plane_stride, ab);
        c->launches++;
        SRCNN_CUDA(c, cudaGetLastError());
        dim3 g2((W + 31) / 32, (ce - cb + 7) / 8);
        k_conv55_strict<<<g2, 256, 0, c->stream>>>(act2, plane_stride, ab, W, H, cb, ce, a.out, a.out_pitch, a.out_row0);
        c->launches++;
        SRCNN_CUDA(c, cudaGetLastError());
    }
    return SRCNN_OK;
}

}  // namespace srcnn
