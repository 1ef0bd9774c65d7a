// color_bicubic_int.cu -- kernel A of the hot path for INTEGER up-scales (x2, x4): the shapes every BASELINE configuration but the
// 384x384 golden pair uses.  Same arithmetic, bit for bit, as the generic kernel in color_bicubic.cu -- cvtColor(BGR2YCrCb)
// src/srcnn.cpp:509, split :540, three resize(..., CV_INTER_CUBIC) :570-583 -- restated for the case where the tap tables are
// periodic: output sample d = S*j + k reads source columns j-2+(k >= S/2) .. +3 with the taps of phase k, whatever j is.  So there
// are S constant tap sets (kernel parameters: constant-bank operands, no table loads), and a window of four source rows
// feeds S output rows.
//
// A tile = 256 output columns x isr*S output rows (isr = 8 or 16 source rows, chosen per launch); one CTA of three warps per
// tile, warp w owns plane w (Y, Cr, Cb), a lane owns 8 adjacent columns.
//   (1) the tile's source footprint (isr+3 rows) is colour-converted into shared memory once: four pixels per step from three
//       aligned 32-bit loads (all of a thread's loads are issued before its first conversion), dp2a for the dot products, one
//       32-bit shared store per plane; replicate border applied here;
//   (2) each lane walks down the footprint rows: per row 8 horizontal sums (16 dp2a on funnel-shifted windows; the int -> float
//       conversion is the dp2a's accumulator starting at the bit pattern of 1.5 * 2^23 and ONE packed subtraction per pair), kept
//       as packed FP32 pairs in a register window of four rows; per row S output rows of
//       v = H0*b0 + (H1*b1 + (H2*b2 + H3*b3)), every product and sum rounded on its own (f2_mul_rn / f2_add_rn), round-half-even,
//       saturate, one 8- or 16-byte store per lane and row.  No shared-memory round trip of the sums, no per-sample addressing.
// Y goes to the padded FP16 plane of the tcgen05 kernel when the context has one (color_bicubic.cu explains the layout).
// A grey source (SRCNN_ORDER_GRAY) has its own kernel below, k_gray_bicubic_int: raw bytes staged, the same walk.  A four-channel
// source (SRCNN_ORDER_BGRA / _RGBA) has k_color4_bicubic_int: a fourth warp walks the alpha plane.
// Measured and not kept (tools/experiments/color_bicubic_int_persistent_tma.cu.txt, DESIGN.md): fetching a tile's raw rows by TMA
// (neutral), persistent CTAs with the next tile's rows prefetched by TMA -- as one block-wide pipeline, with a producer warp, or
// as three per-warp pipelines (all slower: the kernel is bound by instruction issue while a wave of tiles computes, and every
// persistent form added instructions or took warps away from the walk).
#include "color_bicubic.h"

namespace srcnn {

namespace {

// x2 instance: minimum CTAs per SM the register allocation is held to.  Same-box A/B inside the bench step (tools/ab_bench_libs.sh):
// 9 (72 registers, 96 B of spills in the walk) 49.1 GPix/s, 8 (80 registers, 32 B) 49.5-49.8, 6 (91 registers, none) 49.9 -- but
// 1 % slower than 8 in many-wave launches (1024 720p frames: 8.33 vs 8.24 ms); 10 (64 registers) 48.5.
#ifndef SRCNN_KA_MINB
#define SRCNN_KA_MINB 8
#endif
#ifndef SRCNN_KA_MINB4
#define SRCNN_KA_MINB4 5         // x4 instance: 126 registers, no spills -- 168.7 vs 174.6 us per 4K -> 16K frame with 6 (96 registers, 64 B of spills)
#endif
constexpr int kISRMax = 16;         // most source rows a tile advances by (IntTaps::isr; plus 3 rows of apron staged with them)
constexpr int kIRows = kISRMax + 3;
constexpr int kIPitch = 144;       // bytes per converted row: 34 four-pixel groups + one spare word for the 3-word window read
constexpr int kITW = 256;          // output columns per tile
constexpr float kMagic = 12582912.0f;   // 1.5 * 2^23: int bits 0x4B400000 + k is the float 12582912 + k for |k| < 2^22

struct IntTaps {
    uint32_t hk01[4], hk23[4];          // horizontal taps of phase k as signed 16-bit pairs (taps 0,1 / 2,3)
    unsigned long long vb[4][4];        // vertical taps of phase k as FP32 pairs (b, b), b = tap * 2^-22 (exact)
    uint32_t sel[4];                    // byte selectors that turn three source words into four (B, G, R, x) pixel words
    int a_first, i_last;                // first / last source row index i whose output rows S*i + S/2 .. + S-1 are wanted
    int vec_ok;                         // source rows are 4-byte aligned: footprint groups inside the image take 32-bit loads
                                        // (2: 16-byte aligned, four-channel groups take one 128-bit load)
    int isr;                            // source rows a tile advances by (4 .. kISRMax)
    int ntx, nty, ntiles;               // tiles per row of tiles, rows of tiles per frame, tiles in the launch (frames included)
};

// where tile `tile` of a launch lies, for CTAs that cover `tw` output columns
struct TilePos {
    size_t fz;                          // frame
    int X0;                             // first output column
    int a;                              // source row index: footprint row r is source row a - 1 + r
    int F0;                             // first footprint column (a multiple of 4: aligned groups)
    int nit, nsr;                       // source rows the tile advances by; footprint rows
};
template <int S>
__device__ __forceinline__ TilePos tile_pos(const IntTaps& t, int tile, int tw) {
    TilePos r;
    const int bx = tile % t.ntx, rest = tile / t.ntx;
    const int by = rest % t.nty;
    r.fz = (size_t)(rest / t.nty);
    r.X0 = bx * tw;
    r.a = t.a_first + by * t.isr;
    r.F0 = r.X0 / S - 4;
    r.nit = min(t.isr, t.i_last - r.a + 1);
    r.nsr = r.nit + 3;
    return r;
}


__device__ __forceinline__ int dp2a_lo_su(uint32_t k, uint32_t px, int c) {
    int d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(k), "r"(px), "r"(c));
    return d;
}
__device__ __forceinline__ int dp2a_hi_su(uint32_t k, uint32_t px, int c) {
    int d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(k), "r"(px), "r"(c));
    return d;
}
// sat_u8(lo) | sat_u8(hi) << 8 | (upper & 0xFFFF) << 16
__device__ __forceinline__ uint32_t pack2_sat_u8(int lo, int hi, uint32_t upper) {
    uint32_t d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(hi), "r"(lo), "r"(upper));
    return d;
}

// which 4-byte window (in bytes past the lane's first footprint column) output column c of a lane's 8 reads
template <int S>
__host__ __device__ constexpr int win_ofs(int c) {
    // floor((2c + 1 - S) / (2S)) + 1, written for non-negative operands
    return (2 * c + 1 - S + 2 * S) / (2 * S);
}

template <int S>
struct Geo {
    static constexpr int G = kITW / S / 4 + 2;             // four-pixel groups per footprint row (the first starts 4 columns left of the tile)
};

// (1) four (B, G, R, x) pixel words -> one 32-bit word per plane of the converted footprint.  OpenCV RGB2YCrCb_i<uchar>, yuv_shift 14.
// Byte 3 of a pixel word never counts: only the two dp2a.hi read it, against the upper 16-bit halves of kYhi and kR, and both
// halves are zero -- so the x byte may be anything, the alpha byte of a four-channel pixel included.
__device__ __forceinline__ void convert_px4(const uint32_t (&pw)[4], uint8_t* y4, uint8_t* cr4, uint8_t* cb4) {
    const uint32_t kYlo = 1868u | (9617u << 16), kYhi = 4899u, kR = 11682u, kB = 9241u;
    const int cadd = (128 << 14) + 8192;
    int Y[4], Cr[4], Cb[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        Y[j] = dp2a_hi_su(kYhi, pw[j], dp2a_lo_su(kYlo, pw[j], 8192)) >> 14;
        Cr[j] = (dp2a_hi_su(kR, pw[j], cadd) - Y[j] * 11682) >> 14;
        Cb[j] = (dp2a_lo_su(kB, pw[j], cadd) - Y[j] * 9241) >> 14;
    }
    *reinterpret_cast<uint32_t*>(y4) = __byte_perm(__byte_perm(Y[0], Y[1], 0x0040), __byte_perm(Y[2], Y[3], 0x0040), 0x5410);
    *reinterpret_cast<uint32_t*>(cr4) = pack2_sat_u8(Cr[0], Cr[1], pack2_sat_u8(Cr[2], Cr[3], 0u));
    *reinterpret_cast<uint32_t*>(cb4) = pack2_sat_u8(Cb[0], Cb[1], pack2_sat_u8(Cb[2], Cb[3], 0u));
}
// twelve source bytes = four three-byte pixels
__device__ __forceinline__ void convert_group(const IntTaps& t, uint32_t w0, uint32_t w1, uint32_t w2, uint8_t* y4, uint8_t* cr4, uint8_t* cb4) {
    uint32_t pw[4];     // (B, G, R, x) per pixel
    pw[0] = __byte_perm(w0, w0, t.sel[0]);
    pw[1] = __byte_perm(w0, w1, t.sel[1]);
    pw[2] = __byte_perm(w1, w2, t.sel[2]);
    pw[3] = __byte_perm(w2, w2, t.sel[3]);
    convert_px4(pw, y4, cr4, cb4);
}
// the same twelve bytes for a group that crosses the left / right image edge: from clamped pixels of a row that starts at `row`
// (the byte of pixel 0, channel 0)
__device__ __forceinline__ void clamped_group(const uint8_t* row, int gx, int sw, uint32_t (&w)[3]) {
    w[0] = w[1] = w[2] = 0u;
#pragma unroll
    for (int j = 0; j < 12; j++) {
        const int x = clampi(gx + j / 3, 0, sw - 1);
        w[j >> 2] |= (uint32_t)row[3 * (long long)x + (j % 3)] << (8 * (j & 3));
    }
}

// (2) the walk of one warp (one plane) down a tile's converted footprint `plane` (rows kPitch bytes apart): lane's output columns
// x0 .. x0+7 read footprint bytes cb .. cb+7 of a row.  NPL = 4: plane 3 is the alpha plane `pa` (same pitch and frame stride).
template <int S, int kPitch = kIPitch, int NPL = 3>
__device__ __forceinline__ void walk_tile(const ResizeDev& p, const IntTaps& t, const uint8_t* plane, int pl, int lane, int X0, int a,
                                          int nit, size_t fz, uint8_t* pa = nullptr) {
    const int x0 = X0 + 8 * lane;
    if (x0 >= p.ow) return;                        // ow is a multiple of 8 (launch condition)
    const int cb = (8 * lane) / S + 2;
    const uint8_t* const srow = plane + (cb & ~3);
    const int wsh = (cb & 3) * 8;                  // x2: always 16
    const unsigned long long nz = p.negzero2;
    const unsigned long long mm = f2_pack(-kMagic, -kMagic);
    const bool y16 = pl == 0 && p.y16 != nullptr;
    const size_t ostep = y16 ? p.pitch16 : p.pitch;

    auto hsum = [&](int r, unsigned long long (&h)[4]) {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(srow + r * kPitch);
        const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
        uint32_t lo = 0, hi = 0;
        if (S != 2) { lo = __funnelshift_r(w0, w1, wsh); hi = __funnelshift_r(w1, w2, wsh); }
        float f[8];
#pragma unroll
        for (int c = 0; c < 8; c++) {
            const int o = win_ofs<S>(c);
            uint32_t px4;
            if (S == 2) {                  // bytes cb + o .. + 3 straight from the three words (cb & 3 == 2)
                const int sh = 16 + 8 * o;
                px4 = sh < 32 ? __funnelshift_r(w0, w1, sh) : (sh == 32 ? w1 : __funnelshift_r(w1, w2, sh - 32));
            } else {
                px4 = o == 0 ? lo : (o == 4 ? hi : __funnelshift_r(lo, hi, 8 * o));
            }
            const int acc = dp2a_hi_su(t.hk23[c % S], px4, dp2a_lo_su(t.hk01[c % S], px4, 0x4B400000));
            f[c] = __int_as_float(acc);    // = 12582912 + sum, exactly
        }
#pragma unroll
        for (int q = 0; q < 4; q++) h[q] = f2_add_rn(f2_pack(f[2 * q], f[2 * q + 1]), mm);   // = (float)sum, exactly
    };

    // running output pointer: row S*a + S/2 first, one row further per emitted row (dereferenced only for wanted rows)
    int dy = S * a + S / 2;
    uint8_t* outp;
    if (y16) outp = p.y16 + fz * p.y16_frame + ((long long)dy - p.plane_row0) * (long long)p.pitch16 + 2 * (size_t)(x0 + kY16Pad);
    else outp = (pl == 0 ? p.y : (pl == 1 ? p.cr : (NPL == 4 && pl == 3 ? pa : p.cb))) + fz * p.plane_frame + ((long long)dy - p.plane_row0) * (long long)p.pitch + x0;
    uint8_t* const outp0 = outp;

    auto emit = [&](const unsigned long long (&h0)[4], const unsigned long long (&h1)[4], const unsigned long long (&h2)[4],
                    const unsigned long long (&h3)[4]) {
#pragma unroll
        for (int m = 0; m < S; m++) {
            const int ph = (S / 2 + m) % S;
            const bool wanted = dy >= p.row_begin && dy < p.row_end;     // uniform; only the first / last row of tiles has unwanted rows
            uint32_t r[8];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                float va, vb;
                f2_unpack(f2_vtap(h0[q], h1[q], h2[q], h3[q], t.vb[ph][0], t.vb[ph][1], t.vb[ph][2], t.vb[ph][3], nz), va, vb);
                r[2 * q] = sat_u8_rn(va);
                r[2 * q + 1] = sat_u8_rn(vb);
            }
            if (y16) {
                const uint4 hw = make_uint4(u8x2_to_h2(r[0], r[1]), u8x2_to_h2(r[2], r[3]), u8x2_to_h2(r[4], r[5]), u8x2_to_h2(r[6], r[7]));
                if (wanted) *reinterpret_cast<uint4*>(outp) = hw;
            } else {
                const uint32_t lo4 = __byte_perm(__byte_perm(r[0], r[1], 0x0040), __byte_perm(r[2], r[3], 0x0040), 0x5410);
                const uint32_t hi4 = __byte_perm(__byte_perm(r[4], r[5], 0x0040), __byte_perm(r[6], r[7], 0x0040), 0x5410);
                if (wanted) *reinterpret_cast<uint2*>(outp) = make_uint2(lo4, hi4);
            }
            dy++;
            outp += ostep;
        }
    };

    walk_window<unsigned long long[4]>(nit, hsum, emit);

    // FP16 plane: the replicated columns -8..-1 and W..W+7 (conv1 reads Y[clamp(c-4)], src/srcnn.cpp:279) -- by the two
    // lanes that own the first / last eight columns of the image, from what they have just stored
    if (y16 && (x0 == 0 || x0 + 8 == p.ow)) {
        int d = S * a + S / 2;
        uint8_t* o = outp0;
        for (int j = 0; j < nit * S; j++, d++, o += ostep) {
            if (d < p.row_begin || d >= p.row_end) continue;
            const uint4 v = *reinterpret_cast<const uint4*>(o);
            if (x0 == 0) {
                const uint32_t e = __byte_perm(v.x, 0, 0x1010);
                *reinterpret_cast<uint4*>(o - 2 * kY16Pad) = make_uint4(e, e, e, e);
            }
            if (x0 + 8 == p.ow) {
                const uint32_t e = __byte_perm(v.w, 0, 0x3232);
                *reinterpret_cast<uint4*>(o + 16) = make_uint4(e, e, e, e);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// The kernel: one CTA of 3 warps per tile.
// ------------------------------------------------------------------------------------------------
template <int S>
__global__ void __launch_bounds__(96, S == 2 ? SRCNN_KA_MINB : SRCNN_KA_MINB4) k_color_bicubic_int(const ResizeDev p, const IntTaps t) {
    constexpr int G = Geo<S>::G;
    __shared__ __align__(16) uint8_t sP[3][kIRows][kIPitch];
    const int tid = threadIdx.x;
    const int tile = blockIdx.x;
    const auto [fz, X0, a, F0, nit, nsr] = tile_pos<S>(t, tile, kITW);
    const uint8_t* const fsrc = p.src + fz * p.src_frame;

    // (1) colour-convert the footprint; replicate border applied here
    if (t.vec_ok && F0 >= 0 && F0 + 4 * G <= p.sw) {
        // every group lies inside the image and is word-aligned: all of a thread's loads go out before its first conversion
        constexpr int NG = (kIRows * G + 95) / 96;
        uint32_t raw[NG][3];
#pragma unroll
        for (int it = 0; it < NG; it++) {
            const int g = tid + 96 * it;
            if (g < nsr * G) {
                const int r = g / G, q = g - r * G;
                const int gy = clampi(a - 1 + r, 0, p.sh - 1) - p.src_row0;
                const uint32_t* w = reinterpret_cast<const uint32_t*>(fsrc + (size_t)gy * p.src_stride + 3 * (size_t)(F0 + 4 * q));
                raw[it][0] = w[0]; raw[it][1] = w[1]; raw[it][2] = w[2];
            }
        }
#pragma unroll
        for (int it = 0; it < NG; it++) {
            const int g = tid + 96 * it;
            if (g < nsr * G) {
                const int r = g / G, q = g - r * G;
                convert_group(t, raw[it][0], raw[it][1], raw[it][2], &sP[0][r][4 * q], &sP[1][r][4 * q], &sP[2][r][4 * q]);
            }
        }
    } else {
        for (int g = tid; g < nsr * G; g += 96) {
            const int r = g / G, q = g - r * G;
            const int gy = clampi(a - 1 + r, 0, p.sh - 1) - p.src_row0;
            uint32_t w[3];
            clamped_group(fsrc + (size_t)gy * p.src_stride, F0 + 4 * q, p.sw, w);
            convert_group(t, w[0], w[1], w[2], &sP[0][r][4 * q], &sP[1][r][4 * q], &sP[2][r][4 * q]);
        }
    }
    __syncthreads();
    // (2) the walk
    walk_tile<S>(p, t, &sP[tid >> 5][0][0], tid >> 5, tid & 31, X0, a, nit, fz);
    // Launched with programmatic stream serialisation (api.cu, may_start_early) this grid may have started while the merge kernel
    // of the previous whole-path call was still running; nothing here depends on it.  The last tile waits for that kernel at its
    // very end, so that "this grid has finished" still implies "everything before it in the stream has finished" for whatever
    // follows.  A no-op after an ordinary launch.
    if (tile == t.ntiles - 1) asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// Four-channel form (SRCNN_ORDER_BGRA / _RGBA): one CTA of FOUR warps per tile, warp w walks plane w (Y, Cr, Cb, A) with the
// same walk.  A footprint group is 16 source bytes = four pixel words: one 128-bit load when the source is 16-byte aligned, four
// 32-bit loads when it is 4-byte aligned, clamped bytes at the image edges.  A BGRA word already is the (B, G, R, x) word
// convert_px4 takes (the alpha byte drops out of every dp2a); an RGBA word takes one byte permutation.  The alpha plane is byte 3
// of the four words, gathered into one 32-bit shared store.  128 threads: the 96-thread budgets (80 / 126 registers at 8 / 5
// CTAs per SM) would not fit the register file, so the same threads per SM are kept with 6 / 4 CTAs.
// ------------------------------------------------------------------------------------------------
#ifndef SRCNN_KA4_MINB
#define SRCNN_KA4_MINB 6
#endif
#ifndef SRCNN_KA4_MINB4
#define SRCNN_KA4_MINB4 4
#endif

__device__ __forceinline__ void convert_group4(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, bool swap, uint8_t* y4, uint8_t* cr4,
                                               uint8_t* cb4, uint8_t* a4) {
    uint32_t pw[4] = {w0, w1, w2, w3};
    if (swap) {   // (R, G, B, A) -> (B, G, R, A)
#pragma unroll
        for (int j = 0; j < 4; j++) pw[j] = __byte_perm(pw[j], 0, 0x3012);
    }
    convert_px4(pw, y4, cr4, cb4);
    *reinterpret_cast<uint32_t*>(a4) = __byte_perm(__byte_perm(w0, w1, 0x0073), __byte_perm(w2, w3, 0x0073), 0x5410);
}

template <int S>
__global__ void __launch_bounds__(128, S == 2 ? SRCNN_KA4_MINB : SRCNN_KA4_MINB4) k_color4_bicubic_int(const ResizeDev p, const IntTaps t,
                                                                                                      uint8_t* const pa) {
    constexpr int G = Geo<S>::G;
    __shared__ __align__(16) uint8_t sP[4][kIRows][kIPitch];
    const int tid = threadIdx.x;
    const int tile = blockIdx.x;
    const auto [fz, X0, a, F0, nit, nsr] = tile_pos<S>(t, tile, kITW);
    const uint8_t* const fsrc = p.src + fz * p.src_frame;
    const bool swap = p.swapRB;

    // (1) colour-convert the footprint; replicate border applied here
    if (t.vec_ok && F0 >= 0 && F0 + 4 * G <= p.sw) {
        constexpr int NG = (kIRows * G + 127) / 128;
        uint32_t raw[NG][4];
#pragma unroll
        for (int it = 0; it < NG; it++) {
            const int g = tid + 128 * it;
            if (g < nsr * G) {
                const int r = g / G, q = g - r * G;
                const int gy = clampi(a - 1 + r, 0, p.sh - 1) - p.src_row0;
                const uint8_t* px = fsrc + (size_t)gy * p.src_stride + 4 * (size_t)(F0 + 4 * q);
                if (t.vec_ok == 2) {
                    const uint4 v = *reinterpret_cast<const uint4*>(px);
                    raw[it][0] = v.x; raw[it][1] = v.y; raw[it][2] = v.z; raw[it][3] = v.w;
                } else {
                    const uint32_t* w = reinterpret_cast<const uint32_t*>(px);
                    raw[it][0] = w[0]; raw[it][1] = w[1]; raw[it][2] = w[2]; raw[it][3] = w[3];
                }
            }
        }
#pragma unroll
        for (int it = 0; it < NG; it++) {
            const int g = tid + 128 * it;
            if (g < nsr * G) {
                const int r = g / G, q = g - r * G;
                convert_group4(raw[it][0], raw[it][1], raw[it][2], raw[it][3], swap, &sP[0][r][4 * q], &sP[1][r][4 * q], &sP[2][r][4 * q],
                               &sP[3][r][4 * q]);
            }
        }
    } else {
        for (int g = tid; g < nsr * G; g += 128) {
            const int r = g / G, q = g - r * G;
            const int gy = clampi(a - 1 + r, 0, p.sh - 1) - p.src_row0;
            const uint8_t* row = fsrc + (size_t)gy * p.src_stride;
            uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int j = 0; j < 16; j++) {
                const int x = clampi(F0 + 4 * q + j / 4, 0, p.sw - 1);
                w[j >> 2] |= (uint32_t)row[4 * (size_t)x + (j & 3)] << (8 * (j & 3));
            }
            convert_group4(w[0], w[1], w[2], w[3], swap, &sP[0][r][4 * q], &sP[1][r][4 * q], &sP[2][r][4 * q], &sP[3][r][4 * q]);
        }
    }
    __syncthreads();
    // (2) the walk
    walk_tile<S, kIPitch, 4>(p, t, &sP[tid >> 5][0][0], tid >> 5, tid & 31, X0, a, nit, fz, pa);
    // may have started beside the previous call's merge kernel: see k_color_bicubic_int
    if (tile == t.ntiles - 1) asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// One-plane form (SRCNN_ORDER_GRAY): the footprint is the source bytes as they are, with the replicate border.  One CTA of
// three warps takes three ADJACENT tiles: their footprints are one contiguous run of 3 * kITW / S + 8 source columns, staged
// once, and warp w walks tile w from its own offset in it -- the same 96-thread CTA (and occupancy tuning) and the same
// walk as the colour kernel.
// ------------------------------------------------------------------------------------------------
constexpr int kGPitch = 400;       // bytes per staged row: 3 * 128 + 8 columns at x2 (98 words) + the spare word of the window read

// The grey kernel's tile `tile`, also the luma tile of k_yuv_bicubic_int.  L = SRCNN_ORDER_YUY2 / _UYVY: the Y bytes of packed
// 4:2:2 rows (YUY2: bytes 0, 2 of each macropixel; UYVY: 1, 3): a four-pixel group is 8 source bytes (one 64-bit load when
// t.vec_ok == 2, two 32-bit loads when 1) and one byte permutation.  Any other L: a plane of bytes.
template <int S, int L>
__device__ __forceinline__ void gray_tile(const ResizeDev& p, const IntTaps& t, int tile, uint8_t (&sP)[kIRows][kGPitch]) {
    constexpr bool k422 = L == SRCNN_ORDER_YUY2 || L == SRCNN_ORDER_UYVY, kUYVY = L == SRCNN_ORDER_UYVY;
    constexpr int GG = 3 * kITW / S / 4 + 2;       // four-byte groups per staged row
    static_assert(4 * GG + 4 <= kGPitch, "staged row too short");
    const int tid = threadIdx.x;
    const auto [fz, X0, a, F0, nit, nsr] = tile_pos<S>(t, tile, 3 * kITW);   // X0: first column of warp 0's tile
    const uint8_t* const fsrc = p.src + fz * p.src_frame;

    // (1) stage the footprint: all of a thread's loads go out before its first shared store
    constexpr int NG = (kIRows * GG + 95) / 96;
    uint32_t raw[NG];
#pragma unroll
    for (int it = 0; it < NG; it++) {
        const int g = tid + 96 * it;
        if (g < nsr * GG) {
            const int r = g / GG, gx = F0 + 4 * (g - r * GG);
            const uint8_t* row = fsrc + (size_t)(clampi(a - 1 + r, 0, p.sh - 1) - p.src_row0) * p.src_stride;
            if (t.vec_ok && gx >= 0 && gx + 4 <= p.sw) {
                if (!k422) {
                    raw[it] = *reinterpret_cast<const uint32_t*>(row + gx);
                } else {
                    const uint8_t* px = row + 2 * (size_t)gx;
                    uint32_t w0, w1;
                    if (t.vec_ok == 2) {
                        const uint2 v = *reinterpret_cast<const uint2*>(px);
                        w0 = v.x; w1 = v.y;
                    } else {
                        w0 = reinterpret_cast<const uint32_t*>(px)[0]; w1 = reinterpret_cast<const uint32_t*>(px)[1];
                    }
                    raw[it] = __byte_perm(w0, w1, kUYVY ? 0x7531 : 0x6420);
                }
            } else {
                uint32_t v = 0;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const int x = clampi(gx + j, 0, p.sw - 1);
                    v |= (uint32_t)row[!k422 ? x : 2 * x + kUYVY] << (8 * j);
                }
                raw[it] = v;
            }
        }
    }
#pragma unroll
    for (int it = 0; it < NG; it++) {
        const int g = tid + 96 * it;
        if (g < nsr * GG) {
            const int r = g / GG;
            *reinterpret_cast<uint32_t*>(&sP[r][4 * (g - r * GG)]) = raw[it];
        }
    }
    __syncthreads();
    // (2) the walk: warp w's tile starts w * kITW / S staged columns further
    const int w = tid >> 5;
    walk_tile<S, kGPitch>(p, t, &sP[0][w * (kITW / S)], 0, tid & 31, X0 + w * kITW, a, nit, fz);
}

template <int S>
__global__ void __launch_bounds__(96, S == 2 ? SRCNN_KA_MINB : SRCNN_KA_MINB4) k_gray_bicubic_int(const ResizeDev p, const IntTaps t) {
    __shared__ __align__(16) uint8_t sP[kIRows][kGPitch];
    gray_tile<S, SRCNN_ORDER_GRAY>(p, t, blockIdx.x, sP);
}

// ------------------------------------------------------------------------------------------------
// 4:2:0 and packed 4:2:2 frames (SRCNN_ORDER_NV12 / _I420 / _YUY2 / _UYVY, the layout L): ONE launch for luma and chroma.  CTAs
// [0, t.ntiles) are the grey kernel's tiles of the Y plane (gray_tile, into the workspace plane the CNN reads); the rest are
// chroma tiles.  A chroma CTA is three warps on three adjacent 128-column tiles whose footprints are staged once, like the grey
// kernel's, as two shared-memory planes U and V: NV12's pairs are split with two byte permutations per four columns, I420's
// planes are staged as they are, packed 4:2:2 rows give the U and V words of four columns with four byte permutations.  A lane
// owns the SAME 4 columns of both planes, so the 8 horizontal sums per footprint row, the four-row register window and the
// vertical pass are those of walk_tile (which gives a lane 8 columns of one plane); per output row it stores U0 V0 U1 V1 U2 V2
// U3 V3 (NV12, one 8-byte store) or four bytes into each plane.  4:2:0 chroma goes straight into the caller's output (no chroma
// workspace, no CNN); 4:2:2 chroma into the workspace's Cr (U') and Cb (V') planes, which the pack kernel (K-C) reads.  The 4:2:2
// chroma plane is w/2 x h -> ow/2 x oh: x S on both axes, so its vertical taps are the luma ones.  Launch conditions: luma and
// chroma widths multiples of 8, 8-byte aligned luma stores, chroma stores 8-byte (4:2:0) or 4-byte (4:2:2: always true of the
// workspace) aligned.
// ------------------------------------------------------------------------------------------------
struct ChromaDev {
    const uint8_t* src;               // chroma row 0 of frame 0 (NV12: pairs; I420: U; 4:2:2: the packed rows)
    size_t src_pitch, src_v, src_frame;
    uint8_t* dst;
    size_t dst_pitch, dst_v, dst_frame;
    int sw, sh, ow, row_begin, row_end;   // chroma plane sizes, chroma output rows wanted
};
constexpr int kCW = 128;           // chroma columns per warp: 4 per lane, of both planes
template <int S>
struct CGeo {
    static constexpr int G = 3 * kCW / S / 4 + 2;                  // four-column groups per staged row
    static constexpr int kPitch = (4 * G + 4 + 15) / 16 * 16;      // + the spare word of the window read
};

template <int S, int L>
__device__ __forceinline__ void walk_pair(const ChromaDev& q, const IntTaps& t, unsigned long long nz, const uint8_t* su,
                                          const uint8_t* sv, int lane, int X0, int a, int nit, size_t fz) {
    constexpr bool kNV12 = L == SRCNN_ORDER_NV12;
    constexpr int kPitch = CGeo<S>::kPitch;
    const int x0 = X0 + 4 * lane;
    if (x0 >= q.ow) return;                        // ow/2 is a multiple of 8 (launch condition)
    const int cb = (4 * lane) / S + 2;             // footprint byte of the lane's first tap (x0 % S == 0)
    const uint8_t* const ru = su + (cb & ~3);
    const uint8_t* const rv = sv + (cb & ~3);
    const int wsh = (cb & 3) * 8;
    const unsigned long long mm = f2_pack(-kMagic, -kMagic);

    auto hsum = [&](int r, unsigned long long (&h)[4]) {   // h[0], h[1]: U columns 0..3; h[2], h[3]: V columns 0..3
        float f[8];
#pragma unroll
        for (int pl = 0; pl < 2; pl++) {
            const uint32_t* w = reinterpret_cast<const uint32_t*>((pl ? rv : ru) + r * kPitch);
            const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
            const uint32_t lo = __funnelshift_r(w0, w1, wsh), hi = __funnelshift_r(w1, w2, wsh);
#pragma unroll
            for (int c = 0; c < 4; c++) {
                const int o = win_ofs<S>(c);       // 0 .. 2
                const uint32_t px4 = o == 0 ? lo : __funnelshift_r(lo, hi, 8 * o);
                f[4 * pl + c] = __int_as_float(dp2a_hi_su(t.hk23[c % S], px4, dp2a_lo_su(t.hk01[c % S], px4, 0x4B400000)));
            }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) h[k] = f2_add_rn(f2_pack(f[2 * k], f[2 * k + 1]), mm);
    };

    int dy = S * a + S / 2;
    uint8_t* outp = q.dst + fz * q.dst_frame + (long long)dy * (long long)q.dst_pitch + (kNV12 ? 2 : 1) * (size_t)x0;
    auto emit = [&](const unsigned long long (&h0)[4], const unsigned long long (&h1)[4], const unsigned long long (&h2)[4],
                    const unsigned long long (&h3)[4]) {
#pragma unroll
        for (int m = 0; m < S; m++) {
            const int ph = (S / 2 + m) % S;
            const bool wanted = dy >= q.row_begin && dy < q.row_end;
            uint32_t r[8];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                float va, vb;
                f2_unpack(f2_vtap(h0[k], h1[k], h2[k], h3[k], t.vb[ph][0], t.vb[ph][1], t.vb[ph][2], t.vb[ph][3], nz), va, vb);
                r[2 * k] = sat_u8_rn(va);
                r[2 * k + 1] = sat_u8_rn(vb);
            }
            if (kNV12) {   // U0 V0 U1 V1 | U2 V2 U3 V3
                const uint32_t lo = __byte_perm(__byte_perm(r[0], r[4], 0x0040), __byte_perm(r[1], r[5], 0x0040), 0x5410);
                const uint32_t hi = __byte_perm(__byte_perm(r[2], r[6], 0x0040), __byte_perm(r[3], r[7], 0x0040), 0x5410);
                if (wanted) *reinterpret_cast<uint2*>(outp) = make_uint2(lo, hi);
            } else {
                const uint32_t u = __byte_perm(__byte_perm(r[0], r[1], 0x0040), __byte_perm(r[2], r[3], 0x0040), 0x5410);
                const uint32_t v = __byte_perm(__byte_perm(r[4], r[5], 0x0040), __byte_perm(r[6], r[7], 0x0040), 0x5410);
                if (wanted) {
                    *reinterpret_cast<uint32_t*>(outp) = u;
                    *reinterpret_cast<uint32_t*>(outp + q.dst_v) = v;
                }
            }
            dy++;
            outp += q.dst_pitch;
        }
    };

    walk_window<unsigned long long[4]>(nit, hsum, emit);
}

// 4:2:2 rows (L = SRCNN_ORDER_YUY2 / _UYVY): U and V at bytes 1, 3 (YUY2) or 0, 2 (UYVY) of each macropixel, a four-column group
// is 16 source bytes (two 64-bit or four 32-bit loads, per t.vec_ok) and four byte permutations for both planes.
template <int S, int L>
__device__ __forceinline__ void chroma_tile(const ChromaDev& q, const IntTaps& t, unsigned long long nz, int tile, uint8_t* smem) {
    constexpr bool kNV12 = L == SRCNN_ORDER_NV12, k422 = L == SRCNN_ORDER_YUY2 || L == SRCNN_ORDER_UYVY, kUYVY = L == SRCNN_ORDER_UYVY;
    constexpr int G = CGeo<S>::G, kPitch = CGeo<S>::kPitch;
    uint8_t (*sU)[kPitch] = reinterpret_cast<uint8_t (*)[kPitch]>(smem);
    uint8_t (*sV)[kPitch] = sU + kIRows;
    const int tid = threadIdx.x;
    const auto [fz, X0, a, F0, nit, nsr] = tile_pos<S>(t, tile, 3 * kCW);    // X0: first chroma column of warp 0's tile
    const uint8_t* const fsrc = q.src + fz * q.src_frame;

    // (1) stage both footprints: all of a thread's loads go out before its first shared store
    constexpr int NG = (kIRows * G + 95) / 96;
    uint32_t ru[NG], rv[NG];
#pragma unroll
    for (int it = 0; it < NG; it++) {
        const int g = tid + 96 * it;
        if (g < nsr * G) {
            const int r = g / G, gx = F0 + 4 * (g - r * G);
            const uint8_t* row = fsrc + (size_t)clampi(a - 1 + r, 0, q.sh - 1) * q.src_pitch;
            if (t.vec_ok && gx >= 0 && gx + 4 <= q.sw) {
                if (k422) {
                    const uint8_t* px = row + 4 * (size_t)gx;
                    uint32_t w[4];
                    if (t.vec_ok == 2) {
                        const uint2 v0 = reinterpret_cast<const uint2*>(px)[0], v1 = reinterpret_cast<const uint2*>(px)[1];
                        w[0] = v0.x; w[1] = v0.y; w[2] = v1.x; w[3] = v1.y;
                    } else {
#pragma unroll
                        for (int k = 0; k < 4; k++) w[k] = reinterpret_cast<const uint32_t*>(px)[k];
                    }
                    constexpr unsigned kSel = kUYVY ? 0x6240 : 0x7351;    // (U0 U1 V0 V1) of two macropixels
                    const uint32_t lo = __byte_perm(w[0], w[1], kSel), hi = __byte_perm(w[2], w[3], kSel);
                    ru[it] = __byte_perm(lo, hi, 0x5410);
                    rv[it] = __byte_perm(lo, hi, 0x7632);
                } else if (kNV12) {
                    const uint32_t* w = reinterpret_cast<const uint32_t*>(row + 2 * gx);
                    const uint32_t w0 = w[0], w1 = w[1];
                    ru[it] = __byte_perm(w0, w1, 0x6420);
                    rv[it] = __byte_perm(w0, w1, 0x7531);
                } else {
                    ru[it] = *reinterpret_cast<const uint32_t*>(row + gx);
                    rv[it] = *reinterpret_cast<const uint32_t*>(row + q.src_v + gx);
                }
            } else {
                uint32_t u = 0, v = 0;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const int x = clampi(gx + j, 0, q.sw - 1);
                    if (k422) {
                        u |= (uint32_t)row[4 * x + !kUYVY] << (8 * j);
                        v |= (uint32_t)row[4 * x + !kUYVY + 2] << (8 * j);
                    } else {
                        u |= (uint32_t)(kNV12 ? row[2 * x] : row[x]) << (8 * j);
                        v |= (uint32_t)(kNV12 ? row[2 * x + 1] : row[q.src_v + x]) << (8 * j);
                    }
                }
                ru[it] = u;
                rv[it] = v;
            }
        }
    }
#pragma unroll
    for (int it = 0; it < NG; it++) {
        const int g = tid + 96 * it;
        if (g < nsr * G) {
            const int r = g / G, o = 4 * (g - r * G);
            *reinterpret_cast<uint32_t*>(&sU[r][o]) = ru[it];
            *reinterpret_cast<uint32_t*>(&sV[r][o]) = rv[it];
        }
    }
    __syncthreads();
    // (2) the walk: warp w's tile starts w * kCW / S staged columns further
    const int w = tid >> 5;
    walk_pair<S, L>(q, t, nz, &sU[0][w * (kCW / S)], &sV[0][w * (kCW / S)], tid & 31, X0 + w * kCW, a, nit, fz);
}

template <int S, int L>
__global__ void __launch_bounds__(96, S == 2 ? SRCNN_KA_MINB : SRCNN_KA_MINB4) k_yuv_bicubic_int(const ResizeDev p, const IntTaps t,
                                                                                               const ChromaDev q, const IntTaps tc) {
    constexpr int kLuma = kIRows * kGPitch, kChroma = 2 * kIRows * CGeo<S>::kPitch;
    __shared__ __align__(16) uint8_t sm[kLuma > kChroma ? kLuma : kChroma];
    const int b = (int)blockIdx.x;
    if (b < t.ntiles) gray_tile<S, L>(p, t, b, *reinterpret_cast<uint8_t (*)[kIRows][kGPitch]>(sm));
    else chroma_tile<S, L>(q, tc, p.negzero2, b - t.ntiles, sm);
    // A 4:2:2 call may start beside the previous call's merge / pack kernel (api.cu, may_start_early): the last CTA waits for it,
    // as in k_color_bicubic_int.  A 4:2:0 call never starts early (it launches no merge), and leaves the wait out.
    if constexpr (L == SRCNN_ORDER_YUY2 || L == SRCNN_ORDER_UYVY)
        if (b == t.ntiles + tc.ntiles - 1) asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// Grey + alpha frames (SRCNN_ORDER_GRAYA): ONE launch for both planes.  A row of byte pairs (G A G A ...) keeps grey where a YUY2 row
// keeps its Y bytes (the even bytes) and alpha where a UYVY row keeps them (the odd bytes), so both tile kinds are gray_tile's 4:2:2
// luma staging as it is -- group loads of 64 bits when the rows are 8-byte aligned, 32 bits when 4-byte aligned, clamped bytes
// otherwise -- and its walk.  CTAs [0, t.ntiles) stage the even bytes into the plane the CNN reads (p: the FP16 plane or the u8
// Y plane); the rest stage the odd bytes into the workspace's Cr plane (pa: the same source rows, the u8 output plane A' and the
// output rows [r0, r1) -- the halo rows around them are the CNN's).  The source is staged twice, once per tile kind.
// ------------------------------------------------------------------------------------------------
template <int S>
__global__ void __launch_bounds__(96, S == 2 ? SRCNN_KA_MINB : SRCNN_KA_MINB4) k_graya_bicubic_int(const ResizeDev p, const IntTaps t,
                                                                                                 const ResizeDev pa, const IntTaps ta) {
    __shared__ __align__(16) uint8_t sP[kIRows][kGPitch];
    const int b = (int)blockIdx.x;
    if (b < t.ntiles) gray_tile<S, SRCNN_ORDER_YUY2>(p, t, b, sP);
    else gray_tile<S, SRCNN_ORDER_UYVY>(pa, ta, b - t.ntiles, sP);
    // may start beside the previous call's merge / pack kernel (api.cu, may_start_early): the last CTA waits for it, as in
    // k_color_bicubic_int
    if (b == t.ntiles + ta.ntiles - 1) asm volatile("griddepcontrol.wait;" ::: "memory");
}

inline int floordiv(int a, int b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

// one launch of an integer-scale kernel, ordinary or with programmatic stream serialisation
template <typename K, typename... A>
int launch_ka(Ctx* c, K kern, int grid, int threads, bool early, const A&... args) {
    if (early) {   // programmatic dependent launch: may begin before the stream's previous kernel (a merge of ours) has finished
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(threads);
        cfg.dynamicSmemBytes = 0;
        cfg.stream = c->stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        SRCNN_CUDA(c, cudaLaunchKernelEx(&cfg, kern, args...));
    } else {
        kern<<<grid, threads, 0, c->stream>>>(args...);
    }
    c->launches++;
    SRCNN_CUDA(c, cudaGetLastError());
    return SRCNN_OK;
}

// The tiles of one launch of kernel K (kThreads threads per CTA): tile height, rows of tiles and tile count of t, and of tc when
// the launch also has chroma tiles (the same height; their CTAs follow t's).  *ok = false when the launch would have more tiles
// than the kernels index: the geometry is not eligible, and the caller falls back to the generic kernels.
template <auto K, int kThreads>
int plan_tiles(Ctx* c, int nframes, IntTaps& t, IntTaps* tc, bool* ok) {
    static int ctas_per_sm[64] = {};               // per kernel instance and device; a benign race: every writer stores the same value
    int& per_sm = ctas_per_sm[c->device & 63];
    if (per_sm == 0) {
        int n = 0;
        SRCNN_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, K, kThreads, 0));
        per_sm = std::max(1, n);
    }
    // Tile height (same-box A/B, B200): a single 4K frame runs fastest as ~1.5 waves of 8-row tiles (23.6 us; 6 rows: 23.7,
    // 4 rows: 25.1, 12 rows: 25.5, 16 rows = one wave: 27.6 -- the CTAs of one wave wait for their source rows together, and the
    // last wave's tiles run at half occupancy for a whole tile life); launches of many waves (batches, 16K frames, gigapixel
    // bands) take 16-row tiles for the smaller apron (7.5 vs 7.8 ms for 1024 720p frames).  Luma and chroma tiles count together.
    const int resident = per_sm * std::max(1, c->sm_count);
    const int nrows = t.i_last - t.a_first + 1, crows = tc ? tc->i_last - tc->a_first + 1 : 0;
    auto tiles_for = [&](int isr) {
        return ((long long)t.ntx * ((nrows + isr - 1) / isr) + (tc ? (long long)tc->ntx * ((crows + isr - 1) / isr) : 0)) * nframes;
    };
    t.isr = tiles_for(kISRMax) > 2LL * resident ? kISRMax : 8;
    if (c->ka_int_isr >= 4 && c->ka_int_isr <= kISRMax) t.isr = c->ka_int_isr;
    *ok = tiles_for(t.isr) <= 0x3fffffffLL;
    if (!*ok) return SRCNN_OK;
    t.nty = (nrows + t.isr - 1) / t.isr;
    t.ntiles = t.ntx * t.nty * nframes;
    if (tc) {
        tc->isr = t.isr;
        tc->nty = (crows + tc->isr - 1) / tc->isr;
        tc->ntiles = tc->ntx * tc->nty * nframes;
    }
    return SRCNN_OK;
}

// NP = planes: 1 grey, 3 colour, 4 colour + alpha (pa)
template <int S, int NP>
int launch_variant(Ctx* c, const ResizeDev& p, IntTaps& t, uint8_t* pa, int nframes, bool early, bool* done) {
    bool ok = false;
    int rc;
    if constexpr (NP == 4) {
        if ((rc = plan_tiles<k_color4_bicubic_int<S>, 128>(c, nframes, t, nullptr, &ok)) || !ok) return rc;
        rc = launch_ka(c, k_color4_bicubic_int<S>, t.ntiles, 128, early, p, t, pa);
    } else {
        constexpr auto kern = NP == 1 ? k_gray_bicubic_int<S> : k_color_bicubic_int<S>;
        if ((rc = plan_tiles<kern, 96>(c, nframes, t, nullptr, &ok)) || !ok) return rc;
        rc = launch_ka(c, kern, t.ntiles, 96, early, p, t);
    }
    *done = rc == SRCNN_OK;
    return rc;
}

template <int S, int L>
int launch_yuv(Ctx* c, const ResizeDev& p, IntTaps& t, const ChromaDev& q, IntTaps& tc, int nframes, bool early, bool* done) {
    bool ok = false;
    int rc;
    if ((rc = plan_tiles<k_yuv_bicubic_int<S, L>, 96>(c, nframes, t, &tc, &ok)) || !ok) return rc;
    rc = launch_ka(c, k_yuv_bicubic_int<S, L>, t.ntiles + tc.ntiles, 96, early, p, t, q, tc);
    *done = rc == SRCNN_OK;
    return rc;
}

template <int S>
int launch_ga(Ctx* c, const ResizeDev& p, IntTaps& t, const ResizeDev& pa, IntTaps& ta, int nframes, bool early, bool* done) {
    bool ok = false;
    int rc;
    if ((rc = plan_tiles<k_graya_bicubic_int<S>, 96>(c, nframes, t, &ta, &ok)) || !ok) return rc;
    rc = launch_ka(c, k_graya_bicubic_int<S>, t.ntiles + ta.ntiles, 96, early, p, t, pa, ta);
    *done = rc == SRCNN_OK;
    return rc;
}

// the constant tap phases of an integer scale S and the source rows whose output rows [row_begin, row_end) are wanted
void int_taps(const TapTable* tx, const TapTable* ty, int S, int row_begin, int row_end, IntTaps& t) {
    const float sc = 1.0f / 4194304.0f;   // 2^-22, exact
    for (int k = 0; k < 4; k++) {
        const short4 cx = tx->h_coef[k % S], cy = ty->h_coef[k % S];
        t.hk01[k] = (uint32_t)(unsigned short)cx.x | ((uint32_t)(unsigned short)cx.y << 16);
        t.hk23[k] = (uint32_t)(unsigned short)cx.z | ((uint32_t)(unsigned short)cx.w << 16);
        const float b[4] = {(float)cy.x * sc, (float)cy.y * sc, (float)cy.z * sc, (float)cy.w * sc};
        for (int j = 0; j < 4; j++) {
            uint32_t u;
            memcpy(&u, &b[j], 4);
            t.vb[k][j] = (unsigned long long)u | ((unsigned long long)u << 32);
        }
    }
    t.a_first = floordiv(row_begin - S / 2, S);
    t.i_last = floordiv(row_end - 1 - S / 2, S);
}

}  // namespace

int launch_yuv_int(Ctx* c, const ResizeDev& p, const ResizeArgs& a, bool* done) {
    *done = false;
    const Chroma420& ch = a.ch;
    const bool p422 = yuv422(a.order);
    const int S = a.tx->int_scale;
    if (S == 0 || a.ty->int_scale != S || ch.tx->int_scale != S || ch.ty->int_scale != S) return SRCNN_OK;
    if ((a.ow & 7) || (ch.ow & 7) || a.row_end <= a.row_begin || ch.row_end <= ch.row_begin) return SRCNN_OK;
    // stores: luma as in a grey call; chroma 8 bytes (NV12) or 2 x 4 bytes per lane and row, 8-byte aligned chroma rows for 4:2:0
    if ((((uintptr_t)p.y | p.pitch | p.plane_frame) & 7) != 0) return SRCNN_OK;
    if (p.y16 && (((uintptr_t)p.y16 | p.pitch16 | p.y16_frame) & 15) != 0) return SRCNN_OK;
    if ((((uintptr_t)ch.dst | ch.dst_pitch | ch.dst_v | ch.dst_frame) & (p422 ? 3 : 7)) != 0) return SRCNN_OK;

    IntTaps t = {}, tc = {};
    int_taps(a.tx, a.ty, S, a.row_begin, a.row_end, t);
    int_taps(ch.tx, ch.ty, S, ch.row_begin, ch.row_end, tc);
    if (p422) {   // both tile kinds read the same packed rows: 64-bit group loads when they are 8-byte aligned, 32-bit when 4-byte aligned
        const uintptr_t al = (uintptr_t)p.src | p.src_stride | p.src_frame | (uintptr_t)ch.src | ch.src_pitch;
        t.vec_ok = tc.vec_ok = (al & 7) == 0 ? 2 : ((al & 3) == 0 ? 1 : 0);
    } else {
        t.vec_ok = (((uintptr_t)p.src | p.src_stride | p.src_frame) & 3) == 0;
        tc.vec_ok = (((uintptr_t)ch.src | ch.src_pitch | ch.src_v | p.src_frame) & 3) == 0;
    }
    t.ntx = ((a.ow + kITW - 1) / kITW + 2) / 3;    // a CTA per three adjacent tiles, as in a grey call
    tc.ntx = (ch.ow + 3 * kCW - 1) / (3 * kCW);
    ChromaDev q;
    q.src = ch.src; q.src_pitch = ch.src_pitch; q.src_v = ch.src_v; q.src_frame = p.src_frame;
    q.dst = ch.dst; q.dst_pitch = ch.dst_pitch; q.dst_v = ch.dst_v; q.dst_frame = ch.dst_frame;
    q.sw = ch.sw; q.sh = ch.sh; q.ow = ch.ow; q.row_begin = ch.row_begin; q.row_end = ch.row_end;
    // indexed by a.order - SRCNN_ORDER_NV12
    static_assert(SRCNN_ORDER_I420 == SRCNN_ORDER_NV12 + 1 && SRCNN_ORDER_YUY2 == SRCNN_ORDER_NV12 + 2 &&
                  SRCNN_ORDER_UYVY == SRCNN_ORDER_NV12 + 3, "kLaunch lists the YUV orders in enum order");
    using Launch = int (*)(Ctx*, const ResizeDev&, IntTaps&, const ChromaDev&, IntTaps&, int, bool, bool*);
    static constexpr Launch kLaunch[2][4] = {
        {launch_yuv<2, SRCNN_ORDER_NV12>, launch_yuv<2, SRCNN_ORDER_I420>, launch_yuv<2, SRCNN_ORDER_YUY2>, launch_yuv<2, SRCNN_ORDER_UYVY>},
        {launch_yuv<4, SRCNN_ORDER_NV12>, launch_yuv<4, SRCNN_ORDER_I420>, launch_yuv<4, SRCNN_ORDER_YUY2>, launch_yuv<4, SRCNN_ORDER_UYVY>}};
    // a.early is false for every 4:2:0 call: it launches no merge (api.cu)
    return kLaunch[S == 4][a.order - SRCNN_ORDER_NV12](c, p, t, q, tc, std::max(1, a.nframes), a.early, done);
}

int launch_graya_int(Ctx* c, const ResizeDev& p, const ResizeArgs& a, bool* done) {
    *done = false;
    const Chroma420& ch = a.ch;
    const int S = a.tx->int_scale;
    if (S == 0 || a.ty->int_scale != S || (a.ow & 7) || a.row_end <= a.row_begin || ch.row_end <= ch.row_begin) return SRCNN_OK;
    ResizeDev pa = p;   // alpha: the same source rows, into the Cr plane (output row r at ch.dst + r * ch.dst_pitch), no FP16 copy
    pa.y = ch.dst; pa.pitch = ch.dst_pitch; pa.plane_frame = ch.dst_frame; pa.plane_row0 = 0; pa.y16 = nullptr;
    pa.row_begin = ch.row_begin; pa.row_end = ch.row_end;
    // stores: 8 bytes per lane and row into the u8 planes, 16 into the FP16 plane
    if ((((uintptr_t)p.y | p.pitch | p.plane_frame | (uintptr_t)pa.y | pa.pitch | pa.plane_frame) & 7) != 0) return SRCNN_OK;
    if (p.y16 && (((uintptr_t)p.y16 | p.pitch16 | p.y16_frame) & 15) != 0) return SRCNN_OK;

    IntTaps t = {}, ta = {};
    int_taps(a.tx, a.ty, S, a.row_begin, a.row_end, t);
    int_taps(a.tx, a.ty, S, ch.row_begin, ch.row_end, ta);
    // both tile kinds read the same rows of byte pairs: 64-bit group loads when they are 8-byte aligned, 32-bit when 4-byte aligned
    const uintptr_t al = (uintptr_t)p.src | p.src_stride | p.src_frame;
    t.vec_ok = ta.vec_ok = (al & 7) == 0 ? 2 : ((al & 3) == 0 ? 1 : 0);
    t.ntx = ta.ntx = ((a.ow + kITW - 1) / kITW + 2) / 3;   // a CTA per three adjacent tiles, as in a grey call
    const int nframes = std::max(1, a.nframes);
    return S == 2 ? launch_ga<2>(c, p, t, pa, ta, nframes, a.early, done) : launch_ga<4>(c, p, t, pa, ta, nframes, a.early, done);
}

int launch_color_bicubic_int(Ctx* c, const ResizeDev& p, const ResizeArgs& a, bool* done) {
    *done = false;
    const int S = a.tx->int_scale;
    if (S == 0 || a.ty->int_scale != S || (a.ow & 7) || a.row_end <= a.row_begin) return SRCNN_OK;
    // stores: 8 bytes per lane and row into the u8 planes, 16 into the FP16 plane
    const bool four = a.order == SRCNN_ORDER_BGRA || a.order == SRCNN_ORDER_RGBA;
    uint8_t* const pa = four ? a.pl.a : nullptr;
    if ((((uintptr_t)p.y | (uintptr_t)p.cr | (uintptr_t)p.cb | (uintptr_t)pa | p.pitch | p.plane_frame) & 7) != 0) return SRCNN_OK;
    if (p.y16 && (((uintptr_t)p.y16 | p.pitch16 | p.y16_frame) & 15) != 0) return SRCNN_OK;

    IntTaps t;
    int_taps(a.tx, a.ty, S, a.row_begin, a.row_end, t);
    // three words = bytes c0 c1 c2 of pixels 0..3; pixel word = (B, G, R, x): B is c0 for BGR input, c2 for RGB input
    if (p.swapRB) { t.sel[0] = 0x3012; t.sel[1] = 0x6345; t.sel[2] = 0x5234; t.sel[3] = 0x0123; }
    else          { t.sel[0] = 0x3210; t.sel[1] = 0x6543; t.sel[2] = 0x5432; t.sel[3] = 0x0321; }
    t.vec_ok = (((uintptr_t)p.src | p.src_stride | p.src_frame) & 3) == 0;
    if (four && t.vec_ok && (((uintptr_t)p.src | p.src_stride | p.src_frame) & 15) == 0) t.vec_ok = 2;   // 128-bit group loads
    const int nframes = std::max(1, a.nframes);
    const bool gray = a.order == SRCNN_ORDER_GRAY;
    t.ntx = (a.ow + kITW - 1) / kITW;
    if (gray) t.ntx = (t.ntx + 2) / 3;             // a CTA per three adjacent tiles
    if ((long long)t.ntx * (t.i_last - t.a_first + 1) * nframes > 0x3fffffffLL) return SRCNN_OK;
    if (gray) return S == 2 ? launch_variant<2, 1>(c, p, t, pa, nframes, false, done) : launch_variant<4, 1>(c, p, t, pa, nframes, false, done);   // never early (api.cu)
    if (four) return S == 2 ? launch_variant<2, 4>(c, p, t, pa, nframes, a.early, done) : launch_variant<4, 4>(c, p, t, pa, nframes, a.early, done);
    return S == 2 ? launch_variant<2, 3>(c, p, t, pa, nframes, a.early, done) : launch_variant<4, 3>(c, p, t, pa, nframes, a.early, done);
}

}  // namespace srcnn
