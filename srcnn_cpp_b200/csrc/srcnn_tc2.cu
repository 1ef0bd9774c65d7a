// srcnn_tc2.cu -- K-B-tc, second generation: the fused SRCNN kernel as a ROW-WALKING tcgen05 pipeline.
//
// Replaces Convolution99x11 (src/srcnn.cpp:254-325) and Convolution55 (src/srcnn.cpp:189-243) of the
// reference with ONE persistent kernel; the 64- and 32-channel activations never leave the SM.
// Operands are FP16 (Y is exact in FP16; SURVEY Appendix C), accumulators FP32 in TMEM.
//
// Mapping (B200-first, not a translation of the CPU loops):
//   * GEMM M dimension = 128 consecutive PIXELS OF ONE IMAGE ROW (one TMEM lane per pixel column).  A work
//     item is a vertical strip of 124 output columns (lanes 2..125; +-2 lanes are conv3's horizontal reach)
//     walked top to bottom, one image row per step.
//   * conv1 is a dense im2col GEMM whose A operand lives in TENSOR MEMORY as a rolling ring: for every new image
//     row each lane packs its 9 horizontal taps (Y[r][c-4..c+4], FP16) into a 5-column slot of an 11-slot ring
//     (tcgen05.st); conv1 of output row r reads the nine slots of rows r-4..r+4 -- 7 x (M128 N64 K16) MMAs with
//     A from TMEM, K = 112 (90 taps + bias + padding), against one of eleven pre-rotated weight images (which slot
//     holds which kernel row depends on r mod 11; the slot is chosen by ABSOLUTE image row, so a row's summation
//     order does not depend on how the image is cut into strips, segments or bands).  Each pixel's taps are written
//     ONCE and reused by nine rows, so conv1 executes 14 336 FLOP/px instead of the 20 480 of a Toeplitz-weight GEMM
//     off shared memory, and its A operand never touches the shared-memory port.
//   * The bias of conv1 sits in the K padding (a constant-ones ring column times hi+lo FP16 bias rows); conv2
//     borrows the same ones column for its bias MMA.  Epilogues are pure ReLU + FP16 pack.
//   * conv2 = 4+1 x (M128 N32 K16) with A = packed activations written back to TMEM in place; conv3 = "tap
//     GEMM" T[p][tap] = sum_c act2[p][c]*w3[c][tap] (2 x M128 N32 K16) followed by 25 shifted adds per pixel:
//     vertical taps accumulate in registers while the strip is walked (sliding 5-row window), horizontal taps
//     cross lanes through a small shared-memory exchange.
//   * The reference's two border clamps are reproduced exactly: conv1 reads the replicate-clamped Y (applied
//     when a row is staged), conv3 reads act2 AT THE CLAMPED PIXEL (src/srcnn.cpp:203,209) -- out-of-image taps
//     fold onto the edge row of T, the horizontal exchange clamps its lane index; never by padding Y.
//   * Warp specialisation by PHASE, not by tile: per strip pipeline four warpgroups, one thread per TMEM lane in
//     each -- the im2col ring producer, E1 (D1 -> ReLU/pack -> A1), E2 (D2 -> A2) and E3 (tap sums, exchange,
//     store).  The MMAs of a stage are issued by one elected lane of one warp of the warpgroup that produced their
//     A operand (with warp-uniform control flow a single thread issues tcgen05.mma at the tensor-pipe rate;
//     tools/microbench/mma_rate5.cu).  Three rows ("units", 64 TMEM columns each) are in flight per pipeline, two
//     pipelines per CTA share the tensor pipe.
//   * The (strip, row) steps are cut over the pipelines by cost (tc2_partition below): a pipeline's piece of one
//     strip pays for its halo rows and its drain, so pieces that cross a strip boundary get fewer rows.
//
// Executed tensor work per pixel: conv1 2*112*64 = 14 336, conv2 2*80*32 = 5 120, conv3 2*32*32 = 2 048 FLOP
// (x 128/124 for the strip halo); algorithmic 16 064 FLOP/px is what bench.py reports against the roofline.
#include <cuda_fp16.h>
#include <cstdlib>
#include <algorithm>
#include <type_traits>

#include "common.h"

namespace srcnn {
namespace tc2 {

// ---------------------------------------------------------------------------------------------
// geometry
// ---------------------------------------------------------------------------------------------
constexpr int kStripCols = 124;                   // valid output columns per strip = TMEM lanes 2..125
constexpr int kSlots = 11;                        // im2col ring: 11 image rows x 5 TMEM columns (9 taps + pad)
constexpr int kSlotCols = 5;
constexpr int kC1Chunks = 7;                      // conv1 K = 112 = 7 x 16  (56 TMEM columns)
constexpr int kOnesCol = 55;                      // ring column holding (1.0, 1.0): bias rows of conv1 / conv2
constexpr int kUnits = 3;                         // rows in flight per pipeline
constexpr int kUnitCols = 64;
constexpr int kRingOff = kUnits * kUnitCols;      // ring columns [192, 248) of the pipeline's 256
constexpr int kPipeCols = 256;

constexpr int kB1Chunk = 64 * 16 * 2;             // one [N = 64][K = 16] tile
constexpr int kB1Var = kC1Chunks * kB1Chunk;      // one rotation of the conv1 weights
constexpr int kB1Bytes = kSlots * kB1Var;         // 143 360
constexpr int kB2Bytes = 5 * 32 * 16 * 2;         // 4 K steps + bias step
constexpr int kB3Bytes = 2 * 32 * 16 * 2;
constexpr int kWeightBytes = kB1Bytes + kB2Bytes + kB3Bytes;   // 150 528
constexpr int kYRowBytes = 288;                   // staged Y row: 144 FP16 = one TMA bulk copy (the 136 tile columns start 2 or 6 in)
constexpr int kYSlots = 4;
constexpr int kHxBytes = 2 * 5 * 128 * 4;         // horizontal-tap exchange, double buffered: [buf][n][lane] fp32

constexpr int kOffW = 0;
constexpr int kImgB2 = kOffW + kB1Bytes;
constexpr int kImgB3 = kImgB2 + kB2Bytes;
constexpr int kOffY = kOffW + kWeightBytes;
constexpr int kOffHx = kOffY + 2 * kYSlots * kYRowBytes;
constexpr int kOffBar = kOffHx + 2 * kHxBytes;
constexpr int kBarsPerPipe = 13;                  // D1full[3] D2full[3] Tfull[3]: completion barriers of tcgen05.commit; Yfull[4]: staged rows (TMA)
constexpr int kCtrBytes = 32;                     // per pipeline: freed[4] (T rows consumed, one per E3 warp), c1done, pad
constexpr int kOffCtr = (kOffBar + 8 + 2 * kBarsPerPipe * 8 + 15) / 16 * 16;   // 16-byte aligned: freed[4] is read with one 128-bit load
constexpr int kOffTmem = kOffCtr + 2 * kCtrBytes;
constexpr int kOffWd = kOffTmem + 8;               // the launch's watchdog deadline (absolute %globaltimer value, u64)
constexpr int kSmemBytes = kOffTmem + 64;
constexpr int kThreads = 1024;                    // 2 pipelines x (E1, producer, E3, E2) warpgroups
constexpr int kMaxWorkers = 2 * 152;              // pipelines of one launch (B200: 148 SMs); their ranges travel in the kernel parameters
static_assert(kWeightBytes % 64 == 0 && kSmemBytes <= 227 * 1024, "shared memory budget");

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok;
}
__device__ __forceinline__ uint32_t mbar_try_wait_hint(uint32_t bar, uint32_t parity, uint32_t hint_ns) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(hint_ns)
        : "memory");
    return ok;
}
// the watchdog's failure path, out of line: seven instructions (store, fences, trap) that would otherwise sit in the middle
// of every wait loop of the row loops and cost instruction-cache lines there
__device__ __noinline__ void watchdog_die(int* guard, int code) {
    *guard = code;
    __threadfence_system();
    __trap();
}
// Bounded waits: a protocol bug must surface as an error code, never as a hung GPU.  The bound is TIME, not a poll count
// (a legitimate wait under a sanitizer, a profiler or heavy co-tenancy may take any number of polls, and a trap poisons the
// whole process's CUDA context): the launch carries a deadline -- 4 s plus 1 ms per row step of the longest pipeline,
// three orders of magnitude above the real run time; SRCNN_WATCHDOG_MS overrides it, 0 switches it off -- which thread 0
// turns into an absolute %globaltimer value in shared memory.  A wait looks at the clock every 64 Ki polls; the check is
// inline and stateless (a helper that RETURNS would make ptxas save the caller's registers around the call: stack frame,
// spills), only the failure path is out of line.
__device__ __forceinline__ void watchdog_look(uint32_t wd, int* guard, int code) {
    unsigned long long now, deadline;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(deadline) : "r"(wd));
    if (now > deadline) watchdog_die(guard, code);
}
// Plain try_wait: the hardware parks the warp until the phase completes or its own time limit passes (no issue slots
// used meanwhile).  The suspend-time-hint form compiles to a NANOSLEEP.SYNCS loop that wakes on EVERY barrier event of
// the CTA: ncu counted 18 wake-ups per wait, 28 % of all executed instructions, in the highest-priority warps.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, uint32_t wd, int* guard, int code) {
    uint32_t tries = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++tries & 0xFFFFu) == 0u) watchdog_look(wd, guard, code);
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void named_bar(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ uint32_t elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.b32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
    return pred;
}
// one arrive per WARP (barrier count 4 per warpgroup): every lane has fenced its own TMEM / shared-memory writes, the
// warp converges, one lane signals.  128 single-thread arrives per phase wake every parked waiter of the CTA 128 times.
__device__ __forceinline__ void warp_arrive(uint32_t bar, uint32_t leader) {
    __syncwarp();
    if (leader) mbar_arrive(bar);
}
// Progress counters in shared memory (release store by one lane, acquire poll by the consumer): a satisfied poll is one
// shared-memory load, a satisfied mbarrier try_wait costs ~250 cycles here.  mbarriers are kept for what only they can
// do: receiving tcgen05.commit.
__device__ __forceinline__ void ctr_publish(uint32_t addr, uint32_t v) {
    asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void ctr_wait_ge(uint32_t addr, uint32_t need, uint32_t wd, int* guard, int code) {
    uint32_t v, tries = 0;
    for (;;) {
        asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
        if ((int)(v - need) >= 0) return;
        if ((++tries & 0xFFFFu) == 0u) watchdog_look(wd, guard, code);
    }
}
__device__ __forceinline__ void ctr_wait_ge4(uint32_t addr, uint32_t need, uint32_t wd, int* guard, int code) {   // min of four counters
    uint32_t a, b, c, d, tries = 0;
    for (;;) {
        asm volatile("ld.acquire.cta.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(a), "=r"(b), "=r"(c), "=r"(d) : "r"(addr) : "memory");
        if ((int)(a - need) >= 0 && (int)(b - need) >= 0 && (int)(c - need) >= 0 && (int)(d - need) >= 0) return;
        if ((++tries & 0xFFFFu) == 0u) watchdog_look(wd, guard, code);
    }
}
// A warpgroup waits for a tcgen05.commit: ONE warp polls the mbarrier, the other three park in a hardware named barrier
// (no issue slots).  A parked try_wait returns every ~50 cycles; with all four warps of three roles polling, the polls
// were 38 % of all executed instructions.
__device__ __forceinline__ void wg_wait(uint32_t bar, uint32_t parity, bool poller, int barid, uint32_t wd, int* guard, int code) {
    if (poller) {
        mbar_wait(bar, parity, wd, guard, code);
        tc_fence_after();
        tc_fence_before();
    }
    named_bar(barid, 128);
    tc_fence_after();
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// shared-memory matrix descriptor, SWIZZLE_NONE, K-major canonical layout: 8 rows x 16 B core matrices,
// LBO = byte distance between the two K halves of a K=16 step, SBO = byte distance between 8-row groups
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
           (1ull << 46);
}
// instruction descriptor: kind::f16, A=B=FP16, D=FP32, both K-major, M=128
__host__ __device__ constexpr uint32_t idesc_f16(int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a_tmem, uint64_t b, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d),
        "r"(a_tmem), "l"(b), "r"(idesc), "r"(acc)
        : "memory");
}
// same, with the 64-bit shared-memory descriptor given as its two words: consecutive K steps of one operand image
// differ only by an add on the low word (address field), so an issue loop costs one uniform add per MMA
__device__ __forceinline__ uint32_t desc_lo(uint32_t addr, uint32_t lbo_bytes) {
    return ((addr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16);
}
__host__ __device__ constexpr uint32_t desc_hi(uint32_t sbo_bytes) { return (sbo_bytes >> 4) | (1u << 14); }
__device__ __forceinline__ void mma_ts2(uint32_t d, uint32_t a_tmem, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 bd;\n\tsetp.ne.b32 p, %5, 0;\n\tmov.b64 bd, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], bd, %4, p;\n\t}" ::"r"(d),
        "r"(a_tmem), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

#define TM_R(v, o) "=r"(v[o + 0]), "=r"(v[o + 1]), "=r"(v[o + 2]), "=r"(v[o + 3]), "=r"(v[o + 4]), "=r"(v[o + 5]), "=r"(v[o + 6]), "=r"(v[o + 7])
#define TM_W(v, o) "r"(v[o + 0]), "r"(v[o + 1]), "r"(v[o + 2]), "r"(v[o + 3]), "r"(v[o + 4]), "r"(v[o + 5]), "r"(v[o + 6]), "r"(v[o + 7])

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : TM_R(v, 0), TM_R(v, 8), TM_R(v, 16), TM_R(v, 24)
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : TM_R(v, 0), TM_R(v, 8)
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];" : TM_R(v, 0) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld1(uint32_t taddr, uint32_t& v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        TM_W(v, 0), TM_W(v, 8), TM_W(v, 16), TM_W(v, 24)
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* v) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        TM_W(v, 0), TM_W(v, 8)
        : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t* v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), TM_W(v, 0) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};" ::"r"(taddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void tmem_st1(uint32_t taddr, uint32_t a) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(a) : "memory");
}
// ReLU + round-to-nearest FP16 + pack: low half = first element (even K index)
__device__ __forceinline__ uint32_t relu_pack_f16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

// ---------------------------------------------------------------------------------------------
// kernel parameters
// ---------------------------------------------------------------------------------------------
struct Params {
    const uint8_t* y16;    // FP16 Y plane (kY16Pad replicated columns left, >= 6 right), row 0 = image row `row0`; rows [row0, row0+rows)
    size_t pitch16;        // its row pitch in BYTES (multiple of 16)
    size_t pitch;          // row pitch of the u8 chroma planes (fused merge only)
    int W, H;
    int row0, rows;
    int out_begin, out_end;  // image rows to produce
    uint8_t* out;          // Y' plane: row 0 is image row out_row0
    size_t out_pitch;
    int out_row0;
    const uint8_t* cr;     // fused merge (optional, bgr != nullptr): chroma planes, same pitch / row0 as y
    const uint8_t* cb;
    uint8_t* bgr;          // interleaved result, row out_begin first
    size_t bgr_stride;
    int swap_rb;           // 1: R,G,B byte order
    const uint8_t* wimg;   // packed FP16 operand image (kWeightBytes)
    float b3;              // conv3 bias (src/convdata.h:979), added in FP32 by the last epilogue
    int nstrips;           // strips per frame; a batch of frames is nframes x nstrips strips, frame-major
    size_t y16_frame, out_frame;   // byte distance between consecutive frames' FP16 Y planes / Y' planes
    long long total;       // frames x strips x (out_end - out_begin) row steps
    long long bounds[kMaxWorkers + 1];   // pipeline w walks row steps [bounds[w], bounds[w+1]) of the strip-major order (tc2_partition)
    int* guard;
    unsigned long long watchdog_ns;   // time allowance of this launch (0 = no deadline)
    long long* dbg;        // optional timeline (SRCNN_TC_DEBUG=1): clock64 stamps of pipeline 0 of CTA 0, first segment
};
constexpr int kDbgRows = 64, kDbgSlots = 8;
#define TL2(role_, row_, slot_)                                                                                   \
    do {                                                                                                          \
        if constexpr (DBG)                                                                                        \
            if (blockIdx.x == 0 && pipe == 0 && tp == 0 && first_seg &&  \
                (row_) >= 0 && (row_) < kDbgRows)                                                                 \
                p.dbg[(((role_) * kDbgRows) + (row_)) * kDbgSlots + (slot_)] = clock64();                        \
    } while (0)

// same, stamped by lane 0 of the role's MMA-issuing warp (warp 2 of the warpgroup in pipeline 0)
#define TL2W(role_, row_, slot_)                                                                                  \
    do {                                                                                                          \
        if constexpr (DBG)                                                                                        \
            if (blockIdx.x == 0 && pipe == 0 && tp == 64 && first_seg &&  \
                (row_) >= 0 && (row_) < kDbgRows)                                                                 \
                p.dbg[(((role_) * kDbgRows) + (row_)) * kDbgSlots + (slot_)] = clock64();                        \
    } while (0)

// a (unit, phase parity) cursor over the three units of a pipeline: one step per image row, forever
struct UnitCursor {
    uint32_t u = 0, par = 0;
    __device__ __forceinline__ void next() {
        if (++u == (uint32_t)kUnits) { u = 0; par ^= 1u; }
    }
};
__device__ __forceinline__ void st_shared_f32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ float ld_shared_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
// same for the sixteen ring-row barriers
struct RingCursor {
    uint32_t idx = 0, par = 0;
    __device__ __forceinline__ void next() {
        idx = (idx + 1u) & 15u;
        if (idx == 0u) par ^= 1u;
    }
    __device__ __forceinline__ void advance(uint32_t n) {
        const uint32_t q = idx + n;
        idx = q & 15u;
        par ^= (q >> 4) & 1u;
    }
};

// ---- E3 helpers (free functions with explicit state: the five phases of the row ring inline without spills) ----
struct E3Ctx {
    const Params& p;
    uint32_t hx_w;         // shared address of this lane's slot in exchange plane 0 of buffer 0
    uint32_t freed, bars, tml;   // freed: this warp's "T rows consumed" counter
    int tp, pipe, ta, tb, ra, rb;
    bool col_ok, first_seg, poller;
    uint32_t leader;
};
constexpr uint32_t kHxBuf = 5 * 128 * 4;   // one exchange buffer: [n][lane] fp32
// one T row: acc[k] = pending output row rho-2+k (the window slides down one row per step)
// `outp`: Y' plane (plain) or interleaved result (FUSED) pointer of the next row to store; `crp` / `cbp`: chroma (FUSED)
template <int PH, bool DBG, bool FUSED>
__device__ __forceinline__ void e3_step(const E3Ctx& c, const uint32_t (&hx_r)[5], float (&acc)[5][5], const int rho, UnitCursor& uc,
                                        uint32_t& npub, uint32_t& nfreed, uint8_t*& outp, const uint8_t*& crp, const uint8_t*& cbp) {
    constexpr int ROLE = 2;
    const Params& p = c.p;
    const int pipe = c.pipe, tp = c.tp;
    const bool first_seg = c.first_seg;
    (void)p; (void)pipe; (void)tp; (void)first_seg; (void)ROLE;
    const bool has_t = rho <= c.tb;
    uint32_t tv[25];   // the 25 taps: three loads (16 + 8 + 1 columns) instead of one 32-register block
    TL2(2, rho - c.ta, 0);
    if (has_t) {
        wg_wait(c.bars + 48 + uc.u * 8, uc.par, c.poller, 10 + pipe, c.bars + (kOffWd - kOffBar - 8) - pipe * (kBarsPerPipe * 8), p.guard, 40);   // TFULL
        TL2(2, rho - c.ta, 1);
        const uint32_t t = c.tml + uc.u * kUnitCols;
        tmem_ld16(t, tv);     // in flight while the previous row is stored
        tmem_ld8(t + 16, tv + 16);
        tmem_ld1(t + 24, tv[24]);
    }
    if (has_t) {
        tc_wait_ld();
        tc_fence_before();
        __syncwarp();
        nfreed++;
        if (c.leader) ctr_publish(c.freed, nfreed);            // the unit may be overwritten by conv1 of row +3
        TL2(2, rho - c.ta, 2);
        uc.next();
            // T[m*5+n] belongs to output row rho - (m-2): window position k = 4 - m
#pragma unroll
        for (int m = 0; m < 5; m++)
#pragma unroll
            for (int n = 0; n < 5; n++) acc[(4 - m + PH) % 5][n] += __uint_as_float(tv[m * 5 + n]);
        if (rho == 0) {        // rows -1, -2 clamp onto row 0 (src/srcnn.cpp:203)
#pragma unroll
            for (int n = 0; n < 5; n++) {
                acc[(2 + PH) % 5][n] += __uint_as_float(tv[0 * 5 + n]) + __uint_as_float(tv[1 * 5 + n]);
                acc[(3 + PH) % 5][n] += __uint_as_float(tv[0 * 5 + n]);
            }
        }
        if (rho == p.H - 1) {    // rows H, H+1 clamp onto row H-1
#pragma unroll
            for (int n = 0; n < 5; n++) {
                acc[(2 + PH) % 5][n] += __uint_as_float(tv[3 * 5 + n]) + __uint_as_float(tv[4 * 5 + n]);
                acc[(1 + PH) % 5][n] += __uint_as_float(tv[4 * 5 + n]);
            }
        }
    }
    const int r = rho - 2;
    if (r >= c.ra && r < c.rb) {       // output row r is complete: publish its five horizontal-tap partial sums
        uint32_t vcr = 128u, vcb = 128u;
        if (FUSED && c.col_ok) {       // chroma of this pixel: in flight across the exchange
            vcr = *crp;
            vcb = *cbp;
        }
        const uint32_t bo = (npub & 1u) * kHxBuf;   // two buffers alternate: one barrier per row is enough
        npub++;
#pragma unroll
        for (int n = 0; n < 5; n++) st_shared_f32(c.hx_w + bo + n * 512, acc[PH % 5][n]);
        named_bar(10 + pipe, 128);
        TL2(2, rho - c.ta, 3);
        float v[5];
#pragma unroll
        for (int n = 0; n < 5; n++) v[n] = ld_shared_f32(hx_r[n] + bo);
        float sum = v[0];
#pragma unroll
        for (int n = 1; n < 5; n++) sum += v[n];
        sum += p.b3;                                // src/srcnn.cpp:235
        int q = (int)sum;                           // :238 truncation toward zero
        q = min(max(q, 0), 255);
        if constexpr (FUSED) {
            // merge + YCrCb -> BGR (src/srcnn.cpp:637-657; OpenCV's 14-bit fixed point, SURVEY A.1) on the spot: Y' never
            // goes to memory
            if (c.col_ok) {
                const int cr = (int)vcr - 128, cb = (int)vcb - 128;
                const int B = min(max(q + ((cb * 29049 + 8192) >> 14), 0), 255);
                const int G = min(max(q + ((cb * -5636 + cr * -11698 + 8192) >> 14), 0), 255);
                const int R = min(max(q + ((cr * 22987 + 8192) >> 14), 0), 255);
                outp[0] = (uint8_t)(p.swap_rb ? R : B);
                outp[1] = (uint8_t)G;
                outp[2] = (uint8_t)(p.swap_rb ? B : R);
            }
            outp += p.bgr_stride;
            crp += p.pitch;
            cbp += p.pitch;
        } else {
            if (c.col_ok) *outp = (uint8_t)q;
            outp += p.out_pitch;
        }
    }
#pragma unroll
    for (int n = 0; n < 5; n++) acc[PH % 5][n] = 0.f;   // becomes window position 4 of the next row
    TL2(2, rho - c.ta, 4);
}

// One role's whole life: the segment loop of a pipeline.  Each role sits in its own branch of the kernel so that its
// setmaxnreg governs the register allocation of exactly its code.
//   ROLE 0: E1 (+ issues conv2)   1: im2col ring producer (+ issues conv1)   2: E3   3: E2 (+ issues conv3)
// The MMAs of a stage are issued by one elected lane of warp 0 of the warpgroup that produced their A operand.
template <int ROLE, bool DBG, bool FUSED>
__device__ __forceinline__ void role_loop(const Params& p, uint8_t* smem, const uint32_t sbase, const uint32_t wbar, const uint32_t bars,
                                          const uint32_t tm, const uint32_t tml, const uint32_t ring, const int pipe, const int tp) {
    auto D1FULL = [&](uint32_t u) { return bars + (0 + u) * 8; };
    auto D2FULL = [&](uint32_t u) { return bars + (3 + u) * 8; };
    auto TFULL = [&](uint32_t u) { return bars + (6 + u) * 8; };
    const uint32_t ctr = sbase + kOffCtr + pipe * kCtrBytes;   // freed[4] at +0, c1done at +16
    const int W = p.W, H = p.H;
    const int Hb = p.out_end - p.out_begin;
    const int wk = (int)blockIdx.x * 2 + pipe;
    long long lin = p.bounds[wk];
    const long long lin_end = p.bounds[wk + 1];
    const int segbar = 8 + pipe;     // named barrier that closes a segment (the pipeline's four warpgroups)
    bool first_seg = true;
    (void)first_seg;

    // barrier cursors run on across segments (every row / ring row arrives exactly once on its barrier)
    UnitCursor uc;                   // this role's row cursor over the pipeline's three units
    uint32_t rows_done = 0;          // conv1 issuer: rows issued so far (the first three find their unit free)
    uint32_t npub = 0;               // E3: rows published to the horizontal exchange so far
    uint32_t ycount = 0;             // producer: Y rows staged so far (slot and mbarrier phase of the TMA staging ring)
    (void)rows_done; (void)npub; (void)ycount;

    if constexpr (ROLE == 1) {   // the ring starts as finite zeros (stale TMEM bits could be NaN: 0 x NaN = NaN) + the ones column
        uint32_t z[32];
#pragma unroll
        for (int i = 0; i < 32; i++) z[i] = 0u;
        tmem_st32(tml + kRingOff, z);
        tmem_st16(tml + kRingOff + 32, z);
        tmem_st8(tml + kRingOff + 48, z);
        tc_wait_st();
        tmem_st1(tml + kRingOff + kOnesCol, 0x3C003C00u);
        tc_wait_st();
    }
    const uint32_t b1lo = desc_lo(sbase + kOffW, 1024), b2lo = desc_lo(sbase + kImgB2, 512), b3lo = desc_lo(sbase + kImgB3, 512);
    (void)b1lo; (void)b2lo; (void)b3lo;
    // one warp of the warpgroup also issues the stage's MMAs (warp-uniform).  Which one differs per role and pipeline so
    // that the six issuing warps of the CTA spread over the four SM sub-partitions (warp id mod 4) instead of all
    // landing on sub-partition 0.
    const bool warp0 = (tp >> 5) == ((ROLE == 1 ? 0 : 2) + pipe);
    const uint32_t leader = elect_one();
    const uint32_t wd = sbase + kOffWd;
    if (ROLE != 2 && warp0) mbar_wait(wbar, 0, wd, p.guard, 1);   // packed operands have landed in shared memory

    while (lin < lin_end) {
        // ---- one segment: strip `strip`, output rows [ra, rb) ----
        const int gstrip = (int)(lin / Hb);                 // strip of the whole batch
        const int rfirst = (int)(lin - (long long)gstrip * Hb);
        const int frame = gstrip / p.nstrips, strip = gstrip - frame * p.nstrips;
        (void)frame;
        const int cnt = (int)min((long long)(Hb - rfirst), lin_end - lin);
        lin += cnt;
        const int xs = strip * kStripCols;
        const int ra = p.out_begin + rfirst, rb = ra + cnt;
        const int ta = max(ra - 2, 0), tb = min(rb + 1, H - 1);   // act2 / T rows of the segment (image rows)
        const int nT = tb - ta + 1;                               // >= 1
        const int nP = nT + 8;                                    // ring rows: virtual image rows ta-4 .. tb+4
        // ring slot by ABSOLUTE image row (virtual row v -> slot (v + 11) mod 11): a row's conv1 always sees the same K
        // order, so results do not depend on how the image was cut into segments or bands
        const uint32_t slot0 = (uint32_t)((ta - 4 + kSlots) % kSlots);

        if constexpr (ROLE == 0) {
            // ================= E1(i): D1 (64 ch fp32) -> ReLU, FP16 -> A1 (32 columns, in place); then conv2(i) ==========
            for (int i = 0; i < nT; i++) {
                const uint32_t un = tml + uc.u * kUnitCols;
                TL2(0, i, 0);
                wg_wait(D1FULL(uc.u), uc.par, warp0, 3 + pipe, wd, p.guard, 20);
                rows_done++;
                if (warp0 && leader) ctr_publish(ctr + 16, rows_done);   // conv1 of rows_done rows complete: their oldest ring rows may go
                TL2(0, i, 1);
                {
                    // two 32-column loads (a tcgen05.ld round trip costs ~160 cycles whatever its width): half the loads, stores and
                    // waits of a 4 x 16-column walk, same run time
                    uint32_t v[32], w[32];
                    tmem_ld32(un, v);
                    tc_wait_ld();
#pragma unroll
                    for (int c = 0; c < 16; c++) v[c] = relu_pack_f16x2(__uint_as_float(v[2 * c]), __uint_as_float(v[2 * c + 1]));
                    tmem_ld32(un + 32, w);
                    tmem_st16(un, v);          // columns 0..15 were read by the first load (complete)
                    tc_wait_ld();
#pragma unroll
                    for (int c = 0; c < 16; c++) w[c] = relu_pack_f16x2(__uint_as_float(w[2 * c]), __uint_as_float(w[2 * c + 1]));
                    tmem_st16(un + 16, w);
                }
                tc_wait_st();
                tc_fence_before();
                TL2(0, i, 2);
                named_bar(3 + pipe, 128);   // A1 complete in all 128 lanes
                if (warp0) {   // conv2(i): D2 = A1 x W2 + b2 (the ones column of the ring carries the bias)
                    tc_fence_after();
                    TL2W(0, i, 3);
                    if (leader) {
                        const uint32_t ut = tm + uc.u * kUnitCols;
#pragma unroll
                        for (int ks = 0; ks < 4; ks++)
                            mma_ts2(ut + 32, ut + ks * 8, b2lo + ks * 64, desc_hi(128), idesc_f16(32), ks > 0);
                        mma_ts2(ut + 32, ring + 48, b2lo + 4 * 64, desc_hi(128), idesc_f16(32), 1);
                        mma_commit(D2FULL(uc.u));
                    }
                    __syncwarp();
                    TL2W(0, i, 4);
                }
                uc.next();
            }
        } else if constexpr (ROLE == 3) {
            // ================= E2(i): D2 (32 ch fp32 at [32,64)) -> A2 (16 columns at [32,48), in place); then conv3(i) ====
            for (int i = 0; i < nT; i++) {
                const uint32_t un = tml + uc.u * kUnitCols;
                TL2(3, i, 0);
                wg_wait(D2FULL(uc.u), uc.par, warp0, 5 + pipe, wd, p.guard, 21);
                TL2(3, i, 1);
                uint32_t va[32];
                tmem_ld32(un + 32, va);
                tc_wait_ld();
#pragma unroll
                for (int c = 0; c < 16; c++) va[c] = relu_pack_f16x2(__uint_as_float(va[2 * c]), __uint_as_float(va[2 * c + 1]));
                tmem_st16(un + 32, va);
                tc_wait_st();
                tc_fence_before();
                TL2(3, i, 2);
                named_bar(5 + pipe, 128);   // A2 complete in all 128 lanes
                if (warp0) {   // conv3(i) tap GEMM: T = A2 x W3
                    tc_fence_after();
                    TL2W(3, i, 3);
                    if (leader) {
                        const uint32_t ut = tm + uc.u * kUnitCols;
#pragma unroll
                        for (int ks = 0; ks < 2; ks++)
                            mma_ts2(ut, ut + 32 + ks * 8, b3lo + ks * 64, desc_hi(128), idesc_f16(32), ks > 0);
                        mma_commit(TFULL(uc.u));
                    }
                    __syncwarp();
                    TL2W(3, i, 4);
                }
                uc.next();
            }
        } else if constexpr (ROLE == 1) {
            // ================= im2col ring producer =================
            const int ybar = 1 + pipe;
            const uint32_t yst_s = sbase + kOffY + pipe * (kYSlots * kYRowBytes);
            const uint32_t ymb = bars + 9 * 8;                      // Yfull[4]: one mbarrier per staging slot
            // Y rows arrive by TMA: one cp.async.bulk of 288 bytes per ring row, straight from the FP16 plane the colour+bicubic
            // kernel wrote (replicate-padded columns, so the copy never needs a border case), issued two rows ahead by one lane of
            // a warp that does NOT issue conv1 (the issuing warp's serial chain is the pipeline's bottleneck); the same warp waits
            // for the row's bytes in front of the row barrier, so nobody else ever polls.  A strip starts at plane index
            // xs + 2 = 124 s + 2: the copy starts 2 (even strips) or 6 (odd strips) halves earlier, where the address is a
            // multiple of 16 bytes.
            const bool copier = (tp >> 5) == ((pipe + 1) & 3);
            const int odd = strip & 1;
            const uint32_t tile_off = 4u + 8u * (uint32_t)odd;      // byte offset of tile column 0 (image column xs - 6) in a staged row
            // The plane row of ring row q is clamp(clamp(ta-4+q, 0, H-1) - row0, 0, rows-1)
            auto plane_row = [&](int q) { return min(max(min(max(ta - 4 + q, 0), H - 1) - p.row0, 0), p.rows - 1); };
            const uint8_t* ysrc = p.y16 + (size_t)frame * p.y16_frame + 2 * (size_t)(xs - 4 * odd);
            const uint32_t ybase = ycount;                          // staged rows before this segment: slot and phase run on
            auto issue_row = [&](int q) {                           // one lane
                const uint32_t k = ybase + (uint32_t)q, sl = k & (kYSlots - 1);
                mbar_expect_tx(ymb + sl * 8, kYRowBytes);
                bulk_g2s(yst_s + sl * kYRowBytes, ysrc + (size_t)plane_row(q) * p.pitch16, kYRowBytes, ymb + sl * 8);
            };
            auto wait_row = [&](int q) {                            // the copier warp
                const uint32_t k = ybase + (uint32_t)q;
                mbar_wait(ymb + (k & (kYSlots - 1)) * 8, (k >> 2) & 1u, wd, p.guard, 31);
            };
            // A lane that lay beyond the image's right edge in the PREVIOUS segment (last strip of a frame) staged whatever bits the
            // FP16 plane holds past its replicated columns -- possibly NaN or Inf patterns -- and they are still in the ring.  In this
            // segment the lane may be a real column (a batch of frames: strip 0 of the next frame follows), and until a slot is
            // rewritten conv1 multiplies it by zero weights: 0 x NaN = NaN in the first two rows.  So every segment but a pipeline's
            // first starts from a finite ring, like the kernel does (the previous segment has drained: nothing reads the ring now).
            if (!first_seg) {
                uint32_t z[8];
#pragma unroll
                for (int i = 0; i < 8; i++) z[i] = 0u;
#pragma unroll
                for (int i = 0; i < 7; i++) tmem_st8(tml + kRingOff + 8 * i, z);
                tc_wait_st();
                tmem_st1(tml + kRingOff + kOnesCol, 0x3C003C00u);
                tc_wait_st();
            }
            uint32_t slot = slot0;
            uint32_t seen_f[4] = {0u, 0u, 0u, 0u}, seen_c = 0u;   // progress counters as seen one row ago
            uint32_t rot = slot0;                  // conv1 weight rotation = slot of the window's first ring row
            const uint32_t gbase = rows_done;      // global index of the segment's first row
            // One ring row per step.  A single named barrier per row says three things at once: every lane has written ring
            // row t (conv1 of row t-8 may be issued), row t+1 is staged in shared memory, and (warp 0 checked it) the slot of
            // row t+1 is no longer read by any conv1.
            auto step = [&](int t) {
                TL2(1, t, 0);
                // 9 taps of lane tp = tile columns tp .. tp+8 of the staged row
                const uint32_t rowaddr = yst_s + ((ybase + (uint32_t)t) & (kYSlots - 1)) * kYRowBytes + tile_off + ((tp >> 1) << 2);
                uint32_t w[6], o[5];
#pragma unroll
                for (int k = 0; k < 6; k++) asm volatile("ld.shared.b32 %0, [%1];" : "=r"(w[k]) : "r"(rowaddr + 4 * k));
                const uint32_t sh = (tp & 1) * 16;
#pragma unroll
                for (int k = 0; k < 5; k++) o[k] = __funnelshift_r(w[k], w[k + 1], sh);
                o[4] &= 0xFFFFu;
                TL2(1, t, 1);
                const uint32_t sl = tml + kRingOff + slot * kSlotCols;
                tmem_st4(sl, o[0], o[1], o[2], o[3]);
                tmem_st1(sl + 4, o[4]);
                if (copier) {   // row t+2 goes out (its slot held row t-2, read two row barriers ago); row t+1 must have landed
                    if (leader && t + 2 < nP) issue_row(t + 2);
                    if (t + 1 < nP) wait_row(t + 1);
                }
                TL2(1, t, 2);
                tc_wait_st();
                tc_fence_before();
                TL2(1, t, 3);
                if (warp0 && t + 1 >= kSlots) {  // row t+1 reuses the slot of row t+1-11, last read by conv1 of that row
                    // (normally the counter value read one row ago already says so: no poll on the serial chain)
                    const uint32_t need = gbase + (uint32_t)(t + 2 - kSlots);
                    if ((int)(seen_c - need) < 0) ctr_wait_ge(ctr + 16, need, wd, p.guard, 30);
                }
                TL2(1, t, 4);
                named_bar(ybar, 128);
                TL2(1, t, 5);
                if (warp0 && t >= 8) {   // conv1 of row t-8: its last ring row has just been written
                    if (rows_done >= 3u) {   // E3 has read T of row g-3 (again: usually known from last row's look)
                        const uint32_t need = rows_done - 2u;
                        if ((int)(seen_f[0] - need) < 0 || (int)(seen_f[1] - need) < 0 || (int)(seen_f[2] - need) < 0 || (int)(seen_f[3] - need) < 0)
                            ctr_wait_ge4(ctr, need, wd, p.guard, 11);
                    }
                    tc_fence_after();
                    TL2(1, t, 6);
                    if (leader) {
                        const uint32_t d = tm + uc.u * kUnitCols;
                        const uint32_t b = b1lo + rot * (kB1Var >> 4);
#pragma unroll
                        for (int ch = 0; ch < kC1Chunks; ch++)
                            mma_ts2(d, ring + ch * 8, b + ch * (kB1Chunk >> 4), desc_hi(128), idesc_f16(64), ch > 0);
                        mma_commit(D1FULL(uc.u));
                    }
                    __syncwarp();
                    TL2(1, t, 7);
                    uc.next();
                    rows_done++;
                    if (++rot == (uint32_t)kSlots) rot = 0;
                }
                if (warp0) {   // a look at both counters for the NEXT row; the loads are consumed a whole row later.
                    // Relaxed loads: an acquire load makes the warp wait for the value on the spot (ncu: the two waits were a fifth of
                    // the issuing warp's time, and that warp's chain paces the pipeline).  A stale value only sends the next row into
                    // the acquire poll; a fresh one is followed by a control dependency, the row's named barrier and a tcgen05 fence
                    // before anything is overwritten.
                    asm volatile("ld.relaxed.cta.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(seen_f[0]), "=r"(seen_f[1]), "=r"(seen_f[2]), "=r"(seen_f[3]) : "r"(ctr) : "memory");
                    asm volatile("ld.relaxed.cta.shared.u32 %0, [%1];" : "=r"(seen_c) : "r"(ctr + 16) : "memory");
                }
                if (++slot == (uint32_t)kSlots) slot = 0;
            };
            if (copier) {
                if (leader) {
                    issue_row(0);
                    if (nP > 1) issue_row(1);
                }
                wait_row(0);
            }
            named_bar(ybar, 128);   // row 0 staged
            for (int t = 0; t < nP; t++) step(t);
            ycount += (uint32_t)nP;
        } else {
            // ================= E3: conv3 tap sums =================
            const uint32_t hx_s = sbase + kOffHx + pipe * kHxBytes;
            const int x = xs - 2 + tp;                         // image column of this lane
            uint32_t hx_r[5];                                  // exchange slots of the lanes holding act2 at clamp(x + n - 2)  (src/srcnn.cpp:209)
#pragma unroll
            for (int n = 0; n < 5; n++) hx_r[n] = hx_s + n * 512 + 4 * min(max(min(max(x + n - 2, 0), W - 1) - (xs - 2), 0), 127);
            const bool col_ok = (tp >= 2) && (tp <= 125) && (x < W);
            float acc[5][5];                                   // ring of pending output rows x horizontal tap n
#pragma unroll
            for (int k = 0; k < 5; k++)
#pragma unroll
                for (int n = 0; n < 5; n++) acc[k][n] = 0.f;
            // rows are stored in order ra, ra+1, ...
            uint8_t* outp = FUSED ? p.bgr + (size_t)(ra - p.out_begin) * p.bgr_stride + (size_t)3 * (col_ok ? x : 0)
                                  : p.out + (size_t)frame * p.out_frame + (size_t)(ra - p.out_row0) * p.out_pitch + x;
            const uint8_t* crp = FUSED ? p.cr + (size_t)(ra - p.row0) * p.pitch + (col_ok ? x : 0) : nullptr;
            const uint8_t* cbp = FUSED ? p.cb + (size_t)(ra - p.row0) * p.pitch + (col_ok ? x : 0) : nullptr;
            E3Ctx cx{p, hx_s + 4 * tp, ctr + 4 * (uint32_t)(tp >> 5), bars, tml, tp, pipe, ta, tb, ra, rb, col_ok, first_seg, warp0, leader};
            const int last = rb + 1;
            int rho = ta;
            for (; rho + 4 <= last; rho += 5) {   // five rows per trip: the ring position is a compile-time constant
                e3_step<0, DBG, FUSED>(cx, hx_r, acc, rho, uc, npub, rows_done, outp, crp, cbp);
                e3_step<1, DBG, FUSED>(cx, hx_r, acc, rho + 1, uc, npub, rows_done, outp, crp, cbp);
                e3_step<2, DBG, FUSED>(cx, hx_r, acc, rho + 2, uc, npub, rows_done, outp, crp, cbp);
                e3_step<3, DBG, FUSED>(cx, hx_r, acc, rho + 3, uc, npub, rows_done, outp, crp, cbp);
                e3_step<4, DBG, FUSED>(cx, hx_r, acc, rho + 4, uc, npub, rows_done, outp, crp, cbp);
            }
            if (rho <= last) e3_step<0, DBG, FUSED>(cx, hx_r, acc, rho++, uc, npub, rows_done, outp, crp, cbp);
            if (rho <= last) e3_step<1, DBG, FUSED>(cx, hx_r, acc, rho++, uc, npub, rows_done, outp, crp, cbp);
            if (rho <= last) e3_step<2, DBG, FUSED>(cx, hx_r, acc, rho++, uc, npub, rows_done, outp, crp, cbp);
            if (rho <= last) e3_step<3, DBG, FUSED>(cx, hx_r, acc, rho++, uc, npub, rows_done, outp, crp, cbp);
        }
        first_seg = false;
        named_bar(segbar, 4 * 128);   // segment drained: every MMA waited for, ring and units reusable from scratch
    }
}

// ---------------------------------------------------------------------------------------------
// the kernel: 32 warps = 8 warpgroups, one thread per TMEM lane in each.
//   warpgroups 0,1 : E2 of pipeline 0,1        (D2 -> A2; warp 0 issues conv3)
//   warpgroups 2,3 : E1                        (D1 -> ReLU + FP16 pack -> A1; warp 0 issues conv2)
//   warpgroups 4,5 : E3                        (tap sums, horizontal exchange, bias, truncate, clamp, store)
//   warpgroups 6,7 : im2col ring producer      (warp 0 issues conv1)
// ---------------------------------------------------------------------------------------------
template <bool DBG, bool FUSED>
__global__ void __launch_bounds__(kThreads, 1) k_srcnn_tc2(const Params p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // provably warp-uniform: a shuffled value, so ptxas keeps the role branches and the MMA issue paths uniform
    const int wg = warp >> 2;
    // the warp scheduler prefers the highest warp id: the role with the longest serial chain per row gets the highest
    // warpgroups.  wg 0,1: E2 (3)   wg 2,3: E1 (0)   wg 4,5: E3 (2)   wg 6,7: producer + conv1 issue (1)
    const int role = (0x1203 >> ((wg >> 1) * 4)) & 0xF;
    const int pipe = wg & 1;
    const int tp = tid & 127;                                  // TMEM lane = pixel column xs - 2 + tp
    const int quarter = warp & 3;
    // the shared-window base as an opaque, provably uniform register value: left to itself the compiler rematerialises
    // it (S2UR SR_CgaCtaId + ULEA + ...) in front of every barrier / shared-memory access of the row loops
    uint32_t sbase = smem_u32(smem);
    asm volatile("mov.u32 %0, %0;" : "+r"(sbase));
    sbase = __shfl_sync(0xffffffffu, sbase, 0);
    const uint32_t wbar = sbase + kOffBar;
    const uint32_t bars = sbase + kOffBar + 8 + pipe * (kBarsPerPipe * 8);
    volatile uint32_t* tmem_slot = (volatile uint32_t*)(smem + kOffTmem);

    if (tid < 16) reinterpret_cast<volatile uint32_t*>(smem + kOffCtr)[tid] = 0u;   // progress counters
    if (tid == 0) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        const unsigned long long deadline = p.watchdog_ns ? now + p.watchdog_ns : ~0ull;
        asm volatile("st.shared.u64 [%0], %1;" ::"r"(sbase + kOffWd), "l"(deadline) : "memory");
        mbar_init(wbar, 1);
        for (int q = 0; q < 2; q++)
            for (int i = 0; i < kBarsPerPipe; i++)
                mbar_init(sbase + kOffBar + 8 + (q * kBarsPerPipe + i) * 8, 1);   // one tcgen05.commit per phase
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(smem_u32((const void*)tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (tid == 0) {  // weights: one TMA bulk fetch per CTA, shared by both pipelines
        mbar_expect_tx(wbar, kWeightBytes);
        constexpr int kPiece = kWeightBytes / 4;
        static_assert(kPiece % 16 == 0, "bulk copy granularity");
        for (int i = 0; i < 4; i++) bulk_g2s(sbase + kOffW + i * kPiece, p.wimg + i * kPiece, kPiece, wbar);
    }
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tm = tmem_base + pipe * kPipeCols;                   // this pipeline's columns
    const uint32_t tml = tm + ((uint32_t)(quarter * 32) << 16);         // + this warp's lane quarter
    const uint32_t ring = tm + kRingOff;

    // register budget (65 536 at launch = 1024 x 64): producer 48, E2 56, E1 72, E3 80
    if (role == 1) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 48;");
        role_loop<1, DBG, FUSED>(p, smem, sbase, wbar, bars, tm, tml, ring, pipe, tp);
    } else if (role == 3) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
        role_loop<3, DBG, FUSED>(p, smem, sbase, wbar, bars, tm, tml, ring, pipe, tp);
    } else if (role == 0) {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 72;");
        role_loop<0, DBG, FUSED>(p, smem, sbase, wbar, bars, tm, tml, ring, pipe, tp);
    } else {
        asm volatile("setmaxnreg.inc.sync.aligned.u32 80;");
        role_loop<2, DBG, FUSED>(p, smem, sbase, wbar, bars, tm, tml, ring, pipe, tp);
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

}  // namespace tc2

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static inline void put_h2(uint8_t* img, size_t byte_off, float v) {
    const __half h = __float2half_rn(v);
    memcpy(img + byte_off, &h, 2);
}

// Packs the FP32 parameters into the FP16 operand images the kernel's UMMA descriptors expect
// (SWIZZLE_NONE, K-major: element (n,k) of a [N][16] tile at (k/8)*(N*16) + n*16 + (k%8)*2 bytes).  Pure host code:
// `img` (tc2_weight_bytes() bytes) is written in full; tests decode it through srcnn_debug_tc2_weights.
void tc2_pack_weights(const float* P, uint8_t* img) {
    using namespace tc2;
    memset(img, 0, kWeightBytes);
    const float* w1 = P + kOffW1;
    const float* w2 = P + kOffW2;
    const float* w3 = P + kOffW3;
    auto hi_lo = [](float b, float& hi, float& lo) {
        hi = __half2float(__float2half_rn(b));
        lo = b - hi;
    };
    // conv1, eleven rotations: with the window's first image row in ring slot v, slot s holds kernel row
    // j = (s - v) mod 11 (j > 8: a row outside the 9x9 window -> zero weights).  K index k = 10*s + tap
    // (tap 9 = the slot's padding half), k = 110/111 = the ones column -> hi/lo halves of the bias.
    for (int v = 0; v < kSlots; v++)
        for (int n = 0; n < 64; n++) {
            for (int k = 0; k < 16 * kC1Chunks; k++) {
                float val = 0.f;
                if (k < 10 * kSlots) {
                    const int s = k / 10, tap = k % 10;
                    const int j = (s - v + kSlots) % kSlots;
                    if (j <= 8 && tap <= 8) val = w1[(n * 9 + j) * 9 + tap];
                } else if (k == 2 * kOnesCol || k == 2 * kOnesCol + 1) {
                    float hi, lo;
                    hi_lo(P[kOffB1 + n], hi, lo);
                    val = (k == 2 * kOnesCol) ? hi : lo;
                }
                const int ch = k / 16, kk = k % 16;
                put_h2(img, (size_t)v * kB1Var + (size_t)ch * kB1Chunk + (size_t)(kk / 8) * 1024 + (size_t)n * 16 + (kk % 8) * 2, val);
            }
        }
    for (int ks = 0; ks < 4; ks++)  // conv2: B[n = out ch][k = in ch ks*16+k]
        for (int n = 0; n < 32; n++)
            for (int k = 0; k < 16; k++)
                put_h2(img, kImgB2 + (size_t)ks * 1024 + (size_t)(k / 8) * 512 + (size_t)n * 16 + (k % 8) * 2,
                       w2[n * 64 + ks * 16 + k]);
    for (int n = 0; n < 32; n++) {  // conv2 bias step: A = ring columns 48..55, the ones column is K index 4,5 of it
        float hi, lo;
        hi_lo(P[kOffB2 + n], hi, lo);
        const int k0 = 2 * (kOnesCol - 48);
        put_h2(img, kImgB2 + 4 * 1024 + (size_t)(k0 / 8) * 512 + (size_t)n * 16 + (k0 % 8) * 2, hi);
        put_h2(img, kImgB2 + 4 * 1024 + (size_t)((k0 + 1) / 8) * 512 + (size_t)n * 16 + ((k0 + 1) % 8) * 2, lo);
    }
    for (int ks = 0; ks < 2; ks++)  // conv3 tap GEMM: B[n = tap m*5+n][k = in ch]
        for (int n = 0; n < 32; n++)
            for (int k = 0; k < 16; k++)
                put_h2(img, kImgB3 + (size_t)ks * 1024 + (size_t)(k / 8) * 512 + (size_t)n * 16 + (k % 8) * 2,
                       n < 25 ? w3[(ks * 16 + k) * 25 + n] : 0.f);
}

size_t tc2_weight_bytes() { return tc2::kWeightBytes; }

int tc2_prepare_weights(Ctx* c, const float* P) {
    using namespace tc2;
    std::vector<uint8_t> img(kWeightBytes);
    tc2_pack_weights(P, img.data());
    SRCNN_CUDA(c, cudaMalloc(&c->d_tc2_weights, kWeightBytes));
    // pageable source: the runtime has staged `img` when this returns; srcnn_create synchronises the device afterwards
    SRCNN_CUDA(c, cudaMemcpyAsync(c->d_tc2_weights, img.data(), kWeightBytes, cudaMemcpyHostToDevice, c->stream));
    SRCNN_CUDA(c, cudaStreamSynchronize(c->stream));
    c->b3 = P[kOffB3];
    SRCNN_CUDA(c, cudaFuncSetAttribute(tc2::k_srcnn_tc2<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    SRCNN_CUDA(c, cudaFuncSetAttribute(tc2::k_srcnn_tc2<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    SRCNN_CUDA(c, cudaFuncSetAttribute(tc2::k_srcnn_tc2<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    return SRCNN_OK;
}

void tc2_release(Ctx* c) {
    if (c->d_tc2_weights) cudaFree(c->d_tc2_weights);
    c->d_tc2_weights = nullptr;
}

// Cuts the strip-major sequence of row steps (nstrips strips x hb rows) into `nworkers` contiguous ranges of about equal
// COST.  A worker's piece of one strip (a "segment") costs its rows plus `ovh` row steps: eight ring rows and four halo
// rows of conv1..conv3 are recomputed at the top and bottom of every segment, and the pipeline drains at its end.  Cutting
// into equal ROW counts instead (ovh = 0) leaves every worker whose range crosses a strip boundary with two segments and
// the whole launch waiting for them.  The smallest feasible budget per worker is found by bisection; results do not depend
// on the cut (a row's arithmetic is independent of its segment: tests/test_stage_parity.py).
void tc2_partition(int nstrips, int hb, int nworkers, int ovh, long long* bounds) {
    const long long total = (long long)nstrips * hb;
    if (ovh <= 0) {
        for (int w = 0; w <= nworkers; w++) bounds[w] = total * w / nworkers;
        return;
    }
    const int min_seg = 8;   // a shorter piece is not worth a segment of its own unless it finishes the strip
    auto walk = [&](long long budget, long long* out) {
        long long pos = 0;
        for (int w = 0; w < nworkers; w++) {
            if (out) out[w] = pos;
            long long left = budget;
            while (pos < total) {
                const long long in_strip = hb - pos % hb;
                const long long can = left - ovh;
                if (can < std::min<long long>(min_seg, in_strip)) break;
                const long long take = std::min(can, in_strip);
                pos += take;
                left -= take + ovh;
            }
        }
        if (out) out[nworkers] = total;
        return pos >= total;
    };
    long long lo = (total + nworkers - 1) / nworkers + ovh - 1, hi = lo + 1;   // lo: infeasible or unknown, hi: feasible
    while (!walk(hi, nullptr)) { lo = hi; hi += std::max<long long>(1, hi / 8); }
    while (hi - lo > 1) {
        const long long mid = lo + (hi - lo) / 2;
        if (walk(mid, nullptr)) hi = mid; else lo = mid;
    }
    walk(hi, bounds);
    // the last worker took what was left; anything the greedy walk could not place (never happens for a feasible budget)
    // would show as bounds[nworkers] < total, which the walk above rules out
}

int launch_cnn_tc2(Ctx* c, const CnnArgs& a0) {
    using namespace tc2;
    if (a0.out_end <= a0.out_begin) return SRCNN_OK;
    CnnArgs a = a0;
    if (!a.y16) {   // a caller's u8 plane (stage API): the kernel's TMA staging wants the padded FP16 form
        a.pitch16 = y16_pitch_bytes(a.W);
        int rc = ensure(c, c->y16_buf, a.pitch16 * (size_t)a.rows + 512);
        if (rc) return rc;
        rc = launch_y8_to_y16(c, a.y, a.pitch, a.W, a.rows, (uint8_t*)c->y16_buf.p, a.pitch16);
        if (rc) return rc;
        a.y16 = (const uint8_t*)c->y16_buf.p;
    }
    Params p;
    p.y16 = (const uint8_t*)a.y16; p.pitch16 = a.pitch16; p.pitch = a.pitch;
    p.W = a.W; p.H = a.H;
    p.row0 = a.row0; p.rows = a.rows;
    p.out_begin = a.out_begin; p.out_end = a.out_end;
    p.out = a.out; p.out_pitch = a.out_pitch; p.out_row0 = a.out_row0;
    p.cr = a.cr; p.cb = a.cb;
    p.bgr = a.bgr; p.bgr_stride = a.bgr_stride;
    p.swap_rb = a.order == SRCNN_ORDER_RGB ? 1 : 0;
    p.wimg = (const uint8_t*)c->d_tc2_weights;
    p.b3 = c->b3;
    const int nframes = std::max(1, a.nframes);
    if (nframes > 1 && a.bgr) return fail(c, SRCNN_E_ARG, "fused merge does not take a batch of frames");
    const int nstrips1 = (a.W + kStripCols - 1) / kStripCols;
    const int nstrips = nstrips1 * nframes;
    p.nstrips = nstrips1;
    p.y16_frame = a.y16_frame_stride; p.out_frame = a.out_frame_stride;
    p.total = (long long)nstrips * (a.out_end - a.out_begin);
    p.guard = c->d_guard;
    p.dbg = nullptr;
    if (getenv("SRCNN_TC_DEBUG")) {
        const size_t bytes = 4 * kDbgRows * kDbgSlots * sizeof(long long);
        int rc = ensure(c, c->work_buf, bytes);
        if (rc) return rc;
        cudaMemsetAsync(c->work_buf.p, 0, bytes, c->stream);
        p.dbg = (long long*)c->work_buf.p;
    }
    // one persistent CTA per SM; fewer when the image is too small to give every pipeline ~48 row steps
    long long want = (p.total + 95) / 96;
    int grid = (int)std::min<long long>(std::min(c->sm_count, kMaxWorkers / 2), std::max<long long>(1, want));
    {   // the pipelines' ranges (cached: frames of a stream and bands of a frame repeat the same geometry)
        const int hb = a.out_end - a.out_begin;
        Tc2Partition& pt = c->tc2_part;
        if (pt.nstrips != nstrips || pt.hb != hb || pt.nworkers != 2 * grid || pt.ovh != c->tc2_seg_ovh) {
            pt.bounds.resize(kMaxWorkers + 1);
            tc2_partition(nstrips, hb, 2 * grid, c->tc2_seg_ovh, pt.bounds.data());
            pt.nstrips = nstrips; pt.hb = hb; pt.nworkers = 2 * grid; pt.ovh = c->tc2_seg_ovh;
        }
        memcpy(p.bounds, pt.bounds.data(), sizeof(long long) * (2 * grid + 1));
    }
    {   // watchdog allowance: 4 s + 1 ms per row step of the longest pipeline (a row step takes ~0.6 us)
        const long long longest = (p.total + 2 * grid - 1) / (2 * grid) + 64;
        p.watchdog_ns = 4000000000ull + 1000000ull * (unsigned long long)longest;
        if (const char* e = getenv("SRCNN_WATCHDOG_MS")) p.watchdog_ns = 1000000ull * (unsigned long long)std::max(0ll, atoll(e));
    }
    if (p.bgr) k_srcnn_tc2<false, true><<<grid, kThreads, kSmemBytes, c->stream>>>(p);
    else if (p.dbg) k_srcnn_tc2<true, false><<<grid, kThreads, kSmemBytes, c->stream>>>(p);
    else k_srcnn_tc2<false, false><<<grid, kThreads, kSmemBytes, c->stream>>>(p);
    c->launches++;
    SRCNN_CUDA(c, cudaGetLastError());
    return SRCNN_OK;
}

}  // namespace srcnn

// debug hook: copies the last launch's timeline (4 roles x 64 rows x 8 stamps) to the host
extern "C" __attribute__((visibility("default"))) int srcnn_debug_tc2_timeline(srcnn_ctx* c, long long* out) {
    if (!c || !c->work_buf.p) return SRCNN_E_ARG;
    srcnn::DeviceScope scope(c->device);
    cudaStreamSynchronize(c->stream);
    const size_t bytes = 4 * srcnn::tc2::kDbgRows * srcnn::tc2::kDbgSlots * sizeof(long long);
    return cudaMemcpy(out, c->work_buf.p, bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? SRCNN_OK : SRCNN_E_CUDA;
}
