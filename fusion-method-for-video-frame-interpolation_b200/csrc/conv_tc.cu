// conv_tc.cu -- implicit-GEMM 2-D convolution on the 5th-gen tensor cores (tcgen05 + TMEM), fp32 in / fp32 out,
// split-operand error-compensated so the result matches an fp32 FFMA convolution to ~1e-6 relative.
//
// Two operand splits (same kernel, template PREC; same shared-memory bytes per MMA, so the descriptors are identical):
//   PREC_F16X3  (default)  a = a_hi + a_lo with a_hi = fp16(a * 2^s), a_lo = fp16(a * 2^s - a_hi): 11 + 11 mantissa
//                          bits, products exact in the fp32 accumulator; tcgen05.mma.kind::f16 runs at TWICE the
//                          kind::tf32 rate and moves 16 instead of 8 channels per 32-byte K step.  Power-of-two scales
//                          (activations 2^4, weights per layer so that max|w| lands in [2^14, 2^15)) keep both halves
//                          in fp16's normal range; the epilogue multiplies by the exact inverse.  |a| * 2^4 > 65504 sets
//                          an overflow flag the host checks (fvfi_conv2d_overflow_count) -- no silent saturation.
//   PREC_TF32X3            a_hi = rna_tf32(a), a_lo = a - a_hi: the same 11 + 11 bits without any range limit.
//
// Used for the PhaseNet / KernelEstimation / FusionNet convolutions (the only dense contractions on the path;
// reference: torch.nn.Conv2d -> cuDNN, src/phase_net/phase_net.py:190-199, src/fusion_net/fusion_adacofnet.py:19-83,
// src/fusion_net/fusion_net.py:24-36).  A single reduced-precision product (TF32: 10-bit mantissa) does not hold the 1e-4 output
// bound through ~30 layers, so every product a*b is formed as a_lo*b_hi + a_hi*b_lo + a_hi*b_hi from the hi/lo halves of the chosen
// split (default: fp16 halves, tcgen05.mma.kind::f16; PREC_TF32X3: tf32 halves, kind::tf32), three MMAs per K-step accumulating in
// fp32 in TMEM; the dropped a_lo*b_lo term is 2^-22 relative.
//
// Formulation (stride 1, "same" padding, zero or reflect):
//   activations NHWC (torch channels_last), GEMM M = output pixels, N = Cout, K = taps x Cin.
//   A CTA owns an output patch of 16 rows x (8*MT) columns = MT accumulator tiles of M = 128 (16 rows x 8 px),
//   each tile N columns of TMEM.  Per 16-channel chunk the loader warps stage the (16+KH-1) x (8*MT+KW-1) input
//   region ONCE, split into hi/lo, in the no-swizzle K-major canonical layout [kchunk(16B)][pixel][16B]; every
//   filter tap is then just a different descriptor start address into that region (SBO = region row pitch), so
//   the activation is read from L2 once per chunk instead of once per tap.  Weights are pre-packed on the device
//   (hi|lo, canonical layout) and streamed per (chunk, tap) with cp.async.bulk + mbarrier.
//   Warp roles (one per warpgroup, registers split with setmaxnreg): warps 0-7 activation loaders, warps 8-11 epilogue
//   (TMEM -> regs -> bias/activation -> NHWC / planar), warp 12 weight producer, warp 13 TMEM allocator + MMA issuer.
#include <cuda_fp16.h>

#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <mutex>
#include <type_traits>

#include "common.cuh"

namespace fvfi {

constexpr int CV_KCHUNKS = 4;           // 16-byte K chunks per stage = two MMA K steps of 32 bytes
constexpr int CV_UMAX = 12;             // (pixel, K chunk) items a loader thread keeps in flight: a whole K chunk of the tile
constexpr int CV_HDR = 32;              // floats of header in front of the packed weights (scales, precision)
constexpr int CV_X_SHIFT = 4;           // PREC_F16X3: activations are scaled by 2^4 before the fp16 split
constexpr int CV_ROWS = 16;             // output rows per CTA
constexpr int CV_LOADER_WARPS = 8;      // warps 0-7 (two warpgroups): activation loaders
constexpr int CV_LOADERS = 32 * CV_LOADER_WARPS;
constexpr int CV_EPI_WARPS = 4;         // warps 8-11 (one warpgroup): epilogue, warp w owns TMEM lanes 32*(w % 4) .. +31
constexpr int CV_EPI_THREADS = 32 * CV_EPI_WARPS;
constexpr int CV_PRODUCER_WARP = CV_LOADER_WARPS + CV_EPI_WARPS;      // warp 12: weight producer
constexpr int CV_MMA_WARP = CV_PRODUCER_WARP + 1;                     // warp 13: TMEM allocator + MMA issuer; 14, 15 fill the warpgroup
constexpr int CV_THREADS = CV_LOADERS + CV_EPI_THREADS + 128;
// Register budget per role (setmaxnreg, per warpgroup): the launch gives every thread 65536 / 512 = 128; the epilogue and
// producer/MMA warpgroups hand most of theirs to the loaders, which keep a whole K chunk of a tile in flight in registers.
constexpr int CV_REGS_LOADER = 152, CV_REGS_EPI = 144, CV_REGS_MISC = 56;
constexpr int CV_REGS_LAUNCH = 65536 / CV_THREADS;      // what __launch_bounds__(CV_THREADS, 1) gives every thread
static_assert(CV_LOADERS * CV_REGS_LOADER + CV_EPI_THREADS * CV_REGS_EPI + 128 * CV_REGS_MISC <= 65536, "register pool");
constexpr int CV_MAX_ASTAGES = 4;
constexpr int CV_MAX_BSTAGES = 4;
constexpr unsigned CV_SPIN_LIMIT = 200u * 1000u * 1000u;   // bounded waits: trap instead of hanging the GPU

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_ELU = 2, ACT_TANH = 3, ACT_SIGMOID = 4, ACT_SOFTMAX = 5 };   // softmax over channels
enum { PAD_ZERO = 0, PAD_REFLECT = 1 };
enum { PREC_TF32X3 = 0, PREC_F16X3 = 1 };
__host__ __device__ constexpr int cv_cpk(int prec) { return prec == PREC_F16X3 ? 8 : 4; }        // channels per 16-byte K chunk
__host__ __device__ constexpr int cv_chunk(int prec) { return CV_KCHUNKS * cv_cpk(prec); }        // channels per stage

struct ConvArgs {
    const float* x;        // [B,H,W,Cin] NHWC
    const float* wpack;    // packed weights (see pack kernel), behind the CV_HDR-float header
    const float* hdr;      // header of the packed weights: [0] = output scale (exact inverse of the operand scales)
    int* overflow;         // PREC_F16X3: set to 1 when a scaled activation leaves fp16's range
    const float* bias;     // [Npad] or null
    float* y;              // [B,H,W,Cout] NHWC
    int B, H, W, Cin, Cout, Npad, KH, KW, pad_mode, act;
    int ldx, ldy;          // floats per pixel in the input / output storage (channel-slice views)
    int out_nchw;          // 1: y is planar [B,Cout,H,W] (coefficient maps for the warp kernel)
    int cout_store;        // NHWC channels written per pixel: Cout, or round16(Cout) with the padding zero-filled
    int MT, RW, RH, NPIX;  // tiles per CTA, staged region geometry
    int KCS;               // 16-byte units between the K chunks of an A stage: NPIX rounded up to 2 (mod 8), see the host side
    int nchunks, last_ksteps, astages, bstages, tmem_cols;
    int wide, tcols;       // WIDE MMA pairing (Npad <= 32); TMEM columns per accumulator tile (Npad or 2*Npad)
    int nacc;              // TMEM accumulator buffers (2 when they fit: epilogue of tile j-1 overlaps the MMAs of tile j)
    int tiles_x, tiles_y, ntiles;
    unsigned a_stage_bytes, b_stage_bytes;
    const float* res;      // optional residual [B,H,W,>=Cout] NHWC added AFTER the activation (U-Net skip connections), or null
    int ldr;               // floats per pixel of the residual
    // fused bilinear upsampling of the input (torch.nn.Upsample -> Conv2d as ONE kernel): x is [B,Hs,Ws,Cin], the convolution runs
    // on its [H,W] bilinear resampling, which the loaders evaluate while staging -- the upsampled tensor never exists in HBM
    int up, Hs, Ws, up_align;
    float up_sy, up_sx;
    // ... optionally only for the first up_chunks K chunks (channels [0, up_chunks * chunk)): the remaining input channels come from a
    // second tensor x2 [B,H,W,>=Cin - up_chunks*chunk] at the convolution's own resolution -- conv(cat(resize(x), x2)) without the concat
    // (PhaseNet: previous level's features resampled + this level's values, src/phase_net/phase_net.py:138-148)
    const float* x2;
    int ldx2, up_chunks;
};

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    const unsigned addr = smem_u32(bar);
    unsigned done = 0, spins = 0;
    while (true) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) break;
        if (++spins > CV_SPIN_LIMIT) __trap();
    }
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// Called by ALL lanes of the (converged) MMA warp; one elected lane issues.  Keeping the control flow warp-uniform
// lets the compiler keep descriptors in uniform registers instead of R2UR-ing per instruction.
__device__ __forceinline__ void tc_commit(unsigned long long* bar) {
    asm volatile(
        "{\n\t.reg .pred pe;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(unsigned d_tmem, unsigned long long adesc, unsigned long long bdesc,
                                            unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, pe;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// One K=8 step of one filter tap for MT accumulator tiles, 3xTF32: per tile  D += A_lo*B_hi ; D += A_hi*B_lo ; D += A_hi*B_hi.
// A single asm block: the tensor core consumes an MMA of N <= 128 every 40-64 cycles, which one warp can only sustain
// if the issue stream is ~3 instructions per MMA (measured: a C++ loop with per-MMA descriptor arithmetic and elect
// costs ~120 cycles per MMA).  Tile t: A descriptor + 8*t (eight pixels = 8 x 16 B), TMEM columns + t*Npad.
// %4 = B_hi descriptor, %5 = B_lo descriptor, %6 = instruction descriptor (N = Npad), %8 = instruction descriptor with
// N = 2*Npad.  WIDE (Npad <= 32): the packed weights hold [B_hi; B_lo] as one 2*Npad-row operand, so  A_hi x [B_hi; B_lo]
// is ONE MMA writing two accumulators (columns [0,Npad) and [Npad,2Npad), summed by the epilogue) and A_lo x B_hi a second
// one: two instead of three reads of the 4 KB A tile, which is what bounds an SS-mode MMA with N <= 64.
// The second and third product of a step share their A operand (A_hi): the second MMA keeps it in the tensor core's A collector
// buffer (collector::a::fill, SASS .A_KEEP), the third takes it from there (collector::a::lastuse, .A_REUSE) -- two instead of
// three shared-memory reads of the 4 KB A tile per step, the traffic that bounds the N = 64 layers.
#define FVFI_MMA3(KIND, D, AL, AH)                                                                            \
    "@pe tcgen05.mma.cta_group::1.kind::" KIND " [" D "], " AL ", %4, %6, pa;\n\t"                            \
    "@pe tcgen05.mma.cta_group::1.kind::" KIND ".collector::a::fill [" D "], " AH ", %5, %6, pt;\n\t"         \
    "@pe tcgen05.mma.cta_group::1.kind::" KIND ".collector::a::lastuse [" D "], " AH ", %4, %6, pt;\n\t"
#define FVFI_MMA2W(KIND, D, AL, AH)                                                       \
    "@pe tcgen05.mma.cta_group::1.kind::" KIND " [" D "], " AH ", %4, %8, pa;\n\t"        \
    "@pe tcgen05.mma.cta_group::1.kind::" KIND " [" D "], " AL ", %4, %6, pt;\n\t"
#define FVFI_KSTEP_BODY(KIND, MM)                                                                                      \
    if (MT == 1) {                                                                                                     \
        asm volatile(                                                                                                  \
            "{\n\t.reg .pred pe, pa, pt;\n\t"                                                                          \
            "elect.sync _|pe, 0xffffffff;\n\tsetp.ne.b32 pa, %7, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"                       \
            MM(KIND, "%0", "%2", "%3") "}"                                                                             \
            ::"r"(d), "r"(np), "l"(al), "l"(ah), "l"(bh), "l"(bl), "r"(idesc), "r"(acc), "r"(idesc2) : "memory");     \
    } else if (MT == 2) {                                                                                              \
        asm volatile(                                                                                                  \
            "{\n\t.reg .pred pe, pa, pt;\n\t.reg .b64 al1, ah1;\n\t.reg .b32 d1;\n\t"                                  \
            "elect.sync _|pe, 0xffffffff;\n\tsetp.ne.b32 pa, %7, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"                       \
            "add.u64 al1, %2, 8;\n\tadd.u64 ah1, %3, 8;\n\tadd.u32 d1, %0, %1;\n\t"                                    \
            MM(KIND, "%0", "%2", "%3") MM(KIND, "d1", "al1", "ah1") "}"                                                \
            ::"r"(d), "r"(np), "l"(al), "l"(ah), "l"(bh), "l"(bl), "r"(idesc), "r"(acc), "r"(idesc2) : "memory");     \
    } else {                                                                                                           \
        asm volatile(                                                                                                  \
            "{\n\t.reg .pred pe, pa, pt;\n\t.reg .b64 al1, ah1, al2, ah2, al3, ah3;\n\t.reg .b32 d1, d2, d3;\n\t"      \
            "elect.sync _|pe, 0xffffffff;\n\tsetp.ne.b32 pa, %7, 0;\n\tsetp.eq.b32 pt, 0, 0;\n\t"                       \
            "add.u64 al1, %2, 8;\n\tadd.u64 ah1, %3, 8;\n\tadd.u32 d1, %0, %1;\n\t"                                    \
            "add.u64 al2, %2, 16;\n\tadd.u64 ah2, %3, 16;\n\tadd.u32 d2, d1, %1;\n\t"                                  \
            "add.u64 al3, %2, 24;\n\tadd.u64 ah3, %3, 24;\n\tadd.u32 d3, d2, %1;\n\t"                                  \
            MM(KIND, "%0", "%2", "%3") MM(KIND, "d1", "al1", "ah1") MM(KIND, "d2", "al2", "ah2")                       \
            MM(KIND, "d3", "al3", "ah3") "}"                                                                           \
            ::"r"(d), "r"(np), "l"(al), "l"(ah), "l"(bh), "l"(bl), "r"(idesc), "r"(acc), "r"(idesc2) : "memory");     \
    }
// np = TMEM columns per accumulator tile (Npad, or 2*Npad when WIDE)
template <int MT, int PREC, bool WIDE>
__device__ __forceinline__ void tc_mma_kstep(unsigned d, unsigned np, unsigned long long al, unsigned long long ah,
                                             unsigned long long bh, unsigned long long bl, unsigned idesc, unsigned acc,
                                             unsigned idesc2) {
    if (PREC == PREC_F16X3) {
        if (WIDE) { FVFI_KSTEP_BODY("f16", FVFI_MMA2W) } else { FVFI_KSTEP_BODY("f16", FVFI_MMA3) }
    } else {
        if (WIDE) { FVFI_KSTEP_BODY("tf32", FVFI_MMA2W) } else { FVFI_KSTEP_BODY("tf32", FVFI_MMA3) }
    }
}
__device__ __forceinline__ void tc_ld16_issue(unsigned taddr, unsigned* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_ld16(unsigned taddr, float* v) {
    unsigned r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// K-major, SWIZZLE_NONE shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start >> 4 | [16,30) LBO >> 4 (between the two 16 B K-chunks of one MMA) |
//   [32,46) SBO >> 4 (between 8-row core matrices along M/N) | [46,48) version = 1 | [61,64) layout = 0
__device__ __forceinline__ unsigned long long make_desc(unsigned saddr, unsigned lbo_bytes, unsigned sbo_bytes) {
    unsigned long long d = 0;
    d |= (unsigned long long)((saddr >> 4) & 0x3fffu);
    d |= (unsigned long long)((lbo_bytes >> 4) & 0x3fffu) << 16;
    d |= (unsigned long long)((sbo_bytes >> 4) & 0x3fffu) << 32;
    d |= 1ull << 46;
    return d;
}

// 256-bit global accesses (sm_100: LDG.E.256 / STG.E.256): one full 32-byte sector per lane and instruction
__device__ __forceinline__ void ldg256(const float* p, float* v) {
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p));
}
__device__ __forceinline__ void stg256(float* p, const float* v) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}

__device__ __forceinline__ float to_tf32_rna(float x) {
    unsigned r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// Activations of the epilogue.  exp is the hardware ex2 path (__expf, relative error 2^-21): the absolute error of the
// results below is <= 1e-6, an order below the convolution's own rounding; inputs are clamped where exp would overflow.
__device__ __forceinline__ float fast_tanh(float v) {
    const float t = __expf(2.f * fminf(fmaxf(v, -15.f), 15.f));
    return __fdividef(t - 1.f, t + 1.f);
}
__device__ __forceinline__ float fast_sigmoid(float v) { return __fdividef(1.f, 1.f + __expf(-fmaxf(v, -80.f))); }
template <int ACT>
__device__ __forceinline__ float apply_act(float v) {
    switch (ACT) {
        case ACT_RELU: return fmaxf(v, 0.f);
        case ACT_ELU: return v > 0.f ? v : __expf(v) - 1.f;
        case ACT_TANH: return fast_tanh(v);
        case ACT_SIGMOID: return fast_sigmoid(v);
        default: return v;
    }
}

__device__ __forceinline__ int reflect101(int i, int n) {   // torch 'reflect': -1 -> 1, n -> n-2
    if (n == 1) return 0;
    const int period = 2 * (n - 1);
    int m = i % period;
    if (m < 0) m += period;
    return m < n ? m : period - m;
}

// ---- weight packing: OIHW fp32 -> header + [chunk][tap][kc(4)][hi|lo][n(Npad)][16 bytes] --------------------------
// header[0] = output scale (exact inverse of the operand scales), [1] = weight scale, [2] = precision.
__global__ void conv_weight_scale_kernel(const float* __restrict__ w, size_t count, float* __restrict__ hdr, int prec) {
    __shared__ float red[32];
    float m = 0.f;
    if (prec == PREC_F16X3) {                           // 3xTF32 needs no scale (its header is constant)
        size_t i = threadIdx.x;
        float m1 = 0.f, m2 = 0.f, m3 = 0.f;             // four loads in flight per thread
        for (; i + 3 * (size_t)blockDim.x < count; i += 4 * (size_t)blockDim.x) {
            m = fmaxf(m, fabsf(__ldg(w + i)));
            m1 = fmaxf(m1, fabsf(__ldg(w + i + blockDim.x)));
            m2 = fmaxf(m2, fabsf(__ldg(w + i + 2 * (size_t)blockDim.x)));
            m3 = fmaxf(m3, fabsf(__ldg(w + i + 3 * (size_t)blockDim.x)));
        }
        for (; i < count; i += blockDim.x) m = fmaxf(m, fabsf(__ldg(w + i)));
        m = fmaxf(fmaxf(m, m1), fmaxf(m2, m3));
    }
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < (int)(blockDim.x >> 5); ++i) m = fmaxf(m, red[i]);
        float wscale = 1.f, oscale = 1.f;
        if (prec == PREC_F16X3) {
            int e = 0;                                  // 2^e: max|w| * 2^e in [2^14, 2^15)
            if (m > 0.f && isfinite(m)) { int ex; frexpf(m, &ex); e = 15 - ex; }
            e = max(-40, min(40, e));
            wscale = ldexpf(1.f, e);
            oscale = ldexpf(1.f, -e - CV_X_SHIFT);
        }
        hdr[0] = oscale;
        hdr[1] = wscale;
        hdr[2] = (float)prec;
    }
}

template <int PREC>
__global__ void conv_pack_weights_kernel(const float* __restrict__ w, float* __restrict__ packed, int Cout, int Cin, int KH,
                                         int KW, int Npad, int nchunks) {
    constexpr int CPK = cv_cpk(PREC);
    const int taps = KH * KW;
    const float wscale = packed[1];
    float* out32 = packed + CV_HDR;
    __half* out16 = (__half*)(packed + CV_HDR);
    const size_t total = (size_t)nchunks * taps * 2 * CV_KCHUNKS * Npad * CPK;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < total; q += (size_t)gridDim.x * blockDim.x) {
        size_t t = q;
        const int e = (int)(t % CPK); t /= CPK;
        const int n = (int)(t % Npad); t /= Npad;
        const int lo = (int)(t % 2); t /= 2;                  // [B_hi rows; B_lo rows] form one 2*Npad-row operand per K chunk
        const int kc = (int)(t % CV_KCHUNKS); t /= CV_KCHUNKS;
        const int tap = (int)(t % taps); t /= taps;
        const int chunk = (int)t;
        const int c = chunk * (CV_KCHUNKS * CPK) + kc * CPK + e;
        float v = 0.f;
        if (n < Cout && c < Cin) v = w[(((size_t)n * Cin + c) * KH + tap / KW) * KW + tap % KW];
        if (PREC == PREC_F16X3) {
            v *= wscale;
            const __half hi = __float2half_rn(v);
            out16[q] = lo ? __float2half_rn(v - __half2float(hi)) : hi;
        } else {
            unsigned hb;
            asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(hb) : "f"(v));
            const float hi = __uint_as_float(hb);
            out32[q] = lo ? (v - hi) : hi;
        }
    }
}

// ---- the convolution ---------------------------------------------------------------------------------
// Persistent, warp-specialised: one CTA per SM walks the output tiles (tile = blockIdx.x + j * gridDim.x).  The A / B
// shared-memory rings and the (double-buffered) TMEM accumulator keep running across tile boundaries, so the loaders
// fetch tile j+1 while the tensor core works on tile j and the epilogue drains tile j-1.
struct TileCoord { int img, y0, x0; };
__device__ __forceinline__ TileCoord tile_coord(const ConvArgs& A, int tile) {
    TileCoord t;
    const int bx = tile % A.tiles_x, r = tile / A.tiles_x;
    t.x0 = bx * 8 * A.MT;
    t.y0 = (r % A.tiles_y) * CV_ROWS;
    t.img = r / A.tiles_y;
    return t;
}

template <int ACT, int PREC>
__global__ void __launch_bounds__(CV_THREADS, 1) conv_split_kernel(const ConvArgs A) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // layout: [A stages: hi, lo] [B stages] [barriers] [tmem ptr] [pixoff] [bias]
    unsigned char* a_base = smem_raw;
    unsigned char* b_base = a_base + (size_t)A.astages * A.a_stage_bytes;
    unsigned long long* bars = (unsigned long long*)(b_base + (size_t)A.bstages * A.b_stage_bytes);
    unsigned long long* a_full = bars;                                          // [astages] count CV_LOADERS
    unsigned long long* a_empty = bars + CV_MAX_ASTAGES;                        // [astages] count 1 (tcgen05.commit)
    unsigned long long* b_full = bars + 2 * CV_MAX_ASTAGES;                     // [bstages] count 1 + tx
    unsigned long long* b_empty = b_full + CV_MAX_BSTAGES;                      // [bstages] count 1 (tcgen05.commit)
    unsigned long long* acc_full = b_empty + CV_MAX_BSTAGES;                    // [2] count 1 (tcgen05.commit)
    unsigned long long* acc_empty = acc_full + 2;                               // [2] count CV_EPI_THREADS
    unsigned* tmem_ptr = (unsigned*)(acc_empty + 2);
    int* pixoff = (int*)(tmem_ptr + 2);                      // [NPIX] global pixel index of every region pixel, -1 = zero pad
    float* bias_s = (float*)(((size_t)(pixoff + A.NPIX) + 15) & ~(size_t)15);   // [Npad], 16 B aligned
    float2* up_w = (float2*)(bias_s + 256);                  // [NPIX] upsampling loaders: weights of the second source row / column
    int* up_d = (int*)(up_w + A.NPIX);                       // [NPIX] ... and the offsets of the second source row / column
    int* up_off = up_d + A.NPIX;                             // [NPIX] ... and the first source sample (pixoff stays the direct mapping)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int taps = A.KH * A.KW;
    const unsigned a_half = A.a_stage_bytes / 2;             // hi | lo halves of an A stage
    const int nacc = A.nacc;
    const unsigned acc_cols = (unsigned)(A.MT * A.tcols);

    if (threadIdx.x == 0) {
        for (int s = 0; s < A.astages; ++s) { mbar_init(&a_full[s], CV_LOADERS); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < A.bstages; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], CV_EPI_THREADS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int n = threadIdx.x; n < A.Npad; n += CV_THREADS) bias_s[n] = (A.bias && n < A.Cout) ? __ldg(A.bias + n) : 0.f;
    if (warp == CV_MMA_WARP) {   // TMEM allocation by one warp
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(A.tmem_cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem = *tmem_ptr;

    if (warp >= CV_LOADER_WARPS && warp < CV_PRODUCER_WARP) {
        // ================= epilogue warpgroup: TMEM -> registers -> bias/activation -> global =================
        // Dedicated warps (the loaders used to run the epilogue between their two load phases: on the small-N full-resolution
        // layers, where a tile's MMAs take ~6k cycles, the loader path -- epilogue included -- took ~14k and the tensor
        // pipe idled 54 % of the time, profiles/r01_conv_head_summary.txt).
        if (CV_REGS_EPI > CV_REGS_LAUNCH) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(CV_REGS_EPI));
        else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(CV_REGS_EPI));
        const float oscale = __ldg(A.hdr);                         // exact power of two (1 for PREC_TF32X3)
        const bool vec_out = (A.cout_store & 3) == 0 && (A.ldy & 3) == 0 && ((((size_t)A.y) & 15) == 0);
        const bool vec_out8 = (A.cout_store & 7) == 0 && (A.ldy & 7) == 0 && ((((size_t)A.y) & 31) == 0);
        const size_t plane = (size_t)A.H * A.W;
        const int quarter = warp & 3;                              // a warp reads TMEM lanes 32*(warp % 4) .. +31
        const int m = quarter * 32 + lane;                         // accumulator row = TMEM lane
        const bool res_vec = A.res && (A.Cout & 15) == 0 && (A.ldr & 7) == 0 && ((((size_t)A.res) & 31) == 0);

        // ---- epilogue of tile number jt (coordinates T): TMEM -> registers -> bias/activation -> global
        auto epilogue = [&](int jt, const TileCoord& T) {
            const int buf = jt % nacc, use = jt / nacc;
            mbar_wait(&acc_full[buf], use & 1);
            tc_fence_after();
            const int orow = T.y0 + (m >> 3);
            const unsigned tq = tmem + ((unsigned)(quarter * 32) << 16) + (unsigned)buf * acc_cols;
            // bias + activation + store of one 16-column block of accumulator tile t (smax / sinv: softmax only)
            // 16 accumulator columns of this thread's row; WIDE: the two partial accumulators (A_hi B_hi + A_lo B_hi, A_hi B_lo)
            auto ld_acc16 = [&](unsigned taddr, float* v) {
                unsigned r0[16], r1[16];
                tc_ld16_issue(taddr, r0);
                if (A.wide) tc_ld16_issue(taddr + (unsigned)A.Npad, r1);
                tc_ld_wait();
#pragma unroll
                for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r0[i]) + (A.wide ? __uint_as_float(r1[i]) : 0.f);
            };
            // softmax epilogue: same, sequential loads (32 instead of 48 live registers next to the loads in flight)
            auto ld_acc16s = [&](unsigned taddr, float* v) {
                tc_ld16(taddr, v);
                if (A.wide) {
                    float w[16];
                    tc_ld16(taddr + (unsigned)A.Npad, w);
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] += w[i];
                }
            };
            // store of one 16-column block of finished values of accumulator tile t
            auto store16 = [&](int t, int n0, const float* v) {
                const int ocol = T.x0 + t * 8 + (m & 7);
                if (!(orow < A.H && ocol < A.W)) return;
                float* dst = A.out_nchw ? A.y + (size_t)T.img * A.Cout * plane + (size_t)orow * A.W + ocol
                                        : A.y + (((size_t)T.img * A.H + orow) * A.W + ocol) * A.ldy;
                if (A.out_nchw) {
                    // 8 consecutive px per row: full 32 B sectors.  Running pointer + one compare per plane (the indexed form
                    // cost a 64-bit multiply-add per store: 12 instructions per STG, 15 % of the head layers' stall samples).
                    // Measured alternative: staging the tile in shared memory and leaving through TMA tensor stores (single- and
                    // double-buffered) was SLOWER (1.20-1.24 vs 1.10 ms per head layer): with the stores removed altogether the
                    // layer still takes 0.96 ms -- the operand reads of its MMAs (0.72 ms), not these stores, bound it.
                    float* d = dst + (size_t)n0 * plane;
                    const int nv = A.Cout - n0;
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        if (i < nv) *d = v[i];
                        d += plane;
                    }
                } else if (vec_out8) {
#pragma unroll
                    for (int i = 0; i < 16; i += 8)
                        if (n0 + i < A.cout_store) stg256(dst + n0 + i, v + i);
                } else if (vec_out) {
#pragma unroll
                    for (int i = 0; i < 16; i += 4)
                        if (n0 + i < A.cout_store) *(float4*)(dst + n0 + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i)
                        if (n0 + i < A.cout_store) dst[n0 + i] = v[i];
                }
            };
            auto emit = [&](int t, int n0, const float* r, float smax, float sinv) {
                float v[16];
#pragma unroll
                for (int i = 0; i < 16; i += 4) {
                    const float4 b4 = *(const float4*)(bias_s + n0 + i);        // smem broadcast
                    const float z0 = fmaf(r[i], oscale, b4.x), z1 = fmaf(r[i + 1], oscale, b4.y);
                    const float z2 = fmaf(r[i + 2], oscale, b4.z), z3 = fmaf(r[i + 3], oscale, b4.w);
                    if (ACT == ACT_SOFTMAX) {
                        v[i] = __expf(z0 - smax) * sinv; v[i + 1] = __expf(z1 - smax) * sinv;
                        v[i + 2] = __expf(z2 - smax) * sinv; v[i + 3] = __expf(z3 - smax) * sinv;
                    } else {
                        v[i] = apply_act<ACT>(z0); v[i + 1] = apply_act<ACT>(z1);
                        v[i + 2] = apply_act<ACT>(z2); v[i + 3] = apply_act<ACT>(z3);
                    }
                }
                if (ACT != ACT_SOFTMAX && A.res) {
                    // skip connection fused into the epilogue:  y = act(conv(x)) + residual   (fusion_adacofnet.py:128-138: d5 + c5 ...)
                    const int ocol = T.x0 + t * 8 + (m & 7);
                    if (orow < A.H && ocol < A.W) {
                        const float* rp = A.res + (((size_t)T.img * A.H + orow) * A.W + ocol) * A.ldr + n0;
                        if (res_vec) {
                            float q[16];
                            ldg256(rp, q);
                            ldg256(rp + 8, q + 8);
#pragma unroll
                            for (int i = 0; i < 16; ++i) v[i] += q[i];
                        } else {
#pragma unroll
                            for (int i = 0; i < 16; ++i)
                                if (n0 + i < A.Cout) v[i] += __ldg(rp + i);
                        }
                    }
                }
                store16(t, n0, v);
            };
            if (ACT == ACT_SOFTMAX) {
                for (int t = 0; t < A.MT; ++t) {
                    const unsigned tbase = tq + (unsigned)(t * A.tcols);
                    if (A.Npad <= 32) {
                        // the AdaCoF weight heads (25 channels), 16 live values at a time: statistics of columns 16.., then
                        // columns 0..15 finished and stored, then columns 16.. again -- three TMEM reads and two exps per
                        // channel pair instead of four reads and three exps per channel of the general two-pass form
                        float z[16];
                        float m2 = -INFINITY, s2 = 0.f;
                        if (A.Npad > 16) {
                            ld_acc16s(tbase + 16, z);
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                z[i] = (16 + i < A.Cout) ? fmaf(z[i], oscale, bias_s[16 + i]) : -INFINITY;
                                m2 = fmaxf(m2, z[i]);
                            }
#pragma unroll
                            for (int i = 0; i < 16; ++i) s2 += __expf(z[i] - m2);     // exp(-inf) = 0 for the padding
                        }
                        ld_acc16s(tbase, z);
                        float m1 = -INFINITY, s1 = 0.f;
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            z[i] = (i < A.Cout) ? fmaf(z[i], oscale, bias_s[i]) : -INFINITY;
                            m1 = fmaxf(m1, z[i]);
                        }
                        const float smax = fmaxf(m1, m2);
#pragma unroll
                        for (int i = 0; i < 16; ++i) { z[i] = __expf(z[i] - smax); s1 += z[i]; }
                        const float sinv = 1.f / (s1 + (A.Npad > 16 ? s2 * __expf(m2 - smax) : 0.f));
#pragma unroll
                        for (int i = 0; i < 16; ++i) z[i] *= sinv;
                        store16(t, 0, z);
                        if (A.Npad > 16) {
                            ld_acc16s(tbase + 16, z);
                            emit(t, 16, z, smax, sinv);
                        }
                        continue;
                    }
                    float smax = -INFINITY, ssum = 0.f;
                    for (int n0 = 0; n0 < A.Npad; n0 += 16) {          // pass 1 over TMEM: channel max and sum(exp)
                        float v[16];
                        ld_acc16s(tbase + n0, v);
#pragma unroll
                        for (int i = 0; i < 16; ++i)
                            if (n0 + i < A.Cout) {
                                const float z = fmaf(v[i], oscale, bias_s[n0 + i]);
                                if (z > smax) { ssum = ssum * __expf(smax - z); smax = z; }
                                ssum += __expf(z - smax);
                            }
                    }
                    const float sinv = 1.f / ssum;
                    for (int n0 = 0; n0 < A.Npad; n0 += 16) {
                        float r[16];
                        ld_acc16s(tbase + n0, r);
                        emit(t, n0, r, smax, sinv);
                    }
                }
            } else {
                // 16-column blocks (t, n0) of the CTA tile in order, software-pipelined: the TMEM loads of block k+1 are in
                // flight while block k is activated and stored (two register sets; tcgen05.wait::ld covers every load issued
                // so far, hence wait -> issue next -> emit)
                const int nblk = A.MT * (A.Npad >> 4);
                int t_i = 0, n_i = 0, t_e = 0, n_e = 0;                                     // issue / emit cursors
                auto adv = [&](int& t, int& n0) { n0 += 16; if (n0 >= A.Npad) { n0 = 0; ++t; } };
                auto issue_at = [&](unsigned* x, unsigned* y) {
                    const unsigned ta = tq + (unsigned)(t_i * A.tcols + n_i);
                    tc_ld16_issue(ta, x);
                    if (A.wide) tc_ld16_issue(ta + (unsigned)A.Npad, y);
                    adv(t_i, n_i);
                };
                auto emit_at = [&](const unsigned* x, const unsigned* y) {
                    float v[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(x[i]) + (A.wide ? __uint_as_float(y[i]) : 0.f);
                    emit(t_e, n_e, v, 0.f, 1.f);
                    adv(t_e, n_e);
                };
                unsigned a0[16], a1[16], b0[16], b1[16];
                issue_at(a0, a1);
                for (int k = 0; k < nblk; k += 2) {
                    tc_ld_wait();
                    if (k + 1 < nblk) issue_at(b0, b1);
                    emit_at(a0, a1);
                    if (k + 1 < nblk) {
                        tc_ld_wait();
                        if (k + 2 < nblk) issue_at(a0, a1);
                        emit_at(b0, b1);
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(&acc_empty[buf]);          // this thread's TMEM reads of the buffer are done
        };

        {
            int j = 0;
            for (int tile = blockIdx.x; tile < A.ntiles; tile += gridDim.x, ++j) epilogue(j, tile_coord(A, tile));
        }
    } else if (warp < CV_LOADER_WARPS) {
        // ================= activation loaders (region -> hi/lo canonical tiles) =================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(CV_REGS_LOADER));
        const int padT = A.KH / 2, padL = A.KW / 2;
        // 16-byte loads need aligned pixels; a channel count that is not a multiple of 4 is fine when the pixel stride
        // leaves room for the rounded-up group (the producer zero-fills the padding channels, see out layout 2)
        constexpr int CPK = cv_cpk(PREC);
        constexpr int CHUNK = cv_chunk(PREC);
        // the source the plain (issue / finish) path reads: x, or -- behind the upsampled channels -- x2
        const int cshift = A.up ? A.up_chunks * CHUNK : 0;                       // first channel of that source in the weights' order
        const float* xd = (A.up && A.x2) ? A.x2 : A.x;
        const int ldd = (A.up && A.x2) ? A.ldx2 : A.ldx, cind = A.Cin - cshift;
        const int cin4 = (cind + 3) & ~3;
        const bool vec = ((ldd & 3) == 0) && (ldd >= cin4) && ((((size_t)xd) & 15) == 0);
        const int cin8 = (cind + 7) & ~7;
        const bool vec8 = ((ldd & 7) == 0) && (ldd >= cin8) && ((((size_t)xd) & 31) == 0);
        const int cin4u = A.up ? ((min(A.Cin, cshift) + 3) & ~3) : 0;            // channels of the upsampled source
        const float xs = (float)(1 << CV_X_SHIFT);
        float amax = 0.f;
        int g = 0;                                                 // running chunk counter of the A ring

        // ---- one K chunk = two phases.  issue(): ALL of this thread's 16-byte global loads of the chunk go out at once
        // (up to UMAX items of CPK channels stay in registers); finish(): split into hi/lo, store into the A ring.
        constexpr int UMAX = CV_UMAX;                              // NPIX * 4 <= CV_LOADERS * UMAX (checked on the host)
        float v[UMAX][CPK];
        auto chunk_shape = [&](int c, int& ksh) {
            // the last chunk may need only the first MMA K step: K chunks 0,1 are stored first, so just stop early
            ksh = (c == A.nchunks - 1 && A.last_ksteps == 1) ? 1 : 2;            // log2(K chunks to fill)
            return A.NPIX << ksh;
        };
        auto issue = [&](int c, const float* X) {
            int ksh;
            const int total = chunk_shape(c, ksh);
            const int kmask = (1 << ksh) - 1, cbase = c * CHUNK - cshift;
#pragma unroll
            for (int u = 0; u < UMAX; ++u) {
                const int q = threadIdx.x + u * CV_LOADERS;
#pragma unroll
                for (int e = 0; e < CPK; ++e) v[u][e] = 0.f;
                if (q < total) {
                    const int pix = q >> ksh, ch = cbase + (q & kmask) * CPK;   // consecutive threads read one pixel's chunk
                    const int off = pixoff[pix];
                    if (off >= 0 && ch < cin4) {
                        const float* p = X + (size_t)off * ldd + ch;
                        if (vec8 && CPK == 8 && ch + 8 <= cin8) {
                            ldg256(p, v[u]);
                        } else if (vec) {
#pragma unroll
                            for (int e = 0; e < CPK; e += 4) {
                                if (ch + e < cin4) {
                                    const float4 t = __ldg((const float4*)(p + e));
                                    v[u][e] = t.x; v[u][e + 1] = t.y; v[u][e + 2] = t.z; v[u][e + 3] = t.w;
                                }
                            }
                        } else {
#pragma unroll
                            for (int e = 0; e < CPK; ++e)
                                if (ch + e < cind) v[u][e] = __ldg(p + e);
                        }
                    }
                }
            }
        };
        auto finish = [&](int c) {
            const int s = g % A.astages;
            if (g >= A.astages) mbar_wait(&a_empty[s], ((g / A.astages) - 1) & 1);
            ++g;
            float4* hi = (float4*)(a_base + (size_t)s * A.a_stage_bytes);
            float4* lo = (float4*)(a_base + (size_t)s * A.a_stage_bytes + a_half);
            int ksh;
            const int total = chunk_shape(c, ksh);
            const int kmask = (1 << ksh) - 1;
#pragma unroll
            for (int u = 0; u < UMAX; ++u) {
                const int q = threadIdx.x + u * CV_LOADERS;
                if (q < total) {
                    const int o = (q & kmask) * A.KCS + (q >> ksh);
                    if (PREC == PREC_F16X3) {
                        unsigned hw[4], lw[4];
#pragma unroll
                        for (int e = 0; e < 8; e += 2) {
                            const float x0 = v[u][e] * xs, x1 = v[u][e + 1] * xs;
                            amax = fmaxf(amax, fmaxf(fabsf(x0), fabsf(x1)));
                            const __half2 h = __floats2half2_rn(x0, x1);
                            const float2 hf = __half22float2(h);
                            const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
                            hw[e >> 1] = *(const unsigned*)&h;
                            lw[e >> 1] = *(const unsigned*)&l;
                        }
                        hi[o] = make_float4(__uint_as_float(hw[0]), __uint_as_float(hw[1]), __uint_as_float(hw[2]), __uint_as_float(hw[3]));
                        lo[o] = make_float4(__uint_as_float(lw[0]), __uint_as_float(lw[1]), __uint_as_float(lw[2]), __uint_as_float(lw[3]));
                    } else {
                        float4 h;
                        h.x = to_tf32_rna(v[u][0]); h.y = to_tf32_rna(v[u][1]); h.z = to_tf32_rna(v[u][2]); h.w = to_tf32_rna(v[u][3]);
                        hi[o] = h;
                        lo[o] = make_float4(v[u][0] - h.x, v[u][1] - h.y, v[u][2] - h.z, v[u][3] - h.w);
                    }
                }
            }
            fence_async_smem();          // generic-proxy stores -> visible to the tensor-core (async) proxy
            mbar_arrive(&a_full[s]);
        };
        // Upsampling loaders: one item = TWO horizontally adjacent region pixels x one channel group.  The second pixel's sources are
        // the first one's (same source column pair) or share a column with them (its left column is the first one's right column) --
        // 4 or 6 loads per pair instead of 8: the staging is bound by L1 bandwidth (every source sample is wanted by ~4 region pixels),
        // not by latency.  Values are combined with bilerp (the resize kernel's own arithmetic), split and stored at once.
        auto load_cpk = [&](const float* p, float* dst) {
            if (CPK == 8) {
                ldg256(p, dst);
            } else {
                const float4 t = __ldg((const float4*)p);
                dst[0] = t.x; dst[1] = t.y; dst[2] = t.z; dst[3] = t.w;
            }
        };
        auto stage_up = [&](int c, const float* X) {
            const int s = g % A.astages;
            if (g >= A.astages) mbar_wait(&a_empty[s], ((g / A.astages) - 1) & 1);
            ++g;
            float4* hi = (float4*)(a_base + (size_t)s * A.a_stage_bytes);
            float4* lo = (float4*)(a_base + (size_t)s * A.a_stage_bytes + a_half);
            int ksh;
            const int total = chunk_shape(c, ksh) >> 1;             // pixel pairs x channel groups (RW is even: pairs do not straddle rows)
            const int kmask = (1 << ksh) - 1, cbase = c * CHUNK;
            auto put = [&](int o, const float* w) {
                if (PREC == PREC_F16X3) {
                    unsigned hw[4], lw[4];
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {
                        const float x0 = w[e] * xs, x1 = w[e + 1] * xs;
                        amax = fmaxf(amax, fmaxf(fabsf(x0), fabsf(x1)));
                        const __half2 h = __floats2half2_rn(x0, x1);
                        const float2 hf = __half22float2(h);
                        const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
                        hw[e >> 1] = *(const unsigned*)&h;
                        lw[e >> 1] = *(const unsigned*)&l;
                    }
                    hi[o] = make_float4(__uint_as_float(hw[0]), __uint_as_float(hw[1]), __uint_as_float(hw[2]), __uint_as_float(hw[3]));
                    lo[o] = make_float4(__uint_as_float(lw[0]), __uint_as_float(lw[1]), __uint_as_float(lw[2]), __uint_as_float(lw[3]));
                } else {
                    float4 h;
                    h.x = to_tf32_rna(w[0]); h.y = to_tf32_rna(w[1]); h.z = to_tf32_rna(w[2]); h.w = to_tf32_rna(w[3]);
                    hi[o] = h;
                    lo[o] = make_float4(w[0] - h.x, w[1] - h.y, w[2] - h.z, w[3] - h.w);
                }
            };
            for (int q = threadIdx.x; q < total; q += CV_LOADERS) {
                const int pix = (q >> ksh) << 1, kg = q & kmask, ch = cbase + kg * CPK;
                float a0[CPK], b0[CPK], c0[CPK], d0[CPK], a1[CPK], b1[CPK], c1[CPK], d1[CPK];
#pragma unroll
                for (int e = 0; e < CPK; ++e) a0[e] = b0[e] = c0[e] = d0[e] = a1[e] = b1[e] = c1[e] = d1[e] = 0.f;
                const bool chok = ch < cin4u;
                const int off0 = chok ? up_off[pix] : -1, off1 = chok ? up_off[pix + 1] : -1;
                const int e0 = up_d[pix], e1 = up_d[pix + 1];
                const float2 w0 = up_w[pix], w1 = up_w[pix + 1];
                // 0: all four sources of the second pixel are the first one's; 1: its left column is the first one's right column;
                // 2: unrelated (image border / padding)
                const int kind = (off0 >= 0 && off1 == off0 && e1 == e0) ? 0
                               : (off0 >= 0 && off1 == off0 + (e0 & 1) && (e1 >> 1) == (e0 >> 1)) ? 1 : 2;
                if (off0 >= 0) {
                    const float* p = X + (size_t)off0 * A.ldx + ch;
                    const size_t dx = (size_t)(e0 & 1) * A.ldx, dy = (size_t)(e0 >> 1) * A.ldx;
                    load_cpk(p, a0); load_cpk(p + dx, b0); load_cpk(p + dy, c0); load_cpk(p + dy + dx, d0);
                }
                if (off1 >= 0 && kind != 0) {
                    const float* p = X + (size_t)off1 * A.ldx + ch;
                    const size_t dx = (size_t)(e1 & 1) * A.ldx, dy = (size_t)(e1 >> 1) * A.ldx;
                    if (kind == 2) { load_cpk(p, a1); load_cpk(p + dy, c1); }
                    load_cpk(p + dx, b1); load_cpk(p + dy + dx, d1);
                }
                float w[CPK];
                {
                    const float ly = w0.x, lx = w0.y, hy = 1.f - ly, hx = 1.f - lx;
#pragma unroll
                    for (int e = 0; e < CPK; ++e) w[e] = bilerp(hy, hx, ly, lx, a0[e], b0[e], c0[e], d0[e]);
                    put(kg * A.KCS + pix, w);
                }
                {
                    const float ly = w1.x, lx = w1.y, hy = 1.f - ly, hx = 1.f - lx;
#pragma unroll
                    for (int e = 0; e < CPK; ++e) {
                        const float a = kind == 0 ? a0[e] : kind == 1 ? b0[e] : a1[e], cc = kind == 0 ? c0[e] : kind == 1 ? d0[e] : c1[e];
                        const float b = kind == 0 ? b0[e] : b1[e], d = kind == 0 ? d0[e] : d1[e];
                        w[e] = off1 >= 0 ? bilerp(hy, hx, ly, lx, a, b, cc, d) : 0.f;
                    }
                    put(kg * A.KCS + pix + 1, w);
                }
            }
            fence_async_smem();
            mbar_arrive(&a_full[s]);
        };
        // region -> image mapping of a tile (the table is shared by the loaders: barrier before and after the rewrite)
        auto map_tile = [&](const TileCoord& T) {
            asm volatile("bar.sync 1, %0;" ::"n"(CV_LOADERS) : "memory");
            for (int pix = threadIdx.x; pix < A.NPIX; pix += CV_LOADERS) {
                const int r = pix / A.RW, cc = pix - r * A.RW;
                int gy = T.y0 + r - padT, gx = T.x0 + cc - padL;
                bool ok = true;
                if (A.pad_mode == PAD_REFLECT) {
                    gy = reflect101(gy, A.H);
                    gx = reflect101(gx, A.W);
                } else {
                    ok = (gy >= 0 && gy < A.H && gx >= 0 && gx < A.W);
                }
                if (A.up) {        // (gy, gx) is a pixel of the upsampled image: its four sources and weights
                    int y0 = 0, y1 = 0, x0 = 0, x1 = 0;
                    float ly = 0.f, lx = 0.f;
                    if (ok) {
                        bilinear_src(gy, A.up_sy, A.up_align, A.Hs, y0, y1, ly);
                        bilinear_src(gx, A.up_sx, A.up_align, A.Ws, x0, x1, lx);
                    }
                    up_off[pix] = ok ? y0 * A.Ws + x0 : -1;
                    up_w[pix] = make_float2(ly, lx);
                    up_d[pix] = ((y1 - y0) * A.Ws) * 2 + (x1 - x0);
                }
                pixoff[pix] = ok ? gy * A.W + gx : -1;
            }
            asm volatile("bar.sync 1, %0;" ::"n"(CV_LOADERS) : "memory");
        };

        // Stream of (tile, chunk): store chunk k, put chunk k+1's loads in flight.  The A ring (>= 2 stages) lets the
        // loaders run a stage ahead of the tensor core, which is what hides the load latency of the next chunk.
        TileCoord curT = tile_coord(A, blockIdx.x), nextT = curT;
        const float* X = xd + (size_t)curT.img * A.H * A.W * ldd;
        if (A.up) {
            for (int tile = blockIdx.x; tile < A.ntiles; tile += gridDim.x) {
                const TileCoord T = tile_coord(A, tile);
                const float* Xu = A.x + (size_t)T.img * A.Hs * A.Ws * A.ldx;
                X = xd + (size_t)T.img * A.H * A.W * ldd;
                map_tile(T);
                for (int c = 0; c < A.up_chunks; ++c) stage_up(c, Xu);
                for (int c = A.up_chunks; c < A.nchunks; ++c) {      // channels behind the upsampled ones: x2, at full resolution
                    issue(c, X);
                    finish(c);
                }
            }
        } else {
        if ((int)blockIdx.x < A.ntiles) {
            map_tile(curT);
            issue(0, X);
        }
        for (int tile = blockIdx.x; tile < A.ntiles; tile += gridDim.x) {
            for (int c = 0; c < A.nchunks; ++c) {
                finish(c);
                if (c + 1 < A.nchunks) {
                    issue(c + 1, X);
                } else if (tile + (int)gridDim.x < A.ntiles) {
                    nextT = tile_coord(A, tile + gridDim.x);
                    X = xd + (size_t)nextT.img * A.H * A.W * ldd;
                    map_tile(nextT);
                    issue(0, X);
                }
            }
            curT = nextT;
        }
        }
        if (PREC == PREC_F16X3 && !(amax <= 65504.f) && A.overflow) atomicOr(A.overflow, 1);
    } else {
      asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(CV_REGS_MISC));
      if (warp == CV_PRODUCER_WARP) {
        // ================= weight producer =================
        if (lane == 0) {
            int it = 0;
            for (int tile = blockIdx.x; tile < A.ntiles; tile += gridDim.x)
                for (int c = 0; c < A.nchunks; ++c)
                    for (int tp = 0; tp < taps; ++tp, ++it) {
                        const int s = it % A.bstages;
                        if (it >= A.bstages) mbar_wait(&b_empty[s], ((it / A.bstages) - 1) & 1);
                        mbar_expect_tx(&b_full[s], A.b_stage_bytes);
                        bulk_g2s(b_base + (size_t)s * A.b_stage_bytes,
                                 A.wpack + ((size_t)c * taps + tp) * (A.b_stage_bytes / 4), A.b_stage_bytes, &b_full[s]);
                    }
        }
      } else if (warp == CV_MMA_WARP) {
        // ================= MMA issuer: whole warp runs the (uniform) loops, one elected lane issues =================
        {
            // instruction descriptor: D=F32, A=B=TF32 (format 2) or F16 (format 0), K-major both, N = Npad, M = 128
            const unsigned fmt = (PREC == PREC_F16X3) ? 0u : 2u;
            const unsigned idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((unsigned)(A.Npad >> 3) << 17) | ((128u >> 4) << 24);
            const unsigned a_lbo = (unsigned)A.KCS * 16u, a_sbo = (unsigned)A.RW * 16u;
            const unsigned b_lbo = 2u * (unsigned)A.Npad * 16u, b_sbo = 128u;     // K chunks are [hi rows; lo rows] apart
            const unsigned b_half = (unsigned)A.Npad * 16u;                        // B_lo rows follow the B_hi rows
            const unsigned idesc2 = (1u << 4) | (fmt << 7) | (fmt << 10) | ((unsigned)(A.Npad >> 2) << 17) | ((128u >> 4) << 24);
            // descriptors = constant part + (byte offset >> 4) in the 14-bit start-address field (smem < 256 KB: no carry)
            const unsigned long long a_desc0 = make_desc(0, a_lbo, a_sbo), b_desc0 = make_desc(0, b_lbo, b_sbo);
            const unsigned long long a_kstep = (2u * a_lbo) >> 4, b_kstep = (2u * b_lbo) >> 4;
            const unsigned tmem_u = __shfl_sync(0xffffffffu, tmem, 0);
            // The issue loop is specialised on (tiles per CTA, WIDE) and keeps every ring position / phase / descriptor as a
            // running value: on the small-N full-resolution layers a filter tap is only 16 MMAs (~700 tensor-pipe cycles), and
            // the generic loop (runtime MT / WIDE branches, two integer divisions per tap for the ring slots, descriptors
            // rebuilt from the arguments) took ~1300 cycles per tap -- the issuing warp, not the tensor pipe, set the pace
            // (ncu: this warp never waited on a barrier, hmma pipe 29 % active).
            auto mma_loop = [&](auto mt_c, auto wide_c) {
                constexpr int MTV = decltype(mt_c)::value;
                constexpr bool WV = decltype(wide_c)::value;
                const int nchunks = A.nchunks, astages = A.astages, bstages = A.bstages, KW = A.KW, ntiles = A.ntiles;
                const bool last_two = A.last_ksteps == 2;
                const unsigned np = (unsigned)A.tcols, row_skip = (unsigned)(A.RW - A.KW);
                const unsigned a_stage16 = A.a_stage_bytes >> 4, b_stage16 = A.b_stage_bytes >> 4;
                const unsigned a_base16 = smem_u32(a_base) >> 4, b_base16 = smem_u32(b_base) >> 4;
                const unsigned long long a_lo16 = a_half >> 4, b_lo16 = b_half >> 4;
                int sa = 0, sb = 0, j = 0;
                unsigned pha = 0, phb = 0, a_cur16 = a_base16, b_cur16 = b_base16;
                for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++j) {
                    const int buf = (nacc == 2) ? (j & 1) : 0, use = (nacc == 2) ? (j >> 1) : j;
                    if (use > 0) mbar_wait(&acc_empty[buf], (use - 1) & 1);     // epilogue drained this accumulator
                    tc_fence_after();
                    const unsigned tacc = tmem_u + (unsigned)buf * acc_cols;
                    for (int c = 0; c < nchunks; ++c) {
                        mbar_wait(&a_full[sa], pha);
                        const unsigned long long a_hi0 = a_desc0 + a_cur16, a_lo0 = a_hi0 + a_lo16;
                        const bool two = (c < nchunks - 1) || last_two;              // warp-uniform
                        unsigned tap_off = 0;                                        // in 16 B units (one pixel)
                        int dx = 0;
                        for (int tp = 0; tp < taps; ++tp) {
                            mbar_wait(&b_full[sb], phb);
                            tc_fence_after();
                            const unsigned long long dbh0 = b_desc0 + b_cur16, dbl0 = dbh0 + b_lo16;
                            const unsigned acc_first = (c == 0 && tp == 0) ? 0u : 1u;
                            const unsigned long long dah = a_hi0 + tap_off, dal = a_lo0 + tap_off;
                            tc_mma_kstep<MTV, PREC, WV>(tacc, np, dal, dah, dbh0, dbl0, idesc, acc_first, idesc2);
                            if (two)
                                tc_mma_kstep<MTV, PREC, WV>(tacc, np, dal + a_kstep, dah + a_kstep, dbh0 + b_kstep, dbl0 + b_kstep,
                                                            idesc, 1u, idesc2);
                            tc_commit(&b_empty[sb]);           // weights of this (chunk, tap) consumed
                            if (++sb == bstages) { sb = 0; phb ^= 1u; b_cur16 = b_base16; } else { b_cur16 += b_stage16; }
                            ++tap_off;
                            if (++dx == KW) { dx = 0; tap_off += row_skip; }
                        }
                        tc_commit(&a_empty[sa]);               // region of this chunk consumed
                        if (++sa == astages) { sa = 0; pha ^= 1u; a_cur16 = a_base16; } else { a_cur16 += a_stage16; }
                    }
                    tc_commit(&acc_full[buf]);
                }
            };
            using I1 = std::integral_constant<int, 1>;
            using I2 = std::integral_constant<int, 2>;
            using I4 = std::integral_constant<int, 4>;
            if (A.wide) {
                if (A.MT == 4) mma_loop(I4{}, std::true_type{}); else if (A.MT == 2) mma_loop(I2{}, std::true_type{}); else mma_loop(I1{}, std::true_type{});
            } else {
                if (A.MT == 4) mma_loop(I4{}, std::false_type{}); else if (A.MT == 2) mma_loop(I2{}, std::false_type{}); else mma_loop(I1{}, std::false_type{});
            }
        }
        __syncwarp();
      }
    }
    __syncthreads();
    if (warp == CV_MMA_WARP) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(A.tmem_cols));
    }
}

// ---- host side -----------------------------------------------------------------------------------
static int conv_geometry(ConvArgs& a, int prec, size_t* smem_bytes) {
    const int chunk = cv_chunk(prec);
    a.Npad = (a.Cout + 15) & ~15;
    FVFI_CHECK_ARG(a.Npad >= 16 && a.Npad <= 256, "conv: Cout %d not supported (1..256 per launch)", a.Cout);
    a.nchunks = (a.Cin + chunk - 1) / chunk;
    a.last_ksteps = (a.Cin - (a.nchunks - 1) * chunk) > chunk / 2 ? 2 : 1;
    a.b_stage_bytes = (unsigned)a.Npad * CV_KCHUNKS * 16u * 2u;        // hi + lo
    // one persistent CTA per SM: as many A stages as fit (the loaders run that far ahead of the tensor core)
    const int taps = a.KH * a.KW;
    const size_t budget = 222 * 1024;
    static const int force_mt = [] { const char* e = getenv("FVFI_CONV_MT"); return e ? atoi(e) : 0; }();   // tuning override
    for (int mt = 4; mt >= 1; mt >>= 1) {
        if (force_mt && mt > force_mt) continue;
        // WIDE pays for N <= 32 (two A reads instead of three).  Measured again with the dedicated epilogue warps and the lean
        // issue loop: at N = 64 the halved tile (MT = 2: 340 vs 377 TF/s) or a single-buffered accumulator (MT = 4: 308) cost
        // more than the saved A read; the softmax heads are epilogue-bound and keep the one-load-per-block form.
        a.wide = (a.Npad <= 32 && a.act != ACT_SOFTMAX) ? 1 : 0;
        a.tcols = a.wide ? 2 * a.Npad : a.Npad;
        if (mt * a.tcols > 512) continue;
        // Keep the accumulator DOUBLE-BUFFERED (epilogue of tile k under the MMAs of tile k+1) even when that halves the tile:
        // measured at B = 8 (tools/tune_conv_split.py): 512->512 @68x120 282 -> 427 TF/s, 256->256 @136x240 429 -> 523,
        // 128->128 @272x480 408 -> 522, the fused heads 64->448 399 -> 445 (MT = 1 for N > 128, MT = 2 for N = 128).
        if (mt > 1 && 2 * mt * a.tcols > 512) continue;
        if (mt > 1 && 8 * (mt / 2) >= a.W) continue;                   // do not over-tile narrow images
        a.MT = mt;
        a.nacc = (2 * mt * a.tcols <= 512) ? 2 : 1;
        a.RW = 8 * mt + a.KW - 1;
        a.RH = CV_ROWS + a.KH - 1;
        a.NPIX = a.RW * a.RH;
        // K-chunk stride of the A stage = NPIX 16-byte units rounded up to 2 (mod 8): the four K chunks of a pixel (what four
        // consecutive loader lanes store) then start 32 bytes apart modulo the 128-byte bank row, and a quarter-warp's 128-bit
        // stores (two pixels x four K chunks) cover all 32 banks once (ncu on 32->32 @1088x1920: the unpadded stride put K chunks
        // 0/2 and 1/3 on the same banks -- 8 instead of 4 wavefronts per STS.128, 20 M of the layer's 150 M LSU wavefronts)
        a.KCS = a.NPIX + ((2 - a.NPIX) & 7);
        a.a_stage_bytes = (unsigned)a.KCS * CV_KCHUNKS * 16u * 2u;    // hi + lo
        if (a.NPIX * CV_KCHUNKS > CV_LOADERS * CV_UMAX) continue;          // the loaders keep a whole K chunk in registers (UMAX)
        const size_t misc = 512 + (size_t)a.NPIX * 4 + 1024 + 16 + (a.up ? (size_t)a.NPIX * 16 : 0);
        const int min_b = std::min(2, a.nchunks * taps);
        if (misc + 2 * (size_t)a.a_stage_bytes + (size_t)min_b * a.b_stage_bytes > budget) continue;
        // weights first (up to 4 stages of a few KB), the rest goes to activation stages
        int bs = std::min(CV_MAX_BSTAGES, std::max(min_b, (int)((budget - misc - 2 * (size_t)a.a_stage_bytes) / a.b_stage_bytes)));
        int as = (int)((budget - misc - (size_t)bs * a.b_stage_bytes) / a.a_stage_bytes);
        a.bstages = bs;
        a.astages = std::max(2, std::min(CV_MAX_ASTAGES, as));
        int cols = 32;
        while (cols < a.nacc * mt * a.tcols) cols <<= 1;
        a.tmem_cols = cols;
        *smem_bytes = misc + (size_t)a.astages * a.a_stage_bytes + (size_t)a.bstages * a.b_stage_bytes;
        a.tiles_x = ceil_div(a.W, 8 * mt);
        a.tiles_y = ceil_div(a.H, CV_ROWS);
        a.ntiles = a.tiles_x * a.tiles_y * a.B;
        return FVFI_OK;
    }
    set_error("conv: no tile configuration fits (Cout %d, kernel %dx%d)", a.Cout, a.KH, a.KW);
    return FVFI_EINVAL;
}

static int* overflow_flag() {      // one device word per device, zero-initialised; creation is serialised across host threads
    static std::mutex mu;
    static std::atomic<int*> flags[FVFI_MAX_DEVICES];
    const int dev = current_device();
    if (dev < 0 || dev >= FVFI_MAX_DEVICES) return nullptr;
    int* p = flags[dev].load(std::memory_order_acquire);
    if (p) return p;
    std::lock_guard<std::mutex> lock(mu);
    p = flags[dev].load(std::memory_order_relaxed);
    if (!p) {
        if (cudaMalloc(&p, sizeof(int)) != cudaSuccess) return nullptr;
        cudaMemset(p, 0, sizeof(int));
        flags[dev].store(p, std::memory_order_release);
    }
    return p;
}

template <int PREC>
static void (*pick_kernel(int activation))(const ConvArgs) {
    switch (activation) {
        case ACT_RELU: return conv_split_kernel<ACT_RELU, PREC>;
        case ACT_ELU: return conv_split_kernel<ACT_ELU, PREC>;
        case ACT_TANH: return conv_split_kernel<ACT_TANH, PREC>;
        case ACT_SIGMOID: return conv_split_kernel<ACT_SIGMOID, PREC>;
        case ACT_SOFTMAX: return conv_split_kernel<ACT_SOFTMAX, PREC>;
        default: return conv_split_kernel<ACT_NONE, PREC>;
    }
}

}  // namespace fvfi

using namespace fvfi;

extern "C" size_t fvfi_conv2d_packed_weight_floats(int Cout, int Cin, int KH, int KW, int precision) {
    const int Npad = (Cout + 15) & ~15;
    const int chunk = cv_chunk(precision);
    const int nchunks = (Cin + chunk - 1) / chunk;
    return (size_t)CV_HDR + (size_t)nchunks * KH * KW * 2 * CV_KCHUNKS * Npad * 4;   // 16 bytes per (K chunk, n)
}

extern "C" int fvfi_conv2d_pack_weights(const float* weight_oihw, float* packed, int Cout, int Cin, int KH, int KW,
                                        int precision, void* stream) {
    FVFI_CHECK_ARG(weight_oihw && packed && Cout > 0 && Cin > 0 && KH > 0 && KW > 0, "conv_pack_weights: bad argument");
    FVFI_CHECK_ARG(precision == PREC_TF32X3 || precision == PREC_F16X3, "conv_pack_weights: precision must be 0 (3xTF32) or 1 (3xFP16)");
    const int Npad = (Cout + 15) & ~15;
    const int chunk = cv_chunk(precision);
    const int nchunks = (Cin + chunk - 1) / chunk;
    const size_t total = (size_t)nchunks * KH * KW * 2 * CV_KCHUNKS * Npad * cv_cpk(precision);
    const unsigned blocks = (unsigned)((total + 255) / 256 > 4096 ? 4096 : (total + 255) / 256);
    cudaStream_t s = (cudaStream_t)stream;
    conv_weight_scale_kernel<<<1, 1024, 0, s>>>(weight_oihw, (size_t)Cout * Cin * KH * KW, packed, precision);
    FVFI_LAUNCH_CHECK();
    if (precision == PREC_F16X3)
        conv_pack_weights_kernel<PREC_F16X3><<<blocks, 256, 0, s>>>(weight_oihw, packed, Cout, Cin, KH, KW, Npad, nchunks);
    else
        conv_pack_weights_kernel<PREC_TF32X3><<<blocks, 256, 0, s>>>(weight_oihw, packed, Cout, Cin, KH, KW, Npad, nchunks);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_conv2d_overflow_count(void) {
    int* f = overflow_flag();
    if (!f) return -1;
    int v = 0;
    if (cudaMemcpy(&v, f, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
    if (v) cudaMemset(f, 0, sizeof(int));
    return v;
}

extern "C" int fvfi_conv2d_nhwc(const float* x, int x_pixel_stride, const float* packed_weight, const float* bias, float* y,
                                int y_pixel_stride, int B, int H, int W, int Cin, int Cout, int KH, int KW, int pad_mode,
                                int activation, int out_nchw, int precision, void* stream) {
    return fvfi_conv2d_nhwc_residual(x, x_pixel_stride, packed_weight, bias, nullptr, 0, y, y_pixel_stride, B, H, W, Cin, Cout, KH, KW,
                                     pad_mode, activation, out_nchw, precision, stream);
}

extern "C" int fvfi_conv2d_nhwc_residual(const float* x, int x_pixel_stride, const float* packed_weight, const float* bias,
                                         const float* residual, int residual_pixel_stride, float* y, int y_pixel_stride, int B, int H,
                                         int W, int Cin, int Cout, int KH, int KW, int pad_mode, int activation, int out_nchw,
                                         int precision, void* stream) {
    return fvfi_conv2d_nhwc_upsampled(x, x_pixel_stride, 0, 0, 0, nullptr, 0, 0, packed_weight, bias, residual, residual_pixel_stride, y,
                                      y_pixel_stride, B, H, W, Cin, Cout, KH, KW, pad_mode, activation, out_nchw, precision, stream);
}

extern "C" int fvfi_conv2d_nhwc_upsampled(const float* x, int x_pixel_stride, int Hs, int Ws, int align_corners, const float* x_direct,
                                          int x_direct_pixel_stride, int cin_upsampled,
                                          const float* packed_weight, const float* bias, const float* residual,
                                          int residual_pixel_stride, float* y, int y_pixel_stride, int B, int H, int W, int Cin,
                                          int Cout, int KH, int KW, int pad_mode, int activation, int out_nchw, int precision,
                                          void* stream) {
    FVFI_CHECK_ARG(!residual || (activation != ACT_SOFTMAX && residual_pixel_stride >= Cout),
                   "conv2d: a residual needs a pixel stride >= Cout and no softmax");
    FVFI_CHECK_ARG(x && packed_weight && y, "conv2d: null pointer");
    FVFI_CHECK_ARG(B > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0 && B <= 65535, "conv2d: bad dimension");
    FVFI_CHECK_ARG((KH == 1 || KH == 3 || KH == 5) && KW == KH, "conv2d: kernel must be 1x1, 3x3 or 5x5");
    FVFI_CHECK_ARG(pad_mode == PAD_ZERO || pad_mode == PAD_REFLECT, "conv2d: pad_mode must be 0 (zero) or 1 (reflect)");
    FVFI_CHECK_ARG(pad_mode != PAD_REFLECT || (H > KH / 2 && W > KW / 2), "conv2d: reflect padding needs H,W > pad");
    FVFI_CHECK_ARG(activation >= 0 && activation <= 5, "conv2d: bad activation");
    FVFI_CHECK_ARG(activation != ACT_SOFTMAX || Cout <= 256, "conv2d: softmax needs all channels in one call");
    FVFI_CHECK_ARG(precision == PREC_TF32X3 || precision == PREC_F16X3, "conv2d: precision must be 0 (3xTF32) or 1 (3xFP16)");
    ConvArgs a{};
    a.x = x; a.hdr = packed_weight; a.wpack = packed_weight + CV_HDR; a.bias = bias; a.y = y;
    a.ldx = x_pixel_stride; a.ldy = y_pixel_stride; a.out_nchw = (out_nchw == 1) ? 1 : 0;
    a.res = residual; a.ldr = residual_pixel_stride;
    a.up = (Hs > 0 || Ws > 0) ? 1 : 0;
    if (a.up) {
        const int cpk = cv_cpk(precision), cin_r = (Cin + cpk - 1) / cpk * cpk;
        FVFI_CHECK_ARG(Hs > 0 && Ws > 0 && (size_t)Hs * Ws < (1u << 30), "conv2d: bad source size %dx%d for the upsampling loader", Hs, Ws);
        FVFI_CHECK_ARG((x_pixel_stride % cpk) == 0 && (x_direct || x_pixel_stride >= cin_r) && ((size_t)x % (4 * cpk)) == 0,
                       "conv2d: the upsampling loader needs an aligned source whose pixel stride is a multiple of %d and >= %d", cpk, cin_r);
        a.Hs = Hs; a.Ws = Ws; a.up_align = align_corners ? 1 : 0;
        a.up_sy = bilinear_scale(Hs, H, a.up_align);
        a.up_sx = bilinear_scale(Ws, W, a.up_align);
        const int chunk = cv_chunk(precision);
        a.up_chunks = (Cin + chunk - 1) / chunk;
        if (x_direct) {
            FVFI_CHECK_ARG(cin_upsampled > 0 && cin_upsampled < Cin && (cin_upsampled % chunk) == 0,
                           "conv2d: the upsampled part of a two-source input must be a multiple of %d channels (got %d of %d)", chunk,
                           cin_upsampled, Cin);
            FVFI_CHECK_ARG(x_direct_pixel_stride >= Cin - cin_upsampled, "conv2d: x_direct pixel stride smaller than its channel count");
            a.x2 = x_direct; a.ldx2 = x_direct_pixel_stride; a.up_chunks = cin_upsampled / chunk;
        }
    } else {
        FVFI_CHECK_ARG(!x_direct, "conv2d: x_direct needs an upsampled first source");
    }
    a.cout_store = (out_nchw == 2) ? ((Cout + 15) & ~15) : Cout;
    FVFI_CHECK_ARG(out_nchw >= 0 && out_nchw <= 2, "conv2d: output layout must be 0 (NHWC), 1 (NCHW) or 2 (NHWC, zero-padded channels)");
    FVFI_CHECK_ARG(out_nchw != 2 || y_pixel_stride >= a.cout_store, "conv2d: padded NHWC output needs a pixel stride >= round16(Cout)");
    a.overflow = (precision == PREC_F16X3) ? overflow_flag() : nullptr;
    FVFI_CHECK_ARG(x_pixel_stride >= (x_direct ? cin_upsampled : Cin) && (out_nchw || y_pixel_stride >= Cout),
                   "conv2d: pixel stride smaller than channel count");
    a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.KH = KH; a.KW = KW; a.pad_mode = pad_mode; a.act = activation;
    size_t smem = 0;
    if (int rc = conv_geometry(a, precision, &smem)) return rc;
    const int nsm = sm_count();
    dim3 grid((unsigned)std::min(a.ntiles, nsm > 0 ? nsm : 148), 1, 1);
    void (*kern)(const ConvArgs) = (precision == PREC_F16X3) ? pick_kernel<PREC_F16X3>(activation) : pick_kernel<PREC_TF32X3>(activation);
    FVFI_SMEM_OPT_IN(kern, smem);
    kern<<<grid, CV_THREADS, smem, (cudaStream_t)stream>>>(a);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}
