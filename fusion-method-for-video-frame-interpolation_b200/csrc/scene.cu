// scene.cu -- scene-cut detection on 8-bit clips (include/fvfi.h: fvfi_frame_sad_u8, fvfi_scene_cut_decide,
// fvfi_scene_cut_select_u8; DESIGN.md 6b).  Per pair p of a window: the byte SAD of frames p and p + 1, the decision rule
// (mafd / score / threshold, restated in numpy by oracle/scene.py), and the substitution of frame p for the interpolated frame
// at a cut.  All three run on the caller's stream; nothing here synchronises the host.
#include <math.h>

#include "common.cuh"

namespace fvfi {

constexpr int kSadThreads = 256;
constexpr int kSadChunks = 2;           // 16-byte chunks per thread, kSadThreads apart (coalesced)
constexpr int kSelectThreads = 256;
constexpr int kSelectBlocksX = 128;     // blocks per pair of the select grid (grid-stride beyond that)
constexpr int kMaxPairs = 65535;        // grid.y of the select kernel

// 16 bytes at p: one 16-byte load when the frames allow it, 16 byte loads packed little-endian otherwise.
template <bool kVec>
__device__ __forceinline__ uint4 load16(const uint8_t* p) {
    if constexpr (kVec) {
        return __ldg(reinterpret_cast<const uint4*>(p));
    } else {
        unsigned w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
            w[j] = (unsigned)__ldg(p + 4 * j) | (unsigned)__ldg(p + 4 * j + 1) << 8 | (unsigned)__ldg(p + 4 * j + 2) << 16 |
                   (unsigned)__ldg(p + 4 * j + 3) << 24;
        return make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// acc + sum of |a_i - b_i| over the 16 bytes: per-byte absolute differences (SIMD), summed by a dot product with ones.
__device__ __forceinline__ unsigned sad16(uint4 a, uint4 b, unsigned acc) {
    acc = __dp4a(__vabsdiffu4(a.x, b.x), 0x01010101u, acc);
    acc = __dp4a(__vabsdiffu4(a.y, b.y), 0x01010101u, acc);
    acc = __dp4a(__vabsdiffu4(a.z, b.z), 0x01010101u, acc);
    return __dp4a(__vabsdiffu4(a.w, b.w), 0x01010101u, acc);
}

// One thread owns kSadChunks 16-byte chunks of the compared bytes and walks them through every frame of the window, keeping the
// previous frame's chunks in registers: each byte is read from HBM once.  The n % 16 tail bytes belong to the first threads of
// block 0.  Per pair: warp sums (__reduce_add_sync), one block sum in shared memory (double-buffered by pair parity, so one
// barrier per pair), one 64-bit atomic per block.  A block sums at most 256 * 2 * 16 * 255 < 2^32, so 32-bit partial sums are
// exact, and integer addition makes the total independent of the order.
template <bool kVec>
__global__ void __launch_bounds__(kSadThreads) frame_sad_u8_kernel(const uint8_t* __restrict__ frames, size_t stride, size_t nvec,
                                                                   unsigned tail, int pairs, unsigned long long* __restrict__ sad) {
    __shared__ unsigned warp_sums[2][kSadThreads / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t c0 = (size_t)blockIdx.x * (kSadThreads * kSadChunks) + threadIdx.x;
    const bool has_tail = blockIdx.x == 0 && threadIdx.x < tail;
    const size_t tail_off = nvec * 16 + threadIdx.x;
    uint4 prev[kSadChunks];
#pragma unroll
    for (int k = 0; k < kSadChunks; ++k) {
        const size_t c = c0 + (size_t)k * kSadThreads;
        prev[k] = c < nvec ? load16<kVec>(frames + c * 16) : make_uint4(0u, 0u, 0u, 0u);
    }
    unsigned prev_tail = has_tail ? __ldg(frames + tail_off) : 0u;
    for (int p = 0; p < pairs; ++p) {
        const uint8_t* f = frames + (size_t)(p + 1) * stride;
        uint4 cur[kSadChunks];
#pragma unroll
        for (int k = 0; k < kSadChunks; ++k) {
            const size_t c = c0 + (size_t)k * kSadThreads;
            cur[k] = c < nvec ? load16<kVec>(f + c * 16) : make_uint4(0u, 0u, 0u, 0u);
        }
        unsigned s = 0;
        if (has_tail) {
            const unsigned t = __ldg(f + tail_off);
            s = t > prev_tail ? t - prev_tail : prev_tail - t;
            prev_tail = t;
        }
#pragma unroll
        for (int k = 0; k < kSadChunks; ++k) {   // chunks past nvec are zero in both frames
            s = sad16(prev[k], cur[k], s);
            prev[k] = cur[k];
        }
        s = __reduce_add_sync(0xffffffffu, s);
        if (lane == 0) warp_sums[p & 1][warp] = s;
        __syncthreads();
        if (warp == 0) {
            unsigned v = lane < kSadThreads / 32 ? warp_sums[p & 1][lane] : 0u;
            v = __reduce_add_sync(0xffffffffu, v);
            if (lane == 0 && v) atomicAdd(sad + p, (unsigned long long)v);
        }
    }
}

// mafd = sad * 100 / n / 256, each operation rounded to nearest on its own (no FMA), as numpy float64 evaluates it.
__device__ __forceinline__ double mafd_of(unsigned long long s, double n) {
    return __ddiv_rn(__ddiv_rn(__dmul_rn(__ull2double_rn(s), 100.0), n), 256.0);
}

// One thread per pair.  The previous pair's mafd is recomputed from its SAD (not read from mafd, which this launch writes), so
// the pairs are independent; pair 0 takes the carry prev_in (or 0 at the start of a stream).
__global__ void scene_cut_decide_kernel(const unsigned long long* __restrict__ sad, int pairs, double n, const double* prev_in,
                                        double threshold, double* mafd, uint8_t* __restrict__ cut) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= pairs) return;
    const double m = mafd_of(sad[p], n);
    const double prev = p > 0 ? mafd_of(sad[p - 1], n) : (prev_in ? *prev_in : 0.0);
    const double score = fmin(fmax(fmin(m, fabs(__dsub_rn(m, prev))), 0.0), 100.0);
    mafd[p] = m;
    cut[p] = score >= threshold ? 1 : 0;
}

// Grid (chunk, pair): the blocks of an uncut pair read its flag and return; those of a cut pair copy frame p into output p.
template <bool kVec>
__global__ void __launch_bounds__(kSelectThreads) scene_cut_select_u8_kernel(const uint8_t* __restrict__ frames, size_t stride,
                                                                             uint8_t* __restrict__ out, size_t out_stride,
                                                                             size_t frame_bytes, const uint8_t* __restrict__ cut) {
    const int p = blockIdx.y;
    if (!cut[p]) return;
    const uint8_t* src = frames + (size_t)p * stride;
    uint8_t* dst = out + (size_t)p * out_stride;
    const size_t step = (size_t)gridDim.x * kSelectThreads;
    const size_t i0 = (size_t)blockIdx.x * kSelectThreads + threadIdx.x;
    size_t done = 0;
    if (kVec) {
        const size_t nvec = frame_bytes / 16;
        const uint4* s4 = reinterpret_cast<const uint4*>(src);
        uint4* d4 = reinterpret_cast<uint4*>(dst);
        for (size_t i = i0; i < nvec; i += step) d4[i] = __ldg(s4 + i);
        done = nvec * 16;
    }
    for (size_t i = done + i0; i < frame_bytes; i += step) dst[i] = __ldg(src + i);
}

static int check_pairs(const char* fn, int pairs) {
    FVFI_CHECK_ARG(pairs >= 1 && pairs <= kMaxPairs, "%s: pairs must be in [1, %d], got %d", fn, kMaxPairs, pairs);
    return FVFI_OK;
}

}  // namespace fvfi

using namespace fvfi;

extern "C" int fvfi_frame_sad_u8(const uint8_t* frames, size_t stride, size_t n, int pairs, unsigned long long* sad, void* stream) {
    FVFI_CHECK_ARG(frames && sad, "fvfi_frame_sad_u8: null pointer");
    if (int rc = check_pairs("fvfi_frame_sad_u8", pairs)) return rc;
    FVFI_CHECK_ARG(n > 0 && n <= stride, "fvfi_frame_sad_u8: need 0 < n <= stride, got n=%zu stride=%zu", n, stride);
    cudaStream_t s = (cudaStream_t)stream;
    FVFI_CUDA(cudaMemsetAsync(sad, 0, (size_t)pairs * sizeof(unsigned long long), s));
    const size_t nvec = n / 16;
    const unsigned tail = (unsigned)(n % 16);
    const size_t per_block = (size_t)kSadThreads * kSadChunks;
    const unsigned blocks = (unsigned)(nvec ? (nvec + per_block - 1) / per_block : 1);
    if ((uintptr_t)frames % 16 == 0 && stride % 16 == 0)
        frame_sad_u8_kernel<true><<<blocks, kSadThreads, 0, s>>>(frames, stride, nvec, tail, pairs, sad);
    else
        frame_sad_u8_kernel<false><<<blocks, kSadThreads, 0, s>>>(frames, stride, nvec, tail, pairs, sad);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_scene_cut_decide(const unsigned long long* sad, int pairs, size_t n, const double* prev_in, double threshold,
                                     double* mafd, uint8_t* cut, void* stream) {
    FVFI_CHECK_ARG(sad && mafd && cut, "fvfi_scene_cut_decide: null pointer");
    if (int rc = check_pairs("fvfi_scene_cut_decide", pairs)) return rc;
    FVFI_CHECK_ARG(n > 0, "fvfi_scene_cut_decide: n must be positive");
    FVFI_CHECK_ARG(threshold >= 0.0, "fvfi_scene_cut_decide: threshold must be >= 0 and not NaN, got %g", threshold);
    scene_cut_decide_kernel<<<(pairs + 255) / 256, 256, 0, (cudaStream_t)stream>>>(sad, pairs, (double)n, prev_in, threshold, mafd,
                                                                                    cut);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_scene_cut_select_u8(const uint8_t* frames, size_t stride, uint8_t* out, size_t out_stride, size_t frame_bytes,
                                        int pairs, const uint8_t* cut, void* stream) {
    FVFI_CHECK_ARG(frames && out && cut, "fvfi_scene_cut_select_u8: null pointer");
    if (int rc = check_pairs("fvfi_scene_cut_select_u8", pairs)) return rc;
    FVFI_CHECK_ARG(frame_bytes > 0 && frame_bytes <= stride && frame_bytes <= out_stride,
                   "fvfi_scene_cut_select_u8: need 0 < frame_bytes <= stride and <= out_stride, got %zu, %zu, %zu", frame_bytes,
                   stride, out_stride);
    const bool vec = (uintptr_t)frames % 16 == 0 && (uintptr_t)out % 16 == 0 && stride % 16 == 0 && out_stride % 16 == 0;
    const size_t units = vec ? (frame_bytes / 16 ? frame_bytes / 16 : 1) : frame_bytes;
    const size_t bx = (units + kSelectThreads - 1) / kSelectThreads;
    dim3 grid((unsigned)(bx < (size_t)kSelectBlocksX ? bx : (size_t)kSelectBlocksX), (unsigned)pairs);
    if (vec)
        scene_cut_select_u8_kernel<true><<<grid, kSelectThreads, 0, (cudaStream_t)stream>>>(frames, stride, out, out_stride,
                                                                                            frame_bytes, cut);
    else
        scene_cut_select_u8_kernel<false><<<grid, kSelectThreads, 0, (cudaStream_t)stream>>>(frames, stride, out, out_stride,
                                                                                             frame_bytes, cut);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}
