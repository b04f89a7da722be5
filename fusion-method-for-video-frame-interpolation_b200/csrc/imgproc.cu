// imgproc.cu -- the per-pixel stages that the reference bounces to the CPU (SURVEY.md 8(f) f1/f2):
//   RGB <-> Lab   (src/train/transform.py:6-49: skimage.color on the host, then L/100, (a,b+128)/255)
//   Gaussian sigma blur     (scipy.ndimage.gaussian_filter(h, 5), interpolate_twoframe.py:212-213)
//   k x k median            (scipy.ndimage.median_filter(f, size=50), interpolate_twoframe.py:221-222)
// Device-resident replacements so the fusion pipeline never leaves the GPU.
#include "common.cuh"

namespace fvfi {

// ---- colour ------------------------------------------------------------------------------------
// sRGB (IEC 61966-2-1) -> linear -> XYZ (D65 / 2 deg) -> CIE L*a*b*, as skimage.color.rgb2lab.
__device__ __forceinline__ float srgb_to_lin(float c) {
    return c > 0.04045f ? powf((c + 0.055f) / 1.055f, 2.4f) : c / 12.92f;
}
__device__ __forceinline__ float lin_to_srgb(float c) {
    return c > 0.0031308f ? 1.055f * powf(fmaxf(c, 0.f), 1.f / 2.4f) - 0.055f : c * 12.92f;
}
__device__ __forceinline__ float lab_f(float t) { return t > 0.008856f ? cbrtf(t) : 7.787f * t + 16.f / 116.f; }
__device__ __forceinline__ float lab_finv(float f) { return f > 0.2068966f ? f * f * f : (f - 16.f / 116.f) / 7.787f; }

// One pixel: sRGB in [0,1] -> scaled Lab written at dst[0], dst[plane], dst[2*plane] (shared by rgb2lab_kernel and
// rgb8_to_rgb_lab_kernel, so both give the same bits for the same RGB value).
__device__ __forceinline__ void rgb_to_scaled_lab(float sr, float sg, float sb, float* dst, size_t plane) {
    const float r = srgb_to_lin(sr), g = srgb_to_lin(sg), b = srgb_to_lin(sb);
    const float x = (0.412453f * r + 0.357580f * g + 0.180423f * b) / 0.95047f;
    const float y = (0.212671f * r + 0.715160f * g + 0.072169f * b);
    const float z = (0.019334f * r + 0.119193f * g + 0.950227f * b) / 1.08883f;
    const float fx = lab_f(x), fy = lab_f(y), fz = lab_f(z);
    dst[0] = (116.f * fy - 16.f) / 100.f;                    // transform.py:9  L / light
    dst[plane] = (500.f * (fx - fy) + 128.f) / 255.f;        // transform.py:10-11
    dst[2 * plane] = (200.f * (fy - fz) + 128.f) / 255.f;
}

__global__ void rgb2lab_kernel(const float* __restrict__ rgb, float* __restrict__ lab, size_t plane, int B) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.y;
    if (p >= plane) return;
    const float* src = rgb + (size_t)n * 3 * plane + p;
    rgb_to_scaled_lab(src[0], src[plane], src[2 * plane], lab + (size_t)n * 3 * plane + p, plane);
    (void)B;
}

// Decoder frames [T,H,W,3] uint8 (interleaved rgb24) -> planar fp32 RGB [T,3,H,W] (k / 255, correctly rounded: __fdiv_rn, not a
// reciprocal multiply) and planar scaled Lab [T,3,H,W] in one pass.  A warp reads 96 contiguous bytes and writes coalesced planes.
__global__ void __launch_bounds__(256) rgb8_to_rgb_lab_kernel(const uint8_t* __restrict__ rgb8, float* __restrict__ rgb,
                                                              float* __restrict__ lab, size_t plane) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.y;
    if (p >= plane) return;
    const uint8_t* src = rgb8 + ((size_t)n * plane + p) * 3;
    const float r = __fdiv_rn((float)__ldg(src), 255.f), g = __fdiv_rn((float)__ldg(src + 1), 255.f),
                b = __fdiv_rn((float)__ldg(src + 2), 255.f);
    const size_t o = (size_t)n * 3 * plane + p;
    rgb[o] = r;
    rgb[o + plane] = g;
    rgb[o + 2 * plane] = b;
    rgb_to_scaled_lab(r, g, b, lab + o, plane);
}

__global__ void lab2rgb_kernel(const float* __restrict__ lab, float* __restrict__ rgb, size_t plane, int B) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.y;
    if (p >= plane) return;
    const float* src = lab + (size_t)n * 3 * plane + p;
    const float L = src[0] * 100.f;                          // transform.py:31-33
    const float a = src[plane] * 255.f - 128.f, b = src[2 * plane] * 255.f - 128.f;
    const float fy = (L + 16.f) / 116.f;
    const float fx = a / 500.f + fy;
    const float fz = fmaxf(fy - b / 200.f, 0.f);             // skimage clips negative z
    const float x = lab_finv(fx) * 0.95047f, y = lab_finv(fy), z = lab_finv(fz) * 1.08883f;
    const float r = 3.2404813432f * x - 1.5371515163f * y - 0.4985363262f * z;
    const float g = -0.9692549500f * x + 1.8759900015f * y + 0.0415559266f * z;
    const float bl = 0.0556466391f * x - 0.2040413384f * y + 1.0573110696f * z;
    float* dst = rgb + (size_t)n * 3 * plane + p;
    dst[0] = fminf(fmaxf(lin_to_srgb(r), 0.f), 1.f);
    dst[plane] = fminf(fmaxf(lin_to_srgb(g), 0.f), 1.f);
    dst[2 * plane] = fminf(fmaxf(lin_to_srgb(bl), 0.f), 1.f);
    (void)B;
}

// ---- scipy 'reflect' boundary: (d c b a | a b c d | d c b a) ---------------------------------------
__device__ __forceinline__ int reflect_idx(int i, int n) {
    const int period = 2 * n;
    int m = i % period;
    if (m < 0) m += period;
    return m < n ? m : period - 1 - m;
}

// ---- separable Gaussian (one axis per launch), weights in constant-size smem -------------------------
constexpr int GAUSS_MAX_RADIUS = 64;

template <bool ALONG_X>
__global__ void __launch_bounds__(256) gauss1d_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W,
                                                      float sigma, int radius) {
    __shared__ float wts[2 * GAUSS_MAX_RADIUS + 1];
    __shared__ float norm;
    if (threadIdx.x <= radius) {
        const float v = expf(-0.5f * (float)(threadIdx.x * threadIdx.x) / (sigma * sigma));
        wts[radius + threadIdx.x] = v;
        wts[radius - threadIdx.x] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int i = 0; i <= 2 * radius; ++i) s += wts[i];
        norm = 1.f / s;
    }
    __syncthreads();
    const size_t plane = (size_t)H * W;
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= plane) return;
    const int y = (int)(p / W), x = (int)(p - (size_t)y * W);
    const float* src = in + (size_t)blockIdx.y * plane;
    float acc = 0.f;
    for (int t = -radius; t <= radius; ++t) {
        const float v = ALONG_X ? src[(size_t)y * W + reflect_idx(x + t, W)] : src[(size_t)reflect_idx(y + t, H) * W + x];
        acc = fmaf(v, wts[radius + t], acc);
    }
    out[(size_t)blockIdx.y * plane + p] = acc * norm;
}

// Fast path for a compile-time radius (sigma = 5 -> 20, the recipe's call): the generic kernel above issues 2R+1 global loads with a
// reflected index each per output (~330 instructions per pixel).  Here the 2R+1 weights live in registers (full unroll) and
//   * along y: a thread owns one column and GR consecutive output rows; every input row r it loads (GR + 2R loads for GR outputs) is
//     added to all outputs it reaches -- in ascending r, i.e. in the generic kernel's tap order: the results are bit-identical;
//   * along x: a block stages its row segment (+ R on each side, reflected) in shared memory once, a thread owns GX consecutive
//     outputs and walks the GX + 2R staged values the same way.
constexpr int GR = 16, GX = 4, GAUSS_XT = 256;

template <int R>
__device__ __forceinline__ void gauss_weights(float sigma, float* w, float& norm) {       // same arithmetic as the generic kernel
    float s = 0.f;
#pragma unroll
    for (int i = 0; i <= 2 * R; ++i) {
        const int d = i < R ? R - i : i - R;
        w[i] = expf(-0.5f * (float)(d * d) / (sigma * sigma));
    }
#pragma unroll
    for (int i = 0; i <= 2 * R; ++i) s += w[i];
    norm = 1.f / s;
}

template <int R>
__global__ void __launch_bounds__(128) gauss_y_fast_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W,
                                                           float sigma) {
    float w[2 * R + 1], norm;
    gauss_weights<R>(sigma, w, norm);
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= W) return;
    const int y0 = blockIdx.y * GR;
    const size_t plane = (size_t)H * W;
    const float* src = in + (size_t)blockIdx.z * plane + x;
    float acc[GR];
#pragma unroll
    for (int j = 0; j < GR; ++j) acc[j] = 0.f;
#pragma unroll
    for (int rr = 0; rr < GR + 2 * R; ++rr) {                       // input row y0 - R + rr reaches outputs j with |rr - R - j| <= R
        const float v = __ldg(src + (size_t)reflect_idx(y0 - R + rr, H) * W);
#pragma unroll
        for (int j = 0; j < GR; ++j) {
            if (rr - j >= 0 && rr - j <= 2 * R) acc[j] = fmaf(v, w[rr - j], acc[j]);     // tap t = rr - j - R, ascending in rr
        }
    }
    float* dst = out + (size_t)blockIdx.z * plane + x;
#pragma unroll
    for (int j = 0; j < GR; ++j)
        if (y0 + j < H) dst[(size_t)(y0 + j) * W] = acc[j] * norm;
}

template <int R>
__global__ void __launch_bounds__(GAUSS_XT / GX) gauss_x_fast_kernel(const float* __restrict__ in, float* __restrict__ out, int H, int W,
                                                                    float sigma) {
    __shared__ float seg[GAUSS_XT + 2 * R];
    float w[2 * R + 1], norm;
    gauss_weights<R>(sigma, w, norm);
    const int x0 = blockIdx.x * GAUSS_XT, y = blockIdx.y;
    const size_t plane = (size_t)H * W;
    const float* src = in + (size_t)blockIdx.z * plane + (size_t)y * W;
    for (int i = threadIdx.x; i < GAUSS_XT + 2 * R; i += blockDim.x) seg[i] = __ldg(src + reflect_idx(x0 - R + i, W));
    __syncthreads();
    const int xo = threadIdx.x * GX;
    float acc[GX];
#pragma unroll
    for (int j = 0; j < GX; ++j) acc[j] = 0.f;
#pragma unroll
    for (int rr = 0; rr < GX + 2 * R; ++rr) {
        const float v = seg[xo + rr];
#pragma unroll
        for (int j = 0; j < GX; ++j) {
            if (rr - j >= 0 && rr - j <= 2 * R) acc[j] = fmaf(v, w[rr - j], acc[j]);
        }
    }
    float* dst = out + (size_t)blockIdx.z * plane + (size_t)y * W + x0 + xo;
#pragma unroll
    for (int j = 0; j < GX; ++j)
        if (x0 + xo + j < W) dst[j] = acc[j] * norm;
}

// ---- exact k x k median (rank k*k/2, window [i - k/2, i + k - k/2 - 1], reflect) -------------------------
// Order statistics must be exact (scipy's rank filter), so no histogram approximation.
//
// Fast path (median_rank_kernel): a CTA owns a TW x 16 output tile, TW chosen by the launcher so that the region fills the
// 8192-entry sorting network (k = 50: 77 x 16 outputs, 126 x 65 = 8190 samples; a 32-wide tile left 36 % of the network
// sorting padding).  It stages the (TW+k-1)x(16+k-1)
// neighbourhood as (order-preserving key, position) pairs, BITONIC-SORTS it once in shared memory, and
// replaces every sample by its RANK in the region.  A window's median is then "the rank-th set bit" of a
// window-membership bitmap over rank space: one warp per output row builds the bitmap of its first window
// (k*k bit sets) and SLIDES it along x -- k bit clears + k bit sets per pixel.  The wanted set bit is TRACKED, not searched: the warp
// keeps the 256-rank block that holds it and the number of set bits before that block, updated from the ranks that leave / enter the
// window (two ballots per round), so a pixel counts one block (one word per lane + redux.add) and bisects one word with popcounts
// (a full recount of the 256-word bitmap + warp scan + __fns per pixel was half of the kernel: 1.65 -> 1.14 ms per 1080p map).
// The sort keeps 16 consecutive elements per thread in registers for the passes with j <= 8 (1.14 -> 0.90 ms).
// Fallback (median_bisect_kernel): per-thread bisection over the key space, any k <= 96.
__device__ __forceinline__ unsigned f2key(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key2f(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

constexpr int MR_TH = 16, MR_THREADS = MR_TH * 32;
constexpr int MR_MAX_N = 8192;

// element i of the sort array lives at i + (i >> 4): a thread's 16 consecutive elements (the register-local passes) then start
// 34 words apart, which spreads the lanes of a 64-bit access over all banks
__device__ __forceinline__ int mr_sk(int i) { return i + (i >> 4); }
constexpr int MR_E = 16;                                               // elements per thread in the register-local passes

// compare-exchange passes j = JS, JS/2, .., 1 of bitonic stage kk on the 16 elements a thread holds (element e = index base + e)
template <int JS>
__device__ __forceinline__ void mr_local_passes(unsigned long long* v, int base, int kk) {
#pragma unroll
    for (int j = JS; j >= 1; j >>= 1) {
#pragma unroll
        for (int e = 0; e < MR_E; ++e) {
            if ((e & j) == 0) {
                const bool asc = ((base + e) & kk) == 0;
                const unsigned long long a = v[e], b = v[e | j];
                const bool sw = (a > b) == asc;
                v[e] = sw ? b : a;
                v[e | j] = sw ? a : b;
            }
        }
    }
}

__global__ void __launch_bounds__(MR_THREADS) median_rank_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                                 int H, int W, int k, int rank, int npad, int MR_TW) {
    extern __shared__ unsigned long long pairs[];                      // npad + npad/16 (key << 32 | pos), skewed: mr_sk
    const int RW = MR_TW + k - 1, RH = MR_TH + k - 1, n = RW * RH;
    unsigned short* rank_of = (unsigned short*)(pairs + npad + (npad >> 4));   // n
    const int nwords = (n + 31) >> 5;
    const int wpl = (nwords + 31) >> 5;                                // bitmap words per lane
    unsigned* bitmaps = (unsigned*)(rank_of + ((n + 7) & ~7));         // MR_TH x (wpl*32), 16-byte aligned
    const int x0 = blockIdx.x * MR_TW, y0 = blockIdx.y * MR_TH;
    const size_t plane = (size_t)H * W;
    const float* src = in + (size_t)blockIdx.z * plane;
    const int lo_off = k / 2;
    for (int q = threadIdx.x; q < npad; q += MR_THREADS) {
        unsigned long long v = 0xffffffffffffffffull;
        if (q < n) {
            const int r = q / RW, c = q - r * RW;
            const unsigned key = f2key(src[(size_t)reflect_idx(y0 + r - lo_off, H) * W + reflect_idx(x0 + c - lo_off, W)]);
            v = ((unsigned long long)key << 32) | (unsigned)q;
        }
        pairs[mr_sk(q)] = v;
    }
    __syncthreads();
    if (npad == MR_E * MR_THREADS) {
        // Every thread keeps 16 consecutive elements in registers for the passes with j <= 8 (46 of the 91 passes of an 8192-entry
        // network): stages kk = 2 .. 16 entirely, and the last four passes of every later stage -- one shared-memory round trip per
        // stage instead of four.  The passes with j >= 16 go through shared memory, one thread per compare-exchange pair.
        unsigned long long v[MR_E];
        const int base = threadIdx.x * MR_E, pb = mr_sk(base);
#pragma unroll
        for (int e = 0; e < MR_E; ++e) v[e] = pairs[pb + e];
        mr_local_passes<1>(v, base, 2);
        mr_local_passes<2>(v, base, 4);
        mr_local_passes<4>(v, base, 8);
        mr_local_passes<8>(v, base, 16);
#pragma unroll
        for (int e = 0; e < MR_E; ++e) pairs[pb + e] = v[e];
        __syncthreads();
        for (int kk = 32; kk <= npad; kk <<= 1) {
            for (int j = kk >> 1; j >= MR_E; j >>= 1) {
                for (int p = threadIdx.x; p < (npad >> 1); p += MR_THREADS) {
                    const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1));       // p with a zero inserted at bit log2(j)
                    const int pi = mr_sk(i), pj = mr_sk(i | j);
                    const unsigned long long a = pairs[pi], b = pairs[pj];
                    if ((a > b) == ((i & kk) == 0)) { pairs[pi] = b; pairs[pj] = a; }
                }
                __syncthreads();
            }
#pragma unroll
            for (int e = 0; e < MR_E; ++e) v[e] = pairs[pb + e];
            mr_local_passes<8>(v, base, kk);
#pragma unroll
            for (int e = 0; e < MR_E; ++e) pairs[pb + e] = v[e];
            __syncthreads();
        }
    } else {
        for (int kk = 2; kk <= npad; kk <<= 1) {
            for (int j = kk >> 1; j > 0; j >>= 1) {
                for (int p = threadIdx.x; p < (npad >> 1); p += MR_THREADS) {  // one thread per compare-exchange pair
                    const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1));
                    const int pi = mr_sk(i), pj = mr_sk(i | j);
                    const unsigned long long a = pairs[pi], b = pairs[pj];
                    if ((a > b) == ((i & kk) == 0)) { pairs[pi] = b; pairs[pj] = a; }
                }
                __syncthreads();
            }
        }
    }
    for (int r = threadIdx.x; r < n; r += MR_THREADS) rank_of[(unsigned)(pairs[mr_sk(r)] & 0xffffffffu)] = (unsigned short)r;
    const int lane = threadIdx.x & 31, ty = threadIdx.x >> 5;
    unsigned* bm = bitmaps + ty * (wpl * 32);
    for (int i = lane; i < wpl * 32; i += 32) bm[i] = 0u;
    __syncthreads();
    const int y = y0 + ty;
    if (y >= H) return;
    // first window of this output row
    for (int q = lane; q < k * k; q += 32) {
        const int dy = q / k, dx = q - dy * k;
        const unsigned r = rank_of[(ty + dy) * RW + dx];
        atomicOr(&bm[r >> 5], 1u << (r & 31));
    }
    __syncwarp();
    const int xe = min(MR_TW, W - x0);
    // The median's position in rank space moves little from one window to the next, so the warp TRACKS it instead of recounting the
    // whole bitmap per pixel: `ob` = the block of wpl words (one lane's share) that holds the wanted set bit, `excl` = set bits in the
    // blocks before it, kept up to date from the ranks that leave / enter the window (two ballots per update round); per pixel only
    // block ob is counted (one word per lane, redux add) and searched.
    const int bshift = 5 + (wpl == 8 ? 3 : wpl == 4 ? 2 : wpl == 2 ? 1 : 0);      // log2(bits per block) when wpl is a power of two
    const bool pow2 = (wpl & (wpl - 1)) == 0;
    auto block_of = [&](unsigned r) { return pow2 ? (int)(r >> bshift) : (int)(r / (32u * wpl)); };
    unsigned wv = 0;                                                               // lane < wpl: word `lane` of block ob
    auto count_block = [&](int b) {
        wv = lane < wpl ? bm[b * wpl + lane] : 0u;
        return (int)__reduce_add_sync(0xffffffffu, (unsigned)__popc(wv));
    };
    int ob = 0, excl = 0;
    for (int tx = 0; tx < xe; ++tx) {
        if (tx > 0) {   // slide: drop column tx-1, add column tx+k-1
            int delta = 0;
            for (int d0 = 0; d0 < k; d0 += 32) {
                const int dy = d0 + lane;
                bool below_r = false, below_a = false;
                if (dy < k) {
                    const unsigned rr = rank_of[(ty + dy) * RW + tx - 1];
                    atomicAnd(&bm[rr >> 5], ~(1u << (rr & 31)));
                    const unsigned ra = rank_of[(ty + dy) * RW + tx + k - 1];
                    atomicOr(&bm[ra >> 5], 1u << (ra & 31));
                    below_r = block_of(rr) < ob;
                    below_a = block_of(ra) < ob;
                }
                delta += __popc(__ballot_sync(0xffffffffu, below_a)) - __popc(__ballot_sync(0xffffffffu, below_r));
            }
            excl += delta;
            __syncwarp();
        }
        while (rank < excl) {                         // the wanted bit moved into an earlier block
            --ob;
            excl -= count_block(ob);
        }
        int c = count_block(ob);
        while (rank >= excl + c) {                    // ... or into a later one
            excl += c;
            ++ob;
            c = count_block(ob);
        }
        // (rank - excl)-th set bit (0-based) of block ob: word by an inclusive scan of the lanes' popcounts, bit by popcount bisection
        const int pc = __popc(wv);
        int incl = pc;
        for (int o = 1; o < 8; o <<= 1) {             // wpl <= 8 (region <= 8192 samples)
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        const int need = rank - excl - (incl - pc);
        if (lane < wpl && need >= 0 && need < pc) {
            unsigned bit = 0;
            int nd = need;
#pragma unroll
            for (int sft = 16; sft >= 1; sft >>= 1) {
                const int cc = __popc((wv >> bit) & ((1u << sft) - 1u));
                if (nd >= cc) { nd -= cc; bit += sft; }
            }
            const int r = ((ob * wpl + lane) << 5) + (int)bit;
            out[(size_t)blockIdx.z * plane + (size_t)y * W + x0 + tx] = key2f((unsigned)(pairs[mr_sk(r)] >> 32));
        }
        __syncwarp();
    }
}

constexpr int MED_T = 16;

__global__ void __launch_bounds__(MED_T * MED_T) median_bisect_kernel(const float* __restrict__ in, float* __restrict__ out,
                                                                      int H, int W, int k, int rank) {
    extern __shared__ unsigned keys[];
    const int S = MED_T + k - 1;
    const int x0 = blockIdx.x * MED_T, y0 = blockIdx.y * MED_T;
    const size_t plane = (size_t)H * W;
    const float* src = in + (size_t)blockIdx.z * plane;
    const int lo_off = k / 2;
    for (int q = threadIdx.x; q < S * S; q += blockDim.x) {
        const int r = q / S, c = q - r * S;
        keys[q] = f2key(src[(size_t)reflect_idx(y0 + r - lo_off, H) * W + reflect_idx(x0 + c - lo_off, W)]);
    }
    __syncthreads();
    const int tx = threadIdx.x % MED_T, ty = threadIdx.x / MED_T;
    const int x = x0 + tx, y = y0 + ty;
    if (x >= W || y >= H) return;
    const unsigned* base = keys + ty * S + tx;
    unsigned lo = 0u, hi = 0xffffffffu;   // smallest v with count(key <= v) >= rank + 1
    while (lo < hi) {
        const unsigned mid = lo + ((hi - lo) >> 1);
        int cnt = 0;
        for (int r = 0; r < k; ++r) {
            const unsigned* row = base + r * S;
            for (int c = 0; c < k; ++c) cnt += (row[c] <= mid);
        }
        if (cnt >= rank + 1) hi = mid; else lo = mid + 1;
    }
    out[(size_t)blockIdx.z * plane + (size_t)y * W + x] = key2f(lo);
}

}  // namespace fvfi

using namespace fvfi;

extern "C" int fvfi_rgb2lab(const float* rgb, float* lab, int B, int H, int W, void* stream) {
    FVFI_CHECK_ARG(rgb && lab && B > 0 && H > 0 && W > 0 && B <= 65535, "rgb2lab: bad argument");
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), B);
    rgb2lab_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rgb, lab, plane, B);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_rgb8_to_rgb_lab(const uint8_t* rgb8, float* rgb, float* lab, int T, int H, int W, void* stream) {
    FVFI_CHECK_ARG(rgb8 && rgb && lab, "fvfi_rgb8_to_rgb_lab: null pointer");
    FVFI_CHECK_ARG(T > 0 && H > 0 && W > 0 && T <= 65535, "fvfi_rgb8_to_rgb_lab: bad size T=%d H=%d W=%d", T, H, W);
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), T);
    rgb8_to_rgb_lab_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(rgb8, rgb, lab, plane);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_lab2rgb(const float* lab, float* rgb, int B, int H, int W, void* stream) {
    FVFI_CHECK_ARG(rgb && lab && B > 0 && H > 0 && W > 0 && B <= 65535, "lab2rgb: bad argument");
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), B);
    lab2rgb_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(lab, rgb, plane, B);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_gaussian_filter(const float* in, float* out, float* tmp, int N, int H, int W, float sigma,
                                    void* stream) {
    FVFI_CHECK_ARG(in && out && tmp && N > 0 && H > 0 && W > 0 && N <= 65535 && sigma > 0.f, "gaussian_filter: bad argument");
    const int radius = (int)(4.0f * sigma + 0.5f);  // scipy: truncate = 4.0
    FVFI_CHECK_ARG(radius <= GAUSS_MAX_RADIUS, "gaussian_filter: sigma too large (radius %d > %d)", radius, GAUSS_MAX_RADIUS);
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), N);
    // scipy filters axis 0 (rows, i.e. along y) first, then axis 1
    if (radius == 20 && H > 20 && W > 20) {            // the recipe's sigma = 5: register-weight kernels (bit-identical to the generic ones)
        gauss_y_fast_kernel<20><<<dim3(ceil_div(W, 128), ceil_div(H, GR), N), 128, 0, (cudaStream_t)stream>>>(in, tmp, H, W, sigma);
        FVFI_LAUNCH_CHECK();
        gauss_x_fast_kernel<20><<<dim3(ceil_div(W, GAUSS_XT), H, N), GAUSS_XT / GX, 0, (cudaStream_t)stream>>>(tmp, out, H, W, sigma);
        FVFI_LAUNCH_CHECK();
        return FVFI_OK;
    }
    gauss1d_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(in, tmp, H, W, sigma, radius);
    FVFI_LAUNCH_CHECK();
    gauss1d_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(tmp, out, H, W, sigma, radius);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_median_filter(const float* in, float* out, int N, int H, int W, int size, void* stream) {
    FVFI_CHECK_ARG(in && out && N > 0 && H > 0 && W > 0 && N <= 65535, "median_filter: bad argument");
    FVFI_CHECK_ARG(size >= 1 && size <= 96, "median_filter: size must be 1..96");
    const int rank = (size * size) / 2;
    // widest tile whose region fits the sorting network, evened out over the row of tiles
    int tw = MR_MAX_N / (MR_TH + size - 1) - (size - 1);
    if (tw > W) tw = W;
    if (tw >= 1) tw = ceil_div(W, ceil_div(W, tw));
    const int MR_TW = tw;
    const int n = (MR_TW + size - 1) * (MR_TH + size - 1);
    if (MR_TW >= 8 && n <= MR_MAX_N) {
        int npad = 1;
        while (npad < n) npad <<= 1;
        const int nwords = (n + 31) / 32, wpl = (nwords + 31) / 32;
        const size_t smem = (size_t)(npad + (npad >> 4)) * 8 + (size_t)((n + 7) & ~7) * 2 + (size_t)MR_TH * wpl * 32 * 4;
        if (smem > 48 * 1024)
            FVFI_SMEM_OPT_IN(median_rank_kernel, smem);
        dim3 grid(ceil_div(W, MR_TW), ceil_div(H, MR_TH), N);
        median_rank_kernel<<<grid, MR_THREADS, smem, (cudaStream_t)stream>>>(in, out, H, W, size, rank, npad, MR_TW);
        FVFI_LAUNCH_CHECK();
        return FVFI_OK;
    }
    const int S = MED_T + size - 1;
    const size_t smem = (size_t)S * S * sizeof(unsigned);
    if (smem > 48 * 1024)
        FVFI_SMEM_OPT_IN(median_bisect_kernel, smem);
    dim3 grid(ceil_div(W, MED_T), ceil_div(H, MED_T), N);
    median_bisect_kernel<<<grid, MED_T * MED_T, smem, (cudaStream_t)stream>>>(in, out, H, W, size, rank);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

// ---- bilinear resize on NHWC tensors ------------------------------------------------------------------
// torch.nn.Upsample / F.interpolate(mode='bilinear') as the three networks use it: scale 2 with
// align_corners=True (KernelEstimation, fusion_adacofnet.py:31), scale 2 with align_corners=False (FusionNet,
// fusion_net.py:41) and arbitrary output size with align_corners=False (PhaseNet, phase_net.py:138-139).
// One thread = one output pixel x 4 channels (float4); the output may be a channel slice of a wider NHWC
// buffer (y_pixel_stride), which is how PhaseNet's 88-channel concat is assembled without torch.cat.
namespace fvfi {
__device__ __forceinline__ void ldg256f(const float* p, float* v) {      // sm_100 256-bit global load (one sector per lane)
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]), "=f"(v[4]), "=f"(v[5]), "=f"(v[6]), "=f"(v[7])
                 : "l"(p));
}
__device__ __forceinline__ void stg256f(float* p, const float* v) {
    asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
                 "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
                 : "memory");
}

// VEC = channels per thread: 8 (256-bit accesses), 4 (128-bit) or 1 (any stride / alignment).
// grid = (column x channel-group blocks, output rows, images): the row coordinates are uniform per block and nothing is divided
// per thread when the number of channel groups is a power of two (cg_shift >= 0).
template <int VEC>
__global__ void __launch_bounds__(256) resize_bilinear_nhwc_kernel(const float* __restrict__ x, float* __restrict__ y, int Hi,
                                                                   int Wi, int Ho, int Wo, int C, int ldx, int ldy,
                                                                   float sy, float sx, int align_corners,
                                                                   const float* __restrict__ addend, int lda, int relu_in,
                                                                   int cg_n, int cg_shift) {
    const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
    const int ox = cg_shift >= 0 ? (int)(q >> cg_shift) : (int)(q / (unsigned)cg_n);
    if (ox >= Wo) return;
    const int ch = (int)(q - (unsigned)ox * (unsigned)cg_n) * VEC;
    const int oy = blockIdx.y, n = blockIdx.z;
    const size_t p = (size_t)oy * Wo + ox;
    // source coordinates exactly as ATen's area_pixel_compute_source_index
    int y0, y1, x0, x1;
    float ly, lx;
    bilinear_src(oy, sy, align_corners, Hi, y0, y1, ly);
    bilinear_src(ox, sx, align_corners, Wi, x0, x1, lx);
    const float hy = 1.f - ly, hx = 1.f - lx;
    const float* X = x + (size_t)n * Hi * Wi * ldx;
    const float* p00 = X + ((size_t)y0 * Wi + x0) * ldx + ch;
    const float* p01 = X + ((size_t)y0 * Wi + x1) * ldx + ch;
    const float* p10 = X + ((size_t)y1 * Wi + x0) * ldx + ch;
    const float* p11 = X + ((size_t)y1 * Wi + x1) * ldx + ch;
    float* dst = y + ((size_t)n * Ho * Wo + p) * ldy + ch;
    float a[VEC], b[VEC], c[VEC], d[VEC], o[VEC], e[VEC];
    const float* ap = addend ? addend + ((size_t)n * Ho * Wo + p) * lda + ch : nullptr;
    if (VEC == 8) {
        ldg256f(p00, a); ldg256f(p01, b); ldg256f(p10, c); ldg256f(p11, d);
        if (ap) ldg256f(ap, e);
    } else if (VEC == 4) {
        const float4 a4 = __ldg((const float4*)p00), b4 = __ldg((const float4*)p01), c4 = __ldg((const float4*)p10),
                     d4 = __ldg((const float4*)p11);
        a[0] = a4.x; a[1] = a4.y; a[2] = a4.z; a[3] = a4.w;
        b[0] = b4.x; b[1] = b4.y; b[2] = b4.z; b[3] = b4.w;
        c[0] = c4.x; c[1] = c4.y; c[2] = c4.z; c[3] = c4.w;
        d[0] = d4.x; d[1] = d4.y; d[2] = d4.z; d[3] = d4.w;
        if (ap) {
            const float4 e4 = __ldg((const float4*)ap);
            e[0] = e4.x; e[1] = e4.y; e[2] = e4.z; e[3] = e4.w;
        }
    } else {
        a[0] = __ldg(p00); b[0] = __ldg(p01); c[0] = __ldg(p10); d[0] = __ldg(p11);
        if (ap) e[0] = __ldg(ap);
    }
    if (relu_in) {                      // Upsample(ReLU(x)): the activation applies to the source samples (fusion_net.py:61)
#pragma unroll
        for (int i = 0; i < VEC; ++i) { a[i] = fmaxf(a[i], 0.f); b[i] = fmaxf(b[i], 0.f); c[i] = fmaxf(c[i], 0.f); d[i] = fmaxf(d[i], 0.f); }
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) o[i] = bilerp(hy, hx, ly, lx, a[i], b[i], c[i], d[i]);
    if (ap) {                           // + skip connection (fusion_net.py:62)
#pragma unroll
        for (int i = 0; i < VEC; ++i) o[i] += e[i];
    }
    if (VEC == 8) stg256f(dst, o);
    else if (VEC == 4) *(float4*)dst = make_float4(o[0], o[1], o[2], o[3]);
    else dst[0] = o[0];
}

// nn.AvgPool2d(2, 2) on NHWC storage (src/fusion_net/fusion_adacofnet.py:62-70): one thread = one output pixel x VEC channels
// MAX: nn.MaxPool2d(2, stride=2) (FusionNet's encoder, src/fusion_net/fusion_net.py:39,56)
template <int VEC, bool MAX = false>
__global__ void __launch_bounds__(256) avg_pool2_nhwc_kernel(const float* __restrict__ x, float* __restrict__ y, int Hi, int Wi,
                                                             int C, int ldx, int ldy) {
    const int Ho = Hi >> 1, Wo = Wi >> 1;
    const unsigned cg_n = (unsigned)(C + VEC - 1) / VEC;
    const unsigned total = (unsigned)Ho * (unsigned)Wo * cg_n;
    const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= total) return;
    const unsigned p = q / cg_n;
    const int ch = (int)(q - p * cg_n) * VEC;
    const int oy = (int)(p / (unsigned)Wo), ox = (int)(p - (unsigned)oy * (unsigned)Wo);
    const int n = blockIdx.y;
    const float* p00 = x + (((size_t)n * Hi + 2 * oy) * Wi + 2 * ox) * ldx + ch;
    const float* p10 = p00 + (size_t)Wi * ldx;
    float* dst = y + ((size_t)n * Ho * Wo + p) * ldy + ch;
    float a[VEC], b[VEC], c[VEC], d[VEC], o[VEC];
    if (VEC == 8) {
        ldg256f(p00, a); ldg256f(p00 + ldx, b); ldg256f(p10, c); ldg256f(p10 + ldx, d);
    } else {
        a[0] = __ldg(p00); b[0] = __ldg(p00 + ldx); c[0] = __ldg(p10); d[0] = __ldg(p10 + ldx);
    }
#pragma unroll
    for (int i = 0; i < VEC; ++i) o[i] = MAX ? fmaxf(fmaxf(a[i], b[i]), fmaxf(c[i], d[i])) : ((a[i] + b[i]) + (c[i] + d[i])) * 0.25f;
    if (VEC == 8) stg256f(dst, o);
    else dst[0] = o[0];
}
// planar [B,C,H,W] -> channel slice of an NHWC buffer (PhaseNet's concat assembly, src/phase_net/phase_net.py:141):
// coalesced plane reads, one contiguous C-float store per pixel (256-bit when C == 8)
__global__ void __launch_bounds__(256) nchw_to_nhwc_slice_kernel(const float* __restrict__ x, float* __restrict__ y, int C,
                                                                 size_t plane, int ldy) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= plane) return;
    const int n = blockIdx.y;
    const float* src = x + (size_t)n * C * plane + p;
    float* dst = y + ((size_t)n * plane + p) * ldy;
    if (C == 8 && (ldy & 7) == 0 && ((((size_t)y) & 31) == 0)) {
        float v[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) v[c] = __ldg(src + (size_t)c * plane);
        stg256f(dst, v);
    } else {
        for (int c = 0; c < C; ++c) dst[c] = __ldg(src + (size_t)c * plane);
    }
}

// ---- PhaseNet glue (src/train/utils.py:47-127, src/phase_net/phase_net.py:42-105,141,155-156) --------------------------------
// Input side: the decomposition of the frames (channel = plane*nb + band; frame 2 of pair-plane p is plane p + q: q = P for
// [frame-1 planes | frame-2 planes], q = 3 for a clip of consecutive frames decomposed once) goes straight
// into the 4*nb value channels of the NHWC concat of planes [p0, p0+pc):  [phase_1 | phase_2] / pi,  [amp_1 | amp_2] / den[p]
// (den = per-plane max over both frames + eps, from the decomposition's own epilogue) -- separate_vals, get_concat_layers_inf,
// normalize_vals and the concat in ONE pass over the planes (the reference materialises each of them).
template <int NB>
__global__ void __launch_bounds__(256) phasenet_assemble_kernel(const float* __restrict__ phase, const float* __restrict__ amp,
                                                                const float* __restrict__ den, float* __restrict__ y, size_t plane,
                                                                int ldy, int q, int p0) {
    const size_t px = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= plane) return;
    const int p = p0 + blockIdx.y;
    const float* ph1 = phase + (size_t)p * NB * plane + px;
    const float* ph2 = phase + (size_t)(q + p) * NB * plane + px;
    const float* am1 = amp + (size_t)p * NB * plane + px;
    const float* am2 = amp + (size_t)(q + p) * NB * plane + px;
    const float d = __ldg(den + p);
    float v[4 * NB];
#pragma unroll
    for (int c = 0; c < NB; ++c) {
        v[c] = __ldcs(ph1 + (size_t)c * plane) / 3.14159265358979323846f;             // x / math.pi        (phase_net.py:64)
        v[NB + c] = __ldcs(ph2 + (size_t)c * plane) / 3.14159265358979323846f;
        v[2 * NB + c] = __ldg(am1 + (size_t)c * plane) / d;                           // amplitude / max    (phase_net.py:54-57)
        v[3 * NB + c] = __ldg(am2 + (size_t)c * plane) / d;
    }
    float* dst = y + ((size_t)blockIdx.y * plane + px) * ldy;
    if (NB == 4 && (ldy & 7) == 0 && ((((size_t)y) & 31) == 0)) {
        stg256f(dst, v);
        stg256f(dst + 8, v + 8);
    } else {
#pragma unroll
        for (int c = 0; c < 4 * NB; ++c) dst[c] = v[c];
    }
}

// Output side: prediction [pc, 2*nb, h, w] NHWC (tanh outputs) + the RAW amplitudes -> phase_out = pred[:nb] * pi,
// amp_out = beta * amp_2 + (1 - beta) * amp_1 with beta = (pred[nb:] + 1) / 2, at channel (p0+p)*nb + b of the [P*nb,1,h,w]
// outputs: the amplitude blend (phase_net.py:155-156) and reverse_normalize (:80-105) in one pass; normalising by the common
// per-plane maximum and multiplying it back afterwards is the identity up to rounding, so the raw amplitudes are blended.
template <int NB>
__global__ void __launch_bounds__(256) phasenet_outputs_kernel(const float* __restrict__ pred, int ldp, const float* __restrict__ amp,
                                                               float* __restrict__ phase_out, float* __restrict__ amp_out,
                                                               size_t plane, int q, int p0) {
    const size_t px = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (px >= plane) return;
    const int p = p0 + blockIdx.y;
    const float* pr = pred + ((size_t)blockIdx.y * plane + px) * ldp;
    float v[2 * NB];
    if (NB == 4 && (ldp & 7) == 0 && ((((size_t)pred) & 31) == 0)) ldg256f(pr, v);
    else {
#pragma unroll
        for (int c = 0; c < 2 * NB; ++c) v[c] = __ldg(pr + c);
    }
#pragma unroll
    for (int c = 0; c < NB; ++c) {
        const size_t o = ((size_t)p * NB + c) * plane + px;
        const float a1 = __ldg(amp + o), a2 = __ldg(amp + ((size_t)(q + p) * NB + c) * plane + px);
        const float beta = (v[NB + c] + 1.f) / 2.f;
        __stcs(phase_out + o, v[c] * 3.14159265358979323846f);
        __stcs(amp_out + o, beta * a2 + (1.f - beta) * a1);
    }
}

// ---- AdaCoFNet.forward input preparation (src/fusion_net/fusion_adacofnet.py:176-196, src/adacof/utility.py:86-87) ------------
// One pass over the two frames replaces  F.pad(reflect, bottom/right to multiples of 32) x2 -> moduleNormalize x2 -> cat -> NHWC
// (KernelEstimation's input, 6 channels + 2 zero channels)  and  ReplicationPad2d(kpad) x2  (the frames the warp samples):
//   x[b][y][x][0..2] = f0 - mean, [3..5] = f2 - mean, [6..7] = 0          for (y, x) in the reflect-padded Hp x Wp frame
//   p0 / p2[b][c][y'][x'] = reflect-padded frame at clamp(y' - kpad), clamp(x' - kpad)      (un-normalised, :195)
__global__ void __launch_bounds__(256) adacofnet_prep_kernel(const float* __restrict__ f0, const float* __restrict__ f2,
                                                             float* __restrict__ x, float* __restrict__ p0, float* __restrict__ p2,
                                                             int H, int W, int Hp, int Wp, int kpad, float m0, float m1, float m2) {
    const int Hq = Hp + 2 * kpad, Wq = Wp + 2 * kpad;
    const unsigned q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= (unsigned)Hq * (unsigned)Wq) return;
    const int yq = (int)(q / (unsigned)Wq), xq = (int)(q - (unsigned)yq * (unsigned)Wq);
    const int b = blockIdx.y;
    const int yp = min(max(yq - kpad, 0), Hp - 1), xp = min(max(xq - kpad, 0), Wp - 1);      // replicate (clamp)
    const int ys = yp < H ? yp : 2 * (H - 1) - yp, xs = xp < W ? xp : 2 * (W - 1) - xp;      // torch 'reflect' at the far edges
    const size_t plane = (size_t)H * W, planeq = (size_t)Hq * Wq;
    const size_t src = (size_t)b * 3 * plane + (size_t)ys * W + xs, dst = (size_t)b * 3 * planeq + q;
    float a[3], c[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
        a[ch] = __ldg(f0 + src + ch * plane);
        c[ch] = __ldg(f2 + src + ch * plane);
        p0[dst + ch * planeq] = a[ch];
        p2[dst + ch * planeq] = c[ch];
    }
    if (yq - kpad == yp && xq - kpad == xp) {                       // interior of the padded frame: KernelEstimation's input pixel
        float v[8] = {a[0] - m0, a[1] - m1, a[2] - m2, c[0] - m0, c[1] - m1, c[2] - m2, 0.f, 0.f};
        stg256f(x + (((size_t)b * Hp + yp) * Wp + xp) * 8, v);
    }
}

}  // namespace fvfi

extern "C" int fvfi_adacofnet_prep(const float* frame0, const float* frame2, float* x_nhwc8, float* padded0, float* padded2, int B,
                                   int H, int W, int Hp, int Wp, int kpad, const float* mean3_host, void* stream) {
    FVFI_CHECK_ARG(frame0 && frame2 && x_nhwc8 && padded0 && padded2 && mean3_host && B > 0 && B <= 65535 && H > 1 && W > 1,
                   "adacofnet_prep: bad argument");
    FVFI_CHECK_ARG(Hp >= H && Wp >= W && Hp - H < H && Wp - W < W && kpad >= 0, "adacofnet_prep: reflect padding must be smaller than the frame");
    FVFI_CHECK_ARG((((size_t)x_nhwc8) & 31) == 0, "adacofnet_prep: the NHWC output must be 32-byte aligned");
    const size_t total = (size_t)(Hp + 2 * kpad) * (Wp + 2 * kpad);
    FVFI_CHECK_ARG(total < (1ull << 32) - 256, "adacofnet_prep: frame too large");
    dim3 grid((unsigned)((total + 255) / 256), B);
    fvfi::adacofnet_prep_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(frame0, frame2, x_nhwc8, padded0, padded2, H, W, Hp, Wp, kpad,
                                                                        mean3_host[0], mean3_host[1], mean3_host[2]);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

// Shared launches of the two glue kernels: the pair entry points pass N = 2P, q = P; the _offset ones take N and q from the caller.
static int phasenet_assemble_launch(const char* name, const float* phase, const float* amp, const float* den, float* y,
                                    int y_pixel_stride, int N, int P, int q, int p0, int pc, int nb, int H, int W, void* stream) {
    FVFI_CHECK_ARG(phase && amp && den && y, "%s: null pointer", name);
    FVFI_CHECK_ARG(P > 0 && p0 >= 0 && pc > 0 && p0 + pc <= P && pc <= 65535 && H > 0 && W > 0, "%s: bad argument", name);
    FVFI_CHECK_ARG(q > 0 && (long long)p0 + pc - 1 + q < (long long)N, "%s: frame-2 plane offset q=%d out of range (N=%d, p0=%d, pc=%d)",
                   name, q, N, p0, pc);
    FVFI_CHECK_ARG(nb == 4, "%s: nbands must be 4 (got %d)", name, nb);
    FVFI_CHECK_ARG(y_pixel_stride >= 4 * nb, "%s: pixel stride smaller than 4*nbands", name);
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), pc);
    fvfi::phasenet_assemble_kernel<4><<<grid, 256, 0, (cudaStream_t)stream>>>(phase, amp, den, y, plane, y_pixel_stride, q, p0);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

static int phasenet_outputs_launch(const char* name, const float* pred, int pred_pixel_stride, const float* amp, float* phase_out,
                                   float* amp_out, int N, int P, int q, int p0, int pc, int nb, int H, int W, void* stream) {
    FVFI_CHECK_ARG(pred && amp && phase_out && amp_out, "%s: null pointer", name);
    FVFI_CHECK_ARG(P > 0 && p0 >= 0 && pc > 0 && p0 + pc <= P && pc <= 65535 && H > 0 && W > 0, "%s: bad argument", name);
    FVFI_CHECK_ARG(q > 0 && (long long)p0 + pc - 1 + q < (long long)N, "%s: frame-2 plane offset q=%d out of range (N=%d, p0=%d, pc=%d)",
                   name, q, N, p0, pc);
    FVFI_CHECK_ARG(nb == 4, "%s: nbands must be 4 (got %d)", name, nb);
    FVFI_CHECK_ARG(pred_pixel_stride >= 2 * nb, "%s: pixel stride smaller than 2*nbands", name);
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), pc);
    fvfi::phasenet_outputs_kernel<4><<<grid, 256, 0, (cudaStream_t)stream>>>(pred, pred_pixel_stride, amp, phase_out, amp_out, plane, q,
                                                                             p0);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_phasenet_assemble(const float* phase, const float* amp, const float* den, float* y, int y_pixel_stride, int P,
                                      int p0, int pc, int nb, int H, int W, void* stream) {
    return phasenet_assemble_launch("phasenet_assemble", phase, amp, den, y, y_pixel_stride, 2 * P, P, P, p0, pc, nb, H, W, stream);
}

extern "C" int fvfi_phasenet_outputs(const float* pred, int pred_pixel_stride, const float* amp, float* phase_out, float* amp_out,
                                     int P, int p0, int pc, int nb, int H, int W, void* stream) {
    return phasenet_outputs_launch("phasenet_outputs", pred, pred_pixel_stride, amp, phase_out, amp_out, 2 * P, P, P, p0, pc, nb, H, W,
                                   stream);
}

extern "C" int fvfi_phasenet_assemble_offset(const float* phase, const float* amp, const float* den, float* y, int y_pixel_stride,
                                             int N, int P, int q, int p0, int pc, int nb, int H, int W, void* stream) {
    return phasenet_assemble_launch("fvfi_phasenet_assemble_offset", phase, amp, den, y, y_pixel_stride, N, P, q, p0, pc, nb, H, W,
                                    stream);
}

extern "C" int fvfi_phasenet_outputs_offset(const float* pred, int pred_pixel_stride, const float* amp, float* phase_out, float* amp_out,
                                            int N, int P, int q, int p0, int pc, int nb, int H, int W, void* stream) {
    return phasenet_outputs_launch("fvfi_phasenet_outputs_offset", pred, pred_pixel_stride, amp, phase_out, amp_out, N, P, q, p0, pc, nb,
                                   H, W, stream);
}

// torch.cat of planar [B,c_s,H,W] tensors along the channels, written as ONE NHWC tensor (FusionNet's input,
// src/fusion_net/fusion_net.py:47: cat([base, adacof, phase, other, maps], 1)): a thread owns a pixel, reads its NQ*4 channel planes
// (coalesced across the warp) and stores the record as NQ 128-bit words; channels beyond the concatenation are written as zeros.
namespace fvfi {
struct ConcatTable {
    const float* ptr[32];        // plane 0 of the source that supplies channel j (null: zero)
    unsigned long long bstride[32];   // floats between consecutive batch items of that source
};
template <int NQ>
__global__ void __launch_bounds__(256) planar_concat_nhwc_kernel(const ConcatTable T, float* __restrict__ y, size_t plane, int ldy) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= plane) return;
    const int b = blockIdx.y;
    float v[4 * NQ];
#pragma unroll
    for (int j = 0; j < 4 * NQ; ++j) v[j] = T.ptr[j] ? ld_stream(T.ptr[j] + (size_t)b * T.bstride[j] + p) : 0.f;
    float4* dst = reinterpret_cast<float4*>(y + ((size_t)b * plane + p) * ldy);
#pragma unroll
    for (int q = 0; q < NQ; ++q) dst[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}
}  // namespace fvfi

extern "C" int fvfi_planar_concat_nhwc(const float* const* sources, const int* channels, int nsources, float* y, int y_pixel_stride,
                                       int B, int H, int W, void* stream) {
    FVFI_CHECK_ARG(sources && channels && nsources > 0 && y && B > 0 && H > 0 && W > 0 && B <= 65535, "planar_concat_nhwc: bad argument");
    fvfi::ConcatTable T{};
    const size_t plane = (size_t)H * W;
    int C = 0;
    for (int s = 0; s < nsources; ++s) {
        FVFI_CHECK_ARG(sources[s] && channels[s] > 0 && C + channels[s] <= 32, "planar_concat_nhwc: null source or more than 32 channels");
        for (int c = 0; c < channels[s]; ++c, ++C) {
            T.ptr[C] = sources[s] + (size_t)c * plane;
            T.bstride[C] = (unsigned long long)channels[s] * plane;
        }
    }
    const int nq = (C + 3) / 4;
    FVFI_CHECK_ARG((y_pixel_stride % 4) == 0 && y_pixel_stride >= 4 * nq && (((size_t)y) & 15) == 0,
                   "planar_concat_nhwc: y needs a pixel stride that is a multiple of 4 and >= the channel count rounded up to 4, 16-byte aligned");
    dim3 grid((unsigned)((plane + 255) / 256), B);
    cudaStream_t st = (cudaStream_t)stream;
    switch (nq) {
#define FVFI_PC(N) case N: fvfi::planar_concat_nhwc_kernel<N><<<grid, 256, 0, st>>>(T, y, plane, y_pixel_stride); break;
        FVFI_PC(1) FVFI_PC(2) FVFI_PC(3) FVFI_PC(4) FVFI_PC(5) FVFI_PC(6) FVFI_PC(7) FVFI_PC(8)
#undef FVFI_PC
    }
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_nchw_to_nhwc_slice(const float* x, float* y, int y_pixel_stride, int B, int C, int H, int W, void* stream) {
    FVFI_CHECK_ARG(x && y && B > 0 && C > 0 && H > 0 && W > 0 && B <= 65535 && y_pixel_stride >= C, "nchw_to_nhwc_slice: bad argument");
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), B);
    fvfi::nchw_to_nhwc_slice_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, y, C, plane, y_pixel_stride);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_resize_bilinear_nhwc(const float* x, int x_pixel_stride, float* y, int y_pixel_stride, int B, int Hi, int Wi,
                                         int Ho, int Wo, int C, int align_corners, void* stream) {
    return fvfi_resize_bilinear_nhwc_fused(x, x_pixel_stride, nullptr, 0, y, y_pixel_stride, B, Hi, Wi, Ho, Wo, C, align_corners, 0, stream);
}

extern "C" int fvfi_resize_bilinear_nhwc_fused(const float* x, int x_pixel_stride, const float* addend, int addend_pixel_stride,
                                               float* y, int y_pixel_stride, int B, int Hi, int Wi, int Ho, int Wo, int C,
                                               int align_corners, int relu_input, void* stream) {
    FVFI_CHECK_ARG(x && y && B > 0 && Hi > 0 && Wi > 0 && Ho > 0 && Wo > 0 && C > 0 && B <= 65535, "resize_bilinear: bad argument");
    FVFI_CHECK_ARG(x_pixel_stride >= C && y_pixel_stride >= C, "resize_bilinear: pixel stride smaller than channel count");
    FVFI_CHECK_ARG(!addend || addend_pixel_stride >= C, "resize_bilinear: addend pixel stride smaller than channel count");
    const size_t addbits = addend ? ((size_t)addend | ((size_t)addend_pixel_stride * 4)) : 0;
    const int lda = addend_pixel_stride, relu_in = relu_input ? 1 : 0;
    const float sy = fvfi::bilinear_scale(Hi, Ho, align_corners), sx = fvfi::bilinear_scale(Wi, Wo, align_corners);
    const bool a32 = ((((size_t)x) | ((size_t)y) | addbits) & 31) == 0, a16 = ((((size_t)x) | ((size_t)y) | addbits) & 15) == 0;
    const int vec = (a32 && (C & 7) == 0 && (x_pixel_stride & 7) == 0 && (y_pixel_stride & 7) == 0) ? 8
                  : (a16 && (C & 3) == 0 && (x_pixel_stride & 3) == 0 && (y_pixel_stride & 3) == 0) ? 4 : 1;
    const int cg_n = (C + vec - 1) / vec;
    int cg_shift = -1;
    for (int sh = 0; sh < 16; ++sh)
        if ((1 << sh) == cg_n) cg_shift = sh;
    const size_t per_row = (size_t)Wo * cg_n;
    FVFI_CHECK_ARG(per_row < (1ull << 31) && Ho <= 65535, "resize_bilinear: image too large");
    dim3 grid((unsigned)((per_row + 255) / 256), (unsigned)Ho, (unsigned)B);
    cudaStream_t s = (cudaStream_t)stream;
    if (vec == 8)
        fvfi::resize_bilinear_nhwc_kernel<8><<<grid, 256, 0, s>>>(x, y, Hi, Wi, Ho, Wo, C, x_pixel_stride, y_pixel_stride, sy, sx, align_corners, addend, lda, relu_in, cg_n, cg_shift);
    else if (vec == 4)
        fvfi::resize_bilinear_nhwc_kernel<4><<<grid, 256, 0, s>>>(x, y, Hi, Wi, Ho, Wo, C, x_pixel_stride, y_pixel_stride, sy, sx, align_corners, addend, lda, relu_in, cg_n, cg_shift);
    else
        fvfi::resize_bilinear_nhwc_kernel<1><<<grid, 256, 0, s>>>(x, y, Hi, Wi, Ho, Wo, C, x_pixel_stride, y_pixel_stride, sy, sx, align_corners, addend, lda, relu_in, cg_n, cg_shift);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

static int pool2_nhwc(const float* x, int x_pixel_stride, float* y, int y_pixel_stride, int B, int Hi, int Wi, int C, bool is_max,
                      void* stream);
extern "C" int fvfi_max_pool2_nhwc(const float* x, int x_pixel_stride, float* y, int y_pixel_stride, int B, int Hi, int Wi, int C,
                                   void* stream) {
    return pool2_nhwc(x, x_pixel_stride, y, y_pixel_stride, B, Hi, Wi, C, true, stream);
}
extern "C" int fvfi_avg_pool2_nhwc(const float* x, int x_pixel_stride, float* y, int y_pixel_stride, int B, int Hi, int Wi, int C,
                                   void* stream) {
    return pool2_nhwc(x, x_pixel_stride, y, y_pixel_stride, B, Hi, Wi, C, false, stream);
}
static int pool2_nhwc(const float* x, int x_pixel_stride, float* y, int y_pixel_stride, int B, int Hi, int Wi, int C, bool is_max,
                      void* stream) {
    FVFI_CHECK_ARG(x && y && B > 0 && Hi > 1 && Wi > 1 && C > 0 && B <= 65535, "avg_pool2: bad argument");
    FVFI_CHECK_ARG(x_pixel_stride >= C && y_pixel_stride >= C, "avg_pool2: pixel stride smaller than channel count");
    const bool a32 = ((((size_t)x) | ((size_t)y)) & 31) == 0;
    const int vec = (a32 && (C & 7) == 0 && (x_pixel_stride & 7) == 0 && (y_pixel_stride & 7) == 0) ? 8 : 1;
    const size_t total = (size_t)(Hi / 2) * (Wi / 2) * ((C + vec - 1) / vec);
    FVFI_CHECK_ARG(total < (1ull << 32) - 256, "avg_pool2: image too large");
    dim3 grid((unsigned)((total + 255) / 256), B);
    cudaStream_t s = (cudaStream_t)stream;
    if (vec == 8 && is_max) fvfi::avg_pool2_nhwc_kernel<8, true><<<grid, 256, 0, s>>>(x, y, Hi, Wi, C, x_pixel_stride, y_pixel_stride);
    else if (vec == 8) fvfi::avg_pool2_nhwc_kernel<8, false><<<grid, 256, 0, s>>>(x, y, Hi, Wi, C, x_pixel_stride, y_pixel_stride);
    else if (is_max) fvfi::avg_pool2_nhwc_kernel<1, true><<<grid, 256, 0, s>>>(x, y, Hi, Wi, C, x_pixel_stride, y_pixel_stride);
    else fvfi::avg_pool2_nhwc_kernel<1, false><<<grid, 256, 0, s>>>(x, y, Hi, Wi, C, x_pixel_stride, y_pixel_stride);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}
