// adacof.cu -- AdaCoF adaptive-collaboration-of-flows warp for sm_100a.
//
// Replaces the four scalar CuPy/NVRTC kernels of the reference
// (src/adacof/cupy_module/adacof.py:6-258) and the torch elementwise tail of
// AdaCoFNet.forward (src/fusion_net/fusion_adacofnet.py:198-213).
//
// Arithmetic contract (SURVEY.md Appendix B): for output pixel (n,c,i,j)
//   out = sum_{k,l<F} w * ( I[r0,c0](1-a)(1-b) + I[r1,c0] a(1-b) + I[r0,c1](1-a) b + I[r1,c1] a b )
//   A=(int)alpha (TRUNCATION, adacof.py:27-28), a = alpha-A, r0 = clamp(i+k*d+A), r1 = clamp(i+k*d+A+1)
// The four bilinear weights are formed once per tap and shared by the three channels, so the
// rounding association differs from the reference expression by O(1 ulp) per term (tested
// to 2e-6 abs on [0,1] frames; the north-star tolerance is 1e-4).
//
// Kernels in this file ("direct" family): one thread owns one output pixel and ALL channels,
// so every coefficient map (w, alpha, beta) is read from HBM exactly once (the reference
// re-reads them once per channel), lanes of a warp own 32 consecutive pixels of a row so the
// 3*F*F coefficient reads are full 128 B lines, and the frame taps are gathered through the
// read-only L1/L2 path.  The smem-staged "tiled" family lives in adacof_tiled.cu.
#include <cstdlib>

#include "common.cuh"
#include "yuv.cuh"

namespace fvfi {

struct Tap {
    int r0, r1, c0, c1;
    float w00, w10, w01, w11;  // bilinear weights (NOT multiplied by w)
};

__device__ __forceinline__ Tap make_tap(float alpha, float beta, int i0, int j0, int Hin, int Win) {
    Tap t;
    const int A = (int)alpha;  // trunc toward zero -- adacof.py:27
    const int B = (int)beta;   // adacof.py:28
    const float a = alpha - (float)A;
    const float b = beta - (float)B;
    const int r = i0 + A, c = j0 + B;
    t.r0 = min(max(r, 0), Hin - 1);      // adacof.py:30-34
    t.r1 = min(max(r + 1, 0), Hin - 1);  // adacof.py:42-46
    t.c0 = min(max(c, 0), Win - 1);      // adacof.py:36-40
    t.c1 = min(max(c + 1, 0), Win - 1);  // adacof.py:48-52
    const float na = 1.0f - a, nb = 1.0f - b;
    t.w00 = na * nb;
    t.w10 = a * nb;
    t.w01 = na * b;
    t.w11 = a * b;
    return t;
}

// ---------------------------------------------------------------------------------------------
// forward, direct
// ---------------------------------------------------------------------------------------------
template <int C>
__global__ void __launch_bounds__(256)
adacof_fwd_direct(const float* __restrict__ input, const float* __restrict__ weight,
                  const float* __restrict__ off_i, const float* __restrict__ off_j,
                  float* __restrict__ out, int Hin, int Win, int H, int W, int F, int dil) {
    const int j = blockIdx.x * 32 + threadIdx.x;
    const int i = blockIdx.y * 8 + threadIdx.y;
    const int n = blockIdx.z;
    if (j >= W || i >= H) return;
    const size_t plane = (size_t)H * W, plane_in = (size_t)Hin * Win;
    const float* I = input + (size_t)n * C * plane_in;
    size_t q = (size_t)n * F * F * plane + (size_t)i * W + j;
    float acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) acc[c] = 0.f;
    for (int k = 0; k < F; ++k) {
#pragma unroll 5
        for (int l = 0; l < F; ++l, q += plane) {
            const float w = ld_stream(weight + q);
            const float al = ld_stream(off_i + q);
            const float be = ld_stream(off_j + q);
            const Tap t = make_tap(al, be, i + k * dil, j + l * dil, Hin, Win);
            const int o00 = t.r0 * Win + t.c0, o10 = t.r1 * Win + t.c0;
            const int o01 = t.r0 * Win + t.c1, o11 = t.r1 * Win + t.c1;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float* Ic = I + (size_t)c * plane_in;
                const float v = __ldg(Ic + o00) * t.w00 + __ldg(Ic + o10) * t.w10 +
                                __ldg(Ic + o01) * t.w01 + __ldg(Ic + o11) * t.w11;
                acc[c] = fmaf(w, v, acc[c]);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < C; ++c) st_stream(out + ((size_t)n * C + c) * plane + (size_t)i * W + j, acc[c]);
}

// Any channel count: channels in the outer loop (coefficients re-read per channel like the reference).
__global__ void __launch_bounds__(256)
adacof_fwd_direct_anyc(const float* __restrict__ input, const float* __restrict__ weight,
                       const float* __restrict__ off_i, const float* __restrict__ off_j,
                       float* __restrict__ out, int C, int Hin, int Win, int H, int W, int F, int dil) {
    const int j = blockIdx.x * 32 + threadIdx.x;
    const int i = blockIdx.y * 8 + threadIdx.y;
    const int n = blockIdx.z;
    if (j >= W || i >= H) return;
    const size_t plane = (size_t)H * W, plane_in = (size_t)Hin * Win;
    for (int c = 0; c < C; ++c) {
        const float* Ic = input + ((size_t)n * C + c) * plane_in;
        size_t q = (size_t)n * F * F * plane + (size_t)i * W + j;
        float acc = 0.f;
        for (int k = 0; k < F; ++k)
            for (int l = 0; l < F; ++l, q += plane) {
                const float w = __ldg(weight + q);
                const Tap t = make_tap(__ldg(off_i + q), __ldg(off_j + q), i + k * dil, j + l * dil, Hin, Win);
                const float v = __ldg(Ic + t.r0 * Win + t.c0) * t.w00 + __ldg(Ic + t.r1 * Win + t.c0) * t.w10 +
                                __ldg(Ic + t.r0 * Win + t.c1) * t.w01 + __ldg(Ic + t.r1 * Win + t.c1) * t.w11;
                acc = fmaf(w, v, acc);
            }
        out[((size_t)n * C + c) * plane + (size_t)i * W + j] = acc;
    }
}

// ---------------------------------------------------------------------------------------------
// backward, direct: gW, g_alpha, g_beta in one pass (reference: three kernels re-gathering the
// same 12 taps, adacof.py:67-258, plus four new_zeros memsets, :382-385).
//   S_xy = sum_c g_c * I_c[r_x, c_y]
//   gW     = S00 (1-a)(1-b) + S10 a(1-b) + S01 (1-a) b + S11 a b                  (:118-123)
//   gAlpha = w * ( (S10 - S00)(1-b) + (S11 - S01) b )                            (:183-188)
//   gBeta  = w * ( (S01 - S00)(1-a) + (S11 - S10) a )                            (:248-253)
// The optional true gradInput (extension; the reference returns zeros) is a separate scatter kernel below.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adacof_bwd_direct(const float* __restrict__ gout, const float* __restrict__ input,
                  const float* __restrict__ weight, const float* __restrict__ off_i,
                  const float* __restrict__ off_j, float* __restrict__ gin, float* __restrict__ gw,
                  float* __restrict__ goi, float* __restrict__ goj, int Hin, int Win, int H, int W, int F,
                  int dil) {
    constexpr int C = 3;
    const int j = blockIdx.x * 32 + threadIdx.x;
    const int i = blockIdx.y * 8 + threadIdx.y;
    const int n = blockIdx.z;
    if (j >= W || i >= H) return;
    const size_t plane = (size_t)H * W, plane_in = (size_t)Hin * Win;
    const float* I = input + (size_t)n * C * plane_in;
    float g[C];
#pragma unroll
    for (int c = 0; c < C; ++c) g[c] = ld_stream(gout + ((size_t)n * C + c) * plane + (size_t)i * W + j);
    size_t q = (size_t)n * F * F * plane + (size_t)i * W + j;
    for (int k = 0; k < F; ++k) {
#pragma unroll 5
        for (int l = 0; l < F; ++l, q += plane) {
            const float w = ld_stream(weight + q);
            const float al = ld_stream(off_i + q);
            const float be = ld_stream(off_j + q);
            const int A = (int)al, B = (int)be;
            const float a = al - (float)A, b = be - (float)B;
            const int r = i + k * dil + A, cc = j + l * dil + B;
            const int r0 = min(max(r, 0), Hin - 1), r1 = min(max(r + 1, 0), Hin - 1);
            const int c0 = min(max(cc, 0), Win - 1), c1 = min(max(cc + 1, 0), Win - 1);
            const int o00 = r0 * Win + c0, o10 = r1 * Win + c0, o01 = r0 * Win + c1, o11 = r1 * Win + c1;
            float s00 = 0.f, s10 = 0.f, s01 = 0.f, s11 = 0.f;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float* Ic = I + (size_t)c * plane_in;
                s00 = fmaf(g[c], __ldg(Ic + o00), s00);
                s10 = fmaf(g[c], __ldg(Ic + o10), s10);
                s01 = fmaf(g[c], __ldg(Ic + o01), s01);
                s11 = fmaf(g[c], __ldg(Ic + o11), s11);
            }
            const float na = 1.f - a, nb = 1.f - b;
            st_stream(gw + q, s00 * (na * nb) + s10 * (a * nb) + s01 * (na * b) + s11 * (a * b));
            st_stream(goi + q, w * ((s10 - s00) * nb + (s11 - s01) * b));
            st_stream(goj + q, w * ((s01 - s00) * na + (s11 - s10) * a));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// True gradInput (gin_mode = FVFI_GIN_TRUE; NOT in the reference, which returns zeros -- adacof.py:382,445): the adjoint of the
// forward gather, a scatter-add of  gout[c] * w * bilinear weight  into the four taps of every (pixel, k, l).
// WARP-AGGREGATED atomics: a warp owns 32 horizontally adjacent pixels of one tap; neighbouring pixels of a smooth flow field hit
// the same or adjacent frame samples, so for each of the four corners the lanes are grouped by target address
// (__match_any_sync), every group sums its three channel values with shuffles and only the group leader issues the
// red.global.add -- one atomic per DISTINCT address per warp instead of one per lane.  Lanes outside the image contribute to
// no group (address -1 is matched but skipped).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void warp_agg_add3(float* __restrict__ G, size_t plane_in, int o, float v0, float v1, float v2,
                                              unsigned lane) {
    const unsigned peers = __match_any_sync(0xffffffffu, o);
    if (peers == (1u << lane)) {                      // address unique in the warp: plain reductions
        if (o >= 0) {
            atomicAdd(G + o, v0);
            atomicAdd(G + plane_in + o, v1);
            atomicAdd(G + 2 * plane_in + o, v2);
        }
        return;
    }
    // every lane of the group walks the same peer list (same mask -> same trip count), so the shuffles converge per group
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (unsigned m = peers; m; m &= m - 1) {
        const int src = __ffs(m) - 1;
        s0 += __shfl_sync(peers, v0, src);
        s1 += __shfl_sync(peers, v1, src);
        s2 += __shfl_sync(peers, v2, src);
    }
    if (o >= 0 && lane == (unsigned)(__ffs(peers) - 1)) {
        atomicAdd(G + o, s0);
        atomicAdd(G + plane_in + o, s1);
        atomicAdd(G + 2 * plane_in + o, s2);
    }
}

__global__ void __launch_bounds__(256)
adacof_grad_input_scatter(const float* __restrict__ gout, const float* __restrict__ weight, const float* __restrict__ off_i,
                          const float* __restrict__ off_j, float* __restrict__ gin, int Hin, int Win, int H, int W, int F,
                          int dil) {
    constexpr int C = 3;
    const int j = blockIdx.x * 32 + threadIdx.x;         // a warp = 32 adjacent pixels of one row
    const int i = blockIdx.y * 8 + threadIdx.y;
    const int n = blockIdx.z;
    const bool live = j < W && i < H;                    // whole warps stay in the loop: the match/shuffle masks are full
    if (i >= H) return;                                  // uniform per warp (threadIdx.y is the warp index)
    const unsigned lane = threadIdx.x;
    const size_t plane = (size_t)H * W, plane_in = (size_t)Hin * Win;
    float* G = gin + (size_t)n * C * plane_in;
    float g[C] = {0.f, 0.f, 0.f};
    if (live) {
#pragma unroll
        for (int c = 0; c < C; ++c) g[c] = ld_stream(gout + ((size_t)n * C + c) * plane + (size_t)i * W + j);
    }
    size_t q = (size_t)n * F * F * plane + (size_t)i * W + (live ? j : 0);
    for (int k = 0; k < F; ++k) {
        for (int l = 0; l < F; ++l, q += plane) {
            int o00 = -1, o10 = -1, o01 = -1, o11 = -1;
            float w00 = 0.f, w10 = 0.f, w01 = 0.f, w11 = 0.f, w = 0.f;
            if (live) {
                w = ld_stream(weight + q);
                const float al = ld_stream(off_i + q), be = ld_stream(off_j + q);
                const int A = (int)al, B = (int)be;                          // truncation, adacof.py:27-28
                const float a = al - (float)A, b = be - (float)B;
                const int r = i + k * dil + A, cc = j + l * dil + B;
                const int r0 = min(max(r, 0), Hin - 1), r1 = min(max(r + 1, 0), Hin - 1);
                const int c0 = min(max(cc, 0), Win - 1), c1 = min(max(cc + 1, 0), Win - 1);
                o00 = r0 * Win + c0; o10 = r1 * Win + c0; o01 = r0 * Win + c1; o11 = r1 * Win + c1;
                const float na = 1.f - a, nb = 1.f - b;
                w00 = na * nb; w10 = a * nb; w01 = na * b; w11 = a * b;
            }
            const float d0 = g[0] * w, d1 = g[1] * w, d2 = g[2] * w;
            warp_agg_add3(G, plane_in, o00, d0 * w00, d1 * w00, d2 * w00, lane);
            warp_agg_add3(G, plane_in, o10, d0 * w10, d1 * w10, d2 * w10, lane);
            warp_agg_add3(G, plane_in, o01, d0 * w01, d1 * w01, d2 * w01, lane);
            warp_agg_add3(G, plane_in, o11, d0 * w11, d1 * w11, d2 * w11, lane);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// True gradInput, CTA-AGGREGATED form (the default of gin_mode = FVFI_GIN_TRUE): the warp-aggregated kernel above still issues one
// global reduction per (tap, corner, channel) whenever neighbouring lanes hit DIFFERENT samples -- the normal case of a smooth flow
// field: 5e9 reductions for B = 8 at 1088 x 1920, 11.8 ms, atomics-bound.  Here a CTA owns a 64 x 16 output tile and accumulates the
// contributions of its 1024 pixels x F^2 taps x 4 corners in a SHARED-MEMORY image of the frame region the tile can reach
// ((16 + (F-1) d + 2*8 + 1) x (64 + (F-1) d + 2*8 + 1) samples x 3 channels, UNCLAMPED coordinates: 37.7 KB for F = 5, d = 1), then
// flushes every non-zero sample with ONE global reduction at its clamped frame position (clamp-to-edge folds the out-of-frame part of
// the region onto the border samples, adacof.py:30-52) -- 4-9 global reductions per output pixel instead of 300.  Offsets that leave the
// region (beyond the halo of 8) go straight to global memory.  A warp works on 32 adjacent pixels of one row, so for smooth fields its
// shared-memory updates fall on adjacent words (conflict-free); colliding lanes are serialised by the hardware's CAS loop.
// ---------------------------------------------------------------------------------------------
constexpr int GT_W = 64, GT_H = 16, GT_HALO = 8, GT_THREADS = 256;

__global__ void __launch_bounds__(GT_THREADS)
adacof_grad_input_tile(const float* __restrict__ gout, const float* __restrict__ weight, const float* __restrict__ off_i,
                       const float* __restrict__ off_j, float* __restrict__ gin, int Hin, int Win, int H, int W, int F, int dil,
                       int RH, int RW) {
    constexpr int C = 3;
    extern __shared__ float gt_region[];                 // [3][RH * RW]
    const int RP = RH * RW;
    const int i0 = blockIdx.y * GT_H, j0 = blockIdx.x * GT_W, n = blockIdx.z;
    for (int p = threadIdx.x; p < C * RP; p += GT_THREADS) gt_region[p] = 0.f;
    __syncthreads();
    const size_t plane = (size_t)H * W, plane_in = (size_t)Hin * Win;
    float* G = gin + (size_t)n * C * plane_in;
    const int jl = threadIdx.x & (GT_W - 1);             // a warp = 32 adjacent pixels of one row
    const int j = j0 + jl;
    for (int il = threadIdx.x / GT_W; il < GT_H; il += GT_THREADS / GT_W) {
        const int i = i0 + il;
        if (!(i < H && j < W)) continue;
        float g[C];
#pragma unroll
        for (int c = 0; c < C; ++c) g[c] = ld_stream(gout + ((size_t)n * C + c) * plane + (size_t)i * W + j);
        size_t q = (size_t)n * F * F * plane + (size_t)i * W + j;
        for (int k = 0; k < F; ++k) {
          for (int l0 = 0; l0 < F; l0 += 5) {             // up to five taps of the row at a time: their 15 coefficient loads are in flight together
            float wv[5], av[5], bv[5];
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                const bool on = l0 + u < F;
                wv[u] = on ? ld_stream(weight + q + (size_t)u * plane) : 0.f;
                av[u] = on ? ld_stream(off_i + q + (size_t)u * plane) : 0.f;
                bv[u] = on ? ld_stream(off_j + q + (size_t)u * plane) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                const int l = l0 + u;
                if (l >= F) continue;
                const float w = wv[u], al = av[u], be = bv[u];
                const int A = (int)al, B = (int)be;                          // truncation, adacof.py:27-28
                const float a = al - (float)A, b = be - (float)B;
                const float na = 1.f - a, nb = 1.f - b;
                const float w00 = na * nb, w10 = a * nb, w01 = na * b, w11 = a * b;
                const float d0 = g[0] * w, d1 = g[1] * w, d2 = g[2] * w;
                const int rr = il + k * dil + A + GT_HALO, cc = jl + l * dil + B + GT_HALO;     // region coordinates of the (r, c) corner
                if ((unsigned)rr < (unsigned)(RH - 1) && (unsigned)cc < (unsigned)(RW - 1)) {
                    float* R0 = gt_region + rr * RW + cc;
                    atomicAdd(R0, d0 * w00);              atomicAdd(R0 + RP, d1 * w00);              atomicAdd(R0 + 2 * RP, d2 * w00);
                    atomicAdd(R0 + RW, d0 * w10);         atomicAdd(R0 + RP + RW, d1 * w10);         atomicAdd(R0 + 2 * RP + RW, d2 * w10);
                    atomicAdd(R0 + 1, d0 * w01);          atomicAdd(R0 + RP + 1, d1 * w01);          atomicAdd(R0 + 2 * RP + 1, d2 * w01);
                    atomicAdd(R0 + RW + 1, d0 * w11);     atomicAdd(R0 + RP + RW + 1, d1 * w11);     atomicAdd(R0 + 2 * RP + RW + 1, d2 * w11);
                } else {                                  // beyond the halo: global reductions at the clamped positions
                    const int r = i + k * dil + A, cg = j + l * dil + B;
                    const int r0 = min(max(r, 0), Hin - 1), r1 = min(max(r + 1, 0), Hin - 1);
                    const int c0 = min(max(cg, 0), Win - 1), c1 = min(max(cg + 1, 0), Win - 1);
                    float* P00 = G + (size_t)r0 * Win + c0;
                    float* P10 = G + (size_t)r1 * Win + c0;
                    float* P01 = G + (size_t)r0 * Win + c1;
                    float* P11 = G + (size_t)r1 * Win + c1;
                    atomicAdd(P00, d0 * w00); atomicAdd(P00 + plane_in, d1 * w00); atomicAdd(P00 + 2 * plane_in, d2 * w00);
                    atomicAdd(P10, d0 * w10); atomicAdd(P10 + plane_in, d1 * w10); atomicAdd(P10 + 2 * plane_in, d2 * w10);
                    atomicAdd(P01, d0 * w01); atomicAdd(P01 + plane_in, d1 * w01); atomicAdd(P01 + 2 * plane_in, d2 * w01);
                    atomicAdd(P11, d0 * w11); atomicAdd(P11 + plane_in, d1 * w11); atomicAdd(P11 + 2 * plane_in, d2 * w11);
                }
            }
            q += (size_t)min(5, F - l0) * plane;
          }
        }
    }
    __syncthreads();
    for (int p = threadIdx.x; p < RP; p += GT_THREADS) {
        const int r = p / RW, c = p - r * RW;
        const int gr = min(max(i0 - GT_HALO + r, 0), Hin - 1), gc = min(max(j0 - GT_HALO + c, 0), Win - 1);
        float* dst = G + (size_t)gr * Win + gc;
#pragma unroll
        for (int ch = 0; ch < C; ++ch) {
            const float v = gt_region[ch * RP + p];
            if (v != 0.f) atomicAdd(dst + (size_t)ch * plane_in, v);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// AdaCoFNet tail: frame = occ*t1 + (1-occ)*t2 and the flow-variance mask
// (fusion_adacofnet.py:198-213).  One pass per frame using running moments:
//   mean = S1 = sum w*d ;  var = sum w (mean-d)^2 = S2 - mean^2 (2 - S0)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float flow_var(float s0, float s1i, float s2i, float s1j, float s2j) {
    return (s2i - s1i * s1i * (2.f - s0)) + (s2j - s1j * s1j * (2.f - s0));
}

__global__ void __launch_bounds__(256)
adacofnet_tail_kernel(const float* __restrict__ t1, const float* __restrict__ t2, const float* __restrict__ occ,
                      const float* __restrict__ w1, const float* __restrict__ a1, const float* __restrict__ b1,
                      const float* __restrict__ w2, const float* __restrict__ a2, const float* __restrict__ b2,
                      float* __restrict__ frame, float* __restrict__ mask, int C, size_t plane, int FF) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.y;
    if (p >= plane) return;
    if (frame) {
        const float o = occ[(size_t)n * plane + p];
        for (int c = 0; c < C; ++c) {
            const size_t q = ((size_t)n * C + c) * plane + p;
            frame[q] = o * t1[q] + (1.f - o) * t2[q];
        }
    }
    if (mask) {
        float var[2];
#pragma unroll
        for (int f = 0; f < 2; ++f) {
            const float* w = f ? w2 : w1;
            const float* al = f ? a2 : a1;
            const float* be = f ? b2 : b1;
            float s0 = 0.f, s1i = 0.f, s2i = 0.f, s1j = 0.f, s2j = 0.f;
            size_t q = (size_t)n * FF * plane + p;
            for (int t = 0; t < FF; ++t, q += plane) {
                const float ww = ld_stream(w + q), x = ld_stream(al + q), y = ld_stream(be + q);
                s0 += ww;
                s1i = fmaf(ww, x, s1i);
                s2i = fmaf(ww * x, x, s2i);
                s1j = fmaf(ww, y, s1j);
                s2j = fmaf(ww * y, y, s2j);
            }
            var[f] = flow_var(s0, s1i, s2i, s1j, s2j);
        }
        const float m = fminf(fmaxf(fmaxf(var[0], var[1]), 0.f), 20.f);
        mask[(size_t)n * plane + p] = m / 20.f;
    }
}

// ---------------------------------------------------------------------------------------------
// Fused AdaCoFNet synthesis: both warps + occlusion blend + uncertainty mask in one pass
// (fusion_adacofnet.py:195-213).  Each of the six coefficient maps is read from HBM once.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adacofnet_warp_blend_direct(const float* __restrict__ in1, const float* __restrict__ in2,
                            const float* __restrict__ w1, const float* __restrict__ a1,
                            const float* __restrict__ b1, const float* __restrict__ w2,
                            const float* __restrict__ a2, const float* __restrict__ b2,
                            const float* __restrict__ occ, float* __restrict__ t1, float* __restrict__ t2,
                            float* __restrict__ frame, float* __restrict__ mask, int Hin, int Win, int H,
                            int W, int F, int dil) {
    constexpr int C = 3;
    const int j = blockIdx.x * 32 + threadIdx.x;
    const int i = blockIdx.y * 8 + threadIdx.y;
    const int n = blockIdx.z;
    if (j >= W || i >= H) return;
    const size_t plane = (size_t)H * W, plane_in = (size_t)Hin * Win;
    float acc[2][C], var[2];
#pragma unroll
    for (int f = 0; f < 2; ++f) {
        const float* I = (f ? in2 : in1) + (size_t)n * C * plane_in;
        const float* w_ = f ? w2 : w1;
        const float* a_ = f ? a2 : a1;
        const float* b_ = f ? b2 : b1;
        size_t q = (size_t)n * F * F * plane + (size_t)i * W + j;
        float s0 = 0.f, s1i = 0.f, s2i = 0.f, s1j = 0.f, s2j = 0.f;
#pragma unroll
        for (int c = 0; c < C; ++c) acc[f][c] = 0.f;
        for (int k = 0; k < F; ++k) {
#pragma unroll 5
            for (int l = 0; l < F; ++l, q += plane) {
                const float w = ld_stream(w_ + q), al = ld_stream(a_ + q), be = ld_stream(b_ + q);
                s0 += w;
                s1i = fmaf(w, al, s1i);
                s2i = fmaf(w * al, al, s2i);
                s1j = fmaf(w, be, s1j);
                s2j = fmaf(w * be, be, s2j);
                const Tap t = make_tap(al, be, i + k * dil, j + l * dil, Hin, Win);
                const int o00 = t.r0 * Win + t.c0, o10 = t.r1 * Win + t.c0;
                const int o01 = t.r0 * Win + t.c1, o11 = t.r1 * Win + t.c1;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const float* Ic = I + (size_t)c * plane_in;
                    const float v = __ldg(Ic + o00) * t.w00 + __ldg(Ic + o10) * t.w10 +
                                    __ldg(Ic + o01) * t.w01 + __ldg(Ic + o11) * t.w11;
                    acc[f][c] = fmaf(w, v, acc[f][c]);
                }
            }
        }
        var[f] = flow_var(s0, s1i, s2i, s1j, s2j);
    }
    const size_t p = (size_t)i * W + j;
    const float o = occ[(size_t)n * plane + p];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const size_t qo = ((size_t)n * C + c) * plane + p;
        if (t1) st_stream(t1 + qo, acc[0][c]);
        if (t2) st_stream(t2 + qo, acc[1][c]);
        if (frame) st_stream(frame + qo, o * acc[0][c] + (1.f - o) * acc[1][c]);
    }
    if (mask) mask[(size_t)n * plane + p] = fminf(fmaxf(fmaxf(var[0], var[1]), 0.f), 20.f) / 20.f;
}

__device__ __forceinline__ float fusion_blend_px(float base, float x) {
    const float v = base + tanhf(x);                              // fusion_net.py:67-72
    return fminf(fmaxf(v, 0.f), 1.f);                             // fusion_net.py:77
}

__global__ void fusion_blend_kernel(const float* __restrict__ base, const float* __restrict__ x,
                                    float* __restrict__ out, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) out[t] = fusion_blend_px(base[t], x[t]);
}

// The same blend for frames that leave as 8-bit video: planar [B,3,H,W] in, interleaved rgb24 [B,H,W,3] out, rint(v * 255) (round
// half to even); the fp32 frame is never stored.
__global__ void __launch_bounds__(256) fusion_blend_rgb8_kernel(const float* __restrict__ base, const float* __restrict__ x,
                                                                uint8_t* __restrict__ out, size_t plane) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.y;
    if (p >= plane) return;
    const size_t o = (size_t)n * 3 * plane + p;
    uint8_t* dst = out + ((size_t)n * plane + p) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c)
        dst[c] = (uint8_t)__float2uint_rn(fusion_blend_px(__ldcs(base + o + c * plane), __ldcs(x + o + c * plane)) * 255.f);
}

// An 8-bit code from a value on the 0..255 scale: clamp, then round half to even.
__device__ __forceinline__ uint8_t code8(float v) { return (uint8_t)__float2uint_rn(fminf(fmaxf(v, 0.f), 255.f)); }

// Y' = (Kr R' + Kg G') + Kb B', every product and sum rounded on its own (no FMA contraction).
__device__ __forceinline__ float luma(float r, float g, float b, const YuvCoeffs& k) {
    return __fadd_rn(__fadd_rn(__fmul_rn(k.kr, r), __fmul_rn(k.kg, g)), __fmul_rn(k.kb, b));
}

// The same blend for frames that leave as yuv420p [B,3H/2,W] uint8 (include/fvfi.h, fvfi_fusion_blend_yuv420p; oracle/yuv.py restates
// the arithmetic): one thread owns a 2x2 luma block, blends its 4 pixels x 3 channels (float2 __ldcs loads of both rows), writes the
// two uchar2 Y pairs, and Cb / Cr of the block's mean R'G'B' (centre-sited chroma).  The fp32 frame is never stored.
__global__ void __launch_bounds__(256) fusion_blend_yuv420p_kernel(const float* __restrict__ base, const float* __restrict__ x,
                                                                   uint8_t* __restrict__ out, int H, int W, YuvCoeffs k) {
    const int Hc = H / 2, Wc = W / 2;
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.y;
    if (q >= (size_t)Hc * Wc) return;
    const int i = (int)(q / Wc), j = (int)(q - (size_t)i * Wc);
    const size_t plane = (size_t)H * W;
    uint8_t* Y = out + (size_t)n * plane * 3 / 2;
    float v[3][2][2];                                // [channel][row][column]
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
        const size_t o = (size_t)(2 * i + dy) * W + 2 * j;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const size_t f = ((size_t)n * 3 + c) * plane + o;
            const float2 b2 = __ldcs(reinterpret_cast<const float2*>(base + f)), x2 = __ldcs(reinterpret_cast<const float2*>(x + f));
            v[c][dy][0] = fusion_blend_px(b2.x, x2.x);
            v[c][dy][1] = fusion_blend_px(b2.y, x2.y);
        }
        uchar2 yy;
        yy.x = code8(__fadd_rn(k.yoff, __fmul_rn(k.ys, luma(v[0][dy][0], v[1][dy][0], v[2][dy][0], k))));
        yy.y = code8(__fadd_rn(k.yoff, __fmul_rn(k.ys, luma(v[0][dy][1], v[1][dy][1], v[2][dy][1], k))));
        *reinterpret_cast<uchar2*>(Y + o) = yy;
    }
    float m[3];                                      // block mean: ((top-left + top-right) + (bottom-left + bottom-right)) / 4
#pragma unroll
    for (int c = 0; c < 3; ++c) m[c] = __fmul_rn(__fadd_rn(__fadd_rn(v[c][0][0], v[c][0][1]), __fadd_rn(v[c][1][0], v[c][1][1])), 0.25f);
    const float ym = luma(m[0], m[1], m[2], k);
    const size_t oc = (size_t)i * Wc + j;
    Y[plane + oc] = code8(__fadd_rn(128.f, __fmul_rn(k.cs, __fmul_rn(__fsub_rn(m[2], ym), k.kCb))));
    Y[plane + plane / 4 + oc] = code8(__fadd_rn(128.f, __fmul_rn(k.cs, __fmul_rn(__fsub_rn(m[0], ym), k.kCr))));
}

static int check_dims(int B, int C, int Hin, int Win, int H, int W, int F, int dil) {
    FVFI_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0 && F > 0 && dil > 0, "adacof: non-positive dimension");
    // adacof.py:326-327
    FVFI_CHECK_ARG(Hin - ((F - 1) * dil + 1) == H - 1, "adacof: input height %d != H + (F-1)*dilation = %d", Hin,
                   H + (F - 1) * dil);
    FVFI_CHECK_ARG(Win - ((F - 1) * dil + 1) == W - 1, "adacof: input width %d != W + (F-1)*dilation = %d", Win,
                   W + (F - 1) * dil);
    FVFI_CHECK_ARG((size_t)Hin * Win < (size_t)1 << 31, "adacof: frame plane too large for 32-bit tap offsets");
    FVFI_CHECK_ARG(B <= 65535, "adacof: batch > 65535");
    return FVFI_OK;
}

// implemented in adacof_tiled.cu; return 1 if the tiled path handled the call, 0 if not applicable
int adacof_forward_tiled(const float* input, const float* weight, const float* off_i, const float* off_j,
                         float* output, int B, int Hin, int Win, int H, int W, int F, int dil,
                         cudaStream_t s, int* handled);
int adacof_backward_tiled(const float* gout, const float* input, const float* weight, const float* off_i,
                          const float* off_j, float* gw, float* goi, float* goj, int B, int Hin, int Win,
                          int H, int W, int F, int dil, cudaStream_t s, int* handled);

int adacofnet_warp_blend_tiled(const float* in1, const float* in2, const float* w1, const float* a1,
                               const float* b1, const float* w2, const float* a2, const float* b2,
                               const float* occ, float* t1, float* t2, float* frame, float* mask, int B, int Hin,
                               int Win, int H, int W, int F, int dil, cudaStream_t s, int* handled);
// implemented in adacof_tma.cu (F = 5, dilation 1, W % 4 == 0): TMA-streamed coefficient maps, persistent CTAs
int adacof_tma_launch(const float* in1, const float* in2, const float* w1, const float* a1, const float* b1,
                      const float* w2, const float* a2, const float* b2, const float* occ, float* t1, float* t2,
                      float* frame, float* mask, int nframes, int B, int Hin, int Win, int H, int W, int F, int dil,
                      cudaStream_t s, int* handled, const float* bwd_gout = nullptr, float* bwd_gw = nullptr,
                      float* bwd_goi = nullptr, float* bwd_goj = nullptr, int out_rows = 0);

}  // namespace fvfi

using namespace fvfi;

extern "C" int fvfi_adacof_forward(const float* input, const float* weight, const float* off_i,
                                   const float* off_j, float* output, int B, int C, int Hin, int Win, int H,
                                   int W, int F, int dilation, int algo, void* stream) {
    if (int rc = check_dims(B, C, Hin, Win, H, W, F, dilation)) return rc;
    FVFI_CHECK_ARG(input && weight && off_i && off_j && output, "adacof_forward: null pointer");
    FVFI_CHECK_ARG(algo >= 0 && algo <= 3, "adacof_forward: algo must be 0..3");
    cudaStream_t s = (cudaStream_t)stream;
    if (C == 3 && (algo == 0 || algo == 3)) {
        int handled = 0;
        if (int rc = adacof_tma_launch(input, nullptr, weight, off_i, off_j, nullptr, nullptr, nullptr, nullptr, output,
                                       nullptr, nullptr, nullptr, 1, B, Hin, Win, H, W, F, dilation, s, &handled))
            return rc;
        if (handled) return FVFI_OK;
        FVFI_CHECK_ARG(algo != 3, "adacof_forward: TMA algorithm needs F = 5, dilation 1, W %% 4 == 0 and 16-byte aligned maps");
    }
    if (C == 3 && algo != 1) {
        int handled = 0;
        if (int rc = adacof_forward_tiled(input, weight, off_i, off_j, output, B, Hin, Win, H, W, F, dilation, s,
                                          &handled))
            return rc;
        if (handled) return FVFI_OK;
        FVFI_CHECK_ARG(algo != 2, "adacof_forward: tiled algorithm not applicable to F=%d dilation=%d", F,
                       dilation);
    } else {
        FVFI_CHECK_ARG(algo != 2, "adacof_forward: tiled algorithm needs C == 3");
    }
    dim3 block(32, 8), grid(ceil_div(W, 32), ceil_div(H, 8), B);
    if (C == 3)
        adacof_fwd_direct<3><<<grid, block, 0, s>>>(input, weight, off_i, off_j, output, Hin, Win, H, W, F,
                                                     dilation);
    else
        adacof_fwd_direct_anyc<<<grid, block, 0, s>>>(input, weight, off_i, off_j, output, C, Hin, Win, H, W, F,
                                                      dilation);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_adacof_backward(const float* gout, const float* input, const float* weight,
                                    const float* off_i, const float* off_j, float* gin, float* gw, float* goi,
                                    float* goj, int B, int C, int Hin, int Win, int H, int W, int F, int dilation,
                                    int gin_mode, int algo, void* stream) {
    if (int rc = check_dims(B, C, Hin, Win, H, W, F, dilation)) return rc;
    FVFI_CHECK_ARG(C == 3, "adacof_backward: C must be 3 (the reference hard-codes 3 channels, adacof.py:86)");
    FVFI_CHECK_ARG(gout && input && weight && off_i && off_j && gw && goi && goj, "adacof_backward: null pointer");
    FVFI_CHECK_ARG(gin_mode >= 0 && gin_mode <= 2, "adacof_backward: bad gin_mode");
    FVFI_CHECK_ARG(gin_mode == FVFI_GIN_NONE || gin, "adacof_backward: gin is null");
    FVFI_CHECK_ARG(algo >= 0 && algo <= 3, "adacof_backward: algo must be 0..3");
    cudaStream_t s = (cudaStream_t)stream;
    if (gin_mode != FVFI_GIN_NONE)
        FVFI_CUDA(cudaMemsetAsync(gin, 0, (size_t)B * C * Hin * Win * sizeof(float), s));
    if (gin_mode == FVFI_GIN_TRUE) {     // true adjoint (extension): warp-aggregated scatter, independent of the gradient path below
        FVFI_CHECK_ARG((long long)Hin * Win <= 0x7fffffffLL, "adacof_backward: frame too large for the gradInput scatter");
        // default: CTA-aggregated in shared memory (adacof_grad_input_tile); the warp-aggregated kernel when the reachable region
        // does not fit (large F * dilation) or on request (FVFI_GIN_SCATTER=warp: tests / A-B timing)
        const int RH = GT_H + (F - 1) * dilation + 2 * GT_HALO + 1, RW = GT_W + (F - 1) * dilation + 2 * GT_HALO + 1;
        const size_t tile_smem = (size_t)3 * RH * RW * sizeof(float);
        const char* how = getenv("FVFI_GIN_SCATTER");
        if (tile_smem <= 96 * 1024 && !(how && how[0] == 'w')) {
            FVFI_SMEM_OPT_IN(adacof_grad_input_tile, tile_smem);
            dim3 tgrid(ceil_div(W, GT_W), ceil_div(H, GT_H), B);
            adacof_grad_input_tile<<<tgrid, GT_THREADS, tile_smem, s>>>(gout, weight, off_i, off_j, gin, Hin, Win, H, W, F, dilation,
                                                                      RH, RW);
        } else {
            dim3 sblock(32, 8), sgrid(ceil_div(W, 32), ceil_div(H, 8), B);
            adacof_grad_input_scatter<<<sgrid, sblock, 0, s>>>(gout, weight, off_i, off_j, gin, Hin, Win, H, W, F, dilation);
        }
        FVFI_LAUNCH_CHECK();
    }
    if (C == 3 && (algo == 0 || algo == 3)) {
        int handled = 0;
        if (int rc = adacof_tma_launch(input, nullptr, weight, off_i, off_j, nullptr, nullptr, nullptr, nullptr, nullptr,
                                       nullptr, nullptr, nullptr, 0, B, Hin, Win, H, W, F, dilation, s, &handled, gout, gw,
                                       goi, goj))
            return rc;
        if (handled) return FVFI_OK;
        FVFI_CHECK_ARG(algo != 3, "adacof_backward: TMA algorithm needs F = 5, dilation 1, W %% 4 == 0 and 16-byte aligned maps");
    }
    if (algo != 1 && algo != 3) {
        int handled = 0;
        if (int rc = adacof_backward_tiled(gout, input, weight, off_i, off_j, gw, goi, goj, B, Hin, Win, H, W, F,
                                           dilation, s, &handled))
            return rc;
        if (handled) return FVFI_OK;
        FVFI_CHECK_ARG(algo != 2, "adacof_backward: tiled algorithm not applicable to F=%d dilation=%d", F,
                       dilation);
    }
    dim3 block(32, 8), grid(ceil_div(W, 32), ceil_div(H, 8), B);
    adacof_bwd_direct<<<grid, block, 0, s>>>(gout, input, weight, off_i, off_j, nullptr, gw, goi, goj, Hin, Win, H, W, F,
                                             dilation);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_adacofnet_tail(const float* t1, const float* t2, const float* occ, const float* w1,
                                   const float* a1, const float* b1, const float* w2, const float* a2,
                                   const float* b2, float* frame, float* mask, int B, int C, int H, int W, int FF,
                                   void* stream) {
    FVFI_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0 && FF > 0 && B <= 65535, "adacofnet_tail: bad dimension");
    FVFI_CHECK_ARG(!frame || (t1 && t2 && occ), "adacofnet_tail: frame requested without t1/t2/occ");
    FVFI_CHECK_ARG(!mask || (w1 && a1 && b1 && w2 && a2 && b2), "adacofnet_tail: mask requested without maps");
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), B);
    adacofnet_tail_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(t1, t2, occ, w1, a1, b1, w2, a2, b2, frame, mask,
                                                                  C, plane, FF);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_adacofnet_warp_blend_rows(const float* in1, const float* in2, const float* w1, const float* a1,
                                              const float* b1, const float* w2, const float* a2, const float* b2,
                                              const float* occ, float* frame, float* mask, int out_rows, int B, int Hin, int Win,
                                              int H, int W, int F, int dilation, void* stream) {
    if (int rc = check_dims(B, 3, Hin, Win, H, W, F, dilation)) return rc;
    FVFI_CHECK_ARG(in1 && in2 && w1 && a1 && b1 && w2 && a2 && b2 && occ && frame, "adacofnet_warp_blend_rows: null pointer");
    FVFI_CHECK_ARG(out_rows > 0 && out_rows <= H, "adacofnet_warp_blend_rows: out_rows must be in [1, H]");
    int handled = 0;
    if (int rc = adacof_tma_launch(in1, in2, w1, a1, b1, w2, a2, b2, occ, nullptr, nullptr, frame, mask, 2, B, Hin, Win, H, W, F,
                                   dilation, (cudaStream_t)stream, &handled, nullptr, nullptr, nullptr, nullptr, out_rows))
        return rc;
    FVFI_CHECK_ARG(handled, "adacofnet_warp_blend_rows: needs the TMA-streamed kernel (F = 5, dilation 1, W %% 4 == 0, 16-byte aligned maps)");
    return FVFI_OK;
}

extern "C" int fvfi_adacofnet_warp_blend(const float* in1, const float* in2, const float* w1, const float* a1,
                                         const float* b1, const float* w2, const float* a2, const float* b2,
                                         const float* occ, float* t1, float* t2, float* frame, float* mask, int B,
                                         int Hin, int Win, int H, int W, int F, int dilation, void* stream) {
    if (int rc = check_dims(B, 3, Hin, Win, H, W, F, dilation)) return rc;
    FVFI_CHECK_ARG(in1 && in2 && w1 && a1 && b1 && w2 && a2 && b2 && occ, "adacofnet_warp_blend: null input");
    int handled = 0;
    if (int rc = adacof_tma_launch(in1, in2, w1, a1, b1, w2, a2, b2, occ, t1, t2, frame, mask, 2, B, Hin, Win, H, W, F,
                                   dilation, (cudaStream_t)stream, &handled))
        return rc;
    if (handled) return FVFI_OK;
    if (int rc = adacofnet_warp_blend_tiled(in1, in2, w1, a1, b1, w2, a2, b2, occ, t1, t2, frame, mask, B, Hin, Win,
                                            H, W, F, dilation, (cudaStream_t)stream, &handled))
        return rc;
    if (handled) return FVFI_OK;
    dim3 block(32, 8), grid(ceil_div(W, 32), ceil_div(H, 8), B);
    adacofnet_warp_blend_direct<<<grid, block, 0, (cudaStream_t)stream>>>(in1, in2, w1, a1, b1, w2, a2, b2, occ, t1,
                                                                          t2, frame, mask, Hin, Win, H, W, F,
                                                                          dilation);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_fusion_blend(const float* base, const float* x_pre_tanh, float* out, size_t n, void* stream) {
    FVFI_CHECK_ARG(base && x_pre_tanh && out, "fusion_blend: null pointer");
    if (n == 0) return FVFI_OK;
    const int sms = sm_count() > 0 ? sm_count() : 148;
    size_t blocks = (n + 255) / 256;
    if (blocks > (size_t)sms * 16) blocks = (size_t)sms * 16;
    fusion_blend_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(base, x_pre_tanh, out, n);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_fusion_blend_rgb8(const float* base, const float* x_pre_tanh, uint8_t* out, int B, int H, int W, void* stream) {
    FVFI_CHECK_ARG(base && x_pre_tanh && out, "fvfi_fusion_blend_rgb8: null pointer");
    FVFI_CHECK_ARG(B > 0 && H > 0 && W > 0 && B <= 65535, "fvfi_fusion_blend_rgb8: bad size B=%d H=%d W=%d", B, H, W);
    const size_t plane = (size_t)H * W;
    dim3 grid((unsigned)((plane + 255) / 256), B);
    fusion_blend_rgb8_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(base, x_pre_tanh, out, plane);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

extern "C" int fvfi_fusion_blend_yuv420p(const float* base, const float* x_pre_tanh, uint8_t* out, int B, int H, int W, int matrix,
                                         int full_range, void* stream) {
    FVFI_CHECK_ARG(base && x_pre_tanh && out, "fvfi_fusion_blend_yuv420p: null pointer");
    if (int rc = yuv_check("fvfi_fusion_blend_yuv420p", B, H, W, matrix, full_range)) return rc;
    FVFI_CHECK_ARG((uintptr_t)base % 8 == 0 && (uintptr_t)x_pre_tanh % 8 == 0 && (uintptr_t)out % 2 == 0,
                   "fvfi_fusion_blend_yuv420p: base / x_pre_tanh must be 8-byte and out 2-byte aligned");
    const size_t blocks = (size_t)(H / 2) * (W / 2);
    dim3 grid((unsigned)((blocks + 255) / 256), B);
    fusion_blend_yuv420p_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(base, x_pre_tanh, out, H, W, yuv_coeffs(matrix, full_range));
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

// ---------------------------------------------------------------------------------------------
// Host-buffer variants (end-to-end measurement): H2D, kernel, D2H, sync.
// ---------------------------------------------------------------------------------------------
namespace {
struct DevBuf {
    float* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t n) {
        FVFI_CUDA(cudaMalloc(&p, n * sizeof(float)));
        return FVFI_OK;
    }
};
}  // namespace

extern "C" int fvfi_adacof_forward_host(const float* input, const float* weight, const float* off_i,
                                        const float* off_j, float* output, int B, int C, int Hin, int Win, int H,
                                        int W, int F, int dilation) {
    if (int rc = check_dims(B, C, Hin, Win, H, W, F, dilation)) return rc;
    const size_t n_in = (size_t)B * C * Hin * Win, n_k = (size_t)B * F * F * H * W, n_out = (size_t)B * C * H * W;
    DevBuf d_in, d_w, d_a, d_b, d_out;
    if (int rc = d_in.alloc(n_in)) return rc;
    if (int rc = d_w.alloc(n_k)) return rc;
    if (int rc = d_a.alloc(n_k)) return rc;
    if (int rc = d_b.alloc(n_k)) return rc;
    if (int rc = d_out.alloc(n_out)) return rc;
    cudaStream_t s = 0;
    FVFI_CUDA(cudaMemcpyAsync(d_in.p, input, n_in * 4, cudaMemcpyHostToDevice, s));
    FVFI_CUDA(cudaMemcpyAsync(d_w.p, weight, n_k * 4, cudaMemcpyHostToDevice, s));
    FVFI_CUDA(cudaMemcpyAsync(d_a.p, off_i, n_k * 4, cudaMemcpyHostToDevice, s));
    FVFI_CUDA(cudaMemcpyAsync(d_b.p, off_j, n_k * 4, cudaMemcpyHostToDevice, s));
    if (int rc = fvfi_adacof_forward(d_in.p, d_w.p, d_a.p, d_b.p, d_out.p, B, C, Hin, Win, H, W, F, dilation, 0, s))
        return rc;
    FVFI_CUDA(cudaMemcpyAsync(output, d_out.p, n_out * 4, cudaMemcpyDeviceToHost, s));
    FVFI_CUDA(cudaStreamSynchronize(s));
    return FVFI_OK;
}

extern "C" int fvfi_adacof_backward_host(const float* gout, const float* input, const float* weight,
                                         const float* off_i, const float* off_j, float* gw, float* goi, float* goj,
                                         int B, int C, int Hin, int Win, int H, int W, int F, int dilation) {
    if (int rc = check_dims(B, C, Hin, Win, H, W, F, dilation)) return rc;
    const size_t n_in = (size_t)B * C * Hin * Win, n_k = (size_t)B * F * F * H * W, n_out = (size_t)B * C * H * W;
    DevBuf d_g, d_in, d_w, d_a, d_b, d_gw, d_ga, d_gb;
    if (int rc = d_g.alloc(n_out)) return rc;
    if (int rc = d_in.alloc(n_in)) return rc;
    if (int rc = d_w.alloc(n_k)) return rc;
    if (int rc = d_a.alloc(n_k)) return rc;
    if (int rc = d_b.alloc(n_k)) return rc;
    if (int rc = d_gw.alloc(n_k)) return rc;
    if (int rc = d_ga.alloc(n_k)) return rc;
    if (int rc = d_gb.alloc(n_k)) return rc;
    cudaStream_t s = 0;
    FVFI_CUDA(cudaMemcpyAsync(d_g.p, gout, n_out * 4, cudaMemcpyHostToDevice, s));
    FVFI_CUDA(cudaMemcpyAsync(d_in.p, input, n_in * 4, cudaMemcpyHostToDevice, s));
    FVFI_CUDA(cudaMemcpyAsync(d_w.p, weight, n_k * 4, cudaMemcpyHostToDevice, s));
    FVFI_CUDA(cudaMemcpyAsync(d_a.p, off_i, n_k * 4, cudaMemcpyHostToDevice, s));
    FVFI_CUDA(cudaMemcpyAsync(d_b.p, off_j, n_k * 4, cudaMemcpyHostToDevice, s));
    if (int rc = fvfi_adacof_backward(d_g.p, d_in.p, d_w.p, d_a.p, d_b.p, nullptr, d_gw.p, d_ga.p, d_gb.p, B, C,
                                      Hin, Win, H, W, F, dilation, FVFI_GIN_NONE, 0, s))
        return rc;
    FVFI_CUDA(cudaMemcpyAsync(gw, d_gw.p, n_k * 4, cudaMemcpyDeviceToHost, s));
    FVFI_CUDA(cudaMemcpyAsync(goi, d_ga.p, n_k * 4, cudaMemcpyDeviceToHost, s));
    FVFI_CUDA(cudaMemcpyAsync(goj, d_gb.p, n_k * 4, cudaMemcpyDeviceToHost, s));
    FVFI_CUDA(cudaStreamSynchronize(s));
    return FVFI_OK;
}
