// fft_engine.cuh -- shared-memory FFT engine of ARBITRARY length for sm_100a (steerable pyramid, pyramid.cu).
//
// The sqrt(2)-scale steerable pyramid needs 1-D transforms of every length its level-size rule produces
// (1080p: 1080, 764 = 4*191, 540, 382, ...; 1920, 1358 = 2*7*97, 960, 679, ..., 241, ...).  Every transform runs
// entirely in shared memory with register butterflies:
//
//   * smooth lengths (prime factors <= 19): mixed radix with radices {2,3,4,5,7,8,9,11,13,15,16,17,19} -- three
//     stages for 1080 = 8*9*15 and 1920 = 16*8*15.  Rows use an out-of-place autosort (Stockham) network so that
//     input and output are both in natural order (coalesced global traffic); columns use an IN-PLACE
//     decimation-in-frequency network whose digit-reversed output order is free (a column pass writes 64-byte row
//     segments, their order does not matter) -- half the shared memory, twice the resident CTAs.
//   * lengths n = r * p with ONE prime factor p > 19 whose p - 1 is smooth (97, 191, 241, 61, 43, 31, 23 ... -- every such
//     length of the 1080p / 4K pyramids): decimation in time into r interleaved length-p DFTs, each done by RADER's
//     algorithm: a length-p DFT is y0 plus a cyclic convolution of length p - 1 of the inputs taken in the order g^q
//     (g a primitive root of p) with the constant sequence W_p^(g^-q).  fft_put scatters every input straight to its
//     residue block and generator-order slot (pos_in), so the whole transform runs in place in ONE buffer of n slots:
//     in-place DIF of the (p-1)-point sub-sequences, multiply by the precomputed spectrum (stored in DIF order, DC bin
//     carries y0), in-place DIT back, then the in-place DIT radix stages of r across the blocks (their twiddle index goes
//     through `perm`, the blocks being in generator order) -- no zero padding and no copy pass, all passes over n points
//     instead of Bluestein's M >= 2n - 1.
//   * other lengths: Bluestein (chirp-z) on a smooth length M >= 2n-1 chosen by the plan: chirp, in-place DIF,
//     multiply by the precomputed spectrum of the chirp filter (stored in DIF order, pre-scaled by 1/M), in-place
//     DIT (digit-reversed in, natural out), chirp.  No permutation pass anywhere, and no extra pass either: the
//     chirps ride on the callers' fft_put / fft_get, the filter multiply on the last DIF stage -> 2*stages passes.
//
// Only FORWARD (e^{-i...}) butterflies exist; inverse transforms are conj -> forward -> conj, the conjugations
// being fused into the callers' load prologue / store epilogue.
//
// Two shared-memory layouts (template COL):
//   COL = true   batch-interleaved  element (b, i) at (i << ctshift) + b     (tile of 2^ctshift adjacent columns)
//   COL = false  sequence-major     element (b, i) at b*pitch + i [+ (i >> 4) when the plan asks for the skew: the
//                                   smallest butterfly stride is even and would otherwise hit one bank pair]
// All stage code is __host__ __device__ and parameterised by (tid, nthr) so that tests/test_fft_engine_host.py can
// run the very same index math and butterflies on the CPU against numpy.fft.
#pragma once
#include <cuda_runtime.h>

#include "fft_consts.cuh"

namespace fvfi {

#define FVFI_HD __host__ __device__ __forceinline__

constexpr int FFT_MAX_STAGES = 8;

struct FftPlan {
    int n;                       // logical transform length
    int M;                       // machine length and slots per sequence: n (direct, Rader) or the Bluestein convolution length
    int nfac;
    int bluestein;
    int rader;                   // 1: n = rr * rp by decimation in time (inputs scattered by pos_in on the way in, Rader in place,
                                 // outer DIT stages whose twiddle index goes through `perm`); stages [0, nouter) work on length n,
                                 // stages [nouter, nfac) are the sub-FFT of length rq
    int rr, rp, rq, nouter;      // rq = rp - 1
    int pad;                     // sequence-major layout: 1 = skew i + (i >> 4) (smallest butterfly stride is even)
    int fac[FFT_MAX_STAGES];     // radices in network order (product = M; Rader: product = rr * rq)
    int sub[FFT_MAX_STAGES];     // DIF/DIT: butterfly stride m_s (block length = fac*sub); Stockham: Ns (product of earlier radices)
    unsigned mag_sub[FFT_MAX_STAGES];    // ceil(2^32 / sub)
    unsigned mag_items[FFT_MAX_STAGES];  // ceil(2^32 / (M / fac));  Rader sub stages: ceil(2^32 / (rq / fac))
    unsigned mag_ritems[FFT_MAX_STAGES]; // Rader sub stages: ceil(2^32 / (rr * rq / fac))
    const float2* tw;            // W_M^t = exp(-2 pi i t / M), t < M
    const unsigned short* perm;  // direct DIF / Rader: natural index held at position p after the network (null: natural)
    const float2* chirp;         // Bluestein: exp(-i pi k^2 / n), k < n
    const float2* bhat;          // Bluestein: FFT_M(chirp filter) / M in DIF (digit-reversed) order;  Rader: FFT_rq(W_rp^(g^-t)) / rq, DIF order
    const float2* tw2;           // Rader: W_rq^t, t < rq
    const unsigned short* inv;   // Rader: position of natural index k in the result (sequence-major layout reads in natural order)
    const unsigned short* pos_in; // Rader: position input i is written to
};

struct FftCtx { int tid, nthr; };

enum { FFT_STOCKHAM = 0, FFT_DIF = 1, FFT_DIT = 2 };

FVFI_HD float2 cmul(float2 a, float2 b) { return make_float2(fmaf(a.x, b.x, -a.y * b.y), fmaf(a.x, b.y, a.y * b.x)); }
FVFI_HD float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
FVFI_HD float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
FVFI_HD float2 cconj(float2 a) { return make_float2(a.x, -a.y); }
FVFI_HD float2 cmuli_neg(float2 a) { return make_float2(a.y, -a.x); }   // a * (-i)

FVFI_HD unsigned fast_div(unsigned x, unsigned d, unsigned magic) {
#if defined(__CUDA_ARCH__)
    return d == 1 ? x : __umulhi(x, magic);
#else
    return d == 1 ? x : (unsigned)(((unsigned long long)x * magic) >> 32);
#endif
}

template <typename T>
FVFI_HD T ldg_(const T* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

// ------------------------------------------------------------------------------------------------
// register butterflies: v <- DFT_R(v), forward sign
// ------------------------------------------------------------------------------------------------
template <int R> struct Radix {};

FVFI_HD void dft(float2* v, Radix<2>) {
    const float2 a = v[0], b = v[1];
    v[0] = cadd(a, b);
    v[1] = csub(a, b);
}
FVFI_HD void dft(float2* v, Radix<3>) {
    const float2 t1 = cadd(v[1], v[2]);
    const float2 t2 = make_float2(v[0].x - 0.5f * t1.x, v[0].y - 0.5f * t1.y);
    const float2 d = csub(v[1], v[2]);
    const float2 r = cmuli_neg(make_float2(0.86602540378443865f * d.x, 0.86602540378443865f * d.y));
    v[0] = cadd(v[0], t1);
    v[1] = cadd(t2, r);
    v[2] = csub(t2, r);
}
FVFI_HD void dft(float2* v, Radix<4>) {
    const float2 a = cadd(v[0], v[2]), b = csub(v[0], v[2]);
    const float2 c = cadd(v[1], v[3]), d = cmuli_neg(csub(v[1], v[3]));
    v[0] = cadd(a, c);
    v[1] = cadd(b, d);
    v[2] = csub(a, c);
    v[3] = csub(b, d);
}
FVFI_HD void dft(float2* v, Radix<5>) {
    constexpr float c1 = 0.30901699437494742f, c2 = -0.80901699437494742f;
    constexpr float s1 = 0.95105651629515357f, s2 = 0.58778525229247313f;
    const float2 a1 = cadd(v[1], v[4]), a2 = cadd(v[2], v[3]);
    const float2 b1 = csub(v[1], v[4]), b2 = csub(v[2], v[3]);
    const float2 p1 = make_float2(v[0].x + c1 * a1.x + c2 * a2.x, v[0].y + c1 * a1.y + c2 * a2.y);
    const float2 p2 = make_float2(v[0].x + c2 * a1.x + c1 * a2.x, v[0].y + c2 * a1.y + c1 * a2.y);
    const float2 q1 = cmuli_neg(make_float2(s1 * b1.x + s2 * b2.x, s1 * b1.y + s2 * b2.y));
    const float2 q2 = cmuli_neg(make_float2(s2 * b1.x - s1 * b2.x, s2 * b1.y - s1 * b2.y));
    v[0] = make_float2(v[0].x + a1.x + a2.x, v[0].y + a1.y + a2.y);
    v[1] = cadd(p1, q1);
    v[4] = csub(p1, q1);
    v[2] = cadd(p2, q2);
    v[3] = csub(p2, q2);
}

// odd prime P: X[k], X[P-k] from the symmetric / antisymmetric halves, (P-1)^2 real FMAs
template <int P>
FVFI_HD void dft_prime(float2* v) {
    constexpr int H = (P - 1) / 2;
    float2 a[H + 1], b[H + 1];
#pragma unroll
    for (int j = 1; j <= H; ++j) {
        a[j] = cadd(v[j], v[P - j]);
        b[j] = csub(v[j], v[P - j]);
    }
    const float2 x0 = v[0];
    float2 s = x0;
#pragma unroll
    for (int j = 1; j <= H; ++j) s = cadd(s, a[j]);
    v[0] = s;
#pragma unroll
    for (int k = 1; k <= H; ++k) {
        float re = x0.x, im = x0.y, sr = 0.f, si = 0.f;
#pragma unroll
        for (int j = 1; j <= H; ++j) {
            const int t = (j * k) % P;
            const float c = RootTab<P>::c(t), sn = RootTab<P>::s(t);
            re = fmaf(a[j].x, c, re);
            im = fmaf(a[j].y, c, im);
            sr = fmaf(b[j].x, sn, sr);
            si = fmaf(b[j].y, sn, si);
        }
        v[k] = make_float2(re + si, im - sr);
        v[P - k] = make_float2(re - si, im + sr);
    }
}
FVFI_HD void dft(float2* v, Radix<7>) { dft_prime<7>(v); }
FVFI_HD void dft(float2* v, Radix<11>) { dft_prime<11>(v); }
FVFI_HD void dft(float2* v, Radix<13>) { dft_prime<13>(v); }
FVFI_HD void dft(float2* v, Radix<17>) { dft_prime<17>(v); }
FVFI_HD void dft(float2* v, Radix<19>) { dft_prime<19>(v); }

// Cooley-Tukey composite R = R1*R2 with constant twiddles: n = R2*n1 + n2, k = k1 + R1*k2
template <int R1, int R2>
FVFI_HD void dft_ct(float2* v) {
    constexpr int R = R1 * R2;
    float2 a[R2][R1];
#pragma unroll
    for (int n2 = 0; n2 < R2; ++n2) {
        float2 t[R1];
#pragma unroll
        for (int n1 = 0; n1 < R1; ++n1) t[n1] = v[R2 * n1 + n2];
        dft(t, Radix<R1>());
#pragma unroll
        for (int k1 = 0; k1 < R1; ++k1) {
            const int e = n2 * k1;                       // twiddle W_R^e
            float2 x = t[k1];
            if (e == 0) {
            } else if (4 * e == R) {
                x = cmuli_neg(x);
            } else if (2 * e == R) {
                x = make_float2(-x.x, -x.y);
            } else if (4 * e == 3 * R) {
                x = make_float2(-x.y, x.x);
            } else {
                x = cmul(x, make_float2(RootTab<R>::c(e % R), -RootTab<R>::s(e % R)));
            }
            a[n2][k1] = x;
        }
    }
#pragma unroll
    for (int k1 = 0; k1 < R1; ++k1) {
        float2 t[R2];
#pragma unroll
        for (int n2 = 0; n2 < R2; ++n2) t[n2] = a[n2][k1];
        dft(t, Radix<R2>());
#pragma unroll
        for (int k2 = 0; k2 < R2; ++k2) v[k1 + R1 * k2] = t[k2];
    }
}
FVFI_HD void dft(float2* v, Radix<8>) { dft_ct<4, 2>(v); }
FVFI_HD void dft(float2* v, Radix<9>) { dft_ct<3, 3>(v); }
FVFI_HD void dft(float2* v, Radix<16>) { dft_ct<4, 4>(v); }

// Good-Thomas (prime factor) composite, gcd(R1, R2) = 1: no twiddles, only compile-time index maps
__host__ __device__ constexpr int fft_modinv(int a, int m) {
    a %= m;
    for (int x = 1; x < m; ++x)
        if ((a * x) % m == 1) return x;
    return 1;
}
template <int R1, int R2>
FVFI_HD void dft_pfa(float2* v) {
    constexpr int R = R1 * R2;
    constexpr int E1 = R2 * fft_modinv(R2, R1), E2 = R1 * fft_modinv(R1, R2);   // CRT idempotents
    float2 a[R2][R1];
#pragma unroll
    for (int n2 = 0; n2 < R2; ++n2) {
        float2 t[R1];
#pragma unroll
        for (int n1 = 0; n1 < R1; ++n1) t[n1] = v[(R2 * n1 + R1 * n2) % R];
        dft(t, Radix<R1>());
#pragma unroll
        for (int k1 = 0; k1 < R1; ++k1) a[n2][k1] = t[k1];
    }
#pragma unroll
    for (int k1 = 0; k1 < R1; ++k1) {
        float2 t[R2];
#pragma unroll
        for (int n2 = 0; n2 < R2; ++n2) t[n2] = a[n2][k1];
        dft(t, Radix<R2>());
#pragma unroll
        for (int k2 = 0; k2 < R2; ++k2) v[(k1 * E1 + k2 * E2) % R] = t[k2];
    }
}
FVFI_HD void dft(float2* v, Radix<6>) { dft_pfa<2, 3>(v); }
FVFI_HD void dft(float2* v, Radix<10>) { dft_pfa<2, 5>(v); }
FVFI_HD void dft(float2* v, Radix<12>) { dft_pfa<4, 3>(v); }
FVFI_HD void dft(float2* v, Radix<15>) { dft_pfa<3, 5>(v); }

// v[u] *= w^u, u = 1..R-1, powers by doubling (depth log2 R, so the rounding error does not grow with R)
template <int R>
FVFI_HD void twiddle_powers(float2* v, float2 w) {
    float2 p[R > 2 ? R : 2];
    p[1] = w;
#pragma unroll
    for (int u = 2; u < R; ++u) p[u] = cmul(p[u >> 1], p[u - (u >> 1)]);
#pragma unroll
    for (int u = 1; u < R; ++u) v[u] = cmul(v[u], p[u]);
}

// ------------------------------------------------------------------------------------------------
// one network stage over `batch` sequences held in shared memory
// ------------------------------------------------------------------------------------------------
template <bool COL>
FVFI_HD int fft_addr(int b, int i, int ctshift, int pitch, int pad) {
    return COL ? ((i << ctshift) + b) : (b * pitch + i + (pad ? (i >> 4) : 0));
}

// even, so that every row of the sequence-major layout starts 16-byte aligned (rows can be landed by cp.async.bulk)
FVFI_HD int fft_row_pitch(int M, int pad) { return pad ? ((M + (M >> 4) + 2) & ~1) : ((M + 2) & ~1); }

// PAD (sequence-major layout only): the skewed addressing; without it every access is base + u*stride.
template <int R, int KIND, bool COL, bool PAD>
FVFI_HD void fft_stage_impl(const FftPlan& P, int s, const float2* in, float2* out, int batch, int ctshift,
                            int pitch, const float2* post, FftCtx cx, int src_plain = 0) {
    const int M = P.M, items = M / R, total = batch * items;
    const int sub = P.sub[s];
    const unsigned mag_sub = P.mag_sub[s], mag_items = P.mag_items[s];
    const float2* tw = P.tw;             // hoisted: the plan is in global memory and the stage stores could alias it
    constexpr bool LINEAR = COL || !PAD;
    for (int q = cx.tid; q < total; q += cx.nthr) {
        int b, t;
        if (COL) {
            t = q >> ctshift;
            b = q & ((1 << ctshift) - 1);
        } else {
            b = (int)fast_div((unsigned)q, (unsigned)items, mag_items);
            t = q - b * items;
        }
        float2 v[R];
        if (KIND == FFT_STOCKHAM) {
            const int Ns = sub;
            const int hi = (int)fast_div((unsigned)t, (unsigned)Ns, mag_sub);
            const int k = t - hi * Ns;
            if (LINEAR) {
                const float2* src = in + fft_addr<COL>(b, t, ctshift, pitch, 0);
                const int st = COL ? (items << ctshift) : items;
#pragma unroll
                for (int u = 0; u < R; ++u) v[u] = src[u * st];
            } else if (src_plain) {       // first stage of a transform whose rows were landed unskewed (bulk copy): plain reads
                const float2* src = in + fft_addr<COL>(b, t, ctshift, pitch, 0);
#pragma unroll
                for (int u = 0; u < R; ++u) v[u] = src[u * items];
            } else {
#pragma unroll
                for (int u = 0; u < R; ++u) v[u] = in[fft_addr<COL>(b, t + u * items, ctshift, pitch, 1)];
            }
            if (Ns > 1) twiddle_powers<R>(v, ldg_(tw + k * (M / (Ns * R))));
            dft(v, Radix<R>());
            const int o = hi * Ns * R + k;
            if (LINEAR) {
                float2* dst = out + fft_addr<COL>(b, o, ctshift, pitch, 0);
                const int st = COL ? (Ns << ctshift) : Ns;
#pragma unroll
                for (int u = 0; u < R; ++u) dst[u * st] = v[u];
            } else {
#pragma unroll
                for (int u = 0; u < R; ++u) out[fft_addr<COL>(b, o + u * Ns, ctshift, pitch, 1)] = v[u];
            }
        } else {
            const int m = sub;                                    // butterfly stride; block length R*m
            const int c = (int)fast_div((unsigned)t, (unsigned)m, mag_sub);
            const int j = t - c * m;
            const int base = c * R * m + j;
            const int st = COL ? (m << ctshift) : m;
            const int a0 = fft_addr<COL>(b, base, ctshift, pitch, 0);
#pragma unroll
            for (int u = 0; u < R; ++u)
                v[u] = LINEAR ? in[a0 + u * st] : in[fft_addr<COL>(b, base + u * m, ctshift, pitch, 1)];
            if (KIND == FFT_DIT && m > 1) {
                // decimation-in-time Rader: the length-m blocks hold their spectrum in generator order; `perm` names the frequency
                const int jf = P.rader ? (int)ldg_(P.perm + j) : j;
                twiddle_powers<R>(v, ldg_(tw + jf * (M / (R * m))));
            }
            dft(v, Radix<R>());
            if (KIND == FFT_DIF && m > 1) twiddle_powers<R>(v, ldg_(tw + j * (M / (R * m))));
            if (KIND == FFT_DIF && post) {                        // Bluestein: spectrum of the chirp filter, then conj
#pragma unroll
                for (int u = 0; u < R; ++u) v[u] = cconj(cmul(v[u], ldg_(post + base + u * m)));
            }
#pragma unroll
            for (int u = 0; u < R; ++u) {
                if (LINEAR) out[a0 + u * st] = v[u];
                else out[fft_addr<COL>(b, base + u * m, ctshift, pitch, 1)] = v[u];
            }
        }
    }
}

// Rader sub-FFT stage: in-place DIF / DIT butterflies on the (p-1)-point sub-sequences that sit at offset 1 of every length-p
// block of `buf` (rr blocks per sequence).  POST (last DIF stage): multiply by the convolution spectrum, fold y0 (slot 0 of the
// block) into the DC bin, leave X[0] in slot 0, conjugate (the inverse transform is conj -> forward DIT -> conj, the last conj
// being applied by the last DIT stage).
template <int R, int KIND, bool COL>
FVFI_HD void fft_stage_sub_impl(const FftPlan& P, int s, float2* buf, int batch, int ctshift, int pitch, const float2* post,
                                FftCtx cx) {
    const int rq = P.rq, rp = P.rp, qitems = rq / R, items = P.rr * qitems, total = batch * items;
    const int m = P.sub[s];
    const unsigned mag_sub = P.mag_sub[s], mag_q = P.mag_items[s], mag_items = P.mag_ritems[s];
    const float2* tw = P.tw2;
    for (int q = cx.tid; q < total; q += cx.nthr) {
        int b, t;
        if (COL) {
            t = q >> ctshift;
            b = q & ((1 << ctshift) - 1);
        } else {
            b = (int)fast_div((unsigned)q, (unsigned)items, mag_items);
            t = q - b * items;
        }
        const int blk = (int)fast_div((unsigned)t, (unsigned)qitems, mag_q);
        const int tt = t - blk * qitems;
        const int c = (int)fast_div((unsigned)tt, (unsigned)m, mag_sub);
        const int j = tt - c * m;
        const int base = c * R * m + j;                       // position inside the sub-sequence
        const int a0 = fft_addr<COL>(b, blk * rp + 1 + base, ctshift, pitch, 0);
        const int st = COL ? (m << ctshift) : m;
        float2 v[R];
#pragma unroll
        for (int u = 0; u < R; ++u) v[u] = buf[a0 + u * st];
        if (KIND == FFT_DIT && m > 1) twiddle_powers<R>(v, ldg_(tw + j * (rq / (R * m))));
        dft(v, Radix<R>());
        if (KIND == FFT_DIF && m > 1) twiddle_powers<R>(v, ldg_(tw + j * (rq / (R * m))));
        if (KIND == FFT_DIF && post) {
#pragma unroll
            for (int u = 0; u < R; ++u) {
                float2 w = cmul(v[u], ldg_(post + base + u * m));
                if (u == 0 && base == 0) {                    // DC bin of this block: X[0] = y0 + sum, and y0 rides on every output
                    const int a00 = fft_addr<COL>(b, blk * rp, ctshift, pitch, 0);
                    const float2 y0 = buf[a00];
                    buf[a00] = cadd(y0, v[0]);
                    w = cadd(w, y0);
                }
                v[u] = cconj(w);
            }
        }
        // the last stage of the inverse sub-transform finishes the conj -> forward -> conj identity here (the outer radix stages
        // that follow need the true block spectra)
        const bool conj_out = KIND == FFT_DIT && s == P.nouter;
#pragma unroll
        for (int u = 0; u < R; ++u) buf[a0 + u * st] = conj_out ? cconj(v[u]) : v[u];
    }
}

#if defined(__CUDA_ARCH__)
#define FVFI_STAGE_ATTR __device__ __noinline__
#else
#define FVFI_STAGE_ATTR __host__ __device__
#endif

// Out-of-line per (radix, kind, layout): the stage bodies are shared by every kernel of the translation unit.
template <int R, int KIND, bool COL, bool PAD>
FVFI_STAGE_ATTR void fft_stage(const FftPlan* P, int s, const float2* in, float2* out, int batch, int ctshift, int pitch,
                               const float2* post, int tid, int nthr, int src_plain) {
    fft_stage_impl<R, KIND, COL, PAD>(*P, s, in, out, batch, ctshift, pitch, post, FftCtx{tid, nthr}, src_plain);
}

template <int R, int KIND, bool COL>
FVFI_STAGE_ATTR void fft_stage_sub(const FftPlan* P, int s, float2* buf, int batch, int ctshift, int pitch, const float2* post,
                                   int tid, int nthr) {
    fft_stage_sub_impl<R, KIND, COL>(*P, s, buf, batch, ctshift, pitch, post, FftCtx{tid, nthr});
}

template <int KIND, bool COL>
FVFI_HD void fft_run_stage_sub(const FftPlan& P, int s, float2* buf, int batch, int ctshift, int pitch, const float2* post,
                               FftCtx cx) {
#define FVFI_CASE(R) \
    case R: fft_stage_sub<R, KIND, COL>(&P, s, buf, batch, ctshift, pitch, post, cx.tid, cx.nthr); break;
    switch (P.fac[s]) {
        FVFI_CASE(2) FVFI_CASE(3) FVFI_CASE(4) FVFI_CASE(5) FVFI_CASE(6) FVFI_CASE(7) FVFI_CASE(8) FVFI_CASE(9)
        FVFI_CASE(10) FVFI_CASE(11) FVFI_CASE(12) FVFI_CASE(13) FVFI_CASE(15) FVFI_CASE(16) FVFI_CASE(17) FVFI_CASE(19)
        default: break;
    }
#undef FVFI_CASE
}

template <int KIND, bool COL>
FVFI_HD void fft_run_stage(const FftPlan& P, int s, const float2* in, float2* out, int batch, int ctshift, int pitch,
                           const float2* post, FftCtx cx, int src_plain = 0) {
#define FVFI_CASE(R)                                                                                               \
    case R:                                                                                                        \
        if (!COL && P.pad) fft_stage<R, KIND, COL, !COL>(&P, s, in, out, batch, ctshift, pitch, post, cx.tid, cx.nthr, src_plain); \
        else fft_stage<R, KIND, COL, false>(&P, s, in, out, batch, ctshift, pitch, post, cx.tid, cx.nthr, 0);       \
        break;
    switch (P.fac[s]) {
        FVFI_CASE(2) FVFI_CASE(3) FVFI_CASE(4) FVFI_CASE(5) FVFI_CASE(6) FVFI_CASE(7) FVFI_CASE(8) FVFI_CASE(9)
        FVFI_CASE(10) FVFI_CASE(11) FVFI_CASE(12) FVFI_CASE(13) FVFI_CASE(15) FVFI_CASE(16) FVFI_CASE(17) FVFI_CASE(19)
        default: break;
    }
#undef FVFI_CASE
}

FVFI_HD void fft_sync() {
#if defined(__CUDA_ARCH__)
    __syncthreads();
#endif
}

struct FftResult {
    float2* buf;                 // where the transform is
    const unsigned short* perm;  // non-null: position p holds natural index perm[p]
};

// What fft_put / fft_get need from a plan, read ONCE per kernel (the plan lives in global memory: re-reading `bluestein` / `pad`
// per element put an L1 round trip on every load and store of the prologue / epilogue loops).
struct FftIO {
    int bluestein, pad, rader;
    const float2* chirp;
    const unsigned short* inv;
    const unsigned short* pos_in;
};
FVFI_HD FftIO fft_io(const FftPlan& P) { return FftIO{P.bluestein, P.pad, P.rader, P.chirp, P.inv, P.pos_in}; }

// Pitch (floats2 per sequence) of the sequence-major layout for this plan.
FVFI_HD int fft_pitch(const FftPlan& P) { return fft_row_pitch(P.M, P.pad); }

// Callers WRITE their input through fft_put (Bluestein: the chirp is applied on the way in) ...
template <bool COL>
FVFI_HD void fft_put(const FftIO& io, float2* buf, int b, int i, float2 v, int ctshift, int pitch) {
    if (io.bluestein) v = cmul(v, ldg_(io.chirp + i));
    if (io.pos_in) i = (int)ldg_(io.pos_in + i);                 // decimation-in-time Rader: residue block, generator-order slot
    buf[fft_addr<COL>(b, i, ctshift, pitch, io.pad)] = v;
}
// ... and READ the result through fft_get (Bluestein: conj + chirp on the way out).  pos < n; the natural index
// of the value is R.perm ? R.perm[pos] : pos.
template <bool COL>
FVFI_HD float2 fft_get(const FftIO& io, const FftResult& R, int b, int pos, int ctshift, int pitch) {
    if (io.rader) {      // result sits in generator order: the column layout walks positions (R.perm names them), rows look them up
        const int p2 = COL ? pos : (int)ldg_(io.inv + pos);
        return R.buf[fft_addr<COL>(b, p2, ctshift, pitch, 0)];
    }
    const float2 v = R.buf[fft_addr<COL>(b, pos, ctshift, pitch, io.pad)];
    return io.bluestein ? cmul(cconj(v), ldg_(io.chirp + pos)) : v;
}

// Forward DFT of `batch` sequences of logical length P.n, written with fft_put at positions [0, n) of `a`
// (Bluestein transforms need room for P.M positions per sequence).  `b` is the second buffer of the out-of-place
// network (may be null when inplace).  The input must be visible to all threads on entry (caller syncs); on return
// the result is visible (trailing sync) and is read with fft_get.
template <bool COL>
// `src_plain`: the rows of `a` were written WITHOUT the skew (element i of sequence s at s*pitch + i -- what a bulk copy of a row
// delivers) although the plan uses the skewed layout: only valid for the out-of-place (Stockham) network, whose first stage then
// reads plainly and writes skewed.  Plans without skew (Rader, odd first radix) need nothing.
FVFI_HD FftResult fft_forward(const FftPlan& P, float2* a, float2* b, int batch, int ctshift, int pitch, bool inplace,
                              FftCtx cx, int src_plain = 0) {
    const int M = P.M, n = P.n, pad = P.pad;
    if (P.rader) {
        // fft_put has scattered the inputs into residue blocks in generator order; Rader on every block in place, then the
        // radix stages of r across the blocks (twiddle index through `perm`: the blocks are in generator order)
        for (int s = P.nouter; s < P.nfac; ++s) {
            fft_run_stage_sub<FFT_DIF, COL>(P, s, a, batch, ctshift, pitch, s == P.nfac - 1 ? P.bhat : nullptr, cx);
            fft_sync();
        }
        for (int s = P.nfac - 1; s >= P.nouter; --s) {
            fft_run_stage_sub<FFT_DIT, COL>(P, s, a, batch, ctshift, pitch, nullptr, cx);
            fft_sync();
        }
        for (int s = P.nouter - 1; s >= 0; --s) {
            fft_run_stage<FFT_DIT, COL>(P, s, a, a, batch, ctshift, pitch, nullptr, cx);
            fft_sync();
        }
        return FftResult{a, P.perm};
    }
    if (P.bluestein) {
        const int tail = M - n;                              // zero padding of the convolution
        for (int q = cx.tid; q < batch * tail; q += cx.nthr) {
            int bb, i;
            if (COL) { i = q >> ctshift; bb = q & ((1 << ctshift) - 1); } else { bb = q / tail; i = q - bb * tail; }
            a[fft_addr<COL>(bb, n + i, ctshift, pitch, pad)] = make_float2(0.f, 0.f);
        }
        fft_sync();
        for (int s = 0; s < P.nfac; ++s) {
            fft_run_stage<FFT_DIF, COL>(P, s, a, a, batch, ctshift, pitch, s == P.nfac - 1 ? P.bhat : nullptr, cx);
            fft_sync();
        }
        for (int s = P.nfac - 1; s >= 0; --s) {
            fft_run_stage<FFT_DIT, COL>(P, s, a, a, batch, ctshift, pitch, nullptr, cx);
            fft_sync();
        }
        return FftResult{a, nullptr};
    }
    if (inplace) {
        for (int s = 0; s < P.nfac; ++s) {
            fft_run_stage<FFT_DIF, COL>(P, s, a, a, batch, ctshift, pitch, nullptr, cx);
            fft_sync();
        }
        return FftResult{a, P.perm};
    }
    for (int s = 0; s < P.nfac; ++s) {
        fft_run_stage<FFT_STOCKHAM, COL>(P, s, a, b, batch, ctshift, pitch, nullptr, cx, s == 0 ? src_plain : 0);
        fft_sync();
        float2* t = a; a = b; b = t;
    }
    return FftResult{a, nullptr};
}

}  // namespace fvfi
