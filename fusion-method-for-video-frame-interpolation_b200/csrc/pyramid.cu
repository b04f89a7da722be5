// pyramid.cu -- complex steerable pyramid (decompose / reconstruct) for sm_100a.
//
// Replaces steerable.SCFpyr_PyTorch.build / .reconstruct (third party, absent from the reference;
// call sites src/train/pyramid.py:28-33,37,44) fused with Pyramid.coeff_to_values /
// values_to_coeff (src/train/pyramid.py:48-112).  Algorithm: SURVEY.md Appendix A (restated in
// oracle/steerable_shim.py).  B200-first formulation:
//
//  * FLATTENED recursion.  The reference recursion (mask, band IFFT, crop, mask, ...) is linear in
//    the image spectrum X, so band(l,b) = IFFT2_{h_l x w_l}( X[k] * D_l[k] * A_b[k] * (-i)^(nb-1) )
//    with one radial table D_l = lo0 * prod_{j<l} lomask_j * himask_l per level (plan, built on the
//    host in double with the same LUT interpolation the oracle uses) and the angular factor
//    A_b = 2 sqrt(c) cos(theta - pi b/nb)^(nb-1) [cos > 0] evaluated in closed form from the
//    frequency coordinates (no atan2, no table).  Every level depends only on X, so all levels are
//    independent: the large levels are one launch each, all small levels share ONE launch per pass
//    (job table + tile prefix), and reconstruction sums the level spectra in one gather.
//  * Every 1-D transform of any length (764 = 4*191, 1358 = 2*7*97, 241, ...) runs in shared memory
//    with register butterflies (fft_engine.cuh): mixed radix up to 16/15 for smooth lengths (three
//    stages at 1080 / 1920), Bluestein on a smooth length for the rest.  Row passes work on batches
//    of rows (autosort network, natural order in and out, coalesced); column passes on tiles of 8
//    adjacent columns (64-byte row segments) with an in-place network whose digit-reversed output
//    order is absorbed by the store.  Inverse transforms are conj -> forward -> conj with the
//    conjugations fused into the spectrum loader and the output epilogue.
//  * Fused epilogues/prologues: amplitude |z|, phase atan2(im,re), the per-(level,plane) amplitude
//    maximum (PhaseNet.normalize_vals, src/phase_net/phase_net.py:47-59) are produced by the last
//    row pass of the band IFFT -- the complex band never goes to HBM; reconstruction reads
//    (phase, amplitude) and forms A*(cos,sin) in the first row pass (pyramid.py:103-108).
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <map>
#include <memory>
#include <thread>
#include <vector>

#include "common.cuh"
#include "fft_plan.hpp"

namespace fvfi {

constexpr int MAX_LEVELS = 40;
constexpr int MAX_BANDS = 8;
constexpr int MAX_SET = 24;                       // jobs per merged launch
// 9 warps per CTA, 3 CTAs per SM (72 registers): the kernels are latency-bound at 24 resident warps -- same-call A/B on 12 planes of 1080p
// (closing session): 256 threads 5.13 / 6.56 ms decompose / reconstruct, 288: 5.00 / 6.30, 320 (64 registers, spills): 5.04 / 6.32;
// PYR_MIN_CTAS 2: 5.99 / 7.47, 4 (64 registers): 5.19 / 6.58.  Results are bit-identical for any block size.
#ifndef PYR_NTHREADS
#define PYR_NTHREADS 288
#endif
constexpr int PYR_THREADS = PYR_NTHREADS;
#ifndef PYR_MIN_CTAS
#define PYR_MIN_CTAS 3
#endif
#ifndef COL_SMEM_KB
#define COL_SMEM_KB 76
#endif
constexpr size_t COL_SMEM_MAX = COL_SMEM_KB * 1024;   // in-place column tile: at least three CTAs per SM (two for the 113 KB of round 1)
constexpr size_t ROW_SMEM_TARGET = 72 * 1024;     // row batch: three CTAs per SM
constexpr int SMALL_LEVEL_ELEMS = 300 * 520;      // levels at or below this size share one launch per pass

struct LevelGeom {
    int h, w;
    size_t off;          // offset (complex elements, per plane) of this level's spectrum in region C
    float rad2_lo, rad2_hi;  // radial support of D_l in normalised radius^2 (for the gather)
};

struct AngParams {
    int nb, order;
    float cs[MAX_BANDS], sn[MAX_BANDS];
    float scale;      // 2*sqrt(const) (build, one-sided) or sqrt(const) (reconstruct, two-sided)
    float2 fac;       // (-i)^(nb-1) (build) or (i)^(nb-1) (reconstruct)
    int one_sided;
    float inv_hh, inv_hw;  // 2/H, 2/W of the FULL image (grid coordinates, prepare_grid)
};

// One entry per level (0..L-1 bands, L = low residual, L+1 = full-size plane: image FFT / high residual).
struct LevelJob {
    int h, w, nb, is_band;
    int ct_shift, rb;            // column tile = 1 << ct_shift columns; rows per CTA in a row pass
    int col_tiles, row_tiles;
    int ct_shift_c, col_tiles_c; // column tile of the band-combining pass (two buffers per tile)
    unsigned mag_w;              // ceil(2^32 / w)
    long long t_off;             // intermediate T of this level starts at regionB + N * t_off (complex elements)
    long long c_off;             // per-plane offset of the level spectrum in region C
    const float* radial;         // D_l (band levels), low-pass product (L), hi0 (L+1)
    const float* band_build;     // band levels: [nb][h][w] = D_l * one-sided angular mask (decomposition); null otherwise
    const float* band_rec;       // band levels: [nb][h][w] = D_l * two-sided angular mask (reconstruction and its adjoint)
    FftPlan fy, fx;              // column / row transforms
};

struct SetEntry {
    int job, start, mode;
    float scale;             // row-pass output scale; 0 = the IFFT normalisation 1/(h*w)
    const float* p0;
    const float* p1;
    float* q0;
    float* q1;
    float* aux;
};
struct LaunchSet {
    int n, total;
    SetEntry e[MAX_SET];
};

}  // namespace fvfi

struct fvfi_pyr_plan {
    int H, W, height, nbands, L;
    double scale;
    std::vector<fvfi::LevelGeom> lv;            // L band levels + low residual (index L)
    std::vector<fvfi::LevelJob> jobs;           // host copy of the job table (L + 2 entries)
    const fvfi::LevelJob* d_jobs = nullptr;     // device job table
    std::vector<const float*> radial;           // device, per level (index L = low-pass product)
    std::vector<const float*> band_build, band_rec;   // device, per band level: [nb][h_l][w_l] combined radial x angular masks
    const float* hi0 = nullptr;                 // device [H*W], unshifted
    const float* hf_transfer = nullptr;         // device [H*W]: transfer function of  reconstruct(high + finest level of decompose(x))
    std::map<std::pair<int, int>, fvfi::FftPlan> fft_cache;   // (length, stockham) -> plan with device tables
    std::vector<void*> owned;
    size_t level_elems = 0;                     // sum_l h_l*w_l  (l = 0..L)
    fvfi::AngParams ang_build, ang_rec;
};

namespace fvfi {

// ------------------------------------------------------------------------------------------------
// host: plan
// ------------------------------------------------------------------------------------------------
static int next_size(int n, double s) { return (int)ceil((n - 0.5) / s - 1e-9); }

// numpy.interp on an increasing abscissa (end-clamped) -- what upstream's pointOp does.
static double interp(double x, const std::vector<double>& X, const std::vector<double>& Y) {
    const int n = (int)X.size();
    if (x <= X[0]) return Y[0];
    if (x >= X[n - 1]) return Y[n - 1];
    int lo = 0, hi = n - 1;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (X[mid] <= x) lo = mid; else hi = mid;
    }
    const double slope = (Y[hi] - Y[lo]) / (X[hi] - X[lo]);
    return slope * (x - X[lo]) + Y[lo];
}

static inline int sfreq_h(int k, int n) { return k < (n + 1) / 2 ? k : k - n; }

template <typename T>
static int upload(fvfi_pyr_plan* p, const std::vector<T>& v, const T** out) {
    void* d = nullptr;
    FVFI_CUDA(cudaMalloc(&d, v.size() * sizeof(T)));
    p->owned.push_back(d);
    FVFI_CUDA(cudaMemcpy(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = (const T*)d;
    return FVFI_OK;
}


// FFT plan with device-resident tables, cached per (length, network kind)
static int get_fft(fvfi_pyr_plan* p, int n, bool stockham, FftPlan* out) {
    auto key = std::make_pair(n, stockham ? 1 : 0);
    auto it = p->fft_cache.find(key);
    if (it != p->fft_cache.end()) { *out = it->second; return FVFI_OK; }
    HostFftPlan H;
    if (!fft_make_plan(n, stockham, H)) { set_error("pyramid: no FFT plan for length %d", n); return FVFI_EINVAL; }
    FftPlan f = H.p;
    if (int rc = upload(p, H.tw, &f.tw)) return rc;
    f.perm = nullptr;
    f.chirp = nullptr;
    f.bhat = nullptr;
    f.tw2 = nullptr;
    f.inv = nullptr;
    f.pos_in = nullptr;
    if (f.rader) {
        if (int rc = upload(p, H.pos_in, &f.pos_in)) return rc;
        if (int rc = upload(p, H.perm, &f.perm)) return rc;
        if (int rc = upload(p, H.bhat, &f.bhat)) return rc;
        if (int rc = upload(p, H.tw2, &f.tw2)) return rc;
        if (int rc = upload(p, H.inv, &f.inv)) return rc;
    } else if (f.bluestein) {
        if (int rc = upload(p, H.chirp, &f.chirp)) return rc;
        if (int rc = upload(p, H.bhat, &f.bhat)) return rc;
    } else if (!stockham) {
        if (int rc = upload(p, H.perm, &f.perm)) return rc;
    }
    p->fft_cache[key] = f;
    *out = f;
    return FVFI_OK;
}

static size_t row_bytes_per_row(const FftPlan& fx) {
    // Bluestein and Rader run in place; Stockham uses two buffers
    return (size_t)((fx.bluestein || fx.rader) ? 1 : 2) * fft_pitch(fx) * sizeof(float2);
}

static int build_jobs(fvfi_pyr_plan* p) {
    const int L = p->L, nb = p->nbands;
    p->jobs.assign(L + 2, LevelJob{});
    for (int l = 0; l <= L + 1; ++l) {
        LevelJob& J = p->jobs[l];
        const bool full = (l == L + 1);
        J.h = full ? p->H : p->lv[l].h;
        J.w = full ? p->W : p->lv[l].w;
        J.nb = (l < L) ? nb : 1;
        J.is_band = (l < L) ? 1 : 0;
        J.radial = full ? p->hi0 : p->radial[l];
        J.band_build = (l < L) ? p->band_build[l] : nullptr;
        J.band_rec = (l < L) ? p->band_rec[l] : nullptr;
        J.t_off = full ? (long long)nb * (long long)p->level_elems : (long long)nb * (long long)p->lv[l].off;
        J.c_off = full ? 0 : (long long)p->lv[l].off;
        J.mag_w = fft_magic((unsigned)J.w);
        if (int rc = get_fft(p, J.h, false, &J.fy)) return rc;
        if (int rc = get_fft(p, J.w, true, &J.fx)) return rc;
        int cs = 3;
        while (cs > 0 && ((size_t)J.fy.M << cs) * sizeof(float2) > COL_SMEM_MAX) --cs;
        if (((size_t)J.fy.M << cs) * sizeof(float2) > 220 * 1024) { set_error("pyramid: column length %d too large", J.h); return FVFI_EINVAL; }
        J.ct_shift = cs;
        const size_t per_row = row_bytes_per_row(J.fx);
        if (per_row > 220 * 1024) { set_error("pyramid: row length %d too large", J.w); return FVFI_EINVAL; }
        int rb = (int)(ROW_SMEM_TARGET / per_row);
        rb = std::max(1, std::min(std::min(rb, 16), J.h));
        J.rb = rb;
        J.col_tiles = ceil_div(J.w, 1 << cs);
        int cc = cs;                 // combine pass: transform buffer + accumulator, aim for three CTAs per SM
        while (cc > 2 && (((size_t)J.fy.M + J.h) << cc) * sizeof(float2) > 75 * 1024) --cc;
        J.ct_shift_c = cc;
        J.col_tiles_c = ceil_div(J.w, 1 << cc);
        J.row_tiles = ceil_div(J.h, rb);
    }
    const LevelJob* d = nullptr;
    if (int rc = upload(p, p->jobs, &d)) return rc;
    p->d_jobs = d;
    return FVFI_OK;
}

static int build_plan(fvfi_pyr_plan* p) {
    const int H = p->H, W = p->W, L = p->L, nb = p->nbands;
    const double s = p->scale, dlt = log2(s);
    // level sizes (SURVEY.md Appendix A.4 / oracle.steerable_shim.level_sizes)
    p->lv.resize(L + 1);
    p->radial.resize(L + 1);
    int h = H, w = W;
    size_t off = 0;
    for (int l = 0; l <= L; ++l) {
        p->lv[l].h = h;
        p->lv[l].w = w;
        p->lv[l].off = off;
        off += (size_t)h * w;
        h = next_size(h, s);
        w = next_size(w, s);
    }
    p->level_elems = off;
    // the level-size rule stops shrinking at 2 samples: a pyramid that tall has degenerate (repeated) levels
    for (int l = 0; l < L; ++l)
        if (p->lv[l + 1].h >= p->lv[l].h || p->lv[l + 1].w >= p->lv[l].w || p->lv[l + 1].h < 2 || p->lv[l + 1].w < 2) {
            set_error("pyramid: height %d too large for %dx%d", p->height, H, W);
            return FVFI_EINVAL;
        }

    // raised-cosine tables (upstream rcosFn(1, -0.5))
    const int NT = 259;
    std::vector<double> Xr(NT), Yr(NT), YIr(NT);
    for (int i = 0; i < NT; ++i) {
        const double X0 = M_PI * (double)(i - 257) / 512.0;
        double Y = cos(X0) * cos(X0);
        Yr[i] = Y;
        Xr[i] = -0.5 + 2.0 / M_PI * (X0 + M_PI / 4.0);
    }
    Yr[0] = Yr[1];
    Yr[NT - 1] = Yr[NT - 2];
    for (int i = 0; i < NT; ++i) {
        Yr[i] = sqrt(Yr[i]);
        YIr[i] = sqrt(fabs(1.0 - Yr[i] * Yr[i]));
    }
    auto shifted = [&](double d) { std::vector<double> X(Xr); for (auto& x : X) x -= d; return X; };
    std::vector<std::vector<double>> Xlev(L + 1);
    for (int j = 0; j <= L; ++j) Xlev[j] = shifted((j + 1) * dlt);

    auto log_rad = [&](int fy, int fx) {
        double xv = fx * 2.0 / W, yv = fy * 2.0 / H;
        if (fy == 0 && fx == 0) xv = -2.0 / W;  // prepare_grid: DC sample replaced by its left neighbour
        return log2(sqrt(xv * xv + yv * yv));
    };
    auto clean = [](double v) { return fabs(v) < 1e-12 ? 0.0 : v; };

    // hi0 on the full grid
    std::vector<float> hi0_host((size_t)H * W);
    {
        std::vector<float>& t = hi0_host;
        for (int ky = 0; ky < H; ++ky)
            for (int kx = 0; kx < W; ++kx)
                t[(size_t)ky * W + kx] = (float)clean(interp(log_rad(sfreq_h(ky, H), sfreq_h(kx, W)), Xr, Yr));
        if (int rc = upload(p, t, &p->hi0)) return rc;
    }
    // D_l = lo0 * prod_{j<l} lomask_j * himask_l ;  low = lo0 * prod_{j<L} lomask_j
    for (int l = 0; l <= L; ++l) {
        const int hl = p->lv[l].h, wl = p->lv[l].w;
        std::vector<float> t((size_t)hl * wl);
        for (int ky = 0; ky < hl; ++ky)
            for (int kx = 0; kx < wl; ++kx) {
                const double lr = log_rad(sfreq_h(ky, hl), sfreq_h(kx, wl));
                double v = interp(lr, Xr, YIr);
                for (int j = 0; j < l && v != 0.0; ++j) v *= interp(lr, Xlev[j], YIr);
                if (l < L) v *= interp(lr, Xlev[l], Yr);
                t[(size_t)ky * wl + kx] = (float)clean(v);
            }
        if (int rc = upload(p, t, &p->radial[l])) return rc;
        // radial support (log2 radius): himask_l > 0 above -(l+1)dlt - 1 ; lo-product > 0 below -l*dlt (0 for l=0)
        const double lo = (l < L) ? -(l + 1) * dlt - 1.0 : -1e30;
        const double hi = -(double)l * dlt;
        p->lv[l].rad2_lo = (l < L) ? (float)(pow(2.0, 2.0 * lo) * (1.0 - 1e-4)) : -1.f;
        p->lv[l].rad2_hi = (float)(pow(2.0, 2.0 * hi) * (1.0 + 1e-4));
    }
    // Combined band masks  D_l * anglemask_b, with the angular mask computed EXACTLY as the published algorithm does (upstream
    // SCFpyr: angle = arctan2 on the cropped prepare_grid, then np.interp in the 1024-step cos^(nb-1) lookup table shifted by
    // pi*b/nb -- one-sided table for build, two-sided for reconstruct).  A closed-form cos^(nb-1) differs from the interpolated
    // table by up to 3e-6 relative, which PhaseNet turns into 1e-4 .. 5e-3 output differences (phase of weak coefficients);
    // evaluating the table in double here makes the masks equal to the oracle's to float32 rounding.
    {
        const int order_ = nb - 1, lutsize = 1024, NL = 3 * lutsize + 3;      // Xcosn = pi * (-(2*lutsize+1) .. lutsize+1) / lutsize
        double fo_ = 1, f2o_ = 1;
        for (int i = 2; i <= order_; ++i) fo_ *= i;
        for (int i = 2; i <= 2 * order_; ++i) f2o_ *= i;
        const double cst_ = pow(2.0, 2.0 * order_) * fo_ * fo_ / (nb * f2o_);
        std::vector<double> Xc(NL), Y1(NL), Y2(NL);
        for (int i = 0; i < NL; ++i) {
            Xc[i] = M_PI * (double)(i - (2 * lutsize + 1)) / lutsize;
            const double cp = pow(cos(Xc[i]), (double)order_);
            double alpha = fmod(Xc[i] + M_PI, 2.0 * M_PI);                    // numpy %: result has the sign of the divisor
            if (alpha < 0) alpha += 2.0 * M_PI;
            alpha -= M_PI;
            Y1[i] = 2.0 * sqrt(cst_) * cp * (fabs(alpha) < M_PI / 2 ? 1.0 : 0.0);
            Y2[i] = sqrt(cst_) * cp;
        }
        p->band_build.assign(L, nullptr);
        p->band_rec.assign(L, nullptr);
        for (int l = 0; l < L; ++l) {
            const int hl = p->lv[l].h, wl = p->lv[l].w;
            const size_t plane = (size_t)hl * wl;
            std::vector<float> rad(plane);
            FVFI_CUDA(cudaMemcpy(rad.data(), p->radial[l], plane * sizeof(float), cudaMemcpyDeviceToHost));
            std::vector<float> t1((size_t)nb * plane), t2((size_t)nb * plane);
            auto rows = [&](int y_begin, int y_end) {
                std::vector<double> Xs(NL);
                for (int ky = y_begin; ky < y_end; ++ky)
                    for (int kx = 0; kx < wl; ++kx) {
                        const size_t o = (size_t)ky * wl + kx;
                        const double d = rad[o];
                        if (d == 0.0) {
                            for (int b = 0; b < nb; ++b) t1[b * plane + o] = t2[b * plane + o] = 0.f;
                            continue;
                        }
                        const double xv = sfreq_h(kx, wl) * 2.0 / W, yv = sfreq_h(ky, hl) * 2.0 / H;
                        const double ang = atan2(yv, xv);
                        for (int b = 0; b < nb; ++b) {
                            const double sh = M_PI * b / nb;
                            // np.interp(ang, Xc + sh, Y): locate the interval directly (uniform abscissa), then numpy's formula
                            int j = (int)floor((ang - sh - Xc[0]) / (M_PI / lutsize));
                            j = std::max(0, std::min(NL - 2, j));
                            while (j > 0 && Xc[j] + sh > ang) --j;
                            while (j < NL - 2 && Xc[j + 1] + sh <= ang) ++j;
                            const double x0 = Xc[j] + sh, x1 = Xc[j + 1] + sh;
                            const double a1 = (Y1[j + 1] - Y1[j]) / (x1 - x0) * (ang - x0) + Y1[j];
                            const double a2 = (Y2[j + 1] - Y2[j]) / (x1 - x0) * (ang - x0) + Y2[j];
                            // float32 masks multiplied in float32, like the oracle's torch tensors
                            t1[b * plane + o] = (float)d * (float)a1;
                            t2[b * plane + o] = (float)d * (float)a2;
                        }
                    }
            };
            const int nthr = (int)std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
            if (plane < 65536 || nthr == 1) {
                rows(0, hl);
            } else {
                std::vector<std::thread> pool;
                for (int t = 0; t < nthr; ++t) pool.emplace_back(rows, (int)((long long)hl * t / nthr), (int)((long long)hl * (t + 1) / nthr));
                for (auto& th : pool) th.join();
            }
            if (int rc = upload(p, t1, &p->band_build[l])) return rc;
            if (int rc = upload(p, t2, &p->band_rec[l])) return rc;
            if (l == 0) {
                // Decomposing an image and reconstructing ONLY its high residual and finest band level (get_last_value_levels(., 1),
                // src/train/utils.py:242-280) is a linear filter: Re IFFT2( X * T ),  T = hi0^2 + sum_b (D_0 A_b^one)(D_0 A_b^two)
                // ((-i)^(nb-1) (i)^(nb-1) = 1; the coefficients pass through amplitude / phase and back unchanged).  The real part of
                // the inverse transform symmetrises the spectrum, and X is Hermitian (real image): T_sym(k) = (T(k) + T(-k)) / 2.
                std::vector<double> T(plane);
                for (size_t o = 0; o < plane; ++o) {
                    double v = (double)hi0_host[o] * hi0_host[o];
                    for (int b = 0; b < nb; ++b) v += (double)t1[b * plane + o] * (double)t2[b * plane + o];
                    T[o] = v;
                }
                std::vector<float> Ts(plane);
                for (int ky = 0; ky < hl; ++ky)
                    for (int kx = 0; kx < wl; ++kx)
                        Ts[(size_t)ky * wl + kx] = (float)(0.5 * (T[(size_t)ky * wl + kx] + T[(size_t)((hl - ky) % hl) * wl + (wl - kx) % wl]));
                if (int rc = upload(p, Ts, &p->hf_transfer)) return rc;
            }
        }
    }
    // angular parameters
    const int order = nb - 1;
    double fo = 1, f2o = 1;
    for (int i = 2; i <= order; ++i) fo *= i;
    for (int i = 2; i <= 2 * order; ++i) f2o *= i;
    const double cst = pow(2.0, 2.0 * order) * fo * fo / (nb * f2o);
    AngParams a{};
    a.nb = nb;
    a.order = order;
    for (int b = 0; b < nb; ++b) { a.cs[b] = (float)cos(M_PI * b / nb); a.sn[b] = (float)sin(M_PI * b / nb); }
    a.inv_hh = (float)(2.0 / H);
    a.inv_hw = (float)(2.0 / W);
    // (-i)^(nb-1) and (i)^(nb-1)
    const float2 pw_m[4] = {{1, 0}, {0, -1}, {-1, 0}, {0, 1}};
    const float2 pw_p[4] = {{1, 0}, {0, 1}, {-1, 0}, {0, -1}};
    p->ang_build = a;
    p->ang_build.scale = (float)(2.0 * sqrt(cst));
    p->ang_build.fac = pw_m[order & 3];
    p->ang_build.one_sided = 1;
    p->ang_rec = a;
    p->ang_rec.scale = (float)sqrt(cst);
    p->ang_rec.fac = pw_p[order & 3];
    p->ang_rec.one_sided = 0;
    return build_jobs(p);
}


// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int sfreq(int k, int n) { return k < ((n + 1) >> 1) ? k : k - n; }
__device__ __forceinline__ int wrapi(int f, int n) { return f < 0 ? f + n : f; }

// angular factor of band b at signed frequency (fy, fx) of the full grid
__device__ __forceinline__ float ang_factor(const AngParams& A, int b, int fy, int fx) {
    const float xv = (float)fx * A.inv_hw, yv = (float)fy * A.inv_hh;
    const float r2 = xv * xv + yv * yv;
    float c = (r2 > 0.f) ? (xv * A.cs[b] + yv * A.sn[b]) * rsqrtf(r2) : A.cs[b];  // angle(DC) = atan2(0,0) = 0
    if (A.one_sided && !(c > 0.f)) return 0.f;
    float v = A.scale;
    for (int i = 0; i < A.order; ++i) v *= c;
    return v;
}

// atan2f for the phase epilogue: octant reduction + degree-7 minimax in t^2 (|error| < 4e-7 rad, measured against
// float64 over the whole circle in tests/test_pyramid_gpu.py); atan2(0, 0) = 0 like torch.angle; the sign follows
// the sign bit of y (so -0.0 gives -pi on the negative real axis, as atan2f does).
__device__ __forceinline__ float fast_atan2f(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    const float t = (mx > 0.f) ? __fdividef(mn, mx) : 0.f;
    const float s = t * t;
    float r = 3.866738916e-03f;
    r = fmaf(r, s, -2.002674765e-02f);
    r = fmaf(r, s, 4.891432155e-02f);
    r = fmaf(r, s, -8.009681718e-02f);
    r = fmaf(r, s, 1.086575908e-01f);
    r = fmaf(r, s, -1.425704493e-01f);
    r = fmaf(r, s, 1.999868117e-01f);
    r = fmaf(r, s, -3.333332310e-01f);
    r = fmaf(r * s, t, t);
    if (ay > ax) r = 1.57079632679489662f - r;
    if (x < 0.f) r = 3.14159265358979324f - r;
    return copysignf(r, y);
}

__device__ __forceinline__ const SetEntry& find_entry(const LaunchSet& S, int bx) {
    int i = 0;
    while (i + 1 < S.n && bx >= S.e[i + 1].start) ++i;
    return S.e[i];
}

struct PtrTable { const float* p[MAX_BANDS]; };
struct MutPtrTable { float* p[MAX_BANDS]; };

// ------------------------------------------------------------------------------------------------
// K1: row pass, forward, with input prologue.  in -> FFT along x -> T[n][b][y][kx]
//   mode 0: real input  p0[n][y][x]
//   mode 1: polar input phase = p0, amp = p1 at channel (n*nb + b)   (values_to_coeff, pyramid.py:103-108)
//   mode 2: complex interleaved tab.p[b][n][y][x][2] (band tensors [N,h,w,2])
// grid: (row tiles of all jobs, nb, N)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PYR_THREADS, PYR_MIN_CTAS) k_rows_fwd(const LevelJob* __restrict__ jobs, const LaunchSet S, PtrTable tab,
                                                             float2* __restrict__ regionB) {
    extern __shared__ float2 smem[];
    const SetEntry& E = find_entry(S, blockIdx.x);
    const LevelJob& J = jobs[E.job];
    const int mode = E.mode;
    const int nbB = (mode == 0) ? 1 : J.nb;
    const int b = blockIdx.y, n = blockIdx.z, N = gridDim.z;
    if (b >= nbB) return;
    const int h = J.h, w = J.w, rb = J.rb;
    const int y0 = (blockIdx.x - E.start) * rb;
    const int rows = min(rb, h - y0);
    const int pitch = fft_pitch(J.fx);
    const FftIO iox = fft_io(J.fx);
    float2* a = smem;
    float2* bq = smem + (size_t)rb * pitch;
    const unsigned mag_w = J.mag_w;
    const size_t plane = (size_t)h * w;
    constexpr int U = 8;                      // independent global loads in flight per thread
    const int total = rows * w;
    for (int q0 = threadIdx.x; q0 < total; q0 += U * blockDim.x) {
        float2 z[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int q = q0 + u * blockDim.x;
            z[u] = make_float2(0.f, 0.f);
            if (q < total) {
                const size_t pix = (size_t)y0 * w + q;
                if (mode == 0) {
                    z[u].x = __ldg(E.p0 + (size_t)n * plane + pix);
                } else if (mode == 1) {
                    const size_t o = ((size_t)n * nbB + b) * plane + pix;
                    z[u] = make_float2(__ldg(E.p0 + o), __ldg(E.p1 + o));      // (phase, amplitude)
                } else {
                    z[u] = __ldg((const float2*)tab.p[b] + (size_t)n * plane + pix);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int q = q0 + u * blockDim.x;
            if (q < total) {
                const int r = (int)fast_div((unsigned)q, (unsigned)w, mag_w), x = q - r * w;
                float2 v = z[u];
                if (mode == 1) {
                    float sn, cs;
                    sincosf(z[u].x, &sn, &cs);
                    v = make_float2(cs * z[u].y, sn * z[u].y);  // pyramid.py:105-106
                }
                fft_put<false>(iox, a, r, x, v, 0, pitch);
            }
        }
    }
    __syncthreads();
    const FftResult R = fft_forward<false>(J.fx, a, bq, rows, 0, pitch, false, FftCtx{(int)threadIdx.x, (int)blockDim.x});
    float2* dst = regionB + (size_t)N * J.t_off + ((size_t)n * nbB + b) * plane + (size_t)y0 * w;
    for (int q = threadIdx.x; q < rows * w; q += blockDim.x) {
        const int r = (int)fast_div((unsigned)q, (unsigned)w, mag_w), x = q - r * w;
        dst[q] = fft_get<false>(iox, R, r, x, 0, pitch);
    }
}

// ------------------------------------------------------------------------------------------------
// K2: column pass, forward.  T[n][b][:, tile] -> FFT along y ->
//   entry mode 1 (combine, reconstruction of a band level): out = radial * sum_b fft_b * ang_b * (i)^(nb-1)
//   entry mode 0 (plain): out = fft * radial   (use_radial == 0: radial ignored -> image spectrum X)
// out = outbase + n*out_stride (+ J.c_off if add_c_off).   grid: (column tiles of all jobs, 1, N)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PYR_THREADS, PYR_MIN_CTAS) k_cols_fwd(const LevelJob* __restrict__ jobs, const LaunchSet S, AngParams A,
                                                             const float2* __restrict__ regionB, float2* __restrict__ outbase,
                                                             size_t out_stride, int add_c_off, int use_radial,
                                                             const float* __restrict__ radial_override) {
    extern __shared__ float2 smem[];
    const SetEntry& E = find_entry(S, blockIdx.x);
    const LevelJob& J = jobs[E.job];
    const bool combine = E.mode == 1;
    const int nbB = combine ? J.nb : 1;
    const int n = blockIdx.z, N = gridDim.z;
    const int h = J.h, w = J.w, cs = combine ? J.ct_shift_c : J.ct_shift, CT = 1 << cs;
    const int x0 = (blockIdx.x - E.start) << cs;
    const int cols = min(CT, w - x0);
    const int E_ = h << cs;
    const FftIO ioy = fft_io(J.fy);
    float2* a = smem;
    float2* acc = smem + ((size_t)J.fy.M << cs);
    const size_t plane = (size_t)h * w;
    const FftCtx cx{(int)threadIdx.x, (int)blockDim.x};
    FftResult R{a, nullptr};
    for (int b = 0; b < nbB; ++b) {
        const float2* src = regionB + (size_t)N * J.t_off + ((size_t)n * nbB + b) * plane;
        {
            constexpr int U = 8;
            for (int q0 = threadIdx.x; q0 < E_; q0 += U * blockDim.x) {
                float2 z[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int q = q0 + u * blockDim.x;
                    const int y = q >> cs, c = q & (CT - 1);
                    z[u] = make_float2(0.f, 0.f);
                    if (q < E_ && c < cols) z[u] = __ldcs(src + (size_t)y * w + x0 + c);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int q = q0 + u * blockDim.x;
                    if (q < E_) fft_put<true>(ioy, a, q & (CT - 1), q >> cs, z[u], cs, 0);
                }
            }
        }
        __syncthreads();
        R = fft_forward<true>(J.fy, a, nullptr, CT, cs, 0, true, cx);
        if (combine) {
            for (int q = threadIdx.x; q < E_; q += blockDim.x) {
                const int pos = q >> cs, c = q & (CT - 1);
                const int ky = R.perm ? (int)__ldg(R.perm + pos) : pos;
                const float g = __ldg(J.band_rec + ((size_t)b * h + ky) * w + min(x0 + c, w - 1));   // D_l * two-sided angular mask
                const float2 rv = fft_get<true>(ioy, R, c, pos, cs, 0);
                const float2 v = cmul(make_float2(rv.x * g, rv.y * g), A.fac);
                acc[q] = (b == 0) ? v : cadd(acc[q], v);
            }
            __syncthreads();
        }
    }
    const float* radial = (use_radial && !combine) ? (radial_override ? radial_override : J.radial) : nullptr;   // combine: part of band_rec
    float2* dst = outbase + (size_t)n * out_stride + (add_c_off ? (size_t)J.c_off : 0);
    for (int q = threadIdx.x; q < E_; q += blockDim.x) {
        const int pos = q >> cs, c = q & (CT - 1);
        if (c >= cols) continue;
        const int ky = R.perm ? (int)__ldg(R.perm + pos) : pos;
        const size_t o = (size_t)ky * w + x0 + c;
        const float m = radial ? __ldg(radial + o) : 1.f;
        const float2 rv = combine ? acc[q] : fft_get<true>(ioy, R, c, pos, cs, 0);
        dst[o] = make_float2(rv.x * m, rv.y * m);
    }
}

// ------------------------------------------------------------------------------------------------
// K3: column pass of the band IFFT with the spectrum loader (decomposition).
//   value = conj( X[n][fy mod H][fx mod W] * radial[ky][kx] * ang_b * (-i)^(nb-1) ); forward FFT along y; the row pass
//   conjugates again at the very end (IFFT2 = conj FFT2 conj).   out: T[n][b][y][kx]
// grid: (column tiles of all jobs, nb, N)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PYR_THREADS, PYR_MIN_CTAS) k_cols_inv_decomp(const LevelJob* __restrict__ jobs, const LaunchSet S,
                                                                    float2 band_fac, int use_rec_table, int H, int W,
                                                                    const float2* __restrict__ X, float2* __restrict__ regionB) {
    extern __shared__ float2 smem[];
    const SetEntry& E = find_entry(S, blockIdx.x);
    const LevelJob& J = jobs[E.job];
    const int b = blockIdx.y, n = blockIdx.z, N = gridDim.z;
    if (b >= J.nb) return;
    const int h = J.h, w = J.w, cs = J.ct_shift, CT = 1 << cs;
    const int x0 = (blockIdx.x - E.start) << cs;
    const int cols = min(CT, w - x0);
    const int E_ = h << cs;
    const FftIO ioy = fft_io(J.fy);
    const bool band = J.is_band != 0;
    float2* a = smem;
    const float2* Xn = X + (size_t)n * H * W;
    // band levels: the combined radial x angular mask of band b (plan table, equal to the oracle's masks); else the radial mask
    const float* radial = band ? (use_rec_table ? J.band_rec : J.band_build) + (size_t)b * h * w : J.radial;
    {
        constexpr int U = 8;                  // two dependent global loads per element: batch them
        for (int q0 = threadIdx.x; q0 < E_; q0 += U * blockDim.x) {
            float m[U];
            float2 xv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + u * blockDim.x;
                const int ky = q >> cs, c = q & (CT - 1);
                m[u] = (q < E_ && c < cols) ? __ldg(radial + (size_t)ky * w + x0 + c) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + u * blockDim.x;
                const int ky = q >> cs, c = q & (CT - 1);
                const int fy = sfreq(ky, h), fx = sfreq(x0 + c, w);
                xv[u] = make_float2(0.f, 0.f);
                if (m[u] != 0.f) xv[u] = __ldg(Xn + (size_t)wrapi(fy, H) * W + wrapi(fx, W));
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + u * blockDim.x;
                if (q < E_) {
                    float2 v = make_float2(xv[u].x * m[u], xv[u].y * m[u]);
                    if (band) v = cmul(v, band_fac);
                    v.y = -v.y;
                    fft_put<true>(ioy, a, q & (CT - 1), q >> cs, v, cs, 0);
                }
            }
        }
    }
    __syncthreads();
    const FftResult R = fft_forward<true>(J.fy, a, nullptr, CT, cs, 0, true, FftCtx{(int)threadIdx.x, (int)blockDim.x});
    float2* dst = regionB + (size_t)N * J.t_off + ((size_t)n * J.nb + b) * h * w;
    for (int q = threadIdx.x; q < E_; q += blockDim.x) {
        const int pos = q >> cs, c = q & (CT - 1);
        if (c >= cols) continue;
        const int y = R.perm ? (int)__ldg(R.perm + pos) : pos;
        dst[(size_t)y * w + x0 + c] = fft_get<true>(ioy, R, c, pos, cs, 0);
    }
}

// ------------------------------------------------------------------------------------------------
// K4: column pass of the final IFFT of the reconstruction: value = conj( sum over levels of
//   Y_l[n][fy mod h_l][fx mod w_l] (+ high spectrum) ); out: T of the full-size job.   grid: (column tiles, 1, N)
// ------------------------------------------------------------------------------------------------
struct GatherArgs {
    int nlev;                     // number of level spectra (band levels + low)
    LevelGeom lv[MAX_LEVELS];
    unsigned long long active;    // bit l set = level l contributes
    const float2* Y;              // region C base
    size_t plane_stride;          // complex elements per plane in region C
    const float2* Yhigh;          // [N][H][W] or null
};

__global__ void __launch_bounds__(PYR_THREADS, PYR_MIN_CTAS) k_cols_inv_gather(const LevelJob* __restrict__ jobs, int job, const GatherArgs G,
                                                                    float inv_hh, float inv_hw, float2* __restrict__ regionB) {
    extern __shared__ float2 smem[];
    const LevelJob& J = jobs[job];
    const int H = J.h, W = J.w, cs = J.ct_shift, CT = 1 << cs;
    const int x0 = blockIdx.x << cs, n = blockIdx.z, N = gridDim.z;
    const int cols = min(CT, W - x0);
    const int E_ = H << cs;
    const FftIO ioy = fft_io(J.fy);
    float2* a = smem;
    for (int q = threadIdx.x; q < E_; q += blockDim.x) {
        const int ky = q >> cs, c = q & (CT - 1);
        float2 v = make_float2(0.f, 0.f);
        if (c < cols) {
            const int kx = x0 + c;
            const int fy = sfreq(ky, H), fx = sfreq(kx, W);
            const float xv = (float)fx * inv_hw, yv = (float)fy * inv_hh;
            const float r2 = xv * xv + yv * yv;
            if (G.Yhigh) v = G.Yhigh[((size_t)n * H + ky) * W + kx];
            for (int l = 0; l < G.nlev; ++l) {
                const LevelGeom& g = G.lv[l];
                // nested centred windows: once outside, outside of all coarser levels too
                if (fy < -(g.h >> 1) || fy > g.h - 1 - (g.h >> 1) || fx < -(g.w >> 1) || fx > g.w - 1 - (g.w >> 1)) break;
                if (!((G.active >> l) & 1ull)) continue;
                const bool dc = (fy == 0 && fx == 0);
                if (!dc && (r2 <= g.rad2_lo || r2 >= g.rad2_hi)) continue;
                const float2 y = G.Y[(size_t)n * G.plane_stride + g.off + (size_t)wrapi(fy, g.h) * g.w + wrapi(fx, g.w)];
                v = cadd(v, y);
            }
            v.y = -v.y;
        }
        fft_put<true>(ioy, a, c, ky, v, cs, 0);
    }
    __syncthreads();
    const FftResult R = fft_forward<true>(J.fy, a, nullptr, CT, cs, 0, true, FftCtx{(int)threadIdx.x, (int)blockDim.x});
    float2* dst = regionB + (size_t)N * J.t_off + (size_t)n * H * W;
    for (int q = threadIdx.x; q < E_; q += blockDim.x) {
        const int pos = q >> cs, c = q & (CT - 1);
        if (c >= cols) continue;
        const int y = R.perm ? (int)__ldg(R.perm + pos) : pos;
        dst[(size_t)y * W + x0 + c] = fft_get<true>(ioy, R, c, pos, cs, 0);
    }
}

// ------------------------------------------------------------------------------------------------
// K5: row pass of an IFFT with output epilogue.  T[n][b][y][:] -> forward FFT along x -> conj, scale 1/(h*w) ->
//   mode 0: real part -> q0[n][y][x]
//   mode 1: polar: phase -> q0, amplitude -> q1 at channel n*nb + b; per-plane max amplitude -> aux[n]
//           (pyramid.py:63-69, phase_net.py:47-59)
//   mode 2: complex interleaved -> tab.p[b][n][y][x][2]
//   mode 3: backward of the reconstruction: z is dL/d(band); with phase = p0, amplitude = p1 -> dL/dphase -> q0, dL/damp -> q1
// grid: (row tiles of all jobs, nb, N)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PYR_THREADS, PYR_MIN_CTAS) k_rows_inv(const LevelJob* __restrict__ jobs, const LaunchSet S, MutPtrTable tab,
                                                             const float2* __restrict__ regionB) {
    extern __shared__ float2 smem[];
    const SetEntry& E = find_entry(S, blockIdx.x);
    const LevelJob& J = jobs[E.job];
    const int mode = E.mode;
    const int nbB = (mode == 0) ? 1 : J.nb;
    const int b = blockIdx.y, n = blockIdx.z, N = gridDim.z;
    if (b >= nbB) return;
    const int h = J.h, w = J.w, rb = J.rb;
    const int y0 = (blockIdx.x - E.start) * rb;
    const int rows = min(rb, h - y0);
    const int pitch = fft_pitch(J.fx);
    const FftIO iox = fft_io(J.fx);
    float2* a = smem;
    float2* bq = smem + (size_t)rb * pitch;
    const unsigned mag_w = J.mag_w;
    const size_t plane = (size_t)h * w;
    const float2* src = regionB + (size_t)N * J.t_off + ((size_t)n * nbB + b) * plane + (size_t)y0 * w;
    // Rows of the intermediate are contiguous in HBM: when they are 16-byte aligned (even width) and need no transformation on the
    // way in (no Bluestein chirp), one elected thread lands every row at its pitch with cp.async.bulk (bulk async-copy engine,
    // completion on an mbarrier) -- no per-element load / address / store instructions, no registers in flight.
    const bool bulk = !iox.bluestein && !iox.pos_in && !(w & 1) && ((((size_t)src) & 15) == 0) && J.fx.nfac > 0;
    const int src_plain = (bulk && J.fx.pad) ? 1 : 0;     // landed unskewed: the first (out-of-place) stage reads plainly
    if (bulk) {
        unsigned long long* bar = (unsigned long long*)(smem + (size_t)2 * rb * pitch);     // bulk rows are two-buffer plans (row_smem)
        const unsigned bar_s = (unsigned)__cvta_generic_to_shared(bar);
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_s));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned row_bytes = (unsigned)w * (unsigned)sizeof(float2);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_s), "r"(row_bytes * (unsigned)rows) : "memory");
            for (int r = 0; r < rows; ++r)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             ::"r"((unsigned)__cvta_generic_to_shared(a + (size_t)r * pitch)), "l"(src + (size_t)r * w), "r"(row_bytes), "r"(bar_s)
                             : "memory");
        }
        unsigned done = 0, spins = 0;
        while (!done) {
            asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                         : "=r"(done) : "r"(bar_s) : "memory");
            if (++spins > 200000000u) __trap();       // bounded wait: a protocol bug traps instead of hanging the GPU
        }
    } else {
        constexpr int U = 8;                  // independent global loads in flight per thread
        const int total = rows * w;
        for (int q0 = threadIdx.x; q0 < total; q0 += U * blockDim.x) {
            float2 z[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + u * blockDim.x;
                if (q < total) z[u] = __ldcs(src + q);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int q = q0 + u * blockDim.x;
                if (q < total) {
                    const int r = (int)fast_div((unsigned)q, (unsigned)w, mag_w), x = q - r * w;
                    fft_put<false>(iox, a, r, x, z[u], 0, pitch);
                }
            }
        }
    }
    __syncthreads();
    const FftResult R = fft_forward<false>(J.fx, a, bq, rows, 0, pitch, false, FftCtx{(int)threadIdx.x, (int)blockDim.x}, src_plain);
    const float scale = E.scale > 0.f ? E.scale : 1.f / ((float)h * (float)w);
    float mx = 0.f;
    for (int q = threadIdx.x; q < rows * w; q += blockDim.x) {
        const int r = (int)fast_div((unsigned)q, (unsigned)w, mag_w), x = q - r * w;
        const float2 t = fft_get<false>(iox, R, r, x, 0, pitch);
        const float2 z = make_float2(t.x * scale, -t.y * scale);
        const size_t pix = (size_t)y0 * w + q;
        if (mode == 0) {
            E.q0[(size_t)n * plane + pix] = z.x;
        } else if (mode == 1) {
            const size_t o = ((size_t)n * nbB + b) * plane + pix;
            const float ss = fmaf(z.x, z.x, z.y * z.y);
            const float am = ss > 0.f ? ss * rsqrtf(ss) : 0.f;   // torch.abs (pyramid.py:67); rsqrt form: 2 ulp, 3 instructions
            E.q0[o] = fast_atan2f(z.y, z.x);                     // imag(log z)          (pyramid.py:63)
            E.q1[o] = am;
            mx = fmaxf(mx, am);
        } else if (mode == 3) {
            // adjoint of values_to_coeff (pyramid.py:103-108): z = A (cos phi, sin phi), z_bar = dL/d(re, im)
            const size_t o = ((size_t)n * nbB + b) * plane + pix;
            float sn, cs;
            sincosf(__ldg(E.p0 + o), &sn, &cs);
            E.q0[o] = __ldg(E.p1 + o) * (z.y * cs - z.x * sn);     // dL/dphi
            E.q1[o] = z.x * cs + z.y * sn;                         // dL/dA
        } else {
            ((float2*)tab.p[b])[(size_t)n * plane + pix] = z;
        }
    }
    if (mode == 1 && E.aux) {
        for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if ((threadIdx.x & 31) == 0) atomicMax((int*)(E.aux + n), __float_as_int(mx));  // amplitudes are >= 0
    }
}

// ------------------------------------------------------------------------------------------------
// host: launch helpers
// ------------------------------------------------------------------------------------------------
template <typename K>
static int ensure_smem(K kernel, size_t bytes) {
    if (bytes > 227 * 1024) { set_error("pyramid: tile needs %zu B of shared memory (> 227 KB)", bytes); return FVFI_EINVAL; }
    FVFI_SMEM_OPT_IN(kernel, std::max<size_t>(bytes, 48 * 1024));
    return FVFI_OK;
}

static size_t row_smem(const LevelJob& J) { return (size_t)J.rb * row_bytes_per_row(J.fx) + 16; }   // + the mbarrier of the bulk row loads
static size_t col_smem(const LevelJob& J, bool combine) {
    return combine ? ((((size_t)J.fy.M + J.h) << J.ct_shift_c) * sizeof(float2)) : (((size_t)J.fy.M << J.ct_shift) * sizeof(float2));
}

struct SetBuilder {
    const fvfi_pyr_plan* p;
    LaunchSet rows{}, cols{};
    size_t rows_smem = 0, cols_smem = 0;
    int max_nb = 1;
    bool has_combine = false;
    explicit SetBuilder(const fvfi_pyr_plan* plan) : p(plan) {}
    bool full() const { return rows.n >= MAX_SET; }
    bool empty() const { return rows.n == 0; }
    void add(int job, int mode, const float* p0, const float* p1, float* q0, float* q1, float* aux, bool combine_cols,
             float scale = 0.f) {
        const LevelJob& J = p->jobs[job];
        SetEntry e{};
        e.scale = scale;
        e.job = job; e.mode = mode; e.p0 = p0; e.p1 = p1; e.q0 = q0; e.q1 = q1; e.aux = aux;
        e.start = rows.total;
        rows.e[rows.n++] = e;
        rows.total += J.row_tiles;
        e.start = cols.total;
        e.mode = combine_cols ? 1 : 0;
        cols.e[cols.n++] = e;
        cols.total += combine_cols ? J.col_tiles_c : J.col_tiles;
        rows_smem = std::max(rows_smem, row_smem(J));
        cols_smem = std::max(cols_smem, col_smem(J, combine_cols));
        if (mode != 0) max_nb = std::max(max_nb, J.nb);
        has_combine |= combine_cols;
    }
};

static int launch_rows_fwd(const fvfi_pyr_plan* p, const SetBuilder& sb, const PtrTable& tab, int N, float2* regionB, cudaStream_t s) {
    if (int rc = ensure_smem(k_rows_fwd, sb.rows_smem)) return rc;
    dim3 grid(sb.rows.total, sb.max_nb, N);
    k_rows_fwd<<<grid, PYR_THREADS, sb.rows_smem, s>>>(p->d_jobs, sb.rows, tab, regionB);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

static int launch_cols_fwd(const fvfi_pyr_plan* p, const SetBuilder& sb, int N, const float2* regionB, float2* out, size_t stride,
                           int add_c_off, int use_radial, cudaStream_t s, const float* radial_override = nullptr) {
    if (int rc = ensure_smem(k_cols_fwd, sb.cols_smem)) return rc;
    dim3 grid(sb.cols.total, 1, N);
    k_cols_fwd<<<grid, PYR_THREADS, sb.cols_smem, s>>>(p->d_jobs, sb.cols, p->ang_rec, regionB, out, stride, add_c_off, use_radial,
                                                       radial_override);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

static int launch_cols_inv_decomp(const fvfi_pyr_plan* p, const SetBuilder& sb, int N, const float2* X, float2* regionB, cudaStream_t s,
                                  const AngParams* ang = nullptr) {
    if (int rc = ensure_smem(k_cols_inv_decomp, sb.cols_smem)) return rc;
    int nbmax = 1;
    for (int i = 0; i < sb.cols.n; ++i) nbmax = std::max(nbmax, p->jobs[sb.cols.e[i].job].nb);
    dim3 grid(sb.cols.total, nbmax, N);
    k_cols_inv_decomp<<<grid, PYR_THREADS, sb.cols_smem, s>>>(p->d_jobs, sb.cols, ang ? ang->fac : p->ang_build.fac, ang ? 1 : 0, p->H, p->W,
                                                              X, regionB);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

static int launch_rows_inv(const fvfi_pyr_plan* p, const SetBuilder& sb, const MutPtrTable& tab, int N, const float2* regionB, cudaStream_t s) {
    if (int rc = ensure_smem(k_rows_inv, sb.rows_smem)) return rc;
    dim3 grid(sb.rows.total, sb.max_nb, N);
    k_rows_inv<<<grid, PYR_THREADS, sb.rows_smem, s>>>(p->d_jobs, sb.rows, tab, regionB);
    FVFI_LAUNCH_CHECK();
    return FVFI_OK;
}

struct Workspace {
    float2 *A, *B, *C;  // A: N*H*W (X / high spectrum) ; B: N*(nb*level_elems + H*W) (intermediates) ; C: N*level_elems
};

static size_t ws_elems(const fvfi_pyr_plan* p, int N) {
    const size_t HW = (size_t)p->H * p->W;
    return (size_t)N * (HW + ((size_t)p->nbands * p->level_elems + HW) + p->level_elems) + 64;
}

static Workspace carve(const fvfi_pyr_plan* p, int N, void* ws) {
    const size_t HW = (size_t)p->H * p->W;
    Workspace w;
    uintptr_t base = ((uintptr_t)ws + 255) & ~(uintptr_t)255;
    w.A = (float2*)base;
    w.B = w.A + (size_t)N * HW;
    w.C = w.B + (size_t)N * ((size_t)p->nbands * p->level_elems + HW);
    return w;
}

static bool is_small(const LevelJob& J) { return (long long)J.h * J.w <= SMALL_LEVEL_ELEMS; }

// decomposition shared by the polar and complex front ends
static int decompose(const fvfi_pyr_plan* p, const float* img, int N, float* high, float* const* phase,
                     float* const* amp, float* const* bands, float* low, float* amp_max, void* workspace,
                     cudaStream_t s) {
    const int H = p->H, W = p->W, L = p->L, nb = p->nbands;
    const int FULL = L + 1;
    Workspace ws = carve(p, N, workspace);
    PtrTable none{};
    MutPtrTable mnone{};
    // X = FFT2(img): rows (into the full-size intermediate) then columns (into region A)
    {
        SetBuilder sb(p);
        sb.add(FULL, 0, img, nullptr, nullptr, nullptr, nullptr, false);
        if (int rc = launch_rows_fwd(p, sb, none, N, ws.B, s)) return rc;
        if (int rc = launch_cols_fwd(p, sb, N, ws.B, ws.A, (size_t)H * W, 0, 0, s)) return rc;
    }
    if (amp_max) FVFI_CUDA(cudaMemsetAsync(amp_max, 0, (size_t)L * N * sizeof(float), s));
    // every output component is an independent job: big ones get their own launch pair, small ones share one
    SetBuilder small(p);
    auto flush = [&](SetBuilder& sb, const MutPtrTable& tab) -> int {
        if (sb.empty()) return FVFI_OK;
        if (int rc = launch_cols_inv_decomp(p, sb, N, ws.A, ws.B, s)) return rc;
        if (int rc = launch_rows_inv(p, sb, tab, N, ws.B, s)) return rc;
        sb = SetBuilder(p);
        return FVFI_OK;
    };
    auto submit = [&](int job, int mode, float* q0, float* q1, float* aux) -> int {
        if (is_small(p->jobs[job])) {
            small.add(job, mode, nullptr, nullptr, q0, q1, aux, false);
            if (small.full()) return flush(small, mnone);
            return FVFI_OK;
        }
        SetBuilder one(p);
        one.add(job, mode, nullptr, nullptr, q0, q1, aux, false);
        return flush(one, mnone);
    };
    if (high)
        if (int rc = submit(FULL, 0, high, nullptr, nullptr)) return rc;
    for (int l = 0; l < L; ++l) {
        if (phase ? (phase[l] == nullptr) : (bands[l * nb] == nullptr)) continue;
        if (phase) {
            if (int rc = submit(l, 1, phase[l], amp[l], amp_max ? amp_max + (size_t)l * N : nullptr)) return rc;
        } else {
            MutPtrTable t{};
            for (int b = 0; b < nb; ++b) t.p[b] = bands[l * nb + b];
            SetBuilder one(p);
            one.add(l, 2, nullptr, nullptr, nullptr, nullptr, nullptr, false);
            if (int rc = flush(one, t)) return rc;
        }
    }
    if (low)
        if (int rc = submit(L, 0, low, nullptr, nullptr)) return rc;
    return flush(small, mnone);
}

static int reconstruct(const fvfi_pyr_plan* p, const float* high, const float* const* phase, const float* const* amp,
                       const float* const* bands, const float* low, int N, float* img, void* workspace,
                       cudaStream_t s) {
    const int H = p->H, W = p->W, L = p->L, nb = p->nbands;
    const int FULL = L + 1;
    Workspace ws = carve(p, N, workspace);
    PtrTable none{};
    MutPtrTable mnone{};
    GatherArgs G{};
    G.nlev = L + 1;
    G.Y = ws.C;
    G.plane_stride = p->level_elems;
    G.active = 0;
    for (int l = 0; l <= L; ++l) G.lv[l] = p->lv[l];
    SetBuilder small(p);
    auto flush = [&](SetBuilder& sb, const PtrTable& tab) -> int {
        if (sb.empty()) return FVFI_OK;
        if (int rc = launch_rows_fwd(p, sb, tab, N, ws.B, s)) return rc;
        if (int rc = launch_cols_fwd(p, sb, N, ws.B, ws.C, p->level_elems, 1, 1, s)) return rc;
        sb = SetBuilder(p);
        return FVFI_OK;
    };
    for (int l = 0; l < L; ++l) {
        const bool have = phase ? (phase[l] != nullptr && amp[l] != nullptr) : (bands[l * nb] != nullptr);
        if (!have) continue;
        G.active |= 1ull << l;
        if (phase) {
            if (is_small(p->jobs[l])) {
                small.add(l, 1, phase[l], amp[l], nullptr, nullptr, nullptr, true);
                if (small.full())
                    if (int rc = flush(small, none)) return rc;
            } else {
                SetBuilder one(p);
                one.add(l, 1, phase[l], amp[l], nullptr, nullptr, nullptr, true);
                if (int rc = flush(one, none)) return rc;
            }
        } else {
            PtrTable t{};
            for (int b = 0; b < nb; ++b) t.p[b] = bands[l * nb + b];
            SetBuilder one(p);
            one.add(l, 2, nullptr, nullptr, nullptr, nullptr, nullptr, true);
            if (int rc = flush(one, t)) return rc;
        }
    }
    if (low) {
        small.add(L, 0, low, nullptr, nullptr, nullptr, nullptr, false);
        G.active |= 1ull << L;
    }
    if (int rc = flush(small, none)) return rc;
    if (high) {
        SetBuilder one(p);
        one.add(FULL, 0, high, nullptr, nullptr, nullptr, nullptr, false);
        if (int rc = launch_rows_fwd(p, one, none, N, ws.B, s)) return rc;
        if (int rc = launch_cols_fwd(p, one, N, ws.B, ws.A, (size_t)H * W, 0, 1, s)) return rc;
        G.Yhigh = ws.A;
    }
    // gather all level spectra + inverse FFT2
    {
        const LevelJob& J = p->jobs[FULL];
        const size_t smem = col_smem(J, false);
        if (int rc = ensure_smem(k_cols_inv_gather, smem)) return rc;
        dim3 grid(J.col_tiles, 1, N);
        k_cols_inv_gather<<<grid, PYR_THREADS, smem, s>>>(p->d_jobs, FULL, G, p->ang_rec.inv_hh, p->ang_rec.inv_hw, ws.B);
        FVFI_LAUNCH_CHECK();
    }
    SetBuilder fin(p);
    fin.add(FULL, 0, nullptr, nullptr, img, nullptr, nullptr, false);
    return launch_rows_inv(p, fin, mnone, N, ws.B, s);
}

// reconstruct(high + finest level of decompose(img)) as ONE spectral multiplication (plan table hf_transfer): 2 FFT2 instead of 10.
static int highband_filter(const fvfi_pyr_plan* p, const float* img, int N, float* out, void* workspace, cudaStream_t s) {
    const int H = p->H, W = p->W, FULL = p->L + 1;
    Workspace ws = carve(p, N, workspace);
    PtrTable none{};
    MutPtrTable mnone{};
    SetBuilder sb(p);
    sb.add(FULL, 0, img, nullptr, nullptr, nullptr, nullptr, false);
    if (int rc = launch_rows_fwd(p, sb, none, N, ws.B, s)) return rc;
    if (int rc = launch_cols_fwd(p, sb, N, ws.B, ws.A, (size_t)H * W, 0, 1, s, p->hf_transfer)) return rc;
    GatherArgs G{};
    G.nlev = 0;
    G.active = 0;
    G.Y = ws.C;
    G.plane_stride = p->level_elems;
    G.Yhigh = ws.A;
    const LevelJob& J = p->jobs[FULL];
    const size_t smem = col_smem(J, false);
    if (int rc = ensure_smem(k_cols_inv_gather, smem)) return rc;
    dim3 grid(J.col_tiles, 1, N);
    k_cols_inv_gather<<<grid, PYR_THREADS, smem, s>>>(p->d_jobs, FULL, G, p->ang_rec.inv_hh, p->ang_rec.inv_hw, ws.B);
    FVFI_LAUNCH_CHECK();
    SetBuilder fin(p);
    fin.add(FULL, 0, nullptr, nullptr, out, nullptr, nullptr, false);
    return launch_rows_inv(p, fin, mnone, N, ws.B, s);
}

// Backward of reconstruct(): img = Re M(high, bands, low) is real-linear in the complex bands, so dL/d(band) = M^H dL/d(img):
//   FFT2 of the image gradient, then per level the SAME crop / radial mask as the forward, the conjugated two-sided angular
//   factor, an unnormalised IFFT2 at the level size and 1/(H*W) -- i.e. the decomposition machinery with the reconstruction's
//   masks.  The row-pass epilogue chains through z = A e^{i phi} (mode 3) or takes the real part (high / low).
static int reconstruct_backward(const fvfi_pyr_plan* p, const float* gimg, int N, const float* const* phase,
                                const float* const* amp, float* ghigh, float* const* gphase, float* const* gamp, float* glow,
                                void* workspace, cudaStream_t s) {
    const int H = p->H, W = p->W, L = p->L;
    const int FULL = L + 1;
    Workspace ws = carve(p, N, workspace);
    PtrTable none{};
    MutPtrTable mnone{};
    {
        SetBuilder sb(p);
        sb.add(FULL, 0, gimg, nullptr, nullptr, nullptr, nullptr, false);
        if (int rc = launch_rows_fwd(p, sb, none, N, ws.B, s)) return rc;
        if (int rc = launch_cols_fwd(p, sb, N, ws.B, ws.A, (size_t)H * W, 0, 0, s)) return rc;
    }
    AngParams adj = p->ang_rec;
    adj.fac.y = -adj.fac.y;                      // conj((i)^(nb-1))
    const float scale = 1.f / ((float)H * (float)W);
    SetBuilder small(p);
    auto flush = [&](SetBuilder& sb) -> int {
        if (sb.empty()) return FVFI_OK;
        if (int rc = launch_cols_inv_decomp(p, sb, N, ws.A, ws.B, s, &adj)) return rc;
        if (int rc = launch_rows_inv(p, sb, mnone, N, ws.B, s)) return rc;
        sb = SetBuilder(p);
        return FVFI_OK;
    };
    auto submit = [&](int job, int mode, const float* p0, const float* p1, float* q0, float* q1) -> int {
        if (is_small(p->jobs[job])) {
            small.add(job, mode, p0, p1, q0, q1, nullptr, false, scale);
            if (small.full()) return flush(small);
            return FVFI_OK;
        }
        SetBuilder one(p);
        one.add(job, mode, p0, p1, q0, q1, nullptr, false, scale);
        return flush(one);
    };
    if (ghigh)
        if (int rc = submit(FULL, 0, nullptr, nullptr, ghigh, nullptr)) return rc;
    for (int l = 0; l < L; ++l) {
        if (!gphase[l] || !gamp[l]) continue;
        if (!phase[l] || !amp[l]) { set_error("pyr_reconstruct_backward: level %d gradient requested without its values", l); return FVFI_EINVAL; }
        if (int rc = submit(l, 3, phase[l], amp[l], gphase[l], gamp[l])) return rc;
    }
    if (glow)
        if (int rc = submit(L, 0, nullptr, nullptr, glow, nullptr)) return rc;
    return flush(small);
}

}  // namespace fvfi

using namespace fvfi;

extern "C" {

int fvfi_pyr_next_size(int n, double s) { return fvfi::next_size(n, s); }

int fvfi_pyr_plan_create(int H, int W, int height, int nbands, double scale_factor, fvfi_pyr_plan** out) {
    FVFI_CHECK_ARG(out, "pyr_plan_create: null out");
    *out = nullptr;
    FVFI_CHECK_ARG(H >= 4 && W >= 4 && H <= 8192 && W <= 8192, "pyr_plan_create: unsupported image size %dx%d", H, W);
    FVFI_CHECK_ARG(height >= 2 && height - 2 < MAX_LEVELS - 1, "pyr_plan_create: bad height %d", height);
    FVFI_CHECK_ARG(nbands >= 1 && nbands <= MAX_BANDS, "pyr_plan_create: nbands must be 1..%d", MAX_BANDS);
    FVFI_CHECK_ARG(scale_factor > 1.0 && scale_factor <= 4.0, "pyr_plan_create: scale_factor must be in (1,4]");
    fvfi_pyr_plan* p = new fvfi_pyr_plan();
    p->H = H; p->W = W; p->height = height; p->nbands = nbands; p->L = height - 2; p->scale = scale_factor;
    if (int rc = build_plan(p)) { fvfi_pyr_plan_destroy(p); return rc; }
    *out = p;
    return FVFI_OK;
}

void fvfi_pyr_plan_destroy(fvfi_pyr_plan* p) {
    if (!p) return;
    for (void* d : p->owned) cudaFree(d);
    delete p;
}

int fvfi_pyr_num_levels(const fvfi_pyr_plan* p) { return p ? p->L : -1; }

int fvfi_pyr_level_shape(const fvfi_pyr_plan* p, int level, int* h, int* w) {
    FVFI_CHECK_ARG(p && level >= 0 && level <= p->L, "pyr_level_shape: bad level");
    if (h) *h = p->lv[level].h;
    if (w) *w = p->lv[level].w;
    return FVFI_OK;
}

size_t fvfi_pyr_workspace_bytes(const fvfi_pyr_plan* p, int N) {
    if (!p || N <= 0) return 0;
    return ws_elems(p, N) * sizeof(float2) + 256;
}

int fvfi_pyr_decompose(const fvfi_pyr_plan* p, const float* img, int N, float* high, float* const* phase,
                       float* const* amp, float* low, float* amp_max, void* workspace, void* stream) {
    FVFI_CHECK_ARG(p && img && phase && amp && workspace && N > 0 && N <= 65535, "pyr_decompose: bad argument");
    return decompose(p, img, N, high, phase, amp, nullptr, low, amp_max, workspace, (cudaStream_t)stream);
}

int fvfi_pyr_build_complex(const fvfi_pyr_plan* p, const float* img, int N, float* high, float* const* bands,
                           float* low, void* workspace, void* stream) {
    FVFI_CHECK_ARG(p && img && bands && workspace && N > 0 && N <= 65535, "pyr_build_complex: bad argument");
    return decompose(p, img, N, high, nullptr, nullptr, bands, low, nullptr, workspace, (cudaStream_t)stream);
}

int fvfi_pyr_reconstruct(const fvfi_pyr_plan* p, const float* high, const float* const* phase,
                         const float* const* amp, const float* low, int N, float* img, void* workspace,
                         void* stream) {
    FVFI_CHECK_ARG(p && phase && amp && img && workspace && N > 0 && N <= 65535, "pyr_reconstruct: bad argument");
    return reconstruct(p, high, phase, amp, nullptr, low, N, img, workspace, (cudaStream_t)stream);
}

int fvfi_pyr_reconstruct_complex(const fvfi_pyr_plan* p, const float* high, const float* const* bands,
                                 const float* low, int N, float* img, void* workspace, void* stream) {
    FVFI_CHECK_ARG(p && bands && img && workspace && N > 0 && N <= 65535, "pyr_reconstruct_complex: bad argument");
    return reconstruct(p, high, nullptr, nullptr, bands, low, N, img, workspace, (cudaStream_t)stream);
}

int fvfi_pyr_highband_filter(const fvfi_pyr_plan* p, const float* img, int N, float* out, void* workspace, void* stream) {
    FVFI_CHECK_ARG(p && img && out && workspace && N > 0 && N <= 65535, "pyr_highband_filter: bad argument");
    FVFI_CHECK_ARG(p->L >= 1 && p->hf_transfer, "pyr_highband_filter: the plan has no band level");
    return highband_filter(p, img, N, out, workspace, (cudaStream_t)stream);
}

int fvfi_pyr_reconstruct_backward(const fvfi_pyr_plan* p, const float* grad_img, int N, const float* const* phase,
                                  const float* const* amp, float* grad_high, float* const* grad_phase,
                                  float* const* grad_amp, float* grad_low, void* workspace, void* stream) {
    FVFI_CHECK_ARG(p && grad_img && phase && amp && grad_phase && grad_amp && workspace && N > 0 && N <= 65535,
                   "pyr_reconstruct_backward: bad argument");
    return reconstruct_backward(p, grad_img, N, phase, amp, grad_high, grad_phase, grad_amp, grad_low, workspace,
                                (cudaStream_t)stream);
}

}  // extern "C"
