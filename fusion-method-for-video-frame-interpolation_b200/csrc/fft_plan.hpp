// fft_plan.hpp -- host-side planning for fft_engine.cuh: radix selection, Bluestein length, tables (all in double).
#pragma once
#include <math.h>

#include <algorithm>
#include <complex>
#include <vector>

#include "fft_engine.cuh"

namespace fvfi {

struct HostFftPlan {
    FftPlan p{};                       // pointers are filled in by whoever owns the storage (device upload or host test)
    std::vector<float2> tw, chirp, bhat, tw2;
    std::vector<unsigned short> perm, pin, inv, pos_in;
};

// Split n into the radices the engine implements; false if n has a prime factor > 19.
inline bool fft_radices(int n, std::vector<int>& out) {
    out.clear();
    int e2 = 0, e3 = 0, e5 = 0;
    std::vector<int> big;
    int rem = n;
    while (rem % 2 == 0) { rem /= 2; ++e2; }
    while (rem % 3 == 0) { rem /= 3; ++e3; }
    while (rem % 5 == 0) { rem /= 5; ++e5; }
    for (int p : {7, 11, 13, 17, 19})
        while (rem % p == 0) { rem /= p; big.push_back(p); }
    if (rem != 1) return false;
    std::vector<int> odd(big);
    while (e3 >= 1 && e5 >= 1 && (e3 & 1)) { odd.push_back(15); --e3; --e5; }
    while (e3 >= 2) { odd.push_back(9); e3 -= 2; }
    // a lone 2 or 4 would cost a full pass: merge it with a lone 3 / 5 (radix 6, 10, 12)
    std::vector<int> pow2;
    while (e2 >= 4 && e2 != 5 && e2 != 6) { pow2.push_back(16); e2 -= 4; }
    if (e2 == 6) { pow2.push_back(8); pow2.push_back(8); e2 = 0; }
    if (e2 == 5) { pow2.push_back(8); pow2.push_back(4); e2 = 0; }
    if (e2 == 3) { pow2.push_back(8); e2 = 0; }
    if (e2 == 2) {
        if (e3 == 1) { odd.push_back(12); e3 = 0; } else pow2.push_back(4);
        e2 = 0;
    }
    if (e2 == 1) {
        if (e3 == 1) { odd.push_back(6); e3 = 0; }
        else if (e5 >= 1) { odd.push_back(10); --e5; }
        else pow2.push_back(2);
        e2 = 0;
    }
    while (e3 >= 1) { odd.push_back(3); --e3; }
    while (e5 >= 1) { odd.push_back(5); --e5; }
    std::sort(pow2.begin(), pow2.end(), [](int a, int b) { return a > b; });
    std::sort(odd.begin(), odd.end(), [](int a, int b) { return (a & 1) != (b & 1) ? (a & 1) < (b & 1) : a > b; });   // 12/10/6 before odd
    out = pow2;                        // DIF order: power-of-two radices first, odd (conflict-free strides) last
    out.insert(out.end(), odd.begin(), odd.end());
    if (out.empty()) out.push_back(1);
    return (int)out.size() <= FFT_MAX_STAGES;
}

// Reference DFT in double (mixed radix recursion, naive at prime leaves) for the plan tables.
inline void fft_host_dft(std::vector<std::complex<double>>& x) {
    const int n = (int)x.size();
    if (n <= 1) return;
    int r = n;
    for (int d = 2; d * d <= n; ++d)
        if (n % d == 0) { r = d; break; }
    if (r == n) {
        std::vector<std::complex<double>> y(n);
        for (int k = 0; k < n; ++k) {
            std::complex<double> s = 0;
            for (int j = 0; j < n; ++j) s += x[j] * std::polar(1.0, -2.0 * M_PI * (double)((long long)j * k % n) / n);
            y[k] = s;
        }
        x = y;
        return;
    }
    const int m = n / r;
    std::vector<std::vector<std::complex<double>>> sub(r, std::vector<std::complex<double>>(m));
    for (int j = 0; j < n; ++j) sub[j % r][j / r] = x[j];
    for (int q = 0; q < r; ++q) fft_host_dft(sub[q]);
    for (int k = 0; k < n; ++k) {
        std::complex<double> s = 0;
        for (int q = 0; q < r; ++q) s += sub[q][k % m] * std::polar(1.0, -2.0 * M_PI * (double)((long long)q * k % n) / n);
        x[k] = s;
    }
}

inline unsigned fft_magic(unsigned d) { return d <= 1 ? 0u : (unsigned)(((1ull << 32) + d - 1) / d); }

inline long long fft_powmod(long long b, long long e, long long m) {
    long long r = 1 % m;
    b %= m;
    while (e > 0) {
        if (e & 1) r = r * b % m;
        b = b * b % m;
        e >>= 1;
    }
    return r;
}

// n = r * p with exactly one prime factor p > 19 (to the first power), r and p - 1 both products of the implemented radices.
inline bool fft_rader_split(int n, int* r_out, int* p_out) {
    int rem = n;
    for (int q : {2, 3, 5, 7, 11, 13, 17, 19})
        while (rem % q == 0) rem /= q;
    if (rem <= 19) return false;                       // smooth (handled directly) -- or nothing left
    for (int d = 2; (long long)d * d <= rem; ++d)
        if (rem % d == 0) return false;                // more than one large prime factor (or a square): Bluestein
    const int p = rem, r = n / p;
    std::vector<int> t;
    if (!fft_radices(r, t) || !fft_radices(p - 1, t)) return false;
    *r_out = r;
    *p_out = p;
    return true;
}

// Rader plan (see fft_engine.cuh): outer DIT stages for r, sub-FFT stages for q = p - 1, generator-order tables.
inline bool fft_make_rader_plan(int n, int r, int pr, HostFftPlan& H) {
    FftPlan& p = H.p;
    const int q = pr - 1;
    std::vector<int> rad_r, rad_q;
    if (!fft_radices(r, rad_r) || !fft_radices(q, rad_q)) return false;
    if (r == 1) rad_r.clear();
    if ((int)(rad_r.size() + rad_q.size()) > FFT_MAX_STAGES || n > 32767) return false;
    p.M = n;
    p.bluestein = 0;
    p.rader = 1;
    p.rr = r; p.rp = pr; p.rq = q;
    p.nouter = (int)rad_r.size();
    p.nfac = p.nouter + (int)rad_q.size();
    p.pad = 0;
    int prod = 1;
    for (int s = 0; s < p.nouter; ++s) {               // DIT on length n (butterfly stride m_s as for DIF)
        p.fac[s] = rad_r[s];
        prod *= rad_r[s];
        p.sub[s] = n / prod;
        p.mag_sub[s] = fft_magic((unsigned)p.sub[s]);
        p.mag_items[s] = fft_magic((unsigned)(n / rad_r[s]));
    }
    prod = 1;
    for (int i = 0; i < (int)rad_q.size(); ++i) {      // DIF / DIT on length q
        const int s = p.nouter + i;
        p.fac[s] = rad_q[i];
        prod *= rad_q[i];
        p.sub[s] = q / prod;
        p.mag_sub[s] = fft_magic((unsigned)p.sub[s]);
        p.mag_items[s] = fft_magic((unsigned)(q / rad_q[i]));
        p.mag_ritems[s] = fft_magic((unsigned)(r * (q / rad_q[i])));
    }
    H.tw.resize(n);
    for (int t = 0; t < n; ++t) {
        const double a = -2.0 * M_PI * (double)t / (double)n;
        H.tw[t] = make_float2((float)cos(a), (float)sin(a));
    }
    H.tw2.resize(q);
    for (int t = 0; t < q; ++t) {
        const double a = -2.0 * M_PI * (double)t / (double)q;
        H.tw2[t] = make_float2((float)cos(a), (float)sin(a));
    }
    // primitive root g of pr, powers and discrete logarithms
    int g = 0;
    {
        std::vector<int> pf;
        int rem = q;
        for (int d = 2; d * d <= rem; ++d)
            if (rem % d == 0) { pf.push_back(d); while (rem % d == 0) rem /= d; }
        if (rem > 1) pf.push_back(rem);
        for (int c = 2; c < pr && !g; ++c) {
            bool ok = true;
            for (int f : pf) ok = ok && fft_powmod(c, q / f, pr) != 1;
            if (ok) g = c;
        }
        if (!g) return false;
    }
    std::vector<int> gpow(q), dlog(pr, 0);
    for (int t = 0; t < q; ++t) { gpow[t] = (int)fft_powmod(g, t, pr); dlog[gpow[t]] = t; }
    H.pin.assign(pr, 0);
    for (int j = 1; j < pr; ++j) H.pin[j] = (unsigned short)(1 + dlog[j]);        // slot 1 + t holds y[g^t]
    // digit reversal of the sub network (position -> natural bin of the q-point DFT)
    std::vector<int> subperm(q);
    for (int pos = 0; pos < q; ++pos) {
        int rem = pos, k = 0, w = 1;
        for (int s = p.nouter; s < p.nfac; ++s) {
            const int d = rem / p.sub[s];
            rem -= d * p.sub[s];
            k += d * w;
            w *= p.fac[s];
        }
        subperm[pos] = k;
    }
    // convolution kernel b[t] = W_p^(g^-t) = W_p^(g^((q - t) mod q)); spectrum / q in DIF order
    std::vector<std::complex<double>> bk(q);
    for (int t = 0; t < q; ++t) bk[t] = std::polar(1.0, -2.0 * M_PI * (double)gpow[(q - t) % q] / (double)pr);
    fft_host_dft(bk);
    H.bhat.resize(q);
    for (int pos = 0; pos < q; ++pos) {
        const std::complex<double> v = bk[subperm[pos]] / (double)q;
        H.bhat[pos] = make_float2((float)v.real(), (float)v.imag());
    }
    // input i = sum_s d_s prod_{t<s} fac_t + r * j sits at position sum_s d_s sub_s + slot(j); the radix stages of r then run over
    // blocks that hold their spectra in generator order, so X[k2 + rp * K1] ends at position K1 * rp + slot(k2)
    std::vector<int> k2_of_slot(pr, 0);                // slot 1 + m holds X[g^-m]
    for (int m = 0; m < q; ++m) k2_of_slot[1 + m] = gpow[(q - m) % q];
    H.pos_in.assign(n, 0);
    for (int i = 0; i < n; ++i) {
        int rem = i % r, pos = 0;
        for (int s = 0; s < p.nouter; ++s) { pos += (rem % p.fac[s]) * p.sub[s]; rem /= p.fac[s]; }
        H.pos_in[i] = (unsigned short)(pos + H.pin[i / r]);
    }
    H.perm.assign(n, 0);
    H.inv.assign(n, 0);
    for (int pos = 0; pos < n; ++pos) {
        const int k = (pos / pr) * pr + k2_of_slot[pos % pr];
        H.perm[pos] = (unsigned short)k;
        H.inv[k] = (unsigned short)pos;
    }
    H.chirp.clear();
    return true;
}

// Build the plan for length n.  stockham = true: out-of-place autosort order for direct lengths (rows).  rader = false: Bluestein
// for every non-smooth length (lets the host test run the Bluestein code on the lengths Rader would take).
inline bool fft_make_plan(int n, bool stockham, HostFftPlan& H, bool rader = true) {
    FftPlan& p = H.p;
    p = FftPlan{};
    p.n = n;
    std::vector<int> rad;
    {
        int rr = 0, rp = 0;
        if (rader && !fft_radices(n, rad) && fft_rader_split(n, &rr, &rp) && fft_make_rader_plan(n, rr, rp, H)) return true;
        p = FftPlan{};
        p.n = n;
    }
    if (fft_radices(n, rad)) {
        p.M = n;
        p.bluestein = 0;
    } else {
        // Bluestein: smooth M >= 2n-1 minimising M * stages
        long best = -1;
        int bestM = 0;
        for (int M = 2 * n - 1; M <= 4 * n; ++M) {
            std::vector<int> r;
            int rem = M;
            for (int q : {2, 3, 5})
                while (rem % q == 0) rem /= q;
            if (rem != 1 || !fft_radices(M, r)) continue;
            const long cost = (long)M * (long)r.size();
            if (best < 0 || cost < best) { best = cost; bestM = M; }
        }
        if (best < 0) return false;
        p.M = bestM;
        p.bluestein = 1;
        fft_radices(bestM, rad);
        stockham = false;
    }
    const int M = p.M;
    if (M > 65535) return false;
    if (stockham) std::reverse(rad.begin(), rad.end());   // odd radix first: its stride-R stores are conflict free
    p.nfac = (int)rad.size();
    if (rad.size() == 1 && rad[0] == 1) p.nfac = 0;
    int prod = 1;
    for (int s = 0; s < p.nfac; ++s) {
        p.fac[s] = rad[s];
        if (stockham) {
            p.sub[s] = prod;                 // Ns
            prod *= rad[s];
        } else {
            prod *= rad[s];
            p.sub[s] = M / prod;             // m_s
        }
        p.mag_sub[s] = fft_magic((unsigned)p.sub[s]);
        p.mag_items[s] = fft_magic((unsigned)(M / rad[s]));
    }
    // smallest butterfly stride: first Stockham radix / last DIF radix; even -> skewed rows
    p.pad = (p.nfac > 0 && ((stockham ? p.fac[0] : p.fac[p.nfac - 1]) % 2 == 0)) ? 1 : 0;
    H.tw.resize(M);
    for (int t = 0; t < M; ++t) {
        const double a = -2.0 * M_PI * (double)t / (double)M;
        H.tw[t] = make_float2((float)cos(a), (float)sin(a));
    }
    // digit reversal of the DIF network: position p = sum d_s * m_s  <->  natural k = sum d_s * prod_{i<s} fac_i
    H.perm.assign(M, 0);
    if (!stockham) {
        for (int pos = 0; pos < M; ++pos) {
            int rem = pos, k = 0, w = 1;
            for (int s = 0; s < p.nfac; ++s) {
                const int d = rem / p.sub[s];
                rem -= d * p.sub[s];
                k += d * w;
                w *= p.fac[s];
            }
            H.perm[pos] = (unsigned short)k;
        }
    }
    H.chirp.clear();
    H.bhat.clear();
    if (p.bluestein) {
        H.chirp.resize(n);
        std::vector<std::complex<double>> b(M, 0.0);
        for (int k = 0; k < n; ++k) {
            const long long k2 = ((long long)k * k) % (2LL * n);     // exact angle reduction
            const double a = M_PI * (double)k2 / (double)n;
            H.chirp[k] = make_float2((float)cos(a), (float)-sin(a));   // exp(-i pi k^2 / n)
            const std::complex<double> bk = std::polar(1.0, a);        // exp(+i pi k^2 / n)
            b[k] = bk;
            if (k) b[M - k] = bk;
        }
        fft_host_dft(b);
        H.bhat.resize(M);
        for (int pos = 0; pos < M; ++pos) {
            const std::complex<double> v = b[H.perm[pos]] / (double)M;
            H.bhat[pos] = make_float2((float)v.real(), (float)v.imag());
        }
    }
    return true;
}

}  // namespace fvfi
