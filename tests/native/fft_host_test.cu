// Host-side harness for csrc/fft_engine.cuh: runs the SAME stage code (index math, butterflies, Bluestein
// driver) on the CPU with one "thread", so tests/test_fft_engine_host.py can check every length against numpy.fft.
#include <string.h>

#include <vector>

#include "fft_plan.hpp"

using namespace fvfi;

// mode 0: rows layout, out-of-place (Stockham) for direct lengths; mode 1: columns layout, in-place DIF (+perm)
// rader 0: Bluestein for every non-smooth length (fft_make_plan's rader = false); otherwise the plans the library uses.
// in/out: [batch][n][2] floats.  Returns 0, or -1 if no plan.
extern "C" int fft_host_run(int n, int mode, int batch, const float* in, float* out, int* info, int rader) {
    HostFftPlan H;
    const bool col = mode == 1;
    if (!fft_make_plan(n, !col, H, rader != 0)) return -1;
    H.p.tw = H.tw.data();
    H.p.perm = H.p.bluestein ? nullptr : H.perm.data();
    H.p.chirp = H.chirp.data();
    H.p.bhat = H.bhat.data();
    if (H.p.rader) {
        H.p.perm = H.perm.data();
        H.p.tw2 = H.tw2.data();
        H.p.inv = H.inv.data();
        H.p.pos_in = H.pos_in.data();
    }
    const int M = H.p.M;
    int ctshift = 0;
    while ((1 << ctshift) < batch) ++ctshift;
    const int pitch = fft_pitch(H.p);
    const size_t elems = col ? ((size_t)M << ctshift) : (size_t)batch * pitch;
    // garbage-filled on purpose, with a guard zone behind each buffer: the stage code must stay inside [0, elems) -- the bound the
    // kernels size their shared memory by (M << ctshift columns / batch * pitch rows)
    constexpr size_t GUARD = 256;
    const float2 canary = make_float2(-12345.f, 54321.f);
    std::vector<float2> a(elems + GUARD, make_float2(7.f, 7.f)), b(elems + GUARD, make_float2(9.f, 9.f));
    for (size_t i = 0; i < GUARD; ++i) a[elems + i] = b[elems + i] = canary;
    for (int bb = 0; bb < batch; ++bb)
        for (int i = 0; i < n; ++i) {
            const float2 v = make_float2(in[((size_t)bb * n + i) * 2], in[((size_t)bb * n + i) * 2 + 1]);
            if (col) fft_put<true>(fft_io(H.p), a.data(), bb, i, v, ctshift, pitch);
            else fft_put<false>(fft_io(H.p), a.data(), bb, i, v, ctshift, pitch);
        }
    FftResult r = col ? fft_forward<true>(H.p, a.data(), b.data(), batch, ctshift, pitch, true, FftCtx{0, 1})
                      : fft_forward<false>(H.p, a.data(), b.data(), batch, ctshift, pitch, false, FftCtx{0, 1});
    for (int bb = 0; bb < batch; ++bb)
        for (int pos = 0; pos < n; ++pos) {
            const float2 v = col ? fft_get<true>(fft_io(H.p), r, bb, pos, ctshift, pitch) : fft_get<false>(fft_io(H.p), r, bb, pos, ctshift, pitch);
            const int k = (r.perm && (col || !H.p.rader)) ? r.perm[pos] : pos;     // rows of a Rader plan read in natural order (inv table)
            out[((size_t)bb * n + k) * 2] = v.x;
            out[((size_t)bb * n + k) * 2 + 1] = v.y;
        }
    for (size_t i = 0; i < GUARD; ++i)
        if (a[elems + i].x != canary.x || a[elems + i].y != canary.y || b[elems + i].x != canary.x || b[elems + i].y != canary.y) return -2;
    if (info) {
        info[0] = M;
        info[1] = H.p.bluestein + 2 * (H.p.rader != 0);
        info[2] = H.p.nfac;
        for (int s = 0; s < H.p.nfac; ++s) info[3 + s] = H.p.fac[s];
    }
    return 0;
}
