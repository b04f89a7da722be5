// yuv.cuh -- 8-bit yuv420p (I420) constants shared by the entry kernel (imgproc.cu, yuv420p_to_rgb_lab_kernel) and the exit kernel
// (adacof.cu, fusion_blend_yuv420p_kernel).  Every constant is computed in double from Kr, Kb and the range, then rounded to float
// once; oracle/yuv.py computes the same floats the same way, so both sides of the exact-equality tests use the same operands.
#pragma once
#include "common.cuh"

namespace fvfi {

struct YuvCoeffs {
    float kr, kg, kb;        // Y' = (Kr R' + Kg G') + Kb B'
    float kR, kB, kGb, kGr;  // decode: R' = Y' + kR Cr', B' = Y' + kB Cb', G' = (Y' - kGb Cb') - kGr Cr'
    float kCb, kCr;          // encode: Cb' = (B' - Y') kCb, Cr' = (R' - Y') kCr
    float yoff, ys, cs;      // range: Y = yoff + ys Y', Cb = 128 + cs Cb' (limited 16 / 219 / 224, full 0 / 255 / 255)
};

// matrix: 709 (Kr = 0.2126, Kb = 0.0722) or 601 (Kr = 0.299, Kb = 0.114); validated by yuv_check.
inline YuvCoeffs yuv_coeffs(int matrix, int full_range) {
    const double Kr = matrix == 709 ? 0.2126 : 0.299, Kb = matrix == 709 ? 0.0722 : 0.114;
    const double Kg = 1.0 - Kr - Kb;
    YuvCoeffs k;
    k.kr = (float)Kr;
    k.kg = (float)Kg;
    k.kb = (float)Kb;
    k.kR = (float)(2.0 * (1.0 - Kr));
    k.kB = (float)(2.0 * (1.0 - Kb));
    k.kGb = (float)(2.0 * Kb * (1.0 - Kb) / Kg);
    k.kGr = (float)(2.0 * Kr * (1.0 - Kr) / Kg);
    k.kCb = (float)(1.0 / (2.0 * (1.0 - Kb)));
    k.kCr = (float)(1.0 / (2.0 * (1.0 - Kr)));
    k.yoff = full_range ? 0.f : 16.f;
    k.ys = full_range ? 255.f : 219.f;
    k.cs = full_range ? 255.f : 224.f;
    return k;
}

// The size / format arguments both yuv420p entry points share (n = frames).  FVFI_EINVAL with the entry point's name.
inline int yuv_check(const char* name, int n, int H, int W, int matrix, int full_range) {
    FVFI_CHECK_ARG(n > 0 && n <= 65535 && H > 0 && W > 0, "%s: bad size n=%d H=%d W=%d", name, n, H, W);
    FVFI_CHECK_ARG(H % 2 == 0 && W % 2 == 0, "%s: yuv420p needs an even frame size, got H=%d W=%d", name, H, W);
    FVFI_CHECK_ARG(matrix == 709 || matrix == 601, "%s: matrix must be 709 or 601, got %d", name, matrix);
    FVFI_CHECK_ARG(full_range == 0 || full_range == 1, "%s: full_range must be 0 or 1, got %d", name, full_range);
    return FVFI_OK;
}

}  // namespace fvfi
