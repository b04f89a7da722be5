"""oracle/yuv.py -- TEST INFRASTRUCTURE (see oracle/__init__.py).

numpy float32 restatement of the two 8-bit yuv420p conversions of libfvfi (include/fvfi.h: fvfi_yuv420p_to_rgb_lab and
fvfi_fusion_blend_yuv420p), in the kernels' operation order: every float32 product, sum and quotient is rounded on its own (numpy
never fuses them), rint rounds half to even.  The constants are computed in float64 from Kr, Kb and the range and rounded to
float32 once, as csrc/yuv.cuh does, so the device results are compared for exact equality.

Frames are [T,3H/2,W] uint8, 8-bit planar I420 (Y [H,W], then U [H/2,W/2], then V [H/2,W/2], contiguous per frame); chroma is
centre-sited.  For H % 4 == 2 the U plane ends in the middle of a row of that container, so the planes are cut from the flat bytes.
"""
import numpy as np

MATRICES = {"bt709": (0.2126, 0.0722), "bt601": (0.299, 0.114)}

f32 = np.float32


def constants(matrix="bt709", full_range=False):
    Kr, Kb = MATRICES[matrix]
    Kg = 1.0 - Kr - Kb
    c = dict(kr=Kr, kg=Kg, kb=Kb,
             kR=2.0 * (1.0 - Kr), kB=2.0 * (1.0 - Kb), kGb=2.0 * Kb * (1.0 - Kb) / Kg, kGr=2.0 * Kr * (1.0 - Kr) / Kg,
             kCb=1.0 / (2.0 * (1.0 - Kb)), kCr=1.0 / (2.0 * (1.0 - Kr)),
             yoff=0.0 if full_range else 16.0, ys=255.0 if full_range else 219.0, cs=255.0 if full_range else 224.0)
    return {k: f32(v) for k, v in c.items()}


def planes(yuv):
    """[T,3H/2,W] uint8 -> (Y [T,H,W], U [T,H/2,W/2], V [T,H/2,W/2]) views of the flat bytes."""
    yuv = np.ascontiguousarray(yuv, dtype=np.uint8)
    T, rows, W = yuv.shape
    H = 2 * rows // 3
    assert rows * 2 == 3 * H and H % 2 == 0 and W % 2 == 0
    flat = yuv.reshape(T, -1)
    n, m = H * W, H * W // 4
    return (flat[:, :n].reshape(T, H, W), flat[:, n:n + m].reshape(T, H // 2, W // 2),
            flat[:, n + m:].reshape(T, H // 2, W // 2))


def _upsample16(c):
    """[T,Hc,Wc] chroma -> [T,2Hc,2Wc] int32, 16x the [1,3]/4 x [1,3]/4 bilinear upsampling of centre-sited samples:
    9 C[i][j] + 3 C[i][j'] + 3 C[i'][j] + C[i'][j'], i = y/2, i' = i - 1 for even y and i + 1 for odd y (clamped), j' likewise."""
    c = c.astype(np.int32)
    Hc, Wc = c.shape[1:]
    y, x = np.arange(2 * Hc), np.arange(2 * Wc)
    i, j = y // 2, x // 2
    i2 = np.clip(np.where(y % 2, i + 1, i - 1), 0, Hc - 1)
    j2 = np.clip(np.where(x % 2, j + 1, j - 1), 0, Wc - 1)
    g = lambda r, s: c[:, r][:, :, s]
    return 9 * g(i, j) + 3 * g(i, j2) + 3 * g(i2, j) + g(i2, j2)


def decode(yuv, matrix="bt709", full_range=False):
    """yuv420p [T,3H/2,W] uint8 -> the rgb24 codes, planar uint8 [T,3,H,W] (fvfi_yuv420p_to_rgb_lab's rgb is these codes / 255)."""
    k = constants(matrix, full_range)
    Y, U, V = planes(yuv)
    yn = (Y.astype(np.int32) - int(k["yoff"])).astype(f32) / k["ys"]
    den = f32(16) * k["cs"]
    cbn = (_upsample16(U) - 2048).astype(f32) / den
    crn = (_upsample16(V) - 2048).astype(f32) / den
    r = yn + k["kR"] * crn
    g = (yn - k["kGb"] * cbn) - k["kGr"] * crn
    b = yn + k["kB"] * cbn
    rgb = np.stack([r, g, b], 1)
    return np.rint(np.clip(rgb, f32(0), f32(1)) * f32(255)).astype(np.uint8)


def _code8(v):
    return np.clip(np.rint(v), 0, 255).astype(np.uint8)


def encode(rgb, matrix="bt709", full_range=False):
    """R'G'B' values in [0,1], planar float32 [T,3,H,W] (H, W even) -> yuv420p [T,3H/2,W] uint8: Y per pixel, Cb / Cr from the
    2x2 block means ((v00 + v01) + (v10 + v11)) * 0.25 (fvfi_fusion_blend_yuv420p after its blend)."""
    k = constants(matrix, full_range)
    v = np.asarray(rgb, dtype=f32)
    T, C, H, W = v.shape
    assert C == 3 and H % 2 == 0 and W % 2 == 0
    luma = lambda r, g, b: (k["kr"] * r + k["kg"] * g) + k["kb"] * b
    Y = _code8(k["yoff"] + k["ys"] * luma(v[:, 0], v[:, 1], v[:, 2]))
    m = ((v[:, :, 0::2, 0::2] + v[:, :, 0::2, 1::2]) + (v[:, :, 1::2, 0::2] + v[:, :, 1::2, 1::2])) * f32(0.25)
    ym = luma(m[:, 0], m[:, 1], m[:, 2])
    cb = _code8(f32(128) + k["cs"] * ((m[:, 2] - ym) * k["kCb"]))
    cr = _code8(f32(128) + k["cs"] * ((m[:, 0] - ym) * k["kCr"]))
    out = np.concatenate([Y.reshape(T, -1), cb.reshape(T, -1), cr.reshape(T, -1)], 1)
    return out.reshape(T, 3 * H // 2, W)
