"""oracle/scene.py -- TEST INFRASTRUCTURE (see oracle/__init__.py).

numpy restatement of the scene-cut rule of libfvfi (include/fvfi.h: fvfi_frame_sad_u8, fvfi_scene_cut_decide,
fvfi_scene_cut_select_u8; DESIGN.md 6b).  Per pair p = (frame p, frame p + 1) of a stream:
  sad[p]   = sum of |f[p+1][i] - f[p][i]| over the compared bytes (int64): the Y plane (the first H W bytes) of a yuv420p frame,
             all 3 H W bytes of an rgb24 frame;
  mafd[p]  = sad[p] * 100.0 / n / 256.0 in float64, each operation rounded on its own;
  score[p] = clamp(min(mafd[p], |mafd[p] - prev|), 0, 100), prev = mafd[p - 1] of the stream (0 for the first pair);
  cut[p]   = score[p] >= threshold, and then the interpolated frame p is frame p itself, byte for byte.
"""
import numpy as np


def compared_bytes(frames, pix_fmt):
    """[T, n] uint8: the bytes of each frame that the detector compares (pix_fmt 'rgb24' or 'yuv420p')."""
    f = np.ascontiguousarray(frames, dtype=np.uint8)
    flat = f.reshape(f.shape[0], -1)
    if pix_fmt == "yuv420p":
        rows, W = f.shape[1:]
        return flat[:, :2 * rows // 3 * W]
    if pix_fmt != "rgb24":
        raise ValueError(pix_fmt)
    return flat


def sad(frames, pix_fmt):
    """int64 [T - 1]: the byte SAD of every pair of consecutive frames."""
    b = compared_bytes(frames, pix_fmt).astype(np.int64)
    return np.abs(b[1:] - b[:-1]).sum(axis=1, dtype=np.int64)


def mafd(sad_, n):
    return np.asarray(sad_, np.int64).astype(np.float64) * 100.0 / float(n) / 256.0


def decide(sad_, n, threshold, prev=None):
    """(mafd float64 [P], cut bool [P]) for SADs of P consecutive pairs; prev: the stream's mafd before the first of them (None:
    start of the stream, 0)."""
    m = mafd(sad_, n)
    before = np.concatenate(([0.0 if prev is None else float(prev)], m[:-1]))
    score = np.clip(np.minimum(m, np.abs(m - before)), 0.0, 100.0)
    return m, score >= threshold


def detect(frames, pix_fmt, threshold, prev=None):
    """(cut indices [list of int], mafd float64 [T - 1]) of a clip."""
    f = np.asarray(frames)
    n = compared_bytes(f[:1], pix_fmt).shape[1]
    m, cut = decide(sad(f, pix_fmt), n, threshold, prev)
    return [int(i) for i in np.flatnonzero(cut)], m


def substitute(frames, interpolated, cuts):
    """The interpolated frames with frame p in place of interpolated frame p at every cut p."""
    out = np.array(interpolated, dtype=np.uint8, copy=True)
    for p in cuts:
        out[p] = frames[p]
    return out
