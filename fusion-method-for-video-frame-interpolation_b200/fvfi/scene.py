"""Scene-cut detection for 8-bit clips (include/fvfi.h: fvfi_frame_sad_u8, fvfi_scene_cut_decide, fvfi_scene_cut_select_u8;
DESIGN.md 6b).

At a cut, frames t and t + 1 show two unrelated shots and an interpolated frame between them is a ghosted double exposure.  With a
``SceneCutDetector`` passed to ``FusionPipeline.interpolate_sequence`` / ``interpolate_video_host`` (8-bit clips only), every pair
whose score reaches the threshold gets frame t itself, byte for byte, instead of the interpolated frame.  The rule, per pair p:

    sad[p]   = sum |f[p+1] - f[p]| over the Y plane (yuv420p) or all bytes (rgb24) of the frames, n bytes
    mafd[p]  = sad[p] * 100 / n / 256                               (float64, each operation rounded on its own)
    score[p] = clamp(min(mafd[p], |mafd[p] - mafd[p-1]|), 0, 100)   (mafd[-1] = 0 at the start of the stream)
    cut      = score[p] >= threshold

modelled on ffmpeg minterpolate's ``scd=fdiff``: a threshold around 10 means roughly what it means there.  Only the jump in
difference counts, so sustained fast motion does not fire on every pair.  Detection, decision and substitution run on the
device on the frames already uploaded, before a window's result is downloaded: no host round trip, no extra synchronisation.
"""
import math

import torch

from . import _lib


def _frame_stride(frames):
    """Bytes between frames of a uint8 device tensor [F, ...] whose frames are each contiguous."""
    if not frames.is_cuda or frames.dtype != torch.uint8 or frames.dim() < 2:
        raise ValueError("scene-cut kernels take uint8 CUDA tensors [frames, ...]")
    if not frames[0].is_contiguous():
        raise ValueError("scene-cut kernels need each frame contiguous")
    return frames.stride(0)


def frame_sad_u8(frames, n, sad=None):
    """int64 [F - 1]: the byte SAD of every pair of consecutive frames of ``frames`` [F, ...] uint8 over the first ``n`` bytes of
    each frame (fvfi_frame_sad_u8; exact).  ``sad``: optional output tensor."""
    stride = _frame_stride(frames)
    pairs = frames.shape[0] - 1
    if sad is None:
        sad = torch.empty(pairs, dtype=torch.int64, device=frames.device)
    assert sad.dtype == torch.int64 and sad.is_contiguous() and sad.numel() == pairs
    with torch.cuda.device(frames.device):
        _lib.check(_lib.lib().fvfi_frame_sad_u8(frames.data_ptr(), stride, int(n), pairs, sad.data_ptr(), _lib.stream_ptr()))
    return sad


def scene_cut_decide(sad, n, threshold, prev=None, mafd=None, cut=None):
    """(mafd float64 [P], cut uint8 [P]) of the SADs ``sad`` int64 [P] of consecutive pairs of n compared bytes
    (fvfi_scene_cut_decide).  ``prev``: device float64 [1], the stream's mafd before the first pair (None: start of a stream)."""
    P = sad.numel()
    if mafd is None:
        mafd = torch.empty(P, dtype=torch.float64, device=sad.device)
    if cut is None:
        cut = torch.empty(P, dtype=torch.uint8, device=sad.device)
    assert sad.dtype == torch.int64 and mafd.dtype == torch.float64 and cut.dtype == torch.uint8
    assert sad.is_contiguous() and mafd.is_contiguous() and cut.is_contiguous() and mafd.numel() == cut.numel() == P
    assert prev is None or (prev.dtype == torch.float64 and prev.is_cuda)
    with torch.cuda.device(sad.device):
        _lib.check(_lib.lib().fvfi_scene_cut_decide(sad.data_ptr(), P, int(n), _lib.ptr(prev), float(threshold), mafd.data_ptr(),
                                                    cut.data_ptr(), _lib.stream_ptr()))
    return mafd, cut


def scene_cut_select_u8(frames, out, cut):
    """out[p] = frames[p] wherever cut[p] != 0, for the P = out.shape[0] outputs (fvfi_scene_cut_select_u8); other outputs are left
    as they are.  frames [>= P, ...] and out [P, ...] uint8 with frames of equal size."""
    stride, out_stride = _frame_stride(frames), _frame_stride(out)
    P, frame_bytes = out.shape[0], out[0].numel()
    assert frames[0].numel() == frame_bytes and frames.shape[0] >= P and cut.dtype == torch.uint8 and cut.numel() == P
    with torch.cuda.device(out.device):
        _lib.check(_lib.lib().fvfi_scene_cut_select_u8(frames.data_ptr(), stride, out.data_ptr(), out_stride, frame_bytes, P,
                                                       cut.data_ptr(), _lib.stream_ptr()))
    return out


def check_threshold(threshold):
    """float(threshold) if it is a finite number >= 0; ValueError otherwise."""
    try:
        t = float(threshold)
    except (TypeError, ValueError):
        raise ValueError("scene-cut threshold must be a number, got %r" % (threshold,))
    if not math.isfinite(t) or t < 0:
        raise ValueError("scene-cut threshold must be finite and >= 0, got %r" % (threshold,))
    return t


class SceneCutDetector:
    """Scene-cut state of one stream: the threshold, the carried mafd of the last pair seen (a device float64 [1]; None before the
    first pair), the number of pairs seen, and the cuts found so far as global pair indices (``cuts``: pair p lies between
    frames p and p + 1 of the stream).  Pass one detector to every call of a stream, in order: the carry makes the result
    independent of how the stream is cut into calls and windows.  ``reset()`` starts a new stream."""

    def __init__(self, threshold=10.0):
        self.threshold = check_threshold(threshold)
        self.reset()

    def reset(self):
        self.prev = None
        self.pairs_seen = 0
        self._cuts = []
        self._pending = []        # (event, pinned cut flags, global index of their first pair) of calls not yet read

    @property
    def cuts(self):
        """Global indices of the pairs detected as cuts, in order.  The flags of a call reach the host by its own end-of-call
        synchronisation; reading them waits for that copy only."""
        for ev, flags, base in self._pending:
            ev.synchronize()
            self._cuts.extend(base + int(i) for i in torch.nonzero(flags).flatten().tolist())
        self._pending = []
        return list(self._cuts)

    def begin(self, pairs, n, device):
        """The per-call state of a call over ``pairs`` pairs of ``n`` compared bytes (FusionPipeline's clip entry points)."""
        return SceneCall(self, pairs, n, device)


class SceneCall:
    """One call's detection over its windows.  Window k reads the carry from the last pair of window k - 1 (``mafd``, one device
    array per call), window 0 the detector's carry as it was when the call began.  The detector itself changes only in
    ``commit()``, which the entry point runs once when it returns: a call that the 3xFP16 range guard runs a second time
    (conv.range_checked) recomputes the same flags from the same carry, and the detector comes out as if it had run once."""

    def __init__(self, detector, pairs, n, device):
        self.detector, self.pairs, self.n = detector, pairs, n
        self.prev = detector.prev
        self.sad = torch.empty(pairs, dtype=torch.int64, device=device)
        self.mafd = torch.empty(pairs, dtype=torch.float64, device=device)
        self.cut = torch.empty(pairs, dtype=torch.uint8, device=device)
        self.flags = torch.empty(pairs, dtype=torch.uint8, pin_memory=True)
        self.event = None

    def detect(self, frames, a):
        """SAD and decision of the pairs a .. a + B - 1 of the call, from the window's B + 1 uploaded frames [B+1, ...]."""
        b = frames.shape[0] - 1
        sad = frame_sad_u8(frames, self.n, self.sad[a:a + b])
        prev = self.prev if a == 0 else self.mafd[a - 1:a]
        scene_cut_decide(sad, self.n, self.detector.threshold, prev, self.mafd[a:a + b], self.cut[a:a + b])

    def select(self, frames, out, a):
        """Frame a + p of the call in place of the window's interpolated frame p at every cut; after the last window the flags
        start their copy to the host on the same stream."""
        b = out.shape[0]
        scene_cut_select_u8(frames, out, self.cut[a:a + b])
        if a + b == self.pairs:
            self.flags.copy_(self.cut, non_blocking=True)
            self.event = torch.cuda.Event()
            self.event.record()

    def commit(self):
        d = self.detector
        d.prev = self.mafd[-1:]
        d._pending.append((self.event, self.flags, d.pairs_seen))
        d.pairs_seen += self.pairs
