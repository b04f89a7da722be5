"""Drop-in for the reference's ``src/phase_net/phase_net.py`` (PhaseNet, PhaseNetBlock).

Same constructor (``PhaseNet(pyr, device, num_img=2)``), same ``normalize_vals`` / ``forward(vals, m)`` /
``reverse_normalize`` semantics and the same parameter names (``layers.{i}.feature_map.{0,1,3}.*``,
``layers.{i}.prediction_map.0.*``) so ``phase_net.pt`` loads unchanged.  Differences that do not
change results: no ``torch.cuda.empty_cache()`` in the level loop (phase_net.py:145,152), planes can
be processed in chunks to bound the 88-channel concat (SURVEY.md H3), and the alpha/beta blends
(phase_net.py:114-116,155-156) are single fused expressions.
"""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import conv as tc
from .pyramid import DecompValues


class PhaseNetBlock(nn.Module):
    """phase_net.py:179-207."""

    def __init__(self, c_in, c_out, pred_out, kernel_size, device, dropout=0.5):
        super(PhaseNetBlock, self).__init__()
        padding = 1 if kernel_size == (3, 3) else 0
        self.feature_map = nn.Sequential(
            nn.Conv2d(c_in, c_out, kernel_size, padding=padding, padding_mode='reflect'),
            nn.BatchNorm2d(c_out),
            nn.ELU(),
            nn.Conv2d(c_out, c_out, kernel_size, padding=padding, padding_mode='reflect'),
            nn.ELU(),
        )
        self.prediction_map = nn.Sequential(
            nn.Conv2d(c_out, pred_out, (1, 1), padding_mode='reflect'),
            nn.Tanh()
        )
        self.to(device)

    @tc.range_checked
    def forward(self, x):
        if tc.use_tc(x) and not self.training:
            # tcgen05 path: conv+BN(folded)+ELU, conv+ELU, 1x1 conv+tanh -- three fused kernels (phase_net.py:190-200)
            f = tc.conv_bn_module(self.feature_map[0], self.feature_map[1], x, "elu")
            f = tc.conv_module(self.feature_map[3], f, "elu")
            c = tc.conv_module(self.prediction_map[0], f, "tanh")
            return f, c
        if x.is_cuda:
            # training / autograd: the three convolutions -- forward AND backward -- on libfvfi (conv._ConvTC: tcgen05 forward and
            # data gradient, csrc/conv_bwd.cu weight / bias gradients); BatchNorm (batch statistics in train mode) stays torch's
            fm = self.feature_map
            f = fm[2](fm[1](tc.conv_module(fm[0], x, None)))
            f = tc.conv_module(fm[3], f, "elu")
            c = tc.conv_module(self.prediction_map[0], f, "tanh")
            return f, c
        raise NotImplementedError("fvfi PhaseNetBlock runs on CUDA tensors only (no CPU fallback)")

    def forward_resampled(self, feature, direct, size):
        """``forward(cat(interpolate(feature, size), direct))`` without the concatenated tensor: the first convolution's loaders
        resample the previous level's features while they stage them (fvfi_conv2d_nhwc_upsampled, two-source form); ``direct``
        [B, >= c_in - 64, h, w] holds this level's value channels and the resampled previous prediction (phase_net.py:138-148)."""
        assert not self.training and not torch.is_grad_enabled()
        f = tc.conv_bn_module(self.feature_map[0], self.feature_map[1], feature, "elu", upsample=(size, False), x_direct=direct)
        f = tc.conv_module(self.feature_map[3], f, "elu")
        c = tc.conv_module(self.prediction_map[0], f, "tanh")
        return f, c


class PhaseNet(nn.Module):
    """Phase Net for Video Frame Interpolation (phase_net.py:7-177)."""

    def __init__(self, pyr, device, num_img=2):
        super(PhaseNet, self).__init__()
        self.pyr = pyr
        self.device = device
        self.num_img = num_img
        self.layers = self.create_architecture()
        self.to(self.device)
        self.eps = 1e-8
        self.plane_chunk = None  # planes per forward chunk (None = all at once)

    def create_architecture(self):
        n = self.num_img
        if n == 3:
            return nn.ModuleList([
                PhaseNetBlock(n, 64, n - 1, (1, 1), self.device),
                PhaseNetBlock(64 + n - 1 + 8 * n, 64, n * 4, (1, 1), self.device),
                PhaseNetBlock(64 + n * 4 + 8 * n, 64, n * 4, (1, 1), self.device),
                *[PhaseNetBlock(64 + n * 4 + 8 * n, 64, n * 4, (3, 3), self.device) for _ in range(5)]
            ])
        return nn.ModuleList([
            PhaseNetBlock(n, 64, 1, (1, 1), self.device),
            PhaseNetBlock(64 + 1 + 8 * n, 64, 8, (1, 1), self.device),
            PhaseNetBlock(64 + 8 + 8 * n, 64, 8, (1, 1), self.device),
            *[PhaseNetBlock(64 + 8 + 8 * n, 64, 8, (3, 3), self.device) for _ in range(5)]
        ])

    def set_layers(self, start, end, freeze=True):
        for param in self.layers[start:end].parameters():
            param.requires_grad = freeze

    def normalize_vals(self, vals):
        """phase_net.py:42-78: amplitude / (per-plane max + eps), phase / pi, low / (per-plane max + eps).
        The maxima are kept on ``self`` for compatibility (reverse_normalize reads them)."""
        batch_size = int(vals.amplitude[0].shape[0])
        self.max_amplitudes = []
        amplitudes = []
        for amplitude in vals.amplitude:
            max_amplitude = amplitude.reshape(batch_size, -1).max(1)[0] + self.eps
            self.max_amplitudes.append(max_amplitude)
            amplitudes.append(amplitude / max_amplitude.view(-1, 1, 1, 1))
        phases = [x / math.pi for x in vals.phase]
        self.max_low_level = vals.low_level.reshape(batch_size, -1).max(1)[0] + self.eps   # max, not max|.| (:70)
        low_level = vals.low_level / self.max_low_level.view(-1, 1, 1, 1)
        return DecompValues(high_level=vals.high_level, low_level=low_level, amplitude=amplitudes, phase=phases)

    def reverse_normalize(self, vals, m):
        """phase_net.py:80-105."""
        phases = [x * math.pi for x in vals.phase]
        amplitudes = []
        for i in range(m):
            amp = vals.amplitude[i]
            batch_size = int(amp.shape[0] / self.pyr.nbands)
            amplitudes.append((amp.reshape(batch_size, -1) * self.max_amplitudes[i].view(-1, 1)).reshape(amp.shape))
        for _ in range(self.pyr.height - 2 - m):
            phases.append(0)
            amplitudes.append(0)
        low_level = vals.low_level * self.max_low_level.view(-1, 1, 1, 1)
        return DecompValues(high_level=vals.high_level, low_level=low_level, amplitude=amplitudes[::-1],
                            phase=phases[::-1])

    def _forward_planes(self, low, phase, amplitude, m):
        feature, prediction = self.layers[0](low)
        alpha = (prediction[:, 0] + 1) / 2
        low_level = alpha * low[:, 0] + (1 - alpha) * low[:, 1]                      # phase_net.py:114-116
        if self.num_img == 3:
            fusion_alpha = (prediction[:, 1] + 1) / 2
            low_level = fusion_alpha * low_level + (1 - fusion_alpha) * low[:, 2]
        low_level = low_level.unsqueeze(1)
        phases, amplitudes = [], []
        for idx in range(m):
            res = phase[idx].shape[2:]
            if tc.use_tc(feature) and not self.training:
                # NHWC concat assembled in place: resize kernels write straight into their channel slices
                cf, cp, cv = feature.shape[1], prediction.shape[1], phase[idx].shape[1]
                concat = torch.empty((feature.shape[0], cf + 2 * cv + cp, res[0], res[1]), dtype=torch.float32,
                                     device=feature.device, memory_format=torch.channels_last)
                tc.resize_bilinear(feature, res, False, out=concat, out_channel_offset=0)
                tc.put_planar(phase[idx], concat, cf)
                tc.put_planar(amplitude[idx], concat, cf + cv)
                tc.resize_bilinear(prediction, res, False, out=concat, out_channel_offset=cf + 2 * cv)
            else:
                feature_r = F.interpolate(feature, size=tuple(res), mode='bilinear', align_corners=False)
                prediction_r = F.interpolate(prediction, size=tuple(res), mode='bilinear', align_corners=False)
                concat = torch.cat((feature_r, phase[idx], amplitude[idx], prediction_r), 1)
            i = idx + 1 if idx + 1 < len(self.layers) - 1 else len(self.layers) - 1
            feature, prediction = self.layers[i](concat)
            del concat
            beta = (prediction[:, 4:8] + 1) / 2
            amp = beta * amplitude[idx][:, 4:8] + (1 - beta) * amplitude[idx][:, :4]  # phase_net.py:155-156
            if self.num_img == 3:
                fusion_beta = (prediction[:, 8:12] + 1) / 2
                amp = fusion_beta * amp + (1 - fusion_beta) * amplitude[idx][:, 8:12]
            r1, r2 = prediction.shape[2:]
            phases.append(prediction[:, :4].reshape(-1, 1, r1, r2))
            amplitudes.append(amp.reshape(-1, 1, r1, r2))
        return low_level, phases, amplitudes

    @tc.range_checked
    def forward_fused(self, vals, amp_max, m=None, frame2=None):
        """Fused inference form of  separate_vals -> get_concat_layers_inf -> normalize_vals -> forward -> reverse_normalize
        (src/train/utils.py:47-127, phase_net.py:42-177) for two input frames.

        ``vals``: the RAW decomposition (``Pyramid.filter``) of N planes, lists finest first, in which frame 2 of pair-plane p is
        plane p + q, q = ``frame2``: the default N // 2 is ``cat(frame-1 planes, frame-2 planes)`` (N = 2*P); a clip of T'
        consecutive frames decomposed once is q = 3 (pair t = frames t, t + 1), P = N - q.  ``amp_max`` [L, N]: the per-level
        per-plane amplitude maxima from the decomposition's epilogue (``Pyramid.last_amp_max``).  Returns the DecompValues
        ``Pyramid.inv_filter`` consumes (P planes).  The value channels of
        every level's concat are written by ONE kernel straight from the decomposition (fvfi_phasenet_assemble) and the amplitude
        blend + de-normalisation by another (fvfi_phasenet_outputs): the regrouped / normalised / re-scaled copies of the whole
        pyramid that the step-by-step form materialises (~80 GB per 8 frame pairs at 1080p) never exist."""
        from . import _lib
        assert self.num_img == 2 and vals.low_level.is_cuda and not self.training and not torch.is_grad_enabled()
        L, nb = len(vals.phase), self.pyr.nbands
        if m is None:
            m = self.pyr.height - 2
        N = vals.low_level.shape[0]
        q = N // 2 if frame2 is None else int(frame2)
        P = N - q
        assert 0 < q < N, (q, N)
        dev = vals.low_level.device
        low = torch.cat((vals.low_level[:P], vals.low_level[q:q + P]), 1)                  # [P,2,hL,wL] (a few hundred values)
        self.max_low_level = low.reshape(P, -1).max(1)[0] + self.eps                       # max, not max|.| (phase_net.py:70)
        low = low / self.max_low_level.view(-1, 1, 1, 1)
        den = (torch.maximum(amp_max[:, :P], amp_max[:, q:q + P]) + self.eps).contiguous() # [L,P]: max over both frames' bands + eps
        self.max_amplitudes = [den[L - 1 - i] for i in range(m)]                           # coarsest first, as normalize_vals keeps them
        new = lambda *sh: torch.empty(sh, dtype=torch.float32, device=dev)
        phase_out = [new(P * nb, 1, *vals.phase[l].shape[2:]) if l >= L - m else 0 for l in range(L)]
        amp_out = [new(P * nb, 1, *vals.phase[l].shape[2:]) if l >= L - m else 0 for l in range(L)]
        lows = []
        lib = _lib.lib()
        chunk = self.plane_chunk or P
        for p0 in range(0, P, chunk):
            pc = min(chunk, P - p0)
            lo = low[p0:p0 + pc]
            feature, prediction = self.layers[0](lo)
            alpha = (prediction[:, 0] + 1) / 2
            lows.append((alpha * lo[:, 0] + (1 - alpha) * lo[:, 1]).unsqueeze(1))          # phase_net.py:114-116
            for idx in range(m):
                l = L - 1 - idx                                                            # coarsest level first
                ph, am = vals.phase[l], vals.amplitude[l]
                h, w = int(ph.shape[2]), int(ph.shape[3])
                cf, cp, cv = feature.shape[1], prediction.shape[1], 2 * nb
                i = idx + 1 if idx + 1 < len(self.layers) - 1 else len(self.layers) - 1
                if tc.fuse_upsample and cf % 32 == 0:
                    # cat(interpolate(feature), values, interpolate(prediction)) is never built: the value channels and the resampled
                    # prediction go into a compact [.., 24] record, the 64 feature channels are resampled by the loaders of the
                    # level's first convolution
                    cd = (2 * cv + cp + 7) // 8 * 8
                    direct = torch.empty((pc, cd, h, w), dtype=torch.float32, device=dev, memory_format=torch.channels_last)
                    if cd != 2 * cv + cp:
                        direct.zero_()                                                     # padding channels must be finite
                    with torch.cuda.device(dev):
                        _lib.check(lib.fvfi_phasenet_assemble_offset(ph.data_ptr(), am.data_ptr(), den[l].data_ptr(), direct.data_ptr(),
                                                                     direct.stride(3), N, P, q, p0, pc, nb, h, w, _lib.stream_ptr()))
                    tc.resize_bilinear(prediction, (h, w), False, out=direct, out_channel_offset=2 * cv)
                    feature, prediction = self.layers[i].forward_resampled(feature, direct, (h, w))
                    del direct
                else:
                    concat = torch.empty((pc, cf + 2 * cv + cp, h, w), dtype=torch.float32, device=dev,
                                         memory_format=torch.channels_last)
                    tc.resize_bilinear(feature, (h, w), False, out=concat, out_channel_offset=0)
                    with torch.cuda.device(dev):
                        _lib.check(lib.fvfi_phasenet_assemble_offset(ph.data_ptr(), am.data_ptr(), den[l].data_ptr(),
                                                                     concat.data_ptr() + 4 * cf, concat.stride(3), N, P, q, p0, pc, nb,
                                                                     h, w, _lib.stream_ptr()))
                    tc.resize_bilinear(prediction, (h, w), False, out=concat, out_channel_offset=cf + 2 * cv)
                    feature, prediction = self.layers[i](concat)
                    del concat
                pr = tc.to_nhwc(prediction)
                with torch.cuda.device(dev):
                    _lib.check(lib.fvfi_phasenet_outputs_offset(pr.data_ptr(), pr.stride(3), am.data_ptr(), phase_out[l].data_ptr(),
                                                                amp_out[l].data_ptr(), N, P, q, p0, pc, nb, h, w, _lib.stream_ptr()))
        low_level = (lows[0] if len(lows) == 1 else torch.cat(lows, 0)) * self.max_low_level.view(-1, 1, 1, 1)
        H, W = int(vals.phase[0].shape[2]), int(vals.phase[0].shape[3])
        high_level = torch.zeros((1,), dtype=torch.float32, device=dev).expand(P, 1, H, W)  # zeros (phase_net.py:127-128), no storage
        return DecompValues(high_level=high_level, low_level=low_level, amplitude=amp_out, phase=phase_out)

    @tc.range_checked
    def forward(self, vals, m=None):
        """phase_net.py:107-177."""
        if m is None:
            m = self.pyr.height - 2
        P = vals.low_level.shape[0]
        chunk = self.plane_chunk or P
        lows, phs, ams = [], [[] for _ in range(m)], [[] for _ in range(m)]
        for p0 in range(0, P, chunk):
            sl = slice(p0, min(P, p0 + chunk))
            low, ph, am = self._forward_planes(vals.low_level[sl], [x[sl] for x in vals.phase[:m]],
                                               [x[sl] for x in vals.amplitude[:m]], m)
            lows.append(low)
            for i in range(m):
                phs[i].append(ph[i])
                ams[i].append(am[i])
        cat = lambda xs: xs[0] if len(xs) == 1 else torch.cat(xs, 0)
        hl = vals.high_level.shape
        high_level = torch.zeros((hl[0], 1, hl[2], hl[3]), device=vals.low_level.device)   # phase_net.py:127-128
        return self.reverse_normalize(DecompValues(high_level=high_level, low_level=cat(lows),
                                                   phase=[cat(x) for x in phs], amplitude=[cat(x) for x in ams]), m)
