"""Drop-in for the reference's ``src/fusion_net/fusion_net.py`` (FusionNet).

Same constructor, parameter names (``net.*`` dead weights kept for state-dict compatibility,
``encoder_layers.*``, ``bottleneck_layer.*``, ``decoder_layers.*``) and ``forward(base, adacof, phase,
other, maps, save=False, variant=0)``.  The final ``tanh -> base + res -> clamp(0,1)``
(fusion_net.py:67-77) is one fused CUDA kernel (fvfi_fusion_blend), differentiable through
fvfi_fusion_blend_backward (training step, SURVEY.md config 5).
"""
import torch
import torch.nn as nn

from . import _lib, transform
from . import conv as tc


def fusion_blend(base, x):
    """clamp(base + tanh(x), 0, 1) -- fusion_net.py:67-77 (differentiable: fvfi_fusion_blend_backward)."""
    if torch.is_grad_enabled() and (x.requires_grad or base.requires_grad):
        return _FusionBlend.apply(base, x)
    base = base.contiguous()
    x = x.contiguous()
    out = torch.empty_like(base)
    with torch.cuda.device(base.device):
        _lib.check(_lib.lib().fvfi_fusion_blend(base.data_ptr(), x.data_ptr(), out.data_ptr(), base.numel(),
                                                _lib.stream_ptr()))
    return out


def fusion_blend_rgb8(base, x, out=None):
    """The 8-bit form of ``fusion_blend``: planar [B,3,H,W] in, interleaved rgb24 [B,H,W,3] uint8 out,
    rint(clamp(base + tanh(x), 0, 1) * 255) (ties to even); the fp32 frame is never stored (fvfi_fusion_blend_rgb8)."""
    base = base.contiguous()
    x = x.contiguous()
    B, C, H, W = base.shape
    assert C == 3 and x.shape == base.shape
    if out is None:
        out = torch.empty((B, H, W, 3), dtype=torch.uint8, device=base.device)
    assert out.dtype == torch.uint8 and out.shape == (B, H, W, 3) and out.is_contiguous()
    with torch.cuda.device(base.device):
        _lib.check(_lib.lib().fvfi_fusion_blend_rgb8(base.data_ptr(), x.data_ptr(), out.data_ptr(), B, H, W, _lib.stream_ptr()))
    return out


def fusion_blend_yuv420p(base, x, out=None, matrix="bt709", full_range=False):
    """The yuv420p form of ``fusion_blend``: planar [B,3,H,W] in (H, W even), 8-bit planar I420 [B,3H/2,W] uint8 out (Y [H,W],
    then U and V [H/2,W/2] per frame): Y per pixel and Cb / Cr of every 2x2 block's mean of clamp(base + tanh(x), 0, 1), with
    ``matrix`` 'bt709' or 'bt601' and limited or ``full_range``; the fp32 frame is never stored (fvfi_fusion_blend_yuv420p)."""
    mat, full = transform.yuv_args(matrix, full_range)
    base = base.contiguous()
    x = x.contiguous()
    B, C, H, W = base.shape
    assert C == 3 and x.shape == base.shape
    if out is None:
        out = torch.empty((B, 3 * H // 2, W), dtype=torch.uint8, device=base.device)
    assert out.dtype == torch.uint8 and out.shape == (B, 3 * H // 2, W) and out.is_contiguous()
    with torch.cuda.device(base.device):
        _lib.check(_lib.lib().fvfi_fusion_blend_yuv420p(base.data_ptr(), x.data_ptr(), out.data_ptr(), B, H, W, mat, full,
                                                        _lib.stream_ptr()))
    return out


class _FusionBlend(torch.autograd.Function):
    @staticmethod
    def forward(ctx, base, x):
        base, x = base.detach().contiguous().float(), x.detach().contiguous().float()
        ctx.save_for_backward(base, x)
        with torch.no_grad():
            return fusion_blend(base, x)

    @staticmethod
    def backward(ctx, gout):
        base, x = ctx.saved_tensors
        g = gout.detach().contiguous().float()
        gx = torch.empty_like(x)
        gbase = torch.empty_like(base) if ctx.needs_input_grad[0] else None
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().fvfi_fusion_blend_backward(base.data_ptr(), x.data_ptr(), g.data_ptr(), gx.data_ptr(),
                                                             _lib.ptr(gbase), x.numel(), _lib.stream_ptr()))
        return gbase, gx


class FusionNet(torch.nn.Module):

    def __init__(self, num_imgs=5, uncertainty_maps=3, kernel=3, pad=3, dil=3):
        super(FusionNet, self).__init__()
        # never used in forward (fusion_net.py:11-20 vs :46-77) -- kept so fusion_net.pt loads unchanged
        self.net = nn.Sequential(
            nn.Conv2d(3 * num_imgs + uncertainty_maps, 64, kernel_size=kernel, stride=1, padding=pad, dilation=dil),
            nn.ReLU(),
            nn.Conv2d(64, 64, kernel_size=kernel, stride=1, padding=pad, dilation=dil),
            nn.ReLU(),
            nn.Conv2d(64, 64, kernel_size=kernel, stride=1, padding=pad, dilation=dil),
            nn.ReLU(),
            nn.Conv2d(64, 3, kernel_size=kernel, stride=1, padding=pad, dilation=dil),
            nn.Tanh()
        )
        input_channels = 3 * num_imgs + uncertainty_maps
        self.encoder_layers = nn.ModuleList([
            nn.Conv2d(input_channels, 32, kernel_size=5, stride=1, padding=2, padding_mode='reflect'),
            nn.Conv2d(32, 64, kernel_size=5, stride=1, padding=2, padding_mode='reflect'),
            nn.Conv2d(64, 128, kernel_size=3, stride=1, padding=1, padding_mode='reflect')
        ])
        self.bottleneck_layer = nn.Conv2d(128, 128, kernel_size=3, stride=1, padding=1, padding_mode='reflect')
        self.decoder_layers = nn.ModuleList([
            nn.Conv2d(128, 64, kernel_size=5, stride=1, padding=2, padding_mode='reflect'),
            nn.Conv2d(64, 32, kernel_size=5, stride=1, padding=2, padding_mode='reflect'),
            nn.Conv2d(32, 3, kernel_size=1, stride=1),
        ])
        self.relu = nn.ReLU()
        self.tanh = nn.Tanh()
        self.max_pool = nn.MaxPool2d(2, stride=2)
        self.deconvolution = nn.Upsample(scale_factor=2, mode='bilinear')
        self.residuals = []

    def live_parameters(self):
        """Parameters that receive gradients (everything except the dead ``net.*``); the training
        all-reduce bucket is built from these (SURVEY.md 8(e))."""
        return [p for n, p in self.named_parameters() if not n.startswith("net.")]

    @tc.range_checked
    def forward(self, base, adacof, phase, other, maps, save=False, variant=0):
        """fusion_net.py:46-77.  ONE path for inference and training: every convolution (+ its ReLU) is one tcgen05 kernel, pooling,
        ``Upsample(ReLU(x)) + skip`` and the final ``clamp(base + tanh)`` are the fused NHWC kernels; under autograd each of them is
        an autograd Function whose backward is a libfvfi kernel too (csrc/conv_bwd.cu) -- no ATen convolution / pooling /
        interpolation kernel runs in the training step of the trained network."""
        x = self.residual(base, adacof, phase, other, maps)
        anchor = phase if variant == 1 else base
        if save:
            self.residuals.append(torch.sum(torch.tanh(x.detach())).cpu().item())
        return fusion_blend(anchor, x)

    @tc.range_checked
    def residual(self, base, adacof, phase, other, maps):
        """The body of ``forward`` up to the pre-tanh residual x [B,3,H,W] (planar, contiguous): ``forward`` returns
        ``fusion_blend(base, x)``; a caller that wants 8-bit frames ends with ``fusion_blend_rgb8(base, x)`` instead."""
        parts = [base, adacof, phase, other, maps]
        if not all(t.is_cuda for t in parts):
            raise NotImplementedError("fvfi FusionNet runs on CUDA tensors only (no CPU fallback)")
        grad = torch.is_grad_enabled() and (any(t.requires_grad for t in parts) or any(p.requires_grad for p in self.live_parameters()))
        skip = []
        if grad or sum(int(t.shape[1]) for t in parts) > 32:
            x = torch.cat(parts, 1)
            if x.shape[1] % 4:             # zero channels up to a multiple of 4: the weight-gradient kernel then reads float4 pixel quads
                x = nn.functional.pad(x, (0, 0, 0, 0, 0, 4 - x.shape[1] % 4))
            x = tc.to_nhwc(x)
        else:                              # the concatenation written NHWC (18 -> 20 channels) by one kernel: no planar cat, no transposing copy
            x = tc.planar_concat_nhwc(parts)
        for layer in self.encoder_layers:
            x = tc.conv_module(layer, x, "relu")                          # fusion_net.py:52-56
            skip.append(x)
            x = tc.max_pool2(x)
        x = tc.conv_module(self.bottleneck_layer, x, "relu")              # the ReLU of the first decoder step folded in (:58-61)
        for i, (layer, s) in enumerate(zip(self.decoder_layers, skip[::-1])):
            # Upsample(ReLU(x)) + skip as one pass (fvfi_resize_bilinear_nhwc_fused)
            x = tc.resize_bilinear(x, (x.shape[2] * 2, x.shape[3] * 2), False, relu_input=i > 0, add=s)
            x = tc.conv_module(layer, x, None)
        return x.contiguous()
