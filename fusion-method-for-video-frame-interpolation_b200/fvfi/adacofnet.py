"""Drop-in for the reference's ``src/fusion_net/fusion_adacofnet.py`` (KernelEstimation, AdaCoFNet,
make_model) -- the AdaCoFNet variant the fusion pipeline uses (returns 4 tensors).

``AdaCoFNet(args)`` takes ``args.kernel_size``, ``args.dilation``, ``args.gpu_id``;
``forward(frame0, frame2) -> (tensorAdaCoF1, tensorAdaCoF2, frame1, UncertaintyMask)``.
Parameter names (``get_kernel.module*``) match the reference so its checkpoints load.  Lines
195-213 of the reference (two warps, occlusion blend, flow mean/variance, clip/20) run as ONE fused
kernel in inference (fvfi_adacofnet_warp_blend); with autograd enabled the op-level
``FunctionAdaCoF`` is used so gradients reach the kernel-estimation network.
"""
import sys

import torch
from torch.nn import functional as F

from . import adacof
from . import conv as tc


def moduleNormalize(frame):
    """src/adacof/utility.py:86-87."""
    mean = torch.tensor([0.4631, 0.4352, 0.3990], dtype=frame.dtype, device=frame.device).view(1, 3, 1, 1)
    return frame - mean


def make_model(args):
    return AdaCoFNet(args).to(torch.device('cuda:{}'.format(args.gpu_id)))


class KernelEstimation(torch.nn.Module):
    """fusion_adacofnet.py:14-155 (same submodule names and creation order)."""

    def __init__(self, kernel_size):
        super(KernelEstimation, self).__init__()
        self.kernel_size = kernel_size
        nn = torch.nn

        def Basic(ci, co):
            return nn.Sequential(
                nn.Conv2d(ci, co, 3, 1, 1), nn.ReLU(inplace=False),
                nn.Conv2d(co, co, 3, 1, 1), nn.ReLU(inplace=False),
                nn.Conv2d(co, co, 3, 1, 1), nn.ReLU(inplace=False))

        def Upsample(c):
            return nn.Sequential(
                nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True),
                nn.Conv2d(c, c, 3, 1, 1), nn.ReLU(inplace=False))

        def Subnet(ks, tail=None, last_in=None):
            layers = [
                nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(inplace=False),
                nn.Conv2d(64, 64, 3, 1, 1), nn.ReLU(inplace=False),
                nn.Conv2d(64, ks if last_in is None else last_in, 3, 1, 1), nn.ReLU(inplace=False),
                nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True),
                nn.Conv2d(ks if last_in is None else last_in, ks, 3, 1, 1)]
            if tail is not None:
                layers.append(tail)
            return nn.Sequential(*layers)

        ks2 = self.kernel_size ** 2
        self.moduleConv1 = Basic(6, 32)
        self.modulePool1 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.moduleConv2 = Basic(32, 64)
        self.modulePool2 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.moduleConv3 = Basic(64, 128)
        self.modulePool3 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.moduleConv4 = Basic(128, 256)
        self.modulePool4 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.moduleConv5 = Basic(256, 512)
        self.modulePool5 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.moduleDeconv5 = Basic(512, 512)
        self.moduleUpsample5 = Upsample(512)
        self.moduleDeconv4 = Basic(512, 256)
        self.moduleUpsample4 = Upsample(256)
        self.moduleDeconv3 = Basic(256, 128)
        self.moduleUpsample3 = Upsample(128)
        self.moduleDeconv2 = Basic(128, 64)
        self.moduleUpsample2 = Upsample(64)
        self.moduleWeight1 = Subnet(ks2, nn.Softmax(dim=1))
        self.moduleAlpha1 = Subnet(ks2)
        self.moduleBeta1 = Subnet(ks2)
        self.moduleWeight2 = Subnet(ks2, nn.Softmax(dim=1))
        self.moduleAlpha2 = Subnet(ks2)
        self.moduleBeta2 = Subnet(ks2)
        self.moduleOcclusion = Subnet(1, nn.Sigmoid(), last_in=64)

    @staticmethod
    def _seq_tc(seq, x, nchw_last=False, residual=None):
        """Run an nn.Sequential of Conv2d / ReLU / Upsample / Softmax / Sigmoid: conv + activation is one tcgen05 kernel,
        bilinear upsampling is the NHWC resize kernel; with ``nchw_last`` the final conv writes planar NCHW."""
        mods = list(seq)
        last_conv = max(i for i, m in enumerate(mods) if isinstance(m, torch.nn.Conv2d))
        i = 0
        up = None                      # pending Upsample: evaluated by the loaders of the convolution that follows it
        while i < len(mods):
            m = mods[i]
            if isinstance(m, torch.nn.Conv2d):
                nxt = mods[i + 1] if i + 1 < len(mods) else None
                act = {torch.nn.ReLU: "relu", torch.nn.Sigmoid: "sigmoid", torch.nn.Softmax: "softmax"}.get(type(nxt))
                # a conv feeding an Upsample keeps its channels padded to 16 (zeros): resize and the next conv then
                # use 16-byte accesses even for the 25-channel heads
                pad = (i + 2 < len(mods) and isinstance(mods[i + 2], torch.nn.Upsample) and m.out_channels % 4 != 0)
                x = tc.conv_module(m, x, act, nchw_out=nchw_last and i == last_conv, pad_out=pad,
                                   residual=residual if i == last_conv else None,   # skip connection after the last conv + act
                                   upsample=up)
                up = None
                i += 2 if act else 1
            elif (isinstance(m, torch.nn.Upsample) and i + 1 == last_conv and mods[last_conv].out_channels == 1
                  and m.scale_factor == 2 and m.mode == 'bilinear' and m.align_corners):
                # occlusion head: Upsample -> Conv2d(64, 1, 3) -> Sigmoid with the channels contracted before upsampling
                nxt = mods[i + 2] if i + 2 < len(mods) else None
                act = {torch.nn.ReLU: "relu", torch.nn.Sigmoid: "sigmoid"}.get(type(nxt))
                x = tc.upsample2_conv3x3_single(mods[last_conv], x, act)
                i += 3 if act else 2
            elif isinstance(m, torch.nn.Upsample):
                size = (x.shape[2] * 2, x.shape[3] * 2)
                if (m.mode == 'bilinear' and m.scale_factor == 2 and i + 1 < len(mods)
                        and isinstance(mods[i + 1], torch.nn.Conv2d) and mods[i + 1].kernel_size[0] > 1):
                    up = (size, bool(m.align_corners))      # Upsample -> Conv2d: one kernel (fvfi_conv2d_nhwc_upsampled)
                else:
                    x = tc.resize_bilinear(x, size, bool(m.align_corners))
                i += 1
            else:
                x = m(x)
                i += 1
        return x

    def _forward_tc(self, rfield0, rfield2):
        """tcgen05 path of fusion_adacofnet.py:109-155: every conv(+ReLU/sigmoid) is one fused kernel, the
        pooling / bilinear upsampling / softmax run on NHWC tensors, the seven heads are returned NCHW-contiguous
        (the warp kernel streams each coefficient plane)."""
        # 6 input channels padded to 8 (zeros): 16-byte loads in the first convolution
        x = tc.to_nhwc(torch.cat([rfield0, rfield2, rfield0.new_zeros((rfield0.shape[0], 2) + tuple(rfield0.shape[2:]))], 1))
        return self._forward_tc_x(x)

    def _forward_tc_x(self, x):
        """``x``: [B,8,H,W] channels_last = (frame0 - mean | frame2 - mean | two zero channels)."""
        run = self._seq_tc
        pool = tc.avg_pool2                    # modulePool1..5 = AvgPool2d(2, 2), on NHWC with 256-bit accesses
        c1 = run(self.moduleConv1, x)
        c2 = run(self.moduleConv2, pool(c1))
        del c1
        c3 = run(self.moduleConv3, pool(c2))
        c4 = run(self.moduleConv4, pool(c3))
        c5 = run(self.moduleConv5, pool(c4))
        # the skip additions (fusion_adacofnet.py:128-138) ride on the epilogue of the Upsample modules' convolution
        s5 = run(self.moduleUpsample5, run(self.moduleDeconv5, pool(c5)), residual=c5)      # d5 + c5
        s4 = run(self.moduleUpsample4, run(self.moduleDeconv4, s5), residual=c4)            # d4 + c4
        s3 = run(self.moduleUpsample3, run(self.moduleDeconv3, s4), residual=c3)            # d3 + c3
        comb = run(self.moduleUpsample2, run(self.moduleDeconv2, s3), residual=c2)          # d2 + c2
        heads = (self.moduleWeight1, self.moduleAlpha1, self.moduleBeta1, self.moduleWeight2, self.moduleAlpha2,
                 self.moduleBeta2, self.moduleOcclusion)
        # the seven heads start with a 64 -> 64 convolution of the SAME tensor: one 64 -> 448 convolution (N = 256 + 192
        # per tensor-core tile instead of 64, the input staged once instead of seven times); each head continues on its
        # 64-channel slice of the result
        first = self._fused_first(heads)
        y = tc.conv2d(comb, first[0], first[1], "zeros", "relu")
        return tuple(run(torch.nn.Sequential(*list(h)[2:]), y[:, 64 * i:64 * (i + 1)], nchw_last=True)
                     for i, h in enumerate(heads))

    def _fused_first(self, heads):
        """Concatenated weights / biases of the heads' first convolutions, rebuilt when any of them changes."""
        key = tuple((h[0].weight.data_ptr(), h[0].weight._version, h[0].bias._version) for h in heads)
        hit = getattr(self, "_first_cache", None)
        if hit is None or hit[0] != key:
            w = torch.cat([h[0].weight.detach() for h in heads], 0).contiguous()
            b = torch.cat([h[0].bias.detach() for h in heads], 0).contiguous()
            hit = (key, (w, b))
            self._first_cache = hit
        return hit[1]

    @staticmethod
    def _seq_train(seq, x):
        """The same nn.Sequential under autograd: every step is an autograd Function over libfvfi kernels (conv + activation:
        conv._ConvTC, tcgen05 forward and data gradient, csrc/conv_bwd.cu weight / bias gradients; Upsample: conv._ResizeFused);
        only the channel softmax is torch's."""
        mods = list(seq)
        i = 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, torch.nn.Conv2d):
                nxt = mods[i + 1] if i + 1 < len(mods) else None
                act = {torch.nn.ReLU: "relu", torch.nn.Sigmoid: "sigmoid"}.get(type(nxt))
                x = tc.conv_module(m, x, act)
                i += 2 if act else 1
            elif isinstance(m, torch.nn.Upsample):
                assert m.mode == 'bilinear' and m.scale_factor == 2
                x = tc.resize_bilinear(x, (x.shape[2] * 2, x.shape[3] * 2), bool(m.align_corners))
                i += 1
            else:
                x = m(x)
                i += 1
        return x

    def _forward_train(self, rfield0, rfield2):
        """fusion_adacofnet.py:109-155 with gradients: the differentiable counterpart of ``_forward_tc`` (no fused epilogues /
        loaders, one libfvfi autograd Function per module)."""
        x = tc.to_nhwc(torch.cat([rfield0, rfield2, rfield0.new_zeros((rfield0.shape[0], 2) + tuple(rfield0.shape[2:]))], 1))
        run, pool = self._seq_train, tc.avg_pool2
        c1 = run(self.moduleConv1, x)
        c2 = run(self.moduleConv2, pool(c1))
        c3 = run(self.moduleConv3, pool(c2))
        c4 = run(self.moduleConv4, pool(c3))
        c5 = run(self.moduleConv5, pool(c4))
        d5 = run(self.moduleUpsample5, run(self.moduleDeconv5, pool(c5)))
        d4 = run(self.moduleUpsample4, run(self.moduleDeconv4, d5 + c5))
        d3 = run(self.moduleUpsample3, run(self.moduleDeconv3, d4 + c4))
        d2 = run(self.moduleUpsample2, run(self.moduleDeconv2, d3 + c3))
        comb = d2 + c2
        return tuple(run(h, comb) for h in (self.moduleWeight1, self.moduleAlpha1, self.moduleBeta1, self.moduleWeight2,
                                            self.moduleAlpha2, self.moduleBeta2, self.moduleOcclusion))

    @tc.range_checked
    def forward(self, rfield0, rfield2):
        if not rfield0.is_cuda:
            raise NotImplementedError("fvfi KernelEstimation runs on CUDA tensors only (no CPU fallback)")
        grad = torch.is_grad_enabled() and (rfield0.requires_grad or rfield2.requires_grad
                                            or any(p.requires_grad for p in self.parameters()))
        return self._forward_train(rfield0, rfield2) if grad else self._forward_tc(rfield0, rfield2)


class AdaCoFNet(torch.nn.Module):
    """fusion_adacofnet.py:158-240."""

    def __init__(self, args):
        super(AdaCoFNet, self).__init__()
        self.args = args
        self.kernel_size = args.kernel_size
        self.kernel_pad = int(((args.kernel_size - 1) * args.dilation) / 2.0)
        self.dilation = args.dilation
        self.get_kernel = KernelEstimation(self.kernel_size)
        self.modulePad = torch.nn.ReplicationPad2d([self.kernel_pad] * 4)
        self.moduleAdaCoF = adacof.FunctionAdaCoF.apply

    def _forward_fused_prep(self, frame0, frame2, return_warped, want_mask=True):
        """Inference form of lines 176-213: reflect pad / normalise / concat / NHWC and the replicate pad in ONE kernel
        (fvfi_adacofnet_prep), kernel estimation, fused two-warp synthesis."""
        import ctypes
        from . import _lib
        B, _, h0, w0 = frame0.shape
        hp, wp = (h0 + 31) // 32 * 32, (w0 + 31) // 32 * 32
        k = self.kernel_pad
        f0, f2 = frame0.contiguous(), frame2.contiguous()
        x = torch.empty((B, 8, hp, wp), dtype=torch.float32, device=f0.device, memory_format=torch.channels_last)
        p0 = torch.empty((B, 3, hp + 2 * k, wp + 2 * k), dtype=torch.float32, device=f0.device)
        p2 = torch.empty_like(p0)
        mean = (ctypes.c_float * 3)(0.4631, 0.4352, 0.3990)                           # src/adacof/utility.py:86-87
        with torch.cuda.device(f0.device):
            _lib.check(_lib.lib().fvfi_adacofnet_prep(f0.data_ptr(), f2.data_ptr(), x.data_ptr(), p0.data_ptr(), p2.data_ptr(),
                                                      B, h0, w0, hp, wp, k, ctypes.cast(mean, ctypes.c_void_p),
                                                      _lib.stream_ptr()))
        W1, A1, B1, W2, A2, B2, Occ = self.get_kernel._forward_tc_x(x)
        if not return_warped and wp == w0 and hp != h0:
            # only rows were padded: the kernel writes the h0 rows of the result directly (no crop copies)
            r = adacof.adacofnet_warp_blend_rows(p0, p2, W1.contiguous(), A1.contiguous(), B1.contiguous(), W2.contiguous(),
                                                 A2.contiguous(), B2.contiguous(), Occ.contiguous(), self.dilation, h0, want_mask)
            if r is not None:
                return None, None, r[0], r[1]
        t1, t2, frame1, mask = adacof.adacofnet_warp_blend(p0, p2, W1.contiguous(), A1.contiguous(), B1.contiguous(),
                                                           W2.contiguous(), A2.contiguous(), B2.contiguous(),
                                                           Occ.contiguous(), self.dilation, want_t=return_warped)
        if hp != h0 or wp != w0:
            if t1 is not None:
                t1, t2 = t1[:, :, :h0, :w0], t2[:, :, :h0, :w0]
            frame1, mask = frame1[:, :, :h0, :w0].contiguous(), mask[:, :, :h0, :w0].contiguous()
        return t1, t2, frame1, mask

    def load(self, state_dict):
        """The reference wraps models in src/adacof/models/__init__.py:Model whose ``load`` forwards here."""
        self.load_state_dict(state_dict)

    @tc.range_checked
    def forward(self, frame0, frame2, return_warped=True, want_mask=True):
        """fusion_adacofnet.py:172-240.  ``return_warped=False`` / ``want_mask=False`` (extensions, default = the reference's four
        outputs): the two warped frames / the uncertainty mask are returned as None and not computed."""
        h0, w0 = int(frame0.shape[2]), int(frame0.shape[3])
        if h0 != int(frame2.shape[2]) or w0 != int(frame2.shape[3]):
            sys.exit('Frame sizes do not match')                                   # fusion_adacofnet.py:177-178
        if (tc.use_tc(frame0) and not self.training and frame0.shape[1] == 3 and frame0.dtype == torch.float32
                and not (frame0.requires_grad or frame2.requires_grad)):
            return self._forward_fused_prep(frame0, frame2, return_warped, want_mask)
        if h0 % 32 != 0:
            pad_h = 32 - (h0 % 32)
            frame0 = F.pad(frame0, (0, 0, 0, pad_h), mode='reflect')
            frame2 = F.pad(frame2, (0, 0, 0, pad_h), mode='reflect')
        if w0 % 32 != 0:
            pad_w = 32 - (w0 % 32)
            frame0 = F.pad(frame0, (0, pad_w, 0, 0), mode='reflect')
            frame2 = F.pad(frame2, (0, pad_w, 0, 0), mode='reflect')
        W1, A1, B1, W2, A2, B2, Occ = self.get_kernel(moduleNormalize(frame0), moduleNormalize(frame2))
        p0, p2 = self.modulePad(frame0).contiguous(), self.modulePad(frame2).contiguous()
        needs_grad = torch.is_grad_enabled() and any(t.requires_grad for t in (W1, A1, B1, W2, A2, B2, Occ, p0, p2))
        if needs_grad:
            t1 = self.moduleAdaCoF(p0, W1.contiguous(), A1.contiguous(), B1.contiguous(), self.dilation)
            t2 = self.moduleAdaCoF(p2, W2.contiguous(), A2.contiguous(), B2.contiguous(), self.dilation)
            frame1 = Occ * t1 + (1 - Occ) * t2                                       # fusion_adacofnet.py:198
            with torch.no_grad():                                                    # .detach() at :211
                _, mask = adacof.adacofnet_tail(t1.detach(), t2.detach(), Occ.detach().contiguous(),
                                                W1.detach().contiguous(), A1.detach().contiguous(),
                                                B1.detach().contiguous(), W2.detach().contiguous(),
                                                A2.detach().contiguous(), B2.detach().contiguous())
        else:
            t1, t2, frame1, mask = adacof.adacofnet_warp_blend(p0, p2, W1.contiguous(), A1.contiguous(), B1.contiguous(),
                                                               W2.contiguous(), A2.contiguous(), B2.contiguous(),
                                                               Occ.contiguous(), self.dilation, want_t=return_warped)
        if h0 != frame1.shape[2] or w0 != frame1.shape[3]:
            # crop back; NB the reference returns tensorAdaCoF2 as tensorAdaCoF1 when the width was padded
            # (fusion_adacofnet.py:225) -- fixed here, frame1/mask are unaffected.
            if t1 is not None:
                t1, t2 = t1[:, :, :h0, :w0], t2[:, :, :h0, :w0]
            frame1, mask = frame1[:, :, :h0, :w0].contiguous(), mask[:, :, :h0, :w0].contiguous()
        return t1, t2, frame1, mask
