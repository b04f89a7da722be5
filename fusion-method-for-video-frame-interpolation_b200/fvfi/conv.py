"""Tensor-core convolution op (C-ABI: fvfi_conv2d_* in include/fvfi.h): stride-1 "same" convolutions of
the three networks on tcgen05 with split-operand error compensation (3xFP16 default / 3xTF32; fp32-grade results), NHWC activations
(torch ``channels_last``), fused bias + activation.

``conv_module(conv, x, act)`` runs an ``nn.Conv2d`` (weights stay in the module, so reference checkpoints load
unchanged) through the kernel; packed weights are cached per weight version.  Also here: the NHWC helpers around
the convolutions (bilinear resize, 2x2 average pool, planar -> NHWC slice).
"""
import os

import torch

from . import _lib

PRECISIONS = {"tf32x3": 0, "f16x3": 1}
precision = PRECISIONS[os.environ.get("FVFI_CONV_PREC", "f16x3")]   # operand split (include/fvfi.h: FVFI_CONV_*)
range_check = True   # range_checked() forwards verify the 3xFP16 range flag and re-run in 3xTF32 when it was raised
_guard_depth = 0


def overflow_pending():
    """True if a 3xFP16 convolution enqueued on the current stream since the last check saw an activation outside the
    representable range (|x| * 2^4 > 65504).  Synchronises the current stream and clears the flag."""
    import torch as _t
    _t.cuda.current_stream().synchronize()
    return _lib.lib().fvfi_conv2d_overflow_count() > 0


def check_overflow():
    """Raise if a convolution since the last check left the 3xFP16 range (for callers that run the convolutions directly,
    outside the range_checked() module forwards)."""
    if precision == PRECISIONS["f16x3"] and overflow_pending():
        raise FloatingPointError("fvfi.conv: activation beyond the 3xFP16 range (|x| > 4094); use conv.forced_precision('tf32x3')")


class forced_precision:
    """``with forced_precision('tf32x3'):`` -- run the enclosed convolutions with the given operand split."""

    def __init__(self, name):
        self.value = PRECISIONS[name]

    def __enter__(self):
        global precision
        self.old, precision = precision, self.value
        return self

    def __exit__(self, *exc):
        global precision
        precision = self.old


def range_checked(fn):
    """Decorator of the inference entry points (FusionPipeline.forward / fusion_inputs, AdaCoFNet.forward, PhaseNet.forward /
    forward_fused, FusionNet.forward).  The default operand split (3xFP16) represents activations up to |x| = 4094; a kernel that
    meets a larger value raises a device flag instead of saturating.  The OUTERMOST decorated call reads the flag when its work
    is enqueued (one stream synchronisation per call) and, if it was raised, runs the whole call again with the range-unlimited
    3xTF32 split -- the caller never sees an out-of-range result and never has to choose a precision."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        global _guard_depth
        if (_guard_depth > 0 or not range_check or precision != PRECISIONS["f16x3"] or torch.is_grad_enabled()
                or not torch.cuda.is_available() or torch.cuda.is_current_stream_capturing()):
            return fn(*args, **kwargs)
        _guard_depth += 1
        try:
            out = fn(*args, **kwargs)
            if overflow_pending():
                with forced_precision("tf32x3"):
                    out = fn(*args, **kwargs)
        finally:
            _guard_depth -= 1
        return out
    return wrapper


def use_tc(x):
    """The fused inference forwards of the drop-in modules apply to CUDA tensors with autograd off.  (With autograd on, the modules
    run their step-by-step torch graph; FusionNet -- the network the fusion recipe trains -- still takes its convolutions from the
    tensor-core kernel there through ``conv2d``'s autograd Function.)"""
    return x.is_cuda and not torch.is_grad_enabled()


class _ConvTC(torch.autograd.Function):
    """act(conv(pad(x), w) + b), forward AND backward on libfvfi (no cuDNN / ATen convolution on the training path):
    forward = the tcgen05 kernel, activations saved; backward (csrc/conv_bwd.cu, include/fvfi.h "Backward of the same convolutions"):
    ``fvfi_conv2d_grad_act`` (g = gy * act'(y) into a zero canvas + bias gradient), the data gradient as the tcgen05 kernel run
    over that canvas with the flipped / transposed filter in 3xTF32 (+ ``fvfi_reflect_pad_backward_nhwc``), and
    ``fvfi_conv2d_wgrad_nhwc`` (pixel-split fp32 GEMM, fixed summation order).  Replaces what the reference gets from
    torch.nn.Conv2d's autograd in src/fusion_net/trainer.py:246-259."""

    @staticmethod
    def forward(ctx, x, weight, bias, padding_mode, act):
        y = conv2d(x.detach(), weight.detach(), None if bias is None else bias.detach(), padding_mode, act)
        ctx.save_for_backward(x, weight, y)
        ctx.has_bias, ctx.padding_mode, ctx.act = bias is not None, padding_mode, act
        return y

    @staticmethod
    def backward(ctx, gy):
        x, weight, y = ctx.saved_tensors
        assert ctx.act in (None, "none", "relu", "elu", "tanh", "sigmoid"), "no backward for activation %r" % (ctx.act,)
        Cout, Cin, K, _ = weight.shape
        B, Cx, H, W = x.shape
        P = K // 2
        reflect = ctx.padding_mode == "reflect" and P > 0
        need_x, need_w, need_b = ctx.needs_input_grad[0], ctx.needs_input_grad[1], ctx.has_bias and ctx.needs_input_grad[2]
        L, dev, f32 = _lib.lib(), x.device, torch.float32
        gyc, yc, xc = to_nhwc(gy.detach().float()), to_nhwc(y), to_nhwc(x.detach().float())
        border = P if (need_x and reflect) else 0          # the full correlation of the data gradient needs the zero frame
        Hc, Wc = H + 2 * border, W + 2 * border
        canvas = torch.empty((B, Cout, Hc, Wc), dtype=f32, device=dev, memory_format=torch.channels_last)
        gb = torch.empty(Cout, dtype=f32, device=dev) if need_b else None
        with torch.cuda.device(dev):
            ws = torch.empty(L.fvfi_conv2d_grad_act_workspace_floats(B, H, W, Cout, border), dtype=f32, device=dev) if need_b else None
            _lib.check(L.fvfi_conv2d_grad_act(gyc.data_ptr(), gyc.stride(3), yc.data_ptr(), yc.stride(3), canvas.data_ptr(), B, H, W,
                                              Cout, border, ACT[ctx.act], _lib.ptr(gb), _lib.ptr(ws), _lib.stream_ptr()))
            gw = None
            if need_w:
                gw = torch.empty((Cout, Cin, K, K), dtype=f32, device=dev)
                ws2 = torch.empty(L.fvfi_conv2d_wgrad_workspace_floats(B, H, W, Cin, Cout, K), dtype=f32, device=dev)
                _lib.check(L.fvfi_conv2d_wgrad_nhwc(xc.data_ptr(), xc.stride(3), canvas.data_ptr() + 4 * Cout * (border * Wc + border),
                                                    Cout, Wc, Hc * Wc, gw.data_ptr(), B, H, W, Cin, Cout, K, 1 if reflect else 0,
                                                    ws2.data_ptr(), _lib.stream_ptr()))
            gx = None
            if need_x:
                wt = weight.detach().float().flip(2, 3).transpose(0, 1).contiguous()       # [Cin, Cout, K, K], taps mirrored
                with torch.no_grad(), forced_precision("tf32x3"):
                    gxp = conv2d(canvas, wt, None, "zeros", None)                          # [B, Cin, Hc, Wc]
                if reflect:
                    gx = torch.empty((B, Cx, H, W), dtype=f32, device=dev, memory_format=torch.channels_last)
                    if Cx > Cin:
                        gx.zero_()
                    _lib.check(L.fvfi_reflect_pad_backward_nhwc(gxp.data_ptr(), gxp.stride(3), gx.data_ptr(), gx.stride(3), B, H, W,
                                                                Cin, P, _lib.stream_ptr()))
                else:
                    gx = gxp if Cx == Cin else torch.nn.functional.pad(gxp, (0, 0, 0, 0, 0, Cx - Cin))
        return gx, gw, gb, None, None


ACT = {None: 0, "none": 0, "relu": 1, "elu": 2, "tanh": 3, "sigmoid": 4, "softmax": 5}
timing = None    # set to a list to collect (flops, start_event, end_event) per convolution launch (bench.py roofline)


n_split = None   # tuning override (tools/tune_conv_split.py): output channels per launch for Cout > this value


def _split(Cout):
    """Output channels per launch (one launch holds at most 256: the TMEM accumulator is 512 columns)."""
    if n_split is not None and Cout > n_split:
        return n_split
    return 256


def _packed(weight):
    """Packed (hi|lo split, canonical tensor-core layout) copy of a weight tensor, per operand split.  The cache lives ON the
    tensor object (``weight._fvfi_pack``), so it dies with it -- folded / concatenated temporaries do not accumulate; it is
    rebuilt when the tensor's version counter or storage changes (optimizer steps and load_state_dict bump the version; edits
    through ``.data`` do not -- call ``invalidate(weight)`` after those)."""
    key = (weight.data_ptr(), weight._version, tuple(weight.shape), str(weight.device), _split(weight.shape[0]))
    cache = weight.__dict__.setdefault("_fvfi_pack", {})
    hit = cache.get(precision)
    if hit is not None and hit[0] == key:
        return hit[1]
    Cout, Cin, KH, KW = weight.shape
    L = _lib.lib()
    parts = []
    w = weight.detach().contiguous().float()
    step = _split(Cout)
    for o in range(0, Cout, step):
        wo = w[o:o + step].contiguous()
        n = L.fvfi_conv2d_packed_weight_floats(wo.shape[0], Cin, KH, KW, precision)
        buf = torch.empty(n, dtype=torch.float32, device=weight.device)
        with torch.cuda.device(weight.device):
            _lib.check(L.fvfi_conv2d_pack_weights(wo.data_ptr(), buf.data_ptr(), wo.shape[0], Cin, KH, KW, precision,
                                                  _lib.stream_ptr()))
        parts.append((o, wo.shape[0], buf))
    cache[precision] = (key, parts)
    return parts


def invalidate(obj):
    """Drop the cached packed / folded / tap-map weights of a tensor or module (after in-place edits through ``.data``)."""
    for k in ("_fvfi_pack", "_fvfi_fold", "_fvfi_taps", "_first_cache"):
        obj.__dict__.pop(k, None)
    if isinstance(obj, torch.nn.Module):
        for m in obj.children():
            invalidate(m)
        for p in obj.parameters(recurse=False):
            invalidate(p)


def to_nhwc(x):
    """NHWC storage of x; a channel slice of an NHWC tensor is used in place (pixel stride > C), anything else is copied."""
    if x.dim() == 4 and x.stride(1) == 1:
        B, C, H, W = x.shape
        ld = x.stride(3)
        if ld >= C and x.stride(2) == W * ld and (B == 1 or x.stride(0) == H * W * ld):
            return x
    return x.contiguous(memory_format=torch.channels_last)


def conv2d(x, weight, bias=None, padding_mode="zeros", act=None, out=None, nchw_out=False, pad_out=False, residual=None,
           upsample=None, x_direct=None):
    """x [B,Cin,H,W] (any memory format; channels_last avoids a copy) -> [B,Cout,H,W] channels_last
    (``nchw_out=True``: plain contiguous NCHW, written directly by the epilogue).
    Equivalent to act(F.conv2d(pad(x), weight, bias)) with 'same' padding (K//2) in zeros or reflect mode;
    act 'softmax' is over the channel dimension.
    ``residual`` (channels_last [B,Cout,H,W]): added after the activation in the epilogue (skip connection).
    ``pad_out=True``: the result has round16(Cout) channels, the extra ones zero (keeps 16-byte accesses for channel
    counts such as 25).  ``x`` may carry such zero padding channels beyond the weight's Cin.
    ``upsample=((H, W), align_corners)``: the convolution runs on the bilinear resampling of ``x`` to [H, W]
    (torch.nn.Upsample -> Conv2d in one kernel, fvfi_conv2d_nhwc_upsampled); inference only.
    ``x_direct`` [B,C2,H,W] (with ``upsample``): the input is ``cat(resize(x), x_direct)`` along the channels -- the concatenated
    tensor is never built (x.shape[1] must be a multiple of the K chunk: 32 channels, 16 for tf32x3)."""
    if not x.is_cuda:
        raise NotImplementedError("fvfi.conv.conv2d: CUDA tensors only")
    if torch.is_grad_enabled() and (x.requires_grad or weight.requires_grad or (bias is not None and bias.requires_grad)):
        assert upsample is None, "conv2d(upsample=...) is an inference form"
        assert out is None and not nchw_out and not pad_out and residual is None and act != "softmax", \
            "conv2d under autograd supports the plain NHWC form (bias + relu / elu / tanh / sigmoid)"
        return _ConvTC.apply(x, weight, bias, padding_mode, act)
    B, Cin, H, W = x.shape
    Cout, Cin_w, KH, KW = weight.shape
    xd, cin_up = None, 0
    if x_direct is not None:
        chunk = 32 if precision == PRECISIONS["f16x3"] else 16
        assert upsample is not None and Cin % chunk == 0 and Cin + x_direct.shape[1] >= Cin_w > Cin
        assert tuple(x_direct.shape[2:]) == tuple(int(v) for v in upsample[0]) and x_direct.shape[0] == B
        xd, cin_up = to_nhwc(x_direct.float()), Cin
        Cin = Cin_w
    assert Cin >= Cin_w and KH == KW and KH in (1, 3, 5)
    Cin = Cin_w
    xc = to_nhwc(x.float())
    assert xc.stride(1) == 1
    ldx = xc.stride(3)                       # floats per pixel
    Hs = Ws = align = 0
    if upsample is not None:
        cpk = 8 if precision == PRECISIONS["f16x3"] else 4
        if ldx % cpk or ldx < ((cin_up or Cin) + cpk - 1) // cpk * cpk or xc.data_ptr() % (4 * cpk):
            # the upsampling loader wants aligned channel groups: materialise the resampled tensor instead
            up = resize_bilinear(xc, tuple(upsample[0]), bool(upsample[1]))
            if xd is not None:
                up = torch.cat((up[:, :cin_up], xd), 1)
            return conv2d(up, weight, bias, padding_mode, act, out, nchw_out, pad_out, residual)
        Hs, Ws, align = H, W, int(bool(upsample[1]))
        H, W = (int(v) for v in upsample[0])
    if (upsample is None and KH == 1 and Cout <= 8 and Cin % 8 == 0 and Cin <= 128 and ldx % 8 == 0 and xc.data_ptr() % 32 == 0
            and act != "softmax" and out is None and not nchw_out and not pad_out and residual is None):
        return _conv1x1_direct(xc, weight, bias, act)
    if out is None:
        out = torch.empty((B, (Cout + 15) // 16 * 16 if pad_out else Cout, H, W), dtype=torch.float32, device=x.device,
                          memory_format=torch.contiguous_format if nchw_out else torch.channels_last)
    ldy = Cout if nchw_out else out.stride(3)
    if nchw_out:
        assert out.is_contiguous() and Cout <= 256 and not pad_out
    if pad_out:
        assert Cout <= 256
    L = _lib.lib()
    pad_mode = {"zeros": 0, "reflect": 1}[padding_mode]
    b = None if bias is None else bias.detach().contiguous().float()
    rc = None
    if residual is not None:
        assert not nchw_out and act != "softmax" and tuple(residual.shape) == (B, Cout, H, W)
        rc = to_nhwc(residual.float())
    with torch.cuda.device(x.device):
        parts = _packed(weight)
        if timing is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        for (o, n, buf) in parts:
            _lib.check(L.fvfi_conv2d_nhwc_upsampled(xc.data_ptr(), ldx, Hs, Ws, align, None if xd is None else xd.data_ptr(),
                                                    0 if xd is None else xd.stride(3), cin_up, buf.data_ptr(),
                                                    None if b is None else b.data_ptr() + 4 * o,
                                                    None if rc is None else rc.data_ptr() + 4 * o, 0 if rc is None else rc.stride(3),
                                                    out.data_ptr() + 4 * o, ldy, B, H, W, Cin, n, KH, KW, pad_mode, ACT[act],
                                                    1 if nchw_out else (2 if pad_out else 0), precision, _lib.stream_ptr()))
        if timing is not None:
            e1.record()
            timing.append((2.0 * B * H * W * Cin * Cout * KH * KW, e0, e1, len(parts), (B, Cin, Cout, KH, H, W, act), upsample is not None))
    return out


def _conv1x1_direct(xc, weight, bias, act):
    """1x1 convolution with Cout <= 8 as one pass over the NHWC activation (fvfi_conv1x1_nhwc, fp32 FFMA): PhaseNet's
    per-level prediction (phase_net.py:197-200), FusionNet's last layer (fusion_net.py:36)."""
    B, _, H, W = xc.shape
    Cout, Cin = weight.shape[0], weight.shape[1]
    assert B == 1 or xc.stride(0) == H * W * xc.stride(3)
    out = torch.empty((B, Cout, H, W), dtype=torch.float32, device=xc.device, memory_format=torch.channels_last)
    w = weight.detach().reshape(Cout, Cin).contiguous().float()
    b = None if bias is None else bias.detach().contiguous().float()
    with torch.cuda.device(xc.device):
        _lib.check(_lib.lib().fvfi_conv1x1_nhwc(xc.data_ptr(), xc.stride(3), w.data_ptr(), None if b is None else b.data_ptr(),
                                                out.data_ptr(), out.stride(3), B * H * W, Cin, Cout, ACT[act],
                                                _lib.stream_ptr()))
    return out


def upsample2_conv3x3_single(conv, x, act=None):
    """act(conv(Upsample(scale_factor=2, bilinear, align_corners=True)(x))) for a 3x3, zero-padded ``conv`` with ONE output
    channel (KernelEstimation's occlusion head, fusion_adacofnet.py:50-59,103-104) -> contiguous [B,1,2H,2W].
    Upsampling and convolution are linear: the C input channels are contracted first, at half resolution, into the nine
    tap maps (one C -> 9 tensor-core 1x1 convolution), and fvfi_upsample2_tapsum interpolates + sums the shifted taps."""
    assert conv.out_channels == 1 and conv.kernel_size == (3, 3) and conv.padding == (1, 1) and conv.padding_mode == "zeros"
    w = conv.weight
    key = (w.data_ptr(), w._version)
    hit = conv.__dict__.get("_fvfi_taps")
    if hit is None or hit[0] != key:
        C = w.shape[1]
        hit = (key, w.detach()[0].reshape(C, 9).t().reshape(9, C, 1, 1).contiguous())     # [tap = ky*3+kx, c]
        conv.__dict__["_fvfi_taps"] = hit
    B, _, H, W = x.shape
    z = conv2d(x, hit[1], None, "zeros", None, nchw_out=True)                             # planar [B,9,H,W]: coalesced tap reads
    out = torch.empty((B, 1, 2 * H, 2 * W), dtype=torch.float32, device=x.device)
    b = None if conv.bias is None else conv.bias.detach().contiguous().float()
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().fvfi_upsample2_tapsum(z.data_ptr(), 0, None if b is None else b.data_ptr(),
                                                    out.data_ptr(), B, H, W, ACT[act], _lib.stream_ptr()))
    return out


def resize_bilinear(x, size, align_corners, out=None, out_channel_offset=0, relu_input=False, add=None):
    """F.interpolate(x, size=size, mode='bilinear', align_corners=align_corners) on NHWC storage.  ``out`` may be a
    wider channels_last buffer; the result is written to channels [out_channel_offset, out_channel_offset + C).
    ``relu_input``: interpolate max(x, 0); ``add`` ([B,C,Ho,Wo]): added to the result -- FusionNet's decoder step
    ``Upsample(ReLU(x)) + skip`` (fusion_net.py:60-62) as one pass."""
    if torch.is_grad_enabled() and (x.requires_grad or (add is not None and add.requires_grad)):
        assert out is None and out_channel_offset == 0, "resize_bilinear under autograd returns a fresh tensor"
        return _ResizeFused.apply(x, add, (int(size[0]), int(size[1])), bool(align_corners), bool(relu_input))
    B, C, Hi, Wi = x.shape
    Ho, Wo = int(size[0]), int(size[1])
    xc = to_nhwc(x.float())
    if out is None:
        out = torch.empty((B, C, Ho, Wo), dtype=torch.float32, device=x.device, memory_format=torch.channels_last)
    assert out.stride(1) == 1 and out.shape[2] == Ho and out.shape[3] == Wo
    ac = None
    if add is not None:
        assert tuple(add.shape) == (B, C, Ho, Wo)
        ac = to_nhwc(add.float())
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().fvfi_resize_bilinear_nhwc_fused(xc.data_ptr(), xc.stride(3), None if ac is None else ac.data_ptr(),
                                                              0 if ac is None else ac.stride(3),
                                                              out.data_ptr() + 4 * out_channel_offset, out.stride(3), B, Hi, Wi, Ho,
                                                              Wo, C, 1 if align_corners else 0, 1 if relu_input else 0,
                                                              _lib.stream_ptr()))
    return out


def planar_concat_nhwc(tensors):
    """torch.cat(tensors, 1) of contiguous planar [B,c,H,W] tensors as ONE channels_last tensor with the channel count rounded up to 4
    (zeros), written by one kernel (fvfi_planar_concat_nhwc): returns [B, round4(sum c), H, W]."""
    import ctypes
    B, _, H, W = tensors[0].shape
    ts = [t.contiguous().float() for t in tensors]
    assert all(t.is_cuda and t.shape[0] == B and tuple(t.shape[2:]) == (H, W) for t in ts)
    C = sum(int(t.shape[1]) for t in ts)
    C4 = (C + 3) // 4 * 4
    out = torch.empty((B, C4, H, W), dtype=torch.float32, device=ts[0].device, memory_format=torch.channels_last)
    ptrs = (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])
    chans = (ctypes.c_int * len(ts))(*[int(t.shape[1]) for t in ts])
    with torch.cuda.device(out.device):
        _lib.check(_lib.lib().fvfi_planar_concat_nhwc(ctypes.cast(ptrs, ctypes.c_void_p), ctypes.cast(chans, ctypes.c_void_p), len(ts),
                                                      out.data_ptr(), out.stride(3), B, H, W, _lib.stream_ptr()))
    return out


def put_planar(x, out, out_channel_offset):
    """out[:, off:off+C] = x for a contiguous planar x [B,C,H,W] and a channels_last ``out`` (one kernel, no temporaries)."""
    B, C, H, W = x.shape
    x = x.contiguous().float()
    assert out.stride(1) == 1 and out.shape[2] == H and out.shape[3] == W
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().fvfi_nchw_to_nhwc_slice(x.data_ptr(), out.data_ptr() + 4 * out_channel_offset, out.stride(3),
                                                      B, C, H, W, _lib.stream_ptr()))
    return out


def max_pool2(x):
    """nn.MaxPool2d(2, stride=2) on NHWC storage (differentiable: fvfi_max_pool2_backward_nhwc)."""
    if torch.is_grad_enabled() and x.requires_grad:
        return _MaxPool2.apply(x)
    return avg_pool2(x, _fn="fvfi_max_pool2_nhwc")


class _MaxPool2(torch.autograd.Function):
    """nn.MaxPool2d(2, 2) of FusionNet's encoder (fusion_net.py:39,56) for the training step."""

    @staticmethod
    def forward(ctx, x):
        xc = to_nhwc(x.detach().float())
        ctx.save_for_backward(xc)
        return avg_pool2(xc, _fn="fvfi_max_pool2_nhwc")

    @staticmethod
    def backward(ctx, gy):
        (xc,) = ctx.saved_tensors
        B, C, H, W = xc.shape
        g = to_nhwc(gy.detach().float())
        gx = torch.empty((B, C, H, W), dtype=torch.float32, device=xc.device, memory_format=torch.channels_last)
        with torch.cuda.device(xc.device):
            _lib.check(_lib.lib().fvfi_max_pool2_backward_nhwc(xc.data_ptr(), xc.stride(3), g.data_ptr(), g.stride(3), gx.data_ptr(),
                                                               gx.stride(3), B, H, W, C, _lib.stream_ptr()))
        return gx


class _ResizeFused(torch.autograd.Function):
    """y = resize(relu_input ? max(x, 0) : x) + add  (FusionNet's decoder step, fusion_net.py:60-62) for the training step:
    forward fvfi_resize_bilinear_nhwc_fused, backward fvfi_resize_bilinear_backward_nhwc (the addend receives gy itself)."""

    @staticmethod
    def forward(ctx, x, add, size, align_corners, relu_input):
        xc = to_nhwc(x.detach().float())
        with torch.no_grad():
            y = resize_bilinear(xc, size, align_corners, relu_input=relu_input, add=None if add is None else add.detach())
        ctx.save_for_backward(xc)
        ctx.cfg = (size, align_corners, relu_input, add is not None)
        return y

    @staticmethod
    def backward(ctx, gy):
        (xc,) = ctx.saved_tensors
        (Ho, Wo), align, relu_in, has_add = ctx.cfg
        B, C, Hi, Wi = xc.shape
        g = to_nhwc(gy.detach().float())
        gx = None
        if ctx.needs_input_grad[0]:
            gx = torch.empty((B, C, Hi, Wi), dtype=torch.float32, device=xc.device, memory_format=torch.channels_last)
            with torch.cuda.device(xc.device):
                _lib.check(_lib.lib().fvfi_resize_bilinear_backward_nhwc(g.data_ptr(), g.stride(3), xc.data_ptr(), xc.stride(3),
                                                                         gx.data_ptr(), gx.stride(3), B, Hi, Wi, Ho, Wo, C,
                                                                         1 if align else 0, 1 if relu_in else 0, _lib.stream_ptr()))
        return gx, (gy if (has_add and ctx.needs_input_grad[1]) else None), None, None, None


class _AvgPool2(torch.autograd.Function):
    """nn.AvgPool2d(2, 2) of KernelEstimation's encoder (fusion_adacofnet.py:62-70) under autograd."""

    @staticmethod
    def forward(ctx, x):
        ctx.shape = tuple(x.shape)
        with torch.no_grad():
            return avg_pool2(x.detach())

    @staticmethod
    def backward(ctx, gy):
        B, C, H, W = ctx.shape
        g = to_nhwc(gy.detach().float())
        gx = torch.empty((B, C, H, W), dtype=torch.float32, device=g.device, memory_format=torch.channels_last)
        with torch.cuda.device(g.device):
            _lib.check(_lib.lib().fvfi_avg_pool2_backward_nhwc(g.data_ptr(), g.stride(3), gx.data_ptr(), gx.stride(3), B, H, W, C,
                                                               _lib.stream_ptr()))
        return gx


def avg_pool2(x, _fn="fvfi_avg_pool2_nhwc"):
    """nn.AvgPool2d(kernel_size=2, stride=2) on NHWC storage (differentiable: fvfi_avg_pool2_backward_nhwc)."""
    if _fn == "fvfi_avg_pool2_nhwc" and torch.is_grad_enabled() and x.requires_grad:
        return _AvgPool2.apply(x)
    B, C, H, W = x.shape
    xc = to_nhwc(x.float())
    out = torch.empty((B, C, H // 2, W // 2), dtype=torch.float32, device=x.device, memory_format=torch.channels_last)
    with torch.cuda.device(x.device):
        _lib.check(getattr(_lib.lib(), _fn)(xc.data_ptr(), xc.stride(3), out.data_ptr(), out.stride(3), B, H, W, C,
                                                  _lib.stream_ptr()))
    return out


def conv_module(conv, x, act=None, nchw_out=False, pad_out=False, residual=None, upsample=None, x_direct=None):
    """Run an nn.Conv2d (stride 1, dilation 1, padding == K//2) through the tensor-core kernel."""
    k = conv.kernel_size[0]
    assert conv.stride == (1, 1) and conv.dilation == (1, 1) and conv.groups == 1
    assert conv.padding == (k // 2, k // 2) or (k == 1 and conv.padding == (0, 0))
    mode = "zeros" if k == 1 else conv.padding_mode
    return conv2d(x, conv.weight, conv.bias, mode, act, nchw_out=nchw_out, pad_out=pad_out, residual=residual, upsample=upsample,
                  x_direct=x_direct)


def conv_bn_module(conv, bn, x, act=None, upsample=None, x_direct=None):
    """conv -> BatchNorm2d (eval: running statistics) -> act, with the BN affine folded into the weights."""
    key = (conv.weight.data_ptr(), conv.weight._version, None if conv.bias is None else conv.bias._version, bn.weight._version,
           bn.bias._version, bn.running_mean._version, bn.running_var._version)
    hit = conv.__dict__.get("_fvfi_fold")          # lives on the module: replaced (and its packed copy freed) when a version moves
    if hit is None or hit[0] != key:
        scale = (bn.weight / torch.sqrt(bn.running_var + bn.eps)).detach()
        w = (conv.weight.detach() * scale.view(-1, 1, 1, 1)).contiguous()
        b = ((conv.bias.detach() if conv.bias is not None else 0) - bn.running_mean) * scale + bn.bias.detach()
        hit = (key, w, b.contiguous())
        conv.__dict__["_fvfi_fold"] = hit
    k = conv.kernel_size[0]
    mode = "zeros" if k == 1 else conv.padding_mode
    return conv2d(x, hit[1], hit[2], mode, act, upsample=upsample, x_direct=x_direct)
