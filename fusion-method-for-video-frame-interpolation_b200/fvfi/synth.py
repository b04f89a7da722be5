"""Seeded synthetic inputs for benchmarks, smoke runs and profiling drivers: random-init network weights and smooth
synthetic frame pairs (BASELINE.json: "synthetic frame pairs of the named resolutions with random-init weights").

Input GENERATION only -- nothing here is on the timed path.  The networks are this package's own drop-in modules built on
the CPU under ``torch.manual_seed`` (``nn.Module`` default init, BatchNorm running statistics at 0/1), whose parameter
names and creation order equal the reference's (src/phase_net/phase_net.py:21-35, src/fusion_net/fusion_net.py:8-43,
src/fusion_net/fusion_adacofnet.py:14-107), so one seed gives the reference, the oracle and the product the same
``state_dict`` (tests/test_abi.py checks this against the oracle's generator).
"""
import types

import torch


def seeded_state(seed, kernel_size=5):
    """{'phase_net', 'fusion_net', 'adacof'} state_dicts (CPU tensors)."""
    from .adacofnet import AdaCoFNet
    from .fusion_net import FusionNet
    from .phase_net import PhaseNet
    torch.manual_seed(seed)
    pyr = types.SimpleNamespace(height=8, nbands=4)
    cpu = torch.device("cpu")
    return {"phase_net": PhaseNet(pyr, cpu, 2).state_dict(), "fusion_net": FusionNet().state_dict(),
            "adacof": AdaCoFNet(types.SimpleNamespace(kernel_size=kernel_size, dilation=1, gpu_id=0)).state_dict()}


def seeded_frames(B, H, W, seed):
    """Two batches [B,3,H,W] in [0,1]: low-pass noise plus fine noise, the second a shifted crop of the same field
    (smooth, so Lab stays in gamut and the flow is a few pixels)."""
    g = torch.Generator().manual_seed(seed)
    base = torch.rand((B, 3, H // 4 + 2, W // 4 + 2), generator=g)
    up = torch.nn.functional.interpolate(base, size=(H + 8, W + 8), mode='bicubic', align_corners=False).clamp(0.02, 0.98)
    noise = 0.03 * torch.rand((B, 3, H + 8, W + 8), generator=g)
    full = (up + noise).clamp(0, 1)
    return full[:, :, 2:2 + H, 1:1 + W].contiguous(), full[:, :, 5:5 + H, 6:6 + W].contiguous()


def seeded_clip(T, H, W, seed, shift=(2, 3)):
    """A clip [T,3,H,W] in [0,1] of constant motion: frame t is the crop at offset t * shift = (dy, dx) pixels of ONE smooth
    random field (low-pass noise plus fine noise, as seeded_frames).  Negative components move the other way.  A large shift
    (e.g. (12, 24) at 1080p) keeps the warps away from their best case of near-zero flow."""
    dy, dx = int(shift[0]), int(shift[1])
    g = torch.Generator().manual_seed(seed)
    Hf, Wf = H + abs(dy) * (T - 1) + 8, W + abs(dx) * (T - 1) + 8
    base = torch.rand((1, 3, Hf // 4 + 2, Wf // 4 + 2), generator=g)
    up = torch.nn.functional.interpolate(base, size=(Hf, Wf), mode='bicubic', align_corners=False).clamp(0.02, 0.98)
    full = (up + 0.03 * torch.rand((1, 3, Hf, Wf), generator=g)).clamp(0, 1)[0]
    y0 = 4 + (abs(dy) * (T - 1) if dy < 0 else 0)
    x0 = 4 + (abs(dx) * (T - 1) if dx < 0 else 0)
    return torch.stack([full[:, y0 + t * dy:y0 + t * dy + H, x0 + t * dx:x0 + t * dx + W] for t in range(T)]).contiguous()


def to_rgb8(clip):
    """[T,3,H,W] in [0,1] -> the 8-bit interleaved [T,H,W,3] uint8 a decoder delivers (round half to even)."""
    return (clip * 255).round().clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def rgb8_values(frames8):
    """uint8 [T,H,W,3] -> the fp32 planar [T,3,H,W] values k / 255 (correctly rounded: built in float64, then cast)."""
    return (frames8.permute(0, 3, 1, 2).double() / 255).float().contiguous()
