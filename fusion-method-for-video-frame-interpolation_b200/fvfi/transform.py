"""Drop-in for the reference's ``src/train/transform.py`` (rgb2lab, rgb2lab_single, lab2rgb,
lab2rgb_single) -- device-resident: the reference round-trips through skimage on the host CPU
(transform.py:8,19,35,46); here one CUDA kernel per direction, no host copy, same L/100 and
(a,b+128)/255 scaling."""
import torch

from . import _lib


def _run(fn_name, img):
    if not img.is_cuda:
        raise NotImplementedError("fvfi colour transforms run on CUDA tensors only")
    x = img.contiguous().float()
    B, C, H, W = x.shape
    assert C == 3
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(getattr(_lib.lib(), fn_name)(x.data_ptr(), out.data_ptr(), B, H, W, _lib.stream_ptr()))
    return out


def rgb2lab(img, light=100, ab_mul=255, ab_max=128):
    """[B,3,H,W] RGB in [0,1] -> scaled Lab (transform.py:6-14)."""
    assert (light, ab_mul, ab_max) == (100, 255, 128)
    return _run("fvfi_rgb2lab", img)


def rgb2lab_single(img, light=100, ab_mul=255, ab_max=128):
    """[3,H,W] (transform.py:17-25)."""
    return rgb2lab(img.unsqueeze(0), light, ab_mul, ab_max)[0]


def lab2rgb(img, light=100, ab_mul=255, ab_max=128):
    """[B,3,H,W] scaled Lab -> RGB in [0,1] (transform.py:28-37)."""
    assert (light, ab_mul, ab_max) == (100, 255, 128)
    return _run("fvfi_lab2rgb", img)


def rgb8_to_rgb_lab(frames8):
    """Decoder frames [T,H,W,3] uint8 (interleaved rgb24) -> (rgb, lab): planar fp32 [T,3,H,W] RGB (the correctly rounded k / 255)
    and scaled Lab, in one kernel (fvfi_rgb8_to_rgb_lab); ``lab`` equals ``rgb2lab(rgb)`` bit for bit."""
    if not frames8.is_cuda:
        raise NotImplementedError("fvfi colour transforms run on CUDA tensors only")
    assert frames8.dtype == torch.uint8 and frames8.dim() == 4 and frames8.shape[3] == 3
    x = frames8.contiguous()
    T, H, W, _ = x.shape
    rgb = torch.empty((T, 3, H, W), dtype=torch.float32, device=x.device)
    lab = torch.empty_like(rgb)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().fvfi_rgb8_to_rgb_lab(x.data_ptr(), rgb.data_ptr(), lab.data_ptr(), T, H, W, _lib.stream_ptr()))
    return rgb, lab


def lab2rgb_single(img, light=100, ab_mul=255, ab_max=128):
    """[3,H,W] (transform.py:40-49)."""
    return lab2rgb(img.unsqueeze(0), light, ab_mul, ab_max)[0]
