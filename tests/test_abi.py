"""CPU tests of the drop-in boundary: libfvfi.so loads, exports every symbol include/fvfi.h declares, and the
Python mirror keeps the reference's interface (no compute calls -- there is no GPU here)."""
import inspect
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "fvfi.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fvfi_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_are_exported():
    import fvfi
    names = _declared()
    assert len(names) >= 25
    out = subprocess.check_output(["nm", "-D", "--defined-only", fvfi.lib_path()], text=True)
    exported = set(re.findall(r" T (fvfi_[a-z0-9_]+)", out))
    missing = [n for n in names if n not in exported]
    assert not missing, missing


def test_ctypes_prototypes_cover_the_header():
    import fvfi
    from fvfi import _lib
    L = fvfi.lib()
    assert L.fvfi_version() >= 100
    assert set(_declared()) == set(_lib._PROTOS), set(_declared()) ^ set(_lib._PROTOS)
    assert L.fvfi_pyr_next_size(256, 2 ** 0.5) == 181 and L.fvfi_pyr_next_size(181, 2 ** 0.5) == 128
    assert L.fvfi_pyr_next_size(128, 2.0) == 64


def test_no_cpu_fallback_and_reference_signatures():
    import torch
    from fvfi import adacof, pyramid, transform
    from fvfi.adacofnet import AdaCoFNet, KernelEstimation, make_model
    from fvfi.fusion_net import FusionNet
    from fvfi.phase_net import PhaseNet
    # FunctionAdaCoF.forward(ctx, input, weight, offset_i, offset_j, dilation)   (adacof.py:314)
    assert list(inspect.signature(adacof.FunctionAdaCoF.forward).parameters) == \
        ["ctx", "input", "weight", "offset_i", "offset_j", "dilation"]
    assert list(inspect.signature(pyramid.Pyramid.__init__).parameters) == ["self", "height", "nbands", "scale_factor", "device"]
    assert list(inspect.signature(FusionNet.forward).parameters) == \
        ["self", "base", "adacof", "phase", "other", "maps", "save", "variant"]
    assert list(inspect.signature(PhaseNet.__init__).parameters) == ["self", "pyr", "device", "num_img"]
    assert pyramid.DecompValues._fields == ("high_level", "phase", "amplitude", "low_level")
    x = torch.rand(1, 3, 12, 12)
    w = torch.rand(1, 9, 10, 10)
    with pytest.raises(NotImplementedError):          # adacof.py:356-357
        adacof.FunctionAdaCoF.apply(x, w, w, w, 1)
    with pytest.raises(NotImplementedError):
        pyramid.Pyramid(6, 4, 2 ** 0.5, torch.device("cpu")).filter(torch.rand(1, 32, 32))
    with pytest.raises(NotImplementedError):
        transform.rgb2lab(x)


def test_state_dict_keys_match_reference_checkpoints():
    """Key names are the checkpoint-compat contract (SURVEY.md section 5): phase_net.pt / fusion_net.pt / AdaCoF ckpt."""
    import types
    import torch
    from fvfi.adacofnet import AdaCoFNet
    from fvfi.fusion_net import FusionNet
    from fvfi.phase_net import PhaseNet
    pyr = types.SimpleNamespace(height=12, nbands=4)
    pn = PhaseNet(pyr, torch.device("cpu"), 2)
    keys = set(pn.state_dict())
    assert {"layers.0.feature_map.0.weight", "layers.7.feature_map.3.bias", "layers.3.prediction_map.0.weight",
            "layers.1.feature_map.1.running_mean"} <= keys
    assert sum(p.numel() for p in pn.parameters()) == 466745
    assert sum(v.numel() for v in pn.state_dict().values()) == 467777  # SURVEY App. F: values in phase_net.pt
    fn = FusionNet()
    assert sum(p.numel() for p in fn.parameters()) == 629350
    assert sum(p.numel() for p in fn.live_parameters()) == 543331
    assert {"net.0.weight", "encoder_layers.0.weight", "bottleneck_layer.bias", "decoder_layers.2.weight"} <= set(fn.state_dict())
    an = AdaCoFNet(types.SimpleNamespace(kernel_size=5, dilation=1, gpu_id=0))
    assert sum(p.numel() for p in an.parameters()) == 21843427
    assert "get_kernel.moduleConv1.0.weight" in an.state_dict() and "get_kernel.moduleOcclusion.7.bias" in an.state_dict()


def test_state_dicts_load_into_reference_modules(golden_dir):
    """The mirrors' state_dicts have exactly the keys and shapes of the REAL reference modules: the state the reference's own
    PhaseNet / FusionNet loaded strictly to make the committed pipeline fixtures (tests/golden/make_golden_models.py; the
    fixture's checksum pins it) loads strictly into the mirrors, so either side's state_dict loads into the other."""
    import types
    import numpy as np
    import torch
    from fvfi.fusion_net import FusionNet
    from fvfi.phase_net import PhaseNet
    from oracle import fusion_pipeline as fp
    z = np.load(os.path.join(golden_dir, "pipeline_ref_B1_64x64_s0.npz"))
    state = fp.seeded_state(int(z["meta"][3]))
    chk = [float(sum(v.double().sum() for v in state[n].values())) for n in ("phase_net", "fusion_net", "adacof")]
    assert np.allclose(chk, z["checksum"], rtol=1e-9), "seeded init differs from the fixture's"
    PhaseNet(types.SimpleNamespace(height=12, nbands=4), torch.device("cpu"), 2).load_state_dict(state["phase_net"], strict=True)
    FusionNet().load_state_dict(state["fusion_net"], strict=True)


def test_backward_entry_points_validate_arguments():
    """The backward C-ABI (include/fvfi.h "Backward of the same convolutions") rejects bad arguments with FVFI_EINVAL and a message that
    names the entry point, before any CUDA call (so this runs without a GPU)."""
    from fvfi import _lib
    L = _lib.lib()
    cases = [
        ("fvfi_conv2d_wgrad_nhwc", lambda: L.fvfi_conv2d_wgrad_nhwc(None, 18, None, 32, 256, 65536, None, 8, 256, 256, 18, 32, 5, 1, None, None)),
        ("fvfi_conv2d_wgrad_nhwc", lambda: L.fvfi_conv2d_wgrad_nhwc(16, 18, 16, 32, 256, 65536, 16, 8, 256, 256, 18, 32, 4, 1, 16, None)),   # even K
        ("fvfi_conv2d_wgrad_nhwc", lambda: L.fvfi_conv2d_wgrad_nhwc(16, 8, 16, 32, 256, 65536, 16, 8, 256, 256, 18, 32, 5, 1, 16, None)),    # stride < Cin
        ("fvfi_conv2d_wgrad_nhwc", lambda: L.fvfi_conv2d_wgrad_nhwc(16, 18, 16, 32, 2, 4, 16, 1, 2, 2, 18, 32, 5, 1, 16, None)),             # reflect: H <= K/2
        ("fvfi_conv2d_grad_act", lambda: L.fvfi_conv2d_grad_act(None, 32, None, 32, None, 8, 256, 256, 32, 2, 1, None, None, None)),
        ("fvfi_conv2d_grad_act", lambda: L.fvfi_conv2d_grad_act(16, 32, None, 32, 16, 8, 256, 256, 32, 2, 1, None, None, None)),             # ReLU needs y
        ("fvfi_conv2d_grad_act", lambda: L.fvfi_conv2d_grad_act(16, 32, 16, 32, 16, 8, 256, 256, 32, 2, 1, 16, None, None)),                 # gbias needs workspace
        ("fvfi_reflect_pad_backward_nhwc", lambda: L.fvfi_reflect_pad_backward_nhwc(16, 32, 16, 32, 1, 2, 2, 32, 2, None)),                 # H <= P
        ("fvfi_resize_bilinear_backward_nhwc", lambda: L.fvfi_resize_bilinear_backward_nhwc(16, 32, None, 32, 16, 32, 1, 8, 8, 40, 16, 32, 0, 0, None)),
        ("fvfi_resize_bilinear_backward_nhwc", lambda: L.fvfi_resize_bilinear_backward_nhwc(16, 32, None, 32, 16, 32, 1, 8, 8, 16, 16, 32, 0, 1, None)),
        ("fvfi_max_pool2_backward_nhwc", lambda: L.fvfi_max_pool2_backward_nhwc(None, 1, None, 1, None, 1, 1, 4, 4, 1, None)),
        ("fvfi_avg_pool2_backward_nhwc", lambda: L.fvfi_avg_pool2_backward_nhwc(16, 1, 16, 1, 1, 1, 4, 1, None)),                           # Hi < 2
        ("fvfi_fusion_blend_backward", lambda: L.fvfi_fusion_blend_backward(None, None, None, None, None, 10, None)),
    ]
    for name, call in cases:
        rc = call()
        assert rc != 0, name
        assert name in L.fvfi_last_error().decode(), (name, L.fvfi_last_error())
    assert L.fvfi_conv2d_wgrad_workspace_floats(8, 256, 256, 18, 32, 5) >= 32 * 25 * 20
    assert L.fvfi_conv2d_grad_act_workspace_floats(8, 256, 256, 32, 2) >= 32
