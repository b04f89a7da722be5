"""GPU parity tests of the model mirrors, the per-pixel stages and the full fusion pipeline."""
import glob
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import fusion_pipeline as fp

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _strict_fp32():
    """Parity is stated for fp32 arithmetic: cuDNN/cuBLAS TF32 off."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def test_lab_transforms():
    from fvfi import transform
    from oracle import lab
    rgb = torch.rand((2, 3, 37, 53), generator=torch.Generator().manual_seed(0))
    rgb[0, :, 0, :5] = 0.0
    rgb[0, :, 1, :5] = 1.0
    rgb[0, :, 2, :5] = 0.003  # linear segment of the sRGB curve
    got = transform.rgb2lab(rgb.cuda()).cpu()
    ref = fp.rgb2lab_planes(rgb)
    assert float((got - ref).abs().max()) <= 3e-6
    back = transform.lab2rgb(ref.cuda()).cpu()
    assert float((back - fp.lab2rgb_planes(ref)).abs().max()) <= 2e-5
    assert float((transform.rgb2lab_single(rgb[1].cuda()).cpu() - ref[1]).abs().max()) <= 3e-6
    # out-of-gamut Lab (what PhaseNet can produce) is clipped like skimage does
    wild = (ref * 1.6 - 0.3)
    assert float((transform.lab2rgb(wild.cuda()).cpu() - fp.lab2rgb_planes(wild)).abs().max()) <= 1e-4


@pytest.mark.parametrize("H,W", [(64, 96), (19, 33), (120, 70)])
def test_gaussian_and_median_vs_scipy(H, W):
    from scipy.ndimage import gaussian_filter, median_filter
    from fvfi import filters
    x = torch.rand((2, H, W), generator=torch.Generator().manual_seed(1)) * 3 - 1
    g = filters.gaussian_filter(x.cuda(), 5).cpu().numpy()
    ref = np.stack([gaussian_filter(m.numpy(), 5) for m in x])
    assert np.abs(g - ref).max() <= 2e-6
    for size in (50, 7, 4, 1):
        m = filters.median_filter(x.cuda(), size).cpu().numpy()
        ref = np.stack([median_filter(mm.numpy(), size=size) for mm in x])
        assert np.array_equal(m, ref), size       # order statistics: bit exact


@pytest.fixture(params=["inference", "autograd"])
def conv_backend(request):
    """The module tests run twice: under no_grad (the fused tcgen05 inference forwards) and with autograd enabled (the
    differentiable graphs the trainers use: every convolution, pooling and resize step of FusionNet / KernelEstimation / PhaseNetBlock
    is an autograd Function over the same libfvfi kernels).  There is no back-end switch: which form runs is decided by
    torch.is_grad_enabled() alone."""
    with (torch.no_grad() if request.param == "inference" else torch.enable_grad()):
        yield request.param


def test_models_vs_oracle_nets(conv_backend):
    """PhaseNet / FusionNet / AdaCoFNet mirrors vs the oracle restatements with one seeded state_dict."""
    import types
    from fvfi.adacofnet import AdaCoFNet
    from fvfi.fusion_net import FusionNet
    from oracle import nets
    state = fp.seeded_state(7)
    g = torch.Generator().manual_seed(7)
    # FusionNet (fusion_net.py:46-77)
    ins = [torch.rand((2, c, 64, 96), generator=g) for c in (3, 3, 3, 6, 3)]
    ofn = nets.FusionNet().eval()
    ofn.load_state_dict(state["fusion_net"])
    gfn = FusionNet().cuda().eval()
    gfn.load_state_dict(state["fusion_net"])
    with torch.no_grad():
        ref = ofn(*ins)
    got = gfn(*[t.cuda() for t in ins]).detach().cpu()
    # cuDNN fp32 vs oneDNN fp32: different accumulation orders over K = 25*128 products -> a few 1e-5
    print("FusionNet max abs err", float((got - ref).abs().max()))
    assert float((got - ref).abs().max()) <= 1e-4
    # AdaCoFNet incl. reflect padding to /32 (fusion_adacofnet.py:172-240)
    f0, f2 = torch.rand((1, 3, 70, 100), generator=g), torch.rand((1, 3, 70, 100), generator=g)
    oan = nets.AdaCoFNet(5, 1, threads=4).eval()
    oan.load_state_dict(state["adacof"])
    gan = AdaCoFNet(types.SimpleNamespace(kernel_size=5, dilation=1, gpu_id=0)).cuda().eval()
    gan.load_state_dict(state["adacof"])
    with torch.no_grad():
        r = oan(f0, f2)
    o = [t.detach() for t in gan(f0.cuda(), f2.cuda())]
    for a, b, name in zip(o, r, ("t1", "t2", "frame1", "mask")):
        assert a.shape == b.shape, name
        print("AdaCoFNet", name, float((a.cpu() - b).abs().max()))
        assert float((a.cpu() - b).abs().max()) <= 1e-4, name


def _state_for(z, seed):
    """The seeded random-init weights the fixture was made with (pinned by its checksum)."""
    state = fp.seeded_state(seed)
    chk = [float(sum(v.double().sum() for v in state[n].values())) for n in ("phase_net", "fusion_net", "adacof")]
    assert np.allclose(chk, z["checksum"], rtol=1e-9), "weights differ from the fixture's"
    return state


def test_pipeline_vs_reference_golden(golden_dir):
    """Full fusion recipe on the GPU vs the fixtures produced by the reference's own modules on CPU: 64x64, 64x96 (batch 2),
    256x256 (training crop size: pyramid height 12, PhaseNet.layers[7] shared by four levels), 184x328 (Bluestein / Rader FFT
    lengths, AdaCoFNet reflect padding in both axes).
    Bound: 1e-4 max abs on every image of the recipe against the reference (north star); the maps the recipe amplifies carry
    their explicit gain; the fp64 arbiter of the fixture backs anything beyond (tests/_parity.py)."""
    from _parity import WrapAligner, fmt, psnr, stage_report
    from fvfi.pipeline import FusionPipeline
    files = sorted(glob.glob(os.path.join(golden_dir, "pipeline_ref_*.npz")))
    assert len(files) >= 4
    for f in files:
        z = np.load(f)
        B, H, W, seed = [int(v) for v in z["meta"]]
        pipe = FusionPipeline(H, W, "cuda")
        pipe.load_state(_state_for(z, seed))
        pipe.stages = {}
        rgb1, rgb2 = fp.seeded_frames(B, H, W, seed)
        raw = pipe(rgb1.cuda(), rgb2.cuda()).cpu().numpy()            # as shipped: whatever branch the GPU's own rounding picks
        host = pipe.interpolate_host(rgb1.pin_memory(), rgb2.pin_memory())
        assert np.array_equal(host.numpy(), raw)                      # host-buffer entry point == device path
        # parity run on the reference's branch of the wrapped phases (oracle/wrap_align.py)
        pipe.filter_hook = al = WrapAligner(z)
        pipe.stages = {}
        pipe(rgb1.cuda(), rgb2.cuda())
        rep = stage_report(z, pipe.stages)
        print(os.path.basename(f), "wrap flips aligned: %d of %d phase values;" % (al.flips, al.coefficients), fmt(rep))
        bad = [k for k, v in rep.items() if not v["ok"]]
        assert not bad, (bad, fmt(rep))
        for k in ("lab1", "lab2", "ada_pred", "lab_pred", "phase_pred", "base", "final"):
            assert rep[k]["strict"], (k, fmt(rep))                    # the north-star bound itself on every image of the recipe
        assert al.flips <= 1e-5 * al.coefficients                     # a handful of coefficients, not a systematic difference
        st0 = int(z["final__stride"]) if "final__stride" in z.files else 1
        print("  unaligned run: final max abs err %.2e, PSNR %.1f dB" % (float(np.abs(raw[..., ::st0, ::st0] - z["final"]).max()),
                                                                        psnr(raw[..., ::st0, ::st0], z["final"])))
        assert psnr(raw[..., ::st0, ::st0], z["final"]) >= 70


@pytest.mark.parametrize("fused", [True, False])
def test_phasenet_256_vs_reference_golden(golden_dir, fused):
    """BASELINE.json configs[0]: PhaseNet decompose -> predict -> reconstruct on one 256x256 frame pair, random-init weights, against
    the reference's own Pyramid wrapper + PhaseNet on CPU (tests/golden/phasenet_ref_256x256_s5.npz): every predicted level
    (as complex coefficients), the low pass, the reconstructed Lab planes and the RGB frame.  Pyramid(12, 4, sqrt 2):
    levels 256,181,128,91,64,45,32,23,16,11 + low 8 -> layers[7] (phase_net.py:148) serves the four finest levels.
    fused: FusionPipeline.phase_interp (PhaseNet.forward_fused); not fused: the stepwise module API (separate_vals ->
    get_concat_layers_inf -> normalize_vals -> PhaseNet.forward) on the same decomposition."""
    from _parity import WrapAligner, fmt, stage_report
    from fvfi import transform, utils
    from fvfi.pipeline import FusionPipeline
    z = np.load(os.path.join(golden_dir, "phasenet_ref_256x256_s5.npz"))
    B, H, W, seed = [int(v) for v in z["meta"]]
    pipe = FusionPipeline(H, W, "cuda")
    assert pipe.pyr.height == 12
    pipe.load_state(_state_for(z, seed))
    pipe.filter_hook = al = WrapAligner(z)                    # compare on the reference's branch of the wrapped input phases
    pipe.stages = {}
    rgb1, rgb2 = fp.seeded_frames(B, H, W, seed)
    if fused:
        pipe.phase_interp(rgb1.cuda(), rgb2.cuda())
    else:
        pyr, net = pipe.pyr, pipe.phase_net
        with torch.no_grad():
            lab1, lab2 = transform.rgb2lab(rgb1.cuda()), transform.rgb2lab(rgb2.cuda())
            vals = pipe._filter("phasenet", torch.cat((lab1.reshape(-1, H, W), lab2.reshape(-1, H, W)), 0), want_high=False)
            vals_pred = net(net.normalize_vals(utils.get_concat_layers_inf(pyr, utils.separate_vals(vals, 2))))
            lab_pred = pyr.inv_filter_sparse(vals_pred, use_high=False).reshape(B, 3, H, W)
            pipe.stages.update(lab_pred=lab_pred, phase_pred=transform.lab2rgb(lab_pred), low_level=vals_pred.low_level)
            for l, (p, a) in enumerate(zip(vals_pred.phase, vals_pred.amplitude)):
                pipe.stages["phase%d" % l], pipe.stages["amp%d" % l] = p, a
    rep = stage_report(z, pipe.stages)
    print("fused" if fused else "stepwise", "wrap flips aligned: %d of %d" % (al.flips, al.coefficients), fmt(rep))
    assert al.flips <= 1e-5 * al.coefficients
    assert len(rep) == 13                      # 10 levels + low_level + lab_pred + phase_pred
    bad = [k for k, v in rep.items() if not v["ok"]]
    assert not bad, (bad, fmt(rep))
    assert rep["lab_pred"]["err_ref"] <= 1e-4 and rep["phase_pred"]["err_ref"] <= 1e-4      # the north-star bound itself


def test_cuda_graph_replay_matches_eager():
    """FusionPipeline.graphed: the captured launch sequence of a fixed-shape call (256x256 PhaseNet interpolation, and the frozen
    part of the training step) replays to exactly the eager result, for new input values too."""
    from fvfi.pipeline import FusionPipeline
    H = W = 128
    pipe = FusionPipeline(H, W, "cuda")
    pipe.load_state(fp.seeded_state(21))
    a1, a2 = [t.cuda() for t in fp.seeded_frames(2, H, W, 21)]
    b1, b2 = [t.cuda() for t in fp.seeded_frames(2, H, W, 22)]
    with torch.no_grad():
        g = pipe.graphed("phase_interp", a1, a2)
        assert pipe.graphed("phase_interp", a1, a2) is g                 # captured once per (method, shapes)
        for x1, x2 in ((a1, a2), (b1, b2), (a1, a2)):
            assert torch.equal(g(x1, x2).clone(), pipe.phase_interp(x1, x2))
        gi = pipe.graphed("fusion_inputs", a1, a2)
        for x1, x2 in ((b1, b2), (a1, a2)):
            got = [t.clone() for t in gi(x1, x2)]
            ref = pipe.fusion_inputs(x1, x2)
            assert all(torch.equal(p, q) for p, q in zip(got, ref))
        # small frames run the first AdaCoFNet pass on a side stream next to the PhaseNet branch: same values as in sequence
        assert pipe.concurrent_small
        out_c = pipe(a1, a2)
        pipe.concurrent_small = False
        out_s = pipe(a1, a2)
        assert torch.equal(out_c, out_s)


def test_conv_range_guard_reruns_in_tf32x3():
    """|activation| > 4094 leaves the 3xFP16 operand range: the decorated module forwards notice the device flag and run again with
    the 3xTF32 split instead of returning inf/NaN (ADVICE r1: device-resident path)."""
    from fvfi import conv as tc
    from fvfi.fusion_net import FusionNet
    from oracle import nets
    state = fp.seeded_state(13)
    g = torch.Generator().manual_seed(13)
    ins = [torch.rand((1, c, 32, 48), generator=g) for c in (3, 3, 3, 6, 3)]
    ins[3] = ins[3] * 3.0e4                                         # far beyond 4094
    ofn = nets.FusionNet().eval()
    ofn.load_state_dict(state["fusion_net"])
    gfn = FusionNet().cuda().eval()
    gfn.load_state_dict(state["fusion_net"])
    with torch.no_grad():
        ref = ofn(*ins)
        cins = [t.cuda() for t in ins]
        got = gfn(*cins).cpu()
        assert bool(torch.isfinite(got).all())
        with tc.forced_precision("tf32x3"):
            want = gfn(*cins).cpu()
        assert torch.equal(got, want)                               # the guarded call returned the 3xTF32 result
        assert float((got - ref).abs().max()) <= 2e-2               # |x| ~ 3e4 through 7 layers: fp32 rounding of both sides
        assert not tc.overflow_pending()                            # the guard consumed the flag
        x = (torch.rand((1, 16, 32, 48), generator=g) * 3.0e4).cuda()
        w = torch.rand((16, 16, 3, 3), generator=g).cuda()
        tc.conv2d(x, w)                                             # raw op outside a guarded forward: flag stays for the caller
        with pytest.raises(FloatingPointError):
            tc.check_overflow()


def test_training_step_gradients_match_oracle():
    """FusionNet training step (src/fusion_net/trainer.py:246-259): L1 loss on clip(pred,0,1), grads of the live
    parameters equal the oracle's; dead net.* parameters get no gradient."""
    from fvfi.fusion_net import FusionNet
    from oracle import nets
    state = fp.seeded_state(11)
    g = torch.Generator().manual_seed(11)
    ins = [torch.rand((2, c, 32, 32), generator=g) for c in (3, 3, 3, 6, 3)]
    target = torch.rand((2, 3, 32, 32), generator=g)
    ofn = nets.FusionNet()
    ofn.load_state_dict(state["fusion_net"])
    gfn = FusionNet().cuda()
    gfn.load_state_dict(state["fusion_net"])
    lo = torch.nn.functional.l1_loss(target, torch.clip(ofn(*ins), 0, 1))
    lo.backward()
    from fvfi import _lib
    n0 = _lib.lib().fvfi_launch_count()
    pred = gfn(*[t.cuda() for t in ins])
    assert _lib.lib().fvfi_launch_count() - n0 >= 7, "the training forward must run its 7 convolutions on the tcgen05 kernel"
    assert pred.requires_grad
    lg = torch.nn.functional.l1_loss(target.cuda(), torch.clip(pred, 0, 1))
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        lg.backward()
        torch.cuda.synchronize()
    foreign = [e.key for e in prof.key_averages()
               if any(k in e.key.lower() for k in ("cudnn", "convolution", "gemm", "max_pool", "upsample", "wgrad", "dgrad"))
               and "fvfi::" not in e.key]
    assert not foreign, "the backward of the trained network must run on libfvfi kernels: %s" % foreign
    assert abs(float(lo.detach()) - float(lg.detach())) <= 1e-6
    og = dict(ofn.named_parameters())
    for n, p in gfn.named_parameters():
        if n.startswith("net."):
            assert p.grad is None
        else:
            # ReLU / max-pool / clamp masks can flip on a handful of pixels between cuDNN and oneDNN forward
            # values, which changes single gradient entries discretely -> compare in norm as well as max
            d = p.grad.cpu() - og[n].grad
            assert float(d.abs().max()) <= 1e-4, n
            assert float(d.norm()) <= 2e-2 * float(og[n].grad.norm()) + 1e-7, n
    assert len(gfn.live_parameters()) == sum(1 for n, _ in gfn.named_parameters() if not n.startswith("net."))


def test_pipeline_1080p_properties():
    """BASELINE.json configs[2] size (1080x1920): properties that do not need the CPU reference at this size --
    per-sample independence (a batch equals its samples run alone; sub-batching is invisible), finite output in [0,1],
    host-buffer entry point == device path, no 3xFP16 range overflow."""
    from fvfi import conv as tc
    from fvfi.pipeline import FusionPipeline
    H, W = 1080, 1920
    pipe = FusionPipeline(H, W, "cuda")
    pipe.load_state(fp.seeded_state(0))
    r1, r2 = fp.seeded_frames(1, H, W, 3)
    g = torch.Generator().manual_seed(5)
    gains = 0.7 + 0.3 * torch.rand((3, 1, 1, 1), generator=g)
    f1, f2 = (r1 * gains).clamp(0, 1).cuda(), (r2 * gains).clamp(0, 1).cuda()
    pipe.max_batch = 8
    out = pipe(f1, f2)
    assert out.shape == (3, 3, H, W) and bool(torch.isfinite(out).all())
    assert float(out.min()) >= 0.0 and float(out.max()) <= 1.0
    pipe.max_batch = 2                                   # 2 + 1 sub-batches
    out2 = pipe(f1, f2)
    single = pipe(f1[1:2], f2[1:2])
    assert float((out - out2).abs().max()) <= 2e-6       # atomics-free kernels: only launch geometry differs
    assert float((out[1:2] - single).abs().max()) <= 2e-6
    host = pipe.interpolate_host(f1.cpu().pin_memory(), f2.cpu().pin_memory())
    assert float((host - out2.cpu()).abs().max()) <= 2e-6
    tc.check_overflow()


def test_pipeline_4k_runs():
    """BASELINE.json configs[3] size (3840x2160, one pair): the whole recipe runs at 4K (pyramid height 19, AdaCoFNet
    padding to 2176 rows, every convolution / resize / filter kernel at that size) and stays finite in [0,1]."""
    from fvfi import conv as tc
    from fvfi.pipeline import FusionPipeline
    H, W = 2160, 3840
    pipe = FusionPipeline(H, W, "cuda", phase_plane_chunk=3)
    pipe.load_state(fp.seeded_state(0))
    r1, r2 = fp.seeded_frames(1, H, W, 4)
    out = pipe(r1.cuda(), r2.cuda())
    assert out.shape == (1, 3, H, W) and bool(torch.isfinite(out).all())
    assert float(out.min()) >= 0.0 and float(out.max()) <= 1.0
    tc.check_overflow()


def test_phasenet_training_step():
    """PhaseNet training on the new path (SURVEY 8(f) f4): loss = L1(image) + wrapped-phase term back-propagates through
    Pyramid.inv_filter (fvfi_pyr_reconstruct_backward) into every PhaseNet layer; a few Adam steps on a fixed batch lower it."""
    import math
    from fvfi.phase_net import PhaseNet
    from fvfi.pyramid import Pyramid
    from fvfi.trainer import PhaseNetTrainer
    from fvfi.utils import calc_pyr_height
    torch.manual_seed(0)
    H = W = 64
    planes = torch.rand((6, H, W), device="cuda")
    height = calc_pyr_height(planes)
    pyr = Pyramid(height=height, nbands=4, scale_factor=math.sqrt(2), device=torch.device("cuda"))
    net = PhaseNet(pyr, torch.device("cuda"), num_img=2)
    tr = PhaseNetTrainer(pyr, net, lr=1e-3)
    l1, l2 = planes[:3], planes[3:]
    target = 0.5 * (l1 + l2)
    losses = [float(tr.step(l1, l2, target)) for _ in range(6)]
    assert all(math.isfinite(v) for v in losses)
    grads = [p.grad for p in net.parameters() if p.requires_grad]
    assert all(g is not None and bool(torch.isfinite(g).all()) for g in grads)
    # 64x64 -> 6 pyramid levels -> layers[0..6] are exercised; layers[7] (8 tensors) only exists for deeper pyramids
    assert sum(float(g.abs().sum()) > 0 for g in grads) >= len(grads) - 8
    assert losses[-1] < losses[0]


def test_median_full_tiles_and_ties_vs_scipy():
    """The tracked-median path of median_rank_kernel on full-width tiles (77 x 16 outputs for k = 50), several tile rows / columns, window
    sizes with a non-power-of-two bitmap share per lane, and heavily TIED data (values quantised to a few levels, saturated at 0 / 1 the
    way the recipe's clamped uncertainty maps are): bit-equal to scipy's rank filter."""
    from scipy.ndimage import median_filter
    from fvfi import filters
    g = torch.Generator().manual_seed(4)
    x = torch.rand((2, 150, 260), generator=g)
    x[1] = (x[1] * 6).floor() / 5                          # 6 distinct values
    x[0] = (x[0] * 1.6 - 0.3).clamp(0, 1)                  # ~19 % zeros, ~19 % ones
    for size in (50, 31, 21):
        m = filters.median_filter(x.cuda(), size).cpu().numpy()
        ref = np.stack([median_filter(mm.numpy(), size=size) for mm in x])
        assert np.array_equal(m, ref), size


@pytest.mark.parametrize("H,W,chunk", [(64, 96, None), (120, 70, 2)])
def test_phasenet_forward_fused_matches_stepwise(H, W, chunk):
    """PhaseNet.forward_fused (regrouping, normalisation, concat, amplitude blend and de-normalisation fused into two kernels,
    fvfi_phasenet_assemble / fvfi_phasenet_outputs) == separate_vals -> get_concat_layers_inf -> normalize_vals -> forward
    (-> reverse_normalize), the reference's step-by-step plumbing (src/train/utils.py:47-127, phase_net.py:42-177)."""
    import math
    from fvfi import utils
    from fvfi.phase_net import PhaseNet
    from fvfi.pyramid import Pyramid
    torch.manual_seed(3)
    P = 3
    planes = torch.rand((2 * P, H, W), device="cuda")
    height = utils.calc_pyr_height(planes)
    pyr = Pyramid(height=height, nbands=4, scale_factor=math.sqrt(2), device=torch.device("cuda"))
    net = PhaseNet(pyr, torch.device("cuda"), num_img=2).eval()
    net.plane_chunk = chunk
    with torch.no_grad():
        vals = pyr.filter(planes, want_high=False)
        ref = net(net.normalize_vals(utils.get_concat_layers_inf(pyr, utils.separate_vals(vals, 2))))
        out = net.forward_fused(vals, pyr.last_amp_max)
        assert len(out.phase) == len(ref.phase) == height - 2
        for a, b in zip(out.phase + out.amplitude + [out.low_level], ref.phase + ref.amplitude + [ref.low_level]):
            assert a.shape == b.shape
            assert float((a - b).abs().max()) <= 2e-6 * max(1.0, float(b.abs().max()))
        img_a = pyr.inv_filter_sparse(out, use_high=False)
        img_b = pyr.inv_filter_sparse(ref, use_high=False)
        assert float((img_a - img_b).abs().max()) <= 2e-6
        # hierarchical mode (phase_net.py:91-93): only the m coarsest levels are predicted, the finer ones are the int 0
        m = height - 4
        ref_m = net(net.normalize_vals(utils.get_concat_layers_inf(pyr, utils.separate_vals(vals, 2))), m)
        out_m = net.forward_fused(vals, pyr.last_amp_max, m)
        for a, b in zip(out_m.phase + out_m.amplitude, ref_m.phase + ref_m.amplitude):
            if torch.is_tensor(b):
                assert float((a - b).abs().max()) <= 2e-6 * max(1.0, float(b.abs().max()))
            else:
                assert not torch.is_tensor(a) and a == 0 and b == 0
        assert float((pyr.inv_filter_sparse(out_m, use_high=False) - pyr.inv_filter(ref_m)).abs().max()) <= 2e-6


@pytest.mark.parametrize("gain", [4.0, 0.37])
def test_phasenet_output_is_invariant_to_the_input_gain(gain):
    """SURVEY 8(c) invariant (v): normalize_vals divides every level by its own maximum and reverse_normalize multiplies it back
    (src/phase_net/phase_net.py:42-78,80-105), so scaling the decomposed planes by a constant must leave the predicted phases
    unchanged and scale the predicted amplitudes / low pass / reconstruction by exactly that constant (up to the eps = 1e-8 in
    the denominators and fp32 rounding) -- through the GPU decomposition, the fused value plumbing, the tcgen05 convolutions and
    the reconstruction."""
    import math
    from fvfi import utils
    from fvfi.phase_net import PhaseNet
    from fvfi.pyramid import Pyramid
    torch.manual_seed(11)
    H, W, P = 96, 128, 3
    planes = torch.rand((2 * P, H, W), device="cuda")
    height = utils.calc_pyr_height(planes)
    pyr = Pyramid(height=height, nbands=4, scale_factor=math.sqrt(2), device=torch.device("cuda"))
    net = PhaseNet(pyr, torch.device("cuda"), num_img=2).eval()
    with torch.no_grad():
        out1 = net.forward_fused(pyr.filter(planes, want_high=False), pyr.last_amp_max)
        img1 = pyr.inv_filter_sparse(out1, use_high=False)
        outg = net.forward_fused(pyr.filter(gain * planes, want_high=False), pyr.last_amp_max)
        imgg = pyr.inv_filter_sparse(outg, use_high=False)
    tol = 5e-6          # the eps in the denominators and fp32 rounding of the normalised network inputs (~1e-7) through the convolutions
    for l in range(height - 2):
        amax = float(out1.amplitude[l].abs().max())
        assert float((outg.amplitude[l] - gain * out1.amplitude[l]).abs().max()) <= tol * gain * amax
        # phases: compare where the amplitude is not negligible (atan2 of a rounding-level coefficient is arbitrary)
        live = out1.amplitude[l] > 1e-3 * amax
        d = (outg.phase[l] - out1.phase[l])[live]
        d = torch.atan2(torch.sin(d), torch.cos(d))
        assert float(d.abs().max()) <= 2e-4
    assert float((outg.low_level - gain * out1.low_level).abs().max()) <= 1e-5 * gain * float(out1.low_level.abs().max())
    assert float((imgg - gain * img1).abs().max()) <= 2e-5 * gain * float(img1.abs().max())


@pytest.mark.parametrize("B,H,W", [(2, 40, 72), (1, 64, 96), (3, 33, 50)])
def test_adacofnet_prep_kernel(B, H, W):
    """fvfi_adacofnet_prep == reflect pad to multiples of 32 (fusion_adacofnet.py:182-192), moduleNormalize (utility.py:86-87), concat,
    NHWC, and ReplicationPad2d(kernel_pad) (:168,195) of the un-normalised frames -- bit exact (data movement + one subtraction)."""
    import ctypes
    from fvfi import _lib
    from fvfi.adacofnet import moduleNormalize
    torch.manual_seed(5)
    f0, f2 = torch.rand((B, 3, H, W), device="cuda"), torch.rand((B, 3, H, W), device="cuda")
    hp, wp, k = (H + 31) // 32 * 32, (W + 31) // 32 * 32, 2
    x = torch.full((B, 8, hp, wp), 9.0, device="cuda").contiguous(memory_format=torch.channels_last)
    p0 = torch.full((B, 3, hp + 2 * k, wp + 2 * k), 9.0, device="cuda")
    p2 = torch.full_like(p0, 9.0)
    mean = (ctypes.c_float * 3)(0.4631, 0.4352, 0.3990)
    _lib.check(_lib.lib().fvfi_adacofnet_prep(f0.data_ptr(), f2.data_ptr(), x.data_ptr(), p0.data_ptr(), p2.data_ptr(), B, H, W, hp, wp, k,
                                              ctypes.cast(mean, ctypes.c_void_p), _lib.stream_ptr()))

    def pad(f):
        if hp != H:
            f = F.pad(f, (0, 0, 0, hp - H), mode='reflect')
        if wp != W:
            f = F.pad(f, (0, wp - W, 0, 0), mode='reflect')
        return f
    r0, r2 = pad(f0), pad(f2)
    ref_x = torch.cat([moduleNormalize(r0), moduleNormalize(r2), torch.zeros((B, 2, hp, wp), device="cuda")], 1)
    assert torch.equal(x, ref_x)
    rp = torch.nn.ReplicationPad2d([k] * 4)
    assert torch.equal(p0, rp(r0)) and torch.equal(p2, rp(r2))


def test_level0_difference_reconstruction_is_linear():
    """mean_c(recon_{high + level 0}(a_c) - recon_{high + level 0}(b_c)) == recon_{high + level 0}(filter(mean_c(a_c - b_c))): the
    uncertainty branch's h_freq difference (interpolate_twoframe.py:205-209) from ONE decomposed plane per frame pair; also through
    the complex-band entry point (Pyramid.inv_filter_bands)."""
    import math
    from fvfi import utils
    from fvfi.pyramid import Pyramid
    torch.manual_seed(11)
    B, H, W = 2, 72, 104
    a, b = torch.rand((B, 3, H, W), device="cuda"), torch.rand((B, 3, H, W), device="cuda")
    height = utils.calc_pyr_height(a[0])
    pyr = Pyramid(height=height, nbands=4, scale_factor=math.sqrt(2), device=torch.device("cuda"))
    with torch.no_grad():
        va, vb = utils.separate_vals(pyr.filter(torch.cat((a.reshape(-1, H, W), b.reshape(-1, H, W)), 0)), 2)
        ra = pyr.inv_filter_sparse(va, use_low=False, levels=[0]).reshape(B, 3, H, W).mean(1)
        rb = pyr.inv_filter_sparse(vb, use_low=False, levels=[0]).reshape(B, 3, H, W).mean(1)
        v0 = pyr.filter((a - b).mean(1), levels=[0])
        d = pyr.inv_filter_sparse(v0, use_low=False, levels=[0])
        z = torch.stack((torch.cos(v0.phase[0]) * v0.amplitude[0], torch.sin(v0.phase[0]) * v0.amplitude[0]), -1)   # [B*4,1,h,w,2]
        z = z.reshape(B, 4, z.shape[2], z.shape[3], 2)
        d2 = pyr.inv_filter_bands({0: [z[:, i].contiguous() for i in range(4)]}, B, H, W, high=v0.high_level)
    ref = ra - rb
    assert d.shape == ref.shape
    assert float((d - ref).abs().max()) <= 5e-6 * max(1.0, float(ref.abs().max()))
    assert float((d2 - d).abs().max()) <= 5e-6 * max(1.0, float(ref.abs().max()))


def test_phasenet_block_training_gradients_match_torch():
    """PhaseNetBlock in train mode (phase_net.py:179-207): convolutions forward + backward on libfvfi, BatchNorm with batch statistics;
    outputs and every parameter gradient equal torch's eager fp64 evaluation of the same block."""
    import copy
    from fvfi.phase_net import PhaseNetBlock
    torch.manual_seed(3)
    for c_in, k in ((88, (3, 3)), (81, (1, 1)), (2, (1, 1))):
        blk = PhaseNetBlock(c_in, 64, 8, k, torch.device("cuda"))
        blk.train()
        ref = copy.deepcopy(blk).double()
        x = torch.randn((3, c_in, 24, 20), device="cuda")
        gf, gc = torch.randn((3, 64, 24, 20), device="cuda"), torch.randn((3, 8, 24, 20), device="cuda")
        from fvfi import _lib
        n0 = _lib.lib().fvfi_launch_count()
        f, c = blk(x)
        assert _lib.lib().fvfi_launch_count() - n0 >= 3
        (f * gf).sum().add((c * gc).sum()).backward()
        fr = ref.feature_map(x.double())
        cr = ref.prediction_map(fr)
        (fr * gf.double()).sum().add((cr * gc.double()).sum()).backward()
        assert float((f.detach().double() - fr.detach()).abs().max()) <= 2e-5 * float(fr.detach().abs().max())
        assert float((c.detach().double() - cr.detach()).abs().max()) <= 2e-5
        for (n, p), (_, q) in zip(blk.named_parameters(), ref.named_parameters()):
            d = float((p.grad.double() - q.grad).abs().max())
            # the bias in front of the BatchNorm has an exactly zero gradient (the batch mean is removed): fp32 leaves the rounding of
            # a cancelling sum over 1440 pixels of O(10) terms there
            tol = 1e-3 if n == "feature_map.0.bias" else 5e-5 * max(1.0, float(q.grad.abs().max()))
            assert d <= tol, (c_in, n, d, float(q.grad.abs().max()))


def test_kernel_estimation_gradients_match_torch():
    """KernelEstimation under autograd (fusion_adacofnet.py:109-155): every module forward + backward on libfvfi (conv._ConvTC,
    _AvgPool2, _ResizeFused); the seven outputs and all parameter gradients equal torch's eager fp64 evaluation of the same modules."""
    import copy
    from fvfi.adacofnet import KernelEstimation
    from fvfi import _lib
    torch.manual_seed(5)
    ke = KernelEstimation(5).cuda()
    ref = copy.deepcopy(ke).double()
    a, b = torch.rand((1, 3, 64, 96), device="cuda") - 0.4, torch.rand((1, 3, 64, 96), device="cuda") - 0.4
    gouts = [torch.randn((1, c, 64, 96), device="cuda") for c in (25, 25, 25, 25, 25, 25, 1)]
    n0 = _lib.lib().fvfi_launch_count()
    with torch.enable_grad():
        outs = ke(a, b)
        assert _lib.lib().fvfi_launch_count() - n0 >= 46, "46 convolutions on libfvfi"
        sum((o * g).sum() for o, g in zip(outs, gouts)).backward()

    def eager(m, r0, r2):                       # the reference's forward, module by module, in fp64
        x = torch.cat([r0, r2], 1)
        c1 = m.moduleConv1(x)
        c2 = m.moduleConv2(m.modulePool1(c1))
        c3 = m.moduleConv3(m.modulePool2(c2))
        c4 = m.moduleConv4(m.modulePool3(c3))
        c5 = m.moduleConv5(m.modulePool4(c4))
        d5 = m.moduleUpsample5(m.moduleDeconv5(m.modulePool5(c5)))
        d4 = m.moduleUpsample4(m.moduleDeconv4(d5 + c5))
        d3 = m.moduleUpsample3(m.moduleDeconv3(d4 + c4))
        comb = m.moduleUpsample2(m.moduleDeconv2(d3 + c3)) + c2
        return [h(comb) for h in (m.moduleWeight1, m.moduleAlpha1, m.moduleBeta1, m.moduleWeight2, m.moduleAlpha2, m.moduleBeta2,
                                  m.moduleOcclusion)]
    routs = eager(ref, a.double(), b.double())
    sum((o * g.double()).sum() for o, g in zip(routs, gouts)).backward()
    for o, r in zip(outs, routs):
        assert float((o.detach().double() - r.detach()).abs().max()) <= 2e-5 * max(1.0, float(r.detach().abs().max()))
    worst = 0.0
    for (n, p), (_, q) in zip(ke.named_parameters(), ref.named_parameters()):
        d = float((p.grad.double() - q.grad).abs().max())
        # ReLU masks can flip on isolated pixels between the fp32 and fp64 forward; compare in norm as well
        rel = float((p.grad.double() - q.grad).norm()) / (float(q.grad.norm()) + 1e-12)
        worst = max(worst, rel)
        assert rel <= 2e-3, (n, rel, d)
    print("KernelEstimation gradients: worst relative L2 error %.2e" % worst)


def test_fusion_trainer_steps_are_bit_reproducible():
    """FusionTrainer.step (src/fusion_net/trainer.py:222-259 mirror): frozen PhaseNet + AdaCoF under no_grad, FusionNet forward + backward
    on libfvfi, Adam.  Two trainers started from the same weights produce IDENTICAL losses and gradients step after step (no atomics in
    any gradient kernel: the weight gradient sums its pixel ranges in a fixed order), and a few steps on a fixed batch lower the loss."""
    from fvfi.pipeline import FusionPipeline
    from fvfi.trainer import FusionTrainer
    from fvfi import synth
    H = W = 64

    def run():
        pipe = FusionPipeline(H, W, "cuda")
        pipe.load_state(synth.seeded_state(2))
        tr = FusionTrainer(pipe, lr=1e-3)
        a, b = synth.seeded_frames(2, H, W, 9)
        f1, f2 = a.cuda(), b.cuda()
        target = (0.5 * (f1 + f2)).clamp(0, 1)
        losses, flats = [], []
        for _ in range(4):
            losses.append(float(tr.step(f1, f2, target)))
            flats.append(tr.bucket.flat.clone())
        return losses, flats

    l1, g1 = run()
    l2, g2 = run()
    assert l1 == l2, (l1, l2)
    assert all(torch.equal(a, b) for a, b in zip(g1, g2))
    assert all(np.isfinite(v) for v in l1) and l1[-1] < l1[0]
    assert float(g1[0].abs().max()) > 0


def test_adacofnet_row_cropped_synthesis_matches_crop():
    """Frames whose height is not a multiple of 32 but whose width is (1080p: 1080 -> 1088 rows): the fused synthesis writes the unpadded
    rows itself (fvfi_adacofnet_warp_blend_rows) -- frame and uncertainty mask bit-identical to synthesis on the padded size + crop."""
    import types
    from fvfi.adacofnet import AdaCoFNet
    state = fp.seeded_state(8)
    net = AdaCoFNet(types.SimpleNamespace(kernel_size=5, dilation=1, gpu_id=0)).cuda().eval()
    net.load_state_dict(state["adacof"])
    g = torch.Generator().manual_seed(8)
    f0, f2 = torch.rand((2, 3, 70, 96), generator=g).cuda(), torch.rand((2, 3, 70, 96), generator=g).cuda()
    with torch.no_grad():
        _, _, fa, ma = net(f0, f2, return_warped=False)        # rows written directly
        t1, t2, fb, mb = net(f0, f2, return_warped=True)       # padded synthesis, cropped afterwards
    assert fa.shape == (2, 3, 70, 96) and ma.shape == (2, 1, 70, 96) and fa.is_contiguous()
    assert torch.equal(fa, fb) and torch.equal(ma, mb)
