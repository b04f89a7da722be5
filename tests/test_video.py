"""Clip interpolation: the 8-bit conversion and blend kernels, the plane-offset (clip layout) PhaseNet glue, interpolate_sequence /
interpolate_video_host against the pair path, and the raw-video CLI (python -m fvfi.interpolate_video)."""
import io

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _strict_fp32():
    """The pair path and the clip path are compared in fp32: cuDNN/cuBLAS TF32 off."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


# ---- CPU: argument checks of the new entry points and of the CLI -------------------------------------------------------------

def test_clip_entry_points_validate_arguments():
    """Null pointers, bad sizes and a frame-2 plane offset past the last plane are rejected with FVFI_EINVAL and a message naming
    the entry point, before any CUDA call."""
    from fvfi import _lib
    L = _lib.lib()
    cases = [
        ("fvfi_rgb8_to_rgb_lab", lambda: L.fvfi_rgb8_to_rgb_lab(None, 16, 16, 1, 4, 4, None)),
        ("fvfi_rgb8_to_rgb_lab", lambda: L.fvfi_rgb8_to_rgb_lab(16, 16, 16, 0, 4, 4, None)),
        ("fvfi_rgb8_to_rgb_lab", lambda: L.fvfi_rgb8_to_rgb_lab(16, 16, 16, 1, -4, 4, None)),
        ("fvfi_fusion_blend_rgb8", lambda: L.fvfi_fusion_blend_rgb8(16, None, 16, 1, 4, 4, None)),
        ("fvfi_fusion_blend_rgb8", lambda: L.fvfi_fusion_blend_rgb8(16, 16, 16, 1, 4, 0, None)),
        ("fvfi_fusion_blend_rgb8", lambda: L.fvfi_fusion_blend_rgb8(16, 16, 16, 70000, 4, 4, None)),
        # N = 9 planes (3 frames), P = 6, q = 3: the last pair-plane reads plane 8 -- fine; q = 4 would read plane 9
        ("fvfi_phasenet_assemble_offset", lambda: L.fvfi_phasenet_assemble_offset(None, 16, 16, 16, 16, 9, 6, 3, 0, 6, 4, 8, 8, None)),
        ("fvfi_phasenet_assemble_offset", lambda: L.fvfi_phasenet_assemble_offset(16, 16, 16, 16, 16, 9, 6, 4, 0, 6, 4, 8, 8, None)),
        ("fvfi_phasenet_assemble_offset", lambda: L.fvfi_phasenet_assemble_offset(16, 16, 16, 16, 16, 9, 6, 3, 4, 3, 4, 8, 8, None)),
        ("fvfi_phasenet_assemble_offset", lambda: L.fvfi_phasenet_assemble_offset(16, 16, 16, 16, 16, 9, 6, 0, 0, 6, 4, 8, 8, None)),
        ("fvfi_phasenet_assemble_offset", lambda: L.fvfi_phasenet_assemble_offset(16, 16, 16, 16, 8, 9, 6, 3, 0, 6, 4, 8, 8, None)),
        ("fvfi_phasenet_outputs_offset", lambda: L.fvfi_phasenet_outputs_offset(16, 8, None, 16, 16, 9, 6, 3, 0, 6, 4, 8, 8, None)),
        ("fvfi_phasenet_outputs_offset", lambda: L.fvfi_phasenet_outputs_offset(16, 8, 16, 16, 16, 9, 6, 4, 0, 6, 4, 8, 8, None)),
        ("fvfi_phasenet_outputs_offset", lambda: L.fvfi_phasenet_outputs_offset(16, 8, 16, 16, 16, 9, 6, 3, 0, 6, 2, 8, 8, None)),
        ("fvfi_phasenet_outputs_offset", lambda: L.fvfi_phasenet_outputs_offset(16, 8, 16, 16, 16, 9, 6, 3, 0, 0, 4, 8, 8, None)),
    ]
    for name, call in cases:
        rc = call()
        assert rc != 0, name
        assert name in L.fvfi_last_error().decode(), (name, L.fvfi_last_error())


def _cli_rejects(monkeypatch, tmp_path, data, via_pipe, capsys):
    from fvfi import interpolate_video, pipeline

    def no_cuda(*a, **k):
        raise AssertionError("the CLI built the pipeline before rejecting its input")
    monkeypatch.setattr(pipeline, "FusionPipeline", no_cuda)
    monkeypatch.setattr(torch.cuda, "init", no_cuda)
    if via_pipe:
        monkeypatch.setattr("sys.stdin", io.TextIOWrapper(io.BytesIO(data)))
        src = "-"
    else:
        src = str(tmp_path / "in.rgb")
        open(src, "wb").write(data)
    rc = interpolate_video.main(["--size", "6x4", "--seeded-weights", "0", "--input", src, "--output", str(tmp_path / "out.rgb")])
    assert rc == 2
    return capsys.readouterr().err


@pytest.mark.parametrize("via_pipe", [False, True])
def test_cli_rejects_truncated_and_single_frame_clips(monkeypatch, tmp_path, capsys, via_pipe):
    fb = 6 * 4 * 3
    err = _cli_rejects(monkeypatch, tmp_path, bytes(fb), via_pipe, capsys)             # one frame
    assert "at least 2" in err
    err = _cli_rejects(monkeypatch, tmp_path, bytes(fb + fb // 2), via_pipe, capsys)   # a frame and a half
    assert "frame" in err
    if not via_pipe:                                                                   # a regular file is sized up front
        err = _cli_rejects(monkeypatch, tmp_path, bytes(5 * fb + 7), via_pipe, capsys)
        assert "not a whole number" in err


def test_seeded_clip_moves_by_the_shift():
    from fvfi import synth
    clip = synth.seeded_clip(4, 20, 30, 1, shift=(3, -5))
    assert clip.shape == (4, 3, 20, 30) and float(clip.min()) >= 0 and float(clip.max()) <= 1
    # frame t+1 at (y, x) is frame t at (y + 3, x - 5)
    assert torch.equal(clip[1][:, :17, 5:], clip[0][:, 3:, :25])
    f8 = synth.to_rgb8(clip)
    assert f8.shape == (4, 20, 30, 3) and f8.dtype == torch.uint8
    assert float((synth.rgb8_values(f8) - clip).abs().max()) <= 0.5 / 255 + 1e-7


# ---- GPU ------------------------------------------------------------------------------------------------------------------------

def _pipe(H, W, seed=0, max_batch=8):
    from fvfi import synth
    from fvfi.pipeline import FusionPipeline
    pipe = FusionPipeline(H, W, "cuda")
    pipe.load_state(synth.seeded_state(seed))
    pipe.max_batch = max_batch
    return pipe


@gpu
@pytest.mark.parametrize("T,H,W", [(1, 1, 1), (2, 37, 53), (1, 1080, 1920), (1, 16, 16)])
def test_rgb8_to_rgb_lab(T, H, W):
    from fvfi import transform
    g = torch.Generator().manual_seed(T * 7 + H)
    f8 = torch.randint(0, 256, (T, H, W, 3), generator=g, dtype=torch.uint8)
    if H * W >= 256:                                      # every code in every channel
        flat = f8.view(-1, 3)
        for c in range(3):
            flat[:256, c] = torch.roll(torch.arange(256, dtype=torch.uint8), 85 * c)
    table = (torch.arange(256, dtype=torch.float64) / 255).float()      # correctly rounded k/255 (torch's CUDA /255 may not be)
    want_rgb = table[f8.long()].permute(0, 3, 1, 2).contiguous()
    rgb, lab = transform.rgb8_to_rgb_lab(f8.cuda())
    assert torch.equal(rgb.cpu(), want_rgb)
    assert torch.equal(lab, transform.rgb2lab(want_rgb.cuda()))


@gpu
def test_fusion_blend_rgb8():
    from fvfi.fusion_net import fusion_blend, fusion_blend_rgb8
    g = torch.Generator().manual_seed(4)
    base = (torch.rand((2, 3, 37, 53), generator=g) * 2 - 0.5).cuda()      # clamps at 0 and at 1
    x = (torch.randn((2, 3, 37, 53), generator=g) * 2).cuda()
    want = (fusion_blend(base, x).cpu() * 255).round().to(torch.uint8).permute(0, 2, 3, 1)
    got = fusion_blend_rgb8(base, x).cpu()
    assert torch.equal(got, want)
    assert int(got.min()) == 0 and int(got.max()) == 255


@gpu
@pytest.mark.parametrize("Tp,p0,pc", [(4, 0, 9), (5, 3, 7)])
def test_phasenet_glue_offset_entry_points(Tp, p0, pc):
    """q = P equals the pair entry points; q = 3 on a decomposition of T' consecutive frames equals the pair entry points on the
    pair-layout cat of the same frames."""
    from fvfi import _lib
    L = _lib.lib()
    nb, h, w = 4, 13, 21
    g = torch.Generator().manual_seed(Tp)
    ph_f = torch.randn((Tp, 3, nb, h, w), generator=g).cuda()          # per-frame planes of one level (clip layout)
    am_f = torch.rand((Tp, 3, nb, h, w), generator=g).cuda()
    P = 3 * (Tp - 1)
    pair = lambda t: torch.cat((t[:-1], t[1:]), 0).reshape(2 * P * nb, h, w).contiguous()
    clip = lambda t: t.reshape(Tp * 3 * nb, h, w).contiguous()
    den = (torch.rand(P, generator=g) + 0.5).cuda()
    pred = torch.randn((pc, h, w, 2 * nb), generator=g).cuda()
    s = _lib.stream_ptr()

    def assemble(fn, ph, am, *layout):
        y = torch.zeros((pc, h, w, 4 * nb), device="cuda")
        _lib.check(fn(ph.data_ptr(), am.data_ptr(), den.data_ptr(), y.data_ptr(), 4 * nb, *layout, p0, pc, nb, h, w, s))
        return y

    def outputs(fn, am, *layout):
        po, ao = torch.zeros((P * nb, h, w), device="cuda"), torch.zeros((P * nb, h, w), device="cuda")
        _lib.check(fn(pred.data_ptr(), 2 * nb, am.data_ptr(), po.data_ptr(), ao.data_ptr(), *layout, p0, pc, nb, h, w, s))
        return po, ao

    ref_y = assemble(L.fvfi_phasenet_assemble, pair(ph_f), pair(am_f), P)
    ref_o = outputs(L.fvfi_phasenet_outputs, pair(am_f), P)
    assert float(ref_y.abs().sum()) > 0
    assert torch.equal(assemble(L.fvfi_phasenet_assemble_offset, pair(ph_f), pair(am_f), 2 * P, P, P), ref_y)
    assert torch.equal(assemble(L.fvfi_phasenet_assemble_offset, clip(ph_f), clip(am_f), 3 * Tp, P, 3), ref_y)
    for a, b in zip(outputs(L.fvfi_phasenet_outputs_offset, pair(am_f), 2 * P, P, P), ref_o):
        assert torch.equal(a, b)
    for a, b in zip(outputs(L.fvfi_phasenet_outputs_offset, clip(am_f), 3 * Tp, P, 3), ref_o):
        assert torch.equal(a, b)


def _count_excess(a, b, tol):
    return int(((a - b).abs() > tol).sum())


@gpu
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("H,W,T,mb", [(64, 96, 6, 2), (256, 256, 5, 3), (184, 328, 4, 8)])
def test_interpolate_sequence_matches_pairs(H, W, T, mb, fused):
    """The clip path (each frame converted and decomposed once per window, glue in the q = 3 layout) against the pair path on
    frames[:-1], frames[1:] with the same sub-batching."""
    from fvfi import synth
    pipe = _pipe(H, W, seed=2, max_batch=mb)
    pipe.fused_phase_glue = fused
    if H * W <= 512 * 512:
        assert pipe.concurrent_small                        # 64x96 and 256x256 take the side-stream fork
    clip = synth.seeded_clip(T, H, W, 5, shift=(2, -3)).cuda()
    got = pipe.interpolate_sequence(clip)
    want = pipe(clip[:-1], clip[1:])
    assert got.shape == want.shape == (T - 1, 3, H, W)
    err = float((got - want).abs().max())
    assert err <= 2e-6, (err, _count_excess(got, want, 2e-6))


@gpu
def test_interpolate_sequence_rgb8_is_the_quantised_fp32_path():
    from fvfi import synth
    H, W = 64, 96
    pipe = _pipe(H, W, seed=3, max_batch=2)
    f8 = synth.to_rgb8(synth.seeded_clip(6, H, W, 7, shift=(3, 4))).cuda()
    got = pipe.interpolate_sequence(f8)
    ref = pipe.interpolate_sequence(synth.rgb8_values(f8.cpu()).cuda())
    assert got.dtype == torch.uint8 and got.shape == (5, H, W, 3)
    assert torch.equal(got.cpu(), (ref.cpu() * 255).round().to(torch.uint8).permute(0, 2, 3, 1))


@gpu
def test_interpolate_sequence_rejects_bad_clips():
    pipe = _pipe(32, 48)
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(torch.rand((1, 3, 32, 48), device="cuda"))                     # T < 2
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(torch.rand((3, 3, 32, 40), device="cuda"))                     # frame size
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(torch.rand((3, 3, 32, 48), device="cuda", dtype=torch.float64))  # dtype
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(torch.zeros((3, 3, 32, 48), device="cuda", dtype=torch.uint8))   # planar 8-bit
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(torch.rand((3, 32, 48, 3), device="cuda"))                     # interleaved fp32


@gpu
@pytest.mark.parametrize("T,mb", [(6, 4), (4, 8)])
def test_interpolate_video_host(T, mb):
    from fvfi import synth
    H, W = 64, 96
    pipe = _pipe(H, W, seed=4, max_batch=mb)
    f8 = synth.to_rgb8(synth.seeded_clip(T, H, W, 9, shift=(-2, 5))).pin_memory()
    out = pipe.interpolate_video_host(f8)
    assert out.shape == (2 * T - 1, H, W, 3) and out.is_pinned()
    assert torch.equal(out[0::2], f8)
    assert torch.equal(out[1::2], pipe.interpolate_sequence(f8.cuda()).cpu())


@gpu
def test_clip_1080p_large_motion():
    from fvfi import conv as tc
    from fvfi import synth
    H, W, T = 1080, 1920, 10
    pipe = _pipe(H, W, seed=0, max_batch=8)                   # windows of 9 and 2 frames
    clip = synth.seeded_clip(T, H, W, 11, shift=(12, 24)).cuda()
    got = pipe.interpolate_sequence(clip)
    assert got.shape == (T - 1, 3, H, W) and bool(torch.isfinite(got).all())
    assert float(got.min()) >= 0.0 and float(got.max()) <= 1.0
    want = pipe(clip[:-1], clip[1:])
    err = float((got - want).abs().max())
    assert err <= 2e-6, (err, _count_excess(got, want, 2e-6))
    tc.check_overflow()


@gpu
def test_cli_writes_the_bytes_of_interpolate_video_host(tmp_path):
    from fvfi import interpolate_video, synth
    H, W, T = 64, 96, 5
    f8 = synth.to_rgb8(synth.seeded_clip(T, H, W, 13, shift=(1, 2)))
    src, dst = tmp_path / "in.rgb", tmp_path / "out.rgb"
    src.write_bytes(f8.numpy().tobytes())
    assert interpolate_video.main(["--size", "%dx%d" % (W, H), "--seeded-weights", "6", "--input", str(src),
                                   "--output", str(dst)]) == 0
    want = _pipe(H, W, seed=6, max_batch=8).interpolate_video_host(f8.pin_memory())
    assert dst.read_bytes() == want.numpy().tobytes()
