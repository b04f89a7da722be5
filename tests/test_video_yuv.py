"""yuv420p clips: the 4:2:0 entry and exit kernels against oracle/yuv.py (exact), their argument checks, interpolate_sequence /
interpolate_video_host with pix_fmt='yuv420p' against the rgb path, and the raw-video CLI with --pix-fmt yuv420p."""
import io

import numpy as np
import pytest
import torch

from oracle import yuv as oy

gpu = pytest.mark.gpu
FORMATS = [("bt709", False), ("bt709", True), ("bt601", False), ("bt601", True)]


@pytest.fixture(autouse=True)
def _strict_fp32():
    """The yuv path and the rgb path are compared in fp32: cuDNN/cuBLAS TF32 off."""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _solid(rgb):
    """A 2x2 frame of one R'G'B' value, planar float32 [1,3,2,2]."""
    return np.broadcast_to(np.asarray(rgb, np.float32)[None, :, None, None], (1, 3, 2, 2)).copy()


def _yuv_of(frames):
    """(Y, U, V) of the top-left block of each frame of a yuv420p clip."""
    f = np.asarray(frames)
    Y, U, V = oy.planes(f)
    return int(Y[0, 0, 0]), int(U[0, 0, 0]), int(V[0, 0, 0])


# ---- CPU: the oracle's known answers, argument checks of the entry points and of the CLI ---------------------------------------

@pytest.mark.parametrize("rgb,matrix,full_range,want", [
    ((1, 0, 0), "bt709", False, (63, 102, 240)),
    ((1, 0, 0), "bt601", False, (81, 90, 240)),
    ((1, 1, 1), "bt709", False, (235, 128, 128)),
    ((1, 1, 1), "bt709", True, (255, 128, 128)),
    ((1, 1, 1), "bt601", True, (255, 128, 128)),
    ((0, 0, 0), "bt709", False, (16, 128, 128)),
    ((0, 0, 0), "bt709", True, (0, 128, 128)),
    ((0, 0, 0), "bt601", False, (16, 128, 128)),
])
def test_oracle_encode_known_answers(rgb, matrix, full_range, want):
    out = oy.encode(_solid(rgb), matrix, full_range)
    assert out.shape == (1, 3, 2) and out.dtype == np.uint8
    assert (out[0, :2] == want[0]).all()
    assert _yuv_of(out) == want


def test_oracle_decode_known_answer():
    red = np.array([63, 63, 63, 63, 102, 240], np.uint8).reshape(1, 3, 2)     # BT.709 limited pure red
    codes = oy.decode(red).astype(int)
    assert codes.shape == (1, 3, 2, 2)
    assert (np.abs(codes - np.array([255, 0, 0])[None, :, None, None]) <= 1).all(), codes[0, :, 0, 0]
    for matrix, full_range in FORMATS:                                        # grey passes through every format unchanged
        grey = oy.encode(_solid((0.5, 0.5, 0.5)), matrix, full_range)
        assert (np.abs(oy.decode(grey, matrix, full_range).astype(int) - 128) <= 1).all()


def test_oracle_chroma_siting():
    """The [1,3]/4 filter in each direction, centre-sited: a single bright chroma sample spreads to the 4x4 luma pixels around
    its block with weights 9, 3, 3, 1 (out of 16)."""
    c = np.zeros((1, 3, 3), np.uint8)
    c[0, 1, 1] = 16
    up = oy._upsample16(c)[0]
    assert up.shape == (6, 6)
    assert up[2:4, 2:4].tolist() == [[144, 144], [144, 144]]
    assert up[1, 2] == up[4, 3] == up[2, 1] == up[3, 4] == 48 and up[1, 1] == up[4, 4] == 16
    assert up[0].sum() == 0 and up[:, 0].sum() == 0


def test_yuv_entry_points_validate_arguments():
    """Null pointers, non-positive or odd sizes, more than 65535 frames, an unknown matrix, a range flag other than 0 / 1 and
    misaligned pointers are rejected with FVFI_EINVAL and a message naming the entry point, before any CUDA call."""
    from fvfi import _lib
    L = _lib.lib()
    dec, enc = L.fvfi_yuv420p_to_rgb_lab, L.fvfi_fusion_blend_yuv420p
    cases = [
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(None, 16, 16, 1, 4, 4, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, None, 16, 1, 4, 4, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, None, 1, 4, 4, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 0, 4, 4, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 1, -4, 4, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 1, 4, 0, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 1, 5, 4, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 1, 4, 7, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 65536, 4, 4, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 1, 4, 4, 2020, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 1, 4, 4, 601, 2, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 16, 16, 1, 4, 4, 601, -1, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(17, 16, 16, 1, 4, 4, 709, 0, None)),
        ("fvfi_yuv420p_to_rgb_lab", lambda: dec(16, 20, 16, 1, 4, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(None, 16, 16, 1, 4, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, None, 16, 1, 4, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, None, 1, 4, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 16, 0, 4, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 16, 1, 0, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 16, 1, 4, -2, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 16, 1, 3, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 16, 1, 4, 5, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 16, 70000, 4, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 16, 1, 4, 4, 0, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 16, 1, 4, 4, 709, 3, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(20, 16, 16, 1, 4, 4, 709, 0, None)),
        ("fvfi_fusion_blend_yuv420p", lambda: enc(16, 16, 17, 1, 4, 4, 709, 0, None)),
    ]
    for name, call in cases:
        rc = call()
        assert rc == 1, (name, rc)                                   # FVFI_EINVAL
        assert name in L.fvfi_last_error().decode(), (name, L.fvfi_last_error())


def test_python_entry_points_validate_formats():
    from fvfi import transform
    assert transform.yuv_args("bt709", False) == (709, 0) and transform.yuv_args("bt601", True) == (601, 1)
    for bad in (("bt2020", False), ("709", False), ("bt709", 2), ("bt709", "pc")):
        with pytest.raises(ValueError):
            transform.yuv_args(*bad)
    assert transform.yuv420p_frame_size(torch.zeros((2, 6, 4), dtype=torch.uint8)) == (4, 4)
    for bad in (torch.zeros((2, 7, 4), dtype=torch.uint8), torch.zeros((2, 6, 5), dtype=torch.uint8),
                torch.zeros((2, 6, 4), dtype=torch.int16), torch.zeros((6, 4), dtype=torch.uint8)):
        with pytest.raises(ValueError):
            transform.yuv420p_frame_size(bad)


def _no_pipeline(monkeypatch):
    from fvfi import pipeline

    def no_cuda(*a, **k):
        raise AssertionError("the CLI built the pipeline before rejecting its input")
    monkeypatch.setattr(pipeline, "FusionPipeline", no_cuda)
    monkeypatch.setattr(torch.cuda, "init", no_cuda)


def _cli_exit(monkeypatch, argv, capsys):
    """Exit code and stderr of the CLI for argv (argparse errors exit with 2 through SystemExit)."""
    from fvfi import interpolate_video
    _no_pipeline(monkeypatch)
    try:
        rc = interpolate_video.main(argv)
    except SystemExit as e:
        rc = e.code
    return rc, capsys.readouterr().err


@pytest.mark.parametrize("argv,msg", [
    (["--size", "7x4", "--pix-fmt", "yuv420p"], "even"),
    (["--size", "6x5", "--pix-fmt", "yuv420p"], "even"),
    (["--size", "6x4", "--matrix", "bt601"], "yuv420p only"),
    (["--size", "6x4", "--pix-fmt", "rgb24", "--range", "pc"], "yuv420p only"),
    (["--size", "6x4", "--pix-fmt", "yuv420p", "--matrix", "bt2020"], "invalid choice"),
    (["--size", "6x4", "--pix-fmt", "nv12"], "invalid choice"),
])
def test_cli_rejects_bad_format_options(monkeypatch, tmp_path, capsys, argv, msg):
    src = tmp_path / "in.yuv"
    src.write_bytes(bytes(6 * 4 * 3 * 4))                                  # four rgb24 6x4 frames, eight yuv420p ones
    rc, err = _cli_exit(monkeypatch, argv + ["--seeded-weights", "0", "--input", str(src), "--output", str(tmp_path / "o")], capsys)
    assert rc == 2 and msg in err, (rc, err)


def test_cli_yuv_options_parse():
    from fvfi import interpolate_video
    a = interpolate_video.parse_args(["--size", "6x4", "--seeded-weights", "0", "--pix-fmt", "yuv420p"])
    assert (a.pix_fmt, a.matrix, a.range) == ("yuv420p", "bt709", "tv")
    a = interpolate_video.parse_args(["--size", "6x4", "--seeded-weights", "0", "--pix-fmt", "yuv420p", "--matrix", "bt601",
                                      "--range", "pc"])
    assert (a.matrix, a.range) == ("bt601", "pc")
    a = interpolate_video.parse_args(["--size", "6x4", "--seeded-weights", "0"])
    assert a.pix_fmt == "rgb24"


@pytest.mark.parametrize("via_pipe", [False, True])
def test_cli_rejects_truncated_and_single_frame_yuv_clips(monkeypatch, tmp_path, capsys, via_pipe):
    fb = 6 * 4 * 3 // 2                                                      # a 6x4 yuv420p frame: 36 bytes

    def run(data):
        if via_pipe:
            monkeypatch.setattr("sys.stdin", io.TextIOWrapper(io.BytesIO(data)))
            src = "-"
        else:
            src = str(tmp_path / "in.yuv")
            open(src, "wb").write(data)
        return _cli_exit(monkeypatch, ["--size", "6x4", "--pix-fmt", "yuv420p", "--seeded-weights", "0", "--input", src,
                                       "--output", str(tmp_path / "out.yuv")], capsys)
    rc, err = run(bytes(fb))                                                 # one frame
    assert rc == 2 and "at least 2" in err
    rc, err = run(bytes(fb + fb // 2))                                       # a frame and a half
    assert rc == 2 and "frame" in err
    if not via_pipe:                                                         # a regular file is sized up front
        rc, err = run(bytes(5 * fb + 7))
        assert rc == 2 and "not a whole number of %d-byte frames" % fb in err


# ---- GPU ------------------------------------------------------------------------------------------------------------------------

def _pipe(H, W, seed=0, max_batch=8):
    from fvfi import synth
    from fvfi.pipeline import FusionPipeline
    pipe = FusionPipeline(H, W, "cuda")
    pipe.load_state(synth.seeded_state(seed))
    pipe.max_batch = max_batch
    return pipe


def _seeded_yuv(T, H, W, seed, shift, matrix="bt709", full_range=False):
    """A seeded constant-motion clip (fvfi.synth.seeded_clip) encoded to yuv420p by the oracle: uint8 [T,3H/2,W] on the host."""
    from fvfi import synth
    return torch.from_numpy(oy.encode(synth.seeded_clip(T, H, W, seed, shift=shift).numpy(), matrix, full_range))


def _codes(rgb):
    """fp32 values k / 255 [T,3,H,W] -> the codes k (uint8, host)."""
    return (rgb.cpu() * 255).round().to(torch.uint8)


@gpu
@pytest.mark.parametrize("matrix,full_range", FORMATS)
@pytest.mark.parametrize("T,H,W", [(1, 2, 2), (2, 38, 54), (1, 1080, 1920), (1, 6, 10)])
def test_yuv420p_to_rgb_lab(T, H, W, matrix, full_range):
    """Random codes plus every Y, U and V code (where a plane holds 256 samples) against the oracle, bit for bit; the Lab equals
    rgb2lab of the RGB bit for bit, and the RGB is exactly k / 255."""
    from fvfi import transform
    g = torch.Generator().manual_seed(T * 7 + H)
    f = torch.randint(0, 256, (T, 3 * H // 2, W), generator=g, dtype=torch.uint8)
    Y, U, V = (torch.from_numpy(p) for p in oy.planes(f.numpy()))
    for k, p in enumerate((Y, U, V)):
        flat = p.reshape(T, -1)
        if flat.shape[1] >= 256:
            flat[0, :256] = torch.roll(torch.arange(256, dtype=torch.uint8), 85 * k)
    f = torch.cat([Y.reshape(T, -1), U.reshape(T, -1), V.reshape(T, -1)], 1).reshape(T, 3 * H // 2, W)
    rgb, lab = transform.yuv420p_to_rgb_lab(f.cuda(), matrix, full_range)
    assert rgb.shape == lab.shape == (T, 3, H, W)
    want = torch.from_numpy(oy.decode(f.numpy(), matrix, full_range))
    assert torch.equal(_codes(rgb), want), int((_codes(rgb).int() - want.int()).abs().max())
    table = (torch.arange(256, dtype=torch.float64) / 255).float()          # correctly rounded k/255
    assert torch.equal(rgb.cpu(), table[want.long()])
    assert torch.equal(lab, transform.rgb2lab(rgb))
    if H * W >= 1024:                                                       # the clamps at both ends are reached
        assert int(want.min()) == 0 and int(want.max()) == 255


@gpu
@pytest.mark.parametrize("matrix,full_range", FORMATS)
@pytest.mark.parametrize("B,H,W", [(2, 38, 54), (1, 1080, 1920), (1, 2, 2)])
def test_fusion_blend_yuv420p(B, H, W, matrix, full_range):
    """The device blend converted by the oracle equals the fused kernel, byte for byte (clamps at 0 and at 1 included)."""
    from fvfi.fusion_net import fusion_blend, fusion_blend_yuv420p
    g = torch.Generator().manual_seed(B * 5 + H)
    base = (torch.rand((B, 3, H, W), generator=g) * 2 - 0.5).cuda()
    x = (torch.randn((B, 3, H, W), generator=g) * 2).cuda()
    want = torch.from_numpy(oy.encode(fusion_blend(base, x).cpu().numpy(), matrix, full_range))
    got = fusion_blend_yuv420p(base, x, matrix=matrix, full_range=full_range)
    assert got.dtype == torch.uint8 and got.shape == (B, 3 * H // 2, W)
    assert torch.equal(got.cpu(), want), int((got.cpu().int() - want.int()).abs().max())
    out = torch.full_like(got, 7)
    assert fusion_blend_yuv420p(base, x, out, matrix, full_range) is out and torch.equal(out, got)


def _rgb_reference(pipe, clip, matrix, full_range):
    """The rgb path of a yuv420p clip: the entry kernel's rgb24 codes as fp32 k / 255 through interpolate_sequence, encoded to
    yuv420p by the oracle."""
    from fvfi import synth, transform
    rgb, _ = transform.yuv420p_to_rgb_lab(clip.cuda(), matrix, full_range)
    decoded = _codes(rgb).permute(0, 2, 3, 1).contiguous()                   # rgb24 [T,H,W,3]
    ref = pipe.interpolate_sequence(synth.rgb8_values(decoded).cuda())
    return torch.from_numpy(oy.encode(ref.cpu().numpy(), matrix, full_range))


@gpu
@pytest.mark.parametrize("H,W,T,mb,matrix,full_range", [(64, 96, 6, 2, "bt709", False), (184, 328, 4, 2, "bt601", True)])
def test_interpolate_sequence_yuv420p_is_the_rgb_path(H, W, T, mb, matrix, full_range):
    """Windows split (max_batch < T - 1): the yuv420p clip path equals the oracle's encoding of the fp32 path on the decoded
    frames, byte for byte."""
    pipe = _pipe(H, W, seed=3, max_batch=mb)
    clip = _seeded_yuv(T, H, W, 7, (3, -4), matrix, full_range)
    got = pipe.interpolate_sequence(clip.cuda(), pix_fmt="yuv420p", matrix=matrix, full_range=full_range)
    assert got.dtype == torch.uint8 and got.shape == (T - 1, 3 * H // 2, W)
    want = _rgb_reference(pipe, clip, matrix, full_range)
    assert torch.equal(got.cpu(), want), int((got.cpu().int() - want.int()).abs().max())


@gpu
def test_interpolate_sequence_rejects_bad_yuv_clips():
    pipe = _pipe(32, 48)
    u8 = dict(dtype=torch.uint8, device="cuda")
    good = torch.zeros((3, 48, 48), **u8)
    assert pipe.interpolate_sequence(good, pix_fmt="yuv420p").shape == (2, 48, 48)
    for bad in (torch.zeros((1, 48, 48), **u8),                                     # T < 2
                torch.zeros((3, 32, 48), **u8),                                     # the Y plane only
                torch.zeros((3, 48, 50), **u8),                                     # frame size
                torch.zeros((3, 32, 48, 3), **u8),                                  # rgb24 layout
                torch.zeros((3, 48, 48), dtype=torch.float32, device="cuda")):      # dtype
        with pytest.raises(ValueError):
            pipe.interpolate_sequence(bad, pix_fmt="yuv420p")
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(good, pix_fmt="nv12")
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(good, pix_fmt="yuv420p", matrix="bt2020")
    with pytest.raises(ValueError):
        pipe.interpolate_video_host(good.cpu(), pix_fmt="yuv420p", out_host=torch.zeros((4, 48, 48), dtype=torch.uint8))
    odd = _pipe(33, 48)
    with pytest.raises(ValueError):
        odd.interpolate_sequence(torch.zeros((3, 49, 48), **u8), pix_fmt="yuv420p")
    with pytest.raises(ValueError):
        odd.interpolate_video_host(torch.zeros((3, 49, 48), dtype=torch.uint8), pix_fmt="yuv420p")


@gpu
@pytest.mark.parametrize("T,mb", [(6, 4), (4, 8)])
def test_interpolate_video_host_yuv420p(T, mb):
    H, W = 64, 96
    pipe = _pipe(H, W, seed=4, max_batch=mb)
    clip = _seeded_yuv(T, H, W, 9, (-2, 5)).pin_memory()
    out = pipe.interpolate_video_host(clip, pix_fmt="yuv420p")
    assert out.shape == (2 * T - 1, 3 * H // 2, W) and out.dtype == torch.uint8 and out.is_pinned()
    assert torch.equal(out[0::2], clip)
    assert torch.equal(out[1::2], pipe.interpolate_sequence(clip.cuda(), pix_fmt="yuv420p").cpu())


@gpu
def test_clip_1080p_large_motion_yuv420p():
    from fvfi import conv as tc
    H, W, T = 1080, 1920, 10
    pipe = _pipe(H, W, seed=0, max_batch=8)                   # windows of 9 and 2 frames
    clip = _seeded_yuv(T, H, W, 11, (12, 24)).pin_memory()
    out = pipe.interpolate_video_host(clip, pix_fmt="yuv420p")
    assert out.shape == (2 * T - 1, 3 * H // 2, W)
    assert torch.equal(out[0::2], clip)
    assert torch.equal(out[1::2], _rgb_reference(pipe, clip, "bt709", False))
    tc.check_overflow()


@gpu
@pytest.mark.parametrize("opts,matrix,full_range", [([], "bt709", False), (["--matrix", "bt601", "--range", "pc"], "bt601", True)])
def test_cli_writes_the_bytes_of_interpolate_video_host_yuv420p(tmp_path, opts, matrix, full_range):
    from fvfi import interpolate_video
    H, W, T = 64, 96, 5
    clip = _seeded_yuv(T, H, W, 13, (1, 2), matrix, full_range)
    src, dst = tmp_path / "in.yuv", tmp_path / "out.yuv"
    src.write_bytes(clip.numpy().tobytes())
    assert interpolate_video.main(["--size", "%dx%d" % (W, H), "--seeded-weights", "6", "--pix-fmt", "yuv420p", "--input", str(src),
                                   "--output", str(dst)] + opts) == 0
    want = _pipe(H, W, seed=6, max_batch=8).interpolate_video_host(clip.pin_memory(), pix_fmt="yuv420p", matrix=matrix,
                                                                   full_range=full_range)
    assert dst.read_bytes() == want.numpy().tobytes()
    assert len(dst.read_bytes()) == (2 * T - 1) * H * W * 3 // 2
