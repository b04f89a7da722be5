"""Scene-cut detection on 8-bit clips: the rule of oracle/scene.py (known answers), the argument checks of the three entry points
and of the CLI, the SAD / decide / select kernels against the oracle (exact), and interpolate_sequence / interpolate_video_host /
the CLI with a SceneCutDetector on clips with cuts: the cut list, the repeated frames, every other frame unchanged, independence
from the window size and the call split, and the range guard's second run."""
import math

import numpy as np
import pytest
import torch

from oracle import scene as osc
from oracle import yuv as oy

gpu = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _strict_fp32():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _yuv_solid(T, H, W, ys):
    """A yuv420p clip [T,3H/2,W] whose frame t has Y = ys[t] everywhere and neutral chroma."""
    f = np.full((T, 3 * H // 2, W), 128, np.uint8)
    for t, y in enumerate(ys):
        f[t, :H] = y
    return f


# ---- CPU: the oracle's known answers -----------------------------------------------------------------------------------------

def test_oracle_identical_frames():
    f = np.random.default_rng(0).integers(0, 256, (1, 6, 8, 3), dtype=np.uint8).repeat(4, 0)
    assert osc.sad(f, "rgb24").tolist() == [0, 0, 0]
    cuts, m = osc.detect(f, "rgb24", 10.0)
    assert cuts == [] and m.tolist() == [0.0, 0.0, 0.0]


def test_oracle_black_to_white_limited_range():
    H, W = 4, 6
    f = _yuv_solid(2, H, W, [16, 235])
    assert osc.sad(f, "yuv420p").tolist() == [219 * H * W]
    cuts, m = osc.detect(f, "yuv420p", 10.0)
    assert m[0] == 219 * 100 / 256 and cuts == [0]


def test_oracle_first_pair_prev_is_zero():
    f = _yuv_solid(2, 4, 4, [16, 56])                                # mafd = 40 * 100 / 256 = 15.625
    m, cut = osc.decide(osc.sad(f, "yuv420p"), 16, 10.0)
    assert m[0] == 15.625 and cut.tolist() == [True]                  # score = min(15.625, |15.625 - 0|)
    m, cut = osc.decide(osc.sad(f, "yuv420p"), 16, 10.0, prev=15.625)
    assert cut.tolist() == [False]                                    # the same pair after an equal difference: no jump


def test_oracle_consecutive_high_differences_cut_once():
    f = _yuv_solid(4, 4, 4, [16, 235, 16, 16])
    cuts, m = osc.detect(f, "yuv420p", 10.0)
    assert m[0] == m[1] == 219 * 100 / 256 and m[2] == 0
    assert cuts == [0]                                               # pair 1: min(85.5, |85.5 - 85.5|) = 0


def test_oracle_threshold_zero_marks_every_pair():
    f = np.random.default_rng(1).integers(0, 256, (5, 4, 6, 3), dtype=np.uint8)
    f[2] = f[1]
    assert osc.detect(f, "rgb24", 0.0)[0] == [0, 1, 2, 3]


def test_oracle_substitute():
    f = np.arange(4 * 6, dtype=np.uint8).reshape(4, 6)
    mid = np.full((3, 6), 200, np.uint8)
    out = osc.substitute(f, mid, [0, 2])
    assert (out[0] == f[0]).all() and (out[1] == 200).all() and (out[2] == f[2]).all()


# ---- CPU: argument checks ------------------------------------------------------------------------------------------------------

def test_scene_entry_points_validate_arguments():
    """Null pointers, pairs outside [1, 65535], n == 0 or n > stride, frame_bytes beyond a stride and a negative or NaN threshold
    are rejected with FVFI_EINVAL and a message naming the entry point, before any CUDA call."""
    from fvfi import _lib
    L = _lib.lib()
    sad, dec, sel = L.fvfi_frame_sad_u8, L.fvfi_scene_cut_decide, L.fvfi_scene_cut_select_u8
    cases = [
        ("fvfi_frame_sad_u8", lambda: sad(None, 64, 64, 1, 16, None)),
        ("fvfi_frame_sad_u8", lambda: sad(16, 64, 64, 1, None, None)),
        ("fvfi_frame_sad_u8", lambda: sad(16, 64, 64, 0, 16, None)),
        ("fvfi_frame_sad_u8", lambda: sad(16, 64, 64, -3, 16, None)),
        ("fvfi_frame_sad_u8", lambda: sad(16, 64, 64, 65536, 16, None)),
        ("fvfi_frame_sad_u8", lambda: sad(16, 64, 0, 1, 16, None)),
        ("fvfi_frame_sad_u8", lambda: sad(16, 64, 65, 1, 16, None)),
        ("fvfi_scene_cut_decide", lambda: dec(None, 1, 64, None, 10.0, 16, 16, None)),
        ("fvfi_scene_cut_decide", lambda: dec(16, 1, 64, None, 10.0, None, 16, None)),
        ("fvfi_scene_cut_decide", lambda: dec(16, 1, 64, None, 10.0, 16, None, None)),
        ("fvfi_scene_cut_decide", lambda: dec(16, 0, 64, None, 10.0, 16, 16, None)),
        ("fvfi_scene_cut_decide", lambda: dec(16, 65536, 64, None, 10.0, 16, 16, None)),
        ("fvfi_scene_cut_decide", lambda: dec(16, 1, 0, None, 10.0, 16, 16, None)),
        ("fvfi_scene_cut_decide", lambda: dec(16, 1, 64, None, -0.5, 16, 16, None)),
        ("fvfi_scene_cut_decide", lambda: dec(16, 1, 64, None, math.nan, 16, 16, None)),
        ("fvfi_scene_cut_select_u8", lambda: sel(None, 64, 16, 64, 64, 1, 16, None)),
        ("fvfi_scene_cut_select_u8", lambda: sel(16, 64, None, 64, 64, 1, 16, None)),
        ("fvfi_scene_cut_select_u8", lambda: sel(16, 64, 16, 64, 64, 1, None, None)),
        ("fvfi_scene_cut_select_u8", lambda: sel(16, 64, 16, 64, 64, 0, 16, None)),
        ("fvfi_scene_cut_select_u8", lambda: sel(16, 64, 16, 64, 64, 65536, 16, None)),
        ("fvfi_scene_cut_select_u8", lambda: sel(16, 64, 16, 64, 0, 1, 16, None)),
        ("fvfi_scene_cut_select_u8", lambda: sel(16, 32, 16, 64, 64, 1, 16, None)),
        ("fvfi_scene_cut_select_u8", lambda: sel(16, 64, 16, 48, 64, 1, 16, None)),
    ]
    for name, call in cases:
        rc = call()
        assert rc == 1, (name, rc)                                   # FVFI_EINVAL
        assert name in L.fvfi_last_error().decode(), (name, L.fvfi_last_error())


def test_detector_validates_threshold():
    from fvfi.scene import SceneCutDetector
    d = SceneCutDetector()
    assert d.threshold == 10.0 and d.cuts == [] and d.prev is None and d.pairs_seen == 0
    assert SceneCutDetector(0).threshold == 0.0
    for bad in (-1, math.nan, math.inf, "ten", None):
        with pytest.raises(ValueError):
            SceneCutDetector(bad)


def _cli_exit(monkeypatch, argv, capsys):
    """Exit code and stderr of the CLI for argv, with the pipeline and CUDA initialisation made to fail if they are reached."""
    from fvfi import interpolate_video, pipeline

    def no_cuda(*a, **k):
        raise AssertionError("the CLI built the pipeline before rejecting its arguments")
    monkeypatch.setattr(pipeline, "FusionPipeline", no_cuda)
    monkeypatch.setattr(torch.cuda, "init", no_cuda)
    try:
        rc = interpolate_video.main(argv)
    except SystemExit as e:
        rc = e.code
    return rc, capsys.readouterr().err


@pytest.mark.parametrize("opts,msg", [
    (["--scene-log", "cuts.txt"], "--scene-log needs --scene-threshold"),
    (["--scene-threshold", "-1"], "--scene-threshold"),
    (["--scene-threshold", "ten"], "--scene-threshold"),
    (["--scene-threshold", "nan"], "--scene-threshold"),
    (["--scene-threshold", "inf"], "--scene-threshold"),
])
def test_cli_rejects_bad_scene_options(monkeypatch, tmp_path, capsys, opts, msg):
    src = tmp_path / "in.rgb"
    src.write_bytes(bytes(6 * 4 * 3 * 4))
    rc, err = _cli_exit(monkeypatch, ["--size", "6x4", "--seeded-weights", "0", "--input", str(src),
                                      "--output", str(tmp_path / "o")] + opts, capsys)
    assert rc == 2 and msg in err, (rc, err)
    assert not (tmp_path / "o").exists()


def test_cli_scene_options_parse():
    from fvfi import interpolate_video
    a = interpolate_video.parse_args(["--size", "6x4", "--seeded-weights", "0"])
    assert a.scene_threshold is None and a.scene_log is None
    a = interpolate_video.parse_args(["--size", "6x4", "--seeded-weights", "0", "--scene-threshold", "12.5", "--scene-log", "c.txt"])
    assert a.scene_threshold == 12.5 and a.scene_log == "c.txt"
    assert interpolate_video.parse_args(["--size", "6x4", "--seeded-weights", "0", "--scene-threshold", "0"]).scene_threshold == 0.0


# ---- GPU: the kernels ----------------------------------------------------------------------------------------------------------

def _every_byte_frames(T, L, seed):
    """[T, L] uint8: random bytes, with every byte value in frame 0 and (reversed) in the last frame where L >= 256."""
    f = np.random.default_rng(seed).integers(0, 256, (T, L), dtype=np.uint8)
    if L >= 256:
        f[0, :256] = np.arange(256)
        f[-1, :256] = np.arange(256)[::-1]
    return f


@gpu
@pytest.mark.parametrize("pix_fmt,H,W,T", [
    ("rgb24", 37, 53, 17), ("rgb24", 184, 328, 9), ("rgb24", 1080, 1920, 17),
    ("yuv420p", 184, 328, 17), ("yuv420p", 1080, 1920, 9), ("yuv420p", 38, 54, 2),
])
def test_frame_sad_matches_oracle(pix_fmt, H, W, T):
    from fvfi import scene
    shape = (H, W, 3) if pix_fmt == "rgb24" else (3 * H // 2, W)
    f = _every_byte_frames(T, int(np.prod(shape)), H + T).reshape((T,) + shape)
    n = 3 * H * W if pix_fmt == "rgb24" else H * W
    sad = torch.full((T - 1,), -7, dtype=torch.int64, device="cuda")              # the call zeroes its output
    got = scene.frame_sad_u8(torch.from_numpy(f).cuda(), n, sad)
    assert got is sad
    assert got.cpu().numpy().tolist() == osc.sad(f, pix_fmt).tolist()


@gpu
@pytest.mark.parametrize("n,stride,offset,T", [(37 * 53, 2941, 0, 17), (37 * 53, 2941, 3, 5), (4096, 6144, 1, 3), (4096, 6144, 0, 17),
                                               (15, 16, 0, 4), (1, 1, 0, 9)])
def test_frame_sad_unaligned_and_tails(n, stride, offset, T):
    """The byte path (odd stride or base) and the tail of n % 16 bytes: a Y plane of n bytes in frames `stride` bytes apart."""
    from fvfi import scene
    raw = _every_byte_frames(1, offset + T * stride, n + T)[0]
    buf = torch.from_numpy(raw).cuda()
    frames = buf[offset:].as_strided((T, stride), (stride, 1))
    want = np.abs(raw[offset:].reshape(T, stride)[:, :n].astype(np.int64)[1:] - raw[offset:].reshape(T, stride)[:, :n][:-1]).sum(1)
    assert scene.frame_sad_u8(frames, n).cpu().tolist() == want.tolist()


def _bits(x):
    return np.asarray(x, np.float64).view(np.int64)


@gpu
@pytest.mark.parametrize("P,n", [(1, 16), (8, 3 * 1920 * 1080), (300, 37 * 53), (65535, 1920 * 1080)])
def test_decide_matches_oracle(P, n):
    """mafd bit for bit and the cut flags exactly, without and with a carried prev, at thresholds that include exact ties."""
    from fvfi import scene
    rng = np.random.default_rng(P)
    sad = rng.integers(0, 255 * n + 1, P, dtype=np.int64)
    sad[rng.random(P) < 0.5] //= 20                                       # low and high differences next to each other
    m_ref, _ = osc.decide(sad, n, 0.0)
    thresholds = [0.0, 10.0, 33.3, float(np.clip(np.minimum(m_ref, np.abs(m_ref - np.r_[0.0, m_ref[:-1]])), 0, 100)[P // 2])]
    dsad = torch.from_numpy(sad).cuda()
    for prev in (None, 12.345678):
        dprev = None if prev is None else torch.tensor([prev], dtype=torch.float64, device="cuda")
        for thr in thresholds:
            m, cut = scene.scene_cut_decide(dsad, n, thr, dprev)
            want_m, want_cut = osc.decide(sad, n, thr, prev)
            assert (_bits(m.cpu().numpy()) == _bits(want_m)).all()
            assert (cut.cpu().numpy() == want_cut.astype(np.uint8)).all(), (prev, thr)


@gpu
@pytest.mark.parametrize("L,out_pad,offset", [(184 * 328 * 3, 0, 0), (37 * 53 * 3, 0, 0), (4096, 48, 0), (4096, 0, 1), (1080 * 1920 * 3, 0, 0)])
def test_select_copies_cut_frames_only(L, out_pad, offset):
    from fvfi import scene
    P = 9
    frames = torch.from_numpy(_every_byte_frames(P + 1, L, L)).cuda()
    cut = torch.tensor([1, 0, 0, 1, 1, 0, 1, 0, 1], dtype=torch.uint8, device="cuda")
    store = torch.full((offset + P * (L + out_pad),), 0xA5, dtype=torch.uint8, device="cuda")     # sentinel
    out = store[offset:].as_strided((P, L), (L + out_pad, 1))
    scene.scene_cut_select_u8(frames, out, cut)
    host = store.cpu()
    for p in range(P):
        row = host[offset + p * (L + out_pad):offset + p * (L + out_pad) + L]
        assert torch.equal(row, frames[p].cpu()) if cut[p] else bool((row == 0xA5).all()), p
        assert bool((host[offset + p * (L + out_pad) + L:offset + (p + 1) * (L + out_pad)] == 0xA5).all())
    assert bool((host[:offset] == 0xA5).all())


# ---- GPU: the clip paths -------------------------------------------------------------------------------------------------------

H, W = 64, 96
# shots of the test clip: (first frame, brightness offset); each shot is a seeded constant-motion clip at 0.2 of the range plus its
# offset, so a shot change moves every byte by about the offset difference and the motion inside a shot moves it a little
SHOTS = [(0, 0.6), (1, 0.0), (4, 0.6), (6, 0.0), (8, 0.2), (9, 0.8), (10, 0.5)]
T_CLIP = 13
# pairs 0 (the stream's first), 3 and 5 (first and last of the second 3-pair window), 7, 8 and 9 (consecutive: the difference jumps
# from ~2 to ~20 to ~60 and falls to ~30); 9 is also the first pair of the second call when the clip is split at frame 9
CUTS = [0, 3, 5, 7, 8, 9]
SPLIT = 9
_PIPES = {}


def _pipe(max_batch):
    from fvfi import synth
    from fvfi.pipeline import FusionPipeline
    if "pipe" not in _PIPES:
        p = FusionPipeline(H, W, "cuda")
        p.load_state(synth.seeded_state(5))
        _PIPES["pipe"] = p
    _PIPES["pipe"].max_batch = max_batch
    return _PIPES["pipe"]


def _clip(pix_fmt):
    """uint8 host clip with cuts at CUTS: rgb24 [T,H,W,3] or yuv420p [T,3H/2,W]."""
    from fvfi import synth
    bounds = [s for s, _ in SHOTS] + [T_CLIP]
    parts = [synth.seeded_clip(bounds[k + 1] - s, H, W, 20 + k, shift=(1, 2)) * 0.2 + off for k, (s, off) in enumerate(SHOTS)]
    clip = torch.cat(parts).clamp(0, 1)
    if pix_fmt == "yuv420p":
        return torch.from_numpy(oy.encode(clip.numpy()))
    return synth.to_rgb8(clip)


def _fmt(pix_fmt):
    return {"pix_fmt": "yuv420p"} if pix_fmt == "yuv420p" else {}


def test_test_clip_has_the_intended_cuts():
    for pix_fmt in ("rgb24", "yuv420p"):
        cuts, m = osc.detect(_clip(pix_fmt).numpy(), pix_fmt, 10.0)
        assert cuts == CUTS, (pix_fmt, cuts, m)


def _check_stream(frames, got, ref, cuts):
    """got: interpolated frames with the detector, ref: the same call without it."""
    for p in range(got.shape[0]):
        if p in cuts:
            assert torch.equal(got[p], frames[p]), p
        else:
            assert torch.equal(got[p], ref[p]), p


@gpu
@pytest.mark.parametrize("pix_fmt", ["rgb24", "yuv420p"])
@pytest.mark.parametrize("mb", [1, 3, 8])
def test_interpolate_sequence_scene_cuts(pix_fmt, mb):
    from fvfi.scene import SceneCutDetector
    pipe = _pipe(mb)
    clip = _clip(pix_fmt)
    dev = clip.cuda()
    want, mafd = osc.detect(clip.numpy(), pix_fmt, 10.0)
    ref = pipe.interpolate_sequence(dev, **_fmt(pix_fmt)).cpu()
    d = SceneCutDetector(10.0)
    got = pipe.interpolate_sequence(dev, scene_cut=d, **_fmt(pix_fmt)).cpu()
    assert d.cuts == want == CUTS and d.pairs_seen == T_CLIP - 1
    assert _bits(d.prev.cpu().numpy()) == _bits(mafd[-1:])
    _check_stream(clip, got, ref, want)
    # two calls sharing the detector: the carry crosses the boundary (pair SPLIT is the first pair of the second call)
    d2 = SceneCutDetector(10.0)
    a = pipe.interpolate_sequence(dev[:SPLIT + 1], scene_cut=d2, **_fmt(pix_fmt))
    b = pipe.interpolate_sequence(dev[SPLIT:], scene_cut=d2, **_fmt(pix_fmt))
    assert d2.cuts == want and d2.pairs_seen == T_CLIP - 1
    assert _bits(d2.prev.cpu().numpy()) == _bits(mafd[-1:])
    got2 = torch.cat((a, b)).cpu()
    if SPLIT % mb == 0:                         # the same windows: the same bytes
        assert torch.equal(got2, got)
    for p in want:
        assert torch.equal(got2[p], clip[p])


@gpu
def test_carry_decides_the_first_pair_of_a_call():
    """A call that starts right after a cut with an equally large difference is no cut with the carry, and is one on a fresh
    detector (prev = 0): the carry, not the call boundary, decides."""
    from fvfi.scene import SceneCutDetector
    pipe = _pipe(3)
    f = torch.from_numpy(_yuv_solid(3, H, W, [16, 235, 16])).cuda()
    d = SceneCutDetector(10.0)
    first = pipe.interpolate_sequence(f[:2], pix_fmt="yuv420p", scene_cut=d)
    second = pipe.interpolate_sequence(f[1:], pix_fmt="yuv420p", scene_cut=d)
    assert d.cuts == [0] and d.pairs_seen == 2
    assert torch.equal(first[0], f[0])
    assert torch.equal(second, pipe.interpolate_sequence(f[1:], pix_fmt="yuv420p"))     # pair 1: no jump, interpolated
    fresh = SceneCutDetector(10.0)
    alone = pipe.interpolate_sequence(f[1:], pix_fmt="yuv420p", scene_cut=fresh)
    assert fresh.cuts == [0] and torch.equal(alone[0], f[1])
    d.reset()
    assert d.cuts == [] and d.prev is None and d.pairs_seen == 0


@gpu
@pytest.mark.parametrize("pix_fmt", ["rgb24", "yuv420p"])
def test_interpolate_video_host_scene_cuts(pix_fmt):
    from fvfi.scene import SceneCutDetector
    pipe = _pipe(3)
    clip = _clip(pix_fmt).pin_memory()
    ref = pipe.interpolate_video_host(clip, **_fmt(pix_fmt)).clone()
    d = SceneCutDetector(10.0)
    out = pipe.interpolate_video_host(clip, scene_cut=d, **_fmt(pix_fmt))
    assert d.cuts == CUTS
    assert torch.equal(out[0::2], clip)
    _check_stream(clip, out[1::2], ref[1::2], CUTS)
    for p in CUTS:
        assert torch.equal(out[2 * p + 1], out[2 * p])
    # the same stream in two calls with one detector, as the CLI's segments do
    d2 = SceneCutDetector(10.0)
    a = pipe.interpolate_video_host(clip[:SPLIT + 1], scene_cut=d2, **_fmt(pix_fmt)).clone()
    b = pipe.interpolate_video_host(clip[SPLIT:], scene_cut=d2, **_fmt(pix_fmt))
    assert d2.cuts == CUTS
    assert torch.equal(torch.cat((a, b[1:])), out)
    # the device path gives the same frames
    seq = pipe.interpolate_sequence(clip.cuda(), scene_cut=SceneCutDetector(10.0), **_fmt(pix_fmt)).cpu()
    assert torch.equal(out[1::2], seq)


@gpu
@pytest.mark.parametrize("host", [False, True])
def test_range_guard_rerun_counts_once(monkeypatch, host):
    """The 3xFP16 range guard runs a call a second time when a convolution left the range; the detector must come out as if the
    call had run once.  The flag is reported raised once, which selects the 3xTF32 re-run."""
    from fvfi import conv as tc
    from fvfi.scene import SceneCutDetector
    pipe = _pipe(3)
    clip = _clip("rgb24")
    src = clip.pin_memory() if host else clip.cuda()
    call = pipe.interpolate_video_host if host else pipe.interpolate_sequence

    def run(d):
        call(src[:SPLIT + 1], scene_cut=d)
        call(src[SPLIT:], scene_cut=d)
        return d
    ref = run(SceneCutDetector(10.0))
    real, fired = tc.overflow_pending, []

    def once():
        hit = real()
        if not fired:
            fired.append(1)
            return True
        return hit
    d = SceneCutDetector(10.0)
    call(src[:SPLIT + 1], scene_cut=d)
    monkeypatch.setattr(tc, "overflow_pending", once)
    out = call(src[SPLIT:], scene_cut=d)
    monkeypatch.setattr(tc, "overflow_pending", real)
    assert fired == [1]
    assert d.cuts == ref.cuts == CUTS and d.pairs_seen == ref.pairs_seen == T_CLIP - 1
    assert _bits(d.prev.cpu().numpy()) == _bits(ref.prev.cpu().numpy())
    frames_out = out[1::2] if host else out.cpu()
    assert torch.equal(frames_out[0], clip[SPLIT])                 # pair SPLIT is a cut: frame SPLIT repeated


@gpu
def test_float32_clip_with_detector_is_rejected():
    from fvfi import synth
    from fvfi.scene import SceneCutDetector
    pipe = _pipe(3)
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(synth.seeded_clip(3, H, W, 0).cuda(), scene_cut=SceneCutDetector())
    with pytest.raises(ValueError):
        pipe.interpolate_sequence(_clip("rgb24")[:3].cuda(), scene_cut=10.0)


@gpu
@pytest.mark.parametrize("pix_fmt", ["rgb24", "yuv420p"])
def test_cli_scene_threshold(tmp_path, pix_fmt):
    """--batch 2: segments of 8 pairs, so the 12-pair clip takes two segments and pair 8 (a cut) is the first of the second."""
    from fvfi import interpolate_video
    from fvfi.scene import SceneCutDetector
    clip = _clip(pix_fmt)
    src, log = tmp_path / "in.raw", tmp_path / "cuts.txt"
    src.write_bytes(clip.numpy().tobytes())
    base = ["--size", "%dx%d" % (W, H), "--seeded-weights", "5", "--batch", "2", "--pix-fmt", pix_fmt, "--input", str(src)]
    assert interpolate_video.main(base + ["--output", str(tmp_path / "cut.raw"), "--scene-threshold", "10",
                                          "--scene-log", str(log)]) == 0
    assert interpolate_video.main(base + ["--output", str(tmp_path / "plain.raw")]) == 0
    pipe = _pipe(2)
    d = SceneCutDetector(10.0)
    want = pipe.interpolate_video_host(clip.pin_memory(), scene_cut=d, **_fmt(pix_fmt))
    assert (tmp_path / "cut.raw").read_bytes() == want.numpy().tobytes()
    assert log.read_text().split() == [str(p) for p in CUTS] and d.cuts == CUTS
    plain = pipe.interpolate_video_host(clip.pin_memory(), **_fmt(pix_fmt))
    assert (tmp_path / "plain.raw").read_bytes() == plain.numpy().tobytes()
