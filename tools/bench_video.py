"""Clip interpolation vs the pair path on the same clip (1080p, 33 frames = 32 pairs, windows of 8 pairs).

    python tools/bench_video.py --out DIR [--runs 5] [--frames 33] [--size 1920x1080] [--batch 8]

Two comparisons, each timed with a host clock around calls that end in a device synchronise, the arms alternating in one
process after every shape was warmed up:
  host     FusionPipeline.interpolate_video_host with 8-bit rgb24 frames in and out (pinned)  vs  the same with a
           SceneCutDetector(10) (scene-cut detection on; the clip is one shot, but its large motion can mark the stream's first
           pair, whose difference is compared with 0)  vs  the same with yuv420p
           frames (pix_fmt='yuv420p', bt709 limited range: the same clip encoded by the exit kernel)  vs
           interpolate_host(frames[:-1], frames[1:]) on the fp32 values k / 255 of the same frames (pinned)
  device   interpolate_sequence on the fp32 clip (Lab and decomposition once per frame and window)  vs  pipe(frames[:-1], frames[1:])
The clip is fvfi.synth.seeded_clip with a large constant motion (12, 24) px per frame.  Writes DIR/bench_video.json with
interpolated frames/s (min / median over the runs), the H2D and D2H bytes per interpolated frame, the max abs difference
between the arms, the per-launch time of the four 8-bit conversion kernels on one window (CUDA events around back-to-back
launches), the same for the three scene-cut kernels (SAD over rgb24 and over the yuv420p Y plane, decision, substitution with
every pair and with no pair cut), and the card name / power limit / max SM clock read in the same process.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "fusion-method-for-video-frame-interpolation_b200")]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()


def kernel_times(torch, rgb, f8, y8, launches=50):
    """Per-launch time of the entry kernels on one window of frames (rgb [n,3,H,W] fp32, the same frames as rgb24 and yuv420p)
    and of the exit kernels on n - 1 frames: CUDA events around ``launches`` back-to-back calls of the C entry points into
    preallocated buffers, after a warm-up.  Algorithmic bytes per pixel: entry 3 (rgb24) or 1.5 (yuv420p) in + 24 out, exit 24 in
    + 3 or 1.5 out."""
    from fvfi import _lib
    L, s = _lib.lib(), _lib.stream_ptr()
    n, _, H, W = rgb.shape
    o_rgb, o_lab = torch.empty_like(rgb), torch.empty_like(rgb)
    base, x = rgb[1:].contiguous(), torch.zeros_like(rgb[1:])
    o8 = torch.empty((n - 1, H, W, 3), dtype=torch.uint8, device=rgb.device)
    oy = torch.empty((n - 1, 3 * H // 2, W), dtype=torch.uint8, device=rgb.device)
    p = lambda t: t.data_ptr()
    calls = {
        "rgb8_to_rgb_lab": (lambda: L.fvfi_rgb8_to_rgb_lab(p(f8), p(o_rgb), p(o_lab), n, H, W, s), n, 27),
        "yuv420p_to_rgb_lab": (lambda: L.fvfi_yuv420p_to_rgb_lab(p(y8), p(o_rgb), p(o_lab), n, H, W, 709, 0, s), n, 25.5),
        "fusion_blend_rgb8": (lambda: L.fvfi_fusion_blend_rgb8(p(base), p(x), p(o8), n - 1, H, W, s), n - 1, 27),
        "fusion_blend_yuv420p": (lambda: L.fvfi_fusion_blend_yuv420p(p(base), p(x), p(oy), n - 1, H, W, 709, 0, s), n - 1, 25.5),
    }
    res = {}
    for name, (fn, frames, bpp) in calls.items():
        for _ in range(3):
            _lib.check(fn())
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(launches):
            fn()
        t1.record()
        t1.synchronize()
        us = t0.elapsed_time(t1) * 1e3 / launches
        res[name] = {"frames": frames, "us_per_launch": us, "us_per_frame": us / frames,
                     "algorithmic_GB_per_s": bpp * H * W * frames / (us * 1e-6) / 1e9}
    return res


def scene_kernel_times(torch, f8, y8, launches=50):
    """Per-launch time of the scene-cut kernels on one window of n frames (f8 rgb24 [n,H,W,3], y8 yuv420p [n,3H/2,W] on the
    device): CUDA events around ``launches`` back-to-back calls of the C entry points, after a warm-up.  Algorithmic bytes: the SAD
    reads each compared byte once (3 HW per rgb24 frame, HW per yuv420p Y plane); the substitution reads and writes one frame per
    cut pair."""
    from fvfi import _lib
    L, s = _lib.lib(), _lib.stream_ptr()
    n, H, W, _ = f8.shape
    P = n - 1
    sad = torch.empty(P, dtype=torch.int64, device=f8.device)
    mafd = torch.empty(P, dtype=torch.float64, device=f8.device)
    cut = torch.empty(P, dtype=torch.uint8, device=f8.device)
    all_cut, no_cut = torch.ones_like(cut), torch.zeros_like(cut)
    out8 = torch.empty((P, H, W, 3), dtype=torch.uint8, device=f8.device)
    p = lambda t: t.data_ptr()
    fb = 3 * H * W
    calls = {
        "frame_sad_u8 rgb24": (lambda: L.fvfi_frame_sad_u8(p(f8), fb, fb, P, p(sad), s), n * fb),
        "frame_sad_u8 yuv420p Y": (lambda: L.fvfi_frame_sad_u8(p(y8), fb // 2, H * W, P, p(sad), s), n * H * W),
        "scene_cut_decide": (lambda: L.fvfi_scene_cut_decide(p(sad), P, fb, None, 10.0, p(mafd), p(cut), s), P * 17),
        "scene_cut_select_u8 rgb24, every pair cut": (lambda: L.fvfi_scene_cut_select_u8(p(f8), fb, p(out8), fb, fb, P, p(all_cut), s),
                                                      2 * P * fb),
        "scene_cut_select_u8 rgb24, no pair cut": (lambda: L.fvfi_scene_cut_select_u8(p(f8), fb, p(out8), fb, fb, P, p(no_cut), s), P),
    }
    res = {}
    for name, (fn, nbytes) in calls.items():
        for _ in range(3):
            _lib.check(fn())
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(launches):
            fn()
        t1.record()
        t1.synchronize()
        us = t0.elapsed_time(t1) * 1e3 / launches
        res[name] = {"pairs": P, "us_per_launch": us, "us_per_pair": us / P, "algorithmic_GB_per_s": nbytes / (us * 1e-6) / 1e9}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for bench_video.json")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--frames", type=int, default=33)
    ap.add_argument("--size", default="1920x1080")
    ap.add_argument("--batch", type=int, default=8)
    a = ap.parse_args()
    import torch
    from fvfi import synth
    from fvfi.fusion_net import fusion_blend_yuv420p
    from fvfi.pipeline import FusionPipeline
    from fvfi.scene import SceneCutDetector
    if not torch.cuda.is_available():
        raise SystemExit("bench_video needs a GPU")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    W, H = (int(v) for v in a.size.split("x"))
    T, mb = a.frames, a.batch
    pairs = T - 1
    pipe = FusionPipeline(H, W, "cuda")
    pipe.load_state(synth.seeded_state(0))
    pipe.max_batch = mb
    f8 = synth.to_rgb8(synth.seeded_clip(T, H, W, 1, shift=(12, 24))).pin_memory()
    f32 = synth.rgb8_values(f8)                                  # the same frames as fp32 k / 255
    h1, h2 = f32[:-1].contiguous().pin_memory(), f32[1:].contiguous().pin_memory()
    d32 = f32.cuda()
    out8 = torch.empty((2 * T - 1, H, W, 3), dtype=torch.uint8).pin_memory()
    out32 = torch.empty((pairs, 3, H, W), dtype=torch.float32).pin_memory()
    # the same frames as yuv420p: the exit kernel with x = 0 encodes base = k / 255 itself (clamp(base + tanh(0)) = base)
    y8 = fusion_blend_yuv420p(d32, torch.zeros_like(d32)).cpu().pin_memory()
    outy = torch.empty((2 * T - 1, 3 * H // 2, W), dtype=torch.uint8).pin_memory()
    out8s = torch.empty_like(out8).pin_memory()

    def sync(fn):
        def run():
            r = fn()
            torch.cuda.synchronize()
            return r
        return run
    arms = {
        "video_host_rgb8": lambda: pipe.interpolate_video_host(f8, out8),
        "video_host_rgb8_scene": lambda: pipe.interpolate_video_host(f8, out8s, scene_cut=SceneCutDetector(10.0)),
        "video_host_yuv420p": lambda: pipe.interpolate_video_host(y8, outy, pix_fmt="yuv420p"),
        "pairs_host_fp32": lambda: pipe.interpolate_host(h1, h2, out32),
        "sequence_device_fp32": sync(lambda: pipe.interpolate_sequence(d32)),
        "pairs_device_fp32": sync(lambda: pipe(d32[:-1], d32[1:])),
    }
    results = {k: arms[k]() for k in arms}                       # warm-up: every shape, plans, packed weights, allocator
    diff_host = float((results["video_host_rgb8"][1::2].permute(0, 3, 1, 2).float() / 255 - results["pairs_host_fp32"]).abs().max())
    diff_dev = float((results["sequence_device_fp32"] - results["pairs_device_fp32"]).abs().max())
    yuv_even_passthrough = bool(torch.equal(results["video_host_yuv420p"][0::2], y8))
    probe = SceneCutDetector(10.0)
    with_scene = pipe.interpolate_video_host(f8, out8s, scene_cut=probe)
    scene_cuts = probe.cuts
    plain = results["video_host_rgb8"]
    scene_check = torch.equal(with_scene[0::2], f8) and all(
        torch.equal(with_scene[2 * p + 1], f8[p] if p in scene_cuts else plain[2 * p + 1]) for p in range(pairs))
    from fvfi import scene
    sad = scene.frame_sad_u8(f8[:3].cuda(), 3 * H * W).cpu().tolist()
    mafd_first = [v * 100.0 / (3 * H * W) / 256.0 for v in sad]
    del results
    times = {k: [] for k in arms}
    for _ in range(a.runs):
        for pair in (("video_host_rgb8", "video_host_rgb8_scene", "video_host_yuv420p", "pairs_host_fp32"),
                     ("sequence_device_fp32", "pairs_device_fp32")):
            for k in pair:
                t0 = time.perf_counter()
                arms[k]()
                times[k].append(time.perf_counter() - t0)
    windows = [min(mb, pairs - s) for s in range(0, pairs, mb)]
    px = H * W
    bytes_ = {
        "video_host_rgb8": {"h2d": sum(b + 1 for b in windows) * px * 3 / pairs, "d2h": px * 3},
        "video_host_rgb8_scene": {"h2d": sum(b + 1 for b in windows) * px * 3 / pairs, "d2h": px * 3},
        "video_host_yuv420p": {"h2d": sum(b + 1 for b in windows) * px * 3 / 2 / pairs, "d2h": px * 3 / 2},
        "pairs_host_fp32": {"h2d": 2 * 3 * px * 4, "d2h": 3 * px * 4},
        "sequence_device_fp32": {"h2d": 0, "d2h": 0},
        "pairs_device_fp32": {"h2d": 0, "d2h": 0},
    }
    rec = {"card_csv": card(), "size": [W, H], "frames": T, "pairs": pairs, "max_batch": mb, "windows": windows,
           "clip": "fvfi.synth.seeded_clip(seed=1, shift=(12, 24)), 8-bit", "timing": "host clock around calls ending in a synchronise",
           "runs": a.runs, "arms": {}}
    for k, ts in times.items():
        rec["arms"][k] = {"seconds": [round(t, 5) for t in ts],
                          "frames_per_s_median": pairs / statistics.median(ts), "frames_per_s_min": pairs / max(ts),
                          "frames_per_s_max": pairs / min(ts), "spread_pct": 100 * (max(ts) - min(ts)) / statistics.median(ts),
                          "h2d_bytes_per_frame": bytes_[k]["h2d"], "d2h_bytes_per_frame": bytes_[k]["d2h"]}
    rec["max_abs_diff"] = {"video_host_rgb8/255 vs pairs_host_fp32": diff_host, "sequence_device vs pairs_device": diff_dev}
    rec["yuv420p_even_slots_are_the_input"] = yuv_even_passthrough
    rec["scene_cuts_found"] = scene_cuts
    rec["scene_mafd_first_two_pairs"] = mafd_first
    rec["scene_arm_is_plain_arm_with_cut_frames_repeated"] = scene_check
    rec["conversion_kernels"] = kernel_times(torch, d32[:mb + 1], f8[:mb + 1].cuda(), y8[:mb + 1].cuda())
    rec["scene_kernels"] = scene_kernel_times(torch, f8[:mb + 1].cuda(), y8[:mb + 1].cuda())
    rec["speedup_median"] = {"host": rec["arms"]["video_host_rgb8"]["frames_per_s_median"] / rec["arms"]["pairs_host_fp32"]["frames_per_s_median"],
                             "host_yuv420p_vs_rgb8": rec["arms"]["video_host_yuv420p"]["frames_per_s_median"]
                             / rec["arms"]["video_host_rgb8"]["frames_per_s_median"],
                             "host_scene_vs_rgb8": rec["arms"]["video_host_rgb8_scene"]["frames_per_s_median"]
                             / rec["arms"]["video_host_rgb8"]["frames_per_s_median"],
                             "device": rec["arms"]["sequence_device_fp32"]["frames_per_s_median"] / rec["arms"]["pairs_device_fp32"]["frames_per_s_median"]}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_video.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
