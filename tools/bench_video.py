"""Clip interpolation vs the pair path on the same clip (1080p, 33 frames = 32 pairs, windows of 8 pairs).

    python tools/bench_video.py --out DIR [--runs 5] [--frames 33] [--size 1920x1080] [--batch 8]

Two comparisons, each timed with a host clock around calls that end in a device synchronise, the two arms alternating in one
process after every shape was warmed up:
  host     FusionPipeline.interpolate_video_host (8-bit rgb24 frames in and out, pinned)  vs
           interpolate_host(frames[:-1], frames[1:]) on the fp32 values k / 255 of the same frames (pinned)
  device   interpolate_sequence on the fp32 clip (Lab and decomposition once per frame and window)  vs  pipe(frames[:-1], frames[1:])
The clip is fvfi.synth.seeded_clip with a large constant motion (12, 24) px per frame.  Writes DIR/bench_video.json with
interpolated frames/s (min / median over the runs), the H2D and D2H bytes per interpolated frame, the max abs difference
between the arms, and the card name / power limit / max SM clock read in the same process.
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
    from fvfi.pipeline import FusionPipeline
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

    def sync(fn):
        def run():
            r = fn()
            torch.cuda.synchronize()
            return r
        return run
    arms = {
        "video_host_rgb8": lambda: pipe.interpolate_video_host(f8, out8),
        "pairs_host_fp32": lambda: pipe.interpolate_host(h1, h2, out32),
        "sequence_device_fp32": sync(lambda: pipe.interpolate_sequence(d32)),
        "pairs_device_fp32": sync(lambda: pipe(d32[:-1], d32[1:])),
    }
    results = {k: arms[k]() for k in arms}                       # warm-up: every shape, plans, packed weights, allocator
    diff_host = float((results["video_host_rgb8"][1::2].permute(0, 3, 1, 2).float() / 255 - results["pairs_host_fp32"]).abs().max())
    diff_dev = float((results["sequence_device_fp32"] - results["pairs_device_fp32"]).abs().max())
    del results
    times = {k: [] for k in arms}
    for _ in range(a.runs):
        for pair in (("video_host_rgb8", "pairs_host_fp32"), ("sequence_device_fp32", "pairs_device_fp32")):
            for k in pair:
                t0 = time.perf_counter()
                arms[k]()
                times[k].append(time.perf_counter() - t0)
    windows = [min(mb, pairs - s) for s in range(0, pairs, mb)]
    px = H * W
    bytes_ = {
        "video_host_rgb8": {"h2d": sum(b + 1 for b in windows) * px * 3 / pairs, "d2h": px * 3},
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
    rec["speedup_median"] = {"host": rec["arms"]["video_host_rgb8"]["frames_per_s_median"] / rec["arms"]["pairs_host_fp32"]["frames_per_s_median"],
                             "device": rec["arms"]["sequence_device_fp32"]["frames_per_s_median"] / rec["arms"]["pairs_device_fp32"]["frames_per_s_median"]}
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "bench_video.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
