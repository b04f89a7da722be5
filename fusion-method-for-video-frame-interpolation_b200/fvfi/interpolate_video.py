"""Frame-rate doubling of raw 8-bit video: reads rgb24 frames, writes rgb24 frames at twice the frame rate (the input frames
with an interpolated frame between every two of them), so it sits between two ffmpeg pipes:

    ffmpeg -i in.mp4 -f rawvideo -pix_fmt rgb24 - \\
      | python -m fvfi.interpolate_video --size 1920x1080 --state weights.pt \\
      | ffmpeg -f rawvideo -pix_fmt rgb24 -s 1920x1080 -r 60 -i - out.mp4

``--state`` is a ``torch.save`` of {"phase_net", "fusion_net", "adacof"} state dicts; ``--seeded-weights SEED`` uses the
seeded random initialisation of fvfi.synth instead (tests, benchmarks).  The clip is streamed in segments of a few windows
of ``--batch`` pairs, so host and device memory stay bounded for any length.  A regular input file whose size is not a
whole number of frames, or that holds fewer than 2 frames, is rejected before any CUDA work; on a pipe, fewer than 2 frames
are rejected the same way and a partial last frame is an error when the stream ends.
"""
import argparse
import os
import sys

WINDOWS_PER_SEGMENT = 4      # windows of --batch pairs handed to interpolate_video_host per call (uploads overlap compute inside it)


class ClipError(ValueError):
    pass


def _parse_size(s):
    try:
        w, h = (int(v) for v in s.lower().split("x"))
    except ValueError:
        raise argparse.ArgumentTypeError("--size is WxH, e.g. 1920x1080")
    if w <= 0 or h <= 0:
        raise argparse.ArgumentTypeError("--size must be positive")
    return w, h


def parse_args(argv=None):
    ap = argparse.ArgumentParser(prog="python -m fvfi.interpolate_video", description=__doc__.split("\n\n")[0])
    ap.add_argument("--size", type=_parse_size, required=True, help="frame size WxH of the rgb24 stream")
    ap.add_argument("--batch", type=int, default=8, help="frame pairs per window (FusionPipeline.max_batch)")
    w = ap.add_mutually_exclusive_group(required=True)
    w.add_argument("--state", help="torch.save of {'phase_net', 'fusion_net', 'adacof'} state dicts")
    w.add_argument("--seeded-weights", type=int, metavar="SEED", help="seeded random weights (fvfi.synth.seeded_state)")
    ap.add_argument("--input", default="-", help="raw rgb24 input file, or - for stdin")
    ap.add_argument("--output", default="-", help="raw rgb24 output file, or - for stdout")
    a = ap.parse_args(argv)
    if a.batch < 1:
        ap.error("--batch must be at least 1")
    return a


def _read_into(f, view):
    """Fills the byte view from f as far as the stream goes; returns the number of bytes read."""
    n = 0
    while n < len(view):
        k = f.readinto(view[n:])
        if not k:
            break
        n += k
    return n


def _check_regular_file(f, frame_bytes):
    try:
        st = os.fstat(f.fileno())
    except (AttributeError, OSError, ValueError):
        return
    import stat
    if not stat.S_ISREG(st.st_mode):
        return
    size = st.st_size - f.tell()
    if size % frame_bytes:
        raise ClipError("input holds %d bytes, not a whole number of %d-byte frames" % (size, frame_bytes))
    if size // frame_bytes < 2:
        raise ClipError("input holds %d frame(s); interpolation needs at least 2" % (size // frame_bytes))


def run(args, fin, fout):
    W, H = args.size
    frame_bytes = H * W * 3
    _check_regular_file(fin, frame_bytes)
    seg = args.batch * WINDOWS_PER_SEGMENT             # pairs per segment
    import numpy as np
    head = np.empty((2, H, W, 3), dtype=np.uint8)      # the first two frames decide "at least 2 frames" before CUDA is touched
    n = _read_into(fin, memoryview(head).cast("B"))
    if n < 2 * frame_bytes:
        if n % frame_bytes:
            raise ClipError("stream ends inside frame %d (%d bytes; frames are %d bytes)" % (n // frame_bytes, n, frame_bytes))
        raise ClipError("stream holds %d frame(s); interpolation needs at least 2" % (n // frame_bytes))

    import torch
    from .pipeline import FusionPipeline
    from . import synth
    state = (torch.load(args.state, map_location="cpu", weights_only=True) if args.state is not None
             else synth.seeded_state(args.seeded_weights))
    pipe = FusionPipeline(H, W, "cuda")
    pipe.load_state(state)
    pipe.max_batch = args.batch
    frames = torch.empty((seg + 1, H, W, 3), dtype=torch.uint8).pin_memory()
    out = torch.empty((2 * seg + 1, H, W, 3), dtype=torch.uint8).pin_memory()
    fbytes = memoryview(frames.numpy()).cast("B")
    frames.numpy()[:2] = head
    have, first = 2, True                              # frames in the buffer; after a segment, frame 0 is its last frame
    while True:
        got = _read_into(fin, fbytes[have * frame_bytes:])
        if got % frame_bytes:
            raise ClipError("stream ends inside a frame (%d trailing bytes; frames are %d bytes)" % (got % frame_bytes, frame_bytes))
        have += got // frame_bytes
        eof = have < seg + 1                           # the buffer was not filled: the stream has ended
        if have >= 2:
            pipe.interpolate_video_host(frames[:have], out[:2 * have - 1])
            fout.write(memoryview(out.numpy()[0 if first else 1:2 * have - 1]).cast("B"))
            first = False
            frames[0].copy_(frames[have - 1])          # the boundary frame starts the next segment
            have = 1
        if eof:
            break
    fout.flush()


def main(argv=None):
    args = parse_args(argv)
    fin = sys.stdin.buffer if args.input == "-" else open(args.input, "rb")
    try:
        fout = sys.stdout.buffer if args.output == "-" else open(args.output, "wb")
        try:
            run(args, fin, fout)
        finally:
            if fout is not sys.stdout.buffer:
                fout.close()
    except ClipError as e:
        sys.stderr.write("interpolate_video: %s\n" % e)
        return 2
    finally:
        if fin is not sys.stdin.buffer:
            fin.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
