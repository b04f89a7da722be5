"""The end-to-end fusion recipe of the reference (``interp``,
src/fusion_net/interpolate_twoframe.py:82-334) as a device-resident, batched module.

``FusionPipeline(H, W, device)`` owns the three networks (state-dict compatible with the reference's
``phase_net.pt`` / ``fusion_net.pt`` / AdaCoF checkpoints) and the pyramid plan;
``pipe(rgb1, rgb2)`` maps two batches of frames [B,3,H,W] in [0,1] to the interpolated frame
[B,3,H,W].  Nothing leaves the GPU: Lab conversion, pyramid, PhaseNet, the four AdaCoFNet passes
(each = kernel estimation + ONE fused two-warp/blend/uncertainty kernel), Gaussian / median
uncertainty maps and the FusionNet blend all run on the current CUDA stream (the reference makes
>= 9 host round trips per frame, SURVEY.md F7).
"""
import math
import types

import torch

from . import conv as tc
from . import filters, transform, utils
from .adacofnet import AdaCoFNet
from .fusion_net import FusionNet, fusion_blend_rgb8, fusion_blend_yuv420p
from .phase_net import PhaseNet
from .pyramid import Pyramid
from .scene import SceneCutDetector


class GraphedCall:
    """CUDA-graph replay of one fixed-shape entry point of the pipeline (``FusionPipeline.graphed``).

    Small frames (256x256 crops: BASELINE.json configs[0] and the frozen part of the configs[4] training step) are bound by the
    ~400-1000 kernel launches of a call, not by the kernels; capturing the launch sequence once and replaying it removes the
    host from the loop.  Inputs are copied into the captured input buffers; the returned tensors are the captured output
    buffers -- valid until the next call (clone them to keep them).  The 3xFP16 range flag is read after every replay; if a
    replay left the range, the call is repeated eagerly (where the range guard re-runs it with the 3xTF32 split)."""

    def __init__(self, fn, example_inputs, warmup=2):
        self.fn = fn
        self.static_in = [t.clone() for t in example_inputs]
        side = torch.cuda.Stream(self.static_in[0].device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                 # warm-up off the default stream: plans, packed weights, workspaces exist
            for _ in range(warmup):
                fn(*self.static_in)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.static_out = fn(*self.static_in)

    def __call__(self, *inputs):
        for dst, src in zip(self.static_in, inputs):
            dst.copy_(src, non_blocking=True)
        self.graph.replay()
        if tc.range_check and tc.precision == tc.PRECISIONS["f16x3"] and tc.overflow_pending():
            return self.fn(*inputs)
        return self.static_out


class FusionPipeline(torch.nn.Module):
    def __init__(self, H, W, device, kernel_size=5, dilation=1, phase_plane_chunk=None):
        super().__init__()
        self.H, self.W = int(H), int(W)
        self.device = torch.device(device)
        height = utils.calc_pyr_height(torch.empty(3, H, W, device="meta"))                    # :124-129
        self.pyr = Pyramid(height=height, nbands=4, scale_factor=math.sqrt(2), device=self.device)
        self.phase_net = PhaseNet(self.pyr, self.device, num_img=2).eval()                     # :135-137
        self.fusion_net = FusionNet().to(self.device).eval()                                   # :143-145
        self.adacof = AdaCoFNet(types.SimpleNamespace(kernel_size=kernel_size, dilation=dilation, gpu_id=0)
                                ).to(self.device).eval()                                       # :99-103
        self.phase_net.plane_chunk = phase_plane_chunk
        self.stages = None  # set to a dict to capture intermediates (tests)
        self.max_batch = 8  # frame pairs per sub-batch at full HD (see forward)
        self.timing = None  # set to a list to collect (stage, start_event, end_event) (bench)
        self.max_batch_adacof = 16     # largest AdaCoFNet batch at full HD (the 64 -> 448 fused head tensor is 15 GB at 16)
        self._copy_streams = None      # (host -> device, device -> host) side streams of interpolate_host
        self._graphs = {}              # (method, input shapes) -> GraphedCall
        # small frames (<= 512x512) leave most SMs idle in any single kernel: the first AdaCoFNet pass does not depend on the
        # PhaseNet branch, so it runs on a side stream next to it (fork / join by events; also inside a captured CUDA graph)
        self.concurrent_small = True
        self._side_stream = None
        # optional callable (tag, planes, vals) -> vals applied to every decomposition (tests: aligns the branch of phase values
        # at +-pi with the reference's, see tests/_parity.py; None in production)
        self.filter_hook = None

    def graphed(self, method, *example_inputs):
        """``GraphedCall`` of ``self.<method>`` ('forward', 'fusion_inputs', 'phase_interp') for inputs of exactly these shapes:
        captured on first use, replayed afterwards.  ``stages`` / ``timing`` capture must be off."""
        assert self.stages is None and self.timing is None
        key = (method,) + tuple(tuple(t.shape) for t in example_inputs)
        g = self._graphs.get(key)
        if g is None:
            g = self._graphs[key] = GraphedCall(getattr(self, method), example_inputs)
        return g

    def _filter(self, tag, planes, **kw):
        vals = self.pyr.filter(planes, **kw)
        if self.filter_hook is not None:
            vals = self.filter_hook(tag, planes, vals)
        return vals

    def _tick(self, name):
        """Stage timer: CUDA events on the current stream, only when ``self.timing`` is a list."""
        if self.timing is None:
            return
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        self.timing.append((name, ev))

    def load_state(self, state):
        self.phase_net.load_state_dict(state["phase_net"])
        self.fusion_net.load_state_dict(state["fusion_net"])
        self.adacof.load_state_dict(state["adacof"])

    @torch.no_grad()
    @tc.range_checked
    def forward(self, rgb1, rgb2):
        B = rgb1.shape[0]
        if B > self.max_batch:
            # every stage is per-sample, so a large batch is a loop over sub-batches (keeps every tensor
            # below 2^31 elements -- torch's bilinear upsample / cuDNN limit -- and the working set bounded)
            outs = [self.forward(rgb1[i:i + self.max_batch], rgb2[i:i + self.max_batch])
                    for i in range(0, B, self.max_batch)]
            return torch.cat(outs, 0)
        base, ada_pred, phase_pred, other, maps = self.fusion_inputs(rgb1, rgb2)
        final = self.fusion_net(base, ada_pred, phase_pred, other, maps, variant=0)                 # :330
        self._tick('fusion_net')
        if self.stages is not None:
            self.stages["final"] = final
        return final

    @torch.no_grad()
    @tc.range_checked
    def fusion_inputs(self, rgb1, rgb2):
        """Everything of the recipe up to FusionNet's five inputs (``Trainer.predict`` runs exactly this part
        under no_grad, src/fusion_net/trainer.py:65-213)."""
        B, _, H, W = rgb1.shape
        assert (H, W) == (self.H, self.W) and rgb2.shape == rgb1.shape
        self._tick('start')
        lab1, lab2 = transform.rgb2lab(rgb1), transform.rgb2lab(rgb2)                           # :148-149
        planes = torch.cat((lab1.reshape(-1, H, W), lab2.reshape(-1, H, W)), 0)
        return self._fusion_inputs(rgb1, rgb2, lab1, lab2, planes, 3 * B)

    def _fusion_inputs(self, rgb1, rgb2, lab1, lab2, planes, q):
        """The pair-dependent body of ``fusion_inputs``: frames rgb1 / rgb2 [B,3,H,W], their Lab lab1 / lab2 and the Lab planes
        [N,H,W] the PhaseNet branch decomposes, in which frame 2 of pair-plane p is plane p + q.  Pairs: planes = cat(lab1, lab2),
        q = 3B.  A clip of B + 1 frames: planes = Lab of the B + 1 frames (each decomposed once), q = 3, and rgb1 / rgb2 / lab1 /
        lab2 are the views frames[:-1] / frames[1:]."""
        B, _, H, W = rgb1.shape
        pyr, r_shape = self.pyr, (B, 3, H, W)
        fork = self.concurrent_small and H * W <= 512 * 512 and self.timing is None
        if fork:
            main = torch.cuda.current_stream(rgb1.device)
            if self._side_stream is None:
                self._side_stream = torch.cuda.Stream(rgb1.device)
            side = self._side_stream
            side.wait_stream(main)
            with torch.cuda.stream(side):
                _, _, ada_pred, flow_var_map = self.adacof(rgb1, rgb2, return_warped=False)                          # :156
                flow_var_map = flow_var_map.squeeze(1)
        else:
            _, _, ada_pred, flow_var_map = self.adacof(rgb1, rgb2, return_warped=False)                              # :156
            flow_var_map = flow_var_map.squeeze(1)
        self._tick('lab+adacofnet#1')
        # PhaseNet branch (:168-192)
        vals = self._filter("phasenet", planes, want_high=False)
        self._tick('pyr.filter(12 planes/frame)')
        # separate_vals / get_concat_layers_inf / normalize_vals / forward / reverse_normalize with the regrouping and the
        # (de)normalisation fused into the concat assembly and the output kernel (PhaseNet.forward_fused)
        vals_pred = self.phase_net.forward_fused(vals, pyr.last_amp_max, frame2=q)
        del vals
        self._tick('phase_net')
        lab_pred = pyr.inv_filter_sparse(vals_pred, use_high=False).reshape(r_shape)            # high_level is zeros (:127-128)
        del vals_pred
        self._tick('pyr.inv_filter(3 planes/frame)')
        phase_pred = transform.lab2rgb(lab_pred)                                                # :192
        if fork:                                  # join: everything below reads ada_pred
            main.wait_stream(side)
            ada_pred.record_stream(main)
            flow_var_map.record_stream(main)

        def uncertainty_maps():
            # uncertainty maps (:197-225)
            # only level 0 + the high residual (h_freq) and the six coarsest levels + low pass (freq_diff) of these pyramids are ever read
            L = pyr.height - 2
            coarse = list(range(L - 6, L))
            # h_freq - h_freq_ph = mean_c(recon_{high + level 0}(ada_c) - recon_{high + level 0}(phase_c))  (get_last_value_levels(., 1),
            # :205-209).  Decomposition and reconstruction are linear in the image, so this is recon_{high + level 0} of the single
            # plane  xbar = mean_c(ada_c - phase_c): the six colour planes are decomposed on the (tiny) coarse levels only.
            vals_ada, vals_ph = utils.separate_vals(
                self._filter("uncertainty", torch.cat((ada_pred.reshape(-1, H, W), phase_pred.reshape(-1, H, W)), 0), want_high=False,
                             levels=coarse), 2)
            self._tick('lab2rgb+pyr.filter(6 planes/frame)')
            # ... and recon_{high + level 0}(D(x)) is a linear filter of x: one spectral multiplication (Pyramid.highband_filter)
            h_diff = pyr.highband_filter((ada_pred - phase_pred).mean(1))
            h_freq_diff = (h_diff.abs() * 100).clamp(min=0, max=1.0)
            self._tick('pyr.inv_filter(level0 x2)')
            phase_uncertainty = filters.gaussian_filter(h_freq_diff, 5)
            self._tick('gaussian')
            L = len(vals_ph.phase)
            # subtract_values + get_first_value_levels(., 6): only the 6 coarsest levels and the low pass are used
            keep = range(L - 6, L)
            vals_diff = vals_ph._replace(
                low_level=(vals_ph.low_level - vals_ada.low_level).abs(),
                phase=[(vals_ph.phase[l] - vals_ada.phase[l]).abs() if l in keep else None for l in range(L)],
                amplitude=[(vals_ph.amplitude[l] - vals_ada.amplitude[l]).abs() if l in keep else None for l in range(L)])
            freq_diff = pyr.inv_filter_sparse(vals_diff, use_high=False, levels=keep).reshape(r_shape).mean(1) * 30
            del vals_diff, vals_ada, vals_ph
            self._tick('pyr.inv_filter(coarse6)')
            ada_uncertainty = ((freq_diff - filters.median_filter(freq_diff, 50)).abs() * 5).clamp(0, 1)
            self._tick('median50')
            return phase_uncertainty, ada_uncertainty, freq_diff, h_freq_diff

        if fork:                                  # the uncertainty branch and the baseline passes only share their inputs
            side.wait_stream(main)
            with torch.cuda.stream(side):
                phase_uncertainty, ada_uncertainty, freq_diff, h_freq_diff = uncertainty_maps()
        else:
            phase_uncertainty, ada_uncertainty, freq_diff, h_freq_diff = uncertainty_maps()
        # baseline (:228-238)
        if 2 * B <= self.max_batch_adacof:
            # passes 2 and 3 (:229, :233) are independent: ONE AdaCoFNet call on a 2B batch (twice the tiles for the coarse layers)
            inb = self.adacof(torch.cat((rgb1, phase_pred), 0), torch.cat((phase_pred, rgb2), 0), return_warped=False, want_mask=False)[2]
            inb1, inb2 = inb[:B], inb[B:]
        else:
            inb1 = self.adacof(rgb1, phase_pred, return_warped=False, want_mask=False)[2]
            inb2 = self.adacof(phase_pred, rgb2, return_warped=False, want_mask=False)[2]
        base = self.adacof(inb1, inb2, return_warped=False, want_mask=False)[2]
        self._tick('adacofnet#2-4')
        if fork:
            main.wait_stream(side)
            for t in (phase_uncertainty, ada_uncertainty, freq_diff, h_freq_diff):
                t.record_stream(main)
        # fusion (:324-330)
        other = torch.cat([lab1, lab2], 1)
        maps = torch.stack([ada_uncertainty, phase_uncertainty, flow_var_map], 1)
        if self.stages is not None:
            self.stages.update(lab1=lab1, lab2=lab2, ada_pred=ada_pred, flow_var_map=flow_var_map, lab_pred=lab_pred,
                               phase_pred=phase_pred, phase_uncertainty=phase_uncertainty,
                               ada_uncertainty=ada_uncertainty, freq_diff=freq_diff, h_freq_diff=h_freq_diff, base=base)
        return base, ada_pred, phase_pred, other, maps

    @torch.no_grad()
    @tc.range_checked
    def phase_interp(self, rgb1, rgb2):
        """BASELINE.json configs[0] -- the PhaseNet-only interpolation (src/phase_net/interpolate_twoframe.py:52-107; the PhaseNet
        branch of the fusion recipe, src/fusion_net/interpolate_twoframe.py:168-192): rgb2lab -> Pyramid.filter -> PhaseNet ->
        Pyramid.inv_filter -> lab2rgb on [B,3,H,W] frames; the three colour planes of every frame are one batch instead of the
        reference's per-channel loop.  ``self.stages`` (dict) receives lab_pred, phase_pred and the predicted pyramid values."""
        B, _, H, W = rgb1.shape
        assert (H, W) == (self.H, self.W) and rgb2.shape == rgb1.shape
        pyr = self.pyr
        lab1, lab2 = transform.rgb2lab(rgb1), transform.rgb2lab(rgb2)
        vals = self._filter("phasenet", torch.cat((lab1.reshape(-1, H, W), lab2.reshape(-1, H, W)), 0), want_high=False)
        vals_pred = self.phase_net.forward_fused(vals, pyr.last_amp_max)
        lab_pred = pyr.inv_filter_sparse(vals_pred, use_high=False).reshape(B, 3, H, W)
        phase_pred = transform.lab2rgb(lab_pred)
        if self.stages is not None:
            self.stages.update(lab_pred=lab_pred, phase_pred=phase_pred, low_level=vals_pred.low_level)
            for l, (p, a) in enumerate(zip(vals_pred.phase, vals_pred.amplitude)):
                self.stages["phase%d" % l], self.stages["amp%d" % l] = p, a
        return phase_pred

    def _check_clip(self, frames, pix_fmt=None, matrix="bt709", full_range=False):
        """Validates a clip for interpolate_sequence; returns True for 8-bit frames (rgb24 [T,H,W,3] or, with pix_fmt='yuv420p',
        [T,3H/2,W]), False for fp32 [T,3,H,W]."""
        if pix_fmt == "yuv420p":
            transform.yuv_args(matrix, full_range)
            if self.H % 2 or self.W % 2:
                raise ValueError("yuv420p needs an even frame size; this pipeline is %dx%d" % (self.W, self.H))
            want = (3 * self.H // 2, self.W)
            if not torch.is_tensor(frames) or frames.dim() != 3 or frames.dtype != torch.uint8:
                raise ValueError("a yuv420p clip is a uint8 tensor [T,3H/2,W] = [T,%d,%d] for this pipeline" % want)
            if tuple(frames.shape[1:]) != want:
                raise ValueError("yuv420p clip frames must be %s for this %dx%d pipeline, got %s"
                                 % (list(want), self.W, self.H, list(frames.shape[1:])))
        elif pix_fmt is not None:
            raise ValueError("pix_fmt must be None (the dtype and layout decide) or 'yuv420p', got %r" % (pix_fmt,))
        else:
            if not torch.is_tensor(frames) or frames.dim() != 4:
                raise ValueError("a clip is a 4-d tensor: float32 [T,3,H,W] or uint8 [T,H,W,3]")
            if frames.dtype == torch.uint8:
                shape, want = tuple(frames.shape[1:]), (self.H, self.W, 3)
            elif frames.dtype == torch.float32:
                shape, want = tuple(frames.shape[1:]), (3, self.H, self.W)
            else:
                raise ValueError("clip dtype must be torch.float32 ([T,3,H,W] in [0,1]) or torch.uint8 ([T,H,W,3]), got %s"
                                 % frames.dtype)
            if shape != want:
                raise ValueError("%s clip frames must be %s for this %dx%d pipeline, got %s (wrong frame size or layout)"
                                 % (frames.dtype, list(want), self.W, self.H, list(shape)))
        if frames.shape[0] < 2:
            raise ValueError("a clip needs at least 2 frames, got %d" % frames.shape[0])
        return frames.dtype == torch.uint8

    def _scene_call(self, scene_cut, u8, frames, pix_fmt):
        """The per-call state of a SceneCutDetector for a clip that passed _check_clip (None without a detector)."""
        if scene_cut is None:
            return None
        if not isinstance(scene_cut, SceneCutDetector):
            raise ValueError("scene_cut must be a fvfi.scene.SceneCutDetector or None, got %r" % (scene_cut,))
        if not u8:
            raise ValueError("scene-cut detection takes 8-bit clips (rgb24 or yuv420p), not float32 ones")
        n = self.H * self.W * (1 if pix_fmt == "yuv420p" else 3)     # yuv420p: the Y plane; rgb24: every byte
        return scene_cut.begin(frames.shape[0] - 1, n, self.device)

    def _clip_window(self, frames, out=None, pix_fmt=None, matrix="bt709", full_range=False, scene=None, a=0):
        """Interpolates the B pairs of a window of B + 1 consecutive frames (device tensors in interpolate_sequence's formats):
        Lab and the pyramid decomposition run once per frame, the pairs read them as views (clip layout, q = 3).  Writes the B new
        frames into ``out`` (allocated if None) in the input's format.  ``scene`` (a fvfi.scene.SceneCall; 8-bit clips): the
        window's pairs are pairs a .. a + B - 1 of the call; at a detected cut the new frame is replaced by the earlier input
        frame, on this stream, before the caller's download."""
        H, W = self.H, self.W
        yuv = pix_fmt == "yuv420p"
        self._tick('start')
        if scene is not None:
            frames = frames.contiguous()
            scene.detect(frames, a)
        if yuv:
            rgb, lab = transform.yuv420p_to_rgb_lab(frames, matrix, full_range)
        elif frames.dtype == torch.uint8:
            rgb, lab = transform.rgb8_to_rgb_lab(frames)
        else:
            rgb = frames.contiguous()
            lab = transform.rgb2lab(rgb)
        base, ada_pred, phase_pred, other, maps = self._fusion_inputs(rgb[:-1], rgb[1:], lab[:-1], lab[1:], lab.reshape(-1, H, W), 3)
        if yuv:
            x = self.fusion_net.residual(base, ada_pred, phase_pred, other, maps)
            out = fusion_blend_yuv420p(base, x, out, matrix, full_range)
        elif frames.dtype == torch.uint8:
            x = self.fusion_net.residual(base, ada_pred, phase_pred, other, maps)
            out = fusion_blend_rgb8(base, x, out)
        else:
            final = self.fusion_net(base, ada_pred, phase_pred, other, maps, variant=0)
            out = final if out is None else out.copy_(final)
        if scene is not None:
            scene.select(frames, out, a)
        self._tick('fusion_net')
        return out

    @torch.no_grad()
    def interpolate_sequence(self, frames, pix_fmt=None, matrix="bt709", full_range=False, scene_cut=None):
        """The T - 1 in-between frames of a clip on the device: fp32 [T,3,H,W] in [0,1] -> fp32 [T-1,3,H,W], or uint8 [T,H,W,3]
        (rgb24) -> uint8 [T-1,H,W,3] (8-bit in and out: no fp32 frame is stored at either end).  With ``pix_fmt='yuv420p'`` the
        clip is 8-bit planar I420, uint8 [T,3H/2,W] -> [T-1,3H/2,W] (H, W even), converted with ``matrix`` ('bt709' or 'bt601')
        and limited or ``full_range`` at both ends (transform.yuv420p_to_rgb_lab, fusion_net.fusion_blend_yuv420p).  Frame t of
        the result lies between input frames t and t + 1.  Works in windows of ``max_batch`` pairs; a window of B pairs converts
        and decomposes its B + 1 frames once (the pair form ``pipe(frames[:-1], frames[1:])`` does every interior frame twice);
        the frame between two windows is done again in the next one.  ``scene_cut`` (a fvfi.scene.SceneCutDetector, 8-bit clips
        only): result frame t is input frame t, byte for byte, wherever pair t is a scene cut; the detector's carry and cut list
        advance by this call.  ValueError for fewer than 2 frames, a wrong frame size, dtype or layout, or a detector with a
        float32 clip."""
        u8 = self._check_clip(frames, pix_fmt, matrix, full_range)
        if not frames.is_cuda:
            raise ValueError("interpolate_sequence takes device tensors (interpolate_video_host takes host frames)")
        scene = self._scene_call(scene_cut, u8, frames, pix_fmt)
        out = self._sequence_windows(frames, u8, pix_fmt, matrix, full_range, scene)
        if scene is not None:
            scene.commit()          # once, after the range guard's possible second run
        return out

    @tc.range_checked
    def _sequence_windows(self, frames, u8, pix_fmt, matrix, full_range, scene):
        T, mb = frames.shape[0], self.max_batch
        out = torch.empty((T - 1,) + tuple(frames.shape[1:]), dtype=torch.uint8 if u8 else torch.float32, device=frames.device)
        for a in range(0, T - 1, mb):
            b = min(mb, T - 1 - a)
            self._clip_window(frames[a:a + b + 1], out[a:a + b], pix_fmt, matrix, full_range, scene, a)
        return out

    def interpolate_video_host(self, frames_host, out_host=None, pix_fmt=None, matrix="bt709", full_range=False, scene_cut=None):
        """Clip on HOST (pinned) memory: uint8 [T,H,W,3] rgb24 -> uint8 [2T-1,H,W,3], or with ``pix_fmt='yuv420p'`` uint8
        [T,3H/2,W] -> [2T-1,3H/2,W] (``matrix``, ``full_range`` as interpolate_sequence), the input frames at even indices and
        the interpolated ones at odd indices (twice the frame rate).  Windows of ``max_batch`` pairs go up as 8-bit frames and
        come back as 8-bit frames on the two copy streams of interpolate_host, overlapped with the compute of the neighbouring
        windows; the input frames are copied into the even slots on the host meanwhile, byte for byte.  ``scene_cut`` (a
        fvfi.scene.SceneCutDetector): at a detected cut t, odd slot 2t + 1 equals even slot 2t (the earlier frame is repeated);
        the decision and the substitution run on the device before each window's download."""
        layout = "[T,3H/2,W] yuv420p" if pix_fmt == "yuv420p" else "[T,H,W,3]"
        if not torch.is_tensor(frames_host) or frames_host.is_cuda or frames_host.dtype != torch.uint8:
            raise ValueError("interpolate_video_host takes a host uint8 %s tensor (pinned for overlapped copies)" % layout)
        self._check_clip(frames_host, pix_fmt, matrix, full_range)
        scene = self._scene_call(scene_cut, True, frames_host, pix_fmt)
        frames_host = frames_host.contiguous()
        T = frames_host.shape[0]
        shape = (2 * T - 1,) + tuple(frames_host.shape[1:])
        if out_host is None:
            out_host = torch.empty(shape, dtype=torch.uint8).pin_memory()
        if tuple(out_host.shape) != shape or out_host.dtype != torch.uint8 or out_host.is_cuda:
            raise ValueError("out_host must be a host uint8 [%s] tensor" % ",".join(map(str, shape)))
        mb = self.max_batch
        starts = list(range(0, T - 1, mb))
        uploads = [(frames_host[a:a + min(mb, T - 1 - a) + 1],) for a in starts]

        def download(k, out):                  # per-frame contiguous views of the odd slots
            for i in range(out.shape[0]):
                out_host[2 * (starts[k] + i) + 1].copy_(out[i], non_blocking=True)

        def host_work():
            out_host[0::2].copy_(frames_host)
        self._run_windows(uploads, lambda k, frames: self._clip_window(frames, None, pix_fmt, matrix, full_range, scene, starts[k]),
                          download, host_work)
        if scene is not None:
            scene.commit()          # once, after the range guard's possible second run
        return out_host

    def interpolate_host(self, rgb1_host, rgb2_host, out_host=None):
        """End-to-end call on HOST (pinned) tensors [B,3,H,W]: host -> device copies of the frames, the pipeline, device -> host
        copy of the result, all inside the call.  The batch is processed in sub-batches of ``max_batch`` pairs; the copies run
        on two side streams, so sub-batch k+1's frames arrive and sub-batch k-1's result leaves while sub-batch k computes."""
        B, mb = rgb1_host.shape[0], self.max_batch
        if out_host is None:
            out_host = torch.empty((B, 3, self.H, self.W), dtype=torch.float32).pin_memory()
        starts = list(range(0, B, mb))
        uploads = [(rgb1_host[a:a + mb], rgb2_host[a:a + mb]) for a in starts]

        def download(k, out):
            out_host[starts[k]:starts[k] + out.shape[0]].copy_(out, non_blocking=True)
        self._run_windows(uploads, lambda k, rgb1, rgb2: self.forward(rgb1, rgb2), download)
        return out_host

    @torch.no_grad()
    @tc.range_checked       # ONE range check (stream sync) for the whole call; the per-window calls below are nested in it
    def _run_windows(self, uploads, run, download, host_work=None):
        """Stream choreography of the host-buffer entry points: ``uploads`` [k] is the tuple of host tensors of window k; their
        host -> device copies are all queued at once on the input stream (in order), window k's ``run(k, *device_tensors)`` waits for
        its own copies only, and ``download(k, result)`` issues its device -> host copies on the output stream after the window's
        compute.  ``host_work()`` (optional) runs on the host while the device works; the call returns with every result on the
        host."""
        if self._copy_streams is None:
            self._copy_streams = (torch.cuda.Stream(self.device), torch.cuda.Stream(self.device))
        compute = torch.cuda.current_stream(self.device)
        s_in, s_out = self._copy_streams
        s_in.wait_stream(compute)                      # the caller's earlier work on these buffers is ordered before the copies
        staged = []
        for hs in uploads:                             # all uploads are queued at once; they run in order on the input stream
            with torch.cuda.stream(s_in):
                ds = [h.to(self.device, non_blocking=True) for h in hs]
                ev = torch.cuda.Event()
                ev.record(s_in)
            staged.append((ds, ev))
        for k, (ds, ev) in enumerate(staged):
            compute.wait_event(ev)
            for d in ds:
                d.record_stream(compute)
            out = run(k, *ds)
            done = torch.cuda.Event()
            done.record(compute)
            with torch.cuda.stream(s_out):
                s_out.wait_event(done)
                download(k, out)
            out.record_stream(s_out)
        if host_work is not None:
            host_work()
        compute.wait_stream(s_out)                     # the call returns with the result on the host
        compute.synchronize()
