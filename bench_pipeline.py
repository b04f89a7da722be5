"""Pipeline workloads of bench.py.

* PipelineWorkload     BASELINE.json configs[2]: the full fusion recipe (PhaseNet + 4x AdaCoFNet + FusionNet blend) at 1080p,
                       batch 16 on one B200; frame pairs shard across ranks by batch (the default bench line).
* Pipeline4KWorkload   configs[3]: the same recipe at 3840x2160.
* PhaseNet256Workload  configs[0]: PhaseNet decompose -> predict -> reconstruct on one 256x256 frame pair.
Under torchrun (N > 1) the default line also carries a `train` record (configs[4]) and a `pipeline4k` record (configs[3]),
measured outside the headline's timed region (multi_gpu_records).
"""
import json
import os
import time

import numpy as np


def _psnr(a, b):
    mse = float(((a.astype(np.float64) - b.astype(np.float64)) ** 2).mean())
    return 10 * np.log10(1.0 / max(mse, 1e-20))


class PipelineWorkload:
    H, W = 1080, 1920
    B = int(os.environ.get("FVFI_BENCH_BATCH", "16"))
    name = "fusion_pipeline_1080p_batch%d (BASELINE.json configs[2]): PhaseNet + 4x AdaCoFNet + FusionNet" % B
    metric = "interpolated_1080p_frames_per_s"
    dtype = "f32"
    cpu_kind = "port"
    CPU_SAMPLE = (544, 960)        # bounded CPU sample of the main arm (about a quarter of the 1080p area)

    def __init__(self, device, seed):
        import torch
        from fvfi import synth as fp               # seeded synthetic frames / random-init weights (input generation, not timed)
        from fvfi.pipeline import FusionPipeline
        self.torch, self.device = torch, device
        self.pipe = FusionPipeline(self.H, self.W, device, phase_plane_chunk=int(os.environ.get("FVFI_PLANE_CHUNK", "24")))
        self.pipe.max_batch = int(os.environ.get("FVFI_MAX_BATCH", "8" if self.H <= 1080 else "2"))
        self.pipe.load_state(fp.seeded_state(0))
        r1, r2 = fp.seeded_frames(1, self.H, self.W, seed)
        g = torch.Generator().manual_seed(seed)
        # B distinct pairs: per-sample brightness/shift jitter of one smooth synthetic pair
        gains = 0.8 + 0.2 * torch.rand((self.B, 1, 1, 1), generator=g)
        self.h1 = (r1 * gains).clamp(0, 1).contiguous().pin_memory()
        self.h2 = (r2 * gains).clamp(0, 1).contiguous().pin_memory()
        self.out_host = torch.empty((self.B, 3, self.H, self.W)).pin_memory()
        self.d1, self.d2 = self.h1.to(device), self.h2.to(device)
        self.frames_per_step = self.B
        self.launches_per_step = None
        self.stage_ms = {}
        self.nsteps = 0
        self.config_extra = {"convs": "tcgen05 implicit GEMM, %s operand split, persistent (csrc/conv_tc.cu)" % os.environ.get("FVFI_CONV_PREC", "f16x3"),
                             "phase_plane_chunk": self.pipe.phase_net.plane_chunk,
                             "sub_batch": self.pipe.max_batch}

    @classmethod
    def static_config(cls):
        """The `config` object of the JSON line -- identical in the product arm and the reference arm."""
        return {"workload": cls.name, "frames_per_step_per_gpu": cls.B, "frame": "%dx%d" % (cls.W, cls.H),
                "l2": "inputs larger than L2 (no flush needed)", "sharding": "frame pairs by batch, no collectives"}

    def step(self, timed=False):
        self.pipe.timing = [] if timed else None
        self.out = self.pipe(self.d1, self.d2)
        if timed:
            self._pending = getattr(self, "_pending", [])
            self._pending.append(self.pipe.timing)
            self.pipe.timing = None

    def outputs(self):
        """What a caller of the timed step receives: the interpolated frames."""
        return {"frame": self.out}

    def _collect(self):
        for tl in getattr(self, "_pending", []):
            for (n0, e0), (n1, e1) in zip(tl[:-1], tl[1:]):
                if n1 == 'start':
                    continue  # boundary between two sub-batches
                self.stage_ms[n1] = self.stage_ms.get(n1, 0.0) + e0.elapsed_time(e1)
            self.nsteps += 1
        self._pending = []

    def _peaks(self):
        import json
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "MEASURED_PEAKS.json")
        if os.path.exists(path):
            d = json.load(open(path))
            return float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1399.0))), "measured sustained bf16 (MEASURED_PEAKS.json)"
        return 1400.0, "fallback (B200_PROFILING.md, sustained)"

    def _time_conv(self):
        """Per-launch CUDA events around every tcgen05 convolution of ONE extra pipeline step: the step's dominant
        kernel (conv_split_kernel, ~60 % of the step).  achieved = algorithmic FLOPs (2*B*H*W*Cin*Cout*K*K) / time."""
        from fvfi import conv as tc
        torch = self.torch
        tc.timing = []
        self.pipe.timing = None
        self.pipe(self.d1, self.d2)
        torch.cuda.synchronize()
        rec, tc.timing = tc.timing, None
        flops = sum(r[0] for r in rec)
        ms = sum(r[1].elapsed_time(r[2]) for r in rec)
        # per shape class: algorithmic FLOP/s and the algorithmic DRAM bytes (activation in + out, fp32) each launch must move
        classes = {}
        fused = {"launches": 0, "ms": 0.0, "flops": 0.0}
        for fl, e0, e1, nl, (B, Cin, Cout, K, H, W, act), up in rec:
            key = "%d->%d k%d @%dx%d%s%s" % (Cin, Cout, K, H, W, "" if act is None else " " + act, " [resampling in the loader]" if up else "")
            if up:
                fused["launches"] += nl
                fused["ms"] += e0.elapsed_time(e1)
                fused["flops"] += fl
            c = classes.setdefault(key, [0, 0.0, 0.0, 0.0])
            c[0] += nl
            c[1] += fl
            c[2] += e0.elapsed_time(e1)
            c[3] += 4.0 * B * H * W * (Cin + Cout)
        top = sorted(classes.items(), key=lambda kv: -kv[1][2])[:12]
        table = [{"layer": k, "launches": v[0], "ms": round(v[2], 3), "tflops": round(v[1] / v[2] / 1e9, 1),
                  "algorithmic_dram_gb": round(v[3] / 1e9, 3), "dram_gbs_at_this_time": round(v[3] / v[2] / 1e6, 1)} for k, v in top]
        self._fused_up = fused
        self._alg_dram = sum(4.0 * B * H * W * (Cin + Cout) for _, _, _, _, (B, Cin, Cout, K, H, W, act), _ in rec)
        return flops, ms, sum(r[3] for r in rec), table

    def _time_hbm_kernels(self, peak):
        """The hand-written HBM-bound kernels of the step, each timed alone with CUDA events on the step's shapes."""
        torch = self.torch
        from fvfi import adacof
        B, H, W = min(self.B, self.pipe.max_batch), 1088, 1920
        g = torch.Generator(device=self.device).manual_seed(0)
        mk = lambda *s: torch.rand(s, device=self.device, generator=g)
        mkn = lambda *s: torch.randn(s, device=self.device, generator=g)

        def timeit(fn, reps=5):
            for _ in range(3):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps
        out = []
        px = B * H * W
        i1, i2 = mk(B, 3, H + 4, W + 4), mk(B, 3, H + 4, W + 4)
        w1 = torch.softmax(mkn(B, 25, H, W), 1)
        w2 = torch.softmax(mkn(B, 25, H, W), 1)
        occ = mk(B, 1, H, W)
        gout = mkn(B, 3, H, W)
        nb_syn = 4 * (6 * 25 * px + 2 * 3 * B * (H + 4) * (W + 4) + px + 3 * px + px)
        nb_fwd = 4 * (3 * 25 * px + 3 * B * (H + 4) * (W + 4) + 3 * px)
        nb_bwd = 4 * (3 * px + 3 * B * (H + 4) * (W + 4) + 3 * 25 * px + 3 * 25 * px)
        # two offset distributions: what KernelEstimation produces on smooth frames (sub-pixel .. a few pixels, spatially smooth)
        # and the adversarial i.i.d. N(0, 3^2) gather of SURVEY.md 8(d) / BASELINE.json configs[1]
        for label, mkoff in (("smooth offsets U(-0.5,0.5)", lambda: mk(B, 25, H, W) - 0.5),
                             ("i.i.d. offsets N(0,3^2) clipped to +-16 (configs[1])", lambda: (3 * mkn(B, 25, H, W)).clamp_(-16, 16))):
            a1, b1 = mkoff(), mkoff()
            # the second frame gets its OWN three coefficient tensors: nb_syn counts six maps, and re-using frame 1's would turn half of
            # that into L2 hits (ncu, profiles/r02_adacof_final_summary.txt: 5.8 instead of 10.8 GB of DRAM traffic per launch)
            a2, b2 = mkoff(), mkoff()
            ms = timeit(lambda: adacof.adacofnet_warp_blend(i1, i2, w1, a1, b1, w2, a2, b2, occ, 1, want_t=False))
            out.append({"kernel": "adacof_fwd_tma<2,..> fused synthesis (two warps + blend + uncertainty), " + label, "bound": "hbm",
                        "achieved": round(nb_syn / ms / 1e6, 1), "unit": "GB/s", "frac": round(nb_syn / ms / 1e6 / peak, 4),
                        "ms_per_launch": round(ms, 4), "algorithmic_bytes_per_launch": nb_syn,
                        "traffic": 10.925e9 if B == 8 else None})     # ncu dram bytes, profiles/r02_adacof_final_summary.txt
            ms = timeit(lambda: adacof.adacof_forward(i1, w1, a1, b1, 1))
            out.append({"kernel": "adacof_fwd_tma<1,..> warp forward (configs[1] shape B=8), " + label, "bound": "hbm",
                        "achieved": round(nb_fwd / ms / 1e6, 1), "unit": "GB/s", "frac": round(nb_fwd / ms / 1e6 / peak, 4),
                        "ms_per_launch": round(ms, 4), "algorithmic_bytes_per_launch": nb_fwd,
                        "traffic": 5.595e9 if B == 8 else None})      # ncu dram bytes, profiles/r02_adacof_final_summary.txt
            ms = timeit(lambda: adacof.adacof_backward(gout, i1, w1, a1, b1, 1, "none"))
            out.append({"kernel": "adacof_fwd_tma<0,..> fused backward gW/g_alpha/g_beta (configs[1] shape B=8), " + label, "bound": "hbm",
                        "achieved": round(nb_bwd / ms / 1e6, 1), "unit": "GB/s", "frac": round(nb_bwd / ms / 1e6 / peak, 4),
                        "ms_per_launch": round(ms, 4), "algorithmic_bytes_per_launch": nb_bwd,
                        "traffic": 10.590e9 if B == 8 else None})
            if label.startswith("i.i.d."):
                try:     # same-box bar: the reference's own CUDA kernels on the same tensors (oracle/_ref cubins; evidence only)
                    from oracle import ref_kernels
                    if ref_kernels.have(B, 3, H, W, 5, 1):
                        f = timeit(lambda: ref_kernels.forward(i1, w1, a1, b1, 1), 2)
                        b = timeit(lambda: ref_kernels.backward(gout, i1, w1, a1, b1, 1), 2)
                        out.append({"kernel": "REFERENCE CuPy kernels (adacof.py:6-258) compiled for sm_100a, same tensors",
                                    "fwd_ms": round(f, 3), "bwd_ms": round(b, 3)})
                except Exception as ex:
                    out.append({"kernel": "reference kernels", "error": repr(ex)[:160]})
            del a1, b1, a2, b2
        del i1, i2, w1, w2, occ, gout
        torch.cuda.empty_cache()
        N = 12 * B
        x = mk(N, self.H, self.W)
        pyr = self.pipe.pyr
        vals = pyr.filter(x, want_high=False)
        msd = timeit(lambda: pyr.filter(x, want_high=False), 3)
        msr = timeit(lambda: pyr.inv_filter_sparse(vals, use_high=False), 3)
        pb = 72 * self.H * self.W * N - 4 * self.H * self.W * N      # 72 HW per plane-op minus the skipped high residual
        for name, t in (("pyramid decompose (all levels, %d planes)" % N, msd),
                        ("pyramid reconstruct (all levels, %d planes)" % N, msr)):
            out.append({"kernel": name, "bound": "hbm", "achieved": round(pb / t / 1e6, 1), "unit": "GB/s",
                        "frac": round(pb / t / 1e6 / peak, 4), "ms_per_call": round(t, 4), "planes": N,
                        "algorithmic_bytes_per_call": pb})
        return out

    def _ncu_traffic(self, launches):
        """DRAM bytes per launch of the convolution kernel from the committed ncu capture of this step's launch sequence
        (profiles/r02_conv_traffic.json, written by tools/ncu_conv_step.py; a profiler figure, not measured live), next to the
        algorithmic bytes (fp32 activations in + out) of the launches timed here."""
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_conv_traffic.json")
        self._traffic_detail = {"algorithmic_dram_bytes_per_step": self._alg_dram,
                                "algorithmic_dram_bytes_per_launch": self._alg_dram / max(launches, 1)}
        try:
            t = json.load(open(path))
        except Exception:
            return None
        self._traffic_detail.update({"measured_dram_bytes_per_step": t["dram_bytes_per_step"], "measured_launches_per_step": t["launches_per_step"],
                                     "measured_over_algorithmic": round(t["dram_bytes_per_step"] / max(self._alg_dram, 1.0), 3),
                                     "source": t["source"]})
        return t["dram_bytes_per_launch"] if t["launches_per_step"] == launches else t["dram_bytes_per_step"] / max(launches, 1)

    def roofline(self, peak, peak_src):
        """Dominant kernel of the step = the tcgen05 convolution (tensor-bound).  `achieved` counts ALGORITHMIC FLOPs
        (one multiply-add per tap, channel pair and pixel); every one of them is executed as three fp16 tensor-core
        products (3xFP16 split), so the tensor pipe runs 3x that rate (`mma_frac`).  The hand-written HBM-bound kernels
        of the step (fused AdaCoF synthesis, pyramid) follow in `other_kernels`."""
        self._collect()
        tpeak, tsrc = self._peaks()
        flops, ms, launches, table = self._time_conv()
        ach = flops / (ms * 1e-3) / 1e12
        stages = {k: round(v / max(self.nsteps, 1), 3) for k, v in self.stage_ms.items()}
        step_ms = sum(stages.values())
        return {"bound": "tensor", "kernel": "conv_split_kernel<ACT, PREC_F16X3> (all %d launches of one step)" % launches,
                "achieved": round(ach, 1), "peak": tpeak, "unit": "TFLOP/s", "frac": round(ach / tpeak, 4),
                "mma_frac": round(3 * ach / tpeak, 4), "traffic": self._ncu_traffic(launches), "peak_source": tsrc,
                "traffic_detail": self._traffic_detail,
                # `achieved` aggregates several hundred launches of different shapes, so there is no single per-launch DRAM figure:
                # `by_layer_class` lists, per shape class of this step, time, algorithmic TFLOP/s and the ALGORITHMIC DRAM bytes
                # (fp32 activations in + out); measured DRAM bytes of representative launches: profiles/ (ncu --set full)
                "by_layer_class": table,
                # round 2 moved the bilinear resampling in front of KernelEstimation's Upsample blocks / head tails and PhaseNet's
                # level inputs INTO the loaders of these launches (the stand-alone resize kernels they replace were ~45 ms per step
                # outside this kernel in round 1): their time is convolution + resampling, their FLOP count is the convolution's alone
                "launches_with_resampling_loader": {"launches": self._fused_up["launches"], "ms": round(self._fused_up["ms"], 2),
                                                    "tflops": round(self._fused_up["flops"] / max(self._fused_up["ms"], 1e-9) / 1e9, 1)},
                "plain_launches": {"launches": launches - self._fused_up["launches"], "ms": round(ms - self._fused_up["ms"], 2),
                                   "tflops": round((flops - self._fused_up["flops"]) / max(ms - self._fused_up["ms"], 1e-9) / 1e9, 1),
                                   "frac": round((flops - self._fused_up["flops"]) / max(ms - self._fused_up["ms"], 1e-9) / 1e9 / tpeak, 4)},
                "ms_per_step_in_kernel": round(ms, 2), "share_of_step": round(ms / max(step_ms, 1e-9), 3),
                "algorithmic_flops_per_step": flops,
                "other_kernels": self._time_hbm_kernels(peak), "hbm_peak": peak, "hbm_peak_source": peak_src,
                "stage_ms_per_step": stages}

    def e2e(self, steps):
        torch = self.torch
        self.pipe.timing = None
        self.pipe.interpolate_host(self.h1, self.h2, self.out_host)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.pipe.interpolate_host(self.h1, self.h2, self.out_host)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        nb = lambda t: t.numel() * 4
        ok = bool(torch.equal(self.out_host, self.out.cpu()))
        return dt, nb(self.h1) + nb(self.h2), nb(self.out_host), ok

    # ------------------------------------------------------------------------------------------ CPU legs (oracle = the checker)
    @classmethod
    def _cpu_run(cls, H, W, threads, seed, stages=None, decomps=None):
        import torch
        from oracle import fusion_pipeline as fp
        torch.set_num_threads(threads)
        be = fp.oracle_backend(fp.seeded_state(0), hw=(H, W), threads=threads)
        r1, r2 = fp.seeded_frames(1, H, W, seed)
        t0 = time.perf_counter()
        out = fp.interp(be, r1, r2, stages, decomps)
        return time.perf_counter() - t0, (r1, r2, out)

    @classmethod
    def cpu_sample(cls, threads, seed=0, size=None, keep=None):
        """CPU oracle of the same recipe (oracle/fusion_pipeline.py: restated reference modules, scipy filters, C warp) on ONE
        frame pair at ``size`` (default CPU_SAMPLE); frames/s is scaled to the workload's frame by the pixel ratio."""
        H, W = size or cls.CPU_SAMPLE
        stages = {} if keep is not None else None
        decomps = {} if keep is not None else None
        dt, io = cls._cpu_run(H, W, threads, seed, stages, decomps)
        if keep is not None:
            keep.update(size=(H, W), io=io, stages=stages, decomps=decomps)
        scale = (H * W) / float(cls.H * cls.W)
        return scale / dt, dt, ("1 frame pair at %dx%d (%.4f of the %dx%d area), frames/s scaled by the pixel ratio; "
                                "oracle port of the reference recipe: torch CPU + scipy + C warp" % (W, H, scale, cls.W, cls.H))

    @classmethod
    def reference_full(cls, threads):
        """The reference arm's own measurement: ONE full-size frame pair through the CPU port (BASELINE.md section 4: "1 run for
        the 1080p case"), no extrapolation."""
        dt, _ = cls._cpu_run(cls.H, cls.W, threads, 0)
        return 1.0 / dt, dt, "1 frame pair at the FULL %dx%d size, one run; oracle port of the reference recipe: torch CPU + scipy + C warp" % (cls.W, cls.H)

    def parity(self, kept):
        """GPU pipeline vs the oracle output the cpu_baseline leg just computed (same frame pair, same seeded weights)."""
        from fvfi.pipeline import FusionPipeline
        from fvfi import synth
        torch = self.torch
        H, W = kept["size"]
        r1, r2, ref = kept["io"]
        from oracle.wrap_align import WrapAligner
        pipe = FusionPipeline(H, W, self.device)
        pipe.load_state(synth.seeded_state(0))
        ref = ref.numpy()
        raw = pipe(r1.to(self.device), r2.to(self.device)).cpu().numpy()         # as shipped
        # the same call evaluated on the reference's branch of the wrapped phases at the few coefficients on the negative real
        # axis (oracle/wrap_align.py; the reference recipe is discontinuous there, tests/test_models_oracle.py)
        pipe.filter_hook = al = WrapAligner.from_decomps(kept["decomps"])
        pipe.stages = {}
        out = pipe(r1.to(self.device), r2.to(self.device)).cpu().numpy()
        per = {k: float(np.abs(pipe.stages[k].cpu().numpy() - v.numpy()).max()) for k, v in kept["stages"].items()
               if k in pipe.stages and k != "final"}
        e = np.abs(out - ref)
        return {"max_abs_err": float(e.max()), "psnr_db": round(_psnr(out, ref), 2), "size": "%dx%d" % (W, H),
                "rms_err": float(np.sqrt((e.astype(np.float64) ** 2).mean())), "fraction_of_pixels_above_1e-4": float((e > 1e-4).mean()),
                "note": "every IMAGE stage agrees to ~1e-6 (per_stage_max_abs_err); the maximum of `final` comes from isolated pixels of "
                        "the uncertainty maps: the recipe subtracts the phases of two pyramids (src/train/utils.py:322-346), and where a "
                        "coefficient is ~1e-5 of its level maximum its phase turns by 0.01-0.1 rad under a 1e-6 change of the decomposed "
                        "image, amplified x30 x5 before the clamp (DESIGN.md section 5; tools/diag_unc.py)",
                "against": "oracle port of the reference recipe (fp32, CPU) on the same frame pair and weights",
                "branch": "wrapped phases within rounding of +-pi take the reference's sign (%d of %d phase values); "
                          "unaligned run below" % (al.flips, al.coefficients),
                "unaligned": {"max_abs_err": float(np.abs(raw - ref).max()), "psnr_db": round(_psnr(raw, ref), 2)},
                "per_stage_max_abs_err": {k: float("%.3g" % v) for k, v in per.items()}}


class Pipeline4KWorkload(PipelineWorkload):
    """BASELINE.json configs[3]: the same recipe at 3840x2160 (pyramid height 19, AdaCoFNet pads to 2176 rows); frame pairs
    shard across ranks exactly like the 1080p workload.  Not the default bench line (the metric is quoted at 1080p)."""
    H, W = 2160, 3840
    B = int(os.environ.get("FVFI_BENCH_BATCH_4K", "4"))
    name = "fusion_pipeline_4k_batch%d (BASELINE.json configs[3])" % B
    metric = "interpolated_4k_frames_per_s"


class PhaseNet256Workload(PipelineWorkload):
    """BASELINE.json configs[0]: PhaseNet decompose -> phase/amplitude prediction -> reconstruct on one 256x256 RGB frame pair
    (Pyramid(12, 4, sqrt 2)), random-init weights; the reference side is the CPU port at the SAME size (no extrapolation)."""
    H, W = 256, 256
    B = 1
    name = "phasenet_256x256_one_pair (BASELINE.json configs[0]): rgb2lab -> pyramid -> PhaseNet -> reconstruct -> lab2rgb"
    metric = "phasenet_interpolated_256x256_frames_per_s"
    CPU_SAMPLE = (256, 256)

    def step(self, timed=False):
        # launch-bound at this size (~450 launches per call): the launch sequence is captured once and replayed (CUDA graph)
        if os.environ.get("FVFI_NO_GRAPH", "0") == "1":
            self.out = self.pipe.phase_interp(self.d1, self.d2)
        else:
            self.out = self.pipe.graphed("phase_interp", self.d1, self.d2)(self.d1, self.d2)

    def _eager_vs_graph_ms(self):
        torch = self.torch
        res = {}
        for name, fn in (("eager", lambda: self.pipe.phase_interp(self.d1, self.d2)),
                         ("cuda_graph", lambda: self.pipe.graphed("phase_interp", self.d1, self.d2)(self.d1, self.d2))):
            for _ in range(3):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res[name] = round(e0.elapsed_time(e1) / 20, 4)
        return res

    def roofline(self, peak, peak_src):
        torch = self.torch
        pyr = self.pipe.pyr
        self.config_extra = dict(self.config_extra, ms_per_call=self._eager_vs_graph_ms())
        x = torch.rand((6, self.H, self.W), device=self.device)
        for _ in range(3):
            vals = pyr.filter(x, want_high=False)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        for _ in range(10):
            vals = pyr.filter(x, want_high=False)
        e[1].record()
        for _ in range(10):
            pyr.inv_filter_sparse(vals, use_high=False)
        e[2].record()
        torch.cuda.synchronize()
        msd, msr = e[0].elapsed_time(e[1]) / 10, e[1].elapsed_time(e[2]) / 10
        pb = 68 * self.H * self.W * 6
        return {"bound": "hbm", "kernel": "pyramid decompose, 6 planes of 256x256 (latency-bound: 26.7 MB algorithmic)",
                "achieved": round(pb / msd / 1e6, 1), "peak": peak, "unit": "GB/s", "frac": round(pb / msd / 1e6 / peak, 5),
                "traffic": None, "peak_source": peak_src, "ms_per_call": round(msd, 4),
                "other_kernels": [{"kernel": "pyramid reconstruct, 6 planes", "ms_per_call": round(msr, 4),
                                   "achieved": round(pb / msr / 1e6, 1), "unit": "GB/s"}]}

    def e2e(self, steps):
        torch = self.torch
        steps = max(steps, 20)

        def one():
            d1 = self.h1.to(self.device, non_blocking=True)
            d2 = self.h2.to(self.device, non_blocking=True)
            self.out_host.copy_(self.pipe.graphed("phase_interp", d1, d2)(d1, d2), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        one()
        t0 = time.perf_counter()
        for _ in range(steps):
            one()
        dt = (time.perf_counter() - t0) / steps
        nb = lambda t: t.numel() * 4
        return dt, nb(self.h1) + nb(self.h2), nb(self.out_host), bool(torch.equal(self.out_host, self.out.cpu()))

    @classmethod
    def _cpu_run(cls, H, W, threads, seed, stages=None, decomps=None):
        import torch
        from oracle import fusion_pipeline as fp
        torch.set_num_threads(threads)
        be = fp.oracle_backend(fp.seeded_state(0), hw=(H, W), threads=threads)
        r1, r2 = fp.seeded_frames(1, H, W, seed)
        fp.interp_phasenet(be, r1, r2)                    # warm-up (thread pools, FFT plans): this config runs in < 1 s
        t0 = time.perf_counter()
        out = fp.interp_phasenet(be, r1, r2, stages, decomps)
        return time.perf_counter() - t0, (r1, r2, out)

    def parity(self, kept):
        from oracle.wrap_align import WrapAligner
        r1, r2, ref = kept["io"]
        raw = self.pipe.phase_interp(r1.to(self.device), r2.to(self.device)).cpu().numpy()
        self.pipe.filter_hook = al = WrapAligner.from_decomps(kept["decomps"])
        self.pipe.stages = {}
        out = self.pipe.phase_interp(r1.to(self.device), r2.to(self.device)).cpu().numpy()
        st, self.pipe.stages, self.pipe.filter_hook = self.pipe.stages, None, None
        per = {k: float(np.abs(st[k].cpu().numpy() - kept["stages"][k].numpy()).max()) for k in ("lab_pred", "low_level")}
        return {"max_abs_err": float(np.abs(out - ref.numpy()).max()), "psnr_db": round(_psnr(out, ref.numpy()), 2), "size": "256x256",
                "against": "oracle port of the reference PhaseNet interpolation (fp32, CPU), same pair and weights",
                "branch": "wrapped phases within rounding of +-pi take the reference's sign (%d of %d phase values)" % (al.flips, al.coefficients),
                "unaligned": {"max_abs_err": float(np.abs(raw - ref.numpy()).max()), "psnr_db": round(_psnr(raw, ref.numpy()), 2)},
                "per_stage_max_abs_err": {k: float("%.3g" % v) for k, v in per.items()}}


# ----------------------------------------------------------------------------------------------------------------------
# Multi-GPU records of the default line (N > 1): BASELINE.json configs[4] (training step) and configs[3] (4K), outside the
# headline's timed region.  Device-timed, max over ranks.
# ----------------------------------------------------------------------------------------------------------------------
def multi_gpu_records(device, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from fvfi import synth
    from fvfi.pipeline import FusionPipeline
    from fvfi.trainer import FusionTrainer
    out = {}

    def maxr(v):
        t = torch.tensor([v], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- configs[4]: FusionNet training step, 256x256 crops, 8 per GPU (global batch 8 * world), flat-bucket NCCL all-reduce
    H = W = 256
    Bl = 8
    pipe = FusionPipeline(H, W, device)
    pipe.load_state(synth.seeded_state(rank))            # ranks start DIFFERENT on purpose: the trainer broadcasts rank 0's weights
    tr = FusionTrainer(pipe, lr=1e-4)
    a, b = synth.seeded_frames(Bl * world, H, W, 123)     # the same global batch on every rank; each takes its shard
    sl = slice(rank * Bl, (rank + 1) * Bl)
    f1, f2 = a[sl].to(device), b[sl].to(device)
    target = (0.5 * (f1 + f2)).clamp(0, 1)
    # gradient / loss parity of ONE distributed step against a single process on all world*8 samples (rank 0 recomputes every shard)
    with torch.no_grad():
        inputs = pipe.fusion_inputs(f1, f2)
    tr.bucket.zero()
    loss = torch.nn.functional.l1_loss(target, torch.clip(tr.net(*inputs, variant=0), 0, 1))
    loss.backward()
    flat_dist = tr.bucket.all_reduce_mean(tr.group).clone()
    lt = loss.detach().double().reshape(1).clone()
    dist.all_reduce(lt)
    loss_dist = float(lt.item()) / world
    if rank == 0:
        acc = torch.zeros_like(flat_dist)
        lsum = 0.0
        for r in range(world):
            s = slice(r * Bl, (r + 1) * Bl)
            g1, g2 = a[s].to(device), b[s].to(device)
            tg = (0.5 * (g1 + g2)).clamp(0, 1)
            with torch.no_grad():
                ins = pipe.fusion_inputs(g1, g2)
            tr.bucket.zero()
            l = torch.nn.functional.l1_loss(tg, torch.clip(tr.net(*ins, variant=0), 0, 1))
            l.backward()
            acc += tr.bucket.flat
            lsum += float(l.detach())
        acc /= world
        grad_err = float((acc - flat_dist).abs().max())
        grad_ref = float(acc.abs().max())
        loss_single = lsum / world
    steps = 10
    step_ms_mode = {}
    for mode in ("eager", "cuda_graph"):               # frozen PhaseNet / AdaCoF part launched eagerly vs replayed as a CUDA graph
        tr.graph_frozen = mode == "cuda_graph"
        for _ in range(3):
            tr.step(f1, f2, target)
        torch.cuda.synchronize()
        dist.barrier(device_ids=[local_rank])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            tr.step(f1, f2, target)
        e1.record()
        torch.cuda.synchronize()
        step_ms_mode[mode] = maxr(e0.elapsed_time(e1) / steps)
    step_ms = min(step_ms_mode.values())
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier(device_ids=[local_rank])
    a0.record()
    for _ in range(steps):
        tr.bucket.all_reduce_mean(tr.group)
    a1.record()
    torch.cuda.synchronize()
    ar_ms = maxr(a0.elapsed_time(a1) / steps)
    if rank == 0:
        out["train"] = {"config": "BASELINE.json configs[4]: FusionNet training step, 256x256 crops, %d per GPU, global batch %d; frozen "
                                  "PhaseNet + 4x AdaCoFNet forward, FusionNet fwd+bwd, L1, Adam(1e-4)" % (Bl, Bl * world),
                        "ranks": world, "step_ms": round(step_ms, 3), "crops_per_s": round(Bl * world / step_ms * 1e3, 1),
                        "step_ms_by_launch_mode": {k: round(v, 3) for k, v in step_ms_mode.items()},
                        "allreduce_ms": round(ar_ms, 4), "allreduce_floats": int(tr.bucket.flat.numel()),
                        "collective": "one flat fp32 bucket, NCCL all-reduce (sum) + divide",
                        "backward": "libfvfi kernels: data gradient = the tcgen05 convolution over a zero canvas with the flipped filter "
                                    "(3xTF32), weight / bias gradients fp32 split over pixel ranges with a fixed summation order "
                                    "(csrc/conv_bwd.cu); no ATen / cuDNN convolution, pooling or interpolation kernel in the step",
                        "grad_max_abs_diff_vs_single_process": grad_err, "grad_max_abs": grad_ref,
                        "loss_distributed": loss_dist, "loss_single_process": loss_single,
                        "weights": "rank r initialised with seed r, rank 0's broadcast by the trainer"}
    del pipe, tr, inputs, f1, f2, target
    torch.cuda.empty_cache()

    # ---- configs[3]: the recipe at 3840x2160, frame pairs sharded across the ranks (2 per GPU), no collective on the data path
    try:
        H, W, Bl = 2160, 3840, 2
        pipe = FusionPipeline(H, W, device, phase_plane_chunk=6)
        pipe.max_batch = 2
        pipe.load_state(synth.seeded_state(0))
        r1, r2 = synth.seeded_frames(1, H, W, 100 + rank)
        g = torch.Generator().manual_seed(rank)
        gains = 0.8 + 0.2 * torch.rand((Bl, 1, 1, 1), generator=g)
        d1, d2 = (r1 * gains).clamp(0, 1).to(device), (r2 * gains).clamp(0, 1).to(device)
        for _ in range(2):
            o = pipe(d1, d2)
        torch.cuda.synchronize()
        dist.barrier(device_ids=[local_rank])
        steps = 3
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            o = pipe(d1, d2)
        e1.record()
        torch.cuda.synchronize()
        ms = maxr(e0.elapsed_time(e1) / steps)
        ok = bool(torch.isfinite(o).all()) and float(o.min()) >= 0 and float(o.max()) <= 1
        if rank == 0:
            out["pipeline4k"] = {"config": "BASELINE.json configs[3]: full fusion pipeline at 3840x2160, %d frame pairs per GPU sharded "
                                           "by batch over %d GPUs, no collective" % (Bl, world), "ranks": world,
                                 "ms_per_step": round(ms, 2), "frames_4k_per_s": round(Bl * world / ms * 1e3, 3),
                                 "finite_in_unit_range": ok}
    except Exception as ex:      # evidence record only: never fail the headline on it
        if rank == 0:
            out["pipeline4k"] = {"error": repr(ex)[:300]}
    return out
