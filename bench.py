#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native frame-synthesis hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload adacof|pipeline] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by the driver as
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 ... bench.py --gpus N ...
(one rank per GPU; frame pairs are sharded by batch, no collective on the data path -> weak scaling).

Prints ONE JSON line (rank 0).  Keys follow the driver contract: metric/value/unit, ms_per_step,
clocks, e2e (host buffers through the C-ABI / public API, copies inside the timed region),
gpu_launches, roofline (dominant HBM-bound kernel, CUDA-event timed, vs MEASURED_PEAKS.json) and
cpu_baseline (CPU oracle timed on this box's host cores on a bounded sample).

`--impl reference` times the reference arm: the reference's algorithm on the host CPU (the
reference has no CPU AdaCoF path and its pyramid dependency is absent, so this is the oracle
port on all host threads -- "kind": "port"; see DESIGN.md).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "fusion-method-for-video-frame-interpolation_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "interpolated_1080p_frames_per_s"
UNIT = "frames/s"
DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(outputs, path, seed=0):
    """Writes each output of the last timed step as path/<name>.npy (float32).  Outputs of more than DUMP_BYTES in all are
    sampled: the same fraction of every array, flattened, at element indices drawn from a generator seeded with ``seed``, so
    runs with the same arguments store the same elements and two builds can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    total = sum(t.numel() for t in outputs.values())
    keep = (DUMP_BYTES - 4096 * len(outputs)) // 4          # float32 elements, less room for the .npy headers
    rng = np.random.default_rng(seed)
    for name, t in outputs.items():
        t = t.detach()
        if total > keep:
            idx = np.sort(rng.integers(0, t.numel(), t.numel() * keep // total))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop_evt.wait(0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# workload: AdaCoF warp forward+backward, BASELINE.json configs[1]
# ------------------------------------------------------------------------------------------------
class AdaCoFWorkload:
    name = "adacof_F5_d1_fwd+bwd_1080p_batch8 (BASELINE.json configs[1])"
    B, C, H, W, F, D = 8, 3, 1088, 1920, 5, 1   # AdaCoFNet pads 1080 -> 1088 (fusion_adacofnet.py:182-185)
    dtype = "f32"
    metric = METRIC

    @classmethod
    def static_config(cls):
        return {"workload": cls.name, "frames_per_step_per_gpu": cls.B, "l2": "inputs larger than L2 (no flush needed)",
                "sharding": "frame pairs by batch, no collectives"}

    @classmethod
    def reference_full(cls, threads):
        return cls.cpu_sample(threads)

    def __init__(self, device, seed):
        import torch
        self.torch, self.device = torch, device
        B, C, H, W, F, D = self.B, self.C, self.H, self.W, self.F, self.D
        g = torch.Generator(device=device).manual_seed(seed)
        pad = (F - 1) * D
        self.inp = torch.rand((B, C, H + pad, W + pad), device=device, generator=g)
        self.w = torch.softmax(torch.randn((B, F * F, H, W), device=device, generator=g), 1)
        self.oi = (3 * torch.randn((B, F * F, H, W), device=device, generator=g)).clamp_(-16, 16)
        self.oj = (3 * torch.randn((B, F * F, H, W), device=device, generator=g)).clamp_(-16, 16)
        self.gout = torch.randn((B, C, H, W), device=device, generator=g)
        self.out = torch.empty((B, C, H, W), device=device)
        self.ev = []
        px = B * H * W
        # algorithmic bytes per launch (BASELINE.md section 3)
        self.bytes_fwd = 4 * (3 * F * F * px + C * B * (H + pad) * (W + pad) + C * px)
        self.bytes_bwd = 4 * (C * px + C * B * (H + pad) * (W + pad) + 3 * F * F * px + 3 * F * F * px)
        self.frames_per_step = B
        self.launches_per_step = 2

    def step(self, timed=False):
        from fvfi import adacof
        torch = self.torch
        if timed:
            e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            e[0].record()
        adacof.adacof_forward(self.inp, self.w, self.oi, self.oj, self.D, out=self.out)
        if timed:
            e[1].record()
        self.grads = adacof.adacof_backward(self.gout, self.inp, self.w, self.oi, self.oj, self.D, "none")
        if timed:
            e[2].record()
            self.ev.append(e)

    def outputs(self):
        """What a caller of the timed step receives: the warped frames and the three coefficient gradients."""
        _, gw, gi, gj = self.grads
        return {"out": self.out, "grad_weight": gw, "grad_offset_i": gi, "grad_offset_j": gj}

    def roofline(self, peak, peak_src):
        fwd = sum(e[0].elapsed_time(e[1]) for e in self.ev) / len(self.ev)
        bwd = sum(e[1].elapsed_time(e[2]) for e in self.ev) / len(self.ev)
        ach_f = self.bytes_fwd / (fwd * 1e-3) / 1e9
        ach_b = self.bytes_bwd / (bwd * 1e-3) / 1e9
        return {
            "bound": "hbm", "kernel": "adacof_fwd_tma<1,3,2> (TMA-streamed coefficients; offsets ~ N(0, 3^2): the adversarial gather)", "achieved": round(ach_f, 1), "peak": peak,
            "unit": "GB/s", "frac": round(ach_f / peak, 4),
            # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at this size, ncu --set full on the final tree
            # (profiles/r02_adacof_final_summary.txt): 5.395 + 0.200 GB per launch = 1.03 x the algorithmic bytes, i.e. every
            # coefficient map is read from HBM exactly once; backward 5.620 + 4.970 GB = 1.02 x
            "traffic": 5.595e9, "peak_source": peak_src,
            "ms_per_launch": round(fwd, 4), "algorithmic_bytes_per_launch": self.bytes_fwd,
            "other_kernels": [{"kernel": "adacof_fwd_tma<0,3,2> (fused backward: gW, g_alpha, g_beta; TMA-streamed coefficients)", "achieved": round(ach_b, 1),
                               "frac": round(ach_b / peak, 4), "ms_per_launch": round(bwd, 4),
                               "algorithmic_bytes_per_launch": self.bytes_bwd, "traffic": 10.590e9}],
        }

    def reference_gpu_kernels(self, steps=3):
        """Same-box bar: the reference's own CUDA kernels (oracle/_ref cubins), CUDA-event timed."""
        torch = self.torch
        try:
            from oracle import ref_kernels
            if not ref_kernels.have(self.B, self.C, self.H, self.W, self.F, self.D):
                return None
            ts = []
            for it in range(steps + 1):
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                e0.record()
                ref_kernels.forward(self.inp, self.w, self.oi, self.oj, self.D)
                e1.record()
                ref_kernels.backward(self.gout, self.inp, self.w, self.oi, self.oj, self.D)
                e2.record()
                torch.cuda.synchronize()
                if it:
                    ts.append((e0.elapsed_time(e1), e1.elapsed_time(e2)))
            f = sum(t[0] for t in ts) / len(ts)
            b = sum(t[1] for t in ts) / len(ts)
            return {"what": "reference CuPy kernels (adacof.py:6-258) compiled for sm_100a, same inputs",
                    "fwd_ms": round(f, 3), "bwd_ms": round(b, 3),
                    "frames_per_s": round(self.B / ((f + b) * 1e-3), 2)}
        except Exception as ex:  # evidence only; never fail the bench on it
            return {"error": repr(ex)[:200]}

    def e2e(self, steps):
        """fwd+bwd through the C-ABI *_host entry points: pinned host buffers, H2D + kernels + D2H."""
        import ctypes
        torch = self.torch
        from fvfi import _lib
        L = _lib.lib()
        host = {k: getattr(self, k).cpu().pin_memory() for k in ("inp", "w", "oi", "oj", "gout")}
        out = torch.empty(self.out.shape).pin_memory()
        gw, gi, gj = (torch.empty(self.w.shape).pin_memory() for _ in range(3))
        B, C, H, W, F, D = self.B, self.C, self.H, self.W, self.F, self.D
        pad = (F - 1) * D
        dims = (B, C, H + pad, W + pad, H, W, F, D)

        def one():
            _lib.check(L.fvfi_adacof_forward_host(host["inp"].data_ptr(), host["w"].data_ptr(), host["oi"].data_ptr(),
                                                  host["oj"].data_ptr(), out.data_ptr(), *dims))
            _lib.check(L.fvfi_adacof_backward_host(host["gout"].data_ptr(), host["inp"].data_ptr(),
                                                   host["w"].data_ptr(), host["oi"].data_ptr(), host["oj"].data_ptr(),
                                                   gw.data_ptr(), gi.data_ptr(), gj.data_ptr(), *dims))
        one()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            one()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        nb = lambda t: t.numel() * 4
        h2d = (nb(host["inp"]) + 3 * nb(host["w"])) * 2 + nb(host["gout"])
        d2h = nb(out) + 3 * nb(gw)
        ok = bool(torch.allclose(out.cuda(), self.out, atol=1e-6))
        return dt, h2d, d2h, ok

    @classmethod
    def cpu_sample(cls, threads, seed=0):
        """CPU oracle (port of adacof.py:6-258) on a bounded sample: 1 of the 8 frames, full 1088x1920."""
        from oracle import adacof as oa
        inp, w, oi, oj, g = oa.synth(1, cls.C, cls.H, cls.W, cls.F, cls.D, seed)
        t0 = time.perf_counter()
        oa.forward(inp, w, oi, oj, cls.D, threads=threads)
        oa.backward(g, inp, w, oi, oj, cls.D, threads=threads)
        dt = time.perf_counter() - t0
        return 1.0 / dt, dt, "fwd+bwd on 1 of the 8 frames (B=1, 3x1088x1920, F=5), C oracle"


WORKLOADS = {"adacof": AdaCoFWorkload}
try:
    from bench_pipeline import PhaseNet256Workload, Pipeline4KWorkload, PipelineWorkload
    WORKLOADS["pipeline"] = PipelineWorkload
    WORKLOADS["pipeline4k"] = Pipeline4KWorkload
    WORKLOADS["phasenet256"] = PhaseNet256Workload
except ImportError:
    pass
DEFAULT_WORKLOAD = os.environ.get("FVFI_BENCH_WORKLOAD", "pipeline" if "pipeline" in WORKLOADS else "adacof")


def run_reference(args, emit=print):
    """Reference arm: the reference's algorithm for this path on the host CPU with all host threads (the oracle port: the
    reference has no CPU warp and its pyramid package is absent, DESIGN.md section 7).

    `value` comes from ONE run of the workload at its FULL frame size (no extrapolation; BASELINE.md section 4 plans a single run
    for the 1080p case -- it takes about two minutes).  The K "steps" the driver asks for are bounded samples (one frame pair at
    about a quarter of the area) that show how a pixel-ratio extrapolation compares with the full-size run (`extrapolation`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload]
    threads = os.cpu_count() or 1
    t_start = time.perf_counter()
    value, dt_full, sample_full = wl.reference_full(threads)
    times, rates = [], []
    sample = ""
    budget = float(os.environ.get("FVFI_REF_SAMPLE_BUDGET_S", "60"))
    for it in range(args.steps):        # no separate warm-up samples: the full-size run before them has warmed every code path
        fps, dt, sample = wl.cpu_sample(threads, seed=it)
        times.append(dt)
        rates.append(fps)               # scaled to the metric's unit by the pixel ratio
        if time.perf_counter() - t_start - dt_full > budget:
            break
    extr = None
    if rates:
        hm = len(rates) / sum(1.0 / r for r in rates)
        extr = {"sample": sample, "samples_timed": len(rates), "extrapolated_value": round(hm, 5),
                "extrapolated_over_measured": round(hm / value, 3)}
    line = {
        "impl": "reference", "metric": wl.metric, "value": round(value, 5), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dt_full * 1e3, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
        "config": wl.static_config(),
        "measurement": "value = 1 / seconds of ONE full-size run; the %d steps are bounded samples, see `extrapolation`" % len(rates),
        "extrapolation": extr,
        "cpu_baseline": {"value": round(value, 5), "unit": UNIT, "cores": threads,
                         "kind": getattr(wl, "cpu_kind", "port"), "sample": sample_full, "seconds": round(dt_full, 2)},
        "e2e": {"value": round(value, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(json.dumps(line))
    return 0


def _quiet_stdout():
    """Only the JSON line may reach stdout (NCCL / library banners go to stderr): returns a writer for the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    return lambda text: os.write(real, (text + "\n").encode())


def main():
    emit = _quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="fvfi", choices=["fvfi", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-refbar", action="store_true", help="skip timing the reference's own CUDA kernels")
    ap.add_argument("--no-records", action="store_true", help="N > 1: skip the configs[4] training / configs[3] 4K records")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) to DIR/<name>.npy, float32; above %d MB in all, the "
                         "same seeded sample of each output" % (DUMP_BYTES // 10 ** 6))
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "fvfi":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl fvfi)")

    if args.impl == "reference":
        return run_reference(args, emit)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    wl = WORKLOADS[args.workload](device, seed=rank)   # every rank: its own shard of frame pairs
    warmup = max(args.warmup, 3)                        # timing rules: W >= 3
    for _ in range(warmup):
        wl.step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    from fvfi import _lib as _fl
    launches0 = _fl.lib().fvfi_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        wl.step(timed=True)
    e1.record()
    launches = _fl.lib().fvfi_launch_count() - launches0
    barrier()
    clocks = sampler.stop()
    ms = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms.item()) / args.steps
    value = wl.frames_per_step * world / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(wl.outputs(), args.dump_outputs)      # before anything below runs the workload again

    line = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        line = {
            "metric": wl.metric, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
            "config": wl.static_config(),
            "clocks": clocks, "gpu_launches": int(launches),
            "roofline": wl.roofline(peak, peak_src),
        }
        line["config_detail"] = getattr(wl, "config_extra", {})
        bar = wl.reference_gpu_kernels() if hasattr(wl, "reference_gpu_kernels") and not args.no_refbar else None
        if bar:
            line["reference_gpu_kernels"] = bar
    # end-to-end through the host-buffer C-ABI / public API (every rank runs it; max over ranks)
    if not args.no_e2e:
        dt, h2d, d2h, ok = wl.e2e(max(1, min(args.steps, 3)))
        t = torch.tensor([dt], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            line["e2e"] = {"value": round(wl.frames_per_step * world / float(t.item()), 3), "unit": UNIT,
                           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                           "ms_per_step": round(float(t.item()) * 1e3, 3), "matches_device_path": ok}
    if world > 1 and hasattr(wl, "parity") and not args.no_records:
        # BASELINE.json configs[4] (training step + NVLink all-reduce) and configs[3] (4K) on these N GPUs, outside the headline timing
        from bench_pipeline import multi_gpu_records
        del wl.pipe
        torch.cuda.empty_cache()
        rec = multi_gpu_records(device, rank, world, local_rank)
        if rank == 0:
            line.update(rec)
    if rank == 0 and not args.no_cpu:
        if world == 1:
            # the CPU leg runs at N = 1 only: at N > 1 the other ranks would spin in the NCCL barrier on the same host cores
            threads = os.cpu_count() or 1
            kept = {} if hasattr(wl, "parity") else None
            try:
                fps, dt, sample = wl.cpu_sample(threads, keep=kept) if kept is not None else wl.cpu_sample(threads)
            except TypeError:
                fps, dt, sample = wl.cpu_sample(threads)
            line["cpu_baseline"] = {"value": round(fps, 5), "unit": UNIT, "cores": threads,
                                    "kind": getattr(wl, "cpu_kind", "port"), "sample": sample,
                                    "seconds": round(dt, 2)}
            if kept:
                line["parity"] = wl.parity(kept)       # the GPU path against the oracle output just computed
        else:
            line["cpu_baseline"] = None
            line["cpu_baseline_note"] = "timed at N = 1 only (rank 0 would share the host cores with %d ranks polling NCCL)" % (world - 1)
    if rank == 0:
        emit(json.dumps(line))
    if world > 1:
        dist.barrier(device_ids=[local_rank])
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
