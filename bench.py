#!/usr/bin/env python
"""bench.py — sink Msamples/s on the BASELINE.json configs, headline = config 3.

Headline workload ("step" = one pass of the hot path over one batch), per GPU:
    cfg3: 1024 one-minute stereo signals (2 646 000 x 2 Float64 at 44.1 kHz, N(0,1)),
          ToFramerate(x, 48 kHz) |> sink            -> 2 880 000 x 2 each, 90.5 GB per step
the largest BASELINE config that fits one B200 (cfg5's 4096 x 2.95 GB signals run in waves; a wave
of it is reported under `configs`).  One fused polyphase-FIR stage on the FP64 tensor cores
(csrc/k_fir_mma.cuh).

  value      output samples / s, inputs and outputs resident in HBM, CUDA events on the
             launching stream, max over ranks
  e2e        same metric through the public C-ABI call `sigops_plan_run` with HOST buffers
             (H2D + kernels + D2H inside the timed region), pinned and pageable
  roofline   dominant kernel (k_fir_mma): 15.35 algorithmic bytes per output sample / its
             average launch duration (events around every launch), against MEASURED_PEAKS.json
  configs    the same fields for cfg2 (IIR scan), cfg4 (README pipeline x512) and one wave of cfg5
  cpu_baseline  the oracle's C restatement of the reference algorithm on the host cores
             (kind "port": the reference is Julia and cannot run here)

`--impl reference` times that CPU restatement alone on the same config.
`--dump-outputs DIR` writes a fixed sample of the outputs of the last timed step of cfg3 and of each sub-config
(dump_sample); inputs are seeded, so two builds run with the same arguments can be compared output for output.
Normpower sums x² with atomics, so outputs downstream of it (cfg4) may differ in the last bits from run to run.
Multi-GPU: one rank per GPU under torchrun, instances sharded, no data-path collective
(weak scaling: 1024 signals per GPU).  `--single-process` instead drives all N GPUs from ONE
process through `sigops_ctx_create(devices, N)` (the drop-in's own sharding).
"""
import argparse
import ctypes as C
import json
import math
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "sink Msamples/s (Filt+resample+Mix chain) at 1/2/4/8 B200; % of HBM peak"
FS_IN, FS_OUT = 44100.0, 48000.0
N_IN, N_OUT, NCH = 2646000, 2880000, 2
NINST = 1024
WORKLOAD = ("cfg3: 1024 x (2646000x2) Float64 @44.1kHz per GPU, ToFramerate(48kHz) |> sink "
            "(FIRArbitrary polyphase resampler, 32 phases x 38 taps) -> 2880000x2 each")
FIR_BYTES_PER_OUT = 8.0 + 8.0 * FS_IN / FS_OUT          # SURVEY.md §8d: 15.35 B per output sample


# ------------------------------------------------------------------------------------------------
# workloads (graphs are built on zero arrays of the right shape; the data lives on the device)
# ------------------------------------------------------------------------------------------------

def graph_cfg2():
    from signalops import Amplify, Filt, Lowpass, Signal, dB, Hz
    return Signal(np.zeros((480000, 2)), 48000.0 * Hz) >> Filt(Lowpass, 4000.0 * Hz, order=8) >> Amplify(-20 * dB)


def graph_cfg3(x=None):
    from signalops import Hz, Signal, ToFramerate
    x = np.zeros((N_IN, NCH)) if x is None else x
    return ToFramerate(Signal(x, FS_IN * Hz), FS_OUT * Hz)


def graph_cfg4(arrays=None):
    from signalops import (AffineSin, Amplify, Append, Bandstop, Filt, Mix, Normpower, Ramp, Sawtooth, Signal,
                           ToFramerate, Until, dB, Hz, kHz, s, sin)
    fs = 44.1 * kHz
    a = arrays or [np.zeros(88200), np.zeros(220500), np.zeros(44100)]
    s1 = Signal(sin, ω=1 * kHz) >> Until(5 * s) >> Ramp() >> Normpower >> Amplify(-20 * dB)
    s2 = Signal(a[0], fs) >> Normpower >> Amplify(-20 * dB)
    s3 = Signal(Sawtooth(), ω=1 * kHz) >> Until(2 * s) >> Ramp() >> Normpower >> Amplify(-20 * dB)
    s4 = (Signal(a[1], fs) >> Amplify(Signal(AffineSin(0.5, 0.5), ω=5 * Hz)) >> Until(5 * s) >> Normpower
          >> Amplify(-20 * dB))
    x = Signal(sin, ω=1 * kHz) >> Until(1 * s) >> Ramp() >> Normpower >> Amplify(-20 * dB + 5 * dB)
    y = Signal(a[2], fs) >> Until(1 * s) >> Filt(Bandstop, 0.5 * kHz, 2 * kHz) >> Normpower >> Amplify(-20 * dB)
    return Append(s1, s2, s3, s4, Mix(x, y)) >> Normpower >> Amplify(-20 * dB) >> ToFramerate(fs)


def graph_cfg5(x=None, nch=64):
    from signalops import AffineSin, Amplify, Bandpass, Filt, Mix, Ramp, Signal, Until, Hz, kHz, ms, s, sin
    x = np.zeros((5760000, nch)) if x is None else x
    am = Amplify(Signal(x, 96 * kHz), Signal(AffineSin(0.5, 0.5), ω=5 * Hz)) >> Until(60 * s)
    return am >> Filt(Bandpass, 500 * Hz, 4 * kHz) >> Ramp(10 * ms) >> Mix(Signal(sin, ω=1 * kHz) >> Until(60 * s))


SUBCONFIGS = {
    "cfg2": dict(graph=graph_cfg2, ninst=256, kernel="iir_main",
                 workload="cfg2: 256 x (480000x2) Float64 @48kHz, Filt(Lowpass,4kHz,Butterworth 8 = 4 biquads) |> Amplify(-20dB)"),
    "cfg4": dict(graph=graph_cfg4, ninst=512, kernel="map",
                 workload="cfg4: 512 x README pipeline @44.1kHz: Append(5 generated/filtered sounds, each Normpower'd) |> "
                          "Normpower |> Amplify(-20dB) |> ToFramerate(44.1kHz) -> 661500x1 each"),
    "cfg5": dict(graph=graph_cfg5, ninst=16, kernel="iir_main",
                 workload="cfg5 (one wave of the 4096): 16 x (5760000x64) Float64 @96kHz, AM noise |> Filt(Bandpass 0.5-4kHz, "
                          "Butterworth 5 = 5 biquads) |> Ramp(10ms) |> Mix(1kHz tone)"),
}


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------

def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    except Exception:
        return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def ncu_traffic(kernel):
    """dram bytes per launch from the committed `ncu --set full` summary (profiles/ncu_summary.json):
    a capture of the same kernel on a stated batch, NOT a measurement of this run."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


def mem_available_bytes():
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable"):
                return int(ln.split()[1]) * 1024
    except Exception:
        pass
    return 64 << 30


class ClockSampler:
    """SM clock and throttle reasons polled through NVML in a background thread DURING the
    timed region (the same counters `nvidia-smi --query-gpu=clocks.sm,...` prints)."""

    def __init__(self, gpu_index):
        import threading
        self.samples, self.max_mhz = [], None
        self._stop = threading.Event()
        self._ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self._ok = True
        except Exception as e:                                   # pragma: no cover
            self.err = repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        if not self._ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                t = time.perf_counter()
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                try:
                    watts = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    watts = None
                self.samples.append((t, mhz, [k for k, bit in names.items() if mask & bit], watts))
            except Exception:
                pass
            time.sleep(0.002)

    def window(self, t0, t1):
        inside = [x for x in self.samples if t0 <= x[0] <= t1]
        return {"sm_mhz": statistics.median(x[1] for x in inside) if inside else None,
                "sm_mhz_min": min((x[1] for x in inside), default=None),
                "sm_max_mhz": self.max_mhz, "samples": len(inside),
                "power_w_max": max((x[3] for x in inside if x[3] is not None), default=None),
                "reasons": sorted({r for x in inside for r in x[2]})}

    def stop(self):
        self._stop.set()
        self.t.join(timeout=2)


DUMP_BYTES = {"cfg3": 32 << 20, "cfg2": 8 << 20, "cfg4": 8 << 20, "cfg5": 8 << 20}   # 56 MiB in all


def dump_sample(out_dir, name, y):
    """Writes a fixed, seeded sample of one batch output y (ninst, nchannels, nframes), on the device or the
    host, as out_dir/<name>.npy in y's own dtype: up to 8 instances (the first and the last among them) x every
    channel x the first and last frames and a seeded draw of the frames in between, DUMP_BYTES[name] at most.
    The same shape of y always gives the same sample, so two builds can be compared value for value."""
    import torch
    ninst, nch, nframes = y.shape
    rng = np.random.default_rng(1983)
    inst = np.unique(np.concatenate([[0, ninst - 1], rng.permutation(np.arange(1, ninst - 1))[:6]]))
    nf = max(1, DUMP_BYTES[name] // (len(inst) * nch * y.element_size()))
    if nf >= nframes:
        frames = np.arange(nframes)
    else:
        edge = min(1024, nf // 4)
        middle = edge + rng.choice(nframes - 2 * edge, nf - 2 * edge, replace=False)
        frames = np.sort(np.concatenate([np.arange(edge), middle, np.arange(nframes - edge, nframes)]))
    frames = torch.from_numpy(frames).to(y.device)
    s = torch.stack([y[int(i)].index_select(1, frames) for i in inst])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), s.cpu().numpy())


def bind_to_gpu_numa_node(gpu_index):
    """Run this rank (and first-touch its pinned host buffers) on the CPUs local to its GPU, so that the
    end-to-end copies do not cross the socket interconnect.  Best effort: any failure leaves the default."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, m in enumerate(words) for b in range(64) if (int(m) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle's C restatement of the reference algorithm (checker and baseline only)
# ------------------------------------------------------------------------------------------------

def cpu_resample_batch(x, threads, simd=False):
    """x: (nsig, NCH, N_IN) Float64 -> (nsig, NCH, N_OUT) by oracle/cpu_ref.c `oracle_resample_batch`
    (the reference's FilteredSignal block loop over DSP.jl's FIRArbitrary kernel, blocksize 4096).
    simd=True lets the dot products reassociate into vector lanes like DSP.jl's `@simd` loops (timing
    baseline); the parity gate uses the strict left-to-right sums."""
    from oracle import dspjl_ref as D
    r = D.Resampler(FS_OUT / FS_IN)
    r.st.simd = 1 if simd else 0
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.empty((x.shape[0], x.shape[1], N_OUT if x.shape[2] == N_IN else int(math.ceil(x.shape[2] * FS_OUT / FS_IN))))
    dp = C.POINTER(C.c_double)
    D.lib().oracle_resample_batch(x.ctypes.data_as(dp), y.ctypes.data_as(dp), x.shape[0], x.shape[2], y.shape[2],
                                  x.shape[1], C.byref(r.st), 4096, threads)
    return y


def cpu_baseline(seconds_target=12.0, threads=None):
    cores = threads or os.cpu_count() or 1
    rng = np.random.default_rng(1983)
    x1 = rng.standard_normal((1, NCH, N_IN))
    t0 = time.perf_counter()
    cpu_resample_batch(x1, 1, simd=True)
    t1 = time.perf_counter() - t0
    per_core = N_OUT * NCH / t1 / 1e6
    nsig = int(max(cores, min(NINST, cores * max(1, int(seconds_target / max(t1, 1e-3))))))
    nsig = (nsig // cores) * cores
    x = np.broadcast_to(x1, (nsig, NCH, N_IN)).copy()
    t0 = time.perf_counter()
    cpu_resample_batch(x, cores, simd=True)
    t = time.perf_counter() - t0
    return {"value": nsig * N_OUT * NCH / t / 1e6, "unit": "Msamples/s", "cores": cores, "kind": "port",
            "one_core_value": per_core, "seconds": t, "instances": nsig,
            "sample": f"{nsig} of the {NINST} signals (2646000x2 -> 2880000x2 each), {cores} threads, one signal per thread, "
                      f"{t:.1f} s; C restatement of the reference block loop + DSP.jl FIRArbitrary (no Julia in this image)"}


def run_reference(args, rank):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    per_step = 2.0            # bounded sample per step so that warmup+steps finish in a few minutes
    vals = []
    for _ in range(args.warmup + args.steps):
        vals.append(cpu_baseline(seconds_target=per_step, threads=cores))
    vals = vals[args.warmup:]
    v = statistics.median(b["value"] for b in vals)
    nsig = vals[0]["instances"]
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": nsig * N_OUT * NCH / (v * 1e6) * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "instances_per_step": nsig,
                       "note": "reference CPU algorithm (C restatement; the Julia reference cannot run here); "
                               "each step is a bounded sample of the workload"},
            "cpu_baseline": {"value": v, "unit": "Msamples/s", "cores": cores, "kind": "port",
                             "sample": vals[0]["sample"]},
            "e2e": {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------

class DeviceBatch:
    """One lowered plan + `ninst` instances of its inputs/outputs resident on a device."""

    def __init__(self, ctx, graph, ninst, dev, seed, dev_index=0):
        import torch
        from signalops import cabi
        from signalops.lowering import lower
        self.torch, self.cabi = torch, cabi
        t0 = time.perf_counter()
        self.plan = lower(graph)
        self.lower_ms = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        self.cp = cabi.CompiledPlan(ctx, self.plan.tobytes())
        self.plan_create_ms = (time.perf_counter() - t0) * 1e3
        self.ctx, self.ninst, self.dev_index = ctx, ninst, dev_index
        g = torch.Generator(device=dev)
        g.manual_seed(seed)
        tdt = lambda d: torch.float32 if d.dtype == cabi.F32 else torch.float64   # noqa: E731
        self.xs = []
        for d in self.plan.inputs:
            x = torch.empty((ninst, d.nchannels, d.nframes), dtype=tdt(d), device=dev)
            for i0 in range(0, ninst, 64):          # generate in slices: randn_ on one 43 GB tensor is fine, temporaries are not
                x[i0:i0 + 64].normal_(generator=g)
            self.xs.append(x)
        self.ys = [torch.empty((ninst, d.nchannels, d.nframes), dtype=tdt(d), device=dev) for d in self.plan.outputs]
        self.ins, self.outs = self._bufs(self.xs), self._bufs(self.ys)
        self.out_samples = ninst * sum(d.nchannels * d.nframes for d in self.plan.outputs)
        self.alg_bytes = self.cp.algorithmic_bytes() * ninst

    def _bufs(self, ts):
        cabi, torch, n = self.cabi, self.torch, self.ninst
        arr = (cabi.Buffer * (n * max(len(ts), 1)))()
        for i in range(n):
            for k, t in enumerate(ts):
                arr[i * len(ts) + k] = cabi.Buffer(t[i].data_ptr(), t.shape[2], t.shape[1],
                                                   cabi.F32 if t.dtype == torch.float32 else cabi.F64, t.shape[2])
        return arr

    def step(self, stream):
        self.cp.run_device(self.ninst, self.ins, self.outs, stream=stream.cuda_stream, dev_index=self.dev_index)

    def free(self):
        self.cp.close()
        self.xs = self.ys = self.ins = self.outs = None
        self.torch.cuda.empty_cache()


def time_steps(batch, stream, steps, barrier, ctx, sampler=None):
    """K steps bracketed by barrier + synchronize; returns (ms total, per-kind profile, clocks)."""
    import torch
    ctx.set_profiling(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(steps):
        batch.step(stream)
    e1.record(stream)
    barrier()
    t1 = time.perf_counter()
    ms = e0.elapsed_time(e1)
    prof = ctx.profile_collect(batch.dev_index)
    ctx.set_profiling(False)
    return ms, prof, (sampler.window(t0, t1) if sampler else None)


def warm(batch, stream, nmin, seconds):
    import torch
    n, t0 = 0, time.perf_counter()
    while n < nmin or time.perf_counter() - t0 < seconds:
        batch.step(stream)
        n += 1
        if n % 8 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    return n


def parity_cfg3(batch, which):
    """GPU output of whole instances against the C oracle (all 2 880 000 x 2 outputs each)."""
    worst = 0.0
    x = np.stack([batch.xs[0][i].cpu().numpy() for i in which])
    want = cpu_resample_batch(x, min(len(which), os.cpu_count() or 1))
    for k, i in enumerate(which):
        got = batch.ys[0][i].cpu().numpy()
        worst = max(worst, float(np.max(np.abs(got - want[k])) / np.sqrt(np.mean(want[k] ** 2))))
    return worst


def parity_sub(name, batch):
    """Parity gate of a sub-config on the data actually benchmarked (oracle = checker only)."""
    import oracle
    n = batch.ninst
    worst = 0.0
    if name == "cfg2":
        from oracle import dspjl_ref as D
        z, p, k = D.design_zpk("Lowpass", [4000.0], 48000.0, ("butterworth", 8))
        coef, gg = D.zpk2sos_dspjl(z, p, k)
        amp = 10.0 ** (-20 / 20)
        for i in (0, n // 3, 2 * n // 3, n - 1):
            xi = batch.xs[0][i].cpu().numpy()
            want = np.stack([D.sos_filt(xi[c], coef, gg, np.zeros((coef.shape[0], 2))) * amp for c in range(xi.shape[0])])
            got = batch.ys[0][i].cpu().numpy()
            worst = max(worst, float(np.max(np.abs(got - want)) / np.sqrt(np.mean(want ** 2))))
    elif name == "cfg4":
        for i in (0, n - 1):
            bylen = {x.shape[2]: x[i, 0].cpu().numpy().copy() for x in batch.xs}      # the three noise arrays differ in length
            want, _ = oracle.sink(graph_cfg4([bylen[88200], bylen[220500], bylen[44100]]))
            got = batch.ys[0][i].cpu().numpy().T
            worst = max(worst, float(np.max(np.abs(got - want)) / np.sqrt(np.mean(want ** 2))))
    elif name == "cfg5":
        for i in (0, n - 1):
            chans = [0, 63]                 # channels are independent in this chain: check two at full length
            xi = np.ascontiguousarray(batch.xs[0][i][chans].cpu().numpy().T)
            want, _ = oracle.sink(graph_cfg5(xi, nch=len(chans)))
            got = batch.ys[0][i][chans].cpu().numpy().T
            worst = max(worst, float(np.max(np.abs(got - want)) / np.sqrt(np.mean(want ** 2))))
    return worst


def run_subconfig(name, ctx, dev, stream, barrier, rank, steps, min_seconds=0.5, dump_dir=None):
    import torch
    cfg = SUBCONFIGS[name]
    batch = DeviceBatch(ctx, cfg["graph"](), cfg["ninst"], dev, 1983 + 17 * rank)
    nwarm = warm(batch, stream, 3, 0.2)
    err = parity_sub(name, batch)
    tol = 1e-9
    if not err < tol:
        raise SystemExit(f"bench parity check failed for {name}: max err / rms = {err:g}")
    # >= `steps` steps and >= min_seconds of timed region
    ms1, _, _ = time_steps(batch, stream, 1, barrier, ctx)
    k = max(steps, int(math.ceil(min_seconds * 1e3 / max(ms1, 1e-3))))
    ms, prof, _ = time_steps(batch, stream, k, barrier, ctx)
    if dump_dir:
        dump_sample(dump_dir, name, batch.ys[0])
    peak, _ = measured_peaks()
    kind = cfg["kernel"]
    kms, kn = prof.get(kind, (0.0, 0))
    rec = {"workload": cfg["workload"], "instances": cfg["ninst"], "steps": k, "warmup_steps_run": nwarm,
           "ms_per_step": ms / k, "value": batch.out_samples * k / (ms * 1e-3) / 1e6, "unit": "Msamples/s",
           "algorithmic_bytes_per_step": batch.alg_bytes,
           "step_gbs": batch.alg_bytes / (ms / k * 1e-3) / 1e9, "step_frac_of_hbm_peak": batch.alg_bytes / (ms / k * 1e-3) / 1e9 / peak,
           "gpu_launches_per_step": sum(v[1] for v in prof.values()) // k,
           "kernels_ms_per_step": {kk: v[0] / k for kk, v in prof.items()},
           "kernel_launches_per_step": {kk: v[1] // k for kk, v in prof.items()},
           "dominant_kernel": kind, "dominant_kernel_share_of_step": (kms / ms) if ms else None,
           "parity_max_err_over_rms": err, "lower_ms": batch.lower_ms, "plan_create_ms": batch.plan_create_ms}
    batch.free()
    del batch
    torch.cuda.empty_cache()
    return rec


def e2e_run(ctx, cp, x_dev, ninst, steps, barrier, pinned):
    """The reference-facing call with HOST buffers: sigops_plan_run(plan, ninst, in, out)."""
    import torch
    from signalops import cabi
    xh = torch.empty((ninst, NCH, N_IN), dtype=torch.float64, pin_memory=pinned)
    yh = torch.empty((ninst, NCH, N_OUT), dtype=torch.float64, pin_memory=pinned)
    for i0 in range(0, ninst, 64):
        i1 = min(ninst, i0 + 64)
        xh[i0:i1].copy_(x_dev[i0:i1])
    if not pinned:
        yh.zero_()                                   # touch the pages: first-touch faults are not the library's cost
    hin = cabi.CompiledPlan.host_buffers([xh[i].numpy().T for i in range(ninst)])
    hout = cabi.CompiledPlan.host_buffers([yh[i].numpy().T for i in range(ninst)])
    st = cabi.Stats()

    def step():
        cabi._check(cp.lib, ctx.handle, cp.lib.sigops_plan_run(cp.handle, ninst, hin, hout, C.byref(st)))
    step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    barrier()
    sec = time.perf_counter() - t0
    return sec, st, yh


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from signalops import cabi

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    ctx = cabi.Context([local_rank])
    ninst = args.ninst
    batch = DeviceBatch(ctx, graph_cfg3(), ninst, dev, 1983 + rank)
    # a real (non-legacy) stream: handle 0 would mean "library stream + synchronise" to the C ABI
    torch.cuda.synchronize()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    nwarm = warm(batch, stream, max(args.warmup, 3), 0.3)
    barrier()

    # ---- parity gate on the data actually benchmarked: whole instances against the C oracle
    which = sorted({0, ninst // 3, (2 * ninst) // 3, ninst - 1})
    worst = parity_cfg3(batch, which)
    if not worst < 1e-9:
        raise SystemExit(f"bench parity check failed: max err / rms = {worst:g}")

    # ---- timed region: exactly K steps, device resident
    ms, prof, clocks = time_steps(batch, stream, args.steps, barrier, ctx, sampler)
    if args.dump_outputs and rank == 0:
        dump_sample(args.dump_outputs, "cfg3", batch.ys[0])
    # ---- the same loop for >= 2 s (power / thermal behaviour; reported beside the K-step number)
    k_sus = max(args.steps, int(math.ceil(2000.0 / max(ms / args.steps, 1e-3))))
    ms_sus, _, clocks_sus = time_steps(batch, stream, k_sus, barrier, ctx, sampler)
    if world > 1:
        t = torch.tensor([ms, ms_sus], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_sus = float(t[0].item()), float(t[1].item())
    samples_step = batch.out_samples
    value = world * samples_step * args.steps / (ms * 1e-3) / 1e6

    # ---- e2e: host buffers through sigops_plan_run (H2D + kernels + D2H), pinned and pageable
    e2e_ninst = args.e2e_ninst
    if e2e_ninst <= 0:
        per_inst = (N_IN + N_OUT) * NCH * 8
        fit = int(0.35 * mem_available_bytes() / max(world, 1) / per_inst)
        e2e_ninst = max(16, min(ninst, 256, fit // 16 * 16))
    e2e_steps = max(2, min(args.steps, 4))
    sec_pin, st, yh = e2e_run(ctx, batch.cp, batch.xs[0], e2e_ninst, e2e_steps, barrier, pinned=True)
    ref0 = batch.ys[0][0].cpu()
    e2e_err = float((yh[0] - ref0).abs().max() / ref0.pow(2).mean().sqrt())
    st_pin = {k: getattr(st, k) for k in ("h2d_bytes", "d2h_bytes", "h2d_ms", "gpu_ms", "d2h_ms")}
    del yh
    pg_ninst = max(16, e2e_ninst // 4)
    sec_pg, st2, yh2 = e2e_run(ctx, batch.cp, batch.xs[0], pg_ninst, 2, barrier, pinned=False)
    pg_err = float((yh2[0] - ref0).abs().max() / ref0.pow(2).mean().sqrt())
    del yh2
    if world > 1:
        t = torch.tensor([sec_pin, sec_pg], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec_pin, sec_pg = float(t[0].item()), float(t[1].item())
    e2e_value = world * e2e_ninst * N_OUT * NCH * e2e_steps / sec_pin / 1e6
    e2e_pg_value = world * pg_ninst * N_OUT * NCH * 2 / sec_pg / 1e6

    # ---- the call a user makes: sink(list of graphs, GPUSink) — lowering of every graph in Python, page-locked
    # result arrays (pooled after the first call), sigops_plan_run on pageable inputs
    api = None
    if rank == 0:
        from signalops import GPUSink, sink_batch
        napi = 32
        gsink = GPUSink([local_rank])
        xs_api = [np.asfortranarray(batch.xs[0][i].cpu().numpy().T) for i in range(napi)]
        res_api = sink_batch([graph_cfg3(x) for x in xs_api], gsink)       # first call: plan creation, staging ring
        t0 = time.perf_counter()
        nrep = 3
        for _ in range(nrep):
            del res_api
            res_api = sink_batch([graph_cfg3(x) for x in xs_api], gsink)
        sec_api = (time.perf_counter() - t0) / nrep
        api_err = float(np.max(np.abs(res_api[0][0].T - ref0.numpy())) / float(ref0.pow(2).mean().sqrt()))
        api = {"value": napi * N_OUT * NCH / sec_api / 1e6, "unit": "Msamples/s", "instances_per_call": napi,
               "ms_per_call": sec_api * 1e3, "matches_device_run": bool(api_err < 1e-9),
               "what": "sink([ToFramerate(Signal(x,44.1kHz),48kHz) for x in xs], GPUSink()): graph construction, lowering of "
                       "every graph (Python mirror), pageable numpy inputs and results (first-touch page faults of the fresh result arrays included)"}
        del res_api, xs_api
        gsink.close()

    peak, peak_src = measured_peaks()
    fir_ms, fir_n = prof.get("fir", (0.0, 0))
    alg_bytes = FIR_BYTES_PER_OUT * samples_step
    achieved = alg_bytes / (fir_ms / max(fir_n, 1) * 1e-3) / 1e9 if fir_n else None
    launches = int(sum(n for _, n in prof.values()))
    kernels_ms = {k: v[0] / args.steps for k, v in prof.items()}
    dfma, copy_gbs = ctx.measure_peaks(0) if rank == 0 else (None, None)

    # ---- the other BASELINE configs, same fields (rank 0's GPU; they need the 90 GB back first)
    subs = {}
    lower_ms, create_ms = batch.lower_ms, batch.plan_create_ms
    batch.free()
    del batch
    torch.cuda.empty_cache()
    if rank == 0 and args.configs:
        for name in args.configs.split(","):
            if name in SUBCONFIGS:
                subs[name] = run_subconfig(name, ctx, dev, stream, lambda: torch.cuda.synchronize(), rank, args.steps,
                                           dump_dir=args.dump_outputs)
    if sampler:
        sampler.stop()

    if rank == 0:
        fir_launch_ms = fir_ms / max(fir_n, 1)
        # 48 of 38 taps per output are issued (band padding to a multiple of 4 positions): DMMA.8x8x4 work
        dmma_fma = 48.0 * samples_step
        cpu = cpu_baseline()
        line = {
            "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "warmup_steps_run": nwarm, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "instances_per_gpu": ninst, "instances_per_step": ninst,
                       "global_instances": ninst * world,
                       "samples_per_step_per_gpu": samples_step, "parallelism": f"batch-shard x{world}, no collective",
                       "l2": "each step reads 43.3 GB and writes 47.2 GB per GPU: far larger than the 126 MB L2",
                       "parity_max_err_over_rms": worst, "parity_instances_checked": which,
                       "parity_against": "oracle/cpu_ref.c oracle_resample_batch, all 2880000x2 outputs of each instance",
                       "north_star_batch_4096_signals_s": 4096.0 * N_OUT * NCH / (value * 1e6),
                       "lower_ms": lower_ms, "plan_create_ms": create_ms},
            "clocks": clocks,
            "sustained": {"steps": k_sus, "seconds": ms_sus * 1e-3, "ms_per_step": ms_sus / k_sus,
                          "value": world * samples_step * k_sus / (ms_sus * 1e-3) / 1e6, "clocks": clocks_sus},
            "e2e": {"value": e2e_value, "unit": "Msamples/s", "memory": "pinned",
                    "instances_per_step": e2e_ninst,
                    "h2d_bytes_per_step": int(st_pin["h2d_bytes"]), "d2h_bytes_per_step": int(st_pin["d2h_bytes"]),
                    "steps": e2e_steps, "ms_per_step": sec_pin / e2e_steps * 1e3,
                    "matches_device_run": bool(e2e_err < 1e-9), "max_err_over_rms_vs_device_run": e2e_err,
                    "h2d_ms": st_pin["h2d_ms"], "kernels_ms": st_pin["gpu_ms"], "d2h_ms": st_pin["d2h_ms"],
                    "h2d_gbs_per_gpu": st_pin["h2d_bytes"] / max(st_pin["h2d_ms"], 1e-9) / 1e6,
                    "d2h_gbs_per_gpu": st_pin["d2h_bytes"] / max(st_pin["d2h_ms"], 1e-9) / 1e6,
                    "link_gbs_per_gpu": (st_pin["h2d_bytes"] + st_pin["d2h_bytes"]) / (sec_pin / e2e_steps) / 1e9,
                    "limit": "host<->device link (PCIe): 15.35 B cross it per output sample",
                    "pageable": {"value": e2e_pg_value, "unit": "Msamples/s", "instances_per_step": pg_ninst,
                                 "ms_per_step": sec_pg / 2 * 1e3, "matches_device_run": bool(pg_err < 1e-9),
                                 "note": "caller arrays not page-locked (what a Julia Array is): staged through the "
                                         "library's pinned ring"},
                    "public_api": api},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "k_fir_tmap (FP64 tensor-core polyphase FIR: DMMA.8x8x4, tensor-map TMA ring and stores)",
                         "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None,
                         "traffic": ncu_traffic("k_fir_mma_traffic_bytes_per_out_sample") and
                         ncu_traffic("k_fir_mma_traffic_bytes_per_out_sample") * samples_step / max(fir_n // args.steps, 1),
                         "traffic_source": "replayed from profiles/ncu_summary.json (ncu --set full capture of the same kernel, "
                                           "bytes per output sample x this launch's samples); not measured in this run",
                         "peak_source": peak_src, "algorithmic_bytes_per_step": alg_bytes,
                         "algorithmic_bytes_per_out_sample": FIR_BYTES_PER_OUT,
                         "launches_per_step": fir_n // args.steps, "launch_ms": fir_launch_ms,
                         "step_frac": (alg_bytes / (ms / args.steps * 1e-3) / 1e9) / peak,
                         "tensor_fp64": {"dmma_fma_per_out_sample": 48, "useful_fma_per_out_sample": 38,
                                         "dfma_per_s_measured": dfma, "copy_gbs_measured_here": copy_gbs,
                                         "fma_per_s": dmma_fma / (fir_ms / args.steps * 1e-3) if fir_n else None,
                                         "frac_of_measured_fp64_fma_peak": (dmma_fma / (ms / args.steps * 1e-3) / dfma) if dfma else None}},
            "kernels_ms_per_step": kernels_ms,
            "configs": subs,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_single_process(args):
    """All N GPUs driven from ONE process through one context (`sigops_ctx_create(devices, N)`):
    the drop-in's own batch sharding, host buffers in, host buffers out."""
    import torch
    from signalops import cabi
    from signalops.lowering import lower
    n = args.gpus
    ctx = cabi.Context(list(range(n)))
    cp = cabi.CompiledPlan(ctx, lower(graph_cfg3()).tobytes())
    ninst = args.e2e_ninst if args.e2e_ninst > 0 else 64 * n
    g = torch.Generator(device="cuda:0")
    g.manual_seed(1983)
    x = torch.randn((min(ninst, 64), NCH, N_IN), dtype=torch.float64, device="cuda:0", generator=g)
    xh = torch.empty((ninst, NCH, N_IN), dtype=torch.float64, pin_memory=True)
    yh = torch.empty((ninst, NCH, N_OUT), dtype=torch.float64, pin_memory=True)
    for i0 in range(0, ninst, x.shape[0]):
        xh[i0:i0 + x.shape[0]].copy_(x[:min(x.shape[0], ninst - i0)])
    hin = cabi.CompiledPlan.host_buffers([xh[i].numpy().T for i in range(ninst)])
    hout = cabi.CompiledPlan.host_buffers([yh[i].numpy().T for i in range(ninst)])
    st = cabi.Stats()

    def step():
        cabi._check(cp.lib, ctx.handle, cp.lib.sigops_plan_run(cp.handle, ninst, hin, hout, C.byref(st)))
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    sec = time.perf_counter() - t0
    if args.dump_outputs:
        dump_sample(args.dump_outputs, "cfg3", yh)
    which = sorted({0, ninst - 1})
    want = cpu_resample_batch(np.stack([xh[i].numpy() for i in which]), len(which))
    err = max(float(np.max(np.abs(yh[i].numpy() - want[k])) / np.sqrt(np.mean(want[k] ** 2))) for k, i in enumerate(which))
    print(json.dumps({"mode": "single-process", "metric": METRIC, "n_gpus": n, "instances_per_step": ninst, "steps": args.steps,
                      "e2e": {"value": ninst * N_OUT * NCH * args.steps / sec / 1e6, "unit": "Msamples/s",
                              "ms_per_step": sec / args.steps * 1e3, "h2d_bytes_per_step": int(st.h2d_bytes),
                              "d2h_bytes_per_step": int(st.d2h_bytes), "kernels_ms_slowest_device": st.gpu_ms},
                      "parity_max_err_over_rms": err, "config": {"workload": WORKLOAD.replace("1024", str(ninst))}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ninst", type=int, default=NINST, help="signals per GPU and step (BASELINE config 3: 1024)")
    ap.add_argument("--e2e-ninst", type=int, default=0, help="signals per end-to-end step (0 = sized from host memory)")
    ap.add_argument("--configs", default="cfg2,cfg4,cfg5", help="sub-records to add (comma separated; '' = none)")
    ap.add_argument("--single-process", action="store_true", help="drive all --gpus devices from one process/context")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of what the last step computed as DIR/<config>.npy "
                         "(rank 0's cfg3 and each sub-config; 56 MiB at most)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's results; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
    elif args.single_process:
        run_single_process(args)
    else:
        run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
