"""Cost of a traced generator closure on the device, at BASELINE config 5's shape (one wave: 16 signals x 5 760 000
frames x 64 channels, Float64 at 96 kHz, device-resident; 47 GB of input, far larger than L2), and end to end through
the public API.

Cases, alternated within one run (each the median of 5 windows of `steps` steps, CUDA events, after warm-up):
  (a) config 5 as benchmarked: the AM envelope is the enumerated `AffineSin(0.5, 0.5)` leaf;
  (b) the envelope written as the closure `ϕ -> 0.5sin(ϕ) + 0.25sin(2ϕ) + 0.25`: a sub-program of the fused
      tensor-map kernel's input program;
  (c) (b) with SIGOPS_NO_TMAP_LEAVES=1: the per-lane program kernel.
and (d) `sink([...], GPUSink())` of 64 signals of 10 s at 48 kHz of that closure, written with np.sin (traced, run on the
device) and with math.sin (refused by the tracer: evaluated on the host, one Python call per frame), wall time of
the whole call (lowering, host evaluation, copies, kernels).  usage: python tools/gen_closure_step.py [steps]"""
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from signalops import (AffineSin, Amplify, Bandpass, Filt, GPUSink, Hz, Mix, Ramp, Signal, Until, cabi, kHz, ms, s,  # noqa: E402
                       sin, sink)
from signalops.lowering import lower  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
NINST, N, C = 16, 5760000, 64


def cfg5(env):
    am = Amplify(Signal(np.zeros((N, C)), 96 * kHz), Signal(env, ω=5 * Hz)) >> Until(60 * s)
    return am >> Filt(Bandpass, 500 * Hz, 4 * kHz) >> Ramp(10 * ms) >> Mix(Signal(sin, ω=1 * kHz) >> Until(60 * s))


def np_env(p):
    return 0.5 * np.sin(p) + 0.25 * np.sin(2 * p) + 0.25


def math_env(p):
    return 0.5 * math.sin(p) + 0.25 * math.sin(2 * p) + 0.25


def main():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"device: {q[0] if q else 'unknown'}")
    ctx = cabi.Context([0])
    _, copy_gbs = ctx.measure_peaks(0)
    print(f"measured copy peak {copy_gbs:.0f} GB/s; data sheet 7700 GB/s")
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1983)
    x = torch.randn((NINST, C, N), dtype=torch.float64, device="cuda", generator=gen)
    y = torch.empty_like(x)

    def bufs(t):
        arr = (cabi.Buffer * NINST)()
        for i in range(NINST):
            arr[i] = cabi.Buffer(t[i].data_ptr(), N, C, cabi.F64, N)
        return arr

    ins, outs = bufs(x), bufs(y)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cases = {"(a) AffineSin leaf": (AffineSin(0.5, 0.5), False), "(b) closure, fused": (np_env, False),
             "(c) closure, per-lane": (np_env, True)}
    plans = {}
    for name, (env, _) in cases.items():
        plan = lower(cfg5(env))
        assert len(plan.inputs) == 1 and len(plan.outputs) == 1
        plans[name] = cabi.CompiledPlan(ctx, plan.tobytes())
    times = {name: [] for name in cases}
    results = {}

    def run(name, n):
        if cases[name][1]:
            os.environ["SIGOPS_NO_TMAP_LEAVES"] = "1"
        try:
            for _ in range(n):
                plans[name].run_device(NINST, ins, outs, stream=stream.cuda_stream)
        finally:
            os.environ.pop("SIGOPS_NO_TMAP_LEAVES", None)

    for name in cases:
        run(name, 2)
        torch.cuda.synchronize()
        results[name] = y[:, :, ::4099].clone()
    for _ in range(5):
        for name in cases:
            e0.record()
            run(name, steps)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    for name in cases:
        ts = times[name]
        print(f"{name:24s} {float(np.median(ts)):8.3f} ms/step (spread {min(ts):.3f}-{max(ts):.3f})  "
              f"launches {plans[name].launch_count()}")
        plans[name].close()
    b, c = results["(b) closure, fused"], results["(c) closure, per-lane"]
    print(f"(b) against (c): max |diff| / rms = {float(torch.max(torch.abs(b - c)) / torch.sqrt(torch.mean(c ** 2))):.1e}")
    del x, y
    torch.cuda.empty_cache()
    ctx.close()

    g = GPUSink([0])
    for label, env, reps in (("np.sin (traced, device)", np_env, 5), ("math.sin (host evaluation)", math_env, 1)):
        make = lambda: [Signal(env, 48 * kHz, ω=5 * Hz) >> Until(10 * s) for _ in range(64)]   # noqa: E731
        if reps > 1:
            sink(make(), g)          # warm-up (the host-evaluated call takes a minute: timed once, cold)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            sink(make(), g)
            ts.append(time.perf_counter() - t0)
        print(f"(d) sink 64 x 10 s @48 kHz, {label:28s} {1e3 * float(np.median(ts)):9.1f} ms per call ({reps} call(s))")
    g.close()


if __name__ == "__main__":
    main()
