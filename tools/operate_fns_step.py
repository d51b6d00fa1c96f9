"""Cost of traced OperateOn functions on the device, at BASELINE config 2's shape (256 signals x 480 000 frames x 2
channels, Float64, device-resident), against the HBM roofline of the algorithmic bytes.

Chains: the plain config 2 chain (Lowpass order 8, then a gain), `OperateOn(abs)` before its filter, `OperateOn(tanh)`
after it; and a bare elementwise pass (`k_map`) of `tanh` against one of `Amplify` on the same data.  Each is timed as
the median of 5 windows of `steps` graph-replayed steps (CUDA events) after warm-up; the 2 GB inputs do not fit L2.
The roofline is the algorithmic bytes (sigops_plan_algorithmic_bytes) over the measured copy peak of the device and
over the data-sheet 7.7 TB/s.  usage: python tools/operate_fns_step.py [steps]"""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from signalops import Amplify, Filt, Lowpass, Operate, OperateOn, Signal, cabi, dB, kHz  # noqa: E402
from signalops.lowering import lower  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
NINST, N, C = 256, 480000, 2
Z = np.zeros((N, C))
CHAINS = {
    "cfg2": lambda: Signal(Z, 48 * kHz) >> Filt(Lowpass, 4 * kHz, order=8) >> Amplify(-20 * dB),
    "abs >> cfg2": lambda: OperateOn(abs, Signal(Z, 48 * kHz)) >> Filt(Lowpass, 4 * kHz, order=8) >> Amplify(-20 * dB),
    "cfg2 >> tanh": lambda: Signal(Z, 48 * kHz) >> Filt(Lowpass, 4 * kHz, order=8) >> Amplify(-20 * dB) >> Operate(np.tanh),
    "k_map tanh": lambda: OperateOn(np.tanh, Signal(Z, 48 * kHz)),
    "k_map Amplify": lambda: Amplify(Signal(Z, 48 * kHz), -20 * dB),
}


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
    for name, make in CHAINS.items():
        plan = lower(make())
        assert len(plan.inputs) == 1 and len(plan.outputs) == 1
        cp = cabi.CompiledPlan(ctx, plan.tobytes())
        for _ in range(3):
            cp.run_device(NINST, ins, outs, stream=stream.cuda_stream)
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            e0.record()
            for _ in range(steps):
                cp.run_device(NINST, ins, outs, stream=stream.cuda_stream)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / steps)
        t = float(np.median(ts))
        alg = cp.algorithmic_bytes() * NINST
        print(f"{name:14s} {t:7.3f} ms/step (spread {min(ts):.3f}-{max(ts):.3f})  launches {cp.launch_count()}  "
              f"alg {alg / 1e9:.2f} GB  {alg / t / 1e6:6.0f} GB/s = {100 * alg / t / 1e6 / copy_gbs:5.1f}% of measured copy peak, "
              f"{100 * alg / t / 1e6 / 7700:5.1f}% of 7.7 TB/s")
        cp.close()
    ctx.close()


if __name__ == "__main__":
    main()
