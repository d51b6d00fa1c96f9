"""Cost of the long-bank FIR kernel (csrc/k_fir_long.cuh) on device-resident Float64 batches larger than L2, against
the larger of its two bounds: rows * n_out * taps_per_phase FMAs over the FP64 tensor-core rate that tools/dmma_peak.cu
measures (m8n8k4), and the algorithmic bytes (sigops_plan_algorithmic_bytes) over the copy peak of
sigops_measure_peaks.  Both peaks are measured in the same call as the timings; the device name and power limit are
printed beside them.

Cases: 256 x (480 000 x 2) at 48 kHz -> 8 kHz and -> 12 kHz, 64 x (1 920 000 x 2) at 192 kHz -> 48 kHz, and
`FIRFilter` with 511 and 4097 taps on 256 x (480 000 x 2).  Each is timed with CUDA events as the median of 5 windows
of `steps` steps after 3 warm-up steps.  usage: python tools/fir_long_step.py [steps]"""
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import torch
from scipy import signal as sps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from signalops import Filt, Hz, Signal, ToFramerate, cabi, dspjl, kHz  # noqa: E402
from signalops.lowering import STAGE_FIR, lower  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
CASES = [
    ("48k -> 8k", 256, 480000, lambda z: ToFramerate(Signal(z, 48 * kHz), 8 * kHz)),
    ("48k -> 12k", 256, 480000, lambda z: ToFramerate(Signal(z, 48 * kHz), 12 * kHz)),
    ("192k -> 48k", 64, 1920000, lambda z: ToFramerate(Signal(z, 192 * kHz), 48 * kHz)),
    ("FIRFilter 511", 256, 480000, lambda z: Signal(z, 48 * kHz) >> Filt(dspjl.FIRFilter(sps.firwin(511, 0.2)))),
    ("FIRFilter 4097", 256, 480000, lambda z: Signal(z, 48 * kHz) >> Filt(dspjl.FIRFilter(sps.firwin(4097, 0.2)))),
]
C = 2


def dmma_rate():
    """Best m8n8k4 rate tools/dmma_peak.cu reports, in FMA/s (built into a temporary directory)."""
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "dmma_peak")
        subprocess.check_call(["nvcc", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                               os.path.join(ROOT, "tools", "dmma_peak.cu")])
        out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    return max(float(v) for v in re.findall(r"m8n8k4 ([0-9.]+)", out)) * 1e12


def main():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"device: {q[0] if q else 'unknown'}")
    fma_s = dmma_rate()
    ctx = cabi.Context([0])
    _, copy_gbs = ctx.measure_peaks(0)
    print(f"measured DMMA m8n8k4 peak {fma_s / 1e12:.2f} T FMA/s, copy peak {copy_gbs:.0f} GB/s")
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gen = torch.Generator(device="cuda")
    for name, ninst, n, make in CASES:
        plan = lower(make(np.zeros((n, C))))
        st = next(s for s in plan.stages if s.kind == STAGE_FIR)
        n_out = plan.outputs[0].nframes
        gen.manual_seed(1983)
        x = torch.randn((ninst, C, n), dtype=torch.float64, device="cuda", generator=gen)
        y = torch.empty((ninst, C, n_out), dtype=torch.float64, device="cuda")
        ins = (cabi.Buffer * ninst)(*[cabi.Buffer(x[i].data_ptr(), n, C, cabi.F64, n) for i in range(ninst)])
        outs = (cabi.Buffer * ninst)(*[cabi.Buffer(y[i].data_ptr(), n_out, C, cabi.F64, n_out) for i in range(ninst)])
        cp = cabi.CompiledPlan(ctx, plan.tobytes())
        for _ in range(3):
            cp.run_device(ninst, ins, outs, stream=stream.cuda_stream)
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            e0.record()
            for _ in range(steps):
                cp.run_device(ninst, ins, outs, stream=stream.cuda_stream)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / steps)
        t = float(np.median(ts))
        rows = ninst * C
        fmas = rows * n_out * st.taps_per_phase
        alg = cp.algorithmic_bytes() * ninst
        t_fma, t_mem = fmas / fma_s * 1e3, alg / (copy_gbs * 1e9) * 1e3
        bound = "DMMA" if t_fma >= t_mem else "copy"
        print(f"{name:15s} taps/phase {st.taps_per_phase:5d}  {t:8.3f} ms/step (spread {min(ts):.3f}-{max(ts):.3f})  "
              f"{rows * n_out / t / 1e3:8.0f} Msamples/s out  bound {bound} {max(t_fma, t_mem):7.3f} ms "
              f"(DMMA {t_fma:.3f}, copy {t_mem:.3f}) = {100 * max(t_fma, t_mem) / t:5.1f}% of it")
        cp.close()
        del x, y
    ctx.close()


if __name__ == "__main__":
    main()
