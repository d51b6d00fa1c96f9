"""A corpus job as one ragged batch against the alternatives.  1024 stereo clips at 44.1 kHz with seeded lengths uniform in
1-30 s, through `ToFramerate(48 kHz) >> Filt(Lowpass, 8 kHz) >> Normpower >> Amplify(-20 dB)`:
  (a) one ragged `sink(clips, GPUSink())` call,
  (b) one `sink(clip, GPUSink())` call per clip, on the first `--loop` clips (a new plan for every distinct length),
  (c) one equal-length batch of 1024 clips of the mean length (the same useful samples as (a)).
(a) and (c) alternate `--reps` times in the same run; each reports wall time, stats.gpu_ms and useful output Msamples/s.
Then one more ragged call with SIGOPS_DEBUG set gives the frames every wave computed against the frames its clips
need.  The clips are column slices of one pageable pool (the caller's arrays, as a user's would be).  The device name
and power limit are printed first.  usage: python tools/ragged_step.py [--clips 1024] [--loop 128] [--reps 2]"""
import argparse
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from signalops import Amplify, Filt, GPUSink, Lowpass, Normpower, Signal, ToFramerate, dB, kHz, sink  # noqa: E402


def chain(x):
    return Signal(x, 44.1 * kHz) >> ToFramerate(48 * kHz) >> Filt(Lowpass, 8 * kHz) >> Normpower >> Amplify(-20 * dB)


def timed(gpu, sigs):
    t0 = time.perf_counter()
    outs = sink(sigs, gpu) if isinstance(sigs, list) else [sink(sigs, gpu)]
    wall = time.perf_counter() - t0
    useful = sum(o[0].size for o in outs)
    return wall, useful, outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--loop", type=int, default=128)
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"device: {q[0] if q else 'unknown'}", flush=True)
    fs = 44100
    lens = np.random.default_rng(2024).integers(1 * fs, 30 * fs + 1, a.clips)
    total = int(lens.sum())
    pool = np.empty((total, 2), order="F")
    rng = np.random.default_rng(7)
    for c in range(2):
        for lo in range(0, total, 1 << 26):
            pool[lo:lo + (1 << 26), c] = rng.standard_normal(min(1 << 26, total - lo))
    starts = np.concatenate([[0], np.cumsum(lens)[:-1]])
    ragged = [chain(pool[s:s + n]) for s, n in zip(starts, lens)]
    mean = total // a.clips
    equal = [chain(pool[k * mean:(k + 1) * mean]) for k in range(a.clips)]
    print(f"corpus: {a.clips} stereo clips, {lens.min() / fs:.2f}-{lens.max() / fs:.2f} s, {total / fs / 3600:.2f} h in; "
          f"equal-length batch of {mean} frames each", flush=True)
    gpu = GPUSink()
    for name, sigs in (("warm-up ragged", ragged), ("warm-up equal", equal)):
        wall, useful, outs = timed(gpu, sigs)
        del outs
        print(f"{name}: {wall * 1e3:.0f} ms", flush=True)
    res = {"a": [], "c": []}
    for r in range(a.reps):
        for key, sigs in (("a", ragged), ("c", equal)):
            wall, useful, outs = timed(gpu, sigs)
            del outs
            st = gpu.last_stats
            res[key].append((wall, st["gpu_ms"], useful))
            print(f"rep {r} ({key}) {'ragged call' if key == 'a' else 'equal-length batch'}: wall {wall * 1e3:.0f} ms, "
                  f"gpu_ms {st['gpu_ms']:.1f}, h2d_ms {st['h2d_ms']:.1f}, d2h_ms {st['d2h_ms']:.1f}, launches {st['launches']}, "
                  f"useful {useful / wall / 1e6:.0f} Msamples/s", flush=True)
    # (b) the per-clip loop on a subset
    wall_b, useful_b, gpu_b = 0.0, 0, 0.0
    loop = GPUSink()
    for x in ragged[:a.loop]:
        wall, useful, outs = timed(loop, x)
        wall_b += wall
        useful_b += useful
        gpu_b += loop.last_stats["gpu_ms"]
        del outs
    loop.close()
    print(f"(b) per-clip loop over {a.loop} clips: wall {wall_b * 1e3:.0f} ms, gpu_ms {gpu_b:.1f}, "
          f"useful {useful_b / wall_b / 1e6:.0f} Msamples/s", flush=True)
    for key, label in (("a", "(a) ragged call"), ("c", "(c) equal-length batch")):
        w = min(v[0] for v in res[key])
        g = min(v[1] for v in res[key])
        print(f"{label}: best wall {w * 1e3:.0f} ms, best gpu_ms {g:.1f}, useful {res[key][0][2] / w / 1e6:.0f} Msamples/s")
    # computed / useful frames per ragged wave, from the runtime's own debug lines (a fresh sink plans again)
    dbg = GPUSink()
    os.environ["SIGOPS_DEBUG"] = "1"
    with tempfile.TemporaryFile(mode="w+") as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            outs = sink(ragged, dbg)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["SIGOPS_DEBUG"]
        del outs
        f.seek(0)
        waves = [ln.strip() for ln in f if "ragged wave" in ln]
    dbg.close()
    comp = use = 0
    for ln in waves:
        m = re.search(r"computed=(\d+) useful=(\d+)", ln)
        comp += int(m.group(1))
        use += int(m.group(2))
        print(ln)
    print(f"frames computed / useful over {len(waves)} waves: {comp / max(use, 1):.4f}")
    gpu.close()


if __name__ == "__main__":
    main()
