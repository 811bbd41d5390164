"""Cepstrum pitch at frame lengths 300, 400 and 512 samples on bench.py's batch (4096 ragged int16 utterances, the same synth
seeds): call time of each (CUDA events, alternating), per-kernel times from dspfe_timing_*, and the frame count of each.  512
samples run the 512-point chain (pitch_frame_kernel<0>), the others the Bluestein chain (pitch_cep_bluestein_kernel).  Records the
GPU's name and power limit.  Prints one JSON line; --out PATH also writes it to PATH."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "dsp-speech-recognition_b200"))
import dspfe  # noqa: E402
from dspfe import synth  # noqa: E402

FRAME_LENS = (300, 400, 512)


def main(steps=20, warmup=3, out=None):
    dev = torch.device("cuda:0")
    lengths = synth.ragged_lengths(4096, seed=2024)
    pcm16, off = synth.synth_batch_torch(lengths, seed0=555, device=dev)
    off_d = off.to(dev)
    plans = {N: dspfe.PitchPlan(method=0, frame_len=N) for N in FRAME_LENS}
    runs = {N: (lambda pl=pl: pl.detect(pcm16, off_d)) for N, pl in plans.items()}
    for _ in range(warmup):
        for f in runs.values():
            f()
    ms = {N: [] for N in runs}
    for _ in range(steps):
        for N, f in runs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); f(); b.record(); torch.cuda.synchronize()
            ms[N].append(a.elapsed_time(b))
    kernels, frames = {}, {}
    for N, f in runs.items():
        dspfe.timing_begin(); o = f(); marks = dspfe.timing_end()
        agg = {}
        for n, t in marks:
            agg[n] = agg.get(n, 0.0) + t
        kernels[N] = {n: round(t, 4) for n, t in sorted(agg.items(), key=lambda x: -x[1])}
        frames[N] = int(o["frame_off"][-1])
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    med = lambda v: float(np.median(v))
    res = dict(gpu=gpu[0] if gpu else "unknown", utterances=len(lengths), samples=int(pcm16.numel()), steps=steps,
               frames={str(N): v for N, v in frames.items()},
               call_ms={str(N): dict(median=round(med(v), 4), min=round(min(v), 4), max=round(max(v), 4)) for N, v in ms.items()},
               kernels_ms={str(N): v for N, v in kernels.items()})
    line = json.dumps(res)
    print(line)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    main(a.steps, a.warmup, a.out)
