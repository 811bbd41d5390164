"""The general long-frame MFCC kernel (K1L, mfcc_long_kernel) at transform sizes other than the tiled kernels' on a ragged batch
of 4096 int16 utterances: nfft = 1024 (25 ms frames at 16 kHz) and nfft = 2048 (30 ms frames at 44.1 kHz).  Call time of each
(CUDA events, alternating), per-kernel times from dspfe_timing_*, and the GPU's name and power limit.  Prints one JSON line;
--out PATH also writes it to PATH."""
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

CONFIGS = {
    "nfft1024_16k": (16000, dict(frame_len=400, frame_step=160, nfft=1024, window=np.hamming(400), delta_n=2)),
    "nfft2048_44k": (44100, dict(frame_len=1323, frame_step=441, nfft=2048, window=np.hamming(1323), delta_n=2, samplerate=44100)),
}


def main(steps=20, warmup=3, out=None):
    dev = torch.device("cuda:0")
    runs = {}
    for name, (rate, kw) in CONFIGS.items():
        lengths = synth.ragged_lengths(4096, seed=2024) * rate // 16000
        pcm, off = synth.synth_batch_torch(lengths, seed0=555, sr=rate, device=dev)
        plan = dspfe.MfccPlan(**kw)
        runs[name] = (lambda plan=plan, pcm=pcm, off=off.to(dev): plan.mfcc_delta(pcm, off))
    for _ in range(warmup):
        for f in runs.values():
            f()
    ms = {n: [] for n in runs}
    for _ in range(steps):
        for n, f in runs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); f(); b.record(); torch.cuda.synchronize()
            ms[n].append(a.elapsed_time(b))
    kernels = {}
    for n, f in runs.items():
        dspfe.timing_begin(); f(); marks = dspfe.timing_end()
        agg = {}
        for k, t in marks:
            agg[k] = agg.get(k, 0.0) + t
        kernels[n] = {k: round(t, 4) for k, t in sorted(agg.items(), key=lambda x: -x[1])}
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    med = lambda v: float(np.median(v))
    res = dict(gpu=gpu[0] if gpu else "unknown", utterances=4096, steps=steps,
               call_ms={n: dict(median=round(med(v), 4), min=round(min(v), 4), max=round(max(v), 4)) for n, v in ms.items()},
               kernels_ms=kernels)
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
