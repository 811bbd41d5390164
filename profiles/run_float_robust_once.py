"""Robust endpoint detection on float32 samples against int16 on bench.py's batch (4096 ragged utterances, the same synth seeds;
float = int16 * 2^-15): call time of each (CUDA events, alternating), per-kernel times from dspfe_timing_*, host-form call time of
each, and lr equality between the two (exact under the power-of-two scaling).  Records the GPU's name and power limit.  Prints
one JSON line; --out PATH also writes it to PATH."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "dsp-speech-recognition_b200"))
import dspfe  # noqa: E402
from dspfe import synth  # noqa: E402


def main(steps=20, warmup=3, out=None):
    dev = torch.device("cuda:0")
    lengths = synth.ragged_lengths(4096, seed=2024)
    pcm16, off = synth.synth_batch_torch(lengths, seed0=555, device=dev)
    off_h = off.numpy().astype(np.int64)
    off_d = off.to(dev)
    pcmf = (pcm16.float() * 2.0 ** -15).contiguous()
    ep = dspfe.EndpointPlan()
    runs = {"int16": lambda: ep.detect_robust(pcm16, off_d), "float32": lambda: ep.detect_robust_f32(pcmf, off_d)}
    for _ in range(warmup):
        for f in runs.values():
            f()
    ms = {k: [] for k in runs}
    for _ in range(steps):
        for k, f in runs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); f(); b.record(); torch.cuda.synchronize()
            ms[k].append(a.elapsed_time(b))
    kernels = {}
    for k, f in runs.items():
        dspfe.timing_begin(); f(); marks = dspfe.timing_end()
        agg = {}
        for n, t in marks:
            agg[n] = agg.get(n, 0.0) + t
        kernels[k] = {n: round(t, 4) for n, t in sorted(agg.items(), key=lambda x: -x[1])}
    lr16, lrf = runs["int16"](), runs["float32"]()
    # host forms
    h16 = pcm16.cpu().numpy()
    hf = pcmf.cpu().numpy()
    eh = dspfe.EndpointPlan()
    host = {"int16": lambda: eh.detect_robust_host(h16, off_h), "float32": lambda: eh.detect_robust_host_f32(hf, off_h)}
    host_lr = {k: f() for k, f in host.items()}
    host_ms = {k: [] for k in host}
    for _ in range(5):
        for k, f in host.items():
            t0 = time.perf_counter(); f(); host_ms[k].append((time.perf_counter() - t0) * 1e3)
    ident = dict(lr=bool(torch.equal(lr16, lrf)), host_lr=bool(np.array_equal(host_lr["int16"], host_lr["float32"])),
                 host_equals_device=bool(np.array_equal(host_lr["float32"], lrf.cpu().numpy())))
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    med = lambda v: float(np.median(v))
    res = dict(gpu=gpu[0] if gpu else "unknown", utterances=len(lengths), samples=int(pcm16.numel()), steps=steps,
               call_ms={k: dict(median=round(med(v), 4), min=round(min(v), 4), max=round(max(v), 4)) for k, v in ms.items()},
               host_call_ms={k: dict(median=round(med(v), 3), min=round(min(v), 3)) for k, v in host_ms.items()},
               kernels_ms=kernels, lr_equal=ident)
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
