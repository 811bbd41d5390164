#!/usr/bin/env python
"""bench.py -- audio-seconds/second of the PCM -> classifier-features front-end on B200 (BASELINE.json `metric`:
"audio-sec/sec of MFCC+delta+pitch+endpoint at 1/2/4/8 B200; % of HBM roofline").

Workload (default, `--workload frontend`): 4096 ragged synthetic utterances per GPU (0.5-5 s, 16 kHz int16, offset array, no
padding), cut from ONE global list by the length-balanced LPT partition (dspfe/shard.py).  One "step" = one pass of the whole
front-end over the rank's shard, chained per utterance as the reference's callers do it:
    endpoints (model.py:52-53)  ->  MFCC + delta + delta on sig[l:r] (model.py:74-77)
    ->  cepstrum pitch + pitch_feature on preemphasis(sig)[l:r] (pitch_model.py:38-41)  ->  autocorrelation pitch on sig[l:r] (model.py:92)

  value         device-resident throughput (PCM and features in HBM), CUDA events around K steps, max over ranks
  paths         per path (endpoint / mfcc / pitch_cep / pitch_acr): device ms from per-kernel CUDA events on the launching
                stream (dspfe_timing_*), algorithmic bytes, fraction of the measured HBM peak, nominal FP32-pipe fraction
  roofline      the dominant kernel of the step: algorithmic bytes per launch / its event-timed duration vs MEASURED_PEAKS.json
  e2e           the same step through the host-buffer call (dspfe_frontend_host): pinned host PCM -> H2D -> kernels -> D2H of
                every output, slab-pipelined on three streams; host wall clock, max over ranks
  cpu_baseline  the reference front-end on the host cores for a bounded sample of the same utterances (live reference from
                baseline/_ref when installed, else the oracle port)
  pitch_mismatch  pitch-peak lags of the sample against the float64 oracle: frames, differing, near_tie (explained by a
                float64 near-tie, oracle.lag_is_near_tie_*), hard (unexplained; must be 0)

`--impl reference` times the reference front-end on all host cores instead (same config, bounded sample per step).
`--workload mfcc` is the MFCC-only line of BASELINE configs[1] (4096 x 2 s, fused K1 kernel).
`--dump-outputs DIR` writes what the last timed step returned as DIR/<name>.npy (DIR/rank<r>/ when N > 1), at most 64 MB over
all ranks; the inputs are seeded, so two builds run with the same arguments can be compared output for output.  It covers the
GPU workloads only: the reference arm's pool workers hand back no outputs, and returning them would change what it times.
Launch: python bench.py [--gpus N --steps K --warmup W]; for N > 1 via torch.distributed.run (one rank per GPU).
"""
import argparse
import atexit
import json
import os
import signal
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "dsp-speech-recognition_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
os.environ.setdefault("OMP_NUM_THREADS", "1")

# stdout carries the one JSON line and nothing else: everything that writes to file descriptor 1 from here on (NCCL prints its
# version banner there) lands on stderr; emit() writes the line to the original stdout.
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj):
    _JSON_OUT.write(json.dumps(obj) + "\n")
    _JSON_OUT.flush()


import numpy as np  # noqa: E402

SR = 16000
UTT_PER_GPU = 4096
DELTA_N = 2
UNIT = "audio-s/s"
METRIC = "audio-sec/sec of MFCC+delta+pitch+endpoint (full front-end), ragged 0.5-5 s utterances, per-GPU LPT shards"
WORKLOAD = ("configs[3]+[2] on the configs[4] layout: 4096 ragged U{8000..80000}-sample utterances per GPU @16 kHz int16 (offset array), "
            "LPT-sharded from one global list; per utterance endpoint -> MFCC+delta+delta-delta(N=2) on sig[l:r] -> cepstrum pitch + "
            "pitch_feature on preemphasis(sig)[l:r] -> autocorrelation pitch (300-sample frames) on sig[l:r]")
FP32_PEAK = 148 * 128 * 2 * 1.965e9          # FFMA lanes x 2 flop x max SM clock (nominal, for the FP32-pipe fractions)
FFT512_FLOP = 5 * 512 * 9                    # nominal 5 N log2 N of one complex 512-point transform


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_BYTES = 64 * 10**6            # all ranks together


def dump_outputs(d, per_utt, ragged, budget):
    """Writes the outputs of one call as d/<name>.npy: float32 stays float32, every other type becomes float64 (exact for
    the int32 / int64 outputs).  `per_utt` maps a name to an output with one row per utterance; `ragged` maps the name of a
    frame-offset output [U+1] to (those offsets as a NumPy array, {name: per-frame rows}).  When all of it does not fit in
    `budget` bytes, a fixed seeded sample of utterances is written instead, the same utterances in every array, and each
    offset array is rebuilt to index the rows written (what the call returns for those utterances alone).
    d/utterances.npy lists the utterances written, in order."""
    import torch
    os.makedirs(d, exist_ok=True)
    width = lambda t: int(np.prod(t.shape[1:])) * (4 if t.dtype == torch.float32 else 8)
    n_utt = len(next(iter(ragged.values()))[0]) - 1
    files = 1 + len(per_utt) + sum(1 + len(rows) for _, rows in ragged.values())
    fixed = 1024 * files + 8 * len(ragged)                    # .npy headers, the leading zero of each offset array
    cost = 8 + sum(width(t) for t in per_utt.values()) + sum(8 + np.diff(fo) * sum(width(r) for r in rows.values())
                                                             for fo, rows in ragged.values())
    keep = np.arange(n_utt)
    if fixed + int(np.sum(cost)) > budget:
        order = np.random.default_rng(0).permutation(n_utt)
        keep = np.sort(order[: int(np.searchsorted(np.cumsum(cost[order]), budget - fixed, side="right"))])

    written = []

    def save(name, a):
        path = os.path.join(d, name + ".npy")
        np.save(path, np.ascontiguousarray(a, dtype=np.float32 if a.dtype == np.float32 else np.float64))
        written.append(os.path.getsize(path))

    save("utterances", keep)
    sel = torch.from_numpy(keep)
    for k, t in per_utt.items():
        save(k, t[sel.to(t.device)].cpu().numpy())
    for k, (fo, rows) in ragged.items():
        n = np.diff(fo)[keep]
        off = np.concatenate([[0], np.cumsum(n)])
        save(k, off)
        idx = torch.from_numpy(np.arange(off[-1], dtype=np.int64) + np.repeat(fo[keep] - off[:-1], n))
        for name, r in rows.items():
            save(name, r[idx.to(r.device)].cpu().numpy())
    assert sum(written) <= budget, written


def dump(args, rank, world, per_utt, ragged):
    """--dump-outputs: rank r of N > 1 writes to DIR/rank<r>/, each with a 1/N share of DUMP_BYTES."""
    d = args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}")
    dump_outputs(d, per_utt, ragged, DUMP_BYTES // world)


def recorded_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from this round's `ncu --set full` capture of this
    very workload (profiles/r2_traffic.json, written by profiles/summarize_ncu.py), or None when there is no capture."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        with open(path) as f:
            t = json.load(f)
        return t.get(kernel), t.get("_source")
    except (OSError, ValueError):
        return None, None


# ----------------------------------------------------------------------------- CPU legs
# Worker processes are forked before CUDA is touched.  kind "reference" = the unmodified reference package imported from
# baseline/_ref (oracle/install_reference.py), kind "port" = oracle/ref_features.py.
_W = {}


def reference_available():
    return os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "features")) or os.path.isdir("/root/reference/features")


def _w_setup(kind):
    if _W.get("kind") == kind:
        return
    if kind == "reference":
        from oracle import _live_reference as live
        _W["ref"] = live.load()
        _W["quiet"] = live.quiet
    from oracle import ref_features as O
    _W["O"] = O
    _W["kind"] = kind


def _frontend_one(kind, x):
    """The reference's call chain on one int16 utterance; returns audio seconds processed."""
    if kind == "reference":
        ref = _W["ref"]
        with _W["quiet"]():
            l, r = ref.basic_endpoint_detection(x, SR)
            seg = x[l:r]
            m = ref.mfcc(seg, SR)
            d1 = ref.delta(m, DELTA_N); ref.delta(d1, DELTA_N)
            pre = ref.preemphasis(x, coeff=0.97)[l:r]
            try:
                ref.pitch_feature(pre, SR)
            except Exception:      # a half without three usable frames: polyfit raises in the reference
                pass
            ref.pitch_detect_sr(seg, SR, winlen=0.03, step=0.01)
    else:
        O = _W["O"]
        l, r = O.basic_endpoint_detection(x, SR)
        seg = x[l:r]
        O.mfcc_delta39(seg, DELTA_N)
        pre = O.preemphasis(x, 0.97)[l:r]
        try:
            O.pitch_feature(pre, SR)
        except Exception:
            pass
        O.pitch_detect_sr(seg, SR, winlen=0.03, step=0.01)
    return len(x) / SR


def _w_run(job):
    kind, xs = job
    _w_setup(kind)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return sum(_frontend_one(kind, x) for x in xs)


def _w_parity(job):
    """Oracle check of one utterance against what the GPU produced for it (checker only)."""
    import warnings
    _w_setup("port")
    O = _W["O"]
    x, g = job
    res = dict(ep_bad=0, mfcc_err=0.0, cep_frames=0, cep_diff=0, cep_near=0, acr_frames=0, acr_diff=0, acr_near=0, hz_bad=0,
               feat_checked=0, feat_err=0.0, shape_bad=0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        l, r = O.basic_endpoint_detection(x, SR)
        if (l, r) != (int(g["lr"][0]), int(g["lr"][1])):
            res["ep_bad"] = 1
            return res
        seg = x[l:r]
        ref = O.mfcc_delta39(seg, DELTA_N)
        if ref.shape != g["mfcc"].shape:
            res["shape_bad"] += 1
        else:
            res["mfcc_err"] = float(np.max(np.abs(g["mfcc"] - ref) / (1 + np.abs(ref)))) if ref.size else 0.0
        pre = O.preemphasis(x, 0.97)[l:r]
        rows = O.pitch_rows_cep(pre, SR)
        lag = np.array([20 + int(np.argmax(O.peak_score(c))) for c in rows], dtype=np.int64)
        if len(lag) != len(g["cep_lag"]):
            res["shape_bad"] += 1
        else:
            bad = np.nonzero(lag != g["cep_lag"])[0]
            res["cep_frames"], res["cep_diff"] = len(lag), len(bad)
            res["cep_near"] = int(sum(O.lag_is_near_tie_cep(rows[i], g["cep_lag"][i]) for i in bad))
            res["hz_bad"] += int(np.sum(np.asarray(O.robust_pitch_from_lags(g["cep_lag"])) != g["cep_pitch"]))
            if len(bad) == 0:
                try:
                    want = np.asarray(O.pitch_feature(pre, SR), dtype=np.float64)
                except Exception:
                    want = None
                if want is not None and np.all(np.isfinite(want)) and np.all(np.isfinite(g["feat"])):
                    res["feat_checked"] = 1
                    res["feat_err"] = float(np.max(np.abs(g["feat"] - want) / np.maximum(np.abs(want), 1e-9)))
        srows, _ = O.pitch_scores_sr(seg, SR, winlen=0.03, step=0.01)
        srows = np.asarray(srows)
        slag = 20 + np.argmax(srows, axis=1) if len(srows) else np.zeros(0, dtype=np.int64)
        if len(slag) != len(g["acr_lag"]):
            res["shape_bad"] += 1
        else:
            bad = np.nonzero(slag != g["acr_lag"])[0]
            res["acr_frames"], res["acr_diff"] = len(slag), len(bad)
            res["acr_near"] = int(sum(O.lag_is_near_tie_sr(srows[i], g["acr_lag"][i]) for i in bad))
            res["hz_bad"] += int(np.sum(np.asarray(O.robust_pitch_from_lags(g["acr_lag"])) != g["acr_pitch"]))
    return res


def lpt_chunks(xs, n):
    """Deals the utterances to n workers, longest first onto the least loaded (the pool maps one chunk per worker)."""
    order = sorted(range(len(xs)), key=lambda i: -len(xs[i]))
    loads, chunks = [0] * n, [[] for _ in range(n)]
    for i in order:
        k = loads.index(min(loads))
        chunks[k].append(xs[i]); loads[k] += len(xs[i])
    return [c for c in chunks if c]


def make_pool(cores):
    import multiprocessing as mp
    return mp.get_context("fork").Pool(cores)


def cpu_front_end(pool, kind, xs, cores, repeats=1):
    """Times the reference front-end over `xs` on the pool (one warm call per worker first: imports, FFT plan caches)."""
    pool.map(_w_run, [(kind, [xs[0][:8000]])] * cores, chunksize=1)
    jobs = [(kind, c) for c in lpt_chunks(xs, cores)]
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        audio = sum(pool.map(_w_run, jobs, chunksize=1))
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return audio / best, best, audio


def run_reference(args, rank):
    if rank != 0:
        return
    from dspfe import synth
    cores = len(os.sched_getaffinity(0))
    kind = "reference" if reference_available() else "port"
    lengths = synth.ragged_lengths(UTT_PER_GPU * max(args.gpus, 1), seed=2024)
    n = 8 * cores                                   # bounded sample: about 3 s of wall time per step on the box's cores
    xs = [synth.synth_utterance(555 + i, int(lengths[i])) for i in range(n)]
    pool = make_pool(cores)
    pool.map(_w_run, [(kind, [xs[0][:8000]])] * cores, chunksize=1)     # imports, caches
    jobs = [(kind, c) for c in lpt_chunks(xs, cores)]
    audio = sum(len(x) for x in xs) / SR
    dts = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        pool.map(_w_run, jobs, chunksize=1)
        if i >= args.warmup:
            dts.append(time.perf_counter() - t0)
    pool.close()
    dt = float(np.mean(dts))
    value = audio / dt
    sample = (f"{n} of the workload's ragged utterances per step ({audio:.0f} audio-s), "
              + ("the unmodified reference features package (baseline/_ref)" if kind == "reference" else "oracle port (NumPy float64)")
              + f" in {cores} processes, one persistent pool")
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD + " -- bounded sample per step", "sample_utterances": n},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.f, stderr=subprocess.DEVNULL)
            atexit.register(self.p.kill)         # the sampler must not outlive bench.py when a step fails before stop()
        except OSError:
            self.p = None

    def lines(self):
        try:
            return sum(1 for _ in open(self.f.name))
        except OSError:
            return 0

    def wait_first(self, timeout=5.0):
        t0 = time.perf_counter()
        while self.p is not None and self.lines() == 0 and time.perf_counter() - t0 < timeout:
            time.sleep(0.01)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.f.name)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def sample_clocks_under(sampler, step, torch):
    """The timed region lasts milliseconds: keep the very same step running until nvidia-smi has sampled it under load."""
    n0, t0 = sampler.lines(), time.perf_counter()
    while sampler.lines() < n0 + 8 and time.perf_counter() - t0 < 3.0:
        for _ in range(3):
            step()
        torch.cuda.synchronize()
    clocks = sampler.stop()
    clocks["note"] = "sampled every 20 ms from before the timed region until 8 samples had been taken with the same step running"
    return clocks


# ----------------------------------------------------------------------------- GPU arm: full front-end
PATH_OF = {"fe_rel_offsets_kernel": "glue", "fe_finish_kernel": "glue", "ep_prep_kernel": "endpoint", "ep_block_kernel": "endpoint",
           "ep_frame_kernel": "endpoint", "ep_decide_kernel": "endpoint", "prep_kernel": "mfcc", "mfcc_delta_kernel": "mfcc"}


def split_paths(marks):
    """[(kernel, ms)] of one step in launch order -> {path: {kernel: ms}}; the second pitch chain is the autocorrelation one."""
    paths = {"endpoint": {}, "mfcc": {}, "pitch_cep": {}, "pitch_acr": {}, "glue": {}}
    chain = "pitch_cep"
    for name, ms in marks:
        if name.startswith("pitch_") and name == "pitch_prep_kernel" and paths["pitch_cep"]:
            chain = "pitch_acr"
        path = PATH_OF.get(name, chain if name.startswith("pitch_") else "glue")
        paths[path][name] = paths[path].get(name, 0.0) + ms
    return paths


def run_frontend(args, rank, world, local_rank):
    cores = len(os.sched_getaffinity(0))
    pool = make_pool(cores) if rank == 0 else None          # forked before CUDA is initialised in this process
    import torch
    import torch.distributed as dist
    import dspfe
    from dspfe import shard, synth

    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the product path has no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    U = args.utterances
    all_len = synth.ragged_lengths(U * world, seed=2024)
    parts = shard.lpt_partition(all_len, world)
    idx = parts[rank]
    lengths = all_len[idx]
    pcm, off = synth.synth_batch_torch(lengths, seed0=555 + 7919 * rank, device=dev)
    off_np = off.numpy()
    off_d = off.to(dev)
    n_utt, total = len(lengths), int(pcm.numel())
    fe = dspfe.FrontendPlan(delta_n=DELTA_N)
    out = fe.alloc(total, n_utt, device=dev)
    tot = [None]

    def step():
        tot[0] = fe.run(pcm, off_d, off_np, out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.wait_first()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_launch0 = dspfe.launch_count()
    barrier()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = dspfe.launch_count() - n_launch0
    rows, fcep, facr = tot[0]
    # the last timed step's outputs, copied on the device now and written after the clock sampling (later steps reuse `out`)
    last = {k: v.clone() for k, v in out.items()} if args.dump_outputs else None

    # per-kernel device times of the same step: CUDA events on the launching stream around every kernel (3 steps, mean)
    acc = {}
    for _ in range(3):
        dspfe.timing_begin()
        step()
        for path, ks in split_paths(dspfe.timing_end()).items():
            for k, v in ks.items():
                acc.setdefault(path, {}).setdefault(k, []).append(v)
    kern = {path: {k: float(np.mean(v)) for k, v in ks.items()} for path, ks in acc.items()}
    clocks = sample_clocks_under(sampler, step, torch) if sampler else None
    if last:
        fo = {k: last[k].cpu().numpy() for k in ("mfcc_frame_off", "cep_frame_off", "acr_frame_off")}
        dump(args, rank, world, {"lr": last["lr"], "cep_feat": last["cep_feat"]},
             {"mfcc_frame_off": (fo["mfcc_frame_off"], {"mfcc": last["mfcc"][:rows]}),
              "cep_frame_off": (fo["cep_frame_off"], {"cep_pitch": last["cep_pitch"][:fcep], "cep_lag": last["cep_lag"][:fcep]}),
              "acr_frame_off": (fo["acr_frame_off"], {"acr_pitch": last["acr_pitch"][:facr], "acr_lag": last["acr_lag"][:facr]})})

    # end to end through the host-buffer call: pinned host PCM in, pinned host outputs back, every step
    h_pcm = torch.empty(total, dtype=torch.int16).pin_memory()
    h_pcm.copy_(pcm)
    h_out = fe.alloc(total, n_utt, device=None, pinned=True)
    h_pcm_np = h_pcm.numpy()
    for _ in range(2):
        htot = fe.run_host(h_pcm_np, off_np, h_out)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 10))
    for _ in range(e2e_steps):
        fe.run_host(h_pcm_np, off_np, h_out)
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    e2e_ok = bool(htot == (rows, fcep, facr)
                  and torch.equal(h_out["lr"], out["lr"].cpu())
                  and torch.equal(h_out["mfcc"][:rows], out["mfcc"][:rows].cpu())
                  and torch.equal(h_out["cep_lag"][:fcep], out["cep_lag"][:fcep].cpu())
                  and torch.equal(h_out["acr_lag"][:facr], out["acr_lag"][:facr].cpu()))
    d2h = int(n_utt * 8 + rows * 156 + 3 * (n_utt + 1) * 8 + fcep * 12 + facr * 12 + n_utt * 40)
    h2d = int(total * 2 + (n_utt + 1) * 8)

    audio_s = float(lengths.sum()) / SR
    t = torch.tensor([ms_total, e2e_s], dtype=torch.float64, device=dev)
    s = torch.tensor([audio_s, float(h2d), float(d2h), float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
    ms_total, e2e_s = [float(v) for v in t.cpu()]
    audio_all, h2d_all, d2h_all, launches_all = [float(v) for v in s.cpu()]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = ms_total / args.steps
    peak, peak_src = peaks()
    # ---- per-path report (rank 0's shard; SURVEY section 8d byte counts, pitch outputs as built: float64 Hz + int32 lag)
    S = float(lengths.sum())
    fr16 = S / 160.0
    alg = {"endpoint": 2 * S + 8 * n_utt, "mfcc": 2 * S + 156.0 * rows, "pitch_cep": 2 * S + 12.0 * fcep + 40.0 * n_utt,
           "pitch_acr": 2 * S + 12.0 * facr}
    flop = {"pitch_cep": 5 * FFT512_FLOP * fcep, "pitch_acr": 6 * FFT512_FLOP * facr, "mfcc": 14e3 * rows}
    paths = {}
    for path in ("endpoint", "mfcc", "pitch_cep", "pitch_acr"):
        ms = sum(kern.get(path, {}).values())
        e = {"device_ms": ms, "alg_bytes": alg[path], "hbm_frac": alg[path] / (ms * 1e-3) / 1e9 / peak if ms else None,
             "kernels_ms": kern.get(path, {})}
        if path in flop:
            e["fp32_pipe_frac_nominal"] = flop[path] / (ms * 1e-3) / FP32_PEAK if ms else None
        paths[path] = e
    glue_ms = sum(kern.get("glue", {}).values())
    step_alg = 2 * S + 156.0 * rows + 12.0 * (fcep + facr) + 48.0 * n_utt      # PCM counted once (SURVEY section 8d)
    # ---- roofline of the dominant kernel
    flat = [(ms, k, path) for path, ks in kern.items() for k, ms in ks.items()]
    top_ms, top_k, top_path = max(flat)
    nf = fcep if top_path == "pitch_cep" else facr if top_path == "pitch_acr" else rows
    per_unit = {"pitch_cep": 2 * 160 + 12, "pitch_acr": 2 * 160 + 12, "mfcc": 2 * 160 + 156, "endpoint": 2 * 160}[top_path]
    top_alg = float(per_unit) * nf if top_path != "endpoint" else 2 * S
    traffic, traffic_src = recorded_traffic(top_k)
    roof = {"bound": "hbm", "kernel": top_k, "achieved": top_alg / (top_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
            "frac": top_alg / (top_ms * 1e-3) / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
            "alg_bytes_per_launch": top_alg, "launch_ms": top_ms, "share_of_step": top_ms / max(sum(m for m, _, _ in flat), 1e-9),
            "alg_bytes_per_unit": f"{per_unit} B per frame (one 10 ms hop of int16 PCM + the frame's outputs; DESIGN.md section 3)",
            "whole_step": {"alg_bytes": step_alg, "achieved": step_alg / (ms_per_step * 1e-3) / 1e9,
                           "frac": step_alg / (ms_per_step * 1e-3) / 1e9 / peak},
            "note": "the metric asks for the HBM fraction; the pitch transform kernels are bound by shared-memory bandwidth and the FP32 "
                    "pipe, not by HBM (paths.*.fp32_pipe_frac_nominal: 5 N log2 N flops per 512-point transform against 148 x 128 x 2 x 1.965 GHz)"}
    # ---- parity + CPU baseline on a bounded sample of this very batch (rank 0): first 4 x cores utterances
    n_s = min(n_utt, max(32, 4 * cores))
    fo_m = out["mfcc_frame_off"][: n_s + 1].cpu().numpy(); fo_c = out["cep_frame_off"][: n_s + 1].cpu().numpy()
    fo_a = out["acr_frame_off"][: n_s + 1].cpu().numpy()
    g_lr = out["lr"][:n_s].cpu().numpy(); g_m = out["mfcc"][: fo_m[-1]].cpu().numpy().astype(np.float64)
    g_cl = out["cep_lag"][: fo_c[-1]].cpu().numpy(); g_cp = out["cep_pitch"][: fo_c[-1]].cpu().numpy()
    g_al = out["acr_lag"][: fo_a[-1]].cpu().numpy(); g_ap = out["acr_pitch"][: fo_a[-1]].cpu().numpy()
    g_f = out["cep_feat"][:n_s].cpu().numpy()
    pcm_s = pcm[: int(off_np[n_s])].cpu().numpy()
    xs = [pcm_s[off_np[u]:off_np[u + 1]] for u in range(n_s)]
    jobs = [(xs[u], dict(lr=g_lr[u], mfcc=g_m[fo_m[u]:fo_m[u + 1]], cep_lag=g_cl[fo_c[u]:fo_c[u + 1]], cep_pitch=g_cp[fo_c[u]:fo_c[u + 1]],
                         acr_lag=g_al[fo_a[u]:fo_a[u + 1]], acr_pitch=g_ap[fo_a[u]:fo_a[u + 1]], feat=g_f[u])) for u in range(n_s)]
    res = pool.map(_w_parity, jobs, chunksize=1)
    tot_of = lambda k: int(sum(r[k] for r in res))
    mism = {"utterances": n_s, "frames": tot_of("cep_frames") + tot_of("acr_frames"),
            "differing": tot_of("cep_diff") + tot_of("acr_diff"), "near_tie": tot_of("cep_near") + tot_of("acr_near"),
            "hard": tot_of("cep_diff") + tot_of("acr_diff") - tot_of("cep_near") - tot_of("acr_near"),
            "cepstrum": {"frames": tot_of("cep_frames"), "differing": tot_of("cep_diff"), "near_tie": tot_of("cep_near")},
            "autocorrelation": {"frames": tot_of("acr_frames"), "differing": tot_of("acr_diff"), "near_tie": tot_of("acr_near")},
            "hz_inconsistent_with_lags": tot_of("hz_bad"), "endpoint_mismatches": tot_of("ep_bad"), "shape_mismatches": tot_of("shape_bad"),
            "near_tie_rule": "float64 oracle: peak-score bounds with every comparison moved by +-1e-5 max|row| overlap (cepstrum) / "
                             "chosen lag's score within 1e-5 max|row| of the maximum (autocorrelation)"}
    parity = {"mfcc_max_err": float(max(r["mfcc_err"] for r in res)), "mfcc_tolerance": 1e-4,
              "pitch_feature_checked": tot_of("feat_checked"), "pitch_feature_max_rel_err": float(max(r["feat_err"] for r in res)),
              "pitch_feature_tolerance": 1e-6}
    cpu = None
    if world == 1:
        kind = "reference" if reference_available() else "port"
        n_c = min(n_utt, 8 * cores)                 # the same sample size per step as the --impl reference arm
        pcm_c = pcm[: int(off_np[n_c])].cpu().numpy()
        xs_c = [pcm_c[off_np[u]:off_np[u + 1]] for u in range(n_c)]
        v, dt, aud = cpu_front_end(pool, kind, xs_c, cores, repeats=3)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"the first {n_c} utterances of this batch ({aud:.0f} audio-s), best of 3 passes, whole front-end per utterance with "
                         + ("the unmodified reference features package (baseline/_ref)" if kind == "reference" else "the oracle port (NumPy float64)")
                         + f" in {cores} processes, {dt:.1f} s wall"}
    pool.close()
    line = {
        "metric": METRIC, "value": audio_all / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "utterances_per_gpu": U, "audio_s_per_step": audio_all,
                   "shard_imbalance": shard.imbalance(all_len, parts), "sharding": "dspfe.shard.lpt_partition of one global length list",
                   "l2_policy": "PCM per step (%.0f MB per GPU) exceeds the 126 MB L2" % (total * 2 / 1e6),
                   "rows": {"mfcc": rows, "pitch_cep": fcep, "pitch_acr": facr}},
        "paths": paths, "glue_ms": glue_ms, "roofline": roof,
        "e2e": {"value": audio_all / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                "ms_per_step": e2e_s * 1e3, "timer": "host wall clock around the blocking dspfe_frontend_host call, max over ranks",
                "matches_device_path": e2e_ok},
        "pitch_mismatch": mism, "parity": parity,
        "gpu_launches": int(launches_all), "clocks": clocks,
    }
    if cpu:
        line["cpu_baseline"] = cpu
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- GPU arm: MFCC only (BASELINE configs[1])
def run_mfcc(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import dspfe
    from dspfe import synth
    from oracle import ref_features as O   # checker only

    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the product path has no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    U, S = UTT_PER_GPU, 2 * SR
    lengths = np.full(U, S, dtype=np.int64)
    pcm, off = synth.synth_batch_torch(lengths, seed0=1000003 * rank, device=dev)
    off_d = off.to(dev)
    plan = dspfe.MfccPlan(frame_len=400, frame_step=160, numcep=13, delta_n=DELTA_N)
    plan.reserve(U, pcm.numel())
    rows = int(dspfe.frame_counts(lengths, 400, 160).sum())
    out = torch.empty((plan.rows_bound(pcm.numel(), U), 39), dtype=torch.float32, device=dev)
    fo = torch.empty(U + 1, dtype=torch.int64, device=dev)
    audio_s = float(lengths.sum()) / SR
    alg_bytes = 2.0 * float(lengths.sum()) + 156.0 * rows

    def step():
        plan.mfcc_delta(pcm, off_d, out=out, frame_off=fo)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    step()
    torch.cuda.synchronize()
    par = 0.0
    got = out[: 4 * 199].cpu().numpy()
    for u in range(4):
        ref = O.mfcc_delta39(pcm[u * S:(u + 1) * S].cpu().numpy(), DELTA_N)
        par = max(par, float(np.max(np.abs(got[u * 199:(u + 1) * 199] - ref) / (1 + np.abs(ref)))))
    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.wait_first()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    last = (out[:rows].clone(), fo.clone()) if args.dump_outputs else None     # written after the clock sampling
    dspfe.timing_begin()
    for _ in range(args.steps):
        step()
    k_ms = float(np.median([ms for name, ms in dspfe.timing_end() if name == "mfcc_delta_kernel"]))
    clocks = sample_clocks_under(sampler, step, torch) if sampler else None
    if last:
        dump(args, rank, world, {}, {"mfcc_frame_off": (last[1].cpu().numpy(), {"mfcc": last[0]})})
    t = torch.tensor([ms_total, k_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, k_ms = [float(v) for v in t.cpu()]
    if rank == 0:
        ms_per_step = ms_total / args.steps
        peak, peak_src = peaks()
        traffic, traffic_src = recorded_traffic("mfcc_delta_kernel@configs1")
        emit({
            "metric": "audio-sec/sec of MFCC+delta+delta-delta (fused kernel), 4096 x 2 s utterances per B200",
            "value": world * audio_s / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: 4096 x 2 s utterances per GPU @16 kHz int16, 25/10 ms frames, nfft 512, 26 mel, 13 MFCC + delta + "
                                   "delta-delta (N=2) -> float32 [F,39]", "frames_per_gpu": rows, "kernel": plan.info(),
                       "l2_policy": "working set per step (262 MB in + 127 MB out) exceeds the 126 MB L2",
                       "parity_max_err_vs_oracle": par, "tolerance": 1e-4},
            "roofline": {"bound": "hbm", "kernel": "mfcc_delta_kernel", "achieved": alg_bytes / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg_bytes / (k_ms * 1e-3) / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_src, "alg_bytes_per_launch": alg_bytes, "launch_ms": k_ms},
            "gpu_launches": 2 * args.steps, "clocks": clocks})
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="frontend", choices=["frontend", "mfcc"],
                    help="frontend = the metric's workload (default); mfcc = the MFCC-only line of BASELINE configs[1]")
    ap.add_argument("--utterances", type=int, default=UTT_PER_GPU, help="utterances per GPU of the frontend workload")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    # SIGTERM (torch.distributed.run stopping the ranks when one fails) leaves through sys.exit, so the atexit hooks run
    signal.signal(signal.SIGTERM, lambda *_: sys.exit(128 + signal.SIGTERM))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm keeps no outputs")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
    elif args.workload == "frontend":
        run_frontend(args, rank, world, local_rank)
    else:
        run_mfcc(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
