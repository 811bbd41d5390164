"""CPU checks of the float-sample endpoint path: the K2f kernel body on the SIMT emulator against NumPy, and the decision
rule on amplitudes that only float input can produce (NaN, +-inf)."""
import ctypes
import os
import sys

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu  # noqa: E402


def k2f(pcm, offsets, frame_len, frame_step, nthreads=64):
    L = emu.lib()
    L.emu_endpoint_f32.restype = ctypes.c_longlong
    pcm = np.ascontiguousarray(pcm, dtype=np.float32)
    off = np.ascontiguousarray(offsets, dtype=np.int64)
    cap = int(len(pcm) // frame_step + 2 * (len(off) - 1) + 1)
    amp = np.full(cap, np.nan)
    zcr = np.full(cap, -1, dtype=np.int32)
    fo = np.zeros(len(off), dtype=np.int64)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    r = L.emu_endpoint_f32(vp(pcm), ctypes.c_longlong(len(pcm)), vp(off), len(off) - 1, frame_len, frame_step, nthreads, vp(amp),
                           vp(zcr), ctypes.c_longlong(cap), vp(fo))
    assert r >= 0, r
    return amp[:r], zcr[:r], fo


def test_summation_order_every_frame_length():
    """amp of every frame is np.mean(np.abs(row)) bit for bit for frame lengths 1 .. 2048 (frames = rows: step = length)."""
    rng = np.random.default_rng(7)
    bad = []
    for L in range(1, 2049):
        rows = 2 if L > 64 else 3
        x = (rng.standard_normal(rows * L) * rng.choice([1e-3, 1.0, 3e4], rows * L)).astype(np.float32)
        amp, zcr, _ = k2f(x, [0, len(x)], L, L)
        fr = x.astype(np.float64).reshape(rows, L)
        want = np.array([np.mean(np.abs(r)) for r in fr])
        wz = (fr[:, :-1] * fr[:, 1:] < 0).sum(axis=1)
        if not (np.array_equal(amp, want) and np.array_equal(zcr, wz)):
            bad.append(L)
    assert not bad, f"frame lengths with a differing amplitude or zero-crossing count: {bad[:20]}"


def test_ragged_overlapping_frames_vs_oracle():
    from oracle import ref_features as O
    rng = np.random.default_rng(11)
    for rate, cfg_frame, cfg_step in [(16000, 0.03, 0.01), (8000, 0.03, 0.01), (22050, 0.03, 0.01), (16000, 0.03, 0.04)]:
        L, S = int(rate * cfg_frame), int(cfg_step * rate)
        lengths = [0, 1, L - 1, L, L + 1, 3 * S + 7, 5000, 2 * L]
        xs = [(rng.standard_normal(n) * 0.37).astype(np.float32) for n in lengths]
        xs[-1][:] = 0.0                                     # digital silence
        xs[-2][::5] = -0.0
        off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        pcm = np.concatenate(xs + [np.zeros(0, np.float32)])
        for nthreads in (32, 96):
            amp, zcr, fo = k2f(pcm, off + 0, L, S, nthreads)
            for u, x in enumerate(xs):
                fr = O.to_frames(x.astype(np.float64), rate, t=cfg_frame, step=cfg_step)
                np.testing.assert_array_equal(amp[fo[u]:fo[u + 1]], np.array(O.get_amplitude(fr)))
                np.testing.assert_array_equal(zcr[fo[u]:fo[u + 1]], np.array(O.get_zcr(fr)))


def test_amplitude_rule_terminates_on_nan_and_inf():
    import dspfe
    rng = np.random.default_rng(3)
    for F in (1, 5, 40, 120, 700):
        for kind in ("nan", "inf", "-inf", "mixed", "all_nan"):
            a = rng.random(F) * 0.1
            if kind == "all_nan":
                a[:] = np.nan
            else:
                idx = rng.choice(F, max(1, F // 7), replace=False)
                a[idx] = {"nan": np.nan, "inf": np.inf, "-inf": -np.inf}.get(kind, np.nan)
                if kind == "mixed":
                    a[idx[::2]] = np.inf
            for mh in (0.25, 0.125):
                segs = dspfe.amplitude_rule_host(a, mh=mh)
                assert len(segs) >= 1
                for j, k in segs:
                    assert 0 <= j <= F and 0 <= k <= F, (kind, F, segs)
