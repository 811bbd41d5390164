"""CPU checks of the exact pieces of the float32 robust-endpoint gate (endpoint_kernel.cuh acr_lag / acr_gate_frame, which the
device kernel's exact path shares): acr(frame, n) bit for bit against NumPy's summation for every term count up to the longest
built frame, and the gate against the oracle's acr_rule on random, non-finite, all-zero and near-threshold frames."""
import ctypes
import os
import sys
import warnings

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu  # noqa: E402

MAX_LEN = 1536          # kEpGateMaxLen


def _lib():
    L = emu.lib()
    L.emu_acr_lag_f32.restype = ctypes.c_double
    L.emu_acr_lag_f32.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    L.emu_acr_gate_f32.restype = ctypes.c_int
    L.emu_acr_gate_f32.argtypes = [ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    return L


def acr_lag(x, avail, length, n):
    x = np.ascontiguousarray(x, dtype=np.float32)
    return _lib().emu_acr_lag_f32(x.ctypes.data, int(avail), int(length), int(n))


def gate(x, avail, length, n0, n1):
    x = np.ascontiguousarray(x, dtype=np.float32)
    return bool(_lib().emu_acr_gate_f32(x.ctypes.data, int(avail), int(length), int(n0), int(n1)))


def frame64(x, avail, length):
    """framesig's float64 frame: the samples that exist, then zeros."""
    f = np.zeros(length)
    f[:avail] = x[:avail].astype(np.float64)
    return f


def numpy_acr(f, n):
    return np.sum(f * f) / len(f) if n == 0 else np.sum(f[:-n] * f[n:]) / (len(f) - n)


def oracle_gate(f, rate):
    from oracle import ref_features as O
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        acrs = [O.acr(f, n) for n in range(rate // 500, rate // 50)]
        return bool(max(acrs) / O.acr(f, 0) > 0.55)


def families(rng, size):
    """random float32 frames: plain, subnormal, tiny-scaled (x 2^-140) and huge-scaled (x 2^100)"""
    g = rng.standard_normal(size)
    sub = (rng.integers(-2 ** 23, 2 ** 23, size) * 2.0 ** -149).astype(np.float32)
    return {"normal": g.astype(np.float32), "subnormal": sub,
            "tiny": (g.astype(np.float32) * np.float32(2.0 ** -140)).astype(np.float32),
            "huge": (g.astype(np.float32) * np.float32(2.0 ** 100)).astype(np.float32)}


def test_acr_lag_every_term_count_bit_exact():
    """acr(frame, n) equals NumPy's np.sum(f[:-n] * f[n:]) / (len - n) for every term count len - n from 1 to 1536, with and
    without a zero tail, on four families of float32 data; sequential summation differs on some of them, so the order bites."""
    rng = np.random.default_rng(20)
    bad, seq_differs = [], 0
    for k in range(1, MAX_LEN + 1):
        n = int(rng.integers(0, min(40, MAX_LEN - k) + 1))
        length = k + n
        avail = length if k % 3 else int(rng.integers(0, length + 1))
        for name, x in families(rng, length).items():
            f = frame64(x, avail, length)
            got = acr_lag(x, avail, length, n)
            want = numpy_acr(f, n)
            if got != want and not (np.isnan(got) and np.isnan(want)):
                bad.append((k, n, name, got, want))
            prod = f * f if n == 0 else f[:-n] * f[n:]
            seq_differs += int(np.cumsum(prod)[-1] / k != want)
    assert not bad, f"{len(bad)} lag sums differ from NumPy's, e.g. {bad[:5]}"
    assert seq_differs > 100, seq_differs


def test_gate_vs_oracle_random_frames():
    rng = np.random.default_rng(21)
    for rate in (8000, 16000, 22050, 48000):
        length = int(rate * 0.03)
        n0, n1 = rate // 500, min(rate // 50, length)
        for t in range(40):
            period = int(rng.integers(n0 + 1, rate // 50))
            i = np.arange(length)
            x = np.sin(2 * np.pi * i / period) + rng.standard_normal(length) * rng.choice([0.05, 0.5, 1.0, 3.0])
            x = (x * rng.choice([1.0, 2.0 ** -30, 2.0 ** 40, 1e-38 / 3])).astype(np.float32)
            avail = length if t % 4 else int(rng.integers(0, length + 1))
            f = frame64(x, avail, length)
            assert gate(x, avail, length, n0, n1) == oracle_gate(f, rate), (rate, t)


def test_gate_non_finite_and_zero_frames():
    """A NaN, +inf or +-inf sample makes the gate false, as in the oracle; an all-zero frame gives 0 / 0, false."""
    rng = np.random.default_rng(22)
    length, rate = 480, 16000
    base = np.sin(2 * np.pi * np.arange(length) / 100).astype(np.float32)
    cases = {}
    for name, vals in {"nan": [np.nan], "inf": [np.inf], "inf_minf": [np.inf, -np.inf], "minf": [-np.inf]}.items():
        x = base.copy()
        x[rng.choice(length, len(vals), replace=False)] = vals
        cases[name] = x
    cases["zero"] = np.zeros(length, np.float32)
    for name, x in cases.items():
        assert gate(x, length, length, rate // 500, rate // 50) is False, name
        assert oracle_gate(frame64(x, length, length), rate) is False, name


def near_threshold_frame(rate, length, period, seed):
    """periodic + a * noise with the float32 coefficient a bisected until the oracle's decision flips: the frames either side of
    the flip, both a few ulps from acr_rule's 0.55."""
    rng = np.random.default_rng(seed)
    i = np.arange(length)
    p = np.sin(2 * np.pi * i / period) + 0.3 * np.sin(2 * np.pi * 3 * i / period + 0.7)
    noise = rng.standard_normal(length)
    mk = lambda a: (p + np.float64(a) * noise).astype(np.float32)
    lo, hi = np.float32(0.0), np.float32(4.0)
    assert oracle_gate(mk(lo).astype(np.float64), rate) and not oracle_gate(mk(hi).astype(np.float64), rate)
    while np.nextafter(lo, hi) != hi:
        mid = np.float32((np.float64(lo) + np.float64(hi)) / 2)
        if mid in (lo, hi):
            break
        if oracle_gate(mk(mid).astype(np.float64), rate):
            lo = mid
        else:
            hi = mid
    return mk(lo), mk(hi)


def test_gate_near_threshold_frames():
    """Frames that sit about 1e-8 from 0.55, well inside the float32 screening band delta (about 1.3e-4 at 16 kHz): only an exact
    float64 evaluation in NumPy's order decides them the reference's way."""
    checked = 0
    for rate, period, seed in [(16000, 97, 1), (16000, 150, 2), (16000, 61, 3), (8000, 53, 4), (22050, 131, 5), (48000, 400, 6)]:
        length = int(rate * 0.03)
        n0, n1 = rate // 500, rate // 50
        for x, want in zip(near_threshold_frame(rate, length, period, seed), (True, False)):
            f = x.astype(np.float64)
            ratio = max(numpy_acr(f, n) for n in range(n0, n1)) / numpy_acr(f, 0)
            assert abs(ratio - 0.55) < 1e-6, ratio
            assert oracle_gate(f, rate) is want
            assert gate(x, length, length, n0, n1) is want, (rate, period, seed)
            checked += 1
    assert checked == 12
