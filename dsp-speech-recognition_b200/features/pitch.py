"""Drop-in for reference features/pitch.py: cepstrum / autocorrelation pitch and the pitch-SVM features.

Frame-level arithmetic (decimation, centre clipping, the complex FIR band-pass, cepstrum, autocorrelation,
smoothing, peak scoring) runs in the sm_100a kernels K4a/K4b/K5 (csrc/pitch_kernel.cuh) through libdspfe.so;
the per-utterance list logic (octave repair, smooth runs, least-squares fits) is the same C++ the device
kernel K6 runs, reached through the *_host entry points.  There is no CPU fallback for the kernels.
"""
import functools
import pickle  # noqa: F401  (pitch_model.py relies on `from features.pitch import *` exporting pickle, SURVEY A-12)
import re  # noqa: F401

import numpy as np

import dspfe
from . import _gpu
from .preprocess import preemphasis, downsampling  # noqa: F401
from .sigproc import to_frames, window, acr  # noqa: F401
from .endpoint import basic_endpoint_detection, get_amplitude, robust_endpoint_detection  # noqa: F401

try:  # names the reference module re-exports from the host project / scikit-learn (pitch.py:14-23); optional here
    from reader import Reader  # noqa: F401
except Exception:
    Reader = None
try:
    from plotter import plot_frame, show, scatter  # noqa: F401
except Exception:
    def plot_frame(*a, **k):
        return None

    def show(*a, **k):
        return None

    def scatter(*a, **k):
        return None
try:
    from sklearn.ensemble import GradientBoostingClassifier  # noqa: F401
    from sklearn.svm import SVC  # noqa: F401
    from sklearn.preprocessing import scale, RobustScaler  # noqa: F401
    from sklearn.metrics import accuracy_score  # noqa: F401
except Exception:  # scikit-learn is a dependency of the reference's callers, not of the kernels
    pass

_DST_RATE = 10000   # pitch.py:84,100


@functools.lru_cache(maxsize=32)
def _plan(method, rate, dst_rate, frame_len, frame_step, clip, row_len):
    return dspfe.PitchPlan(method=method, samplerate=rate, dst_rate=dst_rate, frame_len=frame_len, frame_step=frame_step,
                           center_clip=clip, row_len=row_len)


def _frame_geometry(winlen, step):
    # to_frames(sig, 10000, winlen, step): int(rate * t), int(step * rate)  (sigproc.py:19)
    return int(_DST_RATE * winlen), int(step * _DST_RATE)


def _detect(sig, rate, winlen, step, method, want_feat=False):
    frame_len, frame_step = _frame_geometry(winlen, step)
    if method == 0 and frame_len < 100:
        # the reference's peak_score reads row[20..99] of every cepstrum row of frame_len values (pitch.py:232)
        raise IndexError(f"index {max(frame_len, 20)} is out of bounds for axis 0 with size {frame_len}")
    if method == 0 and frame_len > 512:
        raise NotImplementedError("cepstrum pitch is built for frames of 100..512 samples at 10 kHz (winlen 0.01..0.0512)")
    if method == 1 and not (20 < frame_len <= 512):
        raise NotImplementedError("autocorrelation pitch is built for frames of 21..512 samples at 10 kHz")
    if frame_step < 1:
        raise NotImplementedError("frame step below one sample")
    x, _ = _gpu.pack_one(sig)
    plan = _plan(method, int(rate), _DST_RATE, frame_len, frame_step, True, 0)
    off = np.array([0, len(x)], dtype=np.int64)
    return plan.detect_host(x, off, want_feat=want_feat), (frame_len, frame_step)


def _frames_of(sig, rate, frame_len, frame_step):
    ds = downsampling(np.asarray(sig), rate, _DST_RATE)
    return dspfe.frames_f64(ds.astype(np.float64), frame_len, frame_step)


def pitch_feature(sig, rate, gender='male'):
    """reference pitch.py:26-47: the five SVM inputs (slope1, slope2, quad1, quad2, median shift) of a signal that
    has been endpoint-trimmed (and pre-emphasised) by the caller.  The reference's two debugging prints are dropped."""
    (pitch, lag, fo, feat), _ = _detect(sig, rate, 0.0512, 0.01, 0, want_feat=True)   # always the default winlen (pitch.py:33)
    return tuple(np.float64(v) for v in feat[0])


def slope(seq):
    """reference pitch.py:49-52: leading coefficient of the degree-1 least-squares fit over x = 0..n-1."""
    return np.float64(dspfe.poly_lead_host(seq, 1))


def quad_params(seq):
    """reference pitch.py:54-57: leading coefficient of the degree-2 fit."""
    return np.float64(dspfe.poly_lead_host(seq, 2))


def peakshift(seq1, seq2):
    """reference pitch.py:59-62."""
    return np.median(seq2) - np.median(seq1)


def sub_endpoint_detect(frames):
    """reference pitch.py:64-81: index of the deepest +-10-frame amplitude valley (len//2 when there is none)."""
    amp = dspfe.row_amplitude_f64(np.asarray(frames, dtype=np.float64), use_sq=2)   # sum |x| per frame, on the device
    return dspfe.sub_endpoint_host(amp)


def pitch_detect(sig, rate, winlen=0.0512, step=0.01, gender='male'):
    """reference pitch.py:83-94: cepstrum pitch.  Returns (list of Hz per frame, frames [F,N] float64), N = int(10000 * winlen).
    N from 100 to 512 samples is built; N < 100 raises IndexError as the reference's peak_score does, N > 512 NotImplementedError."""
    (pitch, lag, fo), (fl, fs) = _detect(sig, rate, winlen, step, 0)
    return [np.float64(v) for v in pitch], _frames_of(sig, rate, fl, fs)


def pitch_detect_sr(sig, rate, winlen=0.0512, step=0.01):
    """reference pitch.py:96-110: autocorrelation pitch.  Returns (list of Hz per frame, frames)."""
    (pitch, lag, fo), (fl, fs) = _detect(sig, rate, winlen, step, 1)
    return [np.float64(v) for v in pitch], _frames_of(sig, rate, fl, fs)


def _frame_rows(frame, rate, method, row_len):
    a = np.asarray(frame, dtype=np.float64)
    if a.ndim != 1:
        raise NotImplementedError("expected one 1-D frame")
    import torch
    if not torch.cuda.is_available():
        raise dspfe.DspfeError(-3, "no CUDA device: the features package has no CPU fallback")
    # one frame = a one-frame utterance that is already at the target rate: no decimation, no clipping
    plan = _plan(method, int(rate), int(rate), len(a), 100, False, row_len)
    x = torch.from_numpy(a.astype(np.float32)).cuda()
    off = torch.tensor([0, len(a)], dtype=torch.int64, device=x.device)
    o = plan.detect(x, off, want_rows=True, want_track=False)
    torch.cuda.synchronize()
    return o["rows"][0].cpu().numpy().astype(np.float64)


def pitch_detect_frame_sr(frame, rate):
    """reference pitch.py:112-132: unbiased autocorrelation of |band-passed frame| at lags 20..199 (list of 180)."""
    if not (20 < len(frame) <= 512):
        raise NotImplementedError("autocorrelation frames of 21..512 samples are built")
    return [np.float64(v) for v in _frame_rows(frame, rate, 1, 0)]


def pitch_detect_frame(frame, rate, gender):
    """reference pitch.py:135-143: |ifft(log|fft(window(frame, 50, 1000, 'hamming'))|)|, all N values of a 1-D frame of
    N = 100..512 samples (N-point transforms, as the reference)."""
    n = np.asarray(frame).shape[-1] if np.ndim(frame) else 0
    if np.ndim(frame) != 1 or not (100 <= n <= 512):
        raise NotImplementedError("the cepstrum kernel is built for 1-D frames of 100..512 samples")
    return _frame_rows(frame, rate, 0, n)


def center_clip(frame, binary=True):
    """reference pitch.py:145-155: clip at the median of the non-negative samples."""
    a = np.asarray(frame)
    if a.ndim != 1 or len(a) > 512:
        raise NotImplementedError("center_clip is built for 1-D frames of up to 512 samples")
    out = dspfe.center_clip_f32(a.astype(np.float32), binary)
    return out.astype(np.int64) if binary else out.astype(np.float64)


def smooth(g, degree=2):
    """reference pitch.py:157-164: in-place running mean over rows (a recurrence), returned as a list of lists."""
    if degree != 2:
        raise NotImplementedError("only degree=2 (the reference's only call) is built")
    a = np.asarray(g, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] > 512:
        raise NotImplementedError("smooth is built for 2-D score arrays of up to 512 columns")
    sm, _, _ = dspfe.smooth_rows_f32(a, mode=1)
    return sm.astype(np.float64).tolist()


def _lags(g, bias):
    return [int(bias + np.argmax(l)) for l in g]


def max_pitch(g, bias=20):
    """reference pitch.py:166-172."""
    return [np.float64(v) for v in dspfe.robust_max_pitch_host(_lags(g, bias), repair=False)]


def greedy_max_pitch(g, bias=20):
    """reference pitch.py:174-189: the first local descent of every row."""
    out = []
    for l in g:
        a = np.asarray(l)
        drop = np.nonzero(a[:-1] > a[1:])[0]
        out.append(1 / (0.0001 * (int(drop[0]) + bias)) if len(drop) else 0)
    return out


def robust_max_pitch(g, bias=20):
    """reference pitch.py:191-206: argmax per row, then forward and backward octave repair."""
    return [np.float64(v) for v in dspfe.robust_max_pitch_host(_lags(g, bias), repair=True)]


def dp_max_pitch(g):
    """reference pitch.py:208-225: Viterbi over lags with a jump penalty (same back-trace start as the reference)."""
    a = np.asarray(g, dtype=np.float64)
    if a.ndim != 2 or a.shape[0] < 2:
        raise NotImplementedError("dp_max_pitch needs a 2-D score array with at least two rows")
    return dspfe.dp_max_pitch_f64(a).tolist()       # device kernel (dspfe_dp_max_pitch)


def peak_score(sig, gender='male'):
    """reference pitch.py:227-242: for lags 20..99, distance to the nearest strictly greater sample."""
    a = np.asarray(sig, dtype=np.float32)
    if a.ndim != 1 or not (100 <= len(a) <= 512):
        raise NotImplementedError("peak_score is built for 1-D rows of 100..512 samples")
    _, sc, _ = dspfe.smooth_rows_f32(a.reshape(1, -1), mode=0, want_score=True, do_smooth=False)
    return [int(v) for v in sc[0]]


def find_smooth_subsequence(pitch, base_tor=3, base_thres=30, bias=0):
    """reference pitch.py:245-279: longest run with at most base_tor jumps larger than base_thres Hz.
    Returns (values, (start + bias, stop + bias))."""
    seg, (i0, j0) = dspfe.smooth_subsequence_host(list(pitch), base_tor, float(base_thres))
    return [np.float64(v) for v in seg], (i0 + bias, j0 + bias)
