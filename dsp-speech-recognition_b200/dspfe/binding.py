"""ctypes binding of include/dspfe.h."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(os.path.dirname(_HERE), "libdspfe.so")
_lib = None


class DspfeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"dspfe error {code}: {msg}")
        self.code = code


class _MfccParams(ctypes.Structure):
    _fields_ = [("samplerate", ctypes.c_int32), ("frame_len", ctypes.c_int32), ("frame_step", ctypes.c_int32),
                ("nfft", ctypes.c_int32), ("nfilt", ctypes.c_int32), ("numcep", ctypes.c_int32),
                ("ceplifter", ctypes.c_int32), ("append_energy", ctypes.c_int32), ("delta_n", ctypes.c_int32),
                ("seg_frames", ctypes.c_int32), ("preemph", ctypes.c_double), ("lowfreq", ctypes.c_double),
                ("highfreq", ctypes.c_double), ("window", ctypes.POINTER(ctypes.c_double))]


def lib_path():
    return _LIB_PATH


def lib():
    """Loads libdspfe.so; fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            raise ImportError(f"{_LIB_PATH} is missing: build it with `python dsp-speech-recognition_b200/build.py` "
                              "(there is no CPU fallback)")
        L = ctypes.CDLL(_LIB_PATH)
        L.dspfe_version.restype = ctypes.c_char_p
        L.dspfe_last_error.restype = ctypes.c_char_p
        L.dspfe_num_frames.restype = ctypes.c_int64
        L.dspfe_num_frames.argtypes = [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32]
        L.dspfe_rows_bound.restype = ctypes.c_int64
        L.dspfe_rows_bound.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]
        L.dspfe_plan_create.argtypes = [ctypes.POINTER(_MfccParams), ctypes.POINTER(ctypes.c_void_p)]
        L.dspfe_plan_reserve.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]
        L.dspfe_plan_destroy.argtypes = [ctypes.c_void_p]
        L.dspfe_plan_destroy.restype = None
        L.dspfe_plan_info.argtypes = [ctypes.c_void_p] + [ctypes.POINTER(ctypes.c_int32)] * 3
        L.dspfe_mfcc_delta.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]
        L.dspfe_mfcc_delta_host.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                            ctypes.c_void_p, ctypes.c_void_p]
        L.dspfe_mfcc_tables_host.argtypes = [ctypes.POINTER(_MfccParams), ctypes.c_void_p, ctypes.c_int32,
                                             ctypes.POINTER(ctypes.c_int32), ctypes.c_void_p]
        L.dspfe_host_alloc.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int64]
        L.dspfe_host_free.argtypes = [ctypes.c_void_p]
        _lib = L
    return _lib


class DspfeUnsupported(DspfeError, NotImplementedError):
    """DSPFE_ERR_UNSUPPORTED: a parameter combination outside the built set (there is no CPU fallback to hand it to)."""


def _check(rc):
    if rc != 0:
        raise (DspfeUnsupported if rc == -2 else DspfeError)(rc, lib().dspfe_last_error().decode())


def mfcc_params(samplerate=16000, frame_len=400, frame_step=160, nfft=512, nfilt=26, numcep=13, ceplifter=22,
                append_energy=True, delta_n=2, seg_frames=0, preemph=0.97, lowfreq=0.0, highfreq=None, window=None):
    """Returns (ctypes struct, keep-alive) for dspfe_mfcc_params; `window` is winfunc(frame_len) or None."""
    p = _MfccParams(int(samplerate), int(frame_len), int(frame_step), int(nfft), int(nfilt), int(numcep),
                    int(ceplifter), int(bool(append_energy)), int(delta_n), int(seg_frames), float(preemph),
                    float(lowfreq or 0.0), float(highfreq or 0.0), None)
    keep = None
    if window is not None:
        keep = np.ascontiguousarray(window, dtype=np.float64)
        if keep.shape != (int(frame_len),):
            raise ValueError("window must have frame_len entries")
        p.window = keep.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    return p, keep


def num_frames(n_samples, frame_len, frame_step):
    return int(lib().dspfe_num_frames(int(n_samples), int(frame_len), int(frame_step)))


def frame_counts(lengths, frame_len, frame_step):
    """framesig's frame count (reference sigproc.py:79-82), vectorised on the host."""
    lengths = np.asarray(lengths, dtype=np.int64)
    return np.where(lengths <= frame_len, 1, 1 + (lengths - frame_len + frame_step - 1) // frame_step).astype(np.int64)


def mfcc_tables_host(**kw):
    """Host-only table construction (no CUDA): returns (blob float32[n], mel_edges float64[nfilt+2])."""
    p, keep = mfcc_params(**kw)
    n = ctypes.c_int32(0)
    _check(lib().dspfe_mfcc_tables_host(ctypes.byref(p), None, 0, ctypes.byref(n), None))
    blob = np.zeros(n.value, dtype=np.float32)
    edges = np.zeros(p.nfilt + 2, dtype=np.float64)
    _check(lib().dspfe_mfcc_tables_host(ctypes.byref(p), blob.ctypes.data_as(ctypes.c_void_p), n.value, ctypes.byref(n),
                                        edges.ctypes.data_as(ctypes.c_void_p)))
    return blob, edges


class MfccPlan:
    """dspfe_plan: parameters + device tables + workspaces for the fused MFCC+delta+delta-delta kernel."""

    def __init__(self, **kw):
        self._p, self._keep = mfcc_params(**kw)
        self.frame_len, self.frame_step = self._p.frame_len, self._p.frame_step
        self.width = 3 * self._p.numcep
        h = ctypes.c_void_p()
        _check(lib().dspfe_plan_create(ctypes.byref(self._p), ctypes.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib().dspfe_plan_destroy(self._h)
            self._h = None

    __del__ = close

    def info(self):
        a, b, c = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
        _check(lib().dspfe_plan_info(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return dict(smem_bytes=a.value, ctas_per_sm=b.value, regs_per_thread=c.value)

    def rows_bound(self, total_samples, n_utt):
        return int(lib().dspfe_rows_bound(self._h, int(total_samples), int(n_utt)))

    def reserve(self, max_utt, max_total_samples):
        _check(lib().dspfe_plan_reserve(self._h, int(max_utt), int(max_total_samples)))

    def mfcc_delta(self, pcm, offsets, trim=None, out=None, frame_off=None, stream=None):
        """Device path.  pcm int16 CUDA tensor [total], offsets int64 CUDA tensor [U+1], optional trim int32
        CUDA tensor [U,2].  Asynchronous on `stream` (default: torch's current stream).  Returns
        (out float32 [rows_bound, 3*numcep], frame_off int64 [U+1]); rows beyond frame_off[-1] are untouched."""
        import torch
        assert pcm.is_cuda and pcm.dtype == torch.int16 and pcm.is_contiguous()
        assert offsets.is_cuda and offsets.dtype == torch.int64 and offsets.is_contiguous()
        n_utt = offsets.numel() - 1
        total = pcm.numel()
        rows = self.rows_bound(total, n_utt)
        if out is None:
            out = torch.empty((rows, self.width), dtype=torch.float32, device=pcm.device)
        assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.shape[0] >= rows
        if frame_off is None:
            frame_off = torch.empty(n_utt + 1, dtype=torch.int64, device=pcm.device)
        tp = None
        if trim is not None:
            assert trim.is_cuda and trim.dtype == torch.int32 and trim.is_contiguous() and trim.shape == (n_utt, 2)
            tp = trim.data_ptr()
        st = stream if stream is not None else torch.cuda.current_stream(pcm.device).cuda_stream
        _check(lib().dspfe_mfcc_delta(self._h, pcm.data_ptr(), total, offsets.data_ptr(), tp, n_utt, out.data_ptr(),
                                      out.shape[0], frame_off.data_ptr(), ctypes.c_void_p(st)))
        return out, frame_off

    def mfcc_delta_host(self, pcm, offsets, out=None):
        """Host path (the reference-facing call): NumPy (or pinned torch CPU) int16 pcm + int64 offsets in, NumPy
        float32 [rows, 3*numcep] out; H2D, kernels and D2H are pipelined inside libdspfe."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n_utt = len(offsets) - 1
        rows = int(frame_counts(np.diff(offsets), self.frame_len, self.frame_step).sum())
        if out is None:
            out = np.empty((rows, self.width), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.shape[0] >= rows
        fo = np.empty(n_utt + 1, dtype=np.int64)
        _check(lib().dspfe_mfcc_delta_host(self._h, pcm.ctypes.data_as(ctypes.c_void_p),
                                           offsets.ctypes.data_as(ctypes.c_void_p), n_utt,
                                           out.ctypes.data_as(ctypes.c_void_p), fo.ctypes.data_as(ctypes.c_void_p)))
        return out[:rows], fo


# ------------------------------------------------------------------------------------------------ endpoint
class _EndpointParams(ctypes.Structure):
    _fields_ = [("samplerate", ctypes.c_int32), ("min_span", ctypes.c_int32), ("cfg_frame", ctypes.c_double),
                ("cfg_step", ctypes.c_double), ("mh1", ctypes.c_double), ("mh2", ctypes.c_double), ("th", ctypes.c_double),
                ("l_sil", ctypes.c_double), ("r_sil", ctypes.c_double), ("sigma", ctypes.c_double),
                ("zcr_max_shift", ctypes.c_double), ("zcr_r_sil", ctypes.c_double)]


def _bind_endpoint(L):
    if getattr(L, "_ep_bound", False):
        return
    L.dspfe_endpoint_params_default.argtypes = [ctypes.POINTER(_EndpointParams), ctypes.c_int32]
    L.dspfe_endpoint_params_default.restype = None
    L.dspfe_endpoint_create.argtypes = [ctypes.POINTER(_EndpointParams), ctypes.POINTER(ctypes.c_void_p)]
    L.dspfe_endpoint_destroy.argtypes = [ctypes.c_void_p]
    L.dspfe_endpoint_destroy.restype = None
    L.dspfe_endpoint_frame_len.argtypes = [ctypes.c_void_p]
    L.dspfe_endpoint_frame_step.argtypes = [ctypes.c_void_p]
    L.dspfe_endpoint_frames_bound.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]
    L.dspfe_endpoint_frames_bound.restype = ctypes.c_int64
    L.dspfe_endpoint.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int32,
                                 ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                 ctypes.c_void_p]
    L.dspfe_endpoint_host.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    L.dspfe_endpoint_decide_host.argtypes = [ctypes.POINTER(_EndpointParams), ctypes.c_void_p, ctypes.c_void_p,
                                             ctypes.c_int32, ctypes.c_void_p]
    L.dspfe_amplitude_rule_host.argtypes = [ctypes.POINTER(_EndpointParams), ctypes.c_void_p, ctypes.c_int32, ctypes.c_double,
                                            ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]
    L.dspfe_zcr_rule_host.argtypes = [ctypes.POINTER(_EndpointParams), ctypes.c_void_p, ctypes.c_int32, ctypes.c_double,
                                      ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]
    L.dspfe_endpoint_robust.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int32,
                                        ctypes.c_void_p, ctypes.c_void_p]
    L.dspfe_endpoint_robust_host.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]
    L.dspfe_amplitude_rule_gated_host.argtypes = [ctypes.POINTER(_EndpointParams), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                                  ctypes.c_double, ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]
    L.dspfe_acr_gate_rows_f64.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    L._ep_bound = True


def endpoint_params(samplerate=16000, cfg_frame=0.03, cfg_step=0.01, **kw):
    L = lib()
    _bind_endpoint(L)
    p = _EndpointParams()
    L.dspfe_endpoint_params_default(ctypes.byref(p), int(samplerate))
    p.cfg_frame, p.cfg_step = float(cfg_frame), float(cfg_step)
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def endpoint_decide_host(asum, zcr, **kw):
    """Host-only replay of the decision rule (no CUDA) on per-frame sum|x| and zero-crossing counts."""
    p = endpoint_params(**kw)
    asum = np.ascontiguousarray(asum, dtype=np.int32)
    zcr = np.ascontiguousarray(zcr, dtype=np.int32)
    lr = np.zeros(2, dtype=np.int32)
    _check(lib().dspfe_endpoint_decide_host(ctypes.byref(p), asum.ctypes.data_as(ctypes.c_void_p),
                                            zcr.ctypes.data_as(ctypes.c_void_p), len(asum), lr.ctypes.data_as(ctypes.c_void_p)))
    return int(lr[0]), int(lr[1])


def amplitude_rule_host(amp, mh=0.25, **kw):
    """amplitude_rule on a float64 list: returns the reference's list of (j, k) segments."""
    p = endpoint_params(**kw)
    amp = np.ascontiguousarray(amp, dtype=np.float64)
    segs = np.zeros((max(len(amp), 1), 2), dtype=np.int32)
    n = ctypes.c_int32(0)
    _check(lib().dspfe_amplitude_rule_host(ctypes.byref(p), amp.ctypes.data_as(ctypes.c_void_p), len(amp), float(mh),
                                           segs.ctypes.data_as(ctypes.c_void_p), len(segs), ctypes.byref(n)))
    return [(int(j), int(k)) for j, k in segs[: n.value]]


def zcr_rule_host(zcr, left, right, l_sil=0.0, **kw):
    p = endpoint_params(**kw)
    zcr = np.ascontiguousarray(zcr, dtype=np.float64)
    jk = np.zeros(2, dtype=np.int32)
    _check(lib().dspfe_zcr_rule_host(ctypes.byref(p), zcr.ctypes.data_as(ctypes.c_void_p), len(zcr), float(l_sil), int(left),
                                     int(right), jk.ctypes.data_as(ctypes.c_void_p)))
    return int(jk[0]), int(jk[1])


class EndpointPlan:
    """dspfe_endpoint_plan: batched basic_endpoint_detection (reference endpoint.py:34)."""

    def __init__(self, **kw):
        self._p = endpoint_params(**kw)
        h = ctypes.c_void_p()
        _check(lib().dspfe_endpoint_create(ctypes.byref(self._p), ctypes.byref(h)))
        self._h = h
        self.frame_len = int(lib().dspfe_endpoint_frame_len(h))
        self.frame_step = int(lib().dspfe_endpoint_frame_step(h))

    def close(self):
        if getattr(self, "_h", None):
            lib().dspfe_endpoint_destroy(self._h)
            self._h = None

    __del__ = close

    def frames_bound(self, total_samples, n_utt):
        return int(lib().dspfe_endpoint_frames_bound(self._h, int(total_samples), int(n_utt)))

    def reserve(self, max_utt, max_total_samples):
        L = lib()
        L.dspfe_endpoint_reserve.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]
        _check(L.dspfe_endpoint_reserve(self._h, int(max_utt), int(max_total_samples)))

    def detect(self, pcm, offsets, want_features=False, stream=None):
        """Device path: pcm int16 CUDA tensor, offsets int64 CUDA tensor [U+1].  Returns lr int32 [U,2]
        (and asum, zcr int32 [frames_bound], frame_off int64 [U+1] when want_features)."""
        import torch
        assert pcm.is_cuda and pcm.dtype == torch.int16 and offsets.is_cuda and offsets.dtype == torch.int64
        n_utt = offsets.numel() - 1
        lr = torch.empty((n_utt, 2), dtype=torch.int32, device=pcm.device)
        st = stream if stream is not None else torch.cuda.current_stream(pcm.device).cuda_stream
        if want_features:
            fb = self.frames_bound(pcm.numel(), n_utt)
            asum = torch.empty(fb, dtype=torch.int32, device=pcm.device)
            zcr = torch.empty(fb, dtype=torch.int32, device=pcm.device)
            fo = torch.empty(n_utt + 1, dtype=torch.int64, device=pcm.device)
            _check(lib().dspfe_endpoint(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), n_utt, lr.data_ptr(),
                                        asum.data_ptr(), zcr.data_ptr(), fo.data_ptr(), fb, ctypes.c_void_p(st)))
            return lr, asum, zcr, fo
        _check(lib().dspfe_endpoint(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), n_utt, lr.data_ptr(),
                                    None, None, None, 0, ctypes.c_void_p(st)))
        return lr

    def detect_robust(self, pcm, offsets, stream=None):
        """robust_endpoint_detection (reference endpoint.py:68) on device tensors: lr int32 [U,2]."""
        import torch
        assert pcm.is_cuda and pcm.dtype == torch.int16 and offsets.is_cuda and offsets.dtype == torch.int64
        n_utt = offsets.numel() - 1
        lr = torch.empty((n_utt, 2), dtype=torch.int32, device=pcm.device)
        st = stream if stream is not None else torch.cuda.current_stream(pcm.device).cuda_stream
        _check(lib().dspfe_endpoint_robust(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), n_utt, lr.data_ptr(), ctypes.c_void_p(st)))
        return lr

    def detect_robust_host(self, pcm, offsets):
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        lr = np.zeros((len(offsets) - 1, 2), dtype=np.int32)
        _check(lib().dspfe_endpoint_robust_host(self._h, pcm.ctypes.data_as(ctypes.c_void_p), offsets.ctypes.data_as(ctypes.c_void_p),
                                                len(offsets) - 1, lr.ctypes.data_as(ctypes.c_void_p)))
        return lr

    def detect_host(self, pcm, offsets, want_features=False):
        """Host path: NumPy int16 pcm + int64 offsets -> lr int32 [U,2] (+ asum, zcr, frame_off)."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n_utt = len(offsets) - 1
        lr = np.zeros((n_utt, 2), dtype=np.int32)
        if not want_features:
            _check(lib().dspfe_endpoint_host(self._h, pcm.ctypes.data_as(ctypes.c_void_p), offsets.ctypes.data_as(ctypes.c_void_p),
                                             n_utt, lr.ctypes.data_as(ctypes.c_void_p), None, None, None))
            return lr
        nf = int(frame_counts(np.diff(offsets), self.frame_len, self.frame_step).sum())
        asum = np.zeros(nf, dtype=np.int32)
        zcr = np.zeros(nf, dtype=np.int32)
        fo = np.zeros(n_utt + 1, dtype=np.int64)
        _check(lib().dspfe_endpoint_host(self._h, pcm.ctypes.data_as(ctypes.c_void_p), offsets.ctypes.data_as(ctypes.c_void_p),
                                         n_utt, lr.ctypes.data_as(ctypes.c_void_p), asum.ctypes.data_as(ctypes.c_void_p),
                                         zcr.ctypes.data_as(ctypes.c_void_p), fo.ctypes.data_as(ctypes.c_void_p)))
        return lr, asum, zcr, fo

    def detect_f32(self, pcm, offsets, want_features=False, stream=None):
        """Device path on float32 samples (dspfe_endpoint_f32): pcm float32 CUDA tensor, offsets int64 CUDA tensor [U+1].
        Returns lr int32 [U,2] (and amp float64, zcr int32 [frames_bound], frame_off int64 [U+1] when want_features)."""
        import torch
        L = lib(); _bind_endpoint_f32(L)
        assert pcm.is_cuda and pcm.dtype == torch.float32 and pcm.is_contiguous()
        assert offsets.is_cuda and offsets.dtype == torch.int64
        n_utt = offsets.numel() - 1
        lr = torch.empty((n_utt, 2), dtype=torch.int32, device=pcm.device)
        st = ctypes.c_void_p(stream if stream is not None else torch.cuda.current_stream(pcm.device).cuda_stream)
        if not want_features:
            _check(L.dspfe_endpoint_f32(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), n_utt, lr.data_ptr(),
                                        None, None, None, 0, st))
            return lr
        fb = self.frames_bound(pcm.numel(), n_utt)
        amp = torch.empty(fb, dtype=torch.float64, device=pcm.device)
        zcr = torch.empty(fb, dtype=torch.int32, device=pcm.device)
        fo = torch.empty(n_utt + 1, dtype=torch.int64, device=pcm.device)
        _check(L.dspfe_endpoint_f32(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), n_utt, lr.data_ptr(),
                                    amp.data_ptr(), zcr.data_ptr(), fo.data_ptr(), fb, st))
        return lr, amp, zcr, fo

    def detect_host_f32(self, pcm, offsets, want_features=False):
        """Host path on float32 samples: NumPy float32 pcm + int64 offsets -> lr int32 [U,2] (+ amp float64, zcr, frame_off)."""
        L = lib(); _bind_endpoint_f32(L)
        pcm = np.ascontiguousarray(pcm, dtype=np.float32)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n_utt = len(offsets) - 1
        lr = np.zeros((n_utt, 2), dtype=np.int32)
        if not want_features:
            _check(L.dspfe_endpoint_host_f32(self._h, _np_ptr(pcm), _np_ptr(offsets), n_utt, _np_ptr(lr), None, None, None))
            return lr
        nf = int(frame_counts(np.diff(offsets), self.frame_len, self.frame_step).sum())
        amp = np.zeros(nf, dtype=np.float64)
        zcr = np.zeros(nf, dtype=np.int32)
        fo = np.zeros(n_utt + 1, dtype=np.int64)
        _check(L.dspfe_endpoint_host_f32(self._h, _np_ptr(pcm), _np_ptr(offsets), n_utt, _np_ptr(lr), _np_ptr(amp), _np_ptr(zcr),
                                         _np_ptr(fo)))
        return lr, amp, zcr, fo

    def detect_robust_f32(self, pcm, offsets, stream=None):
        """robust_endpoint_detection (reference endpoint.py:68) on float32 samples (dspfe_endpoint_robust_f32): pcm float32 CUDA
        tensor, offsets int64 CUDA tensor [U+1].  Returns lr int32 [U,2]."""
        import torch
        L = lib(); _bind_endpoint_f32(L)
        assert pcm.is_cuda and pcm.dtype == torch.float32 and pcm.is_contiguous()
        assert offsets.is_cuda and offsets.dtype == torch.int64
        n_utt = offsets.numel() - 1
        lr = torch.empty((n_utt, 2), dtype=torch.int32, device=pcm.device)
        st = ctypes.c_void_p(stream if stream is not None else torch.cuda.current_stream(pcm.device).cuda_stream)
        _check(L.dspfe_endpoint_robust_f32(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), n_utt, lr.data_ptr(), st))
        return lr

    def detect_robust_host_f32(self, pcm, offsets):
        """Host form of detect_robust_f32: NumPy float32 pcm + int64 offsets -> lr int32 [U,2]."""
        L = lib(); _bind_endpoint_f32(L)
        pcm = np.ascontiguousarray(pcm, dtype=np.float32)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        lr = np.zeros((len(offsets) - 1, 2), dtype=np.int32)
        _check(L.dspfe_endpoint_robust_host_f32(self._h, _np_ptr(pcm), _np_ptr(offsets), len(offsets) - 1, _np_ptr(lr)))
        return lr


def _bind_endpoint_f32(L):
    if getattr(L, "_ep_f32_bound", False):
        return
    vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32
    L.dspfe_endpoint_f32.argtypes = [vp, vp, i64, vp, i32, vp, vp, vp, vp, i64, vp]
    L.dspfe_endpoint_host_f32.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    L.dspfe_endpoint_robust_f32.argtypes = [vp, vp, i64, vp, i32, vp, vp]
    L.dspfe_endpoint_robust_host_f32.argtypes = [vp, vp, vp, i32, vp]
    L._ep_f32_bound = True


# ------------------------------------------------------------------------------------------------ taps + helpers
def _bind_helpers(L):
    if getattr(L, "_h_bound", False):
        return
    vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32
    L.dspfe_mfcc_delta_f32.argtypes = [vp, vp, i64, vp, vp, i32, vp, i64, vp, vp]
    L.dspfe_fbank_f32.argtypes = [vp, vp, i64, vp, i32, vp, i64, vp, vp]
    L.dspfe_spectrum_f32.argtypes = [vp, vp, i64, vp, i32, i32, vp, i64, vp, vp]
    L.dspfe_frames_f64.argtypes = [vp, i64, i32, i32, vp, vp, i64, vp]
    L.dspfe_preemphasis_f64.argtypes = [vp, i64, ctypes.c_double, vp, vp]
    L.dspfe_row_amplitude_f64.argtypes = [vp, i64, i32, i32, vp, vp]
    L.dspfe_row_zcr_f64.argtypes = [vp, i64, i32, vp, vp]
    L.dspfe_row_windowed_amplitude_f64.argtypes = [vp, i64, i32, vp, i32, i32, vp, vp]
    L.dspfe_delta_f32.argtypes = [vp, i64, i32, i32, vp, vp]
    L.dspfe_cmvn_pad_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp]
    L.dspfe_fir_window_f64.argtypes = [vp, i32, ctypes.c_double, ctypes.c_double, ctypes.c_double, i32, vp, vp]
    L.dspfe_acr_f64.argtypes = [vp, i32, i32, vp, vp]
    L._h_bound = True


def _cuda():
    import torch
    if not torch.cuda.is_available():
        raise DspfeError(-3, "no CUDA device: libdspfe has no CPU fallback")
    return torch, torch.device("cuda", torch.cuda.current_device())


def _stream(torch, dev):
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _mfcc_f32(self, pcm, offsets, trim=None):
    """float32-sample variant of MfccPlan.mfcc_delta (device tensors)."""
    import torch
    L = lib(); _bind_helpers(L)
    assert pcm.is_cuda and pcm.dtype == torch.float32 and pcm.is_contiguous()
    n_utt = offsets.numel() - 1
    rows = self.rows_bound(pcm.numel(), n_utt)
    out = torch.empty((rows, self.width), dtype=torch.float32, device=pcm.device)
    fo = torch.empty(n_utt + 1, dtype=torch.int64, device=pcm.device)
    tp = None if trim is None else trim.data_ptr()
    _check(L.dspfe_mfcc_delta_f32(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), tp, n_utt, out.data_ptr(), rows,
                                  fo.data_ptr(), _stream(torch, pcm.device)))
    return out, fo


def _fbank_f32(self, pcm, offsets):
    """[rows, nfilt+1] float32: filterbank energies and the frame energy (reference base.fbank)."""
    import torch
    L = lib(); _bind_helpers(L)
    assert pcm.is_cuda and pcm.dtype == torch.float32 and pcm.is_contiguous()
    n_utt = offsets.numel() - 1
    rows = self.rows_bound(pcm.numel(), n_utt)
    out = torch.empty((rows, self._p.nfilt + 1), dtype=torch.float32, device=pcm.device)
    fo = torch.empty(n_utt + 1, dtype=torch.int64, device=pcm.device)
    _check(L.dspfe_fbank_f32(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), n_utt, out.data_ptr(), rows, fo.data_ptr(),
                             _stream(torch, pcm.device)))
    return out, fo


def _spectrum_f32(self, pcm, offsets, kind=0):
    """[rows, 257] float32: kind 0 power, 1 magnitude, 2 10*log10(power) (reference sigproc.powspec/magspec/logpowspec)."""
    import torch
    L = lib(); _bind_helpers(L)
    assert pcm.is_cuda and pcm.dtype == torch.float32 and pcm.is_contiguous()
    n_utt = offsets.numel() - 1
    rows = self.rows_bound(pcm.numel(), n_utt)
    out = torch.empty((rows, self._p.nfft // 2 + 1), dtype=torch.float32, device=pcm.device)
    fo = torch.empty(n_utt + 1, dtype=torch.int64, device=pcm.device)
    _check(L.dspfe_spectrum_f32(self._h, pcm.data_ptr(), pcm.numel(), offsets.data_ptr(), n_utt, int(kind), out.data_ptr(), rows,
                                fo.data_ptr(), _stream(torch, pcm.device)))
    return out, fo


MfccPlan.mfcc_delta_f32 = _mfcc_f32
MfccPlan.fbank_f32 = _fbank_f32
MfccPlan.spectrum_f32 = _spectrum_f32


def frames_f64(sig, frame_len, frame_step, win=None):
    """framesig on the device: NumPy 1-D signal -> float64 [n_frames, frame_len]."""
    torch, dev = _cuda()
    L = lib(); _bind_helpers(L)
    x = torch.from_numpy(np.ascontiguousarray(sig, dtype=np.float64)).to(dev)
    nf = num_frames(x.numel(), frame_len, frame_step)
    w = None if win is None else torch.from_numpy(np.ascontiguousarray(win, dtype=np.float64)).to(dev)
    out = torch.empty((nf, frame_len), dtype=torch.float64, device=dev)
    _check(L.dspfe_frames_f64(x.data_ptr(), x.numel(), int(frame_len), int(frame_step), None if w is None else w.data_ptr(),
                              out.data_ptr(), nf, _stream(torch, dev)))
    return out.cpu().numpy()


def preemphasis_f64(x, coeff):
    torch, dev = _cuda()
    L = lib(); _bind_helpers(L)
    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(dev)
    y = torch.empty_like(xd)
    _check(L.dspfe_preemphasis_f64(xd.data_ptr(), xd.numel(), float(coeff), y.data_ptr(), _stream(torch, dev)))
    return y.cpu().numpy()


def row_amplitude_f64(frames, use_sq=False):   # use_sq: False mean|x|, True mean x^2, 2 plain sum|x|
    torch, dev = _cuda()
    L = lib(); _bind_helpers(L)
    f = torch.from_numpy(np.ascontiguousarray(frames, dtype=np.float64)).to(dev)
    out = torch.empty(f.shape[0], dtype=torch.float64, device=dev)
    _check(L.dspfe_row_amplitude_f64(f.data_ptr(), f.shape[0], f.shape[1], (2 if use_sq == 2 else int(bool(use_sq))), out.data_ptr(), _stream(torch, dev)))
    return out.cpu().numpy()


def row_windowed_amplitude_f64(frames, window, use_sq=False):
    """get_amplitude(frames, window=<taps>, use_sq) on the device (mean of the 'same' convolution per row)."""
    torch, dev = _cuda()
    L = lib(); _bind_helpers(L)
    f = torch.from_numpy(np.ascontiguousarray(frames, dtype=np.float64)).to(dev)
    w = np.ascontiguousarray(window, dtype=np.float64)
    out = torch.empty(f.shape[0], dtype=torch.float64, device=dev)
    _check(L.dspfe_row_windowed_amplitude_f64(f.data_ptr(), f.shape[0], f.shape[1], _np_ptr(w), len(w), int(bool(use_sq)), out.data_ptr(),
                                              _stream(torch, dev)))
    return out.cpu().numpy()


def row_zcr_f64(frames):
    torch, dev = _cuda()
    L = lib(); _bind_helpers(L)
    f = torch.from_numpy(np.ascontiguousarray(frames, dtype=np.float64)).to(dev)
    out = torch.empty(f.shape[0], dtype=torch.int64, device=dev)
    _check(L.dspfe_row_zcr_f64(f.data_ptr(), f.shape[0], f.shape[1], out.data_ptr(), _stream(torch, dev)))
    return out.cpu().numpy()


def delta_f32(feat, N):
    torch, dev = _cuda()
    L = lib(); _bind_helpers(L)
    f = torch.from_numpy(np.ascontiguousarray(feat, dtype=np.float32)).to(dev)
    out = torch.empty_like(f)
    _check(L.dspfe_delta_f32(f.data_ptr(), f.shape[0], f.shape[1], int(N), out.data_ptr(), _stream(torch, dev)))
    return out.cpu().numpy()


# ------------------------------------------------------------------------------------------------ pitch
class _PitchParams(ctypes.Structure):
    _fields_ = [("samplerate", ctypes.c_int32), ("dst_rate", ctypes.c_int32), ("frame_len", ctypes.c_int32),
                ("frame_step", ctypes.c_int32), ("method", ctypes.c_int32), ("center_clip", ctypes.c_int32),
                ("row_len", ctypes.c_int32), ("reserved", ctypes.c_int32), ("band_lo", ctypes.c_double),
                ("band_hi", ctypes.c_double), ("preemph", ctypes.c_double)]


def _bind_pitch(L):
    if getattr(L, "_p_bound", False):
        return
    vp, i64, i32, f64 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_double
    L.dspfe_pitch_params_default.argtypes = [ctypes.POINTER(_PitchParams), i32]
    L.dspfe_pitch_params_default.restype = None
    L.dspfe_pitch_create.argtypes = [ctypes.POINTER(_PitchParams), ctypes.POINTER(vp)]
    L.dspfe_pitch_destroy.argtypes = [vp]
    L.dspfe_pitch_destroy.restype = None
    L.dspfe_pitch_row_len.argtypes = [vp]
    L.dspfe_pitch_num_frames.argtypes = [vp, i64]
    L.dspfe_pitch_num_frames.restype = i64
    L.dspfe_pitch_frames_bound.argtypes = [vp, i64, i64]
    L.dspfe_pitch_frames_bound.restype = i64
    L.dspfe_pitch.argtypes = [vp, vp, i32, i64, vp, vp, i32, vp, vp, vp, vp, vp, i64, vp]
    L.dspfe_pitch_host.argtypes = [vp, vp, i32, vp, vp, i32, vp, vp, vp, vp]
    L.dspfe_center_clip_f32.argtypes = [vp, i64, i32, i32, vp, vp]
    L.dspfe_track_rows_f32.argtypes = [vp, i64, i32, i32, i32, vp, vp, vp, vp]
    L.dspfe_robust_max_pitch_host.argtypes = [vp, i32, i32, vp]
    L.dspfe_smooth_subsequence_host.argtypes = [vp, i32, i32, f64, vp, ctypes.POINTER(i32), ctypes.POINTER(i32), ctypes.POINTER(i32)]
    L.dspfe_sub_endpoint_host.argtypes = [vp, i32, ctypes.POINTER(i32)]
    L.dspfe_pitch_feature_tail_host.argtypes = [vp, vp, i32, vp]
    L.dspfe_poly_lead_host.argtypes = [vp, i32, i32, ctypes.POINTER(f64)]
    L.dspfe_dp_max_pitch_host.argtypes = [vp, i32, i32, vp]
    L._p_bound = True


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


class PitchPlan:
    """dspfe_pitch_plan: batched pitch_detect (method 0) / pitch_detect_sr (method 1) / pitch_feature
    (reference pitch.py:83, :96, :26)."""

    def __init__(self, method=0, samplerate=16000, dst_rate=10000, frame_len=512, frame_step=100, center_clip=True,
                 row_len=0, band_lo=50.0, band_hi=None, preemph=0.0):
        L = lib(); _bind_pitch(L)
        p = _PitchParams()
        L.dspfe_pitch_params_default(ctypes.byref(p), int(method))
        p.samplerate, p.dst_rate, p.frame_len, p.frame_step = int(samplerate), int(dst_rate), int(frame_len), int(frame_step)
        p.center_clip, p.row_len, p.band_lo, p.preemph = int(bool(center_clip)), int(row_len), float(band_lo), float(preemph)
        if band_hi is not None:
            p.band_hi = float(band_hi)
        self._p = p
        h = ctypes.c_void_p()
        _check(L.dspfe_pitch_create(ctypes.byref(p), ctypes.byref(h)))
        self._h = h
        self.method = int(method)
        self.row_len = int(L.dspfe_pitch_row_len(h))

    def close(self):
        if getattr(self, "_h", None):
            lib().dspfe_pitch_destroy(self._h)
            self._h = None

    __del__ = close

    def frames_bound(self, total_samples, n_utt):
        return int(lib().dspfe_pitch_frames_bound(self._h, int(total_samples), int(n_utt)))

    def reserve(self, max_utt, max_total_samples):
        L = lib()
        L.dspfe_pitch_reserve.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]
        _check(L.dspfe_pitch_reserve(self._h, int(max_utt), int(max_total_samples)))

    def num_frames(self, n_samples):
        return int(lib().dspfe_pitch_num_frames(self._h, int(n_samples)))

    def detect(self, pcm, offsets, trim=None, want_feat=False, want_rows=False, want_track=True, out=None, stream=None):
        """Device path: pcm int16 or float32 CUDA tensor, offsets int64 CUDA tensor [U+1], optional trim int32 [U,2].
        Returns a dict of CUDA tensors: pitch float64 [bound], lag int32 [bound], frame_off int64 [U+1]
        (+ feat float64 [U,5], rows float32 [bound,row_len]); entries beyond frame_off[-1] are untouched.
        `out` may carry preallocated tensors under the same keys."""
        import torch
        assert pcm.is_cuda and pcm.dtype in (torch.int16, torch.float32) and pcm.is_contiguous()
        assert offsets.is_cuda and offsets.dtype == torch.int64 and offsets.is_contiguous()
        n_utt = offsets.numel() - 1
        fb = self.frames_bound(pcm.numel(), n_utt)
        dev = pcm.device
        o = dict(out or {})
        if want_track and o.get("pitch") is None:
            o["pitch"] = torch.empty(fb, dtype=torch.float64, device=dev)
        if want_track and o.get("lag") is None:
            o["lag"] = torch.empty(fb, dtype=torch.int32, device=dev)
        if o.get("frame_off") is None:
            o["frame_off"] = torch.empty(n_utt + 1, dtype=torch.int64, device=dev)
        if want_feat and o.get("feat") is None:
            o["feat"] = torch.empty((n_utt, 5), dtype=torch.float64, device=dev)
        if want_rows and o.get("rows") is None:
            o["rows"] = torch.empty((fb, self.row_len), dtype=torch.float32, device=dev)
        tp = None
        if trim is not None:
            assert trim.is_cuda and trim.dtype == torch.int32 and trim.is_contiguous() and trim.shape == (n_utt, 2)
            tp = trim.data_ptr()
        ptr = lambda k: o[k].data_ptr() if o.get(k) is not None else None
        st = stream if stream is not None else torch.cuda.current_stream(dev).cuda_stream
        _check(lib().dspfe_pitch(self._h, pcm.data_ptr(), int(pcm.dtype == torch.float32), pcm.numel(), offsets.data_ptr(), tp, n_utt,
                                 ptr("pitch"), ptr("lag"), ptr("feat") if want_feat else None, ptr("rows") if want_rows else None,
                                 ptr("frame_off"), fb, ctypes.c_void_p(st)))
        return o

    def detect_host(self, pcm, offsets, trim=None, want_feat=False):
        """Host path: NumPy int16 / float32 pcm + int64 offsets (+ int32 trim [U,2]) ->
        (pitch float64 [F], lag int32 [F], frame_off int64 [U+1][, feat float64 [U,5]])."""
        pcm = np.ascontiguousarray(pcm)
        if pcm.dtype != np.int16:
            pcm = pcm.astype(np.float32, copy=False)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n_utt = len(offsets) - 1
        lens = np.diff(offsets)
        if trim is not None:
            trim = np.ascontiguousarray(trim, dtype=np.int32).reshape(n_utt, 2)
            l = np.clip(trim[:, 0].astype(np.int64), 0, lens); r = np.clip(trim[:, 1].astype(np.int64), 0, lens)
            lens = np.maximum(r - l, 0)
        nf = int(sum(self.num_frames(int(n)) for n in lens))
        pitch = np.zeros(nf, dtype=np.float64)
        lag = np.zeros(nf, dtype=np.int32)
        fo = np.zeros(n_utt + 1, dtype=np.int64)
        feat = np.zeros((n_utt, 5), dtype=np.float64) if want_feat else None
        _check(lib().dspfe_pitch_host(self._h, _np_ptr(pcm), int(pcm.dtype == np.float32), _np_ptr(offsets), _np_ptr(trim), n_utt,
                                      _np_ptr(pitch), _np_ptr(lag), _np_ptr(feat), _np_ptr(fo)))
        return (pitch, lag, fo, feat) if want_feat else (pitch, lag, fo)


def center_clip_f32(rows, binary=True):
    """center_clip (reference pitch.py:145) on [n_rows, len<=512] (or one 1-D frame), on the device."""
    torch, dev = _cuda()
    L = lib(); _bind_pitch(L)
    a = np.ascontiguousarray(rows, dtype=np.float32)
    one = a.ndim == 1
    a2 = a.reshape(1, -1) if one else a
    x = torch.from_numpy(a2).to(dev)
    out = torch.empty_like(x)
    _check(L.dspfe_center_clip_f32(x.data_ptr(), x.shape[0], x.shape[1], int(bool(binary)), out.data_ptr(), _stream(torch, dev)))
    r = out.cpu().numpy()
    return r[0] if one else r


def smooth_rows_f32(rows, mode=0, want_score=False, want_lag=False, do_smooth=True):
    """smooth(g, 2) (reference pitch.py:157) on [n_rows, row_len<=512] float32 on the device; optionally the
    peak_score rows [n_rows, 80] (mode 0) and lag = 20 + first argmax.  Returns (smoothed, score|None, lag|None).
    do_smooth=False scores the rows as given (peak_score alone)."""
    torch, dev = _cuda()
    L = lib(); _bind_pitch(L)
    x = torch.from_numpy(np.ascontiguousarray(rows, dtype=np.float32)).to(dev)
    assert x.dim() == 2
    sm = torch.empty_like(x)
    sc = torch.empty((x.shape[0], 80), dtype=torch.int32, device=dev) if want_score else None
    lg = torch.empty(x.shape[0], dtype=torch.int32, device=dev) if want_lag else None
    _check(L.dspfe_track_rows_f32(x.data_ptr(), x.shape[0], x.shape[1], int(mode), int(bool(do_smooth)), sm.data_ptr(),
                                   None if sc is None else sc.data_ptr(), None if lg is None else lg.data_ptr(), _stream(torch, dev)))
    return sm.cpu().numpy(), None if sc is None else sc.cpu().numpy(), None if lg is None else lg.cpu().numpy()


def robust_max_pitch_host(lags, repair=True):
    """max_pitch / robust_max_pitch (reference pitch.py:166, :191) on integer lags (bias already added)."""
    L = lib(); _bind_pitch(L)
    lags = np.ascontiguousarray(lags, dtype=np.int32)
    out = np.zeros(len(lags), dtype=np.float64)
    _check(L.dspfe_robust_max_pitch_host(_np_ptr(lags), len(lags), int(bool(repair)), _np_ptr(out)))
    return out


def smooth_subsequence_host(pitch, tor=3, thres=30.0):
    """find_smooth_subsequence (reference pitch.py:245): returns (values list, (i0, j0))."""
    L = lib(); _bind_pitch(L)
    pitch = np.ascontiguousarray(pitch, dtype=np.float64)
    seg = np.zeros(len(pitch), dtype=np.float64)
    n, i0, j0 = ctypes.c_int32(0), ctypes.c_int32(0), ctypes.c_int32(0)
    _check(L.dspfe_smooth_subsequence_host(_np_ptr(pitch), len(pitch), int(tor), float(thres), _np_ptr(seg), ctypes.byref(n),
                                           ctypes.byref(i0), ctypes.byref(j0)))
    return seg[: n.value], (i0.value, j0.value)


def sub_endpoint_host(amp):
    L = lib(); _bind_pitch(L)
    amp = np.ascontiguousarray(amp, dtype=np.float64)
    p = ctypes.c_int32(0)
    _check(L.dspfe_sub_endpoint_host(_np_ptr(amp), len(amp), ctypes.byref(p)))
    return p.value


def pitch_feature_tail_host(pitch, amp):
    L = lib(); _bind_pitch(L)
    pitch = np.ascontiguousarray(pitch, dtype=np.float64)
    amp = np.ascontiguousarray(amp, dtype=np.float64)
    out = np.zeros(5, dtype=np.float64)
    _check(L.dspfe_pitch_feature_tail_host(_np_ptr(pitch), _np_ptr(amp), len(pitch), _np_ptr(out)))
    return out


def poly_lead_host(seq, deg):
    L = lib(); _bind_pitch(L)
    seq = np.ascontiguousarray(seq, dtype=np.float64)
    c = ctypes.c_double(0.0)
    _check(L.dspfe_poly_lead_host(_np_ptr(seq), len(seq), int(deg), ctypes.byref(c)))
    return c.value


def dp_max_pitch_host(g):
    """dp_max_pitch (reference pitch.py:208-225) on a [n_rows, n_cols] score array."""
    L = lib(); _bind_pitch(L)
    g = np.ascontiguousarray(g, dtype=np.float64)
    out = np.zeros(g.shape[0], dtype=np.float64)
    _check(L.dspfe_dp_max_pitch_host(_np_ptr(g), g.shape[0], g.shape[1], _np_ptr(out)))
    return out


def dp_max_pitch_f64(g):
    """dp_max_pitch (reference pitch.py:208-225) on the device (dspfe_dp_max_pitch): [n_rows] float64."""
    torch, dev = _cuda()
    L = lib(); _bind_pitch(L)
    L.dspfe_dp_max_pitch.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    x = torch.from_numpy(np.ascontiguousarray(g, dtype=np.float64)).to(dev)
    out = torch.empty(x.shape[0], dtype=torch.float64, device=dev)
    _check(L.dspfe_dp_max_pitch(x.data_ptr(), x.shape[0], x.shape[1], out.data_ptr(), _stream(torch, dev)))
    return out.cpu().numpy()


def fir_window_f64(sig, rate, low_freq, high_freq, hamming):
    """window (reference sigproc.py:22-46) on the device: complex128 [n]."""
    torch, dev = _cuda()
    L = lib(); _bind_helpers(L)
    x = torch.from_numpy(np.ascontiguousarray(sig, dtype=np.float64)).to(dev)
    y = torch.empty((x.numel(), 2), dtype=torch.float64, device=dev)
    _check(L.dspfe_fir_window_f64(x.data_ptr(), x.numel(), float(rate), float(low_freq), float(high_freq), int(bool(hamming)),
                                  y.data_ptr(), _stream(torch, dev)))
    r = y.cpu().numpy()
    return r[:, 0] + 1j * r[:, 1]


def acr_f64(frame, n):
    """acr (reference sigproc.py:48-53) on the device."""
    torch, dev = _cuda()
    L = lib(); _bind_helpers(L)
    x = torch.from_numpy(np.ascontiguousarray(frame, dtype=np.float64)).to(dev)
    out = torch.empty(1, dtype=torch.float64, device=dev)
    _check(L.dspfe_acr_f64(x.data_ptr(), x.numel(), int(n), out.data_ptr(), _stream(torch, dev)))
    return np.float64(out.cpu().numpy()[0])


def cmvn_pad_batch(feat, frame_off, numcep=13, T=200, out=None):
    """The reference trainer's batching epilogue (model.py:75-88, :35-50, :131-135) on device tensors: feat float32
    [rows, 3*numcep] and frame_off int64 [U+1] as written by MfccPlan.mfcc_delta.  Returns (inp float32 [T, U, 3*numcep],
    len0 int32 [U])."""
    import torch
    L = lib(); _bind_helpers(L)
    assert feat.is_cuda and feat.dtype == torch.float32 and feat.is_contiguous() and feat.shape[1] == 3 * numcep
    n_utt = frame_off.numel() - 1
    if out is None:
        out = torch.empty((T, n_utt, 3 * numcep), dtype=torch.float32, device=feat.device)
    len0 = torch.empty(n_utt, dtype=torch.int32, device=feat.device)
    _check(L.dspfe_cmvn_pad_batch(feat.data_ptr(), frame_off.data_ptr(), n_utt, int(numcep), int(T), out.data_ptr(), len0.data_ptr(),
                                  _stream(torch, feat.device)))
    return out, len0


def amplitude_rule_gated_host(amp, gate, mh=0.25, **kw):
    """amplitude_rule(use_acr=True) on a float64 list and the per-frame acr_rule flags."""
    p = endpoint_params(**kw)
    amp = np.ascontiguousarray(amp, dtype=np.float64)
    gate = np.ascontiguousarray(gate, dtype=np.int32)
    segs = np.zeros((max(len(amp), 1), 2), dtype=np.int32)
    n = ctypes.c_int32(0)
    _check(lib().dspfe_amplitude_rule_gated_host(ctypes.byref(p), _np_ptr(amp), _np_ptr(gate), len(amp), float(mh), _np_ptr(segs),
                                                 len(segs), ctypes.byref(n)))
    return [(int(j), int(k)) for j, k in segs[: n.value]]


def acr_gate_rows_f64(frames, rate):
    """acr_rule (reference endpoint.py:142-144) of every row of a float64 frame matrix, on the device: int32 flags."""
    torch, dev = _cuda()
    L = lib(); _bind_endpoint(L)
    f = torch.from_numpy(np.ascontiguousarray(frames, dtype=np.float64)).to(dev)
    g = torch.empty(f.shape[0], dtype=torch.int32, device=dev)
    _check(L.dspfe_acr_gate_rows_f64(f.data_ptr(), f.shape[0], f.shape[1], int(rate), g.data_ptr(), _stream(torch, dev)))
    return g.cpu().numpy()


# ------------------------------------------------------------------------------------------------ ingest
def wav_info(data):
    """Header of one WAV file image (bytes): dict(rate, channels, bits, n_frames, data_offset).  Host only."""
    L = lib()
    L.dspfe_wav_info.argtypes = [ctypes.c_void_p, ctypes.c_int64] + [ctypes.POINTER(ctypes.c_int32)] * 3 + [ctypes.POINTER(ctypes.c_int64)] * 2
    buf = np.frombuffer(data, dtype=np.uint8)
    r, c, b = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    n, o = ctypes.c_int64(), ctypes.c_int64()
    _check(L.dspfe_wav_info(_np_ptr(buf), len(buf), ctypes.byref(r), ctypes.byref(c), ctypes.byref(b), ctypes.byref(n), ctypes.byref(o)))
    return dict(rate=r.value, channels=c.value, bits=b.value, n_frames=n.value, data_offset=o.value)


def wav_scan_paths(paths):
    """Headers only (host): (offsets int64 [n+1] in samples of channel 0, rates int32 [n])."""
    L = lib()
    L.dspfe_wav_scan_paths.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    n = len(paths)
    arr = (ctypes.c_char_p * max(n, 1))(*[os.fsencode(p) for p in paths])
    off = np.zeros(n + 1, dtype=np.int64)
    rates = np.zeros(max(n, 1), dtype=np.int32)
    _check(L.dspfe_wav_scan_paths(arr, n, _np_ptr(off), _np_ptr(rates)))
    return off, rates[:n]


def ingest_wavs(paths):
    """reader.py:67-85 for a list of files: (pcm int16 CUDA tensor [total], offsets int64 NumPy [n+1], rates int32 [n]).
    Channel 0 of every 16-bit PCM WAV file, packed back to back on the current device; the library reads the files."""
    torch, dev = _cuda()
    L = lib()
    L.dspfe_wav_scan_paths.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    L.dspfe_ingest_wav_paths.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                         ctypes.c_void_p]
    n = len(paths)
    arr = (ctypes.c_char_p * max(n, 1))(*[os.fsencode(p) for p in paths])
    off = np.zeros(n + 1, dtype=np.int64)
    rates = np.zeros(max(n, 1), dtype=np.int32)
    _check(L.dspfe_wav_scan_paths(arr, n, _np_ptr(off), _np_ptr(rates)))
    total = int(off[-1])
    pcm = torch.empty(max(total, 1), dtype=torch.int16, device=dev)
    _check(L.dspfe_ingest_wav_paths(arr, n, pcm.data_ptr(), pcm.numel(), _np_ptr(off), _np_ptr(rates), _stream(torch, dev)))
    return pcm[:total], off, rates[:n]


def pitch_num_frames_host(n_samples, samplerate=16000, dst_rate=10000, frame_len=512, frame_step=100, method=0):
    """(pitch frames, decimated length) of an n_samples utterance; host only, no device needed."""
    L = lib(); _bind_pitch(L)
    L.dspfe_pitch_num_frames_host.argtypes = [ctypes.POINTER(_PitchParams), ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)]
    L.dspfe_pitch_num_frames_host.restype = ctypes.c_int64
    p = _PitchParams()
    L.dspfe_pitch_params_default(ctypes.byref(p), int(method))
    p.samplerate, p.dst_rate, p.frame_len, p.frame_step = int(samplerate), int(dst_rate), int(frame_len), int(frame_step)
    ld = ctypes.c_int64(0)
    nf = L.dspfe_pitch_num_frames_host(ctypes.byref(p), int(n_samples), ctypes.byref(ld))
    if nf < 0:
        raise DspfeError(int(nf), L.dspfe_last_error().decode())
    return int(nf), int(ld.value)


# ---------------------------------------------------------------------------------------------- whole front-end
class _FrontendParams(ctypes.Structure):
    _fields_ = [("samplerate", ctypes.c_int32), ("delta_n", ctypes.c_int32), ("acr_frame_len", ctypes.c_int32),
                ("reserved", ctypes.c_int32), ("slab_samples", ctypes.c_int64), ("host_slab_samples", ctypes.c_int64),
                ("cep_preemph", ctypes.c_double)]


class _FrontendOut(ctypes.Structure):
    _fields_ = [("lr", ctypes.c_void_p), ("mfcc", ctypes.c_void_p), ("mfcc_cap", ctypes.c_int64), ("mfcc_frame_off", ctypes.c_void_p),
                ("cep_pitch", ctypes.c_void_p), ("cep_cap", ctypes.c_int64), ("cep_frame_off", ctypes.c_void_p),
                ("cep_feat", ctypes.c_void_p), ("acr_pitch", ctypes.c_void_p), ("acr_cap", ctypes.c_int64),
                ("acr_frame_off", ctypes.c_void_p), ("cep_lag", ctypes.c_void_p), ("acr_lag", ctypes.c_void_p)]


def _bind_frontend(L):
    if getattr(L, "_fe_bound", False):
        return
    vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32
    L.dspfe_frontend_params_default.argtypes = [ctypes.POINTER(_FrontendParams)]
    L.dspfe_frontend_params_default.restype = None
    L.dspfe_frontend_create.argtypes = [ctypes.POINTER(_FrontendParams), ctypes.POINTER(vp)]
    L.dspfe_frontend_destroy.argtypes = [vp]
    L.dspfe_frontend_destroy.restype = None
    L.dspfe_frontend_bounds.argtypes = [vp, i64, i64, vp]
    L.dspfe_frontend.argtypes = [vp, vp, vp, vp, i32, ctypes.POINTER(_FrontendOut), vp, vp]
    L.dspfe_frontend_host.argtypes = [vp, vp, vp, i32, ctypes.POINTER(_FrontendOut), vp]
    L.dspfe_frontend_f32.argtypes = [vp, vp, vp, vp, i32, ctypes.POINTER(_FrontendOut), vp, vp]
    L.dspfe_frontend_host_f32.argtypes = [vp, vp, vp, i32, ctypes.POINTER(_FrontendOut), vp]
    L.dspfe_timing_begin.argtypes = [vp]
    L.dspfe_timing_end.argtypes = [vp, vp, i32, ctypes.POINTER(i32)]
    L.dspfe_launch_count.restype = i64
    L._fe_bound = True


class FrontendPlan:
    """dspfe_frontend_plan: endpoints -> MFCC+delta+delta on sig[l:r] -> cepstrum pitch + pitch_feature on
    preemphasis(sig)[l:r] -> autocorrelation pitch on sig[l:r] for every utterance of a packed ragged batch
    (reference model.py:52-95, pitch_model.py:38-41), walked in slabs with bounded workspaces."""
    KEYS = ("lr", "mfcc", "mfcc_frame_off", "cep_pitch", "cep_frame_off", "cep_feat", "acr_pitch", "acr_frame_off", "cep_lag", "acr_lag")

    def __init__(self, samplerate=16000, delta_n=2, acr_frame_len=300, slab_samples=0, host_slab_samples=0, cep_preemph=0.97):
        L = lib(); _bind_endpoint(L); _bind_pitch(L); _bind_frontend(L)
        p = _FrontendParams()
        L.dspfe_frontend_params_default(ctypes.byref(p))
        p.samplerate, p.delta_n, p.acr_frame_len = int(samplerate), int(delta_n), int(acr_frame_len)
        p.slab_samples, p.host_slab_samples, p.cep_preemph = int(slab_samples), int(host_slab_samples), float(cep_preemph)
        h = ctypes.c_void_p()
        _check(L.dspfe_frontend_create(ctypes.byref(p), ctypes.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            lib().dspfe_frontend_destroy(self._h)
            self._h = None

    __del__ = close

    def bounds(self, total_samples, n_utt):
        """(MFCC rows, cepstrum frames, autocorrelation frames) capacities that hold any batch with these totals."""
        caps = (ctypes.c_int64 * 3)()
        _check(lib().dspfe_frontend_bounds(self._h, int(total_samples), int(n_utt), caps))
        return tuple(int(c) for c in caps)

    def alloc(self, total_samples, n_utt, device=None, pinned=False):
        """Output arrays for a batch: CUDA tensors on `device`, or NumPy arrays (over pinned torch storage if `pinned`)."""
        import torch
        c0, c1, c2 = self.bounds(total_samples, n_utt)
        shapes = dict(lr=((n_utt, 2), torch.int32), mfcc=((c0, 39), torch.float32), mfcc_frame_off=((n_utt + 1,), torch.int64),
                      cep_pitch=((c1,), torch.float64), cep_frame_off=((n_utt + 1,), torch.int64), cep_feat=((n_utt, 5), torch.float64),
                      acr_pitch=((c2,), torch.float64), acr_frame_off=((n_utt + 1,), torch.int64),
                      cep_lag=((c1,), torch.int32), acr_lag=((c2,), torch.int32))
        out = {}
        for k, (shape, dt) in shapes.items():
            if device is not None:
                out[k] = torch.empty(shape, dtype=dt, device=device)
            else:
                t = torch.empty(shape, dtype=dt)
                out[k] = t.pin_memory() if pinned else t
        return out

    @staticmethod
    def _out_struct(o, ptr):
        s = _FrontendOut()
        for k in FrontendPlan.KEYS:
            setattr(s, k, ptr(o[k]) if o.get(k) is not None else None)
        s.mfcc_cap = int(o["mfcc"].shape[0]) if o.get("mfcc") is not None else 0
        s.cep_cap = int(o["cep_pitch"].shape[0]) if o.get("cep_pitch") is not None else 0
        s.acr_cap = int(o["acr_pitch"].shape[0]) if o.get("acr_pitch") is not None else 0
        return s

    def run(self, pcm, offsets, h_offsets, out, stream=None):
        """Device path: pcm int16 CUDA tensor, offsets int64 CUDA tensor [U+1], h_offsets its NumPy copy, `out` from
        alloc(device=...).  Returns (MFCC rows, cepstrum frames, autocorrelation frames) written."""
        import torch
        assert pcm.is_cuda and pcm.dtype == torch.int16 and pcm.is_contiguous()
        assert offsets.is_cuda and offsets.dtype == torch.int64 and offsets.is_contiguous()
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.int64)
        n_utt = len(h_offsets) - 1
        s = self._out_struct(out, lambda t: t.data_ptr())
        tot = (ctypes.c_int64 * 3)()
        st = stream if stream is not None else torch.cuda.current_stream(pcm.device).cuda_stream
        _check(lib().dspfe_frontend(self._h, pcm.data_ptr(), offsets.data_ptr(), _np_ptr(h_offsets), n_utt, ctypes.byref(s), tot,
                                    ctypes.c_void_p(st)))
        return tuple(int(t) for t in tot)

    def run_host(self, pcm, offsets, out):
        """Host path: pcm int16 NumPy array (pinned memory makes the copies asynchronous), offsets int64 NumPy [U+1],
        `out` a dict of NumPy arrays / CPU tensors from alloc(device=None)."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n_utt = len(offsets) - 1
        s = self._out_struct(out, lambda t: t.data_ptr() if hasattr(t, "data_ptr") else t.ctypes.data)
        tot = (ctypes.c_int64 * 3)()
        _check(lib().dspfe_frontend_host(self._h, _np_ptr(pcm), _np_ptr(offsets), n_utt, ctypes.byref(s), tot))
        return tuple(int(t) for t in tot)

    def run_f32(self, pcm, offsets, h_offsets, out, stream=None):
        """run() on float32 samples (dspfe_frontend_f32): pcm float32 CUDA tensor, the rest as for run()."""
        import torch
        assert pcm.is_cuda and pcm.dtype == torch.float32 and pcm.is_contiguous()
        assert offsets.is_cuda and offsets.dtype == torch.int64 and offsets.is_contiguous()
        h_offsets = np.ascontiguousarray(h_offsets, dtype=np.int64)
        n_utt = len(h_offsets) - 1
        s = self._out_struct(out, lambda t: t.data_ptr())
        tot = (ctypes.c_int64 * 3)()
        st = stream if stream is not None else torch.cuda.current_stream(pcm.device).cuda_stream
        _check(lib().dspfe_frontend_f32(self._h, pcm.data_ptr(), offsets.data_ptr(), _np_ptr(h_offsets), n_utt, ctypes.byref(s), tot,
                                        ctypes.c_void_p(st)))
        return tuple(int(t) for t in tot)

    def run_host_f32(self, pcm, offsets, out):
        """run_host() on float32 samples (dspfe_frontend_host_f32): pcm float32 NumPy array, the rest as for run_host()."""
        pcm = np.ascontiguousarray(pcm, dtype=np.float32)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n_utt = len(offsets) - 1
        s = self._out_struct(out, lambda t: t.data_ptr() if hasattr(t, "data_ptr") else t.ctypes.data)
        tot = (ctypes.c_int64 * 3)()
        _check(lib().dspfe_frontend_host_f32(self._h, _np_ptr(pcm), _np_ptr(offsets), n_utt, ctypes.byref(s), tot))
        return tuple(int(t) for t in tot)


def timing_begin(stream=None):
    """Start bracketing every kernel the library launches on `stream` (default: torch's current stream) with CUDA events."""
    import torch
    L = lib(); _bind_frontend(L)
    st = stream if stream is not None else torch.cuda.current_stream().cuda_stream
    _check(L.dspfe_timing_begin(ctypes.c_void_p(st)))


def timing_end(cap=4096):
    """Waits for the stream and returns [(kernel name, ms), ...] in launch order."""
    L = lib(); _bind_frontend(L)
    names = ctypes.create_string_buffer(48 * cap)
    ms = (ctypes.c_float * cap)()
    n = ctypes.c_int32(0)
    _check(L.dspfe_timing_end(names, ms, cap, ctypes.byref(n)))
    k = min(n.value, cap)
    return [(names.raw[48 * i:48 * i + 48].split(b"\0", 1)[0].decode(), float(ms[i])) for i in range(k)]


def launch_count():
    L = lib(); _bind_frontend(L)
    return int(L.dspfe_launch_count())
