"""torch.library custom ops over the batched C-ABI entry points (SURVEY 8b: "each also registered as a torch.library
custom op taking CUDA tensors"; north_star: "thin C-ABI (ctypes / torch custom-op) layer").

    torch.ops.dspfe.endpoint(pcm, offsets, samplerate)                      -> lr int32 [U,2]            (endpoint.py:34)
                                                                            (int16 or float32 samples)
    torch.ops.dspfe.endpoint_robust(pcm, offsets, samplerate)               -> lr int32 [U,2]            (endpoint.py:68)
                                                                            (int16 or float32 samples)
    torch.ops.dspfe.mfcc_delta(pcm, offsets, trim, samplerate, frame_len, frame_step, nfft, delta_n, preemph, hamming)
                                                                            -> (rows float32 [bound,39], frame_off int64 [U+1])
                                                                                                         (base.py:8, :70; model.py:74-77)
    torch.ops.dspfe.pitch(pcm, offsets, trim, method, samplerate, frame_len, preemph)
                                                                            -> (hz float64 [bound], lag int32 [bound], frame_off int64 [U+1])
                                                                                                         (pitch.py:83 / :96)

PyTorch supplies tensors and the current stream; the ops launch the sm_100a kernels of libdspfe.so through the same plans as
the rest of the package (cached per parameter set) and register shape-only fake implementations, so they trace under
torch.export / FakeTensor without a device.  No CPU implementation is registered: a CPU tensor raises NotImplementedError.
Importing this module registers the ops (it is not imported by `import dspfe`, which keeps torch optional there)."""
import functools
import math

import numpy as np
import torch

from . import binding

_lib = torch.library.Library("dspfe", "DEF")
_lib.define("endpoint(Tensor pcm, Tensor offsets, int samplerate=16000) -> Tensor")
_lib.define("endpoint_robust(Tensor pcm, Tensor offsets, int samplerate=16000) -> Tensor")
_lib.define("mfcc_delta(Tensor pcm, Tensor offsets, Tensor? trim=None, int samplerate=16000, int frame_len=400, int frame_step=160, "
            "int nfft=512, int delta_n=2, float preemph=0.97, bool hamming=False) -> (Tensor, Tensor)")
_lib.define("pitch(Tensor pcm, Tensor offsets, Tensor? trim=None, int method=0, int samplerate=16000, int frame_len=512, "
            "float preemph=0.0) -> (Tensor, Tensor, Tensor)")


@functools.lru_cache(maxsize=16)
def _endpoint_plan(samplerate):
    return binding.EndpointPlan(samplerate=samplerate)


@functools.lru_cache(maxsize=32)
def _mfcc_plan(samplerate, frame_len, frame_step, nfft, delta_n, preemph, hamming):
    return binding.MfccPlan(samplerate=samplerate, frame_len=frame_len, frame_step=frame_step, nfft=nfft, delta_n=delta_n, preemph=preemph,
                            window=np.hamming(frame_len) if hamming else None)


@functools.lru_cache(maxsize=32)
def _pitch_plan(method, samplerate, frame_len, preemph):
    return binding.PitchPlan(method=method, samplerate=samplerate, frame_len=frame_len, preemph=preemph)


def _endpoint_cuda(pcm, offsets, samplerate=16000):
    if pcm.dtype == torch.float32:
        return _endpoint_plan(int(samplerate)).detect_f32(pcm.contiguous(), offsets.contiguous())
    return _endpoint_plan(int(samplerate)).detect(pcm.contiguous(), offsets.contiguous())


def _endpoint_robust_cuda(pcm, offsets, samplerate=16000):
    if pcm.dtype == torch.float32:
        return _endpoint_plan(int(samplerate)).detect_robust_f32(pcm.contiguous(), offsets.contiguous())
    return _endpoint_plan(int(samplerate)).detect_robust(pcm.contiguous(), offsets.contiguous())


def _mfcc_cuda(pcm, offsets, trim=None, samplerate=16000, frame_len=400, frame_step=160, nfft=512, delta_n=2, preemph=0.97, hamming=False):
    plan = _mfcc_plan(int(samplerate), int(frame_len), int(frame_step), int(nfft), int(delta_n), float(preemph), bool(hamming))
    t = None if trim is None else trim.contiguous()
    if pcm.dtype == torch.float32:
        return plan.mfcc_delta_f32(pcm.contiguous(), offsets.contiguous(), trim=t)
    return plan.mfcc_delta(pcm.contiguous(), offsets.contiguous(), trim=t)


def _pitch_cuda(pcm, offsets, trim=None, method=0, samplerate=16000, frame_len=512, preemph=0.0):
    plan = _pitch_plan(int(method), int(samplerate), int(frame_len), float(preemph))
    o = plan.detect(pcm.contiguous(), offsets.contiguous(), trim=None if trim is None else trim.contiguous())
    return o["pitch"], o["lag"], o["frame_off"]


_lib.impl("endpoint", _endpoint_cuda, "CUDA")
_lib.impl("endpoint_robust", _endpoint_robust_cuda, "CUDA")
_lib.impl("mfcc_delta", _mfcc_cuda, "CUDA")
_lib.impl("pitch", _pitch_cuda, "CUDA")


# shape-only implementations: the row / frame bounds of the plans depend on sizes alone
@torch.library.register_fake("dspfe::endpoint")
def _(pcm, offsets, samplerate=16000):
    return pcm.new_empty((offsets.shape[0] - 1, 2), dtype=torch.int32)


@torch.library.register_fake("dspfe::endpoint_robust")
def _(pcm, offsets, samplerate=16000):
    return pcm.new_empty((offsets.shape[0] - 1, 2), dtype=torch.int32)


@torch.library.register_fake("dspfe::mfcc_delta")
def _(pcm, offsets, trim=None, samplerate=16000, frame_len=400, frame_step=160, nfft=512, delta_n=2, preemph=0.97, hamming=False):
    n_utt = offsets.shape[0] - 1
    rows = pcm.shape[0] // frame_step + (2 if frame_step > frame_len else 1) * n_utt          # dspfe_rows_bound
    return pcm.new_empty((rows, 39), dtype=torch.float32), offsets.new_empty((n_utt + 1,), dtype=torch.int64)


@torch.library.register_fake("dspfe::pitch")
def _(pcm, offsets, trim=None, method=0, samplerate=16000, frame_len=512, preemph=0.0):
    n_utt = offsets.shape[0] - 1
    g = math.gcd(int(samplerate), 10000)                      # dspfe_pitch_frames_bound: decimation samplerate -> 10 kHz, 100-sample hops
    bound = (pcm.shape[0] // (samplerate // g) + 1) * (10000 // g) // 100 + 3 * n_utt
    return (pcm.new_empty((bound,), dtype=torch.float64), pcm.new_empty((bound,), dtype=torch.int32),
            offsets.new_empty((n_utt + 1,), dtype=torch.int64))
