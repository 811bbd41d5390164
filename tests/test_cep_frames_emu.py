"""Cepstrum pitch at frame lengths other than 512 samples (pitch_cep_bluestein_pair, csrc/pitch_kernel.cuh) on the CPU SIMT
emulator against the float64 oracle, plus the host-only validation and frame counts of the C ABI and the drop-in's argument
checks.  The GPU tests of the same path are tests/test_cep_frames_gpu.py."""
import ctypes
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu  # noqa: E402
import pitchcheck  # noqa: E402
from dspfe import synth  # noqa: E402
from oracle import ref_features as O  # noqa: E402

ROW_N = [100, 128, 199, 200, 250, 256, 300, 307, 400, 480, 500, 511]


def pitch_cep(pcm, offsets, trim=None, frame_len=300, row_len=0, samplerate=16000, center_clip=1, preemph=0.0, want_rows=False):
    """The cepstrum pitch pipeline with the Bluestein chain on the emulator (emu_pitch_cep, tests/emu/emu_cep.cpp), every
    frame length included: 512-sample frames run the Bluestein chain here too.  Returns dict(pitch, lag, frame_off[, rows,
    smoothed])."""
    q = emu.PitchParams(samplerate, 10000, frame_len, 100, 0, center_clip, row_len, 0, 50.0, 1000.0, preemph)
    f32 = np.asarray(pcm).dtype.kind == "f"
    pcm = np.ascontiguousarray(pcm, dtype=np.float32 if f32 else np.int16)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n = len(offsets) - 1
    cap = int(len(pcm) // 100 + 3 * n + 8)
    rl = row_len or min(frame_len, 200)
    out = dict(pitch=np.full(cap, np.nan), lag=np.zeros(cap, dtype=np.int32), frame_off=np.zeros(n + 1, dtype=np.int64))
    rows = np.full((cap, rl), np.nan, dtype=np.float32) if want_rows else None
    sm = np.full((cap, rl), np.nan, dtype=np.float32) if want_rows else None
    tp = None if trim is None else np.ascontiguousarray(trim, dtype=np.int32)
    vp = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    err = ctypes.create_string_buffer(256)
    f = emu.lib().emu_pitch_cep
    f.restype = ctypes.c_longlong
    r = f(ctypes.byref(q), vp(pcm), int(f32), vp(offsets), vp(tp), n, vp(out["pitch"]), vp(out["lag"]), vp(rows), vp(sm), None,
          vp(out["frame_off"]), ctypes.c_longlong(cap), err, 256)
    if r < 0:
        raise RuntimeError(f"emulator: {err.value.decode()} ({r})")
    out["pitch"], out["lag"] = out["pitch"][:r], out["lag"][:r]
    if want_rows:
        out["rows"], out["smoothed"] = rows[:r], sm[:r]
    return out


def clipped_frames(N, count, seed):
    """center_clip(frame, False) of frames cut at random places from decimated synthetic speech, as float32 values."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(count):
        x = O.downsampling(synth.synth_utterance(seed * 100 + i, 4000), 16000, 10000).astype(np.float64)
        s = int(rng.integers(0, len(x) - N))
        out.append(O.center_clip(x[s:s + N], False).astype(np.float32))
    return np.array(out)


def frame_rows(frames, row_len):
    """Each frame as a one-frame utterance at 10 kHz without clipping: the rows tap of pitch_detect_frame."""
    N = frames.shape[1]
    off = np.arange(len(frames) + 1, dtype=np.int64) * N
    return pitch_cep(frames.reshape(-1), off, samplerate=10000, frame_len=N, center_clip=0, row_len=row_len, want_rows=True)["rows"]


@pytest.mark.parametrize("N", ROW_N)
def test_rows_match_oracle(N):
    fr = clipped_frames(N, 7, seed=N)                 # an odd count: the last pair has one frame
    got = frame_rows(fr, N)
    want = O.pitch_detect_frame(fr.astype(np.float64), 10000)
    assert got.shape == want.shape
    for i in range(len(fr)):
        assert np.max(np.abs(got[i] - want[i])) <= pitchcheck.REL_TOL * np.max(np.abs(want[i])), (N, i)


@pytest.mark.parametrize("rate", [16000, 44100])
@pytest.mark.parametrize("N", [300, 307])
def test_lags_ragged_batch_trim_preemphasis(rate, N):
    scale = rate / 16000.0
    lengths = [int(v * scale) for v in (12000, 5000, 300, 20011, 7777)]
    pcm, off = synth.synth_batch(lengths, seed0=91, sr=rate)
    trim = np.array([[1000, 11000], [0, 99999], [10, 200], [3333, 18000], [500, 7000]], dtype=np.int32)
    trim = (trim * scale).astype(np.int32)
    r = pitch_cep(pcm, off, trim=trim, samplerate=rate, frame_len=N, preemph=0.97)
    tot = 0
    for u in range(len(lengths)):
        sig = O.preemphasis(pcm[off[u]:off[u + 1]], 0.97)[trim[u, 0]:trim[u, 1]]
        a, b = r["frame_off"][u], r["frame_off"][u + 1]
        frames, differing, near = pitchcheck.check_lags(0, sig, rate, r["lag"][a:b], r["pitch"][a:b], winlen=N / 10000.0,
                                                        what=f"N={N} rate={rate} u={u}")
        tot += frames
    assert tot == r["frame_off"][-1]


def test_bluestein_at_512_matches_the_512_point_chain():
    lengths = [9000, 5121, 700, 16000]
    pcm, off = synth.synth_batch(lengths, seed0=13)
    ref = emu.pitch(pcm, off, method=0, row_len=512, want_rows=True)
    blu = pitch_cep(pcm, off, frame_len=512, row_len=512, want_rows=True)
    np.testing.assert_array_equal(blu["frame_off"], ref["frame_off"])
    assert blu["rows"].shape == ref["rows"].shape
    for i in range(len(ref["rows"])):
        assert np.max(np.abs(blu["rows"][i] - ref["rows"][i])) <= pitchcheck.REL_TOL * np.max(np.abs(ref["rows"][i])), i
    # and the Bluestein rows against the float64 oracle
    for u in range(len(lengths)):
        fr = O.to_frames(O.downsampling(pcm[off[u]:off[u + 1]], 16000, 10000), 10000, 0.0512, 0.01)
        want = O.pitch_detect_frame(O.center_clip(fr, False), 10000)
        got = blu["rows"][blu["frame_off"][u]:blu["frame_off"][u + 1]]
        assert np.all(np.max(np.abs(got - want), axis=1) <= pitchcheck.REL_TOL * np.max(np.abs(want), axis=1)), u


def test_zero_frame_gives_nan_row_and_silence_gives_reference_lags():
    # log 0 = -inf in every bin -> an all-NaN cepstrum row (SURVEY A-11)
    fr = clipped_frames(300, 3, seed=5)
    fr[1] = 0.0
    rows = frame_rows(fr, 300)
    assert np.all(np.isnan(rows[1])) and np.all(np.isfinite(rows[0])) and np.all(np.isfinite(rows[2]))
    # a silent stretch inside speech: lag 20 on the silent frames, and smooth spreads the NaN rows to their neighbours
    x = synth.synth_utterance(77, 9000)
    x[3000:6000] = 0
    for N in (300, 199):
        r = pitch_cep(x, [0, len(x)], frame_len=N, row_len=N, want_rows=True)
        sm = O.pitch_rows_cep(x, 16000, winlen=N / 10000.0)
        # (the reference's column 0 of a silent row is |sum of -inf| / N = +inf where the kernel has a NaN: both are non-finite,
        # and column 0 takes no part in peak_score)
        np.testing.assert_array_equal(np.isfinite(r["smoothed"]), np.isfinite(sm))
        silent = np.all(np.isnan(sm[:, 1:]), axis=1)
        assert np.any(silent)
        pitchcheck.check_lags(0, x, 16000, r["lag"], r["pitch"], winlen=N / 10000.0, what=f"silence N={N}")
        assert np.all(r["lag"][silent] == 20)


@pytest.mark.parametrize("N", ROW_N)
def test_num_frames_host_matches_oracle(N):
    import dspfe
    for step in (100, 125, 37, 512):
        for n in (0, 1, 999, 1600, 16000, 44100, 123457):
            nf, ld = dspfe.pitch_num_frames_host(n, frame_len=N, frame_step=step, method=0)
            ds = len(O.downsampling(np.zeros(n), 16000, 10000))
            assert ld == ds and nf == O.num_frames(ds, N, step), (N, step, n)


def _host_params(frame_len, row_len=0):
    import dspfe
    from dspfe import binding
    L = dspfe.lib(); binding._bind_pitch(L)
    p = binding._PitchParams()
    L.dspfe_pitch_params_default(ctypes.byref(p), 0)
    p.frame_len, p.row_len = int(frame_len), int(row_len)
    L.dspfe_pitch_num_frames_host.argtypes = [ctypes.POINTER(binding._PitchParams), ctypes.c_int64, ctypes.POINTER(ctypes.c_int64)]
    L.dspfe_pitch_num_frames_host.restype = ctypes.c_int64
    rc = L.dspfe_pitch_num_frames_host(ctypes.byref(p), 16000, None)
    return int(rc), L.dspfe_last_error().decode()


def test_host_validation_of_frame_and_row_lengths():
    for N in (100, 307, 512):
        assert _host_params(N)[0] > 0
        assert _host_params(N, row_len=N)[0] > 0
    for N in (99, 513, 20):
        rc, msg = _host_params(N)
        assert rc == -2 and "100..512" in msg, (N, rc, msg)
    rc, msg = _host_params(300, row_len=301)
    assert rc == -1 and "row_len" in msg
    assert _host_params(300, row_len=99)[0] == -1
    assert _host_params(150)[0] > 0                    # the default row_len is min(N, 200)


def test_mirror_rejects_unbuilt_lengths_before_any_device_call():
    import features
    x = synth.synth_utterance(3, 4000)
    with pytest.raises(IndexError):                   # the reference's peak_score reads sig[20..99]
        features.pitch.pitch_detect(x, 16000, winlen=0.005)
    with pytest.raises(NotImplementedError):
        features.pitch.pitch_detect(x, 16000, winlen=0.06)
    with pytest.raises(NotImplementedError):
        features.pitch.pitch_detect_frame(np.zeros(99), 10000, "male")
    with pytest.raises(NotImplementedError):
        features.pitch.pitch_detect_frame(np.zeros(513), 10000, "male")
