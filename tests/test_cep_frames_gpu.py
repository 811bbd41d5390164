"""GPU tests of the cepstrum pitch at frame lengths other than 512 samples (pitch_cep_bluestein_kernel) through the C ABI,
the torch op and the drop-in.  Lags follow the parity rule of tests/pitchcheck.py: exact, except float64 near-ties, which are
counted; every other difference fails."""
import numpy as np
import pytest

import pitchcheck

pytestmark = pytest.mark.gpu


def _dev():
    import torch
    return torch.device("cuda:0")


def _check_batch(pcm, off, lag, pitch, fo, rate, N, step=0.01, trim=None, preemph=0.0, what=""):
    """check_lags on every utterance of a batch; returns (frames, differing, near-ties)."""
    from oracle import ref_features as O
    tot = np.zeros(3, dtype=np.int64)
    for u in range(len(off) - 1):
        sig = pcm[off[u]:off[u + 1]]
        if preemph:
            sig = O.preemphasis(sig, preemph)
        if trim is not None:
            sig = sig[trim[u, 0]:trim[u, 1]]
        a, b = fo[u], fo[u + 1]
        tot += pitchcheck.check_lags(0, sig, rate, lag[a:b], pitch[a:b], winlen=N / 10000.0, step=step, what=f"{what} u={u}")
    assert tot[0] == fo[-1]
    return tot


@pytest.mark.parametrize("N", [100, 199, 250, 300, 307, 400, 511])
def test_ragged_int16_batches(N):
    import torch
    import dspfe
    from dspfe import synth
    lengths = synth.ragged_lengths(24, seed=N, lo=16000, hi=48000)
    lengths[:4] = [1, 700, 1000 + N, 8001]
    pcm, off = synth.synth_batch(lengths, seed0=3100 + N)
    dev = _dev()
    o = dspfe.PitchPlan(method=0, frame_len=N).detect(torch.from_numpy(pcm).to(dev), torch.from_numpy(off).to(dev))
    fo = o["frame_off"].cpu().numpy()
    lag, pitch = o["lag"].cpu().numpy()[:fo[-1]], o["pitch"].cpu().numpy()[:fo[-1]]
    tot = _check_batch(pcm, off, lag, pitch, fo, 16000, N, what=f"N={N}")
    pitchcheck.record(f"cep_frames_ragged_N{N}", *tot)
    assert tot[0] >= 2900          # 7 lengths: more than 20 000 frames over this test
    assert tot[1] - tot[2] == 0


@pytest.mark.parametrize("rate", [8000, 44100, 48000])
def test_rates_step_trim_preemphasis_float32(rate):
    import torch
    import dspfe
    from dspfe import synth
    lengths = [int(v * rate / 16000) for v in (24000, 9000, 300, 40011, 15000, 3000)]
    pcm, off = synth.synth_batch(lengths, seed0=rate // 7, sr=rate)
    lens = np.diff(off)
    trim = np.stack([lens // 10, lens - lens // 7], axis=1).astype(np.int32)
    dev = _dev()
    pcm_d, off_d, trim_d = torch.from_numpy(pcm).to(dev), torch.from_numpy(off).to(dev), torch.from_numpy(trim).to(dev)
    pcmf = pcm.astype(np.float32) * np.float32(2.0 ** -15)
    for N, step in ((300, 0.0125), (307, 0.01)):
        fs = int(step * 10000)
        for kw, x, xd, t, td in ((dict(preemph=0.97), pcm, pcm_d, trim, trim_d), ({}, pcmf, torch.from_numpy(pcmf).to(dev), None, None)):
            plan = dspfe.PitchPlan(method=0, samplerate=rate, frame_len=N, frame_step=fs, **kw)
            o = plan.detect(xd, off_d, trim=td)
            fo = o["frame_off"].cpu().numpy()
            lag, pitch = o["lag"].cpu().numpy()[:fo[-1]], o["pitch"].cpu().numpy()[:fo[-1]]
            tot = _check_batch(x, off, lag, pitch, fo, rate, N, step=step, trim=t, preemph=kw.get("preemph", 0.0),
                               what=f"rate={rate} N={N} {x.dtype}")
            pitchcheck.record(f"cep_frames_rate{rate}_N{N}_{x.dtype}", *tot)
            assert tot[1] - tot[2] == 0
            # the host path gives the same bits
            hp, hl, hfo = plan.detect_host(x, off, trim=t)
            np.testing.assert_array_equal(hfo, fo)
            np.testing.assert_array_equal(hl, lag)
            np.testing.assert_array_equal(hp, pitch)


def test_rows_tap_against_oracle():
    import torch
    import dspfe
    from dspfe import synth
    from oracle import ref_features as O
    dev = _dev()
    for N in (100, 199, 256, 307, 480, 511):
        rng = np.random.default_rng(N)
        fr = []
        for i in range(9):
            x = O.downsampling(synth.synth_utterance(N * 10 + i, 6000), 16000, 10000).astype(np.float64)
            s = int(rng.integers(0, len(x) - N))
            fr.append(O.center_clip(x[s:s + N], False).astype(np.float32))
        fr = np.array(fr)
        off = np.arange(len(fr) + 1, dtype=np.int64) * N
        plan = dspfe.PitchPlan(method=0, samplerate=10000, frame_len=N, center_clip=False, row_len=N)
        o = plan.detect(torch.from_numpy(fr.reshape(-1)).to(dev), torch.from_numpy(off).to(dev), want_rows=True, want_track=False)
        got = o["rows"].cpu().numpy()[:len(fr)]
        want = O.pitch_detect_frame(fr.astype(np.float64), 10000)
        assert got.shape == want.shape
        err = np.max(np.abs(got - want), axis=1) / np.max(np.abs(want), axis=1)
        assert np.all(err <= pitchcheck.REL_TOL), (N, err.max())


def test_dropin_pitch_detect_and_frame():
    import dspfe
    import features
    from dspfe import synth
    from oracle import ref_features as O
    x = synth.synth_utterance(2024, 30000)
    p, frames = features.pitch.pitch_detect(x, 16000, winlen=0.03)
    wp, wframes = O.pitch_detect(x, 16000, winlen=0.03)
    assert isinstance(p, list) and all(type(v) is np.float64 for v in p) and len(p) == len(wp)
    assert isinstance(frames, np.ndarray) and frames.dtype == np.float64 and frames.shape == wframes.shape == (len(p), 300)
    np.testing.assert_array_equal(frames, wframes)
    # the Hz list is the plan's, and its lags pass the parity rule
    hp, hl, hfo = dspfe.PitchPlan(method=0, frame_len=300).detect_host(x, np.array([0, len(x)]))
    assert p == hp.tolist()
    tot = pitchcheck.check_lags(0, x, 16000, hl, hp, winlen=0.03, what="pitch_detect winlen=0.03")
    assert tot[1] == tot[2]
    fr = O.center_clip(wframes[len(p) // 2], False)
    row = features.pitch.pitch_detect_frame(fr, 10000, "male")
    want = O.pitch_detect_frame(fr, 10000)
    assert isinstance(row, np.ndarray) and row.dtype == np.float64 and row.shape == want.shape == (300,)
    assert np.max(np.abs(row - want)) <= pitchcheck.REL_TOL * np.max(np.abs(want))


def test_utterance_alone_equals_inside_a_batch():
    import torch
    import dspfe
    from dspfe import synth
    dev = _dev()
    lengths = [17000, 5003, 23456, 999, 12000, 30001, 4000]
    pcm, off = synth.synth_batch(lengths, seed0=808)
    for N in (199, 307):
        plan = dspfe.PitchPlan(method=0, frame_len=N)
        big = plan.detect(torch.from_numpy(pcm).to(dev), torch.from_numpy(off).to(dev), want_rows=True)
        bfo = big["frame_off"].cpu().numpy()
        for u in (2, 5):
            x = pcm[off[u]:off[u + 1]]
            one = plan.detect(torch.from_numpy(x).to(dev), torch.tensor([0, len(x)], device=dev), want_rows=True)
            n = int(one["frame_off"][1])
            assert n == bfo[u + 1] - bfo[u]
            for k in ("rows", "lag", "pitch"):
                np.testing.assert_array_equal(one[k].cpu().numpy()[:n], big[k].cpu().numpy()[bfo[u]:bfo[u + 1]], err_msg=f"{k} N={N} u={u}")


def test_torch_op_and_fake():
    import torch
    import dspfe
    import dspfe.torch_ops  # noqa: F401
    from dspfe import synth
    from torch._subclasses.fake_tensor import FakeTensorMode
    dev = _dev()
    lengths = [16000, 4001, 27000]
    pcm, off = synth.synth_batch(lengths, seed0=99)
    pd, od = torch.from_numpy(pcm).to(dev), torch.from_numpy(off).to(dev)
    hz, lag, fo = torch.ops.dspfe.pitch(pd, od, None, 0, 16000, 300, 0.0)
    want = dspfe.PitchPlan(method=0, frame_len=300).detect(pd, od)
    n = int(fo[-1])
    assert torch.equal(fo, want["frame_off"])
    assert torch.equal(hz[:n], want["pitch"][:n]) and torch.equal(lag[:n], want["lag"][:n])
    with FakeTensorMode():
        fp = torch.empty(pcm.shape[0], dtype=torch.int16, device="cuda")
        fo_ = torch.empty(len(lengths) + 1, dtype=torch.int64, device="cuda")
        h, l, q = torch.ops.dspfe.pitch(fp, fo_, None, 0, 16000, 300, 0.0)
        assert h.shape == hz.shape and l.shape == lag.shape and q.shape == fo.shape


def test_timing_names_the_kernel():
    import torch
    import dspfe
    from dspfe import synth
    dev = _dev()
    pcm, off = synth.synth_batch([16000, 9000], seed0=7)
    pd, od = torch.from_numpy(pcm).to(dev), torch.from_numpy(off).to(dev)
    for N, yes, no in ((300, "pitch_cep_bluestein_kernel", "pitch_frame_kernel<0>"), (512, "pitch_frame_kernel<0>", "pitch_cep_bluestein_kernel")):
        plan = dspfe.PitchPlan(method=0, frame_len=N)
        plan.detect(pd, od)
        dspfe.timing_begin()
        plan.detect(pd, od)
        names = [n for n, _ in dspfe.timing_end()]
        assert yes in names and no not in names, (N, names)


def test_digital_silence():
    import dspfe
    z = np.zeros(12000, dtype=np.int16)
    x = np.concatenate([z, (np.arange(9000) % 57 * 300 - 8000).astype(np.int16), z])
    pcm = np.concatenate([z, x])
    off = np.array([0, len(z), len(pcm)], dtype=np.int64)
    pitch, lag, fo = dspfe.PitchPlan(method=0, frame_len=300).detect_host(pcm, off)
    assert np.all(lag[fo[0]:fo[1]] == 20)
    tot = _check_batch(pcm, off, lag, pitch, fo, 16000, 300, what="silence")
    assert tot[1] == tot[2]


def test_unbuilt_requests_raise():
    import torch
    import dspfe
    from dspfe.binding import DspfeUnsupported
    pcm = np.zeros(16000, dtype=np.int16)
    off = np.array([0, len(pcm)], dtype=np.int64)
    plan = dspfe.PitchPlan(method=0, frame_len=300)
    with pytest.raises(DspfeUnsupported):
        plan.detect(torch.from_numpy(pcm).to(_dev()), torch.from_numpy(off).to(_dev()), want_feat=True)
    with pytest.raises(DspfeUnsupported):
        plan.detect_host(pcm, off, want_feat=True)
    for N in (99, 513):
        with pytest.raises(DspfeUnsupported):
            dspfe.PitchPlan(method=0, frame_len=N)
