"""GPU tests of robust endpoint detection on float32 samples (dspfe_endpoint_robust_f32 / _host_f32): bit-exact against the
float64 oracle on non-integer batches and on utterances tuned so that a gate sitting on 0.55 decides where the walk stops, exact
power-of-two scaling against the int16 path, non-finite samples, and the torch op."""
import os
import sys
import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def float_batch(lengths, rate=16000, seed=5):
    """Non-integer float32 samples: synthetic speech x 0.37 plus float noise."""
    from dspfe import synth
    pcm, off = synth.synth_batch(lengths, seed0=700 + seed, sr=rate)
    rng = np.random.default_rng(seed)
    x = (pcm.astype(np.float64) * 0.37 + rng.standard_normal(len(pcm)) * 3.1).astype(np.float32)
    return x, off


def oracle_robust(x, rate, **kw):
    from oracle import ref_features as O
    with np.errstate(all="ignore"), warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return O.robust_endpoint_detection(x, rate, **kw)


def pack(xs):
    off = np.concatenate([[0], np.cumsum([len(x) for x in xs])]).astype(np.int64)
    return np.concatenate(xs).astype(np.float32), off


def both_forms(plan, x, off):
    import torch
    dev = torch.device("cuda:0")
    lr_d = plan.detect_robust_f32(torch.from_numpy(x).to(dev), torch.from_numpy(off).to(dev)).cpu().numpy()
    lr_h = plan.detect_robust_host_f32(x, off)
    np.testing.assert_array_equal(lr_d, lr_h)
    return lr_h


@pytest.mark.parametrize("rate,cfg_frame,cfg_step", [(8000, 0.03, 0.01), (16000, 0.03, 0.01), (22050, 0.03, 0.01),
                                                     (44100, 0.03, 0.01), (48000, 0.03, 0.01), (16000, 0.03, 0.04),
                                                     (16000, 0.0301, 0.01)])
def test_robust_vs_oracle_bit_exact(rate, cfg_frame, cfg_step):
    import dspfe
    from dspfe import synth
    from oracle import ref_features as O
    n = 12 if rate > 40000 else 20
    lengths = list(synth.ragged_lengths(n, seed=rate, lo=rate // 4, hi=3 * rate))
    lengths[:3] = [int(0.03 * rate) + 1, rate // 2, rate]
    if rate == 16000 and cfg_step == 0.01:
        lengths[3] = 170000                                   # more than kEpStageFrames frames: amplitudes from global memory
    x, off = float_batch(lengths, rate)
    x[off[1]:off[2]] = 0.0                                    # digital silence
    plan = dspfe.EndpointPlan(samplerate=rate, cfg_frame=cfg_frame, cfg_step=cfg_step)
    lr = both_forms(plan, x, off)
    differs = 0
    for u in range(len(lengths)):
        sig = x[off[u]:off[u + 1]]
        want = oracle_robust(sig, rate, cfg_frame=cfg_frame, cfg_step=cfg_step)
        assert (int(lr[u, 0]), int(lr[u, 1])) == want, f"utterance {u}"
        differs += want != O.basic_endpoint_detection(sig, rate, cfg_frame=cfg_frame, cfg_step=cfg_step)
    if cfg_step < cfg_frame:      # (with gaps between the frames both rules fall back to the whole signal on this batch)
        assert differs > 0, "the robust rule never departs from the basic one on this batch"


def threshold_utterance(rate, period, seed):
    """Floor noise, a loud voiced segment, then a quieter periodic region whose noise is a * noise.  Its frames stay above the
    low threshold, so the gate alone decides how far the walk right of the voiced segment goes.  The float32 coefficient a is
    bisected until the oracle's robust (l, r) changes: the two utterances either side of the flip differ in a gate whose ratio
    is within float32 rounding of 0.55, far inside the screening band, so the kernel's exact fallback decides them."""
    rng = np.random.default_rng(seed)
    n_sil, n_voc, n_tun = int(0.3 * rate), int(0.6 * rate), int(0.15 * rate)
    i = np.arange(n_voc + n_tun)
    per = np.sin(2 * np.pi * i / period) + 0.4 * np.sin(4 * np.pi * i / period + 0.3)
    level = np.where(i < n_voc, 0.5, 0.1)
    noise = rng.standard_normal(n_voc + n_tun) * np.where(i < n_voc, 0.0, 0.05)
    floor = rng.standard_normal(2 * n_sil + n_voc + n_tun) * 1e-3

    def make(a):
        y = floor.copy()
        y[n_sil:n_sil + n_voc + n_tun] += level * per + np.float64(a) * noise
        return y.astype(np.float32)

    lo, hi = np.float32(0.0), np.float32(3.0)
    r_lo = oracle_robust(make(lo), rate)
    assert r_lo != oracle_robust(make(hi), rate)
    while True:
        mid = np.float32((np.float64(lo) + np.float64(hi)) / 2)
        if mid in (lo, hi):
            break
        if oracle_robust(make(mid), rate) == r_lo:
            lo = mid
        else:
            hi = mid
    return make(lo), make(hi)


@pytest.mark.parametrize("rate", [8000, 16000, 44100])
def test_threshold_flips_match_oracle(rate):
    import dspfe
    xs = []
    for k, period in enumerate([0.006, 0.009, 0.0061, 0.0125]):
        xs.extend(threshold_utterance(rate, int(period * rate), seed=10 * k + rate % 7))
    x, off = pack(xs)
    lr = both_forms(dspfe.EndpointPlan(samplerate=rate), x, off)
    for u in range(len(xs)):
        assert (int(lr[u, 0]), int(lr[u, 1])) == oracle_robust(xs[u], rate), f"utterance {u} (pair {u // 2})"
    for u in range(0, len(xs), 2):
        assert tuple(lr[u]) != tuple(lr[u + 1])


@pytest.mark.parametrize("scale", [2.0 ** -15, 2.0 ** -140, 2.0 ** 100])
def test_power_of_two_scaling_equals_int16_robust(scale):
    """float = int16 x 2^k gives the int16 path's lr: every lag sum of such samples is exact in any order, and the rule is
    invariant under power-of-two scaling (2^-140 makes most samples float32 subnormals, 2^100 puts the squares beyond float32)."""
    import torch
    import dspfe
    from dspfe import synth
    dev = torch.device("cuda:0")
    lengths = synth.ragged_lengths(2048, seed=77)
    pcm16, off = synth.synth_batch_torch(lengths, seed0=91, device=dev)
    od = off.to(dev)
    plan = dspfe.EndpointPlan()
    want = plan.detect_robust(pcm16, od)
    xf = (pcm16.double() * scale).float().contiguous()
    assert torch.equal(xf.double() / scale, pcm16.double())    # the scaled samples are exact
    got = plan.detect_robust_f32(xf, od)
    assert torch.equal(got, want)


def test_non_finite_samples_stay_in_their_utterance():
    import dspfe
    from dspfe import synth
    lengths = list(synth.ragged_lengths(10, seed=4, lo=8000, hi=40000))
    x, off = float_batch(lengths, seed=8)
    plan = dspfe.EndpointPlan()
    clean = both_forms(plan, x, off)
    y = x.copy()
    y[off[3] + 5000] = np.nan
    y[off[7] + 4000] = np.inf
    lr = both_forms(plan, y, off)
    keep = [u for u in range(len(lengths)) if u not in (3, 7)]
    np.testing.assert_array_equal(lr[keep], clean[keep])
    assert (int(lr[7, 0]), int(lr[7, 1])) == oracle_robust(y[off[7]:off[8]], 16000)


def test_torch_op_timing_and_fake():
    import torch
    import dspfe
    import dspfe.torch_ops  # noqa: F401  registers the ops
    from dspfe import synth
    dev = torch.device("cuda:0")
    lengths = [16000, 8000, 30001, 12345]
    pcm, off = synth.synth_batch(lengths, seed0=3)
    p16, od = torch.from_numpy(pcm).to(dev), torch.from_numpy(off).to(dev)
    pf = (p16.float() * 2.0 ** -15).contiguous()
    plan = dspfe.EndpointPlan()
    assert torch.equal(torch.ops.dspfe.endpoint_robust(p16, od), plan.detect_robust(p16, od))
    assert torch.equal(torch.ops.dspfe.endpoint_robust(pf, od, 16000), plan.detect_robust_f32(pf, od))
    with pytest.raises(NotImplementedError):
        torch.ops.dspfe.endpoint_robust(torch.from_numpy(pcm), torch.from_numpy(off))
    dspfe.timing_begin()
    plan.detect_robust_f32(pf, od)
    names = [n for n, _ in dspfe.timing_end()]
    assert "ep_stats_f32_kernel" in names and "ep_decide_robust_kernel<f32>" in names
    assert "ep_decide_robust_kernel" not in names
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        fp = torch.empty(len(pcm), dtype=torch.float32, device="cuda")
        fo = torch.empty(len(lengths) + 1, dtype=torch.int64, device="cuda")
        r = torch.ops.dspfe.endpoint_robust(fp, fo)
        assert r.shape == (len(lengths), 2) and r.dtype == torch.int32
