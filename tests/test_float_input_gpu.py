"""GPU tests of the float32-sample endpoint and front-end entry points (dspfe_endpoint_f32 / _host_f32, dspfe_frontend_f32 /
_host_f32): bit-exact endpoints against the float64 oracle, exact power-of-two scaling against the int16 path, the front-end
equal to the chain of the separate float entry points, slab and host-path invariance, and the oracle on the features."""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def float_batch(lengths, rate=16000, seed=5):
    """Non-integer float32 samples: synthetic speech x 0.37 plus float noise; a few silent utterances."""
    from dspfe import synth
    pcm, off = synth.synth_batch(lengths, seed0=700 + seed, sr=rate)
    rng = np.random.default_rng(seed)
    x = (pcm.astype(np.float64) * 0.37 + rng.standard_normal(len(pcm)) * 3.1).astype(np.float32)
    return x, off


def ragged(rate, n=24, seed=3):
    from dspfe import synth
    L = int(rate * 0.03)
    lengths = list(synth.ragged_lengths(n, seed=seed, lo=rate // 4, hi=3 * rate))
    lengths[:6] = [0, 1, L - 1, L + 1, rate // 2, rate]
    return lengths


def silence(x, off, us):
    for u in us:
        x[off[u]:off[u + 1]] = 0.0
    return x


@pytest.mark.parametrize("rate,cfg_frame,cfg_step", [(8000, 0.03, 0.01), (16000, 0.03, 0.01), (22050, 0.03, 0.01),
                                                     (44100, 0.03, 0.01), (48000, 0.03, 0.01), (16000, 0.03, 0.04),
                                                     (16000, 0.0301, 0.01)])
def test_endpoints_vs_oracle_bit_exact(rate, cfg_frame, cfg_step):
    import torch
    import dspfe
    from oracle import ref_features as O
    lengths = ragged(rate)
    x, off = float_batch(lengths, rate)
    x = silence(x, off, [5])
    plan = dspfe.EndpointPlan(samplerate=rate, cfg_frame=cfg_frame, cfg_step=cfg_step)
    dev = torch.device("cuda:0")
    lr_d, amp_d, zcr_d, fo_d = plan.detect_f32(torch.from_numpy(x).to(dev), torch.from_numpy(off).to(dev), want_features=True)
    lr_h, amp_h, zcr_h, fo_h = plan.detect_host_f32(x, off, want_features=True)
    nf = int(fo_h[-1])
    np.testing.assert_array_equal(lr_d.cpu().numpy(), lr_h)
    np.testing.assert_array_equal(amp_d.cpu().numpy()[:nf], amp_h)
    np.testing.assert_array_equal(zcr_d.cpu().numpy()[:nf], zcr_h)
    np.testing.assert_array_equal(fo_d.cpu().numpy(), fo_h)
    for u in range(len(lengths)):
        sig = x[off[u]:off[u + 1]]
        l, r, amp, z = O.basic_endpoint_detection(sig, rate, return_feature=True, cfg_frame=cfg_frame, cfg_step=cfg_step)
        np.testing.assert_array_equal(amp_h[fo_h[u]:fo_h[u + 1]], np.array(amp), err_msg=f"amp of utterance {u}")
        np.testing.assert_array_equal(zcr_h[fo_h[u]:fo_h[u + 1]], np.array(z), err_msg=f"zcr of utterance {u}")
        assert (int(lr_h[u, 0]), int(lr_h[u, 1])) == (l, r), f"utterance {u}"


def test_power_of_two_scaling_equals_int16_path():
    """float = int16 * 2^-15 gives the int16 path's lr and zcr, and amp = (asum / L) * 2^-15, bit for bit."""
    import torch
    import dspfe
    from dspfe import synth
    lengths = ragged(16000, n=200, seed=9)
    pcm, off = synth.synth_batch(lengths, seed0=31)
    dev = torch.device("cuda:0")
    plan = dspfe.EndpointPlan()
    p16, o = torch.from_numpy(pcm).to(dev), torch.from_numpy(off).to(dev)
    lr, asum, zcr, fo = plan.detect(p16, o, want_features=True)
    lrf, amp, zcrf, fof = plan.detect_f32((p16.float() * 2.0 ** -15).contiguous(), o, want_features=True)
    nf = int(fo[-1])
    np.testing.assert_array_equal(lrf.cpu().numpy(), lr.cpu().numpy())
    np.testing.assert_array_equal(zcrf.cpu().numpy()[:nf], zcr.cpu().numpy()[:nf])
    np.testing.assert_array_equal(amp.cpu().numpy()[:nf], asum.cpu().numpy()[:nf] / 480.0 * 2.0 ** -15)


def to_np(o, tot):
    rows, fc, fa = tot
    return dict(lr=o["lr"].cpu().numpy(), mfcc=o["mfcc"][:rows].cpu().numpy(), mfcc_frame_off=o["mfcc_frame_off"].cpu().numpy(),
                cep_pitch=o["cep_pitch"][:fc].cpu().numpy(), cep_lag=o["cep_lag"][:fc].cpu().numpy(),
                cep_frame_off=o["cep_frame_off"].cpu().numpy(), cep_feat=o["cep_feat"].cpu().numpy(),
                acr_pitch=o["acr_pitch"][:fa].cpu().numpy(), acr_lag=o["acr_lag"][:fa].cpu().numpy(),
                acr_frame_off=o["acr_frame_off"].cpu().numpy())


def host_np(o, tot):
    rows, fc, fa = tot
    g = lambda k: np.asarray(o[k])
    return dict(lr=g("lr"), mfcc=g("mfcc")[:rows], mfcc_frame_off=g("mfcc_frame_off"), cep_pitch=g("cep_pitch")[:fc],
                cep_lag=g("cep_lag")[:fc], cep_frame_off=g("cep_frame_off"), cep_feat=g("cep_feat"), acr_pitch=g("acr_pitch")[:fa],
                acr_lag=g("acr_lag")[:fa], acr_frame_off=g("acr_frame_off"))


def assert_same(a, b, what):
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=f"{what}: {k}")


def fe_batch():
    from dspfe import synth
    lengths = list(synth.ragged_lengths(40, seed=5, lo=6000, hi=50000))
    lengths[:4] = [1, 500, 8000, 80000]
    return float_batch(lengths, seed=8)


def run_device(x, off, **kw):
    import torch
    import dspfe
    dev = torch.device("cuda:0")
    fe = dspfe.FrontendPlan(**kw)
    o = fe.alloc(len(x), len(off) - 1, device=dev)
    tot = fe.run_f32(torch.from_numpy(x).to(dev), torch.from_numpy(off).to(dev), off, o)
    torch.cuda.synchronize()
    return to_np(o, tot)


def test_frontend_equals_separate_float_entry_points():
    import torch
    import dspfe
    x, off = fe_batch()
    got = run_device(x, off)
    dev = torch.device("cuda:0")
    xd, od = torch.from_numpy(x).to(dev), torch.from_numpy(off).to(dev)
    lr = dspfe.EndpointPlan().detect_f32(xd, od)
    out, fo = dspfe.MfccPlan(delta_n=2).mfcc_delta_f32(xd, od, trim=lr)
    cep = dspfe.PitchPlan(method=0, preemph=0.97).detect(xd, od, trim=lr, want_feat=True)
    acr = dspfe.PitchPlan(method=1, frame_len=300).detect(xd, od, trim=lr)
    torch.cuda.synchronize()
    fo = fo.cpu().numpy()
    want = dict(lr=lr.cpu().numpy(), mfcc=out[:fo[-1]].cpu().numpy(), mfcc_frame_off=fo, cep_pitch=cep["pitch"].cpu().numpy(),
                cep_lag=cep["lag"].cpu().numpy(), cep_frame_off=cep["frame_off"].cpu().numpy(), cep_feat=cep["feat"].cpu().numpy(),
                acr_pitch=acr["pitch"].cpu().numpy(), acr_lag=acr["lag"].cpu().numpy(), acr_frame_off=acr["frame_off"].cpu().numpy())
    for k in ("cep_pitch", "cep_lag"):
        want[k] = want[k][: want["cep_frame_off"][-1]]
    for k in ("acr_pitch", "acr_lag"):
        want[k] = want[k][: want["acr_frame_off"][-1]]
    assert_same(got, want, "frontend_f32 vs chain")


def test_slabs_and_host_path_do_not_change_a_bit():
    import dspfe
    x, off = fe_batch()
    ref = run_device(x, off)
    for slab in (20000, 100000, 700001):
        assert_same(run_device(x, off, slab_samples=slab), ref, f"slab {slab}")
    for hs in (30000, 0):
        fe = dspfe.FrontendPlan(host_slab_samples=hs)
        for rep in range(2):
            o = fe.alloc(len(x), len(off) - 1)
            assert_same(host_np(o, fe.run_host_f32(x, off, o)), ref, f"host slab {hs}, call {rep}")
    # offsets that do not start at 0: the same utterances behind a 3-sample prefix
    x2 = np.concatenate([np.full(3, 7.0, np.float32), x])
    fe = dspfe.FrontendPlan(host_slab_samples=30000)
    o = fe.alloc(len(x2), len(off) - 1)
    assert_same(host_np(o, fe.run_host_f32(x2, off + 3, o)), ref, "offset batch")


def test_frontend_vs_oracle():
    from oracle import ref_features as O
    from tol import assert_mfcc_close
    from pitchcheck import check_lags
    x, off = fe_batch()
    got = run_device(x, off)
    for u in range(len(off) - 1):
        sig = x[off[u]:off[u + 1]].astype(np.float64)
        l, r = (int(v) for v in got["lr"][u])
        assert (l, r) == O.basic_endpoint_detection(x[off[u]:off[u + 1]], 16000)[:2]
        fo, ca, cc = got["mfcc_frame_off"], got["acr_frame_off"], got["cep_frame_off"]
        assert_mfcc_close(got["mfcc"][fo[u]:fo[u + 1]], O.mfcc_delta39(sig[l:r], 2), what=f"utterance {u}")
        check_lags(1, sig[l:r], 16000, got["acr_lag"][ca[u]:ca[u + 1]], winlen=0.03, what=f"acr {u}")
        check_lags(0, O.preemphasis(sig, 0.97)[l:r], 16000, got["cep_lag"][cc[u]:cc[u + 1]], what=f"cep {u}")


def test_timing_names_the_statistics_kernel():
    import torch
    import dspfe
    x, off = fe_batch()
    dev = torch.device("cuda:0")
    fe = dspfe.FrontendPlan()
    o = fe.alloc(len(x), len(off) - 1, device=dev)
    xd, od = torch.from_numpy(x).to(dev), torch.from_numpy(off).to(dev)
    fe.run_f32(xd, od, off, o)
    n0 = dspfe.launch_count()
    dspfe.timing_begin()
    fe.run_f32(xd, od, off, o)
    marks = dspfe.timing_end()
    names = [n for n, _ in marks]
    assert "ep_stats_f32_kernel" in names and "ep_decide_kernel<f64>" in names
    assert "ep_block_kernel" not in names
    assert dspfe.launch_count() - n0 == len(marks)


def test_torch_op_dispatches_float32():
    import torch
    import dspfe
    import dspfe.torch_ops  # noqa: F401
    x, off = fe_batch()
    dev = torch.device("cuda:0")
    xd, od = torch.from_numpy(x).to(dev), torch.from_numpy(off).to(dev)
    got = torch.ops.dspfe.endpoint(xd, od, 16000)
    want = dspfe.EndpointPlan().detect_f32(xd, od)
    np.testing.assert_array_equal(got.cpu().numpy(), want.cpu().numpy())
    with pytest.raises(NotImplementedError):
        torch.ops.dspfe.endpoint(torch.from_numpy(x), torch.from_numpy(off), 16000)


def test_nan_sample_stays_in_its_utterance():
    import dspfe
    x, off = fe_batch()
    plan = dspfe.EndpointPlan()
    lr0, amp0, zcr0, fo = plan.detect_host_f32(x, off, want_features=True)
    u = 7
    y = x.copy()
    y[off[u] + (off[u + 1] - off[u]) // 2] = np.nan
    lr1, amp1, zcr1, fo1 = plan.detect_host_f32(y, off, want_features=True)
    others = [v for v in range(len(off) - 1) if v != u]
    np.testing.assert_array_equal(lr1[others], lr0[others])
    for v in others:
        np.testing.assert_array_equal(amp1[fo[v]:fo[v + 1]], amp0[fo[v]:fo[v + 1]])
        np.testing.assert_array_equal(zcr1[fo[v]:fo[v + 1]], zcr0[fo[v]:fo[v + 1]])
    F = int(fo[u + 1] - fo[u])
    assert 0 <= lr1[u, 0] <= lr1[u, 1] <= int(F * 0.01 * 16000)
