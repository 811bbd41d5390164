"""GPU tests of the plans' workspaces, staging buffers, streams and events (csrc/abi_common.h): a plan run on a small batch,
then on one several times larger (every workspace and staging buffer regrows), then on the small one again gives the same
bits as a freshly created plan on each batch, on the device path and on the host-buffer path; and a front-end plan whose
creation fails after some of its sub-plans exist releases them, after which a new plan still gives the expected outputs."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MFCC_SLAB = 8 << 20        # dspfe_mfcc_delta_host's slab (kSlabSamples): a longer utterance is a slab of its own


def make_batch(n, seed, tiny=0, huge=0):
    """n ordinary utterances, with `tiny` 10-sample utterances in the middle (many per host slab: the per-utterance staging
    grows past its floor) and one `huge`-sample utterance at the end."""
    from dspfe import synth
    lengths = list(synth.ragged_lengths(n, seed=seed, lo=6000, hi=50000))
    lengths = lengths[: n // 2] + [10] * tiny + lengths[n // 2:] + ([huge] if huge else [])
    return synth.synth_batch(lengths, seed0=100 * seed)


def small():
    return make_batch(6, 1)


def large(**kw):
    return make_batch(40, 2, **kw)


def assert_same(got, want, what):
    assert got.keys() == want.keys()
    for k in want:
        np.testing.assert_array_equal(got[k], want[k], err_msg=f"{what}: {k}")


def check_growth(new_plan, run, batches, what):
    """run(plan, pcm, off) -> dict of NumPy arrays; one plan over the batches in turn equals a fresh plan on each."""
    plan = new_plan()
    for i, (pcm, off) in enumerate(batches):
        assert_same(run(plan, pcm, off), run(new_plan(), pcm, off), f"{what}, batch {i}")


def cuda(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


@pytest.mark.parametrize("nfft", [512, 1536, 1024])    # K1, K1T and the general kernel K1L (its cepstrum workspace)
def test_mfcc_plan_growth(nfft):
    import dspfe

    def dev(plan, pcm, off):
        out, fo = plan.mfcc_delta(*cuda(pcm, off))
        fo = fo.cpu().numpy()
        return dict(mfcc=out[: fo[-1]].cpu().numpy(), frame_off=fo)

    def host(plan, pcm, off):
        out, fo = plan.mfcc_delta_host(pcm, off)
        return dict(mfcc=out, frame_off=fo)

    s = small()
    check_growth(lambda: dspfe.MfccPlan(nfft=nfft), dev, [s, large(), s], f"MFCC nfft {nfft}, device path")
    # more utterances than a host slot's floor (4096) in one slab, then a slab longer than its floor (kSlabSamples + 8)
    check_growth(lambda: dspfe.MfccPlan(nfft=nfft), host, [s, large(tiny=5000, huge=MFCC_SLAB + 1000), s],
                 f"MFCC nfft {nfft}, host path")


@pytest.mark.parametrize("robust", [False, True])
def test_endpoint_plan_growth(robust):
    import dspfe

    def dev(plan, pcm, off):
        lr = (plan.detect_robust if robust else plan.detect)(*cuda(pcm, off))
        return dict(lr=lr.cpu().numpy())

    def host(plan, pcm, off):
        if robust:
            return dict(lr=plan.detect_robust_host(pcm, off))
        lr, asum, zcr, fo = plan.detect_host(pcm, off, want_features=True)
        return dict(lr=lr, asum=asum, zcr=zcr, frame_off=fo)

    s = small()
    for run, path in ((dev, "device"), (host, "host")):
        check_growth(dspfe.EndpointPlan, run, [s, large(), s], f"{'robust' if robust else 'basic'} endpoints, {path} path")


@pytest.mark.parametrize("method", [0, 1])
def test_pitch_plan_growth(method):
    import dspfe
    feat = method == 0

    def trim_of(off):
        n = np.diff(off)
        return np.stack([n // 10, n - n // 10], axis=1).astype(np.int32)

    def dev(plan, pcm, off):
        o = plan.detect(*cuda(pcm, off), trim=cuda(trim_of(off))[0], want_feat=feat)
        fo = o["frame_off"].cpu().numpy()
        r = dict(pitch=o["pitch"][: fo[-1]].cpu().numpy(), lag=o["lag"][: fo[-1]].cpu().numpy(), frame_off=fo)
        if feat:
            r["feat"] = o["feat"].cpu().numpy()
        return r

    def host(plan, pcm, off):
        return dict(zip(("pitch", "lag", "frame_off", "feat"), plan.detect_host(pcm, off, trim=trim_of(off), want_feat=feat)))

    s = small()
    for run, path in ((dev, "device"), (host, "host")):
        check_growth(lambda: dspfe.PitchPlan(method=method), run, [s, large(), s], f"pitch method {method}, {path} path")


FE_KEYS = dict(mfcc=0, cep_pitch=1, cep_lag=1, acr_pitch=2, acr_lag=2)      # row arrays and the total that bounds them


def fe_to_np(o, tot):
    arr = lambda t: t.cpu().numpy() if hasattr(t, "cpu") else np.asarray(t)
    return {k: arr(v)[: tot[FE_KEYS[k]]] if k in FE_KEYS else arr(v) for k, v in o.items()}


def test_frontend_plan_growth():
    """Device path in slabs of 100000 samples; host path in slabs of 20000 samples, so a batch spans many more slabs than
    the plan has staging slots (kFeSlots = 3) and both lanes, and the tiny utterances put about 2000 utterances in a slab
    (the slots' floor is 1024)."""
    import torch
    import dspfe

    def dev(plan, pcm, off):
        o = plan.alloc(len(pcm), len(off) - 1, device=torch.device("cuda:0"))
        tot = plan.run(*cuda(pcm, off), off, o)
        torch.cuda.synchronize()
        return fe_to_np(o, tot)

    def host(plan, pcm, off):
        o = plan.alloc(len(pcm), len(off) - 1, device=None, pinned=True)
        return fe_to_np(o, plan.run_host(pcm, off, o))

    s, big = small(), large(tiny=3000)
    check_growth(lambda: dspfe.FrontendPlan(slab_samples=100000), dev, [s, big, s], "front-end, device path")
    check_growth(lambda: dspfe.FrontendPlan(host_slab_samples=20000), host, [s, big, s], "front-end, host path")


def test_frontend_create_failure_releases_sub_plans():
    """At 11025 Hz the pitch decimator (11025 -> 10000) is not built: the front-end's creation fails after its endpoint and
    MFCC sub-plans exist.  Those are released with the partial plan, and a valid plan created next still works."""
    import torch
    import dspfe
    from dspfe.binding import DspfeUnsupported
    pcm, off = small()

    def run():
        fe = dspfe.FrontendPlan()
        o = fe.alloc(len(pcm), len(off) - 1, device=torch.device("cuda:0"))
        tot = fe.run(*cuda(pcm, off), off, o)
        torch.cuda.synchronize()
        return fe_to_np(o, tot)

    want = run()
    with pytest.raises(DspfeUnsupported):
        dspfe.FrontendPlan(samplerate=11025)
    assert_same(run(), want, "front-end after a failed create")
