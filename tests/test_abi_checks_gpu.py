"""GPU tests of the argument checks the batched entry points share (include/dspfe.h): for every device form, null and
misaligned samples, a negative or empty batch and a plan that cannot run the call; for every host form, a decreasing
interior offset.  A rejected call queues nothing, so launch_count() does not move.  Also the launch counts of the robust
endpoint host forms: the batch is staged once and the device form runs once."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

OK, INVALID, UNSUPPORTED = 0, -1, -2
LENGTHS = [4000, 2400, 5600]


@pytest.fixture(scope="module")
def env():
    import torch
    from dspfe import binding as B
    from dspfe import synth
    L = B.lib()
    B._bind_endpoint(L); B._bind_endpoint_f32(L); B._bind_helpers(L); B._bind_pitch(L); B._bind_frontend(L)
    dev = torch.device("cuda:0")
    pcm, off = synth.synth_batch(LENGTHS, seed0=41)
    x = (pcm.astype(np.float32) * 0.5)
    e = dict(L=L, B=B, torch=torch, pcm=pcm, x=x, off=off, total=int(off[-1]), n=len(LENGTHS),
             st=ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    e["d_pcm"] = torch.from_numpy(pcm).to(dev)
    e["d_x"] = torch.from_numpy(x).to(dev)
    e["d_off"] = torch.from_numpy(off).to(dev)
    big = 1 << 20
    e["d_f32"] = torch.empty(big, dtype=torch.float32, device=dev)
    e["d_f64"] = torch.empty(big, dtype=torch.float64, device=dev)
    e["d_i32"] = torch.empty(big, dtype=torch.int32, device=dev)
    e["d_i64"] = torch.empty(big, dtype=torch.int64, device=dev)
    e["mfcc"] = B.MfccPlan()
    e["ep"] = B.EndpointPlan()
    e["ep_f32_long"] = B.EndpointPlan(cfg_frame=0.6)       # 9600-sample frames: above the float path's 8192
    e["ep_robust_long"] = B.EndpointPlan(cfg_frame=0.1)    # 1600-sample frames: above the robust gate's 1536
    e["cep"] = B.PitchPlan(method=0)
    e["acr"] = B.PitchPlan(method=1, frame_len=300)
    e["fe"] = B.FrontendPlan()
    yield e
    torch.cuda.synchronize()


def samples(e, dtype, case):
    """(pointer, total samples, n_utt) of the device batch for one case."""
    t = e["d_pcm"] if dtype == "i16" else e["d_x"]
    ptr, total, n = t.data_ptr(), e["total"], e["n"]
    if case == "null":
        ptr = None
    elif case == "misaligned":
        ptr += t.element_size()
        total -= 1
    elif case == "negative":
        n = -1
    elif case == "empty":
        n = 0
    return ptr, total, n


def call_device(e, name, case, plan=None):
    L, st = e["L"], e["st"]
    dtype = "f32" if name.endswith("_f32") or name in ("fbank_f32", "spectrum_f32") else "i16"
    ptr, total, n = samples(e, dtype, case)
    off, f32, f64, i32, i64 = (e[k].data_ptr() for k in ("d_off", "d_f32", "d_f64", "d_i32", "d_i64"))
    cap = 1 << 16
    if name in ("mfcc_delta", "mfcc_delta_f32"):
        return getattr(L, "dspfe_" + name)(e["mfcc"]._h, ptr, total, off, None, n, f32, cap, i64, st)
    if name == "fbank_f32":
        return L.dspfe_fbank_f32(e["mfcc"]._h, ptr, total, off, n, f32, cap, i64, st)
    if name == "spectrum_f32":
        return L.dspfe_spectrum_f32(e["mfcc"]._h, ptr, total, off, n, 0, f32, cap, i64, st)
    if name in ("endpoint", "endpoint_f32"):
        stat = i32 if name == "endpoint" else f64
        return getattr(L, "dspfe_" + name)((plan or e["ep"])._h, ptr, total, off, n, i32, stat, i32 + 4 * cap, i64, cap, st)
    if name in ("endpoint_robust", "endpoint_robust_f32"):
        return getattr(L, "dspfe_" + name)((plan or e["ep"])._h, ptr, total, off, n, i32, st)
    if name in ("pitch", "pitch_f32"):
        feat = f64 + 8 * 2 * cap if plan is not None else None
        return L.dspfe_pitch((plan or e["cep"])._h, ptr, 0 if name == "pitch" else 1, total, off, None, n, f64, i32, feat,
                             None, i64, cap, st)
    if name in ("frontend", "frontend_f32"):
        out = e["B"]._FrontendOut()
        return getattr(L, "dspfe_" + name)(e["fe"]._h, ptr, off, e["off"].ctypes.data, n, ctypes.byref(out), None, st)
    raise KeyError(name)


DEVICE = ["mfcc_delta", "mfcc_delta_f32", "fbank_f32", "spectrum_f32", "endpoint", "endpoint_f32", "endpoint_robust",
          "endpoint_robust_f32", "pitch", "pitch_f32", "frontend", "frontend_f32"]
CASES = [("null", INVALID), ("misaligned", INVALID), ("negative", INVALID), ("empty", OK)]


@pytest.mark.parametrize("name", DEVICE)
@pytest.mark.parametrize("case,code", CASES)
def test_device_batch_check(env, name, case, code):
    e = env
    n0 = e["B"].launch_count()
    rc = call_device(e, name, case)
    assert rc == code, (name, case, e["L"].dspfe_last_error())
    assert e["B"].launch_count() == n0


# plans that cannot run the entry point: endpoint frames above the float path's 8192 or the robust gate's 1536 samples,
# checked before the empty-batch return; pitch_feature on an autocorrelation plan
UNSUPPORTED_PLANS = [("endpoint_f32", "ep_f32_long", "full"), ("endpoint_f32", "ep_f32_long", "empty"),
                     ("endpoint_robust", "ep_robust_long", "full"), ("endpoint_robust", "ep_robust_long", "empty"),
                     ("endpoint_robust_f32", "ep_robust_long", "full"), ("endpoint_robust_f32", "ep_robust_long", "empty"),
                     ("pitch", "acr", "full")]


@pytest.mark.parametrize("name,plan,case", UNSUPPORTED_PLANS)
def test_device_unsupported_plan(env, name, plan, case):
    e = env
    n0 = e["B"].launch_count()
    rc = call_device(e, name, case, plan=e[plan])
    assert rc == UNSUPPORTED, (name, case, e["L"].dspfe_last_error())
    assert e["B"].launch_count() == n0


HOST = ["mfcc_delta_host", "endpoint_host", "endpoint_host_f32", "endpoint_robust_host", "endpoint_robust_host_f32",
        "pitch_host", "pitch_host_f32", "frontend_host", "frontend_host_f32"]


@pytest.mark.parametrize("name", HOST)
def test_host_decreasing_offset(env, name):
    e = env
    L = e["L"]
    off = e["off"].copy()
    off[1], off[2] = off[2], off[1]               # an interior offset goes back; the batch's total stays positive
    assert off[-1] > off[0] and off[2] < off[1]
    h = (e["x"] if name.endswith("_f32") else e["pcm"]).ctypes.data
    o = off.ctypes.data
    n = len(off) - 1
    f64 = np.zeros(1 << 16, dtype=np.float64)
    i32 = np.zeros(1 << 16, dtype=np.int32)
    i64 = np.zeros(n + 1, dtype=np.int64)
    n0 = e["B"].launch_count()
    if name == "mfcc_delta_host":
        rc = L.dspfe_mfcc_delta_host(e["mfcc"]._h, h, o, n, np.zeros(1 << 16, dtype=np.float32).ctypes.data, i64.ctypes.data)
    elif name in ("endpoint_host", "endpoint_host_f32"):
        rc = getattr(L, "dspfe_" + name)(e["ep"]._h, h, o, n, i32.ctypes.data, None, None, i64.ctypes.data)
    elif name.startswith("endpoint_robust_host"):
        rc = getattr(L, "dspfe_" + name)(e["ep"]._h, h, o, n, i32.ctypes.data)
    elif name.startswith("pitch_host"):
        rc = L.dspfe_pitch_host(e["cep"]._h, h, 1 if name.endswith("_f32") else 0, o, None, n, f64.ctypes.data, i32.ctypes.data,
                                None, i64.ctypes.data)
    else:
        rc = getattr(L, "dspfe_" + name)(e["fe"]._h, h, o, n, ctypes.byref(e["B"]._FrontendOut()), None)
    assert rc == INVALID, (name, L.dspfe_last_error())
    assert L.dspfe_last_error() == b"offsets must be non-decreasing"
    assert e["B"].launch_count() == n0


@pytest.mark.parametrize("dtype,launches", [("i16", 5), ("f32", 4)])
def test_robust_host_launches_once(env, dtype, launches):
    """The host form stages the batch and runs the device form once: as many launches as the device form, the same lr."""
    e = env
    plan, B = e["ep"], e["B"]
    if dtype == "i16":
        dev = lambda: plan.detect_robust(e["d_pcm"], e["d_off"]).cpu().numpy()
        host = lambda: plan.detect_robust_host(e["pcm"], e["off"])
    else:
        dev = lambda: plan.detect_robust_f32(e["d_x"], e["d_off"]).cpu().numpy()
        host = lambda: plan.detect_robust_host_f32(e["x"], e["off"])
    n0 = B.launch_count()
    lr_d = dev()
    n1 = B.launch_count()
    lr_h = host()
    n2 = B.launch_count()
    assert n1 - n0 == launches
    assert n2 - n1 == launches
    np.testing.assert_array_equal(lr_h, lr_d)
