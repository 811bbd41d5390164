"""fft512 (csrc/fft_regs.h), the 512-point transform of a packed frame pair that every pitch chain and the long-frame MFCC
kernel call, on its own on the CPU SIMT emulator (emu_fft512, tests/emu/emu_fft512.cpp): forward and inverse against NumPy's
float64 FFT, independence of the two frames of a pair, and the register layout of the result."""
import ctypes
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu"))
import emu  # noqa: E402


def fft512(a, b, inverse=False):
    """Both frames through one warp's fft512; returns the two 512-point results as complex64 in natural order
    (bin k = 32 * register + lane)."""
    x = np.empty((2, 512, 2), dtype=np.float32)
    x[0, :, 0], x[0, :, 1] = a.real, a.imag
    x[1, :, 0], x[1, :, 1] = b.real, b.imag
    out = np.empty_like(x)
    rc = emu.lib().emu_fft512(x.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p), int(inverse))
    assert rc == 0
    y = out[..., 0].astype(np.float64) + 1j * out[..., 1].astype(np.float64)
    return y[0], y[1]


def random_frame(rng, scale=1.0):
    return (rng.standard_normal(512) * scale + 1j * rng.standard_normal(512) * scale).astype(np.complex64)


@pytest.mark.parametrize("seed", range(4))
def test_forward_and_inverse_match_numpy(seed):
    rng = np.random.default_rng(seed)
    a, b = random_frame(rng), random_frame(rng, scale=1e3)
    for inverse in (False, True):
        ya, yb = fft512(a, b, inverse)
        for x, y in ((a, ya), (b, yb)):
            x64 = x.astype(np.complex128)
            ref = 512 * np.fft.ifft(x64) if inverse else np.fft.fft(x64)
            assert np.max(np.abs(y - ref)) <= 2e-6 * np.max(np.abs(ref)), (inverse, np.max(np.abs(y - ref)) / np.max(np.abs(ref)))


def test_real_frames_and_impulses():
    rng = np.random.default_rng(11)
    a = rng.standard_normal(512).astype(np.complex64)             # the chains' forward transforms see real frames
    b = np.zeros(512, dtype=np.complex64)
    b[37] = 1.0
    ya, yb = fft512(a, b)
    ref = np.fft.fft(a.astype(np.complex128))
    assert np.max(np.abs(ya - ref)) <= 2e-6 * np.max(np.abs(ref))
    assert np.max(np.abs(yb - np.exp(-2j * np.pi * 37 * np.arange(512) / 512))) <= 2e-6


@pytest.mark.parametrize("inverse", [False, True])
def test_frames_of_a_pair_are_independent(inverse):
    """The .x frame's result does not depend on the .y frame, to the bit."""
    rng = np.random.default_rng(5)
    a = random_frame(rng)
    ya0, yb0 = fft512(a, np.zeros(512, dtype=np.complex64), inverse)
    ya1, _ = fft512(a, random_frame(rng, scale=1e4), inverse)
    assert np.array_equal(ya0.view(np.float64), ya1.view(np.float64))
    assert not np.any(yb0)


def test_output_layout():
    """Bin k = k1 + 16 kq + 32 k2' leaves in lane 16 kq + k1, register k2': an impulse at bin k of the inverse transform's
    input comes out of the forward transform of exp(2 pi i k n / 512) at (register k >> 5, lane k & 31) alone."""
    n = np.arange(512)
    for k in (0, 1, 15, 16, 17, 31, 32, 255, 256, 300, 497, 511):
        x = np.exp(2j * np.pi * k * n / 512).astype(np.complex64)
        y, _ = fft512(x, np.zeros(512, dtype=np.complex64))
        regs = y.reshape(16, 32)                                  # [register, lane]
        k1, kq, k2 = k & 15, (k >> 4) & 1, k >> 5
        assert abs(regs[k2, 16 * kq + k1] - 512) < 1e-3
        mask = np.ones((16, 32), dtype=bool)
        mask[k2, 16 * kq + k1] = False
        assert np.max(np.abs(regs[mask])) < 1e-3
