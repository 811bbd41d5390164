// Host-side constant tables of the pitch kernels (shared by libdspfe.so and the test emulator):
// parameter validation, the decimator pattern, W1024^k, the 1024-point spectrum of the FIR taps and the Bluestein chirp tables.
#pragma once
#include <cmath>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/dspfe.h"
#include "pitch_kernel.cuh"

namespace dspfe {

// FIR taps of sigproc.window (:33-44), float64: h = 2*pi * w * ifft(Hd), Hd = 1 on bins [int(N*lo/rate), int(N*hi/rate))
inline void fir_taps(int N, double rate, double lo, double hi, bool hamming, std::vector<double>& hr, std::vector<double>& hi_) {
    const double kPi = 3.14159265358979323846;
    int b0 = (int)((double)N * lo / rate), b1 = (int)((double)N * hi / rate);
    if (b0 < 0) b0 = 0;
    if (b1 > N) b1 = N;
    hr.assign(N, 0.0); hi_.assign(N, 0.0);
    for (int n = 0; n < N; ++n) {
        double sr = 0, si = 0;
        for (int b = b0; b < b1; ++b) { const double a = 2 * kPi * (double)((long long)b * n % N) / N; sr += cos(a); si += sin(a); }
        const double w = hamming ? (N > 1 ? 0.54 - 0.46 * cos(2 * kPi * n / (N - 1)) : 1.0) : 1.0;   // np.hamming
        hr[n] = 2 * kPi * w * sr / N; hi_[n] = 2 * kPi * w * si / N;
    }
}

// twiddles of fft512 (fft_regs.h): tws[r*32 + lane] = W512^{n2' (k1 + 16 kq)} for register r of lane 16 q + n2' after the
// radix-2 stage, (kq, k1) = (r >> 3, 8 q + (r & 7)), negated for q = kq = 1; w32[2*k1 + q] = W32^{q k1}
inline void fill_fft512_twiddles(float2* tws, float2* w32) {
    const double kPi = 3.14159265358979323846;
    for (int r = 0; r < 16; ++r)
        for (int lane = 0; lane < 32; ++lane) {
            const int q = lane >> 4, n2 = lane & 15, kq = r >> 3, k1 = 8 * q + (r & 7);
            const double a = -2 * kPi * (double)(n2 * (k1 + 16 * kq)) / 512.0;
            const float sg = q && kq ? -1.f : 1.f;
            tws[r * 32 + lane] = make_float2(sg * (float)cos(a), sg * (float)sin(a));
        }
    for (int k1 = 0; k1 < 16; ++k1) {
        w32[2 * k1] = make_float2(1.f, 0.f);
        w32[2 * k1 + 1] = make_float2((float)cos(-2 * kPi * k1 / 32.0), (float)sin(-2 * kPi * k1 / 32.0));
    }
}

// Bluestein tables of an N-point DFT, N <= 512, as a 1024-point circular convolution (pitch_cep_bluestein_pair), float64 rounded
// once: chirp[n] = w_n = exp(-i pi n^2 / N) for n < N, zero beyond; be[k] / bo[k] = bins 2k / 2k + 1 of FFT1024(b) with
// b[m] = b[1024 - m] = conj(w_m) for m < N, zero elsewhere.  n^2 is reduced mod 2N in integers, so every angle
// pi (n^2 mod 2N) / N lies in [0, 2 pi) and keeps its float64 precision for any n.
inline void fill_cep_bluestein_tables(int N, float2* chirp, float2* be, float2* bo) {
    const double kPi = 3.14159265358979323846;
    std::vector<double> wr(N), wi(N), cr(kPitchFft), ci(kPitchFft);
    for (int n = 0; n < N; ++n) {
        const double a = -kPi * (double)((long long)n * n % (2LL * N)) / N;
        wr[n] = cos(a); wi[n] = sin(a);
    }
    for (int n = 0; n < 512; ++n) chirp[n] = n < N ? make_float2((float)wr[n], (float)wi[n]) : make_float2(0.f, 0.f);
    for (int j = 0; j < kPitchFft; ++j) { cr[j] = cos(-2 * kPi * j / kPitchFft); ci[j] = sin(-2 * kPi * j / kPitchFft); }
    for (int k = 0; k < kPitchFft; ++k) {
        double sr = 0, si = 0;
        for (int m = 1 - N; m < N; ++m) {                          // b[m mod 1024] = conj(w_|m|)
            const int am = m < 0 ? -m : m, j = (int)(((long long)k * (m & (kPitchFft - 1))) & (kPitchFft - 1));
            sr += wr[am] * cr[j] + wi[am] * ci[j]; si += wr[am] * ci[j] - wi[am] * cr[j];
        }
        (k & 1 ? bo : be)[k >> 1] = make_float2((float)sr, (float)si);
    }
}

// Fills the scalar part of PitchParams and the two tables.  Returns 0 or a dspfe_status with `err` set.
inline int build_pitch_tables(const dspfe_pitch_params& q, PitchParams& b, std::vector<float2>& tab, std::string& err) {
    std::memset(&b, 0, sizeof(b));
    if (q.samplerate <= 0 || q.dst_rate <= 0 || q.frame_step < 1) { err = "bad pitch parameters"; return DSPFE_ERR_INVALID_ARG; }
    if (q.method != 0 && q.method != 1) { err = "method must be 0 (cepstrum) or 1 (autocorrelation)"; return DSPFE_ERR_INVALID_ARG; }
    // peak_score (pitch.py:227-242) reads row columns 20..99: the reference raises on shorter cepstrum frames
    if (q.method == 0 && (q.frame_len < kMinLag + kPeakLags || q.frame_len > kCepLen)) { err = "cepstrum frames must have 100..512 samples"; return DSPFE_ERR_UNSUPPORTED; }
    if (q.method == 1 && (q.frame_len <= kMinLag || q.frame_len > 512)) { err = "autocorrelation frames must have 21..512 samples"; return DSPFE_ERR_UNSUPPORTED; }
    if (q.frame_len + q.frame_step > kClipDecCap) { err = "frame_step too large: two frames must fit the clip kernel's sample buffer"; return DSPFE_ERR_UNSUPPORTED; }
    // decimator pattern (preprocess.py:21-28): the k-th kept sample (k >= 1) is floor((k-1)*src/dst) + 1
    if (q.dst_rate >= q.samplerate) { b.ds_in = 1; b.ds_out = 1; b.ds_idx[0] = 1; }
    else {
        long long a = q.samplerate, c = q.dst_rate;
        while (c) { const long long t = a % c; a = c; c = t; }
        b.ds_in = (int)(q.samplerate / a); b.ds_out = (int)(q.dst_rate / a);
        if (b.ds_out > kMaxDsOut) { err = "rate ratio needs a decimator pattern longer than 256"; return DSPFE_ERR_UNSUPPORTED; }
        for (int j = 0; j < b.ds_out; ++j) b.ds_idx[j] = (int)(((long long)j * b.ds_in) / b.ds_out) + 1;
    }
    b.frame_len = q.frame_len; b.frame_step = q.frame_step; b.do_clip = q.center_clip ? 1 : 0; b.mode = q.method;
    b.preemph = q.preemph;
    // cepstrum rows: columns 0..199 decide every peak score; a row shorter than that is the whole cepstrum (the right-hand
    // scan of peak_score ends at the frame length)
    b.row_len = q.method == 0 ? (q.row_len > 0 ? q.row_len : (q.frame_len < kCepCols ? q.frame_len : kCepCols)) : kAcrLags;
    if (q.method == 0 && (b.row_len < kPeakLags + kMinLag || b.row_len > q.frame_len)) { err = "row_len must be in 100..frame_len"; return DSPFE_ERR_INVALID_ARG; }
    b.ds_q32 = 32 / b.ds_out; b.ds_r32 = 32 % b.ds_out;
    b.pre_hi = (float)q.preemph; b.pre_lo = (float)(q.preemph - (double)b.pre_hi);
    // tables, float64 on the host, rounded once: the FFT twiddles, W1024^n and the even / odd bins of the 1024-point
    // spectrum of the FIR taps, all in natural order
    const double kPi = 3.14159265358979323846;
    tab.assign(kTabCepTotal, make_float2(0.f, 0.f));
    fill_fft512_twiddles(tab.data() + kTabTw, tab.data() + kTabW32);
    for (int n = 0; n < 512; ++n) tab[kTabMod + n] = make_float2((float)cos(-2 * kPi * n / 1024.0), (float)sin(-2 * kPi * n / 1024.0));
    std::vector<double> hr, hi;
    fir_taps(q.frame_len, (double)q.dst_rate, q.band_lo, q.band_hi, true, hr, hi);
    for (int k = 0; k < 512; ++k)
        for (int odd = 0; odd < 2; ++odd) {                       // even / odd bins of the 1024-point spectrum of the taps
            const int k1024 = 2 * k + odd;
            double sr = 0, si = 0;
            for (int n = 0; n < q.frame_len; ++n) {
                const double a = -2 * kPi * (double)((long long)k1024 * n % kPitchFft) / kPitchFft, c = cos(a), s_ = sin(a);
                sr += hr[n] * c - hi[n] * s_; si += hr[n] * s_ + hi[n] * c;
            }
            tab[(odd ? kTabHo : kTabHe) + k] = make_float2((float)sr, (float)si);
        }
    if (q.method == 0 && q.frame_len != kCepLen) fill_cep_bluestein_tables(q.frame_len, tab.data() + kTabChirp, tab.data() + kTabBe, tab.data() + kTabBo);
    if (q.method == 1 && acr_short_frames(q.frame_len, b.row_len)) {
        // pitch_acr_quad's split FIR: H_lo = FFT512(taps 0..T), H_hi = FFT512(taps T+1..L-1 left in place), T = 512 - L;
        // kTabHe <- A = (H_lo - i H_hi) / 2, kTabHo <- B = (H_lo + i H_hi) / 2, both with the inverse transform's 1/512
        const int L = q.frame_len, T = 512 - L;
        for (int k = 0; k < 512; ++k) {
            double lr = 0, li = 0, gr = 0, gi = 0;
            for (int n = 0; n < L; ++n) {
                const double a = -2 * kPi * (double)((long long)k * n % 512) / 512.0, c = cos(a), s_ = sin(a);
                const double tr = hr[n] * c - hi[n] * s_, ti = hr[n] * s_ + hi[n] * c;
                if (n <= T) { lr += tr; li += ti; } else { gr += tr; gi += ti; }
            }
            tab[kTabHe + k] = make_float2((float)((lr + gi) / 1024.0), (float)((li - gr) / 1024.0));
            tab[kTabHo + k] = make_float2((float)((lr - gi) / 1024.0), (float)((li + gr) / 1024.0));
        }
    }
    return 0;
}

}  // namespace dspfe
