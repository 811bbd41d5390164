// K4/K5/K6: cepstrum pitch, autocorrelation pitch and the pitch-feature tail over a ragged batch (sm_100a).
//
// Replaces reference features/pitch.py: pitch_detect (:83), pitch_detect_sr (:96), pitch_detect_frame (:135),
// pitch_detect_frame_sr (:112), center_clip (:145), smooth (:157), peak_score (:227), max_pitch (:166),
// robust_max_pitch (:191), pitch_feature (:26) with sub_endpoint_detect (:64), find_smooth_subsequence (:245),
// slope/quad_params/peakshift (:49-62); plus preprocess.downsampling (:21) and sigproc.window (:22), acr (:48).
//
//   K4a/K5a  one warp per 10 kHz frame: gather the frame through the sample-picking decimator (no filter, as
//            the reference), centre-clip at the median of its non-negative samples (exact bitwise selection),
//            apply the one-sided (complex) FIR band-pass as a 1024-point FFT product, then
//              cepstrum:        FFT512 -> log|.| -> IFFT512 -> |.|            -> row of row_len (<= 512) columns
//                               (frames of 100..511 samples: N-point DFTs by Bluestein's chirp, pitch_cep_bluestein_pair)
//              autocorrelation: |y| -> FFT1024 -> |.|^2 -> IFFT1024 -> /(L-n) -> row of 180 lags (20..199)
//   K4b/K5b  one CTA per utterance walks its frames in order, 16 at a time: the reference's in-place running
//            mean (a recurrence over already-smoothed rows, one column per thread), then peak scoring / argmax
//            for the 16 rows in parallel, finally the octave-repair sweeps.
//   K6       one thread per utterance: valley split, longest smooth runs, least-squares slope / curvature and
//            median shift -> the five SVM inputs of pitch_model.py.
#pragma once
#include <math.h>
#include <stdint.h>

#include "simt.h"
#include "fft_regs.h"
#ifndef DSPFE_EMU
#include <cuda_fp16.h>
#endif

#ifndef DSP_HD
#ifdef __CUDACC__
#define DSP_HD __host__ __device__ inline
#else
#define DSP_HD inline
#endif
#endif

namespace dspfe {

constexpr int kPitchFft = 1024;
constexpr int kCepLen = 512;        // cepstrum length (frame length of pitch_detect)
constexpr int kCepCols = 200;       // columns peak_score can reach: lags 20..99 look at most 99 samples either side
constexpr int kAcrLags = 180;       // lags 20..199 (pitch.py:125-129)
constexpr int kMinLag = 20;
constexpr int kPeakLags = 80;       // peak_score evaluates lags 20..99 (pitch.py:232)
constexpr int kMaxDsOut = 256;      // decimator pattern length limit
constexpr int kPitchWarps = 4;      // warps per CTA in K4a/K5a, each carrying a pair of frames
constexpr int kWarpScr = 32 * 17;       // fft512's padded 32x16 transpose tile (float2)
constexpr int kWarpSmemBytes = kWarpScr * 8 + 512 * 16;              // transform kernel: transpose tile | parked spectrum
// table blob offsets, in float2.  The W32 slot is read by no kernel since fft512 takes W32 from immediates; the frame pair
// bodies and the emulator entry points that call them still pass a pointer to it.
constexpr int kTabTw = 0, kTabW32 = kTabTw + 512, kTabMod = kTabW32 + 32, kTabHe = kTabMod + 512, kTabHo = kTabHe + 512,
              kTabTotal = kTabHo + 512;
// the Bluestein tables of pitch_cep_bluestein_pair follow the blob above (filled for cepstrum frames other than 512 samples):
// the chirp w_n = exp(-i pi n^2 / N) for n < N (zero beyond) and the even / odd bins of the 1024-point spectrum of conj(w) wrapped
constexpr int kTabChirp = kTabTotal, kTabBe = kTabChirp + 512, kTabBo = kTabBe + 512, kTabCepTotal = kTabBo + 512;
constexpr int kFrameCtaSmem = (kTabMod * 8) + kPitchWarps * kWarpSmemBytes;                      // shared tables | per-warp areas
constexpr int kClipRun = 8;         // frames per warp of K4a-1, and the padding unit of the slot space (even: pairs never straddle two runs)
constexpr int kTrackThreads = 256;
constexpr int kTrackMaxFrames = 1024;   // utterances up to this many frames keep their lag / Hz track in shared memory
constexpr int kTrackChunk = 32;     // frames smoothed per pass of K4b/K5b (16 for rows wider than 256 columns); 16-frame passes at 8 CTAs/SM
                                    // measured slower (0.68 + 0.41 ms against 0.62 + 0.39 ms)
// autocorrelation rows of lags kMinLag .. kMinLag + row_len - 1: no wrap-around in a 512-point circular correlation
DSP_HD bool acr_short_frames(int frame_len, int row_len) { return frame_len + kMinLag + row_len - 1 <= 512; }
DSP_HD int track_chunk(int row_len) { return row_len <= 256 ? kTrackChunk : kTrackChunk / 2; }

struct PitchParams {
    const void* pcm; int in_f32;         // packed samples: int16 or float32 (16-byte aligned base)
    int64_t total_samples;
    const int64_t* offsets;              // [U+1]
    const int32_t* trim;                 // optional [U,2] (left,right): pitch runs on sig[left:right]
    int n_utt;
    double preemph;                      // y[n] = x[n] - c x[n-1] over the WHOLE utterance before trimming (pitch_model.py:39-41); 0 = off
    int ds_in, ds_out;                   // decimator: output k >= 1 reads input ((k-1)/ds_out)*ds_in + ds_idx[(k-1)%ds_out]
    int32_t ds_idx[kMaxDsOut];
    int frame_len, frame_step;           // at the decimated rate: 512/100 (or 300/100 for the autocorrelation variant)
    int do_clip;                         // center_clip(frame, False) before the band-pass (pitch.py:88,103)
    int no_smooth;                       // taps only: K4b/K5b score the rows as given (peak_score on its own)
    const float2* tab;                   // table blob (kTab* offsets): W512 twiddles, W32, W1024^n, He, Ho (+ chirp, Be, Bo)
    float pre_hi, pre_lo;                // preemph split into float32 head + tail
    int ds_q32, ds_r32;                  // 32 / ds_out, 32 % ds_out
    int mode;                            // 0 cepstrum, 1 autocorrelation
    int row_len;                         // columns per row: cepstrum 200 (fused) or 512 (tap); autocorrelation 180
    int64_t* frame_off;                  // [U+1] prefix sums of pitch frames
    int64_t* slot_off;                   // [U+1] prefix sums of the frame counts rounded up to kClipRun: the work units of K4a/K5a (runs of 8,
                                         //       quads, pairs) are cut in this padded index space, so none of them straddles two utterances and a
                                         //       frame's result does not depend on what else is in the batch
    int64_t* seg_start; int32_t* seg_len; int32_t* ds_len;   // per utterance: trimmed range and decimated length
    float2* clip;                        // [slots/2, 512] clipped frame pairs in slot order (K4a-1 -> K4a-2)
    int4* run_desc;                      // [slots/kClipRun] per run of slots: (first global frame lo, hi, frames that exist, utterance), written by K4a-1
    float* rows;                         // [F_total, row_len] raw rows (K4a/K5a output)
    float* rows_out;                     // optional: smoothed rows (tap of smooth, pitch.py:157)
    int32_t* score;                      // optional [F_total, 80]: peak_score of every smoothed row (tap)
    double* frame_amp;                   // [F_total] sum |x| of each raw frame (sub_endpoint_detect, pitch.py:65)
    double* pitch;                       // [F_total] Hz after robust_max_pitch
    int32_t* lag;                        // [F_total] 20 + argmax (before octave repair)
    double* feat;                        // [U,5] pitch_feature, or null
    double* scratch;                     // [3*F_total] K6 work area
    int64_t max_frames;
    const int32_t* order;                // optional [U]: the utterances by descending frame count (the CTA-per-utterance kernels take
                                         //   them in this order, longest first: no long utterance is left to run alone at the end); null = identity
};

// ---------------------------------------------------------------------------------------------------------
// host/device scalar pieces
// ---------------------------------------------------------------------------------------------------------
// number of decimated samples of an S-sample signal (preprocess.py:21-28: sample 0 is always kept, sample i > 0
// is the k-th kept one when it is the first with i*dst/src > k-1)
DSP_HD int64_t ds_length(int64_t S, const int32_t* ds_idx, int ds_in, int ds_out) {
    if (S <= 0) return 0;
    const int64_t T = S - 1, q = T / ds_in;
    int64_t n = 1 + q * ds_out;
    for (int i = 0; i < ds_out; ++i) n += ((int64_t)ds_idx[i] <= T - q * ds_in) ? 1 : 0;
    return n;
}
DSP_HD int64_t ds_index(int64_t k, const int32_t* ds_idx, int ds_in, int ds_out) {
    if (k <= 0) return 0;
    const int64_t j = k - 1;
    return (j / ds_out) * ds_in + ds_idx[j % ds_out];
}

// robust_max_pitch (pitch.py:191-206) on lags: p = 1/(0.0001*lag), forward then backward octave repair
DSP_HD void robust_pitch(const int32_t* lag, int F, double* pitch) {
    for (int i = 0; i < F; ++i) pitch[i] = 1.0 / (0.0001 * (double)lag[i]);
    for (int i = 1; i < F; ++i)
        if (fabs(2 * pitch[i] - pitch[i - 1]) < 50 && pitch[i] < 170) pitch[i] = 2 * pitch[i];
    for (int i = F - 2; i > 0; --i)
        if (fabs(2 * pitch[i] - pitch[i + 1]) < 50 && pitch[i] < 170) pitch[i] = 2 * pitch[i];
}

// find_smooth_subsequence (pitch.py:245-279): longest run (first on ties) tolerating `tor` jumps > thres.
// Writes the run's accepted values to seg and returns its length; *i0/*j0 = the run's (start, stop) indices.
DSP_HD int smooth_run(const double* pitch, int n, int tor, double thres, double* seg, double* tmp, int* i0, int* j0) {
    int best = 0, i = 0;
    *i0 = 0; *j0 = 0;
    while (i < n) {
        int j = i + 1, k = tor, len = 1;
        double prev = pitch[i];
        tmp[0] = pitch[i];
        bool closed = false;
        while (j < n) {
            if (fabs(pitch[j] - prev) > thres) --k;
            else { tmp[len++] = pitch[j]; prev = pitch[j]; }
            if (!k) { closed = true; break; }
            ++j;
        }
        if (len > best) { best = len; *i0 = i; *j0 = j; for (int q = 0; q < len; ++q) seg[q] = tmp[q]; }
        if (!closed) break;      // reached the end of the sequence
        i = j - tor + 1;
    }
    return best;
}

// least-squares polynomial leading coefficients over x = 0..n-1 (np.polyfit(x, seq, deg)[0]); closed-form
// normal equations about the centred abscissa (odd moments vanish)
DSP_HD double ls_slope(const double* y, int n) {
    const double xm = 0.5 * (n - 1);
    double s2 = 0, t1 = 0;
    for (int i = 0; i < n; ++i) { const double x = i - xm; s2 += x * x; t1 += x * y[i]; }
    return t1 / s2;
}
DSP_HD double ls_quad(const double* y, int n) {
    const double xm = 0.5 * (n - 1);
    double s2 = 0, s4 = 0, t0 = 0, t2 = 0;
    for (int i = 0; i < n; ++i) { const double x = i - xm, x2 = x * x; s2 += x2; s4 += x2 * x2; t0 += y[i]; t2 += x2 * y[i]; }
    return (n * t2 - s2 * t0) / (n * s4 - s2 * s2);   // [s4 s2; s2 n] [a; c] = [t2; t0]
}
DSP_HD double median_inplace(double* a, int n) {   // np.median
    for (int i = 1; i < n; ++i) { double v = a[i]; int j = i - 1; while (j >= 0 && a[j] > v) { a[j + 1] = a[j]; --j; } a[j + 1] = v; }
    return (n & 1) ? a[n / 2] : 0.5 * (a[n / 2 - 1] + a[n / 2]);
}

// sub_endpoint_detect (pitch.py:64-81) on the per-frame sum |x|
DSP_HD int sub_endpoint(const double* amp, int F) {
    int p = 0; double max_score = -1000;
    for (int i = 10; i < F - 10; ++i) {
        bool lower = false;
        for (int j = i - 2; j <= i + 2; ++j) lower = lower || (amp[j] < amp[i]);
        if (lower) continue;
        double s = 0;
        for (int j = i - 10; j <= i + 10; ++j) s += amp[j] - amp[i];
        if (s > max_score) { max_score = s; p = i; }
    }
    return p == 0 ? F / 2 : p;
}

// pitch_feature (pitch.py:26-47) after pitch_detect: amp = sum|x| per raw frame, pitch = Hz per frame.
// work: 3*F doubles.  A half with fewer than three accepted values has no defined curvature: the five
// outputs are NaN and false is returned (the reference raises or returns a minimum-norm fit there).
DSP_HD bool pitch_feature_tail(const double* pitch, const double* amp, int F, double* work, double* out5) {
    const int p = sub_endpoint(amp, F);
    const int p_bias = p > 15 ? 5 : 0;
    double* s1 = work; double* s2 = work + F; double* tmp = work + 2 * F;
    int a, b;
    const int n1 = smooth_run(pitch + p_bias, p - p_bias, 3, 30.0, s1, tmp, &a, &b);
    const int n2 = smooth_run(pitch + p, F - p, 3, 30.0, s2, tmp, &a, &b);
    if (n1 < 3 || n2 < 3) { for (int i = 0; i < 5; ++i) out5[i] = NAN; return false; }
    out5[0] = ls_slope(s1, n1); out5[1] = ls_slope(s2, n2);
    out5[2] = ls_quad(s1, n1); out5[3] = ls_quad(s2, n2);
    const double m1 = median_inplace(s1, n1), m2 = median_inplace(s2, n2);
    out5[4] = m2 - m1;   // peakshift(seq1, seq2) = median(seq2) - median(seq1)
    return true;
}

// ---------------------------------------------------------------------------------------------------------
// warp-cooperative pieces (device + emulator)
// ---------------------------------------------------------------------------------------------------------
// medians of the non-negative entries of two frames at once (np.median(frame[frame >= 0]), pitch.py:146): exact k-th
// order statistics by a bit-sliced radix selection on the float bit patterns; NaN when a frame has no non-negative sample.
// NT = samples per lane (32 * NT >= L): 16 for 512-sample frames, 10 for frames of up to 320 samples.
// Transposes two independent 16 x 16 bit matrices at once: A[r] holds row r of one matrix in its low 16 bits and row r of the
// other in its high 16 bits (Hacker's Delight's masked-swap transpose, masks replicated in both halves; the shifts never
// carry a bit across the halves because every mask clears the top j bits of each half).  Afterwards A[i] holds, per half,
// the plane of bit 15 - i: its bit 15 - r is bit 15 - i of the original row r.
DEVFN void transpose16_dual(unsigned (&A)[16]) {
    unsigned m = 0x00ff00ffu;
#pragma unroll
    for (int j = 8; j != 0; j >>= 1) {
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            if ((k & j) == 0) {
                const unsigned t = (A[k] ^ (A[k + j] >> j)) & m;
                A[k] ^= t;
                A[k + j] ^= t << j;
            }
        }
        m ^= m << (j >> 1);
    }
}
// Integer-valued samples in [0, 32767] (int16 PCM that was neither pre-emphasised nor scaled): 15-bit keys -- one bit-matrix
// transpose and 15 selection steps instead of two and 31.
template <int NT>
DEVFN float2 warp_median_nonneg2_i16(const float (&xa)[NT], const float (&xb)[NT], int L, int lane) {
    unsigned ka[NT], kb[NT];
    int cnt = 0, cntb = 0;
    const bool full = L >= 32 * NT;
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        const float va = xa[t], vb = xb[t];
        const bool in = full || (lane + 32 * t) < L;
        const bool na = in & (va >= 0.f), nb = in & (vb >= 0.f);
        // value + 2^23 has the integer in its low mantissa bits (exact for 0 <= value < 2^23)
        ka[t] = na ? ((unsigned)__float_as_int_compat(va + 8388608.0f) & 0x7fffu) : 0xffffu;
        kb[t] = nb ? ((unsigned)__float_as_int_compat(vb + 8388608.0f) & 0x7fffu) : 0xffffu;
        cnt += na; cntb += nb;
    }
    cnt = warp_redux_add(cnt + (cntb << 16));
    const int ma = cnt & 0xffff, mb = cnt >> 16;
    int rA = (ma - 1) >> 1, rB = (mb - 1) >> 1;
    unsigned Ka = 0, Kb = 0;
    {
        unsigned P[16];
#pragma unroll
        for (int t = 0; t < 16; ++t) P[t] = t < NT ? (ka[t < NT ? t : 0] | (kb[t < NT ? t : 0] << 16)) : 0xffffffffu;
        transpose16_dual(P);                                    // P[i] = plane of key bit 15 - i; bit 15 marks the excluded keys
        unsigned cand = ~P[0];
#pragma unroll
        for (int i = 1; i < 16; ++i) {
            const unsigned z = cand & ~P[i];
            const int c = warp_redux_add(dsp_popc(z & 0xffffu) + (dsp_popc(z >> 16) << 16));
            const int cA = c & 0xffff, cB = c >> 16;
            const bool zA = rA < cA, zB = rB < cB;
            const unsigned sel = (zA ? 0x0000ffffu : 0u) | (zB ? 0xffff0000u : 0u);
            cand = (z & sel) | (cand & P[i] & ~sel);
            if (!zA) { rA -= cA; Ka |= 1u << (15 - i); }
            if (!zB) { rB -= cB; Kb |= 1u << (15 - i); }
        }
    }
    int c = 0; unsigned na = 0xffffu, nb = 0xffffu;
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        c += (ka[t] <= Ka ? 1 : 0) + (kb[t] <= Kb ? 0x10000 : 0);
        if (ka[t] > Ka && ka[t] < na) na = ka[t];
        if (kb[t] > Kb && kb[t] < nb) nb = kb[t];
    }
    c = warp_redux_add(c); na = warp_redux_min(na); nb = warp_redux_min(nb);
    const unsigned Ka2 = ((ma & 1) || (c & 0xffff) >= (ma >> 1) + 1) ? Ka : na;
    const unsigned Kb2 = ((mb & 1) || (c >> 16) >= (mb >> 1) + 1) ? Kb : nb;
    float2 med;
    med.x = ma ? ((float)(int)Ka + (float)(int)Ka2) * 0.5f : NAN;
    med.y = mb ? ((float)(int)Kb + (float)(int)Kb2) * 0.5f : NAN;
    return med;
}
template <int NT>
DEVFN float2 warp_median_nonneg2(const float (&xa)[NT], const float (&xb)[NT], int L, int lane) {
    unsigned ka[NT], kb[NT];
    int cnt = 0, cntb = 0;
    const bool full = L >= 32 * NT;   // uniform: every lane's samples lie inside the frame
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        // branch-free: a sample counts when it lies inside the frame and is >= 0 (-0.0 counts as 0, a NaN does not)
        const float va = xa[t], vb = xb[t];
        const bool in = full || (lane + 32 * t) < L;
        const bool na = in & (va >= 0.f), nb = in & (vb >= 0.f);
        ka[t] = na ? ((unsigned)__float_as_int_compat(va) & 0x7fffffffu) : 0xffffffffu;
        kb[t] = nb ? ((unsigned)__float_as_int_compat(vb) & 0x7fffffffu) : 0xffffffffu;
        cnt += na; cntb += nb;
    }
    cnt = warp_redux_add(cnt + (cntb << 16));
    const int ma = cnt & 0xffff, mb = cnt >> 16;
    const int ra = (ma - 1) >> 1, rb = (mb - 1) >> 1;          // rank of the lower middle element
    unsigned Ka = 0, Kb = 0;
    {
        // Bit-sliced radix select.  The lane's 16 keys of both frames are transposed into bit planes (a 16 x 16 bit-matrix
        // transpose per half-word, frame A in the low halves of the registers and frame B in the high halves, so one
        // sequence of masked swaps serves both): plane[b] has bit t set when key t has bit b set.  One selection step per
        // key bit, most significant first, is then a handful of logic operations per lane: candidates with a zero bit =
        // cand & ~plane, one population count per frame, a warp sum, and the candidate mask keeps the zeros or the ones.
        unsigned H[16], Lo[16];
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            const unsigned a = t < NT ? ka[t < NT ? t : 0] : 0xffffffffu, b = t < NT ? kb[t < NT ? t : 0] : 0xffffffffu;
            H[t] = (a >> 16) | (b & 0xffff0000u);
            Lo[t] = (a & 0xffffu) | (b << 16);
        }
        transpose16_dual(H);
        transpose16_dual(Lo);
        // key bit 31 separates the excluded keys (all ones) from the real ones: its step needs no count
        unsigned cand = ~H[0];
        int rA = ra, rB = rb;
#pragma unroll
        for (int i = 1; i < 32; ++i) {
            const unsigned P = i < 16 ? H[i & 15] : Lo[i & 15];           // plane of key bit 31 - i
            const unsigned z = cand & ~P;
            const int c = warp_redux_add(dsp_popc(z & 0xffffu) + (dsp_popc(z >> 16) << 16));
            const int cA = c & 0xffff, cB = c >> 16;
            const bool zA = rA < cA, zB = rB < cB;                        // the rank lies among the candidates with a zero bit
            const unsigned sel = (zA ? 0x0000ffffu : 0u) | (zB ? 0xffff0000u : 0u);
            cand = (z & sel) | (cand & P & ~sel);
            if (!zA) { rA -= cA; Ka |= 1u << (31 - i); }
            if (!zB) { rB -= cB; Kb |= 1u << (31 - i); }
        }
    }
    // even count: the upper middle element is the same key when enough keys are <= K, else the next larger key
    int c = 0; unsigned na = 0xffffffffu, nb = 0xffffffffu;
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        c += (ka[t] <= Ka ? 1 : 0) + (kb[t] <= Kb ? 0x10000 : 0);
        if (ka[t] > Ka && ka[t] < na) na = ka[t];
        if (kb[t] > Kb && kb[t] < nb) nb = kb[t];
    }
    c = warp_redux_add(c); na = warp_redux_min(na); nb = warp_redux_min(nb);
    const unsigned Ka2 = ((ma & 1) || (c & 0xffff) >= (ma >> 1) + 1) ? Ka : na;
    const unsigned Kb2 = ((mb & 1) || (c >> 16) >= (mb >> 1) + 1) ? Kb : nb;
    float2 med;   // np.median of an even count is (a + b) / 2
    med.x = ma ? (__int_as_float_compat((int)Ka) + __int_as_float_compat((int)Ka2)) * 0.5f : NAN;
    med.y = mb ? (__int_as_float_compat((int)Kb) + __int_as_float_compat((int)Kb2)) * 0.5f : NAN;
    return med;
}
// single-frame form (center_clip tap)
DEVFN float warp_median_nonneg(const float (&x)[16], int L, int lane) { return warp_median_nonneg2<16>(x, x, L, lane).x; }

// center_clip(frame, False) (pitch.py:145-155) on one value
DEVFN float clip_value(float v, float med) {
    // v > med -> v - med;  v < -med -> v + med;  else 0  ==  v - clamp(v, -med, med) for finite v (v - v = +0; a NaN median --
    // a frame without non-negative samples -- leaves the clamp at v, i.e. 0, as both reference comparisons are false)
#ifdef DSPFE_EMU
    if (v > med) return v - med;
    if (v < -med) return v + med;
    return 0.f;
#else
    return v - fmaxf(-med, fminf(v, med));
#endif
}

// frame g -> utterance index: last u with frame_off[u] <= g.  Warp-cooperative 32-ary search: three dependent loads
// for up to 32768 utterances instead of log2(U) of them.
DEVFN int find_utt(const int64_t* frame_off, int n_utt, int64_t g, int lane) {
    int lo = 0, hi = n_utt;   // invariant: frame_off[lo] <= g < frame_off[hi]
    while (hi - lo > 1) {
        const int stride = (hi - lo + 31) >> 5;
        const int i = lo + lane * stride;                       // probes lo, lo + stride, ...
        const bool le = i < hi && frame_off[i] <= g;            // true on a prefix of the lanes (lane 0 always)
        const int c = warp_redux_add(le ? 1 : 0);
        lo += (c - 1) * stride;
        hi = lo + stride < hi ? lo + stride : hi;
    }
    return lo;
}

// Work unit of `per` consecutive slots starting at slot h0 (a multiple of per, per | kClipRun): its utterance, the global index
// of its first frame and how many of its frames exist (0: the unit is padding).
DEVFN void slot_unit(const PitchParams& p, int64_t h0, int per, int lane, int& u, int64_t& g0, int& nvalid) {
    u = find_utt(p.slot_off, p.n_utt, h0, lane);
    const int64_t f0 = p.frame_off[u];
    const int64_t local = h0 - p.slot_off[u], F = p.frame_off[u + 1] - f0;
    const int64_t left = F - local;
    nvalid = left <= 0 ? 0 : (left < per ? (int)left : per);
    g0 = f0 + local;
    if (g0 + nvalid > p.max_frames) nvalid = g0 < p.max_frames ? (int)(p.max_frames - g0) : 0;   // (outputs are sized by the bound: never taken)
}

// The same from the run descriptor K4a-1 left behind (one 16-byte load instead of a three-level search)
DEVFN void slot_unit_from_desc(const PitchParams& p, int64_t h0, int per, int64_t& g0, int& nvalid) {
    const int4 d = ldg(p.run_desc + h0 / kClipRun);
    const int in_run = (int)(h0 % kClipRun);
    const int left = d.z - in_run;
    nvalid = left <= 0 ? 0 : (left < per ? left : per);
    g0 = (((int64_t)d.y << 32) | (int64_t)(unsigned)d.x) + in_run;
}

// Source cursor of one frame for the gather through the sample-picking decimator (preprocess.py:21-28): the lane's
// sample t sits at decimated index k = f*step + lane + 32 t, and k - 1 = a * ds_out + b is advanced by 32 per step
// without a division (k = 0 starts from -1 = (-1, ds_out - 1)).
struct FrameCursor {
    const unsigned char* src;   // sample s of the (trimmed) utterance lives at src + s * esz (global memory or the staged copy)
    int lim;      // relative index of the utterance's first sample (<= 0): pre-emphasis reaches back to it
    int nvalid;   // the lane's samples t < nvalid lie inside both the frame and the decimated signal
    int a, b;     // k - 1 = a * ds_out + b for the lane's current decimated index k
};
// Stages the source span of one frame in shared memory with 16-byte loads (one DRAM latency for the whole frame
// instead of one per group of samples) and returns the cursor; spans that do not fit are read in place.
// span = decimated samples wanted from the frame's first one on (one frame: frame_len; a run of frames: (R-1)*step + frame_len)
DEVFN FrameCursor frame_cursor(const PitchParams& p, int64_t g, int u, int lane, bool valid, unsigned char* stage, int span, int stage_cap) {
    FrameCursor c;
    const int esz = p.in_f32 ? 4 : 2;
    const int64_t start = p.seg_start[u];
    const unsigned char* pcm = reinterpret_cast<const unsigned char*>(p.pcm);
    c.src = pcm + start * esz;
    c.lim = (int)(p.offsets[u] - start);
    const int Ld = valid ? p.ds_len[u] : 0;
    const int kf = (int)(g - p.frame_off[u]) * p.frame_step;
    const int k = kf + lane;
    c.a = k >= 1 ? (k - 1) / p.ds_out : -1;                    // k = 0 starts from -1 = (-1, ds_out - 1): its index
    c.b = k >= 1 ? (k - 1) - c.a * p.ds_out : p.ds_out - 1;    // a*ds_in + ds_idx[b] is negative and clamps to sample 0
    const int kl = kf + span - 1 < Ld - 1 ? kf + span - 1 : Ld - 1;
    const int nlim = (span < Ld - kf ? span : Ld - kf) - lane;   // samples n = lane + 32 t with n < min(span, Ld - kf)
    c.nvalid = nlim > 0 ? (nlim + 31) >> 5 : 0;
    if (kf <= kl) {
        int s_lo = (int)ds_index(kf, p.ds_idx, p.ds_in, p.ds_out) - 1;
        if (s_lo < c.lim) s_lo = c.lim;
        const int s_hi = (int)ds_index(kl, p.ds_idx, p.ds_in, p.ds_out);
        const int64_t b_lo = (start + s_lo) * esz, b_hi = (start + s_hi + 1) * esz, a0 = b_lo & ~(int64_t)15;
        const int nbytes = (int)(b_hi - a0);
        if (nbytes <= stage_cap) {
            const int64_t total_bytes = p.total_samples * esz;
            // four 16-byte loads in flight per lane (a load -> store loop pays one DRAM latency per iteration)
            for (int off0 = lane * 16; off0 < nbytes; off0 += 4 * 512) {
                uint4 v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int off = off0 + k * 512;
                    if (off < nbytes && a0 + off + 16 <= total_bytes) v[k] = ldg(reinterpret_cast<const uint4*>(pcm + a0 + off));
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int off = off0 + k * 512;
                    if (off < nbytes) {
                        if (a0 + off + 16 <= total_bytes) *reinterpret_cast<uint4*>(stage + off) = v[k];
                        else for (int e = 0; e < 16 && a0 + off + e < total_bytes; ++e) stage[off + e] = pcm[a0 + off + e];
                    }
                }
            }
            c.src = stage + (start * esz - a0);
        }
    }
    simt::warp_sync();
    return c;
}
// one sample: pre-emphasised over the whole utterance (preprocess.py:11-19), zero past the decimated length
// (sigproc.py:84-87); then the cursor moves on by 32 decimated samples
template <bool F32, bool PRE>
DEVFN float frame_sample(const PitchParams& p, FrameCursor& c, const int32_t* ds_idx, int t) {
    float v = 0.f;
    if (t < c.nvalid) {
        int s = c.a * p.ds_in + ds_idx[c.b];   // sample index inside the (trimmed) utterance
        s = s > 0 ? s : 0;
        float cur, prev = 0.f;
        if (F32) {
            const float* q = reinterpret_cast<const float*>(c.src) + s;
            cur = q[0]; if (PRE && s > c.lim) prev = q[-1];
        } else {
            const int16_t* q = reinterpret_cast<const int16_t*>(c.src) + s;
            cur = cvt_i16(q[0]); if (PRE && s > c.lim) prev = cvt_i16(q[-1]);
        }
        // x[n] - c*x[n-1] in float64 with NumPy's two roundings (preprocess.py:18), then rounded to float32: exact zeros and
        // signs as in the reference (they decide the membership of the median's sample set, pitch.py:146);
        // PRE = false leaves the sample as it is and skips the load of its predecessor
        if (PRE) {
            // float32 first (c = c_hi + c_lo split: within an ulp of the float64 result); where the two terms cancel -- the only place
            // where the sign or an exact zero can come out differently -- the float64 evaluation decides
            v = dsp_fmaf(-p.pre_lo, prev, dsp_fmaf(-p.pre_hi, prev, cur));
            if (fabsf(v) <= 1e-3f * fabsf(cur)) v = dsp_preemph_f64(p.preemph, cur, prev);
        } else {
            v = cur;
        }
    }
    c.a += p.ds_q32; c.b += p.ds_r32;
    if (c.b >= p.ds_out) { c.b -= p.ds_out; ++c.a; }
    return v;
}
// K4a-1: gather + median + centre clip -> p.clip[pair] (512 float2, frame A in .x, frame B in .y) and p.frame_amp.  Its own
// kernel: it needs few registers and little shared memory, so twice as many warps as the transform kernels hide its load
// and selection latencies.  A warp takes a RUN of kClipRun consecutive frames: consecutive frames of an utterance overlap
// (512 samples every 100), so the run's source span is staged once (16-byte loads), walked once through the sample-picking
// decimator (and the pre-emphasis) into a float buffer of decimated samples, and every frame of the run then reads its
// samples from that buffer with plain contiguous loads -- the index arithmetic is paid per decimated sample, not per
// sample per frame.  Runs are cut in the padded slot space (PitchParams::slot_off): a run belongs to one utterance.
// wsm: per-warp shared memory = stage[kClipStageBytes] | dec[kClipDecCap] float.
constexpr int kClipStageBytes = 4096;        // source span of a run: 1212 decimated samples are 3.9 KB of int16 at 16 -> 10 kHz
constexpr int kClipDecCap = 1280;               // floats: 7 * 100 + 512 decimated samples of a run, rounded up to the unrolled row count
constexpr int kClipWarpSmemBytes = kClipStageBytes + kClipDecCap * 4;
constexpr int kClipCtaSmem = kMaxDsOut * 4 + kPitchWarps * kClipWarpSmemBytes;
template <bool F32, bool PRE>
DEVFN void decimate_span(const PitchParams& p, FrameCursor& c, const int32_t* ds_idx, float* dec, int lane, int rows) {
#pragma unroll 1
    for (int t0 = 0; t0 < rows; t0 += 4) {
#pragma unroll
        for (int j = 0; j < 4; ++j) dec[32 * (t0 + j) + lane] = frame_sample<F32, PRE>(p, c, ds_idx, t0 + j);
    }
}
// I16: raw int16 samples (no pre-emphasis, no float input): integer keys for the median
DSP_HD bool clip_i16_keys(const PitchParams& p) { return !p.in_f32 && p.pre_hi == 0.f && p.pre_lo == 0.f; }
// h0: first slot of the run (a multiple of kClipRun)
template <int NT, bool I16>
DEVFN void pitch_clip_run(const PitchParams& p, int64_t h0, unsigned char* wsm, const int32_t* ds_idx) {
    const int lane = simt::tid() & 31;
    unsigned char* stage = wsm;
    float* dec = reinterpret_cast<float*>(wsm + kClipStageBytes);
    const int L = p.frame_len, step = p.frame_step;
    int u, nf; int64_t g0;
    slot_unit(p, h0, kClipRun, lane, u, g0, nf);
    if (lane == 0) p.run_desc[h0 / kClipRun] = make_int4((int)(g0 & 0xffffffffll), (int)(g0 >> 32), nf, u);   // spares K4a-2 / K5a-2 the search
    if (nf == 0) return;
    const int Ld = p.ds_len[u];
    const int kf0 = (int)(g0 - p.frame_off[u]) * step;              // decimated index of the run's first sample inside the utterance
    const int fit = ((kClipDecCap - L) / step + 1) & ~1;              // frames whose samples fit dec at once (8 for 512 / 100); even: pairs stay together
#pragma unroll 1
    for (int j0 = 0; j0 < nf; j0 += fit) {                            // (one pass unless the framing is unusual)
        const int nj = nf - j0 < fit ? nf - j0 : fit;
        const int span = (nj - 1) * step + L;
        simt::warp_sync();
        FrameCursor c = frame_cursor(p, g0 + j0, u, lane, true, stage, span, kClipStageBytes);
        const int rows = (((span + 31) >> 5) + 3) & ~3;               // rows of 32 decimated samples, rounded to the unroll (rows past the span give zeros)
        const bool pre = p.pre_hi != 0.f || p.pre_lo != 0.f;
        if (p.in_f32) { if (pre) decimate_span<true, true>(p, c, ds_idx, dec, lane, rows); else decimate_span<true, false>(p, c, ds_idx, dec, lane, rows); }
        else { if (pre) decimate_span<false, true>(p, c, ds_idx, dec, lane, rows); else decimate_span<false, false>(p, c, ds_idx, dec, lane, rows); }
        simt::warp_sync();
#pragma unroll 1
        for (int j = j0; j < j0 + nj; j += 2) {
            const bool hasB = j + 1 < nf && j + 1 < j0 + nj;
            float xa[NT], xb[NT], fa = 0.f, fb = 0.f;
            const int base = (j - j0) * step;
            const int cnta = L < Ld - (kf0 + j * step) ? L : Ld - (kf0 + j * step);          // samples inside the decimated signal; zeros after
            const int cntb = hasB ? (L < Ld - (kf0 + (j + 1) * step) ? L : Ld - (kf0 + (j + 1) * step)) : 0;
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const int n = 32 * t + lane;
                const float va = n < cnta ? dec[base + n] : 0.f, vb = n < cntb ? dec[base + step + n] : 0.f;
                xa[t] = va; xb[t] = vb; fa += fabsf(va); fb += fabsf(vb);
            }
            // sum |x| of the raw frames (sub_endpoint_detect, pitch.py:65) in float64 across the warp
            if (p.frame_amp) {
                double sa = (double)fa, sb = (double)fb;
#pragma unroll
                for (int m = 16; m >= 1; m >>= 1) { sa += shfl32_xor_f64(sa, m); sb += shfl32_xor_f64(sb, m); }
                if (lane == 0) { p.frame_amp[g0 + j] = sa; if (hasB) p.frame_amp[g0 + j + 1] = sb; }
            }
            // centre clip at the median of the non-negative samples (pitch.py:145-155); padding zeros are samples too
            float2 med = make_float2(0.f, 0.f);
            if (p.do_clip) med = I16 ? warp_median_nonneg2_i16<NT>(xa, xb, L, lane) : warp_median_nonneg2<NT>(xa, xb, L, lane);
            float2* dst = p.clip + ((h0 + j) >> 1) * 512;
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                float2 o = make_float2(0.f, 0.f);
                if (t < NT && lane + 32 * t < L) {
                    o.x = p.do_clip ? clip_value(xa[t < NT ? t : 0], med.x) : xa[t < NT ? t : 0];
                    o.y = p.do_clip ? clip_value(xb[t < NT ? t : 0], med.y) : xb[t < NT ? t : 0];
                }
                dst[32 * t + lane] = o;
            }
        }
    }
}

// K4a-2 / K5a-2: two consecutive frames (g0, g0 + 1) per warp: FIR band-pass + (cepstrum | autocorrelation) of the clipped
// pair -> p.rows[g, :].  The causal complex FIR y = conv(x, h)[:512] (sigproc.py:22-46) is evaluated through
// the even / odd bins of its 1024-point spectrum, which only takes 512-point transforms:
//     Xe = FFT512(x), Xo = FFT512(x W1024^n);  y[n] = (IFFT512(Xe He)[n] + W1024^-n IFFT512(Xo Ho)[n]) / 2
// and for the cepstrum (pitch.py:135-143) the first inverse transform folds away:
//     FFT512(y) = (Xe He + FFT512(W1024^-n IFFT512(Xo Ho))) / 2.
// The transforms run as a rolled loop over stages (one copy of the routine in the instruction stream: the fully
// inlined chain thrashed the instruction cache).  MODE 0 = cepstrum (5 transforms), 1 = autocorrelation (8).  Autocorrelation
// frames short enough (frame_len + 199 <= 512, e.g. the 300-sample frames of model.py:92) that nothing wraps in 512 points
// take pitch_acr_quad below instead (3 transforms per pair).
// wsm: per-warp shared memory = scr[kWarpScr] float2 | park[512] float4.
template <int MODE>
// h0: the pair's first slot (even); g0: global index of its first frame; hasB: the second frame exists
DEVFN void pitch_fft_pair(const PitchParams& p, int64_t h0, int64_t g0, bool hasB, unsigned char* wsm, const float2* tws, const float2* /*w32s*/) {
    const int lane = simt::tid() & 31;
    float2* scr = reinterpret_cast<float2*>(wsm);
    float4* park = reinterpret_cast<float4*>(scr + kWarpScr);
    float2* xs = p.clip + (h0 >> 1) * 512;      // the clipped frame pair (global memory; the autocorrelation path reuses it for |y|)
    const float2* modA = p.tab + kTabMod;   // W1024^n, n = 32 t + lane
    const float2* HeB = p.tab + kTabHe;     // H1024[2k], k = 32 t + lane
    const float2* HoB = p.tab + kTabHo;     // H1024[2k+1]
    const int L = p.frame_len;
    // (every lane only ever touches its own xs / park entries: no barrier needed around them)
    cpx2 x[16];
    const float2 zero2 = make_float2(0.f, 0.f);
    const float inv1024 = 1.0f / 1024.0f;
    constexpr int kStages = MODE == 0 ? 5 : 8;
    // cepstrum:         0 F(x)        -> park Xe He / 2        autocorrelation: 0 F(x)       -> Xe He
    //                   1 F(x W^n)    -> Xo Ho                                  1 inverse    -> park
    //                   2 inverse     -> W^-n d / 1024                          2 F(x W^n)   -> Xo Ho
    //                   3 forward     -> + park, log|.|                         3 inverse    -> v = |park + W^-n d| / 1024 -> xs
    //                   4 inverse     -> |.| / 512 -> rows                      4 F(v)       -> |Ve|^2      5 inverse -> keep Re
    //                                                                           6 F(v W^n)   -> |Vo|^2      7 inverse -> rows
#pragma unroll 1
    for (int st = 0; st < kStages; ++st) {
        const bool inv = MODE == 0 ? (st == 2 || st == 4) : (st & 1);
        const bool load = MODE == 0 ? st <= 1 : !(st & 1);
        const bool loadmod = MODE == 0 ? st == 1 : (st == 2 || st == 6);
        if (load) {                                          // a real sequence from xs, optionally times W1024^n
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const float2 xv = xs[32 * t + lane];
                float2 m = make_float2(1.f, 0.f);
                if (loadmod) m = ldg(modA + 32 * t + lane);
                x[t].re = f2muls(xv, m.x); x[t].im = f2muls(xv, m.y);
            }
        }
        if (inv) {                                           // inverse = conj . forward . conj
#pragma unroll
            for (int t = 0; t < 16; ++t) x[t].im = f2neg(x[t].im);
        }
        fft512(x, scr, tws, lane);
        if (inv) {
#pragma unroll
            for (int t = 0; t < 16; ++t) x[t].im = f2neg(x[t].im);
        }
        // ---- pointwise table products: He / Ho after a forward transform, conj(W1024^n) after the FIR's inverse
        const bool mulH = MODE == 0 ? st <= 1 : (st == 0 || st == 2);
        const bool mulM = MODE == 0 ? st == 2 : st == 3;
        if (mulH || mulM) {
            const float2* T = mulM ? modA : ((MODE == 0 ? st == 0 : st == 0) ? HeB : HoB);
            const float sr = mulM ? (MODE == 0 ? inv1024 : 1.f) : ((MODE == 0 && st == 0) ? 0.5f : 1.f);
            const float si = mulM ? -sr : sr;
#pragma unroll
            for (int t = 0; t < 16; ++t) { const float2 h = ldg(T + 32 * t + lane); x[t] = cmuls(x[t], h.x * sr, h.y * si); }
        }
        if (MODE == 0) {
            if (st == 0) {                                   // park Xe He / 2
#pragma unroll
                for (int t = 0; t < 16; ++t) park[32 * t + lane] = make_float4(x[t].re.x, x[t].re.y, x[t].im.x, x[t].im.y);
            } else if (st == 3) {                            // FFT512(y) = park + .; log|.|
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    const float4 pk = park[32 * t + lane];
                    const float2 yr = f2add(x[t].re, make_float2(pk.x, pk.y)), yi = f2add(x[t].im, make_float2(pk.z, pk.w));
                    const float2 s2 = f2fma(yi, yi, f2mul(yr, yr));
                    x[t].re = make_float2(0.5f * dsp_fast_logf(s2.x), 0.5f * dsp_fast_logf(s2.y));
                    x[t].im = zero2;
                }
            } else if (st == 4) {                            // |IFFT512| / 512 -> rows
                const float inv512 = 1.0f / 512.0f;
                float* rowa = p.rows + g0 * p.row_len;
                float* rowb = rowa + p.row_len;
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    const int n = 32 * t + lane;
                    if (n < p.row_len) {
                        const float2 s2 = f2fma(x[t].im, x[t].im, f2mul(x[t].re, x[t].re));
                        rowa[n] = dsp_fast_sqrtf(s2.x) * inv512;
                        if (hasB) rowb[n] = dsp_fast_sqrtf(s2.y) * inv512;
                    }
                }
            }
        } else {
            // autocorrelation of v = |y| (pitch.py:112-132, sigproc.py:48-53): r = IFFT1024(|FFT1024(v)|^2), again through
            // the even / odd bins: r[n] = (IFFT512(|Ve|^2)[n] + W1024^-n IFFT512(|Vo|^2)[n]) / 1024
            if (st == 1) {                                   // park the circular part of the convolution
#pragma unroll
                for (int t = 0; t < 16; ++t) park[32 * t + lane] = make_float4(x[t].re.x, x[t].re.y, x[t].im.x, x[t].im.y);
            } else if (st == 3) {                            // v = |park + W1024^-n d| / 1024 -> xs
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    const float4 pk = park[32 * t + lane];
                    const float2 yr = f2add(x[t].re, make_float2(pk.x, pk.y)), yi = f2add(x[t].im, make_float2(pk.z, pk.w));
                    const float2 s2 = f2fma(yi, yi, f2mul(yr, yr));
                    const bool in = 32 * t + lane < L;
                    xs[32 * t + lane] = make_float2(in ? dsp_fast_sqrtf(s2.x) * inv1024 : 0.f, in ? dsp_fast_sqrtf(s2.y) * inv1024 : 0.f);
                }
            } else if (st == 4 || st == 6) {                 // power spectrum
#pragma unroll
                for (int t = 0; t < 16; ++t) { x[t].re = f2fma(x[t].im, x[t].im, f2mul(x[t].re, x[t].re)); x[t].im = zero2; }
            } else if (st == 5) {                            // real parts of the even-bin half, lags < 224
                float2* ge = reinterpret_cast<float2*>(park);
#pragma unroll
                for (int t = 0; t < 7; ++t) ge[32 * t + lane] = x[t].re;
            } else if (st == 7) {                            // combine, unbiased normalisation, rows
                const float2* ge = reinterpret_cast<const float2*>(park);
                float* rowa = p.rows + g0 * p.row_len;
                float* rowb = rowa + p.row_len;
#pragma unroll
                for (int t = 0; t < 7; ++t) {
                    const int n = 32 * t + lane, j = n - kMinLag;
                    if (j >= 0 && j < p.row_len) {
                        const float2 m = ldg(modA + n);
                        // Re(conj(W1024^n) go[n]) = m.x go.re + m.y go.im
                        const float2 r = f2muls(f2add(ge[n], f2fmas(x[t].re, m.x, f2muls(x[t].im, m.y))), inv1024);
                        const float inv_n = (n < L) ? 1.0f / (float)(L - n) : NAN;
                        rowa[j] = r.x * inv_n;
                        if (hasB) rowb[j] = r.y * inv_n;
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K4a-2 for cepstrum frames of 100 <= N < 512 samples (pitch.py:83 with winlen != 0.0512): a frame pair per warp, as
// pitch_fft_pair<0>, but the cepstrum's transforms are N-point DFTs, taken by Bluestein's identity
//     DFT_N(a)[k] = w_k sum_n (a_n w_n) conj(w_{k-n}),   w_n = exp(-i pi n^2 / N),
// a 1024-point circular convolution of s = a w (zero from N on) with b = conj(w) wrapped (b[m] = b[1024 - m] = conj(w_m), m < N):
// b reaches 2N - 1 <= 1023 points, so the first N outputs carry no wrap.  Only magnitudes leave either DFT -- |Y| goes into the
// log, |ifft| into the row -- and |w_k| = 1 drops the post-multiplication; the inverse DFT of the real log|Y| is
// conj(DFT_N(log|Y|)) / N, so it is the same forward chain.  Each 1024-point convolution of an s supported on [0, 512) takes
// four 512-point transforms, as the FIR of pitch_fft_pair<1> does:
//     (s (*) k)[n] = (IFFT512(S_e K_e)[n] + W1024^-n IFFT512(S_o K_o)[n]) / 1024,   S_e = FFT512(s), S_o = FFT512(s W1024^n)
// Three convolutions, 12 transforms per pair:  x (*) h -> y[0..N)  (He, Ho);  (y w) (*) b -> |Y|  (Be, Bo);
// (log|Y| w) (*) b -> |.| / N -> rows.  s is parked for its odd half while the even half runs, then the two swap places.
// wsm: per-warp shared memory = scr[kWarpScr] float2 | park[512] float4 (as pitch_fft_pair).
// ---------------------------------------------------------------------------------------------------------
// h0: the pair's first slot (even); g0: global index of its first frame; hasB: the second frame exists
DEVFN void pitch_cep_bluestein_pair(const PitchParams& p, int64_t h0, int64_t g0, bool hasB, unsigned char* wsm, const float2* tws, const float2* /*w32s*/) {
    const int lane = simt::tid() & 31;
    float2* scr = reinterpret_cast<float2*>(wsm);
    float4* park = reinterpret_cast<float4*>(scr + kWarpScr);
    const float2* xs = p.clip + (h0 >> 1) * 512;      // the clipped frame pair
    const float2* modA = p.tab + kTabMod;             // W1024^n, n = 32 t + lane
    const float2* chirp = p.tab + kTabChirp;          // w_n (zero from N on)
    const int N = p.frame_len;
    const float2 zero2 = make_float2(0.f, 0.f);
    const float inv1024 = 1.0f / 1024.0f;
    cpx2 x[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) { x[t].re = xs[32 * t + lane]; x[t].im = zero2; }
    // stage 4c + 0  F(s)      -> S_e K_e          (s parked first)      c = 0: FIR, K = H;  c = 1, 2: Bluestein, K = B
    //       4c + 1  inverse   -> park <-> x: the even half in, s W1024^n out
    //       4c + 2  forward   -> S_o K_o
    //       4c + 3  inverse   -> v = (park + W1024^-n d) / 1024, then  c = 0: y w;  c = 1: log|v| w;  c = 2: |v| / N -> rows
#pragma unroll 1
    for (int st = 0; st < 12; ++st) {
        const int c = st >> 2, k = st & 3;
        const bool inv = k & 1;
        if (k == 0) {
#pragma unroll
            for (int t = 0; t < 16; ++t) park[32 * t + lane] = make_float4(x[t].re.x, x[t].re.y, x[t].im.x, x[t].im.y);
        }
        if (inv) {                                           // inverse = conj . forward . conj
#pragma unroll
            for (int t = 0; t < 16; ++t) x[t].im = f2neg(x[t].im);
        }
        fft512(x, scr, tws, lane);
        if (inv) {
#pragma unroll
            for (int t = 0; t < 16; ++t) x[t].im = f2neg(x[t].im);
        }
        if (!inv) {                                          // even (k = 0) or odd (k = 2) bins of the kernel's 1024-point spectrum
            const float2* T = p.tab + (c == 0 ? (k == 0 ? kTabHe : kTabHo) : (k == 0 ? kTabBe : kTabBo));
#pragma unroll
            for (int t = 0; t < 16; ++t) { const float2 h = ldg(T + 32 * t + lane); x[t] = cmuls(x[t], h.x, h.y); }
        } else if (k == 1) {                                 // (every lane only ever touches its own park entries)
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const float4 pk = park[32 * t + lane];
                park[32 * t + lane] = make_float4(x[t].re.x, x[t].re.y, x[t].im.x, x[t].im.y);
                const float2 m = ldg(modA + 32 * t + lane);
                cpx2 s; s.re = make_float2(pk.x, pk.y); s.im = make_float2(pk.z, pk.w);
                x[t] = cmuls(s, m.x, m.y);
            }
        } else {
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const int n = 32 * t + lane;
                const float4 pk = park[n];
                const float2 m = ldg(modA + n);
                const cpx2 d = cmuls(x[t], m.x, -m.y);
                cpx2 v;
                v.re = f2muls(f2add(d.re, make_float2(pk.x, pk.y)), inv1024);
                v.im = f2muls(f2add(d.im, make_float2(pk.z, pk.w)), inv1024);
                if (c == 2) {
                    x[t] = v;
                } else {
                    const float2 w = ldg(chirp + n);        // zero from N on: the sequence ends with the frame
                    if (c == 1) {                            // log|Y| (the chirp of the last DFT has modulus 1); 0 * -inf is a NaN
                        const float2 s2 = f2fma(v.im, v.im, f2mul(v.re, v.re));
                        const float2 lg = n < N ? make_float2(0.5f * dsp_fast_logf(s2.x), 0.5f * dsp_fast_logf(s2.y)) : zero2;
                        x[t].re = f2muls(lg, w.x); x[t].im = f2muls(lg, w.y);
                    } else {
                        x[t] = cmuls(v, w.x, w.y);
                    }
                }
            }
            if (c == 2) {                                    // |ifft_N| = |DFT_N| / N -> rows
                const float invN = 1.0f / (float)N;
                float* rowa = p.rows + g0 * p.row_len;
                float* rowb = rowa + p.row_len;
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    const int n = 32 * t + lane;
                    if (n < p.row_len) {
                        const float2 s2 = f2fma(x[t].im, x[t].im, f2mul(x[t].re, x[t].re));
                        rowa[n] = dsp_fast_sqrtf(s2.x) * invN;
                        if (hasB) rowb[n] = dsp_fast_sqrtf(s2.y) * invN;
                    }
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// K5a-2 for frames short enough that nothing wraps in 512 points (acr_short_frames: e.g. the 300-sample frames of
// model.py:92): FOUR consecutive frames (two clipped pairs) per warp, 6 transforms per quad instead of the 12 the
// pair-at-a-time chain (MODE 2 of pitch_fft_pair) takes.  Two uses of "two real sequences in one complex transform":
//   * the FIR.  With T = 512 - L, h = h_lo (taps 0..T) + h_hi (taps T+1..L-1) and x_lo = x[0 .. L-T-2], the first L
//     samples of conv(x, h) are those of conv(x, h_lo) + conv(x_lo, h_hi), and both of these fit 512 points without
//     wrapping (supports end at 511 and at 2L - T - 3 <= 511).  x and x_lo are real, so one forward transform of
//     z = x + i x_lo carries both spectra: X = (Z + Zr*)/2, X_lo = (Z - Zr*)/(2i) with Zr[k] = Z[-k], and
//         FFT512(y) = X H_lo + X_lo H_hi = Z A + Zr* B,   A = (H_lo - i H_hi)/2,  B = (H_lo + i H_hi)/2
//     (tables at kTabHe / kTabHo, the inverse transform's 1/512 folded in).  One forward + one inverse per pair.
//   * the autocorrelation.  v1 = |y| of the first pair and v2 = |y| of the second are real: Z = FFT512(v1 + i v2) gives
//     |V1|^2 = |Z + Zr*|^2 / 4 and |V2|^2 = |Z - Zr*|^2 / 4; both power spectra are real and even, so the inverse transform
//     of |V1|^2 + i |V2|^2 has r1 in its real part and r2 in its imaginary part: one forward + one inverse per quad.
// The partner bins Zr come from the lane 32 - lane (register 15 - t) by shuffles; lane 0 holds the bins 32 t, whose partners
// 32 (16 - t) are its own registers.  So that the update can run in place, the FIR split keeps a one-register look-behind;
// the power spectra are even, so there lane 0 copies bin 32 (16 - t), finished one step earlier, into bin 32 t.
// wsm: per-warp shared memory = scr[kWarpScr] float2 | vpark[32 * kQuadT] float2.
// ---------------------------------------------------------------------------------------------------------
constexpr int kQuadT = 10;                                            // registers that hold samples of a frame of <= 320 samples
constexpr int kQuadWarpSmemBytes = kWarpScr * 8 + 32 * kQuadT * 8;
constexpr int kQuadCtaSmem = (kTabMod * 8) + kPitchWarps * kQuadWarpSmemBytes;
DEVFN cpx2 shfl_c(cpx2 a, int src) {
    cpx2 r;
    r.re.x = __int_as_float_compat(simt::shfl32_i(__float_as_int_compat(a.re.x), src)); r.re.y = __int_as_float_compat(simt::shfl32_i(__float_as_int_compat(a.re.y), src));
    r.im.x = __int_as_float_compat(simt::shfl32_i(__float_as_int_compat(a.im.x), src)); r.im.y = __int_as_float_compat(simt::shfl32_i(__float_as_int_compat(a.im.y), src));
    return r;
}
// KIND 0: x[k] <- x[k] A[k] + conj(x[-k]) B[k];  KIND 1: x[k] <- (|x[k] + conj(x[-k])|^2 + i |x[k] - conj(x[-k])|^2) / 4
template <int KIND>
DEVFN void split_pairs(cpx2 (&x)[16], const float2* A, const float2* B, int lane) {
    const int src = (32 - lane) & 31;
    const bool l0 = lane == 0;
    cpx2 saved = x[0];                                  // KIND 0: lane 0's x[16 - t] before step t - 1 overwrote it
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int a = t, b = 15 - t;
        cpx2 sa = shfl_c(x[b], src), sb = shfl_c(x[a], src);
        const cpx2 za = x[a], zb = x[b];
        if (l0) { sa = KIND == 0 ? saved : za; sb = x[a + 1]; }   // (KIND 1 uses this sa at t = 0 only: bin 0 is its own partner)
        if (KIND == 0) {
            saved = zb;
            const float2 Aa = ldg(A + 32 * a + lane), Ba = ldg(B + 32 * a + lane), Ab = ldg(A + 32 * b + lane), Bb = ldg(B + 32 * b + lane);
            // z A + conj(s) B:  re = z.re A.x - z.im A.y + s.re B.x + s.im B.y;  im = z.re A.y + z.im A.x + s.re B.y - s.im B.x
            x[a].re = f2fmas(sa.im, Ba.y, f2fmas(sa.re, Ba.x, f2fmas(za.im, -Aa.y, f2muls(za.re, Aa.x))));
            x[a].im = f2fmas(sa.im, -Ba.x, f2fmas(sa.re, Ba.y, f2fmas(za.im, Aa.x, f2muls(za.re, Aa.y))));
            x[b].re = f2fmas(sb.im, Bb.y, f2fmas(sb.re, Bb.x, f2fmas(zb.im, -Ab.y, f2muls(zb.re, Ab.x))));
            x[b].im = f2fmas(sb.im, -Bb.x, f2fmas(sb.re, Bb.y, f2fmas(zb.im, Ab.x, f2muls(zb.re, Ab.y))));
        } else {
            const float2 pa_r = f2add(za.re, sa.re), pa_i = f2sub(za.im, sa.im), ma_r = f2sub(za.re, sa.re), ma_i = f2add(za.im, sa.im);
            const float2 pb_r = f2add(zb.re, sb.re), pb_i = f2sub(zb.im, sb.im), mb_r = f2sub(zb.re, sb.re), mb_i = f2add(zb.im, sb.im);
            x[a].re = f2muls(f2fma(pa_i, pa_i, f2mul(pa_r, pa_r)), 0.25f); x[a].im = f2muls(f2fma(ma_i, ma_i, f2mul(ma_r, ma_r)), 0.25f);
            x[b].re = f2muls(f2fma(pb_i, pb_i, f2mul(pb_r, pb_r)), 0.25f); x[b].im = f2muls(f2fma(mb_i, mb_i, f2mul(mb_r, mb_r)), 0.25f);
            if (l0 && t > 0) x[a] = x[16 - t];             // |.|^2 of bin 32 t = that of bin 32 (16 - t), set at step t - 1
        }
    }
}
// h0: the quad's first slot (a multiple of 4); g0: global index of its first frame; nvalid: how many of its frames exist (1..4)
DEVFN void pitch_acr_quad(const PitchParams& p, int64_t h0, int64_t g0, int nvalid, unsigned char* wsm, const float2* tws, const float2* /*w32s*/) {
    const int lane = simt::tid() & 31;
    float2* scr = reinterpret_cast<float2*>(wsm);
    float2* vpark = scr + kWarpScr;
    const float2* tabA = p.tab + kTabHe;
    const float2* tabB = p.tab + kTabHo;
    const int L = p.frame_len;
    const int nlo = 2 * L - 514;                      // x_lo = x[0 .. L - T - 2], T = 512 - L
    const bool has2 = nvalid > 2;                     // the second pair exists (its slot was written by the clip kernel)
    const float2 zero2 = make_float2(0.f, 0.f);
    float2 unscale = make_float2(1.f, 1.f);
    cpx2 x[16];
    // stage 0 F(x + i x_lo) of pair 1 -> Z A + Zr* B      1 inverse -> v1 = |y|, parked
    //       2 the same for pair 2                            3 inverse -> v2;  z = v1 + i v2
    //       4 F(z) -> |V1|^2 + i |V2|^2                    5 inverse -> r1 + i r2 -> rows
#pragma unroll 1
    for (int st = 0; st < 6; ++st) {
        const bool inv = st & 1;
        if (st == 0 || st == 2) {
            const float2* xs = p.clip + ((h0 >> 1) + (st >> 1)) * 512;
            const bool live = st == 0 || has2;
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const int n = 32 * t + lane;
                float2 v = zero2;
                if (t < kQuadT && live) v = xs[n];
                x[t].re = v; x[t].im = n <= nlo ? v : zero2;
            }
        }
        if (inv) {
#pragma unroll
            for (int t = 0; t < 16; ++t) x[t].im = f2neg(x[t].im);
        }
        fft512(x, scr, tws, lane);
        if (st == 0 || st == 2) {
            split_pairs<0>(x, tabA, tabB, lane);
        } else if (st == 1 || st == 3) {                     // v = |y| on the frame, zero beyond it (the conjugation does not change |.|)
            float2 v[kQuadT];
#pragma unroll
            for (int t = 0; t < kQuadT; ++t) {
                const float2 s2 = f2fma(x[t].im, x[t].im, f2mul(x[t].re, x[t].re));
                const bool in = 32 * t + lane < L;
                v[t] = make_float2(in ? dsp_fast_sqrtf(s2.x) : 0.f, in ? dsp_fast_sqrtf(s2.y) : 0.f);
            }
            if (st == 1) {
#pragma unroll
                for (int t = 0; t < kQuadT; ++t) vpark[32 * t + lane] = v[t];      // (a lane only ever touches its own entries)
            } else {
                // Rounding errors of a complex transform leak between its real and imaginary parts at ~1e-7 of the LARGER one:
                // bring the second pair to the first pair's level with a power of two (exact) before packing, undo it after.
                float2 e1 = zero2, e2 = zero2;
#pragma unroll
                for (int t = 0; t < kQuadT; ++t) { const float2 a = vpark[32 * t + lane]; x[t].re = a; e1 = f2fma(a, a, e1); e2 = f2fma(v[t], v[t], e2); }
#pragma unroll
                for (int m = 16; m >= 1; m >>= 1) {
                    e1.x += simt::shfl32_xor(e1.x, m); e1.y += simt::shfl32_xor(e1.y, m);
                    e2.x += simt::shfl32_xor(e2.x, m); e2.y += simt::shfl32_xor(e2.y, m);
                }
                int kx = ((__float_as_int_compat(e1.x) >> 23) - (__float_as_int_compat(e2.x) >> 23)) / 2;    // half the exponent gap of the energies
                int ky = ((__float_as_int_compat(e1.y) >> 23) - (__float_as_int_compat(e2.y) >> 23)) / 2;
                if (!(e1.x > 0.f && e2.x > 0.f && e1.x < 3e38f && e2.x < 3e38f)) kx = 0;
                if (!(e1.y > 0.f && e2.y > 0.f && e1.y < 3e38f && e2.y < 3e38f)) ky = 0;
                kx = kx < -40 ? -40 : (kx > 40 ? 40 : kx); ky = ky < -40 ? -40 : (ky > 40 ? 40 : ky);
                const float2 sc2 = make_float2(__int_as_float_compat((127 + kx) << 23), __int_as_float_compat((127 + ky) << 23));
                unscale = make_float2(__int_as_float_compat((127 - 2 * kx) << 23), __int_as_float_compat((127 - 2 * ky) << 23));
#pragma unroll
                for (int t = 0; t < 16; ++t) {
                    if (t >= kQuadT) x[t].re = zero2;
                    x[t].im = t < kQuadT ? f2mul(v[t < kQuadT ? t : 0], sc2) : zero2;
                }
            }
        } else if (st == 4) {
            split_pairs<1>(x, tabA, tabB, lane);
        }
    }
    // r[n] / 512, unbiased normalisation (sigproc.py:48-53), rows (after the loop: the loop-invariant divisions would otherwise
    // be hoisted out of it and held in registers through every stage)
    const float inv512 = 1.0f / 512.0f;
    float* row = p.rows + g0 * p.row_len;
    const int RL = p.row_len;
    const bool f1 = nvalid > 1, f2 = nvalid > 2, f3 = nvalid > 3;
#pragma unroll
    for (int t = 0; t < 7; ++t) {
        const int n = 32 * t + lane, j = n - kMinLag;
        if (j >= 0 && j < RL) {
            const float sc = (n < L) ? inv512 / (float)(L - n) : NAN;
            row[j] = x[t].re.x * sc;
            if (f1) row[RL + j] = x[t].re.y * sc;
            if (f2) row[2 * RL + j] = -x[t].im.x * unscale.x * sc;   // the inverse is conj . forward . conj: its imaginary part is
            if (f3) row[3 * RL + j] = -x[t].im.y * unscale.y * sc;   // minus the imaginary part left in the registers
        }
    }
}

// K4b / K5b: one CTA (256 threads) per utterance, frames in order, kTrackChunk at a time.  Each pass stages the raw rows of
// the chunk (plus one row of look-ahead) in shared memory with coalesced vector loads, runs the reference's in-place running
// mean on them (one column per thread; rows < i are already smoothed, exactly the reference's recurrence), then one warp per
// row scores the row (peak_score) and takes the arg-max.
// smem (CH = track_chunk(row_len)): float buf[(CH + 1) * row_len] + int sc[CH * 80] + double spitch[kTrackMaxFrames]
//       + int slag[kTrackMaxFrames] + ushort olist[8 * kTrackListPerWarp] (+ 8 bytes of alignment slack).
constexpr int kTrackListPerWarp = kTrackChunk * kPeakLags / (kTrackThreads / 32);     // tasks a warp sees per chunk (all of them may stay open)
DEVFN bool stops(float x, float v) { return !(x <= v); }          // pitch.py:236,239: the scan goes on while sig[j] <= v (a NaN stops it)

DEVFN void pitch_track_cta(const PitchParams& p, float* buf, int* sc, double* spitch) {
    const int u = p.order ? p.order[simt::bid()] : simt::bid();
    const int tid = simt::tid();
    const int lane = tid & 31, warp = tid >> 5;
    const int64_t f0 = p.frame_off[u];
    const int F = (int)(p.frame_off[u + 1] - f0);
    const int RL = p.row_len;
    const int CH = track_chunk(RL);
    const float* rows = p.rows + f0 * RL;
    // the lag track stays in shared memory for the octave-repair sweeps (a thread walking global memory on its own
    // pays a DRAM latency per frame); longer utterances use the global arrays directly
    spitch = reinterpret_cast<double*>((reinterpret_cast<uintptr_t>(spitch) + 7) & ~(uintptr_t)7);   // rows of odd length leave it 4-byte aligned
    int32_t* slag = reinterpret_cast<int32_t*>(spitch + kTrackMaxFrames);
    unsigned short* olist = reinterpret_cast<unsigned short*>(slag + kTrackMaxFrames);                 // per warp: its open (row, lag) tasks
    const bool staged = F <= kTrackMaxFrames;
    int32_t* lagv = staged ? slag : p.lag + f0;
    float s1[2] = {0.f, 0.f}, s2[2] = {0.f, 0.f};    // smoothed rows i-1 and i-2 of this thread's (up to two) columns
    for (int c0 = 0; c0 < F; c0 += CH) {
        const int nrows = F - c0 < CH ? F - c0 : CH;
        const int nload = (c0 + nrows < F ? nrows + 1 : nrows) * RL;          // floats to stage (rows are contiguous)
        const float* src = rows + (int64_t)c0 * RL;
        if ((RL & 3) == 0 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) {
            // eight 16-byte loads in flight per thread (a load -> store loop pays one DRAM latency per iteration)
            const int n4 = nload >> 2;
            for (int i0 = tid; i0 < n4; i0 += 8 * kTrackThreads) {
                float4 v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) { const int i = i0 + k * kTrackThreads; if (i < n4) v[k] = ldg(reinterpret_cast<const float4*>(src) + i); }
#pragma unroll
                for (int k = 0; k < 8; ++k) { const int i = i0 + k * kTrackThreads; if (i < n4) reinterpret_cast<float4*>(buf)[i] = v[k]; }
            }
        } else {
            for (int i = tid; i < nload; i += kTrackThreads) buf[i] = src[i];
        }
        simt::cta_sync();
        if (!p.no_smooth) {
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                const int col = tid + cc * kTrackThreads;
                if (col < RL) {
                    float a2 = s2[cc], a1 = s1[cc];
                    float r0 = buf[col];
                    for (int k = 0; k < nrows; ++k) {
                        const int i = c0 + k;
                        // smooth (pitch.py:157-164): g[i] = mean(g[left:right]) in place, left = max(i-2, 0), right = i+2 if i+2 < F
                        // else F-1; np.mean over axis 0 adds the rows in order (rows < i already smoothed), then divides by the count
                        float gsm, r1 = 0.f;
                        if (i >= 2 && i + 2 < F) {                    // interior: rows i-2, i-1 (smoothed), i, i+1 (raw); /4 is exact as *0.25
                            r1 = buf[(k + 1) * RL + col];
                            gsm = (((a2 + a1) + r0) + r1) * 0.25f;
                        } else {
                            const int right = (i + 2 < F) ? i + 2 : F - 1;
                            const int left = i - 2 > 0 ? i - 2 : 0;
                            float acc = 0.f; bool any = false;
                            if (i - 2 >= 0 && i - 2 < right) { acc = a2; any = true; }
                            if (i - 1 >= 0 && i - 1 < right) { acc = any ? acc + a1 : a1; any = true; }
                            if (i < right) { acc = any ? acc + r0 : r0; any = true; }
                            if (i + 1 < F) r1 = buf[(k + 1) * RL + col];   // raw row i + 1 (inside the chunk or its look-ahead row): the next row's r0
                            if (i + 1 < right) { acc = any ? acc + r1 : r1; any = true; }
                            gsm = any ? acc / (float)(right - left) : NAN;   // empty window: np.mean([]) = NaN
                        }
                        buf[k * RL + col] = gsm;
                        if (p.rows_out) p.rows_out[(f0 + i) * RL + col] = gsm;
                        a2 = a1; a1 = gsm; r0 = r1;
                    }
                    s2[cc] = a2; s1[cc] = a1;
                }
            }
        } else if (p.rows_out) {
            for (int i = tid; i < nrows * RL; i += kTrackThreads) p.rows_out[(f0 + c0) * RL + i] = buf[i];
        }
        simt::cta_sync();
        if (p.mode == 0) {
            // peak_score (pitch.py:227-242) for lags 20..99 of every row of the chunk: min over both sides of the distance to
            // the nearest sample that stops the scan (the left scan ends at index 0, the right one at the row end); only the
            // smaller distance matters, so both sides expand together.
            //   A  one (row, lag) task per thread, distances 1..4 as straight-line code (no loop, no divergence): most lags
            //      stop there.  The others -- the row's peaks at that scale -- go to the warp's own list.
            //   B  the listed tasks, one per lane, eight distances at a time (straight-line) for up to four rounds;
            //   C  what is still open (scores above 36) one task at a time with the 32 lanes spread over the distances.
            const int ntask = nrows * kPeakLags;
            unsigned short* wlist = olist + warp * kTrackListPerWarp;
            int n_open = 0;
            const bool wide = RL >= kMinLag + kPeakLags + 4;              // lags + 4 stay inside the row: no bound checks in A
            for (int t0 = warp * 32; t0 < ntask; t0 += kTrackThreads) {
                const int t = t0 + lane;
                const bool live = t < ntask;
                const int k = live ? t / kPeakLags : 0, c = kMinLag + (live ? t % kPeakLags : 0);
                const float* row = buf + k * RL;
                const float v = row[c];
                const int rmax = c < RL - c ? c : RL - c;             // index 0 / the row end stop the scans
                int sv;
                if (wide) {
                    const bool s1 = stops(row[c - 1], v) || stops(row[c + 1], v), s2 = stops(row[c - 2], v) || stops(row[c + 2], v);
                    const bool s3 = stops(row[c - 3], v) || stops(row[c + 3], v), s4 = stops(row[c - 4], v) || stops(row[c + 4], v);
                    sv = s1 ? 1 : (s2 ? 2 : (s3 ? 3 : (s4 ? 4 : 5)));
                    sv = sv < rmax ? sv : rmax;
                } else {
                    int r = 1;
                    while (r < rmax && r <= 4 && !stops(row[c - r], v) && !stops(row[c + r], v)) ++r;
                    sv = r;
                }
                if (!(v == v)) sv = 0;                                 // a NaN value stops both scans at once
                const bool is_open = live && sv > 4 && sv < rmax;      // all of r = 1..4 passed: go on from r = 5
                if (live) sc[t] = sv;
                const unsigned m = simt::ballot32(is_open);
                if (is_open) wlist[n_open + dsp_popc(m & ((1u << lane) - 1u))] = (unsigned short)t;
                n_open += dsp_popc(m);
            }
            simt::warp_sync();
            for (int i0 = 0; i0 < n_open; i0 += 32) {
                const bool has = i0 + lane < n_open;
                const int t = has ? wlist[i0 + lane] : 0;
                const int k = t / kPeakLags, c = kMinLag + t % kPeakLags;
                const float* row = buf + k * RL;
                const float v = row[c];
                const int rmax = c < RL - c ? c : RL - c;
                int found = -1, r = 5;
                bool pending = has;
#pragma unroll 1
                for (int round = 0; round < 4 && simt::ballot32(pending) != 0; ++round, r += 8) {
                    int first = 8;
#pragma unroll
                    for (int d = 7; d >= 0; --d) {
                        const int rr = r + d < rmax ? r + d : rmax - 1;    // (an index inside the row; past rmax the result is not used)
                        const bool st = r + d < rmax && (stops(row[c - rr], v) || stops(row[c + rr], v));
                        first = st ? d : first;
                    }
                    if (pending) {
                        if (first < 8) { found = r + first; pending = false; }
                        else if (r + 8 >= rmax) { found = rmax; pending = false; }
                    }
                }
                unsigned todo = simt::ballot32(pending);               // r = 37 onwards
                while (todo) {
                    const int src = __builtin_ffs((int)todo) - 1;
                    todo &= todo - 1;
                    const int ck = simt::shfl32_i(k, src), cc = simt::shfl32_i(c, src), cm = simt::shfl32_i(rmax, src);
                    const float cv = __int_as_float_compat(simt::shfl32_i(__float_as_int_compat(v), src));
                    const float* crow = buf + ck * RL;
                    int f = cm;
                    for (int r0 = 37; r0 < cm; r0 += 32) {
                        const int rr = r0 + lane;
                        const bool st = rr < cm && (stops(crow[cc - rr], cv) || stops(crow[cc + rr], cv));
                        const unsigned hit = simt::ballot32(st);
                        if (hit) { f = r0 + __builtin_ffs((int)hit) - 1; break; }
                    }
                    if (lane == src) found = f;
                }
                if (has) sc[t] = found;
            }
            simt::cta_sync();
            for (int k = warp; k < nrows; k += kTrackThreads / 32) {   // first argmax (pitch.py:169), one warp per row
                const int* srow = sc + k * kPeakLags;
                if (p.score) for (int t = lane; t < kPeakLags; t += 32) p.score[(f0 + c0 + k) * kPeakLags + t] = srow[t];
                unsigned key = 0;                                      // (score, first index wins): score * 128 + (127 - index)
                for (int t = lane; t < kPeakLags; t += 32) { const unsigned q = ((unsigned)srow[t] << 7) | (unsigned)(127 - t); key = q > key ? q : key; }
                key = warp_redux_max(key);
                if (lane == 0) lagv[c0 + k] = kMinLag + 127 - (int)(key & 127u);
            }
        } else {
            // np.argmax over the smoothed scores, one warp per row: first maximum, a NaN counts as the maximum.  Values map to
            // unsigned keys in float order (a NaN above +inf); one warp maximum, then the smallest index that attains it.
            for (int k = warp; k < nrows; k += kTrackThreads / 32) {
                const float* row = buf + k * RL;
                unsigned best = 0;
                for (int j = lane; j < RL; j += 32) {
                    const float v = row[j];
                    const unsigned b = (unsigned)__float_as_int_compat(v);
                    const unsigned q = v != v ? 0xffffffffu : (b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u));
                    best = q > best ? q : best;
                }
                const unsigned top = warp_redux_max(best);
                unsigned idx = 0xffffffffu;
                for (int j = lane; j < RL; j += 32) {
                    const float v = row[j];
                    const unsigned b = (unsigned)__float_as_int_compat(v);
                    const unsigned q = v != v ? 0xffffffffu : (b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u));
                    if (q == top && (unsigned)j < idx) idx = (unsigned)j;
                }
                idx = warp_redux_min(idx);
                if (lane == 0) lagv[c0 + k] = kMinLag + (int)idx;
            }
        }
        simt::cta_sync();
    }
    if (!staged) {
        if (tid == 0 && F > 0 && p.pitch) robust_pitch(p.lag + f0, F, p.pitch + f0);
        return;
    }
    // max_pitch (pitch.py:166-172) for every frame in parallel, then the two sequential octave-repair sweeps
    // (robust_max_pitch, pitch.py:191-206) on one thread: compares and doublings only
    for (int i = tid; i < F; i += kTrackThreads) spitch[i] = 1.0 / (0.0001 * (double)slag[i]);
    simt::cta_sync();
    if (tid == 0 && p.pitch) {
        for (int i = 1; i < F; ++i)
            if (fabs(2 * spitch[i] - spitch[i - 1]) < 50 && spitch[i] < 170) spitch[i] = 2 * spitch[i];
        for (int i = F - 2; i > 0; --i)
            if (fabs(2 * spitch[i] - spitch[i + 1]) < 50 && spitch[i] < 170) spitch[i] = 2 * spitch[i];
    }
    simt::cta_sync();
    for (int i = tid; i < F; i += kTrackThreads) {
        p.lag[f0 + i] = slag[i];
        if (p.pitch) p.pitch[f0 + i] = spitch[i];
    }
}

// K6: pitch_feature tail, one warp per utterance.  The utterance's pitch track and frame amplitudes are staged in
// shared memory; the valley search and the two medians run across the lanes, the sequential list logic on lane 0.
// smem: 5 * kFeatMaxFrames doubles.  Longer utterances fall back to lane 0 walking global memory.
constexpr int kFeatMaxFrames = 640;
DEVFN double warp_kth(const double* v, int n, int k, int lane) {   // k-th smallest (0-based) by rank counting; n >= 1
    double out = 0.0; int found = 0;
    for (int e = lane; e < n; e += 32) {
        const double x = v[e];
        int rank = 0;
        for (int j = 0; j < n; ++j) rank += (v[j] < x || (v[j] == x && j < e)) ? 1 : 0;
        if (rank == k) { out = x; found = 1; }
    }
    // exactly one lane found it
    const int src = __builtin_ffs((int)simt::ballot32(found != 0)) - 1;
    return shfl32_f64(out, src);
}
DEVFN void pitch_feature_warp(const PitchParams& p, int u, double* sm) {
    const int lane = simt::tid() & 31;
    const int64_t f0 = p.frame_off[u];
    const int F = (int)(p.frame_off[u + 1] - f0);
    double* out5 = p.feat + 5 * (int64_t)u;
    if (F > kFeatMaxFrames) {
        if (lane == 0) pitch_feature_tail(p.pitch + f0, p.frame_amp + f0, F, p.scratch + 3 * f0, out5);
        return;
    }
    double* pitch = sm; double* amp = sm + kFeatMaxFrames; double* s1 = amp + kFeatMaxFrames; double* s2 = s1 + kFeatMaxFrames;
    double* tmp = s2 + kFeatMaxFrames;
    for (int i = lane; i < F; i += 32) { pitch[i] = p.pitch[f0 + i]; amp[i] = p.frame_amp[f0 + i]; }
    simt::warp_sync();
    // sub_endpoint_detect (pitch.py:64-81): the first index attaining the largest valley score (> -1000), else F/2
    double bs = -1000.0; int bi = 0;
    for (int i = 10 + lane; i < F - 10; i += 32) {
        bool lower = false;
        for (int j = i - 2; j <= i + 2; ++j) lower = lower || (amp[j] < amp[i]);
        if (lower) continue;
        double sc = 0;
        for (int j = i - 10; j <= i + 10; ++j) sc += amp[j] - amp[i];
        if (sc > bs) { bs = sc; bi = i; }
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        const double os = shfl32_xor_f64(bs, m);
        const int oi = simt::shfl32_i(bi, lane ^ m);
        if (os > bs || (os == bs && oi < bi)) { bs = os; bi = oi; }
    }
    const int pv = bi == 0 ? F / 2 : bi;
    const int p_bias = pv > 15 ? 5 : 0;
    // find_smooth_subsequence on both halves (sequential), lanes 0 and 1 take one half each
    int n1 = 0, n2 = 0;
    {
        int a, b, n = 0;
        if (lane == 0) n = smooth_run(pitch + p_bias, pv - p_bias, 3, 30.0, s1, tmp, &a, &b);
        if (lane == 1) n = smooth_run(pitch + pv, F - pv, 3, 30.0, s2, tmp + pv, &a, &b);   // lane 0 uses at most pv entries of tmp
        n1 = simt::shfl32_i(n, 0); n2 = simt::shfl32_i(n, 1);
    }
    simt::warp_sync();
    if (n1 < 3 || n2 < 3) { if (lane < 5) out5[lane] = NAN; return; }
    double r = 0.0;
    if (lane == 0) r = ls_slope(s1, n1);
    if (lane == 1) r = ls_slope(s2, n2);
    if (lane == 2) r = ls_quad(s1, n1);
    if (lane == 3) r = ls_quad(s2, n2);
    if (lane < 4) out5[lane] = r;
    // np.median of both runs by rank counting across the lanes
    const double m1 = 0.5 * (warp_kth(s1, n1, (n1 - 1) >> 1, lane) + warp_kth(s1, n1, n1 >> 1, lane));
    const double m2 = 0.5 * (warp_kth(s2, n2, (n2 - 1) >> 1, lane) + warp_kth(s2, n2, n2 >> 1, lane));
    if (lane == 0) out5[4] = m2 - m1;   // peakshift(seq1, seq2) = median(seq2) - median(seq1)
}

}  // namespace dspfe
