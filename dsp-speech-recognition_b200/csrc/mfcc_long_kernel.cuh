// K1L: MFCC for every transform size other than K1's even-hop nfft = 512 (sm_100a) -- first of all the configuration the
// reference trainer really uses:
// mfcc(sound.reshape(1,-1), rate, winlen=cfg.frame, winstep=cfg.step, nfft=1536, winfunc=np.hamming) (model.py:74), i.e.
// 30 ms Hamming frames of 480 (16 kHz), 1323 (44.1 kHz) or 1440 (48 kHz) samples with hops of 160 / 441 / 480 (the odd hop
// rules out K1's even/odd sample planes), zero padded to 1536 points.  Same arithmetic chain as K1 (sigproc.py:178-185
// pre-emphasis, :66-98 framing, :151-158 power spectrum, base.py:18-32 filterbank, :8-16 log / DCT / lifter / energy).
//
// One warp per pair of consecutive frames (packed FP32: frame A in the .x halves, B in .y).  The 1536-point transform
// of the real frame is a radix-3 decimation in time around the 512-point routine of fft_regs.h:
//     X[k] = sum_{r<3} W1536^{rk} Z_r[k mod 512],   Z_r = FFT512(x[3m + r]),   k = 0..768,
// accumulated per bin in shared memory (a lane only ever touches bins congruent to its lane index, so no barrier is
// needed), then |X|^2 / 1536, triangular mel sums (one filter at a time across the lanes), log, DCT * lifter.
// Delta and delta-delta run in a second kernel over the cepstra (delta_batch_kernel).
//
// Other sizes (round 2; python_speech_features lets the caller choose NFFT, base.py:8 / sigproc.py:136-175): the same
// decimation in time with R = nfft / 512 sub-sequences for nfft = 512 (odd hops, which K1's sample planes rule out), 1024,
// 1536, 2048; for nfft = 512 / D < 512 the frame (at most nfft samples) is zero padded to 512 points and bin k of the short
// transform is bin D k of the long one.  The filterbank (base.py:18) and spectrum (sigproc.py:136-175) taps of these sizes
// leave the same code early (mode 1 / 2).
#pragma once
#include <math.h>
#include <stdint.h>

#include "fft_regs.h"
#include "simt.h"

namespace dspfe {

constexpr int kLongNfft = 1536;                  // the size with the decimation-in-frequency fast path
constexpr int kLongBins = kLongNfft / 2 + 1;     // 769
constexpr int kLongMaxNfft = 2048;
constexpr int kLongWarps = 4;
constexpr int kLongScr = 32 * 17;                // fft512's transpose tile (float2)
// float blob offsets (in floats): fft twiddles | W32 (read by no kernel, as kTabW32) | W1536^k | window | mel tables | dct
constexpr int kLtTw = 0, kLtW32 = kLtTw + 1024, kLtW1536 = kLtW32 + 64, kLtWin = kLtW1536 + 2 * kLongMaxNfft,
              kLtEdge = kLtWin + kLongMaxNfft, kLtInvUp = kLtEdge + 48, kLtInvDn = kLtInvUp + 48, kLtDct = kLtInvDn + 48,
              kLtTotal = kLtDct + 16 * 48;
// per-warp shared memory: transpose tile | X / power per bin | log-mel pair.  The accumulators need nfft/2 + 1 float4 slots; the
// decimation-in-frequency path of nfft = 1536 parks 512 float2 behind 769 + 7 float2 power values, which fits the same area.
#ifdef __CUDACC__
#define LONG_HD __host__ __device__
#else
#define LONG_HD
#endif
LONG_HD constexpr int long_warp_smem(int nfft) { return kLongScr * 8 + ((nfft < kLongNfft ? kLongNfft : nfft) / 2 + 1 + 7) * 16 + 64 * 8; }
LONG_HD constexpr int long_cta_smem(int nfft) { return (kLtW1536 * 4) + kLongWarps * long_warp_smem(nfft); }   // shared twiddles | per-warp areas
constexpr int kLongWarpSmem = long_warp_smem(kLongNfft);
constexpr int kLongCtaSmem = long_cta_smem(kLongNfft);

struct MfccLongParams {
    const void* pcm; int in_f32;
    const int64_t* seg_start;   // [U] first sample of each (trimmed) utterance inside pcm
    const int32_t* seg_len;     // [U]
    const int64_t* frame_off;   // [U+1]
    int n_utt;
    int frame_len, frame_step, nfilt, numcep, append_energy;
    float preemph;
    const float* tab;           // blob (kLt* offsets)
    float* mfcc;                // [F_total, numcep] static cepstra (mode 0), [F_total, nfilt + 1] (mode 1), [F_total, nfft/2 + 1] (mode 2)
    int64_t max_frames;
    int nfft, nbins;            // transform size, nfft / 2 + 1
    int nsub, bin_stride;       // R = max(nfft / 512, 1) sub-sequences; D = max(512 / nfft, 1): bin k = bin D k of the 512-point transform
    int warp_smem;              // long_warp_smem(nfft)
    int mode, spec_kind;        // 0 cepstra | 1 filterbank energies + frame energy | 2 spectrum (0 power, 1 magnitude, 2 10 log10 power)
    // the mel filter edges and slope reciprocals, copied out of the blob: kernel parameters are read through the constant
    // bank with uniform loads, which takes five dependent global loads per filter out of the mel loop
    int32_t mel_edge[48];
    float mel_iu[48], mel_id[48];
};
inline bool long_nfft_ok(int nfft) {
    return nfft == 32 || nfft == 64 || nfft == 128 || nfft == 256 || nfft == 512 || nfft == 1024 || nfft == 1536 || nfft == 2048;
}
inline void long_fill_size_params(MfccLongParams& p, int nfft, int mode, int spec_kind) {
    p.nfft = nfft; p.nbins = nfft / 2 + 1; p.nsub = nfft >= 512 ? nfft / 512 : 1; p.bin_stride = nfft >= 512 ? 1 : 512 / nfft;
    p.warp_smem = long_warp_smem(nfft); p.mode = mode; p.spec_kind = spec_kind;
}
inline void long_fill_mel_params(MfccLongParams& p, const float* host_tab) {
    for (int i = 0; i < 48; ++i) {
        p.mel_edge[i] = reinterpret_cast<const int32_t*>(host_tab + kLtEdge)[i];
        p.mel_iu[i] = host_tab[kLtInvUp + i]; p.mel_id[i] = host_tab[kLtInvDn + i];
    }
}

// warp-cooperative 32-ary form: three dependent loads for up to 32768 utterances instead of log2(U)
DEVFN int long_find_utt_warp(const int64_t* frame_off, int n_utt, int64_t g, int lane) {
    int lo = 0, hi = n_utt;   // invariant: frame_off[lo] <= g < frame_off[hi]
    while (hi - lo > 1) {
        const int stride = (hi - lo + 31) >> 5;
        const int i = lo + lane * stride;
        const bool le = i < hi && frame_off[i] <= g;            // true on a prefix of the lanes (lane 0 always)
        const int c = warp_redux_add(le ? 1 : 0);
        lo += (c - 1) * stride;
        hi = lo + stride < hi ? lo + stride : hi;
    }
    return lo;
}
DEVFN int long_find_utt(const int64_t* frame_off, int n_utt, int64_t g) {
    int lo = 0, hi = n_utt;   // frame_off[lo] <= g < frame_off[hi]
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (frame_off[mid] <= g) lo = mid; else hi = mid; }
    return lo;
}

// a frame's samples: base points at the frame's first sample, sample n is valid for n < lim (= min(frame_len, S - s0)), and
// n = 0 of the utterance's first frame has no predecessor (first = 1)
struct LongFrame { const unsigned char* base; int lim; int first; };
DEVFN float long_sample(const MfccLongParams& p, const LongFrame& f, int n, float w) {
    if (n >= f.lim) return 0.f;
    float cur, prev = 0.f;
    const bool has_prev = n > 0 || !f.first;
    if (p.in_f32) { const float* q = reinterpret_cast<const float*>(f.base); cur = q[n]; if (has_prev) prev = q[n - 1]; }
    else { const int16_t* q = reinterpret_cast<const int16_t*>(f.base); cur = cvt_i16(q[n]); if (has_prev) prev = cvt_i16(q[n - 1]); }
    return dsp_fmaf(-p.preemph, prev, cur) * w;      // y[0] = x[0], y[n] = x[n] - c x[n-1] (sigproc.py:185), times the window
}

// wsm: per-warp shared memory = scr[kLongScr] float2 | acc[kLongBins] float4 | lmel[64] float2
// NFFT: the transform size when known at compile time (1536: the trainer's), else 0
template <int NFFT = 0>
DEVFN void mfcc_long_pair(const MfccLongParams& p, int64_t g0, int64_t total, unsigned char* wsm, const float2* tws, const float2* /*w32s*/) {
    const int lane = simt::tid() & 31;
    float2* scr = reinterpret_cast<float2*>(wsm);
    float4* acc = reinterpret_cast<float4*>(scr + kLongScr);
    const int nfft = NFFT ? NFFT : p.nfft;
    const int nbins = NFFT ? NFFT / 2 + 1 : p.nbins;
    float2* lmel = reinterpret_cast<float2*>(wsm + p.warp_smem) - 64;
    const float2* w1536 = reinterpret_cast<const float2*>(p.tab + kLtW1536);
    const float* win = p.tab + kLtWin;
    const int32_t* edge = p.mel_edge;
    const bool hasB = g0 + 1 < total;
    const int esz = p.in_f32 ? 4 : 2;
    LongFrame fa, fb;
    {
        const int ua = long_find_utt_warp(p.frame_off, p.n_utt, g0, lane);
        const int ub = (hasB && g0 + 1 >= p.frame_off[ua + 1]) ? ua + 1 : ua;
        const int64_t sa = (g0 - p.frame_off[ua]) * p.frame_step;                 // first sample of the frame inside the utterance
        const int64_t sb = hasB ? (g0 + 1 - p.frame_off[ub]) * p.frame_step : 0;
        const int64_t ra = (int64_t)p.seg_len[ua] - sa, rb = hasB ? (int64_t)p.seg_len[ub] - sb : 0;   // samples left from the frame start
        fa.base = reinterpret_cast<const unsigned char*>(p.pcm) + (p.seg_start[ua] + sa) * esz;
        fb.base = reinterpret_cast<const unsigned char*>(p.pcm) + (p.seg_start[ub] + sb) * esz;
        fa.lim = (int)(ra < p.frame_len ? (ra > 0 ? ra : 0) : p.frame_len); fa.first = sa == 0;
        fb.lim = (int)(rb < p.frame_len ? (rb > 0 ? rb : 0) : p.frame_len); fb.first = sb == 0;
    }
    cpx2 x[16];
    const float2 zero2 = make_float2(0.f, 0.f);
    float2 esum = zero2;
    const float sc = 1.0f / (float)nfft;
    // power spectrum of the pair as compact float2 [kLongBins] (8-byte stride: the mel loop's loads are conflict-free; the
    // float4 slots of the accumulation path put consecutive bins 16 bytes apart, a 4-way conflict on every scalar access)
    float2* pw2 = reinterpret_cast<float2*>(acc);
    float2* parked = pw2 + kLongBins + 7;            // [512] the windowed samples between the two passes (inside acc's area)
    if (nfft == kLongNfft && p.frame_len <= 512) {
        // Frames that fit 512 samples (30 ms at 16 kHz = 480): decimation in FREQUENCY.  X[3q + r] = FFT512(x[n] W1536^{n r})[q],
        // and for real x the bins 3q + 2 mirror the bins 3q' + 1 (X[1536 - k] = conj X[k], k = 3q'+1 -> 3(511 - q') + 2), so
        // two transforms in natural order give every power bin straight from the registers: r = 0 -> bins 3q (q <= 256),
        // r = 1 -> bins 3q + 1 (q <= 255) and 3(511 - q) + 2 (q >= 256).  No per-bin accumulation pass, coalesced sample loads.
#pragma unroll 1
        for (int r = 0; r < 2; ++r) {
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const int n = 32 * t + lane;
                float2 v, m = make_float2(1.f, 0.f);
                if (r == 0) {   // windowed, pre-emphasised samples; parked in the unused half of the lane's own bin slots for r = 1
                    const float w = ldg(win + n);
                    v = make_float2(long_sample(p, fa, n, w), long_sample(p, fb, n, w));
                    parked[n] = v;
                } else {
                    v = parked[n];
                    m = ldg(w1536 + n);
                }
                x[t].re = f2muls(v, m.x); x[t].im = f2muls(v, m.y);
            }
            fft512(x, scr, tws, lane);
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const int q = 32 * t + lane;
                const float2 pw = f2muls(f2fma(x[t].im, x[t].im, f2mul(x[t].re, x[t].re)), sc);
                int k = -1;
                if (r == 0) { if (q <= 256) k = 3 * q; }
                else k = q <= 255 ? 3 * q + 1 : 3 * (511 - q) + 2;
                if (k >= 0) { pw2[k] = pw; esum = f2add(esum, pw); }
            }
        }
    } else {
    const int R = NFFT ? (NFFT >= 512 ? NFFT / 512 : 1) : p.nsub, D = NFFT ? (NFFT >= 512 ? 1 : 512 / NFFT) : p.bin_stride, half = nfft >> 1;
#pragma unroll 1
    for (int r = 0; r < R; ++r) {
        // sub-sequence r: element m = 32 t + lane is sample n = R m + r of the frame
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            const int n = R * (32 * t + lane) + r;
            const float w = ldg(win + n);                   // zero past the frame
            x[t].re = make_float2(long_sample(p, fa, n, w), long_sample(p, fb, n, w));
            x[t].im = zero2;
        }
        fft512(x, scr, tws, lane);
        // X[k] += W_nfft^{r k} Z_r[k mod 512] for every bin k = j + 512 c <= nfft / 2, j = 32 t + lane (nfft >= 512);
        // X[k] = Z_0[D k] for the short transforms
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            const int j = 32 * t + lane;
            if (D > 1) {
                if ((j & (D - 1)) == 0 && j / D <= half) acc[j / D] = make_float4(x[t].re.x, x[t].re.y, x[t].im.x, x[t].im.y);
                continue;
            }
            for (int k = j; k <= half; k += 512) {
                cpx2 v = x[t];
                float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
                if (r > 0) {
                    int i = r * k; if (i >= nfft) i -= nfft;     // r k < 2 nfft for R <= 4
                    const float2 w = ldg(w1536 + i); v = cmuls(x[t], w.x, w.y); a = acc[k];
                }
                acc[k] = make_float4(a.x + v.re.x, a.y + v.re.y, a.z + v.im.x, a.w + v.im.y);
            }
        }
    }
    simt::warp_sync();   // the short transforms' bins were written by other lanes
    // power spectrum |X|^2 / NFFT (sigproc.py:158) into the .x / .y of the bin's own slot; frame energy = sum over all bins
    // (bin k's float2 slot pw2[k] lies below its float4 accumulator acc[k] and is only written after acc[k] was read by the
    // same lane; other lanes' accumulators at or below byte 8k + 8 belong to bins <= k/2, read by the same loop iteration or earlier)
    for (int k0 = 0; k0 < nbins; k0 += 32) {
        const int k = k0 + lane;
        float2 pw = zero2;
        if (k < nbins) { const float4 a = acc[k]; pw = make_float2((a.x * a.x + a.z * a.z) * sc, (a.y * a.y + a.w * a.w) * sc); }
        simt::warp_sync();
        if (k < nbins) { pw2[k] = pw; esum.x += pw.x; esum.y += pw.y; }
        simt::warp_sync();
    }
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) { esum.x += simt::shfl32_xor(esum.x, m); esum.y += simt::shfl32_xor(esum.y, m); }
    simt::warp_sync();
    if (p.mode == 2) {   // spectrum tap (sigproc.py:136-175): rows straight to global memory
        const float nf = (float)nfft;
        for (int k = lane; k < nbins; k += 32) {
            float2 v = pw2[k];
            if (p.spec_kind == 1) { v.x = sqrtf(v.x * nf); v.y = sqrtf(v.y * nf); }
            else if (p.spec_kind == 2) { v.x = 10.f * log10f(fmaxf(v.x, 1e-30f)); v.y = 10.f * log10f(fmaxf(v.y, 1e-30f)); }
            p.mfcc[g0 * nbins + k] = v.x;
            if (hasB) p.mfcc[(g0 + 1) * nbins + k] = v.y;
        }
        return;
    }
    // mel filterbank (base.py:40-58): filter j rises over [e_j, e_{j+1}) and falls over [e_{j+1}, e_{j+2}); one filter at a
    // time, its bins spread over the lanes
    const float eps64 = 2.220446049250313e-16f;   // numpy.finfo(float64).eps floor (base.py:26,30)
    const float* inv_up = p.mel_iu;
    const float* inv_dn = p.mel_id;
    // four filters at a time: each lane gathers its share of the four sums, then a transposing reduction (the lanes split
    // the four sums among themselves while they halve the lane distance) brings a filter's total to eight lanes with 12 shuffles
    // per group instead of 10 per filter, and every lane takes the logarithm of one filter only
    for (int j0 = 0; j0 < p.nfilt; j0 += 4) {
        float2 f[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = j0 + u;
            f[u] = zero2;
            if (j < p.nfilt) {
                const int lo = edge[j], mid = edge[j + 1], hi = edge[j + 2];
                const float iu = inv_up[j], id = inv_dn[j];
                for (int k = lo + lane; k < hi; k += 32) {
                    const float w = k < mid ? (float)(k - lo) * iu : (float)(hi - k) * id;
                    const float2 pk = pw2[k];
                    f[u].x = dsp_fmaf(w, pk.x, f[u].x); f[u].y = dsp_fmaf(w, pk.y, f[u].y);
                }
            }
        }
        const bool up16 = (lane & 16) != 0, up8 = (lane & 8) != 0;
        float2 k0 = up16 ? f[2] : f[0], k1 = up16 ? f[3] : f[1];
        const float2 s0 = up16 ? f[0] : f[2], s1 = up16 ? f[1] : f[3];
        k0.x += simt::shfl32_xor(s0.x, 16); k0.y += simt::shfl32_xor(s0.y, 16);
        k1.x += simt::shfl32_xor(s1.x, 16); k1.y += simt::shfl32_xor(s1.y, 16);
        float2 kk = up8 ? k1 : k0;
        const float2 ss = up8 ? k0 : k1;
        kk.x += simt::shfl32_xor(ss.x, 8); kk.y += simt::shfl32_xor(ss.y, 8);
#pragma unroll
        for (int m = 4; m >= 1; m >>= 1) { kk.x += simt::shfl32_xor(kk.x, m); kk.y += simt::shfl32_xor(kk.y, m); }
        const int jm = j0 + (up16 ? 2 : 0) + (up8 ? 1 : 0);
        if ((lane & 7) == 0 && jm < p.nfilt) {
            if (kk.x == 0.f) kk.x = eps64;
            if (kk.y == 0.f) kk.y = eps64;
            if (p.mode == 1) {   // filterbank tap (base.py:18-32): energies, column nfilt = frame energy
                p.mfcc[g0 * (p.nfilt + 1) + jm] = kk.x;
                if (hasB) p.mfcc[(g0 + 1) * (p.nfilt + 1) + jm] = kk.y;
            } else {
                lmel[jm] = make_float2(dsp_fast_logf(kk.x), dsp_fast_logf(kk.y));
            }
        }
    }
    if (esum.x == 0.f) esum.x = eps64;
    if (esum.y == 0.f) esum.y = eps64;
    if (p.mode == 1) {
        if (lane == 0) { p.mfcc[g0 * (p.nfilt + 1) + p.nfilt] = esum.x; if (hasB) p.mfcc[(g0 + 1) * (p.nfilt + 1) + p.nfilt] = esum.y; }
        return;
    }
    if (lane == 0) lmel[p.nfilt] = make_float2(dsp_fast_logf(esum.x), dsp_fast_logf(esum.y));
    simt::warp_sync();
    // DCT-II (ortho) * lifter (base.py:12-14), c0 := log(energy) (base.py:15)
    if (lane < p.numcep) {
        const float* d = p.tab + kLtDct + lane * 48;
        float2 c = zero2;
        for (int j = 0; j < p.nfilt; ++j) { const float2 l = lmel[j]; c.x = dsp_fmaf(d[j], l.x, c.x); c.y = dsp_fmaf(d[j], l.y, c.y); }
        if (lane == 0 && p.append_energy) c = lmel[p.nfilt];
        p.mfcc[g0 * p.numcep + lane] = c.x;
        if (hasB) p.mfcc[(g0 + 1) * p.numcep + lane] = c.y;
    }
    simt::warp_sync();
}

// delta + delta-delta (base.py:70-79 twice, model.py:76-77) over per-utterance cepstra: one thread per (frame, column).
// The second pass pads the DELTA array at the utterance edges (SURVEY Appendix A-5), so it is evaluated as the weighted
// sum of clamped deltas, each a weighted sum of clamped cepstra.
DEVFN void delta_batch_thread(const float* mf, const int64_t* frame_off, int n_utt, int C, int N, float scale, int64_t i, float* out) {
    const int64_t g = i / C;
    const int c = (int)(i - g * C);
    const int u = long_find_utt(frame_off, n_utt, g);
    const int64_t r0 = frame_off[u];
    const int F = (int)(frame_off[u + 1] - r0);
    const int t = (int)(g - r0);
    auto clampf = [&](int a) { return a < 0 ? 0 : (a > F - 1 ? F - 1 : a); };
    auto d1 = [&](int a) {   // delta at the (clamped) frame a
        float acc = 0.f;
        for (int n = 1; n <= N; ++n) acc = dsp_fmaf((float)n, mf[(r0 + clampf(a + n)) * C + c] - mf[(r0 + clampf(a - n)) * C + c], acc);
        return acc * scale;
    };
    float dd = 0.f;
    for (int n = 1; n <= N; ++n) dd = dsp_fmaf((float)n, d1(clampf(t + n)) - d1(clampf(t - n)), dd);
    float* o = out + g * 3 * C;
    o[c] = mf[g * C + c]; o[C + c] = d1(t); o[2 * C + c] = dd * scale;
}

}  // namespace dspfe
