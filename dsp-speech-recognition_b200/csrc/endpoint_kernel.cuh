// K2/K3: energy + zero-crossing endpoint detection over a ragged batch (sm_100a).
//
// Replaces reference features/endpoint.py: get_amplitude (:109), get_zcr (:182), amplitude_rule (:133),
// zcr_rule (:201) and their driver basic_endpoint_detection (:34), on raw int16 PCM.
//   K2a  one warp per hop block (frame_step samples): exact int32 sum |x|, sign changes inside the block,
//        sign change across the boundary to the next block, and the same for the first (frame_len % step)
//        samples (frames that are not a whole number of hops);
//   K2b  one thread per frame: combines the block partials into sum|x| and the zero-crossing count of the
//        frame (zero padding past the end of the utterance is implicit: sigproc.py:84-87);
//   K3   one thread per utterance: the reference's double-threshold state machine, replayed in float64 with
//        NumPy's pairwise summation order so that thresholds, and therefore (left, right), are bit-exact.
// All statistics are integers, so amp = sum/frame_len (one float64 divide on the host) equals the
// reference's np.mean exactly.
//   K2f  float32 samples instead (dspfe_endpoint_f32): the frame statistics in the reference's float64 arithmetic,
//        amp = np.mean(np.abs(frame)) in NumPy's pairwise order (np_pairwise.h) and the exact sign-change count; K3
//        then reads the float64 amplitudes (AmpFromF64).  Its body is also compiled onto the test emulator.
//   K3r  robust_endpoint_detection (endpoint.py:68-92): the rule gated by acr_rule, a CTA per utterance; a template over the sample
//        type (int16: exact integer lag sums, float32: NumPy's pairwise float64 sums, acr_lag).
#pragma once
#include <math.h>
#include <stdint.h>

#include <vector>

#include "dspfe_types.h"
#include "np_pairwise.h"
#include "simt.h"

#ifdef __CUDACC__
#define DSP_HD __host__ __device__ inline
#else
#define DSP_HD inline
#endif

namespace dspfe {

struct EpRule {           // reference call-site constants (endpoint.py:42-45,56,60-64,133,201)
    double cfg_frame;     // 0.03  (config.py:31)
    double cfg_step;      // 0.01  (config.py:32)
    double mh1, mh2;      // 0.25, then 0.125 when the span is shorter than min_span
    double th;            // 0.1 s above the high threshold
    double l_sil, r_sil;  // 0.1 s of assumed silence either side
    double sigma;         // 3
    double zcr_max_shift; // 0.4 s
    double zcr_r_sil;     // 0.1 s
    int min_span;         // 50 frames
    int rate;
};

// numpy's pairwise summation (DOUBLE_pairwise_sum).  Callers pass n <= 64, so only numpy's n < 8 and
// n <= 128 branches are needed (no recursion: device stack stays within the default 1 KB).
DSP_HD double np_pairwise_sum(const double* a, int n) {
    if (n < 8) {
        double res = 0.;
        for (int i = 0; i < n; ++i) res += a[i];
        return res;
    }
    if (n <= 128) {
        double r0 = a[0], r1 = a[1], r2 = a[2], r3 = a[3], r4 = a[4], r5 = a[5], r6 = a[6], r7 = a[7];
        int i = 8;
        for (; i < n - (n % 8); i += 8) {
            r0 += a[i]; r1 += a[i + 1]; r2 += a[i + 2]; r3 += a[i + 3];
            r4 += a[i + 4]; r5 += a[i + 5]; r6 += a[i + 6]; r7 += a[i + 7];
        }
        double res = ((r0 + r1) + (r2 + r3)) + ((r4 + r5) + (r6 + r7));
        for (; i < n; ++i) res += a[i];
        return res;
    }
    return NAN;   // unreachable for n <= 128
}

// np.mean / np.std (population) of up to 64 values, numpy operation order.  n == 0 gives NaN like numpy.
DSP_HD void np_mean_std(const double* a, int n, double* mean, double* std) {
    if (n <= 0) { *mean = NAN; *std = NAN; return; }
    const double m = np_pairwise_sum(a, n) / (double)n;
    double sq[64];
    for (int i = 0; i < n; ++i) { const double d = a[i] - m; sq[i] = d * d; }
    *mean = m;
    *std = sqrt(np_pairwise_sum(sq, n) / (double)n);
}

// Frame statistics come either as exact integer sums (device path: amp = sum|x| / frame_len) or as float64
// values (host entry points that mirror the reference's list-based API).
struct AmpFromSum { const int32_t* s; double len; DSP_HD double operator()(int i) const { return (double)s[i] / len; } };
struct AmpFromF64 { const double* a; DSP_HD double operator()(int i) const { return a[i]; } };
struct ZcrFromI32 { const int32_t* z; DSP_HD double operator()(int i) const { return (double)z[i]; } };

// amplitude_rule (endpoint.py:133-179).  Writes up to seg_cap (j,k) pairs to segs (may be null) and returns the
// number of segments found; *left/*right = first segment start / last segment end, or (0, F) when none qualifies.
// Gate of the expansion loops: always open for the basic rule; robust_endpoint_detection closes it on frames whose
// normalised autocorrelation peak is below 0.55 (acr_rule, endpoint.py:142-144).
// hint(dir, M_L): the walk about to start moves by dir (-1 / +1) per frame and continues while amp > M_L and the gate holds; a
// gate that is expensive may evaluate the frames ahead speculatively (K3r).
struct GateOpen { DSP_HD bool operator()(int) const { return true; } DSP_HD void hint(int, double) {} };
struct GateFromFlags { const int32_t* g; DSP_HD bool operator()(int i) const { return g[i] != 0; } DSP_HD void hint(int, double) {} };

template <class Amp, class Gate = GateOpen>
DSP_HD int amplitude_rule(Amp amp, int F, const EpRule& r, double mh, int* left, int* right, int32_t* segs = nullptr, int seg_cap = 0,
                          Gate gate = Gate()) {
    const int nl = (int)(r.l_sil / r.cfg_step), nr = (int)(r.r_sil / r.cfg_step);
    double sil[64];
    int n = 0;
    // amp[:nl] + amp[-nr:] with Python slice clamping (amp[-0:] is the whole list)
    for (int i = 0; i < nl && i < F && n < 64; ++i) sil[n++] = amp(i);
    for (int i = (nr > 0 && F - nr > 0 ? F - nr : 0); i < F && n < 64; ++i) sil[n++] = amp(i);
    // sorted(sil)[:-2]
    for (int i = 1; i < n; ++i) { double v = sil[i]; int j = i - 1; while (j >= 0 && sil[j] > v) { sil[j + 1] = sil[j]; --j; } sil[j + 1] = v; }
    n = n - 2 > 0 ? n - 2 : 0;
    double s_mean, s_sigma;
    np_mean_std(sil, n, &s_mean, &s_sigma);
    const double T_H = r.th / r.cfg_frame;
    const double M_L = s_mean + r.sigma * s_sigma;
    double amax = amp(0);
    for (int i = 1; i < F; ++i) { const double v = amp(i); amax = v > amax ? v : amax; }
    const double a_hi = amax * mh;
    const double M_H = (M_L > a_hi) ? M_L : a_hi;   // Python max(a_hi, M_L): a NaN M_L keeps a_hi
    int first = -1, last = -1, nseg = 0;
    int i = 0;
    while (i < F) {
        if (amp(i) >= M_H) {
            int j = i, k = i;
            while (k < F && amp(k) > M_H) ++k;
            if ((double)(k - j) < T_H) {
                i = k;
            } else {
                gate.hint(-1, M_L);
                while (j > 0 && amp(j) > M_L && gate(j)) --j;
                gate.hint(+1, M_L);
                while (k < F && amp(k) > M_L && gate(k)) ++k;
                if (first < 0) first = j;
                last = k;
                if (segs && nseg < seg_cap) { segs[2 * nseg] = j; segs[2 * nseg + 1] = k; }
                ++nseg;
                i = k;
            }
        }
        ++i;
    }
    if (first < 0) { *left = 0; *right = F; } else { *left = first; *right = last; }
    return nseg;
}

// zcr_rule (endpoint.py:201-220); l_sil is a parameter of the reference function but its only caller uses 0
template <class Zcr>
DSP_HD void zcr_rule(Zcr zcr, int F, const EpRule& r, double l_sil, int left, int right, int* l2, int* r2) {
    const double max_shift = r.zcr_max_shift / r.cfg_frame;
    const int nl = (int)(l_sil / r.cfg_step), nr = (int)(r.zcr_r_sil / r.cfg_step);
    double sil[64];
    int n = 0;
    for (int i = 0; i < nl && i < F && n < 64; ++i) sil[n++] = zcr(i);
    for (int i = (nr > 0 && F - nr > 0 ? F - nr : 0); i < F && n < 64; ++i) sil[n++] = zcr(i);
    double mu, sg;
    np_mean_std(sil, n, &mu, &sg);
    const double thres = mu + 3 * sg;
    int j = left;
    while (j > 0 && (double)(left - j) <= max_shift && zcr(j) > thres) --j;
    int k = right;
    while (k < F && (double)(k - right) <= max_shift && zcr(k) > thres) ++k;
    *l2 = j; *r2 = k;
}

// basic_endpoint_detection (endpoint.py:34-66): frame-level decision + conversion to sample indices.
template <class Amp>
DSP_HD void endpoint_decide_amp(Amp amp, const int32_t* zcr, int F, const EpRule& r, int32_t* out_lr);
DSP_HD void endpoint_decide(const int32_t* asum, const int32_t* zcr, int F, int frame_len, const EpRule& r, int32_t* out_lr) {
    endpoint_decide_amp(AmpFromSum{asum, (double)frame_len}, zcr, F, r, out_lr);
}
template <class Amp>
DSP_HD void endpoint_decide_amp(Amp amp, const int32_t* zcr, int F, const EpRule& r, int32_t* out_lr) {
    int left, right;
    amplitude_rule(amp, F, r, r.mh1, &left, &right);
    if (right - left < r.min_span) amplitude_rule(amp, F, r, r.mh2, &left, &right);
    int l2, r2;
    zcr_rule(ZcrFromI32{zcr}, F, r, 0.0, left, right, &l2, &r2);
    if (r2 - l2 < r.min_span) { l2 = 0; r2 = F; }
    // int(left2 * cfg.step * rate): float64 product evaluated left to right, truncated (Appendix A-9)
    out_lr[0] = (int32_t)((double)l2 * r.cfg_step * (double)r.rate);
    out_lr[1] = (int32_t)((double)r2 * r.cfg_step * (double)r.rate);
}

// acr_rule (endpoint.py:142-144) from exact integer lag sums: acr(frame, n) = sum_i x[i] x[i+n] / (len - n)
// (sigproc.py:48-53; the products of int16 samples and their sums are exact in the reference's float64 too), gate =
// max_n acr(n) / acr(0) > 0.55 over n in [rate // 500, rate // 50).  best = max_n S_n / (len - n) as computed by the caller.
DSP_HD bool acr_gate_decide(double best, long long s0, int len) {
    const double a0 = (double)s0 / (double)len;
    return best / a0 > 0.55;          // 0 / 0 = NaN compares false, as in the reference
}
// plain sequential form (host entry points, utterances too long for the staged kernel)
DSP_HD bool acr_gate_frame(const int16_t* x, long long avail, int len, int n0, int n1) {
    // x[i] for i < avail, zero beyond (sigproc.py:84-87)
    long long s0 = 0;
    for (int i = 0; i < len && i < avail; ++i) s0 += (long long)x[i] * x[i];
    double best = 0.0; bool any = false;
    for (int n = n0; n < n1 && n < len; ++n) {
        long long sn = 0;
        for (int i = 0; i + n < len && i + n < avail; ++i) sn += (long long)x[i] * x[i + n];
        const double a = (double)sn / (double)(len - n);
        if (!any || a > best) { best = a; any = true; }
    }
    return any && acr_gate_decide(best, s0, len);
}

// acr(frame, n) (sigproc.py:48-53) of a float32 frame x[0..avail) with framesig's float64 zero tail up to len samples: NumPy's
// pairwise float64 sum of the len - n products x[i] x[i+n], divided by len - n; n = 0 is acr(frame, 0).  The product of two
// float32 values is exact in float64 (it neither overflows nor underflows to zero), so only the order of the sum matters, and
// every lag has its own split tree.  Shared by the serial gate below and the exact fallback of K3r's float gate.
DSP_HD double acr_lag(const float* x, int avail, int len, int n) {
    const double s = np_pairwise_sum_any([x, avail, n](int i) { return i + n < avail ? (double)x[i] * (double)x[i + n] : 0.0; }, len - n);
    return s / (double)(len - n);
}
// acr_rule of a float32 frame, serial.  A NaN or +-inf sample makes acr(frame, 0) NaN or +inf, and every ratio NaN, 0 or
// NaN / inf: the gate is false.  An all-zero frame gives 0 / 0, false as well.
DSP_HD bool acr_gate_frame(const float* x, long long avail, int len, int n0, int n1) {
    const int nv = avail < (long long)len ? (avail > 0 ? (int)avail : 0) : len;
    const double a0 = acr_lag(x, nv, len, 0);
    if (!isfinite(a0)) return false;
    double best = 0.0; bool any = false;
    for (int n = n0; n < n1 && n < len; ++n) {
        const double a = acr_lag(x, nv, len, n);
        if (!any || a > best) { best = a; any = true; }
    }
    return any && best / a0 > 0.55;
}

// robust_endpoint_detection (endpoint.py:68-92): amplitude_rule(mh = 0.5) with the gate, zcr_rule, whole-signal fallback
template <class Amp, class Gate>
DSP_HD void endpoint_decide_robust(Amp amp, const int32_t* zcr, int F, const EpRule& r, Gate gate, int32_t* out_lr) {
    int left, right;
    amplitude_rule(amp, F, r, 0.5, &left, &right, nullptr, 0, gate);
    int l2, r2;
    zcr_rule(ZcrFromI32{zcr}, F, r, 0.0, left, right, &l2, &r2);
    if (r2 - l2 < r.min_span) { l2 = 0; r2 = F; }
    out_lr[0] = (int32_t)((double)l2 * r.cfg_step * (double)r.rate);
    out_lr[1] = (int32_t)((double)r2 * r.cfg_step * (double)r.rate);
}

struct EpParams {
    const int16_t* pcm;
    const int64_t* offsets;    // [U+1]
    int n_utt;
    int frame_len, frame_step; // int(rate*cfg.frame), int(cfg.step*rate)  (sigproc.py:19)
    int q, rem;                // frame_len = q*frame_step + rem
    // workspaces / outputs
    int64_t* frame_off;        // [U+1] endpoint-frame prefix sums
    int64_t* block_off;        // [U+1] hop-block prefix sums
    int32_t* blk;              // [total_blocks, 6]: A, Z, C, A', Z', pad
    int32_t* asum;             // [F_total]
    int32_t* zcr;              // [F_total]
    int32_t* lr;               // [U, 2]
    int64_t max_blocks, max_frames;
    EpRule rule;
    int32_t* order;            // optional [U]: the utterances by descending frame count (K3r takes them longest first); null = identity
    const double* amp;         // float-sample path: [F_total] float64 amplitudes written by K2f (K3 reads them instead of asum)
    const float* pcm_f32;      // float-sample path: the samples K3r's gate reads instead of pcm
};

// ---- K2f: frame statistics of float32 samples (basic_endpoint_detection's get_amplitude and get_zcr, endpoint.py:109,182).
// framesig builds the frames in float64 (the zero padding is float64), so every sample enters as its exact float64 value:
//   amp[f] = np.mean(np.abs(frame)): the pairwise sum of the L absolute values, then one division by L;
//   zcr[f] = #{i : x[i] * x[i+1] < 0}: the float64 product of two float32 values is exact and never underflows to zero, so
//            this is the sign test "both nonzero, opposite signs" (a zero, -0.0 included, never counts; NaN never counts).
// The split tree of the pairwise sum depends only on L: the plan lays it out once (np_pairwise_tree).  A CTA takes a run of
// consecutive frames, stages the samples they cover once with 16-byte loads (frames overlap about L / S times), and one
// thread sums one leaf of one frame with pairwise_block; one thread per frame then adds the leaves in the tree's order.
constexpr int kEpF32Threads = 256;
constexpr int kEpF32MaxLen = 8192;        // frame lengths above this are not built (DSPFE_ERR_UNSUPPORTED)
constexpr int kEpF32SpanFloats = 8192;    // staged samples a run aims at (32 KB)

// The split tree of NumPy's pairwise sum of n terms: nleaf leaves (offset, length) in order, then the nleaf - 1 inner nodes
// (left, right) in post order, where node k < nleaf is leaf k and node nleaf + j is inner node j.
inline std::vector<int32_t> np_pairwise_tree(int n, int* nleaf) {
    std::vector<int32_t> leaves, inner;
    struct Walk {
        std::vector<int32_t>& leaves; std::vector<int32_t>& inner;
        int rec(int off, int len) {           // returns the node id with leaves numbered first (fixed up below)
            if (len <= kNpPairwiseBlock) { leaves.push_back(off); leaves.push_back(len); return (int)leaves.size() / 2 - 1; }
            const int n2 = np_pairwise_split(len);
            const int l = rec(off, n2), r = rec(off + n2, len - n2);
            inner.push_back(l); inner.push_back(r);
            return -(int)inner.size() / 2;    // inner node j as -(j + 1)
        }
    } w{leaves, inner};
    w.rec(0, n);
    const int nl = (int)leaves.size() / 2;
    for (auto& v : inner) if (v < 0) v = nl + (-v - 1);
    *nleaf = nl;
    leaves.insert(leaves.end(), inner.begin(), inner.end());
    return leaves;
}

struct EpF32Params {
    const float* pcm;          // 16-byte aligned
    int64_t total_samples;
    const int64_t* offsets;    // [U+1]
    const int64_t* frame_off;  // [U+1] (ep_prep_kernel)
    int n_utt;
    int frame_len, frame_step;
    const int32_t* tree;       // np_pairwise_tree(frame_len)
    int nleaf;
    int run;                   // frames per CTA
    int span_floats;           // staging capacity, a multiple of 4
    int sm_fr, sm_zc, sm_tree, sm_span, sm_total;   // shared-memory carve-up in bytes (nodes at 0)
    int64_t max_frames;
    double* amp;               // [F_total]
    int32_t* zcr;              // [F_total]
};

// frames per CTA and the shared-memory carve-up
inline void ep_f32_layout(EpF32Params& p) {
    const int L = p.frame_len, S = p.frame_step, nl = p.nleaf;
    int run = (kEpF32SpanFloats - L - 4) / S + 1;
    const int by_tasks = (4 * kEpF32Threads) / nl;
    if (run > by_tasks) run = by_tasks;
    if (run < 1) run = 1;
    p.run = run;
    p.span_floats = (int)(((int64_t)(run - 1) * S + L + 3 + 3) & ~(int64_t)3);
    const int node_bytes = run * (2 * nl - 1) * 8;
    p.sm_fr = node_bytes;                                  // [run] (data start, data end) int64 pairs
    p.sm_span = (p.sm_fr + run * 16 + 15) & ~15;
    p.sm_zc = p.sm_span + p.span_floats * 4;
    p.sm_tree = p.sm_zc + run * nl * 4;
    p.sm_total = p.sm_tree + (4 * nl - 2) * 4;
}

// largest u with off[u] <= g
#ifdef __CUDACC__
__device__
#endif
inline int find_owner(const int64_t* off, int n, int64_t g) {
    int lo = 0, hi = n;   // off[lo] <= g < off[hi]
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (off[mid] <= g) lo = mid; else hi = mid; }
    return lo;
}

DEVFN void ep_f32_stats_cta(const EpF32Params& p, unsigned char* smem) {
    double* s_node = reinterpret_cast<double*>(smem);
    int64_t* s_fr = reinterpret_cast<int64_t*>(smem + p.sm_fr);
    float* s_x = reinterpret_cast<float*>(smem + p.sm_span);
    int32_t* s_zc = reinterpret_cast<int32_t*>(smem + p.sm_zc);
    int32_t* s_tree = reinterpret_cast<int32_t*>(smem + p.sm_tree);
    const int tid = simt::tid(), nt = simt::nthreads();
    const int L = p.frame_len, S = p.frame_step, nl = p.nleaf, nnode = 2 * nl - 1;
    int64_t F_total = p.frame_off[p.n_utt];
    if (F_total > p.max_frames) F_total = p.max_frames;
    const int64_t g0 = (int64_t)simt::bid() * p.run;
    if (g0 >= F_total) return;                            // uniform over the CTA
    const int nf = (int)(F_total - g0 < p.run ? F_total - g0 : p.run);
    for (int i = tid; i < 4 * nl - 2; i += nt) s_tree[i] = p.tree[i];
    // the samples of frame g: [ds, de) of the packed buffer, with ds <= de <= end of its utterance; both non-decreasing in g
    for (int f = tid; f < nf; f += nt) {
        const int64_t g = g0 + f;
        const int u = find_owner(p.frame_off, p.n_utt, g);
        const int64_t a = p.offsets[u] + (g - p.frame_off[u]) * S, e = p.offsets[u + 1];
        s_fr[2 * f] = a < e ? a : e;
        s_fr[2 * f + 1] = a + L < e ? a + L : e;
    }
    simt::cta_sync();
    const int64_t lo4 = s_fr[0] & ~(int64_t)3, hi = s_fr[2 * nf - 1];
    const bool staged = hi - lo4 <= p.span_floats;     // a run over many short utterances can cover more: it reads global memory
    if (staged) {
        const int nvec = (int)((hi - lo4 + 3) >> 2);
        for (int v = tid; v < nvec; v += nt) {
            const int64_t s = lo4 + 4 * (int64_t)v;
            float4 w;
            if (s + 4 <= p.total_samples) {
                w = ldg(reinterpret_cast<const float4*>(p.pcm + s));
            } else {
                w.x = s < p.total_samples ? p.pcm[s] : 0.f;
                w.y = s + 1 < p.total_samples ? p.pcm[s + 1] : 0.f;
                w.z = s + 2 < p.total_samples ? p.pcm[s + 2] : 0.f;
                w.w = 0.f;
            }
            *reinterpret_cast<float4*>(s_x + 4 * v) = w;
        }
    }
    simt::cta_sync();
    // one leaf of one frame per thread; samples past the data of the frame are framesig's zero padding
    for (int t = tid; t < nf * nl; t += nt) {
        const int f = t / nl, k = t - f * nl;
        const int64_t ds = s_fr[2 * f];
        const int avail = (int)(s_fr[2 * f + 1] - ds);
        const float* x = staged ? s_x + (ds - lo4) : p.pcm + ds;
        const int o = s_tree[2 * k], n = s_tree[2 * k + 1];
        s_node[f * nnode + k] = pairwise_block([x, o, avail](int i) { const int j = o + i; return j < avail ? fabs((double)x[j]) : 0.0; }, n);
        int zc = 0;
        const int jend = o + n < avail - 1 ? o + n : avail - 1;
        for (int j = o; j < jend; ++j) {
            const float a = x[j], b = x[j + 1];
            zc += ((a < 0.f && b > 0.f) || (a > 0.f && b < 0.f)) ? 1 : 0;
        }
        s_zc[t] = zc;
    }
    simt::cta_sync();
    for (int f = tid; f < nf; f += nt) {
        double* v = s_node + f * nnode;
        for (int j = 0; j < nl - 1; ++j) v[nl + j] = v[s_tree[2 * nl + 2 * j]] + v[s_tree[2 * nl + 2 * j + 1]];
        int zc = 0;
        for (int k = 0; k < nl; ++k) zc += s_zc[f * nl + k];
        p.amp[g0 + f] = v[nnode - 1] / (double)L;
        p.zcr[g0 + f] = zc;
    }
}

#ifdef __CUDACC__
constexpr int kEpPrepThreads = 1024;

// hop blocks an utterance with F frames touches
__device__ inline int64_t ep_blocks(int64_t F, int q, int rem) { return F - 1 + q + (rem > 0 ? 1 : 0); }

__global__ void __launch_bounds__(kEpPrepThreads) ep_prep_kernel(EpParams p) {
    __shared__ long long s_f[kEpPrepThreads], s_b[kEpPrepThreads];
    const int tid = threadIdx.x;
    const int per = (p.n_utt + kEpPrepThreads - 1) / kEpPrepThreads;
    const int u0 = min(tid * per, p.n_utt), u1 = min(u0 + per, p.n_utt);
    long long f = 0, b = 0;
    for (int u = u0; u < u1; ++u) {
        const long long F = num_frames(p.offsets[u + 1] - p.offsets[u], p.frame_len, p.frame_step);
        f += F; b += ep_blocks(F, p.q, p.rem);
    }
    s_f[tid] = f; s_b[tid] = b;
    __syncthreads();
    for (int d = 1; d < kEpPrepThreads; d <<= 1) {
        long long x = tid >= d ? s_f[tid - d] : 0, y = tid >= d ? s_b[tid - d] : 0;
        __syncthreads();
        s_f[tid] += x; s_b[tid] += y;
        __syncthreads();
    }
    long long fo = s_f[tid] - f, bo = s_b[tid] - b;
    for (int u = u0; u < u1; ++u) {
        const long long F = num_frames(p.offsets[u + 1] - p.offsets[u], p.frame_len, p.frame_step);
        p.frame_off[u] = fo; p.block_off[u] = bo;
        fo += F; bo += ep_blocks(F, p.q, p.rem);
    }
    if (tid == kEpPrepThreads - 1) { p.frame_off[p.n_utt] = s_f[tid]; p.block_off[p.n_utt] = s_b[tid]; }
    if (p.order) {   // counting sort by frame count, descending (bins of one frame; the longest utterances share the last bin)
        __syncthreads();
        int* bins = reinterpret_cast<int*>(s_f);
        int* start = reinterpret_cast<int*>(s_b);
        bins[tid] = 0;
        __syncthreads();
        for (int u = u0; u < u1; ++u) {
            const long long F = num_frames(p.offsets[u + 1] - p.offsets[u], p.frame_len, p.frame_step);
            atomicAdd(&bins[F < kEpPrepThreads - 1 ? (int)F : kEpPrepThreads - 1], 1);
        }
        __syncthreads();
        start[tid] = bins[tid];
        __syncthreads();
        for (int d = 1; d < kEpPrepThreads; d <<= 1) {
            const int v = tid + d < kEpPrepThreads ? start[tid + d] : 0;
            __syncthreads();
            start[tid] += v;
            __syncthreads();
        }
        const int mine = start[tid] - bins[tid];
        __syncthreads();
        start[tid] = mine;
        __syncthreads();
        for (int u = u0; u < u1; ++u) {
            const long long F = num_frames(p.offsets[u + 1] - p.offsets[u], p.frame_len, p.frame_step);
            p.order[atomicAdd(&start[F < kEpPrepThreads - 1 ? (int)F : kEpPrepThreads - 1], 1)] = u;
        }
    }
}

// K2a: one THREAD per hop block (frame_step samples): the lane streams its own hop with 16-byte loads and keeps the
// four running integers in registers, so there is no cross-lane reduction and a warp retires 32 hops per pass
// (the first version spent one warp and a five-step shuffle reduction on every hop).  Utterance starts are only
// 2-byte aligned: the aligned middle of the hop goes through uint4 loads, the few samples either side through
// scalar loads.  Samples past the end of the utterance are zeros (sigproc.py:84-87).
// (Round 2 experiments, both reverted: four lanes per hop 0.149 ms and a PAIR of lanes per hop 0.137 ms against 0.111 ms for the lane
// per hop below, all bit-exact.  Sharing a hop between lanes halves / quarters the 128-byte lines a load instruction touches, but
// every extra lane repeats the owner search and the hop geometry -- about 150 instructions against 900 for the hop's samples -- and
// the kernel is bound by instruction issue (45 per 16-byte vector: unpack, |x|, the products' sign bits), not by the line rate.)
struct HopAcc {
    int A, Z, A2, Z2;   // sum |x|, sign changes between neighbours inside the hop; the same over the first `rem` samples
    int prev; int i;    // previous sample, index of the next sample inside the hop
};
__device__ __forceinline__ void hop_push(HopAcc& h, int v, int rem) {
    const int a = v < 0 ? -v : v;
    const int zc = (h.prev * v) < 0 ? 1 : 0;        // |x| <= 32768: the product fits
    h.A += a;
    if (h.i > 0) h.Z += zc;                           // pair (i-1, i)
    if (h.i < rem) { h.A2 += a; if (h.i > 0) h.Z2 += zc; }
    h.prev = v; ++h.i;
}
// eight samples of an aligned vector, none masked, rem == 0: the fast path
__device__ __forceinline__ void hop_push8(HopAcc& h, uint4 w) {
    int v[8];
    v[0] = (int)(short)(w.x & 0xffffu); v[1] = (int)w.x >> 16; v[2] = (int)(short)(w.y & 0xffffu); v[3] = (int)w.y >> 16;
    v[4] = (int)(short)(w.z & 0xffffu); v[5] = (int)w.z >> 16; v[6] = (int)(short)(w.w & 0xffffu); v[7] = (int)w.w >> 16;
    int a = 0, z = ((h.prev * v[0]) >> 31) & (h.i > 0 ? 1 : 0);
#pragma unroll
    for (int k = 0; k < 8; ++k) a += v[k] < 0 ? -v[k] : v[k];
#pragma unroll
    for (int k = 0; k < 7; ++k) z += (unsigned)(v[k] * v[k + 1]) >> 31;
    h.A += a; h.Z += z; h.prev = v[7]; h.i += 8;
}
__global__ void __launch_bounds__(128) ep_block_kernel(EpParams p) {
    const int64_t g = (int64_t)blockIdx.x * 128 + threadIdx.x;
    if (g >= p.block_off[p.n_utt] || g >= p.max_blocks) return;
    const int u = find_owner(p.block_off, p.n_utt, g);
    const int64_t b = g - p.block_off[u];
    const int64_t base = p.offsets[u];
    const int64_t S = p.offsets[u + 1] - base;
    const int64_t s0 = b * p.frame_step;                 // first sample of the hop inside the utterance
    const int16_t* x = p.pcm + base;
    const int step = p.frame_step, rem = p.rem;
    HopAcc h{0, 0, 0, 0, 0, 0};
    int C = 0;
    if (s0 < S) {
        const int64_t n_in = S - s0 < step ? S - s0 : step;          // samples of the hop that exist
        // head: up to the next 16-byte boundary of the packed buffer
        const int64_t addr0 = base + s0;                              // sample index in the packed buffer
        int head = (int)((8 - (addr0 & 7)) & 7);
        if (head > n_in) head = (int)n_in;
        int i = 0;
        for (; i < head; ++i) hop_push(h, (int)x[s0 + i], rem);
        if (rem == 0) {
            const uint4* xv = reinterpret_cast<const uint4*>(p.pcm + addr0 + head);
            const int nvec = (int)((n_in - head) >> 3);
            for (int k = 0; k < nvec; ++k) hop_push8(h, __ldg(xv + k));
            i += 8 * nvec;
        }
        for (; i < n_in; ++i) hop_push(h, (int)x[s0 + i], rem);
        // pair across the boundary to the next hop (the next sample may be past the end: zero)
        if (n_in == step) { const int w = (s0 + step < S) ? (int)x[s0 + step] : 0; C = (h.prev * w) < 0 ? 1 : 0; }
    }
    int32_t* o = p.blk + g * 6;
    o[0] = h.A; o[1] = h.Z; o[2] = C; o[3] = h.A2; o[4] = h.Z2; o[5] = 0;
}

// K2b: one thread per frame
__global__ void __launch_bounds__(256) ep_frame_kernel(EpParams p) {
    const int64_t g = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (g >= p.frame_off[p.n_utt] || g >= p.max_frames) return;
    const int u = find_owner(p.frame_off, p.n_utt, g);
    const int64_t f = g - p.frame_off[u];
    const int32_t* b = p.blk + (p.block_off[u] + f) * 6;
    int A = 0, Z = 0;
    for (int j = 0; j < p.q; ++j) { A += b[6 * j]; Z += b[6 * j + 1]; if (j + 1 < p.q) Z += b[6 * j + 2]; }
    if (p.rem > 0) {
        if (p.q > 0) Z += b[6 * (p.q - 1) + 2];
        A += b[6 * p.q + 3]; Z += b[6 * p.q + 4];
    }
    p.asum[g] = A; p.zcr[g] = Z;
}

// K3: one warp per utterance.  The rule is a sequential state machine over the utterance's frame statistics; the
// warp first stages them in shared memory with coalesced loads (a thread walking global memory on its own pays a full
// DRAM latency per frame), then lane 0 replays the rule.  Utterances longer than kEpStageFrames run from global memory.
constexpr int kEpStageFrames = 1024;
constexpr int kEpDecideWarps = 2;
// amp[i] = sum|x| / frame_len as the reference's float64 mean, computed once per frame by the whole warp: the rule
// compares every frame against its thresholds several times and a float64 division per comparison on one lane was the
// kernel's critical path
template <class Amp>
__device__ __forceinline__ void ep_stage(Amp amp, const int32_t* zcr, int F, double* s_amp, int32_t* s_zcr, int lane) {
    for (int i = lane; i < F; i += 32) { s_amp[i] = amp(i); s_zcr[i] = zcr[i]; }
    __syncwarp();
}
// ---- warp-parallel form of basic_endpoint_detection's decision (endpoint.py:34-66, 133-179, 201-220).
// The thresholds are the reference's float64 expressions evaluated in numpy's order; everything that is order-free runs
// across the lanes: the amplitude maximum (warp max), the sort of the <= 32 silence samples (rank sort), and the
// comparisons of every frame against the thresholds (ballots -> bit masks in shared memory).  The state machine then
// walks bit masks with find-first-set jumps instead of touching every frame.  All lanes execute it redundantly on the same
// shared data (warp-uniform control flow, no broadcasts).
constexpr int kEpMaskWords = kEpStageFrames / 32;
struct EpWarpSmem {
    double amp[kEpStageFrames];
    int32_t zcr[kEpStageFrames];
    double sil[64], sq[64];
    unsigned ge[kEpMaskWords], gt[kEpMaskWords], lo[kEpMaskWords], zt[kEpMaskWords];
};
// smallest index >= i whose bit equals `one` (bits at and beyond F read as "not found"), or F
__device__ __forceinline__ int mask_next(const unsigned* m, int i, int F, bool one) {
    while (i < F) {
        unsigned w = one ? m[i >> 5] : ~m[i >> 5];
        w &= 0xffffffffu << (i & 31);
        if (w) { const int r = (i & ~31) + __ffs((int)w) - 1; return r < F ? r : F; }
        i = (i & ~31) + 32;
    }
    return F;
}
// largest index <= i whose bit is zero, or -1
__device__ __forceinline__ int mask_prev_zero(const unsigned* m, int i) {
    while (i >= 0) {
        unsigned w = ~m[i >> 5];
        w &= 0xffffffffu >> (31 - (i & 31));
        if (w) return (i & ~31) + 31 - __clz((int)w);
        i = (i & ~31) - 1;
    }
    return -1;
}
__device__ __forceinline__ double warp_max_f64(double v) {
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        const double o = __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(v), m), __shfl_xor_sync(0xffffffffu, __double2loint(v), m));
        v = o > v ? o : v;
    }
    return v;
}
// np.mean / np.std of a[0..n) (n <= 64) held in shared memory; sq is shared scratch.  Same operation order as np_mean_std.
__device__ __forceinline__ void warp_mean_std(const double* a, int n, double* sq, int lane, double* mean, double* std) {
    if (n <= 0) { *mean = NAN; *std = NAN; return; }
    const double m = np_pairwise_sum(a, n) / (double)n;
    __syncwarp();
    for (int i = lane; i < n; i += 32) { const double d = a[i] - m; sq[i] = d * d; }
    __syncwarp();
    *mean = m;
    *std = sqrt(np_pairwise_sum(sq, n) / (double)n);
}
// amplitude_rule's scan (endpoint.py:156-179) over the masks ge: amp >= M_H, gt: amp > M_H, lo: amp > M_L
__device__ __forceinline__ void amp_scan_masks(const EpWarpSmem& s, int F, double T_H, int* left, int* right) {
    int first = -1, last = -1, i = 0;
    while (i < F) {
        i = mask_next(s.ge, i, F, true);
        if (i >= F) break;
        int j = i, k = mask_next(s.gt, i, F, false);
        if ((double)(k - j) < T_H) {
            i = k;
        } else {
            if (j > 0) { const int z = mask_prev_zero(s.lo, j); j = z > 0 ? z : 0; }   // while j > 0 and amp[j] > M_L: j -= 1
            k = mask_next(s.lo, k, F, false);                                           // while k < F and amp[k] > M_L: k += 1
            if (first < 0) first = j;
            last = k;
            i = k;
        }
        ++i;
    }
    if (first < 0) { *left = 0; *right = F; } else { *left = first; *right = last; }
}
__device__ __forceinline__ void ep_decide_warp(EpWarpSmem& s, int F, const EpRule& r, int lane, int32_t* out_lr) {
    const int nwords = (F + 31) >> 5;
    // ---- silence model: sorted(amp[:nl] + amp[-nr:])[:-2] (endpoint.py:151-153), n <= 32 here
    const int nl = (int)(r.l_sil / r.cfg_step), nr = (int)(r.r_sil / r.cfg_step);
    const int n_l = nl < F ? nl : F, r0 = (nr > 0 && F - nr > 0) ? F - nr : 0;
    const int n = n_l + (F - r0);
    const double v = lane < n ? s.amp[lane < n_l ? lane : r0 + lane - n_l] : 0.0;
    if (lane < n) s.sq[lane] = v;
    __syncwarp();
    int rank = 0;
    for (int t = 0; t < n; ++t) { const double o = s.sq[t]; rank += (o < v || (o == v && t < lane)) ? 1 : 0; }
    __syncwarp();
    if (lane < n) s.sil[rank] = v;
    double mx = -1.0e300;
    for (int i = lane; i < F; i += 32) { const double a = s.amp[i]; mx = a > mx ? a : mx; }
    const double amax = warp_max_f64(mx);
    __syncwarp();
    double s_mean, s_sigma;
    warp_mean_std(s.sil, n - 2 > 0 ? n - 2 : 0, s.sq, lane, &s_mean, &s_sigma);
    const double T_H = r.th / r.cfg_frame;
    const double M_L = s_mean + r.sigma * s_sigma;
    int left = 0, right = F;
    for (int pass = 0; pass < 2; ++pass) {
        const double a_hi = amax * (pass == 0 ? r.mh1 : r.mh2);
        const double M_H = (M_L > a_hi) ? M_L : a_hi;
        __syncwarp();
        for (int c = 0; c < nwords; ++c) {
            const int i = 32 * c + lane;
            const double a = i < F ? s.amp[i] : 0.0;
            const unsigned ge = __ballot_sync(0xffffffffu, i < F && a >= M_H), gt = __ballot_sync(0xffffffffu, i < F && a > M_H);
            const unsigned lo = __ballot_sync(0xffffffffu, i < F && a > M_L);
            if (lane == 0) { s.ge[c] = ge; s.gt[c] = gt; s.lo[c] = lo; }
        }
        __syncwarp();
        amp_scan_masks(s, F, T_H, &left, &right);
        if (right - left >= r.min_span) break;
    }
    // ---- zcr_rule (endpoint.py:201-220) with l_sil = 0: threshold from the last nr frames
    const int zr = (int)(r.zcr_r_sil / r.cfg_step);
    const int z0 = (zr > 0 && F - zr > 0) ? F - zr : 0;
    const int zn = F - z0;   // <= 32 here
    __syncwarp();
    if (lane < zn) s.sil[lane] = (double)s.zcr[z0 + lane];
    __syncwarp();
    double mu, sg;
    warp_mean_std(s.sil, zn, s.sq, lane, &mu, &sg);
    const double thres = mu + 3 * sg;
    for (int c = 0; c < nwords; ++c) {
        const int i = 32 * c + lane;
        const unsigned zt = __ballot_sync(0xffffffffu, i < F && (double)s.zcr[i < F ? i : 0] > thres);
        if (lane == 0) s.zt[c] = zt;
    }
    __syncwarp();
    // while j > 0 and left - j <= max_shift and zcr[j] > thres: j -= 1   (left - j <= max_shift <=> j >= left - floor(max_shift))
    const double max_shift = r.zcr_max_shift / r.cfg_frame;
    const int ms = (int)floor(max_shift);
    int j = left, k = right;
    if (j > 0 && j < F) {
        int stop = mask_prev_zero(s.zt, j);
        if (stop < left - ms - 1) stop = left - ms - 1;
        j = stop > 0 ? stop : 0;
    }   // (left < F always: it is a frame the scan stood on, or 0)
    if (k < F) {
        int stop = mask_next(s.zt, k, F, false);
        if (stop > right + ms + 1) stop = right + ms + 1;
        k = stop < F ? stop : F;
    }
    int l2 = j, r2 = k;
    if (r2 - l2 < r.min_span) { l2 = 0; r2 = F; }
    if (lane == 0) {
        out_lr[0] = (int32_t)((double)l2 * r.cfg_step * (double)r.rate);
        out_lr[1] = (int32_t)((double)r2 * r.cfg_step * (double)r.rate);
    }
}

// the utterance's amplitudes from the frame starting at f0: int16 path sum|x| / frame_len (AmpFromSum), float path K2f's float64
// values (AmpFromF64)
template <class Amp> __device__ __forceinline__ Amp ep_amp(const EpParams& p, int64_t f0);
template <> __device__ __forceinline__ AmpFromSum ep_amp<AmpFromSum>(const EpParams& p, int64_t f0) { return AmpFromSum{p.asum + f0, (double)p.frame_len}; }
template <> __device__ __forceinline__ AmpFromF64 ep_amp<AmpFromF64>(const EpParams& p, int64_t f0) { return AmpFromF64{p.amp + f0}; }

template <class Amp>
__global__ void __launch_bounds__(32 * kEpDecideWarps) ep_decide_kernel(EpParams p) {
    __shared__ EpWarpSmem s_all[kEpDecideWarps];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int u = blockIdx.x * kEpDecideWarps + w;
    if (u >= p.n_utt) return;
    EpWarpSmem& s = s_all[w];
    const int64_t f0 = p.frame_off[u];
    const int F = (int)(p.frame_off[u + 1] - f0);
    const EpRule& r = p.rule;
    const int nl = (int)(r.l_sil / r.cfg_step), nr = (int)(r.r_sil / r.cfg_step), zr = (int)(r.zcr_r_sil / r.cfg_step);
    if (F <= kEpStageFrames && nl >= 0 && nr >= 1 && nl + nr <= 32 && zr >= 1 && zr <= 32 && r.zcr_max_shift >= 0.0 && r.cfg_frame > 0.0) {
        ep_stage(ep_amp<Amp>(p, f0), p.zcr + f0, F, s.amp, s.zcr, lane);
        ep_decide_warp(s, F, r, lane, p.lr + 2 * u);
    } else if (lane == 0) {
        endpoint_decide_amp(ep_amp<Amp>(p, f0), p.zcr + f0, F, p.rule, p.lr + 2 * u);
    }
}

// K2f on the device
__global__ void __launch_bounds__(kEpF32Threads) ep_stats_f32_kernel(const EpF32Params p) {
    extern __shared__ __align__(16) unsigned char ep_fsm[];
    ep_f32_stats_cta(p, ep_fsm);
}

// K3r gate (acr_rule, endpoint.py:142-144), one warp per frame.  The frame is staged in shared memory as float32 (int16
// samples are exact) with a zero tail.  A lane owns chunks of kGateChunk CONSECUTIVE lags: for a block of eight sample positions
// it loads eight shared values x[i..i+7] (the same for all lanes) and slides a register window over x[i+n..], so every
// shared-memory load feeds kGateChunk fused multiply-adds.  Chunk c goes to lane c mod 32.
//   * screening pass in float32: the lag sums carry a relative error of at most k 2^-24 sum|x_i x_{i+n}| <= k 2^-24 s0 (k terms,
//     Cauchy-Schwarz), i.e. at most delta = 1.5 len 2^-24 len / (len - n_max) on the ratio the rule thresholds at 0.55;
//   * only when the float32 ratio lies within delta of 0.55 the sums are recomputed exactly (float64: products of int16
//     samples and their sums are exact, as in the reference's float64), so the decision is the reference's bit for bit.
constexpr int kEpGateMaxLen = 1536;
constexpr int kGateChunk = 9;
constexpr int kGatePad = 48;        // zero tail: the probe reads up to 38 samples past the frame, the chunked loops 15
// max over the lags n0 .. n0 + nl - 1 of acr(n) = S_n / (len - n), this lane's share (reduce with warp_max_f64).  sx is 16-byte
// aligned: the eight x[i..i+7] every lane needs come from two broadcast 16-byte loads.
// (A split that pairs chunk c with chunk 31 - c on two lanes, so that every lane walks the same number of positions, was
// measured slower -- 3.37 against 2.99 ms: the lanes then read x[i..] at different i, all multiples of eight apart, and the
// loads that were broadcasts turn into 4-way bank conflicts.)
template <typename T>
__device__ __forceinline__ T gate_best(const float* sx, int len, int n0, int nl, int lane, int& best_n) {
    T best = (T)-3.0e38f;
    best_n = n0;
    for (int c = lane; c * kGateChunk < nl; c += 32) {
        const int nb = n0 + c * kGateChunk;              // first lag of the chunk: it has the most terms
        T acc[kGateChunk], w[kGateChunk + 7];
#pragma unroll
        for (int m = 0; m < kGateChunk; ++m) acc[m] = (T)0;
#pragma unroll
        for (int m = 0; m < kGateChunk - 1; ++m) w[m] = (T)sx[nb + m];
        for (int i = 0; i < len - nb; i += 8) {
            // window w[u + m] = x[i + u + nb + m]; terms past the frame multiply the zero tail
#pragma unroll
            for (int u = 0; u < 8; ++u) w[kGateChunk - 1 + u] = (T)sx[i + nb + kGateChunk - 1 + u];
            const float4 a0 = *reinterpret_cast<const float4*>(sx + i), a1 = *reinterpret_cast<const float4*>(sx + i + 4);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const T a = (T)av[u];
#pragma unroll
                for (int m = 0; m < kGateChunk; ++m) acc[m] = fma(a, w[u + m], acc[m]);
            }
#pragma unroll
            for (int m = 0; m < kGateChunk - 1; ++m) w[m] = w[m + 8];
        }
#pragma unroll
        for (int m = 0; m < kGateChunk; ++m) {
            const int n = nb + m;
            if (n < n0 + nl) { const T a = acc[m] / (T)(len - n); if (a > best) { best = a; best_n = n; } }
        }
    }
    return best;
}
// the lane whose value equals the warp maximum hands its lag to everybody (lowest such lane)
__device__ __forceinline__ int warp_arg_of_max(double v, double vmax, int n, int lane) {
    const unsigned m = __ballot_sync(0xffffffffu, v == vmax);
    return __shfl_sync(0xffffffffu, n, m ? __ffs((int)m) - 1 : 0);
}
// The probe and the float32 screening of a staged frame (exact staged values, a0 = acr(frame, 0) of them): 1 / 0 the gate is
// settled, -1 probe_only and not settled, 2 the ratio lies within delta of 0.55 and the exact sums must decide.
__device__ __forceinline__ int gate_screen(const float* sx, int len, int n0, int nl, double a0, int lane, int& pred, bool probe_only) {
    const double delta = 1.5 * (double)len * 5.9604644775390625e-08 * (double)len / (double)(len - (n0 + nl - 1));
    int bn;
    if (delta < 0.01) {
        if (pred >= 0 && nl >= 32) {
            int p0 = pred - 16;
            p0 = p0 < n0 ? n0 : (p0 > n0 + nl - 32 ? n0 + nl - 32 : p0);
            const int n = p0 + lane;
            float acc[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) acc[u] = 0.f;
            for (int i = 0; i < len - p0; i += 8) {      // terms past the frame (i + n >= len) multiply the zero tail
                const float4 a0v = *reinterpret_cast<const float4*>(sx + i), a1v = *reinterpret_cast<const float4*>(sx + i + 4);
                const float av[8] = {a0v.x, a0v.y, a0v.z, a0v.w, a1v.x, a1v.y, a1v.z, a1v.w};
#pragma unroll
                for (int u = 0; u < 8; ++u) acc[u] = fmaf(av[u], sx[i + n + u], acc[u]);
            }
            const float sn = ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
            const double r = (double)(sn / (float)(len - n));
            const double rmax = warp_max_f64(r);
            if (rmax / a0 > 0.55 + delta) { pred = warp_arg_of_max(r, rmax, n, lane); return 1; }
        }
        if (probe_only) return -1;
        const double bf = (double)gate_best<float>(sx, len, n0, nl, lane, bn);
        const double bmax = warp_max_f64(bf);
        const double ratio = bmax / a0;
        if (ratio > 0.55 + delta) { pred = warp_arg_of_max(bf, bmax, bn, lane); return 1; }
        if (ratio < 0.55 - delta) return 0;
    } else if (probe_only) return -1;
    return 2;
}
// The gate of the frame starting at sample b of the utterance x[0..S); warp-uniform result.  `pred` (in): a lag at which the
// neighbouring frame's autocorrelation peaked, or -1; (out) this frame's peak lag when the gate holds.
// With a prediction the warp first PROBES the 32 lags around it, one lag per lane: the rule only asks whether SOME lag exceeds
// 0.55 acr(0), most evaluated frames are voiced (a walk is a run of true gates ended by one false one) and the pitch moves
// slowly, so the probe usually settles the frame for a ninth of the multiply-adds of the full evaluation.  A probe that does not
// clear 0.55 + delta proves nothing and the full evaluation follows.
// probe_only (the speculated frames of a window): 1 = the gate holds, -1 = not settled (the full evaluation is left to the window
// in which the walk actually asks for the frame: speculated frames past the end of a walk are mostly unvoiced)
__device__ int gate_frame_warp(const int16_t* x, long long S, long long b, int len, int n0, int n1, float* sx, int lane, int& pred, bool probe_only) {
    __syncwarp();
    // stage the frame as float32 (exact for int16; mantissa splicing instead of the slow I2F) with a zero tail, summing x^2 on the way;
    // sample pairs through 32-bit loads where the frame starts on a 4-byte boundary
    long long s0i = 0;
    const int nv = (int)(S - b < (long long)len ? (S - b > 0 ? S - b : 0) : (long long)len);      // samples of the frame that exist
    auto cvt = [](int v) { return __uint_as_float(0x4B000000u | (((unsigned)v & 0xffffu) ^ 0x8000u)) - 8421376.0f; };
    if ((reinterpret_cast<uintptr_t>(x + b) & 3) == 0) {
        const int* xw = reinterpret_cast<const int*>(x + b);
        for (int i2 = lane; 2 * i2 < len + kGatePad; i2 += 32) {
            const int i = 2 * i2;
            int lo = 0, hi = 0;
            if (i + 1 < nv) { const int w = __ldg(xw + i2); lo = (int)(short)(w & 0xffff); hi = w >> 16; }
            else if (i < nv) lo = (int)x[b + i];
            *reinterpret_cast<float2*>(sx + i) = make_float2(cvt(lo), cvt(hi));
            s0i += (long long)(lo * lo) + (long long)(hi * hi);                   // each < 2^30: the 32-bit products are exact
        }
    } else {
        for (int i = lane; i < len + kGatePad; i += 32) {
            const int v = i < nv ? (int)x[b + i] : 0;
            sx[i] = cvt(v);
            s0i += (long long)(v * v);
        }
    }
    __syncwarp();
    const int nl = (n1 < len ? n1 : len) - n0;           // lags n0 .. n0 + nl - 1
    if (nl <= 0) return 0;
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) s0i += __shfl_xor_sync(0xffffffffu, s0i, m);
    if (s0i == 0) return 0;                              // 0 / 0 = NaN compares false, as in the reference
    const double a0 = (double)s0i / (double)len;
    const int g = gate_screen(sx, len, n0, nl, a0, lane, pred, probe_only);
    if (g != 2) return g;
    int bn;
    const double bd = gate_best<double>(sx, len, n0, nl, lane, bn);
    const double dmax = warp_max_f64(bd);
    if (dmax / a0 > 0.55) { pred = warp_arg_of_max(bd, dmax, bn, lane); return 1; }   // acr_gate_decide on exact sums
    return 0;
}

// The same gate on float32 samples (x: the utterance, 4-byte aligned).  framesig's frame is float64 and every float32 sample
// enters it exactly, so acr(frame, n) is NumPy's pairwise float64 sum of exact products (acr_lag):
//   * the frame is staged with its zero tail, through 16-byte loads when x + b is 16-byte aligned; a NaN or +-inf sample
//     makes the gate false (acr_gate_frame), an all-zero frame too;
//   * a0 = acr(frame, 0) exactly (acr_lag on the staged, unscaled values);
//   * the staged frame is then scaled by 2^k so that max|x| lies in [1, 2).  The ratio is invariant under power-of-two scaling
//     and the screening's float32 sums neither overflow (above max|x| ~ 1.8e19 they would) nor underflow (quiet input near 1e-20
//     would flush to zero and void the bound).  The probe and the screening then run unchanged with the same delta: its
//     derivation only needs the staged values exact.  Scaling down may round samples below 2^-126 max|x| to subnormals, and the
//     float32 sums may run through subnormals: at most about k 2^-149 on lag sums with a0 >= 1 / len, negligible against delta;
//   * the exact fallback is acr_lag per lag (one lane per lag, unscaled samples from x), a warp max and the 0.55 test.  The
//     chunked float64 FMA order of gate_best<double> is exact for int16 samples only.
__device__ int gate_frame_warp(const float* x, long long S, long long b, int len, int n0, int n1, float* sx, int lane, int& pred, bool probe_only) {
    __syncwarp();
    const int nv = (int)(S - b < (long long)len ? (S - b > 0 ? S - b : 0) : (long long)len);      // samples of the frame that exist
    const float* xb = x + b;
    const int nvec = (len + kGatePad + 3) >> 2;          // the staging area holds kEpGateMaxLen + kGatePad floats, a multiple of 4
    float mx = 0.f;
    bool bad = false;
    if ((reinterpret_cast<uintptr_t>(xb) & 15) == 0) {
        for (int v = lane; v < nvec; v += 32) {
            const int i = 4 * v;
            float4 w;
            if (i + 3 < nv) {
                w = __ldg(reinterpret_cast<const float4*>(xb) + v);
            } else {
                w.x = i < nv ? xb[i] : 0.f; w.y = i + 1 < nv ? xb[i + 1] : 0.f;
                w.z = i + 2 < nv ? xb[i + 2] : 0.f; w.w = i + 3 < nv ? xb[i + 3] : 0.f;
            }
            *reinterpret_cast<float4*>(sx + i) = w;
            const float m = fmaxf(fmaxf(fabsf(w.x), fabsf(w.y)), fmaxf(fabsf(w.z), fabsf(w.w)));
            bad |= !(isfinite(w.x) && isfinite(w.y) && isfinite(w.z) && isfinite(w.w));
            mx = fmaxf(mx, m);
        }
    } else {
        for (int i = lane; i < 4 * nvec; i += 32) {
            const float v = i < nv ? xb[i] : 0.f;
            sx[i] = v;
            bad |= !isfinite(v);
            mx = fmaxf(mx, fabsf(v));
        }
    }
    const int nl = (n1 < len ? n1 : len) - n0;           // lags n0 .. n0 + nl - 1
    if (nl <= 0 || __any_sync(0xffffffffu, bad)) return 0;
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, m));
    if (mx == 0.f) return 0;                             // 0 / 0 = NaN compares false, as in the reference
    __syncwarp();
    const double a0 = acr_lag(sx, nv, len, 0);
    int e;
    frexpf(mx, &e);
    const int k = 1 - e;                                 // mx 2^k in [1, 2)
    __syncwarp();
    if ((reinterpret_cast<uintptr_t>(xb) & 15) == 0) {
        for (int i = 4 * lane; i < 4 * nvec; i += 128) {
            float4 w = *reinterpret_cast<float4*>(sx + i);
            w.x = ldexpf(w.x, k); w.y = ldexpf(w.y, k); w.z = ldexpf(w.z, k); w.w = ldexpf(w.w, k);
            *reinterpret_cast<float4*>(sx + i) = w;
        }
    } else {
        for (int i = lane; i < 4 * nvec; i += 32) sx[i] = ldexpf(sx[i], k);
    }
    __syncwarp();
    const int g = gate_screen(sx, len, n0, nl, ldexp(a0, 2 * k), lane, pred, probe_only);   // a0 of the scaled frame, exact
    if (g != 2) return g;
    double bd = -INFINITY;
    int bn = n0;
    for (int n = n0 + lane; n < n0 + nl; n += 32) {
        const double a = acr_lag(xb, nv, len, n);
        if (a > bd) { bd = a; bn = n; }
    }
    const double dmax = warp_max_f64(bd);
    if (dmax / a0 > 0.55) { pred = warp_arg_of_max(bd, dmax, bn, lane); return 1; }
    return 0;
}

// CTA-cooperative gate of K3r: every thread of the CTA replays the rule in lock step on identical data.  A request for a frame
// that is not in the current window makes the CTA's warps evaluate that frame and the next kEpRobustWarps - 1 frames of the
// walk (those the walk can reach: amp > M_L all the way) at once, one frame per warp; the walk's following requests hit the window.
constexpr int kEpRobustWarps = 4;     // (8 warps: 1.56 -> 1.80 ms with probe-only speculation, 4 warps: 1.40 -> 1.33 ms per 4096 utterances: fewer idle warps at the window barriers)
// Warp 0 alone replays the rule (the first version had all 256 threads do it in lock step: the silence sort, the thresholds and the
// frame walk were a third of the kernel's issue slots); the other warps serve its gate requests.  Requests and results travel
// through shared memory between two named barriers that every thread of the CTA passes once per window.
struct GateRequest { int j, dir, pred, done; double m_l; double pad; };      // 32 bytes: the staging areas behind it stay 16-byte aligned
__device__ __forceinline__ void robust_bar(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(32 * kEpRobustWarps) : "memory"); }
// one window: warp w evaluates frame j + dir * w when the walk can reach it
template <class T, class Amp>
__device__ __forceinline__ int gate_window_warp(const GateRequest& q, const T* x, long long S, int step, int len, int n0, int n1, int F,
                                                Amp amp, float* sx, int w, int lane) {
    const int fj = q.j + q.dir * w;
    bool want = q.dir < 0 ? fj >= 1 : fj < F;
    for (int t = 1; t <= w && want; ++t) want = amp(q.j + q.dir * t) > q.m_l;
    if (q.pred < 0 && w > 0) want = false;     // no peak lag yet (the utterance's first gate): one full evaluation, not eight
    int res = 0, lag = q.pred;
    if (want) {
        const int g = gate_frame_warp(x, S, (long long)fj * step, len, n0, n1, sx + w * (kEpGateMaxLen + kGatePad), lane, lag, w > 0);
        if (g >= 0) res = 2 | g;
    }
    return res | ((lag < 0 ? 0 : lag) << 2);
}
template <class T, class Amp>
struct GateCta {           // lives in warp 0
    const T* x; long long S; int step, len, n0, n1, F;
    Amp amp; float* sx; int* s_res; GateRequest* req;
    int dir; double m_l; int win_base, win_dir, win_known, win_val;
    int pred;                              // the peak lag of the last frame whose gate held (the probe's centre), -1: none yet
    __device__ void hint(int d, double ml) { dir = d; m_l = ml; }
    __device__ bool operator()(int j) {
        const int wi = (j - win_base) * win_dir;
        if (wi >= 0 && wi < kEpRobustWarps && ((win_known >> wi) & 1)) return (win_val >> wi) & 1;
        const int lane = threadIdx.x & 31;
        if (lane == 0) { req->j = j; req->dir = dir; req->pred = pred; req->done = 0; req->m_l = m_l; }
        robust_bar(1);                   // the request is posted (and the previous window's results have been read)
        const int res = gate_window_warp(*req, x, S, step, len, n0, n1, F, amp, sx, 0, lane);
        if (lane == 0) s_res[0] = res;
        robust_bar(2);                   // the results are in
        win_base = j; win_dir = dir; win_known = 0; win_val = 0;
#pragma unroll
        for (int t = 0; t < kEpRobustWarps; ++t) {
            const int r = s_res[t];
            win_known |= ((r >> 1) & 1) << t; win_val |= (r & 1) << t;
            if ((r & 3) == 3) pred = r >> 2;                     // the furthest frame of the window whose gate held
        }
        return win_val & 1;
    }
};
template <class T, class Amp>
__device__ __forceinline__ void robust_cta(const EpParams& p, Amp amp, const int32_t* zcr, int F, const T* x, long long S, float* s_x, int* s_res,
                                           GateRequest* req, int u) {
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = p.rule.rate / 500, n1 = p.rule.rate / 50;
    if (w == 0) {
        GateCta<T, Amp> gate{x, S, p.frame_step, p.frame_len, n0, n1, F, amp, s_x, s_res, req, -1, 0.0, 0, 1, 0, 0, -1};
        int32_t lr[2];
        endpoint_decide_robust(amp, zcr, F, p.rule, gate, lr);
        if (lane == 0) { req->done = 1; p.lr[2 * u] = lr[0]; p.lr[2 * u + 1] = lr[1]; }
        robust_bar(1);                   // releases the serving warps
    } else {
        for (;;) {
            robust_bar(1);
            if (req->done) break;
            const int res = gate_window_warp(*req, x, S, p.frame_step, p.frame_len, n0, n1, F, amp, s_x, w, lane);
            if (lane == 0) s_res[w] = res;
            robust_bar(2);
        }
    }
}

// what K3r reads for each sample type: the samples its gate stages (int16: p.pcm, float32: p.pcm_f32) and the frame amplitudes
// (int16: K2b's sums / frame_len, float32: K2f's float64 values), one frame g at a time or as the source Amp of an utterance
template <class T> struct EpSamples;
template <> struct EpSamples<int16_t> {
    using Amp = AmpFromSum;
    static __device__ __forceinline__ const int16_t* pcm(const EpParams& p) { return p.pcm; }
    static __device__ __forceinline__ double amp(const EpParams& p, int64_t g) { return (double)p.asum[g] / (double)p.frame_len; }
};
template <> struct EpSamples<float> {
    using Amp = AmpFromF64;
    static __device__ __forceinline__ const float* pcm(const EpParams& p) { return p.pcm_f32; }
    static __device__ __forceinline__ double amp(const EpParams& p, int64_t g) { return p.amp[g]; }
};
template <class T>
__global__ void __launch_bounds__(32 * kEpRobustWarps, 6) ep_decide_robust_kernel(EpParams p) {
    extern __shared__ __align__(16) unsigned char ep_rsm[];
    double* s_amp = reinterpret_cast<double*>(ep_rsm);                                   // [kEpStageFrames]
    int32_t* s_zcr = reinterpret_cast<int32_t*>(s_amp + kEpStageFrames);                 // [kEpStageFrames]
    int* s_res = s_zcr + kEpStageFrames;                                                 // [kEpRobustWarps]
    static_assert(kEpRobustWarps % 4 == 0, "the window results keep the request and the staging areas 16-byte aligned");
    GateRequest* req = reinterpret_cast<GateRequest*>(s_res + kEpRobustWarps);
    float* s_x = reinterpret_cast<float*>(req + 1);                                      // [kEpRobustWarps][kEpGateMaxLen + kGatePad], 16-byte aligned
    const int u = p.order ? p.order[blockIdx.x] : (int)blockIdx.x;
    const int64_t f0 = p.frame_off[u];
    const int F = (int)(p.frame_off[u + 1] - f0);
    const T* x = EpSamples<T>::pcm(p) + p.offsets[u];
    const long long S = (long long)(p.offsets[u + 1] - p.offsets[u]);
    if (F <= kEpStageFrames) {
        for (int i = threadIdx.x; i < F; i += blockDim.x) { s_amp[i] = EpSamples<T>::amp(p, f0 + i); s_zcr[i] = p.zcr[f0 + i]; }
        __syncthreads();
        robust_cta(p, AmpFromF64{s_amp}, s_zcr, F, x, S, s_x, s_res, req, u);
    } else {
        robust_cta(p, ep_amp<typename EpSamples<T>::Amp>(p, f0), p.zcr + f0, F, x, S, s_x, s_res, req, u);
    }
}
constexpr int kEpRobustSmem = kEpStageFrames * 12 + kEpRobustWarps * 4 + (int)sizeof(GateRequest) + kEpRobustWarps * (kEpGateMaxLen + kGatePad) * 4;

// the gate of every row of a float64 frame matrix (the list-typed amplitude_rule(use_acr=True, frames=...) API): one warp per row
__global__ void acr_gate_rows_kernel(const double* frames, int64_t n_rows, int len, int n0, int n1, int32_t* gate) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= n_rows) return;
    const double* x = frames + r * len;
    double s0 = 0.0, best = -1.0e300;
    for (int i = lane; i < len; i += 32) s0 += x[i] * x[i];
    for (int n = n0 + lane; n < n1 && n < len; n += 32) {
        double sn = 0.0;
        for (int i = 0; i + n < len; ++i) sn += x[i] * x[i + n];
        const double a = sn / (double)(len - n);
        best = a > best ? a : best;
    }
#pragma unroll
    for (int m = 16; m >= 1; m >>= 1) {
        s0 += __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(s0), m), __shfl_xor_sync(0xffffffffu, __double2loint(s0), m));
        const double o = __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(best), m), __shfl_xor_sync(0xffffffffu, __double2loint(best), m));
        best = o > best ? o : best;
    }
    if (lane == 0) gate[r] = (n0 < n1 && n0 < len && best / (s0 / (double)len) > 0.55) ? 1 : 0;
}
#endif  // __CUDACC__

}  // namespace dspfe
