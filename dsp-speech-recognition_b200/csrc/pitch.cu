// C ABI of the pitch path (include/dspfe.h, "pitch" section).  Kernels: pitch_kernel.cuh.
// No CPU fallback: the device entry points launch CUDA kernels or fail; the *_host list helpers at the end are
// the reference's tiny sequential list functions (same C++ code the device kernels run), not a second path.
#include <cmath>
#include <cstring>
#include <vector>

#include "abi_common.h"
#include "dspfe_types.h"
#include "pitch_kernel.cuh"
#include "pitch_tables.h"

using namespace dspfe;

namespace {

constexpr int kPitchPrepThreads = 1024;

// per-utterance ranges, decimated lengths and the frame prefix sums (single CTA, no host round trip)
__global__ void __launch_bounds__(kPitchPrepThreads) pitch_prep_kernel(PitchParams p) {
    __shared__ long long s_fr[kPitchPrepThreads], s_sl[kPitchPrepThreads];
    const int tid = threadIdx.x;
    const int per = (p.n_utt + kPitchPrepThreads - 1) / kPitchPrepThreads;
    const int u0 = min(tid * per, p.n_utt), u1 = min(u0 + per, p.n_utt);
    long long fr = 0, sl = 0;
    for (int u = u0; u < u1; ++u) {
        long long a = p.offsets[u], len = p.offsets[u + 1] - a;
        if (p.trim) {  // Python slice sig[l:r] with l, r >= 0
            long long l = p.trim[2 * u], r = p.trim[2 * u + 1];
            if (l < 0) l = 0; if (r < 0) r = 0;
            if (l > len) l = len; if (r > len) r = len;
            a += l; len = r > l ? r - l : 0;
        }
        p.seg_start[u] = a; p.seg_len[u] = (int)len;
        const long long ld = ds_length(len, p.ds_idx, p.ds_in, p.ds_out);
        p.ds_len[u] = (int)ld;
        const long long nf = num_frames(ld, p.frame_len, p.frame_step);
        fr += nf; sl += (nf + kClipRun - 1) / kClipRun * kClipRun;
    }
    s_fr[tid] = fr; s_sl[tid] = sl;
    __syncthreads();
    for (int d = 1; d < kPitchPrepThreads; d <<= 1) {
        long long f = tid >= d ? s_fr[tid - d] : 0, g = tid >= d ? s_sl[tid - d] : 0;
        __syncthreads();
        s_fr[tid] += f; s_sl[tid] += g;
        __syncthreads();
    }
    long long fo = s_fr[tid] - fr, so = s_sl[tid] - sl;
    for (int u = u0; u < u1; ++u) {
        p.frame_off[u] = fo; p.slot_off[u] = so;
        const long long nf = num_frames(p.ds_len[u], p.frame_len, p.frame_step);
        fo += nf; so += (nf + kClipRun - 1) / kClipRun * kClipRun;
    }
    if (tid == kPitchPrepThreads - 1) { p.frame_off[p.n_utt] = s_fr[tid]; p.slot_off[p.n_utt] = s_sl[tid]; }
    // the utterances by descending frame count (counting sort, bins of one frame, the longest share the last bin): the order in
    // which the CTA-per-utterance kernels take them.  Positions inside a bin depend on the atomics' order; the results do not.
    int* order = const_cast<int*>(p.order);
    if (order) {
        __syncthreads();
        int* bins = reinterpret_cast<int*>(s_fr);          // [kPitchPrepThreads] (the scan arrays are done)
        bins[tid] = 0;
        __syncthreads();
        for (int u = u0; u < u1; ++u) {
            const long long nf = num_frames(p.ds_len[u], p.frame_len, p.frame_step);
            atomicAdd(&bins[nf < kPitchPrepThreads - 1 ? (int)nf : kPitchPrepThreads - 1], 1);
        }
        __syncthreads();
        // start[b] = utterances in the bins above b: inclusive suffix sums, then shift
        int* start = reinterpret_cast<int*>(s_sl);
        start[tid] = bins[tid];
        __syncthreads();
        for (int d = 1; d < kPitchPrepThreads; d <<= 1) {
            const int v = tid + d < kPitchPrepThreads ? start[tid + d] : 0;
            __syncthreads();
            start[tid] += v;
            __syncthreads();
        }
        const int mine = start[tid] - bins[tid];
        __syncthreads();
        start[tid] = mine;
        __syncthreads();
        for (int u = u0; u < u1; ++u) {
            const long long nf = num_frames(p.ds_len[u], p.frame_len, p.frame_step);
            order[atomicAdd(&start[nf < kPitchPrepThreads - 1 ? (int)nf : kPitchPrepThreads - 1], 1)] = u;
        }
    }
}

// K4a-1: gather + exact median + centre clip, a frame pair per warp
// (4 CTAs/SM at 128 registers without spills beat 5 CTAs/SM at 96 with 100-180 bytes of them)
template <bool I16>
__global__ void __launch_bounds__(32 * kPitchWarps, 4) pitch_clip_kernel(const __grid_constant__ PitchParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    int32_t* ds_idx = reinterpret_cast<int32_t*>(smem);
    const int64_t total = p.slot_off[p.n_utt];
    if (kClipRun * (int64_t)blockIdx.x * kPitchWarps >= total) return;   // the grid is sized for the untrimmed batch
    for (int i = threadIdx.x; i < p.ds_out; i += blockDim.x) ds_idx[i] = p.ds_idx[i];
    __syncthreads();
    const int w = threadIdx.x >> 5;
    const int64_t h0 = kClipRun * ((int64_t)blockIdx.x * kPitchWarps + w);
    if (h0 >= total) return;   // whole warp leaves; only warp-level syncs below
    if (p.frame_len <= 320) pitch_clip_run<10, I16>(p, h0, smem + kMaxDsOut * 4 + w * kClipWarpSmemBytes, ds_idx);   // e.g. the 300-sample frames of model.py:92
    else pitch_clip_run<16, I16>(p, h0, smem + kMaxDsOut * 4 + w * kClipWarpSmemBytes, ds_idx);
}

// K4a-2 / K5a-2: the transforms, a frame pair per warp.  At 128 registers (4 CTAs/SM) the chains spilled 130-230 bytes per
// thread; 3 CTAs/SM without spills measured 3 % faster for the autocorrelation chains and 1 % for the cepstrum (the kernels sit
// on the shared-memory pipe, so the fourth CTA bought nothing).
template <int MODE>
__global__ void __launch_bounds__(32 * kPitchWarps, MODE == 1 ? 3 : 4) pitch_frame_kernel(const __grid_constant__ PitchParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tws = reinterpret_cast<float2*>(smem);                       // W512 twiddles + W32 (kTabMod float2)
    constexpr int kPer = MODE == 2 ? 4 : 2;                              // slots per warp: a quad (pitch_acr_quad) or a pair
    const int64_t total = p.slot_off[p.n_utt];
    if (kPer * (int64_t)blockIdx.x * kPitchWarps >= total) return;   // surplus CTAs leave before touching the tables
    for (int i = threadIdx.x; i < kTabMod; i += blockDim.x) tws[i] = p.tab[i];
    __syncthreads();
    const int w = threadIdx.x >> 5;
    const int64_t h0 = kPer * ((int64_t)blockIdx.x * kPitchWarps + w);
    if (h0 >= total) return;   // whole warp leaves; only warp-level syncs below
    int nvalid; int64_t g0;
    slot_unit_from_desc(p, h0, kPer, g0, nvalid);
    if (nvalid == 0) return;   // padding slots at the end of an utterance
    if (MODE == 2) pitch_acr_quad(p, h0, g0, nvalid, smem + kTabMod * 8 + w * kQuadWarpSmemBytes, tws, tws + kTabW32);
    else pitch_fft_pair<(MODE == 2 ? 1 : MODE)>(p, h0, g0, nvalid > 1, smem + kTabMod * 8 + w * kWarpSmemBytes, tws, tws + kTabW32);
}

// K4a-2 for cepstrum frames of 100..511 samples: the N-point DFTs by Bluestein's chirp (12 transforms per pair), a frame pair per
// warp in the slot space of pitch_frame_kernel<0>
__global__ void __launch_bounds__(32 * kPitchWarps, 3) pitch_cep_bluestein_kernel(const __grid_constant__ PitchParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tws = reinterpret_cast<float2*>(smem);                       // W512 twiddles + W32 (kTabMod float2)
    const int64_t total = p.slot_off[p.n_utt];
    if (2 * (int64_t)blockIdx.x * kPitchWarps >= total) return;         // surplus CTAs leave before touching the tables
    for (int i = threadIdx.x; i < kTabMod; i += blockDim.x) tws[i] = p.tab[i];
    __syncthreads();
    const int w = threadIdx.x >> 5;
    const int64_t h0 = 2 * ((int64_t)blockIdx.x * kPitchWarps + w);
    if (h0 >= total) return;   // whole warp leaves; only warp-level syncs below
    int nvalid; int64_t g0;
    slot_unit_from_desc(p, h0, 2, g0, nvalid);
    if (nvalid == 0) return;   // padding slots at the end of an utterance
    pitch_cep_bluestein_pair(p, h0, g0, nvalid > 1, smem + kTabMod * 8 + w * kWarpSmemBytes, tws, tws + kTabW32);
}

__global__ void __launch_bounds__(kTrackThreads) pitch_track_kernel(const __grid_constant__ PitchParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    float* chunk = reinterpret_cast<float*>(smem);
    int* sc = reinterpret_cast<int*>(chunk + (track_chunk(p.row_len) + 1) * p.row_len);
    pitch_track_cta(p, chunk, sc, reinterpret_cast<double*>(sc + track_chunk(p.row_len) * kPeakLags));
}

__global__ void __launch_bounds__(32) pitch_feature_kernel(const __grid_constant__ PitchParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    pitch_feature_warp(p, p.order ? p.order[blockIdx.x] : (int)blockIdx.x, reinterpret_cast<double*>(smem));
}

// dp_max_pitch (pitch.py:208-225) on the device: Viterbi over the columns of g [n_rows, n_cols] with a jump penalty of 5 per
// column, one CTA, thread j owns column j.  Per row every thread maximises dp[k] - 5 |k - j| + g[i][j] over k in float64 with the
// reference's evaluation order and first-maximum tie rule; the back-trace starts, as in the reference, from the predecessor
// chosen for the LAST column of the last row (`step` as the Python loops leave it), not from the best end state.
constexpr int kDpMaxCols = 1024;
__global__ void __launch_bounds__(kDpMaxCols) dp_max_pitch_kernel(const double* g, int n_rows, int n_cols, int32_t* prev, double* path) {
    extern __shared__ __align__(16) unsigned char smem[];
    double* dp = reinterpret_cast<double*>(smem);            // [2][n_cols]
    const int j = threadIdx.x;
    if (j < n_cols) dp[j] = 0.0;                                // dp[0] = zeros (np.zeros, row 0 is never scored)
    __syncthreads();
    for (int i = 1; i < n_rows; ++i) {
        const double* cur = dp + ((i - 1) & 1) * n_cols;
        double* nxt = dp + (i & 1) * n_cols;
        if (j < n_cols) {
            const double gij = g[(size_t)i * n_cols + j];
            double best = 0.0; int arg = -1;
            for (int k = 0; k < n_cols; ++k) {
                const double r = (cur[k] - 5.0 * (double)(k > j ? k - j : j - k)) + gij;
                if (arg < 0 || r > best) { best = r; arg = k; }
            }
            nxt[j] = best; prev[(size_t)i * n_cols + j] = arg;
        }
        __syncthreads();
    }
    if (j == 0) {
        int step = n_rows > 1 ? prev[(size_t)(n_rows - 1) * n_cols + (n_cols - 1)] : 0;
        for (int i = n_rows - 1; i >= 0; --i) {
            path[i] = 10000.0 / (double)step;
            step = i >= 1 ? prev[(size_t)i * n_cols + step] : 0;    // prev[0] is all zeros in the reference
        }
    }
}

// smooth + peak_score on caller-supplied rows (taps of pitch.py:157 / :227): one "utterance" of n_rows frames
__global__ void pitch_fill_off_kernel(int64_t* frame_off, int64_t n_rows) {
    if (threadIdx.x == 0) { frame_off[0] = 0; frame_off[1] = n_rows; }
}

// center_clip(frame, binary) (pitch.py:145; endpoint.py:20) on rows of up to 512 float32 values, one warp per row
__global__ void center_clip_kernel(const float* in, int64_t n_rows, int len, int binary, float* out) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= n_rows) return;
    float x[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) { const int n = lane + 32 * t; x[t] = n < len ? in[r * len + n] : 0.f; }
    const float med = warp_median_nonneg(x, len, lane);
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        const int n = lane + 32 * t;
        if (n >= len) continue;
        float c;
        if (binary) c = x[t] > med ? 1.f : (x[t] < -med ? -1.f : 0.f);
        else c = clip_value(x[t], med);
        out[r * len + n] = c;
    }
}

}  // namespace

struct dspfe_pitch_plan {
    dspfe_pitch_params prm;
    PitchParams base;          // scalars + table pointers; per-call pointers filled in launch
    HostBatch host;            // host-path staging
    DeviceArray<int32_t> d_trim; DeviceArray<double> d_feat;
    DeviceArray<float2> d_tab;
    // workspaces
    DeviceArray<int64_t> seg_start; DeviceArray<int32_t> seg_len, ds_len; DeviceArray<int64_t> frame_off, slot_off;
    DeviceArray<int32_t> order;
    DeviceArray<float2> clip; DeviceArray<int4> run_desc; DeviceArray<float> rows; DeviceArray<double> frame_amp, pitch;
    DeviceArray<int32_t> lag; DeviceArray<double> scratch;
};

namespace {

int ensure(dspfe_pitch_plan* pl, int64_t n_utt, int64_t frames) {
    int rc = pl->seg_start.reserve(n_utt + 1);
    if (!rc) rc = pl->seg_len.reserve(n_utt + 1);
    if (!rc) rc = pl->ds_len.reserve(n_utt + 1);
    if (!rc) rc = pl->frame_off.reserve(n_utt + 1);
    if (!rc) rc = pl->slot_off.reserve(n_utt + 1);
    if (!rc) rc = pl->order.reserve(n_utt + 1);
    if (!rc) rc = pl->rows.reserve(frames * pl->base.row_len);
    if (!rc) rc = pl->frame_amp.reserve(frames);
    if (!rc) rc = pl->pitch.reserve(frames);
    if (!rc) rc = pl->lag.reserve(frames);
    if (!rc) rc = pl->scratch.reserve(3 * frames);
    const int64_t slots = frames + (kClipRun - 1) * n_utt;       // every utterance's frame count rounded up to a run
    if (!rc) rc = pl->clip.reserve(((slots + 1) / 2) * 512);
    if (!rc) rc = pl->run_desc.reserve(slots / kClipRun + 1);
    return rc;
}

int track_smem(int row_len) { return (track_chunk(row_len) + 1) * row_len * (int)sizeof(float) + track_chunk(row_len) * kPeakLags * (int)sizeof(int) + kTrackMaxFrames * 12 + (kTrackThreads / 32) * kTrackListPerWarp * 2 + 8; }

}  // namespace

extern "C" {

void dspfe_pitch_params_default(dspfe_pitch_params* p, int32_t method) {
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->samplerate = 16000; p->dst_rate = 10000; p->frame_len = 512; p->frame_step = 100; p->method = method;
    p->center_clip = 1; p->row_len = 0; p->band_lo = 50.0; p->band_hi = method == 0 ? 1000.0 : 900.0; p->preemph = 0.0;
}

int dspfe_pitch_create(const dspfe_pitch_params* q, dspfe_pitch_plan** plan) {
    if (!q || !plan) return fail(DSPFE_ERR_INVALID_ARG, "null argument");
    *plan = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(DSPFE_ERR_CUDA, "no CUDA device: libdspfe has no CPU fallback");
    dspfe_pitch_plan* pl = new (std::nothrow) dspfe_pitch_plan();
    if (!pl) return fail(DSPFE_ERR_NOMEM, "out of host memory");
    pl->prm = *q;
    PitchParams& b = pl->base;
    std::vector<float2> tab;
    std::string err;
    const int trc = build_pitch_tables(*q, b, tab, err);
    if (trc) { delete pl; return fail(trc, err); }
    if (int rc = pl->d_tab.reserve(kTabCepTotal)) { delete pl; return rc; }
    cudaError_t e = cudaMemcpy(pl->d_tab.get(), tab.data(), kTabCepTotal * sizeof(float2), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pitch_clip_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kClipCtaSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pitch_clip_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kClipCtaSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pitch_frame_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFrameCtaSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pitch_frame_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kFrameCtaSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pitch_frame_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kQuadCtaSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pitch_cep_bluestein_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kFrameCtaSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pitch_track_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, track_smem(kCepLen));
    if (e != cudaSuccess) { delete pl; return fail(DSPFE_ERR_CUDA, cudaGetErrorString(e)); }
    b.tab = pl->d_tab.get();
    *plan = pl;
    return DSPFE_OK;
}

void dspfe_pitch_destroy(dspfe_pitch_plan* pl) {
    if (!pl) return;
    delete pl;
}

int dspfe_pitch_reserve(dspfe_pitch_plan* pl, int64_t max_utt, int64_t max_total_samples) {
    if (!pl || max_utt < 0 || max_total_samples < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    return ensure(pl, max_utt, dspfe_pitch_frames_bound(pl, max_total_samples, max_utt));
}

int32_t dspfe_pitch_row_len(const dspfe_pitch_plan* pl) { return pl ? pl->base.row_len : -1; }

int64_t dspfe_pitch_frames_bound(const dspfe_pitch_plan* pl, int64_t total_samples, int64_t n_utt) {
    if (!pl) return -1;
    // decimated samples <= S*ds_out/ds_in + 2 per utterance; frames <= decimated/step + 1
    return (total_samples / pl->base.ds_in + 1) * pl->base.ds_out / pl->base.frame_step + 3 * n_utt;
}

int64_t dspfe_pitch_num_frames_host(const dspfe_pitch_params* q, int64_t n_samples, int64_t* n_decimated) {
    if (!q) return -1;
    PitchParams b; std::vector<float2> tab; std::string err;
    const int trc = build_pitch_tables(*q, b, tab, err);
    if (trc) { fail(trc, err); return trc; }
    const int64_t ld = ds_length(n_samples, b.ds_idx, b.ds_in, b.ds_out);
    if (n_decimated) *n_decimated = ld;
    return num_frames(ld, b.frame_len, b.frame_step);
}

int64_t dspfe_pitch_num_frames(const dspfe_pitch_plan* pl, int64_t n_samples) {
    if (!pl) return -1;
    return num_frames(ds_length(n_samples, pl->base.ds_idx, pl->base.ds_in, pl->base.ds_out), pl->base.frame_len, pl->base.frame_step);
}

int dspfe_pitch(dspfe_pitch_plan* pl, const void* d_pcm, int32_t sample_dtype, int64_t total_samples, const int64_t* d_offsets,
                const int32_t* d_trim, int32_t n_utt, double* d_pitch, int32_t* d_lag, double* d_feat, float* d_rows,
                int64_t* d_frame_off, int64_t max_frames, void* stream) {
    if (int rc = check_batch(pl && d_offsets && (sample_dtype == 0 || sample_dtype == 1), n_utt, total_samples, d_pcm)) return rc;
    if (n_utt == 0) return DSPFE_OK;
    const int64_t bound = dspfe_pitch_frames_bound(pl, total_samples, n_utt);
    if ((d_pitch || d_lag || d_rows) && max_frames < bound) return fail(DSPFE_ERR_INVALID_ARG, "max_frames is below dspfe_pitch_frames_bound()");
    if (d_feat && pl->base.mode != 0) return fail(DSPFE_ERR_UNSUPPORTED, "pitch_feature is defined on the cepstrum pitch (pitch.py:33)");
    if (d_feat && pl->base.frame_len != kCepLen)
        return fail(DSPFE_ERR_UNSUPPORTED, "pitch_feature is defined on 512-sample cepstrum frames (pitch.py:33 uses the default winlen)");
    int rc = ensure(pl, n_utt, bound);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    PitchParams p = pl->base;
    p.pcm = d_pcm; p.in_f32 = sample_dtype; p.total_samples = total_samples; p.offsets = d_offsets; p.trim = d_trim; p.n_utt = n_utt;
    p.frame_off = d_frame_off ? d_frame_off : pl->frame_off.get(); p.slot_off = pl->slot_off.get(); p.seg_start = pl->seg_start.get();
    p.seg_len = pl->seg_len.get(); p.ds_len = pl->ds_len.get(); p.clip = pl->clip.get(); p.run_desc = pl->run_desc.get();
    p.rows = d_rows ? d_rows : pl->rows.get(); p.rows_out = nullptr; p.score = nullptr; p.frame_amp = pl->frame_amp.get();
    p.pitch = d_pitch ? d_pitch : pl->pitch.get(); p.lag = d_lag ? d_lag : pl->lag.get(); p.feat = d_feat; p.scratch = pl->scratch.get();
    p.max_frames = bound; p.order = pl->order.get();
    pitch_prep_kernel<<<1, kPitchPrepThreads, 0, st>>>(p);
    LAUNCH_CHECK("pitch_prep_kernel", st);
    const int64_t slots = bound + (int64_t)(kClipRun - 1) * n_utt;
    const unsigned cgrid = (unsigned)((slots + kClipRun * kPitchWarps - 1) / (kClipRun * kPitchWarps));
    if (clip_i16_keys(p)) pitch_clip_kernel<true><<<cgrid, 32 * kPitchWarps, kClipCtaSmem, st>>>(p);
    else pitch_clip_kernel<false><<<cgrid, 32 * kPitchWarps, kClipCtaSmem, st>>>(p);
    LAUNCH_CHECK("pitch_clip_kernel", st);
    // 3: cepstrum frames other than 512 samples (pitch_cep_bluestein_kernel)
    const int fmode = p.mode == 0 ? (p.frame_len == kCepLen ? 0 : 3) : (acr_short_frames(p.frame_len, p.row_len) ? 2 : 1);
    const int per = (fmode == 2 ? 4 : 2) * kPitchWarps;
    const unsigned fgrid = (unsigned)((slots + per - 1) / per);
    if (fmode == 0) pitch_frame_kernel<0><<<fgrid, 32 * kPitchWarps, kFrameCtaSmem, st>>>(p);
    else if (fmode == 3) pitch_cep_bluestein_kernel<<<fgrid, 32 * kPitchWarps, kFrameCtaSmem, st>>>(p);
    else if (fmode == 2) pitch_frame_kernel<2><<<fgrid, 32 * kPitchWarps, kQuadCtaSmem, st>>>(p);
    else pitch_frame_kernel<1><<<fgrid, 32 * kPitchWarps, kFrameCtaSmem, st>>>(p);
    LAUNCH_CHECK(fmode == 0 ? "pitch_frame_kernel<0>" : fmode == 3 ? "pitch_cep_bluestein_kernel" : fmode == 2 ? "pitch_frame_kernel<2>" : "pitch_frame_kernel<1>", st);
    if (d_pitch || d_lag || d_feat) {
        pitch_track_kernel<<<(unsigned)n_utt, kTrackThreads, track_smem(p.row_len), st>>>(p);
        LAUNCH_CHECK("pitch_track_kernel", st);
    }
    if (d_feat) {
        pitch_feature_kernel<<<(unsigned)n_utt, 32, 5 * kFeatMaxFrames * sizeof(double), st>>>(p);
        LAUNCH_CHECK("pitch_feature_kernel", st);
    }
    return DSPFE_OK;
}

int dspfe_pitch_host(dspfe_pitch_plan* pl, const void* h_pcm, int32_t sample_dtype, const int64_t* h_offsets, const int32_t* h_trim,
                     int32_t n_utt, double* h_pitch, int32_t* h_lag, double* h_feat, int64_t* h_frame_off) {
    if (int rc = check_host_batch(pl && (sample_dtype == 0 || sample_dtype == 1), h_offsets, n_utt)) return rc;
    if (n_utt == 0) return DSPFE_OK;
    int rc = pl->d_trim.reserve((int64_t)n_utt * 2);
    if (!rc) rc = pl->d_feat.reserve((int64_t)n_utt * 5);
    if (rc) return rc;
    auto frames_of = [&](int32_t u, int64_t len) {
        if (h_trim) { long long l = h_trim[2 * u]; len = trim_slice(len, l, h_trim[2 * u + 1]); }
        return dspfe_pitch_num_frames(pl, len);
    };
    int64_t total = 0, frames = 0;
    rc = pl->host.stage(h_pcm, sample_dtype ? 4 : 2, h_offsets, n_utt, frames_of, h_frame_off, &total, &frames);
    if (rc) return rc;
    const cudaStream_t st = pl->host.stream();
    if (h_trim) CUDA_TRY(cudaMemcpyAsync(pl->d_trim.get(), h_trim, (int64_t)n_utt * 2 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    const int64_t bound = dspfe_pitch_frames_bound(pl, total, n_utt);
    rc = ensure(pl, n_utt, bound);   // size the workspaces first: their pointers are the outputs of the device call
    if (rc) return rc;
    rc = dspfe_pitch(pl, pl->host.pcm(), sample_dtype, total, pl->host.offsets(), h_trim ? pl->d_trim.get() : nullptr, n_utt, pl->pitch.get(),
                     pl->lag.get(), h_feat ? pl->d_feat.get() : nullptr, nullptr, nullptr, bound, st);
    if (rc) return rc;
    if (h_pitch) CUDA_TRY(cudaMemcpyAsync(h_pitch, pl->pitch.get(), frames * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (h_lag) CUDA_TRY(cudaMemcpyAsync(h_lag, pl->lag.get(), frames * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (h_feat) CUDA_TRY(cudaMemcpyAsync(h_feat, pl->d_feat.get(), (int64_t)n_utt * 5 * sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return DSPFE_OK;
}

/* ---- taps: the reference's per-frame / per-row functions on caller-supplied device arrays ---- */
int dspfe_center_clip_f32(const float* d_in, int64_t n_rows, int32_t len, int32_t binary, float* d_out, void* stream) {
    if (!d_in || !d_out || n_rows < 0 || len < 1) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (len > 512) return fail(DSPFE_ERR_UNSUPPORTED, "center_clip rows longer than 512 samples are not built");
    if (n_rows == 0) return DSPFE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    center_clip_kernel<<<(unsigned)((n_rows + 3) / 4), 128, 0, st>>>(d_in, n_rows, len, binary, d_out);
    LAUNCH_CHECK("center_clip_kernel", st);
    return DSPFE_OK;
}

int dspfe_track_rows_f32(const float* d_rows, int64_t n_rows, int32_t row_len, int32_t mode, int32_t do_smooth, float* d_smoothed,
                         int32_t* d_score, int32_t* d_lag, void* stream) {
    if (!d_rows || n_rows < 1 || row_len < 1 || (mode != 0 && mode != 1)) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (row_len > 2 * kTrackThreads) return fail(DSPFE_ERR_UNSUPPORTED, "rows longer than 512 columns are not built");
    if (mode == 0 && (d_score || d_lag) && row_len < kMinLag + kPeakLags) return fail(DSPFE_ERR_INVALID_ARG, "peak_score needs rows of at least 100 columns");
    cudaStream_t st = (cudaStream_t)stream;
    StreamTemp<int64_t> d_fo; StreamTemp<int32_t> d_lag_tmp;
    CUDA_TRY(d_fo.alloc(2, st));
    if (!d_lag) CUDA_TRY(d_lag_tmp.alloc(n_rows, st));
    pitch_fill_off_kernel<<<1, 32, 0, st>>>(d_fo.get(), n_rows);
    PitchParams p; std::memset(&p, 0, sizeof(p));
    p.n_utt = 1; p.mode = mode; p.row_len = row_len; p.frame_off = d_fo.get(); p.rows = const_cast<float*>(d_rows); p.rows_out = d_smoothed;
    p.no_smooth = do_smooth ? 0 : 1; p.score = mode == 0 ? d_score : nullptr; p.lag = d_lag ? d_lag : d_lag_tmp.get(); p.pitch = nullptr;
    static bool attr_done = false;
    if (!attr_done) { CUDA_TRY(cudaFuncSetAttribute(pitch_track_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, track_smem(kCepLen))); attr_done = true; }
    pitch_track_kernel<<<1, kTrackThreads, track_smem(row_len), st>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(DSPFE_ERR_CUDA, std::string("pitch_track_kernel: ") + cudaGetErrorString(e));
    return DSPFE_OK;
}

/* ---- host-only list helpers (same C++ as the device kernels K4b/K6) ---- */
int dspfe_robust_max_pitch_host(const int32_t* lag, int32_t n, int32_t repair, double* pitch) {
    if (!lag || !pitch || n < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (repair) robust_pitch(lag, n, pitch);
    else for (int i = 0; i < n; ++i) pitch[i] = 1.0 / (0.0001 * (double)lag[i]);
    return DSPFE_OK;
}

int dspfe_smooth_subsequence_host(const double* pitch, int32_t n, int32_t tor, double thres, double* seg, int32_t* seg_len,
                                  int32_t* i0, int32_t* j0) {
    if (!pitch || !seg || !seg_len || !i0 || !j0 || n < 1 || tor < 1) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    std::vector<double> tmp(n);
    int a, b;
    *seg_len = smooth_run(pitch, n, tor, thres, seg, tmp.data(), &a, &b);
    *i0 = a; *j0 = b;
    return DSPFE_OK;
}

int dspfe_sub_endpoint_host(const double* amp, int32_t n_frames, int32_t* p) {
    if (!amp || !p || n_frames < 1) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    *p = sub_endpoint(amp, n_frames);
    return DSPFE_OK;
}

int dspfe_pitch_feature_tail_host(const double* pitch, const double* amp, int32_t n_frames, double* out5) {
    if (!pitch || !amp || !out5 || n_frames < 1) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    std::vector<double> work(3 * (size_t)n_frames);
    pitch_feature_tail(pitch, amp, n_frames, work.data(), out5);
    return DSPFE_OK;
}

int dspfe_dp_max_pitch(const double* d_g, int32_t n_rows, int32_t n_cols, double* d_path, void* stream) {
    if (!d_g || !d_path || n_rows < 2 || n_cols < 1) return fail(DSPFE_ERR_INVALID_ARG, "dp_max_pitch needs at least two rows");
    if (n_cols > kDpMaxCols) return fail(DSPFE_ERR_UNSUPPORTED, "dp_max_pitch is built for up to 1024 columns");
    cudaStream_t st = (cudaStream_t)stream;
    StreamTemp<int32_t> d_prev;
    CUDA_TRY(d_prev.alloc((int64_t)n_rows * n_cols, st));
    const int threads = (n_cols + 31) & ~31;
    dp_max_pitch_kernel<<<1, threads, 2 * n_cols * sizeof(double), st>>>(d_g, n_rows, n_cols, d_prev.get(), d_path);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(DSPFE_ERR_CUDA, std::string("dp_max_pitch_kernel: ") + cudaGetErrorString(e));
    return DSPFE_OK;
}

int dspfe_dp_max_pitch_host(const double* g, int32_t n_rows, int32_t n_cols, double* path) {
    // dp_max_pitch (pitch.py:208-225): Viterbi over lags with a 5-per-step jump penalty.  As in the reference, the
    // back-trace starts from the predecessor chosen for the LAST column of the last row (not from the best end state).
    if (!g || !path || n_rows < 2 || n_cols < 1) return fail(DSPFE_ERR_INVALID_ARG, "dp_max_pitch needs at least two rows");
    std::vector<double> dp((size_t)n_cols, 0.0), nx((size_t)n_cols);
    std::vector<int32_t> prev((size_t)n_rows * n_cols, 0);
    int step = 0;
    for (int i = 1; i < n_rows; ++i) {
        for (int j = 0; j < n_cols; ++j) {
            double best = 0; int arg = -1;
            for (int k = 0; k < n_cols; ++k) {
                const double r = dp[k] - 5.0 * (double)(k > j ? k - j : j - k) + g[(size_t)i * n_cols + j];
                if (arg < 0 || r > best) { best = r; arg = k; }
            }
            nx[j] = best; prev[(size_t)i * n_cols + j] = arg; step = arg;
        }
        dp.swap(nx);
    }
    for (int i = n_rows - 1; i >= 0; --i) { path[i] = 10000.0 / (double)step; step = prev[(size_t)i * n_cols + step]; }
    return DSPFE_OK;
}

int dspfe_poly_lead_host(const double* seq, int32_t n, int32_t deg, double* coef) {
    if (!seq || !coef || n < 1 || (deg != 1 && deg != 2)) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n <= deg) return fail(DSPFE_ERR_UNSUPPORTED, "fewer points than coefficients");
    *coef = deg == 1 ? ls_slope(seq, n) : ls_quad(seq, n);
    return DSPFE_OK;
}

}  // extern "C"
