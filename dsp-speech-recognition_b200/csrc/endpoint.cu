// C ABI of the endpoint-detection path (include/dspfe.h, "endpoint" section).  Kernels: endpoint_kernel.cuh.
#include <cstring>
#include <vector>

#include "abi_common.h"
#include "dspfe_types.h"
#include "endpoint_kernel.cuh"

using namespace dspfe;

struct dspfe_endpoint_plan {
    dspfe_endpoint_params prm;
    EpRule rule;
    int frame_len, frame_step, q, rem;
    HostBatch host;             // host-path staging (int16 or float32 samples)
    DeviceArray<int32_t> d_lr;
    // workspaces
    DeviceArray<int64_t> frame_off, block_off; DeviceArray<int32_t> order;
    DeviceArray<int32_t> blk, asum, zcr;
    DeviceArray<double> amp;    // float-sample path: K2f's float64 amplitudes, one per frame like asum
    // float-sample path: the split tree of the pairwise sum over one frame (np_pairwise_tree), uploaded on first use
    std::vector<int32_t> h_tree; int nleaf = 0;
    DeviceArray<int32_t> tree; bool tree_ready = false;
};

namespace {

int fill_rule(const dspfe_endpoint_params& q, EpRule& r, int& frame_len, int& frame_step) {
    if (q.samplerate <= 0 || !(q.cfg_frame > 0) || !(q.cfg_step > 0)) return fail(DSPFE_ERR_INVALID_ARG, "bad endpoint parameters");
    r.cfg_frame = q.cfg_frame; r.cfg_step = q.cfg_step; r.mh1 = q.mh1; r.mh2 = q.mh2; r.th = q.th;
    r.l_sil = q.l_sil; r.r_sil = q.r_sil; r.sigma = q.sigma; r.zcr_max_shift = q.zcr_max_shift; r.zcr_r_sil = q.zcr_r_sil;
    r.min_span = q.min_span; r.rate = q.samplerate;
    frame_len = (int)((double)q.samplerate * q.cfg_frame);   // to_frames: int(rate * t)   (sigproc.py:19)
    frame_step = (int)(q.cfg_step * (double)q.samplerate);   //            int(step * rate)
    if (frame_len < 1 || frame_step < 1) return fail(DSPFE_ERR_UNSUPPORTED, "endpoint frame length/step below one sample");
    if ((int)(q.l_sil / q.cfg_step) + (int)(q.r_sil / q.cfg_step) > 64 || (int)(q.zcr_r_sil / q.cfg_step) > 64)
        return fail(DSPFE_ERR_UNSUPPORTED, "silence windows longer than 64 frames are not supported");
    return DSPFE_OK;
}

int ensure(dspfe_endpoint_plan* pl, int64_t n_utt, int64_t blocks, int64_t frames) {
    int rc = pl->frame_off.reserve(n_utt + 1);
    if (!rc) rc = pl->order.reserve(n_utt + 1);
    if (!rc) rc = pl->block_off.reserve(n_utt + 1);
    if (!rc) rc = pl->blk.reserve(blocks * 6);
    if (!rc) rc = pl->asum.reserve(frames);
    if (!rc) rc = pl->zcr.reserve(frames);
    if (!rc) rc = pl->amp.reserve(frames);
    return rc;
}

// What differs between the sample types: the frame statistics (int16: sum |x| per frame from K2a + K2b; float32: K2f's
// float64 amplitudes), the EpParams fields that carry the samples and the statistics, the decision kernel's amplitude source,
// and the kernel names the timing reports show.
template <class T> struct EpType;
template <> struct EpType<int16_t> {
    using Stat = int32_t;
    using Amp = AmpFromSum;
    static constexpr const char* kDecide = "ep_decide_kernel";
    static constexpr const char* kRobust = "ep_decide_robust_kernel";
    static const char* unsupported(const dspfe_endpoint_plan*) { return nullptr; }
    static Stat* stat(dspfe_endpoint_plan* pl) { return pl->asum.get(); }
    static void set(EpParams& p, const int16_t* x, Stat* stat) { p.pcm = x; p.asum = stat; }
    static int stats(dspfe_endpoint_plan*, const EpParams& p, int64_t, cudaStream_t st) {
        ep_block_kernel<<<(unsigned)((p.max_blocks + 127) / 128), 128, 0, st>>>(p);
        LAUNCH_CHECK("ep_block_kernel", st);
        ep_frame_kernel<<<(unsigned)((p.max_frames + 255) / 256), 256, 0, st>>>(p);
        LAUNCH_CHECK("ep_frame_kernel", st);
        return DSPFE_OK;
    }
};
template <> struct EpType<float> {
    using Stat = double;
    using Amp = AmpFromF64;
    static constexpr const char* kDecide = "ep_decide_kernel<f64>";
    static constexpr const char* kRobust = "ep_decide_robust_kernel<f32>";
    static const char* unsupported(const dspfe_endpoint_plan* pl) {
        return pl && pl->frame_len > kEpF32MaxLen ? "float-sample endpoint frames longer than 8192 samples are not built" : nullptr;
    }
    static Stat* stat(dspfe_endpoint_plan* pl) { return pl->amp.get(); }
    static void set(EpParams& p, const float* x, Stat* stat) { p.pcm_f32 = x; p.amp = stat; }
    static int stats(dspfe_endpoint_plan* pl, const EpParams& p, int64_t total_samples, cudaStream_t st) {
        if (!pl->tree_ready) {
            int rc = pl->tree.reserve((int64_t)pl->h_tree.size());
            if (rc) return rc;
            CUDA_TRY(cudaMemcpyAsync(pl->tree.get(), pl->h_tree.data(), pl->h_tree.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
            pl->tree_ready = true;
        }
        EpF32Params f;
        f.pcm = p.pcm_f32; f.total_samples = total_samples; f.offsets = p.offsets; f.frame_off = p.frame_off; f.n_utt = p.n_utt;
        f.frame_len = p.frame_len; f.frame_step = p.frame_step; f.tree = pl->tree.get(); f.nleaf = pl->nleaf;
        f.max_frames = p.max_frames; f.amp = const_cast<double*>(p.amp); f.zcr = p.zcr;
        ep_f32_layout(f);
        if (f.sm_total > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(ep_stats_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, f.sm_total));
        ep_stats_f32_kernel<<<(unsigned)((p.max_frames + f.run - 1) / f.run), kEpF32Threads, f.sm_total, st>>>(f);
        LAUNCH_CHECK("ep_stats_f32_kernel", st);
        return DSPFE_OK;
    }
};

const char* robust_unsupported(const dspfe_endpoint_plan* pl) {
    return pl && pl->frame_len > kEpGateMaxLen ? "robust endpoint frames longer than 1536 samples are not built" : nullptr;
}

// K1 (prep), the frame statistics, K3 (decision); `robust` then runs K3r's gated rule over the same statistics, which
// overwrites K3's decision.  Null d_stat / d_zcr / d_frame_off: the plan's workspaces.
template <class T>
int endpoint_device(dspfe_endpoint_plan* pl, const T* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt, int32_t* d_lr,
                    typename EpType<T>::Stat* d_stat, int32_t* d_zcr, int64_t* d_frame_off, int64_t max_frames, void* stream, bool robust = false) {
    const char* unsupported = robust ? robust_unsupported(pl) : EpType<T>::unsupported(pl);
    if (int rc = check_batch(pl && d_offsets && d_lr, n_utt, total_samples, d_pcm, unsupported)) return rc;
    if (n_utt == 0) return DSPFE_OK;
    const int64_t frames_bound = dspfe_endpoint_frames_bound(pl, total_samples, n_utt);
    if ((d_stat || d_zcr) && max_frames < frames_bound) return fail(DSPFE_ERR_INVALID_ARG, "max_frames is below dspfe_endpoint_frames_bound()");
    const int64_t blocks_bound = frames_bound + (int64_t)n_utt * (pl->q + 1);
    int rc = ensure(pl, n_utt, blocks_bound, frames_bound);   // first: growing a workspace moves it
    if (rc) return rc;
    EpParams p;
    std::memset(&p, 0, sizeof(p));
    EpType<T>::set(p, d_pcm, d_stat ? d_stat : EpType<T>::stat(pl));
    p.offsets = d_offsets; p.n_utt = n_utt; p.frame_len = pl->frame_len; p.frame_step = pl->frame_step; p.q = pl->q; p.rem = pl->rem;
    p.frame_off = d_frame_off ? d_frame_off : pl->frame_off.get(); p.block_off = pl->block_off.get(); p.blk = pl->blk.get();
    p.zcr = d_zcr ? d_zcr : pl->zcr.get(); p.lr = d_lr; p.rule = pl->rule; p.order = pl->order.get();
    p.max_blocks = blocks_bound; p.max_frames = frames_bound;
    cudaStream_t st = (cudaStream_t)stream;
    ep_prep_kernel<<<1, kEpPrepThreads, 0, st>>>(p);
    LAUNCH_CHECK("ep_prep_kernel", st);
    rc = EpType<T>::stats(pl, p, total_samples, st);
    if (rc) return rc;
    ep_decide_kernel<typename EpType<T>::Amp><<<(unsigned)((n_utt + kEpDecideWarps - 1) / kEpDecideWarps), 32 * kEpDecideWarps, 0, st>>>(p);
    LAUNCH_CHECK(EpType<T>::kDecide, st);
    if (!robust) return DSPFE_OK;
    CUDA_TRY(cudaFuncSetAttribute(ep_decide_robust_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, kEpRobustSmem));
    CUDA_TRY(cudaFuncSetAttribute(ep_decide_robust_kernel<T>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    ep_decide_robust_kernel<T><<<(unsigned)n_utt, 32 * kEpRobustWarps, kEpRobustSmem, st>>>(p);
    LAUNCH_CHECK(EpType<T>::kRobust, st);
    return DSPFE_OK;
}

// the host-buffer forms: the batch is staged once and the device form run once on the plan's stream
template <class T>
int endpoint_host(dspfe_endpoint_plan* pl, const T* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr,
                  typename EpType<T>::Stat* h_stat, int32_t* h_zcr, int64_t* h_frame_off, bool robust = false) {
    if (int rc = check_host_batch(pl && h_lr, h_offsets, n_utt, robust ? robust_unsupported(pl) : nullptr)) return rc;
    if (n_utt == 0) return DSPFE_OK;
    int64_t total = 0, frames = 0;
    int rc = pl->d_lr.reserve((int64_t)n_utt * 2);
    if (!rc) rc = pl->host.stage(h_pcm, sizeof(T), h_offsets, n_utt, [pl](int32_t, int64_t len) { return num_frames(len, pl->frame_len, pl->frame_step); },
                                 h_frame_off, &total, &frames);
    if (rc) return rc;
    const cudaStream_t st = pl->host.stream();
    rc = endpoint_device<T>(pl, pl->host.pcm<T>(), total, pl->host.offsets(), n_utt, pl->d_lr.get(), nullptr, nullptr, nullptr, 0, st, robust);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(h_lr, pl->d_lr.get(), (int64_t)n_utt * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (h_stat) CUDA_TRY(cudaMemcpyAsync(h_stat, EpType<T>::stat(pl), frames * sizeof(*h_stat), cudaMemcpyDeviceToHost, st));
    if (h_zcr) CUDA_TRY(cudaMemcpyAsync(h_zcr, pl->zcr.get(), frames * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return DSPFE_OK;
}

}  // namespace

extern "C" {

void dspfe_endpoint_params_default(dspfe_endpoint_params* p, int32_t samplerate) {
    if (!p) return;
    p->samplerate = samplerate; p->min_span = 50;
    p->cfg_frame = 0.03; p->cfg_step = 0.01; p->mh1 = 0.25; p->mh2 = 0.125; p->th = 0.100; p->l_sil = 0.100; p->r_sil = 0.100;
    p->sigma = 3.0; p->zcr_max_shift = 0.400; p->zcr_r_sil = 0.100;
}

int dspfe_endpoint_decide_host(const dspfe_endpoint_params* p, const int32_t* asum, const int32_t* zcr, int32_t n_frames, int32_t* lr) {
    if (!p || !asum || !zcr || !lr || n_frames < 1) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    EpRule r; int fl, fs;
    int rc = fill_rule(*p, r, fl, fs);
    if (rc) return rc;
    endpoint_decide(asum, zcr, n_frames, fl, r, lr);
    return DSPFE_OK;
}

int dspfe_amplitude_rule_host(const dspfe_endpoint_params* p, const double* amp, int32_t n_frames, double mh,
                              int32_t* segs, int32_t seg_cap, int32_t* n_segs) {
    if (!p || !amp || !n_segs || n_frames < 1 || seg_cap < 1 || !segs) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    EpRule r; int fl, fs;
    int rc = fill_rule(*p, r, fl, fs);
    if (rc) return rc;
    int left, right;
    const int n = amplitude_rule(AmpFromF64{amp}, n_frames, r, mh, &left, &right, segs, seg_cap);
    if (n == 0) { segs[0] = 0; segs[1] = n_frames; *n_segs = 1; } else { *n_segs = n; }   // reference: [(0, len(amp))]
    return DSPFE_OK;
}

int dspfe_amplitude_rule_gated_host(const dspfe_endpoint_params* p, const double* amp, const int32_t* gate, int32_t n_frames, double mh,
                                    int32_t* segs, int32_t seg_cap, int32_t* n_segs) {
    if (!p || !amp || !gate || !n_segs || n_frames < 1 || seg_cap < 1 || !segs) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    EpRule r; int fl, fs;
    int rc = fill_rule(*p, r, fl, fs);
    if (rc) return rc;
    int left, right;
    const int n = amplitude_rule(AmpFromF64{amp}, n_frames, r, mh, &left, &right, segs, seg_cap, GateFromFlags{gate});
    if (n == 0) { segs[0] = 0; segs[1] = n_frames; *n_segs = 1; } else { *n_segs = n; }
    return DSPFE_OK;
}

int dspfe_acr_gate_rows_f64(const double* d_frames, int64_t n_rows, int32_t len, int32_t samplerate, int32_t* d_gate, void* stream) {
    if (n_rows < 0 || len < 1 || samplerate < 1 || (n_rows > 0 && (!d_frames || !d_gate))) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_rows == 0) return DSPFE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    acr_gate_rows_kernel<<<(unsigned)((n_rows + 3) / 4), 128, 0, st>>>(d_frames, n_rows, len, samplerate / 500, samplerate / 50, d_gate);
    LAUNCH_CHECK("acr_gate_rows_kernel", st);
    return DSPFE_OK;
}

int dspfe_zcr_rule_host(const dspfe_endpoint_params* p, const double* zcr, int32_t n_frames, double l_sil, int32_t left,
                        int32_t right, int32_t* out_jk) {
    if (!p || !zcr || !out_jk || n_frames < 1 || left < 0 || left >= n_frames || right < 0 || right > n_frames)
        return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    EpRule r; int fl, fs;
    int rc = fill_rule(*p, r, fl, fs);
    if (rc) return rc;
    int j, k;
    zcr_rule(AmpFromF64{zcr}, n_frames, r, l_sil, left, right, &j, &k);
    out_jk[0] = j; out_jk[1] = k;
    return DSPFE_OK;
}

int dspfe_endpoint_create(const dspfe_endpoint_params* p, dspfe_endpoint_plan** plan) {
    if (!p || !plan) return fail(DSPFE_ERR_INVALID_ARG, "null argument");
    *plan = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(DSPFE_ERR_CUDA, "no CUDA device: libdspfe has no CPU fallback");
    dspfe_endpoint_plan* pl = new (std::nothrow) dspfe_endpoint_plan();
    if (!pl) return fail(DSPFE_ERR_NOMEM, "out of host memory");
    pl->prm = *p;
    int rc = fill_rule(*p, pl->rule, pl->frame_len, pl->frame_step);
    if (rc) { delete pl; return rc; }
    pl->q = pl->frame_len / pl->frame_step; pl->rem = pl->frame_len % pl->frame_step;
    if (pl->frame_len <= kEpF32MaxLen) pl->h_tree = np_pairwise_tree(pl->frame_len, &pl->nleaf);
    *plan = pl;
    return DSPFE_OK;
}

void dspfe_endpoint_destroy(dspfe_endpoint_plan* pl) {
    if (!pl) return;
    delete pl;
}

int dspfe_endpoint_reserve(dspfe_endpoint_plan* pl, int64_t max_utt, int64_t max_total_samples) {
    if (!pl || max_utt < 0 || max_total_samples < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    const int64_t frames = dspfe_endpoint_frames_bound(pl, max_total_samples, max_utt);
    return ensure(pl, max_utt, frames + max_utt * (pl->q + 1), frames);
}

int32_t dspfe_endpoint_frame_len(const dspfe_endpoint_plan* pl) { return pl ? pl->frame_len : -1; }
int32_t dspfe_endpoint_frame_step(const dspfe_endpoint_plan* pl) { return pl ? pl->frame_step : -1; }

int64_t dspfe_endpoint_frames_bound(const dspfe_endpoint_plan* pl, int64_t total_samples, int64_t n_utt) {
    if (!pl) return -1;
    // framesig's count is 1 + ceil((len - frame_len) / step) <= len / step + 1 per utterance when frame_len >= step, and
    // <= len / step + 2 when cfg.step exceeds cfg.frame (gaps between frames)
    return total_samples / pl->frame_step + (pl->frame_len >= pl->frame_step ? 1 : 2) * n_utt;
}

int dspfe_endpoint(dspfe_endpoint_plan* pl, const int16_t* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                   int32_t* d_lr, int32_t* d_asum, int32_t* d_zcr, int64_t* d_frame_off, int64_t max_frames, void* stream) {
    return endpoint_device(pl, d_pcm, total_samples, d_offsets, n_utt, d_lr, d_asum, d_zcr, d_frame_off, max_frames, stream);
}

int dspfe_endpoint_f32(dspfe_endpoint_plan* pl, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                       int32_t* d_lr, double* d_amp, int32_t* d_zcr, int64_t* d_frame_off, int64_t max_frames, void* stream) {
    return endpoint_device(pl, d_pcm, total_samples, d_offsets, n_utt, d_lr, d_amp, d_zcr, d_frame_off, max_frames, stream);
}

int dspfe_endpoint_robust(dspfe_endpoint_plan* pl, const int16_t* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                          int32_t* d_lr, void* stream) {
    return endpoint_device(pl, d_pcm, total_samples, d_offsets, n_utt, d_lr, nullptr, nullptr, nullptr, 0, stream, true);
}

int dspfe_endpoint_robust_f32(dspfe_endpoint_plan* pl, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                              int32_t* d_lr, void* stream) {
    return endpoint_device(pl, d_pcm, total_samples, d_offsets, n_utt, d_lr, nullptr, nullptr, nullptr, 0, stream, true);
}

int dspfe_endpoint_host(dspfe_endpoint_plan* pl, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr,
                        int32_t* h_asum, int32_t* h_zcr, int64_t* h_frame_off) {
    return endpoint_host(pl, h_pcm, h_offsets, n_utt, h_lr, h_asum, h_zcr, h_frame_off);
}

int dspfe_endpoint_host_f32(dspfe_endpoint_plan* pl, const float* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr,
                            double* h_amp, int32_t* h_zcr, int64_t* h_frame_off) {
    return endpoint_host(pl, h_pcm, h_offsets, n_utt, h_lr, h_amp, h_zcr, h_frame_off);
}

int dspfe_endpoint_robust_host(dspfe_endpoint_plan* pl, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr) {
    return endpoint_host(pl, h_pcm, h_offsets, n_utt, h_lr, nullptr, nullptr, nullptr, true);
}

int dspfe_endpoint_robust_host_f32(dspfe_endpoint_plan* pl, const float* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr) {
    return endpoint_host(pl, h_pcm, h_offsets, n_utt, h_lr, nullptr, nullptr, nullptr, true);
}

}  // extern "C"
