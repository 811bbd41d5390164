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
    Stream stream;              // host path
    // workspaces
    DeviceArray<int64_t> frame_off, block_off; DeviceArray<int32_t> order;
    DeviceArray<int32_t> blk, asum, zcr;
    DeviceArray<double> amp;    // float-sample path: K2f's float64 amplitudes, one per frame like asum
    // float-sample path: the split tree of the pairwise sum over one frame (np_pairwise_tree), uploaded on first use
    std::vector<int32_t> h_tree; int nleaf = 0;
    DeviceArray<int32_t> tree; bool tree_ready = false;
    // host-path staging (int16 or float32 samples)
    DeviceArray<unsigned char> d_pcm;
    DeviceArray<int64_t> d_off; DeviceArray<int32_t> d_lr;
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
    if (!pl || !d_offsets || !d_lr || n_utt < 0 || total_samples < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_utt == 0) return DSPFE_OK;
    if (!d_pcm && total_samples > 0) return fail(DSPFE_ERR_INVALID_ARG, "d_pcm is null");
    if (((uintptr_t)d_pcm & 15) != 0) return fail(DSPFE_ERR_INVALID_ARG, "d_pcm must be 16-byte aligned");
    const int64_t frames_bound = dspfe_endpoint_frames_bound(pl, total_samples, n_utt);
    if ((d_asum || d_zcr) && max_frames < frames_bound) return fail(DSPFE_ERR_INVALID_ARG, "max_frames is below dspfe_endpoint_frames_bound()");
    const int64_t blocks_bound = frames_bound + (int64_t)n_utt * (pl->q + 1);
    int rc = ensure(pl, n_utt, blocks_bound, frames_bound);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    EpParams p;
    p.pcm = d_pcm; p.offsets = d_offsets; p.n_utt = n_utt; p.frame_len = pl->frame_len; p.frame_step = pl->frame_step;
    p.q = pl->q; p.rem = pl->rem; p.frame_off = d_frame_off ? d_frame_off : pl->frame_off.get(); p.block_off = pl->block_off.get();
    p.blk = pl->blk.get(); p.asum = d_asum ? d_asum : pl->asum.get(); p.zcr = d_zcr ? d_zcr : pl->zcr.get(); p.lr = d_lr;
    p.max_blocks = blocks_bound; p.max_frames = frames_bound; p.rule = pl->rule; p.order = pl->order.get();
    ep_prep_kernel<<<1, kEpPrepThreads, 0, st>>>(p);
    LAUNCH_CHECK("ep_prep_kernel", st);
    ep_block_kernel<<<(unsigned)((blocks_bound + 127) / 128), 128, 0, st>>>(p);
    LAUNCH_CHECK("ep_block_kernel", st);
    ep_frame_kernel<<<(unsigned)((frames_bound + 255) / 256), 256, 0, st>>>(p);
    LAUNCH_CHECK("ep_frame_kernel", st);
    ep_decide_kernel<AmpFromSum><<<(unsigned)((n_utt + kEpDecideWarps - 1) / kEpDecideWarps), 32 * kEpDecideWarps, 0, st>>>(p);
    LAUNCH_CHECK("ep_decide_kernel", st);
    return DSPFE_OK;
}

int dspfe_endpoint_f32(dspfe_endpoint_plan* pl, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                       int32_t* d_lr, double* d_amp, int32_t* d_zcr, int64_t* d_frame_off, int64_t max_frames, void* stream) {
    if (!pl || !d_offsets || !d_lr || n_utt < 0 || total_samples < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (pl->frame_len > kEpF32MaxLen) return fail(DSPFE_ERR_UNSUPPORTED, "float-sample endpoint frames longer than 8192 samples are not built");
    if (n_utt == 0) return DSPFE_OK;
    if (!d_pcm && total_samples > 0) return fail(DSPFE_ERR_INVALID_ARG, "d_pcm is null");
    if (((uintptr_t)d_pcm & 15) != 0) return fail(DSPFE_ERR_INVALID_ARG, "d_pcm must be 16-byte aligned");
    const int64_t frames_bound = dspfe_endpoint_frames_bound(pl, total_samples, n_utt);
    if ((d_amp || d_zcr) && max_frames < frames_bound) return fail(DSPFE_ERR_INVALID_ARG, "max_frames is below dspfe_endpoint_frames_bound()");
    const int64_t blocks_bound = frames_bound + (int64_t)n_utt * (pl->q + 1);
    int rc = ensure(pl, n_utt, blocks_bound, frames_bound);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (!pl->tree_ready) {
        rc = pl->tree.reserve((int64_t)pl->h_tree.size());
        if (rc) return rc;
        CUDA_TRY(cudaMemcpyAsync(pl->tree.get(), pl->h_tree.data(), pl->h_tree.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        pl->tree_ready = true;
    }
    EpParams p;
    p.pcm = nullptr; p.offsets = d_offsets; p.n_utt = n_utt; p.frame_len = pl->frame_len; p.frame_step = pl->frame_step;
    p.q = pl->q; p.rem = pl->rem; p.frame_off = d_frame_off ? d_frame_off : pl->frame_off.get(); p.block_off = pl->block_off.get();
    p.blk = pl->blk.get(); p.asum = nullptr; p.zcr = d_zcr ? d_zcr : pl->zcr.get(); p.lr = d_lr;
    p.max_blocks = blocks_bound; p.max_frames = frames_bound; p.rule = pl->rule; p.order = pl->order.get();
    p.amp = d_amp ? d_amp : pl->amp.get();
    EpF32Params f;
    f.pcm = d_pcm; f.total_samples = total_samples; f.offsets = d_offsets; f.frame_off = p.frame_off; f.n_utt = n_utt;
    f.frame_len = pl->frame_len; f.frame_step = pl->frame_step; f.tree = pl->tree.get(); f.nleaf = pl->nleaf;
    f.max_frames = frames_bound; f.amp = const_cast<double*>(p.amp); f.zcr = p.zcr;
    ep_f32_layout(f);
    ep_prep_kernel<<<1, kEpPrepThreads, 0, st>>>(p);
    LAUNCH_CHECK("ep_prep_kernel", st);
    if (f.sm_total > 48 * 1024) CUDA_TRY(cudaFuncSetAttribute(ep_stats_f32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, f.sm_total));
    ep_stats_f32_kernel<<<(unsigned)((frames_bound + f.run - 1) / f.run), kEpF32Threads, f.sm_total, st>>>(f);
    LAUNCH_CHECK("ep_stats_f32_kernel", st);
    ep_decide_kernel<AmpFromF64><<<(unsigned)((n_utt + kEpDecideWarps - 1) / kEpDecideWarps), 32 * kEpDecideWarps, 0, st>>>(p);
    LAUNCH_CHECK("ep_decide_kernel<f64>", st);
    return DSPFE_OK;
}

int dspfe_endpoint_robust(dspfe_endpoint_plan* pl, const int16_t* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                          int32_t* d_lr, void* stream) {
    if (!pl || !d_offsets || !d_lr || n_utt < 0 || total_samples < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_utt == 0) return DSPFE_OK;
    if (!d_pcm && total_samples > 0) return fail(DSPFE_ERR_INVALID_ARG, "d_pcm is null");
    if (pl->frame_len > kEpGateMaxLen) return fail(DSPFE_ERR_UNSUPPORTED, "robust endpoint frames longer than 1536 samples are not built");
    // frame statistics exactly as the basic path (its own decision is discarded), then the gated rule
    int rc = dspfe_endpoint(pl, d_pcm, total_samples, d_offsets, n_utt, d_lr, nullptr, nullptr, nullptr, 0, stream);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t frames_bound = dspfe_endpoint_frames_bound(pl, total_samples, n_utt);
    EpParams p;
    p.pcm = d_pcm; p.offsets = d_offsets; p.n_utt = n_utt; p.frame_len = pl->frame_len; p.frame_step = pl->frame_step;
    p.q = pl->q; p.rem = pl->rem; p.frame_off = pl->frame_off.get(); p.block_off = pl->block_off.get(); p.blk = pl->blk.get();
    p.asum = pl->asum.get(); p.zcr = pl->zcr.get(); p.lr = d_lr; p.max_blocks = 0; p.max_frames = frames_bound; p.rule = pl->rule;
    p.order = pl->order.get();
    CUDA_TRY(cudaFuncSetAttribute(ep_decide_robust_kernel<int16_t>, cudaFuncAttributeMaxDynamicSharedMemorySize, kEpRobustSmem));
    CUDA_TRY(cudaFuncSetAttribute(ep_decide_robust_kernel<int16_t>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    ep_decide_robust_kernel<int16_t><<<(unsigned)n_utt, 32 * kEpRobustWarps, kEpRobustSmem, st>>>(p);
    LAUNCH_CHECK("ep_decide_robust_kernel", st);
    return DSPFE_OK;
}

int dspfe_endpoint_robust_f32(dspfe_endpoint_plan* pl, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                              int32_t* d_lr, void* stream) {
    if (!pl || !d_offsets || !d_lr || n_utt < 0 || total_samples < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (pl->frame_len > kEpGateMaxLen) return fail(DSPFE_ERR_UNSUPPORTED, "robust endpoint frames longer than 1536 samples are not built");
    if (n_utt == 0) return DSPFE_OK;
    // K2f's frame statistics exactly as the basic float path (its own decision is discarded), then the gated rule
    int rc = dspfe_endpoint_f32(pl, d_pcm, total_samples, d_offsets, n_utt, d_lr, nullptr, nullptr, nullptr, 0, stream);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    EpParams p;
    std::memset(&p, 0, sizeof(p));
    p.pcm_f32 = d_pcm; p.offsets = d_offsets; p.n_utt = n_utt; p.frame_len = pl->frame_len; p.frame_step = pl->frame_step;
    p.q = pl->q; p.rem = pl->rem; p.frame_off = pl->frame_off.get(); p.amp = pl->amp.get(); p.zcr = pl->zcr.get(); p.lr = d_lr;
    p.max_frames = dspfe_endpoint_frames_bound(pl, total_samples, n_utt); p.rule = pl->rule; p.order = pl->order.get();
    CUDA_TRY(cudaFuncSetAttribute(ep_decide_robust_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, kEpRobustSmem));
    CUDA_TRY(cudaFuncSetAttribute(ep_decide_robust_kernel<float>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    ep_decide_robust_kernel<float><<<(unsigned)n_utt, 32 * kEpRobustWarps, kEpRobustSmem, st>>>(p);
    LAUNCH_CHECK("ep_decide_robust_kernel<f32>", st);
    return DSPFE_OK;
}

int dspfe_endpoint_robust_host(dspfe_endpoint_plan* pl, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr) {
    if (!pl || !h_offsets || !h_lr || n_utt < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_utt == 0) return DSPFE_OK;
    // stage through the basic host path's buffers (it leaves pcm / offsets on the device), then re-decide with the gate
    int rc = dspfe_endpoint_host(pl, h_pcm, h_offsets, n_utt, h_lr, nullptr, nullptr, nullptr);
    if (rc) return rc;
    const int64_t total = h_offsets[n_utt] - h_offsets[0];
    const cudaStream_t st = pl->stream.get();
    rc = dspfe_endpoint_robust(pl, reinterpret_cast<const int16_t*>(pl->d_pcm.get()), total, pl->d_off.get(), n_utt, pl->d_lr.get(), st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(h_lr, pl->d_lr.get(), (int64_t)n_utt * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return DSPFE_OK;
}

}  // extern "C"

namespace {

// stages a host batch on the plan's stream: the samples into d_pcm, the offsets relative to the first into d_off; *total = the
// sample count, h_frame_off (optional) = the frame prefix sums
template <class T>
int stage_host(dspfe_endpoint_plan* pl, const T* h_pcm, const int64_t* h_offsets, int32_t n_utt, int64_t* h_frame_off, int64_t* total_out,
               int64_t* frames_out) {
    const int64_t base = h_offsets[0], total = h_offsets[n_utt] - base;
    if (total < 0) return fail(DSPFE_ERR_INVALID_ARG, "offsets must be non-decreasing");
    CUDA_TRY(pl->stream.ensure());
    int rc = pl->d_pcm.reserve((total + 8) * (int64_t)sizeof(T));
    if (!rc) rc = pl->d_off.reserve(n_utt + 1);
    if (!rc) rc = pl->d_lr.reserve((int64_t)n_utt * 2);
    if (rc) return rc;
    std::vector<int64_t> rel(n_utt + 1);
    int64_t frames = 0;
    for (int32_t u = 0; u <= n_utt; ++u) {
        rel[u] = h_offsets[u] - base;
        if (u < n_utt) {
            if (h_frame_off) h_frame_off[u] = frames;
            frames += num_frames(h_offsets[u + 1] - h_offsets[u], pl->frame_len, pl->frame_step);
        }
    }
    if (h_frame_off) h_frame_off[n_utt] = frames;
    cudaStream_t st = pl->stream.get();
    if (total > 0) CUDA_TRY(cudaMemcpyAsync(pl->d_pcm.get(), h_pcm + base, total * sizeof(T), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(pl->d_off.get(), rel.data(), (n_utt + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    *total_out = total;
    if (frames_out) *frames_out = frames;
    return DSPFE_OK;
}

// the host-buffer path of either sample type: int16 samples give sum|x| per frame (Stat = int32_t), float32 samples the
// float64 amplitude (Stat = double)
template <class T, class Stat>
int endpoint_host(dspfe_endpoint_plan* pl, const T* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr,
                  Stat* h_stat, int32_t* h_zcr, int64_t* h_frame_off) {
    if (!pl || !h_offsets || !h_lr || n_utt < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_utt == 0) return DSPFE_OK;
    int64_t total = 0, frames = 0;
    int rc = stage_host(pl, h_pcm, h_offsets, n_utt, h_frame_off, &total, &frames);
    if (rc) return rc;
    cudaStream_t st = pl->stream.get();
    const T* d_pcm = reinterpret_cast<const T*>(pl->d_pcm.get());
    if constexpr (sizeof(T) == 2) rc = dspfe_endpoint(pl, d_pcm, total, pl->d_off.get(), n_utt, pl->d_lr.get(), nullptr, nullptr, nullptr, 0, st);
    else rc = dspfe_endpoint_f32(pl, d_pcm, total, pl->d_off.get(), n_utt, pl->d_lr.get(), nullptr, nullptr, nullptr, 0, st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(h_lr, pl->d_lr.get(), (int64_t)n_utt * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    if (h_stat) CUDA_TRY(cudaMemcpyAsync(h_stat, sizeof(T) == 2 ? (void*)pl->asum.get() : (void*)pl->amp.get(), frames * sizeof(Stat), cudaMemcpyDeviceToHost, st));
    if (h_zcr) CUDA_TRY(cudaMemcpyAsync(h_zcr, pl->zcr.get(), frames * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return DSPFE_OK;
}

}  // namespace

extern "C" {

int dspfe_endpoint_host(dspfe_endpoint_plan* pl, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr,
                        int32_t* h_asum, int32_t* h_zcr, int64_t* h_frame_off) {
    return endpoint_host(pl, h_pcm, h_offsets, n_utt, h_lr, h_asum, h_zcr, h_frame_off);
}

int dspfe_endpoint_host_f32(dspfe_endpoint_plan* pl, const float* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr,
                            double* h_amp, int32_t* h_zcr, int64_t* h_frame_off) {
    return endpoint_host(pl, h_pcm, h_offsets, n_utt, h_lr, h_amp, h_zcr, h_frame_off);
}

int dspfe_endpoint_robust_host_f32(dspfe_endpoint_plan* pl, const float* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr) {
    if (!pl || !h_offsets || !h_lr || n_utt < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (pl->frame_len > kEpGateMaxLen) return fail(DSPFE_ERR_UNSUPPORTED, "robust endpoint frames longer than 1536 samples are not built");
    if (n_utt == 0) return DSPFE_OK;
    // the batch is staged once; the device form computes the frame statistics once and then runs the gated rule
    int64_t total = 0;
    int rc = stage_host(pl, h_pcm, h_offsets, n_utt, nullptr, &total, nullptr);
    if (rc) return rc;
    const cudaStream_t st = pl->stream.get();
    rc = dspfe_endpoint_robust_f32(pl, reinterpret_cast<const float*>(pl->d_pcm.get()), total, pl->d_off.get(), n_utt, pl->d_lr.get(), st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(h_lr, pl->d_lr.get(), (int64_t)n_utt * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return DSPFE_OK;
}

}  // extern "C"
