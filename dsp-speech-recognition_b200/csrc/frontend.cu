// C ABI of the whole front-end over one packed ragged batch (include/dspfe.h, "whole front-end" section) and of the
// per-kernel timing facility.  Chains the reference's call sites per utterance -- endpoints (model.py:52-53,
// pitch_model.py:38), MFCC + delta + delta on sig[l:r] (model.py:74-77), pitch_feature on preemphasis(sig)[l:r]
// (pitch_model.py:39-41), pitch_detect_sr on sig[l:r] (model.py:92) -- through the public entry points of the other
// translation units, in slabs of consecutive utterances so that the workspaces stay bounded.  No CPU fallback: this file
// only queues kernels and copies.
#include <algorithm>
#include <cstring>
#include <memory>
#include <vector>

#include "abi_common.h"

using namespace dspfe;

namespace {

constexpr int kFeWidth = 39;          // 3 * numcep of the default MFCC configuration
constexpr int kFeSlots = 3;           // host path: PCM / output staging sets (H2D runs up to two slabs ahead)
constexpr int kFeLanes = 2;           // host path: slabs in flight on the GPU (own plans + stream each), so a slab's tail and its single-CTA
                                      // prefix-sum kernels overlap the next slab's transforms

// rel[i] = off[i] - a0 for i < n: the slab's offsets relative to its 16-byte aligned first sample
__global__ void fe_rel_offsets_kernel(const int64_t* off, int n, int64_t a0, int64_t* rel) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) rel[i] = off[i] - a0;
}

// global row / frame offsets of the slab's utterances (local prefix sums + the rows written by earlier slabs) and the
// slab's totals
struct FeFinish {
    const int64_t* loc[3]; int64_t* glob[3]; int64_t base[3]; int64_t* tot; int n;   // n = utterances + 1
    const int64_t* dbase_in; int64_t* dbase_out;   // host path: the bases live on the device (no host round trip per slab)
};
__global__ void fe_finish_kernel(const FeFinish f) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int64_t base = f.dbase_in ? f.dbase_in[k] : f.base[k];
        if (i < f.n && f.glob[k]) f.glob[k][i] = base + f.loc[k][i];
        if (i == 0) { f.tot[k] = f.loc[k][f.n - 1]; if (f.dbase_out) f.dbase_out[k] = base + f.loc[k][f.n - 1]; }
    }
}

struct FeSlot {
    Event h2d_done, compute_done, d2h_done;
    DeviceArray<unsigned char> d_pcm;    // int16 or float32 samples
    DeviceArray<int64_t> d_rel; PinnedArray<int64_t> h_rel;
    DeviceArray<int32_t> d_lr; DeviceArray<double> d_feat; DeviceArray<int64_t> d_goff[3];
    DeviceArray<float> d_mfcc;
    DeviceArray<double> d_cep, d_acr;
    DeviceArray<int32_t> d_cep_lag, d_acr_lag;
};

struct SubPlanDelete {
    void operator()(dspfe_endpoint_plan* p) const { dspfe_endpoint_destroy(p); }
    void operator()(dspfe_plan* p) const { dspfe_plan_destroy(p); }
    void operator()(dspfe_pitch_plan* p) const { dspfe_pitch_destroy(p); }
};
template <class P> using SubPlan = std::unique_ptr<P, SubPlanDelete>;

}  // namespace

struct FeLane {                       // one slab in flight: the four sub-plans own the workspaces of their kernels
    Stream stream;                                                               // host path only
    Event finish_done;
    // the two pitch chains of a slab run beside its MFCC kernels (they only share the endpoints): side streams, fork / join events
    Stream side[2];
    Event ev_fork, ev_join[2];
    DeviceArray<int64_t> loc_off[3];                                             // slab-local row / frame prefix sums
    DeviceArray<int64_t> d_tot;                                                  // [3] the slab's totals
    SubPlan<dspfe_endpoint_plan> ep; SubPlan<dspfe_plan> mf; SubPlan<dspfe_pitch_plan> cep, acr;
};

struct dspfe_frontend_plan {
    dspfe_frontend_params prm;
    Stream s_copy, s_out;
    FeLane lanes[kFeLanes];               // the device path uses lane 0 on the caller's stream
    FeSlot slots[kFeSlots];
    DeviceArray<int64_t> rel_off;
    DeviceArray<int64_t> d_base;          // [2][3] device-side running bases of the host path (ping-pong between consecutive slabs)
    PinnedArray<int64_t> h_tot;           // [kFeSlots][3]
    // scratch for outputs the caller does not want
    DeviceArray<int32_t> s_lr;
    DeviceArray<float> s_mfcc;
    DeviceArray<double> s_cep, s_acr;
};

namespace {

int create_lane(FeLane& ln, const dspfe_frontend_params& q) {
    dspfe_endpoint_params eq; dspfe_endpoint_params_default(&eq, q.samplerate);
    dspfe_mfcc_params mq; dspfe_mfcc_params_default(&mq);
    mq.samplerate = q.samplerate; mq.delta_n = q.delta_n;
    mq.frame_len = (int32_t)(0.025 * q.samplerate + 0.5); mq.frame_step = (int32_t)(0.01 * q.samplerate + 0.5);
    dspfe_pitch_params cq; dspfe_pitch_params_default(&cq, 0);
    cq.samplerate = q.samplerate; cq.preemph = q.cep_preemph;
    dspfe_pitch_params aq; dspfe_pitch_params_default(&aq, 1);
    aq.samplerate = q.samplerate; aq.frame_len = q.acr_frame_len;
    dspfe_endpoint_plan* ep = nullptr; dspfe_plan* mf = nullptr; dspfe_pitch_plan *cep = nullptr, *acr = nullptr;
    int rc = dspfe_endpoint_create(&eq, &ep);
    if (!rc) rc = dspfe_plan_create(&mq, &mf);
    if (!rc) rc = dspfe_pitch_create(&cq, &cep);
    if (!rc) rc = dspfe_pitch_create(&aq, &acr);
    ln.ep.reset(ep); ln.mf.reset(mf); ln.cep.reset(cep); ln.acr.reset(acr);
    if (!rc) rc = ln.d_tot.reserve(3);
    return rc;
}

// The sample types of the batch: int16 (dspfe_frontend*) and float32 (dspfe_frontend*_f32).  A slab starts at the 16-byte
// aligned sample at or before its first utterance: a multiple of kAlign samples.
template <class T> struct FeSamples;
template <> struct FeSamples<int16_t> {
    static constexpr int kAlign = 8, kDtype = 0;
    static int endpoint(dspfe_endpoint_plan* p, const int16_t* x, int64_t n, const int64_t* off, int32_t nu, int32_t* lr, cudaStream_t st) {
        return dspfe_endpoint(p, x, n, off, nu, lr, nullptr, nullptr, nullptr, 0, st);
    }
    static int mfcc(dspfe_plan* p, const int16_t* x, int64_t n, const int64_t* off, const int32_t* lr, int32_t nu, float* out, int64_t cap,
                    int64_t* fo, cudaStream_t st) {
        return dspfe_mfcc_delta(p, x, n, off, lr, nu, out, cap, fo, st);
    }
};
template <> struct FeSamples<float> {
    static constexpr int kAlign = 4, kDtype = 1;
    static int endpoint(dspfe_endpoint_plan* p, const float* x, int64_t n, const int64_t* off, int32_t nu, int32_t* lr, cudaStream_t st) {
        return dspfe_endpoint_f32(p, x, n, off, nu, lr, nullptr, nullptr, nullptr, 0, st);
    }
    static int mfcc(dspfe_plan* p, const float* x, int64_t n, const int64_t* off, const int32_t* lr, int32_t nu, float* out, int64_t cap,
                    int64_t* fo, cudaStream_t st) {
        return dspfe_mfcc_delta_f32(p, x, n, off, lr, nu, out, cap, fo, st);
    }
};

// the slab's kernels on `st`: endpoints -> MFCC -> cepstrum pitch + pitch_feature -> autocorrelation pitch -> offsets.
// `wait_prev` (host path): the previous slab's finish kernel, which wrote the running bases this slab's finish kernel reads.
template <class T>
int run_slab(dspfe_frontend_plan* pl, FeLane& ln, const T* pcm, int64_t total, const int64_t* rel_off, int32_t nu, int32_t* lr,
             float* mfcc, int64_t mfcc_cap, double* cep, int32_t* cep_lag, int64_t cep_cap, double* feat, double* acr, int32_t* acr_lag,
             int64_t acr_cap, int64_t* const glob[3], const int64_t base[3], cudaStream_t st, const int64_t* dbase_in = nullptr,
             int64_t* dbase_out = nullptr, int64_t* h_tot = nullptr, cudaEvent_t wait_prev = nullptr) {
    int rc = FeSamples<T>::endpoint(ln.ep.get(), pcm, total, rel_off, nu, lr, st);
    if (rc) return rc;
    // MFCC, cepstrum pitch and autocorrelation pitch depend on the endpoints only: three branches, so that the single-CTA
    // prefix sums, the latency-bound pitch_feature kernel and the ragged tails of the track kernels of one branch are filled
    // by the other branches' transforms.  While a per-kernel timing collection is open everything stays on `st`, serially.
    const bool fork = !g_timer.on;
    cudaStream_t sa = st, sb = st;
    if (fork) {
        for (int k = 0; k < 2; ++k) {
            CUDA_TRY(ln.side[k].ensure());
            CUDA_TRY(ln.ev_join[k].ensure());
        }
        CUDA_TRY(ln.ev_fork.ensure());
        CUDA_TRY(cudaEventRecord(ln.ev_fork.get(), st));
        sa = ln.side[0].get(); sb = ln.side[1].get();
        CUDA_TRY(cudaStreamWaitEvent(sa, ln.ev_fork.get(), 0));
        CUDA_TRY(cudaStreamWaitEvent(sb, ln.ev_fork.get(), 0));
    }
    rc = dspfe_pitch(ln.cep.get(), pcm, FeSamples<T>::kDtype, total, rel_off, lr, nu, cep, cep_lag, feat, nullptr, ln.loc_off[1].get(), cep_cap, sa);
    if (rc) return rc;
    rc = dspfe_pitch(ln.acr.get(), pcm, FeSamples<T>::kDtype, total, rel_off, lr, nu, acr, acr_lag, nullptr, nullptr, ln.loc_off[2].get(), acr_cap, sb);
    if (rc) return rc;
    rc = FeSamples<T>::mfcc(ln.mf.get(), pcm, total, rel_off, lr, nu, mfcc, mfcc_cap, ln.loc_off[0].get(), st);
    if (rc) return rc;
    if (fork) {
        CUDA_TRY(cudaEventRecord(ln.ev_join[0].get(), sa));
        CUDA_TRY(cudaEventRecord(ln.ev_join[1].get(), sb));
        CUDA_TRY(cudaStreamWaitEvent(st, ln.ev_join[0].get(), 0));
        CUDA_TRY(cudaStreamWaitEvent(st, ln.ev_join[1].get(), 0));
    }
    if (wait_prev) CUDA_TRY(cudaStreamWaitEvent(st, wait_prev, 0));
    FeFinish f;
    for (int k = 0; k < 3; ++k) { f.loc[k] = ln.loc_off[k].get(); f.glob[k] = glob[k]; f.base[k] = base[k]; }
    f.tot = ln.d_tot.get(); f.n = nu + 1; f.dbase_in = dbase_in; f.dbase_out = dbase_out;
    fe_finish_kernel<<<(unsigned)((nu + 1 + 255) / 256), 256, 0, st>>>(f);
    LAUNCH_CHECK("fe_finish_kernel", st);
    CUDA_TRY(cudaMemcpyAsync(h_tot ? h_tot : pl->h_tot.get(), ln.d_tot.get(), 3 * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    return DSPFE_OK;
}

// next slab of consecutive utterances: at most `cap` samples (one oversized utterance is its own slab)
int32_t slab_end(const int64_t* h_off, int32_t u0, int32_t n_utt, int64_t cap) {
    int32_t u1 = u0 + 1;
    while (u1 < n_utt && h_off[u1 + 1] - h_off[u0] <= cap) ++u1;
    return u1;
}

}  // namespace

extern "C" {

void dspfe_frontend_params_default(dspfe_frontend_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->samplerate = 16000; p->delta_n = 2; p->acr_frame_len = 300; p->cep_preemph = 0.97;
}

void dspfe_frontend_destroy(dspfe_frontend_plan* pl) {
    if (!pl) return;
    delete pl;
}

int dspfe_frontend_create(const dspfe_frontend_params* q, dspfe_frontend_plan** plan) {
    if (!q || !plan) return fail(DSPFE_ERR_INVALID_ARG, "null argument");
    *plan = nullptr;
    if (q->samplerate < 1 || q->delta_n < 1 || q->acr_frame_len < 1 || q->slab_samples < 0 || q->host_slab_samples < 0)
        return fail(DSPFE_ERR_INVALID_ARG, "bad front-end parameter");
    dspfe_frontend_plan* pl = new (std::nothrow) dspfe_frontend_plan();
    if (!pl) return fail(DSPFE_ERR_NOMEM, "out of host memory");
    pl->prm = *q;
    if (pl->prm.slab_samples == 0) pl->prm.slab_samples = 256ll << 20;
    if (pl->prm.host_slab_samples == 0) pl->prm.host_slab_samples = 32ll << 20;
    int rc = create_lane(pl->lanes[0], pl->prm);       // the second lane (host path only) is created on first use
    if (!rc) rc = pl->d_base.reserve(6);
    if (!rc) rc = pl->h_tot.reserve(kFeSlots * 3);
    if (rc) { const std::string keep = g_err; delete pl; g_err = keep; return rc; }
    *plan = pl;
    return DSPFE_OK;
}

int dspfe_frontend_bounds(const dspfe_frontend_plan* pl, int64_t total_samples, int64_t n_utt, int64_t* caps) {
    if (!pl || !caps || total_samples < 0 || n_utt < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    // a slab starts at the 16-byte aligned sample at or before its first utterance: up to 7 extra samples per slab
    const int64_t slabs = total_samples / std::min(pl->prm.slab_samples, pl->prm.host_slab_samples) + 8;   // (+ the host path's short ramp-up / ramp-down slabs)
    const int64_t padded = total_samples + 8 * slabs;
    const FeLane& l0 = pl->lanes[0];
    caps[0] = dspfe_rows_bound(l0.mf.get(), padded, n_utt);
    caps[1] = dspfe_pitch_frames_bound(l0.cep.get(), padded, n_utt) + 3 * slabs;
    caps[2] = dspfe_pitch_frames_bound(l0.acr.get(), padded, n_utt) + 3 * slabs;
    return DSPFE_OK;
}

}  // extern "C"

namespace {

template <class T>
int frontend_device(dspfe_frontend_plan* pl, const T* d_pcm, const int64_t* d_offsets, const int64_t* h_off, int32_t n_utt,
                    const dspfe_frontend_out* o, int64_t* totals, void* stream) {
    constexpr int64_t kAlign = FeSamples<T>::kAlign;
    if (totals) totals[0] = totals[1] = totals[2] = 0;
    const int64_t total_samples = h_off && n_utt > 0 ? h_off[n_utt] - h_off[0] : 0;
    if (int rc = check_batch(pl && d_offsets && h_off && o, n_utt, total_samples, d_pcm)) return rc;
    if (int rc = check_host_batch(true, h_off, n_utt)) return rc;
    if (n_utt == 0) return DSPFE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    int64_t base[3] = {0, 0, 0};
    for (int32_t u0 = 0; u0 < n_utt;) {
        const int32_t u1 = slab_end(h_off, u0, n_utt, pl->prm.slab_samples), nu = u1 - u0;
        const int64_t a0 = h_off[u0] & ~(kAlign - 1), total = h_off[u1] - a0;
        FeLane& ln = pl->lanes[0];
        int rc = DSPFE_OK;
        for (auto& q : ln.loc_off) if (!rc) rc = q.reserve(nu + 1);
        if (!rc) rc = pl->rel_off.reserve(nu + 1);
        if (rc) return rc;
        fe_rel_offsets_kernel<<<(unsigned)((nu + 1 + 255) / 256), 256, 0, st>>>(d_offsets + u0, nu + 1, a0, pl->rel_off.get());
        LAUNCH_CHECK("fe_rel_offsets_kernel", st);
        const int64_t need0 = dspfe_rows_bound(ln.mf.get(), total, nu), need1 = dspfe_pitch_frames_bound(ln.cep.get(), total, nu),
                      need2 = dspfe_pitch_frames_bound(ln.acr.get(), total, nu);
        int32_t* lr = o->lr ? o->lr + 2 * (int64_t)u0 : nullptr;
        float* mfcc = o->mfcc ? o->mfcc + base[0] * kFeWidth : nullptr; int64_t cap0 = o->mfcc_cap - base[0];
        double* cep = o->cep_pitch ? o->cep_pitch + base[1] : nullptr; int64_t cap1 = o->cep_cap - base[1];
        double* acr = o->acr_pitch ? o->acr_pitch + base[2] : nullptr; int64_t cap2 = o->acr_cap - base[2];
        if (!lr) { rc = pl->s_lr.reserve(2 * (int64_t)nu); if (rc) return rc; lr = pl->s_lr.get(); }
        if (!mfcc) { rc = pl->s_mfcc.reserve(need0 * kFeWidth); if (rc) return rc; mfcc = pl->s_mfcc.get(); cap0 = need0; }
        if (!cep) { rc = pl->s_cep.reserve(need1); if (rc) return rc; cep = pl->s_cep.get(); cap1 = need1; }
        if (!acr) { rc = pl->s_acr.reserve(need2); if (rc) return rc; acr = pl->s_acr.get(); cap2 = need2; }
        if (cap0 < need0 || cap1 < need1 || cap2 < need2) return fail(DSPFE_ERR_INVALID_ARG, "output capacity is below dspfe_frontend_bounds()");
        int64_t* glob[3] = {o->mfcc_frame_off ? o->mfcc_frame_off + u0 : nullptr, o->cep_frame_off ? o->cep_frame_off + u0 : nullptr,
                            o->acr_frame_off ? o->acr_frame_off + u0 : nullptr};
        rc = run_slab(pl, ln, d_pcm + a0, total, pl->rel_off.get(), nu, lr, mfcc, cap0, cep, o->cep_lag ? o->cep_lag + base[1] : nullptr, cap1,
                      o->cep_feat ? o->cep_feat + 5 * (int64_t)u0 : nullptr, acr, o->acr_lag ? o->acr_lag + base[2] : nullptr, cap2, glob, base, st);
        if (rc) return rc;
        CUDA_TRY(cudaStreamSynchronize(st));
        for (int k = 0; k < 3; ++k) base[k] += pl->h_tot.get()[k];
        u0 = u1;
    }
    if (totals) for (int k = 0; k < 3; ++k) totals[k] = base[k];
    return DSPFE_OK;
}

template <class T>
int frontend_host(dspfe_frontend_plan* pl, const T* h_pcm, const int64_t* h_off, int32_t n_utt, const dspfe_frontend_out* o,
                  int64_t* totals) {
    constexpr int64_t kAlign = FeSamples<T>::kAlign;
    if (totals) totals[0] = totals[1] = totals[2] = 0;
    if (int rc = check_host_batch(pl && o, h_off, n_utt)) return rc;
    if (n_utt == 0) return DSPFE_OK;
    if (!h_pcm && h_off[n_utt] > h_off[0]) return fail(DSPFE_ERR_INVALID_ARG, "h_pcm is null");
    CUDA_TRY(pl->s_copy.ensure());
    for (auto& ln : pl->lanes) {
        if (!ln.ep) { int rc = create_lane(ln, pl->prm); if (rc) return rc; }
        CUDA_TRY(ln.stream.ensure());
        CUDA_TRY(ln.finish_done.ensure());
    }
    CUDA_TRY(pl->s_out.ensure());
    for (auto& s : pl->slots) {
        CUDA_TRY(s.h2d_done.ensure());
        CUDA_TRY(s.compute_done.ensure());
        CUDA_TRY(s.d2h_done.ensure());
    }
    // the slabs
    std::vector<int32_t> cut{0};                         // short slabs first: the kernels start after a quarter-slab's copy;
    while (cut.back() < n_utt) {                         // short slabs last: nothing overlaps the last slab's kernels and its copy back
        const size_t k = cut.size();
        const int64_t S = pl->prm.host_slab_samples, rem = h_off[n_utt] - h_off[cut.back()];
        int64_t cap = k == 1 ? S / 4 : (k == 2 ? S / 2 : S);
        if (rem > S / 4) cap = std::min(cap, std::max(S / 4, rem / 2));
        cut.push_back(slab_end(h_off, cut.back(), n_utt, cap));
    }
    const int n_slab = (int)cut.size() - 1;
    const int64_t base0 = h_off[0] & ~(kAlign - 1);     // h_pcm is addressed from this sample on (its predecessors are never read)
    auto issue_h2d = [&](int s) -> int {
        FeSlot& sl = pl->slots[s % kFeSlots];
        const int32_t u0 = cut[s], u1 = cut[s + 1], nu = u1 - u0;
        const int64_t a0 = std::max(h_off[u0] & ~(kAlign - 1), base0), total = h_off[u1] - a0;
        const cudaStream_t scopy = pl->s_copy.get();
        CUDA_TRY(cudaStreamWaitEvent(scopy, sl.compute_done.get(), 0));            // the slab that used this slot has been processed
        const int64_t n = nu + 1;
        int rc = sl.d_pcm.reserve((total + 16) * (int64_t)sizeof(T), (pl->prm.host_slab_samples + 16) * (int64_t)sizeof(T));
        if (!rc) rc = sl.d_rel.reserve(n, 1024);
        if (!rc) rc = sl.d_lr.reserve(2 * n, 2 * 1024);
        if (!rc) rc = sl.d_feat.reserve(5 * n, 5 * 1024);
        for (auto& q : sl.d_goff) if (!rc) rc = q.reserve(n, 1024);
        if (!rc) rc = sl.h_rel.reserve(n, 1024);
        if (rc) return rc;
        CUDA_TRY(cudaEventSynchronize(sl.h2d_done.get()));                         // the slot's previous offsets have left h_rel
        for (int32_t i = 0; i <= nu; ++i) sl.h_rel.get()[i] = h_off[u0 + i] - a0;
        // (a0 - base0 .. ) may start before h_off[u0]: those samples belong to the previous utterance and exist in h_pcm
        if (total > 0) CUDA_TRY(cudaMemcpyAsync(sl.d_pcm.get(), h_pcm + a0, total * sizeof(T), cudaMemcpyHostToDevice, scopy));
        CUDA_TRY(cudaMemcpyAsync(sl.d_rel.get(), sl.h_rel.get(), n * sizeof(int64_t), cudaMemcpyHostToDevice, scopy));
        CUDA_TRY(cudaEventRecord(sl.h2d_done.get(), scopy));
        return DSPFE_OK;
    };
    // The kernels of slab s are queued without waiting for slab s - 1, on the other lane (its own plans and stream: two slabs
    // are in flight on the GPU); the running row / frame bases live on the device (d_base[s & 1], written by the previous
    // slab's last kernel, the only cross-lane dependency).  The host only needs a slab's totals to size its
    // D2H copies, and drains slab s - 1 after queuing slab s, so the GPU never waits for the host.
    int64_t base[3] = {0, 0, 0};
    const int64_t zero3[3] = {0, 0, 0};
    CUDA_TRY(cudaMemsetAsync(pl->d_base.get(), 0, 3 * sizeof(int64_t), pl->lanes[0].stream.get()));    // slab 0 runs on lane 0 and reads d_base[0]
    auto drain = [&](int s) -> int {
        FeSlot& sl = pl->slots[s % kFeSlots];
        const int32_t u0 = cut[s], nu = cut[s + 1] - u0;
        CUDA_TRY(cudaEventSynchronize(sl.compute_done.get()));                     // the slab's frame counts are in its h_tot
        const int64_t* ht = pl->h_tot.get() + 3 * (s % kFeSlots);
        const int64_t t0 = ht[0], t1 = ht[1], t2 = ht[2];
        cudaStream_t so = pl->s_out.get();
        CUDA_TRY(cudaStreamWaitEvent(so, sl.compute_done.get(), 0));
        if (o->lr) CUDA_TRY(cudaMemcpyAsync(o->lr + 2 * (int64_t)u0, sl.d_lr.get(), (int64_t)nu * 2 * sizeof(int32_t), cudaMemcpyDeviceToHost, so));
        if (o->mfcc) {
            if (base[0] + t0 > o->mfcc_cap) return fail(DSPFE_ERR_INVALID_ARG, "h_out->mfcc capacity too small");
            CUDA_TRY(cudaMemcpyAsync(o->mfcc + base[0] * kFeWidth, sl.d_mfcc.get(), t0 * kFeWidth * sizeof(float), cudaMemcpyDeviceToHost, so));
        }
        if ((o->cep_pitch || o->cep_lag) && base[1] + t1 > o->cep_cap) return fail(DSPFE_ERR_INVALID_ARG, "h_out cepstrum capacity too small");
        if ((o->acr_pitch || o->acr_lag) && base[2] + t2 > o->acr_cap) return fail(DSPFE_ERR_INVALID_ARG, "h_out autocorrelation capacity too small");
        if (o->cep_pitch) CUDA_TRY(cudaMemcpyAsync(o->cep_pitch + base[1], sl.d_cep.get(), t1 * sizeof(double), cudaMemcpyDeviceToHost, so));
        if (o->acr_pitch) CUDA_TRY(cudaMemcpyAsync(o->acr_pitch + base[2], sl.d_acr.get(), t2 * sizeof(double), cudaMemcpyDeviceToHost, so));
        if (o->cep_lag) CUDA_TRY(cudaMemcpyAsync(o->cep_lag + base[1], sl.d_cep_lag.get(), t1 * sizeof(int32_t), cudaMemcpyDeviceToHost, so));
        if (o->acr_lag) CUDA_TRY(cudaMemcpyAsync(o->acr_lag + base[2], sl.d_acr_lag.get(), t2 * sizeof(int32_t), cudaMemcpyDeviceToHost, so));
        if (o->cep_feat) CUDA_TRY(cudaMemcpyAsync(o->cep_feat + 5 * (int64_t)u0, sl.d_feat.get(), (int64_t)nu * 5 * sizeof(double), cudaMemcpyDeviceToHost, so));
        int64_t* hg[3] = {o->mfcc_frame_off, o->cep_frame_off, o->acr_frame_off};
        for (int k = 0; k < 3; ++k)
            if (hg[k]) CUDA_TRY(cudaMemcpyAsync(hg[k] + u0, sl.d_goff[k].get(), (int64_t)(nu + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, so));
        CUDA_TRY(cudaEventRecord(sl.d2h_done.get(), so));
        base[0] += t0; base[1] += t1; base[2] += t2;
        return DSPFE_OK;
    };
    int rc = issue_h2d(0);
    if (rc) return rc;
    for (int s = 0; s < n_slab; ++s) {
        FeSlot& sl = pl->slots[s % kFeSlots];
        const int32_t u0 = cut[s], u1 = cut[s + 1], nu = u1 - u0;
        const int64_t a0 = std::max(h_off[u0] & ~(kAlign - 1), base0), total = h_off[u1] - a0;
        FeLane& ln = pl->lanes[s % kFeLanes];
        cudaStream_t sc = ln.stream.get();
        const int64_t need0 = dspfe_rows_bound(ln.mf.get(), total, nu), need1 = dspfe_pitch_frames_bound(ln.cep.get(), total, nu),
                      need2 = dspfe_pitch_frames_bound(ln.acr.get(), total, nu);
        CUDA_TRY(cudaStreamWaitEvent(sc, sl.d2h_done.get(), 0));                  // the slot's previous outputs have left
        rc = sl.d_mfcc.reserve(need0 * kFeWidth);
        if (!rc) rc = sl.d_cep.reserve(need1);
        if (!rc) rc = sl.d_acr.reserve(need2);
        if (!rc && o->cep_lag) rc = sl.d_cep_lag.reserve(need1);
        if (!rc && o->acr_lag) rc = sl.d_acr_lag.reserve(need2);
        for (auto& q : ln.loc_off) if (!rc) rc = q.reserve(nu + 1);
        if (rc) return rc;
        CUDA_TRY(cudaStreamWaitEvent(sc, sl.h2d_done.get(), 0));
        int64_t* const goff[3] = {sl.d_goff[0].get(), sl.d_goff[1].get(), sl.d_goff[2].get()};
        rc = run_slab(pl, ln, reinterpret_cast<const T*>(sl.d_pcm.get()), total, sl.d_rel.get(), nu, sl.d_lr.get(), sl.d_mfcc.get(), need0, sl.d_cep.get(),
                      o->cep_lag ? sl.d_cep_lag.get() : nullptr, need1, sl.d_feat.get(), sl.d_acr.get(), o->acr_lag ? sl.d_acr_lag.get() : nullptr,
                      need2, goff, zero3, sc, pl->d_base.get() + 3 * (s & 1), pl->d_base.get() + 3 * ((s + 1) & 1),
                      pl->h_tot.get() + 3 * (s % kFeSlots), s > 0 ? pl->lanes[(s - 1) % kFeLanes].finish_done.get() : nullptr);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(ln.finish_done.get(), sc));
        CUDA_TRY(cudaEventRecord(sl.compute_done.get(), sc));
        if (s + 1 < n_slab) { rc = issue_h2d(s + 1); if (rc) return rc; }          // overlaps this slab's kernels
        if (s >= 1) { rc = drain(s - 1); if (rc) return rc; }                      // (that slab finished while this one was being queued)
    }
    rc = drain(n_slab - 1);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(pl->s_out.get()));
    if (totals) for (int k = 0; k < 3; ++k) totals[k] = base[k];
    return DSPFE_OK;
}

}  // namespace

extern "C" {

int dspfe_frontend(dspfe_frontend_plan* pl, const int16_t* d_pcm, const int64_t* d_offsets, const int64_t* h_off, int32_t n_utt,
                   const dspfe_frontend_out* o, int64_t* totals, void* stream) {
    return frontend_device(pl, d_pcm, d_offsets, h_off, n_utt, o, totals, stream);
}

int dspfe_frontend_f32(dspfe_frontend_plan* pl, const float* d_pcm, const int64_t* d_offsets, const int64_t* h_off, int32_t n_utt,
                       const dspfe_frontend_out* o, int64_t* totals, void* stream) {
    return frontend_device(pl, d_pcm, d_offsets, h_off, n_utt, o, totals, stream);
}

int dspfe_frontend_host(dspfe_frontend_plan* pl, const int16_t* h_pcm, const int64_t* h_off, int32_t n_utt,
                        const dspfe_frontend_out* o, int64_t* totals) {
    return frontend_host(pl, h_pcm, h_off, n_utt, o, totals);
}

int dspfe_frontend_host_f32(dspfe_frontend_plan* pl, const float* h_pcm, const int64_t* h_off, int32_t n_utt,
                            const dspfe_frontend_out* o, int64_t* totals) {
    return frontend_host(pl, h_pcm, h_off, n_utt, o, totals);
}

/* ---- per-kernel timing ---- */
int dspfe_timing_begin(void* stream) {
    StageTimer& t = g_timer;
    t.clear_marks();
    CUDA_TRY(t.ensure_start());
    t.stream = (cudaStream_t)stream;
    CUDA_TRY(cudaEventRecord(t.start, t.stream));
    t.on = true;
    return DSPFE_OK;
}

int dspfe_timing_end(char* names, float* ms, int32_t cap, int32_t* n) {
    StageTimer& t = g_timer;
    if (!t.on) return fail(DSPFE_ERR_INVALID_ARG, "dspfe_timing_begin was not called");
    t.on = false;
    CUDA_TRY(cudaStreamSynchronize(t.stream));
    if (n) *n = (int32_t)t.marks.size();
    cudaEvent_t prev = t.start;
    for (size_t i = 0; i < t.marks.size(); ++i) {
        if ((int32_t)i < cap && names && ms) {
            float v = 0.f;
            CUDA_TRY(cudaEventElapsedTime(&v, prev, t.marks[i].second));
            ms[i] = v;
            std::strncpy(names + 48 * i, t.marks[i].first, 47);
            names[48 * i + 47] = 0;
        }
        prev = t.marks[i].second;
    }
    t.clear_marks();
    return DSPFE_OK;
}

int64_t dspfe_launch_count(void) { return g_timer.launches; }

}  // extern "C"
