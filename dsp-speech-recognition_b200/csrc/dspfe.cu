// libdspfe.so — C ABI (include/dspfe.h) over the sm_100a kernels.  No CPU fallback anywhere in
// this file: every compute entry point launches CUDA kernels or fails with DSPFE_ERR_CUDA.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "abi_common.h"
#include "mfcc_kernel.cuh"
#include "mfcc_long_kernel.cuh"
#include "mfcc_long_tables.h"
#include "mfcc_tables.h"
#include "pitch_tables.h"
#include "prep_kernel.cuh"

using namespace dspfe;

namespace {

template <bool HAS_WIN, int NFULL, bool F32IN, int MODE = 0>
__global__ void __launch_bounds__(kMfccThreads, 4) mfcc_delta_kernel(const __grid_constant__ MfccParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    mfcc_cta<HAS_WIN, NFULL, F32IN, MODE>(p, smem);
}

// K1T: nfft = 1536 for frames of at most 512 samples (model.py:74 at 16 kHz) on K1's tile structure
template <bool HAS_WIN, int NFULL, bool F32IN, bool LONG = false>
__global__ void __launch_bounds__(kMfccThreads, LONG ? 2 : 3) mfcc_tri_kernel(const __grid_constant__ MfccParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    mfcc_cta<HAS_WIN, NFULL, F32IN, 0, true, LONG>(p, smem);
}

// K1L: long frames under nfft = 1536, a frame pair per warp; then delta / delta-delta over the cepstra
template <int NFFT>
__global__ void __launch_bounds__(32 * kLongWarps, 3) mfcc_long_kernel(const __grid_constant__ MfccLongParams p) {
    extern __shared__ __align__(16) unsigned char smem[];
    float2* tws = reinterpret_cast<float2*>(smem);
    const int64_t total = p.frame_off[p.n_utt] < p.max_frames ? p.frame_off[p.n_utt] : p.max_frames;
    if (2 * (int64_t)blockIdx.x * kLongWarps >= total) return;
    for (int i = threadIdx.x; i < kLtW1536 / 2; i += blockDim.x) tws[i] = reinterpret_cast<const float2*>(p.tab)[i];
    __syncthreads();
    const int w = threadIdx.x >> 5;
    const int64_t g0 = 2 * ((int64_t)blockIdx.x * kLongWarps + w);
    if (g0 >= total) return;
    mfcc_long_pair<NFFT>(p, g0, total, smem + kLtW1536 * 4 + w * p.warp_smem, tws, tws + kLtW32 / 2);
}
// delta + delta-delta over per-utterance cepstra (base.py:70-79 twice, model.py:76-77), one CTA per utterance: thread = (row of a
// block of 8, column).  Pass 1 writes the static and delta columns, pass 2 reads the deltas back (edge-clamped on the DELTA
// array, SURVEY Appendix A-5) for the delta-deltas: 4N + 1 loads per output row instead of the 4N^2 + 2N of the one-pass form
// (delta_batch_thread, kept for the CPU emulator), and no per-thread utterance search.  Same arithmetic, same order.
__global__ void __launch_bounds__(128) delta_batch_kernel(const float* mf, const int64_t* frame_off, int n_utt, int C, int N, float scale, int64_t max_frames, float* out) {
    const int u = blockIdx.x;
    const int64_t r0 = frame_off[u];
    const int F = (int)(frame_off[u + 1] - r0);                                   // clamps use the utterance's own frame count
    const int Fw = (int)(r0 + F <= max_frames ? F : (max_frames > r0 ? max_frames - r0 : 0));   // rows that fit the output
    const int c = threadIdx.x & 15, r = threadIdx.x >> 4;
    if (Fw <= 0) return;
    const int W = 3 * C;
    auto clampf = [&](int a) { return a < 0 ? 0 : (a > F - 1 ? F - 1 : a); };
    if (c < C) {
        for (int t = r; t < Fw; t += 8) {
            float acc = 0.f;
            for (int n = 1; n <= N; ++n) acc = dsp_fmaf((float)n, mf[(r0 + clampf(t + n)) * C + c] - mf[(r0 + clampf(t - n)) * C + c], acc);
            float* o = out + (r0 + t) * W;
            o[c] = mf[(r0 + t) * C + c];
            o[C + c] = acc * scale;
        }
    }
    __syncthreads();
    if (c < C) {
        for (int t = r; t < Fw; t += 8) {
            float acc = 0.f;
            for (int n = 1; n <= N; ++n) acc = dsp_fmaf((float)n, out[(r0 + clampf(t + n)) * W + C + c] - out[(r0 + clampf(t - n)) * W + C + c], acc);
            out[(r0 + t) * W + 2 * C + c] = acc * scale;
        }
    }
}

typedef void (*mfcc_kernel_t)(const MfccParams);
// specialisations: rectangular / windowed x frame_len/32 in {12 (25 ms @16 kHz), 15 (30 ms @16 kHz), generic}
mfcc_kernel_t pick_kernel(bool has_win, int frame_len, bool f32, int mode = 0) {
    const int nfull = frame_len >> 5;
    if (mode == 1) return has_win ? mfcc_delta_kernel<true, -1, true, 1> : mfcc_delta_kernel<false, -1, true, 1>;   // taps: float32 input only
    if (mode == 2) return has_win ? mfcc_delta_kernel<true, -1, true, 2> : mfcc_delta_kernel<false, -1, true, 2>;
    if (f32) return has_win ? mfcc_delta_kernel<true, -1, true> : mfcc_delta_kernel<false, -1, true>;
    if (has_win) {
        if (nfull == 12) return mfcc_delta_kernel<true, 12, false>;
        if (nfull == 15) return mfcc_delta_kernel<true, 15, false>;
        return mfcc_delta_kernel<true, -1, false>;
    }
    if (nfull == 12) return mfcc_delta_kernel<false, 12, false>;
    if (nfull == 15) return mfcc_delta_kernel<false, 15, false>;
    return mfcc_delta_kernel<false, -1, false>;
}

mfcc_kernel_t pick_tri_kernel(bool has_win, int frame_len, bool f32) {
    if (frame_len > 512) {   // K1T LONG: 30 ms frames at 22.05 / 44.1 / 48 kHz
        if (f32) return has_win ? mfcc_tri_kernel<true, -1, true, true> : mfcc_tri_kernel<false, -1, true, true>;
        return has_win ? mfcc_tri_kernel<true, -1, false, true> : mfcc_tri_kernel<false, -1, false, true>;
    }
    if (f32) return has_win ? mfcc_tri_kernel<true, -1, true> : mfcc_tri_kernel<false, -1, true>;
    if (has_win) return (frame_len >> 5) == 15 ? mfcc_tri_kernel<true, 15, false> : mfcc_tri_kernel<true, -1, false>;
    return mfcc_tri_kernel<false, -1, false>;
}

MfccConfig to_config(const dspfe_mfcc_params& q) {
    MfccConfig c;
    c.samplerate = q.samplerate; c.frame_len = q.frame_len; c.frame_step = q.frame_step; c.nfft = q.nfft;
    c.count_len = q.frame_len;
    if (q.nfft > 0 && q.frame_len > q.nfft) c.frame_len = q.nfft;   // frames longer than nfft: truncated for the transform, as the reference does
    c.nfilt = q.nfilt; c.numcep = q.numcep; c.ceplifter = q.ceplifter; c.append_energy = q.append_energy;
    c.delta_n = q.delta_n; c.seg_frames = q.seg_frames > 0 ? q.seg_frames : 256;
    c.preemph = q.preemph; c.lowfreq = q.lowfreq; c.highfreq = q.highfreq;
    if (q.window) c.window.assign(q.window, q.window + (c.frame_len > 0 ? c.frame_len : 0));   // (the first nfft entries of a longer window)
    return c;
}

// Per-stream scratch for one in-flight batch.
struct Workspace {
    DeviceArray<float> cep;     // K1L: static cepstra [rows, numcep] between the two kernels
    DeviceArray<int64_t> seg_start; DeviceArray<int32_t> seg_len; DeviceArray<int64_t> frame_off;
    DeviceArray<int32_t> tile_off; DeviceArray<Tile> tiles; DeviceArray<int32_t> ntiles;
    int ensure(int64_t n_utt, int64_t n_tiles) {
        int rc = seg_start.reserve(n_utt + 1);
        if (!rc) rc = seg_len.reserve(n_utt + 1);
        if (!rc) rc = frame_off.reserve(n_utt + 1);
        if (!rc) rc = tile_off.reserve(n_utt + 1);
        if (!rc) rc = tiles.reserve(n_tiles);
        if (!rc) rc = ntiles.reserve(1);
        return rc;
    }
};

constexpr int kSlots = 3;
struct HostSlot {
    Stream stream;
    Workspace ws;
    DeviceArray<int16_t> d_pcm;
    DeviceArray<int64_t> d_off; PinnedArray<int64_t> h_off;
    DeviceArray<float> d_out;
    DeviceArray<int64_t> d_frame_off;
};

}  // namespace

struct dspfe_plan {
    MfccConfig cfg;
    MfccParams layout;          // scalars + offsets filled by build_mfcc_tables; pointers filled per call
    MfccParams layout_f32;      // same for float32 input samples (larger raw staging area)
    DeviceArray<float> d_tables;
    bool has_win = false;
    mfcc_kernel_t kernel = nullptr, kernel_f32 = nullptr, kernel_fbank = nullptr, kernel_spec = nullptr;
    Workspace ws;
    HostSlot slots[kSlots];
    int width = 0;              // 3 * numcep
    bool is_long = false;       // K1L: nfft other than 512, or nfft = 512 with an odd hop
    DeviceArray<float> d_long_tab;
    std::vector<float> h_long_tab;   // host copy: the mel edges travel as kernel parameters
};

namespace {

int launch_mfcc(dspfe_plan* pl, Workspace& ws, const void* d_pcm, bool f32, int64_t total_samples, const int64_t* d_offsets,
                const int32_t* d_trim, int32_t n_utt, float* d_out, int64_t* d_frame_off, cudaStream_t st, int mode = 0, int spec_kind = 0) {
    const int64_t max_tiles = mfcc_max_tiles(total_samples, n_utt, pl->cfg.frame_step, pl->cfg.seg_frames);
    if (max_tiles > 0x7fffffff) return fail(DSPFE_ERR_INVALID_ARG, "batch too large for one launch");
    int rc = ws.ensure(n_utt, max_tiles);
    if (rc) return rc;
    PrepParams pp;
    pp.offsets = d_offsets; pp.trim = d_trim; pp.n_utt = n_utt;
    pp.frame_len = pl->cfg.count_len; pp.frame_step = pl->cfg.frame_step; pp.seg_frames = pl->cfg.seg_frames;
    pp.seg_start = ws.seg_start.get(); pp.seg_len = ws.seg_len.get(); pp.frame_off = d_frame_off ? d_frame_off : ws.frame_off.get();
    pp.tile_off = ws.tile_off.get(); pp.tiles = ws.tiles.get(); pp.ntiles = ws.ntiles.get(); pp.max_tiles = (int)max_tiles;
    prep_kernel<<<1, kPrepThreads, 0, st>>>(pp);
    LAUNCH_CHECK("prep_kernel", st);

    if (pl->is_long || (mode != 0 && pl->d_long_tab.get())) {
        const int64_t rows = dspfe_rows_bound(pl, total_samples, n_utt);
        if (mode == 0) { rc = ws.cep.reserve(rows * pl->cfg.numcep); if (rc) return rc; }
        MfccLongParams lp;
        lp.pcm = d_pcm; lp.in_f32 = f32 ? 1 : 0; lp.seg_start = ws.seg_start.get(); lp.seg_len = ws.seg_len.get(); lp.frame_off = pp.frame_off; lp.n_utt = n_utt;
        lp.frame_len = pl->cfg.frame_len; lp.frame_step = pl->cfg.frame_step; lp.nfilt = pl->cfg.nfilt; lp.numcep = pl->cfg.numcep;
        lp.append_energy = pl->cfg.append_energy; lp.preemph = (float)pl->cfg.preemph; lp.tab = pl->d_long_tab.get(); lp.mfcc = mode == 0 ? ws.cep.get() : d_out; lp.max_frames = rows;
        long_fill_size_params(lp, pl->cfg.nfft, mode, spec_kind);
        long_fill_mel_params(lp, pl->h_long_tab.data());
        const unsigned lgrid = (unsigned)((rows + 2 * kLongWarps - 1) / (2 * kLongWarps));
        if (pl->cfg.nfft == kLongNfft) mfcc_long_kernel<kLongNfft><<<lgrid, 32 * kLongWarps, long_cta_smem(kLongNfft), st>>>(lp);
        else mfcc_long_kernel<0><<<lgrid, 32 * kLongWarps, long_cta_smem(pl->cfg.nfft), st>>>(lp);
        LAUNCH_CHECK("mfcc_long_kernel", st);
        if (mode != 0) return DSPFE_OK;
        int den = 0; for (int i = 1; i <= pl->cfg.delta_n; ++i) den += i * i;
        delta_batch_kernel<<<(unsigned)n_utt, 128, 0, st>>>(ws.cep.get(), pp.frame_off, n_utt, pl->cfg.numcep, pl->cfg.delta_n,
                                                                                          (float)(1.0 / (2.0 * den)), rows, d_out);
        LAUNCH_CHECK("delta_batch_kernel", st);
        return DSPFE_OK;
    }
    MfccParams mp = f32 ? pl->layout_f32 : pl->layout;
    mp.pcm = d_pcm; mp.total_samples = total_samples; mp.seg_start = ws.seg_start.get(); mp.seg_len = ws.seg_len.get();
    mp.frame_off = pp.frame_off; mp.tiles = ws.tiles.get(); mp.ntiles = ws.ntiles.get(); mp.tables = pl->d_tables.get(); mp.out = d_out;
    mp.spec_kind = spec_kind;
    mfcc_kernel_t kern = mode == 1 ? pl->kernel_fbank : mode == 2 ? pl->kernel_spec : (f32 ? pl->kernel_f32 : pl->kernel);
    kern<<<(unsigned)max_tiles, kMfccThreads, mp.sm_total, st>>>(mp);
    LAUNCH_CHECK("mfcc_delta_kernel", st);
    return DSPFE_OK;
}

// the device forms: mode 0 MFCC + delta + delta-delta, 1 the filterbank tap, 2 the spectrum tap of the given kind
int mfcc_device(dspfe_plan* pl, const void* d_pcm, bool f32, int64_t total_samples, const int64_t* d_offsets, const int32_t* d_trim,
                int32_t n_utt, float* d_out, int64_t max_rows, int64_t* d_frame_off, void* stream, int mode = 0, int kind = 0) {
    if (int rc = check_batch(pl && d_offsets && d_out && kind >= 0 && kind <= 2, n_utt, total_samples, d_pcm)) return rc;
    if (n_utt == 0) return DSPFE_OK;
    if (max_rows < dspfe_rows_bound(pl, total_samples, n_utt))
        return fail(DSPFE_ERR_INVALID_ARG, "d_out capacity (max_rows) is below dspfe_rows_bound()");
    return launch_mfcc(pl, pl->ws, d_pcm, f32, total_samples, d_offsets, d_trim, n_utt, d_out, d_frame_off, (cudaStream_t)stream, mode, kind);
}

}  // namespace

extern "C" {

const char* dspfe_version(void) { return "dspfe 0.1 (sm_100a)"; }
const char* dspfe_last_error(void) { return g_err.c_str(); }

void dspfe_mfcc_params_default(dspfe_mfcc_params* p) {
    if (!p) return;
    std::memset(p, 0, sizeof(*p));
    p->samplerate = 16000; p->frame_len = 400; p->frame_step = 160; p->nfft = 512; p->nfilt = 26; p->numcep = 13;
    p->ceplifter = 22; p->append_energy = 1; p->delta_n = 2; p->seg_frames = 0; p->preemph = 0.97;
    p->lowfreq = 0.0; p->highfreq = 0.0; p->window = nullptr;
}

int64_t dspfe_num_frames(int64_t n_samples, int32_t frame_len, int32_t frame_step) {
    if (frame_len < 1 || frame_step < 1) return -1;
    return num_frames(n_samples, frame_len, frame_step);
}

int dspfe_mfcc_tables_host(const dspfe_mfcc_params* p, float* blob, int32_t cap, int32_t* n, double* mel_edges) {
    if (!p || !n) return fail(DSPFE_ERR_INVALID_ARG, "null argument");
    MfccConfig c = to_config(*p);
    MfccParams lay{};
    std::string err;
    std::vector<float> b = build_mfcc_tables(c, lay, err);
    if (!err.empty()) return fail(DSPFE_ERR_UNSUPPORTED, err);
    *n = (int32_t)b.size();
    if (blob) {
        if (cap < *n) return fail(DSPFE_ERR_INVALID_ARG, "blob capacity too small");
        std::memcpy(blob, b.data(), b.size() * sizeof(float));
    }
    if (mel_edges) {
        std::vector<double> e = mel_bin_edges(c);
        std::memcpy(mel_edges, e.data(), e.size() * sizeof(double));
    }
    return DSPFE_OK;
}

int dspfe_plan_create(const dspfe_mfcc_params* p, dspfe_plan** plan) {
    if (!p || !plan) return fail(DSPFE_ERR_INVALID_ARG, "null argument");
    *plan = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(DSPFE_ERR_CUDA, "no CUDA device: libdspfe has no CPU fallback");
    dspfe_plan* pl = new (std::nothrow) dspfe_plan();
    if (!pl) return fail(DSPFE_ERR_NOMEM, "out of host memory");
    pl->cfg = to_config(*p);
    std::memset(&pl->layout, 0, sizeof(pl->layout));
    std::string err;
    // K1 / K1T take nfft = 512 / 1536 at any hop; every other size (and gaps between frames) goes to the general kernel K1L
    const bool tiled = (pl->cfg.nfft == kNfft || pl->cfg.nfft == kTriNfft) &&
                       pl->cfg.frame_step <= pl->cfg.count_len;     // (gaps between frames, winstep > winlen: the general kernel)
    if (!tiled || pl->cfg.nfft != kNfft) {   // (a K1T plan keeps the general kernel for its filterbank / spectrum taps)
        err = mfcc_long_config_check(pl->cfg);
        if (!err.empty()) { delete pl; return fail(DSPFE_ERR_UNSUPPORTED, err); }
        pl->is_long = !tiled; pl->has_win = !pl->cfg.window.empty(); pl->width = 3 * pl->cfg.numcep;
        const std::vector<float> t = build_long_tables(pl->cfg);
        pl->h_long_tab = t;
        if (int rc = pl->d_long_tab.reserve(t.size())) { delete pl; return rc; }
        cudaError_t e = cudaMemcpy(pl->d_long_tab.get(), t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(mfcc_long_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, long_cta_smem(kLongMaxNfft));
        if (e == cudaSuccess) e = cudaFuncSetAttribute(mfcc_long_kernel<kLongNfft>, cudaFuncAttributeMaxDynamicSharedMemorySize, long_cta_smem(kLongNfft));
        if (e != cudaSuccess) { delete pl; return fail(DSPFE_ERR_CUDA, cudaGetErrorString(e)); }
        if (!tiled) { *plan = pl; return DSPFE_OK; }
    }
    std::vector<float> blob = build_mfcc_tables(pl->cfg, pl->layout, err);
    if (err.empty()) { std::memset(&pl->layout_f32, 0, sizeof(pl->layout_f32)); build_mfcc_tables(pl->cfg, pl->layout_f32, err, true); }
    if (!err.empty() && pl->d_long_tab.get()) {   // e.g. a chunk of 16 long frames with a long hop does not fit shared memory: the general kernel takes it
        pl->is_long = true; *plan = pl; return DSPFE_OK;
    }
    if (!err.empty()) { delete pl; return fail(DSPFE_ERR_UNSUPPORTED, err); }
    pl->has_win = !pl->cfg.window.empty();
    pl->width = 3 * pl->cfg.numcep;
    if (int rc = pl->d_tables.reserve(blob.size())) { delete pl; return rc; }
    cudaError_t e = cudaMemcpy(pl->d_tables.get(), blob.data(), blob.size() * sizeof(float), cudaMemcpyHostToDevice);
    const bool tri = pl->cfg.nfft == kTriNfft;
    pl->kernel = tri ? pick_tri_kernel(pl->has_win, pl->cfg.frame_len, false) : pick_kernel(pl->has_win, pl->cfg.frame_len, false);
    pl->kernel_f32 = tri ? pick_tri_kernel(pl->has_win, pl->cfg.frame_len, true) : pick_kernel(pl->has_win, pl->cfg.frame_len, true);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pl->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, pl->layout.sm_total);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pl->kernel_f32, cudaFuncAttributeMaxDynamicSharedMemorySize, pl->layout_f32.sm_total);
    if (!tri) {
        pl->kernel_fbank = pick_kernel(pl->has_win, pl->cfg.frame_len, true, 1);
        pl->kernel_spec = pick_kernel(pl->has_win, pl->cfg.frame_len, true, 2);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(pl->kernel_fbank, cudaFuncAttributeMaxDynamicSharedMemorySize, pl->layout_f32.sm_total);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(pl->kernel_spec, cudaFuncAttributeMaxDynamicSharedMemorySize, pl->layout_f32.sm_total);
    }
    if (e != cudaSuccess) { delete pl; return fail(DSPFE_ERR_CUDA, cudaGetErrorString(e)); }
    *plan = pl;
    return DSPFE_OK;
}

int dspfe_plan_reserve(dspfe_plan* pl, int64_t max_utt, int64_t max_total_samples) {
    if (!pl || max_utt < 0 || max_total_samples < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    return pl->ws.ensure(max_utt, mfcc_max_tiles(max_total_samples, max_utt, pl->cfg.frame_step, pl->cfg.seg_frames));
}

void dspfe_plan_destroy(dspfe_plan* pl) {
    if (!pl) return;
    delete pl;
}

int dspfe_plan_info(const dspfe_plan* pl, int32_t* smem_bytes, int32_t* ctas_per_sm, int32_t* regs_per_thread) {
    if (!pl) return fail(DSPFE_ERR_INVALID_ARG, "null plan");
    cudaFuncAttributes fa;
    int nb = 0;
    if (pl->is_long) {
        if (pl->cfg.nfft == kLongNfft) {
            CUDA_TRY(cudaFuncGetAttributes(&fa, mfcc_long_kernel<kLongNfft>));
            CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, mfcc_long_kernel<kLongNfft>, 32 * kLongWarps, long_cta_smem(pl->cfg.nfft)));
        } else {
            CUDA_TRY(cudaFuncGetAttributes(&fa, mfcc_long_kernel<0>));
            CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, mfcc_long_kernel<0>, 32 * kLongWarps, long_cta_smem(pl->cfg.nfft)));
        }
        if (smem_bytes) *smem_bytes = long_cta_smem(pl->cfg.nfft);
        if (ctas_per_sm) *ctas_per_sm = nb;
        if (regs_per_thread) *regs_per_thread = fa.numRegs;
        return DSPFE_OK;
    }
    CUDA_TRY(cudaFuncGetAttributes(&fa, pl->kernel));
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, pl->kernel, kMfccThreads, pl->layout.sm_total));
    if (smem_bytes) *smem_bytes = pl->layout.sm_total;
    if (ctas_per_sm) *ctas_per_sm = nb;
    if (regs_per_thread) *regs_per_thread = fa.numRegs;
    return DSPFE_OK;
}

int64_t dspfe_rows_bound(const dspfe_plan* pl, int64_t total_samples, int64_t n_utt) {
    if (!pl) return -1;
    // 1 + ceil((S - L) / step) <= S / step + 1 frames per utterance for abutting or overlapping frames, + 2 when step > L (gaps)
    return total_samples / pl->cfg.frame_step + (pl->cfg.frame_step > pl->cfg.count_len ? 2 : 1) * n_utt;
}

int dspfe_mfcc_delta(dspfe_plan* pl, const int16_t* d_pcm, int64_t total_samples, const int64_t* d_offsets,
                     const int32_t* d_trim, int32_t n_utt, float* d_out, int64_t max_rows, int64_t* d_frame_off,
                     void* stream) {
    return mfcc_device(pl, d_pcm, false, total_samples, d_offsets, d_trim, n_utt, d_out, max_rows, d_frame_off, stream);
}

int dspfe_mfcc_delta_f32(dspfe_plan* pl, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets,
                         const int32_t* d_trim, int32_t n_utt, float* d_out, int64_t max_rows, int64_t* d_frame_off,
                         void* stream) {
    return mfcc_device(pl, d_pcm, true, total_samples, d_offsets, d_trim, n_utt, d_out, max_rows, d_frame_off, stream);
}

int dspfe_fbank_f32(dspfe_plan* pl, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                    float* d_out, int64_t max_rows, int64_t* d_frame_off, void* stream) {
    return mfcc_device(pl, d_pcm, true, total_samples, d_offsets, nullptr, n_utt, d_out, max_rows, d_frame_off, stream, 1);
}

int dspfe_spectrum_f32(dspfe_plan* pl, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                       int32_t kind, float* d_out, int64_t max_rows, int64_t* d_frame_off, void* stream) {
    return mfcc_device(pl, d_pcm, true, total_samples, d_offsets, nullptr, n_utt, d_out, max_rows, d_frame_off, stream, 2, kind);
}

int dspfe_mfcc_delta_host(dspfe_plan* pl, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt, float* h_out,
                          int64_t* h_frame_off) {
    if (int rc = check_host_batch(pl && h_out, h_offsets, n_utt)) return rc;
    if (n_utt == 0) return DSPFE_OK;
    const int flen = pl->cfg.count_len, fstep = pl->cfg.frame_step, width = pl->width;
    // slabs of consecutive utterances: <= kSlabSamples samples each (one oversized utterance = its own slab)
    const int64_t kSlabSamples = 8ll << 20;
    int64_t row = 0;
    int slab = 0;
    int32_t u = 0;
    while (u < n_utt) {
        int32_t u_end = u; int64_t samples = 0, rows = 0;
        while (u_end < n_utt) {
            const int64_t len = h_offsets[u_end + 1] - h_offsets[u_end];
            if (u_end > u && samples + len > kSlabSamples) break;
            samples += len; rows += num_frames(len, flen, fstep);
            if (h_frame_off) h_frame_off[u_end] = row + rows - num_frames(len, flen, fstep);
            ++u_end;
        }
        const int32_t nu = u_end - u;
        HostSlot& s = pl->slots[slab % kSlots];
        CUDA_TRY(s.stream.ensure());
        const cudaStream_t st = s.stream.get();
        CUDA_TRY(cudaStreamSynchronize(st));  // the slot's previous slab has fully drained
        int rc = s.d_pcm.reserve(samples + 8, kSlabSamples + 8);
        if (!rc) rc = s.d_off.reserve(nu + 1, 4096);
        if (!rc) rc = s.d_frame_off.reserve(nu + 1, 4096);
        if (!rc) rc = s.h_off.reserve(nu + 1, 4096);
        if (!rc) rc = s.d_out.reserve(dspfe_rows_bound(pl, samples, nu) * width, (kSlabSamples / fstep + 4096) * width);
        if (rc) return rc;
        const int64_t base = h_offsets[u];
        for (int32_t i = 0; i <= nu; ++i) s.h_off.get()[i] = h_offsets[u + i] - base;
        if (samples > 0)
            CUDA_TRY(cudaMemcpyAsync(s.d_pcm.get(), h_pcm + base, samples * sizeof(int16_t), cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(s.d_off.get(), s.h_off.get(), (nu + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        rc = launch_mfcc(pl, s.ws, s.d_pcm.get(), false, samples, s.d_off.get(), nullptr, nu, s.d_out.get(), s.d_frame_off.get(), st);
        if (rc) return rc;
        CUDA_TRY(cudaMemcpyAsync(h_out + row * width, s.d_out.get(), rows * width * sizeof(float), cudaMemcpyDeviceToHost, st));
        row += rows;
        u = u_end;
        ++slab;
    }
    if (h_frame_off) h_frame_off[n_utt] = row;
    for (auto& s : pl->slots)
        if (s.stream.get()) CUDA_TRY(cudaStreamSynchronize(s.stream.get()));
    return DSPFE_OK;
}

int dspfe_host_alloc(void** p, int64_t bytes) {
    if (!p || bytes < 0) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    CUDA_TRY(cudaHostAlloc(p, (size_t)bytes, cudaHostAllocDefault));
    return DSPFE_OK;
}

int dspfe_host_free(void* p) {
    CUDA_TRY(cudaFreeHost(p));
    return DSPFE_OK;
}

}  // extern "C"
