// Small single-purpose kernels behind the reference's helper functions (include/dspfe.h, "helpers").
// They exist so that every arithmetic entry point of the drop-in `features` package runs on the GPU; none
// of them is on the throughput path (the fused kernels never materialise frames).  float64 where the
// reference result is float64 and cheap to reproduce exactly (framing, pre-emphasis, row statistics).
#include <vector>

#include "abi_common.h"
#include "dspfe_types.h"
#include "np_pairwise.h"
#include "pitch_tables.h"

using namespace dspfe;

namespace {

// framesig (sigproc.py:66-98): zero-padded overlapping frames times the window
__global__ void frames_kernel(const double* sig, int64_t n, int frame_len, int frame_step, const double* win, int64_t nframes, double* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nframes * frame_len) return;
    const int64_t f = i / frame_len;
    const int k = (int)(i - f * frame_len);
    const int64_t s = f * frame_step + k;
    const double v = s < n ? sig[s] : 0.0;
    out[i] = win ? v * win[k] : v;
}

// preemphasis (sigproc.py:178-185)
__global__ void preemph_kernel(const double* x, int64_t n, double coeff, double* y) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    y[i] = i == 0 ? x[0] : __dsub_rn(x[i], __dmul_rn(coeff, x[i - 1]));   // product rounded first, as NumPy does (no FMA contraction): bit-exact
}

// numpy's pairwise sum for any n (np_pairwise.h), evaluated without recursion (explicit stack of pending right halves).
// The lambdas capture by value: the flags stay loop invariants of the block sum, which the compiler specialises the loop on.
__device__ double pairwise_block_f64(const double* a, int n, bool absval, bool sq) {
    auto f = [absval, sq](double v) { return sq ? v * v : (absval ? fabs(v) : v); };
    return pairwise_block([f, a](int i) { return f(a[i]); }, n);
}
__device__ double np_sum_any(const double* a, int n, bool absval, bool sq) {
    return pairwise_walk(a, n, [absval, sq](const double* p, int m) { return pairwise_block_f64(p, m, absval, sq); });
}

// get_amplitude (endpoint.py:109-126, window='square'): mean |x| (or x^2) per frame, numpy summation order
__global__ void row_amp_kernel(const double* frames, int64_t nrows, int len, int use_sq, double* out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    const double s = np_sum_any(frames + r * len, len, true, use_sq == 1);
    out[r] = use_sq == 2 ? s : s / (double)len;
}

// get_amplitude with a window (endpoint.py:118-125): mean over n of np.convolve(|x| or x^2, w, 'same')[n] equals
// (1/len) * sum_m v[m] * c[m], where c[m] is the sum of the window taps that the 'same' crop lets sample m meet
__global__ void row_weighted_amp_kernel(const double* frames, int64_t nrows, int len, const double* c, int use_sq, double* out) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (r >= nrows) return;
    const double* x = frames + r * len;
    double acc = 0.0;
    for (int m = lane; m < len; m += 32) { const double v = use_sq ? x[m] * x[m] : fabs(x[m]); acc += v * c[m]; }
#pragma unroll
    for (int k = 16; k >= 1; k >>= 1)
        acc += __hiloint2double(__shfl_xor_sync(0xffffffffu, __double2hiint(acc), k), __shfl_xor_sync(0xffffffffu, __double2loint(acc), k));
    if (lane == 0) out[r] = acc / (double)len;
}

// get_zcr (endpoint.py:182-198)
__global__ void row_zcr_kernel(const double* frames, int64_t nrows, int len, int64_t* out) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    const double* x = frames + r * len;
    int64_t c = 0;
    for (int i = 0; i + 1 < len; ++i) c += (x[i] * x[i + 1] < 0.0) ? 1 : 0;
    out[r] = c;
}

// delta (base.py:70-79) on an arbitrary [F, C] float32 matrix
__global__ void delta_kernel(const float* in, int64_t F, int C, int N, float scale, float* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= F * C) return;
    const int64_t t = i / C;
    const int c = (int)(i - t * C);
    float acc = 0.f;
    for (int n = 1; n <= N; ++n) {
        const int64_t hi = t + n > F - 1 ? F - 1 : t + n, lo = t - n < 0 ? 0 : t - n;
        acc = fmaf((float)n, in[hi * C + c] - in[lo * C + c], acc);
    }
    out[i] = acc * scale;
}

// window (sigproc.py:22-46): y[n] = sum_{m<=n} x[m] h[n-m], complex float64 taps, output truncated to len(x)
__global__ void fir_window_kernel(const double* x, int n, const double* hr, const double* hi, double* y) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double sr = 0.0, si = 0.0;
    for (int m = 0; m <= i; ++m) { const double v = x[m]; sr += v * hr[i - m]; si += v * hi[i - m]; }
    y[2 * i] = sr; y[2 * i + 1] = si;
}

// acr (sigproc.py:48-53): lagged products, then numpy's pairwise sum and the unbiased normalisation
__global__ void lag_products_kernel(const double* x, int len, int n, double* prod) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < len - n) prod[i] = x[i] * x[i + n];
}
__global__ void acr_finish_kernel(const double* prod, int count, int len, int n, double* out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) out[0] = np_sum_any(prod, count, false, false) / (double)(len - n);
}

// Caller-side batching epilogue of model.py (:75-88 CMVN of the static block, :35-50 pad / truncate to T frames,
// :131-135 [T, B, 3C] layout): one CTA per utterance.  Column statistics over ALL frames of the utterance in float64;
// sklearn.preprocessing.scale semantics (population std, a constant column is only centred).
constexpr int kBatchThreads = 128;
__global__ void __launch_bounds__(kBatchThreads) cmvn_pad_kernel(const float* feat, const int64_t* frame_off, int n_utt, int C, int T,
                                                                float* out, int32_t* len0) {
    __shared__ double s_sum[kBatchThreads], s_sq[kBatchThreads];
    __shared__ float s_mean[kMaxNumcep], s_inv[kMaxNumcep];
    const int u = blockIdx.x, tid = threadIdx.x;
    const int64_t r0 = frame_off[u];
    const int F = (int)(frame_off[u + 1] - r0);
    const int W = 3 * C;
    const int per = kBatchThreads / C;               // row lanes per column
    const int c = tid % C, rl = tid / C;
    double sm = 0.0, sq = 0.0;
    if (rl < per)
        for (int t = rl; t < F; t += per) { const double v = feat[(r0 + t) * W + c]; sm += v; sq += v * v; }
    s_sum[tid] = sm; s_sq[tid] = sq;
    __syncthreads();
    if (tid < C) {
        double a = 0.0, b = 0.0;
        for (int k = 0; k < per; ++k) { a += s_sum[tid + k * C]; b += s_sq[tid + k * C]; }
        const double mean = F > 0 ? a / F : 0.0;
        double var = F > 0 ? b / F - mean * mean : 0.0;
        if (var < 0.0) var = 0.0;
        double sd = sqrt(var);
        if (sd < 10.0 * 2.220446049250313e-16 * fmax(1.0, fabs(mean))) sd = 1.0;   // constant column: centre only
        s_mean[tid] = (float)mean; s_inv[tid] = (float)(1.0 / sd);
    }
    __syncthreads();
    const int n = (F < T ? F : T) * W;
    for (int i = tid; i < T * W; i += kBatchThreads) {
        const int t = i / W, col = i - t * W;
        float v = 0.f;
        if (i < n) {
            v = feat[(r0 + t) * W + col];
            if (col < C) v = (v - s_mean[col]) * s_inv[col];
        }
        out[((int64_t)t * n_utt + u) * W + col] = v;
    }
    if (tid == 0 && len0) len0[u] = F < T ? F : T;
}

unsigned grid_for(int64_t n, int bs) { return (unsigned)((n + bs - 1) / bs); }

}  // namespace

extern "C" {

int dspfe_frames_f64(const double* d_sig, int64_t n, int32_t frame_len, int32_t frame_step, const double* d_win,
                     double* d_out, int64_t n_frames, void* stream) {
    if (!d_out || frame_len < 1 || frame_step < 1 || n < 0 || (!d_sig && n > 0)) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_frames != num_frames(n, frame_len, frame_step)) return fail(DSPFE_ERR_INVALID_ARG, "n_frames must equal dspfe_num_frames()");
    cudaStream_t st = (cudaStream_t)stream;
    frames_kernel<<<grid_for(n_frames * frame_len, 256), 256, 0, st>>>(d_sig, n, frame_len, frame_step, d_win, n_frames, d_out);
    LAUNCH_CHECK("frames_kernel", st);
    return DSPFE_OK;
}

int dspfe_preemphasis_f64(const double* d_x, int64_t n, double coeff, double* d_y, void* stream) {
    if (n < 0 || (n > 0 && (!d_x || !d_y))) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n == 0) return DSPFE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    preemph_kernel<<<grid_for(n, 256), 256, 0, st>>>(d_x, n, coeff, d_y);
    LAUNCH_CHECK("preemph_kernel", st);
    return DSPFE_OK;
}

int dspfe_row_amplitude_f64(const double* d_frames, int64_t n_rows, int32_t len, int32_t use_sq, double* d_out, void* stream) {
    if (n_rows < 0 || len < 1 || (n_rows > 0 && (!d_frames || !d_out))) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_rows == 0) return DSPFE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    row_amp_kernel<<<grid_for(n_rows, 128), 128, 0, st>>>(d_frames, n_rows, len, use_sq, d_out);
    LAUNCH_CHECK("row_amp_kernel", st);
    return DSPFE_OK;
}

int dspfe_row_windowed_amplitude_f64(const double* d_frames, int64_t n_rows, int32_t len, const double* h_window, int32_t win_len,
                                     int32_t use_sq, double* d_out, void* stream) {
    if (n_rows < 0 || len < 1 || win_len < 1 || !h_window || (n_rows > 0 && (!d_frames || !d_out))) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_rows == 0) return DSPFE_OK;
    // np.convolve(v, w, 'same') with len(v) = N, len(w) = M: out[n] = full[n + off], off = (min(N,M) - 1) / 2, full[k] = sum_m v[m] w[k-m]
    const int N = len, M = win_len, off = ((N < M ? N : M) - 1) / 2;
    std::vector<double> pre((size_t)M + 1, 0.0), c((size_t)N);
    for (int k = 0; k < M; ++k) pre[k + 1] = pre[k] + h_window[k];
    for (int m = 0; m < N; ++m) {           // taps j = n + off - m with n in [0, max(N,M)) cropped to N outputs... 'same' returns max(N,M) samples
        const int L = N > M ? N : M;
        int lo = off - m, hi = L - 1 + off - m;      // j range over n = 0..L-1
        if (lo < 0) lo = 0;
        if (hi > M - 1) hi = M - 1;
        c[m] = hi >= lo ? pre[hi + 1] - pre[lo] : 0.0;
    }
    cudaStream_t st = (cudaStream_t)stream;
    StreamTemp<double> d_c;
    CUDA_TRY(d_c.alloc(N, st));
    CUDA_TRY(cudaMemcpyAsync(d_c.get(), c.data(), (size_t)N * sizeof(double), cudaMemcpyHostToDevice, st));
    row_weighted_amp_kernel<<<grid_for(n_rows, 4), 128, 0, st>>>(d_frames, n_rows, len, d_c.get(), use_sq, d_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(DSPFE_ERR_CUDA, std::string("row_weighted_amp_kernel: ") + cudaGetErrorString(e));
    return DSPFE_OK;
}

int dspfe_row_zcr_f64(const double* d_frames, int64_t n_rows, int32_t len, int64_t* d_out, void* stream) {
    if (n_rows < 0 || len < 1 || (n_rows > 0 && (!d_frames || !d_out))) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_rows == 0) return DSPFE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    row_zcr_kernel<<<grid_for(n_rows, 128), 128, 0, st>>>(d_frames, n_rows, len, d_out);
    LAUNCH_CHECK("row_zcr_kernel", st);
    return DSPFE_OK;
}

int dspfe_delta_f32(const float* d_in, int64_t n_frames, int32_t n_cols, int32_t N, float* d_out, void* stream) {
    if (N < 1) return fail(DSPFE_ERR_INVALID_ARG, "N must be an integer >= 1");
    if (n_frames < 0 || n_cols < 1 || (n_frames > 0 && (!d_in || !d_out))) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n_frames == 0) return DSPFE_OK;
    int den = 0;
    for (int i = 1; i <= N; ++i) den += i * i;
    cudaStream_t st = (cudaStream_t)stream;
    delta_kernel<<<grid_for(n_frames * n_cols, 256), 256, 0, st>>>(d_in, n_frames, n_cols, N, (float)(1.0 / (2.0 * den)), d_out);
    LAUNCH_CHECK("delta_kernel", st);
    return DSPFE_OK;
}

int dspfe_cmvn_pad_batch(const float* d_feat, const int64_t* d_frame_off, int32_t n_utt, int32_t numcep, int32_t T, float* d_out,
                         int32_t* d_len0, void* stream) {
    if (!d_feat || !d_frame_off || !d_out || n_utt < 0 || T < 1) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (numcep < 1 || numcep > kMaxNumcep) return fail(DSPFE_ERR_UNSUPPORTED, "numcep outside 1..16");
    if (n_utt == 0) return DSPFE_OK;
    cudaStream_t st = (cudaStream_t)stream;
    cmvn_pad_kernel<<<(unsigned)n_utt, kBatchThreads, 0, st>>>(d_feat, d_frame_off, n_utt, numcep, T, d_out, d_len0);
    LAUNCH_CHECK("cmvn_pad_kernel", st);
    return DSPFE_OK;
}

int dspfe_fir_window_f64(const double* d_x, int32_t n, double rate, double low_freq, double high_freq, int32_t hamming,
                         double* d_y, void* stream) {
    if (n < 1 || !d_x || !d_y || !(rate > 0)) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    if (n > 8192) return fail(DSPFE_ERR_UNSUPPORTED, "window() signals longer than 8192 samples are not built");
    std::vector<double> hr, hi;
    fir_taps(n, rate, low_freq, high_freq, hamming != 0, hr, hi);
    cudaStream_t st = (cudaStream_t)stream;
    StreamTemp<double> d_h;
    CUDA_TRY(d_h.alloc(2 * (int64_t)n, st));
    CUDA_TRY(cudaMemcpyAsync(d_h.get(), hr.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_h.get() + n, hi.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    fir_window_kernel<<<grid_for(n, 128), 128, 0, st>>>(d_x, n, d_h.get(), d_h.get() + n, d_y);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(DSPFE_ERR_CUDA, std::string("fir_window_kernel: ") + cudaGetErrorString(e));
    return DSPFE_OK;
}

int dspfe_acr_f64(const double* d_frame, int32_t len, int32_t n, double* d_out, void* stream) {
    if (!d_frame || !d_out || len < 1 || n < 0 || n >= len) return fail(DSPFE_ERR_INVALID_ARG, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    StreamTemp<double> d_prod;
    CUDA_TRY(d_prod.alloc(len - n, st));
    lag_products_kernel<<<grid_for(len - n, 256), 256, 0, st>>>(d_frame, len, n, d_prod.get());
    acr_finish_kernel<<<1, 32, 0, st>>>(d_prod.get(), len - n, len, n, d_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(DSPFE_ERR_CUDA, std::string("acr kernels: ") + cudaGetErrorString(e));
    return DSPFE_OK;
}

}  // extern "C"
