/* dspfe.h — C ABI of libdspfe.so, the B200 (sm_100a) speech front-end.
 *
 * Drop-in boundary for the PCM -> classifier-features path of AuCson/DSP-Speech-Recognition.
 * The reference has no FFI: its boundary is the Python package `features`
 * (features/__init__.py:1-6).  Each entry point below names the reference function(s) it
 * replaces; the Python package `dsp-speech-recognition_b200/features` binds these with ctypes
 * and re-exposes the reference's own names and signatures (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 (DSPFE_OK) or a negative dspfe_status; dspfe_last_error() gives
 *     the message of the calling thread's last failure;
 *   - `d_` pointers are device memory, `h_` pointers host memory; the caller owns all of them;
 *   - device entry points are asynchronous on `stream` (a cudaStream_t passed as void*) and keep
 *     their workspaces inside the plan: ONE call per plan may be in flight at a time (calls on the
 *     same plan must be ordered on one stream or by events; use one plan per concurrent stream --
 *     dspfe_frontend_host does exactly that with two lanes).  A workspace grows only when a larger
 *     batch than ever before arrives, with cudaFree / cudaMalloc, which synchronises the device
 *     once; dspfe_*_reserve() pre-sizes them so that later calls never allocate;
 *   - a packed ragged batch is int16 PCM `pcm[total_samples]` plus `offsets[n_utt+1]` (int64,
 *     samples); utterance u is pcm[offsets[u] .. offsets[u+1]).  No padding between utterances
 *     is required; `d_pcm` itself must be 16-byte aligned.  The `_f32` entry points take the same
 *     layout with float32 samples.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     DSPFE_ERR_CUDA.
 */
#ifndef DSPFE_H_
#define DSPFE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    DSPFE_OK = 0,
    DSPFE_ERR_INVALID_ARG = -1,   /* null pointer, bad size, misaligned buffer */
    DSPFE_ERR_UNSUPPORTED = -2,   /* parameter combination outside the supported set (no CPU fallback) */
    DSPFE_ERR_CUDA = -3,          /* CUDA runtime error (message has the cudaError string) */
    DSPFE_ERR_NOMEM = -4
} dspfe_status;

typedef struct dspfe_plan dspfe_plan;

/* Parameters of the MFCC (+delta) path.  Field meanings follow reference base.py:8-10 `mfcc(...)`.
 * frame_len / frame_step are in samples: the caller applies round_half_up(winlen*samplerate)
 * (reference sigproc.py:77-78). */
typedef struct {
    int32_t samplerate;      /* 16000 */
    int32_t frame_len;       /* 400  (25 ms) */
    int32_t frame_step;      /* 160  (10 ms) */
    int32_t nfft;            /* 512; built: 32..2048 powers of two and 1536 (model.py:74).  512: the tiled kernel K1; 1536: the tiled
                              * kernel K1T; everything else (and frame_step > frame_len): the general kernel K1L */
    int32_t nfilt;           /* 26 */
    int32_t numcep;          /* 13 */
    int32_t ceplifter;       /* 22 (<= 0 disables, base.py:66-68) */
    int32_t append_energy;   /* 1: c0 := log(frame energy), base.py:15 */
    int32_t delta_n;         /* N of delta(feat, N), base.py:70 */
    int32_t seg_frames;      /* tile length in frames (tuning knob; 0 = default) */
    double preemph;          /* 0.97 */
    double lowfreq;          /* 0 */
    double highfreq;         /* <= 0: samplerate / 2 */
    const double* window;    /* host array [frame_len] = winfunc(frame_len), or NULL for rectangular */
} dspfe_mfcc_params;

const char* dspfe_version(void);
const char* dspfe_last_error(void);

/* Reference defaults (base.py:8-10) with delta_n = 2. */
void dspfe_mfcc_params_default(dspfe_mfcc_params* p);

/* framesig's frame count, reference sigproc.py:79-82. */
int64_t dspfe_num_frames(int64_t n_samples, int32_t frame_len, int32_t frame_step);

/* Host-only: build the kernel's constant tables (no CUDA call).  Writes up to `cap` floats to
 * `blob`, the float count to *n, and the 28 mel bin edges (nfilt+2 doubles) to `mel_edges` if
 * non-null.  Lets CPU-only tests check the tables against the oracle. */
int dspfe_mfcc_tables_host(const dspfe_mfcc_params* p, float* blob, int32_t cap, int32_t* n, double* mel_edges);

/* Plan = parameters + device tables + workspaces on the current CUDA device. */
int dspfe_plan_create(const dspfe_mfcc_params* p, dspfe_plan** plan);
int dspfe_plan_reserve(dspfe_plan* plan, int64_t max_utt, int64_t max_total_samples);
void dspfe_plan_destroy(dspfe_plan* plan);
/* shared-memory bytes per CTA and CTAs per SM of the fused kernel (for reports) */
int dspfe_plan_info(const dspfe_plan* plan, int32_t* smem_bytes, int32_t* ctas_per_sm, int32_t* regs_per_thread);

/* Fused MFCC + delta + delta-delta over a packed ragged batch, everything device-resident.
 * Replaces features.mfcc (base.py:8) followed by features.delta twice (base.py:70; as called in
 * model.py:74-77) for every utterance of the batch.
 *   d_offsets   [n_utt+1] int64 utterance boundaries in samples
 *   d_trim      optional [n_utt,2] int32 (left,right) sample indices inside each utterance, as
 *               produced by dspfe_endpoint(); the utterance is replaced by sig[left:right]
 *               (Python slice semantics, model.py:62); NULL = whole utterances
 *   d_out       [rows, 3*numcep] float32, rows >= total frame count
 *   d_frame_off [n_utt+1] int64, written: first output row of each utterance (last = total rows)
 *   max_rows    capacity of d_out in rows; must be >= dspfe_rows_bound(...)  */
int dspfe_mfcc_delta(dspfe_plan* plan, const int16_t* d_pcm, int64_t total_samples,
                     const int64_t* d_offsets, const int32_t* d_trim, int32_t n_utt,
                     float* d_out, int64_t max_rows, int64_t* d_frame_off, void* stream);

/* Same kernel fed with float32 samples (a signal the caller has already scaled, e.g. model.py:62-63 passes
 * sklearn-scaled audio to features.mfcc).  Offsets and trims are in samples as above. */
int dspfe_mfcc_delta_f32(dspfe_plan* plan, const float* d_pcm, int64_t total_samples,
                         const int64_t* d_offsets, const int32_t* d_trim, int32_t n_utt,
                         float* d_out, int64_t max_rows, int64_t* d_frame_off, void* stream);

/* Taps of the same kernel (float32 samples in).  dspfe_fbank_f32 replaces features.fbank (base.py:18-32):
 * d_out [rows, nfilt+1] = filterbank energies, then the total frame energy, both floored at float64 eps.
 * dspfe_spectrum_f32 replaces sigproc.powspec (:151, kind 0), magspec (:136, kind 1) and the un-normalised
 * logpowspec (:161, kind 2): d_out [rows, nfft/2+1].  The plan's preemph / window apply as for the MFCC. */
int dspfe_fbank_f32(dspfe_plan* plan, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                    float* d_out, int64_t max_rows, int64_t* d_frame_off, void* stream);
int dspfe_spectrum_f32(dspfe_plan* plan, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets, int32_t n_utt,
                       int32_t kind, float* d_out, int64_t max_rows, int64_t* d_frame_off, void* stream);

/* Upper bound on output rows for any batch with these totals. */
int64_t dspfe_rows_bound(const dspfe_plan* plan, int64_t total_samples, int64_t n_utt);

/* Same computation through host buffers: H2D copy of pcm/offsets, kernels, D2H copy of the
 * features, pipelined over utterance slabs on internal streams; returns after the result is in
 * h_out.  h_out must hold sum_u num_frames(len_u) rows; h_frame_off [n_utt+1] is written.
 * Pinned host memory (dspfe_host_alloc) makes the copies truly asynchronous. */
int dspfe_mfcc_delta_host(dspfe_plan* plan, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt,
                          float* h_out, int64_t* h_frame_off);

int dspfe_host_alloc(void** p, int64_t bytes);   /* cudaHostAlloc */
int dspfe_host_free(void* p);

/* ------------------------------------------------------------------------------------------------
 * Endpoint detection: short-time amplitude + zero-crossing rate, double-threshold rule.
 * Replaces features.basic_endpoint_detection (endpoint.py:34-66) with its helpers get_amplitude
 * (:109), get_zcr (:182), amplitude_rule (:133) and zcr_rule (:201) for every utterance of a batch.
 * Frame length / step are int(rate*cfg_frame) / int(cfg_step*rate) (sigproc.py:19; config.py:31-32).
 * All outputs are integers and bit-exact against the reference for int16 input.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dspfe_endpoint_plan dspfe_endpoint_plan;

typedef struct {
    int32_t samplerate;      /* 16000 */
    int32_t min_span;        /* 50 frames: shorter spans retry with mh2, then fall back to the whole signal */
    double cfg_frame;        /* 0.03  (config.py:31) */
    double cfg_step;         /* 0.01  (config.py:32) */
    double mh1, mh2;         /* 0.25, 0.125  (endpoint.py:42,45) */
    double th;               /* 0.1 s */
    double l_sil, r_sil;     /* 0.1 s, 0.1 s */
    double sigma;            /* 3 */
    double zcr_max_shift;    /* 0.4 s */
    double zcr_r_sil;        /* 0.1 s (zcr_rule's l_sil is 0) */
} dspfe_endpoint_params;

void dspfe_endpoint_params_default(dspfe_endpoint_params* p, int32_t samplerate);
int dspfe_endpoint_create(const dspfe_endpoint_params* p, dspfe_endpoint_plan** plan);
void dspfe_endpoint_destroy(dspfe_endpoint_plan* plan);
/* pre-sizes the plan's workspaces so that later calls up to these totals allocate nothing */
int dspfe_endpoint_reserve(dspfe_endpoint_plan* plan, int64_t max_utt, int64_t max_total_samples);
int32_t dspfe_endpoint_frame_len(const dspfe_endpoint_plan* plan);
int32_t dspfe_endpoint_frame_step(const dspfe_endpoint_plan* plan);
int64_t dspfe_endpoint_frames_bound(const dspfe_endpoint_plan* plan, int64_t total_samples, int64_t n_utt);

/* Device path.  d_lr [n_utt,2] int32 receives (left,right) sample indices exactly as the reference
 * returns them (right may exceed the utterance length, endpoint.py:64).  Optional outputs (may be
 * NULL): d_asum [frames] int32 = sum |x| per frame (amp = d_asum / frame_len in float64 is the
 * reference's get_amplitude), d_zcr [frames] int32 = get_zcr, d_frame_off [n_utt+1] int64.
 * max_frames = capacity of d_asum / d_zcr, >= dspfe_endpoint_frames_bound(). */
int dspfe_endpoint(dspfe_endpoint_plan* plan, const int16_t* d_pcm, int64_t total_samples, const int64_t* d_offsets,
                   int32_t n_utt, int32_t* d_lr, int32_t* d_asum, int32_t* d_zcr, int64_t* d_frame_off,
                   int64_t max_frames, void* stream);

/* Host-buffer path: H2D, kernels, D2H; returns when the results are in the host arrays. */
int dspfe_endpoint_host(dspfe_endpoint_plan* plan, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt,
                        int32_t* h_lr, int32_t* h_asum, int32_t* h_zcr, int64_t* h_frame_off);

/* Float32 samples (a signal already scaled, e.g. what soundfile / torchaudio return in [-1, 1]; model.py:62-63 scales each
 * utterance before its feature calls): basic_endpoint_detection (endpoint.py:34-66) with the frame statistics in the reference's
 * float64 arithmetic.  framesig pads with float64 zeros, so every sample enters as its exact float64 value:
 *   d_amp [frames] float64 = get_amplitude (endpoint.py:109): np.mean(np.abs(frame)) bit for bit, NumPy's pairwise summation
 *                            order over the frame_len values, then one division by frame_len;
 *   d_zcr [frames] int32  = get_zcr (endpoint.py:182): neighbours x[i], x[i+1] inside the frame (zero padding included) that
 *                            are both nonzero and of opposite sign, i.e. x[i] * x[i+1] < 0, which is exact in float64;
 *   d_lr                  = the same decision rule (K3) on these amplitudes.
 * Bit-exact against the reference for any float32 input.  d_pcm must be 16-byte aligned; utterance starts need only be
 * 4-byte aligned.  Optional outputs, validation and error codes as for dspfe_endpoint (max_frames is the capacity of d_amp /
 * d_zcr).  Frames longer than 8192 samples (int(rate * cfg_frame)) are not built: DSPFE_ERR_UNSUPPORTED.  The float64
 * amplitude workspace is part of the plan and dspfe_endpoint_reserve pre-sizes it. */
int dspfe_endpoint_f32(dspfe_endpoint_plan* plan, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets,
                       int32_t n_utt, int32_t* d_lr, double* d_amp, int32_t* d_zcr, int64_t* d_frame_off,
                       int64_t max_frames, void* stream);
/* Host-buffer form: H2D, kernels, D2H; h_amp [frames] float64, h_zcr, h_frame_off optional. */
int dspfe_endpoint_host_f32(dspfe_endpoint_plan* plan, const float* h_pcm, const int64_t* h_offsets, int32_t n_utt,
                            int32_t* h_lr, double* h_amp, int32_t* h_zcr, int64_t* h_frame_off);

/* robust_endpoint_detection (endpoint.py:68-92): the same frame statistics, amplitude_rule(mh = 0.5) whose expansion is
 * gated by acr_rule (endpoint.py:142-144: max over lags rate//500 .. rate//50 of acr(frame, n) / acr(frame, 0) > 0.55,
 * evaluated from exact integer lag sums), zcr_rule and the whole-signal fallback.  d_lr / h_lr [n_utt,2] int32. */
int dspfe_endpoint_robust(dspfe_endpoint_plan* plan, const int16_t* d_pcm, int64_t total_samples, const int64_t* d_offsets,
                          int32_t n_utt, int32_t* d_lr, void* stream);
int dspfe_endpoint_robust_host(dspfe_endpoint_plan* plan, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr);
/* robust_endpoint_detection (endpoint.py:68-92) on float32 samples: the frame statistics of dspfe_endpoint_f32, then the gated
 * rule with acr_rule evaluated in the reference's float64 arithmetic.  acr(frame, n) (sigproc.py:48-53) is NumPy's pairwise
 * sum of the len - n exact products x[i] x[i+n] divided by len - n, every lag with its own split tree; the gate is
 * max_n acr(n) / acr(0) > 0.55 over the lags rate//500 .. rate//50 below the frame length.  A frame holding a NaN or +-inf
 * sample, and an all-zero frame, fail the gate, as in the reference.  Bit-exact against the reference for any float32 input.
 * Frames longer than 1536 samples are not built: DSPFE_ERR_UNSUPPORTED.  d_pcm must be 16-byte aligned; validation and the
 * other error codes as for dspfe_endpoint_f32.  The host form stages the batch once and computes its statistics once. */
int dspfe_endpoint_robust_f32(dspfe_endpoint_plan* plan, const float* d_pcm, int64_t total_samples, const int64_t* d_offsets,
                              int32_t n_utt, int32_t* d_lr, void* stream);
int dspfe_endpoint_robust_host_f32(dspfe_endpoint_plan* plan, const float* h_pcm, const int64_t* h_offsets, int32_t n_utt, int32_t* h_lr);
/* List form of amplitude_rule(use_acr=True) (endpoint.py:133): gate[n_frames] (0/1) is acr_rule of every frame, which
 * dspfe_acr_gate_rows_f64 computes on the device for a float64 frame matrix [n_rows, len]. */
int dspfe_amplitude_rule_gated_host(const dspfe_endpoint_params* p, const double* amp, const int32_t* gate, int32_t n_frames, double mh,
                                    int32_t* segs, int32_t seg_cap, int32_t* n_segs);
int dspfe_acr_gate_rows_f64(const double* d_frames, int64_t n_rows, int32_t len, int32_t samplerate, int32_t* d_gate, void* stream);

/* Host-only (no CUDA): the decision rule on precomputed frame statistics; lets CPU-only tests check the
 * float64 rule replay (NumPy summation order included) against the oracle. */
int dspfe_endpoint_decide_host(const dspfe_endpoint_params* p, const int32_t* asum, const int32_t* zcr, int32_t n_frames,
                               int32_t* lr);
/* Host-only list forms of the two rules, for the reference's list-based API: amplitude_rule (endpoint.py:133; the
 * l_sil/r_sil/th/sigma of `p` apply, `mh` is the call's high-threshold factor) writes up to seg_cap (j,k) pairs and
 * their count; zcr_rule (endpoint.py:201) writes (j,k).  Same C++ code as the device kernel K3. */
int dspfe_amplitude_rule_host(const dspfe_endpoint_params* p, const double* amp, int32_t n_frames, double mh,
                              int32_t* segs, int32_t seg_cap, int32_t* n_segs);
int dspfe_zcr_rule_host(const dspfe_endpoint_params* p, const double* zcr, int32_t n_frames, double l_sil, int32_t left,
                        int32_t right, int32_t* out_jk);

/* ------------------------------------------------------------------------------------------------
 * Pitch: cepstrum pitch (features.pitch_detect, pitch.py:83-94), autocorrelation pitch (pitch_detect_sr,
 * pitch.py:96-110) and the five SVM inputs of pitch_model.py (pitch_feature, pitch.py:26-47) for every utterance
 * of a packed ragged batch.  Per utterance the kernels replay: downsampling (preprocess.py:21, sample picking) ->
 * to_frames (sigproc.py:11) -> center_clip (pitch.py:145) -> window band-pass (sigproc.py:22) -> cepstrum
 * (pitch.py:135) or autocorrelation scores (pitch.py:112, sigproc.py:48) -> smooth (pitch.py:157) -> peak_score
 * (pitch.py:227) -> robust_max_pitch (pitch.py:191) [-> sub_endpoint_detect (:64), find_smooth_subsequence (:245),
 * slope/quad_params/peakshift (:49-62)].
 * ---------------------------------------------------------------------------------------------- */
typedef struct dspfe_pitch_plan dspfe_pitch_plan;

typedef struct {
    int32_t samplerate;      /* rate of the packed samples, 16000 */
    int32_t dst_rate;        /* 10000: rate the pitch functions decimate to (pitch.py:84,100) */
    int32_t frame_len;       /* int(dst_rate*winlen): 512 (pitch_detect), or 300 for pitch_detect_sr as model.py:92 calls it.
                              * Cepstrum: 100..512 (512 runs the 512-point chain, the others N-point DFTs by Bluestein's chirp);
                              * autocorrelation: 21..512.  Others: DSPFE_ERR_UNSUPPORTED */
    int32_t frame_step;      /* int(step*dst_rate): 100 */
    int32_t method;          /* 0 cepstrum (pitch_detect), 1 autocorrelation (pitch_detect_sr) */
    int32_t center_clip;     /* 1: center_clip(frame, False) before the band-pass (pitch.py:88); 0 for the per-frame taps */
    int32_t row_len;         /* cepstrum columns kept per frame, 100..frame_len; 0 = min(frame_len, 200) (all peak_score can
                              * reach: its right-hand scan ends at the frame length), frame_len for the full-row tap */
    int32_t reserved;
    double band_lo, band_hi; /* band-pass edges in Hz: 50..1000 (pitch.py:137) / 50..900 (pitch.py:124) */
    double preemph;          /* pre-emphasis over the whole utterance before trimming (pitch_model.py:39-41); 0 = none */
} dspfe_pitch_params;

void dspfe_pitch_params_default(dspfe_pitch_params* p, int32_t method);
int dspfe_pitch_create(const dspfe_pitch_params* p, dspfe_pitch_plan** plan);
void dspfe_pitch_destroy(dspfe_pitch_plan* plan);
int dspfe_pitch_reserve(dspfe_pitch_plan* plan, int64_t max_utt, int64_t max_total_samples);   /* pre-sizes the workspaces */
int32_t dspfe_pitch_row_len(const dspfe_pitch_plan* plan);
/* pitch frames of one utterance of n_samples (after decimation and framing) / upper bound for a whole batch */
int64_t dspfe_pitch_num_frames(const dspfe_pitch_plan* plan, int64_t n_samples);
int64_t dspfe_pitch_frames_bound(const dspfe_pitch_plan* plan, int64_t total_samples, int64_t n_utt);
/* the same count without a plan or a device (host only); *n_decimated (optional) = len(downsampling(sig, samplerate, dst_rate)) */
int64_t dspfe_pitch_num_frames_host(const dspfe_pitch_params* p, int64_t n_samples, int64_t* n_decimated);

/* Device path, asynchronous on `stream`.  sample_dtype: 0 = int16, 1 = float32 samples.  d_trim as for
 * dspfe_mfcc_delta (pitch runs on sig[left:right], pitch_model.py:41).  Outputs (each may be NULL):
 *   d_pitch [frames] float64 Hz (robust_max_pitch), d_lag [frames] int32 = 20 + argmax (before the octave repair),
 *   d_feat [n_utt,5] float64 = pitch_feature (cepstrum method at frame_len 512 only, the default winlen pitch.py:33 uses;
 *          other plans fail with DSPFE_ERR_UNSUPPORTED; NaN x5 where a half has < 3 usable frames),
 *   d_rows [frames,row_len] float32 = the per-frame cepstrum / autocorrelation rows before smoothing,
 *   d_frame_off [n_utt+1] int64.  max_frames = capacity in frames, >= dspfe_pitch_frames_bound(). */
int dspfe_pitch(dspfe_pitch_plan* plan, const void* d_pcm, int32_t sample_dtype, int64_t total_samples, const int64_t* d_offsets,
                const int32_t* d_trim, int32_t n_utt, double* d_pitch, int32_t* d_lag, double* d_feat, float* d_rows,
                int64_t* d_frame_off, int64_t max_frames, void* stream);

/* Host-buffer path: H2D, kernels, D2H; returns when the results are in the host arrays (h_trim optional). */
int dspfe_pitch_host(dspfe_pitch_plan* plan, const void* h_pcm, int32_t sample_dtype, const int64_t* h_offsets, const int32_t* h_trim,
                     int32_t n_utt, double* h_pitch, int32_t* h_lag, double* h_feat, int64_t* h_frame_off);

/* Taps on caller-supplied device arrays.
 * center_clip (pitch.py:145 == endpoint.py:20): rows of len <= 512 float32; binary != 0 gives -1/0/1. */
int dspfe_center_clip_f32(const float* d_in, int64_t n_rows, int32_t len, int32_t binary, float* d_out, void* stream);
/* K4b/K5b on caller rows [n_rows,row_len] (row_len <= 512): smooth(g, 2) (pitch.py:157) when do_smooth, then per row either
 * peak_score (pitch.py:227; mode 0, d_score [n_rows,80]) and its first argmax, or the plain first argmax (mode 1);
 * d_lag = 20 + argmax.  d_smoothed receives the rows that were scored.  Outputs may be NULL. */
int dspfe_track_rows_f32(const float* d_rows, int64_t n_rows, int32_t row_len, int32_t mode, int32_t do_smooth, float* d_smoothed,
                         int32_t* d_score, int32_t* d_lag, void* stream);

/* Host-only list helpers, the reference's small sequential functions (same C++ as the device kernels K4b/K6):
 * max_pitch / robust_max_pitch on lags (pitch.py:166,191; repair = 0/1), find_smooth_subsequence (pitch.py:245),
 * sub_endpoint_detect on per-frame sum|x| (pitch.py:64), the pitch_feature tail (pitch.py:33-46) and the leading
 * polyfit coefficient of slope / quad_params (pitch.py:49-57; deg 1 or 2). */
int dspfe_robust_max_pitch_host(const int32_t* lag, int32_t n, int32_t repair, double* pitch);
int dspfe_smooth_subsequence_host(const double* pitch, int32_t n, int32_t tor, double thres, double* seg, int32_t* seg_len,
                                  int32_t* i0, int32_t* j0);
int dspfe_sub_endpoint_host(const double* amp, int32_t n_frames, int32_t* p);
int dspfe_pitch_feature_tail_host(const double* pitch, const double* amp, int32_t n_frames, double* out5);
int dspfe_poly_lead_host(const double* seq, int32_t n, int32_t deg, double* coef);
/* dp_max_pitch (pitch.py:208-225): Viterbi over the columns of g [n_rows,n_cols]; path [n_rows] = 10000 / lag index.
 * dspfe_dp_max_pitch is the device kernel (d_g, d_path device memory, n_cols <= 1024, asynchronous on `stream`);
 * dspfe_dp_max_pitch_host the same recurrence on host arrays (no CUDA), kept for CPU-only checks. */
int dspfe_dp_max_pitch(const double* d_g, int32_t n_rows, int32_t n_cols, double* d_path, void* stream);
int dspfe_dp_max_pitch_host(const double* g, int32_t n_rows, int32_t n_cols, double* path);

/* ------------------------------------------------------------------------------------------------
 * Helpers: the reference's small array functions as device kernels (not on the throughput path; the
 * fused kernels never materialise frames).  All pointers are device memory.
 * ---------------------------------------------------------------------------------------------- */
/* framesig (sigproc.py:66-98) / to_frames (:11): [n_frames, frame_len] float64, zero padded, times d_win if given */
int dspfe_frames_f64(const double* d_sig, int64_t n, int32_t frame_len, int32_t frame_step, const double* d_win,
                     double* d_out, int64_t n_frames, void* stream);
/* preemphasis (sigproc.py:178 == preprocess.py:11) */
int dspfe_preemphasis_f64(const double* d_x, int64_t n, double coeff, double* d_y, void* stream);
/* get_amplitude(frames, 'square', use_sq) (endpoint.py:109): per-row mean |x| (use_sq 0) or x^2 (1) in NumPy's summation
 * order; use_sq 2 = plain sum |x| per row (sub_endpoint_detect, pitch.py:65) */
int dspfe_row_amplitude_f64(const double* d_frames, int64_t n_rows, int32_t len, int32_t use_sq, double* d_out, void* stream);
/* get_amplitude(frames, window=<taps>, use_sq) (endpoint.py:118-125): per-row mean of np.convolve(|x| or x^2, window, 'same');
 * h_window is a host array of win_len taps (np.hamming(len) for window='hamming') */
int dspfe_row_windowed_amplitude_f64(const double* d_frames, int64_t n_rows, int32_t len, const double* h_window, int32_t win_len,
                                     int32_t use_sq, double* d_out, void* stream);
/* get_zcr(frames) (endpoint.py:182) */
int dspfe_row_zcr_f64(const double* d_frames, int64_t n_rows, int32_t len, int64_t* d_out, void* stream);
/* Caller-side batching epilogue of the reference trainer (model.py:75-88, :35-50, :131-135) on K1's rows
 * [F_total, 3*numcep]: the static block is standardised per utterance and column (sklearn scale: population std over
 * all frames, constant columns only centred), delta / delta-delta are passed through, every utterance is truncated or
 * zero padded to T frames, and the batch is written time-major: d_out [T, n_utt, 3*numcep]; d_len0 [n_utt] = min(F, T). */
int dspfe_cmvn_pad_batch(const float* d_feat, const int64_t* d_frame_off, int32_t n_utt, int32_t numcep, int32_t T, float* d_out,
                         int32_t* d_len0, void* stream);
/* window (sigproc.py:22-46): causal complex FIR band-pass of a real signal, d_y [n,2] = (re, im) float64 */
int dspfe_fir_window_f64(const double* d_x, int32_t n, double rate, double low_freq, double high_freq, int32_t hamming,
                         double* d_y, void* stream);
/* acr (sigproc.py:48-53): unbiased autocorrelation of one frame at lag n -> d_out[0] */
int dspfe_acr_f64(const double* d_frame, int32_t len, int32_t n, double* d_out, void* stream);
/* delta(feat, N) (base.py:70) on an arbitrary [n_frames, n_cols] float32 matrix */
int dspfe_delta_f32(const float* d_in, int64_t n_frames, int32_t n_cols, int32_t N, float* d_out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Ingest (reader.py:67-85: scipy.io.wavfile.read + sig[:,0]): 16-bit PCM RIFF/WAVE files, channel 0, into the packed
 * ragged batch.  dspfe_wav_info parses one file image on the host.  dspfe_ingest_wavs takes the images of n files,
 * writes h_offsets [n_files+1] (samples) and h_rates [n_files], streams the sample bytes through pinned staging buffers
 * and de-interleaves channel 0 on the device into d_pcm (capacity in samples); returns when the batch is resident.
 * ---------------------------------------------------------------------------------------------- */
int dspfe_wav_info(const void* bytes, int64_t size, int32_t* rate, int32_t* channels, int32_t* bits, int64_t* n_frames, int64_t* data_offset);
void dspfe_ingest_release(void);   /* frees the staging buffers the ingest path keeps between calls */
int dspfe_ingest_wavs(const void* const* file_bytes, const int64_t* sizes, int32_t n_files, int16_t* d_pcm, int64_t capacity,
                      int64_t* h_offsets, int32_t* h_rates, void* stream);

/* The same from file paths: the library reads the files itself and the sample bytes go straight into the pinned slabs.
 * dspfe_wav_scan_paths only reads the headers (h_offsets[n_files] = total samples, to size d_pcm). */
int dspfe_wav_scan_paths(const char* const* paths, int32_t n_files, int64_t* h_offsets, int32_t* h_rates);
int dspfe_ingest_wav_paths(const char* const* paths, int32_t n_files, int16_t* d_pcm, int64_t capacity, int64_t* h_offsets,
                           int32_t* h_rates, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Whole front-end over one packed ragged batch, as the reference's two callers chain it per utterance:
 *   (l, r) = basic_endpoint_detection(sig, rate)                                   model.py:52-53, pitch_model.py:38
 *   mfcc(sig[l:r]) + delta + delta (N = delta_n)                                   model.py:74-77
 *   pitch_feature(preemphasis(sig, 0.97)[l:r], rate)  (cepstrum pitch + 5 floats)  pitch_model.py:39-41
 *   pitch_detect_sr(sig[l:r], rate, winlen=cfg.frame, step=cfg.step)               model.py:92
 * The batch is walked in slabs of consecutive utterances so that the pitch workspaces (about 3 KB per 10 ms of audio)
 * stay bounded by the slab, whatever the batch size (BASELINE config 5).  Row / frame offsets in the outputs are global.
 * ---------------------------------------------------------------------------------------------- */
typedef struct dspfe_frontend_plan dspfe_frontend_plan;

typedef struct {
    int32_t samplerate;        /* 16000 */
    int32_t delta_n;           /* 2 */
    int32_t acr_frame_len;     /* 300 = int(10000 * cfg.frame), model.py:92 */
    int32_t reserved;
    int64_t slab_samples;      /* device path: samples per slab, 0 = 256 Mi */
    int64_t host_slab_samples; /* host path: samples per pipelined slab, 0 = 32 Mi */
    double cep_preemph;        /* 0.97 (pitch_model.py:39) */
} dspfe_frontend_params;

/* Output arrays (device pointers for dspfe_frontend, host pointers for dspfe_frontend_host); any pointer may be NULL
 * to skip that output's copy (the path still runs).  Capacities are in rows / frames and must cover the untrimmed
 * bounds: dspfe_rows_bound / dspfe_pitch_frames_bound of the whole batch. */
typedef struct {
    int32_t* lr;               /* [n_utt,2] endpoints (left, right) */
    float* mfcc;               /* [mfcc_cap, 39] */
    int64_t mfcc_cap;
    int64_t* mfcc_frame_off;   /* [n_utt+1] */
    double* cep_pitch;         /* [cep_cap] Hz, cepstrum method */
    int64_t cep_cap;
    int64_t* cep_frame_off;    /* [n_utt+1] */
    double* cep_feat;          /* [n_utt,5] pitch_feature */
    double* acr_pitch;         /* [acr_cap] Hz, autocorrelation method */
    int64_t acr_cap;
    int64_t* acr_frame_off;    /* [n_utt+1] */
    int32_t* cep_lag;          /* [cep_cap] 20 + argmax before the octave repair (optional) */
    int32_t* acr_lag;          /* [acr_cap] (optional) */
} dspfe_frontend_out;

void dspfe_frontend_params_default(dspfe_frontend_params* p);
int dspfe_frontend_create(const dspfe_frontend_params* p, dspfe_frontend_plan** plan);
void dspfe_frontend_destroy(dspfe_frontend_plan* plan);
/* capacities that hold any batch with these totals: caps[0] MFCC rows, caps[1] cepstrum frames, caps[2] autocorrelation frames */
int dspfe_frontend_bounds(const dspfe_frontend_plan* plan, int64_t total_samples, int64_t n_utt, int64_t* caps);
/* Device path: PCM and outputs resident.  h_offsets is the host copy of d_offsets (the slab boundaries are cut on the
 * host).  totals[3] (host, optional) receives the MFCC rows / cepstrum frames / autocorrelation frames written.  The call
 * waits for each slab's frame counts (one 24-byte read back per slab) and returns when the last slab has been queued on
 * `stream` and counted, i.e. the outputs are complete when it returns. */
int dspfe_frontend(dspfe_frontend_plan* plan, const int16_t* d_pcm, const int64_t* d_offsets, const int64_t* h_offsets,
                   int32_t n_utt, const dspfe_frontend_out* d_out, int64_t* totals, void* stream);
/* Host-buffer path: slabs are copied H2D, processed and copied back D2H on three internal streams, overlapped. */
int dspfe_frontend_host(dspfe_frontend_plan* plan, const int16_t* h_pcm, const int64_t* h_offsets, int32_t n_utt,
                        const dspfe_frontend_out* h_out, int64_t* totals);
/* The same chain on float32 samples: dspfe_endpoint_f32, dspfe_mfcc_delta_f32 on sig[l:r], dspfe_pitch with sample_dtype 1
 * for both methods (the cepstrum chain's pre-emphasis included).  Outputs, capacities (dspfe_frontend_bounds) and slabs as
 * above; d_pcm 16-byte aligned.  A slab starts at the 16-byte aligned sample at or before its first utterance (a multiple
 * of 4 samples), and host_slab_samples counts samples, so a float slab moves twice the bytes of an int16 one. */
int dspfe_frontend_f32(dspfe_frontend_plan* plan, const float* d_pcm, const int64_t* d_offsets, const int64_t* h_offsets,
                       int32_t n_utt, const dspfe_frontend_out* d_out, int64_t* totals, void* stream);
int dspfe_frontend_host_f32(dspfe_frontend_plan* plan, const float* h_pcm, const int64_t* h_offsets, int32_t n_utt,
                            const dspfe_frontend_out* h_out, int64_t* totals);

/* ------------------------------------------------------------------------------------------------
 * Per-kernel timing for reports (bench.py): between dspfe_timing_begin(stream) and dspfe_timing_end every kernel the
 * library launches on `stream` is bracketed by CUDA events.  dspfe_timing_end waits for the stream and writes up to
 * `cap` records: names[i*48 .. ] = kernel name (NUL terminated, 48 bytes each), ms[i] = its duration; *n = records
 * available.  dspfe_launch_count = kernels launched by the library since it was loaded.
 * ---------------------------------------------------------------------------------------------- */
int dspfe_timing_begin(void* stream);
int dspfe_timing_end(char* names, float* ms, int32_t cap, int32_t* n);
int64_t dspfe_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DSPFE_H_ */
