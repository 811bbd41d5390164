// Emulator entry point for the cepstrum pitch at frame lengths other than 512 samples (pitch_cep_bluestein_pair,
// K4a-2b).  TEST INFRASTRUCTURE ONLY.  The same pipeline as emu_pitch (K4a-1 clip, K4a-2 transforms, K4b track), with the
// Bluestein chain in the transform step.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../dsp-speech-recognition_b200/csrc/dspfe_types.h"
#include "../../dsp-speech-recognition_b200/csrc/pitch_kernel.cuh"
#include "../../dsp-speech-recognition_b200/csrc/pitch_tables.h"
#include "../../include/dspfe.h"

namespace emu { bool run_cta(int bid, int nthreads, void (*body)(void*), void* arg); }
using namespace dspfe;

namespace {
struct CepArgs { PitchParams p; std::vector<unsigned char>* smem; };
void cep_clip_body(void* a) {
    CepArgs* A = (CepArgs*)a;
    const int w = simt::tid() >> 5;
    const int64_t h0 = kClipRun * ((int64_t)simt::bid() * kPitchWarps + w);
    if (h0 >= A->p.slot_off[A->p.n_utt]) return;
    unsigned char* wsm = A->smem->data() + w * kClipWarpSmemBytes;
    const bool i16 = clip_i16_keys(A->p);
    if (A->p.frame_len <= 320) {
        if (i16) pitch_clip_run<10, true>(A->p, h0, wsm, A->p.ds_idx); else pitch_clip_run<10, false>(A->p, h0, wsm, A->p.ds_idx);
    } else {
        if (i16) pitch_clip_run<16, true>(A->p, h0, wsm, A->p.ds_idx); else pitch_clip_run<16, false>(A->p, h0, wsm, A->p.ds_idx);
    }
}
// pitch_cep_bluestein_kernel's body: a frame pair per warp (the device kernel stages the twiddles in shared memory; the
// emulator reads them in place)
void cep_frame_body(void* a) {
    CepArgs* A = (CepArgs*)a;
    const int w = simt::tid() >> 5;
    const int64_t h0 = 2 * ((int64_t)simt::bid() * kPitchWarps + w);
    if (h0 >= A->p.slot_off[A->p.n_utt]) return;
    int nvalid; int64_t g0;
    slot_unit_from_desc(A->p, h0, 2, g0, nvalid);
    if (nvalid == 0) return;
    pitch_cep_bluestein_pair(A->p, h0, g0, nvalid > 1, A->smem->data() + w * kWarpSmemBytes, A->p.tab, A->p.tab + kTabW32);
}
void cep_track_body(void* a) {
    CepArgs* A = (CepArgs*)a;
    float* chunk = reinterpret_cast<float*>(A->smem->data());
    int* sc = reinterpret_cast<int*>(chunk + (track_chunk(A->p.row_len) + 1) * A->p.row_len);
    pitch_track_cta(A->p, chunk, sc, reinterpret_cast<double*>(sc + track_chunk(A->p.row_len) * kPeakLags));
}
}  // namespace

// Same contract as emu_pitch (dspfe_pitch on host pointers, synchronous; no pitch_feature) for cepstrum plans, every frame
// through the Bluestein chain.  At frame_len 512 it fills the Bluestein tables itself: the library sends 512-sample frames
// to pitch_fft_pair<0>, so this cross-checks the two chains on the same clipped frames.  Returns total frames, <0 on error.
extern "C" long long emu_pitch_cep(const dspfe_pitch_params* q, const void* pcm, int in_f32, const long long* offsets, const int* trim,
                                   int n_utt, double* pitch, int* lag, float* rows, float* rows_smoothed, int* score,
                                   long long* frame_off_out, long long max_frames, char* errbuf, int errcap) {
    if (q->method != 0) { std::snprintf(errbuf, errcap, "the Bluestein chain is a cepstrum kernel"); return -2; }
    PitchParams p;
    std::vector<float2> tab;
    std::string err;
    if (build_pitch_tables(*q, p, tab, err)) { std::snprintf(errbuf, errcap, "%s", err.c_str()); return -2; }
    if (q->frame_len == kCepLen) fill_cep_bluestein_tables(kCepLen, tab.data() + kTabChirp, tab.data() + kTabBe, tab.data() + kTabBo);
    std::vector<int64_t> seg_start(n_utt + 1), frame_off(n_utt + 1), slot_off(n_utt + 1);
    std::vector<int32_t> seg_len(n_utt + 1), ds_len(n_utt + 1);
    int64_t fo = 0, so = 0;
    for (int u = 0; u < n_utt; ++u) {
        int64_t a = offsets[u], len = offsets[u + 1] - offsets[u];
        if (trim) {
            int64_t l = trim[2 * u], r = trim[2 * u + 1];
            if (l < 0) l = 0; if (r < 0) r = 0;
            if (l > len) l = len; if (r > len) r = len;
            a += l; len = r > l ? r - l : 0;
        }
        seg_start[u] = a; seg_len[u] = (int32_t)len;
        ds_len[u] = (int32_t)ds_length(len, p.ds_idx, p.ds_in, p.ds_out);
        frame_off[u] = fo; slot_off[u] = so;
        const int64_t nf = num_frames(ds_len[u], p.frame_len, p.frame_step);
        fo += nf; so += (nf + kClipRun - 1) / kClipRun * kClipRun;
    }
    frame_off[n_utt] = fo; slot_off[n_utt] = so;
    if (fo > max_frames) { std::snprintf(errbuf, errcap, "outputs too small"); return -1; }
    if (frame_off_out) std::memcpy(frame_off_out, frame_off.data(), (n_utt + 1) * sizeof(int64_t));
    std::vector<float> rows_own; std::vector<double> amp(fo), pitch_own(fo); std::vector<int32_t> lag_own(fo);
    if (!rows) { rows_own.resize((size_t)fo * p.row_len); rows = rows_own.data(); }
    p.pcm = pcm; p.in_f32 = in_f32; p.total_samples = offsets[n_utt]; p.offsets = (const int64_t*)offsets; p.trim = trim; p.n_utt = n_utt;
    p.tab = tab.data(); p.frame_off = frame_off.data(); p.slot_off = slot_off.data(); p.seg_start = seg_start.data(); p.seg_len = seg_len.data();
    p.ds_len = ds_len.data(); p.rows = rows; p.rows_out = rows_smoothed; p.score = score; p.frame_amp = amp.data();
    p.pitch = pitch ? pitch : pitch_own.data(); p.lag = lag ? lag : lag_own.data(); p.feat = nullptr; p.scratch = nullptr;
    p.max_frames = fo;
    std::vector<float2> clip((size_t)((so + 1) / 2) * 512);
    p.clip = clip.data();
    std::vector<int4> run_desc((size_t)(so / kClipRun + 1));
    p.run_desc = run_desc.data();
    std::vector<unsigned char> smem0(kPitchWarps * kClipWarpSmemBytes + 64);
    CepArgs A0{p, &smem0};
    for (int64_t b = 0; b * kClipRun * kPitchWarps < so + kClipRun * kPitchWarps; ++b) {
        std::memset(smem0.data(), 0xCD, smem0.size());
        if (!emu::run_cta((int)b, 32 * kPitchWarps, cep_clip_body, &A0)) { std::snprintf(errbuf, errcap, "deadlock in clip CTA %lld", (long long)b); return -3; }
    }
    std::vector<unsigned char> smem(kPitchWarps * kWarpSmemBytes + 64);
    CepArgs A{p, &smem};
    for (int64_t b = 0; b * 2 * kPitchWarps < so + 2 * kPitchWarps; ++b) {
        std::memset(smem.data(), 0xCD, smem.size());
        if (!emu::run_cta((int)b, 32 * kPitchWarps, cep_frame_body, &A)) { std::snprintf(errbuf, errcap, "deadlock in frame CTA %lld", (long long)b); return -3; }
    }
    std::vector<unsigned char> smem2((track_chunk(p.row_len) + 1) * p.row_len * sizeof(float) + kTrackChunk * kPeakLags * sizeof(int) + kTrackMaxFrames * 12 + (kTrackThreads / 32) * kTrackListPerWarp * 2 + 8 + 64);
    CepArgs B{p, &smem2};
    for (int u = 0; u < n_utt; ++u) {
        std::memset(smem2.data(), 0xCD, smem2.size());
        if (!emu::run_cta(u, kTrackThreads, cep_track_body, &B)) { std::snprintf(errbuf, errcap, "deadlock in track CTA %d", u); return -3; }
    }
    return fo;
}
