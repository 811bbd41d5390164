// Plain-data parameter blocks shared by host code, the CUDA kernels and the test emulator.
#pragma once
#include <stdint.h>

namespace dspfe {

constexpr int kNfft = 512;            // real FFT length of the MFCC kernel (reference default, base.py:9)
constexpr int kBins = kNfft / 2 + 1;  // 257
constexpr int kGroupLanes = 16;       // lanes that cooperate on one frame pair
constexpr int kMaxNfilt = 40;
constexpr int kMaxNumcep = 16;
constexpr int kMaxDeltaN = 4;
constexpr int kMelSlots = 3;          // mel filter pieces per lane (one per slot)
constexpr int kMelMaxPieces = 4;      // pieces a single mel filter may be cut into
constexpr int kScratchUnits = 272;    // 8-byte units per group: 16x17 transpose tile, >= 257 power bins
constexpr int kTriNfft = 1536;        // K1T: the transform size of model.py:74
constexpr int kMfccThreads = 128;     // 8 groups -> 16 frames per pass of the chunk loop
constexpr int kMfccGroups = kMfccThreads / kGroupLanes;
constexpr int kFramesPerPass = 2 * kMfccGroups;

struct Tile { int utt, f0, nf, pad; };  // output frames [f0, f0+nf) of utterance utt

struct MfccParams {
    // inputs (device pointers)
    const void* pcm;            // packed ragged PCM (int16 or float32 samples), base 16-byte aligned
    int64_t total_samples;      // samples in pcm
    const int64_t* seg_start;   // [U] first sample of each (trimmed) utterance inside pcm
    const int32_t* seg_len;     // [U] samples
    const int64_t* frame_off;   // [U+1] output row of each utterance's frame 0
    const Tile* tiles;          // tile table written by the prep kernel
    const int32_t* ntiles;      // number of valid tiles (device scalar)
    const float* tables;        // constant tables blob (see MfccTables)
    float* out;                 // [F_total, 3*numcep]
    // dims
    int frame_len, frame_step, nfilt, numcep, delta_n, seg_frames, append_energy;
    int spec_kind;              // MODE 2 only: 0 power, 1 magnitude, 2 10*log10(power)
    float preemph, delta_scale, pow_scale;
    // table blob offsets, in floats
    int o_twa, o_twp, o_melw, o_melb, o_melc, o_dct, o_win, dct_stride, tbl_floats;
    int mel_T[kMelSlots];       // iterations per mel slot (uniform over the lanes)
    // shared-memory carve-up, in bytes
    int sm_mbar, sm_scratch, sm_mfcc, sm_fbuf, sm_raw, sm_total;
    int fbuf_floats;            // (kFramesPerPass-1)*step + frame_len: samples one chunk needs
    int fbuf_vecs;              // 8-sample vectors converted per chunk (covers the raw staging area)
    // K1T (nfft = 1536 as three 256-point complex transforms, mfcc_kernel.cuh TRI): bins 3q + c form class c
    int tri;                    // 0: K1 (nfft 512), 1: K1T
    int grp_units;              // 8-byte scratch units per 16-lane group (kScratchUnits)
    int o_tw3, o_tws2;          // [m] float4 (cos a1, cos a2, sin a1, sin a2) of W768^m, W768^2m; W1536^{3q + 2} at [q]
    int o_melw_c[2], o_melb_c[2];   // piece tables: class 0 (= o_melw / o_melb), the joint classes 1 + 2
    int mel_Tc[2][kMelSlots];
};

struct PrepParams {
    const int64_t* offsets;     // [U+1] packed utterance boundaries (samples)
    const int32_t* trim;        // optional [U,2] (left,right) sample indices from the endpoint kernel, or null
    int n_utt;
    int frame_len, frame_step, seg_frames;
    int64_t* seg_start; int32_t* seg_len; int64_t* frame_off; int32_t* tile_off;
    Tile* tiles; int32_t* ntiles; int max_tiles;
};

// frame count rule of framesig (reference sigproc.py:79-82)
inline
#ifdef __CUDACC__
__host__ __device__
#endif
int64_t num_frames(int64_t slen, int frame_len, int frame_step) {
    if (slen <= frame_len) return 1;
    return 1 + (slen - frame_len + frame_step - 1) / frame_step;
}

// Python's slice sig[l:r] with l, r >= 0 of a signal of `len` samples: l and r clamped into [0, len]; returns the slice's
// length and leaves its first sample in l.  (The prep kernels write the clamp out: through this call their SASS differs.)
inline
#ifdef __CUDACC__
__host__ __device__
#endif
long long trim_slice(long long len, long long& l, long long r) {
    if (l < 0) l = 0; if (r < 0) r = 0;
    if (l > len) l = len; if (r > len) r = len;
    return r > l ? r - l : 0;
}

}  // namespace dspfe
