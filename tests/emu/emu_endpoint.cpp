// Emulator entry point for K2f (float-sample endpoint statistics).  TEST INFRASTRUCTURE ONLY.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../dsp-speech-recognition_b200/csrc/endpoint_kernel.cuh"

namespace emu { bool run_cta(int bid, int nthreads, void (*body)(void*), void* arg); }
using namespace dspfe;

namespace {
struct Args { EpF32Params p; std::vector<unsigned char>* smem; };
void body(void* a) { Args* A = (Args*)a; ep_f32_stats_cta(A->p, A->smem->data()); }
}  // namespace

// Same statistics as dspfe_endpoint_f32 on host arrays: amp [frames] float64, zcr [frames] int32, frame_off [n_utt+1].
// Returns the frame count, < 0 on error.
extern "C" long long emu_endpoint_f32(const float* pcm, long long total, const long long* offsets, int n_utt, int frame_len,
                                      int frame_step, int nthreads, double* amp, int* zcr, long long max_frames, long long* frame_off) {
    if (frame_len < 1 || frame_step < 1 || frame_len > kEpF32MaxLen) return -2;
    std::vector<int64_t> fo(n_utt + 1, 0);
    for (int u = 0; u < n_utt; ++u) fo[u + 1] = fo[u] + num_frames(offsets[u + 1] - offsets[u], frame_len, frame_step);
    if (fo[n_utt] > max_frames) return -1;
    std::memcpy(frame_off, fo.data(), (n_utt + 1) * sizeof(int64_t));
    EpF32Params p;
    std::memset(&p, 0, sizeof(p));
    std::vector<int32_t> tree = np_pairwise_tree(frame_len, &p.nleaf);
    p.pcm = pcm; p.total_samples = total; p.offsets = reinterpret_cast<const int64_t*>(offsets); p.frame_off = fo.data(); p.n_utt = n_utt;
    p.frame_len = frame_len; p.frame_step = frame_step; p.tree = tree.data(); p.max_frames = fo[n_utt]; p.amp = amp; p.zcr = zcr;
    ep_f32_layout(p);
    std::vector<unsigned char> smem(p.sm_total + 64);
    Args A{p, &smem};
    for (int64_t b = 0; b * p.run < fo[n_utt] + p.run; ++b) {   // one surplus CTA exercises the early exit
        std::memset(smem.data(), 0xCD, smem.size());
        if (!emu::run_cta((int)b, nthreads, body, &A)) return -3;
    }
    return fo[n_utt];
}
