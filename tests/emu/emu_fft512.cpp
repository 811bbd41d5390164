// Emulator entry point for fft512 (csrc/fft_regs.h) on its own.  TEST INFRASTRUCTURE ONLY.
#include <cmath>
#include <vector>

#include "../../dsp-speech-recognition_b200/csrc/fft_regs.h"
#include "../../dsp-speech-recognition_b200/csrc/pitch_kernel.cuh"
#include "../../dsp-speech-recognition_b200/csrc/pitch_tables.h"

namespace emu { bool run_cta(int bid, int nthreads, void (*body)(void*), void* arg); }
using namespace dspfe;

namespace {
struct FftArgs { const float* in; float* out; int inverse; const float2* tws; float2* scr; };
// one warp, register t of lane l holds element 32 t + l of both frames, before and after the transform
void fft_body(void* a) {
    FftArgs* A = (FftArgs*)a;
    const int lane = simt::tid() & 31;
    cpx2 x[16];
    for (int t = 0; t < 16; ++t) {
        const int n = 32 * t + lane;
        x[t].re = make_float2(A->in[2 * n], A->in[1024 + 2 * n]);
        x[t].im = make_float2(A->in[2 * n + 1], A->in[1024 + 2 * n + 1]);
        if (A->inverse) x[t].im = f2neg(x[t].im);                 // inverse = conj . forward . conj, as the pitch chains take it
    }
    fft512(x, A->scr, A->tws, lane);
    for (int t = 0; t < 16; ++t) {
        if (A->inverse) x[t].im = f2neg(x[t].im);
        const int k = 32 * t + lane;
        A->out[2 * k] = x[t].re.x; A->out[2 * k + 1] = x[t].im.x;
        A->out[1024 + 2 * k] = x[t].re.y; A->out[1024 + 2 * k + 1] = x[t].im.y;
    }
}
}  // namespace

// in / out: two frames of 512 interleaved (re, im) float32 each, frame A then frame B; out[.][k] is the value register k >> 5
// of lane k & 31 holds after the transform.  inverse: the unnormalised inverse.  Returns 0, or -1 if the warp deadlocks.
extern "C" int emu_fft512(const float* in, float* out, int inverse) {
    std::vector<float2> tws(512), w32(32);
    fill_fft512_twiddles(tws.data(), w32.data());
    std::vector<float2> scr(kWarpScr, make_float2(NAN, NAN));      // every tile entry the routine reads must have been written
    FftArgs A{in, out, inverse, tws.data(), scr.data()};
    return emu::run_cta(0, 32, fft_body, &A) ? 0 : -1;
}
