// Emulator entry points for the exact pieces of K3r's float gate (endpoint_kernel.cuh acr_lag / acr_gate_frame, host-and-device
// functions the kernel's exact path shares).  TEST INFRASTRUCTURE ONLY.
#include <cstdint>

#include "../../dsp-speech-recognition_b200/csrc/endpoint_kernel.cuh"

using namespace dspfe;

// acr(frame, n) of a float32 frame x[0..avail) with a zero tail to len samples, and the serial acr_rule over the lags [n0, n1).
extern "C" double emu_acr_lag_f32(const float* x, int avail, int len, int n) { return acr_lag(x, avail, len, n); }
extern "C" int emu_acr_gate_f32(const float* x, long long avail, int len, int n0, int n1) { return acr_gate_frame(x, avail, len, n0, n1) ? 1 : 0; }
