// The host build of the denoiser's passes (denoise_emu.cpp) plus kDenoiseSigmaMin (csrc/rt_denoise.cuh), so that
// tests/test_denoise_edges_cpu.py compares the smallest accepted sigma the filter sees with the one its float64 statement names
// (test infrastructure only).
#include "denoise_emu.cpp"

extern "C" float emu_denoise_sigma_min() { return kDenoiseSigmaMin; }
