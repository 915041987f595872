// pm.cuh -- periodic particle-mesh gravity (pm.cu): deterministic CIC deposit, FFT Poisson solve with a Gaussian
// long-range filter, spectral gradient and CIC interpolation.
#pragma once
#include "common.cuh"

namespace b200 {

constexpr int PM_PHASES = 7;   // deposit, convert, R2C, k-space, C2R (all), interpolation, whole call

int pm_forces(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0, size_t n_targets, int grid, float box,
              float r_split, void* acc3, void* phi, cudaStream_t st);
// Event times (ms) of the phases of the last pm_forces call made with timing enabled (b200_set_timing).
int pm_phase_ms(b200_ctx* ctx, float ms[PM_PHASES]);
void pm_destroy(b200_ctx* ctx);

}  // namespace b200
