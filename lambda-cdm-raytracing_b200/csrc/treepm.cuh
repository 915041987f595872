// treepm.cuh -- the short-range factors of the TreePM force and potential split, shared by the device walk and host checks.
//
// With the Gaussian split radius r_s of the particle mesh (b200_pm_forces_dev) the short-range pair force is
// m d / r^3 * g(r), g(r) = erfc(u) + 2u/sqrt(pi) exp(-u^2), u = r / (2 r_s).  erfc is Abramowitz-Stegun 7.1.26,
// erfc(u) = t P(t) exp(-u^2) with t = 1 / (1 + p u), so g = exp(-u^2) (t P(t) + 2u/sqrt(pi)): one exponential,
// one reciprocal and six FMAs.  Relative error of g, against float64: <= 7.5e-6 for u <= 2.25 (r <= 4.5 r_s,
// the default cut-off); beyond it the absolute error stays below the formula's 1.5e-7 while g itself falls
// (g = 4.4e-4 at u = 3), so the relative error grows to 3.3e-5 at r = 6 r_s.
#pragma once

#ifdef __CUDACC__
#define B200_HD __host__ __device__
#else
#define B200_HD
#include <math.h>
#endif

namespace b200 {

// exp(-u^2) = e and t, P(t) of erfc(u) = t P(t) exp(-u^2), u >= 0.  The device form uses the approximate MUFU
// reciprocal and exponential (relative error about 1e-7 each); the host form is the same expression in IEEE float
// arithmetic.
B200_HD inline void treepm_erfc_parts(float u, float& e, float& t, float& p) {
    const float q = fmaf(0.3275911f, u, 1.0f);
    const float x = -1.442695041f * u * u;                       // -u^2 log2(e)
#ifdef __CUDA_ARCH__
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(q));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x));
#else
    t = 1.0f / q;
    e = exp2f(x);
#endif
    p = fmaf(fmaf(fmaf(fmaf(1.061405429f, t, -1.453152027f), t, 1.421413741f), t, -0.284496736f), t, 0.254829592f);
}

// g(r) at u = r / (2 r_s), u >= 0.
B200_HD inline float treepm_short_g(float u) {
    float e, t, p;
    treepm_erfc_parts(u, e, t, p);
    return e * fmaf(t, p, 1.128379167f * u);                     // 2 / sqrt(pi)
}

// erfc(u), the short-range potential's factor: m erfc(r / 2 r_s) / r.  Absolute error <= 1.5e-7 (the formula's),
// so relative <= 2e-7 for u <= 0.5 and 1e-4 at u = 2.25 (r = 4.5 r_s), where erfc itself is 1.5e-3.
B200_HD inline float treepm_short_erfc(float u) {
    float e, t, p;
    treepm_erfc_parts(u, e, t, p);
    return e * (t * p);
}

}  // namespace b200
