// diag.cu -- device-side diagnostics (SURVEY 8f N4, with the energy sums of direct.cu):
//
//  * force_error: the tree-vs-direct error measure of the reference's Barnes-Hut example
//    (examples/barnes_hut_test.cu:173-189): per particle |a_test - a_ref| / (|a_ref| + 1e-10),
//    averaged and maximised over the particles -- there a host loop over two D2H copies.
//  * power_spectrum: PowerSpectrumAnalyzer::compute_power_spectrum
//    (src/analysis/power_spectrum.cu:53-84): cloud-in-cell mass assignment (:86-134, a host
//    loop in the reference), density contrast (:161-180), forward FFT normalised by 1/G^3
//    (:182-205; cuFFT R2C :387-423), spherical binning in shells of width 2 pi / L with the
//    half-spectrum multiplicities, x volume, optional shot-noise subtraction volume / G^3
//    (:207-285).  Everything stays on the device; only the G/2 bins come back.
#include <math.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "diag.cuh"
#include "fft.cuh"

namespace b200 {
namespace {

constexpr unsigned FULLMASK = 0xffffffffu;

// ---- force error ---------------------------------------------------------------
__global__ void __launch_bounds__(256)
force_error_kernel(const float* __restrict__ a, const float* __restrict__ b, long long n,
                   double* __restrict__ sum, unsigned int* __restrict__ max_bits) {
    double s = 0.0;
    float mx = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float ex = fabsf(a[3 * i] - b[3 * i]), ey = fabsf(a[3 * i + 1] - b[3 * i + 1]),
                    ez = fabsf(a[3 * i + 2] - b[3 * i + 2]);                                  // :176-178
        const float mag = sqrtf(b[3 * i] * b[3 * i] + b[3 * i + 1] * b[3 * i + 1] + b[3 * i + 2] * b[3 * i + 2]);
        const float rel = sqrtf(ex * ex + ey * ey + ez * ez) / (mag + 1e-10f);                // :184
        s += (double)rel;
        mx = fmaxf(mx, rel);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_down_sync(FULLMASK, s, o);
        mx = fmaxf(mx, __shfl_down_sync(FULLMASK, mx, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(sum, s);
        atomicMax(max_bits, __float_as_uint(mx));          // non-negative floats order as unsigned ints
    }
}

// ---- power spectrum --------------------------------------------------------------
__global__ void __launch_bounds__(256)
cic_kernel(const float4* __restrict__ posm, long long n, int G, float inv_spacing, int mass_weighted,
           float* __restrict__ grid) {
    const float Gf = (float)G;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float4 p = posm[i];
        float x = fmodf(p.x * inv_spacing + Gf, Gf);                                          // :93-101
        float y = fmodf(p.y * inv_spacing + Gf, Gf);
        float z = fmodf(p.z * inv_spacing + Gf, Gf);
        // fmodf keeps the dividend's sign: below -box the reference's formula leaves x negative, and a negative
        // index would write before the grid.  x + G may round to G; (ix + dx) % G folds that back to cell 0.
        if (x < 0.f) x += Gf;
        if (y < 0.f) y += Gf;
        if (z < 0.f) z += Gf;
        const int ix = (int)x, iy = (int)y, iz = (int)z;
        const float fx = x - ix, fy = y - iy, fz = z - iz;
        const float m = mass_weighted ? p.w : 1.0f;
#pragma unroll
        for (int dx = 0; dx < 2; ++dx)
#pragma unroll
            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                for (int dz = 0; dz < 2; ++dz) {
                    const float w = (dx ? fx : 1.f - fx) * (dy ? fy : 1.f - fy) * (dz ? fz : 1.f - fz);   // :113-117
                    const int gx = (ix + dx) % G, gy = (iy + dy) % G, gz = (iz + dz) % G;
                    atomicAdd(&grid[((size_t)gx * G + gy) * G + gz], m * w);                  // :124-129
                }
    }
}

__global__ void __launch_bounds__(256)
grid_sum_kernel(const float* __restrict__ grid, long long cells, double* __restrict__ total) {
    double s = 0.0;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < cells; c += (long long)gridDim.x * blockDim.x)
        s += (double)grid[c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(FULLMASK, s, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(total, s);
}

__global__ void __launch_bounds__(256)
contrast_kernel(float* __restrict__ grid, long long cells, const double* __restrict__ total) {
    const float mean = (float)(*total / (double)cells);                                       // :171
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < cells; c += (long long)gridDim.x * blockDim.x)
        grid[c] = mean > 0.0f ? (grid[c] - mean) / mean : 0.0f;                               // :174-179
}

// shells of width dk; per-CTA shared-memory bins (G/2 <= 1024), then one atomic per bin per CTA
__global__ void __launch_bounds__(256)
bin_kernel(const float2* __restrict__ field, int G, float dk, float norm, int n_bins,
           double* __restrict__ power, unsigned long long* __restrict__ counts) {
    extern __shared__ unsigned char smem_raw[];
    double* sp = reinterpret_cast<double*>(smem_raw);
    unsigned int* sc = reinterpret_cast<unsigned int*>(sp + n_bins);
    for (int b = threadIdx.x; b < n_bins; b += blockDim.x) { sp[b] = 0.0; sc[b] = 0u; }
    __syncthreads();
    const int H = G / 2 + 1;
    const long long total = (long long)G * G * H;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int kz = (int)(t % H), ky = (int)((t / H) % G), kx = (int)(t / ((long long)H * G));
        // one IEEE rounding per operation, like the host code: shells whose radius is an exact
        // multiple of dk sit on a bin edge and any contraction would move them
        const float kxv = __fmul_rn((float)((kx <= G / 2) ? kx : kx - G), dk);                // :225-227
        const float kyv = __fmul_rn((float)((ky <= G / 2) ? ky : ky - G), dk);
        const float kzv = __fmul_rn((float)kz, dk);
        const float kmag = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(kxv, kxv), __fmul_rn(kyv, kyv)), __fmul_rn(kzv, kzv)));
        if (kmag == 0.0f) continue;                                                           // :232-233
        const int bin = (int)__fdiv_rn(kmag, dk);                                             // :236
        if (bin >= n_bins) continue;
        const float2 v = field[t];
        const float re = v.x * norm, im = v.y * norm;                                         // :200-204
        const int mult = (kz == 0 || kz == G / 2) ? 1 : 2;                                    // :248
        atomicAdd(&sp[bin], (double)((re * re + im * im) * mult));
        atomicAdd(&sc[bin], (unsigned int)mult);
    }
    __syncthreads();
    for (int b = threadIdx.x; b < n_bins; b += blockDim.x)
        if (sc[b]) { atomicAdd(&power[b], sp[b]); atomicAdd(&counts[b], (unsigned long long)sc[b]); }
}

}  // namespace

int force_error(b200_ctx* ctx, const void* acc_test, const void* acc_ref, size_t n, double* avg, double* max,
                cudaStream_t st) {
    B200_TRY(ctx->energy_out.reserve(2 * sizeof(double)));
    B200_CUDA(cudaMemsetAsync(ctx->energy_out.p, 0, 2 * sizeof(double), st));
    double* sum = ctx->energy_out.as<double>();
    force_error_kernel<<<ctx->sm_count * 4, 256, 0, st>>>((const float*)acc_test, (const float*)acc_ref, (long long)n,
                                                          sum, (unsigned int*)(sum + 1));
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    double h[2];
    B200_CUDA(cudaMemcpyAsync(h, sum, sizeof h, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    unsigned int bits;
    memcpy(&bits, &h[1], sizeof bits);
    float mx;
    memcpy(&mx, &bits, sizeof mx);
    *avg = h[0] / (double)n;
    *max = (double)mx;
    return B200_OK;
}

int power_spectrum(b200_ctx* ctx, const void* posm4, size_t n, int G, float box, int mass_weighted,
                   int shot_noise_correction, float* k_out, float* p_out, int* count_out, cudaStream_t st) {
    const CufftApi* fft = cufft();
    if (!fft) return B200_ERR_UNSUPPORTED;
    const long long cells = (long long)G * G * G;
    const int n_bins = G / 2;                                                                 // :26
    const size_t cplx = (size_t)G * G * (G / 2 + 1) * sizeof(float2);
    B200_TRY(ctx->ic_psi.reserve((size_t)cells * sizeof(float)));       // density grid
    B200_TRY(ctx->ic_wk.reserve(cplx));                                 // delta_k
    B200_TRY(ctx->ic_stats.reserve((1 + 2 * (size_t)n_bins) * sizeof(double)));
    float* grid = ctx->ic_psi.as<float>();
    double* total = ctx->ic_stats.as<double>();
    double* power = total + 1;
    unsigned long long* counts = (unsigned long long*)(power + n_bins);
    B200_CUDA(cudaMemsetAsync(grid, 0, (size_t)cells * sizeof(float), st));                   // :57
    B200_CUDA(cudaMemsetAsync(total, 0, (1 + 2 * (size_t)n_bins) * sizeof(double), st));
    const int pg = ctx->sm_count * 8;
    cic_kernel<<<pg, 256, 0, st>>>((const float4*)posm4, (long long)n, G, (float)G / box, mass_weighted, grid);
    grid_sum_kernel<<<pg, 256, 0, st>>>(grid, cells, total);
    contrast_kernel<<<pg, 256, 0, st>>>(grid, cells, total);
    B200_CUDA(cudaGetLastError());
    cufftHandle plan = 0;
    B200_FFT(fft->Plan3d(&plan, G, G, G, CUFFT_R2C));
    int status = B200_OK;
    cufftResult e = fft->SetStream(plan, st);
    if (e == CUFFT_SUCCESS) e = fft->ExecR2C(plan, grid, (cufftComplex*)ctx->ic_wk.p);
    if (e != CUFFT_SUCCESS) status = 3000 + (int)e;
    if (status == B200_OK) {
        const float dk = 2.0f * (float)M_PI / box;
        bin_kernel<<<pg, 256, (size_t)n_bins * (sizeof(double) + sizeof(unsigned int)), st>>>(
            ctx->ic_wk.as<float2>(), G, dk, 1.0f / (float)cells, n_bins, power, counts);
        if (cudaGetLastError() != cudaSuccess) status = B200_ERR_INVALID;
    }
    ctx->launches += 4;
    std::vector<double> h(1 + 2 * (size_t)n_bins);
    cudaError_t ce = cudaMemcpyAsync(h.data(), total, h.size() * sizeof(double), cudaMemcpyDeviceToHost, st);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(st);          // the plan must outlive its work
    fft->Destroy(plan);
    if (ce != cudaSuccess && status == B200_OK) status = 1000 + (int)ce;
    if (status != B200_OK) return status;
    const float dk = 2.0f * (float)M_PI / box;
    const float volume = box * box * box;
    const unsigned long long* hc = (const unsigned long long*)(h.data() + 1 + n_bins);
    for (int b = 0; b < n_bins; ++b) {
        float p = 0.0f;
        if (hc[b] > 0) p = (float)(h[1 + b] / (double)hc[b]) * volume;                       // :262-267
        if (shot_noise_correction) p -= volume / (float)cells;                                // :271-277
        if (k_out) k_out[b] = (b * dk + (b + 1) * dk) * 0.5f;                                 // :296-298
        if (p_out) p_out[b] = p;
        if (count_out) count_out[b] = (int)hc[b];
    }
    return B200_OK;
}

}  // namespace b200
