// pm.cu -- periodic particle-mesh (PM) gravity: the solver the reference reserves the factory name
// "PMForceComputer" for (src/forces/force_computer_factory.cpp:40-63) and never implements.  The true periodic
// force of the box (uniform neutralising background), O(N + G^3 log G), defined with a Gaussian split radius so that
// it is the long-range half of TreePM from the start.  G = 1; box L, mesh G^3, h = L / G, r_s = r_split:
//
//   wrap + cell   x -> x - L floor(x / L); mesh point i at i h (diag.cu's cic_kernel); cell floor(x / h) mod G
//   deposit       rho = sum m W_CIC / h^3 in int64 fixed point (below), minus the exact mean (k = 0 mode zero)
//   potential     phi_k = -4 pi rho_k exp(-k^2 r_s^2) / (k^2 W(k)^2), W(k) = prod_a sinc^2(k_a h / 2)
//                 (W divided out once for the assignment, once for the interpolation, as GADGET-2)
//   gradient      a_k = -i k_a phi_k, zero on the Nyquist plane of axis a; three C2R; CIC gather at the targets
//   potential out phi = -(interpolated mesh potential), positive, long range only (self term included)
//
// Determinism.  The deposit is the only reduction with a free order.  Each contribution m W is rounded once to an
// integer number of quanta 1 / S, S = 2^e chosen from n * max|m| so that the whole mesh sums below 2^61, and summed
// in int64: integer addition is associative, so the mesh is bitwise the same whatever the storage order of the
// sources, the CTA that handles them or the order in which atomics land.  A CTA first aggregates its contributions
// in a shared-memory hash table (cell -> int64) and flushes each non-zero cell with one global atomic: particles
// stored along a space-filling curve (b200_spatial_order_dev) touch few cells per CTA, so most of the 8N CIC
// contributions never reach global memory.  Random order fills the table to 3/4 and sends the rest straight to
// global atomics -- slower, same integers.  Everything after the deposit is a fixed sequence of element-wise
// kernels, cuFFT transforms and a per-target gather, so a rank computing only part of the targets gets the same
// bits for them as a rank computing all of them.
//
// Buffers (PmState, kept on the context and sized per grid): the int64 mesh, four float G^3 meshes (the density
// in the first, later the three accelerations and the potential), four complex half-spectra.  The k-space kernel
// reads rho_k once and writes all three gradient spectra (and phi_k in place of rho_k): one pass over the
// spectrum instead of one per component, for 3 more complex buffers -- memory is the cheap side here (G = 512:
// 2.2 GB of spectra on a 180 GB card), HBM passes are not.  cuFFT C2R may overwrite its input, which is why each
// spectrum is transformed once.
#include <math.h>
#include <new>
#include <string.h>

#include "common.cuh"
#include "fft.cuh"
#include "pm.cuh"

namespace b200 {

struct PmState {
    int grid = 0;
    cufftHandle r2c = 0, c2r = 0;
    bool plans = false;
    DevBuf mesh;     // int64 fixed-point mass, grid^3
    DevBuf real;     // 4 x float grid^3: density (R2C input), then a_x, a_y, a_z, potential (C2R outputs)
    DevBuf cplx;     // 4 x complex grid^2 (grid/2+1): rho_k (phi_k in place), a_x,k, a_y,k, a_z,k
    DevBuf scal;     // u32 max |m| bits, pad, i64 fixed-point total
    cudaEvent_t ev[PM_PHASES] = {};
    bool timed = false;
};

namespace {

constexpr unsigned FULLMASK = 0xffffffffu;
constexpr int DEP_THREADS = 256;
constexpr int DEP_PER_THREAD = 4;
constexpr int DEP_PER_CTA = DEP_THREADS * DEP_PER_THREAD;
constexpr int TABLE_BITS = 12;
constexpr int TABLE = 1 << TABLE_BITS;               // 4096 cells: 1024 Hilbert-ordered particles touch ~1300
constexpr int TABLE_FILL = TABLE * 3 / 4;            // past this the table is left alone (random storage order)
constexpr int MAX_PROBE = 16;
constexpr size_t DEP_SMEM = TABLE * (sizeof(unsigned long long) + sizeof(int)) + 16;

// Cell index along one axis and the CIC fraction towards the next mesh point.
__device__ __forceinline__ void pm_cell(float p, float box, float inv_h, int G, int& i, float& f) {
    const float x = p - box * floorf(p * (inv_h / (float)G));       // multiply: no IEEE divide subroutine
    const float u = x * inv_h;
    const float fl = floorf(u);
    f = u - fl;
    i = (int)fl % G;                 // u may round to G (x just below L) or below 0 (x = -0 ulp)
    if (i < 0) i += G;
}

// Fixed-point scale: a power of two with S * n * max|m| < 2^61, so the mesh (and its total) cannot overflow.
__device__ __forceinline__ double pm_scale(unsigned mmax_bits, long long n) {
    const double bound = (double)__uint_as_float(mmax_bits) * (double)n;
    if (!(bound > 0.0) || isinf(bound)) return 1.0;
    return ldexp(1.0, 60 - ilogb(bound));
}

__global__ void __launch_bounds__(256)
pm_mass_bound_kernel(const float4* __restrict__ posm, long long n, unsigned* __restrict__ mmax_bits) {
    unsigned mx = 0u;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        mx = max(mx, __float_as_uint(fabsf(posm[i].w)));      // non-negative floats order as unsigned ints
    mx = __reduce_max_sync(FULLMASK, mx);
    if ((threadIdx.x & 31) == 0) atomicMax(mmax_bits, mx);
}

__device__ __forceinline__ void pm_table_add(int* keys, unsigned long long* vals, int* used, int cell,
                                             unsigned long long q, unsigned long long* __restrict__ mesh) {
    unsigned slot = ((unsigned)cell * 0x9E3779B1u) >> (32 - TABLE_BITS);
    for (int probe = 0; probe < MAX_PROBE; ++probe) {
        const int k = ((volatile int*)keys)[slot];
        if (k == cell) { atomicAdd(&vals[slot], q); return; }
        if (k < 0) {
            if (*(volatile int*)used >= TABLE_FILL) break;
            const int prev = atomicCAS(&keys[slot], -1, cell);
            if (prev < 0) atomicAdd(used, 1);
            if (prev < 0 || prev == cell) { atomicAdd(&vals[slot], q); return; }
        }
        slot = (slot + 1) & (TABLE - 1);
    }
    atomicAdd(&mesh[cell], q);
}

// One CTA per DEP_PER_CTA consecutive sources.  Two's-complement adds, so negative masses sum exactly as well.
__global__ void __launch_bounds__(DEP_THREADS)
pm_deposit_kernel(const float4* __restrict__ posm, long long n, int G, float box, float inv_h,
                  const unsigned* __restrict__ mmax_bits, unsigned long long* __restrict__ mesh,
                  unsigned long long* __restrict__ total) {
    extern __shared__ unsigned long long pm_smem[];
    unsigned long long* vals = pm_smem;
    int* keys = reinterpret_cast<int*>(vals + TABLE);
    int* used = keys + TABLE;
    for (int s = threadIdx.x; s < TABLE; s += DEP_THREADS) { keys[s] = -1; vals[s] = 0ull; }
    if (threadIdx.x == 0) *used = 0;
    __syncthreads();
    const double scale = pm_scale(*mmax_bits, n);
    unsigned long long mine = 0ull;
    const long long base = (long long)blockIdx.x * DEP_PER_CTA + threadIdx.x;
#pragma unroll 1
    for (int j = 0; j < DEP_PER_THREAD; ++j) {
        const long long i = base + (long long)j * DEP_THREADS;
        if (i >= n) break;
        const float4 p = posm[i];
        int ix, iy, iz;
        float fx, fy, fz;
        pm_cell(p.x, box, inv_h, G, ix, fx);
        pm_cell(p.y, box, inv_h, G, iy, fy);
        pm_cell(p.z, box, inv_h, G, iz, fz);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int dx = c >> 2, dy = (c >> 1) & 1, dz = c & 1;
            const float w = (dx ? fx : 1.f - fx) * (dy ? fy : 1.f - fy) * (dz ? fz : 1.f - fz);
            const unsigned long long q = (unsigned long long)__double2ll_rn((double)(p.w * w) * scale);
            if (q == 0ull) continue;
            mine += q;
            const int gx = ix + dx == G ? 0 : ix + dx, gy = iy + dy == G ? 0 : iy + dy, gz = iz + dz == G ? 0 : iz + dz;
            pm_table_add(keys, vals, used, (gx * G + gy) * G + gz, q, mesh);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_down_sync(FULLMASK, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(total, mine);
    __syncthreads();
    for (int s = threadIdx.x; s < TABLE; s += DEP_THREADS) {
        const int key = keys[s];
        if (key >= 0 && vals[s]) atomicAdd(&mesh[key], vals[s]);
    }
}

// Integer mesh -> float density minus the exact mean, straight into the R2C input.  mesh - T / cells is split
// as (mesh - q) - r / cells with T = q cells + r: the integer part is exact, so the DC term never meets FP32.
__global__ void __launch_bounds__(256)
pm_convert_kernel(const long long* __restrict__ mesh, long long cells, const long long* __restrict__ total,
                  const unsigned* __restrict__ mmax_bits, long long n, double inv_cell_volume, float* __restrict__ rho) {
    const double f = inv_cell_volume / pm_scale(*mmax_bits, n);
    const long long T = *total;
    const long long q = T / cells;
    const double frac = (double)(T - q * cells) / (double)cells;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < cells; c += (long long)gridDim.x * blockDim.x)
        rho[c] = (float)(((double)(mesh[c] - q) - frac) * f);
}

__device__ __forceinline__ float pm_sinc(int nn, float inv_g) {     // sin(pi n / G) / (pi n / G)
    if (nn == 0) return 1.f;
    const float v = (float)nn * inv_g;
    return sinpif(v) / ((float)M_PI * v);
}

// Green's function x Gaussian filter x deconvolution (x 1 / G^3 for the unnormalised FFT pair), then the
// spectral gradient; phi_k replaces rho_k when the potential is wanted.
__global__ void __launch_bounds__(256)
pm_kspace_kernel(float2* __restrict__ rhok, float2* __restrict__ axk, float2* __restrict__ ayk,
                 float2* __restrict__ azk, int G, float dk, float rs2, float norm, int want_phi) {
    const int H = G / 2 + 1;
    const long long modes = (long long)G * G * H;
    const float inv_g = 1.f / (float)G;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < modes; t += (long long)gridDim.x * blockDim.x) {
        const int kz = (int)(t % H), ky = (int)((t / H) % G), kx = (int)(t / ((long long)H * G));
        const int nx = kx < G / 2 ? kx : kx - G, ny = ky < G / 2 ? ky : ky - G, nz = kz;
        const float kxv = (float)nx * dk, kyv = (float)ny * dk, kzv = (float)nz * dk;
        const float k2 = kxv * kxv + kyv * kyv + kzv * kzv;
        float green = 0.f;
        if (t != 0) {
            const float s = pm_sinc(nx, inv_g) * pm_sinc(ny, inv_g) * pm_sinc(nz, inv_g);
            const float w = s * s;                                            // W(k)
            green = -4.f * (float)M_PI * norm * expf(-k2 * rs2) / (k2 * w * w);
        }
        const float2 r = rhok[t];
        const float2 phi = make_float2(r.x * green, r.y * green);
        // -i k phi = (k phi.im, -k phi.re)
        axk[t] = kx == G / 2 ? make_float2(0.f, 0.f) : make_float2(kxv * phi.y, -kxv * phi.x);
        ayk[t] = ky == G / 2 ? make_float2(0.f, 0.f) : make_float2(kyv * phi.y, -kyv * phi.x);
        azk[t] = kz == G / 2 ? make_float2(0.f, 0.f) : make_float2(kzv * phi.y, -kzv * phi.x);
        if (want_phi) rhok[t] = phi;
    }
}

__global__ void __launch_bounds__(256)
pm_interp_kernel(const float4* __restrict__ tgt, long long n, int G, float box, float inv_h,
                 const float* __restrict__ ax, const float* __restrict__ ay, const float* __restrict__ az,
                 const float* __restrict__ pot, float* __restrict__ acc3, float* __restrict__ phi) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float4 p = tgt[i];
        int ix, iy, iz;
        float fx, fy, fz;
        pm_cell(p.x, box, inv_h, G, ix, fx);
        pm_cell(p.y, box, inv_h, G, iy, fy);
        pm_cell(p.z, box, inv_h, G, iz, fz);
        float sx = 0.f, sy = 0.f, sz = 0.f, sp = 0.f;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int dx = c >> 2, dy = (c >> 1) & 1, dz = c & 1;
            const float w = (dx ? fx : 1.f - fx) * (dy ? fy : 1.f - fy) * (dz ? fz : 1.f - fz);
            const int gx = ix + dx == G ? 0 : ix + dx, gy = iy + dy == G ? 0 : iy + dy, gz = iz + dz == G ? 0 : iz + dz;
            const size_t cell = ((size_t)gx * G + gy) * G + gz;
            sx += w * ax[cell];
            sy += w * ay[cell];
            sz += w * az[cell];
            if (pot) sp += w * pot[cell];
        }
        acc3[3 * i] = sx;
        acc3[3 * i + 1] = sy;
        acc3[3 * i + 2] = sz;
        if (phi) phi[i] = -sp;
    }
}

void destroy_plans(PmState& s) {
    const CufftApi* fft = cufft();
    if (s.plans && fft) { fft->Destroy(s.r2c); fft->Destroy(s.c2r); }
    s.plans = false;
    s.grid = 0;
}

}  // namespace

int pm_forces(b200_ctx* ctx, const void* posm4, size_t n_sources, size_t i0, size_t n_targets, int grid, float box,
              float r_split, void* acc3, void* phi, cudaStream_t st) {
    const CufftApi* fft = cufft();
    if (!fft) return B200_ERR_UNSUPPORTED;
    if (!ctx->pm) {
        B200_CUDA(cudaFuncSetAttribute(pm_deposit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DEP_SMEM));
        ctx->pm = new (std::nothrow) PmState();
        if (!ctx->pm) return B200_ERR_NOMEM;
    }
    PmState& s = *ctx->pm;
    const long long G = grid, cells = G * G * G;
    const size_t modes = (size_t)G * G * (G / 2 + 1);
    B200_TRY(s.mesh.reserve((size_t)cells * sizeof(long long)));
    B200_TRY(s.real.reserve(4 * (size_t)cells * sizeof(float)));
    B200_TRY(s.cplx.reserve(4 * modes * sizeof(float2)));
    B200_TRY(s.scal.reserve(2 * sizeof(long long)));
    if (s.grid != grid) {
        destroy_plans(s);
        B200_FFT(fft->Plan3d(&s.r2c, grid, grid, grid, CUFFT_R2C));
        const cufftResult e = fft->Plan3d(&s.c2r, grid, grid, grid, CUFFT_C2R);
        if (e != CUFFT_SUCCESS) { fft->Destroy(s.r2c); return 3000 + (int)e; }
        s.plans = true;
        s.grid = grid;
    }
    if (ctx->timing && !s.timed) {
        for (int k = 0; k < PM_PHASES; ++k) B200_CUDA(cudaEventCreate(&s.ev[k]));
        s.timed = true;
    }
    const bool timing = ctx->timing;
    auto mark = [&](int k) { if (timing) cudaEventRecord(s.ev[k], st); };

    float* real = s.real.as<float>();
    float2* cplx = s.cplx.as<float2>();
    unsigned* mmax = s.scal.as<unsigned>();
    long long* total = s.scal.as<long long>() + 1;
    const float inv_h = (float)grid / box;
    const long long n = (long long)n_sources;
    const int pg = ctx->sm_count * 8;

    mark(0);
    B200_CUDA(cudaMemsetAsync(s.mesh.p, 0, (size_t)cells * sizeof(long long), st));
    B200_CUDA(cudaMemsetAsync(s.scal.p, 0, 2 * sizeof(long long), st));
    pm_mass_bound_kernel<<<pg, 256, 0, st>>>((const float4*)posm4, n, mmax);
    pm_deposit_kernel<<<ceil_div_i(n, DEP_PER_CTA), DEP_THREADS, DEP_SMEM, st>>>(
        (const float4*)posm4, n, grid, box, inv_h, mmax, s.mesh.as<unsigned long long>(), (unsigned long long*)total);
    B200_CUDA(cudaGetLastError());
    mark(1);
    const double h = (double)box / grid;
    pm_convert_kernel<<<pg, 256, 0, st>>>(s.mesh.as<long long>(), cells, total, mmax, n, 1.0 / (h * h * h), real);
    B200_CUDA(cudaGetLastError());
    mark(2);
    B200_FFT(fft->SetStream(s.r2c, st));
    B200_FFT(fft->ExecR2C(s.r2c, real, (cufftComplex*)cplx));
    mark(3);
    pm_kspace_kernel<<<pg, 256, 0, st>>>(cplx, cplx + modes, cplx + 2 * modes, cplx + 3 * modes, grid,
                                         2.0f * (float)M_PI / box, r_split * r_split, 1.0f / (float)cells, phi != nullptr);
    B200_CUDA(cudaGetLastError());
    mark(4);
    B200_FFT(fft->SetStream(s.c2r, st));
    for (int a = 0; a < 3; ++a)
        B200_FFT(fft->ExecC2R(s.c2r, (cufftComplex*)(cplx + (size_t)(a + 1) * modes), real + (size_t)a * cells));
    if (phi) B200_FFT(fft->ExecC2R(s.c2r, (cufftComplex*)cplx, real + 3 * (size_t)cells));
    mark(5);
    pm_interp_kernel<<<pg, 256, 0, st>>>((const float4*)posm4 + i0, (long long)n_targets, grid, box, inv_h, real,
                                         real + cells, real + 2 * cells, phi ? real + 3 * cells : nullptr,
                                         (float*)acc3, (float*)phi);
    B200_CUDA(cudaGetLastError());
    mark(6);
    ctx->launches += 5;
    return B200_OK;
}

int pm_phase_ms(b200_ctx* ctx, float ms[PM_PHASES]) {
    if (!ctx->timing || !ctx->pm || !ctx->pm->timed) return B200_ERR_STATE;
    PmState& s = *ctx->pm;
    B200_CUDA(cudaEventSynchronize(s.ev[PM_PHASES - 1]));
    for (int k = 0; k + 1 < PM_PHASES; ++k) B200_CUDA(cudaEventElapsedTime(&ms[k], s.ev[k], s.ev[k + 1]));
    B200_CUDA(cudaEventElapsedTime(&ms[PM_PHASES - 1], s.ev[0], s.ev[PM_PHASES - 1]));
    return B200_OK;
}

void pm_destroy(b200_ctx* ctx) {
    if (!ctx->pm) return;
    PmState& s = *ctx->pm;
    destroy_plans(s);
    s.mesh.release(); s.real.release(); s.cplx.release(); s.scal.release();
    if (s.timed)
        for (int k = 0; k < PM_PHASES; ++k) cudaEventDestroy(s.ev[k]);
    delete ctx->pm;
    ctx->pm = nullptr;
}

}  // namespace b200
