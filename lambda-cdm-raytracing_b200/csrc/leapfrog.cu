// leapfrog.cu -- fused Lambda-CDM kick/drift for sm_100a (rows L1-L2).
//
// Replaces leapfrog_update (reference src/physics/lambda_cdm_kernels.cu:290-335),
// which is launched three times per step (kick, drift, kick) and touches every
// array each time.  Here one pass applies up to two half-kicks and the drift:
// 40 B read + 28 B written per particle-step instead of 3 x ~40 B.
// Pure HBM streaming.  A CTA owns a tile of 1024 particles; every global access is a
// fully coalesced 128-bit vector (lane l of a warp touches bytes [16 l, 16 l + 16) of a
// 512-byte run): positions as one float4 per particle, velocities and accelerations
// (3 floats per particle, AoS) as the tile's 768 float4 words staged through shared
// memory, where thread t reads floats 3p .. 3p+2 of its particles (stride 3: no bank
// conflicts).  The n mod 1024 particles behind the last full tile go to the tail kernel
// (a thread owns 4 consecutive particles; 128-bit accesses at a 48/64-byte lane stride).
//
// The arithmetic keeps the reference's operation order with one rounding per
// operation (no FMA contraction) so trajectories are bit-identical to the CPU
// restatement given identical accelerations:
//     v += ((acc*m) * (1/m)) * dt * (1/a^2)        (:307-318; F = acc*m, :217-219)
//     x  = fmodf((x + v*dt) + box, box)            (:322-329)
#include "common.cuh"
#include "leapfrog.cuh"

namespace b200 {
namespace {

__device__ __forceinline__ float kick1(float v, float acc, float m, float minv, float dt, float a2inv) {
    float f = __fmul_rn(acc, m);
    f = __fmul_rn(f, minv);
    f = __fmul_rn(f, dt);
    f = __fmul_rn(f, a2inv);
    return __fadd_rn(v, f);
}

__device__ __forceinline__ float drift1(float x, float v, float dt, float box) {
    x = __fadd_rn(x, __fmul_rn(v, dt));
    if (box > 0.f) x = fmodf(__fadd_rn(x, box), box);
    return x;
}

__device__ __forceinline__ void step_particle(float4& p, float& vx, float& vy, float& vz, float ax,
                                              float ay, float az, int n_kicks, float dt_kick,
                                              float a2inv, float dt_drift, float box) {
    const float minv = __fdiv_rn(1.0f, p.w);
    for (int k = 0; k < n_kicks; ++k) {
        vx = kick1(vx, ax, p.w, minv, dt_kick, a2inv);
        vy = kick1(vy, ay, p.w, minv, dt_kick, a2inv);
        vz = kick1(vz, az, p.w, minv, dt_kick, a2inv);
    }
    if (dt_drift != 0.f) {
        p.x = drift1(p.x, vx, dt_drift, box);
        p.y = drift1(p.y, vy, dt_drift, box);
        p.z = drift1(p.z, vz, dt_drift, box);
    }
}

// The particles behind the last full tile of leapfrog_kernel: 4 per thread, the last group scalar.
__global__ void __launch_bounds__(256)
leapfrog_tail_kernel(float4* __restrict__ posm, float4* __restrict__ vel4, const float4* __restrict__ acc4,
                     long long n, int n_kicks, float dt_kick, float a2inv, float dt_drift, float box) {
    const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // group of 4 particles
    const long long i0 = q * 4;
    if (i0 >= n) return;
    if (i0 + 4 <= n) {
        float4 p[4];
        float v[12], a[12];
#pragma unroll
        for (int k = 0; k < 4; ++k) p[k] = posm[i0 + k];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            float4 t = vel4[q * 3 + k];
            v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w;
            float4 u = acc4[q * 3 + k];
            a[4 * k] = u.x; a[4 * k + 1] = u.y; a[4 * k + 2] = u.z; a[4 * k + 3] = u.w;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k)
            step_particle(p[k], v[3 * k], v[3 * k + 1], v[3 * k + 2], a[3 * k], a[3 * k + 1],
                          a[3 * k + 2], n_kicks, dt_kick, a2inv, dt_drift, box);
        if (n_kicks > 0) {
#pragma unroll
            for (int k = 0; k < 3; ++k)
                vel4[q * 3 + k] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
        }
        if (dt_drift != 0.f) {
#pragma unroll
            for (int k = 0; k < 4; ++k) posm[i0 + k] = p[k];
        }
    } else {   // ragged tail: scalar accesses
        float* vel = reinterpret_cast<float*>(vel4);
        const float* acc = reinterpret_cast<const float*>(acc4);
        for (long long i = i0; i < n; ++i) {
            float4 p = posm[i];
            float vx = vel[3 * i], vy = vel[3 * i + 1], vz = vel[3 * i + 2];
            step_particle(p, vx, vy, vz, acc[3 * i], acc[3 * i + 1], acc[3 * i + 2], n_kicks,
                          dt_kick, a2inv, dt_drift, box);
            vel[3 * i] = vx; vel[3 * i + 1] = vy; vel[3 * i + 2] = vz;
            posm[i] = p;
        }
    }
}

// Tile kernel: full tiles of LF_TILE particles only (the host sends the ragged tail to leapfrog_tail_kernel).
constexpr int LF_THREADS = 256;
constexpr int LF_PER = 4;
constexpr int LF_TILE = LF_THREADS * LF_PER;          // 1024 particles, 768 float4 words of vel / acc

__global__ void __launch_bounds__(LF_THREADS)
leapfrog_kernel(float4* __restrict__ posm, float4* __restrict__ vel4, const float4* __restrict__ acc4,
                int n_tiles, int n_kicks, float dt_kick, float a2inv, float dt_drift, float box) {
    __shared__ __align__(16) float sv[3 * LF_TILE];
    __shared__ __align__(16) float sa[3 * LF_TILE];
    const int t = threadIdx.x;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        float4* pt = posm + (size_t)tile * LF_TILE;
        float4* vt = vel4 + (size_t)tile * (3 * LF_TILE / 4);
        const float4* at = acc4 + (size_t)tile * (3 * LF_TILE / 4);
        float4 p[LF_PER];
#pragma unroll
        for (int j = 0; j < LF_PER; ++j) p[j] = pt[j * LF_THREADS + t];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            reinterpret_cast<float4*>(sv)[j * LF_THREADS + t] = vt[j * LF_THREADS + t];
            reinterpret_cast<float4*>(sa)[j * LF_THREADS + t] = __ldg(at + j * LF_THREADS + t);
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < LF_PER; ++j) {
            const int q = 3 * (j * LF_THREADS + t);
            float vx = sv[q], vy = sv[q + 1], vz = sv[q + 2];
            step_particle(p[j], vx, vy, vz, sa[q], sa[q + 1], sa[q + 2], n_kicks, dt_kick, a2inv, dt_drift, box);
            sv[q] = vx; sv[q + 1] = vy; sv[q + 2] = vz;
        }
        __syncthreads();
        if (n_kicks > 0) {
#pragma unroll
            for (int j = 0; j < 3; ++j) vt[j * LF_THREADS + t] = reinterpret_cast<const float4*>(sv)[j * LF_THREADS + t];
        }
        if (dt_drift != 0.f) {
#pragma unroll
            for (int j = 0; j < LF_PER; ++j) pt[j * LF_THREADS + t] = p[j];
        }
        __syncthreads();          // sv / sa are refilled by the next tile
    }
}

__global__ void pack_posm_kernel(const float* __restrict__ pos3, const float* __restrict__ mass,
                                 long long n, float4* __restrict__ posm) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    posm[i] = make_float4(pos3[3 * i], pos3[3 * i + 1], pos3[3 * i + 2], mass ? mass[i] : 1.0f);
}

__global__ void unpack_pos3_kernel(const float4* __restrict__ posm, long long n, float* __restrict__ pos3) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = posm[i];
    pos3[3 * i] = p.x; pos3[3 * i + 1] = p.y; pos3[3 * i + 2] = p.z;
}

__global__ void scatter_rows_kernel(const float4* __restrict__ src, const int* __restrict__ perm, long long n,
                                    float4* __restrict__ dst) {
    long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) dst[perm[k]] = src[k];
}

__global__ void gather_rows_kernel(const float4* __restrict__ src4, const float* __restrict__ src3,
                                   const int* __restrict__ list, long long n, float4* __restrict__ out4,
                                   float* __restrict__ out3) {
    long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const long long i = list[k];
    if (src4) out4[k] = src4[i];
    if (src3) { out3[3 * k] = src3[3 * i]; out3[3 * k + 1] = src3[3 * i + 1]; out3[3 * k + 2] = src3[3 * i + 2]; }
}

}  // namespace

int scatter_rows(b200_ctx* ctx, const void* src4, const void* perm, size_t n, void* dst4, cudaStream_t st) {
    if (n == 0) return B200_OK;
    scatter_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const float4*)src4, (const int*)perm, (long long)n,
                                                                     (float4*)dst4);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

int gather_rows(b200_ctx* ctx, const void* src4, const void* src3, const void* list, size_t n, void* out4, void* out3,
                cudaStream_t st) {
    if (n == 0) return B200_OK;
    gather_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const float4*)src4, (const float*)src3,
                                                                    (const int*)list, (long long)n, (float4*)out4,
                                                                    (float*)out3);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

int unpack_pos3(b200_ctx* ctx, const void* posm4, size_t n, void* pos3, cudaStream_t st) {
    if (n == 0) return B200_OK;
    unpack_pos3_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const float4*)posm4, (long long)n, (float*)pos3);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

int leapfrog(b200_ctx* ctx, void* posm4, void* vel3, const void* acc3, size_t n, int n_kicks,
             float dt_kick, double a, float dt_drift, float box, cudaStream_t st) {
    if (n == 0) return B200_OK;
    if (n_kicks < 0 || n_kicks > 2 || !(a > 0.0)) return B200_ERR_INVALID;
    if (((uintptr_t)vel3 | (uintptr_t)acc3 | (uintptr_t)posm4) & 15) return B200_ERR_INVALID;
    // lambda_cdm_kernels.cu:308: const float a2_inv = 1.0f / (scale_factor * scale_factor);
    const float a2inv = (float)(1.0f / (a * a));
    const long long full = (long long)n / LF_TILE;                             // particles [0, full * LF_TILE)
    if (full > 0) {
        const long long cap = (long long)ctx->sm_count * 8;                    // 8 CTAs (24 KB of shared memory each) per SM
        leapfrog_kernel<<<(unsigned)(full < cap ? full : cap), LF_THREADS, 0, st>>>(
            (float4*)posm4, (float4*)vel3, (const float4*)acc3, (int)full, n_kicks, dt_kick, a2inv, dt_drift, box);
        ctx->launches += 1;
    }
    const long long done = full * LF_TILE, rest = (long long)n - done;          // tail: a multiple-of-4 offset keeps vel/acc 16-byte aligned
    if (rest > 0) {
        const long long groups = (rest + 3) / 4;
        leapfrog_tail_kernel<<<(unsigned)((groups + 255) / 256), 256, 0, st>>>(
            (float4*)posm4 + done, (float4*)((float*)vel3 + 3 * done), (const float4*)((const float*)acc3 + 3 * done),
            rest, n_kicks, dt_kick, a2inv, dt_drift, box);
        ctx->launches += 1;
    }
    B200_CUDA(cudaGetLastError());
    return B200_OK;
}

int pack_posm(b200_ctx* ctx, const void* pos3, const void* mass, size_t n, void* posm4,
              cudaStream_t st) {
    if (n == 0) return B200_OK;
    pack_posm_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
        (const float*)pos3, (const float*)mass, (long long)n, (float4*)posm4);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

}  // namespace b200
