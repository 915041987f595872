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
#include "blockstep.cuh"

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

// ---- hierarchical time steps: the sync-point pass (DESIGN 3.14) ----------------------------------------------------
// Bin thresholds of the time-step criterion: t[b] = float(dlna^2 / 4^b) for b <= L (host-computed, double first).
struct BinThresholds { float t[BLOCK_MAX_BINS]; };

// The smallest b < L with t[b] |g| <= crit, else L (a non-finite |g| fails every test); |g| with one rounding per
// operation in a fixed order, so that numpy restates it bit for bit.
__device__ __forceinline__ int desired_bin(float gx, float gy, float gz, const BinThresholds& thr, float crit, int L) {
    const float g = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(gx, gx), __fmul_rn(gy, gy)), __fmul_rn(gz, gz)));
    for (int b = 0; b < L; ++b)
        if (__fmul_rn(thr.t[b], g) <= crit) return b;
    return L;
}

constexpr int BK_THREADS = 128;
constexpr int BK_PER = 2;
constexpr int BK_TILE = BK_THREADS * BK_PER;           // 256 particles, 192 float4 words per 3-float array; 2048
                                                       // threads per SM (at 8 CTAs of 512 particles, 1024, the
                                                       // pass took twice leapfrog_kernel's time per byte)
constexpr int BK_WORDS = 3 * BK_TILE / 4;

// Floats [0, nf) of a tile's 3-float rows between global and shared memory: whole 16-byte words as vectors (lane l
// of a warp moves bytes [16 l, 16 l + 16) of a 512-byte run), the one word that the ragged end of n cuts, by floats.
__device__ __forceinline__ void bk_load(float* __restrict__ s, const float* __restrict__ g, int nf) {
    for (int w = threadIdx.x; w < BK_WORDS; w += BK_THREADS) {
        if (4 * w + 4 <= nf) reinterpret_cast<float4*>(s)[w] = reinterpret_cast<const float4*>(g)[w];
        else for (int q = 4 * w; q < nf && q < 4 * w + 4; ++q) s[q] = g[q];
    }
}
__device__ __forceinline__ void bk_store(float* __restrict__ g, const float* __restrict__ s, int nf) {
    for (int w = threadIdx.x; w < BK_WORDS; w += BK_THREADS) {
        if (4 * w + 4 <= nf) reinterpret_cast<float4*>(g)[w] = reinterpret_cast<const float4*>(s)[w];
        else for (int q = 4 * w; q < nf && q < 4 * w + 4; ++q) g[q] = s[q];
    }
}

__device__ __forceinline__ void kick3(float* v, const float* a, float m, float minv, float dt) {
    v[0] = kick1(v[0], a[0], m, minv, dt, 1.0f);
    v[1] = kick1(v[1], a[1], m, minv, dt, 1.0f);
    v[2] = kick1(v[2], a[2], m, minv, dt, 1.0f);
}

// Sync point k of a PM step of S = 2^L sub-steps: closing kicks, rebinning, opening kicks, bin histogram, and with
// drift != 0 the drift of every particle.  fac holds the opening kicks Ko[b][j] at (2^b - 1) + j and the closing
// kicks Kc[b][j] 2^(L+1) - 1 further; Ko[0][0] and Kc[0][0] are also the long-range kicks.  mom, and at k = S acc,
// are written back for the whole tile.
__global__ void __launch_bounds__(BK_THREADS, 16)
block_kick_kernel(float4* __restrict__ posm, float* __restrict__ mom3, float* __restrict__ acc3,
                  const float* __restrict__ long3, const float* __restrict__ short3, unsigned char* __restrict__ bins,
                  long long n, int k, int L, const float* __restrict__ fac, float crit, BinThresholds thr,
                  unsigned* __restrict__ hist, float drift, float box) {
    __shared__ __align__(16) float sv[3 * BK_TILE], sa[3 * BK_TILE], sl[3 * BK_TILE], ss[3 * BK_TILE];
    __shared__ unsigned sh_hist[BLOCK_MAX_BINS];
    const int S = 1 << L;
    const float* Ko = fac;
    const float* Kc = fac + ((2 << L) - 1);
    if (threadIdx.x < BLOCK_MAX_BINS) sh_hist[threadIdx.x] = 0;
    const long long n_tiles = (n + BK_TILE - 1) / BK_TILE;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long base = tile * BK_TILE;
        const int m = (int)(n - base < BK_TILE ? n - base : BK_TILE);
        bk_load(sv, mom3 + 3 * base, 3 * m);
        if (k > 0 || L > 0) {                               // one bin: at k = 0 every particle kicks with acc
            bk_load(sl, long3 + 3 * base, 3 * m);
            bk_load(ss, short3 + 3 * base, 3 * m);
        }
        if (k == 0) bk_load(sa, acc3 + 3 * base, 3 * m);
        __syncthreads();
#pragma unroll
        for (int j = 0; j < BK_PER; ++j) {
            const int q = j * BK_THREADS + threadIdx.x;
            if (q >= m) continue;
            float* v = sv + 3 * q;
            float* a = sa + 3 * q;
            const float* gl = sl + 3 * q;
            const float* gs = ss + 3 * q;
            float4 p = posm[base + q];
            const float mass = p.w, minv = __fdiv_rn(1.0f, mass);
            int b = block_bin(bins[base + q], L);
            bool open = false;
            if (k == 0) {                                   // every step starts: rebin from the stored total
                b = desired_bin(a[0], a[1], a[2], thr, crit, L);
                open = true;
            } else if (block_active(b, k, L)) {             // the step of bin b ends at k
                const float kc = Kc[(1 << b) - 1 + (k >> (L - b)) - 1];
                if (k == S) {
                    a[0] = __fadd_rn(gl[0], gs[0]); a[1] = __fadd_rn(gl[1], gs[1]); a[2] = __fadd_rn(gl[2], gs[2]);
                    if (b == 0) {
                        kick3(v, a, mass, minv, kc);
                    } else {
                        kick3(v, gl, mass, minv, Kc[0]);
                        kick3(v, gs, mass, minv, kc);
                    }
                } else {
                    kick3(v, gs, mass, minv, kc);
                    const int lo = L - (__ffs(k) - 1);       // the longest step that starts on its own grid at k
                    const int want = desired_bin(__fadd_rn(gl[0], gs[0]), __fadd_rn(gl[1], gs[1]),
                                                 __fadd_rn(gl[2], gs[2]), thr, crit, L);
                    b = want > lo ? want : lo;
                    open = true;
                }
            }
            if (open) {                                     // k < S: the (new) step of bin b starts at k
                const float ko = Ko[(1 << b) - 1 + (k >> (L - b))];
                if (k == 0 && b == 0) {
                    kick3(v, a, mass, minv, ko);
                } else {
                    if (k == 0) kick3(v, gl, mass, minv, Ko[0]);
                    kick3(v, gs, mass, minv, ko);
                }
            }
            if (drift != 0.f) {
                p.x = drift1(p.x, v[0], drift, box);
                p.y = drift1(p.y, v[1], drift, box);
                p.z = drift1(p.z, v[2], drift, box);
                posm[base + q] = p;
            }
            bins[base + q] = (unsigned char)b;
            atomicAdd(&sh_hist[b], 1u);
        }
        __syncthreads();
        bk_store(mom3 + 3 * base, sv, 3 * m);
        if (k == S) bk_store(acc3 + 3 * base, sa, 3 * m);
        __syncthreads();                                    // sv / sa are refilled by the next tile
    }
    if (threadIdx.x < BLOCK_MAX_BINS && sh_hist[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh_hist[threadIdx.x]);
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

int block_kick(b200_ctx* ctx, void* posm4, void* mom3, void* acc3, const void* acc_long3, const void* acc_short3,
               void* bins_u8, size_t n, int k, int max_bins, const void* factors, float crit, double dlna,
               void* hist_u32, float drift, float box, cudaStream_t st) {
    if (max_bins < 1 || max_bins > BLOCK_MAX_BINS) return B200_ERR_INVALID;
    const int L = max_bins - 1;
    if (k < 0 || k > (1 << L)) return B200_ERR_INVALID;
    if (!isfinite(drift) || (k == (1 << L) && drift != 0.f)) return B200_ERR_INVALID;
    if (!(crit >= 0.f) || !(dlna >= 0.0) || !isfinite(dlna)) return B200_ERR_INVALID;
    if (!posm4 || !mom3 || !acc3 || !acc_long3 || !acc_short3 || !bins_u8 || !factors || !hist_u32)
        return B200_ERR_INVALID;
    if (((uintptr_t)posm4 | (uintptr_t)mom3 | (uintptr_t)acc3 | (uintptr_t)acc_long3 | (uintptr_t)acc_short3) & 15)
        return B200_ERR_INVALID;
    if (((uintptr_t)factors | (uintptr_t)hist_u32) & 3) return B200_ERR_INVALID;
    B200_CUDA(cudaMemsetAsync(hist_u32, 0, BLOCK_MAX_BINS * sizeof(unsigned), st));
    if (n == 0) return B200_OK;
    BinThresholds thr = {};
    for (int b = 0; b <= L; ++b) thr.t[b] = (float)(dlna * dlna / ldexp(1.0, 2 * b));
    const long long tiles = ((long long)n + BK_TILE - 1) / BK_TILE;
    const long long cap = (long long)ctx->sm_count * 16;   // 16 CTAs per SM (12 KB of shared memory, 32 registers)
    block_kick_kernel<<<(unsigned)(tiles < cap ? tiles : cap), BK_THREADS, 0, st>>>(
        (float4*)posm4, (float*)mom3, (float*)acc3, (const float*)acc_long3, (const float*)acc_short3,
        (unsigned char*)bins_u8, (long long)n, k, L, (const float*)factors, crit, thr, (unsigned*)hist_u32, drift, box);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
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
