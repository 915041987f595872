// direct.cu -- softened direct-sum gravity for sm_100a (rows D1-D3 of SURVEY 8a).
//
// Replaces: the CPU leaf pair loop (reference src/forces/tree_force_computer.cpp:
// 312-347), compute_forces_direct / compute_forces_tiled
// (src/physics/lambda_cdm_kernels.cu:14-56, 144-221) and nbody_force_kernel_shared
// (src/tensorrt/nbody_plugins.cu:53-129).  Not a translation of any of them:
//
//  * sources live in HBM as 8 KB tile-SoA blocks  [tile][x|y|z|m][512]  so one
//    TMA bulk copy (cp.async.bulk + mbarrier, SASS UBLKCP) lands a tile in
//    shared memory already split by component;
//  * the inner loop is written in packed FP32 (fma/mul/add .f32x2 -> FFMA2 /
//    FMUL2 / FADD2): one instruction handles the SAME target against TWO
//    consecutive sources, whose x/y/z/m pairs are adjacent 64-bit words of the
//    smem tile, so no register shuffling is needed; each LDS.128 broadcast
//    feeds 4 sources x R register-blocked targets;
//  * 12 FP32-pipe lane-ops + 1 MUFU.RSQ per interaction (3 sub, 3 fma for
//    r^2+eps^2, rsqrt, 3 mul for m*rinv^3, 3 fma accumulate); no i==j branch
//    (eps > 0 makes the self term exactly 0).  When every source has the same
//    mass (all the reference's generators emit m = 1) a specialised instance
//    drops the mass multiply and the mass LDS -- 11 lane-ops -- and the common
//    mass is applied once in the finalize pass.  Which instance runs is decided
//    on the device (the packer counts masses that differ from the first one),
//    so no host synchronisation is needed: both are enqueued, one returns at
//    its first instruction;
//  * the (target block x source tile) work space is flattened and cut into
//    gridDim.x equal contiguous spans, gridDim.x = SMs x resident CTAs, so
//    there is no tail wave for any N; a span that crosses target-block
//    boundaries writes one partial record per block, and a finalize pass adds
//    the (few) records of a block in fixed order -> deterministic results;
//  * per-tile FP32 partial sums are folded into FP64 running sums, so the
//    round-off does not grow like sqrt(N_sources) (the sequential FP32 CPU
//    loop is 8.6e-6 from FP64 truth at 64 K sources already).
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "direct.cuh"

namespace b200 {

namespace {

typedef unsigned long long u64;

__device__ __forceinline__ u64 pk(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpk(u64 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
    u64 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
    u64 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
    u64 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on an mbarrier.
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes,
                                            uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// -------------------------------------------------------------------------
// float4 (x,y,z,m) -> tile-SoA.  Slots past n are zero-mass sources parked far
// away (1e18): m = 0 silences them in the general kernel, and in the
// equal-mass kernel rinv^3 underflows to exactly 0.
// mass_diff counts sources whose mass differs from the first one.
constexpr float FAR_AWAY = 1.0e18f;

__global__ void pack_tiles_kernel(const float4* __restrict__ posm, long long n, long long n_padded,
                                  float* __restrict__ tiles, int* __restrict__ mass_diff) {
    long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_padded) return;
    float4 p = make_float4(FAR_AWAY, FAR_AWAY, FAR_AWAY, 0.f);
    if (j < n) {
        p = posm[j];
        if (mass_diff && p.w != posm[0].w) atomicAdd(mass_diff, 1);
    }
    long long t = j / DIRECT_TILE_J;
    int o = (int)(j % DIRECT_TILE_J);
    float* base = tiles + t * (4 * DIRECT_TILE_J) + o;
    base[0 * DIRECT_TILE_J] = p.x;
    base[1 * DIRECT_TILE_J] = p.y;
    base[2 * DIRECT_TILE_J] = p.z;
    base[3 * DIRECT_TILE_J] = p.w;
}

constexpr int STAGES = 4;
constexpr int TILE_J = DIRECT_TILE_J;
constexpr int TILE_FLOATS = 4 * TILE_J;
constexpr uint32_t TILE_BYTES = TILE_FLOATS * sizeof(float);

__device__ __forceinline__ const float* tile_ptr(const DirectSources& src, int t) {
    int p = 0, base = 0;
#pragma unroll 1
    while (p < src.n_parts - 1 && t >= src.tile_end[p]) { base = src.tile_end[p]; ++p; }
    return src.tiles[p] + (size_t)(t - base) * TILE_FLOATS;
}

// R targets per thread, THREADS threads per CTA, MINB CTAs per SM.
// UNIT: every source has the same mass (runs only if *mass_diff == 0);
// !UNIT: general masses (runs only if mass_diff is null or *mass_diff != 0).
// POT: accumulate the potential sum_j m_j / sqrt(|d|^2 + eps^2) (the energy diagnostic,
// compute_energy at src/physics/lambda_cdm_kernels.cu:338-408) instead of the
// acceleration: 7 (equal masses) / 8 lane-ops + 1 MUFU per pair, component 0 of the
// partial records only.
//
// PMODE_OPEN: open boundaries.
// PMODE_FLOAT: periodic, minimum image in FP32 (d - box * rint(d / box) with the 1.5 * 2^23 trick): 9 more
//   FP32-pipe lane-ops per pair, exact with respect to the input floats.
// PMODE_FIXED_XY: periodic, x and y in FIXED POINT.  The CTA rewrites the x and y planes of each landed tile in
//   shared memory as 32-bit integers in units of box / 2^32, so x_j - x_i wraps to the minimum image by itself
//   (IADD3) and I2FP brings it back to FP32 -- both on the ALU pipe, which the FP32-pipe-bound loop leaves idle;
//   z keeps the FP32 minimum image.  Per pair 4 ALU + 13 FP32-pipe lane-ops instead of 20 (+15 % measured; all
//   three components in fixed point is slower again, the two pipes overlap only partly).  a_x, a_y come out in
//   fixed-point units and are rescaled in FP64 by the finalize pass.  Positions are quantised to box * 2^-33
//   (1.2e-8 of a 100 box, 1/300 of a float ulp there), which perturbs the force of a pair closer than eps by
//   up to that over eps, relatively: the dispatcher uses this mode only while eps >= 1e-4 box.  In the
//   equal-mass instance the mass plane of the tile is reused for a per-source eps^2 (+inf in the padding slots,
//   whose rsqrt is then exactly 0).
constexpr int PMODE_OPEN = 0, PMODE_FLOAT = 1, PMODE_FIXED_XY = 2;

// x -> units of box / 2^32, modulo 2^32.  The upper half is shifted down by one unit so that a pair exactly
// half a box apart with both positions in [0, box) keeps the sign of its raw separation, as minimum_image
// (lambda_cdm_kernels.cu:122-141) does; plain modular arithmetic would send both to -box/2.  Outside [0, box)
// the image of such a tie is chosen from the wrapped positions and can take either sign (box 100: x_i = -25,
// x_j = 25 gives -50 here, +50 in the FP32 path).  A non-finite x or y saturates in the conversion (+inf lands
// near box, -inf at 0), so the callers first copy it into z, which carries the NaN to every force.
__device__ __forceinline__ uint32_t fixed_point(float x, double units_per_length) {
    uint32_t e = (uint32_t)(unsigned long long)__double2ll_rn((double)x * units_per_length);
    return e - (e >> 31);
}

// (a - b) + c as ONE opaque instruction.
__device__ __forceinline__ int sub3(uint32_t a, uint32_t b, uint32_t c) {
    int d;
    asm("vsub.s32.s32.s32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

template <int R, int THREADS, int MINB, int PMODE, bool UNIT, bool POT = false>
__global__ void __launch_bounds__(THREADS, MINB)
direct_kernel(const DirectSources src, const float4* __restrict__ targets, long long n_targets,
              float eps2, float box, double* __restrict__ partials, long long n_units, int n_tiles,
              const int* __restrict__ mass_diff) {
    constexpr bool PERIODIC = (PMODE == PMODE_FLOAT);
    constexpr bool FIXED = (PMODE == PMODE_FIXED_XY);
    static_assert(!(FIXED && POT), "the potential keeps the FP32 minimum image");
    if (mass_diff != nullptr) {
        const bool uniform = (*mass_diff == 0);
        if (uniform != UNIT) return;
    } else if (UNIT) {
        return;
    }
    constexpr int BLOCK_I = THREADS * R;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* stage_buf = reinterpret_cast<float*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + STAGES * TILE_BYTES);
    // FP64 running sums live in shared memory (touched once per tile): 3R doubles per
    // thread would otherwise cost 6R registers that the inner loop needs for ILP.
    double* dsum = reinterpret_cast<double*>(smem_raw + STAGES * TILE_BYTES + 64);

    const int tid = threadIdx.x;
    const long long G = gridDim.x, c = blockIdx.x;
    const long long u0 = (c * n_units) / G, u1 = ((c + 1) * n_units) / G;
    if (u0 >= u1) return;
    const long long my_units = u1 - u0;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    long long b = u0 / n_tiles;          // current target block
    int t = (int)(u0 % n_tiles);         // current source tile

    if (tid == 0) {
        int tt = t;
        for (int k = 0; k < STAGES - 1 && k < my_units; ++k) {
            mbar_expect_tx(&full[k], TILE_BYTES);
            tma_load_1d(stage_buf + k * TILE_FLOATS, tile_ptr(src, tt), TILE_BYTES, &full[k]);
            if (++tt == n_tiles) tt = 0;
        }
    }
    int t_issue = (int)((u0 + (STAGES - 1)) % n_tiles);   // tile of unit k + STAGES-1

    [[maybe_unused]] const double units = FIXED ? 4294967296.0 / (double)box : 1.0;
    [[maybe_unused]] const uint32_t zero = (uint32_t)(n_tiles >> 31);      // 0 (n_tiles > 0), opaque to the compiler
    const u64 eps2_2 = pk(eps2, eps2);
    constexpr int RF = FIXED ? 1 : R, RI = FIXED ? R : 1;
    [[maybe_unused]] u64 nxi[RF], nyi[RF];                 // packed (-x_i, -x_i) per register-blocked target
    u64 nzi[R];
    [[maybe_unused]] uint32_t ixi[RI], iyi[RI];            // fixed point: x_i in units of box / 2^32
    auto load_targets = [&](long long blk) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            long long i = blk * BLOCK_I + r * THREADS + tid;
            float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < n_targets) p = targets[i];
            if constexpr (FIXED) {
                if (!isfinite(p.x) || !isfinite(p.y)) p.z = p.x + p.y;    // a NaN or inf must not vanish in the conversion
                ixi[r] = fixed_point(p.x, units);
                iyi[r] = fixed_point(p.y, units);
            } else {
                nxi[r] = pk(-p.x, -p.x);
                nyi[r] = pk(-p.y, -p.y);
            }
            nzi[r] = pk(-p.z, -p.z);
            dsum[(0 * R + r) * THREADS + tid] = 0.0;
            dsum[(1 * R + r) * THREADS + tid] = 0.0;
            dsum[(2 * R + r) * THREADS + tid] = 0.0;
        }
    };
    load_targets(b);

    [[maybe_unused]] u64 inv_box2, magic2, nmagic2, nbox2, len2_2;
    if constexpr (FIXED) {
        const float l = (float)(1.0 / units);
        len2_2 = pk(l * l, l * l);      // (box / 2^32)^2: fixed-point units^2 -> length^2
    }
    if constexpr (PERIODIC || FIXED) {
        float ib = 1.0f / box;
        inv_box2 = pk(ib, ib);
        magic2 = pk(12582912.0f, 12582912.0f);      // 1.5 * 2^23: round-to-nearest-integer trick
        nmagic2 = pk(-12582912.0f, -12582912.0f);
        nbox2 = pk(-box, -box);
    }

    for (long long k = 0; k < my_units; ++k) {
        const int s = (int)(k % STAGES);
        if (tid == 0 && k + (STAGES - 1) < my_units) {
            const int sn = (int)((k + STAGES - 1) % STAGES);
            mbar_expect_tx(&full[sn], TILE_BYTES);
            tma_load_1d(stage_buf + sn * TILE_FLOATS, tile_ptr(src, t_issue), TILE_BYTES, &full[sn]);
        }
        if (++t_issue == n_tiles) t_issue = 0;
        mbar_wait(&full[s], (uint32_t)((k / STAGES) & 1));

        if constexpr (FIXED) {
            // rewrite the landed tile in place: x, y -> fixed point; equal-mass instance: mass plane -> eps^2
            // per source, +inf in the padding slots (parked at 1e18 by the packer)
            float* tile = stage_buf + s * TILE_FLOATS;
            for (int j = tid; j < TILE_J; j += THREADS) {
                const float x = tile[j], y = tile[TILE_J + j];
                if (!isfinite(x) || !isfinite(y)) tile[2 * TILE_J + j] = x + y;   // a NaN or inf must not vanish in the conversion
                tile[j] = __uint_as_float(fixed_point(x, units));
                tile[TILE_J + j] = __uint_as_float(fixed_point(y, units));
                if constexpr (UNIT) tile[3 * TILE_J + j] = (x >= 0.5f * FAR_AWAY) ? __int_as_float(0x7f800000) : eps2;
            }
            __syncthreads();
        }

        const ulonglong2* sx = reinterpret_cast<const ulonglong2*>(stage_buf + s * TILE_FLOATS);
        const ulonglong2* sy = sx + TILE_J / 4;
        const ulonglong2* sz = sy + TILE_J / 4;
        const ulonglong2* sm = sz + TILE_J / 4;

        u64 ax[R], ay[R], az[R];
#pragma unroll
        for (int r = 0; r < R; ++r) ax[r] = ay[r] = az[r] = 0ull;

        auto interact = [&](u64 X, u64 Y, u64 Z, u64 M) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                u64 dx, dy, dz;
                if constexpr (FIXED) {
                    // the 32-bit difference IS the minimum image; IADD3 + I2FP run on the ALU pipe
                    // (the third addend is a run-time zero: a three-input add can only be IADD3, whereas ptxas turns
                    // plain subtractions into IMAD.IADD -- on the FP32 pipe this mode is meant to unload)
                    dx = pk(__int2float_rn(sub3((uint32_t)X, ixi[r], zero)), __int2float_rn(sub3((uint32_t)(X >> 32), ixi[r], zero)));
                    dy = pk(__int2float_rn(sub3((uint32_t)Y, iyi[r], zero)), __int2float_rn(sub3((uint32_t)(Y >> 32), iyi[r], zero)));
                    dz = add2(Z, nzi[r]);
                    dz = fma2(add2(fma2(dz, inv_box2, magic2), nmagic2), nbox2, dz);
                } else {
                    dx = add2(X, nxi[r]);
                    dy = add2(Y, nyi[r]);
                    dz = add2(Z, nzi[r]);
                }
                if constexpr (PERIODIC) {
                    u64 qx = add2(fma2(dx, inv_box2, magic2), nmagic2);      // rint(d / box): 3 lane-ops per component
                    u64 qy = add2(fma2(dy, inv_box2, magic2), nmagic2);
                    u64 qz = add2(fma2(dz, inv_box2, magic2), nmagic2);
                    dx = fma2(qx, nbox2, dx);
                    dy = fma2(qy, nbox2, dy);
                    dz = fma2(qz, nbox2, dz);
                }
                u64 r2;
                if constexpr (FIXED) {      // x, y in fixed-point units, z in length units
                    r2 = fma2(fma2(dy, dy, mul2(dx, dx)), len2_2, fma2(dz, dz, UNIT ? M : eps2_2));
                } else {
                    r2 = fma2(dx, dx, eps2_2);
                    r2 = fma2(dy, dy, r2);
                    r2 = fma2(dz, dz, r2);
                }
                float r2a, r2b;
                unpk(r2, r2a, r2b);
                u64 rinv = pk(rsqrt_approx(r2a), rsqrt_approx(r2b));
                if constexpr (POT) {
                    if constexpr (UNIT) ax[r] = add2(ax[r], rinv);
                    else ax[r] = fma2(M, rinv, ax[r]);
                    continue;
                }
                u64 f = mul2(rinv, rinv);
                if constexpr (UNIT) f = mul2(f, rinv);
                else f = mul2(f, mul2(M, rinv));
                ax[r] = fma2(f, dx, ax[r]);
                ay[r] = fma2(f, dy, ay[r]);
                az[r] = fma2(f, dz, az[r]);
            }
        };

#pragma unroll 1      // one LDS.128 group per iteration: ptxas schedules the 2 x R interaction pairs best when left alone
        for (int j4 = 0; j4 < TILE_J / 4; ++j4) {
            const ulonglong2 X = sx[j4], Y = sy[j4], Z = sz[j4];
            ulonglong2 M = make_ulonglong2(0ull, 0ull);
            if constexpr (!UNIT || FIXED) M = sm[j4];
            interact(X.x, Y.x, Z.x, M.x);
            interact(X.y, Y.y, Z.y, M.y);
        }

#pragma unroll
        for (int r = 0; r < R; ++r) {
            float lo, hi;
            unpk(ax[r], lo, hi); dsum[(0 * R + r) * THREADS + tid] += (double)(lo + hi);
            if constexpr (!POT) {
                unpk(ay[r], lo, hi); dsum[(1 * R + r) * THREADS + tid] += (double)(lo + hi);
                unpk(az[r], lo, hi); dsum[(2 * R + r) * THREADS + tid] += (double)(lo + hi);
            }
        }
        if constexpr (FIXED) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // this CTA wrote the stage
        __syncthreads();      // every warp is done with stage s -> it may be refilled

        ++t;
        const bool last = (k == my_units - 1);
        if (t == n_tiles || last) {
            double* rec = partials + (size_t)(c + b) * 3 * BLOCK_I;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                rec[0 * BLOCK_I + r * THREADS + tid] = dsum[(0 * R + r) * THREADS + tid];
                if constexpr (!POT) {
                    rec[1 * BLOCK_I + r * THREADS + tid] = dsum[(1 * R + r) * THREADS + tid];
                    rec[2 * BLOCK_I + r * THREADS + tid] = dsum[(2 * R + r) * THREADS + tid];
                }
            }
            if (t == n_tiles) {
                t = 0;
                ++b;
                if (!last) load_targets(b);
            }
        }
    }
}

// Adds the partial records of each target block in CTA order (fixed -> the
// result does not depend on scheduling), applies the common mass of the
// equal-mass path, and writes float acc3.
__global__ void direct_finalize_kernel(const double* __restrict__ partials, float* __restrict__ acc3,
                                       long long n_targets, int block_i, long long n_units,
                                       int n_tiles, int G, const int* __restrict__ mass_diff,
                                       const float* __restrict__ first_tile, double scale_xy) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_targets) return;
    long long b = i / block_i;
    int o = (int)(i % block_i);
    long long uf = b * n_tiles, ul = uf + n_tiles - 1;
    long long cf = ((uf + 1) * G - 1) / n_units;
    long long cl = ((ul + 1) * G - 1) / n_units;
    double sx = 0.0, sy = 0.0, sz = 0.0;
    for (long long c = cf; c <= cl; ++c) {
        const double* rec = partials + (size_t)(c + b) * 3 * block_i;
        sx += rec[o];
        sy += rec[block_i + o];
        sz += rec[2 * block_i + o];
    }
    if (mass_diff != nullptr && *mass_diff == 0) {
        const double m0 = (double)first_tile[3 * DIRECT_TILE_J];     // mass of source 0
        sx *= m0; sy *= m0; sz *= m0;
    }
    acc3[3 * i + 0] = (float)(sx * scale_xy);        // fixed-point components come out in their own units
    acc3[3 * i + 1] = (float)(sy * scale_xy);
    acc3[3 * i + 2] = (float)sz;
}

// Potential: phi_i = sum of the block's partial records minus the i == i term (the pair loop
// has no self test: with d = 0 it added m_i * rsqrt(eps^2), the very value subtracted here).
__global__ void potential_finalize_kernel(const double* __restrict__ partials, const float4* __restrict__ targets,
                                          float* __restrict__ phi, long long n_targets, int block_i,
                                          long long n_units, int n_tiles, int G, float eps2,
                                          const int* __restrict__ mass_diff,
                                          const float* __restrict__ first_tile) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_targets) return;
    long long b = i / block_i;
    int o = (int)(i % block_i);
    long long uf = b * n_tiles, ul = uf + n_tiles - 1;
    long long cf = ((uf + 1) * G - 1) / n_units;
    long long cl = ((ul + 1) * G - 1) / n_units;
    double s = 0.0;
    for (long long c = cf; c <= cl; ++c) s += partials[(size_t)(c + b) * 3 * block_i + o];
    const double self = (double)rsqrt_approx(eps2);
    if (mass_diff != nullptr && *mass_diff == 0) s = (s - self) * (double)first_tile[3 * DIRECT_TILE_J];
    else s -= self * (double)targets[i].w;
    phi[i] = (float)s;
}

// KE = sum 1/2 m v^2 and PE = -1/2 sum m_i phi_i over the targets, FP64, two fixed-order stages.
constexpr int ENERGY_BLOCKS = 296;
__global__ void __launch_bounds__(256)
energy_partial_kernel(const float4* __restrict__ targets, const float* __restrict__ vel3,
                      const float* __restrict__ phi, long long n, double* __restrict__ part /*[2][gridDim.x]*/) {
    __shared__ double sk[256], sp[256];
    double ke = 0.0, pe = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float4 p = targets[i];
        const double vx = vel3[3 * i], vy = vel3[3 * i + 1], vz = vel3[3 * i + 2];
        ke += 0.5 * (double)p.w * (vx * vx + vy * vy + vz * vz);
        pe -= 0.5 * (double)p.w * (double)phi[i];
    }
    sk[threadIdx.x] = ke; sp[threadIdx.x] = pe;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) { sk[threadIdx.x] += sk[threadIdx.x + s]; sp[threadIdx.x] += sp[threadIdx.x + s]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { part[blockIdx.x] = sk[0]; part[gridDim.x + blockIdx.x] = sp[0]; }
}
__global__ void energy_final_kernel(const double* __restrict__ part, int nblocks, double* __restrict__ out2) {
    if (threadIdx.x < 2) {
        double s = 0.0;
        for (int b = 0; b < nblocks; ++b) s += part[threadIdx.x * nblocks + b];
        out2[threadIdx.x] = s;
    }
}

template <int R, int THREADS, int MINB, int PMODE, bool POT = false>
int launch_direct(b200_ctx* ctx, const DirectSources& src, const float4* targets, size_t n_targets,
                  float eps, float box, float* acc3, const int* mass_diff, cudaStream_t st) {
    constexpr int BLOCK_I = THREADS * R;
    auto kern_g = direct_kernel<R, THREADS, MINB, PMODE, false, POT>;
    auto kern_u = direct_kernel<R, THREADS, MINB, PMODE, true, POT>;
    const size_t smem = STAGES * TILE_BYTES + 64 + (size_t)3 * R * THREADS * sizeof(double);
    // shared-memory opt-in and occupancy are per (device, kernel instance): cached in the context,
    // which belongs to one device and is used by one host thread at a time
    int blocks_per_sm = 0;
    for (int k = 0; k < ctx->n_kernel_cfg; ++k)
        if (ctx->kernel_cfg[k].fn == (const void*)kern_g) blocks_per_sm = ctx->kernel_cfg[k].blocks_per_sm;
    if (blocks_per_sm == 0) {
        int bu = 0;
        B200_CUDA(cudaFuncSetAttribute(kern_g, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        B200_CUDA(cudaFuncSetAttribute(kern_u, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kern_g, THREADS, smem));
        B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bu, kern_u, THREADS, smem));
        if (bu < blocks_per_sm) blocks_per_sm = bu;      // one grid shape for both instances
        if (blocks_per_sm < 1) return B200_ERR_UNSUPPORTED;
        if (ctx->n_kernel_cfg < B200_MAX_KERNEL_CFG) {
            ctx->kernel_cfg[ctx->n_kernel_cfg].fn = (const void*)kern_g;
            ctx->kernel_cfg[ctx->n_kernel_cfg].blocks_per_sm = blocks_per_sm;
            ++ctx->n_kernel_cfg;
        }
    }
    const long long T = ((long long)n_targets + BLOCK_I - 1) / BLOCK_I;
    const int NT = src.total_tiles;
    const long long U = T * NT;
    long long G = (long long)ctx->sm_count * blocks_per_sm;
    if (G > U) G = U;
    B200_TRY(ctx->partials.reserve((size_t)(G + T) * 3 * BLOCK_I * sizeof(double)));
    if (ctx->timing) B200_CUDA(cudaEventRecord(ctx->ev0, st));
    kern_g<<<(unsigned)G, THREADS, smem, st>>>(src, targets, (long long)n_targets, eps * eps, box,
                                               ctx->partials.as<double>(), U, NT, mass_diff);
    if (mass_diff)
        kern_u<<<(unsigned)G, THREADS, smem, st>>>(src, targets, (long long)n_targets, eps * eps, box,
                                                   ctx->partials.as<double>(), U, NT, mass_diff);
    if (ctx->timing) B200_CUDA(cudaEventRecord(ctx->ev1, st));
    B200_CUDA(cudaGetLastError());
    const int fb = 256;
    if constexpr (POT)
        potential_finalize_kernel<<<(unsigned)((n_targets + fb - 1) / fb), fb, 0, st>>>(
            ctx->partials.as<double>(), targets, acc3, (long long)n_targets, BLOCK_I, U, NT, (int)G, eps * eps,
            mass_diff, src.tiles[0]);
    else {
        // PMODE_FIXED_XY: r in length units, d_x and d_y in fixed-point units of box / 2^32
        const double sxy = PMODE == PMODE_FIXED_XY ? (double)box / 4294967296.0 : 1.0;
        direct_finalize_kernel<<<(unsigned)((n_targets + fb - 1) / fb), fb, 0, st>>>(
            ctx->partials.as<double>(), acc3, (long long)n_targets, BLOCK_I, U, NT, (int)G, mass_diff,
            src.tiles[0], sxy);
    }
    B200_CUDA(cudaGetLastError());
    ctx->launches += mass_diff ? 3 : 2;
    return B200_OK;
}

}  // namespace

size_t direct_tiles_bytes(size_t n) {
    size_t nt = (n + DIRECT_TILE_J - 1) / DIRECT_TILE_J;
    return nt * 4 * DIRECT_TILE_J * sizeof(float);
}

// mass_diff (nullable): device int, zeroed here, then incremented once per
// source whose mass differs from source 0's.
int direct_pack_tiles(b200_ctx* ctx, const void* posm4, size_t n, float* tiles, int* mass_diff,
                      cudaStream_t st) {
    size_t nt = (n + DIRECT_TILE_J - 1) / DIRECT_TILE_J;
    long long n_padded = (long long)nt * DIRECT_TILE_J;
    if (n_padded == 0) return B200_OK;
    if (mass_diff) B200_CUDA(cudaMemsetAsync(mass_diff, 0, sizeof(int), st));
    pack_tiles_kernel<<<(unsigned)((n_padded + 255) / 256), 256, 0, st>>>(
        (const float4*)posm4, (long long)n, n_padded, tiles, mass_diff);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

int direct_forces(b200_ctx* ctx, const DirectSources& src, const void* targets4, size_t n_targets,
                  float eps, float box, void* acc3, const int* mass_diff, cudaStream_t st) {
    if (!(eps > 0.f) || box < 0.f) return B200_ERR_INVALID;
    if (n_targets == 0) return B200_OK;
    if (src.total_tiles <= 0) {
        B200_CUDA(cudaMemsetAsync(acc3, 0, n_targets * 3 * sizeof(float), st));
        return B200_OK;
    }
    const float4* tg = (const float4*)targets4;
    float* out = (float*)acc3;
    // Register blocking: 8 targets/thread (one 256-thread CTA per SM, 2048 targets per block) whenever
    // the flattened (target block x source tile) space gives every CTA several units of work
    // and the last, partly filled target block wastes little; 2 targets/thread below that.
    const long long units8 = (((long long)n_targets + 2047) / 2048) * (long long)src.total_tiles;
    const bool small = n_targets < 4 * 2048 || units8 < 4ll * ctx->sm_count;
    if (const char* v = getenv("B200_DIRECT_VARIANT")) {      // tuning hook: "R,THREADS,MINB"
        int r = 0, th = 0, mb = 0;
        if (sscanf(v, "%d,%d,%d", &r, &th, &mb) == 3 && box > 0.f) {
            const bool fp = getenv("B200_DIRECT_PERIODIC_FLOAT") != nullptr;
#define B200_PVARIANT(RR, TH, MB) \
    if (r == RR && th == TH && mb == MB) \
        return fp ? launch_direct<RR, TH, MB, PMODE_FLOAT>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st) \
                  : launch_direct<RR, TH, MB, PMODE_FIXED_XY>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st);
            B200_PVARIANT(4, 256, 1) B200_PVARIANT(8, 256, 1) B200_PVARIANT(4, 512, 1)
#undef B200_PVARIANT
            return B200_ERR_UNSUPPORTED;
        }
        if (sscanf(v, "%d,%d,%d", &r, &th, &mb) == 3 && box == 0.f) {
#define B200_VARIANT(RR, TH, MB) \
    if (r == RR && th == TH && mb == MB) \
        return launch_direct<RR, TH, MB, PMODE_OPEN>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st);
            B200_VARIANT(2, 256, 2) B200_VARIANT(4, 256, 1) B200_VARIANT(4, 256, 2) B200_VARIANT(5, 256, 1)
            B200_VARIANT(6, 256, 1) B200_VARIANT(8, 256, 1) B200_VARIANT(4, 384, 1) B200_VARIANT(4, 512, 1)
            B200_VARIANT(3, 512, 1) B200_VARIANT(6, 128, 2) B200_VARIANT(8, 128, 2) B200_VARIANT(7, 256, 1)
            B200_VARIANT(6, 384, 1) B200_VARIANT(5, 384, 1) B200_VARIANT(8, 192, 1) B200_VARIANT(6, 320, 1)
            B200_VARIANT(10, 256, 1) B200_VARIANT(5, 128, 3) B200_VARIANT(4, 128, 4)
            B200_VARIANT(2, 256, 3) B200_VARIANT(2, 256, 4) B200_VARIANT(3, 256, 2) B200_VARIANT(3, 256, 3)
            B200_VARIANT(2, 512, 2) B200_VARIANT(2, 1024, 1) B200_VARIANT(1, 256, 8) B200_VARIANT(1, 512, 4)
#undef B200_VARIANT
            return B200_ERR_UNSUPPORTED;
        }
    }
    if (box > 0.f) {
        // fixed-point x, y only while the position quantum (box * 2^-33) is below ~1e-6 eps, and never
        // for small problems (launch-bound anyway); B200_DIRECT_PERIODIC_FLOAT forces the FP32 minimum image (A/B)
        const long long units4 = (((long long)n_targets + 2047) / 2048) * (long long)src.total_tiles;
        const bool fixed_ok = eps >= 1e-4f * box && n_targets >= 4 * 2048 && units4 >= 4ll * ctx->sm_count &&
                              getenv("B200_DIRECT_PERIODIC_FLOAT") == nullptr;
        if (fixed_ok)
            return launch_direct<4, 512, 1, PMODE_FIXED_XY>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st);
        return small ? launch_direct<2, 256, 2, PMODE_FLOAT>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st)
                     : launch_direct<4, 256, 1, PMODE_FLOAT>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st);
    }
    return small ? launch_direct<2, 256, 2, PMODE_OPEN>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st)
                 : launch_direct<8, 256, 1, PMODE_OPEN>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st);
}

// Per-target potential phi_i = sum_{j != i} m_j / sqrt(|d|^2 + eps^2) (positive, G = 1).
int direct_potential(b200_ctx* ctx, const DirectSources& src, const void* targets4, size_t n_targets,
                     float eps, float box, void* phi, const int* mass_diff, cudaStream_t st) {
    if (!(eps > 0.f) || box < 0.f) return B200_ERR_INVALID;
    if (n_targets == 0) return B200_OK;
    if (src.total_tiles <= 0) {
        B200_CUDA(cudaMemsetAsync(phi, 0, n_targets * sizeof(float), st));
        return B200_OK;
    }
    const float4* tg = (const float4*)targets4;
    float* out = (float*)phi;
    const long long units6 = (((long long)n_targets + 1535) / 1536) * (long long)src.total_tiles;
    const bool small = n_targets < 4 * 1536 || units6 < 4ll * ctx->sm_count;
    if (box > 0.f) {
        // always the general-mass instance: a padding slot (parked at 1e18) can wrap to distance 0 -- exactly so
        // when box is a power of two -- where only its zero mass silences it (harmless for forces, d = 0; not
        // for a potential)
        return small ? launch_direct<2, 256, 2, PMODE_FLOAT, true>(ctx, src, tg, n_targets, eps, box, out, nullptr, st)
                     : launch_direct<4, 256, 1, PMODE_FLOAT, true>(ctx, src, tg, n_targets, eps, box, out, nullptr, st);
    }
    return small ? launch_direct<2, 256, 2, PMODE_OPEN, true>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st)
                 : launch_direct<6, 256, 1, PMODE_OPEN, true>(ctx, src, tg, n_targets, eps, box, out, mass_diff, st);
}

// out2 (device): [0] = sum 1/2 m v^2, [1] = -1/2 sum m phi over the n targets.
int energy_reduce(b200_ctx* ctx, const void* targets4, const void* vel3, const void* phi, size_t n,
                  double* out2, cudaStream_t st) {
    B200_TRY(ctx->energy_part.reserve(2 * ENERGY_BLOCKS * sizeof(double)));
    energy_partial_kernel<<<ENERGY_BLOCKS, 256, 0, st>>>((const float4*)targets4, (const float*)vel3,
                                                         (const float*)phi, (long long)n,
                                                         ctx->energy_part.as<double>());
    energy_final_kernel<<<1, 32, 0, st>>>(ctx->energy_part.as<double>(), ENERGY_BLOCKS, out2);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 2;
    return B200_OK;
}

}  // namespace b200
