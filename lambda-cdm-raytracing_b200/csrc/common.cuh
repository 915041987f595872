// common.cuh -- context, error plumbing and small device helpers shared by the
// sm_100a kernels of libb200grav.so.
#pragma once
// -DB200_BOUNDS_CHECK (make check-build): device-side asserts on the indices the tree kernels compute -- the
// in-tree stand-in for compute-sanitizer, which is not available on the pool (tools/bounds_check.sh).
#ifdef B200_BOUNDS_CHECK
#include <assert.h>
#define B200_DEV_ASSERT(c) assert(c)
#else
#define B200_DEV_ASSERT(c) ((void)0)
#endif

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "b200grav.h"

#define B200_CUDA(call)                                   \
    do {                                                  \
        cudaError_t e__ = (call);                         \
        if (e__ != cudaSuccess) return 1000 + (int)e__;   \
    } while (0)

#define B200_TRY(call)                  \
    do {                                \
        int s__ = (call);               \
        if (s__ != B200_OK) return s__; \
    } while (0)

// A growable device buffer owned by the context.
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int reserve(size_t need) {
        if (need <= bytes) return B200_OK;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        size_t want = need + need / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { cudaGetLastError(); return B200_ERR_NOMEM; }
        bytes = want;
        return B200_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
    template <class T> T* as() const { return (T*)p; }
};

namespace b200 { struct TreeState; struct ShardState; struct PmState; }   // tree.cu, shard.cu, pm.cu

constexpr int B200_MAX_KERNEL_CFG = 64;
struct KernelCfg { const void* fn; int blocks_per_sm; };   // per-device launch configuration of a kernel instance

struct b200_ctx {
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;        // the context's own stream (host entry points)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timing = false;
    float last_ms = 0.f;
    uint64_t launches = 0;
    KernelCfg kernel_cfg[B200_MAX_KERNEL_CFG];
    int n_kernel_cfg = 0;

    // direct sum scratch
    DevBuf src_tiles;       // tile-SoA sources
    DevBuf partials;        // per (CTA, target block) partial accelerations
    DevBuf zero_flag;       // int that always reads 0 (equal-mass promise of the parts API)
    DevBuf mass_flag;       // int: number of sources whose mass differs from the first
    DevBuf energy_part, energy_phi, energy_out;   // energy diagnostic scratch
    DevBuf ic_wk, ic_tmp, ic_psi, ic_stats;       // initial-conditions scratch (released after each call)
    // host-entry staging
    DevBuf h_pos3, h_vel3, h_mass, h_posm4, h_acc3;
    DevBuf h_tree_posm4;    // particles of the last b200_tree_build_host: stay valid until the next host tree build
    // probe / standalone sort scratch
    DevBuf probe, sort_scratch;

    b200::TreeState* tree = nullptr;
    b200::ShardState* shard = nullptr;    // NCCL communicator (b200_shard_init)
    b200::PmState* pm = nullptr;          // particle-mesh meshes and cuFFT plans, per grid (b200_pm_forces_dev)
};

static inline int ceil_div_i(long long a, long long b) { return (int)((a + b - 1) / b); }
