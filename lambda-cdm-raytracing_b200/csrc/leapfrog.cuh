#pragma once
#include "common.cuh"
namespace b200 {
int leapfrog(b200_ctx* ctx, void* posm4, void* vel3, const void* acc3, size_t n, int n_kicks,
             float dt_kick, double a, float dt_drift, float box, cudaStream_t st);
int unpack_pos3(b200_ctx* ctx, const void* posm4, size_t n, void* pos3, cudaStream_t st);
int scatter_rows(b200_ctx* ctx, const void* src4, const void* perm, size_t n, void* dst4, cudaStream_t st);
int gather_rows(b200_ctx* ctx, const void* src4, const void* src3, const void* list, size_t n, void* out4, void* out3,
                cudaStream_t st);
// sync point k of the hierarchical time steps (b200_block_kick_dev)
int block_kick(b200_ctx* ctx, void* posm4, void* mom3, void* acc3, const void* acc_long3, const void* acc_short3,
               void* bins_u8, size_t n, int k, int max_bins, const void* factors, float crit, double dlna,
               void* hist_u32, float drift, float box, cudaStream_t st);
int pack_posm(b200_ctx* ctx, const void* pos3, const void* mass, size_t n, void* posm4,
              cudaStream_t st);
}
