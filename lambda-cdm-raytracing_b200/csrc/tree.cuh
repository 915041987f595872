#pragma once
#include "common.cuh"
namespace b200 {
void tree_destroy(b200_ctx* ctx);
int tree_build(b200_ctx* ctx, const void* posm4, size_t n, float box, int leaf_cap, int max_depth,
               bool fixed, float eps, cudaStream_t st);
int tree_walk(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, void* acc3, cudaStream_t st);
// octant-sharded build: part `part` of `n_parts` builds the root, its children and the subtrees of its own octants
int tree_build_part(b200_ctx* ctx, const void* posm4, const int* arrival, size_t n, float box, int leaf_cap,
                    int max_depth, int part, int n_parts, cudaStream_t st);
int tree_forest_publish(b200_ctx* ctx, cudaStream_t st);
int tree_forest_root(b200_ctx* ctx, float out[8]);
// targets given as an explicit list of particle slots; acc3 in list order.  Like tree_walk, it walks the
// published forest when the context holds a part build
int tree_walk_list(b200_ctx* ctx, const int* list, size_t n_list, float theta, void* acc3, cudaStream_t st);
// short-range TreePM walk of the fixed-physics tree in a periodic box, added to acc3
int tree_walk_short(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, float box, float r_split, float r_cut,
                    void* acc3, cudaStream_t st);
// short-range TreePM potential (erfc(r / 2 r_s) / r, minus the PM self term), added to phi; theta <= 1/sqrt(3)
int tree_potential_short(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, float box, float r_split,
                         float r_cut, void* phi, cudaStream_t st);
int tree_set_counting(b200_ctx* ctx, int enabled);
int tree_set_periodic(b200_ctx* ctx, float box);
int tree_potential(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, void* phi, cudaStream_t st);
const void* tree_posm(b200_ctx* ctx);
int tree_counters(b200_ctx* ctx, uint64_t counters[3]);
int tree_walk_stats(b200_ctx* ctx, uint64_t stats[6]);
int tree_overflowed(b200_ctx* ctx, int* flag);
int tree_stats(b200_ctx* ctx, size_t* n_nodes, size_t* n_leaves, size_t* depth, size_t* n_stored);
int tree_export(b200_ctx* ctx, int32_t* level, float* center, float* size, int32_t* first_child,
                int64_t* arrivals, int64_t* part_off, int32_t* part_idx, float* mass, float* com);
}
