// blockstep.cuh -- the step-bin rule of the hierarchical (block) time steps, shared by the sync-point pass
// (leapfrog.cu, block_kick) and the active short-range walk (tree.cu, tree_walk_short_active).
#pragma once

namespace b200 {

constexpr int BLOCK_MAX_BINS = 16;

// A PM step is S = 2^L sub-steps (L = max_bins - 1); bin b steps 2^(L - b) of them.  A stored bin above L (not one
// a pass wrote) is read as L.
__device__ __forceinline__ int block_bin(unsigned char b, int L) { return b > L ? L : (int)b; }

// The particle's step (bin b) ends, and its next one starts, at sync point k: k is a multiple of 2^(L - b).
__device__ __forceinline__ bool block_active(int b, int k, int L) { return (k & ((1 << (L - b)) - 1)) == 0; }

}  // namespace b200
