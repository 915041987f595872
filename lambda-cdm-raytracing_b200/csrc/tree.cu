// tree.cu -- Barnes-Hut octree for sm_100a: build + centre of mass (rows T3/T4)
// and the theta-criterion walk (rows T5/T6).
//
// Replaces TreeForceComputer::build_tree_cpu / insert_particle / subdivide_node /
// get_octant / compute_center_of_mass (reference src/forces/tree_force_computer.cpp:
// 130-243) and compute_tree_forces / compute_force_on_particle /
// satisfies_opening_criterion / compute_node_particle_interaction (:245-347).
//
// The reference inserts particles one at a time into a pointer tree; the tree
// it ends up with is nevertheless a pure function of (positions, index order,
// leaf_capacity, max_depth, box):  a node reached by more than leaf_capacity
// particles keeps the first leaf_capacity arrivals (they are never
// redistributed) and routes the rest to its 8 children by a strict ">" test
// against a float centre that follows  c + (+-(size*0.5f))*0.5f.  Since
// arrival order is index order at the root and a STABLE split preserves it,
// the whole build is, per level, one stable segmented 8-way partition:
//
//   classify nodes of the level (u64 scan: split rank | stored-particle offset)
//   digit of every live entry + per-tile 8-bin histogram         (HBM pass 1)
//   scan the tile histograms (8 channels)
//   children of every split node from the prefix counts at its first entry
//   scatter entries to their child segment, order preserved      (HBM pass 2)
//
// All counts live on the device; kernels are persistent grid-stride loops over
// device-side extents, so a build is a fixed launch sequence with no host
// synchronisation (max_depth+1 levels; empty levels cost a few microseconds).
// Nodes are numbered breadth-first, children of a node contiguous -- the same
// canonical numbering the CPU oracle exports, which is what makes the
// bit-exact topology test a plain array compare.
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "blockstep.cuh"
#include "scan.cuh"
#include "shard.cuh"
#include "sort.cuh"
#include "tree.cuh"
#include "treepm.cuh"

namespace b200 {

constexpr int MAX_LEVELS = 64;

struct LevelInfo {
    int node_begin, node_end;   // nodes of this level
    int n_entries;              // live entries (particles that reached this level)
    int n_split;                // nodes of this level that split
    int stored_base;            // offset of this level's stored particles in part_idx
    int pad[3];
};

struct TreeGlobals {
    LevelInfo lv[MAX_LEVELS + 2];
    unsigned int totals[8];     // digit totals of the level being processed
    int error;                  // 1 = node table overflow
    int stored_total;
    unsigned long long counters[6];   // walk (counting instance): nodes visited, cell, pair interactions | pair-row
                                      // lane slots issued, node-visit lanes issued, node-visit lanes awake
    int bbox[6];                // fixed mode: order-preserving int codes of min x,y,z / max x,y,z
    float root[4];              // fixed mode: root cube centre and edge
};

struct TreeState {
    size_t n = 0;
    float box = 0.f;
    int cap = 0, max_depth = 0;
    const float4* posm = nullptr;
    size_t max_nodes = 0, max_split = 0, max_tiles = 0, max_node_tiles = 0;
    bool built = false;
    bool counting = false;
    bool fixed = false;          // "fixed physics" tree: no orphans, data-fitted root, real leaf masses
    float eps = 0.01f;           // softening of the walk (0.01f literal in the faithful mode)
    float periodic_box = 0.f;    // fixed mode only: > 0 = minimum-image separations in the walk
    DevBuf center, com, meta, nstart, ncount, nsplit_rank;
    DevBuf ent_idx[2], ent_node[2], digit;
    DevBuf part_idx;
    DevBuf nodes;                 // walk records, 32 B each, depth-first order: {centre of mass, M} {skip, first leaf pair, edge, leaf count}
    DevBuf leaf_pos, lscan, pscan, leaf_tile_sum;   // leaf sources grouped by parent, pair-interleaved (walk-only)
    DevBuf sub;                   // walk records in the subtree of a node (0: leaf or massless)
    DevBuf slot_node;             // node that stores slot q of part_idx
    DevBuf slot_digit;            // arrival-order builds: root octant of every storage slot (level 0 reads this, not posm)
    DevBuf globals;
    DevBuf tile_hist, tile_warp_prefix, node_tile_sum;
    DevBuf split_node, split_where, split_local, split_cstart;
    DevBuf keys, keys_sorted, perm, sort_scratch, order;
    DevBuf active_list, active_tiles;   // block time steps: the active targets of a sync point, in target order
    size_t order_i0 = 0, order_n = 0;
    bool order_valid = false;
    int order_age = 0;            // builds since the target order was computed
    // The build is a fixed sequence of ~200 launches with no host decision in it: captured once into
    // a CUDA graph and replayed while (inputs pointer, sizes, parameters, scratch buffers) stay the same.
    cudaGraphExec_t graph_exec = nullptr;
    size_t graph_key = 0;
    int graph_launches = 0;
    cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    cudaStream_t body_stream = nullptr;   // capture stream for the bodies of the graph's conditional nodes
    // Part build (octant-sharded octree): this tree holds the root, its 8 children and the subtrees of the
    // octants in oct_mask only; the other octants are empty leaves.  The walk tables of all parts make a FOREST.
    int part = 0, n_parts = 1;
    unsigned oct_mask = 0xffu;
    // arrival[k] = storage slot of the k-th particle the reference would insert (nullptr: slot k).  Lets a run
    // STORE its particles in a space-filling order (compact shards, coherent gathers) while the tree stays the
    // one the reference builds from the original index order.  Particle ids everywhere below are storage slots.
    const int* arrival = nullptr;
    size_t forest_key = 0;        // (posm, arrival, n, box, cap, depth, n_parts) of the forest the slots belong to
    struct ForestSlot {
        DevBuf nodes, leaf_pairs;
        DevBuf leaf_slot;             // received: storage slot of every leaf source (2 per pair, -1 = padding)
        const float4* nodes_at = nullptr;      // where this part's records are: `nodes`, or its slice of the all-gather slab
        const int2* slots_at = nullptr;
        size_t nn = 0, npairs = 0;
        bool valid = false;
    } forest[8];
    DevBuf leaf_slot_send;        // this part's leaf sources as storage slots: what the parts exchange (4 B, not 16 B)
    DevBuf nodes_slab, slots_slab;    // collective publish: all parts' records / slots, one equal-sized slice per part
    DevBuf forest_root;           // {global centre of mass, M} {-, -, root edge, -}
    DevBuf forest_hdr;            // device: int2 {nodes, source pairs} per part
    int* forest_hdr_host = nullptr;   // pinned mirror
    size_t fingerprint() const {
        size_t h = 1469598103934665603ull;
        auto mix = [&h](size_t v) { h = (h ^ v) * 1099511628211ull; };
        mix((size_t)posm); mix(n); mix((size_t)cap); mix((size_t)max_depth); mix(fixed ? 1 : 0);
        mix((size_t)oct_mask); mix((size_t)forest_hdr.p); mix((size_t)arrival);
        unsigned bb, eb;
        memcpy(&bb, &box, 4); memcpy(&eb, &eps, 4);
        mix(bb); mix(eb);
        const DevBuf* all[] = {&center, &com, &meta, &nstart, &ncount, &nsplit_rank, &ent_idx[0], &ent_idx[1],
                               &ent_node[0], &ent_node[1], &digit, &part_idx, &nodes, &leaf_pos,
                               &lscan, &pscan, &sub, &leaf_tile_sum, &slot_node, &slot_digit, &globals, &tile_hist,
                               &tile_warp_prefix, &node_tile_sum, &split_node, &split_where, &split_local,
                               &split_cstart};
        for (const DevBuf* b : all) mix((size_t)b->p);
        return h;
    }
    void drop_graph() {
        if (graph_exec) cudaGraphExecDestroy(graph_exec);
        graph_exec = nullptr; graph_key = 0;
    }
    void release() {
        drop_graph();
        if (body_stream) cudaStreamDestroy(body_stream);
        body_stream = nullptr;
        for (ForestSlot& f : forest) { f.nodes.release(); f.leaf_pairs.release(); f.leaf_slot.release(); f.valid = false; }
        forest_root.release(); forest_hdr.release(); leaf_slot_send.release(); nodes_slab.release(); slots_slab.release();
        if (forest_hdr_host) cudaFreeHost(forest_hdr_host);
        forest_hdr_host = nullptr;
        if (ev_in) cudaEventDestroy(ev_in);
        if (ev_out) cudaEventDestroy(ev_out);
        ev_in = ev_out = nullptr;
        DevBuf* all[] = {&center, &com, &meta, &nstart, &ncount, &nsplit_rank, &ent_idx[0],
                         &ent_idx[1], &ent_node[0], &ent_node[1], &digit, &part_idx, &nodes, &leaf_pos, &lscan, &pscan, &sub, &leaf_tile_sum, &slot_node, &slot_digit,
                         &globals, &tile_hist, &tile_warp_prefix, &node_tile_sum, &split_node,
                         &split_where, &split_local, &split_cstart, &keys, &keys_sorted, &perm,
                         &sort_scratch, &order, &active_list, &active_tiles};
        for (DevBuf* b : all) b->release();
    }
};

namespace {

typedef unsigned long long u64;

constexpr int ET_THREADS = 256;
constexpr int ET_ITEMS = 8;
constexpr int ET_WARPS = ET_THREADS / 32;
constexpr int ENT_TILE = ET_THREADS * ET_ITEMS;       // 2048 entries per tile
constexpr int NODE_TILE = 2048;                        // nodes per scan tile (256 x 8)
constexpr unsigned FULL = 0xffffffffu;

// ------------------------------------------------------------------ init ---
// Fixed mode: bounding box of the particles -> root cube (centre = midpoint, edge = largest
// extent * 1.00001f; 1 when all particles coincide), one rounding per operation.
__device__ __forceinline__ int float_code(float f) {        // order-preserving float -> int
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float code_float(int c) { return __int_as_float(c >= 0 ? c : c ^ 0x7fffffff); }

__global__ void bbox_init_kernel(TreeGlobals* g) {
    if (threadIdx.x < 3) { g->bbox[threadIdx.x] = 0x7fffffff; g->bbox[3 + threadIdx.x] = (int)0x80000000; }
}
__global__ void __launch_bounds__(256)
bbox_kernel(const float4* __restrict__ posm, int n, TreeGlobals* g) {
    float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 p = posm[i];
        lo[0] = fminf(lo[0], p.x); hi[0] = fmaxf(hi[0], p.x);
        lo[1] = fminf(lo[1], p.y); hi[1] = fmaxf(hi[1], p.y);
        lo[2] = fminf(lo[2], p.z); hi[2] = fmaxf(hi[2], p.z);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[k] = fminf(lo[k], __shfl_xor_sync(FULL, lo[k], o));
            hi[k] = fmaxf(hi[k], __shfl_xor_sync(FULL, hi[k], o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&g->bbox[k], float_code(lo[k]));
            atomicMax(&g->bbox[3 + k], float_code(hi[k]));
        }
    }
}
__global__ void root_cube_kernel(TreeGlobals* g) {
    float ext = 0.0f;
    for (int k = 0; k < 3; ++k) {
        const float lo = code_float(g->bbox[k]), hi = code_float(g->bbox[3 + k]);
        g->root[k] = __fmul_rn(__fadd_rn(lo, hi), 0.5f);
        ext = fmaxf(ext, __fsub_rn(hi, lo));
    }
    g->root[3] = ext > 0.0f ? __fmul_rn(ext, 1.00001f) : 1.0f;
}

__global__ void tree_init_kernel(TreeGlobals* g, float4* center, float4* com, int4* meta, int* nstart,
                                 int* ncount, int* ent_idx, int* ent_node, int n, float box, int fixed,
                                 const int* __restrict__ arrival) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        for (int l = 0; l < MAX_LEVELS + 2; ++l) {
            g->lv[l].node_begin = g->lv[l].node_end = 0;
            g->lv[l].n_entries = g->lv[l].n_split = g->lv[l].stored_base = 0;
        }
        g->lv[0].node_begin = 0;
        g->lv[0].node_end = 1;
        g->lv[0].n_entries = n;
        g->error = 0;
        g->stored_total = 0;
        for (int c = 0; c < 6; ++c) g->counters[c] = 0;
        center[0] = fixed ? make_float4(g->root[0], g->root[1], g->root[2], g->root[3])
                          : make_float4(0.f, 0.f, 0.f, box);     // tree_force_computer.cpp:132-133
        com[0] = make_float4(0.f, 0.f, 0.f, 0.f);
        meta[0] = make_int4(-1, -1, 0, 0);
        nstart[0] = 0;
        ncount[0] = n;
    }
    for (; i < n; i += gridDim.x * blockDim.x) {
        ent_idx[i] = arrival ? arrival[i] : i;          // arrival order = the reference's insertion order (:136-140)
        ent_node[i] = 0;
    }
}

// The graph of a build runs the levels below `shallow` only when the tree gets there: three IF nodes (build levels,
// centre-of-mass levels, walk-record levels) armed here, after the last unconditional level has been split.
__global__ void arm_deep_levels_kernel(const TreeGlobals* __restrict__ g, int shallow, cudaGraphConditionalHandle h0,
                                       cudaGraphConditionalHandle h1, cudaGraphConditionalHandle h2) {
    const unsigned deep = g->lv[shallow].node_end > g->lv[shallow].node_begin ? 1u : 0u;
    cudaGraphSetConditional(h0, deep);
    cudaGraphSetConditional(h1, deep);
    cudaGraphSetConditional(h2, deep);
}

// ----------------------------------------------------- K1: classify nodes ---
// value per node: (split ? 1 : 0) << 40 | stored particles (leaf members or orphans)
// keep = arrivals a splitting node retains: cap in the reference's tree (orphans), 0 in the fixed tree
__device__ __forceinline__ u64 node_value(int count, int cap, bool may_split, int keep) {
    const bool split = may_split && count > cap;
    return split ? ((1ull << 40) | (u64)keep) : (u64)count;
}

__global__ void __launch_bounds__(256)
node_reduce_kernel(const TreeGlobals* __restrict__ g, int level, int cap, int keep, int max_depth,
                   const int* __restrict__ ncount, u64* __restrict__ tile_sum) {
    __shared__ u64 sh[8];
    const LevelInfo L = g->lv[level];
    const int n_nodes = L.node_end - L.node_begin;
    const int n_tiles = (n_nodes + NODE_TILE - 1) / NODE_TILE;
    const bool may_split = level < max_depth;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        u64 v = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int k = tile * NODE_TILE + threadIdx.x * 8 + j;
            if (k < n_nodes) v += node_value(ncount[L.node_begin + k], cap, may_split, keep);
        }
        const u64 t = block_sum<8>(v, sh);
        if (threadIdx.x == 0) tile_sum[tile] = t;
    }
}

// single CTA: exclusive scan of the tile sums; publishes the extents of the next level
__global__ void __launch_bounds__(1024)
node_scan_kernel(TreeGlobals* __restrict__ g, int level, u64* __restrict__ tile_sum, int max_nodes) {
    const LevelInfo L = g->lv[level];
    const int n_nodes = L.node_end - L.node_begin;
    const u64 tot = cta_exclusive_scan<1>(tile_sum, (n_nodes + NODE_TILE - 1) / NODE_TILE, 1);
    if (threadIdx.x == 0) {
        const int n_split = (int)(tot >> 40);
        const int stored = (int)(tot & ((1ull << 40) - 1));
        g->lv[level].n_split = n_split;
        g->lv[level].stored_base = g->stored_total;
        g->stored_total += stored;
        long long next_end = (long long)L.node_end + 8ll * n_split;
        if (next_end > max_nodes) { g->error = 1; next_end = L.node_end; g->lv[level].n_split = 0; }
        g->lv[level + 1].node_begin = L.node_end;
        g->lv[level + 1].node_end = (int)next_end;
        g->lv[level + 1].n_entries = 0;         // filled by the histogram scan
        for (int d = 0; d < 8; ++d) g->totals[d] = 0;
    }
}

__global__ void __launch_bounds__(256)
node_apply_kernel(const TreeGlobals* __restrict__ g, int level, int cap, int keep, int max_depth,
                  const int* __restrict__ ncount, const u64* __restrict__ tile_sum,
                  int4* __restrict__ meta, int* __restrict__ nsplit_rank, int* __restrict__ split_node) {
    __shared__ u64 wsum[8];
    const LevelInfo L = g->lv[level];
    if (L.n_split == 0 && g->error) return;
    const int n_nodes = L.node_end - L.node_begin;
    const int n_tiles = (n_nodes + NODE_TILE - 1) / NODE_TILE;
    const bool may_split = level < max_depth;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        u64 v[8], tsum = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int k = tile * NODE_TILE + threadIdx.x * 8 + j;
            v[j] = (k < n_nodes) ? node_value(ncount[L.node_begin + k], cap, may_split, keep) : 0ull;
            tsum += v[j];
        }
        u64 pre = block_exclusive_prefix(tile_sum[tile], tsum, wsum);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int k = tile * NODE_TILE + threadIdx.x * 8 + j;
            if (k < n_nodes) {
                const int node = L.node_begin + k;
                const int rank = (int)(pre >> 40);
                const int off = L.stored_base + (int)(pre & ((1ull << 40) - 1));
                const bool split = (v[j] >> 40) != 0;
                int4 m = meta[node];
                m.x = split ? (L.node_end + 8 * rank) : -1;
                m.z = off;
                m.w = (int)(v[j] & ((1ull << 40) - 1));
                meta[node] = m;
                nsplit_rank[node] = split ? rank : -1;
                if (split) split_node[rank] = node;
            }
            pre += v[j];
        }
    }
}

// ------------------------------------------- K2: digits + tile histograms ---
// entry p of (tile, warp, row, lane) = tile*2048 + warp*256 + row*32 + lane
__device__ __forceinline__ int entry_index(int tile, int warp, int row, int lane) {
    return tile * ENT_TILE + warp * (32 * ET_ITEMS) + row * 32 + lane;
}

// Arrival-order builds (particles stored along a space-filling curve, inserted in their original index order): at
// level 0 every entry is a random slot, and gathering its float4 from a 2^24-particle array costs a DRAM sector per
// entry (0.32 ms of a 1.1 ms part build).  One coalesced pass writes the root octant of every SLOT as a byte; the
// 16 MB table stays in L2 and level 0 gathers from there.
__global__ void __launch_bounds__(256)
slot_digit_kernel(const float4* __restrict__ posm, int n, const float4* __restrict__ center,
                  unsigned char* __restrict__ slot_digit) {
    const float4 c = center[0];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 x = posm[i];
        slot_digit[i] = (unsigned char)((x.x > c.x ? 1 : 0) | (x.y > c.y ? 2 : 0) | (x.z > c.z ? 4 : 0));   // :188-194
    }
}

__device__ __forceinline__ unsigned digit_mask(unsigned bv, unsigned b0, unsigned b1, unsigned b2, int d) {
    return bv & ((d & 1) ? b0 : ~b0) & ((d & 2) ? b1 : ~b1) & ((d & 4) ? b2 : ~b2);
}

__global__ void __launch_bounds__(ET_THREADS)
entry_digit_kernel(const TreeGlobals* __restrict__ g, int level, int keep, unsigned oct_mask,
                   const float4* __restrict__ posm, const float4* __restrict__ center,
                   const int4* __restrict__ meta, const int* __restrict__ nstart,
                   const int* __restrict__ nsplit_rank, const int* __restrict__ ent_idx,
                   const int* __restrict__ ent_node, unsigned char* __restrict__ digit,
                   int* __restrict__ part_idx, int* __restrict__ slot_node,
                   unsigned* __restrict__ tile_hist,
                   unsigned* __restrict__ tile_warp_prefix, int* __restrict__ split_where,
                   unsigned* __restrict__ split_local, const unsigned char* __restrict__ slot_digit) {
    __shared__ unsigned wtot[ET_WARPS][8];
    const LevelInfo L = g->lv[level];
    const int n_ent = L.n_entries;
    const int n_tiles = (n_ent + ENT_TILE - 1) / ENT_TILE;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        unsigned run = 0;             // lane l holds the warp's running count of digit (l & 7)
#pragma unroll
        for (int r = 0; r < ET_ITEMS; ++r) {
            const int p = entry_index(tile, warp, r, lane);
            int d = 8, sr = -1;
            bool first_live = false;
            if (p < n_ent) {
                const int idx = ent_idx[p];
                const int k = ent_node[p];
                const int4 m = meta[k];
                const int rel = p - nstart[k];
                if (m.x < 0 || rel < keep) {
                    part_idx[m.z + rel] = idx;          // leaf member, or orphan of a split node
                    slot_node[m.z + rel] = k;
                } else {
                    if (slot_digit != nullptr) {           // level 0 of an arrival-order build
                        d = slot_digit[idx];
                    } else {
                        const float4 c = center[k];
                        const float4 x = posm[idx];
                        d = (x.x > c.x ? 1 : 0) | (x.y > c.y ? 2 : 0) | (x.z > c.z ? 4 : 0);   // :188-194
                    }
                    if (rel == keep) { first_live = true; sr = nsplit_rank[k]; }
                    // part build: a particle bound for an octant another part owns leaves the build here (the
                    // root's child of that octant stays an empty leaf in this part's tree)
                    if (level == 0 && !((oct_mask >> d) & 1u)) d = 8;
                }
                digit[p] = (unsigned char)d;
            }
            const unsigned bv = __ballot_sync(FULL, d < 8);
            const unsigned b0 = __ballot_sync(FULL, d & 1);
            const unsigned b1 = __ballot_sync(FULL, d & 2);
            const unsigned b2 = __ballot_sync(FULL, d & 4);
            if (__any_sync(FULL, first_live)) {
                // prefix counts of all 8 digits at the first live entry of a split node
#pragma unroll
                for (int dd = 0; dd < 8; ++dd) {
                    const unsigned before = __shfl_sync(FULL, run, dd);
                    const unsigned c = before + __popc(digit_mask(bv, b0, b1, b2, dd) & lt);
                    if (first_live) split_local[(size_t)sr * 8 + dd] = c;
                }
                if (first_live) split_where[sr] = tile * ET_WARPS + warp;
            }
            run += __popc(digit_mask(bv, b0, b1, b2, lane & 7));
        }
        __syncthreads();
        if (lane < 8) wtot[warp][lane] = run;
        __syncthreads();
        if (threadIdx.x < 64) {      // thread (w, d): exclusive prefix over warps of digit d
            const int w = threadIdx.x >> 3, d = threadIdx.x & 7;
            unsigned pre = 0;
            for (int ww = 0; ww < w; ++ww) pre += wtot[ww][d];
            tile_warp_prefix[(size_t)tile * 64 + w * 8 + d] = pre;
            if (w == ET_WARPS - 1) tile_hist[(size_t)tile * 8 + d] = pre + wtot[w][d];
        }
    }
}

// 8 CTAs, CTA d scans channel (octant digit) d over the tiles: 1024 threads x 8 tiles per step, so a
// 16 M-particle level (8192 tiles) is one step of thread-serial + warp + CTA scan.  The next level's
// entry count is the sum of the 8 channel totals (reset by node_scan_kernel, added here).
__global__ void __launch_bounds__(1024)
tile_scan_kernel(TreeGlobals* __restrict__ g, int level, unsigned* __restrict__ tile_hist) {
    const int n_tiles = (g->lv[level].n_entries + ENT_TILE - 1) / ENT_TILE;
    const int d = blockIdx.x;
    const unsigned total = cta_exclusive_scan<8>(tile_hist + d, n_tiles, 8);
    if (threadIdx.x == 0) {
        g->totals[d] = total;
        atomicAdd(&g->lv[level + 1].n_entries, (int)total);
    }
}

// ------------------------------------------------------ K4: make children ---
__global__ void __launch_bounds__(256)
make_children_kernel(const TreeGlobals* __restrict__ g, int level, const int* __restrict__ split_node,
                     const int* __restrict__ split_where, const unsigned* __restrict__ split_local,
                     const unsigned* __restrict__ tile_hist /* scanned */,
                     const unsigned* __restrict__ tile_warp_prefix, unsigned* __restrict__ split_cstart,
                     float4* __restrict__ center, float4* __restrict__ com, int4* __restrict__ meta,
                     int* __restrict__ nstart, int* __restrict__ ncount) {
    const LevelInfo L = g->lv[level];
    const int n_split = L.n_split;
    for (int sr = blockIdx.x * blockDim.x + threadIdx.x; sr < n_split; sr += gridDim.x * blockDim.x) {
        unsigned cs[8], cn[8];
        {
            const int w = split_where[sr];
            const int tile = w / ET_WARPS;
#pragma unroll
            for (int d = 0; d < 8; ++d)
                cs[d] = tile_hist[(size_t)tile * 8 + d] + tile_warp_prefix[(size_t)w * 8 + d] +
                        split_local[(size_t)sr * 8 + d];
        }
        if (sr + 1 < n_split) {
            const int w = split_where[sr + 1];
            const int tile = w / ET_WARPS;
#pragma unroll
            for (int d = 0; d < 8; ++d)
                cn[d] = tile_hist[(size_t)tile * 8 + d] + tile_warp_prefix[(size_t)w * 8 + d] +
                        split_local[(size_t)(sr + 1) * 8 + d];
        } else {
#pragma unroll
            for (int d = 0; d < 8; ++d) cn[d] = g->totals[d];
        }
        unsigned base = 0;
#pragma unroll
        for (int d = 0; d < 8; ++d) { split_cstart[(size_t)sr * 8 + d] = cs[d]; base += cs[d]; }
        const int k = split_node[sr];
        const float4 c = center[k];
        const int4 mk = meta[k];
        const int child0 = mk.x;
        const float half_size = __fmul_rn(c.w, 0.5f);                    // :175
        unsigned off = base;
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            const int id = child0 + d;
            const float hx = (d & 1) ? half_size : -half_size;          // :180-182
            const float hy = (d & 2) ? half_size : -half_size;
            const float hz = (d & 4) ? half_size : -half_size;
            center[id] = make_float4(__fadd_rn(c.x, __fmul_rn(hx, 0.5f)), __fadd_rn(c.y, __fmul_rn(hy, 0.5f)),
                                     __fadd_rn(c.z, __fmul_rn(hz, 0.5f)), half_size);
            com[id] = make_float4(0.f, 0.f, 0.f, 0.f);
            const unsigned cnt = cn[d] - cs[d];
            nstart[id] = (int)off;
            ncount[id] = (int)cnt;
            meta[id] = make_int4(-1, (d < 7) ? id + 1 : mk.y, 0, 0);   // .y = skip pointer
            off += cnt;
        }
    }
}

// ---------------------------------------------------------- K5: scatter ---
__global__ void __launch_bounds__(ET_THREADS)
entry_scatter_kernel(const TreeGlobals* __restrict__ g, int level, const int4* __restrict__ meta,
                     const int* __restrict__ nstart, const int* __restrict__ nsplit_rank,
                     const int* __restrict__ ent_idx, const int* __restrict__ ent_node,
                     const unsigned char* __restrict__ digit, const unsigned* __restrict__ tile_hist,
                     const unsigned* __restrict__ tile_warp_prefix,
                     const unsigned* __restrict__ split_cstart, int* __restrict__ out_idx,
                     int* __restrict__ out_node) {
    const LevelInfo L = g->lv[level];
    if (L.n_split == 0) return;
    const int n_ent = L.n_entries;
    const int n_tiles = (n_ent + ENT_TILE - 1) / ENT_TILE;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        // lane l: global prefix of digit (l & 7) at the start of this warp's rows
        unsigned run = tile_hist[(size_t)tile * 8 + (lane & 7)] +
                       tile_warp_prefix[(size_t)tile * 64 + warp * 8 + (lane & 7)];
#pragma unroll
        for (int r = 0; r < ET_ITEMS; ++r) {
            const int p = entry_index(tile, warp, r, lane);
            const int d = (p < n_ent) ? (int)digit[p] : 8;
            const unsigned bv = __ballot_sync(FULL, d < 8);
            const unsigned b0 = __ballot_sync(FULL, d & 1);
            const unsigned b1 = __ballot_sync(FULL, d & 2);
            const unsigned b2 = __ballot_sync(FULL, d & 4);
            const unsigned before = __shfl_sync(FULL, run, d & 7);
            if (d < 8) {
                const unsigned cpos = before + __popc(digit_mask(bv, b0, b1, b2, d) & lt);
                const int k = ent_node[p];
                const int child = meta[k].x + d;
                const int dst = nstart[child] + (int)(cpos - split_cstart[(size_t)nsplit_rank[k] * 8 + d]);
                B200_DEV_ASSERT(dst >= 0 && dst < g->lv[0].n_entries && child > k);
                out_idx[dst] = ent_idx[p];
                out_node[dst] = child;
            }
            run += __popc(digit_mask(bv, b0, b1, b2, lane & 7));
        }
    }
}

// ------------------------------------------------------- centre of mass ---
__device__ __forceinline__ int tree_node_count(const TreeGlobals* g, int max_depth) {
    int nn = 0;
    for (int L = 0; L <= max_depth; ++L)
        if (g->lv[L].node_end > g->lv[L].node_begin) nn = g->lv[L].node_end;
    return nn;
}

// The stored particles that belong to leaf nodes, in the walk's layout: (x, y, z, particle index bits) -- or,
// in the fixed mode, the float4 as it is (x, y, z, mass): that walk uses real masses and needs no self test.
// The leaf particles of one parent are contiguous and PAIR-INTERLEAVED, pair p = {x0 x1 y0 y1} {z0 z1 w0 w1},
// so that one packed-FP32 instruction of the walk handles two sources (lscan: rank of a leaf's first particle
// among all leaf particles; pscan: first pair of a sibling group).
__global__ void stored_pos_kernel(const TreeGlobals* __restrict__ g, const int* __restrict__ part_idx,
                                  const int* __restrict__ slot_node,
                                  const int4* __restrict__ meta, const int* __restrict__ lscan,
                                  const int* __restrict__ pscan, const float4* __restrict__ posm, int n,
                                  float* __restrict__ leaf_pairs, int fixed) {
    int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= n || q >= g->stored_total) return;            // a part build stores only its octants' particles
    const int idx = part_idx[q];
    float4 p = posm[idx];
    if (!fixed) p.w = __int_as_float(idx);
    const int k = slot_node[q];
    const int4 m = meta[k];
    if (m.x >= 0) return;                                       // an orphan: never a source
    int r = lscan[k] + (q - m.z), pair0 = 0;                    // k == 0: the tree is one leaf
    if (k > 0) { const int grp = (k - 1) >> 3; r -= lscan[1 + 8 * grp]; pair0 = pscan[grp]; }
    float* dst = leaf_pairs + (size_t)(pair0 + (r >> 1)) * 8 + (r & 1);
    dst[0] = p.x; dst[2] = p.y; dst[4] = p.z; dst[6] = p.w;
}
// the unused half of a group's last pair when its particle count is odd: a source that adds exactly 0
// (rinv^3 underflows; index -1 / mass 0)
__global__ void __launch_bounds__(256)
pair_pad_kernel(const TreeGlobals* __restrict__ g, int max_depth, const int* __restrict__ lscan,
                const int* __restrict__ pscan, float* __restrict__ leaf_pairs, int fixed) {
    const int nn = tree_node_count(g, max_depth);
    const int groups = (nn - 1) / 8;
    const int items = groups > 0 ? groups : 1;                  // no groups: the root leaf
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < items; j += gridDim.x * blockDim.x) {
        const int cnt = groups > 0 ? lscan[9 + 8 * j] - lscan[1 + 8 * j] : lscan[1];
        if ((cnt & 1) == 0) continue;
        const int pair0 = groups > 0 ? pscan[j] : 0;
        float* dst = leaf_pairs + (size_t)(pair0 + (cnt >> 1)) * 8 + 1;
        dst[0] = 1.0e18f; dst[2] = 1.0e18f; dst[4] = 1.0e18f;
        dst[6] = fixed ? 0.0f : __int_as_float(-1);
    }
}

// compute_center_of_mass (:196-243): one rounding per operation, reference order.
// One thread per node.  Leaves holding more than 64 particles (the max-depth
// overflow leaves that inputs outside the root cube produce can hold 10^5) are
// summed by the whole warp instead: coalesced gathers, then every lane replays the
// SAME sequential sum from shuffled values, so the result keeps the reference's
// summation order bit for bit while the memory latency is paid once per 32 particles.
constexpr int COM_HUGE = 2048;       // leaves above this size (max-depth overflow leaves only) go to com_huge_kernel

__global__ void __launch_bounds__(256)
com_kernel(const TreeGlobals* __restrict__ g, int level, int4* __restrict__ meta,
           const float4* __restrict__ center, const int* __restrict__ part_idx,
           const float4* __restrict__ posm, float4* __restrict__ com, int* __restrict__ sub) {
    const LevelInfo L = g->lv[level];
    const int n_nodes = L.node_end - L.node_begin;
    const int lane = threadIdx.x & 31;
    const int n_round = (n_nodes + 31) & ~31;            // whole warps stay in the loop together
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += gridDim.x * blockDim.x) {
        const bool have = i < n_nodes;
        const int k = L.node_begin + (have ? i : 0);
        const int4 m = have ? meta[k] : make_int4(0, 0, 0, 0);
        const bool huge = have && m.x < 0 && m.w > COM_HUGE;      // summed by a whole CTA afterwards
        const bool big = have && m.x < 0 && m.w > 64 && !huge;
        float total = 0.f, wx = 0.f, wy = 0.f, wz = 0.f;
        int records = 0;             // walk records in this subtree: internal nodes that carry mass (the walk's visits)
        if (have && !big && !huge) {
            if (m.x < 0) {
                B200_DEV_ASSERT(m.z >= 0 && m.w >= 0 && m.z + m.w <= g->stored_total);
                for (int q = m.z; q < m.z + m.w; ++q) {
                    const float4 p = posm[part_idx[q]];
                    total = __fadd_rn(total, p.w);
                    wx = __fadd_rn(wx, __fmul_rn(p.x, p.w));
                    wy = __fadd_rn(wy, __fmul_rn(p.y, p.w));
                    wz = __fadd_rn(wz, __fmul_rn(p.z, p.w));
                }
            } else {
#pragma unroll
                for (int d = 0; d < 8; ++d) {
                    const float4 c = com[m.x + d];
                    if (c.w > 0.f) {
                        total = __fadd_rn(total, c.w);
                        wx = __fadd_rn(wx, __fmul_rn(c.x, c.w));
                        wy = __fadd_rn(wy, __fmul_rn(c.y, c.w));
                        wz = __fadd_rn(wz, __fmul_rn(c.z, c.w));
                    }
                    records += sub[m.x + d];
                }
                records = (total == 0.0f) ? 0 : records + 1;      // :260 -- a massless cell ends the descent
            }
        }
        if (have) sub[k] = records;                              // leaves: 0
        unsigned todo = __ballot_sync(FULL, big);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const int off = __shfl_sync(FULL, m.z, src), np = __shfl_sync(FULL, m.w, src);
            float t = 0.f, sx = 0.f, sy = 0.f, sz = 0.f;
            for (int base = 0; base < np; base += 32) {
                float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
                if (base + lane < np) p = posm[part_idx[off + base + lane]];
                const int cnt = min(32, np - base);
                for (int j = 0; j < cnt; ++j) {
                    const float px = __shfl_sync(FULL, p.x, j), py = __shfl_sync(FULL, p.y, j);
                    const float pz = __shfl_sync(FULL, p.z, j), pw = __shfl_sync(FULL, p.w, j);
                    t = __fadd_rn(t, pw);
                    sx = __fadd_rn(sx, __fmul_rn(px, pw));
                    sy = __fadd_rn(sy, __fmul_rn(py, pw));
                    sz = __fadd_rn(sz, __fmul_rn(pz, pw));
                }
            }
            if (lane == src) { total = t; wx = sx; wy = sy; wz = sz; }
        }
        if (have && m.x >= 0)       // walk-only field: an internal node's cell edge rides in meta.w
            meta[k].w = __float_as_int(center[k].w);
        if (have && !huge) {
            float4 o = make_float4(0.f, 0.f, 0.f, total);
            if (total > 0.f) {
                o.x = __fdiv_rn(wx, total);
                o.y = __fdiv_rn(wy, total);
                o.z = __fdiv_rn(wz, total);
            }
            com[k] = o;
        }
    }
}

// Leaves of the deepest level that hold thousands of particles (inputs outside the root cube pile up in the
// corner cell: the reference generators' [0, box) convention puts N/8 particles into ONE max-depth leaf).  The sum is
// sequential by definition (:203-215, FP32, insertion order), so one thread adds -- but the whole CTA feeds it:
// 1024-particle tiles are gathered and multiplied by all threads into shared memory, double-buffered, while
// thread 0 runs the four dependent add chains of the previous tile (~4 cycles per particle; the per-warp version
// above pays a dependent global gather every 32 particles: 5 ms for a 131 072-particle leaf, this one 0.4 ms).
__global__ void __launch_bounds__(256)
com_huge_kernel(const TreeGlobals* __restrict__ g, int level, const int4* __restrict__ meta,
                const int* __restrict__ part_idx, const float4* __restrict__ posm, float4* __restrict__ com) {
    constexpr int TILE = 1024;
    __shared__ float4 prod[2][TILE];
    __shared__ float4 acc_s;
    const LevelInfo L = g->lv[level];
    const int n_nodes = L.node_end - L.node_begin;
    for (int i = blockIdx.x; i < n_nodes; i += gridDim.x) {
        const int k = L.node_begin + i;
        const int4 m = meta[k];
        if (!(m.x < 0 && m.w > COM_HUGE)) continue;           // CTA-uniform
        const int np = m.w, off = m.z;
        const int n_tiles = (np + TILE - 1) / TILE;
        float4 r[4];
        auto fetch = [&](int tile) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int q = tile * TILE + j * 256 + threadIdx.x;
                float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
                if (q < np) p = posm[part_idx[off + q]];
                r[j] = make_float4(__fmul_rn(p.x, p.w), __fmul_rn(p.y, p.w), __fmul_rn(p.z, p.w), p.w);
            }
        };
        auto stash = [&](int buf) {
#pragma unroll
            for (int j = 0; j < 4; ++j) prod[buf][j * 256 + threadIdx.x] = r[j];
        };
        if (threadIdx.x == 0) acc_s = make_float4(0.f, 0.f, 0.f, 0.f);
        fetch(0);
        stash(0);
        __syncthreads();
        for (int t = 0; t < n_tiles; ++t) {
            if (t + 1 < n_tiles) fetch(t + 1);                 // loads in flight while thread 0 adds
            if (threadIdx.x == 0) {
                float4 a = acc_s;
                const int cnt = min(TILE, np - t * TILE);
                const float4* src = prod[t & 1];
#pragma unroll 8
                for (int j = 0; j < cnt; ++j) {
                    const float4 v = src[j];
                    a.w = __fadd_rn(a.w, v.w);
                    a.x = __fadd_rn(a.x, v.x);
                    a.y = __fadd_rn(a.y, v.y);
                    a.z = __fadd_rn(a.z, v.z);
                }
                acc_s = a;
            }
            if (t + 1 < n_tiles) stash((t + 1) & 1);
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            const float4 a = acc_s;
            float4 o = make_float4(0.f, 0.f, 0.f, a.w);
            if (a.w > 0.f) { o.x = __fdiv_rn(a.x, a.w); o.y = __fdiv_rn(a.y, a.w); o.z = __fdiv_rn(a.z, a.w); }
            com[k] = o;
        }
        __syncthreads();
    }
}

// ------------------------------------------------- walk-only structures ---
// The walk never visits a leaf node.  A target that opens node X interacts with the particles of
// ALL of X's leaf children (:268-270 makes no distance test for leaves), so those particles are
// laid out contiguously per parent (leaf nodes in node-id order = grouped by parent, children in
// order; orphans stored at internal nodes are left out -- they are never sources) and X's record
// carries the range.
// The walk records -- one per internal node that carries mass -- are stored in DEPTH-FIRST (pre-)ORDER, the order
// the walk visits them in: the record after X's is the first record inside X's subtree if there is one, else the
// first one after it, so "descend" is always id + 1 (no link, and the load can be issued before X's record has
// arrived); `skip` = id + records in X's subtree (com_kernel counts them bottom-up, pack_level_kernel hands out the
// ids top-down); "asleep until the walk leaves this subtree" is one compare, id >= wake.
// The two scans of the build tail share one set of kernels:
//   MODE 0, item = node k:           particles stored in k if k is a leaf            -> lscan
//   MODE 1, item = sibling group j   (nodes 1+8j .. 8+8j, the children of one internal node):
//                                    source PAIRS of the group = ceil(leaf particles / 2) -> pscan
template <int MODE>
__device__ __forceinline__ int scan_items(int nn) { return MODE == 1 ? (nn - 1) / 8 : nn; }
template <int MODE>
__device__ __forceinline__ int scan_value(int k, const int4* __restrict__ meta, const int* __restrict__ lscan) {
    if (MODE == 0) { const int4 m = meta[k]; return m.x < 0 ? m.w : 0; }
    return (lscan[9 + 8 * k] - lscan[1 + 8 * k] + 1) >> 1;
}

// exclusive scan over node ids of the leaf particle counts: tile sums, scan of the sums, apply
template <int MODE>
__global__ void __launch_bounds__(256)
leaf_reduce_kernel(const TreeGlobals* __restrict__ g, int max_depth, const int4* __restrict__ meta,
                   const int* __restrict__ lscan, int* __restrict__ tile_sum) {
    __shared__ int sh[8];
    const int nn = scan_items<MODE>(tree_node_count(g, max_depth));
    const int n_tiles = (nn + NODE_TILE - 1) / NODE_TILE;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int v = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = tile * NODE_TILE + j * 256 + threadIdx.x;
            if (k < nn) v += scan_value<MODE>(k, meta, lscan);
        }
        const int t = block_sum<8>(v, sh);
        if (threadIdx.x == 0) tile_sum[tile] = t;
    }
}
template <int MODE>
__global__ void __launch_bounds__(1024)
leaf_scan_kernel(const TreeGlobals* __restrict__ g, int max_depth, int* __restrict__ tile_sum) {
    const int nn = scan_items<MODE>(tree_node_count(g, max_depth));
    cta_exclusive_scan<1>(tile_sum, (nn + NODE_TILE - 1) / NODE_TILE, 1);
}
// out[k] = sum of the values of items < k (k = 0..items); one tile of 2048 items per CTA pass,
// thread t owns items [8t, 8t+8) of the tile so the in-tile scan is a thread-serial + warp + CTA scan
template <int MODE>
__global__ void __launch_bounds__(256)
leaf_apply_kernel(const TreeGlobals* __restrict__ g, int max_depth, const int4* __restrict__ meta,
                  const int* __restrict__ lscan_in, const int* __restrict__ tile_sum, int* __restrict__ lscan) {
    __shared__ int wsum[8];
    const int nn = scan_items<MODE>(tree_node_count(g, max_depth));
    if (nn == 0 && blockIdx.x == 0 && threadIdx.x == 0) lscan[0] = 0;
    const int n_tiles = (nn + NODE_TILE - 1) / NODE_TILE;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int v[8], tsum = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = tile * NODE_TILE + threadIdx.x * 8 + j;
            v[j] = (k < nn) ? scan_value<MODE>(k, meta, lscan_in) : 0;
            tsum += v[j];
        }
        int pre = block_exclusive_prefix(tile_sum[tile], tsum, wsum);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = tile * NODE_TILE + threadIdx.x * 8 + j;
            if (k < nn) lscan[k] = pre;
            pre += v[j];
            if (k == nn - 1) lscan[nn] = pre;
        }
    }
}
// Walk records of one level, top-down: a node that has an id writes its record and hands ids to its children.
// record = {centre of mass, M} {skip | first source pair of the leaf children | cell edge | their particle count}.
// A root that is a leaf: skip = ROOT_LEAF.  Record 0 is always the root's (a part build's root: its own octants).
constexpr int ROOT_LEAF = -2;
constexpr int FOREST_HDR_INTS = 40;     // per part: {records, source pairs, 6 pad} + the 8 level-1 {com, M}
__global__ void __launch_bounds__(256)
pack_level_kernel(const TreeGlobals* __restrict__ g, int level, int max_depth, const float4* __restrict__ com,
                  const int4* __restrict__ meta, const int* __restrict__ lscan, const int* __restrict__ pscan,
                  const int* __restrict__ sub, int* __restrict__ pre, float4* __restrict__ nodes,
                  int* __restrict__ hdr) {
    const LevelInfo L = g->lv[level];
    const int n_nodes = L.node_end - L.node_begin;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_nodes; i += gridDim.x * blockDim.x) {
        const int k = L.node_begin + i;
        const int4 m = meta[k];
        const int records = sub[k];
        if (hdr && k >= 1 && k <= 8) reinterpret_cast<float4*>(hdr + 8)[k - 1] = com[k];   // forest: root merge input
        if (k == 0) {
            const int nn = tree_node_count(g, max_depth);
            if (hdr) {                                              // sizes of this part's walk tables, overflow flag
                hdr[0] = records > 0 ? records : 1;
                hdr[1] = nn > 1 ? pscan[(nn - 1) / 8] : (lscan[1] + 1) / 2;
                hdr[2] = g->error;
            }
            if (m.x < 0) {                                          // the whole tree is one leaf
                nodes[0] = com[0];
                nodes[1] = make_float4(__int_as_float(ROOT_LEAF), __int_as_float(0), 0.0f, __int_as_float(m.w));
                continue;
            }
            pre[0] = 0;
        } else if (records == 0) {
            continue;                                               // leaf, or massless (:260): never visited
        }
        const int id = pre[k];
        B200_DEV_ASSERT(id >= 0 && id + (records > 0 ? records : 1) <= (sub[0] > 0 ? sub[0] : 1));
        int next = id + 1;
#pragma unroll
        for (int d = 0; d < 8; ++d) {
            const int s = sub[m.x + d];
            if (s > 0) { pre[m.x + d] = next; next += s; }
        }
        // a massless root still gets record 0 (M = 0: the walk stops there, :260); skip = 1 = end of its table
        const int skip = records > 0 ? id + records : 1;
        const int loff = pscan[(m.x - 1) >> 3];                     // first source pair of the children
        const int lcnt = lscan[m.x + 8] - lscan[m.x];               // leaf particles among them
        nodes[2 * id] = com[k];
        nodes[2 * id + 1] = make_float4(__int_as_float(skip), __int_as_float(loff), __int_as_float(m.w),
                                        __int_as_float(lcnt));      // m.w of an internal node = cell edge bits
    }
}

// The parts of a forest exchange their leaf sources as STORAGE SLOTS, not as positions: every rank holds all
// positions already (the all-gather that precedes the build), so 4 bytes per source cross NVLink instead of 16, and
// each rank rebuilds the pair rows of the other parts with one gather pass.  A leaf range's particles are spatial
// neighbours and the particles are stored along a Hilbert curve, so that gather is coherent.
// leaf_pairs: pair p = {x0 x1 y0 y1} {z0 z1 w0 w1}; w = slot bits (the faithful tree), -1 = padding.
__global__ void __launch_bounds__(256)
leaf_slots_kernel(const float* __restrict__ leaf_pairs, int n_pairs, int2* __restrict__ slots) {
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n_pairs; p += gridDim.x * blockDim.x) {
        const float2 w = *reinterpret_cast<const float2*>(leaf_pairs + (size_t)p * 8 + 6);
        slots[p] = make_int2(__float_as_int(w.x), __float_as_int(w.y));
    }
}
__global__ void __launch_bounds__(256)
leaf_expand_kernel(const int2* __restrict__ slots, int n_pairs, const float4* __restrict__ posm,
                   float4* __restrict__ leaf_pairs) {
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n_pairs; p += gridDim.x * blockDim.x) {
        const int2 s = slots[p];
        const float far = 1.0e18f;                            // pair_pad_kernel's padding source
        const float4 a = s.x >= 0 ? posm[s.x] : make_float4(far, far, far, 0.f);
        const float4 b = s.y >= 0 ? posm[s.y] : make_float4(far, far, far, 0.f);
        leaf_pairs[2 * (size_t)p] = make_float4(a.x, b.x, a.y, b.y);
        leaf_pairs[2 * (size_t)p + 1] = make_float4(a.z, b.z, __int_as_float(s.x), __int_as_float(s.y));
    }
}

// Global root of a forest: its centre of mass from the 8 level-1 records of the owning parts, in the order and
// rounding of compute_center_of_mass (:226-241, children 0..7 with M > 0) -- the value the unsharded build gives.
struct ForestTables {
    const float4* nodes[8];
    const ulonglong2* leaf_pairs[8];
    int owner[8];                 // part that owns octant d
    int n_parts;
};
__global__ void forest_root_kernel(ForestTables F, const int* __restrict__ hdr, float4* __restrict__ root) {
    float total = 0.f, wx = 0.f, wy = 0.f, wz = 0.f;
    for (int d = 0; d < 8; ++d) {
        const float4 c = reinterpret_cast<const float4*>(hdr + F.owner[d] * FOREST_HDR_INTS + 8)[d];
        if (c.w > 0.f) {
            total = __fadd_rn(total, c.w);
            wx = __fadd_rn(wx, __fmul_rn(c.x, c.w));
            wy = __fadd_rn(wy, __fmul_rn(c.y, c.w));
            wz = __fadd_rn(wz, __fmul_rn(c.z, c.w));
        }
    }
    float4 o = make_float4(0.f, 0.f, 0.f, total);
    if (total > 0.f) { o.x = __fdiv_rn(wx, total); o.y = __fdiv_rn(wy, total); o.z = __fdiv_rn(wz, total); }
    root[0] = o;
    root[1] = F.nodes[0][1];      // every part's root record carries the same cell edge
}

// ------------------------------------------------------------------ walk ---
__device__ __forceinline__ float rsqrt_fast(float x) {   // one MUFU.RSQ, flush-to-zero
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// Warp-cooperative walk: a warp owns 32 targets that are neighbours on a Hilbert curve and walks the
// UNION of their traversals in lockstep (node id is warp-uniform, so node and leaf
// data are broadcast loads and control flow never diverges).  Every lane still
// applies ITS OWN accept test: a lane that accepts a cell adds the monopole and
// sleeps until the walk leaves that cell's subtree -- which is exactly when the
// walk reaches the cell's skip pointer -- so each target receives precisely the
// interactions, in precisely the depth-first order, of the CPU walk.
// size/|d| < theta taken as size^2 < theta^2 d^2 whenever the two sides differ by more than
// 3e-5 relative (the roundings of either form are < 3e-7), else by the exact IEEE sequence.
// The screening test runs on a contracted |d|^2 (3 lane-ops; within 2e-7 of the reference's rounding, far inside
// the 3e-5 margin), and only an undecided case evaluates the reference's own sequence -- one rounding per
// operation, no contraction.
__device__ __forceinline__ bool accept_cell_d(float size, float dx, float dy, float dz, float d2_fast, float theta,
                                              float theta2) {
    const float t = theta2 * d2_fast;
    const float diff = size * size - t;
    if (fabsf(diff) > 3.0e-5f * t) return diff < 0.0f;
    const float d2 = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
    return __fdiv_rn(size, __fsqrt_rn(d2)) < theta;
}

__device__ __forceinline__ float sqrt_fast(float x) {    // one MUFU.SQRT; 0 at 0
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ unsigned long long w_pk(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void w_unpk(unsigned long long v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ unsigned long long w_add2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long w_mul2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long w_fma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// PERIODIC (fixed-physics walk only): separations are taken to the nearest periodic image, d -= box*round(d/box)
// (the minimum image of compute_forces_direct, src/physics/lambda_cdm_kernels.cu:39-41, which is also what
// the reference's GPU tree kernel applies to its cells, src/forces/barnes_hut_tree.cu:247-254) -- for the
// accept test and the monopole with roundf, for the pair rows with the packed magic-number rounding.
// A cell that reaches across the half-box distance from the target (|d| + edge > box/2 on any axis) is
// always opened: its particles need not share the image of its centre of mass.
// POT (fixed-physics walk, no counters): the same walk accumulating the potential phi_i = sum m / sqrt(|d|^2 + eps^2)
// -- monopole M / r for an accepted cell -- instead of the acceleration; one float per target comes out.
// The pair loop has no self test, so the i == i term m_i / eps is subtracted at the end; that is exact as
// long as a target never accepts a cell that contains itself, i.e. theta <= 1/sqrt(3) (checked by the host).
// One 256-bit read-only load (sm_100 LDG.E.ENL2.256): a walk record, or one pair row of leaf sources, is 32
// bytes, 32-byte aligned -- half the L1 requests of two 128-bit loads.
__device__ __forceinline__ void ld256(const float4* p, float4& a, float4& b) {
    asm("ld.global.nc.v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "l"(p));
}
__device__ __forceinline__ void ld256(const ulonglong2* p, ulonglong2& a, ulonglong2& b) {
    asm("ld.global.nc.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(a.x), "=l"(a.y), "=l"(b.x), "=l"(b.y) : "l"(p));
}

// Launch order of the target groups: the last sixteenth of the sorted target range first, then the range from its
// start.  A rank's targets are a fixed set of storage slots; after a few steps some of them sit just across the
// spatial boundary of the rank's region, and sorting by current Hilbert key collects those at the two ends of the
// range -- thin sheets of particles spread over the whole boundary surface, whose 64-target groups are anything
// but compact and take many times longer to walk.  Started last (the hardware hands out CTAs in index order) the
// ones at the end were a tail of a few dozen warps that kept the kernel alive 20-50 % longer (C4 on 4 GPUs: 10.5
// ms per rank for 9.4 ms of work); started first they cost their share of throughput.  Two contiguous runs, so
// CTAs resident together still walk neighbouring groups.
__device__ __forceinline__ unsigned ends_first(unsigned cta, unsigned n_ctas) {
    const unsigned tail = (n_ctas + 15u) >> 4;
    return cta < tail ? n_ctas - tail + cta : cta - tail;
}

// Counting walks: adds the warp's sums of the six counters to the walk's totals in TreeGlobals::counters.
__device__ __forceinline__ void flush_walk_counters(TreeGlobals* g, u64 c_vis, u64 c_pc, u64 c_pp, u64 c_slots,
                                                    u64 c_nl, u64 c_na) {
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        c_vis += __shfl_down_sync(FULL, c_vis, s);
        c_pc += __shfl_down_sync(FULL, c_pc, s);
        c_pp += __shfl_down_sync(FULL, c_pp, s);
        c_slots += __shfl_down_sync(FULL, c_slots, s);
        c_nl += __shfl_down_sync(FULL, c_nl, s);
        c_na += __shfl_down_sync(FULL, c_na, s);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&g->counters[0], c_vis);
        atomicAdd(&g->counters[1], c_pc);
        atomicAdd(&g->counters[2], c_pp);
        atomicAdd(&g->counters[3], c_slots);
        atomicAdd(&g->counters[4], c_nl);
        atomicAdd(&g->counters[5], c_na);
    }
}

// One target per lane: the "fixed physics" walk -- leaf sources carry their real mass in .w and there is no
// self test (with eps > 0 the self pair adds exactly 0; it is counted), softening = eps.  128-thread CTAs, 9
// resident per SM (56 registers).
// by_slot: acc3 is indexed by the target's position in `order` (an explicit target list), not by index - i0.
// The record of the next visit is requested at the end of a visit.  Requesting it as soon as the successor is
// known (after the vote) measured no gain, and speculative requests (the skip target, or id + 1, before the vote)
// cost time -- every broadcast 256-bit load writes 1 KB into the register file, and in this kernel that return path
// (l1tex lsu writeback, 128 B per clock and SM) is 76 % busy, as busy as the issue slots: a wrong guess is not free.
// SHORT (with PERIODIC): the short-range half of TreePM (b200_tree_walk_short_dev).  Every pair and
// accepted cell is weighted by g(r) = erfc(r / 2 r_s) + r / (r_s sqrt(pi)) exp(-r^2 / 4 r_s^2) of its unsoftened
// minimum-image distance (inv2rs = 1 / (2 r_s)); pairs at r >= r_cut weigh 0 (r^2 >= rcut2).  A cell whose centre
// of mass is at least r_cut + sqrt(3) edge away is cut: accepted with weight 0, its subtree skipped -- every
// particle of the cell lies within sqrt(3) edge of its centre of mass, and the torus distance obeys the triangle
// inequality, so no particle of a cut cell is within r_cut of the target, whether or not the cell straddles the
// half-box distance.  The result is added to acc3.  COUNT: the pair interactions (counter 2) are the pairs inside
// r_cut; the pair-row slots (counter 3) still count every leaf pair issued.  The walk fits the 56 registers of 9
// resident CTAs per SM without spilling; its counting instance spills there and gets 8 (64 registers).
// SHORT and POT: the short-range potential (b200_tree_potential_short_dev), same cut-off and cell cut, a pair or an
// accepted cell adding m erfc(r / 2 r_s) / sqrt(r^2 + eps^2).  Pairs at r = 0 add 0: the particle itself is skipped
// rather than added as m / eps and subtracted, which would round the whole sum at the ulp of m / eps.  The result,
// minus the target's own long-range self term m / (sqrt(pi) r_s) that the PM potential holds and minus the
// short-range potential 4 pi r_s^2 M / box^3 of the uniform background (M = the root's mass; the PM potential has
// only its long range), is added to acc3[i - i0]: the PM potential plus this is the Ewald potential.  No counting
// instance.
template <bool COUNT, bool PERIODIC, bool POT, bool SHORT = false>
__global__ void __launch_bounds__(128, SHORT && COUNT ? 8 : 9)
walk_warp_kernel(const float4* __restrict__ posm, const int* __restrict__ order, int i0, int n_targets,
                 const float4* __restrict__ nodes,
                 const ulonglong2* __restrict__ leaf_pairs, float theta, float theta2, float eps2, float box,
                 float* __restrict__ acc3, TreeGlobals* __restrict__ g, int by_slot, float inv2rs, float rcut,
                 float rcut2) {
    static_assert(!SHORT || PERIODIC, "the short-range walk is periodic");
    typedef unsigned long long u64;
    const int t = ends_first(blockIdx.x, gridDim.x) * blockDim.x + threadIdx.x;
    const bool valid = t < n_targets;
    const int i = valid ? (order ? order[t] : (i0 + t)) : -1;
    float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) p = posm[i];
    float ax = 0.f, ay = 0.f, az = 0.f;                                  // cells
    u64 ax2 = 0ull, ay2 = 0ull, az2 = 0ull;                              // leaf pairs, two sources per lane-op
    // theta2 = theta^2 (0 when theta <= 0: nothing is ever accepted) and eps2 = eps^2 come from the host as kernel
    // parameters: constant-bank operands, no registers
    const u64 eps2_2 = w_pk(eps2, eps2);
    const u64 npx = w_pk(-p.x, -p.x), npy = w_pk(-p.y, -p.y), npz = w_pk(-p.z, -p.z);
    [[maybe_unused]] u64 inv_box2, magic2, nmagic2, nbox2;
    if constexpr (PERIODIC) {
        const float ib = 1.0f / box;
        inv_box2 = w_pk(ib, ib);
        magic2 = w_pk(12582912.0f, 12582912.0f);             // 1.5 * 2^23: round to nearest integer
        nmagic2 = w_pk(-12582912.0f, -12582912.0f);
        nbox2 = w_pk(-box, -box);
    }
    unsigned long long c_vis = valid ? 1 : 0, c_pc = 0, c_pp = 0;        // the root is visited by everyone
    [[maybe_unused]] unsigned long long c_slots = 0, c_nl = 0, c_na = 0;  // lane-utilisation counters (COUNT only)
    constexpr int NEVER = 0x7fffffff;
    int wake = valid ? 0 : NEVER;         // record id at which a sleeping lane resumes: ids grow along the walk, so a
                                          // lane is awake iff id >= wake

    // `cnt` leaf particles stored as pairs from pair `q` on, against this lane's target; on_lane = the
    // lane takes part.  Branch-free packed rows: a lane that is out, or is the particle itself, or a
    // padding slot, adds f = 0.
    auto leaf_range = [&](const ulonglong2* __restrict__ pairs, int q, int cnt, bool on_lane) {
        // A lane that is out takes eps^2 = +inf: rsqrt gives exactly 0 and every row adds 0 -- no select per row.
        // The particle itself needs no test either: d = 0 makes its term exactly 0 (eps > 0).  Padding slots are
        // parked far away with mass 0.
        const float e2 = on_lane ? eps2 : __int_as_float(0x7f800000);
        const u64 e2_2 = w_pk(e2, e2);
        auto row2 = [&](const ulonglong2& a, const ulonglong2& b) {      // a = {x0 x1 | y0 y1}, b = {z0 z1 | w0 w1}
            u64 dx = w_add2(a.x, npx), dy = w_add2(a.y, npy), dz = w_add2(b.x, npz);
            if constexpr (PERIODIC) {
                dx = w_fma2(w_add2(w_fma2(dx, inv_box2, magic2), nmagic2), nbox2, dx);
                dy = w_fma2(w_add2(w_fma2(dy, inv_box2, magic2), nmagic2), nbox2, dy);
                dz = w_fma2(w_add2(w_fma2(dz, inv_box2, magic2), nmagic2), nbox2, dz);
            }
            if constexpr (SHORT) {
                // g of the unsoftened distance, 0 at r >= r_cut; an out lane still has rinv = 0 (eps^2 = +inf)
                u64 d2 = w_mul2(dx, dx);
                d2 = w_fma2(dy, dy, d2);
                d2 = w_fma2(dz, dz, d2);
                float d2a, d2b, r2a, r2b;
                w_unpk(d2, d2a, d2b);
                w_unpk(w_add2(d2, e2_2), r2a, r2b);
                if constexpr (POT) {       // erfc of the unsoftened distance over the softened one; r = 0 adds 0
                    const float ea = d2a < rcut2 && d2a > 0.0f ? treepm_short_erfc(sqrt_fast(d2a) * inv2rs) : 0.0f;
                    const float eb = d2b < rcut2 && d2b > 0.0f ? treepm_short_erfc(sqrt_fast(d2b) * inv2rs) : 0.0f;
                    const u64 rinv = w_pk(rsqrt_fast(r2a), rsqrt_fast(r2b));
                    ax2 = w_fma2(rinv, w_mul2(b.y, w_pk(ea, eb)), ax2);
                    return;
                }
                const bool ina = d2a < rcut2, inb = d2b < rcut2;
                const float ga = ina ? treepm_short_g(sqrt_fast(d2a) * inv2rs) : 0.0f;
                const float gb = inb ? treepm_short_g(sqrt_fast(d2b) * inv2rs) : 0.0f;
                const u64 rinv = w_pk(rsqrt_fast(r2a), rsqrt_fast(r2b));
                if (COUNT) { c_slots += 2; if (on_lane) c_pp += (unsigned)ina + (unsigned)inb; }
                const u64 f = w_mul2(w_mul2(w_mul2(rinv, rinv), rinv), w_mul2(b.y, w_pk(ga, gb)));
                ax2 = w_fma2(f, dx, ax2); ay2 = w_fma2(f, dy, ay2); az2 = w_fma2(f, dz, az2);
                return;
            }
            u64 r2 = w_fma2(dx, dx, e2_2);
            r2 = w_fma2(dy, dy, r2);
            r2 = w_fma2(dz, dz, r2);
            float r2a, r2b;
            w_unpk(r2, r2a, r2b);
            const u64 rinv = w_pk(rsqrt_fast(r2a), rsqrt_fast(r2b));
            if constexpr (POT) {
                ax2 = w_fma2(rinv, b.y, ax2);
                return;
            }
            if (COUNT) c_slots += 2;                                     // every lane issues the row: two source slots
            const u64 f = w_mul2(w_mul2(w_mul2(rinv, rinv), rinv), b.y);  // m / r^3
            ax2 = w_fma2(f, dx, ax2); ay2 = w_fma2(f, dy, ay2); az2 = w_fma2(f, dz, az2);
        };
        if (COUNT && !SHORT && on_lane) c_pp += cnt;
        const ulonglong2* src = pairs + 2 * (size_t)q;
        const int np = (cnt + 1) >> 1;
        int k2 = 0;
        for (; k2 + 2 <= np; k2 += 2) {                  // 2 broadcast 256-bit loads in flight, then 2 packed rows
            ulonglong2 a0, b0, a1, b1;
            ld256(src + 2 * k2, a0, b0);
            ld256(src + 2 * k2 + 2, a1, b1);
            row2(a0, b0); row2(a1, b1);
        }
        if (k2 < np) {
            ulonglong2 a0, b0;
            ld256(src + 2 * k2, a0, b0);
            row2(a0, b0);
        }
    };

    // a build that ran out of node slots (possible only in the fixed tree, whose node count has no a-priori
    // bound short of 2.3 N) left an incomplete tree: fail loudly rather than return a plausible force
    if (g->error) {
        if (valid) {
            const float nan = __int_as_float(0x7fc00000);
            if (POT) acc3[i - i0] = nan;
            else { const size_t o = (size_t)(by_slot ? t : i - i0) * 3; acc3[o] = acc3[o + 1] = acc3[o + 2] = nan; }
        }
        return;
    }
    // One table, records [k, kend) in depth-first order; every record is an internal node that carries mass
    // (pack_level_kernel).  The table has one readable record of padding after kend.
    auto walk_table = [&](const float4* __restrict__ nd, const ulonglong2* __restrict__ pairs, int k, const int kend) {
        auto record = [&](int id) {
            return reinterpret_cast<const float4*>(reinterpret_cast<const char*>(nd) + (size_t)(unsigned)id * 32);
        };
        // One visit.  (c, mf) = {centre of mass, M} {skip | first leaf pair | cell edge | leaf-child particles} of
        // record k; the record of the next visit goes into (cn, mn).  The caller alternates two register sets, so
        // no record is ever moved.
        auto visit = [&](const float4& c, const float4& mf, float4& cn, float4& mn) {
            const int skip = __float_as_int(mf.x), lcnt = __float_as_int(mf.w);
            const bool active = k >= wake;
            if (COUNT) { c_nl += 1; c_na += active; }
            // Branch-free: every lane runs the test and the monopole; a lane that sleeps or opens the cell takes
            // 1/r = 0, so its term is exactly 0.
            float dx = __fsub_rn(c.x, p.x), dy = __fsub_rn(c.y, p.y), dz = __fsub_rn(c.z, p.z);
            if constexpr (PERIODIC) {
                dx = __fsub_rn(dx, __fmul_rn(box, roundf(__fdiv_rn(dx, box))));
                dy = __fsub_rn(dy, __fmul_rn(box, roundf(__fdiv_rn(dy, box))));
                dz = __fsub_rn(dz, __fmul_rn(box, roundf(__fdiv_rn(dz, box))));
            }
            // size/|d| < theta (:309) screened as size^2 < theta^2 |d|^2 on a contracted |d|^2: decided unless the two
            // sides are within 3e-5 of each other (the roundings of either form are < 3e-7)
            const float d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
            const float t2 = theta2 * d2;
            const float diff = fmaf(mf.z, mf.z, -t2);
            bool sure = fabsf(diff) > 3.0e-5f * t2;
            bool accept = diff < 0.0f;
            if constexpr (PERIODIC) {    // a cell reaching across the half-box distance is never a monopole
                const float hb = __fmul_rn(box, 0.5f);
                if (__fadd_rn(fabsf(dx), mf.z) > hb || __fadd_rn(fabsf(dy), mf.z) > hb || __fadd_rn(fabsf(dz), mf.z) > hb) {
                    sure = true; accept = false;
                }
            }
            [[maybe_unused]] bool cut = false;
            if constexpr (SHORT) {       // no particle of the cell within r_cut: accepted with weight 0
                const float reach = fmaf(1.7320509f, mf.z, rcut);           // sqrt(3) rounded up
                cut = d2 >= reach * reach;
                if (cut) { sure = true; accept = true; }
            }
            auto monopole = [&](bool take) {                                 // :280-290; 1/r = 0 for a lane that is out
                if constexpr (SHORT) {
                    const float rinv = (take && !cut) ? rsqrt_fast(d2 + eps2) : 0.0f;
                    if constexpr (POT) {
                        ax = fmaf(c.w * treepm_short_erfc(sqrt_fast(d2) * inv2rs), rinv, ax);
                    } else {
                        const float f = c.w * treepm_short_g(sqrt_fast(d2) * inv2rs) * rinv * rinv * rinv;
                        ax = fmaf(f, dx, ax); ay = fmaf(f, dy, ay); az = fmaf(f, dz, az);
                    }
                    if (COUNT) c_pc += take && !cut;
                    if (take) wake = skip;
                    return;
                }
                const float rinv = take ? rsqrt_fast(d2 + eps2) : 0.0f;
                if constexpr (POT) {
                    ax = fmaf(c.w, rinv, ax);
                } else {
                    const float f = c.w * rinv * rinv * rinv;
                    ax = fmaf(f, dx, ax); ay = fmaf(f, dy, ay); az = fmaf(f, dz, az);
                }
                if (COUNT) c_pc += take;
                if (take) wake = skip;                                       // sleep through this subtree
            };
            int nk = skip;
            if (!__any_sync(FULL, active & !(sure & accept))) {
                monopole(active);        // the common visit: every awake lane accepts the cell outright
            } else {
                if (!sure) {             // the reference's own sequence, one rounding per operation
                    const float d2r = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
                    accept = __fdiv_rn(mf.z, __fsqrt_rn(d2r)) < theta;
                }
                const bool open = active && !accept;
                const bool descend = __any_sync(FULL, open);                 // :293-297
                if (descend) nk = k + 1;
                monopole(active && accept);
                if (descend) {
                    if (COUNT && open) c_vis += 8;                           // its 8 children, leaves included
                    if (lcnt > 0) leaf_range(pairs, __float_as_int(mf.y), lcnt, open);
                }
            }
            B200_DEV_ASSERT(nk > k && nk <= kend);
            if (nk < kend) ld256(record(nk), cn, mn);
            k = nk;
        };
        float4 c0, m0, c1, m1;
        if (k < kend) ld256(record(k), c0, m0);
        while (k < kend) {
            visit(c0, m0, c1, m1);
            if (k >= kend) break;
            visit(c1, m1, c0, m0);
        }
    };
    // the root: massless -> nothing to do (:260); a leaf -> one pair loop (:268-270)
    const float4 c = nodes[0];
    const float4 mf = nodes[1];
    if (c.w != 0.0f) {
        if (__float_as_int(mf.x) == ROOT_LEAF) leaf_range(leaf_pairs, 0, __float_as_int(mf.w), valid);
        else walk_table(nodes, leaf_pairs, 0, __float_as_int(mf.x));         // the root's skip = the record count
    }
    if (valid) {
        float lo, hi;
        w_unpk(ax2, lo, hi); ax += lo + hi;
        if constexpr (SHORT && POT) {
            // minus m / (sqrt(pi) r_s) (2 / sqrt(pi) = 1.128...) and the background's 4 pi r_s^2 M / box^3, M = the
            // root's mass
            const float bg = 3.14159265f * c.w / (inv2rs * inv2rs * box * box * box);
            acc3[i - i0] += fmaf(-p.w, 1.128379167f * inv2rs, ax) - bg;
        } else if constexpr (POT) {
            acc3[i - i0] = ax - p.w * rsqrt_fast(eps2);                  // minus the i == i term of the pair loop
        } else {
            w_unpk(ay2, lo, hi); ay += lo + hi;
            w_unpk(az2, lo, hi); az += lo + hi;
            const size_t o = (size_t)(by_slot ? t : i - i0) * 3;
            if constexpr (SHORT) { ax += acc3[o + 0]; ay += acc3[o + 1]; az += acc3[o + 2]; }
            acc3[o + 0] = ax; acc3[o + 1] = ay; acc3[o + 2] = az;
        }
    }
    if (COUNT) flush_walk_counters(g, c_vis, c_pc, c_pp, c_slots, c_nl, c_na);
}

// Two targets per lane: a warp owns 64 Hilbert-adjacent targets -- lane l holds targets l (A) and 32 + l (B) of the
// group -- and walks the union of their 64 traversals.  One record load (1 KB written into the register file, the
// unit the L1 return path counts) and one visit now serve 64 accept tests, and the whole visit runs in packed FP32:
// a lane's A and B separations, |d|^2, screening test and monopole are the two halves of FADD2 / FFMA2 / FMUL2
// operands.  A leaf range is summed for group A and for group B separately, each only if one of its own 32 targets
// opened the cell, so the pair rows serve compact 32-target groups and the row loads are shared.  Decisions,
// interaction sets and counters are those of a walk of one target at a time.
// The reference's faithful tree only (unit-mass leaf pairs, eps = 0.01 literal from the host).
// FOREST: the octree arrives as the walk tables of several part builds (octant-sharded build: each part holds
// the subtrees of its own octants of the root, the other octants are empty leaves there) plus one merged root
// record.  A target tests the root once, then walks part after part -- octant order, i.e. the depth-first order
// of the whole tree -- with the same loop; node ids are local to a part's table.
// MINB: resident CTAs per SM the register budget is cut for, in units of 64 threads (16 -> 64 registers).
// by_slot: as in walk_warp_kernel.
template <bool COUNT, bool FOREST, int MINB, int THREADS>
__global__ void __launch_bounds__(THREADS, MINB * 64 / THREADS)
walk_warp2_kernel(const float4* __restrict__ posm, const int* __restrict__ order, int i0, int n_targets,
                  const float4* __restrict__ nodes, const ulonglong2* __restrict__ leaf_pairs, float theta,
                  float theta2, float eps2, float* __restrict__ acc3, TreeGlobals* __restrict__ g,
                  const ForestTables* __restrict__ forest, const float4* __restrict__ forest_root, int by_slot) {
    typedef unsigned long long u64;
    const int lane = threadIdx.x & 31;
    const int tA = (ends_first(blockIdx.x, gridDim.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 64 + lane, tB = tA + 32;
    const bool vA = tA < n_targets, vB = tB < n_targets;
    const int iA = vA ? (order ? order[tA] : (i0 + tA)) : -1, iB = vB ? (order ? order[tB] : (i0 + tB)) : -1;
    float4 pA = make_float4(0.f, 0.f, 0.f, 0.f), pB = pA;
    if (vA) pA = posm[iA];
    if (vB) pB = posm[iB];
    if (g->error) {                                                      // incomplete tree: fail loudly
        const float nan = __int_as_float(0x7fc00000);
        if (vA) { const size_t o = (size_t)(by_slot ? tA : iA - i0) * 3; acc3[o] = acc3[o + 1] = acc3[o + 2] = nan; }
        if (vB) { const size_t o = (size_t)(by_slot ? tB : iB - i0) * 3; acc3[o] = acc3[o + 1] = acc3[o + 2] = nan; }
        return;
    }
    const u64 npx = w_pk(-pA.x, -pB.x), npy = w_pk(-pA.y, -pB.y), npz = w_pk(-pA.z, -pB.z);   // {A | B}
    u64 cx = 0ull, cy = 0ull, cz = 0ull;                                 // cells {A | B}
    u64 ax2 = 0ull, ay2 = 0ull, az2 = 0ull, bx2 = 0ull, by2 = 0ull, bz2 = 0ull;   // leaf pairs, two sources per lane-op
    unsigned long long c_vis = (vA ? 1 : 0) + (vB ? 1 : 0), c_pc = 0, c_pp = 0;
    [[maybe_unused]] unsigned long long c_slots = 0, c_nl = 0, c_na = 0;
    constexpr int NEVER = 0x7fffffff;
    int wakeA = vA ? 0 : NEVER, wakeB = vB ? 0 : NEVER;

    // one packed row (two sources) against one target; e2 = eps^2, or +inf for a lane that is out
    auto row = [&](const ulonglong2& a, const ulonglong2& b, float px, float py, float pz, float e2, int self,
                   bool on_lane, u64& sx, u64& sy, u64& sz) {
        const u64 dx = w_add2(a.x, w_pk(-px, -px)), dy = w_add2(a.y, w_pk(-py, -py)), dz = w_add2(b.x, w_pk(-pz, -pz));
        u64 r2 = w_fma2(dx, dx, w_pk(e2, e2));
        r2 = w_fma2(dy, dy, r2);
        r2 = w_fma2(dz, dz, r2);
        float r2a, r2b;
        w_unpk(r2, r2a, r2b);
        const u64 rinv = w_pk(rsqrt_fast(r2a), rsqrt_fast(r2b));
        const u64 f = w_mul2(w_mul2(rinv, rinv), rinv);                  // unit mass (:253, :340)
        sx = w_fma2(f, dx, sx); sy = w_fma2(f, dy, sy); sz = w_fma2(f, dz, sz);
        if (COUNT) {
            c_slots += 2;
            float w0, w1;
            w_unpk(b.y, w0, w1);
            c_pp += (on_lane && __float_as_int(w0) != self && __float_as_int(w0) >= 0) +
                    (on_lane && __float_as_int(w1) != self && __float_as_int(w1) >= 0);
        }
    };
    // `cnt` leaf particles from pair `q` on; group A / B takes part iff anyA / anyB (warp-uniform)
    auto leaf_range = [&](const ulonglong2* __restrict__ pairs, int q, int cnt, bool onA, bool onB, bool anyA, bool anyB) {
        const float inf = __int_as_float(0x7f800000);
        const float eA = onA ? eps2 : inf, eB = onB ? eps2 : inf;
        const ulonglong2* src = pairs + 2 * (size_t)q;
        const int np = (cnt + 1) >> 1;
        if (anyA && anyB) {
            for (int r = 0; r < np; ++r) {
                ulonglong2 a, b;
                ld256(src + 2 * r, a, b);
                row(a, b, pA.x, pA.y, pA.z, eA, iA, onA, ax2, ay2, az2);
                row(a, b, pB.x, pB.y, pB.z, eB, iB, onB, bx2, by2, bz2);
            }
        } else if (anyA) {
            int r = 0;
            for (; r + 2 <= np; r += 2) {
                ulonglong2 a0, b0, a1, b1;
                ld256(src + 2 * r, a0, b0);
                ld256(src + 2 * r + 2, a1, b1);
                row(a0, b0, pA.x, pA.y, pA.z, eA, iA, onA, ax2, ay2, az2);
                row(a1, b1, pA.x, pA.y, pA.z, eA, iA, onA, ax2, ay2, az2);
            }
            if (r < np) { ulonglong2 a, b; ld256(src + 2 * r, a, b); row(a, b, pA.x, pA.y, pA.z, eA, iA, onA, ax2, ay2, az2); }
        } else {
            int r = 0;
            for (; r + 2 <= np; r += 2) {
                ulonglong2 a0, b0, a1, b1;
                ld256(src + 2 * r, a0, b0);
                ld256(src + 2 * r + 2, a1, b1);
                row(a0, b0, pB.x, pB.y, pB.z, eB, iB, onB, bx2, by2, bz2);
                row(a1, b1, pB.x, pB.y, pB.z, eB, iB, onB, bx2, by2, bz2);
            }
            if (r < np) { ulonglong2 a, b; ld256(src + 2 * r, a, b); row(a, b, pB.x, pB.y, pB.z, eB, iB, onB, bx2, by2, bz2); }
        }
    };

    const u64 nth2 = w_pk(-theta2, -theta2), eps2_2 = w_pk(eps2, eps2), nband = w_pk(-3.0e-5f, -3.0e-5f);
    auto walk_table = [&](const float4* __restrict__ nd, const ulonglong2* __restrict__ pairs, int k, const int kend) {
        auto record = [&](int id) {
            return reinterpret_cast<const float4*>(reinterpret_cast<const char*>(nd) + (size_t)(unsigned)id * 32);
        };
        auto visit = [&](const float4& c, const float4& mf, float4& cn, float4& mn) {
            const int skip = __float_as_int(mf.x), lcnt = __float_as_int(mf.w);
            const bool actA = k >= wakeA, actB = k >= wakeB;
            if (COUNT) { c_nl += 2; c_na += (actA ? 1 : 0) + (actB ? 1 : 0); }
            // separations of A and B in the two halves; add.rn(c, -p) is fsub_rn(c, p)
            const u64 dx = w_add2(w_pk(c.x, c.x), npx), dy = w_add2(w_pk(c.y, c.y), npy), dz = w_add2(w_pk(c.z, c.z), npz);
            const u64 d2 = w_fma2(dz, dz, w_fma2(dy, dy, w_mul2(dx, dx)));
            // size^2 - theta^2 |d|^2 and the 3e-5 band around 0, as in the one-target kernel: -t2 = (-theta^2) |d|^2
            const u64 nt2 = w_mul2(nth2, d2);
            const u64 diff = w_fma2(w_pk(mf.z, mf.z), w_pk(mf.z, mf.z), nt2);
            const u64 band = w_mul2(nband, nt2);
            float diffA, diffB, bandA, bandB;
            w_unpk(diff, diffA, diffB);
            w_unpk(band, bandA, bandB);
            const bool sureA = fabsf(diffA) > bandA, sureB = fabsf(diffB) > bandB;
            bool accA = diffA < 0.0f, accB = diffB < 0.0f;
            auto monopole = [&](bool takeA, bool takeB) {                    // :280-290; 1/r = 0 for a target that is out
                float r2A, r2B;
                w_unpk(w_add2(d2, eps2_2), r2A, r2B);
                const float riA = takeA ? rsqrt_fast(r2A) : 0.0f, riB = takeB ? rsqrt_fast(r2B) : 0.0f;
                const u64 ri = w_pk(riA, riB);
                const u64 f = w_mul2(w_mul2(w_mul2(w_pk(c.w, c.w), ri), ri), ri);
                cx = w_fma2(f, dx, cx); cy = w_fma2(f, dy, cy); cz = w_fma2(f, dz, cz);
                if (COUNT) c_pc += (takeA ? 1 : 0) + (takeB ? 1 : 0);
                if (takeA) wakeA = skip;                                     // sleep through this subtree
                if (takeB) wakeB = skip;
            };
            int nk = skip;
            // (bitwise on purpose: four independent compares and one combine, not a chain of dependent predicates)
            if (!__any_sync(FULL, (actA & !(sureA & accA)) | (actB & !(sureB & accB)))) {
                monopole(actA, actB);    // the common visit: every awake target accepts the cell outright
            } else {
                auto exact = [&](float ddx, float ddy, float ddz) {          // :302-310, one rounding per operation
                    const float d2r = __fadd_rn(__fadd_rn(__fmul_rn(ddx, ddx), __fmul_rn(ddy, ddy)), __fmul_rn(ddz, ddz));
                    return __fdiv_rn(mf.z, __fsqrt_rn(d2r)) < theta;
                };
                if (!sureA || !sureB) {
                    float dxA, dxB, dyA, dyB, dzA, dzB;
                    w_unpk(dx, dxA, dxB); w_unpk(dy, dyA, dyB); w_unpk(dz, dzA, dzB);
                    if (!sureA) accA = exact(dxA, dyA, dzA);
                    if (!sureB) accB = exact(dxB, dyB, dzB);
                }
                const bool openA = actA && !accA, openB = actB && !accB;
                const bool anyA = __any_sync(FULL, openA), anyB = __any_sync(FULL, openB);
                if (anyA || anyB) nk = k + 1;                                // :293-297
                monopole(actA && accA, actB && accB);
                if (anyA || anyB) {
                    if (COUNT) c_vis += (openA ? 8 : 0) + (openB ? 8 : 0);   // its 8 children, leaves included
                    if (lcnt > 0) leaf_range(pairs, __float_as_int(mf.y), lcnt, openA, openB, anyA, anyB);
                }
            }
            B200_DEV_ASSERT(nk > k && nk <= kend);
            if (nk < kend) ld256(record(nk), cn, mn);
            k = nk;
        };
        float4 c0, m0, c1, m1;
        if (k < kend) ld256(record(k), c0, m0);
        while (k < kend) {
            visit(c0, m0, c1, m1);
            if (k >= kend) break;
            visit(c1, m1, c0, m0);
        }
    };
    if constexpr (!FOREST) {
        const float4* nd = nodes;
        const ulonglong2* pairs = leaf_pairs;
        const float4 c = nd[0];
        const float4 mf = nd[1];
        if (c.w != 0.0f) {                                                   // :260
            if (__float_as_int(mf.x) == ROOT_LEAF) leaf_range(pairs, 0, __float_as_int(mf.w), vA, vB, true, true);
            else walk_table(nd, pairs, 0, __float_as_int(mf.x));
        }
    } else {
        // the merged root: one accept test per target (:257-300 at depth 0), then part after part
        const float4 c = forest_root[0], mf = forest_root[1];
        if (c.w != 0.0f) {
            if (COUNT) { c_nl += 2; c_na += (vA ? 1 : 0) + (vB ? 1 : 0); }
            float fx[2], fy[2], fz[2];
            bool open[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float4& p = h ? pB : pA;
                const bool valid = h ? vB : vA;
                const float dx = __fsub_rn(c.x, p.x), dy = __fsub_rn(c.y, p.y), dz = __fsub_rn(c.z, p.z);
                const float d2 = fmaf(dz, dz, fmaf(dy, dy, dx * dx));
                const bool accept = accept_cell_d(mf.z, dx, dy, dz, d2, theta, theta2);
                const bool take = valid && accept;
                open[h] = valid && !accept;
                const float rinv = take ? rsqrt_fast(d2 + eps2) : 0.0f;
                const float f = c.w * rinv * rinv * rinv;
                fx[h] = f * dx; fy[h] = f * dy; fz[h] = f * dz;
                if (COUNT) c_pc += take;
                if (take) { if (h) wakeB = NEVER; else wakeA = NEVER; }    // the whole tree is one monopole for this target
            }
            cx = w_pk(fx[0], fx[1]); cy = w_pk(fy[0], fy[1]); cz = w_pk(fz[0], fz[1]);
            const bool anyA = __any_sync(FULL, open[0]), anyB = __any_sync(FULL, open[1]);
            if (anyA || anyB) {
                if (COUNT) c_vis += (open[0] ? 8 : 0) + (open[1] ? 8 : 0);
                const int n_parts = forest->n_parts;
                for (int q = 0; q < n_parts; ++q) {
                    const float4* nd = forest->nodes[q];
                    const ulonglong2* pairs = forest->leaf_pairs[q];
                    const float4 r1 = nd[1];                                 // this part's root record: its own octants
                    if (wakeA != NEVER) wakeA = 0;                           // a target sleeping to the end of a part wakes here
                    if (wakeB != NEVER) wakeB = 0;
                    const int lcnt = __float_as_int(r1.w);
                    if (lcnt > 0) leaf_range(pairs, __float_as_int(r1.y), lcnt, open[0], open[1], anyA, anyB);
                    walk_table(nd, pairs, 1, __float_as_int(r1.x));
                }
            }
        }
    }
    float cxA, cxB, cyA, cyB, czA, czB, lo, hi;
    w_unpk(cx, cxA, cxB); w_unpk(cy, cyA, cyB); w_unpk(cz, czA, czB);
    if (vA) {
        const size_t o = (size_t)(by_slot ? tA : iA - i0) * 3;
        w_unpk(ax2, lo, hi); acc3[o + 0] = cxA + (lo + hi);
        w_unpk(ay2, lo, hi); acc3[o + 1] = cyA + (lo + hi);
        w_unpk(az2, lo, hi); acc3[o + 2] = czA + (lo + hi);
    }
    if (vB) {
        const size_t o = (size_t)(by_slot ? tB : iB - i0) * 3;
        w_unpk(bx2, lo, hi); acc3[o + 0] = cxB + (lo + hi);
        w_unpk(by2, lo, hi); acc3[o + 1] = cyB + (lo + hi);
        w_unpk(bz2, lo, hi); acc3[o + 2] = czB + (lo + hi);
    }
    if (COUNT) flush_walk_counters(g, c_vis, c_pc, c_pp, c_slots, c_nl, c_na);
}

// order[] of a target range holds range-local indices after the sort: shift to global
__global__ void add_offset_kernel(int* __restrict__ v, int n, int off) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) v[t] += off;
}
__global__ void zero_counters_kernel(TreeGlobals* g) {
    for (int c = 0; c < 6; ++c) g->counters[c] = 0;
}

// Compaction of the target order to the particles active at sync point k of the block time steps (DESIGN 3.14):
// tiles of ACT_TILE entries, 8 consecutive per thread; count, single-CTA scan of the tile counts (the total lands in
// tile_sum[n_tiles]), then the stable write of the active entries, whose acc_short rows are zeroed on the way.
constexpr int ACT_TILE = 2048;

__global__ void __launch_bounds__(256)
active_count_kernel(const int* __restrict__ order, const unsigned char* __restrict__ bins, int n, int k, int L,
                    unsigned* __restrict__ tile_sum) {
    __shared__ unsigned sh[8];
    const int n_tiles = (n + ACT_TILE - 1) / ACT_TILE;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        unsigned c = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int t = tile * ACT_TILE + threadIdx.x * 8 + j;
            if (t < n) c += block_active(block_bin(bins[order[t]], L), k, L) ? 1u : 0u;
        }
        const unsigned s = block_sum<8>(c, sh);
        if (threadIdx.x == 0) tile_sum[tile] = s;
    }
}

__global__ void __launch_bounds__(1024)
active_scan_kernel(unsigned* __restrict__ tile_sum, int n_tiles) {
    const unsigned tot = cta_exclusive_scan<1>(tile_sum, n_tiles, 1);
    if (threadIdx.x == 0) tile_sum[n_tiles] = tot;
}

__global__ void __launch_bounds__(256)
active_apply_kernel(const int* __restrict__ order, const unsigned char* __restrict__ bins, int n, int k, int L,
                    const unsigned* __restrict__ tile_sum, int* __restrict__ list, float* __restrict__ acc3) {
    __shared__ unsigned sh[8];
    const int n_tiles = (n + ACT_TILE - 1) / ACT_TILE;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        int idx[8];
        unsigned c = 0, on = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int t = tile * ACT_TILE + threadIdx.x * 8 + j;
            idx[j] = t < n ? order[t] : 0;
            if (t < n && block_active(block_bin(bins[idx[j]], L), k, L)) { on |= 1u << j; ++c; }
        }
        unsigned pos = block_exclusive_prefix(tile_sum[tile], c, sh);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (!(on >> j & 1u)) continue;
            list[pos++] = idx[j];
            float* r = acc3 + 3 * (size_t)idx[j];
            r[0] = r[1] = r[2] = 0.f;
        }
    }
}

}  // namespace

// ---------------------------------------------------------------- host side ---
static TreeState* state(b200_ctx* ctx) {
    if (!ctx->tree) ctx->tree = new TreeState();
    return ctx->tree;
}

void tree_destroy(b200_ctx* ctx) {
    if (ctx->tree) {
        ctx->tree->release();
        delete ctx->tree;
        ctx->tree = nullptr;
    }
}

static int tree_enqueue(b200_ctx* ctx, TreeState* T, cudaStream_t st, bool conditional);

static int tree_build_impl(b200_ctx* ctx, const void* posm4, const int* arrival, size_t n, float box, int leaf_cap,
                           int max_depth, bool fixed, float eps, int part, int n_parts, cudaStream_t st);

int tree_build(b200_ctx* ctx, const void* posm4, size_t n, float box, int leaf_cap, int max_depth,
               bool fixed, float eps, cudaStream_t st) {
    return tree_build_impl(ctx, posm4, nullptr, n, box, leaf_cap, max_depth, fixed, eps, 0, 1, st);
}

// Octants [part * 8 / n_parts, (part + 1) * 8 / n_parts) of the root belong to part `part`.
static unsigned part_octants(int part, int n_parts) {
    unsigned m = 0;
    for (int d = part * 8 / n_parts; d < (part + 1) * 8 / n_parts; ++d) m |= 1u << d;
    return m;
}

int tree_build_part(b200_ctx* ctx, const void* posm4, const int* arrival, size_t n, float box, int leaf_cap,
                    int max_depth, int part, int n_parts, cudaStream_t st) {
    if (n_parts < 1 || n_parts > 8 || part < 0 || part >= n_parts) return B200_ERR_INVALID;
    if (n_parts > 1 && n <= (size_t)leaf_cap) return B200_ERR_UNSUPPORTED;      // the root does not split: nothing to shard
    return tree_build_impl(ctx, posm4, arrival, n, box, leaf_cap, max_depth, false, 0.01f, part, n_parts, st);
}

static int tree_build_impl(b200_ctx* ctx, const void* posm4, const int* arrival, size_t n, float box, int leaf_cap,
                           int max_depth, bool fixed, float eps, int part, int n_parts, cudaStream_t st) {
    if (!posm4 || n == 0) return B200_ERR_INVALID;
    if (fixed ? !(eps > 0.f) : !(box > 0.f)) return B200_ERR_INVALID;
    if (leaf_cap < 1 || max_depth < 0 || max_depth > MAX_LEVELS - 2) return B200_ERR_UNSUPPORTED;
    if (n >= (1ull << 30)) return B200_ERR_UNSUPPORTED;
    TreeState* T = state(ctx);
    T->built = false;
    // The warp grouping of the targets is a performance heuristic (any permutation of the range gives the
    // same forces): particles move little per step, so an order is kept for up to 8 builds.
    if (++T->order_age >= 8) T->order_valid = false;
    T->n = n; T->box = box; T->cap = leaf_cap; T->max_depth = max_depth;
    T->fixed = fixed;
    T->eps = fixed ? eps : 0.01f;
    T->posm = (const float4*)posm4;
    T->part = part; T->n_parts = n_parts;
    T->arrival = arrival;
    T->oct_mask = n_parts > 1 ? part_octants(part, n_parts) : 0xffu;
    if (n_parts > 1) {
        B200_TRY(T->forest_hdr.reserve(8 * FOREST_HDR_INTS * sizeof(int)));
        // The slots belong to one forest: same particle array, arrival order, sizes and parameters.  Every rank of
        // a communicator rebuilds its part in the same step, so all slots go stale together; a single process
        // playing all parts (tests) replaces them one at a time -- and must rebuild every part after the
        // particles have moved.
        size_t key = 1469598103934665603ull;
        auto mix = [&key](size_t v) { key = (key ^ v) * 1099511628211ull; };
        unsigned bb;
        memcpy(&bb, &box, 4);
        mix((size_t)posm4); mix((size_t)arrival); mix(n); mix(bb); mix((size_t)leaf_cap); mix((size_t)max_depth);
        mix((size_t)n_parts);
        if (ctx->shard != nullptr || key != T->forest_key) for (auto& f : T->forest) f.valid = false;
        T->forest_key = key;
        T->forest[part].valid = false;
    }
    // reference tree: every internal node keeps exactly leaf_cap particles => at most n/leaf_cap
    // internal nodes.  Fixed tree: internal nodes of one level hold disjoint sets of > leaf_cap
    // particles, typically ~n/(3 leaf_cap) in all; room for n/2 (deep chains under close pairs) --
    // a tree that needs more reports B200_ERR_NOMEM through tree_stats/tree_export.
    T->max_split = fixed ? n / 2 + 64 : n / (size_t)leaf_cap + 1;
    T->max_nodes = 8 * T->max_split + 1;
    T->max_tiles = (n + ENT_TILE - 1) / ENT_TILE + 1;
    T->max_node_tiles = (T->max_nodes + NODE_TILE - 1) / NODE_TILE + 1;
    B200_TRY(T->center.reserve(T->max_nodes * sizeof(float4)));
    B200_TRY(T->com.reserve(T->max_nodes * sizeof(float4)));
    B200_TRY(T->meta.reserve(T->max_nodes * sizeof(int4)));
    B200_TRY(T->nstart.reserve(T->max_nodes * sizeof(int)));
    B200_TRY(T->ncount.reserve(T->max_nodes * sizeof(int)));
    B200_TRY(T->nsplit_rank.reserve(T->max_nodes * sizeof(int)));
    for (int b = 0; b < 2; ++b) {
        B200_TRY(T->ent_idx[b].reserve(n * sizeof(int)));
        B200_TRY(T->ent_node[b].reserve(n * sizeof(int)));
    }
    B200_TRY(T->digit.reserve(n));
    B200_TRY(T->part_idx.reserve(n * sizeof(int)));
    B200_TRY(T->nodes.reserve((T->max_split + 2) * 2 * sizeof(float4)));     // walk records: internal nodes only
    B200_TRY(T->leaf_pos.reserve((n + T->max_split + 2) * sizeof(float4)));     // pair layout: <= 1 pad slot per parent
    B200_TRY(T->pscan.reserve((T->max_split + 2) * sizeof(int)));
    B200_TRY(T->slot_node.reserve(n * sizeof(int)));
    if (arrival != nullptr) B200_TRY(T->slot_digit.reserve(n));
    B200_TRY(T->lscan.reserve((T->max_nodes + 1) * sizeof(int)));
    B200_TRY(T->sub.reserve((T->max_nodes + 1) * sizeof(int)));
    B200_TRY(T->leaf_tile_sum.reserve(T->max_node_tiles * sizeof(int)));
    B200_TRY(T->globals.reserve(sizeof(TreeGlobals)));
    B200_TRY(T->tile_hist.reserve(T->max_tiles * 8 * sizeof(unsigned)));
    B200_TRY(T->tile_warp_prefix.reserve(T->max_tiles * 64 * sizeof(unsigned)));
    B200_TRY(T->node_tile_sum.reserve(T->max_node_tiles * sizeof(u64)));
    B200_TRY(T->split_node.reserve(T->max_split * sizeof(int)));
    B200_TRY(T->split_where.reserve(T->max_split * sizeof(int)));
    B200_TRY(T->split_local.reserve(T->max_split * 8 * sizeof(unsigned)));
    B200_TRY(T->split_cstart.reserve(T->max_split * 8 * sizeof(unsigned)));

    // graph replay, the deep levels behind IF nodes (B200_NO_GRAPH=1: plain launches).  The graph runs on the
    // context's own stream, ordered after / before the caller's stream by events; a caller that is itself
    // capturing gets the unconditional plain launches on its stream instead (they become part of its graph).
    cudaStreamCaptureStatus cap_status = cudaStreamCaptureStatusNone;
    if (st != nullptr && cudaStreamIsCapturing(st, &cap_status) != cudaSuccess) { cudaGetLastError(); cap_status = cudaStreamCaptureStatusNone; }
    if (getenv("B200_NO_GRAPH") == nullptr && cap_status == cudaStreamCaptureStatusNone && ctx->stream != nullptr) {
        const size_t key = T->fingerprint();
        if (T->graph_exec == nullptr || T->graph_key != key) {
            T->drop_graph();
            cudaGraph_t graph = nullptr;
            if (cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
                const uint64_t before = ctx->launches;
                const int rc = tree_enqueue(ctx, T, ctx->stream, true);
                const cudaError_t ce = cudaStreamEndCapture(ctx->stream, &graph);
                T->graph_launches = (int)(ctx->launches - before);
                ctx->launches = before;
                if (rc == B200_OK && ce == cudaSuccess && graph != nullptr &&
                    cudaGraphInstantiate(&T->graph_exec, graph, 0) == cudaSuccess)
                    T->graph_key = key;
                else
                    T->graph_exec = nullptr;
                if (graph) cudaGraphDestroy(graph);
            }
            cudaGetLastError();
        }
        if (T->graph_exec != nullptr) {
            if (!T->ev_in) {
                B200_CUDA(cudaEventCreateWithFlags(&T->ev_in, cudaEventDisableTiming));
                B200_CUDA(cudaEventCreateWithFlags(&T->ev_out, cudaEventDisableTiming));
            }
            if (st != ctx->stream) {
                B200_CUDA(cudaEventRecord(T->ev_in, st));
                B200_CUDA(cudaStreamWaitEvent(ctx->stream, T->ev_in, 0));
            }
            B200_CUDA(cudaGraphLaunch(T->graph_exec, ctx->stream));
            if (st != ctx->stream) {
                B200_CUDA(cudaEventRecord(T->ev_out, ctx->stream));
                B200_CUDA(cudaStreamWaitEvent(st, T->ev_out, 0));
            }
            ctx->launches += (uint64_t)T->graph_launches;
            T->built = true;
            return B200_OK;
        }
    }
    B200_TRY(tree_enqueue(ctx, T, st, false));
    T->built = true;
    return B200_OK;
}

// The launch sequence of one build (kernels only: no allocation, no host synchronisation).
// conditional (only while `st` is being captured into the build's own graph): levels from `shallow` on -- deeper
// than a uniform distribution of n particles reaches -- go into the bodies of three IF nodes (split levels,
// centre-of-mass levels, walk-record levels) that a one-thread kernel arms when level `shallow` exists.  A tree of
// 2^20 uniform particles ends at level 7 of 20: the unconditional sequence spends 0.2 ms in ~110 empty launches.
static int tree_enqueue(b200_ctx* ctx, TreeState* T, cudaStream_t st, bool conditional) {
    const size_t n = T->n;
    const float box = T->box;
    const int leaf_cap = T->cap, max_depth = T->max_depth;
    const bool fixed = T->fixed;
    TreeGlobals* g = T->globals.as<TreeGlobals>();
    float4* center = T->center.as<float4>();
    float4* com = T->com.as<float4>();
    int4* meta = T->meta.as<int4>();
    int* nstart = T->nstart.as<int>();
    int* ncount = T->ncount.as<int>();
    int* nsr = T->nsplit_rank.as<int>();
    const int pgrid = ctx->sm_count * 8;      // persistent grids: 8 x 256-thread CTAs per SM
    const int keep = fixed ? 0 : leaf_cap;
    int* lscan = T->lscan.as<int>();
    int* pscan = T->pscan.as<int>();
    int* tsum = T->leaf_tile_sum.as<int>();

    // a level cannot hold more nodes than this: trims the grids
    auto level_nodes = [&](int L) {
        const double lvl_nodes = (L < 10) ? (double)(1ull << (3 * L)) : 1e30;
        return (size_t)((lvl_nodes < (double)T->max_nodes) ? lvl_nodes : (double)T->max_nodes);
    };
    auto split_levels = [&](int L0, int L1, cudaStream_t s) {               // levels L0..L1: one stable 8-way partition each
        for (int L = L0; L <= L1; ++L) {
            const int cur = L & 1, nxt = cur ^ 1;
            const size_t nb = level_nodes(L);
            const int ngrid = (int)((nb + NODE_TILE - 1) / NODE_TILE < (size_t)pgrid ? (nb + NODE_TILE - 1) / NODE_TILE : (size_t)pgrid);
            const int egrid = (int)(T->max_tiles < (size_t)pgrid ? T->max_tiles : (size_t)pgrid);
            const int sgrid = (int)((nb + 255) / 256 < (size_t)pgrid ? (nb + 255) / 256 : (size_t)pgrid);
            node_reduce_kernel<<<ngrid, 256, 0, s>>>(g, L, leaf_cap, keep, max_depth, ncount, T->node_tile_sum.as<u64>());
            node_scan_kernel<<<1, 1024, 0, s>>>(g, L, T->node_tile_sum.as<u64>(), (int)T->max_nodes);
            node_apply_kernel<<<ngrid, 256, 0, s>>>(g, L, leaf_cap, keep, max_depth, ncount, T->node_tile_sum.as<u64>(),
                                                    meta, nsr, T->split_node.as<int>());
            entry_digit_kernel<<<egrid, ET_THREADS, 0, s>>>(
                g, L, keep, T->oct_mask, T->posm, center, meta, nstart, nsr, T->ent_idx[cur].as<int>(),
                T->ent_node[cur].as<int>(), T->digit.as<unsigned char>(), T->part_idx.as<int>(),
                T->slot_node.as<int>(), T->tile_hist.as<unsigned>(), T->tile_warp_prefix.as<unsigned>(), T->split_where.as<int>(),
                T->split_local.as<unsigned>(),
                (L == 0 && T->arrival != nullptr) ? T->slot_digit.as<unsigned char>() : nullptr);
            tile_scan_kernel<<<8, 1024, 0, s>>>(g, L, T->tile_hist.as<unsigned>());
            make_children_kernel<<<sgrid, 256, 0, s>>>(g, L, T->split_node.as<int>(), T->split_where.as<int>(),
                                                       T->split_local.as<unsigned>(), T->tile_hist.as<unsigned>(),
                                                       T->tile_warp_prefix.as<unsigned>(),
                                                       T->split_cstart.as<unsigned>(), center, com, meta, nstart, ncount);
            entry_scatter_kernel<<<egrid, ET_THREADS, 0, s>>>(
                g, L, meta, nstart, nsr, T->ent_idx[cur].as<int>(), T->ent_node[cur].as<int>(),
                T->digit.as<unsigned char>(), T->tile_hist.as<unsigned>(), T->tile_warp_prefix.as<unsigned>(),
                T->split_cstart.as<unsigned>(), T->ent_idx[nxt].as<int>(), T->ent_node[nxt].as<int>());
        }
        return 7 * (L1 - L0 + 1);
    };
    auto com_levels = [&](int Lhi, int Llo, cudaStream_t s) {                // bottom-up: levels Lhi..Llo
        int launched = 0;
        for (int L = Lhi; L >= Llo; --L) {
            const size_t nb = level_nodes(L);
            const int cgrid = (int)((nb + 255) / 256 < (size_t)pgrid ? (nb + 255) / 256 : (size_t)pgrid);
            com_kernel<<<cgrid, 256, 0, s>>>(g, L, meta, center, T->part_idx.as<int>(), T->posm, com, T->sub.as<int>());
            ++launched;
            if (L == max_depth || leaf_cap > COM_HUGE) {      // only the deepest level can hold leaves above leaf_cap
                com_huge_kernel<<<ctx->sm_count, 256, 0, s>>>(g, L, meta, T->part_idx.as<int>(), T->posm, com);
                ++launched;
            }
        }
        return launched;
    };
    // walk records in depth-first order: ids handed down level by level (nsplit_rank is free after the split levels
    // and holds them)
    auto pack_levels = [&](int L0, int L1, cudaStream_t s) {
        for (int L = L0; L <= L1; ++L) {
            const size_t nb = level_nodes(L);
            const int grid = (int)((nb + 255) / 256 < (size_t)pgrid ? (nb + 255) / 256 : (size_t)pgrid);
            pack_level_kernel<<<grid, 256, 0, s>>>(
                g, L, max_depth, com, meta, lscan, pscan, T->sub.as<int>(), nsr, T->nodes.as<float4>(),
                T->forest_hdr.p ? T->forest_hdr.as<int>() + FOREST_HDR_INTS * T->part : nullptr);
        }
        return L1 - L0 + 1;
    };

    // first level that goes behind the IF nodes: two levels more than n / leaf_cap leaves fill when spread evenly
    int shallow = max_depth + 1;
    cudaGraphConditionalHandle cond[3] = {0, 0, 0};
    cudaGraph_t capture_graph = nullptr;
    if (conditional) {
        int lv = 0;
        for (size_t cells = 1; cells * (size_t)leaf_cap < n && lv < MAX_LEVELS; cells *= 8) ++lv;
        shallow = lv + 3;
        cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
        if (shallow > max_depth ||
            cudaStreamGetCaptureInfo(st, &status, nullptr, &capture_graph, nullptr, nullptr) != cudaSuccess ||
            status != cudaStreamCaptureStatusActive || capture_graph == nullptr) {
            cudaGetLastError();
            shallow = max_depth + 1;
        } else {
            for (int k = 0; k < 3; ++k)
                B200_CUDA(cudaGraphConditionalHandleCreate(&cond[k], capture_graph, 0, cudaGraphCondAssignDefault));
            if (!T->body_stream) B200_CUDA(cudaStreamCreateWithFlags(&T->body_stream, cudaStreamNonBlocking));
        }
    }
    const bool deep = shallow <= max_depth;
    // An IF node after everything captured so far on st; its body = whatever `body` launches on the body stream.
    auto if_deep = [&](cudaGraphConditionalHandle h, auto&& body) -> int {
        cudaStreamCaptureStatus status;
        const cudaGraphNode_t* deps = nullptr;
        size_t n_deps = 0;
        B200_CUDA(cudaStreamGetCaptureInfo(st, &status, nullptr, nullptr, &deps, &n_deps));
        cudaGraphNodeParams p = {};
        p.type = cudaGraphNodeTypeConditional;
        p.conditional.handle = h;
        p.conditional.type = cudaGraphCondTypeIf;
        p.conditional.size = 1;
        cudaGraphNode_t node = nullptr;
        B200_CUDA(cudaGraphAddNode(&node, capture_graph, deps, n_deps, &p));
        B200_CUDA(cudaStreamUpdateCaptureDependencies(st, &node, 1, cudaStreamSetCaptureDependencies));
        cudaGraph_t body_graph = p.conditional.phGraph_out[0];
        B200_CUDA(cudaStreamBeginCaptureToGraph(T->body_stream, body_graph, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
        body(T->body_stream);
        cudaGraph_t same = nullptr;
        B200_CUDA(cudaStreamEndCapture(T->body_stream, &same));
        return B200_OK;
    };

    if (fixed) {
        bbox_init_kernel<<<1, 32, 0, st>>>(g);
        bbox_kernel<<<pgrid, 256, 0, st>>>(T->posm, (int)n, g);
        root_cube_kernel<<<1, 1, 0, st>>>(g);
        ctx->launches += 3;
    }
    tree_init_kernel<<<pgrid, 256, 0, st>>>(g, center, com, meta, nstart, ncount, T->ent_idx[0].as<int>(),
                                            T->ent_node[0].as<int>(), (int)n, box, fixed ? 1 : 0, T->arrival);
    ctx->launches += 1;
    if (T->arrival != nullptr) {
        slot_digit_kernel<<<pgrid, 256, 0, st>>>(T->posm, (int)n, center, T->slot_digit.as<unsigned char>());
        ctx->launches += 1;
    }
    ctx->launches += split_levels(0, deep ? shallow - 1 : max_depth, st);
    B200_CUDA(cudaGetLastError());
    if (deep) {
        // launches inside the bodies are not counted: they run only for trees deeper than `shallow` levels
        arm_deep_levels_kernel<<<1, 1, 0, st>>>(g, shallow, cond[0], cond[1], cond[2]);
        ctx->launches += 1;
        B200_TRY(if_deep(cond[0], [&](cudaStream_t s) { split_levels(shallow, max_depth, s); }));
        B200_TRY(if_deep(cond[1], [&](cudaStream_t s) { com_levels(max_depth, shallow, s); }));
        ctx->launches += com_levels(shallow - 1, 0, st);
    } else {
        ctx->launches += com_levels(max_depth, 0, st);
    }
    // walk-only structures: leaf particles grouped by parent, then the records
    leaf_reduce_kernel<0><<<pgrid, 256, 0, st>>>(g, max_depth, meta, nullptr, tsum);
    leaf_scan_kernel<0><<<1, 1024, 0, st>>>(g, max_depth, tsum);
    leaf_apply_kernel<0><<<pgrid, 256, 0, st>>>(g, max_depth, meta, nullptr, tsum, lscan);
    leaf_reduce_kernel<1><<<pgrid, 256, 0, st>>>(g, max_depth, meta, lscan, tsum);
    leaf_scan_kernel<1><<<1, 1024, 0, st>>>(g, max_depth, tsum);
    leaf_apply_kernel<1><<<pgrid, 256, 0, st>>>(g, max_depth, meta, lscan, tsum, pscan);
    stored_pos_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(
        g, T->part_idx.as<int>(), T->slot_node.as<int>(), meta, lscan, pscan, T->posm, (int)n,
        T->leaf_pos.as<float>(), fixed ? 1 : 0);
    pair_pad_kernel<<<pgrid, 256, 0, st>>>(g, max_depth, lscan, pscan, T->leaf_pos.as<float>(), fixed ? 1 : 0);
    ctx->launches += 8;
    ctx->launches += pack_levels(0, deep ? shallow - 1 : max_depth, st);
    if (deep) B200_TRY(if_deep(cond[2], [&](cudaStream_t s) { pack_levels(shallow, max_depth, s); }));
    B200_CUDA(cudaGetLastError());
    return B200_OK;
}

// Hilbert order of the targets [i0, i0+n): stable sort of their 30-bit keys; kept across builds (order_age).
static int tree_target_order(b200_ctx* ctx, TreeState* T, size_t i0, size_t n_targets, cudaStream_t st) {
    if (T->order_valid && T->order_i0 == i0 && T->order_n == n_targets) return B200_OK;
    B200_TRY(T->keys.reserve(n_targets * sizeof(uint32_t)));
    B200_TRY(T->keys_sorted.reserve(n_targets * sizeof(uint32_t)));
    B200_TRY(T->order.reserve(n_targets * sizeof(int)));
    B200_TRY(T->sort_scratch.reserve(sort_scratch_bytes(n_targets)));
    B200_TRY(hilbert_keys(ctx, T->posm + i0, n_targets, T->box,
                          T->fixed ? T->globals.as<TreeGlobals>()->root : nullptr, T->keys.as<uint32_t>(), st));
    B200_TRY(sort_pairs(ctx, T->keys.as<uint32_t>(), n_targets, T->keys_sorted.as<uint32_t>(),
                        T->order.as<int>(), 30, T->sort_scratch.p, st));
    if (i0) {
        add_offset_kernel<<<(unsigned)((n_targets + 255) / 256), 256, 0, st>>>(T->order.as<int>(),
                                                                               (int)n_targets, (int)i0);
        ctx->launches += 1;
    }
    B200_CUDA(cudaGetLastError());
    T->order_valid = true; T->order_i0 = i0; T->order_n = n_targets; T->order_age = 0;
    return B200_OK;
}

// The fixed-physics walk (one target per lane, 128-thread CTAs) of the targets order[0 .. n_targets), or of
// [i0, i0 + n_targets) when order is null: accelerations, or with POT the potentials.
template <bool COUNT, bool POT>
static void launch_fixed_walk(const TreeState* T, const int* order, size_t i0, size_t n_targets, float theta,
                              float* out, int by_slot, cudaStream_t st) {
    const unsigned grid = (unsigned)((n_targets + 127) / 128);
    const float theta2 = theta > 0.f ? theta * theta : 0.f;
    auto kernel = T->periodic_box > 0.f ? walk_warp_kernel<COUNT, true, POT> : walk_warp_kernel<COUNT, false, POT>;
    kernel<<<grid, 128, 0, st>>>(T->posm, order, (int)i0, (int)n_targets, T->nodes.as<float4>(),
                                 T->leaf_pos.as<ulonglong2>(), theta, theta2, T->eps * T->eps, T->periodic_box, out,
                                 T->globals.as<TreeGlobals>(), by_slot, 0.f, 0.f, 0.f);
}

// The faithful tree's walk (two targets per lane), of this context's tree or (FOREST) of the published forest.
template <bool COUNT, bool FOREST, int MINB, int THREADS>
static void launch_walk2(const TreeState* T, const int* order, size_t i0, size_t n_targets, float theta,
                         float* acc3, int by_slot, cudaStream_t st) {
    const unsigned groups = (unsigned)((n_targets + 63) / 64);           // 64 targets per warp
    const float theta2 = theta > 0.f ? theta * theta : 0.f;
    const float eps2 = 0.01f * 0.01f;                                   // :281-282, :334-335
    const ForestTables* forest = T->forest_root.p ? (const ForestTables*)(T->forest_root.as<char>() + 64) : nullptr;
    walk_warp2_kernel<COUNT, FOREST, MINB, THREADS><<<(groups * 32 + THREADS - 1) / THREADS, THREADS, 0, st>>>(
        T->posm, order, (int)i0, (int)n_targets, T->nodes.as<float4>(), T->leaf_pos.as<ulonglong2>(), theta, theta2,
        eps2, acc3, T->globals.as<TreeGlobals>(), forest, T->forest_root.as<float4>(), by_slot);
}

// Targets: the index range [i0, i0 + n_targets) (list == nullptr; warps are formed from a Hilbert order of the
// range computed here; acc3 indexed by index - i0) or an explicit list of particle indices (warps = runs of 32
// list entries, acc3 in list order).  forest: walk the published forest of part builds, else this context's tree.
static int tree_walk_impl(b200_ctx* ctx, const int* list, size_t i0, size_t n_targets, float theta, void* acc3,
                          cudaStream_t st) {
    TreeState* T = ctx->tree;
    if (!T || !T->built) return B200_ERR_STATE;
    if (n_targets == 0) return B200_OK;
    if (!acc3 || (!list && i0 + n_targets > T->n)) return B200_ERR_INVALID;
    const bool forest = T->n_parts > 1;       // a part build alone is not the whole tree: its walk is the forest's
    if (forest) {
        if (T->fixed) return B200_ERR_STATE;
        for (int q = 0; q < T->n_parts; ++q)
            if (!T->forest[q].valid) return B200_ERR_STATE;               // a part has not been published since its rebuild
    }
    const int* order = list;
    if (!list) {
        B200_TRY(tree_target_order(ctx, T, i0, n_targets, st));
        order = T->order.as<int>();
    }
    const int by_slot = list ? 1 : 0;
    if (T->counting) {
        zero_counters_kernel<<<1, 1, 0, st>>>(T->globals.as<TreeGlobals>());
        ctx->launches += 1;
    }
    if (ctx->timing) B200_CUDA(cudaEventRecord(ctx->ev0, st));
    float* out = (float*)acc3;
    // The faithful tree's instances: 256-thread CTAs, in which adjacent groups share the L1.  The forest instance
    // keeps 8 more values live (part loop): at 64 registers they spill inside the walk loop; 72 registers (7 CTAs of
    // 128 threads) measured 4.5 % faster on 8 GPUs.
    if (forest) {
        if (T->counting) launch_walk2<true, true, 12, 256>(T, order, i0, n_targets, theta, out, by_slot, st);
        else launch_walk2<false, true, 14, 128>(T, order, i0, n_targets, theta, out, by_slot, st);
    } else if (T->fixed) {
        if (T->counting) launch_fixed_walk<true, false>(T, order, i0, n_targets, theta, out, by_slot, st);
        else launch_fixed_walk<false, false>(T, order, i0, n_targets, theta, out, by_slot, st);
    } else {
        if (T->counting) launch_walk2<true, false, 12, 256>(T, order, i0, n_targets, theta, out, by_slot, st);
        else launch_walk2<false, false, 16, 256>(T, order, i0, n_targets, theta, out, by_slot, st);
    }
    if (ctx->timing) B200_CUDA(cudaEventRecord(ctx->ev1, st));
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

int tree_walk(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, void* acc3, cudaStream_t st) {
    return tree_walk_impl(ctx, nullptr, i0, n_targets, theta, acc3, st);
}

int tree_walk_list(b200_ctx* ctx, const int* list, size_t n_list, float theta, void* acc3, cudaStream_t st) {
    if (n_list && !list) return B200_ERR_INVALID;
    return tree_walk_impl(ctx, list, 0, n_list, theta, acc3, st);
}

// The short-range TreePM walk (walk_warp_kernel, SHORT) of the targets [i0, i0 + n_targets) of the fixed-physics
// tree, in the periodic box `box` whatever tree_set_periodic holds: added to acc3.
static int launch_short_walk(b200_ctx* ctx, TreeState* T, const int* order, size_t i0, size_t n_targets, float theta,
                             float box, float r_split, float r_cut, void* acc3, cudaStream_t st);

int tree_walk_short(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, float box, float r_split, float r_cut,
                    void* acc3, cudaStream_t st) {
    TreeState* T = ctx->tree;
    if (!T || !T->built || !T->fixed) return B200_ERR_STATE;
    // r_cut < box / 2: the minimum image is the only image of a source within reach
    if (!(box > 0.f) || !(r_split > 0.f) || !(r_cut > 0.f) || !(r_cut < 0.5f * box)) return B200_ERR_INVALID;
    if (n_targets == 0) return B200_OK;
    if (!acc3 || i0 + n_targets > T->n) return B200_ERR_INVALID;
    B200_TRY(tree_target_order(ctx, T, i0, n_targets, st));
    return launch_short_walk(ctx, T, T->order.as<int>(), i0, n_targets, theta, box, r_split, r_cut, acc3, st);
}

// walk_warp_kernel<SHORT> of the targets order[0 .. n_targets) (particle indices), added to acc3[index - i0]; a
// plain function rather than a template, so that the instances stay where they were in the module
static int launch_short_walk(b200_ctx* ctx, TreeState* T, const int* order, size_t i0, size_t n_targets, float theta,
                             float box, float r_split, float r_cut, void* acc3, cudaStream_t st) {
    if (T->counting) {
        zero_counters_kernel<<<1, 1, 0, st>>>(T->globals.as<TreeGlobals>());
        ctx->launches += 1;
    }
    if (ctx->timing) B200_CUDA(cudaEventRecord(ctx->ev0, st));
    const unsigned grid = (unsigned)((n_targets + 127) / 128);
    const float theta2 = theta > 0.f ? theta * theta : 0.f;
    auto kernel = T->counting ? walk_warp_kernel<true, true, false, true> : walk_warp_kernel<false, true, false, true>;
    kernel<<<grid, 128, 0, st>>>(T->posm, order, (int)i0, (int)n_targets, T->nodes.as<float4>(),
                                 T->leaf_pos.as<ulonglong2>(), theta, theta2, T->eps * T->eps, box, (float*)acc3,
                                 T->globals.as<TreeGlobals>(), 0, 0.5f / r_split, r_cut, r_cut * r_cut);
    if (ctx->timing) B200_CUDA(cudaEventRecord(ctx->ev1, st));
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

// The short-range walk of the particles of [0, n) active at sync point k of the block time steps: the Hilbert order
// of [0, n) compacted to them (its warps stay spatially coherent), their acc_short rows zeroed, then the walk adds
// into them.  The count comes back to the host for the launch size.
int tree_walk_short_active(b200_ctx* ctx, const void* bins_u8, size_t n, int k, int max_bins, float theta, float box,
                           float r_split, float r_cut, void* acc_short3, size_t* n_active, cudaStream_t st) {
    if (!n_active) return B200_ERR_INVALID;
    *n_active = 0;
    TreeState* T = ctx->tree;
    if (!T || !T->built || !T->fixed || T->n != n) return B200_ERR_STATE;
    if (!(box > 0.f) || !(r_split > 0.f) || !(r_cut > 0.f) || !(r_cut < 0.5f * box)) return B200_ERR_INVALID;
    if (max_bins < 1 || max_bins > BLOCK_MAX_BINS) return B200_ERR_INVALID;
    const int L = max_bins - 1;
    if (k < 0 || k > (1 << L) || !bins_u8 || !acc_short3) return B200_ERR_INVALID;
    B200_TRY(tree_target_order(ctx, T, 0, n, st));
    if (k == 0 || k == (1 << L)) {                      // every step ends: the whole Hilbert order, no count to read
        B200_CUDA(cudaMemsetAsync(acc_short3, 0, n * 3 * sizeof(float), st));
        *n_active = n;
        return launch_short_walk(ctx, T, T->order.as<int>(), 0, n, theta, box, r_split, r_cut, acc_short3, st);
    }
    const int n_tiles = (int)((n + ACT_TILE - 1) / ACT_TILE);
    B200_TRY(T->active_list.reserve(n * sizeof(int)));
    B200_TRY(T->active_tiles.reserve((n_tiles + 1) * sizeof(unsigned)));
    const unsigned grid = (unsigned)(n_tiles < ctx->sm_count * 4 ? n_tiles : ctx->sm_count * 4);
    const unsigned char* bins = (const unsigned char*)bins_u8;
    unsigned* tiles = T->active_tiles.as<unsigned>();
    active_count_kernel<<<grid, 256, 0, st>>>(T->order.as<int>(), bins, (int)n, k, L, tiles);
    active_scan_kernel<<<1, 1024, 0, st>>>(tiles, n_tiles);
    active_apply_kernel<<<grid, 256, 0, st>>>(T->order.as<int>(), bins, (int)n, k, L, tiles,
                                              T->active_list.as<int>(), (float*)acc_short3);
    ctx->launches += 3;
    unsigned count = 0;
    B200_CUDA(cudaMemcpyAsync(&count, tiles + n_tiles, sizeof count, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    B200_CUDA(cudaGetLastError());
    *n_active = count;
    if (count == 0) return B200_OK;
    return launch_short_walk(ctx, T, T->active_list.as<int>(), 0, count, theta, box, r_split, r_cut, acc_short3, st);
}

// The short-range TreePM potential (walk_warp_kernel, SHORT and POT) of the same targets, added to phi: the checks
// of tree_walk_short plus the theta bound of tree_potential.
int tree_potential_short(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, float box, float r_split,
                         float r_cut, void* phi, cudaStream_t st) {
    TreeState* T = ctx->tree;
    if (!T || !T->built || !T->fixed) return B200_ERR_STATE;
    if (!(box > 0.f) || !(r_split > 0.f) || !(r_cut > 0.f) || !(r_cut < 0.5f * box)) return B200_ERR_INVALID;
    if (!(theta <= 0.57735f)) return B200_ERR_UNSUPPORTED;  // a target must never accept a cell containing itself
    if (n_targets == 0) return B200_OK;
    if (!phi || i0 + n_targets > T->n) return B200_ERR_INVALID;
    B200_TRY(tree_target_order(ctx, T, i0, n_targets, st));
    walk_warp_kernel<false, true, true, true><<<(unsigned)((n_targets + 127) / 128), 128, 0, st>>>(
        T->posm, T->order.as<int>(), (int)i0, (int)n_targets, T->nodes.as<float4>(), T->leaf_pos.as<ulonglong2>(),
        theta, theta > 0.f ? theta * theta : 0.f, T->eps * T->eps, box, (float*)phi, T->globals.as<TreeGlobals>(), 0,
        0.5f / r_split, r_cut, r_cut * r_cut);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

// ---- forest of part builds -------------------------------------------------------------------
namespace {
__global__ void set_forest_kernel(ForestTables F, ForestTables* dst) { *dst = F; }
}

// Makes this part's walk tables (node records, leaf offsets, leaf source pairs) available to every walker:
// with a communicator of n_parts ranks (b200_shard_init) the parts exchange their tables over NCCL -- sizes first
// (one 160-byte all-gather and a host read-back), then two all-gathers of equal-sized slices -- node records and the
// leaf sources as storage slots, from which every rank rebuilds the pair rows locally; without one (a
// single process building the parts one after another) the tables are copied into this context's slot.
// When all slots are current the merged root record and the table directory are written.
int tree_forest_publish(b200_ctx* ctx, cudaStream_t st) {
    TreeState* T = ctx->tree;
    if (!T || !T->built || T->n_parts < 2 || T->fixed) return B200_ERR_STATE;
    const int P = T->n_parts, part = T->part;
    int rank = 0, world = 1;
    shard_info(ctx, &rank, &world);
    const bool collective = ctx->shard != nullptr && world > 1;
    if (collective && (world != P || rank != part)) return B200_ERR_STATE;
    constexpr size_t HDR_BYTES = FOREST_HDR_INTS * sizeof(int);
    if (!T->forest_hdr_host) B200_CUDA(cudaMallocHost((void**)&T->forest_hdr_host, 8 * HDR_BYTES));
    int* hdr = T->forest_hdr.as<int>();
    if (collective) B200_TRY(shard_allgather_bytes(ctx, hdr + FOREST_HDR_INTS * part, hdr, HDR_BYTES, st));
    B200_CUDA(cudaMemcpyAsync(T->forest_hdr_host, hdr, 8 * HDR_BYTES, cudaMemcpyDeviceToHost, st));
    B200_CUDA(cudaStreamSynchronize(st));
    size_t max_nn = 1, max_pairs = 1;
    for (int q = 0; q < P; ++q) {
        if (!collective && q != part) continue;
        const int* h = T->forest_hdr_host + FOREST_HDR_INTS * q;
        if (h[2]) return B200_ERR_NOMEM;                                  // a part ran out of node slots
        if (h[0] < 1) return B200_ERR_STATE;
        max_nn = (size_t)h[0] > max_nn ? (size_t)h[0] : max_nn;
        max_pairs = (size_t)h[1] > max_pairs ? (size_t)h[1] : max_pairs;
    }
    // this part's leaf sources as slots
    const size_t own_pairs = (size_t)T->forest_hdr_host[FOREST_HDR_INTS * part + 1];
    B200_TRY(T->leaf_slot_send.reserve((max_pairs + 1) * sizeof(int2)));
    const int xgrid = ctx->sm_count * 8;
    leaf_slots_kernel<<<xgrid, 256, 0, st>>>(T->leaf_pos.as<float>(), (int)own_pairs, T->leaf_slot_send.as<int2>());
    ctx->launches += 1;
    if (collective) {
        // two all-gathers of equal-sized slices (the largest part's sizes; what lies behind a part's own size is
        // never read) instead of one broadcast per table and owner: NCCL's best-performing collective, one launch each
        const size_t node_stride = (max_nn + 1) * 2 * sizeof(float4);     // + the record of padding the walk may read
        const size_t slot_stride = max_pairs * sizeof(int2);
        if (node_stride > T->nodes.bytes) return B200_ERR_STATE;           // cannot happen: records <= n / leaf_cap + 1
        B200_TRY(T->nodes_slab.reserve(P * node_stride));
        B200_TRY(T->slots_slab.reserve(P * slot_stride));
        B200_TRY(shard_allgather_bytes(ctx, T->nodes.p, T->nodes_slab.p, node_stride, st));
        B200_TRY(shard_allgather_bytes(ctx, T->leaf_slot_send.p, T->slots_slab.p, slot_stride, st));
        for (int q = 0; q < P; ++q) {
            TreeState::ForestSlot& f = T->forest[q];
            f.nn = (size_t)T->forest_hdr_host[FOREST_HDR_INTS * q];
            f.npairs = (size_t)T->forest_hdr_host[FOREST_HDR_INTS * q + 1];
            f.nodes_at = reinterpret_cast<const float4*>(T->nodes_slab.as<char>() + q * node_stride);
            f.slots_at = reinterpret_cast<const int2*>(T->slots_slab.as<char>() + q * slot_stride);
            B200_TRY(f.leaf_pairs.reserve((f.npairs + 1) * 2 * sizeof(float4)));
            f.valid = true;
        }
    } else {
        TreeState::ForestSlot& f = T->forest[part];
        f.nn = (size_t)T->forest_hdr_host[FOREST_HDR_INTS * part];        // walk records (internal nodes)
        f.npairs = own_pairs;
        B200_TRY(f.nodes.reserve((f.nn + 1) * 2 * sizeof(float4)));       // + the record of padding the walk may read
        B200_TRY(f.leaf_pairs.reserve((f.npairs + 1) * 2 * sizeof(float4)));
        B200_TRY(f.leaf_slot.reserve((f.npairs + 1) * sizeof(int2)));
        B200_CUDA(cudaMemcpyAsync(f.nodes.p, T->nodes.p, f.nn * 2 * sizeof(float4), cudaMemcpyDeviceToDevice, st));
        if (f.npairs)
            B200_CUDA(cudaMemcpyAsync(f.leaf_slot.p, T->leaf_slot_send.p, f.npairs * sizeof(int2), cudaMemcpyDeviceToDevice, st));
        f.nodes_at = f.nodes.as<float4>();
        f.slots_at = f.leaf_slot.as<int2>();
        f.valid = true;
    }
    // pair rows of the received parts from the positions this rank holds (its own part, in a collective publish:
    // a copy of the rows it built)
    for (int q = 0; q < P; ++q) {
        if (!collective && q != part) continue;
        TreeState::ForestSlot& f = T->forest[q];
        if (f.npairs == 0) continue;
        if (collective && q == part) {
            B200_CUDA(cudaMemcpyAsync(f.leaf_pairs.p, T->leaf_pos.p, f.npairs * 2 * sizeof(float4), cudaMemcpyDeviceToDevice, st));
        } else {
            leaf_expand_kernel<<<xgrid, 256, 0, st>>>(f.slots_at, (int)f.npairs, T->posm, f.leaf_pairs.as<float4>());
            ctx->launches += 1;
        }
    }
    B200_CUDA(cudaGetLastError());
    ctx->launches += 0;
    bool all = true;
    for (int q = 0; q < P; ++q) all = all && T->forest[q].valid;
    if (all) {
        ForestTables F;
        memset(&F, 0, sizeof F);
        F.n_parts = P;
        for (int q = 0; q < P; ++q) {
            F.nodes[q] = T->forest[q].nodes_at;
            F.leaf_pairs[q] = T->forest[q].leaf_pairs.as<ulonglong2>();
            for (int d = q * 8 / P; d < (q + 1) * 8 / P; ++d) F.owner[d] = q;
        }
        // forest_root buffer: [0, 32) the merged root record, [64, 64 + sizeof F) the table directory
        B200_TRY(T->forest_root.reserve(64 + sizeof(ForestTables)));
        forest_root_kernel<<<1, 1, 0, st>>>(F, hdr, T->forest_root.as<float4>());
        set_forest_kernel<<<1, 1, 0, st>>>(F, (ForestTables*)(T->forest_root.as<char>() + 64));
        ctx->launches += 2;
        B200_CUDA(cudaGetLastError());
    }
    return B200_OK;
}

// {x, y, z, M} {first, skip, edge, leaf count} of the merged root (host; synchronises)
int tree_forest_root(b200_ctx* ctx, float out[8]) {
    TreeState* T = ctx->tree;
    if (!T || !T->forest_root.p) return B200_ERR_STATE;
    B200_CUDA(cudaDeviceSynchronize());
    B200_CUDA(cudaMemcpy(out, T->forest_root.p, 8 * sizeof(float), cudaMemcpyDeviceToHost));
    return B200_OK;
}

// Potential of the targets [i0, i0 + n) from the fixed-physics tree (phi: float[n_targets], positive).
int tree_potential(b200_ctx* ctx, size_t i0, size_t n_targets, float theta, void* phi, cudaStream_t st) {
    TreeState* T = ctx->tree;
    if (!T || !T->built) return B200_ERR_STATE;
    if (!T->fixed) return B200_ERR_UNSUPPORTED;            // the reference's tree has unit-mass leaves and orphans
    if (!(theta <= 0.57735f)) return B200_ERR_UNSUPPORTED;  // a target must never accept a cell containing itself
    if (n_targets == 0) return B200_OK;
    if (!phi || i0 + n_targets > T->n) return B200_ERR_INVALID;
    B200_TRY(tree_target_order(ctx, T, i0, n_targets, st));
    launch_fixed_walk<false, true>(T, T->order.as<int>(), i0, n_targets, theta, (float*)phi, 0, st);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

const void* tree_posm(b200_ctx* ctx) { return ctx->tree ? (const void*)ctx->tree->posm : nullptr; }

int tree_set_periodic(b200_ctx* ctx, float box) {
    if (box < 0.f) return B200_ERR_INVALID;
    state(ctx)->periodic_box = box;
    return B200_OK;
}

int tree_set_counting(b200_ctx* ctx, int enabled) {
    state(ctx)->counting = enabled != 0;
    return B200_OK;
}

static int fetch_globals(b200_ctx* ctx, TreeState* T, TreeGlobals* h) {
    B200_CUDA(cudaStreamSynchronize(ctx->stream));
    B200_CUDA(cudaDeviceSynchronize());
    B200_CUDA(cudaMemcpy(h, T->globals.p, sizeof(TreeGlobals), cudaMemcpyDeviceToHost));
    return B200_OK;
}

// 1 if the last build overflowed its node table (synchronises)
int tree_overflowed(b200_ctx* ctx, int* flag) {
    TreeState* T = ctx->tree;
    if (!T || !T->built) return B200_ERR_STATE;
    TreeGlobals h;
    B200_TRY(fetch_globals(ctx, T, &h));
    *flag = h.error ? 1 : 0;
    return B200_OK;
}

int tree_counters(b200_ctx* ctx, uint64_t counters[3]) {
    TreeState* T = ctx->tree;
    if (!T || !T->built) return B200_ERR_STATE;
    TreeGlobals h;
    B200_TRY(fetch_globals(ctx, T, &h));
    for (int k = 0; k < 3; ++k) counters[k] = h.counters[k];
    return B200_OK;
}

// all six counters of the last counting walk (see TreeGlobals::counters)
int tree_walk_stats(b200_ctx* ctx, uint64_t stats[6]) {
    TreeState* T = ctx->tree;
    if (!T || !T->built) return B200_ERR_STATE;
    TreeGlobals h;
    B200_TRY(fetch_globals(ctx, T, &h));
    for (int k = 0; k < 6; ++k) stats[k] = h.counters[k];
    return B200_OK;
}

int tree_stats(b200_ctx* ctx, size_t* n_nodes, size_t* n_leaves, size_t* depth, size_t* n_stored) {
    TreeState* T = ctx->tree;
    if (!T || !T->built) return B200_ERR_STATE;
    TreeGlobals h;
    B200_TRY(fetch_globals(ctx, T, &h));
    if (h.error) return B200_ERR_NOMEM;
    size_t nn = 0, dep = 0;
    for (int L = 0; L <= T->max_depth; ++L)
        if (h.lv[L].node_end > h.lv[L].node_begin) { nn = (size_t)h.lv[L].node_end; dep = (size_t)L + 1; }
    if (n_nodes) *n_nodes = nn;
    if (depth) *depth = dep;
    if (n_stored) *n_stored = (size_t)h.stored_total;
    if (n_leaves) {
        std::vector<int4> m(nn);
        B200_CUDA(cudaMemcpy(m.data(), T->meta.p, nn * sizeof(int4), cudaMemcpyDeviceToHost));
        size_t c = 0;
        for (size_t k = 0; k < nn; ++k) c += (m[k].x < 0);
        *n_leaves = c;
    }
    return B200_OK;
}

int tree_export(b200_ctx* ctx, int32_t* level, float* center, float* size, int32_t* first_child,
                int64_t* arrivals, int64_t* part_off, int32_t* part_idx, float* mass, float* com) {
    TreeState* T = ctx->tree;
    if (!T || !T->built) return B200_ERR_STATE;
    TreeGlobals h;
    B200_TRY(fetch_globals(ctx, T, &h));
    if (h.error) return B200_ERR_NOMEM;
    size_t nn = 0;
    for (int L = 0; L <= T->max_depth; ++L)
        if (h.lv[L].node_end > h.lv[L].node_begin) nn = (size_t)h.lv[L].node_end;
    if (level)
        for (int L = 0; L <= T->max_depth; ++L)
            for (int k = h.lv[L].node_begin; k < h.lv[L].node_end; ++k) level[k] = L;
    if (center || size) {
        std::vector<float4> c(nn);
        B200_CUDA(cudaMemcpy(c.data(), T->center.p, nn * sizeof(float4), cudaMemcpyDeviceToHost));
        for (size_t k = 0; k < nn; ++k) {
            if (center) { center[3 * k] = c[k].x; center[3 * k + 1] = c[k].y; center[3 * k + 2] = c[k].z; }
            if (size) size[k] = c[k].w;
        }
    }
    if (first_child || part_off) {
        std::vector<int4> m(nn);
        B200_CUDA(cudaMemcpy(m.data(), T->meta.p, nn * sizeof(int4), cudaMemcpyDeviceToHost));
        for (size_t k = 0; k < nn; ++k) {
            if (first_child) first_child[k] = m[k].x;
            if (part_off) part_off[k] = m[k].z;
        }
        if (part_off) part_off[nn] = h.stored_total;
    }
    if (arrivals) {
        std::vector<int> a(nn);
        B200_CUDA(cudaMemcpy(a.data(), T->ncount.p, nn * sizeof(int), cudaMemcpyDeviceToHost));
        for (size_t k = 0; k < nn; ++k) arrivals[k] = a[k];
    }
    if (part_idx)
        B200_CUDA(cudaMemcpy(part_idx, T->part_idx.p, (size_t)h.stored_total * sizeof(int), cudaMemcpyDeviceToHost));
    if (mass || com) {
        std::vector<float4> c(nn);
        B200_CUDA(cudaMemcpy(c.data(), T->com.p, nn * sizeof(float4), cudaMemcpyDeviceToHost));
        for (size_t k = 0; k < nn; ++k) {
            if (com) { com[3 * k] = c[k].x; com[3 * k + 1] = c[k].y; com[3 * k + 2] = c[k].z; }
            if (mass) mass[k] = c[k].w;
        }
    }
    return B200_OK;
}

}  // namespace b200
