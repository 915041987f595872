// sort.cu -- Morton keys (row T1) and a stable LSD radix sort of (key, index)
// pairs (row T2) for sm_100a.
//
// Replaces compute_morton_codes_kernel + morton3D (reference
// src/forces/barnes_hut_tree.cu:33-55, include/forces/barnes_hut_tree.hpp:11-27)
// and thrust::sequence + thrust::sort_by_key (barnes_hut_tree.cu:358,383-401).
// Hand-written, CUB-style: 8-bit digits, per pass  (1) per-tile digit
// histogram, (2) per-digit exclusive scan over tiles, (3) scatter with a
// warp-match (match.any) stable rank inside the tile.  Integer/byte work that
// is HBM-bound: 20 B per element per pass, coalesced 128-bit loads, tiles of
// 4096 keys so a 16 M sort is 4096 CTAs (~28 per SM).
#include "common.cuh"
#include "scan.cuh"
#include "sort.cuh"

namespace b200 {
namespace {

constexpr int RS_THREADS = 256;
constexpr int RS_ITEMS = 16;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;   // 4096 keys per CTA
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RADIX = 256;

__device__ __forceinline__ uint32_t expand_bits(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

__device__ __forceinline__ uint32_t morton3d(float x, float y, float z) {
    x = fminf(fmaxf(__fmul_rn(x, 1024.0f), 0.0f), 1023.0f);
    y = fminf(fmaxf(__fmul_rn(y, 1024.0f), 0.0f), 1023.0f);
    z = fminf(fmaxf(__fmul_rn(z, 1024.0f), 0.0f), 1023.0f);
    return expand_bits((uint32_t)x) * 4 + expand_bits((uint32_t)y) * 2 + expand_bits((uint32_t)z);
}

__global__ void morton_kernel(const float4* __restrict__ posm, long long n, float box,
                              uint32_t* __restrict__ keys) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 p = posm[i];
    // IEEE divide (the reference builds with --use_fast_math; the host morton3D it
    // must agree with does not) -- barnes_hut_tree.cu:44-51
    float x = __fdiv_rn(p.x, box), y = __fdiv_rn(p.y, box), z = __fdiv_rn(p.z, box);
    x = __fsub_rn(x, floorf(x));
    y = __fsub_rn(y, floorf(y));
    z = __fsub_rn(z, floorf(z));
    keys[i] = morton3d(x, y, z);
}

// Hilbert-curve keys on the same 1024^3 lattice (Skilling's transpose algorithm, then bit
// interleave).  Internal use only: the ORDER in which the walk groups targets into warps.
// A Hilbert curve has no jumps, so 32 consecutive targets form a more compact set than 32
// consecutive Morton keys do, and the union of their traversals is smaller.  The lattice is
// centred so that the origin-centred root cube [-box/2, box/2) maps onto it without wrapping.
// root_dev (nullable): device float[4] = cube centre and edge (the fixed tree's data-fitted root).
__global__ void hilbert_kernel(const float4* __restrict__ posm, long long n, float box,
                               const float* __restrict__ root_dev, uint32_t* __restrict__ keys) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = posm[i];
    float cx = 0.f, cy = 0.f, cz = 0.f;
    if (root_dev) { cx = root_dev[0]; cy = root_dev[1]; cz = root_dev[2]; box = root_dev[3]; }
    const float s = 1024.0f / box;
    uint32_t X[3];
    X[0] = (uint32_t)fminf(fmaxf((p.x - cx) * s + 512.0f, 0.0f), 1023.0f);
    X[1] = (uint32_t)fminf(fmaxf((p.y - cy) * s + 512.0f, 0.0f), 1023.0f);
    X[2] = (uint32_t)fminf(fmaxf((p.z - cz) * s + 512.0f, 0.0f), 1023.0f);
    const uint32_t M = 1u << 9;
    for (uint32_t Q = M; Q > 1; Q >>= 1) {              // inverse undo
        const uint32_t P = Q - 1;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            if (X[d] & Q) X[0] ^= P;
            else { const uint32_t t = (X[0] ^ X[d]) & P; X[0] ^= t; X[d] ^= t; }
        }
    }
    X[1] ^= X[0];                                       // Gray encode
    X[2] ^= X[1];
    uint32_t t = 0;
    for (uint32_t Q = M; Q > 1; Q >>= 1)
        if (X[2] & Q) t ^= Q - 1;
    X[0] ^= t; X[1] ^= t; X[2] ^= t;
    keys[i] = expand_bits(X[0]) * 4 + expand_bits(X[1]) * 2 + expand_bits(X[2]);
}

// warp w of the CTA owns keys [tile*RS_TILE + w*512, +512), 16 rows of 32: the
// (warp, row, lane) order is the key order, which is what makes ranks stable.
__device__ __forceinline__ long long item_index(long long tile, int warp, int row, int lane) {
    return tile * RS_TILE + warp * (32 * RS_ITEMS) + row * 32 + lane;
}

__global__ void __launch_bounds__(RS_THREADS)
rs_hist_kernel(const uint32_t* __restrict__ keys, long long n, int shift, int n_tiles,
               uint32_t* __restrict__ hist /* [RADIX][n_tiles] */) {
    __shared__ uint32_t sh[RADIX];
    const long long tile = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    sh[threadIdx.x] = 0;
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_ITEMS; ++r) {
        long long i = item_index(tile, warp, r, lane);
        if (i < n) atomicAdd(&sh[(keys[i] >> shift) & 0xFFu], 1u);
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * n_tiles + tile] = sh[threadIdx.x];
}

// One CTA per digit: exclusive scan of that digit's per-tile counts (in place)
// and the digit total.
__global__ void __launch_bounds__(1024)
rs_scan_kernel(uint32_t* __restrict__ hist, int n_tiles, uint32_t* __restrict__ totals) {
    const uint32_t total = cta_exclusive_scan<1>(hist + (size_t)blockIdx.x * n_tiles, n_tiles, 1);
    if (threadIdx.x == 0) totals[blockIdx.x] = total;
}

__global__ void __launch_bounds__(RS_THREADS)
rs_scatter_kernel(const uint32_t* __restrict__ keys_in, const int32_t* __restrict__ vals_in,
                  uint32_t* __restrict__ keys_out, int32_t* __restrict__ vals_out, long long n,
                  int shift, int n_tiles, const uint32_t* __restrict__ hist,
                  const uint32_t* __restrict__ totals) {
    __shared__ uint32_t warp_cnt[RS_WARPS][RADIX];   // per-warp digit counters -> bases
    __shared__ uint32_t digit_base[RADIX];
    __shared__ uint32_t wsum[RS_WARPS];
    const long long tile = blockIdx.x;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;

    for (int k = threadIdx.x; k < RS_WARPS * RADIX; k += RS_THREADS) (&warp_cnt[0][0])[k] = 0;
    // global base of each digit = exclusive scan of totals (256 values, one per thread)
    digit_base[threadIdx.x] =
        block_exclusive_prefix(hist[(size_t)threadIdx.x * n_tiles + tile], totals[threadIdx.x], wsum);
    __syncthreads();

    uint32_t key[RS_ITEMS];
    int32_t val[RS_ITEMS];
    uint32_t rank[RS_ITEMS];
#pragma unroll
    for (int r = 0; r < RS_ITEMS; ++r) {
        long long i = item_index(tile, warp, r, lane);
        const bool ok = i < n;
        key[r] = ok ? keys_in[i] : 0xFFFFFFFFu;
        val[r] = ok ? (vals_in ? vals_in[i] : (int32_t)i) : -1;
        const uint32_t d = (key[r] >> shift) & 0xFFu;
        // invalid slots only exist at the very end of the last tile; giving them a
        // rank keeps the warp converged, they are not written.
        const uint32_t peers = __match_any_sync(0xffffffffu, ok ? d : 0x100u);
        const uint32_t before = warp_cnt[warp][ok ? d : 0];
        rank[r] = before + __popc(peers & lt);
        __syncwarp();
        if (ok && (peers & lt) == 0) warp_cnt[warp][d] = before + __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    // per digit: exclusive prefix over warps (key order = warp order)
    {
        const int d = threadIdx.x;
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < RS_WARPS; ++w) {
            uint32_t c = warp_cnt[w][d];
            warp_cnt[w][d] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_ITEMS; ++r) {
        long long i = item_index(tile, warp, r, lane);
        if (i < n) {
            const uint32_t d = (key[r] >> shift) & 0xFFu;
            const uint32_t dst = digit_base[d] + warp_cnt[warp][d] + rank[r];
            keys_out[dst] = key[r];
            vals_out[dst] = val[r];
        }
    }
}

}  // namespace

int morton_keys(b200_ctx* ctx, const void* posm4, size_t n, float box, uint32_t* keys,
                cudaStream_t st) {
    if (n == 0) return B200_OK;
    if (!(box > 0.f)) return B200_ERR_INVALID;
    morton_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const float4*)posm4, (long long)n,
                                                               box, keys);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

int hilbert_keys(b200_ctx* ctx, const void* posm4, size_t n, float box, const float* root_dev,
                 uint32_t* keys, cudaStream_t st) {
    if (n == 0) return B200_OK;
    if (!root_dev && !(box > 0.f)) return B200_ERR_INVALID;
    hilbert_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const float4*)posm4, (long long)n,
                                                               box, root_dev, keys);
    B200_CUDA(cudaGetLastError());
    ctx->launches += 1;
    return B200_OK;
}

size_t sort_scratch_bytes(size_t n) {
    size_t n_tiles = (n + RS_TILE - 1) / RS_TILE;
    // two ping-pong (key, val) buffers + histogram + totals
    return 2 * n * sizeof(uint32_t) + 2 * n * sizeof(int32_t) + RADIX * n_tiles * sizeof(uint32_t) +
           RADIX * sizeof(uint32_t) + 1024;
}

// Stable ascending sort of (keys_in[i], i) on bits [0, end_bit).  scratch must
// hold sort_scratch_bytes(n).  Results land in keys_out / perm_out.
int sort_pairs(b200_ctx* ctx, const uint32_t* keys_in, size_t n, uint32_t* keys_out,
               int32_t* perm_out, int end_bit, void* scratch, cudaStream_t st) {
    if (n == 0) return B200_OK;
    if (n >= (1ull << 31)) return B200_ERR_UNSUPPORTED;
    const int n_tiles = (int)((n + RS_TILE - 1) / RS_TILE);
    unsigned char* s = (unsigned char*)scratch;
    uint32_t* kA = (uint32_t*)s; s += n * sizeof(uint32_t);
    uint32_t* kB = (uint32_t*)s; s += n * sizeof(uint32_t);
    int32_t* vA = (int32_t*)s; s += n * sizeof(int32_t);
    int32_t* vB = (int32_t*)s; s += n * sizeof(int32_t);
    uint32_t* hist = (uint32_t*)s; s += (size_t)RADIX * n_tiles * sizeof(uint32_t);
    uint32_t* totals = (uint32_t*)s;
    const int passes = (end_bit + 7) / 8;
    const uint32_t* kin = keys_in;
    const int32_t* vin = nullptr;           // pass 0 generates the identity (thrust::sequence)
    for (int p = 0; p < passes; ++p) {
        const bool last = (p == passes - 1);
        uint32_t* kout = last ? keys_out : ((p & 1) ? kB : kA);
        int32_t* vout = last ? perm_out : ((p & 1) ? vB : vA);
        rs_hist_kernel<<<n_tiles, RS_THREADS, 0, st>>>(kin, (long long)n, p * 8, n_tiles, hist);
        rs_scan_kernel<<<RADIX, 1024, 0, st>>>(hist, n_tiles, totals);
        rs_scatter_kernel<<<n_tiles, RS_THREADS, 0, st>>>(kin, vin, kout, vout, (long long)n, p * 8,
                                                          n_tiles, hist, totals);
        B200_CUDA(cudaGetLastError());
        ctx->launches += 3;
        kin = kout;
        vin = vout;
    }
    return B200_OK;
}

}  // namespace b200
