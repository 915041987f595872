// scan.cuh -- CTA-wide integer sums and prefix sums shared by the tree build (tree.cu) and the radix
// sort (sort.cu).  Every value is an integer, so the results do not depend on the order of the adds.
#pragma once

namespace b200 {

// inclusive prefix sum over the 32 lanes of a full warp
template <typename T>
__device__ __forceinline__ T warp_inclusive_scan(T x) {
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

// sum of v over a CTA of WARPS warps, returned to every thread; sh holds WARPS values
template <int WARPS, typename T>
__device__ __forceinline__ T block_sum(T v, T* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    T t = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) t += sh[w];
    return t;
}

// base + the sum of `sum` over the threads of the CTA before this one; sh holds one value per warp
template <typename T>
__device__ __forceinline__ T block_exclusive_prefix(T base, T sum, T* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const T x = warp_inclusive_scan(sum);
    __syncthreads();
    if (lane == 31) sh[warp] = x;
    __syncthreads();
    T pre = base + (x - sum);
#pragma unroll 1        // at most 31 iterations; unrolled, the tree build's apply kernels took 0.4-0.7 us longer
    for (int w = 0; w < warp; ++w) pre += sh[w];
    return pre;
}

// In-place exclusive scan of the n values data[i * stride] by a single CTA of 1024 threads; returns the total to
// every thread.  Thread t holds PER consecutive values of each chunk of 1024 * PER, and a carry joins the chunks.
template <int PER, typename T>
__device__ __forceinline__ T cta_exclusive_scan(T* data, int n, int stride) {
    __shared__ T wsum[32];
    __shared__ T carry_s, chunk_s;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024 * PER) {
        T v[PER], sum = 0;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int i = base + threadIdx.x * PER + j;
            v[j] = (i < n) ? data[(size_t)i * stride] : T(0);
            sum += v[j];
        }
        const T x = warp_inclusive_scan(sum);
        if (lane == 31) wsum[warp] = x;
        __syncthreads();
        if (warp == 0) {
            const T w = wsum[lane];
            const T xs = warp_inclusive_scan(w);
            wsum[lane] = xs - w;        // exclusive prefix of the warp sums
            if (lane == 31) chunk_s = xs;
        }
        __syncthreads();
        T pre = carry_s + wsum[warp] + (x - sum);
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int i = base + threadIdx.x * PER + j;
            if (i < n) data[(size_t)i * stride] = pre;
            pre += v[j];
        }
        __syncthreads();
        if (threadIdx.x == 0) carry_s += chunk_s;
        __syncthreads();
    }
    return carry_s;
}

}  // namespace b200
