// Device building blocks of the merge, ICP, frontier and route kernels: a block-wide scan, a
// single-CTA scan of per-block counts and a grid barrier for cooperative launches.
#pragma once
#include <cuda_runtime.h>

namespace occ {

// Block-wide exclusive scan of one value per thread, T = unsigned int or unsigned long long (the
// type of s_warp; v is converted to it).  Every thread of the block calls it; blockDim.x is a
// multiple of 32 and at most 1024.  Returns the sum of v over the lower threads and sets *total
// to the sum over the block, in every thread.  s_warp holds 33 shared entries; it can be reused
// as soon as the call returns.
template <class T, class V>
__device__ __forceinline__ T block_exclusive_scan(V value, T* s_warp /* 33 */, T* total) {
    const T v = (T)value;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        T w = (lane < (int)(blockDim.x >> 5)) ? s_warp[lane] : T(0);
        T winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            T t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        s_warp[lane] = winc - w;          // exclusive warp offsets
        if (lane == 31) s_warp[32] = winc;   // block total
    }
    __syncthreads();
    T res = s_warp[warp] + inc - v;
    *total = s_warp[32];
    __syncthreads();
    return res;
}

// Single-CTA exclusive scan of n per-block counts in place: a[i] = carry + a[0] + ... + a[i - 1],
// stored in 32 bits.  Each thread takes kItems consecutive counts per round of blockDim.x * kItems.
// Every thread of the one CTA calls it; all get carry + the sum of the n counts.
template <int kItems>
__device__ __forceinline__ unsigned long long cta_scan_in_place(unsigned int* a, int n, unsigned long long carry) {
    __shared__ unsigned int s_warp[33];
    for (int start = 0; start < n; start += (int)blockDim.x * kItems) {
        const int i0 = start + (int)threadIdx.x * kItems;
        unsigned int v[kItems], sum = 0;
#pragma unroll
        for (int j = 0; j < kItems; ++j) { v[j] = (i0 + j < n) ? a[i0 + j] : 0u; sum += v[j]; }
        unsigned int total;
        unsigned int run = (unsigned int)carry + block_exclusive_scan(sum, s_warp, &total);
#pragma unroll
        for (int j = 0; j < kItems; ++j) {
            if (i0 + j < n) a[i0 + j] = run;
            run += v[j];
        }
        carry += total;
    }
    return carry;
}

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Grid-wide barrier over co-resident CTAs (cooperative launch).  bar[0] counts arrivals, bar[1] is
// free for the caller's exit count, bar[2] is the release word and bar[3] the verdict the LAST
// arriver computed (`last_arriver()` runs in exactly one thread of the grid, after every CTA's
// pre-barrier writes are visible and before anybody is released), so a decision every CTA must
// agree on is single-sourced: nobody re-derives it from state a faster CTA may already be
// overwriting in the next phase.  The words start at zero; `target` starts at zero in every CTA.
// A CTA that waits longer than kGridBarrierTimeoutNs, or finds *abort_flag set, gives up (returns
// false, sets *abort_flag): a missing CTA can then no longer hang the device.
constexpr unsigned long long kGridBarrierTimeoutNs = 2000000000ull;

template <class F>
__device__ __forceinline__ bool grid_barrier(unsigned int* bar, unsigned int& target, int* abort_flag, int* verdict, F&& last_arriver) {
    __shared__ int s_ok, s_verdict;
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        int ok = 1;
        __threadfence();
        if (atomicAdd(bar, 1u) == target - 1u) {               // last arriver: decide, publish, release
            __threadfence();
            reinterpret_cast<volatile unsigned int*>(bar)[3] = (unsigned int)last_arriver();
            __threadfence();
            reinterpret_cast<volatile unsigned int*>(bar)[2] = target;
        } else {
            const unsigned long long t0 = global_ns();
            unsigned int spins = 0;
            while (reinterpret_cast<volatile unsigned int*>(bar)[2] < target) {
                if (((++spins) & 1023u) == 0u &&
                    (*reinterpret_cast<volatile int*>(abort_flag) || global_ns() - t0 > kGridBarrierTimeoutNs)) {
                    atomicExch(abort_flag, 1);
                    ok = 0;
                    break;
                }
            }
        }
        __threadfence();
        s_ok = ok;
        s_verdict = (int)reinterpret_cast<volatile unsigned int*>(bar)[3];
    }
    __syncthreads();
    if (verdict) *verdict = s_verdict;
    return s_ok != 0;
}

__device__ __forceinline__ bool grid_barrier(unsigned int* bar, unsigned int& target, int* abort_flag) {
    return grid_barrier(bar, target, abort_flag, nullptr, [] { return 0; });
}

}  // namespace occ
