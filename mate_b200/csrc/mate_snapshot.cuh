// mate_snapshot.cuh -- device-side state snapshots (mate_b200_save_state / mate_b200_load_state): one gather and one
// scatter kernel over the per-environment struct-of-arrays members of a state block.
//
// The host code (mate_b200.cu) describes every array of for_each_state_array as a SnapArray: its live rows
// ([row * bpad + env]) and its section of the payload ([row * count + i]).  Block row y of a launch handles one row of
// one array; the threads of a block walk consecutive entries, so the side that is contiguous (the payload, and the
// state wherever the index map is the identity) is read and written in whole 32-lane runs of 4-, 8- or 16-byte words.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace mate {

constexpr int kSnapMaxArrays = 16;   // for_each_state_array visits 15
constexpr int kSnapThreads = 256;
constexpr int kSnapPerThread = 4;    // entries per thread, loaded before any is stored

struct SnapArray {
    char* state;     // live rows [rows][bpad]
    char* payload;   // payload section [rows][count]
    int rows;        // > 0
    int elem;        // bytes per element: 4, 8 or 16
};

struct SnapTable {
    SnapArray a[kSnapMaxArrays];
    int n;                    // arrays in `a`
    int rows;                 // sum of a[k].rows (= gridDim.y)
    int bpad, num_envs, count;
    float* stats;             // the handle's 16 statistics accumulators
    float* payload_stats;     // their place at the end of the payload
    int copy_stats;           // scatter only: load the statistics too (resume)
    uint32_t* ready;          // scatter only: prepared-episode tags, zeroed for every loaded environment (nullptr = none)
};

// the array and row of block row y (static indices only, so that the table stays in the parameter bank)
__device__ __forceinline__ SnapArray snap_row(const SnapTable& t, int y, int* row) {
    SnapArray out = t.a[0];
    bool found = false;
#pragma unroll
    for (int k = 0; k < kSnapMaxArrays; ++k) {
        if (!found && k < t.n) {
            if (y < t.a[k].rows) { out = t.a[k]; found = true; }
            else y -= t.a[k].rows;
        }
    }
    *row = y;
    return out;
}

// payload entry i <- live environment env[i] (identity without a list); an entry whose environment is outside
// [0, num_envs) is left unwritten
template <typename T>
__device__ __forceinline__ void snap_gather_row(const SnapArray& a, int row, const SnapTable& t, const int32_t* __restrict__ env) {
    const T* __restrict__ src = reinterpret_cast<const T*>(a.state) + (size_t)row * t.bpad;
    T* __restrict__ dst = reinterpret_cast<T*>(a.payload) + (size_t)row * t.count;
    const int first = blockIdx.x * (kSnapThreads * kSnapPerThread) + threadIdx.x;
    T v[kSnapPerThread];
    bool ok[kSnapPerThread];
#pragma unroll
    for (int u = 0; u < kSnapPerThread; ++u) {
        const int i = first + u * kSnapThreads;
        int e = i;
        ok[u] = i < t.count;
        if (ok[u] && env != nullptr) { e = __ldg(env + i); ok[u] = e >= 0 && e < t.num_envs; }
        if (ok[u]) v[u] = src[e];
    }
#pragma unroll
    for (int u = 0; u < kSnapPerThread; ++u)
        if (ok[u]) __stcs(dst + first + u * kSnapThreads, v[u]);
}

// live environment d <- payload entry src[d] (identity without a map); an environment whose entry is outside
// [0, count) is left unchanged
template <typename T>
__device__ __forceinline__ void snap_scatter_row(const SnapArray& a, int row, const SnapTable& t, const int32_t* __restrict__ map,
                                                 bool first_row) {
    const T* __restrict__ src = reinterpret_cast<const T*>(a.payload) + (size_t)row * t.count;
    T* __restrict__ dst = reinterpret_cast<T*>(a.state) + (size_t)row * t.bpad;
    const int first = blockIdx.x * (kSnapThreads * kSnapPerThread) + threadIdx.x;
    T v[kSnapPerThread];
    bool ok[kSnapPerThread];
#pragma unroll
    for (int u = 0; u < kSnapPerThread; ++u) {
        const int d = first + u * kSnapThreads;
        int s = d;
        ok[u] = d < t.num_envs;
        if (ok[u] && map != nullptr) s = __ldg(map + d);
        ok[u] = ok[u] && s >= 0 && s < t.count;
        if (ok[u]) v[u] = src[s];   // cached: a branching load reads a few entries many times
    }
#pragma unroll
    for (int u = 0; u < kSnapPerThread; ++u) {
        const int d = first + u * kSnapThreads;
        if (ok[u]) {
            dst[d] = v[u];
            if (first_row && t.ready != nullptr) t.ready[d] = 0u;   // its prepared next episode belongs to the old state
        }
    }
}

__global__ void __launch_bounds__(kSnapThreads) snapshot_gather_kernel(const __grid_constant__ SnapTable t, const int32_t* __restrict__ env) {
    int row;
    const SnapArray a = snap_row(t, blockIdx.y, &row);
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 16) t.payload_stats[threadIdx.x] = t.stats[threadIdx.x];
    if (blockIdx.x == 0 && row == a.rows - 1) {   // the section's alignment padding is zeroed: equal states give equal payloads
        const size_t end = (size_t)a.rows * t.count * a.elem;
        if (threadIdx.x < (256 - end % 256) % 256) a.payload[end + threadIdx.x] = 0;
    }
    if (a.elem == 16) snap_gather_row<uint4>(a, row, t, env);
    else if (a.elem == 8) snap_gather_row<unsigned long long>(a, row, t, env);
    else snap_gather_row<uint32_t>(a, row, t, env);
}

__global__ void __launch_bounds__(kSnapThreads) snapshot_scatter_kernel(const __grid_constant__ SnapTable t, const int32_t* __restrict__ map) {
    int row;
    const SnapArray a = snap_row(t, blockIdx.y, &row);
    if (t.copy_stats && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 16) t.stats[threadIdx.x] = t.payload_stats[threadIdx.x];
    const bool first_row = blockIdx.y == 0;
    if (a.elem == 16) snap_scatter_row<uint4>(a, row, t, map, first_row);
    else if (a.elem == 8) snap_scatter_row<unsigned long long>(a, row, t, map, first_row);
    else snap_scatter_row<uint32_t>(a, row, t, map, first_row);
}

// `entries`: payload entries (gather) or live environments (scatter) the launch covers
inline dim3 snapshot_grid(const SnapTable& t, int entries) {
    const int per_block = kSnapThreads * kSnapPerThread;
    return dim3((unsigned)((entries + per_block - 1) / per_block), (unsigned)t.rows);
}

}  // namespace mate
