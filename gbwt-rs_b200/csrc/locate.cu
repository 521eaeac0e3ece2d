// locate.cu -- gbwt_b200_locate / gbwt_b200_locate_states (gbwt_b200.h): one lane per BWT position walks Record::lf
// until it meets a locate sample (record_scan.cuh: gbwt_locate), and the sort that turns the samples of the build walk
// (kernels.cuh: k_build_locate) into the table the walks search.
#include "locate.h"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>

#include "record_scan.cuh"

namespace gbwt_b200 {

namespace {

constexpr int LOCATE_THREADS = 256;

unsigned grid_of(uint64_t n, int sm_count) {
    const uint64_t blocks = (n + LOCATE_THREADS - 1) / LOCATE_THREADS;
    const uint64_t wave = static_cast<uint64_t>(std::max(1, sm_count)) * (2048 / LOCATE_THREADS);
    return static_cast<unsigned>(std::max<uint64_t>(1, std::min(blocks, wave)));
}

// One atomic per warp for the LF-step counter (GBWT_B200_LOCATE_STATS).
__device__ __forceinline__ void add_steps(unsigned long long* steps, uint64_t mine) {
    if (steps == nullptr) return;
    for (int d = 16; d > 0; d >>= 1) mine += __shfl_down_sync(0xFFFFFFFFu, mine, d);
    if ((threadIdx.x & 31u) == 0 && mine != 0) atomicAdd(steps, static_cast<unsigned long long>(mine));
}

// first[r] = first slot of record r in the sorted keys (lower bound of r << 32), r = 0 .. records.
__global__ void __launch_bounds__(LOCATE_THREADS) k_locate_first(const uint64_t* __restrict__ keys, uint64_t count, uint64_t records,
                                                                 uint32_t* __restrict__ first) {
    for (uint64_t r = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; r <= records; r += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const uint64_t key = r << 32;
        uint64_t lo = 0, hi = count;
        while (lo < hi) {
            const uint64_t mid = lo + (hi - lo) / 2;
            if (__ldg(keys + mid) < key) lo = mid + 1; else hi = mid;
        }
        first[r] = static_cast<uint32_t>(lo);
    }
}

// Loops are warp-uniform in their trip count (grid stride over a multiple of 32 lanes), so the step counter's shuffles
// see full warps.
__global__ void __launch_bounds__(LOCATE_THREADS) k_locate(IndexView ix, LocateView lv, const gbwt_b200_pos* __restrict__ positions,
                                                           uint64_t n, gbwt_b200_occurrence* __restrict__ out,
                                                           unsigned long long* __restrict__ steps) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t base = blockIdx.x * static_cast<uint64_t>(blockDim.x); base < n; base += stride) {
        const uint64_t q = base + threadIdx.x;
        uint64_t taken = 0;
        if (q < n) {
            const gbwt_b200_pos p = positions[q];
            gbwt_b200_occurrence o;
            gbwt_locate(ix, lv, p.node, p.offset, o, taken);
            out[q] = o;
        }
        add_steps(steps, taken);
    }
}

// take[q] = how many occurrences of state q are written (its count, clipped to its output slot); counts[q] = its count.
__global__ void __launch_bounds__(LOCATE_THREADS) k_locate_take(const gbwt_b200_state* __restrict__ states, uint64_t n,
                                                                const uint64_t* __restrict__ out_offsets, uint64_t* __restrict__ take,
                                                                uint64_t* __restrict__ counts) {
    for (uint64_t q = blockIdx.x * static_cast<uint64_t>(blockDim.x) + threadIdx.x; q < n; q += static_cast<uint64_t>(gridDim.x) * blockDim.x) {
        const gbwt_b200_state st = states[q];
        const uint64_t count = st.end > st.start ? st.end - st.start : 0;
        if (counts != nullptr) counts[q] = count;
        if (take != nullptr) {
            const uint64_t lo = out_offsets[q], hi = out_offsets[q + 1], slot = hi > lo ? hi - lo : 0;
            take[q] = count < slot ? count : slot;
        }
    }
}

// One lane per occurrence: lane p finds its state in the exclusive scan of take[] (neighbouring lanes take neighbouring
// offsets of the same state, so they start in the same record), then walks.
__global__ void __launch_bounds__(LOCATE_THREADS) k_locate_states(IndexView ix, LocateView lv, const gbwt_b200_state* __restrict__ states,
                                                                  uint64_t n, const uint64_t* __restrict__ scan,
                                                                  const uint64_t* __restrict__ take, const uint64_t* __restrict__ out_offsets,
                                                                  uint64_t out_base, gbwt_b200_occurrence* __restrict__ out,
                                                                  unsigned long long* __restrict__ steps) {
    const uint64_t total = scan[n - 1] + take[n - 1];
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * blockDim.x;
    for (uint64_t base = blockIdx.x * static_cast<uint64_t>(blockDim.x); base < total; base += stride) {
        const uint64_t p = base + threadIdx.x;
        uint64_t taken = 0;
        if (p < total) {
            uint64_t lo = 0, hi = n;  // last q with scan[q] <= p (states that take nothing share their scan value)
            while (hi - lo > 1) {
                const uint64_t mid = lo + (hi - lo) / 2;
                if (__ldg(scan + mid) <= p) lo = mid; else hi = mid;
            }
            const uint64_t k = p - __ldg(scan + lo);
            const gbwt_b200_state st = states[lo];
            gbwt_b200_occurrence o;
            gbwt_locate(ix, lv, st.node, st.start + k, o, taken);
            out[__ldg(out_offsets + lo) - out_base + k] = o;
        }
        add_steps(steps, taken);
    }
}

}  // namespace

cudaError_t locate_sort_samples(uint64_t* keys, LocateSample* samples, uint64_t count, uint64_t records, LocateSample* table,
                                uint32_t* first, int sm_count, cudaStream_t s) {
    int end_bit = 32;
    while (end_bit < 64 && (records >> (end_bit - 32)) != 0) end_bit++;
    uint64_t* keys_out = nullptr;
    void* temp = nullptr;
    size_t temp_bytes = 0;
    cudaError_t e = cudaSuccess;
    if (count > 0) {
        // (count <= 2^32 - 1, checked by the caller; CUB takes the item count as a signed 64-bit value here)
        e = cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys, keys, samples, table, static_cast<int64_t>(count), 0, end_bit, s);
        if (e == cudaSuccess) e = cudaMallocAsync(reinterpret_cast<void**>(&keys_out), count * sizeof(uint64_t), s);
        if (e == cudaSuccess) e = cudaMallocAsync(&temp, std::max<size_t>(temp_bytes, 16), s);
        if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys, keys_out, samples, table, static_cast<int64_t>(count), 0, end_bit, s);
    }
    if (e == cudaSuccess) {
        k_locate_first<<<grid_of(records + 1, sm_count), LOCATE_THREADS, 0, s>>>(keys_out, count, records, first);
        e = cudaGetLastError();
    }
    if (temp != nullptr) cudaFreeAsync(temp, s);
    if (keys_out != nullptr) cudaFreeAsync(keys_out, s);
    return e;
}

cudaError_t launch_locate(const IndexView& ix, const LocateView& lv, const gbwt_b200_pos* positions, uint64_t n,
                          gbwt_b200_occurrence* out, unsigned long long* steps, int sm_count, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    k_locate<<<grid_of(n, sm_count), LOCATE_THREADS, 0, s>>>(ix, lv, positions, n, out, steps);
    return cudaGetLastError();
}

cudaError_t launch_locate_states(const IndexView& ix, const LocateView& lv, const gbwt_b200_state* states, uint64_t n,
                                 const uint64_t* out_offsets, uint64_t base, gbwt_b200_occurrence* out, uint64_t* counts,
                                 unsigned long long* steps, int sm_count, cudaStream_t s) {
    if (n == 0) return cudaSuccess;
    if (out == nullptr) {
        k_locate_take<<<grid_of(n, sm_count), LOCATE_THREADS, 0, s>>>(states, n, nullptr, nullptr, counts);
        return cudaGetLastError();
    }
    uint64_t *take = nullptr, *scan = nullptr;
    void* temp = nullptr;
    size_t temp_bytes = 0;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&take), n * sizeof(uint64_t), s);
    if (e == cudaSuccess) e = cudaMallocAsync(reinterpret_cast<void**>(&scan), n * sizeof(uint64_t), s);
    if (e == cudaSuccess) {
        k_locate_take<<<grid_of(n, sm_count), LOCATE_THREADS, 0, s>>>(states, n, out_offsets, take, counts);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(nullptr, temp_bytes, take, scan, static_cast<int64_t>(n), s);
    if (e == cudaSuccess) e = cudaMallocAsync(&temp, std::max<size_t>(temp_bytes, 16), s);
    if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(temp, temp_bytes, take, scan, static_cast<int64_t>(n), s);
    if (e == cudaSuccess) {
        // (the total is read on the device: no round trip to size the grid; a full wave loops over it)
        k_locate_states<<<grid_of(uint64_t(1) << 40, sm_count), LOCATE_THREADS, 0, s>>>(ix, lv, states, n, scan, take, out_offsets, base, out, steps);
        e = cudaGetLastError();
    }
    if (temp != nullptr) cudaFreeAsync(temp, s);
    if (take != nullptr) cudaFreeAsync(take, s);
    if (scan != nullptr) cudaFreeAsync(scan, s);
    return e;
}

}  // namespace gbwt_b200
