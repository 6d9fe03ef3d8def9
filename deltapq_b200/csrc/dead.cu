// Deleted nodes (dpq_index_delete / dpq_index_undelete): vector ids -> bits of the per-index bitmap that
// the scan kernels test before they append a candidate.  Not on the search path: one sort of the ids and
// one pass over the shard's positions per call.
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>

#include "kernels.cuh"

namespace dpq {

cudaError_t sort_ids(const uint32_t* d_in, uint32_t* d_out, int n, void* d_temp, size_t* temp_bytes, cudaStream_t st) {
    return cub::DeviceRadixSort::SortKeys(d_temp, *temp_bytes, d_in, d_out, n, 0, 32, st);
}

// One thread per 32-position word: each of its nodes' ids is binary-searched in the sorted id list, and the
// word is written once (no atomics).  Then the block's popcounts are summed into *count.
__global__ void __launch_bounds__(256) mark_dead_kernel(const uint32_t* __restrict__ ids, int64_t n_ids,
                                                        const uint32_t* __restrict__ pos2id, uint32_t base_pos, int64_t n_local,
                                                        bool set, uint32_t* __restrict__ dead, unsigned long long* __restrict__ count) {
    __shared__ unsigned s_sum;
    if (threadIdx.x == 0) s_sum = 0u;
    __syncthreads();
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t n_words = (n_local + 31) / 32;
    unsigned bits = 0u;
    if (w < n_words) {
        uint32_t found = 0u;
        for (int b = 0; b < 32; ++b) {
            const int64_t i = w * 32 + b;
            if (i >= n_local) break;
            const uint32_t id = pos2id ? pos2id[i] : base_pos + (uint32_t)i;
            int64_t lo = 0, hi = n_ids;  // first listed id >= id
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (ids[mid] < id) lo = mid + 1;
                else hi = mid;
            }
            if (lo < n_ids && ids[lo] == id) found |= 1u << b;
        }
        const uint32_t old = dead[w];
        const uint32_t v = set ? (old | found) : (old & ~found);
        dead[w] = v;
        bits = (unsigned)__popc(v);
    }
    bits = __reduce_add_sync(0xffffffffu, bits);
    if ((threadIdx.x & 31) == 0 && bits) atomicAdd(&s_sum, bits);
    __syncthreads();
    if (threadIdx.x == 0 && s_sum) atomicAdd(count, (unsigned long long)s_sum);
}

void launch_mark_dead(const uint32_t* d_ids, int64_t n_ids, const uint32_t* d_pos2id, uint32_t base_pos, int64_t n_local,
                      bool set, uint32_t* d_dead, unsigned long long* d_count, cudaStream_t st) {
    const int64_t n_words = (n_local + 31) / 32;
    const unsigned blocks = (unsigned)std::max<int64_t>(1, (n_words + 255) / 256);
    mark_dead_kernel<<<blocks, 256, 0, st>>>(d_ids, n_ids, d_pos2id, base_pos, n_local, set, d_dead, d_count);
}

}  // namespace dpq
