// Compaction (dpq_index_compact / dpq_multi_compact): the live nodes of an open index are gathered on the
// device, in ascending local position, into the unpadded [n_live][M] code layout and the id table that
// dpq_tree_build* take, and the new tree's vec_id (a row of that layout) is mapped back to the carried ids.
// Not on the search path: one count pass, one CUB scan and one gather per call.
#include <cub/device/device_scan.cuh>

#include "compact.cuh"

namespace dpq {

namespace {

// live bits of 32-node word w: not deleted and below n
__device__ __forceinline__ uint32_t live_bits(const uint32_t* __restrict__ dead, int64_t n, int64_t w) {
    const int64_t rest = n - 32 * w;
    const uint32_t valid = rest >= 32 ? 0xFFFFFFFFu : ((1u << rest) - 1u);
    return (dead ? ~dead[w] : 0xFFFFFFFFu) & valid;
}

__global__ void live_count_kernel(const uint32_t* __restrict__ dead, int64_t n, int64_t words, uint32_t* __restrict__ cnt) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w < words) cnt[w] = (uint32_t)__popc(live_bits(dead, n, w));
}

// Node i, when live, goes to row off[i / 32] + (live nodes below it in its word): its padded word of NF bytes
// un-padded to M bytes, its id pos2id[i] (or base_pos + i without a table).
template <int NF>
__global__ void live_gather_kernel(const uint8_t* __restrict__ codes, int64_t n, int M, const uint32_t* __restrict__ dead,
                                   const uint32_t* __restrict__ off, const uint32_t* __restrict__ pos2id, uint32_t base_pos,
                                   uint8_t* __restrict__ out_codes, uint32_t* __restrict__ out_ids) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t j = i;
    if (dead) {
        const uint32_t live = live_bits(dead, n, i >> 5);
        const uint32_t b = (uint32_t)(i & 31);
        if (!((live >> b) & 1u)) return;
        j = (int64_t)off[i >> 5] + __popc(live & ((1u << b) - 1u));
    }
    uint32_t w[NF / 4];
    if constexpr (NF == 8) {
        const uint2 v = reinterpret_cast<const uint2*>(codes)[i];
        w[0] = v.x;
        w[1] = v.y;
    } else {
        const uint4 v = reinterpret_cast<const uint4*>(codes)[i];
        w[0] = v.x;
        w[1] = v.y;
        w[2] = v.z;
        w[3] = v.w;
    }
    uint8_t* dst = out_codes + (size_t)j * M;
#pragma unroll
    for (int m = 0; m < NF; ++m)
        if (m < M) dst[m] = (uint8_t)(w[m >> 2] >> (8 * (m & 3)));
    out_ids[j] = pos2id ? pos2id[i] : base_pos + (uint32_t)i;
}

__global__ void map_ids_kernel(uint32_t* __restrict__ vec, int64_t n, const uint32_t* __restrict__ ids) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n) vec[p] = ids[vec[p]];
}

unsigned grid(int64_t n) { return (unsigned)((n + 255) / 256); }

}  // namespace

cudaError_t count_live(const uint32_t* d_dead, int64_t n, uint32_t* d_cnt, uint32_t* d_off, void* d_temp, size_t* temp_bytes,
                       cudaStream_t st) {
    const int64_t words = (n + 31) / 32;
    if (!d_temp) return cub::DeviceScan::ExclusiveSum(nullptr, *temp_bytes, d_cnt, d_off, (int)(words + 1), st);
    cudaError_t e = cudaMemsetAsync(d_cnt + words, 0, 4, st);
    if (e != cudaSuccess) return e;
    if (words) live_count_kernel<<<grid(words), 256, 0, st>>>(d_dead, n, words, d_cnt);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    return cub::DeviceScan::ExclusiveSum(d_temp, *temp_bytes, d_cnt, d_off, (int)(words + 1), st);
}

cudaError_t gather_live(const uint8_t* d_codes, int nf, int64_t n, int M, const uint32_t* d_dead, const uint32_t* d_off,
                        const uint32_t* d_pos2id, uint32_t base_pos, uint8_t* d_out_codes, uint32_t* d_out_ids, cudaStream_t st) {
    if (nf != 8 && nf != 16) return cudaErrorInvalidValue;  // only the code-array layout has padded words
    if (n == 0) return cudaSuccess;
    if (nf == 8)
        live_gather_kernel<8><<<grid(n), 256, 0, st>>>(d_codes, n, M, d_dead, d_off, d_pos2id, base_pos, d_out_codes, d_out_ids);
    else
        live_gather_kernel<16><<<grid(n), 256, 0, st>>>(d_codes, n, M, d_dead, d_off, d_pos2id, base_pos, d_out_codes, d_out_ids);
    return cudaGetLastError();
}

cudaError_t map_tree_ids(uint32_t* d_vec_id, int64_t n, const uint32_t* d_ids, cudaStream_t st) {
    if (n > 0) map_ids_kernel<<<grid(n), 256, 0, st>>>(d_vec_id, n, d_ids);
    return cudaGetLastError();
}

}  // namespace dpq
