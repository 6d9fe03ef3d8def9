// Appended nodes (dpq_index_add / dpq_index_add_vectors): an add batch is sorted on the device by code word
// (subspace 0 most significant, ties by input row) and gathered into the tail of the code array, so that
// consecutive appended positions share centroids the way DFS neighbours of the tree do and the coarse scan's
// row reuse (DESIGN §4.1) keeps working on them.  Not on the search path: one or two radix sorts and one
// gather per call.
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>

#include "kernels.cuh"

namespace dpq {

// Sort key of one code: code bytes [8 * word, 8 * word + 8) of the zero-padded word, the first of them the most
// significant byte.
__device__ __forceinline__ uint64_t code_key(const uint8_t* __restrict__ row, int M, int word) {
    uint64_t k = 0;
#pragma unroll
    for (int b = 0; b < 8; ++b) {
        const int m = word * 8 + b;
        k = (k << 8) | (m < M ? row[m] : 0u);
    }
    return k;
}

// keys[i] = key of input row perm[i] (row i when perm is null); vals[i] = that row
__global__ void add_keys_kernel(const uint8_t* __restrict__ codes, int64_t n, int M, int word, const uint32_t* __restrict__ perm,
                                uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t r = perm ? perm[i] : (uint32_t)i;
    keys[i] = code_key(codes + (size_t)r * M, M, word);
    vals[i] = r;
}

// Appended node i takes input row r = perm[i] (or i): its padded code word, its id (ids[r], or its position when
// ids is null) and, at the row's own index, its position.
template <int NF>
__global__ void add_gather_kernel(const uint8_t* __restrict__ codes, int64_t n, int M, const uint32_t* __restrict__ perm,
                                  const uint32_t* __restrict__ ids, uint32_t first_pos, uint8_t* __restrict__ out_codes,
                                  uint32_t* __restrict__ out_ids, uint32_t* __restrict__ out_pos) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t r = perm ? perm[i] : (uint32_t)i;
    const uint8_t* row = codes + (size_t)r * M;
    uint32_t w[NF / 4];
#pragma unroll
    for (int j = 0; j < NF / 4; ++j) {
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int m = 4 * j + b;
            v |= (uint32_t)(m < M ? row[m] : 0u) << (8 * b);
        }
        w[j] = v;
    }
    if constexpr (NF == 8) reinterpret_cast<uint2*>(out_codes)[i] = make_uint2(w[0], w[1]);
    else reinterpret_cast<uint4*>(out_codes)[i] = make_uint4(w[0], w[1], w[2], w[3]);
    const uint32_t pos = first_pos + (uint32_t)i;
    if (out_ids) out_ids[i] = ids ? ids[r] : pos;
    out_pos[r] = pos;
}

cudaError_t sort_add_batch(const uint8_t* d_codes, int64_t n, int M, int nf, uint64_t* d_keys, uint32_t* d_vals, void* d_temp,
                           size_t* temp_bytes, cudaStream_t st) {
    const int N = (int)n;
    // the narrow shape has one pass over subspaces 0..7; the wide shape sorts by subspaces 8..15 first, then
    // stably by 0..7.  Bytes of subspaces >= M are zero in every key: the sort skips their bits.
    const int passes = nf == 16 ? 2 : 1;
    const int low_begin = 8 * std::max(0, nf - M);
    if (!d_temp) {
        size_t t = 0;
        cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, t, d_keys, d_keys + n, d_vals, d_vals + n, N, 0, 64, st);
        *temp_bytes = t;
        return e;
    }
    const unsigned blocks = (unsigned)((n + 255) / 256);
    for (int p = 0; p < passes; ++p) {
        const int word = passes - 1 - p;
        // pass 0 reads the rows in input order; pass 1 the order pass 0 left in d_vals + n
        add_keys_kernel<<<blocks, 256, 0, st>>>(d_codes, n, M, word, p ? d_vals + n : nullptr, d_keys, d_vals);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
        e = cub::DeviceRadixSort::SortPairs(d_temp, *temp_bytes, d_keys, d_keys + n, d_vals, d_vals + n, N, p == 0 ? low_begin : 0,
                                            64, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

cudaError_t launch_add_gather(const uint8_t* d_codes, int64_t n, int M, int nf, const uint32_t* d_perm, const uint32_t* d_ids,
                              uint32_t first_pos, uint8_t* d_out_codes, uint32_t* d_out_ids, uint32_t* d_out_pos, cudaStream_t st) {
    const unsigned blocks = (unsigned)((n + 255) / 256);
    if (nf == 8)
        add_gather_kernel<8><<<blocks, 256, 0, st>>>(d_codes, n, M, d_perm, d_ids, first_pos, d_out_codes, d_out_ids, d_out_pos);
    else
        add_gather_kernel<16><<<blocks, 256, 0, st>>>(d_codes, n, M, d_perm, d_ids, first_pos, d_out_codes, d_out_ids, d_out_pos);
    return cudaGetLastError();
}

}  // namespace dpq
