// compact.cu: the device half of dpq_index_compact / dpq_multi_compact.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace dpq {
// d_cnt [words + 1] (words = ceil(n / 32)) receives the live nodes of each 32-node word of the dead bitmap (d_dead
// null: all live), d_off [words + 1] their exclusive sum: d_off[words] = the live count.  d_temp = null:
// *temp_bytes receives the scan's scratch size and nothing runs.
cudaError_t count_live(const uint32_t* d_dead, int64_t n, uint32_t* d_cnt, uint32_t* d_off, void* d_temp, size_t* temp_bytes,
                       cudaStream_t st);
// Live node i (local position, ascending) -> row r: d_out_codes[r] = its code word of nf padded bytes cut to M,
// d_out_ids[r] = d_pos2id[i], or base_pos + i when d_pos2id is null.  d_off from count_live (unused without d_dead).
// nf other than 8 or 16 (not a code-array layout): cudaErrorInvalidValue, nothing runs.
cudaError_t gather_live(const uint8_t* d_codes, int nf, int64_t n, int M, const uint32_t* d_dead, const uint32_t* d_off,
                        const uint32_t* d_pos2id, uint32_t base_pos, uint8_t* d_out_codes, uint32_t* d_out_ids, cudaStream_t st);
// d_vec_id[p] = d_ids[d_vec_id[p]] for p < n: a tree built over gathered rows reports the rows' carried ids
cudaError_t map_tree_ids(uint32_t* d_vec_id, int64_t n, const uint32_t* d_ids, cudaStream_t st);
}  // namespace dpq
