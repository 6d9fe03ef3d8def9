// dpq_tree: the result object of dpq_tree_build / dpq_tree_from_edges (include/dpq.h), shared by
// the host layout (tree_build.cpp) and the device layout (layout.cu).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

struct dpq_tree {
    int M = 0, K = 0;
    int64_t n = 0;
    uint32_t root = 0;
    int64_t n_diffs = 0;
    int64_t edge_us = 0, layout_us = 0;  // wall time of the two build stages (dpq_tree_build)
    std::vector<uint32_t> edges;  // [n-1][2]
    std::vector<uint32_t> vec_id, parent_pos, child_num;
    std::vector<uint8_t> depth;
    std::vector<float> max_dist, max_dist2p;
    std::vector<uint8_t> payload;
    std::vector<uint8_t> codes_by_pos;  // [n][M]
    // Device-resident result (dpq_tree_build_device): what the index needs stays in HBM and the host
    // vectors above stay empty (43 bytes per node of host memory and PCIe traffic at 10^9 codes).
    bool on_device = false;
    int device = 0;
    void* d_codes_by_pos = nullptr;   // uint8 [n][M]
    void* d_depth = nullptr;          // uint8 [n]
    void* d_vec_id = nullptr;         // uint32 [n]
    void* d_payload = nullptr;        // the byte stream, payload_bytes
    void* d_roff = nullptr;           // uint64 [n-1]: stream offset of node p's record - M, at index p - 1
    int64_t payload_bytes = 0;
    std::vector<int64_t> depth_hist;  // nodes per depth (device build)
    ~dpq_tree();
};

namespace dpq {
// dmain:107-116: the K x K centroid distance tables that order the children, [M][K][K]
void centroid_tables(const float* cw, int M, int K, int Ds, std::vector<float>& T);
// DFS layout + stream on the GPU (layout.cu): fills every array of *t from t->edges / t->root.
// codes: [n][M] host pointer.  Returns 0 or a DPQ_ERR_* code (text via dpq_last_error).
// d_edges: the edges already on the device (uint32 [n-1][2]) or nullptr to upload t->edges; keep_on_device:
// leave the result in HBM (dpq_tree::on_device) instead of copying every array to the host; keep_qnode_fields (with
// keep_on_device): also copy parent_pos, child_num, max_dist and max_dist2p to the host vectors (dpq_index_compact).
int layout_tree_device(const uint8_t* codes, int64_t n, int M, int K, const float* cw, int Ds, dpq_tree* t,
                       const uint32_t* d_edges = nullptr, bool keep_on_device = false, bool keep_qnode_fields = false);
// edge search with the result left on the device: *d_edges_out is a cudaMalloc'ed uint32 [n-1][2] array the
// caller frees; codes may be a host or a device pointer (edges.cu)
int find_edges_device(const uint8_t* codes, int64_t n, int M, int K, int max_height_folds, int method,
                      uint32_t** d_edges_out, uint32_t* root_id);
void tree_release_device(dpq_tree* t);  // layout.cu
int tree_copy_device(const dpq_tree* t, const void* src, void* dst, size_t bytes);
// depth-1 subtree shards of a device-resident tree (same deal as the stream reader, program.cpp)
int tree_shard_bounds(const dpq_tree* t, int n_ranks, std::vector<int64_t>* bounds, std::vector<int64_t>* bytes);
int depth_hist_device(int device, const uint8_t* d_depth, int64_t n, int64_t* hist17);
// the on-disk stream decoded on the GPU into a device-resident tree (program_dev.cu); payload / pos2id: host
int decode_stream_device(const uint8_t* payload, int64_t n_bytes, int64_t n, int M, int K, const uint32_t* pos2id,
                         dpq_tree** out);
// DPQ_ERR_ARG when a code byte is >= K (host or device pointer; no-op for K == 256)
int check_code_range(const uint8_t* codes, int64_t n, int M, int K);
}  // namespace dpq
