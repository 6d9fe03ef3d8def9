// DeltaTree build, stages 2-3 on the device: edges -> DFS layout -> byte stream.
//
// Reference: edges_to_tree_index_approx_dfs_layout (DCAT.h:1334-1487; CSR :1067-1104; farthest
// descendant :1396-1417; child order :1421-1426; DFS numbering :1156-1183) and
// qnodes_to_compressed_codes_opt (DCAT.h:1765-1842).  tree_build.cpp holds the same stage as a
// sequential host walk (dpq_tree_from_edges, no GPU needed); this file is its data-parallel
// form, used by dpq_tree_build, and the two are compared bit for bit by the GPU tests.
//
// The reference numbers the nodes with a recursive pre-order walk.  A pre-order position is a
// sum along the root path:  pos(v) = sum over the ancestors-or-self a != root of
// (1 + total subtree size of the siblings ordered before a), so the walk becomes
//
//   parent_kernel     parent[child], child count per parent                   (DCAT.h:1067-1104)
//   far_kernel        per node, <= 16 hops up: farthest descendant per node and per child
//                     branch; float max is exact, so atomicMax on the bit patterns (DCAT.h:1396-1417)
//   climb_kernel      depth of every node, descendants per node (one atomic per ancestor)
//   cub radix sort    stable sort of the edges by (parent, far_via descending): children in the
//                     reference's order, emission order on ties                (DCAT.h:1421-1426)
//   cub exclusive sum subtree sizes in child-list order -> offset of each child from its parent
//   pos_kernel        position = sum of the offsets along the root path        (DCAT.h:1156-1183)
//   emit_kernel       arrays by position (vec_id, parent_pos, child_num, depth, max_dist, codes)
//   reclen_kernel     stream record length per position, cub exclusive sum -> byte offsets
//   stream_kernel     every node writes its own record                         (DCAT.h:1765-1842)
//
// The working set is ~70 B/node: a 125M-code shard of the 1B-code workload lays out in HBM.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <cub/cub.cuh>
#include <string>
#include <vector>

#include "../../include/dpq.h"
#include "tree_internal.h"

namespace dpq {
int api_fail(int code, const std::string& msg);
int api_check_device();
int api_device();
}  // namespace dpq

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return dpq::api_fail(DPQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

namespace {

constexpr uint32_t NONE = 0xFFFFFFFFu;
enum : uint32_t { ERR_TWO_PARENTS = 1, ERR_NOT_SPANNING = 2, ERR_TOO_DEEP = 4, ERR_NIBBLE = 8, ERR_RANGE = 16 };

struct Buf {
    void* p = nullptr;
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, std::max<size_t>(bytes, 16)); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
    }
    template <class T>
    T* as() const {
        return reinterpret_cast<T*>(p);
    }
    ~Buf() { release(); }
};

inline unsigned blocks(int64_t n, int t = 256) { return (unsigned)((n + t - 1) / t); }

__global__ void fill_kernel(uint32_t* a, int64_t n, uint32_t v) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = v;
}

__global__ void parent_kernel(const uint32_t* __restrict__ edges, int64_t E, int64_t n, uint32_t root,
                              uint32_t* __restrict__ parent, uint32_t* __restrict__ n_kids,
                              uint32_t* __restrict__ err) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const uint32_t p = edges[2 * e], c = edges[2 * e + 1];
    if (p >= n || c >= n) {
        atomicOr(err, ERR_RANGE);
        return;
    }
    if (c == root || atomicExch(&parent[c], p) != NONE) atomicOr(err, ERR_TWO_PARENTS);
    atomicAdd(&n_kids[p], 1u);
}

// CT.h:827-835: float sum over m ascending of the centroid-table entries
template <int MAXM>
__device__ __forceinline__ float pair_dist(const uint8_t* x, const uint8_t* __restrict__ y, int M, int K,
                                           const float* __restrict__ T) {
    float s = 0.0f;
    for (int m = 0; m < M; ++m) s = __fadd_rn(s, T[((size_t)m * K + x[m]) * K + y[m]]);
    return s;
}

// DCAT.h:1396-1417: every node raises the "farthest descendant" of its <= 16 nearest ancestors
// (far) and of the child branch it hangs under (far_via).  Distances are >= 0, so the float
// maximum is the maximum of the bit patterns.
__global__ void far_kernel(const uint8_t* __restrict__ codes, int64_t n, int M, int K,
                           const uint32_t* __restrict__ parent, const float* __restrict__ T,
                           uint32_t* __restrict__ far, uint32_t* __restrict__ far_via) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    uint8_t x[16];
    for (int m = 0; m < M; ++m) x[m] = codes[(size_t)v * M + m];
    uint32_t below = (uint32_t)v;
    uint32_t anc = parent[v];
    for (int hop = 0; anc != NONE && hop < 16; ++hop) {
        const uint32_t d = __float_as_uint(pair_dist<16>(x, codes + (size_t)anc * M, M, K, T));
        if (d > far[anc]) atomicMax(&far[anc], d);
        if (d > far_via[below]) atomicMax(&far_via[below], d);
        below = anc;
        anc = parent[anc];
    }
}

// depth of every node and the number of descendants of every node but the root (the root's is
// n - 1 by definition; skipping it keeps n atomics off one address)
__global__ void climb_kernel(int64_t n, uint32_t root, const uint32_t* __restrict__ parent,
                             uint8_t* __restrict__ depth, uint32_t* __restrict__ desc, uint32_t* __restrict__ err) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    if ((uint32_t)v == root) {
        depth[v] = 0;
        desc[v] = (uint32_t)(n - 1);
        return;
    }
    uint32_t a = parent[v];
    int hops = 1;
    while (a != root) {
        if (a == NONE) {
            atomicOr(err, ERR_NOT_SPANNING);
            return;
        }
        if (++hops > 255) {
            atomicOr(err, ERR_TOO_DEEP);
            return;
        }
        atomicAdd(&desc[a], 1u);
        a = parent[a];
    }
    depth[v] = (uint8_t)hops;
}

// child-list sort key: parent ascending, then far_via descending; the stable sort keeps the
// emission order among equal keys, as std::stable_sort over each child list does
__global__ void kidkey_kernel(const uint32_t* __restrict__ edges, int64_t E, const uint32_t* __restrict__ far_via,
                              unsigned long long* __restrict__ key, uint32_t* __restrict__ kid) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const uint32_t p = edges[2 * e], c = edges[2 * e + 1];
    key[e] = ((unsigned long long)p << 32) | (unsigned long long)(0xFFFFFFFFu - far_via[c]);
    kid[e] = c;
}

__global__ void kidsize_kernel(const uint32_t* __restrict__ kid, int64_t E, const uint32_t* __restrict__ desc,
                               unsigned long long* __restrict__ sz) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < E) sz[j] = (unsigned long long)desc[kid[j]] + 1ull;
}

// off[c] = 1 + subtree sizes of the siblings listed before c
__global__ void kidoff_kernel(const uint32_t* __restrict__ kid, int64_t E, const uint32_t* __restrict__ parent,
                              const uint32_t* __restrict__ first, const unsigned long long* __restrict__ pre,
                              uint32_t* __restrict__ off) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= E) return;
    const uint32_t c = kid[j];
    off[c] = (uint32_t)(1ull + pre[j] - pre[first[parent[c]]]);
}

__global__ void pos_kernel(int64_t n, uint32_t root, const uint32_t* __restrict__ parent,
                           const uint32_t* __restrict__ off, uint32_t* __restrict__ pos) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    uint32_t p = 0;
    for (uint32_t a = (uint32_t)v; a != root; a = parent[a]) p += off[a];
    pos[v] = p;
}

__global__ void emit_kernel(int64_t n, int M, uint32_t root, const uint8_t* __restrict__ codes,
                            const uint32_t* __restrict__ parent, const uint32_t* __restrict__ pos,
                            const uint32_t* __restrict__ desc, const uint8_t* __restrict__ depth,
                            const uint32_t* __restrict__ far, const uint32_t* __restrict__ far_via,
                            uint32_t* __restrict__ vec_id, uint32_t* __restrict__ parent_pos,
                            uint32_t* __restrict__ child_num, uint8_t* __restrict__ depth_p,
                            float* __restrict__ max_dist, float* __restrict__ max_dist2p,
                            uint8_t* __restrict__ codes_p, uint32_t* __restrict__ err) {
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const uint32_t p = pos[v];
    if (p >= n) {
        atomicOr(err, ERR_NOT_SPANNING);
        return;
    }
    vec_id[p] = (uint32_t)v;
    parent_pos[p] = (uint32_t)v == root ? NONE : pos[parent[v]];
    child_num[p] = desc[v];
    depth_p[p] = depth[v];
    max_dist[p] = __fsqrt_rn(__uint_as_float(far[v]));
    max_dist2p[p] = __fsqrt_rn(__uint_as_float(far_via[v]));
    if (M == 8) {
        reinterpret_cast<uint2*>(codes_p)[p] = reinterpret_cast<const uint2*>(codes)[v];
    } else {
        for (int m = 0; m < M; ++m) codes_p[(size_t)p * M + m] = codes[(size_t)v * M + m];
    }
}

__device__ __forceinline__ uint32_t diff_bitmap(const uint8_t* __restrict__ codes_p, int M, uint32_t p, uint32_t q) {
    uint32_t bm = 0;
    for (int m = 0; m < M; ++m) bm |= (uint32_t)(codes_p[(size_t)p * M + m] != codes_p[(size_t)q * M + m]) << m;
    return bm;
}

// record p (1 <= p < n) = [depth byte if p is odd] + ceil(M/8) bitmap bytes + one byte per
// changed subspace; len[p - 1] so that the exclusive sum starts at the first record
__global__ void reclen_kernel(int64_t n, int M, const uint8_t* __restrict__ codes_p,
                              const uint32_t* __restrict__ parent_pos, const uint8_t* __restrict__ depth_p,
                              unsigned long long* __restrict__ len, uint32_t* __restrict__ err) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x + 1;
    if (p >= n) return;
    if (depth_p[p] > (M > 8 ? 15 : 7)) atomicOr(err, ERR_NIBBLE);  // M <= 8: the reader masks nibbles with &7 (DCAT.h:3794)
    const uint32_t bm = diff_bitmap(codes_p, M, (uint32_t)p, parent_pos[p]);
    len[p - 1] = (unsigned long long)((M + 7) / 8 + __popc(bm) + (int)(p & 1));
}

__global__ void stream_kernel(int64_t n, int M, const uint8_t* __restrict__ codes_p,
                              const uint32_t* __restrict__ parent_pos, const uint8_t* __restrict__ depth_p,
                              const unsigned long long* __restrict__ off, uint8_t* __restrict__ out) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    if (p == 0) {
        for (int m = 0; m < M; ++m) out[m] = codes_p[m];
        return;
    }
    uint8_t* o = out + (size_t)M + off[p - 1];
    if (p & 1) *o++ = (uint8_t)(depth_p[p] | (p + 1 < n ? depth_p[p + 1] << 4 : 0));
    const uint32_t bm = diff_bitmap(codes_p, M, (uint32_t)p, parent_pos[p]);
    for (int b = 0; b < (M + 7) / 8; ++b) *o++ = (uint8_t)(bm >> (8 * b));
    for (int m = 0; m < M; ++m)
        if ((bm >> m) & 1u) *o++ = codes_p[(size_t)p * M + m];
}

}  // namespace

dpq_tree::~dpq_tree() { dpq::tree_release_device(this); }

namespace dpq {

void tree_release_device(dpq_tree* t) {
    if (!t->on_device) return;
    cudaSetDevice(t->device);
    for (void** p : {&t->d_codes_by_pos, &t->d_depth, &t->d_vec_id, &t->d_payload, &t->d_roff}) {
        if (*p) cudaFree(*p);
        *p = nullptr;
    }
    (void)cudaGetLastError();
}

// Depth-1 subtree shards of a device-resident tree, exactly as the stream reader deals them
// (program.cpp: a depth-1 node whose record starts at stream byte `off` goes to rank
// floor(off * n_ranks / n_bytes), and takes its subtree along): first[c] = the first depth-1 position
// dealt to rank c.
__global__ void shard_first_kernel(const uint8_t* __restrict__ depth, const unsigned long long* __restrict__ roff,
                                   int64_t n, int M, unsigned long long n_bytes, int n_ranks,
                                   unsigned int* __restrict__ first) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x + 1;
    if (p >= n || depth[p] != 1) return;
    const unsigned long long off = (unsigned long long)M + roff[p - 1];
    int c = (int)(off * (unsigned long long)n_ranks / n_bytes);
    if (c >= n_ranks) c = n_ranks - 1;
    atomicMin(&first[c], (unsigned int)p);
}

// bounds[r] .. bounds[r + 1] = the positions of shard r (rank 0 also holds the root at position 0);
// bytes[r] = stream bytes of the shard's records (+ M root bytes for rank 0)
int tree_shard_bounds(const dpq_tree* t, int n_ranks, std::vector<int64_t>* bounds, std::vector<int64_t>* bytes) {
    CU(cudaSetDevice(t->device));
    const int64_t n = t->n;
    Buf d_first;
    CU(d_first.alloc((size_t)n_ranks * 4));
    CU(cudaMemset(d_first.p, 0xFF, (size_t)n_ranks * 4));
    if (n > 1)
        shard_first_kernel<<<blocks(n - 1), 256>>>((const uint8_t*)t->d_depth, (const unsigned long long*)t->d_roff, n, t->M,
                                                   (unsigned long long)t->payload_bytes, n_ranks, d_first.as<unsigned int>());
    std::vector<unsigned int> first((size_t)n_ranks);
    CU(cudaMemcpy(first.data(), d_first.p, (size_t)n_ranks * 4, cudaMemcpyDeviceToHost));
    bounds->assign((size_t)n_ranks + 1, n);
    for (int r = n_ranks - 1; r >= 1; --r)
        (*bounds)[(size_t)r] = std::min<int64_t>((*bounds)[(size_t)r + 1], first[(size_t)r] == 0xFFFFFFFFu ? n : (int64_t)first[(size_t)r]);
    (*bounds)[0] = 0;
    bytes->assign((size_t)n_ranks, 0);
    auto off_of = [&](int64_t p, unsigned long long* o) -> int {  // stream offset of node p's record (p >= 1), or the end
        if (p >= n) {
            *o = (unsigned long long)t->payload_bytes;
            return DPQ_OK;
        }
        unsigned long long v = 0;
        CU(cudaMemcpy(&v, (const unsigned long long*)t->d_roff + (p - 1), 8, cudaMemcpyDeviceToHost));
        *o = v + (unsigned long long)t->M;
        return DPQ_OK;
    };
    for (int r = 0; r < n_ranks; ++r) {
        const int64_t lo = std::max<int64_t>((*bounds)[(size_t)r], 1), hi = (*bounds)[(size_t)r + 1];
        unsigned long long a = 0, b = 0;
        int rc;
        if (hi > lo) {
            if ((rc = off_of(lo, &a)) || (rc = off_of(hi, &b))) return rc;
        }
        (*bytes)[(size_t)r] = (int64_t)(b - a) + (r == 0 ? t->M : 0);
    }
    return DPQ_OK;
}

int depth_hist_device(int device, const uint8_t* d_depth, int64_t n, int64_t* hist17);

__global__ void code_range_kernel(const uint8_t* __restrict__ codes, int64_t bytes, int K, uint32_t* __restrict__ bad) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < bytes; i += stride)
        if (codes[i] >= K) *bad = 1u;
}

// every code byte must be a centroid id < K: a larger byte (foreign or corrupt codes file, -k mismatch)
// would index the K x K centroid tables and the ADC table rows out of bounds.  codes: host or device.
int check_code_range(const uint8_t* codes, int64_t n, int M, int K) {
    if (K >= 256) return DPQ_OK;
    const int64_t bytes = n * M;
    cudaPointerAttributes pa;
    const bool on_dev = cudaPointerGetAttributes(&pa, codes) == cudaSuccess && pa.type == cudaMemoryTypeDevice;
    (void)cudaGetLastError();
    bool bad = false;
    if (on_dev) {
        Buf d_bad;
        CU(d_bad.alloc(16));
        CU(cudaMemset(d_bad.p, 0, 16));
        code_range_kernel<<<1184, 256>>>(codes, bytes, K, d_bad.as<uint32_t>());
        uint32_t f = 0;
        CU(cudaMemcpy(&f, d_bad.p, 4, cudaMemcpyDeviceToHost));
        bad = f != 0;
    } else {
        for (int64_t i = 0; i < bytes && !bad; ++i) bad = codes[i] >= K;
    }
    if (bad) return api_fail(DPQ_ERR_ARG, "codes hold a centroid id >= K");
    return DPQ_OK;
}

// dpq_tree_copy of a device-resident tree: D2H of one of its arrays
int tree_copy_device(const dpq_tree* t, const void* src, void* dst, size_t bytes) {
    CU(cudaSetDevice(t->device));
    if (bytes) CU(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return DPQ_OK;
}

__global__ void depth_hist_kernel(const uint8_t* __restrict__ depth, int64_t n, unsigned long long* __restrict__ hist) {
    __shared__ unsigned int s[17];
    if (threadIdx.x < 17) s[threadIdx.x] = 0u;
    __syncthreads();
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) atomicAdd(&s[min((int)depth[i], 16)], 1u);
    __syncthreads();
    if (threadIdx.x < 17 && s[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (unsigned long long)s[threadIdx.x]);
}

int depth_hist_device(int device, const uint8_t* d_depth, int64_t n, int64_t* hist17) {
    CU(cudaSetDevice(device));
    Buf d_hist;
    CU(d_hist.alloc(17 * 8));
    CU(cudaMemset(d_hist.p, 0, 17 * 8));
    if (n > 0) depth_hist_kernel<<<592, 256>>>(d_depth, n, d_hist.as<unsigned long long>());
    unsigned long long hist[17];
    CU(cudaMemcpy(hist, d_hist.p, sizeof(hist), cudaMemcpyDeviceToHost));
    for (int i = 0; i < 17; ++i) hist17[i] = (int64_t)hist[i];
    return DPQ_OK;
}

int layout_tree_device(const uint8_t* codes, int64_t n, int M, int K, const float* cw, int Ds, dpq_tree* t,
                       const uint32_t* d_edges_in, bool keep_on_device, bool keep_qnode_fields) {
    int rc = api_check_device();
    if (rc) return rc;
    CU(cudaSetDevice(api_device()));
    const int64_t E = n - 1;
    const uint32_t root = t->root;
    if (root >= (uint64_t)n) return api_fail(DPQ_ERR_FORMAT, "dpq_tree: root id out of range");
    if (M > 16) return api_fail(DPQ_ERR_ARG, "dpq_tree: M <= 16");
    const int bmb = (M + 7) / 8;

    std::vector<float> T;
    centroid_tables(cw, M, K, Ds, T);

    Buf d_codes, d_T, d_edges, d_parent, d_nkids, d_first, d_far, d_farvia, d_depth, d_desc, d_err, d_tmp;
    Buf d_key, d_key2, d_kid, d_kid2, d_sz, d_pre, d_off, d_pos;
    CU(d_codes.alloc((size_t)n * M));
    CU(d_T.alloc(T.size() * 4));
    CU(d_edges.alloc((size_t)std::max<int64_t>(E, 1) * 8));
    CU(d_parent.alloc((size_t)n * 4));
    CU(d_nkids.alloc((size_t)(n + 1) * 4));
    CU(d_first.alloc((size_t)(n + 1) * 4));
    CU(d_far.alloc((size_t)n * 4));
    CU(d_farvia.alloc((size_t)n * 4));
    CU(d_depth.alloc((size_t)n));
    CU(d_desc.alloc((size_t)n * 4));
    CU(d_err.alloc(16));
    CU(cudaMemcpy(d_codes.p, codes, (size_t)n * M, cudaMemcpyDefault));
    CU(cudaMemcpy(d_T.p, T.data(), T.size() * 4, cudaMemcpyHostToDevice));
    if (E) CU(cudaMemcpy(d_edges.p, d_edges_in ? (const void*)d_edges_in : (const void*)t->edges.data(), (size_t)E * 8,
                         cudaMemcpyDefault));
    CU(cudaMemset(d_nkids.p, 0, (size_t)(n + 1) * 4));
    CU(cudaMemset(d_far.p, 0, (size_t)n * 4));
    CU(cudaMemset(d_farvia.p, 0, (size_t)n * 4));
    CU(cudaMemset(d_desc.p, 0, (size_t)n * 4));
    CU(cudaMemset(d_err.p, 0, 16));
    uint32_t* err = d_err.as<uint32_t>();
    uint32_t* parent = d_parent.as<uint32_t>();
    fill_kernel<<<blocks(n), 256>>>(parent, n, NONE);

    auto failed = [&](uint32_t* flags) -> int {
        *flags = 0;
        CU(cudaMemcpy(flags, err, 4, cudaMemcpyDeviceToHost));
        return DPQ_OK;
    };
    auto describe = [&](uint32_t f) -> int {
        if (f & ERR_RANGE) return api_fail(DPQ_ERR_FORMAT, "dpq_tree: edge endpoint out of range");
        if (f & ERR_TWO_PARENTS) return api_fail(DPQ_ERR_FORMAT, "dpq_tree: edges do not form a tree (a node has two parents)");
        if (f & ERR_NOT_SPANNING) return api_fail(DPQ_ERR_FORMAT, "dpq_tree: edges do not span all codes from the root");
        if (f & ERR_TOO_DEEP) return api_fail(DPQ_ERR_FORMAT, "dpq_tree: tree deeper than 255 levels (or a cycle)");
        if (f & ERR_NIBBLE) return api_fail(DPQ_ERR_FORMAT, "dpq_tree: tree too deep for the stream's depth nibble (depth <= 7 when M <= 8: the reader masks with &7, DCAT.h:3794; <= 15 otherwise)");
        return DPQ_OK;
    };
    uint32_t flags = 0;

    if (E) parent_kernel<<<blocks(E), 256>>>(d_edges.as<uint32_t>(), E, n, root, parent, d_nkids.as<uint32_t>(), err);
    if ((rc = failed(&flags))) return rc;
    if (flags) return describe(flags);

    // one temp buffer for the cub calls
    size_t tmp_bytes = 0, tb = 0;
    CU(d_key.alloc((size_t)std::max<int64_t>(E, 1) * 8));
    CU(d_key2.alloc((size_t)std::max<int64_t>(E, 1) * 8));
    CU(d_kid.alloc((size_t)std::max<int64_t>(E, 1) * 4));
    CU(d_kid2.alloc((size_t)std::max<int64_t>(E, 1) * 4));
    {
        cub::DoubleBuffer<unsigned long long> kb(d_key.as<unsigned long long>(), d_key2.as<unsigned long long>());
        cub::DoubleBuffer<uint32_t> vb(d_kid.as<uint32_t>(), d_kid2.as<uint32_t>());
        CU(cub::DeviceRadixSort::SortPairs(nullptr, tb, kb, vb, (int)std::max<int64_t>(E, 1), 0, 64));
        tmp_bytes = std::max(tmp_bytes, tb);
        CU(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_nkids.as<uint32_t>(), d_first.as<uint32_t>(), (int)(n + 1)));
        tmp_bytes = std::max(tmp_bytes, tb);
        CU(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_key.as<unsigned long long>(), d_key2.as<unsigned long long>(), (int)n));
        tmp_bytes = std::max(tmp_bytes, tb);
    }
    CU(d_tmp.alloc(tmp_bytes));

    tb = tmp_bytes;
    CU(cub::DeviceScan::ExclusiveSum(d_tmp.p, tb, d_nkids.as<uint32_t>(), d_first.as<uint32_t>(), (int)(n + 1)));
    far_kernel<<<blocks(n), 256>>>(d_codes.as<uint8_t>(), n, M, K, parent, d_T.as<float>(), d_far.as<uint32_t>(),
                                   d_farvia.as<uint32_t>());
    climb_kernel<<<blocks(n), 256>>>(n, root, parent, d_depth.as<uint8_t>(), d_desc.as<uint32_t>(), err);
    if ((rc = failed(&flags))) return rc;
    if (flags) return describe(flags);

    CU(d_off.alloc((size_t)n * 4));
    CU(d_pos.alloc((size_t)n * 4));
    CU(cudaMemset(d_off.p, 0, (size_t)n * 4));
    if (E) {
        kidkey_kernel<<<blocks(E), 256>>>(d_edges.as<uint32_t>(), E, d_farvia.as<uint32_t>(),
                                          d_key.as<unsigned long long>(), d_kid.as<uint32_t>());
        cub::DoubleBuffer<unsigned long long> kb(d_key.as<unsigned long long>(), d_key2.as<unsigned long long>());
        cub::DoubleBuffer<uint32_t> vb(d_kid.as<uint32_t>(), d_kid2.as<uint32_t>());
        tb = tmp_bytes;
        CU(cub::DeviceRadixSort::SortPairs(d_tmp.p, tb, kb, vb, (int)E, 0, 64));
        const uint32_t* kid = vb.Current();
        // the key buffers are free again: subtree sizes and their exclusive sum live there
        unsigned long long* sz = kb.Current();
        unsigned long long* pre = kb.Alternate();
        kidsize_kernel<<<blocks(E), 256>>>(kid, E, d_desc.as<uint32_t>(), sz);
        tb = tmp_bytes;
        CU(cub::DeviceScan::ExclusiveSum(d_tmp.p, tb, sz, pre, (int)E));
        kidoff_kernel<<<blocks(E), 256>>>(kid, E, parent, d_first.as<uint32_t>(), pre, d_off.as<uint32_t>());
    }
    pos_kernel<<<blocks(n), 256>>>(n, root, parent, d_off.as<uint32_t>(), d_pos.as<uint32_t>());
    CU(cudaGetLastError());
    d_kid.release();
    d_kid2.release();
    d_edges.release();
    d_nkids.release();
    d_first.release();

    Buf d_vec, d_ppos, d_cnum, d_depthp, d_md, d_md2, d_codesp;
    CU(d_vec.alloc((size_t)n * 4));
    CU(d_ppos.alloc((size_t)n * 4));
    CU(d_cnum.alloc((size_t)n * 4));
    CU(d_depthp.alloc((size_t)n));
    CU(d_md.alloc((size_t)n * 4));
    CU(d_md2.alloc((size_t)n * 4));
    CU(d_codesp.alloc((size_t)n * M));
    emit_kernel<<<blocks(n), 256>>>(n, M, root, d_codes.as<uint8_t>(), parent, d_pos.as<uint32_t>(),
                                    d_desc.as<uint32_t>(), d_depth.as<uint8_t>(), d_far.as<uint32_t>(),
                                    d_farvia.as<uint32_t>(), d_vec.as<uint32_t>(), d_ppos.as<uint32_t>(),
                                    d_cnum.as<uint32_t>(), d_depthp.as<uint8_t>(), d_md.as<float>(),
                                    d_md2.as<float>(), d_codesp.as<uint8_t>(), err);
    // stream: record lengths -> byte offsets -> every node writes its record
    unsigned long long* len = d_key.as<unsigned long long>();
    unsigned long long* roff = d_key2.as<unsigned long long>();
    unsigned long long total = (unsigned long long)M;
    if (E) {
        reclen_kernel<<<blocks(E), 256>>>(n, M, d_codesp.as<uint8_t>(), d_ppos.as<uint32_t>(), d_depthp.as<uint8_t>(),
                                          len, err);
        tb = tmp_bytes;
        CU(cub::DeviceScan::ExclusiveSum(d_tmp.p, tb, len, roff, (int)E));
        unsigned long long last_off = 0, last_len = 0;
        CU(cudaMemcpy(&last_off, roff + (E - 1), 8, cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(&last_len, len + (E - 1), 8, cudaMemcpyDeviceToHost));
        total += last_off + last_len;
    }
    if ((rc = failed(&flags))) return rc;
    if (flags) return describe(flags);
    t->n_diffs = (int64_t)total - M - (int64_t)bmb * E - n / 2;  // M = 8: total = 8 + n_diffs + (3(n-1)+1)/2
    Buf d_out;
    CU(d_out.alloc((size_t)total));
    stream_kernel<<<blocks(n), 256>>>(n, M, d_codesp.as<uint8_t>(), d_ppos.as<uint32_t>(), d_depthp.as<uint8_t>(), roff,
                                      d_out.as<uint8_t>());
    CU(cudaGetLastError());
    if (keep_on_device) {  // hand the buffers the index needs to the tree object; nothing crosses PCIe
        int64_t hist[17];
        if ((rc = depth_hist_device(api_device(), d_depthp.as<uint8_t>(), n, hist))) return rc;
        t->depth_hist.assign(hist, hist + 17);
        if (keep_qnode_fields) {  // what the QNode records need beyond the device arrays
            t->parent_pos.resize((size_t)n);
            t->child_num.resize((size_t)n);
            t->max_dist.resize((size_t)n);
            t->max_dist2p.resize((size_t)n);
            CU(cudaMemcpy(t->parent_pos.data(), d_ppos.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(t->child_num.data(), d_cnum.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(t->max_dist.data(), d_md.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
            CU(cudaMemcpy(t->max_dist2p.data(), d_md2.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
        }
        CU(cudaDeviceSynchronize());
        t->on_device = true;
        t->device = api_device();
        t->payload_bytes = (int64_t)total;
        t->d_codes_by_pos = d_codesp.p;
        t->d_depth = d_depthp.p;
        t->d_vec_id = d_vec.p;
        t->d_payload = d_out.p;
        t->d_roff = d_key2.p;
        d_codesp.p = d_depthp.p = d_vec.p = d_out.p = d_key2.p = nullptr;
        return DPQ_OK;
    }

    t->vec_id.resize((size_t)n);
    t->parent_pos.resize((size_t)n);
    t->child_num.resize((size_t)n);
    t->depth.resize((size_t)n);
    t->max_dist.resize((size_t)n);
    t->max_dist2p.resize((size_t)n);
    t->codes_by_pos.resize((size_t)n * M);
    t->payload.resize((size_t)total);
    CU(cudaMemcpy(t->vec_id.data(), d_vec.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t->parent_pos.data(), d_ppos.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t->child_num.data(), d_cnum.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t->depth.data(), d_depthp.p, (size_t)n, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t->max_dist.data(), d_md.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t->max_dist2p.data(), d_md2.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t->codes_by_pos.data(), d_codesp.p, (size_t)n * M, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(t->payload.data(), d_out.p, (size_t)total, cudaMemcpyDeviceToHost));
    return DPQ_OK;
}

}  // namespace dpq
