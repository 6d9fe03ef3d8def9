// Multi-GPU search behind the C ABI (include/dpq.h: dpq_multi_*): one process, one host thread,
// one DeltaTree shard per GPU (whole depth-1 subtrees, SURVEY 8e), local top-k on every GPU,
// ONE collective -- an NCCL all-gather of the Q x k result keys over NVLink -- and a k-way merge
// kernel.  This is what the drop-in `deltapq -task query -gpus N` uses; bench.py does the same
// with torch.distributed as the NCCL plumbing.
//
// NCCL is bound at run time (dlopen "libnccl.so.2"), so libdpq.so has no link-time dependency on
// it and single-GPU users never load it.
#include <cuda_runtime.h>

#include <chrono>
#include <dlfcn.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/dpq.h"

namespace dpq {
int api_fail(int code, const std::string& msg);
int api_check_device();
int index_live_nodes(dpq_index* ix, uint8_t** d_codes, uint32_t** d_ids, int64_t* n_live);  // api.cu
void index_take_ids(dpq_index* ix, std::vector<uint32_t>* ids);
}

namespace {

// the slice of nccl.h this file needs (ABI-stable since NCCL 2.x)
typedef struct ncclComm* ncclComm_t;
typedef int ncclResult_t;  // 0 = ncclSuccess
constexpr int kNcclUint64 = 5;  // ncclUint64 in ncclDataType_t
struct Nccl {
    void* lib = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string load() {
        if (lib) return std::string();
        // DPQ_NCCL_LIB names a specific library (e.g. the copy a framework already ships); else the system one
        const char* env = getenv("DPQ_NCCL_LIB");
        if (env && env[0]) lib = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            if (lib) break;
            lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
        }
        if (!lib) return std::string("cannot load libnccl.so.2: ") + dlerror();
#define DPQ_SYM(field, sym)                                                  \
    field = reinterpret_cast<decltype(field)>(dlsym(lib, sym));              \
    if (!field) return std::string("libnccl lacks ") + sym;
        DPQ_SYM(CommInitAll, "ncclCommInitAll")
        DPQ_SYM(CommDestroy, "ncclCommDestroy")
        DPQ_SYM(AllGather, "ncclAllGather")
        DPQ_SYM(GroupStart, "ncclGroupStart")
        DPQ_SYM(GroupEnd, "ncclGroupEnd")
        DPQ_SYM(GetErrorString, "ncclGetErrorString")
#undef DPQ_SYM
        return std::string();
    }
};
Nccl g_nccl;

}  // namespace

struct dpq_multi {
    int n = 0, M = 0, K = 0, Ds = 0;  // n = GPUs
    std::vector<dpq_index*> ix;          // every shard (one per GPU) or forest part (dealt round-robin)
    std::vector<int> dev;                // device of ix[i]
    std::vector<std::vector<int>> on;    // indexes living on each device
    std::vector<cudaStream_t> st;        // one stream per device, shared by its indexes
    std::vector<ncclComm_t> comm;
    std::vector<void*> d_q, d_loc, d_one, d_all;  // per device: queries, per-index lists, their merge, gathered lists
    void* d_out = nullptr;  // device 0
    size_t q_cap = 0, k_cap = 0;
    void* h_stage = nullptr;
    size_t h_cap = 0;
    std::vector<uint32_t> pos2id;  // position -> vector id over the whole position space
    size_t last = 0;               // the index whose positions end the position space: it takes every add
    bool forest = false;           // dpq_multi_open_parts: ix are forest parts, else subtree shards of one tree
    std::vector<float> cw;         // the codebook: dpq_multi_compact builds a tree with it
    int64_t open_us = 0, nccl_us = 0;  // wall time of opening the shards / of ncclCommInitAll
};

#define CUM(call)                                                                                   \
    do {                                                                                            \
        cudaError_t e_ = (call);                                                                    \
        if (e_ != cudaSuccess)                                                                      \
            return dpq::api_fail(DPQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)
#define NCM(call)                                                                                        \
    do {                                                                                                 \
        ncclResult_t r_ = (call);                                                                        \
        if (r_ != 0) return dpq::api_fail(DPQ_ERR_CUDA, std::string(#call) + ": " + g_nccl.GetErrorString(r_)); \
    } while (0)

namespace {

// vec_id of every position from the 60-byte QNode records (DCAT.h:79-101), plus `add`
bool read_vec_ids(const char* path, size_t n, uint32_t* dst, uint32_t add, std::string* err) {
    FILE* f = fopen(path, "rb");
    if (!f) {
        *err = std::string("cannot open ") + path;
        return false;
    }
    std::vector<uint8_t> rec(60 * 4096);
    size_t done = 0;
    bool ok = true;
    while (ok && done < n) {
        const size_t want = std::min<size_t>(4096, n - done);
        ok = fread(rec.data(), 60, want, f) == want;
        for (size_t i = 0; ok && i < want; ++i) {
            uint32_t v;
            memcpy(&v, rec.data() + 60 * i, 4);
            dst[done + i] = v + add;
        }
        done += want;
    }
    fclose(f);
    if (!ok) *err = "QNode file truncated";
    return ok;
}

// streams, NCCL communicators: after every index is open
int finish_multi_open(dpq_multi* m) {
    const int n_gpus = m->n;
    m->st.assign((size_t)n_gpus, nullptr);
    m->d_q.assign((size_t)n_gpus, nullptr);
    m->d_loc.assign((size_t)n_gpus, nullptr);
    m->d_one.assign((size_t)n_gpus, nullptr);
    m->d_all.assign((size_t)n_gpus, nullptr);
    for (int r = 0; r < n_gpus; ++r) {
        CUM(cudaSetDevice(r));
        CUM(cudaStreamCreateWithFlags(&m->st[(size_t)r], cudaStreamNonBlocking));
        for (int i : m->on[(size_t)r]) {
            int rc = dpq_index_set_stream(m->ix[(size_t)i], m->st[(size_t)r]);
            if (rc) return rc;
        }
    }
    dpq_set_device(0);
    if (n_gpus > 1) {
        m->comm.assign((size_t)n_gpus, nullptr);
        std::vector<int> devs((size_t)n_gpus);
        for (int r = 0; r < n_gpus; ++r) devs[(size_t)r] = r;
        const auto t0 = std::chrono::steady_clock::now();
        ncclResult_t r_ = g_nccl.CommInitAll(m->comm.data(), n_gpus, devs.data());
        m->nccl_us = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
        if (r_ != 0) {
            m->comm.clear();
            return dpq::api_fail(DPQ_ERR_CUDA, std::string("ncclCommInitAll: ") + g_nccl.GetErrorString(r_));
        }
    }
    return DPQ_OK;
}

int begin_multi_open(int n_gpus, int n_index, int M, int K, dpq_multi** out) {
    if (n_gpus > dpq_device_count())
        return dpq::api_fail(DPQ_ERR_CUDA, "dpq_multi_open: fewer CUDA devices than -gpus");
    if (n_gpus > 1) {
        std::string err = g_nccl.load();
        if (!err.empty()) return dpq::api_fail(DPQ_ERR_CUDA, err);
    }
    dpq_multi* m = new dpq_multi();
    m->n = n_gpus;
    m->M = M;
    m->K = K;
    m->ix.assign((size_t)n_index, nullptr);
    m->dev.assign((size_t)n_index, 0);
    m->on.assign((size_t)n_gpus, std::vector<int>());
    *out = m;
    return DPQ_OK;
}

}  // namespace

extern "C" {

int dpq_multi_open_file(const char* tree_path, const char* qnode_path, int M, int K, int n_gpus, dpq_multi** out) {
    if (!tree_path || !out || n_gpus < 1) return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_open_file: bad argument");
    *out = nullptr;
    dpq_multi* m = nullptr;
    int rc = begin_multi_open(n_gpus, n_gpus, M, K, &m);
    if (rc) return rc;
    const auto t_open0 = std::chrono::steady_clock::now();
    {
        // one host thread per shard: the stream decode is sequential (seconds per 10^8 nodes), the
        // shards are independent and the device selection is per thread, so the open takes one decode
        // time instead of n_gpus of them
        for (int r = 0; r < n_gpus; ++r) {
            m->dev[(size_t)r] = r;
            m->on[(size_t)r].push_back(r);
        }
        std::vector<int> rcs((size_t)n_gpus, 0);
        std::vector<std::string> errs((size_t)n_gpus);
        auto worker = [&](int r) {
            int r_ = dpq_set_device(r);
            if (!r_) r_ = dpq_index_open_file(tree_path, nullptr, M, K, r, n_gpus, &m->ix[(size_t)r]);
            rcs[(size_t)r] = r_;
            if (r_) errs[(size_t)r] = dpq_last_error();  // thread-local text: carry it to the caller's thread
        };
        std::vector<std::thread> th;
        for (int r = 1; r < n_gpus; ++r) th.emplace_back(worker, r);
        worker(0);
        for (auto& t : th) t.join();
        for (int r = 0; r < n_gpus && !rc; ++r)
            if (rcs[(size_t)r]) rc = dpq::api_fail(rcs[(size_t)r], errs[(size_t)r]);
    }
    m->open_us = std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t_open0).count();
    m->last = (size_t)n_gpus - 1;
    if (!rc) rc = finish_multi_open(m);
    if (!rc && qnode_path) {
        const int64_t n_codes = dpq_index_stat(m->ix[0], "n_codes");
        m->pos2id.resize((size_t)n_codes);
        std::string err;
        if (!read_vec_ids(qnode_path, m->pos2id.size(), m->pos2id.data(), 0u, &err)) rc = dpq::api_fail(DPQ_ERR_IO, err);
    }
    if (rc) {
        std::string keep = dpq_last_error();
        dpq_multi_close(m);
        return dpq::api_fail(rc, keep);
    }
    *out = m;
    return DPQ_OK;
}

int dpq_multi_open_parts(const char* const* tree_paths, const char* const* qnode_paths, const int64_t* first_pos,
                         int n_parts, int M, int K, int n_gpus, dpq_multi** out) {
    if (!tree_paths || !first_pos || !out || n_parts < 1 || n_gpus < 1)
        return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_open_parts: bad argument");
    *out = nullptr;
    if (n_gpus > n_parts) n_gpus = n_parts;
    dpq_multi* m = nullptr;
    int rc = begin_multi_open(n_gpus, n_parts, M, K, &m);
    if (rc) return rc;
    m->forest = true;
    int64_t span = 0;
    {
        // parts are dealt round-robin to the GPUs and opened concurrently: the host decode of a stream is
        // sequential (seconds per 10^8 nodes), the parts are independent, the device selection is per thread
        for (int p = 0; p < n_parts; ++p) {
            m->dev[(size_t)p] = p % n_gpus;
            m->on[(size_t)(p % n_gpus)].push_back(p);
        }
        std::vector<int> rcs((size_t)n_parts, 0);
        std::vector<std::string> errs((size_t)n_parts);
        const int n_threads = std::max(1, std::min(n_parts, (int)std::thread::hardware_concurrency()));
        auto worker = [&](int t) {
            for (int p = t; p < n_parts; p += n_threads) {
                int r_ = dpq_set_device(m->dev[(size_t)p]);
                if (!r_) r_ = dpq_index_open_part_file(tree_paths[p], nullptr, M, K, first_pos[p], &m->ix[(size_t)p]);
                rcs[(size_t)p] = r_;
                if (r_) errs[(size_t)p] = dpq_last_error();  // thread-local text: carry it to the caller's thread
            }
        };
        std::vector<std::thread> th;
        for (int t = 1; t < n_threads; ++t) th.emplace_back(worker, t);
        worker(0);
        for (auto& t : th) t.join();
        for (int p = 0; p < n_parts && !rc; ++p)
            if (rcs[(size_t)p]) rc = dpq::api_fail(rcs[(size_t)p], errs[(size_t)p]);
        for (int p = 0; p < n_parts && !rc; ++p)
            span = std::max<int64_t>(span, first_pos[p] + dpq_index_stat(m->ix[(size_t)p], "n_codes"));
        for (int p = 0; p < n_parts; ++p)
            if (first_pos[p] >= first_pos[m->last]) m->last = (size_t)p;
    }
    if (!rc) rc = finish_multi_open(m);
    if (!rc && qnode_paths) {  // ids of part p = first_pos[p] + its own vec_id (parts are id ranges)
        m->pos2id.resize((size_t)span);
        for (size_t i = 0; i < m->pos2id.size(); ++i) m->pos2id[i] = (uint32_t)i;
        for (int p = 0; p < n_parts && !rc; ++p) {
            if (!qnode_paths[p]) continue;
            std::string err;
            const int64_t np = dpq_index_stat(m->ix[(size_t)p], "n_codes");
            if (!read_vec_ids(qnode_paths[p], (size_t)np, m->pos2id.data() + first_pos[p], (uint32_t)first_pos[p], &err))
                rc = dpq::api_fail(DPQ_ERR_IO, err);
        }
    }
    if (rc) {
        std::string keep = dpq_last_error();
        dpq_multi_close(m);
        return dpq::api_fail(rc, keep);
    }
    *out = m;
    return DPQ_OK;
}

int dpq_multi_set_codebook(dpq_multi* m, const float* codewords, int Ds) {
    if (!m || !codewords) return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_set_codebook: null");
    m->Ds = Ds;
    m->cw.assign(codewords, codewords + (size_t)m->M * m->K * Ds);
    for (size_t i = 0; i < m->ix.size(); ++i) {
        CUM(cudaSetDevice(m->dev[i]));
        int rc = dpq_index_set_codebook(m->ix[i], codewords, Ds);
        if (rc) return rc;
    }
    CUM(cudaSetDevice(0));
    return DPQ_OK;
}

int dpq_multi_search(dpq_multi* m, const float* queries, int Q, int topk, uint32_t* out_pos, uint32_t* out_id,
                     float* out_dist) {
    if (!m || !queries || Q < 1 || topk < 1) return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_search: bad argument");
    if (m->Ds < 1) return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_search: codebook not set");
    constexpr int kMaxBatch = 32768;  // bounds the per-index scratch (float tables: 8 KB per query at M = 8), as dpq_index_search
    if (Q > kMaxBatch) {
        const size_t D = (size_t)m->M * m->Ds;
        for (int q0 = 0; q0 < Q; q0 += kMaxBatch) {
            const int nq = std::min(kMaxBatch, Q - q0);
            const size_t o = (size_t)q0 * topk;
            int rc = dpq_multi_search(m, queries + (size_t)q0 * D, nq, topk, out_pos ? out_pos + o : nullptr,
                                      out_id ? out_id + o : nullptr, out_dist ? out_dist + o : nullptr);
            if (rc) return rc;
        }
        return DPQ_OK;
    }
    const size_t qbytes = (size_t)Q * m->M * m->Ds * 4, kbytes = (size_t)Q * topk * 8;
    if (m->h_cap < qbytes + kbytes) {
        if (m->h_stage) cudaFreeHost(m->h_stage);
        m->h_stage = nullptr;
        CUM(cudaMallocHost(&m->h_stage, qbytes + kbytes));
        m->h_cap = qbytes + kbytes;
    }
    if (m->q_cap < qbytes || m->k_cap < kbytes) {
        for (int r = 0; r < m->n; ++r) {
            CUM(cudaSetDevice(r));
            for (void** p : {&m->d_q[(size_t)r], &m->d_loc[(size_t)r], &m->d_one[(size_t)r], &m->d_all[(size_t)r]})
                if (*p) {
                    cudaFree(*p);
                    *p = nullptr;
                }
            CUM(cudaMalloc(&m->d_q[(size_t)r], qbytes));
            CUM(cudaMalloc(&m->d_loc[(size_t)r], kbytes * std::max<size_t>(m->on[(size_t)r].size(), 1)));
            CUM(cudaMalloc(&m->d_one[(size_t)r], kbytes));
            CUM(cudaMalloc(&m->d_all[(size_t)r], kbytes * (size_t)m->n));
        }
        CUM(cudaSetDevice(0));
        if (m->d_out) cudaFree(m->d_out);
        CUM(cudaMalloc(&m->d_out, kbytes));
        m->q_cap = qbytes;
        m->k_cap = kbytes;
    }
    float* hq = reinterpret_cast<float*>(m->h_stage);
    uint64_t* hk = reinterpret_cast<uint64_t*>(reinterpret_cast<char*>(m->h_stage) + qbytes);
    memcpy(hq, queries, qbytes);
    // every GPU: queries in, local top-k (global positions) of each of its shards / parts, merged
    // into one list per GPU
    std::vector<const void*> mine((size_t)m->n, nullptr);
    for (int r = 0; r < m->n; ++r) {
        CUM(cudaSetDevice(r));
        CUM(cudaMemcpyAsync(m->d_q[(size_t)r], hq, qbytes, cudaMemcpyHostToDevice, m->st[(size_t)r]));
        const std::vector<int>& on = m->on[(size_t)r];
        for (size_t j = 0; j < on.size(); ++j) {
            int rc = dpq_index_search_device(m->ix[(size_t)on[j]], reinterpret_cast<const float*>(m->d_q[(size_t)r]), Q, topk,
                                             reinterpret_cast<uint64_t*>(reinterpret_cast<char*>(m->d_loc[(size_t)r]) + j * kbytes));
            if (rc) return rc;
        }
        mine[(size_t)r] = m->d_loc[(size_t)r];
        if (on.size() > 1) {
            int rc = dpq_merge_topk_device(m->ix[(size_t)on[0]], reinterpret_cast<const uint64_t*>(m->d_loc[(size_t)r]),
                                           (int)on.size(), Q, topk, reinterpret_cast<uint64_t*>(m->d_one[(size_t)r]));
            if (rc) return rc;
            mine[(size_t)r] = m->d_one[(size_t)r];
        }
    }
    const void* merged = mine[0];
    if (m->n > 1) {  // the only collective: all-gather of the key lists, then the k-way merge
        NCM(g_nccl.GroupStart());
        for (int r = 0; r < m->n; ++r)
            NCM(g_nccl.AllGather(mine[(size_t)r], m->d_all[(size_t)r], (size_t)Q * topk, kNcclUint64,
                                 m->comm[(size_t)r], m->st[(size_t)r]));
        NCM(g_nccl.GroupEnd());
        CUM(cudaSetDevice(0));
        int rc = dpq_merge_topk_device(m->ix[(size_t)m->on[0][0]], reinterpret_cast<const uint64_t*>(m->d_all[0]), m->n, Q,
                                       topk, reinterpret_cast<uint64_t*>(m->d_out));
        if (rc) return rc;
        merged = m->d_out;
    }
    CUM(cudaSetDevice(0));
    CUM(cudaMemcpyAsync(hk, merged, kbytes, cudaMemcpyDeviceToHost, m->st[0]));
    for (size_t i = 0; i < m->ix.size(); ++i) {
        CUM(cudaSetDevice(m->dev[i]));
        int rc = dpq_index_sync(m->ix[i]);  // stream sync + fallback overflow check
        if (rc) return rc;
    }
    CUM(cudaSetDevice(0));
    for (size_t i = 0; i < (size_t)Q * topk; ++i) {
        const uint32_t pos = (uint32_t)hk[i];
        const uint32_t bits = (uint32_t)(hk[i] >> 32);
        if (out_pos) out_pos[i] = pos;
        if (out_dist) memcpy(&out_dist[i], &bits, 4);
        if (out_id) out_id[i] = (pos < m->pos2id.size()) ? m->pos2id[pos] : pos;
    }
    return DPQ_OK;
}

// Shard and part indexes are opened without pos2id, so they take global positions: the ids are translated with
// the QNode table first (when there is one), then every index is given the same position list and keeps its own.
static int multi_mark_dead(dpq_multi* m, const uint32_t* ids, int64_t n, bool set, const char* what) {
    int rc = dpq::api_check_device();
    if (rc) return rc;
    if (!m) return dpq::api_fail(DPQ_ERR_ARG, std::string(what) + ": null handle");
    if (n < 0 || (n > 0 && !ids)) return dpq::api_fail(DPQ_ERR_ARG, std::string(what) + ": ids is null or n < 0");
    if (n == 0) return DPQ_OK;
    std::vector<uint32_t> pos;
    const uint32_t* list = ids;
    if (!m->pos2id.empty()) {
        std::vector<uint32_t> sorted(ids, ids + n);
        std::sort(sorted.begin(), sorted.end());
        for (size_t p = 0; p < m->pos2id.size(); ++p)
            if (std::binary_search(sorted.begin(), sorted.end(), m->pos2id[p])) pos.push_back((uint32_t)p);
        list = pos.data();
        n = (int64_t)pos.size();
    }
    for (size_t i = 0; i < m->ix.size(); ++i) {
        CUM(cudaSetDevice(m->dev[i]));
        rc = set ? dpq_index_delete(m->ix[i], list, n) : dpq_index_undelete(m->ix[i], list, n);
        if (rc) return rc;
    }
    CUM(cudaSetDevice(0));
    return DPQ_OK;
}

int dpq_multi_delete(dpq_multi* m, const uint32_t* ids, int64_t n) { return multi_mark_dead(m, ids, n, true, "dpq_multi_delete"); }
int dpq_multi_undelete(dpq_multi* m, const uint32_t* ids, int64_t n) {
    return multi_mark_dead(m, ids, n, false, "dpq_multi_undelete");
}

// The index that ends the position space takes the batch with ids = its positions (shard and part indexes have no
// id table); the handle's own table maps those positions to the caller's ids.
// D = 0: data are codes; else vectors of D floats.
static int multi_add(dpq_multi* m, const void* data, int64_t n, int D, const uint32_t* ids, uint32_t* out_pos, const char* what) {
    int rc = dpq::api_check_device();
    if (rc) return rc;
    if (!m) return dpq::api_fail(DPQ_ERR_ARG, std::string(what) + ": null handle");
    if (n < 0 || (n > 0 && !data)) return dpq::api_fail(DPQ_ERR_ARG, std::string(what) + ": input is null or n < 0");
    if (n > 0x7FFFFFFFLL) return dpq::api_fail(DPQ_ERR_ARG, std::string(what) + ": more than 2^31 - 1 rows in one call");
    if (D < 0) return dpq::api_fail(DPQ_ERR_ARG, std::string(what) + ": D must be >= 1");
    if (n == 0) return DPQ_OK;
    dpq_index* ix = m->ix[m->last];
    std::vector<uint32_t> pos((size_t)n), hid;
    if (ids) {  // host or device pointer
        hid.resize((size_t)n);
        CUM(cudaMemcpy(hid.data(), ids, (size_t)n * 4, cudaMemcpyDefault));
    }
    CUM(cudaSetDevice(m->dev[m->last]));
    rc = D ? dpq_index_add_vectors(ix, static_cast<const float*>(data), n, D, nullptr, pos.data())
           : dpq_index_add(ix, static_cast<const uint8_t*>(data), n, nullptr, pos.data());
    if (rc) return rc;
    if (ids || !m->pos2id.empty()) {
        const size_t end = (size_t)*std::max_element(pos.begin(), pos.end()) + 1, old = m->pos2id.size();
        if (end > old) {
            m->pos2id.resize(end);
            for (size_t p = old; p < end; ++p) m->pos2id[p] = (uint32_t)p;
        }
        for (size_t j = 0; j < pos.size(); ++j) m->pos2id[pos[j]] = ids ? hid[j] : pos[j];
    }
    if (out_pos) CUM(cudaMemcpy(out_pos, pos.data(), (size_t)n * 4, cudaMemcpyDefault));
    CUM(cudaSetDevice(0));
    return DPQ_OK;
}

int dpq_multi_add(dpq_multi* m, const uint8_t* codes, int64_t n, const uint32_t* ids, uint32_t* out_pos) {
    return multi_add(m, codes, n, 0, ids, out_pos, "dpq_multi_add");
}
int dpq_multi_add_vectors(dpq_multi* m, const float* x, int64_t n, int D, const uint32_t* ids, uint32_t* out_pos) {
    return multi_add(m, x, n, D < 1 ? -1 : D, ids, out_pos, "dpq_multi_add_vectors");
}

// The handle reports ids through its table, indexed by global position; a position it does not cover is its own id.
static uint32_t id_of(const std::vector<uint32_t>& tab, uint32_t pos) { return pos < tab.size() ? tab[pos] : pos; }

// Forest parts: each part is compacted in place on its GPU (dpq_index_compact keeps first_pos); the ids it carries
// are the global positions the handle knew, translated through the old table into the new one part by part, so a
// failure in a later part leaves a consistent handle.
static int compact_parts(dpq_multi* m) {
    int64_t span = 0;
    for (size_t p = 0; p < m->ix.size(); ++p) {
        const int64_t live = dpq_index_stat(m->ix[p], "n_local") - dpq_index_stat(m->ix[p], "n_deleted");
        if (live < 1) return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_compact: part " + std::to_string(p) + " has no live node");
        span = std::max(span, dpq_index_stat(m->ix[p], "base_pos") + dpq_index_stat(m->ix[p], "n_local"));
    }
    const std::vector<uint32_t> old = m->pos2id;
    if (m->pos2id.size() < (size_t)span) {
        const size_t from = m->pos2id.size();
        m->pos2id.resize((size_t)span);
        for (size_t i = from; i < m->pos2id.size(); ++i) m->pos2id[i] = (uint32_t)i;
    }
    for (size_t p = 0; p < m->ix.size(); ++p) {
        dpq_index* ix = m->ix[p];
        const int64_t first = dpq_index_stat(ix, "base_pos"), n_old = dpq_index_stat(ix, "n_local");
        CUM(cudaSetDevice(m->dev[p]));
        int rc = dpq_index_compact(ix, nullptr);
        if (rc) return rc;
        std::vector<uint32_t> ids;
        dpq::index_take_ids(ix, &ids);
        for (size_t i = 0; i < ids.size(); ++i) m->pos2id[(size_t)first + i] = id_of(old, ids[i]);
        for (int64_t q = first + (int64_t)ids.size(); q < first + n_old; ++q) m->pos2id[(size_t)q] = (uint32_t)q;  // no node
    }
    CUM(cudaSetDevice(0));
    return DPQ_OK;
}

// Subtree shards: every shard's live codes and positions are gathered on its GPU, copied in rank order (= global
// position order) to GPU 0, built into one tree there, and its stream is dealt to the GPUs again as
// dpq_multi_open_file deals a file.  The new shards replace the old ones only once all of them are open.
static int compact_shards(dpq_multi* m) {
    const size_t n = m->ix.size();
    std::vector<uint8_t*> codes(n, nullptr);
    std::vector<uint32_t*> pos(n, nullptr);
    std::vector<int64_t> cnt(n, 0);
    std::vector<dpq_index*> fresh(n, nullptr);
    uint8_t* all_codes = nullptr;
    uint32_t* all_pos = nullptr;
    dpq_tree* t = nullptr;
    auto cleanup = [&](int rc) {
        for (size_t r = 0; r < n; ++r) {
            cudaSetDevice(m->dev[r]);
            if (codes[r]) cudaFree(codes[r]);
            if (pos[r]) cudaFree(pos[r]);
            if (fresh[r]) dpq_index_close(fresh[r]);
        }
        cudaSetDevice(0);
        if (all_codes) cudaFree(all_codes);
        if (all_pos) cudaFree(all_pos);
        dpq_tree_free(t);
        (void)cudaGetLastError();
        dpq_set_device(0);
        return rc;
    };
    const std::string keep_err = "dpq_multi_compact: ";
    auto cuda_fail = [&](cudaError_t e) { return cleanup(dpq::api_fail(DPQ_ERR_CUDA, keep_err + cudaGetErrorString(e))); };
    int64_t total = 0;
    for (size_t r = 0; r < n; ++r) {
        int rc = dpq::index_live_nodes(m->ix[r], &codes[r], &pos[r], &cnt[r]);  // shards have no id table: ids = positions
        if (rc) return cleanup(rc);
        total += cnt[r];
    }
    if (total == 0) return cleanup(dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_compact: every node is deleted (a tree needs at least one node)"));
    const int M = m->M, K = m->K;
    int rc = dpq_set_device(0);
    if (rc) return cleanup(rc);
    cudaError_t e = cudaMalloc(&all_codes, (size_t)total * M);
    if (e == cudaSuccess) e = cudaMalloc(&all_pos, (size_t)total * 4);
    for (size_t r = 0, off = 0; r < n && e == cudaSuccess; off += (size_t)cnt[r], ++r) {
        if (!cnt[r]) continue;  // another GPU's memory: peer or host-staged copies, whatever the platform has
        e = cudaMemcpyAsync(all_codes + off * M, codes[r], (size_t)cnt[r] * M, cudaMemcpyDefault, m->st[0]);
        if (e == cudaSuccess) e = cudaMemcpyAsync(all_pos + off, pos[r], (size_t)cnt[r] * 4, cudaMemcpyDefault, m->st[0]);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(m->st[0]);
    if (e != cudaSuccess) return cuda_fail(e);
    if ((rc = dpq_tree_build_device(all_codes, total, M, K, m->cw.data(), m->Ds, 1, 1, &t))) return cleanup(rc);
    std::vector<uint8_t> payload((size_t)dpq_tree_size(t, "payload"));
    std::vector<uint32_t> row((size_t)total), old_pos((size_t)total);
    if ((rc = dpq_tree_copy(t, "payload", payload.data())) || (rc = dpq_tree_copy(t, "vec_id", row.data()))) return cleanup(rc);
    if ((e = cudaMemcpy(old_pos.data(), all_pos, (size_t)total * 4, cudaMemcpyDeviceToHost)) != cudaSuccess) return cuda_fail(e);
    std::vector<uint32_t> tab((size_t)total);
    for (size_t p = 0; p < tab.size(); ++p) tab[p] = id_of(m->pos2id, old_pos[row[p]]);
    for (size_t r = 0; r < n; ++r) {
        if ((rc = dpq_set_device(m->dev[r])) ||
            (rc = dpq_index_open(payload.data(), (int64_t)payload.size(), total, M, K, nullptr, (int)r, (int)n, &fresh[r])) ||
            (rc = dpq_index_set_codebook(fresh[r], m->cw.data(), m->Ds)) || (rc = dpq_index_set_stream(fresh[r], m->st[r])))
            return cleanup(rc);
    }
    for (size_t r = 0; r < n; ++r) {
        cudaSetDevice(m->dev[r]);
        dpq_index_close(m->ix[r]);
        m->ix[r] = fresh[r];
        fresh[r] = nullptr;
    }
    m->pos2id.swap(tab);
    return cleanup(DPQ_OK);
}

int dpq_multi_compact(dpq_multi* m) {
    int rc = dpq::api_check_device();
    if (rc) return rc;
    if (!m) return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_compact: null handle");
    if (m->Ds < 1 || m->cw.empty()) return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_compact: codebook not set");
    for (dpq_index* ix : m->ix)  // checked for every index first: the handle stays unchanged
        if (dpq_index_stat(ix, "engine") != 2)
            return dpq::api_fail(DPQ_ERR_ARG, "dpq_multi_compact: compaction needs the code-array engine (this handle runs the first-generation engine, DPQ_ENGINE=1)");
    return m->forest ? compact_parts(m) : compact_shards(m);
}

int64_t dpq_multi_stat(dpq_multi* m, int rank, const char* name) {
    if (m && name && std::string(name) == "multi_nccl_init_us") return m->nccl_us;
    if (m && name && std::string(name) == "multi_open_us") return m->open_us;
    if (!m || rank < 0 || rank >= (int)m->ix.size()) return -1;
    return dpq_index_stat(m->ix[(size_t)rank], name);
}

void dpq_multi_close(dpq_multi* m) {
    if (!m) return;
    for (size_t r = 0; r < m->comm.size(); ++r)
        if (m->comm[r]) g_nccl.CommDestroy(m->comm[r]);
    for (size_t i = 0; i < m->ix.size(); ++i) {
        cudaSetDevice(m->dev[i]);
        if (m->ix[i]) dpq_index_close(m->ix[i]);
    }
    for (int r = 0; r < m->n; ++r) {
        cudaSetDevice(r);
        if ((size_t)r < m->st.size() && m->st[(size_t)r]) cudaStreamDestroy(m->st[(size_t)r]);
        for (std::vector<void*>* v : {&m->d_q, &m->d_loc, &m->d_one, &m->d_all})
            if ((size_t)r < v->size() && (*v)[(size_t)r]) cudaFree((*v)[(size_t)r]);
    }
    cudaSetDevice(0);
    if (m->d_out) cudaFree(m->d_out);
    if (m->h_stage) cudaFreeHost(m->h_stage);
    (void)cudaGetLastError();
    dpq_set_device(0);
    delete m;
}

}  // extern "C"
