// C ABI of libdpq.so (include/dpq.h): handle management, buffer plumbing, kernel sequencing.
// No compute happens on the host here; without a usable CUDA device every entry point
// fails with DPQ_ERR_CUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/dpq.h"
#include "compact.cuh"
#include "encode_tc.cuh"
#include "kernels.cuh"
#include "tree_internal.h"

namespace {

thread_local std::string g_err;
thread_local int g_device = 0;  // like CUDA's current device: one selection per host thread

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
int check_device();
#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(DPQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));    \
    } while (0)

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {  // drops the contents when it reallocates
        if (bytes <= cap) return DPQ_OK;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            (void)cudaGetLastError();
            return fail(DPQ_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
        }
        cap = want;
        return DPQ_OK;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T>
    T* as() const {
        return reinterpret_cast<T*>(p);
    }
};

// A scratch buffer released on every return path (DevBuf itself has none: index members outlive calls).
struct Scratch {
    DevBuf b;
    ~Scratch() { b.release(); }
};

// True when p is device memory of `device`, which an index's kernels may read directly.  Host memory and memory of
// another device (no peer access is enabled) are copied to the index's device first, with cudaMemcpyDefault.
bool on_device(const void* p, int device) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice && at.device == device;
}

}  // namespace

struct dpq_index {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    // per search call: total begin, scan begin, scan end, total end, coarse-scan kernel begin / end.
    // Calls since the last
    // "timing_reset" keep their own events so a bench loop can time K steps without syncing.
    std::vector<cudaEvent_t> evs;
    int timed_calls = 0;
    cudaEvent_t* ev = nullptr;  // the last call's four events
    dpq::ScanProgram prog;  // host copy (ops/codes released after upload)
    int Ds = 0;
    // device-resident tree
    DevBuf d_ops, d_chunks, d_anc, d_codes, d_pos2id, d_cw, d_ovf;
    DevBuf d_qlut8, d_cand8, d_cnt8, d_ovf8, d_flagged2, d_cap0, d_cap1, d_part8, d_done8, d_ps_codes, d_stage8;
    int sm_slots8 = 0;  // %nsmid of the device: SM slots of the coarse scan's staging buffers (0 = not asked yet)
    int ps_R = 0;  // presample nodes currently gathered in d_ps_codes
    int last_coarse = 0;
    int last_sample_stride = 0, last_refine_stride = 0;  // strides of the sampled coarse passes of the last search
    int last_device_queries = 0;  // queries of the last dpq_index_search_device call (a host-buffer search runs sub-batches)
    int64_t last_items8 = 0;
    int n_chunks = 0;
    size_t ops_bytes = 0;
    bool has_pos2id = false;
    std::vector<uint32_t> pos2id_host;  // local slice
    int64_t pos_shift = 0;              // dpq_index_open_part: added to every reported position
    // options
    int opt_slices = 0, opt_pack = 2, opt_warps = 16, opt_slack = -1, opt_force_fallback = 0;
    int opt_epoch = 128, opt_trigger = 0, opt_ramp = 1;
    int opt_latency = -1;      // -1 auto (Q <= 16, topk <= 32, M <= 8), 0 off, 1 on: lanes = nodes scan (scan1.cu)
    int last_latency = 0;
    DevBuf d_cand1, d_cnt1;    // latency mode: candidate positions [Q][ccap], counts + overflow flags
    int opt_coarse = -1;       // -1 auto, 0 off, 1 on: 8-bit coarse pass + exact re-score (scan8.cu)
    int opt_sample = 0;        // the sample pass walks every opt_sample-th batch (0 = auto: 8 / 16 / 32 / 64 by tree size)
    int opt_slices_s = 0;      // slices of the sample pass (0 = auto)
    int opt_seed = -1;         // 0: sampled 15-bit scan gives the cap; 1 / -1 (default): exact presample -> sampled
                               // coarse scan -> exact re-score
    int opt_parts8 = 0;        // CTAs per query of the exact re-score (0 auto)
    int opt_warp_rescore = -1; // -1 auto (narrow shape, topk <= 32), 0 / 1: warp-per-query form of the exact re-score
    int opt_refine = -1;       // stride of a second, denser sampled coarse pass that tightens the cap before the
                               // full pass (0: none; -1 auto: 4 for the wide shape with topk > 32)
    int opt_presample = 0;     // nodes scored exactly per query to seed the sample pass (0 auto: 2048, or 4096 for topk > 32)
    int opt_bcap8 = 0, opt_warps8 = 24, opt_levels8 = 80;  // bcap8 0 = auto (512 narrow, 2048 wide)
    int opt_reuse8 = 1;        // 1: the narrow coarse scan reads only the table rows whose code byte changed (scan8.cu); 0: all
    int opt_stage8 = 512;      // survivor records a coarse-scan warp stages before it drains them into the lists (scan8.cu)
    int opt_stight = 100;      // percent of the presample cap the first sampled pass accepts (100 = all of it)
    int64_t opt_coarse_min = 100000;  // nodes in the shard from which the coarse search pays (gpurun_out/probe22.log)
    int opt_dbg_bound = 0x8000;  // developer probe: initial exclusive bound (results are wrong below 0x8000)
    int chunk_nodes = 512;
    // scratch
    DevBuf d_queries, d_lutf, d_scale, d_qlut, d_cand, d_cnt, d_flagged, d_ctrl, d_bound, d_key, d_gthr, d_fpart;
    void* h_stage = nullptr;  // pinned staging for the host-buffer path
    size_t h_stage_cap = 0;
    int64_t host_us[3] = {0, 0, 0};  // last dpq_index_search: enqueue, wait for the GPU, unpack (host wall clock)
    // stats
    int last_launches = 0;
    int64_t last_fallback = 0;
    bool timing_valid = false;
    // deleted nodes: one bit per local position (null until the first dpq_index_delete = nothing deleted)
    DevBuf d_dead, d_del_ids, d_del_tmp;
    int64_t n_deleted = 0;
    int64_t last_delete_us = 0;  // host wall clock of the last dpq_index_delete / _undelete (ends in a stream sync)
    const uint32_t* dead() const { return d_dead.p ? d_dead.as<uint32_t>() : nullptr; }
    // appended nodes (dpq_index_add): only the index whose positions end the position space accepts them
    bool ends_range = true;    // false for shards rank < n_ranks - 1
    int opt_add_order = 1;     // 1: an add batch is laid out sorted by code word; 0: in input order
    int64_t n_added = 0;
    int64_t last_add_us = 0;   // host wall clock of the last dpq_index_add / _add_vectors (ends in a stream sync)
    int n_ranks = 1;           // shards the tree was split into when this index was opened
    std::vector<float> cw_host;  // the codebook again: a compaction's layout builds its centroid tables on the host
    // host wall clock of the last dpq_index_compact: whole call, gather, edge search, layout (each ends in a sync)
    int64_t compact_us[4] = {0, 0, 0, 0};
};

namespace {

int choose_geometry(const dpq_index* ix, int Q, int topk, dpq::ScanGeom* g) {
    const dpq::ScanProgram& P = ix->prog;
    g->M = P.M;
    g->K = P.K;
    g->rb = P.fmt.rb;
    g->pack = ix->opt_pack == 2 ? 2 : 1;
    g->levels = P.fmt.levels();
    g->n_warps = std::max(1, std::min(16, ix->opt_warps));
    const size_t rows_bytes = (size_t)4 << g->rb;
    int slack = ix->opt_slack >= 0 ? ix->opt_slack : std::max(6, topk / 4);
    g->kp = std::min(256, topk + slack);
    if (topk > 256 || g->kp < topk) return fail(DPQ_ERR_ARG, "topk must be <= 256");
    g->kps = g->kp <= 32 ? g->kp : 0;
    g->bcap = std::min(512, ((g->kp + 31) / 32) * 32 + 32);
    const size_t overhead = (size_t)g->n_warps * (g->levels * 128 + 512) + 32 * g->pack * 4 * (1 + g->kps) + 64;
    int qgl = (int)((dpq::kMaxSmem - overhead) / rows_bytes);
    qgl = std::min(qgl, 32);
    if (qgl < 1) return fail(DPQ_ERR_ARG, "ADC table does not fit in shared memory");
    // do not spread a small batch over more lanes than needed
    int need = (Q + g->pack - 1) / g->pack;
    if (need < qgl) qgl = std::max(1, need);
    g->qgl = qgl;
    g->qpg = qgl * g->pack;
    g->n_groups = (Q + g->qpg - 1) / g->qpg;
    int n_slices = ix->opt_slices;
    if (n_slices <= 0) {
        int by_fill = (148 * 6 + g->n_groups - 1) / g->n_groups;
        int by_work = std::max(1, ix->n_chunks / (2 * g->n_warps));
        n_slices = std::max(1, std::min(by_fill, by_work));
    }
    n_slices = std::min(n_slices, std::max(1, ix->n_chunks));
    while ((int64_t)n_slices * g->n_warps > 2048) --n_slices;
    g->n_slices = n_slices;
    g->smem_bytes = (size_t)qgl * rows_bytes + overhead;
    return DPQ_OK;
}

// v2: 56 queries per group; pick the number of tree slices so that (a) the items fill whole
// waves of 148 one-CTA SMs and (b) an item is a whole number of rounds (16 warps x 4 strands
// x chunk_nodes nodes) as nearly as possible.
int choose_geometry2(const dpq_index* ix, int Q, int topk, dpq::ScanGeom* g, int n_chunks_eff = -1) {
    const dpq::ScanProgram& P = ix->prog;
    g->M = P.M;
    g->K = P.K;
    const dpq::V2Shape sh = P.shape;
    g->rb = sh.rows == 2048 ? 11 : 12;
    g->pack = 2;
    g->levels = 0;
    g->n_warps = std::max(2, std::min(16, ix->opt_warps));
    // slack: extra candidates re-scored exactly so that the rounding-bound proof in select_kernel
    // succeeds; deeper lists are denser in distance, so the slack grows with topk
    int slack = ix->opt_slack >= 0 ? ix->opt_slack : (topk <= 32 ? std::max(6, topk / 4) : topk / 2);
    g->kp = std::min(256, topk + slack);
    if (topk > 256) return fail(DPQ_ERR_ARG, "topk must be <= 256");
    g->kps = 0;
    g->bcap = g->kp <= 64 ? 256 : (g->kp <= 128 ? 512 : 1024);
    g->qgl = sh.lpg;
    g->qpg = sh.qb();
    g->n_groups = (Q + sh.qb() - 1) / sh.qb();
    const int n_chunks = n_chunks_eff > 0 ? n_chunks_eff : ix->n_chunks;
    int n_slices = n_chunks_eff > 0 ? ix->opt_slices_s : ix->opt_slices;
    if (n_slices <= 0) {
        const int chunks_per_round = g->n_warps * sh.spw();
        double best = -1.0;
        n_slices = 1;
        for (int s = 1; s <= 64 && s <= std::max(1, n_chunks / chunks_per_round); ++s) {
            const int64_t items = (int64_t)g->n_groups * s;
            const int64_t waves = (items + 147) / 148;
            const double eff_wave = (double)items / (double)(waves * 148);
            const double cpi = (double)n_chunks / s;
            const double rounds = std::ceil(cpi / chunks_per_round);
            const double eff = eff_wave * (cpi / chunks_per_round) / rounds;
            if (eff > best + 1e-9) {
                best = eff;
                n_slices = s;
            }
        }
    }
    n_slices = std::max(1, std::min(n_slices, std::max(1, n_chunks)));
    g->n_slices = n_slices;
    g->smem_bytes = 0;
    return DPQ_OK;
}

int upload(DevBuf& b, const void* src, size_t bytes, cudaStream_t st) {
    int rc = b.ensure(std::max<size_t>(bytes, 16));
    if (rc) return rc;
    if (bytes) CU(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, st));
    return DPQ_OK;
}

// Keeps the first `used` bytes of b and makes room for `need`: a new block of at least 1.5x the old capacity (many
// small adds stay amortised), the contents copied device to device on st, every byte past `used` zeroed, then the
// old block freed.
int grow(DevBuf& b, size_t used, size_t need, cudaStream_t st) {
    if (need <= b.cap) return DPQ_OK;
    const size_t want = std::max(need, b.cap + b.cap / 2) + 256;
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return fail(DPQ_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e));
    }
    if (used) e = cudaMemcpyAsync(p, b.p, used, cudaMemcpyDeviceToDevice, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(static_cast<char*>(p) + used, 0, want - used, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // searches still in flight read the old block
    if (e != cudaSuccess) {
        cudaFree(p);
        return fail(DPQ_ERR_CUDA, std::string("growing a device buffer: ") + cudaGetErrorString(e));
    }
    b.release();
    b.p = p;
    b.cap = want;
    return DPQ_OK;
}

int finish_open(dpq_index* ix, const uint32_t* pos2id) {
    dpq::ScanProgram& P = ix->prog;
    CU(cudaSetDevice(ix->device));
    CU(cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking));
    int rc;
    if ((rc = upload(ix->d_ops, P.ops.data(), P.ops.size() * 4, ix->stream))) return rc;
    if ((rc = upload(ix->d_chunks, P.chunks.data(), P.chunks.size() * sizeof(dpq::ChunkDesc), ix->stream)))
        return rc;
    if ((rc = upload(ix->d_anc, P.anc.data(), P.anc.size(), ix->stream))) return rc;
    if ((rc = upload(ix->d_codes, P.codes.data(), P.codes.size(), ix->stream))) return rc;
    ix->n_chunks = (int)P.chunks.size();
    ix->ops_bytes = P.ops.size() * 4;
    if (P.v2) {  // the code array IS the program: chunk c = nodes [c * 64, c * 64 + 64)
        ix->n_chunks = (int)((P.n_local + P.v2_chunk_nodes - 1) / P.v2_chunk_nodes);
        ix->ops_bytes = P.codes.size();
    }
    if (pos2id) {
        ix->has_pos2id = true;
        const int64_t b = P.base_pos - ix->pos_shift;  // pos2id is indexed by the tree's own positions
        ix->pos2id_host.assign(pos2id + b, pos2id + b + P.n_local);
    }
    CU(cudaStreamSynchronize(ix->stream));
    // the device copy is authoritative from here on
    std::vector<uint32_t>().swap(P.ops);
    std::vector<uint8_t>().swap(P.codes);
    std::vector<uint8_t>().swap(P.anc);
    std::vector<dpq::ChunkDesc>().swap(P.chunks);
    return DPQ_OK;
}

int check_device() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        (void)cudaGetLastError();
        return fail(DPQ_ERR_CUDA, "no CUDA device available (libdpq has no CPU fallback)");
    }
    if (g_device >= n) return fail(DPQ_ERR_CUDA, "selected device index out of range");
    return DPQ_OK;
}

}  // namespace

namespace dpq {  // shared with secondary.cu / edges.cu
int api_fail(int code, const std::string& msg) { return fail(code, msg); }
int api_check_device() { return check_device(); }
int api_device() { return g_device; }
}  // namespace dpq

extern "C" {

int dpq_version(void) { return 100; }
const char* dpq_last_error(void) { return g_err.c_str(); }

int dpq_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        (void)cudaGetLastError();
        return 0;
    }
    return n;
}

int dpq_set_device(int device) {
    int n = dpq_device_count();
    if (device < 0 || device >= n) return fail(DPQ_ERR_CUDA, "dpq_set_device: no such device");
    g_device = device;
    CU(cudaSetDevice(device));
    return DPQ_OK;
}

static int open_tree_shard_impl(dpq_tree* t, int rank, int n_ranks, int64_t first_pos, dpq_index** out);

static int open_common(const uint8_t* payload, int64_t n_bytes, int64_t n_codes, int M, int K,
                       const uint32_t* pos2id, int rank, int n_ranks, int64_t first_pos, dpq_index** out) {
    if (!payload || !out) return fail(DPQ_ERR_ARG, "dpq_index_open: null argument");
    *out = nullptr;
    if (first_pos < 0 || first_pos + n_codes > 0xFFFFFFFFLL)
        return fail(DPQ_ERR_ARG, "dpq_index_open_part: positions must stay below 2^32 - 1");
    int rc = check_device();
    if (rc) return rc;
    // DPQ_ENGINE=1 in the environment keeps the first-generation op program / kernel
    const char* eng = getenv("DPQ_ENGINE");
    const char* host_dec = getenv("DPQ_HOST_DECODE");  // 1: decode the stream on one host core (program.cpp) instead of the GPU
    if (!(eng && eng[0] == '1') && !(host_dec && host_dec[0] == '1') && dpq::v2_shape_ok(M, K)) {
        if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(DPQ_ERR_FORMAT, "dpq_index_open: bad rank / n_ranks");
        dpq_tree* t = nullptr;
        rc = dpq::decode_stream_device(payload, n_bytes, n_codes, M, K, pos2id, &t);  // program_dev.cu
        if (rc) return fail(rc, std::string("dpq_index_open: ") + g_err);
        rc = open_tree_shard_impl(t, rank, n_ranks, first_pos, out);
        delete t;
        return rc;
    }
    dpq_index* ix = new dpq_index();
    ix->device = g_device;
    std::string err = dpq::compile_program(payload, n_bytes, n_codes, M, K, rank, n_ranks,
                                           ix->chunk_nodes, &ix->prog, eng && eng[0] == '1' ? 1 : 0);
    if (err.empty() && first_pos && !ix->prog.v2) err = "a forest part needs the fixed-record program (M <= 16, M*K <= 4096)";
    if (!err.empty()) {
        delete ix;
        return fail(DPQ_ERR_FORMAT, "dpq_index_open: " + err);
    }
    ix->ends_range = rank == n_ranks - 1;
    ix->n_ranks = n_ranks;
    if (first_pos) {  // one tree of a forest: every position this index reports is shifted
        ix->pos_shift = first_pos;
        ix->prog.base_pos += first_pos;
    }
    rc = finish_open(ix, pos2id);
    if (rc) {
        dpq_index_close(ix);
        return rc;
    }
    *out = ix;
    return DPQ_OK;
}

int dpq_index_open(const uint8_t* payload, int64_t n_bytes, int64_t n_codes, int M, int K,
                   const uint32_t* pos2id, int rank, int n_ranks, dpq_index** out) {
    return open_common(payload, n_bytes, n_codes, M, K, pos2id, rank, n_ranks, 0, out);
}

int dpq_index_open_part(const uint8_t* payload, int64_t n_bytes, int64_t n_codes, int M, int K,
                        const uint32_t* pos2id, int64_t first_pos, dpq_index** out) {
    return open_common(payload, n_bytes, n_codes, M, K, pos2id, 0, 1, first_pos, out);
}

static int open_file_common(const char* tree_path, const char* qnode_path, int M, int K, int rank,
                            int n_ranks, int64_t first_pos, dpq_index** out) {
    if (!tree_path || !out) return fail(DPQ_ERR_ARG, "dpq_index_open_file: null argument");
    FILE* f = fopen(tree_path, "rb");
    if (!f) return fail(DPQ_ERR_IO, std::string("cannot open ") + tree_path);
    int64_t hdr[2];
    if (fread(hdr, 8, 2, f) != 2) {
        fclose(f);
        return fail(DPQ_ERR_FORMAT, "tree file shorter than its header");
    }
    if (hdr[0] < 1 || hdr[1] < M) {
        fclose(f);
        return fail(DPQ_ERR_FORMAT, "bad tree file header");
    }
    std::vector<uint8_t> payload((size_t)hdr[1]);
    size_t got = fread(payload.data(), 1, payload.size(), f);
    fclose(f);
    if (got != payload.size()) return fail(DPQ_ERR_FORMAT, "tree file truncated");
    std::vector<uint32_t> pos2id;
    if (qnode_path) {  // 60-byte QNode records, vec_id at offset 0 (DCAT.h:79-101)
        FILE* q = fopen(qnode_path, "rb");
        if (!q) return fail(DPQ_ERR_IO, std::string("cannot open ") + qnode_path);
        pos2id.resize((size_t)hdr[0]);
        std::vector<uint8_t> rec(60 * 4096);
        size_t done = 0;
        while (done < pos2id.size()) {
            size_t want = std::min<size_t>(4096, pos2id.size() - done);
            if (fread(rec.data(), 60, want, q) != want) {
                fclose(q);
                return fail(DPQ_ERR_FORMAT, "QNode file truncated");
            }
            for (size_t i = 0; i < want; ++i) memcpy(&pos2id[done + i], rec.data() + 60 * i, 4);
            done += want;
        }
        fclose(q);
    }
    return open_common(payload.data(), hdr[1], hdr[0], M, K, qnode_path ? pos2id.data() : nullptr, rank, n_ranks,
                       first_pos, out);
}

int dpq_index_open_tree(dpq_tree* t, int64_t first_pos, dpq_index** out) {
    if (!t || !out) return fail(DPQ_ERR_ARG, "dpq_index_open_tree: null argument");
    *out = nullptr;
    const int M = t->M, K = t->K;
    const int64_t n = t->n;
    if (t->on_device) {
        if (first_pos) return fail(DPQ_ERR_ARG, "dpq_index_open_tree: a device-resident tree opens at first_pos 0 (use dpq_index_open_tree_shard)");
        return dpq_index_open_tree_shard(t, 0, 1, out);
    }
    const char* eng = getenv("DPQ_ENGINE");
    if ((eng && eng[0] == '1') || !dpq::v2_shape_ok(M, K))  // first-generation program: through the byte stream
        return open_common(t->payload.data(), (int64_t)t->payload.size(), n, M, K, t->vec_id.data(), 0, 1, first_pos, out);
    if (first_pos < 0 || first_pos + n > 0xFFFFFFFFLL)
        return fail(DPQ_ERR_ARG, "dpq_index_open_tree: positions must stay below 2^32 - 1");
    if ((int64_t)t->codes_by_pos.size() != n * M || (int64_t)t->depth.size() != n)
        return fail(DPQ_ERR_ARG, "dpq_index_open_tree: the tree has no layout arrays");
    int rc = check_device();
    if (rc) return rc;
    dpq_index* ix = new dpq_index();
    ix->device = g_device;
    dpq::ScanProgram& P = ix->prog;
    P.M = M;
    P.K = K;
    P.fmt.rb = (M * K <= 2048) ? 11 : 12;
    P.v2 = true;
    P.shape = dpq::v2_shape(M, K);
    P.cstride = P.shape.nf;
    P.n_codes = n;
    P.n_bytes = (int64_t)t->payload.size();
    P.base_pos = first_pos;
    P.n_local = n;
    P.local_bytes = P.n_bytes;
    P.n_diffs = t->n_diffs;
    P.depth_hist.assign(17, 0);
    for (int64_t i = 0; i < n; ++i) P.depth_hist[std::min<int>(t->depth[(size_t)i], 16)]++;
    ix->pos_shift = first_pos;
    auto bail = [&](int code) {
        dpq_index_close(ix);
        return code;
    };
    if (cudaSetDevice(ix->device) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(DPQ_ERR_CUDA, "dpq_index_open_tree: stream setup failed"));
    // the code array by position IS the device program; pad to the scan's word stride when M < stride
    cudaError_t e = cudaSuccess;
    if (M == P.cstride) {
        if ((rc = upload(ix->d_codes, t->codes_by_pos.data(), (size_t)n * M, ix->stream))) return bail(rc);
    } else {
        DevBuf d_raw;
        if ((rc = upload(d_raw, t->codes_by_pos.data(), (size_t)n * M, ix->stream)) ||
            (rc = ix->d_codes.ensure((size_t)n * P.cstride))) {
            d_raw.release();
            return bail(rc);
        }
        e = dpq::launch_pad_codes(d_raw.as<uint8_t>(), n, M, P.cstride, ix->d_codes.as<uint8_t>(), ix->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ix->stream);
        d_raw.release();
    }
    // the first-generation buffers stay empty (16-byte placeholders keep the launch arguments valid)
    if ((rc = ix->d_ops.ensure(16)) || (rc = ix->d_chunks.ensure(16)) || (rc = ix->d_anc.ensure(16))) return bail(rc);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ix->stream);
    if (e != cudaSuccess) return bail(fail(DPQ_ERR_CUDA, std::string("dpq_index_open_tree: ") + cudaGetErrorString(e)));
    ix->n_chunks = (int)((n + P.v2_chunk_nodes - 1) / P.v2_chunk_nodes);
    ix->ops_bytes = (size_t)n * P.cstride;
    ix->has_pos2id = true;
    ix->pos2id_host = t->vec_id;
    *out = ix;
    return DPQ_OK;
}

// Shard `rank` of `n_ranks` of a tree that dpq_tree_build[_device] just produced: whole depth-1
// subtrees balanced by stream bytes, the same deal as dpq_index_open(payload, ..., rank, n_ranks).
// A device-resident tree never leaves HBM: the shard's slice of the code array is copied device to
// device (and padded to the word stride when M is not 8 / 16).
static int open_tree_shard_impl(dpq_tree* t, int rank, int n_ranks, int64_t first_pos, dpq_index** out);

int dpq_index_open_tree_shard(dpq_tree* t, int rank, int n_ranks, dpq_index** out) {
    if (!t || !out) return fail(DPQ_ERR_ARG, "dpq_index_open_tree_shard: null argument");
    *out = nullptr;
    if (n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(DPQ_ERR_ARG, "dpq_index_open_tree_shard: bad rank / n_ranks");
    const int M = t->M, K = t->K;
    const int64_t n = t->n;
    const char* eng = getenv("DPQ_ENGINE");
    const bool gen1 = (eng && eng[0] == '1') || !dpq::v2_shape_ok(M, K);
    if (!t->on_device) {
        if (n_ranks == 1 && !gen1) return dpq_index_open_tree(t, 0, out);
        return open_common(t->payload.data(), (int64_t)t->payload.size(), n, M, K, t->vec_id.data(), rank, n_ranks, 0, out);
    }
    if (gen1) return fail(DPQ_ERR_ARG, "dpq_index_open_tree_shard: a device-resident tree needs the code-array engine");
    return open_tree_shard_impl(t, rank, n_ranks, 0, out);
}

// Fills ix (device, stream set; nothing loaded yet) with shard `rank` of `n_ranks` of a device-resident tree;
// first_pos shifts every reported position (forest parts).  On failure the caller closes ix.
static int load_tree_shard(dpq_index* ix, dpq_tree* t, int rank, int n_ranks, int64_t first_pos) {
    const int M = t->M, K = t->K;
    const int64_t n = t->n;
    int rc;
    std::vector<int64_t> bounds, bytes;
    if ((rc = dpq::tree_shard_bounds(t, n_ranks, &bounds, &bytes))) return rc;
    int64_t lo = bounds[(size_t)rank], hi = bounds[(size_t)rank + 1];
    if (hi == lo) lo = hi = n;  // an empty shard reports base_pos = n_codes like the stream reader (program.cpp)
    ix->ends_range = rank == n_ranks - 1;
    ix->n_ranks = n_ranks;
    dpq::ScanProgram& P = ix->prog;
    P.M = M;
    P.K = K;
    P.fmt.rb = (M * K <= 2048) ? 11 : 12;
    P.v2 = true;
    P.shape = dpq::v2_shape(M, K);
    P.cstride = P.shape.nf;
    P.n_codes = n;
    P.n_bytes = t->payload_bytes;
    P.base_pos = lo + first_pos;
    ix->pos_shift = first_pos;
    P.n_local = hi - lo;
    P.local_bytes = bytes[(size_t)rank];
    {   // changed subspaces = record bytes - bitmap bytes - depth bytes (one per odd position)
        const int64_t rlo = std::max<int64_t>(lo, 1), recs = std::max<int64_t>(hi - rlo, 0);
        const int64_t odd = recs > 0 ? ((hi - 1 + 1) / 2 - (rlo - 1 + 1) / 2) : 0;  // odd p in [rlo, hi)
        P.n_diffs = bytes[(size_t)rank] - (rank == 0 ? M : 0) - (int64_t)((M + 7) / 8) * recs - odd;
    }
    int64_t hist[17] = {0};
    if ((rc = dpq::depth_hist_device(ix->device, (const uint8_t*)t->d_depth + lo, P.n_local, hist))) return rc;
    P.depth_hist.assign(hist, hist + 17);
    if ((rc = ix->d_codes.ensure((size_t)std::max<int64_t>(P.n_local, 1) * P.cstride))) return rc;
    cudaError_t e = cudaSuccess;
    const uint8_t* src = (const uint8_t*)t->d_codes_by_pos + (size_t)lo * M;
    if (P.n_local > 0) {
        if (M == P.cstride)
            e = cudaMemcpyAsync(ix->d_codes.p, src, (size_t)P.n_local * M, cudaMemcpyDeviceToDevice, ix->stream);
        else
            e = dpq::launch_pad_codes(src, P.n_local, M, P.cstride, ix->d_codes.as<uint8_t>(), ix->stream);
    }
    if ((rc = ix->d_ops.ensure(16)) || (rc = ix->d_chunks.ensure(16)) || (rc = ix->d_anc.ensure(16))) return rc;
    if (t->d_vec_id) {
        ix->pos2id_host.resize((size_t)P.n_local);
        if (e == cudaSuccess && P.n_local > 0)
            e = cudaMemcpyAsync(ix->pos2id_host.data(), (const uint32_t*)t->d_vec_id + lo, (size_t)P.n_local * 4,
                                cudaMemcpyDeviceToHost, ix->stream);
        ix->has_pos2id = true;
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ix->stream);
    if (e != cudaSuccess) return fail(DPQ_ERR_CUDA, std::string("dpq_index_open_tree_shard: ") + cudaGetErrorString(e));
    ix->n_chunks = (int)((P.n_local + P.v2_chunk_nodes - 1) / P.v2_chunk_nodes);
    ix->ops_bytes = (size_t)P.n_local * P.cstride;
    return DPQ_OK;
}

// device-resident tree -> index of one shard; first_pos shifts every reported position (forest parts)
static int open_tree_shard_impl(dpq_tree* t, int rank, int n_ranks, int64_t first_pos, dpq_index** out) {
    if (first_pos < 0 || first_pos + t->n > 0xFFFFFFFFLL) return fail(DPQ_ERR_ARG, "dpq_index_open: positions must stay below 2^32 - 1");
    int rc = check_device();
    if (rc) return rc;
    if (g_device != t->device) return fail(DPQ_ERR_ARG, "dpq_index_open_tree_shard: the tree lives on another device");
    dpq_index* ix = new dpq_index();
    ix->device = g_device;
    if (cudaSetDevice(ix->device) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ix->stream, cudaStreamNonBlocking) != cudaSuccess) {
        dpq_index_close(ix);
        return fail(DPQ_ERR_CUDA, "dpq_index_open_tree_shard: stream setup failed");
    }
    if ((rc = load_tree_shard(ix, t, rank, n_ranks, first_pos))) {
        dpq_index_close(ix);
        return rc;
    }
    *out = ix;
    return DPQ_OK;
}

int dpq_index_open_file(const char* tree_path, const char* qnode_path, int M, int K, int rank,
                        int n_ranks, dpq_index** out) {
    return open_file_common(tree_path, qnode_path, M, K, rank, n_ranks, 0, out);
}

int dpq_index_open_part_file(const char* tree_path, const char* qnode_path, int M, int K, int64_t first_pos,
                             dpq_index** out) {
    return open_file_common(tree_path, qnode_path, M, K, 0, 1, first_pos, out);
}

int dpq_index_set_codebook(dpq_index* ix, const float* cw, int Ds) {
    if (!ix || !cw || Ds < 1) return fail(DPQ_ERR_ARG, "dpq_index_set_codebook: bad argument");
    CU(cudaSetDevice(ix->device));
    ix->Ds = Ds;
    const size_t n = (size_t)ix->prog.M * ix->prog.K * Ds;
    int rc = upload(ix->d_cw, cw, n * sizeof(float), ix->stream);
    if (rc) return rc;
    CU(cudaStreamSynchronize(ix->stream));
    ix->cw_host.assign(cw, cw + n);
    return DPQ_OK;
}

int dpq_index_set_stream(dpq_index* ix, void* cuda_stream) {
    if (!ix) return fail(DPQ_ERR_ARG, "dpq_index_set_stream: null");
    CU(cudaSetDevice(ix->device));
    CU(cudaStreamSynchronize(ix->stream));
    if (ix->own_stream && ix->stream) CU(cudaStreamDestroy(ix->stream));
    ix->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    ix->own_stream = false;
    return DPQ_OK;
}

int dpq_index_set_option(dpq_index* ix, const char* name, int64_t v) {
    if (!ix || !name) return fail(DPQ_ERR_ARG, "dpq_index_set_option: null argument");
    std::string n(name);
    if (n == "slices") ix->opt_slices = (int)v;
    else if (n == "pack") ix->opt_pack = (int)v;
    else if (n == "warps") ix->opt_warps = (int)v;
    else if (n == "slack") ix->opt_slack = (int)v;
    else if (n == "force_fallback") ix->opt_force_fallback = (int)v;
    else if (n == "timing_reset") ix->timed_calls = 0;
    else if (n == "epoch") ix->opt_epoch = (int)v;
    else if (n == "trigger") ix->opt_trigger = (int)v;
    else if (n == "ramp") ix->opt_ramp = (int)v;
    else if (n == "dbg_bound") ix->opt_dbg_bound = (int)v;
    else if (n == "coarse") ix->opt_coarse = (int)v;
    else if (n == "latency") ix->opt_latency = (int)v;
    else if (n == "sample") ix->opt_sample = std::max(0, (int)v);
    else if (n == "bcap8") ix->opt_bcap8 = v <= 0 ? 0 : std::max(32, (int)v);
    else if (n == "warps8") ix->opt_warps8 = std::max(2, std::min(24, (int)v));
    else if (n == "reuse8") ix->opt_reuse8 = v != 0;
    else if (n == "stage8") ix->opt_stage8 = std::max(32, std::min(1 << 16, (int)v));
    else if (n == "coarse_min") ix->opt_coarse_min = v;
    else if (n == "seed") ix->opt_seed = (int)v;
    else if (n == "refine") ix->opt_refine = (int)v;
    else if (n == "parts8") ix->opt_parts8 = std::max(0, std::min(16, (int)v));
    else if (n == "warp_rescore") ix->opt_warp_rescore = (int)v;
    else if (n == "slices_s") ix->opt_slices_s = (int)v;
    else if (n == "presample") ix->opt_presample = v <= 0 ? 0 : std::max(64, std::min(8192, (int)v));
    else if (n == "levels8") ix->opt_levels8 = std::max(31, std::min(123, (int)v));
    else if (n == "stight") ix->opt_stight = std::max(50, std::min(100, (int)v));
    else if (n == "add_order") ix->opt_add_order = v != 0;
    else return fail(DPQ_ERR_ARG, "unknown option " + n);
    return DPQ_OK;
}

// The device copy of the id table, uploaded on the index's stream the first time a search, a delete or a compaction
// needs it; later changes (dpq_index_add) keep both copies in step.
static int upload_pos2id(dpq_index* ix) {
    if (!ix->has_pos2id || ix->d_pos2id.p) return DPQ_OK;
    int rc = ix->d_pos2id.ensure(std::max<size_t>(ix->pos2id_host.size(), 1) * 4);
    if (rc) return rc;
    CU(cudaMemcpyAsync(ix->d_pos2id.p, ix->pos2id_host.data(), ix->pos2id_host.size() * 4, cudaMemcpyHostToDevice, ix->stream));
    return DPQ_OK;
}

// dpq_index_delete / dpq_index_undelete: the ids are sorted on the device, then every 32-position word of the
// bitmap is rebuilt from a binary search of its nodes' ids (dead.cu).  The caller's stream orders the change
// before every later search; the call returns once it is complete.
static int mark_dead(dpq_index* ix, const uint32_t* ids, int64_t n, bool set, const char* what) {
    const auto t0 = std::chrono::steady_clock::now();
    int rc = check_device();
    if (rc) return rc;
    if (!ix) return fail(DPQ_ERR_ARG, std::string(what) + ": null index");
    if (n < 0 || (n > 0 && !ids)) return fail(DPQ_ERR_ARG, std::string(what) + ": ids is null or n < 0");
    if (n > 0x7FFFFFFFLL) return fail(DPQ_ERR_ARG, std::string(what) + ": more than 2^31 - 1 ids in one call");
    const dpq::ScanProgram& P = ix->prog;
    if (!P.v2)
        return fail(DPQ_ERR_ARG, std::string(what) +
                                     ": deletion needs the code-array engine (this index runs the first-generation engine, DPQ_ENGINE=1)");
    if (n == 0 || (!set && !ix->d_dead.p)) {
        ix->last_delete_us = 0;
        return DPQ_OK;
    }
    CU(cudaSetDevice(ix->device));
    cudaStream_t st = ix->stream;
    const size_t words = (size_t)((P.n_local + 31) / 32);
    if (!ix->d_dead.p) {  // first delete: the bitmap appears, all live
        if ((rc = ix->d_dead.ensure(std::max<size_t>(words, 1) * 4))) return rc;
        CU(cudaMemsetAsync(ix->d_dead.p, 0, ix->d_dead.cap, st));
    }
    if ((rc = upload_pos2id(ix))) return rc;
    // [n raw ids][n sorted ids][count], then the sort's scratch
    const size_t ids_bytes = ((size_t)n * 4 + 15) / 16 * 16;
    size_t tmp_bytes = 0;
    CU(dpq::sort_ids(nullptr, nullptr, (int)n, nullptr, &tmp_bytes, st));
    if ((rc = ix->d_del_ids.ensure(2 * ids_bytes + 16)) || (rc = ix->d_del_tmp.ensure(std::max<size_t>(tmp_bytes, 16)))) return rc;
    uint32_t* d_raw = ix->d_del_ids.as<uint32_t>();
    uint32_t* d_sorted = reinterpret_cast<uint32_t*>(ix->d_del_ids.as<char>() + ids_bytes);
    unsigned long long* d_count = reinterpret_cast<unsigned long long*>(ix->d_del_ids.as<char>() + 2 * ids_bytes);
    CU(cudaMemcpyAsync(d_raw, ids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CU(dpq::sort_ids(d_raw, d_sorted, (int)n, ix->d_del_tmp.p, &tmp_bytes, st));
    CU(cudaMemsetAsync(d_count, 0, 8, st));
    dpq::launch_mark_dead(d_sorted, n, ix->has_pos2id ? ix->d_pos2id.as<uint32_t>() : nullptr, (uint32_t)P.base_pos, P.n_local, set,
                          ix->d_dead.as<uint32_t>(), d_count, st);
    CU(cudaGetLastError());
    unsigned long long count = 0;
    CU(cudaMemcpyAsync(&count, d_count, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ix->n_deleted = (int64_t)count;
    if (count == 0) ix->d_dead.release();  // nothing deleted: the searches are back on the kernels without liveness tests
    ix->last_delete_us =
        (int64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    return DPQ_OK;
}

int dpq_index_delete(dpq_index* ix, const uint32_t* ids, int64_t n) { return mark_dead(ix, ids, n, true, "dpq_index_delete"); }
int dpq_index_undelete(dpq_index* ix, const uint32_t* ids, int64_t n) { return mark_dead(ix, ids, n, false, "dpq_index_undelete"); }

// dpq_index_add / dpq_index_add_vectors: the checks both share.  *done = true when there is nothing to do.
static int add_check(dpq_index* ix, const void* data, int64_t n, const char* what, bool* done) {
    *done = true;
    int rc = check_device();
    if (rc) return rc;
    if (!ix) return fail(DPQ_ERR_ARG, std::string(what) + ": null index");
    if (n < 0 || (n > 0 && !data)) return fail(DPQ_ERR_ARG, std::string(what) + ": input is null or n < 0");
    if (n > 0x7FFFFFFFLL) return fail(DPQ_ERR_ARG, std::string(what) + ": more than 2^31 - 1 rows in one call");
    const dpq::ScanProgram& P = ix->prog;
    if (!P.v2)
        return fail(DPQ_ERR_ARG, std::string(what) +
                                     ": adding needs the code-array engine (this index runs the first-generation engine, DPQ_ENGINE=1)");
    if (!ix->ends_range)
        return fail(DPQ_ERR_ARG, std::string(what) + ": only the last shard (or a whole tree, or a forest part) accepts adds");
    if (P.base_pos + P.n_local + n > 0xFFFFFFFFLL)
        return fail(DPQ_ERR_ARG, std::string(what) + ": an appended position would reach 0xFFFFFFFF");
    if (n == 0) {
        ix->last_add_us = 0;
        return DPQ_OK;
    }
    *done = false;
    return DPQ_OK;
}

// Appends n nodes whose codes d_in [n][M] are on the device: sorted by code word on the device (add.cu) unless
// add_order = 0, then the padded words go to the tail of d_codes, the ids to the tail of the id table and the
// positions to out_pos.  ids / out_pos may be host or device pointers.  Host state changes only once the device
// work has completed, so a failed call leaves the index as it was.
static int append_nodes(dpq_index* ix, const uint8_t* d_in, int64_t n, const uint32_t* ids, uint32_t* out_pos,
                        std::chrono::steady_clock::time_point t0) {
    dpq::ScanProgram& P = ix->prog;
    cudaStream_t st = ix->stream;
    const int M = P.M, cs = P.cstride;
    const int64_t n_old = P.n_local, n_new = n_old + n;
    const uint32_t first = (uint32_t)(P.base_pos + n_old);
    const bool table = ix->has_pos2id || ids;
    int rc;
    // scratch: [keys 2n][values 2n][ids n][tail ids n][positions n], then the sort's
    size_t tmp_bytes = 0;
    if (ix->opt_add_order) CU(dpq::sort_add_batch(nullptr, n, M, cs, nullptr, nullptr, nullptr, &tmp_bytes, st));
    const size_t n4 = ((size_t)n * 4 + 15) / 16 * 16;
    const size_t off_vals = (size_t)n * 16, off_ids = off_vals + 2 * n4, off_tail = off_ids + n4, off_pos = off_tail + n4,
                 off_tmp = off_pos + n4;
    Scratch s;
    if ((rc = s.b.ensure(off_tmp + tmp_bytes + 16))) return rc;
    char* base = s.b.as<char>();
    uint32_t* d_ids = ids ? reinterpret_cast<uint32_t*>(base + off_ids) : nullptr;
    uint32_t* d_tail = table ? reinterpret_cast<uint32_t*>(base + off_tail) : nullptr;
    uint32_t* d_pos = reinterpret_cast<uint32_t*>(base + off_pos);
    if (ids) CU(cudaMemcpyAsync(d_ids, ids, (size_t)n * 4, cudaMemcpyDefault, st));
    const uint32_t* perm = nullptr;
    if (ix->opt_add_order) {
        uint32_t* vals = reinterpret_cast<uint32_t*>(base + off_vals);
        CU(dpq::sort_add_batch(d_in, n, M, cs, s.b.as<uint64_t>(), vals, base + off_tmp, &tmp_bytes, st));
        perm = vals + n;
    }
    // room for the new nodes (and a zero pad word: the latency scan reads nodes in pairs)
    if ((rc = grow(ix->d_codes, (size_t)n_old * cs, (size_t)(n_new + 1) * cs, st))) return rc;
    CU(dpq::launch_add_gather(d_in, n, M, cs, perm, d_ids, first, ix->d_codes.as<uint8_t>() + (size_t)n_old * cs, d_tail, d_pos, st));
    if (ix->d_dead.p && (rc = grow(ix->d_dead, (size_t)(n_old + 31) / 32 * 4, (size_t)(n_new + 31) / 32 * 4, st))) return rc;
    if (table && ix->d_pos2id.p) {  // the device copy of the id table, once a search or a delete has uploaded it
        if ((rc = grow(ix->d_pos2id, (size_t)n_old * 4, (size_t)n_new * 4, st))) return rc;
        CU(cudaMemcpyAsync(ix->d_pos2id.as<uint32_t>() + n_old, d_tail, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    }
    std::vector<uint32_t> tail(table ? (size_t)n : 0);
    if (table) CU(cudaMemcpyAsync(tail.data(), d_tail, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    if (out_pos) CU(cudaMemcpyAsync(out_pos, d_pos, (size_t)n * 4, cudaMemcpyDefault, st));
    CU(cudaStreamSynchronize(st));
    if (table) {
        if (!ix->has_pos2id) {  // the first add that names ids: the nodes so far keep id = position
            ix->pos2id_host.resize((size_t)n_old);
            for (int64_t i = 0; i < n_old; ++i) ix->pos2id_host[(size_t)i] = (uint32_t)(P.base_pos + i);
            ix->has_pos2id = true;
        }
        ix->pos2id_host.insert(ix->pos2id_host.end(), tail.begin(), tail.end());
    }
    P.n_local = n_new;
    ix->n_chunks = (int)((n_new + P.v2_chunk_nodes - 1) / P.v2_chunk_nodes);
    ix->ops_bytes = (size_t)n_new * cs;
    // the presample's gathered nodes were strided by the old n_local; presample_kernel tests dead bits at the new stride
    ix->ps_R = 0;
    ix->n_added += n;
    ix->last_add_us = (int64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    return DPQ_OK;
}

int dpq_index_add(dpq_index* ix, const uint8_t* codes, int64_t n, const uint32_t* ids, uint32_t* out_pos) {
    const auto t0 = std::chrono::steady_clock::now();
    bool done = true;
    int rc = add_check(ix, codes, n, "dpq_index_add", &done);
    if (rc || done) return rc;
    CU(cudaSetDevice(ix->device));
    const int M = ix->prog.M, K = ix->prog.K;
    const uint8_t* d_in = codes;
    Scratch staged;
    if (!on_device(codes, ix->device)) {  // host memory, or another device's
        if ((rc = staged.b.ensure((size_t)n * M))) return rc;
        CU(cudaMemcpyAsync(staged.b.p, codes, (size_t)n * M, cudaMemcpyDefault, ix->stream));
        d_in = staged.b.as<uint8_t>();
    }
    if (K < 256) {  // a code byte >= K would index past the tables; the check runs on the legacy stream
        CU(cudaStreamSynchronize(ix->stream));
        if ((rc = dpq::check_code_range(d_in, n, M, K))) return rc;
    }
    return append_nodes(ix, d_in, n, ids, out_pos, t0);
}

// Encoded on the device with the index's codebook by the kernels and path choice of dpq_encode (tensor cores for
// Ds in {4, 8, 16} unless DPQ_ENCODE_TC=0), so the codes are bit-identical to its; input that is not on the
// index's device is staged in chunks of at most 2^20 rows.
int dpq_index_add_vectors(dpq_index* ix, const float* x, int64_t n, int D, const uint32_t* ids, uint32_t* out_pos) {
    const auto t0 = std::chrono::steady_clock::now();
    bool done = true;
    int rc = add_check(ix, x, n, "dpq_index_add_vectors", &done);
    if (rc || done) return rc;
    const int M = ix->prog.M, K = ix->prog.K, Ds = ix->Ds;
    if (!ix->d_cw.p || Ds < 1) return fail(DPQ_ERR_ARG, "dpq_index_add_vectors: no codebook (dpq_index_set_codebook first)");
    if (D < 1 || D > M * Ds) return fail(DPQ_ERR_ARG, "dpq_index_add_vectors: D must be in 1 .. M * Ds");
    CU(cudaSetDevice(ix->device));
    cudaStream_t st = ix->stream;
    const char* env = getenv("DPQ_ENCODE_TC");
    const bool tc = dpq::encode_tc_supported(M, K, Ds) && !(env && env[0] == '0');
    const bool on_dev = on_device(x, ix->device);  // else host memory or another device's: staged in chunks
    const int64_t chunk = on_dev ? n : std::min<int64_t>(n, (int64_t)1 << 20);
    Scratch s_codes, s_x, s_tc;
    DevBuf &d_codes = s_codes.b, &d_x = s_x.b, &d_tc = s_tc.b;
    if ((rc = d_codes.ensure((size_t)n * M)) || (!on_dev && (rc = d_x.ensure((size_t)chunk * D * 4)))) return rc;
    int n_sms = 148;
    if (tc) {  // [operand blocks][error word]
        CU(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, ix->device));
        if ((rc = d_tc.ensure(dpq::encode_tc_scratch_bytes(M) + 16))) return rc;
        CU(cudaMemsetAsync(d_tc.as<char>() + dpq::encode_tc_scratch_bytes(M), 0, 4, st));
    }
    uint32_t* d_err = reinterpret_cast<uint32_t*>(d_tc.as<char>() + (tc ? dpq::encode_tc_scratch_bytes(M) : 0));
    for (int64_t s0 = 0; s0 < n; s0 += chunk) {
        const int64_t c = std::min(chunk, n - s0);
        const float* src = x + (size_t)s0 * D;
        if (!on_dev) {
            CU(cudaMemcpyAsync(d_x.p, src, (size_t)c * D * 4, cudaMemcpyDefault, st));
            src = d_x.as<float>();
        }
        uint8_t* dst = d_codes.as<uint8_t>() + (size_t)s0 * M;
        if (tc) CU(dpq::launch_encode_tc(ix->d_cw.as<float>(), M, K, Ds, src, c, D, dst, d_tc.as<unsigned char>(), d_err, n_sms, st));
        else CU(dpq::launch_encode(ix->d_cw.as<float>(), M, K, Ds, src, c, D, dst, st));
        if (!on_dev) CU(cudaStreamSynchronize(st));  // the staging buffer is reused by the next chunk
    }
    if (tc) {
        uint32_t err = 0;
        CU(cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (err) return fail(DPQ_ERR_CUDA, "dpq_index_add_vectors: a tensor-core completion barrier never fired");
    }
    return append_nodes(ix, d_codes.as<uint8_t>(), n, ids, out_pos, t0);
}

// The live nodes of ix in ascending local position, gathered on its stream (compact.cu): *d_codes [n_live][M]
// unpadded, *d_ids [n_live] the id each node reports (pos2id[pos], else its position).  Both are cudaMalloc'ed for
// the caller to free; with no live node both stay null.  Returns once the device work is complete.
static int live_nodes(dpq_index* ix, uint8_t** d_codes, uint32_t** d_ids, int64_t* n_live) {
    *d_codes = nullptr;
    *d_ids = nullptr;
    *n_live = 0;
    const dpq::ScanProgram& P = ix->prog;
    cudaStream_t st = ix->stream;
    const int64_t n = P.n_local, words = (n + 31) / 32;
    int rc;
    if ((rc = upload_pos2id(ix))) return rc;
    const uint32_t* dead = ix->dead();
    Scratch off, codes, ids;  // off: [live offsets words + 1][live counts words + 1][the scan's scratch]
    int64_t count = n;
    if (dead) {
        size_t tmp = 0;
        CU(dpq::count_live(dead, n, nullptr, nullptr, nullptr, &tmp, st));
        const size_t off_bytes = ((size_t)(words + 1) * 4 + 255) / 256 * 256;
        if ((rc = off.b.ensure(2 * off_bytes + tmp))) return rc;
        CU(dpq::count_live(dead, n, reinterpret_cast<uint32_t*>(off.b.as<char>() + off_bytes), off.b.as<uint32_t>(),
                           off.b.as<char>() + 2 * off_bytes, &tmp, st));
        uint32_t c = 0;
        CU(cudaMemcpyAsync(&c, off.b.as<uint32_t>() + words, 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        count = c;
    }
    if (count == 0) return DPQ_OK;
    if ((rc = codes.b.ensure((size_t)count * P.M)) || (rc = ids.b.ensure((size_t)count * 4))) return rc;
    CU(dpq::gather_live(ix->d_codes.as<uint8_t>(), P.cstride, n, P.M, dead, off.b.as<uint32_t>(),
                        ix->has_pos2id ? ix->d_pos2id.as<uint32_t>() : nullptr, (uint32_t)P.base_pos, codes.b.as<uint8_t>(),
                        ids.b.as<uint32_t>(), st));
    CU(cudaStreamSynchronize(st));
    *d_codes = codes.b.as<uint8_t>();
    *d_ids = ids.b.as<uint32_t>();
    codes.b.p = ids.b.p = nullptr;  // handed to the caller
    *n_live = count;
    return DPQ_OK;
}

// Gather the live nodes, build their tree on the device (the edge search and layout of dpq_tree_build_device with
// the defaults of `deltapq -task approx_tree`: -h 1, -method 1), map its vec_id to the carried ids, load it into a
// new index state on the same stream, and only then swap that state in: a failure at any step leaves ix as it was.
int dpq_index_compact(dpq_index* ix, dpq_tree** out_tree) {
    using clk = std::chrono::steady_clock;
    const auto t0 = clk::now();
    auto us = [](clk::time_point a, clk::time_point b) { return (int64_t)std::chrono::duration_cast<std::chrono::microseconds>(b - a).count(); };
    if (out_tree) *out_tree = nullptr;
    int rc = check_device();
    if (rc) return rc;
    if (!ix) return fail(DPQ_ERR_ARG, "dpq_index_compact: null index");
    const dpq::ScanProgram& P = ix->prog;
    if (!P.v2)
        return fail(DPQ_ERR_ARG,
                    "dpq_index_compact: compaction needs the code-array engine (this index runs the first-generation engine, DPQ_ENGINE=1)");
    if (ix->n_ranks > 1)
        return fail(DPQ_ERR_ARG, "dpq_index_compact: this index is one shard of a tree split over several ranks (dpq_multi_compact compacts those)");
    if (!ix->d_cw.p || ix->cw_host.empty()) return fail(DPQ_ERR_ARG, "dpq_index_compact: no codebook (dpq_index_set_codebook first)");
    const int M = P.M, K = P.K;
    CU(cudaSetDevice(ix->device));
    struct Restore {  // the build runs on the thread's selected device, which is the index's for the call's duration
        int d;
        ~Restore() { g_device = d; }
    } restore{g_device};
    g_device = ix->device;
    uint8_t* d_live = nullptr;
    uint32_t* d_ids = nullptr;
    int64_t n_live = 0;
    rc = live_nodes(ix, &d_live, &d_ids, &n_live);
    Scratch live_codes, live_ids;  // released on every return path
    live_codes.b.p = d_live;
    live_ids.b.p = d_ids;
    if (rc) return rc;
    if (n_live == 0) return fail(DPQ_ERR_ARG, "dpq_index_compact: every node is deleted (a tree needs at least one node)");
    const auto t1 = clk::now();
    std::unique_ptr<dpq_tree> t(new dpq_tree());
    t->M = M;
    t->K = K;
    t->n = n_live;
    uint32_t* d_edges = nullptr;
    rc = dpq::find_edges_device(d_live, n_live, M, K, 1, 1, &d_edges, &t->root);
    const auto t2 = clk::now();
    if (!rc) rc = dpq::layout_tree_device(d_live, n_live, M, K, ix->cw_host.data(), ix->Ds, t.get(), d_edges, true, out_tree != nullptr);
    if (d_edges) cudaFree(d_edges);
    const auto t3 = clk::now();
    if (rc) return rc;
    t->edge_us = us(t1, t2);
    t->layout_us = us(t2, t3);
    // the layout ended in a device synchronisation; the new state is filled on the index's stream
    CU(dpq::map_tree_ids(static_cast<uint32_t*>(t->d_vec_id), n_live, d_ids, ix->stream));
    dpq_index* nx = new dpq_index();
    nx->device = ix->device;
    nx->stream = ix->stream;
    nx->own_stream = false;
    rc = load_tree_shard(nx, t.get(), 0, 1, ix->pos_shift);  // ends in a stream synchronisation
    if (!rc && out_tree) {  // the host form dpq_tree_build returns (the QNode fields came with the layout)
        t->vec_id.resize((size_t)n_live);
        t->depth.resize((size_t)n_live);
        t->codes_by_pos.resize((size_t)n_live * M);
        t->payload.resize((size_t)t->payload_bytes);
        if (!(rc = dpq::tree_copy_device(t.get(), t->d_vec_id, t->vec_id.data(), t->vec_id.size() * 4)) &&
            !(rc = dpq::tree_copy_device(t.get(), t->d_depth, t->depth.data(), t->depth.size())) &&
            !(rc = dpq::tree_copy_device(t.get(), t->d_codes_by_pos, t->codes_by_pos.data(), t->codes_by_pos.size())))
            rc = dpq::tree_copy_device(t.get(), t->d_payload, t->payload.data(), t->payload.size());
    }
    if (rc) {
        dpq_index_close(nx);
        return rc;
    }
    // swap: positions renumbered from base_pos, ids carried, tombstones and the appended tail gone
    std::swap(ix->d_codes, nx->d_codes);
    ix->prog = nx->prog;
    ix->pos2id_host.swap(nx->pos2id_host);
    ix->has_pos2id = true;
    ix->n_chunks = nx->n_chunks;
    ix->ops_bytes = nx->ops_bytes;
    ix->d_pos2id.release();  // uploaded again from pos2id_host when a search or a delete needs it
    ix->d_dead.release();
    ix->n_deleted = 0;
    ix->n_added = 0;
    ix->ps_R = 0;  // the presample's nodes were gathered from the old code array
    dpq_index_close(nx);  // frees the old code array
    if (out_tree) {
        dpq::tree_release_device(t.get());
        t->on_device = false;
        *out_tree = t.release();
    }
    const auto t4 = clk::now();
    ix->compact_us[0] = us(t0, t4);
    ix->compact_us[1] = us(t0, t1);
    ix->compact_us[2] = us(t1, t2);
    ix->compact_us[3] = us(t2, t3);
    return DPQ_OK;
}

// slices of a pass over n_chunks chunks for n_groups query groups: whole waves of 148 one-CTA SMs and
// whole rounds (warps x strands chunks) per item, as nearly as possible
static int pick_slices(int n_groups, int n_chunks, int chunks_per_round, int max_slices) {
    double best = -1.0;
    int pick = 1;
    // an item is at least a quarter round: sampled passes are small, and an SM without a CTA costs more than a
    // partly filled round (ncu: the 1/32 sample pass of the wide shape ran on 54 of 148 SMs)
    for (int s = 1; s <= max_slices && s <= std::max(1, 4 * n_chunks / chunks_per_round); ++s) {
        const int64_t items = (int64_t)n_groups * s;
        const int64_t waves = (items + 147) / 148;
        const double cpi = (double)n_chunks / s;
        const double eff = (double)items / (double)(waves * 148) * (cpi / chunks_per_round) / std::ceil(cpi / chunks_per_round);
        if (eff > best + 1e-9) {
            best = eff;
            pick = s;
        }
    }
    return pick;
}

// the presample's node set gathered once per (index, R)
static int ensure_sample_codes(dpq_index* ix, int R) {
    if (ix->ps_R == R && ix->d_ps_codes.p) return DPQ_OK;
    int rc = ix->d_ps_codes.ensure((size_t)R * ix->prog.cstride);
    if (rc) return rc;
    dpq::launch_gather_sample(ix->d_codes.as<uint8_t>(), ix->prog.cstride, ix->prog.n_local, R, ix->d_ps_codes.as<uint8_t>(), ix->stream);
    ix->ps_R = R;
    return DPQ_OK;
}

// Latency mode: exact tables -> exact presample (cap0) -> [scan1 over every S-th chunk -> exact re-score ->
// cap1] -> scan1 over the whole shard -> exact re-score -> exact fallback for overflowed lists.
static int search_latency(dpq_index* ix, const float* d_queries, int Q, int topk, uint64_t* d_out_key) {
    const dpq::ScanProgram& P = ix->prog;
    const size_t MK = (size_t)P.M * P.K;
    const int ccap = 32768;
    int rc;
    if ((rc = ix->d_lutf.ensure((size_t)Q * MK * 4))) return rc;
    if ((rc = ix->d_scale.ensure((size_t)Q * 16 * 4 + 64))) return rc;
    if ((rc = ix->d_cand1.ensure((size_t)Q * ccap * 4))) return rc;
    if ((rc = ix->d_cnt1.ensure((size_t)Q * 8 * 2))) return rc;
    if ((rc = ix->d_cap0.ensure((size_t)Q * 4))) return rc;
    if ((rc = ix->d_cap1.ensure((size_t)Q * 4))) return rc;
    if ((rc = ix->d_flagged.ensure((size_t)Q * 4))) return rc;
    if ((rc = ix->d_bound.ensure((size_t)Q * 4))) return rc;
    if ((rc = ix->d_ctrl.ensure(64))) return rc;
    if ((rc = ix->d_fpart.ensure((size_t)Q * dpq::fallback_slices(topk) * topk * 8))) return rc;
    cudaStream_t st = ix->stream;
    uint32_t* ctrl = ix->d_ctrl.as<uint32_t>();
    {
        const int slot = std::min(ix->timed_calls, 4095);
        while ((int)ix->evs.size() < 6 * (slot + 1)) {
            cudaEvent_t e;
            CU(cudaEventCreate(&e));
            ix->evs.push_back(e);
        }
        ix->ev = ix->evs.data() + 6 * slot;
        ix->timed_calls = slot + 1;
    }
    int launches = 0;
    CU(cudaEventRecord(ix->ev[0], st));
    CU(cudaMemsetAsync(ctrl, 0, 64, st));
    dpq::launch_lut_small(ix->d_cw.as<float>(), P.M, P.K, ix->Ds, d_queries, Q, ix->d_lutf.as<float>(), ix->d_scale.as<float>(), st);
    CU(cudaEventRecord(ix->ev[1], st));
    float* cap0 = ix->d_cap0.as<float>();
    float* cap1 = ix->d_cap1.as<float>();
    if ((rc = ensure_sample_codes(ix, 2048))) return rc;
    dpq::launch_presample(ix->d_lutf.as<float>(), ix->d_ps_codes.as<uint8_t>(), P.cstride, P.n_local, P.M, P.K, Q, topk, 2048, cap0,
                          ix->dead(), st);
    launches += 2;
    uint32_t* cnt = ix->d_cnt1.as<uint32_t>();  // [0..Q) counts, [Q..2Q) overflow flags; a second pair behind for the final pass
    dpq::Scan1Args s1;
    s1.codes = ix->d_codes.as<uint8_t>();
    s1.n_local = P.n_local;
    s1.base_pos = (uint32_t)P.base_pos;
    s1.lutf = ix->d_lutf.as<float>();
    s1.mmax = ix->d_scale.as<float>();
    s1.M = P.M;
    s1.K = P.K;
    s1.Q = Q;
    s1.n_pairs = (Q + 1) / 2;
    s1.cand = ix->d_cand1.as<uint32_t>();
    s1.ccap = ccap;
    s1.dead = ix->dead();
    dpq::Rescore1Args r1;
    r1.cand = s1.cand;
    r1.ccap = ccap;
    r1.lutf = s1.lutf;
    r1.codes = s1.codes;
    r1.cstride = P.cstride;
    r1.base_pos = P.base_pos;
    r1.M = P.M;
    r1.K = P.K;
    r1.Q = Q;
    r1.topk = topk;
    r1.n_parts = std::max(1, std::min(16, 2048 / topk));
    {
        if ((rc = ix->d_part8.ensure((size_t)Q * r1.n_parts * topk * 8))) return rc;
        const bool fresh = ix->d_done8.cap < (size_t)Q * 4;
        if ((rc = ix->d_done8.ensure((size_t)Q * 4))) return rc;
        if (fresh) CU(cudaMemsetAsync(ix->d_done8.p, 0, ix->d_done8.cap, st));
    }
    r1.part = ix->d_part8.as<uint64_t>();
    r1.part_done = ix->d_done8.as<uint32_t>();
    const int64_t n_chunks = (P.n_local + 2047) / 2048;
    auto ranges_for = [&](int64_t chunks) { return (int)std::max<int64_t>(1, std::min<int64_t>(chunks, 148 / s1.n_pairs)); };
    CU(cudaMemsetAsync(cnt, 0, (size_t)Q * 16, st));
    const float* cap = cap0;
    // presample: k-th of 2048 nodes -> about topk * n / 2048 nodes under cap0; a first pass over every S-th
    // chunk (about a million nodes) tightens the cap when the whole shard would overflow the candidate lists
    if ((double)P.n_local / 2048.0 * topk > ccap / 4) {
        const int S = (int)std::max<int64_t>(2, P.n_local >> 20);
        s1.chunk_stride = S;
        s1.cap = cap0;
        s1.cand_cnt = cnt;
        s1.ovf = cnt + Q;
        s1.n_ranges = ranges_for((n_chunks + S - 1) / S);
        CU(dpq::launch_scan1(s1, st));
        r1.cand_cnt = s1.cand_cnt;
        r1.ovf = s1.ovf;
        r1.out_key = nullptr;
        r1.cap_in = cap0;
        r1.cap_out = cap1;
        r1.flagged = nullptr;
        r1.n_flagged = nullptr;
        r1.max_flagged = 0;
        r1.bound = nullptr;
        dpq::launch_rescore1(r1, st);
        launches += 2;
        cap = cap1;
    }
    s1.chunk_stride = 1;
    s1.cap = cap;
    s1.cand_cnt = cnt + 2 * Q;
    s1.ovf = cnt + 3 * Q;
    s1.n_ranges = ranges_for(n_chunks);
    CU(cudaEventRecord(ix->ev[4], st));
    CU(dpq::launch_scan1(s1, st));
    CU(cudaEventRecord(ix->ev[5], st));
    r1.cand_cnt = s1.cand_cnt;
    r1.ovf = s1.ovf;
    r1.out_key = d_out_key;
    r1.cap_in = cap;
    r1.cap_out = nullptr;
    r1.flagged = ix->d_flagged.as<uint32_t>();
    r1.n_flagged = ctrl + 2;
    r1.max_flagged = Q;
    r1.bound = ix->d_bound.as<float>();
    dpq::launch_rescore1(r1, st);
    CU(cudaEventRecord(ix->ev[2], st));
    dpq::FallbackArgs fb;
    fb.flagged = r1.flagged;
    fb.n_flagged = ctrl + 2;
    fb.max_flagged = Q;
    fb.lutf = s1.lutf;
    fb.bound = r1.bound;
    fb.codes = s1.codes;
    fb.cstride = P.cstride;
    fb.base_pos = P.base_pos;
    fb.n_local = P.n_local;
    fb.M = P.M;
    fb.K = P.K;
    fb.topk = topk;
    fb.part = ix->d_fpart.as<uint64_t>();
    fb.out_key = d_out_key;
    fb.dead = ix->dead();
    dpq::launch_fallback(fb, st);
    launches += 4;
    CU(cudaEventRecord(ix->ev[3], st));
    CU(cudaGetLastError());
    ix->last_launches = launches;
    ix->last_coarse = 0;
    ix->last_latency = 1;
    ix->last_device_queries = Q;
    ix->timing_valid = true;
    return DPQ_OK;
}

int dpq_index_search_device(dpq_index* ix, const float* d_queries, int Q, int topk,
                            uint64_t* d_out_key) {
    if (!ix || !d_queries || !d_out_key) return fail(DPQ_ERR_ARG, "dpq_index_search: null argument");
    if (Q < 1 || topk < 1) return fail(DPQ_ERR_ARG, "dpq_index_search: Q and topk must be >= 1");
    if (ix->Ds < 1) return fail(DPQ_ERR_ARG, "dpq_index_search: codebook not set");
    CU(cudaSetDevice(ix->device));
    dpq::ScanGeom g;
    const dpq::ScanProgram& P = ix->prog;
    {   // latency mode (scan1.cu): a handful of queries, lanes = nodes, the code array streams once per query pair
        const bool can = P.v2 && P.shape.nf == 8 && Q <= 16 && topk <= 32;
        const bool auto_on = P.n_local >= 4096 && (double)P.n_local * topk <= 6e9;
        ix->last_latency = 0;
        if (can && ix->opt_latency != 0 && !ix->opt_force_fallback && (ix->opt_latency == 1 || auto_on))
            return search_latency(ix, d_queries, Q, topk, d_out_key);
    }
    // coarse search (scan8.cu): 15-bit scan over a 1/S sample -> cap per query -> 8-bit scan of
    // the whole tree -> exact re-score.  Trees large enough to pay, result lists up to 128.
    const bool coarse_auto = P.n_local >= ix->opt_coarse_min && topk <= (P.shape.nf == 8 ? 64 : 128);
    const bool coarse = P.v2 && topk <= 128 && ix->opt_coarse != 0 && (ix->opt_coarse == 1 || coarse_auto);
    const dpq::C8Shape c8 = dpq::c8_shape(P.shape.nf);  // 112 queries per CTA in both shapes
    const int spw = P.shape.spw();
    const int levels8 = std::min(ix->opt_levels8, 127 - c8.slack);  // the test constant stays <= 128
    // sample stride: a sparser sample is cheaper to scan but gives a looser cap (more coarse survivors to
    // re-score).  Measured optimum: 32 at 1M nodes (+2 % over 16; 64 is slower), 64 at 125M nodes (+9 %;
    // 256 overflows candidate lists): the sample keeps at least ~30K nodes (gpurun_out/b_opt.json runs).
    int S_auto = P.n_local >= 2000000 ? 64 : (P.n_local >= 1000000 ? 32 : (P.n_local >= 400000 ? 16 : 8));
    // wide shape, short lists: a denser sample (1M codes, M = 16, top-10: 2.42 ms at 16 vs 2.8 ms at 32)
    if (P.shape.nf == 16 && topk <= 32 && S_auto > 16 && P.n_local < 2000000) S_auto = 16;
    // Large shards, seeded pipeline: a 1/64 sample of 10^8..10^9 nodes is millions of nodes, far too many to scan
    // under the presample's loose cap (0.5 % quantile: tens of thousands of survivors per query, appended and
    // re-scored: 0.36 s of a 1.10 s step on a 250M-node shard).  Two levels instead: a ~64K-node sample under
    // the presample cap, then the 1/64 sample under THAT cap (the refine pass below), then the whole shard.
    int S_big = 0;
    if (coarse && ix->opt_seed != 0 && ix->opt_sample == 0 && ix->opt_refine < 0 && P.n_local / 64 > 262144) {
        S_big = 128;
        while (S_big < 16384 && P.n_local / S_big > 98304) S_big <<= 1;
    }
    const int S = !coarse ? 1 : (ix->opt_sample > 0 ? ix->opt_sample : (S_big ? S_big : S_auto));
    const int n_chunks_sample = (((ix->n_chunks + spw - 1) / spw + S - 1) / S) * spw;  // chunks the sample pass walks
    int rc = P.v2 ? choose_geometry2(ix, Q, topk, &g, coarse ? n_chunks_sample : -1) : choose_geometry(ix, Q, topk, &g);
    if (rc) return rc;
    ix->last_coarse = coarse ? 1 : 0;
    ix->last_sample_stride = coarse ? S : 0;
    ix->last_device_queries = Q;
    // geometry of the coarse passes: 112-query groups, 4 strands per warp
    const int warps8 = ix->opt_warps8;
    const int bcap8 = ix->opt_bcap8 > 0 ? ix->opt_bcap8 : (P.shape.nf == 8 ? 512 : 4096);  // survivors per (slice, query)
    // the sample pass is a coarse scan seeded by an exact presample (default: 4.20 vs 4.28 ms per step at C2 once
    // the re-score and presample kernels fetched codes with vector loads); seed=0 keeps the 15-bit sample pass
    const bool seeded = coarse && ix->opt_seed != 0;
    const int n_chunks_sample8 = (((ix->n_chunks + 3) / 4 + S - 1) / S) * 4;
    // second refinement level: a denser sampled coarse pass (stride S2 < S) under the first cap.  Long result
    // lists need it: the cap of a 1/S sample is about the (k S)-th distance of the tree, and the coarse filter
    // passes a multiple of that many nodes (26K survivors per query at top-100, S = 32, M = 16).
    int S2 = ix->opt_refine >= 0 ? ix->opt_refine : (S_big ? 64 : (P.shape.nf == 16 && topk > 32 ? 8 : 0));
    if (!coarse || S2 < 2 || S2 >= S) S2 = 0;
    ix->last_refine_stride = S2;
    const int n_chunks_refine8 = S2 ? (((ix->n_chunks + 3) / 4 + S2 - 1) / S2) * 4 : 0;
    int g8_groups = 0, g8_slices = 1, g8_slices_s = 1, g8_slices_r = 1;
    if (coarse) {
        g8_groups = (Q + c8.qb - 1) / c8.qb;
        g8_slices = ix->opt_slices > 0 ? ix->opt_slices : pick_slices(g8_groups, ix->n_chunks, warps8 * 4, 96);
        g8_slices = std::max(1, std::min(std::min(g8_slices, 128), std::max(1, ix->n_chunks)));  // <= R8_MAXSL
        if (seeded) g8_slices_s = pick_slices(g8_groups, n_chunks_sample8, warps8 * 4, 96);
        if (S2) g8_slices_r = pick_slices(g8_groups, n_chunks_refine8, warps8 * 4, 96);
    }
    // exact re-score: CTAs per query.  Long lists / the wide shape have thousands of survivors per query with a
    // heavy tail: several CTAs per query (ranges of slices) and a last-arrival merge
    const int r8_parts = !coarse ? 1 : (ix->opt_parts8 > 0 ? ix->opt_parts8 : ((P.shape.nf == 16 || topk > 32) ? 8 : 1));
    const size_t MK = (size_t)P.M * P.K;
    const size_t rows = (size_t)1 << g.rb;
    const size_t LW = 32 * (size_t)g.pack;
    const size_t n_items = (size_t)g.n_groups * g.n_slices;
    const int max_flagged = Q;
    if ((rc = ix->d_lutf.ensure((size_t)Q * MK * 4))) return rc;
    // [padded Q] doubles (15-bit scale), then [Q][16] floats (per-subspace table maxima)
    const size_t scale_bytes = (size_t)g.n_groups * g.qpg * 8;
    if ((rc = ix->d_scale.ensure(scale_bytes + (size_t)Q * 16 * 4))) return rc;
    if (P.v2) {
        if ((rc = ix->d_cand.ensure(n_items * g.qpg * g.bcap * 8))) return rc;
        if ((rc = ix->d_cnt.ensure(n_items * g.qpg * 4))) return rc;
        if ((rc = ix->d_ovf.ensure((size_t)g.n_groups * g.qpg * 4))) return rc;
        if ((rc = ix->d_qlut.ensure((size_t)g.n_groups * P.shape.lut_bytes()))) return rc;
    } else {
        if ((rc = ix->d_qlut.ensure((size_t)g.n_groups * g.qgl * rows * 4))) return rc;
        if ((rc = ix->d_cand.ensure(n_items * g.n_warps * g.bcap * LW * 8))) return rc;
        if ((rc = ix->d_cnt.ensure(n_items * g.n_warps * LW * 4))) return rc;
        if ((rc = ix->d_ovf.ensure(16))) return rc;
    }
    if ((rc = ix->d_gthr.ensure((size_t)g.n_groups * g.qpg * 4))) return rc;
    if ((rc = ix->d_flagged.ensure((size_t)max_flagged * 4))) return rc;
    if ((rc = ix->d_ctrl.ensure(64))) return rc;
    if ((rc = ix->d_bound.ensure((size_t)Q * 4))) return rc;
    if ((rc = ix->d_fpart.ensure((size_t)max_flagged * dpq::fallback_slices(topk) * topk * 8))) return rc;
    if (coarse) {
        const size_t items8 = (size_t)g8_groups * std::max(std::max(g8_slices, g8_slices_s), g8_slices_r);
        ix->last_items8 = (int64_t)g8_groups * g8_slices;
        if ((rc = ix->d_cap0.ensure((size_t)Q * 4))) return rc;
        if ((rc = ix->d_cap1.ensure((size_t)Q * 4))) return rc;
        if ((rc = ix->d_qlut8.ensure((size_t)g8_groups * c8.lut_bytes()))) return rc;
        if ((rc = ix->d_cand8.ensure(items8 * c8.qb * bcap8 * 4))) return rc;
        if ((rc = ix->d_cnt8.ensure(items8 * c8.qb * 4))) return rc;
        if ((rc = ix->d_ovf8.ensure((size_t)g8_groups * c8.qb * 4))) return rc;
        if ((rc = ix->d_flagged2.ensure((size_t)max_flagged * 4))) return rc;
        if (!ix->sm_slots8) CU(dpq::scan8_sm_slots(ix->d_flagged2.as<int>(), &ix->sm_slots8, ix->stream));
        if ((rc = ix->d_stage8.ensure((size_t)ix->sm_slots8 * 24 * ix->opt_stage8 * 8))) return rc;
        if (r8_parts > 1) {
            if ((rc = ix->d_part8.ensure((size_t)Q * r8_parts * topk * 8))) return rc;
            const bool fresh = ix->d_done8.cap < (size_t)Q * 4;
            if ((rc = ix->d_done8.ensure((size_t)Q * 4))) return rc;
            if (fresh) CU(cudaMemsetAsync(ix->d_done8.p, 0, ix->d_done8.cap, ix->stream));  // counters reset themselves afterwards
        }
    }
    cudaStream_t st = ix->stream;
    // ctrl words: [0] queries flagged by select_kernel, [2] by the final rescore8_kernel,
    // [3] scratch (flags of the sample phase of the coarse search, which needs no fallback)
    uint32_t* ctrl = ix->d_ctrl.as<uint32_t>();
    {
        const int slot = std::min(ix->timed_calls, 4095);
        while ((int)ix->evs.size() < 6 * (slot + 1)) {
            cudaEvent_t e;
            CU(cudaEventCreate(&e));
            ix->evs.push_back(e);
        }
        ix->ev = ix->evs.data() + 6 * slot;
        ix->timed_calls = slot + 1;
    }
    int launches = 0;
    CU(cudaEventRecord(ix->ev[0], st));
    CU(cudaMemsetAsync(ctrl, 0, 64, st));
    if (P.v2) {
        dpq::launch_lut2(ix->d_cw.as<float>(), P.M, P.K, ix->Ds, d_queries, Q, ix->d_lutf.as<float>(),
                         ix->d_scale.as<double>(), reinterpret_cast<float*>(ix->d_scale.as<char>() + scale_bytes),
                         seeded ? nullptr : ix->d_qlut.as<uint16_t>(),
                         ix->d_gthr.as<uint32_t>(), ix->d_ovf.as<uint32_t>(), g.n_groups, P.shape,
                         (uint32_t)ix->opt_dbg_bound, st);
        launches += seeded ? 1 : 3;
    } else {
        dpq::launch_lut(ix->d_cw.as<float>(), P.M, P.K, ix->Ds, d_queries, Q, ix->d_lutf.as<float>(),
                        ix->d_scale.as<double>(), ix->d_qlut.as<uint32_t>(), ix->d_gthr.as<uint32_t>(), g, st);
        launches += 1;
    }
    dpq::ScanArgs sa;
    sa.g = g;
    sa.ops = ix->d_ops.as<uint4>();
    sa.chunks = ix->d_chunks.as<dpq::ChunkDesc>();
    sa.anc = ix->d_anc.as<uint8_t>();
    sa.n_chunks = ix->n_chunks;
    sa.qlut = ix->d_qlut.as<uint32_t>();
    sa.cand = ix->d_cand.as<uint64_t>();
    sa.cand_cnt = ix->d_cnt.as<uint32_t>();
    sa.gthr = ix->d_gthr.as<uint32_t>();
    sa.Q = Q;
    CU(cudaEventRecord(ix->ev[1], st));
    if (P.v2 && !seeded) {
        dpq::Scan2Args s2;
        s2.shape = P.shape;
        s2.codes = ix->d_codes.as<uint8_t>();
        s2.n_local = P.n_local;
        s2.base_pos = (uint32_t)P.base_pos;
        s2.n_chunks = ix->n_chunks;
        s2.chunk_nodes = P.v2_chunk_nodes;
        s2.bt_stride = S;
        s2.qlut = ix->d_qlut.as<uint16_t>();
        s2.cand = sa.cand;
        s2.cand_cnt = sa.cand_cnt;
        s2.gthr = sa.gthr;
        s2.ovf = ix->d_ovf.as<uint32_t>();
        s2.Q = Q;
        s2.n_groups = g.n_groups;
        s2.n_slices = g.n_slices;
        s2.n_warps = g.n_warps;
        s2.kp = g.kp;
        s2.bcap = g.bcap;
        s2.trigger = ix->opt_trigger > 0 ? std::min(ix->opt_trigger, g.bcap / 2) : std::min(2 * g.kp, g.bcap / 2);
        s2.epoch = std::max(1, ix->opt_epoch);
        s2.ramp = ix->opt_ramp;
        s2.dead = ix->dead();
        CU(dpq::launch_scan2(s2, st));
        ++launches;
    } else if (!seeded) {
        CU(dpq::launch_scan(sa, st));
        ++launches;
    }
    if (!coarse) CU(cudaEventRecord(ix->ev[2], st));
    float* cap0 = ix->d_cap0.as<float>();
    float* cap1 = ix->d_cap1.as<float>();
    dpq::SelectArgs se;
    se.g = g;
    se.v2 = P.v2 ? 1 : 0;
    se.ovf = ix->d_ovf.as<uint32_t>();
    se.cand = sa.cand;
    se.cand_cnt = sa.cand_cnt;
    se.lutf = ix->d_lutf.as<float>();
    se.scale = ix->d_scale.as<double>();
    se.codes = ix->d_codes.as<uint8_t>();
    se.cstride = P.cstride;
    se.base_pos = P.base_pos;
    se.n_local = P.n_local;
    se.Q = Q;
    se.topk = topk;
    se.out_key = d_out_key;
    se.flagged = ix->d_flagged.as<uint32_t>();
    se.max_flagged = max_flagged;
    se.force_fallback = ix->opt_force_fallback;
    // Coarse search: the sample pass only has to deliver a valid cap >= the true k-th distance, and
    // select_kernel's bound[q] -- the exact k-th distance among the re-scored sample nodes, which are
    // real nodes of the tree -- already is one (FLT_MAX when the sample held fewer than k nodes).  Its
    // proof-failure / overflow flags concern the exactness of the SAMPLE's top-k only and are ignored.
    se.n_flagged = coarse ? ctrl + 3 : ctrl;
    se.bound = coarse ? cap1 : ix->d_bound.as<float>();
    if (!seeded) {
        dpq::launch_select(se, st);
        ++launches;
    }
    dpq::FallbackArgs fa;
    fa.flagged = se.flagged;
    fa.n_flagged = ctrl;
    fa.max_flagged = max_flagged;
    fa.lutf = se.lutf;
    fa.bound = ix->d_bound.as<float>();
    fa.codes = se.codes;
    fa.cstride = P.cstride;
    fa.base_pos = P.base_pos;
    fa.n_local = P.n_local;
    fa.M = P.M;
    fa.K = P.K;
    fa.topk = topk;
    fa.part = ix->d_fpart.as<uint64_t>();
    fa.out_key = d_out_key;
    fa.dead = ix->dead();
    if (!coarse) {
        dpq::launch_fallback(fa, st);
        launches += 2;
    } else {
        dpq::Scan8Args s8;
        s8.codes = ix->d_codes.as<uint8_t>();
        s8.n_local = P.n_local;
        s8.base_pos = (uint32_t)P.base_pos;
        s8.n_chunks = ix->n_chunks;
        s8.chunk_nodes = P.v2_chunk_nodes;
        s8.qlut8 = ix->d_qlut8.as<uint8_t>();
        s8.cand = ix->d_cand8.as<uint32_t>();
        s8.cand_cnt = ix->d_cnt8.as<uint32_t>();
        s8.ovf = ix->d_ovf8.as<uint32_t>();
        s8.Q = Q;
        s8.n_groups = g8_groups;
        s8.n_warps = warps8;
        s8.bcap = bcap8;
        s8.thresh = levels8 + c8.slack + 1;
        s8.nf = c8.nf;
        s8.reuse = ix->opt_reuse8;
        s8.dead = ix->dead();
        s8.stage = ix->d_stage8.as<uint2>();
        s8.stage_cap = ix->opt_stage8;
        dpq::Rescore8Args r8;
        r8.cand = s8.cand;
        r8.cand_cnt = s8.cand_cnt;
        r8.ovf = s8.ovf;
        r8.n_groups = g8_groups;
        r8.bcap = bcap8;
        r8.qb = c8.qb;
        r8.lutf = se.lutf;
        r8.codes = se.codes;
        r8.cstride = P.cstride;
        r8.base_pos = P.base_pos;
        r8.M = P.M;
        r8.K = P.K;
        r8.Q = Q;
        r8.topk = topk;
        r8.part = ix->d_part8.as<uint64_t>();
        r8.part_done = ix->d_done8.as<uint32_t>();
        r8.warp_form = ix->opt_warp_rescore >= 0 ? ix->opt_warp_rescore : (P.shape.nf == 8 ? 1 : 0);
        auto parts_for = [&](int slices) { return std::max(1, std::min(std::min(r8_parts, slices), std::max(1, 2048 / topk))); };
        if (seeded) {
            // cap0: exact k-th distance over a small strided set of nodes -> coarse scan of the
            // sample (every S-th batch) -> exact re-score -> cap1 = the sample's k-th distance
            const int R = ix->opt_presample > 0 ? ix->opt_presample : (topk > 32 ? 4096 : 2048);
            if ((rc = ensure_sample_codes(ix, R))) return rc;
            dpq::launch_presample(se.lutf, ix->d_ps_codes.as<uint8_t>(), P.cstride, P.n_local, P.M, P.K, Q, topk, R, cap0, ix->dead(), st);
            // The first sampled pass only has to FIND k nodes below the presample cap, not all of them: quantising
            // with levels8 * 100 / stight levels per cap while the test constant stays at levels8 accepts distances
            // up to ~stight % of cap0 -- fewer survivors to append and re-score.  A query whose sample holds fewer than
            // k such nodes keeps cap0 (valid, looser).
            dpq::launch_pack8(se.lutf, cap0, P.M, P.K, Q, levels8 * 100 / ix->opt_stight, ix->d_qlut8.as<uint8_t>(), s8.ovf, g8_groups,
                              c8.nf, st);
            s8.bt_stride = S;
            s8.n_slices = g8_slices_s;
            CU(dpq::launch_scan8(s8, st));
            r8.n_slices = g8_slices_s;
            r8.n_parts = parts_for(g8_slices_s);
            r8.out_key = nullptr;
            r8.cap_in = cap0;
            r8.cap_out = cap1;
            r8.flagged = nullptr;
            r8.n_flagged = nullptr;
            r8.max_flagged = 0;
            r8.bound = nullptr;
            dpq::launch_rescore8(r8, st);
            launches += 4;
        }
        const float* cap = cap1;
        if (S2) {  // cap1 -> coarse scan of every S2-th batch -> exact re-score -> cap2 (kept in the cap0 buffer)
            dpq::launch_pack8(se.lutf, cap1, P.M, P.K, Q, levels8, ix->d_qlut8.as<uint8_t>(), s8.ovf, g8_groups, c8.nf, st);
            s8.bt_stride = S2;
            s8.n_slices = g8_slices_r;
            CU(dpq::launch_scan8(s8, st));
            r8.n_slices = g8_slices_r;
            r8.n_parts = parts_for(g8_slices_r);
            r8.out_key = nullptr;
            r8.cap_in = cap1;
            r8.cap_out = cap0;
            r8.flagged = nullptr;
            r8.n_flagged = nullptr;
            r8.max_flagged = 0;
            r8.bound = nullptr;
            dpq::launch_rescore8(r8, st);
            launches += 3;
            cap = cap0;
        }
        dpq::launch_pack8(se.lutf, cap, P.M, P.K, Q, levels8, ix->d_qlut8.as<uint8_t>(), s8.ovf, g8_groups, c8.nf, st);
        s8.bt_stride = 1;
        s8.n_slices = g8_slices;
        CU(cudaEventRecord(ix->ev[4], st));
        CU(dpq::launch_scan8(s8, st));
        CU(cudaEventRecord(ix->ev[5], st));
        r8.n_slices = g8_slices;
        r8.n_parts = parts_for(g8_slices);
        r8.out_key = d_out_key;
        r8.cap_in = cap;
        r8.cap_out = nullptr;
        r8.flagged = ix->d_flagged2.as<uint32_t>();
        r8.n_flagged = ctrl + 2;
        r8.max_flagged = max_flagged;
        r8.bound = ix->d_bound.as<float>();
        dpq::launch_rescore8(r8, st);
        CU(cudaEventRecord(ix->ev[2], st));
        dpq::FallbackArgs fb = fa;
        fb.flagged = r8.flagged;
        fb.n_flagged = ctrl + 2;
        dpq::launch_fallback(fb, st);
        launches += 5;
    }
    CU(cudaEventRecord(ix->ev[3], st));
    CU(cudaGetLastError());
    ix->last_launches = launches;
    ix->timing_valid = true;
    return DPQ_OK;
}

int dpq_index_sync(dpq_index* ix) {
    if (!ix) return fail(DPQ_ERR_ARG, "dpq_index_sync: null");
    CU(cudaSetDevice(ix->device));
    CU(cudaStreamSynchronize(ix->stream));
    if (ix->d_ctrl.p) {
        uint32_t ctrl[4] = {0, 0, 0, 0};
        CU(cudaMemcpy(ctrl, ix->d_ctrl.p, 16, cudaMemcpyDeviceToHost));
        ix->last_fallback = (int64_t)ctrl[0] + ctrl[2];
    }
    return DPQ_OK;
}

int dpq_index_search(dpq_index* ix, const float* queries, int Q, int topk, uint32_t* out_pos,
                     uint32_t* out_id, float* out_dist) {
    if (!ix || !queries) return fail(DPQ_ERR_ARG, "dpq_index_search: null argument");
    if (Q < 1 || topk < 1) return fail(DPQ_ERR_ARG, "dpq_index_search: Q and topk must be >= 1");
    CU(cudaSetDevice(ix->device));
    const size_t D = (size_t)ix->prog.M * ix->Ds;
    constexpr int kMaxBatch = 32768;  // bounds the per-search scratch (float tables: 8 KB per query at M = 8)
    if (Q > kMaxBatch) {
        int64_t fb = 0;
        for (int q0 = 0; q0 < Q; q0 += kMaxBatch) {
            const int n = std::min(kMaxBatch, Q - q0);
            const size_t o = (size_t)q0 * topk;
            int rc = dpq_index_search(ix, queries + (size_t)q0 * D, n, topk, out_pos ? out_pos + o : nullptr,
                                      out_id ? out_id + o : nullptr, out_dist ? out_dist + o : nullptr);
            if (rc) return rc;
            fb += ix->last_fallback;
        }
        ix->last_fallback = fb;
        return DPQ_OK;
    }
    const size_t qbytes = (size_t)Q * D * 4, nk = (size_t)Q * topk, kbytes = nk * 8;
    // pinned, device-mapped staging: [queries][pos][id][dist][ctrl words]; a caller buffer that is
    // already page-locked (dpq_malloc_host, cudaHostRegister) is read directly
    const size_t need = qbytes + 3 * nk * 4 + 256;
    if (ix->h_stage_cap < need) {
        if (ix->h_stage) cudaFreeHost(ix->h_stage);
        ix->h_stage = nullptr;
        ix->h_stage_cap = 0;
        CU(cudaHostAlloc(&ix->h_stage, need, cudaHostAllocMapped));
        ix->h_stage_cap = need;
    }
    int rc;
    const auto t_begin = std::chrono::steady_clock::now();
    float* hq = reinterpret_cast<float*>(ix->h_stage);
    uint32_t* h_pos = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ix->h_stage) + qbytes);
    uint32_t* h_id = h_pos + nk;
    uint32_t* h_dist = h_id + nk;
    uint32_t* hc = h_dist + nk;
    // No copy engine in the way: the kernels read the queries from page-locked HOST memory through its
    // device mapping (unified addressing) -- the ADC-table kernel pulls each query's D floats over PCIe
    // exactly once while it computes -- and unpack_kernel writes positions, ids (pos2id lives on the
    // device) and distances straight into the mapped staging buffer.  ONE stream synchronisation, then
    // three sequential copies into the caller's arrays.  (The sub-batch pipeline H2D || search || D2H on
    // two streams lost more to four small searches than the overlap won; the id translation on the host
    // was a 100K-element random gather: 0.2-0.45 ms per 10K x 10 results.)
    void* dq = nullptr;
    cudaPointerAttributes pa;
    const bool pinned = cudaPointerGetAttributes(&pa, queries) == cudaSuccess && pa.type == cudaMemoryTypeHost &&
                        cudaHostGetDevicePointer(&dq, const_cast<float*>(queries), 0) == cudaSuccess && dq;
    (void)cudaGetLastError();
    if (!pinned) {
        memcpy(hq, queries, qbytes);
        CU(cudaHostGetDevicePointer(&dq, hq, 0));
    }
    // result arrays: a caller array that is page-locked is written by the kernel itself (no staging, no
    // copy afterwards); the others go through the mapped staging buffer
    auto mapped = [&](void* host) -> uint32_t* {
        if (!host) return nullptr;
        void* d = nullptr;
        cudaPointerAttributes at;
        const bool ok = cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost &&
                        cudaHostGetDevicePointer(&d, host, 0) == cudaSuccess && d;
        (void)cudaGetLastError();
        return ok ? reinterpret_cast<uint32_t*>(d) : nullptr;
    };
    void* d_stage_out = nullptr;
    CU(cudaHostGetDevicePointer(&d_stage_out, h_pos, 0));
    uint32_t* const ds = reinterpret_cast<uint32_t*>(d_stage_out);
    uint32_t* const o_pos = mapped(out_pos);
    uint32_t* const o_id = mapped(out_id);
    uint32_t* const o_dist = mapped(out_dist);
    if ((rc = ix->d_key.ensure(kbytes))) return rc;
    const bool want_id = out_id != nullptr;
    if (want_id && (rc = upload_pos2id(ix))) return rc;
    rc = dpq_index_search_device(ix, reinterpret_cast<const float*>(dq), Q, topk, ix->d_key.as<uint64_t>());
    if (rc) return rc;
    dpq::launch_unpack(ix->d_key.as<uint64_t>(), nk, want_id && ix->has_pos2id ? ix->d_pos2id.as<uint32_t>() : nullptr,
                       (uint32_t)ix->prog.base_pos, out_pos ? (o_pos ? o_pos : ds) : nullptr,
                       out_id ? (o_id ? o_id : ds + nk) : nullptr, out_dist ? (o_dist ? o_dist : ds + 2 * nk) : nullptr,
                       ix->d_ctrl.p ? ix->d_ctrl.as<uint32_t>() : nullptr, ds + 3 * nk, ix->stream);
    CU(cudaGetLastError());
    const auto t_enq = std::chrono::steady_clock::now();
    CU(cudaStreamSynchronize(ix->stream));  // the one host sync of the call
    const auto t_sync = std::chrono::steady_clock::now();
    ix->last_fallback = (int64_t)hc[0] + hc[2];
    if (out_pos && !o_pos) memcpy(out_pos, h_pos, nk * 4);
    if (out_id && !o_id) memcpy(out_id, h_id, nk * 4);
    if (out_dist && !o_dist) memcpy(out_dist, h_dist, nk * 4);
    const auto t_end = std::chrono::steady_clock::now();
    auto us = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return (int64_t)std::chrono::duration_cast<std::chrono::microseconds>(b - a).count();
    };
    ix->host_us[0] = us(t_begin, t_enq);
    ix->host_us[1] = us(t_enq, t_sync);
    ix->host_us[2] = us(t_sync, t_end);
    return DPQ_OK;
}

int dpq_merge_topk_device(dpq_index* ix, const uint64_t* d_keys, int n_lists, int Q, int topk,
                          uint64_t* d_out_key) {
    if (!ix || !d_keys || !d_out_key) return fail(DPQ_ERR_ARG, "dpq_merge_topk_device: null");
    if (n_lists < 1 || n_lists > 64) return fail(DPQ_ERR_ARG, "dpq_merge_topk_device: 1..64 lists");
    CU(cudaSetDevice(ix->device));
    dpq::launch_merge(d_keys, n_lists, Q, topk, d_out_key, ix->stream);
    CU(cudaGetLastError());
    return DPQ_OK;
}

int dpq_malloc(void** dptr, size_t bytes) {
    if (!dptr) return fail(DPQ_ERR_ARG, "dpq_malloc: null");
    int rc = check_device();
    if (rc) return rc;
    CU(cudaSetDevice(g_device));
    CU(cudaMalloc(dptr, bytes));
    return DPQ_OK;
}
int dpq_free(void* dptr) {
    CU(cudaFree(dptr));
    return DPQ_OK;
}
int dpq_memcpy_h2d(void* dst, const void* src, size_t bytes) {
    CU(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    return DPQ_OK;
}
int dpq_memcpy_d2h(void* dst, const void* src, size_t bytes) {
    CU(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return DPQ_OK;
}
int dpq_malloc_host(void** hptr, size_t bytes) {
    if (!hptr) return fail(DPQ_ERR_ARG, "dpq_malloc_host: null");
    int rc = check_device();
    if (rc) return rc;
    CU(cudaMallocHost(hptr, bytes));
    return DPQ_OK;
}
int dpq_free_host(void* hptr) {
    CU(cudaFreeHost(hptr));
    return DPQ_OK;
}

int64_t dpq_index_stat(dpq_index* ix, const char* name) {
    if (!ix || !name) return -1;
    std::string n(name);
    const dpq::ScanProgram& P = ix->prog;
    if (n == "n_codes") return P.n_codes;
    if (n == "n_bytes") return P.local_bytes;
    if (n == "n_bytes_total") return P.n_bytes;
    if (n == "n_local") return P.n_local;
    if (n == "base_pos") return P.base_pos;
    if (n == "n_diffs") return P.n_diffs;
    if (n == "n_chunks") return ix->n_chunks;
    if (n == "ops_bytes") return (int64_t)ix->ops_bytes;
    if (n == "last_launches") return ix->last_launches;
    if (n == "engine") return P.v2 ? 2 : 1;
    if (n == "last_coarse") return ix->last_coarse;
    if (n == "last_sample_stride") return ix->last_sample_stride;
    if (n == "last_refine_stride") return ix->last_refine_stride;
    if (n == "last_latency") return ix->last_latency;
    if (n == "last_host_enqueue_us") return ix->host_us[0];
    if (n == "last_host_wait_us") return ix->host_us[1];
    if (n == "last_host_unpack_us") return ix->host_us[2];
    if (n == "last_device_queries") return ix->last_device_queries;
    if (n == "cand8_total") {  // developer statistic: coarse survivors of the last search
        if (!ix->last_coarse || !ix->d_cnt8.p) return -1;
        cudaSetDevice(ix->device);
        std::vector<uint32_t> c(ix->d_cnt8.cap / 4);
        if (cudaStreamSynchronize(ix->stream) != cudaSuccess) return -1;
        if (cudaMemcpy(c.data(), ix->d_cnt8.p, c.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
        int64_t t = 0;
        for (size_t i = 0; i < (size_t)ix->last_items8 * dpq::c8_shape(P.shape.nf).qb && i < c.size(); ++i) t += c[i];
        return t;
    }
    if (n == "v2_delta_nodes") return 0;  // the code-array engine has no delta records (kept for older tools)
    if (n == "device_bytes_per_node") return P.n_local > 0 ? (int64_t)((ix->ops_bytes + (P.v2 ? 0 : ix->d_codes.cap)) / (size_t)P.n_local) : 0;
    if (n == "last_fallback") return ix->last_fallback;
    if (n == "n_deleted") return ix->n_deleted;
    if (n == "last_delete_us") return ix->last_delete_us;
    if (n == "n_added") return ix->n_added;
    if (n == "last_add_us") return ix->last_add_us;
    if (n == "last_compact_us") return ix->compact_us[0];
    if (n == "last_compact_gather_us") return ix->compact_us[1];
    if (n == "last_compact_edge_us") return ix->compact_us[2];
    if (n == "last_compact_layout_us") return ix->compact_us[3];
    if (n == "last_compact_build_us") return ix->compact_us[2] + ix->compact_us[3];
    if (n.rfind("depth_hist_", 0) == 0) {
        size_t d = (size_t)atoi(n.c_str() + 11);
        return d < P.depth_hist.size() ? P.depth_hist[d] : 0;
    }
    if (n == "timed_calls") return ix->timed_calls;
    const bool last = n == "last_scan_us" || n == "last_total_us" || n == "last_lut_us" || n == "last_scan8_us";
    const bool sum = n == "sum_scan_ns" || n == "sum_total_ns" || n == "sum_lut_ns" || n == "sum_scan8_ns";
    if (last || sum) {  // "last_*": the last search; "sum_*": all searches since "timing_reset"
        if (!ix->timing_valid || !ix->ev) return -1;
        cudaSetDevice(ix->device);
        if (cudaEventSynchronize(ix->ev[3]) != cudaSuccess) return -1;
        const int which = n.find("scan8") != std::string::npos ? 3 : (n.find("scan") != std::string::npos ? 0 : (n.find("lut") != std::string::npos ? 1 : 2));
        if (which == 3 && !ix->last_coarse && !ix->last_latency) return -1;  // scan8 or, in latency mode, the full scan1 pass
        double total_ms = 0;
        const int first = last ? ix->timed_calls - 1 : 0;
        for (int c = first; c < ix->timed_calls; ++c) {
            cudaEvent_t* e = ix->evs.data() + 6 * c;
            float ms = 0;
            cudaEvent_t a = which == 3 ? e[4] : (which == 0 ? e[1] : e[0]);
            cudaEvent_t b = which == 3 ? e[5] : (which == 0 ? e[2] : (which == 1 ? e[1] : e[3]));
            if (cudaEventElapsedTime(&ms, a, b) != cudaSuccess) return -1;
            total_ms += ms;
        }
        return last ? (int64_t)(total_ms * 1e3 + 0.5) : (int64_t)(total_ms * 1e6 + 0.5);
    }
    return -1;
}

void dpq_index_close(dpq_index* ix) {
    if (!ix) return;
    cudaSetDevice(ix->device);
    if (ix->stream) cudaStreamSynchronize(ix->stream);
    for (DevBuf* b : {&ix->d_cap0, &ix->d_cap1, &ix->d_qlut8, &ix->d_cand8, &ix->d_cnt8, &ix->d_ovf8, &ix->d_flagged2, &ix->d_ovf, &ix->d_cand1, &ix->d_cnt1, &ix->d_part8, &ix->d_done8, &ix->d_ps_codes, &ix->d_stage8, &ix->d_ops, &ix->d_chunks, &ix->d_anc, &ix->d_codes, &ix->d_pos2id, &ix->d_cw,
                      &ix->d_queries, &ix->d_lutf, &ix->d_scale, &ix->d_qlut, &ix->d_cand, &ix->d_cnt,
                      &ix->d_flagged, &ix->d_ctrl, &ix->d_bound, &ix->d_key, &ix->d_fpart,
                      &ix->d_gthr, &ix->d_dead, &ix->d_del_ids, &ix->d_del_tmp})
        b->release();
    if (ix->h_stage) cudaFreeHost(ix->h_stage);
    for (auto& e : ix->evs)
        if (e) cudaEventDestroy(e);
    if (ix->stream && ix->own_stream) cudaStreamDestroy(ix->stream);
    (void)cudaGetLastError();
    delete ix;
}

int dpq_adc_tables(const float* cw, int M, int K, int Ds, const float* queries, int Q, float* lut) {
    if (!cw || !queries || !lut || M < 1 || M > 16 || K < 1 || K > 256 || Ds < 1 || Q < 1)
        return fail(DPQ_ERR_ARG, "dpq_adc_tables: bad argument");
    int rc = check_device();
    if (rc) return rc;
    CU(cudaSetDevice(g_device));
    DevBuf d_cw, d_q, d_l;
    size_t cwb = (size_t)M * K * Ds * 4, qb = (size_t)Q * M * Ds * 4, lb = (size_t)Q * M * K * 4;
    if ((rc = d_cw.ensure(cwb)) || (rc = d_q.ensure(qb)) || (rc = d_l.ensure(lb))) return rc;
    CU(cudaMemcpy(d_cw.p, cw, cwb, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_q.p, queries, qb, cudaMemcpyHostToDevice));
    dpq::launch_lut_plain(d_cw.as<float>(), M, K, Ds, d_q.as<float>(), Q, d_l.as<float>(), 0);
    CU(cudaGetLastError());
    CU(cudaMemcpy(lut, d_l.p, lb, cudaMemcpyDeviceToHost));
    d_cw.release();
    d_q.release();
    d_l.release();
    return DPQ_OK;
}

}  // extern "C"

namespace dpq {  // for dpq_multi_compact (multi.cu)
int index_live_nodes(dpq_index* ix, uint8_t** d_codes, uint32_t** d_ids, int64_t* n_live) {
    if (!ix->prog.v2)
        return fail(DPQ_ERR_ARG, "dpq_multi_compact: compaction needs the code-array engine (this handle runs the first-generation engine, DPQ_ENGINE=1)");
    CU(cudaSetDevice(ix->device));
    return live_nodes(ix, d_codes, d_ids, n_live);
}
// A forest part compacted inside a multi-GPU handle: its id table (the global positions the handle gave its nodes)
// moves to *ids, and the part reports positions as ids again, as every part of a handle does.
void index_take_ids(dpq_index* ix, std::vector<uint32_t>* ids) {
    ids->swap(ix->pos2id_host);
    std::vector<uint32_t>().swap(ix->pos2id_host);
    ix->has_pos2id = false;
    cudaSetDevice(ix->device);
    ix->d_pos2id.release();
}
}  // namespace dpq
