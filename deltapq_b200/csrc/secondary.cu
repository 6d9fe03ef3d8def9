// Secondary kernels of the DeltaPQ pipeline (in scope per BASELINE.json north_star):
//   encode_kernel        PQTree::EncodePlain nearest-centroid argmin (pq_tree.cpp:215-237)
//   edge_diff_kernel     per-edge changed-subspace bitmap / diff count (DCAT.h:196-238)
//   gt_dist / gt_select  exact brute-force ground truth (pmain:138-166)
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/dpq.h"
#include "encode_tc.cuh"
#include "gt_tc.cuh"

namespace dpq {
int api_fail(int code, const std::string& msg);  // api_common.cu
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

// ------------------------------------------------------------------------ encode -------
// Block = 256 vectors x one subspace.  The subspace's K x Ds codebook slice sits in shared
// memory (every thread reads the same word: broadcast); each thread keeps its Ds-float
// sub-vector in registers.  Arithmetic is the reference's, op for op: float subtract, float
// multiply, float add (no FMA: __f*_rn intrinsics are never contracted), strict <, so ties
// go to the lowest centroid id and the codes are bit-exact.
template <int DS>
__global__ void __launch_bounds__(256) encode_kernel(const float* __restrict__ cw, int M, int K,
                                                     const float* __restrict__ x, int64_t n, int D,
                                                     uint8_t* __restrict__ codes) {
    extern __shared__ float s_cw[];  // [K][DS]
    const int m = blockIdx.y;
    for (int i = threadIdx.x; i < K * DS; i += blockDim.x) s_cw[i] = cw[(size_t)m * K * DS + i];
    __syncthreads();
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    float xr[DS];
#pragma unroll
    for (int d = 0; d < DS; ++d) {
        int col = m * DS + d;
        xr[d] = col < D ? x[(size_t)v * D + col] : 0.0f;  // zero padding (pq_tree.cpp:194-198)
    }
    float best = FLT_MAX;
    int best_k = -1;  // nothing below FLT_MAX (overflow, NaN): the reference writes (uchar)-1 (pq_tree.cpp:217, 235)
    for (int k = 0; k < K; ++k) {
        const float* c = s_cw + k * DS;
        float dist = 0.0f;
#pragma unroll
        for (int d = 0; d < DS; ++d) {
            float diff = __fsub_rn(xr[d], c[d]);
            dist = __fadd_rn(dist, __fmul_rn(diff, diff));
        }
        if (dist < best) {
            best = dist;
            best_k = k;
        }
    }
    codes[(size_t)v * M + m] = (uint8_t)best_k;
}

// any Ds: sub-vector staged in shared memory as [d][thread]
__global__ void __launch_bounds__(256) encode_kernel_any(const float* __restrict__ cw, int M, int K,
                                                         int Ds, const float* __restrict__ x,
                                                         int64_t n, int D, uint8_t* __restrict__ codes) {
    extern __shared__ float s_mem[];
    float* s_cw = s_mem;            // [K][Ds]
    float* s_x = s_mem + K * Ds;    // [Ds][256]
    const int m = blockIdx.y;
    for (int i = threadIdx.x; i < K * Ds; i += blockDim.x) s_cw[i] = cw[(size_t)m * K * Ds + i];
    const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int d = 0; d < Ds; ++d) {
        int col = m * Ds + d;
        s_x[d * 256 + threadIdx.x] = (v < n && col < D) ? x[(size_t)v * D + col] : 0.0f;
    }
    __syncthreads();
    if (v >= n) return;
    float best = FLT_MAX;
    int best_k = -1;  // nothing below FLT_MAX (overflow, NaN): the reference writes (uchar)-1 (pq_tree.cpp:217, 235)
    for (int k = 0; k < K; ++k) {
        const float* c = s_cw + k * Ds;
        float dist = 0.0f;
        for (int d = 0; d < Ds; ++d) {
            float diff = __fsub_rn(s_x[d * 256 + threadIdx.x], c[d]);
            dist = __fadd_rn(dist, __fmul_rn(diff, diff));
        }
        if (dist < best) {
            best = dist;
            best_k = k;
        }
    }
    codes[(size_t)v * M + m] = (uint8_t)best_k;
}

// bvecs components (utils.cpp:43-71 reads them into floats): rows of D bytes `stride` bytes apart
__global__ void u8_to_float_kernel(const uint8_t* __restrict__ src, int64_t n, int D, int64_t stride, int64_t skip,
                                   float* __restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * D) return;
    const int64_t v = i / D;
    dst[i] = (float)src[v * stride + skip + (i - v * D)];
}

}  // namespace

namespace dpq {  // also used by dpq_index_add_vectors (api.cu)

cudaError_t launch_encode(const float* d_cw, int M, int K, int Ds, const float* d_x, int64_t n, int D,
                          uint8_t* d_codes, cudaStream_t st) {
    dim3 grid((unsigned)((n + 255) / 256), (unsigned)M), block(256);
    size_t sm = (size_t)K * Ds * 4;
#define DPQ_ENC(DSV)                                                                              \
    case DSV:                                                                                     \
        cudaFuncSetAttribute(encode_kernel<DSV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm); \
        encode_kernel<DSV><<<grid, block, sm, st>>>(d_cw, M, K, d_x, n, D, d_codes);             \
        break;
    switch (Ds) {
        DPQ_ENC(4)
        DPQ_ENC(8)
        DPQ_ENC(16)
        DPQ_ENC(32)
        DPQ_ENC(60)
        default: {
            size_t sm2 = sm + (size_t)Ds * 256 * 4;
            if (sm2 > 227 * 1024) return cudaErrorInvalidValue;
            cudaFuncSetAttribute(encode_kernel_any, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm2);
            encode_kernel_any<<<grid, block, sm2, st>>>(d_cw, M, K, Ds, d_x, n, D, d_codes);
        }
    }
#undef DPQ_ENC
    return cudaGetLastError();
}

}  // namespace dpq

namespace {

// ------------------------------------------------------------------------ edge diffs ---
__global__ void edge_diff_kernel(const uint8_t* __restrict__ codes, int M, const uint32_t* __restrict__ edges,
                                 int64_t n_edges, uint32_t* __restrict__ bitmaps,
                                 unsigned long long* __restrict__ total) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int nd = 0;
    if (e < n_edges) {
        const uint8_t* a = codes + (size_t)edges[2 * e] * M;
        const uint8_t* b = codes + (size_t)edges[2 * e + 1] * M;
        uint32_t bm = 0;
        if (M == 8) {  // XOR of the packed codes, then a per-byte non-zero mask
            uint64_t xa = *reinterpret_cast<const uint64_t*>(a) ^ *reinterpret_cast<const uint64_t*>(b);
#pragma unroll
            for (int m = 0; m < 8; ++m) bm |= ((xa >> (8 * m)) & 0xFFull) ? (1u << m) : 0u;
        } else {
            for (int m = 0; m < M; ++m) bm |= (a[m] != b[m]) ? (1u << m) : 0u;
        }
        bitmaps[e] = bm;
        nd = __popc(bm);
    }
    for (int o = 16; o; o >>= 1) nd += __shfl_xor_sync(0xffffffffu, nd, o);
    if ((threadIdx.x & 31) == 0 && nd) atomicAdd(total, (unsigned long long)nd);
}

// ------------------------------------------------------------------------ ground truth -
// Distances in the reference's arithmetic (pmain:150-156): float difference, float product,
// double running sum over d ascending; narrowed to float when it enters the heap.
// Tile: 128 base vectors x 8 queries per block, base tile staged through shared memory.
constexpr int GT_TB = 128, GT_TQ = 8;
// qlist (optional): the launch covers the Q queries qlist[0..Q) of the query array; dist rows follow
// the list order.
__global__ void __launch_bounds__(GT_TB) gt_dist_kernel(const float* __restrict__ base, int64_t n,
                                                        const float* __restrict__ queries, int Q, int D,
                                                        float* __restrict__ dist /*[Q][n]*/,
                                                        const uint32_t* __restrict__ qlist) {
    extern __shared__ float s_q[];  // [GT_TQ][D]
    const int q0 = blockIdx.y * GT_TQ;
    for (int i = threadIdx.x; i < GT_TQ * D; i += blockDim.x) {
        int qq = q0 + i / D;
        s_q[i] = qq < Q ? queries[(size_t)(qlist ? qlist[qq] : (uint32_t)qq) * D + i % D] : 0.0f;
    }
    __syncthreads();
    const int64_t v = (int64_t)blockIdx.x * GT_TB + threadIdx.x;
    if (v >= n) return;
    double acc[GT_TQ];
#pragma unroll
    for (int j = 0; j < GT_TQ; ++j) acc[j] = 0.0;
    const float* x = base + (size_t)v * D;
    for (int d = 0; d < D; ++d) {
        float xv = x[d];
#pragma unroll
        for (int j = 0; j < GT_TQ; ++j) {
            float diff = __fsub_rn(xv, s_q[j * D + d]);
            acc[j] = __dadd_rn(acc[j], (double)__fmul_rn(diff, diff));
        }
    }
#pragma unroll
    for (int j = 0; j < GT_TQ; ++j)
        if (q0 + j < Q) dist[(size_t)(q0 + j) * n + v] = (float)acc[j];
}

// One block per query: merge this chunk's distances into the running sorted top-k
// (keys = float bits << 32 | id; ascending; ties keep the lower id like the reference's
// strict < against the heap top while ids arrive in ascending order).
constexpr int GT_SEL_T = 256, GT_BUF = 2048;
__global__ void __launch_bounds__(GT_SEL_T) gt_select_kernel(const float* __restrict__ dist, int64_t n,
                                                             int64_t id0, int topk,
                                                             unsigned long long* __restrict__ state /*[Q][topk]*/,
                                                             const uint32_t* __restrict__ qlist) {
    __shared__ unsigned long long s_buf[GT_BUF];
    __shared__ int s_n;
    __shared__ unsigned long long s_bound;
    const int q = blockIdx.x;  // row of dist; the state row is the listed query
    unsigned long long* st = state + (size_t)(qlist ? qlist[q] : (uint32_t)q) * topk;
    // buffer starts with the current state
    for (int i = threadIdx.x; i < topk; i += blockDim.x) s_buf[i] = st[i];
    if (threadIdx.x == 0) {
        s_n = topk;
        s_bound = st[topk - 1];
    }
    __syncthreads();
    const float* dq = dist + (size_t)q * n;
    auto compact = [&]() {  // sort s_buf[0..s_n) ascending, keep topk, refresh bound
        int cnt = s_n;
        int np2 = 1;
        while (np2 < cnt) np2 <<= 1;
        for (int i = cnt + threadIdx.x; i < np2; i += blockDim.x) s_buf[i] = ~0ull;
        __syncthreads();
        for (int k = 2; k <= np2; k <<= 1)
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int i = threadIdx.x; i < np2; i += blockDim.x) {
                    int ixj = i ^ j;
                    if (ixj > i) {
                        unsigned long long a = s_buf[i], b = s_buf[ixj];
                        bool up = (i & k) == 0;
                        if ((a > b) == up) {
                            s_buf[i] = b;
                            s_buf[ixj] = a;
                        }
                    }
                }
                __syncthreads();
            }
        if (threadIdx.x == 0) {
            s_n = topk;
            s_bound = s_buf[topk - 1];
        }
        __syncthreads();
    };
    for (int64_t base_i = 0; base_i < n; base_i += GT_SEL_T) {
        int64_t i = base_i + threadIdx.x;
        unsigned long long key = ~0ull;
        if (i < n) key = ((unsigned long long)__float_as_uint(dq[i]) << 32) | (unsigned)(id0 + i);
        bool take = key < s_bound;
        // at most GT_SEL_T pushes per step: compact first if they might not fit
        if (s_n + GT_SEL_T > GT_BUF) {
            __syncthreads();
            compact();
            take = key < s_bound;
        }
        if (take) {
            int slot = atomicAdd(&s_n, 1);
            s_buf[slot] = key;
        }
        __syncthreads();
    }
    compact();
    for (int i = threadIdx.x; i < topk; i += blockDim.x) st[i] = s_buf[i];
}

struct Buf {
    void* p = nullptr;
    ~Buf() {
        if (p) cudaFree(p);
    }
};

}  // namespace

struct dpq_gt {
    int Q, D, topk;
    float* d_q = nullptr;
    unsigned long long* d_state = nullptr;
    float* d_base = nullptr;
    float* d_dist = nullptr;
    size_t base_cap = 0, dist_cap = 0;
    // tensor-core filter path (gt_tc.cu): topk <= 64 unless DPQ_GT_TC=0
    bool tc = false, seeded = false;
    int tc_form = 2;  // 2: pipelined (pre-split operands, TMA, warp-specialised roles); 1: synchronous form
    unsigned char *d_qsplit = nullptr, *d_xsplit = nullptr;
    size_t xsplit_cap = 0;
    int n_sms = 148;
    float *d_qn = nullptr, *d_xn = nullptr;  // [3][Q] / [3][x_cap]: ||v||^2 low, high, ||v|| high
    size_t x_cap = 0;
    float *d_thr = nullptr, *d_qerr = nullptr;
    uint32_t *d_cand = nullptr, *d_cnt = nullptr, *d_flag = nullptr, *d_ctl = nullptr;  // ctl: [0] flagged, [1] error
    int64_t tc_vectors = 0, tc_candidates = 0, tc_flagged = 0;  // statistics
    double tc_filter_ms = 0.0, tc_rescore_ms = 0.0;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
};

namespace {
constexpr int64_t GT_TC_STEP = 131072;  // base vectors per filter launch: the cap tightens between launches
// vectors scored densely first, so that every query has a finite cap.  The first launch's survivors
// are about k * step / seed per query: 4096 keeps them (and the exact re-score) small -- a 1024 seed
// tripled the re-score time -- and 64 per wanted neighbour keeps long lists inside the candidate slots
inline int64_t gt_tc_seed(int topk) { return std::min<int64_t>(8192, std::max<int64_t>(4096, 64LL * topk)); }
constexpr int GT_TC_CAND = 4096;        // candidate slots per query per launch

// dense exact path over base[0..n) (device) for the queries qlist[0..nq) (nullptr: all)
int gt_dense(dpq_gt* st, const float* d_base, int64_t n, int64_t id0, const uint32_t* qlist, int nq) {
    const int64_t step = std::max<int64_t>(1, std::min<int64_t>(n, ((int64_t)256 << 20) / ((int64_t)nq * 4)));
    const size_t db = (size_t)step * nq * 4;
    if (db > st->dist_cap) {
        if (st->d_dist) cudaFree(st->d_dist);
        st->d_dist = nullptr;
        st->dist_cap = 0;
        CU(cudaMalloc(&st->d_dist, db));
        st->dist_cap = db;
    }
    const size_t sm = (size_t)GT_TQ * st->D * 4;
    cudaFuncSetAttribute(gt_dist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
    for (int64_t s = 0; s < n; s += step) {
        const int64_t c = std::min(step, n - s);
        dim3 grid((unsigned)((c + GT_TB - 1) / GT_TB), (unsigned)((nq + GT_TQ - 1) / GT_TQ));
        gt_dist_kernel<<<grid, GT_TB, sm>>>(d_base + (size_t)s * st->D, c, st->d_q, nq, st->D, st->d_dist, qlist);
        gt_select_kernel<<<nq, GT_SEL_T>>>(st->d_dist, c, id0 + s, st->topk, st->d_state, qlist);
        CU(cudaGetLastError());
    }
    return DPQ_OK;
}

// tensor-core filter + exact re-score over base[0..n) (device, norms already in d_xn)
int gt_tc_range(dpq_gt* st, const float* d_base, int64_t n, int64_t id0, int64_t xoff) {
    const int Q = st->Q;
    // err <= c_err ||x|| ||q||: 2 x (dropped split terms 4 x 2^-18 + fp32 accumulation of 3 D products)
    const int dpad = (st->D + 63) / 64 * 64;
    const float c_err = 2.02f * (4.0f / 262144.0f + (3.0f * dpad + 8.0f) / 8388608.0f);
    CU(dpq::launch_gt_thr(st->d_state, st->topk, Q, st->d_qn, st->d_qn + Q, st->d_qn + 2 * (size_t)Q, c_err, st->d_thr,
                          st->d_qerr, 0));
    CU(cudaMemsetAsync(st->d_cnt, 0, (size_t)Q * 4));
    CU(cudaMemsetAsync(st->d_ctl, 0, 16));  // [0] flagged queries, [1] error flag
    dpq::GtTcArgs a;
    a.base = d_base;
    a.queries = st->d_q;
    a.n = n;
    a.Q = Q;
    a.D = st->D;
    a.x_nlo = st->d_xn + xoff;
    a.x_len = st->d_xn + 2 * st->x_cap + xoff;
    a.thr = st->d_thr;
    a.qerr = st->d_qerr;
    a.cand = st->d_cand;
    a.cand_cnt = st->d_cnt;
    a.cand_cap = GT_TC_CAND;
    a.error = st->d_ctl + 1;
    a.q_split = nullptr;
    a.x_split = nullptr;
    for (auto& e : st->ev)
        if (!e) CU(cudaEventCreate(&e));
    CU(cudaEventRecord(st->ev[0], 0));
    if (st->tc_form == 2) {
        const size_t need = dpq::gt_split_bytes(n, st->D, false);
        if (need > st->xsplit_cap) {
            if (st->d_xsplit) cudaFree(st->d_xsplit);
            st->d_xsplit = nullptr;
            st->xsplit_cap = 0;
            CU(cudaMalloc(&st->d_xsplit, need));
            st->xsplit_cap = need;
        }
        CU(dpq::launch_gt_split(d_base, n, st->D, false, st->d_xsplit, 0));
        a.q_split = st->d_qsplit;
        a.x_split = st->d_xsplit;
        CU(dpq::launch_gt_tc_filter2(a, st->n_sms, 0));
    } else {
        CU(dpq::launch_gt_tc_filter(a, st->n_sms, 0));
    }
    CU(cudaEventRecord(st->ev[1], 0));
    CU(dpq::launch_gt_rescore(a, id0, st->topk, st->d_state, st->d_flag, st->d_ctl, 0));
    CU(cudaEventRecord(st->ev[2], 0));
    uint32_t ctl[2] = {0, 0};
    CU(cudaMemcpy(ctl, st->d_ctl, 8, cudaMemcpyDeviceToHost));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, st->ev[0], st->ev[1]) == cudaSuccess) st->tc_filter_ms += ms;
    if (cudaEventElapsedTime(&ms, st->ev[1], st->ev[2]) == cudaSuccess) st->tc_rescore_ms += ms;
    if (ctl[1]) return dpq::api_fail(DPQ_ERR_CUDA, "ground truth: a tensor-core completion barrier never fired");
    st->tc_vectors += n;
    st->tc_flagged += ctl[0];
    if (ctl[0]) return gt_dense(st, d_base, n, id0, st->d_flag, (int)ctl[0]);  // overflowed candidate lists
    return DPQ_OK;
}

// ------------------------------------------------------------------------ encode driver -------
int64_t g_enc_tc = 0, g_enc_kernel_us = 0;

bool is_device_ptr(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice;
}

// One encode call: the codebook on the device, the path choice (tensor cores for Ds in {4, 8, 16} unless
// DPQ_ENCODE_TC=0, else the SIMT kernel), the kernels' device time.
struct Encoder {
    Buf d_cw, d_scratch, d_err;
    int M = 0, K = 0, Ds = 0, n_sms = 148;
    bool tc = false;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    double ms = 0.0;
    ~Encoder() {
        for (auto e : ev)
            if (e) cudaEventDestroy(e);
    }
    int init(const float* cw, int M_, int K_, int Ds_) {
        M = M_, K = K_, Ds = Ds_;
        g_enc_tc = 0, g_enc_kernel_us = 0;
        CU(cudaMalloc(&d_cw.p, (size_t)M * K * Ds * 4));
        CU(cudaMemcpy(d_cw.p, cw, (size_t)M * K * Ds * 4, cudaMemcpyDefault));
        const char* env = getenv("DPQ_ENCODE_TC");
        tc = dpq::encode_tc_supported(M, K, Ds) && !(env && env[0] == '0');
        if (tc) {
            CU(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dpq::api_device()));  // (cudaGetDeviceProperties takes milliseconds)
            CU(cudaMalloc(&d_scratch.p, dpq::encode_tc_scratch_bytes(M)));
            CU(cudaMalloc(&d_err.p, 4));
            CU(cudaMemset(d_err.p, 0, 4));
        }
        CU(cudaEventCreate(&ev[0]));
        CU(cudaEventCreate(&ev[1]));
        return DPQ_OK;
    }
    int run(const float* d_x, int64_t n, int D, uint8_t* d_codes) {
        CU(cudaEventRecord(ev[0], 0));
        if (tc)
            CU(dpq::launch_encode_tc((const float*)d_cw.p, M, K, Ds, d_x, n, D, d_codes, (unsigned char*)d_scratch.p,
                                     (uint32_t*)d_err.p, n_sms, 0));
        else
            CU(dpq::launch_encode((const float*)d_cw.p, M, K, Ds, d_x, n, D, d_codes, 0));
        CU(cudaEventRecord(ev[1], 0));
        CU(cudaEventSynchronize(ev[1]));
        float t = 0.0f;
        CU(cudaEventElapsedTime(&t, ev[0], ev[1]));
        ms += t;
        return DPQ_OK;
    }
    int finish() {
        if (tc) {
            uint32_t err = 0;
            CU(cudaMemcpy(&err, d_err.p, 4, cudaMemcpyDeviceToHost));
            if (err) return dpq::api_fail(DPQ_ERR_CUDA, "encode: a tensor-core completion barrier never fired");
        }
        g_enc_tc = tc ? 1 : 0;
        g_enc_kernel_us = (int64_t)(ms * 1e3);
        return DPQ_OK;
    }
};
}  // namespace

extern "C" {

int dpq_encode(const float* cw, int M, int K, int Ds, const float* x, int64_t n, int D, uint8_t* codes) {
    if (!cw || !x || !codes || M < 1 || M > 64 || K < 1 || K > 256 || Ds < 1 || n < 0 || D < 1 ||
        D > M * Ds)
        return dpq::api_fail(DPQ_ERR_ARG, "dpq_encode: bad argument");
    int rc = dpq::api_check_device();
    if (rc) return rc;
    if (n == 0) return DPQ_OK;
    CU(cudaSetDevice(dpq::api_device()));
    Encoder enc;
    if ((rc = enc.init(cw, M, K, Ds))) return rc;
    if (is_device_ptr(x) && is_device_ptr(codes)) {  // device-resident input and output: no staging
        if ((rc = enc.run(x, n, D, codes))) return rc;
        return enc.finish();
    }
    Buf d_x, d_c;
    const int64_t chunk = std::min<int64_t>(n, (int64_t)1 << 20);
    CU(cudaMalloc(&d_x.p, (size_t)chunk * D * 4));
    CU(cudaMalloc(&d_c.p, (size_t)chunk * M));
    for (int64_t s = 0; s < n; s += chunk) {
        int64_t c = std::min(chunk, n - s);
        CU(cudaMemcpy(d_x.p, x + (size_t)s * D, (size_t)c * D * 4, cudaMemcpyDefault));
        if ((rc = enc.run((const float*)d_x.p, c, D, (uint8_t*)d_c.p))) return rc;
        CU(cudaMemcpy(codes + (size_t)s * M, d_c.p, (size_t)c * M, cudaMemcpyDefault));
    }
    return enc.finish();
}

int dpq_encode_u8(const float* cw, int M, int K, int Ds, const uint8_t* x, int64_t n, int D, int64_t row_stride,
                  int64_t row_offset, uint8_t* codes) {
    if (!cw || !x || !codes || M < 1 || M > 64 || K < 1 || K > 256 || Ds < 1 || n < 0 || D < 1 || D > M * Ds ||
        row_offset < 0 || row_stride < row_offset + D)
        return dpq::api_fail(DPQ_ERR_ARG, "dpq_encode_u8: bad argument");
    int rc = dpq::api_check_device();
    if (rc) return rc;
    if (n == 0) return DPQ_OK;
    CU(cudaSetDevice(dpq::api_device()));
    Encoder enc;
    if ((rc = enc.init(cw, M, K, Ds))) return rc;
    Buf d_raw, d_x, d_c;
    const int64_t chunk = std::min<int64_t>(n, (int64_t)1 << 20);
    CU(cudaMalloc(&d_raw.p, (size_t)chunk * row_stride));
    CU(cudaMalloc(&d_x.p, (size_t)chunk * D * 4));
    CU(cudaMalloc(&d_c.p, (size_t)chunk * M));
    for (int64_t s = 0; s < n; s += chunk) {
        const int64_t c = std::min(chunk, n - s);
        // the last record may end before a whole stride (no trailing padding in the caller's buffer)
        const size_t raw_bytes = (size_t)(c - 1) * row_stride + (size_t)(row_offset + D);
        CU(cudaMemcpy(d_raw.p, x + (size_t)s * row_stride, raw_bytes, cudaMemcpyDefault));
        u8_to_float_kernel<<<(unsigned)((c * D + 255) / 256), 256>>>((const uint8_t*)d_raw.p, c, D, row_stride, row_offset,
                                                                     (float*)d_x.p);
        if ((rc = enc.run((const float*)d_x.p, c, D, (uint8_t*)d_c.p))) return rc;
        CU(cudaMemcpy(codes + (size_t)s * M, d_c.p, (size_t)c * M, cudaMemcpyDefault));
    }
    return enc.finish();
}

int64_t dpq_encode_stat(const char* name) {
    if (!name) return -1;
    const std::string s(name);
    if (s == "tc") return g_enc_tc;                 // 1: the last encode call ran on the tensor cores
    if (s == "kernel_us") return g_enc_kernel_us;   // device time of its encode kernels (CUDA events)
    return -1;
}

int dpq_edge_diffs(const uint8_t* codes, int64_t n_codes, int M, const uint32_t* edges, int64_t n_edges,
                   uint32_t* bitmaps, int64_t* n_diffs) {
    if (!codes || !edges || M < 1 || M > 32 || n_edges < 0)
        return dpq::api_fail(DPQ_ERR_ARG, "dpq_edge_diffs: bad argument");
    int rc = dpq::api_check_device();
    if (rc) return rc;
    CU(cudaSetDevice(dpq::api_device()));
    if (n_diffs) *n_diffs = 0;
    if (n_edges == 0) return DPQ_OK;
    Buf d_codes, d_edges, d_bm, d_tot;
    CU(cudaMalloc(&d_codes.p, (size_t)n_codes * M + 8));
    CU(cudaMalloc(&d_edges.p, (size_t)n_edges * 8));
    CU(cudaMalloc(&d_bm.p, (size_t)n_edges * 4));
    CU(cudaMalloc(&d_tot.p, 8));
    CU(cudaMemcpy(d_codes.p, codes, (size_t)n_codes * M, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_edges.p, edges, (size_t)n_edges * 8, cudaMemcpyHostToDevice));
    CU(cudaMemset(d_tot.p, 0, 8));
    edge_diff_kernel<<<(unsigned)((n_edges + 255) / 256), 256>>>((const uint8_t*)d_codes.p, M,
                                                                (const uint32_t*)d_edges.p, n_edges,
                                                                (uint32_t*)d_bm.p,
                                                                (unsigned long long*)d_tot.p);
    CU(cudaGetLastError());
    if (bitmaps) CU(cudaMemcpy(bitmaps, d_bm.p, (size_t)n_edges * 4, cudaMemcpyDeviceToHost));
    unsigned long long tot = 0;
    CU(cudaMemcpy(&tot, d_tot.p, 8, cudaMemcpyDeviceToHost));
    if (n_diffs) *n_diffs = (int64_t)tot;
    return DPQ_OK;
}

int dpq_groundtruth_begin(const float* queries, int Q, int D, int topk, dpq_gt** out) {
    if (!queries || !out || Q < 1 || D < 1 || topk < 1 || topk > 1024)
        return dpq::api_fail(DPQ_ERR_ARG, "dpq_groundtruth_begin: bad argument");
    int rc = dpq::api_check_device();
    if (rc) return rc;
    CU(cudaSetDevice(dpq::api_device()));
    dpq_gt* st = new dpq_gt();
    st->Q = Q;
    st->D = D;
    st->topk = topk;
    CU(cudaMalloc(&st->d_q, (size_t)Q * D * 4));
    CU(cudaMalloc(&st->d_state, (size_t)Q * topk * 8));
    CU(cudaMemcpy(st->d_q, queries, (size_t)Q * D * 4, cudaMemcpyHostToDevice));
    // (FLT_MAX, 0xFFFFFFFF) sentinels: results[i][j].second = FLT_MAX (pmain:609-611)
    std::vector<unsigned long long> init((size_t)Q * topk, ((unsigned long long)0x7F7FFFFFu << 32) | 0xFFFFFFFFull);
    CU(cudaMemcpy(st->d_state, init.data(), init.size() * 8, cudaMemcpyHostToDevice));
    const char* env = getenv("DPQ_GT_TC");
    st->tc = topk <= 64 && !(env && env[0] == '0');
    if (st->tc) {
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, dpq::api_device()));
        st->n_sms = prop.multiProcessorCount;
        CU(cudaMalloc(&st->d_qn, (size_t)Q * 3 * 4));
        CU(cudaMalloc(&st->d_thr, (size_t)Q * 4));
        CU(cudaMalloc(&st->d_qerr, (size_t)Q * 4));
        CU(cudaMalloc(&st->d_cand, (size_t)Q * GT_TC_CAND * 4));
        CU(cudaMalloc(&st->d_cnt, (size_t)Q * 4));
        CU(cudaMalloc(&st->d_flag, (size_t)Q * 4));
        CU(cudaMalloc(&st->d_ctl, 16));
        CU(dpq::launch_gt_prep(st->d_q, Q, D, st->d_qn, st->d_qn + Q, st->d_qn + 2 * (size_t)Q, 0));
        st->tc_form = (env && env[0] == '1') ? 1 : 2;
        if (st->tc_form == 2) {
            CU(cudaMalloc(&st->d_qsplit, dpq::gt_split_bytes(Q, D, true)));
            CU(dpq::launch_gt_split(st->d_q, Q, D, true, st->d_qsplit, 0));
        }
    }
    *out = st;
    return DPQ_OK;
}

int dpq_groundtruth_chunk(dpq_gt* st, const float* base, int64_t n, int64_t id0) {
    if (!st || !base || n < 0) return dpq::api_fail(DPQ_ERR_ARG, "dpq_groundtruth_chunk: bad argument");
    CU(cudaSetDevice(dpq::api_device()));
    // upload granularity: the dense path is bounded by its [Q][step] distance buffer, the tensor-core
    // path by the candidate lists (the cap tightens between launches)
    const int64_t step = st->tc ? GT_TC_STEP
                                : std::max<int64_t>(1, std::min<int64_t>(n, ((int64_t)256 << 20) / ((int64_t)st->Q * 4)));
    for (int64_t s = 0; s < n; s += step) {
        const int64_t c = std::min(step, n - s);
        const size_t bb = (size_t)c * st->D * 4;
        if (bb > st->base_cap) {
            if (st->d_base) cudaFree(st->d_base);
            st->d_base = nullptr;
            st->base_cap = 0;
            CU(cudaMalloc(&st->d_base, bb));
            st->base_cap = bb;
        }
        CU(cudaMemcpy(st->d_base, base + (size_t)s * st->D, bb, cudaMemcpyDefault));
        int rc;
        if (!st->tc) {
            if ((rc = gt_dense(st, st->d_base, c, id0 + s, nullptr, st->Q))) return rc;
            continue;
        }
        if ((size_t)c > st->x_cap) {
            if (st->d_xn) cudaFree(st->d_xn);
            st->d_xn = nullptr;
            st->x_cap = 0;
            CU(cudaMalloc(&st->d_xn, (size_t)c * 3 * 4));
            st->x_cap = (size_t)c;
        }
        CU(dpq::launch_gt_prep(st->d_base, c, st->D, st->d_xn, st->d_xn + st->x_cap, st->d_xn + 2 * st->x_cap, 0));
        int64_t s0 = 0;
        if (!st->seeded) {  // the first vectors densely: afterwards every query has k exact distances
            s0 = std::min<int64_t>(c, gt_tc_seed(st->topk));
            if ((rc = gt_dense(st, st->d_base, s0, id0 + s, nullptr, st->Q))) return rc;
            st->seeded = true;
        }
        if (c > s0 && (rc = gt_tc_range(st, st->d_base + (size_t)s0 * st->D, c - s0, id0 + s + s0, s0))) return rc;
    }
    CU(cudaDeviceSynchronize());
    return DPQ_OK;
}

int64_t dpq_groundtruth_stat(dpq_gt* st, const char* name) {
    if (!st || !name) return -1;
    const std::string w(name);
    if (w == "tc") return st->tc ? st->tc_form : 0;
    if (w == "tc_vectors") return st->tc_vectors;
    if (w == "tc_flagged") return st->tc_flagged;
    if (w == "tc_filter_us") return (int64_t)(st->tc_filter_ms * 1e3);
    if (w == "tc_rescore_us") return (int64_t)(st->tc_rescore_ms * 1e3);
    return -1;
}

int dpq_groundtruth_finish(dpq_gt* st, uint32_t* out_id, float* out_dist) {
    if (!st) return dpq::api_fail(DPQ_ERR_ARG, "dpq_groundtruth_finish: null");
    std::vector<unsigned long long> keys((size_t)st->Q * st->topk);
    cudaError_t e = cudaMemcpy(keys.data(), st->d_state, keys.size() * 8, cudaMemcpyDeviceToHost);
    cudaFree(st->d_q);
    cudaFree(st->d_state);
    if (st->d_base) cudaFree(st->d_base);
    if (st->d_dist) cudaFree(st->d_dist);
    for (void* p : {(void*)st->d_qn, (void*)st->d_xn, (void*)st->d_thr, (void*)st->d_qerr, (void*)st->d_cand,
                    (void*)st->d_cnt, (void*)st->d_flag, (void*)st->d_ctl, (void*)st->d_qsplit, (void*)st->d_xsplit})
        if (p) cudaFree(p);
    for (auto& e : st->ev)
        if (e) cudaEventDestroy(e);
    if (getenv("DPQ_GT_STATS"))
        fprintf(stderr, "dpq_groundtruth: tensor-core path %s, %lld vectors filtered, %lld query re-runs on the dense path\n",
                st->tc ? "on" : "off", (long long)st->tc_vectors, (long long)st->tc_flagged);
    delete st;
    if (e != cudaSuccess) return dpq::api_fail(DPQ_ERR_CUDA, cudaGetErrorString(e));
    for (size_t i = 0; i < keys.size(); ++i) {
        uint32_t bits = (uint32_t)(keys[i] >> 32);
        if (out_id) out_id[i] = (uint32_t)keys[i];
        if (out_dist) memcpy(&out_dist[i], &bits, 4);
    }
    return DPQ_OK;
}

}  // extern "C"
