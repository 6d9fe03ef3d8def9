// Hand-written sm_100a kernels of the DeltaPQ query hot path.
//
//   lut_kernel      ADC tables (reference DCAT.h:3750-3758), exact + quantised/swizzled
//   scan_kernel     DeltaTree delta scan (reference DCAT.h:3786-3882) over the compiled
//                   op program, lanes = queries, fused per-warp top-k' candidate lists
//   select_kernel   merge of the per-warp lists + exact re-score (reference heap,
//                   DCAT.h:3853-3889) + rigorous margin check
//   fallback_*      exact scan for queries whose margin check failed
//   merge_kernel    k-way merge of per-GPU top-k lists after the NCCL gather
//
// Numerics.  The reference accumulates float table entries in double along the tree path;
// its node distance is therefore (to ~1e-16) float(sum of the node's M table entries).
// scan_kernel instead runs the same parent -> child delta recurrence in EXACT integer
// arithmetic on a fixed-point copy of the table (no error accumulates along a path, the
// only error is the <= 0.5 unit rounding of each of the M entries), keeps topk + slack
// candidates per query, and select_kernel re-scores those with the float table in double.
// A query whose exact k-th distance is not separated from the first rejected fixed-point
// distance by the rounding bound is re-run by the exact fallback, so results never depend
// on the fixed-point precision.
#include "kernels.cuh"

#include <cfloat>

namespace dpq {

// ------------------------------------------------------------------------ ADC tables ---
// One CTA per (virtual) query; thread = centroid (adc_entry: kernels.cuh).
__global__ void __launch_bounds__(256) lut_kernel(const float* __restrict__ cw, int M, int K, int Ds,
                                                  const float* __restrict__ queries, int Q,
                                                  float* __restrict__ lutf, double* __restrict__ scale,
                                                  uint32_t* __restrict__ qlut, uint32_t* __restrict__ gthr,
                                                  ScanGeom g) {
    extern __shared__ float s_q[];  // M*Ds
    __shared__ int s_max[16];
    const int vq = blockIdx.x;  // virtual query (padding lanes of the last group included)
    const int k = threadIdx.x;
    const int rows = 1 << g.rb;
    // destination of this query inside the swizzled group table
    const int grp = vq / g.qpg, sub = vq % g.qpg;
    const int lane = sub % g.qgl, half = sub / g.qgl;
    uint32_t* dst = qlut ? qlut + ((size_t)grp * g.qgl + lane) * rows : nullptr;
    if (vq >= Q) {  // padding: all-zero table so the lane computes harmless zeros
        if (dst)
            for (int r = k; r < rows; r += blockDim.x) {
                if (g.pack == 1) dst[r] = 0;
                else reinterpret_cast<uint16_t*>(dst)[2 * r + half] = 0;
            }
        return;
    }
    for (int i = k; i < M * Ds; i += blockDim.x) s_q[i] = queries[(size_t)vq * M * Ds + i];
    if (k < 16) s_max[k] = 0;
    __syncthreads();
    float* out = lutf + (size_t)vq * M * K;
    for (int m = 0; m < M; ++m) {
        float v = 0.0f;
        if (k < K) {
            v = adc_entry(cw + ((size_t)m * K + k) * Ds, s_q + m * Ds, Ds);
            out[m * K + k] = v;
        }
        // v >= 0 so integer order == float order
        int vi = __float_as_int(v);
        for (int o = 16; o; o >>= 1) vi = max(vi, __shfl_xor_sync(0xffffffffu, vi, o));
        if ((k & 31) == 0) atomicMax(&s_max[m], vi);
    }
    if (!qlut) return;
    __syncthreads();
    double sum = 0.0;
    for (int m = 0; m < M; ++m) sum += (double)__int_as_float(s_max[m]);
    const double qmax = g.pack == 1 ? (double)(1u << 30) : (double)(32767 - 16);
    // a sum that is not positive (NaN from a NaN query component, or 0) scales by 0, as an infinite one does: every
    // entry 0, a filter that passes every node, the exact re-score and fallback decide
    const double s = sum > 0.0 ? qmax / sum : 0.0;
    if (k == 0) {
        scale[vq] = s;
        gthr[vq] = g.pack == 1 ? kInf31 : 0x8000u;
    }
    // rows beyond M*K are never addressed; entry (m,k) lives at word (row ^ lane).  Every entry is clamped to
    // [0, qmax] before packing (a no-op for a finite positive sum; NaN -> 0): no value can leave its lane.
    if (k < K)
        for (int m = 0; m < M; ++m) {
            uint32_t v = (uint32_t)__double2ll_rn(fmin(fmax((double)out[m * K + k] * s, 0.0), qmax));
            int r = (m * K + k) ^ lane;
            if (g.pack == 1) dst[r] = v;
            else reinterpret_cast<uint16_t*>(dst)[2 * r + half] = (uint16_t)v;
        }
}

void launch_lut(const float* d_cw, int M, int K, int Ds, const float* d_queries, int Q,
                float* d_lutf, double* d_scale, uint32_t* d_qlut, uint32_t* d_gthr, const ScanGeom& g,
                cudaStream_t st) {
    int nvq = g.n_groups * g.qpg;
    lut_kernel<<<nvq, 256, (size_t)M * Ds * sizeof(float), st>>>(d_cw, M, K, Ds, d_queries, Q, d_lutf,
                                                              d_scale, d_qlut, d_gthr, g);
}
void launch_lut_plain(const float* d_cw, int M, int K, int Ds, const float* d_queries, int Q,
                      float* d_lutf, cudaStream_t st) {
    ScanGeom g{};
    g.rb = 11;
    g.pack = 1;
    g.qgl = 1;
    g.qpg = 1;
    lut_kernel<<<Q, 256, (size_t)M * Ds * sizeof(float), st>>>(d_cw, M, K, Ds, d_queries, Q, d_lutf,
                                                            nullptr, nullptr, nullptr, g);
}

// ------------------------------------------------------------------------ scan ---------
// CTA = (query group, tree slice).  Shared memory: the group's fixed-point ADC table,
// [lane][row ^ lane] so that the 32 lanes of a warp, all reading the SAME row, hit 32
// different banks; per-warp op windows; per-warp depth stacks; per-query shared bounds.
// Each warp pulls chunks of the op program and runs the delta recurrence with lanes =
// queries: one table row read per changed subspace for the old and the new centroid.
//
// Candidates: a node whose distance is below the query's current bound is APPENDED to that
// (warp, query)'s buffer in global scratch (one store); when a buffer fills, the whole warp
// compacts it to its kp smallest keys (rank by counting through shuffles) and tightens the
// bound, which is shared through shared memory (CTA) and global memory (other slices).

// Warp-cooperative compaction of one buffer: keeps the min(n, kp) smallest of its n keys,
// sorted ascending, and returns the kept count (uniform).  *kth = distance part of the
// kp-th smallest key when n >= kp.
template <int MAXPER>
__device__ __forceinline__ int compact_buffer_t(uint64_t* buf, int n, int kp, int lane, uint32_t* kth) {
    __syncwarp();
    const int per = (n + 31) >> 5;
    uint64_t mine[MAXPER];
    int rank[MAXPER];
#pragma unroll
    for (int t = 0; t < MAXPER; ++t) {
        mine[t] = ~0ull;
        rank[t] = 0;
        if (t < per) {
            int i = t * 32 + lane;
            if (i < n) mine[t] = buf[i];
        }
    }
#pragma unroll
    for (int u = 0; u < MAXPER; ++u) {
        if (u < per) {
            for (int j = 0; j < 32; ++j) {
                uint64_t o = __shfl_sync(0xffffffffu, mine[u], j);
#pragma unroll
                for (int t = 0; t < MAXPER; ++t)
                    if (t < per) rank[t] += o < mine[t];
            }
        }
    }
    __syncwarp();
    const int keep = n < kp ? n : kp;
    uint32_t kd = 0;
#pragma unroll
    for (int t = 0; t < MAXPER; ++t) {
        if (t < per) {
            int i = t * 32 + lane;
            if (i < n && rank[t] < keep) buf[rank[t]] = mine[t];  // keys are unique
            if (i < n && rank[t] == kp - 1) kd = (uint32_t)(mine[t] >> 32);
        }
    }
    for (int o = 16; o; o >>= 1) kd |= __shfl_xor_sync(0xffffffffu, kd, o);
    *kth = kd;
    __syncwarp();
    return keep;
}

__device__ __noinline__ int compact_buffer_big(uint64_t* buf, int n, int kp, int lane, uint32_t* kth) {
    return compact_buffer_t<16>(buf, n, kp, lane, kth);  // buffers hold at most 512 keys
}
__device__ __forceinline__ int compact_buffer(uint64_t* buf, int n, int kp, int lane, uint32_t* kth) {
    if (n <= 32) return compact_buffer_t<1>(buf, n, kp, lane, kth);
    return compact_buffer_big(buf, n, kp, lane, kth);
}

// Lock-free insert of distance v into a CTA-shared ascending array A[0..n) that keeps the n
// smallest distances any warp of the CTA has seen for one query.  Each step is one
// atomicMin that leaves min(old, carry) in the slot and carries max(old, carry) on: the
// multiset {slots} + {carried values} is preserved and the array stays sorted under any
// interleaving, so A[n-1] is always a valid bound once no slot holds the initial ~0.
__device__ __forceinline__ void shared_topk_insert(uint32_t* A, int n, uint32_t v) {
    int p = n - 1;
    if (v >= A[p]) return;
    while (p > 0 && A[p - 1] > v) --p;  // slots before p are <= v and only ever decrease
    uint32_t c = v;
    for (int i = p; i < n && c != 0xFFFFFFFFu; ++i) {
        const uint32_t old = atomicMin(&A[i], c);
        c = old > c ? old : c;
    }
}

template <int PACK>
struct CandCtx {  // per-thread constants of the candidate slow path (lives in local memory)
    uint64_t* bufs;   // this warp's buffers [32*PACK][bcap]
    uint32_t* s_thr;  // CTA-shared exclusive bounds [32*PACK]
    uint32_t* gthr;   // global exclusive bounds
    int kp, bcap, lane;
    int qidx[PACK];
    bool valid[PACK];
    uint32_t livemask;
};
template <int PACK>
struct CandState {  // per-thread mutable state, kept in registers
    int cnt[PACK];
    uint32_t own[PACK];  // own exclusive bound (kp-th distance + 1 after a compaction)
};

// warp-uniform: compact the buffer of (lane l, half h), publish the tightened bound
template <int PACK>
__device__ __forceinline__ void cand_compact(const CandCtx<PACK>* cx, CandState<PACK>& st, int l, int h) {
    int n = __shfl_sync(0xffffffffu, st.cnt[h], l);
    uint32_t kth = 0;
    int keep = compact_buffer(cx->bufs + (size_t)(l + 32 * h) * cx->bcap, n, cx->kp, cx->lane, &kth);
    if (cx->lane == l) {
        st.cnt[h] = keep;
        if (n >= cx->kp) {
            st.own[h] = kth + 1u;
            atomicMin(&cx->s_thr[cx->lane + 32 * h], kth + 1u);
            atomicMin(&cx->gthr[cx->qidx[h]], kth + 1u);
        }
    }
}

// Window-boundary maintenance (whole warp, out of line): compact every buffer that could
// overflow during the next op window (at most `room` appends), then refresh the bounds.
template <int PACK>
__device__ __noinline__ CandState<PACK> cand_maintain(const CandCtx<PACK>* cx, CandState<PACK> st, int room) {
#pragma unroll
    for (int h = 0; h < PACK; ++h) {
        uint32_t full = __ballot_sync(0xffffffffu, st.cnt[h] + room > cx->bcap);
        while (full) {
            int l = __ffs(full) - 1;
            full &= full - 1;
            cand_compact(cx, st, l, h);
        }
    }
    return st;
}

template <int PACK>
__device__ __noinline__ CandState<PACK> cand_finish(const CandCtx<PACK>* cx, CandState<PACK> st) {
#pragma unroll
    for (int h = 0; h < PACK; ++h) {
        uint32_t todo = __ballot_sync(0xffffffffu, st.cnt[h] > 0);
        while (todo) {
            int l = __ffs(todo) - 1;
            todo &= todo - 1;
            cand_compact(cx, st, l, h);
        }
    }
    return st;
}

template <int RB, int PACK>
__global__ void __launch_bounds__(512, 1) scan_kernel(const ScanArgs a) {
    constexpr int ROWS = 1 << RB;
    constexpr int LEVELS = RB == 11 ? 8 : 16;
    constexpr uint32_t FMASK = (uint32_t)(ROWS - 1) << 2;
    constexpr int TSH = RB + 2;
    constexpr int LW = 32 * PACK;
    constexpr uint32_t XINF = PACK == 1 ? kInf31 : 0x8000u;  // exclusive bound "accept all"
    extern __shared__ __align__(128) unsigned char smem[];
    const ScanGeom& g = a.g;
    uint32_t* s_lut = reinterpret_cast<uint32_t*>(smem);
    uint4* s_ring = reinterpret_cast<uint4*>(s_lut + (size_t)g.qgl * ROWS);  // [n_warps][32]
    uint32_t* s_stack = reinterpret_cast<uint32_t*>(s_ring + (size_t)g.n_warps * 32);  // [n_warps][LEVELS][32]
    uint32_t* s_thr = s_stack + (size_t)g.n_warps * LEVELS * 32;                        // [LW]
    uint32_t* s_top = s_thr + LW;  // [LW][kps]: CTA-shared kps smallest distances per query
    int* s_next = reinterpret_cast<int*>(s_top + (size_t)LW * g.kps);
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_next + 2);

    const int item = blockIdx.x;
    const int slice = item / g.n_groups, grp = item % g.n_groups;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c_lo = (int)((int64_t)a.n_chunks * slice / g.n_slices);
    const int c_hi = (int)((int64_t)a.n_chunks * (slice + 1) / g.n_slices);

    if (threadIdx.x == 0) {
        mbar_init(s_bar, 1);
        *s_next = c_lo;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // TMA bulk copy of the group's table: qgl regions of ROWS*4 bytes
        const uint32_t bytes = (uint32_t)g.qgl * ROWS * 4u;
        mbar_expect_tx(s_bar, bytes);
        const unsigned char* src = reinterpret_cast<const unsigned char*>(a.qlut) + (size_t)grp * bytes;
        for (uint32_t o = 0; o < bytes; o += ROWS * 4u) bulk_g2s(smem + o, src + o, ROWS * 4u, s_bar);
    }

    const int ql = lane < g.qgl ? lane : g.qgl - 1;  // idle lanes alias the last region
    // a (lane, half) is valid when it maps to a real query of this group
    bool valid[PACK];
    int qidx[PACK];
    uint32_t livemask = 0;
#pragma unroll
    for (int h = 0; h < PACK; ++h) {
        qidx[h] = grp * g.qpg + h * g.qgl + lane;
        valid[h] = lane < g.qgl && qidx[h] < a.Q;
        if (valid[h]) livemask |= PACK == 1 ? 1u : (0x8000u << (16 * h));
    }
    const bool live = livemask != 0;
    if (warp == 0) {  // seed the CTA-shared bounds from the global ones (other slices)
#pragma unroll
        for (int h = 0; h < PACK; ++h) s_thr[lane + 32 * h] = valid[h] ? a.gthr[qidx[h]] : XINF;
    }
    for (int i = threadIdx.x; i < LW * g.kps; i += blockDim.x) s_top[i] = 0xFFFFFFFFu;
    __syncthreads();
    mbar_wait(s_bar, 0);

    const uint32_t Lx = ((uint32_t)ql << (RB + 2)) | ((uint32_t)ql << 2);
    const unsigned char* lutb = smem;
    uint32_t* stack = s_stack + (size_t)warp * LEVELS * 32 + lane;
    uint4* ring = s_ring + warp * 32;
#define DPQ_LUT(off) (*reinterpret_cast<const uint32_t*>(lutb + (off)))

    // candidate buffers of this warp: [LW][bcap]
    CandCtx<PACK> cx;
    cx.bufs = a.cand + ((size_t)item * g.n_warps + warp) * (size_t)LW * g.bcap;
    cx.s_thr = s_thr;
    cx.gthr = a.gthr;
    cx.kp = g.kp;
    cx.bcap = g.bcap;
    cx.lane = lane;
    cx.livemask = livemask;
    CandState<PACK> st;
    uint64_t* bp[PACK];  // this lane's buffer per half
    uint32_t xb[PACK];   // exclusive distance bound per half (0 = reject everything)
#pragma unroll
    for (int h = 0; h < PACK; ++h) {
        cx.qidx[h] = qidx[h];
        cx.valid[h] = valid[h];
        st.cnt[h] = 0;
        st.own[h] = XINF;
        bp[h] = cx.bufs + (size_t)(lane + 32 * h) * g.bcap;
        xb[h] = 0;
    }
    uint32_t thr = 0;  // PACK 1: exclusive bound; PACK 2: packed ((X-1)|0x8000) per half
    constexpr int WIN_ROOM = 16 + 1;  // appends between two maintenance points (16 quads + the root)
    const int bcap = g.bcap;
    const int kps = g.kps;
    uint32_t gb[PACK];    // last global bound seen / published
    uint32_t* topq[PACK]; // this lane's shared top-kps array per half
#pragma unroll
    for (int h = 0; h < PACK; ++h) {
        gb[h] = XINF;
        topq[h] = s_top + (size_t)(lane + 32 * h) * kps;
    }

#define DPQ_IS_CAND(d) (PACK == 1 ? ((d) < thr) : (((thr - (d)) & livemask) != 0u))
    // inline append (no call in the hot loop): one store + counter bump per accepted half
#define DPQ_APPEND(d, p)                                                              \
    {                                                                                 \
        _Pragma("unroll") for (int h = 0; h < PACK; ++h) {                            \
            const uint32_t dh = PACK == 1 ? (d) : (((d) >> (16 * h)) & 0xFFFFu);      \
            if (dh < xb[h]) {                                                         \
                bp[h][st.cnt[h]] = ((uint64_t)dh << 32) | (p);                        \
                ++st.cnt[h];                                                          \
                if (kps) shared_topk_insert(topq[h], kps, dh);                        \
            }                                                                         \
        }                                                                             \
    }
    // window boundary: make room for WIN_ROOM appends, then reload the shared bounds
#define DPQ_WINDOW_BOUNDARY()                                                         \
    {                                                                                 \
        bool tight = false;                                                           \
        _Pragma("unroll") for (int h = 0; h < PACK; ++h) tight |= st.cnt[h] + WIN_ROOM > bcap; \
        if (__any_sync(0xffffffffu, tight)) st = cand_maintain(&cx, st, WIN_ROOM);    \
        _Pragma("unroll") for (int h = 0; h < PACK; ++h) {                            \
            uint32_t x = min(st.own[h], s_thr[lane + 32 * h]);                        \
            if (kps) {                                                                \
                const uint32_t t = topq[h][kps - 1];                                  \
                if (t < x) x = t + 1u; /* ties stay candidates */                     \
            }                                                                         \
            if (valid[h] && x < gb[h]) { /* publish to the other slices */            \
                atomicMin(&a.gthr[qidx[h]], x);                                       \
                gb[h] = x;                                                            \
            }                                                                         \
            xb[h] = valid[h] ? x : 0u;                                                \
        }                                                                             \
        if (PACK == 1) {                                                              \
            thr = xb[0];                                                              \
        } else {                                                                      \
            const uint32_t x0 = valid[0] ? xb[0] : 1u, x1 = valid[PACK - 1] ? xb[PACK - 1] : 1u; \
            thr = ((x0 - 1u) | 0x8000u) | (((x1 - 1u) | 0x8000u) << 16);              \
        }                                                                             \
    }

    // 8 table reads of one quad -> signed sum of (new - old) over its 4 ops (zero ops cancel)
#define DPQ_QUAD_DELTA(Q, OUT)                                                        \
    {                                                                                 \
        const uint32_t f0 = DPQ_LUT(((Q).x & FMASK) ^ Lx), t0 = DPQ_LUT((((Q).x >> TSH) & FMASK) ^ Lx); \
        const uint32_t f1 = DPQ_LUT(((Q).y & FMASK) ^ Lx), t1 = DPQ_LUT((((Q).y >> TSH) & FMASK) ^ Lx); \
        const uint32_t f2 = DPQ_LUT(((Q).z & FMASK) ^ Lx), t2 = DPQ_LUT((((Q).z >> TSH) & FMASK) ^ Lx); \
        const uint32_t f3 = DPQ_LUT(((Q).w & FMASK) ^ Lx), t3 = DPQ_LUT((((Q).w >> TSH) & FMASK) ^ Lx); \
        OUT = (t0 - f0 + t1) + (t2 - f1 - f2) + (t3 - f3);                            \
    }

    for (;;) {
        int c = 0;
        if (lane == 0) c = atomicAdd(s_next, 1);
        c = __shfl_sync(0xffffffffu, c, 0);
        if (c >= c_hi) break;
        const ChunkDesc cd = a.chunks[c];
        const int n_anc = (int)(cd.n_anc_flags & 0xFFu);
        const uint4* qp = a.ops + cd.quad_begin;
        const int n_quads = (int)cd.n_quads;
        // op ring: 32 quads in two halves of 16; the whole ring is filled up front, then the
        // half the consumer has left is refilled from `pre` (loaded one half ahead)
        uint4 pre = make_uint4(0, 0, 0, 0);
        if (lane < n_quads) pre = __ldg(qp + lane);
#pragma unroll
        for (int h = 0; h < PACK; ++h)
            if (valid[h]) {  // bounds published by other slices of this query group
                const uint32_t gx = __ldcg(&a.gthr[qidx[h]]);
                if (gx < gb[h]) {
                    gb[h] = gx;
                    atomicMin(&s_thr[lane + 32 * h], gx);
                }
            }
        DPQ_WINDOW_BOUNDARY()
        // chunk prologue: full M-term sums for the ancestors of the first node
        uint32_t par = 0;
        {
            const uint8_t* anc = a.anc + (size_t)c * LEVELS * g.M;
            for (int lev = 0; lev < n_anc; ++lev) {
                uint32_t d = 0;
                for (int m = 0; m < g.M; ++m) {
                    uint32_t row4 = (uint32_t)(m * g.K + anc[lev * g.M + m]) << 2;
                    d += DPQ_LUT(row4 ^ Lx);
                }
                stack[lev * 32] = d;
                par = d;
                if (lev == 0 && (cd.n_anc_flags & CHUNK_EMIT_ROOT)) {
                    if (__any_sync(0xffffffffu, DPQ_IS_CAND(d))) DPQ_APPEND(d, 0u)
                }
            }
        }
        __syncwarp();  // every lane is done with the previous chunk's ring
        ring[lane] = pre;
        __syncwarp();
        int filled = 32;
        if (lane < 16 && filled + lane < n_quads) pre = __ldg(qp + filled + lane);
        uint32_t pos = cd.first_pos;
        int p = 0;
        uint4 A = ring[0];
        while (p < n_quads) {
            if (p >= filled - 16 && filled < n_quads) {  // left a half behind: refill it
                DPQ_WINDOW_BOUNDARY()
                __syncwarp();
                if (lane < 16) ring[(filled & 31) + lane] = pre;
                __syncwarp();
                filled += 16;
                if (lane < 16 && filled + lane < n_quads) pre = __ldg(qp + filled + lane);
            }
            const uint32_t w0 = A.x;
            const int nq = (int)(w0 >> 30) + 1;
            const int pn = p + nq;
            const uint4 An = ring[pn & 31];  // next record's first quad, requested early
            uint32_t delta;
            DPQ_QUAD_DELTA(A, delta)
            for (int e = 1; e < nq; ++e) {
                const uint4 B = ring[(p + e) & 31];
                uint32_t dB;
                DPQ_QUAD_DELTA(B, dB)
                delta += dB;
            }
            const uint32_t d = par + delta;
            if (__any_sync(0xffffffffu, DPQ_IS_CAND(d))) DPQ_APPEND(d, pos)
            if (w0 & (OP_CHILD | OP_AUX)) {
                const uint32_t lev = (w0 & 3u) | ((w0 >> RB) & 0xCu);
                if (w0 & OP_CHILD) {
                    par = d;
                    if (w0 & OP_AUX) stack[lev * 32] = d;
                } else {
                    par = stack[lev * 32];
                }
            }
            ++pos;
            p = pn;
            A = An;
        }
    }
#undef DPQ_QUAD_DELTA
#undef DPQ_LUT
#undef DPQ_IS_CAND
#undef DPQ_APPEND
#undef DPQ_WINDOW_BOUNDARY
    // final compaction: every buffer becomes a sorted list of at most kp keys
    st = cand_finish(&cx, st);
#pragma unroll
    for (int h = 0; h < PACK; ++h)
        a.cand_cnt[((size_t)item * g.n_warps + warp) * LW + lane + 32 * h] = (uint32_t)st.cnt[h];
}

cudaError_t launch_scan(const ScanArgs& a, cudaStream_t st) {
    const ScanGeom& g = a.g;
    dim3 grid((unsigned)(g.n_groups * g.n_slices)), block((unsigned)(g.n_warps * 32));
    void (*k)(const ScanArgs) = nullptr;
    if (g.rb == 11 && g.pack == 1) k = scan_kernel<11, 1>;
    else if (g.rb == 11 && g.pack == 2) k = scan_kernel<11, 2>;
    else if (g.rb == 12 && g.pack == 1) k = scan_kernel<12, 1>;
    else if (g.rb == 12 && g.pack == 2) k = scan_kernel<12, 2>;
    else return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem_bytes);
    if (e != cudaSuccess) return e;
    k<<<grid, block, g.smem_bytes, st>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------ select -------
// One warp per query: k'-way merge of the per-(slice, warp) sorted candidate lists, exact
// re-score of the k' winners, sort by (exact distance, position), margin check.
constexpr int SEL_WARPS = 4;
constexpr int SEL_MAXKP = 256;
constexpr int SEL_MAXLISTS_PER_LANE = 64;

__global__ void __launch_bounds__(SEL_WARPS * 32) select_kernel(const SelectArgs a) {
    __shared__ uint64_t s_sel[SEL_WARPS][SEL_MAXKP];
    __shared__ uint64_t s_exact[SEL_WARPS][SEL_MAXKP];
    const ScanGeom& g = a.g;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int q = blockIdx.x * SEL_WARPS + w;
    if (q >= a.Q) return;
    const int LW = a.v2 ? g.qpg : 32 * g.pack;
    const int grp = q / g.qpg, sub = q % g.qpg;
    const int sl = a.v2 ? sub : (sub % g.qgl) + 32 * (sub / g.qgl);
    const int lists_per_item = a.v2 ? 1 : g.n_warps;  // v2: one CTA-wide list per (slice, query)
    const int n_lists = g.n_slices * lists_per_item;
    const int kp = g.kp;

    // cursors over this lane's lists (list id = lane + 32*j)
    uint16_t cur[SEL_MAXLISTS_PER_LANE];
    uint16_t len[SEL_MAXLISTS_PER_LANE];
    const int my = (n_lists - lane + 31) / 32;
    auto list_base = [&](int id) -> const uint64_t* {
        int s = id / lists_per_item, ww = id % lists_per_item;
        size_t item = (size_t)s * g.n_groups + grp;
        return a.cand + ((item * lists_per_item + ww) * (size_t)LW + sl) * g.bcap;
    };
    for (int j = 0; j < my; ++j) {
        int id = lane + 32 * j;
        int s = id / lists_per_item, ww = id % lists_per_item;
        size_t item = (size_t)s * g.n_groups + grp;
        len[j] = (uint16_t)a.cand_cnt[(item * lists_per_item + ww) * LW + sl];
        cur[j] = 0;
    }
    int n_sel = 0;
    for (int r = 0; r < kp; ++r) {
        uint64_t best = ~0ull;
        int bj = -1;
        for (int j = 0; j < my; ++j)
            if (cur[j] < len[j]) {
                uint64_t k = list_base(lane + 32 * j)[cur[j]];
                if (k < best) {
                    best = k;
                    bj = j;
                }
            }
        uint64_t m = best;
        for (int o = 16; o; o >>= 1) {
            uint64_t t = __shfl_xor_sync(0xffffffffu, m, o);
            m = t < m ? t : m;
        }
        if (m == ~0ull) break;
        if (best == m && bj >= 0) cur[bj]++;  // keys are unique (position is part of the key)
        if (lane == 0) s_sel[w][r] = m;
        n_sel = r + 1;
    }
    __syncwarp();
    // exact re-score: float(sum in double of the node's M float table entries)
    const float* lut = a.lutf + (size_t)q * g.M * g.K;
    for (int j = lane; j < n_sel; j += 32) {
        uint32_t pos = (uint32_t)s_sel[w][j];
        const uint8_t* code = a.codes + (size_t)((int64_t)pos - a.base_pos) * a.cstride;
        const double d = exact_dist(lut, code, a.cstride, g.M, g.K);
        s_exact[w][j] = ((uint64_t)__float_as_uint((float)d) << 32) | pos;
    }
    __syncwarp();
    // rank sort (keys unique) and output
    uint64_t kth_exact = 0;
    for (int j = lane; j < n_sel; j += 32) {
        uint64_t k = s_exact[w][j];
        int rank = 0;
        for (int i = 0; i < n_sel; ++i) rank += s_exact[w][i] < k;
        if (rank < a.topk) a.out_key[(size_t)q * a.topk + rank] = k;
        if (rank == a.topk - 1) kth_exact = k;
    }
    for (int j = n_sel + lane; j < a.topk; j += 32)
        a.out_key[(size_t)q * a.topk + j] = ((uint64_t)__float_as_uint(FLT_MAX) << 32) | 0xFFFFFFFFull;
    for (int o = 16; o; o >>= 1) {
        uint64_t t = __shfl_xor_sync(0xffffffffu, kth_exact, o);
        kth_exact = t > kth_exact ? t : kth_exact;
    }
    if (lane == 0) {
        // Every node NOT among the k' winners has fixed-point distance >= G (the k'-th).
        // Its exact distance is >= (G - E) / scale with E = M/2 + 2 rounding units.
        uint32_t flag = 0;
        float bound = FLT_MAX;
        if (n_sel >= a.topk) bound = __uint_as_float((uint32_t)(kth_exact >> 32));
        if (n_sel == kp) {
            double G = (double)(uint32_t)(s_sel[w][kp - 1] >> 32);
            double E = 0.5 * g.M + 2.0;
            if (!((double)bound * a.scale[q] + E < G)) flag = 1;
        }
        if (a.force_fallback) flag = 1;
        if (a.v2 && a.ovf[(size_t)grp * g.qpg + sub]) flag = 1;  // dropped candidates: redo exactly
        a.bound[q] = bound;
        if (flag) {
            uint32_t slot = atomicAdd(a.n_flagged, 1u);
            if (slot < (uint32_t)a.max_flagged) a.flagged[slot] = (uint32_t)q;
        }
    }
}

void launch_select(const SelectArgs& a, cudaStream_t st) {
    int blocks = (a.Q + SEL_WARPS - 1) / SEL_WARPS;
    select_kernel<<<blocks, SEL_WARPS * 32, 0, st>>>(a);
}

// ------------------------------------------------------------------------ fallback -----
// Exact plain ADC scan over the decoded codes for the (rare) flagged queries: one CTA per
// flagged query walks every node of the shard, scores it in the reference's arithmetic (float
// table entries, double sum) and keeps a running top-k in shared memory.  The acceptance test is
// on the full 64-bit key (distance bits << 32 | position, strict), so any number of nodes tying
// at the k-th distance is handled: the buffer is reduced to the k best keys (bitonic sort)
// whenever it is more than half full, and the k-th key becomes the new exclusive bound.
constexpr int FB_T = 1024;  // FB_BUF (kernels.cuh) >= FB_T + 256 (topk <= 256)

// grid = (slices, query slots): block (s, y) scans slice s of the shard for the flagged queries y, y + gridDim.y, ...
// and leaves its k best keys in part[f][s][topk]; fallback_merge_kernel sorts a query's slices together.
// DEAD: nodes whose bit is set in a.dead are skipped.
template <bool DEAD>
__global__ void __launch_bounds__(FB_T) fallback_kernel(const FallbackArgs a) {
    extern __shared__ __align__(16) unsigned char fb_smem[];
    uint64_t* s_keys = reinterpret_cast<uint64_t*>(fb_smem);  // [FB_BUF]
    float* s_lut = reinterpret_cast<float*>(s_keys + FB_BUF);  // [M*K]
    __shared__ uint32_t s_n;
    __shared__ unsigned long long s_thr;
    const int n_flagged = min((int)*a.n_flagged, a.max_flagged);
    const int MK = a.M * a.K;
    const int slice = blockIdx.x, n_slices = gridDim.x;
    const int64_t lo = a.n_local * slice / n_slices, hi = a.n_local * (slice + 1) / n_slices;
    for (int f = blockIdx.y; f < n_flagged; f += gridDim.y) {
        const uint32_t q = a.flagged[f];
        stage_table(s_lut, a.lutf + (size_t)q * MK, MK, threadIdx.x, FB_T);
        if (threadIdx.x == 0) {
            s_n = 0u;
            // inclusive bound: every node with distance <= bound[q] (any position) is a candidate
            s_thr = ((unsigned long long)__float_as_uint(a.bound[q]) << 32) | 0xFFFFFFFFull;
        }
        __syncthreads();
        for (int64_t base = lo; base < hi; base += FB_T) {
            const int64_t i = base + threadIdx.x;
            if (i < hi && !(DEAD && node_dead(a.dead, (uint32_t)i))) {
                const uint8_t* code = a.codes + (size_t)i * a.cstride;
                const double d = exact_dist(s_lut, code, a.cstride, a.M, a.K);
                const uint64_t key = ((uint64_t)__float_as_uint((float)d) << 32) | (uint32_t)(i + a.base_pos);
                if (key <= s_thr) s_keys[atomicAdd(&s_n, 1u)] = key;  // < FB_BUF: compacted above FB_BUF - FB_T
            }
            __syncthreads();
            if (s_n > (uint32_t)(FB_BUF - FB_T)) fb_compact(s_keys, &s_n, &s_thr, a.topk);
        }
        fb_compact(s_keys, &s_n, &s_thr, a.topk);
        uint64_t* part = a.part + ((size_t)f * n_slices + slice) * a.topk;
        for (int i = threadIdx.x; i < a.topk; i += FB_T) part[i] = i < (int)s_n ? s_keys[i] : ~0ull;
        __syncthreads();
    }
}

// one CTA per flagged query: the slices' k best keys (<= FB_BUF of them) sorted together -> out_key
__global__ void __launch_bounds__(256) fallback_merge_kernel(const FallbackArgs a, int n_slices) {
    __shared__ uint64_t s_keys[FB_BUF];
    __shared__ uint32_t s_n;
    __shared__ unsigned long long s_thr;
    const int n_flagged = min((int)*a.n_flagged, a.max_flagged);
    for (int f = blockIdx.x; f < n_flagged; f += gridDim.x) {
        const uint32_t q = a.flagged[f];
        const int total = n_slices * a.topk;
        const uint64_t* part = a.part + (size_t)f * total;
        for (int i = threadIdx.x; i < total; i += blockDim.x) s_keys[i] = part[i];
        if (threadIdx.x == 0) {
            s_n = (uint32_t)total;  // empty slots are ~0 keys: they sort to the end
            s_thr = ~0ull;
        }
        __syncthreads();
        fb_compact(s_keys, &s_n, &s_thr, a.topk);
        for (int i = threadIdx.x; i < a.topk; i += blockDim.x)
            a.out_key[(size_t)q * a.topk + i] =
                s_keys[i] != ~0ull ? s_keys[i] : (((uint64_t)__float_as_uint(FLT_MAX) << 32) | 0xFFFFFFFFull);
        __syncthreads();
    }
}

// Latency mode: exact re-score of scan1's candidate lists.  A query's list is cut into gridDim.y ranges, one
// CTA each (a handful of queries must still fill the machine); the last CTA of a query to arrive merges the
// ranges' k best (same running top-k).
constexpr int R1_T = 256;
__global__ void __launch_bounds__(R1_T) rescore1_kernel(const Rescore1Args a) {
    extern __shared__ __align__(16) unsigned char fb_smem[];
    uint64_t* s_keys = reinterpret_cast<uint64_t*>(fb_smem);   // [FB_BUF]
    float* s_lut = reinterpret_cast<float*>(s_keys + FB_BUF);  // [M*K]
    __shared__ uint32_t s_n;
    __shared__ unsigned long long s_thr;
    __shared__ int s_last, s_real;
    const int q = blockIdx.x, part = blockIdx.y, n_parts = gridDim.y;
    const int MK = a.M * a.K;
    stage_table(s_lut, a.lutf + (size_t)q * MK, MK, threadIdx.x, R1_T);
    if (threadIdx.x == 0) {
        s_n = 0u;
        s_thr = ~0ull;
        s_real = 0;
    }
    __syncthreads();
    const int total = (int)min(a.cand_cnt[q], (uint32_t)a.ccap);
    const int lo = (int)((int64_t)total * part / n_parts), hi = (int)((int64_t)total * (part + 1) / n_parts);
    const uint32_t* cand = a.cand + (size_t)q * a.ccap;
    for (int base = lo; base < hi; base += R1_T) {
        const int i = base + threadIdx.x;
        if (i < hi) {
            const uint32_t pos = cand[i];
            const uint8_t* code = a.codes + (size_t)((int64_t)pos - a.base_pos) * a.cstride;
            const double d = exact_dist(s_lut, code, a.cstride, a.M, a.K);
            const uint64_t key = ((uint64_t)__float_as_uint((float)d) << 32) | pos;
            if (key <= s_thr) s_keys[atomicAdd(&s_n, 1u)] = key;
        }
        __syncthreads();
        if (s_n > (uint32_t)max(256, 2 * a.topk)) fb_compact(s_keys, &s_n, &s_thr, a.topk);  // early: small sorts, tight bound
    }
    fb_compact(s_keys, &s_n, &s_thr, a.topk);
    const int k = a.topk;
    if (n_parts > 1) {
        uint64_t* mine = a.part + ((size_t)q * n_parts + part) * k;
        for (int i = threadIdx.x; i < k; i += R1_T) mine[i] = i < (int)s_n ? s_keys[i] : ~0ull;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = atomicAdd(&a.part_done[q], 1u) == (uint32_t)(n_parts - 1);
        __syncthreads();
        if (!s_last) return;
        __threadfence();
        const uint64_t* all = a.part + (size_t)q * n_parts * k;
        for (int i = threadIdx.x; i < n_parts * k; i += R1_T) s_keys[i] = __ldcg(all + i);
        if (threadIdx.x == 0) {
            s_n = (uint32_t)(n_parts * k);  // empty slots are ~0 keys: they sort to the end
            s_thr = ~0ull;
            a.part_done[q] = 0u;
        }
        __syncthreads();
        fb_compact(s_keys, &s_n, &s_thr, k);
    }
    int c = 0;
    for (int i = threadIdx.x; i < (int)s_n; i += R1_T) c += s_keys[i] != ~0ull;
    if (c) atomicAdd(&s_real, c);
    __syncthreads();
    const int n = s_real;
    if (a.out_key)
        for (int i = threadIdx.x; i < k; i += R1_T)
            a.out_key[(size_t)q * k + i] = i < n ? s_keys[i] : (((uint64_t)__float_as_uint(FLT_MAX) << 32) | 0xFFFFFFFFull);
    if (threadIdx.x == 0) {
        // the k best found are real nodes: their k-th distance bounds the true k-th from above
        const float found = n >= k ? __uint_as_float((uint32_t)(s_keys[k - 1] >> 32)) : FLT_MAX;
        const float known = a.cap_in ? a.cap_in[q] : FLT_MAX;
        const float cap = fminf(found, known);
        if (a.cap_out) a.cap_out[q] = cap;
        if (a.flagged) {
            a.bound[q] = cap;
            if (a.ovf[q]) {  // dropped candidates may hide a true top-k node: exact fallback
                const uint32_t slot = atomicAdd(a.n_flagged, 1u);
                if (slot < (uint32_t)a.max_flagged) a.flagged[slot] = (uint32_t)q;
            }
        }
    }
}

void launch_rescore1(const Rescore1Args& a, cudaStream_t st) {
    const size_t sm = (size_t)FB_BUF * sizeof(uint64_t) + (size_t)a.M * a.K * sizeof(float);
    rescore1_kernel<<<dim3((unsigned)a.Q, (unsigned)(a.n_parts > 1 ? a.n_parts : 1)), R1_T, sm, st>>>(a);
}

void launch_fallback(const FallbackArgs& a, cudaStream_t st) {
    // Always enqueued: the kernel reads the flagged count on the device and exits at once when it
    // is zero, so the common path needs no host round trip.
    // The shard is cut into slices so that a handful of flagged queries still fill the machine.
    const size_t sm = (size_t)FB_BUF * sizeof(uint64_t) + (size_t)a.M * a.K * sizeof(float);
    const int n_slices = fallback_slices(a.topk);
    const int qslots = a.max_flagged < 64 ? a.max_flagged : 64;
    (a.dead ? fallback_kernel<true> : fallback_kernel<false>)<<<dim3((unsigned)n_slices, (unsigned)qslots), FB_T, sm, st>>>(a);
    fallback_merge_kernel<<<a.max_flagged < 296 ? a.max_flagged : 296, 256, 0, st>>>(a, n_slices);
}

// ------------------------------------------------------------------------ merge --------
__global__ void merge_kernel(const uint64_t* __restrict__ keys, int n_lists, int Q, int topk,
                             uint64_t* __restrict__ out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    int cur[64];
    for (int l = 0; l < n_lists; ++l) cur[l] = 0;
    for (int r = 0; r < topk; ++r) {
        uint64_t best = ~0ull;
        int bl = -1;
        for (int l = 0; l < n_lists; ++l)
            if (cur[l] < topk) {
                uint64_t k = keys[((size_t)l * Q + q) * topk + cur[l]];
                if (k < best) {
                    best = k;
                    bl = l;
                }
            }
        if (bl >= 0) cur[bl]++;
        out[(size_t)q * topk + r] =
            bl >= 0 ? best : (((uint64_t)__float_as_uint(FLT_MAX) << 32) | 0xFFFFFFFFull);
    }
}

__global__ void unpack_kernel(const uint64_t* __restrict__ keys, size_t n, const uint32_t* __restrict__ pos2id,
                              uint32_t base_pos, uint32_t* __restrict__ out_pos, uint32_t* __restrict__ out_id,
                              uint32_t* __restrict__ out_dist, const uint32_t* __restrict__ ctrl, uint32_t* __restrict__ out_ctrl) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 4 && out_ctrl) out_ctrl[i] = ctrl ? ctrl[i] : 0u;
    if (i >= n) return;
    const uint64_t k = keys[i];
    const uint32_t pos = (uint32_t)k;
    if (out_pos) out_pos[i] = pos;
    if (out_id) out_id[i] = (pos2id && pos != 0xFFFFFFFFu) ? pos2id[pos - base_pos] : pos;
    if (out_dist) out_dist[i] = (uint32_t)(k >> 32);
}

void launch_unpack(const uint64_t* d_keys, size_t n, const uint32_t* d_pos2id, uint32_t base_pos, uint32_t* out_pos,
                   uint32_t* out_id, uint32_t* out_dist, const uint32_t* d_ctrl, uint32_t* out_ctrl, cudaStream_t st) {
    unpack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_keys, n, d_pos2id, base_pos, out_pos, out_id, out_dist, d_ctrl,
                                                                out_ctrl);
}

void launch_merge(const uint64_t* d_keys, int n_lists, int Q, int topk, uint64_t* d_out,
                  cudaStream_t st) {
    merge_kernel<<<(Q + 127) / 128, 128, 0, st>>>(d_keys, n_lists, Q, topk, d_out);
}

}  // namespace dpq
