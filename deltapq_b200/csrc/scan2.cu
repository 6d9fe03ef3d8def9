// Second-generation DeltaTree scan for sm_100a (M <= 16): the 15-bit fixed-point scan.
//
// What the first-generation kernel's ncu capture showed (profiles/r1_summary.md): that scan is
// bound by instruction issue, not by shared-memory wavefronts or HBM: 136 warp instructions per
// node for 48 queries, most of it per-node control (variable-length records, depth stack, ring
// refills) and address arithmetic for one 32-bit table read per (lane, lookup).  This kernel
// removes that overhead structurally:
//
//   * the shard is its nodes' PQ codes by DFS position, 8 (M <= 8) or 16 bytes per node
//     (dpq_internal.h "v2"); every node gets the full M-term lookup -- the delta rule would read
//     2 x 4.3..5.2 table rows per node instead of 8 -- so there is no record decoding, no depth
//     stack and no dependence between nodes;
//   * the warp is four quarter-warp STRANDS (eight 4-lane strands in the wide shape), each
//     walking its own 64-node chunk, so one instruction advances four (eight) nodes;
//   * the fixed-point ADC table is laid out [m * 256 + centroid][56 queries] (112-byte rows) and
//     read with 128-bit loads: lane j of a strand gets queries 8j..8j+7 of the row in one
//     LDS.128, the lanes of a strand cover one contiguous row = one conflict-free wavefront; the
//     row address is centroid * row_bytes + base (one IMAD), the subspace offset m * 256 * row_bytes
//     is the load's immediate;
//   * all arithmetic is packed 2 x 15-bit in 32-bit integer adds (exact, see kernels.cu);
//   * top-k: CTA-wide candidate buffers (one per query, in global scratch) appended with one
//     shared-memory atomic + one store; at epoch boundaries (every 128 iterations, ramping up
//     from 1) a CTA barrier lets the owner warp of a query compact its buffer to the k' best and
//     tighten the bound, which is shared through shared memory (CTA) and global memory (the
//     other tree slices of the same query group).
//
// The table for 56 queries fills shared memory (229,376 of 232,448 bytes); the codes stream from
// L2/HBM through L1 with one 8- or 16-byte load per strand per node.
#include "kernels.cuh"

#include <cfloat>
#include <type_traits>

namespace dpq {

namespace {

constexpr int MAXQB = 64;  // s_thr / s_cnt slots (56 or 24 used)

}  // namespace

// ------------------------------------------------------------------------ ADC tables ---
// Exact float tables [Q][M*K] (reference arithmetic, DCAT.h:3754-3757, same expression as
// adc_entry).  Block = (8 queries, one subspace) x one thread per centroid: every codebook value is
// loaded once and feeds eight independent accumulation chains (the chain is a dependent
// float -> double -> float sequence, so the eight queries are the ILP).  One subspace per block keeps
// the grid at (Q / 8) * M short blocks: with whole queries per block (1250 blocks of 256 threads at
// C2, four or five resident per SM) the last wave ran a third full.
// mmax[q][16]: the per-subspace maxima of the table (scale2_kernel derives the 15-bit scale from them).
constexpr int LUT2_QPB = 8;
__global__ void __launch_bounds__(256) lut2_kernel(const float* __restrict__ cw, int M, int K, int Ds,
                                                   const float* __restrict__ queries, int Q,
                                                   float* __restrict__ lutf, float* __restrict__ mmax) {
    extern __shared__ __align__(16) float s_q[];  // [Ds][LUT2_QPB]: the eight queries' values of one dimension are adjacent
    __shared__ int s_max[LUT2_QPB];
    const int q0 = blockIdx.x * LUT2_QPB;
    const int m = blockIdx.y;
    const int k = threadIdx.x;
    const int D = M * Ds;
    for (int i = k; i < LUT2_QPB * Ds; i += blockDim.x) {
        const int j = i / Ds, d = i % Ds;  // contiguous global reads per query, transposed store
        const int q = q0 + j;
        s_q[d * LUT2_QPB + j] = q < Q ? queries[(size_t)q * D + m * Ds + d] : 0.0f;
    }
    if (k < LUT2_QPB) s_max[k] = 0;
    __syncthreads();
    float acc[LUT2_QPB];
#pragma unroll
    for (int j = 0; j < LUT2_QPB; ++j) acc[j] = 0.0f;
    if (k < K) {
        // The accumulator is rounded to float after every term INSIDE the double domain (add and
        // subtract 2^(E+29), see round_to_float_in_double): branch free, one F2F per term instead of
        // three.  The sum only grows, so the rare ranges where that shortcut differs from the float
        // conversion are detected per chain -- a nonzero partial sum below 2^-126 (float subnormals
        // keep fewer bits) or a final value from 2^127 up (the conversion may overflow) -- and such an
        // entry is recomputed by adc_entry, which takes the conversion path.
        double accd[LUT2_QPB];
        unsigned emin[LUT2_QPB];  // smallest (exponent field - 1) seen by the chain; a zero sum wraps to the top
#pragma unroll
        for (int j = 0; j < LUT2_QPB; ++j) {
            accd[j] = 0.0;
            emin[j] = 0xFFFFFFFFu;
        }
        const float* c = cw + ((size_t)m * K + k) * Ds;
        const float4* qrow = reinterpret_cast<const float4*>(s_q);
        auto term = [&](int d, float cv) {
            const float4 qa = qrow[2 * d], qb = qrow[2 * d + 1];
            const float qv[LUT2_QPB] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w};
#pragma unroll
            for (int j = 0; j < LUT2_QPB; ++j) {
                const double diff = (double)__fsub_rn(cv, qv[j]);
                // diff is a widened float: diff * diff is exact in double, so one fused multiply-add
                // rounds exactly like the reference's multiply then add
                const double sum = __fma_rn(diff, diff, accd[j]);
                const int e = __double2hiint(sum) & 0x7FF00000;
                emin[j] = min(emin[j], (unsigned)e - 1u);
                const double big = __hiloint2double(e + (29 << 20), 0);
                accd[j] = __dsub_rn(__dadd_rn(sum, big), big);
            }
        };
        if ((Ds & 3) == 0) {  // the centroid's values four at a time, the next four in flight
            const float4* c4 = reinterpret_cast<const float4*>(c);
            float4 nxt = __ldg(c4);
            for (int d4 = 0; d4 < Ds / 4; ++d4) {
                const float4 cur = nxt;
                if (d4 + 1 < Ds / 4) nxt = __ldg(c4 + d4 + 1);
                term(4 * d4, cur.x);
                term(4 * d4 + 1, cur.y);
                term(4 * d4 + 2, cur.z);
                term(4 * d4 + 3, cur.w);
            }
        } else {
            for (int d = 0; d < Ds; ++d) term(d, c[d]);
        }
#pragma unroll
        for (int j = 0; j < LUT2_QPB; ++j) {
            // 0 < some partial sum < 2^-126, or a final value from 2^127 up: the conversion path decides
            if (emin[j] < 0x38100000u - 1u || (__double2hiint(accd[j]) & 0x7FF00000) >= 0x47E00000) {
                float r = 0.0f;
                for (int d = 0; d < Ds; ++d) {
                    const float diff = __fsub_rn(c[d], s_q[d * LUT2_QPB + j]);
                    r = (float)__dadd_rn((double)r, __dmul_rn((double)diff, (double)diff));
                }
                acc[j] = r;
            } else {
                acc[j] = (float)accd[j];
            }
        }
    }
#pragma unroll
    for (int j = 0; j < LUT2_QPB; ++j) {
        if (k < K && q0 + j < Q) lutf[(size_t)(q0 + j) * M * K + m * K + k] = acc[j];
        int vi = __float_as_int(acc[j]);  // >= 0: integer order == float order
        vi = __reduce_max_sync(0xffffffffu, vi);
        if ((k & 31) == 0) atomicMax(&s_max[j], vi);
    }
    __syncthreads();
    if (k < LUT2_QPB && q0 + k < Q) mmax[(size_t)(q0 + k) * 16 + m] = __int_as_float(s_max[k]);
}

// 15-bit fixed-point scale per query from the per-subspace maxima (the 15-bit scan only)
__global__ void scale2_kernel(const float* __restrict__ mmax, int M, int Q, double* __restrict__ scale) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    double sum = 0.0;
    for (int m = 0; m < M; ++m) sum += (double)mmax[(size_t)q * 16 + m];
    scale[q] = sum > 0.0 ? (double)(32767 - 16) / sum : 0.0;  // NaN or 0: scale 0, the filter passes every node
}

// Small batches (latency mode): one block per (query, subspace), so that even a single query spreads
// over M SMs and the dependent accumulation chain is Ds long instead of M * Ds.  Same arithmetic.
// mmax[q][16]: the per-subspace maxima (the fixed-point scale is derived from their sum).
__global__ void __launch_bounds__(256) lut_small_kernel(const float* __restrict__ cw, int M, int K, int Ds,
                                                        const float* __restrict__ queries, float* __restrict__ lutf,
                                                        float* __restrict__ mmax) {
    extern __shared__ float s_q[];  // [Ds]
    __shared__ int s_max;
    const int q = blockIdx.x, m = blockIdx.y, k = threadIdx.x;
    const int D = M * Ds;
    for (int i = k; i < Ds; i += blockDim.x) s_q[i] = queries[(size_t)q * D + m * Ds + i];
    if (k == 0) s_max = 0;
    __syncthreads();
    float acc = 0.0f;
    if (k < K) {
        acc = adc_entry(cw + ((size_t)m * K + k) * Ds, s_q, Ds);
        lutf[(size_t)q * M * K + m * K + k] = acc;
    }
    int vi = __float_as_int(acc);  // >= 0: integer order == float order
    for (int o = 16; o; o >>= 1) vi = max(vi, __shfl_xor_sync(0xffffffffu, vi, o));
    if ((k & 31) == 0) atomicMax(&s_max, vi);
    __syncthreads();
    if (k == 0) mmax[q * 16 + m] = __int_as_float(s_max);
}

void launch_lut_small(const float* d_cw, int M, int K, int Ds, const float* d_queries, int Q, float* d_lutf, float* d_mmax,
                      cudaStream_t st) {
    lut_small_kernel<<<dim3((unsigned)Q, (unsigned)M), 256, (size_t)Ds * sizeof(float), st>>>(d_cw, M, K, Ds, d_queries, d_lutf, d_mmax);
}

// Quantise + transpose into the scan layout [group][m * 256 + centroid][QB] u16; rows of subspaces
// >= M or centroids >= K and queries >= Q are zero.  Block = 64 rows of one group; reads and writes are both coalesced.
__global__ void __launch_bounds__(256) pack2_kernel(const float* __restrict__ lutf, const double* __restrict__ scale,
                                                    int M, int K, int Q, int QB, int rows, uint16_t* __restrict__ qlut,
                                                    uint32_t* __restrict__ gthr, uint32_t* __restrict__ ovf,
                                                    uint32_t bound0) {
    const int MK = M * K;
    __shared__ uint16_t tile[64 * MAXQB];
    const int grp = blockIdx.x, row0 = blockIdx.y * 64;
    for (int i = threadIdx.x; i < 64 * QB; i += blockDim.x) {
        const int ql = i >> 6, r = i & 63;
        const int q = grp * QB + ql, row = row0 + r;
        uint16_t v = 0;
        const int m = row >> 8, c = row & 255;  // scan-table row = m * 256 + centroid
        // clamped to the 15-bit range scale2_kernel scales to (a no-op for a finite positive sum; NaN -> 0): no
        // entry can wrap into bit 15 and carry or borrow into the neighbouring query's lane
        if (q < Q && m < M && c < K)
            v = (uint16_t)__double2ll_rn(fmin(fmax((double)lutf[(size_t)q * MK + m * K + c] * scale[q], 0.0), 32767.0 - 16.0));
        tile[r * QB + ql] = v;
    }
    __syncthreads();
    uint32_t* dst = reinterpret_cast<uint32_t*>(qlut + ((size_t)grp * rows + row0) * QB);
    const uint32_t* src = reinterpret_cast<const uint32_t*>(tile);
    for (int i = threadIdx.x; i < 64 * QB / 2; i += blockDim.x) dst[i] = src[i];
    if (blockIdx.y == 0 && threadIdx.x < QB) {
        gthr[grp * QB + threadIdx.x] = bound0;  // exclusive bound; 0x8000 = accept everything
        ovf[grp * QB + threadIdx.x] = 0u;
    }
}

void launch_lut2(const float* d_cw, int M, int K, int Ds, const float* d_queries, int Q, float* d_lutf,
                 double* d_scale, float* d_mmax, uint16_t* d_qlut, uint32_t* d_gthr, uint32_t* d_ovf, int n_groups,
                 const V2Shape& sh, uint32_t bound0, cudaStream_t st) {
    const size_t lsm = (size_t)LUT2_QPB * Ds * sizeof(float);
    if (lsm > 48 * 1024) cudaFuncSetAttribute(lut2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lsm);
    lut2_kernel<<<dim3((unsigned)((Q + LUT2_QPB - 1) / LUT2_QPB), (unsigned)M), 256, lsm, st>>>(d_cw, M, K, Ds, d_queries, Q, d_lutf,
                                                                                            d_mmax);
    if (!d_qlut) return;
    scale2_kernel<<<(Q + 255) / 256, 256, 0, st>>>(d_mmax, M, Q, d_scale);
    pack2_kernel<<<dim3((unsigned)n_groups, (unsigned)(sh.rows / 64)), 256, 0, st>>>(d_lutf, d_scale, M, K, Q, sh.qb(), sh.rows,
                                                                                    d_qlut, d_gthr, d_ovf, bound0);
}

// ------------------------------------------------------------------------ scan ---------
// warp-cooperative: keep the min(n, kp) smallest of buf[0..n), sorted ascending (keys unique)
template <int MAXPER>
__device__ __forceinline__ int compact2_t(uint64_t* buf, int n, int kp, int lane, uint32_t* kth) {
    const int per = (n + 31) >> 5;
    uint64_t mine[MAXPER];
    int rank[MAXPER];
#pragma unroll
    for (int t = 0; t < MAXPER; ++t) {
        mine[t] = ~0ull;
        rank[t] = 0;
        if (t < per) {
            int i = t * 32 + lane;
            if (i < n) mine[t] = __ldcg(buf + i);
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
            if (i < n && rank[t] < keep) __stcg(buf + rank[t], mine[t]);
            if (i < n && rank[t] == kp - 1) kd = (uint32_t)(mine[t] >> 32);
        }
    }
    for (int o = 16; o; o >>= 1) kd |= __shfl_xor_sync(0xffffffffu, kd, o);
    *kth = kd;
    __syncwarp();
    return keep;
}
__device__ __noinline__ int compact2(uint64_t* buf, int n, int kp, int lane, uint32_t* kth) {
    // more than 512 keys (bcap = 1024, kp <= 256): reduce the first 512 to their kp best, slide the
    // tail down behind them, repeat.  Keeps the register footprint of this (called) function small:
    // a 1024-key variant made the scan loop of the calling kernel spill.
    while (n > 512) {
        uint32_t dummy;
        const int keep = compact2_t<16>(buf, 512, kp, lane, &dummy);
        const int tail = n - 512;
        for (int i = 0; i < tail; i += 32) {  // destination is always below every unread key
            uint64_t v = 0;
            if (i + lane < tail) v = __ldcg(buf + 512 + i + lane);
            __syncwarp();
            if (i + lane < tail) __stcg(buf + keep + i + lane, v);
            __syncwarp();
        }
        n = keep + tail;
    }
    if (n <= 64) return compact2_t<2>(buf, n, kp, lane, kth);
    if (n <= 256) return compact2_t<8>(buf, n, kp, lane, kth);
    return compact2_t<16>(buf, n, kp, lane, kth);
}

struct Own2 {  // what an owner warp needs to compact one query's buffer
    uint64_t* cand;    // this item's buffers [56][bcap]
    uint32_t* s_cnt;
    uint32_t* s_thr;
    uint32_t* gthr;    // this group's global bounds [56]
    int kp, bcap, lane;
};
__device__ __noinline__ void own_compact(const Own2* o, int ql, int trigger) {
    int n = (int)o->s_cnt[ql];
    if (n > o->bcap) n = o->bcap;
    if (n < trigger || n == 0) return;
    __threadfence_block();
    uint32_t kth = 0;
    const int keep = compact2(o->cand + (size_t)ql * o->bcap, n, o->kp, o->lane, &kth);
    if (o->lane == 0) {
        o->s_cnt[ql] = (uint32_t)keep;
        if (n >= o->kp) {
            atomicMin(&o->s_thr[ql], kth + 1u);
            atomicMin(&o->gthr[ql], kth + 1u);
        }
    }
}

// NF table fields per node (= code stride), LPG active 16-byte lanes per strand, SW lanes per strand.
// DEAD: a.dead is the deleted-node bitmap; a deleted node is never appended, so the bounds the epoch compactions
// take from the appended candidates stay k'-th distances of live nodes.  DEAD = false is the kernel without the test.
template <int NF, int LPG, int SW, bool DEAD>
__global__ void __launch_bounds__(512, 1) scan2_kernel(const std::conditional_t<DEAD, Scan2Args, Scan2Core> a) {
    constexpr int QB = LPG * 8;                  // queries per CTA
    constexpr int ROWS = NF * 256;
    constexpr int ROWB = LPG * 16;               // table row bytes
    constexpr int LUT_BYTES = ROWS * ROWB;
    constexpr int SPW = 32 / SW;                 // strands per warp = chunks in flight per warp
    constexpr int SUB = 256 * ROWB;              // table bytes per subspace
    using CodeT = typename CodeWord<NF>::type;   // uint2 (8 codes) or uint4 (16 codes)
    extern __shared__ __align__(128) unsigned char smem[];
    uint32_t* s_thr = reinterpret_cast<uint32_t*>(smem + LUT_BYTES);  // [64] exclusive bounds
    uint32_t* s_cnt = s_thr + MAXQB;                                  // [64] candidates per query
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_cnt + MAXQB);

    const int item = blockIdx.x;
    const int slice = item / a.n_groups, grp = item % a.n_groups;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strand = lane / SW, j = lane % SW;
    const int jj = j < LPG ? j : LPG - 1;  // the idle last lane of a strand aliases its neighbour
    // slices are whole batches of SPW chunks; bt_stride > 1 walks every bt_stride-th batch only
    // (the sample pass of the coarse search)
    const int n_bt = ((a.n_chunks + SPW - 1) / SPW + a.bt_stride - 1) / a.bt_stride;
    const int b_lo = (int)((int64_t)n_bt * slice / a.n_slices);
    const int b_hi = (int)((int64_t)n_bt * (slice + 1) / a.n_slices);
    uint32_t* gthr = a.gthr + (size_t)grp * QB;

    if (threadIdx.x == 0) {
        mbar_init(s_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // TMA bulk copy of the group's table
        mbar_expect_tx(s_bar, (uint32_t)LUT_BYTES);
        const unsigned char* src = reinterpret_cast<const unsigned char*>(a.qlut) + (size_t)grp * LUT_BYTES;
        for (uint32_t o = 0; o < (uint32_t)LUT_BYTES; o += 32768u) bulk_g2s(smem + o, src + o, 32768u, s_bar);
    }
    if (threadIdx.x < MAXQB) {
        const int q = grp * QB + threadIdx.x;
        s_thr[threadIdx.x] = (threadIdx.x < QB && q < a.Q) ? __ldcg(&gthr[threadIdx.x]) : 1u;
        s_cnt[threadIdx.x] = 0u;
    }
    __syncthreads();
    mbar_wait(s_bar, 0);

    // my 8 queries: ql = jj*8 + 2k + h (word k, half h).  A dead half (idle lane, or a query
    // beyond Q in the last group) gets the bound word 0x7FFF: thr - d never has bit 15.
    uint32_t lut_base = smem_u32(smem) + (uint32_t)jj * 16u;
    asm volatile("" : "+r"(lut_base));  // keep it one register: address = lut_base + centroid * ROWB (+ immediate)
    uint64_t* my_cand = a.cand + (size_t)item * QB * a.bcap;
    Own2 own{my_cand, s_cnt, s_thr, gthr, a.kp, a.bcap, lane};
    const int trigger = a.trigger;
    const int n_live = j < LPG ? min(8, max(0, a.Q - (grp * QB + jj * 8))) : 0;  // my live queries

    uint32_t thr[4];
    auto reload_thr = [&]() {
        const uint4 t0 = *reinterpret_cast<const uint4*>(s_thr + jj * 8);
        const uint4 t1 = *reinterpret_cast<const uint4*>(s_thr + jj * 8 + 4);
        const uint32_t x[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t lo = 2 * k < n_live ? ((x[2 * k] - 1u) | 0x8000u) : 0x7FFFu;
            const uint32_t hi = 2 * k + 1 < n_live ? ((x[2 * k + 1] - 1u) | 0x8000u) : 0x7FFFu;
            thr[k] = lo | (hi << 16);
        }
    };
    reload_thr();

    const int n_rounds = (b_hi - b_lo + a.n_warps - 1) / a.n_warps;
    const int C = a.chunk_nodes;
    const CodeT* codes = reinterpret_cast<const CodeT*>(a.codes);
    int since = 0, epoch_len = a.ramp ? 1 : a.epoch;
    constexpr int PF = 128 / (int)sizeof(CodeT);  // nodes per 128-byte line

    for (int round = 0; round < n_rounds; ++round) {
        const int bt = b_lo + round * a.n_warps + warp;
        const int c = bt * a.bt_stride * SPW + strand;
        int n_nodes = 0;
        uint32_t pos = 0;
        uint32_t nix = 0;  // node index in the shard (32-bit index off the uniform base pointer)
        if (bt < b_hi && c < a.n_chunks) {
            nix = (uint32_t)c * (uint32_t)C;
            n_nodes = (int)min((int64_t)C, a.n_local - (int64_t)nix);
            pos = a.base_pos + nix;
        }
        CodeT rec = CodeWord<NF>::zero(), nxt;
        if (n_nodes > 0) rec = __ldg(codes + nix);
#pragma unroll 1
        for (int it = 0; it < C; ++it) {
            ++nix;
            if ((it & (PF - 1)) == 0) {  // warp-uniform: one L2 prefetch per 128-byte line of codes, three lines ahead
                if (it + 3 * PF + 1 < n_nodes) prefetch_l2(codes + nix + 3 * PF);
            }
            nxt = CodeWord<NF>::zero();
            if (it + 1 < n_nodes) nxt = __ldg(codes + nix);
            // d = sum of the node's NF table rows (pad bytes read all-zero rows)
            uint32_t d[4];
            if constexpr (NF == 8) {
                // eight 128-bit table reads in flight: this lane's 8 queries of each row
                const uint4 A0 = lds128o<0 * SUB>(rowaddr<ROWB>(lut_base, rec.x, 0));
                const uint4 A1 = lds128o<1 * SUB>(rowaddr<ROWB>(lut_base, rec.x, 1));
                const uint4 A2 = lds128o<2 * SUB>(rowaddr<ROWB>(lut_base, rec.x, 2));
                const uint4 A3 = lds128o<3 * SUB>(rowaddr<ROWB>(lut_base, rec.x, 3));
                const uint4 A4 = lds128o<4 * SUB>(rowaddr<ROWB>(lut_base, rec.y, 0));
                const uint4 A5 = lds128o<5 * SUB>(rowaddr<ROWB>(lut_base, rec.y, 1));
                const uint4 A6 = lds128o<6 * SUB>(rowaddr<ROWB>(lut_base, rec.y, 2));
                const uint4 A7 = lds128o<7 * SUB>(rowaddr<ROWB>(lut_base, rec.y, 3));
                d[0] = (A0.x + A1.x + A2.x) + (A3.x + A4.x + A5.x) + (A6.x + A7.x);
                d[1] = (A0.y + A1.y + A2.y) + (A3.y + A4.y + A5.y) + (A6.y + A7.y);
                d[2] = (A0.z + A1.z + A2.z) + (A3.z + A4.z + A5.z) + (A6.z + A7.z);
                d[3] = (A0.w + A1.w + A2.w) + (A3.w + A4.w + A5.w) + (A6.w + A7.w);
            } else {
                const uint32_t w4[4] = {rec.x, rec.y, rec.z, rec.w};
                d[0] = d[1] = d[2] = d[3] = 0u;
#pragma unroll
                for (int h = 0; h < 2; ++h) {  // two halves of eight reads keep the register footprint of the narrow shape
                    const uint32_t wa = w4[2 * h], wb = w4[2 * h + 1];
                    const uint4 A0 = lds128v(rowaddr<ROWB>(lut_base, wa, 0), (8 * h + 0) * SUB);
                    const uint4 A1 = lds128v(rowaddr<ROWB>(lut_base, wa, 1), (8 * h + 1) * SUB);
                    const uint4 A2 = lds128v(rowaddr<ROWB>(lut_base, wa, 2), (8 * h + 2) * SUB);
                    const uint4 A3 = lds128v(rowaddr<ROWB>(lut_base, wa, 3), (8 * h + 3) * SUB);
                    const uint4 A4 = lds128v(rowaddr<ROWB>(lut_base, wb, 0), (8 * h + 4) * SUB);
                    const uint4 A5 = lds128v(rowaddr<ROWB>(lut_base, wb, 1), (8 * h + 5) * SUB);
                    const uint4 A6 = lds128v(rowaddr<ROWB>(lut_base, wb, 2), (8 * h + 6) * SUB);
                    const uint4 A7 = lds128v(rowaddr<ROWB>(lut_base, wb, 3), (8 * h + 7) * SUB);
                    d[0] += (A0.x + A1.x + A2.x) + (A3.x + A4.x + A5.x) + (A6.x + A7.x);
                    d[1] += (A0.y + A1.y + A2.y) + (A3.y + A4.y + A5.y) + (A6.y + A7.y);
                    d[2] += (A0.z + A1.z + A2.z) + (A3.z + A4.z + A5.z) + (A6.z + A7.z);
                    d[3] += (A0.w + A1.w + A2.w) + (A3.w + A4.w + A5.w) + (A6.w + A7.w);
                }
            }
            // candidate test: bit 15 / 31 of (thr - d) survives iff d < bound, per packed half
            const uint32_t am = it < n_nodes ? 0x80008000u : 0u;
            const uint32_t h0 = thr[0] - d[0], h1 = thr[1] - d[1], h2 = thr[2] - d[2], h3 = thr[3] - d[3];
            const uint32_t hit = (h0 | h1 | h2 | h3) & am;
            if (__any_sync(0xffffffffu, hit != 0u)) {
                // rare path: one bit per (word, half) that is below its bound
                uint32_t bits = 0;
                bits |= ((h0 & am) >> 15 & 1u) | ((h0 & am) >> 30 & 2u);
                bits |= (((h1 & am) >> 15 & 1u) | ((h1 & am) >> 30 & 2u)) << 2;
                bits |= (((h2 & am) >> 15 & 1u) | ((h2 & am) >> 30 & 2u)) << 4;
                bits |= (((h3 & am) >> 15 & 1u) | ((h3 & am) >> 30 & 2u)) << 6;
                if constexpr (DEAD)
                    if (bits != 0u && node_dead(a.dead, pos - a.base_pos)) bits = 0u;
                while (bits) {
                    const int b = __ffs(bits) - 1;
                    bits &= bits - 1;
                    const uint32_t dw = b < 4 ? (b < 2 ? d[0] : d[1]) : (b < 6 ? d[2] : d[3]);
                    const uint32_t dist = (dw >> (16 * (b & 1))) & 0xFFFFu;
                    const int ql = jj * 8 + b;
                    const uint32_t slot = atomicAdd(&s_cnt[ql], 1u);
                    if (slot < (uint32_t)a.bcap)
                        __stcg(my_cand + (size_t)ql * a.bcap + slot, ((uint64_t)dist << 32) | pos);
                    else
                        a.ovf[(size_t)grp * QB + ql] = 1u;  // exact fallback will redo this query
                }
            }
            rec = nxt;
            ++pos;
            if (++since == epoch_len) {  // epoch boundary (uniform over the CTA)
                since = 0;
                if (epoch_len < a.epoch) epoch_len <<= 1;
                bool need = false;
                {  // warp w owns queries w, w + n_warps, ...
                    const int ql = warp + a.n_warps * lane;
                    if (ql < QB && (int)s_cnt[ql] >= trigger) need = true;
                }
                const int any_need = __syncthreads_or(need);
                if (warp == 0) {  // bounds published by the other slices of this query group
                    for (int ql = lane; ql < QB; ql += 32)
                        if (grp * QB + ql < a.Q) atomicMin(&s_thr[ql], __ldcg(&gthr[ql]));
                }
                if (any_need) {
                    for (int ql = warp; ql < QB; ql += a.n_warps) own_compact(&own, ql, trigger);
                    __syncthreads();
                }
                reload_thr();
            }
        }
    }
    // final compaction: every buffer becomes a sorted list of at most kp keys
    __syncthreads();
    for (int ql = warp; ql < QB; ql += a.n_warps) {
        own_compact(&own, ql, 1);
        if (lane == 0) a.cand_cnt[(size_t)item * QB + ql] = min(s_cnt[ql], (uint32_t)a.kp);
    }
}

cudaError_t launch_scan2(const Scan2Args& a, cudaStream_t st) {
    const size_t smem = (size_t)a.shape.lut_bytes() + MAXQB * 4 * 2 + 16;
    // 16 warps x 128 registers: more warps spill and ran 2x slower (gpurun_out/probe12.log)
    const dim3 grid((unsigned)(a.n_groups * a.n_slices)), block((unsigned)(a.n_warps * 32));
    cudaError_t e;
    if (a.dead) {
        void (*k)(const Scan2Args) = a.shape.nf == 8 ? scan2_kernel<8, 7, 8, true> : scan2_kernel<16, 3, 4, true>;
        e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        k<<<grid, block, smem, st>>>(a);
    } else {
        void (*k)(const Scan2Core) = a.shape.nf == 8 ? scan2_kernel<8, 7, 8, false> : scan2_kernel<16, 3, 4, false>;
        e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        k<<<grid, block, smem, st>>>(a);
    }
    return cudaGetLastError();
}

}  // namespace dpq
