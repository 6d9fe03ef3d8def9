// Coarse search: the whole tree is scanned with a small-integer table in packed 8-bit arithmetic.
// Narrow shape (M <= 8): 5-bit entries stored one per byte, four queries per 32-bit word, sixteen
// per 128-bit table read, 112 queries per CTA, i.e. HALF the shared-memory wavefronts per (node,
// query) of the 15-bit scan (scan2.cu), which is bound by exactly those wavefronts
// (profiles/r1_summary.md).  Wide shape (M <= 16): 4-bit entries (sixteen of them fit a byte sum)
// stored TWO per byte: a table row is 56 bytes = 112 queries, the 4096-row table fills shared memory
// exactly like the narrow one, a lane reads 16 queries per 64-bit load and splits even / odd nibbles
// into byte sums (three logic ops per word).  Round 1 kept one entry per byte (48-byte rows, 48
// queries per CTA): two 48-byte rows of one quarter-warp phase overlap in banks 75 % of the time;
// the nibble table needs half the wavefronts per (node, query).
//
// Why it is exact.  Before this pass the 15-bit scan runs over a 1/S sample of the tree and
// select_kernel gives cap_q = the exact k-th distance over the sample (real nodes), an upper bound
// of the true k-th distance T_q.  Coarse entry = min(SAT, rint(lut / unit)) with unit = cap_q / L
// (L = 80 levels; entries saturate at SAT = 31 / 15 so that the M of them never carry out of a
// byte).  Saturation only lowers a sum, and rounding adds at most 0.5 per entry, so a node with
// distance d <= T_q <= cap_q has coarse sum <= d / unit + M/2 <= L + M/2: EVERY true top-k node
// passes the test "sum < L + M/2 + 1".  (rint() is taken of the double product lut * (L / cap);
// both roundings are below 2^-52 relative, far inside the half-unit the integer test leaves: the sum
// of M roundings is at most M/2 and the bound is the next integer.)  The survivors (a few hundred
// per query) are re-scored exactly (float tables, double sum, reference arithmetic) by
// rescore8_kernel, which keeps the k best by (distance, position).  A candidate buffer that
// overflows flags its query for the exact fallback.  No result ever depends on the coarse values.
//
// The kernels are scan2's strand design (one code word per node, four nodes per warp step) with the
// candidate machinery reduced to a staged append: the bound is the same constant for every query, so
// there are no epochs, barriers or compactions.
#include "kernels.cuh"

#include <algorithm>
#include <cfloat>

namespace dpq {

__global__ void cap_from_keys_kernel(const uint64_t* __restrict__ keys, int topk, int Q, float* __restrict__ cap) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < Q) cap[q] = __uint_as_float((uint32_t)(keys[(size_t)q * topk + topk - 1] >> 32));
}
void launch_cap_from_keys(const uint64_t* d_keys, int topk, int Q, float* d_cap, cudaStream_t st) {
    cap_from_keys_kernel<<<(Q + 255) / 256, 256, 0, st>>>(d_keys, topk, Q, d_cap);
}

// The presample's node set (R evenly strided nodes of the shard) is the same for every query: their codes
// are gathered once per index into a compact array, so that a query's block reads them with coalesced
// loads instead of R strided ones (189 us -> see profiles/r2_summary.md at C2).
__global__ void gather_sample_kernel(const uint8_t* __restrict__ codes, int cstride, int64_t n_local, int R, int64_t stride,
                                     uint8_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    const int64_t node = (int64_t)i * stride;
    for (int b = 0; b < cstride; ++b) out[(size_t)i * cstride + b] = node < n_local ? codes[(size_t)node * cstride + b] : 0;
}
void launch_gather_sample(const uint8_t* d_codes, int cstride, int64_t n_local, int R, uint8_t* d_out, cudaStream_t st) {
    const int64_t stride = n_local / R > 0 ? n_local / R : 1;
    gather_sample_kernel<<<(R + 255) / 256, 256, 0, st>>>(d_codes, cstride, n_local, R, stride, d_out);
}

// One block per query: an upper bound of the distance of each of R evenly strided nodes (the query's float
// table in shared memory; the nodes' codes come from the compact array of launch_gather_sample), then an
// upper bound of the k-th smallest by bisection on the leading 14 bits of the float patterns (distances are
// non-negative, so the integer order of the bits is the float order; the answer is the top of the bucket:
// at most 1.6 % above the k-th value).  cap only has to be a VALID bound of the query's true k-th distance --
// it seeds the quantisation of the sample pass -- so neither the float sums nor the bucket cost exactness;
// the kernel is instruction-issue bound (ncu: 90 % issue active), and 31 bisection rounds of shuffles and
// barriers were most of its instructions.
// DEAD: a sample node whose bit is set in `dead` counts as +inf (the cap must be the k-th distance of live nodes).
template <int PS_T, bool DEAD>
__global__ void __launch_bounds__(PS_T) presample_kernel(const float* __restrict__ lutf, const uint8_t* __restrict__ sample_codes, int cstride,
                                                         int64_t n_local, int M, int K, int topk, int R,
                                                         float* __restrict__ cap, const uint32_t* __restrict__ dead) {
    extern __shared__ __align__(16) float s_lut[];  // M*K
    __shared__ int s_cnt[2][PS_T / 32];
    const int q = blockIdx.x;
    const int MK = M * K;
    stage_table(s_lut, lutf + (size_t)q * MK, MK, threadIdx.x, PS_T);
    __syncthreads();
    constexpr int PER = 16;  // R <= PS_T * PER
    constexpr int DROP = 17;  // pattern bits below the bucket
    uint32_t v[PER];
    const int64_t stride = n_local / R > 0 ? n_local / R : 1;
#pragma unroll
    for (int t = 0; t < PER; ++t) {
        const int i = t * PS_T + threadIdx.x;
        v[t] = 0x7F800000u >> DROP;  // +inf: never counted
        if (i < R && (int64_t)i * stride < n_local && !(DEAD && node_dead(dead, (uint32_t)((int64_t)i * stride))))
            v[t] = __float_as_uint(dist_upper_bound(s_lut, sample_codes + (size_t)i * cstride, cstride, M, K)) >> DROP;
    }
    // smallest bucket x with count(v <= x) >= topk
    uint32_t lo = 0, hi = 0x7F7FFFFFu >> DROP;  // FLT_MAX's bucket
    int it = 0;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        int c = 0;
#pragma unroll
        for (int t = 0; t < PER; ++t) c += v[t] <= mid;
        c = __reduce_add_sync(0xffffffffu, c);
        if ((threadIdx.x & 31) == 0) s_cnt[it & 1][threadIdx.x >> 5] = c;
        __syncthreads();  // one barrier per round: the next round writes the other buffer
        int tot = 0;
#pragma unroll
        for (int w = 0; w < PS_T / 32; ++w) tot += s_cnt[it & 1][w];
        if (tot >= topk) hi = mid;
        else lo = mid + 1;
        ++it;
    }
    // top of the bucket; FLT_MAX when the sample holds fewer than k nodes
    if (threadIdx.x == 0) cap[q] = __uint_as_float((lo << DROP) | ((1u << DROP) - 1u));
}
void launch_presample(const float* d_lutf, const uint8_t* d_sample_codes, int cstride, int64_t n_local, int M, int K, int Q,
                      int topk, int R, float* d_cap, const uint32_t* d_dead, cudaStream_t st) {
    // 16 values per thread: 128 threads for R <= 2048, 512 threads up to 8192
    const size_t sm = (size_t)M * K * sizeof(float);
    const bool small = R <= 128 * 16;
    auto k = small ? (d_dead ? presample_kernel<128, true> : presample_kernel<128, false>)
                   : (d_dead ? presample_kernel<512, true> : presample_kernel<512, false>);
    k<<<Q, small ? 128 : 512, sm, st>>>(d_lutf, d_sample_codes, cstride, n_local, M, K, topk, R, d_cap, d_dead);
}

// Coarse tables [group][m * 256 + centroid][112 queries]: NIB = false: one byte per entry (112-byte
// rows); NIB = true: two 4-bit entries per byte (56-byte rows, query ql in byte ql / 2, nibble ql & 1).
template <int ROWS, int SAT, bool NIB>
__global__ void __launch_bounds__(256) pack8_kernel(const float* __restrict__ lutf, const float* __restrict__ capv,
                                                    int M, int K, int Q, int levels, uint8_t* __restrict__ qlut8,
                                                    uint32_t* __restrict__ ovf) {
    constexpr int QB = 112;
    constexpr int ROWB = NIB ? 56 : 112;
    __shared__ __align__(16) uint8_t tile[64 * 112];
    __shared__ double s_inv[QB];
    const int grp = blockIdx.x, row0 = blockIdx.y * 64;
    const int MK = M * K;
    if (threadIdx.x < QB) {
        const int q = grp * QB + threadIdx.x;
        double inv = 0.0;
        if (q < Q) {
            const float cap = capv[q];
            // cap == FLT_MAX: the sample held fewer than k nodes; every entry quantises to 0 and
            // every node becomes a candidate (correct, merely slow: tiny trees only)
            inv = cap > 0.0f ? (double)levels / (double)cap : 0.0;
            if (cap == 0.0f) inv = 1e30;  // k exact matches: only zero entries stay below the bound
        }
        s_inv[threadIdx.x] = inv;
        if (blockIdx.y == 0) ovf[grp * QB + threadIdx.x] = 0u;
    }
    __syncthreads();
    // 28 entries per thread, seven loads in flight at a time (one load per round trip made the kernel
    // latency-bound: 53 us for 82 MB of L2-resident tables)
    constexpr int PER = 64 * QB / 256, BATCH = 7;
    static_assert(PER % BATCH == 0, "tile shape");
#pragma unroll 1
    for (int it0 = 0; it0 < PER; it0 += BATCH) {
        float f[BATCH];  // negative = no such entry (table entries are sums of squares)
#pragma unroll
        for (int u = 0; u < BATCH; ++u) {
            const int i = (it0 + u) * 256 + threadIdx.x;
            const int ql = i >> 6, r = i & 63;
            const int q = grp * QB + ql, row = row0 + r;
            const int m = row >> 8, c = row & 255;
            f[u] = (q < Q && m < M && c < K) ? __ldg(lutf + (size_t)q * MK + m * K + c) : -1.0f;
        }
#pragma unroll
        for (int u = 0; u < BATCH; ++u) {
            const int i = (it0 + u) * 256 + threadIdx.x;
            const int ql = i >> 6, r = i & 63;
            uint8_t v = 0;
            if (f[u] >= 0.0f) {
                const double x = (double)f[u] * s_inv[ql];
                v = x >= (double)SAT ? (uint8_t)SAT : (uint8_t)__double2int_rn(x);
            }
            tile[r * QB + ql] = v;
        }
    }
    __syncthreads();
    uint32_t* dst = reinterpret_cast<uint32_t*>(qlut8 + ((size_t)grp * ROWS + row0) * ROWB);
    if (!NIB) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(tile);
        for (int i = threadIdx.x; i < 64 * QB / 4; i += blockDim.x) dst[i] = src[i];
    } else {
        // eight consecutive queries (one 64-bit tile word) -> one 32-bit word of nibbles
        const uint2* src = reinterpret_cast<const uint2*>(tile);
        for (int i = threadIdx.x; i < 64 * QB / 8; i += blockDim.x) {
            const uint2 w = src[i];
            const uint32_t lo = (w.x & 0x0Fu) | ((w.x >> 4) & 0xF0u) | ((w.x >> 8) & 0xF00u) | ((w.x >> 12) & 0xF000u);
            const uint32_t hi = (w.y & 0x0Fu) | ((w.y >> 4) & 0xF0u) | ((w.y >> 8) & 0xF00u) | ((w.y >> 12) & 0xF000u);
            dst[i] = lo | (hi << 16);
        }
    }
}

void launch_pack8(const float* d_lutf, const float* d_cap, int M, int K, int Q, int levels, uint8_t* d_qlut8,
                  uint32_t* d_ovf, int n_groups, int nf, cudaStream_t st) {
    if (nf == 8)
        pack8_kernel<2048, 31, false><<<dim3((unsigned)n_groups, 2048 / 64), 256, 0, st>>>(d_lutf, d_cap, M, K, Q, levels, d_qlut8, d_ovf);
    else
        pack8_kernel<4096, 15, true><<<dim3((unsigned)n_groups, 4096 / 64), 256, 0, st>>>(d_lutf, d_cap, M, K, Q, levels, d_qlut8, d_ovf);
}

// Both shapes: 112 queries per CTA, a strand is a quarter warp (8 lanes, 7 active), lane jj of a
// strand owns queries jj*16 .. jj*16+15 in four 32-bit words of byte sums.
//   NF = 8 : LDS.128 of the 112-byte row, word k byte b = query jj*16 + 4k + b
//   NF = 16: LDS.64 of the 56-byte row (nibbles); sums E0, O0, E1, O1 = even / odd nibbles of the two
//            loaded words: word w (k = w >> 1, parity p = w & 1) byte b = query jj*16 + 8k + 2b + p
//
// Survivors are staged, not appended in the node loop.  A lane whose node passes for any of its 16
// queries writes one 8-byte record {position, jj << 4 | hit bits} to its warp's staging buffer in
// global memory; the slot is a warp-uniform counter plus the lane's rank in the step's ballot, so a
// step with hits has no atomics, no divergent loops and nothing that waits on a returned value.  The per-hit
// atomicAdd + store it replaces held most of the kernel's instructions and stall samples on the
// steps that took it (DESIGN.md section 8).  The warp expands its records into the per-(item, query)
// lists (drain8) whenever the next step could overflow its buffer and once at the end: the lists,
// their counts (clipped at bcap) and the overflow flags are exactly those of an in-loop append, in
// another order within a list, which nothing downstream depends on.  The staging capacity changes
// only how often a warp drains.  A buffer belongs to (SM, warp): one CTA per SM (checked at launch).
// DEAD: a.dead is the deleted-node bitmap; a lane whose node is deleted stages nothing.  The test
// sits inside the rare branch (one bitmap word per lane with a hit), before the ballot: testing in the
// drain instead stages every deleted node that passes, and with most of the tree deleted the loose
// cap of the live nodes passes many (25 % slower at 99 % deleted).  DEAD = false is the kernel without it.
template <int NF>
__device__ __forceinline__ void drain8(const uint2* __restrict__ rec, int n, uint32_t* s_cnt, uint32_t* __restrict__ my_cand,
                                    const Scan8Args& a, int grp, int lane) {
    constexpr int QB = 112;
    __syncwarp();  // the warp's records are visible to all of its lanes
    for (int i0 = 0; i0 < n; i0 += 32) {  // warp-uniform loops: the node loop stays convergent
        uint32_t m = 0u, pos = 0u;
        int jj = 0;
        if (i0 + lane < n) {
            const uint2 r = __ldcg(rec + i0 + lane);
            m = r.y & 0x0F0F0F0Fu;  // bit 8 b + k: byte b of word k
            jj = (int)(r.y >> 4) & 7;
            pos = r.x;
        }
        while (__any_sync(0xffffffffu, m != 0u)) {
            if (m) {
                const int bit = __ffs(m) - 1;
                m &= m - 1;
                const int b = bit >> 3, k = bit & 3;
                const int q = NF == 8 ? 4 * k + b : 8 * (k >> 1) + 2 * b + (k & 1);
                const int ql = jj * 16 + q;
                const uint32_t slot = atomicAdd(&s_cnt[ql], 1u);
                if (slot < (uint32_t)a.bcap) __stcg(my_cand + (size_t)ql * a.bcap + slot, pos);
                else a.ovf[(size_t)grp * QB + ql] = 1u;
            }
        }
    }
    __syncwarp();  // every record is read before the buffer is refilled
}

template <int NF, bool REUSE, bool DEAD>
__global__ void __launch_bounds__(768, 1) scan8_kernel(const Scan8Args a) {
    constexpr int QB = 112;                      // queries per CTA
    constexpr int ROWS = NF * 256;
    constexpr int ROWB = NF == 8 ? 112 : 56;     // table row bytes
    constexpr int LANEB = NF == 8 ? 16 : 8;      // bytes of a row one lane reads
    constexpr int LUT_BYTES = ROWS * ROWB;
    constexpr int SPW = 4;                       // strands per warp = chunks in flight per warp
    constexpr int SUB = 256 * ROWB;              // table bytes per subspace
    using CodeT = typename CodeWord<NF>::type;
    extern __shared__ __align__(128) unsigned char smem[];
    uint32_t* s_cnt = reinterpret_cast<uint32_t*>(smem + LUT_BYTES);  // [128] candidates per query
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(s_cnt + 128);

    const int item = blockIdx.x;
    const int slice = item / a.n_groups, grp = item % a.n_groups;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int strand = lane >> 3, j = lane & 7;
    const int jj = j < 7 ? j : 6;
    const int n_bt = ((a.n_chunks + SPW - 1) / SPW + a.bt_stride - 1) / a.bt_stride;  // batches this launch walks
    const int b_lo = (int)((int64_t)n_bt * slice / a.n_slices);
    const int b_hi = (int)((int64_t)n_bt * (slice + 1) / a.n_slices);

    if (threadIdx.x == 0) {
        mbar_init(s_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // TMA bulk copy of the group's coarse table
        mbar_expect_tx(s_bar, (uint32_t)LUT_BYTES);
        const unsigned char* src = a.qlut8 + (size_t)grp * LUT_BYTES;
        for (uint32_t o = 0; o < (uint32_t)LUT_BYTES; o += 32768u) bulk_g2s(smem + o, src + o, 32768u, s_bar);
    }
    if (threadIdx.x < 128) s_cnt[threadIdx.x] = 0u;
    __syncthreads();
    mbar_wait(s_bar, 0);

    // Per byte: hit iff sum < thresh (<= 128), tested as bit 7 of (0x80 + thresh - 1 - low7(sum))
    // with bit 7 of the sum clear; a dead byte (idle lane / query beyond Q) gets the constant 0x7F,
    // which never sets bit 7.
    uint32_t lut_base = smem_u32(smem) + (uint32_t)jj * (uint32_t)LANEB;
    asm volatile("" : "+r"(lut_base));
    const int n_live = j < 7 ? min(16, max(0, a.Q - (grp * QB + jj * 16))) : 0;
    uint32_t cmpc[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        cmpc[k] = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int r = NF == 8 ? 4 * k + b : 8 * (k >> 1) + 2 * b + (k & 1);  // query of (word k, byte b) within the lane
            cmpc[k] |= (r < n_live ? (0x80u + (uint32_t)a.thresh - 1u) : 0x7Fu) << (8 * b);
        }
    }
    uint32_t* my_cand = a.cand + (size_t)item * QB * a.bcap;
    const int n_rounds = (b_hi - b_lo + a.n_warps - 1) / a.n_warps;
    const int C = a.chunk_nodes;
    const CodeT* codes = reinterpret_cast<const CodeT*>(a.codes);
    constexpr int PF = 128 / (int)sizeof(CodeT);  // nodes per 128-byte line

    // Row reuse (REUSE, narrow shape): a strand walks consecutive DFS positions, and a node often shares
    // a centroid with the node before it in some subspaces (21 % of the rows of the 1M SIFT-shaped tree,
    // tools/row_reuse_stats.py).  The eight rows stay in registers across nodes and a row is read only
    // when its code byte changed: one LOP3 with a predicate output per row, and a skipped read sends no
    // shared-memory wavefront for that strand.  The rows, and so the sums, are the same as when every
    // row is read.  REUSE = false reads all of them every node.  The wide scan does not reuse rows: it
    // is issue-bound, and the sixteen predicates made it slower (profiles/r3_summary.md).
    static_assert(NF == 8 || !REUSE, "row reuse is narrow-shape only");
    uint4 A[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) A[r] = make_uint4(0u, 0u, 0u, 0u);

    // this warp's staging buffer: [SM][24 warps][stage_cap] records
    uint32_t smid;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));
    uint2* stage = a.stage + ((size_t)smid * 24 + (size_t)warp) * (size_t)a.stage_cap;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const uint32_t jj_tag = (uint32_t)jj << 4;
    int n_staged = 0;  // warp-uniform

    // One node of a strand: its M rows (NF = 8: those whose code byte changed, REUSE), the byte sums, the
    // SWAR hit test, and on a hit one staged record.  ok: the node exists.
    auto node = [&](const CodeT w, const uint2 chg, const bool ok, const uint32_t p) {
        uint32_t d[4];
        if constexpr (NF == 8) {
            const uint32_t w2[2] = {w.x, w.y};
            const uint32_t ch2[2] = {REUSE ? chg.x : ~0u, REUSE ? chg.y : ~0u};
#pragma unroll
            for (int r = 0; r < 8; ++r)
                lds128_if(A[r], rowaddr<ROWB>(lut_base, w2[r >> 2], r & 3) + (uint32_t)(r * SUB), ch2[r >> 2] & (0xFFu << (8 * (r & 3))));
            d[0] = (A[0].x + A[1].x + A[2].x) + (A[3].x + A[4].x + A[5].x) + (A[6].x + A[7].x);
            d[1] = (A[0].y + A[1].y + A[2].y) + (A[3].y + A[4].y + A[5].y) + (A[6].y + A[7].y);
            d[2] = (A[0].z + A[1].z + A[2].z) + (A[3].z + A[4].z + A[5].z) + (A[6].z + A[7].z);
            d[3] = (A[0].w + A[1].w + A[2].w) + (A[3].w + A[4].w + A[5].w) + (A[6].w + A[7].w);
        } else {
            const uint32_t w4[4] = {w.x, w.y, w.z, w.w};
            d[0] = d[1] = d[2] = d[3] = 0u;
#pragma unroll
            for (int h = 0; h < 4; ++h) {  // four rows at a time: four 64-bit reads in flight per step
                const uint2 A0 = lds64(rowaddr<ROWB>(lut_base, w4[h], 0) + (uint32_t)((4 * h + 0) * SUB));
                const uint2 A1 = lds64(rowaddr<ROWB>(lut_base, w4[h], 1) + (uint32_t)((4 * h + 1) * SUB));
                const uint2 A2 = lds64(rowaddr<ROWB>(lut_base, w4[h], 2) + (uint32_t)((4 * h + 2) * SUB));
                const uint2 A3 = lds64(rowaddr<ROWB>(lut_base, w4[h], 3) + (uint32_t)((4 * h + 3) * SUB));
                constexpr uint32_t LO = 0x0F0F0F0Fu;
                d[0] += ((A0.x & LO) + (A1.x & LO)) + ((A2.x & LO) + (A3.x & LO));
                d[1] += (((A0.x >> 4) & LO) + ((A1.x >> 4) & LO)) + (((A2.x >> 4) & LO) + ((A3.x >> 4) & LO));
                d[2] += ((A0.y & LO) + (A1.y & LO)) + ((A2.y & LO) + (A3.y & LO));
                d[3] += (((A0.y >> 4) & LO) + ((A1.y >> 4) & LO)) + (((A2.y >> 4) & LO) + ((A3.y >> 4) & LO));
            }
        }
        const uint32_t am = ok ? 0x80808080u : 0u;
        const uint32_t h0 = (cmpc[0] - (d[0] & 0x7F7F7F7Fu)) & ~d[0];
        const uint32_t h1 = (cmpc[1] - (d[1] & 0x7F7F7F7Fu)) & ~d[1];
        const uint32_t h2 = (cmpc[2] - (d[2] & 0x7F7F7F7Fu)) & ~d[2];
        const uint32_t h3 = (cmpc[3] - (d[3] & 0x7F7F7F7Fu)) & ~d[3];
        uint32_t hit = (h0 | h1 | h2 | h3) & am;
        if (__any_sync(0xffffffffu, hit != 0u)) {  // the ballot and the fold stay off the common path
            // a deleted node stages nothing: under a heavily deleted tree most nodes that pass are deleted
            if constexpr (DEAD)
                if (hit != 0u && node_dead(a.dead, p - a.base_pos)) hit = 0u;
            const uint32_t bal = __ballot_sync(0xffffffffu, hit != 0u);
            // bit 8 b + k of the fold: byte b of word k is below the bound
            const uint32_t hb = (((h0 & am) >> 7) | ((h1 & am) >> 6)) | (((h2 & am) >> 5) | ((h3 & am) >> 4));
            if (hit) __stcg(stage + n_staged + __popc(bal & lt_mask), make_uint2(p, hb | jj_tag));
            n_staged += __popc(bal);
            if (n_staged > a.stage_cap - 32) {  // a step stages at most 28 records
                drain8<NF>(stage, n_staged, s_cnt, my_cand, a, grp, lane);
                n_staged = 0;
            }
        }
    };

    for (int round = 0; round < n_rounds; ++round) {
        const int bt = b_lo + round * a.n_warps + warp;
        const int c = bt * a.bt_stride * SPW + strand;
        int n_nodes = 0;
        uint32_t pos = 0, nix = 0;
        if (bt < b_hi && c < a.n_chunks) {
            nix = (uint32_t)c * (uint32_t)C;
            n_nodes = (int)min((int64_t)C, a.n_local - (int64_t)nix);
            pos = a.base_pos + nix;
        }
        // code bytes that differ from the strand's previous node: at a chunk start all of them, on an
        // idle strand none (past a chunk's last node the code is 0: one read of the changed rows, then none)
        uint2 chg = n_nodes > 0 ? make_uint2(~0u, ~0u) : make_uint2(0u, 0u);
        if constexpr (NF == 8) {
            // Two nodes' code words per 128-bit load (C is even, so a pair never straddles 16 bytes): half
            // the load wavefronts of one LDG.64 per node, double-buffered one pair ahead.
            const uint4* pairs = reinterpret_cast<const uint4*>(codes);
            auto load_pair = [&](uint32_t at, int first) {  // nodes `first`, `first` + 1 of the chunk
                uint4 v = make_uint4(0u, 0u, 0u, 0u);
                if (first + 1 < n_nodes) v = __ldg(pairs + (at >> 1));
                else if (first < n_nodes) { const uint2 h = __ldg(codes + at); v.x = h.x; v.y = h.y; }
                return v;
            };
            uint4 cur = load_pair(nix, 0);
#pragma unroll 1
            for (int it = 0; it < C; it += 2) {
                nix += 2;
                if ((it & (PF - 1)) == 0) {  // warp-uniform: one L2 prefetch per 128-byte line of codes, three lines ahead
                    if (it + 3 * PF + 1 < n_nodes) prefetch_l2(codes + nix - 1 + 3 * PF);
                }
                const uint4 nxt = load_pair(nix, it + 2);
                node(make_uint2(cur.x, cur.y), chg, it < n_nodes, pos);
                node(make_uint2(cur.z, cur.w), make_uint2(cur.z ^ cur.x, cur.w ^ cur.y), it + 1 < n_nodes, pos + 1u);
                chg = make_uint2(nxt.x ^ cur.z, nxt.y ^ cur.w);
                cur = nxt;
                pos += 2u;
            }
        } else {
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
                node(rec, chg, it < n_nodes, pos);
                rec = nxt;
                ++pos;
            }
        }
    }
    if (n_staged) drain8<NF>(stage, n_staged, s_cnt, my_cand, a, grp, lane);
    __syncthreads();
    for (int ql = threadIdx.x; ql < QB; ql += blockDim.x)
        a.cand_cnt[(size_t)item * QB + ql] = min(s_cnt[ql], (uint32_t)a.bcap);
}

__global__ void nsmid_kernel(int* out) {
    uint32_t n;
    asm("mov.u32 %0, %%nsmid;" : "=r"(n));
    *out = (int)n;
}
cudaError_t scan8_sm_slots(int* d_tmp, int* n_slots, cudaStream_t st) {
    nsmid_kernel<<<1, 1, 0, st>>>(d_tmp);
    cudaError_t e = cudaMemcpyAsync(n_slots, d_tmp, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    return e;
}

cudaError_t launch_scan8(const Scan8Args& a, cudaStream_t st) {
    const C8Shape sh = c8_shape(a.nf);
    const size_t smem = (size_t)sh.lut_bytes() + 128 * 4 + 16;
    void (*k)(const Scan8Args) =
        a.dead ? (a.nf == 16 ? scan8_kernel<16, false, true> : a.reuse ? scan8_kernel<8, true, true> : scan8_kernel<8, false, true>)
               : (a.nf == 16 ? scan8_kernel<16, false, false> : a.reuse ? scan8_kernel<8, true, false> : scan8_kernel<8, false, false>);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // the staging buffers are indexed by SM: a second resident CTA would share them
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, a.n_warps * 32, smem);
    if (e != cudaSuccess) return e;
    if (per_sm > 1 || a.n_warps > 24 || a.stage_cap < 32 || !a.stage || (a.chunk_nodes & 1)) return cudaErrorInvalidConfiguration;
    k<<<(unsigned)(a.n_groups * a.n_slices), (unsigned)(a.n_warps * 32), smem, st>>>(a);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------ exact re-score --
// One CTA per query: the query's exact float table is staged in shared memory, every coarse
// survivor is scored exactly (float entries, double sum of the node's M entries = what the
// reference's double accumulation rounds to) and the k best keys (distance bits << 32 | position)
// are kept by the block-wide running top-k (fb_compact): the buffer is sorted and cut to k whenever
// it fills, and the k-th key becomes the acceptance bound.  The per-(slice, query) candidate lists
// are addressed as one flat index space so that every step scores blockDim.x candidates no matter
// how they are spread over the slices.
constexpr int R8_T = 256;
constexpr int R8_MAXSL = 128;  // slices per group the flattened candidate index can address

__global__ void __launch_bounds__(R8_T) rescore8_kernel(const Rescore8Args a) {
    extern __shared__ __align__(16) unsigned char r8_smem[];
    uint64_t* s_keys = reinterpret_cast<uint64_t*>(r8_smem);   // [FB_BUF]
    float* s_lut = reinterpret_cast<float*>(s_keys + FB_BUF);  // [M*K]
    __shared__ uint32_t s_off[R8_MAXSL + 1];  // exclusive prefix of the per-slice counts
    __shared__ uint32_t s_n;
    __shared__ unsigned long long s_thr;
    __shared__ int s_last;
    const int q = blockIdx.x;
    // a query's candidate lists are cut into n_parts ranges of slices, one CTA each: candidate counts
    // are heavy tailed (a query in a dense region passes 20x the average), and one CTA per query
    // made the kernel wait for its slowest block
    const int part = blockIdx.y, n_parts = gridDim.y;
    const int sl_lo = a.n_slices * part / n_parts, sl_hi = a.n_slices * (part + 1) / n_parts;
    const int n_sl = sl_hi - sl_lo;
    const int grp = q / a.qb, ql = q % a.qb;
    const int MK = a.M * a.K;
    stage_table(s_lut, a.lutf + (size_t)q * MK, MK, threadIdx.x, R8_T);
    if (threadIdx.x < 32) {  // warp 0: counts of this part's slices, exclusive prefix
        const int lane = threadIdx.x;
        uint32_t run = 0;
        for (int s0 = 0; s0 < n_sl; s0 += 32) {
            const int s = s0 + lane;
            uint32_t c = 0;
            if (s < n_sl) c = a.cand_cnt[((size_t)(sl_lo + s) * a.n_groups + grp) * a.qb + ql];
            uint32_t incl = c;
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (s < n_sl) s_off[s] = run + incl - c;
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) {
            s_off[n_sl] = run;
            s_n = 0u;
            // a valid cap known beforehand bounds the candidates worth keeping (inclusive, any position)
            const float cap = a.cap_in ? a.cap_in[q] : FLT_MAX;
            s_thr = ((unsigned long long)__float_as_uint(cap) << 32) | 0xFFFFFFFFull;
        }
    }
    __syncthreads();
    const int total = (int)s_off[n_sl];
    for (int base = 0; base < total; base += R8_T) {
        const int i = base + threadIdx.x;
        if (i < total) {
            int lo = 0, hi = n_sl;  // slice s with off[s] <= i < off[s+1]
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (s_off[mid] <= (uint32_t)i) lo = mid;
                else hi = mid;
            }
            const size_t item = (size_t)(sl_lo + lo) * a.n_groups + grp;
            const uint32_t pos = __ldcg(a.cand + (item * a.qb + ql) * (size_t)a.bcap + ((uint32_t)i - s_off[lo]));
            const uint8_t* code = a.codes + (size_t)((int64_t)pos - a.base_pos) * a.cstride;
            const double d = exact_dist(s_lut, code, a.cstride, a.M, a.K);
            const uint64_t key = ((uint64_t)__float_as_uint((float)d) << 32) | pos;
            if (key <= s_thr) s_keys[atomicAdd(&s_n, 1u)] = key;  // < FB_BUF: compacted well below FB_BUF - R8_T
        }
        __syncthreads();
        // compact early (a small sort) so that the k-th key becomes the bound soon: later candidates are
        // then rejected by one compare instead of being stored and sorted
        if (s_n > (uint32_t)max(256, 2 * a.topk)) fb_compact(s_keys, &s_n, &s_thr, a.topk);
    }
    fb_compact(s_keys, &s_n, &s_thr, a.topk);
    const int k = a.topk;
    if (n_parts > 1) {
        // leave this part's k best in the scratch list; the last CTA of the query to arrive merges them
        uint64_t* mine = a.part + ((size_t)q * n_parts + part) * k;
        for (int i = threadIdx.x; i < k; i += R8_T) mine[i] = i < (int)s_n ? s_keys[i] : ~0ull;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_last = atomicAdd(&a.part_done[q], 1u) == (uint32_t)(n_parts - 1);
        __syncthreads();
        if (!s_last) return;
        __threadfence();
        const uint64_t* all = a.part + (size_t)q * n_parts * k;
        for (int i = threadIdx.x; i < n_parts * k; i += R8_T) s_keys[i] = __ldcg(all + i);
        if (threadIdx.x == 0) {
            s_n = (uint32_t)(n_parts * k);  // empty slots are ~0 keys: they sort to the end
            s_thr = ~0ull;
            a.part_done[q] = 0u;  // ready for the next pass
        }
        __syncthreads();
        fb_compact(s_keys, &s_n, &s_thr, k);
    }
    int n = (int)s_n;
    if (n_parts > 1) {  // count the real keys among the k kept
        __shared__ int s_real;
        if (threadIdx.x == 0) s_real = 0;
        __syncthreads();
        int c = 0;
        for (int i = threadIdx.x; i < n; i += R8_T) c += s_keys[i] != ~0ull;
        if (c) atomicAdd(&s_real, c);
        __syncthreads();
        n = s_real;
    }
    if (a.out_key)
        for (int i = threadIdx.x; i < k; i += R8_T)
            a.out_key[(size_t)q * k + i] = i < n ? s_keys[i] : (((uint64_t)__float_as_uint(FLT_MAX) << 32) | 0xFFFFFFFFull);
    if (threadIdx.x == 0) {
        // the k best found are real nodes: their k-th distance bounds the true k-th from above even
        // when candidates were dropped
        const float found = n >= k ? __uint_as_float((uint32_t)(s_keys[k - 1] >> 32)) : FLT_MAX;
        const float known = a.cap_in ? a.cap_in[q] : FLT_MAX;
        if (a.cap_out) a.cap_out[q] = fminf(found, known);
        if (a.flagged) {
            // a dropped candidate (buffer overflow) may hide a true top-k node: exact fallback, bounded
            // by the best k found so far
            a.bound[q] = fminf(found, known);
            if (a.ovf[(size_t)grp * a.qb + ql]) {
                const uint32_t slot = atomicAdd(a.n_flagged, 1u);
                if (slot < (uint32_t)a.max_flagged) a.flagged[slot] = (uint32_t)q;
            }
        }
    }
}

// (Measured and rejected: two interleaved queries per warp, so that 10 000 queries fit one wave of resident
// warps -- 235 us against 168 us at C2: candidate counts are heavy tailed, the longest query decides.)
// Short lists (topk <= 32) with a few hundred survivors per query: ONE WARP per query, no barriers: the
// keys live in a small shared-memory buffer that is reduced by rank counting whenever it fills.  (The
// CTA-per-query form above pays a table load and ~50 barrier stages of sorting per query: 289 us against
// this form's time at C2, 10 000 queries x 900 survivors.)
constexpr int R8W_WARPS = 4;
constexpr int R8W_BUF = 96;  // >= topk + 64

__device__ __forceinline__ int r8w_compact(uint64_t* buf, int n, int k, int lane) {
    // keep the min(n, k) smallest of buf[0..n) sorted ascending (keys unique); n <= R8W_BUF
    uint64_t mine[R8W_BUF / 32];
    int rank[R8W_BUF / 32];
#pragma unroll
    for (int t = 0; t < R8W_BUF / 32; ++t) {
        mine[t] = ~0ull;
        rank[t] = 0;
        if (t * 32 + lane < n) mine[t] = buf[t * 32 + lane];
    }
    __syncwarp();
    for (int i = 0; i < n; ++i) {
        const uint64_t o = buf[i];  // broadcast read
#pragma unroll
        for (int t = 0; t < R8W_BUF / 32; ++t) rank[t] += o < mine[t];
    }
    __syncwarp();
    const int keep = n < k ? n : k;
#pragma unroll
    for (int t = 0; t < R8W_BUF / 32; ++t)
        if (t * 32 + lane < n && rank[t] < keep) buf[rank[t]] = mine[t];
    __syncwarp();
    return keep;
}

__global__ void __launch_bounds__(R8W_WARPS * 32) rescore8w_kernel(const Rescore8Args a) {
    __shared__ uint64_t s_buf[R8W_WARPS][R8W_BUF];
    __shared__ uint32_t s_off[R8W_WARPS][R8_MAXSL + 1];  // exclusive prefix of the per-slice counts
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int q = blockIdx.x * R8W_WARPS + w;
    if (q >= a.Q) return;
    const int grp = q / a.qb, ql = q % a.qb;
    const float* lut = a.lutf + (size_t)q * a.M * a.K;
    uint64_t* buf = s_buf[w];
    uint32_t* off = s_off[w];
    uint32_t run = 0;
    for (int s0 = 0; s0 < a.n_slices; s0 += 32) {
        const int s = s0 + lane;
        uint32_t c = 0;
        if (s < a.n_slices) c = a.cand_cnt[((size_t)s * a.n_groups + grp) * a.qb + ql];
        uint32_t incl = c;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (s < a.n_slices) off[s] = run + incl - c;
        run += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) off[a.n_slices] = run;
    __syncwarp();
    const int total = (int)run;
    const int k = a.topk;
    int n = 0;
    // inclusive bound: a valid cap known beforehand, then the k-th best key so far
    const float known = a.cap_in ? a.cap_in[q] : FLT_MAX;
    uint64_t bound = ((uint64_t)__float_as_uint(known) << 32) | 0xFFFFFFFFull;
    // Two candidates per lane per round, every load of both issued before either is used (indices are
    // clamped instead of branched around): a round is a chain of three dependent memory round trips
    // (position -> code -> table entries), and one candidate per lane left the warp waiting on each of them.
    constexpr int U = 2;
    for (int i0 = 0; i0 < total; i0 += 32 * U) {
        uint32_t pos[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int i = min(i0 + 32 * u + lane, total - 1);
            int lo = 0, hi = a.n_slices;  // slice s with off[s] <= i < off[s+1]
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (off[mid] <= (uint32_t)i) lo = mid;
                else hi = mid;
            }
            const size_t item = (size_t)lo * a.n_groups + grp;
            pos[u] = __ldcg(a.cand + (item * a.qb + ql) * (size_t)a.bcap + ((uint32_t)i - off[lo]));
        }
        uint64_t keys[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint8_t* code = a.codes + (size_t)((int64_t)pos[u] - a.base_pos) * a.cstride;
            keys[u] = ((uint64_t)__float_as_uint((float)exact_dist(lut, code, a.cstride, a.M, a.K)) << 32) | pos[u];
            if (i0 + 32 * u + lane >= total) keys[u] = ~0ull;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t key = keys[u];
            const bool take = key <= bound;
            const uint32_t mk = __ballot_sync(0xffffffffu, take);
            if (mk) {
                if (n + 32 > R8W_BUF) {  // make room: reduce to the k best, tighten the bound
                    n = r8w_compact(buf, n, k, lane);
                    if (n == k) bound = buf[k - 1] - 1ull;
                    __syncwarp();
                }
                const bool still = take && key <= bound;
                const uint32_t mk2 = __ballot_sync(0xffffffffu, still);
                if (still) buf[n + __popc(mk2 & ((1u << lane) - 1u))] = key;
                n += __popc(mk2);
                __syncwarp();
            }
        }
    }
    n = r8w_compact(buf, n, k, lane);
    if (a.out_key)
        for (int i = lane; i < k; i += 32)
            a.out_key[(size_t)q * k + i] = i < n ? buf[i] : (((uint64_t)__float_as_uint(FLT_MAX) << 32) | 0xFFFFFFFFull);
    const float found = n >= k ? __uint_as_float((uint32_t)(buf[k - 1] >> 32)) : FLT_MAX;
    if (lane == 0 && a.cap_out) a.cap_out[q] = fminf(found, known);
    if (lane == 0 && a.flagged) {
        a.bound[q] = fminf(found, known);
        if (a.ovf[(size_t)grp * a.qb + ql]) {
            const uint32_t slot = atomicAdd(a.n_flagged, 1u);
            if (slot < (uint32_t)a.max_flagged) a.flagged[slot] = (uint32_t)q;
        }
    }
}

void launch_rescore8(const Rescore8Args& a, cudaStream_t st) {
    if (a.n_parts <= 1 && a.topk <= 32 && a.warp_form) {
        rescore8w_kernel<<<(a.Q + R8W_WARPS - 1) / R8W_WARPS, R8W_WARPS * 32, 0, st>>>(a);
        return;
    }
    const size_t sm = (size_t)FB_BUF * sizeof(uint64_t) + (size_t)a.M * a.K * sizeof(float);
    rescore8_kernel<<<dim3((unsigned)a.Q, (unsigned)std::max(1, a.n_parts)), R8_T, sm, st>>>(a);
}

}  // namespace dpq
