// Latency-mode scan for a handful of queries (Q <= 16, M <= 8): LANES = NODES.
//
// The batched kernels (scan2.cu / scan8.cu) put lanes = queries: a table row read serves 56 / 112
// queries, and the pass is bound by the shared-memory data pipe at 8 wavefronts per node per query
// group -- whether the group holds 112 queries or one.  For one or two queries that is 20x the
// time HBM needs to stream the code array once (SURVEY App. F: "lanes = nodes with 1-2 queries per
// pass is the only physically HBM-bound regime").  Here every lane scores its own node:
//
//   * a warp reads 32 consecutive nodes' codes (8 B/node, 128-bit loads of two nodes per lane,
//     the next chunk's loads in flight while the current one is scored): the tree streams from HBM
//     exactly once per PAIR of queries, fully coalesced;
//   * the table is the pair's fixed-point ADC table, two 16-bit entries per 32-bit word (one per
//     query: entry = rint(lut * 65500 / sum of the per-subspace maxima), so the M entries of a node
//     sum below 2^16 and the packed add never carries between the halves), replicated 16 times in
//     shared memory (2048 entries x 16 copies x 4 B = 128 KB): lane l reads copy l % 16, so only
//     lanes l and l + 16 can collide (two wavefronts per lookup instead of ~3.5 for one copy);
//   * the address of subspace m's entry is ((code >> (8m - 6)) & 0x3FC0) | lane_base: one shift and
//     one LOP3 (the table sits on a 16 KB boundary), the subspace offset m * 16 KB is the load's
//     immediate: four instructions per lookup for two queries;
//   * top-k: the bound is a constant per query (cap * scale + rounding slack), a hit appends the
//     node's position to the query's candidate list; rescore1_kernel (kernels.cu) scores the
//     candidates exactly (float tables, double sum: the reference's arithmetic) and keeps the k best
//     by (distance, position).  The cap comes from an exact presample (2048 strided nodes) and, on
//     large trees, a first pass of this kernel over every S-th chunk.  A node with exact distance
//     d <= cap has fixed-point sum <= cap * scale + M/2 (rounding adds at most 0.5 per entry), so no
//     true top-k node is dropped; results never depend on the fixed point.
//
// Bound (DESIGN.md): 8 lookups x 2 wavefronts per 32 nodes = 0.5 wavefront per node per query pair
// against 8 B/node of HBM: the shared-memory pipe allows 2 nodes/clk/SM = 69 % of the HBM copy
// peak; the kernel is built to sit at that ceiling and its dram__bytes_read is the tree size.
#include "kernels.cuh"

#include <cfloat>

namespace dpq {

constexpr int S1_T = 1024;            // threads per CTA, one CTA per SM
constexpr int S1_CHUNK = 2 * S1_T;    // nodes per CTA iteration (two per thread: one 128-bit load)
constexpr int S1_TABLE = 2048 * 16 * 4;

// (x & 0x3FC0) | base in ONE LOP3 (the compiler turns the OR of disjoint bit fields into an add)
__device__ __forceinline__ uint32_t field_addr(uint32_t x, uint32_t base) {
    uint32_t d;
    asm("lop3.b32 %0, %1, 0x3FC0, %2, 0xEA;" : "=r"(d) : "r"(x), "r"(base));
    return d;
}

// DEAD: a.dead is the deleted-node bitmap; a deleted node is never appended.  DEAD = false has no test.
template <bool DEAD>
__global__ void __launch_bounds__(S1_T, 1) scan1_kernel(const Scan1Args a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    // table on a 16 KB boundary: address bits 6..13 are the centroid field of the lookup
    const uint32_t s_base = smem_u32(smem_raw);
    const uint32_t t_base = (s_base + 16383u) & ~16383u;
    unsigned char* table = smem_raw + (t_base - s_base);
    const int pair = blockIdx.x % a.n_pairs, range = blockIdx.x / a.n_pairs;
    const int q0 = 2 * pair, q1 = 2 * pair + 1;
    const bool live1 = q1 < a.Q;
    const int MK = a.M * a.K;
    // fixed-point scale of each query: 65500 / sum of the per-subspace maxima, so that a node's M entries
    // sum below 2^16 (+ M/2 of rounding).  A sum that is not finite and positive (a NaN or infinite query
    // component) scales by 0: every entry 0, the filter passes every node and the exact re-score decides.
    auto scale_of = [&](int q) -> double {
        double sum = 0.0;
        for (int m = 0; m < a.M; ++m) sum += (double)a.mmax[q * 16 + m];
        return sum > 0.0 ? 65500.0 / sum : 0.0;
    };
    // entries clamped to the lane's range before packing (NaN -> 0): no value reaches the partner's half
    auto entry = [&](int q, int i, double sc) -> uint32_t {
        return (uint32_t)__double2int_rn(fmin(fmax((double)a.lutf[(size_t)q * MK + i] * sc, 0.0), 65500.0));
    };
    const double sc0 = scale_of(q0);
    const double sc1 = live1 ? scale_of(q1) : 0.0;
    for (int e = threadIdx.x; e < 2048; e += S1_T) {
        const int m = e >> 8, c = e & 255;
        uint32_t w = 0;
        if (m < a.M && c < a.K) {
            const uint32_t v0 = entry(q0, m * a.K + c, sc0);
            const uint32_t v1 = live1 ? entry(q1, m * a.K + c, sc1) : 0u;
            w = v0 | (v1 << 16);
        }
        uint4* dst = reinterpret_cast<uint4*>(table + (size_t)e * 64);
        const uint4 w4 = make_uint4(w, w, w, w);
        dst[0] = w4;
        dst[1] = w4;
        dst[2] = w4;
        dst[3] = w4;
    }
    // inclusive fixed-point bounds: every node with exact distance <= cap passes
    auto bound_of = [&](int q, double sc) -> uint32_t {
        const float cap = a.cap[q];
        if (!(cap < FLT_MAX)) return 0xFFFFFu;  // no cap known: everything passes (tiny trees)
        const double b = floor((double)cap * sc) + 0.5 * a.M + 2.0;
        return b >= 1048575.0 ? 0xFFFFFu : (uint32_t)b;
    };
    const uint32_t thr0 = bound_of(q0, sc0);
    const uint32_t thr1 = live1 ? bound_of(q1, sc1) : 0u;
    __syncthreads();

    const uint32_t lane_base = t_base + (uint32_t)(threadIdx.x & 15) * 4u;
    // 32-bit indices: a shard holds fewer than 2^32 nodes (positions are 32-bit)
    const uint32_t n_local = (uint32_t)a.n_local;
    const uint32_t n_chunks = (n_local + S1_CHUNK - 1) / S1_CHUNK;
    const uint32_t n_walk = (n_chunks + (uint32_t)a.chunk_stride - 1) / (uint32_t)a.chunk_stride;  // chunks this launch walks
    const uint32_t w_lo = (uint32_t)((uint64_t)n_walk * range / a.n_ranges);
    const uint32_t w_hi = (uint32_t)((uint64_t)n_walk * (range + 1) / a.n_ranges);
    const uint4* codes = reinterpret_cast<const uint4*>(a.codes);  // two nodes per uint4
    const uint32_t n_pairs_of_nodes = (n_local + 1) / 2;
    const uint32_t step = (uint32_t)a.chunk_stride * (S1_CHUNK / 2);  // node pairs between walked chunks

    uint32_t i2 = w_lo * step + threadIdx.x;  // index of my node pair in the current chunk
    uint4 cur = make_uint4(0u, 0u, 0u, 0u);
    if (w_lo < w_hi && i2 < n_pairs_of_nodes) cur = __ldcs(codes + i2);
    for (uint32_t w = w_lo; w < w_hi; ++w) {
        uint4 nxt = make_uint4(0u, 0u, 0u, 0u);
        const uint32_t i2n = i2 + step;
        if (w + 1 < w_hi && i2n < n_pairs_of_nodes) nxt = __ldcs(codes + i2n);
        if (w + 3 < w_hi) prefetch_l2(codes + i2 + 3 * step);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const uint32_t lo = h ? cur.z : cur.x, hi = h ? cur.w : cur.y;
            uint32_t acc = lds32(field_addr(lo << 6, lane_base));
            acc += lds32(field_addr(lo >> 2, lane_base) + 1u * 16384u);
            acc += lds32(field_addr(lo >> 10, lane_base) + 2u * 16384u);
            acc += lds32(field_addr(lo >> 18, lane_base) + 3u * 16384u);
            acc += lds32(field_addr(hi << 6, lane_base) + 4u * 16384u);
            acc += lds32(field_addr(hi >> 2, lane_base) + 5u * 16384u);
            acc += lds32(field_addr(hi >> 10, lane_base) + 6u * 16384u);
            acc += lds32(field_addr(hi >> 18, lane_base) + 7u * 16384u);
            const uint32_t node = i2 * 2u + (uint32_t)h;
            const bool in = node < n_local;
            const bool hit0 = in && (acc & 0xFFFFu) <= thr0;
            const bool hit1 = in && live1 && (acc >> 16) <= thr1;
            if ((hit0 || hit1) && !(DEAD && node_dead(a.dead, node))) {  // rare: append the position to the query's candidate list
                const uint32_t pos = a.base_pos + node;
                if (hit0) {
                    const uint32_t slot = atomicAdd(&a.cand_cnt[q0], 1u);
                    if (slot < (uint32_t)a.ccap) a.cand[(size_t)q0 * a.ccap + slot] = pos;
                    else a.ovf[q0] = 1u;
                }
                if (hit1) {
                    const uint32_t slot = atomicAdd(&a.cand_cnt[q1], 1u);
                    if (slot < (uint32_t)a.ccap) a.cand[(size_t)q1 * a.ccap + slot] = pos;
                    else a.ovf[q1] = 1u;
                }
            }
        }
        cur = nxt;
        i2 = i2n;
    }
}

cudaError_t launch_scan1(const Scan1Args& a, cudaStream_t st) {
    const size_t smem = (size_t)S1_TABLE + 16384;
    void (*k)(const Scan1Args) = a.dead ? scan1_kernel<true> : scan1_kernel<false>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k<<<(unsigned)(a.n_pairs * a.n_ranges), S1_T, smem, st>>>(a);
    return cudaGetLastError();
}

}  // namespace dpq
