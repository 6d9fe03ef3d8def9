// Kernel-side declarations (launch wrappers implemented in kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

#include "dpq_internal.h"

namespace dpq {

constexpr int kMaxSmem = 232448;  // 227 KB opt-in per CTA on sm_100
constexpr uint32_t kInf31 = 0x7FFFFFFFu;

// ------------------------------------------------------------------------ PTX helpers --
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// TMA bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n.reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n}\n"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(phase)
            : "memory");
    }
}
__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
    return v;
}
// table address of a record field: base + field * 16 (one IMAD) -- first-generation records
__device__ __forceinline__ uint32_t fld(uint32_t base, uint32_t field) {
    uint32_t r;
    asm("mad.lo.u32 %0, %1, 16, %2;" : "=r"(r) : "r"(field), "r"(base));
    return r;
}
// Code-array engine (dpq_internal.h "v2"): a node is NF code bytes in one 8- or 16-byte word.
template <int NF>
struct CodeWord;
template <>
struct CodeWord<8> {
    using type = uint2;
    __device__ static __forceinline__ uint2 zero() { return make_uint2(0u, 0u); }
};
template <>
struct CodeWord<16> {
    using type = uint4;
    __device__ static __forceinline__ uint4 zero() { return make_uint4(0u, 0u, 0u, 0u); }
};
// table address of centroid byte `byte` of `word`: base + centroid * ROWB (PRMT + IMAD); the
// subspace offset is added as a constant that ptxas folds into the load's immediate
template <int ROWB>
__device__ __forceinline__ uint32_t rowaddr(uint32_t base, uint32_t word, int byte) {
    return __byte_perm(word, 0u, 0x4440u + (uint32_t)byte) * (uint32_t)ROWB + base;
}
__device__ __forceinline__ uint4 lds128v(uint32_t saddr, int off) { return lds128(saddr + (uint32_t)off); }
template <int OFF>
__device__ __forceinline__ uint4 lds128o(uint32_t saddr) {
    return lds128(saddr + (uint32_t)OFF);
}
__device__ __forceinline__ uint32_t lds32(uint32_t saddr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(saddr));
    return v;
}
__device__ __forceinline__ uint2 lds64(uint32_t saddr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(saddr));
    return v;
}
// Loads only when `load` != 0; otherwise v keeps what it held (a skipped load sends no wavefront).
// The test is written into the asm so that ptxas makes it one LOP3 with a predicate output.
__device__ __forceinline__ void lds128_if(uint4& v, uint32_t saddr, uint32_t load) {
    asm volatile(
        "{\n.reg .pred p;\n"
        "setp.ne.b32 p, %5, 0;\n"
        "@p ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];\n}\n"
        : "+r"(v.x), "+r"(v.y), "+r"(v.z), "+r"(v.w)
        : "r"(saddr), "r"(load));
}
// hints: pull the line three lines ahead of the record cursor into L2 (hides HBM latency when the
// tree does not fit L2; a 16M-code tree ran 3.4x off the shared-memory bound without it), and the
// next line into L1
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

// Deleted nodes (dpq_index_delete): one bit per local position, bit (i & 31) of word i >> 5.  A null bitmap means
// nothing is deleted; the scan kernels then run their instantiation without any liveness test.
__device__ __forceinline__ bool node_dead(const uint32_t* __restrict__ dead, uint32_t i) {
    return (__ldg(dead + (i >> 5)) >> (i & 31u)) & 1u;
}

struct ScanGeom {
    int M, K, rb;      // rows = 1 << rb words per query-lane
    int pack;          // 1: one 31-bit query per lane; 2: two 15-bit queries per lane
    int qgl;           // query lanes per group (<= 32)
    int qpg;           // queries per group = qgl * pack
    int n_groups;      // ceil(Q / qpg)
    int n_slices;      // tree slices (chunk ranges) per group
    int n_warps;       // warps per CTA
    int kp;            // candidates kept per (warp, query): topk + slack, <= 256
    int kps;           // CTA-shared top-distance array length per query (kp, or 0 = disabled)
    int bcap;          // candidate buffer capacity per (warp, query): multiple of 32, >= 2*kp, <= 512
    int levels;        // depth stack levels
    size_t smem_bytes;
};

struct ScanArgs {
    ScanGeom g;
    const uint4* ops;
    const ChunkDesc* chunks;
    const uint8_t* anc;
    int n_chunks;
    const uint32_t* qlut;   // [n_groups][qgl][rows]   (swizzled, see lut kernel)
    uint64_t* cand;         // [n_items][n_warps][32*pack][bcap]
    uint32_t* gthr;         // [n_groups*qpg] exclusive distance bounds shared across slices
    uint32_t* cand_cnt;     // [n_items][n_warps][32*pack]
    int Q;
};

// ADC tables: exact float table [Q][M*K] + per-query scale + quantised swizzled table.
void launch_lut(const float* d_cw, int M, int K, int Ds, const float* d_queries, int Q,
                float* d_lutf, double* d_scale, uint32_t* d_qlut, uint32_t* d_gthr,
                const ScanGeom& g, cudaStream_t st);
// plain float tables only (dpq_adc_tables)
void launch_lut_plain(const float* d_cw, int M, int K, int Ds, const float* d_queries, int Q,
                      float* d_lutf, cudaStream_t st);

cudaError_t launch_scan(const ScanArgs& a, cudaStream_t st);

// ---- second-generation scan (scan2.cu) --------------------------------------------------
struct Scan2Core {
    V2Shape shape;
    const uint8_t* codes;         // [n_local][shape.nf] codes by position (8- or 16-byte aligned words)
    int64_t n_local;
    uint32_t base_pos;            // global position of node 0 of the shard
    int n_chunks, chunk_nodes;    // chunk c = nodes [c * chunk_nodes, ...)
    int bt_stride;                // 1: every batch; S: every S-th batch (sample pass)
    const uint16_t* qlut;         // [n_groups][2048][56] fixed-point tables
    uint64_t* cand;               // [n_items][56][bcap] candidate keys (dist << 32 | pos)
    uint32_t* cand_cnt;           // [n_items][56]
    uint32_t* gthr;               // [n_groups*56] exclusive bounds shared across tree slices
    uint32_t* ovf;                // [n_groups*56] a candidate buffer overflowed: query needs the exact fallback
    int Q, n_groups, n_slices, n_warps;
    int kp, bcap, trigger, epoch, ramp;
};
// The kernel without deletions takes Scan2Core: a larger parameter block alone changed its code generation.
struct Scan2Args : Scan2Core {
    const uint32_t* dead;         // deleted-node bitmap by local position, or null: a deleted node is never appended
};
// d_qlut == nullptr: float tables only (the coarse pipeline quantises them itself)
// d_mmax: [Q][16] floats of scratch (per-subspace table maxima; d_scale is derived from it when d_qlut is set)
void launch_lut2(const float* d_cw, int M, int K, int Ds, const float* d_queries, int Q, float* d_lutf,
                 double* d_scale, float* d_mmax, uint16_t* d_qlut, uint32_t* d_gthr, uint32_t* d_ovf, int n_groups,
                 const V2Shape& sh, uint32_t bound0, cudaStream_t st);
cudaError_t launch_scan2(const Scan2Args& a, cudaStream_t st);
// small batches: exact tables + per-subspace maxima mmax[Q][16], one block per (query, subspace)
void launch_lut_small(const float* d_cw, int M, int K, int Ds, const float* d_queries, int Q, float* d_lutf, float* d_mmax,
                      cudaStream_t st);
// program_dev.cu: codes [n][M] -> padded code words [n][stride] (stride 8 or 16, pad bytes 0)
cudaError_t launch_pad_codes(const uint8_t* codes, int64_t n, int M, int stride, uint8_t* out, cudaStream_t st);

// ---- coarse search (scan8.cu): 8-bit packed filter over the whole tree + exact re-score ----
// Coarse tables (scan8.cu).  The unit is cap / L with L > SAT ("levels", default 80): finer than the
// saturation point, so a large entry saturates.  Saturation only lowers a coarse sum (more false
// positives, never a false negative); a node within the cap has coarse sum <= L + M * 0.5, so the
// test is "sum < L + slack + 1".  On the 1M SIFT-shaped tree L = 80 leaves 4.5x fewer survivors
// than L = 31.
//   narrow (M <= 8):  one byte per entry, saturation 31 (8 x 31 <= 255), 112-byte rows, slack 4
//   wide   (M <= 16): two 4-bit entries per byte, saturation 15 (16 x 15 <= 255), 56-byte rows, slack 8
// Both serve 112 queries per CTA and fill shared memory (2048 x 112 = 4096 x 56 = 229,376 bytes).
struct C8Shape {
    int nf;         // table fields per node: 8 (narrow) or 16 (wide)
    int qb;         // queries per CTA
    int rows;       // table rows
    int row_bytes;
    int sat;        // saturation value of an entry
    int slack;      // rounding slack of a sum: nf / 2
    int lut_bytes() const { return rows * row_bytes; }
};
inline C8Shape c8_shape(int nf) { return nf == 8 ? C8Shape{8, 112, 2048, 112, 31, 4} : C8Shape{16, 112, 4096, 56, 15, 8}; }
struct Scan8Args {
    const uint8_t* codes;         // [n_local][nf] codes by position
    int64_t n_local;
    uint32_t base_pos;
    int n_chunks, chunk_nodes;
    int bt_stride;                // 1: every batch; S: every S-th batch (sample pass)
    const uint8_t* qlut8;         // [n_groups][rows][qb] coarse tables
    uint32_t* cand;               // [n_items][qb][bcap] candidate positions
    uint32_t* cand_cnt;           // [n_items][qb]
    uint32_t* ovf;                // [n_groups*qb]
    int Q, n_groups, n_slices, n_warps, bcap;
    int thresh;                   // hit iff coarse sum < thresh (= levels + slack + 1 <= 128)
    int nf;                       // 8: narrow shape, 16: wide shape (C8Shape)
    int reuse;                    // narrow shape, 1: a strand keeps its table rows and reads only those of changed code bytes
    const uint32_t* dead;         // deleted-node bitmap by local position, or null: a deleted node is never appended
    uint2* stage;                 // [SM slots][24 warps][stage_cap] survivor records (one resident CTA per SM)
    int stage_cap;                // records per warp, >= 32: how often a warp drains, never what it finds
};
// coarse tables: entry = min(SAT, rint(lut / unit)), unit = cap / levels, cap = the query's exact k-th
// distance over the sample; transposed to [group][m * 256 + centroid][112 queries]
void launch_pack8(const float* d_lutf, const float* d_cap, int M, int K, int Q, int levels, uint8_t* d_qlut8,
                  uint32_t* d_ovf, int n_groups, int nf, cudaStream_t st);
// cap of every query from the key lists of a finished search: cap[q] = distance of out_key[q][topk-1]
void launch_cap_from_keys(const uint64_t* d_keys, int topk, int Q, float* d_cap, cudaStream_t st);
// the presample's nodes (R evenly strided nodes of the shard, R <= 8192) gathered into a compact array [R][cstride]
void launch_gather_sample(const uint8_t* d_codes, int cstride, int64_t n_local, int R, uint8_t* d_out, cudaStream_t st);
// cap0[q] = exact k-th smallest distance over those R nodes (float tables, reference arithmetic): a valid,
// loose upper bound of the true k-th distance that seeds the sample pass.  d_dead (may be null): deleted sample
// nodes count as +inf, so the cap stays the k-th distance of live nodes
void launch_presample(const float* d_lutf, const uint8_t* d_sample_codes, int cstride, int64_t n_local, int M, int K, int Q,
                      int topk, int R, float* d_cap, const uint32_t* d_dead, cudaStream_t st);
cudaError_t launch_scan8(const Scan8Args& a, cudaStream_t st);
// number of %smid values of the device (the SM slots of Scan8Args::stage); d_tmp: one device int; syncs st
cudaError_t scan8_sm_slots(int* d_tmp, int* n_slots, cudaStream_t st);
struct Rescore8Args {
    const uint32_t* cand;
    const uint32_t* cand_cnt;
    const uint32_t* ovf;
    int n_groups, n_slices, bcap;
    int qb;                       // queries per group (C8Shape::qb)
    const float* lutf;            // [Q][M*K]
    const uint8_t* codes;         // node i's code = codes + i * cstride
    int cstride;
    int64_t base_pos;
    int M, K, Q, topk;
    uint64_t* out_key;            // [Q][topk] (may be null for the sample pass)
    const float* cap_in;          // [Q] a valid upper bound of the k-th distance known beforehand (may be null)
    float* cap_out;               // [Q] min(cap_in, k-th exact distance found), may be null
    uint32_t* flagged;            // queries whose candidate buffer overflowed -> exact fallback (may be null)
    uint32_t* n_flagged;
    int max_flagged;
    float* bound;                 // [Q] exact distance bound for the fallback
    int warp_form;                // 1: short lists may take the warp-per-query kernel (narrow shape, few survivors)
    int n_parts;                  // CTAs per query (ranges of slices); > 1: part / part_done scratch is used
    uint64_t* part;               // [Q][n_parts][topk] per-part results (n_parts * topk <= FB_BUF)
    uint32_t* part_done;          // [Q] zeroed arrival counters (the last CTA of a query merges and resets its counter)
};
void launch_rescore8(const Rescore8Args& a, cudaStream_t st);

// Rounds a non-negative double to the nearest float (ties to even) WITHOUT leaving the double domain:
// adding and subtracting 2^(E+29), E = the operand's exponent, drops exactly the 29 mantissa bits a float
// lacks, with the double adder's own round-to-nearest-even.  Two DADD + a few integer ops instead of the
// F2F.F32.F64 / F2F.F64.F32 pair, which run at a quarter of the FP64 add rate and bound the ADC-table
// kernel.  Zero, float subnormals and the top binade (where the float conversion may overflow) take the
// conversion itself.
// (the conversion path is a real call: inlined, the compiler if-converts the branch and executes both
// paths for every term -- ncu showed three F2F per term again)
static __device__ __noinline__ double round_to_float_by_conversion(double s) { return (double)(float)s; }
__device__ __forceinline__ double round_to_float_in_double(double s) {
    const int e = __double2hiint(s) & 0x7FF00000;
    if ((unsigned)(e - 0x38100000) <= (unsigned)(0x47D00000 - 0x38100000)) {  // 2^-126 <= s < 2^127
        const double c = __hiloint2double(e + (29 << 20), 0);
        return __dsub_rn(__dadd_rn(s, c), c);
    }
    return round_to_float_by_conversion(s);
}

// One ADC table entry in the reference's arithmetic (DCAT.h:3754-3757): float accumulator,
// each term the double square of the float difference, rounded back to float after every add.
__device__ __forceinline__ float adc_entry(const float* __restrict__ c, const float* q, int Ds) {
    double acc = 0.0;  // always holds a float-representable value
    for (int d = 0; d < Ds; ++d) {
        const double diff = (double)__fsub_rn(c[d], q[d]);
        acc = round_to_float_in_double(__fma_rn(diff, diff, acc));  // diff * diff is exact in double: same rounding as multiply, add
    }
    return (float)acc;
}

struct SelectArgs {
    ScanGeom g;
    int v2;                  // 1: lists are per (slice) with 56 queries per group (scan2.cu)
    const uint32_t* ovf;     // v2: per-query overflow flags
    const uint64_t* cand;
    const uint32_t* cand_cnt;
    const float* lutf;       // [Q][M*K]
    const double* scale;     // [Q]
    const uint8_t* codes;    // node i's code = codes + i * cstride
    int cstride;
    int64_t base_pos;
    int64_t n_local;
    int Q, topk;
    uint64_t* out_key;       // [Q][topk]
    uint32_t* flagged;       // [max_flagged] compacted ids of queries needing the fallback
    uint32_t* n_flagged;     // [1]
    int max_flagged;
    float* bound;            // [Q]: exact distance bound for the fallback
    int force_fallback;
};
void launch_select(const SelectArgs& a, cudaStream_t st);

// A query's float table [M*K] -> shared memory, 16 bytes per load and a thread's loads in flight together
// (s_lut 16-byte aligned; the table rows of lutf are when M*K is a multiple of four)
__device__ __forceinline__ void stage_table(float* s_lut, const float* __restrict__ src, int MK, int tid, int T) {
    if ((MK & 3) == 0) {
        const float4* s4 = reinterpret_cast<const float4*>(src);
        float4* d4 = reinterpret_cast<float4*>(s_lut);
#pragma unroll 4
        for (int i = tid; i < MK / 4; i += T) d4[i] = __ldg(s4 + i);
    } else {
        for (int i = tid; i < MK; i += T) s_lut[i] = src[i];
    }
}

// Exact distance of one node in the reference's arithmetic: float table entries summed in double.
// The node's code is fetched with ONE vector load when the stride is 8 or 16 bytes (the code-array
// engine): sixteen byte loads per candidate, each lane on another line, made the exact kernels
// L1-transaction bound (ncu launch list, round 2).
__device__ __forceinline__ double exact_dist(const float* __restrict__ lut, const uint8_t* __restrict__ code, int cstride,
                                             int M, int K) {
    double d = 0.0;
    if (cstride == 8) {
        const uint2 w = *reinterpret_cast<const uint2*>(code);
        const uint32_t ww[2] = {w.x, w.y};
#pragma unroll
        for (int m = 0; m < 8; ++m)
            if (m < M) d += (double)lut[m * K + ((ww[m >> 2] >> (8 * (m & 3))) & 0xFFu)];
    } else if (cstride == 16) {
        const uint4 w = *reinterpret_cast<const uint4*>(code);
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int m = 0; m < 16; ++m)
            if (m < M) d += (double)lut[m * K + ((ww[m >> 2] >> (8 * (m & 3))) & 0xFFu)];
    } else {
        for (int m = 0; m < M; ++m) d += (double)lut[m * K + code[m]];
    }
    return d;
}

// Upper bound of exact_dist from float adds only (no conversions): the float sum of M non-negative
// entries is within (M - 1) * 2^-24 of the real sum, the exact value within 2^-24 of it.
__device__ __forceinline__ float dist_upper_bound(const float* __restrict__ lut, const uint8_t* __restrict__ code, int cstride,
                                                  int M, int K) {
    float d = 0.0f;
    if (cstride == 8) {
        const uint2 w = *reinterpret_cast<const uint2*>(code);
        const uint32_t ww[2] = {w.x, w.y};
#pragma unroll
        for (int m = 0; m < 8; ++m)
            if (m < M) d += lut[m * K + ((ww[m >> 2] >> (8 * (m & 3))) & 0xFFu)];
    } else if (cstride == 16) {
        const uint4 w = *reinterpret_cast<const uint4*>(code);
        const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int m = 0; m < 16; ++m)
            if (m < M) d += lut[m * K + ((ww[m >> 2] >> (8 * (m & 3))) & 0xFFu)];
    } else {
        for (int m = 0; m < M; ++m) d += lut[m * K + code[m]];
    }
    return __fmul_ru(d, 1.0f + 1.0f / 131072.0f);  // M <= 64 terms: 2^-17 covers 64 * 2^-24 with room
}

// Block-wide running top-k used by the exact kernels (fallback, re-score): s_keys[0 .. *s_n) holds
// candidate keys (distance bits << 32 | position, unique); the call sorts them (bitonic, whole CTA),
// keeps the topk smallest and makes the k-th key the new exclusive bound *s_thr.  Every thread of
// the CTA must call it; *s_n is read after a barrier.
constexpr int FB_BUF = 2048;
__device__ __forceinline__ void fb_compact(uint64_t* s_keys, uint32_t* s_n, unsigned long long* s_thr, int topk) {
    const int T = (int)blockDim.x;
    const int n = (int)*s_n;  // uniform: read after a barrier
    int np2 = 1;
    while (np2 < n) np2 <<= 1;
    for (int i = n + threadIdx.x; i < np2; i += T) s_keys[i] = ~0ull;
    __syncthreads();
    for (int k = 2; k <= np2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < np2; i += T) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const uint64_t x = s_keys[i], y = s_keys[ixj];
                    const bool up = (i & k) == 0;
                    if ((x > y) == up) {
                        s_keys[i] = y;
                        s_keys[ixj] = x;
                    }
                }
            }
            __syncthreads();
        }
    if (threadIdx.x == 0) {
        *s_n = (uint32_t)(n < topk ? n : topk);
        if (n >= topk) *s_thr = s_keys[topk - 1] - 1ull;  // keys are unique: only strictly better keys pass
    }
    __syncthreads();
}

// Exact fallback for flagged queries: a running top-k over every node of the shard (kernels.cu).
struct FallbackArgs {
    const uint32_t* flagged;    // [max_flagged] query ids
    const uint32_t* n_flagged;  // [1] device-side count
    int max_flagged;
    const float* lutf;
    const float* bound;         // [Q] inclusive distance bound known to hold the k-th best (FLT_MAX: none)
    const uint8_t* codes;       // node i's code = codes + i * cstride
    int cstride;
    int64_t base_pos, n_local;
    int M, K, topk;
    uint64_t* part;             // [max_flagged][fallback_slices(topk)][topk] per-slice results
    uint64_t* out_key;          // [Q][topk]
    const uint32_t* dead;       // deleted-node bitmap by local position, or null
};
// slices of the exact fallback: as many as fit the merge buffer (slices x topk <= FB_BUF), at most 16
inline int fallback_slices(int topk) { return topk >= 1 ? (FB_BUF / topk < 16 ? (FB_BUF / topk < 1 ? 1 : FB_BUF / topk) : 16) : 1; }
void launch_fallback(const FallbackArgs& a, cudaStream_t st);

void launch_merge(const uint64_t* d_keys, int n_lists, int Q, int topk, uint64_t* d_out,
                  cudaStream_t st);
// keys (distance bits << 32 | position) -> positions, ids (pos2id[pos - base_pos], or the position when
// pos2id is null), distance bits, each to its own array (null = not wanted; device-mapped host memory is
// fine); the four control words of the search are copied to out_ctrl alongside
void launch_unpack(const uint64_t* d_keys, size_t n, const uint32_t* d_pos2id, uint32_t base_pos, uint32_t* out_pos,
                   uint32_t* out_id, uint32_t* out_dist, const uint32_t* d_ctrl, uint32_t* out_ctrl, cudaStream_t st);

// ---- latency mode (scan1.cu): lanes = nodes, two queries per pass over the code array ----
struct Scan1Args {
    const uint8_t* codes;         // [n_local][8] codes by position (16-byte aligned)
    int64_t n_local;
    uint32_t base_pos;
    const float* lutf;            // [Q][M*K] exact tables
    const float* mmax;            // [Q][16] per-subspace maxima of the tables (lut_small_kernel)
    const float* cap;             // [Q] inclusive distance bound (FLT_MAX: none)
    int M, K, Q;
    int n_pairs;                  // ceil(Q / 2): query pairs, each pair has its own CTAs
    int n_ranges;                 // tree ranges per pair (n_pairs * n_ranges CTAs, one per SM)
    int chunk_stride;             // 1: every 2048-node chunk; S: every S-th chunk (sample pass)
    uint32_t* cand;               // [Q][ccap] candidate positions
    uint32_t* cand_cnt;           // [Q]
    uint32_t* ovf;                // [Q]
    int ccap;
    const uint32_t* dead;         // deleted-node bitmap by local position, or null: a deleted node is never appended
};
cudaError_t launch_scan1(const Scan1Args& a, cudaStream_t st);
// exact re-score of scan1's candidate lists: one CTA per query, running top-k on (distance, position)
struct Rescore1Args {
    const uint32_t* cand;         // [Q][ccap]
    const uint32_t* cand_cnt;     // [Q]
    const uint32_t* ovf;          // [Q]
    int ccap;
    const float* lutf;
    const uint8_t* codes;
    int cstride;
    int64_t base_pos;
    int M, K, Q, topk;
    uint64_t* out_key;            // [Q][topk] or null (sample pass)
    const float* cap_in;          // [Q]
    float* cap_out;               // [Q] min(cap_in, exact k-th distance found), or null
    uint32_t* flagged;            // queries whose list overflowed -> exact fallback (or null)
    uint32_t* n_flagged;
    int max_flagged;
    float* bound;                 // [Q] bound for the fallback
    int n_parts;                  // CTAs per query (ranges of the candidate list); n_parts * topk <= FB_BUF
    uint64_t* part;               // [Q][n_parts][topk]
    uint32_t* part_done;          // [Q] zeroed arrival counters (self-resetting)
};
void launch_rescore1(const Rescore1Args& a, cudaStream_t st);

// ---- deletion (dead.cu): ids -> bits of the deleted-node bitmap ------------------------------------
// d_ids [n_ids] sorted ascending; node i (local position) has id pos2id[i], or base_pos + i when pos2id is null.
// set = true: sets the bit of every node whose id is listed; false: clears it.  Every 32-node word is written
// by one thread; *d_count (zeroed by the caller) receives the number of set bits of the whole bitmap.
void launch_mark_dead(const uint32_t* d_ids, int64_t n_ids, const uint32_t* d_pos2id, uint32_t base_pos, int64_t n_local,
                      bool set, uint32_t* d_dead, unsigned long long* d_count, cudaStream_t st);
// CUB radix sort of n ids (d_temp = null: *temp_bytes receives the scratch size and nothing runs)
cudaError_t sort_ids(const uint32_t* d_in, uint32_t* d_out, int n, void* d_temp, size_t* temp_bytes, cudaStream_t st);

// ---- appended nodes (add.cu): the layout of an add batch --------------------------------------------
// Sorts the rows of d_codes [n][M] by their padded code word of nf bytes (subspace 0 most significant; ties by
// input row, the sorts being stable).  d_keys: [2n], d_vals: [2n]; the order (input row of each appended node)
// is left in d_vals + n.  d_temp = null: *temp_bytes receives the scratch size and nothing runs.
cudaError_t sort_add_batch(const uint8_t* d_codes, int64_t n, int M, int nf, uint64_t* d_keys, uint32_t* d_vals, void* d_temp,
                           size_t* temp_bytes, cudaStream_t st);
// Appended node i = input row d_perm[i] (row i when d_perm is null): its code word padded to nf bytes goes to
// d_out_codes [n][nf], its id (d_ids[row], or its position when d_ids is null) to d_out_ids [n] (skipped when
// null), and its position first_pos + i to d_out_pos[row].
cudaError_t launch_add_gather(const uint8_t* d_codes, int64_t n, int M, int nf, const uint32_t* d_perm, const uint32_t* d_ids,
                              uint32_t first_pos, uint8_t* d_out_codes, uint32_t* d_out_ids, uint32_t* d_out_pos, cudaStream_t st);
// secondary.cu: the SIMT encoder (any Ds)
cudaError_t launch_encode(const float* d_cw, int M, int K, int Ds, const float* d_x, int64_t n, int D, uint8_t* d_codes,
                          cudaStream_t st);

}  // namespace dpq
