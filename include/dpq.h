/* dpq.h -- C ABI of the B200-native DeltaPQ query hot path (libdpq.so).
 *
 * The reference (RunhuiWang/DeltaPQ) has no plugin/FFI layer: its hot path is a set of free
 * functions in deltapq_create_approx_tree.h ("DCAT.h") called from the per-query loop of
 * deltapq_approx_tree_main.cpp ("dmain") and main.cpp ("pmain").  Each entry point below
 * names the reference function / call site it replaces.  Plain C: opaque handles, int
 * status returns (0 = ok, negative = error, text via dpq_last_error()), caller-owned
 * buffers, no C++ or torch types.  One handle is used from one host thread at a time.
 * There is no CPU fallback: every compute entry point fails with DPQ_ERR_CUDA when no
 * sm_100 device is usable.
 */
#ifndef DPQ_H
#define DPQ_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define DPQ_OK 0
#define DPQ_ERR_ARG (-1)    /* bad argument / unsupported shape */
#define DPQ_ERR_CUDA (-2)   /* CUDA runtime error or no device */
#define DPQ_ERR_FORMAT (-3) /* malformed tree stream / file */
#define DPQ_ERR_IO (-4)
#define DPQ_ERR_NOMEM (-5)

typedef struct dpq_index dpq_index;

/* ---- library ------------------------------------------------------------------------ */
int dpq_version(void);
const char* dpq_last_error(void); /* thread-local text of the last failure */
int dpq_device_count(void);       /* number of visible CUDA devices (0 without a GPU) */
int dpq_set_device(int device);   /* device used by this host thread's calls and by handles it creates afterwards */

/* ---- DeltaTree index (the scan operand) --------------------------------------------- */
/* Opens a compressed DeltaTree ("DTC", SURVEY App. A.5; writer DCAT.h:1765-1842) that is
 * already in host memory.  payload = the stream WITHOUT its 16-byte header, exactly what
 * query_processing_scan_compressed_codes_opt_in_memory (DCAT.h:3731) takes.  pos2id maps a
 * DFS position to the vector id (QNode.vec_id, DCAT.h:79) and may be NULL.
 * The stream is uploaded and decoded ON THE GPU (program_dev.cu) into the device program: the
 * nodes' codes by DFS position, 8 bytes per node at M <= 8 (16 at M <= 16).  DPQ_HOST_DECODE=1
 * keeps the sequential host decoder.
 *
 * rank / n_ranks shard the tree by whole depth-1 subtrees balanced by stream bytes
 * (SURVEY 8e): rank r keeps only its subtrees, prefixed by the global root code; reported
 * positions stay GLOBAL.  Rank 0 also scores the root.  Use rank=0,n_ranks=1 for the
 * whole tree. */
int dpq_index_open(const uint8_t* payload, int64_t n_bytes, int64_t n_codes, int M, int K,
                   const uint32_t* pos2id, int rank, int n_ranks, dpq_index** out);

/* One tree of a FOREST: the code set is cut into parts by vector id, every part gets its own
 * DeltaTree (dpq_tree_build on the GPU that will scan it), and the parts' local top-k lists
 * merge with dpq_merge_topk_device exactly as subtree shards do.  (The reference builds ONE
 * tree over all codes; so does dpq_tree_build_device + dpq_index_open_tree_shard below, which
 * is what config C5 runs.  The forest is for code sets that arrive in pieces.)  The whole tree is kept; first_pos is added to every position the index
 * reports, so positions are unique across the forest (part p of equal parts: p * n_codes);
 * pos2id is this tree's own [n_codes] table (callers add the part's first vector id). */
int dpq_index_open_part(const uint8_t* payload, int64_t n_bytes, int64_t n_codes, int M, int K,
                        const uint32_t* pos2id, int64_t first_pos, dpq_index** out);

/* Same, reading "<dataset>/M{M}K{K}_Approx_compressed_codes_opt_N{N}" style files
 * (header int64 n_codes, int64 n_bytes; DCAT.h:2822-2824).  qnode_path (the 60-byte/node
 * "..._Approx_TreeNodesDFS_N{N}" file, DCAT.h:1484) may be NULL. */
int dpq_index_open_file(const char* tree_path, const char* qnode_path, int M, int K, int rank,
                        int n_ranks, dpq_index** out);

/* Opens a tree that dpq_tree_build / dpq_tree_from_edges just produced, without going through its
 * byte stream: the device scan program is the tree's code array by DFS position (8 bytes per node at
 * M = 8), uploaded as it is instead of decoding the sequential stream on the host.
 * Same index as dpq_index_open_part(payload, ..., vec_id, first_pos); t stays owned by the caller
 * and may be freed afterwards.  (dpq_tree is declared further down.) */
struct dpq_tree;
int dpq_index_open_tree(struct dpq_tree* t, int64_t first_pos, dpq_index** out);

/* Shard `rank` of `n_ranks` of such a tree: whole depth-1 subtrees balanced by stream bytes (SURVEY
 * 8e; subtree ranges as in DCAT.h:1156-1183), the same deal as dpq_index_open(payload, ..., rank,
 * n_ranks); positions stay global.  With a device-resident tree (dpq_tree_build_device) nothing
 * crosses PCIe: the shard's slice of the code array is copied device to device.  This is how the
 * 10^9-code tree of config C5 is opened on 1 / 2 / 4 / 8 GPUs. */
int dpq_index_open_tree_shard(struct dpq_tree* t, int rank, int n_ranks, dpq_index** out);

/* dpq_index_open_part reading the part's files (tree file with its 16-byte header; 60-byte
 * QNode file or NULL). */
int dpq_index_open_part_file(const char* tree_path, const char* qnode_path, int M, int K, int64_t first_pos,
                             dpq_index** out);

/* Codebook [M][K][Ds] as PQ::ReadCodewords returns it (pq.cpp:288-312). */
int dpq_index_set_codebook(dpq_index* idx, const float* codewords, int Ds);

/* Run this handle's work on the caller's CUDA stream (a cudaStream_t; NULL = the legacy
 * default stream) instead of the handle's own, so that a host that already owns streams
 * and events (bench.py: torch.cuda.current_stream()) can order and time the searches and
 * the NCCL gather on one stream.  The handle does not take ownership. */
int dpq_index_set_stream(dpq_index* idx, void* cuda_stream);

/* Tuning knobs (optional): "slices", "warps", "slack" (extra candidates re-scored exactly),
 * "epoch", "trigger", "ramp" (candidate collection of the 15-bit scan); "coarse" (-1 auto, 0 off,
 * 1 on), "sample", "seed" (1: the sample pass is a coarse scan seeded by an exact presample),
 * "refine" (stride of a second, denser sample pass; automatic on shards above 16.8M nodes), "stight"
 * (percent of the presample cap the first sampled pass accepts, default 100), "presample", "parts8",
 * "levels8", "bcap8", "warps8", "coarse_min" (coarse search); "latency" (-1 auto, 0 off, 1 on: lanes =
 * nodes scan for a handful of queries); "add_order" (1 default: an add batch is laid out sorted by code word, 0:
 * in input order);
 * first-generation engine only: "pack" (1 = 31-bit, 2 = 2x15-bit filter). */
int dpq_index_set_option(dpq_index* idx, const char* name, int64_t value);

/* Deletes vectors from an open index (an extension: the reference's trees are rebuilt to drop a vector).  An id
 * is the value this handle reports as out_id: pos2id[pos] when the index has a pos2id table, else the position
 * (a forest part: its own vec_id, as dpq_index_open_part says).  Deletions accumulate; deleting an id twice is
 * harmless; ids with no node in this shard are ignored, so every shard can be given the same list; n = 0 does
 * nothing; ids == NULL with n > 0 is DPQ_ERR_ARG.  A deleted node stays in the tree as a tombstone: it is still
 * scanned but never reported, and every search returns the top-k over the LIVE nodes with the usual rule
 * (ascending distance, ties by lower position, the same distance bits), padded with (0xFFFFFFFF, FLT_MAX) when
 * fewer than topk nodes are live.  The bitmap (one bit per node of the shard) appears on the first delete.
 * dpq_index_undelete clears the same bits; once nothing is deleted the index answers exactly as one that never
 * had deletions.  The call runs on the index's stream (the caller's after dpq_index_set_stream) and returns
 * once the change is complete: every search issued after it sees it.  Deletions reach a file through
 * dpq_index_compact, which drops the deleted nodes from a rebuilt tree.
 * The first-generation engine (DPQ_ENGINE=1) has no deletion: DPQ_ERR_ARG.  Stat "n_deleted": nodes of this
 * shard currently deleted; "last_delete_us": host wall time of the last call. */
int dpq_index_delete(dpq_index* idx, const uint32_t* ids, int64_t n);
int dpq_index_undelete(dpq_index* idx, const uint32_t* ids, int64_t n);

/* Adds vectors to an open index (an extension, like deletion).  codes is [n][M]; x is [n][D] floats with
 * D <= M*Ds, zero-padded like dpq_encode and encoded on the device with this index's codebook
 * (dpq_index_set_codebook first, else DPQ_ERR_ARG) by the same kernels, so the codes are bit-identical to
 * dpq_encode's.  codes / x / ids / out_pos may be host pointers or device pointers of any device: input that is
 * not on the index's device is copied there first (no peer access is needed).  ids may be NULL: a node's id is then
 * its position.  out_pos (may be NULL) receives the position given to input row i at out_pos[i].
 * Positions: appended nodes continue this index's range, base_pos + n_local, + 1, ... and every search path
 * scores them exactly like tree nodes.  Only an index whose range ends the position space accepts adds: a whole
 * tree, the last shard (rank = n_ranks - 1, also when it is empty) or a forest part; another shard returns
 * DPQ_ERR_ARG.  A lone forest part continues at first_pos + n_codes + j: keeping those positions clear of the next
 * part is the caller's job (dpq_multi_add does it).  A position reaching 0xFFFFFFFF is DPQ_ERR_ARG and changes
 * nothing; so are n > 2^31 - 1, a null codes / x with n > 0, a code byte >= K and the first-generation engine
 * (DPQ_ENGINE=1).  n = 0 does nothing.
 * Layout: each call's batch is sorted on the device by code word (subspace 0 most significant, ties by input
 * row) and appended in that order, so that neighbouring positions share centroids as DFS neighbours of the tree
 * do; set_option("add_order", 0) appends in input order instead.
 * Ids: an index without a pos2id table keeps none while ids is NULL (id = position); the first add that names
 * ids creates one, identity over the nodes it already had.  Duplicate ids are allowed: dpq_index_delete removes
 * every node that carries the id, and a node added after its id was deleted is live (the bitmap is per node).
 * The call runs on the index's stream and returns once the change is complete.  Adds reach a file through
 * dpq_index_compact, which builds them into the tree.  Stats: "n_added" (appended nodes), "last_add_us"; "n_local" counts appended nodes, "n_codes" does not. */
int dpq_index_add(dpq_index* idx, const uint8_t* codes, int64_t n, const uint32_t* ids, uint32_t* out_pos);
int dpq_index_add_vectors(dpq_index* idx, const float* x, int64_t n, int D, const uint32_t* ids, uint32_t* out_pos);

/* Compacts an open index (an extension, like deletion and adds; the reference rebuilds its trees): the live nodes,
 * tree nodes and appended ones alike, are gathered on the device in ascending position, a new DeltaTree is built
 * over them on the device (the edge search and layout of dpq_tree_build_device with -h 1, -method 1 and this
 * index's codebook), and it replaces the index's tree.  Afterwards no node is deleted or appended: n_codes = n_local
 * = the live count, and n_bytes, n_diffs, n_chunks and the depth histogram are the new tree's.
 * Positions are renumbered: the new tree's DFS order, from the same base_pos (a forest part keeps first_pos).
 * Ids are not: every node reports the id it reported before, and the index always has an id table afterwards (an
 * index that had none reports each node's old position as its id).  Deletions, adds and searches continue on the
 * new tree as on any other (adds take the positions after the live count).  Options, stream and codebook are kept.
 * out_tree (may be NULL) receives the new tree as dpq_tree_build(live codes) returns it, vec_id mapped to the ids:
 * "payload", "vec_id", "depth", "codes_by_pos", "n_codes", "n_diffs" and, at M = 8, "qnodes" (vec_id field = the
 * id), which are the bytes of the reference's files; the caller writes them and frees the tree with dpq_tree_free.
 * Without out_tree nothing but the index's own id table leaves the device.
 * DPQ_ERR_ARG, index unchanged: a shard of a tree split over n_ranks > 1 (dpq_multi_compact), no codebook, the
 * first-generation engine (DPQ_ENGINE=1), no live node.  Any failure (e.g. out of memory during the edge search)
 * leaves the index unchanged and searchable.  The gather runs on the index's stream, the build on the device's
 * legacy stream; the call returns once everything is complete.  Stats: "last_compact_us" (host wall time),
 * "last_compact_gather_us", "last_compact_edge_us", "last_compact_layout_us", "last_compact_build_us" (edge search
 * + layout). */
int dpq_index_compact(dpq_index* idx, struct dpq_tree** out_tree);

/* Replaces the per-query loop dmain:328-344 calling
 * query_processing_scan_compressed_codes_opt_o_direct (DCAT.h:2805) /
 * ..._in_memory (DCAT.h:3731): ADC table build, DeltaTree scan, top-k.
 * queries [Q][M*Ds] host floats; outputs [Q][topk], ascending distance, ties by lower
 * position: out_pos = DFS position (what the reference returns), out_id = pos2id[pos]
 * (NULL allowed), out_dist = float(sum of the node's M table entries), i.e. the value
 * the reference's double accumulation rounds to.  Entries beyond the number of nodes in
 * the shard are (0xFFFFFFFF, FLT_MAX). */
int dpq_index_search(dpq_index* idx, const float* queries, int Q, int topk, uint32_t* out_pos,
                     uint32_t* out_id, float* out_dist);

/* Device-resident variant: all pointers are DEVICE pointers, work is enqueued on the
 * index stream; call dpq_index_sync() before reading.  Used by bench.py ("value": inputs
 * resident in HBM) and by the multi-GPU driver, which all-gathers out_key over NCCL.
 * out_key [Q][topk] = (uint64) float_bits(dist) << 32 | pos, ascending. */
int dpq_index_search_device(dpq_index* idx, const float* d_queries, int Q, int topk,
                            uint64_t* d_out_key);
int dpq_index_sync(dpq_index* idx);

/* Merge n_lists sorted top-k key lists per query (device pointers; [n_lists][Q][topk])
 * into one [Q][topk]: the post-gather step of the sharded scan (SURVEY 8e). */
int dpq_merge_topk_device(dpq_index* idx, const uint64_t* d_keys, int n_lists, int Q, int topk,
                          uint64_t* d_out_key);

/* ---- multi-GPU search, one process (SURVEY 8e) ------------------------------------------ */
/* One shard per GPU (devices 0..n_gpus-1, whole depth-1 subtrees balanced by stream bytes),
 * local top-k with global positions on every GPU, ONE collective (NCCL all-gather of the
 * Q x k keys over NVLink, libnccl.so.2 bound at run time) and the k-way merge kernel.  Used by
 * `deltapq -task query -gpus N`.  Same argument meaning as dpq_index_open_file / _search. */
typedef struct dpq_multi dpq_multi;
int dpq_multi_open_file(const char* tree_path, const char* qnode_path, int M, int K, int n_gpus,
                        dpq_multi** out);
/* Forest variant (`deltapq -task query -parts P`, the 1B-code layout): n_parts independently
 * built trees (files of `deltapq -task approx_tree -parts P`), part p reporting positions
 * first_pos[p] + its own DFS position and ids first_pos[p] + its own vec_id (parts are vector-id
 * ranges); the parts are dealt round-robin to the GPUs, each GPU merges its parts' lists, then
 * the same single all-gather + merge.  qnode_paths (or single entries) may be NULL. */
int dpq_multi_open_parts(const char* const* tree_paths, const char* const* qnode_paths, const int64_t* first_pos,
                         int n_parts, int M, int K, int n_gpus, dpq_multi** out);
int dpq_multi_set_codebook(dpq_multi* m, const float* codewords, int Ds);
int dpq_multi_search(dpq_multi* m, const float* queries, int Q, int topk, uint32_t* out_pos,
                     uint32_t* out_id, float* out_dist);
int64_t dpq_multi_stat(dpq_multi* m, int rank, const char* name); /* dpq_index_stat of one shard / part */
/* dpq_index_delete / _undelete for every shard or part.  The ids are vector ids: with a QNode file they are
 * translated to global positions through it first; without one an id is the global position.  Every shard /
 * part is given the same list and keeps the nodes it holds. */
int dpq_multi_delete(dpq_multi* m, const uint32_t* ids, int64_t n);
int dpq_multi_undelete(dpq_multi* m, const uint32_t* ids, int64_t n);
/* dpq_index_add / _add_vectors for the handle: the whole batch goes to the index that ends the position space
 * (the last shard, or the part with the largest first_pos) and the new positions continue the global space.
 * The handle's id table grows with them (created as identity when it was empty and ids are given), so that
 * dpq_multi_search reports the ids and dpq_multi_delete takes them.  As for dpq_index_add, the inputs may be on
 * any device.  Every add lands on that one GPU, a known imbalance of the search load until dpq_multi_compact. */
int dpq_multi_add(dpq_multi* m, const uint8_t* codes, int64_t n, const uint32_t* ids, uint32_t* out_pos);
int dpq_multi_add_vectors(dpq_multi* m, const float* x, int64_t n, int D, const uint32_t* ids, uint32_t* out_pos);
/* dpq_index_compact for the handle (dpq_multi_set_codebook first).  Subtree shards (dpq_multi_open_file): the live
 * nodes of every shard are gathered in global position order onto GPU 0, one tree is built there and dealt to the
 * GPUs again by whole depth-1 subtrees balanced by stream bytes, as dpq_multi_open_file deals a file, so appended
 * nodes are spread over every GPU.  Forest parts (dpq_multi_open_parts): every part is compacted in place on its
 * GPU and keeps its first_pos.  Positions are renumbered, ids kept (the handle's id table is rebuilt; without one
 * before, a node's id is its old global position).  DPQ_ERR_ARG, handle unchanged: no codebook, the first-generation
 * engine (DPQ_ENGINE=1), no live node (shards) or a part without a live node (parts).  With n_gpus > 1 the gather
 * onto GPU 0 copies across devices with cudaMemcpyAsync (peer or host-staged). */
int dpq_multi_compact(dpq_multi* m);
void dpq_multi_close(dpq_multi* m);

/* Raw device allocation helpers for hosts without a CUDA binding (ctypes, cgo, JNI). */
int dpq_malloc(void** dptr, size_t bytes);
int dpq_free(void* dptr);
int dpq_memcpy_h2d(void* dst, const void* src, size_t bytes);
int dpq_memcpy_d2h(void* dst, const void* src, size_t bytes);
int dpq_malloc_host(void** hptr, size_t bytes); /* pinned */
int dpq_free_host(void* hptr);

/* Introspection: "n_codes", "n_bytes" (algorithmic stream bytes of this shard),
 * "n_local" (nodes scanned by this rank), "n_diffs", "n_chunks", "ops_bytes",
 * "last_launches" (kernels launched by the last search), "last_fallback" (queries that
 * took the exact fallback in the last search), "last_scan_us" (scan kernel time of the
 * last search, CUDA events), "last_total_us"; "sum_scan_ns" / "sum_lut_ns" / "sum_total_ns" /
 * "timed_calls": the same summed over every search since set_option("timing_reset");
 * "last_coarse" (1 when the last search used the sample -> 8-bit coarse scan -> exact re-score
 * path), "last_latency" (1: latency mode), "last_scan8_us" / "sum_scan8_ns" (the coarse scan kernel
 * alone; in latency mode the full scan1 pass), "device_bytes_per_node", "engine"; "n_deleted",
 * "last_delete_us" (dpq_index_delete); "n_added", "last_add_us" (dpq_index_add); "last_compact_us" and its stages
 * (dpq_index_compact). */
int64_t dpq_index_stat(dpq_index* idx, const char* name);

void dpq_index_close(dpq_index* idx);

/* Host-only introspection of the tree compiler (no GPU needed): compiles the stream exactly
 * as dpq_index_open does and lets a test copy the device program out and interpret it.
 * `what`: "ops" (uint32), "chunks" (4 x uint32 each), "anc" (uint8), "codes" (uint8),
 * scalars "n_ops", "n_chunks", "n_local", "base_pos", "rb", "levels", "n_bytes", "n_diffs". */
typedef struct dpq_program dpq_program;
int dpq_program_compile(const uint8_t* payload, int64_t n_bytes, int64_t n_codes, int M, int K,
                        int rank, int n_ranks, int chunk_nodes, dpq_program** out);
int64_t dpq_program_size(dpq_program* p, const char* what); /* bytes for arrays, value for scalars */
int dpq_program_copy(dpq_program* p, const char* what, void* dst);
void dpq_program_free(dpq_program* p);

/* ---- stand-alone kernels ------------------------------------------------------------- */
/* ADC tables of Q queries, lut[Q][M][K] (DCAT.h:2841-2849 / :3750-3758), host buffers. */
int dpq_adc_tables(const float* codewords, int M, int K, int Ds, const float* queries, int Q,
                   float* lut);

/* PQTree::EncodePlain (pq_tree.cpp:192-253) over n vectors x[n][D], D <= M*Ds (zero
 * padded): codes[n][M], bit-exact (sequential FP32, no FMA, strict <).  x and codes may be
 * host or device pointers (unified addressing; device-resident x and codes are used in place);
 * codewords is a host pointer.  Ds in {4, 8, 16}: the K scores of 128 vectors come from one
 * tcgen05.mma group (bf16 hi/lo split) used as a filter, and only the centroids within the
 * rigorous error bound of the best score are re-scored in the reference's arithmetic
 * (encode_tc.cu; DPQ_ENCODE_TC=0 selects the SIMT kernel); other Ds: SIMT kernel. */
int dpq_encode(const float* codewords, int M, int K, int Ds, const float* x, int64_t n, int D,
               uint8_t* codes);

/* Same for uint8 components (bvecs, utils.cpp:43-71 converts them to float before EncodePlain):
 * vector i = the D bytes at x + i * row_stride + row_offset, so a block of raw .bvecs records
 * (4-byte dimension header + D bytes each) is passed as it was read: row_stride = D + 4,
 * row_offset = 4.  The conversion runs on the device; a quarter of the bytes cross PCIe. */
int dpq_encode_u8(const float* codewords, int M, int K, int Ds, const uint8_t* x, int64_t n, int D,
                  int64_t row_stride, int64_t row_offset, uint8_t* codes);
/* About the calling thread's process-wide last encode call: "tc" (1 = tensor-core path),
 * "kernel_us" (device time of its encode kernels, CUDA events); -1 for an unknown name. */
int64_t dpq_encode_stat(const char* name);

/* find_edges_by_diff_approx (DCAT.h:1207-1332) with the canonical stable-sort tie rule:
 * edges[n_codes-1][2] = (parent id, child id) in emission order, *root_id. */
int dpq_find_edges(const uint8_t* codes, int64_t n_codes, int M, int K, int max_height_folds,
                   int method, uint32_t* edges, uint32_t* root_id);

/* create_approx_tree (DCAT.h:970-1065), the whole `deltapq -task approx_tree` computation:
 * edge search on the GPU (dpq_find_edges), then the DFS layout
 * edges_to_tree_index_approx_dfs_layout (DCAT.h:1334-1487) and the stream writer
 * qnodes_to_compressed_codes_opt (DCAT.h:1730-1845), also on the GPU (layout.cu; the
 * sequential host form of the same stage is dpq_tree_from_edges).  codewords [M][K][Ds] feed the K x K
 * centroid tables (dmain:101-118) that order the children.  dpq_tree_from_edges is the host
 * half alone (no GPU needed).  Arrays are fetched by name with dpq_tree_size / dpq_tree_copy:
 *   "edges" uint32[n-1][2] (the ..._Approx_Edges file body), "root_id",
 *   per DFS position: "vec_id" "parent_pos" "child_num" (uint32), "depth" (uint8),
 *   "max_dist" "max_dist2p" (float), "codes_by_pos" uint8[n][M];
 *   "qnodes": the (n+1) x 60-byte ..._Approx_TreeNodesDFS file body (M == 8 only);
 *   "payload": the ..._Approx_compressed_codes_opt stream without its 16-byte header
 *   (M > 8: extension format, ceil(M/8) bitmap bytes); scalars "n_diffs", "n_codes",
 *   "edge_us" / "layout_us" (wall time of the two stages of dpq_tree_build). */
typedef struct dpq_tree dpq_tree;
int dpq_tree_build(const uint8_t* codes, int64_t n_codes, int M, int K, const float* codewords, int Ds,
                   int max_height_folds, int method, dpq_tree** out);
int dpq_tree_from_edges(const uint8_t* codes, int64_t n_codes, int M, int K, const float* codewords,
                        int Ds, const uint32_t* edges, uint32_t root_id, dpq_tree** out);
/* dpq_tree_build with the result left in HBM: codes may be a host or a DEVICE pointer, the edges
 * go from the edge search to the layout without leaving the device, and of the layout only what an
 * index needs is kept (codes by position, depth, vec_id, the byte stream and its record offsets).
 * dpq_tree_size / dpq_tree_copy serve "vec_id", "depth", "codes_by_pos", "payload" (copied to the
 * host on request) and the scalars ("on_device" = 1, "depth_hist_<d>"); open it with
 * dpq_index_open_tree_shard.  One tree over 10^9 codes (DCAT.h:970-1065 builds ONE tree over all N,
 * guard N < INT_MAX at :982) needs about 110 GB of HBM during the edge search and none of the
 * 43 bytes per node of host memory the host-resident form takes. */
int dpq_tree_build_device(const uint8_t* codes, int64_t n_codes, int M, int K, const float* codewords, int Ds,
                          int max_height_folds, int method, dpq_tree** out);
int64_t dpq_tree_size(dpq_tree* t, const char* what); /* bytes for arrays, value for scalars */
int dpq_tree_copy(dpq_tree* t, const char* what, void* dst);
void dpq_tree_free(dpq_tree* t);

/* check_num_diffs / dfs_node_layout diff extraction (DCAT.h:196-238, 1156-1183): for each
 * edge the changed-subspace bitmap (bit m set <=> codes differ in subspace m);
 * returns the total number of diffs through *n_diffs. */
int dpq_edge_diffs(const uint8_t* codes, int64_t n_codes, int M, const uint32_t* edges,
                   int64_t n_edges, uint32_t* bitmaps, int64_t* n_diffs);

/* Exact brute-force ground truth (pmain:138-166, 569-669): base[n][D] (ids id0..),
 * queries[Q][D]; accumulates into a state created by dpq_groundtruth_begin.  For topk <= 64
 * the Q x n x D inner products run on the tensor cores (tcgen05, bf16 hi + lo split, fp32
 * accumulators in TMEM) as a filter with a rigorous error bound, and only the candidates that
 * can reach a query's top-k are re-scored in the reference's arithmetic (float difference,
 * float product, double sum): results are identical to the plain exact kernels, which
 * DPQ_GT_TC=0 in the environment selects for everything.  base may be a host or device pointer.
 * dpq_groundtruth_stat: "tc" (1 when the filter path is on), "tc_vectors" (base vectors that went
 * through it), "tc_flagged" (query re-runs on the plain path after a candidate list overflowed),
 * "tc_filter_us" / "tc_rescore_us" (summed CUDA-event time of the two kernels). */
typedef struct dpq_gt dpq_gt;
int dpq_groundtruth_begin(const float* queries, int Q, int D, int topk, dpq_gt** out);
int dpq_groundtruth_chunk(dpq_gt* st, const float* base, int64_t n, int64_t id0);
int64_t dpq_groundtruth_stat(dpq_gt* st, const char* name);
int dpq_groundtruth_finish(dpq_gt* st, uint32_t* out_id, float* out_dist); /* frees st */

#ifdef __cplusplus
}
#endif
#endif
