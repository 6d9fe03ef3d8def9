// deltapq -- drop-in for the reference's `deltapq` binary (deltapq_approx_tree_main.cpp) for the
// tasks approx_tree / query (+ query_im, batch_query: same in-memory batched semantics), same
// flags (-dataset -ext -task -m -k -h -diff -N -query_size -topk -method -debug) and the same
// files (SURVEY App. A.3-A.5).  Compute runs on the GPU through libdpq.
#include "cli_common.hpp"

#include <algorithm>
#include <thread>

using namespace cli;

static std::string base_name(const std::string& dataset, int M, int K) {
    return dataset + "/M" + std::to_string(M) + "K" + std::to_string(K);
}

static std::string nodes_file(const std::string& dataset, int M, int K, const std::string& sfx) {
    return base_name(dataset, M, K) + "_Approx_TreeNodesDFS" + sfx + (M == 8 ? "" : ".vec_id");
}
static std::string tree_file(const std::string& dataset, int M, int K, const std::string& sfx) {
    return base_name(dataset, M, K) + "_Approx_compressed_codes_opt" + sfx;
}

// the node file (QNode records at M = 8, else the position -> vec_id extension file) and the tree file with its
// 16-byte header of a tree of N nodes, under the names of suffix `sfx`
static int write_tree(const std::string& dataset, int M, int K, dpq_tree* t, long long N, const std::string& sfx) {
    const std::string f_nodes = nodes_file(dataset, M, K, sfx), f_tree = tree_file(dataset, M, K, sfx);
    if (M == 8) {  // QNode records exist for M == 8 only (DCAT.h:79-101)
        std::vector<uint8_t> qn((size_t)dpq_tree_size(t, "qnodes"));
        DPQ_TRY(dpq_tree_copy(t, "qnodes", qn.data()));
        if (!write_file(f_nodes, nullptr, 0, qn.data(), qn.size())) return die("cannot write " + f_nodes);
    } else {
        std::vector<uint32_t> v((size_t)N);
        DPQ_TRY(dpq_tree_copy(t, "vec_id", v.data()));
        if (!write_file(f_nodes, nullptr, 0, v.data(), v.size() * 4)) return die("cannot write vec_id file");
    }
    std::vector<uint8_t> payload((size_t)dpq_tree_size(t, "payload"));
    DPQ_TRY(dpq_tree_copy(t, "payload", payload.data()));
    int64_t hdr[2] = {(int64_t)N, (int64_t)payload.size()};  // DCAT.h:1840-1842
    if (!write_file(f_tree, hdr, 16, payload.data(), payload.size())) return die("cannot write " + f_tree);
    std::cout << "n_diffs " << dpq_tree_size(t, "n_diffs") << " number of bytes " << payload.size() << std::endl;
    return 0;
}

// one tree: `codes` [n][M] -> the three files of create_approx_tree (DCAT.h:970-1065) with suffix `sfx`
static int build_one(const std::string& dataset, int M, int K, int H, int method, const uint8_t* codes, long long N,
                     const Codebook& cb, const std::string& sfx) {
    const std::string f_edges = base_name(dataset, M, K) + "H" + std::to_string(H) + "_Approx_Edges" + sfx;
    dpq_tree* t = nullptr;
    if (file_exists(f_edges)) {  // stage caching by file existence (DCAT.h:1230-1242)
        std::vector<uint32_t> e((size_t)(2 * (N - 1) + 1));
        FILE* f = fopen(f_edges.c_str(), "rb");
        bool ok = f && fread(e.data(), 4, e.size(), f) == e.size();
        if (f) fclose(f);
        if (!ok) return die("stale or truncated " + f_edges);
        std::cout << "edges read from " << f_edges << std::endl;
        DPQ_TRY(dpq_tree_from_edges(codes, N, M, K, cb.cw.data(), cb.Ds, e.data() + 1, e[0], &t));
    } else {
        DPQ_TRY(dpq_tree_build(codes, N, M, K, cb.cw.data(), cb.Ds, H, method, &t));
        std::vector<uint32_t> e((size_t)(2 * (N - 1) + 1));
        e[0] = (uint32_t)dpq_tree_size(t, "root_id");
        if (N > 1) DPQ_TRY(dpq_tree_copy(t, "edges", e.data() + 1));
        if (!write_file(f_edges, nullptr, 0, e.data(), e.size() * 4)) return die("cannot write " + f_edges);
    }
    const int rc = write_tree(dataset, M, K, t, N, sfx);
    dpq_tree_free(t);
    return rc;
}

// -parts P (extension, the 1B-code layout): part p = vector ids [p*N/P, (p+1)*N/P), its own tree,
// files suffixed ".part{p}of{P}"
static std::string part_suffix(int p, int P) { return ".part" + std::to_string(p) + "of" + std::to_string(P); }
static long long part_begin(long long N, int p, int P) { return (long long)((__int128)N * p / P); }

static int approx_tree(const Args& a, const std::string& dataset, int M, int K) {
    long long N = a.num("-N", -1);
    const int H = (int)a.num("-h", 1), method = (int)a.num("-method", 1);
    const int P = (int)a.num("-parts", 1);
    // -diff is parsed but ignored like the reference (dmain:126: diff_argument = PQ_M)
    std::vector<uint8_t> codes;
    long long nn = 0;
    std::string cpath = dataset + "/codes.bin.plain.M" + std::to_string(M) + "K" + std::to_string(K) + "N" +
                        std::to_string(N);  // dmain:76-77
    if (!read_codes(cpath, M, codes, nn)) return die("cannot read " + cpath);
    if (N == -1) N = nn;
    if (N > nn) return die("-N exceeds the number of codes in " + cpath);
    if (P < 1 || P > N) return die("-parts must be between 1 and N");
    Codebook cb;
    std::string cw = base_name(dataset, M, K) + "codewords.txt";
    if (!read_codebook(cw, cb) || cb.M != M || cb.K != K) return die("cannot read codebook " + cw);
    std::cout << "M = " << M << "\nK = " << K << "\nN = " << N << "\n" << dataset << std::endl;
    const std::string sfx = method_suffix(method) + "_N" + std::to_string(N);
    double t0 = now_s();
    if (P == 1) {
        if (int rc = build_one(dataset, M, K, H, method, codes.data(), N, cb, sfx)) return rc;
    } else {
        // -gpus G: the parts are independent trees, so GPU g builds parts g, g + G, ... on its own host thread
        int G = (int)a.num("-gpus", 1);
        G = std::max(1, std::min(std::min(G, P), dpq_device_count()));
        std::vector<int> rcs((size_t)G, 0);
        auto worker = [&](int g) {
            if (dpq_set_device(g) != DPQ_OK) {
                rcs[(size_t)g] = 1;
                return;
            }
            for (int p = g; p < P && !rcs[(size_t)g]; p += G) {
                const long long b = part_begin(N, p, P), e = part_begin(N, p + 1, P);
                rcs[(size_t)g] = build_one(dataset, M, K, H, method, codes.data() + (size_t)b * M, e - b, cb, sfx + part_suffix(p, P));
            }
        };
        std::vector<std::thread> th;
        for (int g = 1; g < G; ++g) th.emplace_back(worker, g);
        worker(0);
        for (auto& t : th) t.join();
        for (int g = 0; g < G; ++g)
            if (rcs[(size_t)g]) return die("approx_tree -parts: building a part failed on GPU " + std::to_string(g));
        std::cout << P << " parts on " << G << " GPU(s)" << std::endl;
    }
    std::cout << "approx tree built in " << now_s() - t0 << " sec" << std::endl;
    return 0;
}

static int query(const Args& a, const std::string& dataset, const std::string& ext, int M, int K) {
    long long N = a.num("-N", -1);
    int query_size = (int)a.num("-query_size", -1), top_k = (int)a.num("-topk", 1);
    const int method = (int)a.num("-method", 1);
    const bool debug = a.has("-debug");
    Codebook cb;
    std::string cw = base_name(dataset, M, K) + "codewords.txt";
    if (!read_codebook(cw, cb) || cb.M != M || cb.K != K) return die("cannot read codebook " + cw);
    VecFile qf;
    if (!qf.open(dataset + "/query." + ext, ext)) return die("cannot open " + dataset + "/query." + ext);
    std::vector<float> raw;
    long long nq = qf.read(10000, raw);  // dmain:303: ReadTopN(..., 10000)
    if (query_size != -1 && query_size < nq) nq = query_size;  // dmain:306-308
    const int D = qf.D, Dp = M * cb.Ds;
    if (D > Dp) return die("query dimension exceeds M*Ds of the codebook");
    std::vector<float> q((size_t)nq * Dp, 0.f);
    for (long long i = 0; i < nq; ++i) memcpy(&q[i * Dp], &raw[i * D], (size_t)D * 4);
    const std::string sfx = method_suffix(method) + "_N" + std::to_string(N);
    const std::string f_tree = tree_file(dataset, M, K, sfx);
    const std::string f_nodes = base_name(dataset, M, K) + "_Approx_TreeNodesDFS" + sfx;
    // -gpus N (extension): the tree is sharded by depth-1 subtrees over N GPUs of this box, the
    // per-GPU top-k lists are all-gathered over NCCL and merged (dpq_multi_*, SURVEY 8e)
    const int n_gpus = (int)a.num("-gpus", 1);
    const int P = (int)a.num("-parts", 1);  // extension: the forest written by approx_tree -parts P
    const char* nodes_arg = (M == 8 && file_exists(f_nodes)) ? f_nodes.c_str() : nullptr;
    std::vector<uint32_t> pos((size_t)nq * top_k), id(pos.size());
    std::vector<float> dist(pos.size());
    const bool compact = a.has("-compact");
    if (compact && (P > 1 || n_gpus > 1)) return die("-compact works on the single-GPU index only (not with -gpus or -parts)");
    dpq_index* ix = nullptr;
    dpq_multi* mx = nullptr;
    if (P > 1) {
        if (N < P) return die("-parts needs -N >= parts");
        std::vector<std::string> tp((size_t)P), np((size_t)P);
        std::vector<const char*> tpc((size_t)P), npc((size_t)P);
        std::vector<int64_t> first((size_t)P);
        for (int p = 0; p < P; ++p) {
            tp[(size_t)p] = f_tree + part_suffix(p, P);
            np[(size_t)p] = f_nodes + part_suffix(p, P);
            tpc[(size_t)p] = tp[(size_t)p].c_str();
            npc[(size_t)p] = (M == 8 && file_exists(np[(size_t)p])) ? np[(size_t)p].c_str() : nullptr;
            first[(size_t)p] = part_begin(N, p, P);
        }
        DPQ_TRY(dpq_multi_open_parts(tpc.data(), npc.data(), first.data(), P, M, K, n_gpus, &mx));
        DPQ_TRY(dpq_multi_set_codebook(mx, cb.cw.data(), cb.Ds));
    } else if (n_gpus > 1) {
        DPQ_TRY(dpq_multi_open_file(f_tree.c_str(), nodes_arg, M, K, n_gpus, &mx));
        DPQ_TRY(dpq_multi_set_codebook(mx, cb.cw.data(), cb.Ds));
    } else {
        DPQ_TRY(dpq_index_open_file(f_tree.c_str(), nodes_arg, M, K, 0, 1, &ix));
        DPQ_TRY(dpq_index_set_codebook(ix, cb.cw.data(), cb.Ds));
    }
    const std::string added = a.str("-add", "");
    if (!added.empty()) {  // extension: vectors (-ext format) appended to the open index with ids N + i
        VecFile af;
        if (!af.open(added, ext)) return die("cannot open " + added);
        std::vector<float> xa;
        const long long na = af.read(0x7FFFFFFFLL, xa);
        if (af.D > Dp) return die("-add: vector dimension exceeds M*Ds of the codebook");
        if (N < 0 || N + na > 0xFFFFFFFFLL) return die("-add needs -N, and ids N + i below 2^32 - 1");
        std::vector<uint32_t> aid((size_t)na);
        for (long long i = 0; i < na; ++i) aid[(size_t)i] = (uint32_t)(N + i);
        if (mx) DPQ_TRY(dpq_multi_add_vectors(mx, xa.data(), na, af.D, aid.data(), nullptr));
        else DPQ_TRY(dpq_index_add_vectors(ix, xa.data(), na, af.D, aid.data(), nullptr));
    }
    const std::string deleted = a.str("-deleted", "");
    if (!deleted.empty()) {  // extension: vector ids (decimal, whitespace separated) that no query may return
        std::ifstream dfs(deleted);
        if (!dfs) return die("cannot open " + deleted);
        std::vector<uint32_t> del;
        unsigned long long v = 0;
        while (dfs >> v) {
            if (v > 0xFFFFFFFFull) return die("-deleted: id out of range in " + deleted);
            del.push_back((uint32_t)v);
        }
        if (!dfs.eof()) return die("-deleted: " + deleted + " holds something other than decimal ids");
        if (mx) DPQ_TRY(dpq_multi_delete(mx, del.data(), (int64_t)del.size()));
        else DPQ_TRY(dpq_index_delete(ix, del.data(), (int64_t)del.size()));
    }
    if (compact) {  // extension: the tree rebuilt over the live nodes, written as the files of -method 1 -N <live count>
        dpq_tree* t = nullptr;
        DPQ_TRY(dpq_index_compact(ix, &t));
        const long long n_live = dpq_tree_size(t, "n_codes");
        const std::string csfx = method_suffix(1) + "_N" + std::to_string(n_live);  // the compaction builds with -method 1
        for (const std::string& f : {nodes_file(dataset, M, K, csfx), tree_file(dataset, M, K, csfx)})
            if (file_exists(f)) {
                dpq_tree_free(t);
                return die("-compact: " + f + " exists and is not overwritten");
            }
        const int rc = write_tree(dataset, M, K, t, n_live, csfx);
        dpq_tree_free(t);
        if (rc) return rc;
        std::cout << "compacted: " << n_live << " live nodes, query them with -method 1 -N " << n_live << std::endl;
    }
    const int reps = (int)a.num("-repeat", 1);  // extension: repeat the batch (the first call pays allocations)
    double t0 = now_s();
    for (int it = 0; it < reps; ++it) {
        if (it == reps - 1) t0 = now_s();
        if (mx) DPQ_TRY(dpq_multi_search(mx, q.data(), (int)nq, top_k, pos.data(), id.data(), dist.data()));
        else DPQ_TRY(dpq_index_search(ix, q.data(), (int)nq, top_k, pos.data(), id.data(), dist.data()));
    }
    double dt = now_s() - t0;
    if (debug)  // dmain:340-343: "pos dist" of the nearest neighbour per query (+ the vector id)
        for (long long i = 0; i < nq; ++i)
            std::cout << pos[(size_t)i * top_k] << " " << dist[(size_t)i * top_k] << " id " << id[(size_t)i * top_k]
                      << std::endl;
    std::cout << dt / nq * 1000 << " [msec/query]" << std::endl;  // dmain:345
    const std::string out = a.str("-results", "");
    if (!out.empty()) {  // extension (SURVEY 8f-4): "id,dist," lines like the ground-truth file
        std::ofstream ofs(out);
        ofs << nq << "," << top_k << "\n";
        for (long long i = 0; i < nq; ++i) {
            for (int t = 0; t < top_k; ++t) ofs << id[(size_t)i * top_k + t] << "," << dist[(size_t)i * top_k + t] << ",";
            ofs << "\n";
        }
    }
    if (ix) dpq_index_close(ix);
    if (mx) dpq_multi_close(mx);
    return 0;
}

int main(int argc, char** argv) {
    Args a{argc, argv};
    std::string dataset = a.str("-dataset", ""), ext = a.str("-ext", "fvecs"), task = a.str("-task", "approx_tree");
    int M = (int)a.num("-m", 8), K = (int)a.num("-k", 256);
    if (dataset.empty()) return die("usage: deltapq -dataset DIR -task approx_tree|query|query_im|batch_query -m M -k K -h 1 -diff M -N N [-query_size Q] [-topk k] [-method 1|2] [-debug] [-results FILE] [-gpus N] [-parts P] [-repeat R] [-add FILE] [-deleted FILE] [-compact (writes the files of -method 1 -N <live count>)]");
    if (task == "approx_tree") return approx_tree(a, dataset, M, K);
    if (task == "query" || task == "query_im" || task == "batch_query") return query(a, dataset, ext, M, K);
    return die("deltapq: task '" + task + "' is outside the B200 hot-path scope (approx_tree, query, query_im, batch_query)");
}
