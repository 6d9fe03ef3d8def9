"""Developer probe (NOT bench.py, not a product path): search time before and after dpq_index_compact, the time of
the compaction and its stages, and the search time of an index opened fresh from dpq_tree_build(live codes).
Usage: python tools/bench_compact.py OUT.json [--quick]
Workloads: the bench tree (1M SIFT-shaped codes, M = 8, seeds 1 / 2 / 3, 10K queries, top-10) and the 1M-code
M = 16 tree at top-100.  Edits: added in {0, 10, 50} % of n (SIFT-shaped vectors, seed 5, ids n + i), then deleted in
{10, 50, 90} % of all nodes, uniformly by id (seed 6).  Search time = libdpq events ("last_total_us"), best of 5
after 2 warm-up calls; L2 is not flushed between calls, as in bench.py.  Compaction time = host wall clock of the
call and its stage stats (gather, edge search, layout; the rest is the swap).  The compacted index must return
exactly what the fresh index returns (positions, ids, distance bits) for every query, and that is recorded.
--quick: 100K codes, 1K queries, one edit set per shape (a rehearsal of the script, not a measurement)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

import datagen as dg
import deltapq_b200 as dpq


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def best_search(ix, queries, k):
    for _ in range(2):
        ix.search(queries, k)
    best, res = None, None
    for _ in range(5):
        r = ix.search(queries, k)
        us = ix.stat("last_total_us")
        if best is None or us < best:
            best, res = us, r
    return best / 1e3, res


def run(M, n, Q, k, edits, gpu):
    base = dg.sift_like(n, 128, seed=1)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(20000, 128, seed=3), M, 256, iters=6))
    queries = dg.sift_like(Q, 128, seed=2)
    t = dpq.tree_build(dpq.encode(cw, base), cw, want=("payload", "vec_id", "codes_by_pos"))
    extra = dg.sift_like(n // 2, 128, seed=5)
    extra_codes = dpq.encode(cw, extra)
    recs = []
    for added, deleted in edits:
        ix = dpq.DeltaTreeIndex(t["payload"], n, M, 256, pos2id=t["vec_id"])
        ix.set_codebook(cw)
        n_add = int(n * added)
        codes = t["codes_by_pos"]
        ids = t["vec_id"]
        if n_add:
            app_ids = np.arange(n, n + n_add, dtype=np.uint32)
            pos = ix.add(extra_codes[:n_add], app_ids)
            order = np.argsort(pos)
            codes = np.concatenate([codes, extra_codes[:n_add][order]])
            ids = np.concatenate([ids, app_ids[order]])
        gone = np.random.default_rng(6).permutation(ids)[: int(len(ids) * deleted)]
        ix.delete(gone)
        before_ms, _ = best_search(ix, queries, k)
        dead = np.isin(ids, gone)
        live_codes, live_ids = np.ascontiguousarray(codes[~dead]), ids[~dead]
        ix.compact(want=None)
        st = {s: ix.stat("last_compact_" + s + "us") for s in ("", "gather_", "edge_", "layout_")}
        after_ms, after = best_search(ix, queries, k)
        fresh = dpq.tree_build(live_codes, cw, want=("payload", "vec_id"))
        fx = dpq.DeltaTreeIndex(fresh["payload"], len(live_ids), M, 256, pos2id=live_ids[fresh["vec_id"]])
        fx.set_codebook(cw)
        fresh_ms, fres = best_search(fx, queries, k)
        rec = dict(M=M, n=n, Q=Q, topk=k, added_frac=added, deleted_frac=deleted, n_live=len(live_ids),
                   search_before_ms=before_ms, compact_ms=st[""] / 1e3, gather_ms=st["gather_"] / 1e3,
                   edge_ms=st["edge_"] / 1e3, layout_ms=st["layout_"] / 1e3,
                   swap_ms=(st[""] - st["gather_"] - st["edge_"] - st["layout_"]) / 1e3, search_after_ms=after_ms,
                   search_fresh_ms=fresh_ms, fresh_tree_build_edge_ms=fresh["edge_us"] / 1e3,
                   fresh_tree_build_layout_ms=fresh["layout_us"] / 1e3,
                   equal_to_fresh=all(np.array_equal(u, v) for u, v in zip(after, fres)),
                   last_fallback=ix.stat("last_fallback"), l2_flushed=False, gpu=gpu)
        print(json.dumps(rec), flush=True)
        recs.append(rec)
        ix.close()
        fx.close()
    return recs


def main(out, quick):
    gpu = gpu_info()
    n, Q = (100_000, 1000) if quick else (1_000_000, 10_000)
    grid = [(a, d) for a in (0.0, 0.1, 0.5) for d in (0.1, 0.5, 0.9)]
    edits = [(0.1, 0.5)] if quick else grid
    recs = run(8, n, Q, 10, edits, gpu) + run(16, n, Q, 100, edits, gpu)
    with open(out, "w") as f:
        json.dump(recs, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1], "--quick" in sys.argv[2:])
