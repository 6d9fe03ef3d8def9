"""Developer probe (NOT bench.py, not a product path): search time, coarse survivors and fallbacks with a
fraction of the tree deleted (dpq_index_delete), and the time of the delete call itself.
Usage: python tools/bench_delete.py OUT_PREFIX
Three workloads: the bench tree (1M SIFT-shaped codes, M = 8, 10K queries, top-10), the same tree at Q = 8
(latency mode), and a 1M-code M = 16 tree at top-100.  Deletion sets: uniform fractions 0 .. 99 % and 10 % as
one contiguous DFS range.  Search time = libdpq events ("last_total_us"), best of 5 after 2 warm-up calls; L2 is
not flushed between calls (the 8 MB code array of the M = 8 tree stays L2-resident, as in bench.py).  Every set
is checked against a numpy oracle (plain ADC over the codes by position, deleted nodes dropped) for 20 queries.
Writes OUT_PREFIX_<workload>.json, one record per deletion set."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

import datagen as dg
import deltapq_b200 as dpq

FRACS = [0.0, 0.01, 0.10, 0.50, 0.90, 0.99]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def node_dist(lut_q, cbp):
    d = np.zeros(len(cbp), np.float64)
    for m in range(cbp.shape[1]):
        d += lut_q[m][cbp[:, m]].astype(np.float64)
    return d.astype(np.float32)


def oracle_ok(pos, dist, lut, cbp, dead, k, rows):
    for i in rows:
        nd = node_dist(lut[i], cbp)
        live = np.flatnonzero(~dead)
        order = live[np.lexsort((live, nd[live]))][:k]
        epos = np.full(k, 0xFFFFFFFF, np.int64)
        edist = np.full(k, np.finfo(np.float32).max, np.float32)
        epos[: len(order)] = order
        edist[: len(order)] = nd[order]
        if not (np.array_equal(pos[i].astype(np.int64), epos) and np.array_equal(dist[i].view(np.uint32), edist.view(np.uint32))):
            return False
    return True


def run(name, M, n, Q, k, out_prefix):
    base = dg.sift_like(n, 128, seed=1)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(20000, 128, seed=3), M, 256, iters=6))
    queries = dg.sift_like(max(Q, 20), 128, seed=2)[:Q]
    codes = dpq.encode(cw, base)
    t = dpq.tree_build(codes, cw, want=("payload", "vec_id", "codes_by_pos", "depth"))
    cbp, vid = t["codes_by_pos"], t["vec_id"]
    lut = dpq.adc_tables(cw, queries[:20])
    ix = dpq.DeltaTreeIndex(t["payload"], n, M, 256, pos2id=vid)
    ix.set_codebook(cw)
    rng = np.random.default_rng(7)
    d1 = np.flatnonzero(t["depth"] == 1)
    sets = [("uniform_%g%%" % (100 * f), rng.random(n) < f) for f in FRACS]
    contig = np.zeros(n, bool)
    lo = int(d1[np.searchsorted(d1, n // 3)])  # from a depth-1 subtree boundary: one contiguous DFS range of 10 % of the nodes
    lo = min(lo, n - n // 10)
    contig[lo: lo + n // 10] = True
    sets.append(("contiguous_10%", contig))
    recs = []
    for label, dead in sets:
        ix.undelete(vid)
        t0 = time.perf_counter()
        ix.delete(vid[dead])
        call_ms = (time.perf_counter() - t0) * 1e3
        assert ix.stat("n_deleted") == dead.sum()
        for _ in range(2):
            ix.search(queries, k)
        best = None
        for _ in range(5):
            pos, ids, dist = ix.search(queries, k)
            tot = ix.stat("last_total_us")
            if best is None or tot < best:
                best = tot
        rec = dict(workload=name, set=label, n_deleted=int(dead.sum()), Q=Q, topk=k, search_ms=best / 1e3,
                   qps=round(Q / (best * 1e-6)), delete_call_ms=round(call_ms, 3), delete_us_stat=ix.stat("last_delete_us"),
                   survivors_per_query=(round(ix.stat("cand8_total") / Q, 1) if ix.stat("last_coarse") else "no coarse pass"),
                   last_fallback=ix.stat("last_fallback"), last_latency=ix.stat("last_latency"),
                   oracle_20_queries=oracle_ok(pos, dist, lut, cbp, dead, k, range(min(20, Q))),
                   l2_flushed=False, gpu=gpu_info())
        print(json.dumps(rec), flush=True)
        recs.append(rec)
    ix.close()
    with open(f"{out_prefix}_{name}.json", "w") as f:
        json.dump(recs, f, indent=1)


if __name__ == "__main__":
    prefix = sys.argv[1]
    run("m8_q10000_top10", 8, 1_000_000, 10_000, 10, prefix)
    run("m8_q8_top10_latency", 8, 1_000_000, 8, 10, prefix)
    run("m16_q10000_top100", 16, 1_000_000, 10_000, 100, prefix)
