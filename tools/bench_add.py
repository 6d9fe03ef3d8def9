"""Developer probe (NOT bench.py, not a product path): searches over a tree with appended nodes
(dpq_index_add_vectors), and the throughput of the add calls themselves.
Usage: python tools/bench_add.py OUT.json
Workload: the bench tree (bench.py's data: 1M SIFT-shaped codes, M = 8, seeds 1 / 2 / 3), 10K queries, top-10, with
0 %, 1 %, 10 % and 50 % of n appended as SIFT-shaped vectors (seed 5), laid out sorted by code word
(add_order 1, the default) or in input order (add_order 0); the two orders alternate, twice each.  Search time =
libdpq events ("last_total_us" for the step, "last_scan8_us" for the full coarse pass), best of 5 after 2 warm-up
calls; L2 is not flushed between calls, as in bench.py.  Every search is checked against a numpy oracle (plain
ADC over the codes by position, appended codes included) for 20 queries.  The appended segment's table-row reuse
is counted on the CPU with tools/row_reuse_stats.py's counter, over the layout the library reported (out_pos).
Add throughput: dpq_index_add (host codes) and dpq_index_add_vectors (host floats) of 10^3, 10^5 and 10^6 rows
into a freshly opened index, host wall clock of the call (it ends in a stream sync), best of 3."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np

import datagen as dg
import deltapq_b200 as dpq
from row_reuse_stats import row_stats

N, Q, K = 1_000_000, 10_000, 10
FRACS = [0.0, 0.01, 0.10, 0.50]


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def node_dist(lut_q, cbp):
    d = np.zeros(len(cbp), np.float64)
    for m in range(cbp.shape[1]):
        d += lut_q[m][cbp[:, m]].astype(np.float64)
    return d.astype(np.float32)


def oracle_ok(pos, dist, lut, cbp, k, rows):
    for i in rows:
        nd = node_dist(lut[i], cbp)
        order = np.lexsort((np.arange(len(nd)), nd))[:k]
        if not (np.array_equal(pos[i].astype(np.int64), order) and np.array_equal(dist[i], nd[order])):
            return False
    return True


def main(out):
    base = dg.sift_like(N, 128, seed=1)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(20000, 128, seed=3), 8, 256, iters=6))
    queries = dg.sift_like(Q, 128, seed=2)
    extra = dg.sift_like(N // 2, 128, seed=5)
    extra_codes = dpq.encode(cw, extra)
    t = dpq.tree_build(dpq.encode(cw, base), cw, want=("payload", "vec_id", "codes_by_pos"))
    lut = dpq.adc_tables(cw, queries[:20])
    gpu = gpu_info()
    tree_rows = row_stats(t["codes_by_pos"])

    def open_ix(order):
        ix = dpq.DeltaTreeIndex(t["payload"], N, 8, 256, pos2id=t["vec_id"])
        ix.set_codebook(cw)
        ix.set_option("add_order", order)
        return ix

    recs = []
    for rnd in range(2):
        for frac in FRACS:
            for order in (1, 0):
                if frac == 0 and order == 0:
                    continue  # nothing appended: the same index
                ix = open_ix(order)
                n_add = int(N * frac)
                app = np.zeros((0, 8), np.uint8)
                if n_add:
                    pos = ix.add_vectors(extra[:n_add])
                    app = extra_codes[:n_add][np.argsort(pos)]
                for _ in range(2):
                    ix.search(queries, K)
                best = None
                for _ in range(5):
                    p, _, d = ix.search(queries, K)
                    tot, s8 = ix.stat("last_total_us"), ix.stat("last_scan8_us")
                    if best is None or tot < best[0]:
                        best = (tot, s8)
                rec = dict(round=rnd, added_frac=frac, n_added=n_add, add_order=order, Q=Q, topk=K, search_ms=best[0] / 1e3,
                           scan8_ms=best[1] / 1e3, qps=round(Q / (best[0] * 1e-6)), last_coarse=ix.stat("last_coarse"),
                           last_sample_stride=ix.stat("last_sample_stride"),
                           survivors_per_query=round(ix.stat("cand8_total") / Q, 1), last_fallback=ix.stat("last_fallback"),
                           oracle_20_queries=oracle_ok(p, d, lut, np.concatenate([t["codes_by_pos"], app]), K, range(20)),
                           appended_rows_per_node=(round(row_stats(app)["rows_per_node"], 3) if n_add else None),
                           tree_rows_per_node=round(tree_rows["rows_per_node"], 3), l2_flushed=False, gpu=gpu)
                print(json.dumps(rec), flush=True)
                recs.append(rec)
                ix.close()
    codes_all = np.concatenate([extra_codes, extra_codes])
    x_all = np.concatenate([extra, extra])
    for rows in (1000, 100_000, 1_000_000):
        for what in ("add", "add_vectors"):
            best = None
            for _ in range(3):
                ix = open_ix(1)
                t0 = time.perf_counter()
                if what == "add":
                    ix.add(codes_all[:rows])
                else:
                    ix.add_vectors(x_all[:rows])
                dt = time.perf_counter() - t0
                us = ix.stat("last_add_us")
                ix.close()
                if best is None or dt < best[0]:
                    best = (dt, us)
            rec = dict(throughput=what, rows=rows, call_ms=round(best[0] * 1e3, 3), last_add_us=best[1],
                       rows_per_s=round(rows / best[0]), gpu=gpu)
            print(json.dumps(rec), flush=True)
            recs.append(rec)
    with open(out, "w") as f:
        json.dump(recs, f, indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
