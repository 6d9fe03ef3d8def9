"""Table rows the coarse scan (scan8.cu) reads per node, counted on the CPU from a tree's DFS codes.

A strand walks `chunk_nodes` consecutive positions and keeps its table rows in registers: at a chunk
start it reads all NF rows (NF = 8 narrow, 16 wide), then only the rows whose code byte differs from
the previous node.  Past the last node of a short chunk the code word is 0 (one read of the rows that
differ from it, then none).  Without reuse (reuse8=0) every step reads NF rows.  A pass with batch
stride S walks the chunks of every S-th batch of four (the sample passes).

Predicted shared-memory wavefronts per (node, 112-query group), narrow shape: each row a strand reads
is one 128-byte wavefront; round 2 measured 8.69 per (node, group) for 8 rows, of which 8.06 were the
rows (bank conflicts: x 8.06 / 8) and 0.63 the code-word delivery and candidate appends
(profiles/r2_summary.md).  Wide shape: a 64-bit row read of one strand is half a wavefront; two
strands of a half warp share one when their rows do not conflict, so the count lies between the
half-warp requests (no conflicts) and the strand rows (every pair conflicts).

Usage:
  python tools/row_reuse_stats.py --sift 1000000 [--m 8] [--stride 1 8]   # bench tree (CPU oracle build)
  python tools/row_reuse_stats.py --golden sift_n4000_m8 [--stride 1 4]
"""
import argparse
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np

from oracle import pyoracle as po

SPW = 4  # strands (chunks in flight) per warp
R2_ROW_FACTOR, R2_OTHER = 8.06 / 8, 8.69 - 8.06  # narrow shape, round 2 capture


def dfs_codes_sift(n, M):
    """The bench tree: bench.py's synthetic data (seeds 1 / 2 / 3), built by the CPU oracle."""
    import datagen as dg
    base = dg.sift_like(n, 128, seed=1)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(20000, 128, seed=3), M, 256, iters=6))
    t = time.time()
    codes = po.encode(cw, base)
    _, _, _, payload = po.build_tree(codes, cw)
    print(f"oracle tree: {n} codes, M={M}, {len(payload)} stream bytes, {time.time() - t:.1f} s", flush=True)
    return po.decode(payload, n, M)[0]


def dfs_codes_golden(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    n = int(z["n"]) if "n" in z.files else len(z["codes"])
    if "payload" in z.files:
        M = int(z["M"])
        return po.decode(z["payload"], n, M)[0]
    codes, cw = z["codes"], z["cw"]
    return po.decode(po.build_tree(codes, cw)[3], len(codes), codes.shape[1])[0]


def row_stats(codes, chunk_nodes=64, stride=1):
    n, M = codes.shape
    NF = 8 if M <= 8 else 16
    C = chunk_nodes
    n_chunks = (n + C - 1) // C
    words = np.zeros((n_chunks * C, NF), np.uint8)  # padded code words; 0 past the last node
    words[:n, :M] = codes
    chg = np.ones_like(words, dtype=bool)
    chg[1:] = words[1:] != words[:-1]
    chg[::C] = True  # chunk start: all rows
    chg = chg.reshape(n_chunks, C, NF)
    walked = (np.arange(n_chunks) // SPW) % stride == 0
    real = np.minimum(C, n - np.arange(n_chunks) * C)
    nodes = int(real[walked].sum())
    reads = int(chg[walked].sum())
    full = int(walked.sum()) * C * NF
    out = dict(nodes=nodes, chunks=int(walked.sum()), nf=NF, rows_per_node=reads / nodes, rows_per_node_full=full / nodes,
               rows_equal_to_previous=1.0 - reads / full)
    if NF == 8:
        out["pred_wavefronts_per_node_group"] = reads / nodes * R2_ROW_FACTOR + R2_OTHER
        out["pred_wavefronts_per_node_group_full"] = full / nodes * R2_ROW_FACTOR + R2_OTHER
    else:
        # half-warp requests: strands (0, 1) and (2, 3) of a batch step together; pad to whole batches
        n_b = (n_chunks + SPW - 1) // SPW
        pad = np.zeros((n_b * SPW, C, NF), bool)
        pad[:n_chunks] = chg
        pair = pad.reshape(n_b, 2, 2, C, NF).any(axis=2)  # [batch][pair][step][row]
        wb = (np.arange(n_b) % stride) == 0
        out["halfwarp_requests_per_node"] = float(pair[wb].sum()) / nodes
        out["halfwarp_requests_per_node_full"] = float(wb.sum()) * 2 * C * NF / nodes
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    src = ap.add_mutually_exclusive_group(required=True)
    src.add_argument("--sift", type=int, metavar="N", help="bench-shaped synthetic tree of N codes")
    src.add_argument("--golden", metavar="NAME", help="tests/golden/NAME.npz")
    ap.add_argument("--m", type=int, default=8, help="subspaces of the --sift tree (8 narrow, 16 wide)")
    ap.add_argument("--chunk-nodes", type=int, default=64)
    ap.add_argument("--stride", type=int, nargs="+", default=[1], help="batch strides to count (1 = the full pass)")
    args = ap.parse_args()
    codes = dfs_codes_sift(args.sift, args.m) if args.sift else dfs_codes_golden(args.golden)
    for s in args.stride:
        st = row_stats(codes, args.chunk_nodes, s)
        print(f"stride {s}: " + ", ".join(f"{k} {v:.4g}" if isinstance(v, float) else f"{k} {v}" for k, v in st.items()))


if __name__ == "__main__":
    main()
