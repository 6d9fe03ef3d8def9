import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import numpy as np, datagen as dg, deltapq_b200 as dpq
os.environ["DPQ_EDGE_STATS"] = "1"
M = int(sys.argv[1]); N = int(sys.argv[2])
base = dg.sift_like(N, 128, seed=1)
cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(20000, 128, seed=3), M, 256, iters=6))
codes = dpq.encode(cw, base)
t = time.time(); e, r = dpq.find_edges(codes, 256, 1, 1); print("find_edges", time.time() - t)
