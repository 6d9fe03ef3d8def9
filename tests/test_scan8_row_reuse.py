"""GPU: the coarse scan with row reuse (reuse8=1, the default: a strand keeps its table rows in
registers and reads only those whose code byte changed since its previous node) gives exactly what
the scan that reads every row gives (reuse8=0).  The coarse sums are the same integers, so the
candidate counts (cand8_total) match as well as the final positions, ids and distances."""
import numpy as np
import pytest

import datagen as dg
import deltapq_b200 as dpq
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

CHUNK_NODES = 64  # nodes a strand walks per chunk (dpq_internal.h v2_chunk_nodes)


def _queries(base, n, seed, jitter):
    rng = np.random.default_rng(seed)
    q = base[rng.integers(0, len(base), n)] + rng.integers(-jitter, jitter + 1, (n, base.shape[1]))
    return np.clip(q, 0, 255).astype(np.float32)


def _both(ix, queries, k):
    """(pos, ids, dist, cand8_total, fallback) with reuse8 = 0 and with reuse8 = 1, same index."""
    out = []
    for reuse in (0, 1):
        ix.set_option("reuse8", reuse)
        pos, ids, dist = ix.search(queries, k)
        assert ix.stat("last_coarse") == 1
        out.append((pos, ids, dist, ix.stat("cand8_total"), ix.stat("last_fallback")))
    return out


def _assert_same(a, b):
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[1], b[1])
    assert np.array_equal(a[2], b[2])
    assert a[3] == b[3] and a[3] > 0  # the same coarse survivors: the sums did not change
    assert a[4] == b[4]


@pytest.mark.parametrize("opts", [dict(), dict(sample=1), dict(sample=4), dict(slices=3, warps8=24), dict(bcap8=32)],
                         ids=["default", "sample1", "sample4", "slices3_warps24", "bcap32"])
def test_narrow_reuse_matches_full_reads(golden4000, opts):
    g = golden4000
    n = int(g["n"])
    assert n % CHUNK_NODES != 0  # the last chunk is short
    ix = dpq.DeltaTreeIndex(g["payload"], n, int(g["M"]), int(g["K"]), pos2id=g["vec_id"])
    ix.set_codebook(g["cw"])
    ix.set_option("coarse", 1)
    for name, v in opts.items():
        ix.set_option(name, v)
    queries = _queries(g["queries"], 130, 23, 12)  # 130: not a multiple of the 112 queries of a CTA
    for k in (1, 10, 40):
        old, new = _both(ix, queries, k)
        _assert_same(old, new)
    if opts.get("bcap8") == 32:
        assert new[4] > 0  # overflowing candidate buffers took the exact fallback in both forms
    # and the answers are the oracle's
    for i in range(0, len(queries), 13):
        _, odist = po.scan(g["payload"], n, g["cw"], queries[i], 40)
        assert np.array_equal(new[2][i], odist)
    ix.close()


@pytest.mark.parametrize("opts", [dict(), dict(sample=2), dict(bcap8=32)], ids=["default", "sample2", "bcap32"])
def test_wide_reuse_matches_full_reads(golden_m16, opts):
    g = golden_m16
    codes, cw = g["codes"], g["cw"]
    n = len(codes)
    assert n % CHUNK_NODES != 0
    _, _, lay, payload = po.build_tree(codes, cw)
    ix = dpq.DeltaTreeIndex(payload, n, 16, 256, pos2id=lay["vec_id"])
    ix.set_codebook(cw)
    ix.set_option("coarse", 1)
    for name, v in opts.items():
        ix.set_option(name, v)
    queries = np.concatenate([g["queries"], _queries(g["queries"], 113, 5, 9)]).astype(np.float32)
    for k in (10, 100):
        old, new = _both(ix, queries, k)
        _assert_same(old, new)
    if opts.get("bcap8") == 32:
        assert new[4] > 0
    ix.close()


def test_reuse_on_a_tree_of_many_chunks():
    """30 001 codes (469 chunks, the last one 49 nodes), 1 000 queries (9 groups, the last partly
    filled): several rounds per warp and several slices, through the automatic sample pass."""
    n = 30001
    base = dg.sift_like(n, 128, seed=11)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(5000, 128, seed=12), 8, 256, iters=3))
    codes = dpq.encode(cw, base)
    tree = dpq.tree_build(codes, cw)
    ix = dpq.DeltaTreeIndex(tree["payload"], n, 8, 256, pos2id=tree["vec_id"])
    ix.set_codebook(cw)
    ix.set_option("coarse", 1)
    queries = dg.sift_like(1000, 128, seed=13)
    old, new = _both(ix, queries, 10)
    _assert_same(old, new)
    ix.close()
