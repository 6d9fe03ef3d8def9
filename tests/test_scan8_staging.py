"""GPU: the coarse scan stages its survivors per warp and expands them into the per-(item, query)
lists when the warp's buffer could overflow and once at the end (scan8.cu, drain8).  The staging
capacity only changes how often a warp drains: a tiny buffer (stage8=32: a drain after nearly every
step that has a survivor) gives exactly what the default gives -- the same positions, ids and
distances, the same coarse survivors (cand8_total) and the same exact-fallback queries."""
import numpy as np
import pytest

import datagen as dg
import deltapq_b200 as dpq
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

TINY = 32  # the smallest capacity: one step's records (at most 28) always fit


def _queries(base, n, seed, jitter):
    rng = np.random.default_rng(seed)
    q = base[rng.integers(0, len(base), n)] + rng.integers(-jitter, jitter + 1, (n, base.shape[1]))
    return np.clip(q, 0, 255).astype(np.float32)


def _both(ix, queries, k):
    """(pos, ids, dist, cand8_total, fallback) with the default staging capacity and with TINY."""
    out = []
    for cap in (512, TINY):
        ix.set_option("stage8", cap)
        pos, ids, dist = ix.search(queries, k)
        assert ix.stat("last_coarse") == 1
        out.append((pos, ids, dist, ix.stat("cand8_total"), ix.stat("last_fallback")))
    return out


def _assert_same(a, b):
    assert np.array_equal(a[0], b[0])
    assert np.array_equal(a[1], b[1])
    assert np.array_equal(a[2], b[2])
    assert a[3] == b[3] and a[3] > 0
    assert a[4] == b[4]


def _open(payload, n, M, vec_id, cw, opts):
    ix = dpq.DeltaTreeIndex(payload, n, M, 256, pos2id=vec_id)
    ix.set_codebook(cw)
    ix.set_option("coarse", 1)
    for name, v in opts.items():
        ix.set_option(name, v)
    return ix


@pytest.mark.parametrize("opts", [dict(), dict(sample=1), dict(sample=4), dict(slices=3, warps8=24), dict(bcap8=32),
                                  dict(reuse8=0)],
                         ids=["default", "sample1", "sample4", "slices3_warps24", "bcap32", "noreuse"])
def test_narrow_tiny_staging_matches_default(golden4000, opts):
    g = golden4000
    n = int(g["n"])
    ix = _open(g["payload"], n, int(g["M"]), g["vec_id"], g["cw"], opts)
    queries = _queries(g["queries"], 130, 23, 12)  # 130: not a multiple of the 112 queries of a CTA
    for k in (1, 10, 40):
        a, b = _both(ix, queries, k)
        _assert_same(a, b)
    if opts.get("bcap8") == 32:
        assert b[4] > 0  # overflowing candidate lists took the exact fallback with either capacity
    for i in range(0, len(queries), 13):
        _, odist = po.scan(g["payload"], n, g["cw"], queries[i], 40)
        assert np.array_equal(b[2][i], odist)
    ix.close()


@pytest.mark.parametrize("opts", [dict(), dict(sample=1), dict(bcap8=32)], ids=["default", "sample1", "bcap32"])
def test_wide_tiny_staging_matches_default(golden_m16, opts):
    g = golden_m16
    codes, cw = g["codes"], g["cw"]
    n = len(codes)
    _, _, lay, payload = po.build_tree(codes, cw)
    ix = _open(payload, n, 16, lay["vec_id"], cw, opts)
    queries = np.concatenate([g["queries"], _queries(g["queries"], 113, 5, 9)]).astype(np.float32)
    for k in (10, 100):
        a, b = _both(ix, queries, k)
        _assert_same(a, b)
    if opts.get("bcap8") == 32:
        assert b[4] > 0
    ix.close()


@pytest.mark.parametrize("deleted", [False, True], ids=["live", "deleted"])
def test_narrow_tiny_staging_with_deleted_nodes(golden4000, deleted):
    """A deleted node's records are dropped by the drain: with either capacity no deleted id comes back."""
    g = golden4000
    n = int(g["n"])
    ix = _open(g["payload"], n, int(g["M"]), g["vec_id"], g["cw"], dict(sample=4))
    dead_ids = g["vec_id"][np.random.default_rng(41).random(n) < 0.3]
    if deleted:
        ix.delete(dead_ids)
    queries = _queries(g["queries"], 130, 29, 12)
    a, b = _both(ix, queries, 10)
    _assert_same(a, b)
    assert not deleted or not np.isin(b[1], dead_ids).any()
    ix.close()


def _sift_tree(n, seed):
    base = dg.sift_like(n, 128, seed=seed)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(5000, 128, seed=seed + 1), 8, 256, iters=3))
    codes = dpq.encode(cw, base)
    tree = dpq.tree_build(codes, cw)
    return tree, cw


def test_tiny_staging_on_a_tree_of_many_chunks():
    """30 001 codes (469 chunks, the last one 49 nodes), 1 000 queries (9 groups, the last partly
    filled): several rounds per warp and several slices, a deleted set on the second pass."""
    n = 30001
    tree, cw = _sift_tree(n, 11)
    ix = _open(tree["payload"], n, 8, tree["vec_id"], cw, {})
    queries = dg.sift_like(1000, 128, seed=13)
    a, b = _both(ix, queries, 10)
    _assert_same(a, b)
    ix.delete(tree["vec_id"][np.random.default_rng(5).random(n) < 0.1])
    a, b = _both(ix, queries, 10)
    _assert_same(a, b)
    ix.close()


def test_tiny_staging_on_the_bench_shape():
    """1M codes, M = 8, 10 000 queries, top-10: the shape of the benchmark."""
    n = 1_000_000
    tree, cw = _sift_tree(n, 903)
    ix = _open(tree["payload"], n, 8, tree["vec_id"], cw, {})
    queries = dg.sift_like(10000, 128, seed=904)
    a, b = _both(ix, queries, 10)
    _assert_same(a, b)
    ix.close()
