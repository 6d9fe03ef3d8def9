"""A query's answer does not depend on the batch it rides in.

Every search kernel packs several queries into one table word or one shared table: scan1 (latency mode) holds
a query pair in one 32-bit word, scan2 and the first-generation engine at pack=2 hold two 15-bit entries per
word, scan8 holds four queries per word and 112 queries per CTA.  A lane or pair mapping error, or a table entry
that leaves its lane, changes ANOTHER query's answer, and a per-query comparison with the oracle run on
well-formed batches never sees it.  So, on every search path (forced by options, the path stat asserted):

  * a permuted batch gives the permuted rows, bit for bit, at batch sizes around each lane geometry;
  * a query searched alone gives the same row as inside a batch, whichever hostile query sits next to it (its
    pair partner on either side, the same 16-query lane, the same group, the next group): NaN or +-inf
    components, components so large that whole table rows overflow to inf, distance 0, the all-zero query, a
    duplicate, a query whose candidate lists overflow;
  * every row with a defined answer equals plain ADC over the codes by position: the oracle's float tables,
    each node's M entries summed in double and rounded to float, ties by lower position.

A query with a NaN or infinite component has no defined answer of its own; its call succeeds and its row
holds k entries, but the row's contents are not pinned here."""
import numpy as np
import pytest

import datagen as dg
import deltapq_b200 as dpq
from oracle import pyoracle as po
from test_gpu_delete import PAD, check, node_dist

gpu = pytest.mark.gpu
K_TOP = 10

# path -> options.  latency=0 everywhere else: a query searched alone on a tree of 4096+ nodes would otherwise
# switch to latency mode, and the solo row would come from another path than the batch.
PATHS = {
    "latency": dict(latency=1),                                   # scan1, query pairs
    "coarse": dict(coarse=1, latency=0),                          # presample-seeded coarse scan (scan8)
    "coarse_sample15": dict(coarse=1, seed=0, latency=0),         # coarse scan after the 15-bit sample pass
    "coarse_overflow": dict(coarse=1, bcap8=32, latency=0),       # candidate lists overflow -> exact fallback
    "scan15": dict(coarse=0, latency=0),                          # 15-bit scan + select (scan2)
    "gen1_pack1": dict(pack=1, latency=0),                        # first-generation engine (DPQ_ENGINE=1)
    "gen1_pack2": dict(pack=2, latency=0),
    "fallback": dict(force_fallback=1, latency=0),                # exact fallback for every query
}
CASES = [(t, p) for t in ("g4000", "t30k") for p in PATHS] + [("m16", "coarse"), ("m16", "scan15")]
# batch sizes around the lane geometry: query pairs (odd Q leaves the last pair half-empty), lut2_kernel's
# 8-query blocks, 16-query lanes, scan2's 56-query groups and scan8's 112-query CTAs
QS = (1, 2, 3, 7, 8, 9, 15, 16, 55, 56, 57, 111, 112, 113, 223, 224, 225)
QS_LATENCY = (1, 2, 3, 15, 16)
DEFINED = ("recon", "zero", "dup", "cluster")  # hostile queries whose own answer is defined


# ------------------------------------------------------------------------------------------- trees --
def _tree(n, seed, cluster=0):
    base = dg.sift_like(n, 128, seed=seed)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(20000, 128, seed=seed + 1), 8, 256, iters=4))
    codes = dpq.encode(cw, base)
    if cluster:  # a dense cluster: `cluster` copies of one code, contiguous in DFS order
        codes = np.concatenate([codes, np.repeat(codes[:1], cluster, 0)])
    t = dpq.tree_build(codes, cw, want=("payload", "vec_id", "codes_by_pos"))
    t.update(cw=cw, n=len(codes), M=8, cluster_code=codes[0] if cluster else None)
    return t


def _from_payload(payload, n, M, cw, vec_id):
    return dict(payload=payload, n=n, M=M, cw=cw, vec_id=np.asarray(vec_id, np.uint32),
                codes_by_pos=po.decode(payload, n, M)[0], cluster_code=None)


@pytest.fixture(scope="module")
def g4000(golden4000):
    g = golden4000
    return _from_payload(g["payload"], int(g["n"]), 8, g["cw"], g["vec_id"])


@pytest.fixture(scope="module")
def t30k():
    return _tree(30_000, 3901, cluster=3000)


@pytest.fixture(scope="module")
def m16(golden_m16):
    g = golden_m16
    _, _, lay, payload = po.build_tree(g["codes"], g["cw"])
    return _from_payload(payload, len(g["codes"]), 16, g["cw"], lay["vec_id"])


@pytest.fixture(scope="module")
def tree120k():
    return _tree(120_000, 3903)


# ------------------------------------------------------------------------------------------- helpers --
def open_path(t, path, monkeypatch, cw=None):
    if path.startswith("gen1"):
        monkeypatch.setenv("DPQ_ENGINE", "1")
    else:
        monkeypatch.delenv("DPQ_ENGINE", raising=False)
    ix = dpq.DeltaTreeIndex(t["payload"], t["n"], t["M"], 256, pos2id=t["vec_id"])
    ix.set_codebook(t["cw"] if cw is None else cw)
    for k, v in PATHS.get(path, {}).items():
        ix.set_option(k, v)
    assert ix.stat("engine") == (1 if path.startswith("gen1") else 2)
    return ix


def search(ix, path, queries, k=K_TOP):
    """ix.search, and proof of the path it took"""
    out = ix.search(queries, k)
    assert ix.stat("last_latency") == (1 if path == "latency" else 0)
    assert ix.stat("last_coarse") == (1 if path.startswith("coarse") else 0)
    if path == "fallback":
        assert ix.stat("last_fallback") > 0
    return out


class Reference:
    """plain ADC over the codes by position, per query (cached by the query's bytes)"""

    def __init__(self, t, cw=None):
        self.t, self.cw, self.nd = t, t["cw"] if cw is None else cw, {}
        self.dead = np.zeros(t["n"], bool)

    def dist(self, q):
        key = np.asarray(q, np.float32).tobytes()
        if key not in self.nd:
            self.nd[key] = node_dist(po.lut(self.cw, q), self.t["codes_by_pos"])
        return self.nd[key]

    def check(self, q, pos, ids, dist, k=K_TOP):
        check(pos, ids, dist, self.dist(q), self.dead, k, self.t["vec_id"])


def same_row(a, b, i, j, ctx=""):
    """row i of result a == row j of result b: positions, ids and distance bits"""
    pa, ia, da = a
    pb, ib, db = b
    assert np.array_equal(pa[i], pb[j]) and np.array_equal(ia[i], ib[j]), (ctx, i, j, pa[i], pb[j])
    assert np.array_equal(da[i].view(np.uint32), db[j].view(np.uint32)), (ctx, i, j, da[i], db[j])


def recon(cw, code):
    """the exact reconstruction of a code: distance 0 to every node that holds it"""
    return np.concatenate([cw[m, code[m]] for m in range(cw.shape[0])]).astype(np.float32)


def hostile_queries(t, victim):
    M, _, Ds = t["cw"].shape
    D = M * Ds
    base = dg.sift_like(1, D, seed=3905)[0]

    def with_(idx, v):
        q = base.copy()
        q[idx] = v
        return q

    h = {
        "nan_first": with_(0, np.nan),
        "nan_last": with_(D - 1, np.nan),
        "nan_all": np.full(D, np.nan, np.float32),
        "pinf": with_(D // 2, np.inf),
        "ninf": with_(D // 2, -np.inf),
        "huge": with_(slice(0, Ds), 3e19),  # subspace 0's table row overflows to inf
        "recon": recon(t["cw"], t["codes_by_pos"][t["n"] // 3]),
        "zero": np.zeros(D, np.float32),
        "dup": victim.copy(),
    }
    if t["cluster_code"] is not None:
        h["cluster"] = recon(t["cw"], t["cluster_code"])
    return h


def check_undefined_row(t, pos, ids):
    """a query without a defined answer: k entries, each a real position with its id, or padding"""
    real = pos != PAD
    assert np.all(pos[real] < t["n"])
    assert np.array_equal(ids[real], t["vec_id"][pos[real].astype(np.int64)])


# ------------------------------------------------------------------------------------------- 1. permutation --
@gpu
@pytest.mark.parametrize("tree,path", CASES)
def test_permuted_batch_gives_permuted_rows(request, monkeypatch, tree, path):
    t = request.getfixturevalue(tree)
    ix = open_path(t, path, monkeypatch)
    ref = Reference(t)
    rng = np.random.default_rng(3907)
    pool = dg.sift_like(225, t["M"] * t["cw"].shape[2], seed=3909)
    fallbacks = 0
    for Q in QS_LATENCY if path == "latency" else QS:
        b = pool[:Q]
        p = rng.permutation(Q)
        a = search(ix, path, b)
        fallbacks += ix.stat("last_fallback")
        ap = search(ix, path, b[p])
        for j in range(Q):
            same_row(a, ap, p[j], j, ctx=f"Q={Q}")
        for i in range(0, Q, 13):
            ref.check(b[i], a[0][i], a[1][i], a[2][i])
    if path == "coarse_overflow":
        assert fallbacks > 0
    ix.close()


# ------------------------------------------------------------------------------------------- 2-4. hostile neighbours --
@gpu
@pytest.mark.parametrize("tree,path", CASES)
def test_alone_equals_in_a_batch_with_hostile_neighbours(request, monkeypatch, tree, path):
    t = request.getfixturevalue(tree)
    ix = open_path(t, path, monkeypatch)
    ref = Reference(t)
    D = t["M"] * t["cw"].shape[2]
    victims = dg.sift_like(6, D, seed=3911)
    V = len(victims)
    solo = [search(ix, path, victims[j: j + 1]) for j in range(V)]
    for j in range(V):
        ref.check(victims[j], *(x[0] for x in solo[j]))
    # batch rows are the victims in turn; the hostile query replaces row h: row h ^ 1 is its pair partner (h even
    # and odd), rows of h's 16-query lane, of its 56- / 112-query group and of the next group are all victims
    if path == "latency":
        Qb, spots = 16, (6, 7, 15)
    else:
        Qb, spots = 232, (20, 21, 55, 111)
    batch = victims[np.arange(Qb) % V]
    base = search(ix, path, batch)
    for i in range(Qb):
        same_row(base, solo[i % V], i, 0)
    base_fallback = ix.stat("last_fallback")
    for name, hq in hostile_queries(t, victims[0]).items():
        for h in spots:
            b = batch.copy()
            b[h] = hq
            r = search(ix, path, b)
            for i in range(Qb):
                if i != h:
                    same_row(r, solo[i % V], i, 0, ctx=f"hostile {name} at row {h}")
            if name in DEFINED:
                ref.check(hq, r[0][h], r[1][h], r[2][h])
            else:
                check_undefined_row(t, r[0][h], r[1][h])
            if name == "cluster" and path in ("coarse", "coarse_sample15"):
                # its candidate lists overflow (a slice holds more than 512 nodes at distance 0): it alone goes to
                # the exact fallback
                assert ix.stat("last_fallback") > base_fallback, (name, h)
        if name in DEFINED:  # and alone
            r = search(ix, path, hq[None])
            ref.check(hq, r[0][0], r[1][0], r[2][0])
    ix.close()


# ------------------------------------------------------------------------------------------- 5. infinite distances --
@gpu
@pytest.mark.parametrize("tree,path", CASES)
def test_overflowing_distances_with_k_finite(request, monkeypatch, tree, path):
    """A few centroids of subspace 0 hold components of 1e19: the nodes that use them are at distance +inf, every
    query's table has inf entries (so every fixed-point scale is 0 and every filter passes everything)."""
    t = request.getfixturevalue(tree)
    cw = t["cw"].copy()
    used = np.unique(t["codes_by_pos"][:, 0])
    cw[0, used[:3]] = 1e19
    ix = open_path(t, path, monkeypatch, cw=cw)
    ref = Reference(t, cw)
    D = t["M"] * t["cw"].shape[2]
    queries = dg.sift_like(16 if path == "latency" else 130, D, seed=3913)
    assert np.isinf(ref.dist(queries[0])).any() and np.isfinite(ref.dist(queries[0])).sum() >= K_TOP
    batch = search(ix, path, queries)
    for i in range(len(queries)):
        ref.check(queries[i], batch[0][i], batch[1][i], batch[2][i])
    for i in range(0, len(queries), 11):
        same_row(batch, search(ix, path, queries[i: i + 1]), i, 0)
    ix.close()


# ------------------------------------------------------------------------------------------- 6. bench scale --
@gpu
def test_automatic_path_at_bench_scale(tree120k, monkeypatch):
    """10 000 SIFT-shaped queries on a 120K-node tree, no options, with 20 hostile queries mixed in"""
    t = tree120k
    ix = open_path(t, "automatic", monkeypatch)  # no options
    ref = Reference(t)
    Q = 10_000
    rng = np.random.default_rng(3915)
    queries = dg.sift_like(Q, 128, seed=3917)
    hostile = hostile_queries(t, queries[0])
    names = list(hostile) * 3
    spots = rng.choice(np.arange(1, Q), 20, replace=False)
    undefined = np.zeros(Q, bool)
    for s, name in zip(spots, names):
        queries[s] = hostile[name]
        undefined[s] = name not in DEFINED
    a = ix.search(queries, K_TOP)
    assert ix.stat("last_coarse") == 1 and ix.stat("last_latency") == 0
    p = rng.permutation(Q)
    ap = ix.search(queries[p], K_TOP)
    for j in range(Q):
        if not undefined[p[j]]:
            same_row(a, ap, p[j], j)
    victims = [0] + list(rng.choice(np.flatnonzero(~undefined), 29, replace=False))
    for i in victims + [s for s in spots if not undefined[s]]:
        ref.check(queries[i], a[0][i], a[1][i], a[2][i])
    for s in spots[undefined[spots]]:
        check_undefined_row(t, a[0][s], a[1][s])
    ix.close()
