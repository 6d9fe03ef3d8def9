"""Deleting vectors from an open index (dpq_index_delete / dpq_multi_delete): every search path returns the
exact top-k over the LIVE nodes -- ascending distance, ties by lower position, the same distance bits -- padded
with (0xFFFFFFFF, FLT_MAX) when fewer than k nodes are live.  The oracle is the per-node distance (the oracle
scan, or plain ADC over the codes by position: float table entries summed in double) with the deleted nodes
dropped.  The last test runs without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import datagen as dg
import deltapq_b200 as dpq
from helpers import assert_topk_equal
from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "deltapq_b200", "bin")
PAD = 0xFFFFFFFF
gpu = pytest.mark.gpu


def node_dist(lut_q, codes_by_pos):
    """distance of every node (by position) for one query: float(double sum of its M float table entries)"""
    d = np.zeros(len(codes_by_pos), np.float64)
    for m in range(codes_by_pos.shape[1]):
        d += lut_q[m][codes_by_pos[:, m]].astype(np.float64)
    return d.astype(np.float32)


def expected(nd, dead, k, base_pos=0):
    """top-k over live nodes by (distance, position); positions are base_pos + local index"""
    live = np.flatnonzero(~dead)
    order = live[np.lexsort((live, nd[live]))][:k]
    pos = np.full(k, PAD, np.int64)
    dist = np.full(k, np.finfo(np.float32).max, np.float32)
    pos[: len(order)] = order + base_pos
    dist[: len(order)] = nd[order]
    return pos, dist


def check(pos, ids, dist, nd, dead, k, vec_id=None, base_pos=0):
    """one query: bit-equal distances, the same positions, no deleted node, ids by the table"""
    epos, edist = expected(nd, dead, k, base_pos)
    assert np.array_equal(dist.view(np.uint32), edist.view(np.uint32)), (dist, edist)
    real = epos != PAD
    if real.any():
        assert_topk_equal(pos[real] - base_pos, dist[real], epos[real] - base_pos, edist[real], node_dist=nd)
    assert np.array_equal(pos.astype(np.int64), epos)
    assert not dead[(pos[real] - base_pos).astype(np.int64)].any()
    if vec_id is not None and ids is not None:
        assert np.array_equal(ids[real], vec_id[(pos[real] - base_pos).astype(np.int64)])
        assert np.all(ids[~real] == PAD)


def random_dead(n, frac, seed):
    return np.random.default_rng(seed).random(n) < frac


def open_golden(g, **opts):
    ix = dpq.DeltaTreeIndex(g["payload"], int(g["n"]), int(g["M"]), int(g["K"]), pos2id=g["vec_id"])
    ix.set_codebook(g["cw"])
    for k, v in opts.items():
        ix.set_option(k, v)
    return ix


def golden_node_dist(g, queries):
    n = int(g["n"])
    return [po.scan(g["payload"], n, g["cw"], q, 1, want_node_dist=True)[2] for q in queries]


@pytest.fixture(scope="module")
def q130():
    return dg.sift_like(130, 128, seed=907)


@pytest.fixture(scope="module")
def tree120k():
    return _tree(120_000, 901)


@pytest.fixture(scope="module")
def tree1m():
    return _tree(1_000_000, 903)


def _tree(n, seed):
    base = dg.sift_like(n, 128, seed=seed)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(20000, 128, seed=seed + 1), 8, 256, iters=4))
    codes = dpq.encode(cw, base)
    t = dpq.tree_build(codes, cw, want=("payload", "vec_id", "codes_by_pos", "depth", "qnodes"))
    t["cw"], t["n"] = cw, n
    return t


def open_tree(t, **opts):
    ix = dpq.DeltaTreeIndex(t["payload"], t["n"], 8, 256, pos2id=t["vec_id"])
    ix.set_codebook(t["cw"])
    for k, v in opts.items():
        ix.set_option(k, v)
    return ix


# ------------------------------------------------------------------------------------------- every path --
@gpu
@pytest.mark.parametrize("opts,nq", [(dict(coarse=1), 130), (dict(coarse=0), 130), (dict(coarse=1, seed=0), 130),
                                     (dict(force_fallback=1), 130), (dict(coarse=1, bcap8=32), 130),
                                     (dict(latency=1), 9), (dict(coarse=1, latency=0), 9)])
def test_golden4000_every_path(golden4000, q130, opts, nq):
    g = golden4000
    queries = q130[:nq]
    nd = golden_node_dist(g, queries)
    dead = random_dead(int(g["n"]), 0.3, 11)
    ix = open_golden(g, **opts)
    ix.delete(g["vec_id"][dead])
    assert ix.stat("n_deleted") == dead.sum()
    for k in (10, 64) if opts.get("latency") != 1 else (10,):
        pos, ids, dist = ix.search(queries, k)
        if opts.get("latency") == 1:
            assert ix.stat("last_latency") == 1
        for i in range(nq):
            check(pos[i], ids[i], dist[i], nd[i], dead, k, g["vec_id"])
    if opts.get("bcap8") == 32:
        assert ix.stat("last_fallback") > 0  # overflowed lists went to the exact fallback, which skips dead nodes too
    ix.close()


@gpu
@pytest.mark.parametrize("opts", [dict(coarse=1), dict(coarse=1, refine=4), dict(coarse=0), dict(coarse=1, bcap8=32)])
@pytest.mark.parametrize("k", [10, 100])
def test_wide_shape(golden_m16, opts, k):
    g = golden_m16
    codes, cw = g["codes"], g["cw"]
    _, _, lay, payload = po.build_tree(codes, cw)
    n = len(codes)
    queries = np.concatenate([g["queries"], dg.sift_like(9, 128, seed=905)])
    nd = [po.scan(payload, n, cw, q, 1, want_node_dist=True)[2] for q in queries]
    vec_id = np.asarray(lay["vec_id"], np.uint32)
    dead = random_dead(n, 0.3, 12)
    ix = dpq.DeltaTreeIndex(payload, n, 16, 256, pos2id=vec_id)
    ix.set_codebook(cw)
    for kk, v in opts.items():
        ix.set_option(kk, v)
    ix.delete(vec_id[dead])
    pos, ids, dist = ix.search(queries, k)
    if opts.get("refine"):
        assert ix.stat("last_refine_stride") == 4
    for i in range(len(queries)):
        check(pos[i], ids[i], dist[i], nd[i], dead, k, vec_id)
    ix.close()


@gpu
@pytest.mark.parametrize("which", ["tree120k", "tree1m"])
def test_automatic_paths_on_larger_trees(request, which):
    t = request.getfixturevalue(which)
    n = t["n"]
    queries = dg.sift_like(150, 128, seed=909)
    lut = dpq.adc_tables(t["cw"], queries)
    dead = random_dead(n, 0.3, 13)
    ix = open_tree(t)
    ix.delete(t["vec_id"][dead])
    pos, ids, dist = ix.search(queries, 10)
    assert ix.stat("last_coarse") == 1
    for i in range(0, 150, 8):
        check(pos[i], ids[i], dist[i], node_dist(lut[i], t["codes_by_pos"]), dead, 10, t["vec_id"])
    for lat in (-1, 1):  # latency mode, automatic and forced
        ix.set_option("latency", lat)
        pos, ids, dist = ix.search(queries[:8], 10)
        assert ix.stat("last_latency") == 1
        for i in range(8):
            check(pos[i], ids[i], dist[i], node_dist(lut[i], t["codes_by_pos"]), dead, 10, t["vec_id"])
    ix.close()


@gpu
@pytest.mark.parametrize("R", [2, 3])
def test_shard_split_merges_to_whole(golden4000, q130, R):
    g = golden4000
    n, k, Q = int(g["n"]), 10, 130
    dead = random_dead(n, 0.3, 14)
    ids_del = g["vec_id"][dead]
    whole = open_golden(g)
    whole.delete(ids_del)
    wpos, _, wdist = whole.search(q130, k)
    dq = dpq.DeviceBuffer(q130.nbytes).upload(q130)
    dk = dpq.DeviceBuffer(R * Q * k * 8)
    do = dpq.DeviceBuffer(Q * k * 8)
    shards = []
    for r in range(R):
        ix = dpq.DeltaTreeIndex(g["payload"], n, 8, 256, pos2id=g["vec_id"], rank=r, n_ranks=R)
        ix.set_codebook(g["cw"])
        ix.delete(ids_del)  # the same list: each shard keeps the ids it holds
        base = ix.stat("base_pos")
        assert ix.stat("n_deleted") == dead[base: base + ix.stat("n_local")].sum()
        ix.search_device(dq.ptr, Q, k, dk.ptr.value + r * Q * k * 8)
        ix.sync()
        shards.append(ix)
    assert sum(s.stat("n_deleted") for s in shards) == dead.sum()
    shards[0].merge_device(dk.ptr, R, Q, k, do.ptr)
    shards[0].sync()
    pos, dist = dpq.unpack_keys(do.download(np.uint64, (Q, k)))
    assert np.array_equal(dist, wdist) and np.array_equal(pos, wpos)
    for s in shards + [whole]:
        s.close()
    for b in (dq, dk, do):
        b.free()


@gpu
def test_forest_part(q130):
    base = dg.sift_like(9000, 128, seed=21)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(3000, 128, seed=22), 8, 256, iters=3))
    codes = dpq.encode(cw, base)
    a, b = 2500, 9000
    t = dpq.tree_build(codes[a:b], cw, want=("payload", "vec_id", "codes_by_pos"))
    ix = dpq.DeltaTreeIndex(t["payload"], b - a, 8, 256, pos2id=t["vec_id"], first_pos=a)
    ix.set_codebook(cw)
    dead = random_dead(b - a, 0.3, 15)
    ix.delete(t["vec_id"][dead])  # a part's ids are its own vec_ids
    assert ix.stat("n_deleted") == dead.sum()
    lut = dpq.adc_tables(cw, q130)
    pos, ids, dist = ix.search(q130, 10)
    for i in range(0, 130, 5):
        check(pos[i], ids[i], dist[i], node_dist(lut[i], t["codes_by_pos"]), dead, 10, t["vec_id"], base_pos=a)
    ix.close()


@gpu
def test_device_resident_tree_shards(q130):
    n, M = 30000, 8
    base = dg.sift_like(n, 128, seed=61)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(3000, 128, seed=62), M, 256, iters=3))
    codes = dpq.encode(cw, base)
    dcodes = dpq.DeviceBuffer(codes.nbytes).upload(codes)
    dt = dpq.DeviceTree(dcodes.ptr.value, n, M, cw)
    vec_id = dt.fetch("vec_id", np.uint32)
    cbp = dt.fetch("codes_by_pos", np.uint8).reshape(-1, M)
    dead = random_dead(n, 0.3, 16)
    lut = dpq.adc_tables(cw, q130)
    for r in range(3):
        ix = dt.shard(r, 3)
        ix.set_codebook(cw)
        ix.delete(vec_id[dead])
        lo, nl = ix.stat("base_pos"), ix.stat("n_local")
        pos, ids, dist = ix.search(q130, 10)
        for i in range(0, 130, 7):
            nd = node_dist(lut[i], cbp[lo: lo + nl])
            check(pos[i], ids[i], dist[i], nd, dead[lo: lo + nl], 10, vec_id[lo: lo + nl], base_pos=lo)
        ix.close()
    dt.free()
    dcodes.free()


@gpu
def test_two_level_sample_on_a_large_shard_half_deleted():
    n, M, K, Q, k = 20_000_000, 8, 256, 300, 10
    rng = np.random.default_rng(5)
    codes = rng.integers(0, K, size=(n, M), dtype=np.uint8)
    cw = dg.roundtrip_codebook((rng.random((M, K, 16)) * 120).astype(np.float32))
    queries = (rng.random((Q, 128)) * 120).astype(np.float32)
    dcodes = dpq.DeviceBuffer(codes.nbytes).upload(codes)
    dt = dpq.DeviceTree(dcodes.ptr.value, n, M, cw)
    vec_id = dt.fetch("vec_id", np.uint32)
    ix = dt.shard(0, 1)
    ix.set_codebook(cw)
    dead_ids = np.flatnonzero(rng.random(n) < 0.5).astype(np.uint32)  # vector ids = rows of `codes`
    ix.delete(dead_ids)
    assert ix.stat("n_deleted") == len(dead_ids)
    pos, ids, dist = ix.search(queries, k)
    assert ix.stat("last_coarse") == 1 and ix.stat("last_refine_stride") == 64
    dead_row = np.zeros(n, bool)
    dead_row[dead_ids] = True
    lut = dpq.adc_tables(cw, queries[:3])
    for i in range(3):  # plain ADC over the codes by vector id
        d32 = node_dist(lut[i], codes)
        d32[dead_row] = np.inf
        best = np.sort(d32, kind="stable")[:k]
        assert np.array_equal(dist[i], best)
        assert np.array_equal(d32[ids[i]], dist[i])
        assert not dead_row[ids[i]].any()
    assert np.array_equal(vec_id[pos[:3].astype(np.int64)], ids[:3])
    ix.close()
    dt.free()
    dcodes.free()


# ------------------------------------------------------------------------------------------- attacks on the caps --
@gpu
@pytest.mark.parametrize("R", [2048, 4096])
def test_delete_exactly_the_presample(tree120k, q130, R):
    t = tree120k
    n = t["n"]
    dead = np.zeros(n, bool)
    dead[np.arange(R) * (n // R)] = True  # the nodes the presample scores
    ix = open_tree(t, presample=R)
    ix.delete(t["vec_id"][dead])
    lut = dpq.adc_tables(t["cw"], q130)
    for k, nq in ((10, 130), (10, 8), (50, 130)):
        pos, ids, dist = ix.search(q130[:nq], k)
        for i in range(0, nq, 9):
            check(pos[i], ids[i], dist[i], node_dist(lut[i], t["codes_by_pos"]), dead, k, t["vec_id"])
    ix.close()


@gpu
def test_delete_each_querys_true_top50(tree120k, q130):
    t = tree120k
    lut = dpq.adc_tables(t["cw"], q130)
    ix = open_tree(t)
    for i in (0, 33, 77, 129):
        nd = node_dist(lut[i], t["codes_by_pos"])
        order = np.lexsort((np.arange(t["n"]), nd))
        dead = np.zeros(t["n"], bool)
        dead[order[:50]] = True
        ix.delete(t["vec_id"][dead])
        for qs in (q130, q130[i: i + 1]):  # batched and latency mode
            pos, ids, dist = ix.search(qs, 10)
            row = i if len(qs) > 1 else 0
            assert np.array_equal(pos[row].astype(np.int64), order[50:60])
            check(pos[row], ids[row], dist[row], nd, dead, 10, t["vec_id"])
        ix.undelete(t["vec_id"][dead])
        assert ix.stat("n_deleted") == 0
    ix.close()


@gpu
def test_delete_a_whole_depth1_subtree_and_the_root(tree120k, q130):
    t = tree120k
    n = t["n"]
    d1 = np.flatnonzero(t["depth"] == 1)
    ends = np.append(d1[1:], n)
    j = int(np.argmax(ends - d1))  # the largest depth-1 subtree: a contiguous DFS range
    lut = dpq.adc_tables(t["cw"], q130)
    for rng_ in ((d1[j], ends[j]), (0, 1)):
        dead = np.zeros(n, bool)
        dead[rng_[0]: rng_[1]] = True
        for opts in (dict(), dict(coarse=0), dict(latency=1)):
            ix = open_tree(t, **opts)
            ix.delete(t["vec_id"][dead])
            nq = 8 if opts.get("latency") else 130
            pos, ids, dist = ix.search(q130[:nq], 10)
            for i in range(0, nq, 6):
                check(pos[i], ids[i], dist[i], node_dist(lut[i], t["codes_by_pos"]), dead, 10, t["vec_id"])
            ix.close()


@gpu
@pytest.mark.parametrize("opts", [dict(), dict(coarse=1), dict(coarse=0), dict(latency=1), dict(force_fallback=1)])
def test_all_but_five_and_everything(golden4000, q130, opts):
    g = golden4000
    n = int(g["n"])
    queries = q130[:9]
    nd = golden_node_dist(g, queries)
    ix = open_golden(g, **opts)
    dead = np.ones(n, bool)
    dead[[0, 17, 1999, 2500, n - 1]] = False
    ix.delete(g["vec_id"][dead])
    pos, ids, dist = ix.search(queries, 10)
    for i in range(len(queries)):
        check(pos[i], ids[i], dist[i], nd[i], dead, 10, g["vec_id"])
        assert np.all(pos[i][5:] == PAD) and np.all(dist[i][5:] == np.finfo(np.float32).max)
    ix.delete(g["vec_id"])
    assert ix.stat("n_deleted") == n
    pos, ids, dist = ix.search(queries, 10)
    assert np.all(pos == PAD) and np.all(ids == PAD) and np.all(dist == np.finfo(np.float32).max)
    ix.close()


# ------------------------------------------------------------------------------------------- bookkeeping --
@gpu
def test_undelete_restores_the_index_exactly(tree120k, q130):
    t = tree120k
    fresh = open_tree(t)
    ix = open_tree(t)
    dead = random_dead(t["n"], 0.3, 17)
    for qs in (q130, q130[:8]):
        a = fresh.search(qs, 10)
        ref = (fresh.stat("cand8_total"), fresh.stat("last_fallback"))
        ix.delete(t["vec_id"][dead])
        ix.search(qs, 10)
        ix.undelete(t["vec_id"][dead])
        assert ix.stat("n_deleted") == 0
        b = ix.search(qs, 10)
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
        assert (ix.stat("cand8_total"), ix.stat("last_fallback")) == ref
    fresh.close()
    ix.close()


@gpu
def test_repeated_cumulative_absent_and_persistent(golden4000, q130):
    g = golden4000
    n = int(g["n"])
    vid = g["vec_id"]
    nd = golden_node_dist(g, q130[:20])
    ix = open_golden(g, coarse=1)
    A, B = random_dead(n, 0.2, 18), random_dead(n, 0.2, 19)
    ix.delete([])
    assert ix.stat("n_deleted") == 0
    ix.delete(vid[A])
    ix.delete(vid[A])  # twice: harmless
    assert ix.stat("n_deleted") == A.sum()
    ix.delete(np.concatenate([vid[B], np.arange(n, n + 500, dtype=np.uint32)]))  # absent ids are ignored
    both = A | B
    assert ix.stat("n_deleted") == both.sum()
    ix.set_codebook(g["cw"])   # deletions survive a new codebook ...
    ix.set_option("coarse", 0)  # ... and options
    for opts in ((), (("coarse", 1),)):
        for kv in opts:
            ix.set_option(*kv)
        pos, ids, dist = ix.search(q130[:20], 10)
        for i in range(20):
            check(pos[i], ids[i], dist[i], nd[i], both, 10, vid)
    ix.undelete(vid[A])  # clears A's bits, B's stay
    assert ix.stat("n_deleted") == (B & ~A).sum()
    pos, ids, dist = ix.search(q130[:20], 10)
    for i in range(20):
        check(pos[i], ids[i], dist[i], nd[i], B & ~A, 10, vid)
    ix.close()


@gpu
def test_bad_arguments_and_first_generation_engine(golden4000, monkeypatch):
    g = golden4000
    ix = open_golden(g)
    L = dpq.lib()
    assert L.dpq_index_delete(ix._h, None, 3) == -1
    assert L.dpq_index_undelete(ix._h, None, 3) == -1
    assert L.dpq_index_delete(ix._h, None, 0) == 0
    ix.close()
    monkeypatch.setenv("DPQ_ENGINE", "1")
    ix = open_golden(g)
    assert ix.stat("engine") == 1
    ids = np.arange(5, dtype=np.uint32)
    assert L.dpq_index_delete(ix._h, ids.ctypes.data_as(C.c_void_p), 5) == -1
    assert b"code-array engine" in L.dpq_last_error()
    ix.close()


# ------------------------------------------------------------------------------------------- multi-GPU --
def _write_tree_files(d, t, n):
    tree_path, qnode_path = os.path.join(d, "tree"), os.path.join(d, "qnodes")
    with open(tree_path, "wb") as f:
        f.write(np.array([n, len(t["payload"])], np.int64).tobytes())
        f.write(t["payload"].tobytes())
    t["qnodes"].tofile(qnode_path)
    return tree_path, qnode_path


@gpu
def test_multi_index_deletes_like_a_single_index(tree120k, q130, tmp_path):
    t = tree120k
    n = t["n"]
    tree_path, qnode_path = _write_tree_files(str(tmp_path), t, n)
    ng = min(2, dpq.device_count())
    m = dpq.MultiIndex(tree_path, 8, 256, ng, qnode_path=qnode_path)
    m.set_codebook(t["cw"])
    single = open_tree(t)
    dead = random_dead(n, 0.3, 20)
    del_ids = t["vec_id"][dead]
    m.delete(del_ids)
    single.delete(del_ids)
    assert sum(m.stat(r, "n_deleted") for r in range(ng)) == dead.sum()
    for qs in (q130, q130[:8]):
        mpos, mids, mdist = m.search(qs, 10)
        spos, sids, sdist = single.search(qs, 10)
        assert np.array_equal(mpos, spos) and np.array_equal(mids, sids) and np.array_equal(mdist, sdist)
        assert not np.isin(mids, del_ids).any()
    m.undelete(del_ids)
    assert sum(m.stat(r, "n_deleted") for r in range(ng)) == 0
    m.close()
    single.close()


# ------------------------------------------------------------------------------------------- CLI --
@gpu
@pytest.mark.parametrize("parts", [1, 2])
def test_cli_query_with_deleted_ids(tmp_path, parts):
    n, nq, M, K, k = 6000, 40, 8, 256, 10
    d = str(tmp_path)
    dg.make_dataset(d, n, nq, M=M, K=K, d=128, seed=37)
    common = ["-m", str(M), "-k", str(K), "-N", str(n), "-ext", "fvecs"]
    run = lambda cmd: subprocess.run(cmd, capture_output=True, text=True)
    r = run([BIN + "/pqtree", "-dataset", d, "-task", "encode"] + common)
    assert r.returncode == 0, r.stderr
    extra = ["-parts", str(parts)] if parts > 1 else []
    r = run([BIN + "/deltapq", "-dataset", d, "-task", "approx_tree", "-h", "1", "-diff", "8"] + common + extra)
    assert r.returncode == 0, r.stderr
    del_ids = np.flatnonzero(random_dead(n, 0.3, 21))
    with open(d + "/ids.txt", "w") as f:
        f.write(" ".join(map(str, del_ids[: len(del_ids) // 2])) + "\n")
        f.write("\n".join(map(str, del_ids[len(del_ids) // 2:])) + "\n")
    r = run([BIN + "/deltapq", "-dataset", d, "-task", "query", "-query_size", str(nq), "-topk", str(k), "-deleted",
             d + "/ids.txt", "-results", d + "/out.txt"] + common + extra)
    assert r.returncode == 0, r.stderr
    lines = open(d + "/out.txt").read().splitlines()
    assert lines[0] == f"{nq},{k}"
    got = [np.array(ln.rstrip(",").split(","), np.float64).reshape(-1, 2) for ln in lines[1:]]
    ids = np.array([g[:, 0] for g in got], np.int64)
    dist = np.array([g[:, 1] for g in got])
    assert not np.isin(ids, del_ids).any()
    # the library's answer: plain ADC over the vector ids' codes, deleted ids dropped
    cw = dg.read_codebook(d + f"/M{M}K{K}codewords.txt")
    codes = dg.read_codes(d + f"/codes.bin.plain.M{M}K{K}N{n}", M)
    queries = dg.read_vecs(d + "/query.fvecs")[:nq]
    lut = dpq.adc_tables(cw, queries)
    dead = np.zeros(n, bool)
    dead[del_ids] = True
    for i in range(nq):
        nd = node_dist(lut[i], codes)
        _, edist = expected(nd, dead, k)
        np.testing.assert_allclose(dist[i], edist, rtol=1e-5)
        np.testing.assert_allclose(nd[ids[i]], edist, rtol=1e-5)
    r = run([BIN + "/deltapq", "-dataset", d, "-task", "query", "-query_size", "2", "-deleted", d + "/nope.txt"]
            + common + extra)
    assert r.returncode != 0 and "nope.txt" in r.stderr


# ------------------------------------------------------------------------------------------- no GPU --
def test_delete_entry_points_fail_loudly_without_gpu():
    if dpq.device_count() > 0:
        pytest.skip("a GPU is present")
    L = dpq.lib()
    ids = np.arange(3, dtype=np.uint32)
    for name in ("dpq_index_delete", "dpq_index_undelete", "dpq_multi_delete", "dpq_multi_undelete"):
        assert getattr(L, name)(None, ids.ctypes.data_as(C.c_void_p), 3) == -2, name
        assert b"no CUDA device" in L.dpq_last_error(), name
