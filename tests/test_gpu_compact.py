"""Compacting an open index (dpq_index_compact / dpq_multi_compact): the tree is rebuilt on the device over the live
nodes, positions are renumbered and ids kept.  Afterwards every search path returns the exact top-k over the live
nodes (plain ADC, bit-equal distances, ties by lower position), byte for byte what an index opened from
dpq.tree_build(live codes) returns, and the tree handed back is the bytes of that fresh build with vec_id mapped to
the carried ids.  The last test runs without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import datagen as dg
import deltapq_b200 as dpq
from oracle import pyoracle as po
from test_gpu_add import Model, _tree, _write_tree_files, codes_of, golden_model, open_golden
from test_gpu_delete import node_dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "deltapq_b200", "bin")
gpu = pytest.mark.gpu
WANT = ("payload", "vec_id", "qnodes", "codes_by_pos")


@pytest.fixture(scope="module")
def q130():
    return dg.sift_like(130, 128, seed=2907)


def edit(ix, model, cw, n_add, del_every, seed):
    """adds n_add codes with fresh ids, then deletes every del_every-th node by id; returns the dead mask"""
    add = codes_of(cw, n_add, seed=seed)
    ids = np.arange(10_000_000, 10_000_000 + n_add, dtype=np.uint32)
    model.add(add, ids, ix.add(add, ids))
    gone = model.ids[::del_every]
    ix.delete(gone)
    return np.isin(model.ids, gone)


def live_of(model, dead):
    return np.ascontiguousarray(model.codes[~dead]), model.ids[~dead]


def fresh_index(t, n, M, ids, opts, cw, first_pos=None):
    ix = dpq.DeltaTreeIndex(t["payload"], n, M, 256, pos2id=ids, first_pos=first_pos)
    ix.set_codebook(cw)
    for k, v in opts.items():
        ix.set_option(k, v)
    return ix


def check_tree_equals_fresh(out, fresh, live_ids, M):
    """the compacted tree's files are a fresh build's bytes, vec_id mapped to the carried ids"""
    mapped = live_ids[fresh["vec_id"]]
    assert np.array_equal(out["payload"], fresh["payload"])
    assert np.array_equal(out["vec_id"], mapped)
    assert out["n_codes"] == len(live_ids) and out["n_diffs"] == fresh["n_diffs"]
    if M == 8:
        a, b = out["qnodes"].reshape(-1, 60), fresh["qnodes"].reshape(-1, 60)
        assert np.array_equal(a[:, 4:], b[:, 4:])
        assert np.array_equal(a[:-1, :4].copy().view(np.uint32).ravel(), mapped)
    else:
        assert "qnodes" not in out
    return mapped


def same_results(a, b, queries, k):
    for u, v in zip(a.search(queries, k), b.search(queries, k)):
        assert np.array_equal(u, v)


# ------------------------------------------------------------------------------------------- every path --
@gpu
@pytest.mark.parametrize("opts,nq", [(dict(coarse=1), 130), (dict(coarse=0), 130), (dict(coarse=1, seed=0), 130),
                                     (dict(force_fallback=1), 130), (dict(coarse=1, bcap8=32), 130),
                                     (dict(latency=1), 9), (dict(coarse=1, latency=0), 9)])
def test_golden4000_every_path(golden4000, q130, opts, nq):
    g = golden4000
    ix = open_golden(g, **opts)
    model = golden_model(g)
    dead = edit(ix, model, g["cw"], 1500, 3, seed=41)
    live_codes, live_ids = live_of(model, dead)
    n_live = len(live_ids)
    out = ix.compact(want=WANT)
    fresh = dpq.tree_build(live_codes, g["cw"], want=WANT)
    mapped = check_tree_equals_fresh(out, fresh, live_ids, 8)
    assert np.array_equal(out["codes_by_pos"], fresh["codes_by_pos"])
    assert (ix.stat("n_codes"), ix.stat("n_local"), ix.stat("n_deleted"), ix.stat("n_added")) == (n_live, n_live, 0, 0)
    assert ix.stat("n_bytes") == len(out["payload"]) and ix.stat("n_diffs") == out["n_diffs"]
    assert ix.stat("last_compact_us") >= ix.stat("last_compact_build_us") > 0
    queries = q130[:nq]
    lut = dpq.adc_tables(g["cw"], queries)
    other = fresh_index(fresh, n_live, 8, mapped, opts, g["cw"])
    after = Model(fresh["codes_by_pos"], mapped)
    for k in (10, 64) if opts.get("latency") != 1 else (10,):
        pos, ids, dist = ix.search(queries, k)
        if opts.get("latency") == 1:
            assert ix.stat("last_latency") == 1
        after.check(lut, pos, ids, dist, k)
        for u, v in zip((pos, ids, dist), other.search(queries, k)):
            assert np.array_equal(u, v)
    ix.close()
    other.close()


# ------------------------------------------------------------------------------------------- files --
@gpu
def test_written_files_reopen_like_the_compacted_index(golden4000, q130, tmp_path):
    g = golden4000
    ix = open_golden(g, coarse=1)
    model = golden_model(g)
    dead = edit(ix, model, g["cw"], 800, 4, seed=42)
    n_live = int((~dead).sum())
    out = ix.compact()
    assert set(out) >= {"payload", "vec_id", "qnodes"} and "codes_by_pos" not in out
    tree_path, qnode_path = _write_tree_files(str(tmp_path), out, n_live)
    re = dpq.DeltaTreeIndex.from_file(tree_path, 8, 256, qnode_path=qnode_path)
    re.set_codebook(g["cw"])
    re.set_option("coarse", 1)
    same_results(ix, re, q130, 10)
    assert ix.compact(want=None) is None and ix.stat("n_local") == n_live  # nothing left to drop
    re.close()
    ix.close()


# ------------------------------------------------------------------------------------------- ids and state --
@gpu
def test_ids_state_and_later_edits(golden4000, q130):
    g = golden4000
    n = int(g["n"])
    lut = dpq.adc_tables(g["cw"], q130)
    # no id table: every node keeps its old position as its id
    ix = dpq.DeltaTreeIndex(g["payload"], n, 8, 256)
    ix.set_codebook(g["cw"])
    model = Model(golden_model(g).codes, np.arange(n, dtype=np.uint32))
    add = codes_of(g["cw"], 700, seed=43)
    model.add(add, None, ix.add(add))
    gone = np.arange(0, n + 700, 5, dtype=np.uint32)
    ix.delete(gone)
    dead = np.isin(model.ids, gone)
    live_codes, live_ids = live_of(model, dead)
    out = ix.compact(want=("vec_id", "codes_by_pos", "payload"))
    after = Model(out["codes_by_pos"], out["vec_id"])
    assert np.array_equal(np.sort(out["vec_id"]), live_ids)
    after.check(lut, *ix.search(q130, 10), 10)
    # delete by the carried ids, then add: positions continue after n_live, and both stay exact
    n_live = len(live_ids)
    gone2 = live_ids[::7]
    ix.delete(gone2)
    assert ix.stat("n_deleted") == len(gone2)
    more = codes_of(g["cw"], 300, seed=44)
    pos = ix.add(more, np.arange(50_000, 50_300, dtype=np.uint32))
    assert pos.min() == n_live
    after.add(more, np.arange(50_000, 50_300, dtype=np.uint32), pos)
    dead2 = np.isin(after.ids, gone2)
    for opts in (dict(coarse=1), dict(coarse=0), dict(latency=1)):
        for k, v in opts.items():
            ix.set_option(k, v)
        qs = q130[:9] if opts.get("latency") else q130
        after.check(lut, *ix.search(qs, 10), 10, dead=dead2)
    ix.close()


@gpu
def test_presample_is_regathered_after_a_compaction():
    t = _tree(30_000, 2901)
    n, R = t["n"], 2048
    for opts in (dict(coarse=1, presample=R), dict(latency=1)):
        ix = dpq.DeltaTreeIndex(t["payload"], n, 8, 256, pos2id=t["vec_id"])
        ix.set_codebook(t["cw"])
        for k, v in opts.items():
            ix.set_option(k, v)
        ix.delete(t["vec_id"][1::2])
        ix.search(t["base"][:9], 10)  # gathers the presample from the old code array
        out = ix.compact(want=("vec_id", "codes_by_pos"))
        n_live = len(out["vec_id"])
        dead = np.zeros(n_live, bool)
        dead[np.arange(R) * (n_live // R)] = True  # exactly the nodes the new presample scores
        ix.delete(out["vec_id"][dead])
        # right on top of those nodes: a stale presample would give k = 1 a cap from nodes that are not there
        queries = t["base"][out["vec_id"][dead][::37]]
        qs = queries[:9] if opts.get("latency") else queries
        lut = dpq.adc_tables(t["cw"], qs)
        model = Model(out["codes_by_pos"], out["vec_id"])
        for k in (1, 2, 10):
            model.check(lut, *ix.search(qs, k), k, dead=dead)
        ix.close()


# ------------------------------------------------------------------------------------------- shapes and handles --
@gpu
def test_wide_shape(golden_m16):
    g = golden_m16
    codes, cw = g["codes"], g["cw"]
    _, _, lay, payload = po.build_tree(codes, cw)
    n = len(codes)
    vec_id = np.asarray(lay["vec_id"], np.uint32)
    ix = dpq.DeltaTreeIndex(payload, n, 16, 256, pos2id=vec_id)
    ix.set_codebook(cw)
    ix.set_option("coarse", 1)
    model = Model(dpq.compile_program(payload, n, 16, 256)["codes"], vec_id)
    dead = edit(ix, model, cw, 2 * n + 1, 3, seed=45)
    live_codes, live_ids = live_of(model, dead)
    out = ix.compact()
    fresh = dpq.tree_build(live_codes, cw, want=WANT)
    mapped = check_tree_equals_fresh(out, fresh, live_ids, 16)
    queries = np.concatenate([g["queries"], dg.sift_like(9, 128, seed=2905)])
    other = fresh_index(fresh, len(live_ids), 16, mapped, dict(coarse=1), cw)
    Model(fresh["codes_by_pos"], mapped).check(dpq.adc_tables(cw, queries), *ix.search(queries, 100), 100)
    same_results(ix, other, queries, 100)
    ix.close()
    other.close()


@gpu
def test_forest_part_keeps_first_pos(q130):
    base = dg.sift_like(9000, 128, seed=46)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(3000, 128, seed=47), 8, 256, iters=3))
    codes = dpq.encode(cw, base)
    a, b = 2500, 9000
    t = dpq.tree_build(codes[a:b], cw, want=("payload", "vec_id", "codes_by_pos"))
    ix = dpq.DeltaTreeIndex(t["payload"], b - a, 8, 256, pos2id=t["vec_id"], first_pos=a)
    ix.set_codebook(cw)
    model = Model(t["codes_by_pos"], t["vec_id"], base_pos=a)
    dead = edit(ix, model, cw, 1500, 4, seed=48)
    live_codes, live_ids = live_of(model, dead)
    out = ix.compact()
    assert ix.stat("base_pos") == a
    fresh = dpq.tree_build(live_codes, cw, want=WANT)
    mapped = check_tree_equals_fresh(out, fresh, live_ids, 8)
    other = fresh_index(fresh, len(live_ids), 8, mapped, {}, cw, first_pos=a)
    Model(fresh["codes_by_pos"], mapped, base_pos=a).check(dpq.adc_tables(cw, q130), *ix.search(q130, 10), 10,
                                                           rows=range(0, 130, 5))
    same_results(ix, other, q130, 10)
    assert ix.add(codes_of(cw, 10, seed=49)).min() == a + len(live_ids)
    ix.close()
    other.close()


@gpu
def test_device_resident_tree_and_shards(q130):
    t = _tree(20_000, 2903)
    n, M = t["n"], 8
    codes = dpq.encode(t["cw"], t["base"])
    dcodes = dpq.DeviceBuffer(codes.nbytes).upload(codes)
    dt = dpq.DeviceTree(dcodes.ptr.value, n, M, t["cw"])
    vec_id = dt.fetch("vec_id", np.uint32)
    cbp = dt.fetch("codes_by_pos", np.uint8).reshape(-1, M)
    # a shard of two is refused and stays as it was
    sh = dt.shard(1, 2)
    sh.set_codebook(t["cw"])
    before = sh.search(q130, 10)
    with pytest.raises(dpq.DpqError, match="shard"):
        sh.compact()
    for u, v in zip(before, sh.search(q130, 10)):
        assert np.array_equal(u, v)
    sh.close()
    # the whole tree compacts
    ix = dt.shard(0, 1)
    ix.set_codebook(t["cw"])
    model = Model(cbp, vec_id)
    dead = edit(ix, model, t["cw"], 3000, 2, seed=50)
    live_codes, live_ids = live_of(model, dead)
    out = ix.compact()
    fresh = dpq.tree_build(live_codes, t["cw"], want=WANT)
    mapped = check_tree_equals_fresh(out, fresh, live_ids, 8)
    Model(fresh["codes_by_pos"], mapped).check(dpq.adc_tables(t["cw"], q130), *ix.search(q130, 10), 10,
                                               rows=range(0, 130, 7))
    ix.close()
    dt.free()
    dcodes.free()


# ------------------------------------------------------------------------------------------- errors --
@gpu
def test_errors_leave_the_index_unchanged(golden4000, q130, monkeypatch):
    g = golden4000
    n = int(g["n"])
    L = dpq.lib()

    def refused(ix, what):
        before = ix.search(q130, 10) if ix.Ds else None
        stats = [ix.stat(s) for s in ("n_local", "n_deleted", "n_added", "n_bytes")]
        assert L.dpq_index_compact(ix._h, None) == -1
        assert what in L.dpq_last_error()
        assert stats == [ix.stat(s) for s in ("n_local", "n_deleted", "n_added", "n_bytes")]
        if before is not None:
            for u, v in zip(before, ix.search(q130, 10)):
                assert np.array_equal(u, v)

    ix = dpq.DeltaTreeIndex(g["payload"], n, 8, 256, pos2id=g["vec_id"])
    ix.delete(g["vec_id"][::2])
    refused(ix, b"codebook")
    ix.set_codebook(g["cw"])
    ix.delete(g["vec_id"])
    refused(ix, b"every node is deleted")
    ix.undelete(g["vec_id"][:5])
    ix.compact(want=None)
    assert ix.stat("n_local") == 5
    ix.close()
    monkeypatch.setenv("DPQ_ENGINE", "1")
    ix = open_golden(g)
    assert ix.stat("engine") == 1
    refused(ix, b"code-array engine")
    ix.close()


# ------------------------------------------------------------------------------------------- multi-GPU handle --
@gpu
def test_multi_index_refuses_the_first_generation_engine(golden4000, q130, tmp_path, monkeypatch):
    g = golden4000
    n = int(g["n"])
    tree_path = os.path.join(str(tmp_path), "tree")
    with open(tree_path, "wb") as f:
        f.write(np.array([n, len(g["payload"])], np.int64).tobytes())
        f.write(np.asarray(g["payload"], np.uint8).tobytes())
    monkeypatch.setenv("DPQ_ENGINE", "1")
    m = dpq.MultiIndex(tree_path, 8, 256, 1)
    m.set_codebook(g["cw"])
    assert m.stat(0, "engine") == 1
    before = m.search(q130, 10)
    L = dpq.lib()
    assert L.dpq_multi_compact(m._h) == -1
    assert b"code-array engine" in L.dpq_last_error()
    assert m.stat(0, "n_local") == n
    for u, v in zip(before, m.search(q130, 10)):
        assert np.array_equal(u, v)
    m.close()


@gpu
@pytest.mark.parametrize("ng", [1, 2])
def test_multi_index_compacts_like_a_single_index(q130, tmp_path, ng):
    if dpq.device_count() < ng:
        pytest.skip("needs %d GPUs" % ng)
    t = _tree(30_000, 2904)
    n = t["n"]
    tree_path, qnode_path = _write_tree_files(str(tmp_path), t, n)
    m = dpq.MultiIndex(tree_path, 8, 256, ng, qnode_path=qnode_path)
    m.set_codebook(t["cw"])
    single = dpq.DeltaTreeIndex(t["payload"], n, 8, 256, pos2id=t["vec_id"])
    single.set_codebook(t["cw"])
    x = dg.sift_like(9000, 128, seed=51)
    ids = np.arange(n + 100, n + 9100, dtype=np.uint32)
    assert np.array_equal(m.add_vectors(x, ids), single.add_vectors(x, ids))
    gone = np.concatenate([ids[::4], t["vec_id"][::3]])
    m.delete(gone)
    single.delete(gone)
    assert m.stat(ng - 1, "n_added") == 9000
    m.compact()
    single.compact(want=None)
    assert sum(m.stat(r, "n_local") for r in range(ng)) == single.stat("n_local")
    assert all(m.stat(r, "n_added") == 0 and m.stat(r, "n_deleted") == 0 for r in range(ng))
    if ng > 1:  # the appended nodes are dealt with the tree: every GPU holds a share by stream bytes
        assert m.stat(ng - 1, "n_local") < single.stat("n_local") * 0.75
    for qs in (q130, q130[:8]):
        for u, v in zip(m.search(qs, 10), single.search(qs, 10)):
            assert np.array_equal(u, v)
    # later deletes and adds through the handle keep working on the new shards
    g2 = ids[1::9]
    m.delete(g2)
    single.delete(g2)
    more = dg.sift_like(500, 128, seed=52)
    assert np.array_equal(m.add_vectors(more, ids[:500] + 20000), single.add_vectors(more, ids[:500] + 20000))
    for u, v in zip(m.search(q130, 10), single.search(q130, 10)):
        assert np.array_equal(u, v)
    m.close()
    single.close()


@gpu
def test_multi_forest_parts_compact_in_place(q130, tmp_path):
    base = dg.sift_like(8000, 128, seed=53)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(3000, 128, seed=54), 8, 256, iters=3))
    codes = dpq.encode(cw, base)
    bounds = [0, 3000, 8000]
    L = dpq.lib()
    L.dpq_multi_open_parts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.POINTER(C.c_void_p)]
    paths, qpaths, models = [], [], []
    for p in range(2):
        t = dpq.tree_build(codes[bounds[p]: bounds[p + 1]], cw, want=("payload", "vec_id", "codes_by_pos", "qnodes"))
        tp, qp = _write_tree_files(str(tmp_path), t, bounds[p + 1] - bounds[p], tag=str(p))
        paths.append(tp.encode())
        qpaths.append(qp.encode())
        models.append(Model(t["codes_by_pos"], t["vec_id"] + bounds[p]))  # ids of part p = first_pos + vec_id
    tp_arr = (C.c_char_p * 2)(*paths)
    qp_arr = (C.c_char_p * 2)(*qpaths)
    first = np.array(bounds[:2], np.int64)
    ng = min(2, dpq.device_count())
    m = dpq.MultiIndex.__new__(dpq.MultiIndex)
    m._h = C.c_void_p()
    assert L.dpq_multi_open_parts(tp_arr, qp_arr, first.ctypes.data_as(C.c_void_p), 2, 8, 256, ng, C.byref(m._h)) == 0
    m.set_codebook(cw)
    add = codes_of(cw, 2000, seed=55)
    ids = np.arange(8000, 10000, dtype=np.uint32)
    pos = m.add(add, ids)
    models[1].add(add, ids, pos - 3000)
    gone = np.concatenate([ids[::3], np.arange(0, 8000, 5, dtype=np.uint32)])
    m.delete(gone)
    m.compact()
    live = [live_of(md, np.isin(md.ids, gone)) for md in models]
    lut = dpq.adc_tables(cw, q130)
    mp, mi, md = m.search(q130, 10)
    # each part is now a fresh tree over its live nodes, at its first_pos
    all_codes, all_ids = [], []
    for p in range(2):
        fresh = dpq.tree_build(live[p][0], cw, want=("vec_id", "codes_by_pos"))
        assert m.stat(p, "n_local") == len(live[p][1]) and m.stat(p, "base_pos") == bounds[p]
        all_codes.append(fresh["codes_by_pos"])
        all_ids.append(live[p][1][fresh["vec_id"]])
        gap = bounds[p + 1] - bounds[p] - len(live[p][1]) if p == 0 else 0
        all_codes.append(np.full((gap, 8), 0, np.uint8))
        all_ids.append(np.full(gap, 0xFFFFFFFF, np.uint32))
    codes_by_pos, ids_by_pos = np.concatenate(all_codes), np.concatenate(all_ids)
    dead = ids_by_pos == 0xFFFFFFFF  # the positions part 0 no longer holds
    for i in range(0, 130, 5):
        nd = node_dist(lut[i], codes_by_pos)
        nd[dead] = np.inf
        order = np.lexsort((np.arange(len(nd)), nd))[:10]
        assert np.array_equal(md[i], nd[order]) and np.array_equal(mp[i], order)
        assert np.array_equal(mi[i], ids_by_pos[order])
    m.close()


# ------------------------------------------------------------------------------------------- 1M codes --
@gpu
def test_1m_tree_half_deleted_tenth_added():
    t = _tree(1_000_000, 2906)
    n = t["n"]
    ix = dpq.DeltaTreeIndex(t["payload"], n, 8, 256, pos2id=t["vec_id"])
    ix.set_codebook(t["cw"])
    model = Model(t["codes_by_pos"], t["vec_id"])
    x = dg.sift_like(100_000, 128, seed=56)
    ids = np.arange(n, n + 100_000, dtype=np.uint32)
    model.add(dpq.encode(t["cw"], x), ids, ix.add_vectors(x, ids))
    gone = np.random.default_rng(57).permutation(model.ids)[: len(model.ids) // 2]
    ix.delete(gone)
    ix.compact(want=None)
    _, live_ids = live_of(model, np.isin(model.ids, gone))
    assert ix.stat("n_local") == len(live_ids)
    queries = np.concatenate([t["base"][:10] + 0.25, dg.sift_like(10, 128, seed=58)])
    pos, ids_, dist = ix.search(queries, 10)
    assert ix.stat("last_coarse") == 1 and ix.stat("last_fallback") == 0
    live_codes, live_ids = live_of(model, np.isin(model.ids, gone))
    lut = dpq.adc_tables(t["cw"], queries)
    # the oracle needs the new positions: the same order the compacted index reports, from a fresh build
    fresh = dpq.tree_build(live_codes, t["cw"], want=("vec_id", "codes_by_pos"))
    Model(fresh["codes_by_pos"], live_ids[fresh["vec_id"]]).check(lut, pos, ids_, dist, 10)
    ix.close()


# ------------------------------------------------------------------------------------------- CLI --
@gpu
def test_cli_compact_writes_files_that_answer_the_same(tmp_path):
    n, nq, M, K, k, na = 6000, 40, 8, 256, 10, 1500
    d = str(tmp_path)
    dg.make_dataset(d, n, nq, M=M, K=K, d=128, seed=59)
    common = ["-m", str(M), "-k", str(K), "-ext", "fvecs"]
    run = lambda cmd: subprocess.run(cmd, capture_output=True, text=True)  # noqa: E731
    r = run([BIN + "/pqtree", "-dataset", d, "-task", "encode", "-N", str(n)] + common)
    assert r.returncode == 0, r.stderr
    r = run([BIN + "/deltapq", "-dataset", d, "-task", "approx_tree", "-h", "1", "-diff", "8", "-N", str(n)] + common)
    assert r.returncode == 0, r.stderr
    x = dg.sift_like(na, 128, seed=60)
    dg.write_vecs(d + "/add.fvecs", x)
    del_ids = np.concatenate([np.arange(0, n, 3), np.arange(n, n + na, 7)])
    with open(d + "/ids.txt", "w") as f:
        f.write(" ".join(map(str, del_ids)) + "\n")
    n_live = n + na - len(del_ids)
    edit_args = ["-add", d + "/add.fvecs", "-deleted", d + "/ids.txt", "-compact"]
    query = [BIN + "/deltapq", "-dataset", d, "-task", "query", "-query_size", str(nq), "-topk", str(k)] + common
    r = run(query + ["-N", str(n), "-results", d + "/a.txt"] + edit_args)
    assert r.returncode == 0, r.stderr
    assert f"{n_live} live nodes, query them with -method 1 -N {n_live}" in r.stdout
    assert os.path.exists(d + f"/M{M}K{K}_Approx_TreeNodesDFS_N{n_live}")
    r = run(query + ["-N", str(n_live), "-results", d + "/b.txt"])
    assert r.returncode == 0, r.stderr
    assert open(d + "/a.txt").read() == open(d + "/b.txt").read()
    r = run(query + ["-N", str(n), "-results", d + "/c.txt"] + edit_args)  # the files exist: not overwritten
    assert r.returncode != 0 and "not overwritten" in r.stderr
    r = run(query + ["-N", str(n), "-gpus", "2"] + edit_args)  # refused before any index is opened
    assert r.returncode != 0 and "single-GPU index only" in r.stderr


# ------------------------------------------------------------------------------------------- no GPU --
def test_compact_entry_points_fail_loudly_without_gpu():
    if dpq.device_count() > 0:
        pytest.skip("a GPU is present")
    L = dpq.lib()
    assert L.dpq_index_compact(None, None) == -2
    assert b"no CUDA device" in L.dpq_last_error()
    assert L.dpq_multi_compact(None) == -2
    assert b"no CUDA device" in L.dpq_last_error()
