"""Adding vectors to an open index (dpq_index_add / dpq_multi_add): appended nodes take the positions after the
index's range and every search path returns the exact top-k over tree and appended nodes together -- ascending
distance, ties by lower position, the same distance bits.  The oracle is plain ADC over the codes by position
(the tree's, then the appended codes in position order): float table entries summed in double.  The last test
runs without a GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import datagen as dg
import deltapq_b200 as dpq
from oracle import pyoracle as po
from test_gpu_delete import check, node_dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "deltapq_b200", "bin")
gpu = pytest.mark.gpu


class Model:
    """codes and ids by local position of one index, appended nodes included"""

    def __init__(self, codes_by_pos, vec_id, base_pos=0):
        self.codes = np.asarray(codes_by_pos, np.uint8)
        self.ids = np.asarray(vec_id, np.uint32)
        self.base = base_pos

    def add(self, codes, ids, pos):
        n0, n = len(self.codes), len(codes)
        pos = np.asarray(pos, np.int64)
        assert np.array_equal(np.sort(pos), self.base + n0 + np.arange(n))  # contiguous, after the range
        order = np.argsort(pos)
        self.codes = np.concatenate([self.codes, np.asarray(codes, np.uint8)[order]])
        self.ids = np.concatenate([self.ids, (pos if ids is None else np.asarray(ids))[order].astype(np.uint32)])

    def check(self, lut, pos, ids, dist, k, dead=None, rows=None):
        dead = np.zeros(len(self.codes), bool) if dead is None else dead
        for i in rows if rows is not None else range(len(pos)):
            check(pos[i], ids[i], dist[i], node_dist(lut[i], self.codes), dead, k, self.ids, base_pos=self.base)


def codes_of(cw, n, seed):
    return dpq.encode(cw, dg.sift_like(n, cw.shape[0] * cw.shape[2], seed=seed))


def golden_model(g):
    return Model(dpq.compile_program(g["payload"], int(g["n"]), int(g["M"]), int(g["K"]))["codes"], g["vec_id"])


def open_golden(g, **opts):
    ix = dpq.DeltaTreeIndex(g["payload"], int(g["n"]), int(g["M"]), int(g["K"]), pos2id=g["vec_id"])
    ix.set_codebook(g["cw"])
    for k, v in opts.items():
        ix.set_option(k, v)
    return ix


@pytest.fixture(scope="module")
def q130():
    return dg.sift_like(130, 128, seed=1907)


def _tree(n, seed):
    base = dg.sift_like(n, 128, seed=seed)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(20000, 128, seed=seed + 1), 8, 256, iters=4))
    codes = dpq.encode(cw, base)
    t = dpq.tree_build(codes, cw, want=("payload", "vec_id", "codes_by_pos", "qnodes"))
    t["cw"], t["n"], t["base"] = cw, n, base
    return t


def open_tree(t, **opts):
    ix = dpq.DeltaTreeIndex(t["payload"], t["n"], 8, 256, pos2id=t["vec_id"])
    ix.set_codebook(t["cw"])
    for k, v in opts.items():
        ix.set_option(k, v)
    return ix


@pytest.fixture(scope="module")
def tree30k():
    return _tree(30_000, 1901)


# ------------------------------------------------------------------------------------------- every path --
@gpu
@pytest.mark.parametrize("opts,nq", [(dict(coarse=1), 130), (dict(coarse=0), 130), (dict(coarse=1, seed=0), 130),
                                     (dict(force_fallback=1), 130), (dict(coarse=1, bcap8=32), 130),
                                     (dict(latency=1), 9), (dict(coarse=1, latency=0), 9)])
@pytest.mark.parametrize("frac", [0.1, 1.0, 3.0])
def test_golden4000_every_path(golden4000, q130, opts, nq, frac):
    g = golden4000
    n = int(g["n"])
    ix = open_golden(g, **opts)
    model = golden_model(g)
    add = codes_of(g["cw"], int(n * frac), seed=11)
    ids = np.arange(n, n + len(add), dtype=np.uint32)
    model.add(add, ids, ix.add(add, ids))
    assert ix.stat("n_added") == len(add) and ix.stat("n_local") == n + len(add) and ix.stat("n_codes") == n
    queries = q130[:nq]
    lut = dpq.adc_tables(g["cw"], queries)
    for k in (10, 64) if opts.get("latency") != 1 else (10,):
        pos, ids_, dist = ix.search(queries, k)
        if opts.get("latency") == 1:
            assert ix.stat("last_latency") == 1
        model.check(lut, pos, ids_, dist, k)
    ix.close()


@gpu
@pytest.mark.parametrize("k", [10, 100])
def test_wide_shape(golden_m16, k):
    g = golden_m16
    codes, cw = g["codes"], g["cw"]
    _, _, lay, payload = po.build_tree(codes, cw)
    n = len(codes)
    vec_id = np.asarray(lay["vec_id"], np.uint32)
    ix = dpq.DeltaTreeIndex(payload, n, 16, 256, pos2id=vec_id)
    ix.set_codebook(cw)
    ix.set_option("coarse", 1)
    ix.set_option("refine", 4)
    model = Model(dpq.compile_program(payload, n, 16, 256)["codes"], vec_id)
    add = codes_of(cw, 2 * n + 1, seed=12)
    model.add(add, None, ix.add(add))  # no ids: the table grows with the positions
    queries = np.concatenate([g["queries"], dg.sift_like(9, 128, seed=1905)])
    pos, ids, dist = ix.search(queries, k)
    assert ix.stat("last_refine_stride") == 4
    model.check(dpq.adc_tables(cw, queries), pos, ids, dist, k)
    ix.close()


# ------------------------------------------------------------------------------------------- layout --
@gpu
def test_one_call_equals_sixty_calls_and_input_order(golden4000, q130):
    g = golden4000
    n = int(g["n"])
    rng = np.random.default_rng(3)
    sizes = [1, 63, 64, 65, 2, 127, 129, 3] + [int(v) for v in rng.integers(1, 90, size=52)]  # chunk ends
    sizes[-1] += (n + sum(sizes) + 1) % 2  # an odd n_local: the last code word pair is half padding
    add = codes_of(g["cw"], int(sum(sizes)), seed=13)
    ids = np.arange(10**6, 10**6 + len(add), dtype=np.uint32)
    lut = dpq.adc_tables(g["cw"], q130)
    one, many, plain = open_golden(g), open_golden(g), open_golden(g, add_order=0)
    m_one, m_many, m_plain = golden_model(g), golden_model(g), golden_model(g)
    p_one = one.add(add, ids)
    m_one.add(add, ids, p_one)
    p_plain = plain.add(add, ids)
    assert np.array_equal(p_plain, n + np.arange(len(add)))  # input order
    m_plain.add(add, ids, p_plain)
    s = 0
    for c in sizes:
        m_many.add(add[s: s + c], ids[s: s + c], many.add(add[s: s + c], ids[s: s + c]))
        s += c
    assert many.stat("n_local") % 2 == 1
    for opts in (dict(coarse=1), dict(coarse=0), dict(latency=1)):
        nq = 9 if opts.get("latency") else 130
        res = {}
        for name, ix, m in (("one", one, m_one), ("many", many, m_many), ("plain", plain, m_plain)):
            for kk, v in opts.items():
                ix.set_option(kk, v)
            res[name] = ix.search(q130[:nq], 10)
            m.check(lut, *res[name], 10)
        for name in ("many", "plain"):
            assert np.array_equal(res[name][2].view(np.uint32), res["one"][2].view(np.uint32))
        # the same input rows: map the sorted index's appended positions to rows, then to input-order positions
        row_of = np.full(n + len(add), -1, np.int64)
        row_of[p_one.astype(np.int64)] = np.arange(len(add))
        pos1 = res["one"][0].astype(np.int64)
        app = pos1 >= n
        mapped = pos1.copy()
        mapped[app] = p_plain[row_of[pos1[app]]]
        for i in range(nq):
            nd_plain = node_dist(lut[i], m_plain.codes)
            assert np.array_equal(nd_plain[mapped[i]], res["one"][2][i])
    for ix in (one, many, plain):
        ix.close()


@gpu
def test_ties_and_exact_match(golden4000):
    g = golden4000
    n = int(g["n"])
    ix = open_golden(g, coarse=1)
    model = golden_model(g)
    cw = g["cw"]
    twin = model.codes[[17, 2500]]  # equal to tree codes
    rng = np.random.default_rng(4)
    while True:
        fresh = rng.integers(0, 256, size=(1, 8), dtype=np.uint8)
        if not (model.codes == fresh).all(axis=1).any():
            break
    add = np.concatenate([twin, fresh])
    model.add(add, None, ix.add(add))
    recon = lambda c: np.concatenate([cw[m, c[m]] for m in range(8)])[None, :]  # noqa: E731
    for row, c in enumerate(add):
        q = recon(c)
        lut = dpq.adc_tables(cw, q)
        for opts in (dict(coarse=1), dict(coarse=0), dict(latency=1)):
            for kk, v in opts.items():
                ix.set_option(kk, v)
            pos, ids, dist = ix.search(q, 10)
            model.check(lut, pos, ids, dist, 10)
            hits = np.flatnonzero((model.codes == c).all(axis=1))  # the tree's twin, then the appended node
            assert len(hits) == (2 if row < 2 else 1) and hits[-1] >= n
            assert np.array_equal(pos[0][: len(hits)], hits)  # equal distances: lower position first
    ix.close()


@gpu
@pytest.mark.parametrize("which", ["golden4000", "golden_m16"])
def test_batch_is_laid_out_sorted_by_code(request, which):
    g = request.getfixturevalue(which)
    M = int(g["M"])
    if which == "golden_m16":
        payload = po.build_tree(g["codes"], g["cw"])[3]
        ix = dpq.DeltaTreeIndex(payload, int(g["n"]), M, 256)
    else:
        ix = open_golden(g)
    add = codes_of(g["cw"], 3000, seed=33)
    add = np.concatenate([add, add[::7], add[5::11]])  # equal codes: ties keep input-row order
    add[::13, M - 1] = add[::13, 0]  # vary the last subspaces too (the wide shape's low word)
    add[::17, :] = add[::17, ::-1]
    pos = ix.add(add)
    rows = np.arange(len(add))
    expect = np.lexsort((rows,) + tuple(add[:, m] for m in reversed(range(M))))  # subspace 0 most significant
    assert np.array_equal(np.argsort(pos), expect)
    ix.set_option("add_order", 0)
    pos0 = ix.add(add)
    assert np.array_equal(pos0, pos.max() + 1 + rows)
    ix.close()


# ------------------------------------------------------------------------------------------- presample --
@gpu
def test_presample_is_regathered_after_an_add(tree30k):
    t = tree30k
    n = t["n"]
    R = 2048
    dead = np.zeros(n, bool)
    dead[np.arange(R) * (n // R)] = True  # exactly the nodes the presample scores before the add
    # right on top of deleted nodes: a stale presample (old nodes, dead bits tested at the new stride) would count
    # them live and give k = 1 a cap of ~0 that drops the true nearest live node
    queries = t["base"][t["vec_id"][dead][::37]]
    for opts in (dict(coarse=1, presample=R), dict(latency=1)):
        ix = open_tree(t, **opts)
        model = Model(t["codes_by_pos"], t["vec_id"])
        ix.delete(t["vec_id"][dead])
        ix.search(queries, 10)  # gathers the presample at the old stride
        add = codes_of(t["cw"], n, seed=14)
        model.add(add, None, ix.add(add))  # the stride doubles
        full_dead = np.concatenate([dead, np.zeros(n, bool)])
        qs = queries[:9] if opts.get("latency") else queries
        lut = dpq.adc_tables(t["cw"], qs)
        for k in (1, 2, 10):
            pos, ids, dist = ix.search(qs, k)
            model.check(lut, pos, ids, dist, k, dead=full_dead)
        ix.close()


# ------------------------------------------------------------------------------------------- delete --
@gpu
def test_interaction_with_delete(golden4000, q130):
    g = golden4000
    n = int(g["n"])
    queries = q130[:40]
    lut = dpq.adc_tables(g["cw"], queries)
    for opts in (dict(coarse=1), dict(coarse=0), dict(latency=1)):
        ix = open_golden(g, **opts)
        model = golden_model(g)
        qs, lq = (queries[:9], lut[:9]) if opts.get("latency") else (queries, lut)
        ix.delete([777777])  # not present yet
        add = codes_of(g["cw"], 3000, seed=15)
        ids = np.arange(777000, 780000, dtype=np.uint32)  # holds 777777: deleted before it was added, live now
        model.add(add, ids, ix.add(add, ids))
        assert ix.stat("n_deleted") == 0
        dead = np.zeros(len(model.codes), bool)
        model.check(lq, *ix.search(qs, 10), 10, dead=dead)
        gone = ids[::3]
        ix.delete(gone)
        dead = np.isin(model.ids, gone)
        assert ix.stat("n_deleted") == len(gone)
        model.check(lq, *ix.search(qs, 10), 10, dead=dead)
        ix.undelete(gone[::2])
        dead = np.isin(model.ids, gone[1::2])
        model.check(lq, *ix.search(qs, 10), 10, dead=dead)
        ix.delete(g["vec_id"])  # every tree node: only appended nodes remain
        dead |= np.arange(len(model.codes)) < n
        pos, ids_, dist = ix.search(qs, 10)
        model.check(lq, pos, ids_, dist, 10, dead=dead)
        assert (pos >= n).all()
        more = codes_of(g["cw"], 100, seed=16)  # the bitmap grows: new nodes are live
        model.add(more, None, ix.add(more))
        dead = np.concatenate([dead, np.zeros(100, bool)])
        model.check(lq, *ix.search(qs, 10), 10, dead=dead)
        ix.close()


# ------------------------------------------------------------------------------------------- encoder --
@gpu
@pytest.mark.parametrize("tc", ["1", "0"])
def test_add_vectors_encodes_like_dpq_encode(golden4000, q130, monkeypatch, tc):
    monkeypatch.setenv("DPQ_ENCODE_TC", tc)
    g = golden4000
    x = dg.sift_like(5000, 128, seed=17)
    codes = dpq.encode(g["cw"], x)
    assert dpq.encode_stat("tc") == (tc == "1")
    a, b = open_golden(g, add_order=0), open_golden(g, add_order=0)
    pa = a.add_vectors(x)
    pb = b.add(codes)
    assert np.array_equal(pa, pb)
    lut = dpq.adc_tables(g["cw"], q130)
    model = golden_model(g)
    model.add(codes, None, pa)
    for ix in (a, b):
        ix.set_option("coarse", 1)
    ra, rb = a.search(q130, 64), b.search(q130, 64)
    for u, v in zip(ra, rb):
        assert np.array_equal(u, v)
    model.check(lut, *ra, 64)
    # sorted layout: the order is a function of the codes alone
    c = open_golden(g)
    assert np.array_equal(c.add_vectors(x), open_golden(g).add(codes))
    c.close()
    a.close()
    b.close()


@gpu
def test_device_pointers(golden4000, q130):
    g = golden4000
    L = dpq.lib()
    x = dg.sift_like(3000, 128, seed=18)
    codes = dpq.encode(g["cw"], x)
    ids = np.arange(50000, 53000, dtype=np.uint32)
    dx = dpq.DeviceBuffer(x.nbytes).upload(x)
    dc = dpq.DeviceBuffer(codes.nbytes).upload(codes)
    di = dpq.DeviceBuffer(ids.nbytes).upload(ids)
    dp = dpq.DeviceBuffer(ids.nbytes)
    host = open_golden(g)
    ref = host.add(codes, ids)
    for fn, buf, extra in ((L.dpq_index_add, dc, ()), (L.dpq_index_add_vectors, dx, (128,))):
        ix = open_golden(g)
        assert fn(ix._h, buf.ptr, 3000, *extra, di.ptr, dp.ptr) == 0
        assert np.array_equal(dp.download(np.uint32, 3000), ref)
        for u, v in zip(ix.search(q130, 10), host.search(q130, 10)):
            assert np.array_equal(u, v)
        ix.close()
    host.close()
    for b in (dx, dc, di, dp):
        b.free()


# ------------------------------------------------------------------------------------------- shards --
@gpu
def test_shards_only_the_last_accepts(golden4000, q130):
    g = golden4000
    n, Q, k, R = int(g["n"]), 130, 10, 3
    add = codes_of(g["cw"], 900, seed=19)
    ids = np.arange(n, n + 900, dtype=np.uint32)
    whole = open_golden(g)
    wp = whole.add(add, ids)
    wpos, wids, wdist = whole.search(q130, k)
    dq = dpq.DeviceBuffer(q130.nbytes).upload(q130)
    dk = dpq.DeviceBuffer(R * Q * k * 8)
    do = dpq.DeviceBuffer(Q * k * 8)
    shards = []
    for r in range(R):
        ix = dpq.DeltaTreeIndex(g["payload"], n, 8, 256, pos2id=g["vec_id"], rank=r, n_ranks=R)
        ix.set_codebook(g["cw"])
        if r < R - 1:
            with pytest.raises(dpq.DpqError, match="last shard"):
                ix.add(add, ids)
            assert ix.stat("n_added") == 0
        else:
            assert np.array_equal(ix.add(add, ids), wp)
        ix.search_device(dq.ptr, Q, k, dk.ptr.value + r * Q * k * 8)
        ix.sync()
        shards.append(ix)
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
    model = Model(t["codes_by_pos"], t["vec_id"], base_pos=a)
    add = codes_of(cw, 1500, seed=23)
    pos_ = ix.add(add)
    assert pos_.min() == b
    model.add(add, None, pos_)
    lut = dpq.adc_tables(cw, q130)
    model.check(lut, *ix.search(q130, 10), 10, rows=range(0, 130, 5))
    ix.close()


@gpu
def test_device_resident_tree_shards(tree30k, q130):
    t = tree30k
    n, M = t["n"], 8
    codes = dpq.encode(t["cw"], t["base"])
    dcodes = dpq.DeviceBuffer(codes.nbytes).upload(codes)
    dt = dpq.DeviceTree(dcodes.ptr.value, n, M, t["cw"])
    vec_id = dt.fetch("vec_id", np.uint32)
    cbp = dt.fetch("codes_by_pos", np.uint8).reshape(-1, M)
    lut = dpq.adc_tables(t["cw"], q130)
    add = codes_of(t["cw"], 5000, seed=24)
    for r in range(3):
        ix = dt.shard(r, 3)
        ix.set_codebook(t["cw"])
        if r < 2:
            assert dpq.lib().dpq_index_add(ix._h, add.ctypes.data_as(C.c_void_p), 10, None, None) == -1
            ix.close()
            continue
        lo, nl = ix.stat("base_pos"), ix.stat("n_local")
        assert lo + nl == n
        model = Model(cbp[lo:], vec_id[lo:], base_pos=lo)
        ids = np.arange(n, n + 5000, dtype=np.uint32)
        model.add(add, ids, ix.add(add, ids))
        model.check(lut, *ix.search(q130, 10), 10, rows=range(0, 130, 7))
        ix.close()
    dt.free()
    dcodes.free()


def _write_tree_files(d, t, n, tag=""):
    tree_path, qnode_path = os.path.join(d, "tree" + tag), os.path.join(d, "qnodes" + tag)
    with open(tree_path, "wb") as f:
        f.write(np.array([n, len(t["payload"])], np.int64).tobytes())
        f.write(t["payload"].tobytes())
    t["qnodes"].tofile(qnode_path)
    return tree_path, qnode_path


@gpu
@pytest.mark.parametrize("ng", [1, 2])
def test_multi_index_adds_like_a_single_index(tree30k, q130, tmp_path, ng):
    if dpq.device_count() < ng:
        pytest.skip("needs %d GPUs" % ng)
    t = tree30k
    n = t["n"]
    tree_path, qnode_path = _write_tree_files(str(tmp_path), t, n)
    m = dpq.MultiIndex(tree_path, 8, 256, ng, qnode_path=qnode_path)
    m.set_codebook(t["cw"])
    single = open_tree(t)
    x = dg.sift_like(4000, 128, seed=25)
    ids = np.arange(n + 100, n + 4100, dtype=np.uint32)
    assert np.array_equal(m.add_vectors(x, ids), single.add_vectors(x, ids))
    assert np.array_equal(m.add(dpq.encode(t["cw"], x[:70])), single.add(dpq.encode(t["cw"], x[:70])))
    assert m.stat(ng - 1, "n_added") == 4070
    # device input on GPU 0, while the index that takes the adds lives on GPU ng - 1: copied across first
    dpq.set_device(0)
    x2 = dg.sift_like(500, 128, seed=35)
    dx = dpq.DeviceBuffer(x2.nbytes).upload(x2)
    dc = dpq.DeviceBuffer(x2.shape[0] * 8).upload(dpq.encode(t["cw"], x2))
    dp = dpq.DeviceBuffer(x2.shape[0] * 4)
    L = dpq.lib()
    assert L.dpq_multi_add_vectors(m._h, dx.ptr, 500, 128, None, dp.ptr) == 0, L.dpq_last_error()
    assert np.array_equal(dp.download(np.uint32, 500), single.add_vectors(x2))
    assert L.dpq_multi_add(m._h, dc.ptr, 500, None, dp.ptr) == 0, L.dpq_last_error()
    assert np.array_equal(dp.download(np.uint32, 500), single.add(dpq.encode(t["cw"], x2)))
    for b in (dx, dc, dp):
        b.free()
    for step in ("added", "deleted"):
        if step == "deleted":
            gone = np.concatenate([ids[::4], t["vec_id"][::5]])
            m.delete(gone)
            single.delete(gone)
        for qs in (q130, q130[:8]):
            for u, v in zip(m.search(qs, 10), single.search(qs, 10)):
                assert np.array_equal(u, v)
    m.close()
    single.close()


@gpu
def test_multi_forest_parts_add_to_the_last_part(q130, tmp_path):
    base = dg.sift_like(8000, 128, seed=26)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(dg.sift_like(3000, 128, seed=27), 8, 256, iters=3))
    codes = dpq.encode(cw, base)
    bounds = [0, 3000, 8000]
    L = dpq.lib()
    L.dpq_multi_open_parts.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.POINTER(C.c_void_p)]
    paths, qpaths, cbp = [], [], []
    for p in range(2):
        t = dpq.tree_build(codes[bounds[p]: bounds[p + 1]], cw, want=("payload", "vec_id", "codes_by_pos", "qnodes"))
        tp, qp = _write_tree_files(str(tmp_path), t, bounds[p + 1] - bounds[p], tag=str(p))
        paths.append(tp.encode())
        qpaths.append(qp.encode())
        cbp.append(t["codes_by_pos"])
    tp_arr = (C.c_char_p * 2)(*paths)
    qp_arr = (C.c_char_p * 2)(*qpaths)
    first = np.array(bounds[:2], np.int64)
    m = dpq.MultiIndex.__new__(dpq.MultiIndex)
    m._h = C.c_void_p()
    assert L.dpq_multi_open_parts(tp_arr, qp_arr, first.ctypes.data_as(C.c_void_p), 2, 8, 256, 1, C.byref(m._h)) == 0
    m.set_codebook(cw)
    add = codes_of(cw, 2000, seed=28)
    ids = np.arange(8000, 10000, dtype=np.uint32)
    pos = m.add(add, ids)
    assert pos.min() == 8000 and m.stat(1, "n_added") == 2000 and m.stat(0, "n_added") == 0
    all_codes = np.concatenate(cbp + [add[np.argsort(pos)]])
    app_ids = ids[np.argsort(pos)]
    lut = dpq.adc_tables(cw, q130)
    mp, mi, md = m.search(q130, 10)
    for i in range(0, 130, 5):
        nd = node_dist(lut[i], all_codes)
        order = np.lexsort((np.arange(len(nd)), nd))[:10]
        assert np.array_equal(md[i], nd[order]) and np.array_equal(mp[i], order)
    sel = mp >= 8000  # the added ids, through the handle's id table
    assert sel.any() and np.array_equal(mi[sel], app_ids[mp[sel].astype(np.int64) - 8000])
    m.close()


# ------------------------------------------------------------------------------------------- 1M codes --
@gpu
def test_1m_tree_with_1_and_10_percent_added():
    t = _tree(1_000_000, 1903)
    n = t["n"]
    queries = dg.sift_like(150, 128, seed=1909)
    lut = dpq.adc_tables(t["cw"], queries)
    ix = open_tree(t)
    model = Model(t["codes_by_pos"], t["vec_id"])
    for total, seed in ((10_000, 29), (100_000, 30)):
        x = dg.sift_like(total - ix.stat("n_added"), 128, seed=seed)
        ids = np.arange(n + ix.stat("n_added"), n + total, dtype=np.uint32)
        model.add(dpq.encode(t["cw"], x), ids, ix.add_vectors(x, ids))
        pos, ids_, dist = ix.search(queries, 10)
        assert ix.stat("last_coarse") == 1
        model.check(lut, pos, ids_, dist, 10, rows=range(0, 150, 8))
    ix.close()


# ------------------------------------------------------------------------------------------- errors --
@gpu
def test_errors_and_stats(golden4000, monkeypatch):
    g = golden4000
    n = int(g["n"])
    L = dpq.lib()
    add = codes_of(g["cw"], 6, seed=31)
    p = add.ctypes.data_as(C.c_void_p)
    # a part placed right below the sentinel: 5 more positions fit, a sixth would reach 0xFFFFFFFF
    top = 0xFFFFFFFF - n - 5
    ix = dpq.DeltaTreeIndex(g["payload"], n, 8, 256, pos2id=g["vec_id"], first_pos=top)
    ix.set_codebook(g["cw"])
    assert L.dpq_index_add(ix._h, p, 6, None, None) == -1
    assert b"0xFFFFFFFF" in L.dpq_last_error()
    assert ix.stat("n_local") == n and ix.stat("n_added") == 0
    pos = ix.add(add[:5])
    assert pos.max() == 0xFFFFFFFE
    assert L.dpq_index_add(ix._h, p, 1, None, None) == -1
    ix.close()
    ix = open_golden(g)
    assert L.dpq_index_add(ix._h, None, 3, None, None) == -1
    assert L.dpq_index_add(ix._h, None, 0, None, None) == 0
    assert L.dpq_index_add(ix._h, p, 1 << 31, None, None) == -1
    assert L.dpq_index_add_vectors(ix._h, p, 2, 129, None, None) == -1  # D > M * Ds
    ix.add(add)
    ix.add(add[:2])
    assert (ix.stat("n_added"), ix.stat("n_local"), ix.stat("n_codes")) == (8, n + 8, n)
    assert ix.stat("device_bytes_per_node") == 8 and ix.stat("last_add_us") >= 0
    ix.close()
    ix = dpq.DeltaTreeIndex(g["payload"], n, 8, 256, pos2id=g["vec_id"])  # no codebook
    x = dg.sift_like(4, 128, seed=32)
    with pytest.raises(dpq.DpqError, match="codebook"):
        ix.add_vectors(x)
    ix.add(add)  # codes need no codebook
    ix.close()
    monkeypatch.setenv("DPQ_ENGINE", "1")
    ix = open_golden(g)
    assert ix.stat("engine") == 1
    assert L.dpq_index_add(ix._h, p, 6, None, None) == -1
    assert b"code-array engine" in L.dpq_last_error()
    ix.close()


# ------------------------------------------------------------------------------------------- CLI --
@gpu
@pytest.mark.parametrize("parts", [1, 2])
def test_cli_query_with_added_vectors(tmp_path, parts):
    n, nq, M, K, k, na = 6000, 40, 8, 256, 10, 1500
    d = str(tmp_path)
    dg.make_dataset(d, n, nq, M=M, K=K, d=128, seed=37)
    common = ["-m", str(M), "-k", str(K), "-N", str(n), "-ext", "fvecs"]
    run = lambda cmd: subprocess.run(cmd, capture_output=True, text=True)  # noqa: E731
    r = run([BIN + "/pqtree", "-dataset", d, "-task", "encode"] + common)
    assert r.returncode == 0, r.stderr
    extra = ["-parts", str(parts)] if parts > 1 else []
    r = run([BIN + "/deltapq", "-dataset", d, "-task", "approx_tree", "-h", "1", "-diff", "8"] + common + extra)
    assert r.returncode == 0, r.stderr
    queries = dg.read_vecs(d + "/query.fvecs")[:nq]
    x = np.concatenate([queries[:20] + 0.5, dg.sift_like(na - 20, 128, seed=38)]).astype(np.float32)
    dg.write_vecs(d + "/add.fvecs", x)
    del_ids = np.arange(n, n + na, 7)  # the deleted file may name added ids
    with open(d + "/ids.txt", "w") as f:
        f.write(" ".join(map(str, del_ids)) + "\n")
    r = run([BIN + "/deltapq", "-dataset", d, "-task", "query", "-query_size", str(nq), "-topk", str(k), "-add",
             d + "/add.fvecs", "-deleted", d + "/ids.txt", "-results", d + "/out.txt"] + common + extra)
    assert r.returncode == 0, r.stderr
    lines = open(d + "/out.txt").read().splitlines()
    assert lines[0] == f"{nq},{k}"
    got = [np.array(ln.rstrip(",").split(","), np.float64).reshape(-1, 2) for ln in lines[1:]]
    ids = np.array([g_[:, 0] for g_ in got], np.int64)
    dist = np.array([g_[:, 1] for g_ in got])
    assert (ids >= n).any() and not np.isin(ids, del_ids).any()
    cw = dg.read_codebook(d + f"/M{M}K{K}codewords.txt")
    codes = np.concatenate([dg.read_codes(d + f"/codes.bin.plain.M{M}K{K}N{n}", M), dpq.encode(cw, x)])
    lut = dpq.adc_tables(cw, queries)
    dead = np.zeros(n + na, bool)
    dead[del_ids] = True
    for i in range(nq):
        nd = node_dist(lut[i], codes)
        nd[dead] = np.inf
        np.testing.assert_allclose(dist[i], np.sort(nd)[:k], rtol=1e-5)
        np.testing.assert_allclose(nd[ids[i]], dist[i], rtol=1e-5)


# ------------------------------------------------------------------------------------------- no GPU --
def test_add_entry_points_fail_loudly_without_gpu():
    if dpq.device_count() > 0:
        pytest.skip("a GPU is present")
    L = dpq.lib()
    codes = np.zeros((3, 8), np.uint8)
    p = codes.ctypes.data_as(C.c_void_p)
    for name in ("dpq_index_add", "dpq_multi_add"):
        assert getattr(L, name)(None, p, 3, None, None) == -2, name
        assert b"no CUDA device" in L.dpq_last_error(), name
    for name in ("dpq_index_add_vectors", "dpq_multi_add_vectors"):
        assert getattr(L, name)(None, p, 3, 128, None, None) == -2, name
        assert b"no CUDA device" in L.dpq_last_error(), name
