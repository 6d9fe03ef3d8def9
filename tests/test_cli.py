"""Drop-in command line tools (deltapq_b200/bin/pqtree, deltapq): same flags and files as the
reference binaries.  GPU test: the task chain encode -> approx_tree -> query on BASELINE
configs[0] (10K x 128, M=8 K=256 h=1, 100 queries top-10) writes files that are byte-identical
to what the UNMODIFIED reference binaries (oracle/_ref, canonical stable-sort tree build) write,
and prints the same nearest neighbour per query."""
import filecmp
import os
import shutil
import subprocess

import numpy as np
import pytest

import datagen as dg
from oracle import pyoracle as po

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "deltapq_b200", "bin")


def run(cmd, **kw):
    return subprocess.run(cmd, capture_output=True, text=True, **kw)


def test_cli_binaries_exist_and_reject_bad_input(tmp_path):
    for b in ("pqtree", "deltapq"):
        assert os.access(os.path.join(BIN, b), os.X_OK), b
        r = run([os.path.join(BIN, b)])
        assert r.returncode != 0 and "usage" in r.stderr
    r = run([os.path.join(BIN, "deltapq"), "-dataset", str(tmp_path), "-task", "query", "-N", "10"])
    assert r.returncode != 0 and "codebook" in r.stderr
    r = run([os.path.join(BIN, "pqtree"), "-dataset", str(tmp_path), "-task", "recall"])
    assert r.returncode != 0 and "scope" in r.stderr


def test_cli_fails_loudly_without_gpu(tmp_path):
    import deltapq_b200 as dpq
    if dpq.device_count() > 0:
        pytest.skip("a GPU is present")
    dg.make_dataset(str(tmp_path), 300, 5, M=8, K=256, d=128, seed=3, n_learn=600)
    r = run([os.path.join(BIN, "pqtree"), "-dataset", str(tmp_path), "-task", "encode", "-N", "300"])
    assert r.returncode != 0 and "no CUDA device" in r.stderr


@pytest.mark.gpu
def test_cli_chain_matches_reference_binaries(tmp_path):
    n, nq, M, K, k = 10000, 100, 8, 256, 10
    ours, ref = str(tmp_path / "ours"), str(tmp_path / "ref")
    dg.make_dataset(ours, n, nq, M=M, K=K, d=128, seed=31)
    shutil.copytree(ours, ref)
    common = ["-m", str(M), "-k", str(K), "-N", str(n), "-ext", "fvecs"]
    r = run([BIN + "/pqtree", "-dataset", ours, "-task", "encode"] + common)
    assert r.returncode == 0, r.stderr
    r = run([BIN + "/deltapq", "-dataset", ours, "-task", "approx_tree", "-h", "1", "-diff", "8"] + common)
    assert r.returncode == 0, r.stderr
    r = run([BIN + "/deltapq", "-dataset", ours, "-task", "query", "-query_size", str(nq), "-topk", str(k), "-debug",
             "-results", ours + "/results.txt"] + common)
    assert r.returncode == 0, r.stderr
    assert "[msec/query]" in r.stdout
    mine = [ln.split() for ln in r.stdout.splitlines() if " id " in ln]
    assert len(mine) == nq
    names = [f"codes.bin.plain.M{M}K{K}N{n}", f"M{M}K{K}H1_Approx_Edges_N{n}", f"M{M}K{K}_Approx_TreeNodesDFS_N{n}",
             f"M{M}K{K}_Approx_compressed_codes_opt_N{n}"]
    have_ref = all(os.path.exists(os.path.join(po.REF_DIR, b)) for b in ("pqtree", "deltapq_canon", "deltapq"))
    if have_ref:
        r = run([po.REF_DIR + "/pqtree", "-dataset", ref, "-task", "encode"] + common)
        assert r.returncode == 0, r.stderr[-2000:]
        r = run([po.REF_DIR + "/deltapq_canon", "-dataset", ref, "-task", "approx_tree", "-h", "1", "-diff", "8"] + common)
        assert r.returncode == 0, r.stderr[-2000:]
        for nm in names:
            assert filecmp.cmp(os.path.join(ours, nm), os.path.join(ref, nm), shallow=False), nm
        r = run([po.REF_DIR + "/deltapq", "-dataset", ref, "-task", "query", "-query_size", str(nq), "-topk", str(k),
                 "-debug"] + common)
        assert r.returncode == 0, r.stderr[-2000:]
        theirs = [ln.split() for ln in r.stdout.splitlines() if len(ln.split()) == 2 and ln.split()[0].isdigit()]
        assert len(theirs) >= nq
        for a, b in zip(mine, theirs[:nq]):  # reference prints "pos dist" of the top-1 (dmain:341)
            assert abs(float(a[1]) - float(b[1])) <= 1e-5 * float(b[1])
    else:  # no reference binaries on this box: the oracle restatement of the same files
        base = dg.read_vecs(ours + "/base.fvecs")
        cw = dg.read_codebook(ours + f"/M{M}K{K}codewords.txt")
        codes = po.encode(cw, base)
        assert np.array_equal(dg.read_codes(os.path.join(ours, names[0]), M), codes)
        edges, root, lay, payload = po.build_tree(codes, cw)
        e = np.fromfile(os.path.join(ours, names[1]), np.uint32)
        assert e[0] == root and np.array_equal(e[1:].reshape(-1, 2), edges)
        assert np.array_equal(np.fromfile(os.path.join(ours, names[2]), np.uint8), po.qnodes8(codes, lay))
        nc, pl = dg.read_dtc(os.path.join(ours, names[3]))
        assert nc == n and np.array_equal(pl, payload)
    # results file: vector ids + distances against the oracle scan
    cw = dg.read_codebook(ours + f"/M{M}K{K}codewords.txt")
    nc, pl = dg.read_dtc(os.path.join(ours, names[3]))
    qn = np.fromfile(os.path.join(ours, names[2]), np.uint8).reshape(n + 1, 60)
    vec_id = qn[:n, 0:4].copy().view(np.uint32).ravel()
    queries = dg.read_vecs(ours + "/query.fvecs")
    lines = open(ours + "/results.txt").read().splitlines()
    assert lines[0] == f"{nq},{k}"
    for i in (0, 17, 99):
        vals = lines[1 + i].rstrip(",").split(",")
        ids = np.array(vals[0::2], np.int64)
        opos, odist = po.scan(pl, n, cw, queries[i], k)
        np.testing.assert_allclose(np.array(vals[1::2], np.float64), odist, rtol=1e-5)
        assert ids[0] == vec_id[opos[0]] or odist[0] == odist[1]


@pytest.mark.gpu
def test_cli_groundtruth_and_learn(tmp_path):
    d = str(tmp_path)
    base, queries, _ = dg.make_dataset(d, 5000, 20, M=8, K=256, d=128, seed=41)
    dg.write_vecs(d + "/learn.fvecs", dg.sift_like(3000, 128, seed=44))
    os.makedirs(d + "/groundtruth")
    r = run([BIN + "/pqtree", "-dataset", d, "-task", "groundtruth", "-N", "5000", "-query_size", "20", "-topk", "5"])
    assert r.returncode == 0, r.stderr
    lines = open(d + "/groundtruth/N5000Top5.txt").read().splitlines()
    assert lines[0] == "20,5"
    oid, odist = po.groundtruth(base, queries, 5)
    for i in range(20):
        vals = lines[1 + i].rstrip(",").split(",")
        assert [int(v) for v in vals[0::2]] == list(oid[i]) or len(set(odist[i])) < 5
        assert [float(v) for v in vals[1::2]] == [float("%g" % v) for v in odist[i]]
    r = run([BIN + "/pqtree", "-dataset", d, "-task", "learn", "-m", "8", "-k", "16", "-train_size", "2000"])
    assert r.returncode == 0, r.stderr
    cw = dg.read_codebook(d + "/M8K16codewords.txt")
    assert cw.shape == (8, 16, 16) and np.isfinite(cw).all() and len(np.unique(cw[0], axis=0)) == 16


@pytest.mark.gpu
def test_cli_query_multi_gpu_matches_single_gpu(tmp_path):
    """`deltapq -task query -gpus 2`: one shard per GPU, NCCL all-gather of the top-k keys, merge
    kernel (dpq_multi_*).  Result file identical to the single-GPU run.  Needs 2 GPUs."""
    import deltapq_b200 as dpq
    if dpq.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    n, nq, M, K, k = 60000, 500, 8, 256, 10
    d = str(tmp_path)
    dg.make_dataset(d, n, nq, M=M, K=K, d=128, seed=51)
    common = ["-dataset", d, "-m", str(M), "-k", str(K), "-N", str(n), "-ext", "fvecs"]
    for cmd in ([BIN + "/pqtree", "-task", "encode"], [BIN + "/deltapq", "-task", "approx_tree", "-h", "1", "-diff", "8"]):
        r = run(cmd + common)
        assert r.returncode == 0, r.stderr
    outs = []
    for g in (1, 2):
        out = f"{d}/res{g}.txt"
        r = run([BIN + "/deltapq", "-task", "query", "-query_size", str(nq), "-topk", str(k), "-gpus", str(g),
                 "-results", out] + common)
        assert r.returncode == 0, r.stderr
        outs.append(open(out).read())
    assert outs[0] == outs[1]


def _parse_results(path):
    lines = open(path).read().strip().split("\n")
    nq, k = (int(v) for v in lines[0].split(","))
    ids = np.zeros((nq, k), np.int64)
    dist = np.zeros((nq, k), np.float64)
    for i, line in enumerate(lines[1:]):
        vals = line.rstrip(",").split(",")
        ids[i] = [int(v) for v in vals[0::2]]
        dist[i] = [float(v) for v in vals[1::2]]
    return ids, dist


@pytest.mark.gpu
def test_cli_forest_parts_match_single_tree(tmp_path):
    """`deltapq -task approx_tree -parts 3` + `-task query -parts 3` (the 1B-code layout: one tree
    per vector-id range, dpq_multi_open_parts): same distances as the single-tree query and the
    same ids wherever the distance is not tied; with 2 GPUs also `-gpus 2`."""
    import deltapq_b200 as dpq
    n, nq, M, K, k = 30001, 200, 8, 256, 10
    d = str(tmp_path)
    dg.make_dataset(d, n, nq, M=M, K=K, d=128, seed=61)
    common = ["-dataset", d, "-m", str(M), "-k", str(K), "-N", str(n), "-ext", "fvecs"]
    for cmd in ([BIN + "/pqtree", "-task", "encode"],
                [BIN + "/deltapq", "-task", "approx_tree", "-h", "1", "-diff", "8"],
                [BIN + "/deltapq", "-task", "approx_tree", "-h", "1", "-diff", "8", "-parts", "3"]):
        r = run(cmd + common)
        assert r.returncode == 0, r.stderr
    assert os.path.exists(f"{d}/M8K256_Approx_compressed_codes_opt_N{n}.part2of3")
    if dpq.device_count() >= 2:  # -gpus 2: one builder thread per GPU, byte-identical part files
        d2 = str(tmp_path / "g2")
        os.makedirs(d2)
        for f in ("base.fvecs", "query.fvecs", "M8K256codewords.txt", f"codes.bin.plain.M8K256N{n}"):
            shutil.copy(os.path.join(d, f), d2)
        r = run([BIN + "/deltapq", "-task", "approx_tree", "-h", "1", "-diff", "8", "-parts", "3", "-gpus", "2",
                 "-dataset", d2] + common[2:])
        assert r.returncode == 0, r.stderr
        for p in range(3):
            for stem in ("M8K256_Approx_compressed_codes_opt", "M8K256_Approx_TreeNodesDFS", "M8K256H1_Approx_Edges"):
                assert filecmp.cmp(f"{d}/{stem}_N{n}.part{p}of3", f"{d2}/{stem}_N{n}.part{p}of3", shallow=False), (stem, p)
    q = [BIN + "/deltapq", "-task", "query", "-query_size", str(nq), "-topk", str(k)]
    r = run(q + ["-results", f"{d}/whole.txt"] + common)
    assert r.returncode == 0, r.stderr
    wid, wdist = _parse_results(f"{d}/whole.txt")
    for g in (1, 2):
        if g > dpq.device_count():
            continue
        r = run(q + ["-parts", "3", "-gpus", str(g), "-results", f"{d}/parts{g}.txt"] + common)
        assert r.returncode == 0, r.stderr
        pid, pdist = _parse_results(f"{d}/parts{g}.txt")
        assert np.array_equal(pdist, wdist)
        for i in range(nq):
            untied = np.array([np.sum(wdist[i] == v) == 1 and v < wdist[i, -1] for v in wdist[i]])
            assert np.array_equal(pid[i][untied], wid[i][untied]), i


@pytest.mark.gpu
def test_cli_encode_bvecs_equals_fvecs(tmp_path):
    """`pqtree -task encode -ext bvecs` (SIFT1B's format; raw records go to the device through
    dpq_encode_u8) writes the same codes file as the fvecs run on the same components, and the
    reference binary agrees when it is available."""
    n, M, K = 7000, 8, 256
    d = str(tmp_path / "b")
    f = str(tmp_path / "f")
    base, _, _ = dg.make_dataset(f, n, 10, M=M, K=K, d=128, seed=71)
    os.makedirs(d)
    dg.write_vecs(d + "/base.bvecs", base, ext="bvecs")
    shutil.copy(f + f"/M{M}K{K}codewords.txt", d)
    for path, ext in ((f, "fvecs"), (d, "bvecs")):
        r = run([BIN + "/pqtree", "-dataset", path, "-task", "encode", "-m", str(M), "-k", str(K), "-N", str(n), "-ext", ext])
        assert r.returncode == 0, r.stderr
    name = f"/codes.bin.plain.M{M}K{K}N{n}"
    assert filecmp.cmp(d + name, f + name, shallow=False)
    if os.path.exists(os.path.join(po.REF_DIR, "pqtree")):
        rdir = str(tmp_path / "r")
        os.makedirs(rdir)
        shutil.copy(d + "/base.bvecs", rdir)
        shutil.copy(f + f"/M{M}K{K}codewords.txt", rdir)
        r = run([po.REF_DIR + "/pqtree", "-dataset", rdir, "-task", "encode", "-m", str(M), "-k", str(K), "-N", str(n), "-ext", "bvecs"])
        if r.returncode == 0 and os.path.exists(rdir + name):
            assert filecmp.cmp(rdir + name, d + name, shallow=False)
