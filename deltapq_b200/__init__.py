"""deltapq_b200 -- thin ctypes binding over libdpq.so (the C ABI in include/dpq.h).

This is plumbing for tests and bench.py, not the product: the product is the CUDA library
and the C++ command-line tools built from deltapq_b200/csrc.  There is no CPU fallback; if
libdpq.so is missing or no GPU is visible the calls raise.
"""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdpq.so")

# every symbol include/dpq.h declares (tests check the library exports all of them)
SYMBOLS = [
    "dpq_version", "dpq_last_error", "dpq_device_count", "dpq_set_device",
    "dpq_index_open", "dpq_index_open_part", "dpq_index_open_file", "dpq_index_open_part_file",
    "dpq_multi_open_parts", "dpq_index_open_tree", "dpq_index_open_tree_shard", "dpq_tree_build_device",
    "dpq_index_set_codebook", "dpq_index_set_option",
    "dpq_index_set_stream",
    "dpq_index_search", "dpq_index_search_device", "dpq_index_sync", "dpq_merge_topk_device",
    "dpq_malloc", "dpq_free", "dpq_memcpy_h2d", "dpq_memcpy_d2h", "dpq_malloc_host",
    "dpq_free_host", "dpq_index_stat", "dpq_index_close", "dpq_adc_tables", "dpq_encode", "dpq_encode_u8", "dpq_encode_stat",
    "dpq_find_edges", "dpq_edge_diffs", "dpq_groundtruth_begin", "dpq_groundtruth_chunk",
    "dpq_groundtruth_finish", "dpq_groundtruth_stat", "dpq_program_compile", "dpq_program_size", "dpq_program_copy",
    "dpq_program_free", "dpq_tree_build", "dpq_tree_from_edges", "dpq_tree_size", "dpq_tree_copy",
    "dpq_tree_free", "dpq_multi_open_file", "dpq_multi_set_codebook", "dpq_multi_search", "dpq_multi_stat",
    "dpq_multi_close", "dpq_index_delete", "dpq_index_undelete", "dpq_multi_delete", "dpq_multi_undelete",
    "dpq_index_add", "dpq_index_add_vectors", "dpq_multi_add", "dpq_multi_add_vectors",
    "dpq_index_compact", "dpq_multi_compact",
]


class DpqError(RuntimeError):
    pass


def build(verbose=False):
    """Compile libdpq.so in tree for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-j8", "-C", os.path.join(HERE, "csrc")], capture_output=not verbose, text=True)
    if r.returncode != 0:
        raise DpqError("building libdpq.so failed:\n" + (r.stdout or "") + (r.stderr or ""))


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DpqError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
    L.dpq_last_error.restype = C.c_char_p
    L.dpq_index_open.argtypes = [vp, i64, i64, i32, i32, vp, i32, i32, C.POINTER(vp)]
    L.dpq_index_open_part.argtypes = [vp, i64, i64, i32, i32, vp, i64, C.POINTER(vp)]
    L.dpq_index_open_tree.argtypes = [vp, i64, C.POINTER(vp)]
    L.dpq_index_open_tree_shard.argtypes = [vp, i32, i32, C.POINTER(vp)]
    L.dpq_tree_build_device.argtypes = [vp, i64, i32, i32, vp, i32, i32, i32, C.POINTER(vp)]
    L.dpq_index_open_file.argtypes = [C.c_char_p, C.c_char_p, i32, i32, i32, i32, C.POINTER(vp)]
    L.dpq_index_set_codebook.argtypes = [vp, vp, i32]
    L.dpq_index_set_option.argtypes = [vp, C.c_char_p, i64]
    L.dpq_index_set_stream.argtypes = [vp, vp]
    L.dpq_index_search.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    L.dpq_index_search_device.argtypes = [vp, vp, i32, i32, vp]
    L.dpq_index_sync.argtypes = [vp]
    L.dpq_merge_topk_device.argtypes = [vp, vp, i32, i32, i32, vp]
    L.dpq_malloc.argtypes = [C.POINTER(vp), sz]
    L.dpq_free.argtypes = [vp]
    L.dpq_memcpy_h2d.argtypes = [vp, vp, sz]
    L.dpq_memcpy_d2h.argtypes = [vp, vp, sz]
    L.dpq_malloc_host.argtypes = [C.POINTER(vp), sz]
    L.dpq_free_host.argtypes = [vp]
    L.dpq_index_stat.restype = i64
    L.dpq_index_stat.argtypes = [vp, C.c_char_p]
    L.dpq_index_close.argtypes = [vp]
    L.dpq_index_close.restype = None
    L.dpq_adc_tables.argtypes = [vp, i32, i32, i32, vp, i32, vp]
    L.dpq_encode.argtypes = [vp, i32, i32, i32, vp, i64, i32, vp]
    L.dpq_encode_u8.argtypes = [vp, i32, i32, i32, vp, i64, i32, i64, i64, vp]
    L.dpq_encode_stat.argtypes = [C.c_char_p]
    L.dpq_encode_stat.restype = C.c_int64
    L.dpq_find_edges.argtypes = [vp, i64, i32, i32, i32, i32, vp, C.POINTER(C.c_uint32)]
    L.dpq_edge_diffs.argtypes = [vp, i64, i32, vp, i64, vp, C.POINTER(i64)]
    L.dpq_groundtruth_begin.argtypes = [vp, i32, i32, i32, C.POINTER(vp)]
    L.dpq_groundtruth_chunk.argtypes = [vp, vp, i64, i64]
    L.dpq_groundtruth_finish.argtypes = [vp, vp, vp]
    L.dpq_groundtruth_stat.restype = i64
    L.dpq_groundtruth_stat.argtypes = [vp, C.c_char_p]
    L.dpq_program_compile.argtypes = [vp, i64, i64, i32, i32, i32, i32, i32, C.POINTER(vp)]
    L.dpq_program_size.restype = i64
    L.dpq_program_size.argtypes = [vp, C.c_char_p]
    L.dpq_program_copy.argtypes = [vp, C.c_char_p, vp]
    L.dpq_program_free.argtypes = [vp]
    L.dpq_program_free.restype = None
    L.dpq_tree_build.argtypes = [vp, i64, i32, i32, vp, i32, i32, i32, C.POINTER(vp)]
    L.dpq_tree_from_edges.argtypes = [vp, i64, i32, i32, vp, i32, vp, C.c_uint32, C.POINTER(vp)]
    L.dpq_tree_size.restype = i64
    L.dpq_tree_size.argtypes = [vp, C.c_char_p]
    L.dpq_tree_copy.argtypes = [vp, C.c_char_p, vp]
    L.dpq_tree_free.argtypes = [vp]
    L.dpq_tree_free.restype = None
    L.dpq_multi_open_file.argtypes = [C.c_char_p, C.c_char_p, i32, i32, i32, C.POINTER(vp)]
    L.dpq_multi_set_codebook.argtypes = [vp, vp, i32]
    L.dpq_multi_search.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    L.dpq_multi_stat.restype = i64
    L.dpq_multi_stat.argtypes = [vp, i32, C.c_char_p]
    L.dpq_multi_close.argtypes = [vp]
    L.dpq_multi_close.restype = None
    for name in ("dpq_index_delete", "dpq_index_undelete", "dpq_multi_delete", "dpq_multi_undelete"):
        getattr(L, name).argtypes = [vp, vp, i64]
    for name in ("dpq_index_add", "dpq_multi_add"):
        getattr(L, name).argtypes = [vp, vp, i64, vp, vp]
    for name in ("dpq_index_add_vectors", "dpq_multi_add_vectors"):
        getattr(L, name).argtypes = [vp, vp, i64, i32, vp, vp]
    L.dpq_index_compact.argtypes = [vp, C.POINTER(vp)]
    L.dpq_multi_compact.argtypes = [vp]
    _lib = L
    return L


def _check(rc):
    if rc != 0:
        raise DpqError(f"libdpq error {rc}: {lib().dpq_last_error().decode()}")


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def device_count():
    return lib().dpq_device_count()


def set_device(dev):
    _check(lib().dpq_set_device(dev))


class DeviceBuffer:
    """Raw device allocation through the C ABI (no torch / cuda-python needed)."""

    def __init__(self, nbytes):
        self.ptr = C.c_void_p()
        self.nbytes = nbytes
        _check(lib().dpq_malloc(C.byref(self.ptr), max(nbytes, 16)))

    def upload(self, arr):
        arr = np.ascontiguousarray(arr)
        assert arr.nbytes <= self.nbytes
        _check(lib().dpq_memcpy_h2d(self.ptr, _ptr(arr), arr.nbytes))
        return self

    def download(self, dtype, shape):
        out = np.empty(shape, dtype)
        assert out.nbytes <= self.nbytes
        _check(lib().dpq_memcpy_d2h(_ptr(out), self.ptr, out.nbytes))
        return out

    def free(self):
        if self.ptr:
            lib().dpq_free(self.ptr)
            self.ptr = C.c_void_p()


def pinned_array(shape, dtype):
    """numpy array over page-locked host memory from dpq_malloc_host (kept alive by the array);
    dpq_index_search copies from such a buffer without staging."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    _check(lib().dpq_malloc_host(C.byref(p), max(n, 16)))
    buf = (C.c_char * n).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    _PINNED.append((arr, p))  # never freed before process exit: the array may outlive any scope
    return arr


_PINNED = []


def _id_array(ids):
    ids = np.ascontiguousarray(np.asarray(ids).reshape(-1), np.uint32)
    return ids, (_ptr(ids) if ids.size else None)


def _add(fn, h, data, ids, D=None):
    """dpq_index_add / dpq_multi_add (D None: data are codes [n][M] uint8) or their _add_vectors forms (data
    [n][D] float32) -> the position given to each input row."""
    if D is None:
        data = np.ascontiguousarray(data, np.uint8)
    else:
        data = np.ascontiguousarray(data, np.float32)
    n = data.shape[0]
    p_ids = None
    if ids is not None:
        ids = np.ascontiguousarray(np.asarray(ids).reshape(-1), np.uint32)
        assert ids.size == n
        p_ids = _ptr(ids)
    pos = np.empty(n, np.uint32)
    if D is None:
        _check(fn(h, _ptr(data), n, p_ids, _ptr(pos)))
    else:
        _check(fn(h, _ptr(data), n, data.shape[1], p_ids, _ptr(pos)))
    return pos


def unpack_keys(keys):
    """uint64 keys (float bits << 32 | pos) -> (pos uint32, dist float32)."""
    keys = np.asarray(keys, np.uint64)
    pos = (keys & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    dist = (keys >> np.uint64(32)).astype(np.uint32).view(np.float32)
    return pos, dist


class DeltaTreeIndex:
    """Host mirror of the reference's query entry points (DCAT.h:2805 / :3731): open a
    compressed DeltaTree, set the codebook, search batches of queries."""

    def __init__(self, payload, n_codes, M, K, pos2id=None, rank=0, n_ranks=1, first_pos=None):
        """first_pos: open the tree as one part of a forest (dpq_index_open_part): the whole
        tree, positions reported as first_pos + DFS position."""
        payload = np.ascontiguousarray(payload, np.uint8)
        self.M, self.K = M, K
        self._h = C.c_void_p()
        p2i = None
        if pos2id is not None:
            self._p2i = np.ascontiguousarray(pos2id, np.uint32)
            p2i = _ptr(self._p2i)
        if first_pos is not None:
            _check(lib().dpq_index_open_part(_ptr(payload), payload.nbytes, n_codes, M, K, p2i, int(first_pos),
                                             C.byref(self._h)))
        else:
            _check(lib().dpq_index_open(_ptr(payload), payload.nbytes, n_codes, M, K, p2i, rank, n_ranks,
                                        C.byref(self._h)))
        self.Ds = None

    @classmethod
    def from_file(cls, tree_path, M, K, qnode_path=None, rank=0, n_ranks=1):
        self = cls.__new__(cls)
        self.M, self.K = M, K
        self._h = C.c_void_p()
        _check(lib().dpq_index_open_file(tree_path.encode(), qnode_path.encode() if qnode_path else None,
                                         M, K, rank, n_ranks, C.byref(self._h)))
        self.Ds = None
        return self

    def set_codebook(self, cw):
        cw = np.ascontiguousarray(cw, np.float32)
        assert cw.shape[0] == self.M and cw.shape[1] == self.K
        self.Ds = cw.shape[2]
        _check(lib().dpq_index_set_codebook(self._h, _ptr(cw), self.Ds))

    def set_option(self, name, value):
        _check(lib().dpq_index_set_option(self._h, name.encode(), int(value)))

    def set_stream(self, cuda_stream):
        """cuda_stream: integer cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream)."""
        _check(lib().dpq_index_set_stream(self._h, C.c_void_p(cuda_stream)))

    def stat(self, name):
        return int(lib().dpq_index_stat(self._h, name.encode()))

    def search(self, queries, topk, out=None):
        """Host buffers in, host buffers out: (pos [Q][k], id [Q][k], dist [Q][k]).  out: a tuple of
        caller-owned result arrays to fill (the C ABI's caller-owned buffers) instead of new ones."""
        q = np.ascontiguousarray(queries, np.float32)
        Q = q.shape[0]
        if out is None:
            out = (np.empty((Q, topk), np.uint32), np.empty((Q, topk), np.uint32), np.empty((Q, topk), np.float32))
        pos, ids, dist = out
        assert pos.shape == ids.shape == dist.shape == (Q, topk) and pos.flags.c_contiguous
        _check(lib().dpq_index_search(self._h, _ptr(q), Q, topk, _ptr(pos), _ptr(ids), _ptr(dist)))
        return pos, ids, dist

    def delete(self, ids):
        """dpq_index_delete: the vector ids (what search reports as ids) stop appearing in results."""
        ids, p = _id_array(ids)
        _check(lib().dpq_index_delete(self._h, p, ids.size))

    def undelete(self, ids):
        ids, p = _id_array(ids)
        _check(lib().dpq_index_undelete(self._h, p, ids.size))

    def add(self, codes, ids=None):
        """dpq_index_add: codes [n][M] appended (ids None: id = position); returns each row's position."""
        return _add(lib().dpq_index_add, self._h, codes, ids)

    def add_vectors(self, x, ids=None):
        """dpq_index_add_vectors: x [n][D] encoded with the index's codebook and appended; returns the positions."""
        return _add(lib().dpq_index_add_vectors, self._h, x, ids, D=np.asarray(x).shape[1])

    def compact(self, want=("payload", "vec_id", "qnodes")):
        """dpq_index_compact: the tree is rebuilt over the live nodes (positions renumbered, ids kept).  Returns the
        new tree's arrays by name, as tree_build does (vec_id = the carried ids; "qnodes" at M = 8 only), or None
        with want=None, in which case only the index's id table leaves the device."""
        if want is None:
            _check(lib().dpq_index_compact(self._h, None))
            return None
        t = C.c_void_p()
        _check(lib().dpq_index_compact(self._h, C.byref(t)))
        return _tree_out(t, self.M, want)

    def search_device(self, d_queries_ptr, Q, topk, d_out_ptr):
        _check(lib().dpq_index_search_device(self._h, d_queries_ptr, Q, topk, d_out_ptr))

    def merge_device(self, d_keys_ptr, n_lists, Q, topk, d_out_ptr):
        _check(lib().dpq_merge_topk_device(self._h, d_keys_ptr, n_lists, Q, topk, d_out_ptr))

    def sync(self):
        _check(lib().dpq_index_sync(self._h))

    def close(self):
        if self._h:
            lib().dpq_index_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class MultiIndex:
    """dpq_multi_*: one process drives one subtree shard per GPU (devices 0..n_gpus-1), NCCL
    all-gather of the key lists (libnccl bound at run time) + device merge: `deltapq -task query
    -gpus N` without torch."""

    def __init__(self, tree_path, M, K, n_gpus, qnode_path=None):
        self.M, self.K, self.n_gpus = M, K, n_gpus
        self._h = C.c_void_p()
        _check(lib().dpq_multi_open_file(tree_path.encode(), qnode_path.encode() if qnode_path else None, M, K, n_gpus,
                                         C.byref(self._h)))

    def set_codebook(self, cw):
        cw = np.ascontiguousarray(cw, np.float32)
        _check(lib().dpq_multi_set_codebook(self._h, _ptr(cw), cw.shape[2]))

    def search(self, queries, topk):
        q = np.ascontiguousarray(queries, np.float32)
        Q = q.shape[0]
        pos = np.empty((Q, topk), np.uint32)
        ids = np.empty((Q, topk), np.uint32)
        dist = np.empty((Q, topk), np.float32)
        _check(lib().dpq_multi_search(self._h, _ptr(q), Q, topk, _ptr(pos), _ptr(ids), _ptr(dist)))
        return pos, ids, dist

    def delete(self, ids):
        """dpq_multi_delete: vector ids (through the QNode file when one was given, else positions)."""
        ids, p = _id_array(ids)
        _check(lib().dpq_multi_delete(self._h, p, ids.size))

    def undelete(self, ids):
        ids, p = _id_array(ids)
        _check(lib().dpq_multi_undelete(self._h, p, ids.size))

    def add(self, codes, ids=None):
        """dpq_multi_add: appended to the index that ends the position space; returns the global positions."""
        return _add(lib().dpq_multi_add, self._h, codes, ids)

    def add_vectors(self, x, ids=None):
        return _add(lib().dpq_multi_add_vectors, self._h, x, ids, D=np.asarray(x).shape[1])

    def compact(self):
        """dpq_multi_compact: one tree over the live nodes, dealt to the GPUs again (forest: every part rebuilt)."""
        _check(lib().dpq_multi_compact(self._h))

    def stat(self, rank, name):
        return int(lib().dpq_multi_stat(self._h, rank, name.encode()))

    def close(self):
        if self._h:
            lib().dpq_multi_close(self._h)
            self._h = C.c_void_p()


def adc_tables(cw, queries):
    cw = np.ascontiguousarray(cw, np.float32)
    q = np.ascontiguousarray(queries, np.float32)
    M, K, Ds = cw.shape
    out = np.empty((q.shape[0], M, K), np.float32)
    _check(lib().dpq_adc_tables(_ptr(cw), M, K, Ds, _ptr(q), q.shape[0], _ptr(out)))
    return out


def encode(cw, x):
    cw = np.ascontiguousarray(cw, np.float32)
    x = np.ascontiguousarray(x, np.float32)
    M, K, Ds = cw.shape
    codes = np.empty((x.shape[0], M), np.uint8)
    _check(lib().dpq_encode(_ptr(cw), M, K, Ds, _ptr(x), x.shape[0], x.shape[1], _ptr(codes)))
    return codes


def encode_stat(name):
    """dpq_encode_stat: "tc" / "kernel_us" of the last encode call."""
    return int(lib().dpq_encode_stat(name.encode()))


def encode_u8(cw, raw, n, D, row_stride, row_offset):
    """dpq_encode_u8 over a buffer of raw uint8 records (e.g. the bytes of a .bvecs file)."""
    cw = np.ascontiguousarray(cw, np.float32)
    raw = np.ascontiguousarray(raw, np.uint8)
    M, K, Ds = cw.shape
    codes = np.empty((n, M), np.uint8)
    _check(lib().dpq_encode_u8(_ptr(cw), M, K, Ds, _ptr(raw), n, D, row_stride, row_offset, _ptr(codes)))
    return codes


def find_edges(codes, K=256, h=1, method=1):
    codes = np.ascontiguousarray(codes, np.uint8)
    n, M = codes.shape
    edges = np.zeros((max(n - 1, 1), 2), np.uint32)
    root = C.c_uint32(0)
    _check(lib().dpq_find_edges(_ptr(codes), n, M, K, h, method, _ptr(edges), C.byref(root)))
    return edges[: n - 1], int(root.value)


def edge_diffs(codes, edges):
    codes = np.ascontiguousarray(codes, np.uint8)
    edges = np.ascontiguousarray(edges, np.uint32)
    bm = np.empty(edges.shape[0], np.uint32)
    nd = C.c_int64(0)
    _check(lib().dpq_edge_diffs(_ptr(codes), codes.shape[0], codes.shape[1], _ptr(edges), edges.shape[0],
                                _ptr(bm), C.byref(nd)))
    return bm, int(nd.value)


_TREE_ARRAYS = (("edges", np.uint32), ("vec_id", np.uint32), ("parent_pos", np.uint32), ("child_num", np.uint32),
                ("depth", np.uint8), ("max_dist", np.float32), ("max_dist2p", np.float32),
                ("codes_by_pos", np.uint8), ("payload", np.uint8), ("qnodes", np.uint8))


def _tree_out(h, M, want=None):
    try:
        out = {}
        for name, dt in _TREE_ARRAYS:
            if want is not None and name not in want:
                continue
            nb = lib().dpq_tree_size(h, name.encode())
            if nb < 0:
                continue
            arr = np.empty(nb // np.dtype(dt).itemsize, dt)
            if nb:
                _check(lib().dpq_tree_copy(h, name.encode(), _ptr(arr)))
            out[name] = arr
        for name in ("root_id", "n_diffs", "n_codes", "edge_us", "layout_us"):
            out[name] = int(lib().dpq_tree_size(h, name.encode()))
        if "edges" in out:
            out["edges"] = out["edges"].reshape(-1, 2)
        if "codes_by_pos" in out:
            out["codes_by_pos"] = out["codes_by_pos"].reshape(-1, M)
        return out
    finally:
        lib().dpq_tree_free(h)


def tree_build(codes, cw, h=1, method=1, want=None, open_index_at=None):
    """`deltapq -task approx_tree` (DCAT.h:970): GPU edge search + GPU layout + stream.
    want: names of the arrays to fetch (default all; at 10^8 nodes the QNode file body alone
    is 6 GB).  open_index_at: also open the tree as an index (first_pos = that value) straight
    from the layout arrays; returned under "index"."""
    codes = np.ascontiguousarray(codes, np.uint8)
    cw = np.ascontiguousarray(cw, np.float32)
    n, M = codes.shape
    t = C.c_void_p()
    _check(lib().dpq_tree_build(_ptr(codes), n, M, cw.shape[1], _ptr(cw), cw.shape[2], h, method, C.byref(t)))
    if open_index_at is not None:  # dpq_index_open_tree: program compiled on the GPU from the layout arrays
        ix = DeltaTreeIndex.__new__(DeltaTreeIndex)
        ix.M, ix.K, ix.Ds = M, cw.shape[1], None
        ix._h = C.c_void_p()
        try:
            _check(lib().dpq_index_open_tree(t, int(open_index_at), C.byref(ix._h)))
        except Exception:
            lib().dpq_tree_free(t)
            raise
        out = _tree_out(t, M, want)
        out["index"] = ix
        return out
    return _tree_out(t, M, want)


class DeviceTree:
    """dpq_tree_build_device: one DeltaTree built and kept in HBM (the 10^9-code layout).  codes_ptr
    is a DEVICE pointer to [n][M] codes (or a numpy array).  shard(rank, n_ranks) opens whole depth-1
    subtrees as an index (dpq_index_open_tree_shard)."""

    def __init__(self, codes, n, M, cw, h=1, method=1):
        cw = np.ascontiguousarray(cw, np.float32)
        self.M, self.K, self.n = M, cw.shape[1], n
        self._t = C.c_void_p()
        if isinstance(codes, np.ndarray):
            self._keep = np.ascontiguousarray(codes, np.uint8)
            ptr = _ptr(self._keep)
        else:
            ptr = C.c_void_p(int(codes))
        _check(lib().dpq_tree_build_device(ptr, n, M, self.K, _ptr(cw), cw.shape[2], h, method, C.byref(self._t)))

    def stat(self, name):
        return int(lib().dpq_tree_size(self._t, name.encode()))

    def fetch(self, name, dtype):
        nb = self.stat(name)
        arr = np.empty(nb // np.dtype(dtype).itemsize, dtype)
        if nb:
            _check(lib().dpq_tree_copy(self._t, name.encode(), _ptr(arr)))
        return arr

    def shard(self, rank=0, n_ranks=1):
        ix = DeltaTreeIndex.__new__(DeltaTreeIndex)
        ix.M, ix.K, ix.Ds = self.M, self.K, None
        ix._h = C.c_void_p()
        _check(lib().dpq_index_open_tree_shard(self._t, rank, n_ranks, C.byref(ix._h)))
        return ix

    def free(self):
        if self._t:
            lib().dpq_tree_free(self._t)
            self._t = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def encode_device(cw, d_x_ptr, n, D, d_codes_ptr):
    """dpq_encode with DEVICE buffers x [n][D] float32 -> codes [n][M] (raw pointers)."""
    cw = np.ascontiguousarray(cw, np.float32)
    M, K, Ds = cw.shape
    _check(lib().dpq_encode(_ptr(cw), M, K, Ds, C.c_void_p(d_x_ptr), n, D, C.c_void_p(d_codes_ptr)))


def tree_from_edges(codes, cw, edges, root_id):
    """Host half of the build only (layout + stream), no GPU needed."""
    codes = np.ascontiguousarray(codes, np.uint8)
    cw = np.ascontiguousarray(cw, np.float32)
    edges = np.ascontiguousarray(edges, np.uint32)
    n, M = codes.shape
    t = C.c_void_p()
    _check(lib().dpq_tree_from_edges(_ptr(codes), n, M, cw.shape[1], _ptr(cw), cw.shape[2], _ptr(edges),
                                     int(root_id), C.byref(t)))
    return _tree_out(t, M)


def groundtruth(base, queries, topk, chunk=100000, stats=None):
    """stats: optional dict that receives dpq_groundtruth_stat's counters (tensor-core path)."""
    base = np.ascontiguousarray(base, np.float32)
    q = np.ascontiguousarray(queries, np.float32)
    st = C.c_void_p()
    _check(lib().dpq_groundtruth_begin(_ptr(q), q.shape[0], q.shape[1], topk, C.byref(st)))
    for s in range(0, base.shape[0], chunk):
        blk = base[s:s + chunk]
        _check(lib().dpq_groundtruth_chunk(st, _ptr(blk), blk.shape[0], s))
    if stats is not None:
        for name in ("tc", "tc_vectors", "tc_flagged"):
            stats[name] = int(lib().dpq_groundtruth_stat(st, name.encode()))
    ids = np.empty((q.shape[0], topk), np.uint32)
    dist = np.empty((q.shape[0], topk), np.float32)
    _check(lib().dpq_groundtruth_finish(st, _ptr(ids), _ptr(dist)))
    return ids, dist


def compile_program(payload, n_codes, M, K, rank=0, n_ranks=1, chunk_nodes=256, engine=0):
    """Host-only: the device scan program of one shard as numpy arrays (for tests).
    engine 0: the code-array program (prog["v2"] == 1: "codes_padded" [n_local][cstride] is
    what the scan kernels read, "codes" its first M columns); engine 1: the first-generation op
    program (ops / chunks / anc)."""
    payload = np.ascontiguousarray(payload, np.uint8)
    h = C.c_void_p()
    _check(lib().dpq_program_compile(_ptr(payload), payload.nbytes, n_codes, M, K, rank, n_ranks,
                                     -chunk_nodes if engine == 1 else chunk_nodes, C.byref(h)))
    try:
        out = {}
        for name, dt in (("ops", np.uint32), ("chunks", np.uint32), ("anc", np.uint8), ("codes", np.uint8)):
            nb = lib().dpq_program_size(h, name.encode())
            arr = np.empty(nb // np.dtype(dt).itemsize, dt)
            if nb:
                _check(lib().dpq_program_copy(h, name.encode(), _ptr(arr)))
            out[name] = arr
        for name in ("n_local", "base_pos", "rb", "levels", "n_bytes", "n_diffs", "n_chunks", "v2",
                     "v2_nf", "v2_lpg", "cstride"):
            out[name] = int(lib().dpq_program_size(h, name.encode()))
        out["chunks"] = out["chunks"].reshape(-1, 4)
        out["codes_padded"] = out["codes"].reshape(-1, max(out["cstride"], 1))
        out["codes"] = np.ascontiguousarray(out["codes_padded"][:, :M])
        out["anc"] = out["anc"].reshape(-1, out["levels"], M)
        out["M"], out["K"] = M, K
        return out
    finally:
        lib().dpq_program_free(h)
