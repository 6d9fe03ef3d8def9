#!/usr/bin/env python
"""bench.py -- queries/sec of the DeltaPQ query hot path (ADC tables -> DeltaTree scan ->
top-k) on B200, through libdpq.so's C ABI (include/dpq.h).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): SIFT1M-shaped synthetic, 1M x 128-d, M=8 K=256 h=1,
10K queries, top-10.  One step = one pass of the hot path over one batch of 10K queries.
The tree is produced by the product's own pipeline (GPU encode, GPU edge search, GPU DFS
layout + stream writer); only the cpu_baseline leg / --impl reference touch oracle/.

N > 1 (torchrun, one rank per GPU).  Primary number: the 16 MB tree is replicated and the
QUERIES are the sharded units (10K per GPU per step, weak scaling): independent batches, no
data-path collective.  Secondary block "tree_sharded": the same tree sharded by whole depth-1 subtrees
(SURVEY 8e, the 1B-code design), every rank scans its shard for the same 10K queries, the
per-rank top-k key lists are all-gathered over NCCL and merged on the device (strong scaling);
its merged result is checked against the unsharded one in the same run.
PyTorch is plumbing here (device buffers, stream, events, torch.distributed).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))  # datagen: synthetic data + file formats (tooling)

METRIC = "queries/sec @top10 on 1M-code DeltaTree (SIFT1M-shaped synthetic, M=8 K=256)"
UNIT = "queries/s"
WORKLOAD = ("SIFT1M-shaped synthetic 1Mx128 M=8 K=256 h=1, 10K queries per GPU per step, top-10 "
            "(BASELINE configs[1])")
N_CODES, N_QUERIES, DIM, PQ_M, PQ_K, TOPK = 1_000_000, 10_000, 128, 8, 256, 10


def synth(n_codes, n_queries):
    import datagen as dg
    base = dg.sift_like(n_codes, DIM, seed=1)
    learn = dg.sift_like(20000, DIM, seed=3)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(learn, PQ_M, PQ_K, iters=6))
    queries = dg.sift_like(n_queries, DIM, seed=2)
    return base, cw, queries


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                       "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        self.f.seek(0)
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 8:
                continue
            try:
                sm.append(float(c[1]))
                smax.append(float(c[2]))
                power.append(float(c[3]))
            except ValueError:
                continue
            for nm, v in zip(names, c[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # under load = samples at or above the median power draw
        med_p = float(np.median(power))
        load = [s for s, p in zip(sm, power) if p >= med_p] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": float(max(power))}


# ------------------------------------------------------------------------ reference arm --
_REF_STATE = {}


def _ref_init(payload, n_codes, cw):
    """Runs once in every worker process: the tree and codebook stay resident in the worker."""
    _REF_STATE["tree"] = (payload, n_codes, cw)


def _ref_worker(job):
    """One process = one single-threaded reference scanner (its globals are not thread safe)."""
    queries, topk = job
    payload, n_codes, cw = _REF_STATE["tree"]
    from oracle import pyoracle as po
    if po.have_ref():
        _, _, secs = po.ref_scan(payload, n_codes, cw, queries, topk)
        return secs
    t = time.perf_counter()
    for q in queries:
        po.scan(payload, n_codes, cw, q, topk)
    return time.perf_counter() - t


def cpu_reference_tree(base, cw):
    """CPU-only tree for the reference arm (oracle/ builder; same seeds => same tree)."""
    from oracle import pyoracle as po
    import multiprocessing as mp
    cores = len(os.sched_getaffinity(0))
    parts = np.array_split(base, max(1, cores))
    with mp.get_context("fork").Pool(cores) as pool:
        codes = np.concatenate(pool.starmap(po.encode, [(cw, p) for p in parts]))
    _, _, lay, payload = po.build_tree(codes, cw)
    return payload


def run_reference(args):
    """The reference's own CPU implementation of the path on all host cores: one persistent
    single-threaded scanner process per core (the reference's query function keeps its state in
    globals, so threads cannot share a process), started and warmed OUTSIDE the timed region; a
    step hands every scanner its slice of a bounded sample of the 10K-query batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    from oracle import pyoracle as po
    base, cw, queries = synth(args.n_codes, args.queries)
    payload = cpu_reference_tree(base, cw)
    del base
    cores = len(os.sched_getaffinity(0))
    per_proc = args.ref_queries_per_proc
    kind = "reference" if po.have_ref() else "port"
    n_step = cores * per_proc
    pool = mp.get_context("fork").Pool(cores, initializer=_ref_init, initargs=(payload, args.n_codes, cw))

    def step(i):
        # a different window of the query set every step (wraps around the 10K queries)
        idx = (np.arange(n_step) + i * n_step) % len(queries)
        qs = queries[idx]
        jobs = [(np.ascontiguousarray(qs[p * per_proc:(p + 1) * per_proc]), TOPK) for p in range(cores)]
        pool.map(_ref_worker, jobs, chunksize=1)

    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(args.steps):
        step(args.warmup + i)
    dt = time.perf_counter() - t0
    pool.close()
    pool.join()
    nq = n_step * args.steps
    qps = nq / dt
    sample = (f"{n_step} of the {args.queries} queries per step ({per_proc} per process, {cores} persistent "
              f"single-threaded reference scanners side by side: DCAT.h:3731 in-memory scan via oracle/_ref; "
              f"workers forked and warmed before the timed region)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "n_codes": args.n_codes, "queries_per_step": n_step, "topk": TOPK, "n_bytes": int(len(payload)),
                   "note": "same tree and query set as the GPU arm; each step is a bounded sample of the 10K-query batch"},
        "cpu_baseline": {"value": qps, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": qps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))
    return 0


# ------------------------------------------------------------------------ GPU arm -------
def timed_steps(torch, stream, flush, steps, step_fn, barrier):
    """K steps, device time per step; a 256 MiB write before every step flushes L2 (outside
    the events).  Returns the summed device milliseconds."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    for a, b in ev:
        flush.zero_()
        a.record(stream)
        step_fn()
        b.record(stream)
    barrier()
    return float(sum(a.elapsed_time(b) for a, b in ev))


def dump_outputs(out_dir, pos, ids, dist):
    """--dump-outputs: the top-k of the last timed step (all queries, rank 0's batch), as a caller of
    dpq_index_search receives it: DFS positions, vector ids (float64: every uint32 is exact) and
    distances (float32, as computed), one row per query in ascending distance.  Past 64 MB in all, a
    fixed seeded sample of the queries is kept and query_rows.npy names them.  The inputs are seeded,
    so two builds run with the same arguments can be compared array by array."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"positions": np.asarray(pos, np.float64), "ids": np.asarray(ids, np.float64),
              "distances": np.asarray(dist, np.float32)}
    row_bytes = sum(a[0].nbytes for a in arrays.values())
    max_rows = (64_000_000 - 4096) // (row_bytes + 8)  # 4 KB for the .npy headers
    if len(pos) > max_rows:
        rows = np.sort(np.random.default_rng(0).choice(len(pos), max_rows, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["query_rows"] = rows.astype(np.float64)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_gpu(args):
    import torch
    import deltapq_b200 as dpq

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not os.path.exists(dpq.LIB_PATH):
        raise SystemExit("libdpq.so is missing: run __graft_entry__.build() (no CPU fallback exists)")
    if dpq.device_count() < 1 or not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (libdpq has no CPU fallback)")
    torch.cuda.set_device(local)
    dpq.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    gloo = dist.new_group(backend="gloo") if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def host_barrier():  # waits on the CPU: the GPUs stay free for whoever works meanwhile
        torch.cuda.synchronize()
        dist.barrier(group=gloo)

    def max_over_ranks(*vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t.tolist()]

    # ---- workload: product pipeline only (encode -> approx_tree -> index) -----------------
    t_setup = time.perf_counter()
    base, cw, queries0 = synth(args.n_codes, args.queries)
    codes = dpq.encode(cw, base)
    tree = dpq.tree_build(codes, cw, h=1, method=1)
    payload = tree["payload"]
    del base
    Q, k = args.queries, TOPK
    stream = torch.cuda.current_stream()

    def open_index(r, n):
        ix_ = dpq.DeltaTreeIndex(payload, args.n_codes, PQ_M, PQ_K, pos2id=tree["vec_id"], rank=r, n_ranks=n)
        ix_.set_codebook(cw)
        for kv in (args.opts.split(",") if args.opts else []):
            kk, v = kv.split("=")
            ix_.set_option(kk, int(v))
        ix_.set_stream(stream.cuda_stream)
        return ix_

    # Primary mode.  The 1M-code tree is 16 MB on the device: every GPU holds the whole tree
    # and answers ITS OWN batch of 10K queries (the units of work are queries: weak scaling,
    # per-GPU batch fixed).  The batches are independent, so the primary step has no collective
    # (the exchange step of the path -- all-gather of key lists + merge -- is what the tree_sharded
    # and c5 blocks below measure).  N = 1 is the plain single-GPU run.
    ix = open_index(0, 1)
    t_setup = time.perf_counter() - t_setup
    if world > 1:
        import datagen as dg
        queries = dg.sift_like(Q, DIM, seed=2 + 1000 * rank)  # a different batch per rank
    else:
        queries = queries0
    d_q = torch.from_numpy(queries).to(dev)
    d_key = torch.empty((Q, k), dtype=torch.int64, device=dev)
    d_all = torch.empty((world, Q, k), dtype=torch.int64, device=dev) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step_device():
        ix.search_device(d_q.data_ptr(), Q, k, d_key.data_ptr())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)  # nvidia-smi start-up: the first sample must not land after the timed region
    for _ in range(args.warmup):
        flush.zero_()
        step_device()
    barrier()
    ix.set_option("timing_reset", 1)
    total_ms = timed_steps(torch, stream, flush, args.steps, step_device, barrier)
    scan_ns = ix.stat("sum_scan_ns")
    lut_ns = ix.stat("sum_lut_ns")
    calls = ix.stat("timed_calls")
    coarse = ix.stat("last_coarse") == 1
    scan8_ns = ix.stat("sum_scan8_ns") if coarse else 0
    fallback = ix.stat("last_fallback")
    launches_per_step = ix.stat("last_launches")

    # ---- e2e: the reference-facing C-ABI call dpq_index_search with HOST buffers (pinned staging
    # inside libdpq, H2D of the queries + D2H of the results inside the timed region)
    # The queries live in page-locked host memory (dpq_malloc_host), which libdpq copies from
    # directly; results land in ordinary numpy arrays.
    h_queries = dpq.pinned_array(queries.shape, np.float32)
    h_queries[...] = queries
    # caller-owned result arrays, reused; page-locked like the queries, so the last kernel of a search writes them
    # over PCIe itself (pageable arrays work too: staging buffer + three copies, ~50 us more per call)
    res = (dpq.pinned_array((Q, k), np.uint32), dpq.pinned_array((Q, k), np.uint32), dpq.pinned_array((Q, k), np.float32))
    pos, ids, dst = ix.search(h_queries, k, out=res)  # warm the pinned staging
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pos, ids, dst = ix.search(h_queries, k, out=res)
    barrier()
    e2e_s = time.perf_counter() - t0
    e2e_host = {"enqueue_us": ix.stat("last_host_enqueue_us"), "gpu_wait_us": ix.stat("last_host_wait_us"),
                "unpack_us": ix.stat("last_host_unpack_us")}
    clocks = sampler.stop() if rank == 0 else None
    total_ms, e2e_s, scan_ms_max = max_over_ranks(total_ms, e2e_s, scan_ns / 1e6)

    out_pos, out_dist = dpq.unpack_keys(d_key.cpu().numpy().view(np.uint64))
    assert np.all(np.diff(out_dist.astype(np.float64), axis=1) >= 0), "top-k not ascending"
    assert np.array_equal(out_dist, dst) and np.array_equal(out_pos, pos), "device and host paths disagree"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_pos, ids, out_dist)

    # ---- secondary mode at N > 1: the SAME tree sharded by depth-1 subtrees over the ranks
    # (SURVEY 8e, the 1B-code design): every rank scans its shard for the same 10K queries, one
    # NCCL all-gather of the local top-k keys, device merge.  Strong scaling on a 16 MB tree.
    tree_sharded = None
    if world > 1:
        sh = open_index(rank, world)
        d_q0 = torch.from_numpy(queries0).to(dev)
        d_loc = torch.empty((Q, k), dtype=torch.int64, device=dev)
        d_mrg = torch.empty((Q, k), dtype=torch.int64, device=dev)

        def step_sharded():
            sh.search_device(d_q0.data_ptr(), Q, k, d_loc.data_ptr())
            dist.all_gather_into_tensor(d_all.view(-1), d_loc.view(-1))
            sh.merge_device(d_all.data_ptr(), world, Q, k, d_mrg.data_ptr())

        for _ in range(args.warmup):
            flush.zero_()
            step_sharded()
        barrier()
        sh.set_option("timing_reset", 1)
        ms = timed_steps(torch, stream, flush, args.steps, step_sharded, barrier)
        sh_scan = sh.stat("sum_scan_ns") / 1e6 / max(sh.stat("timed_calls"), 1)
        ms, sh_scan = max_over_ranks(ms, sh_scan)
        # the merged result must equal the unsharded search of the same queries
        ix.search_device(d_q0.data_ptr(), Q, k, d_key.data_ptr())
        torch.cuda.synchronize()
        same = bool(torch.equal(d_key, d_mrg))
        tree_sharded = {"value": Q * args.steps / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / args.steps,
                        "scan_ms_max_over_ranks": sh_scan, "scaling": "strong", "equals_unsharded": same,
                        "n_local_nodes": sh.stat("n_local"),
                        "what": f"1M-code tree sharded by depth-1 subtrees over {world} GPUs, same 10K queries, "
                                f"NCCL all-gather of {Q * k * 8} B/rank + device merge"}
        assert same, "sharded + merged top-k differs from the unsharded result"
        sh.close()

    # ---- the C++ multi-GPU path (dpq_multi_*, NCCL bound at run time, no torch): rank 0 saves the tree and
    # runs tools/multi_probe.py in a SUBPROCESS with a timeout; the other ranks wait on the host
    multi_cpp = None
    if not args.no_multi_cpp:
        if rank == 0:
            import shutil
            tmpd = tempfile.mkdtemp(prefix="dpq_multi_")
            try:
                with open(os.path.join(tmpd, "tree.bin"), "wb") as f:
                    f.write(np.array([args.n_codes, len(payload)], np.int64).tobytes())
                    f.write(payload.tobytes())
                qn = np.zeros((args.n_codes + 1, 60), np.uint8)
                qn[:args.n_codes, 0:4] = tree["vec_id"].astype(np.uint32).view(np.uint8).reshape(-1, 4)
                qn.tofile(os.path.join(tmpd, "qnodes.bin"))
                del qn
                np.savez(os.path.join(tmpd, "multi_probe.npz"), cw=cw, queries=queries0, topk=k, n_codes=args.n_codes)
                r = subprocess.run([sys.executable, "-B", os.path.join(ROOT, "tools", "multi_probe.py"), tmpd, str(world), "5"],
                                   capture_output=True, text=True, timeout=420)
                last = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
                multi_cpp = json.loads(last[-1]) if last else {"error": (r.stderr or r.stdout)[-300:], "rc": r.returncode}
            except Exception as e:  # recorded, never fatal
                multi_cpp = {"error": repr(e)[:300]}
            finally:
                shutil.rmtree(tmpd, ignore_errors=True)
        if world > 1:
            host_barrier()

    # ---- C5: one tree over 10^9 codes, subtree shards over the ranks (own block, never fails the line)
    c5 = None
    if args.c5_codes > 0:
        t_c5 = time.perf_counter()
        try:
            del flush
            torch.cuda.empty_cache()
            c5 = c5_block(torch, dpq, dist, dev, rank, world, args, stream, barrier, max_over_ranks)
        except Exception as e:  # recorded, the primary line stands
            import traceback
            c5 = {"error": repr(e)[:300], "trace": traceback.format_exc()[-600:]}
        c5["block_s"] = round(time.perf_counter() - t_c5, 1)
        torch.cuda.empty_cache()

    n_bytes_total = ix.stat("n_bytes_total")
    peak, peak_src = measured_peak()
    # algorithmic bytes of one scan launch (SURVEY 8d): Q queries x (stream bytes + 4 D query
    # floats + 8 k result bytes)
    alg_bytes = Q * (ix.stat("n_bytes") + 4 * DIM + 8 * k)
    scan_s = (scan_ns / 1e9) / max(calls, 1)
    # dominant kernel: the coarse scan (one launch = all Q queries over the whole tree) when the
    # three-phase search ran, else the 15-bit scan
    dom_s = (scan8_ns / 1e9) / max(calls, 1) if coarse else scan_s
    dom_name = "scan8_kernel" if coarse else ("scan2_kernel" if ix.stat("engine") == 2 else "scan_kernel")
    achieved = alg_bytes / dom_s / 1e9
    qps = world * Q * args.steps / (total_ms / 1e3)
    e2e_qps = world * Q * args.steps / e2e_s

    if rank == 0:
        cpu_base, parity = None, None
        if world == 1 and not args.no_cpu_baseline:
            cpu_base, parity = cpu_baseline(payload, args.n_codes, cw, queries, args.cpu_baseline_queries, out_pos, out_dist)
        elif not args.no_cpu_baseline:
            # N > 1: the CPU baseline is an N = 1 number, the parity check is not: rank 0's answers for a short
            # sample of its own batch against the reference CPU scan (about a second; the other ranks wait)
            _, parity = cpu_baseline(payload, args.n_codes, cw, queries, min(100, args.cpu_baseline_queries), out_pos, out_dist)
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "scan_traffic.json")
        if os.path.exists(tpath):
            try:
                traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        # Roofline of the dominant kernel.  The coarse scan is bound by the shared-memory / LSU data
        # pipe, not by HBM (the 8 MB code array is L2 resident and one pass serves 112 queries):
        # every (node, 112-query group) costs 8 table-row reads = 8 shared-memory wavefronts of 128 B,
        # one wavefront per clock per SM.  achieved = algorithmic wavefront bytes / kernel time; peak =
        # 148 SMs x 128 B x SM clock (sampled under load).  The SURVEY 8d figure (stream bytes x
        # queries: an EFFECTIVE bandwidth that grows with the batch) and the physical DRAM traffic are
        # reported beside it under their own names.
        n_local = ix.stat("n_local")
        qpg = 112 if coarse else 56
        groups = (Q + qpg - 1) // qpg
        wf_per_node = 8
        alg_wavefronts = n_local * groups * wf_per_node
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        lsu_peak = 148 * 128 * sm_mhz * 1e6 / 1e9  # GB/s of shared-memory wavefronts
        lsu_achieved = alg_wavefronts * 128 / dom_s / 1e9
        line = {
            "metric": METRIC, "value": qps, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8 coarse filter + u16 fixed-point sample + f64 exact re-score",
            "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "n_codes": args.n_codes, "queries_per_step": world * Q, "topk": k, "n_bytes": n_bytes_total,
                       "mean_diffs_per_node": round((n_bytes_total - 8 - (3 * (args.n_codes - 1) + 1) // 2) / (args.n_codes - 1), 3),
                       "depth_hist": [ix.stat(f"depth_hist_{d}") for d in range(9)],
                       "device_bytes_per_node": ix.stat("device_bytes_per_node"),
                       "disk_bytes_per_node": round(n_bytes_total / args.n_codes, 3),
                       "sharding": "whole tree on one GPU" if world == 1 else
                                   f"queries sharded: {world} replicas of the tree, {Q} independent queries per GPU per step, no data-path collective",
                       "l2": "256 MiB buffer written before every timed step (L2 flush, outside the events)",
                       "tree": "built by libdpq (GPU encode + GPU edge search + GPU DFS layout and stream)",
                       "setup_s": round(t_setup, 1), "opts": args.opts or "default"},
            "roofline": {"bound": "smem_lsu", "achieved": lsu_achieved, "peak": lsu_peak, "unit": "GB/s",
                         "frac": lsu_achieved / lsu_peak, "traffic": traffic, "kernel": dom_name,
                         "kernel_ms_per_launch": dom_s * 1e3,
                         "algorithmic_wavefronts_per_launch": alg_wavefronts,
                         "wavefronts_per_node_per_group": wf_per_node, "queries_per_group": qpg,
                         "peak_source": f"148 SMs x 128 B/clk x {sm_mhz:.0f} MHz (nvidia-smi under load); one shared-memory wavefront per clock per SM",
                         "effective_hbm_gbs": achieved, "effective_hbm_x_peak": achieved / peak,
                         "hbm_peak_gbs": peak, "hbm_peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "dram_gbs": (traffic / dom_s / 1e9) if traffic else None,
                         "note": "per GPU. frac = shared-memory wavefronts the algorithm needs / kernel time / pipe peak. "
                                 "effective_hbm_* = SURVEY 8d bytes (Q x (stream bytes + 4D + 8k)) / kernel time: above 1 because one "
                                 "L2-resident pass serves 112 queries; traffic / dram_gbs = physical DRAM bytes per launch from the "
                                 "committed ncu capture (profiles/scan_traffic.json)"},
            "cpu_baseline": cpu_base,
            "parity": parity,
            "e2e": {"value": e2e_qps, "unit": UNIT, "h2d_bytes_per_step": world * Q * DIM * 4,
                    "d2h_bytes_per_step": world * Q * k * 8, "host_breakdown_last_call": e2e_host,
                    "how": "dpq_index_search with the queries and the caller's result arrays in page-locked host memory: the kernels "
                           "read the queries and write positions / ids / distances through the device mapping of that memory "
                           "(PCIe traffic inside the timed region), one stream sync"},
            "gpu_launches": int(launches_per_step * args.steps),
            "clocks": clocks,
            "breakdown_ms_per_step": {"lut": lut_ns / 1e6 / max(calls, 1), "all_scan_phases": scan_s * 1e3,
                                      "coarse_scan_kernel": dom_s * 1e3 if coarse else None,
                                      "scan_max_over_ranks": scan_ms_max / max(calls, 1), "exact_fallback_queries": fallback},
            "tree_sharded": tree_sharded,
            "multi_cpp": multi_cpp,
            "c5": c5,
        }
        print(json.dumps(line))
        if parity is not None and not parity["ok"]:
            raise SystemExit("parity check against the reference CPU scan FAILED: " + str(parity.get("why")))
    ix.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------ C5: 10^9 codes --
def gen_codes_device(torch, dpq, dev, cw, n, seed, out, chunk=1 << 21):
    """SIFT-like bvecs-shaped vectors (tests/datagen.sift_like's mixture, drawn with torch on the
    device: integer components 0..255) -> codes [n][8] written into `out` (a device uint8 tensor),
    never storing the vectors."""
    n_clusters, sigma, nb, w = 256, 14.0, DIM // 16, 16
    crng = np.random.default_rng(1234567)  # the centres of datagen.sift_like
    centres = torch.from_numpy(np.clip(crng.gamma(2.0, 22.0, size=(nb, n_clusters, w)), 0, 255)).to(dev, torch.float32)
    pop = 1.0 / np.arange(1, n_clusters + 1) ** 0.7
    pop = torch.from_numpy(pop / pop.sum()).to(dev, torch.float32)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    for s_ in range(0, n, chunk):
        c = min(chunk, n - s_)
        x = torch.empty((c, DIM), dtype=torch.float32, device=dev)
        for b in range(nb):
            cid = torch.multinomial(pop, c, replacement=True, generator=g)
            blk = centres[b][cid] + sigma * torch.randn((c, w), device=dev, generator=g)
            x[:, b * w:(b + 1) * w] = blk.round_().clamp_(0, 255)
        dpq.encode_device(cw, x.data_ptr(), c, DIM, out[s_:].data_ptr())
        del x
    torch.cuda.synchronize()


def plain_adc_topk_device(torch, dpq, cw, codes_dev, queries, k, slab=1 << 27):
    """Exact top-k of plain ADC over ALL codes for a few queries (float table entries, double sum =
    the reference's arithmetic), on the device in slabs: [(dist float32 [k], vector id int64 [k])]."""
    tabs = dpq.adc_tables(cw, queries)  # [q][M][K] float32
    out = []
    n = codes_dev.shape[0]
    for t in tabs:
        tt = torch.from_numpy(t).to(codes_dev.device, torch.float64)
        best_d, best_i = None, None
        for s_ in range(0, n, slab):
            blk = codes_dev[s_:s_ + slab]
            d = torch.zeros(blk.shape[0], dtype=torch.float64, device=codes_dev.device)
            for m in range(PQ_M):
                d += tt[m][blk[:, m].long()]
            d32 = d.to(torch.float32)
            v, i = torch.topk(d32, min(4 * k, d32.shape[0]), largest=False, sorted=True)
            i = i + s_
            best_d = v if best_d is None else torch.cat([best_d, v])
            best_i = i if best_i is None else torch.cat([best_i, i])
            del d, d32, blk
        bd, bi = best_d.cpu().numpy(), best_i.cpu().numpy().astype(np.int64)
        order = np.lexsort((bi, bd))[:4 * k]
        out.append((bd[order], bi[order]))
    return out


def c5_block(torch, dpq, dist, dev, rank, world, args, stream, barrier, max_over_ranks):
    """BASELINE configs[4] / north_star: ONE DeltaTree over 10^9 SIFT1B-shaped codes, sharded by
    whole depth-1 subtrees over the GPUs (SURVEY 8e), local top-k per GPU with global positions, one
    NCCL all-gather of Q x k keys per rank, device merge.  Every rank builds the same tree on its own
    GPU (the build is a global sort: replicas, DESIGN.md section 6) and keeps only its shard."""
    import datagen as dg
    n_total, Q, k = args.c5_codes, args.queries, TOPK
    out = {"n_codes": n_total, "queries_per_step": Q, "topk": k}
    t0 = time.perf_counter()
    learn = dg.sift_like(20000, DIM, seed=3)
    cw = dg.roundtrip_codebook(dg.kmeans_codebook(learn, PQ_M, PQ_K, iters=6))
    queries = dg.sift_like(Q, DIM, seed=2)
    torch.cuda.empty_cache()
    setup_err = None
    try:
        codes = torch.empty((n_total, PQ_M), dtype=torch.uint8, device=dev)
    except Exception as e:  # out of memory: every rank must agree to skip before any collective
        setup_err = repr(e)[:200]
    if world > 1:
        flag = torch.tensor([1.0 if setup_err else 0.0], device=dev)
        dist.all_reduce(flag)
        if float(flag[0]) > 0:
            return {"error": "setup failed on some rank: " + str(setup_err)}
    elif setup_err:
        return {"error": "setup failed: " + setup_err}
    n_gen = 8  # generated in 8 seeded pieces (the same data for every world size)
    for p in range(n_gen):
        lo, hi = n_total * p // n_gen, n_total * (p + 1) // n_gen
        gen_codes_device(torch, dpq, dev, cw, hi - lo, 1000 + p, codes[lo:hi])
    t1 = time.perf_counter()
    nq_chk = min(args.c5_check_queries, Q)
    truth = plain_adc_topk_device(torch, dpq, cw, codes, queries[:nq_chk], k) if nq_chk else []
    torch.cuda.empty_cache()
    t2 = time.perf_counter()
    tree = dpq.DeviceTree(codes.data_ptr(), n_total, PQ_M, cw)
    t3 = time.perf_counter()
    del codes
    torch.cuda.empty_cache()
    ix = tree.shard(rank, world)
    ix.set_codebook(cw)
    ix.set_stream(stream.cuda_stream)
    n_bytes = tree.stat("payload")
    n_diffs = tree.stat("n_diffs")
    out["setup_s"] = {"gen_encode": round(t1 - t0, 1), "plain_adc_truth": round(t2 - t1, 1),
                      "edge_search": round(tree.stat("edge_us") / 1e6, 1), "layout_stream": round(tree.stat("layout_us") / 1e6, 1),
                      "open_shard": round(time.perf_counter() - t3, 1)}
    out["tree"] = {"n_bytes": n_bytes, "disk_bytes_per_node": round(n_bytes / n_total, 3),
                   "mean_diffs_per_node": round(n_diffs / max(n_total - 1, 1), 3),
                   "depth_hist": [tree.stat(f"depth_hist_{d}") for d in range(9)],
                   "device_bytes_per_node": ix.stat("device_bytes_per_node"),
                   "built": "one tree over all codes by dpq_tree_build_device on every rank's GPU (edge search + layout + stream, "
                            "nothing leaves HBM); shard = whole depth-1 subtrees balanced by stream bytes"}
    # rank 0 at N = 1 keeps the stream for the reference CPU sample and the ids of the check queries
    payload = tree.fetch("payload", np.uint8) if (rank == 0 and world == 1 and args.c5_ref_queries > 0) else None
    vec_id = tree.fetch("vec_id", np.uint32) if nq_chk else None
    tree.free()
    torch.cuda.empty_cache()

    d_q = torch.from_numpy(queries).to(dev)
    d_loc = torch.empty((Q, k), dtype=torch.int64, device=dev)
    d_all = torch.empty((world, Q, k), dtype=torch.int64, device=dev)
    d_mrg = torch.empty((Q, k), dtype=torch.int64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        ix.search_device(d_q.data_ptr(), Q, k, d_loc.data_ptr())
        if world > 1:
            dist.all_gather_into_tensor(d_all.view(-1), d_loc.view(-1))
            ix.merge_device(d_all.data_ptr(), world, Q, k, d_mrg.data_ptr())
        else:
            d_mrg.copy_(d_loc)

    steps = max(1, min(args.steps, args.c5_steps))
    for _ in range(3):
        flush.zero_()
        step()
    barrier()
    ix.set_option("timing_reset", 1)
    total_ms = timed_steps(torch, stream, flush, steps, step, barrier)
    calls = max(ix.stat("timed_calls"), 1)
    scan8_ms = ix.stat("sum_scan8_ns") / 1e6 / calls
    scan_ms = ix.stat("sum_scan_ns") / 1e6 / calls
    lut_ms = ix.stat("sum_lut_ns") / 1e6 / calls
    ix.sync()
    fallback = ix.stat("last_fallback")
    n_local = ix.stat("n_local")
    (total_ms, scan8_max) = max_over_ranks(total_ms, scan8_ms)
    # e2e: host buffers through dpq_index_search on the shard, keys gathered and merged
    h_q = dpq.pinned_array(queries.shape, np.float32)
    h_q[...] = queries
    barrier()
    te = time.perf_counter()
    pos, ids, dst = ix.search(h_q, k)
    if world > 1:
        keys = (dst.view(np.uint32).astype(np.uint64) << np.uint64(32)) | pos
        d_keys = torch.from_numpy(keys.view(np.int64)).to(dev)
        dist.all_gather_into_tensor(d_all.view(-1), d_keys.view(-1))
        ix.merge_device(d_all.data_ptr(), world, Q, k, d_mrg.data_ptr())
        _ = d_mrg.cpu()
    barrier()
    (e2e_s,) = max_over_ranks(time.perf_counter() - te)

    step()
    torch.cuda.synchronize()
    mpos, mdist = dpq.unpack_keys(d_mrg.cpu().numpy().view(np.uint64))
    ok = bool(np.all(np.diff(mdist.astype(np.float64), axis=1) >= 0))
    check = None
    if nq_chk:
        same = True
        for q in range(nq_chk):
            td, ti = truth[q]
            same &= bool(np.array_equal(td[:k], mdist[q]))
            kth = td[k - 1]
            got = {int(vec_id[p_]) for p_, d_ in zip(mpos[q], mdist[q]) if d_ < kth}
            want = {int(i_) for i_, d_ in zip(ti, td) if d_ < kth}
            same &= got == want
        check = {"queries": nq_chk, "equals_plain_adc_over_all_codes": bool(same)}
        ok &= bool(same)
    qps = Q * steps / (total_ms / 1e3)
    out.update({"value": qps, "unit": UNIT, "ms_per_step": total_ms / steps, "steps": steps, "warmup": 3,
                "scaling": "strong", "n_local_nodes_rank0": n_local,
                "sharding": f"one tree, {world} shard(s) of whole depth-1 subtrees; same {Q} queries on every shard; "
                            f"NCCL all-gather of {Q * k * 8} B/rank + device merge",
                "e2e": {"value": Q / e2e_s, "unit": UNIT, "h2d_bytes_per_step": world * Q * DIM * 4,
                        "d2h_bytes_per_step": world * Q * k * 8},
                "breakdown_ms_per_step": {"lut": lut_ms, "all_scan_phases": scan_ms, "coarse_scan_kernel_max_over_ranks": scan8_max,
                                          "exact_fallback_queries": fallback},
                "check": check, "ok": ok})
    groups = (Q + 111) // 112
    sm_mhz = 1965.0
    out["roofline"] = {"bound": "smem_lsu", "kernel": "scan8_kernel", "kernel_ms_per_launch": scan8_ms,
                       "achieved": n_local * groups * 8 * 128 / (scan8_ms / 1e3) / 1e9, "peak": 148 * 128 * sm_mhz * 1e6 / 1e9,
                       "unit": "GB/s", "frac": (n_local * groups * 8 * 128 / (scan8_ms / 1e3) / 1e9) / (148 * 128 * sm_mhz * 1e6 / 1e9),
                       "hbm_floor_ms": n_local * 8 / 6553e9 * 1e3 * groups,
                       "note": "rank 0's shard; one pass of the 8 B/node code array per 112-query group"}
    if payload is not None:
        from oracle import pyoracle as po
        from helpers import assert_topk_equal
        nq = args.c5_ref_queries
        kind = "reference" if po.have_ref() else "port"
        tq = time.perf_counter()
        if kind == "reference":
            rpos, rdist, secs = po.ref_scan(payload, n_total, cw, np.ascontiguousarray(queries[:nq]), k)
        else:
            rpos = np.empty((nq, k), np.int32)
            rdist = np.empty((nq, k), np.float32)
            for i in range(nq):
                rpos[i], rdist[i] = po.scan(payload, n_total, cw, queries[i], k)
            secs = time.perf_counter() - tq
        rpos = np.where(rpos == n_total, n_total - 1, rpos)
        pok, why = True, None
        try:
            assert_topk_equal(mpos[:nq], mdist[:nq], rpos, rdist)
        except AssertionError as e:
            pok, why = False, str(e)[:300]
        out["cpu_baseline"] = {"value": nq / secs, "unit": UNIT, "cores": 1, "kind": kind,
                               "sample": f"{nq} queries over the same {n_total}-code tree, in-memory scan (DCAT.h:3731), 1 thread, {secs:.1f} s"}
        out["parity"] = {"queries": nq, "ok": pok, "dist_bit_equal": bool(np.array_equal(mdist[:nq], rdist)),
                         "against": kind + " CPU scan of the same queries on the same tree"}
        if why:
            out["parity"]["why"] = why
        out["ok"] = bool(out["ok"] and pok)
    ix.close()
    return out


def cpu_baseline(payload, n_codes, cw, queries, n_q, gpu_pos, gpu_dist):
    """The reference's own CPU scan (oracle/_ref when it was built, else the oracle port) on a
    bounded sample of the same workload, one thread (the reference query path is single
    threaded by design).  Its results are the parity check of THIS run: the GPU's top-k for the
    same queries on the same tree must match them (distances within 1e-5 relative -- bit-equal
    on this integer-valued data -- ids modulo ties at 1e-5: tests/helpers.assert_topk_equal)."""
    from oracle import pyoracle as po
    from helpers import assert_topk_equal, REL_TOL
    kind = "reference" if po.have_ref() else "port"
    qs = np.ascontiguousarray(queries[:n_q])
    t = time.perf_counter()
    if kind == "reference":
        rpos, rdist, secs = po.ref_scan(payload, n_codes, cw, qs, TOPK)
    else:
        rpos = np.empty((n_q, TOPK), np.int32)
        rdist = np.empty((n_q, TOPK), np.float32)
        for i, q in enumerate(qs):
            rpos[i], rdist[i] = po.scan(payload, n_codes, cw, q, TOPK)
        secs = time.perf_counter() - t
    # the reference reports the trailing node of an even-N tree at position N (SURVEY App. C.1)
    rpos = np.where(rpos == n_codes, n_codes - 1, rpos)
    g_d = gpu_dist[:n_q].astype(np.float64)
    r_d = rdist.astype(np.float64)
    max_rel = float(np.max(np.abs(g_d - r_d) / np.maximum(np.abs(r_d), 1e-30)))
    ok, why = True, None
    try:
        assert_topk_equal(gpu_pos[:n_q], gpu_dist[:n_q], rpos, rdist)
    except AssertionError as e:  # reported in the line, then the run fails
        ok, why = False, str(e)[:300]
    parity = {"queries": int(n_q), "ok": ok, "max_rel": max_rel, "tol": REL_TOL,
              "dist_bit_equal": bool(np.array_equal(gpu_dist[:n_q], rdist)),
              "ids_equal_modulo_ties": ok, "against": kind + " CPU scan of the same queries on the same tree"}
    if why:
        parity["why"] = why
    base = {"value": n_q / secs, "unit": UNIT, "cores": 1, "kind": kind,
            "sample": f"first {n_q} of the {len(queries)} queries on the same 1M-code tree, in-memory scan "
                      f"(DCAT.h:3731), 1 thread, {secs:.1f} s"}
    return base, parity


class StdoutToStderr:
    """Everything libraries print on fd 1 while the bench runs (e.g. NCCL's version banner) goes
    to stderr; stdout carries exactly the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


def main():
    sys.dont_write_bytecode = True  # the bench leaves the source tree as it found it (it may be read-only)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="dpq", choices=["dpq", "reference"])
    ap.add_argument("--n-codes", type=int, default=N_CODES)
    ap.add_argument("--queries", type=int, default=N_QUERIES)
    ap.add_argument("--opts", default="", help="libdpq tuning options, e.g. pack=2,warps=16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-baseline-queries", type=int, default=600)
    ap.add_argument("--ref-queries-per-proc", type=int, default=100)
    ap.add_argument("--no-multi-cpp", action="store_true", help="skip the C++ multi-GPU probe (tools/multi_probe.py)")
    ap.add_argument("--c5-codes", type=int, default=1_000_000_000,
                    help="codes of the single-tree C5 block (0 = skip the block)")
    ap.add_argument("--c5-steps", type=int, default=3)
    ap.add_argument("--c5-check-queries", type=int, default=4)
    ap.add_argument("--c5-ref-queries", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the top-k of the last timed step to DIR/{positions,ids,distances}.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    if args.warmup < 3:
        args.warmup = 3
    holder = []
    real_print = print

    def capture(*a, **k):  # run_* print their JSON line last; emit it after fd 1 is restored
        holder.append(" ".join(str(x) for x in a))

    with StdoutToStderr():
        import builtins
        builtins.print = capture
        try:
            rc = run_reference(args) if args.impl == "reference" else run_gpu(args)
        finally:
            builtins.print = real_print
    for line in holder:
        real_print(line, flush=True)
    return rc


if __name__ == "__main__":
    sys.exit(main())
