#!/usr/bin/env python
"""bench.py -- batched Cobweb predict throughput on B200 (see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference] [--workload cfg1|cfg2|cfg3|cfg4]
                  [--mode fused|fp32] [--shard query|store] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic queries: dense cobweb_predict_fast
semantics (every query against every node, path product, top-k) on a tree built by the engine's own
ifit from synthetic embeddings of the BASELINE.json shape.  One JSON line on stdout (rank 0).  Under
torchrun the node store is built on rank 0 and broadcast over NCCL, each rank answers its own batch
(weak scaling) and the results are all-gathered on the device inside the timed step.

--dump-outputs DIR writes the ids and scores of the last timed step as DIR/<name>.npy.  The inputs are seeded, so
two builds of the project run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it (it may be read-only)
DUMP_MAX_BYTES = 64 * 10**6

WORKLOADS = {
    # name: (docs, dim, queries per GPU, k, corpus kind, BASELINE.json config it is)
    "cfg1": (1000, 384, 100, 10, "unit", "configs[0] 1,000 docs x 384-d (MiniLM shape), 100 queries"),
    "cfg2": (1500, 1024, 300, 10, "unit", "configs[1] QQP-shape 1,500 docs x 1024-d, 300 queries"),
    "cfg3": (100000, 768, 10000, 10, "unit", "configs[2] MS-MARCO-shape 100k passages x 768-d, 10k-query batch"),
    "cfg4": (1000000, 1024, 16384, 10, "unit", "configs[3] 1M docs x 1024-d, query batches sharded over GPUs"),
}
GOLDEN = {"cfg1": "cfg1_unit_1000x384", "cfg2": "cfg2_unit_1500x1024"}


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def dump_outputs(out_dir, ids, scores):
    """The last timed step's answer as out_dir/ids.npy (float64: exact for any sentence id) and out_dir/scores.npy
    (float32).  A batch beyond DUMP_MAX_BYTES in all is cut to a fixed seeded sample of its query rows, whose row
    numbers go to out_dir/rows.npy."""
    arrays = {"ids": np.asarray(ids, np.float64), "scores": np.asarray(scores, np.float32)}
    n = len(arrays["ids"])
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    budget = DUMP_MAX_BYTES - 3 * 1024  # the .npy headers
    if n * row_bytes > budget:
        rows = np.sort(np.random.default_rng(0).choice(n, budget // (row_bytes + 8), replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"[bench] outputs of the last timed step -> {out_dir}: " + ", ".join(f"{k} {a.shape}" for k, a in arrays.items()))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for j, nm in enumerate(names) if any(len(r) >= 7 and r[3 + j].lower() == "active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def build_tree(docs, dim, kind):
    """Setup (untimed): synthetic corpus -> engine ifit on the device.  Returns (wrapper, x, secs)."""
    import torch
    from rag_cobweb_b200 import CobwebWrapper, synth
    x = synth.corpus(docs, dim, kind, seed=0)
    xd = torch.from_numpy(x).cuda()  # the instances are resident in HBM when the timed build starts
    # one-time costs out of the way (library + CUDA module load, first allocations): a 64-row tree that is thrown away
    CobwebWrapper(corpus=[None] * 64, corpus_embeddings=xd[:64].clone())
    torch.cuda.synchronize()
    t0 = time.time()
    w = CobwebWrapper(corpus=[None] * docs, corpus_embeddings=xd)
    torch.cuda.synchronize()
    return w, x, time.time() - t0


def oracle_from_engine(w):
    """Load the engine-built tree into the CPU oracle (setup for the CPU baseline legs and the parity block)."""
    from oracle.cobweb_oracle import OracleTree
    b = w.tree.bfs()
    mean, m2 = w.tree.store.rows(b["order"])
    t = OracleTree(w.tree.d)
    t.load(b["parent"], b["count"], b["nsent"], mean, m2)
    pos = np.full(int(b["order"].max()) + 1, -1, np.int64)
    pos[b["order"]] = np.arange(len(b["order"]))
    t.leaf_of_sentence = pos[w._leaf_of_sentence].astype(np.int32)
    t.n_sentences = len(t.leaf_of_sentence)
    t.build_index()
    return t


def oracle_topk(ot, q, k):
    """The oracle's dense predict for a few queries: (ids [nq, k], scores [nq, k]), ties by sentence id."""
    from oracle.cobweb_oracle import leaf_scores, topk
    ns, _ = ot.dense_scores(q, fast=True)
    ls = leaf_scores(ns, ot.index["path_idx"], ot.index["path_w"])
    out = [topk(row, k) for row in ls]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])


def cpu_predict_rate(ot, q, k, min_seconds=3.0, max_rounds=50):
    """queries/s of the oracle port's dense predict (OpenMP over the threads set by oracle.set_threads)."""
    done, t0 = 0, time.time()
    while True:
        oracle_topk(ot, q, k)
        done += len(q)
        if time.time() - t0 >= min_seconds or done >= max_rounds * len(q):
            break
    return done / (time.time() - t0)


def host_threads():
    """All the host threads the CPU arm may use -- set explicitly: torchrun exports OMP_NUM_THREADS=1."""
    from oracle import cobweb_oracle
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return cobweb_oracle.set_threads(n)


def run_reference(args, wl):
    """--impl reference: the reference's CPU implementation of the path (oracle port, since the
    Python reference cannot travel to this box) on the host cores, same config and metric."""
    docs, dim, qn, k, kind, cfg = wl
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from rag_cobweb_b200 import synth
    cores = host_threads()
    sample = 16
    w, x, build_s = build_tree(docs, dim, kind)
    ot = oracle_from_engine(w)
    q, _ = synth.queries(x, sample, kind, seed=1)
    for _ in range(max(args.warmup, 1)):
        cpu_predict_rate(ot, q, k, min_seconds=0.0, max_rounds=1)
    t0 = time.time()
    for _ in range(args.steps):
        ids, scores = oracle_topk(ot, q, k)
    dt = time.time() - t0
    v = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": "cobweb_predict_fast queries/sec", "value": v, "unit": "queries/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg, "docs": docs, "dim": dim, "k": k, "queries_per_step": sample,
                   "note": "per-query throughput on a bounded sample: %d queries per step against all nodes (the engine arm "
                           "answers %d per step)" % (sample, qn),
                   "tree": "built by the engine's ifit in setup, loaded into the CPU port"},
        "cpu_baseline": {"value": v, "unit": "queries/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} queries per step against all {ot.index['means'].shape[0]} nodes, OpenMP, "
                                   f"{cores} threads set explicitly"},
        "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ids, scores)
    print(json.dumps(line), flush=True)


def run_engine(args, wl):
    # keep stdout clean for the single JSON line: libraries (NCCL's version banner) write to fd 1
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = _run_engine(args, wl)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if line is not None:
        print(json.dumps(line), flush=True)


def reference_tree_parity(name, k=10):
    """configs[0] / configs[1]: the REFERENCE's tree (its recorded decisions replayed by the oracle, fixture
    tests/golden/<name>.npz) beside the tree the engine builds by itself from the same rows, both queried by the
    engine: recall@k of each and how far the two answer lists agree.  The two trees differ at the decisions the
    fixture marks as summation noise of the reference (DESIGN.md section 3)."""
    import torch
    from oracle.cobweb_oracle import OracleTree
    from rag_cobweb_b200 import CobwebWrapper, synth
    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    if not os.path.exists(path):
        return None
    g = np.load(path)
    n, d, kind = int(g["n"]), int(g["d"]), str(g["kind"])
    x = synth.corpus(n, d, kind, seed=0)
    nq = min(300, n)
    q, targets = synth.queries(x, nq, kind, seed=1)
    ref = OracleTree(d)
    dec = g["ops"][g["ops"] < 4]
    leaves, _, st = ref.ifit_guided(x, dec, g["dec_b1"], g["dec_b2"])
    rb = ref.bfs()
    assert np.array_equal(rb["parent"], g["bfs_parent"]) and np.array_equal(rb["count"], g["bfs_count"]), "replayed tree != fixture"
    mean, m2 = ref.rows(rb["order"])
    w_ref = CobwebWrapper(corpus=[None], corpus_embeddings=torch.from_numpy(x[:1]).cuda())
    w_ref.tree.load_arrays(rb["parent"], rb["count"], rb["nsent"], mean, m2)
    pos = np.full(int(rb["order"].max()) + 1, -1, np.int64)
    pos[rb["order"]] = np.arange(len(rb["order"]))
    w_ref.sentences, w_ref._leaf_of_sentence = [None] * n, pos[leaves].astype(np.int32)
    w_ref._invalidate_prediction_index()
    w_eng = CobwebWrapper(corpus=[None] * n, corpus_embeddings=torch.from_numpy(x).cuda())
    ids_r = w_ref.predict_fast_batch(q, k)[0].cpu().numpy()
    ids_e = w_eng.predict_fast_batch(q, k)[0].cpu().numpy()
    rec = lambda ids: float(np.mean([t in g_ for t, g_ in zip(targets, ids)]))
    return {"fixture": name, "docs": n, "dim": d, "queries": nq, "recall_at_k_reference_tree": rec(ids_r),
            "recall_at_k_engine_tree": rec(ids_e), "nodes_reference_tree": int(len(rb["order"])),
            "nodes_engine_tree": int(len(w_eng.tree.bfs()["order"])),
            "top1_agreement": float(np.mean(ids_r[:, 0] == ids_e[:, 0])),
            "topk_overlap": float(np.mean([len(set(a) & set(b)) / k for a, b in zip(ids_r, ids_e)]))}


def _run_engine(args, wl):
    import torch
    import torch.distributed as dist
    from rag_cobweb_b200 import _lib, parallel, synth
    docs, dim, qn, k, kind, cfg = wl
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    peaks, peak_src = measured_peaks()

    # ---------------------------------------------------------------- setup (untimed)
    if rank == 0 and args.snapshot and os.path.exists(args.snapshot):
        # a tree built by an earlier run of this bench on this box (the 1M-document build takes minutes): same tree
        from rag_cobweb_b200 import CobwebWrapper
        t0 = time.time()
        w = CobwebWrapper.load_snapshot(args.snapshot)
        x = synth.corpus(docs, dim, kind, seed=0)
        meta = json.load(open(args.snapshot + ".json"))
        assert (meta["docs"], meta["dim"], meta["kind"]) == (docs, dim, kind) and len(w.sentences) == docs, "snapshot of another workload"
        build_s, counters = meta["build_s"], meta["counters"]
        log(f"[bench] snapshot {args.snapshot} loaded in {time.time() - t0:.1f}s (built in {build_s:.1f}s)")
    elif rank == 0:
        w, x, build_s = build_tree(docs, dim, kind)
        counters = w.tree.store.counters()
        log(f"[bench] ifit {docs}x{dim}: {build_s:.1f}s = {docs / build_s:.0f} inserts/s")
        if args.snapshot:
            t0 = time.time()
            w.save_snapshot(args.snapshot)
            json.dump({"docs": docs, "dim": dim, "kind": kind, "build_s": build_s, "counters": counters}, open(args.snapshot + ".json", "w"))
            log(f"[bench] snapshot written to {args.snapshot} in {time.time() - t0:.1f}s")
    else:
        from rag_cobweb_b200 import CobwebWrapper
        x = synth.corpus(docs, dim, kind, seed=0)
        w = CobwebWrapper(corpus=[None], corpus_embeddings=torch.from_numpy(x[:1]).cuda())
        build_s, counters = None, None
    if world > 1:
        t0 = time.time()
        parallel.broadcast_store(w.tree, src=0)
        leaf = torch.from_numpy(w._leaf_of_sentence if rank == 0 else np.zeros(docs, np.int32)).cuda()
        dist.broadcast(leaf, 0)
        w._leaf_of_sentence = leaf.cpu().numpy()
        w.sentences = [None] * docs
        w._invalidate_prediction_index()
        torch.cuda.synchronize()
        log(f"[bench] rank {rank}: store broadcast {time.time() - t0:.2f}s")
    w.set_dense_mode(args.mode)
    torch.cuda.synchronize()
    t0 = time.time()
    w.build_prediction_index()
    torch.cuda.synchronize()
    index_build_s = time.time() - t0
    ix = w._index
    fused = ix.fused_ready(k)  # small index / large k: the engine answers on the FP32 pipe whatever the mode
    # this rank's batch: global batch = world * qn, contiguous shards
    q_all, targets_all = synth.queries(x, qn * world, kind, seed=1, targets=np.arange(qn * world) % docs)
    lo, hi = parallel.shard_bounds(qn * world, world, rank)
    q_host = torch.from_numpy(q_all[lo:hi]).pin_memory()
    q_dev = q_host.cuda()
    out_sid_h = torch.empty((qn, k), dtype=torch.int32).pin_memory()
    out_val_h = torch.empty((qn, k), dtype=torch.float32).pin_memory()

    store_mode = args.shard == "store" and world > 1
    if store_mode:
        # every rank answers the same global batch (the first qn queries) against its shard of the store
        q_host = torch.from_numpy(q_all[:qn]).pin_memory()
        q_dev = q_host.cuda()
        lo, hi = 0, qn
        w.predict_fast_sharded(q_dev[:64], k)  # builds this rank's shard index
    gather = parallel.ResultGather(qn * world, k, world) if (world > 1 and not store_mode) else None

    def step_device():
        if store_mode:
            return w.predict_fast_sharded(q_dev, k)
        ids, vals, _ = ix.predict(q_dev, k)
        if gather is not None:
            ids, vals = gather(ids, vals)
        return ids, vals

    def step_host():
        if store_mode:
            w.predict_fast_sharded(q_host.cuda(non_blocking=True), k)[0].cpu()
            return
        if gather is None:
            ix.predict_host(q_host, k, out_sid_h, out_val_h)
            return
        # N > 1: pinned host queries -> device, answer, all-gather ON THE DEVICE, one D2H of this rank's rows
        qd = q_host.cuda(non_blocking=True)
        ids, vals, _ = ix.predict(qd, k)
        gather(ids, vals)
        out_sid_h.copy_(ids, non_blocking=True)
        out_val_h.copy_(vals, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def timed(fn, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    last_step = [None]

    def step_device_kept():
        last_step[0] = step_device()

    for _ in range(max(args.warmup, 3)):
        step_device()
        step_host()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev = timed(step_device_kept, args.steps)
    # copied now: the all-gather reuses its buffers in the next call
    last_out = [t.cpu().numpy() for t in last_step[0]] if args.dump_outputs and rank == 0 else None
    ms_host = timed(step_host, args.steps)
    # the stages of one fused chunk (CUDA events inside cw_fused_profile) / the FP32 score kernel alone
    nq_k = min(qn, ix.fused_workspace(qn, k)["cap_q"]) if fused else min(qn, ix.chunk_queries())
    stages = None
    if fused:
        reps = [ix.profile_stages(q_dev[:nq_k], k) for _ in range(max(args.steps, 3))]
        stages = {name: float(np.median([r[name] for r in reps])) for name in reps[0]}
    else:
        ix.node_scores(q_dev[:nq_k])
        ms_kernel = timed(lambda: ix.node_scores(q_dev[:nq_k]), max(args.steps, 5)) / max(args.steps, 5)
    clocks = sampler.stop() if rank == 0 else None
    fstats = dict(ix.stats)

    # the FP32 form on the same batch: its step time, and the identity of the results
    fp32 = None
    if fused:
        ids_t, vals_t, _ = ix.predict(q_dev, k)
        ids_f, vals_f, _ = ix.predict(q_dev, k, mode="fp32")
        ms_dev32 = timed(lambda: ix.predict(q_dev, k, mode="fp32"), 2) / 2
        fp32 = {"queries_per_s": qn / (ms_dev32 * 1e-3), "ms_per_step": ms_dev32,
                "ids_identical": bool(torch.equal(ids_t, ids_f)), "scores_bit_identical": bool(torch.equal(vals_t, vals_f))}

    # FP32-FMA issue peak measured live (back-to-back FFMA chains, CUDA events, best of 5)
    L = _lib.load()
    sink = torch.zeros(4, device="cuda")
    ffma = 0.0
    for _ in range(5):
        blocks, threads, iters = 148 * 8, 256, 8000
        L.cw_ffma_peak(blocks, threads, 10, sink.data_ptr(), None)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.cw_ffma_peak(blocks, threads, iters, sink.data_ptr(), None)
        e1.record()
        torch.cuda.synchronize()
        ffma = max(ffma, 2.0 * blocks * threads * iters * 64 / e0.elapsed_time(e1) / 1e9)

    # secondary: best-first predict (cobweb_predict semantics) on a slice of the batch
    nbf = min(qn, 2048)
    w.tree.categorize_batch(q_dev[:nbf], retrieve_k=k, max_nodes=w.max_init_search)
    ms_bf = timed(lambda: w.tree.categorize_batch(q_dev[:nbf], retrieve_k=k, max_nodes=w.max_init_search), 3) / 3
    bf = w.tree.categorize_batch(q_dev[:nbf], retrieve_k=k, max_nodes=w.max_init_search)
    bf_rows = float(bf["lp_calls"].float().mean().item())

    # the reference's own usage pattern and published metric: ONE query per call through the reference-shaped API
    # (benchmark_utils.py:803-831 quotes ms per query), host vector in, python list of ids out
    single = None
    if not store_mode:
        w.cobweb_predict_fast(q_all[0], k=k, return_ids=True, is_embedding=True)
        torch.cuda.synchronize()
        n1 = 200
        t0 = time.time()
        for i in range(n1):
            w.cobweb_predict_fast(q_all[i % qn], k=k, return_ids=True, is_embedding=True)
        ms1 = (time.time() - t0) / n1 * 1e3
        one = q_dev[:1].contiguous()
        ix.predict_small(one, k)
        ms1_dev = timed(lambda: ix.predict_small(one, k), 50) / 50
        bytes1 = 8.0 * ix.nn * dim + 4.0 * ix.nn + 4.0 * dim  # the node operands once
        single = {"ms_per_query_api": ms1, "ms_per_query_device": ms1_dev,
                  "hbm_frac": bytes1 / (ms1 * 1e-3) / 1e9 / peaks["hbm_gbs"],
                  "hbm_frac_device": bytes1 / (ms1_dev * 1e-3) / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes": bytes1,
                  "api": "CobwebWrapper.cobweb_predict_fast -> cw_small_predict_host (one C call per query)"}

    # context (SURVEY 8d): the reference's brute-force inner-product baseline (retrieve_torch_dot, its stand-in for FAISS
    # IndexFlatIP) on the same corpus and queries -- library GEMM + top-k
    from rag_cobweb_b200.evaluate import retrieve_dot_batch
    x_dev = torch.from_numpy(x).cuda()
    retrieve_dot_batch(x_dev, q_dev, k)
    ms_dot = timed(lambda: retrieve_dot_batch(x_dev, q_dev, k), 3) / 3
    dot_ids = retrieve_dot_batch(x_dev, q_dev, k).cpu().numpy()
    brute = {"gpu_queries_per_s": qn / (ms_dot * 1e-3),
             "recall_at_k": float(np.mean([t in g for t, g in zip(targets_all[lo:hi], dot_ids)])),
             "note": "torch.matmul + torch.topk over the raw embeddings (retrieve_torch_dot semantics); a different retrieval "
                     "function than Cobweb's path-averaged log-likelihood, listed for context only"}
    del x_dev
    if world == 1 and not args.no_cpu_baseline:
        xs, qs = torch.from_numpy(x), torch.from_numpy(q_all[:512])
        torch.topk(qs @ xs.T, k, dim=1)
        t0 = time.time()
        torch.topk(qs @ xs.T, k, dim=1)
        brute["cpu_queries_per_s"] = 512 / (time.time() - t0)
        brute["cpu_sample"] = f"512 queries, torch CPU matmul + topk, {torch.get_num_threads()} threads"

    # correctness inside the bench: recall@k of the timed configuration (target among returned ids)
    ids, vals = step_device()
    got = ids.cpu().numpy()[lo:hi] if gather is not None else ids.cpu().numpy()
    got_v = vals.cpu().numpy()[lo:hi] if gather is not None else vals.cpu().numpy()
    recall = float(np.mean([t in g for t, g in zip(targets_all[lo:hi], got)]))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return None

    # ---------------------------------------------------------------- parity block (rank 0)
    parity = {"audit": {"audited_queries": fstats["audited"], "mismatches": fstats["audit_mismatch"],
                        "every": ix.audit_every,
                        "note": "always-on: one query in `every` is answered again by the exact small-batch path on the device "
                                "and compared bit for bit, in every call including the timed ones"}}
    if not args.no_cpu_baseline:
        host_threads()
        ot = oracle_from_engine(w)
        ns = 16
        o_ids, o_vals = oracle_topk(ot, q_all[lo:lo + ns], k)
        e_ids, e_vals = got[:ns], got_v[:ns]
        parity["oracle_topk"] = {
            "queries": ns, "ids_identical": float(np.mean((o_ids == e_ids).all(1))),
            "set_overlap": float(np.mean([len(set(a) & set(b)) / k for a, b in zip(o_ids, e_ids)])),
            "max_rel_score_diff": float(np.max(np.abs(o_vals - e_vals) / np.abs(o_vals))),
            "note": "oracle (CPU restatement, plain fp32 accumulation) vs engine on the same engine-built tree; ids can "
                    "differ only where two leaf scores agree to ~1e-6 relative"}
        if world == 1:
            for cfgname, fixture in GOLDEN.items():
                t0 = time.time()
                parity[cfgname] = reference_tree_parity(fixture, k)
                log(f"[bench] parity {cfgname}: {time.time() - t0:.1f}s {parity[cfgname]}")

    # ---------------------------------------------------------------- config 5 sample: streaming ifit (N = 1 only)
    stream = None
    if world == 1 and not args.no_cpu_baseline:
        from rag_cobweb_b200 import CobwebTorchTree
        n5 = 50000
        x5 = torch.from_numpy(synth.corpus(n5, 256, "whitened", seed=0)).cuda()
        t5 = CobwebTorchTree((256,))
        torch.cuda.synchronize()
        t0 = time.time()
        t5.ifit_batch(x5, tag_sentences=True)
        torch.cuda.synchronize()
        dt5 = time.time() - t0
        c5 = t5.store.counters()
        stream = {"inserts_per_s": n5 / dt5, "sample": f"first {n5} inserts of configs[4] (whitened 256-d stream)",
                  "levels_per_insert": c5["levels"] / n5, "rows_per_insert": c5["rows"] / n5,
                  "us_per_level_step": dt5 / c5["levels"] * 1e6}
        del t5, x5

    # ---------------------------------------------------------------- CPU baseline (rank 0, N = 1 only)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle.cobweb_oracle import OracleTree
        cores = host_threads()
        sample = 16
        rate = cpu_predict_rate(ot, q_all[:sample], k, min_seconds=8.0)
        o2 = OracleTree(dim)
        n_ins = min(docs, 1500)
        t0 = time.time()
        o2.ifit(x[:n_ins])
        ifit_rate = n_ins / (time.time() - t0)
        o5 = OracleTree(256)
        t0 = time.time()
        o5.ifit(synth.corpus(1500, 256, "whitened", seed=0))
        ifit5_rate = 1500 / (time.time() - t0)
        cpu = {"value": rate, "unit": "queries/s", "cores": cores, "kind": "port",
               "sample": f"{sample} queries x all {ix.nn} nodes per pass, repeated for >= 8 s, OpenMP over {cores} threads",
               "ifit_inserts_per_s": ifit_rate, "ifit_sample": f"first {n_ins} inserts, 1 thread",
               "ifit_cfg5_inserts_per_s": ifit5_rate, "ifit_cfg5_sample": "first 1500 whitened 256-d inserts, 1 thread"}

    # ---------------------------------------------------------------- roofline of the dominant kernel
    nn, n_pos = ix.nn, ix.n_pos
    traffic_file = os.path.join(ROOT, "profiles", "traffic_r02.json")
    traffic_db = json.load(open(traffic_file)) if os.path.exists(traffic_file) else {}

    def traffic_of(kernel):
        t = traffic_db.get(kernel)
        if t and t.get("workload") == {"docs": docs, "dim": dim, "queries": nq_k}:
            return t["dram_bytes_read"] + t["dram_bytes_write"]
        return None

    if fused:
        hx = ix.hx
        n_int, n_leaf = hx["n_int"], hx["n_leaf"]
        f1 = hx["leaf_layout"] == _lib.H_F1
        # per (query, row): the reference's direct form is 2 FMAs per attribute = 4 D flops (SURVEY 8d) whichever way the
        # kernel contracts; what the tensor pipe EXECUTES: internal rows 3 fp16 products over 2 D features = 12 D flops,
        # leaf rows one product over D (one-variance rows) or 2 D features = 2 D / 4 D flops
        dom = max(("internal_scores_f16x3", "leaf_filter_f16"), key=lambda s: stages[s])
        rows_dom = n_leaf if dom == "leaf_filter_f16" else n_int
        ms_dom = stages[dom]
        alg = 4.0 * nq_k * rows_dom * dim
        exe = (2.0 if f1 else 4.0) * nq_k * rows_dom * dim if dom == "leaf_filter_f16" else 12.0 * nq_k * rows_dom * dim
        op_bytes = (2.0 if f1 else 4.0) * dim if dom == "leaf_filter_f16" else 8.0 * dim  # fp16 operand bytes per row
        # operand bytes through L2 -> SM: the one-product kernels work on half tiles (128 query rows + 256 index rows per
        # tile, two CTAs per SM), the three-product kernel on 256 + 256 (ncu xbar2l1tex: 20.1 / 12.7 GB at cfg3,
        # profiles/r02_fused_ncu_full.md -- the rest is the epilogue's ancestor-sum loads)
        tq = 128 if dom == "leaf_filter_f16" else 256
        tiles = ((nq_k + tq - 1) // tq) * ((rows_dom + 255) // 256)
        l2_bytes = tiles * (tq + 256) * op_bytes
        peak = peaks["bf16_tflops"]
        achieved = alg / (ms_dom * 1e-3) / 1e12
        score_ms = stages["internal_scores_f16x3"] + stages["sample_threshold"] + stages["leaf_filter_f16"]
        roofline = {
            "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": traffic_of("h_score_kernel_filter" if dom == "leaf_filter_f16" else "h_score_kernel_node"),
            "kernel": "h_score_kernel<%s>" % ("1 product, FILTER" if dom == "leaf_filter_f16" else "3 products, NODE"),
            "kernel_ms": ms_dom, "rows": rows_dom, "queries": nq_k,
            "flops_per_launch": alg, "executed_flops_per_launch": exe, "executed_tflops": exe / (ms_dom * 1e-3) / 1e12,
            "executed_frac": exe / (ms_dom * 1e-3) / 1e12 / peak,
            "l2_to_sm_bytes_per_launch": l2_bytes, "l2_to_sm_tb_s": l2_bytes / (ms_dom * 1e-3) / 1e12,
            "bound_note": "two limits together (DESIGN.md section 5, Bounds): operand ingest per SM -- with the epilogue's "
                          "arithmetic compiled out the kernel takes 1.45 ms = 12.5 TB/s L2->SM = 44 B/clk per SM -- and a drain "
                          "of the accumulator that overlaps the other CTA's MMAs only partly (one half-tile CTA per SM: 2.93 ms)",
            "peak_source": f"kind::f16 dense = the bf16 burst peak, {peak_src}",
            "note": "achieved = ALGORITHMIC flops of the dominant kernel's rows (4 per query, row and attribute: the "
                    "reference's direct form) / its CUDA-event time; executed_* = what the tensor pipe really does. The "
                    "fp16 filter executes LESS than the algorithmic count (one product over D features instead of two over "
                    "2D), so achieved can exceed the tensor peak; the honest utilisation figure is executed_frac",
            "whole_index": {"flops": 4.0 * nq_k * nn * dim, "score_kernels_ms": score_ms,
                            "tflops": 4.0 * nq_k * nn * dim / (score_ms * 1e-3) / 1e12,
                            "frac_of_tf32_peak": 4.0 * nq_k * nn * dim / (score_ms * 1e-3) / 1e12 / (peak / 2.0),
                            "note": "all three score launches (internal rows, sampled tiles, leaf filter) together against "
                                    "4 Q Nn D and the TF32 dense peak = half the bf16 peak: the figure round 1 reported as frac"},
            "algorithmic_bytes": 8.0 * nn * dim + 4.0 * nn + 4.0 * nq_k * dim + 8.0 * nq_k * k,
        }
        launches_per_chunk = (1 + (2 if hx["n_int"] else 0) + (2 if hx["n_s"] else 1) + 3 + 5 * _lib.FUSED_FB_ROUNDS + 1 +
                              (6 if ix.audit_every else 0))
        chunks = (qn + ix.fused_workspace(qn, k)["cap_q"] - 1) // ix.fused_workspace(qn, k)["cap_q"]
    else:
        flops = 4.0 * nq_k * nn * dim
        alg_bytes = 8.0 * nn * dim + 4.0 * nn + 4.0 * nq_k * dim + 4.0 * nq_k * nn
        achieved = flops / (ms_kernel * 1e-3) / 1e12
        roofline = {"bound": "fp32", "achieved": achieved, "peak": ffma, "unit": "TFLOP/s", "frac": achieved / ffma,
                    "traffic": traffic_of("dense_score_kernel"), "algorithmic_bytes": alg_bytes, "kernel": "dense_score_kernel",
                    "kernel_ms": ms_kernel, "flops_per_launch": flops,
                    "peak_source": "FFMA issue peak measured in this run (cw_ffma_peak)",
                    "hbm_frac": alg_bytes / (ms_kernel * 1e-3) / 1e9 / peaks["hbm_gbs"], "hbm_peak_source": peak_src}
        launches_per_chunk = 4 if qn > _lib.SMALL_Q else 3
        chunks = (qn + ix.chunk_queries() - 1) // ix.chunk_queries()
    total_q = qn if store_mode else qn * world
    line = {
        "metric": "cobweb_predict_fast queries/sec", "value": total_q * args.steps / (ms_dev * 1e-3), "unit": "queries/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev / args.steps,
        "higher_is_better": True, "scaling": "strong" if store_mode else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": cfg, "docs": docs, "dim": dim, "nodes": nn, "queries_per_gpu": qn, "k": k,
                   "parallelism": (f"store sharded x{world} (sentences + ancestor nodes), NCCL all-gather + top-k merge"
                                   if store_mode else f"replicated store, query-sharded x{world}, one all_gather_into_tensor "
                                                      "of the packed results on the device") if world > 1 else "single GPU",
                   "l2": "inputs exceed L2 (node operands %.0f MB fp32 / %.0f MB fp16 per pass)" % (8.0 * nn * dim / 1e6, 2.4 * nn * dim / 1e6),
                   "scoring": ("fused: tcgen05 kind::f16 -- internal rows with split operands (3 products), leaf rows with ONE "
                               "fp16 product as a filter with a derived error bound -- then exact FP32 refine / re-score; ids "
                               "and scores bit-identical to the FP32-pipe path (dtype f32 names the result arithmetic)")
                   if fused else "fp32: FP32-pipe FFMA2 kernel"},
        "e2e": {"value": total_q * args.steps / (ms_host * 1e-3), "unit": "queries/s",
                "h2d_bytes_per_step": int(qn * dim * 4), "d2h_bytes_per_step": int(qn * k * 8),
                "api": (("cw_fused_predict_host" if fused else "cw_predict_dense_host") + " (one C-ABI call per batch, pinned host "
                        "buffers)") if gather is None and not store_mode else
                       "pinned host queries -> device, cw_fused_predict, all-gather on the device, D2H of this rank's rows"},
        "gpu_launches": launches_per_chunk * chunks * args.steps,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "recall_at_k": recall,
        "parity": parity,
        "stages_ms": stages,
        "fused_stats": {**fstats, "candidates_per_query": fstats["candidates"] / max(fstats["queries"], 1),
                        "refined_per_query": fstats["refined"] / max(fstats["queries"], 1),
                        "rescored_per_query": fstats["rescored"] / max(fstats["queries"], 1)} if fused else None,
        "fp32_path": fp32,
        "brute_force_ip": brute,
        "single_query": single,
        "index_build_s": index_build_s,
        "index_bytes": ix.bytes(),
        "ffma_peak_tflops": ffma,
        "queries_answered": int(qn * (2 * max(args.warmup, 3) + 2 * args.steps)),
        "best_first": {"queries_per_s": nbf * world / (ms_bf * 1e-3), "rows_scored_per_query": bf_rows,
                       "queries": nbf, "hbm_frac": nbf * bf_rows * (8.0 * dim + 4) / (ms_bf * 1e-3) / 1e9 / peaks["hbm_gbs"],
                       "note": "cobweb_predict semantics (CobwebTorchTree._cobweb_categorize), algorithmic bytes = rows scored x (8D+4)"},
        "ifit_stream_cfg5": stream,
        "ifit": {"inserts_per_s": docs / build_s, "seconds": build_s, "levels_per_insert": counters["levels"] / docs,
                 "rows_per_insert": counters["rows"] / docs,
                 "hbm_frac": (counters["rows"] + counters["levels"] + docs) * (8.0 * dim + 4) / build_s / 1e9 / peaks["hbm_gbs"]},
    }
    if last_out is not None:
        dump_outputs(args.dump_outputs, *last_out)
    if world > 1:
        dist.destroy_process_group()
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--docs", type=int)
    ap.add_argument("--queries", type=int)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--snapshot", help="binary snapshot of the built tree: written after the build if missing, loaded instead of "
                                       "building if present (several runs of the 1M-document workload on one box)")
    ap.add_argument("--mode", default="fused", choices=["fused", "fp32"],
                    help="fused (default): tcgen05 fp16 pipeline (3-product internal rows, 1-product leaf filter with a derived "
                         "bound) + exact FP32 refine / re-score; fp32: everything on the FP32 pipe.  The results are identical")
    ap.add_argument("--shard", default="query", choices=["query", "store"],
                    help="N>1: 'query' replicates the store and shards the batch (weak scaling, default); "
                         "'store' shards sentences+nodes, every rank answers the whole batch, per-rank top-k "
                         "lists are merged after an NCCL all-gather (strong scaling)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the ids and scores the last one computed as DIR/<name>.npy "
                         f"(at most {DUMP_MAX_BYTES // 10**6} MB: a larger batch is cut to a fixed seeded sample of its rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    wl = list(WORKLOADS[args.workload])
    if args.docs:
        wl[0] = args.docs
    if args.queries:
        wl[2] = args.queries
    import __graft_entry__
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        __graft_entry__._load_build_module().build()
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_engine(args, wl)


if __name__ == "__main__":
    main()
