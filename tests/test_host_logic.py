"""CPU tests of the host-side logic: topology processing against the oracle's index, the JSON
wire format, weight schedules, the C-ABI library's exported symbols, and the multi-process
query-sharding plumbing (gloo, world_size 2)."""
import ctypes
import json
import os
import re
import socket

import numpy as np
import pytest
import torch

from oracle.cobweb_oracle import OracleTree
from rag_cobweb_b200 import _lib, parallel, serialize, synth, topology

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_tree(n=300, d=32, kind="unit"):
    x = synth.corpus(n, d, kind, seed=0)
    t = OracleTree(d)
    leaves = t.ifit(x)
    return x, t, leaves


def flat_topology(t):
    """Store-style arrays (child_off/cnt/pool) from an oracle tree, node id = BFS index."""
    b = t.bfs()
    n = len(b["order"])
    cnt = b["nchild"].astype(np.int64)
    off = np.cumsum(cnt) - cnt
    pool = np.zeros(max(int(cnt.sum()), 1), np.int32)
    fill = np.zeros(n, np.int64)
    for i in range(1, n):
        p = b["parent"][i]
        pool[off[p] + fill[p]] = i
        fill[p] += 1
    return b, off.astype(np.int32), cnt.astype(np.int32), pool


def test_bfs_and_paths_match_oracle_index():
    x, t, leaves = oracle_tree()
    b, off, cnt, pool = flat_topology(t)
    order, parent_b, depth = topology.bfs_order(0, off, cnt, pool)
    assert np.array_equal(order, np.arange(len(order)))
    assert np.array_equal(parent_b, b["parent"]) and np.array_equal(depth, b["depth"])
    ix = t.build_index(level_weights=[1.0, 0.5, 0.25])
    pos = np.full(int(b["order"].max()) + 1, -1)
    pos[b["order"]] = np.arange(len(b["order"]))
    p = topology.sentence_paths(order, parent_b, depth, pos[leaves], [1.0, 0.5, 0.25])
    # positions are a permutation of sentence ids, grouped by leaf in tree order
    assert sorted(p["pos_sid"].tolist()) == list(range(len(leaves)))
    assert (np.diff(pos[leaves][p["pos_sid"]]) >= 0).all()
    # per sentence the path and the weights are the oracle's (build_prediction_index semantics)
    assert np.array_equal(p["path_idx"].T[np.argsort(p["pos_sid"])], ix["path_idx"])
    assert np.array_equal(p["path_w"].T[np.argsort(p["pos_sid"])], ix["path_w"])
    # per-position records: length, shared prefix with the previous position, leaf row, sentence id
    rec = p["pos_rec"]
    assert np.array_equal(rec[:, 0], p["path_len"]) and np.array_equal(rec[:, 3], p["pos_sid"])
    for i in range(len(rec)):
        col = p["path_idx"][:, i]
        assert rec[i, 2] == col[rec[i, 0] - 1]
        if i:
            prev = p["path_idx"][:, i - 1]
            m = 0
            while m < rec[i, 0] and rec[i, 0] == rec[i - 1, 0] and col[m] == prev[m]:
                m += 1
            assert rec[i, 1] == m
    assert rec[0, 1] == 0 and (rec[1:, 1] >= rec[1:, 0] - 1).mean() > 0.5  # siblings share all but the leaf
    # the (len, depth) weight table the kernel uses holds exactly those values
    for j in range(p["max_len"]):
        ok = p["path_idx"][j] >= 0
        assert np.array_equal(p["w_table"][p["path_len"][ok], j], p["path_w"][j][ok])


def test_restrict_to_paths_keeps_exactly_the_ancestors():
    x, t, leaves = oracle_tree(200, 8)
    b, off, cnt, pool = flat_topology(t)
    order, parent_b, depth = topology.bfs_order(0, off, cnt, pool)
    pos = np.full(int(b["order"].max()) + 1, -1)
    pos[b["order"]] = np.arange(len(b["order"]))
    some = pos[leaves][::7]
    o2, p2, d2 = topology.restrict_to_paths(order, parent_b, depth, some, len(order))
    want = set()
    for leaf in some:
        nd = int(leaf)
        while nd >= 0:
            want.add(nd)
            nd = int(parent_b[nd])
    assert set(o2.tolist()) == want and list(o2) == sorted(want)
    assert p2[0] == -1 and all(o2[p2[i]] == parent_b[o2[i]] for i in range(1, len(o2)))
    assert np.array_equal(d2, depth[o2])


def test_sentence_paths_rejects_dangling_leaf():
    x, t, leaves = oracle_tree(60, 8)
    b, off, cnt, pool = flat_topology(t)
    order, parent_b, depth = topology.bfs_order(0, off, cnt, pool)
    with pytest.raises(ValueError):
        topology.sentence_paths(order[:-1], parent_b[:-1], depth[:-1], [len(order) - 1], n_slots=len(order))


def test_weight_schedules_match_reference_formulas():
    g = topology.generate_weight_schedule
    assert g("constant", 3, value=2.0) == [2.0, 2.0, 2.0]
    assert g("linear", 3, start=1.0, end=3.0) == [1.0, 2.0, 3.0]
    assert g("linear", 3, start=1.0, end=3.0, direction="decrease") == [3.0, 2.0, 1.0]
    assert g("linear", 1, start=5.0) == [5.0]
    assert g("quadratic", 3) == [1.0, 0.25, 1 / 9]
    assert g("quadratic", 2, start_n=0) == [1.0, 1.0]
    assert g("exponential", 3, base=0.5) == [1.0, 0.5, 0.25]
    with pytest.raises(ValueError):
        g("cubic", 3)


def test_json_wire_format_roundtrip_and_reference_shape():
    x, t, leaves = oracle_tree(120, 16)
    b = t.bfs()
    mean, m2 = t.rows(b["order"])
    pos = np.full(int(b["order"].max()) + 1, -1)
    pos[b["order"]] = np.arange(len(b["order"]))
    sids = [[] for _ in b["order"]]
    for sid, leaf in enumerate(leaves):
        sids[pos[leaf]].append(sid)
    params = dict(use_info=True, acuity_cutoff=False, use_kl=True, shape=[16], alpha=1e-8, prior_var=0.0585)
    doc = serialize.dump_tree_json(params, b["parent"], b["count"], mean, m2, sids)
    data = json.loads(doc)
    # the reference's document shape (CobwebTorchTree.py:67-81, CobwebTorchNode.py:741-772)
    assert set(data) == {"use_info", "acuity_cutoff", "use_kl", "shape", "alpha", "prior_var", "root"}
    assert set(data["root"]) == {"count", "mean", "meanSq", "sentence_id", "children"}
    assert len(data["root"]["children"]) == b["nchild"][0]
    p2, parent2, count2, mean2, m22, sids2 = serialize.load_tree_json(doc)
    assert p2 == params
    assert np.array_equal(parent2, b["parent"]) and np.array_equal(count2, b["count"])
    assert np.array_equal(mean2, mean) and np.array_equal(m22, m2)  # fp32 -> decimal -> fp32 is lossless
    assert sids2 == sids


def test_library_exports_every_declared_symbol():
    """The C ABI loads without a GPU and exports every function include/cobweb_b200.h declares."""
    hdr = open(os.path.join(ROOT, "include", "cobweb_b200.h")).read()
    declared = set(re.findall(r"^\s*(?:int|int64_t|const char \*)\s*(cw_\w+)\(", hdr, flags=re.M))
    assert declared == set(_lib.EXPORTS)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name)
    assert lib.cw_version() == 100
    assert ctypes.sizeof(_lib.CwStore) == 24 + 14 * 8
    assert lib.cw_topk_chunks(1025) == 3 and lib.cw_xt_floats(129, 20) == 2 * 2 * 16 * 128  # 2 chunks + the threshold slot
    # fp16 operand sets: layout F1 = 32 attributes per slab, F2 = 16; one-product sets pack two slabs into a stage
    assert lib.cw_h_stages(768, _lib.H_F1, 1) == 12 and lib.cw_h_stages(768, _lib.H_F2, 3) == 48 and lib.cw_h_stages(33, _lib.H_F1, 1) == 1
    assert lib.cw_h_a_bytes(257, 20, _lib.H_F2, 3) == 2 * 2 * 32768 and lib.cw_h_b_bytes(300, 9, _lib.H_F1, 1) == 2 * 1 * 32768
    assert lib.cw_small_scratch_words(1025, 10) == 32 * 3 * 10 * 2
    assert ctypes.sizeof(_lib.CwDenseWork) == 7 * 8 and ctypes.sizeof(_lib.CwHSet) == 6 * 4 + 2 * 8
    assert ctypes.sizeof(_lib.CwFusedIndex) == ctypes.sizeof(_lib.CwIndex) + 16 + 2 * 40 + 8 * 8 + 6 * 4
    assert ctypes.sizeof(_lib.CwFusedWork) == 2 * 8 + 7 * 8 + 8 + 13 * 8 + 8


def test_engine_refuses_to_run_without_cuda():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from rag_cobweb_b200 import CobwebB200Error, CobwebTorchTree, CobwebWrapper
    with pytest.raises(CobwebB200Error):
        CobwebTorchTree((8,))
    with pytest.raises(CobwebB200Error):
        CobwebWrapper(corpus=[None], corpus_embeddings=np.zeros((1, 8), np.float32))


def test_shard_bounds_cover_everything():
    for n in (0, 1, 7, 10, 64):
        for w in (1, 2, 3, 8):
            spans = [parallel.shard_bounds(n, w, r) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


def test_merge_topk_orders_by_score_then_id():
    ids = torch.tensor([[5, 2, -1, 9, 7, 1]], dtype=torch.int32)
    vals = torch.tensor([[1.0, 3.0, 99.0, 3.0, 0.5, 3.0]])
    i, v = parallel.merge_topk(ids, vals, 4)
    assert i.tolist() == [[1, 2, 9, 5]] and v.tolist() == [[3.0, 3.0, 3.0, 1.0]]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q, ret):
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        x, t, _ = oracle_tree(200, 16)
        t.build_index()
        qs, _ = synth.queries(x, q, "unit", seed=1)
        k = 5

        def local_predict(batch):  # stand-in for the per-GPU engine call
            _, ls = t.dense_scores(batch)
            ids = np.argsort(-ls, axis=1, kind="stable")[:, :k].astype(np.int32)
            return torch.from_numpy(ids), torch.from_numpy(np.take_along_axis(ls, ids.astype(np.int64), 1))

        # query-sharded mode: each rank answers its shard, one all-gather returns the batch
        lo, hi = parallel.shard_bounds(q, world, rank)
        ids, vals = local_predict(qs[lo:hi])
        gi, gv = parallel.gather_results(ids, vals, q)
        full_i, full_v = local_predict(qs)
        ok1 = torch.equal(gi, full_i) and torch.equal(gv, full_v)
        # the re-usable form: sizes from shard_bounds, one packed collective, same buffers on every call
        g = parallel.ResultGather(q, k, device="cpu")
        for _ in range(2):
            gi2, gv2 = g(ids, vals)
            ok1 = ok1 and torch.equal(gi2, full_i) and torch.equal(gv2, full_v)
        # store-sharded mode: each rank scores only its sentences, candidates merged after all-gather
        _, ls = t.dense_scores(qs)
        slo, shi = parallel.shard_bounds(ls.shape[1], world, rank)
        part = ls[:, slo:shi]
        pid = np.argsort(-part, axis=1, kind="stable")[:, :k]
        cand_i = torch.from_numpy((pid + slo).astype(np.int32))
        cand_v = torch.from_numpy(np.take_along_axis(part, pid, 1))
        ci, cv = parallel.gather_candidates(cand_i, cand_v)
        mi, mv = parallel.merge_topk(ci, cv, k)
        ok2 = torch.equal(mi, full_i) and torch.equal(mv, full_v)
        ret[rank] = (ok1, ok2)
    finally:
        dist.destroy_process_group()


def test_query_sharding_world_size_2_gloo():
    import torch.multiprocessing as mp
    world, q = 2, 11  # odd batch: shards of different size
    mgr = mp.Manager()
    ret = mgr.dict()
    port = _free_port()
    mp.spawn(_worker, args=(world, port, q, ret), nprocs=world, join=True)
    assert dict(ret) == {0: (True, True), 1: (True, True)}


def test_evaluator_matches_the_reference_loop():
    """metrics_from_ids == the reference's per-query loop (benchmark_utils.py:794-820, transcribed here with
    sklearn's ndcg_score called the way the reference calls it), including short result lists."""
    from sklearn.metrics import ndcg_score
    from rag_cobweb_b200.evaluate import get_eval_ks, metrics_from_ids
    rng = np.random.default_rng(0)
    nq, top_k, n_docs = 300, 20, 60
    retrieved = np.stack([rng.permutation(n_docs)[:top_k] for _ in range(nq)])
    retrieved[5, 7:] = -1   # fewer than top_k documents came back
    retrieved[6, 1:] = -1
    targets = rng.integers(0, n_docs, nq)
    targets[:40] = retrieved[:40, 0]  # some first-rank hits
    ks = get_eval_ks(top_k)
    assert ks == [2, 3, 5, 10, 20]
    want = {f"{m}@{k}": 0.0 for k in ks for m in ("recall", "mrr", "ndcg")}
    for row, target in zip(retrieved, targets):
        docs = [d for d in row.tolist() if d >= 0]
        for k in ks:
            top = docs[:k]
            if target in top:
                want[f"recall@{k}"] += 1
                want[f"mrr@{k}"] += 1 / (top.index(target) + 1)
            relevance = [1 if d == target else 0 for d in top]
            if sum(relevance) > 0 and len(relevance) > 1:
                want[f"ndcg@{k}"] += ndcg_score([sorted(relevance, reverse=True)], [relevance])
            elif sum(relevance) > 0:
                want[f"ndcg@{k}"] += 1.0  # sklearn rejects single-document lists; the only document is the hit
    got = metrics_from_ids("x", retrieved, targets, top_k, seconds=1.5)
    for key, v in want.items():
        assert got[key] == round(v / nq, 4), key
    assert got["method"] == "x" and got["time_taken"] == 1.5 and got["avg_latency_ms"] == 5.0


def test_bench_dump_outputs_whole_or_seeded_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: a batch under the cap is written whole (ids exact as float64); a larger one as the same
    seeded sample of rows on every call, under the cap, with its row numbers."""
    import bench
    rng = np.random.default_rng(2)
    ids = rng.integers(0, 1 << 30, (500, 10)).astype(np.int32)
    scores = rng.standard_normal((500, 10)).astype(np.float32)
    bench.dump_outputs(str(tmp_path / "whole"), ids, scores)
    assert sorted(os.listdir(tmp_path / "whole")) == ["ids.npy", "scores.npy"]
    got = np.load(tmp_path / "whole" / "ids.npy")
    assert got.dtype == np.float64 and np.array_equal(got.astype(np.int32), ids)
    assert np.array_equal(np.load(tmp_path / "whole" / "scores.npy"), scores)
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 3 * 1024 + 100 * 128)
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), ids, scores)
    files = {f: np.load(tmp_path / "a" / f) for f in ("ids.npy", "scores.npy", "rows.npy")}
    rows = files["rows.npy"].astype(np.int64)
    assert len(rows) == 100 and (np.diff(rows) > 0).all()
    assert np.array_equal(files["ids.npy"], ids[rows]) and np.array_equal(files["scores.npy"], scores[rows])
    assert all(np.array_equal(a, np.load(tmp_path / "b" / f)) for f, a in files.items())
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_MAX_BYTES


def test_fused_layout_reproduces_the_path_sums():
    """(C[parent] + w_leaf s_leaf) / len over the fused layout == sum_j (w_j / len) s_j over the root->leaf paths
    (CobwebWrapper.py:160-169), every sentence appears exactly once, sampled tiles lead."""
    rng = np.random.default_rng(3)
    n_nodes = 4000
    parent = np.full(n_nodes, -1, np.int64)
    for i in range(1, n_nodes):
        parent[i] = rng.integers(max(0, i - 60), i)
    child_cnt = np.bincount(parent[1:], minlength=n_nodes).astype(np.int32)
    child_off = (np.cumsum(child_cnt) - child_cnt).astype(np.int32)
    pool = np.argsort(parent[1:], kind="stable").astype(np.int32) + 1
    order, parent_b, depth = topology.bfs_order(0, child_off, child_cnt, pool)
    leaves = np.nonzero(child_cnt == 0)[0]
    leaf_of_sentence = np.concatenate([leaves, leaves[:37], leaves[:5]])  # some leaves hold two or three sentences
    leaf_of_sentence = leaf_of_sentence[rng.permutation(len(leaf_of_sentence))]
    lw = [1.0, 0.5, 2.0, 1.5]
    F = topology.fused_layout(order, parent_b, depth, leaf_of_sentence, lw, n_slots=n_nodes, tile=64, sample_every=4)
    s = rng.standard_normal(len(order))                       # one query's node scores by index row
    C = np.zeros(len(F["int_rows"]))
    for lvl in range(len(F["level_off"]) - 1):                # top-down, one level at a time
        a, b = F["level_off"][lvl], F["level_off"][lvl + 1]
        par = F["int_parent"][a:b]
        C[a:b] = np.where(par >= 0, C[np.maximum(par, 0)], 0.0) + F["int_w"][a:b].astype(np.float64) * s[F["int_rows"][a:b]]
    par = F["leaf_parent"]
    leaf_score = (np.where(par >= 0, C[np.maximum(par, 0)], 0.0) + F["leaf_w"].astype(np.float64) * s[F["leaf_rows"]]) * \
        F["leaf_inv_len"].astype(np.float64)
    P = topology.sentence_paths(order, parent_b, depth, leaf_of_sentence, lw, n_slots=n_nodes)
    want = np.zeros(len(leaf_of_sentence))
    for p in range(len(leaf_of_sentence)):
        ln = P["path_len"][p]
        want[P["pos_sid"][p]] = sum(P["level_w"][j] / ln * s[P["path_idx"][j, p]] for j in range(ln))
    got = np.full(len(leaf_of_sentence), np.nan)
    for leaf in range(len(F["leaf_rows"])):
        got[F["sent_ids"][F["sent_off"][leaf]:F["sent_off"][leaf + 1]]] = leaf_score[leaf]
    np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-9)
    assert sorted(F["sent_ids"].tolist()) == list(range(len(leaf_of_sentence)))
    ns = F["n_sample_tiles"]
    n_leaf = len(F["leaf_rows"])
    assert ns == ((n_leaf + 3) // 4) // 64 and ns > 0 and len(F["flat_pos_rec"]) == F["sent_off"][ns * 64]
    assert np.array_equal(F["leaf_len"], depth[F["leaf_rows"]] + 1) and F["leaf_len"].dtype == np.int32
    assert sorted(F["leaf_rows"].tolist()) == sorted(np.unique(topology.sentence_paths(order, parent_b, depth, leaf_of_sentence, lw, n_slots=n_nodes)["pos_rec"][:, 2]).tolist())
    assert (F["flat_pos_rec"][:, 2] < ns * 64).all() and (np.diff(F["flat_pos_rec"][:, 2]) >= 0).all()


def test_fused_mode_host_policy():
    """Host-side policy of the fused mode (no GPU needed): which requests it serves, how the counters of a call are
    folded into DenseIndex.stats, and that an audit mismatch widens eps."""
    import warnings
    from rag_cobweb_b200 import _lib
    from rag_cobweb_b200.wrapper import DenseIndex
    ix = DenseIndex.__new__(DenseIndex)
    ix.mode, ix.nn, ix.hx = "fused", 20000, {"smem_ok": True}
    assert ix.fused_ready(1) and ix.fused_ready(_lib.FUSED_MAX_K) and not ix.fused_ready(_lib.FUSED_MAX_K + 1) and not ix.fused_ready(0)
    ix.nn = DenseIndex.TENSOR_MIN_NODES - 1     # small index: the FP32 pipe is the shorter path
    assert not ix.fused_ready(10)
    ix.nn, ix.mode = 20000, "fp32"
    assert not ix.fused_ready(10)
    ix.stats = {"queries": 0, "flagged": 0, "unresolved": 0, "cand_overflow": 0, "line_fail": 0, "list_overflow": 0,
                "candidates": 0, "audited": 0, "audit_mismatch": 0, "refined": 0, "rescored": 0}
    ix.eps_scale = DenseIndex.EPS_SCALE
    st = np.zeros(_lib.FUSED_STATS, np.int32)
    st[0], st[2], st[3], st[5], st[8] = 3, 1, 2, 10000, 5
    st[6:8] = np.array([(1 << 32) + 7], np.uint64).view(np.int32)   # 64-bit candidate counter
    ix._account(st)
    assert ix.stats["flagged"] == 3 and ix.stats["cand_overflow"] == 1 and ix.stats["line_fail"] == 2
    assert ix.stats["queries"] == 10000 and ix.stats["candidates"] == (1 << 32) + 7 and ix.stats["audited"] == 5
    assert ix.eps_scale == DenseIndex.EPS_SCALE
    st[:] = 0
    st[9] = 1
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        ix._account(st)
    assert ix.stats["audit_mismatch"] == 1 and ix.eps_scale == 4 * DenseIndex.EPS_SCALE and len(rec) == 1


def test_device_topology_matches_host_topology():
    """topology_device (torch ops on the store's tensors, SURVEY 8f-1) == topology (numpy statements) on random trees:
    BFS numbering, per-sentence paths / position records, fused layout -- with level weights, leaves holding several
    sentences, shuffled child pools and dead slots."""
    from rag_cobweb_b200 import topology_device as td
    rng = np.random.default_rng(11)
    for n_nodes, lw, tile, every in ((1, None, 64, 4), (50, None, 16, 2), (3000, [1.0, 0.5, 2.0, 1.5], 64, 4), (2500, None, 64, 8)):
        parent = np.full(n_nodes, -1, np.int64)
        for i in range(1, n_nodes):
            parent[i] = rng.integers(max(0, i - 40), i)
        child_cnt = np.bincount(parent[1:], minlength=n_nodes).astype(np.int32)
        # child lists at scattered pool offsets (lists are allocated with slack and out of order in the real store)
        caps = child_cnt + rng.integers(0, 3, n_nodes).astype(np.int32)
        perm = rng.permutation(n_nodes)
        off = np.zeros(n_nodes, np.int64)
        off[perm] = np.cumsum(caps[perm]) - caps[perm]
        pool = np.full(int(caps.sum()) + 1, -7, np.int32)
        fill = np.zeros(n_nodes, np.int64)
        for i in range(1, n_nodes):
            p = parent[i]
            pool[off[p] + fill[p]] = i
            fill[p] += 1
        child_off = off.astype(np.int32)
        order, parent_b, depth = topology.bfs_order(0, child_off, child_cnt, pool)
        t = lambda a: torch.as_tensor(a)
        o2, p2, d2 = td.bfs_order(0, t(child_off), t(child_cnt), t(pool))
        assert np.array_equal(o2.numpy(), order) and np.array_equal(p2.numpy(), parent_b) and np.array_equal(d2.numpy(), depth)
        leaves = np.nonzero(child_cnt == 0)[0]
        los = np.concatenate([leaves, leaves[: len(leaves) // 7], leaves[:3]])
        los = los[rng.permutation(len(los))]
        P = topology.sentence_paths(order, parent_b, depth, los, lw, n_slots=n_nodes)
        P2 = td.sentence_paths(o2, p2, d2, t(los), lw, n_slots=n_nodes)
        assert P2["max_len"] == P["max_len"] and np.array_equal(P2["path_idx"].numpy(), P["path_idx"].T)
        assert np.array_equal(P2["pos_rec"].numpy(), P["pos_rec"]) and np.allclose(P2["level_w"], P["level_w"])
        assert np.array_equal(P2["pos_leaf_row"].numpy(), P["pos_rec"][:, 2]) and P2["path_lens"] == np.unique(P["pos_rec"][:, 0]).tolist()
        if n_nodes == 1:
            continue
        F = topology.fused_layout(order, parent_b, depth, los, lw, n_slots=n_nodes, tile=tile, sample_every=every)
        F2 = td.fused_layout(o2, p2, d2, t(los), lw, n_slots=n_nodes, tile=tile, sample_every=every)
        for key in ("int_rows", "int_parent", "int_w", "level_off", "leaf_rows", "leaf_parent", "leaf_w", "leaf_inv_len", "leaf_len",
                    "sent_off", "sent_ids"):
            assert np.array_equal(F2[key].numpy(), np.asarray(F[key])), (n_nodes, key)
        assert F2["n_sample_tiles"] == F["n_sample_tiles"] and F2["max_len"] == F["max_len"]
