"""GPU parity tests: the sm_100a engine (through the reference-shaped Python API, which calls
the C ABI of libcobweb_b200.so) against the CPU oracle and the golden fixtures recorded from
the reference.  Bars (BASELINE.json north_star):
  * integer / index results bit-exact: decision traces, tree structure, leaf of every
    instance, best-first pop order, rows scored per query;
  * node statistics bit-exact (they involve no reduction);
  * dense log-likelihood scores within 1e-5 relative of the oracle (fp32 FMA accumulation vs
    the oracle's pairwise-binary64 sum; the north_star tolerance is 1e-4);
  * the path product bit-exact given the same node scores; top-k = exact arg-sort of them.
"""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
EPS32 = float(np.finfo(np.float32).eps)

from oracle.cobweb_oracle import OracleTree, leaf_scores as oracle_leaf_scores  # noqa: E402
from rag_cobweb_b200 import CobwebTorchTree, CobwebWrapper, DenseIndex, synth  # noqa: E402

DenseIndex.TENSOR_MIN_NODES = 0  # the tests' trees are small: keep the tensor-core modes on the tensor cores


def pos_of(b):
    pos = np.full(int(b["order"].max()) + 1, -1, np.int64)
    pos[b["order"]] = np.arange(len(b["order"]))
    return pos


def assert_same_tree(tree, ref, leaves=None, ref_leaves=None):
    b, rb = tree.bfs(), ref.bfs()
    assert np.array_equal(b["parent"], rb["parent"])
    assert np.array_equal(b["count"], rb["count"])
    assert np.array_equal(b["nchild"], rb["nchild"])
    assert np.array_equal(b["nsent"], rb["nsent"])
    mean, m2 = tree.store.rows(b["order"])
    rmean, rm2 = ref.rows(rb["order"])
    assert np.array_equal(mean, rmean)
    assert np.array_equal(m2, rm2)
    pos, rpos = pos_of(b), pos_of(rb)
    if leaves is not None:
        assert np.array_equal(pos[leaves], rpos[ref_leaves])
    return pos, rpos


def build_pair(n, d, kind, seed=0, dups=False, **kw):
    x = synth.corpus(n, d, kind, seed=seed)
    if dups:
        x[n // 4:n // 4 + 10] = x[5:15]
    tree = CobwebTorchTree((d,), **kw)
    ref = OracleTree(d, use_info=kw.get("use_info", True), use_kl=kw.get("use_kl", True),
                     acuity_cutoff=kw.get("acuity_cutoff", False), prior_var=kw.get("prior_var"))
    return x, tree, ref


@pytest.mark.parametrize("n,d,kind", [(300, 64, "unit"), (500, 128, "unit"), (400, 384, "unit"), (300, 1024, "unit"),
                                      (500, 256, "whitened"), (300, 30, "unit"), (200, 7, "whitened"),
                                      (150, 2048, "unit")])
def test_ifit_bit_exact_vs_oracle(n, d, kind):
    x, tree, ref = build_pair(n, d, kind)
    leaves, ops, off = tree.ifit_batch(x, tag_sentences=True, trace=True)
    rl, rops, roff = ref.ifit(x, trace=True)
    assert np.array_equal(ops, rops) and np.array_equal(off, roff)
    assert_same_tree(tree, ref, leaves.cpu().numpy(), rl)


@pytest.mark.parametrize("kw", [dict(use_kl=False), dict(use_info=False), dict(acuity_cutoff=True),
                                dict(prior_var=0.01)])
def test_ifit_modes(kw):
    x, tree, ref = build_pair(300, 96, "whitened", **kw)
    leaves, ops, off = tree.ifit_batch(x, tag_sentences=True, trace=True)
    rl, rops, roff = ref.ifit(x, trace=True)
    assert np.array_equal(ops, rops)
    assert_same_tree(tree, ref, leaves.cpu().numpy(), rl)


def test_ifit_duplicates_and_single_calls():
    x, tree, ref = build_pair(200, 32, "unit", dups=True)
    rl, rops, _ = ref.ifit(x, tag_sentences=False, trace=True)
    assert (rops == 4).sum() > 5  # the leaf-increment branch is exercised
    got = [tree.ifit(torch.from_numpy(v)).node_id for v in x]  # reference-style one-at-a-time API
    pos, rpos = assert_same_tree(tree, ref)
    assert np.array_equal(pos[np.asarray(got)], rpos[rl])


def test_ifit_cluster_sizes_agree():
    """The thread-block-cluster size only changes who scores which child: results are identical."""
    from rag_cobweb_b200 import _lib
    L = _lib.load()
    x, _, ref = build_pair(400, 384, "unit")
    rl, rops, _ = ref.ifit(x, trace=True)
    try:
        for ncta in (1, 2, 4, 8, 16):
            _lib.check(L.cw_set_ifit_cluster(ncta))
            tree = CobwebTorchTree((384,))
            leaves, ops, _ = tree.ifit_batch(x, tag_sentences=True, trace=True)
            assert np.array_equal(ops, rops), ncta
            assert_same_tree(tree, ref, leaves.cpu().numpy(), rl)
        assert L.cw_set_ifit_cluster(3) != 0
    finally:
        L.cw_set_ifit_cluster(0)


def test_ifit_fast_arithmetic_is_ieee():
    """The branch-free division / logarithm of the ifit scoring jobs give the bits of the IEEE division and of the
    strict log on 2e8 pseudo-random and edge operands (zero numerators, all-ones mantissas, equal mantissas)."""
    from rag_cobweb_b200 import _lib
    L = _lib.load()
    out = torch.zeros(3, dtype=torch.int64, device="cuda")
    _lib.check(L.cw_selftest_arith(1 << 18, 800, 12345, out.data_ptr(), _lib.stream_ptr()), "cw_selftest_arith")
    bad_div, bad_log, tested = out.cpu().tolist()
    assert tested > 1e8
    assert bad_div == 0 and bad_log == 0


def test_derived_rows_follow_the_statistics():
    """cw_store.var / .tf (compute_var and its log, cached per node) are what the ifit kernel scores children from.  After
    every kind of update (increment, new, merge, split, fringe split, duplicates) they equal a fresh derivation from
    (m2, count) bit for bit, for every live node and every scoring mode; a tree reloaded from its arrays (derived rows
    rebuilt by cw_store_derive) keeps growing exactly like the oracle's."""
    for kw in (dict(), dict(use_kl=False), dict(use_info=False), dict(acuity_cutoff=True)):
        x, tree, ref = build_pair(700, 96, "whitened", dups=True, **kw)
        tree.ifit_batch(x[:400], tag_sentences=True)
        st = tree.store
        n_used = int(st.header()[1])
        live = (st.parent[:n_used] > -2) & (st.count[:n_used] > 0)
        var_k, tf_k = st.var[:n_used].clone(), st.tf[:n_used].clone()
        st.derive(n_used)
        assert torch.equal(st.var[:n_used][live], var_k[live]) and torch.equal(st.tf[:n_used][live], tf_k[live]), kw
        # the same tree rebuilt from its arrays (what load_json / load_snapshot do), then 300 more inserts
        b = tree.bfs()
        mean, m2 = st.rows(b["order"])
        tree2 = CobwebTorchTree((96,), **kw)
        tree2.load_arrays(b["parent"], b["count"], b["nsent"], mean, m2)
        leaves2 = tree2.ifit_batch(x[400:], tag_sentences=True)
        rl = ref.ifit(x)
        assert_same_tree(tree2, ref, leaves2.cpu().numpy(), rl[400:])


def test_ifit_is_deterministic_under_repetition():
    """The cluster protocol of cw_ifit (scores through distributed shared memory, CTAs running phases ahead of each other)
    must not let timing into the result: the same stream gives the same decision trace every time, for every cluster
    size, on shapes with one-warp and multi-warp teams and with many rounds per phase (high fan-out)."""
    from rag_cobweb_b200 import _lib
    L = _lib.load()
    try:
        for n, d, kind in ((4000, 128, "unit"), (3000, 768, "unit"), (4000, 256, "whitened")):
            x = torch.from_numpy(synth.corpus(n, d, kind, seed=3)).cuda()
            want = None
            for rep, ncta in enumerate((0, 0, 0, 8, 16, 4, 0)):
                _lib.check(L.cw_set_ifit_cluster(ncta))
                tree = CobwebTorchTree((d,))
                _, ops, off = tree.ifit_batch(x, tag_sentences=True, trace=True)
                if want is None:
                    want = (ops, off)
                assert np.array_equal(ops, want[0]) and np.array_equal(off, want[1]), (n, d, kind, rep, ncta)
    finally:
        L.cw_set_ifit_cluster(0)


def test_child_pool_compaction_keeps_the_tree():
    """Child lists are rewritten contiguously (leaked chunks dropped) without changing the tree, and
    inserts continue bit-exactly afterwards."""
    x, tree, ref = build_pair(2400, 64, "whitened")
    tree.ifit_batch(x[:1200], tag_sentences=True)
    used_before = int(tree.store.header()[3])
    b0 = tree.bfs()
    tree.store.compact_pool()
    assert int(tree.store.header()[3]) <= used_before
    b1 = tree.bfs()
    assert all(np.array_equal(b0[k], b1[k]) for k in ("order", "parent", "count", "nchild", "nsent"))
    leaves2 = tree.ifit_batch(x[1200:], tag_sentences=True)
    rl = ref.ifit(x)
    assert_same_tree(tree, ref, leaves2.cpu().numpy(), rl[1200:])


def test_ifit_capacity_growth_midway():
    x, tree, ref = build_pair(3000, 64, "unit")
    tree.IFIT_CHUNK = 700  # several launches, several reallocations of the store
    leaves = tree.ifit_batch(x, tag_sentences=True)
    rl = ref.ifit(x)
    assert tree.store.cap > 1024
    assert_same_tree(tree, ref, leaves.cpu().numpy(), rl)


@pytest.mark.parametrize("name", ["tiny_unit_64", "dups_unit_200x32", "unit_300x128", "whitened_600x256"])
def test_ifit_matches_reference_golden(golden_dir, name):
    """Cases where the reference's own decisions are free of fp32-summation-noise ties: the
    engine reproduces the reference tree outright."""
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    n, d, kind = int(g["n"]), int(g["d"]), str(g["kind"])
    x = synth.corpus(n, d, kind, seed=0)
    if name.startswith("dups"):
        x[50:60] = x[10:20]
        x[150:155] = x[10:15]
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    b = w.tree.bfs()
    assert np.array_equal(b["parent"], g["bfs_parent"])
    assert np.array_equal(b["count"], g["bfs_count"])
    pos = pos_of(b)
    assert np.array_equal(pos[w._leaf_of_sentence], g["leaf_of_sentence"])
    mean, m2 = w.tree.store.rows(b["order"][:1])
    assert np.array_equal(mean[0], g["mean_row0"]) and np.array_equal(m2[0], g["m2_row0"])
    # queries: best-first pop order and rows scored are the reference's; dense scores to fp32
    q, _ = synth.queries(x, g["rank_scores"].shape[0], kind, seed=1)
    k = int(g["k"])
    leaves, nfound, calls = w.predict_batch(q, k)
    assert np.array_equal(pos[leaves], g["bf_leaves"])
    assert np.array_equal(calls, g["bf_lp_calls"])
    best = w.tree.categorize_batch(q)["best"].cpu().numpy()
    assert np.array_equal(pos[best], g["cat_best"])
    rank = w.rank_scores_batch(q).cpu().numpy()
    np.testing.assert_allclose(rank, g["rank_scores"], rtol=2e-5)
    w.build_prediction_index()
    ns = w._index.node_scores(torch.from_numpy(q).cuda()).cpu().numpy()
    # score = -0.5 * (sumlog + quad) can cancel to ~0: absolute floor of a few ulps of |sumlog|
    floor = 8 * EPS32 * float(w._index.sumlog.abs().max())
    np.testing.assert_allclose(ns, g["node_scores"], rtol=2e-5, atol=floor)


@pytest.mark.parametrize("n,d,kind,k", [(600, 128, "unit", 10), (500, 256, "whitened", 5), (300, 1024, "unit", 10)])
def test_categorize_bit_exact_vs_oracle(n, d, kind, k):
    x, tree, ref = build_pair(n, d, kind)
    tree.ifit_batch(x, tag_sentences=True)
    ref.ifit(x)
    pos, rpos = assert_same_tree(tree, ref)
    q, _ = synth.queries(x, 64, kind, seed=1)
    r = tree.categorize_batch(q, retrieve_k=k, max_nodes=100000)
    rl, rnf, _, rcalls = ref.categorize(q, k=k, max_nodes=100000)
    assert np.array_equal(pos[r["leaves"].cpu().numpy()], rpos[rl])
    assert np.array_equal(r["nfound"].cpu().numpy(), rnf)
    assert np.array_equal(r["lp_calls"].cpu().numpy(), rcalls)
    # retrieve_k=None over the whole tree, greedy descent, and a max_nodes cut-off
    for kw in (dict(), dict(greedy=True), dict(max_nodes=7), dict(use_best=False, max_nodes=5)):
        got = tree.categorize_batch(q, **kw)
        _, _, rbest, rc = ref.categorize(q, k=0, **kw)
        assert np.array_equal(pos[got["best"].cpu().numpy()], rpos[rbest]), kw
        assert np.array_equal(got["lp_calls"].cpu().numpy(), rc), kw
    # reference error behaviour: more leaves requested than exist -> IndexError (CobwebTorchTree.py:289)
    with pytest.raises(IndexError):
        tree.categorize(q[0], retrieve_k=n + 5)
    one = tree.categorize(q[0], retrieve_k=3)
    assert [pos[h.node_id] for h in one] == list(rpos[rl[0, :3]])


@pytest.mark.parametrize("n,d,kind", [(700, 128, "unit"), (500, 256, "whitened"), (400, 1024, "unit"), (300, 100, "unit")])
def test_dense_predict_vs_oracle(n, d, kind):
    x = synth.corpus(n, d, kind, seed=0)
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    ref = OracleTree(d)
    ref.ifit(x)
    q, targets = synth.queries(x, 200, kind, seed=1)
    k = 10
    w.build_prediction_index()
    ix = ref.build_index()
    # index operands: sum of log-variances bit-exact
    assert np.array_equal(w._index.sumlog[: w._index.nn].cpu().numpy(), ix["sumlog"])
    rns, rls = ref.dense_scores(q)
    qd = torch.from_numpy(q).cuda()
    ns = w._index.node_scores(qd).cpu().numpy()
    # score = -0.5 * (sumlog + quad) can cancel to ~0: absolute floor of a few ulps of |sumlog|
    floor = 8 * EPS32 * float(np.abs(ix["sumlog"]).max())
    np.testing.assert_allclose(ns, rns, rtol=1e-5, atol=floor)
    ids, vals, leaf = w._index.predict(qd, k, want_leaf_scores=True)
    leaf, ids, vals = leaf.cpu().numpy(), ids.cpu().numpy(), vals.cpu().numpy()
    np.testing.assert_allclose(leaf, rls, rtol=1e-5, atol=floor)
    # path product: bit-exact given the same node scores (sequential fp32 FMA, root first)
    assert np.array_equal(leaf, oracle_leaf_scores(ns, ix["path_idx"], ix["path_w"]))
    # top-k: exact arg-sort of the engine's own leaf scores, ties by ascending sentence id
    want = np.argsort(-leaf, axis=1, kind="stable")[:, :k]
    assert np.array_equal(ids, want)
    assert np.array_equal(vals, np.take_along_axis(leaf, want, 1))
    # against the oracle's ranking: identical except inside fp32 near-ties
    rwant = np.argsort(-rls, axis=1, kind="stable")[:, :k]
    for i in range(len(q)):
        if not np.array_equal(rwant[i], ids[i]):
            s = rls[i]
            lo = s[rwant[i, -1]]
            near = set(np.nonzero(np.abs(s - lo) <= 2e-5 * abs(lo))[0])
            assert (set(rwant[i]) ^ set(ids[i])) <= near
    # recall@10 parity with the oracle (SURVEY 8d: target document among the returned ids)
    rec = np.mean([t in g for t, g in zip(targets, ids)])
    rrec = np.mean([t in g for t, g in zip(targets, rwant)])
    assert rec == rrec
    # host-buffer entry point (H2D + kernels + D2H in one C call) gives the same answer
    hs, hv = w._index.predict_host(q, k)
    assert np.array_equal(hs.numpy(), ids) and np.array_equal(hv.numpy(), vals)
    # reference-shaped single-query API
    assert w.cobweb_predict_fast(q[0], k=k, return_ids=True, is_embedding=True) == list(ids[0])
    np.testing.assert_array_equal(w.cobweb_rank_scores(torch.from_numpy(q[0]), is_embedding=True).cpu().numpy(), leaf[0])


def test_level_weights_and_large_k():
    n, d = 300, 64
    x = synth.corpus(n, d, "unit", seed=0)
    w = CobwebWrapper(corpus=[str(i) for i in range(n)], corpus_embeddings=x)
    ref = OracleTree(d)
    ref.ifit(x)
    q, _ = synth.queries(x, 16, "unit", seed=1)
    w.set_weight_schedule("exponential", max_depth=12, base=0.5)
    lw = w.get_level_weights()
    ref.build_index(level_weights=lw)
    _, rls = ref.dense_scores(q)
    np.testing.assert_allclose(w.rank_scores_batch(q).cpu().numpy(), rls, rtol=1e-5)
    # k >= number of sentences returns everything, sorted (CobwebWrapper.py:246-251)
    out = w.cobweb_predict_fast(q[0], k=n + 10, return_ids=True, is_embedding=True)
    assert sorted(out) == list(range(n))
    assert w.cobweb_predict_fast(q[0], k=3, is_embedding=True) == [str(i) for i in out[:3]]
    res = w.cobweb_predict(q[0], k=4, return_ids=True, is_embedding=True)
    rl, _, _, _ = ref.categorize(q[:1], k=4, max_nodes=100000)
    ref_sids = [int(np.nonzero(ref.leaf_of_sentence == l)[0][0]) for l in rl[0]]
    assert res == ref_sids


def test_json_roundtrip_on_device():
    n, d = 250, 48
    x = synth.corpus(n, d, "whitened", seed=0)
    w = CobwebWrapper(corpus=[f"s{i}" for i in range(n)], corpus_embeddings=x)
    q, _ = synth.queries(x, 8, "whitened", seed=1)
    before = w.predict_fast_batch(q, 5)[0].cpu().numpy()
    bf_before = [w.cobweb_predict(v, k=3, return_ids=True, is_embedding=True) for v in q]
    w2 = CobwebWrapper.load_json(w.dump_json())
    assert w2.sentences == w.sentences
    b, b2 = w.tree.bfs(), w2.tree.bfs()
    assert np.array_equal(b["parent"], b2["parent"]) and np.array_equal(b["count"], b2["count"])
    assert np.array_equal(w2.predict_fast_batch(q, 5)[0].cpu().numpy(), before)
    assert [w2.cobweb_predict(v, k=3, return_ids=True, is_embedding=True) for v in q] == bf_before
    # the tree keeps learning after a reload
    w2.add_sentences(["extra"], x[:1] + 0.01)
    assert len(w2) == n + 1


def test_properties_at_scale():
    """Size-independent invariants on a tree far larger than the oracle is asked to build:
    count conservation, leaves-only sentences, self-retrieval."""
    n, d = 20000, 256
    x = synth.corpus(n, d, "whitened", seed=0)
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    t = w.tree.store.topology()
    b = w.tree.bfs()
    assert b["count"][0] == n
    kids = b["nchild"] > 0
    csum = np.zeros(len(b["order"]))
    np.add.at(csum, b["parent"][1:], b["count"][1:])
    assert np.array_equal(csum[kids], b["count"][kids])          # every internal count = sum of children
    assert (b["nsent"][kids] == 0).all() and b["nsent"].sum() == n  # sentences live on leaves only
    assert (t["child_cnt"][w._leaf_of_sentence] == 0).all()
    q = x[:512]
    ids, vals = w.predict_fast_batch(q, 10)
    assert np.mean([i in g for i, g in enumerate(ids.cpu().numpy())]) > 0.99  # a document retrieves itself
    # the tensor-core path at this size (several node tiles per SM, whitened operands = the cancellation-heavy case):
    # same ids, same scores, on a batch that is not a multiple of any tile
    w.set_dense_mode("fused")
    qb, _ = synth.queries(x, 3001, "whitened", seed=2)
    ids_t, vals_t = w.predict_fast_batch(np.concatenate([q, qb]), 10)
    w.set_dense_mode("fp32")
    ids_f, vals_f = w.predict_fast_batch(np.concatenate([q, qb]), 10)
    assert torch.equal(ids_t, ids_f) and torch.equal(vals_t, vals_f)
    st = w._index.stats
    assert torch.equal(ids_t[:512], ids) and st["flagged"] <= 32 and st["audit_mismatch"] == 0 and st["queries"] == 512 + 3513, st
    # oracle cross-check on the engine-built tree: load it into the oracle, compare best-first on a sample
    mean, m2 = w.tree.store.rows(b["order"])
    ref = OracleTree(d)
    ref.load(b["parent"], b["count"], b["nsent"], mean, m2)
    qs, _ = synth.queries(x, 16, "whitened", seed=1)
    r = w.tree.categorize_batch(qs, retrieve_k=10, max_nodes=100000)
    rl, _, _, rc = ref.categorize(qs, k=10, max_nodes=100000)
    pos = pos_of(b)
    assert np.array_equal(pos[r["leaves"].cpu().numpy()], rl)  # oracle slots == BFS index after load()
    assert np.array_equal(r["lp_calls"].cpu().numpy(), rc)


def test_edge_cases_empty_and_tiny_trees():
    """Empty tree, single-instance tree, k larger than the corpus, ragged batch sizes."""
    d = 16
    tree = CobwebTorchTree((d,))
    x = synth.corpus(5, d, "unit", seed=3)
    # categorize on an empty tree returns the (empty) root like the reference's loop does
    assert tree.categorize(x[0]).node_id == tree.root.node_id
    with pytest.raises(IndexError):
        tree.categorize(x[0], retrieve_k=1)
    leaf = tree.ifit(x[0])
    assert leaf.node_id == tree.root.node_id and float(tree.root.count) == 1.0
    assert np.array_equal(tree.root.mean.cpu().numpy(), x[0])
    assert tree.root.children == [] and tree.root.parent is None
    # a second, different instance fringe-splits the root
    leaf2 = tree.ifit(x[1])
    assert len(tree.root.children) == 2 and leaf2.parent == tree.root and float(tree.root.count) == 2.0
    ref = OracleTree(d)
    ref.ifit(x[:2], tag_sentences=False)
    assert_same_tree(tree, ref)
    # wrapper on a 3-document corpus: k beyond the corpus returns everything, best-first too
    w = CobwebWrapper(corpus=["a", "b", "c"], corpus_embeddings=x[:3])
    assert sorted(w.cobweb_predict_fast(x[0], k=10, return_ids=True, is_embedding=True)) == [0, 1, 2]
    assert w.cobweb_predict_fast(x[1], k=1, is_embedding=True) == ["b"]
    assert w.cobweb_predict(x[2], k=1, return_ids=True, is_embedding=True) == [2]
    with pytest.raises(IndexError):
        w.cobweb_predict(x[0], k=7, return_ids=True, is_embedding=True)
    # ragged batches around the tile sizes of the dense path
    n = 400
    xs = synth.corpus(n, 40, "unit", seed=0)
    w2 = CobwebWrapper(corpus=[None] * n, corpus_embeddings=xs)
    q, _ = synth.queries(xs, 300, "unit", seed=1)
    full = w2.predict_fast_batch(q, 7)[0].cpu().numpy()
    for nq in (1, 31, 33, 127, 129, 257):
        assert np.array_equal(w2.predict_fast_batch(q[:nq], 7)[0].cpu().numpy(), full[:nq])
    # wrong dimension is rejected
    with pytest.raises(ValueError):
        w2.tree.ifit_batch(np.zeros((2, 41), np.float32))


def test_store_sharded_predict_matches_full():
    """SURVEY 8e row 2: every rank indexes only its share of the sentences and the nodes on their
    paths; merged per-rank top-k == the single-index answer.  Ranks emulated one after another."""
    from rag_cobweb_b200 import parallel
    n, d, k = 1500, 96, 10
    x = synth.corpus(n, d, "unit", seed=0)
    x[700:720] = x[10:30]  # duplicates: several sentences per leaf
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    q, _ = synth.queries(x, 100, "unit", seed=1)
    full_i, full_v = w.predict_fast_batch(q, k)
    for world in (2, 3):
        parts = [w.predict_fast_sharded(q, k, world=world, rank=r) for r in range(world)]
        nodes = []
        for r in range(world):
            w.predict_fast_sharded(q[:1], k, world=world, rank=r)
            nodes.append(w._shard_index.nn)
        assert max(nodes) < 0.8 * w._index.nn  # a shard really holds fewer nodes than the whole tree
        ci = torch.cat([p[0] for p in parts], 1)
        cv = torch.cat([p[1] for p in parts], 1)
        mi, mv = parallel.merge_topk(ci, cv, k)
        assert torch.equal(mi, full_i) and torch.equal(mv, full_v)
    # the same through the tensor-core modes (a shard index carries global sentence ids and its own row subset)
    for mode in ("fused",):
        w.set_dense_mode(mode)
        w._shard_key = None
        parts = [w.predict_fast_sharded(q, k, world=2, rank=r) for r in range(2)]
        mi, mv = parallel.merge_topk(torch.cat([p[0] for p in parts], 1), torch.cat([p[1] for p in parts], 1), k)
        assert torch.equal(mi, full_i) and torch.equal(mv, full_v), mode
    w.set_dense_mode("fp32")


def test_whitening_transform_matches_reference(golden_dir, tmp_path):
    """PCAICAWhiteningModel.transform on the device vs the reference's own outputs (fixture recorded
    by tests/golden/make_golden.py whitening).  fp32 GEMMs: 1e-4 relative to the row scale."""
    from rag_cobweb_b200 import PCAICAWhiteningModel
    g = np.load(os.path.join(golden_dir, "whitening_pcaica.npz"))
    m = PCAICAWhiteningModel(g["mean"], g["pca_components"], g["ica_unmixing"], g["pca_explained_var"], float(g["eps"]))
    for got, want in ((m.transform(g["x"]), g["y_ica"]), (m.transform(g["x"], is_ica=False), g["y_pca"]),
                      (m.transform(g["x"][0]), g["y_single"])):
        assert got.shape == want.shape
        np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * np.abs(want).max())
    # pickle layout of the reference (save / load), ragged batch sizes, and use as a wrapper front-end
    path = str(tmp_path / "w.pkl")
    m.save(path)
    m2 = PCAICAWhiteningModel.load(path)
    np.testing.assert_array_equal(m2.transform(g["x"][:3]), m.transform(g["x"])[:3])
    big = np.tile(g["x"], (5, 1))[:301]
    np.testing.assert_array_equal(m.transform(big)[:64], m.transform(g["x"]))
    yd = m.transform_device(g["x"])
    w = CobwebWrapper(corpus=[None] * len(yd), corpus_embeddings=yd)  # whitened vectors never leave the device
    assert w.cobweb_predict_fast(yd[3], k=1, return_ids=True, is_embedding=True) == [3]


def test_rank_scores_gradient_matches_torch_autograd():
    """Backward of cobweb_rank_scores w.r.t. the query against torch autograd of the reference's
    own expression (CobwebWrapper.py:283-292) evaluated in float64 on the oracle's index arrays."""
    n, d, nq = 500, 48, 37
    x = synth.corpus(n, d, "whitened", seed=0)
    x[100:110] = x[5:15]
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    ref = OracleTree(d)
    ref.ifit(x)
    ix = ref.build_index(level_weights=[1.0, 0.5, 2.0])
    w.set_level_weights([1.0, 0.5, 2.0])
    q, _ = synth.queries(x, nq, "whitened", seed=1)
    rng = np.random.default_rng(5)
    gl = rng.standard_normal((nq, n)).astype(np.float32)
    # engine
    Q = torch.from_numpy(q).cuda().requires_grad_(True)
    leaf = w.rank_scores_batch(Q)
    (leaf * torch.from_numpy(gl).cuda()).sum().backward()
    got = Q.grad.cpu().numpy()
    # torch reference (float64): node log-probs, path product as a dense matrix, autograd
    M, V = torch.from_numpy(ix["means"]).double(), torch.from_numpy(ix["vars"]).double()
    P = torch.zeros(n, M.shape[0], dtype=torch.float64)
    for l in range(n):
        for j, b in enumerate(ix["path_idx"][l]):
            if b >= 0:
                P[l, b] += float(ix["path_w"][l, j])
    Qr = torch.from_numpy(q).double().requires_grad_(True)
    s_nodes = -0.5 * (torch.log(V).sum(1)[None, :] + (((Qr[:, None, :] - M[None]) ** 2) / V[None]).sum(2))
    leaf_r = s_nodes @ P.T
    (leaf_r * torch.from_numpy(gl).double()).sum().backward()
    want = Qr.grad.numpy()
    np.testing.assert_allclose(leaf.detach().cpu().numpy(), leaf_r.detach().numpy(), rtol=1e-5, atol=1e-3)
    np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-4 * np.abs(want).max())
    # single-query reference-style call: gradient of the sum of all leaf scores
    x1 = torch.from_numpy(q[0]).cuda().requires_grad_(True)
    w.cobweb_rank_scores(x1, is_embedding=True).sum().backward()
    x1r = torch.from_numpy(q[0]).double().requires_grad_(True)
    s1 = -0.5 * (torch.log(V).sum(1) + (((x1r[None, :] - M) ** 2) / V).sum(1))
    (s1 @ P.T).sum().backward()
    np.testing.assert_allclose(x1.grad.cpu().numpy(), x1r.grad.numpy(), rtol=1e-4, atol=1e-4 * np.abs(x1r.grad.numpy()).max())


def test_wrapper_input_conventions():
    """The reference's callers pass lists, numpy rows, tensors and text + encode_func
    (CobwebWrapper.py:13-80, benchmark_utils.py:465-581): all of them work."""
    rng = np.random.default_rng(11)
    vocab = {f"doc {i}": rng.standard_normal(24).astype(np.float32) for i in range(60)}
    encode = lambda texts: np.stack([vocab[t] for t in texts])  # noqa: E731
    texts = list(vocab)
    w_text = CobwebWrapper(corpus=texts, encode_func=encode)                      # text only
    emb = encode(texts)
    w_np = CobwebWrapper(corpus=texts, corpus_embeddings=emb)                     # numpy matrix
    w_list = CobwebWrapper(corpus=texts, corpus_embeddings=emb.tolist())          # python lists
    w_t = CobwebWrapper(corpus=None, corpus_embeddings=torch.from_numpy(emb))     # tensor, embedding-only entries
    for w in (w_np, w_list, w_t):
        assert np.array_equal(w.tree.bfs()["parent"], w_text.tree.bfs()["parent"])
    assert w_t.sentences == [None] * 60 and len(w_text) == 60
    # query by text (encode_func), by numpy row positionally like retrieve_cobweb_basic, by tensor
    assert w_text.cobweb_predict_fast("doc 7", k=1) == ["doc 7"]
    assert w_np.cobweb_predict_fast(emb[7], k=1, return_ids=True) == [7]          # identity encode_func([q])[0]
    assert w_np.cobweb_predict(torch.from_numpy(emb[9]), k=1, return_ids=True, is_embedding=True) == [9]
    # add_sentences appends with running ids and invalidates the index
    w_np.build_prediction_index()
    extra = rng.standard_normal((3, 24)).astype(np.float32)
    w_np.add_sentences(["x", "y", "z"], extra)
    assert not w_np._prediction_index_valid and len(w_np) == 63
    assert w_np.cobweb_predict_fast(extra[1], k=1, is_embedding=True) == ["y"]
    assert set(w_np.sentence_to_node) == set(range(63))
    leaf = w_np.sentence_to_node[61]
    assert 61 in w_np.cobweb_predict(extra[1], k=1, return_ids=True, is_embedding=True) and leaf.children == []
    info = w_np.get_weight_schedule_info()
    assert info["schedule_type"] is None and w_np.get_prediction_index_info()["index_valid"]


@pytest.mark.parametrize("n,d,kind,k", [(700, 128, "unit", 10), (900, 256, "whitened", 5), (400, 1024, "unit", 10),
                                        (300, 100, "unit", 3), (1500, 40, "whitened", 16), (600, 384, "unit", 30)])
def test_fused_predict_matches_fp32_path(n, d, kind, k):
    """"fused" dense predict (cw_half.cu: fp16x3 internal rows -> cumulative sums, one-product fp16 leaf filter with its
    derived error bound, exact refine + re-score in the finish kernel) returns the FP32-pipe path's ids AND scores bit
    for bit, through the device call, the one-call host entry and the reference-shaped API; the cumulative ancestor
    sums it builds agree with the FP32 node scores far inside the 1e-4 relative bar of the contract."""
    x = synth.corpus(n, d, kind, seed=3)
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    q, _ = synth.queries(x, 333, kind, seed=4)  # not a multiple of the 256-query tile
    qd = torch.from_numpy(q).cuda()
    w.build_prediction_index()
    ix = w._index
    ns32 = ix.node_scores(qd).clone()
    ids32, v32, _ = ix.predict(qd, k)
    ix.set_mode("fused")
    assert ix.fused_ready(k)
    ids, vals, _ = ix.predict(qd, k)
    assert torch.equal(ids, ids32) and torch.equal(vals, v32)
    st = dict(ix.stats)
    assert st["queries"] == 333 and st["audit_mismatch"] == 0 and st["audited"] >= 1 and st["unresolved"] == 0, st
    assert st["flagged"] <= 4, st  # the line test holds for (nearly) every query on continuous data
    # root row of the cumulative sums = the root's node score: fp16 split operands vs the FP32 kernel
    F = ix.hx["F"]
    root = ix._hws["S"][0, :333]
    x2 = float((qd * qd).sum(1).max())
    floor = 2.0 ** -18 * 2.0 * (x2 / w.tree.store.prior_var + ix.hx["fi"].hmax)
    want = ns32[:, int(F["int_rows"][0])] * float(F["int_w"][0])
    assert bool(((root - want).abs() <= 1e-5 * want.abs() + floor).all()), float((root - want).abs().max())
    hs, hv = ix.predict_host(q, k)
    assert np.array_equal(hs.numpy(), ids32.cpu().numpy()) and np.array_equal(hv.numpy(), v32.cpu().numpy())
    # reference-shaped API (one query: the exact small-batch path)
    w.set_dense_mode("fused")
    assert w.cobweb_predict_fast(q[0], k=k, return_ids=True, is_embedding=True) == list(ids32[0].cpu().numpy())


def test_fused_predict_flagged_queries_and_fallbacks():
    """Queries the device cannot decide (duplicates: more equal-scoring sentences than the finish kernel's lists hold), k
    beyond the fused range, fewer sentences than k, a level-weight schedule: always the FP32 path's answer."""
    rng = np.random.default_rng(5)
    base = synth.corpus(40, 64, "unit", seed=6)
    # leaves with 150, 70 and 40 identical sentences: 150 > CW_FUSED_MAX_SENT
    x = np.concatenate([np.repeat(base[:1], 150, axis=0), np.repeat(base[1:2], 70, axis=0), np.repeat(base[2:3], 40, axis=0),
                        base[3:]]).astype(np.float32)
    x = x[rng.permutation(len(x))]
    w = CobwebWrapper(corpus=[None] * len(x), corpus_embeddings=x)
    q = np.concatenate([base[:3] + 1e-3, synth.queries(x, 61, "unit", seed=7)[0]]).astype(np.float32)
    qd = torch.from_numpy(q).cuda()
    for weights in (None, [1.0, 0.5, 2.0, 1.0, 0.25]):
        if weights is not None:
            w.set_level_weights(weights)
        w.build_prediction_index()
        ix = w._index
        for k in (1, 10, 30, 40, 128):  # 128: the fallback's top-k fills all four register slots of the merge
            ix.set_mode("fp32")
            ids32, v32, _ = ix.predict(qd, k, small=False)
            ix.set_mode("fused")
            for call in ("device", "host"):
                f0 = ix.stats["flagged"]
                if call == "device":
                    ids, vals, _ = ix.predict(qd, k, small=False)
                    assert torch.equal(ids, ids32) and torch.equal(vals, v32), (k, weights)
                else:
                    hs, hv = ix.predict_host(q, k)
                    assert np.array_equal(hs.numpy(), ids32.cpu().numpy()) and np.array_equal(hv.numpy(), v32.cpu().numpy()), k
                if k == 10 and weights is None:
                    # a query next to the 150-sentence leaf ranks it first: its sentences overflow the finish kernel's
                    # list, the query is flagged and answered by the exact small-batch path on the device
                    assert ix.stats["flagged"] - f0 >= 1 and ix.stats["unresolved"] == 0, ix.stats
    assert ix.stats["audit_mismatch"] == 0
    # fewer sentences than k
    w2 = CobwebWrapper(corpus=[None] * 12, corpus_embeddings=base[:12])
    w2.build_prediction_index()
    a, b, _ = w2._index.predict(qd, 20, small=False)
    c, e, _ = w2._index.set_mode("fused").predict(qd, 20, small=False)
    assert torch.equal(a, c) and torch.equal(b, e)
    # more flagged queries than the device-side rounds take (2 x 32): every query sits on the 150-sentence leaf
    qq = (np.repeat(base[:1], 200, axis=0) + 1e-4 * rng.standard_normal((200, 64))).astype(np.float32)
    w.set_level_weights(None)   # default weights: the query's own leaf ranks first
    w.build_prediction_index()
    ix = w._index
    ix.set_mode("fp32")
    i32, f32v, _ = ix.predict(torch.from_numpy(qq).cuda(), 10, small=False)
    ix.set_mode("fused")
    u0 = ix.stats["unresolved"]
    ids, vals, _ = ix.predict(torch.from_numpy(qq).cuda(), 10, small=False)
    assert torch.equal(ids, i32) and torch.equal(vals, f32v) and ix.stats["unresolved"] - u0 >= 100, ix.stats
    hs, hv = ix.predict_host(qq, 10)
    assert np.array_equal(hs.numpy(), i32.cpu().numpy()) and np.array_equal(hv.numpy(), f32v.cpu().numpy())


def test_small_batch_exact_path():
    """cw_small_predict (thread-per-node FP32 chains, HBM-bound for one query) = the big FP32 kernels bit for bit, for
    1..32 queries, odd D, through the device call, the host call and cobweb_predict_fast.  k = 64 puts rank k-1 in lane 31
    of the second register slot, 65 and 128 use the third and fourth slots of the merge and of the insertion loop."""
    for n, d, kind, k in ((900, 100, "unit", 10), (2000, 256, "whitened", 5), (300, 7, "whitened", 1), (600, 1030, "unit", 40),
                          (2000, 64, "unit", 64), (2500, 33, "whitened", 65), (3000, 128, "unit", 128)):
        x = synth.corpus(n, d, kind, seed=31)
        w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
        q, _ = synth.queries(x, 40, kind, seed=32)
        qd = torch.from_numpy(q).cuda()
        w.build_prediction_index()
        ix = w._index
        ids32, v32, _ = ix.predict(qd, k, small=False)
        for nq in (1, 2, 3, 8, 17, 32):
            a, b = ix.predict_small(qd[:nq].contiguous(), k)
            assert torch.equal(a, ids32[:nq]) and torch.equal(b, v32[:nq]), (n, d, nq)
            hs, hv = ix.predict_host(q[:nq], k)
            assert np.array_equal(hs.numpy(), ids32[:nq].cpu().numpy()) and np.array_equal(hv.numpy(), v32[:nq].cpu().numpy())
        assert w.cobweb_predict_fast(q[3], k=k, return_ids=True, is_embedding=True) == list(ids32[3].cpu().numpy())


def test_batched_evaluator_on_device():
    """evaluate_cobweb (evaluate_retrieval semantics, benchmark_utils.py:710-833) in both predict modes and the
    brute-force inner-product baseline (retrieve_torch_dot, :602-614) on a corpus with known targets."""
    from rag_cobweb_b200.evaluate import evaluate_cobweb, evaluate_dot, metrics_from_ids
    n, d = 800, 64
    x = synth.corpus(n, d, "unit", seed=8)
    q, targets = synth.queries(x, 200, "unit", seed=9)
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    fast = evaluate_cobweb(w, q, targets, top_k=10, mode="fast")
    ids, _ = w.predict_fast_batch(q, 10)
    assert fast["recall@10"] == round(float(np.mean([t in g for t, g in zip(targets, ids.cpu().numpy())])), 4)
    assert fast["recall@2"] <= fast["recall@5"] <= fast["recall@10"] and fast["mrr@10"] <= fast["recall@10"]
    w.set_dense_mode("fused")
    assert {k: v for k, v in evaluate_cobweb(w, q, targets, top_k=10, mode="fast").items() if "@" in k} == \
        {k: v for k, v in fast.items() if "@" in k}
    basic = evaluate_cobweb(w, q, targets, top_k=10, mode="basic")
    ref_ids = [w.cobweb_predict(qq, k=10, return_ids=True, is_embedding=True)[:10] for qq in q[:50]]
    pad = np.array([r + [-1] * (10 - len(r)) for r in ref_ids])
    assert metrics_from_ids("b", pad, targets[:50], 10, 0.0)["recall@10"] == \
        evaluate_cobweb(w, q[:50], targets[:50], top_k=10, mode="basic")["recall@10"]
    dot = evaluate_dot(x, q, targets, top_k=10)
    assert dot["recall@10"] >= 0.99 and basic["recall@10"] > 0.5


@pytest.mark.parametrize("n,d,kind,k,weights", [(6000, 64, "unit", 10, None), (5000, 96, "whitened", 5, [1.0, 0.5, 2.0, 1.5]),
                                                (700, 128, "unit", 10, None), (3000, 40, "unit", 16, None)])
def test_fused_predict_sampled_threshold_and_overflow(n, d, kind, k, weights):
    """The fused pipeline with a sampled threshold (6000/5000/3000 leaves = strided sample tiles; 700 = one sampled tile
    with a coarser stride), leaves with several sentences (duplicated documents), level weights,
    and candidate-buffer overflow: ids and scores bit-identical to the FP32-pipe path."""
    x = synth.corpus(n, d, kind, seed=11)
    x[100:130] = x[7]          # a leaf with 31 sentences
    x[200:203] = x[9]
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    if weights is not None:
        w.set_level_weights(weights)
    q, _ = synth.queries(x, 517, kind, seed=12)
    q[:3] = x[[7, 9, 11]] + 1e-3
    qd = torch.from_numpy(q).cuda()
    w.build_prediction_index()
    ix = w._index
    ids32, v32, _ = ix.predict(qd, k)
    ix.set_mode("fused")
    assert ix.mode == "fused" and ix.hx["n_s"] == ix.hx["n_leaf"] // 2048 + (512 <= ix.hx["n_leaf"] < 2048) >= 1
    ids, vals, _ = ix.predict(qd, k)
    assert torch.equal(ids, ids32) and torch.equal(vals, v32)
    hs, hv = ix.predict_host(q, k)
    assert np.array_equal(hs.numpy(), ids32.cpu().numpy()) and np.array_equal(hv.numpy(), v32.cpu().numpy())
    assert ix.stats["flagged"] <= 16 and ix.stats["audit_mismatch"] == 0, ix.stats
    if ix.hx["n_s"]:
        # the sampled threshold really filters: far fewer candidates than leaves
        assert ix.stats["candidates"] / ix.stats["queries"] < 0.2 * ix.hx["n_leaf"], ix.stats
    a, b, _ = ix.predict(qd[:40], k, small=False)  # one partial tile
    assert torch.equal(a, ids32[:40]) and torch.equal(b, v32[:40])
    # several chunks per call (work buffers sized for 256 queries): device and host entry
    budget, ix.SCORE_BUDGET_BYTES, ix._hws = ix.SCORE_BUDGET_BYTES, 1, None
    assert ix.fused_chunk_queries() == 256
    a, b, _ = ix.predict(qd, k)
    hs, hv = ix.predict_host(q, k)
    assert torch.equal(a, ids32) and torch.equal(b, v32) and np.array_equal(hs.numpy(), ids32.cpu().numpy())
    assert np.array_equal(hv.numpy(), v32.cpu().numpy())
    ix.SCORE_BUDGET_BYTES, ix._hws = budget, None
    # candidate-buffer overflow: with 8 slots per query nearly every query overflows, is flagged by the finish kernel and
    # answered by the exact path -- same result
    ix.FUSED_CAP, ix._hws, f0 = 8, None, ix.stats["cand_overflow"]
    a, b, _ = ix.predict(qd, k)
    assert torch.equal(a, ids32) and torch.equal(b, v32) and ix.stats["cand_overflow"] - f0 > 100


def test_fused_predict_small_and_odd_shapes():
    """The fused mode against the FP32 path on shapes around the tile edges: tiny trees, attribute counts that are not
    multiples of the 32-feature slab, k = 1, acuity cutoff, a custom prior variance, one-query batches; and a tree whose
    leaves do NOT have one variance for all attributes (loaded statistics), which takes the general operand layout."""
    cases = [(40, 7, "whitened", 1, {}), (257, 33, "unit", 4, {}), (2500, 200, "unit", 4, dict(acuity_cutoff=True)),
             (900, 9, "whitened", 3, dict(prior_var=0.01)), (3000, 17, "unit", 10, {})]
    for n, d, kind, k, kw in cases:
        x = synth.corpus(n, d, kind, seed=21)
        w = CobwebWrapper(corpus=[None], corpus_embeddings=x[:1])
        w.tree, w.sentences, w._leaf_of_sentence = CobwebTorchTree((d,), **kw), [], np.zeros(0, np.int32)  # tree with these flags
        w.add_sentences([None] * n, x)
        q, _ = synth.queries(x, 70, kind, seed=22)
        qd = torch.from_numpy(q).cuda()
        w.build_prediction_index()
        ix = w._index
        ids32, v32, _ = ix.predict(qd, k)
        ix.set_mode("fused")
        assert ix.hx["leaf_layout"] == 1
        for batch in (qd, qd[:1]):
            a, b, _ = ix.predict(batch, k, small=False)
            assert torch.equal(a, ids32[: len(batch)]) and torch.equal(b, v32[: len(batch)]), (n, d, kind, k, len(batch))
        assert ix.stats["audit_mismatch"] == 0
    # anisotropic leaves: perturb the M2 rows of the leaves so that their variances differ per attribute
    n, d, k = 2000, 48, 10
    x = synth.corpus(n, d, "whitened", seed=23)
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    leaves = torch.as_tensor(np.unique(w._leaf_of_sentence), device="cuda").long()
    g = torch.Generator(device="cuda").manual_seed(1)
    w.tree.store.m2[leaves] = 0.05 * torch.rand((len(leaves), d), device="cuda", generator=g)
    q, _ = synth.queries(x, 300, "whitened", seed=24)
    qd = torch.from_numpy(q).cuda()
    w.force_rebuild_index()
    ix = w._index
    ids32, v32, _ = ix.predict(qd, k, mode="fp32")
    ix.set_mode("fused")
    assert ix.hx["leaf_layout"] == 2
    a, b, _ = ix.predict(qd, k)
    assert torch.equal(a, ids32) and torch.equal(b, v32) and ix.stats["audit_mismatch"] == 0


def test_ifit_greedy_mode(golden_dir):
    """COBWEB_GREEDY_MODE (src/utils/constants.py; CobwebTorchTree.py:209-213): the kernel takes "new" at every internal
    node.  Equal to the reference's recorded tree, and to the oracle beyond the scoring lists' fan-out limit (the flat
    tree's root has one child per instance)."""
    from rag_cobweb_b200 import constants
    g = np.load(os.path.join(golden_dir, "greedy_unit_150x24.npz"))
    x = synth.corpus(150, 24, "unit", seed=0)
    x[40:50] = x[5:15]
    constants.COBWEB_GREEDY_MODE = True
    try:
        tree = CobwebTorchTree((24,))          # reads the module switch like the reference does
    finally:
        constants.COBWEB_GREEDY_MODE = False
    assert tree.greedy_mode and not CobwebTorchTree((24,)).greedy_mode
    tree.ifit_batch(x)
    b = tree.bfs()
    mean, m2 = tree.store.rows(b["order"])
    assert np.array_equal(b["parent"], g["bfs_parent"]) and np.array_equal(b["count"], g["bfs_count"])
    assert np.array_equal(mean, g["mean"]) and np.array_equal(m2, g["m2"])
    n, d = 3000, 16
    x = synth.corpus(n, d, "whitened", seed=2)
    tree, ref = CobwebTorchTree((d,), greedy_mode=True), OracleTree(d, greedy=True)
    leaves = tree.ifit_batch(x, tag_sentences=True).cpu().numpy()
    assert_same_tree(tree, ref, leaves, ref.ifit(x))
    assert tree.bfs()["nchild"][0] == n > 2048


def test_reference_json_fixture_and_snapshot(golden_dir, tmp_path):
    """A document written by the REFERENCE's dump_json (fixture): load -> the reference's own rank scores (2e-5), re-dump
    byte-identical; binary snapshot of the same wrapper: load -> identical answers."""
    import json
    doc = open(os.path.join(golden_dir, "reference_tree_80x12.json")).read()
    ans = np.load(os.path.join(golden_dir, "reference_tree_80x12_answers.npz"))
    w = CobwebWrapper.load_json(json.dumps({"tree": json.loads(doc), "sentences": [f"s{i}" for i in range(80)],
                                            "embedding_dim": 12}))
    assert w.tree.dump_json() == doc
    x = synth.corpus(80, 12, "unit", seed=0)
    x[30:33] = x[4]
    q, _ = synth.queries(x, 6, "unit", seed=1)
    got = w.rank_scores_batch(q).cpu().numpy()
    np.testing.assert_allclose(got, ans["rank_scores"], rtol=2e-5, atol=1e-5)
    assert [float(w.sentence_to_node[i].count) for i in range(80)] == ans["leaf_count"].tolist()
    # reading .sentence_id on a handle must not disturb later dumps / predicts (round-1 advisor finding)
    assert sorted(w.sentence_to_node[4].sentence_id) == [4, 30, 31, 32] or 4 in w.sentence_to_node[4].sentence_id
    ids0, v0 = w.predict_fast_batch(q, 5)
    means, vars_ = w.get_node_path_stats(7)
    assert means.shape == vars_.shape and means.shape[1] == 12 and w.get_node_path_stats(10 ** 6) == (None, None)
    path = str(tmp_path / "w.cwb")
    w.save_snapshot(path)
    w2 = CobwebWrapper.load_snapshot(path)
    assert w2.sentences == w.sentences and w2.tree.dump_json() == doc
    ids1, v1 = w2.predict_fast_batch(q, 5)
    assert torch.equal(ids0, ids1) and torch.equal(v0, v1)
    assert w2.cobweb_predict(q[0], k=3, return_ids=True, is_embedding=True) == w.cobweb_predict(q[0], k=3, return_ids=True, is_embedding=True)
    # a wrapper built here: .sentence_id before and after adding sentences, JSON and snapshot agree
    w3 = CobwebWrapper(corpus=[f"t{i}" for i in range(40)], corpus_embeddings=x[:40])
    assert w3.sentence_to_node[0].sentence_id == [0]
    w3.add_sentences([f"t{i}" for i in range(40, 80)], x[40:])
    assert 79 in w3.sentence_to_node[79].sentence_id and len(w3.cobweb_predict(q[0], k=3, return_ids=True, is_embedding=True)) >= 3
    w4 = CobwebWrapper.load_json(w3.dump_json())
    assert np.array_equal(w4._leaf_of_sentence >= 0, np.ones(80, bool)) and w4.tree.dump_json() == w3.tree.dump_json()
    w3.add_sentences(["x", "y", "z"], x[:2])   # more sentences than vectors: the reference zips (CobwebWrapper.py:70)
    assert len(w3) == 82 and len(w3._leaf_of_sentence) == 82


@pytest.mark.parametrize("name", ["cfg1_unit_1000x384", "cfg2_unit_1500x1024"])
def test_baseline_configs_vs_oracle(golden_dir, name):
    """BASELINE configs[0] (1,000 x 384) and configs[1] (1,500 x 1024) at full size: ifit traces / trees / statistics
    bit-exact against the oracle, best-first retrieval identical, dense scores within 1e-5; and the reference's OWN tree
    (fixture decisions replayed) queried by the engine returns the reference's recorded node scores."""
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    n, d, kind, k = int(g["n"]), int(g["d"]), str(g["kind"]), int(g["k"])
    x = synth.corpus(n, d, kind, seed=0)
    tree, ref = CobwebTorchTree((d,)), OracleTree(d)
    leaves, ops, offs = tree.ifit_batch(x, tag_sentences=True, trace=True)
    rl, rops, roffs = ref.ifit(x, trace=True)
    assert np.array_equal(ops, rops) and np.array_equal(offs, roffs)
    pos, rpos = assert_same_tree(tree, ref, leaves.cpu().numpy(), rl)
    q, _ = synth.queries(x, 64, kind, seed=1)
    r = tree.categorize_batch(q, retrieve_k=k, max_nodes=100000)
    cl, _, _, cc = ref.categorize(q, k=k, max_nodes=100000)
    assert np.array_equal(pos[r["leaves"].cpu().numpy()], rpos[cl]) and np.array_equal(r["lp_calls"].cpu().numpy(), cc)
    # the reference's tree: guided replay -> engine store -> node scores vs the reference's recorded ones
    ref2 = OracleTree(d)
    dec = g["ops"][g["ops"] < 4]
    l2, _, _ = ref2.ifit_guided(x, dec, g["dec_b1"], g["dec_b2"])
    rb = ref2.bfs()
    mean, m2 = ref2.rows(rb["order"])
    w = CobwebWrapper(corpus=[None], corpus_embeddings=x[:1])
    w.tree.load_arrays(rb["parent"], rb["count"], rb["nsent"], mean, m2)
    p2 = pos_of(rb)
    w.sentences, w._leaf_of_sentence = [None] * n, p2[l2].astype(np.int32)
    w._invalidate_prediction_index()
    w.build_prediction_index()
    qg, _ = synth.queries(x, g["rank_scores"].shape[0], kind, seed=1)
    ns = w._index.node_scores(torch.from_numpy(qg).cuda()).cpu().numpy()
    np.testing.assert_allclose(ns, g["node_scores"], rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(w.rank_scores_batch(qg).cpu().numpy(), g["rank_scores"], rtol=2e-5, atol=1e-4)
