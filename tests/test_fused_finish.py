"""The fused predict's finish stage (select -> exact pair scores -> line test -> exact pair scores -> path sums and top-k,
rag-cobweb_b200/csrc/cw_half.cu) on what the other fused tests do not reach: refine lists longer than one round of
exact rows and past CW_FUSED_KC1 (trees built directly, so the leaves are known), paths near the fused mode's depth limit (the ancestor lists), and chunks whose query
count is not a multiple of the queries per CTA.  Each case compares with the FP32 path bit for bit."""
import functools

import numpy as np
import pytest
import torch

from rag_cobweb_b200 import CobwebTorchTree, CobwebWrapper, synth

pytestmark = pytest.mark.gpu
KC1 = 64


def fused_vs_fp32(ix, qd, k):
    ids32, v32, _ = ix.predict(qd, k, mode="fp32")
    ix.TENSOR_MIN_NODES = 0  # these trees are small: run them on the fused pipeline all the same
    ix.set_mode("fused")
    assert ix.fused_ready(k)
    s0 = dict(ix.stats)
    ids, vals, _ = ix.predict(qd, k, small=False)
    st = {n: ix.stats[n] - s0[n] for n in ix.stats}
    assert torch.equal(ids, ids32) and torch.equal(vals, v32)
    assert st["queries"] == qd.shape[0] and st["unresolved"] == 0 and st["audit_mismatch"] == 0, st
    return st


@functools.lru_cache(maxsize=None)
def star(n_tied, d=16):
    """A root with n_tied leaves one part in 10^6 apart and 20 distant ones (one sentence each, prior_var = 1).  The
    tied leaves' a1 differ far less than their filter bound E, so every one of them is kept and needs the exact term."""
    rng = np.random.default_rng(n_tied)
    x0 = rng.standard_normal(d)
    leaves = np.concatenate([x0 + 1e-6 * rng.standard_normal((n_tied, d)), x0 + 3.0 + rng.standard_normal((20, d))])
    L = len(leaves)
    parent = np.concatenate([[-1], np.zeros(L, np.int64)])
    count = np.concatenate([[L], np.ones(L)])
    mean = np.concatenate([leaves.mean(0, keepdims=True), leaves])
    m2 = np.zeros_like(mean)
    m2[0] = ((leaves - mean[0]) ** 2).sum(0)
    nsent = np.concatenate([[0], np.ones(L, np.int32)]).astype(np.int32)
    leaf_of_sentence = rng.permutation(np.arange(1, L + 1)).astype(np.int32)
    mean32 = mean.astype(np.float32)
    w = CobwebWrapper(corpus=[None], corpus_embeddings=mean32[1:2])
    w.tree = CobwebTorchTree((d,), prior_var=1.0)
    w.tree.load_arrays(parent, count.astype(np.float32), nsent, mean32, m2.astype(np.float32))
    w.sentences, w._leaf_of_sentence = [None] * L, leaf_of_sentence
    w._invalidate_prediction_index()
    w.build_prediction_index()
    return w, x0.astype(np.float32)


@pytest.mark.parametrize("n_tied,k", [(40, 1), (40, 30), (100, 1), (100, 10), (100, 30)])
def test_refine_list_past_kc1(n_tied, k):
    """40 tied leaves: a refine list of 40 (three rounds of exact rows); 100: the list is cut at KC1 by (a1 desc, row
    asc) and U comes from the cut ones.  The ties cannot be told apart by the line test, so such queries are flagged
    and answered by the exact path: never wrong."""
    w, x0 = star(n_tied)
    rng = np.random.default_rng(k)
    q = x0 + 1e-3 * rng.standard_normal((37, len(x0))).astype(np.float32)
    st = fused_vs_fp32(w._index, torch.from_numpy(q).cuda(), k)
    assert st["refined"] == min(n_tied, KC1) * 37, st


@functools.lru_cache(maxsize=None)
def caterpillar(max_len, d=16):
    """A tree of depth max_len - 1: every internal node has one internal child and one leaf child (the deepest has two
    leaves), in BFS order, with consistent count / mean / m2; leaves hold 1 to 3 identical sentences."""
    L = max_len
    rng = np.random.default_rng(max_len)
    nn = 2 * L - 1
    internal = np.array([0] + [2 * t - 1 for t in range(1, L - 1)])
    leaf = np.array([2 * j for j in range(1, L - 1)] + [2 * L - 3, 2 * L - 2])
    parent = np.full(nn, -1, np.int64)
    parent[internal[1:]] = internal[:-1]
    parent[leaf[:L - 1]] = internal
    parent[leaf[L - 1]] = internal[L - 2]
    c = 1 + (np.arange(L) % 3 == 0) + (np.arange(L) % 5 == 0)
    count, mean, m2 = np.zeros(nn), np.zeros((nn, d)), np.zeros((nn, d))
    count[leaf], mean[leaf] = c, rng.standard_normal((L, d))
    for row in internal[::-1]:
        kids = np.nonzero(parent == row)[0]
        na, nb = count[kids[0]], count[kids[1]]
        delta = mean[kids[1]] - mean[kids[0]]
        count[row] = na + nb
        mean[row] = mean[kids[0]] + delta * nb / (na + nb)
        m2[row] = m2[kids[0]] + m2[kids[1]] + delta * delta * na * nb / (na + nb)
    nsent = np.zeros(nn, np.int32)
    nsent[leaf] = c
    leaf_of_sentence = rng.permutation(np.repeat(leaf, c)).astype(np.int32)
    mean32, m232 = mean.astype(np.float32), m2.astype(np.float32)
    w = CobwebWrapper(corpus=[None], corpus_embeddings=mean32[leaf[:1]])
    w.tree = CobwebTorchTree((d,), prior_var=1.0)
    w.tree.load_arrays(parent, count.astype(np.float32), nsent, mean32, m232)
    w.sentences, w._leaf_of_sentence = [None] * len(leaf_of_sentence), leaf_of_sentence
    w._invalidate_prediction_index()
    w.build_prediction_index()
    return w, mean32[leaf]


@pytest.mark.parametrize("max_len", [300, 500])
def test_deep_tree_through_fused_mode(max_len):
    """Paths of up to 500 nodes: the survivors' ancestor lists run to CW_FUSED_MSURV x max_len entries per query."""
    w, leaf_vecs = caterpillar(max_len)
    ix = w._index
    assert ix.max_len == max_len
    rng = np.random.default_rng(1)
    q = leaf_vecs[rng.integers(0, len(leaf_vecs), 45)] + 0.1 * rng.standard_normal((45, leaf_vecs.shape[1])).astype(np.float32)
    st = fused_vs_fp32(ix, torch.from_numpy(q).cuda(), 10)
    assert st["rescored"] > 0, st


def test_query_counts_off_the_cta_grid():
    """Chunks of 1, 7, 259 and 523 queries (and 256-query chunks with a remainder of 11): the per-query kernels take 8
    queries per CTA, the exact-score kernel 4."""
    x = synth.corpus(1500, 48, "whitened", seed=21)
    w = CobwebWrapper(corpus=[None] * len(x), corpus_embeddings=x)
    w.build_prediction_index()
    ix = w._index
    q, _ = synth.queries(x, 523, "whitened", seed=22)
    qd = torch.from_numpy(q).cuda()
    for n in (1, 7, 259, 523):
        st = fused_vs_fp32(ix, qd[:n], 10)
        assert st["flagged"] <= 4, st
    budget, ix.SCORE_BUDGET_BYTES, ix._hws = ix.SCORE_BUDGET_BYTES, 1, None
    try:
        assert ix.fused_chunk_queries() == 256
        st = fused_vs_fp32(ix, qd[:267], 7)
        assert st["flagged"] <= 4, st
    finally:
        ix.SCORE_BUDGET_BYTES, ix._hws = budget, None
