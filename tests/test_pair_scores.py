"""Exact scores of chosen (query, sentence) pairs (CobwebWrapper.score_sentences / rerank, cw_pair_scores and
cw_pair_scores_bwd in rag-cobweb_b200/csrc/cw_pairs.cu).

Forward: bit for bit rank_scores_batch(Q).gather(1, ids) on every valid entry and -inf on padding, across D (tails that
are not a multiple of 32), data kinds, level schedules, batch sizes, list widths (one past CW_PAIR_MAX_M, so two
column blocks), sharing patterns (random ids with repeats, siblings, every depth), deep caterpillar trees and a single
query whose list is spread over many (query, row block) work items.

Backward, against a float64 reference built from the index's own {r, mb} rows:
  dx[q, d] = -sum_c G[q, c] sum_j w(len_c, j) (x_d r_bd + mb_bd) r_bd,  b = path(ids[q, c], j).
Error bound (eps = 2^-23, u = eps / 2): the kernel sums G w into one coefficient per listed row (at most m terms, one
rounding of each fp32 weight and product), then sums gs (x r + mb) r over the n listed rows (x r + mb fused, two more
roundings per term).  Every term of the exact sum carries a relative error of at most (m + n + 4) u to first order, so
the check is (m + n + 8) * eps * T per element, T = sum of |G w (x r + mb) r| over every (c, j).  The same bound plus the
rank-score backward's (nn + 8) * eps * T covers the difference to rank_scores_batch(Q).backward(G scattered).
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from rag_cobweb_b200 import CobwebTorchTree, CobwebWrapper, DenseIndex, _lib, synth

pytestmark = pytest.mark.gpu
EPS32 = float(np.finfo(np.float32).eps)
WEIGHTS = [1.0, 0.5, 2.0, 0.25, 1.5]


# ------------------------------------------------------------------ trees
@functools.lru_cache(maxsize=None)
def corpus_tree(d, kind="unit", n=2000, weights=None):
    x = synth.corpus(n, d, kind, seed=d)
    x[300:340] = x[5]  # one leaf with 41 sentences: positions whose whole path repeats
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    w.set_dense_mode("fp32")
    if weights is not None:
        w.set_level_weights(list(weights))
    w.build_prediction_index()
    return w, x


@functools.lru_cache(maxsize=None)
def caterpillar(max_len, d=16):
    """Depth max_len - 1: every internal node has one internal child and one leaf child (the deepest has two leaves),
    BFS rows, consistent count / mean / m2, 1 to 3 sentences per leaf, sentence ids shuffled over the positions."""
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
    mean32 = mean.astype(np.float32)
    w = CobwebWrapper(corpus=[None], corpus_embeddings=mean32[leaf[:1]])
    w.tree = CobwebTorchTree((d,), prior_var=1.0)
    w.tree.load_arrays(parent, count.astype(np.float32), nsent, mean32, m2.astype(np.float32))
    w.sentences, w._leaf_of_sentence = [None] * len(leaf_of_sentence), leaf_of_sentence
    w._invalidate_prediction_index()
    w.set_dense_mode("fp32")
    w.build_prediction_index()
    return w, mean32[leaf]


def random_ids(rng, n, nq, m):
    """Ids with repeats inside a row and about one in eight -1."""
    ids = rng.integers(0, n, (nq, m))
    if m > 1:
        ids[:, m // 2] = ids[:, 0]
    ids[rng.random((nq, m)) < 0.125] = -1
    return torch.from_numpy(ids.astype(np.int32)).cuda()


def queries(x, nq, seed):
    q, _ = synth.queries(x, nq, "unit", seed=seed)
    return torch.from_numpy(q).cuda()


# ------------------------------------------------------------------ checks
def check_forward(w, Q, ids):
    got = w.score_sentences(Q, ids)
    leaf = w.rank_scores_batch(Q)
    valid = ids >= 0
    want = leaf.gather(1, ids.clamp_min(0).long())
    assert got.shape == ids.shape and got.dtype == torch.float32
    assert torch.equal(got[valid], want[valid]), f"{int((got[valid] != want[valid]).sum())} scores differ"
    assert bool((got[~valid] == float("-inf")).all())
    return got


def grad_reference(index, x, ids, G):
    """float64 dx and the per-element bound (module docstring) from the index's rows and paths."""
    rows = index.rows().double().cpu().numpy()             # [nn, D, 2]
    path = index.path_idx.cpu().numpy()
    rec = index.pos_rec.cpu().numpy()
    pos = index.pos_of_sid().cpu().numpy()
    lw = index.level_w.cpu().numpy()
    x = x.astype(np.float64)
    nq, m = ids.shape
    dx, T = np.zeros_like(x), np.zeros_like(x)
    n_rows = 0
    for q in range(nq):
        gs = {}
        for c in range(m):
            sid = ids[q, c]
            if sid < 0:
                continue
            p = pos[sid]
            ln = rec[p, 0]
            for j in range(ln):
                b = path[p, j]
                wj = float(np.float32(lw[j] / ln))
                gs.setdefault(b, []).append(float(G[q, c]) * wj)
        n_rows = max(n_rows, sum(len(v) for v in gs.values()))
        for b, terms in gs.items():
            r, mb = rows[b, :, 0], rows[b, :, 1]
            t = (x[q] * r + mb) * r
            dx[q] -= sum(terms) * t
            T[q] += sum(abs(v) for v in terms) * np.abs(t)
    return dx, T, n_rows


def assert_within(got, want, bound, what):
    err = np.abs(np.asarray(got, np.float64) - want)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} elements outside the bound; first at "
                           f"{np.argwhere(bad)[0].tolist()}, worst err / bound {np.nanmax(err / np.maximum(bound, 1e-300)):.3g}")


def check_backward(w, Q, ids, seed):
    index = w._index
    nq, m = ids.shape
    G = torch.from_numpy(np.random.default_rng(seed).standard_normal((nq, m)).astype(np.float32)).cuda()
    Gw = torch.where(ids >= 0, G, 0.0)
    Qt = Q.clone().requires_grad_(True)
    w.score_sentences(Qt, ids).backward(Gw)
    got = Qt.grad.clone()
    dx, T, n_rows = grad_reference(index, Q.cpu().numpy(), ids.cpu().numpy(), G.cpu().numpy())
    bound = (m + n_rows + 8) * EPS32 * T
    assert_within(got.cpu().numpy(), dx, bound, "pair backward vs float64")
    # the dense backward on the same gradient scattered into [nq, L]
    Gs = torch.zeros((nq, len(w)), device="cuda")
    valid = ids >= 0
    qi = torch.arange(nq, device="cuda")[:, None].expand(nq, m)
    Gs.index_put_((qi[valid], ids[valid].long()), G[valid], accumulate=True)
    Qr = Q.clone().requires_grad_(True)
    w.rank_scores_batch(Qr).backward(Gs)
    assert_within(got.cpu().numpy(), Qr.grad.cpu().numpy(), bound + (index.nn + 8) * EPS32 * T, "pair vs rank backward")
    # the same bits on a second run
    Qt2 = Q.clone().requires_grad_(True)
    w.score_sentences(Qt2, ids).backward(Gw)
    assert torch.equal(Qt2.grad, got)
    return got


# ------------------------------------------------------------------ forward
@pytest.mark.parametrize("d,kind,weights", [
    pytest.param(7, "unit", None, id="D7-unit"),
    pytest.param(100, "whitened", WEIGHTS, id="D100-whitened-nonuniform-weights"),
    pytest.param(768, "unit", WEIGHTS, id="D768-unit-nonuniform-weights"),
    pytest.param(1030, "whitened", None, id="D1030-whitened-tail-6"),
])
def test_forward_bit_exact(d, kind, weights):
    """nq in {1, 33, 300} x m in {1, 31, 33, 500}, and m = CW_PAIR_MAX_M + 76 (two column blocks), random ids with
    repeats and -1."""
    w, x = corpus_tree(d, kind, weights=None if weights is None else tuple(weights))
    rng = np.random.default_rng(d)
    for nq in (1, 33, 300):
        Q = queries(x, nq, seed=nq + d)
        for m in (1, 31, 33, 500):
            check_forward(w, Q, random_ids(rng, len(w), nq, m))
    Q = queries(x, 33, seed=d)
    check_forward(w, Q, random_ids(rng, len(w), 33, _lib.PAIR_MAX_M + 76))


def test_forward_sharing_patterns():
    """All candidates the sentences under one parent (maximal sharing), candidates at every depth, one shared list
    given as [m], and a single [D] query."""
    w, x = corpus_tree(100)
    index = w._index
    rec, path = index.pos_rec.cpu().numpy(), index.path_idx.cpu().numpy()
    par = path[np.arange(len(rec)), rec[:, 0] - 2]
    best = np.bincount(par).argmax()
    sib = rec[par == best, 3]
    assert len(sib) >= 8
    Q = queries(x, 33, seed=5)
    check_forward(w, Q, torch.from_numpy(np.tile(sib, (33, 1)).astype(np.int32)).cuda())
    depths = np.unique(rec[:, 0])
    assert len(depths) >= 4
    per_depth = np.concatenate([rec[rec[:, 0] == ln, 3][:6] for ln in depths])
    ids = torch.from_numpy(np.tile(per_depth, (33, 1)).astype(np.int32)).cuda()
    check_forward(w, Q, ids)
    shared = w.score_sentences(Q, ids[0])
    assert torch.equal(shared, w.score_sentences(Q, ids))
    one = w.score_sentences(Q[0], ids[0])
    assert one.shape == (ids.shape[1],) and torch.equal(one, shared[0])


@pytest.mark.parametrize("max_len", [600, 1000])
def test_forward_deep_caterpillar(max_len):
    w, leaf_vecs = caterpillar(max_len)
    assert w._index.max_len == max_len
    rng = np.random.default_rng(max_len)
    q = (leaf_vecs[rng.integers(0, len(leaf_vecs), 33)] + 0.05 * rng.standard_normal((33, leaf_vecs.shape[1])))
    Q = torch.from_numpy(q.astype(np.float32)).cuda()
    check_forward(w, Q, random_ids(rng, len(w), 33, 200))
    check_backward(w, Q[:3].contiguous(), random_ids(rng, len(w), 3, 40), seed=max_len)


def test_forward_one_query_long_list():
    """One query with 3000 candidates, every sentence once plus repeats: three column blocks, each list spread over
    hundreds of (query, row block) work items."""
    w, x = corpus_tree(100)
    rng = np.random.default_rng(1)
    ids = np.concatenate([rng.permutation(len(w)), rng.integers(0, len(w), 1000)])[None, :3000]
    check_forward(w, queries(x, 1, seed=9), torch.from_numpy(ids.astype(np.int32)).cuda())


# ------------------------------------------------------------------ rerank
@pytest.mark.parametrize("mode", ["fp32", "fused"])
def test_rerank_equals_predict(mode):
    w, x = corpus_tree(100, n=3000)
    w.set_dense_mode(mode)
    w._index.TENSOR_MIN_NODES = 0  # a small tree: run it on the fused pipeline all the same
    try:
        Q = queries(x, 300, seed=11)
        all_ids = torch.arange(len(w), dtype=torch.int32, device="cuda")
        for k in (1, 10, 128):
            want_i, want_v = w.predict_fast_batch(Q, k)
            got_i, got_v = w.rerank(Q, all_ids, k)
            assert torch.equal(got_i, want_i) and torch.equal(got_v, want_v), k
        top_i, _ = w.predict_fast_batch(Q, 128)
        want_i, want_v = w.predict_fast_batch(Q, 10)
        got_i, got_v = w.rerank(Q, top_i, 10)
        assert torch.equal(got_i, want_i) and torch.equal(got_v, want_v)
    finally:
        w._index.TENSOR_MIN_NODES = DenseIndex.TENSOR_MIN_NODES
        w.set_dense_mode("fp32")


def test_rerank_padding_and_repeats():
    w, x = corpus_tree(100)
    Q = queries(x, 2, seed=3)
    ids = torch.tensor([[5, -1, 5, 9], [-1, -1, -1, 2]], dtype=torch.int32, device="cuda")
    got_i, got_v = w.rerank(Q, ids, 6)
    s = w.score_sentences(Q, ids)
    assert got_i.shape == (2, 6) and got_i.dtype == torch.int32
    assert sorted(got_i[0, :3].tolist()) == [5, 5, 9] and got_i[0, 3:].tolist() == [-1, -1, -1]
    assert got_i[1].tolist() == [2, -1, -1, -1, -1, -1] and float(got_v[1, 0]) == float(s[1, 3])
    assert bool((got_v[:, 3:] == float("-inf")).all()) and bool((got_v[0, :2] >= got_v[0, 1:3]).all())


# ------------------------------------------------------------------ backward
@pytest.mark.parametrize("d,weights", [
    pytest.param(7, None, id="D7"),
    pytest.param(100, WEIGHTS, id="D100-nonuniform-weights"),
    pytest.param(1030, None, id="D1030"),
])
def test_backward(d, weights):
    w, x = corpus_tree(d, "whitened" if d == 1030 else "unit", weights=None if weights is None else tuple(weights))
    rng = np.random.default_rng(d)
    for nq, m in ((1, 31), (33, 33), (5, _lib.PAIR_MAX_M + 10)):
        check_backward(w, queries(x, nq, seed=d + m), random_ids(rng, len(w), nq, m), seed=d + nq)


def test_backward_padding_and_repeats():
    w, x = corpus_tree(100)
    Q = queries(x, 2, seed=4)

    def grad(ids, G):
        Qt = Q.clone().requires_grad_(True)
        w.score_sentences(Qt, torch.tensor(ids, dtype=torch.int32, device="cuda")).backward(
            torch.tensor(G, dtype=torch.float32, device="cuda"))
        return Qt.grad

    assert bool((grad([[-1, -1], [-1, -1]], [[3.0, 1.0], [2.0, 5.0]]) == 0).all())
    a = grad([[7, -1], [8, 9]], [[1.5, 0.0], [1.0, -2.0]])
    assert torch.equal(a, grad([[7, -1], [8, 9]], [[1.5, 123.0], [1.0, -2.0]]))  # a padding entry's G is never read
    twice = grad([[7, 7], [8, 9]], [[1.0, 0.5], [1.0, -2.0]])
    once = grad([[7, -1], [8, 9]], [[1.5, 0.0], [1.0, -2.0]])
    assert torch.allclose(twice, once, rtol=1e-5, atol=1e-6) and torch.equal(twice[1], once[1])


# ------------------------------------------------------------------ errors
def test_errors():
    w, x = corpus_tree(100)
    Q = queries(x, 2, seed=2)
    with pytest.raises(ValueError):
        w.score_sentences(Q, torch.tensor([[0, -2]], device="cuda").expand(2, -1))
    with pytest.raises(ValueError):
        w.score_sentences(Q, [len(w)])
    with pytest.raises(ValueError):
        w.rerank(Q, [len(w) + 5], 1)
    shard = DenseIndex(w.tree, w._leaf_of_sentence, None, sentence_ids=np.arange(0, len(w), 2))
    with pytest.raises(ValueError, match="shard"):
        shard.pair_scores(Q, torch.zeros((2, 1), dtype=torch.int32, device="cuda"))
    index = w._index
    m = _lib.PAIR_MAX_M + 1
    ids = torch.zeros((2, m), dtype=torch.int32, device="cuda")
    out = torch.empty((2, m), device="cuda")
    scratch = torch.empty(16, dtype=torch.int32, device="cuda")
    L = _lib.load()
    rc = L.cw_pair_scores(C.byref(index.ix), index.rows().data_ptr(), index.pos_of_sid().data_ptr(), index.n_pos,
                          Q.data_ptr(), 2, ids.data_ptr(), m, out.data_ptr(), scratch.data_ptr(), _lib.stream_ptr())
    assert rc == _lib.CW_E_ARG and f"m={m}" in L.cw_last_error().decode()
