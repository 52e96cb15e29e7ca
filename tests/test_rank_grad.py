"""Backward of the rank scores (cw_rank_scores_bwd, rag-cobweb_b200/csrc/cw_grad.cu) against float64 references built
from the CPU oracle's index arrays, on the grid shapes and branches of its two kernels:

  kernel 1, paths_transpose_kernel:  gs[n, q] = sum over the positions l below node n of path_w[l, depth n] * G[q, l]
  kernel 2, rank_grad_kernel:        dx[q, d] = -sum_n gs[n, q] (x_qd - mean_nd) / var_nd

Error bounds (eps = 2^-23, u = eps / 2):
  * gs: node n sums n_terms(n) products w * G: the first product of a run is rounded once, the rest of the run is fused
    multiply-adds, runs and chunks are joined by atomicAdd in any order.  Any order of summing m terms stays within
    gamma_(m-1) * sum |terms| of the exact sum, and the rounded product adds u * |w G|, so the first-order bound is
    n_terms * u * sum |w G|.  The check is n_terms * eps * sum |w G| per element (c = 1: twice the first-order bound,
    which covers the higher-order terms since n_terms * u << 1).  A bound relative to the largest element instead would
    hide one dropped leaf contribution at the root.
  * dx from the kernel's own gs: r = 1/sqrtf(var) and mb = -mean * r carry at most 1.5u and 2.5u; the kernel's r * r and
    mb * r add one rounding each (4u of 1/var, 5u of mean/var); the two sums over the nn index rows add gamma_nn; the
    final x * a1 + a2 at most 2u.  First order: (nn + 7) u * sum_n |gs| (|x| r^2 + |mb r|).  The check is
    (nn + 8) * eps times that sum.  x * a1 + a2 cancels when x is near the means, so a relative tolerance is wrong there.
  * dx through the wrapper (gs not visible): the same with |gs_ref| + E_n in place of |gs|, plus
    sum_n E_n (|x| r^2 + |mb r|), where E_n is the gs bound above.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from oracle.cobweb_oracle import OracleTree, leaf_scores as oracle_leaf_scores
from rag_cobweb_b200 import CobwebTorchTree, CobwebWrapper, _lib, synth

pytestmark = pytest.mark.gpu
EPS32 = float(np.finfo(np.float32).eps)
LONG_WEIGHTS = [1.0 + 0.25 * (j % 5) for j in range(40)]  # longer than any path of the trees below


# ------------------------------------------------------------------ trees
def oracle_for(w):
    """The engine's tree loaded into the oracle (slots = BFS rows of the engine's index) with the same sentence map."""
    b = w.tree.bfs()
    mean, m2 = w.tree.store.rows(b["order"])
    ref = OracleTree(w.tree.d)
    ref.load(b["parent"], b["count"], b["nsent"], mean, m2)
    pos = np.full(int(b["order"].max()) + 1, -1, np.int64)
    pos[b["order"]] = np.arange(len(b["order"]))
    ref.leaf_of_sentence = pos[w._leaf_of_sentence].astype(np.int32)
    ref.n_sentences = len(w._leaf_of_sentence)
    return ref


@functools.lru_cache(maxsize=None)
def corpus_tree(d):
    """3000 documents (about 12 position chunks of 250 in kernel 1), one of them 301 times: a leaf whose sentences run
    across a chunk boundary (positions with m == len on both sides), and one 41 times."""
    n = 3000
    x = synth.corpus(n, d, "unit", seed=0)
    x[500:800] = x[7]
    x[1500:1540] = x[9]
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    return w, oracle_for(w), x


@functools.lru_cache(maxsize=None)
def caterpillar(max_len, d=16):
    """A tree of depth max_len - 1 in which every internal node has one internal child and one leaf child (the deepest
    internal node has two leaves), built in BFS order (level t = [internal t, leaf t-1]) with consistent count / mean /
    m2.  Leaves sit at every depth, so consecutive positions have different path lengths (stored prefix 0) while sharing
    every ancestor but the last.  Leaves hold 1 to 3 identical sentences; sentence ids are shuffled over the positions.
    prior_var = 1 keeps every variance >= 1, so every node score is <= 0 and leaf sums of up to 1000 terms do not cancel
    (the forward check against the oracle is relative)."""
    L = max_len
    rng = np.random.default_rng(max_len)
    nn = 2 * L - 1
    internal = np.array([0] + [2 * t - 1 for t in range(1, L - 1)])       # row of internal node t
    leaf = np.array([2 * j for j in range(1, L - 1)] + [2 * L - 3, 2 * L - 2])  # row of leaf j (leaf j is a child of internal j)
    parent = np.full(nn, -1, np.int64)
    parent[internal[1:]] = internal[:-1]
    parent[leaf[:L - 1]] = internal
    parent[leaf[L - 1]] = internal[L - 2]
    c = 1 + (np.arange(L) % 3 == 0) + (np.arange(L) % 5 == 0)
    count, mean, m2 = np.zeros(nn), np.zeros((nn, d)), np.zeros((nn, d))
    count[leaf], mean[leaf] = c, rng.standard_normal((L, d))
    for row in internal[::-1]:   # children have larger rows: combine them bottom-up (Chan et al. pairwise update)
        kids = np.nonzero(parent == row)[0]
        na, nb = count[kids[0]], count[kids[1]]
        delta = mean[kids[1]] - mean[kids[0]]
        count[row] = na + nb
        mean[row] = mean[kids[0]] + delta * nb / (na + nb)
        m2[row] = m2[kids[0]] + m2[kids[1]] + delta * delta * na * nb / (na + nb)
    nsent = np.zeros(nn, np.int32)
    nsent[leaf] = c
    leaf_of_sentence = rng.permutation(np.repeat(leaf, c)).astype(np.int32)
    n = len(leaf_of_sentence)
    mean32, m232 = mean.astype(np.float32), m2.astype(np.float32)
    w = CobwebWrapper(corpus=[None], corpus_embeddings=mean32[leaf[:1]])
    w.tree = CobwebTorchTree((d,), prior_var=1.0)
    w.tree.load_arrays(parent, count.astype(np.float32), nsent, mean32, m232)
    w.sentences, w._leaf_of_sentence = [None] * n, leaf_of_sentence
    w._invalidate_prediction_index()
    ref = OracleTree(d, prior_var=1.0)
    ref.load(parent, count.astype(np.float32), nsent, mean32, m232)
    ref.leaf_of_sentence, ref.n_sentences = leaf_of_sentence, n
    return w, ref, mean32[leaf]


def index_pair(w, ref, weights):
    """Engine index and oracle index arrays for one level-weight list; the engine's per-position paths must be the
    oracle's per-sentence paths."""
    w.set_level_weights(weights)
    w.build_prediction_index()
    index = w._index
    ix = ref.build_index(level_weights=weights)
    rec = index.pos_rec.cpu().numpy()
    path = index.path_idx.cpu().numpy()
    assert ix["path_idx"].shape[1] == index.max_len
    assert np.array_equal(path, ix["path_idx"][rec[:, 3]])
    return index, ix


# ------------------------------------------------------------------ references
def node_grad_ref(ix, G):
    """float64 gs_ref [nn, nq], sum |w G| [nn, nq] and the number of terms per node [nn], one level at a time."""
    P, W = ix["path_idx"], ix["path_w"].astype(np.float64)
    nn, nq = ix["means"].shape[0], G.shape[0]
    Gt = G.T.astype(np.float64)
    gs, ab, terms = np.zeros((nn, nq)), np.zeros((nn, nq)), np.zeros(nn)
    for j in range(P.shape[1]):
        ok = P[:, j] >= 0
        t = W[ok, j, None] * Gt[ok]
        np.add.at(gs, P[ok, j], t)
        np.add.at(ab, P[ok, j], np.abs(t))
        np.add.at(terms, P[ok, j], 1.0)
    return gs, ab, terms


def query_grad_ref(ix, x, gs, extra=None):
    """float64 dx[q, d] = -sum_n gs[n, q] (x_qd - mean_nd) / var_nd and its error bound (module docstring); extra = the
    per-element bound of gs when gs is the reference rather than the values the kernel read."""
    mu, iv, x = ix["means"].astype(np.float64), 1.0 / ix["vars"].astype(np.float64), x.astype(np.float64)
    dx = -(x * (gs.T @ iv) - gs.T @ (mu * iv))
    scale = lambda g: np.abs(x) * (g.T @ iv) + g.T @ (np.abs(mu) * iv)  # noqa: E731  sum_n g (|x| r^2 + |mb r|)
    g = np.abs(gs) if extra is None else np.abs(gs) + extra
    bound = (len(mu) + 8) * EPS32 * scale(g)
    if extra is not None:
        bound += scale(extra)
    return dx, bound


def assert_within(got, want, bound, what):
    err = np.abs(np.asarray(got, np.float64) - want)
    bad = ~(err <= bound)   # NaN fails
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} elements outside the bound; first at "
                           f"{np.argwhere(bad)[0].tolist()}, worst err / bound {np.nanmax(err / np.maximum(bound, 1e-300)):.3g}")


def bwd_direct(index, Q, G, pad=5):
    """cw_rank_scores_bwd on caller-owned buffers: gs scratch [nn, nq + pad] (an ldq larger than nq), grad_q prefilled
    with NaN (an element the kernel does not write fails every check)."""
    nq = Q.shape[0]
    gs = torch.full((index.nn, nq + pad), float("nan"), device="cuda")
    out = torch.full_like(Q, float("nan"))
    _lib.check(_lib.load().cw_rank_scores_bwd(C.byref(index.ix), Q.data_ptr(), nq, G.data_ptr(), gs.data_ptr(), nq + pad,
                                              out.data_ptr(), _lib.stream_ptr()), "cw_rank_scores_bwd")
    return gs.cpu().numpy(), out.cpu().numpy()


def transpose_chunk_len(n_pos, nq):
    """Positions per chunk of kernel 1 (the launch formula of cw_rank_scores_bwd)."""
    groups = (nq + 31) // 32
    want = max(1, min((148 * 32 + groups - 1) // groups, (n_pos + 255) // 256))
    return -(-n_pos // want)


def branch_positions(index, nq):
    """Positions at which kernel 1 takes each of its branches: first and last of every chunk, a path-length change, a
    stored prefix of 0 with shared leading nodes (most shared first), further sentences of one leaf, and the first
    position of a chunk whose leaf continues from the previous chunk (if any)."""
    rec, path = index.pos_rec.cpu().numpy(), index.path_idx.cpu().numpy()
    n, cl = len(rec), transpose_chunk_len(index.n_pos, nq)
    firsts = list(range(0, n, cl))
    lasts = [min(n, p + cl) - 1 for p in firsts]
    p = np.arange(1, n)
    len_change = p[rec[1:, 0] != rec[:-1, 0]]
    lead = np.cumprod((path[1:] == path[:-1]) & (path[1:] >= 0), axis=1).sum(1)
    zero = (rec[1:, 1] == 0) & (lead > 0) & (p % cl != 0)
    shared0 = p[zero][np.argsort(-lead[zero], kind="stable")]
    same_leaf = p[rec[1:, 2] == rec[:-1, 2]]
    straddle = [c for c in firsts[1:] if rec[c, 2] == rec[c - 1, 2]]
    assert len(len_change) and len(shared0) and len(same_leaf)
    picks = firsts + lasts + list(len_change[:4]) + list(shared0[:4]) + list(same_leaf[::max(1, len(same_leaf) // 8)]) + straddle
    return sorted(set(int(v) for v in picks)), straddle


# ------------------------------------------------------------------ checks
def check_one_hot(index, ix, Q, picks, rng):
    """One 1.0 per query at a chosen position: gs must be the fp32 path weights of that one path bit for bit and exactly
    0 everywhere else (padding columns of the ldq stride included).  Any dropped, doubled or misrouted flush fails."""
    nq = Q.shape[0]
    rec = index.pos_rec.cpu().numpy()
    for lo in range(0, len(picks), nq):
        chosen = np.array(picks[lo:lo + nq] + list(rng.integers(0, index.n_pos, max(0, nq - len(picks[lo:lo + nq])))))
        sid = rec[chosen, 3]
        G = np.zeros((nq, index.n_pos), np.float32)
        G[np.arange(nq), sid] = 1.0
        gs, _ = bwd_direct(index, Q, torch.from_numpy(G).cuda())
        want = np.zeros((index.nn, nq), np.float32)
        for q, s in enumerate(sid):
            ok = ix["path_idx"][s] >= 0
            want[ix["path_idx"][s][ok], q] = ix["path_w"][s][ok]
        bad = np.argwhere(gs[:, :nq] != want)
        assert len(bad) == 0, f"{len(bad)} wrong gs elements; first [node, query] {bad[0].tolist()} at position {chosen[bad[0][1]]}"
        assert (gs[:, nq:] == 0).all()


def check_dense(index, ix, x, rng, wrapper=None):
    """Random G: kernel 1 against gs_ref, kernel 2 against the reference of the kernel's own gs (direct call), and the
    whole backward through rank_scores_batch(Q).backward(G) against the reference of gs_ref."""
    nq = x.shape[0]
    G = rng.standard_normal((nq, index.n_pos)).astype(np.float32)
    Q, Gd = torch.from_numpy(x).cuda(), torch.from_numpy(G).cuda()
    gs, dx = bwd_direct(index, Q, Gd)
    gs_ref, ab, terms = node_grad_ref(ix, G)
    e_gs = terms[:, None] * EPS32 * ab
    assert_within(gs[:, :nq], gs_ref, e_gs, "gs")
    want, bound = query_grad_ref(ix, x, gs[:, :nq].astype(np.float64))
    assert_within(dx, want, bound, "grad_q (direct call)")
    if wrapper is not None:
        Qt = Q.clone().requires_grad_(True)
        wrapper.rank_scores_batch(Qt).backward(Gd)
        want, bound = query_grad_ref(ix, x, gs_ref, e_gs)
        assert_within(Qt.grad.cpu().numpy(), want, bound, "grad_q (rank_scores_batch backward)")
    return G


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("nq,weights", [
    pytest.param(1, None, id="nq1-one-warp-31-idle-lanes-default-weights"),
    pytest.param(33, [1.0, 0.5, 2.0], id="nq33-two-warps-one-cta-weights-1-0.5-2"),
    pytest.param(129, LONG_WEIGHTS, id="nq129-two-query-ctas-last-holds-1-query-weights-longer-than-depth"),
    pytest.param(300, None, id="nq300-three-query-ctas-last-partly-idle"),
])
def test_paths_transpose_kernel(nq, weights):
    """Kernel 1 over 3000 positions in 12 chunks: one-hot G at every branch position (bit-exact), then a random G."""
    w, ref, x = corpus_tree(100)
    index, ix = index_pair(w, ref, weights)
    assert transpose_chunk_len(index.n_pos, nq) == 250
    rng = np.random.default_rng(nq)
    q, _ = synth.queries(x, nq, "unit", seed=nq)
    picks, straddle = branch_positions(index, nq)
    assert straddle, "no leaf's sentences cross a chunk boundary"
    check_one_hot(index, ix, torch.from_numpy(q).cuda(), picks, rng)
    check_dense(index, ix, q, rng)


@pytest.mark.parametrize("d,weights", [
    pytest.param(7, None, id="D7-one-d-tile-one-padded-k-tile"),
    pytest.param(100, [1.0, 0.5, 2.0], id="D100-two-d-tiles-last-36-wide-padded-k-tile"),
    pytest.param(130, LONG_WEIGHTS, id="D130-three-d-tiles-last-2-wide"),
])
def test_query_gradient(d, weights):
    """Kernel 2 on 1, 33, 129 and 300 queries (partial 64-query tiles, 1 to 5 query tiles) for D that span one to
    three 64-wide attribute tiles and are not multiples of the 16-attribute k-tile; direct call and autograd."""
    w, ref, x = corpus_tree(d)
    index, ix = index_pair(w, ref, weights)
    for nq in (1, 33, 129, 300):
        q, _ = synth.queries(x, nq, "unit", seed=d + nq)
        check_dense(index, ix, q, np.random.default_rng(d + nq), wrapper=w)


def test_rank_scores_backward_wrapper_paths():
    """_RankScores.backward in 256-query steps (600 queries: 3 steps), a CPU float64 leaf tensor, and a column-strided
    view: each gradient within the bound of the float64 reference (kernel 1 joins chunks with atomicAdd in no fixed
    order, so two runs agree to the bound, not bit for bit)."""
    w, ref, x = corpus_tree(100)
    index, ix = index_pair(w, ref, [1.0, 0.5, 2.0])
    nq = 600
    q, _ = synth.queries(x, nq, "unit", seed=3)
    G = np.random.default_rng(3).standard_normal((nq, index.n_pos)).astype(np.float32)
    Gd = torch.from_numpy(G).cuda()
    gs_ref, ab, terms = node_grad_ref(ix, G)
    e_gs = terms[:, None] * EPS32 * ab
    want, bound = query_grad_ref(ix, q, gs_ref, e_gs)
    # chunked backward: SCORE_BUDGET_BYTES = 1 -> chunk_queries() = 256
    budget, index.SCORE_BUDGET_BYTES = index.SCORE_BUDGET_BYTES, 1
    try:
        assert index.chunk_queries() == 256
        Qt = torch.from_numpy(q).cuda().requires_grad_(True)
        w.rank_scores_batch(Qt).backward(Gd)
        assert_within(Qt.grad.cpu().numpy(), want, bound, "chunked backward")
    finally:
        index.SCORE_BUDGET_BYTES = budget
    Qt = torch.from_numpy(q).cuda().requires_grad_(True)
    w.rank_scores_batch(Qt).backward(Gd)
    assert_within(Qt.grad.cpu().numpy(), want, bound, "unchunked backward")
    # CPU float64 leaf: the gradient comes back through .to(cuda, float32) as float64 on the CPU
    Qc = torch.from_numpy(q.astype(np.float64)).requires_grad_(True)
    w.rank_scores_batch(Qc).backward(Gd)
    assert Qc.grad.dtype == torch.float64 and Qc.grad.device.type == "cpu"
    assert_within(Qc.grad.numpy(), want, bound, "float64 CPU leaf")
    # column-strided view of a [nq, 2D] leaf, and its contiguous copy
    base = torch.zeros((nq, 2 * q.shape[1]), device="cuda")
    base[:, ::2] = torch.from_numpy(q).cuda()
    base.requires_grad_(True)
    view = base[:, ::2]
    assert not view.is_contiguous()
    w.rank_scores_batch(view).backward(Gd)
    g = base.grad.cpu().numpy()
    assert (g[:, 1::2] == 0).all()
    assert_within(g[:, ::2], want, bound, "strided view")
    Qv = view.detach().clone().requires_grad_(True)
    w.rank_scores_batch(Qv).backward(Gd)
    assert_within(Qv.grad.cpu().numpy(), want, bound, "contiguous copy of the view")


@pytest.mark.parametrize("max_len", [
    pytest.param(120, id="len120-4-warps-opt-in-smem"),
    pytest.param(600, id="len600-2-warps-beyond-4-warp-smem"),
    pytest.param(1000, id="len1000-1-warp"),
])
def test_deep_tree(max_len):
    """Paths as deep as the forward path kernel takes (it accepts max_len up to 1024): forward scores against the
    oracle, the path product bit-exact, top-128 (all four register slots of the merge, rank 63 and 127 in lane 31)
    against an exact stable arg-sort, and the backward against the float64 reference.  Kernel 1 needs 536 bytes per
    level with 4 warps per CTA: above 48 KiB from max_len 92, above a B200 CTA's 227 KiB from 434 (2 warps), above
    2 warps' from 855 (1 warp)."""
    w, ref, leaf_vecs = caterpillar(max_len)
    index, ix = index_pair(w, ref, None)
    assert index.max_len == max_len and index.n_pos >= 128
    rng = np.random.default_rng(max_len)
    nq, k = 129, 128
    q = (leaf_vecs[rng.integers(0, len(leaf_vecs), nq)] + 0.05 * rng.standard_normal((nq, leaf_vecs.shape[1]))).astype(np.float32)
    qd = torch.from_numpy(q).cuda()
    ns = index.node_scores(qd).cpu().numpy()
    rns, rls = ref.dense_scores(q)
    floor = 8 * EPS32 * float(np.abs(ix["sumlog"]).max())
    np.testing.assert_allclose(ns, rns, rtol=1e-5, atol=floor)
    ids, vals, leaf = index.predict(qd, k, want_leaf_scores=True)
    ids, vals, leaf = ids.cpu().numpy(), vals.cpu().numpy(), leaf.cpu().numpy()
    np.testing.assert_allclose(leaf, rls, rtol=1e-5, atol=floor)
    assert np.array_equal(leaf, oracle_leaf_scores(ns, ix["path_idx"], ix["path_w"]))
    want = np.argsort(-leaf, axis=1, kind="stable")[:, :k]
    assert np.array_equal(ids, want)
    assert np.array_equal(vals, np.take_along_axis(leaf, want, 1))
    a, b, _ = index.predict(qd, k, small=False)   # the kernel instance without leaf scores
    assert np.array_equal(a.cpu().numpy(), ids) and np.array_equal(b.cpu().numpy(), vals)
    a, b = index.predict_small(qd[:8].contiguous(), k)
    assert np.array_equal(a.cpu().numpy(), ids[:8]) and np.array_equal(b.cpu().numpy(), vals[:8])
    picks, _ = branch_positions(index, nq)
    check_one_hot(index, ix, qd, picks, rng)
    check_dense(index, ix, q, rng, wrapper=w)


def test_backward_rejects_paths_one_warp_cannot_hold():
    """max_len 1700 needs 140 bytes per level with one warp per CTA, more than a B200 CTA has: an argument error that
    names max_len, not a CUDA error.  (The forward path kernel rejects such a tree too: max_len above 1024.)"""
    w, _, leaf_vecs = caterpillar(1700, d=4)
    w.build_prediction_index()
    index = w._index
    Q = torch.from_numpy(leaf_vecs[:3]).cuda()
    G = torch.zeros((3, index.n_pos), device="cuda")
    gs = torch.zeros((index.nn, 3), device="cuda")
    out = torch.zeros_like(Q)
    L = _lib.load()
    rc = L.cw_rank_scores_bwd(C.byref(index.ix), Q.data_ptr(), 3, G.data_ptr(), gs.data_ptr(), 3, out.data_ptr(), _lib.stream_ptr())
    assert rc == _lib.CW_E_ARG and "max_len=1700" in L.cw_last_error().decode()
    with pytest.raises(_lib.CobwebB200Error, match="max_len"):
        w.rank_scores_batch(Q)
