"""Tag-filtered dense retrieval: CobwebWrapper.set_sentence_tags and predict_fast_batch(Q, k, query_tags=...), backed by
cw_dense_paths_topk_tagged, cw_small_predict_tagged and cw_fused_predict_tagged.

Sentence s is eligible for query q iff tags[s] & query_tags[q] != 0.  The reference is rank_scores_batch(Q) (the FP32
form) restricted to the eligible sentences, ranked by (score desc, id asc) in numpy and padded with -1 / -inf; every path
must give the same bits.
"""
import functools

import numpy as np
import pytest
import torch

from rag_cobweb_b200 import CobwebWrapper, DenseIndex, _lib, synth

pytestmark = pytest.mark.gpu
ALL = -1  # every bit set (0xffffffff as an int32 word)


# ------------------------------------------------------------------ trees
@functools.lru_cache(maxsize=None)
def tree(n, d, kind, dups=1):
    x = synth.corpus(n, d, kind, seed=n + d)
    if dups > 1:  # every vector dups times: leaves that hold several sentences
        x = np.ascontiguousarray(np.repeat(x, dups, axis=0))
    return CobwebWrapper(corpus=[None] * len(x), corpus_embeddings=x), x


def fresh(n, d, kind, mode, dups=1):
    """The cached tree with its tags cleared, in the given dense mode."""
    w, x = tree(n, d, kind, dups)
    w.set_sentence_tags(np.arange(len(w)), 0)
    w.set_dense_mode(mode)
    w.build_prediction_index()
    return w, x


def big(kind):
    w, x = fresh(16000, 48, kind, "fused")
    assert w._index.nn >= DenseIndex.TENSOR_MIN_NODES and w._index.mode == "fused"
    return w, x


def queries(x, nq, seed):
    q, _ = synth.queries(x, nq, "unit", seed=seed)
    return torch.from_numpy(q).cuda()


def random_tags(w, bits, seed):
    """Each sentence gets one of `bits` tag bits."""
    rng = np.random.default_rng(seed)
    t = (1 << rng.integers(0, bits, len(w))).astype(np.int64)
    w.set_sentence_tags(np.arange(len(w)), t)
    return t


def random_masks(nq, bits, seed):
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.integers(1, 1 << bits, nq).astype(np.int32)).cuda()


# ------------------------------------------------------------------ reference and checks
def reference(w, Q, qt, k):
    leaf = w.rank_scores_batch(Q).cpu().numpy()
    tags = w.get_sentence_tags().cpu().numpy()
    qt = np.broadcast_to(np.asarray(qt.cpu() if torch.is_tensor(qt) else qt, np.int64).astype(np.int32), (Q.shape[0],))
    k = min(k, leaf.shape[1])
    ids = np.full((Q.shape[0], k), -1, np.int32)
    vals = np.full((Q.shape[0], k), -np.inf, np.float32)
    for q in range(Q.shape[0]):
        e = np.nonzero(tags & qt[q])[0]
        o = e[np.lexsort((e, -leaf[q, e]))][:k]
        ids[q, : len(o)], vals[q, : len(o)] = o, leaf[q, o]
    return torch.from_numpy(ids).cuda(), torch.from_numpy(vals).cuda()


def check(w, Q, qt, k):
    got_i, got_v = w.predict_fast_batch(Q, k, query_tags=qt)
    want_i, want_v = reference(w, Q, qt, k)
    assert got_i.dtype == torch.int32 and got_i.shape == want_i.shape
    bad = (got_i != want_i).any(1) | (got_v != want_v).any(1)
    assert not bool(bad.any()), f"{int(bad.sum())} rows differ, first {int(torch.nonzero(bad)[0])}"
    return got_i, got_v


# ------------------------------------------------------------------ the three device paths and k > CW_MAX_K
@pytest.mark.parametrize("k", [1, 10, 31, 128])
def test_fp32_mode_mixed_masks(k):
    w, x = fresh(2000, 64, "unit", "fp32")
    random_tags(w, 8, seed=k)
    check(w, queries(x, 100, seed=k), random_masks(100, 8, seed=k + 1), k)


@pytest.mark.parametrize("kind", ["unit", "whitened"])
@pytest.mark.parametrize("k", [1, 10, 30])
def test_fused_mode_mixed_masks(kind, k):
    w, x = big(kind)
    w._index.audit_every = 16
    w._index._audit_phase = 0  # the audit runs in one call out of CW_FUSED_AUDIT_STRIDE: make it this one
    random_tags(w, 8, seed=k)
    s0 = dict(w._index.stats)
    check(w, queries(x, 300, seed=k), random_masks(300, 8, seed=k + 2), k)
    st = w._index.stats
    assert st["queries"] - s0["queries"] >= 300 and st["audited"] > s0["audited"] and st["audit_mismatch"] == 0


@pytest.mark.parametrize("nq", [1, 7, 32])
@pytest.mark.parametrize("mode", ["fp32", "fused"])
def test_small_path(nq, mode):
    w, x = big("unit") if mode == "fused" else fresh(2000, 64, "unit", "fp32")
    random_tags(w, 4, seed=nq)
    check(w, queries(x, nq, seed=nq), random_masks(nq, 4, seed=nq), 10)


def test_k_past_max_k():
    w, x = fresh(2000, 64, "unit", "fp32")
    random_tags(w, 4, seed=200)
    check(w, queries(x, 40, seed=200), random_masks(40, 4, seed=200), 200)


# ------------------------------------------------------------------ masks
@pytest.mark.parametrize("mode", ["fp32", "fused"])
def test_all_ones_equals_untagged(mode):
    w, x = big("unit") if mode == "fused" else fresh(2000, 64, "unit", "fp32")
    w.set_sentence_tags(np.arange(len(w)), ALL)
    for nq in (5, 300):
        Q = queries(x, nq, seed=nq)
        i0, v0 = w.predict_fast_batch(Q, 10)
        i1, v1 = w.predict_fast_batch(Q, 10, query_tags=ALL)
        assert torch.equal(i0, i1) and torch.equal(v0, v1)
        i2, _ = w.predict_fast_batch(Q, 10, query_tags=torch.full((nq,), 1 << 31, dtype=torch.int64))  # bit 31 alone
        assert torch.equal(i0, i2)


@pytest.mark.parametrize("mode", ["fp32", "fused"])
def test_mask_zero_gives_padding(mode):
    w, x = big("unit") if mode == "fused" else fresh(2000, 64, "unit", "fp32")
    w.set_sentence_tags(np.arange(len(w)), ALL)
    for nq in (3, 300):
        i, v = w.predict_fast_batch(queries(x, nq, seed=3), 10, query_tags=0)
        assert bool((i == -1).all()) and bool((v == float("-inf")).all())


@pytest.mark.parametrize("mode", ["fp32", "fused"])
def test_selective_tag(mode):
    w, x = big("unit") if mode == "fused" else fresh(2000, 64, "unit", "fp32")
    rng = np.random.default_rng(5)
    chosen = rng.choice(len(w), max(2, len(w) // 1000), replace=False)
    w.set_sentence_tags(chosen, 1 << 7)
    Q = queries(x, 300, seed=5)
    mixed = torch.where(torch.arange(300, device="cuda") % 2 == 0, 1 << 7, ALL).to(torch.int32)
    check(w, Q, mixed, 10)
    i, _ = check(w, Q, 1 << 7, 30 if mode == "fused" else 40)
    assert bool((i[:, len(chosen):] == -1).all())


@pytest.mark.parametrize("mode", ["fp32", "fused"])
def test_fewer_than_k_eligible(mode):
    w, x = big("unit") if mode == "fused" else fresh(2000, 64, "unit", "fp32")
    w.set_sentence_tags([3, 900, 1500, 1501, 7], 1 << 3)
    for nq in (4, 300):
        i, _ = check(w, queries(x, nq, seed=8), 1 << 3, 10)
        assert bool((i[:, 5:] == -1).all()) and bool((i[:, :5] >= 0).all())


@pytest.mark.parametrize("k", [1, 10, 30])
def test_duplicate_sentences_with_mixed_tags(k):
    """Four sentences per leaf, one of them eligible: a leaf counts its eligible sentences only."""
    w, x = fresh(4000, 32, "unit", "fused", dups=4)
    w._index.TENSOR_MIN_NODES = 0  # a 4000-leaf tree: run it on the fused pipeline all the same
    w._index.audit_every = 8
    sid = np.arange(len(w))
    w.set_sentence_tags(sid, np.where(sid % 4 == 1, 1, 2))
    Q = queries(x, 300, seed=k)
    check(w, Q, 1, k)
    check(w, Q, torch.where(torch.arange(300, device="cuda") % 3 == 0, 1, 3).to(torch.int32), k)
    check(w, Q[:9], 1, k)
    assert w._index.stats["audit_mismatch"] == 0


def test_eligibility_outside_the_sampled_tiles_flags_and_stays_exact():
    w, x = big("whitened")
    ix = w._index
    hx = ix.hx
    n_s = hx["n_s"] * _lib.H_TILE
    assert n_s > 0
    off, sids = hx["sent_off"].cpu().numpy(), hx["sent_ids"].cpu().numpy()
    outside = sids[off[n_s]:]
    w.set_sentence_tags(outside, 1)
    flagged = ix.stats["flagged"]
    check(w, queries(x, 300, seed=9), 1, 10)
    assert ix.stats["flagged"] > flagged and ix.stats["audit_mismatch"] == 0


# ------------------------------------------------------------------ derived tags, lifecycle, arguments
def test_leaf_tags_are_the_or_over_each_leaf():
    w, x = fresh(4000, 32, "unit", "fused", dups=4)
    random_tags(w, 16, seed=1)
    ix = w._index
    t = ix.tag_arrays(w._tag_words(), w._tag_version)
    tags = w.get_sentence_tags().cpu().numpy()
    off, sids = ix.hx["sent_off"].cpu().numpy(), ix.hx["sent_ids"].cpu().numpy()
    want = np.array([np.bitwise_or.reduce(tags[sids[off[r]:off[r + 1]]]) for r in range(len(off) - 1)], np.int32)
    assert np.array_equal(t["leaf"].cpu().numpy(), want)
    assert np.array_equal(t["pos"].cpu().numpy(), tags[ix.pos_rec[:, 3].cpu().numpy()])


def test_lifecycle_retag_add_and_snapshot(tmp_path):
    x = synth.corpus(600, 32, "unit", seed=4)
    w = CobwebWrapper(corpus=[None] * 500, corpus_embeddings=x[:500])
    w.save_snapshot(str(tmp_path / "plain.snap"))
    assert bool((CobwebWrapper.load_snapshot(str(tmp_path / "plain.snap")).get_sentence_tags() == 0).all())
    Q = queries(x, 40, seed=4)
    w.set_sentence_tags(np.arange(0, 500, 2), 1)
    check(w, Q, 1, 10)
    w.set_sentence_tags(np.arange(0, 500, 2), 2)  # the next call sees the new tags
    i, _ = w.predict_fast_batch(Q, 10, query_tags=1)
    assert bool((i == -1).all())
    check(w, Q, 2, 10)
    w.add_sentences([None] * 100, x[500:])
    t = w.get_sentence_tags()
    assert t.shape == (600,) and bool((t[500:] == 0).all())
    check(w, Q, ALL, 10)
    w.set_sentence_tags([550, 551], [4, 0xFFFFFFFF])
    w.save_snapshot(str(tmp_path / "tagged.snap"))
    w2 = CobwebWrapper.load_snapshot(str(tmp_path / "tagged.snap"))
    assert torch.equal(w2.get_sentence_tags(), w.get_sentence_tags())
    for m in (4, 2, ALL):
        assert all(torch.equal(a, b) for a, b in zip(w2.predict_fast_batch(Q, 10, query_tags=m),
                                                     w.predict_fast_batch(Q, 10, query_tags=m)))


def test_argument_errors():
    w, x = fresh(2000, 64, "unit", "fp32")
    n = len(w)
    for ids, tags in (([n], 1), ([-1], 1), ([1, 1], 1), ([1.0], 1), ([1, 2], [1]), ([1], 1 << 32), ([1], -(1 << 31) - 1),
                      ([1], 0.5), ([[1]], 1)):
        with pytest.raises(ValueError):
            w.set_sentence_tags(ids, tags)
    Q = queries(x, 5, seed=1)
    for qt in ([1, 2], 1.5, torch.ones(5, dtype=torch.bool), 1 << 32):
        with pytest.raises(ValueError):
            w.predict_fast_batch(Q, 10, query_tags=qt)
    shard = DenseIndex(w.tree, w._leaf_of_sentence, sentence_ids=np.arange(0, n, 2))
    with pytest.raises(ValueError):
        shard.predict(Q, 10, query_tags=torch.ones(5, dtype=torch.int32, device="cuda"), sent_tags=w._tag_words(),
                      tag_version=0)
    assert w.predict_fast_batch(Q, 0, query_tags=1)[0].shape == (5, 0)
