"""The FP32 form of dense predict (the form that defines every retrieval answer, DESIGN.md section 5) bit for bit against a
CPU model of its arithmetic, on every launch shape of its kernels.

The model (OracleTree.fp32_scores / fp32_operands, oracle/cobweb_oracle.c) restates the specified operation sequence:
r = 1 / sqrt(var), mb = -(mean * r); per (query, node) one chain over d ascending, u = fma(x, r, mb), acc = fma(u, u, acc)
from acc = +0; s = -0.5 * (sumlog + acc); each leaf an fp32 FMA chain root first with weights (float)(level_w[j] / len);
results ordered by (score desc, sentence id asc), padded with -1 / -inf only when a row has fewer than k sentences.

The CPU tests check the model itself: libm fmaf against exact rational arithmetic, and the model against float64 within
a bound derived from the operation sequence.  The GPU tests compare the engine's outputs with the model as int32 views
(so -0 and +0 differ): node scores (index_tiles_kernel, tile_queries_kernel, dense_score_kernel), the R / MB tiles and
the row-major rows (index_rows_kernel), the leaf matrix and top-k (paths_topk_kernel, merge_topk_kernel), the small-batch
path (small_scores_kernel<QB>, paths_small_kernel) and the host entry points.  Every case asserts, through Python mirrors
of the launch formulas, that it reaches the branch it is named after.
"""
import functools
from fractions import Fraction

import numpy as np
import pytest
import torch

from oracle.cobweb_oracle import OracleTree, fmaf, topk
from rag_cobweb_b200 import CobwebB200Error, CobwebTorchTree, CobwebWrapper, _lib, synth

EPS = 2.0 ** -24          # unit roundoff of binary32
TK, TN, STAGES, SM_DC, PT_MAXLEN = 16, 128, 4, 256, 1024   # cw_dense.cu


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def assert_bits(got, want, what=""):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.nonzero(bits(got) != bits(want))
    assert not len(bad[0]), f"{what}: {len(bad[0])} values differ, first at {tuple(int(b[0]) for b in bad)}: " \
                            f"{got[tuple(b[0] for b in bad)]!r} vs {want[tuple(b[0] for b in bad)]!r}"


# ------------------------------------------------------------------ exact arithmetic (CPU)
def round_f32(x):
    """Fraction -> nearest binary32 (ties to even), overflow to +-inf; exact zero -> +0."""
    if x == 0:
        return np.float32(0.0)
    neg, a = x < 0, abs(x)
    e = a.numerator.bit_length() - a.denominator.bit_length()
    if Fraction(2) ** e > a:
        e -= 1
    qe = max(e, -126) - 23                       # exponent of the quantum at a (subnormals: 2^-149)
    s = a / Fraction(2) ** qe
    n, rem = divmod(s.numerator, s.denominator)
    if 2 * rem > s.denominator or (2 * rem == s.denominator and n & 1):
        n += 1
    v = n * Fraction(2) ** qe
    r = np.float32(np.inf) if v >= Fraction(2) ** 128 else np.float32(float(v))
    return -r if neg else r


def exact_fma(a, b, c):
    a, b, c = np.float32(a), np.float32(b), np.float32(c)
    p = Fraction(float(a)) * Fraction(float(b))
    s = p + Fraction(float(c))
    if s == 0 and p == 0 and c == 0:   # exact zero of zeros: -0 only if both addends are -0
        neg = (np.signbit(a) != np.signbit(b)) and np.signbit(c)
        return np.float32(-0.0) if neg else np.float32(0.0)
    return round_f32(s)


def fma_triples(rng, n):
    """Random triples of mixed magnitude plus the edges of the model's chain."""
    def rnd(m, lo, hi):
        return (rng.choice([-1.0, 1.0], m) * rng.uniform(1.0, 2.0, m) * 2.0 ** rng.integers(lo, hi, m)).astype(np.float32)
    a, b, c = rnd(n, -30, 30), rnd(n, -30, 30), rnd(n, -60, 60)
    m, r = rnd(n, -20, 20), rnd(n, -20, 20)
    err = (m, r, -(m * r))                                         # fma(m, r, -fl(m r)): the rounding error of m r
    ulp = np.spacing(np.abs(m * r)).astype(np.float32)
    cancel = (m, r, (-(m * r) + rng.integers(-3, 4, n) * ulp).astype(np.float32))   # sums a few ulps from zero
    tiny = (rnd(n, -80, -60), rnd(n, -80, -60), rnd(n, -149, -126))   # subnormal and underflowing results
    u = rnd(n, -75, -63)
    square = (u, u, np.zeros(n, np.float32))                       # acc = fma(u, u, +0) below the normal range
    big = (rnd(n, 62, 66), rnd(n, 62, 66), rnd(n, 100, 127))        # overflow to inf
    zeros = (np.array([0.0, -0.0, 0.0, -0.0, 1.0, -1.0], np.float32), np.array([1.0, 1.0, -1.0, -1.0, 0.0, 0.0], np.float32),
             np.array([-0.0, -0.0, -0.0, -0.0, -0.0, 0.0], np.float32))
    parts = [(a, b, c), err, cancel, tiny, square, big, zeros]
    return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))


def test_fmaf_is_correctly_rounded():
    """The model's fused multiply-add (libm fmaf through the oracle library) equals exact rational arithmetic rounded
    once to binary32, ties to even, on random triples and on the chain's edges: the rounding error of a product, sums
    that cancel to a few ulps, subnormal results, squares that underflow, overflow and signed zeros."""
    rng = np.random.default_rng(0)
    a, b, c = fma_triples(rng, 600)
    assert len(a) > 3000
    got = fmaf(a, b, c)
    want = np.array([exact_fma(x, y, z) for x, y, z in zip(a, b, c)], np.float32)
    assert_bits(got, want, "fmaf")
    # the edges are live: results that are subnormal, exactly zero, the rounding error of a product, and infinite
    assert (np.abs(want) < np.finfo(np.float32).tiny).sum() > 100 and np.isinf(want).sum() > 100
    assert np.count_nonzero(want[600:1200]) > 500   # fma(m, r, -fl(m r)) is the product's rounding error, rarely 0


# ------------------------------------------------------------------ trees from arrays
def agg_root(count, mean, m2):
    """count / mean / m2 of a parent from its children's (the merge the store keeps)."""
    n = count.sum()
    mu = (count[:, None] * mean).sum(0) / n
    return n, mu, (m2 + count[:, None] * (mean - mu) ** 2).sum(0)


REGIMES = {  # name -> (prior_var, mean offset, leaf spread, query noise, acuity cutoff)
    "normal": (None, 0.0, 1.0, 0.3, False),
    "offset": (1e-6, 1e3, 1e-2, 1e-3, False),     # |mean| >> sigma: mb = -(mean r) carries the error term |mean r| 2^-24
    "prior_small": (1e-6, 0.0, 1.0, 1e-3, False),
    "prior_large": (1e3, 0.0, 30.0, 10.0, False),
    "acuity": (None, 0.0, 1.0, 0.3, True),         # var = max(m2 / count, prior): some attributes at the prior
}


def flat_arrays(d, n_leaves, regime, seed):
    """root -> n_leaves leaves (one to three sentences each; leaves with several sentences have a spread), or with
    n_leaves = 0 a root that holds three sentences itself.  Arrays in BFS order; returns dict(parent, count, nsent, mean,
    m2, leaf_of_sentence, prior_var, acuity_cutoff, qscale)."""
    prior, off, spread, qscale, cutoff = REGIMES[regime]
    rng = np.random.default_rng(seed)
    if n_leaves == 0:
        mean = (off + spread * rng.standard_normal((1, d))).astype(np.float32)
        m2 = (3 * spread ** 2 * rng.uniform(0.05, 1.0, (1, d))).astype(np.float32)
        return dict(parent=np.array([-1]), count=np.array([3.0], np.float32), nsent=np.array([3], np.int32), mean=mean, m2=m2,
                    leaf_of_sentence=np.zeros(3, np.int32), prior_var=prior, acuity_cutoff=cutoff, qscale=qscale)
    c = (1 + (np.arange(n_leaves) % 3 == 1) + (np.arange(n_leaves) % 5 == 2)).astype(np.float64)
    mean = off + spread * rng.standard_normal((n_leaves, d))
    m2 = (c - 1)[:, None] * (0.3 * spread) ** 2 * rng.uniform(0.0, 2.0, (n_leaves, d))
    n, mu, rm2 = agg_root(c, mean, m2)
    leaves = np.arange(1, n_leaves + 1)
    return dict(parent=np.concatenate([[-1], np.zeros(n_leaves, np.int64)]), count=np.concatenate([[n], c]).astype(np.float32),
                nsent=np.concatenate([[0], c]).astype(np.int32), mean=np.vstack([mu, mean]).astype(np.float32),
                m2=np.vstack([rm2, m2]).astype(np.float32),
                leaf_of_sentence=rng.permutation(np.repeat(leaves, c.astype(np.int64))).astype(np.int32),
                prior_var=prior, acuity_cutoff=cutoff, qscale=qscale)


def queries_near(mean, nq, qscale, seed):
    """A third of the queries equal to a row of mean, a third 1e-3 qscale away, a third qscale away."""
    rng = np.random.default_rng(seed)
    base = mean[rng.integers(0, len(mean), nq)].astype(np.float64)
    noise = rng.standard_normal(base.shape) * np.where(np.arange(nq) % 3 == 0, 0.0,
                                                       np.where(np.arange(nq) % 3 == 1, 1e-3, 1.0))[:, None]
    return (base + qscale * noise).astype(np.float32)


def oracle_from_arrays(t, level_weights=None):
    ref = OracleTree(t["mean"].shape[1], prior_var=t["prior_var"], acuity_cutoff=t["acuity_cutoff"])
    ref.load(t["parent"], t["count"], t["nsent"], t["mean"], t["m2"])
    ref.leaf_of_sentence = np.asarray(t["leaf_of_sentence"], np.int32)
    ref.n_sentences = len(ref.leaf_of_sentence)
    ix = ref.build_index(level_weights)
    assert np.array_equal(ix["bfs"]["order"], np.arange(len(t["parent"])))   # slot i is index row i
    return ref


# ------------------------------------------------------------------ the model against float64 (CPU)
def f64_bound(ref, Q):
    """float64 node scores -0.5 (sum log v + sum (x - mu)^2 / v) of the store's fp32 mean and var, and the bound on
    |model - float64| that the model's operation sequence implies.

    With eps = 2^-24, u = (x - mu) r the exact term and r = v^-1/2:
      r^ = fl(1 / fl(sqrt v)) = r (1 + d_r), |d_r| <= e_r = 2 eps / (1 - eps)        (two roundings)
      mb^ = -fl(mu r^) = -mu r^ (1 + d3)                                              (one rounding)
      u^ = fl(x r^ + mb^) = ((x - mu) r^ - mu r^ d3)(1 + d4)                          (one rounding)
    so |u^ - u| <= e_u = |u| (e_r + eps (1 + e_r)) + |mu| r (1 + e_r) eps (1 + eps) + 2^-149;
    the |mu r| eps term is the whole error when x = mu.  Then
      |u^2 - u^2| <= e_u (2 |u| + e_u), and the FMA chain over D nonnegative terms adds at most gamma_D sum u^2 with
      gamma_D = D eps / (1 - D eps) and sum u^2 <= sum (|u| + e_u)^2 (plus D 2^-150 for results below the normal range);
      sumlog is within one ulp per logf of sum log v, plus the binary64 sum's error and one binary32 rounding;
      fl(sumlog + acc) adds one rounding, -0.5 * is exact.
    The float64 reference itself is within 4 D 2^-53 of the exact value relative to its absolute terms."""
    ix = ref.index
    mu, v = ix["means"].astype(np.float64), ix["vars"].astype(np.float64)
    D = mu.shape[1]
    Q = Q.astype(np.float64)
    r = 1.0 / np.sqrt(v)                                               # [nn, D]
    u = (Q[:, None, :] - mu[None]) * r[None]                           # [nq, nn, D]
    lv = np.log(v)
    s64 = -0.5 * (lv.sum(1)[None] + (u * u).sum(2))
    e_r = 2 * EPS / (1 - EPS)
    e_u = np.abs(u) * (e_r + EPS * (1 + e_r)) + (np.abs(mu) * r * (1 + e_r) * EPS * (1 + EPS))[None] + 2.0 ** -149
    g_d = D * EPS / (1 - D * EPS)
    e_acc = (e_u * (2 * np.abs(u) + e_u)).sum(2) + g_d * ((np.abs(u) + e_u) ** 2).sum(2) + D * 2.0 ** -150
    sl = ix["sumlog"].astype(np.float64)
    ulp_log = np.spacing(np.abs(lv).astype(np.float32) * np.float32(1 + 2 * EPS)).astype(np.float64)
    e_sl = ulp_log.sum(1) + 4 * D * 2.0 ** -53 * np.abs(lv).sum(1) + EPS * np.abs(sl)
    acc_hi = (u * u).sum(2) + e_acc
    e_add = EPS * (np.abs(sl)[None] + e_sl[None] + acc_hi)
    e_ref = 4 * D * 2.0 ** -53 * (np.abs(lv).sum(1)[None] + (u * u).sum(2))
    return s64, 0.5 * (e_acc + e_sl[None] + e_add) + e_ref


@pytest.mark.parametrize("regime", ["at_means", "offset", "prior_1e-6", "prior_1e3", "acuity"])
def test_model_within_float64_bound(regime):
    """The model's node scores are within the derived bound of float64 on adversarial data: queries equal to node means
    (the error is then all rounding of mb), |mean| >> sigma, prior_var from 1e-6 to 1e3, acuity cutoff; the leaf chain is
    within gamma_len sum |w_j s_j| plus the weights' rounding of the float64 path sum of the model's node scores."""
    name = {"at_means": "normal", "prior_1e-6": "prior_small", "prior_1e3": "prior_large"}.get(regime, regime)
    t = flat_arrays(96, 40, name, seed=3)
    ref = oracle_from_arrays(t, level_weights=[1.0, 0.5, 2.0, 1.5])
    Q = queries_near(t["mean"], 60, t["qscale"], seed=4)
    if regime == "at_means":
        Q = t["mean"][np.arange(60) % len(t["mean"])].copy()
    if regime == "acuity":   # the cutoff is live: some variances sit at the prior, others above it
        pv = np.float32(ref.prior_var)
        assert (ref.index["vars"] == pv).mean() > 0.1 and (ref.index["vars"] > pv).mean() > 0.1
    node, leaf = ref.fp32_scores(Q)
    s64, bound = f64_bound(ref, Q)
    err = np.abs(node.astype(np.float64) - s64)
    assert np.all(err <= bound), f"worst error / bound {float((err / bound).max()):.3g}"
    # leaf chain: fp32 FMA over len terms, weights (float)(lw[j] / len)
    ix = ref.index
    pidx, pw = ix["path_idx"], ix["path_w"].astype(np.float64)
    lw = [1.0, 0.5, 2.0, 1.5]
    lens = (pidx >= 0).sum(1)
    w64 = np.array([[(lw[j] if j < len(lw) else 1.0) / n if j < n else 0.0 for j in range(pidx.shape[1])] for n in lens])
    s = node.astype(np.float64)[:, np.maximum(pidx, 0)] * (pidx >= 0)          # [nq, L, max_len]
    l64 = (s * w64[None]).sum(2)
    lbound = (lens * EPS / (1 - lens * EPS))[None] * np.abs(s * pw[None]).sum(2) + (np.abs(pw - w64)[None] * np.abs(s)).sum(2)
    assert np.all(np.abs(leaf - l64) <= lbound + 2.0 ** -149 * lens[None])


# ------------------------------------------------------------------ engine side (GPU)
def engine_from_arrays(t, level_weights=None):
    mean32 = np.asarray(t["mean"], np.float32)
    w = CobwebWrapper(corpus=[None], corpus_embeddings=np.zeros((1, 8), np.float32))   # the tree is replaced below
    w.tree = CobwebTorchTree((mean32.shape[1],), prior_var=t["prior_var"], acuity_cutoff=t["acuity_cutoff"])
    w.tree.load_arrays(t["parent"], t["count"], t["nsent"], mean32, t["m2"])
    w.sentences, w._leaf_of_sentence = [None] * len(t["leaf_of_sentence"]), np.asarray(t["leaf_of_sentence"], np.int32)
    if level_weights is not None:
        w.set_level_weights(list(level_weights))
    w._invalidate_prediction_index()
    w.build_prediction_index()
    return w


def oracle_of(w):
    """The oracle holding the engine's tree (rows in the index's BFS order) and the same sentence paths."""
    b = w.tree.bfs()
    mean, m2 = w.tree.store.rows(b["order"])
    pos = np.full(int(b["order"].max()) + 1, -1, np.int64)
    pos[b["order"]] = np.arange(len(b["order"]))
    t = dict(parent=b["parent"], count=b["count"], nsent=b["nsent"], mean=mean, m2=m2,
             leaf_of_sentence=pos[np.asarray(w._leaf_of_sentence)], prior_var=float(w.tree.prior_var.item()),
             acuity_cutoff=w.tree.acuity_cutoff)
    return oracle_from_arrays(t, w._level_weights)


def model_topk(leaf, k):
    out = [topk(row, k) for row in leaf]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])


def check_operands(ix, ref):
    """R / MB tiles [node tile][k tile][16][128] decoded to [row, d]: the model's r and mb, padding exactly +0; the
    row-major rows {r, mb}; sumlog."""
    r, mb = ref.fp32_operands()
    nn, D = r.shape
    for name, t, want in (("R", ix.R, r), ("MB", ix.MB, mb)):
        got = t.view(ix.n_ntiles, ix.n_ktiles, TK, TN).permute(0, 3, 1, 2).reshape(ix.n_ntiles * TN, ix.n_ktiles * TK)
        got = got.cpu().numpy()
        assert_bits(got[:nn, :D], want, name)
        pad = bits(got).copy()
        pad[:nn, :D] = 0
        assert not pad.any(), f"{name}: padding is not +0"
    rows = ix.rows().cpu().numpy()
    assert_bits(rows[..., 0], r, "rows r")
    assert_bits(rows[..., 1], mb, "rows mb")
    assert_bits(ix.sumlog[:nn].cpu().numpy(), ref.index["sumlog"], "sumlog")


def check_fp32_form(w, ref, Q, ks, host=True):
    """Node scores, the leaf matrix (LEAF variant), top-k of the FP32 path without leaf scores, and the host entry
    point, each against the model bit for bit.  Returns the model's (node, leaf)."""
    ix = w._index
    Qd = torch.from_numpy(Q).cuda()
    node, leaf = ref.fp32_scores(Q)
    assert_bits(ix.node_scores(Qd).cpu().numpy(), node, "node scores")
    for k in ks:
        want_i, want_v = model_topk(leaf, k)
        ids, vals, lg = ix.predict(Qd, k, want_leaf_scores=True, mode="fp32")
        assert_bits(lg.cpu().numpy(), leaf, "leaf scores")
        assert np.array_equal(ids.cpu().numpy(), want_i), f"top-{k} ids (LEAF variant)"
        assert_bits(vals.cpu().numpy(), want_v, f"top-{k} scores (LEAF variant)")
        ids, vals, _ = ix.predict(Qd, k, mode="fp32", small=False)
        assert np.array_equal(ids.cpu().numpy(), want_i), f"top-{k} ids"
        assert_bits(vals.cpu().numpy(), want_v, f"top-{k} scores")
        if host:
            hs, hv = ix.predict_host(Q, k)
            assert np.array_equal(hs.numpy(), want_i), f"host top-{k} ids"
            assert_bits(hv.numpy(), want_v, f"host top-{k} scores")
    return node, leaf


# launch mirrors (cw_dense.cu)
def n_ktiles(d):
    return (d + TK - 1) // TK


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def paths_launch(k, max_len, n_pos, nq):
    """(wpb, n_chunks, chunk_len) of paths_topk_launch."""
    per_warp = k * 256 + max_len * 132 + 64 * 32 + 8 * 3 * 32 * 4
    fixed = ((max_len + 1) & ~1) * 8
    wpb, best = 1, 0
    for c in range(8, 0, -1):
        blk = fixed + c * per_warp
        if blk > 200 * 1024:
            continue
        warps = (227 * 1024) // (blk + 1024) * c
        if warps > best:
            best, wpb = warps, c
    gblocks = ((nq + 31) // 32 + wpb - 1) // wpb
    want = max(1, min(sms() * (best // wpb) // gblocks, (n_pos + 1023) // 1024))
    chunk_len = (n_pos + want - 1) // want
    return wpb, (n_pos + chunk_len - 1) // chunk_len, chunk_len


def small_launch(nq, n_pos):
    """(QB, n_chunks, chunk_len) of cw_small_predict."""
    qb = next(b for b in (1, 2, 4, 8, 16, 32) if nq <= b)
    per_q = min(32 * ((n_pos + 1023) // 1024) // nq, 1024)
    chunk_len = max((n_pos + per_q - 1) // per_q, 256)
    chunk_len = (chunk_len + 31) & ~31
    return qb, (n_pos + chunk_len - 1) // chunk_len, chunk_len


DENSE_SHAPES = [  # D, nn, nq, regime: n_ktiles 1, 3, 4, 5, 8, 9, 128, 256 (fewer, as many and more k-tiles than the
    (1, 129, 129, "normal"),          # 4 stages); nn 1, 127, 128, 129, 257; nq 1, 127, 128, 129
    (33, 127, 128, "offset"),
    (64, 128, 127, "prior_small"),
    (65, 257, 1, "prior_large"),
    (128, 1, 129, "normal"),
    (144, 129, 128, "acuity"),
    (2048, 257, 129, "normal"),
    (4096, 129, 127, "offset"),
]


@functools.lru_cache(maxsize=None)
def flat_case(d, nn, regime, seed=0, level_weights=None):
    t = flat_arrays(d, nn - 1, regime, seed)
    w = engine_from_arrays(t, level_weights)
    return w, oracle_of(w), t


@pytest.mark.gpu
@pytest.mark.parametrize("d,nn,nq,regime", [pytest.param(*s, id=f"D{s[0]}-nn{s[1]}-nq{s[2]}-{s[3]}") for s in DENSE_SHAPES])
def test_dense_shapes(d, nn, nq, regime):
    w, ref, t = flat_case(d, nn, regime)
    ix = w._index
    assert ix.nn == nn and ix.n_ktiles == n_ktiles(d) and ix.n_ntiles == (nn + TN - 1) // TN
    check_operands(ix, ref)
    Q = queries_near(t["mean"], nq, t["qscale"], seed=nq)
    check_fp32_form(w, ref, Q, ks=(1, 10))
    if nq == 1:
        node, leaf = ref.fp32_scores(Q)
        assert ix.predict_one(Q[0], 10) == list(model_topk(leaf, 10)[0][0])


def test_shape_coverage():
    """The shapes above cover what their names say: k-tiles fewer than, equal to and beyond the pipeline's stages,
    D % 16 != 0, partial node and query tiles."""
    kt = {n_ktiles(d) for d, _, _, _ in DENSE_SHAPES}
    assert {1, 3, 4, 5, 8, 9} <= kt and max(kt) >= 128 and min(kt) < STAGES
    assert any(d % TK for d, _, _, _ in DENSE_SHAPES)
    assert {1, 127, 128, 129, 257} <= {nn for _, nn, _, _ in DENSE_SHAPES}
    assert {1, 127, 128, 129} <= {nq for _, _, nq, _ in DENSE_SHAPES}


@pytest.mark.gpu
def test_chunked_call():
    """SCORE_BUDGET_BYTES = 1: 256-query chunks and a remainder of 11 queries, scored into a matrix with ldq = 256 >
    cw_score_ldq(11) = 128."""
    w, ref, t = flat_case(48, 200, "normal", seed=1)
    ix = w._index
    Q = queries_near(t["mean"], 2 * 256 + 11, t["qscale"], seed=5)
    budget, ix.SCORE_BUDGET_BYTES, ws = ix.SCORE_BUDGET_BYTES, 1, ix._ws
    try:
        ix._ws = None
        assert ix.chunk_queries() == 256
        chunks = list(ix._fp32_chunks(len(Q), 10))
        assert len(chunks) == 3 and chunks[-1][0] == slice(512, 523)
        assert chunks[-1][1]["ldq"] == 256 > _lib.load().cw_score_ldq(11)
        Qd = torch.from_numpy(Q).cuda()
        _, leaf = ref.fp32_scores(Q)
        for k in (10, 40):
            want_i, want_v = model_topk(leaf, k)
            ids, vals, lg = ix.predict(Qd, k, want_leaf_scores=True, mode="fp32")
            assert_bits(lg.cpu().numpy(), leaf, "leaf scores")
            assert np.array_equal(ids.cpu().numpy(), want_i) and np.array_equal(bits(vals.cpu().numpy()), bits(want_v))
            ids, vals, _ = ix.predict(Qd, k, mode="fp32")
            assert np.array_equal(ids.cpu().numpy(), want_i) and np.array_equal(bits(vals.cpu().numpy()), bits(want_v))
            hs, hv = ix.predict_host(Q, k)
            assert np.array_equal(hs.numpy(), want_i) and np.array_equal(bits(hv.numpy()), bits(want_v))
    finally:
        ix.SCORE_BUDGET_BYTES, ix._ws = budget, ws


SMALL_SHAPES = [(1, 257), (2, 1030), (3, 2048), (4, 257), (5, 1030), (8, 2048), (9, 257), (16, 1030), (17, 2048), (32, 257)]


@pytest.mark.gpu
@pytest.mark.parametrize("nq,d", [pytest.param(nq, d, id=f"nq{nq}-D{d}") for nq, d in SMALL_SHAPES])
def test_small_path(nq, d):
    """small_scores_kernel<QB> at every QB boundary, with D > SM_DC = 256 so that the queries are staged in several
    passes; paths_small_kernel and the merge.  k = n_pos returns every leaf score, in order."""
    w, ref, t = flat_case(d, 80, "normal", seed=2)
    ix = w._index
    qb, _, _ = small_launch(nq, ix.n_pos)
    assert qb >= nq > qb // 2 and (n_ktiles(d) + SM_DC // TK - 1) // (SM_DC // TK) >= 2
    assert ix.n_pos <= _lib.MAX_K
    Q = queries_near(t["mean"], nq, t["qscale"], seed=nq + 7)
    Qd = torch.from_numpy(Q).cuda()
    _, leaf = ref.fp32_scores(Q)
    for k in (1, 10, ix.n_pos):
        assert ix._route(nq, k, "fp32") == "small"
        want_i, want_v = model_topk(leaf, k)
        ids, vals, _ = ix.predict(Qd, k)
        assert np.array_equal(ids.cpu().numpy(), want_i), f"top-{k} ids"
        assert_bits(vals.cpu().numpy(), want_v, f"top-{k} scores")
        hs, hv = ix.predict_host(Q, k)
        assert np.array_equal(hs.numpy(), want_i) and np.array_equal(bits(hv.numpy()), bits(want_v))
    if nq == 1:
        assert ix.predict_one(Q[0], 10) == list(model_topk(leaf, 10)[0][0])


# ------------------------------------------------------------------ path product and top-k
def binary_arrays(nn, d, seed, mult):
    """Complete binary tree in BFS numbering (children of i: 2i + 1, 2i + 2): leaves on two depths, so consecutive
    positions share m = len - 1, len - 2, len - 3 and fewer levels, and the path length changes.  Leaf j holds mult[j]
    identical sentences; the leaves 2i + 1, 2i + 2 of every fifth parent are exact duplicates (equal scores)."""
    rng = np.random.default_rng(seed)
    parent = np.concatenate([[-1], (np.arange(1, nn) - 1) // 2])
    leaves = np.array([i for i in range(nn) if 2 * i + 1 >= nn])
    nl = len(leaves)
    c = np.asarray(mult, np.float64)[:nl]
    mean = np.zeros((nn, d))
    m2 = np.zeros((nn, d))
    count = np.zeros(nn)
    lm = rng.standard_normal((nl, d))
    lm2 = (c - 1)[:, None] * 0.01 * rng.uniform(0.0, 2.0, (nl, d))
    for j, i in enumerate(leaves):
        if i % 2 == 0 and (i // 2) % 5 == 0 and j > 0 and leaves[j - 1] == i - 1 and c[j] == c[j - 1]:
            lm[j], lm2[j] = lm[j - 1], lm2[j - 1]
    mean[leaves], m2[leaves], count[leaves] = lm, lm2, c
    for i in range(nn - 1, -1, -1):
        kids = [k for k in (2 * i + 1, 2 * i + 2) if k < nn]
        if kids:
            count[i], mean[i], m2[i] = agg_root(count[kids], mean[kids], m2[kids])
    nsent = np.zeros(nn, np.int32)
    nsent[leaves] = c
    return dict(parent=parent, count=count.astype(np.float32), nsent=nsent, mean=mean.astype(np.float32),
                m2=m2.astype(np.float32), leaf_of_sentence=rng.permutation(np.repeat(leaves, c.astype(np.int64))).astype(np.int32),
                prior_var=None, acuity_cutoff=False, qscale=0.3, leaves=leaves)


BIN_NN, BIN_D, BIN_NQ = 2647, 32, 45


def bin_mult(nn):
    nl = sum(1 for i in range(nn) if 2 * i + 1 >= nn)
    j = np.arange(nl)
    return 1 + (j % 3 == 0) + (j % 7 == 2) + 2 * (j % 11 == 5)


@functools.lru_cache(maxsize=None)
def binary_case(level_weights=None):
    t = binary_arrays(BIN_NN, BIN_D, 11, bin_mult(BIN_NN))
    w = engine_from_arrays(t, level_weights)
    return w, oracle_of(w), t


def pos_records(ix):
    return ix.pos_rec.cpu().numpy().astype(np.int64)   # {len, m, leaf row, sid}


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 31, 32, 33, 64, 128])
def test_paths_topk(k):
    """paths_topk_kernel (K32 for k <= 32, the pass-of-32 insertion above) and merge_topk_kernel on 2195 positions
    in three chunks per query: one chunk boundary inside a run of sentences of one leaf (m == len, equal scores split
    between chunks, ordered by id), one where a leaf follows its sibling (m == len - 1); prefixes m = len - 1 .. len - 3
    and shorter, a change of path length, sentence ids permuted against positions, exact-duplicate sibling leaves; 45
    queries (a partial query group).  Queries at the leaves whose runs straddle the boundaries make the ties count."""
    w, ref, t = binary_case()
    ix = w._index
    rec = pos_records(ix)
    n_pos, max_len = ix.n_pos, ix.max_len
    _, n_chunks, chunk_len = paths_launch(k, max_len, n_pos, BIN_NQ)
    assert n_pos > 1024 and n_chunks >= 2 and BIN_NQ % 32
    bnd = [c * chunk_len for c in range(1, n_chunks)]
    lens, m = rec[:, 0], rec[:, 1]
    assert any(m[p] == lens[p] for p in bnd), "no chunk boundary inside a run of one leaf's sentences"
    assert any(m[p] == lens[p] - 1 for p in bnd), "no chunk boundary between sibling leaves"
    gap = lens[1:] - m[1:]
    same_len = lens[1:] == lens[:-1]
    assert {0, 1, 2, 3} <= set(gap[same_len]) and (gap[same_len] >= 4).any() and (~same_len).any()
    assert len(np.unique(lens)) == 2 and not np.array_equal(rec[:, 3], np.arange(n_pos))
    # queries: the leaves whose sentences straddle a boundary, and others
    leaf_rows = [rec[p, 2] for p in bnd] + [rec[p - 1, 2] for p in bnd]
    rng = np.random.default_rng(k)
    Q = np.concatenate([t["mean"][leaf_rows], queries_near(t["mean"][t["leaves"]], BIN_NQ - len(leaf_rows), 0.3, seed=k)])
    Q = Q.astype(np.float32)
    Q[1::4] += (1e-4 * rng.standard_normal(Q[1::4].shape)).astype(np.float32)
    _, leaf = check_fp32_form(w, ref, Q, ks=(k,), host=False)
    want_i, want_v = model_topk(leaf, k)
    if k >= 2:   # equal scores across chunks are in the answer
        assert any(len(set(v)) < len(v) for v in want_v[:, :k])


@pytest.mark.gpu
@pytest.mark.parametrize("k", [20, 64])
def test_k_at_least_n_pos(k):
    """k >= n_pos (15 sentences): every list is short, padded with -1 / -inf, for K32 and the k > 32 insertion."""
    w, ref, t = flat_case(24, 11, "normal", seed=4)
    assert w._index.n_pos == 15 < k
    Q = queries_near(t["mean"], 40, t["qscale"], seed=9)
    check_fp32_form(w, ref, Q, ks=(k,))
    ids, vals = w._index.predict_small(torch.from_numpy(Q[:9]).cuda(), k)
    want_i, want_v = model_topk(ref.fp32_scores(Q[:9])[1], k)
    assert np.array_equal(ids.cpu().numpy(), want_i) and np.array_equal(bits(vals.cpu().numpy()), bits(want_v))
    assert (want_i[:, 15:] == -1).all()


LEVEL_WEIGHTS = {
    "default": None,
    "mixed": (1.0, 0.5, 2.0, 1.5),
    "exponential": tuple(0.5 ** i for i in range(12)),
    "zero": (1.0, 0.0, 1.0, 0.75, 1.0, 0.0, 2.0),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LEVEL_WEIGHTS))
def test_level_weights(name):
    """Path weights (float)(level_w[j] / len) with the default weights, mixed ones, an exponential schedule and one
    with zero weights, on the complete binary tree (two path lengths), through the big and the small path."""
    lw = LEVEL_WEIGHTS[name]
    w, ref, t = binary_case(lw)
    ix = w._index
    assert np.array_equal(ix._level_w_host[:len(lw)], lw) if lw else ix._level_w_host[0] == 1.0
    Q = queries_near(t["mean"][t["leaves"]], 40, 0.3, seed=3)
    check_fp32_form(w, ref, Q, ks=(10, 40), host=False)
    _, leaf = ref.fp32_scores(Q[:6])
    for k in (10, 40):
        ids, vals = ix.predict_small(torch.from_numpy(Q[:6]).cuda(), k)
        want_i, want_v = model_topk(leaf, k)
        assert np.array_equal(ids.cpu().numpy(), want_i) and np.array_equal(bits(vals.cpu().numpy()), bits(want_v))


@pytest.mark.gpu
def test_k_above_max_k():
    """k > 128 in predict_fast_batch: the leaf matrix sorted by torch.sort, the same ranking as the model's."""
    w, ref, t = binary_case()
    Q = queries_near(t["mean"][t["leaves"]], 40, 0.3, seed=8)
    ids, vals = w.predict_fast_batch(Q, 200)
    want_i, want_v = model_topk(ref.fp32_scores(Q)[1], 200)
    assert np.array_equal(ids.cpu().numpy(), want_i) and np.array_equal(bits(vals.cpu().numpy()), bits(want_v))


@pytest.mark.gpu
@pytest.mark.parametrize("max_len", [PT_MAXLEN, PT_MAXLEN + 1])
def test_deep_paths(max_len):
    """Paths of PT_MAXLEN = 1024 nodes through paths_topk_kernel; at 1025 the big path refuses with CobwebB200Error and
    the small path (no such limit) still answers."""
    from test_fused_finish import caterpillar
    w, leaf_vecs = caterpillar(max_len)
    ix = w._index
    assert ix.max_len == max_len
    ref = oracle_of(w)
    rng = np.random.default_rng(max_len)
    Q = (leaf_vecs[rng.integers(0, len(leaf_vecs), 40)] + 0.1 * rng.standard_normal((40, leaf_vecs.shape[1]))).astype(np.float32)
    Q[::5] = leaf_vecs[rng.integers(0, len(leaf_vecs), 8)]
    Qd = torch.from_numpy(Q).cuda()
    if max_len <= PT_MAXLEN:
        check_fp32_form(w, ref, Q, ks=(10, 40))
    else:
        with pytest.raises(CobwebB200Error):
            ix.predict(Qd, 10, small=False)
    _, leaf = ref.fp32_scores(Q[:5])
    ids, vals = ix.predict_small(Qd[:5], 10)
    want_i, want_v = model_topk(leaf, 10)
    assert np.array_equal(ids.cpu().numpy(), want_i) and np.array_equal(bits(vals.cpu().numpy()), bits(want_v))


@pytest.mark.gpu
@pytest.mark.parametrize("n,d,kind", [(400, 64, "unit"), (300, 200, "whitened")])
def test_ifit_trees_with_duplicates(n, d, kind):
    """Trees built by ifit, with repeated documents: the prefix patterns and duplicate runs of real data."""
    x = synth.corpus(n, d, kind, seed=0)
    x[n // 4:n // 4 + 10] = x[5:15]
    x[n // 2:n // 2 + 3] = x[7]
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=x)
    w.build_prediction_index()
    ref = oracle_of(w)
    rec = pos_records(w._index)
    assert (rec[1:, 1] == rec[1:, 0]).any()                     # sentences sharing a leaf
    q, _ = synth.queries(x, 70, kind, seed=1)
    q[::7] = x[5:15]
    check_operands(w._index, ref)
    check_fp32_form(w, ref, q, ks=(10, 33))


# ------------------------------------------------------------------ non-finite scores
@functools.lru_cache(maxsize=None)
def overflow_case():
    """prior_var = 1e-37, D = 64: a one-sentence leaf has var 1e-37 and r ~ 3e18, so any query about 1 away from it sums
    u^2 past FLT_MAX and its leaf score is -inf; a query at a leaf's mean scores that leaf (and its duplicate) finitely."""
    t = flat_arrays(64, 48, "normal", seed=6)
    t["prior_var"] = 1e-37
    t["count"][1:] = 1.0
    t["m2"][1:] = 0.0
    t["nsent"][1:] = 1
    t["mean"][2] = t["mean"][1]                               # an exact duplicate leaf
    t["count"][0], t["mean"][0], t["m2"][0] = agg_root(np.ones(48), t["mean"][1:].astype(np.float64), np.zeros((48, 64)))
    t["count"] = t["count"].astype(np.float32)
    t["mean"], t["m2"] = t["mean"].astype(np.float32), t["m2"].astype(np.float32)
    t["leaf_of_sentence"] = np.random.default_rng(6).permutation(np.arange(1, 49)).astype(np.int32)
    w = engine_from_arrays(t)
    return w, oracle_of(w), t


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5, 40])
@pytest.mark.parametrize("path", ["fp32", "small"])
def test_fewer_finite_scores_than_k(path, k):
    """Rows with fewer finite leaf scores than k: the -inf sentences fill the rest of the list in id order, on the
    K32 insertion, the k > 32 insertion and the small path alike."""
    w, ref, t = overflow_case()
    ix = w._index
    nq = 40 if path == "fp32" else 9
    Q = t["mean"][1 + np.arange(nq) % 48].copy()
    node, leaf = ref.fp32_scores(Q)
    finite = np.isfinite(leaf).sum(1)
    assert (finite >= 1).all() and (finite < k).all() and np.isinf(node).any()
    want_i, want_v = model_topk(leaf, k)
    assert (want_i >= 0).all()
    Qd = torch.from_numpy(Q).cuda()
    assert ix._route(nq, k, "fp32") == path
    ids, vals, _ = ix.predict(Qd, k, mode="fp32")
    assert np.array_equal(ids.cpu().numpy(), want_i), "ids"
    assert_bits(vals.cpu().numpy(), want_v, "scores")
    if path == "fp32":
        assert_bits(ix.node_scores(Qd).cpu().numpy(), node, "node scores")
        ids, vals, lg = ix.predict(Qd, k, want_leaf_scores=True, mode="fp32")
        assert_bits(lg.cpu().numpy(), leaf, "leaf scores")
        assert np.array_equal(ids.cpu().numpy(), want_i) and np.array_equal(bits(vals.cpu().numpy()), bits(want_v))
