"""Best-first categorize (categorize_kernel, rag-cobweb_b200/csrc/cw_categorize.cu) and the index's sums of log-variances
(index_sumlog_kernel, csrc/cw_index.cu) against the CPU oracle, bit for bit, on every branch of their team reduction.

Both kernels score a row with a team of Gp = pow2_ceil(ceil(D / 4)) threads: group4 over the four attributes of a lane,
a butterfly over tw = min(Gp, 32) lanes, and a cross-warp step when the team spans wpt = Gp / 32 > 1 warps.  A CTA holds
NT = max(Gp, 256) / Gp teams.  The trees are loaded from arrays (node i of the arrays is node id i in the store and slot i
in the oracle), so D reaches CW_MAX_D = 4096 and the test picks the exact statistics.

Retrieval returns an order, and sibling log-probs of ordinary data lie far apart, so a kernel that loses the last bits
still pops in the oracle's order.  The probe trees make the order depend on the last bit: a base leaf, and probe
siblings pushed before it that differ from it in one attribute p each.  The probe's mean at p is moved away from the query
by the fewest float32 steps (found with the oracle) that raise its float32 -log_prob above the base's, so the oracle pops
the base first; a kernel that drops or misrounds the term of p ties the probe with the base or undercuts it, and the probe
pops first (push order).  Every probe asserts that it is live: with attribute p put back to the base value the oracle's
order changes.
"""
import numpy as np
import pytest
import torch

from oracle.cobweb_oracle import OracleTree, default_prior_var
from rag_cobweb_b200 import CobwebTorchTree, DenseIndex, _lib

pytestmark = pytest.mark.gpu
NO_LIMIT = 1 << 62


def launch_shape(d):
    """(Gp, NT) of categorize_kernel and index_sumlog_kernel at dimension d (the launch formulas of cw_categorize and
    cw_index_build)."""
    gp = 1
    while gp < (d + 3) // 4:
        gp <<= 1
    return gp, max(gp, 256) // gp


# ------------------------------------------------------------------ float32 steps
def f32_ord(v):
    """float32 -> integer that orders like the value (+0 and -0 both 0)."""
    b = int(np.float32(v).view(np.int32))
    return b if b >= 0 else -(b & 0x7fffffff)


def ord_f32(o):
    return np.uint32(o if o >= 0 else (-o) | 0x80000000).view(np.float32)


def step_away(v, x, n):
    """v moved n float32 steps further from x."""
    return ord_f32(f32_ord(v) + (n if v >= x else -n))


# ------------------------------------------------------------------ probe trees (oracle side: runs without a GPU)
def row_neg(ref, count, mean, m2, x):
    """float32 -log_prob of one node row (the oracle's arithmetic), through a one-node tree."""
    ref.load([-1], [count], [1], mean[None], m2[None])
    return np.float32(-ref.log_prob(0, x))


def size_probe(ref, count, base, m2, x, p):
    """The base row with attribute p moved away from x[p] by the fewest float32 steps that raise its -log_prob above the
    base's; returns (row, gap in float32 steps of -log_prob)."""
    base_neg = row_neg(ref, count, base, m2, x)
    row = base.copy()

    def neg(n):
        row[p] = step_away(base[p], x[p], n)
        return row_neg(ref, count, row, m2, x)

    hi = 1
    while not neg(hi) > base_neg:
        hi *= 2
        assert hi < 1 << 30 and np.isfinite(row[p]), f"attribute {p} cannot move the score"
    lo = hi // 2 if hi > 1 else 0
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if neg(mid) > base_neg:
            hi = mid
        else:
            lo = mid
    gap = f32_ord(neg(hi)) - f32_ord(base_neg)
    return row.copy(), gap


def probe_attrs(d):
    """Where the reduction changes hands: the first group4 boundary (0, 3, 4), the first and last attribute of every
    warp's 128-attribute span of a team (128 j, 128 j - 1), both ends of the last full group, each real attribute of a
    partial last group, and D - 1."""
    full = d // 4
    s = {0, 3, 4, 4 * full - 4, 4 * full - 1, d - 1}
    s.update(a for j in range(0, d + 1, 128) for a in (j, j - 1))
    s.update(range(4 * full, d))
    return sorted(a for a in s if 0 <= a < d)


def probe_tree(d, kw, count, base, m2, x, attrs):
    """Flat tree: root -> [one probe per attribute of attrs, the base leaf, fillers].  Fillers (the base row with one
    attribute 1000 (j + 1) steps further from the query) give the root more children than a CTA has teams, so one
    expansion takes several rounds.  Returns the tree's arrays, the oracle answer with k = all leaves, and the gaps."""
    ref = OracleTree(d, **kw)
    rows, gaps = [], []
    for p in attrs:
        row, gap = size_probe(ref, count, base, m2, x, p)
        rows.append(row)
        gaps.append(gap)
    n_fill = max(2, launch_shape(d)[1] + 4 - len(attrs))
    for j in range(n_fill):
        row = base.copy()
        a = (7 * j) % d
        row[a] = step_away(base[a], x[a], 1000 * (j + 1))
        rows.append(row)
    nl = len(rows) + 1
    leaf_mean = np.stack(rows[:len(attrs)] + [base] + rows[len(attrs):])
    t = dict(d=d, kw=kw, x=x, nl=nl, gaps=gaps,
             parent=np.array([-1] + [0] * nl), count=np.array([count * nl] + [count] * nl, np.float32),
             nsent=np.array([0] + [1] * nl, np.int32),
             mean=np.concatenate([base[None], leaf_mean]).astype(np.float32),
             m2=np.concatenate([np.full((1, d), count * nl, np.float32), np.broadcast_to(m2, (nl, d))]).astype(np.float32))
    t["want"] = oracle_answer(t, ref)
    # liveness: attribute p of probe i put back to the base value changes the order
    for i, p in enumerate(attrs):
        mean = t["mean"].copy()
        mean[1 + i] = base
        order = oracle_answer(dict(t, mean=mean), ref)[0]
        assert not np.array_equal(order, t["want"][0]), f"probe of attribute {p} is not decisive"
    return t


def oracle_answer(t, ref=None):
    """(leaves in retrieval order with k = all leaves, nfound, best, lp_calls) of the oracle for t's query."""
    if ref is None:
        ref = OracleTree(t["d"], **t["kw"])
    ref.load(t["parent"], t["count"], t["nsent"], t["mean"], t["m2"])
    leaves, nfound, _, calls = ref.categorize(t["x"][None], k=t["nl"])
    _, _, best, _ = ref.categorize(t["x"][None], k=0)
    return leaves[0], nfound[0], best[0], calls[0]


FORMS = {  # leaf count, m2 and scoring flags of each form of log_prob
    "cached": (1, lambda rng, d: np.zeros(d, np.float32), {}),                         # var = prior on every attribute
    "count2": (2, lambda rng, d: rng.uniform(0.02, 0.5, d).astype(np.float32), {}),  # cached var / tf rows differ
    "long_form": (2, lambda rng, d: rng.uniform(0.02, 0.5, d).astype(np.float32), dict(use_info=False)),
    "acuity_cutoff": (2, lambda rng, d: rng.uniform(0.0, 0.25, d).astype(np.float32), dict(acuity_cutoff=True)),
}


def ulp_probe_tree(d, form, seed=0):
    rng = np.random.default_rng(seed + d)
    count, m2_of, kw = FORMS[form]
    base = rng.standard_normal(d).astype(np.float32)
    x = (base + 0.5 * rng.standard_normal(d)).astype(np.float32)
    t = probe_tree(d, kw, count, base, m2_of(rng, d), x, probe_attrs(d))
    assert max(t["gaps"]) <= 4, t["gaps"]  # each probe sits a few float32 steps above the base
    return t


# The fallback division of the cached form: the decisive attribute's numerator 0.5 (x - mean)^2 or variance lies outside
# [2^-60, 2^60), where cat_div_core's range checks send all four divisions of the lane to the plain IEEE division.
# regime: (mean scale, query offset scale on the other attributes (numerators inside the window), base mean at the probed
# attributes (None: as the others), query offset there, prior_var); leaves have count 1 and m2 = 0, so var = prior_var.
FALLBACK = {
    "num_below_window": (2.0 ** -9, 2.0 ** -29, None, 2.0 ** -31, 2.0 ** -59),  # numerator 2^-63, variance 2^-59
    "num_zero": (1.0, 0.5, None, 0.0, None),                                   # query on the mean: +0, fast path
    "num_above_window": (1.0, 0.5, 2.0 ** 31, 2.0 ** 31, None),                # numerator 2^61
    "var_below_window": (1.0, 0.5, None, 0.5, 2.0 ** -64),
    "var_subnormal": (2.0 ** -9, 2.0 ** -29, None, 2.0 ** -29, 2.0 ** -130),   # the fast path's reciprocal flushes to 0
}


def fallback_tree(d, regime, seed=0):
    rng = np.random.default_rng(seed + d)
    scale, off, probe_mean, probe_off, prior = FALLBACK[regime]
    attrs = [0, 5, d - 1]
    base = (scale * rng.uniform(1.0, 2.0, d)).astype(np.float32)
    if probe_mean is not None:
        base[attrs] = probe_mean
    x = (base + off * rng.uniform(1.0, 2.0, d)).astype(np.float32)
    x[attrs] = base[attrs] - np.float32(probe_off)
    kw = {} if prior is None else dict(prior_var=prior)
    t = probe_tree(d, kw, 1, base, np.zeros(d, np.float32), x, attrs)
    # the regime holds at the probed attribute of the base row and of its probe row
    pv = np.float32(default_prior_var() if prior is None else prior)
    for i, p in enumerate(attrs):
        for which, row in (("base", base), ("probe", t["mean"][1 + i])):
            df = np.float32(x[p] - row[p])
            num = np.float32(0.5) * np.float32(df * df)
            ok = dict(num_below_window=0 < num < 2.0 ** -60, num_zero=(num == 0) == (which == "base"),
                      num_above_window=num >= 2.0 ** 60, var_below_window=pv < 2.0 ** -60,
                      var_subnormal=pv < np.finfo(np.float32).tiny)[regime]
            assert ok, (regime, p, which, float(num))
    return t


# ------------------------------------------------------------------ engine side
def engine_tree(t):
    tree = CobwebTorchTree((t["d"],), **t["kw"])
    tree.load_arrays(t["parent"], t["count"], t["nsent"], t["mean"], t["m2"])
    return tree


def assert_same_answer(tree, t):
    want_leaves, want_nf, want_best, want_calls = t["want"]
    r = tree.categorize_batch(t["x"][None], retrieve_k=t["nl"])
    assert np.array_equal(r["leaves"][0].cpu().numpy(), want_leaves)
    assert int(r["nfound"][0]) == want_nf and int(r["lp_calls"][0]) == want_calls
    assert int(tree.categorize_batch(t["x"][None])["best"][0]) == want_best


def assert_sumlog(tree, t):
    """DenseIndex.sumlog (index_sumlog_kernel) equals the oracle's bit for bit; it does not depend on the sentences."""
    ix = DenseIndex(tree, np.zeros(0, np.int32))
    ref = OracleTree(t["d"], **t["kw"])
    ref.load(t["parent"], t["count"], t["nsent"], t["mean"], t["m2"])
    want = ref.build_index()["sumlog"]
    assert ix.nn == len(want)
    assert np.array_equal(ix.sumlog[:ix.nn].cpu().numpy(), want)


SHAPES = [(7, "gp2-nt128"), (33, "gp16-partial-group"), (64, "gp16-two-teams-per-warp"),
          (100, "gp32-one-team-per-warp-7-idle-lanes"), (1024, "gp256-nt1-wpt8"), (2052, "gp1024-513-groups"),
          (4093, "gp1024-partial-last-group"), (4096, "gp1024-wpt32")]


@pytest.mark.parametrize("form", list(FORMS))
@pytest.mark.parametrize("d", [pytest.param(d, id=f"D{d}-{name}") for d, name in SHAPES])
def test_ulp_probes(d, form):
    t = ulp_probe_tree(d, form)
    tree = engine_tree(t)
    assert_same_answer(tree, t)
    assert_sumlog(tree, t)


@pytest.mark.parametrize("regime", list(FALLBACK))
@pytest.mark.parametrize("d", [pytest.param(33, id="D33-scalar-loads"), pytest.param(64, id="D64-float4-loads")])
def test_fallback_division(d, regime):
    t = fallback_tree(d, regime)
    tree = engine_tree(t)
    assert_same_answer(tree, t)
    assert_sumlog(tree, t)


@pytest.mark.parametrize("d", [pytest.param(7, id="D7-nt128"), pytest.param(100, id="D100-nt8"),
                               pytest.param(4096, id="D4096-wpt32")])
def test_heap_ties(d):
    """root -> A, B; A -> a1, a2 and B -> b1, b2, all four leaves one row.  A scores above B, so A is expanded first and
    a1, a2 are pushed before b1, b2; on the tie in -log_prob the lower parent score pops first (b1, b2), and siblings pop
    in push order (b1 before b2, a1 before a2)."""
    rng = np.random.default_rng(d)
    x = rng.standard_normal(d).astype(np.float32)
    mean = np.stack([x, x + 0.1, x + 0.2] + [x + 1.0] * 4).astype(np.float32)
    t = dict(d=d, kw={}, x=x, nl=4, parent=np.array([-1, 0, 0, 1, 1, 2, 2]),
             count=np.array([4, 2, 2, 1, 1, 1, 1], np.float32), nsent=np.array([0, 0, 0, 1, 1, 1, 1], np.int32),
             mean=mean, m2=np.ones((7, d), np.float32))
    t["want"] = oracle_answer(t)
    assert list(t["want"][0]) == [5, 6, 3, 4]
    assert_same_answer(engine_tree(t), t)


# ------------------------------------------------------------------ several queries per CTA
def two_level(d, n_mid, n_leaf, seed, leaf_var=None):
    """root -> n_mid internal nodes -> n_leaf leaves each, BFS order.  Internal nodes are wide (variance about 4), leaves
    narrow, so a query far from every cluster expands every internal node before its first leaf."""
    rng = np.random.default_rng(seed)
    centre = 3.0 * rng.standard_normal((n_mid, d))
    leaf = np.repeat(centre, n_leaf, 0) + 0.3 * rng.standard_normal((n_mid * n_leaf, d))
    nn = 1 + n_mid + n_mid * n_leaf
    parent = np.concatenate([[-1], np.zeros(n_mid, np.int64), 1 + np.repeat(np.arange(n_mid), n_leaf)])
    count = np.concatenate([[n_mid * n_leaf], np.full(n_mid, n_leaf), np.ones(n_mid * n_leaf)]).astype(np.float32)
    mean = np.concatenate([np.zeros((1, d)), centre, leaf]).astype(np.float32)
    m2 = np.zeros((nn, d), np.float32)
    m2[0] = 10.0 * n_mid * n_leaf
    m2[1:1 + n_mid] = 4.0 * n_leaf * rng.uniform(0.8, 1.2, (n_mid, d))
    if leaf_var is not None:
        m2[1 + n_mid:] = leaf_var * rng.uniform(0.5, 1.5, (n_mid * n_leaf, d))
    nsent = (np.arange(nn) > n_mid).astype(np.int32)
    return dict(d=d, kw={}, parent=parent, count=count, nsent=nsent, mean=mean, m2=m2, leaf=leaf.astype(np.float32))


def categorize_direct(tree, Q, k, n_ctas, max_nodes=NO_LIMIT, greedy=False, use_best=True, alone=False):
    """cw_categorize on caller-owned buffers with the wrapper's frontier bound (n_live_bound rows per CTA); outputs
    prefilled with values the kernel never writes.  alone: one launch per query (grid of one CTA)."""
    L = _lib.load()
    nq = Q.shape[0]
    fcap = int(tree.store.header()[_lib.HDR_N_USED]) + 1
    frontier = torch.empty(n_ctas * fcap * 4, dtype=torch.int32, device="cuda")
    leaves = torch.full((nq, max(k, 1)), -7, dtype=torch.int32, device="cuda")
    nfound = torch.full((nq,), -7, dtype=torch.int32, device="cuda")
    best = torch.full((nq,), -7, dtype=torch.int32, device="cuda")
    calls = torch.full((nq,), -7, dtype=torch.int64, device="cuda")
    spans = [(q, 1) for q in range(nq)] if alone else [(0, nq)]
    for q, n in spans:
        _lib.check(L.cw_categorize(tree.store.struct(), Q[q].data_ptr(), n, k, max_nodes, int(greedy), int(use_best),
                                   n_ctas, frontier.data_ptr(), fcap, leaves[q].data_ptr(), nfound[q:].data_ptr(),
                                   best[q:].data_ptr(), calls[q:].data_ptr(), _lib.stream_ptr()), "cw_categorize")
    out = [best.cpu().numpy(), calls.cpu().numpy()]
    if k:
        out = [leaves.cpu().numpy(), nfound.cpu().numpy()] + out[1:]
    return out


MULTI_CASES = {  # launch options -> what the outputs hold
    "k3": dict(k=3),
    "k0-max_nodes4": dict(k=0, max_nodes=4),
    "k0-greedy": dict(k=0, greedy=True),
    "k0-last_popped-max_nodes9": dict(k=0, use_best=False, max_nodes=9),
}


def test_several_queries_per_cta():
    """About 1500 queries on one launch: a query near a leaf stops after a few pops with a frontier of about 90 entries,
    every third query lies far from every cluster and opens a frontier of about 1600.  n_ctas = 1, 3 and 592 give each
    CTA about 1500, 500 and 2.5 queries in a row, so each query starts on the frontier slice, xs, F and reduction buffers
    a very different query left behind.  Every answer equals the oracle's and the same query answered alone."""
    d, n_mid, n_leaf = 32, 64, 25
    t = two_level(d, n_mid, n_leaf, seed=5)
    rng = np.random.default_rng(6)
    nq = 1500
    near = t["leaf"][rng.integers(0, len(t["leaf"]), nq)] + 0.01 * rng.standard_normal((nq, d))
    far = 12.0 * rng.standard_normal((nq, d))
    Qn = np.where((np.arange(nq) % 3 == 0)[:, None], far, near).astype(np.float32)
    tree = engine_tree(t)
    ref = OracleTree(d)
    ref.load(t["parent"], t["count"], t["nsent"], t["mean"], t["m2"])
    Q = torch.from_numpy(Qn).cuda()
    assert nq > _lib.load().cw_categorize_ctas()
    for name, kw in MULTI_CASES.items():
        k = kw["k"]
        opts = dict(max_nodes=kw.get("max_nodes", NO_LIMIT), greedy=kw.get("greedy", False),
                    use_best=kw.get("use_best", True))
        rl, rnf, rbest, rcalls = ref.categorize(Qn, k=k, **opts)
        want = [rl, rnf, rcalls] if k else [rbest, rcalls]
        if name == "k3":   # the mix holds: some queries score every node, others stop after a few pops
            assert rcalls.max() == len(t["parent"]) and np.median(rcalls) < 100
        for n_ctas in (1, 3, 592, "alone"):
            got = categorize_direct(tree, Q, k, 1 if n_ctas == "alone" else n_ctas, alone=n_ctas == "alone", **opts)
            for g, w in zip(got, want):
                assert np.array_equal(g, w), (name, n_ctas)
    r = tree.categorize_batch(Qn, retrieve_k=3)
    rl, rnf, _, rcalls = ref.categorize(Qn, k=3)
    assert np.array_equal(r["leaves"].cpu().numpy(), rl) and np.array_equal(r["nfound"].cpu().numpy(), rnf)
    assert np.array_equal(r["lp_calls"].cpu().numpy(), rcalls)


# ------------------------------------------------------------------ sumlog beyond one grid pass
@pytest.mark.parametrize("d", [pytest.param(1024, id="D1024-nt1"), pytest.param(2052, id="D2052-nt1"),
                               pytest.param(4096, id="D4096-nt1")])
def test_sumlog_second_grid_pass(d):
    """3061 rows at NT = 1: the grid of index_sumlog_kernel is capped at 148 * 16 = 2368 CTAs, so the last 693 rows are
    written by the second pass of its grid-stride loop."""
    t = two_level(d, 60, 50, seed=d, leaf_var=0.2)
    assert len(t["parent"]) > 148 * 16 and launch_shape(d)[1] == 1
    assert_sumlog(engine_tree(t), t)
