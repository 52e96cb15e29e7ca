"""The fused predict's internal operand set holds path sums (rag-cobweb_b200/csrc/cw_half.cu, hn_build_kernel): row n
carries B'_n = sum_{j in path(n)} w_j B_j and h'_n = sum_j w_j h_j, so the three-product score kernel writes the ancestor
sums C[n] = sum_j w_j s_j that the leaf filter and the finish stage read, with no cumulative-sum pass.  Checked here
against float64 references built from the store's own rows: C for every internal row and query, the decoded operand
image, answers bit-identical to the FP32 path, and one call's kernel list."""
import numpy as np
import pytest
import torch

from rag_cobweb_b200 import CobwebWrapper, synth
from test_fused_finish import caterpillar

pytestmark = pytest.mark.gpu
SCHEDULE = [1.0, 0.5, 2.0, 1.5]


def build(x, weights):
    w = CobwebWrapper(corpus=[None] * len(x), corpus_embeddings=x)
    if weights is not None:
        w.set_level_weights(weights)
    w.build_prediction_index()
    return w


def fused_predict(ix, qd, k=10):
    """The fused call, checked bit for bit against the FP32 path."""
    ids32, v32, _ = ix.predict(qd, k, mode="fp32")
    ix.TENSOR_MIN_NODES = 0  # small trees: run them on the fused pipeline all the same
    ix.set_mode("fused")
    assert ix.fused_ready(k) and ix.hx["n_int"] > 0
    ids, vals, _ = ix.predict(qd, k, small=False)
    assert torch.equal(ids, ids32) and torch.equal(vals, v32)
    assert ix.stats["unresolved"] == 0 and ix.stats["audit_mismatch"] == 0, ix.stats


def float64_reference(w, ix):
    """Per internal row in float64: the node operands iv = 1/var and m = -2 mean/var (the store's fp32 variance, as the
    kernels take it), h = -0.5 (sumlog + sum_d mean^2/var), and their path sums with the level weights, plus
    W = sum over the path of |w_j|."""
    F, st = ix.hx["F"], w.tree.store
    node = ix.order.long()[F["int_rows"].long()]
    mu = st.mean[node].double()
    iv = 1.0 / w.tree.compute_var(st.m2[node], st.count[node][:, None]).double()
    m = -2.0 * mu * iv
    h = -0.5 * (ix.sumlog[F["int_rows"].long()].double() + (mu * mu * iv).sum(1))
    par, wv, off = F["int_parent"].long(), F["int_w"].double(), F["level_off"].tolist()
    Biv, Bm, Hp, W = (torch.zeros_like(t) for t in (iv, m, h, h))
    for a, b in zip(off[:-1], off[1:]):                 # parents sit in the level above
        p = par[a:b]
        has = (p >= 0)
        pc = p.clamp_min(0)
        for acc, own in ((Biv, iv), (Bm, m)):
            acc[a:b] = torch.where(has[:, None], acc[pc], 0.0) + wv[a:b, None] * own[a:b]
        Hp[a:b] = torch.where(has, Hp[pc], 0.0) + wv[a:b] * h[a:b]
        W[a:b] = torch.where(has, W[pc], 0.0) + wv[a:b].abs()
    return dict(iv=iv, m=m, h=h, Biv=Biv, Bm=Bm, Hp=Hp, W=W)


def check_ancestor_sums(w, ix, qd):
    """Device C (the score matrix S after a fused call) against sum_j w_j s_j in float64.  Allowed: half of eps's
    operand term, 0.5 * eps_scale * T * W (T = 2 (|x|^2 / prior + hmax) bounds the contraction's magnitude, W =
    sum_path |w_j|), plus one fp32 ulp of the score magnitude 0.5 W (lmax + hmax + T) for the rounding of h' and of the
    epilogue's result (eps's ulp term takes 4 + 3 sqrt(max_len) of those)."""
    R, fi = float64_reference(w, ix), ix.hx["fi"]
    x = qd.double()
    s = R["h"][:, None] - 0.5 * (R["iv"] @ (x * x).T + R["m"] @ x.T)        # [n_int, nq] node scores
    F = ix.hx["F"]
    par, wv, off = F["int_parent"].long(), F["int_w"].double(), F["level_off"].tolist()
    Cref = torch.zeros_like(s)
    for a, b in zip(off[:-1], off[1:]):
        p = par[a:b]
        Cref[a:b] = torch.where((p >= 0)[:, None], Cref[p.clamp_min(0)], 0.0) + wv[a:b, None] * s[a:b]
    n_int, nq = ix.hx["n_int"], qd.shape[0]
    Cgot = ix._hws["S"][:n_int, :nq].double()
    T = 2.0 * ((x * x).sum(1) / float(w.tree.store.prior_var) + fi.hmax)    # [nq]
    op = 0.5 * ix.eps_scale * T[None, :] * R["W"][:, None]
    ulp = 2.0 ** -23 * 0.5 * (fi.lmax + fi.hmax + T[None, :]) * R["W"][:, None]
    err = (Cgot - Cref).abs()
    assert bool(torch.isfinite(Cgot).all())
    assert bool((err <= op + ulp).all()), float((err / (op + ulp)).max())


@pytest.mark.parametrize("d,kind,weights", [
    (7, "unit", None), (7, "whitened", SCHEDULE),
    (33, "unit", SCHEDULE), (33, "whitened", None),
    (128, "unit", None), (128, "whitened", SCHEDULE),
    (768, "unit", SCHEDULE), (768, "whitened", None),
    (1030, "unit", None), (1030, "whitened", SCHEDULE),
])
def test_ancestor_sums_vs_float64(d, kind, weights):
    """Trees from the engine's own ifit at D = 7 ... 1030 (a partial last slab of 16 attributes at 7, 33 and 1030),
    unit and whitened data, the default weights and a non-uniform schedule."""
    x = synth.corpus(500, d, kind, seed=d)
    w = build(x, weights)
    ix = w._index
    q, _ = synth.queries(x, 128, kind, seed=d + 1)
    qd = torch.from_numpy(q).cuda()
    fused_predict(ix, qd)
    check_ancestor_sums(w, ix, qd)


@pytest.mark.parametrize("max_len", [300, 500])
@pytest.mark.parametrize("weights", [None, SCHEDULE])
def test_ancestor_sums_deep_paths(max_len, weights):
    """Caterpillar trees: internal rows whose operands sum 299 and 499 rows, the deepest the fused mode takes."""
    w, leaf_vecs = caterpillar.__wrapped__(max_len)   # a fresh tree: the level weights change it
    if weights is not None:
        w.set_level_weights(weights)
        w.build_prediction_index()
    ix = w._index
    assert ix.max_len == max_len
    rng = np.random.default_rng(max_len + 7)
    q = leaf_vecs[rng.integers(0, len(leaf_vecs), 64)] + 0.1 * rng.standard_normal((64, leaf_vecs.shape[1])).astype(np.float32)
    qd = torch.from_numpy(q).cuda()
    fused_predict(ix, qd)
    check_ancestor_sums(w, ix, qd)


def test_decoded_operand_image():
    """The internal set's fp16 image (hi + lo, 64-byte swizzle, per-row power-of-two scale) decodes to the float64 path
    sums B' to 2^-22 of the row maximum, and its h' to fp32 rounding; the padding of the last slab is zero."""
    d = 40
    x = synth.corpus(400, d, "whitened", seed=11)
    w = build(x, SCHEDULE)
    ix = w._index
    ix.set_mode("fused")
    hx = ix.hx
    n_int, n_sl = hx["n_int"], (d + 15) // 16
    nt = (n_int + 255) // 256
    img = hx["B_int"].view(torch.float16).view(nt, n_sl, 2, 256, 4, 8).double()
    val = img[:, :, 0] + img[:, :, 1]                                        # [tile, slab, row, 16-byte chunk, 8]
    r = torch.arange(256, device=val.device)
    phys = torch.arange(4, device=val.device)[None, :] ^ ((r[:, None] >> 1) & 3)    # logical chunk -> stored chunk
    val = val.gather(3, phys[None, None, :, :, None].expand(nt, n_sl, 256, 4, 8))
    val = val.permute(0, 2, 3, 1, 4)                                         # [tile, row, chunk, slab, 8]
    scale = -2.0 * hx["rc_int"].view(-1, 2)[:, 1].double()                   # 2^-s per row
    iv_img = val[:, :, :2].permute(0, 1, 3, 2, 4).reshape(nt * 256, n_sl * 16) * scale[:, None]
    m_img = val[:, :, 2:].permute(0, 1, 3, 2, 4).reshape(nt * 256, n_sl * 16) * scale[:, None]
    assert not bool(iv_img[:, d:].any()) and not bool(m_img[:, d:].any())
    R = float64_reference(w, ix)
    rowmax = torch.maximum(R["Biv"].abs().amax(1), R["Bm"].abs().amax(1))[:, None]
    tol = 2.0 ** -22 * rowmax * (1 + 1e-5)
    assert bool(((iv_img[:n_int, :d] - R["Biv"]).abs() <= tol).all())
    assert bool(((m_img[:n_int, :d] - R["Bm"]).abs() <= tol).all())
    h_img = hx["rc_int"].view(-1, 2)[:n_int, 0].double()
    assert bool(((h_img - R["Hp"]).abs() <= 2.0 ** -23 * R["Hp"].abs()).all())


def test_no_cumulative_sum_launch():
    """One fused call launches the score kernel and no cumulative-sum kernel."""
    x = synth.corpus(1500, 64, "unit", seed=3)
    w = build(x, None)
    ix = w._index
    q, _ = synth.queries(x, 300, "unit", seed=4)
    qd = torch.from_numpy(q).cuda()
    fused_predict(ix, qd)                       # builds the operand sets and the work buffers
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ix.predict(qd, 10, small=False)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any("h_score_kernel" in n for n in names), names
    assert not [n for n in names if "cumsum" in n.lower()], names
