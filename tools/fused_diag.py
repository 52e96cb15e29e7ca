"""Stage-by-stage check of the fused tcgen05 predict (cw_half.cu) against the FP32 form on one tree:
cumulative ancestor sums (against a float64 sum of the FP32 node scores, and as a fraction of eps), filter scores and
their error bound, candidate counts, final ids/scores, timing.
  python tools/fused_diag.py [docs] [dim] [unit|whitened] [queries] [k]"""
import ctypes as C
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rag_cobweb_b200 import CobwebWrapper, DenseIndex, _lib, synth  # noqa: E402

n, d, kind, nq, k = (int(sys.argv[1]) if len(sys.argv) > 1 else 30000, int(sys.argv[2]) if len(sys.argv) > 2 else 128,
                     sys.argv[3] if len(sys.argv) > 3 else "unit", int(sys.argv[4]) if len(sys.argv) > 4 else 1000,
                     int(sys.argv[5]) if len(sys.argv) > 5 else 10)
DenseIndex.TENSOR_MIN_NODES = 0
x = synth.corpus(n, d, kind, seed=0)
w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=torch.from_numpy(x).cuda())
q, targets = synth.queries(x, nq, kind, seed=1)
qd = torch.from_numpy(q).cuda()
w.build_prediction_index()
ix = w._index
ix.audit_every = 64
ids32, v32, leaf32 = ix.predict(qd, k, want_leaf_scores=True, mode="fp32")
ns32 = ix.node_scores(qd).clone()          # [nq, nn]
ix.set_mode("fused")
hx = ix.hx
F = hx["F"]
print(f"tree {n}x{d} {kind}: nn {ix.nn}, internal {hx['n_int']}, leaves {hx['n_leaf']}, sample tiles {hx['n_s']}, "
      f"leaf layout F{hx['leaf_layout']}, max_len {ix.max_len}, e1max {hx['fi'].e1max:.3e}, hmax {hx['fi'].hmax:.3f}", flush=True)
ids, vals, _ = ix.predict(qd, k, small=False)
torch.cuda.synchronize()
print("stats", ix.stats, flush=True)
same_i = (ids == ids32).all(1)
same_v = (vals == v32).all(1)
print(f"ids identical {float(same_i.float().mean()):.4f}, scores bit-identical {float(same_v.float().mean()):.4f}", flush=True)
hw = ix._hws
# ---- cumulative sums of the internal rows
if hx["n_int"]:
    int_rows = torch.as_tensor(F["int_rows"], device="cuda")
    par = F["int_parent"]
    wv = F["int_w"]
    S = ns32[:, int_rows].double().T.contiguous()   # [n_int, nq]
    Cref = torch.zeros_like(S)
    off = F["level_off"]
    for lv in range(len(off) - 1):
        r = torch.arange(off[lv], off[lv + 1], device="cuda")
        p = torch.as_tensor(par[off[lv]:off[lv + 1]], device="cuda").long()
        base = torch.where((p >= 0)[:, None], Cref[p.clamp_min(0)], torch.zeros_like(S[r]))
        Cref[r] = base + torch.as_tensor(wv[off[lv]:off[lv + 1]], device="cuda").double()[:, None] * S[r]
    Cgot = hw["S"][: hx["n_int"], :nq].double()
    err = (Cgot - Cref).abs()
    print(f"cumulative sums: max abs err {float(err.max()):.3e} (max |C| {float(Cref.abs().max()):.3f}); root row err "
          f"{float(err[0].max()):.3e}", flush=True)
    # against eps of each query (cw_half.cu eps_of); C enters a leaf score divided by the path length, which is left out
    fi = hx["fi"]
    tq = 2.0 * ((qd.double() ** 2).sum(1) / fi.prior_var + fi.hmax)
    op = fi.wfac * fi.eps_scale * tq
    eps = op + fi.wfac * 2.0 ** -23 * (4.0 + 3.0 * ix.max_len ** 0.5) * 0.5 * (fi.lmax + fi.hmax + tq)
    print(f"cumulative sums vs eps: max |C - C_ref| / eps {float((err / eps[None, :]).max()):.4f}, / eps operand term "
          f"(eps_scale T wfac) {float((err / op[None, :]).max()):.4f}", flush=True)
# ---- filter candidates: a1 vs the exact leaf score, against the bound
cnt = hw["cnt"][:nq].cpu().numpy()
print(f"candidates per query: mean {cnt.mean():.1f} median {np.median(cnt):.0f} max {cnt.max()} (cap {ix.FUSED_CAP})", flush=True)
rc = hx["rc_leaf"].view(-1, 8)
qv = hw["qv"][:nq]
sent_off = torch.as_tensor(F["sent_off"], device="cuda").long()
sent_ids = torch.as_tensor(F["sent_ids"], device="cuda").long()
worst, worst_ratio = 0.0, 0.0
for qi in range(0, nq, max(1, nq // 50)):
    c = min(int(cnt[qi]), ix.FUSED_CAP)
    if c == 0:
        continue
    rows = hw["cand_row"][qi, :c].long()
    a1 = hw["cand_val"][qi, :c]
    sid0 = sent_ids[sent_off[rows]]
    ex = leaf32[qi, sid0]
    bound = rc[rows, 4] * qv[qi, 2]
    e = (a1 - ex).abs()
    worst = max(worst, float(e.max()))
    worst_ratio = max(worst_ratio, float((e / bound.clamp_min(1e-30)).max()))
    # every exact top-k sentence must be among the candidates
    cand_sids = set()
    for r in rows.cpu().tolist():
        cand_sids.update(sent_ids[sent_off[r]:sent_off[r + 1]].cpu().tolist())
    missing = [s for s in ids32[qi].cpu().tolist() if s >= 0 and s not in cand_sids]
    if missing:
        print(f"  query {qi}: exact top-k sentences missing from the candidates: {missing}; tau {float(hw['tau'][qi]):.5f}", flush=True)
print(f"filter: max |a1 - exact| {worst:.3e}, max ratio to the bound e1*||a|| {worst_ratio:.3f} (must be < 1)", flush=True)
# ---- host entry point
hs, hv = ix.predict_host(q, k)
print(f"host entry: ids identical {np.mean((hs.numpy() == ids32.cpu().numpy()).all(1)):.4f} scores "
      f"{np.mean((hv.numpy() == v32.cpu().numpy()).all(1)):.4f}", flush=True)
# ---- small path
ss, sv = ix.predict_small(qd[:32].contiguous(), k)
print(f"small path (32): ids identical {float((ss == ids32[:32]).all(1).float().mean()):.4f} scores "
      f"{float((sv == v32[:32]).all(1).float().mean()):.4f}", flush=True)
s1, v1 = ix.predict_small(qd[:1].contiguous(), k)
print(f"small path (1): {bool((s1 == ids32[:1]).all())} {bool((v1 == v32[:1]).all())}", flush=True)
# ---- timing
def timed(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps
t_f = timed(lambda: ix.predict(qd, k, small=False))
t_32 = timed(lambda: ix.predict(qd, k, mode="fp32", small=False), reps=2)
t_s1 = timed(lambda: ix.predict_small(qd[:1], k), reps=20)
t_s32 = timed(lambda: ix.predict_small(qd[:32], k), reps=10)
print(f"timing: fused {t_f:.3f} ms ({nq / t_f * 1e3:.0f} q/s), fp32 {t_32:.3f} ms, small(1) {t_s1:.3f} ms, small(32) {t_s32:.3f} ms")
print("stats", ix.stats)
for rep in range(2):
    print("stages (ms):", {k_: round(v, 3) for k_, v in ix.profile_stages(qd[: ix.fused_workspace(nq, k)["cap_q"]], k).items()})
t_h = timed(lambda: ix.predict_host(q, k))
print(f"host entry: {t_h:.3f} ms ({nq / t_h * 1e3:.0f} q/s)")
import time
t0 = time.time()
for i in range(50):
    w.cobweb_predict_fast(q[i % nq], k=k, return_ids=True, is_embedding=True)
print(f"cobweb_predict_fast single query: {(time.time() - t0) / 50 * 1e3:.3f} ms")
