"""CPU tests of DenseIndex's dispatch: which C entry points a device, host or tag-filtered predict calls, with which
query counts, k, rows and query tags, and which calls it refuses.  No GPU and no built library: _lib.load() is
replaced by a fake that records every cw_* call, and the index is assembled from CPU tensors."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from rag_cobweb_b200 import _lib
from rag_cobweb_b200.wrapper import DenseIndex

D, N_POS = 8, 50
SIZE_QUERIES = ("cw_xt_floats", "cw_score_ldq", "cw_topk_chunks", "cw_small_scratch_words", "cw_fused_flag_words",
                "cw_h_a_bytes")
# argument positions of (Q, nq, k, tag filter, output ids) in the recorded entry points (include/cobweb_b200.h)
ARGS = {
    "cw_small_predict": (1, 2, 7, None, None),
    "cw_small_predict_tagged": (2, 3, 8, 1, None),
    "cw_small_predict_host": (1, 2, 3, None, None),
    "cw_fused_predict": (2, 3, 4, None, 5),
    "cw_fused_predict_tagged": (3, 4, 5, 2, 6),
    "cw_fused_predict_host": (2, 3, 4, None, None),
    "cw_dense_node_scores": (1, 2, None, None, None),
    "cw_dense_paths_topk": (None, 3, 4, None, 6),
    "cw_dense_paths_topk_tagged": (None, 4, 5, 1, 6),
    "cw_predict_dense_host": (2, 3, 4, None, None),
    "cw_leaf_tags": (None, None, None, None, None),
}
FP32_MARK = 7   # what the fake FP32 top-k writes into every id it returns


def _ints(ptr, n, ctype=C.c_int32):
    return (ctype * n).from_address(ptr)


class FakeLib:
    """Records the work entry points as (name, nq, k) plus the rows (Q[:, 0]) and query tags they were given.  Fused
    device calls write the statistics word of unresolved rows and SID_UNRESOLVED into the rows listed in
    `unresolved`; the FP32 top-k writes FP32_MARK."""

    def __init__(self):
        self.calls, self.detail, self.unresolved = [], [], ()

    def __getattr__(self, name):
        if name in SIZE_QUERIES:
            return lambda *a: 4
        if name not in ARGS:
            return lambda *a: 0
        return lambda *a: self._record(name, a)

    def _record(self, name, a):
        iq, inq, ik, itf, isid = ARGS[name]
        nq = a[inq] if inq is not None else None
        k = a[ik] if ik is not None else None
        self.calls.append((name, nq, k))
        d = {}
        if iq is not None and nq:
            d["rows"] = tuple(int(v) for v in np.ctypeslib.as_array(_ints(a[iq], nq * D, C.c_float)).reshape(nq, D)[:, 0])
        if itf is not None and nq:
            d["tags"] = tuple(_ints(a[itf]._obj.query_tags, nq))
        if name in ("cw_fused_predict", "cw_fused_predict_tagged"):
            w = a[1]._obj
            d["audit_phase"] = w.audit_phase
            st = _ints(w.stats, _lib.FUSED_STATS)
            rows = [r for r in self.unresolved if r < nq]
            st[1], st[5] = len(rows), nq
            sid = _ints(a[isid], nq * k)
            for i in range(nq * k):
                sid[i] = 0
            for r in rows:
                sid[r * k] = _lib.SID_UNRESOLVED
        elif name == "cw_fused_predict_host":
            a[7][5] = nq
        elif isid is not None and nq and k:
            sid = _ints(a[isid], nq * k)
            for i in range(nq * k):
                sid[i] = FP32_MARK
        self.detail.append(d)
        return 0


@pytest.fixture
def fake(monkeypatch):
    lib = FakeLib()
    stream = types.SimpleNamespace(cuda_stream=0, synchronize=lambda: None)
    monkeypatch.setattr(_lib, "load", lambda: lib)
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **kw: stream)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **kw: self)

    def build_fused(ix):
        lib.calls.append(("_build_fused", None, None))
        lib.detail.append({})
        ix.hx = fused_operands()

    monkeypatch.setattr(DenseIndex, "_build_fused", build_fused)
    return lib


def fused_operands(smem_ok=True):
    return {"n_int": 10, "n_leaf": 5, "leaf_layout": _lib.H_F2, "smem_ok": smem_ok, "fi": _lib.CwFusedIndex(),
            "sent_off": torch.zeros(6, dtype=torch.int32), "sent_ids": torch.zeros(N_POS, dtype=torch.int32)}


def make_index(mode="fused", hx=True, nn=20000, n_pos=N_POS, shard=False):
    """A DenseIndex as __init__ leaves it (plus the fused operands when hx), on CPU tensors; chunks of 256 queries."""
    ix = DenseIndex.__new__(DenseIndex)
    ix.tree = types.SimpleNamespace(device=torch.device("cpu"), d=D)
    ix.ix = _lib.CwIndex()
    ix.nn, ix.ld, ix.n_pos, ix.max_len = nn, 128, n_pos, 4
    ix.pos_rec = torch.zeros((n_pos, 4), dtype=torch.int32)
    ix.pos_rec[:, 3] = torch.arange(n_pos - 1, -1, -1)
    ix.sentence_ids = np.arange(n_pos) if shard else None
    ix._ws = ix._sm = ix._hws = ix.hx = ix._rows = ix._pos_of_sid = ix._tag_cache = None
    if hx:
        ix.hx = fused_operands()
    ix.mode = mode
    ix.eps_scale, ix.audit_every, ix._audit_phase = DenseIndex.EPS_SCALE, DenseIndex.AUDIT_EVERY, 0
    ix.stats = {"queries": 0, "flagged": 0, "unresolved": 0, "cand_overflow": 0, "line_fail": 0, "list_overflow": 0,
                "candidates": 0, "audited": 0, "audit_mismatch": 0, "refined": 0, "rescored": 0}
    ix.SCORE_BUDGET_BYTES = 1   # chunk_queries() == 256
    return ix


def queries(nq):
    Q = torch.zeros((nq, D), dtype=torch.float32)
    Q[:, 0] = torch.arange(nq, dtype=torch.float32)
    return Q


def query_tags(nq):
    return torch.arange(100, 100 + nq, dtype=torch.int32)


SENT_TAGS = torch.ones(N_POS, dtype=torch.int32)


def tag_kw(nq, tagged):
    return dict(query_tags=query_tags(nq), sent_tags=SENT_TAGS, tag_version=1) if tagged else {}


# ---------------------------------------------------------------- the routing grid
K = (0, 1, 30, 31, 128)   # k = 0 asks for leaf scores on the device
S, F, P = "small", "fused", "fp32"
# the pipeline of an untagged device call with the fused operands built, nn >= TENSOR_MIN_NODES, per (mode, small) and
# nq, for each k of K
ROUTES = {
    ("fused", True): {0: (P, P, P, P, P), 1: (P, S, S, S, S), 32: (P, S, S, S, S), 33: (P, F, F, P, P), 1000: (P, F, F, P, P)},
    ("fused", False): {0: (P, P, P, P, P), 1: (P, F, F, P, P), 32: (P, F, F, P, P), 33: (P, F, F, P, P), 1000: (P, F, F, P, P)},
    ("fp32", True): {0: (P, P, P, P, P), 1: (P, S, S, S, S), 32: (P, S, S, S, S), 33: (P, P, P, P, P), 1000: (P, P, P, P, P)},
    ("fp32", False): {0: (P, P, P, P, P), 1: (P, P, P, P, P), 32: (P, P, P, P, P), 33: (P, P, P, P, P), 1000: (P, P, P, P, P)},
}
CHUNKS = {0: (), 1: (1,), 32: (32,), 33: (33,), 1000: (256, 256, 256, 232)}


def device_calls(route, nq, k, tagged):
    t = "_tagged" if tagged else ""
    if route == S:
        return [("cw_small_predict" + t, nq, k)]
    if route == F:
        return [("cw_fused_predict" + t, nq, k)]
    return [c for n in CHUNKS[nq] for c in (("cw_dense_node_scores", n, None), ("cw_dense_paths_topk" + t, n, k))]


def host_calls(route, nq, k):
    if route == S:
        return [("cw_small_predict_host", nq, k)]
    if route == F:
        return [("cw_fused_predict_host", nq, k)]
    return [("cw_predict_dense_host", n, k) for n in CHUNKS[nq]]


@pytest.mark.parametrize("nq", sorted(CHUNKS))
@pytest.mark.parametrize("small", [True, False])
@pytest.mark.parametrize("mode,per_call", [("fused", False), ("fp32", False), ("fused", True), ("fp32", True)])
def test_device_routing(fake, mode, per_call, small, nq):
    """Untagged device calls: the mode from the index or from the call, with and without the small-batch path."""
    for i, k in enumerate(K):
        ix = make_index(mode={"fused": "fp32", "fp32": "fused"}[mode] if per_call else mode)
        fake.calls.clear()
        sids, vals, leaf = ix.predict(queries(nq), k, want_leaf_scores=k == 0, mode=mode if per_call else None, small=small)
        route = ROUTES[(mode, small)][nq][i]
        assert fake.calls == device_calls(route, nq, k, False), (route, k)
        assert sids.shape == vals.shape == (nq, max(k, 1))
        assert (leaf is None) == (k != 0) and (leaf is None or leaf.shape == (nq, N_POS))
        assert ix._audit_phase == (route == F)


@pytest.mark.parametrize("nq", sorted(CHUNKS))
@pytest.mark.parametrize("small", [True, False])
@pytest.mark.parametrize("mode,per_call", [("fused", False), ("fp32", False), ("fused", True), ("fp32", True)])
def test_tagged_routing(fake, mode, per_call, small, nq):
    """Tag-filtered device calls take the same pipelines through their _tagged entry points; the leaf tags are derived
    once; an empty batch returns the padding."""
    for i, k in enumerate(K):
        ix = make_index(mode={"fused": "fp32", "fp32": "fused"}[mode] if per_call else mode)
        fake.calls.clear()
        kw = dict(mode=mode if per_call else None, small=small, query_tags=query_tags(nq), sent_tags=SENT_TAGS, tag_version=1)
        if k == 0:
            with pytest.raises(ValueError, match="leaf scores are not filtered by tags"):
                ix.predict(queries(nq), k, want_leaf_scores=True, **kw)
            with pytest.raises(ValueError, match="k must lie"):
                ix.predict(queries(nq), k, **kw)
            assert fake.calls == []
            continue
        sids, vals, leaf = ix.predict(queries(nq), k, **kw)
        route = ROUTES[(mode, small)][nq][i]
        want = [("cw_leaf_tags", None, None)] + device_calls(route, nq, k, True) if nq else []
        assert fake.calls == want, (route, k)
        assert leaf is None and sids.shape == vals.shape == (nq, k)
        if route == S:   # the small path writes nothing here: the prefilled padding shows
            assert bool((sids == -1).all()) and bool((vals == float("-inf")).all())


@pytest.mark.parametrize("nq", sorted(CHUNKS))
@pytest.mark.parametrize("mode", ["fused", "fp32"])
def test_host_routing(fake, mode, nq):
    """predict_host routes like a device call with the index's mode and the small-batch path allowed."""
    for i, k in enumerate(K):
        ix = make_index(mode=mode)
        fake.calls.clear()
        sid, val = ix.predict_host(queries(nq).numpy(), k)
        route = ROUTES[(mode, True)][nq][i]
        assert fake.calls == host_calls(route, nq, k), (route, k)
        assert sid.shape == val.shape == (nq, k)
        assert ix._audit_phase == (route == F)
        assert ix.stats["queries"] == (nq if route == F else 0)


# ---------------------------------------------------------------- edge cases
def test_fp32_chunks_get_their_rows_and_tags(fake):
    ix = make_index(mode="fp32")
    ix.predict(queries(1000), 10)
    assert [d["rows"][0] for d in fake.detail if "rows" in d] == [0, 256, 512, 768]
    fake.calls.clear()
    fake.detail.clear()
    ix.predict(queries(1000), 10, query_tags=query_tags(1000), sent_tags=SENT_TAGS, tag_version=1)
    assert [c[0] for c in fake.calls] == ["cw_leaf_tags"] + ["cw_dense_node_scores", "cw_dense_paths_topk_tagged"] * 4
    assert [d["rows"][0] for d in fake.detail if "rows" in d] == [0, 256, 512, 768]
    assert [d["tags"] for d in fake.detail if "tags" in d] == [tuple(range(100 + lo, 100 + min(1000, lo + 256)))
                                                                for lo in (0, 256, 512, 768)]


@pytest.mark.parametrize("tagged", [False, True])
def test_below_tensor_min_nodes_or_without_smem(fake, tagged):
    """A small index, or a path too long for the finish stage's shared memory, is answered by the FP32 chunks."""
    kw = tag_kw(33, tagged)
    pre = [("cw_leaf_tags", None, None)] if tagged else []
    want = pre + [("cw_dense_node_scores", 33, None), ("cw_dense_paths_topk" + ("_tagged" if tagged else ""), 33, 10)]
    ix = make_index(nn=DenseIndex.TENSOR_MIN_NODES - 1)
    ix.predict(queries(33), 10, **kw)
    assert fake.calls == want
    assert not ix.fused_ready(10)
    fake.calls.clear()
    ix = make_index()
    ix.hx["smem_ok"] = False
    ix.predict(queries(33), 10, **kw)
    assert fake.calls == want
    assert not ix.fused_ready(10)
    fake.calls.clear()
    ix = make_index(nn=DenseIndex.TENSOR_MIN_NODES)
    ix.predict(queries(33), 10, **kw)
    assert fake.calls == pre + [("cw_fused_predict" + ("_tagged" if tagged else ""), 33, 10)]
    assert ix.fused_ready(10)


@pytest.mark.parametrize("tagged", [False, True])
def test_fused_operands_built_on_first_fused_call(fake, tagged):
    """mode "fused" without the operands builds them first, even when the call then takes the small-batch path; an
    index with no sentences never builds them; host calls never do."""
    kw = tag_kw(1, tagged)
    t = "_tagged" if tagged else ""
    pre = [("cw_leaf_tags", None, None)] if tagged else []
    ix = make_index(mode="fused", hx=False)
    ix.predict(queries(1), 10, **kw)
    assert fake.calls == [("_build_fused", None, None)] + pre + [("cw_small_predict" + t, 1, 10)]
    fake.calls.clear()
    ix = make_index(mode="fp32", hx=False)
    ix.predict(queries(1), 10, mode="fused", small=False, **kw)
    assert fake.calls == [("_build_fused", None, None)] + pre + [("cw_fused_predict" + t, 1, 10)]
    fake.calls.clear()
    ix = make_index(mode="fp32", hx=False)
    ix.predict(queries(40), 10, **tag_kw(40, tagged))
    assert fake.calls == [("cw_dense_node_scores", 40, None), ("cw_dense_paths_topk" + t, 40, 10)]
    fake.calls.clear()
    ix = make_index(mode="fused", hx=False)
    ix.predict_host(queries(40).numpy(), 10)
    assert fake.calls == [("cw_predict_dense_host", 40, 10)] and ix.hx is None


def test_index_without_sentences(fake):
    """n_pos = 0: no operands are built; untagged calls run the FP32 chunks, tagged calls return the padding."""
    ix = make_index(mode="fused", hx=False, n_pos=0)
    ix.predict(queries(5), 10)
    assert fake.calls == [("cw_dense_node_scores", 5, None), ("cw_dense_paths_topk", 5, 10)]
    fake.calls.clear()
    s, v, _ = ix.predict(queries(5), 10, query_tags=query_tags(5), sent_tags=SENT_TAGS, tag_version=1)
    assert fake.calls == [] and bool((s == -1).all()) and bool((v == float("-inf")).all()) and s.shape == (5, 10)
    ix.predict_host(queries(5).numpy(), 10)
    assert fake.calls == [("cw_predict_dense_host", 5, 10)] and ix.hx is None


@pytest.mark.parametrize("tagged", [False, True])
def test_unresolved_rows_rerun_on_fp32(fake, tagged):
    """Rows the fused call leaves at SID_UNRESOLVED (statistics word 1) are answered again by the FP32 chunks with
    exactly those rows and, on tagged calls, their query tags; the other rows keep the fused answer."""
    fake.unresolved = (3, 40, 999)
    ix = make_index()
    kw = tag_kw(1000, tagged)
    t = "_tagged" if tagged else ""
    sids, _, _ = ix.predict(queries(1000), 10, **kw)
    pre = [("cw_leaf_tags", None, None)] if tagged else []
    assert fake.calls == pre + [("cw_fused_predict" + t, 1000, 10), ("cw_dense_node_scores", 3, None),
                                ("cw_dense_paths_topk" + t, 3, 10)]
    assert fake.detail[-2]["rows"] == (3, 40, 999)
    if tagged:
        assert fake.detail[-1]["tags"] == (103, 140, 1099)
    assert ix.stats["unresolved"] == 3 and ix.stats["queries"] == 1000
    first = sids[:, 0].tolist()
    assert [i for i, s in enumerate(first) if s == FP32_MARK] == [3, 40, 999]
    assert all(s == 0 for i, s in enumerate(first) if i not in (3, 40, 999))


@pytest.mark.parametrize("tagged", [False, True])
def test_audit_phase_steps_once_per_fused_call(fake, tagged):
    ix = make_index()
    kw = tag_kw(64, tagged)
    for _ in range(3):
        ix.predict(queries(64), 10, **kw)
    ix.predict(queries(64), 10, mode="fp32", **kw)
    ix.predict(queries(8), 10, **kw)
    assert [d["audit_phase"] for d in fake.detail if "audit_phase" in d] == [0, 1, 2]
    assert ix._audit_phase == 3
    ix.predict_host(queries(64).numpy(), 10)
    assert ix._audit_phase == 4


def test_errors(fake):
    """Every refusal, checked before any work is issued, in the order the checks are made."""
    Q, qt = queries(4), query_tags(4)
    tags = dict(query_tags=qt, sent_tags=SENT_TAGS, tag_version=1)
    shard = make_index(shard=True)
    with pytest.raises(ValueError, match="sentence shard"):
        shard.predict(Q, 0, want_leaf_scores=True, mode="bogus")
    with pytest.raises(ValueError, match="mode must be"):
        make_index().predict(Q, 10, mode="bogus")
    with pytest.raises(ValueError, match="leaf scores are not filtered by tags"):
        shard.predict(Q, 10, want_leaf_scores=True, mode="bogus", **tags)
    with pytest.raises(ValueError, match="sentence shard"):
        shard.predict(Q, 0, mode="bogus", **tags)
    with pytest.raises(ValueError, match="mode must be"):
        make_index().predict(Q, 0, mode="bogus", **tags)
    for k in (0, _lib.MAX_K + 1):
        with pytest.raises(ValueError, match="k must lie"):
            make_index().predict(Q, k, **tags)
    with pytest.raises(ValueError, match="k must lie"):
        make_index(n_pos=0).predict(queries(0), 0, query_tags=query_tags(0), sent_tags=SENT_TAGS, tag_version=1)
    assert fake.calls == []
    s, _, _ = shard.predict(Q, 10)   # a shard answers untagged calls without leaf scores
    assert s.shape == (4, 10) and fake.calls == [("cw_small_predict", 4, 10)]


def test_one_query_paths_create_no_tensors(fake, monkeypatch):
    """predict_one and predict_host's small branch, once the buffers exist, allocate no torch tensors."""
    ix = make_index()
    q = queries(1).numpy()[0]
    Qh, out_s, out_v = queries(3), torch.empty((3, 10), dtype=torch.int32), torch.empty((3, 10))
    ix.predict_one(q, 10)
    for name in ("empty", "zeros", "full", "tensor", "as_tensor", "from_numpy"):
        monkeypatch.setattr(torch, name, lambda *a, **kw: pytest.fail("a tensor was created"))
    fake.calls.clear()
    assert len(ix.predict_one(q, 10)) == 10
    ix.predict_host(Qh, 10, out_s, out_v)
    assert fake.calls == [("cw_small_predict_host", 1, 10), ("cw_small_predict_host", 3, 10)]


def test_fused_ready_reads_mode_hx_nn_and_k_only():
    ix = DenseIndex.__new__(DenseIndex)
    ix.mode, ix.nn, ix.hx = "fused", DenseIndex.TENSOR_MIN_NODES, {"smem_ok": True}
    assert [ix.fused_ready(k) for k in (0, 1, _lib.FUSED_MAX_K, _lib.FUSED_MAX_K + 1)] == [False, True, True, False]
    ix.hx = None
    assert not ix.fused_ready(1)
