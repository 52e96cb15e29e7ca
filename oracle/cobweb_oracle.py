"""ctypes front-end of the CPU oracle (oracle/cobweb_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs -- never by the product package.  The class mirrors the
slice of the reference API the parity tests need: ifit / categorize / dense scores, each
restating the reference function named in the C source.
"""
import ctypes as C
import math
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libcobweb_oracle.so")
_lib = None

OP_NAMES = ["best", "new", "merge", "split", "leaf", "fringe"]


def build(force=False):
    src = os.path.join(_HERE, "cobweb_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE, "-B", "libcobweb_oracle.so"])
    return _SO


def default_prior_var():
    """1 / (2 * e * pi) evaluated as the reference does (CobwebTorchTree.py:35-40):
    python-double 2*e times the fp32 pi tensor, reciprocal in fp32."""
    return float(np.float32(1.0) / (np.float32(2 * math.e) * np.float32(math.pi)))


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        fp, ip, lp = C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_long)
        L.co_create.restype = C.c_void_p
        L.co_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
        L.co_free.argtypes = [C.c_void_p]
        L.co_ifit.restype = C.c_long
        L.co_ifit.argtypes = [C.c_void_p, fp, C.c_long, ip, C.POINTER(C.c_byte), lp, C.c_long, C.c_int]
        L.co_ifit_guided.restype = C.c_long
        L.co_ifit_guided.argtypes = [C.c_void_p, fp, C.c_long, ip, C.POINTER(C.c_byte), ip, ip, C.c_long, fp,
                                     C.POINTER(C.c_double), C.c_int]
        for f in ("co_num_slots", "co_root", "co_num_nodes"):
            getattr(L, f).restype = C.c_int
            getattr(L, f).argtypes = [C.c_void_p]
        L.co_score_calls.restype = C.c_long
        L.co_score_calls.argtypes = [C.c_void_p]
        L.co_bfs.restype = C.c_int
        L.co_bfs.argtypes = [C.c_void_p, ip, ip, fp, ip, ip, ip]
        L.co_get_rows.argtypes = [C.c_void_p, ip, C.c_int, fp, fp]
        L.co_load.argtypes = [C.c_void_p, C.c_int, ip, fp, ip, fp, fp]
        L.co_log_prob.restype = C.c_float
        L.co_log_prob.argtypes = [C.c_void_p, C.c_int, fp]
        L.co_categorize.argtypes = [C.c_void_p, fp, C.c_long, C.c_int, C.c_long, C.c_int, C.c_int, ip, ip, ip, lp]
        L.co_index_stats.argtypes = [C.c_void_p, ip, C.c_int, fp, fp, fp]
        L.co_dense_scores.argtypes = [C.c_int, C.c_long, fp, C.c_int, fp, fp, fp, C.c_long, C.c_int, ip, fp, fp, fp]
        L.co_leaf_scores.argtypes = [C.c_long, C.c_int, fp, C.c_long, C.c_int, ip, fp, fp]
        L.co_dense_scores_fast.argtypes = [C.c_int, C.c_long, fp, C.c_int, fp, fp, fp, fp]
        L.co_topk.argtypes = [fp, C.c_long, C.c_int, ip, fp]
        L.co_fp32_operands.argtypes = [C.c_int, C.c_int, fp, fp, fp, fp]
        L.co_fp32_node_scores.argtypes = [C.c_int, C.c_long, fp, C.c_int, fp, fp, fp, fp]
        L.co_fmaf_array.argtypes = [C.c_long, fp, fp, fp, fp]
        L.co_logf.restype = C.c_float
        L.co_logf.argtypes = [C.c_float]
        L.co_sum_public.restype = C.c_float
        L.co_sum_public.argtypes = [C.c_int, fp]
        L.co_compute_score.restype = C.c_float
        L.co_compute_score.argtypes = [C.c_void_p, fp, fp, fp, fp]
        _lib = L
    return _lib


def set_threads(n):
    """OpenMP threads of the dense baseline loops; returns the count in effect (bench.py: all host threads)."""
    L = lib()
    L.co_set_threads.restype = C.c_int
    L.co_set_threads.argtypes = [C.c_int]
    return int(L.co_set_threads(int(n)))


def _f(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _i(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _l(a):
    return a.ctypes.data_as(C.POINTER(C.c_long))


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


class OracleTree:
    """Restates CobwebTorchTree (+ the wrapper's sentence bookkeeping and dense index)."""

    def __init__(self, d, prior_var=None, use_info=True, use_kl=True, acuity_cutoff=False, greedy=False):
        self.d = int(d)
        self.prior_var = default_prior_var() if prior_var is None else float(prior_var)
        self._h = lib().co_create(self.d, self.prior_var, int(use_info), int(use_kl), int(acuity_cutoff))
        if greedy:  # COBWEB_GREEDY_MODE = True (src/utils/constants.py)
            lib().co_set_greedy.argtypes = [C.c_void_p, C.c_int]
            lib().co_set_greedy(self._h, 1)
        self.n_sentences = 0
        self.leaf_of_sentence = np.zeros(0, dtype=np.int32)  # node slot per sentence id

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.co_free(self._h)
            self._h = None

    # -- ifit ---------------------------------------------------------------------------
    def ifit(self, X, tag_sentences=True, trace=False):
        """Insert rows of X in order. Returns leaf slots [n] (and per-insert op traces)."""
        X = _f32(np.atleast_2d(X))
        n = X.shape[0]
        leaves = np.empty(n, dtype=np.int32)
        if trace:
            cap = 64 * n + 64
            tr = np.zeros(cap, dtype=np.int8)
            off = np.zeros(n + 1, dtype=np.int64)
            nt = lib().co_ifit(self._h, _f(X), n, _i(leaves), tr.ctypes.data_as(C.POINTER(C.c_byte)), _l(off), cap,
                               int(tag_sentences))
            assert nt <= cap
        else:
            lib().co_ifit(self._h, _f(X), n, _i(leaves), None, None, 0, int(tag_sentences))
        if tag_sentences:
            self.leaf_of_sentence = np.concatenate([self.leaf_of_sentence, leaves])
            self.n_sentences += n
        return (leaves, tr[:nt], off) if trace else leaves

    def ifit_guided(self, X, ops, b1, b2, tag_sentences=True):
        """Replay recorded internal-node decisions (golden dec_* arrays; ops = the 0..3 codes
        only).  Returns (leaves, pus [ndec,4], dict(rank_disagree, op_disagree, rank_margin,
        op_margin, used))."""
        X = _f32(np.atleast_2d(X))
        n = X.shape[0]
        ops = np.ascontiguousarray(ops, np.int8)
        b1 = np.ascontiguousarray(b1, np.int32)
        b2 = np.ascontiguousarray(b2, np.int32)
        leaves = np.empty(n, dtype=np.int32)
        pus = np.full((len(ops), 4), np.nan, np.float32)
        stats = np.zeros(4, np.float64)
        used = lib().co_ifit_guided(self._h, _f(X), n, _i(leaves), ops.ctypes.data_as(C.POINTER(C.c_byte)), _i(b1),
                                    _i(b2), len(ops), _f(pus), stats.ctypes.data_as(C.POINTER(C.c_double)),
                                    int(tag_sentences))
        if tag_sentences:
            self.leaf_of_sentence = np.concatenate([self.leaf_of_sentence, leaves])
            self.n_sentences += n
        return leaves, pus, dict(rank_disagree=int(stats[0]), op_disagree=int(stats[1]), rank_margin=stats[2],
                                 op_margin=stats[3], used=int(used))

    @property
    def score_calls(self):
        return lib().co_score_calls(self._h)

    # -- structure ----------------------------------------------------------------------
    def bfs(self):
        """dict(order=node slots in BFS order, parent (BFS idx), count, nchild, nsent, depth)."""
        ns = lib().co_num_slots(self._h)
        order = np.empty(ns, np.int32); parent = np.empty(ns, np.int32); count = np.empty(ns, np.float32)
        nchild = np.empty(ns, np.int32); nsent = np.empty(ns, np.int32); depth = np.empty(ns, np.int32)
        n = lib().co_bfs(self._h, _i(order), _i(parent), _f(count), _i(nchild), _i(nsent), _i(depth))
        return dict(order=order[:n], parent=parent[:n], count=count[:n], nchild=nchild[:n], nsent=nsent[:n],
                    depth=depth[:n])

    def rows(self, slots):
        slots = np.ascontiguousarray(slots, dtype=np.int32)
        mean = np.empty((len(slots), self.d), np.float32)
        m2 = np.empty((len(slots), self.d), np.float32)
        lib().co_get_rows(self._h, _i(slots), len(slots), _f(mean), _f(m2))
        return mean, m2

    def load(self, parent, count, nsent, mean, m2):
        """Replace the tree (nodes topologically ordered, siblings in child order)."""
        parent = np.ascontiguousarray(parent, np.int32)
        nsent = np.ascontiguousarray(nsent, np.int32)
        lib().co_load(self._h, len(parent), _i(parent), _f(_f32(count)), _i(nsent), _f(_f32(mean)), _f(_f32(m2)))

    # -- best-first ---------------------------------------------------------------------
    def log_prob(self, slot, x):
        return lib().co_log_prob(self._h, int(slot), _f(_f32(x)))

    def categorize(self, Q, k=0, max_nodes=None, greedy=False, use_best=True):
        """k > 0: (leaves [nq,k] slots (-1 padded), nfound, best, lp_calls); k == 0: retrieve_k=None."""
        Q = _f32(np.atleast_2d(Q))
        nq = Q.shape[0]
        leaves = np.full((nq, max(k, 1)), -1, np.int32)
        nfound = np.zeros(nq, np.int32)
        best = np.zeros(nq, np.int32)
        calls = np.zeros(nq, np.int64)
        mn = (1 << 62) if max_nodes is None or max_nodes == float("inf") else int(max_nodes)
        lib().co_categorize(self._h, _f(Q), nq, int(k), mn, int(greedy), int(use_best), _i(leaves), _i(nfound),
                            _i(best), _l(calls))
        return leaves, nfound, best, calls

    # -- dense index --------------------------------------------------------------------
    def build_index(self, level_weights=None):
        """build_prediction_index (CobwebWrapper.py:91-208): BFS node matrices + per-sentence
        root->leaf paths with weights level_w[depth]/path_len (fp32)."""
        b = self.bfs()
        nn = len(b["order"])
        means = np.empty((nn, self.d), np.float32); vars_ = np.empty((nn, self.d), np.float32)
        sumlog = np.empty(nn, np.float32)
        lib().co_index_stats(self._h, _i(b["order"]), nn, _f(means), _f(vars_), _f(sumlog))
        pos = np.full(lib().co_num_slots(self._h), -1, np.int32)
        pos[b["order"]] = np.arange(nn, dtype=np.int32)
        maxlen = int(b["depth"].max()) + 1
        L = self.n_sentences
        path_idx = np.full((L, maxlen), -1, np.int32)
        path_w = np.zeros((L, maxlen), np.float32)
        lw = [1.0] * 6 if level_weights is None else list(level_weights)
        leaf_b = pos[self.leaf_of_sentence]
        for sid in range(L):
            p, node = [], int(leaf_b[sid])
            while node >= 0:
                p.append(node)
                node = int(b["parent"][node])
            p.reverse()
            for dep, nb in enumerate(p):
                w = lw[dep] if dep < len(lw) else 1.0
                path_idx[sid, dep] = nb
                path_w[sid, dep] = np.float32(w / len(p))
        self.index = dict(bfs=b, means=means, vars=vars_, sumlog=sumlog, path_idx=path_idx, path_w=path_w,
                          leaf_b=leaf_b)
        return self.index

    def dense_scores(self, Q, fast=False):
        """(node_scores [nq, Nn] in BFS order, leaf_scores [nq, L] by sentence id)."""
        ix = self.index
        Q = _f32(np.atleast_2d(Q))
        nq, nn, L = Q.shape[0], ix["means"].shape[0], ix["path_idx"].shape[0]
        ns = np.empty((nq, nn), np.float32)
        ls = np.empty((nq, L), np.float32)
        if fast:
            lib().co_dense_scores_fast(self.d, nq, _f(Q), nn, _f(ix["means"]), _f(ix["vars"]), _f(ix["sumlog"]), _f(ns))
            return ns, None
        lib().co_dense_scores(self.d, nq, _f(Q), nn, _f(ix["means"]), _f(ix["vars"]), _f(ix["sumlog"]), L,
                              ix["path_idx"].shape[1], _i(ix["path_idx"]), _f(ix["path_w"]), _f(ns), _f(ls))
        return ns, ls

    def fp32_operands(self):
        """(r, mb) [nn, D] of the engine's FP32 form in BFS order: r = 1 / sqrt(var), mb = -(mean * r)."""
        ix = self.index
        r, mb = np.empty_like(ix["vars"]), np.empty_like(ix["vars"])
        lib().co_fp32_operands(self.d, r.shape[0], _f(ix["means"]), _f(ix["vars"]), _f(r), _f(mb))
        return r, mb

    def fp32_scores(self, Q):
        """(node_scores [nq, Nn], leaf_scores [nq, L]) of the engine's FP32 form bit for bit: the node score chain
        u = fma(x, r, mb), acc = fma(u, u, acc) over d ascending, -0.5 * (sumlog + acc); then the path product."""
        ix = self.index
        Q = _f32(np.atleast_2d(Q))
        nq, nn, L = Q.shape[0], ix["means"].shape[0], ix["path_idx"].shape[0]
        ns = np.empty((nq, nn), np.float32)
        lib().co_fp32_node_scores(self.d, nq, _f(Q), nn, _f(ix["means"]), _f(ix["vars"]), _f(ix["sumlog"]), _f(ns))
        return ns, leaf_scores(ns, ix["path_idx"], ix["path_w"])


def fmaf(a, b, c):
    """Elementwise fmaf(a, b, c) in binary32, the fused multiply-add of fp32_scores."""
    a, b, c = np.broadcast_arrays(_f32(a), _f32(b), _f32(c))
    a, b, c = _f32(a), _f32(b), _f32(c)
    out = np.empty(a.shape, np.float32)
    lib().co_fmaf_array(a.size, _f(a), _f(b), _f(c), _f(out))
    return out


def leaf_scores(node_scores, path_idx, path_w):
    """Sparse path product of the reference (sequential binary32 FMA, root first)."""
    ns = _f32(np.atleast_2d(node_scores))
    path_idx = np.ascontiguousarray(path_idx, np.int32)
    path_w = _f32(path_w)
    out = np.empty((ns.shape[0], path_idx.shape[0]), np.float32)
    lib().co_leaf_scores(ns.shape[0], ns.shape[1], _f(ns), path_idx.shape[0], path_idx.shape[1], _i(path_idx),
                         _f(path_w), _f(out))
    return out


def topk(scores, k):
    scores = _f32(scores)
    idx = np.empty(k, np.int32)
    val = np.empty(k, np.float32)
    lib().co_topk(_f(scores), len(scores), k, _i(idx), _f(val))
    return idx, val
