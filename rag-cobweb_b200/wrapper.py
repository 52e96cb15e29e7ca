"""CobwebWrapper with the reference's signatures (src/cobweb/CobwebWrapper.py), backed by the
device node store and kernels.

Reference surface kept: __init__(corpus, corpus_embeddings, encode_func) :13, add_sentences :52,
build_prediction_index :91, cobweb_predict_indexed :210, cobweb_rank_scores :267,
set_level_weights :335, set_weight_schedule :348, get_level_weights :410,
get_weight_schedule_info :414, force_rebuild_index :422, cobweb_predict_fast :428,
cobweb_predict :435, print_tree :463, dump_json :484, load_json :501, __len__ :557, attributes
sentences / sentence_to_node / tree / device / max_init_search.  visualize_subtrees (graphviz
rendering) is out of scope and raises NotImplementedError.
Additive: predict_fast_batch / predict_batch / rank_scores_batch for query batches; set_sentence_tags /
get_sentence_tags and predict_fast_batch(..., query_tags=) for tag-filtered retrieval.

Deliberate differences (DESIGN.md "Tie-breaking"): no 1e-6*randn noise and no in-leaf
random.shuffle -- exact ties are broken by ascending sentence id.
"""
import base64
import ctypes as C
import json
import os

import numpy as np
import torch

from . import _lib, topology, topology_device
from .tree import CobwebNode, CobwebTorchTree


class DenseIndex:
    """Device-resident prediction index (build_prediction_index, CobwebWrapper.py:91-208)."""

    SCORE_BUDGET_BYTES = 24 << 30  # node-score scratch per query chunk (180 GB of HBM: one chunk for 16k queries x 313k internal rows)
    # How the top-k of a query batch is computed (ids and scores are the same bit for bit in both modes):
    #   "fp32"   every (query, node) score on the FP32 pipe, (x*r + mb)^2 per triple (cw_dense.cu), path product and
    #            top-k over the [nodes, queries] score matrix: the form that DEFINES the result;
    #   "fused"  tcgen05 fp16 pipeline (cw_half.cu): internal rows with path-summed split operands (hi + lo, three
    #            products), whose scores are the ancestor sums; leaf rows with ONE fp16 product as a filter with a derived error bound;
    #            the survivors are re-scored with the FP32 form's exact arithmetic; queries the device cannot decide
    #            (and an always-on audit sample) go through the exact small-batch path.
    # Batches of up to SMALL_Q queries take the exact small-batch path in every mode (one query: HBM-bound).
    MODES = ("fp32", "fused")
    FUSED_CAP = 768               # candidate slots per query of the filtering epilogue
    TENSOR_MIN_NODES = 16384      # smaller indexes are answered on the FP32 pipe (launch-bound there; same result)
    EPS_SCALE = 2.0 ** -18        # |fp16x3 ancestor sums - fp32| relative to the operand magnitudes (cw_half.cu eps_of)
    AUDIT_EVERY = 2048            # one query in AUDIT_EVERY is answered again by the exact path and compared (0 = off)
    PAIR_BUDGET_BYTES = 4 << 30   # pair-scoring scratch per query chunk (row lists, their scores, the level maps)

    def __init__(self, tree, leaf_of_sentence, level_weights=None, sentence_ids=None):
        """leaf_of_sentence[i] = leaf node id of sentence i.  sentence_ids (optional, sorted global
        ids) restricts the index to a shard of the sentences: only the nodes on their root->leaf
        paths are indexed and scored, returned ids stay global (store-sharded mode, SURVEY 8e)."""
        L = _lib.load()
        self.tree = tree
        dev = tree.device
        # topology on the device (topology_device.py mirrors the numpy statements in topology.py): the store's arrays
        # are not copied to the host, so the index is rebuilt after add_sentences in milliseconds (SURVEY 8f-1)
        st = tree.store
        h = st.header()
        n_used, root = int(h[_lib.HDR_N_USED]), int(h[_lib.HDR_ROOT])
        order, parent_b, depth = topology_device.bfs_order(root, st.child_off, st.child_cnt, st.child_pool)
        leaf_np = np.asarray(leaf_of_sentence)
        if len(leaf_np) and int(leaf_np.min()) < 0:
            raise ValueError("a sentence has no leaf (leaf_of_sentence < 0): the sentence list and the tree do not match")
        self.sentence_ids = None
        if sentence_ids is not None:
            # a shard of the sentences: only the nodes on their paths are indexed (host statement; built once per shard)
            self.sentence_ids = np.asarray(sentence_ids, np.int64)
            leaf_np = leaf_np[self.sentence_ids]
            o, p_, d_ = topology.restrict_to_paths(order.cpu().numpy(), parent_b.cpu().numpy(), depth.cpu().numpy(), leaf_np, n_used)
            order, parent_b, depth = (torch.as_tensor(a_, device=dev) for a_ in (o, p_, d_))
        leaf_dev = torch.as_tensor(leaf_np.astype(np.int64), device=dev)
        self._topo = (order, parent_b, depth, leaf_dev, level_weights, n_used)
        self.nn = int(order.numel())
        self.max_depth = int(depth.max()) + 1
        d = tree.d
        self.n_ntiles = (self.nn + _lib.TILE_N - 1) // _lib.TILE_N
        self.n_ktiles = (d + _lib.TILE_K - 1) // _lib.TILE_K
        self.ld = self.n_ntiles * _lib.TILE_N  # rows of the node-major score matrix
        tile_elems = self.n_ntiles * self.n_ktiles * _lib.TILE_K * _lib.TILE_N
        self.R = torch.empty(tile_elems, dtype=torch.float32, device=dev)
        self.MB = torch.empty(tile_elems, dtype=torch.float32, device=dev)
        self.sumlog = torch.zeros(self.ld, dtype=torch.float32, device=dev)
        self.order = order.to(torch.int32)
        self.n_pos = int(leaf_dev.numel())
        ix = _lib.CwIndex()
        ix.D, ix.nn, ix.n_ntiles, ix.n_ktiles = d, self.nn, self.n_ntiles, self.n_ktiles
        ix.R, ix.MB, ix.sumlog = self.R.data_ptr(), self.MB.data_ptr(), self.sumlog.data_ptr()
        if self.n_pos:
            p = topology_device.sentence_paths(order, parent_b, depth, leaf_dev, level_weights, n_slots=n_used)
            self.max_len = p["max_len"]
            self.path_idx = p["path_idx"]  # [n_pos, max_len]
            self._level_w_host = np.asarray(p["level_w"], np.float64)
            self.level_w = torch.as_tensor(self._level_w_host, dtype=torch.float64, device=dev)
            self._pos_leaf_row = p["pos_leaf_row"]   # ascending: positions are sorted by leaf row
            self._path_lens = np.asarray(p["path_lens"], np.int64)
            self.pos_rec = p["pos_rec"]  # [n_pos, 4]
            if self.sentence_ids is not None:  # local position ids -> global ids
                self.pos_rec[:, 3] = torch.as_tensor(self.sentence_ids, device=dev)[self.pos_rec[:, 3].long()].to(torch.int32)
            ix.n_pos, ix.max_len = self.n_pos, self.max_len
            ix.path_idx, ix.pos_rec, ix.level_w = self.path_idx.data_ptr(), self.pos_rec.data_ptr(), self.level_w.data_ptr()
        self.ix = ix
        _lib.check(L.cw_index_build(tree.store.struct(), self.order.data_ptr(), self.nn, C.byref(ix), _lib.stream_ptr()),
                   "cw_index_build")
        self._ws = None
        self._sm = None
        self._hws = None
        self.hx = None
        self._rows = None
        self._pos_of_sid = None
        self._tag_cache = None
        self.mode = "fp32"
        self.eps_scale = self.EPS_SCALE
        self.audit_every = self.AUDIT_EVERY
        self._audit_phase = 0
        self.stats = {"queries": 0, "flagged": 0, "unresolved": 0, "cand_overflow": 0, "line_fail": 0, "list_overflow": 0,
                      "candidates": 0, "audited": 0, "audit_mismatch": 0, "refined": 0, "rescored": 0}

    # ------------------------------------------------------------------ modes
    def set_mode(self, mode):
        """Select how predict / predict_host compute the top-k; "fused" builds its operand sets on first use."""
        if mode not in self.MODES:
            raise ValueError(f"mode must be one of {self.MODES}")
        if mode == "fused":
            if not self.n_pos:
                return self
            if self.hx is None:
                self._build_fused()
        self.mode = mode
        return self

    def fused_ready(self, k):
        """True if a top-k request is served by the fused pipeline (else: the FP32 form)."""
        return self._route(1, k, self.mode, small=False) == "fused"

    def _route(self, nq, k, mode, small=True, leaf=False):
        """The pipeline of a call for the top-k of nq queries: "small" (the exact small-batch path), "fused" or "fp32".
        Every pipeline returns the same ids and scores; this rule only decides which is fastest."""
        if small and not leaf and 1 <= k <= _lib.MAX_K and 0 < nq <= _lib.SMALL_Q and self.n_pos:
            return "small"
        if (mode == "fused" and not leaf and self.hx is not None and 1 <= k <= _lib.FUSED_MAX_K and
                self.nn >= self.TENSOR_MIN_NODES and self.hx["smem_ok"] and nq > 0):
            return "fused"
        return "fp32"

    def _build_fused(self):
        """Operands of the fused mode: fp16 operand sets for the internal rows (hi + lo) and the leaf rows (hi), per-leaf
        records, row-major {r, mb} rows for the exact arithmetic, the constants of eps (topology.fused_layout)."""
        L, dev, d = _lib.load(), self.tree.device, self.tree.d
        order, parent_b, depth, leaf_dev, level_weights, n_used = self._topo
        F = topology_device.fused_layout(order, parent_b, depth, leaf_dev, level_weights, n_slots=n_used,
                                         sentence_ids=None if self.sentence_ids is None else torch.as_tensor(self.sentence_ids, device=dev),
                                         tile=_lib.H_TILE)
        st, store = _lib.stream_ptr(), self.tree.store.struct()
        n_int, n_leaf = int(F["int_rows"].numel()), int(F["leaf_rows"].numel())
        hx = {"F": F, "n_int": n_int, "n_leaf": n_leaf, "n_s": int(F["n_sample_tiles"])}
        hx["leaf_rows"] = F["leaf_rows"]
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        iso = L.cw_h_rows_isotropic(store, self.order.data_ptr(), hx["leaf_rows"].data_ptr(), n_leaf, flag.data_ptr(), st)
        if iso < 0:
            _lib.check(iso, "cw_h_rows_isotropic")
        hx["leaf_layout"] = _lib.H_F1 if iso == 1 else _lib.H_F2

        def hset(rows_t, n_rows, layout, nprod, internal, leaf):
            hs = _lib.CwHSet()
            hs.n_rows, hs.n_ntiles = n_rows, (n_rows + _lib.H_TILE - 1) // _lib.H_TILE
            hs.n_stages, hs.nprod, hs.layout = L.cw_h_stages(d, layout, nprod), nprod, layout
            B = torch.empty(L.cw_h_b_bytes(n_rows, d, layout, nprod), dtype=torch.uint8, device=dev)
            rc = torch.empty(hs.n_ntiles * _lib.H_TILE * (2 if nprod == 3 else 8), dtype=torch.float32, device=dev)
            hs.B, hs.rc = B.data_ptr(), rc.data_ptr()
            ptrs = [t.data_ptr() if t is not None else None for t in internal + leaf]
            _lib.check(L.cw_h_set_build(store, self.order.data_ptr(), rows_t.data_ptr(), self.sumlog.data_ptr(), C.byref(hs),
                                        *ptrs, st), "cw_h_set_build")
            return hs, B, rc

        fi = _lib.CwFusedIndex()
        fi.ix = self.ix
        fi.n_int, fi.n_leaf, fi.n_sample_tiles = n_int, n_leaf, hx["n_s"]
        if n_int:
            hx["int_rows"] = F["int_rows"]
            # internal rows: operands summed along the path with the level weights (their scores are the ancestor sums)
            fi.internal, hx["B_int"], hx["rc_int"] = hset(hx["int_rows"], n_int, _lib.H_F2, 3, [F["int_parent"], F["int_w"]],
                                                          [None] * 4)
            hx["int_parent"], hx["int_w"], hx["level_off"] = F["int_parent"], F["int_w"], F["level_off"]
            fi.int_parent, fi.int_w, fi.level_off = hx["int_parent"].data_ptr(), hx["int_w"].data_ptr(), hx["level_off"].data_ptr()
            fi.n_levels = int(F["level_off"].numel()) - 1
        hx["leaf_aux"] = [F["leaf_w"], F["leaf_inv_len"], F["leaf_parent"], F["leaf_len"]]
        fi.leaves, hx["B_leaf"], hx["rc_leaf"] = hset(hx["leaf_rows"], n_leaf, hx["leaf_layout"], 1, [None] * 2, hx["leaf_aux"])
        hx["leaf_pos"] = torch.searchsorted(self._pos_leaf_row, F["leaf_rows"].to(torch.int64)).to(torch.int32)
        hx["sent_off"], hx["sent_ids"] = F["sent_off"], F["sent_ids"]
        fi.leaf_row_b, fi.leaf_pos = hx["leaf_rows"].data_ptr(), hx["leaf_pos"].data_ptr()
        fi.sent_off, fi.sent_ids = hx["sent_off"].data_ptr(), hx["sent_ids"].data_ptr()
        hx["rows"] = self.rows()
        fi.rows = hx["rows"].data_ptr()
        # constants of eps: hmax = max_b sum_d mean^2/var (= sum_d mb^2), lmax = max_b |sumlog|,
        # wfac = max over path lengths of sum_j |level_w[j]| / len; e1max = largest rounding-error coefficient of a leaf
        hmax = 0.0
        for lo in range(0, self.nn, 65536):
            hmax = max(hmax, float(hx["rows"][lo:lo + 65536, :, 1].double().square().sum(1).max()))
        fi.hmax = hmax * (1.0 + 1e-6) + 1e-6
        fi.lmax = float(self.sumlog[: self.nn].abs().max())
        cw = np.cumsum(np.abs(self._level_w_host))
        fi.wfac = float(max(1.0, (cw[self._path_lens - 1] / self._path_lens).max()))
        fi.e1max = float(hx["rc_leaf"].view(-1, 8)[:n_leaf, 4].max())
        fi.eps_scale = self.eps_scale
        fi.prior_var = float(self.tree.prior_var.item())
        torch.cuda.current_stream().synchronize()
        hx["fi"] = fi
        hx["smem_ok"] = self.max_len <= 512
        self.hx = hx

    def rows(self):
        """Row-major {r, mb} rows [nn, D, 2] (cw_index_rows_build), built on first use: the operands of the exact
        arithmetic in the fused finish stage and in pair scoring."""
        if self._rows is None:
            rows = torch.empty((self.nn, self.tree.d, 2), dtype=torch.float32, device=self.tree.device)
            _lib.check(_lib.load().cw_index_rows_build(self.tree.store.struct(), self.order.data_ptr(), self.nn,
                                                       rows.data_ptr(), _lib.stream_ptr()), "cw_index_rows_build")
            self._rows = rows
        return self._rows

    def pos_of_sid(self):
        """[n_pos] int32: position (row of path_idx) of each sentence id, the inverse of pos_rec[:, 3]; built on first use."""
        if self._pos_of_sid is None:
            p = torch.full((self.n_pos,), -1, dtype=torch.int32, device=self.tree.device)
            p[self.pos_rec[:, 3].long()] = torch.arange(self.n_pos, dtype=torch.int32, device=p.device)
            self._pos_of_sid = p
        return self._pos_of_sid

    def tag_arrays(self, sent_tags, version):
        """What the tagged kernels read of the sentences' tag words sent_tags [n sentences] int32, derived once per tag
        version: "pos" [n_pos] the tag of each position's sentence and, once the fused operands exist, "leaf" [n_leaf] the
        OR of the tags of each fused leaf row's sentences (cw_leaf_tags)."""
        c = self._tag_cache
        if c is None or c["version"] != version:
            c = self._tag_cache = {"version": version, "sent": sent_tags, "leaf": None,
                                   "pos": sent_tags[self.pos_rec[:, 3].long()].contiguous()}
        if c["leaf"] is None and self.hx is not None:
            hx = self.hx
            leaf = torch.empty(hx["n_leaf"], dtype=torch.int32, device=sent_tags.device)
            _lib.check(_lib.load().cw_leaf_tags(hx["sent_off"].data_ptr(), hx["sent_ids"].data_ptr(), hx["n_leaf"],
                                                sent_tags.data_ptr(), leaf.data_ptr(), _lib.stream_ptr()), "cw_leaf_tags")
            c["leaf"] = leaf
        return c

    def bytes(self):
        b = (self.R.numel() + self.MB.numel() + self.sumlog.numel()) * 4
        if self._rows is not None:
            b += self._rows.numel() * 4
        if self.hx is not None:
            b += sum(self.hx[n].numel() * self.hx[n].element_size() for n in ("B_int", "rc_int", "B_leaf", "rc_leaf")
                     if n in self.hx)
        return b

    # ------------------------------------------------------------------ work buffers
    def chunk_queries(self):
        return int(max(256, min(65535, self.SCORE_BUDGET_BYTES // (self.ld * 4)) // 256 * 256))  # whole 256-query tiles

    def workspace(self, nq, k):
        """Device work buffers of the FP32 form for chunks of up to nq queries and top-k up to k (grown on demand)."""
        ws = self._ws
        if ws and ws["cap_q"] >= nq and ws["cap_k"] >= k:
            return ws
        L, dev = _lib.load(), self.tree.device
        nq = max(nq, ws["cap_q"]) if ws else nq
        k = max(k, ws["cap_k"], 1) if ws else max(k, 1)
        self._ws = ws = None
        ldq = int(L.cw_score_ldq(nq))
        ws = dict(
            cap_q=nq, cap_k=k, ldq=ldq,
            q=torch.empty((nq, self.tree.d), dtype=torch.float32, device=dev),
            xt=torch.empty(L.cw_xt_floats(nq, self.tree.d), dtype=torch.float32, device=dev),  # k-major query tiles
            scores=torch.empty((self.ld, ldq), dtype=torch.float32, device=dev),  # node-major
            sid=torch.empty((nq, k), dtype=torch.int32, device=dev),
            val=torch.empty((nq, k), dtype=torch.float32, device=dev),
            scratch=torch.empty(max(1, nq * L.cw_topk_chunks(max(self.n_pos, 1)) * k * 2), dtype=torch.int32, device=dev),
        )
        w = ws["w"] = _lib.CwDenseWork()
        w.Q_dev, w.xt_scratch, w.node_scores, w.ldq = ws["q"].data_ptr(), ws["xt"].data_ptr(), ws["scores"].data_ptr(), ldq
        w.out_sid_dev, w.out_score_dev, w.scratch = ws["sid"].data_ptr(), ws["val"].data_ptr(), ws["scratch"].data_ptr()
        self._ws = ws
        return ws

    def _fp32_chunks(self, nq, k):
        """Chunks of up to chunk_queries() queries for the FP32 form: yields (row slice, workspace)."""
        step = self.chunk_queries()
        for lo in range(0, nq, step):
            yield slice(lo, min(nq, lo + step)), self.workspace(min(step, nq), k)

    def small_workspace(self, k):
        """Buffers of the exact small-batch path (cw_small_predict)."""
        sm = self._sm
        if sm and sm["cap_k"] >= k:
            return sm
        L, dev, Q = _lib.load(), self.tree.device, _lib.SMALL_Q
        k = max(k, sm["cap_k"]) if sm else max(k, 10)
        self._sm = sm = dict(
            cap_k=k,
            Q=torch.empty((Q, self.tree.d), dtype=torch.float32, device=dev),
            scores=torch.empty((self.ld, Q), dtype=torch.float32, device=dev),
            scratch=torch.empty(L.cw_small_scratch_words(max(self.n_pos, 1), k), dtype=torch.int32, device=dev),
            sid=torch.empty((Q, k), dtype=torch.int32, device=dev),
            val=torch.empty((Q, k), dtype=torch.float32, device=dev),
            n=torch.zeros(1, dtype=torch.int32, device=dev),
            sid_host=torch.empty((Q, k), dtype=torch.int32).pin_memory(),
            val_host=torch.empty((Q, k), dtype=torch.float32).pin_memory(),
        )
        # sm_Q, sm_scores, sm_scratch, sm_sid, sm_val, sm_n of every small-batch entry point and of cw_fused_work
        sm["ptrs"] = tuple(sm[n].data_ptr() for n in ("Q", "scores", "scratch", "sid", "val", "n"))
        return sm

    def fused_chunk_queries(self):
        n_int_pad = (self.hx["n_int"] + _lib.H_TILE - 1) // _lib.H_TILE * _lib.H_TILE
        per_query = (max(n_int_pad, 1) + _lib.load().cw_fused_flag_words(1, self.max_len)) * 4  # node scores + finish lists
        return int(max(256, min(32768, self.SCORE_BUDGET_BYTES // per_query) // 256 * 256))

    def fused_workspace(self, nq, k):
        """cw_fused_work for chunks of up to nq queries (rounded to whole tiles, at most fused_chunk_queries())."""
        L, dev, d, hx = _lib.load(), self.tree.device, self.tree.d, self.hx
        cap_q = min((max(nq, 1) + _lib.H_TILE - 1) // _lib.H_TILE * _lib.H_TILE, self.fused_chunk_queries())
        sm = self.small_workspace(k)
        hw = self._hws
        if hw and hw["cap_q"] >= cap_q and hw["cap_k"] >= k and hw["sm"] is sm:
            return hw
        self._hws = hw = None
        n_int_pad = (hx["n_int"] + _lib.H_TILE - 1) // _lib.H_TILE * _lib.H_TILE
        cap = self.FUSED_CAP
        hw = dict(
            cap_q=cap_q, cap_k=k, sm=sm,
            Q=torch.empty((cap_q, d), dtype=torch.float32, device=dev),
            A_int=torch.empty(max(16, L.cw_h_a_bytes(cap_q, d, _lib.H_F2, 3) if hx["n_int"] else 16), dtype=torch.uint8, device=dev),
            A_leaf=torch.empty(L.cw_h_a_bytes(cap_q, d, hx["leaf_layout"], 1), dtype=torch.uint8, device=dev),
            qv=torch.empty((cap_q, 4), dtype=torch.float32, device=dev),
            S=torch.empty((max(n_int_pad, 1), cap_q), dtype=torch.float32, device=dev),
            slots=torch.empty((cap_q, 32), dtype=torch.int32, device=dev),
            tau=torch.empty(cap_q, dtype=torch.float32, device=dev),
            cnt=torch.zeros(cap_q, dtype=torch.int32, device=dev),
            cand_val=torch.empty((cap_q, cap), dtype=torch.float32, device=dev),
            cand_row=torch.empty((cap_q, cap), dtype=torch.int32, device=dev),
            flag=torch.zeros(L.cw_fused_flag_words(cap_q, self.max_len), dtype=torch.int32, device=dev),
            sid=torch.empty((cap_q, k), dtype=torch.int32, device=dev),
            val=torch.empty((cap_q, k), dtype=torch.float32, device=dev),
            stats=torch.zeros(_lib.FUSED_STATS, dtype=torch.int32, device=dev),
            stats_host=torch.zeros(_lib.FUSED_STATS, dtype=torch.int32).pin_memory(),
        )
        w = _lib.CwFusedWork()
        w.cap_q, w.ldq, w.cap, w.fin_ml = cap_q, cap_q, cap, self.max_len
        w.Q_dev, w.A_int, w.A_leaf, w.qv, w.S = (hw[n].data_ptr() for n in ("Q", "A_int", "A_leaf", "qv", "S"))
        w.slots, w.tau, w.cnt, w.cand_val, w.cand_row = (hw[n].data_ptr() for n in ("slots", "tau", "cnt", "cand_val", "cand_row"))
        w.flag, w.out_sid_dev, w.out_val_dev, w.stats = (hw[n].data_ptr() for n in ("flag", "sid", "val", "stats"))
        w.sm_Q, w.sm_scores, w.sm_scratch, w.sm_sid, w.sm_val, w.sm_n = sm["ptrs"]
        hw["w"] = w
        self._hws = hw
        return hw

    def _fused_struct(self, hw):
        """The work struct with this call's audit settings; the index struct with the current eps."""
        w, fi = hw["w"], self.hx["fi"]
        w.audit_every = int(self.audit_every)
        w.audit_phase = self._audit_phase
        self._audit_phase += 1
        fi.eps_scale = self.eps_scale
        return fi, w

    def _account(self, st):
        """Fold the counters of one fused call (CW_FUSED_STATS words) into self.stats; an audit mismatch means the
        statistical part of eps did not hold: widen it and say so."""
        s = self.stats
        s["flagged"] += int(st[0]); s["unresolved"] += int(st[1]); s["cand_overflow"] += int(st[2])
        s["line_fail"] += int(st[3]); s["list_overflow"] += int(st[4]); s["queries"] += int(st[5])
        s["candidates"] += int(np.asarray(st[6:8], np.int32).view(np.uint64)[0])
        s["audited"] += int(st[8]); s["audit_mismatch"] += int(st[9]); s["refined"] += int(st[10]); s["rescored"] += int(st[11])
        if int(st[9]):
            self.eps_scale *= 4.0
            import warnings
            warnings.warn(f"cobweb-b200: {int(st[9])} audited quer(ies) differed from the exact path; eps widened to "
                          f"{self.eps_scale:.3g} (DenseIndex.stats['audit_mismatch'])")

    # ------------------------------------------------------------------ predict
    def node_scores(self, Q):
        """[nq, nn] node log-likelihood scores in index (BFS) order (CobwebWrapper.py:283-287), FP32 form."""
        nq = Q.shape[0]
        ws = self.workspace(nq, 0)
        _lib.check(_lib.load().cw_dense_node_scores(C.byref(self.ix), Q.data_ptr(), nq, ws["xt"].data_ptr(),
                                                    ws["scores"].data_ptr(), ws["ldq"], _lib.stream_ptr()), "cw_dense_node_scores")
        return ws["scores"][: self.nn, :nq].T

    def predict_small(self, Q, k):
        """Exact small-batch path for up to SMALL_Q queries on the device (cw_small_predict)."""
        sids = torch.empty((Q.shape[0], k), dtype=torch.int32, device=Q.device)
        vals = torch.empty((Q.shape[0], k), dtype=torch.float32, device=Q.device)
        self._run_small(Q, k, sids, vals)
        return sids, vals

    def predict(self, Q, k, want_leaf_scores=False, mode=None, small=True, query_tags=None, sent_tags=None, tag_version=None):
        """Device batch -> (sids [nq,k] int32, scores [nq,k], leaf_scores [nq,L] or None).  mode overrides self.mode for
        this call; small=False keeps batches of up to SMALL_Q queries off the small-batch path (tests).  query_tags [nq]
        int32 (with the sentences' tag words sent_tags and their version): only sentences s with
        sent_tags[s] & query_tags[q] != 0 are ranked (k in 1..MAX_K), short rows padded with -1 / -inf."""
        if query_tags is not None and want_leaf_scores:
            raise ValueError("leaf scores are not filtered by tags")
        if self.sentence_ids is not None and (want_leaf_scores or query_tags is not None):
            what = "leaf scores" if want_leaf_scores else "tag filters"
            raise ValueError(f"{what} are indexed by global sentence id; not available on a sentence shard")
        mode = mode or self.mode
        if mode not in self.MODES:
            raise ValueError(f"mode must be one of {self.MODES}")
        nq, tf = Q.shape[0], None
        if query_tags is None:
            sids = torch.empty((nq, max(k, 1)), dtype=torch.int32, device=Q.device)
            vals = torch.empty((nq, max(k, 1)), dtype=torch.float32, device=Q.device)
        else:
            if not 1 <= k <= _lib.MAX_K:
                raise ValueError(f"k must lie in [1, {_lib.MAX_K}]")
            sids = torch.full((nq, k), -1, dtype=torch.int32, device=Q.device)
            vals = torch.full((nq, k), float("-inf"), dtype=torch.float32, device=Q.device)
            if not nq or not self.n_pos:
                return sids, vals, None
        if mode == "fused" and self.hx is None and self.n_pos:
            self._build_fused()
        if query_tags is not None:
            t = self.tag_arrays(sent_tags, tag_version)
            tf = _lib.CwTagFilter()
            tf.query_tags, tf.pos_tags, tf.sent_tags = query_tags.data_ptr(), t["pos"].data_ptr(), sent_tags.data_ptr()
            tf.leaf_tags = t["leaf"].data_ptr() if t["leaf"] is not None else None
        leaf = torch.empty((nq, self.n_pos), dtype=torch.float32, device=Q.device) if want_leaf_scores else None
        route = self._route(nq, k, mode, small, want_leaf_scores)
        if route == "small":
            self._run_small(Q, k, sids, vals, tf)
        elif route == "fused":
            self._run_fused(Q, k, sids, vals, tf, query_tags)
        else:
            self._run_fp32(Q, k, sids, vals, tf, query_tags, leaf)
        return sids, vals, leaf

    # Each runner writes the top-k of the queries Q into sids / vals.  Given a tag filter tf (and the query tags qt it
    # points to), it calls the _tagged form of its entry points, which take the untagged form's arguments plus tf.
    def _run_small(self, Q, k, sids, vals, tf=None):
        """The exact small-batch path (cw_small_predict[_tagged]) for up to SMALL_Q queries."""
        L, sm = _lib.load(), self.small_workspace(k)
        args = (Q.data_ptr(), Q.shape[0], None, None, 0, 0, k, *sm["ptrs"], sids.data_ptr(), vals.data_ptr(), _lib.stream_ptr())
        if tf is None:
            _lib.check(L.cw_small_predict(C.byref(self.ix), *args), "cw_small_predict")
        else:
            _lib.check(L.cw_small_predict_tagged(C.byref(self.ix), C.byref(tf), *args), "cw_small_predict_tagged")

    def _run_fused(self, Q, k, sids, vals, tf=None, qt=None):
        """The fused pipeline (cw_fused_predict[_tagged]); the FP32 form answers the rows it leaves unresolved."""
        L, nq = _lib.load(), Q.shape[0]
        hw = self.fused_workspace(nq, k)
        fi, w = self._fused_struct(hw)
        hw["stats"].zero_()
        args = (Q.data_ptr(), nq, k, sids.data_ptr(), vals.data_ptr(), _lib.stream_ptr())
        if tf is None:
            _lib.check(L.cw_fused_predict(C.byref(fi), C.byref(w), *args), "cw_fused_predict")
        else:
            _lib.check(L.cw_fused_predict_tagged(C.byref(fi), C.byref(w), C.byref(tf), *args), "cw_fused_predict_tagged")
        hw["stats_host"].copy_(hw["stats"], non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the one read-back of a call: counters (flagged / audit)
        st = hw["stats_host"].numpy().copy()
        self._account(st)
        if st[1]:  # more flagged queries in a chunk than the device-side rounds take: the FP32 form answers them
            idx = torch.nonzero(sids[:, 0] == _lib.SID_UNRESOLVED).view(-1)
            s2, v2 = sids[idx], vals[idx]
            self._run_fp32(Q[idx].contiguous(), k, s2, v2, tf, qt[idx].contiguous() if tf is not None else None)
            sids[idx], vals[idx] = s2, v2

    def _run_fp32(self, Q, k, sids, vals, tf=None, qt=None, leaf=None):
        """The FP32 form chunk by chunk: node scores (cw_dense_node_scores), then path sums and top-k
        (cw_dense_paths_topk[_tagged]); leaf [nq, n_pos] (untagged only) also receives every sentence's score."""
        L, st = _lib.load(), _lib.stream_ptr()
        for r, ws in self._fp32_chunks(Q.shape[0], k):
            q = Q[r]
            _lib.check(L.cw_dense_node_scores(C.byref(self.ix), q.data_ptr(), q.shape[0], ws["xt"].data_ptr(),
                                              ws["scores"].data_ptr(), ws["ldq"], st), "cw_dense_node_scores")
            if tf is None:
                _lib.check(L.cw_dense_paths_topk(C.byref(self.ix), ws["scores"].data_ptr(), ws["ldq"], q.shape[0], k,
                                                 leaf[r].data_ptr() if leaf is not None else None, sids[r].data_ptr(),
                                                 vals[r].data_ptr(), ws["scratch"].data_ptr(), st), "cw_dense_paths_topk")
            else:
                tf.query_tags = qt[r].data_ptr()
                _lib.check(L.cw_dense_paths_topk_tagged(C.byref(self.ix), C.byref(tf), ws["scores"].data_ptr(), ws["ldq"],
                                                        q.shape[0], k, sids[r].data_ptr(), vals[r].data_ptr(),
                                                        ws["scratch"].data_ptr(), st), "cw_dense_paths_topk_tagged")

    def predict_one(self, q, k):
        """One query (contiguous float32 numpy row) -> list of k sentence ids: the shortest way through the exact
        small-batch path (one C call: H2D, two kernels + merge, D2H, sync; no torch objects created)."""
        sm = self.small_workspace(k)
        sid, val = sm["sid_host"], sm["val_host"]
        _lib.check(_lib.load().cw_small_predict_host(C.byref(self.ix), q.ctypes.data, 1, k, *sm["ptrs"], sid.data_ptr(),
                                                     val.data_ptr(), _lib.stream_ptr()), "cw_small_predict_host")
        return sid.view(-1)[:k].tolist()

    # ------------------------------------------------------------------ pair scores
    def _pair_calls(self, ids):
        """Column blocks of at most PAIR_MAX_M candidates and query chunks that fit PAIR_BUDGET_BYTES of scratch:
        yields (query slice, column slice, scratch)."""
        L, (nq, m) = _lib.load(), ids.shape
        mb = min(m, _lib.PAIR_MAX_M)
        per_query = int(L.cw_pair_scratch_words(1, mb, self.max_len))
        _lib.check(min(per_query, 0), "cw_pair_scratch_words")
        step = max(1, min(nq, self.PAIR_BUDGET_BYTES // (4 * per_query)))
        scratch = torch.empty(max(1, step * per_query), dtype=torch.int32, device=ids.device)
        for c0 in range(0, m, mb):
            for q0 in range(0, nq, step):
                yield slice(q0, min(nq, q0 + step)), slice(c0, min(m, c0 + mb)), scratch

    def _pair_check(self):
        if self.sentence_ids is not None:
            raise ValueError("pair scores are indexed by global sentence id; not available on a sentence shard")

    def pair_scores(self, Q, ids):
        """[nq, m] exact leaf scores of sentences ids[q, c] (-1 = padding -> -inf) for queries Q [nq, D], bit for bit the
        FP32 form's (cw_pair_scores).  Ids must lie in [-1, n_pos)."""
        self._pair_check()
        L = _lib.load()
        out = torch.empty(ids.shape, dtype=torch.float32, device=Q.device)
        if not self.n_pos or not ids.numel():
            return out.fill_(float("-inf"))
        rows, pos = self.rows(), self.pos_of_sid()
        for qs, cs, scratch in self._pair_calls(ids):
            cand = ids[qs, cs].contiguous()
            o = torch.empty(cand.shape, dtype=torch.float32, device=Q.device)
            q = Q[qs]
            _lib.check(L.cw_pair_scores(C.byref(self.ix), rows.data_ptr(), pos.data_ptr(), self.n_pos, q.data_ptr(),
                                        q.shape[0], cand.data_ptr(), cand.shape[1], o.data_ptr(), scratch.data_ptr(),
                                        _lib.stream_ptr()), "cw_pair_scores")
            out[qs, cs] = o
        return out

    def pair_scores_bwd(self, Q, ids, grad_out):
        """dL/dQ [nq, D] for dL/d(pair_scores(Q, ids)) = grad_out [nq, m] (cw_pair_scores_bwd); column blocks are added
        in order, so the result is the same bits on every run."""
        self._pair_check()
        L = _lib.load()
        grad = torch.zeros_like(Q)
        if not self.n_pos or not ids.numel():
            return grad
        rows, pos = self.rows(), self.pos_of_sid()
        part = torch.empty_like(Q) if ids.shape[1] > _lib.PAIR_MAX_M else None
        for qs, cs, scratch in self._pair_calls(ids):
            cand = ids[qs, cs].contiguous()
            g = grad_out[qs, cs].contiguous().to(torch.float32)
            q = Q[qs]
            dst = grad[qs] if part is None else part[qs]
            _lib.check(L.cw_pair_scores_bwd(C.byref(self.ix), rows.data_ptr(), pos.data_ptr(), self.n_pos, q.data_ptr(),
                                            q.shape[0], cand.data_ptr(), cand.shape[1], g.data_ptr(), dst.data_ptr(),
                                            scratch.data_ptr(), _lib.stream_ptr()), "cw_pair_scores_bwd")
            if part is not None:
                grad[qs] += part[qs]
        return grad

    STAGES = ("query_operands", "internal_scores_f16x3", "cumulative_sums", "sample_threshold", "leaf_filter_f16", "finish",
              "fallback_audit_tail")

    def profile_stages(self, Q, k):
        """Per-stage device times (ms, CUDA events inside cw_fused_profile) of ONE fused chunk: dict stage -> ms."""
        hw = self.fused_workspace(Q.shape[0], k)
        if Q.shape[0] > hw["cap_q"]:
            raise ValueError("profile_stages takes one chunk")
        fi, w = self._fused_struct(hw)
        sids = torch.empty((Q.shape[0], k), dtype=torch.int32, device=Q.device)
        vals = torch.empty((Q.shape[0], k), dtype=torch.float32, device=Q.device)
        ms = (C.c_float * _lib.FUSED_STAGES)()
        _lib.check(_lib.load().cw_fused_profile(C.byref(fi), C.byref(w), Q.data_ptr(), Q.shape[0], k, sids.data_ptr(),
                                                vals.data_ptr(), ms, _lib.stream_ptr()), "cw_fused_profile")
        return dict(zip(self.STAGES, [float(v) for v in ms]))

    def predict_host(self, Q_host, k, out_sid=None, out_val=None):
        """Host batch (numpy / pinned tensor) -> host ids/scores through ONE C-ABI call per batch:
        cw_fused_predict_host ("fused" mode), cw_small_predict_host (up to SMALL_Q queries) or cw_predict_dense_host
        (FP32 form); H2D + kernels + D2H + sync inside."""
        L = _lib.load()
        Qh = Q_host if torch.is_tensor(Q_host) else torch.from_numpy(np.ascontiguousarray(Q_host, np.float32))
        nq = Qh.shape[0]
        if out_sid is None:
            out_sid = torch.empty((nq, k), dtype=torch.int32)
            out_val = torch.empty((nq, k), dtype=torch.float32)
        route = self._route(nq, k, self.mode)
        if route == "small":
            sm = self.small_workspace(k)
            _lib.check(L.cw_small_predict_host(C.byref(self.ix), Qh.data_ptr(), nq, k, *sm["ptrs"], out_sid.data_ptr(),
                                               out_val.data_ptr(), _lib.stream_ptr()), "cw_small_predict_host")
        elif route == "fused":
            hw = self.fused_workspace(nq, k)
            fi, w = self._fused_struct(hw)
            st = (C.c_int32 * _lib.FUSED_STATS)()
            _lib.check(L.cw_fused_predict_host(C.byref(fi), C.byref(w), Qh.data_ptr(), nq, k, out_sid.data_ptr(),
                                               out_val.data_ptr(), st, _lib.stream_ptr()), "cw_fused_predict_host")
            self._account(np.asarray(list(st), np.int32))
        else:
            for r, ws in self._fp32_chunks(nq, k):
                q = Qh[r]
                _lib.check(L.cw_predict_dense_host(C.byref(self.ix), C.byref(ws["w"]), q.data_ptr(), q.shape[0], k,
                                                   out_sid[r].data_ptr(), out_val[r].data_ptr(), _lib.stream_ptr()),
                           "cw_predict_dense_host")
        return out_sid, out_val


class _RankScores(torch.autograd.Function):
    """cobweb_rank_scores with a gradient w.r.t. the queries (cw_rank_scores_bwd)."""

    @staticmethod
    def forward(ctx, Q, index):
        _, _, leaf = index.predict(Q.detach(), 0, want_leaf_scores=True, mode="fp32")
        ctx.index = index
        ctx.save_for_backward(Q.detach())
        return leaf

    @staticmethod
    def backward(ctx, grad_leaf):
        (Q,) = ctx.saved_tensors
        ix = ctx.index
        nq = Q.shape[0]
        out = torch.empty_like(Q)
        step = max(32, min(nq, ix.chunk_queries()))
        for lo in range(0, nq, step):
            n = min(step, nq - lo)
            gs = torch.empty((ix.nn, n), dtype=torch.float32, device=Q.device)
            g = grad_leaf[lo:lo + n].contiguous().to(torch.float32)
            _lib.check(_lib.load().cw_rank_scores_bwd(C.byref(ix.ix), Q[lo:lo + n].data_ptr(), n, g.data_ptr(), gs.data_ptr(),
                                                      n, out[lo:lo + n].data_ptr(), _lib.stream_ptr()), "cw_rank_scores_bwd")
        return out, None


class _PairScores(torch.autograd.Function):
    """score_sentences with a gradient w.r.t. the queries (cw_pair_scores_bwd)."""

    @staticmethod
    def forward(ctx, Q, ids, index):
        ctx.index = index
        ctx.save_for_backward(Q.detach(), ids)
        return index.pair_scores(Q.detach(), ids)

    @staticmethod
    def backward(ctx, grad_out):
        Q, ids = ctx.saved_tensors
        return ctx.index.pair_scores_bwd(Q, ids, grad_out.contiguous()), None, None


class CobwebWrapper:
    def __init__(self, corpus=None, corpus_embeddings=None, encode_func=lambda x: x):
        _lib.require_cuda()
        self.encode_func = encode_func
        self.sentences = []
        self.device = "cuda"
        self.max_init_search = 100000
        self._index = None
        self._level_weights = None
        self._weight_schedule = None
        self._schedule_params = {}
        self.max_depth = 0
        self._leaf_of_sentence = np.zeros(0, np.int32)

        if corpus_embeddings is not None:
            if isinstance(corpus_embeddings, list):
                corpus_embeddings = torch.tensor(corpus_embeddings)
            embedding_shape = corpus_embeddings.shape[1:]
        elif corpus and len(corpus) > 0:
            sample_emb = self.encode_func([corpus[0]])
            embedding_shape = sample_emb.shape[1:]
        else:
            raise ValueError("CobwebWrapper needs a corpus or corpus_embeddings to size the tree")
        self.tree = CobwebTorchTree(shape=embedding_shape, device=self.device)
        if corpus_embeddings is not None:
            if corpus is None:
                corpus = [None] * len(corpus_embeddings)
            self.add_sentences(corpus, corpus_embeddings)
        elif corpus is not None and len(corpus) > 0:
            self.add_sentences(corpus)

    # ------------------------------------------------------------------ build
    def add_sentences(self, new_sentences, new_vectors=None):
        """CobwebWrapper.add_sentences (CobwebWrapper.py:52-80): one ifit per row, in order; the
        leaf -> sentence-id bookkeeping is done by the kernel (n_sent) and the id map below."""
        if new_vectors is None:
            new_embeddings = self.encode_func(new_sentences)
        else:
            new_embeddings = new_vectors
            if isinstance(new_embeddings, list):
                new_embeddings = torch.tensor(new_embeddings)
            if new_embeddings.shape[1] != self.tree.shape[0]:
                print(f"[Warning] Provided vector dim {new_embeddings.shape[1]} != tree dim {self.tree.shape[0]}, re-encoding...")
                new_embeddings = self.encode_func(new_sentences)
        X = self.tree._as_device_mat(new_embeddings)
        n = min(len(new_sentences), X.shape[0])  # the reference zips sentences with embeddings (CobwebWrapper.py:70)
        new_sentences = list(new_sentences[:n])
        try:
            leaves = self.tree.ifit_batch(X[:n], tag_sentences=True).cpu().numpy()
        except _lib.CobwebB200Error as e:
            # rows inserted before the failure stay in the tree (their n_sent is tagged): keep wrapper and tree consistent
            done = int(getattr(e, "completed", 0))
            if done:
                self._record(new_sentences[:done], e.leaves[:done].cpu().numpy())
            raise
        self._record(new_sentences, leaves)

    def _record(self, new_sentences, leaves):
        self.sentences.extend(new_sentences)
        self._leaf_of_sentence = np.concatenate([self._leaf_of_sentence, np.asarray(leaves, np.int32)])
        self.tree._sent_stale = True   # node.sentence_id lists are rebuilt from the id map on next access
        self.tree._sent_loader = self._load_sentence_lists
        self._invalidate_prediction_index()

    @property
    def sentence_to_node(self):
        """sentence id -> concept handle (CobwebWrapper.py:77)."""
        return {i: CobwebNode(self.tree, int(n)) for i, n in enumerate(self._leaf_of_sentence)}

    def _load_sentence_lists(self):
        """leaf -> [sentence ids] from the id map (leaf.sentence_id.append of CobwebWrapper.py:73-77, done lazily)."""
        from .tree import SentenceList
        sent = {}
        order = np.argsort(self._leaf_of_sentence, kind="stable")
        for sid in order:
            nid = int(self._leaf_of_sentence[sid])
            if nid >= 0:
                sent.setdefault(nid, SentenceList(self.tree, nid)).extend([int(sid)])
        return sent

    def _sync_sentence_lists(self):
        self.tree._sync_sentences()

    def _invalidate_prediction_index(self):
        self._index = None
        self._shard_key = None
        self._shard_index = None

    @property
    def _prediction_index_valid(self):
        return self._index is not None

    def build_prediction_index(self):
        """CobwebWrapper.build_prediction_index (CobwebWrapper.py:91-208)."""
        if self._index is not None:
            return
        ix = DenseIndex(self.tree, self._leaf_of_sentence, self._level_weights)
        self._index = ix.set_mode(self._resolve_mode(ix))
        self.max_depth = max(self.max_depth, self._index.max_depth)

    # Mode of the dense index (DenseIndex.MODES; both return the same ids and scores).  "auto": the fused tcgen05
    # pipeline for indexes of AUTO_TENSOR_NODES nodes and more -- it builds fp16 operand copies, which 180 GB of HBM
    # is there for -- and the FP32 pipe below (launch-bound at that size).
    dense_mode = os.environ.get("COBWEB_B200_DENSE_MODE", "auto")
    AUTO_TENSOR_NODES = DenseIndex.TENSOR_MIN_NODES

    def _resolve_mode(self, index):
        if self.dense_mode != "auto":
            return self.dense_mode
        return "fused" if index.nn >= self.AUTO_TENSOR_NODES else "fp32"

    def set_dense_mode(self, mode):
        """Additive: how cobweb_predict_fast / predict_fast_batch compute the top-k -- "auto" (default), "fp32" (FP32
        pipe) or "fused" (tcgen05 fp16 filter + exact re-score).  See DenseIndex.MODES."""
        if mode != "auto" and mode not in DenseIndex.MODES:
            raise ValueError(f"mode must be 'auto' or one of {DenseIndex.MODES}")
        self.dense_mode = mode
        if self._index is not None:
            self._index.set_mode(self._resolve_mode(self._index))
        if getattr(self, "_shard_index", None) is not None:
            self._shard_index.set_mode(self._resolve_mode(self._shard_index))

    def force_rebuild_index(self):
        self._invalidate_prediction_index()
        self.build_prediction_index()

    # ------------------------------------------------------------------ level weights
    def set_level_weights(self, weights):
        self._level_weights = weights
        self._weight_schedule = None
        self._invalidate_prediction_index()

    def set_weight_schedule(self, schedule_type, max_depth=10, **kwargs):
        if self._prediction_index_valid:
            max_depth = self.max_depth
        self._weight_schedule = schedule_type
        self._schedule_params = kwargs
        self._level_weights = topology.generate_weight_schedule(schedule_type, max_depth, **kwargs)
        self._invalidate_prediction_index()

    def get_level_weights(self):
        return self._level_weights if self._level_weights is not None else [1.0, 1.0, 1.0, 1.0]

    def get_weight_schedule_info(self):
        return {"schedule_type": self._weight_schedule, "schedule_params": self._schedule_params,
                "current_weights": self.get_level_weights()}

    def get_prediction_index_info(self):
        ix = self._index
        return {"index_valid": ix is not None, "total_nodes": ix.nn if ix else 0,
                "leaf_paths_cached": ix.n_pos if ix else 0, "means_cached": ix is not None, "vars_cached": ix is not None}

    # ------------------------------------------------------------------ dense predict
    def _embed(self, input, is_embedding):
        emb = input if is_embedding else self.encode_func([input])[0]
        return self.tree._as_device_vec(emb).reshape(1, -1)

    # ------------------------------------------------------------------ sentence tags
    @staticmethod
    def _as_tag_words(v, n, what):
        """Integers in [-2^31, 2^32) (a scalar, broadcast, or [n]) -> device int32 [n] with the same 32 bits."""
        t = torch.as_tensor(v, device="cuda")
        if t.dtype.is_floating_point or t.dtype.is_complex or t.dtype == torch.bool or t.dim() > 1:
            raise ValueError(f"{what} must be integers: a scalar or a vector")
        t = t.to(torch.int64)
        if t.dim() == 0:
            t = t.expand(n)
        elif t.numel() != n:
            raise ValueError(f"{what} has {t.numel()} entries for {n}")
        if t.numel() and bool(((t < -(1 << 31)) | (t >= (1 << 32))).any()):
            raise ValueError(f"{what} must be 32-bit words (integers in [-2^31, 2^32))")
        return torch.where(t >= (1 << 31), t - (1 << 32), t).to(torch.int32).contiguous()

    def _tag_words(self):
        """Device int32 [len(self)]: the tag word of every sentence; sentences never tagged (added since) have 0."""
        t, n = getattr(self, "_tags", None), len(self)
        if t is None or t.numel() != n:
            new = torch.zeros(n, dtype=torch.int32, device=self.device)
            if t is not None:
                new[: min(n, t.numel())] = t[: min(n, t.numel())]
            self._tags = new
            self._tag_version = getattr(self, "_tag_version", 0) + 1
        return self._tags

    def set_sentence_tags(self, ids, tags):
        """Additive: set the 32-bit tag word of sentences ids [m] to tags ([m] or one value for all; integers in
        [-2^31, 2^32), read as 32 bits).  Every sentence starts with tag 0.  predict_fast_batch(Q, k, query_tags=...) ranks
        for query q only the sentences s with tags[s] & query_tags[q] != 0."""
        cur = self._tag_words()
        ids = torch.as_tensor(ids, device=self.device)
        if ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool or ids.dim() > 1:
            raise ValueError("ids must be an integer vector of sentence ids")
        ids = ids.reshape(-1).to(torch.int64)
        n = len(self)
        if ids.numel() and bool(((ids < 0) | (ids >= n)).any()):
            raise ValueError(f"sentence ids must lie in [0, {n})")
        if torch.unique(ids).numel() != ids.numel():
            raise ValueError("ids must not repeat")
        words = self._as_tag_words(tags, ids.numel(), "tags")
        new = cur.clone()
        new[ids] = words
        self._tags = new
        self._tag_version += 1

    def get_sentence_tags(self):
        """Additive: the tag word of every sentence, device int32 [len(self)] (a copy)."""
        return self._tag_words().clone()

    def predict_fast_batch(self, Q, k=5, query_tags=None):
        """Batched cobweb_predict_fast(return_ids=True): device tensors (ids [nq,k], scores [nq,k]).  query_tags
        (additive): a mask per query ([nq]) or one for all; query q then ranks only the sentences s with
        tags[s] & query_tags[q] != 0 (set_sentence_tags), and rows with fewer than k of them are padded with -1 / -inf.
        Scores are the same bits as rank_scores_batch(Q)."""
        self.build_prediction_index()
        Q = self.tree._as_device_mat(Q)
        k = min(int(k), self._index.n_pos)
        if query_tags is not None:
            return self._predict_fast_tagged(Q, k, query_tags)
        if k > _lib.MAX_K:
            _, _, leaf = self._index.predict(Q, 0, want_leaf_scores=True, mode="fp32")
            vals, ids = torch.sort(leaf, dim=1, descending=True, stable=True)
            return ids[:, :k].to(torch.int32), vals[:, :k]
        sids, vals, _ = self._index.predict(Q, k)
        return sids, vals

    def _predict_fast_tagged(self, Q, k, query_tags):
        qt = self._as_tag_words(query_tags, Q.shape[0], "query_tags")
        tags = self._tag_words()
        if k < 1:
            return (torch.empty((Q.shape[0], 0), dtype=torch.int32, device=Q.device),
                    torch.empty((Q.shape[0], 0), dtype=torch.float32, device=Q.device))
        if k <= _lib.MAX_K:
            sids, vals, _ = self._index.predict(Q, k, query_tags=qt, sent_tags=tags, tag_version=self._tag_version)
            return sids, vals
        # the leaf matrix with ineligible entries at -inf; eligible entries first, each part in (score desc, id asc)
        _, _, leaf = self._index.predict(Q, 0, want_leaf_scores=True, mode="fp32")
        elig = (tags.unsqueeze(0) & qt.unsqueeze(1)) != 0
        vals, ids = torch.sort(leaf.masked_fill_(~elig, float("-inf")), dim=1, descending=True, stable=True)
        e = elig.gather(1, ids)
        _, o = torch.sort((~e).to(torch.uint8), dim=1, stable=True)
        ids, vals, e = ids.gather(1, o)[:, :k], vals.gather(1, o)[:, :k], e.gather(1, o)[:, :k]
        return torch.where(e, ids, -1).to(torch.int32), vals

    def predict_fast_sharded(self, Q, k=5, world=None, rank=None):
        """Store-sharded dense predict (SURVEY 8e, trees beyond one HBM): this rank indexes and
        scores only its contiguous share of the sentences (in tree order) plus the nodes on their
        paths, then per-rank top-k lists are all-gathered and merged.  Same ids and scores as
        predict_fast_batch.  With world/rank given explicitly and no process group, returns this
        shard's candidates (used by the single-GPU test that emulates the ranks one after another)."""
        import torch.distributed as dist
        from . import parallel
        live = dist.is_available() and dist.is_initialized()
        if world is None:
            world, rank = (dist.get_world_size(), dist.get_rank()) if live else (1, 0)
        key = (world, rank, len(self.sentences))
        if getattr(self, "_shard_key", None) != key:
            t = self.tree.store.topology()
            order, parent_b, depth = topology.bfs_order(t["root"], t["child_off"], t["child_cnt"], t["child_pool"])
            row_of = np.full(t["n_used"], -1, np.int64)
            row_of[order] = np.arange(len(order))
            tree_order = np.lexsort((np.arange(len(self._leaf_of_sentence)), row_of[self._leaf_of_sentence]))
            lo, hi = parallel.shard_bounds(len(tree_order), world, rank)
            self._shard_index = DenseIndex(self.tree, self._leaf_of_sentence, self._level_weights,
                                           sentence_ids=np.sort(tree_order[lo:hi]))
            self._shard_index.set_mode(self._resolve_mode(self._shard_index))
            self._shard_key = key
        Q = self.tree._as_device_mat(Q)
        kk = min(int(k), self._shard_index.n_pos, _lib.MAX_K)
        ids, vals, _ = self._shard_index.predict(Q, kk)
        if kk < k:  # pad so every rank contributes the same number of candidates
            pad = k - kk
            ids = torch.cat([ids, torch.full((ids.shape[0], pad), -1, dtype=ids.dtype, device=ids.device)], 1)
            vals = torch.cat([vals, torch.full((vals.shape[0], pad), float("-inf"), device=vals.device)], 1)
        if live and world > 1:
            ci, cv = parallel.gather_candidates(ids, vals)
            return parallel.merge_topk(ci, cv, k)
        return ids, vals

    def rank_scores_batch(self, Q):
        """Batched cobweb_rank_scores: [nq, L] leaf scores indexed by sentence id.  Differentiable
        w.r.t. Q when Q is a CUDA tensor that requires grad (the training use of the reference,
        src/training/cobweb_query_train.py:104-126)."""
        self.build_prediction_index()
        if torch.is_tensor(Q) and Q.requires_grad:
            Qd = Q.to(device=self.device, dtype=torch.float32)
            Qd = Qd.reshape(1, -1) if Qd.dim() == 1 else Qd
            return _RankScores.apply(Qd.contiguous(), self._index)
        _, _, leaf = self._index.predict(self.tree._as_device_mat(Q), 0, want_leaf_scores=True, mode="fp32")
        return leaf

    def score_sentences(self, Q, ids):
        """Additive: the Cobweb leaf scores of chosen sentences, bit for bit rank_scores_batch(Q)[q, ids[q, c]], without
        scoring the rest of the tree.  Q [nq, D] or [D]; ids [nq, m] sentence ids per query, or [m] for the same list
        for every query; -1 is padding and scores -inf.  Returns [nq, m] float32 on the device ([m] for a [D] query).
        Differentiable w.r.t. Q when Q requires grad; padding gets no gradient, a repeated id gets the sum of its
        entries' gradients."""
        self.build_prediction_index()
        single = torch.is_tensor(Q) and Q.dim() == 1 or not torch.is_tensor(Q) and np.ndim(Q) == 1
        if torch.is_tensor(Q) and Q.requires_grad:
            if Q.dim() not in (1, 2) or Q.shape[-1] != self.tree.d:
                raise ValueError(f"Q must be [nq, {self.tree.d}] or [{self.tree.d}]")
            Qd = Q.to(device=self.device, dtype=torch.float32).reshape(-1, self.tree.d).contiguous()
        else:
            Qd = self.tree._as_device_mat(Q).reshape(-1, self.tree.d).contiguous()
        ids = torch.as_tensor(ids, device=Qd.device)
        if ids.dtype.is_floating_point or ids.dtype == torch.bool or ids.dim() not in (1, 2):
            raise ValueError("ids must be an integer tensor of shape [m] or [nq, m]")
        if ids.dim() == 1:
            ids = ids.unsqueeze(0).expand(Qd.shape[0], -1)
        elif ids.shape[0] != Qd.shape[0]:
            raise ValueError(f"ids has {ids.shape[0]} rows for {Qd.shape[0]} queries")
        n = len(self)
        if ids.numel() and bool(((ids < -1) | (ids >= n)).any()):
            raise ValueError(f"sentence ids must lie in [-1, {n}) (-1 = padding)")
        ids = ids.to(torch.int32).contiguous()
        if Qd.requires_grad:
            out = _PairScores.apply(Qd, ids, self._index)
        else:
            out = self._index.pair_scores(Qd, ids)
        return out[0] if single else out

    def rerank(self, Q, ids, k):
        """Additive: the k best of the given candidates by exact Cobweb score, ranked like predict_fast_batch (score
        desc, sentence id asc).  Q [nq, D] or [D]; ids as in score_sentences.  Returns (ids [nq, k] int32, scores [nq, k])
        ([k] each for a [D] query), padded with -1 / -inf when fewer than k valid candidates exist.  Entries are ranked
        as given: an id passed twice can appear twice."""
        k = int(k)
        if k < 0:
            raise ValueError("k must be >= 0")
        with torch.no_grad():
            scores = self.score_sentences(Q.detach() if torch.is_tensor(Q) else Q, ids)
        single = scores.dim() == 1
        scores = scores.unsqueeze(0) if single else scores
        ids = torch.as_tensor(ids, device=scores.device).to(torch.int32).reshape(-1, scores.shape[1])
        ids = ids.expand(scores.shape[0], -1)
        # (score desc, id asc), padding last: sort by id (padding as the largest), then stably by score
        tie = torch.where(ids < 0, torch.iinfo(torch.int32).max, ids)
        _, o1 = torch.sort(tie, dim=1, stable=True)
        s2, o2 = torch.sort(scores.gather(1, o1), dim=1, descending=True, stable=True)
        top_ids, top_val = ids.gather(1, o1.gather(1, o2))[:, :k], s2[:, :k]
        if top_ids.shape[1] < k:
            pad = k - top_ids.shape[1]
            top_ids = torch.cat([top_ids, top_ids.new_full((top_ids.shape[0], pad), -1)], 1)
            top_val = torch.cat([top_val, top_val.new_full((top_val.shape[0], pad), float("-inf"))], 1)
        return (top_ids[0], top_val[0]) if single else (top_ids, top_val)

    def cobweb_predict_indexed(self, input, k=5, return_ids=False, is_embedding=False):
        """CobwebWrapper.cobweb_predict_indexed (CobwebWrapper.py:210-265), noise-free."""
        self.build_prediction_index()
        if len(self.sentences) == 0:
            return []
        kk = min(int(k), self._index.n_pos)
        if 1 <= kk <= _lib.MAX_K:
            emb = input if is_embedding else self.encode_func([input])[0]
            emb = emb.detach().cpu().numpy() if torch.is_tensor(emb) else emb
            q = np.ascontiguousarray(emb, dtype=np.float32).reshape(-1)
            if q.shape[0] != self.tree.d:
                raise ValueError(f"instance dim {q.shape[0]} != tree dim {self.tree.d}")
            sids = self._index.predict_one(q, kk)
        else:
            ids, _ = self.predict_fast_batch(self._embed(input, is_embedding), k)
            sids = ids[0].cpu().tolist()
        out = []
        for sid in sids:
            if 0 <= sid < len(self.sentences):
                out.append(sid if return_ids else self.sentences[sid])
        return out

    def cobweb_predict_fast(self, input, k=5, return_ids=False, is_embedding=False):
        return self.cobweb_predict_indexed(input, k, return_ids, is_embedding)

    def cobweb_rank_scores(self, input, is_embedding=False):
        """CobwebWrapper.cobweb_rank_scores (CobwebWrapper.py:267-294); differentiable w.r.t. a tensor
        input that requires grad, like the reference's torch expression."""
        self.build_prediction_index()
        if len(self.sentences) == 0:
            return torch.empty(0, device=self.device)
        x = input if is_embedding else self.encode_func([input])[0]
        if torch.is_tensor(x) and x.requires_grad:
            return self.rank_scores_batch(x.reshape(1, -1))[0]
        return self.rank_scores_batch(self.tree._as_device_vec(x).reshape(1, -1))[0]

    # ------------------------------------------------------------------ best-first predict
    def predict_batch(self, Q, k=5):
        """Batched cobweb_predict: returns (leaves [nq,k] node ids on the host, nfound [nq],
        lp_calls [nq])."""
        r = self.tree.categorize_batch(Q, retrieve_k=k, use_best=True, max_nodes=self.max_init_search)
        return r["leaves"].cpu().numpy(), r["nfound"].cpu().numpy(), r["lp_calls"].cpu().numpy()

    def cobweb_predict(self, input, k=5, return_ids=False, is_embedding=False):
        """CobwebWrapper.cobweb_predict (CobwebWrapper.py:435-461)."""
        emb = input if is_embedding else self.encode_func([input])[0]
        leaves = self.tree.categorize(emb, use_best=True, max_nodes=self.max_init_search, retrieve_k=k)
        self._sync_sentence_lists()
        results = []
        for leaf in leaves:
            for sid in sorted(self.tree._sent.get(leaf.node_id, [])):
                if sid is None or sid >= len(self.sentences):
                    continue
                results.append(sid if return_ids else self.sentences[sid])
        return results

    # ------------------------------------------------------------------ misc
    def print_tree(self):
        self._sync_sentence_lists()
        b = self.tree.bfs()
        kids = [[] for _ in b["order"]]
        for i in range(1, len(b["order"])):
            kids[b["parent"][i]].append(i)

        def rec(i, depth):
            nid = int(b["order"][i])
            print(f"{'  ' * depth}- Node ID {nid} Sentence ID: {list(self.tree._sent.get(nid, []))}")
            for c in kids[i]:
                rec(c, depth + 1)

        print("\nCobweb Sentence Clustering Tree:")
        rec(0, 0)

    def dump_json(self, save_path=None):
        """CobwebWrapper.dump_json (CobwebWrapper.py:484-497)."""
        self._sync_sentence_lists()
        state = {"tree": json.loads(self.tree.dump_json()), "sentences": self.sentences,
                 "embedding_dim": self.tree.shape[0]}
        if save_path:
            with open(save_path, "w") as f:
                json.dump(state, f, indent=2)
        return json.dumps(state, indent=2)

    @staticmethod
    def load_json(json_data, encode_func=lambda x: x):
        """CobwebWrapper.load_json (CobwebWrapper.py:500-555).  The reference's version crashes on
        list-valued sentence ids (SURVEY.md 4); this one restores the id -> leaf map."""
        data = json.loads(json_data) if isinstance(json_data, str) else json_data
        w = CobwebWrapper.__new__(CobwebWrapper)
        w.encode_func = encode_func
        w.device = "cuda"
        w.sentences = data.get("sentences", [])
        w.max_init_search = data.get("max_init_search", 100000)
        w._index, w._level_weights, w._weight_schedule, w._schedule_params, w.max_depth = None, None, None, {}, 0
        w.tree = CobwebTorchTree(shape=(int(data["embedding_dim"]),), device=w.device)
        w.tree.load_json(json.dumps(data["tree"]))
        leaf = np.full(len(w.sentences), -1, np.int32)
        for nid, lst in w.tree._sent.items():
            for sid in lst:
                if 0 <= sid < len(leaf):
                    leaf[sid] = nid
        w._leaf_of_sentence = leaf
        return w

    def save_snapshot(self, path):
        """Additive (SURVEY 8f-2): binary snapshot of tree + sentence map + sentences; a 1M-node tree is a few seconds of
        streaming instead of gigabytes of decimal JSON.  load_snapshot restores an equivalent wrapper."""
        extra = {"sentences": self.sentences if any(s is not None for s in self.sentences) else None,
                 "n_sentences": len(self.sentences), "max_init_search": self.max_init_search, "level_weights": self._level_weights}
        tags = self._tag_words()
        if bool((tags != 0).any()):  # little-endian int32 words, base64 (a snapshot without them loads as all 0)
            extra["sentence_tags"] = base64.b64encode(tags.cpu().numpy().astype("<i4").tobytes()).decode()
        self.tree.save_snapshot(path, self._leaf_of_sentence, extra=extra)

    @staticmethod
    def load_snapshot(path, encode_func=lambda x: x):
        w = CobwebWrapper.__new__(CobwebWrapper)
        w.encode_func, w.device = encode_func, "cuda"
        w._index, w._weight_schedule, w._schedule_params, w.max_depth = None, None, {}, 0
        w._shard_key = w._shard_index = None
        w.tree = CobwebTorchTree(shape=(1,), device=w.device)
        leaf, extra = w.tree.load_snapshot(path)
        w._leaf_of_sentence = np.asarray(leaf, np.int32)
        w.sentences = extra.get("sentences") or [None] * int(extra.get("n_sentences", len(leaf)))
        w.max_init_search = extra.get("max_init_search", 100000)
        w._level_weights = extra.get("level_weights")
        w.tree._sent_stale, w.tree._sent_loader = True, w._load_sentence_lists
        if extra.get("sentence_tags"):
            t = np.frombuffer(base64.b64decode(extra["sentence_tags"]), "<i4").astype(np.int32)
            w._tags, w._tag_version = torch.as_tensor(t, device=w.device), 1
        return w

    def get_node_path_stats(self, sentence_id):
        """CobwebWrapper.get_node_path_stats (CobwebWrapper.py:297-313): (means [len, D], vars [len, D]) of the nodes on
        the root -> leaf path of a sentence, root first; (None, None) for an unknown sentence."""
        if not 0 <= sentence_id < len(self._leaf_of_sentence) or self._leaf_of_sentence[sentence_id] < 0:
            return None, None
        node, path = int(self._leaf_of_sentence[sentence_id]), []
        par = self.tree.store.parent
        while node >= 0:
            path.append(node)
            node = int(par[node].item())
        idx = torch.as_tensor(path[::-1], device=self.tree.device)
        st = self.tree.store
        cnt = st.count[idx].unsqueeze(1)
        var = torch.where(cnt > 0, self.tree.compute_var(st.m2[idx], cnt.clamp_min(1e-30)),
                          self.tree.prior_var.expand_as(st.m2[idx]))
        return st.mean[idx].clone(), var

    def visualize_subtrees(self, directory, num_leaves=6):
        raise NotImplementedError("graphviz rendering is outside the hot-path scope (SURVEY.md section 2, row 3)")

    def __len__(self):
        return len(self.sentences)
