"""cw_pair_scores / cw_pair_scores_bwd take the [nn, D, 2] row buffer only 16-byte aligned: fn_exact_kernel fetches it
with bulk copies, whose source addresses must be 16-byte aligned.  The argument check runs on the host, and the calls
below ask for no work (nq = m = 0), so nothing is launched and no GPU is needed: the index's pointers are never read."""
import ctypes as C

from rag_cobweb_b200 import _lib


def test_pair_scores_reject_unaligned_rows():
    L = _lib.load()
    ix = _lib.CwIndex()
    ix.D, ix.nn, ix.n_pos, ix.max_len = 8, 4, 4, 2
    ix.path_idx, ix.level_w, ix.pos_rec, ix.sumlog = 1 << 20, 2 << 20, 3 << 20, 4 << 20
    for rows in (5 << 20, (5 << 20) + 8, (5 << 20) + 4):
        want = _lib.CW_E_ARG if rows % 16 else 0
        rc = L.cw_pair_scores(C.byref(ix), rows, None, 4, None, 0, None, 0, None, None, None)
        assert rc == want and (not want or "16-byte aligned" in L.cw_last_error().decode())
        rc = L.cw_pair_scores_bwd(C.byref(ix), rows, None, 4, None, 0, None, 0, None, None, None, None)
        assert rc == want and (not want or "16-byte aligned" in L.cw_last_error().decode())
