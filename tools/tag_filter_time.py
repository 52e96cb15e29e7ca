"""Times tag-filtered dense retrieval (predict_fast_batch(Q, k, query_tags=...)) against the unfiltered call on one GPU.

  python tools/tag_filter_time.py [--snapshot PATH] [--docs 100000] [--dim 768] [--queries 10000] [--out FILE]

The tree is the engine's ifit of the cfg3 corpus (synth.corpus unit, seed 0), or a bench.py --snapshot of it.  Every
sentence carries one of 32 tag bits (uniform, seeded); each query's mask has b random bits, b in {1, 4, 16, 32}, so
about b/32 of the sentences are eligible.  Filtered and unfiltered calls alternate in the same run.  Reported per case:
CUDA-event time (median of the timed runs after two warm-up runs) and queries/s; for the fused path also the flagged
queries and the filter's candidates per query (DenseIndex.stats) of one call.  Also: the cost of deriving the position
and leaf tags after a retag, the FP32 path at k = 50 (past the fused path's k) and the small-batch path at nq = 1."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rag_cobweb_b200 import CobwebWrapper, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--snapshot")
ap.add_argument("--docs", type=int, default=100000)
ap.add_argument("--dim", type=int, default=768)
ap.add_argument("--queries", type=int, default=10000)
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--out")
args = ap.parse_args()
lines = []


def log(s):
    print(s, flush=True)
    lines.append(s)


def timed(fn, reps):
    """Median ms over reps runs after two warm-up runs (CUDA events around each run)."""
    for _ in range(2):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
log(f"device: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi[0] if smi else 'n/a'}")
n, d, nq = args.docs, args.dim, args.queries
x = synth.corpus(n, d, "unit", seed=0)
t0 = time.time()
if args.snapshot and os.path.exists(args.snapshot):
    w = CobwebWrapper.load_snapshot(args.snapshot)
    assert len(w) == n and w.tree.d == d, "snapshot of another workload"
    how = f"snapshot {args.snapshot}"
else:
    w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=torch.from_numpy(x).cuda())
    how = "ifit"
w.build_prediction_index()
ix = w._index
torch.cuda.synchronize()
log(f"tree {n} x {d} unit ({how}, {time.time() - t0:.1f} s): {ix.nn} index rows, max_len {ix.max_len}, mode {ix.mode}")
q, _ = synth.queries(x, nq, "unit", seed=1)
Q = torch.from_numpy(q).cuda()
rng = np.random.default_rng(0)
w.set_sentence_tags(np.arange(n), (1 << rng.integers(0, 32, n)).astype(np.int64))

tags = w._tag_words()


def derive():
    ix._tag_cache = None
    ix.tag_arrays(tags, w._tag_version)


log(f"deriving pos_tags [{ix.n_pos}] and leaf_tags [{ix.hx['n_leaf'] if ix.hx else 0}] after a retag: "
    f"{timed(derive, args.reps):.3f} ms")


def masks(bits, count):
    m = np.zeros(count, np.int64)
    for i in range(count):
        m[i] = int(np.bitwise_or.reduce(1 << rng.choice(32, bits, replace=False)))
    return torch.from_numpy(m).cuda()


def stats_of(fn):
    s0 = dict(ix.stats)
    fn()
    return {k: ix.stats[k] - s0[k] for k in ("queries", "flagged", "candidates")}


log("")
log(f"k 10, nq {nq}, mode {ix.mode}: unfiltered and filtered calls alternated (median of {args.reps} timed runs)")
for bits in (1, 4, 16, 32):
    qt = masks(bits, nq)
    plain = lambda: w.predict_fast_batch(Q, 10)  # noqa: E731
    tagged = lambda: w.predict_fast_batch(Q, 10, query_tags=qt)  # noqa: E731
    tp, tt = [], []
    for _ in range(2):
        tp.append(timed(plain, args.reps))
        tt.append(timed(tagged, args.reps))
    sp, st = stats_of(plain), stats_of(tagged)
    cq = lambda s: s["candidates"] / max(1, s["queries"])  # noqa: E731
    log(f"mask bits {bits:>2}: unfiltered {min(tp):8.3f} ms ({nq / min(tp) * 1e3:11.0f} q/s)  filtered {min(tt):8.3f} ms "
        f"({nq / min(tt) * 1e3:11.0f} q/s)  flagged {sp['flagged']} / {st['flagged']}  candidates/query "
        f"{cq(sp):7.1f} / {cq(st):7.1f}  (unfiltered / filtered)")

log("")
qt = masks(4, nq)
tp = timed(lambda: w.predict_fast_batch(Q, 50), 3)
tt = timed(lambda: w.predict_fast_batch(Q, 50, query_tags=qt), 3)
log(f"FP32 path, k 50, nq {nq}, mask bits 4: unfiltered {tp:8.3f} ms ({nq / tp * 1e3:9.0f} q/s)  filtered {tt:8.3f} ms "
    f"({nq / tt * 1e3:9.0f} q/s)")
Q1, qt1 = Q[:1].contiguous(), qt[:1].contiguous()
tp = timed(lambda: w.predict_fast_batch(Q1, 10), 20)
tt = timed(lambda: w.predict_fast_batch(Q1, 10, query_tags=qt1), 20)
log(f"small path, k 10, nq 1, mask bits 4: unfiltered {tp:8.3f} ms  filtered {tt:8.3f} ms")
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
