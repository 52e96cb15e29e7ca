"""Times score_sentences (exact (query, sentence) pair scores, cw_pairs.cu) forward and forward + backward against the
dense baseline it replaces, rank_scores_batch(Q) + gather and its backward, on one GPU.

  python tools/pair_scores_time.py [--snapshot PATH] [--docs 100000] [--dim 768] [--queries 10000] [--out FILE]

The tree is the engine's ifit of the cfg3 corpus (synth.corpus unit, seed 0), or a bench.py --snapshot of it.
Candidates: the top-m of predict_fast_batch (clustered: the paths share most ancestors) and uniformly random ids (little
sharing), m in {10, 100, 1000}, for the whole query batch and for one query with m = 1000.  Reported per case: CUDA-event
time (median of the timed repetitions after warm-up), distinct index rows per query (exact, on a sample of queries),
algorithmic bytes = distinct rows x (8 D + 4) per query, and that over the forward time.  The rows of a cfg3 tree
(100k sentences x 768 x 8 bytes, ~1 GB) do not fit the 126 MB L2, but the clustered lists reread the upper levels, which
do: the effective rate can exceed HBM bandwidth there."""
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
ap.add_argument("--reps", type=int, default=5)
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
path, pos = ix.path_idx, ix.pos_of_sid()
row_bytes = 8 * d + 4


def distinct_rows(ids, sample=200):
    """Mean number of distinct index rows on the candidates' paths per query, over up to `sample` queries."""
    tot = 0
    qs = np.linspace(0, ids.shape[0] - 1, min(sample, ids.shape[0])).astype(np.int64)
    for qi in qs:
        p = path[pos[ids[qi].long()].long()]
        tot += int(torch.unique(p[p >= 0]).numel())
    return tot / len(qs)


def case(label, Qc, ids, reps):
    nqc, m = ids.shape
    fwd = timed(lambda: w.score_sentences(Qc, ids), reps)
    G = torch.randn(ids.shape, device="cuda")
    Qg = Qc.clone().requires_grad_(True)

    def fb():
        Qg.grad = None
        w.score_sentences(Qg, ids).backward(G)
    both = timed(fb, reps)
    dr = distinct_rows(ids)
    gb = dr * row_bytes * nqc / 1e9
    log(f"{label:<34} nq {nqc:>5} m {m:>4}: fwd {fwd:9.3f} ms  fwd+bwd {both:9.3f} ms  distinct rows/query {dr:8.1f}  "
        f"algorithmic bytes {gb:8.3f} GB  -> {gb / fwd * 1e3:8.1f} GB/s fwd")
    return fwd, both


log("")
log("score_sentences (median of %d timed runs after 2 warm-up runs)" % args.reps)
for m in (10, 100, 1000):
    top, _ = w.predict_fast_batch(Q, m)
    case(f"top-{m} of predict_fast_batch", Q, top, args.reps)
    rnd = torch.from_numpy(rng.integers(0, n, (nq, m)).astype(np.int32)).cuda()
    case("uniform random ids", Q, rnd, args.reps)
Q1 = Q[:1].contiguous()
top1, _ = w.predict_fast_batch(Q1, 1000)
case("one query, top-1000 of predict", Q1, top1, 20)
case("one query, random ids", Q1, torch.from_numpy(rng.integers(0, n, (1, 1000)).astype(np.int32)).cuda(), 20)
one = timed(lambda: w.predict_fast_batch(Q1, 10), 20)
log(f"predict_fast_batch, one query, k 10 (same run): {one:.3f} ms")

log("")
log("baseline: rank_scores_batch(Q) [nq, L] + gather, and its backward with the pair gradient scattered into [nq, L]")
for m in (10, 1000):
    ids = torch.from_numpy(rng.integers(0, n, (nq, m)).astype(np.int32)).cuda()
    fwd = timed(lambda: w.rank_scores_batch(Q).gather(1, ids.long()), 3)
    G = torch.randn(ids.shape, device="cuda")
    Qg = Q.clone().requires_grad_(True)

    def fb():
        Qg.grad = None
        leaf = w.rank_scores_batch(Qg)
        leaf.gather(1, ids.long()).backward(G)
    both = timed(fb, 3)
    log(f"rank_scores_batch + gather           nq {nq:>5} m {m:>4}: fwd {fwd:9.3f} ms  fwd+bwd {both:9.3f} ms")
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
