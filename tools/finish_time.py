"""Where the fused predict's finish stage spends its time, and what its two exact-row launches move.

  python tools/finish_time.py [--docs 100000] [--dim 768] [--queries 10000] [--calls 10] [--out FILE]

The tree is the engine's ifit of the bench corpus (synth.corpus unit, seed 0), the queries are bench.py's (seed 1).
Reported, in one run: the card, its power limit and SM clocks; the per-launch device times of the finish stage's five
kernels (torch.profiler over --calls predict calls, median per launch); the stage times of one chunk from
cw_fused_profile (CUDA events); and for each fn_exact_kernel launch the row bytes it reads, list length x 8 D summed
over the queries (the lengths are the meta words FM_NSEL / FM_NANC of the finish scratch after one call), as TB/s
and as bytes per clock per SM at the card's maximum SM clock."""
import argparse
import collections
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from rag_cobweb_b200 import CobwebWrapper, synth, _lib  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--docs", type=int, default=100000)
ap.add_argument("--dim", type=int, default=768)
ap.add_argument("--queries", type=int, default=10000)
ap.add_argument("--k", type=int, default=10)
ap.add_argument("--calls", type=int, default=10)
ap.add_argument("--out")
args = ap.parse_args()
lines = []


def log(s):
    print(s, flush=True)
    lines.append(s)


def smi(fields):
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={fields}", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    return [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")] if r.returncode == 0 and r.stdout.strip() else []


# meta words of the finish scratch (cw_half.cu): FM_NSEL, FM_NANC, ..., the survivors from word 8, CW_FUSED_MSURV of them
hdr = open(os.path.join(ROOT, "include", "cobweb_b200.h")).read()
MSURV = int(re.search(r"#define CW_FUSED_MSURV (\d+)", hdr).group(1))
FM_NSEL, FM_NANC, FM_STRIDE = 0, 1, 8 + MSURV
FINISH = ("fn_select_kernel", "fn_exact_kernel", "fn_line_kernel", "fn_topk_kernel")

assert torch.cuda.is_available(), "finish_time.py measures on the GPU"
props = torch.cuda.get_device_properties(0)
name, plimit, sm_max = (smi("name,power.limit,clocks.max.sm") + ["n/a"] * 3)[:3]
log(f"device: {props.name}, {props.multi_processor_count} SMs; nvidia-smi: {name}, power limit {plimit} W, "
    f"max SM clock {sm_max} MHz")
n, d, nq, k = args.docs, args.dim, args.queries, args.k
x = synth.corpus(n, d, "unit", seed=0)
t0 = time.time()
w = CobwebWrapper(corpus=[None] * n, corpus_embeddings=torch.from_numpy(x).cuda())
w.build_prediction_index()
ix = w._index
torch.cuda.synchronize()
log(f"tree {n} x {d} unit (ifit + index, {time.time() - t0:.1f} s): {ix.nn} index rows, max_len {ix.max_len}, "
    f"mode {ix.mode}")
q, _ = synth.queries(x, nq, "unit", seed=1, targets=np.arange(nq) % n)
Q = torch.from_numpy(q).cuda()
assert ix.fused_ready(k), "the index answers on the FP32 pipe at this size: no finish stage to time"
for _ in range(3):
    ix.predict(Q, k)
torch.cuda.synchronize()

hw = ix.fused_workspace(nq, k)
cap_q = hw["cap_q"]
assert nq <= cap_q, "more queries than one fused chunk: the meta words hold the last chunk only"
base = 4 + cap_q + _lib.SMALL_Q
meta = hw["flag"][base:base + cap_q * FM_STRIDE].view(cap_q, FM_STRIDE)[:nq].cpu().numpy()
row_bytes = 8 * d
lists = {"refine": meta[:, FM_NSEL].astype(np.int64), "ancestors": meta[:, FM_NANC].astype(np.int64)}
for lab, v in lists.items():
    log(f"{lab:<9} list: {v.mean():6.2f} rows per query (max {v.max()}), {v.sum() * row_bytes / 1e9:.3f} GB of rows")

# per-launch device times: every finish kernel of --calls predict calls; exact launches alternate refine / ancestors
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(args.calls):
        ix.predict(Q, k)
    torch.cuda.synchronize()
with tempfile.TemporaryDirectory() as td:
    path = os.path.join(td, "trace.json")
    prof.export_chrome_trace(path)
    events = json.load(open(path))["traceEvents"]
kern = sorted((e for e in events if e.get("cat") == "kernel" and any(f in e.get("name", "") for f in FINISH)),
              key=lambda e: e["ts"])
times = collections.defaultdict(list)
n_exact = 0
for e in kern:
    f = next(f for f in FINISH if f in e["name"])
    if f == "fn_exact_kernel":
        f += " (refine)" if n_exact % 2 == 0 else " (ancestors)"
        n_exact += 1
    times[f].append(e["dur"])
sm_now = (smi("clocks.sm") + ["n/a"])[0]
clk_hz = float(sm_max) * 1e6 if sm_max.replace(".", "").isdigit() else float("nan")
log("")
log(f"finish launches, median over {args.calls} predict calls (torch.profiler; SM clock after the run {sm_now} MHz; "
    f"B/clk per SM at the max SM clock {sm_max} MHz over {props.multi_processor_count} SMs)")
order = ["fn_select_kernel", "fn_exact_kernel (refine)", "fn_line_kernel", "fn_exact_kernel (ancestors)", "fn_topk_kernel"]
total = 0.0
for f in order:
    us = float(np.median(times[f])) if times[f] else float("nan")
    total += us
    s = f"  {f:<28} {us:8.1f} us  ({len(times[f])} launches)"
    lab = {"fn_exact_kernel (refine)": "refine", "fn_exact_kernel (ancestors)": "ancestors"}.get(f)
    if lab:
        by = float(lists[lab].sum() * row_bytes)
        s += (f"  rows {by / 1e9:.3f} GB -> {by / (us * 1e-6) / 1e12:5.2f} TB/s, "
              f"{by / (us * 1e-6) / clk_hz / props.multi_processor_count:5.1f} B/clk per SM")
    log(s)
log(f"  {'sum of the five':<28} {total:8.1f} us")
reps = [ix.profile_stages(Q, k) for _ in range(5)]
log("stages of one chunk (cw_fused_profile, CUDA events, median of 5): " +
    ", ".join(f"{s} {np.median([r[s] for r in reps]):.3f} ms" for s in reps[0]))
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
