"""Per-kernel CUDA time of one bench step, split by stream: where the merge fold's time goes.

    python profiles/fold_kernels_time.py [--reads 50000000] [--genes 60000] [--warmup 2]

The data set is bench.py's configs[3] on one GPU, built the way bench.py builds it (make_tables, make_dataset over every
chromosome, device resident), with bench.py's update-gtf parameters.  After the warm-up steps one step (lrb_pipeline_run +
lrb_update_run) runs under torch.profiler with CUDA activities; the kernels of the trace are summed by (stream, name).  The main
stream is the one that runs the step's first kernel: filter, classification and the updated_T fold; the side stream runs the four
class folds of the summary.  The trace goes to a temporary directory.  Prints the card name and power limit, then one table per
stream (kernel, launches, total ms), largest first, and the busy time of each stream."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=50_000_000)
    ap.add_argument("--genes", type=int, default=60_000)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from lr2rmats_b200 import api, cabi

    anno, rr = bench.make_tables(args.genes)
    reads, sj = bench.make_dataset(anno, rr, args.reads, range(bench.N_CHROM), seed=3)
    fp, ep = cabi.FilterParams.default(), cabi.ExonParams.default()
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)
    ctx = api.Context(0)
    ctx.set_anno(anno.soa()); ctx.set_rm(rr); ctx.set_sj(sj)
    ctx.upload(reads.soa()); ctx.sync()
    for _ in range(args.warmup):
        ctx.pipeline_run(fp, ep); ctx.update_run(up); ctx.sync()
    torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as tmp:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ctx.pipeline_run(fp, ep); ctx.update_run(up); ctx.sync()
        path = os.path.join(tmp, "step.pt.trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    kernels = [e for e in events if e.get("cat") == "kernel"]
    if not kernels:
        raise SystemExit("the trace holds no kernels")
    main_stream = min(kernels, key=lambda e: e["ts"])["args"]["stream"]
    per = defaultdict(lambda: [0, 0.0])
    busy = defaultdict(float)
    for e in kernels:
        s = "main" if e["args"]["stream"] == main_stream else f"side (stream {e['args']['stream']})"
        per[(s, e["name"])][0] += 1
        per[(s, e["name"])][1] += e["dur"] / 1e3
        busy[s] += e["dur"] / 1e3
    print(f"card: {card()}")
    print(f"configs[3]: {args.reads} primaries, {reads.n} records, one step after {args.warmup} warm-up steps, device resident")
    for s in sorted(busy, key=lambda s: (s != "main", s)):
        print(f"\n[{s}] kernel time {busy[s]:.2f} ms")
        rows = sorted(((n, c, t) for (ss, n), (c, t) in per.items() if ss == s), key=lambda r: -r[2])
        for n, c, t in rows:
            print(f"  {t:9.3f} ms  {c:4d}x  {n}")
    ctx.close()


if __name__ == "__main__":
    main()
