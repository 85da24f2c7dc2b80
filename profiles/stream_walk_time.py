"""Time of the CIGAR walk with the pool resident (lrb_batch_upload + lrb_pipeline_run) against the pool streamed from pinned host
memory (lrb_batch_attach + lrb_pipeline_run) at several chunk sizes, on bench.py's configs[2] shape (ONT-like reads, 60 k genes).

    python profiles/stream_walk_time.py [--reads 10000000] [--steps 3] [--warmup 1] [--out FILE]

Every column of the batch lives in pinned memory (lrb_host_alloc), so the copies can overlap the walk.  Every timed window starts after a device
synchronise and is measured twice: CUDA events on the context stream (lrb_mark / lrb_elapsed_ms) and a host clock that stops after
the final synchronise.  Also timed alone: the upload (every column, pool included) and the pipeline pass over the resident batch, so
the streamed pass can be set against its two bounds, the H2D copy of the pool and the walk.  The filter / exon results of every
streamed run are checked against the resident run.  Prints one JSON line with the card name and power limit."""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def pinned_copy(L, a):
    """a in pinned host memory (freed by the caller with lrb_host_free)."""
    p = L.lrb_host_alloc(a.nbytes)
    if not p:
        raise MemoryError(f"lrb_host_alloc({a.nbytes}) failed")
    v = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(a.nbytes,)).view(a.dtype)
    v[:] = a
    return p, v


def digest(ctx):
    """sha1 of the filter and exon results (score only where the record passes: it is undefined elsewhere)."""
    f, e = ctx.filter_fetch(), ctx.exon_fetch()
    h = hashlib.sha1()
    for x in [f["pass_"], np.where(f["pass_"].astype(bool), f["score"], 0), f["keep_idx"]] + [e[k] for k in ("tid", "is_rev", "exon_off", "exon_start", "exon_end")]:
        h.update(np.ascontiguousarray(x).tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000, help="ONT-like primaries (bench.py --c2-reads)")
    ap.add_argument("--genes", type=int, default=60_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--chunks", default="0,67108864,16777216,4194304,1048576", help="chunk sizes in ops (0: the library's choice)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from lr2rmats_b200 import api, cabi
    fp, ep = cabi.FilterParams.default(), cabi.ExonParams.default()
    anno, rr = bench.make_tables(args.genes)
    reads, sj = bench.make_dataset(anno, rr, args.reads, range(bench.N_CHROM), seed=3, ont=True)
    L = api.load_library()
    pinned = {k: pinned_copy(L, np.ascontiguousarray(v)) for k, v in reads.soa().items()}
    soa = {k: v for k, (_, v) in pinned.items()}
    n_ops = int(reads.cigar_off[-1])
    ctx = api.Context(0)
    ctx.set_rm(rr)

    def timed(fn):
        ms, wall = [], []
        for it in range(args.warmup + args.steps):
            ctx.sync()
            t0 = time.perf_counter(); ctx.mark(0)
            fn()
            ctx.mark(1); ctx.sync(); t1 = time.perf_counter()
            if it >= args.warmup:
                ms.append(ctx.elapsed_ms(0, 1)); wall.append((t1 - t0) * 1e3)
        return dict(event_ms=round(float(np.mean(ms)), 3), event_ms_min=round(float(np.min(ms)), 3), wall_ms=round(float(np.mean(wall)), 3))

    res = {"card": card(), "reads": int(reads.n), "cigar_ops": n_ops, "pool_bytes": 4 * n_ops, "ops_per_read": round(n_ops / reads.n, 1),
           "steps": args.steps, "warmup": args.warmup}
    res["upload"] = timed(lambda: ctx.upload(soa))
    res["pipeline_resident"] = timed(lambda: ctx.pipeline_run(fp, ep))
    res["upload_pipeline"] = timed(lambda: (ctx.upload(soa), ctx.pipeline_run(fp, ep)))
    ref = digest(ctx)
    res["upload_GBs"] = round(sum(v.nbytes for v in soa.values()) / (res["upload"]["event_ms"] * 1e-3) / 1e9, 2)
    res["attach_pipeline"] = {}
    for k in (int(x) for x in args.chunks.split(",")):
        r = timed(lambda: (ctx.attach(soa, k), ctx.pipeline_run(fp, ep)))
        r.update(ctx.cigar_stream_diag())
        r["same_as_resident"] = digest(ctx) == ref
        res["attach_pipeline"][str(k)] = r
    ctx.close()
    for p, _ in pinned.values():
        L.lrb_host_free(p)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
