"""Time of the filter stage (lrb_filter_run) on a resident batch: bench.py's configs[1] shape (1 M Iso-Seq-like reads), its configs[2]
shape (10 M ONT-like reads), and an adversarial batch of 10 M records of which only every 10 000th can pass (ten copies of the
configs[1] batch, all records but every 10 000th made unmapped with FLAG 4): there each passing record's qname-run selection walks
back over 10 000 failing records to find its run predecessor.

    python profiles/filter_stage_time.py [--steps 10] [--warmup 3] [--rounds 2] [--lib LABEL=PATH ...] [--out FILE]

--lib names a build of liblr2rmats_b200.so (default: this tree's); with several, the rounds alternate between them on the same data
in one process, so that two versions of the library are compared under the same conditions.  The batch is uploaded once per library
and round, outside the timed window.  Every timed window starts after a device synchronise and an L2 flush (a 256 MiB write, untimed)
and is measured twice: CUDA events on the context stream (lrb_mark / lrb_elapsed_ms) and a host clock that stops after the final
synchronise.  Per library the kernel launches of one filter_run and a digest of its result are reported, so that the versions can be
checked to compute the same.  Prints one JSON line with the card name and power limit."""
import argparse
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


_libs = {}


def context_on(path):
    """A context of the library at `path` (loaded once, its prototypes declared by api.load_library)."""
    from lr2rmats_b200 import api
    saved = api._lib, api.LIB_PATH
    api._lib, api.LIB_PATH = _libs.get(path), path
    try:
        _libs[path] = api.load_library()
        return api.Context(0)
    finally:
        api._lib, api.LIB_PATH = saved


def digest(f):
    """sha1 of a filter result (score / intron_n only where the record passes: they are undefined elsewhere)."""
    m = f["pass_"].astype(bool)
    h = hashlib.sha1()
    for x in (f["pass_"], np.where(m, f["score"], 0), np.where(m, f["intron_n"], 0), f["keep_idx"]):
        h.update(np.ascontiguousarray(x).tobytes())
    return h.hexdigest()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--lib", action="append", default=[], metavar="LABEL=PATH")
    ap.add_argument("--c1-reads", type=int, default=1_000_000)
    ap.add_argument("--c2-reads", type=int, default=10_000_000)
    ap.add_argument("--genes", type=int, default=60_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    libs = dict(s.split("=", 1) for s in args.lib) or {"this": os.path.join(ROOT, "lr2rmats_b200", "csrc", "liblr2rmats_b200.so")}
    import torch
    from lr2rmats_b200 import cabi, synth
    fp = cabi.FilterParams.default()
    anno, rr = bench.make_tables(args.genes)
    c1, _ = bench.make_dataset(anno, rr, args.c1_reads, range(bench.N_CHROM), seed=3, ont=False)
    adv = synth.concat_reads([c1] * 10)
    adv.flag = np.where(np.arange(adv.n) % 10_000 == 0, adv.flag, adv.flag | 4).astype(np.uint16)
    c2, _ = bench.make_dataset(anno, rr, args.c2_reads, range(bench.N_CHROM), seed=3, ont=True)
    batches = {"configs[1] (Iso-Seq-like)": c1, "configs[2] (ONT-like)": c2, "adversarial (1 in 10 000 can pass)": adv}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")

    res = {"card": card(), "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds, "libs": libs,
           "l2": "flushed before every timed window (256 MiB write, untimed)", "configs": {}}
    for name, reads in batches.items():
        soa = reads.soa()
        r = res["configs"][name] = {"reads": int(reads.n), "cigar_ops_per_read": round(int(reads.cigar_off[-1]) / reads.n, 1)}
        for rnd in range(args.rounds):
            for label, path in libs.items():
                ctx = context_on(path)
                ctx.set_rm(rr); ctx.upload(soa); ctx.sync()
                ms, wall = [], []
                for it in range(args.warmup + args.steps):
                    flush.fill_(1); torch.cuda.synchronize(0); ctx.sync()
                    t0 = time.perf_counter(); ctx.mark(0)
                    ctx.filter_run(fp)
                    ctx.mark(1); ctx.sync(); t1 = time.perf_counter()
                    if it >= args.warmup:
                        ms.append(ctx.elapsed_ms(0, 1)); wall.append((t1 - t0) * 1e3)
                l0 = ctx.launch_count(); ctx.filter_run(fp); launches = ctx.launch_count() - l0
                f = ctx.filter_fetch()
                out = r.setdefault(label, {"event_ms": [], "event_ms_min": [], "wall_ms": []})
                out["event_ms"].append(round(float(np.mean(ms)), 3)); out["event_ms_min"].append(round(float(np.min(ms)), 3))
                out["wall_ms"].append(round(float(np.mean(wall)), 3))
                out.update(launches=int(launches), digest=digest(f), passing=int(f["pass_"].sum()), kept=int(len(f["keep_idx"])))
                ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
