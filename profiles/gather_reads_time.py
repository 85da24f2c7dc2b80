"""Time of the per-read gather of a sharded run: lrb_update_gather_reads (count all-gather, compaction of the rank's exon chains,
gatherv to rank 0, rebase on the root) and lrb_gather_fetch_reads (device-to-host copy of the gathered per-read results on rank 0).

Run under torchrun, one process per GPU:
    torchrun --nproc_per_node N profiles/gather_reads_time.py [--reads 50000000] [--steps 5] [--warmup 2]
The data set is bench.py's configs[3] (--reads primaries over 24 chromosomes, Iso-Seq-like), sharded by chromosome the way
bench.py does it: rank r generates and owns the r-th contiguous block of chromosomes.  Each rank runs filter + bam2gtf + update-gtf
on its shard once and the table gather (lrb_update_gather, whose BED rows / counters the fetch returns); then every step times
the two calls separately, each with a host clock between a barrier and the call's return (both end in a stream synchronise).
Rank 0 prints one JSON line with the card name and power limit."""
import argparse
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=50_000_000)
    ap.add_argument("--genes", type=int, default=60_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    rank, world, local_rank = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    import torch
    import torch.distributed as dist
    from lr2rmats_b200 import api, cabi
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    anno, rr = bench.make_tables(args.genes)
    chroms = list(range(bench.N_CHROM * rank // world, bench.N_CHROM * (rank + 1) // world))
    reads, sj_part = bench.make_dataset(anno, rr, args.reads, chroms, seed=3, procs=max(1, (os.cpu_count() or 1) // world))
    sj = bench.gather_sj(dist, torch, sj_part, world)
    ns = [torch.zeros(1, device="cuda", dtype=torch.int64) for _ in range(world)]
    dist.all_gather(ns, torch.tensor([reads.n], device="cuda", dtype=torch.int64))
    name_base = int(sum(int(x) for x in ns[:rank]))

    ctx = api.Context(local_rank)
    idt = torch.zeros(api.COMM_ID_BYTES, dtype=torch.uint8, device="cuda")
    if rank == 0:
        idt.copy_(torch.frombuffer(bytearray(api.comm_id()), dtype=torch.uint8))
    dist.broadcast(idt, 0)
    ctx.comm_init(bytes(idt.cpu().numpy().tobytes()), rank, world)
    ctx.tables_broadcast(0, *((anno.soa(), rr, sj) if rank == 0 else (None, None, None)))
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)
    ctx.upload(reads.soa())
    ctx.pipeline_run(cabi.FilterParams.default(), cabi.ExonParams.default())
    ctx.update_run(up)
    ctx.update_gather(name_base)

    def timed(f):
        dist.barrier(); torch.cuda.synchronize()
        t = time.perf_counter(); f(); return (time.perf_counter() - t) * 1e3

    t_gather, t_fetch = [], []
    for i in range(args.warmup + args.steps):
        g = timed(lambda: ctx.update_gather_reads(name_base))
        f = timed(lambda: ctx.gather_fetch_reads(raw=True))
        if i >= args.warmup:
            t_gather.append(g); t_fetch.append(f)
    if rank == 0:
        r = ctx.gather_fetch_reads(); u, fl = r["update"], r["filter"]
        n_rows, n_exon = u["ex"]["n_reads"], len(u["ex"]["exon_start"])
        moved = sum(a.nbytes for d in (u, u["ex"], u["novel"], u["updated"], fl) for a in d.values() if isinstance(a, np.ndarray) and a.ndim == 1)
        print(json.dumps(dict(card=card(), world=world, records=int(len(fl["pass_"])), rows=int(n_rows), exons=int(n_exon),
                              fetched_bytes=int(moved), steps=args.steps, warmup=args.warmup,
                              gather_reads_ms=dict(mean=float(np.mean(t_gather)), min=float(np.min(t_gather)), max=float(np.max(t_gather))),
                              fetch_reads_ms=dict(mean=float(np.mean(t_fetch)), min=float(np.min(t_fetch)), max=float(np.max(t_fetch))))), flush=True)
    ctx.comm_destroy(); ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
