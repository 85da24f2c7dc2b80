"""Driver of the sharded multi-GPU run (one process per GPU): the host-side logic above the C ABI's multi-GPU layer.

    cuts = plan_shards(batch, world)            # same on every rank: locus-aligned, qname-run-safe, balanced by CIGAR ops
    ctx.comm_init(id, rank, world)              # id = api.comm_id() on rank 0, shipped by the launcher (torch.distributed, a file, MPI)
    ctx.tables_broadcast(0, anno, rm, sj)       # rank 0 passes the tables, the others None
    res = run_shard(ctx, shard_soa, name_base, fp, ep, up)   # rank 0: the merged result; others: None
    res = run_shard(..., reads=True)            # + res["reads"]: the per-read results (update-gtf -a/-A/-k/-v/-u, filter's records)

Everything numeric happens in the CUDA library; this file only slices arrays and orders calls.
"""
from __future__ import annotations

import numpy as np

from . import api

_REF_OPS = np.zeros(16, bool); _REF_OPS[[0, 2, 3, 7, 8]] = True      # M D N = X consume the reference (bam_cigar2rlen, htslib/sam.c:334)


def ref_span(batch: dict) -> np.ndarray:
    """(start, end) 1-based inclusive reference span per record, from pos + the reference-consuming CIGAR ops."""
    off = np.asarray(batch["cigar_off"]).astype(np.int64)
    cig = np.asarray(batch["cigar"])
    n = len(off) - 1
    consumed = np.where(_REF_OPS[cig & 15], (cig >> 4).astype(np.int64), 0)
    cs = np.zeros(len(cig) + 1, np.int64); np.cumsum(consumed, out=cs[1:])
    rlen = cs[off[1:]] - cs[off[:-1]]
    start = np.asarray(batch["pos"]).astype(np.int64) + 1
    return start[:n], start[:n] + np.maximum(rlen, 1) - 1


def plan_shards(batch: dict, n_shards: int) -> np.ndarray:
    """Cut positions (n_shards + 1) into ONE (tid,start)-sorted, name-grouped record stream.  A cut is placed only where the
    record starts beyond every earlier end on its chromosome (loci are independent, SURVEY App. B.3) and never inside a
    qname run (bam_filter.c:129-159 compares neighbours); shards are balanced by CIGAR ops + a per-record constant."""
    start, end = ref_span(batch)
    qh = np.asarray(batch["qname_hash"])
    n = len(start)
    if n:
        head = np.ones(n, bool); head[1:] = qh[1:] != qh[:-1]
        head_idx = np.maximum.accumulate(np.where(head, np.arange(n), 0))
        start = start[head_idx]                      # a record inside a qname run inherits the run head's start: never "beyond"
    off = np.asarray(batch["cigar_off"]).astype(np.int64)
    weight = np.diff(off) + 16
    return api.shard_cuts(batch["tid"], start.astype(np.int32), end.astype(np.int32), n_shards, weight=weight)


def take_shard(batch: dict, lo: int, hi: int) -> dict:
    off = np.asarray(batch["cigar_off"]).astype(np.int64)
    d = {k: np.ascontiguousarray(np.asarray(batch[k])[lo:hi]) for k in ("tid", "pos", "flag", "l_qseq", "nm", "xs", "qname_hash")}
    d["cigar_off"] = (off[lo:hi + 1] - off[lo]).astype(np.uint64)
    d["cigar"] = np.ascontiguousarray(np.asarray(batch["cigar"])[off[lo]:off[hi]])
    return d


def take_rows(batch: dict, idx) -> dict:
    """Sub-batch of the records idx (in that order), e.g. filter's kept records."""
    idx = np.asarray(idx, np.int64)
    off = np.asarray(batch["cigar_off"]).astype(np.int64)
    d = {k: np.ascontiguousarray(np.asarray(batch[k])[idx]) for k in ("tid", "pos", "flag", "l_qseq", "nm", "xs", "qname_hash")}
    lens = off[idx + 1] - off[idx]
    o = np.zeros(len(idx) + 1, np.int64); np.cumsum(lens, out=o[1:])
    src = np.repeat(off[idx] - o[:-1], lens) + np.arange(o[-1])
    d["cigar_off"] = o.astype(np.uint64); d["cigar"] = np.ascontiguousarray(np.asarray(batch["cigar"])[src])
    return d


def run_shard(ctx: api.Context, shard: dict | None, name_base: int, fp, ep, up, filtered: bool = True, fetch: bool = True,
              reads: bool = False):
    """One rank's part: upload, (filter +) CIGAR walk, update, gather to rank 0.  Returns the merged result on rank 0.
    reads: also gather the per-read results; rank 0's result then has them under "reads" (Context.gather_fetch_reads)."""
    if shard is not None:
        ctx.upload(shard)
    if filtered:
        ctx.pipeline_run(fp, ep)
    else:
        ctx.exon_run(ep)
    ctx.update_run(up)
    try:
        ctx.update_gather(name_base)
    finally:
        if reads:                                   # collective: every rank joins it, also where the root's table gather failed
            ctx.update_gather_reads(name_base)
    if not fetch:
        return None
    res = ctx.gather_fetch()
    if reads:
        res["reads"] = ctx.gather_fetch_reads(want_filter=filtered)
    return res
