#!/usr/bin/env python
"""bench.py -- alignments/sec through filter + bam2gtf + update-gtf (BASELINE.json's metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--reads R] [--genes G] [--shape iso|ont] [--dump-outputs DIR]

Workload (the same ONE data set for every N: strong scaling): BASELINE.json configs[3] -- R synthetic spliced alignments
(default 50 M primaries, Iso-Seq-like as configs[1], + secondaries / rRNA / low-identity / low-coverage rejects) against a
60 k-gene / ~200 k-transcript annotation with a STAR SJ.out.tab table (short-read validation of novel junctions) and an rRNA
remove table, "sharded by chromosome": the 24 chromosomes are dealt to the N ranks as N contiguous blocks of the coordinate-sorted
stream (every rank generates only its own block; a block boundary is a locus gap, SURVEY App. B.3).

A step = the whole job once: every rank runs the fused filter + CIGAR walk (`lrb_pipeline_run`) and classification / SJ support /
split / merge fold / summary sets (`lrb_update_run`) on its shard, then `lrb_update_gather` sends the per-shard updated_T tables, BED
rows and known-gene pairs to rank 0 over NCCL and merges them canonically there (ordered concatenation, gene sets recomputed over
the gathered table, counters summed) -- the gather and the merge are INSIDE the timed region.  At N = 1 there is nothing to gather.

  value     device-resident: the shard is in HBM when the timed region starts; CUDA events on the library stream, L2 flushed
            (untimed) between steps, K steps, max over ranks; value = all alignments of the data set / that time.
  e2e       the same step from HOST buffers: pinned H2D of the shard + the stages + gather/merge + D2H of the merged result
            (updated table, BED rows, summary, kept-record list) to host memory; wall clock, max over ranks.
  roofline  dominant kernel: algorithmic bytes per launch / its CUDA-event duration vs MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline, files_e2e (N = 1): the UNMODIFIED reference binary (oracle/_ref/lr2rmats), one thread, on a bounded sample of the
            same stream, and the drop-in CLI on the same files (wall clock files in -> files out, outputs compared byte for byte).
  other_configs (N = 1): configs[1] (1 M Iso-Seq-like) and configs[2] (10 M ONT-like, indel-dense CIGARs) device-resident.

--dump-outputs DIR: after the device-resident steps, what the last one computed is written as DIR/<name>.npy (see dump_outputs), so
that two builds run with the same arguments (hence the same seeded data set) can be compared output for output.

--impl reference: the reference's own CPU implementation (its CLI, unmodified binary) on the host cores: one process per
locus-aligned shard of a bounded sample of the same stream, all cores.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "long-read alignments/sec filter+bam2gtf+update-gtf"
UNIT = "alignments/s"
N_CHROM = 24


_T0 = time.time()


def log(*a):
    print(f"[{time.time() - _T0:7.1f}s]", *a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------- workload
def make_tables(n_genes):
    from lr2rmats_b200 import synth
    anno = synth.make_annotation(n_genes, n_chrom=N_CHROM, seed=1)
    rr = synth.make_rrna(anno, 2000 if n_genes >= 20000 else max(10, n_genes // 30), seed=2)
    return anno, rr


def make_workload(n_reads, n_genes, seed, ont=False):
    """One batch drawn over the whole annotation at once (tests and profiling drivers; the bench itself builds its data set per chromosome)."""
    from lr2rmats_b200 import synth
    anno, rr = make_tables(n_genes)
    return anno, rr, synth.make_reads(anno, n_reads, seed=seed, ont=ont, reject_frac=0.2, rrna=rr)


def make_sj_table(reads, ep=None, frac=0.7, seed=5):
    """SJ.out.tab rows from the read-derived junctions (N ops of at least min_intron bases)."""
    from lr2rmats_b200 import synth
    return synth.make_sj_from_reads(reads, frac=frac, seed=seed, min_intron=ep.min_intron if ep is not None else 3)


_G = {}


def _chrom_task(task):
    """One chromosome of the data set: reads + the SJ rows its junctions give (pool worker; the annotation is inherited by fork)."""
    from lr2rmats_b200 import synth
    c, n, seed, ont = task
    r = synth.make_reads(_G["anno"], n, seed=seed + 7919 * c, ont=ont, reject_frac=0.2, rrna=_G["rr"], chrom=c, qid_base=c * (1 << 32))
    sj = synth.make_sj_from_reads(r, frac=0.7, seed=seed + 31 * c + 5)
    return c, r, sj


def make_dataset(anno, rr, total_reads, chroms, seed=3, ont=False, procs=None):
    """Reads of the chromosomes `chroms` (total_reads is the size of the WHOLE 24-chromosome data set) + their SJ rows."""
    from lr2rmats_b200 import synth
    import multiprocessing as mp
    per = np.full(N_CHROM, total_reads // N_CHROM); per[: total_reads % N_CHROM] += 1
    tasks = [(int(c), int(per[c]), seed, ont) for c in chroms]
    procs = max(1, min(len(tasks), procs or (os.cpu_count() or 1)))
    _G["anno"], _G["rr"] = anno, rr
    if procs > 1 and total_reads >= 200_000:
        with mp.get_context("fork").Pool(procs) as pool:
            parts = sorted(pool.map(_chrom_task, tasks, chunksize=1), key=lambda x: x[0])
    else:
        parts = [_chrom_task(t) for t in tasks]
    reads = synth.concat_reads([p[1] for p in parts])
    sj = {k: np.concatenate([p[2][k] for p in parts]) for k in ("tid", "don", "acc", "uniq_c", "multi_c")}
    return reads, sj


def algorithmic_bytes(n_records, n_ops, n_exons_rows):
    """SURVEY.md 8(d): 53 + 4c + 13e bytes per alignment (c CIGAR ops, e exons)."""
    return 53 * int(n_records) + 4 * int(n_ops) + 13 * int(n_exons_rows)


def locus_cuts(reads, n_parts, lo=0, hi=None):
    """numpy restatement of the locus-gap rule for the reference arm (which must not load the CUDA library): cut positions in
    [lo, hi) where a record starts beyond every earlier end on its chromosome and does not continue a qname run."""
    hi = reads.n if hi is None else hi
    off = reads.cigar_off.astype(np.int64); cig = reads.cigar
    op = cig[off[lo]:off[hi]] & 15
    consumed = np.where((op == 0) | (op == 2) | (op == 3) | (op == 7) | (op == 8), (cig[off[lo]:off[hi]] >> 4).astype(np.int64), 0)
    cs = np.zeros(len(consumed) + 1, np.int64); np.cumsum(consumed, out=cs[1:])
    o = off[lo:hi + 1] - off[lo]
    start = reads.pos[lo:hi].astype(np.int64) + 1
    end = start + np.maximum(cs[o[1:]] - cs[o[:-1]], 1) - 1
    key_s = ((reads.tid[lo:hi].astype(np.int64) + 1) << 32) | start
    key_e = ((reads.tid[lo:hi].astype(np.int64) + 1) << 32) | end
    before = np.concatenate([[0], np.maximum.accumulate(key_e)[:-1]])
    ok = key_s > before
    ok[1:] &= reads.qname_hash[lo + 1:hi] != reads.qname_hash[lo:hi - 1]
    cand = np.nonzero(ok)[0]
    cuts = [0]
    for k in range(1, n_parts):
        want = (hi - lo) * k // n_parts
        j = np.searchsorted(cand, want)
        c = int(cand[j]) if j < len(cand) else hi - lo
        cuts.append(max(c, cuts[-1]))
    cuts.append(hi - lo)
    return [lo + c for c in cuts]


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.p, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.p:
            self.p.terminate()
            try:
                self.p.wait(timeout=3)
            except Exception:
                self.p.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------- reference (CPU) arm
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "lr2rmats")
CLI_BIN = os.path.join(ROOT, "lr2rmats_b200", "host", "lr2rmats-b200")
UPD_ARGS = "-s -l 3 -J 1 -j sj.tab"


def write_inputs(anno, rr, reads, sj, workdir, cuts):
    """The reference's input files (SAM text with SEQ, GTFs, SJ.out.tab): one SAM per [cuts[k], cuts[k+1]) slice of the stream."""
    from lr2rmats_b200 import synth
    synth.write_gtf(os.path.join(workdir, "anno.gtf"), anno)
    synth.write_rm_gtf(os.path.join(workdir, "rm.gtf"), rr, anno.chrom_names)
    synth.write_sj(os.path.join(workdir, "sj.tab"), sj, anno.chrom_names)
    for k in range(len(cuts) - 1):
        synth.write_sam(os.path.join(workdir, f"in{k}.sam"), reads.take(np.arange(cuts[k], cuts[k + 1])), with_seq=True)


def run_cli(binary, workdir, n_parts, tag):
    """filter -> update-gtf (pass 2: -s -l 3 -J 1 -j SJ, with summary and BED) through a CLI, one process per slice.  Wall seconds."""
    script = ("set -e; cd {w}; {b} filter -r rm.gtf in{k}.sam > {t}f{k}.bam 2>/dev/null; "
              "{b} update-gtf " + UPD_ARGS + " {t}f{k}.bam anno.gtf -y {t}s{k}.txt -E {t}e{k}.bed -o {t}u{k}.gtf 2>/dev/null")
    t0 = time.perf_counter()
    procs = [subprocess.Popen(["bash", "-c", script.format(w=workdir, b=binary, k=k, t=tag)]) for k in range(n_parts)]
    rcs = [p.wait() for p in procs]
    dt = time.perf_counter() - t0
    if any(rcs):
        raise RuntimeError(f"{binary} failed: {rcs}")
    return dt


def sample_of_stream(args, n_sample, ont=False):
    """A bounded sample of the bench workload: the first ~n_sample records of chromosome 1 of the SAME data set (same depth, same
    annotation, same SJ table rows of that chromosome), ending at a locus gap."""
    anno, rr = make_tables(args.genes)
    per_chrom = args.reads // N_CHROM
    reads, sj = make_dataset(anno, rr, args.reads, [0], seed=3, ont=ont, procs=1)
    if reads.n > n_sample:
        cuts = locus_cuts(reads, max(2, int(round(reads.n / n_sample))))
        reads = reads.take(np.arange(0, cuts[1]))
    return anno, rr, reads, sj, per_chrom


def workload_name(args, n_total=None, n_ops=None):
    shape = "ONT-like (indel-dense CIGARs)" if args.shape == "ont" else "Iso-Seq-like"
    return (f"configs[3]: {args.reads} {shape} primary alignments (+ secondaries and 20 % filter rejects) vs {args.genes} genes, STAR SJ table, rRNA table; "
            f"filter(-v .67 -q .75 -s .98 -r) + bam2gtf + update-gtf {UPD_ARGS.replace(' sj.tab', '')} with summary/BED; ONE data set sharded by chromosome over the ranks")


def bench_reference(args, rank, world):
    if rank != 0:
        return
    if not (os.path.isfile(REF_BIN) and os.access(REF_BIN, os.X_OK)):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/lr2rmats was not built in the build container"}))
        return
    anno, rr, reads, sj, _ = sample_of_stream(args, args.ref_reads, ont=(args.shape == "ont"))
    cores = os.cpu_count() or 1
    cuts = locus_cuts(reads, cores)
    cuts = sorted(set(cuts)); used = len(cuts) - 1
    times = []
    wd = tempfile.mkdtemp(prefix="lrb_ref_")
    try:
        write_inputs(anno, rr, reads, sj, wd, cuts)
        for it in range(args.warmup + args.steps):
            dt = run_cli(REF_BIN, wd, used, "r")
            if it >= args.warmup:
                times.append(dt)
    finally:
        shutil.rmtree(wd, ignore_errors=True)
    ms = 1e3 * float(np.mean(times))
    val = reads.n / (ms / 1e3)
    sample = (f"first {reads.n} records of chromosome 1 of the same data set ({len(sj['tid'])} SJ rows), cut at locus gaps into {used} shards, one unmodified "
              f"reference process (`filter` | `update-gtf {UPD_ARGS}` -y -E -o, SAM text with SEQ in) per shard on {used} of {cores} cores")
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
           "config": {"workload": workload_name(args), "sample_reads": int(reads.n), "sample": sample},
           "cpu_baseline": {"value": val, "unit": UNIT, "cores": used, "kind": "reference", "sample": sample},
           "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "files_e2e": {"value": val, "unit": UNIT, "seconds": ms / 1e3, "what": "wall clock, SAM / GTF / SJ files in -> BAM, updated GTF, BED, summary files out"},
           "gpu_launches": 0}
    print(json.dumps(out))


# --------------------------------------------------------------------------------------------------- our arm
def pinned_copy(arr):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
    return t, t.numpy()


DUMP_CAP = 1 << 18          # elements per dumped array: the 21 arrays stay below 64 MiB of float64


def dump_outputs(out_dir, res, keep_idx):
    """The arrays a caller of the timed step receives -- the updated_T table (table_*), the BED rows (bed_*), the summary counters and
    filter's kept-record list -- as float64 .npy files (every value is an integer below 2^53, so it is stored exactly).  An array longer
    than DUMP_CAP is replaced by its elements at DUMP_CAP sorted positions drawn with its length as the seed: two runs whose arrays have
    the same length dump the same positions."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"summary": res["summary"], "keep_idx": keep_idx}
    arrays.update({f"table_{k}": v for k, v in res["table"].items()})
    arrays.update({f"bed_{k}": v for k, v in res["bed"].items()})
    for name, a in arrays.items():
        a = np.asarray(a)
        if len(a) > DUMP_CAP:
            a = a[np.sort(np.random.default_rng(len(a)).choice(len(a), DUMP_CAP, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a.astype(np.float64))


def gather_sj(dist, torch, sj, world):
    """Every rank made the SJ rows of its own chromosomes: all-gather them (plumbing) so that rank 0 holds the whole table."""
    if dist is None:
        return sj
    rows = np.stack([sj[k].astype(np.int32) for k in ("tid", "don", "acc", "uniq_c", "multi_c")], 1) if len(sj["tid"]) else np.zeros((0, 5), np.int32)
    n = torch.tensor([len(rows)], device="cuda", dtype=torch.int64)
    ns = [torch.zeros(1, device="cuda", dtype=torch.int64) for _ in range(world)]
    dist.all_gather(ns, n)
    ns = [int(x) for x in ns]; mx = max(max(ns), 1)
    buf = torch.zeros((mx, 5), device="cuda", dtype=torch.int32); buf[: len(rows)] = torch.from_numpy(rows).cuda()
    bufs = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(bufs, buf)
    allr = np.concatenate([b[:k].cpu().numpy() for b, k in zip(bufs, ns)], 0)
    return dict(tid=allr[:, 0].copy(), don=allr[:, 1].copy(), acc=allr[:, 2].copy(), uniq_c=allr[:, 3].copy(), multi_c=allr[:, 4].copy())


def resident_config(ctx, api, cabi, torch, dev, n_reads, n_genes, ont, steps, warmup, flush, peak):
    """One of the single-GPU configs of BASELINE.json, device resident: ms per step, alignments/s, scan-kernel roofline."""
    fp, ep = cabi.FilterParams.default(), cabi.ExonParams.default()
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)
    anno, rr = make_tables(n_genes)
    reads, sj = make_dataset(anno, rr, n_reads, range(N_CHROM), seed=3, ont=ont)
    ctx.set_anno(anno.soa()); ctx.set_rm(rr); ctx.set_sj(sj)
    ctx.upload(reads.soa()); ctx.sync(); ctx.timing(True)
    times, scan, stages = [], [], []
    for it in range(warmup + steps):
        flush.fill_(1); torch.cuda.synchronize(dev)
        ctx.mark(0); ctx.pipeline_run(fp, ep); s1 = ctx.timing_get()[0]; ctx.update_run(up); ctx.mark(1)
        if it >= warmup:
            times.append(ctx.elapsed_ms(0, 1)); scan.append(s1["k_scan"]); stages.append(ctx.timing_get()[0])
    ms = float(np.mean(times)); ks = float(np.mean(scan))
    r = ctx.update_fetch_table(want_bed=False)
    n_ops = int(reads.cigar_off[-1])
    ne = int(r["table"]["exon_off"][-1]) if len(r["table"]["cov"]) else 0
    scan_bytes = reads.n * 40 + 4 * n_ops
    st = {k: round(float(np.mean([s[k] for s in stages])), 4) for k in ("classify", "merge", "summary", "k_fold")}
    return {"reads": int(reads.n), "cigar_ops_per_read": round(n_ops / reads.n, 1), "ms_per_step": ms, "value": reads.n / (ms * 1e-3), "unit": UNIT,
            "updated_transcripts": len(r["table"]["cov"]), "updated_exons": ne, "stage_ms": dict(st, k_scan=round(ks, 4)),
            "scan_kernel": {"ms": ks, "algorithmic_bytes": int(scan_bytes), "achieved_GBs": scan_bytes / (ks * 1e-3) / 1e9, "frac": scan_bytes / (ks * 1e-3) / 1e9 / peak}}


def bench_ours(args, rank, world, local_rank):
    # the JSON line must be the only thing on stdout: libraries that print there (NCCL's version banner) go to stderr until the end
    sys.stdout.flush(); real_stdout = os.dup(1); os.dup2(2, 1)
    import torch
    from lr2rmats_b200 import api, cabi
    dist = None
    if world > 1:

        import torch.distributed as dist_
        dist = dist_
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = local_rank
    fp, ep = cabi.FilterParams.default(), cabi.ExonParams.default()
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)

    # ---- workload: ONE data set; rank r owns (and generates) the r-th block of chromosomes; rank 0's tables go to every GPU over NVLink
    t0 = time.time()
    anno, rr = make_tables(args.genes)
    chroms = list(range(N_CHROM * rank // world, N_CHROM * (rank + 1) // world))
    reads, sj_part = make_dataset(anno, rr, args.reads, chroms, seed=3, ont=(args.shape == "ont"), procs=max(1, (os.cpu_count() or 1) // world))
    sj = gather_sj(dist, torch, sj_part, world)
    ctx = api.Context(dev)
    name_base = 0
    if world > 1:
        idt = torch.zeros(api.COMM_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(api.comm_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        ctx.comm_init(bytes(idt.cpu().numpy().tobytes()), rank, world)
        if rank == 0:
            ctx.tables_broadcast(0, anno.soa(), rr, sj)          # ncclBroadcast HBM -> HBM: the other ranks never touch the tables on the host
        else:
            ctx.tables_broadcast(0, None, None, None)
        ns = [torch.zeros(1, device="cuda", dtype=torch.int64) for _ in range(world)]
        dist.all_gather(ns, torch.tensor([reads.n], device="cuda", dtype=torch.int64))
        name_base = int(sum(int(x) for x in ns[:rank]))
    else:
        ctx.set_anno(anno.soa()); ctx.set_rm(rr); ctx.set_sj(sj)
    n_ops = int(reads.cigar_off[-1])
    log(f"[rank {rank}] workload ready in {time.time() - t0:.1f}s: chromosomes {chroms[0] + 1}-{chroms[-1] + 1}, {reads.n} alignments, {n_ops} CIGAR ops, "
        f"{anno.n_trans} transcripts, {len(sj['tid'])} SJ rows")

    soa = reads.soa()
    keep, pinned = [], {}
    for k, v in soa.items():
        t, a = pinned_copy(v); keep.append(t); pinned[k] = a
    batch, bk = cabi.make_batch(pinned)
    h2d_bytes = int(sum(a.nbytes for a in pinned.values()))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{dev}")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev); ctx.sync()

    def step_resident():
        ctx.pipeline_run(fp, ep)
        ctx.update_run(up)
        if world > 1:
            ctx.update_gather(name_base)

    # ---- device-resident timing
    ctx.upload_struct(batch); ctx.sync()
    ctx.timing(True)
    for i in range(args.warmup):
        if i == 0:
            ctx.pipeline_run(fp, ep); ctx.sync(); log(f"[rank {rank}] first pipeline_run done: {ctx.timing_get()[0]}")
        step_resident(); ctx.sync()
        log(f"[rank {rank}] warm-up step {i} done: {ctx.timing_get()[0]}")
    clocks = ClockSampler(dev); clocks.start()
    times, stage_ms, gather_ms, launches = [], [], [], 0
    barrier()
    for _ in range(args.steps):
        flush.fill_(1); torch.cuda.synchronize(dev)           # L2 flush, untimed
        if dist is not None:
            dist.barrier()                                    # every rank enters the step together: the step time is the slowest rank's
        l0 = ctx.launch_count()
        ctx.mark(0)
        ctx.pipeline_run(fp, ep); s1 = ctx.timing_get()[0]
        ctx.update_run(up); s2 = ctx.timing_get()[0]
        if world > 1:
            ctx.update_gather(name_base)
        ctx.mark(1)
        times.append(ctx.elapsed_ms(0, 1))
        launches += ctx.launch_count() - l0
        stage_ms.append(dict(s2, filter=s1["filter"], k_scan=s1["k_scan"]))
        if world > 1:
            gather_ms.append(ctx.gather_timing())
    barrier()
    ms_step = float(np.mean(times))
    log(f"[rank {rank}] device-resident: {ms_step:.3f} ms/step")
    tb = ctx.update_fetch_table(want_bed=True)
    n_kept = int(ctx.filter_fetch_keep(raw=True)[0])
    ne_rows = None
    local_summary = tb["summary"].copy()
    n_upd_local, n_upd_exons_local = len(tb["table"]["cov"]), int(tb["table"]["exon_off"][-1]) if len(tb["table"]["cov"]) else 0
    merged = ctx.gather_fetch() if world > 1 else tb
    summary = merged["summary"].copy() if rank == 0 else local_summary
    n_upd_total = len(merged["table"]["cov"]) if rank == 0 else 0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, merged, ctx.filter_fetch_keep())
        log(f"[rank {rank}] outputs of the last timed step written to {args.dump_outputs}")
    del tb, merged

    # ---- end to end from HOST buffers: upload of the shard from pinned memory, the stages, gather + merge, and the merged
    # result (what `update-gtf -o -y -E` prints, plus filter's kept-record list) back in host memory.  At N = 1 `--e2e-contexts`
    # contexts (one stream + one host thread each) keep that many steps in flight, the way a multi-batch caller drives the library;
    # with a communicator per context that is not safe across ranks, so N > 1 runs one step at a time.
    def step_e2e(cx):
        cx.upload_struct(batch)
        cx.pipeline_run(fp, ep)
        cx.update_run(up)
        nk, _ = cx.filter_fetch_keep(raw=True)
        if world > 1:
            cx.update_gather(name_base)
            t, b, _s = cx.gather_fetch(raw=True)
        else:
            t, b, _s = cx.update_fetch_table(raw=True)
        nt = int(t.n); nte = int(t.exon_off[nt]) if nt else 0
        return int(nk * 4 + nt * (4 * 9 + 2) + 4 + nte * 8 + b.n * 18 + 19 * 4)

    ctx.timing(False)
    n_ctx = max(1, args.e2e_contexts) if world == 1 else 1
    ctxs = [ctx]
    for _ in range(n_ctx - 1):
        cx = api.Context(dev)
        cx.set_anno(anno.soa()); cx.set_rm(rr); cx.set_sj(sj)
        ctxs.append(cx)
    last = {}

    def worker(k, n_steps):
        for _ in range(n_steps):
            last[k] = step_e2e(ctxs[k])

    def run_e2e(n_steps):
        share = [n_steps // n_ctx + (1 if k < n_steps % n_ctx else 0) for k in range(n_ctx)]
        th = [threading.Thread(target=worker, args=(k, share[k])) for k in range(n_ctx) if share[k]]
        t1 = time.perf_counter()
        for x in th:
            x.start()
        for x in th:
            x.join()
        return 1e3 * (time.perf_counter() - t1)

    run_e2e(max(n_ctx, min(args.warmup, 3)))
    log(f"[rank {rank}] e2e warm-up done")
    flush.fill_(1); torch.cuda.synchronize(dev)
    barrier()
    e2e_total_ms = run_e2e(args.steps)
    barrier()
    log(f"[rank {rank}] e2e: {e2e_total_ms / args.steps:.3f} ms/step")
    d2h_bytes = last[0]
    e2e_ms = e2e_total_ms / args.steps
    for cx in ctxs[1:]:
        cx.sync(); cx.close()
    clk = clocks.stop()

    # ---- max over ranks, totals over ranks
    n_total, ops_total, kept_total = reads.n, n_ops, n_kept
    rank_ms = [ms_step]
    if dist is not None:
        t = torch.tensor([ms_step, e2e_ms], device="cuda", dtype=torch.float64)
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        rank_ms = [float(x[0]) for x in allt]
        ms_step, e2e_ms = max(float(x[0]) for x in allt), max(float(x[1]) for x in allt)
        cnt = torch.tensor([reads.n, launches, h2d_bytes, d2h_bytes, n_ops, n_kept, n_upd_exons_local], device="cuda", dtype=torch.int64); dist.all_reduce(cnt)
        n_total, launches, h2d_bytes, d2h_bytes, ops_total, kept_total, upd_exons_total = (int(x) for x in cnt)
    if rank != 0:
        if dist is not None:
            ctx.comm_destroy(); dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (rank 0's launches)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0)); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s"
    st = {k: float(np.mean([s[k] for s in stage_ms])) for k in stage_ms[0]}
    if gather_ms:
        st["gather"] = float(np.mean([g[0] for g in gather_ms])); st["root_merge"] = float(np.mean([g[1] for g in gather_ms]))
    # rows / exons of rank 0's shard: exon slots of the kept rows ~ updated exons are not the same thing; use the library's own counts
    ex = ctx.exon_fetch() if False else None
    ne_rank0 = int(round(7.2 * n_kept))                      # refined below from the fetched exon table when cheap
    try:
        r0 = ctx.update_fetch()
        ne_rank0 = int(r0["ex"]["exon_off"][-1]); n_novel_cand = len(r0["novel"]["read"]); del r0
    except Exception:
        n_novel_cand = n_kept
    # per-kernel algorithmic bytes (DESIGN.md section 4): scan reads 31 B/record + CIGAR, writes 9 B/record filter outputs,
    # 25 B/row + 8 B/exon; classify reads 21 B/row + 8 B/exon and writes 13 B/row + 1 B/exon; fold reads 28 B/candidate + 8 B/exon
    scan_bytes = reads.n * (31 + 9) + 4 * n_ops + n_kept * 25 + ne_rank0 * 8
    classify_bytes = n_kept * (21 + 13) + ne_rank0 * 9
    kernels = {"cigar_scan_kernel": (st["k_scan"], scan_bytes), "classify_row_kernel": (st["classify"], classify_bytes),
               "fold kernels (fold_prepare..fold_big/merge_fold)": (st["k_fold"], n_novel_cand * 28 + ne_rank0 * 8)}
    dom = max(kernels, key=lambda k: kernels[k][0])
    dms, dbytes = kernels[dom]
    achieved = dbytes / (dms * 1e-3) / 1e9 if dms > 0 else 0.0
    path_bytes = algorithmic_bytes(n_total, ops_total, ne_rank0 * (n_total / max(reads.n, 1)))
    traffic = traffic_note = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        tk = tj["kernels"].get(dom.split(" ")[0])
        if tk:                                        # measured on a smaller data set of the same shape: scaled to this launch by the record count
            traffic = int(tk["dram_bytes"] * reads.n / tj["reads"])
            traffic_note = f"ncu dram bytes of a {tj['reads']}-record capture ({tk.get('what', dom)}) scaled by records; see profiles/r02_traffic.json"
    except Exception:
        pass

    # ---- N = 1 extras: the reference binary and the drop-in CLI on a bounded sample (files in -> files out), configs[1] / configs[2]
    cpu = files = others = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            if os.path.isfile(REF_BIN) and os.access(REF_BIN, os.X_OK):
                a2, rr2, rd2, sj2, _ = sample_of_stream(args, args.cpu_reads, ont=(args.shape == "ont"))
                wd = tempfile.mkdtemp(prefix="lrb_cpu_")
                try:
                    write_inputs(a2, rr2, rd2, sj2, wd, [0, rd2.n])
                    dt = run_cli(REF_BIN, wd, 1, "r")
                    sample = f"first {rd2.n} records of chromosome 1 of the same data set ({len(sj2['tid'])} SJ rows)"
                    cpu = {"value": rd2.n / dt, "unit": UNIT, "cores": 1, "kind": "reference",
                           "sample": sample + f": unmodified reference `filter` | `update-gtf {UPD_ARGS}` -y -E -o, {dt:.1f} s wall, 1 thread"}
                    if os.path.isfile(CLI_BIN):
                        run_cli(CLI_BIN, wd, 1, "w")                       # first process on this box pays the CUDA start-up once
                        dt2 = run_cli(CLI_BIN, wd, 1, "o")
                        same = all(open(os.path.join(wd, f"r{x}0.{e}"), "rb").read() == open(os.path.join(wd, f"o{x}0.{e}"), "rb").read()
                                   for x, e in (("s", "txt"), ("e", "bed"), ("u", "gtf")))
                        files = {"value": rd2.n / dt2, "unit": UNIT, "seconds": dt2, "reference_seconds": dt, "speedup": dt / dt2, "outputs_identical": bool(same),
                                 "what": "wall clock of the drop-in CLI (lr2rmats-b200 filter | update-gtf), SAM / GTF / SJ files in -> BAM, updated GTF, BED, summary files out, "
                                         "CUDA context creation included; same files as cpu_baseline", "sample": sample}
                finally:
                    shutil.rmtree(wd, ignore_errors=True)
        except Exception as e:  # noqa: BLE001
            cpu = {"value": None, "unit": UNIT, "cores": 1, "kind": "reference", "sample": f"failed: {e}"}
    log("cpu_baseline / files_e2e legs done")
    if world == 1 and not args.no_other_configs:
        try:
            ctx.timing(True)
            others = {"configs[1] (1 M Iso-Seq-like, 60 k genes)": resident_config(ctx, api, cabi, torch, dev, 1_000_000, 60_000, False, 5, 3, flush, peak),
                      "configs[2] (10 M ONT-like, 60 k genes)": resident_config(ctx, api, cabi, torch, dev, args.c2_reads, 60_000, True, 3, 2, flush, peak)}
        except Exception as e:  # noqa: BLE001
            others = {"failed": str(e)}

    out = {
        "metric": METRIC, "value": n_total / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": workload_name(args), "alignments_total": int(n_total), "cigar_ops_total": int(ops_total), "kept_after_filter": int(kept_total),
                   "transcripts": int(anno.n_trans), "sj_rows": int(len(sj["tid"])), "rrna_entries": int(len(rr["tid"])),
                   "sharding": f"{world} contiguous chromosome blocks of one coordinate-sorted stream; tables ncclBroadcast from rank 0; per-shard tables gathered to rank 0 "
                               "(count all-gather + send/recv) and merged there inside the timed step" if world > 1 else "single GPU: no gather",
                   "l2": "flushed between steps (256 MiB write, untimed); per-step inputs exceed L2"},
        "e2e": {"value": n_total / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes, "ms_per_step": e2e_ms,
                "contexts_in_flight": n_ctx, "result": "merged updated_T table + BED rows + summary on rank 0, kept-record list per rank"},
        "gpu_launches": int(launches),
        "clocks": clk,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                     "traffic_note": traffic_note, "peak_source": peak_src, "algorithmic_bytes_per_launch": int(dbytes), "kernel_ms": dms, "rank": 0,
                     "all_kernels": {k: {"ms": v[0], "algorithmic_bytes": int(v[1]), "frac": (v[1] / (v[0] * 1e-3) / 1e9 / peak) if v[0] > 0 else None} for k, v in kernels.items()},
                     "path": {"algorithmic_bytes_per_step": int(path_bytes), "achieved": path_bytes / (ms_step * 1e-3) / 1e9,
                              "frac": path_bytes / (ms_step * 1e-3) / 1e9 / peak / world, "note": "whole job, per GPU: bytes / step time / N / peak"}},
        "stage_ms": st, "rank_ms": rank_ms,
        "cpu_baseline": cpu, "files_e2e": files, "other_configs": others,
        "merged": {"updated_transcripts": int(n_upd_total), "summary_counters": [int(x) for x in summary], "rank0_diag": ctx.update_diag()},
    }
    sys.stdout.flush(); os.dup2(real_stdout, 1)
    print(json.dumps(out), flush=True)
    os.dup2(2, 1)
    if dist is not None:
        ctx.comm_destroy(); dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=50_000_000, help="primary alignments of the whole data set (configs[3]: 50 M)")
    ap.add_argument("--genes", type=int, default=60_000)
    ap.add_argument("--shape", default="iso", choices=["iso", "ont"])
    ap.add_argument("--cpu-reads", type=int, default=300_000, help="sample size of the cpu_baseline / files_e2e legs (the reference's summary is quadratic, so its rate falls with the sample)")
    ap.add_argument("--ref-reads", type=int, default=800_000, help="sample size per step of --impl reference (cut into one shard per core)")
    ap.add_argument("--c2-reads", type=int, default=10_000_000, help="size of the configs[2] leg (ONT-like)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--e2e-contexts", type=int, default=3, help="lrb contexts (streams + host threads) kept in flight by the e2e leg at N = 1")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (rank 0's results)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        bench_reference(args, rank, world)
    else:
        bench_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
