"""ctypes binding of liblr2rmats_b200.so (the C ABI of include/lr2rmats_b200.h) for tests and bench.py.

This is plumbing only: numpy arrays in, numpy arrays out, every bit of compute happens in the CUDA library.  There is no
CPU path: `Context()` raises when the library is not built or no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import cabi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "liblr2rmats_b200.so")
CLI_PATH = os.path.join(_HERE, "host", "lr2rmats-b200")

ENTRY_POINTS = [
    "lrb_ctx_create", "lrb_ctx_destroy", "lrb_last_error", "lrb_version", "lrb_anno_upload", "lrb_rm_upload", "lrb_sj_upload",
    "lrb_batch_upload", "lrb_chains_upload", "lrb_filter_run", "lrb_exon_run", "lrb_pipeline_run", "lrb_update_run", "lrb_unique_run",
    "lrb_sync", "lrb_rows_sort", "lrb_filter_fetch", "lrb_exon_fetch", "lrb_update_fetch", "lrb_unique_fetch", "lrb_filter", "lrb_bam2gtf",
    "lrb_update_gtf", "lrb_unique_gtf", "lrb_timing_enable", "lrb_timing_get", "lrb_launch_count", "lrb_shard_cuts",
    "lrb_mark", "lrb_elapsed_ms", "lrb_host_alloc", "lrb_host_free", "lrb_update_fetch_table", "lrb_filter_fetch_keep",
    "lrb_comm_id", "lrb_comm_init", "lrb_comm_destroy", "lrb_comm_rank", "lrb_tables_broadcast", "lrb_update_gather", "lrb_gather_fetch",
    "lrb_gather_timing", "lrb_shard_cuts_weighted", "lrb_update_diag", "lrb_bam2sj", "lrb_sort3", "lrb_update_gather_reads",
    "lrb_gather_fetch_reads", "lrb_fold_census", "lrb_batch_attach", "lrb_cigar_stream_diag",
]

# lrb_fold_census counters per stream, in the order of the LRB_FC_* enum
FOLD_CENSUS_NAMES = ["flat", "tier0", "tier1", "merge_overflow", "merge_verify", "norows", "d_small", "d_large", "single", "indexed"]

T_NAMES = ["filter", "exon", "classify", "merge", "summary", "k_scan", "k_fold"]


class LrbError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"lr2rmats_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load_library():
    """dlopen the CUDA library and declare prototypes.  Raises if it is not built (run __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise FileNotFoundError(f"{LIB_PATH} is missing: build it with `make -C lr2rmats_b200/csrc` (there is no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    P = C.POINTER
    vp = C.c_void_p
    L.lrb_ctx_create.argtypes = [C.c_int, P(vp)]
    L.lrb_ctx_destroy.argtypes = [vp]; L.lrb_ctx_destroy.restype = None
    L.lrb_last_error.argtypes = [vp]; L.lrb_last_error.restype = C.c_char_p
    L.lrb_version.restype = C.c_char_p
    L.lrb_anno_upload.argtypes = [vp, P(cabi.Anno)]
    L.lrb_rm_upload.argtypes = [vp, P(cabi.Anno)]
    L.lrb_sj_upload.argtypes = [vp, P(cabi.Sj)]
    L.lrb_batch_upload.argtypes = [vp, P(cabi.Batch)]
    L.lrb_batch_attach.argtypes = [vp, P(cabi.Batch), C.c_int64]
    L.lrb_chains_upload.argtypes = [vp, P(cabi.Chains)]
    L.lrb_filter_run.argtypes = [vp, P(cabi.FilterParams)]
    L.lrb_exon_run.argtypes = [vp, P(cabi.ExonParams), C.c_int]
    L.lrb_pipeline_run.argtypes = [vp, P(cabi.FilterParams), P(cabi.ExonParams)]
    L.lrb_update_run.argtypes = [vp, P(cabi.UpdateParams)]
    L.lrb_unique_run.argtypes = [vp, P(cabi.UpdateParams)]
    L.lrb_sync.argtypes = [vp]
    L.lrb_rows_sort.argtypes = [vp]
    L.lrb_filter_fetch.argtypes = [vp, P(cabi.FilterResult)]
    L.lrb_exon_fetch.argtypes = [vp, P(cabi.ExonResult)]
    L.lrb_filter_fetch_keep.argtypes = [vp, P(C.c_int64), P(cabi.u32p)]
    L.lrb_update_fetch.argtypes = [vp, P(cabi.UpdateResult)]
    L.lrb_unique_fetch.argtypes = [vp, P(cabi.UniqueResult)]
    L.lrb_update_fetch_table.argtypes = [vp, P(cabi.TransTable), P(cabi.BedList), P(C.c_int32 * cabi.S_COUNT)]
    L.lrb_filter.argtypes = [vp, P(cabi.Batch), P(cabi.FilterParams), P(cabi.FilterResult)]
    L.lrb_bam2gtf.argtypes = [vp, P(cabi.Batch), P(cabi.ExonParams), P(cabi.ExonResult)]
    L.lrb_update_gtf.argtypes = [vp, P(cabi.Batch), P(cabi.ExonParams), P(cabi.UpdateParams), P(cabi.UpdateResult)]
    L.lrb_unique_gtf.argtypes = [vp, P(cabi.Batch), P(cabi.ExonParams), P(cabi.UpdateParams), P(cabi.UniqueResult)]
    L.lrb_timing_enable.argtypes = [vp, C.c_int]
    L.lrb_timing_get.argtypes = [vp, P(C.c_float * 7), P(C.c_int64)]
    L.lrb_mark.argtypes = [vp, C.c_int]
    L.lrb_elapsed_ms.argtypes = [vp, C.c_int, C.c_int, P(C.c_float)]
    L.lrb_host_alloc.argtypes = [C.c_size_t]; L.lrb_host_alloc.restype = C.c_void_p
    L.lrb_host_free.argtypes = [C.c_void_p]; L.lrb_host_free.restype = None
    L.lrb_launch_count.argtypes = [vp]; L.lrb_launch_count.restype = C.c_int64
    L.lrb_shard_cuts.argtypes = [cabi.i32p, cabi.i32p, cabi.i32p, C.c_int64, C.c_int, P(C.c_int64)]
    L.lrb_shard_cuts_weighted.argtypes = [cabi.i32p, cabi.i32p, cabi.i32p, P(C.c_int64), C.c_int64, C.c_int, P(C.c_int64)]
    L.lrb_comm_id.argtypes = [C.c_void_p]
    L.lrb_comm_init.argtypes = [vp, C.c_void_p, C.c_int, C.c_int]
    L.lrb_comm_destroy.argtypes = [vp]
    L.lrb_comm_rank.argtypes = [vp, P(C.c_int), P(C.c_int)]
    L.lrb_tables_broadcast.argtypes = [vp, C.c_int, P(cabi.Anno), P(cabi.Anno), P(cabi.Sj)]
    L.lrb_update_gather.argtypes = [vp, C.c_int64]
    L.lrb_gather_fetch.argtypes = [vp, P(cabi.TransTable), P(cabi.BedList), P(C.c_int32 * cabi.S_COUNT)]
    L.lrb_gather_timing.argtypes = [vp, P(C.c_float), P(C.c_float)]
    L.lrb_update_gather_reads.argtypes = [vp, C.c_int64]
    L.lrb_gather_fetch_reads.argtypes = [vp, P(cabi.UpdateResult), P(cabi.FilterResult)]
    L.lrb_update_diag.argtypes = [vp, P(C.c_int64), P(C.c_int64)]
    L.lrb_fold_census.argtypes = [vp, P(C.c_int64), C.c_int]
    L.lrb_cigar_stream_diag.argtypes = [vp, P(C.c_int64), P(C.c_int64)]
    L.lrb_bam2sj.argtypes = [vp, P(cabi.Batch), cabi.u8p, P(cabi.SjParams), P(cabi.Sj)]
    L.lrb_sort3.argtypes = [vp, cabi.u32p, cabi.u32p, cabi.u32p, C.c_int64, P(cabi.u32p)]
    _lib = L
    return L


class Context:
    """One lrb_ctx (one device, one stream).  Mirrors the C ABI one to one."""

    def __init__(self, device: int = 0):
        self.L = load_library()
        self.h = C.c_void_p()
        rc = self.L.lrb_ctx_create(device, C.byref(self.h))
        if rc != 0:
            raise LrbError(rc, "lrb_ctx_create failed (no CUDA device? there is no CPU fallback)")
        self._keep = {}

    def close(self):
        if self.h:
            self.L.lrb_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise LrbError(rc, self.L.lrb_last_error(self.h).decode())

    # ---- tables
    def set_anno(self, soa: dict | None):
        if soa is None:
            self._ck(self.L.lrb_anno_upload(self.h, None)); return
        a, k = cabi.make_anno(soa); self._keep["anno"] = k
        self._ck(self.L.lrb_anno_upload(self.h, C.byref(a)))

    def set_rm(self, soa: dict | None):
        if soa is None:
            self._ck(self.L.lrb_rm_upload(self.h, None)); return
        a, k = cabi.make_anno(soa); self._keep["rm"] = k
        self._ck(self.L.lrb_rm_upload(self.h, C.byref(a)))

    def set_sj(self, soa: dict | None):
        if soa is None or len(soa["tid"]) == 0:
            self._ck(self.L.lrb_sj_upload(self.h, None)); return
        s, k = cabi.make_sj(soa); self._keep["sj"] = k
        self._ck(self.L.lrb_sj_upload(self.h, C.byref(s)))

    # ---- device-resident stages
    def upload(self, batch_soa: dict):
        b, k = cabi.make_batch(batch_soa); self._keep["batch"] = (b, k)
        self._ck(self.L.lrb_batch_upload(self.h, C.byref(b)))

    def attach(self, batch_soa: dict, chunk_ops: int = 0):
        """The batch without its CIGAR pool on the device: the walk streams batch_soa["cigar"] from host memory in chunks of at most
        chunk_ops ops (0: the library chooses).  The arrays stay referenced here until the next upload / attach or close()."""
        b, k = cabi.make_batch(batch_soa); self._keep["batch"] = (b, k)
        self._ck(self.L.lrb_batch_attach(self.h, C.byref(b), int(chunk_ops)))

    def upload_struct(self, b):
        self._ck(self.L.lrb_batch_upload(self.h, C.byref(b)))

    def upload_chains(self, soa: dict):
        c, k = cabi.make_chains(soa); self._keep["chains"] = k
        self._ck(self.L.lrb_chains_upload(self.h, C.byref(c)))

    def filter_run(self, p): self._ck(self.L.lrb_filter_run(self.h, C.byref(p)))
    def exon_run(self, p, use_keep_list=False): self._ck(self.L.lrb_exon_run(self.h, C.byref(p), 1 if use_keep_list else 0))
    def pipeline_run(self, fp, ep): self._ck(self.L.lrb_pipeline_run(self.h, C.byref(fp), C.byref(ep)))
    def update_run(self, p): self._ck(self.L.lrb_update_run(self.h, C.byref(p)))
    def unique_run(self, p): self._ck(self.L.lrb_unique_run(self.h, C.byref(p)))
    def sync(self): self._ck(self.L.lrb_sync(self.h))
    def rows_sort(self): self._ck(self.L.lrb_rows_sort(self.h))          # device-side `samtools sort` of the kept rows

    def filter_fetch(self) -> dict:
        r = cabi.FilterResult(); self._ck(self.L.lrb_filter_fetch(self.h, C.byref(r))); return cabi.filter_to_np(r)

    def filter_fetch_keep(self, raw=False):
        n = C.c_int64(); p = cabi.u32p()
        self._ck(self.L.lrb_filter_fetch_keep(self.h, C.byref(n), C.byref(p)))
        return (int(n.value), p) if raw else cabi._arr(p, n.value, np.uint32)

    def exon_fetch(self) -> dict:
        r = cabi.ExonResult(); self._ck(self.L.lrb_exon_fetch(self.h, C.byref(r))); return cabi.exon_to_np(r)

    def update_fetch(self, raw=False):
        r = cabi.UpdateResult(); self._ck(self.L.lrb_update_fetch(self.h, C.byref(r)))
        return r if raw else cabi.update_to_np(r)

    def update_fetch_table(self, raw=False, want_bed=True):
        """updated_T as a self-contained table + BED rows + summary counters (what update-gtf -o/-y/-E print)."""
        t = cabi.TransTable(); b = cabi.BedList(); s = (C.c_int32 * cabi.S_COUNT)()
        self._ck(self.L.lrb_update_fetch_table(self.h, C.byref(t), C.byref(b) if want_bed else None, C.byref(s)))
        if raw:
            return t, b, s
        return dict(table=cabi.table_to_np(t), bed=cabi.bed_to_np(b) if want_bed else None, summary=np.array(list(s), np.int32))

    def unique_fetch(self) -> dict:
        r = cabi.UniqueResult(); self._ck(self.L.lrb_unique_fetch(self.h, C.byref(r))); return cabi.unique_to_np(r)

    # ---- one-call forms (host buffers in, host buffers out)
    def filter(self, batch_soa, p) -> dict:
        b, k = cabi.make_batch(batch_soa); r = cabi.FilterResult()
        self._ck(self.L.lrb_filter(self.h, C.byref(b), C.byref(p), C.byref(r))); return cabi.filter_to_np(r)

    def bam2gtf(self, batch_soa, p) -> dict:
        b, k = cabi.make_batch(batch_soa); r = cabi.ExonResult()
        self._ck(self.L.lrb_bam2gtf(self.h, C.byref(b), C.byref(p), C.byref(r))); return cabi.exon_to_np(r)

    def update_gtf(self, batch_soa, ep, up) -> dict:
        r = cabi.UpdateResult()
        if batch_soa is None:
            self._ck(self.L.lrb_update_gtf(self.h, None, C.byref(ep), C.byref(up), C.byref(r)))
        else:
            b, k = cabi.make_batch(batch_soa)
            self._ck(self.L.lrb_update_gtf(self.h, C.byref(b), C.byref(ep), C.byref(up), C.byref(r)))
        return cabi.update_to_np(r)

    def bam2sj(self, batch_soa, is_uniq, sp) -> dict:
        b, k = cabi.make_batch(batch_soa); r = cabi.Sj()
        u = np.ascontiguousarray(is_uniq, np.uint8)
        self._ck(self.L.lrb_bam2sj(self.h, C.byref(b), u.ctypes.data_as(cabi.u8p), C.byref(sp), C.byref(r)))
        return cabi.sj_to_np(r)

    def sort3(self, k0, k1, k2) -> np.ndarray:
        """Stable sort by three unsigned keys (the `sort -n` of src/sort_gtf.sh); returns the permutation."""
        a = [np.ascontiguousarray(k, np.uint32) for k in (k0, k1, k2)]
        p = cabi.u32p()
        self._ck(self.L.lrb_sort3(self.h, *[x.ctypes.data_as(cabi.u32p) for x in a], len(a[0]), C.byref(p)))
        return cabi._arr(p, len(a[0]), np.uint32).copy()

    def unique_gtf(self, batch_soa, ep, up) -> dict:
        r = cabi.UniqueResult()
        if batch_soa is None:
            self._ck(self.L.lrb_unique_gtf(self.h, None, C.byref(ep), C.byref(up), C.byref(r)))
        else:
            b, k = cabi.make_batch(batch_soa)
            self._ck(self.L.lrb_unique_gtf(self.h, C.byref(b), C.byref(ep), C.byref(up), C.byref(r)))
        return cabi.unique_to_np(r)

    # ---- multi-GPU (one process per GPU; see lr2rmats_b200/multi.py for the driver)
    def comm_init(self, comm_id: bytes, rank: int, n_ranks: int):
        _prefer_bundled_nccl()
        self._comm_id = C.create_string_buffer(bytes(comm_id), COMM_ID_BYTES)
        self._ck(self.L.lrb_comm_init(self.h, self._comm_id, rank, n_ranks))

    def comm_destroy(self): self._ck(self.L.lrb_comm_destroy(self.h))

    def tables_broadcast(self, root: int, anno: dict | None, rm: dict | None, sj: dict | None):
        """Collective: the root passes its host tables, every other rank passes None."""
        a = r = s = None
        if anno is not None: a, self._keep["anno"] = cabi.make_anno(anno)
        if rm is not None: r, self._keep["rm"] = cabi.make_anno(rm)
        if sj is not None and len(sj["tid"]): s, self._keep["sj"] = cabi.make_sj(sj)
        self._ck(self.L.lrb_tables_broadcast(self.h, root, C.byref(a) if a is not None else None, C.byref(r) if r is not None else None,
                                             C.byref(s) if s is not None else None))

    def update_gather(self, name_base: int): self._ck(self.L.lrb_update_gather(self.h, int(name_base)))

    def gather_fetch(self, raw=False, want_bed=True):
        t = cabi.TransTable(); b = cabi.BedList(); s = (C.c_int32 * cabi.S_COUNT)()
        self._ck(self.L.lrb_gather_fetch(self.h, C.byref(t), C.byref(b) if want_bed else None, C.byref(s)))
        if raw:
            return t, b, s
        return dict(table=cabi.table_to_np(t), bed=cabi.bed_to_np(b) if want_bed else None, summary=np.array(list(s), np.int32))

    def update_gather_reads(self, name_base: int): self._ck(self.L.lrb_update_gather_reads(self.h, int(name_base)))

    def gather_fetch_reads(self, want_filter=True, want_update=True, raw=False):
        """Rank 0: the per-read results of the whole stream, as update_fetch() / filter_fetch() give them on one GPU; other ranks: empty."""
        u = cabi.UpdateResult() if want_update else None
        f = cabi.FilterResult() if want_filter else None
        self._ck(self.L.lrb_gather_fetch_reads(self.h, C.byref(u) if u is not None else None, C.byref(f) if f is not None else None))
        if raw:
            return u, f
        return dict(update=cabi.update_to_np(u) if u is not None else None, filter=cabi.filter_to_np(f) if f is not None else None)

    def gather_timing(self):
        a = C.c_float(); b = C.c_float(); self._ck(self.L.lrb_gather_timing(self.h, C.byref(a), C.byref(b))); return float(a.value), float(b.value)

    def update_diag(self):
        a = C.c_int64(); b = C.c_int64(); self._ck(self.L.lrb_update_diag(self.h, C.byref(a), C.byref(b)))
        return dict(pieces_across_chromosomes=int(a.value), one_locus_replays=int(b.value))

    def cigar_stream_diag(self) -> dict:
        """Of the last CIGAR walk: chunks of an attached pool walked, and the most ops one chunk staged on the device (0, 0: uploaded pool)."""
        a = C.c_int64(); b = C.c_int64(); self._ck(self.L.lrb_cigar_stream_diag(self.h, C.byref(a), C.byref(b)))
        return dict(chunks=int(a.value), max_staged_ops=int(b.value))

    def fold_census(self) -> dict:
        """Loci per merge-fold path since the context was created, {"main": {name: n}, "side": {name: n}} (names: FOLD_CENSUS_NAMES).
        Counted only when LRB_TEST_FOLD_CENSUS=1 was in the environment when the context was created; all zero otherwise."""
        k = len(FOLD_CENSUS_NAMES)
        out = (C.c_int64 * (2 * k))()
        n = self.L.lrb_fold_census(self.h, out, 2 * k)
        if n != 2 * k:
            raise LrbError(n, f"lrb_fold_census returned {n} counters, the binding knows {2 * k}")
        return {s: dict(zip(FOLD_CENSUS_NAMES, list(out)[i * k:(i + 1) * k])) for i, s in enumerate(("main", "side"))}

    # ---- measurement
    def timing(self, on=True): self._ck(self.L.lrb_timing_enable(self.h, 1 if on else 0))

    def timing_get(self):
        ms = (C.c_float * 7)(); n = C.c_int64()
        self._ck(self.L.lrb_timing_get(self.h, C.byref(ms), C.byref(n)))
        return dict(zip(T_NAMES, list(ms))), int(n.value)

    def launch_count(self) -> int:
        return int(self.L.lrb_launch_count(self.h))

    def mark(self, slot: int): self._ck(self.L.lrb_mark(self.h, slot))

    def elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float(); self._ck(self.L.lrb_elapsed_ms(self.h, a, b, C.byref(ms))); return float(ms.value)


COMM_ID_BYTES = 128


def _prefer_bundled_nccl():
    """The library binds NCCL at run time (dlopen of libnccl.so.2).  In a Python process that also imports torch, both must end up
    on the SAME copy: torch's own (site-packages/nvidia/nccl) is newer than the system one, and the dynamic loader reuses whichever
    libnccl.so.2 came first for everybody.  Point the library at torch's copy unless the caller chose one (LRB_NCCL_LIB)."""
    if os.environ.get("LRB_NCCL_LIB"):
        return
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for d in (spec.submodule_search_locations if spec else []):
            cand = os.path.join(d, "lib", "libnccl.so.2")
            if os.path.isfile(cand):
                os.environ["LRB_NCCL_LIB"] = cand
                return
    except Exception:
        pass


def comm_id() -> bytes:
    """ncclGetUniqueId through the library: call on ONE rank and ship the bytes to the others."""
    _prefer_bundled_nccl()
    L = load_library()
    buf = C.create_string_buffer(COMM_ID_BYTES)
    rc = L.lrb_comm_id(buf)
    if rc != 0:
        raise LrbError(rc, "lrb_comm_id (libnccl.so.2 not loadable?)")
    return buf.raw


def shard_cuts(tid, start, end, n_shards: int, weight=None) -> np.ndarray:
    L = load_library()
    tid = np.ascontiguousarray(tid, np.int32); start = np.ascontiguousarray(start, np.int32); end = np.ascontiguousarray(end, np.int32)
    cuts = (C.c_int64 * (n_shards + 1))()
    w = None
    if weight is not None:
        weight = np.ascontiguousarray(weight, np.int64); w = weight.ctypes.data_as(C.POINTER(C.c_int64))
    rc = L.lrb_shard_cuts_weighted(tid.ctypes.data_as(cabi.i32p), start.ctypes.data_as(cabi.i32p), end.ctypes.data_as(cabi.i32p), w, len(tid), n_shards, cuts)
    if rc != 0:
        raise LrbError(rc, "lrb_shard_cuts_weighted")
    return np.array(list(cuts), np.int64)
