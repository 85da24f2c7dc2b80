"""TEST-ONLY ctypes binding of the CPU restatement (oracle/liboracle_port.so) and helpers to run the compiled
reference binary (oracle/_ref/lr2rmats).  Never imported by the product."""
from __future__ import annotations

import ctypes as C
import gzip
import hashlib
import json
import os
import subprocess

import numpy as np

from lr2rmats_b200 import cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
REF_BIN = os.path.join(ORACLE_DIR, "_ref", "lr2rmats")
PORT_BIN = os.path.join(ORACLE_DIR, "_ref", "lr2rmats_port")
REF_SORT_SCRIPT = os.path.join(ORACLE_DIR, "_ref", "sort_gtf.sh")          # the reference's src/sort_gtf.sh, copied by `make ref`
PORT_SO = os.path.join(ORACLE_DIR, "liboracle_port.so")


def build_oracle():
    """(Re)build whatever can be built: the port always (gcc only), the reference when /root/reference is mounted."""
    subprocess.run(["make", "-s", "-C", ORACLE_DIR, "all"], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)


def have_ref_bin() -> bool:
    return os.path.isfile(REF_BIN) and os.access(REF_BIN, os.X_OK)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(PORT_SO):
            build_oracle()
        L = C.CDLL(PORT_SO)
        P = C.POINTER
        L.orc_filter.argtypes = [P(cabi.Batch), P(cabi.Anno), P(cabi.FilterParams), P(cabi.FilterResult)]
        L.orc_bam2gtf.argtypes = [P(cabi.Batch), cabi.u32p, C.c_int64, P(cabi.ExonParams), P(cabi.ExonResult)]
        L.orc_update.argtypes = [P(cabi.ExonResult), P(cabi.Anno), P(cabi.Sj), P(cabi.UpdateParams), P(cabi.UpdateResult)]
        L.orc_unique.argtypes = [P(cabi.ExonResult), P(cabi.UpdateParams), P(cabi.UniqueResult)]
        L.orc_bam2sj.argtypes = [P(cabi.Batch), cabi.u8p, P(cabi.SjParams), P(cabi.Sj)]
        for f in ("orc_free_filter", "orc_free_exon", "orc_free_update", "orc_free_unique", "orc_free_sj"):
            getattr(L, f).restype = None
        _lib = L
    return _lib


def filter(batch_soa: dict, rm_soa: dict | None, params: cabi.FilterParams) -> dict:
    b, k1 = cabi.make_batch(batch_soa)
    rm, k2 = cabi.make_anno(rm_soa) if rm_soa is not None else (None, None)
    res = cabi.FilterResult()
    rc = lib().orc_filter(C.byref(b), C.byref(rm) if rm is not None else None, C.byref(params), C.byref(res))
    assert rc == 0
    out = cabi.filter_to_np(res)
    lib().orc_free_filter(C.byref(res))
    return out


def bam2gtf(batch_soa: dict, params: cabi.ExonParams, sel=None) -> dict:
    b, k1 = cabi.make_batch(batch_soa)
    res = cabi.ExonResult()
    if sel is not None:
        sel = np.ascontiguousarray(sel, np.uint32)
        rc = lib().orc_bam2gtf(C.byref(b), sel.ctypes.data_as(cabi.u32p), len(sel), C.byref(params), C.byref(res))
    else:
        rc = lib().orc_bam2gtf(C.byref(b), None, 0, C.byref(params), C.byref(res))
    assert rc == 0
    out = cabi.exon_to_np(res)
    lib().orc_free_exon(C.byref(res))
    return out


def update(chains: dict, anno_soa: dict, sj_soa: dict | None, params: cabi.UpdateParams):
    ex, k1 = cabi.exon_struct_from_np(chains)
    a, k2 = cabi.make_anno(anno_soa)
    sj, k3 = cabi.make_sj(sj_soa) if sj_soa is not None and len(sj_soa["tid"]) else (None, None)
    res = cabi.UpdateResult()
    rc = lib().orc_update(C.byref(ex), C.byref(a), C.byref(sj) if sj is not None else None, C.byref(params), C.byref(res))
    if rc != 0:
        return rc, None
    out = cabi.update_to_np(res)
    lib().orc_free_update(C.byref(res))
    return 0, out


def unique(chains: dict, params: cabi.UpdateParams):
    ex, k1 = cabi.exon_struct_from_np(chains)
    res = cabi.UniqueResult()
    rc = lib().orc_unique(C.byref(ex), C.byref(params), C.byref(res))
    if rc != 0:
        return rc, None
    out = cabi.unique_to_np(res)
    lib().orc_free_unique(C.byref(res))
    return 0, out


def bam2sj(batch_soa: dict, is_uniq, params: cabi.SjParams) -> dict:
    b, k1 = cabi.make_batch(batch_soa)
    u = np.ascontiguousarray(is_uniq, np.uint8)
    res = cabi.Sj()
    rc = lib().orc_bam2sj(C.byref(b), u.ctypes.data_as(cabi.u8p), C.byref(params), C.byref(res))
    assert rc == 0
    out = {k: v.copy() for k, v in cabi.sj_to_np(res).items()}
    lib().orc_free_sj(C.byref(res))
    return out


REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "ref_digests.json")


def digest(path) -> str:
    """sha256 of a file's bytes; of the decompressed stream for a .bam (its deflate bytes depend on zlib)."""
    with (gzip.open(path) if str(path).endswith(".bam") else open(path, "rb")) as f:
        return hashlib.sha256(f.read()).hexdigest()


def stored_digests(key: str, got: dict | None) -> dict:
    """Entry `key` of tests/golden/ref_digests.json: digests of the reference's outputs on a test's generated inputs (or of those
    inputs), so that the comparison with the reference holds where it is not built.  `got` maps names to the digests the test
    computed from the reference's own run; with LRB_RECORD_REF_DIGESTS=1 they are (re)recorded instead."""
    table = {}
    if os.path.exists(REF_DIGESTS):
        with open(REF_DIGESTS) as f:
            table = json.load(f)
    if os.environ.get("LRB_RECORD_REF_DIGESTS") == "1" and got is not None:
        table[key] = got
        with open(REF_DIGESTS, "w") as f:
            json.dump(table, f, indent=1, sort_keys=True)
            f.write("\n")
    assert key in table, f"no entry {key} in tests/golden/ref_digests.json"
    return table[key]


def ref_digests(key: str, run_ref, paths: dict, available=None) -> dict:
    """Digests of what the reference writes to `paths` (name -> file) when `run_ref()` runs it: computed live where it is built
    (`available`, by default the reference binary) and checked against the stored ones, the stored ones elsewhere."""
    if not (have_ref_bin() if available is None else available):
        return stored_digests(key, None)
    run_ref()
    got = {name: digest(p) for name, p in paths.items()}
    assert stored_digests(key, got) == got, f"{key}: the reference's outputs differ from entry {key} of tests/golden/ref_digests.json"
    return got


def check_inputs(key: str, paths: dict) -> None:
    """The generated inputs must be the ones the stored reference digests were taken on."""
    got = {name: digest(p) for name, p in paths.items()}
    assert stored_digests(key, got) == got, f"{key}: the generated inputs changed; re-record tests/golden/ref_digests.json with the reference binary"


def run_bin(binary: str, args: list, stdout_path: str | None = None, check=True):
    with open(stdout_path, "wb") if stdout_path else open(os.devnull, "wb") as so:
        p = subprocess.run([binary] + [str(a) for a in args], stdout=so, stderr=subprocess.PIPE)
    if check and p.returncode != 0:
        raise RuntimeError(f"{binary} {args} failed rc={p.returncode}: {p.stderr.decode()[-2000:]}")
    return p
