"""A batch attached with lrb_batch_attach keeps its CIGAR pool in host memory; the walk streams it through the device in chunks.
Every result must be bit-identical to the one of the same batch uploaded whole (lrb_batch_upload), whatever the chunk size --
from two chunks down to chunks smaller than one tile -- and the device must never have staged more than a chunk."""
import os

import numpy as np
import pytest

from lr2rmats_b200 import cabi, synth
from tests.test_golden import CASES, replay

pytestmark = pytest.mark.gpu

FP, EP = cabi.FilterParams.default(), cabi.ExonParams.default()
# update-gtf -s -l 3 -J 1 -j sj.tab, summary on
UP = cabi.UpdateParams.default(split_trans=1, full_level=3, min_sj_cnt=1, want_summary=1)


@pytest.fixture(scope="module")
def data():
    anno = synth.make_annotation(1500, n_chrom=4, seed=31)
    rr = synth.make_rrna(anno, 40, seed=32)
    iso = synth.make_reads(anno, 32000, seed=33, ont=False, reject_frac=0.2, rrna=rr)
    ont = synth.make_reads(anno, 4000, seed=34, ont=True, reject_frac=0.2, rrna=rr)
    sj = {k: synth.make_sj_from_reads(r, frac=0.7, seed=35) for k, r in (("iso", iso), ("ont", ont))}
    return dict(anno=anno, rr=rr, iso=iso, ont=ont, sj=sj)


def tile_reads(reads):
    """Records per tile of the walk: 256 for short CIGARs, 32 (one warp) for long ones (> 48 ops per record on average)."""
    return 32 if int(reads.cigar_off[-1]) > 48 * reads.n else 256


def tile_ops(reads):
    """CIGAR ops per tile of the walk."""
    off, starts = reads.cigar_off.astype(np.int64), np.arange(0, reads.n, tile_reads(reads))
    return off[np.minimum(starts + tile_reads(reads), reads.n)] - off[starts]


def snap(x):
    """A deep copy: fetched arrays are views of pinned buffers the next fetch reuses."""
    if isinstance(x, dict):
        return {k: snap(v) for k, v in x.items()}
    return x.copy() if isinstance(x, np.ndarray) else x


def filter_valid(f):
    """score / intron_n are only defined where the record passes."""
    m = f["pass_"].astype(bool)
    return dict(pass_=f["pass_"], score=np.where(m, f["score"], 0), intron_n=np.where(m, f["intron_n"], 0), keep_idx=f["keep_idx"])


def assert_same(a, b, path=""):
    assert set(a) == set(b), (path, set(a) ^ set(b))
    for k in a:
        if isinstance(a[k], dict):
            assert_same(a[k], b[k], path + "/" + k)
        elif isinstance(a[k], np.ndarray):
            assert a[k].dtype == b[k].dtype and a[k].shape == b[k].shape, (path + "/" + k, a[k].shape, b[k].shape)
            if not np.array_equal(a[k], b[k]):
                i = int(np.nonzero(a[k] != b[k])[0][0])
                raise AssertionError(f"{path}/{k} differs first at {i}: {a[k][i]} vs {b[k][i]} ({int((a[k] != b[k]).sum())} diffs)")
        else:
            assert a[k] == b[k], path + "/" + k


def run_all(ctx, load, with_update=True, ep=EP):
    """Every stage that walks the CIGARs, each after a fresh load of the batch, then the update stage on the fused pass's rows.
    Returns the fetched results and the stream diagnostics of each walk."""
    out, diag = {}, {}
    load(); ctx.filter_run(FP); out["filter"] = filter_valid(snap(ctx.filter_fetch())); diag["filter"] = ctx.cigar_stream_diag()
    load(); ctx.exon_run(ep); out["exon"] = snap(ctx.exon_fetch()); diag["exon"] = ctx.cigar_stream_diag()
    load(); ctx.filter_run(FP); ctx.exon_run(ep, use_keep_list=True); out["exon_keep"] = snap(ctx.exon_fetch()); diag["exon_keep"] = ctx.cigar_stream_diag()
    load(); ctx.pipeline_run(FP, ep); diag["pipeline"] = ctx.cigar_stream_diag()
    out["pipeline_filter"] = filter_valid(snap(ctx.filter_fetch())); out["pipeline_exon"] = snap(ctx.exon_fetch())
    if with_update:
        ctx.rows_sort(); ctx.update_run(UP)
        out["update"] = snap(ctx.update_fetch())
        t = ctx.update_fetch_table()
        out["table"] = snap(dict(t["table"], summary=t["summary"], **{"bed_" + k: v for k, v in t["bed"].items()}))
    return out, diag


@pytest.fixture(scope="module")
def uploaded(data):
    """Results of the uploaded path, per shape."""
    from lr2rmats_b200 import api
    ctx = api.Context(0)
    res = {}
    for which in ("iso", "ont"):
        ctx.set_anno(data["anno"].soa()); ctx.set_rm(data["rr"]); ctx.set_sj(data["sj"][which])
        out, diag = run_all(ctx, lambda: ctx.upload(data[which].soa()))
        assert all(d == dict(chunks=0, max_staged_ops=0) for d in diag.values()), diag
        res[which] = out
    ctx.close()
    return res


@pytest.fixture(scope="module")
def ctx():
    from lr2rmats_b200 import api
    c = api.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("which", ["iso", "ont"])
@pytest.mark.parametrize("chunks", [2, 7, 100, "sub_tile"])
def test_attached_equals_uploaded(ctx, data, uploaded, which, chunks):
    reads = data[which]
    n_ops, per_tile = int(reads.cigar_off[-1]), tile_ops(reads)
    n_tiles = len(per_tile)
    assert n_tiles > 100, "the fixture must have enough tiles for ~100 chunks"
    # sub_tile: every tile but the (partial) last one holds more ops than a chunk, so each is staged alone
    chunk_ops = max(1, int(per_tile[:-1].min()) // 2) if chunks == "sub_tile" else n_ops // chunks
    ctx.set_anno(data["anno"].soa()); ctx.set_rm(data["rr"]); ctx.set_sj(data["sj"][which])
    out, diag = run_all(ctx, lambda: ctx.attach(reads.soa(), chunk_ops))
    for k in uploaded[which]:
        assert_same(out[k], uploaded[which][k], k)
    # a chunk holds whole tiles and at most chunk_ops ops (its first op rounded down to a multiple of 4 included), unless one tile
    # alone holds more
    bound = max(chunk_ops, int(per_tile.max()) + 3)
    for stage, d in diag.items():
        assert d["chunks"] > 1, (stage, d)
        assert 0 < d["max_staged_ops"] <= bound, (stage, d, bound)
        if chunks == "sub_tile":
            assert d["chunks"] == n_tiles, (stage, d)
        else:
            assert chunks <= d["chunks"] <= 2 * chunks + 1, (stage, d)
    assert out["update"]["updated"]["cand"].size > 0


def test_exon_pool_regrow_across_chunks():
    """Reads of one long run of introns with min_exon 0: every N op closes an (empty) exon, so the exons outrun the pool's first
    estimate (half an exon per op, one per record, + 4096) and the walk is repeated, every chunk of it, with the exact size."""
    from lr2rmats_b200 import api
    n, k = 400, 200
    cig = np.array([(10 << 4) | 0] + [(100 << 4) | 3] * k + [(10 << 4) | 0], np.uint32)
    soa = dict(tid=np.zeros(n, np.int32), pos=(np.arange(n, dtype=np.int32) * 50 + 1000), flag=np.zeros(n, np.uint16),
               l_qseq=np.full(n, 20, np.int32), nm=np.zeros(n, np.int32), xs=np.zeros(n, np.int8),
               qname_hash=np.arange(n, dtype=np.uint64) + 1, cigar_off=(np.arange(n + 1, dtype=np.uint64) * len(cig)), cigar=np.tile(cig, n))
    ep = cabi.ExonParams.default(min_exon=0)
    n_ops = n * len(cig)
    res = []
    for attach in (False, True):
        ctx = api.Context(0)                       # fresh: the exon pool starts at its estimate
        out, diag = run_all(ctx, (lambda: ctx.attach(soa, n_ops // 5)) if attach else (lambda: ctx.upload(soa)), with_update=False, ep=ep)
        ctx.close()
        res.append(out)
        if attach:
            assert all(d["chunks"] > 1 for d in diag.values()), diag
    assert len(res[0]["exon"]["exon_start"]) > n_ops // 2 + n + 4096, "the batch must outrun the exon pool estimate"
    for key in res[0]:
        assert_same(res[1][key], res[0][key], key)


def test_attach_contract(ctx, data):
    """A negative chunk size is refused; an upload after an attach brings the pool back to the device (no streaming)."""
    from lr2rmats_b200 import api
    reads = data["iso"]
    with pytest.raises(api.LrbError):
        ctx.attach(reads.soa(), -1)
    ctx.set_rm(data["rr"])
    ctx.attach(reads.soa(), 0); ctx.filter_run(FP)
    d = ctx.cigar_stream_diag()
    assert d["chunks"] >= 1 and 0 < d["max_staged_ops"] <= max(1 << 26, int(tile_ops(reads).max()) + 3), d
    a = filter_valid(snap(ctx.filter_fetch()))
    ctx.upload(reads.soa()); ctx.filter_run(FP)
    assert ctx.cigar_stream_diag() == dict(chunks=0, max_staged_ops=0)
    assert_same(filter_valid(snap(ctx.filter_fetch())), a)


@pytest.mark.parametrize("case,cname", CASES)
def test_cli_streamed_pool_matches_reference_golden(case, cname, tmp_path, monkeypatch):
    """The CLI's attached path (LRB_TEST_CHUNK_OPS: every batch attached, 8-op chunks, so every tile is a chunk of its own) gives
    the reference binary's output files byte for byte."""
    from lr2rmats_b200 import api
    monkeypatch.setenv("LRB_TEST_CHUNK_OPS", "8")
    assert os.path.exists(api.CLI_PATH), "product CLI not built (run __graft_entry__.build())"
    replay(api.CLI_PATH, case, cname, tmp_path)
