"""The premise of lrb_update_gather_reads, on the CPU restatement: the per-read results of filter + bam2gtf + update-gtf run per
shard, concatenated with each shard's row / exon / record indices shifted to the whole stream, are those of the whole stream.
Shards come from multi.plan_shards (locus-aligned, never inside a qname run).

concat_update / concat_filter are the numpy statement of that rebasing; tests/test_gather_reads_gpu.py checks the CUDA gather
against them too."""
import numpy as np
import pytest

from lr2rmats_b200 import cabi, multi, synth
from tests import oracle_port as op
from tests.test_gpu_parity import assert_dict_equal


def _starts(sizes):
    return np.concatenate([[0], np.cumsum(sizes, dtype=np.int64)])


def concat_update(parts, name_bases):
    """Per-shard update results (cabi.update_to_np shape, without summary / bed) -> the whole stream's.
    ex.read_idx, keep_idx: + the shard's first record; ex.exon_off: + exons of the shards before; known_idx, unrecog_idx,
    novel.read: + rows of the shards before; updated.cand: + novel entries of the shards before; everything else unchanged."""
    rows = _starts([p["ex"]["n_reads"] for p in parts])
    exons = _starts([len(p["ex"]["exon_start"]) for p in parts])
    novel = _starts([len(p["novel"]["read"]) for p in parts])

    def cat(get, add=None):
        return np.concatenate([get(p) if add is None else (get(p).astype(np.int64) + add[r]).astype(get(p).dtype)
                               for r, p in enumerate(parts)])
    ex = dict(n_reads=int(rows[-1]),
              read_idx=None if any(p["ex"]["read_idx"] is None for p in parts) else cat(lambda p: p["ex"]["read_idx"], name_bases),
              tid=cat(lambda p: p["ex"]["tid"]), is_rev=cat(lambda p: p["ex"]["is_rev"]),
              exon_off=np.concatenate([cat(lambda p: p["ex"]["exon_off"][:-1], exons), np.array([exons[-1]], np.uint32)]),
              exon_start=cat(lambda p: p["ex"]["exon_start"]), exon_end=cat(lambda p: p["ex"]["exon_end"]))
    upd = {k: cat(lambda p, k=k: p["updated"][k], novel if k == "cand" else None) for k in parts[0]["updated"]}
    return dict(ex=ex, cls=cat(lambda p: p["cls"]), ref_anno=cat(lambda p: p["ref_anno"]), exon_flag=cat(lambda p: p["exon_flag"]),
                known_idx=cat(lambda p: p["known_idx"], rows), unrecog_idx=cat(lambda p: p["unrecog_idx"], rows),
                novel={k: cat(lambda p, k=k: p["novel"][k], rows if k == "read" else None) for k in parts[0]["novel"]},
                updated=upd)


def concat_filter(parts, name_bases):
    """Per-shard filter results (cabi.filter_to_np shape) -> the whole stream's: keep_idx + the shard's first record."""
    return dict(pass_=np.concatenate([p["pass_"] for p in parts]), score=np.concatenate([p["score"] for p in parts]),
                intron_n=np.concatenate([p["intron_n"] for p in parts]),
                keep_idx=np.concatenate([(p["keep_idx"].astype(np.int64) + b).astype(np.uint32) for p, b in zip(parts, name_bases)]))


def per_read(u):
    """An update result without the parts lrb_update_gather merges (summary, BED rows)."""
    return {k: v for k, v in u.items() if k not in ("summary", "bed")}


@pytest.fixture(scope="module")
def data():
    anno = synth.make_annotation(400, n_chrom=4, seed=51)
    rr = synth.make_rrna(anno, 8, seed=52)
    iso = synth.make_reads(anno, 20000, seed=53, ont=False, reject_frac=0.2, rrna=rr)
    ont = synth.make_reads(anno, 4000, seed=54, ont=True, reject_frac=0.2, rrna=rr)
    return dict(anno=anno.soa(), rr=rr, iso=iso, ont=ont, sj={s: synth.make_sj_from_reads(r, frac=0.7, seed=55) for s, r in (("iso", iso), ("ont", ont))})


def run_port(batch, data, sj, up):
    of = op.filter(batch, data["rr"], cabi.FilterParams.default())
    ex = op.bam2gtf(batch, cabi.ExonParams.default(), sel=of["keep_idx"])
    rc, u = op.update(ex, data["anno"], sj, up)
    assert rc == 0
    return of, u


@pytest.mark.parametrize("level", [1, 3, 5])
@pytest.mark.parametrize("summary", [0, 1])
@pytest.mark.parametrize("shape", ["iso", "ont"])
def test_shards_concatenate_to_whole_stream(data, shape, summary, level):
    batch = data[shape].soa()
    sj = data["sj"][shape]
    up = cabi.UpdateParams.default(full_level=level, split_trans=1, min_sj_cnt=1, want_summary=summary)
    whole_f, whole_u = run_port(batch, data, sj, up)
    assert (whole_u["novel"]["piece"] >= 0).any() and len(whole_u["updated"]["cand"])
    assert level == 1 or (len(whole_u["known_idx"]) and len(whole_u["unrecog_idx"]))      # -l 1 lists neither
    for n_shards in (2, 4, 8):
        cuts = multi.plan_shards(batch, n_shards)
        assert len(set(cuts.tolist())) == n_shards + 1, "degenerate shards"
        parts = [run_port(multi.take_shard(batch, int(lo), int(hi)), data, sj, up) for lo, hi in zip(cuts[:-1], cuts[1:])]
        assert_dict_equal(concat_filter([f for f, _ in parts], cuts[:-1]), whole_f, f"{n_shards} shards: filter")
        assert_dict_equal(concat_update([per_read(u) for _, u in parts], cuts[:-1]), per_read(whole_u), f"{n_shards} shards: update")
