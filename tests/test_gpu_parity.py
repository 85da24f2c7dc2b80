"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle on the same seeded inputs --
bit-exact on every output array -- plus size-independent properties (shard invariance, fused == unfused, idempotence)."""
import os
import numpy as np
import pytest

from lr2rmats_b200 import cabi, synth
from tests import oracle_port as op

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from lr2rmats_b200 import api
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def data():
    anno = synth.make_annotation(1500, n_chrom=4, seed=21)
    rr = synth.make_rrna(anno, 40, seed=22)
    iso = synth.make_reads(anno, 30000, seed=23, ont=False, reject_frac=0.2, rrna=rr)
    ont = synth.make_reads(anno, 4000, seed=24, ont=True, reject_frac=0.2, rrna=rr)
    return dict(anno=anno, rr=rr, iso=iso, ont=ont)


def assert_dict_equal(a, b, path=""):
    assert set(a) == set(b), (path, set(a) ^ set(b))
    for k in a:
        if isinstance(a[k], dict):
            assert_dict_equal(a[k], b[k], path + "/" + k)
        elif a[k] is None or b[k] is None:
            assert a[k] is None and b[k] is None, path + "/" + k
        elif isinstance(a[k], np.ndarray):
            assert a[k].shape == b[k].shape, (path + "/" + k, a[k].shape, b[k].shape)
            if not np.array_equal(a[k], b[k]):
                i = int(np.nonzero(a[k] != b[k])[0][0])
                raise AssertionError(f"{path}/{k} differs first at {i}: {a[k][i]} vs {b[k][i]} ({int((a[k] != b[k]).sum())} diffs)")
        else:
            assert a[k] == b[k], path + "/" + k


def filter_valid(f):
    """score / intron_n are only defined where pass (the reference leaves them unset otherwise)."""
    m = f["pass_"].astype(bool)
    return dict(pass_=f["pass_"], score=np.where(m, f["score"], 0), intron_n=np.where(m, f["intron_n"], 0), keep_idx=f["keep_idx"])


@pytest.mark.parametrize("which", ["iso", "ont"])
@pytest.mark.parametrize("with_rm", [True, False])
def test_filter(ctx, data, which, with_rm):
    r = data[which]
    fp = cabi.FilterParams.default()
    ctx.set_rm(data["rr"] if with_rm else None)
    g = ctx.filter(r.soa(), fp)
    o = op.filter(r.soa(), data["rr"] if with_rm else None, fp)
    assert_dict_equal(filter_valid(g), filter_valid(o))
    assert 0 < len(o["keep_idx"]) < r.n


def test_filter_params(ctx, data):
    r = data["iso"]
    ctx.set_rm(data["rr"])
    for fp in (cabi.FilterParams.default(cov_rate=0.9, map_qual=0.9, sec_rat=0.5), cabi.FilterParams.default(min_intron_n=2),
               cabi.FilterParams.default(sec_rat=1.5), cabi.FilterParams.default(cov_rate=0.0, map_qual=0.0)):
        assert_dict_equal(filter_valid(ctx.filter(r.soa(), fp)), filter_valid(op.filter(r.soa(), data["rr"], fp)))


@pytest.mark.parametrize("which", ["iso", "ont"])
def test_bam2gtf(ctx, data, which):
    r = data[which]
    for ep in (cabi.ExonParams.default(), cabi.ExonParams.default(min_exon=1, min_intron=30, max_delet=2), cabi.ExonParams.default(min_exon=40)):
        g = ctx.bam2gtf(r.soa(), ep); o = op.bam2gtf(r.soa(), ep)
        g["read_idx"] = None
        assert_dict_equal(g, o)


def test_exon_with_keep_list_and_fused(ctx, data):
    r = data["iso"]
    fp, ep = cabi.FilterParams.default(), cabi.ExonParams.default()
    ctx.set_rm(data["rr"])
    of = op.filter(r.soa(), data["rr"], fp)
    oe = op.bam2gtf(r.soa(), ep, sel=of["keep_idx"])
    # unfused: filter stage, then the walk restricted to the keep list
    ctx.upload(r.soa()); ctx.filter_run(fp); ctx.exon_run(ep, use_keep_list=True)
    assert_dict_equal(ctx.exon_fetch(), oe)
    # fused single pass
    ctx.upload(r.soa()); ctx.pipeline_run(fp, ep)
    assert_dict_equal(ctx.exon_fetch(), oe)
    assert_dict_equal(filter_valid(ctx.filter_fetch()), filter_valid(of))


def _kept_chains(data, which):
    r = data[which]
    of = op.filter(r.soa(), data["rr"], cabi.FilterParams.default())
    kept = r.take(of["keep_idx"])
    return kept, op.bam2gtf(kept.soa(), cabi.ExonParams.default())


@pytest.mark.parametrize("which", ["iso", "ont"])
@pytest.mark.parametrize("level", [1, 2, 3, 4, 5])
def test_update_pass1(ctx, data, which, level):
    kept, chains = _kept_chains(data, which)
    up = cabi.UpdateParams.default(full_level=level)
    ctx.set_anno(data["anno"].soa()); ctx.set_sj(None)
    g = ctx.update_gtf(kept.soa(), cabi.ExonParams.default(), up)
    rc, o = op.update(chains, data["anno"].soa(), None, up)
    assert rc == 0
    o["ex"]["read_idx"] = g["ex"]["read_idx"]
    assert_dict_equal(g, o)
    assert len(o["updated"]["cand"]) > 0


@pytest.mark.parametrize("which", ["iso", "ont"])
@pytest.mark.parametrize("kw", [dict(split_trans=1), dict(split_trans=0), dict(split_trans=1, ss_dis=4, min_sj_cnt=2),
                                dict(split_trans=1, use_multi=1, force_strand=1, full_level=5), dict(split_trans=1, end_dis=30)])
def test_update_pass2_sj(ctx, data, which, kw):
    kept, chains = _kept_chains(data, which)
    sj = synth.make_sj((chains["tid"], chains["exon_off"], chains["exon_start"], chains["exon_end"]), 0.7, seed=5)
    args = dict(full_level=3); args.update(kw)
    up = cabi.UpdateParams.default(**args)
    ctx.set_anno(data["anno"].soa()); ctx.set_sj(sj)
    g = ctx.update_gtf(kept.soa(), cabi.ExonParams.default(), up)
    rc, o = op.update(chains, data["anno"].soa(), sj, up)
    assert rc == 0
    o["ex"]["read_idx"] = g["ex"]["read_idx"]
    assert_dict_equal(g, o)
    if kw.get("split_trans"):
        assert (o["novel"]["piece"] >= 0).sum() > 0, "the fixture must exercise split pieces"


@pytest.mark.parametrize("which", ["iso", "ont"])
def test_unique(ctx, data, which):
    kept, chains = _kept_chains(data, which)
    for kw in (dict(), dict(force_strand=1), dict(ss_dis=6), dict(end_dis=25, single_exon_ovlp_frac=0.5)):
        up = cabi.UpdateParams.default(**kw)
        g = ctx.unique_gtf(kept.soa(), cabi.ExonParams.default(), up)
        rc, o = op.unique(chains, up)
        assert rc == 0
        o["ex"]["read_idx"] = g["ex"]["read_idx"]
        assert_dict_equal(g, o)


def test_chains_input_mode(ctx, data):
    """-m g: read-derived transcripts given as exon chains (read_gtf_trans) instead of CIGARs."""
    kept, chains = _kept_chains(data, "iso")
    up = cabi.UpdateParams.default(full_level=3)
    ctx.set_anno(data["anno"].soa()); ctx.set_sj(None)
    ctx.upload_chains(dict(tid=chains["tid"], is_rev=chains["is_rev"], exon_off=chains["exon_off"], exon_start=chains["exon_start"], exon_end=chains["exon_end"]))
    g = ctx.update_gtf(None, cabi.ExonParams.default(), up)
    rc, o = op.update(chains, data["anno"].soa(), None, up)
    assert_dict_equal(g, o)


def test_edge_cases(ctx, data):
    anno = data["anno"]
    ctx.set_anno(anno.soa()); ctx.set_sj(None); ctx.set_rm(None)
    ep, fp, up = cabi.ExonParams.default(), cabi.FilterParams.default(), cabi.UpdateParams.default()
    # empty batch
    empty = data["iso"].take(np.zeros(0, np.int64))
    assert ctx.filter(empty.soa(), fp)["keep_idx"].size == 0
    assert ctx.bam2gtf(empty.soa(), ep)["n_reads"] == 0
    g = ctx.update_gtf(empty.soa(), ep, up)
    assert g["ex"]["n_reads"] == 0 and g["updated"]["cand"].size == 0
    # a single read
    one = data["iso"].take(np.array([5]))
    assert_dict_equal(filter_valid(ctx.filter(one.soa(), fp)), filter_valid(op.filter(one.soa(), None, fp)))
    # hand-made CIGARs: very long (> staging capacity, > 64 exons), leading N, zero-length CIGAR / unmapped
    M, I, D, N, S = synth.M, synth.I, synth.D, synth.N, synth.S
    def w(l, o): return (l << 4) | o
    long_c = []
    for k in range(3000):
        long_c += [w(30 + k % 7, M), w(100 + k % 13, N)] if k % 3 else [w(20, M), w(2, I), w(15, M), w(60, D)]
    long_c.append(w(50, M))
    cigs = [long_c, [w(100, N), w(50, M)], [w(5, S), w(40, M), w(2, N), w(40, M), w(51, D), w(10, M), w(5, S)], [], [w(70, M)] * 1]
    rds = synth.Reads()
    rds.tid = np.array([0, 0, 0, -1, 1], np.int32); rds.pos = np.array([1000, 2000, 3000, -1, 500], np.int32)
    rds.flag = np.array([0, 16, 0, 4, 0], np.uint16); rds.nm = np.array([3, 0, 1, 0, 0], np.int32); rds.xs = np.array([0, ord('+'), ord('-'), 0, 7], np.int8)
    qn = lambda c: sum((x >> 4) for x in c if (x & 15) in (M, I, S, 7, 8))
    rds.l_qseq = np.array([qn(c) for c in cigs], np.int32); rds.qid = np.arange(5); rds.qname_hash = synth.splitmix64(np.arange(5))
    rds.cigar = np.array(sum(cigs, []), np.uint32); rds.cigar_off = np.cumsum([0] + [len(c) for c in cigs]).astype(np.uint64)
    for e in (ep, cabi.ExonParams.default(min_exon=0, min_intron=0, max_delet=0)):
        g = ctx.bam2gtf(rds.soa(), e); o = op.bam2gtf(rds.soa(), e); g["read_idx"] = None
        assert_dict_equal(g, o)
    assert_dict_equal(filter_valid(ctx.filter(rds.soa(), fp)), filter_valid(op.filter(rds.soa(), None, fp)))
    # update on a batch with an unmapped record fails loudly like the reference (it aborts)
    from lr2rmats_b200 import api
    with pytest.raises(api.LrbError) as ei:
        ctx.update_gtf(rds.soa(), ep, up)
    assert ei.value.code == -5
    # unsorted reads are rejected
    rev = data["iso"].take(np.arange(200)[::-1])
    with pytest.raises(api.LrbError) as ei:
        ctx.update_gtf(rev.soa(), ep, up)
    assert ei.value.code == -4
    # the mapped subset (long chain of > 64 exons included) goes through update and unique
    sub = rds.take(np.array([4]))    # tid 1 read alone
    mapped = rds.take(np.array([0, 1, 2]))
    g = ctx.update_gtf(mapped.soa(), ep, up); ch = op.bam2gtf(mapped.soa(), ep)
    rc, o = op.update(ch, anno.soa(), None, up); o["ex"]["read_idx"] = g["ex"]["read_idx"]
    assert_dict_equal(g, o)
    g = ctx.unique_gtf(mapped.soa(), ep, up); rc, o = op.unique(ch, up); o["ex"]["read_idx"] = g["ex"]["read_idx"]
    assert_dict_equal(g, o)


def test_random_cigars(ctx, data):
    """Arbitrary op sequences (adjacent cuts, leading / trailing N and D, empty exons, clips in odd places): the CIGAR
    walk and the filter statistics against the oracle, thread mode (short) and warp mode (long)."""
    ctx.set_rm(None)
    rng = np.random.default_rng(11)
    fp = cabi.FilterParams.default()
    for lo, hi, n in ((1, 24, 3000), (60, 400, 300)):
        cigs = []
        for _ in range(n):
            k = int(rng.integers(lo, hi))
            ops = rng.choice([0, 0, 0, 1, 2, 2, 3, 3, 3, 4, 7, 8], size=k)
            lens = np.where(rng.random(k) < 0.3, rng.integers(0, 6, k), rng.integers(1, 400, k))
            cigs.append(((lens.astype(np.uint32) << 4) | ops.astype(np.uint32)).tolist())
        rds = synth.Reads()
        rds.tid = np.zeros(n, np.int32); rds.pos = np.sort(rng.integers(0, 1_000_000, n)).astype(np.int32)
        rds.flag = rng.choice([0, 16], size=n).astype(np.uint16); rds.nm = rng.integers(0, 10, n).astype(np.int32)
        rds.xs = rng.choice([0, ord('+'), ord('-')], size=n).astype(np.int8)
        rds.l_qseq = np.array([max(1, sum((x >> 4) for x in c if (x & 15) in (0, 1, 4, 7, 8))) for c in cigs], np.int32)
        rds.qid = np.arange(n); rds.qname_hash = synth.splitmix64(np.arange(n))
        rds.cigar = np.array(sum(cigs, []), np.uint32); rds.cigar_off = np.cumsum([0] + [len(c) for c in cigs]).astype(np.uint64)
        for e in (cabi.ExonParams.default(), cabi.ExonParams.default(min_exon=0, min_intron=0, max_delet=0), cabi.ExonParams.default(min_exon=30, min_intron=3, max_delet=2)):
            g = ctx.bam2gtf(rds.soa(), e); o = op.bam2gtf(rds.soa(), e); g["read_idx"] = None
            assert_dict_equal(g, o)
        assert_dict_equal(filter_valid(ctx.filter(rds.soa(), fp)), filter_valid(op.filter(rds.soa(), None, fp)))
        # fused filter + walk: the chains of the kept records
        ctx.upload(rds.soa()); ctx.pipeline_run(fp, cabi.ExonParams.default())
        keep = ctx.filter_fetch()["keep_idx"]
        g = ctx.exon_fetch(); o = op.bam2gtf(rds.take(keep).soa(), cabi.ExonParams.default())
        for k in ("exon_off", "exon_start", "exon_end", "is_rev"):
            assert np.array_equal(g[k], o[k]), k


def test_stream_scan_edge_cases(ctx, data):
    """The long-CIGAR streaming kernel (mean ops > 48): reads of 0 / 1 / 2 ops and unmapped records between long reads, runs of
    empty reads at tile and warp-span borders, short internal exons that vanish, a read whose exons overflow the staging
    slots (tile redone by the warp walk), several tiles, sub-batches that start at odd word offsets."""
    ctx.set_rm(None)
    rng = np.random.default_rng(5)
    fp = cabi.FilterParams.default()
    def w(l, o): return (int(l) << 4) | int(o)
    cigs = []
    for i in range(700):
        kind = int(rng.integers(0, 12))
        if kind == 0: c = []
        elif kind == 1: c = [w(rng.integers(1, 300), rng.choice([0, 3, 2, 4]))]
        elif kind == 2: c = [w(30, 0), w(rng.integers(1, 200), 3)]
        elif kind == 3:                              # many tiny internal exons (holes) between real ones
            c = []
            for k in range(int(rng.integers(20, 120))): c += [w(rng.integers(1, 6), 0), w(rng.integers(3, 90), 3)]
            c.append(w(40, 0))
        elif kind == 4 and i % 5 == 0:               # far more exons than the staging slots of a warp
            c = []
            for k in range(int(rng.integers(300, 700))): c += [w(rng.integers(3, 50), 0), w(rng.integers(60, 90), 2 if k % 4 == 0 else 3)]
            c.append(w(10, 0))
        else:
            k = int(rng.integers(100, 900))
            ops = rng.choice([0, 0, 0, 0, 1, 2, 2, 3, 7, 8], size=k)
            lens = np.where(ops == 3, rng.integers(1, 2000, k), rng.integers(1, 60, k))
            c = [w(5, 4)] + ((lens.astype(np.uint32) << 4) | ops.astype(np.uint32)).tolist() + [w(7, 4)]
        cigs.append(c)
    for lo in range(100, 140): cigs[lo] = []          # a run of empty reads around the first tile border (128)
    n = len(cigs)
    rds = synth.Reads()
    rds.tid = np.zeros(n, np.int32); rds.pos = np.sort(rng.integers(0, 1_000_000, n)).astype(np.int32)
    rds.flag = rng.choice([0, 16], size=n).astype(np.uint16); rds.nm = rng.integers(0, 10, n).astype(np.int32)
    empty = np.array([len(c) == 0 for c in cigs])
    rds.flag[empty & (rng.random(n) < 0.5)] = 4       # some of the empty ones are unmapped records
    rds.xs = rng.choice([0, ord('+'), ord('-')], size=n).astype(np.int8)
    rds.l_qseq = np.array([max(1, sum((x >> 4) for x in c if (x & 15) in (0, 1, 4, 7, 8))) for c in cigs], np.int32)
    rds.qid = np.arange(n); rds.qname_hash = synth.splitmix64(np.arange(n))
    rds.cigar = np.array(sum(cigs, []), np.uint32); rds.cigar_off = np.cumsum([0] + [len(c) for c in cigs]).astype(np.uint64)
    assert rds.cigar.size / n > 48
    for sub in (rds, rds.take(np.arange(3, n)), rds.take(np.arange(131, 400))):
        for e in (cabi.ExonParams.default(), cabi.ExonParams.default(min_exon=0, min_intron=0, max_delet=0), cabi.ExonParams.default(min_exon=30, min_intron=3, max_delet=2)):
            g = ctx.bam2gtf(sub.soa(), e); o = op.bam2gtf(sub.soa(), e); g["read_idx"] = None
            assert_dict_equal(g, o)
        assert_dict_equal(filter_valid(ctx.filter(sub.soa(), fp)), filter_valid(op.filter(sub.soa(), None, fp)))
        ctx.upload(sub.soa()); ctx.pipeline_run(fp, cabi.ExonParams.default())
        keep = ctx.filter_fetch()["keep_idx"]
        g = ctx.exon_fetch(); o = op.bam2gtf(sub.take(keep).soa(), cabi.ExonParams.default())
        for k in ("exon_off", "exon_start", "exon_end", "is_rev"):
            assert np.array_equal(g[k], o[k]), k


def test_shard_invariance(ctx, data):
    """SURVEY App. B.3: cutting the read stream at locus gaps and processing shards independently reproduces the unsharded
    result (the multi-GPU decomposition).  Checked here on one GPU, shard after shard."""
    from lr2rmats_b200 import api
    kept, chains = _kept_chains(data, "iso")
    off = chains["exon_off"].astype(np.int64)
    cuts = api.shard_cuts(chains["tid"], chains["exon_start"][off[:-1]], chains["exon_end"][off[1:] - 1], 4)
    up = cabi.UpdateParams.default(full_level=3, want_summary=0)
    ctx.set_anno(data["anno"].soa()); ctx.set_sj(None)
    whole = ctx.update_gtf(kept.soa(), cabi.ExonParams.default(), up)
    cov, fs, le, n_upd = [], [], [], 0
    for k in range(4):
        part = kept.take(np.arange(cuts[k], cuts[k + 1]))
        g = ctx.update_gtf(part.soa(), cabi.ExonParams.default(), up)
        cov.append(g["updated"]["cov"]); fs.append(g["updated"]["first_start"]); le.append(g["updated"]["last_end"])
    assert np.array_equal(np.concatenate(cov), whole["updated"]["cov"])
    assert np.array_equal(np.concatenate(fs), whole["updated"]["first_start"])
    assert np.array_equal(np.concatenate(le), whole["updated"]["last_end"])


def test_idempotent_and_launches(ctx, data):
    kept, chains = _kept_chains(data, "iso")
    up = cabi.UpdateParams.default(full_level=3)
    ctx.set_anno(data["anno"].soa()); ctx.set_sj(None)
    n0 = ctx.launch_count()
    a = ctx.update_gtf(kept.soa(), cabi.ExonParams.default(), up)
    n1 = ctx.launch_count()
    b = ctx.update_gtf(kept.soa(), cabi.ExonParams.default(), up)
    assert_dict_equal(a, b)
    assert n1 - n0 >= 10, "the CUDA kernels must actually have been launched"


def _table_from_full(g, name_idx_from_read_idx=True):
    """What lrb_update_fetch_table must return, derived from the full result tables (emit.cpp put_list_row, use_merged)."""
    ex, nov, upd = g["ex"], g["novel"], g["updated"]
    c = upd["cand"].astype(np.int64)
    row = nov["read"][c].astype(np.int64); lo = ex["exon_off"][row].astype(np.int64) + nov["exon_lo"][c]; n = nov["exon_n"][c].astype(np.int64)
    piece = nov["piece"][c]
    off = np.zeros(len(c) + 1, np.uint32); off[1:] = np.cumsum(n)
    es = np.concatenate([ex["exon_start"][a:a + k] for a, k in zip(lo, n)]) if len(c) else np.zeros(0, np.int32)
    ee = np.concatenate([ex["exon_end"][a:a + k] for a, k in zip(lo, n)]) if len(c) else np.zeros(0, np.int32)
    es = es.copy(); ee = ee.copy()
    es[off[:-1]] = upd["first_start"]; ee[off[1:] - 1] = upd["last_end"]
    rev = ex["is_rev"][row]
    return dict(name_idx=(ex["read_idx"][row] if ex["read_idx"] is not None else row.astype(np.uint32)), piece=piece, t_tid=upd["t_tid"], t_start=upd["t_start"],
                t_end=upd["t_end"], t_rev=np.where(piece >= 0, 0, rev).astype(np.uint8), e_tid=ex["tid"][row], e_rev=rev, cov=upd["cov"],
                ref_anno=g["ref_anno"][row], exon_off=off, exon_start=es, exon_end=ee)


@pytest.mark.parametrize("which", ["iso", "ont"])
def test_update_fetch_table(ctx, data, which):
    """The self-contained updated_T table (+ BED + summary) equals what the full per-read tables give."""
    kept, chains = _kept_chains(data, which)
    sj = synth.make_sj((chains["tid"], chains["exon_off"], chains["exon_start"], chains["exon_end"]), 0.7, seed=5)
    up = cabi.UpdateParams.default(full_level=3, split_trans=1)
    ctx.set_anno(data["anno"].soa()); ctx.set_sj(sj)
    g = ctx.update_gtf(kept.soa(), cabi.ExonParams.default(), up)
    t = ctx.update_fetch_table()
    assert_dict_equal(t["table"], _table_from_full(g))
    assert_dict_equal(t["bed"], g["bed"])
    assert np.array_equal(t["summary"], g["summary"])
    assert (t["table"]["piece"] >= 0).sum() > 0


def test_unique_unsorted_concatenation(ctx, data):
    """unique-gtf -m g on a CONCATENATION of samples (Snakefile:189-192: not globally sorted): loci then mix chromosomes and
    the early-stop quirks of merge_trans (update_gtf.c:148) decide; the fold must follow the port there too."""
    _, chains = _kept_chains(data, "iso")
    off = chains["exon_off"].astype(np.int64)
    n = len(chains["tid"])
    rng = np.random.default_rng(7)
    halves = [np.sort(rng.choice(n, n // 2, replace=False)), np.sort(rng.choice(n, n // 3, replace=False)), np.arange(0, n, 5)[::-1].copy()]
    order = np.concatenate(halves)
    cnt = (off[1:] - off[:-1])[order]
    eo = np.zeros(len(order) + 1, np.uint32); eo[1:] = np.cumsum(cnt)
    idx = np.concatenate([np.arange(off[r], off[r + 1]) for r in order])
    cat = dict(tid=chains["tid"][order].copy(), is_rev=chains["is_rev"][order].copy(), exon_off=eo,
               exon_start=chains["exon_start"][idx].copy(), exon_end=chains["exon_end"][idx].copy())
    for kw in (dict(), dict(force_strand=1), dict(ss_dis=3)):
        up = cabi.UpdateParams.default(**kw)
        ctx.upload_chains(cat)
        g = ctx.unique_gtf(None, cabi.ExonParams.default(), up)
        rc, o = op.unique(dict(cat, read_idx=None, n_reads=len(order)), up)
        assert rc == 0
        o["ex"]["read_idx"] = g["ex"]["read_idx"]
        assert_dict_equal(g, o)


def _shuffle_runs(reads, seed):
    """Name-grouped but NOT coordinate-sorted: whole qname runs in random order (what `filter` reads and writes)."""
    h = reads.qname_hash
    starts = np.r_[0, np.nonzero(h[1:] != h[:-1])[0] + 1]; ends = np.r_[starts[1:], len(h)]
    order = np.random.default_rng(seed).permutation(len(starts))
    return reads.take(np.concatenate([np.arange(starts[k], ends[k]) for k in order]))


def _samtools_order(kept):
    """samtools sort's coordinate key (bam_sort.c bam1_lt): tid, pos, reverse-strand flag; stable."""
    key = (kept.tid.astype(np.int64) << 32) | ((kept.pos.astype(np.int64) + 1) << 1) | ((kept.flag & 16) != 0).astype(np.int64)
    return np.argsort(key, kind="stable")


@pytest.mark.parametrize("which,one_chrom", [("iso", False), ("ont", False), ("iso", True)])
def test_rows_sort_replaces_samtools_sort(ctx, data, which, one_chrom):
    """filter -> [device radix sort] -> update-gtf on coordinate-UNSORTED input equals the oracle on the samtools-sorted
    kept records (Snakefile:90), row for row; the row -> record map comes back in read_idx."""
    reads = data[which]
    if one_chrom:
        reads = reads.take(np.nonzero(reads.tid <= 0)[0])          # keys below 2^32: one radix pass less
    sh = _shuffle_runs(reads, 11)
    fp, ep = cabi.FilterParams.default(), cabi.ExonParams.default()
    up = cabi.UpdateParams.default(full_level=3, split_trans=1)
    of = op.filter(sh.soa(), data["rr"], fp)
    kept = sh.take(of["keep_idx"])
    order = _samtools_order(kept)
    assert (np.diff(order) < 0).sum() > len(order) // 4, "the fixture must really be unsorted"
    oex = op.bam2gtf(kept.take(order).soa(), ep)
    sj = synth.make_sj((oex["tid"], oex["exon_off"], oex["exon_start"], oex["exon_end"]), 0.7, seed=5)
    rc, ou = op.update(oex, data["anno"].soa(), sj, up)
    assert rc == 0
    ctx.set_anno(data["anno"].soa()); ctx.set_rm(data["rr"]); ctx.set_sj(sj)
    ctx.upload(sh.soa()); ctx.pipeline_run(fp, ep)
    with pytest.raises(Exception):
        ctx.update_run(up)                                         # unsorted input is refused (LRB_E_UNSORTED), not silently mis-swept
    ctx.upload(sh.soa()); ctx.pipeline_run(fp, ep); ctx.rows_sort(); ctx.rows_sort(); ctx.update_run(up)
    gu = ctx.update_fetch()
    assert np.array_equal(gu["ex"]["read_idx"], of["keep_idx"][order])
    ou["ex"]["read_idx"] = gu["ex"]["read_idx"]
    assert_dict_equal(gu, ou)
    assert len(ou["updated"]["cand"]) > 100


def test_cli_sort_input(data, tmp_path):
    """LRB_SORT_INPUT=1: `lr2rmats-b200 update-gtf` on filter's unsorted BAM == the reference binary on the sorted records (run where it
    is built, known by the digests of entry cli_sort_input of tests/golden/ref_digests.json elsewhere)."""
    import os, subprocess
    from lr2rmats_b200 import api
    anno, rr = data["anno"], data["rr"]
    sh = _shuffle_runs(data["iso"], 12)
    synth.write_gtf(tmp_path / "anno.gtf", anno); synth.write_rm_gtf(tmp_path / "rm.gtf", rr, anno.chrom_names)
    synth.write_sam(tmp_path / "in.sam", sh, with_seq=True)
    of = op.filter(sh.soa(), rr, cabi.FilterParams.default())
    kept = sh.take(of["keep_idx"])
    synth.write_sam(tmp_path / "sorted.sam", kept.take(_samtools_order(kept)), with_seq=True)     # stands in for `samtools sort`
    op.check_inputs("cli_sort_input_inputs", {fn: tmp_path / fn for fn in ("anno.gtf", "rm.gtf", "in.sam", "sorted.sam")})
    outs = ["-y", "@sum.txt", "-E", "@bed", "-A", "@detail.txt", "-k", "@known.gtf", "-o", "@updated.gtf"]
    want = op.ref_digests("cli_sort_input", lambda: op.run_bin(op.REF_BIN, ["update-gtf", "-l", "3", str(tmp_path / "sorted.sam"), str(tmp_path / "anno.gtf")]
                                                                         + [x.replace("@", str(tmp_path) + "/ref.") for x in outs]),
                          {fn: tmp_path / f"ref.{fn}" for fn in ("sum.txt", "bed", "detail.txt", "known.gtf", "updated.gtf")})
    with open(tmp_path / "f.bam", "wb") as f:
        subprocess.run([api.CLI_PATH, "filter", "-r", str(tmp_path / "rm.gtf"), str(tmp_path / "in.sam")], stdout=f, stderr=subprocess.DEVNULL, check=True)
    env = dict(os.environ, LRB_SORT_INPUT="1")
    subprocess.run([api.CLI_PATH, "update-gtf", "-l", "3", str(tmp_path / "f.bam"), str(tmp_path / "anno.gtf")] + [x.replace("@", str(tmp_path) + "/our.") for x in outs],
                   stderr=subprocess.DEVNULL, check=True, env=env)
    for fn in ("sum.txt", "bed", "detail.txt", "known.gtf", "updated.gtf"):
        assert op.digest(tmp_path / f"our.{fn}") == want[fn], fn
    # the table-only fetch path (-o / -y / -E alone)
    few = ["-y", "@sum.txt", "-E", "@bed", "-o", "@updated.gtf"]
    subprocess.run([api.CLI_PATH, "update-gtf", "-l", "3", str(tmp_path / "f.bam"), str(tmp_path / "anno.gtf")] + [x.replace("@", str(tmp_path) + "/few.") for x in few],
                   stderr=subprocess.DEVNULL, check=True, env=env)
    for fn in ("sum.txt", "bed", "updated.gtf"):
        assert op.digest(tmp_path / f"few.{fn}") == want[fn], fn
    p = subprocess.run([api.CLI_PATH, "update-gtf", "-l", "3", str(tmp_path / "f.bam"), str(tmp_path / "anno.gtf")], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE)
    assert p.returncode != 0                                       # without the knob the unsorted BAM is refused, as documented


@pytest.mark.gpu
def test_undersized_novel_list_is_retried(tmp_path):
    """novel_T is sized optimistically (pieces are rare); when it turns out too small the fold must see an EMPTY list (its tail was never
    written), and the pass is repeated with the exact size.  LRB_TEST_SMALL_NOVEL_CAP forces that on the first attempt."""
    import subprocess
    from lr2rmats_b200 import api
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "syn_iso")
    outs = []
    for small in ("0", "1"):
        o = tmp_path / f"s{small}"; o.mkdir()
        env = dict(os.environ, LRB_TEST_SMALL_NOVEL_CAP=small)
        p = subprocess.run([api.CLI_PATH, "update-gtf", "-s", "-l", "3", "-J", "1", "-j", os.path.join(d, "sj.tab"), os.path.join(d, "in.sam"), os.path.join(d, "anno.gtf"),
                            "-y", "summary.txt", "-E", "bed.bed", "-o", "updated.gtf", "-v", "novel.gtf"], cwd=o, env=env, stderr=subprocess.PIPE)
        assert p.returncode == 0, p.stderr.decode()[-1000:]
        outs.append({f: open(o / f, "rb").read() for f in ("summary.txt", "bed.bed", "updated.gtf", "novel.gtf")})
    assert outs[0] == outs[1]
    exp = os.path.join(d, "expected", "p2s")
    for f, g in (("summary.txt", "summary.txt"), ("bed.bed", "novel_exon.bed"), ("updated.gtf", "updated.gtf"), ("novel.gtf", "novel.gtf")):
        assert outs[1][f] == open(os.path.join(exp, g), "rb").read(), f


@pytest.mark.gpu
def test_single_locus_replay_equals_locus_fold(tmp_path):
    """The one-locus replay of the updated_T fold (what a split piece meeting another chromosome falls back to) gives the
    same tables as the locus-parallel fold on data without such a meeting: run the CLI with and without LRB_FORCE_SINGLE_FOLD."""
    import subprocess
    from lr2rmats_b200 import api
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "syn_iso")
    outs = []
    for force in ("0", "1"):
        o = tmp_path / f"f{force}"; o.mkdir()
        env = dict(os.environ, LRB_FORCE_SINGLE_FOLD=force)
        p = subprocess.run([api.CLI_PATH, "update-gtf", "-s", "-l", "3", "-J", "1", "-j", os.path.join(d, "sj.tab"), os.path.join(d, "in.sam"), os.path.join(d, "anno.gtf"),
                            "-y", "summary.txt", "-E", "bed.bed", "-o", "updated.gtf"], cwd=o, env=env, stderr=subprocess.PIPE)
        assert p.returncode == 0, p.stderr.decode()[-1000:]
        outs.append({f: open(o / f, "rb").read() for f in ("summary.txt", "bed.bed", "updated.gtf")})
    assert outs[0] == outs[1]


@pytest.mark.parametrize("summary", [1, 0])
def test_cross_chromosome_piece_replay(ctx, summary):
    """Every read twice, on chromosomes 1-2 and on clones of them at the same coordinates: the split pieces of the clones meet equal
    chains on the originals, which the reference merges across chromosomes (a piece's back-scan never stops, update_gtf.c:148; golden
    c8_xlocus).  The fold must notice, and every table equals the port's.  With -d 0 the pieces are settled by rounds on the device;
    with -d 2 junctions match approximately, the probe of the set kernels proves nothing and the fold is replayed as one locus."""
    anno = synth.make_annotation(1500, n_chrom=2, seed=41)
    reads = synth.make_reads(anno, 12_000, seed=43, reject_frac=0.0)
    sj = synth.make_sj_from_reads(reads, frac=0.7, seed=44)
    a2, both, s2 = synth.clone_chromosome(anno.soa(), reads, sj, 2)
    ep = cabi.ExonParams.default()
    oex = op.bam2gtf(both.soa(), ep)
    ctx.set_anno(a2); ctx.set_sj(s2)
    for ss_dis in (0, 2):
        up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=summary, ss_dis=ss_dis)
        rc, ou = op.update(oex, a2, s2, up)
        assert rc == 0
        replays = ctx.update_diag()["one_locus_replays"]
        gu = ctx.update_gtf(both.soa(), ep, up)
        ou["ex"]["read_idx"] = gu["ex"]["read_idx"]
        assert_dict_equal(gu, ou, f"-d {ss_dis}")
        # the case is live: at least one piece of a clone chromosome was absorbed by an original (cov > 1 on a piece)
        upd = gu["updated"]; piece = gu["novel"]["piece"][upd["cand"]]
        assert ((piece >= 0) & (upd["cov"] > 1)).sum() > 0, ss_dis
        d = ctx.update_diag()
        if ss_dis == 0:
            assert d["pieces_across_chromosomes"] > 0, d     # settled by the rounds on the device, not by the one-locus replay
        else:
            assert d["one_locus_replays"] > replays, d       # the detect probe sent the fold to the one-locus replay


@pytest.mark.parametrize("which", ["iso", "ont"])
def test_bam2sj(ctx, data, which):
    """bam2sj (parse_bam.c:896-985) on the device against the port's replay of the reference's sorted insertion: distinct junctions in
    (tid, don, acc) order with unique / multi read counts; proper-pair filter (the only mode the reference can reach), -i."""
    r = data[which]
    rng = np.random.default_rng(7)
    soa = dict(r.soa())
    flag = soa["flag"].copy()
    paired = rng.random(r.n) < 0.7
    flag[paired] |= np.uint16(3)
    flag[rng.random(r.n) < 0.02] |= np.uint16(4)
    soa["flag"] = flag
    uniq = (rng.random(r.n) < 0.8).astype(np.uint8)
    for sp in (cabi.SjParams.default(), cabi.SjParams.default(min_intron=400), cabi.SjParams.default(pair_only=0)):
        g = ctx.bam2sj(soa, uniq, sp); o = op.bam2sj(soa, uniq, sp)
        assert_dict_equal(g, o)
        assert len(o["tid"]) > 100 and (o["uniq_c"] + o["multi_c"]).max() > 1
    # a stream that is not ordered by reference id is refused (the reference's insertion would leave an unsorted table)
    from lr2rmats_b200 import api
    rev = {k: (v[::-1].copy() if k not in ("cigar", "cigar_off") else v) for k, v in soa.items()}
    lens = np.diff(soa["cigar_off"].astype(np.int64))[::-1]
    rev["cigar_off"] = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    rev["cigar"] = np.concatenate([soa["cigar"][int(a):int(b)] for a, b in zip(soa["cigar_off"][:-1][::-1], soa["cigar_off"][1:][::-1])]) if r.n < 10000 else None
    if rev["cigar"] is not None:
        with pytest.raises(api.LrbError) as e:
            ctx.bam2sj(rev, uniq[::-1].copy(), cabi.SjParams.default())
        assert e.value.code == -4


def test_sort3_is_a_stable_lexicographic_sort(ctx):
    """lrb_sort3 (the `sort -n -k1..-k4` of src/sort_gtf.sh on the device): equals numpy's stable lexsort, ties keep the input order."""
    rng = np.random.default_rng(11)
    for n in (0, 1, 5, 4097, 300_000):
        k0 = rng.integers(0, 40, n).astype(np.uint32); k1 = rng.integers(0, 2**32 - 1, n, dtype=np.uint64).astype(np.uint32) // np.uint32(1 << 12)
        k2 = rng.integers(0, 3, n).astype(np.uint32) * np.uint32(0x7fffffff)
        got = ctx.sort3(k0, k1, k2)
        want = np.lexsort((np.arange(n), k2, k1, k0)).astype(np.uint32)
        assert np.array_equal(got, want)


@pytest.mark.parametrize("shape", ["iso", "ont"])
def test_deep_loci_against_port(ctx, shape):
    """Deep data: hundreds of reads per gene, so nearly every candidate sits in a locus beyond the 64-candidate masks of the flat fold
    (identity classes through the table, tabulated class relation, warp replay with the survivors in shared memory; the four class folds
    of the summary as sub-streams).  Every table and all counters equal the port's sequential merge_trans."""
    anno = synth.make_annotation(120, n_chrom=3, seed=61)
    rr = synth.make_rrna(anno, 4, seed=62)
    reads = synth.make_reads(anno, 60_000 if shape == "iso" else 25_000, seed=63, ont=(shape == "ont"), reject_frac=0.2, rrna=rr)
    sj = synth.make_sj_from_reads(reads, frac=0.7, seed=64)
    fp, ep = cabi.FilterParams.default(), cabi.ExonParams.default()
    for up in (cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1),
               cabi.UpdateParams.default(full_level=5, split_trans=0, want_summary=1, force_strand=1)):
        of = op.filter(reads.soa(), rr, fp)
        kept = reads.take(of["keep_idx"])
        oex = op.bam2gtf(kept.soa(), ep)
        rc, ou = op.update(oex, anno.soa(), sj, up)
        assert rc == 0
        ctx.set_anno(anno.soa()); ctx.set_rm(rr); ctx.set_sj(sj)
        ctx.upload(reads.soa())
        ctx.pipeline_run(fp, ep)
        ctx.update_run(up)
        gu = ctx.update_fetch()
        ou["ex"]["read_idx"] = gu["ex"]["read_idx"]
        assert_dict_equal(gu, ou)
        n_upd = len(gu["updated"]["cand"])
        assert len(of["keep_idx"]) / max(n_upd, 1) > 4          # deep: most candidates are absorbed
    # unique-gtf on the same deep stream (one fold over all rows)
    rc, oq = op.unique(oex, cabi.UpdateParams.default())
    gq = ctx.unique_gtf(kept.soa(), ep, cabi.UpdateParams.default())
    oq["ex"]["read_idx"] = gq["ex"]["read_idx"]
    assert_dict_equal(gq, oq)
