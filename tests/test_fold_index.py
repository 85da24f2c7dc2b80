"""The class index of fold_big_kernel against the CPU port.

With tabulated class rows and no end tests (end_dis = INT_MAX, the default) the big-locus replay decides a multi-exon candidate from
the newest slot of each class in its relation row and from per-chunk bounds of the stop rule, instead of scanning back through the
survivors; single-exon candidates, loci of more than 127 classes and a finite -e keep the back-scan.  Every output must equal the
port's bit for bit, and the fold census (LRB_TEST_FOLD_CENSUS) counts the candidates the index decided ("indexed"), so each case
also shows which path ran."""
import numpy as np
import pytest

from lr2rmats_b200 import cabi, synth
from tests import fold_loci as fl
from tests import oracle_port as op
from tests.test_fold_regimes import census_of, ctx, run_unique  # noqa: F401  (ctx: the census-enabled context fixture)
from tests.test_fold_regimes_port import RECIPES, STAIRS
from tests.test_gpu_parity import assert_dict_equal

pytestmark = pytest.mark.gpu

EP = cabi.ExonParams.default()


def multi_exon(loc):
    return sum(len(ex) > 1 for _, ex in loc.chains)


def singles_then_late_classes():
    """Tier 1 with class rows: 60 two-exon survivors with duplicates and partials, then 150 single-exon chains that overlap nothing
    (each one a survivor: the locus outgrows tier 0's 128 slots), then five late classes twice each, decided behind the singles."""
    loc = fl.block("singles_tier1", 1, 0, 60, dups=40, partials=10, seed=9)
    for i in range(150):
        loc.add([(100 + 120 * i, 150 + 120 * i)])
    for j in range(5):
        for _ in range(2):
            loc.add([(18_000 + 10 * j, 18_150), (18_300 + 10 * j, 19_500)])
    loc.survivors = loc.novel = None
    return fl._order(loc)


# case -> (locus builder, parameters); every locus has more than 64 candidates: one big-locus replay
CASES = {
    # -c with both strands: the class rows leave out pairs of different strands
    "strands_tier0_c": (RECIPES["strands_tier0"], dict(force_strand=1)),
    "stairs_tier0_c": (lambda: STAIRS["stairs_tier0"](strands=True), dict(force_strand=1)),
    "stairs_c": (lambda: fl.stairs("stairs_c", 1, 0, 15, variants=3, copies=2, singles=1, seed=5, strands=True), dict(force_strand=1)),
    "stairs_tier1_c": (lambda: STAIRS["stairs_tier1"](strands=True), dict(force_strand=1)),
    # single-exon-heavy loci: single-exon candidates keep the back-scan between indexed multi-exon ones
    "singles_block": (lambda: fl.block("singles_block", 1, 0, 60, dups=40, partials=10, singles=300, seed=7), {}),
    "singles_stairs": (lambda: fl.stairs("singles_stairs", 1, 0, 20, variants=3, copies=2, singles=8, seed=8), {}),
    "singles_tier1": (singles_then_late_classes, {}),
    # 127 classes are tabulated and indexed; 128 are not: the relation cache and the back-scan
    "rows_127": (RECIPES["rows_127"], {}),
    "rows_128": (RECIPES["rows_128"], {}),
    # a finite -e: the end tests make the event depend on the slot, the back-scan decides
    "stairs_tier0_e30": (lambda: STAIRS["stairs_tier0"](), dict(end_dis=30)),
    "stairs_c_e30": (lambda: fl.stairs("stairs_c", 1, 0, 15, variants=3, copies=2, singles=1, seed=5, strands=True), dict(end_dis=30, force_strand=1)),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_index_on_built_locus(ctx, name):
    build, kw = CASES[name]
    loc = build()
    up = cabi.UpdateParams.default(**kw)
    assert len(loc.chains) > 64
    _, cen = run_unique(ctx, [loc], up)
    # the whole locus is one big-locus replay: the index decides every multi-exon candidate when the classes are tabulated and there
    # are no end tests, else none
    indexed = up.end_dis == np.iinfo(np.int32).max and fl.n_classes(loc.chains, by_strand=bool(up.force_strand)) <= 127
    assert cen["main"]["indexed"] == (multi_exon(loc) if indexed else 0), (name, cen["main"])
    if name in ("stairs_c", "singles_tier1", "rows_127"):
        assert indexed, name                                  # the cases meant to reach the index do


DEEP_PARAMS = {
    "summary": dict(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1),          # split pieces inside the big loci
    "summary_c": dict(full_level=5, split_trans=1, min_sj_cnt=1, want_summary=1, force_strand=1),
    "summary_e30": dict(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1, end_dis=30),
}


@pytest.mark.parametrize("params", sorted(DEEP_PARAMS))
@pytest.mark.parametrize("shape", ["iso", "ont"])
def test_index_on_deep_data(ctx, shape, params):
    """Deep generated loci (hundreds of reads per gene) through filter, bam2gtf and update-gtf with the summary's class folds, then
    unique-gtf on the same rows: every table and counter equals the port's; the index decides candidates on both streams under the
    default end_dis and none under -e 30."""
    anno = synth.make_annotation(120, n_chrom=3, seed=71)
    rr = synth.make_rrna(anno, 4, seed=72)
    reads = synth.make_reads(anno, 60_000 if shape == "iso" else 25_000, seed=73, ont=(shape == "ont"), reject_frac=0.2, rrna=rr)
    sj = synth.make_sj_from_reads(reads, frac=0.7, seed=74)
    fp = cabi.FilterParams.default()
    up = cabi.UpdateParams.default(**DEEP_PARAMS[params])
    of = op.filter(reads.soa(), rr, fp)
    kept = reads.take(of["keep_idx"])
    oex = op.bam2gtf(kept.soa(), EP)
    rc, ou = op.update(oex, anno.soa(), sj, up)
    assert rc == 0
    ctx.set_anno(anno.soa()); ctx.set_rm(rr); ctx.set_sj(sj)
    ctx.upload(reads.soa())
    ctx.pipeline_run(fp, EP)
    _, cen = census_of(ctx, lambda: ctx.update_run(up))
    gu = ctx.update_fetch()
    ou["ex"]["read_idx"] = gu["ex"]["read_idx"]
    assert_dict_equal(gu, ou)
    assert cen["main"]["tier0"] > 0 and cen["side"]["tier0"] > 0, cen
    if up.end_dis == np.iinfo(np.int32).max:
        assert cen["main"]["indexed"] > 0 and cen["side"]["indexed"] > 0, cen
    else:
        assert cen["main"]["indexed"] == 0 and cen["side"]["indexed"] == 0, cen
    uq = cabi.UpdateParams.default(force_strand=up.force_strand, end_dis=up.end_dis)
    rc, oq = op.unique(oex, uq)
    assert rc == 0
    gq, cen = census_of(ctx, lambda: ctx.unique_gtf(kept.soa(), EP, uq))
    oq["ex"]["read_idx"] = gq["ex"]["read_idx"]
    assert_dict_equal(gq, oq)
    assert (cen["main"]["indexed"] > 0) == (up.end_dis == np.iinfo(np.int32).max), cen
    ctx.set_rm(None)
