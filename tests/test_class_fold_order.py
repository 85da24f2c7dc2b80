"""The class folds of the summary on the class-ordered list, against the CPU port.

update-gtf's summary folds the rows of each class (known, novel reliable, novel unreliable, unrecognized) as a list of its own
(update_gtf.c:501-528).  The device folds them in one pass on the side stream: the rows are cut into loci in row order, then inside
each locus grouped by class (launch_class_order), and each (locus, class) replay walks only its own range.  When a class's survivors
outgrow tier 0's slots, tier 1 goes on from tier 0's saved state.  Every output must equal the port's bit for bit, and the fold
census must show the loci of the union of the classes."""
from collections import Counter

import numpy as np
import pytest

from lr2rmats_b200 import cabi, synth
from tests import fold_loci as fl
from tests import oracle_port as op
from tests.test_fold_regimes import assert_paths, census_of, ctx  # noqa: F401  (ctx: the census-enabled context fixture)
from tests.test_fold_regimes_port import RECIPES
from tests.test_gpu_parity import _samtools_order, _shuffle_runs
from tests.test_gpu_parity import assert_dict_equal

pytestmark = pytest.mark.gpu

EP = cabi.ExonParams.default()


def four_classes(name, tid, base, n, reliable=40, unreliable=40, unrecog=30, seed=0):
    """One big locus whose rows take the four classes in random order: known chains (single-exon reads over the annotation's
    single-exon transcript), novel chains on the annotation's donor with `reliable` acceptors the junction table supports and
    `unreliable` ones it lacks, unrecognized chains on sites the annotation lacks.  Starts in [base, base + 100), so every class runs
    through the whole locus.  Returns the locus and its junction table."""
    rng = np.random.default_rng(seed)
    loc = fl.Locus(name, tid, base)
    don, end = base + 1000, base + 20000
    acc_rel = [base + 2003 + 10 * j for j in range(reliable)]
    acc_unrel = [base + 6003 + 10 * j for j in range(unreliable)]
    for _ in range(n):
        s, e = base + int(rng.integers(0, 100)), end + int(rng.integers(-60, 60))
        k = int(rng.integers(0, 4))
        if k == 0:
            loc.add([(base + int(rng.integers(0, 30)), base + 600 - int(rng.integers(0, 30)))])
        elif k == 1:
            loc.add([(s, don), (acc_rel[int(rng.integers(0, reliable))], e)])
        elif k == 2:
            loc.add([(s, don), (acc_unrel[int(rng.integers(0, unreliable))], e)])
        else:
            j = int(rng.integers(0, unrecog))
            loc.add([(s, base + 1203 + 10 * j), (base + 9007 + 10 * j, e)])
    loc.anno = [(0, [(base, base + 600)]), (0, [(base + 500, don), (base + 19003, end + 100)])]
    sj = [(tid, don + 1, a - 1) for a in acc_rel]
    return fl._order(loc), sj


def sj_table(rows):
    rows = sorted(rows)
    i32 = lambda k: np.array([r[k] for r in rows], np.int32)      # noqa: E731
    return dict(tid=i32(0), don=i32(1), acc=i32(2), uniq_c=np.full(len(rows), 10, np.int32), multi_c=np.zeros(len(rows), np.int32))


def run_summary(ctx, loci, sj, up):
    """update-gtf with the summary on, device against port; returns the port's output and the census."""
    ch, _, loci = fl.chains_of(loci)
    anno = fl.anno_of(loci)
    rc, o = op.update(ch, anno, sj, up)
    assert rc == 0
    ctx.set_anno(anno); ctx.set_sj(sj)
    ctx.upload_chains(fl.upload_form(ch))
    g, cen = census_of(ctx, lambda: ctx.update_gtf(None, EP, up))
    assert_dict_equal(g, o, "update summary")
    return o, cen


def classes_of(cls):
    known, site, unrel = (cls & cabi.C_KNOWN) != 0, (cls & cabi.C_KNOWN_SITE) != 0, (cls & cabi.C_UNRELIABLE) != 0
    return np.select([known, site & ~unrel, site & unrel], [0, 1, 2], 3)


def unrecog_then_singles():
    """Unrecognized rows: 20 two-exon classes twice each (the second copy absorbed by the class index), then 150 single-exon chains
    that overlap nothing (the 129th survivor overflows tier 0 with the index holding 20 classes), then five late classes twice
    each, decided by tier 1 on the index it took over.  The novel rows of the locus (60 survivors) stay in tier 0."""
    loc = fl.block("unrecog_singles", 1, 0, 60, dups=40, partials=10, unrecog=20, seed=9)
    for i in range(150):
        loc.add([(100 + 120 * i, 150 + 120 * i)])
    for j in range(5):
        for _ in range(2):
            loc.add([(18_000 + 10 * j, 18_150), (18_300 + 10 * j, 19_500)])
    loc.survivors = loc.novel = None
    return fl._order(loc)


def test_four_classes_interleaved(ctx):
    """A big locus (600 rows) whose four classes alternate at random: each class replay walks only its own rows."""
    loc, sj = four_classes("four", 1, 0, 600, seed=11)
    up = cabi.UpdateParams.default(want_summary=1)
    o, cen = run_summary(ctx, [loc], sj_table(sj), up)
    k = classes_of(o["cls"])
    assert set(k.tolist()) == {0, 1, 2, 3}
    assert (np.diff(k) != 0).sum() > 300, "the classes are interleaved"
    assert sum(cen["side"][p] for p in ("flat", "tier0", "tier1", "merge_overflow", "merge_verify")) == 1, cen["side"]
    assert cen["side"]["tier0"] == 1, cen["side"]


def test_class_beyond_its_own_reach(ctx):
    """Novel chains in two groups: the second starts beyond every end of the first, but a long unrecognized chain in between
    reaches past it.  Cut on the union of the classes that is one locus (the side stream's census shows one), while the updated_T
    fold, which sees the novel chains alone, cuts it in two."""
    a = fl.block("first", 1, 0, 40, dups=40, partials=5)
    b = fl.block("second", 1, 30_000, 40, dups=40, partials=5, seed=1)
    loc = fl.Locus("union", 1, 0, a.chains + b.chains + [(0, [(90, 1208), (55_007, 60_000)])], a.anno + b.anno)
    loc = fl._order(loc)
    up = cabi.UpdateParams.default(want_summary=1)
    o, cen = run_summary(ctx, [loc], None, up)
    assert fl.n_loci([c for c, k in zip(loc.chains, classes_of(o["cls"])) if k == 1]) == 2
    assert_paths(cen["side"], Counter(tier0=1), "class folds: one union locus")
    assert_paths(cen["main"], Counter(tier0=2), "updated_T: two loci")


@pytest.mark.parametrize("name", ["tabulated", "untabulated"])
def test_tier1_resumes(ctx, name):
    """A class outgrows tier 0's 128 slots in the middle of its range and tier 1 goes on from tier 0's state: with class rows (the
    class index decided earlier candidates; single-exon survivors push the locus over) and without (more than 127 classes: the
    back-scan and the relation cache).  Next to it the other classes of the locus stay in tier 0."""
    if name == "tabulated":
        loc = unrecog_then_singles()
    else:
        loc = RECIPES["tier1_129"]()
    up = cabi.UpdateParams.default(want_summary=1)
    o, cen = run_summary(ctx, [loc], None, up)
    assert_paths(cen["side"], Counter(tier1=1), f"{name}: class folds")
    assert cen["side"]["norows"] == (name == "untabulated"), cen["side"]
    # the same locus a second time in the batch, next to a four-class locus: both tiers, several entries, list positions past 0
    four, sj = four_classes("four", 2, 0, 400, seed=12)
    o2, cen = run_summary(ctx, [loc, four], sj_table(sj), up)
    assert_paths(cen["side"], Counter(tier1=1, tier0=1), f"{name}: class folds beside a four-class locus")


def test_unsorted_with_summary(ctx):
    """Deep loci from an unsorted stream (name-grouped runs in random order): filter, the device sort, then update-gtf with the
    summary on.  The class folds run on the sorted rows, not in record order; every output, the four uniq_* counters included,
    equals the port's on the samtools-sorted records."""
    anno = synth.make_annotation(120, n_chrom=3, seed=81)
    rr = synth.make_rrna(anno, 4, seed=82)
    reads = _shuffle_runs(synth.make_reads(anno, 60_000, seed=83, ont=False, reject_frac=0.2, rrna=rr), 12)
    fp = cabi.FilterParams.default()
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)
    of = op.filter(reads.soa(), rr, fp)
    kept = reads.take(of["keep_idx"])
    order = _samtools_order(kept)
    assert (np.diff(order) < 0).sum() > len(order) // 8, "the stream must really be unsorted"
    oex = op.bam2gtf(kept.take(order).soa(), EP)
    sj = synth.make_sj((oex["tid"], oex["exon_off"], oex["exon_start"], oex["exon_end"]), 0.7, seed=85)
    rc, ou = op.update(oex, anno.soa(), sj, up)
    assert rc == 0
    ctx.set_anno(anno.soa()); ctx.set_rm(rr); ctx.set_sj(sj)
    ctx.upload(reads.soa()); ctx.pipeline_run(fp, EP); ctx.rows_sort()
    _, cen = census_of(ctx, lambda: ctx.update_run(up))
    gu = ctx.update_fetch()
    ou["ex"]["read_idx"] = gu["ex"]["read_idx"]
    assert_dict_equal(gu, ou)
    assert min(ou["summary"][[11, 14, 16, 18]]) > 0, ou["summary"]
    assert cen["side"]["tier0"] > 0, cen["side"]
    ctx.set_rm(None)
