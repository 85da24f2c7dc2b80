"""Every path of the device's merge fold, placed on its boundaries on purpose and checked against the CPU port.

launch_merge_fold (lr2rmats_b200/csrc/lrb_update.cu) sends each locus down one of several paths with fixed capacities between them:
the flat kernels (<= 64 candidates, <= 32 survivors), fold_big_kernel's tier 0 (128 survivors) and tier 1 (416), merge_fold_kernel
after an overflow or at >= 32768 candidates, the class-relation rows (<= 127 classes per locus and sub-stream, else the relation cache),
merge_fold_kernel<8> / <32> for -d > 0 (<= 32 / >= 33 candidates), and the one-locus replay.  Each case below is a hand-built locus
(tests/fold_loci.py; the recipes are checked against the port without a device in test_fold_regimes_port.py) run through unique-gtf
and update-gtf (summary off and on: on, the four class folds run the same loci as sub-streams on the side stream).  The outputs must
equal the port's bit for bit, the port's own output must show the case is the one it claims (survivors per locus), and the fold census
(LRB_TEST_FOLD_CENSUS, lrb_fold_census) must show that the targeted path folded the locus.

Not covered: a real 64-bit hash collision of two different chains (the flat fold's collision check, hard = 1 by collision, and the
class verification of the big loci, hard = 3).  It cannot be built by hand."""
import os
from collections import Counter

import numpy as np
import pytest

from lr2rmats_b200 import cabi, synth
from tests import fold_loci as fl
from tests import oracle_port as op
from tests.test_fold_regimes_port import RECIPES, STAIRS, member_locus
from tests.test_gpu_parity import assert_dict_equal

pytestmark = pytest.mark.gpu

EP = cabi.ExonParams.default()
# the paths a locus is folded by, one per locus (lrb_fold_census); "norows" counts (locus, sub-stream) pairs on top
PATHS = ("flat", "tier0", "tier1", "merge_overflow", "merge_verify", "d_small", "d_large")


@pytest.fixture(scope="module")
def ctx():
    from lr2rmats_b200 import api
    old = os.environ.get("LRB_TEST_FOLD_CENSUS")
    os.environ["LRB_TEST_FOLD_CENSUS"] = "1"             # read by lrb_ctx_create
    try:
        c = api.Context(0)
    finally:
        if old is None:
            del os.environ["LRB_TEST_FOLD_CENSUS"]
        else:
            os.environ["LRB_TEST_FOLD_CENSUS"] = old
    yield c
    c.close()


def census_of(ctx, call):
    before = ctx.fold_census()
    out = call()
    after = ctx.fold_census()
    return out, {s: {k: after[s][k] - before[s][k] for k in after[s]} for s in after}


def run_unique(ctx, loci, up, unsorted=False):
    ch, owner, loci = fl.chains_of(loci)
    if unsorted:                                           # the loci's runs in reverse order: a concatenation of sorted samples
        ch, owner = reverse_loci(ch, owner)
    rc, o = op.unique(ch, up)
    assert rc == 0
    ctx.upload_chains(fl.upload_form(ch))
    g, cen = census_of(ctx, lambda: ctx.unique_gtf(None, EP, up))
    assert_dict_equal(g, o, "unique")
    return fl.survivors_per_locus(o["uniq"]["cand"], owner, len(loci)), cen


def run_update(ctx, loci, up):
    ch, owner, loci = fl.chains_of(loci)
    anno = fl.anno_of(loci)
    rc, o = op.update(ch, anno, None, up)
    assert rc == 0
    ctx.set_anno(anno); ctx.set_sj(None)
    ctx.upload_chains(fl.upload_form(ch))
    g, cen = census_of(ctx, lambda: ctx.update_gtf(None, EP, up))
    assert_dict_equal(g, o, f"update summary={up.want_summary}")
    return fl.survivors_per_locus(o["updated"]["cand"], fl.novel_owner(o, owner), len(loci)), cen, g


def reverse_loci(ch, owner):
    order = np.concatenate([np.nonzero(owner == k)[0] for k in sorted(set(owner.tolist()), reverse=True)])
    off = ch["exon_off"].astype(np.int64)
    es = np.concatenate([ch["exon_start"][off[i]:off[i + 1]] for i in order])
    ee = np.concatenate([ch["exon_end"][off[i]:off[i + 1]] for i in order])
    noff = np.concatenate([[0], np.cumsum(np.diff(off)[order])]).astype(np.uint32)
    return dict(ch, tid=ch["tid"][order], is_rev=ch["is_rev"][order], exon_off=noff, exon_start=es, exon_end=ee), owner[order]


def assert_paths(got, want: Counter, where):
    """The census of one fold stream equals the expected number of loci per path (every path, so nothing else ran)."""
    seen = {k: got[k] for k in PATHS}
    assert seen == {k: want.get(k, 0) for k in PATHS}, f"{where}: wanted {dict(want)}, the census shows {seen}"


# case -> (locus builder, parameters, path of its locus in unique-gtf / in update-gtf's updated_T fold / in the class folds)
def _case(build, path, main=None, side=None, **up):
    return build, up, (path, main or path, side or path)


def norows(path, streams, force):
    """(locus, sub-stream) pairs of the census's "norows": a locus the warp replay takes (whatever path finished it) gets class rows
    per sub-stream unless its multi-exon classes there outnumber the 127 rows.  streams: the chains of each sub-stream, (is_rev, exons)."""
    if path in ("flat", "d_small", "d_large"):
        return 0
    return sum(fl.n_classes(chains, by_strand=force) > 127 for chains in streams)


def update_streams(loc, g):
    """The chains of the updated_T fold (novel_T) and of the four class folds (known / novel reliable / novel unreliable /
    unrecognized, update_gtf.c:501-528), strands as classification left them (the reference's strand of a matched transcript)."""
    rev, cls = g["ex"]["is_rev"], g["cls"]
    rows = [(int(rev[r]), ex) for r, (_, ex) in enumerate(loc.chains)]
    known, site, unrel = (cls & cabi.C_KNOWN) != 0, (cls & cabi.C_KNOWN_SITE) != 0, (cls & cabi.C_UNRELIABLE) != 0
    masks = (known, ~known & site & ~unrel, ~known & site & unrel, ~known & ~site)
    return [rows[r] for r in g["novel"]["read"]], [[rows[r] for r in np.nonzero(m)[0]] for m in masks]


CASES = {
    # 1. flat boundary: 32 survivors fit the flat kernel's slots, the 33rd sends the locus to tier 0; 65 candidates go there directly
    "flat_32": _case(RECIPES["flat_32"], "flat"),
    "flat_33": _case(RECIPES["flat_33"], "tier0"),
    "big_65": _case(RECIPES["big_65"], "tier0"),
    # 2. tier 0 holds 128 survivors, tier 1 416; the 417th sends the locus to merge_fold_kernel
    "tier0_128": _case(RECIPES["tier0_128"], "tier0"),
    "tier1_129": _case(RECIPES["tier1_129"], "tier1"),
    "tier1_416": _case(RECIPES["tier1_416"], "tier1"),
    "merge_417": _case(RECIPES["merge_417"], "merge_overflow"),
    # 3. class rows: 127 classes are tabulated, 128 fall back to the per-warp relation cache
    "rows_127": _case(RECIPES["rows_127"], "tier0"),
    "rows_128": _case(RECIPES["rows_128"], "tier0"),
    # 4. member limit: 32767 candidates still replay in tier 0 (16-bit candidate offsets at their edge), 32768 go to merge_fold_kernel
    "members_32767": _case(lambda: member_locus("members_32767"), "tier0"),
    "members_32768": _case(lambda: member_locus("members_32768"), "merge_overflow"),
    # 5. -d > 0: lane groups of 8 up to 32 candidates, whole warps from 33 on
    "d2_32": _case(RECIPES["d_32"], "d_small", ss_dis=2),
    "d2_33": _case(RECIPES["d_33"], "d_large", ss_dis=2),
    # 6. strands with -c, in tier 0
    "strands_force": _case(RECIPES["strands_tier0"], "tier0", force_strand=1),
    "strands_free": _case(RECIPES["strands_tier0"], "tier0"),
    # 7. sub-streams: one class of the locus outgrows tier 0 in the class folds, the others do not
    "novel_tier1": _case(RECIPES["novel_tier1"], "tier1"),
    "unrecog_tier1": _case(RECIPES["unrecog_tier1"], "tier1", main="flat", side="tier1"),
    # tier 1 with the class rows (the other tier-1 cases have more than 127 classes); in update-gtf the single-exon chains are
    # unrecognized, so neither the updated_T fold nor a class sub-stream outgrows tier 0
    "tier1_rows": _case(RECIPES["tier1_rows"], "tier1", main="tier0", side="tier0", end_dis=0),
}
# 6. dynamic ends in the big tiers: identity under a finite -e, single-exon merges under -f, -c with both strands
for st in STAIRS:
    path = st.split("_")[1]
    for tag, kw in (("e0", dict(end_dis=0)), ("e5", dict(end_dis=5)), ("e30", dict(end_dis=30)), ("f05", dict(single_exon_ovlp_frac=0.5)),
                    ("f1", dict(single_exon_ovlp_frac=1.0)), ("c", dict(force_strand=1, end_dis=30))):
        strands = "force_strand" in kw
        CASES[f"{st}_{tag}"] = _case(lambda st=st, strands=strands: STAIRS[st](strands=strands), path, **kw)


def check_survivors(name, loc, n, novel):
    """From the port's output alone: the locus is the case it claims."""
    if loc.survivors is not None:
        assert n == loc.survivors, (name, n)
    if novel is not None and loc.novel is not None:
        assert novel == loc.novel, (name, novel)
    if name == "tier1_rows":
        assert 128 < n <= 416 and novel <= 128
    if name.startswith("stairs_tier0"):
        assert n <= 128
    elif name.startswith("stairs_tier1"):
        assert 128 < novel <= 416 and n <= 416


@pytest.mark.parametrize("name", sorted(CASES))
def test_fold_regime(ctx, name):
    build, kw, (p_uniq, p_main, p_side) = CASES[name]
    loc = build()
    up = cabi.UpdateParams.default(**kw)
    force = bool(up.force_strand)
    if name.startswith("rows_"):                             # the class-rows boundary itself: 127 classes tabulated, 128 not
        assert norows(p_uniq, [loc.chains], force) == (name == "rows_128")
    surv, cen = run_unique(ctx, [loc], up)
    assert_paths(cen["main"], Counter({p_uniq: 1}), f"{name} unique-gtf: {p_uniq}")
    assert cen["main"]["norows"] == norows(p_uniq, [loc.chains], force), (f"{name} unique-gtf: norows", cen)
    for ws in (0, 1):
        up.want_summary = ws
        novel, cen, g = run_update(ctx, [loc], up)
        check_survivors(name, loc, int(surv[0]), int(novel[0]))
        main_chains, class_streams = update_streams(loc, g)
        assert_paths(cen["main"], Counter({p_main: 1}), f"{name} update-gtf updated_T: {p_main}")
        assert cen["main"]["norows"] == norows(p_main, [main_chains], force), (f"{name} updated_T: norows", cen)
        if ws:
            assert_paths(cen["side"], Counter({p_side: 1}), f"{name} update-gtf class folds: {p_side}")
            assert cen["side"]["norows"] == norows(p_side, class_streams, force), (f"{name} class folds: norows", cen)
        else:
            assert not any(cen["side"].values()), (name, cen)


def test_one_locus_replay(ctx):
    """unique-gtf on a concatenation of sorted samples is folded as ONE locus: the replay of the whole list, here in tier 1."""
    loci = [RECIPES["flat_32"](), fl.block("second", 1, fl.SPAN, 128, dups=30)]
    surv, cen = run_unique(ctx, loci, cabi.UpdateParams.default(), unsorted=True)
    assert surv.tolist() == [32, 128]
    assert cen["main"]["single"] == 1
    assert_paths(cen["main"], Counter(tier1=1), "one-locus replay: tier1")


def ladder_loci():
    """Every default-parameter case's locus and both staircases in one batch on two chromosomes (alternating), so that concurrent
    claims of tiers, lists and counters meet; with the number of loci expected on each path."""
    cases = [(n, b, paths) for n, (b, kw, paths) in sorted(CASES.items()) if not kw]
    cases += [(n, STAIRS[n], (n.split("_")[1],) * 3) for n in sorted(STAIRS)]
    loci, want = [], {"unique": Counter(), "main": Counter(), "side": Counter()}
    for i, (n, build, paths) in enumerate(cases):
        loci.append(fl.moved(build(), 1 + i % 2, (i // 2) * fl.SPAN))
        for k, p in zip(("unique", "main", "side"), paths):
            want[k][p] += 1
    return loci, want


def test_ladder_twice(ctx):
    loci, want = ladder_loci()
    up = cabi.UpdateParams.default()
    first, cen = run_unique(ctx, loci, up)
    assert_paths(cen["main"], want["unique"], "ladder unique-gtf")
    again, _ = run_unique(ctx, loci, up)
    assert np.array_equal(first, again)
    up.want_summary = 1
    res = []
    for _ in range(2):
        novel, cen, g = run_update(ctx, loci, up)
        assert_paths(cen["main"], want["main"], "ladder update-gtf updated_T")
        assert_paths(cen["side"], want["side"], "ladder update-gtf class folds")
        res.append(g)
    assert_dict_equal(res[0], res[1], "ladder run twice")


def test_census_of_deep_data(ctx):
    """test_deep_loci_against_port's data with the census on: which paths deep generated data reach.  Asserted is only what the data
    guarantee (most candidates in loci beyond the flat kernels' 64); the counts are printed."""
    anno = synth.make_annotation(120, n_chrom=3, seed=61)
    rr = synth.make_rrna(anno, 4, seed=62)
    fp = cabi.FilterParams.default()
    for shape in ("iso", "ont"):
        reads = synth.make_reads(anno, 60_000 if shape == "iso" else 25_000, seed=63, ont=(shape == "ont"), reject_frac=0.2, rrna=rr)
        sj = synth.make_sj_from_reads(reads, frac=0.7, seed=64)
        for up in (cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1),
                   cabi.UpdateParams.default(full_level=5, split_trans=0, want_summary=1, force_strand=1)):
            ctx.set_anno(anno.soa()); ctx.set_rm(rr); ctx.set_sj(sj)
            ctx.upload(reads.soa())
            ctx.pipeline_run(fp, EP)
            _, cen = census_of(ctx, lambda: ctx.update_run(up))
            print(f"deep {shape} -l {up.full_level} -s {up.split_trans} -c {up.force_strand}: census {cen}")
            assert cen["main"]["tier0"] > 0 and cen["side"]["tier0"] > 0, cen
        _, cen = census_of(ctx, lambda: ctx.unique_gtf(reads.take(op.filter(reads.soa(), rr, fp)["keep_idx"]).soa(), EP, cabi.UpdateParams.default()))
        print(f"deep {shape} unique-gtf: census {cen['main']}")
        assert cen["main"]["tier0"] > 0, cen
    ctx.set_rm(None)
