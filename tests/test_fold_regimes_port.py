"""The hand-built loci of tests/fold_loci.py against the CPU port alone: each recipe must be the case it claims to be -- one locus of
the stated size, the stated number of multi-exon classes, and (where the recipe fixes it) the stated number of survivors of
uniq_trans and of the updated_T fold of update-gtf.  A broken fixture is caught here, without a device; test_fold_regimes.py then
relies on these counts to put the device's fold on each boundary of its paths."""
import numpy as np
import pytest

from lr2rmats_b200 import cabi
from tests import fold_loci as fl
from tests import oracle_port as op

RECIPES = {
    "flat_32": lambda: fl.block("flat_32", 1, 0, 32, dups=32),
    "flat_33": lambda: fl.block("flat_33", 1, 0, 33, dups=31),
    "big_65": lambda: fl.block("big_65", 1, 0, 10, dups=55),
    "tier0_128": lambda: fl.block("tier0_128", 1, 0, 128, dups=30, partials=12),
    "tier1_129": lambda: fl.block("tier1_129", 1, 0, 129, dups=30, partials=12),
    "tier1_416": lambda: fl.block("tier1_416", 1, 0, 416, dups=30, partials=20),
    "merge_417": lambda: fl.block("merge_417", 1, 0, 417, dups=30, partials=20),
    "rows_127": lambda: fl.rows("rows_127", 1, 0, 127),
    "rows_128": lambda: fl.rows("rows_128", 1, 0, 128),
    "d_32": lambda: fl.block("d_32", 1, 0, 10, dups=22),
    "d_33": lambda: fl.block("d_33", 1, 0, 10, dups=23),
    "strands_tier0": lambda: fl.block("strands_tier0", 1, 0, 40, dups=40, partials=10, strands=True),
    "novel_tier1": lambda: fl.block("novel_tier1", 1, 0, 150, dups=30, unrecog=60),
    "unrecog_tier1": lambda: fl.block("unrecog_tier1", 1, 0, 20, unrecog=140),
    # tier 1 with class rows: single-exon chains add survivors but no classes (with -e 0 no two of them merge)
    "tier1_rows": lambda: fl.block("tier1_rows", 1, 0, 100, singles=100),
}
# (candidates, expected size) of the member-limit loci: built only where asked, they are large
MEMBER = {"members_32767": 32767, "members_32768": 32768}
STAIRS = {"stairs_tier0": lambda **kw: fl.stairs("stairs_tier0", 1, 0, 12, variants=2, copies=2, singles=1, **kw),
          "stairs_tier1": lambda **kw: fl.stairs("stairs_tier1", 1, 0, 33, variants=3, copies=1, singles=1, **kw)}


def member_locus(name):
    return fl.block(name, 1, 0, 3, dups=MEMBER[name] - 3)


def port_counts(loc, up=None):
    """Survivors of the locus in the port's unique-gtf fold and in its update-gtf updated_T fold."""
    up = up or cabi.UpdateParams.default()
    ch, owner, _ = fl.chains_of([loc])
    rc, oq = op.unique(ch, up)
    assert rc == 0
    rc, ou = op.update(ch, fl.anno_of([loc]), None, up)
    assert rc == 0
    return len(oq["uniq"]["cand"]), len(ou["updated"]["cand"]), ou


def test_every_multi_exon_chain_of_a_block_is_novel():
    """update-gtf's classes come from the annotation as the module says: multi-exon survivors, duplicates and partials novel,
    `unrecog` chains and single-exon chains unrecognized."""
    loc = fl.block("mix", 1, 0, 12, dups=10, partials=5, singles=4, unrecog=6)
    ch, _, _ = fl.chains_of([loc])
    rc, ou = op.update(ch, fl.anno_of([loc]), None, cabi.UpdateParams.default())
    assert rc == 0
    n_ex = np.diff(ch["exon_off"].astype(np.int64))
    known = (ou["cls"] & cabi.C_KNOWN) != 0
    site = (ou["cls"] & cabi.C_KNOWN_SITE) != 0
    assert known.sum() == 0
    assert (site & ~known).sum() == 12 + 10 + 5
    assert (~site & ~known).sum() == 4 + 12 and (~site & (n_ex == 1)).sum() == 4
    assert len(ou["novel"]["read"]) == 12 + 10 + 5


@pytest.mark.parametrize("name", sorted(RECIPES))
def test_recipe_is_what_it_claims(name):
    loc = RECIPES[name]()
    assert fl.n_loci(loc.chains) == 1
    assert fl.n_classes(loc.chains) == loc.classes
    nq, nu, _ = port_counts(loc)
    assert nu == loc.novel
    if loc.survivors is not None:
        assert nq == loc.survivors


def test_tier1_rows_recipe():
    """With -e 0 the single-exon chains all survive: more survivors than tier 0's 128 slots, candidates within tier 1's 416, and
    no more multi-exon classes than the 127 relation rows hold."""
    loc = RECIPES["tier1_rows"]()
    nq, _, _ = port_counts(loc, cabi.UpdateParams.default(end_dis=0))
    assert 128 < nq <= len(loc.chains) <= 416 and loc.classes <= 127


def test_recipe_sizes():
    """The candidate counts the GPU cases rely on: 64 / 64 / 65 for the flat boundary, 32 / 33 for -d > 0's two group widths."""
    size = {k: len(RECIPES[k]().chains) for k in ("flat_32", "flat_33", "big_65", "d_32", "d_33")}
    assert size == dict(flat_32=64, flat_33=64, big_65=65, d_32=32, d_33=33)
    for k in ("tier1_416", "merge_417", "tier1_129"):
        assert len(RECIPES[k]().chains) <= 500                # the port's back-scan is O(candidates x survivors)


@pytest.mark.parametrize("name", sorted(MEMBER))
def test_member_limit_recipe(name):
    loc = member_locus(name)
    assert len(loc.chains) == MEMBER[name] and fl.n_loci(loc.chains) == 1
    nq, nu, _ = port_counts(loc)
    assert nq == nu == 3
    # the last survivor is the locus's last candidate: the largest offset inside the locus
    assert loc.chains[-1][1][1][0] == 2003 + 10 * 2


@pytest.mark.parametrize("name", sorted(STAIRS))
def test_stairs_recipe(name):
    """The staircase is one locus; the stop rule on (extended) ends leaves some class with more than one survivor; for the tier-1 case
    the classes alone outnumber tier 0's 128 slots and the candidates fit tier 1's 416, whatever end_dis does to identity."""
    loc = STAIRS[name]()
    assert fl.n_loci(loc.chains) == 1
    assert fl.n_classes(loc.chains) == loc.classes
    m = len(loc.chains)
    if name == "stairs_tier0":
        assert 64 < m <= 128
    else:
        assert loc.classes > 128 and m <= 416
    ch, _, _ = fl.chains_of([loc])
    rc, oq = op.unique(ch, cabi.UpdateParams.default())
    assert rc == 0
    multi = [fl.junctions(loc.chains[c][1]) for c in oq["uniq"]["cand"] if len(loc.chains[c][1]) > 1]
    assert len(multi) > len(set(multi)), "no class kept two survivors: the stop rule was never decisive"
    # identical chains absorbed: cov > 1 somewhere, and an absorbed copy extended an end
    assert oq["uniq"]["cov"].max() > 1
