"""Hand-built loci for the merge fold (merge_trans / uniq_trans): exon chains whose survivor count, class count and locus size are
known by construction, so that a case can be placed on a boundary of the fold's paths (flat kernels, the two warp-replay tiers,
merge_fold_kernel, the class-relation rows) on purpose.  Shared by test_fold_regimes_port.py (the recipes against the CPU port) and
test_fold_regimes.py (the device against the port).

Every multi-exon chain of a locus has a donor that its locus's annotation transcript also has, and no acceptor of it, so update-gtf
classifies it as a novel transcript (a known site, not every site known: oracle/port/lr2rmats_port.c site_check) and folds it into
updated_T.  `unrecog` chains use donors and acceptors the annotation lacks: unrecognized, like the single-exon chains (the annotations
have no single-exon transcript).  No chain is known: the class folds of the summary see two of their four sub-streams."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

SPAN = 200_000          # distance between the bases of two loci of one chromosome: no chain of a locus reaches the next one


@dataclass
class Locus:
    name: str
    tid: int
    base: int
    chains: list = field(default_factory=list)      # (is_rev, [(start, end), ...]) in fold order
    anno: list = field(default_factory=list)        # the annotation transcripts: (is_rev, [(start, end), ...])
    survivors: int | None = None                    # unique-gtf survivors with default parameters, by construction
    classes: int | None = None                      # distinct multi-exon chains (internal boundaries), by construction
    novel: int | None = None                        # survivors of update-gtf's updated_T fold (novel chains only), by construction

    def add(self, exons, rev=0):
        self.chains.append((int(rev), [(int(s), int(e)) for s, e in exons]))


def junctions(exons):
    return tuple(x for (s0, e0), (s1, e1) in zip(exons[:-1], exons[1:]) for x in (e0, s1))


def n_classes(chains, by_strand=False):
    return len({(len(ex), junctions(ex)) + ((rev,) if by_strand else ()) for rev, ex in chains if len(ex) > 1})


def n_loci(chains):
    """Locus cuts of the fold (a chain that starts beyond every earlier end starts a locus), on chains in fold order."""
    run, k = -1, 0
    for _, ex in chains:
        if ex[0][0] > run:
            k += 1
        run = max(run, ex[-1][1])
    return k


def _order(loc: Locus):
    """(tid, start) order, as update-gtf and unique-gtf require; ties keep the order of construction (stable)."""
    st = np.array([ex[0][0] for _, ex in loc.chains], np.int64)
    loc.chains = [loc.chains[i] for i in np.argsort(st, kind="stable")]
    return loc


def block(name, tid, base, survivors, dups=0, partials=0, singles=0, unrecog=0, seed=0, strands=False):
    """`survivors` 2-exon chains with one shared donor and pairwise distinct acceptors (equal exon counts, different junctions: none
    absorbs another), then `dups` copies of them with jittered first start and last end (cov > 1, extended ends), `partials` 3-exon
    chains that begin with a survivor's junction (check_iden 2: dropped), `singles` single-exon chains and `unrecog` 2-exon chains on
    sites the annotation lacks (`unrecog` distinct ones, each twice).  The first
    starts of the survivors lie in [base, base + 40), of the duplicates too, of the partials in [base + 50, base + 60): every chain
    that could absorb a partial comes first.  The last survivor starts at base + 45, after every duplicate: it is the locus's last
    survivor, at the locus's largest candidate offsets.  strands: random strands (all chains of a class on one strand)."""
    rng = np.random.default_rng(seed)
    loc = Locus(name, tid, base)
    don, end = base + 1000, base + 20000
    acc = [base + 2003 + 10 * j for j in range(survivors)]
    rev = rng.integers(0, 2, survivors) if strands else np.zeros(survivors, np.int64)
    for j in range(survivors):
        fs = base + 45 if j == survivors - 1 and survivors > 1 else base + int(rng.integers(0, 40))
        loc.add([(fs, don), (acc[j], end + int(rng.integers(-40, 40)))], rev[j])
    pool = max(survivors - 1, 1)
    for _ in range(dups):
        j = int(rng.integers(0, pool))
        loc.add([(base + int(rng.integers(0, 40)), don), (acc[j], end + int(rng.integers(-60, 60)))], rev[j])
    for _ in range(partials):
        j = int(rng.integers(0, survivors))
        loc.add([(base + 50 + int(rng.integers(0, 10)), don), (acc[j], base + 15000), (base + 16003, end + int(rng.integers(-40, 40)))], rev[j])
    for _ in range(singles):
        s = base + 60 + int(rng.integers(0, 400))
        loc.add([(s, s + 300 + int(rng.integers(0, 200)))], rng.integers(0, 2) if strands else 0)
    for j in range(unrecog):
        for _ in range(2):
            loc.add([(base + 60 + int(rng.integers(0, 30)), base + 1203 + 10 * j), (base + 9007 + 10 * j, end + int(rng.integers(-40, 40)))])
    loc.anno = [(0, [(base + 500, don), (base + 19003, end + 100)])]
    loc.classes = n_classes(loc.chains)
    loc.survivors = None if singles else survivors + unrecog   # single-exon merges: the port decides
    loc.novel = survivors
    return _order(loc)


def rows(name, tid, base, n_classes_, dups=20, seed=0):
    """One long chain of 17 exons, then `n_classes_ - 1` distinct shorter chains, each a run of its junctions (partial relation with
    the long chain and with each other where the runs nest: many set bits in the class rows), then duplicates of the long chain.  All
    are absorbed by the long chain: one survivor, `n_classes_` classes."""
    rng = np.random.default_rng(seed)
    loc = Locus(name, tid, base)
    nex = 17
    ex = [(base + 1000 * i + (0 if i == 0 else 3), base + 1000 * i + 300) for i in range(nex)]
    ex[-1] = (ex[-1][0], base + 1000 * (nex - 1) + 900)
    runs = [(i, j) for i in range(nex - 1) for j in range(i + 1, nex) if (i, j) != (0, nex - 1)]   # exons i..j, >= one junction
    assert n_classes_ - 1 <= len(runs)
    pick = [runs[k] for k in rng.permutation(len(runs))[: n_classes_ - 1]]
    loc.add(ex)
    for i, j in pick:
        sub = [list(e) for e in ex[i:j + 1]]
        sub[0][0] = max(sub[0][0], sub[0][1] - 200 + int(rng.integers(0, 100)))
        sub[-1][1] = sub[-1][1] - int(rng.integers(0, 100))
        loc.add(sub)
    for _ in range(dups):
        loc.add([(base + int(rng.integers(0, 50)), ex[0][1])] + ex[1:-1] + [(ex[-1][0], ex[-1][1] + int(rng.integers(-80, 80)))])
    # annotation: every donor of the long chain, none of its acceptors
    loc.anno = [(0, [(e - 20, e) for _, e in ex[:-1]] + [(ex[-1][0] - 20, ex[-1][1] + 100)])]
    loc.survivors, loc.novel, loc.classes = 1, 1, n_classes_
    return _order(loc)


def stairs(name, tid, base, steps, variants=3, copies=2, singles=0, seed=0, strands=False):
    """A staircase of `steps` groups 1000 apart, each a long chain (`variants` acceptors: classes) that reaches 2.5 steps ahead, a short
    chain inside the group's first 150 bases, copies of the long chains that start after the short chain ends, and short-chain
    duplicates whose jittered last end may or may not reach past that start.  A copy is absorbed by its long chain only when the
    back-scan gets past the short entry (update_gtf.c:148, the start against T.end as earlier absorptions extended it); otherwise the
    copy stays as one more survivor of its class.  Jitter of first starts / last ends makes end_dis decide identity too."""
    rng = np.random.default_rng(seed)
    loc = Locus(name, tid, base)
    donors = []
    for k in range(steps):
        s = base + 1000 * k
        r = lambda: int(rng.integers(0, 2)) if strands else 0      # noqa: E731
        sd, ld = s + 70, s + 200
        donors += [sd, ld]
        for v in range(variants):
            loc.add([(s + int(rng.integers(0, 20)), ld), (s + 301 + 10 * v, s + 3500 + int(rng.integers(-30, 30)))], r())
        loc.add([(s + 50, sd), (s + 91, s + 120 + int(rng.integers(0, 10)))], r())
        for _ in range(copies):
            ls = s + 120 + int(rng.integers(0, 60))
            loc.add([(ls, ld), (s + 301 + 10 * int(rng.integers(0, variants)), s + 3500 + int(rng.integers(-30, 30)))], r())
            loc.add([(s + 50 + int(rng.integers(-3, 4)), sd), (s + 91, s + 110 + int(rng.integers(0, 80)))], r())
        for _ in range(singles):
            a = s + int(rng.integers(0, 600))
            loc.add([(a, a + 100 + int(rng.integers(0, 300)))], r())
    loc.anno = [(0, [(d - 15, d) for d in sorted(donors)] + [(base + 1000 * steps + 4000, base + 1000 * steps + 4100)])]
    loc.classes = steps * (variants + 1)
    return _order(loc)


# ------------------------------------------------------------------------------------------------------------------ batches
def moved(loc: Locus, tid: int, base: int) -> Locus:
    """The same locus on chromosome `tid` at `base` (chains and annotation shifted together)."""
    d = base - loc.base
    mv = lambda ex: [(s + d, e + d) for s, e in ex]      # noqa: E731
    return Locus(loc.name, tid, base, [(r, mv(ex)) for r, ex in loc.chains], [(r, mv(ex)) for r, ex in loc.anno], loc.survivors,
                 loc.classes, loc.novel)


def chains_of(loci):
    """Exon chains (update-gtf -m g / unique-gtf input) of loci on their chromosomes, in (tid, start) order, and the locus of each."""
    loci = sorted(loci, key=lambda l: (l.tid, l.base))
    tid, rev, off, es, ee, owner = [], [], [0], [], [], []
    for li, l in enumerate(loci):
        for r, ex in l.chains:
            tid.append(l.tid); rev.append(r); owner.append(li)
            es += [s for s, _ in ex]; ee += [e for _, e in ex]; off.append(len(es))
    ch = dict(n_reads=len(tid), tid=np.array(tid, np.int32), is_rev=np.array(rev, np.uint8), exon_off=np.array(off, np.uint32),
              exon_start=np.array(es, np.int32), exon_end=np.array(ee, np.int32), read_idx=None)
    return ch, np.array(owner, np.int64), loci


def upload_form(ch):
    return {k: ch[k] for k in ("tid", "is_rev", "exon_off", "exon_start", "exon_end")}


def anno_of(loci):
    """The loci's annotation transcripts as an lrb_anno table ((tid, start) order, one gene each)."""
    loci = sorted(loci, key=lambda l: (l.tid, l.base))
    tid, st, en, rev, gene, off, es, ee = [], [], [], [], [], [0], [], []
    for l in loci:
        for r, ex in l.anno:
            tid.append(l.tid); st.append(ex[0][0]); en.append(ex[-1][1]); rev.append(r); gene.append(len(gene))
            es += [s for s, _ in ex]; ee += [e for _, e in ex]; off.append(len(es))
    i32 = lambda a: np.array(a, np.int32)      # noqa: E731
    return dict(tid=i32(tid), start=i32(st), end=i32(en), is_rev=np.array(rev, np.uint8), gene=i32(gene),
                exon_off=np.array(off, np.uint32), exon_start=i32(es), exon_end=i32(ee))


def survivors_per_locus(cand, owner, n_loci_):
    """Entries of a fold's output (updated_T / unique list) per locus; `cand` maps entries to chains (rows).  An entry is never removed
    once appended, so this is the fold's survivor count of each locus."""
    return np.bincount(owner[np.asarray(cand, np.int64)], minlength=n_loci_)


def novel_owner(update_out, owner):
    """Locus of each novel_T entry of an update-gtf result (updated_T's cand indexes novel_T)."""
    return owner[update_out["novel"]["read"].astype(np.int64)]
