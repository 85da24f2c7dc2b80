"""The qname-run selection of the filter against the port, on batches built so that the failing records sit where a selection could go
wrong: inside runs (failing by FLAG 4, by low coverage, by rRNA overlap), in stretches longer than a tile of the walk between two
records of one run, everywhere between a passing first and a passing last record, and everywhere.  The filter result of lrb_filter,
of lrb_filter_run and of lrb_pipeline_run, and the exon chains of lrb_filter_run + lrb_exon_run(use_keep_list) and of
lrb_pipeline_run, must equal the port's, with the batch uploaded and attached."""
import numpy as np
import pytest

from lr2rmats_b200 import cabi, synth
from tests import oracle_port as op
from tests.test_gpu_parity import assert_dict_equal, filter_valid

pytestmark = pytest.mark.gpu

FP, EP = cabi.FilterParams.default(), cabi.ExonParams.default()
TILE = {"iso": 256, "ont": 32}                      # records per tile of the walk: short CIGARs / long CIGARs (> 48 ops per record)
FAIL = ("unmapped", "lowcov", "rrna")


@pytest.fixture(scope="module")
def donors():
    """Per shape a batch and its records by filter outcome: passing, failing by low coverage, failing by rRNA overlap only."""
    anno = synth.make_annotation(800, n_chrom=3, seed=41)
    rr = synth.make_rrna(anno, 40, seed=42)
    out = dict(rr=rr)
    for which, n, ont in (("iso", 6000, False), ("ont", 1500, True)):
        r = synth.make_reads(anno, n, seed=43, ont=ont, reject_frac=0.4, rrna=rr)
        with_rm, without = op.filter(r.soa(), rr, FP)["pass_"].astype(bool), op.filter(r.soa(), None, FP)["pass_"].astype(bool)
        first = r.cigar[r.cigar_off[:-1].astype(np.int64)]
        clip = np.where((first & 15) == 4, first >> 4, 0).astype(np.int64)
        lowcov = (r.l_qseq - clip) / r.l_qseq < FP.cov_rate
        pools = dict(pass_=np.nonzero(with_rm)[0], lowcov=np.nonzero(lowcov & ((r.flag & 4) == 0))[0], rrna=np.nonzero(without & ~with_rm)[0])
        assert all(len(p) >= 20 for p in pools.values()), {k: len(p) for k, p in pools.items()}
        out[which] = (r, pools)
    return out


def assemble(donor, spec, seed):
    """The batch of spec = [(kind, qname id)], kind "pass" or one of FAIL; an unmapped record is a passing one with FLAG 4 set."""
    r, pools = donor
    rng = np.random.default_rng(seed)
    kinds = [k for k, _ in spec]
    idx = [int(rng.choice(pools["pass_" if k in ("pass", "unmapped") else k])) for k in kinds]
    b = r.take(np.asarray(idx, np.int64))
    b.flag = np.where(np.array([k == "unmapped" for k in kinds], bool), b.flag | 4, b.flag).astype(np.uint16)
    b.qname_hash = synth.splitmix64(np.asarray([q for _, q in spec], np.int64))
    return b


def failing(rng, n, qids):
    """n failing records of every kind, each with one of qids."""
    return [(FAIL[i % 3], int(rng.choice(qids))) for i in rng.permutation(n)]


def make_spec(which, case, seed):
    rng = np.random.default_rng(seed)
    stretch = 2 * TILE[which] + TILE[which] // 2 + 7
    if case == "empty":
        return []
    if case == "runs":                              # runs of 1-4 passing records with failing ones inside, of its qname or another
        spec, q = [], 1000
        for _ in range({"iso": 900, "ont": 250}[which]):
            q = q - 2 if rng.random() < 0.1 else q + 1          # now and then a qname seen two runs back
            recs = [("pass", q)] * int(rng.integers(1, 5)) + failing(rng, int(rng.integers(0, 4)), [q, q + 50000])
            spec += [recs[i] for i in rng.permutation(len(recs))]
        return spec
    if case == "split":                             # one run cut by more than two tiles of failing records, runs around it
        head = [("pass", 1), ("pass", 1), ("pass", 2)]
        return head + [("pass", 7)] + failing(rng, stretch, [7, 8, 9]) + [("pass", 7), ("pass", 7)] + [("pass", 10), ("lowcov", 10), ("pass", 11)]
    if case in ("ends_one_run", "ends_two_runs"):   # passing records at 0 and n - 1 only
        return [("pass", 5)] + failing(rng, stretch, [5, 6, 7]) + [("pass", 5 if case == "ends_one_run" else 6)]
    if case == "all_fail":
        return failing(rng, 4 * stretch, list(range(40)))
    raise ValueError(case)


@pytest.fixture(scope="module")
def ctx():
    from lr2rmats_b200 import api
    c = api.Context(0)
    yield c
    c.close()


CASES = ["runs", "split", "ends_one_run", "ends_two_runs", "all_fail", "empty"]


@pytest.mark.parametrize("load", ["upload", "attach"])
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("which", ["iso", "ont"])
def test_filter_selection_matches_port(ctx, donors, which, case, load):
    b = assemble(donors[which], make_spec(which, case, seed=CASES.index(case)), seed=7)
    soa, rr = b.soa(), donors["rr"]
    if b.n:                                         # the walk runs in the tile shape the case is built for
        assert (int(b.cigar_off[-1]) > 48 * b.n) == (which == "ont")
    of = op.filter(soa, rr, FP)
    oe = op.bam2gtf(soa, EP, sel=of["keep_idx"])
    want = filter_valid(of)
    if case in ("split", "ends_one_run", "ends_two_runs"):
        assert b.n > 2 * TILE[which]
    if case == "all_fail":
        assert not want["pass_"].any()
    ctx.set_rm(rr)

    def put():
        if load == "upload":
            ctx.upload(soa)
        else:
            ctx.attach(soa, max(1, int(b.cigar_off[-1]) // 5))

    # (each fetch is compared before the next one reuses its pinned buffers)
    if load == "upload":
        assert_dict_equal(filter_valid(ctx.filter(soa, FP)), want, "lrb_filter")
    put(); ctx.filter_run(FP)
    assert_dict_equal(filter_valid(ctx.filter_fetch()), want, "filter_run")
    ctx.exon_run(EP, use_keep_list=True)
    assert_dict_equal(ctx.exon_fetch(), oe, "filter_run + exon_run(use_keep_list)")
    put(); ctx.pipeline_run(FP, EP)
    assert_dict_equal(filter_valid(ctx.filter_fetch()), want, "pipeline_run")
    assert_dict_equal(ctx.exon_fetch(), oe, "pipeline_run exons")
