"""Both classification kernels against the CPU port.

launch_classify (lr2rmats_b200/csrc/lrb_update.cu) classifies the common case (-d 0, at most 32 exons, monotone chains) with
classify_row_kernel and leaves the rest to classify_kernel, which implements the same rules without those restrictions.  On the
synthetic data almost every row takes the row kernel, so the general kernel's -d 0 path would go untested.  A context created with
LRB_TEST_CLASSIFY_GENERAL=1 never launches the row kernel and sends every row through classify_kernel.  Each case below runs
update-gtf once on an ordinary context and once on such a context; both must equal the port on every output array, and the second
must have launched exactly one kernel fewer."""
import os

import pytest

from lr2rmats_b200 import cabi, synth
from tests import oracle_port as op
from tests.test_gpu_parity import assert_dict_equal

pytestmark = pytest.mark.gpu

EP = cabi.ExonParams.default()


def _context(general):
    from lr2rmats_b200 import api
    old = os.environ.get("LRB_TEST_CLASSIFY_GENERAL")
    os.environ["LRB_TEST_CLASSIFY_GENERAL"] = "1" if general else "0"      # read by lrb_ctx_create
    try:
        return api.Context(0)
    finally:
        if old is None:
            del os.environ["LRB_TEST_CLASSIFY_GENERAL"]
        else:
            os.environ["LRB_TEST_CLASSIFY_GENERAL"] = old


@pytest.fixture(scope="module")
def ctxs():
    row, general = _context(False), _context(True)
    yield row, general
    general.close()
    row.close()


@pytest.fixture(scope="module")
def data():
    """The seeded data of test_gpu_parity: per shape the kept reads, their chains (port) and a short-read SJ table."""
    anno = synth.make_annotation(1500, n_chrom=4, seed=21)
    rr = synth.make_rrna(anno, 40, seed=22)
    out = dict(anno=anno.soa())
    for which, n, seed, ont in (("iso", 30000, 23, False), ("ont", 4000, 24, True)):
        r = synth.make_reads(anno, n, seed=seed, ont=ont, reject_frac=0.2, rrna=rr)
        kept = r.take(op.filter(r.soa(), rr, cabi.FilterParams.default())["keep_idx"])
        chains = op.bam2gtf(kept.soa(), EP)
        sj = synth.make_sj((chains["tid"], chains["exon_off"], chains["exon_start"], chains["exon_end"]), 0.7, seed=5)
        out[which] = (kept.soa(), chains, sj)
    return out


def run_both(ctxs, data, which, sj_on, up):
    kept, chains, sj = data[which]
    sj = sj if sj_on else None
    rc, o = op.update(chains, data["anno"], sj, up)
    assert rc == 0
    launches = []
    for ctx in ctxs:
        ctx.set_anno(data["anno"]); ctx.set_sj(sj)
        n0 = ctx.launch_count()
        g = ctx.update_gtf(kept, EP, up)
        launches.append(ctx.launch_count() - n0)
        o["ex"]["read_idx"] = g["ex"]["read_idx"]
        assert_dict_equal(g, o, "general kernel" if ctx is ctxs[1] else "row kernel")
    assert launches[1] == launches[0] - 1, f"classify_row_kernel must not run under the hook: launches {launches}"
    return o


@pytest.mark.parametrize("which", ["iso", "ont"])
@pytest.mark.parametrize("sj_on", [False, True])
@pytest.mark.parametrize("level", [1, 2, 3, 4, 5])
def test_levels(ctxs, data, which, sj_on, level):
    o = run_both(ctxs, data, which, sj_on, cabi.UpdateParams.default(full_level=level))
    assert len(o["updated"]["cand"]) > 0


# -s, -c, -e 30, and -j / -J (min_sj_cnt / use_multi): each with the SJ table, where the short-read support is checked
@pytest.mark.parametrize("which", ["iso", "ont"])
@pytest.mark.parametrize("kw", [dict(split_trans=1), dict(force_strand=1), dict(end_dis=30), dict(min_sj_cnt=3),
                                dict(use_multi=1, min_sj_cnt=3, split_trans=1)])
def test_options(ctxs, data, which, kw):
    up = cabi.UpdateParams.default(**dict(dict(full_level=3), **kw))
    o = run_both(ctxs, data, which, True, up)
    assert (o["cls"] & cabi.C_SJ_CHECKED).any(), "the fixture must exercise the short-read SJ check"
    if kw.get("split_trans"):
        assert (o["novel"]["piece"] >= 0).sum() > 0, "the fixture must exercise split pieces"
