"""Result lifetime (include/lr2rmats_b200.h): the arrays a fetch hands out stay valid until the next fetch of the SAME kind.  Each test
keeps the raw result struct of one kind, copies its arrays right after the fetch, lets other kinds run and fetch on the same context,
and checks that the struct's arrays still hold what they held.  The other kind runs once beforehand as well, so that its pinned
buffers already have their full size: the check then reads memory that stays allocated however the kinds share it."""
import ctypes as C

import numpy as np
import pytest

from lr2rmats_b200 import cabi, synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from lr2rmats_b200 import api
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def data():
    anno = synth.make_annotation(300, n_chrom=2, seed=81)
    rr = synth.make_rrna(anno, 10, seed=82)
    reads = synth.make_reads(anno, 8000, seed=83, ont=False, reject_frac=0.2, rrna=rr)
    return dict(anno=anno, rr=rr, reads=reads, sj=synth.make_sj_from_reads(reads, frac=0.7, seed=84))


def assert_same(a, b, path=""):
    assert set(a) == set(b), path
    for k in a:
        if isinstance(a[k], dict):
            assert_same(a[k], b[k], path + "/" + k)
        elif isinstance(a[k], np.ndarray):
            assert np.array_equal(a[k], b[k]), f"{path}/{k} changed"
        else:
            assert a[k] == b[k], f"{path}/{k} changed"


def test_filter_result_survives_sort3_and_bam2sj(ctx, data):
    r = data["reads"]
    soa = dict(r.soa())
    flag = soa["flag"].copy()
    flag[:150] |= np.uint16(3)                      # a few proper pairs: bam2sj writes junctions only for them
    soa["flag"] = flag
    uniq = np.ones(r.n, np.uint8)
    rng = np.random.default_rng(85)
    keys = [rng.integers(0, 1 << 20, r.n // 4).astype(np.uint32) for _ in range(3)]
    ctx.set_rm(data["rr"])
    ctx.upload(soa)
    ctx.filter_run(cabi.FilterParams.default())
    ctx.sort3(*keys)
    ctx.bam2sj(soa, uniq, cabi.SjParams.default())
    ctx.upload(soa)
    ctx.filter_run(cabi.FilterParams.default())

    res = cabi.FilterResult()
    ctx._ck(ctx.L.lrb_filter_fetch(ctx.h, C.byref(res)))
    want = cabi.filter_to_np(res)
    assert res.n == r.n and 0 < res.n_keep < r.n

    ctx.sort3(*keys)
    assert_same(cabi.filter_to_np(res), want, "filter after sort3")
    sj = ctx.bam2sj(soa, uniq, cabi.SjParams.default())
    assert len(sj["tid"]) > 0
    assert_same(cabi.filter_to_np(res), want, "filter after bam2sj")


def test_update_result_survives_unique(ctx, data):
    fp, ep = cabi.FilterParams.default(), cabi.ExonParams.default()
    up = cabi.UpdateParams.default(want_summary=1)
    ctx.set_anno(data["anno"].soa()); ctx.set_rm(data["rr"]); ctx.set_sj(data["sj"])
    ctx.upload(data["reads"].soa())
    ctx.pipeline_run(fp, ep)
    ctx.unique_run(up)
    ctx.unique_fetch()

    res = cabi.UpdateResult()
    ctx.update_run(up)
    ctx._ck(ctx.L.lrb_update_fetch(ctx.h, C.byref(res)))
    want = cabi.update_to_np(res)
    assert res.updated.n > 0 and res.bed.n > 0

    ctx.unique_run(up)
    q = ctx.unique_fetch()
    assert len(q["uniq"]["cand"]) > 0
    got = cabi.update_to_np(res)
    assert_same(got["updated"], want["updated"], "updated")
    assert_same(got["bed"], want["bed"], "bed")
    assert_same(got, want, "update result")
