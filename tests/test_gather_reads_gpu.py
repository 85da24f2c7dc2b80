"""lrb_update_gather_reads / lrb_gather_fetch_reads: the per-read results of a sharded run, gathered on rank 0, against what one GPU
returns for the whole stream (lrb_update_fetch + lrb_filter_fetch) and against the numpy concatenation of the ranks' own fetches
(tests/test_gather_reads_port.py).  The one-rank cases run on one GPU; the N-rank cases need N visible GPUs."""
import ctypes as C
import os
import pickle
import subprocess
import sys

import numpy as np
import pytest

from lr2rmats_b200 import api, cabi, multi, synth
from tests.test_gather_reads_port import concat_filter, concat_update, per_read
from tests.test_gpu_parity import assert_dict_equal, filter_valid
from tests.test_multi_gpu import n_gpus, workload
from tests.test_result_lifetime import assert_same

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
FP, EP = cabi.FilterParams.default(), cabi.ExonParams.default()


def one_rank(anno, rr, sj):
    ctx = api.Context(0)
    ctx.comm_init(api.comm_id(), 0, 1)
    ctx.tables_broadcast(0, anno.soa(), rr, sj)
    return ctx


@pytest.mark.parametrize("split,summary", [(1, 1), (0, 1), (1, 0), (0, 0)])
def test_one_rank_equals_fetch(split, summary):
    anno, rr, reads, sj = workload(40_000, 2000)
    up = cabi.UpdateParams.default(full_level=3, split_trans=split, min_sj_cnt=1, want_summary=summary)
    ctx = one_rank(anno, rr, sj)
    got = multi.run_shard(ctx, reads.soa(), 0, FP, EP, up, reads=True)["reads"]
    want_u, want_f = ctx.update_fetch(), ctx.filter_fetch()
    ctx.comm_destroy(); ctx.close()
    assert_dict_equal(got["update"], want_u)
    assert_dict_equal(got["filter"], want_f)
    assert len(want_u["known_idx"]) and len(want_u["unrecog_idx"]) and len(want_u["updated"]["cand"]) > 1000
    assert not split or (want_u["novel"]["piece"] >= 0).any()
    assert (len(want_u["bed"]["tid"]) > 0) == bool(summary)


def test_one_rank_chains_have_no_read_idx():
    anno, rr, reads, sj = workload(20_000, 1500)
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)
    ex = api.Context(0)
    ex.set_rm(rr); ex.upload(reads.soa()); ex.pipeline_run(FP, EP)
    chains = ex.exon_fetch(); ex.close()
    ctx = one_rank(anno, rr, sj)
    ctx.upload_chains({k: chains[k] for k in ("tid", "is_rev", "exon_off", "exon_start", "exon_end")})
    ctx.update_run(up)
    ctx.update_gather(0); ctx.update_gather_reads(0)
    got = ctx.gather_fetch_reads(want_filter=False)["update"]
    want = ctx.update_fetch()
    with pytest.raises(api.LrbError) as e:
        ctx.gather_fetch_reads(want_update=False)            # no filter stage ran
    ctx.comm_destroy(); ctx.close()
    assert e.value.code == -2
    assert got["ex"]["read_idx"] is None and want["ex"]["read_idx"] is None
    assert_dict_equal(got, want)
    assert len(want["updated"]["cand"]) > 500


def test_one_rank_results_outlive_other_fetches():
    """The gather-reads result kind has pinned buffers of its own: its structs survive lrb_gather_fetch, lrb_update_fetch and
    lrb_filter_fetch, and theirs survive it."""
    anno, rr, reads, sj = workload(20_000, 1500)
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)
    ctx = one_rank(anno, rr, sj)
    multi.run_shard(ctx, reads.soa(), 0, FP, EP, up, fetch=False, reads=True)
    ctx.gather_fetch(); ctx.update_fetch(); ctx.filter_fetch(); ctx.gather_fetch_reads()     # every kind at full size once
    gu, gf = ctx.gather_fetch_reads(raw=True)
    want_g = (cabi.update_to_np(gu), cabi.filter_to_np(gf))
    ctx.gather_fetch()
    u = cabi.UpdateResult(); ctx._ck(ctx.L.lrb_update_fetch(ctx.h, C.byref(u)))
    f = cabi.FilterResult(); ctx._ck(ctx.L.lrb_filter_fetch(ctx.h, C.byref(f)))
    want_u, want_f = cabi.update_to_np(u), cabi.filter_to_np(f)
    assert_same(cabi.update_to_np(gu), want_g[0], "gathered update after the other fetches")
    assert_same(cabi.filter_to_np(gf), want_g[1], "gathered filter after the other fetches")
    ctx.gather_fetch_reads()
    assert_same(cabi.update_to_np(u), want_u, "update after gather_fetch_reads")
    assert_same(cabi.filter_to_np(f), want_f, "filter after gather_fetch_reads")
    ctx.comm_destroy(); ctx.close()
    assert gu.updated.n > 0 and gu.bed.n > 0 and gf.n_keep > 0


def test_one_rank_update_needs_table_gather():
    anno, rr, reads, sj = workload(10_000, 1000)
    ctx = one_rank(anno, rr, sj)
    ctx.upload(reads.soa()); ctx.pipeline_run(FP, EP); ctx.update_run(cabi.UpdateParams.default(full_level=3, min_sj_cnt=1))
    ctx.update_gather_reads(0)
    with pytest.raises(api.LrbError) as e:
        ctx.gather_fetch_reads()
    f = ctx.gather_fetch_reads(want_update=False)["filter"]
    want = ctx.filter_fetch()
    # a table gather of an EARLIER update run does not go with these reads either
    ctx.update_gather(0)
    ctx.update_run(cabi.UpdateParams.default(full_level=5, min_sj_cnt=1))
    ctx.update_gather_reads(0)
    with pytest.raises(api.LrbError) as e2:
        ctx.gather_fetch_reads()
    ctx.update_gather(0)
    got = ctx.gather_fetch_reads(want_filter=False)["update"]
    want_u = ctx.update_fetch()
    ctx.comm_destroy(); ctx.close()
    assert e.value.code == -2 and e2.value.code == -2
    assert_dict_equal(f, want)
    assert_dict_equal(got, want_u)


# ---------------------------------------------------------------------------------------------------------- N ranks
def single_gpu(anno, rr, reads, sj, up):
    ctx = api.Context(0)
    ctx.set_anno(anno.soa()); ctx.set_rm(rr); ctx.set_sj(sj)
    ctx.upload(reads.soa()); ctx.pipeline_run(FP, EP); ctx.update_run(up)
    u, f = ctx.update_fetch(), ctx.filter_fetch()
    ctx.close()
    return u, f


def run_world(tmp_path, world, anno_soa, rr, reads, sj, cuts=None, split=1, summary=1, level=3, run_shard=False):
    wl = tmp_path / "wl.npz"
    d = {"b_" + k: v for k, v in reads.soa().items()}
    d.update({"a_" + k: v for k, v in anno_soa.items()}); d.update({"r_" + k: v for k, v in rr.items()}); d.update({"s_" + k: v for k, v in sj.items()})
    d.update(p_full_level=level, p_split=split, p_summary=summary)
    if cuts is not None:
        d["cuts"] = np.asarray(cuts, np.int64)
    if run_shard:
        d["p_run_shard"] = 1
    np.savez(wl, **d)
    procs = [subprocess.Popen([sys.executable, os.path.join(HERE, "gather_reads_worker.py"), str(wl), str(tmp_path), str(r), str(world)],
                              stderr=subprocess.PIPE, stdout=subprocess.PIPE) for r in range(world)]
    for p in procs:
        try:
            out, err = p.communicate(timeout=600)
        except subprocess.TimeoutExpired:
            for q in procs: q.kill()
            raise
        assert p.returncode == 0, err.decode()[-3000:]
    load = lambda name: pickle.load(open(tmp_path / name, "rb"))
    if run_shard:
        return [load(f"run_shard{r}.pkl") for r in range(world)]
    return load("merged.pkl"), [load(f"rank{r}.pkl") for r in range(world)]


def check_world(got, ranks, want_u, want_f):
    assert got["code"] == 0 and got["update_code"] == 0
    assert_dict_equal(got["update"], want_u)
    assert_dict_equal(filter_valid(got["filter"]), filter_valid(want_f))
    bases = got["cuts"][:-1]
    assert_dict_equal(per_read(got["update"]), concat_update([per_read(r["update"]) for r in ranks], bases))
    assert_dict_equal(got["filter"], concat_filter([r["filter"] for r in ranks], bases))


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("shape", ["iso", "ont"])
def test_gathered_reads_equal_single_gpu(tmp_path, world, shape):
    if n_gpus() < world:
        pytest.skip(f"needs {world} GPUs")
    anno, rr, reads, sj = workload(60_000 if shape == "ont" else 200_000, 8000, ont=(shape == "ont"))
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)
    want_u, want_f = single_gpu(anno, rr, reads, sj, up)
    got, ranks = run_world(tmp_path, world, anno.soa(), rr, reads, sj)
    assert len(set(got["cuts"].tolist())) == world + 1, "degenerate shards"
    check_world(got, ranks, want_u, want_f)
    assert (want_u["novel"]["piece"] >= 0).any()


@pytest.mark.parametrize("empty_rank", [0, 1])
def test_empty_shard(tmp_path, empty_rank):
    if n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    anno, rr, reads, sj = workload(40_000, 2000)
    up = cabi.UpdateParams.default(full_level=3, split_trans=1, min_sj_cnt=1, want_summary=1)
    want_u, want_f = single_gpu(anno, rr, reads, sj, up)
    cuts = [0, 0, reads.n] if empty_rank == 0 else [0, reads.n, reads.n]
    got, ranks = run_world(tmp_path, 2, anno.soa(), rr, reads, sj, cuts=cuts)
    assert ranks[empty_rank]["filter"]["pass_"].size == 0
    check_world(got, ranks, want_u, want_f)


def test_after_cross_shard_piece(tmp_path):
    """The table gather reports LRB_E_XSHARD on the root (the workload of test_cross_shard_piece_is_reported); every rank still
    returns from the per-read gather, the root's update fetch has no BED rows / counters to give, its filter fetch does."""
    if n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    anno = synth.make_annotation(1500, n_chrom=2, seed=41)
    rr = synth.make_rrna(anno, 10, seed=42)
    reads = synth.make_reads(anno, 20_000, seed=43, reject_frac=0.2, rrna=rr)
    sj = synth.make_sj_from_reads(reads, frac=0.7, seed=44)
    a2, both, s2 = synth.clone_chromosome(anno.soa(), reads, sj, 2)
    ctx = api.Context(0)
    ctx.set_rm(rr); ctx.upload(both.soa()); ctx.pipeline_run(FP, EP)
    want_f = ctx.filter_fetch(); ctx.close()
    got, ranks = run_world(tmp_path, 2, a2, rr, both, s2)
    assert got["code"] == -8 and got["update_code"] == -2
    assert_dict_equal(filter_valid(got["filter"]), filter_valid(want_f))
    assert_dict_equal(got["filter"], concat_filter([r["filter"] for r in ranks], got["cuts"][:-1]))


def test_run_shard_after_cross_shard_piece(tmp_path):
    """multi.run_shard(..., reads=True) on the workload above: the root's table gather raises LRB_E_XSHARD, the other ranks' does
    not; every rank still joins the per-read gather and returns (none is left waiting in the collective)."""
    if n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    anno = synth.make_annotation(1500, n_chrom=2, seed=41)
    rr = synth.make_rrna(anno, 10, seed=42)
    reads = synth.make_reads(anno, 20_000, seed=43, reject_frac=0.2, rrna=rr)
    sj = synth.make_sj_from_reads(reads, frac=0.7, seed=44)
    a2, both, s2 = synth.clone_chromosome(anno.soa(), reads, sj, 2)
    codes = [r["code"] for r in run_world(tmp_path, 2, a2, rr, both, s2, run_shard=True)]
    assert codes == [-8, 0]
