"""One rank of a sharded run that gathers the per-read results (tests/test_gather_reads_gpu.py spawns `world` of these, one per GPU).
usage: gather_reads_worker.py <workload.npz> <out_dir> <rank> <world>
The workload may fix the shard cuts ("cuts"); otherwise multi.plan_shards picks them.  With "p_run_shard" the rank runs
multi.run_shard(..., reads=True) and only records what it raised.  Every rank writes its own update / filter
fetch to rank<r>.pkl; rank 0 also writes what lrb_update_gather returned and the gathered per-read results to merged.pkl."""
import os
import pickle
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lr2rmats_b200 import api, cabi, multi  # noqa: E402


def main():
    path, out, rank, world = sys.argv[1], sys.argv[2], int(sys.argv[3]), int(sys.argv[4])
    z = np.load(path)
    batch = {k[2:]: z[k] for k in z.files if k.startswith("b_")}
    idf = os.path.join(out, "comm.id")
    if rank == 0:
        open(idf + ".tmp", "wb").write(api.comm_id()); os.rename(idf + ".tmp", idf)
    t0 = time.time()
    while not os.path.exists(idf):
        if time.time() - t0 > 120: sys.exit("no communicator id")
        time.sleep(0.05)
    ctx = api.Context(rank)
    ctx.comm_init(open(idf, "rb").read(), rank, world)
    tabs = [None, None, None]
    if rank == 0:
        tabs = [{k[2:]: z[k] for k in z.files if k.startswith(p)} for p in ("a_", "r_", "s_")]
    ctx.tables_broadcast(0, *tabs)
    cuts = z["cuts"] if "cuts" in z.files else multi.plan_shards(batch, world)
    up = cabi.UpdateParams.default(full_level=int(z["p_full_level"]), split_trans=int(z["p_split"]), min_sj_cnt=1, want_summary=int(z["p_summary"]))
    lo, hi = int(cuts[rank]), int(cuts[rank + 1])
    if "p_run_shard" in z.files:
        try:
            multi.run_shard(ctx, multi.take_shard(batch, lo, hi), lo, cabi.FilterParams.default(), cabi.ExonParams.default(), up, reads=True)
            code = 0
        except api.LrbError as e:
            code = e.code
        with open(os.path.join(out, f"run_shard{rank}.pkl"), "wb") as f:
            pickle.dump(dict(code=code), f)
        ctx.comm_destroy(); ctx.close()
        return
    ctx.upload(multi.take_shard(batch, lo, hi))
    ctx.pipeline_run(cabi.FilterParams.default(), cabi.ExonParams.default())
    ctx.update_run(up)
    try:
        ctx.update_gather(lo)
        code = 0
    except api.LrbError as e:
        code = e.code
    ctx.update_gather_reads(lo)                     # on every rank, whatever the table gather returned
    with open(os.path.join(out, f"rank{rank}.pkl"), "wb") as f:
        pickle.dump(dict(update=ctx.update_fetch(), filter=ctx.filter_fetch()), f)
    if rank == 0:
        d = dict(code=code, cuts=np.asarray(cuts))
        try:
            d["update"] = ctx.gather_fetch_reads(want_filter=False)["update"]
            d["update_code"] = 0
        except api.LrbError as e:
            d["update_code"] = e.code
        d["filter"] = ctx.gather_fetch_reads(want_update=False)["filter"]
        with open(os.path.join(out, "merged.pkl"), "wb") as f:
            pickle.dump(d, f)
    ctx.comm_destroy(); ctx.close()


if __name__ == "__main__":
    main()
