// main.cpp -- the product binary `lr2rmats-b200`: the drop-in CLI (cli.cpp) bound to the CUDA library through the C ABI.
// There is no CPU engine in this binary: without a CUDA device every subcommand fails loudly.
#include <cstdio>
#include <cstdlib>
#include <future>
#include <unistd.h>
#include "lrb_host.h"

namespace {
// The CUDA context (driver initialisation, a second or more on a multi-GPU box) is created on a helper thread while the
// subcommand decodes its input files; the first engine call joins it.
struct CudaEngine {
    lrb_ctx *ctx = nullptr; std::future<int> pending;
    lrb_ctx *get()
    {
        if (pending.valid()) {
            int rc = pending.get();
            if (rc != LRB_OK) {
                fprintf(stderr, "[lr2rmats-b200] cannot create a CUDA context (code %d): this build has no CPU fallback\n", rc);
                exit(2);
            }
        }
        return ctx;
    }
};

int set_tables(void *s, const lrb_anno *a, const lrb_anno *rm, const lrb_sj *sj)
{
    lrb_ctx *c = ((CudaEngine *)s)->get(); int rc;
    if ((rc = lrb_anno_upload(c, a))) return rc;
    if ((rc = lrb_rm_upload(c, rm))) return rc;
    return lrb_sj_upload(c, sj);
}
// A batch goes to the device with its CIGAR pool (lrb_batch_upload).  When that, or a later stage of the same engine call, runs out
// of device memory, the call runs once more with the batch attached (lrb_batch_attach: the pool streams from host memory through
// the walk).  Every engine call is a pure function of its inputs, so the second run gives what the first would have.
// LRB_TEST_CHUNK_OPS=n (test hook): every call takes the attached path from the start, in chunks of n ops.
int64_t test_chunk_ops() { static const int64_t n = getenv("LRB_TEST_CHUNK_OPS") ? atoll(getenv("LRB_TEST_CHUNK_OPS")) : 0; return n; }
template <class F> int with_pool_fallback(F &&call)
{
    if (test_chunk_ops() > 0) return call(test_chunk_ops());
    const int rc = call(-1);
    return rc == LRB_E_NOMEM ? call(0) : rc;
}
// chunk_ops < 0: upload the batch, pool included; otherwise attach it with chunks of chunk_ops ops (0: the library's choice)
int load(lrb_ctx *c, const lrb_batch *b, int64_t chunk_ops) { return chunk_ops < 0 ? lrb_batch_upload(c, b) : lrb_batch_attach(c, b, chunk_ops); }

int do_filter(void *s, const lrb_batch *b, const lrb_filter_params *p, lrb_filter_result *o)
{
    lrb_ctx *c = ((CudaEngine *)s)->get();
    return with_pool_fallback([&](int64_t k) { int rc;
        if ((rc = load(c, b, k)) || (rc = lrb_filter_run(c, p))) return rc;
        return lrb_filter_fetch(c, o); });
}
int do_bam2gtf(void *s, const lrb_batch *b, const lrb_exon_params *p, lrb_exon_result *o)
{
    lrb_ctx *c = ((CudaEngine *)s)->get();
    return with_pool_fallback([&](int64_t k) { int rc;
        if ((rc = load(c, b, k)) || (rc = lrb_exon_run(c, p, 0))) return rc;
        return lrb_exon_fetch(c, o); });
}
int do_sort3(void *s, const uint32_t *a, const uint32_t *b, const uint32_t *c, int64_t n, const uint32_t **perm) { return lrb_sort3(((CudaEngine *)s)->get(), a, b, c, n, perm); }
int do_bam2sj(void *s, const lrb_batch *b, const uint8_t *u, const lrb_sj_params *p, lrb_sj *o) { return lrb_bam2sj(((CudaEngine *)s)->get(), b, u, p, o); }
// LRB_SORT_INPUT=1: update-gtf takes a BAM that is NOT coordinate sorted (filter's output as it is) and sorts the rows on the
// device -- the `samtools sort` hop of the pipeline (Snakefile:90) without the extra BAM round trip
bool sort_input() { static const bool on = getenv("LRB_SORT_INPUT") && atoi(getenv("LRB_SORT_INPUT")) != 0; return on; }

// the rows of an update / unique run: the batch's exon chains (b), or the given chains (-m g)
int load_rows(lrb_ctx *c, const lrb_batch *b, const lrb_chains *ch, const lrb_exon_params *ep, int64_t chunk_ops)
{
    int rc;
    if (!b) return lrb_chains_upload(c, ch);
    if ((rc = load(c, b, chunk_ops))) return rc;
    return lrb_exon_run(c, ep, 0);
}
int do_update(void *s, const lrb_batch *b, const lrb_chains *ch, const lrb_exon_params *ep, const lrb_update_params *up, lrb_update_result *o)
{
    lrb_ctx *c = ((CudaEngine *)s)->get();
    return with_pool_fallback([&](int64_t k) { int rc;
        if ((rc = load_rows(c, b, ch, ep, k))) return rc;
        if (sort_input() && (rc = lrb_rows_sort(c))) return rc;
        if ((rc = lrb_update_run(c, up))) return rc;
        return lrb_update_fetch(c, o); });
}
int do_update_table(void *s, const lrb_batch *b, const lrb_chains *ch, const lrb_exon_params *ep, const lrb_update_params *up,
                    lrb_trans_table *tab, lrb_bed_list *bed, int32_t *summary)
{
    lrb_ctx *c = ((CudaEngine *)s)->get();
    return with_pool_fallback([&](int64_t k) { int rc;
        if ((rc = load_rows(c, b, ch, ep, k))) return rc;
        if (sort_input() && (rc = lrb_rows_sort(c))) return rc;
        if ((rc = lrb_update_run(c, up))) return rc;
        return lrb_update_fetch_table(c, tab, bed, summary); });
}
int do_unique(void *s, const lrb_batch *b, const lrb_chains *ch, const lrb_exon_params *ep, const lrb_update_params *up, lrb_unique_result *o)
{
    lrb_ctx *c = ((CudaEngine *)s)->get();
    return with_pool_fallback([&](int64_t k) { int rc;
        if ((rc = load_rows(c, b, ch, ep, k)) || (rc = lrb_unique_run(c, up))) return rc;
        return lrb_unique_fetch(c, o); });
}
const char *err(void *s) { return lrb_last_error(((CudaEngine *)s)->get()); }
}  // namespace

int main(int argc, char **argv)
{
    CudaEngine ce; lrb::Engine eng;
    if (argc >= 3) {                                  // usage-only invocations need no device
        const char *dev = getenv("LRB_DEVICE");
        const int device = dev ? atoi(dev) : 0;
        ce.pending = std::async(std::launch::async, [&ce, device] { return lrb_ctx_create(device, &ce.ctx); });
    }
    eng.self = &ce; eng.set_tables = set_tables; eng.filter = do_filter; eng.bam2gtf = do_bam2gtf; eng.bam2sj = do_bam2sj; eng.sort3 = do_sort3; eng.update = do_update; eng.update_table = getenv("LRB_FULL_FETCH") ? nullptr : do_update_table;
    eng.unique = do_unique; eng.error = err;
    lrb::IoTrace tr;
    int rc = lrb::cli_main(argc, argv, eng);
    if (ce.pending.valid()) ce.pending.wait();        // usage errors return before any engine call
    // orderly teardown: leaving the context to the driver's process cleanup (_exit) was measured to slow down the context
    // creation of the NEXT process by more than a second (LRB_QUICK_EXIT=1 keeps that variant)
    if (getenv("LRB_QUICK_EXIT")) { fflush(NULL); tr.lap("total"); _exit(rc); }
    if (ce.ctx) lrb_ctx_destroy(ce.ctx);
    tr.lap("total");
    return rc;
}
