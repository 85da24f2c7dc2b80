// lrb_capi.cu -- the C ABI of liblr2rmats_b200.so (include/lr2rmats_b200.h): context, HBM residency, stage
// orchestration on one CUDA stream, pinned result buffers.  No compute happens on the host here beyond building the
// small lookup indices of the replicated tables (prefix-max keys, the remove-GTF index) at upload time.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include "lrb_ctx.cuh"

using namespace lrbk;

namespace {

// r backed by `cols`, sized for cap rows (r.n stays the caller's)
int setup_rows(lrb_ctx *c, DRows &r, RowsCols<Buf> &cols, int64_t cap)
{
    if (int rc = ensure(c, cols, Extent{std::max<int64_t>(cap, 1)})) return rc;
    r = view(cols, r); r.cap = cap;
    return LRB_OK;
}
int setup_list(lrb_ctx *c, DTransList &l, ListCols<Buf> &cols, int64_t n)
{
    if (int rc = ensure(c, cols, Extent{std::max<int64_t>(n, 1)})) return rc;
    l = view(cols, DTransList{n, n});
    return LRB_OK;
}
int setup_exons(lrb_ctx *c, int64_t cap)
{
    size_t n = (size_t)std::max<int64_t>(cap, 1);
    NEED(c->e_s, n * 4); NEED(c->e_e, n * 4); NEED(c->e_f, n);
    c->ex.cap = (int64_t)std::min(c->e_s.cap / 4, std::min(c->e_e.cap / 4, c->e_f.cap));
    c->ex.es = c->e_s.as<int32_t>(); c->ex.ee = c->e_e.as<int32_t>(); c->ex.flag = c->e_f.as<uint8_t>();
    return LRB_OK;
}

// tiles of the CIGAR walk: short CIGARs (Iso-Seq like) are walked thread per read on staged tiles of 256 reads, long CIGARs
// (ONT like) by the streaming kernel on warp tiles
bool scan_stream_mode(int64_t n, int64_t n_cigar) { return n > 0 && (double)n_cigar / (double)n > 48.0; }
int scan_tile_reads(bool stream_mode) { return stream_mode ? stream_reads_per_tile() : scan_reads_per_tile(); }

// the CIGAR walk of one scan attempt (look-back state zeroed by the caller): one launch over the resident pool, or the chunks of an
// attached pool.  A chunk's launch takes its tiles from its first one on, so its first tile looks back at the last tile of the
// chunk before, complete by then (same stream): rows and exons are placed as by one launch, with no host round trip in between.
int walk_cigars(lrb_ctx *c, ScanArgs a, int n_tiles, bool stream_mode, size_t smem)
{
    c->n_chunks_walked = 0; c->max_staged_ops = 0;
    if (!c->attached) {
        a.ops = c->b.cigar; a.op_base = 0; a.tile_base = 0;
        CK(cudaMemsetAsync(a.ticket, 0, 4, c->st));
        launch_cigar_scan(a, n_tiles, stream_mode, smem, c->st);
        return LRB_OK;
    }
    // + 4 words: the last bulk copy of the streaming kernel rounds its length up to 16 bytes
    for (Buf &s : c->stage) NEED(s, (size_t)(c->stage_ops + 4) * 4);
    const size_t nk = c->chunks.size();
    auto copy_chunk = [&](size_t k) -> int {         // chunk k -> staging buffer k & 1, once the walk of chunk k - 2 is done with it
        const OpChunk &ch = c->chunks[k]; const int s = (int)(k & 1);
        CK(cudaStreamWaitEvent(c->st_copy, c->ev_walked[s], 0));
        if (ch.op_end > ch.op_base)
            CK(cudaMemcpyAsync(c->stage[s].p, c->h_cigar + ch.op_base, (size_t)(ch.op_end - ch.op_base) * 4, cudaMemcpyHostToDevice, c->st_copy));
        CK(cudaEventRecord(c->ev_copied[s], c->st_copy));
        return LRB_OK;
    };
    int rc;
    if (nk && (rc = copy_chunk(0))) return rc;
    for (size_t k = 0; k < nk; ++k) {
        if (k + 1 < nk && (rc = copy_chunk(k + 1))) return rc;
        const OpChunk &ch = c->chunks[k]; const int s = (int)(k & 1);
        CK(cudaStreamWaitEvent(c->st, c->ev_copied[s], 0));
        a.ops = c->stage[s].as<uint32_t>(); a.op_base = ch.op_base; a.tile_base = ch.tile0;
        CK(cudaMemsetAsync(a.ticket, 0, 4, c->st));
        launch_cigar_scan(a, ch.tile1 - ch.tile0, stream_mode, smem, c->st);
        CK(cudaEventRecord(c->ev_walked[s], c->st));
        c->max_staged_ops = std::max<int64_t>(c->max_staged_ops, (int64_t)(ch.op_end - ch.op_base));
    }
    c->n_chunks_walked = (int64_t)nk;
    return LRB_OK;
}

// the scan stage in one of its three modes: 0 filter, 1 exon chains (of the records in sel_mask, or of all), 2 both in one fused pass.
// On return the counts are known on the host.  A walk that computes the filter is followed by the qname-run selection on the record
// stream and the ordered compaction of the kept records: into the keep list (mode 0), or into the keep list and the kept rows, rows2
// (mode 2, whose walk writes the rows at their record index).  Mode 0 writes no rows.  Rows, exons and kept records come back in one
// round trip.  If the exon pool was too small the walk is repeated once with its exact size (all chunks of an attached pool again).
int run_scan(lrb_ctx *c, int mode, const lrb_filter_params *fp, const lrb_exon_params *ep, const uint8_t *sel_mask)
{
    const int64_t n = c->b.n;
    const bool do_filter = mode != 1, do_exon = mode != 0;
    int rc;
    if ((rc = ensure_tiles(c, n)) != LRB_OK) return rc;
    if (do_exon && (rc = setup_rows(c, c->rows, c->rows_cols, n)) != LRB_OK) return rc;
    if (do_filter) {
        NEED(c->f_pass, (size_t)n + 1); NEED(c->f_score, (size_t)n * 4 + 4); NEED(c->f_intron, (size_t)n * 4 + 4);
        NEED(c->f_keep_rec_mask, (size_t)n + 1); NEED(c->f_keep_idx, (size_t)n * 4 + 4);
    }
    if (mode == 2 && (rc = setup_rows(c, c->rows2, c->rows2_cols, n)) != LRB_OK) return rc;
    // the counts of a walk, t = (rows, exons, kept records); the fused pass's rows are indexed by record
    auto take = [&](const uint64_t *t) {
        c->ex.n = (int64_t)t[1];
        if (do_filter) c->n_keep = (int64_t)t[2];
        if (do_exon) c->rows.n = mode == 2 ? n : (int64_t)t[0];
        if (mode == 2) c->rows2.n = c->n_keep;
    };
    if (n == 0) { const uint64_t none[3] = {0, 0, 0}; take(none); return do_exon ? setup_exons(c, 16) : LRB_OK; }
    const double avg = (double)c->b.n_cigar / (double)n;
    const bool stream_mode = scan_stream_mode(n, c->b.n_cigar);
    const int R = scan_tile_reads(stream_mode);
    int stage_words = (int)(R * avg * 1.3) + 256; stage_words = (stage_words + 255) & ~255; stage_words = std::max(2048, std::min(12288, stage_words));
    if (stream_mode) stage_words = 0;
    const int n_tiles = (int)((n + R - 1) / R);
    if (mode != 0) {
        int64_t bound = c->b.n_cigar + n + 16, est = c->b.n_cigar / 2 + n + 4096;
        rc = setup_exons(c, std::min(bound, std::max(est, c->ex.cap)));
        // the estimate is 4.5 B per op, more than the pool: an attached batch that cannot hold it walks once to count its exons
        // (the walk writes none when they do not fit), then again with the exact size
        if (rc == LRB_E_NOMEM && c->attached) rc = setup_exons(c, n + 4096);
        if (rc != LRB_OK) return rc;
    }
    for (int attempt = 0;; ++attempt) {
        ScanArgs a{};
        a.b = c->b; if (fp) a.fp = *fp; if (ep) a.ep = *ep; a.rm = c->rm; a.mode = mode; a.sel_mask = sel_mask;
        a.pass = c->f_pass.as<uint8_t>(); a.score = c->f_score.as<int32_t>(); a.intron_n = c->f_intron.as<int32_t>();
        a.rows = c->rows; a.ex = c->ex; a.tile_state = c->tile_state.as<uint64_t>(); a.ticket = d_ticket(c); a.totals = d_totals(c);
        a.reads_per_tile = R; a.stage_words = stage_words; a.rows_by_record = mode == 2 ? 1 : 0;
        CK(cudaMemsetAsync(c->tile_state.p, 0, (size_t)n_tiles * 8, c->st));
        CK(cudaMemsetAsync(c->scalars.p, 0, 8 * 8, c->st));
        size_t smem = (size_t)stage_words * 4;
        tick(c, EV_SCAN0);
        if ((rc = walk_cigars(c, a, n_tiles, stream_mode, smem)) != LRB_OK) return rc;
        tick(c, EV_SCAN1);
        CK(cudaGetLastError());
        if (do_filter) {                             // run selection on the record stream -> compaction (+ row gather)
            uint8_t *keep = c->f_keep_rec_mask.as<uint8_t>();
            CK(cudaMemsetAsync(keep, 0, (size_t)n, c->st));
            launch_select_records(c->b, c->f_pass.as<uint8_t>(), c->f_score.as<int32_t>(), c->f_intron.as<int32_t>(), *fp, keep, c->st);
            if (mode == 2)
                launch_compact_gather(keep, n, c->rows, c->rows2, c->f_keep_idx.as<uint32_t>(), c->tile_state.as<uint64_t>(), d_ticket(c), d_totals(c) + 2, c->st);
            else launch_compact_mask(keep, n, c->f_keep_idx.as<uint32_t>(), c->tile_state.as<uint64_t>(), d_ticket(c), d_totals(c) + 2, c->st);
            CK(cudaGetLastError());
        }
        uint64_t t[3] = {0, 0, 0};
        if ((rc = read_totals(c, t, do_filter ? 3 : 2)) != LRB_OK) return rc;
        take(t);
        if (c->timing) cudaEventElapsedTime(&c->ms[LRB_T_K_SCAN], c->ev[EV_SCAN0], c->ev[EV_SCAN1]);
        if (!do_exon || c->ex.n <= c->ex.cap) return LRB_OK;
        if (attempt == 1) return fail(c, LRB_E_NOMEM, "exon pool still too small after regrow");
        if ((rc = setup_exons(c, c->ex.n + 16)) != LRB_OK) return rc;          // exact size known now: walk again
    }
}

// The stages that walk the CIGARs, run_scan in their mode: checks, timing, launch count, and what is current afterwards -- the filter
// result (modes 0, 2), the rows and exon chains (modes 1, 2).
int scan_stage(lrb_ctx *c, const char *who, int mode, const lrb_filter_params *fp, const lrb_exon_params *ep, bool use_keep_list)
{
    if (!c || (mode != 1 && !fp) || (mode != 0 && !ep)) return LRB_E_ARG;
    if (!c->have_batch) return fail(c, LRB_E_ARG, std::string(who) + ": no batch uploaded");
    if (use_keep_list && !c->have_filter) return fail(c, LRB_E_ARG, std::string(who) + ": keep list requested but lrb_filter_run has not run");
    CK(cudaSetDevice(c->device));
    const int64_t l0 = total_launches(); tick(c, EV_BEGIN);
    if (int rc = run_scan(c, mode, fp, ep, use_keep_list ? c->f_keep_rec_mask.as<uint8_t>() : nullptr)) return rc;
    tick(c, EV_END);
    if (mode != 1) c->have_filter = true;
    if (mode == 0) c->have_exons = false;
    else { c->cur = mode == 2 ? &c->rows2 : &c->rows; c->rows_compact = mode == 1; c->have_exons = true; c->have_update = c->have_unique = false; }
    c->launches_last = total_launches() - l0;
    if (c->timing) {
        CK(cudaStreamSynchronize(c->st));
        cudaEventElapsedTime(&c->ms[mode == 1 ? LRB_T_EXON : LRB_T_FILTER], c->ev[EV_BEGIN], c->ev[EV_END]);
        if (mode == 2) c->ms[LRB_T_EXON] = 0;
    }
    return LRB_OK;
}

int setup_merge(lrb_ctx *c, MergeBufs &m, int64_t n_cand)
{
    size_t n = (size_t)std::max<int64_t>(n_cand, 1);
    NEED(m.tlist, n * 8); NEED(m.head, n); NEED(m.locus_start, (n + 1) * 4); NEED(m.locus_cnt, n * 4); NEED(m.alive, n);
    NEED(m.rep, n * 4); NEED(m.lstart, n * 4); NEED(m.evmask, n * 8); NEED(m.samemask, n * 8); NEED(m.hard, n); NEED(m.desc, n * 2); NEED(m.relsym, n * 8); NEED(m.ckey, (2 * n + 64) * 8); NEED(m.cmin, (2 * n + 64) * 4); NEED(m.cord, n); NEED(m.clist, n * 4); NEED(m.crow, n * 16); NEED(m.fb_list, n * 8); NEED(m.fb_cnt, 64); NEED(m.fb_state, fold_resume_bytes((int64_t)n));
    const Extent e{(int64_t)n};
    int rc;
    if ((rc = ensure(c, m.w, e)) || (rc = ensure(c, m.o, e)) || (rc = ensure(c, m.cd, e))) return rc;
    return LRB_OK;
}

// what a merge fold does beyond folding its list
struct FoldOpts {
    const uint8_t *kls = nullptr;                   // set: every row is folded, as four independent sub-streams (class id per row) in one
    uint32_t *class_alive = nullptr;                // pass; the list is built here, in class order (launch_class_order), and only the
                                                    // survivors per sub-stream are counted (class_alive)
    bool time_fold = false;                         // EV_FOLD0 / EV_FOLD1 around the fold kernels
    bool side = false;                              // on the side stream, with its own look-back state
    bool single_locus = false;                      // the whole list is ONE locus: the back-scan replayed entry by entry
    bool xl = false;                                // split pieces that meet another chromosome are marked by the xl_* kernels
};

// merge fold over `list`, asynchronous.  n_cand is the number of candidates, or (n_cand_dev != nullptr) the host's upper
// bound of a count that lives on the device.  With o.kls `list` is only the storage the class-ordered list of every row is built in.
// Without o.kls the survivors are compacted into m.o_*.
// totals[0] <- number of loci, totals[1] <- number of survivors (device).
int run_merge_async(lrb_ctx *c, MergeBufs &m, const DTransList &list, int64_t n_cand, const uint64_t *n_cand_dev, const lrb_update_params &up,
                    uint64_t *totals, const FoldOpts &o)
{
    int rc;
    cudaStream_t st = o.side ? c->st2 : c->st;
    if ((rc = setup_merge(c, m, n_cand)) != LRB_OK) return rc;
    if (o.side) { NEED(c->tile_state2, (size_t)(n_cand / 8 + 1024) * 8); }
    else if ((rc = ensure_tiles(c, n_cand)) != LRB_OK) return rc;
    m.n_out = 0; m.n_loci = 0;
    CK(cudaMemsetAsync(totals, 0, 16, st));
    if (n_cand == 0) return LRB_OK;
    MergeArgs a{};
    a.rows = *c->cur; a.ex = c->ex; a.up = up; a.list = list; a.n_cand = n_cand; a.n_cand_dev = n_cand_dev;
    a.tlist = m.tlist.as<uint32_t>(); a.head = m.head.as<uint8_t>(); a.locus_start = m.locus_start.as<uint32_t>(); a.locus_cnt = m.locus_cnt.as<uint32_t>();
    a.alive = m.alive.as<uint8_t>();
    a.rep = m.rep.as<uint32_t>(); a.lstart = m.lstart.as<uint32_t>(); a.evmask = m.evmask.as<uint64_t>(); a.samemask = m.samemask.as<uint64_t>(); a.hard = m.hard.as<uint8_t>(); a.desc = m.desc.as<uint16_t>(); a.relsym = m.relsym.as<uint64_t>(); a.ckey = m.ckey.as<uint64_t>(); a.cmin = m.cmin.as<uint32_t>(); a.cord = m.cord.as<uint8_t>(); a.clist = m.clist.as<uint32_t>(); a.crow = m.crow.as<uint64_t>(); a.fb_list = m.fb_list.as<uint32_t>(); a.fb_cnt = m.fb_cnt.as<uint32_t>(); a.fb_state = m.fb_state.p;
    a.n_indexed = c->fold_census ? a.fb_cnt + 5 : nullptr;
    a.work = view(m.w, DMerged{n_cand, n_cand}); a.out = view(m.o, DMerged{n_cand, n_cand}); a.cd = view(m.cd, CandSoA{});
    a.tile_state = o.side ? c->tile_state2.as<uint64_t>() : c->tile_state.as<uint64_t>(); a.ticket = o.side ? d_ticket2(c) : d_ticket(c); a.totals = totals;
    a.kls = o.kls; a.class_alive = o.class_alive; a.single_locus = o.single_locus ? 1 : 0;
    if (o.xl) {
        // split pieces that meet another chromosome (xl_* kernels): marks per candidate, a key set sized for the pieces' junctions
        // (pieces are a small share of the candidates), lists in buffers the fold is done with by then
        const uint64_t tcap = std::max<uint64_t>(1u << 16, (uint64_t)n_cand / 2);
        NEED(c->xl_key, tcap * 8); NEED(c->xl_min, tcap * 4); NEED(c->xl_max, tcap * 4); NEED(c->xl_cnt, 64);
        a.forced = c->xl_forced.as<uint8_t>();
        c->xl = XlArgs{c->xl_key.as<unsigned long long>(), c->xl_min.as<uint32_t>(), c->xl_max.as<uint32_t>(), tcap, a.clist, a.lstart, (uint32_t)std::min<int64_t>(n_cand, 1 << 20),
                       a.relsym, c->xl_cnt.as<uint32_t>()};
    }
    if (o.kls) {
        NEED(m.cbase, ((size_t)n_cand + 1) * 16); NEED(m.cperm, (size_t)n_cand * 4); NEED(m.ckls, (size_t)n_cand);
        a.cbase = m.cbase.as<uint4>(); a.kls = m.ckls.as<uint8_t>(); a.presegmented = 1;
        launch_class_order(a, o.kls, m.cperm.as<uint32_t>(), m.ckls.as<uint8_t>(), st);
        DTransList rows_list = list;                // a view: its columns are the list's
        launch_rows_as_list(a.rows, m.cperm.as<uint32_t>(), n_cand, rows_list, st);
    }
    m.args = a;
    launch_merge_prepare(a, st);
    if (o.time_fold) tick(c, EV_FOLD0);
    launch_merge_fold(a, st);                        // locus count is consumed on the device: no host round trip
    if (o.time_fold) tick(c, EV_FOLD1);
    if (c->fold_census) CK(merge_fold_census(a, st, c->census[o.side ? 1 : 0]));
    if (o.xl) launch_xlocus_detect(a, c->xl, st);
    if (o.kls) launch_merge_class_counts(a, st);
    else launch_merge_finish(a, st);
    CK(cudaGetLastError());
    return LRB_OK;
}

int run_merge(lrb_ctx *c, MergeBufs &m, const DTransList &list, int64_t n_cand, const lrb_update_params &up, bool single_locus)
{
    int rc;
    FoldOpts o; o.time_fold = true; o.single_locus = single_locus;
    if ((rc = run_merge_async(c, m, list, n_cand, nullptr, up, d_totals(c), o)) != LRB_OK) return rc;
    uint64_t t[2];
    if ((rc = read_totals(c, t, 2)) != LRB_OK) return rc;
    m.n_loci = (int64_t)t[0]; m.n_out = (int64_t)t[1];
    if (c->timing && n_cand) cudaEventElapsedTime(&c->ms[LRB_T_K_FOLD], c->ev[EV_FOLD0], c->ev[EV_FOLD1]);
    return LRB_OK;
}

}  // namespace

// ====================================================================================================== C ABI
extern "C" {

const char *lrb_version(void) { return "lr2rmats_b200 0.1 (sm_100a)"; }

int lrb_ctx_create(int device, lrb_ctx **out)
{
    if (!out) return LRB_E_ARG;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { cudaGetLastError(); return LRB_E_NODEVICE; }
    if (device < 0 || device >= ndev) return LRB_E_ARG;
    if (cudaSetDevice(device) != cudaSuccess) { cudaGetLastError(); return LRB_E_CUDA; }
    lrb_ctx *c = new lrb_ctx();
    c->device = device;
    if (cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking) != cudaSuccess) { delete c; return LRB_E_CUDA; }
    if (cudaStreamCreateWithFlags(&c->st2, cudaStreamNonBlocking) != cudaSuccess) { cudaStreamDestroy(c->st); delete c; return LRB_E_CUDA; }
    cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming); cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming);
    if (cudaStreamCreateWithFlags(&c->st3, cudaStreamNonBlocking) != cudaSuccess) { cudaStreamDestroy(c->st2); cudaStreamDestroy(c->st); delete c; return LRB_E_CUDA; }
    cudaEventCreateWithFlags(&c->ev_fork3, cudaEventDisableTiming); cudaEventCreateWithFlags(&c->ev_join3, cudaEventDisableTiming);
    if (cudaStreamCreateWithFlags(&c->st_copy, cudaStreamNonBlocking) != cudaSuccess) { cudaStreamDestroy(c->st3); cudaStreamDestroy(c->st2); cudaStreamDestroy(c->st); delete c; return LRB_E_CUDA; }
    for (int i = 0; i < 2; ++i) { cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming); cudaEventCreateWithFlags(&c->ev_walked[i], cudaEventDisableTiming); }
    { const char *e = getenv("LRB_TEST_SMALL_NOVEL_CAP"); if (e) c->test_small_novel_cap = atoi(e) != 0; }      // test hook: novel_T sized too small on the first attempt
    { const char *e = getenv("LRB_FORCE_SINGLE_FOLD"); if (e) c->force_single_fold = atoi(e) != 0; }    // test hook: updated_T always folded by the one-locus replay
    { const char *e = getenv("LRB_TEST_FOLD_CENSUS"); if (e) c->fold_census = atoi(e) != 0; }       // test hook: loci tallied by fold path (lrb_fold_census)
    { const char *e = getenv("LRB_TEST_CLASSIFY_GENERAL"); if (e) c->classify_general = atoi(e) != 0; }   // test hook: every row through classify_kernel
    if (!c->scalars.ensure(512) || !c->h_scalars.ensure(512)) { delete c; return LRB_E_NOMEM; }
    cudaMemsetAsync(c->scalars.p, 0, 512, c->st);
    for (cudaEvent_t &e : c->ev) cudaEventCreate(&e);
    for (int i = 0; i < 8; ++i) cudaEventCreate(&c->marks[i]);
    memset(c->ms, 0, sizeof c->ms); memset(c->summary, 0, sizeof c->summary);
    c->launches0 = total_launches();
    *out = c;
    return LRB_OK;
}

void lrb_ctx_destroy(lrb_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->st); cudaStreamSynchronize(c->st2); cudaStreamSynchronize(c->st3); cudaStreamSynchronize(c->st_copy);
    lrbk::multi_release(c);
    for (cudaEvent_t e : c->ev) cudaEventDestroy(e);
    for (int i = 0; i < 8; ++i) cudaEventDestroy(c->marks[i]);
    cudaEventDestroy(c->ev_fork); cudaEventDestroy(c->ev_join);
    cudaEventDestroy(c->ev_fork3); cudaEventDestroy(c->ev_join3); cudaStreamDestroy(c->st3);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(c->ev_copied[i]); cudaEventDestroy(c->ev_walked[i]); }
    cudaStreamDestroy(c->st_copy);
    cudaStreamDestroy(c->st2); cudaStreamDestroy(c->st);
    delete c;                                       // frees the device and pinned buffers
}

const char *lrb_last_error(const lrb_ctx *c) { return c ? c->err.c_str() : "null context"; }

// -------------------------------------------------------------------------------------------------- tables
int lrb_anno_upload(lrb_ctx *c, const lrb_anno *a)
{
    if (!c) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    c->anno = DAnno{};
    if (!a || a->n_trans == 0) return LRB_OK;
    const int32_t n = a->n_trans;
    std::vector<uint64_t> pm((size_t)n);
    uint64_t run = 0;
    for (int32_t i = 0; i < n; ++i) {               // P_j, SURVEY App. B.1
        uint64_t k = ((uint64_t)(uint32_t)(a->tid[i] + 1) << 32) | (uint32_t)a->end[i];
        run = std::max(run, k); pm[(size_t)i] = run;
    }
    std::vector<uint8_t> mono((size_t)n);
    for (int32_t i = 0; i < n; ++i) {
        uint8_t m = 1;
        for (uint32_t k = a->exon_off[i] + 1; k < a->exon_off[i + 1]; ++k)
            if (a->exon_start[k] <= a->exon_start[k - 1] || a->exon_end[k] <= a->exon_end[k - 1]) { m = 0; break; }
        mono[(size_t)i] = m;
    }
    AnnoCols<const void *> src;
    src.tid = a->tid; src.start = a->start; src.end = a->end; src.gene = a->gene; src.is_rev = a->is_rev; src.exon_off = a->exon_off;
    src.es = a->exon_start; src.ee = a->exon_end; src.pmax_key = pm.data(); src.mono = mono.data();
    if (int rc = copy(c, c->anno_cols, src, Extent{n, a->n_exon}, cudaMemcpyHostToDevice)) return rc;
    CK(cudaStreamSynchronize(c->st));               // pm is a local
    c->anno = view(c->anno_cols, DAnno{n, a->n_exon});
    return LRB_OK;
}

int lrb_rm_upload(lrb_ctx *c, const lrb_anno *rmt)
{
    if (!c) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    c->rm = DRmIndex{};
    if (!rmt || rmt->n_trans == 0) return LRB_OK;
    // entries visible to remove_overlap()'s early exit (bam_filter.c:54-57): for a read on tid t the scan stops after the
    // first entry with tid > t, so only entries in front of it exist for t.  Group them per tid, sort by start, running max end.
    const int32_t n = rmt->n_trans;
    std::map<int32_t, std::vector<std::pair<int32_t, int32_t>>> groups;
    std::vector<int32_t> pmax_tid((size_t)n);
    int32_t run = INT32_MIN;
    for (int32_t i = 0; i < n; ++i) { run = std::max(run, rmt->tid[i]); pmax_tid[(size_t)i] = run; }
    for (int32_t i = 0; i < n; ++i) {
        int32_t t = rmt->tid[i];
        // visible iff no earlier-or-equal position has prefix max tid > t  <=>  pmax_tid[i] <= t (i itself has tid t)
        if (pmax_tid[(size_t)i] > t) continue;
        groups[t].push_back({rmt->start[i], rmt->end[i]});
    }
    std::vector<int32_t> gt, go{0}, st, pe;
    for (auto &g : groups) {
        std::sort(g.second.begin(), g.second.end());
        int32_t m = INT32_MIN;
        for (auto &iv : g.second) { m = std::max(m, iv.second); st.push_back(iv.first); pe.push_back(m); }
        gt.push_back(g.first); go.push_back((int32_t)st.size());
    }
    RmCols<const void *> src;
    src.g_tid = gt.data(); src.g_off = go.data(); src.start = st.data(); src.pmax_end = pe.data();
    if (int rc = copy(c, c->rm_cols, src, Extent{(int64_t)gt.size(), (int64_t)st.size()}, cudaMemcpyHostToDevice)) return rc;
    CK(cudaStreamSynchronize(c->st));
    c->rm = view(c->rm_cols, DRmIndex{(int32_t)gt.size(), (int32_t)st.size()});
    return LRB_OK;
}

int lrb_sj_upload(lrb_ctx *c, const lrb_sj *s)
{
    if (!c) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    c->sj = DSj{};
    if (!s || s->n == 0) return LRB_OK;
    const int64_t n = s->n;
    std::vector<uint64_t> pm((size_t)n), dk((size_t)n);
    uint64_t run = 0;
    for (int64_t i = 0; i < n; ++i) {               // Q_i, SURVEY App. B.2
        uint64_t k = ((uint64_t)(uint32_t)(s->tid[i] + 1) << 32) | (uint32_t)s->acc[i];
        run = std::max(run, k); pm[(size_t)i] = run;
        dk[(size_t)i] = ((uint64_t)(uint32_t)(s->tid[i] + 1) << 32) | (uint32_t)s->don[i];
        if (i && dk[(size_t)i] < dk[(size_t)i - 1]) return fail(c, LRB_E_ARG, "SJ table is not sorted by (tid,don,acc)");
    }
    SjCols<const void *> src;
    src.tid = s->tid; src.don = s->don; src.acc = s->acc; src.cnt_u = s->uniq_c; src.cnt_m = s->multi_c; src.pmax_key = pm.data(); src.don_key = dk.data();
    if (int rc = copy(c, c->sj_cols, src, Extent{n}, cudaMemcpyHostToDevice)) return rc;
    CK(cudaStreamSynchronize(c->st));
    c->sj = view(c->sj_cols, DSj{n});
    return LRB_OK;
}

// --------------------------------------------------------------------------------------------------- batch
// the fixed-width columns of b -> HBM, and the CIGAR pool with them unless it stays in host memory (attach: chunk_ops >= 0)
static int load_batch(lrb_ctx *c, const lrb_batch *b, int64_t chunk_ops)
{
    if (!c || !b || b->n < 0) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    const bool attach = chunk_ops >= 0;
    const size_t n = (size_t)b->n;
    const size_t nc = n ? b->cigar_off[n] : 0;
    if (b->n >= (1ll << 31) - 1) return fail(c, LRB_E_ARG, "batch too large: at most 2^31-2 records per batch");
    if (n && b->cigar_off[0] != 0) return fail(c, LRB_E_ARG, "cigar_off[0] must be 0");
    if (nc >= (1ull << 40)) return fail(c, LRB_E_ARG, "batch too large: at most 2^40 CIGAR ops per batch");
    c->have_batch = false; c->attached = false; c->h_cigar = nullptr; c->chunks.clear();
    if (attach) c->batch_cols.cigar.release();      // the pool's device column is returned before anything else is sized
    else { c->stage[0].release(); c->stage[1].release(); }
    static const uint64_t no_cigar = 0;             // cigar_off of an empty batch
    BatchCols<const void *> src;
    src.tid = b->tid; src.pos = b->pos; src.l_qseq = b->l_qseq; src.nm = b->nm; src.flag = b->flag; src.xs = b->xs; src.qhash = b->qname_hash;
    src.cigar_off = n ? b->cigar_off : &no_cigar; src.cigar = b->cigar;
    if (int rc = copy(c, c->batch_cols, src, Extent{(int64_t)n, attach ? 0 : (int64_t)nc}, cudaMemcpyHostToDevice)) return rc;
    c->b = view(c->batch_cols, DBatch{b->n, (int64_t)nc});
    if (attach) {
        c->batch_cols.cigar.release(); c->b.cigar = nullptr;      // (copy() sized it for an empty pool)
        if (chunk_ops == 0) {                       // two staging buffers of at most 1/64 of the free memory each, 4 MB .. 256 MB
            size_t fr = 0, tot = 0;
            CK(cudaMemGetInfo(&fr, &tot));
            chunk_ops = std::max<int64_t>(1 << 20, std::min<int64_t>(1 << 26, (int64_t)(fr / 64 / 4)));
        }
        // chunks of whole tiles, staged from op_base = (the first tile's first op) rounded down to a multiple of 4; a chunk takes
        // tiles while its staged ops stay within chunk_ops, and at least one
        const bool sm = scan_stream_mode((int64_t)n, (int64_t)nc);
        const int64_t R = scan_tile_reads(sm), n_tiles = ((int64_t)n + R - 1) / R;
        auto tile_end = [&](int64_t t) { return b->cigar_off[std::min<int64_t>((int64_t)n, (t + 1) * R)]; };
        c->stage_ops = 0;
        for (int64_t t = 0; t < n_tiles;) {
            OpChunk ch; ch.tile0 = (int)t; ch.op_base = b->cigar_off[t * R] & ~3ull;
            do ++t; while (t < n_tiles && tile_end(t) - ch.op_base <= (uint64_t)chunk_ops);
            ch.tile1 = (int)t; ch.op_end = tile_end(t - 1);
            c->chunks.push_back(ch);
            c->stage_ops = std::max<int64_t>(c->stage_ops, (int64_t)(ch.op_end - ch.op_base));
        }
        c->h_cigar = b->cigar; c->attached = true;
    }
    c->have_batch = true; c->have_filter = c->have_exons = c->have_update = c->have_unique = false;
    return LRB_OK;
}

int lrb_batch_upload(lrb_ctx *c, const lrb_batch *b) { return load_batch(c, b, -1); }

int lrb_batch_attach(lrb_ctx *c, const lrb_batch *b, int64_t chunk_ops)
{
    if (chunk_ops < 0) return LRB_E_ARG;
    return load_batch(c, b, chunk_ops);
}

// rows straight from exon chains (-m g input): start/end/ex_beg/ex_n derived on device
__global__ void chains_rows_kernel(DRows rows, const uint32_t *__restrict__ off, const int32_t *__restrict__ es, const int32_t *__restrict__ ee, int64_t n,
                                   uint8_t *nonmono)
{
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    uint32_t lo = off[r], hi = off[r + 1];
    uint8_t nm = 0;                                  // GTF chains may be anything; CIGAR chains always ascend
    for (uint32_t k = lo + 1; k < hi; ++k) if (es[k] < es[k - 1] || ee[k] < ee[k - 1]) nm = 1;
    nonmono[r] = nm;
    rows.read_idx[r] = (uint32_t)r; rows.ex_beg[r] = lo; rows.ex_n[r] = hi - lo;
    rows.start[r] = hi > lo ? es[lo] : 0; rows.end[r] = hi > lo ? ee[hi - 1] : 0;
}

int lrb_chains_upload(lrb_ctx *c, const lrb_chains *ch)
{
    if (!c || !ch || ch->n < 0) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    const int64_t n = ch->n; const int64_t ne = n ? ch->exon_off[n] : 0;
    int rc;
    if ((rc = setup_rows(c, c->rows, c->rows_cols, n))) return rc;
    if ((rc = setup_exons(c, ne + 16))) return rc;
    if ((rc = h2d(c, c->rows_cols.tid, ch->tid, (size_t)n))) return rc;
    if ((rc = h2d(c, c->rows_cols.is_rev, ch->is_rev, (size_t)n))) return rc;
    if ((rc = h2d(c, c->e_s, ch->exon_start, (size_t)ne))) return rc;
    if ((rc = h2d(c, c->e_e, ch->exon_end, (size_t)ne))) return rc;
    if ((rc = h2d(c, c->u_noff, ch->exon_off, (size_t)n + 1))) return rc;          // scratch for the offsets
    NEED(c->r_nonmono, (size_t)std::max<int64_t>(n, 1));
    if (n) { chains_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->st>>>(c->rows, c->u_noff.as<uint32_t>(), c->ex.es, c->ex.ee, n, c->r_nonmono.as<uint8_t>()); CK(cudaGetLastError()); }
    c->rows.n = n; c->ex.n = ne; c->cur = &c->rows; c->rows_compact = true;
    c->b.n = 0; c->have_batch = false; c->have_filter = false; c->have_exons = true; c->have_update = c->have_unique = false;
    return LRB_OK;
}

// -------------------------------------------------------------------------------------------------- stages
int lrb_filter_run(lrb_ctx *c, const lrb_filter_params *p) { return scan_stage(c, "lrb_filter_run", 0, p, nullptr, false); }
int lrb_exon_run(lrb_ctx *c, const lrb_exon_params *p, int use_keep_list) { return scan_stage(c, "lrb_exon_run", 1, nullptr, p, use_keep_list != 0); }
int lrb_pipeline_run(lrb_ctx *c, const lrb_filter_params *fp, const lrb_exon_params *ep) { return scan_stage(c, "lrb_pipeline_run", 2, fp, ep, false); }

// the error flags of the update / unique input checks (d_err) as a status
static int err_status(lrb_ctx *c, uint32_t e)
{
    if (e & 2u) return fail(c, LRB_E_UNMAPPED, "unmapped record / empty exon chain in update/unique input (the reference aborts here, bam2gtf.c:95-100)");
    if (e & 1u) return fail(c, LRB_E_UNSORTED, "reads are not sorted by (tid,start) (update_gtf.c:41)");
    return LRB_OK;
}

static int check_err_flags(lrb_ctx *c, uint32_t *flags)
{
    CK(cudaMemcpyAsync(c->h_scalars.p, d_err(c), 4, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    memcpy(flags, c->h_scalars.p, 4);
    return err_status(c, *flags);
}

__global__ void invert_mask_kernel(const uint8_t *a, uint8_t *o, int64_t n)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) o[i] = !a[i];
}

// empty-chain / sortedness check for unique (classification does it for update)
__global__ void rows_check_kernel(DRows rows, uint32_t *err, int check_sorted)
{
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows.n) return;
    if (rows.ex_n[r] == 0) atomicOr(err, 2u);
    if (check_sorted && r > 0) {                     // bit 2: not sorted by (tid,start) -- allowed for unique (a concatenation of samples)
        const int pt = rows.tid[r - 1], ps = rows.start[r - 1], ct = rows.tid[r], cs = rows.start[r];
        if (pt > ct || (pt == ct && ps > cs)) atomicOr(err, 4u);
    }
}

// ---- the update stage in steps; what one step hands to the next
struct UpdateRun {
    const lrb_update_params *up;
    bool xl_exact, detect, run_sets, single;        // see lrb_update_run
    int64_t cap, n_novel;                           // novel_T: capacity, entries
    SummaryArgs sa;                                 // the summary sets over updated_T (run_sets)
};

// the stage's round trips through h_scalars (UpdateScalars): the copies `parts` names, in this order, then one synchronization.
// RB_SCALARS: totals, ticket, error flags.  RB_SET_COUNTS: y_counts without the class sizes, which keep the value of an earlier read.
enum { RB_SCALARS = 1, RB_BED = 2, RB_COUNTS = 4, RB_SET_COUNTS = 8, RB_NELEM = 16, RB_XL = 32 };
static int read_back(lrb_ctx *c, unsigned parts)
{
    UpdateScalars *hs = c->h_scalars.as<UpdateScalars>();
    if (parts & RB_SCALARS) CK(cudaMemcpyAsync(hs, c->scalars.p, T_SLOTS * 8 + 8, cudaMemcpyDeviceToHost, c->st));
    if (parts & RB_BED) CK(cudaMemcpyAsync(&hs->t[T_BED], d_totals(c) + T_BED, 8, cudaMemcpyDeviceToHost, c->st));
    if (parts & (RB_COUNTS | RB_SET_COUNTS)) CK(cudaMemcpyAsync(hs->counts, c->y_counts.p, (parts & RB_COUNTS) ? 64 : 48, cudaMemcpyDeviceToHost, c->st));
    if (parts & RB_NELEM) CK(cudaMemcpyAsync(&hs->n_elem, c->y_nelem.p, 16, cudaMemcpyDeviceToHost, c->st));
    if (parts & RB_XL) CK(cudaMemcpyAsync(hs->xl, c->xl_cnt.p, XL_NCNT * 4, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    return LRB_OK;
}

// The class folds run on the side stream.  The main stream waits for them before their counters are read or reset, and before the
// stage returns early: they share the context's buffers and counters with whatever runs next.
static int join_class_folds(lrb_ctx *c, const lrb_update_params *up)
{
    if (up->want_summary) CK(cudaStreamWaitEvent(c->st, c->ev_join, 0));
    return LRB_OK;
}

// classification (+ SJ support)
static int update_classify(lrb_ctx *c, const lrb_update_params *up)
{
    DRows &rows = *c->cur; const int64_t n = rows.n; const size_t nn = (size_t)std::max<int64_t>(n, 1);
    int rc;
    NEED(c->u_cls, nn * 4); NEED(c->u_ref, nn * 4); NEED(c->u_nnovel, nn * 4);
    NEED(c->u_mk, nn); NEED(c->u_known, nn * 4); NEED(c->u_unrecog, nn * 4); NEED(c->u_ck, nn);
    NEED(c->y_counts, 64); NEED(c->y_nelem, 64);       // y_nelem: element count, then (at +16) the six tickets of sum_scans_kernel
    if ((rc = ensure_tiles(c, std::max<int64_t>(n, c->ex.n)))) return rc;
    CK(cudaMemsetAsync(d_err(c), 0, 4, c->st));
    tick(c, EV_BEGIN);
    ClassArgs ca{};
    ca.rows = rows; ca.ex = c->ex; ca.anno = c->anno; ca.sj = c->sj; ca.up = *up;
    ca.row_nonmono = c->have_batch ? nullptr : c->r_nonmono.as<uint8_t>();
    ca.cls = c->u_cls.as<uint32_t>(); ca.ref = c->u_ref.as<int32_t>(); ca.n_novel = c->u_nnovel.as<uint32_t>(); ca.err_flags = d_err(c);
    launch_classify(ca, c->classify_general ? nullptr : c->u_mk.as<uint8_t>(), c->st);     // u_mk: scratch for the slow-row mask
    CK(cudaGetLastError());
    tick(c, EV_CLASSIFIED);
    return LRB_OK;
}

// Lists, the updated_T fold, the class folds and the element count of the summary sets: one stream of launches, every count stays on
// the device; ONE copy brings them all back.  novel_T is sized optimistically (pieces are rare); if it turns out too small the step is
// repeated once with the exact size.  The class folds are left running on the side stream underneath the steps that follow.
static int update_lists_and_folds(lrb_ctx *c, UpdateRun &u, int pass)
{
    const lrb_update_params *up = u.up;
    DRows &rows = *c->cur; const int64_t n = rows.n;
    uint64_t *T = d_totals(c);
    const UpdateScalars &hs = *c->h_scalars.as<UpdateScalars>();
    int rc;
    if (n == 0) {
        if ((rc = setup_list(c, c->novel, c->novel_cols, 0))) return rc;
        c->mg.n_out = c->mg.n_loci = 0; tick(c, EV_LISTED); tick(c, EV_FOLDED);
        u.n_novel = 0;
        return LRB_OK;
    }
    for (int attempt = 0;; ++attempt) {
        if ((rc = setup_list(c, c->novel, c->novel_cols, u.cap))) return rc;
        CK(cudaMemsetAsync(c->y_counts.p, 0, 64, c->st)); CK(cudaMemsetAsync(c->y_nelem.p, 0, 16, c->st));
        ListArgs la{};
        la.rows = rows; la.ex = c->ex; la.up = *up; la.cls = c->u_cls.as<uint32_t>(); la.n_novel = c->u_nnovel.as<uint32_t>(); la.novel = c->novel;
        la.known = c->u_known.as<uint32_t>(); la.unrecog = c->u_unrecog.as<uint32_t>();
        la.kls = up->want_summary ? c->u_ck.as<uint8_t>() : nullptr; la.class_n = c->y_counts.as<uint32_t>() + 12;
        la.tile_state = c->tile_state.as<uint64_t>(); la.ticket = d_ticket(c); la.totals = T + T_NOVEL;
        launch_build_lists(la, c->st);
        CK(cudaGetLastError());
        if (attempt == 0 && pass == 0) tick(c, EV_LISTED);
        if (up->want_summary) {
            // class counts + uniq_* folds over bam_T (update_gtf.c:501-528): the four classes partition the rows; they are
            // folded in ONE pass over all rows, each candidate seeing only the entries of its own class.  Independent of the
            // updated_T fold and of the sets: forked onto the side stream.
            if ((rc = setup_list(c, c->tmp_list, c->tmp_cols, n))) return rc;
            CK(cudaEventRecord(c->ev_fork, c->st)); CK(cudaStreamWaitEvent(c->st2, c->ev_fork, 0));
            FoldOpts o; o.kls = c->u_ck.as<uint8_t>(); o.class_alive = c->y_counts.as<uint32_t>() + 8; o.side = true;
            if ((rc = run_merge_async(c, c->mg2, c->tmp_list, n, nullptr, *up, T + T_LOCI2, o))) return rc;
            CK(cudaEventRecord(c->ev_join, c->st2));
        }
        // updated_T = merge fold over novel_T (update_gtf.c:949,956)
        if (u.xl_exact) { NEED(c->xl_forced, (size_t)std::max<int64_t>(u.cap, 1)); CK(cudaMemsetAsync(c->xl_forced.p, 0, (size_t)std::max<int64_t>(u.cap, 1), c->st)); }
        FoldOpts o; o.time_fold = true; o.single_locus = u.single; o.xl = u.xl_exact;
        if ((rc = run_merge_async(c, c->mg, c->novel, u.cap, T + T_NOVEL, *up, T + T_LOCI, o))) return rc;
        if (attempt == 0 && pass == 0) tick(c, EV_FOLDED);
        if (u.run_sets) {
            // sets over updated_T: element count (sizes the hash table)
            const size_t capn = (size_t)std::max<int64_t>(u.cap, 1);
            NEED(c->y_barcnt, capn * 16); NEED(c->y_barseg, capn * 16); NEED(c->y_genebar, capn * 8); NEED(c->y_bedcnt, capn * 4); NEED(c->y_bedoff, capn * 4);
            SummaryArgs &sa = u.sa;
            sa = SummaryArgs{}; sa.sets = up->want_summary ? SUM_ALL : 0; sa.probe = u.detect ? 1 : 0;
            sa.rows = rows; sa.ex = c->ex; sa.list = c->novel; sa.n_upd = u.cap; sa.n_upd_dev = T + T_UPD;
            sa.upd = view(c->mg.o, DMerged{u.cap, u.cap});
            sa.ref = c->u_ref.as<int32_t>(); sa.anno_gene = c->anno.gene;
            sa.bar_cnt = c->y_barcnt.as<uint32_t>(); sa.bar_seg = c->y_barseg.as<uint32_t>(); sa.gene_bar = c->y_genebar.as<uint64_t>();
            sa.bed_cnt = c->y_bedcnt.as<uint32_t>(); sa.bed_off = c->y_bedoff.as<uint32_t>(); sa.counts = c->y_counts.as<uint32_t>();
            launch_summary_count(sa, c->y_nelem.as<unsigned long long>(), c->st);
            CK(cudaGetLastError());
        }
        // the one round trip: totals, error flags, class sizes, element count
        if ((rc = read_back(c, RB_SCALARS | RB_COUNTS | RB_NELEM | (u.xl_exact ? RB_XL : 0)))) return rc;
        if (hs.err & 3u) { join_class_folds(c, up); return err_status(c, hs.err); }
        u.n_novel = (int64_t)hs.t[T_NOVEL]; c->n_known = (int64_t)hs.t[T_KNOWN]; c->n_unrecog = (int64_t)hs.t[T_UNREC];
        if (u.n_novel <= u.cap) break;
        if ((rc = join_class_folds(c, up))) return rc;          // novel_T did not fit: the counters are reset for one more attempt
        if (attempt >= 1) return fail(c, LRB_E_CUDA, "novel_T size changed between passes");
        u.cap = u.n_novel; c->novel_cap_hint = u.n_novel + u.n_novel / 16;
    }
    c->mg.n_loci = (int64_t)hs.t[T_LOCI]; c->mg.n_out = (int64_t)hs.t[T_UPD];
    return LRB_OK;
}

// Split pieces absorbed by an entry on another chromosome (xl_exact): fold again with the marks until they are stable (round k fixes the
// k-th affected piece at the latest), then let the absorbing entries take cov / ends, compact and count again.  *settled = false: more
// hits than the lists hold, or no fixed point in 32 rounds.
static int update_settle_pieces(lrb_ctx *c, UpdateRun &u, bool *settled)
{
    const UpdateScalars &hs = *c->h_scalars.as<UpdateScalars>();
    int rc;
    *settled = true;
    if (!u.xl_exact || c->cur->n == 0 || !(hs.xl[XL_OVERFLOW] || hs.xl[XL_CHANGED])) return LRB_OK;
    for (int round = 0; !hs.xl[XL_OVERFLOW] && hs.xl[XL_CHANGED] && round < 32; ++round) {
        launch_xlocus_reset(c->mg.args, c->xl, c->st);
        launch_merge_fold(c->mg.args, c->st);
        launch_xlocus_detect(c->mg.args, c->xl, c->st);
        if ((rc = read_back(c, RB_XL))) return rc;
    }
    if (hs.xl[XL_OVERFLOW] || hs.xl[XL_CHANGED]) { *settled = false; return LRB_OK; }
    c->n_xlocus_pieces = hs.xl[XL_NFORCED];
    launch_xlocus_apply(c->mg.args, c->xl, c->st);
    CK(cudaMemsetAsync(d_totals(c) + T_UPD, 0, 8, c->st));
    launch_merge_finish(c->mg.args, c->st);
    if (u.run_sets) { CK(cudaMemsetAsync(c->y_nelem.p, 0, 16, c->st)); launch_summary_count(u.sa, c->y_nelem.as<unsigned long long>(), c->st); }
    CK(cudaGetLastError());
    if ((rc = read_back(c, RB_SCALARS | RB_NELEM))) return rc;
    c->mg.n_out = (int64_t)hs.t[T_UPD];
    return LRB_OK;
}

// Summary sets (print_trans_summary, update_gtf.c:421-587) and / or the probe for pieces that meet another chromosome, then the second
// round trip.  The class folds are joined in front of it, so they overlap the sets.
static int update_sets(lrb_ctx *c, UpdateRun &u)
{
    const lrb_update_params *up = u.up;
    const int64_t n = c->cur->n, nu = c->mg.n_out;
    const UpdateScalars &hs = *c->h_scalars.as<UpdateScalars>();
    SummaryArgs &sa = u.sa;
    int rc;
    const int64_t n_known_reads = up->want_summary ? (int64_t)hs.counts[12] : 0;
    sa.n_upd = nu; sa.n_upd_dev = nullptr; sa.upd.n = nu;
    // distinct table keys: one per exon element, up to two per gene / site / junction element (the tid-0 phase and the
    // segment phase key them differently), one per known read; the table stays below that bound's next power of two
    // (load <= 0.8 in the worst case, ~0.4 on the bench shape; the slot index is a multiply-high, so no power of two is needed)
    const uint64_t worst = 2 * hs.n_elem - std::min(hs.n_exon_elem, hs.n_elem) + (uint64_t)n_known_reads;
    const uint64_t capn = worst + worst / 4 + 1024;
    NEED(c->h_khi, capn * sizeof(HashSlot));
    CK(cudaMemsetAsync(c->h_khi.p, 0xFF, capn * sizeof(HashSlot), c->st));
    sa.tab.cap = capn; sa.tab.slots = c->h_khi.as<HashSlot>();
    // BED rows are the first occurrences of the exon set: at most one per counted element
    const size_t nb = (size_t)std::max<uint64_t>(hs.n_elem, 1);
    if ((rc = ensure(c, c->bed, Extent{(int64_t)nb}))) return rc;
    sa.bed_tid = c->bed.tid.as<int32_t>(); sa.bed_start = c->bed.start.as<int32_t>(); sa.bed_end = c->bed.end.as<int32_t>(); sa.bed_score = c->bed.score.as<int32_t>();
    sa.bed_type = c->bed.type.as<uint8_t>(); sa.bed_rev = c->bed.is_rev.as<uint8_t>();
    if (c->want_kg_pairs && up->want_summary) { NEED(c->kg_pairs, (size_t)std::max<int64_t>(n_known_reads, 1) * 8); sa.kg_pairs = c->kg_pairs.as<int2>(); }
    CK(cudaMemsetAsync(c->y_counts.p, 0, 32, c->st));
    launch_summary_sets(sa, c->u_cls.as<uint32_t>(), n, c->tile_state.as<uint64_t>(), (uint32_t *)(c->y_nelem.as<uint8_t>() + 16), d_totals(c) + T_BED, c->st,
                        c->st3, c->ev_fork3, c->ev_join3);
    CK(cudaGetLastError());
    if ((rc = join_class_folds(c, up))) return rc;
    return read_back(c, RB_BED | RB_SET_COUNTS);
}

// c->summary from the counters of both round trips (the class sizes are the first one's)
static void update_fill_summary(lrb_ctx *c)
{
    const UpdateScalars &hs = *c->h_scalars.as<UpdateScalars>();
    const uint32_t *cnt = hs.counts; const int64_t nu = c->mg.n_out;
    int32_t *s = c->summary;
    const int cnt_idx[4] = {LRB_S_KNOWN_TRANS, LRB_S_NOVEL_RELIABLE, LRB_S_NOVEL_UNRELIABLE, LRB_S_UNRECOG};
    const int uniq_idx[4] = {LRB_S_UNIQ_KNOWN, LRB_S_UNIQ_RELIABLE, LRB_S_UNIQ_UNRELIABLE, LRB_S_UNIQ_UNRECOG};
    for (int k = 0; k < 4; ++k) s[cnt_idx[k]] = (int32_t)cnt[12 + k];
    s[LRB_S_NOVEL_BAM] = s[LRB_S_NOVEL_RELIABLE] + s[LRB_S_NOVEL_UNRELIABLE];
    for (int k = 0; k < 4; ++k) s[uniq_idx[k]] = (int32_t)cnt[8 + k];
    c->n_bed = nu ? (int64_t)hs.t[T_BED] : 0;
    s[LRB_S_UPD_GENES] = (int32_t)cnt[CNT_G]; s[LRB_S_NOVEL_TRANS] = (int32_t)nu; s[LRB_S_NOVEL_PARTIAL] = (int32_t)cnt[CNT_PARTIAL];
    s[LRB_S_NOVEL_FULL] = (int32_t)nu - (int32_t)cnt[CNT_PARTIAL]; s[LRB_S_NOVEL_EXONS] = (int32_t)cnt[CNT_E]; s[LRB_S_NOVEL_SITES] = (int32_t)(cnt[CNT_D] + cnt[CNT_A]);
    s[LRB_S_NOVEL_JUNC] = (int32_t)cnt[CNT_J]; s[LRB_S_KNOWN_GENES] = (int32_t)cnt[CNT_KG];
    c->n_kg_pairs = (int64_t)cnt[CNT_KG];
}

int lrb_update_run(lrb_ctx *c, const lrb_update_params *up)
{
    if (!c || !up) return LRB_E_ARG;
    if (!c->have_exons) return fail(c, LRB_E_ARG, "lrb_update_run: exon chains missing (run lrb_exon_run / lrb_pipeline_run / lrb_chains_upload)");
    CK(cudaSetDevice(c->device));
    const int64_t l0 = total_launches(), n = c->cur->n;
    int rc;
    memset(c->summary, 0, sizeof c->summary); c->n_bed = 0; c->last_up = *up; c->n_known = c->n_unrecog = 0; c->n_xlocus_pieces = 0;
    ++c->update_gen;
    if ((rc = update_classify(c, up))) return rc;
    // A split piece scans the WHOLE of updated_T in the reference (its tid/start/end are 0, update_gtf.c:148 never stops it), so it
    // can be absorbed by a chain on another chromosome.  The locus-parallel fold cannot see that.  With the default exact matching
    // (-d 0, no -D) that is settled in rounds on the device (xl_* kernels in lrb_update.cu): exact and cheap.  Otherwise the set
    // kernels probe for the necessary condition (a junction of a piece that also exists on another chromosome, CNT_XLOCUS) and the
    // fold is then replayed once more as ONE locus (merge_fold_kernel: the exact back-scan, entry by entry).  With -d > 0 junctions
    // match approximately and the exact-key probe proves nothing: any surviving piece sends the fold to the replay.
    UpdateRun u{};
    u.up = up;
    u.xl_exact = up->split_trans != 0 && up->ss_dis == 0 && up->end_dis == 0x7fffffff && !c->force_single_fold;
    u.detect = up->split_trans != 0 && !u.xl_exact; u.run_sets = up->want_summary || u.detect; u.single = c->force_single_fold;
    u.cap = up->split_trans ? n + n / 8 + 1024 : n;
    u.cap = std::max<int64_t>(u.cap, std::min<int64_t>(c->novel_cap_hint, n + c->ex.n / 2 + 1));
    if (c->test_small_novel_cap) u.cap = std::max<int64_t>(1, n / 4);   // test hook: forces the undersized-list retry
    for (int pass = 0; pass < 2; ++pass) {                              // the second pass is the one-locus replay
        if ((rc = update_lists_and_folds(c, u, pass))) return rc;
        bool settled;
        if ((rc = update_settle_pieces(c, u, &settled))) return rc;
        if (!settled) {                                                 // way 1 into the replay: the xl marks do not settle
            if ((rc = join_class_folds(c, up))) return rc;
            u.single = true; c->n_xlocus_replays++;
            continue;
        }
        c->novel.n = u.n_novel; c->novel.cap = std::max<int64_t>(u.cap, 0);
        if (c->timing && n && pass == 0) { CK(cudaStreamSynchronize(c->st)); cudaEventElapsedTime(&c->ms[LRB_T_K_FOLD], c->ev[EV_FOLD0], c->ev[EV_FOLD1]); }
        if (!u.run_sets || n == 0) break;
        if ((rc = update_sets(c, u))) return rc;
        const uint32_t *cnt = c->h_scalars.as<UpdateScalars>()->counts;
        if (u.detect && !u.single && (cnt[CNT_XLOCUS] != 0 || (up->ss_dis > 0 && cnt[CNT_PARTIAL] != 0))) {
            u.single = true; c->n_xlocus_replays++;                     // way 2 into the replay: the probe
            continue;
        }
        if (up->want_summary) update_fill_summary(c);
        break;
    }
    tick(c, EV_UPDATED);
    c->have_update = true; c->launches_last = total_launches() - l0;
    if (c->timing) {
        CK(cudaStreamSynchronize(c->st));
        cudaEventElapsedTime(&c->ms[LRB_T_CLASSIFY], c->ev[EV_BEGIN], c->ev[EV_CLASSIFIED]);
        float lists = 0; cudaEventElapsedTime(&lists, c->ev[EV_CLASSIFIED], c->ev[EV_LISTED]);
        cudaEventElapsedTime(&c->ms[LRB_T_MERGE], c->ev[EV_LISTED], c->ev[EV_FOLDED]); c->ms[LRB_T_MERGE] += lists;
        cudaEventElapsedTime(&c->ms[LRB_T_SUMMARY], c->ev[EV_FOLDED], c->ev[EV_UPDATED]);
    }
    return LRB_OK;
}

int lrb_unique_run(lrb_ctx *c, const lrb_update_params *up)
{
    if (!c || !up) return LRB_E_ARG;
    if (!c->have_exons) return fail(c, LRB_E_ARG, "lrb_unique_run: exon chains missing");
    CK(cudaSetDevice(c->device));
    int64_t l0 = total_launches();
    DRows &rows = *c->cur; const int64_t n = rows.n;
    int rc;
    CK(cudaMemsetAsync(d_err(c), 0, 4, c->st));
    tick(c, EV_BEGIN);
    if (n) { rows_check_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->st>>>(rows, d_err(c), 1); CK(cudaGetLastError()); }
    uint32_t flags = 0;
    if ((rc = check_err_flags(c, &flags))) return rc;
    if ((rc = setup_list(c, c->tmp_list, c->tmp_cols, n))) return rc;
    launch_rows_as_list(rows, nullptr, n, c->tmp_list, c->st);
    // unique-gtf's input may be a concatenation of sorted samples (Snakefile:189-192).  The locus cuts (App. B.3) are only
    // proven for (tid,start)-sorted streams, so an unsorted list is folded as ONE locus: the back-scan of merge_trans is
    // replayed entry by entry (merge_fold_kernel), early-termination quirks included.
    if ((rc = run_merge(c, c->mg, c->tmp_list, n, *up, (flags & 4u) != 0))) return rc;
    // shared_T = rows the fold absorbed: complement of the alive mask (kept in mg.alive); mg.head is free again
    NEED(c->q_shared, (size_t)std::max<int64_t>(n, 1) * 4);
    c->n_shared = 0;
    if (n) {
        invert_mask_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->st>>>(c->mg.alive.as<uint8_t>(), c->mg.head.as<uint8_t>(), n);
        launch_compact_mask(c->mg.head.as<uint8_t>(), n, c->q_shared.as<uint32_t>(), c->tile_state.as<uint64_t>(), d_ticket(c), d_totals(c), c->st);
        CK(cudaGetLastError());
        uint64_t t; if ((rc = read_totals(c, &t, 1))) return rc;
        c->n_shared = (int64_t)t;
    }
    tick(c, EV_END);
    c->have_unique = true; c->launches_last = total_launches() - l0;
    if (c->timing) { CK(cudaStreamSynchronize(c->st)); cudaEventElapsedTime(&c->ms[LRB_T_MERGE], c->ev[EV_BEGIN], c->ev[EV_END]); }
    return LRB_OK;
}

// Coordinate sort of the current rows on the device: what `samtools sort` does between `lr2rmats filter` and
// `lr2rmats update-gtf` (Snakefile:90), without leaving HBM.  Stable LSD radix sort on tid << 32 | (pos + 1) << 1 | FLAG 0x10.
int lrb_rows_sort(lrb_ctx *c)
{
    if (!c) return LRB_E_ARG;
    if (!c->have_exons) return fail(c, LRB_E_ARG, "lrb_rows_sort: exon chains missing (run lrb_exon_run / lrb_pipeline_run / lrb_chains_upload)");
    CK(cudaSetDevice(c->device));
    int64_t l0 = total_launches();
    if (c->cur == &c->rows3) return LRB_OK;                           // sorted already (every upload / stage run resets cur)
    DRows &rows = *c->cur; const int64_t n = rows.n; int rc;
    if (n == 0) return LRB_OK;
    if (n >= (int64_t)1 << 32) return fail(c, LRB_E_ARG, "lrb_rows_sort: more than 2^32 rows");
    const size_t nn = (size_t)n;
    NEED(c->s_key0, nn * 8); NEED(c->s_key1, nn * 8); NEED(c->s_idx0, nn * 4); NEED(c->s_idx1, nn * 4);
    NEED(c->s_hist, (size_t)256 * (size_t)lrbk::sort_tiles(n) * 4);
    if ((rc = setup_rows(c, c->rows3, c->rows3_cols, n))) return rc;
    unsigned long long *d_max = (unsigned long long *)(d_totals(c) + 3);
    CK(cudaMemsetAsync(d_max, 0, 8, c->st));
    launch_sort_keys(rows, c->have_batch ? c->b.flag : nullptr, c->s_key0.as<uint64_t>(), c->s_idx0.as<uint32_t>(), d_max, c->st);
    CK(cudaGetLastError());
    uint64_t t[4];
    if ((rc = read_totals(c, t, 4))) return rc;
    int bits = 0; for (uint64_t m = t[3]; m; m >>= 1) ++bits;
    uint64_t *k[2] = {c->s_key0.as<uint64_t>(), c->s_key1.as<uint64_t>()}; uint32_t *v[2] = {c->s_idx0.as<uint32_t>(), c->s_idx1.as<uint32_t>()};
    int cur = 0;
    for (int shift = 0; shift < bits; shift += 8) {                  // only the digits the largest key has
        launch_sort_pass(k[cur], v[cur], k[cur ^ 1], v[cur ^ 1], n, shift, c->s_hist.as<uint32_t>(), c->st);
        cur ^= 1;
    }
    c->rows3.n = n;
    launch_rows_permute(rows, c->rows3, v[cur], c->st);
    CK(cudaGetLastError());
    c->cur = &c->rows3; c->rows_compact = false; c->have_update = c->have_unique = false;
    c->launches_last = total_launches() - l0;
    return LRB_OK;
}

int lrb_sync(lrb_ctx *c)
{
    if (!c) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->st));
    return LRB_OK;
}

// ------------------------------------------------------------------------------------------------- fetches
int lrb_filter_fetch(lrb_ctx *c, lrb_filter_result *out)
{
    if (!c || !out) return LRB_E_ARG;
    if (!c->have_filter) return fail(c, LRB_E_ARG, "lrb_filter_fetch: filter stage has not run");
    CK(cudaSetDevice(c->device));
    const size_t n = (size_t)c->b.n; int rc;
    FilterOut &o = c->out_filter;
    if ((rc = d2h(c, o.pass, c->f_pass.as<uint8_t>(), n))) return rc;
    if ((rc = d2h(c, o.score, c->f_score.as<int32_t>(), n))) return rc;
    if ((rc = d2h(c, o.intron, c->f_intron.as<int32_t>(), n))) return rc;
    if ((rc = d2h(c, o.keep_idx, c->f_keep_idx.as<uint32_t>(), (size_t)c->n_keep))) return rc;
    CK(cudaStreamSynchronize(c->st));
    out->n = c->b.n; out->pass = o.pass.as<uint8_t>(); out->score = o.score.as<int32_t>(); out->intron_n = o.intron.as<int32_t>();
    out->n_keep = c->n_keep; out->keep_idx = o.keep_idx.as<uint32_t>();
    return LRB_OK;
}

int lrb_filter_fetch_keep(lrb_ctx *c, int64_t *n_keep, const uint32_t **keep_idx)
{
    if (!c || !n_keep || !keep_idx) return LRB_E_ARG;
    if (!c->have_filter) return fail(c, LRB_E_ARG, "lrb_filter_fetch_keep: filter stage has not run");
    CK(cudaSetDevice(c->device));
    int rc;
    if ((rc = d2h(c, c->out_filter.keep_idx, c->f_keep_idx.as<uint32_t>(), (size_t)c->n_keep))) return rc;
    CK(cudaStreamSynchronize(c->st));
    *n_keep = c->n_keep; *keep_idx = c->out_filter.keep_idx.as<uint32_t>();
    return LRB_OK;
}

// compact copy of the exon data of the current rows (rows may reference a sparse subset of the pool after the fused pass)
__global__ void exon_gather_kernel(DRows rows, DExons ex, const uint32_t *__restrict__ off, int32_t *es, int32_t *ee, uint8_t *fl, int with_flags)
{
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows.n) return;
    uint32_t b = rows.ex_beg[r], n = rows.ex_n[r], o = off[r];
    for (uint32_t j = 0; j < n; ++j) { es[o + j] = ex.es[b + j]; ee[o + j] = ex.ee[b + j]; if (with_flags) fl[o + j] = ex.flag[b + j]; }
}

}  // extern "C" (reopened below)

int lrbk::compact_exons(lrb_ctx *c, bool with_flags, CompactExons *out)
{
    DRows &rows = *c->cur; const int64_t n = rows.n; int rc;
    *out = CompactExons{rows.ex_beg, c->ex.es, c->ex.ee, c->ex.flag, c->ex.n};
    if (c->rows_compact) return LRB_OK;
    // exclusive scan of ex_n -> offsets, then gather into scratch (the summary hash buffers are free at fetch time)
    if ((rc = ensure_tiles(c, n))) return rc;
    NEED(c->u_sub, ((size_t)n + 1) * 4);
    launch_scan_sum_u32(rows.ex_n, c->u_sub.as<uint32_t>(), n, c->tile_state.as<uint64_t>(), d_ticket(c), d_totals(c), c->st);
    uint64_t t; if ((rc = read_totals(c, &t, 1))) return rc;
    const int64_t ne = n ? (int64_t)t : 0;
    const size_t k = (size_t)std::max<int64_t>(ne, 1);
    NEED(c->y_barcnt, k * 4); NEED(c->y_barseg, k * 4); NEED(c->y_bedcnt, k);
    *out = CompactExons{c->u_sub.as<uint32_t>(), c->y_barcnt.as<int32_t>(), c->y_barseg.as<int32_t>(), c->y_bedcnt.as<uint8_t>(), ne};
    if (n) {
        exon_gather_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->st>>>(rows, c->ex, out->off, (int32_t *)out->es, (int32_t *)out->ee,
                                                                              (uint8_t *)out->flag, with_flags ? 1 : 0);
        CK(cudaGetLastError());
    }
    return LRB_OK;
}

extern "C" {

static int fetch_exons(lrb_ctx *c, ExonsOut &o, lrb_exon_result *out, bool with_flags, const uint8_t **flags_out)
{
    DRows &rows = *c->cur; const int64_t n = rows.n; int rc;
    if ((rc = d2h(c, o.read_idx, rows.read_idx, (size_t)n))) return rc;
    if ((rc = d2h(c, o.tid, rows.tid, (size_t)n))) return rc;
    if ((rc = d2h(c, o.is_rev, rows.is_rev, (size_t)n))) return rc;
    NEEDP(o.off, ((size_t)n + 1) * 4);
    CompactExons ce;
    if ((rc = compact_exons(c, with_flags, &ce))) return rc;
    const int64_t ne = ce.n_exon;
    if (n) CK(cudaMemcpyAsync(o.off.p, ce.off, (size_t)n * 4, cudaMemcpyDeviceToHost, c->st));
    if ((rc = d2h(c, o.es, ce.es, (size_t)ne))) return rc;
    if ((rc = d2h(c, o.ee, ce.ee, (size_t)ne))) return rc;
    if (with_flags && (rc = d2h(c, o.flag, ce.flag, (size_t)ne))) return rc;
    CK(cudaStreamSynchronize(c->st));
    o.off.as<uint32_t>()[n] = (uint32_t)ne;
    out->n_reads = n; out->read_idx = c->have_batch ? o.read_idx.as<uint32_t>() : nullptr; out->tid = o.tid.as<int32_t>();
    out->is_rev = o.is_rev.as<uint8_t>(); out->exon_off = o.off.as<uint32_t>();
    out->exon_start = o.es.as<int32_t>(); out->exon_end = o.ee.as<int32_t>();
    if (flags_out) *flags_out = with_flags ? o.flag.as<uint8_t>() : nullptr;
    return LRB_OK;
}

int lrb_exon_fetch(lrb_ctx *c, lrb_exon_result *out)
{
    if (!c || !out) return LRB_E_ARG;
    if (!c->have_exons) return fail(c, LRB_E_ARG, "lrb_exon_fetch: exon stage has not run");
    CK(cudaSetDevice(c->device));
    return fetch_exons(c, c->out_exons, out, false, nullptr);
}

int lrb_update_fetch(lrb_ctx *c, lrb_update_result *out)
{
    if (!c || !out) return LRB_E_ARG;
    if (!c->have_update) return fail(c, LRB_E_ARG, "lrb_update_fetch: update stage has not run");
    CK(cudaSetDevice(c->device));
    memset(out, 0, sizeof *out);
    int rc; const int64_t n = c->cur->n;
    UpdateOut &o = c->out_update;
    if ((rc = fetch_exons(c, o.ex, &out->ex, true, &out->exon_flag))) return rc;
    if ((rc = d2h(c, o.cls, c->u_cls.as<uint32_t>(), (size_t)n))) return rc;
    if ((rc = d2h(c, o.ref, c->u_ref.as<int32_t>(), (size_t)n))) return rc;
    if ((rc = d2h(c, o.known, c->u_known.as<uint32_t>(), (size_t)c->n_known))) return rc;
    if ((rc = d2h(c, o.unrecog, c->u_unrecog.as<uint32_t>(), (size_t)c->n_unrecog))) return rc;
    if ((rc = copy(c, o.novel, c->novel_cols, Extent{c->novel.n}, cudaMemcpyDeviceToHost))) return rc;
    if ((rc = copy(c, o.updated, c->mg.o, Extent{c->mg.n_out}, cudaMemcpyDeviceToHost))) return rc;
    if ((rc = copy(c, o.bed, c->bed, Extent{c->n_bed}, cudaMemcpyDeviceToHost))) return rc;
    CK(cudaStreamSynchronize(c->st));
    out->cls = o.cls.as<uint32_t>(); out->ref_anno = o.ref.as<int32_t>();
    out->n_known = c->n_known; out->known_idx = o.known.as<uint32_t>(); out->n_unrecog = c->n_unrecog; out->unrecog_idx = o.unrecog.as<uint32_t>();
    out->novel.n = c->novel.n; out->novel.read = o.novel.row.as<uint32_t>(); out->novel.exon_lo = o.novel.lo.as<uint32_t>();
    out->novel.exon_n = o.novel.cnt.as<uint32_t>(); out->novel.piece = o.novel.piece.as<int32_t>();
    out->updated = merged_result(o.updated, c->mg.n_out); out->bed = view(o.bed, lrb_bed_list{c->n_bed});
    memcpy(out->summary, c->summary, sizeof c->summary);
    return LRB_OK;
}

// ---- updated_T as a self-contained table (what print_read_trans needs), gathered on the device
struct TabArgs {
    DRows rows; DExons ex; DTransList list; DMerged upd; const int32_t *ref; int rows_have_read_idx;
    uint32_t *name_idx; int32_t *piece, *t_tid, *t_start, *t_end, *e_tid, *cov, *ref_out; uint8_t *t_rev, *e_rev; uint32_t *cnt;
    const uint32_t *off; int32_t *es, *ee; uint8_t *fl;
};
__global__ void tab_rows_kernel(TabArgs a)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.upd.n) return;
    const uint32_t cd = a.upd.cand[i], row = a.list.row[cd];
    const int piece = a.list.piece[cd];
    const uint8_t rev = a.rows.is_rev[row];
    a.name_idx[i] = a.rows_have_read_idx ? a.rows.read_idx[row] : row;
    a.piece[i] = piece; a.t_tid[i] = a.upd.tid[i]; a.t_start[i] = a.upd.start[i]; a.t_end[i] = a.upd.end[i];
    a.t_rev[i] = piece >= 0 ? 0 : rev; a.e_tid[i] = a.rows.tid[row]; a.e_rev[i] = rev; a.cov[i] = a.upd.cov[i]; a.ref_out[i] = a.ref[row];
    a.cnt[i] = a.list.cnt[cd];
}
__global__ void tab_exons_kernel(TabArgs a)
{
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.upd.n) return;
    const uint32_t cd = a.upd.cand[i], row = a.list.row[cd];
    const uint32_t gb = a.rows.ex_beg[row] + a.list.lo[cd], o = a.off[i];
    const int n = (int)a.list.cnt[cd];
    for (int j = 0; j < n; ++j) {
        a.es[o + j] = j == 0 ? a.upd.fs[i] : a.ex.es[gb + j];
        a.ee[o + j] = j == n - 1 ? a.upd.le[i] : a.ex.ee[gb + j];
        if (a.fl) a.fl[o + j] = a.ex.flag[gb + j];
    }
}

}  // extern "C" (reopened below)

// updated_T as a self-contained table in device memory (c->tab): rows + exon offsets + exon pools (+ the exon flag bytes for the
// gather root of a multi-GPU run).  One host round trip (the exon total).
int lrbk::build_update_table(lrb_ctx *c, int64_t *n_exon_out, bool with_flags)
{
    int rc;
    const int64_t nu = c->mg.n_out, k = std::max<int64_t>(nu, 1);
    TableCols<Buf> &tb = c->tab;
    if ((rc = ensure(c, tb, Extent{k, -1}))) return rc;                // the exon columns once their total is known
    NEED(c->tb_cnt, (size_t)k * 4);
    TabArgs a{};
    a.rows = *c->cur; a.ex = c->ex; a.list = c->novel; a.ref = c->u_ref.as<int32_t>(); a.rows_have_read_idx = c->have_batch ? 1 : 0;
    a.upd = view(c->mg.o, DMerged{nu, nu});
    a.name_idx = tb.name_idx.as<uint32_t>(); a.piece = tb.piece.as<int32_t>(); a.t_tid = tb.t_tid.as<int32_t>(); a.t_start = tb.t_start.as<int32_t>();
    a.t_end = tb.t_end.as<int32_t>(); a.e_tid = tb.e_tid.as<int32_t>(); a.cov = tb.cov.as<int32_t>(); a.ref_out = tb.ref_anno.as<int32_t>();
    a.t_rev = tb.t_rev.as<uint8_t>(); a.e_rev = tb.e_rev.as<uint8_t>(); a.cnt = c->tb_cnt.as<uint32_t>(); a.off = tb.exon_off.as<uint32_t>();
    int64_t ne = 0;
    if (nu) {
        if ((rc = ensure_tiles(c, nu))) return rc;
        tab_rows_kernel<<<(unsigned)((nu + 255) / 256), 256, 0, c->st>>>(a);
        launch_scan_sum_u32(a.cnt, tb.exon_off.as<uint32_t>(), nu, c->tile_state.as<uint64_t>(), d_ticket(c), d_totals(c), c->st);
        CK(cudaGetLastError());
        uint64_t t; if ((rc = read_totals(c, &t, 1))) return rc;
        ne = (int64_t)t;
        if ((rc = ensure(c, tb, Extent{k, ne}))) return rc;
        if (with_flags) NEED(c->tb_flag, (size_t)std::max<int64_t>(ne, 1));
        a.es = tb.exon_start.as<int32_t>(); a.ee = tb.exon_end.as<int32_t>(); a.fl = with_flags ? c->tb_flag.as<uint8_t>() : nullptr;
        tab_exons_kernel<<<(unsigned)((nu + 255) / 256), 256, 0, c->st>>>(a);
        CK(cudaGetLastError());
    }
    *n_exon_out = ne;
    return LRB_OK;
}

extern "C" {

int lrb_update_fetch_table(lrb_ctx *c, lrb_trans_table *tab, lrb_bed_list *bed, int32_t *summary)
{
    if (!c) return LRB_E_ARG;
    if (!c->have_update) return fail(c, LRB_E_ARG, "lrb_update_fetch_table: update stage has not run");
    CK(cudaSetDevice(c->device));
    int rc;
    if (summary) memcpy(summary, c->summary, sizeof c->summary);
    UpdateOut &o = c->out_update;
    if (bed) {
        if (!c->last_up.want_summary) return fail(c, LRB_E_ARG, "lrb_update_fetch_table: BED rows need want_summary");
        if ((rc = copy(c, o.bed, c->bed, Extent{c->n_bed}, cudaMemcpyDeviceToHost))) return rc;
        *bed = view(o.bed, lrb_bed_list{c->n_bed});
    }
    if (tab) {
        int64_t ne = 0;
        if ((rc = lrbk::build_update_table(c, &ne, false))) return rc;
        const int64_t nu = c->mg.n_out;
        if ((rc = copy(c, o.tab, c->tab, Extent{nu, ne}, cudaMemcpyDeviceToHost))) return rc;
        CK(cudaStreamSynchronize(c->st));
        o.tab.exon_off.as<uint32_t>()[nu] = (uint32_t)ne;
        *tab = view(o.tab, lrb_trans_table{nu});
    } else CK(cudaStreamSynchronize(c->st));
    return LRB_OK;
}

int lrb_unique_fetch(lrb_ctx *c, lrb_unique_result *out)
{
    if (!c || !out) return LRB_E_ARG;
    if (!c->have_unique) return fail(c, LRB_E_ARG, "lrb_unique_fetch: unique stage has not run");
    CK(cudaSetDevice(c->device));
    memset(out, 0, sizeof *out);
    int rc;
    UniqueOut &o = c->out_unique;
    if ((rc = fetch_exons(c, o.ex, &out->ex, false, nullptr))) return rc;
    if ((rc = copy(c, o.uniq, c->mg.o, Extent{c->mg.n_out}, cudaMemcpyDeviceToHost))) return rc;
    if ((rc = d2h(c, o.shared, c->q_shared.as<uint32_t>(), (size_t)c->n_shared))) return rc;
    CK(cudaStreamSynchronize(c->st));
    out->uniq = merged_result(o.uniq, c->mg.n_out);
    out->n_shared = c->n_shared; out->shared_idx = o.shared.as<uint32_t>();
    return LRB_OK;
}

// -------------------------------------------------------------------------------------------- one-call forms
int lrb_filter(lrb_ctx *c, const lrb_batch *b, const lrb_filter_params *p, lrb_filter_result *out)
{
    int rc;
    if ((rc = lrb_batch_upload(c, b))) return rc;
    if ((rc = lrb_filter_run(c, p))) return rc;
    return lrb_filter_fetch(c, out);
}
int lrb_bam2gtf(lrb_ctx *c, const lrb_batch *b, const lrb_exon_params *p, lrb_exon_result *out)
{
    int rc;
    if ((rc = lrb_batch_upload(c, b))) return rc;
    if ((rc = lrb_exon_run(c, p, 0))) return rc;
    return lrb_exon_fetch(c, out);
}
int lrb_update_gtf(lrb_ctx *c, const lrb_batch *b, const lrb_exon_params *ep, const lrb_update_params *up, lrb_update_result *out)
{
    int rc;
    if (b) { if ((rc = lrb_batch_upload(c, b))) return rc; if ((rc = lrb_exon_run(c, ep, 0))) return rc; }
    if ((rc = lrb_update_run(c, up))) return rc;
    return lrb_update_fetch(c, out);
}
int lrb_unique_gtf(lrb_ctx *c, const lrb_batch *b, const lrb_exon_params *ep, const lrb_update_params *up, lrb_unique_result *out)
{
    int rc;
    if (b) { if ((rc = lrb_batch_upload(c, b))) return rc; if ((rc = lrb_exon_run(c, ep, 0))) return rc; }
    if ((rc = lrb_unique_run(c, up))) return rc;
    return lrb_unique_fetch(c, out);
}

// ------------------------------------------------------------------------------------------------ measurement
int lrb_timing_enable(lrb_ctx *c, int on) { if (!c) return LRB_E_ARG; c->timing = on != 0; return LRB_OK; }
int lrb_timing_get(lrb_ctx *c, float ms[LRB_T_COUNT], int64_t *n_launches)
{
    if (!c) return LRB_E_ARG;
    if (ms) memcpy(ms, c->ms, sizeof c->ms);
    if (n_launches) *n_launches = c->launches_last;
    return LRB_OK;
}
int64_t lrb_launch_count(const lrb_ctx *c) { return c ? total_launches() - c->launches0 : 0; }
int lrb_mark(lrb_ctx *c, int slot)
{
    if (!c || slot < 0 || slot >= 8) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaEventRecord(c->marks[slot], c->st));
    return LRB_OK;
}
int lrb_elapsed_ms(lrb_ctx *c, int a, int b, float *ms)
{
    if (!c || !ms || a < 0 || a >= 8 || b < 0 || b >= 8) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    CK(cudaEventSynchronize(c->marks[b]));
    CK(cudaEventElapsedTime(ms, c->marks[a], c->marks[b]));
    return LRB_OK;
}
int lrb_update_diag(const lrb_ctx *c, int64_t *pieces, int64_t *replays)
{
    if (!c) return LRB_E_ARG;
    if (pieces) *pieces = c->n_xlocus_pieces;
    if (replays) *replays = c->n_xlocus_replays;
    return LRB_OK;
}
int lrb_cigar_stream_diag(const lrb_ctx *c, int64_t *chunks, int64_t *max_staged_ops)
{
    if (!c) return LRB_E_ARG;
    if (chunks) *chunks = c->n_chunks_walked;
    if (max_staged_ops) *max_staged_ops = c->max_staged_ops;
    return LRB_OK;
}
int lrb_fold_census(const lrb_ctx *c, int64_t *out, int n)
{
    if (!c || n < 0 || (n > 0 && !out)) return LRB_E_ARG;
    if (n > 0) memcpy(out, c->census, sizeof(int64_t) * (size_t)std::min(n, 2 * LRB_FC_COUNT));
    return 2 * LRB_FC_COUNT;
}
void *lrb_host_alloc(size_t bytes) { void *p = nullptr; if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; } return p; }
void lrb_host_free(void *p) { if (p) cudaFreeHost(p); }

// ----------------------------------------------------------------------------------------------------- shards
int lrb_shard_cuts_weighted(const int32_t *tid, const int32_t *start, const int32_t *end, const int64_t *weight, int64_t n, int n_shards, int64_t *cuts)
{
    if (n_shards <= 0 || !cuts || n < 0) return LRB_E_ARG;
    // a cut is exact where the read starts beyond every earlier end on its chromosome (SURVEY App. B.3);
    // take the first such position at or after each ideal boundary (k/n_shards of the total weight)
    cuts[0] = 0; cuts[n_shards] = n;
    __int128 total = 0;
    if (weight) for (int64_t i = 0; i < n; ++i) total += weight[i]; else total = n;
    uint64_t run = 0; int k = 1; __int128 acc = 0, want = n_shards > 1 ? total / n_shards : total;
    for (int64_t i = 0; i < n && k < n_shards; ++i) {
        uint64_t ks = ((uint64_t)(uint32_t)(tid[i] + 1) << 32) | (uint32_t)start[i];
        if (acc >= want && i > cuts[k - 1] && ks > run) { cuts[k++] = i; want = total * k / n_shards; }
        uint64_t ke = ((uint64_t)(uint32_t)(tid[i] + 1) << 32) | (uint32_t)end[i];
        if (ke > run) run = ke;
        acc += weight ? weight[i] : 1;
    }
    for (; k < n_shards; ++k) cuts[k] = n;
    return LRB_OK;
}
int lrb_shard_cuts(const int32_t *tid, const int32_t *start, const int32_t *end, int64_t n, int n_shards, int64_t *cuts)
{
    return lrb_shard_cuts_weighted(tid, start, end, nullptr, n, n_shards, cuts);
}

}  // extern "C"
