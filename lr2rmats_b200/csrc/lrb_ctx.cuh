// lrb_ctx.cuh -- the context behind the C ABI (private to the library): device / pinned buffers, streams, stage state and
// the small helpers every stage uses.  Shared by lrb_capi.cu (single-GPU stages) and lrb_multi.cu (NCCL layer).
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>
#include "lrb_common.cuh"
#include "lrb_kernels.cuh"
#include "lrb_summary.cuh"

namespace lrbk {

extern int64_t g_launches_update, g_launches_summary, g_launches_sort;

// grow-only buffer, contents not preserved on growth: device memory (Buf) or pinned host memory (PBuf), freed with its owner
template <cudaError_t (*Alloc)(void **, size_t), cudaError_t (*Free)(void *)> struct Mem {
    void *p = nullptr; size_t cap = 0;
    Mem() = default;
    Mem(const Mem &) = delete; Mem &operator=(const Mem &) = delete;
    ~Mem() { release(); }
    bool ensure(size_t bytes)
    {
        if (bytes <= cap) return true;
        if (p) Free(p);
        size_t nc = bytes + bytes / 4 + 256;
        if (Alloc(&p, nc) != cudaSuccess) { p = nullptr; cap = 0; cudaGetLastError(); return false; }
        cap = nc; return true;
    }
    void release() { if (p) Free(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};
using Buf = Mem<cudaMalloc, cudaFree>;
using PBuf = Mem<cudaMallocHost, cudaFreeHost>;

// ---- tables: one struct per table states its columns once.  XCols<Buf> holds the table in HBM, XCols<PBuf> its pinned copy,
// XCols<const void *> the host arrays of an upload.  cols(f, g...) calls f(per, element size, the column of each g) per column.
// The columns are named like the pointers of the table's kernel view or result struct, which view() points at them.
enum Per {
    ROW,                                            // one entry per row
    ROW1,                                           // n + 1 entries (offsets given by the host)
    OFFS,                                           // n + 1 exon offsets of which n are built on the device: the one past the end,
                                                    // the exon total, is written by whoever receives the table
    EXON                                            // one entry per exon (per entry of the table's second count)
};
struct Extent {
    int64_t n = 0, ne = 0;                          // rows, exons; ne < 0: exon columns are left alone (not known yet)
    int64_t held(Per p) const { return p == ROW ? n : p == EXON ? ne : n + 1; }
    int64_t moved(Per p) const { return p == ROW1 ? n + 1 : p == EXON ? ne : n; }
};

template <class B> struct BatchCols {               // DBatch; the CIGAR ops are its "exons"
    B tid, pos, l_qseq, nm, flag, xs, qhash, cigar_off, cigar;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.tid...); f(ROW, 4, g.pos...); f(ROW, 4, g.l_qseq...); f(ROW, 4, g.nm...); f(ROW, 2, g.flag...); f(ROW, 1, g.xs...);
        f(ROW, 8, g.qhash...); f(ROW1, 8, g.cigar_off...); f(EXON, 4, g.cigar...);
    }
};
template <class B> struct AnnoCols {                // DAnno
    B tid, start, end, gene, is_rev, exon_off, es, ee, pmax_key, mono;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.tid...); f(ROW, 4, g.start...); f(ROW, 4, g.end...); f(ROW, 4, g.gene...); f(ROW, 1, g.is_rev...); f(ROW1, 4, g.exon_off...);
        f(EXON, 4, g.es...); f(EXON, 4, g.ee...); f(ROW, 8, g.pmax_key...); f(ROW, 1, g.mono...);
    }
};
template <class B> struct SjCols {                  // DSj
    B tid, don, acc, cnt_u, cnt_m, pmax_key, don_key;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.tid...); f(ROW, 4, g.don...); f(ROW, 4, g.acc...); f(ROW, 4, g.cnt_u...); f(ROW, 4, g.cnt_m...); f(ROW, 8, g.pmax_key...); f(ROW, 8, g.don_key...);
    }
};
template <class B> struct RmCols {                  // DRmIndex; rows: the per-tid groups, exons: their entries
    B g_tid, g_off, start, pmax_end;
    template <class F, class... G> static void cols(F &&f, G &...g) { f(ROW, 4, g.g_tid...); f(ROW1, 4, g.g_off...); f(EXON, 4, g.start...); f(EXON, 4, g.pmax_end...); }
};
template <class B> struct RowsCols {                // DRows
    B read_idx, tid, start, end, is_rev, ex_beg, ex_n;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.read_idx...); f(ROW, 4, g.tid...); f(ROW, 4, g.start...); f(ROW, 4, g.end...); f(ROW, 1, g.is_rev...); f(ROW, 4, g.ex_beg...); f(ROW, 4, g.ex_n...);
    }
};
template <class B> struct ListCols {                // DTransList
    B row, lo, cnt, piece;
    template <class F, class... G> static void cols(F &&f, G &...g) { f(ROW, 4, g.row...); f(ROW, 4, g.lo...); f(ROW, 4, g.cnt...); f(ROW, 4, g.piece...); }
};
template <class B> struct MergedCols {              // DMerged
    B cand, cov, tid, start, end, fs, le;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.cand...); f(ROW, 4, g.cov...); f(ROW, 4, g.tid...); f(ROW, 4, g.start...); f(ROW, 4, g.end...); f(ROW, 4, g.fs...); f(ROW, 4, g.le...);
    }
};
template <class B> struct CandCols {                // CandSoA
    B tid, start, end, rev, n, fs, le, gbeg, hash, j0, sig;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.tid...); f(ROW, 4, g.start...); f(ROW, 4, g.end...); f(ROW, 4, g.rev...); f(ROW, 4, g.n...); f(ROW, 4, g.fs...); f(ROW, 4, g.le...);
        f(ROW, 4, g.gbeg...); f(ROW, 8, g.hash...); f(ROW, 8, g.j0...); f(ROW, 8, g.sig...);
    }
};
template <class B> struct TableCols {               // lrb_trans_table: updated_T as a self-contained table
    B name_idx, piece, t_tid, t_start, t_end, t_rev, e_tid, e_rev, cov, ref_anno, exon_off, exon_start, exon_end;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.name_idx...); f(ROW, 4, g.piece...); f(ROW, 4, g.t_tid...); f(ROW, 4, g.t_start...); f(ROW, 4, g.t_end...); f(ROW, 1, g.t_rev...);
        f(ROW, 4, g.e_tid...); f(ROW, 1, g.e_rev...); f(ROW, 4, g.cov...); f(ROW, 4, g.ref_anno...); f(OFFS, 4, g.exon_off...);
        f(EXON, 4, g.exon_start...); f(EXON, 4, g.exon_end...);
    }
};
template <class B> struct BedCols {                 // lrb_bed_list
    B tid, start, end, score, type, is_rev;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.tid...); f(ROW, 4, g.start...); f(ROW, 4, g.end...); f(ROW, 4, g.score...); f(ROW, 1, g.type...); f(ROW, 1, g.is_rev...);
    }
};
template <class B> struct ReadCols {                // lrb_update_result's per-read part: bam_T chains (lrb_exon_result), class words, flags
    B read_idx, tid, is_rev, cls, ref_anno, exon_off, exon_start, exon_end, exon_flag;
    template <class F, class... G> static void cols(F &&f, G &...g)
    {
        f(ROW, 4, g.read_idx...); f(ROW, 4, g.tid...); f(ROW, 1, g.is_rev...); f(ROW, 4, g.cls...); f(ROW, 4, g.ref_anno...); f(OFFS, 4, g.exon_off...);
        f(EXON, 4, g.exon_start...); f(EXON, 4, g.exon_end...); f(EXON, 1, g.exon_flag...);
    }
};
template <class B> struct FilterCols {              // lrb_filter_result; rows: the records, exons: the kept records
    B pass, score, intron_n, keep_idx;
    template <class F, class... G> static void cols(F &&f, G &...g) { f(ROW, 1, g.pass...); f(ROW, 4, g.score...); f(ROW, 4, g.intron_n...); f(EXON, 4, g.keep_idx...); }
};
template <class B> struct JuncCols {                // lrb_sj: the bam2sj output
    B tid, don, acc, uniq_c, multi_c;
    template <class F, class... G> static void cols(F &&f, G &...g) { f(ROW, 4, g.tid...); f(ROW, 4, g.don...); f(ROW, 4, g.acc...); f(ROW, 4, g.uniq_c...); f(ROW, 4, g.multi_c...); }
};

// v (a kernel view or a result struct) with its pointers at the columns of g; its counts are the caller's
template <class G, class V> V view(const G &g, V v)
{
    G::cols([](Per, size_t, auto &ptr, const auto &col) { ptr = (std::remove_reference_t<decltype(ptr)>)col.p; }, v, g);
    return v;
}

inline lrb_merged_list merged_result(const MergedCols<PBuf> &h, int64_t n)
{
    lrb_merged_list o; o.n = n; o.cand = h.cand.as<uint32_t>(); o.cov = h.cov.as<int32_t>(); o.t_tid = h.tid.as<int32_t>(); o.t_start = h.start.as<int32_t>();
    o.t_end = h.end.as<int32_t>(); o.first_start = h.fs.as<int32_t>(); o.last_end = h.le.as<int32_t>();
    return o;
}

// ---- pinned results: one set per result kind, so that a fetch of one kind leaves the results of the others intact
struct ExonsOut { PBuf read_idx, tid, is_rev, off, es, ee, flag; };    // lrb_exon_result (+ the exon flags of an update result)
struct FilterOut { PBuf pass, score, intron, keep_idx; };
struct UpdateOut {                                  // lrb_update_fetch, lrb_update_fetch_table
    ExonsOut ex; PBuf cls, ref, known, unrecog; ListCols<PBuf> novel; MergedCols<PBuf> updated; BedCols<PBuf> bed; TableCols<PBuf> tab;
};
struct UniqueOut { ExonsOut ex; MergedCols<PBuf> uniq; PBuf shared; };

struct MergeBufs {                                  // scratch + output of one merge fold
    Buf tlist, head, locus_start, locus_cnt, alive, rep, lstart, evmask, samemask, hard, desc, relsym, ckey, cmin, cord, clist, crow, fb_list, fb_cnt, fb_state;
    Buf cbase, cperm, ckls;                         // class folds: class order of the rows (launch_class_order)
    MergedCols<Buf> w, o;                           // work list, survivors
    CandCols<Buf> cd;
    int64_t n_out = 0, n_loci = 0;
    MergeArgs args;                                 // of the last fold (refolds of the split-piece rounds reuse them)
};

// timing events (ev[]): the marks of the stage that runs, then the two kernels timed on their own
enum {
    EV_BEGIN = 0, EV_END = 1,                                           // filter, exon, pipeline, unique
    EV_CLASSIFIED = 1, EV_LISTED = 2, EV_FOLDED = 3, EV_UPDATED = 4,    // update
    EV_SCAN0 = 8, EV_SCAN1, EV_FOLD0, EV_FOLD1, EV_COUNT
};

struct MultiState;                                  // lrb_multi.cu

struct OpChunk {                                    // one chunk of an attached CIGAR pool: tiles [tile0, tile1), ops [op_base, op_end)
    int tile0, tile1; uint64_t op_base, op_end;
};

}  // namespace lrbk

struct lrb_ctx {
    using Buf = lrbk::Buf; using PBuf = lrbk::PBuf; using MergeBufs = lrbk::MergeBufs; using DAnno = lrbk::DAnno; using DSj = lrbk::DSj; using DRmIndex = lrbk::DRmIndex;
    using DBatch = lrbk::DBatch; using DRows = lrbk::DRows; using DExons = lrbk::DExons; using DTransList = lrbk::DTransList;
    lrbk::MultiState *multi = nullptr;              // NCCL communicator + gather buffers (lrb_comm_init)

    int device = 0; cudaStream_t st = nullptr; std::string err;
    // side stream: work of a stage that is independent of its main chain (the class folds of the summary) runs here,
    // forked / joined with events, on its own look-back state
    cudaStream_t st2 = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    cudaStream_t st3 = nullptr; cudaEvent_t ev_fork3 = nullptr, ev_join3 = nullptr;       // exon chain of the summary sets
    // tables
    DAnno anno; DSj sj; DRmIndex rm;
    lrbk::AnnoCols<Buf> anno_cols; lrbk::SjCols<Buf> sj_cols; lrbk::RmCols<Buf> rm_cols;
    // batch
    DBatch b; lrbk::BatchCols<Buf> batch_cols;
    bool have_batch = false;
    // an attached batch (lrb_batch_attach): b.cigar is NULL, the walk streams the caller's host pool through two staging buffers,
    // chunk k + 1 copied on st_copy while chunk k is walked on st.  The chunks are whole tiles of the walk, planned at attach.
    const uint32_t *h_cigar = nullptr; bool attached = false;
    std::vector<lrbk::OpChunk> chunks; int64_t stage_ops = 0;       // the plan; the most ops one chunk stages
    Buf stage[2]; cudaStream_t st_copy = nullptr; cudaEvent_t ev_copied[2] = {}, ev_walked[2] = {};
    int64_t n_chunks_walked = 0, max_staged_ops = 0;                // lrb_cigar_stream_diag: of the last walk
    // filter
    Buf f_pass, f_score, f_intron, f_keep_rec_mask, f_keep_idx;
    int64_t n_keep = 0; bool have_filter = false;
    // rows + exons
    DRows rows, rows2, rows3; DRows *cur = nullptr; DExons ex;      // rows3: the coordinate-sorted copy made by lrb_rows_sort
    lrbk::RowsCols<Buf> rows_cols, rows2_cols, rows3_cols; Buf r_nonmono;
    Buf s_key0, s_key1, s_idx0, s_idx1, s_hist;                      // lrb_rows_sort
    Buf e_s, e_e, e_f;
    bool have_exons = false, rows_compact = false;
    // update
    Buf u_cls, u_ref, u_nnovel, u_noff, u_mk, u_ck, u_known, u_unrecog, u_sub;
    DTransList novel; lrbk::ListCols<Buf> novel_cols;
    DTransList tmp_list; lrbk::ListCols<Buf> tmp_cols;
    MergeBufs mg, mg2;
    int64_t n_known = 0, n_unrecog = 0, novel_cap_hint = 0; bool have_update = false, have_unique = false;
    int32_t summary[LRB_S_COUNT];
    bool force_single_fold = false, test_small_novel_cap = false, want_kg_pairs = false; int64_t n_xlocus_replays = 0, n_xlocus_pieces = 0, n_kg_pairs = 0; Buf kg_pairs;
    bool fold_census = false; int64_t census[2][LRB_FC_COUNT] = {};   // test hook LRB_TEST_FOLD_CENSUS: loci per fold path, main / side stream
    bool classify_general = false;                  // test hook LRB_TEST_CLASSIFY_GENERAL: classify_row_kernel is not launched
    Buf xl_key, xl_min, xl_max, xl_cnt, xl_forced; lrbk::XlArgs xl;      // split pieces that meet another chromosome (xl_* kernels)
    // summary
    Buf h_khi, y_barcnt, y_barseg, y_genebar, y_bedcnt, y_bedoff, y_counts, y_nelem;
    lrbk::BedCols<Buf> bed; int64_t n_bed = 0;
    // updated_T as a table (build_update_table); the exon flags only for the gather root, tb_cnt is scratch
    lrbk::TableCols<Buf> tab; Buf tb_flag, tb_cnt;
    // bam2sj
    Buf j_cnt, j_off, j_uq, j_tid, j_don, j_acc, j_u, j_head, j_hpos; lrbk::JuncCols<Buf> junc;
    // unique
    Buf q_shared; int64_t n_shared = 0;
    // look-back state, small device scalars and their pinned mirror
    Buf tile_state, tile_state2, scalars; PBuf h_scalars;
    // pinned results, one set per kind
    lrbk::FilterOut out_filter; lrbk::ExonsOut out_exons; lrbk::UpdateOut out_update; lrbk::UniqueOut out_unique; lrbk::JuncCols<PBuf> out_junc; PBuf out_perm;
    // timing
    bool timing = false; cudaEvent_t ev[lrbk::EV_COUNT]; cudaEvent_t marks[8]; float ms[LRB_T_COUNT]; int64_t launches0 = 0, launches_last = 0;
    lrb_update_params last_up;
    int64_t update_gen = 0;                         // bumped by every lrb_update_run: ties a gathered result to the run it came from
};

namespace lrbk {

int build_update_table(lrb_ctx *c, int64_t *n_exon_out, bool with_flags);      // lrb_capi.cu
// the current rows' exon chains (+ flags) in the layout of lrb_exon_result, in HBM: n offsets from 0 (the exon total is the caller's),
// the chains back to back.  Rows that are not compact are gathered into summary scratch (free once the update stage has run) after
// one host round trip for the exon total.  The pointers stay valid until the next stage run or compaction.
struct CompactExons { const uint32_t *off; const int32_t *es, *ee; const uint8_t *flag; int64_t n_exon; };
int compact_exons(lrb_ctx *c, bool with_flags, CompactExons *out);                // lrb_capi.cu
void multi_release(lrb_ctx *c);                                                   // lrb_multi.cu

inline int64_t total_launches() { return lrbk::count_launches() + lrbk::g_launches_update + lrbk::g_launches_summary + lrbk::g_launches_sort; }

inline int fail(lrb_ctx *c, int code, const std::string &msg) { c->err = msg; return code; }
#define CK(call)                                                                                               \
    do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(c, LRB_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } while (0)
#define NEED(buf, bytes) do { if (!(buf).ensure(bytes)) return fail(c, LRB_E_NOMEM, "device allocation failed: " #buf); } while (0)
#define NEEDP(buf, bytes) do { if (!(buf).ensure(bytes)) return fail(c, LRB_E_NOMEM, "pinned allocation failed: " #buf); } while (0)

// device scalars: [0..31] uint64 totals, then uint32 ticket, err flags.  Slots 0..7 are scratch of the stage that is
// running; the update stage parks its results in fixed slots so that ONE copy brings them all to the host:
enum { T_NOVEL = 8, T_KNOWN = 9, T_UNREC = 10, T_LOCI = 11, T_UPD = 12, T_LOCI2 = 13, T_BED = 16, T_SLOTS = 32 };
inline uint64_t *d_totals(lrb_ctx *c) { return c->scalars.as<uint64_t>(); }
inline uint32_t *d_ticket(lrb_ctx *c) { return (uint32_t *)(c->scalars.as<uint64_t>() + T_SLOTS); }
inline uint32_t *d_err(lrb_ctx *c) { return d_ticket(c) + 1; }
inline uint32_t *d_ticket2(lrb_ctx *c) { return d_ticket(c) + 2; }          // ticket of the side stream

// the update stage's pinned round trip (h_scalars, 512 bytes): the device scalars, then the counters it brings back with them
struct UpdateScalars {
    uint64_t t[T_SLOTS]; uint32_t ticket, err;      // d_totals, d_ticket, d_err
    uint32_t counts[16];                            // y_counts
    uint64_t n_elem, n_exon_elem;                   // y_nelem
    uint32_t xl[XL_NCNT];                           // xl_cnt
};
static_assert(sizeof(UpdateScalars) <= 512, "h_scalars holds 512 bytes");

inline int read_totals(lrb_ctx *c, uint64_t *out, int n)
{
    CK(cudaMemcpyAsync(c->h_scalars.p, d_totals(c), 8 * (size_t)n, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    memcpy(out, c->h_scalars.p, 8 * (size_t)n);
    return LRB_OK;
}

inline int ensure_tiles(lrb_ctx *c, int64_t n_items)
{
    int64_t tiles = n_items / 8 + 1024;             // generous for every tiling used (>= n/256/8, n/reads_per_tile>=8)
    NEED(c->tile_state, (size_t)tiles * 8);
    return LRB_OK;
}

inline void tick(lrb_ctx *c, int k) { if (c->timing) cudaEventRecord(c->ev[k], c->st); }

template <class T> int h2d(lrb_ctx *c, Buf &dst, const T *src, size_t n)
{
    NEED(dst, std::max<size_t>(n, 1) * sizeof(T));
    if (n) CK(cudaMemcpyAsync(dst.p, src, n * sizeof(T), cudaMemcpyHostToDevice, c->st));
    return LRB_OK;
}
template <class T> int d2h(lrb_ctx *c, PBuf &dst, const T *src, size_t n)
{
    NEEDP(dst, std::max<size_t>(n, 1) * sizeof(T));
    if (n) CK(cudaMemcpyAsync(dst.p, src, n * sizeof(T), cudaMemcpyDeviceToHost, c->st));
    return LRB_OK;
}

// f(per, element size, columns...) over the columns of g, gs... until one returns an error
template <class G, class F, class... Gs> int each_col(F &&f, G &g, Gs &...gs)
{
    int rc = LRB_OK;
    G::cols([&](Per p, size_t esz, auto &...col) { if (rc == LRB_OK) rc = f(p, esz, col...); }, g, gs...);
    return rc;
}
// every column of g (device or pinned) sized for e, at least one entry each
template <class G> int ensure(lrb_ctx *c, G &g, Extent e)
{
    return each_col([&](Per p, size_t esz, auto &b) {
        const int64_t k = e.held(p);
        if (k >= 0 && !b.ensure(std::max<int64_t>(k, 1) * esz)) return fail(c, LRB_E_NOMEM, "allocation failed for a table of " + std::to_string(e.n) + " rows");
        return LRB_OK;
    }, g);
}
// the columns of src -> those of dst, sized for e first: host arrays -> HBM (an upload) or HBM -> pinned (a fetch, which leaves
// an OFFS column's last entry to the caller)
inline const void *addr(const void *p) { return p; }
inline const void *addr(const Buf &b) { return b.p; }
template <class D, class S> int copy(lrb_ctx *c, D &dst, S &src, Extent e, cudaMemcpyKind kind)
{
    if (int rc = ensure(c, dst, e)) return rc;
    return each_col([&](Per p, size_t esz, auto &d, const auto &s) {
        if (e.moved(p)) CK(cudaMemcpyAsync(d.p, addr(s), (size_t)e.moved(p) * esz, kind, c->st));
        return LRB_OK;
    }, dst, src);
}

}  // namespace lrbk
