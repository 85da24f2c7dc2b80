// lrb_multi.cu -- the multi-GPU layer of the C ABI (SURVEY.md 8e): one process per GPU, one NCCL communicator per context.
//
//   lrb_tables_broadcast   the annotation / remove / SJ tables go from the root's HBM to every rank's HBM (ncclBroadcast over
//                          NVLink); no rank but the root parses or uploads them
//   lrb_update_gather      after lrb_update_run on every rank (each on its locus-aligned shard of ONE sorted read stream):
//                          counts all-gathered, the per-shard updated_T tables / BED rows / known-gene pairs sent to rank 0
//                          (ncclSend / ncclRecv, a gatherv), and the canonical merge on rank 0:
//                            * tables and BED rows concatenate in shard order (SURVEY App. B.3);
//                            * counters add up, EXCEPT the gene sets -- a gene can span two loci, and gene equality ignores the
//                              chromosome (update_gtf.c:176-179): Updated_Genes is recomputed over the gathered table with the
//                              same barrier-aware kernels as on one GPU, Genes_of_Known... is the union of the shards' pairs;
//                            * the tid-0 site / junction keys of split pieces (SURVEY Q14.4) are probed across shards and the
//                              three sets recomputed over the gathered table when two shards share one;
//                            * a split piece whose junction also exists in ANOTHER shard could have been absorbed there in the
//                              reference (Q14.2): that is reported as LRB_E_XSHARD, the caller reruns unsharded.
//
// NCCL is bound at run time (dlopen of libnccl.so.2): the library loads on a box without NCCL, and inside a process that already
// carries NCCL (torch) it binds to that copy instead of a second one.
#include <dlfcn.h>
#include <nccl.h>
#include <vector>
#include "lrb_ctx.cuh"

namespace lrbk {

struct NcclApi {
    void *h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi *nccl_api(std::string *err)
{
    static NcclApi api; static bool tried = false; static std::string why;
    if (!tried) {
        tried = true;
        const char *names[] = {getenv("LRB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
        for (const char *nm : names) { if (nm && *nm && (api.h = dlopen(nm, RTLD_NOW | RTLD_LOCAL))) break; }
        if (!api.h) why = std::string("libnccl.so.2 not found (") + (dlerror() ? dlerror() : "dlopen failed") + "); set LRB_NCCL_LIB";
        else {
#define LRB_SYM(field, name) do { *(void **)&api.field = dlsym(api.h, name); if (!api.field) why = std::string("NCCL symbol missing: ") + name; } while (0)
            LRB_SYM(GetUniqueId, "ncclGetUniqueId"); LRB_SYM(CommInitRank, "ncclCommInitRank"); LRB_SYM(CommDestroy, "ncclCommDestroy");
            LRB_SYM(Broadcast, "ncclBroadcast"); LRB_SYM(AllGather, "ncclAllGather"); LRB_SYM(Send, "ncclSend"); LRB_SYM(Recv, "ncclRecv");
            LRB_SYM(GroupStart, "ncclGroupStart"); LRB_SYM(GroupEnd, "ncclGroupEnd"); LRB_SYM(GetErrorString, "ncclGetErrorString");
#undef LRB_SYM
        }
    }
    if (!why.empty()) { if (err) *err = why; return nullptr; }
    return &api;
}

static constexpr int META_WORDS = 40, MAX_RANKS = 64;
enum { M_NU = 0, M_NE, M_NBED, M_NKG, M_NAME_BASE, M_PARTIAL, M_WANT_SUMMARY, M_SUMMARY0 /* .. + LRB_S_COUNT */ };

struct MultiState {
    NcclApi *api = nullptr; ncclComm_t comm = nullptr; int rank = 0, n_ranks = 1;
    Buf meta_dev, shard_end_dev, flags_dev; PBuf meta_host;
    // gathered on the root
    TableCols<Buf> g; Buf g_flag; BedCols<Buf> g_bed; Buf g_kg;
    Buf v_ident, v_zeros, v_cnt, v_fs, v_le;          // the gathered table in the shape the set kernels read
    Buf tab, y_barcnt, y_barseg, y_genebar, y_bedcnt, y_bedoff, y_counts, y_nelem, tiles, xs_pl, xs_hx, xs_cnt;
    int64_t n = 0, n_exon = 0, n_bed = 0; int32_t summary[LRB_S_COUNT]; bool have = false, daj_recomputed = false;
    TableCols<PBuf> out_tab; BedCols<PBuf> out_bed;  // lrb_gather_fetch
    float ms_gather = 0, ms_merge = 0; cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
};

void multi_release(lrb_ctx *c)
{
    MultiState *m = c->multi;
    if (!m) return;
    if (m->comm && m->api) m->api->CommDestroy(m->comm);
    for (cudaEvent_t &e : m->ev) if (e) cudaEventDestroy(e);
    delete m; c->multi = nullptr;                   // frees its buffers
}

#define NK(call)                                                                                                           \
    do { ncclResult_t r_ = (call); if (r_ != ncclSuccess) return fail(c, LRB_E_NCCL, std::string(#call) + ": " + m->api->GetErrorString(r_)); } while (0)

// exon offsets of shard r start at 0: shift them to the shard's place in the gathered pools; name_idx becomes an index into
// the whole read stream
struct RebaseArgs { int64_t row_end[MAX_RANKS]; int64_t exon_base[MAX_RANKS]; int64_t name_base[MAX_RANKS]; int n; };
__global__ void rebase_kernel(RebaseArgs a, uint32_t *exon_off, uint32_t *name_idx, int64_t n, int64_t n_exon)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) exon_off[n] = (uint32_t)n_exon;
    if (i >= n) return;
    int k = 0; while (k < a.n - 1 && i >= a.row_end[k]) ++k;
    exon_off[i] += (uint32_t)a.exon_base[k]; name_idx[i] += (uint32_t)a.name_base[k];
}

}  // namespace lrbk

using namespace lrbk;

extern "C" {

int lrb_comm_id(void *id_out)
{
    if (!id_out) return LRB_E_ARG;
    std::string why; NcclApi *api = nccl_api(&why);
    if (!api) return LRB_E_NCCL;
    ncclUniqueId id;
    if (api->GetUniqueId(&id) != ncclSuccess) return LRB_E_NCCL;
    static_assert(sizeof(ncclUniqueId) == LRB_COMM_ID_BYTES, "ncclUniqueId size");
    memcpy(id_out, &id, sizeof id);
    return LRB_OK;
}

int lrb_comm_init(lrb_ctx *c, const void *id_bytes, int rank, int n_ranks)
{
    if (!c || !id_bytes || n_ranks < 1 || n_ranks > MAX_RANKS || rank < 0 || rank >= n_ranks) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    std::string why; NcclApi *api = nccl_api(&why);
    if (!api) return fail(c, LRB_E_NCCL, why);
    multi_release(c);
    MultiState *m = new MultiState(); c->multi = m;
    m->api = api; m->rank = rank; m->n_ranks = n_ranks;
    ncclUniqueId id; memcpy(&id, id_bytes, sizeof id);
    NK(api->CommInitRank(&m->comm, n_ranks, id, rank));
    NEED(m->meta_dev, (size_t)MAX_RANKS * META_WORDS * 8); NEED(m->shard_end_dev, MAX_RANKS * 8); NEED(m->flags_dev, 64);
    NEEDP(m->meta_host, (size_t)MAX_RANKS * META_WORDS * 8);
    for (cudaEvent_t &e : m->ev) CK(cudaEventCreate(&e));
    c->want_kg_pairs = true;
    return LRB_OK;
}

int lrb_comm_destroy(lrb_ctx *c)
{
    if (!c) return LRB_E_ARG;
    cudaSetDevice(c->device); cudaStreamSynchronize(c->st);
    multi_release(c); c->want_kg_pairs = false;
    return LRB_OK;
}

int lrb_comm_rank(const lrb_ctx *c, int *rank, int *n_ranks)
{
    if (!c || !c->multi) return LRB_E_ARG;
    if (rank) *rank = c->multi->rank;
    if (n_ranks) *n_ranks = c->multi->n_ranks;
    return LRB_OK;
}

// ------------------------------------------------------------------------------------------------ tables over NVLink
int lrb_tables_broadcast(lrb_ctx *c, int root, const lrb_anno *anno, const lrb_anno *rm, const lrb_sj *sj)
{
    if (!c) return LRB_E_ARG;
    MultiState *m = c->multi;
    if (!m) return fail(c, LRB_E_ARG, "lrb_tables_broadcast: no communicator (lrb_comm_init)");
    if (root < 0 || root >= m->n_ranks) return LRB_E_ARG;
    CK(cudaSetDevice(c->device));
    int rc;
    const bool is_root = m->rank == root;
    if (is_root) {                                   // the root builds the device tables (prefix-max keys, remove index) once
        if ((rc = lrb_anno_upload(c, anno))) return rc;
        if ((rc = lrb_rm_upload(c, rm))) return rc;
        if ((rc = lrb_sj_upload(c, sj))) return rc;
    }
    int64_t *hd = m->meta_host.as<int64_t>();
    if (is_root) { hd[0] = c->anno.n; hd[1] = c->anno.n_exon; hd[2] = c->sj.n; hd[3] = c->rm.n_groups; hd[4] = c->rm.n; }
    if (is_root) CK(cudaMemcpyAsync(m->meta_dev.p, hd, 5 * 8, cudaMemcpyHostToDevice, c->st));
    NK(m->api->Broadcast(m->meta_dev.p, m->meta_dev.p, 5, ncclInt64, root, m->comm, c->st));
    CK(cudaMemcpyAsync(hd, m->meta_dev.p, 5 * 8, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    const int64_t na = hd[0], nae = hd[1], ns = hd[2], ng = hd[3], nr = hd[4];
    const Extent e_anno{na, nae}, e_sj{ns}, e_rm{ng, nr};
    if (!is_root && ((na && (rc = ensure(c, c->anno_cols, e_anno))) || (ns && (rc = ensure(c, c->sj_cols, e_sj))) || (nr && (rc = ensure(c, c->rm_cols, e_rm)))))
        return rc;
    auto bcast = [&](Extent e) {
        return [&, e](Per p, size_t esz, Buf &b) {
            const size_t bytes = (size_t)e.moved(p) * esz;
            if (bytes) NK(m->api->Broadcast(b.p, b.p, bytes, ncclChar, root, m->comm, c->st));
            return LRB_OK;
        };
    };
    NK(m->api->GroupStart());
    if ((na && (rc = each_col(bcast(e_anno), c->anno_cols))) || (ns && (rc = each_col(bcast(e_sj), c->sj_cols))) || (nr && (rc = each_col(bcast(e_rm), c->rm_cols))))
        return rc;
    NK(m->api->GroupEnd());
    if (!is_root) {
        c->anno = na ? view(c->anno_cols, DAnno{(int32_t)na, nae}) : DAnno{};
        c->sj = ns ? view(c->sj_cols, DSj{ns}) : DSj{};
        c->rm = nr ? view(c->rm_cols, DRmIndex{(int32_t)ng, (int32_t)nr}) : DRmIndex{};
    }
    CK(cudaStreamSynchronize(c->st));
    return LRB_OK;
}

// ------------------------------------------------------------------------------------------- gather + canonical merge
int lrb_update_gather(lrb_ctx *c, int64_t name_base)
{
    if (!c) return LRB_E_ARG;
    MultiState *m = c->multi;
    if (!m) return fail(c, LRB_E_ARG, "lrb_update_gather: no communicator (lrb_comm_init)");
    if (!c->have_update) return fail(c, LRB_E_ARG, "lrb_update_gather: update stage has not run");
    CK(cudaSetDevice(c->device));
    int rc; const int R = m->n_ranks, me = m->rank; const bool root = me == 0;
    const int64_t l0 = total_launches();
    m->have = false;
    CK(cudaEventRecord(m->ev[0], c->st));
    // ---- this shard's updated_T as a self-contained table
    int64_t ne = 0;
    if ((rc = build_update_table(c, &ne, true))) return rc;
    const int64_t nu = c->mg.n_out, nbed = c->last_up.want_summary ? c->n_bed : 0, nkg = c->last_up.want_summary ? c->n_kg_pairs : 0;
    // ---- counts of every rank
    int64_t *mh = m->meta_host.as<int64_t>(), *mine = mh + (size_t)me * META_WORDS;
    memset(mine, 0, META_WORDS * 8);
    mine[M_NU] = nu; mine[M_NE] = ne; mine[M_NBED] = nbed; mine[M_NKG] = nkg; mine[M_NAME_BASE] = name_base;
    mine[M_PARTIAL] = c->summary[LRB_S_NOVEL_PARTIAL]; mine[M_WANT_SUMMARY] = c->last_up.want_summary;
    for (int k = 0; k < LRB_S_COUNT; ++k) mine[M_SUMMARY0 + k] = c->summary[k];
    int64_t *md = m->meta_dev.as<int64_t>();
    CK(cudaMemcpyAsync(md + (size_t)me * META_WORDS, mine, META_WORDS * 8, cudaMemcpyHostToDevice, c->st));
    NK(m->api->AllGather(md + (size_t)me * META_WORDS, md, META_WORDS, ncclInt64, m->comm, c->st));
    CK(cudaMemcpyAsync(mh, md, (size_t)R * META_WORDS * 8, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    std::vector<int64_t> o_n(R + 1, 0), o_e(R + 1, 0), o_b(R + 1, 0), o_k(R + 1, 0);
    bool want_summary = true;
    for (int r = 0; r < R; ++r) {
        const int64_t *x = mh + (size_t)r * META_WORDS;
        o_n[r + 1] = o_n[r] + x[M_NU]; o_e[r + 1] = o_e[r] + x[M_NE]; o_b[r + 1] = o_b[r] + x[M_NBED]; o_k[r + 1] = o_k[r] + x[M_NKG];
        want_summary = want_summary && x[M_WANT_SUMMARY] != 0;
    }
    const int64_t N = o_n[R], NE = o_e[R], NB = o_b[R], NK_ = o_k[R];
    if (NE >= ((int64_t)1 << 32) || N >= ((int64_t)1 << 31)) return fail(c, LRB_E_ARG, "lrb_update_gather: gathered table exceeds 2^32 exons / 2^31 transcripts");
    // ---- gatherv: every rank sends its part of each column, the root receives each part at the shard's offset and then copies its own
    if (root) {
        const int64_t n1 = std::max<int64_t>(N, 1), e1 = std::max<int64_t>(NE, 1);
        if ((rc = ensure(c, m->g, Extent{n1, e1})) || (rc = ensure(c, m->g_bed, Extent{std::max<int64_t>(NB, 1)}))) return rc;
        NEED(m->g_flag, (size_t)e1); NEED(m->g_kg, (size_t)std::max<int64_t>(NK_, 1) * 8);
    }
    auto parts = [&](bool own, const std::vector<int64_t> &row_off) {
        return [&, own, rows = &row_off](Per p, size_t esz, Buf &src, Buf &dst) {
            const std::vector<int64_t> &off = p == EXON ? o_e : *rows;            // an OFFS column moves n entries: the root rebases them
            if (own) { if (off[1]) CK(cudaMemcpyAsync(dst.p, src.p, (size_t)off[1] * esz, cudaMemcpyDeviceToDevice, c->st)); }
            else if (!root) { const int64_t cnt = off[me + 1] - off[me]; if (cnt) NK(m->api->Send(src.p, (size_t)cnt * esz, ncclChar, 0, m->comm, c->st)); }
            else for (int r = 1; r < R; ++r) {
                const int64_t cnt = off[r + 1] - off[r];
                if (cnt) NK(m->api->Recv((char *)dst.p + (size_t)off[r] * esz, (size_t)cnt * esz, ncclChar, r, m->comm, c->st));
            }
            return LRB_OK;
        };
    };
    auto gather = [&](bool own) {
        int rc2;
        if ((rc2 = each_col(parts(own, o_n), c->tab, m->g)) || (rc2 = parts(own, o_n)(EXON, 1, c->tb_flag, m->g_flag)) ||
            (rc2 = each_col(parts(own, o_b), c->bed, m->g_bed)))
            return rc2;
        return parts(own, o_k)(ROW, 8, c->kg_pairs, m->g_kg);
    };
    NK(m->api->GroupStart());
    if ((rc = gather(false))) return rc;
    NK(m->api->GroupEnd());
    if (root && (rc = gather(true))) return rc;
    CK(cudaEventRecord(m->ev[1], c->st));
    if (!root) {
        CK(cudaStreamSynchronize(c->st));
        CK(cudaEventElapsedTime(&m->ms_gather, m->ev[0], m->ev[1])); m->ms_merge = 0;
        c->launches_last = total_launches() - l0;
        return LRB_OK;
    }
    // ---- canonical merge on the root
    RebaseArgs ra{}; ra.n = R;
    for (int r = 0; r < R; ++r) { ra.row_end[r] = o_n[r + 1]; ra.exon_base[r] = o_e[r]; ra.name_base[r] = mh[(size_t)r * META_WORDS + M_NAME_BASE]; }
    rebase_kernel<<<(unsigned)(N / 256 + 1), 256, 0, c->st>>>(ra, m->g.exon_off.as<uint32_t>(), m->g.name_idx.as<uint32_t>(), N, NE);
    CK(cudaGetLastError());
    m->n = N; m->n_exon = NE; m->n_bed = want_summary ? NB : 0; m->daj_recomputed = false;
    memset(m->summary, 0, sizeof m->summary);
    int64_t partial = 0;
    for (int r = 0; r < R; ++r) {
        const int64_t *x = mh + (size_t)r * META_WORDS;
        for (int k = 0; k < LRB_S_COUNT; ++k) m->summary[k] += (int32_t)x[M_SUMMARY0 + k];
        partial += x[M_PARTIAL];
    }
    const bool detect = c->last_up.split_trans != 0;
    if (N > 0 && (want_summary || detect)) {
        const size_t n1 = (size_t)N;
        for (Buf *b : {&m->v_ident, &m->v_zeros, &m->v_cnt, &m->v_fs, &m->v_le}) NEED(*b, n1 * 4);
        NEED(m->y_barcnt, n1 * 16); NEED(m->y_barseg, n1 * 16); NEED(m->y_genebar, n1 * 8); NEED(m->y_bedcnt, n1 * 4); NEED(m->y_bedoff, n1 * 4);
        NEED(m->y_counts, 64); NEED(m->y_nelem, 64); NEED(m->tiles, (size_t)(N / 256 + 1024) * 8 * 6);
        const TableCols<Buf> &g = m->g;
        GatheredTable gt; gt.n = N; gt.n_exon = NE; gt.exon_off = g.exon_off.as<uint32_t>(); gt.es = g.exon_start.as<int32_t>(); gt.ee = g.exon_end.as<int32_t>();
        launch_table_view(gt, m->v_ident.as<uint32_t>(), m->v_zeros.as<uint32_t>(), m->v_cnt.as<uint32_t>(), m->v_fs.as<int32_t>(), m->v_le.as<int32_t>(), c->st);
        std::vector<int64_t> ends(o_n.begin() + 1, o_n.end());
        memcpy(mh + (size_t)MAX_RANKS * META_WORDS - MAX_RANKS, ends.data(), (size_t)R * 8);            // pinned staging behind the metas
        CK(cudaMemcpyAsync(m->shard_end_dev.p, mh + (size_t)MAX_RANKS * META_WORDS - MAX_RANKS, (size_t)R * 8, cudaMemcpyHostToDevice, c->st));
        SummaryArgs sa{};
        sa.rows.n = N; sa.rows.tid = g.e_tid.as<int32_t>(); sa.rows.is_rev = g.e_rev.as<uint8_t>(); sa.rows.ex_beg = g.exon_off.as<uint32_t>(); sa.rows.ex_n = m->v_cnt.as<uint32_t>();
        sa.ex.n = NE; sa.ex.es = g.exon_start.as<int32_t>(); sa.ex.ee = g.exon_end.as<int32_t>(); sa.ex.flag = m->g_flag.as<uint8_t>();
        sa.list.n = N; sa.list.row = m->v_ident.as<uint32_t>(); sa.list.lo = m->v_zeros.as<uint32_t>(); sa.list.cnt = m->v_cnt.as<uint32_t>(); sa.list.piece = g.piece.as<int32_t>();
        sa.upd.n = N; sa.upd.cand = m->v_ident.as<uint32_t>(); sa.upd.cov = g.cov.as<int32_t>(); sa.upd.tid = g.t_tid.as<int32_t>(); sa.upd.start = g.t_start.as<int32_t>();
        sa.upd.end = g.t_end.as<int32_t>(); sa.upd.fs = m->v_fs.as<int32_t>(); sa.upd.le = m->v_le.as<int32_t>();
        sa.ref = g.ref_anno.as<int32_t>(); sa.anno_gene = c->anno.gene; sa.n_upd = N;
        sa.bar_cnt = m->y_barcnt.as<uint32_t>(); sa.bar_seg = m->y_barseg.as<uint32_t>(); sa.gene_bar = m->y_genebar.as<uint64_t>();
        sa.bed_cnt = m->y_bedcnt.as<uint32_t>(); sa.bed_off = m->y_bedoff.as<uint32_t>(); sa.counts = m->y_counts.as<uint32_t>();
        sa.shard_end = m->shard_end_dev.as<int64_t>(); sa.n_shards = R; sa.probe = detect ? 1 : 0;
        if (detect) {
            NEED(m->xs_pl, n1 * 4); NEED(m->xs_hx, n1 * 4); NEED(m->xs_cnt, 64);
            sa.xs_pl = m->xs_pl.as<uint32_t>(); sa.xs_hx = m->xs_hx.as<uint32_t>(); sa.xs_cnt = m->xs_cnt.as<uint32_t>(); sa.xs_cap = (uint32_t)std::min<int64_t>(N, 0x7fffffff);
        }
        // pieces anywhere: their tid-0 site / junction keys may coincide across shards (probe needs those elements in the table)
        const bool pieces = partial > 0 || detect;
        for (int pass = 0; pass < 2; ++pass) {
            // pass 0: gene set (+ the probes); pass 1 (only after a coincidence): gene, site and junction sets over the whole table
            sa.sets = (want_summary ? SUM_G : 0) | (pass == 1 ? SUM_DAJ : 0);
            SummaryArgs cnt_args = sa; cnt_args.sets = sa.sets | ((pieces && want_summary) ? SUM_DAJ : 0);
            CK(cudaMemsetAsync(m->y_nelem.p, 0, 64, c->st)); CK(cudaMemsetAsync(m->y_counts.p, 0, 64, c->st)); CK(cudaMemsetAsync(m->flags_dev.p, 0, 64, c->st));
            if (detect) CK(cudaMemsetAsync(m->xs_cnt.p, 0, 64, c->st));
            launch_summary_count(cnt_args, m->y_nelem.as<unsigned long long>(), c->st);
            CK(cudaMemcpyAsync(mh, m->y_nelem.p, 16, cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
            const uint64_t n_elem = (uint64_t)mh[0];
            const uint64_t worst = 2 * n_elem + (uint64_t)NK_, capn = worst + worst / 4 + 1024;
            NEED(m->tab, capn * sizeof(HashSlot));
            CK(cudaMemsetAsync(m->tab.p, 0xFF, capn * sizeof(HashSlot), c->st));
            sa.tab.cap = capn; sa.tab.slots = m->tab.as<HashSlot>();
            if (pass == 0 && pieces && want_summary) launch_tid0_coincidence(sa, m->flags_dev.as<uint32_t>(), c->st);
            launch_summary_sets(sa, nullptr, 0, m->tiles.as<uint64_t>(), (uint32_t *)(m->y_nelem.as<uint8_t>() + 16), d_totals(c) + T_BED, c->st, c->st, nullptr, nullptr);
            if (want_summary && NK_ > 0) launch_pairs_distinct(sa.tab, m->g_kg.as<int2>(), NK_, m->y_counts.as<uint32_t>() + CNT_KG, c->st);
            CK(cudaGetLastError());
            uint32_t *hp = (uint32_t *)mh;
            CK(cudaMemcpyAsync(hp, m->y_counts.p, 48, cudaMemcpyDeviceToHost, c->st));
            CK(cudaMemcpyAsync(hp + 16, m->flags_dev.p, 4, cudaMemcpyDeviceToHost, c->st));
            CK(cudaStreamSynchronize(c->st));
            if (detect && hp[CNT_XLOCUS])
                return fail(c, LRB_E_XSHARD, "a split piece shares a junction with a transcript of another shard: the reference may merge them across shards "
                                             "(update_gtf.c:148 never stops a piece's back-scan); rerun this input unsharded");
            if (want_summary) {
                m->summary[LRB_S_UPD_GENES] = (int32_t)hp[CNT_G]; m->summary[LRB_S_KNOWN_GENES] = (int32_t)hp[CNT_KG];
                if (pass == 1) { m->summary[LRB_S_NOVEL_SITES] = (int32_t)(hp[CNT_D] + hp[CNT_A]); m->summary[LRB_S_NOVEL_JUNC] = (int32_t)hp[CNT_J]; m->daj_recomputed = true; }
            }
            if (pass == 0 && hp[16] == 0) break;
        }
    }
    CK(cudaEventRecord(m->ev[2], c->st));
    CK(cudaStreamSynchronize(c->st));
    CK(cudaEventElapsedTime(&m->ms_gather, m->ev[0], m->ev[1])); CK(cudaEventElapsedTime(&m->ms_merge, m->ev[1], m->ev[2]));
    m->have = true;
    c->launches_last = total_launches() - l0;
    return LRB_OK;
}

int lrb_gather_fetch(lrb_ctx *c, lrb_trans_table *tab, lrb_bed_list *bed, int32_t *summary)
{
    if (!c) return LRB_E_ARG;
    MultiState *m = c->multi;
    if (!m) return fail(c, LRB_E_ARG, "lrb_gather_fetch: no communicator (lrb_comm_init)");
    CK(cudaSetDevice(c->device));
    if (m->rank != 0) {                              // only the root holds the merged result
        if (tab) memset(tab, 0, sizeof *tab);
        if (bed) memset(bed, 0, sizeof *bed);
        if (summary) memset(summary, 0, sizeof(int32_t) * LRB_S_COUNT);
        return LRB_OK;
    }
    if (!m->have) return fail(c, LRB_E_ARG, "lrb_gather_fetch: lrb_update_gather has not run");
    if (summary) memcpy(summary, m->summary, sizeof m->summary);
    int rc;
    if (tab && (rc = copy(c, m->out_tab, m->g, Extent{m->n, m->n_exon}, cudaMemcpyDeviceToHost))) return rc;
    if (bed && (rc = copy(c, m->out_bed, m->g_bed, Extent{m->n_bed}, cudaMemcpyDeviceToHost))) return rc;
    CK(cudaStreamSynchronize(c->st));
    if (tab) { m->out_tab.exon_off.as<uint32_t>()[m->n] = (uint32_t)m->n_exon; *tab = view(m->out_tab, lrb_trans_table{m->n}); }
    if (bed) *bed = view(m->out_bed, lrb_bed_list{m->n_bed});
    return LRB_OK;
}

int lrb_gather_timing(lrb_ctx *c, float *ms_gather, float *ms_merge)
{
    if (!c || !c->multi) return LRB_E_ARG;
    if (ms_gather) *ms_gather = c->multi->ms_gather;
    if (ms_merge) *ms_merge = c->multi->ms_merge;
    return LRB_OK;
}

}  // extern "C"
