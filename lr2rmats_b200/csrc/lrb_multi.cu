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
//   lrb_update_gather_reads  the per-read results (bam_T chains, class words, known / unrecog / novel lists, the filter's
//                          records and keep list) of every shard go to rank 0 the same way; they need no merge: each row is
//                          a function of its read and the replicated tables, so the root only concatenates the shards and
//                          shifts their row / exon / record indices to the whole stream (App. B.3).
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
// the per-rank block of lrb_update_gather_reads
enum { R_REC = 0, R_KEEP, R_ROWS, R_EXON, R_KNOWN, R_UNREC, R_NOVEL, R_UPD, R_NAME_BASE, R_FILTER, R_READ_IDX, R_WORDS };
static_assert(R_WORDS <= META_WORDS, "meta block");

struct GatherReads {                                // lrb_update_gather_reads, gathered on the root
    ReadCols<Buf> rd; Buf known, unrecog; ListCols<Buf> novel; MergedCols<Buf> upd; FilterCols<Buf> filt;
    int64_t n_rec = 0, n_keep = 0, n_rows = 0, n_exon = 0, n_known = 0, n_unrecog = 0, n_novel = 0, n_upd = 0;
    int64_t gen = -1;                               // lrb_ctx::update_gen of the run gathered
    bool have = false, with_filter = false, with_read_idx = false;
    // lrb_gather_fetch_reads
    ReadCols<PBuf> o_rd; PBuf o_known, o_unrecog; ListCols<PBuf> o_novel; MergedCols<PBuf> o_upd; BedCols<PBuf> o_bed; FilterCols<PBuf> o_filt;
};

struct MultiState {
    NcclApi *api = nullptr; ncclComm_t comm = nullptr; int rank = 0, n_ranks = 1;
    Buf meta_dev, shard_end_dev, flags_dev; PBuf meta_host;
    // gathered on the root
    TableCols<Buf> g; Buf g_flag; BedCols<Buf> g_bed; Buf g_kg;
    Buf v_ident, v_zeros, v_cnt, v_fs, v_le;          // the gathered table in the shape the set kernels read
    Buf tab, y_barcnt, y_barseg, y_genebar, y_bedcnt, y_bedoff, y_counts, y_nelem, tiles, xs_pl, xs_hx, xs_cnt;
    int64_t n = 0, n_exon = 0, n_bed = 0; int32_t summary[LRB_S_COUNT]; bool have = false, daj_recomputed = false;
    int64_t gen = -1;                               // lrb_ctx::update_gen of the run merged
    TableCols<PBuf> out_tab; BedCols<PBuf> out_bed;  // lrb_gather_fetch
    GatherReads reads;
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

// Indices of shard r count from 0 within the shard (exon offsets, rows, novel entries, records): the root shifts them to the
// shard's place in the gathered whole.  A segmented add over a few uint32 columns in one launch, blockIdx.y = column: element i
// lies in shard k, the first with i < end[k], and gets add[k].  *term = term_val writes an OFFS column's last entry.
static constexpr int REBASE_COLS = 7;
struct RebaseCol { uint32_t *p; int64_t n; uint32_t end[MAX_RANKS], add[MAX_RANKS]; };
struct RebaseArgs { RebaseCol col[REBASE_COLS]; int n_cols, n_shards; uint32_t *term, term_val; };
static_assert(sizeof(RebaseArgs) <= 4096, "kernel parameter space");
__global__ void rebase_kernel(const __grid_constant__ RebaseArgs a)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (a.term && i == 0 && blockIdx.y == 0) *a.term = a.term_val;
    const RebaseCol &c = a.col[blockIdx.y];
    if (i >= c.n) return;
    int k = 0; while (k < a.n_shards - 1 && i >= c.end[k]) ++k;
    c.p[i] += c.add[k];
}

// a column of the gathered shards: shard r holds entries [off[r], off[r + 1]) and gets add[r]
static void rebase_col(RebaseArgs &a, void *p, const std::vector<int64_t> &off, const std::vector<int64_t> &add)
{
    RebaseCol &col = a.col[a.n_cols++];
    col.p = (uint32_t *)p; col.n = off[a.n_shards];
    for (int r = 0; r < a.n_shards; ++r) { col.end[r] = (uint32_t)off[r + 1]; col.add[r] = (uint32_t)add[r]; }
}

static int launch_rebase(lrb_ctx *c, const RebaseArgs &a)
{
    int64_t n = 0;
    for (int j = 0; j < a.n_cols; ++j) n = std::max(n, a.col[j].n);
    rebase_kernel<<<dim3((unsigned)(n / 256 + 1), (unsigned)a.n_cols), 256, 0, c->st>>>(a);
    CK(cudaGetLastError());
    return LRB_OK;
}

// one table's part of a gatherv to the root, as an each_col callback: a rank sends rows [rows[me], rows[me + 1]) and exons
// [exons[me], exons[me + 1]) of each column, the root receives part r at that offset (both inside one ncclGroup); own: the root
// copies its own part instead.  An OFFS column moves n entries: the root rebases them.
static auto gather_parts(lrb_ctx *c, MultiState *m, bool own, const std::vector<int64_t> &rows, const std::vector<int64_t> &exons)
{
    return [c, m, own, &rows, &exons](Per p, size_t esz, auto &src, Buf &dst) {
        const std::vector<int64_t> &off = p == EXON ? exons : rows;
        const int me = m->rank;
        if (own) { if (off[1]) CK(cudaMemcpyAsync(dst.p, addr(src), (size_t)off[1] * esz, cudaMemcpyDeviceToDevice, c->st)); }
        else if (me != 0) { const int64_t cnt = off[me + 1] - off[me]; if (cnt) NK(m->api->Send(addr(src), (size_t)cnt * esz, ncclChar, 0, m->comm, c->st)); }
        else for (int r = 1; r < m->n_ranks; ++r) {
            const int64_t cnt = off[r + 1] - off[r];
            if (cnt) NK(m->api->Recv((char *)dst.p + (size_t)off[r] * esz, (size_t)cnt * esz, ncclChar, r, m->comm, c->st));
        }
        return LRB_OK;
    };
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
    auto parts = [&](bool own, const std::vector<int64_t> &row_off) { return gather_parts(c, m, own, row_off, o_e); };
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
    std::vector<int64_t> names(R);
    for (int r = 0; r < R; ++r) names[r] = mh[(size_t)r * META_WORDS + M_NAME_BASE];
    RebaseArgs ra{}; ra.n_shards = R; ra.term = m->g.exon_off.as<uint32_t>() + N; ra.term_val = (uint32_t)NE;
    rebase_col(ra, m->g.exon_off.p, o_n, o_e); rebase_col(ra, m->g.name_idx.p, o_n, names);
    if ((rc = launch_rebase(c, ra))) return rc;
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
    m->have = true; m->gen = c->update_gen;
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

// ------------------------------------------------------------------------------------------- gather of the per-read results
int lrb_update_gather_reads(lrb_ctx *c, int64_t name_base)
{
    if (!c) return LRB_E_ARG;
    MultiState *m = c->multi;
    if (!m) return fail(c, LRB_E_ARG, "lrb_update_gather_reads: no communicator (lrb_comm_init)");
    if (!c->have_update) return fail(c, LRB_E_ARG, "lrb_update_gather_reads: update stage has not run");
    CK(cudaSetDevice(c->device));
    int rc; const int R = m->n_ranks, me = m->rank; const bool root = me == 0;
    const int64_t l0 = total_launches();
    GatherReads &gr = m->reads;
    gr.have = false;
    // ---- this shard's exon chains in the layout lrb_update_fetch hands out
    CompactExons ce;
    if ((rc = compact_exons(c, true, &ce))) return rc;
    const DRows &rows = *c->cur;
    // ---- counts of every rank
    int64_t *mh = m->meta_host.as<int64_t>(), *mine = mh + (size_t)me * META_WORDS;
    memset(mine, 0, META_WORDS * 8);
    mine[R_REC] = c->have_filter ? c->b.n : 0; mine[R_KEEP] = c->have_filter ? c->n_keep : 0; mine[R_ROWS] = rows.n; mine[R_EXON] = ce.n_exon;
    mine[R_KNOWN] = c->n_known; mine[R_UNREC] = c->n_unrecog; mine[R_NOVEL] = c->novel.n; mine[R_UPD] = c->mg.n_out;
    mine[R_NAME_BASE] = name_base; mine[R_FILTER] = c->have_filter; mine[R_READ_IDX] = c->have_batch;
    int64_t *md = m->meta_dev.as<int64_t>();
    CK(cudaMemcpyAsync(md + (size_t)me * META_WORDS, mine, META_WORDS * 8, cudaMemcpyHostToDevice, c->st));
    NK(m->api->AllGather(md + (size_t)me * META_WORDS, md, META_WORDS, ncclInt64, m->comm, c->st));
    CK(cudaMemcpyAsync(mh, md, (size_t)R * META_WORDS * 8, cudaMemcpyDeviceToHost, c->st));
    CK(cudaStreamSynchronize(c->st));
    // o_x[r]: entries of x in the shards before r
    std::vector<int64_t> o_rec(R + 1, 0), o_keep(R + 1, 0), o_rows(R + 1, 0), o_exon(R + 1, 0), o_known(R + 1, 0), o_unrec(R + 1, 0), o_novel(R + 1, 0),
        o_upd(R + 1, 0), names(R);
    bool with_filter = true, with_read_idx = true;
    for (int r = 0; r < R; ++r) {
        const int64_t *x = mh + (size_t)r * META_WORDS;
        o_rec[r + 1] = o_rec[r] + x[R_REC]; o_keep[r + 1] = o_keep[r] + x[R_KEEP]; o_rows[r + 1] = o_rows[r] + x[R_ROWS];
        o_exon[r + 1] = o_exon[r] + x[R_EXON]; o_known[r + 1] = o_known[r] + x[R_KNOWN]; o_unrec[r + 1] = o_unrec[r] + x[R_UNREC];
        o_novel[r + 1] = o_novel[r] + x[R_NOVEL]; o_upd[r + 1] = o_upd[r] + x[R_UPD]; names[r] = x[R_NAME_BASE];
        with_filter = with_filter && x[R_FILTER] != 0; with_read_idx = with_read_idx && x[R_READ_IDX] != 0;
    }
    const int64_t lim = (int64_t)1 << 32;
    if (o_exon[R] >= lim || o_rows[R] >= lim || o_novel[R] >= lim || (with_filter && o_rec[R] >= lim))
        return fail(c, LRB_E_ARG, "lrb_update_gather_reads: gathered results exceed 2^32 exons / records");
    // ---- gatherv of every column, as in lrb_update_gather
    if (root) {
        if ((rc = ensure(c, gr.rd, Extent{o_rows[R], o_exon[R]})) || (rc = ensure(c, gr.novel, Extent{o_novel[R]})) || (rc = ensure(c, gr.upd, Extent{o_upd[R]})) ||
            (with_filter && (rc = ensure(c, gr.filt, Extent{o_rec[R], o_keep[R]}))))
            return rc;
        NEED(gr.known, (size_t)std::max<int64_t>(o_known[R], 1) * 4); NEED(gr.unrecog, (size_t)std::max<int64_t>(o_unrec[R], 1) * 4);
    }
    ReadCols<const void *> my_rd{rows.read_idx, rows.tid, rows.is_rev, c->u_cls.p, c->u_ref.p, ce.off, ce.es, ce.ee, ce.flag};
    FilterCols<const void *> my_filt{c->f_pass.p, c->f_score.p, c->f_intron.p, c->f_keep_idx.p};
    auto gather = [&](bool own) {
        int rc2;
        if ((rc2 = each_col(gather_parts(c, m, own, o_rows, o_exon), my_rd, gr.rd)) ||
            (rc2 = gather_parts(c, m, own, o_known, o_exon)(ROW, 4, c->u_known, gr.known)) ||
            (rc2 = gather_parts(c, m, own, o_unrec, o_exon)(ROW, 4, c->u_unrecog, gr.unrecog)) ||
            (rc2 = each_col(gather_parts(c, m, own, o_novel, o_exon), c->novel_cols, gr.novel)) ||
            (rc2 = each_col(gather_parts(c, m, own, o_upd, o_exon), c->mg.o, gr.upd)))
            return rc2;
        return with_filter ? each_col(gather_parts(c, m, own, o_rec, o_keep), my_filt, gr.filt) : LRB_OK;
    };
    NK(m->api->GroupStart());
    if ((rc = gather(false))) return rc;
    NK(m->api->GroupEnd());
    if (root) {
        if ((rc = gather(true))) return rc;
        // ---- shard-local indices -> indices of the whole stream (the exon total of ex.exon_off is written by the fetch)
        RebaseArgs ra{}; ra.n_shards = R;
        if (with_read_idx) rebase_col(ra, gr.rd.read_idx.p, o_rows, names);
        rebase_col(ra, gr.rd.exon_off.p, o_rows, o_exon);
        rebase_col(ra, gr.known.p, o_known, o_rows); rebase_col(ra, gr.unrecog.p, o_unrec, o_rows); rebase_col(ra, gr.novel.row.p, o_novel, o_rows);
        rebase_col(ra, gr.upd.cand.p, o_upd, o_novel);
        if (with_filter) rebase_col(ra, gr.filt.keep_idx.p, o_keep, names);
        if ((rc = launch_rebase(c, ra))) return rc;
        gr.n_rec = o_rec[R]; gr.n_keep = o_keep[R]; gr.n_rows = o_rows[R]; gr.n_exon = o_exon[R]; gr.n_known = o_known[R]; gr.n_unrecog = o_unrec[R];
        gr.n_novel = o_novel[R]; gr.n_upd = o_upd[R]; gr.with_filter = with_filter; gr.with_read_idx = with_read_idx;
    }
    CK(cudaStreamSynchronize(c->st));
    gr.have = root; gr.gen = c->update_gen;
    c->launches_last = total_launches() - l0;
    return LRB_OK;
}

int lrb_gather_fetch_reads(lrb_ctx *c, lrb_update_result *update, lrb_filter_result *filter)
{
    if (!c) return LRB_E_ARG;
    MultiState *m = c->multi;
    if (!m) return fail(c, LRB_E_ARG, "lrb_gather_fetch_reads: no communicator (lrb_comm_init)");
    CK(cudaSetDevice(c->device));
    if (update) memset(update, 0, sizeof *update);
    if (filter) memset(filter, 0, sizeof *filter);
    if (m->rank != 0) return LRB_OK;                 // only the root holds the gathered results
    GatherReads &gr = m->reads;
    if (!gr.have) return fail(c, LRB_E_ARG, "lrb_gather_fetch_reads: lrb_update_gather_reads has not run");
    if (update && (!m->have || m->gen != gr.gen))
        return fail(c, LRB_E_ARG, "lrb_gather_fetch_reads: an update result takes its BED rows and counters from lrb_update_gather, which has not "
                                  "succeeded for the lrb_update_run these reads come from");
    if (filter && !gr.with_filter) return fail(c, LRB_E_ARG, "lrb_gather_fetch_reads: the filter stage did not run on every shard");
    int rc;
    if (update) {
        if ((rc = copy(c, gr.o_rd, gr.rd, Extent{gr.n_rows, gr.n_exon}, cudaMemcpyDeviceToHost))) return rc;
        if ((rc = d2h(c, gr.o_known, gr.known.as<uint32_t>(), (size_t)gr.n_known))) return rc;
        if ((rc = d2h(c, gr.o_unrecog, gr.unrecog.as<uint32_t>(), (size_t)gr.n_unrecog))) return rc;
        if ((rc = copy(c, gr.o_novel, gr.novel, Extent{gr.n_novel}, cudaMemcpyDeviceToHost))) return rc;
        if ((rc = copy(c, gr.o_upd, gr.upd, Extent{gr.n_upd}, cudaMemcpyDeviceToHost))) return rc;
        if ((rc = copy(c, gr.o_bed, m->g_bed, Extent{m->n_bed}, cudaMemcpyDeviceToHost))) return rc;
    }
    if (filter && (rc = copy(c, gr.o_filt, gr.filt, Extent{gr.n_rec, gr.n_keep}, cudaMemcpyDeviceToHost))) return rc;
    CK(cudaStreamSynchronize(c->st));
    if (update) {
        const ReadCols<PBuf> &h = gr.o_rd;
        h.exon_off.as<uint32_t>()[gr.n_rows] = (uint32_t)gr.n_exon;
        lrb_exon_result &ex = update->ex;
        ex.n_reads = gr.n_rows; ex.read_idx = gr.with_read_idx ? h.read_idx.as<uint32_t>() : nullptr; ex.tid = h.tid.as<int32_t>();
        ex.is_rev = h.is_rev.as<uint8_t>(); ex.exon_off = h.exon_off.as<uint32_t>(); ex.exon_start = h.exon_start.as<int32_t>(); ex.exon_end = h.exon_end.as<int32_t>();
        update->cls = h.cls.as<uint32_t>(); update->ref_anno = h.ref_anno.as<int32_t>(); update->exon_flag = h.exon_flag.as<uint8_t>();
        update->n_known = gr.n_known; update->known_idx = gr.o_known.as<uint32_t>(); update->n_unrecog = gr.n_unrecog; update->unrecog_idx = gr.o_unrecog.as<uint32_t>();
        update->novel.n = gr.n_novel; update->novel.read = gr.o_novel.row.as<uint32_t>(); update->novel.exon_lo = gr.o_novel.lo.as<uint32_t>();
        update->novel.exon_n = gr.o_novel.cnt.as<uint32_t>(); update->novel.piece = gr.o_novel.piece.as<int32_t>();
        update->updated = merged_result(gr.o_upd, gr.n_upd); update->bed = view(gr.o_bed, lrb_bed_list{m->n_bed});
        memcpy(update->summary, m->summary, sizeof m->summary);
    }
    if (filter) {
        *filter = view(gr.o_filt, lrb_filter_result{});
        filter->n = gr.n_rec; filter->n_keep = gr.n_keep;
    }
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
