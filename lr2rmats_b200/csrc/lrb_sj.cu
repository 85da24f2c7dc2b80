// lrb_sj.cu -- `lr2rmats bam2sj` on the device (parse_bam.c: bam2sj_core :896-924, gen_sj :402-442, sj_update_group :353-380).
//
// The reference walks every record's CIGAR, emits (tid, don, acc) for each N op of at least `intron_len` bases (don = first, acc =
// last intron base, 1-based) and keeps a sorted array of distinct junctions by linear search + memmove, counting unique- and
// multi-mapped reads (NH:i == 1 or not) per junction.  Here:
//   sj_count_kernel / sj_emit_kernel   thread per record: qualifying N ops counted, offsets by a look-back scan, junctions written
//   radix sort                         stable LSD passes of lrb_sort.cu: by acc, then by tid << 32 | don  (= the array order the
//                                      reference's insertion keeps for a tid-monotone record stream)
//   sj_heads_kernel + compaction       first of every run of equal (tid, don, acc)
//   sj_reduce_kernel                   thread per distinct junction: uniq / multi counts over its run
// Skipped records, as in bam2sj_core: unmapped (:909), and -- since read_type is PAIR_T and no option can change it (:76, :997) --
// everything that is not a proper pair (:914): single-end long reads give the header lines only (SURVEY f-3).
// The strand / motif columns come from the genome FASTA (intr_deri_str :319-337): a per-junction table lookup the host CLI does.
#include "lrb_ctx.cuh"

namespace lrbk {

struct SjArgs {
    DBatch b; const uint8_t *is_uniq; lrb_sj_params p;
    uint32_t *cnt, *off;                            // per record: qualifying N ops, exclusive offsets
    int32_t *j_tid, *j_don, *j_acc; uint8_t *j_uniq; // per emitted junction
    uint32_t *err;
};
LRB_DEVINL bool sj_record_passes(const SjArgs &a, int64_t i) { const uint16_t f = a.b.flag[i]; return !(f & 4u) && (!a.p.pair_only || (f & 2u)); }

__global__ void __launch_bounds__(256) sj_count_kernel(SjArgs a)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.b.n) return;
    uint32_t c = 0;
    if (sj_record_passes(a, i)) {
        for (uint64_t k = a.b.cigar_off[i]; k < a.b.cigar_off[i + 1]; ++k) { const uint32_t w = a.b.cigar[k]; c += (w & 15u) == 3u && (int)(w >> 4) >= a.p.min_intron; }
        // the reference's sorted insert (sj_sch_group :339-351) compares don before it looks at tid: its array stays ordered only for a
        // tid-monotone stream.  Anything else is refused instead of guessed at.
        if (i > 0 && !(a.b.flag[i - 1] & 4u) && a.b.tid[i - 1] > a.b.tid[i]) atomicOr(a.err, 1u);
    }
    a.cnt[i] = c;
}
__global__ void __launch_bounds__(256) sj_emit_kernel(SjArgs a)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.b.n || a.cnt[i] == 0) return;
    uint32_t o = a.off[i];
    int end = a.b.pos[i];                            // gen_sj: end = start - 1 with start = pos + 1
    const uint8_t u = a.is_uniq ? a.is_uniq[i] : 0;
    for (uint64_t k = a.b.cigar_off[i]; k < a.b.cigar_off[i + 1]; ++k) {
        const uint32_t w = a.b.cigar[k], op = w & 15u; const int l = (int)(w >> 4);
        if (op == 3u) {
            if (l >= a.p.min_intron) { a.j_tid[o] = a.b.tid[i]; a.j_don[o] = end + 1; a.j_acc[o] = end + l; a.j_uniq[o] = u; ++o; }
            end += l;
        } else if (op == 0u || op == 7u || op == 8u || op == 2u) end += l;      // M = X D consume the reference (:421-428)
    }
}
__global__ void __launch_bounds__(256) sj_key_kernel(const int32_t *__restrict__ tid, const int32_t *__restrict__ don, const int32_t *__restrict__ acc,
                                                     const uint32_t *__restrict__ perm, uint64_t *keys, uint32_t *idx, int64_t n, int stage)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (stage == 0) { keys[i] = (uint32_t)acc[i]; idx[i] = (uint32_t)i; }
    else { const uint32_t s = perm[i]; keys[i] = ((uint64_t)(uint32_t)tid[s] << 32) | (uint32_t)don[s]; }
}
__global__ void __launch_bounds__(256) sj_heads_kernel(const int32_t *__restrict__ tid, const int32_t *__restrict__ don, const int32_t *__restrict__ acc,
                                                       const uint32_t *__restrict__ perm, uint8_t *head, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool h = i == 0;
    if (!h) { const uint32_t s = perm[i], q = perm[i - 1]; h = tid[s] != tid[q] || don[s] != don[q] || acc[s] != acc[q]; }
    head[i] = h ? 1 : 0;
}
__global__ void __launch_bounds__(256) sj_reduce_kernel(const int32_t *__restrict__ tid, const int32_t *__restrict__ don, const int32_t *__restrict__ acc,
                                                        const uint8_t *__restrict__ uniq, const uint32_t *__restrict__ perm, const uint32_t *__restrict__ head_pos,
                                                        int64_t n_distinct, int64_t n, int32_t *o_tid, int32_t *o_don, int32_t *o_acc, int32_t *o_u, int32_t *o_m)
{
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_distinct) return;
    const int64_t lo = head_pos[k], hi = k + 1 < n_distinct ? head_pos[k + 1] : n;
    int u = 0;
    for (int64_t i = lo; i < hi; ++i) u += uniq[perm[i]];
    const uint32_t s = perm[lo];
    o_tid[k] = tid[s]; o_don[k] = don[s]; o_acc[k] = acc[s]; o_u[k] = u; o_m[k] = (int)(hi - lo) - u;
}

// Stable sort of n records by three keys (k0, k1, k2; most significant first, compared as unsigned): 4 radix passes over k2, then 8 over
// k0 << 32 | k1.  *perm <- the sorted order (in s_idx0 / s_idx1).
static int sort3_device(lrb_ctx *c, const int32_t *k0, const int32_t *k1, const int32_t *k2, int64_t n, const uint32_t **perm)
{
    const size_t m = (size_t)n;
    NEED(c->s_key0, m * 8); NEED(c->s_key1, m * 8); NEED(c->s_idx0, m * 4); NEED(c->s_idx1, m * 4); NEED(c->s_hist, (size_t)256 * (size_t)sort_tiles(n) * 4);
    uint64_t *k[2] = {c->s_key0.as<uint64_t>(), c->s_key1.as<uint64_t>()}; uint32_t *v[2] = {c->s_idx0.as<uint32_t>(), c->s_idx1.as<uint32_t>()};
    const unsigned bl = (unsigned)((n + 255) / 256);
    int cur = 0;
    sj_key_kernel<<<bl, 256, 0, c->st>>>(k0, k1, k2, nullptr, k[0], v[0], n, 0);
    for (int shift = 0; shift < 32; shift += 8) { launch_sort_pass(k[cur], v[cur], k[cur ^ 1], v[cur ^ 1], n, shift, c->s_hist.as<uint32_t>(), c->st); cur ^= 1; }
    sj_key_kernel<<<bl, 256, 0, c->st>>>(k0, k1, k2, v[cur], k[cur], nullptr, n, 1);
    for (int shift = 0; shift < 64; shift += 8) { launch_sort_pass(k[cur], v[cur], k[cur ^ 1], v[cur ^ 1], n, shift, c->s_hist.as<uint32_t>(), c->st); cur ^= 1; }
    *perm = v[cur];
    return LRB_OK;
}

}  // namespace lrbk
using namespace lrbk;

extern "C" int lrb_bam2sj(lrb_ctx *c, const lrb_batch *b, const uint8_t *is_uniq, const lrb_sj_params *p, lrb_sj *out)
{
    if (!c || !p || !out) return LRB_E_ARG;
    int rc;
    if (b && (rc = lrb_batch_upload(c, b))) return rc;
    if (!c->have_batch) return fail(c, LRB_E_ARG, "lrb_bam2sj: no batch uploaded");
    if (c->attached) return fail(c, LRB_E_ARG, "lrb_bam2sj: the batch is attached (its CIGARs are in host memory): pass it to lrb_bam2sj");
    CK(cudaSetDevice(c->device));
    const int64_t l0 = total_launches();
    const int64_t n = c->b.n; const size_t nn = (size_t)std::max<int64_t>(n, 1);
    memset(out, 0, sizeof *out);
    NEED(c->j_cnt, nn * 4); NEED(c->j_off, (nn + 1) * 4); NEED(c->j_uq, nn);
    if ((rc = ensure_tiles(c, n))) return rc;
    if (is_uniq && n) CK(cudaMemcpyAsync(c->j_uq.p, is_uniq, (size_t)n, cudaMemcpyHostToDevice, c->st));
    SjArgs a{}; a.b = c->b; a.is_uniq = is_uniq ? c->j_uq.as<uint8_t>() : nullptr; a.p = *p; a.cnt = c->j_cnt.as<uint32_t>(); a.off = c->j_off.as<uint32_t>(); a.err = d_err(c);
    CK(cudaMemsetAsync(d_err(c), 0, 4, c->st));
    int64_t nj = 0;
    if (n) {
        sj_count_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->st>>>(a);
        launch_scan_sum_u32(a.cnt, a.off, n, c->tile_state.as<uint64_t>(), d_ticket(c), d_totals(c), c->st);
        CK(cudaGetLastError());
        uint64_t t; if ((rc = read_totals(c, &t, 1))) return rc;
        nj = (int64_t)t;
        uint32_t e = 0; CK(cudaMemcpy(&e, d_err(c), 4, cudaMemcpyDeviceToHost));
        if (e & 1u) return fail(c, LRB_E_UNSORTED, "lrb_bam2sj: records are not ordered by reference id (the reference's sorted insert, parse_bam.c:339-351, only keeps its order for such a stream)");
    }
    if (nj >= ((int64_t)1 << 32)) return fail(c, LRB_E_ARG, "lrb_bam2sj: more than 2^32 junction occurrences in one batch");
    int64_t nd = 0;
    if (nj) {
        const size_t m = (size_t)nj;
        NEED(c->j_tid, m * 4); NEED(c->j_don, m * 4); NEED(c->j_acc, m * 4); NEED(c->j_u, m); NEED(c->j_head, m); NEED(c->j_hpos, m * 4);
        if ((rc = ensure_tiles(c, nj))) return rc;
        a.j_tid = c->j_tid.as<int32_t>(); a.j_don = c->j_don.as<int32_t>(); a.j_acc = c->j_acc.as<int32_t>(); a.j_uniq = c->j_u.as<uint8_t>();
        sj_emit_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->st>>>(a);
        const uint32_t *perm;
        if ((rc = sort3_device(c, a.j_tid, a.j_don, a.j_acc, nj, &perm))) return rc;
        sj_heads_kernel<<<(unsigned)((nj + 255) / 256), 256, 0, c->st>>>(a.j_tid, a.j_don, a.j_acc, perm, c->j_head.as<uint8_t>(), nj);
        launch_compact_mask(c->j_head.as<uint8_t>(), nj, c->j_hpos.as<uint32_t>(), c->tile_state.as<uint64_t>(), d_ticket(c), d_totals(c), c->st);
        CK(cudaGetLastError());
        uint64_t t; if ((rc = read_totals(c, &t, 1))) return rc;
        nd = (int64_t)t;
        JuncCols<Buf> &o = c->junc;
        if ((rc = ensure(c, o, Extent{nd}))) return rc;
        sj_reduce_kernel<<<(unsigned)((nd + 255) / 256), 256, 0, c->st>>>(a.j_tid, a.j_don, a.j_acc, a.j_uniq, perm, c->j_hpos.as<uint32_t>(), nd, nj,
                                                                             o.tid.as<int32_t>(), o.don.as<int32_t>(), o.acc.as<int32_t>(), o.uniq_c.as<int32_t>(), o.multi_c.as<int32_t>());
        CK(cudaGetLastError());
        if ((rc = copy(c, c->out_junc, o, Extent{nd}, cudaMemcpyDeviceToHost))) return rc;
        CK(cudaStreamSynchronize(c->st));
    }
    *out = view(c->out_junc, lrb_sj{nd});
    c->launches_last = total_launches() - l0;
    return LRB_OK;
}

// Stable sort of n records by three unsigned keys (most significant first): the `sort -n -k1 -n -k2 -n -k3 -n -k4` of src/sort_gtf.sh:29
// (chromosome rank, transcript start, transcript end; the fourth key, the line number, is the input order a stable sort keeps).
extern "C" int lrb_sort3(lrb_ctx *c, const uint32_t *k0, const uint32_t *k1, const uint32_t *k2, int64_t n, const uint32_t **perm)
{
    if (!c || !perm || n < 0 || (n && (!k0 || !k1 || !k2))) return LRB_E_ARG;
    if (n >= ((int64_t)1 << 32)) return fail(c, LRB_E_ARG, "lrb_sort3: more than 2^32 records");
    CK(cudaSetDevice(c->device));
    const int64_t l0 = total_launches();
    *perm = nullptr;
    if (n == 0) { NEEDP(c->out_perm, 4); *perm = c->out_perm.as<uint32_t>(); return LRB_OK; }
    const size_t m = (size_t)n; int rc;
    // the three key columns ride in the junction buffers (tid = k0, don = k1, acc = k2)
    if ((rc = h2d(c, c->j_tid, (const int32_t *)k0, m)) || (rc = h2d(c, c->j_don, (const int32_t *)k1, m)) || (rc = h2d(c, c->j_acc, (const int32_t *)k2, m))) return rc;
    const uint32_t *sorted;
    if ((rc = sort3_device(c, c->j_tid.as<int32_t>(), c->j_don.as<int32_t>(), c->j_acc.as<int32_t>(), n, &sorted))) return rc;
    CK(cudaGetLastError());
    if ((rc = d2h(c, c->out_perm, sorted, m))) return rc;
    CK(cudaStreamSynchronize(c->st));
    *perm = c->out_perm.as<uint32_t>();
    c->launches_last = total_launches() - l0;
    return LRB_OK;
}
