// lrb_scan.cu -- K1: the fused CIGAR pass (filter statistics + exon chains) and the qname-run selection.
//
// Replaces, for a whole batch at once:
//   gtf_filter()      bam_filter.c:61-86   (coverage / NM identity / remove-GTF overlap, score)
//   remove_overlap()  bam_filter.c:49-59
//   gen_exon()        bam2gtf.c:31-78      (CIGAR walk -> exon chain)
//   the best/second-best qname-run state machine of bam_filter(), bam_filter.c:129-159
//
// Layout: one CTA owns a tile of `reads_per_tile` consecutive records.  Their CIGAR words are one contiguous range of
// the pool, staged into shared memory with coalesced loads and walked from there -- by one thread per read when
// CIGARs are short (Iso-Seq like), or by one warp per read with ballot / shuffle prefix scans when they are long
// (ONT like).  Exons are produced in a second walk over the staged words once the tile's output offset is known from
// a decoupled look-back over (rows, exons), staged in shared memory and written out coalesced: the CIGAR pool is read
// from HBM exactly once and every output array is written exactly once, in read order.
#include "lrb_common.cuh"
#include "lrb_kernels.cuh"

namespace lrbk {

static int64_t g_launches = 0;
int64_t count_launches() { return g_launches; }
#define LRB_COUNT_LAUNCH() (++g_launches)

static constexpr int SCAN_THREADS = 256;

enum { OP_M = 0, OP_I, OP_D, OP_N, OP_S, OP_H, OP_P, OP_EQ, OP_X, OP_B };

LRB_DEVINL bool op_ref(unsigned op) { return (0x18Du >> op) & 1u; }   // M D N = X consume reference (bits 0,2,3,7,8)

// op `off` of the batch, from wherever the launch's ops are (see ScanArgs::ops)
LRB_DEVINL const uint32_t *op_ptr(const ScanArgs &a, uint64_t off) { return a.ops + (off - a.op_base); }

struct WalkStats { int n_exon, intron_n, del_len, ref_len, first_start, last_end; };

// ---- sequential walk (one thread).  EMIT writes exons to es/ee.
template <bool EMIT>
LRB_DEVINL void walk_seq(const uint32_t *c, int n_c, int pos, const lrb_exon_params &ep, int *es, int *ee, WalkStats &w)
{
    int n = 0, start = pos + 1, end = pos, intron = 0, del = 0, first_start = pos + 1;
    for (int i = 0; i < n_c; ++i) {
        uint32_t x = c[i]; int l = (int)(x >> 4); unsigned op = x & 15u;
        bool cut = (op == OP_N && l >= ep.min_intron) || (op == OP_D && l > ep.max_delet);
        if (op == OP_N) ++intron; else if (op == OP_D) del += l;
        if (cut) {
            if (n == 0 || (end - start + 1) >= ep.min_exon) { if (EMIT) { es[n] = start; ee[n] = end; } ++n; }
            start = end + l + 1;
        }
        if (op_ref(op)) end += l;
    }
    if (EMIT) { es[n] = start; ee[n] = end; }
    ++n;
    w.n_exon = n; w.intron_n = intron; w.del_len = del; w.ref_len = end - pos; w.first_start = first_start; w.last_end = end;
}

// ---- sequential walk that also keeps the exons: exon k (all but the last) is parked in the words 2k, 2k+1 of the read's own
// staged CIGAR, which the walk has consumed by then whenever cuts are not adjacent and the CIGAR does not start with one
// (word 2k+1 <= index of the cut that closes exon k).  A CIGAR that breaks this sets *ovf and is walked again later.
LRB_DEVINL void walk_seq_inplace(uint32_t *c, int n_c, int pos, const lrb_exon_params &ep, WalkStats &w, bool *ovf, int *last_start)
{
    int n = 0, start = pos + 1, end = pos, intron = 0, del = 0; bool over = false;
    for (int i = 0; i < n_c; ++i) {
        uint32_t x = c[i]; int l = (int)(x >> 4); unsigned op = x & 15u;
        bool cut = (op == OP_N && l >= ep.min_intron) || (op == OP_D && l > ep.max_delet);
        if (op == OP_N) ++intron; else if (op == OP_D) del += l;
        if (cut) {
            if (n == 0 || (end - start + 1) >= ep.min_exon) {
                if (2 * n + 1 <= i && !over) { c[2 * n] = (uint32_t)start; c[2 * n + 1] = (uint32_t)end; } else over = true;
                ++n;
            }
            start = end + l + 1;
        }
        if (op_ref(op)) end += l;
    }
    ++n;
    *ovf = over; *last_start = start;
    w.n_exon = n; w.intron_n = intron; w.del_len = del; w.ref_len = end - pos; w.first_start = pos + 1; w.last_end = end;
}

// ---- cooperative walk (one warp, lanes over ops, 32 ops per step)
template <bool EMIT>
LRB_DEVINL void walk_warp(const uint32_t *c, int n_c, int pos, const lrb_exon_params &ep, int *es, int *ee, WalkStats &w)
{
    const int lane = lane_id();
    int carry_ref = 0;               // reference bases consumed by earlier steps
    int last_cut_after = pos;        // `end` right after the latest cut op (start of the open exon - 1)
    bool seen_cut = false;
    int n = 0, intron = 0, del = 0;
    for (int base = 0; base < n_c; base += 32) {
        int i = base + lane;
        uint32_t x = i < n_c ? c[i] : 0xFu;                     // op 15: consumes nothing
        int l = (int)(x >> 4); unsigned op = x & 15u;
        int rc = (op <= 8 && op_ref(op)) ? l : 0;
        bool cut = (op == OP_N && l >= ep.min_intron) || (op == OP_D && l > ep.max_delet);
        intron += __popc(__ballot_sync(FULL, op == OP_N));
        int dl = op == OP_D ? l : 0;
        int inc = rc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(FULL, inc, o); int d = __shfl_up_sync(FULL, dl, o); if (lane >= o) { inc += t; dl += d; } }
        del += __shfl_sync(FULL, dl, 31);
        int end_after = pos + carry_ref + inc, end_before = end_after - rc;
        unsigned cutmask = __ballot_sync(FULL, cut);
        unsigned prev = cutmask & ((1u << lane) - 1u);
        int src = prev ? 31 - __clz(prev) : 0;
        int prev_after = __shfl_sync(FULL, end_after, src);
        int start = (prev ? prev_after : last_cut_after) + 1;
        bool first_cut = cut && !seen_cut && prev == 0;
        bool emit = cut && (first_cut || (end_before - start + 1) >= ep.min_exon);
        unsigned emask = __ballot_sync(FULL, emit);
        if (EMIT && emit) { int k = n + __popc(emask & ((1u << lane) - 1u)); es[k] = start; ee[k] = end_before; }
        n += __popc(emask);
        if (cutmask) { last_cut_after = __shfl_sync(FULL, end_after, 31 - __clz(cutmask)); seen_cut = true; }
        carry_ref += __shfl_sync(FULL, inc, 31);
    }
    if (EMIT && lane == 0) { es[n] = last_cut_after + 1; ee[n] = pos + carry_ref; }
    ++n;
    w.n_exon = n; w.intron_n = intron; w.del_len = del; w.ref_len = carry_ref; w.first_start = pos + 1; w.last_end = pos + carry_ref;
}

// remove_overlap() through the per-tid index (see DRmIndex)
LRB_DEVINL bool rm_hit(const DRmIndex &rm, int tid, int pos, int rlen)
{
    if (rm.n_groups == 0) return false;
    int lo = 0, hi = rm.n_groups;
    while (lo < hi) { int m = (lo + hi) >> 1; if (rm.g_tid[m] < tid) lo = m + 1; else hi = m; }
    if (lo >= rm.n_groups || rm.g_tid[lo] != tid) return false;
    int b = rm.g_off[lo], e = rm.g_off[lo + 1], qe = pos + rlen - 1;
    // last entry with start <= qe
    int l2 = b, h2 = e;
    while (l2 < h2) { int m = (l2 + h2) >> 1; if (rm.start[m] <= qe) l2 = m + 1; else h2 = m; }
    if (l2 == b) return false;
    return rm.pmax_end[l2 - 1] >= pos;            // !(pos > end): 0-based pos against 1-based end, as the reference
}

// gtf_filter() predicate after the walk (bam_filter.c:73-84); mixed float/double compares kept as in C
LRB_DEVINL bool filter_pass(const ScanArgs &a, int64_t r, uint32_t c0, uint32_t c1, int n_c, const WalkStats &w, int *score)
{
    if (a.b.flag[r] & 4) return false;
    int l_qseq = a.b.l_qseq[r], qlen = l_qseq;
    if (n_c > 0) {
        unsigned op0 = c0 & 15u, op1 = c1 & 15u;
        if (op0 == OP_S || op0 == OP_H) qlen -= (int)(c0 >> 4);
        if (n_c > 1 && (op1 == OP_S || op1 == OP_H)) qlen -= (int)(c1 >> 4);
    }
    if (__ddiv_rn((double)qlen, (double)l_qseq) < (double)a.fp.cov_rate) return false;
    int sc = qlen - a.b.nm[r] + w.del_len;
    if ((float)sc < __fmul_rn(a.fp.map_qual, (float)qlen)) return false;
    if (rm_hit(a.rm, a.b.tid[r], a.b.pos[r], w.ref_len)) return false;
    *score = sc;
    return true;
}

// Short CIGARs (Iso-Seq like): one thread per read on a staged tile.  Long CIGARs go through cigar_stream_kernel below.
__global__ void __launch_bounds__(SCAN_THREADS) cigar_scan_kernel(ScanArgs a)
{
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t *s_words = smem;                                   // stage_words
    __shared__ uint32_t s_scan[33];
    __shared__ int s_cnt[SCAN_THREADS], s_start[SCAN_THREADS], s_end[SCAN_THREADS];
    __shared__ uint8_t s_mask[SCAN_THREADS];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_excl;

    const int tid = threadIdx.x, R = a.reads_per_tile;
    if (tid == 0) s_tile = a.tile_base + atomicAdd(a.ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile;
    const int64_t r0 = (int64_t)tile * R, r1 = min(a.b.n, r0 + R);
    const int nr = (int)(r1 - r0);
    const uint64_t w_lo = a.b.cigar_off[r0], w_hi = a.b.cigar_off[r1];
    const uint64_t nw = w_hi - w_lo;
    const bool staged = nw <= (uint64_t)a.stage_words;
    const bool do_filter = a.mode != 1, do_exon = a.mode != 0;
    if (staged) {
        // coalesced stage: scalar head up to 16-byte alignment, then 128-bit streaming loads
        const uint32_t *src = op_ptr(a, w_lo);
        uint32_t head = (uint32_t)((4 - (w_lo & 3)) & 3); if (head > nw) head = (uint32_t)nw;
        if ((uint32_t)tid < head) s_words[tid] = ldg_stream_u32(src + tid);
        uint32_t nv = ((uint32_t)nw - head) >> 2;
        const uint4 *v = (const uint4 *)(src + head);
        for (uint32_t i = tid; i < nv; i += SCAN_THREADS) {
            uint4 q = ldg_stream_u4(v + i);
            uint32_t o = head + 4 * i;
            s_words[o] = q.x; s_words[o + 1] = q.y; s_words[o + 2] = q.z; s_words[o + 3] = q.w;
        }
        uint32_t tail = head + 4 * nv;
        if (tail + tid < nw) s_words[tail + tid] = ldg_stream_u32(src + tail + tid);
    }
    s_cnt[tid] = 0; s_mask[tid] = 0;
    __syncthreads();

    // ---- walk 1: statistics, exon count, filter predicate
    auto read_ptr = [&](int64_t r) -> const uint32_t * {
        const uint64_t off = a.b.cigar_off[r];
        return staged ? (s_words + (off - w_lo)) : op_ptr(a, off);
    };
    bool parked = false, park_ovf = false; int park_last_start = 0;      // exons parked in the staged words by walk 1
    if (tid < nr) {
        int64_t r = r0 + tid;
        const uint32_t *c = read_ptr(r); int n_c = (int)(a.b.cigar_off[r + 1] - a.b.cigar_off[r]);
        const uint32_t c0 = n_c > 0 ? c[0] : 0u, c1 = n_c > 0 ? c[n_c - 1] : 0u;
        WalkStats w;
        if (staged && do_exon) { parked = true; walk_seq_inplace(const_cast<uint32_t *>(c), n_c, a.b.pos[r], a.ep, w, &park_ovf, &park_last_start); }
        else walk_seq<false>(c, n_c, a.b.pos[r], a.ep, nullptr, nullptr, w);
        bool mask;
        if (do_filter) {
            int sc = 0; bool p = filter_pass(a, r, c0, c1, n_c, w, &sc);
            a.pass[r] = p ? 1 : 0;
            if (p) { a.score[r] = sc; a.intron_n[r] = w.intron_n; }
            mask = p;
        } else mask = a.sel_mask ? (a.sel_mask[r] != 0) : true;
        const bool unmapped = (a.b.flag[r] & 4) != 0;
        s_mask[tid] = mask ? 1 : 0;
        s_cnt[tid] = (mask && do_exon && !unmapped) ? w.n_exon : 0;
        s_start[tid] = w.first_start; s_end[tid] = w.last_end;
    }
    __syncthreads();

    // ---- tile offsets: block scan of (rows, exons) + look-back across tiles
    uint32_t my_row = s_mask[tid], my_ex = (uint32_t)s_cnt[tid], rows_total, ex_total;
    uint32_t row_excl = block_excl_sum(my_row, s_scan, &rows_total);
    uint32_t ex_excl = block_excl_sum(my_ex, s_scan, &ex_total);
    if (warp_id() == 0) {
        uint64_t e = lookback_exclusive(a.tile_state, tile, pack_pair(rows_total, ex_total), OpAdd());
        if (lane_id() == 0) s_excl = e;
    }
    __syncthreads();
    const uint32_t row_base = pair_hi(s_excl), ex_base = pair_lo(s_excl);
    if (r1 == a.b.n && tid == 0) { a.totals[0] = (uint64_t)row_base + rows_total; a.totals[1] = (uint64_t)ex_base + ex_total; }

    if (!do_exon) return;

    // ---- row records
    if (tid < nr && my_row) {
        int64_t r = r0 + tid; uint32_t row = a.rows_by_record ? (uint32_t)r : row_base + row_excl;
        if ((int64_t)row < a.rows.cap) {
            int8_t xs = a.b.xs[r];
            a.rows.read_idx[row] = (uint32_t)r;
            a.rows.tid[row] = a.b.tid[r];
            a.rows.is_rev[row] = xs == 0 ? ((a.b.flag[r] & 16) != 0) : (xs == '+' ? 0 : 1);    // bam2gtf.c:35-37
            a.rows.start[row] = s_start[tid]; a.rows.end[row] = s_end[tid];
            a.rows.ex_beg[row] = ex_base + ex_excl; a.rows.ex_n[row] = my_ex;
        }
    }
    if (ex_total == 0) return;

    // ---- walk 2: each read's parked exons move straight to the pools (no staging buffer: 6 resident CTAs per SM cover
    // the look-back waits)
    const bool room = (int64_t)ex_base + ex_total <= a.ex.cap;   // host re-runs with a larger pool otherwise
    if (!room) return;
    if (tid < nr && my_ex) {
        int64_t r = r0 + tid;
        const uint32_t *c = read_ptr(r); int n_c = (int)(a.b.cigar_off[r + 1] - a.b.cigar_off[r]);
        int *es = a.ex.es + ex_base + ex_excl, *ee = a.ex.ee + ex_base + ex_excl;
        if (parked && !park_ovf) {                            // move the parked exons; the open one is still in registers
            const int last = (int)my_ex - 1;
            for (int k = 0; k < last; ++k) { es[k] = (int)c[2 * k]; ee[k] = (int)c[2 * k + 1]; }
            es[last] = park_last_start; ee[last] = s_end[tid];
        } else {
            if (parked) c = op_ptr(a, a.b.cigar_off[r]);      // the staged copy is partly overwritten: walk the pool
            WalkStats w; walk_seq<true>(c, n_c, a.b.pos[r], a.ep, es, ee, w);
        }
    }
}

// ------------------------------------------------------------------------------------ long CIGARs: streaming scan
// ONT-like reads carry hundreds of ops, so the pass is a stream over the CIGAR pool with a segmented scan on top.
//
//   * a WARP owns a tile of <= 32 consecutive reads = ONE contiguous range of the pool, and is autonomous: own ticket,
//     own shared-memory ring, own staging slots, no block-wide synchronisation anywhere (a CTA is only a container);
//   * the warp pulls its range through the ring with 1-D TMA bulk copies (cp.async.bulk + mbarrier complete_tx,
//     ST_STAGES rounds in flight: the loads of the next rounds run under the scan of the current one) and consumes it
//     in rounds of 256 ops, 8 consecutive ops per lane (two conflict-free 128-bit shared loads);
//   * what a sequential walk carries from op to op is a flat prefix over the tile, read boundaries ignored: reference
//     bases consumed (32-bit, modular), deletion bases, N ops, cut ops -- two warp scans per round; per-read values are
//     differences of that prefix between the read's last and first op, so the pool is read exactly ONCE;
//   * the flat prefix of the reference bases is written back over the ops in the ring, so the (few) cut ops find the
//     exon end in front of them and the exon start behind them with two shared loads; exon k of a read lands in staging
//     slot (cuts so far in the tile) + (reads so far in the tile), whatever the read boundaries are;
//   * read boundaries are warp-uniform events: lane j keeps the statistics of read j of the tile in registers and
//     finishes it (filter predicate, short internal exons dropped as bam2gtf.c:45 does, row, exons to the pools).
// Output placement: the fused pipeline writes rows at their record index, so a tile only needs room for its exons -- one
// atomicAdd; the other modes keep the pools in read order with the (rows, exons) look-back, one word per warp tile.
// A tile whose exons overflow the staging slots is redone by walk_warp (two walks per read).
static constexpr int ST_THREADS = 128, ST_WARPS = ST_THREADS / 32;
static constexpr int ST_R = 32;                     // reads per warp tile: one lane per read
static constexpr int ST_ROUND = 256;                // ops per warp round = 8 per lane = one ring stage
static constexpr int ST_STAGES = 3;
static constexpr int ST_EXW = 512;                  // exon staging slots per warp tile

LRB_DEVINL uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
LRB_DEVINL void mbar_init(uint64_t *bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory"); }
LRB_DEVINL void mbar_expect_tx(uint64_t *bar, uint32_t bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory"); }
LRB_DEVINL void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
LRB_DEVINL bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}

// one step of an inclusive warp scan: shfl.up hands back "source lane in range" as a predicate, the add rides on it
LRB_DEVINL void scan_up_add(uint32_t &v, int o)
{
    asm volatile("{\n.reg .u32 t;\n.reg .pred p;\nshfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff;\n@p add.u32 %0, %0, t;\n}" : "+r"(v) : "r"(o));
}

struct StreamWarp {
    alignas(128) uint32_t ring[ST_STAGES][ST_ROUND];
    alignas(16) uint32_t dpre[ST_ROUND];            // flat prefix of the deletion bases behind every op of the round
    int es[ST_EXW], ee[ST_EXW];
    alignas(8) uint64_t bar[ST_STAGES];
    uint2 dslot[ST_R];                              // x: pos - (flat reference prefix at the read's first op), y: reads with ops before it in the tile
    int off[ST_R + 1];
};

__global__ void __launch_bounds__(ST_THREADS) cigar_stream_kernel(ScanArgs a, int n_tiles)
{
    __shared__ StreamWarp s_warp[ST_WARPS];
    StreamWarp &S = s_warp[warp_id()];
    const int lane = lane_id();
    const bool do_filter = a.mode != 1, do_exon = a.mode != 0;
    int tile = 0;
    if (lane == 0) { tile = (int)atomicAdd(a.ticket, 1u); for (int s = 0; s < ST_STAGES; ++s) mbar_init(&S.bar[s], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    tile = __shfl_sync(FULL, tile, 0);
    if (tile >= n_tiles) return;                     // (the grid is rounded up to whole CTAs)
    tile += a.tile_base;
    const int64_t r0 = (int64_t)tile * ST_R, r1 = min(a.b.n, r0 + ST_R);
    const int nr = (int)(r1 - r0);
    const uint64_t w_lo = a.b.cigar_off[r0], w_hi = a.b.cigar_off[r1];
    const bool huge = w_hi - w_lo >= (1ull << 30);   // cannot happen with 16-bit n_cigar (32 x 65535 ops); guard anyway
    const int nw = huge ? 0 : (int)(w_hi - w_lo);
    const int64_t rr = r0 + lane;                    // this lane's read
    const bool mine = lane < nr;
    const int my_beg = mine ? (int)(min(a.b.cigar_off[rr], w_hi) - w_lo) : nw, my_end = mine ? (int)(min(a.b.cigar_off[rr + 1], w_hi) - w_lo) : nw;
    const int my_pos = mine ? a.b.pos[rr] : 0;
    // the record fields the filter predicate needs and the read's first / last op: loaded now, used after the stream
    const uint32_t my_flag = mine ? a.b.flag[rr] : 4u;
    const uint32_t c0 = (mine && my_end > my_beg) ? *op_ptr(a, w_lo + (uint64_t)my_beg) : 0u, c1 = (mine && my_end > my_beg) ? *op_ptr(a, w_lo + (uint64_t)my_end - 1) : 0u;
    S.off[lane] = my_beg; if (lane == 31) S.off[32] = my_end;
    int my_ref = 0, my_del = 0, my_int = 0; uint32_t my_ncut = 0, my_sbeg = 0;
    bool ovf = huge;
    __syncwarp();

    // ---- phase A: stream the tile's ops
    if (nw > 0) {
        uint32_t *ring = &S.ring[0][0];
        const uint64_t g_abs = w_lo & ~3ull;                         // 16-byte aligned start of the stream
        const int lead = (int)(w_lo - g_abs);                        // pad words in front of the tile (0..3)
        const int n_words = lead + nw;
        const int n_chunks = (n_words + ST_ROUND - 1) / ST_ROUND;
        const uint32_t *src = op_ptr(a, g_abs);                      // op_base is a multiple of 4: still 16-byte aligned
        auto issue = [&](int c) {
            const int s = c % ST_STAGES;
            int words = n_words - c * ST_ROUND; words = words > ST_ROUND ? ST_ROUND : ((words + 3) & ~3);
            mbar_expect_tx(&S.bar[s], (uint32_t)words * 4u);
            bulk_g2s(ring + s * ST_ROUND, src + (size_t)c * ST_ROUND, (uint32_t)words * 4u, &S.bar[s]);
        };
        if (lane == 0) for (int c = 0; c < ST_STAGES && c < n_chunks; ++c) issue(c);
        const uint32_t nonempty = __ballot_sync(FULL, my_end > my_beg);
        // warp-uniform state of the read being walked
        int r = __ffs(nonempty) - 1;                                 // first read with ops (nw > 0: it exists)
        int nb = __shfl_sync(FULL, my_end, r);                       // its end
        uint32_t baseS = 0, baseD = 0, baseN = 0, baseC = 0;         // flat prefixes at its first op
        uint32_t ridx = 0;                                           // reads with ops started before it
        uint32_t carryS = 0, carryD = 0, carryN = 0, carryC = 0;     // flat prefixes at the start of the round
        if (lane == r) { S.dslot[r] = make_uint2((uint32_t)my_pos, 0u); my_sbeg = 0; }
        bool done = false;
        for (int c = 0; c < n_chunks && !done; ++c) {
            const int s = c % ST_STAGES;
            while (!mbar_try_wait(&S.bar[s], (uint32_t)(c / ST_STAGES) & 1u)) { }
            uint32_t *rw = ring + s * ST_ROUND;
            const int g = c * ST_ROUND - lead;                       // tile op index of the round's first word
            const int i0 = g + 8 * lane;
            // (lanes 4..7 of every quarter warp fetch their two quads in swapped order: the eight 16-byte accesses of a
            // shared-memory phase then fall into eight different bank groups)
            const int hsw = (lane >> 2) & 1;
            const uint4 qa = *reinterpret_cast<const uint4 *>(rw + 8 * lane + 4 * hsw), qb = *reinterpret_cast<const uint4 *>(rw + 8 * lane + 4 - 4 * hsw);
            const uint4 q0 = hsw ? qb : qa, q1 = hsw ? qa : qb;
            uint32_t x[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
            if (g < 0 || g + ST_ROUND > nw) {                        // first / last round: words outside the tile consume nothing (op 15)
#pragma unroll
                for (int k = 0; k < 8; ++k) if (i0 + k < 0 || i0 + k >= nw) x[k] = 0xFu;
            }
            // lane-local prefixes BEHIND every op go to shared memory at once (the reference bases over the ops themselves);
            // the lane's own offsets exS / exD are added by whoever reads them
            uint32_t sp[8], dp[8], cm = 0, nm = 0, sacc = 0, dacc = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t l = x[k] >> 4, op = x[k] & 15u;
                if ((0x18Du >> op) & 1u) sacc += l;
                const bool isd = op == OP_D, isn = op == OP_N;
                if (isd) dacc += l;
                const bool cut = (isn && (int)l >= a.ep.min_intron) || (isd && (int)l > a.ep.max_delet);
                nm |= (isn ? 1u : 0u) << k; cm |= (cut ? 1u : 0u) << k;
                sp[k] = sacc; dp[k] = dacc;
            }
            *reinterpret_cast<uint4 *>(rw + 8 * lane) = make_uint4(sp[0], sp[1], sp[2], sp[3]);
            *reinterpret_cast<uint4 *>(rw + 8 * lane + 4) = make_uint4(sp[4], sp[5], sp[6], sp[7]);
            *reinterpret_cast<uint4 *>(S.dpre + 8 * lane) = make_uint4(dp[0], dp[1], dp[2], dp[3]);
            *reinterpret_cast<uint4 *>(S.dpre + 8 * lane + 4) = make_uint4(dp[4], dp[5], dp[6], dp[7]);
            // three warp scans: reference bases, deletion bases, (N ops : cut ops) packed (<= 256 each per round)
            uint32_t incS = sacc, incD = dacc;
            const uint32_t ncp = ((uint32_t)__popc(nm) << 16) | (uint32_t)__popc(cm);
            uint32_t incP = ncp;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { scan_up_add(incS, o); scan_up_add(incD, o); scan_up_add(incP, o); }
            const uint32_t exS = carryS + incS - sacc, exD = carryD + incD - dacc;
            const uint32_t exP = incP - ncp, exN = carryN + (exP >> 16), exC = carryC + (exP & 0xffffu);
            __syncwarp();
            int rL = r, nbL = nb;                                    // read of the round's first op: where the cut ops start looking for theirs
            // ---- read boundaries of this round, warp-uniform: position nb lies behind op nb - 1
            const int gend = g + ST_ROUND;
            while (nb <= gend) {
                const int p = nb - 1 - g;                            // word of the read's last op
                const uint32_t low = (2u << (p & 7)) - 1u;
                const uint32_t Sb = rw[p] + __shfl_sync(FULL, exS, p >> 3), Db = S.dpre[p] + __shfl_sync(FULL, exD, p >> 3);
                const uint32_t Nb = __shfl_sync(FULL, exN + __popc(nm & low), p >> 3), Cb = __shfl_sync(FULL, exC + __popc(cm & low), p >> 3);
                if (lane == r) { my_ref = (int)(Sb - baseS); my_del = (int)(Db - baseD); my_int = (int)(Nb - baseN); my_ncut = Cb - baseC; }
                const uint32_t rest = r >= 31 ? 0u : (nonempty & ~((2u << r) - 1u));
                if (!rest) { done = true; break; }
                r = __ffs(rest) - 1; nb = __shfl_sync(FULL, my_end, r);
                baseS = Sb; baseD = Db; baseN = Nb; baseC = Cb; ++ridx;
                if (lane == r) { S.dslot[r] = make_uint2((uint32_t)my_pos - Sb, ridx); my_sbeg = Cb + ridx; }
            }
            __syncwarp();
            // ---- cut ops: exon end in front of the cut, exon start behind it
            if (do_exon) {
                uint32_t m = cm;
                while (m) {
                    const int k = __ffs(m) - 1; m &= m - 1;
                    const int i = i0 + k, wi = 8 * lane + k;
                    while (i >= nbL) { ++rL; nbL = S.off[rL + 1]; }
                    const uint2 ds = S.dslot[rL];
                    const uint32_t s_after = exS + rw[wi], s_before = k ? exS + rw[wi - 1] : exS;
                    const uint32_t sl = exC + __popc(cm & ((1u << k) - 1u)) + ds.y;
                    if (sl + 1 < (uint32_t)ST_EXW) { S.ee[sl] = (int)(ds.x + s_before); S.es[sl + 1] = (int)(ds.x + s_after) + 1; }
                    else ovf = true;
                }
            }
            // ---- carries into the next round
            const uint32_t totP = __shfl_sync(FULL, incP, 31);
            carryS += __shfl_sync(FULL, incS, 31); carryD += __shfl_sync(FULL, incD, 31); carryN += totP >> 16; carryC += totP & 0xffffu;
            __syncwarp();
            if (lane == 0 && c + ST_STAGES < n_chunks) { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); issue(c + ST_STAGES); }
        }
    }
    ovf = __any_sync(FULL, ovf || (mine && my_end > my_beg && my_sbeg + my_ncut >= (uint32_t)ST_EXW));

    // ---- phase B: lane j finishes read j of the tile
    WalkStats ws; ws.n_exon = 0; ws.intron_n = 0; ws.del_len = 0; ws.ref_len = 0; ws.first_start = my_pos + 1; ws.last_end = my_pos;
    uint32_t f0 = c0, f1 = c1; const int n_c = my_end - my_beg;
    if (!ovf) {
        if (mine) {
            if (n_c > 0) {
                ws.ref_len = my_ref; ws.del_len = my_del; ws.intron_n = my_int;
                int n = (int)my_ncut + 1;
                if (do_exon) {
                    int *xs = S.es + my_sbeg, *xe = S.ee + my_sbeg;
                    xs[0] = my_pos + 1; xe[n - 1] = my_pos + my_ref;
                    if (n > 2) {                                 // short internal exons vanish (bam2gtf.c:45), the first and the last stay
                        int o = 1;
                        for (int k = 1; k < n - 1; ++k) if (xe[k] - xs[k] + 1 >= a.ep.min_exon) { xs[o] = xs[k]; xe[o] = xe[k]; ++o; }
                        xs[o] = xs[n - 1]; xe[o] = xe[n - 1]; n = o + 1;
                    }
                }
                ws.n_exon = n;
            } else ws.n_exon = 1;
            ws.last_end = my_pos + ws.ref_len;
        }
    } else {
        for (int li = 0; li < nr; ++li) {                        // staging overflow: one warp walk per read
            const int64_t q = r0 + li;
            const uint32_t *cg = op_ptr(a, a.b.cigar_off[q]); const int nc = (int)(a.b.cigar_off[q + 1] - a.b.cigar_off[q]);
            WalkStats t; walk_warp<false>(cg, nc, a.b.pos[q], a.ep, nullptr, nullptr, t);
            if (lane == li) ws = t;
        }
    }
    bool mask = false;
    if (mine) {
        if (do_filter) {
            int sc = 0; const bool p = filter_pass(a, rr, f0, f1, n_c, ws, &sc);
            a.pass[rr] = p ? 1 : 0;
            if (p) { a.score[rr] = sc; a.intron_n[rr] = ws.intron_n; }
            mask = p;
        } else mask = a.sel_mask ? (a.sel_mask[rr] != 0) : true;
    }
    const uint32_t my_row = mask ? 1u : 0u;
    const uint32_t my_ex = (mask && do_exon && !(my_flag & 4u)) ? (uint32_t)ws.n_exon : 0u;
    // ---- placement: warp scan of (rows, exons), then one atomicAdd (rows by record) or the look-back across warp tiles
    uint32_t row_inc = my_row, ex_inc = my_ex;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(FULL, row_inc, o), u = __shfl_up_sync(FULL, ex_inc, o); if (lane >= o) { row_inc += t; ex_inc += u; } }
    const uint32_t rows_total = __shfl_sync(FULL, row_inc, 31), ex_total = __shfl_sync(FULL, ex_inc, 31);
    const uint32_t row_excl = row_inc - my_row, ex_excl = ex_inc - my_ex;
    uint32_t row_base = 0, ex_base = 0;
    if (a.rows_by_record) {
        unsigned long long eb = 0;
        if (lane == 0) {
            if (rows_total) atomicAdd((unsigned long long *)&a.totals[0], (unsigned long long)rows_total);
            if (ex_total) eb = atomicAdd((unsigned long long *)&a.totals[1], (unsigned long long)ex_total);
        }
        ex_base = (uint32_t)__shfl_sync(FULL, eb, 0);
    } else {
        const uint64_t e = __shfl_sync(FULL, lookback_exclusive(a.tile_state, tile, pack_pair(rows_total, ex_total), OpAdd()), 0);
        row_base = pair_hi(e); ex_base = pair_lo(e);
        if (r1 == a.b.n && lane == 0) { a.totals[0] = (uint64_t)row_base + rows_total; a.totals[1] = (uint64_t)ex_base + ex_total; }
    }
    if (!do_exon) return;
    if (my_row) {
        const uint32_t row = a.rows_by_record ? (uint32_t)rr : row_base + row_excl;
        if ((int64_t)row < a.rows.cap) {
            const int8_t xs = a.b.xs[rr];
            a.rows.read_idx[row] = (uint32_t)rr;
            a.rows.tid[row] = a.b.tid[rr];
            a.rows.is_rev[row] = xs == 0 ? ((a.b.flag[rr] & 16) != 0) : (xs == '+' ? 0 : 1);    // bam2gtf.c:35-37
            a.rows.start[row] = ws.first_start; a.rows.end[row] = ws.last_end;
            a.rows.ex_beg[row] = ex_base + ex_excl; a.rows.ex_n[row] = my_ex;
        }
    }
    if (ex_total == 0) return;
    if ((int64_t)ex_base + ex_total > a.ex.cap) return;          // host re-runs with a larger pool
    if (!ovf) {
        if (my_ex) {
            int *es = a.ex.es + ex_base + ex_excl, *ee = a.ex.ee + ex_base + ex_excl;
            if (n_c == 0) { es[0] = my_pos + 1; ee[0] = my_pos; }    // no ops at all: the open exon (bam2gtf.c:74-76)
            else {
                const int *xs = S.es + my_sbeg, *xe = S.ee + my_sbeg;
                for (uint32_t k = 0; k < my_ex; ++k) { es[k] = xs[k]; ee[k] = xe[k]; }
            }
        }
    } else {
        for (int li = 0; li < nr; ++li) {
            const uint32_t cnt = __shfl_sync(FULL, my_ex, li), lo = __shfl_sync(FULL, ex_excl, li);
            if (!cnt) continue;
            const int64_t q = r0 + li;
            const uint32_t *cg = op_ptr(a, a.b.cigar_off[q]); const int nc = (int)(a.b.cigar_off[q + 1] - a.b.cigar_off[q]);
            WalkStats t; walk_warp<true>(cg, nc, a.b.pos[q], a.ep, a.ex.es + ex_base + lo, a.ex.ee + ex_base + lo, t);
        }
    }
}

int stream_reads_per_tile() { return ST_R; }
int scan_reads_per_tile() { return SCAN_THREADS; }

void launch_cigar_scan(const ScanArgs &a, int n_tiles, bool stream_mode, size_t smem_bytes, cudaStream_t st)
{
    if (n_tiles <= 0) return;
    if (stream_mode) cigar_stream_kernel<<<(n_tiles + ST_WARPS - 1) / ST_WARPS, ST_THREADS, 0, st>>>(a, n_tiles);
    else {
        cudaFuncSetAttribute(cigar_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
        cigar_scan_kernel<<<n_tiles, SCAN_THREADS, smem_bytes, st>>>(a);
    }
    LRB_COUNT_LAUNCH();
}

// ---------------------------------------------------------------------------------------- qname-run selection
// The reference's state machine (bam_filter.c:133-153; SURVEY Q3) sees the passing records in input order, so a run is a stretch
// of equal qname hashes over the passing subsequence, walked here through the pass mask: no compacted row list -- and no host
// round trip for its size -- is needed in front of the selection.  The head record of each run replays the machine.
__global__ void select_records_kernel(const uint64_t *__restrict__ qhash, const uint8_t *__restrict__ pass, int64_t n,
                                      const int32_t *__restrict__ score, const int32_t *__restrict__ intron_n, lrb_filter_params fp, uint8_t *keep_rec_mask)
{
    int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n || !pass[r]) return;
    const uint64_t h = qhash[r];
    int64_t p = r - 1;
    while (p >= 0 && !pass[p]) --p;
    if (p >= 0 && qhash[p] == h) return;                        // not a run head
    int b_score = score[r], s_score = 0, b_intron = intron_n[r]; int64_t best = r;
    for (int64_t j = r + 1; j < n; ++j) {
        if (!pass[j]) continue;
        if (qhash[j] != h) break;
        int sc = score[j];
        if (sc > b_score) { best = j; s_score = b_score; b_score = sc; b_intron = intron_n[j]; }
        else if (sc > s_score) s_score = sc;
    }
    if ((float)s_score < __fmul_rn(fp.sec_rat, (float)b_score) && b_intron >= fp.min_intron_n) keep_rec_mask[best] = 1;
}
void launch_select_records(const DBatch &b, const uint8_t *pass, const int32_t *score, const int32_t *intron_n, lrb_filter_params fp,
                           uint8_t *keep_rec_mask, cudaStream_t st)
{
    if (b.n <= 0) return;
    select_records_kernel<<<(unsigned)((b.n + 255) / 256), 256, 0, st>>>(b.qhash, pass, b.n, score, intron_n, fp, keep_rec_mask);
    LRB_COUNT_LAUNCH();
}

// ordered compaction of the kept records + gather of their (record-indexed) rows into the compact row table
__global__ void __launch_bounds__(256) compact_gather_kernel(const uint8_t *__restrict__ mask, int64_t n, DRows src, DRows dst, uint32_t *keep_idx,
                                                             uint64_t *tile_state, uint32_t *ticket, uint64_t *total)
{
    constexpr int ITEMS = 8;
    __shared__ uint32_t s_scan[33];
    __shared__ uint32_t s_tile; __shared__ uint64_t s_excl;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile;
    const int64_t base = ((int64_t)tile * 256 + threadIdx.x) * ITEMS;
    uint32_t cnt = 0, m = 0;
    if (base + ITEMS <= n) {                                     // 8 mask bytes in one load (base is a multiple of 8)
        const uint2 q = *(const uint2 *)(mask + base);
#pragma unroll
        for (int i = 0; i < 4; ++i) { if ((q.x >> (8 * i)) & 0xffu) m |= 1u << i; if ((q.y >> (8 * i)) & 0xffu) m |= 1u << (4 + i); }
    } else {
        for (int i = 0; i < ITEMS; ++i) if (base + i < n && mask[base + i]) m |= 1u << i;
    }
    cnt = __popc(m);
    uint32_t tot, excl = block_excl_sum(cnt, s_scan, &tot);
    if (warp_id() == 0) { uint64_t e = lookback_exclusive(tile_state, tile, tot, OpAdd()); if (lane_id() == 0) s_excl = e; }
    __syncthreads();
    uint32_t o = (uint32_t)s_excl + excl;
    while (m) {
        const int i = __ffs(m) - 1; m &= m - 1;
        const uint32_t s = (uint32_t)(base + i);
        keep_idx[o] = s;
        dst.read_idx[o] = s; dst.tid[o] = src.tid[s]; dst.start[o] = src.start[s]; dst.end[o] = src.end[s];
        dst.is_rev[o] = src.is_rev[s]; dst.ex_beg[o] = src.ex_beg[s]; dst.ex_n[o] = src.ex_n[s];
        ++o;
    }
    if ((int64_t)(tile + 1) * 256 * ITEMS >= n && threadIdx.x == 0) *total = s_excl + tot;
}
void launch_compact_gather(const uint8_t *mask, int64_t n, const DRows &src, DRows &dst, uint32_t *keep_idx,
                           uint64_t *tile_state, uint32_t *ticket, uint64_t *total, cudaStream_t st)
{
    if (n <= 0) { cudaMemsetAsync(total, 0, 8, st); return; }
    int64_t per = 256 * 8, bl = (n + per - 1) / per;
    cudaMemsetAsync(tile_state, 0, (size_t)bl * 8, st); cudaMemsetAsync(ticket, 0, 4, st);
    compact_gather_kernel<<<(unsigned)bl, 256, 0, st>>>(mask, n, src, dst, keep_idx, tile_state, ticket, total);
    LRB_COUNT_LAUNCH();
}

// -------------------------------------------------------------------------------------------- mask compaction
static constexpr int CM_THREADS = 256, CM_ITEMS = 8;
__global__ void __launch_bounds__(CM_THREADS) compact_mask_kernel(const uint8_t *__restrict__ mask, int64_t n, uint32_t *out,
                                                                  uint64_t *tile_state, uint32_t *ticket, uint64_t *total)
{
    __shared__ uint32_t s_scan[33];
    __shared__ uint32_t s_tile; __shared__ uint64_t s_excl;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile;
    const int64_t base = ((int64_t)tile * CM_THREADS + threadIdx.x) * CM_ITEMS;
    uint32_t cnt = 0; uint8_t m[CM_ITEMS];
#pragma unroll
    for (int i = 0; i < CM_ITEMS; ++i) { m[i] = (base + i < n) ? mask[base + i] : 0; cnt += m[i] != 0; }
    uint32_t tot, excl = block_excl_sum(cnt, s_scan, &tot);
    if (warp_id() == 0) { uint64_t e = lookback_exclusive(tile_state, tile, tot, OpAdd()); if (lane_id() == 0) s_excl = e; }
    __syncthreads();
    uint32_t o = (uint32_t)s_excl + excl;
#pragma unroll
    for (int i = 0; i < CM_ITEMS; ++i)
        if (m[i]) out[o++] = (uint32_t)(base + i);
    if ((int64_t)(tile + 1) * CM_THREADS * CM_ITEMS >= n && threadIdx.x == 0) *total = s_excl + tot;
}

void launch_compact_mask(const uint8_t *mask, int64_t n, uint32_t *out, uint64_t *tile_state, uint32_t *ticket, uint64_t *total, cudaStream_t st)
{
    if (n <= 0) { cudaMemsetAsync(total, 0, 8, st); return; }
    int64_t per = (int64_t)CM_THREADS * CM_ITEMS, bl = (n + per - 1) / per;
    cudaMemsetAsync(tile_state, 0, (size_t)bl * 8, st); cudaMemsetAsync(ticket, 0, 4, st);
    compact_mask_kernel<<<(unsigned)bl, CM_THREADS, 0, st>>>(mask, n, out, tile_state, ticket, total);
    LRB_COUNT_LAUNCH();
}

// ----------------------------------------------------------------------------------------------- generic scans
static constexpr int GS_THREADS = 256, GS_ITEMS = 8;
__global__ void __launch_bounds__(GS_THREADS) scan_sum_u32_kernel(const uint32_t *__restrict__ in, uint32_t *out, int64_t n,
                                                                  uint64_t *tile_state, uint32_t *ticket, uint64_t *total)
{
    __shared__ uint32_t s_scan[33]; __shared__ uint32_t s_tile; __shared__ uint64_t s_excl;
    if (threadIdx.x == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile;
    const int64_t base = ((int64_t)tile * GS_THREADS + threadIdx.x) * GS_ITEMS;
    uint32_t v[GS_ITEMS], sum = 0;
#pragma unroll
    for (int i = 0; i < GS_ITEMS; ++i) { v[i] = (base + i < n) ? in[base + i] : 0; sum += v[i]; }
    uint32_t tot, excl = block_excl_sum(sum, s_scan, &tot);
    if (warp_id() == 0) { uint64_t e = lookback_exclusive(tile_state, tile, tot, OpAdd()); if (lane_id() == 0) s_excl = e; }
    __syncthreads();
    uint32_t o = (uint32_t)s_excl + excl;
#pragma unroll
    for (int i = 0; i < GS_ITEMS; ++i) if (base + i < n) { out[base + i] = o; o += v[i]; }
    if ((int64_t)(tile + 1) * GS_THREADS * GS_ITEMS >= n && threadIdx.x == 0 && total) *total = s_excl + tot;
}
void launch_scan_sum_u32(const uint32_t *in, uint32_t *out_excl, int64_t n, uint64_t *tile_state, uint32_t *ticket, uint64_t *total, cudaStream_t st)
{
    if (n <= 0) { if (total) cudaMemsetAsync(total, 0, 8, st); return; }
    int64_t per = (int64_t)GS_THREADS * GS_ITEMS, bl = (n + per - 1) / per;
    cudaMemsetAsync(tile_state, 0, (size_t)bl * 8, st); cudaMemsetAsync(ticket, 0, 4, st);
    scan_sum_u32_kernel<<<(unsigned)bl, GS_THREADS, 0, st>>>(in, out_excl, n, tile_state, ticket, total);
    LRB_COUNT_LAUNCH();
}

}  // namespace lrbk
