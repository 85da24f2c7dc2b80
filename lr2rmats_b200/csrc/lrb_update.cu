// lrb_update.cu -- K3/K4/K5: classification against the annotation, short-read SJ support, split pieces, and the
// locus-parallel greedy merge fold.
//
// Replaces, for all reads at once:
//   check_with_anno_trans / comp_trans / check_full / set_full / check_splice_site   update_gtf.c:629-696,717-835
//   check_with_short_sj / check_short_sj / check_short_sj1                           update_gtf.c:589-627,698-709
//   split_trans                                                                       update_gtf.c:837-913
//   merge_trans / merge_trans1 / merge_trans2 + check_iden                            update_gtf.c:98-163, gtf.c:54-92
//
// The reference's two monotone cursors are replaced by closed forms over prefix-max keys (SURVEY App. B.1/B.2), which
// makes every read independent; the order-dependent merge fold is exact per locus (App. A.6/B.3) and loci run in
// parallel, one warp each, the warp evaluating a whole window of the back-scan per step.
#include <cstdlib>
#include <climits>
#include <vector>
#include "lrb_common.cuh"
#include "lrb_kernels.cuh"

namespace lrbk {

extern int64_t g_launches_update;
int64_t g_launches_update = 0;
#define LRB_COUNT_LAUNCH() (++g_launches_update)

static constexpr int CL_THREADS = 256;
static constexpr int CL_ITERS = 4;                    // rows per block = (CL_THREADS / G) * CL_ITERS

LRB_DEVINL bool ex_ovlp(int s1, int e1, int s2, int e2) { return !(s1 > e2 || s2 > e1); }
// exon_overlap_frac (update_gtf.c:80-89): double quotient rounded to float
LRB_DEVINL float ovlp_frac(int s1, int e1, int s2, int e2)
{
    if (s1 > e2 || s2 > e1) return 0.0f;
    int ov = min(e1, e2) - max(s1, s2) + 1;
    int ml = min(e1 - s1 + 1, e2 - s2 + 1);
    return (float)__ddiv_rn((double)ov, (double)ml + 0.0);
}

// first index in [0,n) with a[idx] >= key (small sorted exon arrays of one transcript)
LRB_DEVINL int small_lower_bound(const int *a, int n, int key)
{
    int lo = 0, hi = n;
    while (lo < hi) { int mid = (lo + hi) >> 1; if (a[mid] < key) lo = mid + 1; else hi = mid; }
    return lo;
}

// ------------------------------------------------------------------------- classification rules (both kernels below)
// A rule that lanes share is templated on the group width G (G lanes per read, G == 1: one thread per read); all lanes of a group
// call it with the same arguments.
LRB_DEVINL uint64_t tid_key(int tid) { return (uint64_t)(uint32_t)(tid + 1) << 32; }     // high half of the (tid+1)<<32 | coordinate keys

// Rows are sorted by (tid,start), so the annotation cursor F(b), the SJ cursor S(b) and the first SJ row at or after start - dis are
// monotone in the row index: six searches bracket them for the rows [r0, r1) of a tile.  Search q: F (q = 0, 1), S (2, 3), the donor
// row (4, 5), each at the first (even q) and the last (odd q) row.
template <int G>
LRB_DEVINL int tile_window(const ClassArgs &a, int q, int64_t r0, int64_t r1, unsigned gm, int gl)
{
    const int64_t rr = (q & 1) ? r1 - 1 : r0;
    const uint64_t tk = tid_key(a.rows.tid[rr]);
    const int st = a.rows.start[rr];
    if (q < 2) return (int)group_upper_bound<G, uint64_t>(gm, gl, a.anno.pmax_key, 0, a.anno.n, tk | (uint32_t)st);
    if (!a.sj.n) return 0;
    if (q < 4) return (int)group_upper_bound<G, uint64_t>(gm, gl, a.sj.pmax_key, 0, a.sj.n, tk | (uint32_t)st);
    return (int)group_lower_bound<G, uint64_t>(gm, gl, a.sj.don_key, 0, a.sj.n, tk | (uint32_t)max(st - a.up.ss_dis, 0));
}
struct TileWin { int Flo, Fhi, Slo, Shi, Dlo, Dhi; };
LRB_DEVINL TileWin tile_windows(const int *s) { return {s[0], max(s[0], s[1]), s[2], max(s[2], s[3]), s[4], max(s[4], s[5])}; }

// the closed forms need the rows in (tid,start) order: a row out of order sets err_flags bit 0
LRB_DEVINL void check_row_order(const ClassArgs &a, int64_t row, int tid_b, int start_b)
{
    if (row == 0) return;
    const int pt = a.rows.tid[row - 1], ps = a.rows.start[row - 1];
    if (pt > tid_b || (pt == tid_b && ps > start_b)) atomicOr(a.err_flags, 1u);
}

// comp_trans (the sweep of update_gtf.c:792-835): the transcript lies after the read (< 0: the sweep ends) or before it (> 0: skipped)
LRB_DEVINL bool anno_after(int tid_b, int end_b, int at, int as) { return tid_b < at || (tid_b == at && end_b <= as); }
LRB_DEVINL bool anno_before(int tid_b, int start_b, int at, int ae) { return at < tid_b || (at == tid_b && ae <= start_b); }

struct ClassState {
    int lfull = 0, rfull = 0, lnoth = 1, rnoth = 1;   // check_full
    int known = 0, known_site = 0, ref = -1;
};

// check_full, update_gtf.c:629-681: the read's first exon [b0s, b0e] and last exon [bls, ble] against transcript (xs, xe, na)
template <int G>
LRB_DEVINL void check_full(ClassState &c, int level, int b0s, int b0e, int bls, int ble, const int *xs, const int *xe, int na, unsigned gm, int gl)
{
    if ((c.lfull && c.rfull) || level > 4) return;
    const int a0s = xs[0], a0e = xe[0], als = xs[na - 1], ale = xe[na - 1];
    if (level == 1) {
        if (!c.lfull && b0e == a0e) c.lfull = 1;
        if (!c.rfull && bls == als) c.rfull = 1;
    } else if (level == 2) {
        if (!c.lfull && ex_ovlp(b0s, b0e, a0s, a0e)) c.lfull = 1;
        if (!c.rfull && ex_ovlp(bls, ble, als, ale)) c.rfull = 1;
    } else if (level == 3 || level == 4) {
        bool need_l = false, need_r = false;
        if (!c.lfull) { if (ex_ovlp(b0s, b0e, a0s, a0e)) c.lfull = 1; else need_l = c.lnoth; }
        if (level == 3 && !c.rfull) { if (ex_ovlp(bls, ble, als, ale)) c.rfull = 1; else need_r = c.rnoth; }
        if (need_l | need_r) {
            int lany = 0, rany = 0;
            for (int k = gl; k < na; k += G) { const int s2 = xs[k], e2 = xe[k]; lany |= ex_ovlp(b0s, b0e, s2, e2); rany |= ex_ovlp(bls, ble, s2, e2); }
            if (need_l && group_or<G>(gm, lany)) c.lnoth = 0;
            if (need_r && group_or<G>(gm, rany)) c.rnoth = 0;
        }
    }
}

// update_gtf.c:806-811: a single-exon read is known through a single-exon transcript it overlaps by at least -f
LRB_DEVINL bool single_exon_known(const ClassArgs &a, int b0s, int b0e, int a0s, int a0e)
{
    return ovlp_frac(b0s, b0e, a0s, a0e) >= a.up.single_exon_ovlp_frac;
}

// check_splice_site's verdict for transcript i (update_gtf.c:812-821): every splice site of the read inside the overlap matches -> known,
// and the sweep ends (true); some match -> known_site through this transcript
LRB_DEVINL bool splice_verdict(ClassState &c, int n, int ovl, int iden, int i)
{
    if (2 * (n - 1) == ovl && ovl == iden) { c.known = 1; c.ref = i; return true; }
    if (iden > 0) { c.known_site = 1; c.ref = i; }
    return false;
}

// set_full, update_gtf.c:683-696
LRB_DEVINL int set_full(const ClassState &c, int level)
{
    if (level == 5) return 1;
    if (level == 4) return c.lfull || c.lnoth;
    if (level == 3) return (c.lfull || c.lnoth) && (c.rfull || c.rnoth);
    return c.lfull && c.rfull;
}

// check_with_short_sj, update_gtf.c:589-627, cursor closed form (App. B.2): false when the SJ cursor S(b) has no junction row left that
// starts inside the read.  Else R0 = the first row with the read's tid and donor >= start - dis, never below S.
template <int G>
LRB_DEVINL bool sj_cursor(const ClassArgs &a, const TileWin &w, uint64_t key_b, int tid_b, int start_b, int end_b, unsigned gm, int gl, int64_t &R0)
{
    const int64_t S = group_upper_bound<G, uint64_t>(gm, gl, a.sj.pmax_key, w.Slo, w.Shi, key_b);
    if (S >= a.sj.n) return false;
    const int st = a.sj.tid[S];
    if (st > tid_b || (st == tid_b && a.sj.don[S] >= end_b)) return false;
    R0 = group_lower_bound<G, uint64_t>(gm, gl, a.sj.don_key, w.Dlo, w.Dhi, tid_key(tid_b) | (uint32_t)max(start_b - a.up.ss_dis, 0));
    if (R0 < S) R0 = S;
    return true;
}

// check_short_sj / check_short_sj1 (:698-709) for the intron [is, ie]: an SJ row with the read's tid, donor in [is-dis, is+dis] and below
// ie, acceptor within dis of ie and enough reads (-j, -J).  The rows are searched from `from` on (gallop, then bisect); `from` moves to
// the first row of the donor window, where the search for a later intron of a chain with ascending introns may start.
LRB_DEVINL bool sj_supported(const ClassArgs &a, int tid_b, int is, int ie, int64_t &from)
{
    const int dis = a.up.ss_dis;
    const uint64_t tk = tid_key(tid_b);
    int dlo = is - dis; if (dlo < 0) dlo = 0;
    int64_t dhi = (int64_t)is + dis + 1; if (dhi > ie) dhi = ie; if (dhi < 0) dhi = 0;
    const uint64_t klo = tk | (uint32_t)dlo, khi = tk | (uint64_t)dhi;
    int64_t lo = from, step = 1, hi = from;
    while (hi < a.sj.n && a.sj.don_key[hi] < klo) { lo = hi + 1; hi += step; step <<= 1; }
    if (hi > a.sj.n) hi = a.sj.n;
    lo = lower_bound_dev<uint64_t>(a.sj.don_key, lo, hi, klo);
    from = lo;
    for (int64_t q = lo; q < a.sj.n; ++q) {
        if (a.sj.don_key[q] >= khi) break;
        if (iabs_dev(a.sj.acc[q] - ie) <= dis) {
            const int c = a.up.use_multi ? a.sj.cnt_u[q] + a.sj.cnt_m[q] : a.sj.cnt_u[q];
            if (c >= a.up.min_sj_cnt) return true;
        }
    }
    return false;
}

// split_trans (update_gtf.c:837-913): the chain of n exons is cut after every unreliable junction; a piece of at least two exons with a
// novel and a known junction is emitted as emit(first exon, last exon).  novel_junc(k) / unreliable(k): flags of junction k (< n - 1).
template <class NovelJ, class Unrel, class Emit>
LRB_DEVINL void split_trans(int n, NovelJ novel_junc, Unrel unreliable, Emit emit)
{
    int last = 0, has_novel = 0, has_known = 0;
    for (int k = 0; k <= n - 1; ++k) {
        const bool at_end = k == n - 1;
        if (!at_end) { if (novel_junc(k)) has_novel = 1; else has_known = 1; }
        if (at_end || unreliable(k)) {
            if (has_novel && has_known && k - last >= 1) emit(last, k);
            last = k + 1; has_novel = 0; has_known = 0;
        }
    }
}

LRB_DEVINL uint32_t class_word(const ClassState &c, int full, int sj_checked, int unreliable)
{
    return (c.known ? LRB_C_KNOWN : 0) | (c.known_site ? LRB_C_KNOWN_SITE : 0) | (unreliable ? LRB_C_UNRELIABLE : 0) | (full ? LRB_C_FULL : 0) |
           (c.lfull ? LRB_C_LFULL : 0) | (c.rfull ? LRB_C_RFULL : 0) | (c.lnoth ? LRB_C_LNOTH : 0) | (c.rnoth ? LRB_C_RNOTH : 0) |
           (sj_checked ? LRB_C_SJ_CHECKED : 0);
}

// ------------------------------------------------------------------------------------- classification, lane group per read
// G lanes per read (power of two), CL_SLOTS exon slots per read staged in shared memory
template <int G, int CL_SLOTS>
__global__ void __launch_bounds__(CL_THREADS) classify_kernel(ClassArgs a, const uint8_t *__restrict__ only)
{
    constexpr int GPB = CL_THREADS / G;
    constexpr int STRIDE = CL_SLOTS + G;             // STRIDE = G * odd: the 32/G groups of a warp land on disjoint banks
    static_assert(((STRIDE / G) & 1) == 1 && STRIDE % G == 0, "bank-conflict-free stride");
    __shared__ int s_es[GPB][STRIDE], s_ee[GPB][STRIDE];
    __shared__ uint8_t s_fl[GPB][STRIDE];
    __shared__ int s_win[6];
    const int g = threadIdx.x / G, gl = threadIdx.x % G;
    const unsigned gm = group_mask<G>();
    const int dis = a.up.ss_dis, level = a.up.full_level;

    const int64_t r0 = (int64_t)blockIdx.x * GPB * CL_ITERS;
    const int64_t r1 = min(a.rows.n, r0 + (int64_t)GPB * CL_ITERS);
    if (only) {                                      // nothing left for this block after classify_row_kernel?
        int any = 0;
        for (int64_t r = r0 + threadIdx.x; r < r1; r += CL_THREADS) any |= only[r];
        if (!__syncthreads_or(any)) return;
    }
    if (threadIdx.x < 6) s_win[threadIdx.x] = tile_window<1>(a, threadIdx.x, r0, r1, FULL, 0);      // one thread per search
    __syncthreads();
    const TileWin w = tile_windows(s_win);

    for (int64_t row = r0 + g; row < r1; row += GPB) {
        if (only && !only[row]) continue;               // classified by classify_row_kernel
        const int n = (int)a.rows.ex_n[row];
        const uint32_t beg = a.rows.ex_beg[row];
        const int tid_b = a.rows.tid[row], start_b = a.rows.start[row], end_b = a.rows.end[row];
        if (n == 0) { if (gl == 0) { atomicOr(a.err_flags, 2u); a.cls[row] = 0; a.ref[row] = -1; a.n_novel[row] = 0; } continue; }
        if (gl == 0) check_row_order(a, row, tid_b, start_b);
        // exon chain + flags: shared memory when it fits, else straight on the HBM arrays
        const bool in_smem = n <= CL_SLOTS;
        int *es = in_smem ? s_es[g] : a.ex.es + beg, *ee = in_smem ? s_ee[g] : a.ex.ee + beg;
        uint8_t *fl = in_smem ? s_fl[g] : a.ex.flag + beg;
        __syncwarp(gm);
        for (int j = gl; j < n; j += G) {
            if (in_smem) { es[j] = a.ex.es[beg + j]; ee[j] = a.ex.ee[beg + j]; }
            fl[j] = (j < n - 1) ? (LRB_F_NOVEL_EXON | LRB_F_NOVEL_DON | LRB_F_NOVEL_ACC | LRB_F_NOVEL_JUNC) : LRB_F_NOVEL_EXON;
        }
        __syncwarp(gm);
        const int b0s = es[0], b0e = ee[0], bls = es[n - 1], ble = ee[n - 1];

        // ---- annotation window: F(b) by a cooperative search on the prefix-max keys, sweep to the first "after"
        const uint64_t key_b = tid_key(tid_b) | (uint32_t)start_b;
        ClassState c;
        for (int i = (int)group_upper_bound<G, uint64_t>(gm, gl, a.anno.pmax_key, w.Flo, w.Fhi, key_b); i < a.anno.n; ++i) {
            const int at = a.anno.tid[i], as_ = a.anno.start[i], ae_ = a.anno.end[i];
            if (anno_after(tid_b, end_b, at, as_)) break;
            if (anno_before(tid_b, start_b, at, ae_)) continue;
            const uint32_t ao = a.anno.exon_off[i]; const int na = (int)(a.anno.exon_off[i + 1] - ao);
            const int *xs = a.anno.es + ao, *xe = a.anno.ee + ao;
            check_full<G>(c, level, b0s, b0e, bls, ble, xs, xe, na, gm, gl);
            if (n == 1 && na == 1) {
                if (single_exon_known(a, b0s, b0e, xs[0], xe[0])) { c.ref = i; c.known = 1; break; }
            } else if (n > 1 && na > 1) {                                                  // check_splice_site :717-779
                const int os = max(start_b, as_), oe = min(end_b, ae_);
                int ovl = 0, iden = 0;
                if (dis == 0 && a.anno.mono[i]) {
                    // exact-match fast path: exon starts and ends of this transcript are strictly increasing, so every read
                    // coordinate matches at most one annotation exon -- two binary searches per read exon replace the
                    // na x n sweep, and the pair counts of the reference become match counts.
                    for (int j = gl; j < n; j += G) {
                        const int bs = es[j], be = ee[j];
                        const int ie = small_lower_bound(xe, na, be), is = small_lower_bound(xs, na, bs);
                        const bool hit_e = ie < na && xe[ie] == be, hit_s = is < na && xs[is] == bs;
                        uint8_t f = fl[j], f0 = f;
                        if (j < n - 1) {
                            const int sn = es[j + 1];
                            ovl += (be >= os && be <= oe) + (sn >= os && sn <= oe);
                            if (hit_e && ie < na - 1) {
                                if (be >= os && be <= oe) { ++iden; f &= ~LRB_F_NOVEL_DON; }
                                if (xs[ie + 1] == sn) f &= ~LRB_F_NOVEL_JUNC;
                            }
                            if (hit_s && is >= 1 && bs >= os && bs <= oe) { ++iden; f &= ~LRB_F_NOVEL_ACC; }
                        }
                        if (hit_s && hit_e && is == ie) f &= ~LRB_F_NOVEL_EXON;
                        if (f != f0) fl[j] = f;
                    }
                } else {
                    for (int j = gl; j < n - 1; j += G) {
                        int e = ee[j], s = es[j + 1];
                        ovl += (e >= os && e <= oe) + (s >= os && s <= oe);
                    }
                    for (int k = 0; k < na; ++k) {
                        const int a_s = xs[k], a_e = xe[k];
                        const bool has_next = k < na - 1;
                        const int a_sn = has_next ? xs[k + 1] : 0;
                        const bool don_ok = has_next && a_e >= os && a_e <= oe;
                        const bool acc_ok = k >= 1 && a_s >= os && a_s <= oe;
                        for (int j = gl; j < n; j += G) {
                            const int bs = es[j], be = ee[j];
                            uint8_t f = fl[j], f0 = f;
                            const bool de = iabs_dev(a_e - be) <= dis, ds = iabs_dev(a_s - bs) <= dis;
                            if (j < n - 1) {
                                if (don_ok && de) { ++iden; f &= ~LRB_F_NOVEL_DON; }
                                if (acc_ok && ds) { ++iden; f &= ~LRB_F_NOVEL_ACC; }
                                if (has_next && de && iabs_dev(a_sn - es[j + 1]) <= dis) f &= ~LRB_F_NOVEL_JUNC;
                            }
                            if (ds && de) f &= ~LRB_F_NOVEL_EXON;
                            if (f != f0) fl[j] = f;
                        }
                    }
                }
                if (splice_verdict(c, n, group_sum<G>(gm, ovl), group_sum<G>(gm, iden), i)) break;
            }
        }
        int is_rev = a.rows.is_rev[row];
        if (c.ref != -1) is_rev = a.anno.is_rev[c.ref];                                   // update_gtf.c:823-833
        const int full = set_full(c, level);
        __syncwarp(gm);

        // ---- short-read SJ support; a chain here need not have ascending introns, so every intron is searched from R0
        int sj_checked = 0, unreliable = 0;
        if (full && !c.known && c.known_site && a.sj.n > 0) {
            sj_checked = 1;
            int64_t R0;
            unreliable = !sj_cursor<G>(a, w, key_b, tid_b, start_b, end_b, gm, gl, R0);
            if (!unreliable) {
                int bad = 0;
                for (int j = gl; j < n - 1; j += G) {
                    int64_t from = R0;
                    if ((fl[j] & LRB_F_NOVEL_JUNC) && !sj_supported(a, tid_b, ee[j] + 1, es[j + 1] - 1, from)) { fl[j] |= LRB_F_UNRELIABLE; bad = 1; }
                }
                unreliable = group_or<G>(gm, bad);
            }
        }
        __syncwarp(gm);

        // ---- novel_T contribution: the read itself, or its split pieces
        uint32_t nn = 0;
        if (full && !c.known && c.known_site) {
            if (!sj_checked || !unreliable) nn = 1;
            else if (a.up.split_trans && gl == 0)
                split_trans(n, [&](int k) { return (fl[k] & LRB_F_NOVEL_JUNC) != 0; }, [&](int k) { return (fl[k] & LRB_F_UNRELIABLE) != 0; },
                            [&](int, int) { ++nn; });
        }
        if (in_smem) for (int j = gl; j < n; j += G) a.ex.flag[beg + j] = fl[j];
        if (gl == 0) {
            a.cls[row] = class_word(c, full, sj_checked, unreliable);
            a.ref[row] = c.ref;
            a.rows.is_rev[row] = (uint8_t)is_rev;
            a.n_novel[row] = nn;
        }
    }
}

// ---------------------------------------------------------------------------------- classification, thread per read
// The common case (exact splice-site matching, reads and window transcripts with increasing exon coordinates, at most
// 32 exons per read) runs here; every other read is flagged in `slow` and goes through classify_kernel above, which
// implements the same rules without those restrictions.  One thread replays the reference's sweep for one read: the 32
// reads of a warp are neighbours in (tid,start) order, so they sweep the same transcripts -- annotation loads are warp
// broadcasts and the lanes stay converged.  Per (read, transcript) pair one merge walk over the two sorted exon lists
// replaces the reference's three nested loops; the four per-exon flag arrays live in four 32-bit registers.

template <int CR_THREADS, int CR_MINB>
__global__ void __launch_bounds__(CR_THREADS, CR_MINB) classify_row_kernel(ClassArgs a, uint8_t *__restrict__ slow, const uint8_t *__restrict__ row_nonmono, int by_exon_count)
{
    __shared__ int s_win[6];
    __shared__ int s_hist[34]; __shared__ uint8_t s_perm[CR_THREADS];
    int t = threadIdx.x;
    const int dis = a.up.ss_dis, level = a.up.full_level;
    const int64_t r0 = (int64_t)blockIdx.x * CR_THREADS, r1 = min(a.rows.n, r0 + (int64_t)CR_THREADS);
    for (int q = warp_id(); q < 6; q += CR_THREADS / 32) {          // six cooperative 33-ary searches, warps 0..3
        const int v = tile_window<32>(a, q, r0, r1, FULL, lane_id());
        if (lane_id() == 0) s_win[q] = v;
    }
    __syncthreads();
    if (by_exon_count) {
        // the rows of the tile are dealt to the threads in order of their exon count (stable counting sort in shared memory):
        // the lanes of a warp then run merge walks of the same length, at the price of sweeping different transcripts
        if (t < 34) s_hist[t] = 0;
        __syncthreads();
        const int64_t rr = r0 + t;
        int key = 33, rank = 0;
        if (rr < r1) { const int nn = (int)a.rows.ex_n[rr]; key = nn < 0 ? 0 : nn > 32 ? 32 : nn; }
        // rank inside the key class = number of earlier threads with the same key (warp ballots + per-warp offsets)
        const unsigned peers = __match_any_sync(FULL, key);
        const int lane = lane_id();
        rank = __popc(peers & ((1u << lane) - 1u));
        __shared__ int s_wcnt[CR_THREADS / 32][34];
        for (int q = t; q < (CR_THREADS / 32) * 34; q += CR_THREADS) (&s_wcnt[0][0])[q] = 0;
        __syncthreads();
        if (rank == 0) s_wcnt[warp_id()][key] = __popc(peers);
        __syncthreads();
        if (t < 34) { int acc = 0; for (int w = 0; w < CR_THREADS / 32; ++w) { const int v = s_wcnt[w][t]; s_wcnt[w][t] = acc; acc += v; } s_hist[t] = acc; }
        __syncthreads();
        if (t == 0) { int acc = 0; for (int k = 0; k < 34; ++k) { const int v = s_hist[k]; s_hist[k] = acc; acc += v; } }
        __syncthreads();
        s_perm[s_hist[key] + s_wcnt[warp_id()][key] + rank] = (uint8_t)t;
        __syncthreads();
        t = s_perm[t];
    }
    const int64_t row = r0 + t;
    if (row >= r1) return;
    const TileWin w = tile_windows(s_win);
    const int n = (int)a.rows.ex_n[row];
    const uint32_t beg = a.rows.ex_beg[row];
    const int tid_b = a.rows.tid[row], start_b = a.rows.start[row], end_b = a.rows.end[row];
    check_row_order(a, row, tid_b, start_b);
    if (dis != 0 || n < 1 || n > 32 || (row_nonmono && row_nonmono[row])) { slow[row] = 1; return; }
    const int *__restrict__ es = a.ex.es + beg, *__restrict__ ee = a.ex.ee + beg;
    const int b0s = es[0], b0e = ee[0], bls = es[n - 1], ble = ee[n - 1];
    const uint64_t key_b = tid_key(tid_b) | (uint32_t)start_b;

    // ---- annotation window: F(b) on the prefix-max keys, sweep to the first "after" (update_gtf.c:792-835)
    ClassState c;
    uint32_t c_don = 0, c_acc = 0, c_junc = 0, c_exon = 0;                                     // cleared novel_* flags, bit j
    for (int i = (int)upper_bound_dev<uint64_t>(a.anno.pmax_key, w.Flo, w.Fhi, key_b); i < a.anno.n; ++i) {
        const int at = a.anno.tid[i], as_ = a.anno.start[i];
        if (anno_after(tid_b, end_b, at, as_)) break;
        const int ae_ = a.anno.end[i];
        if (anno_before(tid_b, start_b, at, ae_)) continue;
        if (!a.anno.mono[i]) { slow[row] = 1; return; }                                         // nothing was written yet
        const uint32_t ao = a.anno.exon_off[i]; const int na = (int)(a.anno.exon_off[i + 1] - ao);
        const int *__restrict__ xs = a.anno.es + ao, *__restrict__ xe = a.anno.ee + ao;
        check_full<1>(c, level, b0s, b0e, bls, ble, xs, xe, na, FULL, 0);
        if (n == 1 && na == 1) {
            if (single_exon_known(a, b0s, b0e, xs[0], xe[0])) { c.ref = i; c.known = 1; break; }
        } else if (n > 1 && na > 1) {                                                           // check_splice_site :717-779, exact matching
            const int os = max(start_b, as_), oe = min(end_b, ae_);
            int ovl = 0, iden = 0, ps = 0, pe = 0, bs = b0s, be = b0e;
            {   // both cursors jump over the transcript's exons in front of the read (the skipped prefix of a 5'-truncated read)
                // by one paired binary search; its trip count depends on na only, so the lanes sweeping this transcript stay converged
                int ls = na, le = na;
                while (ls | le) {
                    const int hs = ls >> 1, he = le >> 1;
                    const int vs = ls ? xs[ps + hs] : INT_MAX, ve = le ? xe[pe + he] : INT_MAX;
                    if (vs < bs) { ps += hs + 1; ls -= hs + 1; } else ls = hs;
                    if (ve < be) { pe += he + 1; le -= he + 1; } else le = he;
                }
            }
            for (int j = 0; j < n; ++j) {
                // advance both cursors to the first annotation start >= bs / end >= be.  The usual step is 0..2 exons: the two
                // next values of each list are fetched together (four independent loads, one latency) and the cursors move by
                // selects; only a longer jump (the skipped prefix of a truncated read) walks
                int s0 = ps < na ? xs[ps] : INT_MAX, s1 = ps + 1 < na ? xs[ps + 1] : INT_MAX;
                int e0 = pe < na ? xe[pe] : INT_MAX, e1 = pe + 1 < na ? xe[pe + 1] : INT_MAX;
                if (s0 < bs) {
                    ++ps; s0 = s1;
                    if (s0 < bs) { ++ps; s0 = INT_MAX; while (ps < na && (s0 = xs[ps]) < bs) { ++ps; s0 = INT_MAX; } }
                }
                if (e0 < be) {
                    ++pe; e0 = e1;
                    if (e0 < be) { ++pe; e0 = INT_MAX; while (pe < na && (e0 = xe[pe]) < be) { ++pe; e0 = INT_MAX; } }
                }
                const bool hit_s = s0 == bs, hit_e = e0 == be;
                const uint32_t bit = 1u << j;
                if (hit_s && hit_e && ps == pe) c_exon |= bit;
                if (j < n - 1) {
                    const int sn = es[j + 1];
                    ovl += (be >= os && be <= oe) + (sn >= os && sn <= oe);
                    if (hit_e && pe < na - 1) {
                        if (be >= os && be <= oe) { ++iden; c_don |= bit; }
                        if (xs[pe + 1] == sn) c_junc |= bit;
                    }
                    if (hit_s && ps >= 1 && bs >= os && bs <= oe) { ++iden; c_acc |= bit; }
                    bs = sn; be = ee[j + 1];
                }
            }
            if (splice_verdict(c, n, ovl, iden, i)) break;
        }
    }
    const int full = set_full(c, level);

    // ---- short-read SJ support: the introns of a chain here ascend, so each search starts where the last one ended
    int sj_checked = 0, unreliable = 0;
    uint32_t unrel = 0;
    if (full && !c.known && c.known_site && a.sj.n > 0) {
        sj_checked = 1;
        int64_t R0;
        unreliable = !sj_cursor<1>(a, w, key_b, tid_b, start_b, end_b, FULL, 0, R0);
        if (!unreliable) {
            uint32_t nj = ~c_junc & (n >= 2 ? (0xffffffffu >> (33 - n)) : 0u);              // novel junctions j < n-1, ascending
            while (nj) {
                const int j = __ffs(nj) - 1; nj &= nj - 1;
                if (!sj_supported(a, tid_b, ee[j] + 1, es[j + 1] - 1, R0)) unrel |= 1u << j;
            }
            unreliable = unrel != 0;
        }
    }

    // ---- novel_T contribution: the read itself, or its split pieces
    uint32_t nn = 0;
    if (full && !c.known && c.known_site) {
        if (!sj_checked || !unreliable) nn = 1;
        else if (a.up.split_trans)
            split_trans(n, [&](int k) { return !((c_junc >> k) & 1u); }, [&](int k) { return ((unrel >> k) & 1u) != 0; }, [&](int, int) { ++nn; });
    }
    uint8_t *fl = a.ex.flag + beg;
    for (int j = 0; j < n; ++j) {
        uint32_t f = ((c_exon >> j) & 1u) ? 0u : LRB_F_NOVEL_EXON;
        if (j < n - 1) {
            if (!((c_don >> j) & 1u)) f |= LRB_F_NOVEL_DON;
            if (!((c_acc >> j) & 1u)) f |= LRB_F_NOVEL_ACC;
            if (!((c_junc >> j) & 1u)) f |= LRB_F_NOVEL_JUNC;
            if ((unrel >> j) & 1u) f |= LRB_F_UNRELIABLE;
        }
        fl[j] = (uint8_t)f;
    }
    slow[row] = 0;
    a.cls[row] = class_word(c, full, sj_checked, unreliable);
    a.ref[row] = c.ref;
    if (c.ref != -1) a.rows.is_rev[row] = a.anno.is_rev[c.ref];                                 // update_gtf.c:823-833
    a.n_novel[row] = nn;
}

template <int G, int SLOTS> static void launch_classify_t(const ClassArgs &a, const uint8_t *only, cudaStream_t st)
{
    constexpr int per_block = (CL_THREADS / G) * CL_ITERS;
    int64_t bl = (a.rows.n + per_block - 1) / per_block;
    classify_kernel<G, SLOTS><<<(unsigned)bl, CL_THREADS, 0, st>>>(a, only);
}
void launch_classify(const ClassArgs &a, uint8_t *slow, cudaStream_t st)
{
    if (a.rows.n <= 0) return;
    // the common case (-d 0) row by row with rows dealt to lanes by exon count (128 threads, 8 CTAs per SM: measured best on B200,
    // profiles/r01_v13_classify_*_ab.txt); what that kernel flags as slow (> 32 exons, non-monotone chains) and every row of -d > 0 goes
    // through the general kernel, 4 lanes per row
    const uint8_t *only = nullptr;
    if (a.up.ss_dis == 0 && slow) {
        classify_row_kernel<128, 8><<<(unsigned)((a.rows.n + 127) / 128), 128, 0, st>>>(a, slow, a.row_nonmono, 1); LRB_COUNT_LAUNCH();
        only = slow;
    }
    launch_classify_t<4, 16>(a, only, st); LRB_COUNT_LAUNCH();
}

// ------------------------------------------------------------------ class lists: novel_T / known_T / unrecog_T in one pass
// One pass over the classified rows builds, in row order: novel_T (whole reads and the split pieces of split_trans,
// update_gtf.c:837-913), the known_T and unrecog_T row lists (:941-962), and -- for the summary -- the class of every row
// (0 known, 1 novel with all junctions reliable, 2 novel with an unreliable junction, 3 unrecognized; :501-528) with the class
// sizes.  Three running counts ride on two look-back chains; the list sizes stay on the device (totals[0..2]).
static constexpr int LS_THREADS = 256, LS_ITEMS = 4;
__global__ void __launch_bounds__(LS_THREADS) build_lists_kernel(ListArgs a)
{
    __shared__ uint32_t s_scan[33];
    __shared__ uint32_t s_tile, s_class[4]; __shared__ uint64_t s_excl[2];
    if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
    if (threadIdx.x < 4) s_class[threadIdx.x] = 0;
    __syncthreads();
    const int tile = (int)s_tile;
    const int64_t base = ((int64_t)tile * LS_THREADS + threadIdx.x) * LS_ITEMS;
    uint32_t cw[LS_ITEMS], nn[LS_ITEMS], nn_sum = 0, kn_sum = 0, un_sum = 0, flags = 0, ccnt = 0;   // ccnt: four 8-bit class counters
#pragma unroll
    for (int i = 0; i < LS_ITEMS; ++i) {
        cw[i] = 0; nn[i] = 0;
        if (base + i < a.rows.n) {
            const uint32_t c = a.cls[base + i];
            cw[i] = c; nn[i] = a.n_novel[base + i];
            const bool full = c & LRB_C_FULL, known = c & LRB_C_KNOWN, ks = c & LRB_C_KNOWN_SITE, ur = c & LRB_C_UNRELIABLE;
            const uint32_t kn = full && known, un = full && !known && !ks;
            flags |= (kn | (un << 1)) << (2 * i);
            nn_sum += nn[i]; kn_sum += kn; un_sum += un;
            if (a.kls) { const int k = known ? 0 : (ks ? (ur ? 2 : 1) : 3); a.kls[base + i] = (uint8_t)k; ccnt += 1u << (8 * k); }
        }
    }
    if (a.kls) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) ccnt += __shfl_xor_sync(FULL, ccnt, o);     // <= 128 per class and warp: no carry between the bytes
        if (lane_id() == 0) for (int q = 0; q < 4; ++q) { const uint32_t v = (ccnt >> (8 * q)) & 0xffu; if (v) atomicAdd(&s_class[q], v); }
    }
    uint32_t nn_tot, kn_tot, un_tot;
    uint32_t nn_ex = block_excl_sum(nn_sum, s_scan, &nn_tot), kn_ex = block_excl_sum(kn_sum, s_scan, &kn_tot), un_ex = block_excl_sum(un_sum, s_scan, &un_tot);
    if (warp_id() == 0) {
        const uint64_t e0 = lookback_exclusive(a.tile_state, tile, pack_pair(nn_tot, kn_tot), OpAdd());
        const uint64_t e1 = lookback_exclusive(a.tile_state + a.n_tiles, tile, (uint64_t)un_tot, OpAdd());
        if (lane_id() == 0) { s_excl[0] = e0; s_excl[1] = e1; }
    }
    __syncthreads();
    if (a.kls && threadIdx.x < 4 && s_class[threadIdx.x]) atomicAdd(&a.class_n[threadIdx.x], s_class[threadIdx.x]);
    const uint32_t nn_base = pair_hi(s_excl[0]), kn_base = pair_lo(s_excl[0]), un_base = (uint32_t)s_excl[1];
    if (tile == a.n_tiles - 1 && threadIdx.x == 0) {
        a.totals[0] = (uint64_t)nn_base + nn_tot; a.totals[1] = (uint64_t)kn_base + kn_tot; a.totals[2] = (uint64_t)un_base + un_tot;
    }
    uint32_t o = nn_base + nn_ex, ko = kn_base + kn_ex, uo = un_base + un_ex;
#pragma unroll
    for (int i = 0; i < LS_ITEMS; ++i) {
        const int64_t row = base + i;
        if (row >= a.rows.n) break;
        if ((flags >> (2 * i)) & 1u) a.known[ko++] = (uint32_t)row;
        if ((flags >> (2 * i)) & 2u) a.unrecog[uo++] = (uint32_t)row;
        if (!nn[i]) continue;
        const uint32_t o0 = o; o += nn[i];
        if ((int64_t)o0 + nn[i] > a.novel.cap) continue;             // list sized too small: the host sees the total and repeats the pass
        const uint32_t c = cw[i];
        const int n = (int)a.rows.ex_n[row];
        if (!((c & LRB_C_SJ_CHECKED) && (c & LRB_C_UNRELIABLE))) {
            a.novel.row[o0] = (uint32_t)row; a.novel.lo[o0] = 0; a.novel.cnt[o0] = (uint32_t)n; a.novel.piece[o0] = -1;
            continue;
        }
        const uint8_t *fl = a.ex.flag + a.rows.ex_beg[row];
        int k2 = 0; uint32_t w = o0;
        split_trans(n, [&](int k) { return (fl[k] & LRB_F_NOVEL_JUNC) != 0; }, [&](int k) { return (fl[k] & LRB_F_UNRELIABLE) != 0; }, [&](int lo, int hi) {
            a.novel.row[w] = (uint32_t)row; a.novel.lo[w] = (uint32_t)lo; a.novel.cnt[w] = (uint32_t)(hi - lo + 1); a.novel.piece[w] = k2;
            ++w; ++k2;
        });
    }
}
void launch_build_lists(ListArgs a, cudaStream_t st)
{
    if (a.rows.n <= 0) { cudaMemsetAsync(a.totals, 0, 24, st); return; }
    a.n_tiles = (int)((a.rows.n + LS_THREADS * LS_ITEMS - 1) / (LS_THREADS * LS_ITEMS));
    cudaMemsetAsync(a.tile_state, 0, (size_t)a.n_tiles * 16, st); cudaMemsetAsync(a.ticket, 0, 4, st);
    build_lists_kernel<<<(unsigned)a.n_tiles, LS_THREADS, 0, st>>>(a);
    LRB_COUNT_LAUNCH();
}

__global__ void rows_as_list_kernel(DRows rows, const uint32_t *__restrict__ subset, int64_t n, DTransList out)
{
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    uint32_t row = subset ? subset[k] : (uint32_t)k;
    out.row[k] = row; out.lo[k] = 0; out.cnt[k] = rows.ex_n[row]; out.piece[k] = -1;
}
void launch_rows_as_list(const DRows &rows, const uint32_t *subset, int64_t n, DTransList &out, cudaStream_t st)
{
    if (n <= 0) return;
    rows_as_list_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(rows, subset, n, out);
    LRB_COUNT_LAUNCH();
}

// --------------------------------------------------------------------------------------------------- merge fold
// Candidate SoA (one row per transcript entering the fold), built once by merge_cand_kernel:
//   tid/start/end/rev : trans_t fields (0/0/0/0 for split pieces, SURVEY Q14)      n, gbeg : exon slots in the pools
//   fs/le             : exon[0].start, exon[n-1].end                               hash    : of the internal boundaries
LRB_DEVINL uint64_t mixh(uint64_t h, uint32_t v) { h ^= v; h *= 0x9E3779B97F4A7C15ull; h ^= h >> 29; return h; }
// membership signature of a chain's junctions: two bits per junction in 64 (a Bloom filter with two hash functions: short chains, the
// bulk of the pairs a deep locus compares, pass a foreign junction ~4x less often than with one bit)
LRB_DEVINL uint64_t junc_mask(uint64_t jk) { jk *= 0xD6E8FEB86659FD93ull; return (1ull << (jk >> 58)) | (1ull << ((jk >> 52) & 63u)); }
LRB_DEVINL bool sig_has(uint64_t sig, uint64_t jk) { const uint64_t m = junc_mask(jk); return (sig & m) == m; }

// (clamped to the host bound: an undersized list is detected and redone by the host, the kernels must only stay in bounds)
// (an undersized list -- more candidates on the device than the host's bound -- folds as EMPTY: its tail was never written, the host
// sees the true count in the same round trip and repeats the pass with the exact size)
LRB_DEVINL int64_t cand_count(const MergeArgs &a) { if (!a.n_cand_dev) return a.n_cand; const int64_t n = (int64_t)*a.n_cand_dev; return n > a.n_cand ? 0 : n; }
// the candidates [ls, le) of locus loc
LRB_DEVINL void locus_range(const MergeArgs &a, int64_t n_loci, int64_t loc, int64_t &ls, int64_t &le)
{
    ls = a.locus_start[loc]; le = (loc + 1 < n_loci) ? a.locus_start[loc + 1] : cand_count(a);
}
// class order (launch_class_order): the candidates [cs, ce) of sub-stream k of the locus loc that starts at ls
LRB_DEVINL void class_range(const MergeArgs &a, int64_t loc, int64_t ls, int k, int64_t &cs, int64_t &ce)
{
    const uint4 b0 = a.cbase[loc], b1 = a.cbase[loc + 1];
    const uint32_t n0 = b1.x - b0.x, n1 = b1.y - b0.y, n2 = b1.z - b0.z, n3 = b1.w - b0.w;
    cs = ls + (k > 0 ? n0 : 0u) + (k > 1 ? n1 : 0u) + (k > 2 ? n2 : 0u);
    ce = cs + (k == 0 ? n0 : k == 1 ? n1 : k == 2 ? n2 : n3);
}
// the candidates a replay of (locus, sub-stream my) walks: with sub-streams their own range, else the whole locus
LRB_DEVINL void replay_range(const MergeArgs &a, int64_t n_loci, int64_t loc, int my, int64_t &ls, int64_t &le, int64_t &cs, int64_t &ce)
{
    locus_range(a, n_loci, loc, ls, le);
    if (a.kls) class_range(a, loc, ls, my, cs, ce); else { cs = ls; ce = le; }
}

// Hand-off state of a locus, kept at its head in hard[]: the path that folds the locus next.  A kernel writes it only to hand the
// locus on, so the last value names the path that finished it (merge_fold_census).
enum LocusPath : uint8_t {
    LP_FLAT = 0,                // fold_seq_kernel (at most FF_MAX candidates)
    LP_TIER0 = 1,               // fold_big_kernel tier 0: beyond the flat masks, or given up by the flat kernels
    LP_MERGE_OVER = 2,          // merge_fold_kernel: tier 1's slots overflowed, or FB_MAXREL candidates or more
    LP_MERGE_VERIFY = 3,        // merge_fold_kernel: class verification failed
    LP_TIER1 = 4,               // fold_big_kernel tier 1: tier 0's slots overflowed
};
LRB_DEVINL bool for_merge_fold(int h) { return h == LP_MERGE_OVER || h == LP_MERGE_VERIFY; }
// the other in-band hand-offs of the fold's scratch
static constexpr uint32_t LSTART_DEEP = 0xffffffffu;    // lstart[c]: the locus is deeper than the flat masks: not for the flat relation kernels
static constexpr uint16_t DESC_BIG = 0xFFFFu;           // desc[c]: a member of a locus of the big-locus path (the flat kernels are done with desc by then)
static constexpr uint8_t CLASSES_UNTABULATED = 0xffu;   // locus_cnt byte: too many classes for the relation rows: fold_big_kernel uses its cache

// One pass over the candidates: flatten (CandSoA), running max of (tid,end) across tiles (look-back, max), locus heads
// (a candidate that starts beyond every earlier end on its chromosome, App. B.3) and their compaction into locus_start
// (second look-back chain, sum).  The number of candidates may live on the device (n_cand_dev): the grid is sized by the
// host's upper bound and surplus tiles only pass the chain on.
static constexpr int FP_THREADS = 256, FP_ITEMS = 4;
// The locus heads of one tile (FP_THREADS threads, items [c0, c0 + FP_ITEMS) per thread, look-back chain `state` under max): head[c]
// for every item, bit i of the result for item i.  keys(c, key_start, key_end): (tid + 1) << 32 | first start / last end of item c.
template <class Keys>
LRB_DEVINL uint32_t tile_locus_heads(uint64_t *state, int tile, int64_t c0, int64_t n, bool single_locus, uint8_t *head_out, Keys keys)
{
    __shared__ uint64_t s_w[FP_THREADS / 32], s_excl;
    const int lane = lane_id(), w = warp_id();
    uint64_t key_end[FP_ITEMS], key_start[FP_ITEMS], run = 0;
#pragma unroll
    for (int i = 0; i < FP_ITEMS; ++i) {
        key_end[i] = 0; key_start[i] = 0;
        if (c0 + i < n) keys(c0 + i, key_start[i], key_end[i]);
        run = key_end[i] > run ? key_end[i] : run;
    }
    // inclusive max over the block (one value per thread: the max of its items)
    uint64_t inc = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const uint64_t t = __shfl_up_sync(FULL, inc, o); if (lane >= o && t > inc) inc = t; }
    if (lane == 31) s_w[w] = inc;
    __syncthreads();
    uint64_t pre = 0, tot = 0;
    for (int k = 0; k < FP_THREADS / 32; ++k) { const uint64_t v = s_w[k]; if (k < w && v > pre) pre = v; if (v > tot) tot = v; }
    uint64_t left = __shfl_up_sync(FULL, inc, 1); if (lane == 0) left = 0;
    const uint64_t tpre = left > pre ? left : pre;                             // exclusive prefix max of this thread inside the tile
    if (w == 0) { const uint64_t e = lookback_exclusive(state, tile, tot, OpMax()); if (lane == 0) s_excl = e; }
    __syncthreads();
    uint64_t before = s_excl > tpre ? s_excl : tpre;
    uint32_t head = 0;
#pragma unroll
    for (int i = 0; i < FP_ITEMS; ++i) {
        if (c0 + i < n) {
            const bool h = (c0 + i == 0) || (!single_locus && key_start[i] > before);
            if (h) head |= 1u << i;
            head_out[c0 + i] = h ? 1 : 0;
            before = key_end[i] > before ? key_end[i] : before;
        }
    }
    return head;
}

__global__ void __launch_bounds__(FP_THREADS) fold_prepare_kernel(MergeArgs a)
{
    __shared__ uint32_t s_scan[33];
    __shared__ uint32_t s_tile; __shared__ uint64_t s_excl;
    if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile, lane = lane_id(), w = warp_id();
    const int64_t n_cand = cand_count(a);
    const int64_t c0 = ((int64_t)tile * FP_THREADS + threadIdx.x) * FP_ITEMS;
    // locus segmentation first (cheap loads, two look-back chains): the per-exon work below then overlaps the chains of later tiles
    if (!a.presegmented) {
        const uint32_t head = tile_locus_heads(a.tile_state, tile, c0, n_cand, a.single_locus, a.head, [&](int64_t c, uint64_t &ks, uint64_t &ke) {
            const uint32_t rw = a.list.row[c]; const int ni = (int)a.list.cnt[c];
            const uint32_t g = a.rows.ex_beg[rw] + a.list.lo[c];
            const uint64_t tk = (uint64_t)(uint32_t)(a.rows.tid[rw] + 1) << 32;
            ke = tk | (uint32_t)a.ex.ee[g + ni - 1];                               // real coordinates: locus segmentation
            ks = tk | (uint32_t)a.ex.es[g];
        });
        uint32_t htot; const uint32_t hex = block_excl_sum(__popc(head), s_scan, &htot);
        if (w == 0) { const uint64_t e = lookback_exclusive(a.tile_state + a.n_tiles, tile, (uint64_t)htot, OpAdd()); if (lane == 0) s_excl = e; }
        __syncthreads();
        uint32_t ho = (uint32_t)s_excl + hex;
#pragma unroll
        for (int i = 0; i < FP_ITEMS; ++i) if ((head >> i) & 1u) a.locus_start[ho++] = (uint32_t)(c0 + i);
        if (tile == a.n_tiles - 1 && threadIdx.x == 0) a.totals[0] = s_excl + htot;
    }
    // flatten the candidates: trans-level fields, chain hash, junction signature.  Striped over the tile (thread t takes the
    // candidates t, t + 256, ...): the exon ranges of neighbouring threads are adjacent in the pools, so the per-exon loads of a
    // warp fall into a few lines instead of one line per lane
    const int64_t t0 = (int64_t)tile * FP_THREADS * FP_ITEMS;
#pragma unroll 1
    for (int i = 0; i < FP_ITEMS; ++i) {
        const int64_t c = t0 + (int64_t)i * FP_THREADS + threadIdx.x;
        if (c >= n_cand) break;
        const uint32_t rw = a.list.row[c]; const int ni = (int)a.list.cnt[c];
        const uint32_t g = a.rows.ex_beg[rw] + a.list.lo[c];
        const int fsi = a.ex.es[g], lei = a.ex.ee[g + ni - 1], rt = a.rows.tid[rw];
        const bool pc = a.list.piece[c] >= 0;
        a.cd.tid[c] = pc ? 0 : rt; a.cd.start[c] = pc ? 0 : fsi; a.cd.end[c] = pc ? 0 : lei;
        int mono = 2;                               // bit 1: exon ends never decrease (always true for CIGAR chains)
        uint64_t h = 0x243F6A8885A308D3ull ^ (uint64_t)ni, sig = 0, j0 = 0;
        int prev_e = 0;
        for (int j = 0; j < ni - 1; ++j) {
            const int e_i = a.ex.ee[g + j];
            const uint32_t e = (uint32_t)e_i, s2 = (uint32_t)a.ex.es[g + j + 1];
            if (j > 0 && prev_e > e_i) mono = 0;
            prev_e = e_i;
            h = mixh(h, e); h = mixh(h, s2);
            const uint64_t jk = ((uint64_t)e << 32) | s2;
            if (j == 0) j0 = jk;
            sig |= junc_mask(jk);
        }
        a.cd.rev[c] = (pc ? 0 : a.rows.is_rev[rw]) | mono;
        a.cd.n[c] = ni; a.cd.gbeg[c] = g; a.cd.fs[c] = fsi; a.cd.le[c] = lei;
        a.cd.hash[c] = h; a.cd.j0[c] = j0; a.cd.sig[c] = sig;
    }
}
void launch_merge_prepare(MergeArgs a, cudaStream_t st)
{
    if (a.n_cand <= 0) { cudaMemsetAsync(a.totals, 0, 16, st); return; }
    a.n_tiles = (int)((a.n_cand + FP_THREADS * FP_ITEMS - 1) / (FP_THREADS * FP_ITEMS));
    cudaMemsetAsync(a.tile_state, 0, (size_t)a.n_tiles * 16, st); cudaMemsetAsync(a.ticket, 0, 4, st);
    fold_prepare_kernel<<<(unsigned)a.n_tiles, FP_THREADS, 0, st>>>(a); LRB_COUNT_LAUNCH();
}

// Class order for the class folds (update_gtf.c:501-528 folds each class's rows as a list of its own).  A candidate never sees another
// sub-stream's entries (fold_event), so grouping the rows of a locus by class, each group in row order, hands every sub-stream the same
// sequence, and its replay walks only its own range.  The loci are cut on all rows in row order (fold_prepare_kernel's rule), not
// on the permuted list: the cuts, and so every locus and its path, stay what they are.
//   class_order_kernel    per tile of rows: locus heads (look-back, max), then one look-back (sum) of the head count and the class
//                         counts (class 3 is what the others leave); per row its locus and its rank among the earlier rows of its
//                         class, per locus the class counts before its head (cbase)
//   class_scatter_kernel  per row: its candidate index (the locus's class ranges follow from two neighbours in cbase)
__global__ void __launch_bounds__(FP_THREADS) class_order_kernel(MergeArgs a, const uint8_t *__restrict__ row_kls, uint2 *loc_rank)
{
    __shared__ uint32_t s_scan[33];
    __shared__ uint32_t s_tile; __shared__ uint64_t s_excl[2];
    if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile, lane = lane_id(), w = warp_id();
    const int64_t n = a.n_cand;
    const int64_t c0 = ((int64_t)tile * FP_THREADS + threadIdx.x) * FP_ITEMS;
    const uint32_t head = tile_locus_heads(a.tile_state, tile, c0, n, a.single_locus, a.head, [&](int64_t r, uint64_t &ks, uint64_t &ke) {
        const uint32_t g = a.rows.ex_beg[r]; const int ni = (int)a.rows.ex_n[r];
        const uint64_t tk = (uint64_t)(uint32_t)(a.rows.tid[r] + 1) << 32;
        ke = tk | (uint32_t)a.ex.ee[g + ni - 1];
        ks = tk | (uint32_t)a.ex.es[g];
    });
    uint32_t k[FP_ITEMS], hk0 = __popc(head), k12 = 0;                         // 16-bit counters in pairs: a tile has 1024 rows
#pragma unroll
    for (int i = 0; i < FP_ITEMS; ++i) {
        k[i] = c0 + i < n ? row_kls[c0 + i] : 3u;
        hk0 += k[i] == 0 ? 1u << 16 : 0u; k12 += k[i] == 1 ? 1u : k[i] == 2 ? 1u << 16 : 0u;
    }
    uint32_t t_hk0, t_k12;
    const uint32_t e_hk0 = block_excl_sum(hk0, s_scan, &t_hk0), e_k12 = block_excl_sum(k12, s_scan, &t_k12);
    if (w == 0) {
        const uint64_t x = lookback_exclusive(a.tile_state + a.n_tiles, tile, pack_pair(t_hk0 & 0xFFFFu, t_hk0 >> 16), OpAdd());
        const uint64_t y = lookback_exclusive(a.tile_state + 2 * a.n_tiles, tile, pack_pair(t_k12 & 0xFFFFu, t_k12 >> 16), OpAdd());
        if (lane == 0) { s_excl[0] = x; s_excl[1] = y; }
    }
    __syncthreads();
    uint32_t loc = pair_hi(s_excl[0]) + (e_hk0 & 0xFFFFu);                    // loci that start before this thread's first row
    uint32_t r0 = pair_lo(s_excl[0]) + (e_hk0 >> 16), r1 = pair_hi(s_excl[1]) + (e_k12 & 0xFFFFu), r2 = pair_lo(s_excl[1]) + (e_k12 >> 16);
    uint32_t r3 = (uint32_t)c0 - r0 - r1 - r2;                                 // rows of each class before it
#pragma unroll
    for (int i = 0; i < FP_ITEMS; ++i) {
        if (c0 + i >= n) break;
        if ((head >> i) & 1u) { a.locus_start[loc] = (uint32_t)(c0 + i); a.cbase[loc] = make_uint4(r0, r1, r2, r3); ++loc; }
        const uint32_t rank = k[i] == 0 ? r0++ : k[i] == 1 ? r1++ : k[i] == 2 ? r2++ : r3++;
        loc_rank[c0 + i] = make_uint2(loc - 1, rank);
    }
    if (tile == a.n_tiles - 1 && threadIdx.x == 0) {
        const uint32_t n_loci = pair_hi(s_excl[0]) + (t_hk0 & 0xFFFFu);
        const uint32_t q0 = pair_lo(s_excl[0]) + (t_hk0 >> 16), q1 = pair_hi(s_excl[1]) + (t_k12 & 0xFFFFu), q2 = pair_lo(s_excl[1]) + (t_k12 >> 16);
        a.totals[0] = n_loci;
        a.cbase[n_loci] = make_uint4(q0, q1, q2, (uint32_t)n - q0 - q1 - q2);
    }
}
__global__ void __launch_bounds__(256) class_scatter_kernel(MergeArgs a, const uint8_t *__restrict__ row_kls, const uint2 *__restrict__ loc_rank,
                                                            uint32_t *perm, uint8_t *cand_kls)
{
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.n_cand) return;
    const int k = row_kls[r]; const uint2 lr = loc_rank[r];
    const uint4 b0 = a.cbase[lr.x];
    int64_t cs, ce; class_range(a, lr.x, a.locus_start[lr.x], k, cs, ce);
    const int64_t c = cs + lr.y - (k == 0 ? b0.x : k == 1 ? b0.y : k == 2 ? b0.z : b0.w);
    perm[c] = (uint32_t)r; cand_kls[c] = (uint8_t)k;
}
void launch_class_order(MergeArgs a, const uint8_t *row_kls, uint32_t *perm, uint8_t *cand_kls, cudaStream_t st)
{
    if (a.n_cand <= 0) return;
    a.n_tiles = (int)((a.n_cand + FP_THREADS * FP_ITEMS - 1) / (FP_THREADS * FP_ITEMS));
    uint2 *loc_rank = reinterpret_cast<uint2 *>(a.tlist);                      // tlist: n_cand * 8 bytes, not needed before the fold
    cudaMemsetAsync(a.tile_state, 0, (size_t)a.n_tiles * 24, st); cudaMemsetAsync(a.ticket, 0, 4, st);
    class_order_kernel<<<(unsigned)a.n_tiles, FP_THREADS, 0, st>>>(a, row_kls, loc_rank); LRB_COUNT_LAUNCH();
    class_scatter_kernel<<<(unsigned)((a.n_cand + 255) / 256), 256, 0, st>>>(a, row_kls, loc_rank, perm, cand_kls); LRB_COUNT_LAUNCH();
}

// check_iden (gtf.c:54-92) between candidate t and fold entry E (first start / last end may have been extended)
struct Entry { int n; uint32_t gbeg; int fs, le; uint64_t hash; int mono; uint64_t j0, sig; };
// candidate c as an entry of T, with its (possibly extended) first start fs and last end le
LRB_DEVINL Entry entry_of(const CandSoA &cd, int64_t c, int fs, int le) { return {cd.n[c], cd.gbeg[c], fs, le, cd.hash[c], cd.rev[c] & 2, cd.j0[c], cd.sig[c]}; }
LRB_DEVINL int x_s(const DExons &ex, const Entry &e, int i) { return i == 0 ? e.fs : ex.es[e.gbeg + i]; }
LRB_DEVINL int x_e(const DExons &ex, const Entry &e, int i) { return i == e.n - 1 ? e.le : ex.ee[e.gbeg + i]; }
// the partial match of gtf.c:76-91: does the chain s (fewer exons, at least two; s_j0 its first junction) continue the chain l from the
// first occurrence of its first junction on, every boundary within ss_dis?  l_mono: the exon ends of l never decrease
LRB_DEVINL bool chain_continues(const DExons &ex, uint32_t l_gbeg, int l_n, bool l_mono, uint64_t s_j0, uint32_t s_gbeg, int s_n, int ss_dis)
{
    const int s_e0 = (int)(uint32_t)(s_j0 >> 32), s_s1 = (int)(uint32_t)s_j0;
    int i = 0;
    const bool jump = ss_dis == 0 && l_mono;
    if (jump) {                                                  // exact matching on non-decreasing ends: jump to the first candidate
        int lo = 0, hi = l_n - 1;
        while (lo < hi) { int mid = (lo + hi) >> 1; if (ex.ee[l_gbeg + mid] < s_e0) lo = mid + 1; else hi = mid; }
        i = lo;
    }
    for (; i < l_n - 1; ++i) {
        const int le_i = ex.ee[l_gbeg + i];
        if (jump && le_i > s_e0) return false;
        if (iabs_dev(le_i - s_e0) <= ss_dis && iabs_dev(ex.es[l_gbeg + i + 1] - s_s1) <= ss_dis) {
            int j = 1;
            for (i = i + 1; i < l_n - 1 && j < s_n - 1; ++i, ++j) {
                if (iabs_dev(ex.ee[l_gbeg + i] - ex.ee[s_gbeg + j]) > ss_dis) return false;
                if (iabs_dev(ex.es[l_gbeg + i + 1] - ex.es[s_gbeg + j + 1]) > ss_dis) return false;
            }
            return true;
        }
    }
    return false;
}
LRB_DEVINL int chain_iden(const DExons &ex, const Entry &t1, const Entry &t2, int ss_dis, int end_dis)
{
    const Entry &l = t1.n >= t2.n ? t1 : t2, &s = t1.n >= t2.n ? t2 : t1;
    if (t1.n == t2.n) {
        if (ss_dis == 0 && t1.hash != t2.hash) return -1;        // some internal boundary differs
        if (iabs_dev(l.fs - s.fs) > end_dis) return -1;
        for (int i = 0; i < l.n - 1; ++i) {
            if (iabs_dev(x_e(ex, l, i) - x_e(ex, s, i)) > ss_dis) return -1;
            if (iabs_dev(x_s(ex, l, i + 1) - x_s(ex, s, i + 1)) > ss_dis) return -1;
        }
        if (iabs_dev(l.le - s.le) > end_dis) return -1;
        return 0;
    }
    if (iabs_dev(l.fs - s.fs) > end_dis) return -1;
    if (ss_dis == 0 && !sig_has(l.sig, s.j0)) return -1;   // the first junction of s is not a junction of l
    if (!chain_continues(ex, l.gbeg, l.n, l.mono, s.j0, s.gbeg, s.n, ss_dis)) return -1;
    if (iabs_dev(l.le - s.le) > end_dis) return -1;
    return 2;
}

// ---- one step of merge_trans's back-scan (update_gtf.c:145-160), shared by the replays of merge_fold_kernel and fold_big_kernel
enum { EV_NONE = 0, EV_STOP = 1, EV_MERGE = 2, EV_DROP = 3 };
// merge_trans2's single-exon test (update_gtf.c:122-140); its first two tests are check_iden's end tests
LRB_DEVINL bool ends_match(const MergeArgs &a, int t_fs, int t_le, int e_fs, int e_le)
{
    return iabs_dev(t_fs - e_fs) <= a.up.end_dis && iabs_dev(t_le - e_le) <= a.up.end_dis;
}
LRB_DEVINL bool single_exon_match(const MergeArgs &a, int t_fs, int t_le, int e_fs, int e_le)
{
    return ends_match(a, t_fs, t_le, e_fs, e_le) && ovlp_frac(t_fs, t_le, e_fs, e_le) >= a.up.single_exon_ovlp_frac;
}
// The event of entry e for candidate t: visible = e is of t's sub-stream, stop = the stop rule (:148), same_strand (:149, under -c).
// multi(): the relation of two multi-exon chains whose ends passed the end tests (0 identical, 2 partial, -1 none).
template <class Multi>
LRB_DEVINL int fold_event(const MergeArgs &a, bool visible, bool stop, bool same_strand, int t_n, int t_fs, int t_le, int e_n, int e_fs, int e_le, Multi multi)
{
    if (!visible) return EV_NONE;
    if (stop) return EV_STOP;
    if (a.up.force_strand && !same_strand) return EV_NONE;
    if (t_n == 1 && e_n == 1) return single_exon_match(a, t_fs, t_le, e_fs, e_le) ? EV_MERGE : EV_NONE;          // merge_trans2
    if (t_n > 1 && e_n > 1 && ends_match(a, t_fs, t_le, e_fs, e_le)) {                                           // merge_trans1 :98-119
        const int r = multi();
        return r == 0 ? EV_MERGE : r == 2 ? EV_DROP : EV_NONE;
    }
    return EV_NONE;
}
// A lane group tests G entries at once (lane l: the entry base - l).  The lowest lane with an event holds the entry nearest to the end
// of T and decides: -1 no event in this window, 0 the scan stops (t is appended), 1 t is absorbed (that lane has run absorb()) or dropped.
template <int G, class Absorb>
LRB_DEVINL int fold_winner(unsigned gm, int gl, int ev, Absorb absorb)
{
    const int sh = (lane_id() / G) * G;
    const unsigned m = (__ballot_sync(gm, ev != EV_NONE) >> sh) & lane_bits<G>();
    if (!m) return -1;
    const int win = __ffs(m) - 1;
    const int wev = __shfl_sync(gm, ev, sh + win);
    if (wev == EV_MERGE && gl == win) absorb();
    return wev == EV_STOP ? 0 : 1;
}
// merge_trans1 / merge_trans2 (update_gtf.c:104-111, 130-137): the entry counts t and takes t's first start / last end where they extend it
LRB_DEVINL void absorb_into(int &cov, int &fs, int &start, int &le, int &end, int t_fs, int t_le)
{
    cov += 1;
    if (t_fs < fs) { fs = t_fs; start = t_fs; }
    if (t_le > le) { le = t_le; end = t_le; }
}
// a candidate nothing of its locus absorbs is not appended when an entry of an earlier locus absorbs it (xl_* below); the writer lane
// records (forced = 3) that it happened in this fold
LRB_DEVINL bool absorbed_elsewhere(const MergeArgs &a, int64_t c, bool writer)
{
    if (!a.forced || !a.forced[c]) return false;
    if (writer) a.forced[c] = 3;
    return true;
}
// the internal boundaries of two chains of n exons are equal (on the pools: what a class key or chain hash only suggests)
LRB_DEVINL bool same_chain(const DExons &ex, uint32_t g1, uint32_t g2, int n)
{
    bool same = true;
    for (int i = 0; i < n - 1; ++i) same = same && ex.ee[g1 + i] == ex.ee[g2 + i] && ex.es[g1 + i + 1] == ex.es[g2 + i + 1];
    return same;
}

static constexpr int MF_THREADS = 128;
// G lanes per locus; tlist[ls + k] = candidate index of the k-th entry of the locus' T; mutable entry data lives at work[cand].
// Loci of [min_m, max_m] candidates, and those whose hand-off state is in hard_mask.  The whole-warp instance is held to 40 registers
// (12 blocks per SM): left free, the compiler takes more registers to avoid a few spills.
template <int G>
__global__ void __launch_bounds__(MF_THREADS, G == 32 ? 12 : 0) merge_fold_kernel(MergeArgs a, int min_m, int max_m, int hard_mask)
{
    const int64_t n_loci = (int64_t)a.totals[0];
    constexpr int GPB = MF_THREADS / G;
    const int gl = threadIdx.x % G;
    const unsigned gm = group_mask<G>();
    const CandSoA &cd = a.cd;
    for (int64_t loc = (int64_t)blockIdx.x * GPB + threadIdx.x / G; loc < n_loci; loc += (int64_t)gridDim.x * GPB) {
        int64_t ls, le; locus_range(a, n_loci, loc, ls, le);
        if ((le - ls < min_m || le - ls > max_m) && !(hard_mask && ((hard_mask >> a.hard[ls]) & 1))) continue;   // other loci: flat kernels / another group width
        int cnt = 0;
        for (int64_t c = ls; c < le; ++c) {
            const int t_tid = cd.tid[c], t_start = cd.start[c], t_rev = cd.rev[c] & 1;
            const Entry te = entry_of(cd, c, cd.fs[c], cd.le[c]);
            int result = 0;                                      // 0 append, 1 absorbed / dropped
            for (int base = cnt - 1; base >= 0; base -= G) {
                const int k = base - gl;
                int ev = EV_NONE;
                uint32_t ec = 0;
                if (k >= 0) {
                    ec = a.tlist[ls + k];
                    const int e_fs = a.work.fs[ec], e_le = a.work.le[ec];
                    ev = fold_event(a, !a.kls || a.kls[ec] == a.kls[c], t_tid > cd.tid[ec] || t_start > a.work.end[ec], t_rev == (cd.rev[ec] & 1),
                                    te.n, te.fs, te.le, cd.n[ec], e_fs, e_le, [&] { return chain_iden(a.ex, te, entry_of(cd, ec, e_fs, e_le), a.up.ss_dis, a.up.end_dis); });
                }
                const int w = fold_winner<G>(gm, gl, ev, [&] { absorb_into(a.work.cov[ec], a.work.fs[ec], a.work.start[ec], a.work.le[ec], a.work.end[ec], te.fs, te.le); });
                if (w >= 0) { result = w; break; }
            }
            __syncwarp(gm);
            if (result == 0 && absorbed_elsewhere(a, c, gl == 0)) result = 1;
            if (result == 0) {
                if (gl == 0) {
                    a.tlist[ls + cnt] = (uint32_t)c; a.alive[c] = 1;
                    a.work.cov[c] = 1; a.work.start[c] = t_start; a.work.end[c] = cd.end[c]; a.work.fs[c] = te.fs; a.work.le[c] = te.le;
                }
                ++cnt;
            } else if (gl == 0) a.alive[c] = 0;
            __syncwarp(gm);
        }
    }
}

static constexpr int FF_MAX = 64;                   // loci up to this many candidates; larger ones -> fold_big_kernel

// ------------------------------------------------------------------------------- big loci (ss_dis == 0): classes + warp replay
// Deep data (hundreds of reads per gene) puts most candidates into loci beyond the 64-candidate masks of the flat fold.  Replaying
// those through merge_fold_kernel costs a chain of dependent L2 / HBM loads per survivor visited (candidate fields, then both exon
// chains for every identity or partial-match test): ~2.4 us per candidate.  With exact splice-site matching the tests are STATIC:
//   fold_big_mark_kernel     warp per locus: members of loci beyond the masks (or left over by the flat kernels) learn their locus head;
//   fold_class_insert/verify thread per member: identity class = the first member of the locus with the same (chromosome, exon count,
//                            chain hash, strand if -c, sub-stream), through one lock-free table; verified ONCE on the exon pools
//                            (a 64-bit collision sends the locus to merge_fold_kernel);
//   fold_big_kernel          warp per locus, the ordered replay itself with the survivors in SHARED memory: identity is an integer
//                            compare of class ids, the partial-match relation between two classes (junction-signature pre-filter, then
//                            the pools) is decided once and kept in a direct-mapped per-warp cache, the stop rule reads the slots.
//                            32 survivors per step, 32 candidates loaded per batch, one per lane.
// A locus whose survivors outgrow the slots of both tiers (LP_MERGE_OVER) is redone by merge_fold_kernel -- exact either way.
static constexpr int FB_THREADS = 128, FB_MAXREL = 32768;
// G lanes per locus: lane l reads slot base - l (conflict free inside the group); two tiers -- 8 lanes / 64 slots for the common
// locus (a few dozen survivors: four loci per warp), a whole warp / 416 slots for what outgrows that
template <int SLOTS, int CACHE>
struct FbSlots {
    uint64_t j0[SLOTS], sig[SLOTS];
    int fs[SLOTS], le[SLOTS], end[SLOTS], start[SLOTS], tid[SLOTS], cov[SLOTS];
    uint32_t gbeg[SLOTS], cand[SLOTS], meta[SLOTS], rep[SLOTS];       // meta: n << 8 | mono bit 1 | rev bit 0
    uint32_t cache[CACHE];                          // partial-match relation of two classes: valid 31 | result 30 | relA 29:15 | relB 14:0
    uint32_t pad[8];                                // group stride = 8 banks mod 32: the four 8-lane groups of a warp read disjoint banks
};
struct ClassTab { unsigned long long *key; uint32_t *minidx; uint64_t cap; };

__global__ void __launch_bounds__(256) fold_big_mark_kernel(MergeArgs a)
{
    const int64_t n_loci = (int64_t)a.totals[0];
    const int lane = lane_id();
    for (int64_t loc = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / 32; loc < n_loci; loc += (int64_t)gridDim.x * blockDim.x / 32) {
        int64_t ls, le; locus_range(a, n_loci, loc, ls, le);
        if (le - ls <= FF_MAX && a.hard[ls] == LP_FLAT) continue;
        // the later passes walk this list, not all loci; an entry is (locus, sub-stream): the four class folds of the summary run over
        // their own ranges of the locus (class order) and never see each other's entries, so each gets its own replay, and a sub-stream
        // without rows in the locus gets none (nor class rows: zero classes)
        if (lane < (a.kls ? 4 : 1)) {
            int64_t cs = ls, ce = le;
            if (a.kls) class_range(a, loc, ls, lane, cs, ce);
            if (ce == cs) ((uint8_t *)&a.locus_cnt[loc])[lane] = 0;
            else {
                const uint32_t i = atomicAdd(&a.fb_cnt[0], 1u);
                if (i < (uint32_t)a.n_cand) a.fb_list[i] = ((uint32_t)loc << 2) | (uint32_t)lane; else a.hard[ls] = LP_MERGE_OVER;    // (cannot happen for loci beyond the masks)
            }
        }
        for (int64_t c = ls + lane; c < le; c += 32) { a.desc[c] = DESC_BIG; a.lstart[c] = (uint32_t)ls; }
    }
}
LRB_DEVINL uint64_t class_key(const MergeArgs &a, int64_t c, uint32_t ls)
{
    const CandSoA &cd = a.cd;
    uint64_t k = mixh(cd.hash[c], (uint32_t)cd.n[c] | ((a.kls ? (uint32_t)a.kls[c] : 0u) << 16) | ((a.up.force_strand ? (uint32_t)(cd.rev[c] & 1) : 0u) << 20));
    k = mixh(k, ls);                                // classes are per locus (check_iden itself never looks at the chromosome)
    return k == ~0ull ? 0x1234567ull : k;
}
LRB_DEVINL uint64_t class_slot(const ClassTab &t, uint64_t k) { return __umul64hi(k * 0x9E3779B97F4A7C15ull, t.cap); }
__global__ void __launch_bounds__(256) fold_class_insert_kernel(MergeArgs a, ClassTab t)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cand_count(a) || a.desc[c] != DESC_BIG || a.cd.n[c] < 2) return;
    const uint64_t k = class_key(a, c, a.lstart[c]);
    uint64_t s = class_slot(t, k);
    for (;;) {
        const unsigned long long p = atomicCAS(&t.key[s], ~0ull, (unsigned long long)k);
        if (p == ~0ull || p == k) { atomicMin(&t.minidx[s], (uint32_t)c); return; }
        s = s + 1 == t.cap ? 0 : s + 1;
    }
}
__global__ void __launch_bounds__(256) fold_class_verify_kernel(MergeArgs a, ClassTab t)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cand_count(a) || a.desc[c] != DESC_BIG) return;
    const CandSoA &cd = a.cd;
    const int nc = cd.n[c];
    if (nc < 2) { a.rep[c] = (uint32_t)c; return; }
    const uint32_t ls = a.lstart[c];
    const uint64_t k = class_key(a, c, ls);
    uint64_t s = class_slot(t, k);
    while (t.key[s] != k) s = s + 1 == t.cap ? 0 : s + 1;
    const uint32_t r = t.minidx[s];
    a.rep[c] = r;
    if (r == (uint32_t)c) return;
    bool same = r >= ls && cd.n[r] == nc;           // same key in another locus (only an unsorted concatenation can do that) or a collision
    if (same) {
        same = same_chain(a.ex, cd.gbeg[c], cd.gbeg[r], nc);
        if (a.up.force_strand) same = same && ((cd.rev[c] ^ cd.rev[r]) & 1) == 0;
        if (a.kls) same = same && a.kls[c] == a.kls[r];
    }
    if (!same) a.hard[ls] = LP_MERGE_VERIFY;        // merge_fold_kernel replays this locus on the pools
}

// Warp per big locus: the multi-exon classes of the locus get dense ordinals in order of first occurrence (single-exon candidates share
// the pseudo class FB_SINGLE: their relation is dynamic, decided on the slots), and the STATIC relation between every two classes of
// the locus (identity on the diagonal, partial match elsewhere: gtf.c:76-91 on the chains of the two representatives) becomes a
// 128-bit row per class.  The replay then needs no exon pool at all: "can this survivor absorb the candidate" is one bit test.
// Loci with more than FB_MAXCLS classes keep locus_cnt = CLASSES_UNTABULATED and the replay falls back to its relation cache.
static constexpr int FB_MAXCLS = 127; static constexpr uint32_t FB_SINGLE = 127u;
__global__ void __launch_bounds__(256) fold_class_rows_kernel(MergeArgs a, uint32_t *next_entry)
{
    // per warp: the classes of the locus (exon count, sub-stream, junction signature, first junction, representative)
    __shared__ uint64_t s_sig[8][128], s_j0[8][128]; __shared__ uint32_t s_rep[8][128]; __shared__ uint32_t s_nk[8][128];
    const int64_t n_loci = (int64_t)a.totals[0], n_big = min((int64_t)a.fb_cnt[0], a.n_cand);
    const int lane = lane_id(), w = warp_id();
    const CandSoA &cd = a.cd;
    for (;;) {
        uint32_t bi = 0;
        if (lane == 0) bi = atomicAdd(next_entry, 1u);               // entries differ by orders of magnitude in size: claimed one at a time
        bi = __shfl_sync(FULL, bi, 0);
        if ((int64_t)bi >= n_big) return;
        const int64_t loc = a.fb_list[bi] >> 2; const int my = (int)(a.fb_list[bi] & 3u);
        int64_t ls, le, cs, ce; replay_range(a, n_loci, loc, my, ls, le, cs, ce);
        if (for_merge_fold(a.hard[ls])) continue;
        int K = 0;
        for (int64_t c0 = cs; c0 < ce; c0 += 32) {
            const int64_t c = c0 + lane;
            const bool headc = c < ce && cd.n[c] > 1 && a.rep[c] == (uint32_t)c;
            const unsigned b = __ballot_sync(FULL, headc);
            if (headc) {
                const int o = K + __popc(b & ((1u << lane) - 1u));
                if (o < FB_MAXCLS) {                 // rows live at the representative's own index: a class of the locus, whatever its sub-stream
                    a.cord[c] = (uint8_t)o; a.crow[2 * c] = o < 64 ? 1ull << o : 0; a.crow[2 * c + 1] = o >= 64 ? 1ull << (o - 64) : 0;
                    s_sig[w][o] = cd.sig[c]; s_j0[w][o] = cd.j0[c]; s_rep[w][o] = (uint32_t)c; s_nk[w][o] = (uint32_t)cd.n[c];
                }
            }
            K += __popc(b);
        }
        if (lane == 0) ((uint8_t *)&a.locus_cnt[loc])[my] = K <= FB_MAXCLS ? (uint8_t)K : CLASSES_UNTABULATED;
        if (K > FB_MAXCLS) continue;
        __syncwarp();
        for (int64_t c = cs + lane; c < ce; c += 32) {
            if (cd.n[c] < 2) a.cord[c] = (uint8_t)FB_SINGLE;
            else if (a.rep[c] != (uint32_t)c) a.cord[c] = a.cord[a.rep[c]];
        }
        for (int p = lane; p < K * K; p += 32) {
            const int i = p / K, j = p - i * K;
            if (i >= j) continue;
            const int nA = (int)s_nk[w][i], nB = (int)s_nk[w][j];
            if (nA == nB) continue;                                  // equal exon counts: identical or unrelated, never partial
            const int L = nA > nB ? i : j, Sh = nA > nB ? j : i;
            const uint64_t sj0 = s_j0[w][Sh];
            if (!sig_has(s_sig[w][L], sj0)) continue;
            const uint32_t cl = s_rep[w][L], cs = s_rep[w][Sh];
            // under -c a survivor of the other strand never absorbs (fold_event): the rows leave such pairs out, so that the class
            // index of fold_big_kernel sees only same-strand classes (the back-scan tests the strand first and reads no row for them)
            if (a.up.force_strand && ((cd.rev[cl] ^ cd.rev[cs]) & 1)) continue;
            if (!chain_continues(a.ex, cd.gbeg[cl], cd.n[cl], (cd.rev[cl] & 2) != 0, sj0, cd.gbeg[cs], cd.n[cs], 0)) continue;
            atomicOr((unsigned long long *)&a.crow[2 * (size_t)s_rep[w][i] + (j >> 6)], 1ull << (j & 63));
            atomicOr((unsigned long long *)&a.crow[2 * (size_t)s_rep[w][j] + (i >> 6)], 1ull << (i & 63));
        }
        __syncwarp();
    }
}

// The class index of a replay: with tabulated rows and no end tests (end_dis = INT_MAX: check_iden's end tests always pass) the
// event of a slot for a multi-exon candidate t does not depend on the slot's position: STOP where t_tid > tid or t_start > end,
// else MERGE / DROP where the slot's class is in t's row (same class / partial match), else NONE.  The back-scan takes the newest
// slot with an event, so its winner is max(F, A): F the newest stopping slot, A the newest slot of a class in t's row.  A comes from
// last[o], the newest slot of class o (lane l keeps l, l + 32, l + 64, l + 96); F needs only be looked for at or above A, and only
// in 32-slot chunks whose lower bounds of tid and end allow a stop (lane j keeps chunk j's; tid is fixed and end only grows, so a
// bound stays a lower bound).  A split piece (tid = start = 0) never stops.
struct FbIndex {
    int last[4] = {-1, -1, -1, -1};
    int lo_tid = INT_MAX, lo_end = INT_MAX;
};
// -1: no slot stops or absorbs at or above A (t is appended), else 0 (a slot stops the scan: t is appended) or 1 (absorbed / dropped)
template <int SLOTS, int CACHE>
LRB_DEVINL int fold_index_decide(FbSlots<SLOTS, CACHE> &S, FbIndex &ix, int cnt, int lane, int t_tid, int t_start, int t_fs, int t_le,
                                 uint32_t t_ord, uint64_t t_row0, uint64_t t_row1)
{
    int A = -1;
    if ((t_row0 >> lane) & 1ull) A = max(A, ix.last[0]);
    if ((t_row0 >> (lane + 32)) & 1ull) A = max(A, ix.last[1]);
    if ((t_row1 >> lane) & 1ull) A = max(A, ix.last[2]);
    if ((t_row1 >> (lane + 32)) & 1ull) A = max(A, ix.last[3]);
    A = __reduce_max_sync(FULL, A);
    unsigned maybe = __ballot_sync(FULL, lane * 32 + 31 >= A && (t_tid > ix.lo_tid || t_start > ix.lo_end));
    while (maybe) {
        const int j = 31 - __clz(maybe);                         // newest chunk first
        maybe &= ~(1u << j);
        const int k = j * 32 + lane;
        const bool live = k < cnt;
        if (__any_sync(FULL, live && k >= A && (t_tid > S.tid[k] || t_start > S.end[k]))) return 0;
        const int e = __reduce_min_sync(FULL, live ? S.end[k] : INT_MAX);     // no stop there: the bound becomes exact again
        if (lane == j) ix.lo_end = e;
    }
    if (A < 0) return -1;
    if (lane == 0 && (S.cand[A] >> 16) == t_ord) absorb_into(S.cov[A], S.fs[A], S.start[A], S.le[A], S.end[A], t_fs, t_le);
    return 1;
}
// slot `slot` takes a candidate of class ord (FB_SINGLE: none)
LRB_DEVINL void fold_index_append(FbIndex &ix, int lane, int slot, uint32_t ord, int tid, int end)
{
    if (ord != FB_SINGLE && lane == (int)(ord & 31u)) {
        const int s = (int)(ord >> 5);
        ix.last[0] = s == 0 ? slot : ix.last[0]; ix.last[1] = s == 1 ? slot : ix.last[1];
        ix.last[2] = s == 2 ? slot : ix.last[2]; ix.last[3] = s == 3 ? slot : ix.last[3];
    }
    if (lane == (slot >> 5)) { ix.lo_tid = min(ix.lo_tid, tid); ix.lo_end = min(ix.lo_end, end); }
}

// Tier 0's replay when its slots ran out, kept for tier 1 to go on from: the slots, each lane's class index (slot numbers and chunk
// bounds mean the same with tier 1's slots), the candidate that found the slots full (tier 1 decides it again: a candidate to be
// appended changed nothing) and the count of indexed decisions so far.  The relation cache is not kept: it only remembers relations
// tier 1 can work out again.  One per entry of tier 1's list, at the entry's index.
static constexpr int FB_SLOTS0 = 128;
struct FbSaved {
    uint64_t j0[FB_SLOTS0], sig[FB_SLOTS0];
    int fs[FB_SLOTS0], le[FB_SLOTS0], end[FB_SLOTS0], start[FB_SLOTS0], tid[FB_SLOTS0], cov[FB_SLOTS0];
    uint32_t gbeg[FB_SLOTS0], cand[FB_SLOTS0], meta[FB_SLOTS0], rep[FB_SLOTS0];
    FbIndex ix[32];
    int64_t next; uint32_t n_indexed;
};
// a tier-1 entry holds more than FB_SLOTS0 candidates of its own (a range no other entry shares)
size_t fold_resume_bytes(int64_t n_cand) { return (size_t)(n_cand / (FB_SLOTS0 + 1) + 1) * sizeof(FbSaved); }
template <int SLOTS, int CACHE>
LRB_DEVINL void fb_save(FbSaved &d, const FbSlots<SLOTS, CACHE> &S, const FbIndex &ix, int lane, int64_t next, uint32_t n_indexed)
{
    static_assert(SLOTS == FB_SLOTS0, "tier 0 saves");
    for (int k = lane; k < FB_SLOTS0; k += 32) {
        d.j0[k] = S.j0[k]; d.sig[k] = S.sig[k]; d.fs[k] = S.fs[k]; d.le[k] = S.le[k]; d.end[k] = S.end[k]; d.start[k] = S.start[k];
        d.tid[k] = S.tid[k]; d.cov[k] = S.cov[k]; d.gbeg[k] = S.gbeg[k]; d.cand[k] = S.cand[k]; d.meta[k] = S.meta[k]; d.rep[k] = S.rep[k];
    }
    d.ix[lane] = ix;
    if (lane == 0) { d.next = next; d.n_indexed = n_indexed; }
}
template <int SLOTS, int CACHE>
LRB_DEVINL void fb_load(FbSlots<SLOTS, CACHE> &S, FbIndex &ix, const FbSaved &d, int lane)
{
    static_assert(SLOTS >= FB_SLOTS0, "tier 1 resumes");
    for (int k = lane; k < FB_SLOTS0; k += 32) {
        S.j0[k] = d.j0[k]; S.sig[k] = d.sig[k]; S.fs[k] = d.fs[k]; S.le[k] = d.le[k]; S.end[k] = d.end[k]; S.start[k] = d.start[k];
        S.tid[k] = d.tid[k]; S.cov[k] = d.cov[k]; S.gbeg[k] = d.gbeg[k]; S.cand[k] = d.cand[k]; S.meta[k] = d.meta[k]; S.rep[k] = d.rep[k];
    }
    ix = d.ix[lane];
}

// tier 0: loci beyond the masks or left over by the flat kernels (LP_TIER0); overflow -> LP_TIER1, which goes on from where tier 0
// stopped.  tier 1: overflow -> LP_MERGE_OVER.
// Tier 0 runs 6 blocks per SM (its slots take 222 KB of shared memory): at most 80 registers.
template <int G, int SLOTS, int CACHE, int TIER>
__global__ void __launch_bounds__(FB_THREADS, TIER == 0 ? 6 : 1) fold_big_kernel(MergeArgs a, uint32_t *next_locus)
{
    static_assert(G == 32 && SLOTS <= 32 * 32, "the class index takes a whole warp, one chunk of 32 slots per lane");
    extern __shared__ __align__(16) unsigned char fb_smem[];
    FbSlots<SLOTS, CACHE> &S = reinterpret_cast<FbSlots<SLOTS, CACHE> *>(fb_smem)[threadIdx.x / G];
    const int64_t n_loci = (int64_t)a.totals[0];
    const int lane = threadIdx.x % G;
    const unsigned gm = group_mask<G>();
    const CandSoA &cd = a.cd;
    for (;;) {
        // loci are claimed one at a time (their sizes differ by orders of magnitude)
        // tier 0 walks the list of big loci (fold_big_mark_kernel), tier 1 the list of those whose survivors outgrew tier 0's slots
        const uint32_t *list = TIER == 0 ? a.fb_list : a.fb_list + a.n_cand;
        const uint32_t n_list = min(a.fb_cnt[TIER == 0 ? 0 : 2], (uint32_t)a.n_cand);
        uint32_t li = 0;
        if (lane == 0) li = atomicAdd(next_locus, 1u);
        li = __shfl_sync(gm, li, 0, G);
        if (li >= n_list) return;
        const int64_t loc = (int64_t)(list[li] >> 2); const int my = (int)(list[li] & 3u);      // (locus, sub-stream)
        int64_t ls, le, cs, ce; replay_range(a, n_loci, loc, my, ls, le, cs, ce);
        const int hd = a.hard[ls];
        if (TIER == 0 ? for_merge_fold(hd) : hd != LP_TIER1) continue;
        if (le - ls >= FB_MAXREL) { if (lane == 0) a.hard[ls] = LP_MERGE_OVER; continue; }
        const bool use_rows = ((const uint8_t *)&a.locus_cnt[loc])[my] != CLASSES_UNTABULATED;      // the static relation of the sub-stream's classes is tabulated
        if (!use_rows) for (int i = lane; i < CACHE; i += G) S.cache[i] = 0;
        // multi-exon candidates are decided by the class index; single-exon ones (their overlap test reads the moving first start /
        // last end), untabulated classes and finite end_dis keep the back-scan, the only exact path for them
        const bool indexed = use_rows && a.up.end_dis == INT_MAX;
        FbIndex ix; uint32_t n_indexed = 0;
        int cnt = 0; bool overflow = false;
        int64_t from = cs, next = 0;                                 // next: the candidate that found the slots full
        if constexpr (TIER == 1) {
            const FbSaved &d = reinterpret_cast<const FbSaved *>(a.fb_state)[li];
            fb_load(S, ix, d, lane); cnt = FB_SLOTS0; from = d.next; n_indexed = d.n_indexed;
        }
        __syncwarp(gm);
        for (int64_t c0 = from; c0 < ce && !overflow; c0 += G) {
            // 32 candidates, one per lane
            const int64_t cl = c0 + lane; const bool have = cl < ce;
            const int l_tid = have ? cd.tid[cl] : 0, l_start = have ? cd.start[cl] : 0, l_end = have ? cd.end[cl] : 0, l_rv = have ? cd.rev[cl] : 0;
            const int l_n = have ? cd.n[cl] : 0, l_fs = have ? cd.fs[cl] : 0, l_le = have ? cd.le[cl] : 0; const uint32_t l_gbeg = have ? cd.gbeg[cl] : 0;
            const uint64_t l_j0 = have ? cd.j0[cl] : 0, l_sig = have ? cd.sig[cl] : 0;
            const uint32_t l_rep = have ? a.rep[cl] : 0;
            const uint32_t l_ord = (have && use_rows) ? a.cord[cl] : FB_SINGLE;
            const uint64_t l_row0 = l_ord != FB_SINGLE ? a.crow[2 * (size_t)l_rep] : 0, l_row1 = l_ord != FB_SINGLE ? a.crow[2 * (size_t)l_rep + 1] : 0;
            int l_alive = 0;
            const int nb = (int)min((int64_t)G, ce - c0);
            for (int q = 0; q < nb; ++q) {
                const int t_tid = __shfl_sync(gm, l_tid, q, G), t_start = __shfl_sync(gm, l_start, q, G), t_end = __shfl_sync(gm, l_end, q, G), t_rv = __shfl_sync(gm, l_rv, q, G);
                const int t_n = __shfl_sync(gm, l_n, q, G), t_fs = __shfl_sync(gm, l_fs, q, G), t_le = __shfl_sync(gm, l_le, q, G);
                const uint32_t t_gbeg = __shfl_sync(gm, l_gbeg, q, G), t_rep = __shfl_sync(gm, l_rep, q, G);
                const uint64_t t_j0 = __shfl_sync(gm, l_j0, q, G), t_sig = __shfl_sync(gm, l_sig, q, G);
                const uint64_t t_row0 = __shfl_sync(gm, l_row0, q, G), t_row1 = __shfl_sync(gm, l_row1, q, G);
                const uint32_t t_ord = __shfl_sync(gm, l_ord, q, G);
                const uint32_t t_rel = t_rep - (uint32_t)ls;
                int result = 0;                                      // 0 append, 1 absorbed / dropped
                if (indexed && t_ord != FB_SINGLE) {
                    result = fold_index_decide(S, ix, cnt, lane, t_tid, t_start, t_fs, t_le, t_ord, t_row0, t_row1) > 0;
                    ++n_indexed;
                } else for (int base = cnt - 1; base >= 0; base -= G) {
                    const int k = base - lane;
                    int ev = EV_NONE;
                    if (k >= 0) {
                        const uint32_t mt = S.meta[k];
                        const int e_n = (int)(mt >> 8);
                        // the static relation of two multi-exon classes: the class rows, else the identity of the representatives or the
                        // partial match (the shorter chain's first junction must be a junction of the longer, then the cached relation)
                        ev = fold_event(a, true, t_tid > S.tid[k] || t_start > S.end[k], (t_rv & 1) == (int)(mt & 1u),
                                        t_n, t_fs, t_le, e_n, S.fs[k], S.le[k], [&] {
                            if (use_rows) {
                                const uint32_t e_ord = S.cand[k] >> 16;
                                if (!((((e_ord & 64u) ? t_row1 : t_row0) >> (e_ord & 63u)) & 1ull)) return -1;
                                return e_ord == t_ord ? 0 : 2;
                            }
                            if (t_n == e_n) return S.rep[k] == t_rep ? 0 : -1;
                            const bool t_long = t_n > e_n;
                            const uint64_t lsig = t_long ? t_sig : S.sig[k], sj0 = t_long ? S.j0[k] : t_j0;
                            if (!sig_has(lsig, sj0)) return -1;
                            const uint32_t e_rel = S.rep[k] - (uint32_t)ls;
                            const uint32_t pair = (t_rel << 15) | e_rel;
                            const uint32_t ci = ((t_rel * 0x9E37u) ^ (e_rel * 0x85EBu) ^ (e_rel >> 5)) & (CACHE - 1);
                            const uint32_t ce = S.cache[ci];
                            bool rel;
                            if ((ce >> 31) && (ce & 0x3FFFFFFFu) == pair) rel = (ce >> 30) & 1u;
                            else {
                                rel = t_long ? chain_continues(a.ex, t_gbeg, t_n, (t_rv & 2) != 0, sj0, S.gbeg[k], e_n, 0)
                                             : chain_continues(a.ex, S.gbeg[k], e_n, (mt & 2u) != 0, sj0, t_gbeg, t_n, 0);
                                S.cache[ci] = 0x80000000u | (rel ? 0x40000000u : 0u) | pair;
                            }
                            return rel ? 2 : -1;
                        });
                    }
                    const int w = fold_winner<G>(gm, lane, ev, [&] { absorb_into(S.cov[k], S.fs[k], S.start[k], S.le[k], S.end[k], t_fs, t_le); });
                    if (w >= 0) { result = w; break; }
                }
                __syncwarp(gm);
                if (result == 0 && absorbed_elsewhere(a, c0 + q, lane == 0)) result = 1;
                if (result == 0) {
                    if (cnt == SLOTS) { overflow = true; next = c0 + q; n_indexed -= indexed && t_ord != FB_SINGLE; break; }
                    if (lane == 0) {
                        S.j0[cnt] = t_j0; S.sig[cnt] = t_sig; S.fs[cnt] = t_fs; S.le[cnt] = t_le; S.end[cnt] = t_end; S.start[cnt] = t_start;
                        S.tid[cnt] = t_tid; S.cov[cnt] = 1; S.gbeg[cnt] = t_gbeg; S.cand[cnt] = (uint32_t)(c0 + q - ls) | (t_ord << 16); S.rep[cnt] = t_rep;
                        S.meta[cnt] = ((uint32_t)t_n << 8) | (uint32_t)(t_rv & 3);
                    }
                    fold_index_append(ix, lane, cnt, t_ord, t_tid, t_end);
                    ++cnt;
                    if (lane == q) l_alive = 1;
                }
                __syncwarp(gm);
            }
            if (have && (!overflow || cl < next)) a.alive[cl] = (uint8_t)l_alive;
        }
        if (overflow) {                                              // tier 1 goes on from here; merge_fold_kernel redoes the locus from scratch
            if constexpr (TIER == 0) {
                uint32_t i = 0;
                if (lane == 0) i = atomicAdd(&a.fb_cnt[2], 1u);
                i = __shfl_sync(gm, i, 0, G);
                fb_save(reinterpret_cast<FbSaved *>(a.fb_state)[i], S, ix, lane, next, n_indexed);
                if (lane == 0) { a.hard[ls] = LP_TIER1; a.fb_list[a.n_cand + i] = list[li]; }
            } else if (lane == 0) a.hard[ls] = LP_MERGE_OVER;
            __syncwarp(gm);
            continue;
        }
        if (a.n_indexed && lane == 0 && n_indexed) atomicAdd(a.n_indexed, n_indexed);
        for (int k = lane; k < cnt; k += G) {
            const int64_t c = ls + (S.cand[k] & 0xFFFFu);
            a.work.cov[c] = S.cov[k]; a.work.start[c] = S.start[k]; a.work.end[c] = S.end[k]; a.work.fs[c] = S.fs[k]; a.work.le[c] = S.le[k];
        }
        __syncwarp(gm);
    }
}

// ------------------------------------------------------------------------------------------ flat fold (ss_dis == 0)
// With exact splice-site matching the relation between two multi-exon chains is STATIC (internal boundaries only; the
// mutable first start / last end enter through the end_dis tests alone), identity is transitive, and the partial-match
// relation is a relation between identity classes.  That moves every exon-pool access out of the ordered part:
//   fold_rep_kernel   thread per candidate: its identity class = first earlier candidate of the locus with the same
//                     (exon count, chain hash[, strand]), verified once on the pools (a hash collision hands the locus
//                     to the big-locus path, LP_TIER0);
//   fold_rel_kernel   thread per candidate: bit mask (over the <= 64 earlier candidates of its locus) of the entries that
//                     could absorb it -- same class, a class in partial-match relation (junction-signature pre-filter,
//                     verified on the pools, decided once per class representative), other single-exon reads;
//   fold_seq_kernel   thread per locus: the ordered fold itself on that mask and an alive mask held in registers: walk
//                     the alive entries from the newest, stop on the reference's stop rule (dynamic end), take the first
//                     confirmed event.  A warp folds 32 loci in lock step.

__global__ void __launch_bounds__(256) fold_rep_kernel(MergeArgs a)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cand_count(a)) return;
    const CandSoA &cd = a.cd;
    const bool force = a.up.force_strand != 0;
    const int nc = cd.n[c], rvc = cd.rev[c] & 1;
    const uint64_t hc = cd.hash[c];
    const uint8_t kc = a.kls ? a.kls[c] : 0;
    int64_t e = c, r = c;
    int steps = 0;
    while (!a.head[e]) {
        if (++steps >= FF_MAX) { a.lstart[c] = LSTART_DEEP; a.rep[c] = (uint32_t)c; a.desc[c] = 0; return; }   // deeper than the masks reach
        --e;
        if (nc > 1 && cd.n[e] == nc && cd.hash[e] == hc && (!force || (cd.rev[e] & 1) == rvc) && (!a.kls || a.kls[e] == kc)) r = e;
    }
    if (r != c && !same_chain(a.ex, cd.gbeg[c], cd.gbeg[r], nc)) a.hard[e] = LP_TIER0;     // a hash collision: not for the flat kernels
    a.rep[c] = (uint32_t)r; a.lstart[c] = (uint32_t)e;
    // class descriptor for the relation passes: [0:5] representative (locus-local), [6] single exon, [7] strand, [8:9] sub-stream
    a.desc[c] = (uint16_t)((uint32_t)(r - e) | (nc == 1 ? 64u : 0u) | ((uint32_t)rvc << 7) | ((uint32_t)kc << 8));
    a.relsym[c] = 0;
}

// partial-match relation between the class representatives of a locus (threads of non-representatives leave at once):
// relsym[r] gets a bit for every representative r' (earlier or later) whose class can absorb / be absorbed by r's
__global__ void __launch_bounds__(256) fold_relrep_kernel(MergeArgs a)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cand_count(a)) return;
    const uint32_t ls = a.lstart[c];
    if (ls == LSTART_DEEP) return;
    const uint32_t d = a.desc[c];
    if ((d & 64u) || (d & 63u) != (uint32_t)c - ls) return;          // single exon, or not the representative of its class
    const CandSoA &cd = a.cd;
    const bool force = a.up.force_strand != 0;
    const int nc = cd.n[c];
    const uint64_t sig_c = cd.sig[c], j0_c = cd.j0[c];
    const uint32_t gb_c = cd.gbeg[c];
    const bool mono_c = (cd.rev[c] & 2) != 0;
    for (uint32_t e = ls; e < (uint32_t)c; ++e) {
        const uint32_t de = a.desc[e];
        if ((de & 64u) || (de & 63u) != e - ls || ((de ^ d) & 0x300u)) continue;             // single / not a representative / other sub-stream
        if (force && ((de ^ d) & 128u)) continue;
        const int ne = cd.n[e];
        if (ne == nc) continue;
        bool hit;
        if (nc > ne) {
            const uint64_t j0_e = cd.j0[e];
            hit = sig_has(sig_c, j0_e) && chain_continues(a.ex, gb_c, nc, mono_c, j0_e, cd.gbeg[e], ne, 0);
        } else
            hit = sig_has(cd.sig[e], j0_c) && chain_continues(a.ex, cd.gbeg[e], ne, (cd.rev[e] & 2) != 0, j0_c, gb_c, nc, 0);
        if (hit) {
            atomicOr((unsigned long long *)&a.relsym[c], 1ull << (e - ls));
            atomicOr((unsigned long long *)&a.relsym[e], 1ull << ((uint32_t)c - ls));
        }
    }
}

// per candidate: the mask (over the <= 63 earlier candidates of its locus) of the entries that could absorb it -- members of its
// own class (identical chains), members of classes in partial-match relation, other single-exon reads -- and, for class
// folds, the mask of the earlier candidates of its own sub-stream
__global__ void __launch_bounds__(256) fold_relasm_kernel(MergeArgs a)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cand_count(a)) return;
    const uint32_t ls = a.lstart[c];
    if (ls == LSTART_DEEP) return;
    const uint32_t d = a.desc[c];
    const bool force = a.up.force_strand != 0;
    uint64_t mask = 0, same = 0;
    if (d & 64u) {
        for (uint32_t e = ls; e < (uint32_t)c; ++e) {
            const uint32_t de = a.desc[e];
            const uint64_t bit = 1ull << (e - ls);
            if (!((de ^ d) & 0x300u)) { same |= bit; if ((de & 64u) && !(force && ((de ^ d) & 128u))) mask |= bit; }
        }
    } else {
        const uint32_t r = d & 63u;
        const uint64_t rel = a.relsym[ls + r] | (1ull << r);          // classes in partial-match relation, and its own
        for (uint32_t e = ls; e < (uint32_t)c; ++e) {
            const uint32_t de = a.desc[e];
            const uint64_t bit = 1ull << (e - ls);
            if (!((de ^ d) & 0x300u)) same |= bit;
            if (!(de & 64u) && ((rel >> (de & 63u)) & 1ull)) mask |= bit;
        }
    }
    a.evmask[c] = mask;
    if (a.kls) a.samemask[c] = same;
}

// thread per locus.  The entries of T (the survivors so far) live in shared-memory slots in insertion order -- the back-scan
// of merge_trans is a walk down the slots; a locus with more than FS_SLOTS survivors is handed to fold_big_kernel.
// A slot keeps exon[0].start / exon[last].end; T.start / T.end equal them except for a split piece that was not extended
// yet (0 / 0, SURVEY Q14) -- two flag bits.
// T.tid of an entry is not stored: the candidates of a locus carry one non-zero tid (checked; a locus mixing chromosomes -- unsorted
// input -- goes to fold_big_kernel), so "t.tid > T.tid" (update_gtf.c:148) can only hold for an entry with tid 0 (a split piece,
// flag bit 4) under a candidate with tid > 0.
static constexpr int FS_THREADS = 64;
template <int FS_SLOTS>
__global__ void __launch_bounds__(FS_THREADS) fold_seq_kernel(MergeArgs a)
{
    __shared__ int s_fs[FS_SLOTS][FS_THREADS], s_le[FS_SLOTS][FS_THREADS];
    __shared__ uint8_t s_cov[FS_SLOTS][FS_THREADS], s_rep[FS_SLOTS][FS_THREADS], s_cand[FS_SLOTS][FS_THREADS], s_flag[FS_SLOTS][FS_THREADS];
    const int t = threadIdx.x;
    const int64_t loc = (int64_t)blockIdx.x * FS_THREADS + t;
    const int64_t n_loci = (int64_t)a.totals[0];
    if (loc >= n_loci) return;
    int64_t ls, le; locus_range(a, n_loci, loc, ls, le);
    if (le - ls > FF_MAX || a.hard[ls] != LP_FLAT) return;
    const int m = (int)(le - ls);
    const CandSoA &cd = a.cd;
    const bool end_free = a.up.end_dis == 0x7fffffff;                // the default: check_iden's end tests always pass
    uint64_t alive = 0;
    int cnt = 0, ltid = 0;
    // candidate k+1 is loaded while candidate k is folded
    int t_tid = cd.tid[ls], t_start = cd.start[ls], t_end = cd.end[ls], nc = cd.n[ls], fs = cd.fs[ls], lend = cd.le[ls];
    uint32_t rc = a.rep[ls]; uint64_t ev = a.evmask[ls], same = a.kls ? a.samemask[ls] : ~0ull;
    for (int k = 0; k < m; ++k) {
        const int64_t c = ls + k;
        const int c_tid = t_tid, c_start = t_start, c_end = t_end, c_n = nc, c_fs = fs, c_le = lend;
        const uint32_t c_rep = rc - (uint32_t)ls; const uint64_t c_ev = ev, c_same = same;
        if (k + 1 < m) {
            t_tid = cd.tid[c + 1]; t_start = cd.start[c + 1]; t_end = cd.end[c + 1]; nc = cd.n[c + 1]; fs = cd.fs[c + 1]; lend = cd.le[c + 1];
            rc = a.rep[c + 1]; ev = a.evmask[c + 1]; if (a.kls) same = a.samemask[c + 1];
        }
        if (c_tid != 0) {                                             // unsorted input can put two chromosomes into one locus: not for the slots
            if (ltid == 0) ltid = c_tid; else if (c_tid != ltid) { a.hard[ls] = LP_TIER0; return; }
        }
        int kind = 0, hit = 0;                                        // kind: 0 append, 1 merge (identical), 2 drop (partial)
        for (int sl = cnt - 1; sl >= 0; --sl) {
            const int b = s_cand[sl][t];
            if (!(c_ev & alive & ((2ull << b) - 1ull))) break;        // no candidate event at or below this entry: append whatever the stops say
            if (!((c_same >> b) & 1ull)) continue;                    // another sub-stream: invisible
            const int efs = s_fs[sl][t], ele = s_le[sl][t];
            const int fl = s_flag[sl][t];
            const int e_end = (fl & 2) ? 0 : ele;                     // T.end
            if (((fl & 4) && c_tid > 0) || c_start > e_end) break;    // update_gtf.c:148
            if ((c_ev >> b) & 1ull) {
                const bool ok = c_n == 1 ? single_exon_match(a, c_fs, c_le, efs, ele) : end_free || ends_match(a, c_fs, c_le, efs, ele);
                if (ok) { hit = sl; kind = (c_n == 1 || s_rep[sl][t] == (uint8_t)c_rep) ? 1 : 2; break; }
            }
        }
        if (kind == 1) {
            s_cov[hit][t] += 1;                                       // <= 64 candidates per locus: fits a byte
            if (c_fs < s_fs[hit][t]) { s_fs[hit][t] = c_fs; s_flag[hit][t] &= ~1; }
            if (c_le > s_le[hit][t]) { s_le[hit][t] = c_le; s_flag[hit][t] &= ~2; }
        } else if (kind == 0 && absorbed_elsewhere(a, c, true)) {
            kind = 3;
        } else if (kind == 0) {
            if (cnt == FS_SLOTS) { a.hard[ls] = LP_TIER0; return; }   // too many survivors for the slots: fold_big_kernel redoes the locus
            alive |= 1ull << k;
            s_fs[cnt][t] = c_fs; s_le[cnt][t] = c_le; s_cov[cnt][t] = 1;
            s_rep[cnt][t] = (uint8_t)c_rep; s_cand[cnt][t] = (uint8_t)k;
            s_flag[cnt][t] = (uint8_t)((c_start != c_fs ? 1 : 0) | (c_end != c_le ? 2 : 0) | (c_tid == 0 ? 4 : 0));   // bits 0,1: only an unextended piece (start = end = 0)
            ++cnt;
        }
        a.alive[c] = kind == 0 ? 1 : 0;
    }
    for (int sl = 0; sl < cnt; ++sl) {
        const int64_t c = ls + s_cand[sl][t];
        const int f = s_flag[sl][t], efs = s_fs[sl][t], ele = s_le[sl][t];
        a.work.cov[c] = s_cov[sl][t]; a.work.start[c] = (f & 1) ? cd.start[c] : efs; a.work.end[c] = (f & 2) ? cd.end[c] : ele; a.work.fs[c] = efs; a.work.le[c] = ele;
    }
}

// survivors of the fold, compacted in candidate order with their mutated fields (one pass, look-back sum)
static constexpr int FF_ITEMS = 8;
__global__ void __launch_bounds__(FP_THREADS) fold_finish_kernel(MergeArgs a)
{
    __shared__ uint32_t s_scan[33];
    __shared__ uint32_t s_tile; __shared__ uint64_t s_excl;
    if (threadIdx.x == 0) s_tile = atomicAdd(a.ticket, 1u);
    __syncthreads();
    const int tile = (int)s_tile;
    const int64_t c0 = ((int64_t)tile * FP_THREADS + threadIdx.x) * FF_ITEMS, n = cand_count(a);
    uint32_t al = 0, cnt = 0;
#pragma unroll
    for (int i = 0; i < FF_ITEMS; ++i) if (c0 + i < n && a.alive[c0 + i]) { al |= 1u << i; ++cnt; }
    uint32_t tot; const uint32_t ex = block_excl_sum(cnt, s_scan, &tot);
    if (warp_id() == 0) { const uint64_t e = lookback_exclusive(a.tile_state, tile, (uint64_t)tot, OpAdd()); if (lane_id() == 0) s_excl = e; }
    __syncthreads();
    uint32_t k = (uint32_t)s_excl + ex;
#pragma unroll
    for (int i = 0; i < FF_ITEMS; ++i)
        if ((al >> i) & 1u) {
            const int64_t c = c0 + i;
            a.out.cand[k] = (uint32_t)c; a.out.cov[k] = a.work.cov[c]; a.out.tid[k] = a.cd.tid[c]; a.out.start[k] = a.work.start[c]; a.out.end[k] = a.work.end[c];
            a.out.fs[k] = a.work.fs[c]; a.out.le[k] = a.work.le[c];
            ++k;
        }
    if (tile == a.n_tiles - 1 && threadIdx.x == 0) a.totals[1] = s_excl + tot;
}
void launch_merge_finish(MergeArgs a, cudaStream_t st)
{
    if (a.n_cand <= 0) return;
    a.n_tiles = (int)((a.n_cand + FP_THREADS * FF_ITEMS - 1) / (FP_THREADS * FF_ITEMS));
    cudaMemsetAsync(a.tile_state, 0, (size_t)a.n_tiles * 8, st); cudaMemsetAsync(a.ticket, 0, 4, st);
    fold_finish_kernel<<<(unsigned)a.n_tiles, FP_THREADS, 0, st>>>(a); LRB_COUNT_LAUNCH();
}

void launch_merge_fold(const MergeArgs &a, cudaStream_t st)
{
    if (a.n_cand <= 0) return;
    // Grids are sized for the worst case (every candidate its own locus); the locus count is read on the device.
    if (a.up.ss_dis == 0) {
        cudaMemsetAsync(a.hard, 0, (size_t)a.n_cand, st);
        const unsigned bl = (unsigned)((a.n_cand + 255) / 256);
        fold_rep_kernel<<<bl, 256, 0, st>>>(a); LRB_COUNT_LAUNCH();
        fold_relrep_kernel<<<bl, 256, 0, st>>>(a); LRB_COUNT_LAUNCH();
        fold_relasm_kernel<<<bl, 256, 0, st>>>(a); LRB_COUNT_LAUNCH();
        const unsigned bs = (unsigned)((a.n_cand + FS_THREADS - 1) / FS_THREADS);
        fold_seq_kernel<32><<<bs, FS_THREADS, 0, st>>>(a); LRB_COUNT_LAUNCH();
        // loci beyond the masks and the ones the flat kernels gave up on: classes through one table, then warp per locus with the survivors
        // in shared memory; what outgrows the slots there (LP_MERGE_OVER) is replayed from global memory
        int64_t bl2 = (a.n_cand / (FF_MAX + 1) + 1 + 3) / 4 + 8; if (bl2 > 148 * 8) bl2 = 148 * 8;
        using S0 = FbSlots<FB_SLOTS0, 256>; using S1 = FbSlots<416, 1024>;
        auto k0 = fold_big_kernel<32, FB_SLOTS0, 256, 0>; auto k1 = fold_big_kernel<32, 416, 1024, 1>;
        const size_t smem0 = sizeof(S0) * (FB_THREADS / 32), smem1 = sizeof(S1) * (FB_THREADS / 32);
        static bool attr = false;
        if (!attr) { cudaFuncSetAttribute(k0, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem0); cudaFuncSetAttribute(k1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1); attr = true; }
        ClassTab tab{(unsigned long long *)a.ckey, a.cmin, (uint64_t)a.n_cand * 2 + 64};
        cudaMemsetAsync(a.ckey, 0xFF, tab.cap * 8, st); cudaMemsetAsync(a.cmin, 0xFF, tab.cap * 4, st);
        cudaMemsetAsync(a.fb_cnt, 0, 32, st);                     // [0] big loci, [1] tier-0 claims, [2] tier-0 overflows, [3] tier-1 claims, [4] class-row claims, [5] n_indexed
        int64_t blm = (a.n_cand / 8 + 255) / 256 + 1; if (blm > 148 * 8) blm = 148 * 8;
        fold_big_mark_kernel<<<(unsigned)blm, 256, 0, st>>>(a); LRB_COUNT_LAUNCH();
        fold_class_insert_kernel<<<bl, 256, 0, st>>>(a, tab); LRB_COUNT_LAUNCH();
        fold_class_verify_kernel<<<bl, 256, 0, st>>>(a, tab); LRB_COUNT_LAUNCH();
        fold_class_rows_kernel<<<(unsigned)blm, 256, 0, st>>>(a, a.fb_cnt + 4); LRB_COUNT_LAUNCH();
        // one warp per locus, loci claimed from the lists: a whole warp measured fastest (8 / 16 lanes per locus: 17.5 / 15.8 ms per
        // step against 14.2 ms on the 10 M-read data set -- the lane groups of a warp diverge)
        int64_t blb = (a.n_cand / (FF_MAX + 1) + 1) / (FB_THREADS / 32) + 1; if (blb > 148 * 6) blb = 148 * 6;
        k0<<<(unsigned)blb, FB_THREADS, smem0, st>>>(a, a.fb_cnt + 1); LRB_COUNT_LAUNCH();
        if (blb > 148 * 2) blb = 148 * 2;
        k1<<<(unsigned)blb, FB_THREADS, smem1, st>>>(a, a.fb_cnt + 3); LRB_COUNT_LAUNCH();
        merge_fold_kernel<32><<<(unsigned)bl2, MF_THREADS, 0, st>>>(a, 0x7fffffff, 0x7fffffff, (1 << LP_MERGE_OVER) | (1 << LP_MERGE_VERIFY));
        LRB_COUNT_LAUNCH();
        return;
    }
    // inexact splice-site matching (-d > 0): the relation is neither static nor transitive -- lane groups replay the fold
    {
        constexpr int GPB = MF_THREADS / 8;
        int64_t bl = (a.n_cand + GPB - 1) / GPB; if (bl > 148 * 12) bl = 148 * 12;
        merge_fold_kernel<8><<<(unsigned)bl, MF_THREADS, 0, st>>>(a, 1, 32, 0);
        LRB_COUNT_LAUNCH();
    }
    {
        int64_t bl = (a.n_cand / 33 + 1 + 3) / 4; if (bl > 148 * 8) bl = 148 * 8;
        merge_fold_kernel<32><<<(unsigned)bl, MF_THREADS, 0, st>>>(a, 33, 0x7fffffff, 0);
        LRB_COUNT_LAUNCH();
    }
}

// Test hook (lrb_fold_census): after launch_merge_fold on the same stream, read the locus table back and tally each locus by the path
// that folded it: the final LocusPath at its head.  A big locus's locus_cnt holds one byte per sub-stream, written by
// fold_class_rows_kernel unless class verification had already sent the locus to merge_fold_kernel (LP_MERGE_VERIFY): that byte is
// stale then and not read.
cudaError_t merge_fold_census(const MergeArgs &a, cudaStream_t st, int64_t *k)
{
    uint64_t n_loci = 0, n_dev = (uint64_t)a.n_cand;
    cudaError_t e;
    if ((e = cudaMemcpyAsync(&n_loci, a.totals, 8, cudaMemcpyDeviceToHost, st))) return e;
    if (a.n_cand_dev && (e = cudaMemcpyAsync(&n_dev, a.n_cand_dev, 8, cudaMemcpyDeviceToHost, st))) return e;
    if ((e = cudaStreamSynchronize(st))) return e;
    const int64_t n = n_dev > (uint64_t)a.n_cand ? 0 : (int64_t)n_dev;      // as cand_count: an undersized list is folded empty
    if (a.n_cand <= 0 || n == 0 || n_loci == 0) return cudaSuccess;
    const bool exact = a.up.ss_dis == 0;
    std::vector<uint32_t> ls(n_loci), cnt(n_loci); std::vector<uint8_t> hard(n);
    if ((e = cudaMemcpyAsync(ls.data(), a.locus_start, n_loci * 4, cudaMemcpyDeviceToHost, st))) return e;
    if (exact && (e = cudaMemcpyAsync(cnt.data(), a.locus_cnt, n_loci * 4, cudaMemcpyDeviceToHost, st))) return e;
    if (exact && (e = cudaMemcpyAsync(hard.data(), a.hard, (size_t)n, cudaMemcpyDeviceToHost, st))) return e;
    uint32_t n_indexed = 0;
    if (exact && a.n_indexed && (e = cudaMemcpyAsync(&n_indexed, a.n_indexed, 4, cudaMemcpyDeviceToHost, st))) return e;
    if ((e = cudaStreamSynchronize(st))) return e;
    k[LRB_FC_INDEXED] += n_indexed;
    for (uint64_t loc = 0; loc < n_loci; ++loc) {
        const int64_t m = (loc + 1 < n_loci ? (int64_t)ls[loc + 1] : n) - (int64_t)ls[loc];
        if (a.single_locus) ++k[LRB_FC_SINGLE];
        if (!exact) { ++k[m <= 32 ? LRB_FC_D_SMALL : LRB_FC_D_LARGE]; continue; }   // merge_fold_kernel<8> / <32>
        const int h = hard[ls[loc]];
        if (h == LP_FLAT && m <= FF_MAX) { ++k[LRB_FC_FLAT]; continue; }
        ++k[h <= LP_TIER0 ? LRB_FC_TIER0 : h == LP_TIER1 ? LRB_FC_TIER1 : h == LP_MERGE_OVER ? LRB_FC_MERGE_OVER : LRB_FC_MERGE_VERIFY];
        if (h == LP_MERGE_VERIFY) continue;
        for (int s = 0; s < (a.kls ? 4 : 1); ++s) k[LRB_FC_NOROWS] += ((const uint8_t *)&cnt[loc])[s] == CLASSES_UNTABULATED;
    }
    return cudaSuccess;
}

// ------------------------------------------------------------------------------ split pieces that meet ANOTHER chromosome
// A split piece carries tid = start = end = 0 (SURVEY Q14), so its back-scan in merge_trans never stops (update_gtf.c:148): after the
// entries of its own locus it walks ALL earlier entries of updated_T, on every chromosome, and the first one with check_iden != -1
// absorbs it.  The locus-parallel fold cannot see that.  It is settled in rounds instead:
//   detect   after a fold: the junctions of the surviving (or already forced) pieces go into a small key set; every surviving entry
//            probes it (its first junction among a piece's junctions / a piece's first junction among its own: the necessary condition
//            of gtf.c:61-91); the few hits are joined with the pieces and check_iden is evaluated exactly; best[p] = nearest earlier
//            entry on another chromosome that absorbs p;
//   force    pieces with such an entry are marked; if the marks changed, the fold runs again with them: a marked piece that finds
//            nothing in its own locus is NOT appended (and no longer a barrier there);
//   apply    once the marks are stable: the absorbing entries take cov / first start / last end as merge_trans1 would (update_gtf.c:104-111).
// What a piece meets depends only on earlier entries, so round k fixes the k-th affected piece at the latest.  Steady state (no piece
// meets anything): one round, three small kernels.
LRB_DEVINL uint64_t xl_key(uint32_t kind, uint32_t e, uint32_t s) { uint64_t k = mixh(mixh(0x51ED270B3Full + kind, e), s); return k == ~0ull ? 0x77ull : k; }
LRB_DEVINL bool xl_upsert(const XlArgs &x, uint64_t k, uint32_t rt)
{
    uint64_t s = __umul64hi(k * 0x9E3779B97F4A7C15ull, x.tcap);
    for (int probes = 0; probes < 4096; ++probes) {
        const unsigned long long p = atomicCAS(&x.tkey[s], ~0ull, (unsigned long long)k);
        if (p == ~0ull || p == k) { atomicMin(&x.tmin[s], rt); atomicMax(&x.tmax[s], rt + 1u); return true; }
        s = s + 1 == x.tcap ? 0 : s + 1;
    }
    return false;
}
LRB_DEVINL bool xl_other_chrom(const XlArgs &x, uint64_t k, uint32_t rt)      // is the key owned by a piece of another chromosome?
{
    uint64_t s = __umul64hi(k * 0x9E3779B97F4A7C15ull, x.tcap);
    for (int probes = 0; probes < 4096; ++probes) {
        const unsigned long long p = x.tkey[s];
        if (p == ~0ull) return false;
        if (p == k) return x.tmin[s] != rt || x.tmax[s] != rt + 1u;
        s = s + 1 == x.tcap ? 0 : s + 1;
    }
    return true;
}
__global__ void __launch_bounds__(256) xl_insert_kernel(MergeArgs a, XlArgs x)
{
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cand_count(a) || a.list.piece[c] < 0) return;
    const int n = a.cd.n[c];
    if (n < 2 || !(a.alive[c] || a.forced[c])) return;
    const uint32_t i = atomicAdd(&x.cnt[XL_NPL], 1u);
    x.pl[i] = (uint32_t)c; x.best[c] = 0;
    const uint32_t g = a.cd.gbeg[c], rt = (uint32_t)a.rows.tid[a.list.row[c]];
    bool ok = true;
    for (int j = 0; j < n - 1; ++j) {
        const uint32_t e = (uint32_t)a.ex.ee[g + j], s = (uint32_t)a.ex.es[g + j + 1];
        ok = ok && xl_upsert(x, xl_key(0, e, s), rt);
        if (j == 0) ok = ok && xl_upsert(x, xl_key(1, e, s), rt);
    }
    if (!ok) x.cnt[XL_OVERFLOW] = 1u;
}
__global__ void __launch_bounds__(256) xl_probe_kernel(MergeArgs a, XlArgs x)
{
    if (x.cnt[XL_NPL] == 0) return;
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= cand_count(a) || !a.alive[c]) return;
    const int n = a.cd.n[c];
    if (n < 2) return;
    const uint32_t g = a.cd.gbeg[c], rt = (uint32_t)a.rows.tid[a.list.row[c]];
    bool hit = xl_other_chrom(x, xl_key(0, (uint32_t)a.ex.ee[g], (uint32_t)a.ex.es[g + 1]), rt);
    for (int j = 0; j < n - 1 && !hit; ++j) hit = xl_other_chrom(x, xl_key(1, (uint32_t)a.ex.ee[g + j], (uint32_t)a.ex.es[g + j + 1]), rt);
    if (!hit) return;
    const uint32_t k = atomicAdd(&x.cnt[XL_NHX], 1u);
    if (k < x.hx_cap) x.hx[k] = (uint32_t)c; else x.cnt[XL_OVERFLOW] = 1u;
}
// pieces x hits: exact check_iden of the piece against the surviving entry (dynamic first start / last end of the entry)
__global__ void __launch_bounds__(256) xl_join_kernel(MergeArgs a, XlArgs x)
{
    const uint32_t n_pl = x.cnt[XL_NPL], n_hx = min(x.cnt[XL_NHX], x.hx_cap);
    const CandSoA &cd = a.cd;
    for (uint32_t h = blockIdx.y; h < n_hx; h += gridDim.y) {
        const uint32_t e = x.hx[h];
        const int e_tid = a.rows.tid[a.list.row[e]];
        const Entry E = entry_of(cd, e, a.work.fs[e], a.work.le[e]);
        for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_pl; i += gridDim.x * blockDim.x) {
            const uint32_t p = x.pl[i];
            if (e >= p || a.rows.tid[a.list.row[p]] == e_tid) continue;          // only EARLIER entries, and its own chromosome is the fold's business
            if (a.up.force_strand && ((cd.rev[e] ^ cd.rev[p]) & 1)) continue;    // pieces carry is_rev 0 in cd.rev (update_gtf.c:149)
            const Entry P = entry_of(cd, p, cd.fs[p], cd.le[p]);
            const int r = chain_iden(a.ex, P, E, 0, a.up.end_dis);
            if (r == 0 || r == 2) atomicMax((unsigned long long *)&x.best[p], ((unsigned long long)(e + 1u) << 2) | (r == 0 ? 1ull : 2ull));
        }
    }
}
__global__ void __launch_bounds__(256) xl_force_kernel(MergeArgs a, XlArgs x)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= x.cnt[XL_NPL]) return;
    const uint32_t p = x.pl[i];
    const bool want = x.best[p] != 0, is = a.forced[p] != 0;
    if (want != is) { a.forced[p] = want ? 1 : 0; atomicAdd(&x.cnt[XL_CHANGED], 1u); }     // else: 3 (absorbed across chromosomes in the fold that just ran) stays for xl_apply
    if (want) atomicAdd(&x.cnt[XL_NFORCED], 1u);
}
// before a fold runs again: "absorbed across chromosomes in the last fold" (3) is history
__global__ void __launch_bounds__(256) xl_reset_kernel(MergeArgs a, XlArgs x)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < x.cnt[XL_NPL] && a.forced[x.pl[i]] == 3) a.forced[x.pl[i]] = 1;
}
void launch_xlocus_reset(const MergeArgs &a, const XlArgs &x, cudaStream_t st)
{
    if (a.n_cand <= 0) return;
    xl_reset_kernel<<<(unsigned)((a.n_cand / 16 + 255) / 256 + 1), 256, 0, st>>>(a, x); LRB_COUNT_LAUNCH();
}
// the marks are stable: entries that absorbed a piece by identity take cov + 1 and the piece's ends (merge_trans1, update_gtf.c:104-111)
__global__ void __launch_bounds__(256) xl_apply_kernel(MergeArgs a, XlArgs x, int pass)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= x.cnt[XL_NPL]) return;
    const uint32_t p = x.pl[i];
    if (a.forced[p] != 3 || (x.best[p] & 3ull) != 1ull) return;                  // absorbed inside its locus after all / dropped as a partial match
    const uint32_t e = (uint32_t)(x.best[p] >> 2) - 1u;
    if (pass == 0) { atomicAdd(&a.work.cov[e], 1); atomicMin(&a.work.fs[e], a.cd.fs[p]); atomicMax(&a.work.le[e], a.cd.le[p]); }
    else {                                           // T.start / T.end follow an extension (:108-111); equal values race benignly
        if (a.work.fs[e] < a.cd.fs[e]) a.work.start[e] = a.work.fs[e];
        if (a.work.le[e] > a.cd.le[e]) a.work.end[e] = a.work.le[e];
    }
}
void launch_xlocus_detect(const MergeArgs &a, const XlArgs &x, cudaStream_t st)
{
    if (a.n_cand <= 0) return;
    cudaMemsetAsync(x.tkey, 0xFF, x.tcap * 8, st); cudaMemsetAsync(x.tmin, 0xFF, x.tcap * 4, st); cudaMemsetAsync(x.tmax, 0, x.tcap * 4, st);
    cudaMemsetAsync(x.cnt, 0, XL_NCNT * 4, st);
    const unsigned bl = (unsigned)((a.n_cand + 255) / 256);
    xl_insert_kernel<<<bl, 256, 0, st>>>(a, x); LRB_COUNT_LAUNCH();
    xl_probe_kernel<<<bl, 256, 0, st>>>(a, x); LRB_COUNT_LAUNCH();
    xl_join_kernel<<<dim3(64, 64), 256, 0, st>>>(a, x); LRB_COUNT_LAUNCH();
    int64_t blp = (a.n_cand / 16 + 255) / 256 + 1;                   // pieces are a small share of the candidates; the kernel checks the true count
    xl_force_kernel<<<(unsigned)blp, 256, 0, st>>>(a, x); LRB_COUNT_LAUNCH();
}
void launch_xlocus_apply(const MergeArgs &a, const XlArgs &x, cudaStream_t st)
{
    if (a.n_cand <= 0) return;
    int64_t blp = (a.n_cand / 16 + 255) / 256 + 1;
    for (int pass = 0; pass < 2; ++pass) { xl_apply_kernel<<<(unsigned)blp, 256, 0, st>>>(a, x, pass); LRB_COUNT_LAUNCH(); }
}

__global__ void __launch_bounds__(256) merge_class_counts_kernel(MergeArgs a)
{
    __shared__ uint32_t s_class[4];
    if (threadIdx.x < 4) s_class[threadIdx.x] = 0;
    __syncthreads();
    const int64_t n = cand_count(a);
    uint32_t ccnt = 0;                                               // four 8-bit counters
    for (int64_t c = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4, i = 0; i < 4 && c + i < n; ++i)
        if (a.alive[c + i]) ccnt += 1u << (8 * a.kls[c + i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ccnt += __shfl_xor_sync(FULL, ccnt, o);         // <= 128 per class and warp
    if (lane_id() == 0) for (int q = 0; q < 4; ++q) { const uint32_t v = (ccnt >> (8 * q)) & 0xffu; if (v) atomicAdd(&s_class[q], v); }
    __syncthreads();
    if (threadIdx.x < 4 && s_class[threadIdx.x]) atomicAdd(&a.class_alive[threadIdx.x], s_class[threadIdx.x]);
}
void launch_merge_class_counts(const MergeArgs &a, cudaStream_t st)
{
    if (a.n_cand <= 0) return;
    merge_class_counts_kernel<<<(unsigned)((a.n_cand + 1023) / 1024), 256, 0, st>>>(a);
    LRB_COUNT_LAUNCH();
}

}  // namespace lrbk
