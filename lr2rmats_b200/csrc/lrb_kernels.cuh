// lrb_kernels.cuh -- device-side data layout and kernel launchers shared by the .cu files of liblr2rmats_b200.so.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/lr2rmats_b200.h"

namespace lrbk {

// ---- record batch resident in HBM (structure of arrays; mirrors lrb_batch)
struct DBatch {
    int64_t n = 0, n_cigar = 0;
    int32_t *tid = nullptr, *pos = nullptr, *l_qseq = nullptr, *nm = nullptr;
    uint16_t *flag = nullptr;
    int8_t *xs = nullptr;
    uint64_t *qhash = nullptr;
    uint64_t *cigar_off = nullptr; uint32_t *cigar = nullptr;
};

// ---- remove table (-r GTF) as an index: per tid the entries visible to remove_overlap()'s early exit
// (bam_filter.c:54-57), sorted by start with a running max of end.
struct DRmIndex {
    int32_t n_groups = 0, n = 0;
    int32_t *g_tid = nullptr, *g_off = nullptr;     // n_groups, n_groups+1
    int32_t *start = nullptr, *pmax_end = nullptr;  // n
};

// ---- annotation in HBM: transcripts in file order + exon pools + prefix-max keys for the cursor closed form
struct DAnno {
    int32_t n = 0; int64_t n_exon = 0;
    int32_t *tid = nullptr, *start = nullptr, *end = nullptr, *gene = nullptr;
    uint8_t *is_rev = nullptr;
    uint32_t *exon_off = nullptr;
    int32_t *es = nullptr, *ee = nullptr;
    uint64_t *pmax_key = nullptr;                   // P_j = max_{i<=j} ((tid_i+1)<<32 | end_i)   (SURVEY App. B.1)
    uint8_t *mono = nullptr;                        // 1: exon starts and exon ends of the transcript strictly increase
};
struct DSj {
    int64_t n = 0;
    int32_t *tid = nullptr, *don = nullptr, *acc = nullptr, *cnt_u = nullptr, *cnt_m = nullptr;
    uint64_t *pmax_key = nullptr;                   // Q_i = max_{k<=i} ((tid_k+1)<<32 | acc_k)   (SURVEY App. B.2)
    uint64_t *don_key = nullptr;                    // (tid+1)<<32 | don  (non-decreasing: table is sorted)
};

// ---- read rows (the reads that went through the CIGAR walk, in record order)
struct DRows {
    int64_t n = 0, cap = 0;
    uint32_t *read_idx = nullptr;                   // record index in the batch
    int32_t *tid = nullptr, *start = nullptr, *end = nullptr;   // trans_t.tid / start / end
    uint8_t *is_rev = nullptr;
    uint32_t *ex_beg = nullptr, *ex_n = nullptr;    // exon slots [ex_beg, ex_beg+ex_n) in the pools
};
struct DExons {
    int64_t n = 0, cap = 0;
    int32_t *es = nullptr, *ee = nullptr;
    uint8_t *flag = nullptr;                        // LRB_F_* per slot (classification output)
};

struct ScanArgs {
    DBatch b;
    lrb_filter_params fp; lrb_exon_params ep;
    DRmIndex rm;
    int mode;                                       // 0 filter only (writes no rows), 1 exon only, 2 fused
    const uint8_t *sel_mask;                        // mode 1: records to walk (NULL = all)
    uint8_t *pass; int32_t *score, *intron_n;       // filter outputs (record level)
    DRows rows; DExons ex;
    uint64_t *tile_state; uint32_t *ticket;         // look-back state (zeroed per walk), tile ticket (zeroed per launch)
    uint64_t *totals;                               // [0] rows, [1] exons
    int reads_per_tile, stage_words;
    int rows_by_record;                             // 1: a passing record's row is written at its record index (no row compaction)
    // the ops of the launch's tiles: op k of the batch (cigar_off[r] <= k < cigar_off[r + 1] for a record r of these tiles) is
    // ops[k - op_base].  The whole pool (ops = b.cigar, op_base = 0), or one chunk of it staged from host memory (op_base a
    // multiple of 4, so that the 16-byte alignment of the pool holds in the staging buffer).
    const uint32_t *ops; uint64_t op_base;
    int tile_base;                                  // a launch walks tiles [tile_base, tile_base + its grid's tiles)
};

void launch_cigar_scan(const ScanArgs &a, int n_tiles, bool stream_mode, size_t smem_bytes, cudaStream_t st);
int stream_reads_per_tile();                        // tile size of the long-CIGAR streaming kernel
int scan_reads_per_tile();                          // tile size of the short-CIGAR kernel
// ordered compaction of the set positions of a byte mask: out[k] = index of k-th nonzero
void launch_compact_mask(const uint8_t *mask, int64_t n, uint32_t *out, uint64_t *tile_state, uint32_t *ticket, uint64_t *total, cudaStream_t st);
void launch_select_records(const DBatch &b, const uint8_t *pass, const int32_t *score, const int32_t *intron_n, lrb_filter_params fp,
                           uint8_t *keep_rec_mask, cudaStream_t st);
void launch_compact_gather(const uint8_t *mask, int64_t n, const DRows &src_by_record, DRows &dst, uint32_t *keep_idx,
                           uint64_t *tile_state, uint32_t *ticket, uint64_t *total, cudaStream_t st);

// ---- classification
struct ClassArgs {
    DRows rows; DExons ex; DAnno anno; DSj sj;
    lrb_update_params up;
    uint32_t *cls; int32_t *ref;
    uint32_t *n_novel;                              // per row: 0, 1 (whole read) or number of split pieces
    uint32_t *err_flags;                            // bit0 unsorted, bit1 unmapped/empty chain
    const uint8_t *row_nonmono;                     // NULL: every row's exon starts/ends are non-decreasing (always true for CIGAR chains)
};
void launch_classify(const ClassArgs &a, uint8_t *slow_rows_scratch, cudaStream_t st);   // scratch: one byte per row

// ---- novel_T / known / unrecog lists + merge fold
struct DTransList {                                 // transcript rows of a list (whole reads or split pieces)
    int64_t n = 0, cap = 0;
    uint32_t *row = nullptr, *lo = nullptr, *cnt = nullptr; int32_t *piece = nullptr;
};
struct ListArgs {
    DRows rows; DExons ex; lrb_update_params up;
    const uint32_t *cls; const uint32_t *n_novel;
    DTransList novel; uint32_t *known, *unrecog;    // novel.cap bounds the writes; the true size is totals[0]
    uint8_t *kls; uint32_t *class_n;                // optional (summary): class per row, class sizes [4]
    uint64_t *tile_state; uint32_t *ticket; uint64_t *totals;   // [0] novel, [1] known, [2] unrecog
    int n_tiles;
};
void launch_build_lists(ListArgs a, cudaStream_t st);

struct DMerged {
    int64_t n = 0, cap = 0;
    uint32_t *cand = nullptr; int32_t *cov = nullptr, *tid = nullptr, *start = nullptr, *end = nullptr, *fs = nullptr, *le = nullptr;
};
struct CandSoA {                                    // flattened fold candidates (see fold_prepare_kernel)
    int32_t *tid = nullptr, *start = nullptr, *end = nullptr, *rev = nullptr, *n = nullptr, *fs = nullptr, *le = nullptr;
    uint32_t *gbeg = nullptr; uint64_t *hash = nullptr;
    uint64_t *j0 = nullptr;                         // first junction (exon[0].end << 32 | exon[1].start), 0 for single-exon chains
    uint64_t *sig = nullptr;                        // 64-bit membership signature of all junctions of the chain
};
struct MergeArgs {
    DRows rows; DExons ex; lrb_update_params up; CandSoA cd;
    DTransList list;                                // candidates in fold order
    const uint32_t *subset;                         // optional: rows subset as whole-read candidates (list.n==0): indices into rows
    int64_t n_cand;                                 // candidates (host value, or the host's upper bound when n_cand_dev is set)
    const uint64_t *n_cand_dev;                     // optional: the true count, produced on the device
    int n_tiles;
    int single_locus;                               // 1: the whole list is ONE locus (unsorted input: no cut is safe, the fold is replayed in order)
    int presegmented;                               // 1: head, locus_start and totals[0] were written by launch_class_order
    const uint8_t *kls;                             // optional: sub-stream id per candidate (class folds: four independent folds in one pass); NULL: one stream
    uint4 *cbase;                                   // with kls: per locus the candidates of each sub-stream before its head, [n_loci] the totals
                                                    // (the list is in class order: inside a locus the sub-streams follow each other, class_range)
    uint64_t *samemask;                             // flat fold with kls: earlier candidates of the locus in the same sub-stream
    uint32_t *class_alive;                          // [4] surviving entries per sub-stream
    // scratch
    uint32_t *tlist;                                // merge_fold_kernel: candidate index of each entry of T, at the locus' offset
    uint8_t *head;                                  // locus head flags
    uint32_t *locus_start;                          // compacted heads (+ sentinel)
    DMerged work;                                   // per-candidate slots (T entries live at their locus' range)
    uint32_t *locus_cnt;                            // big loci: number of multi-exon classes per sub-stream (CLASSES_UNTABULATED: too many for the relation rows)
    uint8_t *alive;                                 // per candidate: 1 = an entry of T after the fold (0: absorbed / dropped)
    uint32_t *rep, *lstart; uint64_t *evmask;       // flat fold: class representative, locus head, absorber mask per candidate
    uint16_t *desc; uint64_t *relsym;               // flat fold: class descriptor per candidate; per representative the related representatives
    uint8_t *hard;                                  // per locus head: the path that folds the locus next (LocusPath, lrb_update.cu)
    uint8_t *cord; uint64_t *crow;                  // big loci: class ordinal per candidate; per representative its 128-bit relation row
    uint32_t *clist;                                // not used by the fold: the split-piece rounds' piece list (XlArgs::pl)
    // lent to XlArgs once the fold is done, as well: lstart as its hit list hx, relsym as best
    uint32_t *fb_list, *fb_cnt;                     // big loci: [0, n_cand) list of their locus ordinals, [n_cand, 2 n_cand) those that outgrew tier 0; counters
    void *fb_state;                                 // big loci: tier 0's replay state per entry that outgrew it (fold_resume_bytes)
    uint64_t *ckey; uint32_t *cmin;                 // class table of the big loci: 2 * n_cand + 64 slots
    uint32_t *n_indexed;                            // optional (fold census): multi-exon candidates fold_big_kernel decided by its class index
    DMerged out;                                    // compacted result
    uint8_t *forced;                                // optional (split pieces, see XlArgs): 1 = this piece is absorbed by an entry of an earlier locus when its own locus has nothing for it (3: that happened in the last fold)
    uint64_t *tile_state; uint32_t *ticket; uint64_t *totals;  // [0] n_loci, [1] n_out
};
// split pieces that meet another chromosome (lrb_update.cu, xl_* kernels)
enum { XL_NPL = 0, XL_NHX = 1, XL_CHANGED = 2, XL_NFORCED = 3, XL_OVERFLOW = 4, XL_NCNT = 8 };
struct XlArgs {
    unsigned long long *tkey; uint32_t *tmin, *tmax; uint64_t tcap;   // key set of the pieces' junctions with the range of chromosomes that own each
    uint32_t *pl, *hx; uint32_t hx_cap;             // piece list, hit list (surviving entries that share a key with a piece of another chromosome)
    uint64_t *best;                                 // per candidate: (absorbing entry + 1) << 2 | 1 identical / 2 partial
    uint32_t *cnt;                                  // XL_* counters (device)
};
void launch_xlocus_detect(const MergeArgs &a, const XlArgs &x, cudaStream_t st);    // after launch_merge_fold, before launch_merge_finish
void launch_xlocus_apply(const MergeArgs &a, const XlArgs &x, cudaStream_t st);
void launch_xlocus_reset(const MergeArgs &a, const XlArgs &x, cudaStream_t st);     // before the fold runs again with new marks
// class folds: the rows (a.rows, all of them, a.n_cand) cut into loci in row order, then each locus's rows grouped by their class
// row_kls (known, reliable, unreliable, unrecognized), each group in row order: perm[c] = row of candidate c, cand_kls[c] = its class;
// head, locus_start, cbase and totals[0] as launch_merge_prepare would leave them for the rows in row order (a.tlist is scratch)
void launch_class_order(MergeArgs a, const uint8_t *row_kls, uint32_t *perm, uint8_t *cand_kls, cudaStream_t st);
void launch_merge_prepare(MergeArgs a, cudaStream_t st);            // candidates, locus heads, locus_start; totals[0] = number of loci
void launch_merge_fold(const MergeArgs &a, cudaStream_t st);        // number of loci is read from a.totals[0] on the device
size_t fold_resume_bytes(int64_t n_cand);                           // size of MergeArgs::fb_state
cudaError_t merge_fold_census(const MergeArgs &a, cudaStream_t st, int64_t *counts);   // test hook: synchronises st, adds to counts[LRB_FC_*]
void launch_merge_class_counts(const MergeArgs &a, cudaStream_t st);
void launch_merge_finish(MergeArgs a, cudaStream_t st);             // survivors compacted into a.out; totals[1] = their number

// lrb_sort.cu: stable LSD radix sort of rows by samtools' coordinate key
int sort_tiles(int64_t n);
void launch_sort_keys(const DRows &rows, const uint16_t *flag, uint64_t *keys, uint32_t *idx, unsigned long long *max_key, cudaStream_t st);
void launch_sort_pass(const uint64_t *kin, const uint32_t *vin, uint64_t *kout, uint32_t *vout, int64_t n, int shift, uint32_t *hist, cudaStream_t st);
void launch_rows_permute(const DRows &in, const DRows &out, const uint32_t *perm, cudaStream_t st);

// generic device scans used by the stages above
void launch_scan_sum_u32(const uint32_t *in, uint32_t *out_excl, int64_t n, uint64_t *tile_state, uint32_t *ticket, uint64_t *total, cudaStream_t st);

int64_t count_launches();   // kernels launched by this library since load (every launch_* bumps it)

}  // namespace lrbk
