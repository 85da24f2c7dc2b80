/* lr2rmats_b200.h -- C ABI of the B200-native lr2rmats hot path.
 *
 * The reference (Xinglab/lr2rmats) has no plugin/FFI layer: its data-parallel
 * seams are plain C functions inside one binary (SURVEY.md section 8b).  Every
 * entry point below replaces one of those seams and cites it.  All pointers are
 * plain host pointers to structure-of-arrays buffers, sizes are explicit, no
 * CUDA or torch types cross this boundary.  Functions return LRB_OK (0) or a
 * negative LRB_E_* code; nothing in the library calls exit()/abort() (the
 * reference's err_fatal() does, utils.c:91-111 -- the CLI keeps that behaviour
 * above this boundary).
 *
 * Threading: one host thread per lrb_ctx.  A ctx owns one CUDA device, one
 * stream, all device memory and the pinned host result buffers it hands out.
 * Result pointers stay valid until the next *_run/_fetch call of the same kind
 * on that ctx or lrb_ctx_destroy().  Each kind has pinned buffers of its own:
 *   filter  lrb_filter_fetch, lrb_filter, lrb_filter_fetch_keep
 *   exons   lrb_exon_fetch, lrb_bam2gtf
 *   update  lrb_update_fetch, lrb_update_gtf, lrb_update_fetch_table
 *   unique  lrb_unique_fetch, lrb_unique_gtf
 *   bam2sj  lrb_bam2sj
 *   sort3   lrb_sort3
 *   gather  lrb_gather_fetch
 *   gather reads  lrb_gather_fetch_reads
 */
#ifndef LR2RMATS_B200_H
#define LR2RMATS_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRB_OK            0
#define LRB_E_CUDA       -1   /* CUDA runtime error (message in lrb_last_error) */
#define LRB_E_ARG        -2   /* bad argument / missing prerequisite stage */
#define LRB_E_NOMEM      -3
#define LRB_E_UNSORTED   -4   /* update/unique need (tid,start)-sorted reads (update_gtf.c:41) */
#define LRB_E_UNMAPPED   -5   /* unmapped record given to update/unique (reference aborts, bam2gtf.c:95-100) */
#define LRB_E_NODEVICE   -6   /* no CUDA device: there is NO CPU fallback */
#define LRB_E_NCCL       -7   /* NCCL missing or a collective failed (message in lrb_last_error) */
#define LRB_E_XSHARD     -8   /* multi-GPU merge: a split piece shares a junction with a transcript of another shard; the
                                 reference could merge them (update_gtf.c:148) -- rerun this input unsharded */

/* ------------------------------------------------------------------ inputs */

/* One batch of alignment records decoded from BAM/SAM (bam1_core_t fields the
 * path consumes, htslib/sam.h:149-158, plus the NM / XS:A aux tags and a hash
 * of the query name).  CIGAR words are BAM-packed (len<<4|op, sam.h:65-84). */
typedef struct {
    int64_t         n;           /* records */
    const int32_t  *tid;         /* core.tid, -1 = no reference */
    const int32_t  *pos;         /* core.pos, 0-based */
    const uint16_t *flag;        /* core.flag */
    const int32_t  *l_qseq;      /* core.l_qseq */
    const int32_t  *nm;          /* NM:i value (bam_aux2i), 0 when absent */
    const int8_t   *xs;          /* XS:A value (bam_aux2A): 0 = tag absent */
    const uint64_t *qname_hash;  /* 64-bit hash of qname; equal names <=> equal hash */
    const uint64_t *cigar_off;   /* n+1 offsets into cigar[] (64-bit: a batch may hold more than 2^32 CIGAR ops) */
    const uint32_t *cigar;       /* cigar_off[n] words */
} lrb_batch;

/* Annotation transcripts exactly as read_anno_trans() builds anno_T
 * (gtf.c:468-521): FILE ORDER, exons ascending by (start,end) per transcript,
 * tid = bam_name2id() (-1 when the chromosome is not in the BAM header).
 * `gene` is an interned id of the gene_id string (equal string <=> equal id),
 * which is all the path needs of it (update_gtf.c:176-179). */
typedef struct {
    int32_t         n_trans;
    int64_t         n_exon;
    const int32_t  *tid, *start, *end;   /* per transcript */
    const uint8_t  *is_rev;
    const int32_t  *gene;
    const uint32_t *exon_off;            /* n_trans+1 */
    const int32_t  *exon_start, *exon_end;
} lrb_anno;

/* STAR SJ.out.tab rows as read_sj_group() leaves them (gtf.c:431-449):
 * sorted by (tid,don,acc); tid from the cname table seeded by the BAM header. */
typedef struct {
    int64_t         n;
    const int32_t  *tid, *don, *acc, *uniq_c, *multi_c;
} lrb_sj;

/* Read-derived transcripts given directly as exon chains (the `-m g` GTF input
 * mode, read_gtf_trans gtf.c:524-595), bypassing the CIGAR walk. */
typedef struct {
    int64_t         n;
    const int32_t  *tid;
    const uint8_t  *is_rev;
    const uint32_t *exon_off;            /* n+1 */
    const int32_t  *exon_start, *exon_end;
} lrb_chains;

/* --------------------------------------------------------------- parameters */

typedef struct {               /* bam_filter.c:100 (floats parsed by atof into float) */
    float   cov_rate;          /* -v  0.67 */
    float   map_qual;          /* -q  0.75 */
    float   sec_rat;           /* -s  0.98 */
    int32_t min_intron_n;      /* -i  0    */
} lrb_filter_params;

typedef struct {               /* bam2gtf.c:122, gtf.h:118-120 */
    int32_t min_exon;          /* -e 3  */
    int32_t min_intron;        /* -i 3  */
    int32_t max_delet;         /* -t 50 */
} lrb_exon_params;

typedef struct {               /* sj_para, parse_bam.c:71-84 (the fields bam2sj_core reads) */
    int32_t min_intron;        /* -i 3 (INTRON_MIN_LEN, gtf.h:118) */
    int32_t pair_only;         /* read_type == PAIR_T: 1 in the reference whatever the options say (parse_bam.c:76,997) */
} lrb_sj_params;

typedef struct {               /* update_gtf_para, update_gtf.h:8-15; defaults update_gtf.c:24-35 */
    int32_t min_sj_cnt;        /* -J 1 */
    int32_t ss_dis;            /* -d 0 */
    int32_t end_dis;           /* -D 0x7fffffff */
    int32_t full_level;        /* -l 5 */
    int32_t split_trans;       /* -s 0 */
    int32_t use_multi;         /* -M 0 */
    int32_t force_strand;      /* -c 0 */
    float   single_exon_ovlp_frac; /* -f 0.80 */
    int32_t want_summary;      /* compute print_trans_summary()'s sets/counts (-y / -E) */
} lrb_update_params;

/* ------------------------------------------------------------------ results */

typedef struct {               /* gtf_filter + qname-run selection, bam_filter.c:61-86,129-159 */
    int64_t         n;
    const uint8_t  *pass;      /* gtf_filter()==0 */
    const int32_t  *score;     /* valid where pass */
    const int32_t  *intron_n;  /* valid where pass */
    int64_t         n_keep;    /* records written by sam_write1, in output order */
    const uint32_t *keep_idx;
} lrb_filter_result;

/* Exon chains (gen_exon bam2gtf.c:31-78 + set_trans_name gtf.c:94-100).  Row r
 * describes record read_idx[r] (read_idx==NULL: identity).  Unmapped records
 * give an empty chain (gen_trans returns 0, bam2gtf.c:82). */
typedef struct {
    int64_t         n_reads;
    const uint32_t *read_idx;
    const int32_t  *tid;       /* per row */
    const uint8_t  *is_rev;    /* per row: XS:A or FLAG 0x10 (after update: annotation strand when assigned) */
    const uint32_t *exon_off;  /* n_reads+1 */
    const int32_t  *exon_start, *exon_end;
} lrb_exon_result;

/* per-read class word */
#define LRB_C_KNOWN       0x001u   /* trans_t.known */
#define LRB_C_KNOWN_SITE  0x002u   /* has_known_site */
#define LRB_C_UNRELIABLE  0x004u   /* has_unreliable_junction */
#define LRB_C_FULL        0x008u
#define LRB_C_LFULL       0x010u
#define LRB_C_RFULL       0x020u
#define LRB_C_LNOTH       0x040u
#define LRB_C_RNOTH       0x080u
#define LRB_C_SJ_CHECKED  0x100u   /* check_with_short_sj() was evaluated for this read */

/* per-exon-slot flag byte, slot j of a read (bits 1-4 only meaningful for j < exon_n-1) */
#define LRB_F_NOVEL_EXON  0x01u    /* novel_exon_flag[j] */
#define LRB_F_NOVEL_DON   0x02u    /* novel_site_flag[2j] */
#define LRB_F_NOVEL_ACC   0x04u    /* novel_site_flag[2j+1] */
#define LRB_F_NOVEL_JUNC  0x08u    /* novel_junction_flag[j] */
#define LRB_F_UNRELIABLE  0x10u    /* unreliable_junction_flag[j] */

/* summary.txt counters in file order (update_gtf.c:537-569) */
enum {
    LRB_S_ANNO_GENES = 0, LRB_S_ANNO_TRANS,
    LRB_S_UPD_GENES, LRB_S_NOVEL_TRANS, LRB_S_NOVEL_FULL, LRB_S_NOVEL_PARTIAL,
    LRB_S_NOVEL_EXONS, LRB_S_NOVEL_SITES, LRB_S_NOVEL_JUNC,
    LRB_S_KNOWN_TRANS, LRB_S_KNOWN_GENES, LRB_S_UNIQ_KNOWN,
    LRB_S_NOVEL_BAM, LRB_S_NOVEL_RELIABLE, LRB_S_UNIQ_RELIABLE, LRB_S_NOVEL_UNRELIABLE, LRB_S_UNIQ_UNRELIABLE,
    LRB_S_UNRECOG, LRB_S_UNIQ_UNRECOG,
    LRB_S_COUNT
};

/* A transcript row of novel_T / updated_T / a unique-gtf list: a whole read or
 * a split piece (split_trans update_gtf.c:837-913).  Exon slots are
 * [exon_lo, exon_lo+exon_n) of read `read` (row of the exon result). */
typedef struct {
    int64_t         n;
    const uint32_t *read;      /* row in the exon result */
    const uint32_t *exon_lo;   /* first exon slot within the read */
    const uint32_t *exon_n;
    const int32_t  *piece;     /* -1 whole read, else k of "<id>.split.<k>" */
} lrb_trans_list;

/* merge_trans() output (update_gtf.c:144-163): surviving rows of a transcript
 * list with the mutated fields (cov, T.start/T.end, exon[0].start, exon[last].end). */
typedef struct {
    int64_t         n;
    const uint32_t *cand;      /* row in the transcript list that was folded */
    const int32_t  *cov;
    const int32_t  *t_tid, *t_start, *t_end;  /* trans_t.tid/start/end (0/0/0 quirk for pieces, SURVEY Q14) */
    const int32_t  *first_start, *last_end;   /* exon[0].start, exon[n-1].end */
} lrb_merged_list;

typedef struct {               /* novel_exon.bed rows, update_gtf.c:571-576 */
    int64_t         n;
    const int32_t  *tid, *start, *end, *score;
    const uint8_t  *type;      /* 0 T, 1 I, 2 S */
    const uint8_t  *is_rev;
} lrb_bed_list;

typedef struct {               /* check_trans + print_trans_summary, update_gtf.c:936-965,421-587 */
    lrb_exon_result  ex;       /* bam_T chains, strands flipped to the annotation's where assigned */
    const uint32_t  *cls;      /* per read LRB_C_* */
    const int32_t   *ref_anno; /* ref_anno_i (-1: gene "NA") */
    const uint8_t   *exon_flag;/* per exon slot LRB_F_* (parallel to ex.exon_start) */
    int64_t          n_known;   const uint32_t *known_idx;    /* known_T rows   */
    int64_t          n_unrecog; const uint32_t *unrecog_idx;  /* unrecog_T rows */
    lrb_trans_list   novel;    /* novel_T (whole reads and split pieces, in order) */
    lrb_merged_list  updated;  /* updated_T = merge_trans fold over novel_T */
    int32_t          summary[LRB_S_COUNT]; /* anno counters [0],[1] are left 0: the host owns them */
    lrb_bed_list     bed;
} lrb_update_result;

/* Self-contained rows of a transcript list as print_read_trans() needs them
 * (gtf.c:607-632): everything the default outputs of update-gtf (-o updated GTF,
 * -y summary, -E BED) require, without the per-read tables.  Names stay on the
 * host: name_idx is the record index of the batch (or the chain index for -m g
 * input); pieces print "<name>.split.<piece>". */
typedef struct {
    int64_t         n;
    const uint32_t *name_idx;
    const int32_t  *piece;     /* -1 whole read */
    const int32_t  *t_tid, *t_start, *t_end;  /* transcript line: trans_t.tid/start/end (0/0/0 for pieces, SURVEY Q14) */
    const uint8_t  *t_rev;     /* transcript line strand (0 for pieces) */
    const int32_t  *e_tid;     /* exon lines: the read's chromosome */
    const uint8_t  *e_rev;     /* exon lines strand; also selects descending exon order */
    const int32_t  *cov;
    const int32_t  *ref_anno;  /* gene_id / gene_name source (-1: "NA") */
    const uint32_t *exon_off;  /* n+1 */
    const int32_t  *exon_start, *exon_end;    /* first start / last end already extended by the fold */
} lrb_trans_table;

typedef struct {               /* uniq_trans, unique_gtf.c:73-84 */
    lrb_exon_result  ex;
    lrb_merged_list  uniq;     /* unique_T (cand = read row) */
    int64_t          n_shared; const uint32_t *shared_idx;   /* shared_T rows (-I) */
} lrb_unique_result;

/* ------------------------------------------------------------- entry points */

typedef struct lrb_ctx lrb_ctx;

int  lrb_ctx_create(int device, lrb_ctx **out);
void lrb_ctx_destroy(lrb_ctx *ctx);
const char *lrb_last_error(const lrb_ctx *ctx);
const char *lrb_version(void);

/* Tables, replicated per device.  Replaces read_anno_trans (gtf.c:468) for the
 * annotation and the -r remove GTF (bam_filter.c:122-125), read_sj_group (gtf.c:431). */
int lrb_anno_upload(lrb_ctx *ctx, const lrb_anno *anno);
int lrb_rm_upload(lrb_ctx *ctx, const lrb_anno *rm);      /* only tid/start/end are used */
int lrb_sj_upload(lrb_ctx *ctx, const lrb_sj *sj);        /* sj==NULL or n==0: no -j */

/* Record batch -> device (async on the ctx stream; pinned source recommended). */
int lrb_batch_upload(lrb_ctx *ctx, const lrb_batch *batch);
/* Record batch -> device WITHOUT its CIGAR pool, for a batch whose pool does not fit the device (4 B per op; an ONT read carries
 * hundreds of ops).  The fixed-width columns are copied as lrb_batch_upload copies them; the context's device copy of an earlier
 * pool is freed.  The later lrb_filter_run, lrb_exon_run and lrb_pipeline_run stream the pool from batch->cigar through two
 * device staging buffers, in chunks of whole walk tiles of at most chunk_ops ops (the copy of the next chunk runs under the walk
 * of the current one); every result is the one lrb_batch_upload gives.  A tile whose own ops exceed chunk_ops (a tile is 256
 * records when the batch averages <= 48 ops per record, 32 otherwise) is staged alone, in staging grown for it.  chunk_ops == 0:
 * the library sizes the chunks from the free device memory (cudaMemGetInfo).
 * Contract: batch->cigar stays valid and unchanged until the next lrb_batch_upload / lrb_batch_attach or lrb_ctx_destroy.  Pinned
 * memory (lrb_host_alloc) lets the copies overlap the walk; pageable memory gives the same results, serialised.  lrb_bam2sj needs
 * the batch passed to it (b != NULL) after an attach.  LRB_E_ARG if chunk_ops < 0. */
int lrb_batch_attach(lrb_ctx *ctx, const lrb_batch *batch, int64_t chunk_ops);
int lrb_chains_upload(lrb_ctx *ctx, const lrb_chains *chains);   /* -m g input */

/* Device-resident stages (no host<->device copies of per-read data). */
int lrb_filter_run(lrb_ctx *ctx, const lrb_filter_params *p);                 /* bam_filter.c:130-159 */
int lrb_exon_run(lrb_ctx *ctx, const lrb_exon_params *p, int use_keep_list);  /* bam2gtf.c:89-110 / :150-156 */
int lrb_pipeline_run(lrb_ctx *ctx, const lrb_filter_params *fp, const lrb_exon_params *ep); /* fused filter + exon pass */
int lrb_update_run(lrb_ctx *ctx, const lrb_update_params *p);                 /* update_gtf.c:936-965 (+421-587) */
int lrb_unique_run(lrb_ctx *ctx, const lrb_update_params *p);                 /* unique_gtf.c:73-84 */
/* Coordinate sort of the current rows on the device (after lrb_exon_run / lrb_pipeline_run / lrb_chains_upload, before
 * lrb_update_run): replaces the external `samtools sort` between `lr2rmats filter` and `lr2rmats update-gtf`
 * (Snakefile:90); update_gtf needs (tid,start)-sorted input (update_gtf.c:41).  Stable, samtools' coordinate key
 * tid << 32 | (pos + 1) << 1 | FLAG 0x10; row r of the later results refers to record read_idx[r] of the batch. */
int lrb_rows_sort(lrb_ctx *ctx);
int lrb_sync(lrb_ctx *ctx);

/* `lr2rmats bam2sj` (bam2sj_core parse_bam.c:896-924 + gen_sj :402-442 + sj_update_group :353-380): the distinct splice
 * junctions (tid, don = first, acc = last intron base) of the batch, ordered by (tid, don, acc), with the numbers of unique-
 * (NH:i == 1: is_uniq[i] != 0) and multi-mapped records over each.  b == NULL: the batch uploaded last.  The record stream
 * must be ordered by reference id (LRB_E_UNSORTED otherwise: the reference's insertion only keeps its order then).  The
 * strand / motif columns of print_sj (:974-985) are a genome lookup per junction (intr_deri_str :319-337) left to the caller. */
int lrb_bam2sj(lrb_ctx *ctx, const lrb_batch *b, const uint8_t *is_uniq, const lrb_sj_params *p, lrb_sj *out);

/* Stable sort of n records by three unsigned keys, most significant first; *perm (pinned, owned by the ctx) = record indices
 * in sorted order.  Replaces the `sort -n -k1 -n -k2 -n -k3 -n -k4` of src/sort_gtf.sh:29 -- chromosome rank, transcript
 * start, transcript end, and the line number as the input order a stable sort keeps (Snakefile:192, the pipeline's last step). */
int lrb_sort3(lrb_ctx *ctx, const uint32_t *k0, const uint32_t *k1, const uint32_t *k2, int64_t n, const uint32_t **perm);

/* Results -> pinned host buffers owned by the ctx. */
int lrb_filter_fetch(lrb_ctx *ctx, lrb_filter_result *out);
int lrb_filter_fetch_keep(lrb_ctx *ctx, int64_t *n_keep, const uint32_t **keep_idx); /* only the records sam_write1 would emit */
int lrb_exon_fetch(lrb_ctx *ctx, lrb_exon_result *out);
int lrb_update_fetch(lrb_ctx *ctx, lrb_update_result *out);
int lrb_unique_fetch(lrb_ctx *ctx, lrb_unique_result *out);
/* updated_T as a self-contained table + BED rows + summary counters: the part of lrb_update_fetch that
 * `update-gtf -o/-y/-E` prints (print_read_trans gtf.c:607-632, update_gtf.c:535-576); any argument may be NULL. */
int lrb_update_fetch_table(lrb_ctx *ctx, lrb_trans_table *updated, lrb_bed_list *bed, int32_t summary[LRB_S_COUNT]);

/* One-call forms with HOST buffers (upload + run + fetch), the calls the
 * reference's subcommands would make where they call gtf_filter /
 * read_bam_trans / check_trans / uniq_trans today. */
int lrb_filter(lrb_ctx *ctx, const lrb_batch *b, const lrb_filter_params *p, lrb_filter_result *out);
int lrb_bam2gtf(lrb_ctx *ctx, const lrb_batch *b, const lrb_exon_params *p, lrb_exon_result *out);
int lrb_update_gtf(lrb_ctx *ctx, const lrb_batch *b, const lrb_exon_params *ep,
                   const lrb_update_params *up, lrb_update_result *out);
int lrb_unique_gtf(lrb_ctx *ctx, const lrb_batch *b, const lrb_exon_params *ep,
                   const lrb_update_params *up, lrb_unique_result *out);

/* Measurement hooks (bench.py): CUDA-event time of the last *_run call on the
 * ctx stream, per kernel family, and the number of kernels it launched. */
#define LRB_T_FILTER   0
#define LRB_T_EXON     1
#define LRB_T_CLASSIFY 2
#define LRB_T_MERGE    3
#define LRB_T_SUMMARY  4
#define LRB_T_K_SCAN   5   /* the cigar_scan kernel alone */
#define LRB_T_K_FOLD   6   /* the merge_fold kernel alone (updated_T fold) */
#define LRB_T_COUNT    7
int lrb_timing_enable(lrb_ctx *ctx, int on);
int lrb_timing_get(lrb_ctx *ctx, float ms[LRB_T_COUNT], int64_t *n_launches);
int64_t lrb_launch_count(const lrb_ctx *ctx);   /* kernels launched since ctx creation */
/* CUDA events on the ctx stream (the stream every kernel of this library is launched on): slot in [0,8) */
int lrb_mark(lrb_ctx *ctx, int slot);
int lrb_elapsed_ms(lrb_ctx *ctx, int slot_from, int slot_to, float *ms);   /* synchronises on slot_to */
/* Diagnostics of the last lrb_update_run: split pieces that were absorbed by an entry on ANOTHER chromosome (the reference's
 * back-scan of a piece never stops, update_gtf.c:148; settled in rounds on the device) and folds replayed as one locus. */
int lrb_update_diag(const lrb_ctx *ctx, int64_t *pieces_across_chromosomes, int64_t *one_locus_replays);
/* Diagnostics of the last CIGAR walk (lrb_filter_run / lrb_exon_run / lrb_pipeline_run; the repeat of a walk whose exon pool
 * was regrown counts alone): chunks of an attached batch's pool walked, and the most ops one chunk staged on the device.
 * Both 0 for a batch uploaded with its pool. */
int lrb_cigar_stream_diag(const lrb_ctx *ctx, int64_t *chunks, int64_t *max_staged_ops);
/* Fold census, a test hook: which path of the merge fold (update-gtf's updated_T and class folds, unique-gtf) folded each locus.
 * Counted only when LRB_TEST_FOLD_CENSUS is set to a non-zero number at lrb_ctx_create; each fold then reads its locus table back
 * and synchronises its stream.  Cumulative over the context's life; the repeated folds that settle split pieces absorbed on another
 * chromosome are not counted.  Per locus unless stated, by the final state of the fold:
 *   -d 0:  FLAT         <= 64 candidates, folded by the flat kernels
 *          TIER0        > 64 candidates or given up by the flat kernels, folded by the 128-slot warp replay
 *          TIER1        outgrew tier 0, folded by the 416-slot replay
 *          MERGE_OVER   outgrew tier 1, or >= 32768 candidates: replayed by merge_fold_kernel
 *          MERGE_VERIFY a class hash collision: replayed by merge_fold_kernel
 *          NOROWS       (locus, sub-stream) pairs of the warp replay with more than 127 multi-exon classes (no relation rows)
 *   -d >0: D_SMALL / D_LARGE  loci of <= 32 / >= 33 candidates
 *   both:  SINGLE       loci of folds replayed as one locus (also counted above)
 *   -d 0:  INDEXED      multi-exon candidates the warp replay decided by its class index (tabulated classes, no end tests)
 *                       instead of a back-scan; per candidate
 * Counters [0, LRB_FC_COUNT) are the folds on the main stream (updated_T, unique-gtf), [LRB_FC_COUNT, 2 * LRB_FC_COUNT) those on
 * the side stream (update-gtf's four class folds of the summary).  Writes min(n, 2 * LRB_FC_COUNT) counters to out and returns
 * 2 * LRB_FC_COUNT. */
enum { LRB_FC_FLAT, LRB_FC_TIER0, LRB_FC_TIER1, LRB_FC_MERGE_OVER, LRB_FC_MERGE_VERIFY, LRB_FC_NOROWS, LRB_FC_D_SMALL, LRB_FC_D_LARGE,
       LRB_FC_SINGLE, LRB_FC_INDEXED, LRB_FC_COUNT };
int lrb_fold_census(const lrb_ctx *ctx, int64_t *out, int n);
/* pinned host memory for record batches (what the host decoder fills) */
void *lrb_host_alloc(size_t bytes);
void lrb_host_free(void *p);

/* ---------------------------------------------------------------- multi-GPU
 * One process per GPU, one lrb_ctx per process, one NCCL communicator per ctx (SURVEY.md 8e; the reference is a single
 * thread -- its analogue is one `lr2rmats update-gtf` per chromosome shard and a `cat` of the outputs, App. B.3).
 *
 *   1. the caller cuts ONE (tid,start)-sorted read stream into locus-aligned shards (lrb_shard_cuts / _weighted);
 *   2. lrb_comm_id on one rank, the 128 bytes shipped to the others by whatever launched them, lrb_comm_init on all;
 *   3. lrb_tables_broadcast: the root's annotation / remove / SJ tables are replicated HBM -> HBM over NVLink
 *      (replaces read_anno_trans / read_sj_group on every other rank);
 *   4. every rank runs its shard (lrb_batch_upload, lrb_pipeline_run / lrb_exon_run, lrb_update_run);
 *   5. lrb_update_gather: per-shard updated_T tables, BED rows and known-gene pairs go to rank 0 (count all-gather +
 *      send/recv gatherv) and are merged canonically there: ordered concatenation, counters summed, the gene sets
 *      (Updated_Genes, Genes_of_Known...: add_simp_gene update_gtf.c:175-189,503-506 -- a gene can span two loci)
 *      recomputed / unioned over the gathered table, the piece-aware tid-0 sets (update_gtf.c:421-534, SURVEY A.8)
 *      recomputed when two shards share a tid-0 key;
 *   6. lrb_gather_fetch on rank 0: the result exactly as one GPU (and the reference) would produce it for the whole stream.
 *
 * The per-read outputs (update-gtf -a/-A/-k/-v/-u, the records `lr2rmats filter` writes) need no merge: every row is a function
 * of its read and the replicated tables, and shards never cut a qname run, so the shards' results concatenate (App. B.3):
 *   5'. lrb_update_gather_reads: per-shard bam_T chains, class words, known / unrecog / novel lists, updated_T entries and
 *       the filter's per-record results go to rank 0 (count all-gather + send/recv gatherv), which shifts their row / exon /
 *       record indices to the whole stream;
 *   6'. lrb_gather_fetch_reads on rank 0: what lrb_update_fetch / lrb_filter_fetch return on one GPU for the whole stream.
 */
#define LRB_COMM_ID_BYTES 128
int lrb_comm_id(void *id_out /* LRB_COMM_ID_BYTES */);
int lrb_comm_init(lrb_ctx *ctx, const void *id, int rank, int n_ranks);
int lrb_comm_destroy(lrb_ctx *ctx);
int lrb_comm_rank(const lrb_ctx *ctx, int *rank, int *n_ranks);
/* rank `root` passes its host tables (any may be NULL), the other ranks pass NULL; collective */
int lrb_tables_broadcast(lrb_ctx *ctx, int root, const lrb_anno *anno, const lrb_anno *rm, const lrb_sj *sj);
/* collective, after lrb_update_run on every rank.  name_base = index of this shard's first record in the whole read
 * stream (name_idx of the merged table then indexes the whole stream).  LRB_E_XSHARD: see above. */
int lrb_update_gather(lrb_ctx *ctx, int64_t name_base);
/* rank 0: merged updated_T + BED rows + summary (anno counters [0],[1] left 0); other ranks: empty.  Any argument may be NULL. */
int lrb_gather_fetch(lrb_ctx *ctx, lrb_trans_table *updated, lrb_bed_list *bed, int32_t summary[LRB_S_COUNT]);
int lrb_gather_timing(lrb_ctx *ctx, float *ms_gather, float *ms_merge);   /* CUDA-event times of the last lrb_update_gather */
/* collective, after lrb_update_run on every rank (each on its shard of ONE stream); name_base as for lrb_update_gather.
 * Does not depend on the outcome of lrb_update_gather: every rank may call it even where the root got LRB_E_XSHARD.
 * LRB_E_ARG on every rank when the gathered results exceed 2^32 exons or records. */
int lrb_update_gather_reads(lrb_ctx *ctx, int64_t name_base);
/* rank 0: what lrb_update_fetch / lrb_filter_fetch return on ONE GPU for the whole stream; other ranks: zeroed, LRB_OK.
 * Either argument may be NULL.  update: ex.read_idx is NULL when the shards were chains (lrb_chains_upload); its BED rows and
 * summary come from lrb_update_gather, which must have succeeded after the same lrb_update_run (LRB_E_ARG otherwise).  filter: LRB_E_ARG unless
 * the filter stage ran on every shard (lrb_pipeline_run / lrb_filter_run). */
int lrb_gather_fetch_reads(lrb_ctx *ctx, lrb_update_result *update, lrb_filter_result *filter);

/* Read shards are cut at locus gaps (SURVEY App. B.3: where a read starts beyond every earlier end on its chromosome the
 * outputs concatenate exactly); this helper finds n_shards-1 such cuts near the ideal boundaries on the host.
 * _weighted balances the shards by `weight` (e.g. CIGAR ops per read) instead of by read count. */
int lrb_shard_cuts(const int32_t *tid, const int32_t *start, const int32_t *end, int64_t n,
                   int n_shards, int64_t *cuts /* n_shards+1 */);
int lrb_shard_cuts_weighted(const int32_t *tid, const int32_t *start, const int32_t *end, const int64_t *weight, int64_t n,
                            int n_shards, int64_t *cuts /* n_shards+1 */);

#ifdef __cplusplus
}
#endif
#endif /* LR2RMATS_B200_H */
