/* minimap_b200.h -- the minimap2 C API surface of the AirLift fork, served by the B200 build.
 *
 * Same type layouts and function names as the reference's minimap.h (src/minimap2-master_remapping/
 * minimap.h:53-150,180-376), so a caller of mm_set_opt / mm_idx_reader_* / mm_map_file_frag / mm_map_frag
 * recompiles against this header unchanged.  Differences, all behind the API:
 *   - mm_idx_t::B no longer points at per-bucket khash tables; it holds the handle of the HBM-resident index;
 *   - mapping is batched: mm_map_file_frag() drives the GPU stages once per mini-batch instead of once
 *     per fragment, and the mm_map_frag()/mm_map() calls that are waiting at the same time, from any number of threads,
 *     are mapped together as one mini-batch;
 *   - a CUDA device is required: every entry point fails with an [ERROR] on stderr otherwise.
 */
#ifndef MINIMAP_B200_H
#define MINIMAP_B200_H
#include <stdint.h>
#include <stdio.h>
#include <sys/types.h>
#include "mmg.h"

/* mapping flags (minimap.h:8-38) */
#define MM_F_NO_DIAG       0x001
#define MM_F_NO_DUAL       0x002
#define MM_F_CIGAR         0x004
#define MM_F_OUT_SAM       0x008
#define MM_F_NO_QUAL       0x010
#define MM_F_OUT_CG        0x020
#define MM_F_OUT_CS        0x040
#define MM_F_SPLICE        0x080
#define MM_F_SPLICE_FOR    0x100
#define MM_F_SPLICE_REV    0x200
#define MM_F_NO_LJOIN      0x400
#define MM_F_OUT_CS_LONG   0x800
#define MM_F_SR            0x1000
#define MM_F_FRAG_MODE     0x2000
#define MM_F_NO_PRINT_2ND  0x4000
#define MM_F_2_IO_THREADS  0x8000
#define MM_F_LONG_CIGAR    0x10000
#define MM_F_INDEPEND_SEG  0x20000
#define MM_F_SPLICE_FLANK  0x40000
#define MM_F_SOFTCLIP      0x80000
#define MM_F_FOR_ONLY      0x100000
#define MM_F_REV_ONLY      0x200000
#define MM_F_HEAP_SORT     0x400000
#define MM_F_ALL_CHAINS    0x800000
#define MM_F_OUT_MD        0x1000000
#define MM_F_COPY_COMMENT  0x2000000
#define MM_F_EQX           0x4000000
#define MM_F_PAF_NO_HIT    0x8000000
#define MM_F_NO_END_FLT    0x10000000
#define MM_F_HARD_MLEVEL   0x20000000
#define MM_F_SAM_HIT_ONLY  0x40000000

#define MM_I_HPC      0x1
#define MM_I_NO_SEQ   0x2
#define MM_I_NO_NAME  0x4

#define MM_IDX_MAGIC  "MMI\2"
#define MM_MAX_SEG    255

#ifdef __cplusplus
extern "C" {
#endif

typedef struct { uint64_t x, y; } mm128_t;
typedef struct { size_t n, m; mm128_t *a; } mm128_v;

typedef struct { char *name; uint64_t offset; uint32_t len; } mm_idx_seq_t;

typedef struct {
	int32_t b, w, k, flag;
	uint32_t n_seq;
	int32_t index;
	mm_idx_seq_t *seq;
	uint32_t *S;                 /* 4-bit packed reference (host copy; the device holds its own) */
	struct mm_idx_bucket_s *B;   /* hidden: here, the device-side index state */
	struct mm_idx_intv_s *I;
	void *km, *h;
} mm_idx_t;

typedef struct {
	uint32_t capacity;
	int32_t dp_score, dp_max, dp_max2;
	uint32_t n_ambi:30, trans_strand:2;
	uint32_t n_cigar;
	uint32_t cigar[];
} mm_extra_t;

typedef struct {
	int32_t id, cnt, rid, score;
	int32_t qs, qe, rs, re;
	int32_t parent, subsc;
	int32_t as;
	int32_t mlen, blen;
	int32_t n_sub;
	int32_t score0;
	uint32_t mapq:8, split:2, rev:1, inv:1, sam_pri:1, proper_frag:1, pe_thru:1, seg_split:1, seg_id:8, split_inv:1, dummy:7;
	uint32_t hash;
	float div;
	mm_extra_t *p;
} mm_reg1_t;

typedef struct { short k, w, flag, bucket_bits; int mini_batch_size; uint64_t batch_size; } mm_idxopt_t;

typedef struct {
	int64_t flag;
	int seed;
	int sdust_thres;
	int max_qlen;
	int bw;
	int max_gap, max_gap_ref;
	int max_frag_len;
	int max_chain_skip, max_chain_iter;
	int min_cnt;
	int min_chain_score;
	float mask_level;
	float pri_ratio;
	int best_n;
	int max_join_long, max_join_short;
	int min_join_flank_sc;
	float min_join_flank_ratio;
	int a, b, q, e, q2, e2;
	int sc_ambi;
	int noncan;
	int junc_bonus;
	int zdrop, zdrop_inv;
	int end_bonus;
	int min_dp_max;
	int min_ksw_len;
	int anchor_ext_len, anchor_ext_shift;
	float max_clip_ratio;
	int pe_ori, pe_bonus;
	float mid_occ_frac;
	int32_t min_mid_occ;
	int32_t mid_occ;
	int32_t max_occ;
	int mini_batch_size;
	int64_t max_sw_mat;
	const char *split_prefix;
} mm_mapopt_t;

typedef struct {
	int is_idx, n_parts;
	int64_t idx_size;
	mm_idxopt_t opt;
	FILE *fp_out;
	union { struct mm_bseq_file_s *seq; FILE *idx; } fp;
} mm_idx_reader_t;

typedef struct mm_tbuf_s mm_tbuf_t;

extern int mm_verbose, mm_dbg_flag;
extern double mm_realtime0;

/* options (options.c) */
int mm_set_opt(const char *preset, mm_idxopt_t *io, mm_mapopt_t *mo);
int mm_check_opt(const mm_idxopt_t *io, const mm_mapopt_t *mo);
void mm_mapopt_update(mm_mapopt_t *opt, const mm_idx_t *mi);
void mm_mapopt_max_intron_len(mm_mapopt_t *opt, int max_intron_len);
void mm_idxopt_init(mm_idxopt_t *opt);
void mm_mapopt_init(mm_mapopt_t *opt);

/* index (index.c) */
mm_idx_reader_t *mm_idx_reader_open(const char *fn, const mm_idxopt_t *opt, const char *fn_out);
mm_idx_t *mm_idx_reader_read(mm_idx_reader_t *r, int n_threads);
void mm_idx_reader_close(mm_idx_reader_t *r);
int mm_idx_reader_eof(const mm_idx_reader_t *r);
void mm_idx_dump(FILE *fp, const mm_idx_t *mi);   /* index.c:438: byte-identical .mmi */
mm_idx_t *mm_idx_load(FILE *fp);                   /* index.c:479: one index part from a .mmi */
int64_t mm_idx_is_idx(const char *fn);
mm_idx_t *mm_idx_str(int w, int k, int is_hpc, int bucket_bits, int n, const char **seq, const char **name);
void mm_idx_stat(const mm_idx_t *idx);
void mm_idx_destroy(mm_idx_t *mi);
#ifndef MM_FN
#define MM_FN
#endif
MM_FN int mm_idx_getseq(const mm_idx_t *mi, uint32_t rid, uint32_t st, uint32_t en, uint8_t *seq);
int32_t mm_idx_cal_max_occ(const mm_idx_t *mi, float f);
int mm_idx_name2id(const mm_idx_t *mi, const char *name); /* -1 when no target has that name */

/* mapping (map.c) */
mm_tbuf_t *mm_tbuf_init(void);
void mm_tbuf_destroy(mm_tbuf_t *b);
mm_reg1_t *mm_map(const mm_idx_t *mi, int l_seq, const char *seq, int *n_regs, mm_tbuf_t *b, const mm_mapopt_t *opt, const char *name);
void mm_map_frag(const mm_idx_t *mi, int n_segs, const int *qlens, const char **seqs, int *n_regs, mm_reg1_t **regs, mm_tbuf_t *b,
                 const mm_mapopt_t *opt, const char *qname);
int mm_map_file(const mm_idx_t *idx, const char *fn, const mm_mapopt_t *opt, int n_threads);
int mm_map_file_frag(const mm_idx_t *idx, int n_segs, const char **fn, const mm_mapopt_t *opt, int n_threads);

/* cs / MD of a hit (format.c, mm_gen_cs / mm_gen_MD), the string alone: *buf is realloc'd to *max_len bytes and the length
 * is returned; seq is the query as mapped; km is not used.  The PAF/SAM writers print the same strings. */
int mm_gen_cs(void *km, char **buf, int *max_len, const mm_idx_t *mi, const mm_reg1_t *r, const char *seq, int no_iden);
int mm_gen_MD(void *km, char **buf, int *max_len, const mm_idx_t *mi, const mm_reg1_t *r, const char *seq);

/* FASTA/FASTQ (gzip'd or not) one record at a time, as the mapper reads it (bseq.c): mm_fastx_read returns the sequence
 * length, or -1 at the end; the strings (qual and comment may be 0) stay valid until the next call */
typedef struct mm_fastx_s mm_fastx_t;
mm_fastx_t *mm_fastx_open(const char *fn, int with_comment);
int mm_fastx_read(mm_fastx_t *r, const char **name, const char **seq, const char **qual, const char **comment);
void mm_fastx_close(mm_fastx_t *r);

/* B200 additions */
int mm_b200_set_devices(int n_gpus, const int *dev_ids); /* before building the index; default: device 0 */
/* one process per GPU: rank 0 builds the index, exports its flat device image (mm_b200_idx_image), the other ranks allocate
 * the same shape (mm_b200_idx_alloc), a collective fills the five buffers, mm_b200_idx_finalize completes the replica */
int mm_b200_idx_image(const mm_idx_t *mi, mmg_idx_image_t *img);
mm_idx_t *mm_b200_idx_alloc(const char *fasta, const mm_idxopt_t *opt, const mmg_idx_image_t *shape, mmg_idx_image_t *ptrs);
mm_idx_t *mm_b200_idx_alloc_named(const mm_idxopt_t *opt, int n_seq, const char *const *names, const uint32_t *lens,
                                  const mmg_idx_image_t *shape, mmg_idx_image_t *ptrs); /* same, without re-reading the FASTA */
int mm_b200_idx_seq(const mm_idx_t *mi, int i, const char **name, uint32_t *len);
int mm_b200_idx_finalize(mm_idx_t *mi);
/* options this build does not implement (splice, -D/-X/--dual=no, -T, --split-prefix) are refused, never ignored: 0 if
 * opt can be mapped with, else -1 after an [ERROR] line.  MM_F_INDEPEND_SEG (--no-pairing) maps the two reads of a pair
 * one by one in mm_map_file_frag() and mm_b200_map_batch(es); mm_map_frag() maps the segments it is given jointly, as the
 * reference does.  mm_map_frag()/mm_map() may be called from any number of threads at once, each with its own mm_tbuf_t:
 * one dispatcher thread per index (started by the first call, joined by mm_idx_destroy) maps the calls that are waiting
 * with equal options as shared mini-batches on every GPU of the index, and a lone caller is never held back to fill one.
 * Calling them while mm_b200_map_batch(es) or mm_map_file(_frag) maps on the same index is not supported. */
int mm_b200_check_opt(const mm_mapopt_t *opt);
const char *mm_b200_opt_error(const mm_mapopt_t *opt); /* the message mm_b200_check_opt prints (no "[ERROR] "), or 0: nothing printed */
/* An index loaded from a .mmi written with --idx-no-seq keeps no sequence (mi->S is null): it maps, but CIGARs (-a, -c, --cs,
 * --MD: MM_F_CIGAR) cannot be computed against it.  mm_b200_seq_error returns the message for that case, or 0; the mapping calls
 * refuse it as they refuse mm_b200_check_opt's options (the batch calls return -1, mm_map_frag exits) */
const char *mm_b200_seq_error(const mm_idx_t *mi, const mm_mapopt_t *opt);
/* the minimizer lists of the first part of a no-sequence .mmi, as its loader hands them to mmg_idx_build_lists (see mmg.h);
 * returns the number of distinct minimizers, or -1 with the loader's message printed */
int64_t mm_b200_mmi_lists(const char *fn, uint64_t **key, uint32_t **cnt, uint64_t **src, uint64_t *n_p, uint64_t **p);
void mm_b200_mmi_lists_free(uint64_t *key, uint32_t *cnt, uint64_t *src, uint64_t *p);
/* name keys of the self/dual-hit filters (see "name keys" in mmg.h): sorted[] receives the n names in strcmp order (a NULL name
 * counts as ""), tkey[] the target key of each; mm_b200_name_ukey gives the unit key of qname against those sorted names
 * (MMG_NAME_NONE for a NULL qname) */
void mm_b200_name_order(int n, const char *const *names, const char **sorted, uint32_t *tkey);
uint32_t mm_b200_name_ukey(int n, const char *const *sorted, const char *qname);
/* host seconds spent on unit keys by the mappers since the last reset (summed over shards) */
double mm_b200_name_key_time(int reset);
int mm_b200_set_lanes(int lanes); /* streams (with their arenas) per GPU, 1..8; before building the index */

/* Batch interface = the drop-in cut point of SURVEY.md §8b (worker_pipeline step 1, map.c:590-593): a mini-batch of
 * fragments with HOST buffers in, malloc'd mm_reg1_t arrays out.  mode 0 maps (upload + all stages); modes 1 / 2 split
 * that into "stage the reads in HBM" and "map the resident batch" so that device-resident throughput can be timed. */
typedef struct mm_b200_reader_s mm_b200_reader_t;
typedef struct mm_b200_batch_s mm_b200_batch_t;
mm_b200_reader_t *mm_b200_open_reads(int n_fp, const char **fn);
void mm_b200_close_reads(mm_b200_reader_t *r);
mm_b200_batch_t *mm_b200_read_batch(mm_b200_reader_t *r, const mm_mapopt_t *opt, int batch_bases);
void mm_b200_batch_info(const mm_b200_batch_t *b, int *n_seq, int *n_frag, int64_t *n_bases);
int  mm_b200_map_batch(const mm_idx_t *mi, const mm_mapopt_t *opt, int n_threads, mm_b200_batch_t *b, int mode);
void mm_b200_reset_batch(mm_b200_batch_t *b);
uint64_t mm_b200_batch_digest(const mm_b200_batch_t *b, int64_t *n_hits);
/* columns of a row of mm_b200_batch_hits: read (index in the batch), rid, rs, re, qs, qe, rev, mapq, score, primary (parent == id),
 * sam_pri, proper_frag, mlen, blen, dp_score, dp_max, n_cigar */
#define MM_B200_HIT_COLS 17
/* the hits of a mapped batch: one row per hit into rows (n_hits x MM_B200_HIT_COLS) and the CIGARs of all hits, concatenated,
 * into cigar; either may be 0 to only count.  Returns the number of hits; *n_cigar receives the number of CIGAR words. */
int64_t mm_b200_batch_hits(const mm_b200_batch_t *b, int64_t *rows, uint32_t *cigar, int64_t *n_cigar);
void mm_b200_write_batch(const mm_idx_t *mi, const mm_mapopt_t *opt, mm_b200_batch_t *b); /* prints and frees */
void mm_b200_free_batch(mm_b200_batch_t *b);
/* n mini-batches through mm_b200_map_batch with two of them in flight (needs an even number of lanes >= 2): batch i uses lane
 * group i % 2 of every GPU, so one batch's upload, serial tails and host finish run under the other's kernels */
int  mm_b200_set_in_flight(int n); /* mini-batches mm_b200_map_batches keeps in flight (default 2); must divide the number of lanes */
int  mm_b200_batches_in_flight(const mm_idx_t *mi, const mm_mapopt_t *opt); /* what mm_b200_map_batches overlaps for these options */
int  mm_b200_map_batches(const mm_idx_t *mi, const mm_mapopt_t *opt, int n_threads, mm_b200_batch_t **b, int n, int mode);
int  mm_b200_n_devices(const mm_idx_t *mi);

/* Hits for bindings that do not mirror mm_reg1_t (airlift_b200/mappy.py): one malloc'd block, released with mm_b200_hits_free,
 * holding n_hits rows of MM_B200_HITS_COLS integers, the CIGAR words of every hit in row order, and the cs (short form) / MD
 * strings asked for, each NUL-terminated.  Columns: frag, seg_id, rid, rs, re, qs, qe, rev, mapq, primary (id == parent), mlen,
 * blen, n_ambi, trans_strand, dp_score, dp_max, n_cigar, cigar_off, cs_off, cs_len, md_off, md_len (string offsets: -1 when
 * not made). */
#define MM_B200_HITS_COLS 22
#define MM_B200_HITS_CS   0x1
#define MM_B200_HITS_MD   0x2
typedef struct { int64_t n_hits, n_cigar, n_str; const int64_t *rows; const uint32_t *cigar; const char *str; } mm_b200_hits_t;
/* one fragment of one or two reads through mm_map_frag (any thread): the second read is given as sequenced, mapped as its reverse
 * complement, and its hits are reported in its own orientation, as the PAF writer prints a pair */
mm_b200_hits_t *mm_b200_map_hits(const mm_idx_t *mi, const mm_mapopt_t *opt, int n_segs, const int *qlens, const char **seqs,
                                 const char *qname, int flags);
mm_b200_hits_t *mm_b200_batch_hits_flat(const mm_idx_t *mi, const mm_b200_batch_t *b, int flags); /* of a mapped batch */
void mm_b200_hits_free(mm_b200_hits_t *h);
/* a batch of n_frag fragments from memory, for mm_b200_map_batch(es): fragment f has n_segs[f] reads, the next ones of
 * qlens / seqs, named names[f] (names may be 0) */
mm_b200_batch_t *mm_b200_make_batch(int n_frag, const int *n_segs, const int *qlens, const char *const *seqs, const char *const *names);
void mm_b200_path_counts(const mm_idx_t *mi, uint64_t out[8], int reset); /* see mmg_path_counts (mmg.h) */

typedef struct { /* accumulated over mm_b200_map_batch / mm_map_file_frag calls; seconds and counts */
	double t_total, t_upload, t_seedchain, t_seedchain_kernels, t_hits, t_align_host, t_ksw_total, t_ksw_kernel, t_finish;
	uint64_t n_frag, n_reads, n_bases, n_minimizers, n_anchors, n_chain_iter, n_dp_jobs, n_dp_cells, n_dp_rounds, h2d_bytes, d2h_bytes, n_dp_jobs_fast, n_dp_cells_fast;
} mm_b200_stats_t;
void mm_b200_stats(mm_b200_stats_t *out, int reset);
void mm_b200_set_serial(int on);                        /* shards of a GPU take turns on the device (clean per-kernel timing) */
void mm_b200_profile(const mm_idx_t *mi, int enable);   /* CUDA-event timing of every kernel launch */
int  mm_b200_profile_fetch(const mm_idx_t *mi, int max, const char **names, double *ms, long *launches);
void mm_b200_report(const mm_idx_t *mi, FILE *fp);
long mm_b200_launch_count(const mm_idx_t *mi, int reset); /* kernels launched on all streams of all GPUs */
void mm_write_sam_hdr(const mm_idx_t *mi, const char *rg, const char *ver, int argc, char *argv[]);

#ifdef __cplusplus
}
#endif
#endif
