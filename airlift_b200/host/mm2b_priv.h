/* mm2b_priv.h -- host-side internals of the B200 mapper (counterpart of the reference's mmpriv.h). */
#ifndef MM2B_PRIV_H
#define MM2B_PRIV_H
#include <stdlib.h>
#include <string.h>
#include <assert.h>
#include <pthread.h>
/* hits.c, aln.c and llsw.c are also compiled for the device (csrc/mmg_post.cu includes this header and them inside a
 * namespace with MM_DEVICE_BUILD defined and MM_FN = __device__), so that the GPU runs the very same bookkeeping code */
#ifndef MM_FN
#define MM_FN
#endif
#include "minimap_b200.h"
#include "mmg.h"

#define MM_VERSION_B200 "2.17-r954-b200"


#define MM_PARENT_UNSET   (-1)
#define MM_PARENT_TMP_PRI (-2)

#define MM_DBG_NO_KALLOC     0x1
#define MM_DBG_PRINT_QNAME   0x2
#define MM_DBG_PRINT_SEED    0x4
#define MM_DBG_PRINT_ALN_SEQ 0x8

#define MM_SEED_LONG_JOIN  (1ULL<<40)
#define MM_SEED_IGNORE     (1ULL<<41)
#define MM_SEED_TANDEM     (1ULL<<42)
#define MM_SEED_SELF       (1ULL<<43)
#define MM_SEED_SEG_SHIFT  48
#define MM_SEED_SEG_MASK   (0xffULL<<(MM_SEED_SEG_SHIFT))

#define KSW_NEG_INF (-0x40000000)
#define KSW_EZ_SCORE_ONLY  0x01
#define KSW_EZ_RIGHT       0x02
#define KSW_EZ_APPROX_MAX  0x08
#define KSW_EZ_EXTZ_ONLY   0x40
#define KSW_EZ_REV_CIGAR   0x80

MM_FN static inline uint32_t mm_roundup32(uint32_t x) { --x; x |= x >> 1; x |= x >> 2; x |= x >> 4; x |= x >> 8; x |= x >> 16; return ++x; }
#define mm_seq4_get(s, i) ((s)[(i)>>3] >> (((i)&7)<<2) & 0xf)

typedef struct { unsigned l, m; char *s; } mm_str_t;

/* one sequence record (bseq.h:14-17) */
typedef struct { int l_seq, rid; char *name, *seq, *qual, *comment; } mm_bseq1_t;
typedef struct mm_bseq_file_s mm_bseq_file_t;

/* per-segment chains after mm_seg_gen (mmpriv.h:46-50) */
typedef struct { int n_u, n_a; uint64_t *u; mm128_t *a; } mm_seg_t;

/* hidden part of mm_idx_t */
#define MM_B200_MAX_LANES 8  /* a batch is cut in `lanes` shards per GPU (own stream each) so that one shard's host work overlaps another's kernels */
struct mm_idx_bucket_s {
	int n_dev, lanes;
	int dev_id[16];
	mmg_ctx_t *ctx[16 * MM_B200_MAX_LANES]; /* ctx[d * lanes + lane]: own stream and arenas, same device */
	mmg_idx_t *didx[16];
	struct { const void *batch; int f0, f1; } staged[16 * MM_B200_MAX_LANES][MMG_STAGE_SLOTS]; /* which shard the ctx's staging slots hold */
	pthread_mutex_t up_token[16];  /* device path: the shards of a GPU stage their reads one after the other */
	pthread_mutex_t gpu_token[16]; /* with lanes > 1: one shard per GPU runs device stages at a time, the others do their host stages */
	int32_t max_occ_cache_set; float max_occ_cache_f; int32_t max_occ_cache;
	pthread_mutex_t apiq_mu;  /* guards the lazy start of apiq */
	struct mm_apiq_s *apiq;   /* mm_map_frag()/mm_map(): request queue and its dispatcher thread (apiq.c); 0 until the first call */
	pthread_mutex_t key_mu; /* guards the lazy set-up of the name keys */
	const char **sorted_names; /* the target names in strcmp order, once the name keys were made (namekey.c) */
};

extern unsigned char seq_nt4_table[256];
extern unsigned char seq_comp_table[256];

/* misc.c: shard-lifetime bump arena.  Everything whose lifetime ends with the mini-batch shard (work arrays, per-mate
 * anchor copies, the DP job cache, temporaries) is carved from recycled 256 KB blocks; the stage functions select the
 * shard's arena through a thread-local pointer.  API-visible blocks (mm_reg1_t arrays, mm_extra_t) stay on malloc because
 * callers free() them. */
#define MM_ARENA_MAX_PARTIAL 64
typedef struct mm_ablock_s { struct mm_ablock_s *next; size_t cap; } mm_ablock_t;
typedef struct {
	mm_ablock_t *blocks;      /* every block handed out for this arena */
	pthread_mutex_t mu;
	uint64_t gen;             /* changes on release, so a stale thread-local bump pointer is never reused */
	int n_partial;
	struct { char *cur, *end; } partial[MM_ARENA_MAX_PARTIAL]; /* blocks that exited workers left half full */
} mm_arena_t;
extern __thread mm_arena_t *mm_tls_arena;
void mm_arena_init(mm_arena_t *a);
MM_FN void *mm_amalloc(size_t n);
MM_FN void *mm_acalloc(size_t n, size_t sz);
MM_FN void *mm_arealloc(void *p, size_t old_bytes, size_t new_bytes);
MM_FN void mm_afree(void *p);
void mm_arena_thread_done(void);
void mm_arena_release(mm_arena_t *a);
void mm_b200_tune_malloc(void);


/* The reference sorts with klib's in-place MSD byte radix sort (insertion sort at <= 64 elements).  Where equal
 * keys can meet, the order they end up in is observable downstream (SURVEY.md H1), so the same permutation
 * is performed here: count, then cycle elements into their buckets starting from the lowest non-empty one.
 * TABLES declares cnt[256], hd[256], tl[256] (on the stack for the host, from the arena for the device). */
#define RS_SMALL 64
#define RS_TABLES_STACK(T) size_t cnt[256]; T *hd[256], *tl[256];
#define RS_TABLES_ARENA(T) size_t *cnt = (size_t*)mm_amalloc(256 * sizeof(size_t)); T **hd = (T**)mm_amalloc(256 * sizeof(T*)), **tl = (T**)mm_amalloc(256 * sizeof(T*));

#define RADIX_IMPL(NAME, T, KEY, TABLES) \
MM_FN static void NAME##_ins(T *b, T *e) \
{ \
	T *i, *j; \
	for (i = b + 1; i < e; ++i) { \
		if (!(KEY(*i) < KEY(*(i - 1)))) continue; \
		T t = *i; \
		for (j = i; j > b && KEY(t) < KEY(*(j - 1)); --j) *j = *(j - 1); \
		*j = t; \
	} \
} \
MM_FN static void NAME##_lvl(T *b, T *e, int sh) \
{ \
	TABLES(T) T *i; int d; \
	memset(cnt, 0, 256 * sizeof(size_t)); \
	for (i = b; i != e; ++i) ++cnt[(KEY(*i) >> sh) & 0xff]; \
	for (d = 0, i = b; d < 256; ++d) hd[d] = i, i += cnt[d], tl[d] = i; \
	for (d = 0; d < 256;) { \
		int to; \
		if (hd[d] == tl[d]) { ++d; continue; } \
		to = (int)((KEY(*hd[d]) >> sh) & 0xff); \
		if (to == d) { ++hd[d]; continue; } \
		{ T carry = *hd[d], sw; \
		  do { sw = carry; carry = *hd[to]; *hd[to]++ = sw; to = (int)((KEY(carry) >> sh) & 0xff); } while (to != d); \
		  *hd[d]++ = carry; } \
	} \
	if (sh == 0) return; \
	sh = sh > 8 ? sh - 8 : 0; \
	for (d = 0, i = b; d < 256; i = tl[d], ++d) { \
		if (tl[d] - i > RS_SMALL) NAME##_lvl(i, tl[d], sh); \
		else if (tl[d] - i > 1) NAME##_ins(i, tl[d]); \
	} \
} \
MM_FN void NAME(T *beg, T *end) \
{ \
	if (end - beg <= RS_SMALL) NAME##_ins(beg, end); \
	else NAME##_lvl(beg, end, 56); \
}
#define RS_KEY_X(v) ((v).x)
#define RS_KEY_ID(v) (v)

/* misc.c */
double cputime(void);
double realtime(void);
long peakrss(void);
void mm_err_puts(const char *str);
MM_FN void radix_sort_128x(mm128_t *beg, mm128_t *end);
MM_FN void radix_sort_64(uint64_t *beg, uint64_t *end);

/* seqio.c */
mm_bseq_file_t *mm_bseq_open(const char *fn);
void mm_bseq_close(mm_bseq_file_t *fp);
mm_bseq1_t *mm_bseq_read3(mm_bseq_file_t *fp, int chunk_size, int with_qual, int with_comment, int frag_mode, int *n_);
mm_bseq1_t *mm_bseq_read_frag2(int n_fp, mm_bseq_file_t **fp, int chunk_size, int with_qual, int with_comment, int *n_);
int mm_bseq_eof(mm_bseq_file_t *fp);
void mm_bseq_set_readahead(mm_bseq_file_t *fp, int packed);
void mm_bseq_free1(mm_bseq1_t *s, int packed);
int mm_qname_len(const char *s);
int mm_qname_same(const char *s1, const char *s2);
void mm_revcomp_bseq(mm_bseq1_t *s);
int mm_bseq_pack1(mm_bseq1_t *s, const char *name, const char *seq, int l_seq);

/* hits.c */
#ifndef MM_DEVICE_BUILD
uint32_t mm_frag_hash(const char *qname, int qlen_sum, int seed);
#endif
MM_FN mm_reg1_t *mm_gen_regs(uint32_t hash, int qlen, int n_u, uint64_t *u, mm128_t *a);
MM_FN void mm_split_reg(mm_reg1_t *r, mm_reg1_t *r2, int n, int qlen, mm128_t *a);
MM_FN void mm_sync_regs(int n_regs, mm_reg1_t *regs);
MM_FN int mm_squeeze_a(int n_regs, mm_reg1_t *regs, mm128_t *a);
MM_FN int mm_set_sam_pri(int n, mm_reg1_t *r);
MM_FN void mm_set_parent(float mask_level, int n, mm_reg1_t *r, int sub_diff, int hard_mask_level);
MM_FN void mm_select_sub(float pri_ratio, int min_diff, int best_n, int *n_, mm_reg1_t *r);
MM_FN void mm_select_sub_multi(float pri_ratio, float pri1, float pri2, int max_gap_ref, int min_diff, int best_n, int n_segs, const int *qlens, int *n_, mm_reg1_t *r);
MM_FN void mm_filter_regs(const mm_mapopt_t *opt, int qlen, int *n_regs, mm_reg1_t *regs);
MM_FN void mm_join_long(const mm_mapopt_t *opt, int qlen, int *n_regs, mm_reg1_t *regs, mm128_t *a);
MM_FN void mm_hit_sort(int *n_regs, mm_reg1_t *r);
void mm_set_mapq(int n_regs, mm_reg1_t *regs, int min_chain_sc, int match_sc, int rep_len, int is_sr);
void mm_est_err(const mm_idx_t *mi, int qlen, int n_regs, mm_reg1_t *regs, const mm128_t *a, int32_t n, const uint64_t *mini_pos);
MM_FN mm_seg_t *mm_seg_gen(uint32_t hash, int n_segs, const int *qlens, int n_regs0, const mm_reg1_t *regs0, int *n_regs, mm_reg1_t **regs, const mm128_t *a);
MM_FN void mm_seg_free(int n_segs, mm_seg_t *segs);
void mm_pair(int max_gap_ref, int dp_bonus, int sub_diff, int match_sc, const int *qlens, int *n_regs, mm_reg1_t **regs);

/* llsw.c: local alignment score used by the inversion test (ksw_ll_qinit + ksw_ll_i16, ksw2_ll_sse.c) */
MM_FN int mm_ll_i16(int qlen, const uint8_t *query, int tlen, const uint8_t *target, int m, const int8_t *mat, int gapo, int gape, int *qe, int *te);

/* aln.c: resumable alignment of one segment's regions; DP goes through a job cache */
typedef struct {
	mmg_ksw_job_t job;
	mmg_extz_t ez;
	uint32_t *cigar;   /* owned */
	int done;
} mm_dpjob_t;

typedef struct {
	int n, m, n_sent;  /* jobs [n_sent, n) have not been submitted yet */
	mm_dpjob_t *a;
} mm_dpcache_t;

typedef struct { int rev, rid, rs, qs, len, score, zdrop_code; } mm_fillmemo_t; /* ungapped stretch already scored */

typedef struct {       /* alignment progress of one segment (mm_align_skeleton, align.c:857-913, made resumable) */
	int seq_id, qlen, n_regs, i, n_a, started, finished, inv_wait, planned;
	const char *qstr;
	const uint32_t *q4; uint64_t q4_off; /* device build: the read as 4-bit codes in the resident batch (instead of qstr) */
	uint8_t *qseq0[2];
	mm_reg1_t *regs;
	mm128_t *a;
	mm_dpcache_t cache;
	int n_fill, m_fill;
	mm_fillmemo_t *fill;
} mm_alnseg_t;

MM_FN void mm_aln_begin(mm_alnseg_t *s, int seq_id, int qlen, const char *qstr, int n_regs, mm_reg1_t *regs, mm128_t *a);
/* returns 1 when every region is aligned (regs/n_regs final, filtered and sorted), 0 when new DP jobs were queued */
MM_FN int mm_aln_step(mm_alnseg_t *s, const mm_mapopt_t *opt, const mm_idx_t *mi);
MM_FN void mm_aln_end(mm_alnseg_t *s);

/* fmt.c */
void mm_write_paf3(mm_str_t *s, const mm_idx_t *mi, const mm_bseq1_t *t, const mm_reg1_t *r, int opt_flag, int rep_len);
void mm_write_sam3(mm_str_t *s, const mm_idx_t *mi, const mm_bseq1_t *t, int seg_idx, int reg_idx, int n_seg, const int *n_regss,
                   const mm_reg1_t *const* regss, int opt_flag, int rep_len);

/* namekey.c: name keys of the self/dual-hit filters (include/mmg.h) */
int mm_b200_name_keys_ready(const mm_idx_t *mi);  /* target keys on every device replica (first call computes them); 0 or -1 */
uint32_t mm_b200_unit_key(const mm_idx_t *mi, const char *qname); /* after mm_b200_name_keys_ready */

/* mapper.c */
mmg_ctx_t *mm_b200_ctx(const mm_idx_t *mi, int dev_slot);
mmg_idx_t *mm_b200_didx(const mm_idx_t *mi, int dev); /* the device index on GPU dev of the index */
void mm_mapopt_to_dev(const mm_mapopt_t *opt, mmg_mapopt_t *d);

/* a mini-batch of fragments (the reference's step_t, map.c:449-456, minus the per-thread buffers); mm_b200_batch_t is one */
typedef struct {
	int n_seq, n_frag;
	mm_bseq1_t *seq;
	int *n_reg, *seg_off, *n_seg, *rep_len, *frag_gap;
	mm_reg1_t **reg;
	long order; /* position in the input (file driver: batches of two mappers leave in this order) */
} step_t;

/* apiq.c: mm_map_frag() callers of any number of threads enqueue requests; one dispatcher thread per index maps what is
 * queued when it comes round, as up to two mini-batches through `map`, and hands every caller its own hits */
typedef struct { const mm_idx_t *mi; const mm_mapopt_t *opt; int n_threads; } mm_apiq_round_t; /* what `map` receives as its first argument */
typedef int (*mm_apiq_map_f)(void *round, step_t **b, int n);               /* 0, or -1 when mapping failed */
typedef int (*mm_apiq_in_flight_f)(const mm_idx_t *mi, const mm_mapopt_t *opt); /* batches `map` overlaps for these options */
/* maps one fragment; the first call on an index starts its dispatcher with `map` and `in_flight` */
void mm_apiq_map_frag(const mm_idx_t *mi, mm_apiq_map_f map, mm_apiq_in_flight_f in_flight, const mm_mapopt_t *opt, int n_segs,
                      const int *qlens, const char **seqs, const char *qname, int *n_regs, mm_reg1_t **regs, int *rep_len, int *frag_gap);
void mm_apiq_stop(struct mm_idx_bucket_s *B); /* maps what is queued, then stops and joins the dispatcher */

#endif
