/* mmg.h -- C-ABI of the B200 device layer for the AirLift/minimap2 re-alignment hot path.
 *
 * Plain C: opaque handles, pointers and sizes only.  Every function returns 0 on success or
 * a negative MMG_E* code; mmg_last_error() describes the last failure on the calling thread.
 * There is no CPU fallback anywhere behind this interface: without a CUDA device
 * mmg_init() fails with MMG_ENODEV and nothing else can be called.
 *
 * Reference interfaces replaced (paths relative to src/minimap2-master_remapping/):
 *   mmg_sketch        <- mm_sketch                    mmpriv.h:60   sketch.c:77
 *   mmg_idx_build     <- mm_idx_str / mm_idx_gen      minimap.h:274 index.c:385,353
 *   mmg_idx_get       <- mm_idx_get                   mmpriv.h:70   index.c:81
 *   mmg_idx_cal_max_occ <- mm_idx_cal_max_occ         mmpriv.h:71   index.c:164
 *   mmg_collect_seeds <- collect_seed_hits(_heap)     map.c:149,215
 *   mmg_chain_dp      <- mm_chain_dp                  mmpriv.h:72   chain.c:22
 *   mmg_ksw_extd2     <- ksw_extd2_sse                ksw2.h:60     ksw2_extd2_sse.c:19
 *   mmg_seed_chain_batch / mmg_ksw_batch are the batched forms the mapper (mm_map_frag,
 *   map.c:272) drives: one call per mini-batch stage instead of one call per fragment.
 */
#ifndef MMG_H
#define MMG_H
#include <stdint.h>
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MMG_OK       0
#define MMG_ENODEV  (-1)  /* no usable CUDA device */
#define MMG_ECUDA   (-2)  /* a CUDA call or kernel failed */
#define MMG_EINVAL  (-3)  /* bad argument */
#define MMG_ENOMEM  (-4)
#define MMG_ELIMIT  (-5)  /* a documented device-side limit was exceeded (e.g. w > 64) */

typedef struct { uint64_t x, y; } mmg128_t;       /* == mm128_t (minimap.h:53) */
typedef struct mmg_ctx_s mmg_ctx_t;               /* one per GPU: stream, scratch arenas */
typedef struct mmg_idx_s mmg_idx_t;               /* device-resident minimizer index */

const char *mmg_last_error(void);
int  mmg_device_count(void);
int  mmg_init(int device, mmg_ctx_t **ctx);
void mmg_destroy(mmg_ctx_t *ctx);
int  mmg_device(const mmg_ctx_t *ctx);
void *mmg_stream(const mmg_ctx_t *ctx);           /* the cudaStream_t every launch of this ctx uses */
/* kernels launched by this context since the last call (for bench.py's gpu_launches) */
long mmg_launch_count(mmg_ctx_t *ctx, int reset);
/* bytes copied host->device / device->host on the ctx stream since the last reset */
void mmg_copy_bytes(mmg_ctx_t *ctx, uint64_t *h2d, uint64_t *d2h, int reset);
/* per-kernel device time (CUDA events around every launch of this ctx); names[] receives static strings */
void mmg_profile_enable(mmg_ctx_t *ctx, int on);
int  mmg_profile_fetch(mmg_ctx_t *ctx, int max, const char **names, double *ms, long *launches);
/* work items that took each data-dependent path since the last reset: out[0] fragments re-chained with max_occ (map.c:353-375),
 * [1] fragments whose seed-merge order was replayed on ranks, [2] ... literally, [3] fragments whose hit tree was built by a warp,
 * [4] extra DP rounds after z-drop cuts, [5] hits cut at a z-drop, [6] seed hits whose merge order was replayed (pops of [1]),
 * [7] seed hits dropped by the self/dual filters (-D, --dual=no; see "name keys" below) */
void mmg_path_counts(mmg_ctx_t *ctx, uint64_t out[8], int reset);
/* process-wide: how often a device ([0]) or pinned host ([1]) buffer of any ctx was re-allocated since the last reset; a
 * re-allocation synchronises the whole device, so a steady state should show none */
void mmg_growth_counts(uint64_t out[2], int reset);

/* ------------------------------------------------------------------ index */
/* Build the index on the device from n_seq ASCII sequences (not NUL-terminated; lens[] given).
 * Positions returned per minimizer are identical, in value and order, to mm_idx_get's. */
int  mmg_idx_build(mmg_ctx_t *ctx, int w, int k, int is_hpc, int n_seq, const char *const *seqs, const uint32_t *lens,
                   mmg_idx_t **idx);
void mmg_idx_free(mmg_idx_t *idx);
int64_t mmg_idx_n_minimizers(const mmg_idx_t *idx);   /* occurrences */
int64_t mmg_idx_n_keys(const mmg_idx_t *idx);         /* distinct minimizers */
uint64_t mmg_idx_total_len(const mmg_idx_t *idx);
size_t mmg_idx_bytes(const mmg_idx_t *idx);           /* HBM footprint */
/* copy the 4-bit packed reference (mm_idx_t::S layout, mmpriv.h:28-29) to the host: (total_len+7)/8 words */
int  mmg_idx_copy_S(const mmg_idx_t *idx, uint32_t *S_host);
int  mmg_idx_cal_max_occ(mmg_idx_t *idx, float f, int32_t *thres);
/* batched mm_idx_get: for each minier[i] write n[i] and up to max_pos positions at pos + i*max_pos */
int  mmg_idx_get(mmg_ctx_t *ctx, const mmg_idx_t *idx, int n_q, const uint64_t *minier, int32_t *n, int max_pos, uint64_t *pos);
/* flat device image for replication to other GPUs (one NCCL broadcast per buffer) */
typedef struct {
	int32_t w, k, is_hpc, n_seq;
	uint64_t total_len, n_slots, n_pos;
	void *d_S, *d_seq_off, *d_seq_len, *d_slots, *d_pos;  /* device pointers */
	size_t bytes_S, bytes_seq_off, bytes_seq_len, bytes_slots, bytes_pos;
	int64_t n_keys;
} mmg_idx_image_t;
int  mmg_idx_export(const mmg_idx_t *idx, mmg_idx_image_t *img);
/* allocate an empty index of the same shape on ctx's device; fill img->d_* with its pointers */
int  mmg_idx_alloc_like(mmg_ctx_t *ctx, mmg_idx_image_t *img, mmg_idx_t **idx);
/* replicate src (on its device) into a new index on ctx's device with a peer/NVLink copy */
int  mmg_idx_clone_to(mmg_ctx_t *ctx, const mmg_idx_t *src, mmg_idx_t **dst);
/* after the buffers of an mmg_idx_alloc_like() index were filled (e.g. by an NCCL broadcast) */
int  mmg_idx_finalize(mmg_idx_t *idx);
int64_t mmg_idx_n_singletons(const mmg_idx_t *idx);
/* every distinct minimizer in the order the reference's index file keeps them (mm_idx_dump, index.c:438-477, after
 * worker_post, index.c:191-243): by bucket = minimizer & ((1<<b)-1), then by minimizer>>b.  keys[i] = minimizer, bit 63
 * set when it occurs once; vals[i] = that one position, or first<<32|n with `first` indexing pos[].  pos (may be NULL)
 * receives all mmg_idx_n_minimizers() positions grouped by minimizer, ascending within a group (index.c:230).
 * keys/vals hold mmg_idx_n_keys() entries (host memory). */
int  mmg_idx_export_sorted(mmg_ctx_t *ctx, const mmg_idx_t *idx, int b, uint64_t *keys, uint64_t *vals, uint64_t *pos);
int  mmg_memcpy_d2d(void *dst, const void *src, size_t bytes);

/* Name keys.  The self/dual-hit filters of the all-vs-all modes (MM_F_NO_DIAG / MM_F_NO_DUAL, skip_seed at map.c:125-147) need
 * the sign of strcmp(qname, tname) for the mapping unit's name qname (a fragment's first read, or one read under --no-pairing)
 * and the target's name tname.  Names never reach the device; the host sorts the n_seq target names with strcmp (a missing
 * name counts as "") and sends two kinds of integers instead:
 *   target key  tkey[rid] = 2 * #{targets whose name < name(rid)} + 1           (equal names: equal keys)
 *   unit key    ukey      = 2 * #{targets whose name < qname} + (1 if some target is named qname, else 0)
 * so that ukey == tkey[rid] means cmp == 0, tkey[rid] < ukey means cmp > 0 and tkey[rid] > ukey means cmp < 0.
 * MMG_NAME_NONE as a unit key turns both filters off for the unit (the reference's `qname == NULL`). */
#define MMG_NAME_NONE 0xffffffffu
/* tkey: n_seq target keys, kept in HBM next to the index (replaces earlier keys) */
int  mmg_idx_set_name_keys(mmg_idx_t *idx, const uint32_t *tkey);

/* ----------------------------------------------------- per-kernel entry points */
/* mm_sketch on the device.  Returns the count in *n_out; writes min(count, cap) entries. */
int  mmg_sketch(mmg_ctx_t *ctx, const char *str, int len, int w, int k, uint32_t rid, int is_hpc,
                mmg128_t *out, int cap, int *n_out);

/* collect_seed_hits / collect_seed_hits_heap for ONE fragment whose minimizers are given.
 * a_out must hold a_cap anchors; *n_a receives the anchor count (even if > a_cap). */
int  mmg_collect_seeds(mmg_ctx_t *ctx, const mmg_idx_t *idx, int heap_sort, int64_t flag, int max_occ,
                       int n_mv, const mmg128_t *mv, int qlen, mmg128_t *a_out, int64_t a_cap, int64_t *n_a,
                       int *rep_len, int *n_mini_pos, uint64_t *mini_pos);
/* the same for a fragment whose unit key is ukey, against an index with name keys: the self/dual filters apply when flag asks for them */
int  mmg_collect_seeds_named(mmg_ctx_t *ctx, const mmg_idx_t *idx, int heap_sort, int64_t flag, int max_occ, int n_mv, const mmg128_t *mv,
                             int qlen, uint32_t ukey, mmg128_t *a_out, int64_t a_cap, int64_t *n_a, int *rep_len, int *n_mini_pos,
                             uint64_t *mini_pos);

/* mm_chain_dp for ONE anchor array: a[] (n) is replaced by the compacted chains, u[] gets score<<32|cnt */
int  mmg_chain_dp(mmg_ctx_t *ctx, int max_dist_x, int max_dist_y, int bw, int max_skip, int max_iter, int min_cnt,
                  int min_sc, int is_cdna, int n_segs, int64_t n, mmg128_t *a, int *n_u, uint64_t *u);

typedef struct {            /* ksw_extz_t (ksw2.h:23-32) without the heap pointer */
	uint32_t max; int32_t zdropped;
	int32_t max_q, max_t, mqe, mqe_t, mte, mte_q, score;
	int32_t n_cigar, reach_end;
} mmg_extz_t;
/* ksw_extd2_sse for ONE pair (query/target are 0..4 codes); cigar must hold qlen+tlen entries */
int  mmg_ksw_extd2(mmg_ctx_t *ctx, int qlen, const uint8_t *query, int tlen, const uint8_t *target, int8_t m,
                   const int8_t *mat, int8_t q, int8_t e, int8_t q2, int8_t e2, int w, int zdrop, int end_bonus,
                   int flag, mmg_extz_t *ez, uint32_t *cigar);

/* ------------------------------------------------------------- batched stages */
typedef struct {            /* the subset of mm_mapopt_t / mm_idx_t the device stages read */
	int64_t flag;           /* MM_F_* (minimap.h:8-38): HEAP_SORT, FOR_ONLY, REV_ONLY, NO_DIAG, NO_DUAL, SR, SPLICE */
	int32_t mid_occ, max_occ;
	int32_t bw, max_gap, max_gap_ref, max_frag_len;
	int32_t max_chain_skip, max_chain_iter, min_cnt, min_chain_score;
	int32_t pe_ori;
	int32_t a, b, q, e, q2, e2, sc_ambi;
} mmg_mapopt_t;

typedef struct {            /* one mini-batch of fragments: inputs are HOST pointers */
	int32_t n_frag, n_seq;
	const int32_t *n_seg;   /* [n_frag] segments per fragment (map.c:453) */
	const int32_t *seg_off; /* [n_frag] first read of each fragment */
	const int32_t *seq_len; /* [n_seq] */
	const uint64_t *seq_off;/* [n_seq] offset of each read in `bases` */
	const char *bases;      /* concatenated ASCII reads, original orientation */
	uint64_t n_bases;
	/* [n_seq] 1 = reverse-complement the read before mapping, whatever fragment it is in (--no-pairing, map.c:458-498: the mates
	 * of a pair are flipped as for a pair but mapped one by one); null: the mates are flipped per pe_ori within each fragment */
	const uint8_t *flip;
	/* [n_frag] unit keys (see "name keys"), which the self/dual filters need; null: the batch has none */
	const uint32_t *ukey;
} mmg_batch_t;

typedef struct {            /* per-fragment chaining output, HOST arrays owned by the ctx (valid until the next batch call) */
	int32_t n_frag;
	const int32_t *n_u;     /* [n_frag] chains */
	const int32_t *n_a;     /* [n_frag] anchors kept in chains */
	const int32_t *rep_len; /* [n_frag] */
	const int32_t *n_mini;  /* [n_frag] query minimizers below the occurrence cut-off */
	const int32_t *rechained; /* [n_frag] 1 if the max_occ re-chain (map.c:353-375) was taken */
	const uint64_t *u_off, *a_off, *mini_off; /* [n_frag+1] prefix offsets into the flat arrays */
	const uint64_t *u;      /* score<<32|cnt */
	const mmg128_t *a;      /* chained anchors, chain by chain */
	const uint64_t *mini_pos;
	double t_h2d_ms, t_kernels_ms, t_d2h_ms;
	uint64_t n_minimizers, n_anchors, n_chain_iter; /* work counters for the roofline */
} mmg_chains_t;

/* upload + encode reads (mate flip per pe_ori, map.c:467-469), then sketch -> seed -> chain (+ re-chain) */
int  mmg_seed_chain_batch(mmg_ctx_t *ctx, const mmg_idx_t *idx, const mmg_mapopt_t *opt, const mmg_batch_t *batch,
                          mmg_chains_t *out);
/* Uploads go through the ctx's MMG_STAGE_SLOTS pinned staging slots.  A caller fills a slot with mmg_stage and uploads it
 * with mmg_upload_stage, so that it can fill one slot for its next batch while the batch uploaded from the other is mapped.
 * mmg_stage first waits until the device has read what the slot's last upload copied, so the host never overwrites data a
 * copy still reads.  The upload makes its batch the resident one: it replaces the previous batch, flips and unit keys included.
 * mmg_seed_chain_resident refuses (MMG_EINVAL) options with MM_F_NO_DIAG or MM_F_NO_DUAL when the index has no target keys
 * or the batch was uploaded without unit keys. */
#define MMG_STAGE_SLOTS 2
typedef struct {            /* writable pinned arrays of one staging slot, laid out as the fields of mmg_batch_t */
	char *bases;            /* [n_bases] */
	int32_t *seq_len;       /* [n_seq] */
	uint64_t *seq_off;      /* [n_seq] */
	int32_t *n_seg, *seg_off; /* [n_frag] */
	uint8_t *flip;          /* [n_seq] when asked for, else null */
	uint32_t *ukey;         /* [n_frag] when asked for, else null */
} mmg_stage_t;
int  mmg_stage(mmg_ctx_t *ctx, int slot, int n_frag, int n_seq, uint64_t n_bases, int with_flip, int with_ukey, mmg_stage_t *out);
/* upload what the slot holds and encode the reads (mate flip per the slot's flip table or pe_ori, map.c:467-469) */
int  mmg_upload_stage(mmg_ctx_t *ctx, const mmg_mapopt_t *opt, int slot);
/* the upload half of mmg_seed_chain_batch, so that a caller can time device-resident work separately: the batch's host arrays
 * are copied into slot 0 (mmg_stage), then uploaded from there */
int  mmg_batch_upload(mmg_ctx_t *ctx, const mmg_mapopt_t *opt, const mmg_batch_t *batch);

int  mmg_seed_chain_resident(mmg_ctx_t *ctx, const mmg_idx_t *idx, const mmg_mapopt_t *opt, mmg_chains_t *out, int download);

typedef struct {            /* one DP job against the resident batch and index (align.c:313 call sites) */
	int32_t seq_id;         /* read in the resident batch */
	int32_t q_rev;          /* 0: read as mapped; 1: its reverse complement (qseq0[rev], align.c:865-870) */
	int32_t q_start, q_len; /* slice of that strand */
	int32_t rid, t_start, t_len; /* reference slice */
	int32_t reversed;       /* 1: both slices are reversed before DP (left extension, align.c:694-695) */
	int32_t w, zdrop, end_bonus, flag;
} mmg_ksw_job_t;

typedef struct {
	mmg_extz_t ez;
	uint64_t cigar_off;     /* into the flat cigar array returned by mmg_ksw_batch */
} mmg_ksw_res_t;

/* run n_jobs DP jobs; res[] (n_jobs) is caller-allocated; *cigars points to a ctx-owned HOST array */
int  mmg_ksw_batch(mmg_ctx_t *ctx, const mmg_idx_t *idx, const mmg_mapopt_t *opt, int n_jobs, const mmg_ksw_job_t *jobs,
                   mmg_ksw_res_t *res, const uint32_t **cigars, double *kernel_ms, uint64_t *cells);
/* jobs and true-band cells the last mmg_ksw_batch() ran in the thread-per-job fast form (band never clips) and in the literal 16-lane form */
void mmg_ksw_last_split(const mmg_ctx_t *ctx, uint64_t *jobs_fast, uint64_t *cells_fast, uint64_t *jobs_literal, uint64_t *cells_literal);
/* page-locked job / result arrays owned by the ctx (kept across batches) for mmg_ksw_batch; plain malloc'd arrays work too, slower */
int  mmg_job_buffers(mmg_ctx_t *ctx, size_t n_jobs, mmg_ksw_job_t **jobs, mmg_ksw_res_t **res);

/* ------------------------------------------- post-chaining stages on the device (short-read presets)
 * What mm_map_frag does between mm_chain_dp and its return (map.c:376-406: mm_gen_regs, chain_post, mm_seg_gen,
 * mm_align_skeleton with its ksw_extd2 calls, mm_update_extra, filters, mm_set_mapq, mm_pair) for every fragment of the
 * resident batch, right after mmg_seed_chain_resident(download = 0).  The host receives one blob of finished records. */
typedef struct {
	const int32_t *n_reg;        /* [n_seq] hits per read */
	const int64_t *blob_off;     /* [n_seq+1] byte offset of each read's records in blob */
	const unsigned char *blob;   /* per read: n_reg mm_reg1_t, then for every hit with p != 0 its mm_extra_t + cigar, padded to 8 bytes */
	const int32_t *rep_len;      /* [n_frag] */
	double t_device_ms, t_ksw_ms;
	uint64_t n_dp_jobs, n_dp_cells, n_dp_rounds, n_dp_jobs_fast, n_dp_cells_fast;
	int32_t finished;            /* 1: MAPQ, pairing and the mate un-flip (map.c:392-406,486-497) were done on the device as well */
} mmg_post_out_t;
/* mapopt_full: the caller's mm_mapopt_t (minimap.h:107-150) as bytes; idx_flag: mm_idx_t::flag; frag_hash[n_frag]: the
 * per-fragment salt of map.c:291-293 (it depends on the read name, which never leaves the host) */
int  mmg_post_chain(mmg_ctx_t *ctx, const mmg_idx_t *idx, const mmg_mapopt_t *opt, const void *mapopt_full, size_t mapopt_bytes, int idx_flag,
                    const uint32_t *frag_hash, mmg_post_out_t *out);

#ifdef __cplusplus
}
#endif
#endif
