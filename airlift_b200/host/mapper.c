/* mapper.c -- the mini-batch mapper: read -> map (GPU stages + host bookkeeping) -> write.
 *
 * Drop-in for the reference's file-level driver (mm_map_file_frag and worker_pipeline, map.c:557-696):
 * same three ordered steps, same records on stdout.  Step 1 no longer calls mm_map_frag once per
 * fragment (worker_for, map.c:458-498); it runs each mini-batch through
 *     upload -> K1 sketch -> K2 seed -> K3 chain          (one device call, mmg_seed_chain_batch)
 *     chains -> hits, primary/secondary, per-mate split    (host threads; hits.c)
 *     rounds of { collect DP jobs -> K4 batch -> resume }  (aln.c + mmg_ksw_batch)
 *     MAPQ, pairing, mate un-flip                          (host threads)
 * with the fragments of a batch cut into one contiguous range per GPU.
 */
#include <stdio.h>
#include <errno.h>
#include <pthread.h>
#include "mm2b_priv.h"

/* ------------------------------------------------------------------ work / time counters (for bench.py and -v4) */

static mm_b200_stats_t g_stats;
static double g_t_name_keys; /* kept apart: mm_b200_stats_t is mirrored by callers */
static pthread_mutex_t g_stats_mu = PTHREAD_MUTEX_INITIALIZER;

double mm_b200_name_key_time(int reset)
{
	double t;
	pthread_mutex_lock(&g_stats_mu);
	t = g_t_name_keys;
	if (reset) g_t_name_keys = 0;
	pthread_mutex_unlock(&g_stats_mu);
	return t;
}

void mm_b200_stats(mm_b200_stats_t *out, int reset)
{
	pthread_mutex_lock(&g_stats_mu);
	if (out) *out = g_stats;
	if (reset) memset(&g_stats, 0, sizeof(g_stats));
	pthread_mutex_unlock(&g_stats_mu);
}

/* ------------------------------------------------------------------ a tiny parallel-for */

typedef struct { void (*fn)(void*, long, int); void *data; long n; volatile long next; int n_threads; } pfor_t;
typedef struct { pfor_t *pf; int tid; } pfor_arg_t;

static void *pfor_worker(void *p)
{
	pfor_arg_t *a = (pfor_arg_t*)p;
	for (;;) {
		const long i = __sync_fetch_and_add(&a->pf->next, 16);
		long j;
		if (i >= a->pf->n) break;
		for (j = i; j < i + 16 && j < a->pf->n; ++j) a->pf->fn(a->pf->data, j, a->tid);
	}
	mm_arena_thread_done(); /* what is left of this worker's arena block goes to the next worker */
	return 0;
}

static void parallel_for(int n_threads, void (*fn)(void*, long, int), void *data, long n)
{
	if (n_threads <= 1 || n < 32) { long i; for (i = 0; i < n; ++i) fn(data, i, 0); return; }
	{
		pfor_t pf = {fn, data, n, 0, n_threads};
		pthread_t *tid = (pthread_t*)alloca((size_t)n_threads * sizeof(pthread_t));
		pfor_arg_t *arg = (pfor_arg_t*)alloca((size_t)n_threads * sizeof(pfor_arg_t));
		int i;
		for (i = 0; i < n_threads; ++i) { arg[i].pf = &pf, arg[i].tid = i; pthread_create(&tid[i], 0, pfor_worker, &arg[i]); }
		for (i = 0; i < n_threads; ++i) pthread_join(tid[i], 0);
	}
}

/* ------------------------------------------------------------------ per-fragment state */

typedef struct {
	int n_segs, qlen_sum, rep_len, frag_gap, active, finished, n_regs0, n_u, n_mini;
	uint32_t hash;
	int *qlens;           /* [n_segs] */
	mm128_t *a;           /* chained anchors of the fragment (owned copy) */
	uint64_t *u, *mini;
	mm_reg1_t *regs0;
	mm_seg_t *seg;        /* per-mate chains when n_segs > 1 */
	mm_alnseg_t *aln;     /* [n_segs] */
} frag_t;

typedef struct {          /* one GPU's share of a mini-batch */
	const mm_idx_t *mi;
	const mm_mapopt_t *opt;
	mmg_ctx_t *ctx;
	mmg_idx_t *didx;
	mmg_mapopt_t dopt;
	int n_threads, f0, f1, s0; /* fragments [f0,f1); s0 = first read */
	mm_bseq1_t *seq;
	int *n_seg, *seg_off, *n_reg, *rep_len, *frag_gap;
	mm_reg1_t **reg;
	frag_t *fr;
	mmg_chains_t ch;
	mm_b200_stats_t st;
	mmg_post_out_t post;  /* device path: packed hits of every read of the shard */
	uint32_t *frag_hash;
	mm_arena_t arena;     /* per-fragment state of this shard: anchors, chains, per-mate copies, DP cache, temporaries */
	pthread_mutex_t *gpu_token; /* held during device stages when the GPU is shared by several shards */
	pthread_mutex_t *up_token;  /* device path: the shards of a GPU upload one after the other, so that the second upload runs under the first shard's kernels */
	size_t *job_off;      /* [nf+1] first job of each fragment in the current DP round */
	mmg_ksw_job_t *jobs;
	mmg_ksw_res_t *res;
	const uint32_t *cig;
	char *stage_dst; const uint64_t *stage_off;
	size_t m_jobs;
	int rc;
	int ci, slot, ops;    /* ctx index in the bucket, its staging slot this shard uses, SH_* */
	const void *batch;    /* the mini-batch the shard belongs to (identifies what a slot holds) */
	const uint8_t *flip;  /* --no-pairing: [read] 1 if the read is mapped reverse-complemented, decided by the pair it was read in; 0: by pe_ori and the fragment */
	uint32_t *ukey;       /* self/dual filters: name key of every unit of the shard, written into the staging slot */
	double t_name_keys;
} shard_t;

static inline int mate_is_flipped(const mm_mapopt_t *opt, int n_segs, int j)
{ /* map.c:468 */
	return n_segs == 2 && ((j == 0 && (opt->pe_ori >> 1 & 1)) || (j == 1 && (opt->pe_ori & 1)));
}

/* segment j of a fragment of ns reads whose first read is `off` */
static inline int read_is_flipped(const shard_t *sh, int ns, int j, int off)
{
	return sh->flip ? sh->flip[off + j] : mate_is_flipped(sh->opt, ns, j);
}

static int chain_gap_ref(const mm_mapopt_t *opt, int qlen_sum)
{ /* map.c:344-349 */
	int g;
	if (opt->max_gap_ref > 0) return opt->max_gap_ref;
	if (opt->max_frag_len > 0) { g = opt->max_frag_len - qlen_sum; return g < opt->max_gap ? opt->max_gap : g; }
	return opt->max_gap;
}

static int use_device_path(const mm_idx_t *mi, const mm_mapopt_t *opt);
static void stage_align(void *data, long i, int tid);
static void stage_finish(void *data, long i, int tid);

/* chains -> hits for fragment i of the shard (map.c:376-388, 390-400 up to the DP) */
static void stage_hits(void *data, long i, int tid)
{
	shard_t *sh = (shard_t*)data;
	const mm_mapopt_t *opt = sh->opt;
	const mm_idx_t *mi = sh->mi;
	const int f = sh->f0 + (int)i, off = sh->seg_off[f], ns = sh->n_seg[f];
	frag_t *fr = &sh->fr[i];
	const mmg_chains_t *ch = &sh->ch;
	int j, is_sr = !!(opt->flag & MM_F_SR);
	memset(fr, 0, sizeof(*fr));
	mm_tls_arena = &sh->arena;
	fr->n_segs = ns;
	fr->qlens = (int*)mm_amalloc((size_t)ns * sizeof(int));
	for (j = 0; j < ns; ++j) {
		sh->n_reg[off + j] = 0, sh->reg[off + j] = 0;
		fr->qlens[j] = sh->seq[off + j].l_seq, fr->qlen_sum += fr->qlens[j];
	}
	if (fr->qlen_sum == 0 || ns <= 0 || ns > MM_MAX_SEG) return;
	if (opt->max_qlen > 0 && fr->qlen_sum > opt->max_qlen) return;
	for (j = 0; j < ns; ++j) /* host copy in mapping orientation, undone in stage_finish (map.c:467-469,489) */
		if (read_is_flipped(sh, ns, j, off)) mm_revcomp_bseq(&sh->seq[off + j]);
	fr->hash = mm_frag_hash(sh->seq[off].name, fr->qlen_sum, opt->seed);
	fr->frag_gap = chain_gap_ref(opt, fr->qlen_sum);
	fr->rep_len = ch->rep_len[i];
	fr->n_u = ch->n_u[i];
	fr->n_mini = ch->n_mini[i];
	if (fr->n_u > 0) {
		/* used in place: the fragment's slice of the ctx's pinned download stays untouched until this shard's next batch */
		fr->u = (uint64_t*)(ch->u + ch->u_off[i]);
		fr->a = (mm128_t*)(ch->a + ch->a_off[i]);
	}
	fr->regs0 = mm_gen_regs(fr->hash, fr->qlen_sum, fr->n_u, fr->u, fr->a);
	fr->n_regs0 = fr->n_u;
	if (!(opt->flag & MM_F_ALL_CHAINS)) { /* chain_post, map.c:249-258 */
		mm_set_parent(opt->mask_level, fr->n_regs0, fr->regs0, opt->a * 2 + opt->b, opt->flag & MM_F_HARD_MLEVEL);
		if (ns <= 1) mm_select_sub(opt->pri_ratio, mi->k * 2, opt->best_n, &fr->n_regs0, fr->regs0);
		else mm_select_sub_multi(opt->pri_ratio, 0.2f, 0.7f, fr->frag_gap, mi->k * 2, opt->best_n, ns, fr->qlens, &fr->n_regs0, fr->regs0);
		if (!(opt->flag & (MM_F_SPLICE|MM_F_SR|MM_F_NO_LJOIN))) mm_join_long(opt, fr->qlen_sum, &fr->n_regs0, fr->regs0, fr->a);
	}
	if (!is_sr) mm_est_err(mi, fr->qlen_sum, fr->n_regs0, fr->regs0, fr->a, fr->n_mini, ch->mini_pos + ch->mini_off[i]);
	fr->aln = (mm_alnseg_t*)mm_acalloc(ns, sizeof(mm_alnseg_t));
	if (ns == 1) {
		sh->n_reg[off] = fr->n_regs0, sh->reg[off] = fr->regs0;
		mm_aln_begin(&fr->aln[0], off - sh->s0, fr->qlens[0], sh->seq[off].seq, fr->n_regs0, fr->regs0, fr->a);
	} else {
		fr->seg = mm_seg_gen(fr->hash, ns, fr->qlens, fr->n_regs0, fr->regs0, &sh->n_reg[off], &sh->reg[off], fr->a);
		free(fr->regs0); fr->regs0 = 0;
		for (j = 0; j < ns; ++j) {
			mm_set_parent(opt->mask_level, sh->n_reg[off + j], sh->reg[off + j], opt->a * 2 + opt->b, opt->flag & MM_F_HARD_MLEVEL);
			mm_aln_begin(&fr->aln[j], off + j - sh->s0, fr->qlens[j], sh->seq[off + j].seq, sh->n_reg[off + j], sh->reg[off + j], fr->seg[j].a);
		}
	}
	fr->active = (opt->flag & MM_F_CIGAR) ? 1 : 0;
	mm_tls_arena = 0;
	if (fr->active) stage_align(data, i, tid); /* first walk (requests the DP jobs) while the fragment is still in cache */
}

/* one resumable pass over the regions of an active fragment (align_regs, map.c:260-270) */
static void stage_align(void *data, long i, int tid)
{
	shard_t *sh = (shard_t*)data;
	frag_t *fr = &sh->fr[i];
	const mm_mapopt_t *opt = sh->opt;
	int j, all_done = 1;
	if (!fr->active) return;
	mm_tls_arena = &sh->arena;
	for (j = 0; j < fr->n_segs; ++j) {
		mm_alnseg_t *s = &fr->aln[j];
		const int off = sh->seg_off[sh->f0 + i] + j;
		if (s->finished) continue;
		if (mm_aln_step(s, opt, sh->mi)) {
			if (!(opt->flag & MM_F_ALL_CHAINS)) {
				mm_set_parent(opt->mask_level, s->n_regs, s->regs, opt->a * 2 + opt->b, opt->flag & MM_F_HARD_MLEVEL);
				mm_select_sub(opt->pri_ratio, sh->mi->k * 2, opt->best_n, &s->n_regs, s->regs);
				mm_set_sam_pri(s->n_regs, s->regs);
			}
			sh->n_reg[off] = s->n_regs, sh->reg[off] = s->regs;
		} else all_done = 0;
	}
	if (all_done) fr->active = 0;
	mm_tls_arena = 0;
	if (all_done) stage_finish(data, i, tid); /* MAPQ, pairing, release: same thread, same cache lines */
}

/* copy the DP jobs a fragment queued in this round into the shard's job array */
static void stage_gather_jobs(void *data, long i, int tid)
{
	shard_t *sh = (shard_t*)data;
	frag_t *fr = &sh->fr[i];
	size_t k = sh->job_off[i];
	int j, q;
	if (!fr->active) return;
	for (j = 0; j < fr->n_segs; ++j) {
		const mm_dpcache_t *c = &fr->aln[j].cache;
		for (q = c->n_sent; q < c->n; ++q) sh->jobs[k++] = c->a[q].job;
	}
}

/* hand the results of this round back to the job caches, in the order they were gathered */
static void stage_scatter_results(void *data, long i, int tid)
{
	shard_t *sh = (shard_t*)data;
	frag_t *fr = &sh->fr[i];
	size_t k = sh->job_off[i];
	int j;
	if (!fr->active) return;
	mm_tls_arena = &sh->arena;
	for (j = 0; j < fr->n_segs; ++j) {
		mm_dpcache_t *c = &fr->aln[j].cache;
		for (; c->n_sent < c->n; ++c->n_sent, ++k) {
			mm_dpjob_t *dj = &c->a[c->n_sent];
			dj->ez = sh->res[k].ez;
			if (dj->ez.n_cigar > 0) {
				dj->cigar = (uint32_t*)mm_amalloc((size_t)dj->ez.n_cigar * 4);
				memcpy(dj->cigar, sh->cig + sh->res[k].cigar_off, (size_t)dj->ez.n_cigar * 4);
			}
			dj->done = 1;
		}
	}
}

/* MAPQ, pairing, release, mate un-flip (map.c:392-406, 486-497) */
static void stage_finish(void *data, long i, int tid)
{
	shard_t *sh = (shard_t*)data;
	frag_t *fr = &sh->fr[i];
	const mm_mapopt_t *opt = sh->opt;
	const int f = sh->f0 + (int)i, off = sh->seg_off[f], ns = fr->n_segs, is_sr = !!(opt->flag & MM_F_SR);
	int j, k, mapped;
	if (fr->finished) return;
	fr->finished = 1;
	mm_tls_arena = &sh->arena;
	mapped = !(fr->qlen_sum == 0 || ns <= 0 || ns > MM_MAX_SEG || (opt->max_qlen > 0 && fr->qlen_sum > opt->max_qlen));
	if (mapped) {
		for (j = 0; j < ns; ++j) mm_set_mapq(sh->n_reg[off + j], sh->reg[off + j], opt->min_chain_score, opt->a, fr->rep_len, is_sr);
		if (ns == 2 && opt->pe_ori >= 0 && (opt->flag & MM_F_CIGAR))
			mm_pair(fr->frag_gap, opt->pe_bonus, opt->a * 2 + opt->b, opt->a, fr->qlens, &sh->n_reg[off], &sh->reg[off]);
		for (j = 0; j < ns; ++j)
			if (read_is_flipped(sh, ns, j, off)) {
				mm_revcomp_bseq(&sh->seq[off + j]);
				for (k = 0; k < sh->n_reg[off + j]; ++k) {
					mm_reg1_t *r = &sh->reg[off + j][k];
					const int t = r->qs;
					r->qs = fr->qlens[j] - r->qe, r->qe = fr->qlens[j] - t, r->rev = !r->rev;
				}
			}
	}
	for (j = 0; j < ns; ++j) sh->rep_len[off + j] = fr->rep_len, sh->frag_gap[off + j] = fr->frag_gap;
	mm_tls_arena = 0;
}

static void shard_fail(shard_t *sh, const char *what)
{
	fprintf(stderr, "[ERROR] %s: %s\n", what, mmg_last_error());
	sh->rc = -1;
}

static void stage_copy_read(void *data, long i, int tid)
{
	shard_t *sh = (shard_t*)data;
	const mm_bseq1_t *t = &sh->seq[sh->s0 + i];
	memcpy(sh->stage_dst + sh->stage_off[i], t->seq, t->l_seq);
}

static inline int use_name_filters(const mm_mapopt_t *opt) { return (opt->flag & (MM_F_NO_DIAG | MM_F_NO_DUAL)) != 0; }

static void stage_unit_key(void *data, long i, int tid)
{ /* the unit's name is its first read's (worker_for passes it to mm_map_frag, map.c:475-485) */
	shard_t *sh = (shard_t*)data;
	sh->ukey[i] = mm_b200_unit_key(sh->mi, sh->seq[sh->seg_off[sh->f0 + i]].name);
}

/* what map_step_group does with every shard: fill a pinned staging slot of its ctx (host), upload the slot (H2D + 4-bit
 * encode), map the resident batch */
enum { SH_STAGE = 1, SH_SEND = 2, SH_MAP = 4 };

/* the host part of an upload: the reads of units [f0,f1), their four tables, the flips and the unit keys into staging slot
 * sh->slot of the ctx.  mm_b200_map_batches runs it for a lane group's next mini-batch while the current one is mapped. */
static void shard_stage(shard_t *sh)
{
	struct mm_idx_bucket_s *B = sh->mi->B;
	const int nf = sh->f1 - sh->f0;
	const double t0 = realtime();
	int i, n_seq = 0;
	uint64_t n_bases = 0, o;
	mmg_stage_t st;
	B->staged[sh->ci][sh->slot].batch = 0; /* the slot holds nothing whole until the end */
	for (i = sh->f0; i < sh->f1; ++i) n_seq += sh->n_seg[i];
	for (i = 0; i < n_seq; ++i) n_bases += sh->seq[sh->s0 + i].l_seq;
	if (mmg_stage(sh->ctx, sh->slot, nf, n_seq, n_bases, sh->flip != 0, use_name_filters(sh->opt), &st) != MMG_OK) {
		shard_fail(sh, "cannot allocate the staging buffers");
		return;
	}
	if (sh->flip) memcpy(st.flip, sh->flip + sh->s0, (size_t)n_seq); /* the reads are uploaded as read; the device flips them from this table */
	if (st.ukey) {
		const double tk = realtime();
		sh->ukey = st.ukey;
		parallel_for(sh->n_threads, stage_unit_key, sh, nf);
		sh->t_name_keys += realtime() - tk;
	}
	for (i = 0, o = 0; i < n_seq; ++i) {
		st.seq_len[i] = sh->seq[sh->s0 + i].l_seq, st.seq_off[i] = o;
		o += st.seq_len[i];
	}
	sh->stage_dst = st.bases, sh->stage_off = st.seq_off;
	parallel_for(sh->n_threads, stage_copy_read, sh, n_seq);
	for (i = 0; i < nf; ++i) st.n_seg[i] = sh->n_seg[sh->f0 + i], st.seg_off[i] = sh->seg_off[sh->f0 + i] - sh->s0;
	B->staged[sh->ci][sh->slot].batch = sh->batch, B->staged[sh->ci][sh->slot].f0 = sh->f0, B->staged[sh->ci][sh->slot].f1 = sh->f1;
	if (getenv("MM2_B200_TRACE")) fprintf(stderr, "[T::upload] staged %d reads in %.4f s\n", n_seq, realtime() - t0);
	sh->st.n_frag += nf, sh->st.n_reads += n_seq, sh->st.n_bases += n_bases;
	sh->st.t_upload += realtime() - t0;
}

/* the device part: upload what the slot holds */
static void shard_send(shard_t *sh)
{
	const double t0 = realtime();
	if (mmg_upload_stage(sh->ctx, &sh->dopt, sh->slot) != MMG_OK) {
		shard_fail(sh, "read upload failed");
		return;
	}
	if (getenv("MM2_B200_TRACE")) fprintf(stderr, "[T::upload] device upload %.4f s\n", realtime() - t0);
	sh->st.t_upload += realtime() - t0;
}

/* ---- device path (short-read presets): hits, per-mate split, alignment walk and CIGAR post-processing run on the GPU
 * (csrc/mmg_post.cu: designed device stages over flat arrays, mmg_hits.h / mmg_aln.h / mmg_post.h, MAPQ and pairing included); the
 * host computes the name hash before and unpacks the result blob into malloc'd API objects after */

static void stage_dev_hash(void *data, long i, int tid)
{
	shard_t *sh = (shard_t*)data;
	const int f = sh->f0 + (int)i, off = sh->seg_off[f], ns = sh->n_seg[f];
	int j, qlen_sum = 0;
	for (j = 0; j < ns; ++j) qlen_sum += sh->seq[off + j].l_seq;
	sh->frag_hash[i] = mm_frag_hash(sh->seq[off].name, qlen_sum, sh->opt->seed);
}

/* blob -> malloc'd mm_reg1_t / mm_extra_t (minimap.h:317-331 ownership), then MAPQ, pairing, mate un-flip (map.c:392-406, 486-497) */
static void stage_dev_finish(void *data, long i, int tid)
{
	shard_t *sh = (shard_t*)data;
	const mm_mapopt_t *opt = sh->opt;
	const int f = sh->f0 + (int)i, off = sh->seg_off[f], ns = sh->n_seg[f], is_sr = !!(opt->flag & MM_F_SR);
	int j, k, qlen_sum = 0, frag_gap, mapped, qlens[MM_MAX_SEG];
	const int rep_len = sh->post.rep_len[i];
	for (j = 0; j < ns && j < MM_MAX_SEG; ++j) qlens[j] = sh->seq[off + j].l_seq, qlen_sum += qlens[j];
	frag_gap = chain_gap_ref(opt, qlen_sum);
	for (j = 0; j < ns; ++j) {
		const int rr = off + j - sh->s0, n = sh->post.n_reg[rr];
		const unsigned char *b = sh->post.blob + sh->post.blob_off[rr], *e = b + (size_t)n * sizeof(mm_reg1_t);
		mm_reg1_t *regs = 0;
		if (n > 0) {
			regs = (mm_reg1_t*)malloc((size_t)n * sizeof(mm_reg1_t));
			memcpy(regs, b, (size_t)n * sizeof(mm_reg1_t));
			for (k = 0; k < n; ++k)
				if (regs[k].p) {
					const mm_extra_t *src = (const mm_extra_t*)e;
					const size_t bytes = sizeof(mm_extra_t) + (size_t)src->n_cigar * 4, cap = (size_t)src->capacity * 4;
					regs[k].p = (mm_extra_t*)malloc(cap > bytes ? cap : bytes);
					memcpy(regs[k].p, src, bytes);
					e += (bytes + 7) & ~(size_t)7;
				}
		}
		sh->n_reg[off + j] = n, sh->reg[off + j] = regs;
	}
	mapped = !(qlen_sum == 0 || ns <= 0 || ns > MM_MAX_SEG || (opt->max_qlen > 0 && qlen_sum > opt->max_qlen));
	if (mapped && !sh->post.finished) { /* a device layer that stops before MAPQ leaves these three steps to the host */
		for (j = 0; j < ns; ++j) mm_set_mapq(sh->n_reg[off + j], sh->reg[off + j], opt->min_chain_score, opt->a, rep_len, is_sr);
		if (ns == 2 && opt->pe_ori >= 0 && (opt->flag & MM_F_CIGAR))
			mm_pair(frag_gap, opt->pe_bonus, opt->a * 2 + opt->b, opt->a, qlens, &sh->n_reg[off], &sh->reg[off]);
		for (j = 0; j < ns; ++j)
			if (read_is_flipped(sh, ns, j, off)) /* the host copy of the read was never flipped on this path: only the coordinates are */
				for (k = 0; k < sh->n_reg[off + j]; ++k) {
					mm_reg1_t *r = &sh->reg[off + j][k];
					const int t = r->qs;
					r->qs = qlens[j] - r->qe, r->qe = qlens[j] - t, r->rev = !r->rev;
				}
	}
	for (j = 0; j < ns; ++j) sh->rep_len[off + j] = rep_len, sh->frag_gap[off + j] = frag_gap;
}

static int g_serial_shards = 0;
/* bench.py's kernel-profile pass: the shards of a GPU take turns on the device, so that per-kernel CUDA-event times are not
 * stretched by kernels of the other shard running next to them */
void mm_b200_set_serial(int on) { g_serial_shards = on; }

static int use_device_path(const mm_idx_t *mi, const mm_mapopt_t *opt)
{ /* the device post-chaining stages cover the short-read presets; =/X CIGARs and HPC indexes take the host stages */
	static int host_only = -1;
	if (host_only < 0) host_only = getenv("MM2_B200_HOSTPATH") != 0;
	return !host_only && (opt->flag & MM_F_SR) && !(opt->flag & (MM_F_SPLICE | MM_F_EQX)) && !(mi->flag & MM_I_HPC);
}

static void *dev_hash_main(void *data)
{
	shard_t *sh = (shard_t*)data;
	parallel_for(sh->n_threads, stage_dev_hash, sh, sh->f1 - sh->f0);
	return 0;
}

static void *map_shard_dev(shard_t *sh)
{
	const int nf = sh->f1 - sh->f0;
	double t0 = realtime(), t1;
	pthread_t th_hash;
	int rc;
	sh->frag_hash = (uint32_t*)malloc((size_t)nf * 4);
	pthread_create(&th_hash, 0, dev_hash_main, sh); /* the name hashes are computed while the device sketches, seeds and chains */
	if (sh->gpu_token) pthread_mutex_lock(sh->gpu_token);
	rc = mmg_seed_chain_resident(sh->ctx, sh->didx, &sh->dopt, &sh->ch, 0);
	if (sh->gpu_token) pthread_mutex_unlock(sh->gpu_token);
	t1 = realtime();
	pthread_join(th_hash, 0);
	if (rc != MMG_OK) { free(sh->frag_hash); sh->frag_hash = 0; shard_fail(sh, "seed/chain stage failed"); return 0; }
	sh->st.t_seedchain += t1 - t0, sh->st.t_seedchain_kernels += sh->ch.t_kernels_ms * 1e-3;
	sh->st.n_minimizers += sh->ch.n_minimizers, sh->st.n_anchors += sh->ch.n_anchors, sh->st.n_chain_iter += sh->ch.n_chain_iter;
	t0 = realtime(); sh->st.t_hits += t0 - t1;
	if (sh->gpu_token) pthread_mutex_lock(sh->gpu_token);
	rc = mmg_post_chain(sh->ctx, sh->didx, &sh->dopt, sh->opt, sizeof(mm_mapopt_t), sh->mi->flag, sh->frag_hash, &sh->post);
	if (sh->gpu_token) pthread_mutex_unlock(sh->gpu_token);
	free(sh->frag_hash); sh->frag_hash = 0;
	if (rc != MMG_OK) { shard_fail(sh, "post-chaining device stages failed"); return 0; }
	t1 = realtime();
	sh->st.t_ksw_total += t1 - t0, sh->st.t_ksw_kernel += sh->post.t_ksw_ms * 1e-3;
	sh->st.n_dp_jobs += sh->post.n_dp_jobs, sh->st.n_dp_cells += sh->post.n_dp_cells, sh->st.n_dp_rounds += sh->post.n_dp_rounds;
	sh->st.n_dp_jobs_fast += sh->post.n_dp_jobs_fast, sh->st.n_dp_cells_fast += sh->post.n_dp_cells_fast;
	parallel_for(sh->n_threads, stage_dev_finish, sh, nf);
	sh->st.t_finish += realtime() - t1;
	return 0;
}

/* map the fragments [f0,f1) whose reads are resident on the shard's GPU */
static void *map_shard(void *data)
{
	shard_t *sh = (shard_t*)data;
	const int nf = sh->f1 - sh->f0;
	int i, j;
	double t0, t1;
	if (nf <= 0 || sh->rc) return 0;
	if (use_device_path(sh->mi, sh->opt)) return map_shard_dev(sh);
	t0 = realtime();
	if (sh->gpu_token) pthread_mutex_lock(sh->gpu_token);
	i = mmg_seed_chain_resident(sh->ctx, sh->didx, &sh->dopt, &sh->ch, 1);
	if (sh->gpu_token) pthread_mutex_unlock(sh->gpu_token);
	if (i != MMG_OK) { shard_fail(sh, "seed/chain stage failed"); return 0; }
	t1 = realtime();
	sh->st.t_seedchain += t1 - t0, sh->st.t_seedchain_kernels += sh->ch.t_kernels_ms * 1e-3;
	sh->st.n_minimizers += sh->ch.n_minimizers, sh->st.n_anchors += sh->ch.n_anchors, sh->st.n_chain_iter += sh->ch.n_chain_iter;

	sh->fr = (frag_t*)calloc(nf, sizeof(frag_t));
	parallel_for(sh->n_threads, stage_hits, sh, nf);
	t0 = realtime(); sh->st.t_hits += t0 - t1;
	if (sh->opt->flag & MM_F_CIGAR) {
		size_t m_jobs = 0;
		int round = 0;
		sh->job_off = (size_t*)malloc((size_t)(nf + 1) * sizeof(size_t));
		for (;;) { /* DP rounds: walk the regions, send what they asked for, hand the results back */
			size_t n_jobs = 0;
			int n_active = 0;
			double ta = realtime(), tb, kms = 0;
			uint64_t cells = 0;
			if (round++ > 0) parallel_for(sh->n_threads, stage_align, sh, nf);
			for (i = 0; i < nf; ++i) { /* new jobs per fragment -> offsets */
				const frag_t *fr = &sh->fr[i];
				sh->job_off[i] = n_jobs;
				if (!fr->active) continue;
				++n_active;
				for (j = 0; j < fr->n_segs; ++j) n_jobs += (size_t)(fr->aln[j].cache.n - fr->aln[j].cache.n_sent);
			}
			sh->job_off[nf] = n_jobs;
			tb = realtime(); sh->st.t_align_host += tb - ta;
			if (n_active == 0) break;
			if (n_jobs == 0) { fprintf(stderr, "[ERROR] alignment made no progress\n"); sh->rc = -1; break; }
			if (n_jobs > m_jobs) { /* page-locked arrays kept by the ctx: they cross PCIe every round */
				m_jobs = n_jobs + n_jobs / 4;
				if (mmg_job_buffers(sh->ctx, m_jobs, &sh->jobs, &sh->res) != MMG_OK) { shard_fail(sh, "cannot allocate page-locked job arrays"); break; }
			}
			parallel_for(sh->n_threads, stage_gather_jobs, sh, nf);
			ta = realtime(); sh->st.t_align_host += ta - tb;
			if (sh->gpu_token) pthread_mutex_lock(sh->gpu_token);
			j = mmg_ksw_batch(sh->ctx, sh->didx, &sh->dopt, (int)n_jobs, sh->jobs, sh->res, &sh->cig, &kms, &cells);
			if (sh->gpu_token) pthread_mutex_unlock(sh->gpu_token);
			if (j != MMG_OK) { shard_fail(sh, "DP stage failed"); break; }
			tb = realtime();
			sh->st.t_ksw_total += tb - ta, sh->st.t_ksw_kernel += kms * 1e-3;
			sh->st.n_dp_jobs += n_jobs, sh->st.n_dp_cells += cells, sh->st.n_dp_rounds += 1;
			{ uint64_t jf = 0, cf = 0; mmg_ksw_last_split(sh->ctx, &jf, &cf, 0, 0); sh->st.n_dp_jobs_fast += jf, sh->st.n_dp_cells_fast += cf; }
			parallel_for(sh->n_threads, stage_scatter_results, sh, nf);
			sh->st.t_align_host += realtime() - tb;
		}
		free(sh->job_off);
		sh->jobs = 0, sh->res = 0, sh->job_off = 0;
	}
	t0 = realtime();
	parallel_for(sh->n_threads, stage_finish, sh, nf);
	sh->st.t_finish += realtime() - t0;
	free(sh->fr); sh->fr = 0;
	mm_arena_release(&sh->arena); /* gone in one sweep */
	return 0;
}

/* ------------------------------------------------------------------ the three-step pipeline */

typedef struct {
	int mini_batch_size, n_processed, n_threads, n_fp;
	const mm_mapopt_t *opt;
	mm_bseq_file_t **fp;
	const mm_idx_t *mi;
	mm_str_t str;
	int failed;
} pipeline_t;

static step_t *step_read(pipeline_t *p)
{ /* map.c:561-589 */
	const int with_qual = (!!(p->opt->flag & MM_F_OUT_SAM) && !(p->opt->flag & MM_F_NO_QUAL));
	const int with_comment = !!(p->opt->flag & MM_F_COPY_COMMENT);
	const int frag_mode = (p->n_fp > 1 || !!(p->opt->flag & MM_F_FRAG_MODE));
	step_t *s = (step_t*)calloc(1, sizeof(step_t));
	int i, j;
	if (p->n_fp > 1) s->seq = mm_bseq_read_frag2(p->n_fp, p->fp, p->mini_batch_size, with_qual, with_comment, &s->n_seq);
	else s->seq = mm_bseq_read3(p->fp[0], p->mini_batch_size, with_qual, with_comment, frag_mode, &s->n_seq);
	if (s->seq == 0) { free(s); return 0; }
	for (i = 0; i < s->n_seq; ++i) s->seq[i].rid = p->n_processed++;
	s->n_reg = (int*)calloc(5 * (size_t)s->n_seq, sizeof(int));
	s->seg_off = s->n_reg + s->n_seq, s->n_seg = s->seg_off + s->n_seq, s->rep_len = s->n_seg + s->n_seq, s->frag_gap = s->rep_len + s->n_seq;
	s->reg = (mm_reg1_t**)calloc(s->n_seq, sizeof(mm_reg1_t*));
	for (i = 1, j = 0; i <= s->n_seq; ++i)
		if (i == s->n_seq || !frag_mode || !mm_qname_same(s->seq[i-1].name, s->seq[i].name)) {
			s->n_seg[s->n_frag] = i - j;
			s->seg_off[s->n_frag++] = j;
			j = i;
		}
	return s;
}

/* whether the shard's staging slot holds this shard, filled by an earlier SH_STAGE call */
static int slot_holds(const shard_t *sh)
{
	const struct mm_idx_bucket_s *B = sh->mi->B;
	return B->staged[sh->ci][sh->slot].batch == sh->batch && B->staged[sh->ci][sh->slot].f0 == sh->f0 && B->staged[sh->ci][sh->slot].f1 == sh->f1;
}

static void *shard_run(void *data)
{
	shard_t *sh = (shard_t*)data;
	const int send = !!(sh->ops & SH_SEND);
	if (sh->f1 <= sh->f0) return 0;
	if (send && sh->up_token) pthread_mutex_lock(sh->up_token);
	if ((sh->ops & SH_STAGE) || (send && !slot_holds(sh))) shard_stage(sh);
	if (send && !sh->rc) shard_send(sh);
	if (send && sh->up_token) pthread_mutex_unlock(sh->up_token);
	if (sh->ops & SH_MAP) map_shard(sh);
	return 0;
}

/* ops (SH_*): what to do with every shard of the step.  SH_SEND without SH_STAGE stages a shard first unless its slot holds it.
 * slot: the staging slot of every ctx this call uses.
 * group/n_groups: the lanes of every GPU are split into n_groups sets and this call uses set `group`, so that calls on
 * different groups may run at the same time (mm_b200_map_batches) */
static int map_step_group(const mm_idx_t *mi, const mm_mapopt_t *opt, int n_threads, step_t *s, int ops, int group, int n_groups, int slot)
{
	struct mm_idx_bucket_s *B = mi->B;
	const int lanes = B->lanes / n_groups;  /* shards per GPU of this call, each with its own stream */
	const int n_dev = B->n_dev * lanes;
	shard_t *sh = (shard_t*)calloc(n_dev, sizeof(shard_t));
	pthread_t *tid = (pthread_t*)calloc(n_dev, sizeof(pthread_t));
	int d, f = 0, rc = 0;
	int64_t tot = 0, acc = 0;
	const double t_start = realtime();
	/* the mapping units: the fragments as read, or with --no-pairing every read on its own (worker_for, map.c:475-485); the
	 * writer keeps the step's own fragment tables, so that records still print as pairs */
	int n_unit = s->n_frag, *u_seg = s->n_seg, *u_off = s->seg_off, *u_tab = 0;
	uint8_t *u_flip = 0;
	mm_b200_tune_malloc();
	if (mm_b200_check_opt(opt) < 0 || (use_name_filters(opt) && mm_b200_name_keys_ready(mi) < 0)) { free(sh); free(tid); return -1; }
	if (opt->flag & MM_F_INDEPEND_SEG) {
		int k, j;
		u_tab = (int*)malloc(2 * (size_t)s->n_seq * sizeof(int) + 1);
		u_flip = (uint8_t*)malloc((size_t)s->n_seq + 1);
		n_unit = s->n_seq, u_seg = u_tab, u_off = u_tab + s->n_seq;
		for (d = 0; d < s->n_seq; ++d) u_seg[d] = 1, u_off[d] = d;
		for (k = 0; k < s->n_frag; ++k) /* the mates are still flipped as the pair they were read in (map.c:467-469) */
			for (j = 0; j < s->n_seg[k]; ++j) u_flip[s->seg_off[k] + j] = mate_is_flipped(opt, s->n_seg[k], j);
	}
	for (d = 0; d < s->n_seq; ++d) tot += s->seq[d].l_seq;
	for (d = 0; d < n_dev; ++d) { /* contiguous unit ranges balanced by bases; a unit is never cut (with --no-pairing a pair may be) */
		shard_t *h = &sh[d];
		/* device path with two shards per GPU: the first shard is the smaller one, so that its upload (the only one no kernel
		 * can hide) is short and the second, larger upload runs under its kernels */
		const int64_t goal = (lanes == 2 && use_device_path(mi, opt)) ? (tot * (d / 2) + (d % 2 == 0 ? tot * 3 / 10 : tot)) / B->n_dev : tot * (d + 1) / n_dev;
		const int gpu = d / lanes;
		h->mi = mi, h->opt = opt, h->ci = gpu * B->lanes + group * lanes + d % lanes, h->ctx = B->ctx[h->ci], h->didx = B->didx[gpu];
		mm_mapopt_to_dev(opt, &h->dopt);
		mm_arena_init(&h->arena);
		/* lanes of one GPU alternate between device and host stages, so each may use that GPU's whole share of host threads */
		h->n_threads = n_threads / B->n_dev > 0 ? n_threads / B->n_dev : 1;
		/* host path: the lanes of a GPU take turns on the device while the others run host stages; device path: their kernels
		 * may overlap freely (the latency-bound tails of one shard fill the gaps of the other) */
		h->gpu_token = B->lanes > 1 && (!use_device_path(mi, opt) || g_serial_shards) ? &B->gpu_token[gpu] : 0;
		h->up_token = B->lanes > 1 && use_device_path(mi, opt) ? &B->up_token[gpu] : 0;
		h->slot = slot, h->ops = ops, h->batch = s;
		h->seq = s->seq, h->n_seg = u_seg, h->seg_off = u_off, h->n_reg = s->n_reg, h->rep_len = s->rep_len, h->frag_gap = s->frag_gap, h->reg = s->reg;
		h->flip = u_flip;
		h->f0 = f;
		while (f < n_unit && (acc < goal || d == n_dev - 1)) {
			int j;
			for (j = 0; j < u_seg[f]; ++j) acc += s->seq[u_off[f] + j].l_seq;
			++f;
		}
		h->f1 = f;
		if (h->f1 > h->f0) h->s0 = u_off[h->f0];
	}
	if (n_dev == 1) shard_run(&sh[0]);
	else {
		for (d = 0; d < n_dev; ++d) pthread_create(&tid[d], 0, shard_run, &sh[d]);
		for (d = 0; d < n_dev; ++d) pthread_join(tid[d], 0);
	}
	pthread_mutex_lock(&g_stats_mu);
	for (d = 0; d < n_dev; ++d) {
		const mm_b200_stats_t *t = &sh[d].st;
		uint64_t h2d = 0, d2h = 0;
		if (sh[d].rc) rc = -1;
		mmg_copy_bytes(sh[d].ctx, &h2d, &d2h, 1);
		g_stats.t_upload += t->t_upload, g_stats.t_seedchain += t->t_seedchain, g_stats.t_seedchain_kernels += t->t_seedchain_kernels;
		g_stats.t_hits += t->t_hits, g_stats.t_align_host += t->t_align_host, g_stats.t_ksw_total += t->t_ksw_total;
		g_stats.t_ksw_kernel += t->t_ksw_kernel, g_stats.t_finish += t->t_finish;
		g_stats.n_frag += t->n_frag, g_stats.n_reads += t->n_reads, g_stats.n_bases += t->n_bases, g_stats.n_minimizers += t->n_minimizers;
		g_stats.n_anchors += t->n_anchors, g_stats.n_chain_iter += t->n_chain_iter, g_stats.n_dp_jobs += t->n_dp_jobs;
		g_stats.n_dp_cells += t->n_dp_cells, g_stats.n_dp_rounds += t->n_dp_rounds, g_stats.h2d_bytes += h2d, g_stats.d2h_bytes += d2h;
		g_stats.n_dp_jobs_fast += t->n_dp_jobs_fast, g_stats.n_dp_cells_fast += t->n_dp_cells_fast;
		g_t_name_keys += sh[d].t_name_keys;
	}
	g_stats.t_total += realtime() - t_start;
	pthread_mutex_unlock(&g_stats_mu);
	if (getenv("MM2_B200_TRACE")) /* per-batch stage times of every shard */
		for (d = 0; d < n_dev; ++d) {
			const mm_b200_stats_t *t = &sh[d].st;
			fprintf(stderr, "[T::map_step] at %.3f: %.3f s, shard %d: %d frags, upload %.3f seed/chain %.3f (kernels %.3f) hits %.3f align %.3f dp %.3f (kernel %.3f) finish %.3f\n",
					realtime() - mm_realtime0, realtime() - t_start, d, sh[d].f1 - sh[d].f0, t->t_upload, t->t_seedchain, t->t_seedchain_kernels, t->t_hits, t->t_align_host, t->t_ksw_total, t->t_ksw_kernel, t->t_finish);
		}
	free(sh); free(tid); free(u_tab); free(u_flip);
	return rc;
}

/* the mode of mm_b200_map_batch(es): 0 stage, upload and map; 1 stage and upload; 2 map what mode 1 left resident */
static int mode_ops(int mode) { return mode == 1 ? SH_STAGE | SH_SEND : mode == 2 ? SH_MAP : SH_STAGE | SH_SEND | SH_MAP; }

static int step_map(pipeline_t *p, step_t *s) { return map_step_group(p->mi, p->opt, p->n_threads, s, SH_STAGE | SH_SEND | SH_MAP, 0, 1, 0); }

/* Several mini-batches, two in flight: batch i runs on lane group i % 2 of every GPU, so the upload, the latency-bound tails
 * (the serial replays of a few repeat-family fragments) and the host finish of one batch run under the kernels of the other.
 * This is worker_pipeline's overlap of its three steps (map.c:553-652, kt_pipeline with n_threads = 3) carried into the
 * mapping step itself.  Results are complete, batch by batch, when the call returns. */
static int g_in_flight = 2;
int mm_b200_set_in_flight(int n) { if (n < 1 || n > MM_B200_MAX_LANES) return -1; g_in_flight = n; return 0; }
typedef struct { const mm_idx_t *mi; const mm_mapopt_t *opt; int n_threads, mode, group, n_groups, n; step_t **b; int rc; } mb_arg_t;
typedef struct { mb_arg_t *a; int i, slot, n_threads; } mb_stage_t;
static void *map_batches_stage(void *data)
{ /* host staging of batch i into the pinned slot the lane group does not map from */
	mb_stage_t *t = (mb_stage_t*)data;
	map_step_group(t->a->mi, t->a->opt, t->n_threads, t->a->b[t->i], SH_STAGE, t->a->group, t->a->n_groups, t->slot);
	return 0;
}

static void *map_batches_main(void *data)
{
	mb_arg_t *a = (mb_arg_t*)data;
	int i, slot = 0;
	if (a->mode != 0) { /* upload only / map resident: nothing to overlap */
		for (i = a->group; i < a->n; i += a->n_groups)
			if (map_step_group(a->mi, a->opt, a->n_threads, a->b[i], mode_ops(a->mode), a->group, a->n_groups, 0) != 0) a->rc = -1;
		return 0;
	}
	{ mb_stage_t t0 = {a, a->group, 0, a->n_threads}; if (a->group < a->n) map_batches_stage(&t0); }
	for (i = a->group; i < a->n; i += a->n_groups, slot ^= 1) {
		const int nx = i + a->n_groups;
		pthread_t tid;
		mb_stage_t t = {a, nx, slot ^ 1, a->n_threads > 2 ? a->n_threads / 2 : 1};
		if (nx < a->n) pthread_create(&tid, 0, map_batches_stage, &t); /* the next batch of this group is staged while this one is mapped */
		if (map_step_group(a->mi, a->opt, a->n_threads, a->b[i], SH_SEND | SH_MAP, a->group, a->n_groups, slot) != 0) a->rc = -1;
		if (nx < a->n) pthread_join(tid, 0);
	}
	return 0;
}

int mm_b200_batches_in_flight(const mm_idx_t *mi, const mm_mapopt_t *opt)
{ /* how many mini-batches mm_b200_map_batches overlaps for these options (1: one after the other) */
	int n_groups = g_in_flight;
	while (n_groups > 1 && mi->B->lanes % n_groups) --n_groups;
	if (!use_device_path(mi, opt) || g_serial_shards || n_groups < 1) n_groups = 1;
	return n_groups;
}

int mm_b200_map_batches(const mm_idx_t *mi, const mm_mapopt_t *opt, int n_threads, mm_b200_batch_t **b, int n, int mode)
{
	int n_groups = g_in_flight < n ? g_in_flight : n;
	mb_arg_t a[MM_B200_MAX_LANES];
	pthread_t tid[MM_B200_MAX_LANES];
	int g, rc = 0;
	if (n_threads < 1) n_threads = 1;
	while (n_groups > 1 && mi->B->lanes % n_groups) --n_groups;
	if (!use_device_path(mi, opt) || g_serial_shards || n_groups < 1) n_groups = 1;
	for (g = 0; g < n_groups; ++g) {
		a[g].mi = mi, a[g].opt = opt, a[g].n_threads = n_threads / n_groups > 0 ? n_threads / n_groups : 1, a[g].mode = mode;
		a[g].group = g, a[g].n_groups = n_groups, a[g].n = n, a[g].b = (step_t**)b, a[g].rc = 0;
	}
	if (n_groups == 1) map_batches_main(&a[0]);
	else {
		for (g = 0; g < n_groups; ++g) pthread_create(&tid[g], 0, map_batches_main, &a[g]);
		for (g = 0; g < n_groups; ++g) pthread_join(tid[g], 0);
	}
	for (g = 0; g < n_groups; ++g) if (a[g].rc) rc = -1;
	return rc;
}

/* Step 2 (map.c:594-650, no --split-prefix).  Records are formatted by the worker threads, one output buffer per block of
 * fragments, and the buffers leave through stdout in input order: the bytes are those of one puts() per record. */
typedef struct { pipeline_t *p; step_t *s; int frags_per_chunk; char **buf; size_t *len; } write_job_t;

static inline void out_append(char **o, size_t *ol, size_t *om, const char *rec, size_t l)
{
	if (*ol + l + 1 > *om) { *om = (*ol + l + 1) * 2 > (1 << 20) ? (*ol + l + 1) * 2 : (1 << 20); *o = (char*)realloc(*o, *om); }
	memcpy(*o + *ol, rec, l);
	(*o)[*ol + l] = '\n';
	*ol += l + 1;
}

static void write_chunk(void *data, long c, int tid)
{
	write_job_t *w = (write_job_t*)data;
	pipeline_t *p = w->p;
	step_t *s = w->s;
	const mm_idx_t *mi = p->mi;
	const int k0 = (int)c * w->frags_per_chunk, k1 = k0 + w->frags_per_chunk < s->n_frag ? k0 + w->frags_per_chunk : s->n_frag;
	mm_str_t str = {0, 0, 0};
	char *o = 0;
	size_t ol = 0, om = 0;
	int i, j, k;
	for (k = k0; k < k1; ++k) {
		const int seg_st = s->seg_off[k], seg_en = s->seg_off[k] + s->n_seg[k];
		for (i = seg_st; i < seg_en; ++i) {
			mm_bseq1_t *t = &s->seq[i];
			if (s->n_reg[i] > 0) {
				for (j = 0; j < s->n_reg[i]; ++j) {
					mm_reg1_t *r = &s->reg[i][j];
					assert(!r->sam_pri || r->id == r->parent);
					if ((p->opt->flag & MM_F_NO_PRINT_2ND) && r->id != r->parent) continue;
					if (p->opt->flag & MM_F_OUT_SAM)
						mm_write_sam3(&str, mi, t, i - seg_st, j, s->n_seg[k], &s->n_reg[seg_st], (const mm_reg1_t*const*)&s->reg[seg_st], (int)p->opt->flag, s->rep_len[i]);
					else mm_write_paf3(&str, mi, t, r, (int)p->opt->flag, s->rep_len[i]);
					out_append(&o, &ol, &om, str.s, str.l);
				}
			} else if ((p->opt->flag & MM_F_PAF_NO_HIT) || ((p->opt->flag & MM_F_OUT_SAM) && !(p->opt->flag & MM_F_SAM_HIT_ONLY))) {
				if (p->opt->flag & MM_F_OUT_SAM)
					mm_write_sam3(&str, mi, t, i - seg_st, -1, s->n_seg[k], &s->n_reg[seg_st], (const mm_reg1_t*const*)&s->reg[seg_st], (int)p->opt->flag, s->rep_len[i]);
				else mm_write_paf3(&str, mi, t, 0, (int)p->opt->flag, s->rep_len[i]);
				out_append(&o, &ol, &om, str.s, str.l);
			}
		}
		for (i = seg_st; i < seg_en; ++i) {
			for (j = 0; j < s->n_reg[i]; ++j) free(s->reg[i][j].p);
			free(s->reg[i]);
		}
	}
	free(str.s);
	w->buf[c] = o, w->len[c] = ol;
}

static void step_write(pipeline_t *p, step_t *s)
{
	write_job_t w;
	const int fpc = 256, n_chunks = (s->n_frag + fpc - 1) / fpc;
	int c;
	w.p = p, w.s = s, w.frags_per_chunk = fpc;
	w.buf = (char**)calloc(n_chunks > 0 ? n_chunks : 1, sizeof(char*));
	w.len = (size_t*)calloc(n_chunks > 0 ? n_chunks : 1, sizeof(size_t));
	{
		const double t0 = realtime();
		parallel_for(p->n_threads, write_chunk, &w, n_chunks);
		if (getenv("MM2_B200_TRACE")) fprintf(stderr, "[T::write] formatted %d chunks in %.3f s\n", n_chunks, realtime() - t0);
	}
	for (c = 0; c < n_chunks; ++c) {
		if (w.len[c] && fwrite(w.buf[c], 1, w.len[c], stdout) != w.len[c]) { /* a short write is fatal (misc.c:123-131) */
			perror("[ERROR] failed to write the results");
			exit(EXIT_FAILURE);
		}
		free(w.buf[c]);
	}
	free(w.buf); free(w.len);
	/* the reads were allocated by the read-ahead threads: sixteen workers returning them to those two malloc arenas contend on
	 * their locks (it was half of the writer's time), one thread does not */
	for (c = 0; c < s->n_seq; ++c) mm_bseq_free1(&s->seq[c], 1);
	if (mm_verbose >= 3)
		fprintf(stderr, "[M::%s::%.3f*%.2f] mapped %d sequences\n", "worker_pipeline", realtime() - mm_realtime0, cputime() / (realtime() - mm_realtime0), s->n_seq);
	free(s->reg); free(s->n_reg); free(s->seq);
	free(s);
}

/* Ordered hand-off between the three steps: one slot per edge, so that reading batch n+1, mapping batch n and
 * writing batch n-1 overlap while records still leave in input order (kthread.c:97-159 gives the same guarantee). */
typedef struct { pthread_mutex_t mu; pthread_cond_t cv; step_t *item; int has, closed; } slot_t;

static void slot_init(slot_t *q) { pthread_mutex_init(&q->mu, 0); pthread_cond_init(&q->cv, 0); q->item = 0, q->has = q->closed = 0; }
static void slot_put(slot_t *q, step_t *s)
{
	pthread_mutex_lock(&q->mu);
	while (q->has) pthread_cond_wait(&q->cv, &q->mu);
	q->item = s, q->has = 1;
	pthread_cond_broadcast(&q->cv);
	pthread_mutex_unlock(&q->mu);
}
static void slot_close(slot_t *q)
{
	pthread_mutex_lock(&q->mu);
	while (q->has) pthread_cond_wait(&q->cv, &q->mu);
	q->closed = 1;
	pthread_cond_broadcast(&q->cv);
	pthread_mutex_unlock(&q->mu);
}
static step_t *slot_get(slot_t *q)
{
	step_t *s = 0;
	pthread_mutex_lock(&q->mu);
	while (!q->has && !q->closed) pthread_cond_wait(&q->cv, &q->mu);
	if (q->has) { s = q->item; q->has = 0; pthread_cond_broadcast(&q->cv); }
	pthread_mutex_unlock(&q->mu);
	return s;
}

typedef struct { pipeline_t *p; slot_t *in, *out; } stage_arg_t;

static void *reader_main(void *a)
{
	stage_arg_t *g = (stage_arg_t*)a;
	step_t *s;
	const int trace = getenv("MM2_B200_TRACE") != 0;
	double t0 = realtime();
	while (!g->p->failed && (s = step_read(g->p)) != 0) {
		if (trace) fprintf(stderr, "[T::read] at %.3f: %d reads parsed in %.3f s\n", realtime() - mm_realtime0, s->n_seq, realtime() - t0);
		slot_put(g->out, s);
		t0 = realtime();
	}
	slot_close(g->out);
	return 0;
}

static void *writer_main(void *a)
{
	stage_arg_t *g = (stage_arg_t*)a;
	step_t *s;
	while ((s = slot_get(g->in)) != 0) {
		const double t0 = realtime();
		const int n = s->n_seq;
		step_write(g->p, s);
		if (getenv("MM2_B200_TRACE")) fprintf(stderr, "[T::write] at %.3f: %d reads written in %.3f s\n", realtime() - mm_realtime0, n, realtime() - t0);
	}
	return 0;
}

/* The mapping step with two mini-batches in flight (mm_b200_map_batches' overlap inside the file driver): two mappers, one per
 * lane group, take the batches alternately; a turn counter hands them to the writer in input order.  The second group's arenas
 * cost ~0.5 s to allocate and as much to release (tens of GB at human size), so it only joins after MM2_B200_WARM_BATCHES
 * mini-batches (default 16): short runs pay nothing, long runs map 6.5 M instead of 5.1 M reads/s in steady state. */
typedef struct { pthread_mutex_t mu; pthread_cond_t cv; long turn; } turn_t;
typedef struct { pipeline_t *p; slot_t *in, *out; turn_t *turn; int group, lane_groups, n_threads; } mapper_arg_t;

static void *mapper_main(void *a)
{
	mapper_arg_t *m = (mapper_arg_t*)a;
	pipeline_t *p = m->p;
	step_t *s;
	int i;
	while ((s = slot_get(m->in)) != 0) {
		const long idx = s->order;
		if (!p->failed && map_step_group(p->mi, p->opt, m->n_threads, s, SH_STAGE | SH_SEND | SH_MAP, m->group, m->lane_groups, 0) != 0) p->failed = 1;
		pthread_mutex_lock(&m->turn->mu);
		while (m->turn->turn != idx) pthread_cond_wait(&m->turn->cv, &m->turn->mu);
		pthread_mutex_unlock(&m->turn->mu);
		if (p->failed) { /* keep draining so the reader can finish; nothing more is written */
			for (i = 0; i < s->n_seq; ++i) mm_bseq_free1(&s->seq[i], 1);
			free(s->reg); free(s->n_reg); free(s->seq); free(s);
		} else slot_put(m->out, s);
		pthread_mutex_lock(&m->turn->mu);
		++m->turn->turn;
		pthread_cond_broadcast(&m->turn->cv);
		pthread_mutex_unlock(&m->turn->mu);
	}
	return 0;
}

int mm_map_file_frag(const mm_idx_t *idx, int n_segs, const char **fn, const mm_mapopt_t *opt, int n_threads)
{
	pipeline_t pl;
	slot_t q_read, q_write;
	stage_arg_t ra, wa;
	pthread_t t_read, t_write;
	step_t *s;
	int i;
	if (n_segs < 1) return -1;
	if (idx == 0 || idx->B == 0 || idx->B->n_dev < 1) { fprintf(stderr, "[ERROR] the index is not resident on a GPU\n"); return -1; }
	if (mm_b200_check_opt(opt) < 0) return -1;
	memset(&pl, 0, sizeof(pl));
	pl.n_fp = n_segs;
	pl.fp = (mm_bseq_file_t**)calloc(n_segs, sizeof(mm_bseq_file_t*));
	for (i = 0; i < n_segs; ++i)
		if ((pl.fp[i] = mm_bseq_open(fn[i])) == 0) {
			int j;
			if (mm_verbose >= 1) fprintf(stderr, "ERROR: failed to open file '%s': %s\n", fn[i], strerror(errno));
			for (j = 0; j < i; ++j) mm_bseq_close(pl.fp[j]);
			free(pl.fp);
			return -1;
		}
	for (i = 0; i < n_segs; ++i) mm_bseq_set_readahead(pl.fp[i], 1); /* parse each file ahead in its own thread */
	pl.opt = opt, pl.mi = idx;
	pl.n_threads = n_threads > 1 ? n_threads : 1;
	pl.mini_batch_size = opt->mini_batch_size;
	slot_init(&q_read); slot_init(&q_write);
	ra.p = wa.p = &pl, ra.in = 0, ra.out = &q_read, wa.in = &q_write, wa.out = 0;
	pthread_create(&t_read, 0, reader_main, &ra);
	pthread_create(&t_write, 0, writer_main, &wa);
	if (idx->B->lanes >= 4 && idx->B->lanes % 2 == 0) {
		/* four streams per GPU: the device path keeps two mini-batches in flight, one per lane group; the host path (long-read
		 * presets) maps one batch at a time on the first group, i.e. on two streams as before */
		const int n_map = mm_b200_batches_in_flight(idx, opt) >= 2 ? 2 : 1;
		slot_t q_map[2];
		turn_t turn;
		mapper_arg_t ma[2];
		pthread_t t_map[2];
		long n_in = 0;
		const long warm = getenv("MM2_B200_WARM_BATCHES") ? atol(getenv("MM2_B200_WARM_BATCHES")) : 16;
		int g;
		pthread_mutex_init(&turn.mu, 0); pthread_cond_init(&turn.cv, 0); turn.turn = 0;
		for (g = 0; g < n_map; ++g) {
			slot_init(&q_map[g]);
			ma[g].p = &pl, ma[g].in = &q_map[g], ma[g].out = &q_write, ma[g].turn = &turn, ma[g].group = g, ma[g].lane_groups = 2;
			ma[g].n_threads = pl.n_threads / n_map > 0 ? pl.n_threads / n_map : 1;
			pthread_create(&t_map[g], 0, mapper_main, &ma[g]);
		}
		while ((s = slot_get(&q_read)) != 0) {
			s->order = n_in;
			slot_put(&q_map[n_map == 2 && n_in >= warm ? n_in % 2 : 0], s);
			++n_in;
		}
		for (g = 0; g < n_map; ++g) slot_close(&q_map[g]);
		for (g = 0; g < n_map; ++g) pthread_join(t_map[g], 0);
	} else
	while ((s = slot_get(&q_read)) != 0) {
		if (!pl.failed && step_map(&pl, s) != 0) pl.failed = 1;
		if (pl.failed) { /* keep draining so the reader can finish; nothing more is written */
			for (i = 0; i < s->n_seq; ++i) mm_bseq_free1(&s->seq[i], 1);
			free(s->reg); free(s->n_reg); free(s->seq); free(s);
			continue;
		}
		slot_put(&q_write, s);
	}
	slot_close(&q_write);
	pthread_join(t_read, 0);
	pthread_join(t_write, 0);
	free(pl.str.s);
	for (i = 0; i < pl.n_fp; ++i) mm_bseq_close(pl.fp[i]);
	free(pl.fp);
	if (pl.failed) { fprintf(stderr, "[ERROR] mapping failed; no CPU fallback exists\n"); exit(1); }
	return 0;
}

int mm_map_file(const mm_idx_t *idx, const char *fn, const mm_mapopt_t *opt, int n_threads)
{
	return mm_map_file_frag(idx, 1, &fn, opt, n_threads);
}

/* ------------------------------------------------------------------ per-fragment API (shared mini-batches, apiq.c) */

struct mm_tbuf_s { int rep_len, frag_gap; };
const char *mm_b200_opt_error(const mm_mapopt_t *opt)
{ /* what the device stages do not implement is refused with a message; nothing is silently dropped */
#define NOT_SUPPORTED " is not supported by this build"
	if (opt->flag & MM_F_SPLICE) return "spliced alignment (--splice, ksw_exts2)" NOT_SUPPORTED;
	/* the short-read presets' device post stages (aln_plan_sr, mmg_aln.h) do not bound the extension of a self-chain (MM_SEED_SELF) */
	if ((opt->flag & (MM_F_NO_DIAG | MM_F_NO_DUAL)) && (opt->flag & MM_F_SR))
		return "the self/dual-hit filters of the all-vs-all modes (-D, -X, --dual=no, ava-ont, ava-pb; map.c:128-137)" NOT_SUPPORTED;
	if (opt->sdust_thres > 0) return "SDUST masking of query minimizers (-T, map.c:41-62)" NOT_SUPPORTED;
	if (opt->split_prefix) return "--split-prefix (the index is a single part in HBM)" NOT_SUPPORTED;
	return 0;
#undef NOT_SUPPORTED
}

int mm_b200_check_opt(const mm_mapopt_t *opt)
{
	const char *msg = mm_b200_opt_error(opt);
	if (msg == 0) return 0;
	fprintf(stderr, "[ERROR] %s\n", msg);
	return -1;
}

mm_tbuf_t *mm_tbuf_init(void) { return (mm_tbuf_t*)calloc(1, sizeof(mm_tbuf_t)); }
void mm_tbuf_destroy(mm_tbuf_t *b) { free(b); }

/* what the request queue maps a round with: the batch path on every GPU of the index */
static int apiq_map_batches(void *round, step_t **b, int n)
{
	const mm_apiq_round_t *r = (const mm_apiq_round_t*)round;
	return mm_b200_map_batches(r->mi, r->opt, r->n_threads, (mm_b200_batch_t**)b, n, 0);
}

void mm_map_frag(const mm_idx_t *mi, int n_segs, const int *qlens, const char **seqs, int *n_regs, mm_reg1_t **regs, mm_tbuf_t *b,
                 const mm_mapopt_t *opt, const char *qname)
{ /* map.c:272-424, for the fragments of all concurrent callers at once */
	int j, rep_len = 0, frag_gap = 0;
	for (j = 0; j < n_segs; ++j) n_regs[j] = 0, regs[j] = 0;
	if (n_segs <= 0 || n_segs > MM_MAX_SEG) return;
	if (mi == 0 || mi->B == 0 || mi->B->n_dev < 1) { fprintf(stderr, "[ERROR] the index is not resident on a GPU\n"); exit(1); }
	if (mm_b200_check_opt(opt) < 0 || (use_name_filters(opt) && mm_b200_name_keys_ready(mi) < 0)) exit(1);
	mm_apiq_map_frag(mi, apiq_map_batches, mm_b200_batches_in_flight, opt, n_segs, qlens, seqs, qname, n_regs, regs, &rep_len, &frag_gap);
	if (b) b->rep_len = rep_len, b->frag_gap = frag_gap;
}

mm_reg1_t *mm_map(const mm_idx_t *mi, int qlen, const char *seq, int *n_regs, mm_tbuf_t *b, const mm_mapopt_t *opt, const char *qname)
{
	mm_reg1_t *regs;
	mm_map_frag(mi, 1, &qlen, &seq, n_regs, &regs, b, opt, qname);
	return regs;
}

/* ------------------------------------------------------------------ batch API (what bench.py and embedders call) */

struct mm_b200_reader_s { pipeline_t pl; };

mm_b200_reader_t *mm_b200_open_reads(int n_fp, const char **fn)
{
	mm_b200_reader_t *r = (mm_b200_reader_t*)calloc(1, sizeof(*r));
	int i;
	r->pl.n_fp = n_fp;
	r->pl.fp = (mm_bseq_file_t**)calloc(n_fp, sizeof(mm_bseq_file_t*));
	for (i = 0; i < n_fp; ++i)
		if ((r->pl.fp[i] = mm_bseq_open(fn[i])) == 0) {
			int j;
			for (j = 0; j < i; ++j) mm_bseq_close(r->pl.fp[j]);
			free(r->pl.fp); free(r);
			return 0;
		}
	for (i = 0; i < n_fp; ++i) mm_bseq_set_readahead(r->pl.fp[i], 1);
	return r;
}

void mm_b200_close_reads(mm_b200_reader_t *r)
{
	int i;
	if (r == 0) return;
	for (i = 0; i < r->pl.n_fp; ++i) mm_bseq_close(r->pl.fp[i]);
	free(r->pl.fp); free(r->pl.str.s); free(r);
}

mm_b200_batch_t *mm_b200_read_batch(mm_b200_reader_t *r, const mm_mapopt_t *opt, int batch_bases)
{
	r->pl.opt = opt, r->pl.mini_batch_size = batch_bases;
	return (mm_b200_batch_t*)step_read(&r->pl);
}

void mm_b200_batch_info(const mm_b200_batch_t *b, int *n_seq, int *n_frag, int64_t *n_bases)
{
	const step_t *s = (const step_t*)b;
	int64_t t = 0;
	int i;
	for (i = 0; i < s->n_seq; ++i) t += s->seq[i].l_seq;
	if (n_seq) *n_seq = s->n_seq;
	if (n_frag) *n_frag = s->n_frag;
	if (n_bases) *n_bases = t;
}

int mm_b200_map_batch(const mm_idx_t *mi, const mm_mapopt_t *opt, int n_threads, mm_b200_batch_t *b, int mode)
{
	return map_step_group(mi, opt, n_threads > 1 ? n_threads : 1, (step_t*)b, mode_ops(mode), 0, 1, 0);
}

/* drop the hits of a mapped batch so that it can be mapped again */
void mm_b200_reset_batch(mm_b200_batch_t *b)
{
	step_t *s = (step_t*)b;
	int i, j;
	for (i = 0; i < s->n_seq; ++i) {
		for (j = 0; j < s->n_reg[i]; ++j) free(s->reg[i][j].p);
		free(s->reg[i]);
		s->reg[i] = 0, s->n_reg[i] = 0;
	}
}

/* order-independent digest of the hits of a batch (coordinates, strand, MAPQ, CIGAR, scores) */
uint64_t mm_b200_batch_digest(const mm_b200_batch_t *b, int64_t *n_hits)
{
	const step_t *s = (const step_t*)b;
	uint64_t h = 1469598103934665603ULL;
	int64_t n = 0;
	int i, j;
	uint32_t k;
#define MIX(v) do { h ^= (uint64_t)(v); h *= 1099511628211ULL; } while (0)
	for (i = 0; i < s->n_seq; ++i)
		for (j = 0; j < s->n_reg[i]; ++j) {
			const mm_reg1_t *r = &s->reg[i][j];
			MIX(i); MIX(r->rid); MIX(r->rs); MIX(r->re); MIX(r->qs); MIX(r->qe); MIX(r->rev); MIX(r->mapq); MIX(r->score); MIX(r->parent == r->id);
			if (r->p) { MIX(r->p->dp_max); MIX(r->p->dp_score); for (k = 0; k < r->p->n_cigar; ++k) MIX(r->p->cigar[k]); }
			++n;
		}
#undef MIX
	if (n_hits) *n_hits = n;
	return h;
}

/* the hits of a mapped batch as rows of MM_B200_HIT_COLS integers, in read order, and their CIGARs concatenated in the same order */
int64_t mm_b200_batch_hits(const mm_b200_batch_t *b, int64_t *rows, uint32_t *cigar, int64_t *n_cigar)
{
	const step_t *s = (const step_t*)b;
	int64_t n = 0, nc = 0;
	int i, j;
	for (i = 0; i < s->n_seq; ++i)
		for (j = 0; j < s->n_reg[i]; ++j, ++n) {
			const mm_reg1_t *r = &s->reg[i][j];
			const uint32_t k = r->p ? r->p->n_cigar : 0;
			if (rows) {
				int64_t *o = rows + n * MM_B200_HIT_COLS;
				o[0] = i, o[1] = r->rid, o[2] = r->rs, o[3] = r->re, o[4] = r->qs, o[5] = r->qe, o[6] = r->rev, o[7] = r->mapq;
				o[8] = r->score, o[9] = r->parent == r->id, o[10] = r->sam_pri, o[11] = r->proper_frag, o[12] = r->mlen, o[13] = r->blen;
				o[14] = r->p ? r->p->dp_score : 0, o[15] = r->p ? r->p->dp_max : 0, o[16] = k;
			}
			if (cigar && k) memcpy(cigar + nc, r->p->cigar, k * sizeof(uint32_t));
			nc += k;
		}
	if (n_cigar) *n_cigar = nc;
	return n;
}

void mm_b200_write_batch(const mm_idx_t *mi, const mm_mapopt_t *opt, mm_b200_batch_t *b)
{
	pipeline_t pl;
	memset(&pl, 0, sizeof(pl));
	pl.opt = opt, pl.mi = mi;
	step_write(&pl, (step_t*)b);
	free(pl.str.s);
}

void mm_b200_free_batch(mm_b200_batch_t *b)
{
	step_t *s = (step_t*)b;
	int i;
	mm_b200_reset_batch(b);
	for (i = 0; i < s->n_seq; ++i) mm_bseq_free1(&s->seq[i], 1);
	free(s->reg); free(s->n_reg); free(s->seq); free(s);
}

mmg_ctx_t *mm_b200_ctx(const mm_idx_t *mi, int dev_slot) { return mi->B->ctx[dev_slot]; }
int mm_b200_n_devices(const mm_idx_t *mi) { return mi->B->n_dev; }

void mm_b200_profile(const mm_idx_t *mi, int enable)
{
	int d;
	for (d = 0; d < mi->B->n_dev * mi->B->lanes; ++d) mmg_profile_enable(mi->B->ctx[d], enable);
}

/* per-kernel device time and launch counts since profiling was enabled (device slot 0..n-1 summed) */
int mm_b200_profile_fetch(const mm_idx_t *mi, int max, const char **names, double *ms, long *launches)
{
	int d, n = 0, i, j;
	for (d = 0; d < mi->B->n_dev * mi->B->lanes; ++d) {
		const char *nm[64]; double t[64]; long l[64];
		const int k = mmg_profile_fetch(mi->B->ctx[d], 64, nm, t, l);
		for (i = 0; i < k; ++i) {
			for (j = 0; j < n; ++j) if (strcmp(names[j], nm[i]) == 0) break;
			if (j == n) { if (n == max) continue; names[n] = nm[i], ms[n] = 0, launches[n] = 0, ++n; }
			ms[j] += t[i], launches[j] += l[i];
		}
	}
	return n;
}

void mm_b200_report(const mm_idx_t *mi, FILE *fp)
{
	mm_b200_stats_t s;
	const char *nm[64]; double t[64]; long l[64];
	int i, n;
	mm_b200_stats(&s, 0);
	fprintf(fp, "[M::b200] batches: %.3f s total = upload %.3f + seed/chain %.3f (kernels %.3f) + hits %.3f + align host %.3f + DP %.3f (kernel %.3f) + finish %.3f\n",
			s.t_total, s.t_upload, s.t_seedchain, s.t_seedchain_kernels, s.t_hits, s.t_align_host, s.t_ksw_total, s.t_ksw_kernel, s.t_finish);
	fprintf(fp, "[M::b200] reads %lu, bases %lu, minimizers %lu, anchors %lu, chain iterations %lu, DP jobs %lu in %lu rounds, DP cells %lu, H2D %lu B, D2H %lu B\n",
			(unsigned long)s.n_reads, (unsigned long)s.n_bases, (unsigned long)s.n_minimizers, (unsigned long)s.n_anchors, (unsigned long)s.n_chain_iter,
			(unsigned long)s.n_dp_jobs, (unsigned long)s.n_dp_rounds, (unsigned long)s.n_dp_cells, (unsigned long)s.h2d_bytes, (unsigned long)s.d2h_bytes);
	n = mm_b200_profile_fetch(mi, 64, nm, t, l);
	for (i = 0; i < n; ++i) fprintf(fp, "[M::b200] kernel %-18s %8ld launches %10.3f ms\n", nm[i], l[i], t[i]);
	{
		uint64_t pc[8];
		mm_b200_path_counts(mi, pc, 0);
		fprintf(fp, "[M::b200] paths: rechained %lu, heap_rank_replay %lu, heap_literal_replay %lu, warp_tree %lu, zdrop_rounds %lu, zdrop_cuts %lu\n",
				(unsigned long)pc[0], (unsigned long)pc[1], (unsigned long)pc[2], (unsigned long)pc[3], (unsigned long)pc[4], (unsigned long)pc[5]);
	}
}

void mm_b200_path_counts(const mm_idx_t *mi, uint64_t out[8], int reset)
{ /* work items that took each data-dependent device path (mmg_path_counts), summed over the shards' contexts */
	int d, i;
	for (i = 0; i < 8; ++i) out[i] = 0;
	for (d = 0; d < mi->B->n_dev * mi->B->lanes; ++d) {
		uint64_t t[8];
		mmg_path_counts(mi->B->ctx[d], t, reset);
		for (i = 0; i < 8; ++i) out[i] += t[i];
	}
}

long mm_b200_launch_count(const mm_idx_t *mi, int reset)
{
	long n = 0;
	int d;
	for (d = 0; d < mi->B->n_dev * mi->B->lanes; ++d) n += mmg_launch_count(mi->B->ctx[d], reset);
	return n;
}
