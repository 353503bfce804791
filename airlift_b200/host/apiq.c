/* apiq.c -- the per-fragment API (mm_map_frag / mm_map) served from shared mini-batches.
 *
 * Library clients call mm_map_frag() from many threads, each with its own mm_tbuf_t (map.c:272-424 is re-entrant).  Mapping
 * one fragment per device round trip would leave the GPUs idle between calls, so every call becomes a request in a queue
 * of its index and one dispatcher thread per index maps what is queued when the device comes free: the requests whose
 * options equal those of the oldest one, cut into mini-batches of at most opt->mini_batch_size bases, two of them at once
 * when the batch path keeps two in flight.  Nothing waits for a batch to fill: a lone caller gets one round trip per call.
 * The hits go back to their callers, who own them as before (minimap.h:317-331).
 */
#include <stdio.h>
#include <unistd.h>
#include "mm2b_priv.h"

typedef struct apiq_req_s {
	struct apiq_req_s *next;
	mm_mapopt_t opt;        /* normalised: see apiq_normalise() */
	int n_segs, done;
	int64_t n_bases;
	mm_bseq1_t *seg;        /* [n_segs] copies of the segments; every segment carries the copy of the name */
	int *n_regs, rep_len, frag_gap;
	mm_reg1_t **regs;       /* the caller's arrays */
	pthread_cond_t cv;      /* signalled with done = 1, under the queue's mutex */
} apiq_req_t;

struct mm_apiq_s {
	pthread_mutex_t mu;
	pthread_cond_t cv;      /* a request arrived, or stop */
	apiq_req_t *head, *tail;
	int stop, n_threads;
	pthread_t tid;
	const mm_idx_t *mi;
	mm_apiq_map_f map;
	mm_apiq_in_flight_f in_flight;
};

/* mm_map_frag() maps the segments it is given jointly whatever MM_F_INDEPEND_SEG says (the flag is read by the file driver,
 * worker_for map.c:475-485), and its callers pass them in mapping orientation (worker_for flips the mates around the call,
 * map.c:467-469,486-497): pe_ori = 0 keeps `pe_ori >= 0` (pairing on, map.c:404) while naming no mate to flip */
static void apiq_normalise(mm_mapopt_t *o)
{
	if (o->pe_ori > 0) o->pe_ori = 0;
	o->flag &= ~(int64_t)MM_F_INDEPEND_SEG;
}

static int same_str(const char *a, const char *b) { return a == b || (a && b && strcmp(a, b) == 0); }

/* field by field: the padding of mm_mapopt_t holds whatever the caller's stack held */
static int same_opt(const mm_mapopt_t *a, const mm_mapopt_t *b)
{
#define EQ(f) (a->f == b->f)
	return EQ(flag) && EQ(seed) && EQ(sdust_thres) && EQ(max_qlen) && EQ(bw) && EQ(max_gap) && EQ(max_gap_ref) && EQ(max_frag_len) &&
		EQ(max_chain_skip) && EQ(max_chain_iter) && EQ(min_cnt) && EQ(min_chain_score) && EQ(mask_level) && EQ(pri_ratio) && EQ(best_n) &&
		EQ(max_join_long) && EQ(max_join_short) && EQ(min_join_flank_sc) && EQ(min_join_flank_ratio) && EQ(a) && EQ(b) && EQ(q) && EQ(e) &&
		EQ(q2) && EQ(e2) && EQ(sc_ambi) && EQ(noncan) && EQ(junc_bonus) && EQ(zdrop) && EQ(zdrop_inv) && EQ(end_bonus) && EQ(min_dp_max) &&
		EQ(min_ksw_len) && EQ(anchor_ext_len) && EQ(anchor_ext_shift) && EQ(max_clip_ratio) && EQ(pe_ori) && EQ(pe_bonus) &&
		EQ(mid_occ_frac) && EQ(min_mid_occ) && EQ(mid_occ) && EQ(max_occ) && EQ(mini_batch_size) && EQ(max_sw_mat) &&
		same_str(a->split_prefix, b->split_prefix);
#undef EQ
}

/* the requests of a list as one mini-batch; the segments are the requests' copies, not duplicated again */
static step_t *batch_of(apiq_req_t *r)
{
	step_t *s = (step_t*)calloc(1, sizeof(step_t));
	apiq_req_t *t;
	int j;
	for (t = r; t; t = t->next) s->n_seq += t->n_segs, ++s->n_frag;
	s->seq = (mm_bseq1_t*)calloc(s->n_seq, sizeof(mm_bseq1_t));
	s->n_reg = (int*)calloc(5 * (size_t)s->n_seq, sizeof(int));
	s->seg_off = s->n_reg + s->n_seq, s->n_seg = s->seg_off + s->n_seq, s->rep_len = s->n_seg + s->n_seq, s->frag_gap = s->rep_len + s->n_seq;
	s->reg = (mm_reg1_t**)calloc(s->n_seq, sizeof(mm_reg1_t*));
	s->n_seq = s->n_frag = 0;
	for (t = r; t; t = t->next) {
		s->seg_off[s->n_frag] = s->n_seq, s->n_seg[s->n_frag++] = t->n_segs;
		for (j = 0; j < t->n_segs; ++j, ++s->n_seq) s->seq[s->n_seq] = t->seg[j], s->seq[s->n_seq].rid = s->n_seq;
	}
	return s;
}

/* the hits of each fragment to its request; the caller owns them from here on */
static void batch_hand_back(step_t *s, apiq_req_t *r)
{
	int f, j;
	for (f = 0; r; r = r->next, ++f) {
		const int off = s->seg_off[f];
		for (j = 0; j < r->n_segs; ++j) r->n_regs[j] = s->n_reg[off + j], r->regs[j] = s->reg[off + j];
		r->rep_len = s->rep_len[off], r->frag_gap = s->frag_gap[off];
	}
	free(s->seq); free(s->n_reg); free(s->reg); free(s);
}

/* moves the next round's requests from the queue into lists b[0..n): those with the head's options, in arrival order, cut at
 * opt->mini_batch_size bases per batch (a batch holds at least one request); the others stay queued in their order */
static int take_round(struct mm_apiq_s *q, apiq_req_t **b, mm_mapopt_t *opt)
{
	apiq_req_t **pp = &q->head, *tail[2] = {0, 0};
	int64_t bases[2] = {0, 0};
	int g = 0, n_max;
	*opt = q->head->opt;
	n_max = q->in_flight(q->mi, opt) >= 2 ? 2 : 1;
	b[0] = b[1] = 0;
	while (*pp) {
		apiq_req_t *r = *pp;
		if (!same_opt(&r->opt, opt)) { pp = &r->next; continue; }
		if (b[g] && bases[g] + r->n_bases > opt->mini_batch_size) {
			if (g + 1 == n_max) break;
			++g;
		}
		*pp = r->next, r->next = 0;
		if (tail[g]) tail[g]->next = r;
		else b[g] = r;
		tail[g] = r, bases[g] += r->n_bases;
	}
	for (q->tail = q->head; q->tail && q->tail->next; q->tail = q->tail->next) {}
	return g + 1;
}

static void *apiq_main(void *data)
{
	struct mm_apiq_s *q = (struct mm_apiq_s*)data;
	pthread_mutex_lock(&q->mu);
	for (;;) {
		apiq_req_t *b[2], *r;
		step_t *s[2];
		mm_mapopt_t opt;
		mm_apiq_round_t round;
		int n, i;
		while (q->head == 0 && !q->stop) pthread_cond_wait(&q->cv, &q->mu);
		if (q->head == 0) break; /* stopped, and nothing is left */
		n = take_round(q, b, &opt);
		pthread_mutex_unlock(&q->mu);
		for (i = 0; i < n; ++i) s[i] = batch_of(b[i]);
		round.mi = q->mi, round.opt = &opt, round.n_threads = q->n_threads;
		if (q->map(&round, s, n) != 0) { fprintf(stderr, "[ERROR] mapping failed; no CPU fallback exists\n"); exit(1); }
		for (i = 0; i < n; ++i) batch_hand_back(s[i], b[i]);
		pthread_mutex_lock(&q->mu);
		for (i = 0; i < n; ++i)
			while ((r = b[i]) != 0) { b[i] = r->next; r->done = 1; pthread_cond_signal(&r->cv); } /* r lives on its caller's stack */
	}
	pthread_mutex_unlock(&q->mu);
	return 0;
}

static struct mm_apiq_s *apiq_start(const mm_idx_t *mi, mm_apiq_map_f map, mm_apiq_in_flight_f in_flight)
{
	struct mm_apiq_s *q = (struct mm_apiq_s*)calloc(1, sizeof(*q));
	const long n_cpu = sysconf(_SC_NPROCESSORS_ONLN);
	pthread_mutex_init(&q->mu, 0);
	pthread_cond_init(&q->cv, 0);
	q->mi = mi, q->map = map, q->in_flight = in_flight;
	q->n_threads = n_cpu < 1 ? 1 : n_cpu > 16 ? 16 : (int)n_cpu; /* host stages of a round */
	if (pthread_create(&q->tid, 0, apiq_main, q) != 0) { fprintf(stderr, "[ERROR] cannot start the mapping thread\n"); exit(1); }
	return q;
}

void mm_apiq_stop(struct mm_idx_bucket_s *B)
{
	struct mm_apiq_s *q;
	pthread_mutex_lock(&B->apiq_mu);
	q = B->apiq, B->apiq = 0;
	pthread_mutex_unlock(&B->apiq_mu);
	if (q == 0) return;
	pthread_mutex_lock(&q->mu);
	q->stop = 1;
	pthread_cond_signal(&q->cv);
	pthread_mutex_unlock(&q->mu);
	pthread_join(q->tid, 0);
	pthread_cond_destroy(&q->cv);
	pthread_mutex_destroy(&q->mu);
	free(q);
}

void mm_apiq_map_frag(const mm_idx_t *mi, mm_apiq_map_f map, mm_apiq_in_flight_f in_flight, const mm_mapopt_t *opt, int n_segs,
                      const int *qlens, const char **seqs, const char *qname, int *n_regs, mm_reg1_t **regs, int *rep_len, int *frag_gap)
{
	struct mm_idx_bucket_s *B = mi->B;
	struct mm_apiq_s *q;
	apiq_req_t r;
	char *name = qname ? strdup(qname) : 0;
	int j;
	memset(&r, 0, sizeof(r));
	r.opt = *opt;
	apiq_normalise(&r.opt);
	r.n_segs = n_segs, r.n_regs = n_regs, r.regs = regs;
	r.seg = (mm_bseq1_t*)calloc(n_segs, sizeof(mm_bseq1_t));
	for (j = 0; j < n_segs; ++j) {
		r.seg[j].l_seq = qlens[j], r.seg[j].name = name, r.seg[j].seq = (char*)malloc((size_t)qlens[j] + 1);
		memcpy(r.seg[j].seq, seqs[j], qlens[j]); r.seg[j].seq[qlens[j]] = 0;
		r.n_bases += qlens[j];
	}
	pthread_cond_init(&r.cv, 0);
	pthread_mutex_lock(&B->apiq_mu);
	if (B->apiq == 0) B->apiq = apiq_start(mi, map, in_flight);
	q = B->apiq;
	pthread_mutex_unlock(&B->apiq_mu);
	pthread_mutex_lock(&q->mu);
	if (q->tail) q->tail->next = &r;
	else q->head = &r;
	q->tail = &r;
	pthread_cond_signal(&q->cv);
	while (!r.done) pthread_cond_wait(&r.cv, &q->mu);
	pthread_mutex_unlock(&q->mu);
	pthread_cond_destroy(&r.cv);
	*rep_len = r.rep_len, *frag_gap = r.frag_gap;
	for (j = 0; j < n_segs; ++j) free(r.seg[j].seq);
	free(r.seg); free(name);
}
