/* Drives the mm_map_frag request queue (airlift_b200/host/apiq.c) from many threads with a fake batch mapper, built with
 * ThreadSanitizer by tests/test_api_queue_tsan.py.
 *
 * The fake writes one mm_reg1_t per segment whose fields encode the segment's bytes and the identity of the options the round
 * was mapped with; every caller checks that it got exactly its own result.  The fake also counts batches that mix option
 * sets, batches above the base cap, and rounds of more than one fragment.  One line of counts goes to stdout. */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <dirent.h>
#include <unistd.h>
#include "mm2b_priv.h"

#define N_OPT 3
#define CAP   1500 /* mini_batch_size of every option set: small, so that a backlog needs two batches */

static mm_idx_t g_mi;
static mm_mapopt_t g_opt[N_OPT];
static int g_n_threads, g_n_calls;
/* written by the dispatcher only, read after it was joined */
static long n_rounds, n_batches, n_two_batch_rounds, n_multi_frag, max_frag, n_mixed, n_over_cap, n_bad_opt;
static int n_errors; /* callers */

static uint32_t fnv(const char *s, int l)
{
	uint32_t h = 2166136261u;
	int i;
	for (i = 0; i < l; ++i) h = (h ^ (uint8_t)s[i]) * 16777619u;
	return h;
}

static int opt_id_of_name(const char *name)
{
	const char *p = strrchr(name, 'o');
	return p ? atoi(p + 1) : -1;
}

static int fake_map(void *round, step_t **b, int n)
{
	const mm_apiq_round_t *r = (const mm_apiq_round_t*)round;
	const int id = r->opt->seed - 11; /* the option sets differ in their seed */
	int i, f, j;
	++n_rounds, n_batches += n;
	if (n > 1) ++n_two_batch_rounds;
	if (r->mi != &g_mi || r->n_threads < 1 || r->n_threads > 16 || r->opt->pe_ori > 0 || (r->opt->flag & MM_F_INDEPEND_SEG)) ++n_bad_opt;
	for (i = 0; i < n; ++i) {
		step_t *s = b[i];
		int64_t bases = 0;
		if (s->n_frag > 1) ++n_multi_frag;
		if (s->n_frag > max_frag) max_frag = s->n_frag;
		for (f = 0; f < s->n_frag; ++f) {
			const int off = s->seg_off[f];
			if (opt_id_of_name(s->seq[off].name) != id) ++n_mixed;
			for (j = 0; j < s->n_seg[f]; ++j) {
				const mm_bseq1_t *t = &s->seq[off + j];
				mm_reg1_t *g = (mm_reg1_t*)calloc(1, sizeof(mm_reg1_t));
				if (t->seq[t->l_seq] != 0) ++n_bad_opt; /* the copies are NUL-terminated */
				g->rid = id, g->qs = t->l_seq, g->hash = fnv(t->seq, t->l_seq), g->score = j, g->cnt = s->n_seg[f];
				s->n_reg[off + j] = 1, s->reg[off + j] = g;
				s->rep_len[off + j] = (int)(fnv(t->name, (int)strlen(t->name)) & 0xffff), s->frag_gap[off + j] = 1000 * id + s->n_seg[f];
				bases += t->l_seq;
			}
		}
		if (s->n_frag > 1 && bases > CAP) ++n_over_cap;
	}
	usleep(200); /* a device round trip: lets a backlog build up */
	return 0;
}

static int fake_in_flight(const mm_idx_t *mi, const mm_mapopt_t *opt) { (void)mi; (void)opt; return 2; }

static void *caller(void *data)
{
	const int tid = (int)(long)data;
	unsigned seed = 1234u + tid;
	char buf[2][320], name[64];
	int c, j, k;
	for (c = 0; c < g_n_calls; ++c) {
		const int id = (tid + c) % N_OPT, n_segs = 1 + (rand_r(&seed) & 1);
		int qlens[2], n_regs[2], rep_len = -1, frag_gap = -1, bad = 0;
		const char *seqs[2] = {buf[0], buf[1]};
		mm_reg1_t *regs[2];
		for (j = 0; j < n_segs; ++j) {
			qlens[j] = 20 + rand_r(&seed) % 280;
			for (k = 0; k < qlens[j]; ++k) buf[j][k] = "ACGT"[rand_r(&seed) & 3];
			buf[j][qlens[j]] = 'X'; /* not NUL-terminated: the queue copies qlens[j] bytes */
		}
		snprintf(name, sizeof(name), "t%d.c%d.o%d", tid, c, id);
		mm_apiq_map_frag(&g_mi, fake_map, fake_in_flight, &g_opt[id], n_segs, qlens, seqs, name, n_regs, regs, &rep_len, &frag_gap);
		for (j = 0; j < n_segs; ++j) {
			const mm_reg1_t *g = regs[j];
			if (n_regs[j] != 1 || g == 0 || g->rid != id || g->qs != qlens[j] || g->hash != fnv(buf[j], qlens[j]) || g->score != j || g->cnt != n_segs) bad = 1;
			free(regs[j]);
		}
		if (rep_len != (int)(fnv(name, (int)strlen(name)) & 0xffff) || frag_gap != 1000 * id + n_segs) bad = 1;
		if (bad) __atomic_fetch_add(&n_errors, 1, __ATOMIC_RELAXED);
	}
	return 0;
}

static int n_tasks(void)
{
	DIR *d = opendir("/proc/self/task");
	struct dirent *e;
	int n = 0;
	if (d == 0) return -1;
	while ((e = readdir(d)) != 0) if (e->d_name[0] != '.') ++n;
	closedir(d);
	return n;
}

/* joined threads may linger in /proc for a moment (want < 0: wait until the count stops changing) */
static int n_tasks_settled(int want)
{
	int i, n = n_tasks(), prev = -2;
	for (i = 0; i < 200 && (want < 0 ? n != prev : n != want); ++i) { usleep(10000); prev = n, n = n_tasks(); }
	return n;
}

static void *idle(void *data) { return data; }

int main(int argc, char *argv[])
{
	pthread_t *tid;
	int i, t_before, t_running, t_after;
	g_n_threads = argc > 1 ? atoi(argv[1]) : 32;
	g_n_calls = argc > 2 ? atoi(argv[2]) : 2000;
	g_mi.B = (struct mm_idx_bucket_s*)calloc(1, sizeof(struct mm_idx_bucket_s));
	pthread_mutex_init(&g_mi.B->apiq_mu, 0);
	for (i = 0; i < N_OPT; ++i) {
		memset(&g_opt[i], 0xa5, sizeof(mm_mapopt_t)); /* padding differs from set to set; the fields decide */
		g_opt[i].flag = MM_F_SR | MM_F_CIGAR, g_opt[i].seed = 11 + i, g_opt[i].pe_ori = 0, g_opt[i].mini_batch_size = CAP;
		g_opt[i].split_prefix = 0, g_opt[i].mask_level = 0.5f, g_opt[i].pri_ratio = 0.8f, g_opt[i].min_join_flank_ratio = 0.5f;
		g_opt[i].max_clip_ratio = 1.0f, g_opt[i].mid_occ_frac = 2e-4f;
	}
	g_opt[1].pe_ori = 0 << 1 | 1;                    /* FR: normalised to 0 */
	g_opt[2].flag |= MM_F_INDEPEND_SEG;              /* cleared: mm_map_frag maps jointly */
	tid = (pthread_t*)calloc(g_n_threads, sizeof(pthread_t));
	pthread_create(&tid[0], 0, idle, 0); /* the sanitizer starts its own helper thread with the first thread: counted from here */
	pthread_join(tid[0], 0);
	t_before = n_tasks_settled(-1);
	for (i = 0; i < g_n_threads; ++i) pthread_create(&tid[i], 0, caller, (void*)(long)i);
	for (i = 0; i < g_n_threads; ++i) pthread_join(tid[i], 0);
	t_running = n_tasks_settled(t_before + 1); /* the dispatcher */
	mm_apiq_stop(g_mi.B);
	t_after = n_tasks_settled(t_before);
	printf("calls %ld errors %d rounds %ld batches %ld two_batch_rounds %ld multi_frag %ld max_frag %ld mixed %ld over_cap %ld bad_opt %ld "
		   "tasks_before %d tasks_running %d tasks_after %d\n", (long)g_n_threads * g_n_calls, n_errors, n_rounds, n_batches, n_two_batch_rounds,
		   n_multi_frag, max_frag, n_mixed, n_over_cap, n_bad_opt, t_before, t_running, t_after);
	free(tid);
	pthread_mutex_destroy(&g_mi.B->apiq_mu);
	free(g_mi.B);
	return 0;
}
