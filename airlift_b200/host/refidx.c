/* refidx.c -- the host face of the index: read the reference FASTA, have the device build the minimizer
 * table (mmg_idx_build), keep names / lengths / the 4-bit sequence for the host-side stages.
 * Reference: index.c (mm_idx_reader_*, mm_idx_gen, mm_idx_str, mm_idx_getseq, mm_idx_cal_max_occ, mm_idx_stat). */
#include <stdio.h>
#include <fcntl.h>
#include <unistd.h>
#include "mm2b_priv.h"

static int g_n_dev = 1, g_dev[16] = {0}, g_lanes = 2;

int mm_b200_set_lanes(int lanes)
{
	if (lanes < 1 || lanes > MM_B200_MAX_LANES) return -1;
	g_lanes = lanes;
	return 0;
}

int mm_b200_set_devices(int n_gpus, const int *dev_ids)
{
	int i;
	if (n_gpus < 1 || n_gpus > 16) return -1;
	g_n_dev = n_gpus;
	for (i = 0; i < n_gpus; ++i) g_dev[i] = dev_ids ? dev_ids[i] : i;
	return 0;
}

static void die_gpu(const char *what)
{
	fprintf(stderr, "[ERROR] %s: %s\n", what, mmg_last_error());
	exit(1);
}

/* an mm_idx_t with names, lengths and the GPU contexts, without its device index yet */
static mm_idx_t *idx_shell(int w, int k, int b, int flag, int n, const uint32_t *len, char **name)
{
	mm_idx_t *mi = (mm_idx_t*)calloc(1, sizeof(mm_idx_t));
	struct mm_idx_bucket_s *B = (struct mm_idx_bucket_s*)calloc(1, sizeof(*B));
	uint64_t sum = 0;
	int i, d;
	if (k * 2 < b) b = k * 2;
	if (w < 1) w = 1;
	mi->w = w, mi->k = k, mi->b = b, mi->flag = flag, mi->n_seq = n, mi->B = B;
	mi->seq = (mm_idx_seq_t*)calloc(n, sizeof(mm_idx_seq_t));
	for (i = 0; i < n; ++i) {
		mi->seq[i].name = (name && name[i] && !(flag & MM_I_NO_NAME)) ? strdup(name[i]) : 0;
		mi->seq[i].len = len[i], mi->seq[i].offset = sum;
		sum += len[i];
	}
	B->n_dev = g_n_dev;
	B->lanes = g_lanes;
	pthread_mutex_init(&B->apiq_mu, 0);
	pthread_mutex_init(&B->key_mu, 0);
	for (d = 0; d < g_n_dev; ++d) {
		int l;
		pthread_mutex_init(&B->gpu_token[d], 0);
		pthread_mutex_init(&B->up_token[d], 0);
		B->dev_id[d] = g_dev[d];
		for (l = 0; l < B->lanes; ++l)
			if (mmg_init(g_dev[d], &B->ctx[d * B->lanes + l]) != MMG_OK) die_gpu("cannot initialise the GPU");
	}
	return mi;
}

static void idx_replicate(mm_idx_t *mi)
{
	int d;
	for (d = 1; d < mi->B->n_dev; ++d) /* replicate over NVLink; nothing else ever crosses GPUs */
		if (mmg_idx_clone_to(mi->B->ctx[d * mi->B->lanes], mi->B->didx[0], &mi->B->didx[d]) != MMG_OK) die_gpu("index replication failed");
}

/* build the device index from in-memory sequences and wrap it in an mm_idx_t */
static mm_idx_t *idx_from_seqs(int w, int k, int b, int flag, int n, char **seq, const uint32_t *len, char **name)
{
	mm_idx_t *mi = idx_shell(w, k, b, flag, n, len, name);
	uint64_t sum = 0;
	int i;
	for (i = 0; i < n; ++i) sum += len[i];
	if (mmg_idx_build(mi->B->ctx[0], mi->w, k, !!(flag & MM_I_HPC), n, (const char *const*)seq, len, &mi->B->didx[0]) != MMG_OK) die_gpu("index construction failed");
	idx_replicate(mi);
	/* the host keeps the packed sequence: CIGAR post-processing and cs/MD read it (index.c:152-162) */
	mi->S = (uint32_t*)calloc((sum + 7) / 8 + 1, 4);
	if (mmg_idx_copy_S(mi->B->didx[0], mi->S) != MMG_OK) die_gpu("cannot fetch the packed reference");
	return mi;
}

void mm_idx_destroy(mm_idx_t *mi)
{
	uint32_t i;
	int d;
	if (mi == 0) return;
	if (mi->B) {
		mm_apiq_stop(mi->B); /* no thread outlives the index */
		for (d = 0; d < mi->B->n_dev; ++d) mmg_idx_free(mi->B->didx[d]);
		for (d = 0; d < mi->B->n_dev * mi->B->lanes; ++d) mmg_destroy(mi->B->ctx[d]);
		free(mi->B->sorted_names);
		free(mi->B);
	}
	for (i = 0; i < mi->n_seq; ++i) free(mi->seq[i].name);
	free(mi->seq); free(mi->S); free(mi);
}

mm_idx_t *mm_idx_str(int w, int k, int is_hpc, int bucket_bits, int n, const char **seq, const char **name)
{ /* index.c:385-432 */
	uint32_t *len;
	mm_idx_t *mi;
	int i, flag = 0;
	if (n <= 0) return 0;
	if (is_hpc) flag |= MM_I_HPC;
	if (name == 0) flag |= MM_I_NO_NAME;
	if (bucket_bits < 0) bucket_bits = 14;
	len = (uint32_t*)malloc((size_t)n * 4);
	for (i = 0; i < n; ++i) len[i] = (uint32_t)strlen(seq[i]);
	mi = idx_from_seqs(w, k, bucket_bits, flag, n, (char**)seq, len, (char**)name);
	free(len);
	return mi;
}

int mm_idx_getseq(const mm_idx_t *mi, uint32_t rid, uint32_t st, uint32_t en, uint8_t *seq)
{ /* index.c:152-162 */
	uint64_t i, st1, en1;
	if (mi->S == 0 || rid >= mi->n_seq || st >= mi->seq[rid].len) return -1; /* S: null for an index loaded without sequences */
	if (en > mi->seq[rid].len) en = mi->seq[rid].len;
	st1 = mi->seq[rid].offset + st, en1 = mi->seq[rid].offset + en;
	for (i = st1; i < en1; ++i) seq[i - st1] = mm_seq4_get(mi->S, i);
	return (int)(en - st);
}

int mm_idx_name2id(const mm_idx_t *mi, const char *name)
{ /* a linear scan: bindings look a name up once per call, and the index keeps no name table */
	uint32_t i;
	if (name == 0) return -1;
	for (i = 0; i < mi->n_seq; ++i)
		if (mi->seq[i].name && strcmp(mi->seq[i].name, name) == 0) return (int)i;
	return -1;
}

int32_t mm_idx_cal_max_occ(const mm_idx_t *mi, float f)
{
	int32_t t = 0;
	if (mmg_idx_cal_max_occ(mi->B->didx[0], f, &t) != MMG_OK) die_gpu("mm_idx_cal_max_occ");
	return t;
}

void mm_idx_stat(const mm_idx_t *mi)
{ /* index.c:100-122 */
	uint64_t len = 0;
	uint32_t i;
	const int64_t n = mmg_idx_n_keys(mi->B->didx[0]), sum = mmg_idx_n_minimizers(mi->B->didx[0]);
	extern int64_t mmg_idx_n_singletons(const mmg_idx_t *idx);
	const int64_t n1 = mmg_idx_n_singletons(mi->B->didx[0]);
	fprintf(stderr, "[M::%s] kmer size: %d; skip: %d; is_hpc: %d; #seq: %d\n", __func__, mi->k, mi->w, mi->flag & MM_I_HPC, mi->n_seq);
	for (i = 0; i < mi->n_seq; ++i) len += mi->seq[i].len;
	fprintf(stderr, "[M::%s::%.3f*%.2f] distinct minimizers: %d (%.2f%% are singletons); average occurrences: %.3lf; average spacing: %.3lf\n",
			__func__, realtime() - mm_realtime0, cputime() / (realtime() - mm_realtime0), (int)n, 100.0 * n1 / n, (double)sum / n, (double)len / sum);
}

/* ---- index files (index.c:438-531).  A .mmi keeps, per bucket, the position array p[] and the (key, value) pairs of a
 * klib hash table in slot order.  The device table has another shape, so mm_idx_dump() asks the device for the keys in
 * bucket order and replays khash's placement (khash.h:232-330) on slot numbers alone: the file comes out byte for byte
 * as the reference writes it.  mm_idx_load() takes the parameters, names and the 4-bit sequence from the file and
 * re-derives the tables on the GPU -- they are a function of exactly those -- then checks the counts the file states.  A file
 * written without sequences (MM_I_NO_SEQ) has nothing to re-derive from: its minimizer lists go to mmg_idx_build_lists. */

typedef struct { int32_t *slot; uint8_t *live, *taken; uint32_t cap; } kh_replay_t;

static void kh_replay_reserve(kh_replay_t *o, uint32_t nb)
{
	if (nb <= o->cap) return;
	o->slot = (int32_t*)realloc(o->slot, (size_t)nb * 4);
	o->live = (uint8_t*)realloc(o->live, nb);
	o->taken = (uint8_t*)realloc(o->taken, nb);
	o->cap = nb;
}

/* Slot of each of n distinct keys inserted in array order into an empty table pre-sized for n (index.c:211-212,219).
 * h[e] is the 32-bit hash of entry e.  Returns the table size; o->slot[i] = entry in slot i, or -1. */
static uint32_t kh_replay(kh_replay_t *o, const uint32_t *h, uint32_t n)
{
	uint32_t nb = 4, bound, e, i, step;
	while (nb < n) nb <<= 1;
	kh_replay_reserve(o, nb);
	memset(o->slot, 0xff, (size_t)nb * 4);
	bound = (uint32_t)(nb * 0.77 + 0.5);
	for (e = 0; e < n; ++e) {
		if (e >= bound) { /* load limit reached: the table doubles and every entry is re-placed where it stands */
			const uint32_t old = nb, mask = nb * 2 - 1;
			uint32_t j;
			nb <<= 1;
			kh_replay_reserve(o, nb);
			for (j = 0; j < old; ++j) o->live[j] = o->slot[j] >= 0;
			memset(o->taken, 0, nb);
			for (j = 0; j < old; ++j) {
				int32_t cur;
				if (!o->live[j]) continue;
				cur = o->slot[j], o->live[j] = 0;
				for (;;) { /* an entry landing on one that has not moved yet takes its place and evicts it */
					for (i = h[cur] & mask, step = 0; o->taken[i]; i = (i + (++step)) & mask) {}
					o->taken[i] = 1;
					if (i < old && o->live[i]) { const int32_t t = o->slot[i]; o->slot[i] = cur, cur = t, o->live[i] = 0; }
					else { o->slot[i] = cur; break; }
				}
			}
			for (j = 0; j < nb; ++j) if (!o->taken[j]) o->slot[j] = -1;
			bound = (uint32_t)(nb * 0.77 + 0.5);
		}
		for (i = h[e] & (nb - 1), step = 0; o->slot[i] >= 0; i = (i + (++step)) & (nb - 1)) {}
		o->slot[i] = (int32_t)e;
	}
	return nb;
}

/* test hook: slot order for n hashes; slot_out must hold 2 * max(4, n rounded up to a power of two) entries */
uint32_t mm_b200_kh_replay(const uint32_t *h, uint32_t n, int32_t *slot_out)
{
	kh_replay_t o = {0, 0, 0, 0};
	const uint32_t nb = kh_replay(&o, h, n);
	memcpy(slot_out, o.slot, (size_t)nb * 4);
	free(o.slot); free(o.live); free(o.taken);
	return nb;
}

#define KEY_ONCE (1ULL << 63)

void mm_idx_dump(FILE *fp, const mm_idx_t *mi)
{
	const int64_t n_keys = mmg_idx_n_keys(mi->B->didx[0]), n_pos = mmg_idx_n_minimizers(mi->B->didx[0]);
	uint64_t *keys = (uint64_t*)malloc((size_t)(n_keys + 1) * 8), *vals = (uint64_t*)malloc((size_t)(n_keys + 1) * 8);
	uint64_t *pos = (uint64_t*)malloc((size_t)(n_pos + 1) * 8), *p = 0, sum_len = 0;
	uint32_t x[5], i, *h = 0, m_h = 0, m_p = 0;
	const uint64_t bmask = (1ULL << mi->b) - 1;
	kh_replay_t o = {0, 0, 0, 0};
	int64_t at = 0;
	if (mmg_idx_export_sorted(mi->B->ctx[0], mi->B->didx[0], mi->b, keys, vals, pos) != MMG_OK) die_gpu("mm_idx_dump");
	x[0] = mi->w, x[1] = mi->k, x[2] = mi->b, x[3] = mi->n_seq, x[4] = mi->flag;
	fwrite(MM_IDX_MAGIC, 1, 4, fp);
	fwrite(x, 4, 5, fp);
	for (i = 0; i < mi->n_seq; ++i) {
		const uint8_t l = mi->seq[i].name ? (uint8_t)strlen(mi->seq[i].name) : 0;
		fwrite(&l, 1, 1, fp);
		if (l) fwrite(mi->seq[i].name, 1, l, fp);
		fwrite(&mi->seq[i].len, 4, 1, fp);
		sum_len += mi->seq[i].len;
	}
	for (i = 0; i < 1U << mi->b; ++i) {
		int64_t end = at;
		uint32_t size, e, nb, n_p = 0, start_p = 0;
		while (end < n_keys && ((keys[end] & ~KEY_ONCE) & bmask) == i) ++end;
		size = (uint32_t)(end - at);
		for (e = 0; e < size; ++e) if (!(keys[at + e] & KEY_ONCE)) n_p += (uint32_t)vals[at + e];
		if (n_p > m_p) { m_p = n_p + (n_p >> 1); p = (uint64_t*)realloc(p, (size_t)m_p * 8); }
		if (size > m_h) { m_h = size + (size >> 1); h = (uint32_t*)realloc(h, (size_t)m_h * 4); }
		for (e = 0; e < size; ++e) { /* p[]: the position lists of the repeated minimizers, in key order (index.c:226-233) */
			const uint64_t k = keys[at + e], v = vals[at + e];
			h[e] = (uint32_t)((k & ~KEY_ONCE) >> mi->b);
			if (!(k & KEY_ONCE)) {
				const uint32_t n = (uint32_t)v;
				memcpy(p + start_p, pos + (v >> 32), (size_t)n * 8);
				vals[at + e] = (uint64_t)start_p << 32 | n;
				start_p += n;
			}
		}
		fwrite(&n_p, 4, 1, fp);
		fwrite(p, 8, n_p, fp);
		fwrite(&size, 4, 1, fp);
		if (size) {
			nb = kh_replay(&o, h, size);
			for (e = 0; e < nb; ++e) {
				uint64_t y[2];
				const int32_t t = o.slot[e];
				if (t < 0) continue;
				y[0] = (keys[at + t] & ~KEY_ONCE) >> mi->b << 1 | keys[at + t] >> 63, y[1] = vals[at + t];
				fwrite(y, 8, 2, fp);
			}
		}
		at = end;
	}
	if (!(mi->flag & MM_I_NO_SEQ)) fwrite(mi->S, 4, (sum_len + 7) / 8, fp);
	fflush(fp);
	free(keys); free(vals); free(pos); free(p); free(h); free(o.slot); free(o.live); free(o.taken);
}

/* The minimizer lists of one index part written without sequences, as mmg_idx_build_lists takes them.  Per bucket i the file
 * holds p[] and the {key, val} pairs of its hash table (index.c:438-477): key = minimizer >> b << 1 | singleton, val = the
 * position of a singleton, else start << 32 | n with start indexing the bucket's p[].  Here: key = minimizer (| KEY_ONCE for a
 * singleton), in the file's order; src = the singleton's position, or the run's first entry in p[], all buckets' p[] in one array. */
typedef struct { int64_t n_keys; uint64_t n_p, m_keys, m_p; uint64_t *key, *src, *p; uint32_t *cnt; } mmi_lists_t;

static void mmi_lists_free(mmi_lists_t *l) { free(l->key); free(l->src); free(l->p); free(l->cnt); }

/* 0; -1 when the file ends early; -2 when a run lies outside its bucket's p[] */
static int mmi_read_lists(FILE *fp, int b, mmi_lists_t *l)
{
	uint64_t *kv = 0, m_kv = 0;
	uint32_t i, j;
	int rc = 0;
	memset(l, 0, sizeof(*l));
	for (i = 0; i < 1U << b && rc == 0; ++i) {
		int32_t n;
		uint32_t size;
		const uint64_t p0 = l->n_p;
		if (fread(&n, 4, 1, fp) != 1 || n < 0) { rc = -1; break; }
		if (l->n_p + n > l->m_p) { l->m_p = l->n_p + n + ((l->n_p + n) >> 1); l->p = (uint64_t*)realloc(l->p, l->m_p * 8); }
		if (fread(l->p + l->n_p, 8, n, fp) != (size_t)n) { rc = -1; break; }
		l->n_p += n;
		if (fread(&size, 4, 1, fp) != 1) { rc = -1; break; }
		if ((uint64_t)l->n_keys + size > l->m_keys) {
			l->m_keys = l->n_keys + size + ((l->n_keys + size) >> 1);
			l->key = (uint64_t*)realloc(l->key, l->m_keys * 8), l->src = (uint64_t*)realloc(l->src, l->m_keys * 8);
			l->cnt = (uint32_t*)realloc(l->cnt, l->m_keys * 4);
		}
		if (2 * (uint64_t)size > m_kv) { m_kv = 2 * (uint64_t)size; kv = (uint64_t*)realloc(kv, m_kv * 8); }
		if (fread(kv, 16, size, fp) != size) { rc = -1; break; }
		for (j = 0; j < size; ++j) {
			const uint64_t y0 = kv[2 * j], y1 = kv[2 * j + 1], m = y0 >> 1 << b | i;
			const int64_t e = l->n_keys++;
			if (y0 & 1) l->key[e] = m | KEY_ONCE, l->cnt[e] = 1, l->src[e] = y1;
			else {
				l->key[e] = m, l->cnt[e] = (uint32_t)y1, l->src[e] = p0 + (y1 >> 32);
				if ((y1 >> 32) + (uint32_t)y1 > (uint64_t)n) { rc = -2; break; }
			}
		}
	}
	free(kv);
	if (rc) mmi_lists_free(l), memset(l, 0, sizeof(*l));
	return rc;
}

/* test hook: the lists of the first part of a no-sequence index file, exactly as mm_idx_load hands them to mmg_idx_build_lists.
 * Returns the number of distinct minimizers, or -1 with the loader's message; free the arrays with mm_b200_mmi_lists_free */
int64_t mm_b200_mmi_lists(const char *fn, uint64_t **key, uint32_t **cnt, uint64_t **src, uint64_t *n_p, uint64_t **p)
{
	FILE *fp = fopen(fn, "rb");
	char magic[4];
	uint32_t x[5], i, len;
	mmi_lists_t l;
	int rc = -1;
	if (fp == 0) return -1;
	if (fread(magic, 1, 4, fp) != 4 || strncmp(magic, MM_IDX_MAGIC, 4) != 0 || fread(x, 4, 5, fp) != 5 || !(x[4] & MM_I_NO_SEQ)) {
		fprintf(stderr, "[ERROR] not an index file written without sequences\n");
		fclose(fp);
		return -1;
	}
	for (i = 0; i < x[3]; ++i) {
		uint8_t nl;
		if (fread(&nl, 1, 1, fp) != 1 || fseeko(fp, nl, SEEK_CUR) != 0 || fread(&len, 4, 1, fp) != 1) break;
	}
	if (i == x[3]) rc = mmi_read_lists(fp, (int)x[2], &l);
	fclose(fp);
	if (rc == -1) { fprintf(stderr, "[ERROR] the index file is truncated\n"); return -1; }
	if (rc < 0) { fprintf(stderr, "[ERROR] the index file lists positions outside their bucket\n"); return -1; }
	*key = l.key, *cnt = l.cnt, *src = l.src, *n_p = l.n_p, *p = l.p;
	return l.n_keys;
}

void mm_b200_mmi_lists_free(uint64_t *key, uint32_t *cnt, uint64_t *src, uint64_t *p) { free(key); free(cnt); free(src); free(p); }

mm_idx_t *mm_idx_load(FILE *fp)
{
	char magic[4], **seq, **name;
	uint32_t x[5], i, *len, *S;
	uint64_t sum_len = 0, off = 0, n_keys = 0, n_listed = 0, j;
	mm_idx_t *mi;
	if (fread(magic, 1, 4, fp) != 4) return 0;
	if (strncmp(magic, MM_IDX_MAGIC, 4) != 0) return 0;
	if (fread(x, 4, 5, fp) != 5) return 0;
	seq = (char**)calloc(x[3], sizeof(char*)), name = (char**)calloc(x[3], sizeof(char*)), len = (uint32_t*)calloc(x[3], 4);
	for (i = 0; i < x[3]; ++i) {
		uint8_t l;
		if (fread(&l, 1, 1, fp) != 1) goto truncated;
		if (l) {
			name[i] = (char*)calloc((size_t)l + 1, 1);
			if (fread(name[i], 1, l, fp) != l) goto truncated;
		}
		if (fread(&len[i], 4, 1, fp) != 1) goto truncated;
		sum_len += len[i];
	}
	if (x[4] & MM_I_NO_SEQ) { /* no sequence to re-derive the tables from: the device builds them from the file's lists */
		mmi_lists_t l;
		const int rc = mmi_read_lists(fp, (int)x[2], &l);
		if (rc == -1) goto truncated;
		if (rc < 0) { fprintf(stderr, "[ERROR] the index file lists positions outside their bucket\n"); exit(1); }
		mi = idx_shell((int)x[0], (int)x[1], (int)x[2], (int)x[4], (int)x[3], len, name);
		if (mmg_idx_build_lists(mi->B->ctx[0], mi->w, mi->k, !!(mi->flag & MM_I_HPC), mi->n_seq, len, l.n_keys, l.key, l.cnt, l.src, l.n_p, l.p,
		                        &mi->B->didx[0]) != MMG_OK)
			die_gpu("index construction failed");
		idx_replicate(mi); /* mi->S stays null: nothing on the host may read the sequence */
		mmi_lists_free(&l);
		for (i = 0; i < x[3]; ++i) free(name[i]);
		free(seq); free(name); free(len);
		return mi;
	}
	for (i = 0; i < 1U << x[2]; ++i) { /* the tables are rebuilt from the sequence; only their sizes are taken from the file */
		int32_t n;
		uint32_t size;
		if (fread(&n, 4, 1, fp) != 1 || fseeko(fp, (off_t)n * 8, SEEK_CUR) != 0) goto truncated;
		if (fread(&size, 4, 1, fp) != 1 || fseeko(fp, (off_t)size * 16, SEEK_CUR) != 0) goto truncated;
		n_listed += (uint64_t)n, n_keys += size;
	}
	S = (uint32_t*)malloc(((sum_len + 7) / 8 + 1) * 4);
	if (fread(S, 4, (sum_len + 7) / 8, fp) != (sum_len + 7) / 8) goto truncated;
	for (i = 0; i < x[3]; ++i) {
		seq[i] = (char*)malloc((size_t)len[i] + 1);
		for (j = 0; j < len[i]; ++j) seq[i][j] = "ACGTN"[mm_seq4_get(S, off + j) > 4 ? 4 : mm_seq4_get(S, off + j)];
		seq[i][len[i]] = 0;
		off += len[i];
	}
	free(S);
	mi = idx_from_seqs((int)x[0], (int)x[1], (int)x[2], (int)x[4], (int)x[3], seq, len, name);
	for (i = 0; i < x[3]; ++i) { free(seq[i]); free(name[i]); }
	free(seq); free(name); free(len);
	if ((uint64_t)mmg_idx_n_keys(mi->B->didx[0]) != n_keys ||
		(uint64_t)(mmg_idx_n_minimizers(mi->B->didx[0]) - mmg_idx_n_singletons(mi->B->didx[0])) != n_listed) {
		fprintf(stderr, "[ERROR] the index file states %llu distinct minimizers and %llu listed positions, its sequences give %lld and %lld\n",
				(unsigned long long)n_keys, (unsigned long long)n_listed, (long long)mmg_idx_n_keys(mi->B->didx[0]),
				(long long)(mmg_idx_n_minimizers(mi->B->didx[0]) - mmg_idx_n_singletons(mi->B->didx[0])));
		exit(1);
	}
	return mi;
truncated:
	fprintf(stderr, "[ERROR] the index file is truncated\n");
	exit(1);
}

/* ---- reader (index.c:533-602) */

int64_t mm_idx_is_idx(const char *fn)
{
	int fd, is_idx = 0;
	int64_t off_end;
	char magic[4];
	if (strcmp(fn, "-") == 0) return 0;
	fd = open(fn, O_RDONLY);
	if (fd < 0) return -1;
	if ((off_end = lseek(fd, 0, SEEK_END)) >= 4) {
		lseek(fd, 0, SEEK_SET);
		if (read(fd, magic, 4) == 4 && strncmp(magic, MM_IDX_MAGIC, 4) == 0) is_idx = 1;
	}
	close(fd);
	return is_idx ? off_end : 0;
}

mm_idx_reader_t *mm_idx_reader_open(const char *fn, const mm_idxopt_t *opt, const char *fn_out)
{
	const int64_t is_idx = mm_idx_is_idx(fn);
	mm_idx_reader_t *r;
	if (is_idx < 0) return 0;
	r = (mm_idx_reader_t*)calloc(1, sizeof(mm_idx_reader_t));
	r->is_idx = is_idx > 0;
	if (opt) r->opt = *opt;
	else mm_idxopt_init(&r->opt);
	if (r->is_idx) {
		r->fp.idx = fopen(fn, "rb");
		r->idx_size = is_idx;
		if (r->fp.idx == 0) { free(r); return 0; }
	} else {
		r->fp.seq = mm_bseq_open(fn);
		if (r->fp.seq == 0) { free(r); return 0; }
	}
	if (fn_out) r->fp_out = fopen(fn_out, "wb");
	return r;
}

void mm_idx_reader_close(mm_idx_reader_t *r)
{
	if (r->is_idx) fclose(r->fp.idx);
	else mm_bseq_close(r->fp.seq);
	if (r->fp_out) fclose(r->fp_out);
	free(r);
}

int mm_idx_reader_eof(const mm_idx_reader_t *r)
{
	return r->is_idx ? (feof(r->fp.idx) || ftello(r->fp.idx) == r->idx_size) : mm_bseq_eof(r->fp.seq);
}

static mm_idx_t *idx_gen(mm_idx_reader_t *r);

mm_idx_t *mm_idx_reader_read(mm_idx_reader_t *r, int n_threads)
{
	mm_idx_t *mi;
	(void)n_threads;
	if (r->is_idx) {
		mi = mm_idx_load(r->fp.idx);
		if (mi && mm_verbose >= 2 && (mi->k != r->opt.k || mi->w != r->opt.w || (mi->flag & MM_I_HPC) != (r->opt.flag & MM_I_HPC)))
			fprintf(stderr, "[WARNING]\033[1;31m Indexing parameters (-k, -w or -H) overridden by parameters used in the prebuilt index.\033[0m\n");
	} else mi = idx_gen(r);
	if (mi) {
		if (r->fp_out) mm_idx_dump(r->fp_out, mi);
		mi->index = r->n_parts++;
	}
	return mi;
}

static mm_idx_t *idx_gen(mm_idx_reader_t *r)
{ /* one index part: sequences are taken in mini-batches until batch_size bases are exceeded (index.c:284-331,353-372) */
	mm_bseq_file_t *fp = r->fp.seq;
	const uint64_t batch_size = r->opt.batch_size;
	const int mini = (uint64_t)r->opt.mini_batch_size < batch_size ? r->opt.mini_batch_size : (int)batch_size;
	char **seq = 0, **name = 0;
	uint32_t *len = 0;
	int n = 0, m = 0, i;
	uint64_t sum_len = 0;
	mm_idx_t *mi;
	if (fp == 0 || mm_bseq_eof(fp)) return 0;
	while (sum_len <= batch_size) {
		int n_seq;
		mm_bseq1_t *s = mm_bseq_read3(fp, mini, 0, 0, 0, &n_seq);
		if (s == 0) break;
		for (i = 0; i < n_seq; ++i) {
			if (n == m) {
				m = m ? m << 1 : 64;
				seq = (char**)realloc(seq, (size_t)m * sizeof(char*)); name = (char**)realloc(name, (size_t)m * sizeof(char*));
				len = (uint32_t*)realloc(len, (size_t)m * 4);
			}
			if (s[i].l_seq == 0 && mm_verbose >= 2) fprintf(stderr, "[WARNING] the length database sequence '%s' is 0\n", s[i].name);
			seq[n] = s[i].seq, name[n] = s[i].name, len[n] = (uint32_t)s[i].l_seq;
			sum_len += (uint64_t)s[i].l_seq;
			++n;
		}
		free(s);
	}
	if (n == 0) return 0;
	mi = idx_from_seqs(r->opt.w, r->opt.k, r->opt.bucket_bits, r->opt.flag, n, seq, len, name);
	for (i = 0; i < n; ++i) { free(seq[i]); free(name[i]); }
	free(seq); free(name); free(len);
	return mi;
}

/* ---- index replication across processes (one process per GPU): rank 0 builds, the others receive the flat
 * device image through a collective the caller runs (bench.py: NCCL broadcast over NVLink) */

int mm_b200_idx_image(const mm_idx_t *mi, mmg_idx_image_t *img) { return mmg_idx_export(mi->B->didx[0], img); }

/* the replica's host side: names/lengths as given, the minimizer table, positions and packed sequence allocated uninitialised on
 * the GPU with the shape given by `shape`; their device pointers are returned in `ptrs` */
mm_idx_t *mm_b200_idx_alloc_named(const mm_idxopt_t *opt, int n_seq, const char *const *names, const uint32_t *lens,
                                  const mmg_idx_image_t *shape, mmg_idx_image_t *ptrs)
{
	mm_idx_t *mi;
	struct mm_idx_bucket_s *B;
	int i, b = opt->bucket_bits;
	uint64_t sum = 0;
	for (i = 0; i < n_seq; ++i) sum += lens[i];
	if (n_seq != shape->n_seq || sum != shape->total_len) {
		fprintf(stderr, "[ERROR] the sequence table does not match the index being received (%d sequences, %lu bases expected)\n", shape->n_seq, (unsigned long)shape->total_len);
		exit(1);
	}
	mi = (mm_idx_t*)calloc(1, sizeof(mm_idx_t));
	B = (struct mm_idx_bucket_s*)calloc(1, sizeof(*B));
	if (opt->k * 2 < b) b = opt->k * 2;
	mi->w = opt->w < 1 ? 1 : opt->w, mi->k = opt->k, mi->b = b, mi->flag = opt->flag, mi->B = B, mi->n_seq = n_seq;
	mi->seq = (mm_idx_seq_t*)calloc(n_seq > 0 ? n_seq : 1, sizeof(mm_idx_seq_t));
	for (i = 0, sum = 0; i < n_seq; ++i) {
		mi->seq[i].name = names && names[i] ? strdup(names[i]) : 0, mi->seq[i].len = lens[i], mi->seq[i].offset = sum;
		sum += lens[i];
	}
	B->n_dev = 1, B->lanes = g_lanes, B->dev_id[0] = g_dev[0];
	pthread_mutex_init(&B->apiq_mu, 0);
	pthread_mutex_init(&B->key_mu, 0);
	pthread_mutex_init(&B->gpu_token[0], 0);
	pthread_mutex_init(&B->up_token[0], 0);
	for (i = 0; i < B->lanes; ++i)
		if (mmg_init(g_dev[0], &B->ctx[i]) != MMG_OK) die_gpu("cannot initialise the GPU");
	*ptrs = *shape;
	if (mmg_idx_alloc_like(B->ctx[0], ptrs, &B->didx[0]) != MMG_OK) die_gpu("cannot allocate the index replica");
	return mi;
}

/* same, names/lengths read from the FASTA the source rank indexed */
mm_idx_t *mm_b200_idx_alloc(const char *fn, const mm_idxopt_t *opt, const mmg_idx_image_t *shape, mmg_idx_image_t *ptrs)
{
	mm_bseq_file_t *fp = mm_bseq_open(fn);
	mm_idx_t *mi;
	char **names = (char**)calloc(shape->n_seq > 0 ? shape->n_seq : 1, sizeof(char*));
	uint32_t *lens = (uint32_t*)calloc(shape->n_seq > 0 ? shape->n_seq : 1, 4);
	int n_seq, i, d = 0;
	if (fp == 0) return 0;
	while (d < shape->n_seq) {
		mm_bseq1_t *s = mm_bseq_read3(fp, 1 << 28, 0, 0, 0, &n_seq);
		if (s == 0) break;
		for (i = 0; i < n_seq && d < shape->n_seq; ++i, ++d) { names[d] = s[i].name, lens[d] = (uint32_t)s[i].l_seq; free(s[i].seq); }
		for (; i < n_seq; ++i) { free(s[i].seq); free(s[i].name); }
		free(s);
	}
	mm_bseq_close(fp);
	mi = mm_b200_idx_alloc_named(opt, d, (const char *const*)names, lens, shape, ptrs);
	for (i = 0; i < d; ++i) free(names[i]);
	free(names); free(lens);
	return mi;
}

/* name and length of sequence i (for callers that replicate the index to other processes) */
int mm_b200_idx_seq(const mm_idx_t *mi, int i, const char **name, uint32_t *len)
{
	if (i < 0 || (uint32_t)i >= mi->n_seq) return -1;
	*name = mi->seq[i].name, *len = mi->seq[i].len;
	return 0;
}

int mm_b200_idx_finalize(mm_idx_t *mi)
{
	uint64_t sum = 0;
	uint32_t i;
	for (i = 0; i < mi->n_seq; ++i) sum += mi->seq[i].len;
	if (mmg_idx_finalize(mi->B->didx[0]) != MMG_OK) die_gpu("index replica");
	if (!mmg_idx_has_seq(mi->B->didx[0])) return 0;
	mi->S = (uint32_t*)calloc((sum + 7) / 8 + 1, 4);
	if (mmg_idx_copy_S(mi->B->didx[0], mi->S) != MMG_OK) die_gpu("cannot fetch the packed reference");
	return 0;
}
