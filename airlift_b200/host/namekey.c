/* namekey.c -- the name order the self/dual-hit filters need (-D, -X, --dual=no, ava-ont, ava-pb; skip_seed, map.c:125-147).
 * The device never sees a name, only the integer keys described under "name keys" in include/mmg.h; this module is the one
 * place that builds them: target keys once per index, unit keys per mini-batch. */
#include <stdio.h>
#include "mm2b_priv.h"

static inline const char *name_or_empty(const char *s) { return s ? s : ""; }

static int cmp_name(const void *a, const void *b) { return strcmp(*(const char *const*)a, *(const char *const*)b); }

void mm_b200_name_order(int n, const char *const *names, const char **sorted, uint32_t *tkey)
{
	int i;
	for (i = 0; i < n; ++i) sorted[i] = name_or_empty(names[i]);
	qsort(sorted, n, sizeof(char*), cmp_name);
	for (i = 0; i < n; ++i) { /* 2 * (number of names below) + 1, by binary search in the sorted names */
		const char *s = name_or_empty(names[i]);
		int lo = 0, hi = n;
		while (lo < hi) { const int mid = (lo + hi) >> 1; if (strcmp(sorted[mid], s) < 0) lo = mid + 1; else hi = mid; }
		tkey[i] = 2 * (uint32_t)lo + 1;
	}
}

uint32_t mm_b200_name_ukey(int n, const char *const *sorted, const char *qname)
{
	int lo = 0, hi = n;
	if (qname == 0) return MMG_NAME_NONE;
	while (lo < hi) { const int mid = (lo + hi) >> 1; if (strcmp(sorted[mid], qname) < 0) lo = mid + 1; else hi = mid; }
	return 2 * (uint32_t)lo + (lo < n && strcmp(sorted[lo], qname) == 0 ? 1 : 0);
}

int mm_b200_name_keys_ready(const mm_idx_t *mi)
{ /* the target keys of the index on every device replica, computed on first use */
	struct mm_idx_bucket_s *B = mi->B;
	int rc = 0, d;
	pthread_mutex_lock(&B->key_mu);
	if (B->sorted_names == 0) {
		const char **names = (const char**)malloc(((size_t)mi->n_seq + 1) * sizeof(char*));
		uint32_t *tkey = (uint32_t*)malloc(((size_t)mi->n_seq + 1) * 4), i;
		B->sorted_names = (const char**)malloc(((size_t)mi->n_seq + 1) * sizeof(char*));
		for (i = 0; i < mi->n_seq; ++i) names[i] = mi->seq[i].name;
		mm_b200_name_order((int)mi->n_seq, names, B->sorted_names, tkey);
		for (d = 0; d < B->n_dev && rc == 0; ++d)
			if (mmg_idx_set_name_keys(B->didx[d], tkey) != MMG_OK) {
				fprintf(stderr, "[ERROR] cannot upload the target name keys: %s\n", mmg_last_error());
				rc = -1;
			}
		if (rc) { free(B->sorted_names); B->sorted_names = 0; }
		free(names); free(tkey);
	}
	pthread_mutex_unlock(&B->key_mu);
	return rc;
}

uint32_t mm_b200_unit_key(const mm_idx_t *mi, const char *qname)
{
	return mm_b200_name_ukey((int)mi->n_seq, mi->B->sorted_names, qname);
}
