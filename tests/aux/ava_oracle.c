/* TEST ORACLE (never linked into the product): collect_seed_hits / collect_seed_hits_heap (map.c:149-247) with the whole of
 * skip_seed (map.c:125-147), restated with the literal names and strcmp -- never the integer name keys the device uses.
 * The index lookup and klib's radix sort come from the plain-C oracle (oracle/mm2_oracle.c), which this file is linked with.
 *
 * tnames/tlens: name and length of every target; qname: the unit's name (NULL turns the self/dual filters off, as in the
 * reference); *n_named: seed hits the self/dual filters dropped. */
#include <stdlib.h>
#include <string.h>
#include "mm2_oracle.h"

#define F_NO_DIAG 0x001
#define F_NO_DUAL 0x002
#define F_FOR_ONLY 0x100000
#define F_REV_ONLY 0x200000
#define SEED_TANDEM (1ULL << 42)
#define SEED_SELF (1ULL << 43)
#define SEED_SEG_SHIFT 48

typedef struct { uint32_t n, q_pos, q_span, seg_id, is_tandem; const uint64_t *cr; } match_t;

/* map.c:125-147; returns 0 (keep), 1 (strand filter) or 2 (self/dual filter) */
static int skip_seed(int64_t flag, uint64_t r, const match_t *q, const char *qname, int qlen, const char *const *tnames,
                     const uint32_t *tlens, int *is_self)
{
	*is_self = 0;
	if (qname && (flag & (F_NO_DIAG | F_NO_DUAL))) {
		const char *tname = tnames[r >> 32] ? tnames[r >> 32] : "";
		const int cmp = strcmp(qname, tname);
		if ((flag & F_NO_DIAG) && cmp == 0 && (int)tlens[r >> 32] == qlen) {
			if ((uint32_t)r >> 1 == (q->q_pos >> 1)) return 2;
			if ((r & 1) == (q->q_pos & 1)) *is_self = 1;
		}
		if ((flag & F_NO_DUAL) && cmp > 0) return 2;
	}
	if (flag & (F_FOR_ONLY | F_REV_ONLY)) {
		if ((r & 1) == (q->q_pos & 1)) { if (flag & F_REV_ONLY) return 1; }
		else if (flag & F_FOR_ONLY) return 1;
	}
	return 0;
}

static void make_anchor(orc128_t *p, uint64_t r, const match_t *q, int qlen, int is_self)
{ /* map.c:176-187 == map.c:232-241 */
	int32_t rpos = (uint32_t)r >> 1;
	if ((r & 1) == (q->q_pos & 1)) {
		p->x = (r & 0xffffffff00000000ULL) | rpos;
		p->y = (uint64_t)q->q_span << 32 | q->q_pos >> 1;
	} else {
		p->x = 1ULL << 63 | (r & 0xffffffff00000000ULL) | rpos;
		p->y = (uint64_t)q->q_span << 32 | (uint32_t)(qlen - ((q->q_pos >> 1) + 1 - q->q_span) - 1);
	}
	p->y |= (uint64_t)q->seg_id << SEED_SEG_SHIFT;
	if (q->is_tandem) p->y |= SEED_TANDEM;
	if (is_self) p->y |= SEED_SELF;
}

static void heap_down(size_t i, size_t n, orc128_t *l)
{ /* ksort.h:43-53 with heap_lt(a,b) = a.x > b.x */
	size_t k = i;
	orc128_t tmp = l[i];
	while ((k = (k << 1) + 1) < n) {
		if (k != n - 1 && l[k].x > l[k + 1].x) ++k;
		if (l[k].x > tmp.x) break;
		l[i] = l[k]; i = k;
	}
	l[i] = tmp;
}

int64_t orc_collect_seeds_named(const orc_idx_t *mi, const char *const *tnames, const uint32_t *tlens, const char *qname, int heap_sort,
                                int64_t flag, int max_occ, int n_mv, const orc128_t *mv, int qlen, orc128_t *a, int *rep_len,
                                int *n_mini_pos, int64_t *n_named)
{
	match_t *m = (match_t*)malloc((n_mv + 1) * sizeof(match_t));
	int i, n_m = 0, rep_st = 0, rep_en = 0, n_mp = 0, is_self, sk;
	int64_t n_a = 0, nn = 0;
	*rep_len = 0;
	for (i = 0; i < n_mv; ++i) { /* collect_matches, map.c:90-123 */
		const orc128_t *p = &mv[i];
		uint32_t q_pos = (uint32_t)p->y, q_span = p->x & 0xff;
		int t;
		const uint64_t *cr = orc_idx_get(mi, p->x >> 8, &t);
		if (t >= max_occ) {
			int en = (q_pos >> 1) + 1, st = en - q_span;
			if (st > rep_en) { *rep_len += rep_en - rep_st; rep_st = st, rep_en = en; }
			else rep_en = en;
		} else {
			match_t *q = &m[n_m++];
			q->q_pos = q_pos, q->q_span = q_span, q->cr = cr, q->n = t, q->seg_id = (uint32_t)(p->y >> 32);
			q->is_tandem = (i > 0 && p->x >> 8 == mv[i - 1].x >> 8) || (i < n_mv - 1 && p->x >> 8 == mv[i + 1].x >> 8);
			n_a += q->n;
			++n_mp;
		}
	}
	*rep_len += rep_en - rep_st;
	*n_mini_pos = n_mp;
	if (a == 0) { free(m); return n_a; }
	if (heap_sort) { /* map.c:149-213 */
		orc128_t *heap = (orc128_t*)malloc((n_m + 1) * sizeof(orc128_t));
		size_t hs = 0;
		int64_t n_for = 0, n_rev = 0, j;
		for (i = 0; i < n_m; ++i)
			if (m[i].n > 0) { heap[hs].x = m[i].cr[0]; heap[hs].y = (uint64_t)i << 32; ++hs; }
		if (hs > 1) for (j = (int64_t)(hs >> 1) - 1; j >= 0; --j) heap_down((size_t)j, hs, heap);
		while (hs > 0) {
			match_t *q = &m[heap->y >> 32];
			uint64_t r = heap->x;
			if ((sk = skip_seed(flag, r, q, qname, qlen, tnames, tlens, &is_self)) == 0) {
				if ((r & 1) == (q->q_pos & 1)) make_anchor(&a[n_for++], r, q, qlen, is_self);
				else make_anchor(&a[n_a - (++n_rev)], r, q, qlen, is_self);
			} else nn += sk == 2;
			if ((uint32_t)heap->y < q->n - 1) {
				++heap[0].y;
				heap[0].x = m[heap[0].y >> 32].cr[(uint32_t)heap[0].y];
			} else {
				heap[0] = heap[hs - 1];
				--hs;
			}
			heap_down(0, hs, heap);
		}
		free(heap);
		for (j = 0; j < n_rev >> 1; ++j) {
			orc128_t t = a[n_a - 1 - j];
			a[n_a - 1 - j] = a[n_a - (n_rev - j)];
			a[n_a - (n_rev - j)] = t;
		}
		if (n_a > n_for + n_rev) { /* map.c:208-211 */
			memmove(a + n_for, a + n_a - n_rev, n_rev * sizeof(orc128_t));
			n_a = n_for + n_rev;
		}
	} else { /* map.c:215-247 */
		int64_t o = 0;
		for (i = 0; i < n_m; ++i) {
			uint32_t k;
			for (k = 0; k < m[i].n; ++k) {
				if ((sk = skip_seed(flag, m[i].cr[k], &m[i], qname, qlen, tnames, tlens, &is_self)) != 0) { nn += sk == 2; continue; }
				make_anchor(&a[o++], m[i].cr[k], &m[i], qlen, is_self);
			}
		}
		n_a = o;
		orc_radix_sort_128x(a, a + n_a);
	}
	free(m);
	*n_named = nn;
	return n_a;
}
