/* flat.c -- the hits of a mapping as one flat block, for bindings that do not mirror mm_reg1_t (airlift_b200/mappy.py).
 * A fragment goes through mm_map_frag() (the request queue of apiq.c), a batch built from memory through mm_b200_map_batch(es);
 * either way the result is one malloc'd mm_b200_hits_t. */
#include <stdio.h>
#include "mm2b_priv.h"

typedef struct { int frag, seg, n_regs; const mm_reg1_t *regs; const char *seq; } hit_src_t; /* the hits of one read */

static int64_t *row_of(mm_b200_hits_t *h, int64_t i) { return (int64_t*)h->rows + i * MM_B200_HITS_COLS; }

/* rows, CIGARs and the cs / MD strings flags asks for, of every read in src[0..n) */
static mm_b200_hits_t *hits_pack(const mm_idx_t *mi, int n, const hit_src_t *src, int flags)
{
	int64_t n_hits = 0, n_cigar = 0, k = 0, c = 0;
	mm_str_t str = {0, 0, 0};
	char *buf = 0;
	int m_buf = 0, i, j;
	size_t head, bytes;
	mm_b200_hits_t *h;
	for (i = 0; i < n; ++i)
		for (j = 0; j < src[i].n_regs; ++j, ++n_hits)
			if (src[i].regs[j].p) n_cigar += src[i].regs[j].p->n_cigar;
	head = (sizeof(mm_b200_hits_t) + 7) & ~(size_t)7;
	bytes = head + (size_t)n_hits * MM_B200_HITS_COLS * sizeof(int64_t) + (size_t)n_cigar * sizeof(uint32_t);
	h = (mm_b200_hits_t*)malloc(bytes);
	h->n_hits = n_hits, h->n_cigar = n_cigar, h->n_str = 0;
	h->rows = (int64_t*)((char*)h + head);
	h->cigar = (uint32_t*)((char*)h + head + (size_t)n_hits * MM_B200_HITS_COLS * sizeof(int64_t));
	for (i = 0; i < n; ++i)
		for (j = 0; j < src[i].n_regs; ++j, ++k) {
			const mm_reg1_t *r = &src[i].regs[j];
			const uint32_t nc = r->p ? r->p->n_cigar : 0;
			int64_t *o = row_of(h, k);
			int f;
			o[0] = src[i].frag, o[1] = src[i].seg, o[2] = r->rid, o[3] = r->rs, o[4] = r->re, o[5] = r->qs, o[6] = r->qe, o[7] = r->rev;
			o[8] = r->mapq, o[9] = r->id == r->parent, o[10] = r->mlen, o[11] = r->blen;
			o[12] = r->p ? r->p->n_ambi : 0, o[13] = r->p ? r->p->trans_strand : 0;
			o[14] = r->p ? r->p->dp_score : 0, o[15] = r->p ? r->p->dp_max : 0, o[16] = nc, o[17] = c;
			if (nc) memcpy((uint32_t*)h->cigar + c, r->p->cigar, nc * sizeof(uint32_t));
			c += nc;
			for (f = 0; f < 2; ++f) { /* f = 0: cs (short form, --cs), 1: MD */
				int l;
				o[18 + 2 * f] = -1, o[19 + 2 * f] = 0;
				if (!(flags & (f ? MM_B200_HITS_MD : MM_B200_HITS_CS)) || r->p == 0) continue;
				l = f ? mm_gen_MD(0, &buf, &m_buf, mi, r, src[i].seq) : mm_gen_cs(0, &buf, &m_buf, mi, r, src[i].seq, 1);
				o[18 + 2 * f] = str.l, o[19 + 2 * f] = l;
				if (str.l + (size_t)l + 1 > str.m) str.m = mm_roundup32((uint32_t)(str.l + l + 1)), str.s = (char*)realloc(str.s, str.m);
				memcpy(str.s + str.l, buf, l), str.l += l, str.s[str.l++] = 0;
			}
		}
	free(buf);
	if (str.l > 0) { /* the strings go at the end of the block */
		h = (mm_b200_hits_t*)realloc(h, bytes + str.l);
		h->rows = (int64_t*)((char*)h + head);
		h->cigar = (uint32_t*)((char*)h + head + (size_t)n_hits * MM_B200_HITS_COLS * sizeof(int64_t));
		h->str = (char*)h + bytes, h->n_str = str.l;
		memcpy((char*)h->str, str.s, str.l);
	} else h->str = 0;
	free(str.s);
	return h;
}

static void free_regs(int n, mm_reg1_t *r)
{
	int i;
	for (i = 0; i < n; ++i) free(r[i].p);
	free(r);
}

mm_b200_hits_t *mm_b200_map_hits(const mm_idx_t *mi, const mm_mapopt_t *opt, int n_segs, const int *qlens, const char **seqs,
                                 const char *qname, int flags)
{
	int n_regs[2] = {0, 0}, j, k;
	mm_reg1_t *regs[2] = {0, 0};
	const char *mseq[2];
	char *rc = 0;
	hit_src_t src[2];
	mm_b200_hits_t *h;
	if (n_segs < 1 || n_segs > 2) return 0;
	mseq[0] = seqs[0];
	if (n_segs == 2) { /* read 2 is mapped as its reverse complement (map.c:467-469 with the fr orientation) */
		mm_bseq1_t t;
		rc = (char*)malloc((size_t)qlens[1] + 1);
		memcpy(rc, seqs[1], qlens[1]), rc[qlens[1]] = 0;
		memset(&t, 0, sizeof(t));
		t.seq = rc, t.l_seq = qlens[1];
		mm_revcomp_bseq(&t);
		mseq[1] = rc;
	}
	mm_map_frag(mi, n_segs, qlens, mseq, n_regs, regs, 0, opt, qname);
	free(rc);
	if (n_segs == 2) /* ... and reported in its own orientation, as the file driver prints it (map.c:486-497) */
		for (k = 0; k < n_regs[1]; ++k) {
			mm_reg1_t *r = &regs[1][k];
			const int t = r->qs;
			r->qs = qlens[1] - r->qe, r->qe = qlens[1] - t, r->rev = !r->rev;
		}
	for (j = 0; j < n_segs; ++j) src[j].frag = 0, src[j].seg = j, src[j].n_regs = n_regs[j], src[j].regs = regs[j], src[j].seq = seqs[j];
	h = hits_pack(mi, n_segs, src, flags);
	for (j = 0; j < n_segs; ++j) free_regs(n_regs[j], regs[j]);
	return h;
}

mm_b200_hits_t *mm_b200_batch_hits_flat(const mm_idx_t *mi, const mm_b200_batch_t *b, int flags)
{
	const step_t *s = (const step_t*)b;
	hit_src_t *src = (hit_src_t*)malloc(((size_t)s->n_seq + 1) * sizeof(hit_src_t));
	mm_b200_hits_t *h;
	int f, j;
	for (f = 0; f < s->n_frag; ++f)
		for (j = 0; j < s->n_seg[f]; ++j) {
			const int i = s->seg_off[f] + j;
			src[i].frag = f, src[i].seg = j, src[i].n_regs = s->n_reg[i], src[i].regs = s->reg[i], src[i].seq = s->seq[i].seq;
		}
	h = hits_pack(mi, s->n_seq, src, flags);
	free(src);
	return h;
}

void mm_b200_hits_free(mm_b200_hits_t *h) { free(h); }

mm_b200_batch_t *mm_b200_make_batch(int n_frag, const int *n_segs, const int *qlens, const char *const *seqs, const char *const *names)
{
	step_t *s = (step_t*)calloc(1, sizeof(step_t));
	int f, j;
	for (f = 0; f < n_frag; ++f) s->n_seq += n_segs[f];
	s->seq = (mm_bseq1_t*)calloc((size_t)s->n_seq + 1, sizeof(mm_bseq1_t));
	s->n_reg = (int*)calloc(5 * ((size_t)s->n_seq + 1), sizeof(int));
	s->seg_off = s->n_reg + s->n_seq, s->n_seg = s->seg_off + s->n_seq, s->rep_len = s->n_seg + s->n_seq, s->frag_gap = s->rep_len + s->n_seq;
	s->reg = (mm_reg1_t**)calloc((size_t)s->n_seq + 1, sizeof(mm_reg1_t*));
	s->n_seq = 0;
	for (f = 0; f < n_frag; ++f) {
		s->seg_off[f] = s->n_seq, s->n_seg[f] = n_segs[f];
		for (j = 0; j < n_segs[f]; ++j, ++s->n_seq) {
			if (mm_bseq_pack1(&s->seq[s->n_seq], names ? names[f] : 0, seqs[s->n_seq], qlens[s->n_seq]) < 0) {
				s->n_frag = f;
				mm_b200_free_batch((mm_b200_batch_t*)s);
				return 0;
			}
			s->seq[s->n_seq].rid = s->n_seq;
		}
	}
	s->n_frag = n_frag;
	return (mm_b200_batch_t*)s;
}
