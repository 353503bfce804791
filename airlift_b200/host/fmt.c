/* fmt.c -- SAM / PAF records.  Output is the contract: byte-identical to the reference's format.c
 * (header :116-135, tags :276-302, PAF :304-330, SAM :387-544, cs/MD :137-250); the builder below is
 * a plain append-only string with integer printing, no varargs. */
#include <stdio.h>
#include "mm2b_priv.h"

static char g_rg_id[256];

static inline void sb_room(mm_str_t *s, size_t extra)
{
	if ((size_t)s->l + extra + 1 > s->m) {
		s->m = mm_roundup32((uint32_t)(s->l + extra + 1));
		s->s = (char*)realloc(s->s, s->m);
	}
}
static inline void sb_mem(mm_str_t *s, const char *p, size_t n) { sb_room(s, n); memcpy(s->s + s->l, p, n); s->l += n; s->s[s->l] = 0; }
static inline void sb_str(mm_str_t *s, const char *p) { sb_mem(s, p, strlen(p)); }
static inline void sb_chr(mm_str_t *s, int c) { sb_room(s, 1); s->s[s->l++] = (char)c; s->s[s->l] = 0; }
static inline void sb_u32(mm_str_t *s, uint32_t x)
{
	char buf[16]; int l = 0;
	do { buf[l++] = (char)('0' + x % 10); x /= 10; } while (x);
	sb_room(s, l);
	while (l > 0) s->s[s->l++] = buf[--l];
	s->s[s->l] = 0;
}
static inline void sb_int(mm_str_t *s, int c)
{
	if (c < 0) { sb_chr(s, '-'); sb_u32(s, (uint32_t)(-(int64_t)c)); }
	else sb_u32(s, (uint32_t)c);
}
/* "\t" + tag + value helpers */
static inline void sb_tag_i(mm_str_t *s, const char *tag, int v) { sb_str(s, tag); sb_int(s, v); }

static void unescape(char *s)
{ /* \t and \\ (format.c:67-80) */
	char *p, *q;
	for (p = q = s; *p; ++p) {
		if (*p == '\\') {
			++p;
			if (*p == 't') *q++ = '\t';
			else if (*p == '\\') *q++ = '\\';
		} else *q++ = *p;
	}
	*q = 0;
}

static void write_rg(mm_str_t *str, const char *s)
{ /* format.c:82-114 */
	char *p, *q, *r, *line = 0;
	memset(g_rg_id, 0, 256);
	if (s == 0) return;
	if (strstr(s, "@RG") != s) {
		if (mm_verbose >= 1) fprintf(stderr, "[ERROR] the read group line is not started with @RG\n");
		return;
	}
	if (strstr(s, "\t") != NULL) {
		if (mm_verbose >= 1) fprintf(stderr, "[ERROR] the read group line contained literal <tab> characters -- replace with escaped tabs: \\t\n");
		return;
	}
	line = strdup(s);
	unescape(line);
	if ((p = strstr(line, "\tID:")) == 0) {
		if (mm_verbose >= 1) fprintf(stderr, "[ERROR] no ID within the read group line\n");
		free(line); return;
	}
	p += 4;
	for (q = p; *q && *q != '\t' && *q != '\n'; ++q) {}
	if (q - p + 1 > 256) {
		if (mm_verbose >= 1) fprintf(stderr, "[ERROR] @RG:ID is longer than 255 characters\n");
		free(line); return;
	}
	for (q = p, r = g_rg_id; *q && *q != '\t' && *q != '\n'; ++q) *r++ = *q;
	sb_str(str, line); sb_chr(str, '\n');
	free(line);
}

void mm_write_sam_hdr(const mm_idx_t *idx, const char *rg, const char *ver, int argc, char *argv[])
{
	mm_str_t str = {0, 0, 0};
	int i;
	sb_room(&str, 1); str.s[0] = 0;
	if (idx)
		for (i = 0; i < (int)idx->n_seq; ++i) {
			sb_str(&str, "@SQ\tSN:"); sb_str(&str, idx->seq[i].name); sb_tag_i(&str, "\tLN:", idx->seq[i].len); sb_chr(&str, '\n');
		}
	if (rg) write_rg(&str, rg);
	sb_str(&str, "@PG\tID:minimap2\tPN:minimap2");
	if (ver) { sb_str(&str, "\tVN:"); sb_str(&str, ver); }
	if (argc > 1) {
		sb_str(&str, "\tCL:minimap2");
		for (i = 1; i < argc; ++i) { sb_chr(&str, ' '); sb_str(&str, argv[i]); }
	}
	mm_err_puts(str.s);
	free(str.s);
}

/* ---- cs / MD (format.c:137-250) */

static void write_cs(mm_str_t *s, const uint8_t *tseq, const uint8_t *qseq, const mm_reg1_t *r, char *tmp, int no_iden, int write_tag)
{
	int i, q_off = 0, t_off = 0;
	if (write_tag) sb_str(s, "\tcs:Z:");
	for (i = 0; i < (int)r->p->n_cigar; ++i) {
		const int op = r->p->cigar[i] & 0xf, len = r->p->cigar[i] >> 4;
		int j;
		if (op == 0 || op == 7 || op == 8) {
			int l_tmp = 0;
			for (j = 0; j < len; ++j) {
				if (qseq[q_off + j] != tseq[t_off + j]) {
					if (l_tmp > 0) {
						if (!no_iden) { tmp[l_tmp] = 0; sb_chr(s, '='); sb_str(s, tmp); }
						else { sb_chr(s, ':'); sb_int(s, l_tmp); }
						l_tmp = 0;
					}
					sb_chr(s, '*'); sb_chr(s, "acgtn"[tseq[t_off + j]]); sb_chr(s, "acgtn"[qseq[q_off + j]]);
				} else tmp[l_tmp++] = "ACGTN"[qseq[q_off + j]];
			}
			if (l_tmp > 0) {
				if (!no_iden) { tmp[l_tmp] = 0; sb_chr(s, '='); sb_str(s, tmp); }
				else { sb_chr(s, ':'); sb_int(s, l_tmp); }
			}
			q_off += len, t_off += len;
		} else if (op == 1) {
			for (j = 0, tmp[len] = 0; j < len; ++j) tmp[j] = "acgtn"[qseq[q_off + j]];
			sb_chr(s, '+'); sb_str(s, tmp);
			q_off += len;
		} else if (op == 2) {
			for (j = 0, tmp[len] = 0; j < len; ++j) tmp[j] = "acgtn"[tseq[t_off + j]];
			sb_chr(s, '-'); sb_str(s, tmp);
			t_off += len;
		} else {
			sb_chr(s, '~'); sb_chr(s, "acgtn"[tseq[t_off]]); sb_chr(s, "acgtn"[tseq[t_off + 1]]);
			sb_int(s, len); sb_chr(s, "acgtn"[tseq[t_off + len - 2]]); sb_chr(s, "acgtn"[tseq[t_off + len - 1]]);
			t_off += len;
		}
	}
	assert(t_off == r->re - r->rs && q_off == r->qe - r->qs);
}

static void write_md(mm_str_t *s, const uint8_t *tseq, const uint8_t *qseq, const mm_reg1_t *r, char *tmp, int write_tag)
{
	int i, q_off = 0, t_off = 0, l_MD = 0;
	if (write_tag) sb_str(s, "\tMD:Z:");
	for (i = 0; i < (int)r->p->n_cigar; ++i) {
		const int op = r->p->cigar[i] & 0xf, len = r->p->cigar[i] >> 4;
		int j;
		if (op == 0 || op == 7 || op == 8) {
			for (j = 0; j < len; ++j) {
				if (qseq[q_off + j] != tseq[t_off + j]) { sb_int(s, l_MD); sb_chr(s, "ACGTN"[tseq[t_off + j]]); l_MD = 0; }
				else ++l_MD;
			}
			q_off += len, t_off += len;
		} else if (op == 1) q_off += len;
		else if (op == 2) {
			for (j = 0, tmp[len] = 0; j < len; ++j) tmp[j] = "ACGTN"[tseq[t_off + j]];
			sb_int(s, l_MD); sb_chr(s, '^'); sb_str(s, tmp);
			l_MD = 0, t_off += len;
		} else if (op == 3) t_off += len;
	}
	if (l_MD > 0) sb_int(s, l_MD);
	assert(t_off == r->re - r->rs && q_off == r->qe - r->qs);
}

/* the cs (is_md: MD) string of r appended to s, after its "\tcs:Z:" / "\tMD:Z:" tag when write_tag; seq is the query as it was
 * mapped (format.c:137-250).  The PAF/SAM writers and mm_gen_cs / mm_gen_MD share it. */
static void write_cs_or_md(mm_str_t *s, const mm_idx_t *mi, const char *seq, const mm_reg1_t *r, int no_iden, int is_md, int write_tag)
{
	int i;
	const int ql = r->qe - r->qs, tl = r->re - r->rs;
	uint8_t *qseq, *tseq;
	char *tmp;
	if (r->p == 0) return;
	qseq = (uint8_t*)malloc(ql > 0 ? ql : 1);
	tseq = (uint8_t*)malloc(tl > 0 ? tl : 1);
	tmp = (char*)malloc((tl > ql ? tl : ql) + 1);
	mm_idx_getseq(mi, r->rid, r->rs, r->re, tseq);
	if (!r->rev) for (i = r->qs; i < r->qe; ++i) qseq[i - r->qs] = seq_nt4_table[(uint8_t)seq[i]];
	else for (i = r->qs; i < r->qe; ++i) { const uint8_t c = seq_nt4_table[(uint8_t)seq[i]]; qseq[r->qe - i - 1] = c >= 4 ? 4 : 3 - c; }
	if (is_md) write_md(s, tseq, qseq, r, tmp, write_tag);
	else write_cs(s, tseq, qseq, r, tmp, no_iden, write_tag);
	free(qseq); free(tseq); free(tmp);
}

static int gen_cs_or_md(char **buf, int *max_len, const mm_idx_t *mi, const mm_reg1_t *r, const char *seq, int no_iden, int is_md)
{ /* mm_gen_cs_or_MD (format.c): the string alone, in a buffer the caller keeps across calls */
	mm_str_t s;
	s.s = *buf, s.l = 0, s.m = *max_len > 0 ? (unsigned)*max_len : 0;
	write_cs_or_md(&s, mi, seq, r, no_iden, is_md, 0);
	if (s.s && s.m > 0) s.s[s.l] = 0;
	*buf = s.s, *max_len = (int)s.m;
	return (int)s.l;
}

int mm_gen_cs(void *km, char **buf, int *max_len, const mm_idx_t *mi, const mm_reg1_t *r, const char *seq, int no_iden)
{
	(void)km;
	return gen_cs_or_md(buf, max_len, mi, r, seq, no_iden, 0);
}

int mm_gen_MD(void *km, char **buf, int *max_len, const mm_idx_t *mi, const mm_reg1_t *r, const char *seq)
{
	(void)km;
	return gen_cs_or_md(buf, max_len, mi, r, seq, 0, 1);
}

static double event_identity(const mm_reg1_t *r)
{ /* format.c:262-274: matches over (block length with each gap counted once) */
	int32_t i, n_gapo = 0, n_gap = 0;
	if (r->p == 0) return -1.0f;
	for (i = 0; i < (int32_t)r->p->n_cigar; ++i) {
		const int32_t op = r->p->cigar[i] & 0xf, len = r->p->cigar[i] >> 4;
		if (op == 1 || op == 2) ++n_gapo, n_gap += len;
	}
	return (double)r->mlen / (r->blen - n_gap + n_gapo);
}

static void write_tags(mm_str_t *s, const mm_reg1_t *r)
{ /* format.c:276-302 */
	int type;
	if (r->id == r->parent) type = r->inv ? 'I' : 'P';
	else type = r->inv ? 'i' : 'S';
	if (r->p) {
		sb_tag_i(s, "\tNM:i:", r->blen - r->mlen + r->p->n_ambi); sb_tag_i(s, "\tms:i:", r->p->dp_max);
		sb_tag_i(s, "\tAS:i:", r->p->dp_score); sb_tag_i(s, "\tnn:i:", r->p->n_ambi);
		if (r->p->trans_strand == 1 || r->p->trans_strand == 2) { sb_str(s, "\tts:A:"); sb_chr(s, "?+-?"[r->p->trans_strand]); }
	}
	sb_str(s, "\ttp:A:"); sb_chr(s, type); sb_tag_i(s, "\tcm:i:", r->cnt); sb_tag_i(s, "\ts1:i:", r->score);
	if (r->parent == r->id) sb_tag_i(s, "\ts2:i:", r->subsc);
	if (r->p) {
		char buf[16];
		const double div = 1.0 - event_identity(r);
		if (div == 0.0) buf[0] = '0', buf[1] = 0;
		else snprintf(buf, 16, "%.4f", 1.0 - event_identity(r));
		sb_str(s, "\tde:f:"); sb_str(s, buf);
	} else if (r->div >= 0.0f && r->div <= 1.0f) {
		char buf[16];
		if (r->div == 0.0f) buf[0] = '0', buf[1] = 0;
		else snprintf(buf, 16, "%.4f", r->div);
		sb_str(s, "\tdv:f:"); sb_str(s, buf);
	}
	if (r->split) sb_tag_i(s, "\tzd:i:", r->split);
}

void mm_write_paf3(mm_str_t *s, const mm_idx_t *mi, const mm_bseq1_t *t, const mm_reg1_t *r, int opt_flag, int rep_len)
{ /* format.c:304-330 */
	s->l = 0;
	sb_room(s, 1); s->s[0] = 0;
	if (r == 0) {
		sb_str(s, t->name); sb_chr(s, '\t'); sb_int(s, t->l_seq); sb_str(s, "\t0\t0\t*\t*\t0\t0\t0\t0\t0\t0");
		if (rep_len >= 0) sb_tag_i(s, "\trl:i:", rep_len);
		return;
	}
	sb_str(s, t->name); sb_chr(s, '\t'); sb_int(s, t->l_seq); sb_chr(s, '\t'); sb_int(s, r->qs); sb_chr(s, '\t'); sb_int(s, r->qe);
	sb_chr(s, '\t'); sb_chr(s, "+-"[r->rev]); sb_chr(s, '\t');
	if (mi->seq[r->rid].name) sb_str(s, mi->seq[r->rid].name);
	else sb_int(s, r->rid);
	sb_chr(s, '\t'); sb_int(s, mi->seq[r->rid].len); sb_chr(s, '\t'); sb_int(s, r->rs); sb_chr(s, '\t'); sb_int(s, r->re);
	sb_chr(s, '\t'); sb_int(s, r->mlen); sb_chr(s, '\t'); sb_int(s, r->blen); sb_chr(s, '\t'); sb_int(s, r->mapq);
	write_tags(s, r);
	if (rep_len >= 0) sb_tag_i(s, "\trl:i:", rep_len);
	if (r->p && (opt_flag & MM_F_OUT_CG)) {
		uint32_t k;
		sb_str(s, "\tcg:Z:");
		for (k = 0; k < r->p->n_cigar; ++k) { sb_int(s, r->p->cigar[k] >> 4); sb_chr(s, "MIDNSHP=XB"[r->p->cigar[k] & 0xf]); }
	}
	if (r->p && (opt_flag & (MM_F_OUT_CS|MM_F_OUT_MD)))
		write_cs_or_md(s, mi, t->seq, r, !(opt_flag & MM_F_OUT_CS_LONG), opt_flag & MM_F_OUT_MD, 1);
	if ((opt_flag & MM_F_COPY_COMMENT) && t->comment) { sb_chr(s, '\t'); sb_str(s, t->comment); }
}

static void sam_seq(mm_str_t *s, const char *seq, int l, int rev, int comp)
{ /* format.c:337-349 */
	if (rev) {
		int i;
		sb_room(s, l);
		for (i = 0; i < l; ++i) {
			const int c = seq[l - 1 - i]; /* plain char on purpose: bytes >= 128 stay as they are */
			s->s[s->l + i] = (char)(c < 128 && comp ? seq_comp_table[c] : c);
		}
		s->l += l; s->s[s->l] = 0;
	} else sb_mem(s, seq, l);
}

static const mm_reg1_t *sam_primary(int n_regs, const mm_reg1_t *regs)
{
	int i;
	for (i = 0; i < n_regs; ++i) if (regs[i].sam_pri) return &regs[i];
	assert(n_regs == 0);
	return NULL;
}

static void sam_cigar(mm_str_t *s, int sam_flag, int in_tag, int qlen, const mm_reg1_t *r, int opt_flag)
{ /* format.c:361-385 */
	uint32_t k, clip[2];
	if (r->p == 0) { sb_chr(s, '*'); return; }
	clip[0] = r->rev ? qlen - r->qe : r->qs;
	clip[1] = r->rev ? r->qs : qlen - r->qe;
	if (in_tag) {
		const int op = (sam_flag & 0x800) && !(opt_flag & MM_F_SOFTCLIP) ? 5 : 4;
		sb_str(s, "\tCG:B:I");
		if (clip[0]) { sb_chr(s, ','); sb_u32(s, clip[0] << 4 | op); }
		for (k = 0; k < r->p->n_cigar; ++k) { sb_chr(s, ','); sb_u32(s, r->p->cigar[k]); }
		if (clip[1]) { sb_chr(s, ','); sb_u32(s, clip[1] << 4 | op); }
	} else {
		const int ch = (sam_flag & 0x800) && !(opt_flag & MM_F_SOFTCLIP) ? 'H' : 'S';
		assert(clip[0] < (uint32_t)qlen && clip[1] < (uint32_t)qlen);
		if (clip[0]) { sb_int(s, clip[0]); sb_chr(s, ch); }
		for (k = 0; k < r->p->n_cigar; ++k) { sb_int(s, r->p->cigar[k] >> 4); sb_chr(s, "MIDNSHP=XB"[r->p->cigar[k] & 0xf]); }
		if (clip[1]) { sb_int(s, clip[1]); sb_chr(s, ch); }
	}
}

void mm_write_sam3(mm_str_t *s, const mm_idx_t *mi, const mm_bseq1_t *t, int seg_idx, int reg_idx, int n_seg, const int *n_regss,
                   const mm_reg1_t *const* regss, int opt_flag, int rep_len)
{ /* format.c:387-544 */
	const int max_bam_cigar_op = 65535;
	int flag, n_regs = n_regss[seg_idx], cigar_in_tag = 0;
	int this_rid = -1, this_pos = -1;
	const mm_reg1_t *regs = regss[seg_idx], *r_prev = NULL, *r_next = NULL;
	const mm_reg1_t *r = n_regs > 0 && reg_idx < n_regs && reg_idx >= 0 ? &regs[reg_idx] : NULL;

	if (n_seg > 1) { /* primaries of the neighbouring segments */
		int i;
		const int next_sid = (seg_idx + 1) % n_seg;
		r_next = sam_primary(n_regss[next_sid], regss[next_sid]);
		if (n_seg > 2) {
			for (i = 1; i <= n_seg - 1; ++i) {
				const int prev_sid = (seg_idx + n_seg - i) % n_seg;
				if (n_regss[prev_sid] > 0) { r_prev = sam_primary(n_regss[prev_sid], regss[prev_sid]); break; }
			}
		} else r_prev = r_next;
	}

	s->l = 0;
	sb_room(s, 1); s->s[0] = 0;
	sb_str(s, t->name);
	if (n_seg > 1) s->l = mm_qname_len(t->name); /* drop /1 or /2 */

	flag = n_seg > 1 ? 0x1 : 0x0;
	if (r == 0) flag |= 0x4;
	else {
		if (r->rev) flag |= 0x10;
		if (r->parent != r->id) flag |= 0x100;
		else if (!r->sam_pri) flag |= 0x800;
	}
	if (n_seg > 1) {
		if (r && r->proper_frag) flag |= 0x2;
		if (seg_idx == 0) flag |= 0x40;
		else if (seg_idx == n_seg - 1) flag |= 0x80;
		if (r_next == NULL) flag |= 0x8;
		else if (r_next->rev) flag |= 0x20;
	}
	sb_chr(s, '\t'); sb_int(s, flag);

	if (r == 0) {
		if (r_prev) {
			this_rid = r_prev->rid, this_pos = r_prev->rs;
			sb_chr(s, '\t'); sb_str(s, mi->seq[this_rid].name); sb_chr(s, '\t'); sb_int(s, this_pos + 1); sb_str(s, "\t0\t*");
		} else sb_str(s, "\t*\t0\t0\t*");
	} else {
		this_rid = r->rid, this_pos = r->rs;
		sb_chr(s, '\t'); sb_str(s, mi->seq[r->rid].name); sb_chr(s, '\t'); sb_int(s, r->rs + 1); sb_chr(s, '\t'); sb_int(s, r->mapq); sb_chr(s, '\t');
		if ((opt_flag & MM_F_LONG_CIGAR) && r->p && r->p->n_cigar > (uint32_t)(max_bam_cigar_op - 2)) {
			int n_cigar = r->p->n_cigar;
			if (r->qs != 0) ++n_cigar;
			if (r->qe != t->l_seq) ++n_cigar;
			if (n_cigar > max_bam_cigar_op) cigar_in_tag = 1;
		}
		if (cigar_in_tag) {
			int slen;
			if ((flag & 0x900) == 0 || (opt_flag & MM_F_SOFTCLIP)) slen = t->l_seq;
			else if (flag & 0x100) slen = 0;
			else slen = r->qe - r->qs;
			sb_int(s, slen); sb_chr(s, 'S'); sb_int(s, r->re - r->rs); sb_chr(s, 'N');
		} else sam_cigar(s, flag, 0, t->l_seq, r, opt_flag);
	}

	if (n_seg > 1) { /* RNEXT, PNEXT, TLEN */
		int tlen = 0;
		if (this_rid >= 0 && r_next) {
			if (this_rid == r_next->rid) {
				if (r) {
					const int this_pos5 = r->rev ? r->re - 1 : this_pos;
					const int next_pos5 = r_next->rev ? r_next->re - 1 : r_next->rs;
					tlen = next_pos5 - this_pos5;
				}
				sb_str(s, "\t=\t");
			} else { sb_chr(s, '\t'); sb_str(s, mi->seq[r_next->rid].name); sb_chr(s, '\t'); }
			sb_int(s, r_next->rs + 1); sb_chr(s, '\t');
		} else if (r_next) {
			sb_chr(s, '\t'); sb_str(s, mi->seq[r_next->rid].name); sb_chr(s, '\t'); sb_int(s, r_next->rs + 1); sb_chr(s, '\t');
		} else if (this_rid >= 0) {
			sb_str(s, "\t=\t"); sb_int(s, this_pos + 1); sb_chr(s, '\t');
		} else sb_str(s, "\t*\t0\t");
		if (tlen > 0) ++tlen;
		else if (tlen < 0) --tlen;
		sb_int(s, tlen); sb_chr(s, '\t');
	} else sb_str(s, "\t*\t0\t0\t");

	if (r == 0) { /* SEQ, QUAL */
		sam_seq(s, t->seq, t->l_seq, 0, 0);
		sb_chr(s, '\t');
		if (t->qual) sam_seq(s, t->qual, t->l_seq, 0, 0);
		else sb_chr(s, '*');
	} else if ((flag & 0x900) == 0 || (opt_flag & MM_F_SOFTCLIP)) {
		sam_seq(s, t->seq, t->l_seq, r->rev, r->rev);
		sb_chr(s, '\t');
		if (t->qual) sam_seq(s, t->qual, t->l_seq, r->rev, 0);
		else sb_chr(s, '*');
	} else if (flag & 0x100) {
		sb_str(s, "*\t*");
	} else {
		sam_seq(s, t->seq + r->qs, r->qe - r->qs, r->rev, r->rev);
		sb_chr(s, '\t');
		if (t->qual) sam_seq(s, t->qual + r->qs, r->qe - r->qs, r->rev, 0);
		else sb_chr(s, '*');
	}

	if (g_rg_id[0]) { sb_str(s, "\tRG:Z:"); sb_str(s, g_rg_id); }
	if (n_seg > 2) sb_tag_i(s, "\tFI:i:", seg_idx);
	if (r) {
		write_tags(s, r);
		if (r->parent == r->id && r->p && n_regs > 1 && regs && r >= regs && r - regs < n_regs) { /* SA: other primary lines */
			int i, n_sa = 0;
			for (i = 0; i < n_regs; ++i)
				if (i != r - regs && regs[i].parent == regs[i].id && regs[i].p) ++n_sa;
			if (n_sa > 0) {
				sb_str(s, "\tSA:Z:");
				for (i = 0; i < n_regs; ++i) {
					const mm_reg1_t *q = &regs[i];
					int l_M, l_I = 0, l_D = 0, clip5, clip3;
					if (r == q || q->parent != q->id || q->p == 0) continue;
					if (q->qe - q->qs < q->re - q->rs) l_M = q->qe - q->qs, l_D = (q->re - q->rs) - l_M;
					else l_M = q->re - q->rs, l_I = (q->qe - q->qs) - l_M;
					clip5 = q->rev ? t->l_seq - q->qe : q->qs;
					clip3 = q->rev ? q->qs : t->l_seq - q->qe;
					sb_str(s, mi->seq[q->rid].name); sb_chr(s, ','); sb_int(s, q->rs + 1); sb_chr(s, ','); sb_chr(s, "+-"[q->rev]); sb_chr(s, ',');
					if (clip5) { sb_int(s, clip5); sb_chr(s, 'S'); }
					if (l_M) { sb_int(s, l_M); sb_chr(s, 'M'); }
					if (l_I) { sb_int(s, l_I); sb_chr(s, 'I'); }
					if (l_D) { sb_int(s, l_D); sb_chr(s, 'D'); }
					if (clip3) { sb_int(s, clip3); sb_chr(s, 'S'); }
					sb_chr(s, ','); sb_int(s, q->mapq); sb_chr(s, ','); sb_int(s, q->blen - q->mlen + q->p->n_ambi); sb_chr(s, ';');
				}
			}
		}
		if (r->p && (opt_flag & (MM_F_OUT_CS|MM_F_OUT_MD)))
			write_cs_or_md(s, mi, t->seq, r, !(opt_flag & MM_F_OUT_CS_LONG), opt_flag & MM_F_OUT_MD, 1);
		if (cigar_in_tag) sam_cigar(s, flag, 1, t->l_seq, r, opt_flag);
	}
	if (rep_len >= 0) sb_tag_i(s, "\trl:i:", rep_len);
	if ((opt_flag & MM_F_COPY_COMMENT) && t->comment) { sb_chr(s, '\t'); sb_str(s, t->comment); }
	s->s[s->l] = 0;
}
