/* seqio.c -- gz FASTA/FASTQ reader and mini-batch assembly.
 * Observable behaviour follows the reference's kseq.h:192-233 (record grammar) and bseq.c:58-162
 * (U->T, batch sizing, mate grouping); SURVEY.md App. C lists the rules.  Implementation is a small
 * pull parser over a 256 KiB inflate window. */
#include <zlib.h>
#include <stdio.h>
#include <ctype.h>
#include <pthread.h>
#include "mm2b_priv.h"

#define IO_BUF (256 * 1024)
#define CHECK_PAIR_THRES 1000000

typedef struct {
	gzFile fp;
	unsigned char *buf;
	int beg, end, eof;
} gzstream_t;

typedef struct { mm_str_t name, comment, seq, qual; int last_char; } record_t;

/* Query files are parsed by a read-ahead thread per file (mm_bseq_set_readahead): blocks of records travel through a
 * small ring, so that the two mate files of a paired run are parsed concurrently and ahead of the mapper. */
#define RA_BLOCK 4096
#define RA_RING 8
typedef struct { mm_bseq1_t *a; int n, ret; } ra_block_t; /* ret: what ended the block (>= 0: more follow; -1: end of file; -2: bad record) */

/* Packed records of a read-ahead stream live in slabs: one malloc per ~1 MB of records instead of one per record (malloc and free
 * were a sixth of the parser's time).  A record is [slab_t* | name\0 seq\0 qual\0 comment\0]; the slab counts its live records
 * plus the producer while it is still filling it, and whoever drops the last reference frees it (mm_bseq_free1 from any thread). */
typedef struct { int live; } slab_t;
#define SLAB_BYTES (1 << 20)
static inline void slab_unref(slab_t *h) { if (__atomic_sub_fetch(&h->live, 1, __ATOMIC_ACQ_REL) == 0) free(h); }

struct mm_bseq_file_s {
	gzstream_t st;
	record_t rec;
	slab_t *slab; size_t slab_used, slab_cap; /* slab being filled by this stream's producer */
	mm_bseq1_t pending; /* a record read ahead while completing a pair (bseq.c:100-110) */
	int packed;         /* records are one malloc block owned by `name` (seq/qual/comment point inside it) */
	int ra_on, ra_started, ra_stop, ra_with_qual, ra_with_comment;
	pthread_t ra_thread;
	pthread_mutex_t ra_mu;
	pthread_cond_t ra_cv;
	ra_block_t ring[RA_RING];
	uint64_t ra_head, ra_tail; /* blocks [head, tail) are ready */
	ra_block_t cur;            /* block being consumed */
	int cur_i, ra_final;       /* ra_final: the status that ended the stream, once the consumer has seen it */
};

static int next_bseq(mm_bseq_file_t *fp, mm_bseq1_t *out, int with_qual, int with_comment);

static inline int st_fill(gzstream_t *s)
{
	if (s->eof) return 0;
	s->beg = 0;
	s->end = gzread(s->fp, s->buf, IO_BUF);
	if (s->end < IO_BUF) s->eof = 1;
	if (s->end < 0) s->end = 0;
	return s->end;
}

static inline int st_getc(gzstream_t *s)
{
	if (s->beg >= s->end && st_fill(s) == 0) return -1;
	return s->buf[s->beg++];
}

static inline void str_reserve(mm_str_t *s, size_t need)
{
	if (s->m < need) { s->m = mm_roundup32((uint32_t)need); s->s = (char*)realloc(s->s, s->m); }
}

/* read up to a delimiter (is_line: '\n', else any whitespace); the delimiter is consumed and returned in *dret.
 * Returns the string length or -1 at end of file.  A single trailing '\r' is dropped from line reads. */
static int st_until(gzstream_t *s, int is_line, mm_str_t *str, int *dret, int append)
{
	if (dret) *dret = 0;
	if (!append) str->l = 0;
	if (s->beg >= s->end && s->eof) return -1;
	for (;;) {
		int i;
		if (s->beg >= s->end && st_fill(s) == 0) break;
		if (is_line) { unsigned char *p = (unsigned char*)memchr(s->buf + s->beg, '\n', s->end - s->beg); i = p ? (int)(p - s->buf) : s->end; }
		else for (i = s->beg; i < s->end; ++i) if (isspace(s->buf[i])) break;
		str_reserve(str, (size_t)str->l + (i - s->beg) + 1);
		memcpy(str->s + str->l, s->buf + s->beg, i - s->beg);
		str->l += i - s->beg;
		s->beg = i + 1;
		if (i < s->end) { if (dret) *dret = s->buf[i]; break; }
	}
	if (str->s == 0) { str->m = 1; str->s = (char*)calloc(1, 1); }
	else if (is_line && str->l > 1 && str->s[str->l - 1] == '\r') --str->l;
	str->s[str->l] = 0;
	return (int)str->l;
}

/* >=0 sequence length; -1 end of file; -2 truncated/mismatched quality */
static int read_record(gzstream_t *st, record_t *r)
{
	int c;
	if (r->last_char == 0) {
		while ((c = st_getc(st)) != -1 && c != '>' && c != '@') {}
		if (c == -1) return -1;
		r->last_char = c;
	}
	r->comment.l = r->seq.l = r->qual.l = 0;
	if (st_until(st, 0, &r->name, &c, 0) < 0) return -1;
	if (c != '\n') st_until(st, 1, &r->comment, 0, 0);
	if (r->seq.s == 0) { r->seq.m = 256; r->seq.s = (char*)malloc(r->seq.m); }
	while ((c = st_getc(st)) != -1 && c != '>' && c != '+' && c != '@') {
		if (c == '\n') continue;
		str_reserve(&r->seq, (size_t)r->seq.l + 2);
		r->seq.s[r->seq.l++] = (char)c;
		st_until(st, 1, &r->seq, 0, 1);
	}
	if (c == '>' || c == '@') r->last_char = c;
	str_reserve(&r->seq, (size_t)r->seq.l + 2);
	r->seq.s[r->seq.l] = 0;
	if (c != '+') return (int)r->seq.l;
	str_reserve(&r->qual, r->seq.m);
	while ((c = st_getc(st)) != -1 && c != '\n') {}
	if (c == -1) return -2;
	while (st_until(st, 1, &r->qual, 0, 1) >= 0 && r->qual.l < r->seq.l) {}
	r->last_char = 0;
	if (r->seq.l != r->qual.l) return -2;
	return (int)r->seq.l;
}

mm_bseq_file_t *mm_bseq_open(const char *fn)
{
	gzFile f = fn && strcmp(fn, "-") ? gzopen(fn, "r") : gzdopen(0, "r");
	mm_bseq_file_t *fp;
	if (f == 0) return 0;
	gzbuffer(f, 1 << 20);
	fp = (mm_bseq_file_t*)calloc(1, sizeof(*fp));
	fp->st.fp = f;
	fp->st.buf = (unsigned char*)malloc(IO_BUF);
	pthread_mutex_init(&fp->ra_mu, 0);
	pthread_cond_init(&fp->ra_cv, 0);
	return fp;
}

void mm_bseq_close(mm_bseq_file_t *fp)
{
	if (fp == 0) return;
	if (fp->ra_started) { /* stop the read-ahead thread and drop what it had queued */
		int i;
		pthread_mutex_lock(&fp->ra_mu);
		fp->ra_stop = 1;
		pthread_cond_broadcast(&fp->ra_cv);
		pthread_mutex_unlock(&fp->ra_mu);
		for (;;) { /* keep draining so that a producer blocked on a full ring can finish */
			mm_bseq1_t t;
			if (next_bseq(fp, &t, fp->ra_with_qual, fp->ra_with_comment) < 0) break;
			mm_bseq_free1(&t, fp->packed);
		}
		pthread_join(fp->ra_thread, 0);
		while (fp->ra_head < fp->ra_tail) {
			ra_block_t *b = &fp->ring[fp->ra_head++ % RA_RING];
			for (i = 0; i < b->n; ++i) mm_bseq_free1(&b->a[i], fp->packed);
			free(b->a);
		}
	}
	if (fp->pending.seq) mm_bseq_free1(&fp->pending, fp->packed);
	if (fp->slab) slab_unref(fp->slab); /* records already handed out keep their slabs alive */
	free(fp->rec.name.s); free(fp->rec.comment.s); free(fp->rec.seq.s); free(fp->rec.qual.s);
	free(fp->st.buf);
	gzclose(fp->st.fp);
	free(fp);
}

int mm_bseq_eof(mm_bseq_file_t *fp)
{
	if (fp->ra_on) return fp->ra_final < 0 && fp->pending.seq == 0;
	return fp->st.eof && fp->st.beg >= fp->st.end && fp->pending.seq == 0;
}

static inline void fix_u(char *q, int l)
{ /* U -> T, u -> t (bseq.c:72-74) */
	int i;
	for (i = 0; i < l; ++i) q[i] -= ((q[i] | 0x20) == 'u');
}

/* one record from its four pieces; packed: a single block [name\0 seq\0 qual\0 comment\0] owned by `name` */
static char *slab_alloc(mm_bseq_file_t *fp, size_t need)
{ /* room for a back-pointer and `need` bytes of strings, 8-byte aligned */
	const size_t tot = (sizeof(slab_t*) + need + 7) & ~(size_t)7;
	char *p;
	if (fp->slab == 0 || fp->slab_used + tot > fp->slab_cap) {
		const size_t cap = sizeof(slab_t) + 8 + tot > SLAB_BYTES ? sizeof(slab_t) + 8 + tot : SLAB_BYTES;
		if (fp->slab) slab_unref(fp->slab); /* the producer is done with the old one */
		fp->slab = (slab_t*)malloc(cap);
		fp->slab->live = 1;                 /* the producer's own reference */
		fp->slab_used = (sizeof(slab_t) + 7) & ~(size_t)7, fp->slab_cap = cap;
	}
	p = (char*)fp->slab + fp->slab_used;
	fp->slab_used += tot;
	__atomic_add_fetch(&fp->slab->live, 1, __ATOMIC_RELAXED);
	*(slab_t**)p = fp->slab;
	return p + sizeof(slab_t*);
}

static void make_bseq(mm_bseq_file_t *fp, mm_bseq1_t *s, int packed, const char *name, int l_name, const char *seq, int l_seq, const char *qual, int l_qual,
                      const char *comment, int l_comment)
{
	if (l_name == 0) fprintf(stderr, "[WARNING]\033[1;31m empty sequence name in the input.\033[0m\n");
	if (packed) {
		char *b = slab_alloc(fp, (size_t)l_name + l_seq + (qual ? l_qual + 1 : 0) + (comment ? l_comment + 1 : 0) + 2);
		s->name = b; memcpy(b, name, l_name); b[l_name] = 0; b += l_name + 1;
		s->seq = b; memcpy(b, seq, l_seq); b[l_seq] = 0; b += l_seq + 1;
		s->qual = 0, s->comment = 0;
		if (qual) { s->qual = b; memcpy(b, qual, l_qual); b[l_qual] = 0; b += l_qual + 1; }
		if (comment) { s->comment = b; memcpy(b, comment, l_comment); b[l_comment] = 0; }
	} else {
		s->name = (char*)malloc((size_t)l_name + 1); memcpy(s->name, name, l_name); s->name[l_name] = 0;
		s->seq = (char*)malloc((size_t)l_seq + 1); memcpy(s->seq, seq, l_seq); s->seq[l_seq] = 0;
		s->qual = 0, s->comment = 0;
		if (qual) { s->qual = (char*)malloc((size_t)l_qual + 1); memcpy(s->qual, qual, l_qual); s->qual[l_qual] = 0; }
		if (comment) { s->comment = (char*)malloc((size_t)l_comment + 1); memcpy(s->comment, comment, l_comment); s->comment[l_comment] = 0; }
	}
	if (memchr(s->seq, 'U', l_seq) || memchr(s->seq, 'u', l_seq)) fix_u(s->seq, l_seq); /* two vector scans instead of a byte loop over every read */
	s->l_seq = l_seq;
	s->rid = 0;
}

static void record_to_bseq(mm_bseq_file_t *fp, const record_t *r, mm_bseq1_t *s, int packed, int with_qual, int with_comment)
{
	make_bseq(fp, s, packed, r->name.s, (int)r->name.l, r->seq.s, (int)r->seq.l, with_qual && r->qual.l ? r->qual.s : 0, (int)r->qual.l,
	          with_comment && r->comment.l ? r->comment.s : 0, (int)r->comment.l);
}

/* The common case, a four-line FASTQ record lying entirely inside the inflate window, is cut out with four memchr()
 * calls; anything else (FASTA, wrapped lines, '\r', a record straddling the window, ...) takes the general parser above,
 * which defines the behaviour.  Returns 1 if a record was produced, 0 if the general parser must be used. */
static int fastq_fast_path(mm_bseq_file_t *fp, mm_bseq1_t *out, int with_qual, int with_comment)
{
	gzstream_t *st = &fp->st;
	const unsigned char *b = st->buf, *e = st->buf + st->end, *p0 = st->buf + st->beg, *p1, *p2, *p3, *p4, *ws;
	int l_name, l_seq;
	if (fp->rec.last_char != 0 || p0 >= e || *p0 != '@') return 0;
	if ((p1 = (const unsigned char*)memchr(p0, '\n', e - p0)) == 0) return 0;
	if ((p2 = (const unsigned char*)memchr(p1 + 1, '\n', e - (p1 + 1))) == 0) return 0;
	if (p2 + 1 >= e || p2[1] != '+') return 0;
	if ((p3 = (const unsigned char*)memchr(p2 + 1, '\n', e - (p2 + 1))) == 0) return 0;
	if ((p4 = (const unsigned char*)memchr(p3 + 1, '\n', e - (p3 + 1))) == 0) return 0;
	l_seq = (int)(p2 - p1 - 1);
	if (l_seq <= 0 || p4 - p3 - 1 != l_seq) return 0;
	if (p1[-1] == '\r' || p2[-1] == '\r' || p4[-1] == '\r') return 0;
	if (p4 + 1 < e && p4[1] != '@') return 0;                 /* not followed by a record start: leave it to the general parser */
	if (p4 + 1 >= e && !st->eof) return 0;                     /* cannot see what follows */
	/* kseq looks at the first character of a sequence line only (kseq.h:186: `while ((c = ks_getc(ks)) >= 0 && c != '>' && c != '+'
	 * && c != '@')`, the rest of the line goes through ks_getuntil2); l_seq > 0, so p1[1] is that character */
	if (p1[1] == '>' || p1[1] == '@' || p1[1] == '+') return 0;
	for (ws = p0 + 1; ws < p1; ++ws) if (isspace(*ws)) break; /* name ends at the first white space; the rest of the line is the comment */
	l_name = (int)(ws - (p0 + 1));
	make_bseq(fp, out, fp->packed, (const char*)p0 + 1, l_name, (const char*)p1 + 1, l_seq, with_qual ? (const char*)p3 + 1 : 0, l_seq,
	          with_comment && ws < p1 && p1 - ws - 1 > 0 ? (const char*)ws + 1 : 0, ws < p1 ? (int)(p1 - ws - 1) : 0);
	st->beg = (int)(p4 + 1 - b);
	return 1;
}

/* next record straight from the file: >= 0 sequence length (record in *out); -1 end of file; -2 bad record */
static int next_direct(mm_bseq_file_t *fp, mm_bseq1_t *out, int with_qual, int with_comment)
{
	int ret;
	if (fp->st.beg >= fp->st.end && !fp->st.eof && fp->rec.last_char == 0) st_fill(&fp->st);
	if (fastq_fast_path(fp, out, with_qual, with_comment)) return out->l_seq;
	ret = read_record(&fp->st, &fp->rec);
	if (ret >= 0) record_to_bseq(fp, &fp->rec, out, fp->packed, with_qual, with_comment);
	return ret;
}

static void *ra_main(void *arg)
{
	mm_bseq_file_t *fp = (mm_bseq_file_t*)arg;
	for (;;) {
		ra_block_t blk;
		blk.a = (mm_bseq1_t*)malloc(RA_BLOCK * sizeof(mm_bseq1_t)), blk.n = 0, blk.ret = 0;
		while (blk.n < RA_BLOCK && (blk.ret = next_direct(fp, &blk.a[blk.n], fp->ra_with_qual, fp->ra_with_comment)) >= 0) ++blk.n;
		pthread_mutex_lock(&fp->ra_mu);
		/* a full ring always drains: the consumer takes blocks, and mm_bseq_close() keeps taking them after it asked us to stop */
		while (fp->ra_tail - fp->ra_head == RA_RING) pthread_cond_wait(&fp->ra_cv, &fp->ra_mu);
		if (fp->ra_stop && blk.ret >= 0) blk.ret = -1; /* asked to stop: this block is the last one, the consumer must see an end */
		fp->ring[fp->ra_tail % RA_RING] = blk; ++fp->ra_tail;
		pthread_cond_broadcast(&fp->ra_cv);
		pthread_mutex_unlock(&fp->ra_mu);
		if (blk.ret < 0) break;
	}
	return 0;
}

/* next record of the file, through the read-ahead ring when it is enabled */
static int next_bseq(mm_bseq_file_t *fp, mm_bseq1_t *out, int with_qual, int with_comment)
{
	if (!fp->ra_on) return next_direct(fp, out, with_qual, with_comment);
	if (!fp->ra_started) {
		fp->ra_with_qual = with_qual, fp->ra_with_comment = with_comment, fp->ra_started = 1;
		pthread_create(&fp->ra_thread, 0, ra_main, fp);
	}
	for (;;) {
		if (fp->cur_i < fp->cur.n) { *out = fp->cur.a[fp->cur_i++]; return out->l_seq; }
		if (fp->cur.a) { free(fp->cur.a); fp->cur.a = 0; fp->cur.n = fp->cur_i = 0; if (fp->cur.ret < 0) fp->ra_final = fp->cur.ret; }
		if (fp->ra_final < 0) return fp->ra_final;
		pthread_mutex_lock(&fp->ra_mu);
		while (fp->ra_tail == fp->ra_head) pthread_cond_wait(&fp->ra_cv, &fp->ra_mu);
		fp->cur = fp->ring[fp->ra_head % RA_RING]; ++fp->ra_head; fp->cur_i = 0;
		pthread_cond_broadcast(&fp->ra_cv);
		pthread_mutex_unlock(&fp->ra_mu);
	}
}

void mm_bseq_set_readahead(mm_bseq_file_t *fp, int packed)
{ /* query files: parse ahead in a thread of its own; `packed` records are single blocks released with mm_bseq_free1() */
	fp->ra_on = 1, fp->packed = packed;
}

void mm_bseq_free1(mm_bseq1_t *s, int packed)
{
	if (packed) { if (s->name) slab_unref(*(slab_t**)(s->name - sizeof(slab_t*))); }
	else { free(s->seq); free(s->name); free(s->qual); free(s->comment); }
	s->seq = s->name = s->qual = s->comment = 0;
}

typedef struct { int n, m; mm_bseq1_t *a; } bseq_v;

static inline mm_bseq1_t *vec_next(bseq_v *v)
{
	if (v->n == v->m) { v->m = v->m ? v->m << 1 : 256; v->a = (mm_bseq1_t*)realloc(v->a, (size_t)v->m * sizeof(mm_bseq1_t)); }
	return &v->a[v->n++];
}

int mm_qname_len(const char *s)
{ /* a trailing "/<digit>" is not part of the fragment name (bseq.h:31-36) */
	int l = (int)strlen(s);
	return l >= 3 && s[l-1] >= '0' && s[l-1] <= '9' && s[l-2] == '/' ? l - 2 : l;
}

int mm_qname_same(const char *s1, const char *s2)
{
	int l1 = mm_qname_len(s1), l2 = mm_qname_len(s2);
	return l1 == l2 && strncmp(s1, s2, l1) == 0;
}

void mm_revcomp_bseq(mm_bseq1_t *s)
{ /* bseq.h:46-58 */
	int i, l = s->l_seq;
	for (i = 0; i < l >> 1; ++i) {
		int t = (unsigned char)s->seq[l - i - 1];
		s->seq[l - i - 1] = seq_comp_table[(unsigned char)s->seq[i]];
		s->seq[i] = seq_comp_table[t];
	}
	if (l & 1) s->seq[l >> 1] = seq_comp_table[(unsigned char)s->seq[l >> 1]];
	if (s->qual)
		for (i = 0; i < l >> 1; ++i) { char t = s->qual[l - i - 1]; s->qual[l - i - 1] = s->qual[i], s->qual[i] = t; }
}

mm_bseq1_t *mm_bseq_read3(mm_bseq_file_t *fp, int chunk_size, int with_qual, int with_comment, int frag_mode, int *n_)
{ /* bseq.c:80-117 */
	int64_t size = 0;
	int ret;
	bseq_v a = {0, 0, 0};
	*n_ = 0;
	if (fp->pending.seq) {
		*vec_next(&a) = fp->pending;
		size = fp->pending.l_seq;
		memset(&fp->pending, 0, sizeof(mm_bseq1_t));
	}
	for (;;) {
		mm_bseq1_t t;
		if ((ret = next_bseq(fp, &t, with_qual, with_comment)) < 0) break;
		*vec_next(&a) = t;
		size += t.l_seq;
		if (size >= chunk_size) {
			if (frag_mode && a.a[a.n-1].l_seq < CHECK_PAIR_THRES) { /* never split a pair across batches */
				while (next_bseq(fp, &fp->pending, with_qual, with_comment) >= 0) {
					if (mm_qname_same(fp->pending.name, a.a[a.n-1].name)) {
						*vec_next(&a) = fp->pending;
						memset(&fp->pending, 0, sizeof(mm_bseq1_t));
					} else break;
				}
			}
			break;
		}
	}
	if (ret < -1) fprintf(stderr, "[WARNING]\033[1;31m wrong FASTA/FASTQ record. Continue anyway.\033[0m\n");
	*n_ = a.n;
	return a.a;
}

mm_bseq1_t *mm_bseq_read_frag2(int n_fp, mm_bseq_file_t **fp, int chunk_size, int with_qual, int with_comment, int *n_)
{ /* bseq.c:129-157: zip the files record by record; stop at the shortest */
	int i;
	int64_t size = 0;
	bseq_v a = {0, 0, 0};
	*n_ = 0;
	if (n_fp < 1) return 0;
	for (;;) {
		int n_read = 0;
		mm_bseq1_t t[MM_MAX_SEG];
		for (i = 0; i < n_fp && i < MM_MAX_SEG; ++i)
			if (next_bseq(fp[i], &t[i], with_qual, with_comment) >= 0) ++n_read; else memset(&t[i], 0, sizeof(t[i]));
		if (n_read < n_fp) {
			if (n_read > 0)
				fprintf(stderr, "[W::%s]\033[1;31m query files have different number of records; extra records skipped.\033[0m\n", __func__);
			for (i = 0; i < n_fp && i < MM_MAX_SEG; ++i) if (t[i].seq) mm_bseq_free1(&t[i], fp[i]->packed);
			break;
		}
		for (i = 0; i < n_fp; ++i) {
			*vec_next(&a) = t[i];
			size += t[i].l_seq;
		}
		if (size >= chunk_size) break;
	}
	*n_ = a.n;
	return a.a;
}

int mm_bseq_pack1(mm_bseq1_t *s, const char *name, const char *seq, int l_seq)
{ /* a packed record (see slab_t) on a slab of its own, for batches built from memory; 0, or -1 when out of memory */
	const size_t l_name = name ? strlen(name) : 0, off = (sizeof(slab_t) + 7) & ~(size_t)7;
	char *p = (char*)malloc(off + sizeof(slab_t*) + l_name + 1 + (size_t)l_seq + 1), *b;
	if (p == 0) return -1;
	((slab_t*)p)->live = 1;
	*(slab_t**)(p + off) = (slab_t*)p;
	b = p + off + sizeof(slab_t*);
	memset(s, 0, sizeof(*s));
	s->name = b, memcpy(b, name ? name : "", l_name + 1);
	s->seq = b + l_name + 1, memcpy(s->seq, seq, l_seq), s->seq[l_seq] = 0;
	s->l_seq = l_seq;
	return 0;
}

/* ---- record-at-a-time reader for bindings (mappy.fastx_read): the records mm_bseq_read3 gives, one per call */

struct mm_fastx_s { mm_bseq_file_t *fp; mm_bseq1_t *a; int n, i, with_comment; };

mm_fastx_t *mm_fastx_open(const char *fn, int with_comment)
{
	mm_fastx_t *r;
	mm_bseq_file_t *fp = mm_bseq_open(fn);
	if (fp == 0) return 0;
	r = (mm_fastx_t*)calloc(1, sizeof(*r));
	r->fp = fp, r->with_comment = with_comment;
	return r;
}

static void fastx_drop(mm_fastx_t *r)
{
	int i;
	for (i = 0; i < r->n; ++i) mm_bseq_free1(&r->a[i], 0);
	free(r->a);
	r->a = 0, r->n = r->i = 0;
}

int mm_fastx_read(mm_fastx_t *r, const char **name, const char **seq, const char **qual, const char **comment)
{
	const mm_bseq1_t *t;
	if (r->i == r->n) {
		fastx_drop(r);
		r->a = mm_bseq_read3(r->fp, 1, 1, r->with_comment, 0, &r->n); /* chunk of one base: one record (more after empty ones) */
		if (r->n == 0) return -1;
	}
	t = &r->a[r->i++];
	*name = t->name, *seq = t->seq, *qual = t->qual, *comment = t->comment;
	return t->l_seq;
}

void mm_fastx_close(mm_fastx_t *r)
{
	if (r == 0) return;
	fastx_drop(r);
	mm_bseq_close(r->fp);
	free(r);
}
