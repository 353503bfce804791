// mmg_core.h -- per-thread building blocks of the device stages.
//
// Every function here is __host__ __device__ so that the exact code the kernels run can also
// be compiled by g++ into the CPU-side emulation harness used by the `-m "not gpu"` tests
// (tests/emu/).  The product library only ever calls them from kernels.
//
// Reference behaviour each block reproduces (paths relative to
// /root/reference/src/minimap2-master_remapping/): see the comment on each function.
#pragma once
#include <stdint.h>
#include <stddef.h>

#if defined(__CUDACC__)
#define MMG_HD __host__ __device__ __forceinline__
#define MMG_HDN __host__ __device__
#else
#define MMG_HD inline
#define MMG_HDN
#endif

struct mm128 { uint64_t x, y; };

#define MMG_NONE 0xffffffffffffffffULL
#define MMG_MAX_W 64               // ring buffer size of the sketch state machine (reference allows 255)
#define MMG_SEED_TANDEM (1ULL << 42)  // mmpriv.h:18
#define MMG_SEED_SELF (1ULL << 43)    // mmpriv.h:19
#define MMG_SEED_SEG_SHIFT 48         // mmpriv.h:21
#define MMG_SEED_SEG_MASK (0xffULL << MMG_SEED_SEG_SHIFT)
#define MMG_NAME_NONE 0xffffffffu     // name key of a unit without a name (include/mmg.h)
#define MMG_F_NO_DIAG 0x001LL         // minimap.h:8
#define MMG_F_NO_DUAL 0x002LL
#define MMG_F_FOR_ONLY 0x100000LL     // minimap.h:28
#define MMG_F_REV_ONLY 0x200000LL
#define MMG_F_HEAP_SORT 0x400000LL
#define MMG_F_SR 0x1000LL
#define MMG_F_SPLICE 0x080LL

// ------------------------------------------------------------------ sequences
// 4-bit packed bases, 8 per word, identical to mm_idx_t::S (mmpriv.h:28-29)
MMG_HD int mmg_seq4_get(const uint32_t *S, uint64_t i) { return S[i >> 3] >> ((i & 7) << 2) & 0xf; }

MMG_HD int mmg_nt4(uint8_t c)  // seq_nt4_table, sketch.c:9-26
{
	if (c < 4) return c;
	switch (c | 0x20) { case 'a': return 0; case 'c': return 1; case 'g': return 2; case 't': case 'u': return 3; default: return 4; }
}

MMG_HD uint64_t mmg_hash64(uint64_t key, uint64_t mask)  // sketch.c:28-38
{
	key = (~key + (key << 21)) & mask;
	key = key ^ key >> 24;
	key = ((key + (key << 3)) + (key << 8)) & mask;
	key = key ^ key >> 14;
	key = ((key + (key << 2)) + (key << 4)) & mask;
	key = key ^ key >> 28;
	key = (key + (key << 31)) & mask;
	return key;
}

// ------------------------------------------------------------------ K1: sketch
// One work unit = the emission events of positions [emit_start, emit_end) of one sequence
// (sketch.c:89-140), plus the final flush (sketch.c:141-142) when emit_end == len.
// A unit that does not start at 0 replays a warm-up prefix from a blank state; the replay
// is long enough once (a) the last w ring entries were produced with a k-mer validity equal
// to the true one and (b) every `l` threshold compares the same way as in the full scan
// (l >= w+2k, or l resynchronised exactly by an ambiguous base after >= k shifted bases).
// If the first warm-up is too short (N runs, palindromic k-mers) it is retried 4x longer,
// down to position 0, where the state is exact by definition.
struct SketchUnit {
	uint64_t off;       // base offset of the sequence in the packed array
	int32_t len;        // sequence length
	uint32_t rid;       // goes to y>>32
	uint64_t y_add;     // collect_minimizers' `sum<<1` for segments after the first (map.c:71-72)
	int32_t emit_start, emit_end;
};

template <bool kWrite>
MMG_HDN inline int mmg_sketch_unit(const uint32_t *S, const SketchUnit &un, int w, int k, int is_hpc, mm128 *out)
{
	const uint64_t shift1 = 2 * (k - 1), mask = (1ULL << 2 * k) - 1;
	const int len = un.len;
	int warm = w + 2 * k + 16;
	for (;;) {
		uint64_t kmer0 = 0, kmer1 = 0;
		mm128 ring[MMG_MAX_W], best = {MMG_NONE, MMG_NONE};
		int hp_q[32], hp_front = 0, hp_count = 0;
		int i, j, l = 0, ring_pos = 0, best_pos = 0, span = 0, n = 0;
		int ws = un.emit_start - warm, eq_pushes = 0, n_shift = 0;
		bool exact = false, resync = false; // exact: l equals the l of a scan from position 0
		if (ws < 0 || is_hpc) ws = 0;
		for (j = 0; j < w; ++j) ring[j].x = ring[j].y = MMG_NONE;
		uint32_t word = 0;
		{ uint64_t o = un.off + ws; if (o & 7) word = S[o >> 3]; }
		for (i = ws; i < un.emit_end; ++i) {
			const uint64_t o = un.off + i;
			if ((o & 7) == 0) word = S[o >> 3];
			int c = word >> ((o & 7) << 2) & 0xf;
			if (i == un.emit_start && ws > 0 && !(eq_pushes >= w && (exact || l >= w + 2 * k))) { resync = true; break; }
			const bool keep = i >= un.emit_start;
			mm128 info = {MMG_NONE, MMG_NONE};
			if (c < 4) {
				int z;
				if (is_hpc) { // sketch.c:94-104 (only reached with ws == 0: whole-sequence units)
					int run = 1;
					if (i + 1 < len && mmg_seq4_get(S, un.off + i + 1) == c) {
						for (run = 2; i + run < len; ++run)
							if (mmg_seq4_get(S, un.off + i + run) != c) break;
						i += run - 1;
						word = S[(un.off + i) >> 3];
					}
					hp_q[(hp_count++ + hp_front) & 0x1f] = run;
					span += run;
					if (hp_count > k) { span -= hp_q[hp_front++]; hp_front &= 0x1f; --hp_count; }
				} else span = l + 1 < k ? l + 1 : k;
				if (n_shift < k) ++n_shift;
				kmer0 = (kmer0 << 2 | (uint64_t)c) & mask;
				kmer1 = (kmer1 >> 2) | (3ULL ^ (uint64_t)c) << shift1;
				if (kmer0 == kmer1) continue; // sketch.c:108
				z = kmer0 < kmer1 ? 0 : 1;
				++l;
				if (l >= k && span < 256) {
					info.x = mmg_hash64(z ? kmer1 : kmer0, mask) << 8 | (uint64_t)span;
					info.y = ((uint64_t)un.rid << 32 | (uint32_t)i << 1 | (uint32_t)z) + un.y_add;
				}
				eq_pushes = (exact || l >= k) ? eq_pushes + 1 : 0; // this ring entry equals the full scan's
			} else {
				l = 0, hp_count = hp_front = 0, span = 0;
				if (n_shift >= k) exact = true; // k-mer registers complete: from here on l is the true l
				++eq_pushes;                    // an N pushes the empty entry in either scan
			}
#define MMG_EMIT(v) do { if (keep) { if (kWrite) out[n] = (v); ++n; } } while (0)
			ring[ring_pos] = info;
			if (l == w + k - 1 && best.x != MMG_NONE) { // sketch.c:117-122
				for (j = ring_pos + 1; j < w; ++j) if (best.x == ring[j].x && ring[j].y != best.y) MMG_EMIT(ring[j]);
				for (j = 0; j < ring_pos; ++j)     if (best.x == ring[j].x && ring[j].y != best.y) MMG_EMIT(ring[j]);
			}
			if (info.x <= best.x) { // sketch.c:123-125
				if (l >= w + k && best.x != MMG_NONE) MMG_EMIT(best);
				best = info, best_pos = ring_pos;
			} else if (ring_pos == best_pos) { // sketch.c:126-137
				if (l >= w + k - 1 && best.x != MMG_NONE) MMG_EMIT(best);
				best.x = MMG_NONE;
				for (j = ring_pos + 1; j < w; ++j) if (best.x >= ring[j].x) best = ring[j], best_pos = j;
				for (j = 0; j <= ring_pos; ++j)    if (best.x >= ring[j].x) best = ring[j], best_pos = j;
				if (l >= w + k - 1 && best.x != MMG_NONE) {
					for (j = ring_pos + 1; j < w; ++j) if (best.x == ring[j].x && best.y != ring[j].y) MMG_EMIT(ring[j]);
					for (j = 0; j <= ring_pos; ++j)    if (best.x == ring[j].x && best.y != ring[j].y) MMG_EMIT(ring[j]);
				}
			}
			if (++ring_pos == w) ring_pos = 0;
		}
		if (resync) { warm *= 4; continue; }
		if (un.emit_end >= len && best.x != MMG_NONE) { // sketch.c:141-142
			if (kWrite) out[n] = best;
			++n;
		}
#undef MMG_EMIT
		return n;
	}
}

// ------------------------------------------------------------------ K2: index lookup
// Open-addressing table of 16-byte slots {key, val}: one 32-byte sector per probe.
//   key = minimizer hash (x>>8) | singleton<<63;  empty = ~0
//   val = position (singleton, index.c:223-225)  or  start<<32|n into pos[] (index.c:231)
// mm_idx_get (index.c:81-98) returns (n, pointer); here (n, val) with the same meaning.
struct IdxSlot { uint64_t key, val; };
#define MMG_SLOT_EMPTY 0xffffffffffffffffULL
#define MMG_SLOT_SINGLE (1ULL << 63)

MMG_HD uint64_t mmg_slot_hash(uint64_t minier, int shift) { return (minier * 0x9E3779B97F4A7C15ULL) >> shift; }

struct IdxView {
	const uint32_t *S;
	const uint64_t *seq_off;
	const uint32_t *seq_len;
	const uint32_t *tkey;      // name key of every target (mmg_idx_set_name_keys); null until set
	const IdxSlot *slots;
	const uint64_t *pos;
	uint64_t slot_mask;
	int32_t slot_shift, n_seq, w, k;
};

// returns n; *val = the position when n == 1, else the start index into pos[]
MMG_HD int mmg_idx_probe(const IdxView &ix, uint64_t minier, uint64_t *val)
{
	uint64_t i = mmg_slot_hash(minier, ix.slot_shift);
	for (;;) {
#if defined(__CUDA_ARCH__)
		const ulonglong2 s = __ldg(reinterpret_cast<const ulonglong2*>(ix.slots) + i);
		const uint64_t key = s.x, v = s.y;
#else
		const uint64_t key = ix.slots[i].key, v = ix.slots[i].val;
#endif
		if (key == MMG_SLOT_EMPTY) { *val = 0; return 0; }
		if ((key & ~MMG_SLOT_SINGLE) == minier) {
			if (key & MMG_SLOT_SINGLE) { *val = v; return 1; }
			*val = v >> 32;
			return (int)(uint32_t)v;
		}
		i = (i + 1) & ix.slot_mask;
	}
}

// collect_matches (map.c:90-123) for one fragment whose lookups (m_n) are done:
// marks the minimizers below the occurrence cut-off, sums their hits, accumulates rep_len,
// and records mini_pos (map.c:117).  Returns n_a.
MMG_HDN inline int64_t mmg_frag_plan(const mm128 *mv, const int32_t *m_n, int n_mv, int max_occ, int *rep_len_out,
                                     int *n_mini_out, uint64_t *mini_pos)
{
	int rep_st = 0, rep_en = 0, rep_len = 0, n_mini = 0;
	int64_t n_a = 0;
	for (int i = 0; i < n_mv; ++i) {
		const uint32_t q_pos = (uint32_t)mv[i].y, q_span = (uint32_t)(mv[i].x & 0xff);
		const int t = m_n[i];
		if (t >= max_occ) {
			const int en = (int)(q_pos >> 1) + 1, st = en - (int)q_span;
			if (st > rep_en) { rep_len += rep_en - rep_st; rep_st = st, rep_en = en; }
			else rep_en = en;
		} else {
			n_a += t;
			if (mini_pos) mini_pos[n_mini] = (uint64_t)q_span << 32 | q_pos >> 1;
			++n_mini;
		}
	}
	*rep_len_out = rep_len + (rep_en - rep_st);
	*n_mini_out = n_mini;
	return n_a;
}

// The self/dual-hit filters of skip_seed compare the mapping unit's name with the target's.  The device sees the names only as
// the order keys of include/mmg.h: tkey[rid] per target, ukey per unit (MMG_NAME_NONE: the filters are off for the unit).
struct NameFilt { const uint32_t *tkey, *tlen; uint32_t ukey; };

#define MMG_SKIP_KEEP 0
#define MMG_SKIP_STRAND 1  // dropped by --for-only / --rev-only
#define MMG_SKIP_NAME 2    // dropped by -D (diagonal of a self-hit) or --dual=no (target name sorts below the unit's)

// skip_seed, map.c:125-147; qlen is the unit's summed length.  *is_self: same-strand anchor of a unit mapped onto the target of
// its own name and length (MMG_SEED_SELF).  Nothing is read from nf unless a name filter is on.
MMG_HD int mmg_skip_seed(int64_t flag, uint64_t r, uint32_t q_pos, const NameFilt &nf, int qlen, bool *is_self)
{
	*is_self = false;
	if ((flag & (MMG_F_NO_DIAG | MMG_F_NO_DUAL)) && nf.ukey != MMG_NAME_NONE) {
		const uint32_t rid = (uint32_t)(r >> 32), tk = nf.tkey[rid];
		if ((flag & MMG_F_NO_DIAG) && tk == nf.ukey && (int)nf.tlen[rid] == qlen) {
			if ((uint32_t)r >> 1 == q_pos >> 1) return MMG_SKIP_NAME;
			if ((r & 1) == (q_pos & 1)) *is_self = true;
		}
		if ((flag & MMG_F_NO_DUAL) && tk < nf.ukey) return MMG_SKIP_NAME;
	}
	if (flag & (MMG_F_FOR_ONLY | MMG_F_REV_ONLY)) {
		if ((r & 1) == (q_pos & 1)) { if (flag & MMG_F_REV_ONLY) return MMG_SKIP_STRAND; }
		else if (flag & MMG_F_FOR_ONLY) return MMG_SKIP_STRAND;
	}
	return MMG_SKIP_KEEP;
}

// Strand-only forms of the functions below, for callers without name keys (the self/dual filters off): the strand filters,
// no self bit, no count of hits dropped by name
MMG_HD bool mmg_skip_seed(int64_t flag, uint64_t r, uint32_t q_pos)
{
	const NameFilt nf = {nullptr, nullptr, MMG_NAME_NONE};
	bool self;
	return mmg_skip_seed(flag, r, q_pos, nf, 0, &self) != MMG_SKIP_KEEP;
}

MMG_HD bool mmg_is_tandem(const mm128 *mv, int n_mv, int i)  // map.c:113-115
{
	const uint64_t h = mv[i].x >> 8;
	return (i > 0 && h == mv[i - 1].x >> 8) || (i < n_mv - 1 && h == mv[i + 1].x >> 8);
}

MMG_HD mm128 mmg_make_anchor(uint64_t r, const mm128 &m, bool tandem, bool self, int qlen)  // map.c:176-187 / 232-241
{
	const uint32_t q_pos = (uint32_t)m.y, q_span = (uint32_t)(m.x & 0xff), seg_id = (uint32_t)(m.y >> 32);
	const uint32_t rpos = (uint32_t)r >> 1;
	mm128 p;
	if ((r & 1) == (q_pos & 1)) {
		p.x = (r & 0xffffffff00000000ULL) | rpos;
		p.y = (uint64_t)q_span << 32 | q_pos >> 1;
	} else {
		p.x = 1ULL << 63 | (r & 0xffffffff00000000ULL) | rpos;
		p.y = (uint64_t)q_span << 32 | (uint32_t)(qlen - (int)((q_pos >> 1) + 1 - q_span) - 1);
	}
	p.y |= (uint64_t)seg_id << MMG_SEED_SEG_SHIFT;
	if (tandem) p.y |= MMG_SEED_TANDEM;
	if (self) p.y |= MMG_SEED_SELF;
	return p;
}
MMG_HD mm128 mmg_make_anchor(uint64_t r, const mm128 &m, bool tandem, int qlen) { return mmg_make_anchor(r, m, tandem, false, qlen); }

MMG_HD uint64_t mmg_hit_pos(const uint64_t *pos, int n, uint64_t val, uint32_t j) { return n == 1 ? val : pos[val + j]; }

// binary heap keyed on x with klib's sift-down (ksort.h:43-53 with heap_lt(a,b) = a.x > b.x, map.c:80)
MMG_HD void mmg_heap_down(size_t i, size_t n, mm128 *l)
{
	size_t k = i;
	mm128 tmp = l[i];
	while ((k = (k << 1) + 1) < n) {
		if (k != n - 1 && l[k].x > l[k + 1].x) ++k;
		if (l[k].x > tmp.x) break;
		l[i] = l[k]; i = k;
	}
	l[i] = tmp;
}

// collect_seed_hits_heap (map.c:149-213): k-way merge of the per-minimizer position lists.
// heap[] is scratch with room for n_mv entries.  a[] has room for n_a_planned anchors.
// Equal-x anchors come out in the heap's own order (SURVEY.md H2), hence the literal replay.
// *n_named receives the hits the self/dual filters dropped (here and in mmg_fill_flat).  kNamed = false compiles the filters out
// (options without MMG_F_NO_DIAG / MMG_F_NO_DUAL), so that the kernels of the other presets keep their registers.
#define MMG_NAMED_FLAG(kNamed, flag) ((kNamed) ? (flag) : (flag) & ~(MMG_F_NO_DIAG | MMG_F_NO_DUAL))
template <bool kNamed = true>
MMG_HDN inline int64_t mmg_fill_heap(const mm128 *mv, const int32_t *m_n, const uint64_t *m_val, int n_mv, int max_occ,
                                     const uint64_t *pos, int64_t flag, const NameFilt &nf, int qlen, int64_t n_a_planned, mm128 *heap,
                                     mm128 *a, int64_t *n_named)
{
	size_t hs = 0;
	int64_t n_for = 0, n_rev = 0, n_a = n_a_planned, n_nm = 0;
	for (int i = 0; i < n_mv; ++i)
		if (m_n[i] > 0 && m_n[i] < max_occ) {
			heap[hs].x = mmg_hit_pos(pos, m_n[i], m_val[i], 0);
			heap[hs].y = (uint64_t)i << 32;
			++hs;
		}
	if (hs > 1) for (int64_t j = (int64_t)(hs >> 1) - 1; j >= 0; --j) mmg_heap_down((size_t)j, hs, heap);
	while (hs > 0) {
		const int i = (int)(heap[0].y >> 32);
		const uint64_t r = heap[0].x;
		bool self;
		const int sk = mmg_skip_seed(MMG_NAMED_FLAG(kNamed, flag), r, (uint32_t)mv[i].y, nf, qlen, &self);
		if (sk == MMG_SKIP_KEEP) {
			const mm128 an = mmg_make_anchor(r, mv[i], mmg_is_tandem(mv, n_mv, i), self, qlen);
			if ((r & 1) == ((uint32_t)mv[i].y & 1)) a[n_for++] = an;
			else a[n_a - (++n_rev)] = an;
		} else n_nm += sk == MMG_SKIP_NAME;
		if ((uint32_t)heap[0].y < (uint32_t)m_n[i] - 1) {
			++heap[0].y;
			heap[0].x = mmg_hit_pos(pos, m_n[i], m_val[i], (uint32_t)heap[0].y);
		} else {
			heap[0] = heap[hs - 1];
			--hs;
		}
		if (hs > 0) mmg_heap_down(0, hs, heap);
	}
	for (int64_t j = 0; j < n_rev >> 1; ++j) { // map.c:203-207
		mm128 t = a[n_a - 1 - j];
		a[n_a - 1 - j] = a[n_a - (n_rev - j)];
		a[n_a - (n_rev - j)] = t;
	}
	if (n_a > n_for + n_rev) { // map.c:208-211 (only with strand or self/dual filters)
		for (int64_t j = 0; j < n_rev; ++j) a[n_for + j] = a[n_a - n_rev + j];
		n_a = n_for + n_rev;
	}
	*n_named = n_nm;
	return n_a;
}
MMG_HDN inline int64_t mmg_fill_heap(const mm128 *mv, const int32_t *m_n, const uint64_t *m_val, int n_mv, int max_occ,
                                     const uint64_t *pos, int64_t flag, int qlen, int64_t n_a_planned, mm128 *heap, mm128 *a)
{
	const NameFilt nf = {nullptr, nullptr, MMG_NAME_NONE};
	int64_t nn;
	return mmg_fill_heap<false>(mv, m_n, m_val, n_mv, max_occ, pos, flag, nf, qlen, n_a_planned, heap, a, &nn);
}

// The same merge replayed on RANKS.  Which of two equal positions leaves the heap first depends on the heap's shape, so the
// order of equal-x anchors can only come from running klib's heap (SURVEY.md H2); but the heap only ever COMPARES positions.
// A device-wide sort gives every planned hit the index of the first hit with its position (equal positions: equal index), and
// the replay then runs on 32-bit words `rank << 8 | list` without touching the position arrays: same comparisons, same
// sift-downs, same pops.  K[s]: rank of planned slot s (slots of list j: first[j] .. first[j] + cnt[j]); pop[t] receives the
// slot popped t-th.  Lists: up to 256; ranks: below 2^24.  heap/cur: n_lists words of scratch each.
MMG_HD void mmg_rank_heap_down(uint32_t i, uint32_t n, uint32_t *l)
{
	uint32_t k = i;
	const uint32_t tmp = l[i];
	while ((k = (k << 1) + 1) < n) {
		if (k != n - 1 && (l[k] >> 8) > (l[k + 1] >> 8)) ++k;
		if ((l[k] >> 8) > (tmp >> 8)) break;
		l[i] = l[k]; i = k;
	}
	l[i] = tmp;
}

MMG_HDN inline int64_t mmg_heap_replay_ranks(int n_lists, const int32_t *first, const int32_t *cnt, const uint32_t *K, uint32_t *heap, uint32_t *cur, uint32_t *pop)
{
	uint32_t hs = 0;
	int64_t t = 0;
	for (int j = 0; j < n_lists; ++j) { heap[hs++] = K[first[j]] << 8 | (uint32_t)j; cur[j] = 0; }
	if (hs > 1) for (int32_t j = (int32_t)(hs >> 1) - 1; j >= 0; --j) mmg_rank_heap_down((uint32_t)j, hs, heap);
	while (hs > 0) {
		const uint32_t j = heap[0] & 0xff;
		pop[t++] = (uint32_t)first[j] + cur[j];
		if (cur[j] + 1 < (uint32_t)cnt[j]) { ++cur[j]; heap[0] = K[(uint32_t)first[j] + cur[j]] << 8 | j; }
		else { heap[0] = heap[hs - 1]; --hs; }
		if (hs > 0) mmg_rank_heap_down(0, hs, heap);
	}
	return t;
}

// --- klib's in-place MSD radix sort (ksort.h:101-151) replayed exactly, recursion turned into an
// explicit stack (stack[] needs n/65+2 frames).  Needed wherever equal keys may meet in an array of
// more than 64 elements: the order they end in is defined by this permutation (SURVEY.md H1).
struct RsFrame { int64_t beg, end; int32_t shift; int32_t pad; };

template <class T, class KeyFn>
MMG_HDN inline void mmg_rs_insertion(T *a, int64_t beg, int64_t end, KeyFn key)
{
	for (int64_t i = beg + 1; i < end; ++i)
		if (key(a[i]) < key(a[i - 1])) {
			T tmp = a[i];
			int64_t j;
			for (j = i; j > beg && key(tmp) < key(a[j - 1]); --j) a[j] = a[j - 1];
			a[j] = tmp;
		}
}

template <class T, class KeyFn>
MMG_HDN inline void mmg_rs_sort_exact(T *a, int64_t n, RsFrame *stack, KeyFn key)
{
	if (n <= 64) { mmg_rs_insertion(a, 0, n, key); return; }
	int top = 0;
	stack[top].beg = 0, stack[top].end = n, stack[top].shift = 56; ++top;
	while (top > 0) {
		const RsFrame fr = stack[--top];
		const int s = fr.shift;
		int64_t head[256], tail[256];
		for (int d = 0; d < 256; ++d) tail[d] = 0;
		for (int64_t i = fr.beg; i < fr.end; ++i) ++tail[key(a[i]) >> s & 0xff];
		{
			int64_t at = fr.beg;
			for (int d = 0; d < 256; ++d) { head[d] = at; at += tail[d]; tail[d] = at; }
		}
		for (int d = 0; d < 256;) { // ksort.h:126-138
			if (head[d] != tail[d]) {
				int to = (int)(key(a[head[d]]) >> s & 0xff);
				if (to != d) {
					T carry = a[head[d]], swap;
					do {
						swap = carry; carry = a[head[to]]; a[head[to]++] = swap;
						to = (int)(key(carry) >> s & 0xff);
					} while (to != d);
					a[head[d]++] = carry;
				} else ++head[d];
			} else ++d;
		}
		if (s) { // ksort.h:140-145
			const int ns = s > 8 ? s - 8 : 0;
			int64_t lo = fr.beg;
			for (int d = 0; d < 256; ++d) {
				const int64_t hi = tail[d];
				if (hi - lo > 64) { stack[top].beg = lo, stack[top].end = hi, stack[top].shift = ns; ++top; }
				else if (hi - lo > 1) mmg_rs_insertion(a, lo, hi, key);
				lo = hi;
			}
		}
	}
}

struct KeyX { MMG_HD uint64_t operator()(const mm128 &v) const { return v.x; } };

// collect_seed_hits (map.c:215-247): fill in query order, then radix_sort_128x
template <bool kNamed = true>
MMG_HDN inline int64_t mmg_fill_flat(const mm128 *mv, const int32_t *m_n, const uint64_t *m_val, int n_mv, int max_occ,
                                     const uint64_t *pos, int64_t flag, const NameFilt &nf, int qlen, mm128 *a, RsFrame *stack,
                                     int64_t *n_named)
{
	int64_t o = 0, n_nm = 0;
	for (int i = 0; i < n_mv; ++i) {
		if (m_n[i] <= 0 || m_n[i] >= max_occ) continue;
		const bool tandem = mmg_is_tandem(mv, n_mv, i);
		for (uint32_t j = 0; j < (uint32_t)m_n[i]; ++j) {
			const uint64_t r = mmg_hit_pos(pos, m_n[i], m_val[i], j);
			bool self;
			const int sk = mmg_skip_seed(MMG_NAMED_FLAG(kNamed, flag), r, (uint32_t)mv[i].y, nf, qlen, &self);
			if (sk != MMG_SKIP_KEEP) { n_nm += sk == MMG_SKIP_NAME; continue; }
			a[o++] = mmg_make_anchor(r, mv[i], tandem, self, qlen);
		}
	}
	mmg_rs_sort_exact(a, o, stack, KeyX());
	*n_named = n_nm;
	return o;
}
MMG_HDN inline int64_t mmg_fill_flat(const mm128 *mv, const int32_t *m_n, const uint64_t *m_val, int n_mv, int max_occ,
                                     const uint64_t *pos, int64_t flag, int qlen, mm128 *a, RsFrame *stack)
{
	const NameFilt nf = {nullptr, nullptr, MMG_NAME_NONE};
	int64_t nn;
	return mmg_fill_flat<false>(mv, m_n, m_val, n_mv, max_occ, pos, flag, nf, qlen, a, stack, &nn);
}

// ------------------------------------------------------------------ K3: chaining
struct ChainParams {  // mm_chain_dp's scalar arguments (chain.c:22)
	int32_t max_dist_x, max_dist_y, bw, max_skip, max_iter, min_cnt, min_sc, is_cdna, n_segs;
};

MMG_HD int mmg_ilog2_32(uint32_t v)  // chain.c:15-20
{
#if defined(__CUDA_ARCH__)
	return 31 - __clz((int)v);
#else
	return 31 - __builtin_clz(v);
#endif
}

// score of extending predecessor j to anchor i (chain.c:54-72); returns false when j is not eligible
MMG_HD bool mmg_chain_score(const ChainParams &P, uint64_t ri, int32_t qi, int32_t q_span, int32_t sidi, const mm128 &aj,
                            float avg_qspan, int32_t *sc_out)
{
	const int64_t dr = (int64_t)(ri - aj.x);
	const int32_t dq = qi - (int32_t)aj.y;
	const int32_t sidj = (int32_t)((aj.y & MMG_SEED_SEG_MASK) >> MMG_SEED_SEG_SHIFT);
	int32_t dd, sc, log_dd, min_d;
	if ((sidi == sidj && dr == 0) || dq <= 0) return false;
	if ((sidi == sidj && dq > P.max_dist_y) || dq > P.max_dist_x) return false;
	dd = (int32_t)(dr > dq ? dr - dq : dq - dr);
	if (sidi == sidj && dd > P.bw) return false;
	if (P.n_segs > 1 && !P.is_cdna && sidi == sidj && dr > P.max_dist_y) return false;
	min_d = dq < dr ? dq : (int32_t)dr;
	sc = min_d > q_span ? q_span : min_d;
	log_dd = dd ? mmg_ilog2_32((uint32_t)dd) : 0;
	// (int)(dd * .01 * avg_qspan): int->double, double multiplies, truncation (chain.c:67,72)
	const int32_t c_lin = (int32_t)((double)dd * .01 * (double)avg_qspan);
	if (P.is_cdna || sidi != sidj) {
		const int32_t c_log = log_dd;
		if (sidi != sidj && dr == 0) ++sc;
		else if (dr > dq || sidi != sidj) sc -= c_lin < c_log ? c_lin : c_log;
		else sc -= c_lin + (c_log >> 1);
	} else sc -= c_lin + (log_dd >> 1);
	*sc_out = sc;
	return true;
}

struct KeyU64 { MMG_HD uint64_t operator()(const uint64_t &v) const { return v; } };

// heap sort, ascending; used where the reference radix-sorts keys that are unique or fully identical
MMG_HDN inline void mmg_sort_u64(uint64_t *a, int64_t n)
{
	if (n <= 64) { mmg_rs_insertion(a, 0, n, KeyU64()); return; }
	for (int64_t start = n / 2 - 1; start >= 0; --start) {
		int64_t i = start; uint64_t tmp = a[i];
		for (;;) { int64_t c = 2 * i + 1; if (c >= n) break; if (c + 1 < n && a[c + 1] > a[c]) ++c; if (a[c] <= tmp) break; a[i] = a[c]; i = c; }
		a[i] = tmp;
	}
	for (int64_t end = n - 1; end > 0; --end) {
		uint64_t tmp = a[end]; a[end] = a[0];
		int64_t i = 0;
		for (;;) { int64_t c = 2 * i + 1; if (c >= end) break; if (c + 1 < end && a[c + 1] > a[c]) ++c; if (a[c] <= tmp) break; a[i] = a[c]; i = c; }
		a[i] = tmp;
	}
}

// Everything in mm_chain_dp after the DP fill (chain.c:87-160), for one anchor array.
//   f,p,t,v : the four int32 work arrays (contiguous: f | p | t | v, 16*n bytes, reused for w[])
//   u       : 2*n uint64 of scratch (u then u2)
//   b       : n mm128 of scratch
//   a       : in: sorted anchors; out: compacted chains in final order.  Returns n_u; *n_v_out = anchors kept.
MMG_HDN inline int mmg_chain_backtrack(const ChainParams &P, int64_t n, mm128 *a, int32_t *f, int32_t *p, int32_t *t, int32_t *v,
                                       uint64_t *u, mm128 *b, RsFrame *stack, int64_t *n_v_out)
{
	int32_t n_u = 0, n_v = 0, k;
	int64_t i, j;
	for (i = 0; i < n; ++i) t[i] = 0;
	for (i = 0; i < n; ++i) if (p[i] >= 0) t[p[i]] = 1;
	for (i = 0; i < n; ++i)
		if (t[i] == 0 && v[i] >= P.min_sc) {
			j = i;
			while (j >= 0 && f[j] < v[j]) j = p[j];
			if (j < 0) j = i;
			u[n_u++] = (uint64_t)f[j] << 32 | (uint64_t)j;
		}
	*n_v_out = 0;
	if (n_u == 0) return 0;
	mmg_sort_u64(u, n_u); // chain.c:107 (keys unique or identical)
	for (i = 0; i < n_u >> 1; ++i) { uint64_t x = u[i]; u[i] = u[n_u - i - 1], u[n_u - i - 1] = x; }
	for (i = 0; i < n; ++i) t[i] = 0;
	for (i = n_v = k = 0; i < n_u; ++i) { // chain.c:115-129
		const int32_t n_v0 = n_v, k0 = k;
		j = (int32_t)u[i];
		do { v[n_v++] = (int32_t)j; t[j] = 1; j = p[j]; } while (j >= 0 && t[j] == 0);
		if (j < 0) {
			if (n_v - n_v0 >= P.min_cnt) u[k++] = u[i] >> 32 << 32 | (uint64_t)(n_v - n_v0);
		} else if ((int32_t)(u[i] >> 32) - f[j] >= P.min_sc) {
			if (n_v - n_v0 >= P.min_cnt) u[k++] = ((u[i] >> 32) - (uint64_t)f[j]) << 32 | (uint64_t)(n_v - n_v0);
		}
		if (k0 == k) n_v = n_v0;
	}
	n_u = k;
	for (i = 0, k = 0; i < n_u; ++i) { // chain.c:137-141
		const int32_t k0 = k, ni = (int32_t)u[i];
		for (j = 0; j < ni; ++j) b[k] = a[v[k0 + (ni - j - 1)]], ++k;
	}
	mm128 *w = reinterpret_cast<mm128*>(f); // f|p|t|v are dead from here (chain.c:133,142)
	for (i = k = 0; i < n_u; ++i) { // chain.c:146-149
		w[i].x = b[k].x, w[i].y = (uint64_t)k << 32 | (uint64_t)i;
		k += (int32_t)u[i];
	}
	mmg_rs_sort_exact(w, n_u, stack, KeyX()); // chain.c:150
	uint64_t *u2 = u + n;
	for (i = k = 0; i < n_u; ++i) { // chain.c:152-157
		const int32_t jj = (int32_t)w[i].y, nn = (int32_t)u[jj];
		u2[i] = u[jj];
		const mm128 *src = &b[w[i].y >> 32];
		for (int32_t q = 0; q < nn; ++q) a[k + q] = src[q];
		k += nn;
	}
	for (i = 0; i < n_u; ++i) u[i] = u2[i];
	*n_v_out = k;
	return n_u;
}

// the DP fill of mm_chain_dp (chain.c:41-85), one thread walking the anchors in order
MMG_HDN inline uint64_t mmg_chain_fill_seq(const ChainParams &P, int64_t n, const mm128 *a, int32_t *f, int32_t *p, int32_t *t, int32_t *v)
{
	uint64_t sum_qspan = 0, n_iter = 0;
	int64_t i, j, st = 0;
	for (i = 0; i < n; ++i) sum_qspan += a[i].y >> 32 & 0xff, t[i] = 0;
	const float avg_qspan = (float)sum_qspan / (float)n; // chain.c:42
	for (i = 0; i < n; ++i) {
		const uint64_t ri = a[i].x;
		int64_t max_j = -1;
		const int32_t qi = (int32_t)a[i].y, q_span = (int32_t)(a[i].y >> 32 & 0xff);
		int32_t max_f = q_span, n_skip = 0;
		const int32_t sidi = (int32_t)((a[i].y & MMG_SEED_SEG_MASK) >> MMG_SEED_SEG_SHIFT);
		while (st < i && ri > a[st].x + (uint64_t)P.max_dist_x) ++st;
		if (i - st > P.max_iter) st = i - P.max_iter;
		for (j = i - 1; j >= st; --j) {
			int32_t sc;
			++n_iter;
			if (!mmg_chain_score(P, ri, qi, q_span, sidi, a[j], avg_qspan, &sc)) continue;
			sc += f[j];
			if (sc > max_f) {
				max_f = sc, max_j = j;
				if (n_skip > 0) --n_skip;
			} else if (t[j] == (int32_t)i) {
				if (++n_skip > P.max_skip) break;
			}
			if (p[j] >= 0) t[p[j]] = (int32_t)i;
		}
		f[i] = max_f, p[i] = (int32_t)max_j;
		v[i] = max_j >= 0 && v[max_j] > max_f ? v[max_j] : max_f;
	}
	return n_iter;
}

// ------------------------------------------------------------------ K4: ksw_extd2 pieces
#define MMG_KSW_NEG_INF (-0x40000000)
#define MMG_EZ_SCORE_ONLY 0x01
#define MMG_EZ_RIGHT 0x02
#define MMG_EZ_GENERIC_SC 0x04
#define MMG_EZ_APPROX_MAX 0x08
#define MMG_EZ_APPROX_DROP 0x10
#define MMG_EZ_EXTZ_ONLY 0x40
#define MMG_EZ_REV_CIGAR 0x80

struct KswEz {  // == mmg_extz_t
	uint32_t max; int32_t zdropped;
	int32_t max_q, max_t, mqe, mqe_t, mte, mte_q, score;
	int32_t n_cigar, reach_end;
};

struct KswGeom {  // per-job constants derived as in ksw2_extd2_sse.c:60-97
	int32_t qlen, tlen, w, tlen_, qlen_, n_col_, long_thres, long_diff;
	int32_t q, e, q2, e2, qe_pre, sc_mch, sc_mis, sc_N, m1;
	int32_t bail; // 1: returns before any DP (ksw2_extd2_sse.c:68,92)
};

MMG_HD KswGeom mmg_ksw_geom(int qlen, int tlen, int m, const int8_t *mat, int q, int e, int q2, int e2, int w)
{
	KswGeom g;
	g.qe_pre = q + e; // ksw2_extd2_sse.c:60 (before the swap at :70)
	g.bail = (m <= 1 || qlen <= 0 || tlen <= 0);
	if (q2 + e2 < q + e) { int t = q; q = q2, q2 = t; t = e, e = e2, e2 = t; }
	g.q = q, g.e = e, g.q2 = q2, g.e2 = e2;
	g.qlen = qlen, g.tlen = tlen;
	g.sc_mch = mat[0], g.sc_mis = mat[1];
	g.sc_N = mat[m * m - 1] == 0 ? -e2 : mat[m * m - 1];
	g.m1 = m - 1;
	if (w < 0) w = tlen > qlen ? tlen : qlen;
	g.w = w;
	g.tlen_ = (tlen + 15) / 16;
	int nc = qlen < tlen ? qlen : tlen;
	g.n_col_ = ((nc < w + 1 ? nc : w + 1) + 15) / 16 + 1;
	g.qlen_ = (qlen + 15) / 16;
	int min_sc = mat[1];
	for (int t = 1; t < m * m; ++t) min_sc = min_sc < mat[t] ? min_sc : mat[t];
	if (-min_sc > 2 * (q + e)) g.bail = 1;
	g.long_thres = e != e2 ? (q2 - q) / (e - e2) - 1 : 0;
	if (q2 + e2 + g.long_thres * e2 > q + e + g.long_thres * e) ++g.long_thres;
	g.long_diff = g.long_thres * (e - e2) - (q2 - q) - e2;
	return g;
}

// band of anti-diagonal r (ksw2_extd2_sse.c:124-139); false when the band is empty
MMG_HD bool mmg_ksw_band(const KswGeom &g, int r, int *st0, int *en0)
{
	int st = 0, en = g.tlen - 1;
	if (st < r - g.qlen + 1) st = r - g.qlen + 1;
	if (en > r) en = r;
	if (st < (r - g.w + 1) >> 1) st = (r - g.w + 1) >> 1;
	if (en > (r + g.w) >> 1) en = (r + g.w) >> 1;
	*st0 = st, *en0 = en;
	return st <= en;
}

MMG_HD int mmg_ksw_first_col(const KswGeom &g, int r)  // v1/u[r] boundary value (ksw2_extd2_sse.c:150,154)
{
	return r == 0 ? -g.q - g.e : r < g.long_thres ? -g.e : r == g.long_thres ? g.long_diff : -g.e2;
}

struct KswCell { int8_t u, v, x, y, x2, y2; uint8_t d; };

// one DP cell: z = s; a = x[t-1]+v[t-1]; b = y[t]+u[t]; ... (ksw2_extd2_sse.c:30-58,184-313); int8 wrap-around kept
template <int kMode /*0 score only, 1 left-aligned gaps, 2 right-aligned gaps*/>
MMG_HD KswCell mmg_ksw_cell(const KswGeom &g, int8_t z, int8_t xt1, int8_t vt1, int8_t ut, int8_t yt, int8_t x2t1, int8_t y2t)
{
	KswCell c;
	int8_t a = (int8_t)(xt1 + vt1), b = (int8_t)(yt + ut), a2 = (int8_t)(x2t1 + vt1), b2 = (int8_t)(y2t + ut), tmp;
	uint8_t d = 0;
	if (kMode == 0) {
		z = z > a ? z : a; z = z > b ? z : b; z = z > a2 ? z : a2; z = z > b2 ? z : b2;
	} else if (kMode == 1) {
		d = a > z ? 1 : 0;   z = z > a ? z : a;
		d = b > z ? 2 : d;   z = z > b ? z : b;
		d = a2 > z ? 3 : d;  z = z > a2 ? z : a2;
		d = b2 > z ? 4 : d;  z = z > b2 ? z : b2;
	} else {
		d = z > a ? 0 : 1;   z = z > a ? z : a;
		d = z > b ? d : 2;   z = z > b ? z : b;
		d = z > a2 ? d : 3;  z = z > a2 ? z : a2;
		d = z > b2 ? d : 4;  z = z > b2 ? z : b2;
	}
	z = z < (int8_t)g.sc_mch ? z : (int8_t)g.sc_mch;
	c.u = (int8_t)(z - vt1);
	c.v = (int8_t)(z - ut);
	tmp = (int8_t)(z - g.q);  a = (int8_t)(a - tmp);   b = (int8_t)(b - tmp);
	tmp = (int8_t)(z - g.q2); a2 = (int8_t)(a2 - tmp); b2 = (int8_t)(b2 - tmp);
	const int8_t qe = (int8_t)(g.q + g.e), qe2 = (int8_t)(g.q2 + g.e2);
	if (kMode != 2) { // continuation iff strictly positive
		c.x  = (int8_t)((a  > 0 ? a  : 0) - qe);  if (kMode && a  > 0) d |= 0x08;
		c.y  = (int8_t)((b  > 0 ? b  : 0) - qe);  if (kMode && b  > 0) d |= 0x10;
		c.x2 = (int8_t)((a2 > 0 ? a2 : 0) - qe2); if (kMode && a2 > 0) d |= 0x20;
		c.y2 = (int8_t)((b2 > 0 ? b2 : 0) - qe2); if (kMode && b2 > 0) d |= 0x40;
	} else { // continuation iff non-negative
		c.x  = (int8_t)((a  < 0 ? 0 : a)  - qe);  if (!(a  < 0)) d |= 0x08;
		c.y  = (int8_t)((b  < 0 ? 0 : b)  - qe);  if (!(b  < 0)) d |= 0x10;
		c.x2 = (int8_t)((a2 < 0 ? 0 : a2) - qe2); if (!(a2 < 0)) d |= 0x20;
		c.y2 = (int8_t)((b2 < 0 ? 0 : b2) - qe2); if (!(b2 < 0)) d |= 0x40;
	}
	c.d = d;
	return c;
}

MMG_HD int8_t mmg_ksw_score(const KswGeom &g, uint8_t tb, uint8_t qb)  // ksw2_extd2_sse.c:160-171
{
	int8_t z = tb == qb ? (int8_t)g.sc_mch : (int8_t)g.sc_mis;
	if (tb == (uint8_t)g.m1 || qb == (uint8_t)g.m1) z = (int8_t)g.sc_N;
	return z;
}

// order in which the reference's exact-max scan (ksw2_extd2_sse.c:319-349) prefers equal scores:
// H[en0] first, then the four strided lanes (each keeping its first hit, merged lane 0..3), then the tail
MMG_HD uint32_t mmg_ksw_max_rank(int t, int st0, int en0)
{
	if (t == en0) return 0;
	const int en1 = st0 + (en0 - st0) / 4 * 4;
	if (t < en1) return 1u + ((uint32_t)((t - st0) & 3) << 24) + (uint32_t)((t - st0) >> 2);
	return 1u + (4u << 24) + (uint32_t)(t - en1);
}

MMG_HD void mmg_ksw_reset(KswEz *ez)  // ksw_reset_extz, ksw2.h:153-158
{
	ez->max_q = ez->max_t = ez->mqe_t = ez->mte_q = -1;
	ez->max = 0, ez->score = ez->mqe = ez->mte = MMG_KSW_NEG_INF;
	ez->n_cigar = 0, ez->zdropped = 0, ez->reach_end = 0;
}

MMG_HD int mmg_ksw_zdrop(KswEz *ez, int32_t H, int r, int t, int zdrop, int e)  // ksw_apply_zdrop, ksw2.h:160-176 (is_rot)
{
	if (H > (int32_t)ez->max) {
		ez->max = (uint32_t)H, ez->max_t = t, ez->max_q = r - t;
	} else if (t >= ez->max_t && r - t >= ez->max_q) {
		const int tl = t - ez->max_t, ql = (r - t) - ez->max_q;
		const int l = tl > ql ? tl - ql : ql - tl;
		if (zdrop >= 0 && (int32_t)ez->max - H > zdrop + l * e) { ez->zdropped = 1; return 1; }
	}
	return 0;
}

// ksw_backtrack (ksw2.h:119-151; is_rot=1, min_intron_len=0) + ksw_push_cigar (ksw2.h:103-113).
// off[r]/off_end[r] are recomputed from the geometry instead of being stored.
MMG_HDN inline int mmg_ksw_backtrack(const KswGeom &g, int is_rev, const uint8_t *p, int i0, int j0, uint32_t *cigar)
{
	int n = 0, i = i0, j = j0, state = 0;
	const int n_col = g.n_col_ * 16;
#define MMG_PUSH(op, len) do { if (n == 0 || (uint32_t)(op) != (cigar[n - 1] & 0xf)) cigar[n++] = (uint32_t)(len) << 4 | (uint32_t)(op); else cigar[n - 1] += (uint32_t)(len) << 4; } while (0)
	while (i >= 0 && j >= 0) {
		int force_state = -1, st0, en0;
		const int r = i + j;
		mmg_ksw_band(g, r, &st0, &en0);
		const int off = st0 / 16 * 16, off_end = (en0 + 16) / 16 * 16 - 1;
		if (i < off) force_state = 2;
		if (i > off_end) force_state = 1;
		const uint32_t tmp = force_state < 0 ? p[(size_t)r * n_col + i - off] : 0;
		if (state == 0) state = tmp & 7;
		else if (!(tmp >> (state + 2) & 1)) state = 0;
		if (state == 0) state = tmp & 7;
		if (force_state >= 0) state = force_state;
		if (state == 0) { MMG_PUSH(0, 1); --i, --j; }
		else if (state == 1 || state == 3) { MMG_PUSH(2, 1); --i; }
		else { MMG_PUSH(1, 1); --j; }
	}
	if (i >= 0) MMG_PUSH(2, i + 1);
	if (j >= 0) MMG_PUSH(1, j + 1);
#undef MMG_PUSH
	if (!is_rev)
		for (int k = 0; k < n >> 1; ++k) { uint32_t t = cigar[k]; cigar[k] = cigar[n - 1 - k]; cigar[n - 1 - k] = t; }
	return n;
}

// which traceback (if any) runs after the DP (ksw2_extd2_sse.c:381-391)
MMG_HD bool mmg_ksw_trace_start(const KswGeom &g, int flag, int end_bonus, KswEz *ez, int *i0, int *j0)
{
	if (!ez->zdropped && !(flag & MMG_EZ_EXTZ_ONLY)) { *i0 = g.tlen - 1, *j0 = g.qlen - 1; return true; }
	if (!ez->zdropped && (flag & MMG_EZ_EXTZ_ONLY) && ez->mqe + end_bonus > (int)ez->max) {
		ez->reach_end = 1; *i0 = ez->mqe_t, *j0 = g.qlen - 1; return true;
	}
	if (ez->max_t >= 0 && ez->max_q >= 0) { *i0 = ez->max_t, *j0 = ez->max_q; return true; }
	return false;
}

// ksw_extd2 for one job walked by ONE thread: the 16 int8 lanes of each SSE block are visited in order with the
// previous lane's old x/v/x2 carried in registers, so the result is the reference's lane for lane (same widened band,
// stale lanes, spill of the score chunk into sf[], exact-max tie order).  `mem` holds u|v|x|y|x2|y2|s|sf|qr as laid out
// by mmg_ksw_mem_bytes(); the caller has filled sf[] (target, zero padded) and qr[] (reversed query, zero padded).
// This is the form used for the short-read job mix (hundreds of thousands of tiny DPs): one job per thread.
template <int kMode>
MMG_HDN inline void mmg_ksw_scalar_run(const KswGeom &g, int flag, int zdrop, int8_t *mem, int32_t *H, uint8_t *p, KswEz &ez)
{
	const int tl16 = g.tlen_ * 16, qlen = g.qlen, tlen = g.tlen;
	int8_t *u = mem, *v = u + tl16, *x = v + tl16, *y = x + tl16, *x2 = y + tl16, *y2 = x2 + tl16, *s = y2 + tl16;
	const uint8_t *sf = reinterpret_cast<const uint8_t*>(s + tl16), *qr = sf + tl16;
	const bool approx = (flag & MMG_EZ_APPROX_MAX) != 0;
	const int8_t n1 = (int8_t)(-g.q - g.e), n2 = (int8_t)(-g.q2 - g.e2);
	for (int i = 0; i < tl16; ++i) { u[i] = v[i] = x[i] = y[i] = n1; x2[i] = y2[i] = n2; s[i] = 0; H[i] = MMG_KSW_NEG_INF; }
	int last_st = -1, last_en = -1;
	int32_t H0 = 0, last_H0_t = 0;
	for (int r = 0; r < qlen + tlen - 1; ++r) {
		int st0, en0;
		if (!mmg_ksw_band(g, r, &st0, &en0)) { ez.zdropped = 1; break; }
		const int st = st0 / 16 * 16, en = (en0 + 16) / 16 * 16 - 1;
		int8_t x1, x21, v1;
		if (st > 0) {
			if (st - 1 >= last_st && st - 1 <= last_en) x1 = x[st - 1], x21 = x2[st - 1], v1 = v[st - 1];
			else x1 = n1, x21 = n2, v1 = n1;
		} else x1 = n1, x21 = n2, v1 = (int8_t)mmg_ksw_first_col(g, r);
		if (en >= r) y[r] = n1, y2[r] = n2, u[r] = (int8_t)mmg_ksw_first_col(g, r);
		{
			const uint8_t *qrr = qr + (qlen - 1 - r);
			for (int t = st0; t <= en0; t += 16)
				for (int l = 0; l < 16; ++l) s[t + l] = mmg_ksw_score(g, sf[t + l], qrr[t + l]);
		}
		for (int blk = st / 16; blk <= en / 16; ++blk) {
			const int base = blk * 16;
			uint8_t *pr = kMode ? p + ((size_t)r * g.n_col_ + (blk - st / 16)) * 16 : nullptr;
#pragma unroll 4
			for (int l = 0; l < 16; ++l) {
				const int i = base + l;
				const int8_t xo = x[i], vo = v[i], x2o = x2[i];
				const KswCell c = mmg_ksw_cell<kMode>(g, s[i], x1, v1, u[i], y[i], x21, y2[i]);
				u[i] = c.u, v[i] = c.v, x[i] = c.x, y[i] = c.y, x2[i] = c.x2, y2[i] = c.y2;
				if (kMode) pr[l] = c.d;
				x1 = xo, v1 = vo, x21 = x2o;
			}
		}
		if (!approx) {
			int32_t max_H, max_t, H_en0;
			if (r > 0) {
				H_en0 = en0 > 0 ? H[en0 - 1] + u[en0] : H[en0] + v[en0];
				int32_t bh = H_en0, bt = en0; uint32_t br = 0;
				for (int t = st0; t < en0; ++t) {
					const int32_t h = H[t] + v[t];
					H[t] = h;
					const uint32_t rk = mmg_ksw_max_rank(t, st0, en0);
					if (h > bh || (h == bh && rk < br)) bh = h, bt = t, br = rk;
				}
				H[en0] = H_en0;
				max_H = bh, max_t = bt;
			} else { H_en0 = v[0] - g.qe_pre; H[0] = H_en0; max_H = H_en0, max_t = 0; }
			if (en0 == tlen - 1 && H_en0 > ez.mte) ez.mte = H_en0, ez.mte_q = r - en;
			if (r - st0 == qlen - 1) { const int32_t hs = H[st0]; if (hs > ez.mqe) ez.mqe = hs, ez.mqe_t = st0; }
			if (mmg_ksw_zdrop(&ez, max_H, r, max_t, zdrop, g.e2)) break;
			if (r == qlen + tlen - 2 && en0 == tlen - 1) ez.score = H[tlen - 1];
		} else {
			if (r > 0) {
				if (last_H0_t >= st0 && last_H0_t <= en0 && last_H0_t + 1 >= st0 && last_H0_t + 1 <= en0) {
					const int32_t d0 = v[last_H0_t], d1 = u[last_H0_t + 1];
					if (d0 > d1) H0 += d0; else H0 += d1, ++last_H0_t;
				} else if (last_H0_t >= st0 && last_H0_t <= en0) H0 += v[last_H0_t];
				else ++last_H0_t, H0 += u[last_H0_t];
			} else H0 = v[0] - g.qe_pre, last_H0_t = 0;
			if ((flag & MMG_EZ_APPROX_DROP) && mmg_ksw_zdrop(&ez, H0, r, last_H0_t, zdrop, g.e2)) break;
			if (r == qlen + tlen - 2 && en0 == tlen - 1) ez.score = H0;
		}
		last_st = st, last_en = en;
	}
}

MMG_HDN inline void mmg_ksw_scalar(const KswGeom &g, int flag, int zdrop, int end_bonus, int8_t *mem, int32_t *H, uint8_t *p, KswEz *ez_out, uint32_t *cigar)
{
	KswEz ez;
	mmg_ksw_reset(&ez);
	const bool with_cigar = !(flag & MMG_EZ_SCORE_ONLY);
	if (!with_cigar) mmg_ksw_scalar_run<0>(g, flag, zdrop, mem, H, p, ez);
	else if (!(flag & MMG_EZ_RIGHT)) mmg_ksw_scalar_run<1>(g, flag, zdrop, mem, H, p, ez);
	else mmg_ksw_scalar_run<2>(g, flag, zdrop, mem, H, p, ez);
	int i0, j0;
	if (with_cigar && mmg_ksw_trace_start(g, flag, end_bonus, &ez, &i0, &j0))
		ez.n_cigar = mmg_ksw_backtrack(g, !!(flag & MMG_EZ_REV_CIGAR), p, i0, j0, cigar);
	*ez_out = ez;
}

// ---- K4 fast form: jobs whose band never binds ------------------------------------------------------------------
// When [st0,en0] is the whole anti-diagonal for every r (ksw2_extd2_sse.c:124-139 with a band that never clips), no valid
// cell ever reads one of the stale out-of-band lanes of the SSE program (every predecessor is itself a valid cell or one of
// the explicitly initialised first-row/first-column values), the traceback never leaves the matrix, and the exact-max scan
// only sees valid cells.  The result is then the plain difference-form DP, so one thread can sweep each anti-diagonal over
// exactly its valid cells.  Per-cell state (u,v,x,y,x2,y2 and a 16-bit H) is one 64-bit word in a circular window of
// min(qlen,tlen)+1 slots; element i of every per-job array sits at [i*stride] so that the threads of a CTA interleave.
MMG_HD bool mmg_ksw_band_clips(const KswGeom &g, int r)
{
	int st = 0, en = g.tlen - 1;
	if (st < r - g.qlen + 1) st = r - g.qlen + 1;
	if (en > r) en = r;
	return st < ((r - g.w + 1) >> 1) || en > ((r + g.w) >> 1);
}

MMG_HD int mmg_ksw_fast_pw(int qlen, int tlen) { return ((qlen < tlen ? qlen : tlen) + 3) & ~3; } // traceback row width
MMG_HD size_t mmg_ksw_fast_p_bytes(int qlen, int tlen) { return ((size_t)(qlen + tlen - 1) * mmg_ksw_fast_pw(qlen, tlen) + 15) & ~(size_t)15; }
// limits of the fast form's packed max key (score << 11 | preference): scores stay far below 2^20 and an anti-diagonal
// has at most 1024 cells
MMG_HD bool mmg_ksw_fast_ok(const KswGeom &g)
{
	int m = g.sc_mch > -g.sc_mis ? g.sc_mch : -g.sc_mis;
	if (m < -g.sc_N) m = -g.sc_N;
	if (m < g.q + g.e) m = g.q + g.e;
	if (m < g.q2 + g.e2) m = g.q2 + g.e2;
	return (int64_t)(g.qlen + g.tlen + 2) * m < 500000 && (g.qlen < g.tlen ? g.qlen : g.tlen) <= 1023;
}

#ifndef MMG_KSW_RANGE   // the emulation harness defines this to prove that no value of a valid cell leaves the int8 range
#define MMG_KSW_RANGE(v) ((void)0)
#endif

struct KswCell32 { int32_t u, v, x, y, x2, y2; uint32_t d; };

// mmg_ksw_cell in 32-bit registers: identical as long as nothing wraps, which holds for valid cells (checked by the
// emulation tests through MMG_KSW_RANGE; ksw2's scoring constraints, options.c:171-180, are what guarantee it)
template <int kMode>
MMG_HD KswCell32 mmg_ksw_cell32(const KswGeom &g, int32_t z, int32_t xt1, int32_t vt1, int32_t ut, int32_t yt, int32_t x2t1, int32_t y2t)
{
	KswCell32 c;
	int32_t a = xt1 + vt1, b = yt + ut, a2 = x2t1 + vt1, b2 = y2t + ut, tmp;
	uint32_t d = 0;
	MMG_KSW_RANGE(a); MMG_KSW_RANGE(b); MMG_KSW_RANGE(a2); MMG_KSW_RANGE(b2);
	if (kMode == 0) {
		z = z > a ? z : a; z = z > b ? z : b; z = z > a2 ? z : a2; z = z > b2 ? z : b2;
	} else if (kMode == 1) {
		d = a > z ? 1 : 0;   z = z > a ? z : a;
		d = b > z ? 2 : d;   z = z > b ? z : b;
		d = a2 > z ? 3 : d;  z = z > a2 ? z : a2;
		d = b2 > z ? 4 : d;  z = z > b2 ? z : b2;
	} else {
		d = z > a ? 0 : 1;   z = z > a ? z : a;
		d = z > b ? d : 2;   z = z > b ? z : b;
		d = z > a2 ? d : 3;  z = z > a2 ? z : a2;
		d = z > b2 ? d : 4;  z = z > b2 ? z : b2;
	}
	z = z < g.sc_mch ? z : g.sc_mch;
	c.u = z - vt1;
	c.v = z - ut;
	tmp = z - g.q;  a -= tmp;  b -= tmp;
	MMG_KSW_RANGE(tmp);
	tmp = z - g.q2; a2 -= tmp; b2 -= tmp;
	MMG_KSW_RANGE(tmp); MMG_KSW_RANGE(c.u); MMG_KSW_RANGE(c.v); MMG_KSW_RANGE(a); MMG_KSW_RANGE(b); MMG_KSW_RANGE(a2); MMG_KSW_RANGE(b2);
	const int32_t qe = g.q + g.e, qe2 = g.q2 + g.e2;
	if (kMode != 2) {
		c.x  = (a  > 0 ? a  : 0) - qe;  if (kMode && a  > 0) d |= 0x08;
		c.y  = (b  > 0 ? b  : 0) - qe;  if (kMode && b  > 0) d |= 0x10;
		c.x2 = (a2 > 0 ? a2 : 0) - qe2; if (kMode && a2 > 0) d |= 0x20;
		c.y2 = (b2 > 0 ? b2 : 0) - qe2; if (kMode && b2 > 0) d |= 0x40;
	} else {
		c.x  = (a  < 0 ? 0 : a)  - qe;  if (!(a  < 0)) d |= 0x08;
		c.y  = (b  < 0 ? 0 : b)  - qe;  if (!(b  < 0)) d |= 0x10;
		c.x2 = (a2 < 0 ? 0 : a2) - qe2; if (!(a2 < 0)) d |= 0x20;
		c.y2 = (b2 < 0 ? 0 : b2) - qe2; if (!(b2 < 0)) d |= 0x40;
	}
	MMG_KSW_RANGE(c.x); MMG_KSW_RANGE(c.y); MMG_KSW_RANGE(c.x2); MMG_KSW_RANGE(c.y2);
	c.d = d;
	return c;
}

// state word of a cell: u | v<<8 | x<<16 | y<<24 | x2<<32 | y2<<40 | target base<<48
#define MMG_KSW_PACK6(u, v, x, y, x2, y2) ((uint64_t)((uint32_t)((u) & 0xff) | (uint32_t)((v) & 0xff) << 8 | (uint32_t)((x) & 0xff) << 16 | (uint32_t)(y) << 24) | \
	(uint64_t)((uint32_t)((x2) & 0xff) | (uint32_t)((y2) & 0xff) << 8) << 32)
#define MMG_KSW_TB_MASK 0x00ff000000000000ULL

template <int kMode>
MMG_HDN inline void mmg_ksw_fast_run(const KswGeom &g, int flag, int zdrop, uint64_t *S, const uint8_t *tb, const uint8_t *qb, int stride,
                                     uint32_t *p /* rows of mmg_ksw_fast_pw() bytes */, KswEz &ez)
{
	const int qlen = g.qlen, tlen = g.tlen;
	const int W = (qlen < tlen ? qlen : tlen) + 1, PWw = mmg_ksw_fast_pw(qlen, tlen) >> 2;
	const bool approx = (flag & MMG_EZ_APPROX_MAX) != 0;
	const int32_t n1 = -g.q - g.e, n2 = -g.q2 - g.e2;
	uint64_t *const S_end = S + (size_t)W * stride;
	uint64_t *sp_st = S;      // window slot of cell st0
	int32_t Hst = 0;          // H of cell st0 of the previous anti-diagonal
	int32_t H0 = 0, last_H0_t = 0;
	for (int r = 0; r < qlen + tlen - 1; ++r) {
		const int st0 = r - qlen + 1 > 0 ? r - qlen + 1 : 0, en0 = r < tlen - 1 ? r : tlen - 1, n = en0 - st0 + 1;
		const int32_t fc = mmg_ksw_first_col(g, r);
		int32_t cx, cv, cx2; // x, v, x2 of cell t-1 on the previous anti-diagonal
		if (st0 == 0) cx = n1, cx2 = n2, cv = fc;
		else {
			const uint64_t w = *(sp_st == S ? S_end - stride : sp_st - stride);
			cv = (int8_t)(w >> 8), cx = (int8_t)(w >> 16), cx2 = (int8_t)(w >> 32);
		}
		if (r < tlen) { // the cell entering on the first row: boundary u/y/y2 (ksw2_extd2_sse.c:152-156) and its target base
			uint64_t *sn = sp_st + (size_t)(n - 1) * stride;
			if (sn >= S_end) sn -= (size_t)W * stride;
			*sn = MMG_KSW_PACK6(fc, n1, n1, n1, n2, n2) | (uint64_t)tb[(size_t)r * stride] << 48;
		}
		uint64_t *sp = sp_st;
		const uint8_t *qp = qb + (size_t)(r - st0) * stride;
		// exact max: E_k = H(r,st0+k) - H(r,st0) + u_0 accumulates from u - v of neighbouring cells; key = E<<11 | preference
		int32_t E = 0, best = INT32_MIN;
		const int en1k = (n - 1) / 4 * 4;
		uint32_t pw = 0;
		uint32_t *prow = p + (size_t)r * PWw;
		int32_t v_last = 0;
		for (int k = 0; k < n; ++k) {
			const uint64_t w = *sp;
			const int32_t ou = (int8_t)w, ov = (int8_t)(w >> 8), ox = (int8_t)(w >> 16), oy = (int8_t)(w >> 24), ox2 = (int8_t)(w >> 32), oy2 = (int8_t)(w >> 40);
			const uint32_t tbase = (uint32_t)(w >> 48) & 0xff, qbase = *qp;
			int32_t s = tbase == qbase ? g.sc_mch : g.sc_mis;
			if ((tbase | qbase) & 4) s = g.sc_N; // codes are 0..4: either one is N
			const KswCell32 c = mmg_ksw_cell32<kMode>(g, s, cx, cv, ou, oy, cx2, oy2);
			*sp = MMG_KSW_PACK6(c.u, c.v, c.x, c.y, c.x2, c.y2) | (w & MMG_KSW_TB_MASK);
			cx = ox, cv = ov, cx2 = ox2;
			if (kMode) {
				pw = pw >> 8 | c.d << 24;
				if ((k & 3) == 3) prow[k >> 2] = pw;
			}
			E += c.u;
			{
				const int32_t rk = k < en1k ? ((k & 3) << 8 | k >> 2) : (4 << 8 | (k - en1k));
				const int32_t key = E * 2048 + (2046 - rk);
				best = best > key ? best : key;
			}
			E -= c.v; v_last = c.v;
			sp += stride; if (sp == S_end) sp = S;
			qp -= stride;
		}
		if (kMode && (n & 3)) prow[n >> 2] = pw >> ((4 - (n & 3)) << 3);
		if (!approx) {
			const uint64_t w0 = *sp_st;
			const int32_t u0 = (int8_t)w0, v0 = (int8_t)(w0 >> 8);
			const int32_t H_st0 = r == 0 ? v0 - g.qe_pre : Hst + (st0 > 0 ? u0 : v0);
			const int32_t off = H_st0 - u0, H_en0 = off + E + v_last;
			int32_t bh, bt;
			{ // the cell en0 wins every tie (ksw2_extd2_sse.c:319-349 starts from it)
				const int32_t key = (E + v_last) * 2048 + 2047;
				best = best > key ? best : key;
				const int32_t low = best & 2047;
				bh = ((best - low) >> 11) + off; // exact: best - low is a multiple of 2048
				if (low == 2047) bt = en0;
				else { const int32_t rk = 2046 - low; bt = (rk >> 8) == 4 ? st0 + en1k + (rk & 255) : st0 + ((rk & 255) << 2) + (rk >> 8); }
			}
			Hst = H_st0;
			if (en0 == tlen - 1 && H_en0 > ez.mte) ez.mte = H_en0, ez.mte_q = r - ((en0 + 16) / 16 * 16 - 1); // the widened end (ksw2_extd2_sse.c:352)
			if (r - st0 == qlen - 1 && H_st0 > ez.mqe) ez.mqe = H_st0, ez.mqe_t = st0;
			if (mmg_ksw_zdrop(&ez, bh, r, bt, zdrop, g.e2)) break;
			if (r == qlen + tlen - 2 && en0 == tlen - 1) ez.score = H_en0;
		} else { // ksw2_extd2_sse.c:359-375, reading the cells just written
#define MMG_FAST_AT(t_) S[(size_t)(((int)((sp_st - S) / stride) + ((t_) - st0)) % W) * stride]
			if (r > 0) {
				if (last_H0_t >= st0 && last_H0_t <= en0 && last_H0_t + 1 >= st0 && last_H0_t + 1 <= en0) {
					const int32_t d0 = (int8_t)(MMG_FAST_AT(last_H0_t) >> 8), d1 = (int8_t)MMG_FAST_AT(last_H0_t + 1);
					if (d0 > d1) H0 += d0; else H0 += d1, ++last_H0_t;
				} else if (last_H0_t >= st0 && last_H0_t <= en0) H0 += (int8_t)(MMG_FAST_AT(last_H0_t) >> 8);
				else { ++last_H0_t; H0 += (int8_t)MMG_FAST_AT(last_H0_t); }
			} else H0 = (int8_t)(S[0] >> 8) - g.qe_pre, last_H0_t = 0;
#undef MMG_FAST_AT
			if ((flag & MMG_EZ_APPROX_DROP) && mmg_ksw_zdrop(&ez, H0, r, last_H0_t, zdrop, g.e2)) break;
			if (r == qlen + tlen - 2 && en0 == tlen - 1) ez.score = H0;
		}
		if (r + 2 - qlen > 0) { sp_st += stride; if (sp_st == S_end) sp_st = S; } // st0 of the next anti-diagonal is one further
	}
}

MMG_HDN inline int mmg_ksw_backtrack_fast(const KswGeom &g, int is_rev, const uint8_t *p, int i0, int j0, uint32_t *cigar)
{ // ksw_backtrack (ksw2.h:119-151) over the fast form's rows; the walk cannot leave the band, so no forced states
	int n = 0, i = i0, j = j0, state = 0;
	const int pw = mmg_ksw_fast_pw(g.qlen, g.tlen);
#define MMG_PUSH(op, len) do { if (n == 0 || (uint32_t)(op) != (cigar[n - 1] & 0xf)) cigar[n++] = (uint32_t)(len) << 4 | (uint32_t)(op); else cigar[n - 1] += (uint32_t)(len) << 4; } while (0)
	while (i >= 0 && j >= 0) {
		const int r = i + j, st0 = r - g.qlen + 1 > 0 ? r - g.qlen + 1 : 0;
		const uint32_t tmp = p[(size_t)r * pw + i - st0];
		if (state == 0) state = tmp & 7;
		else if (!(tmp >> (state + 2) & 1)) state = 0;
		if (state == 0) state = tmp & 7;
		if (state == 0) { MMG_PUSH(0, 1); --i, --j; }
		else if (state == 1 || state == 3) { MMG_PUSH(2, 1); --i; }
		else { MMG_PUSH(1, 1); --j; }
	}
	if (i >= 0) MMG_PUSH(2, i + 1);
	if (j >= 0) MMG_PUSH(1, j + 1);
#undef MMG_PUSH
	if (!is_rev)
		for (int k = 0; k < n >> 1; ++k) { uint32_t t = cigar[k]; cigar[k] = cigar[n - 1 - k]; cigar[n - 1 - k] = t; }
	return n;
}

// one job, one thread: S/tb/qb as described above (tb[t], qb[j] already filled), p = this job's traceback rows
MMG_HDN inline void mmg_ksw_fast(const KswGeom &g, int flag, int zdrop, int end_bonus, uint64_t *S, const uint8_t *tb, const uint8_t *qb, int stride,
                                 uint32_t *p, KswEz *ez_out, uint32_t *cigar)
{
	KswEz ez;
	mmg_ksw_reset(&ez);
	const bool with_cigar = !(flag & MMG_EZ_SCORE_ONLY);
	if (!with_cigar) mmg_ksw_fast_run<0>(g, flag, zdrop, S, tb, qb, stride, p, ez);
	else if (!(flag & MMG_EZ_RIGHT)) mmg_ksw_fast_run<1>(g, flag, zdrop, S, tb, qb, stride, p, ez);
	else mmg_ksw_fast_run<2>(g, flag, zdrop, S, tb, qb, stride, p, ez);
	int i0, j0;
	if (with_cigar && mmg_ksw_trace_start(g, flag, end_bonus, &ez, &i0, &j0))
		ez.n_cigar = mmg_ksw_backtrack_fast(g, !!(flag & MMG_EZ_REV_CIGAR), reinterpret_cast<const uint8_t*>(p), i0, j0, cigar);
	*ez_out = ez;
}

// bytes of lane memory for one job, laid out as the reference does (ksw2_extd2_sse.c:99-102):
// u | v | x | y | x2 | y2 | s | sf | qr (+16 spare), all tlen_*16 except qr
MMG_HD size_t mmg_ksw_mem_bytes(int qlen, int tlen) { return ((size_t)((tlen + 15) / 16) * 8 + (size_t)((qlen + 15) / 16) + 1) * 16; }
