// mmg_stages.cu -- the batched sketch -> seed -> chain stages (K1, K2, K3) and their
// single-call test entry points.  Reference path: mm_map_frag, map.c:272-377.
#include <cub/cub.cuh>
#include "mmg_ctx.cuh"
#include "mmg_regheap.h"
#include "mmg_sketchwarp.h"
#include "mmg_rswarp.h"

int mmg_run_sketch(mmg_ctx_t *c, const uint32_t *d_S, const SketchUnit *d_units, int n_units, int w, int k, int is_hpc,
                   DevBuf &cnt, DevBuf &off, DevBuf &out, int64_t *total, bool short_reads, uint64_t stage_slots);

#define MMG_READ_CHUNK 4096   // reads longer than this are sketched in chunks

// ------------------------------------------------------------------ kernels

// ASCII reads -> 4-bit codes, one word (8 bases) per thread; flipped reads are reverse-complemented
// (mm_revcomp_bseq, bseq.h:46-58, applied to mates per pe_ori at map.c:467-469)
__global__ void k_encode_reads(const uint8_t *__restrict__ ascii, const uint64_t *__restrict__ seq_off, const int32_t *__restrict__ seq_len,
                               const uint64_t *__restrict__ q_off, const uint8_t *__restrict__ flip, int n_seq, uint64_t n_words,
                               uint32_t *__restrict__ Q)
{
	const uint64_t wi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (wi >= n_words) return;
	const uint64_t b0 = wi * 8;
	int lo = 0, hi = n_seq - 1; // last read with q_off <= b0
	while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (q_off[mid] <= b0) lo = mid; else hi = mid - 1; }
	const int r = lo, len = seq_len[r];
	const uint64_t base = b0 - q_off[r];
	const uint8_t *s = ascii + seq_off[r];
	const bool fl = flip[r] != 0;
	uint32_t word = 0;
	for (int j = 0; j < 8; ++j) {
		const uint64_t i = base + j;
		int c = 4;
		if (i < (uint64_t)len) {
			if (!fl) c = mmg_nt4(s[i]);
			else { c = mmg_nt4(s[len - 1 - i]); c = c < 4 ? 3 - c : 4; }
		}
		word |= (uint32_t)c << (4 * j);
	}
	Q[wi] = word;
}

// K2a: one lookup per query minimizer (mm_idx_get at map.c:103)
__global__ void k_lookup(IdxView ix, const mm128 *__restrict__ mv, int64_t n, int32_t *__restrict__ m_n, uint64_t *__restrict__ m_val)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	uint64_t val;
	m_n[i] = mmg_idx_probe(ix, mv[i].x >> 8, &val);
	m_val[i] = val;
}

struct FragTab {  // per-fragment tables of the resident batch
	const int32_t *unit0;      // [n_frag+1] first sketch unit of each fragment
	const int64_t *unit_off;   // [n_units+1] first minimizer of each unit
	const int32_t *qlen;       // [n_frag] summed segment lengths
};

struct NameTabs {  // the self/dual filters' name keys (include/mmg.h): per target of the index, per fragment of the resident batch
	const uint32_t *tkey, *tlen, *ukey;  // ukey null: the filters are off
};

__device__ __forceinline__ NameFilt name_filt(const NameTabs &nt, int f)
{
	NameFilt n;
	n.tkey = nt.tkey, n.tlen = nt.tlen, n.ukey = nt.ukey ? nt.ukey[f] : MMG_NAME_NONE;
	return n;
}

__device__ __forceinline__ int frag_of_anchor(const int64_t *aoff, int n_list, int64_t g)
{ // last li with aoff[li] <= g
	int lo = 0, hi = n_list - 1;
	while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (aoff[mid] <= g) lo = mid; else hi = mid - 1; }
	return lo;
}

// K2b: collect_matches bookkeeping per fragment (map.c:90-123)
__global__ void k_plan(FragTab ft, const int32_t *__restrict__ list, int n_list, const mm128 *__restrict__ mv, const int32_t *__restrict__ m_n,
                       int max_occ, int32_t *__restrict__ na, int32_t *__restrict__ rep, int32_t *__restrict__ nmini,
                       uint64_t *__restrict__ mini /* may be null */, uint8_t *__restrict__ replay /* may be null */, int32_t *__restrict__ m_aoff)
{
	const int li = blockIdx.x * blockDim.x + threadIdx.x;
	if (li >= n_list) return;
	const int f = list ? list[li] : li;
	const int64_t b = ft.unit_off[ft.unit0[f]], e = ft.unit_off[ft.unit0[f + 1]];
	int r, nm;
	const int64_t n_a = mmg_frag_plan(mv + b, m_n + b, (int)(e - b), max_occ, &r, &nm, mini ? mini + b : nullptr);
	na[li] = (int32_t)n_a, rep[li] = r, nmini[li] = nm;
	{ // first anchor slot of every minimizer inside the fragment (k_expand finds an anchor's minimizer by bisection)
		int32_t run = 0;
		for (int i = 0; i < (int)(e - b); ++i) {
			m_aoff[b + i] = run;
			const int n = m_n[b + i];
			if (n > 0 && n < max_occ) run += n;
		}
	}
	if (replay) {
		// Positions of different minimizers are disjoint, so two heap entries can only tie when two kept query minimizers
		// carry the same hash (tandem k-mers, overlapping mates; SURVEY.md H2).  Only those fragments need the heap replayed.
		const int m = (int)(e - b);
		uint8_t dup = m > 256 ? 1 : 0;
		for (int i = 0; i < m && !dup; ++i) {
			if (m_n[b + i] <= 0 || m_n[b + i] >= max_occ) continue;
			const uint64_t h = mv[b + i].x >> 8;
			for (int j = i + 1; j < m; ++j)
				if (mv[b + j].x >> 8 == h && m_n[b + j] > 0 && m_n[b + j] < max_occ) { dup = 1; break; }
		}
		if (dup) { // 1: the heap is replayed on ranks (k_heap_replay); 2: too many lists or anchors for its packed words -> literal replay (k_fill)
			int kept = 0;
			for (int i = 0; i < m; ++i) kept += m_n[b + i] > 0 && m_n[b + i] < max_occ;
			dup = (kept <= 256 && n_a < (1 << 24)) ? 1 : 2;
		}
		replay[li] = dup;
	}
}

// K2c, sort form (fragments without repeated hashes): every planned anchor slot finds its (minimizer, hit), and emits the
// heap's pop key (strand class, reference position incl. strand bit) with the anchor's y as payload
template <bool kNamed>
__global__ void k_expand(FragTab ft, const int32_t *__restrict__ list, int n_list, const mm128 *__restrict__ mv, const int32_t *__restrict__ m_n,
                         const uint64_t *__restrict__ m_val, const uint64_t *__restrict__ pos, int max_occ, int64_t flag,
                         const int64_t *__restrict__ aoff, const uint8_t *__restrict__ replay, int64_t n_total,
                         uint64_t *__restrict__ key, uint64_t *__restrict__ val, int32_t *__restrict__ n_skipped, const int32_t *__restrict__ m_aoff,
                         NameTabs nt, unsigned long long *__restrict__ n_named)
{
	const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (g >= n_total) return;
	const int li = frag_of_anchor(aoff, n_list, g);
	if (replay[li] == 2) return; // segment of length zero in the sort
	const int f = list ? list[li] : li;
	const int64_t b = ft.unit_off[ft.unit0[f]], e = ft.unit_off[ft.unit0[f + 1]];
	int64_t i = g - aoff[li];
	int m;
	{ // last minimizer whose first slot is <= i: it is a kept one, because dropped minimizers have empty slot ranges
		int lo = 0, hi = (int)(e - b) - 1;
		while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (m_aoff[b + mid] <= i) lo = mid; else hi = mid - 1; }
		m = lo;
		i -= m_aoff[b + m];
	}
	const mm128 mz = mv[b + m];
	const uint64_t r = mmg_hit_pos(pos, m_n[b + m], m_val[b + m], (uint32_t)i);
	if (replay[li] == 1) { key[g] = r, val[g] = (uint64_t)(g - aoff[li]); return; } // heap replay: ordered by position alone, the planned slot as payload
	bool self;
	const int sk = mmg_skip_seed(MMG_NAMED_FLAG(kNamed, flag), r, (uint32_t)mz.y, name_filt(nt, f), kNamed ? ft.qlen[f] : 0, &self);
	if (sk != MMG_SKIP_KEEP) {
		key[g] = MMG_NONE, val[g] = 0; atomicAdd(&n_skipped[li], 1);
		if (kNamed && sk == MMG_SKIP_NAME) atomicAdd(n_named, 1ULL);
		return;
	}
	const mm128 an = mmg_make_anchor(r, mz, mmg_is_tandem(mv + b, (int)(e - b), m), self, ft.qlen[f]);
	key[g] = (an.x & (1ULL << 63)) | r; // r < 2^63
	val[g] = an.y; // the self bit rides here
}

__global__ void k_sort_segments(int n_list, const int64_t *__restrict__ aoff, const uint8_t *__restrict__ replay, int64_t *__restrict__ seg_b, int64_t *__restrict__ seg_e)
{
	const int li = blockIdx.x * blockDim.x + threadIdx.x;
	if (li >= n_list) return;
	seg_b[li] = aoff[li];
	seg_e[li] = replay[li] == 2 ? aoff[li] : aoff[li + 1];
}

__global__ void k_emit_sorted(int n_list, const int64_t *__restrict__ aoff, const uint8_t *__restrict__ replay, int64_t n_total,
                              const uint64_t *__restrict__ key, const uint64_t *__restrict__ val, const int32_t *__restrict__ n_skipped,
                              int32_t *__restrict__ na, mm128 *__restrict__ a, uint8_t *__restrict__ tie /* may be null */)
{
	const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (g >= n_total) return;
	const int li = frag_of_anchor(aoff, n_list, g);
	if (replay[li]) return;
	const uint64_t k = key[g];
	if (g == aoff[li]) na[li] = (int32_t)(aoff[li + 1] - aoff[li]) - n_skipped[li];
	if (k == MMG_NONE) return;
	const uint64_t r = k & ~(1ULL << 63);
	mm128 an;
	an.x = (k & (1ULL << 63)) | (r & 0xffffffff00000000ULL) | ((uint32_t)r >> 1);
	an.y = val[g];
	a[g] = an;
	if (tie && g > aoff[li]) { // radix-sort form (collect_seed_hits, map.c:215-247): two anchors with the same x leave klib's sort in an order only a replay gives
		const uint64_t kp = key[g - 1], rp = kp & ~(1ULL << 63);
		if (((kp & (1ULL << 63)) | (rp & 0xffffffff00000000ULL) | ((uint32_t)rp >> 1)) == an.x) tie[li] = 1;
	}
}

// K2c, radix-sort form, fragments in which two anchors share x: the anchors in query order (the planned slots k_expand filled,
// minus the skipped seeds) and klib's radix sort replayed by a warp (mmg_rswarp.h).  work[] is free until the chain fill.
__global__ void __launch_bounds__(128)
k_fill_flat_warp(int n_list, const int64_t *__restrict__ aoff, const uint8_t *__restrict__ tie, const uint64_t *__restrict__ key,
                 const uint64_t *__restrict__ val, int32_t *__restrict__ na, mm128 *__restrict__ a, int32_t *__restrict__ work, RsFrame *__restrict__ stack)
{
	__shared__ int32_t s_head[4][256], s_tail[4][256];
	const int li = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
	if (li >= n_list || tie[li] != 1) return;
	const int64_t ao = aoff[li];
	const int32_t n_plan = (int32_t)(aoff[li + 1] - ao);
	mm128 *A = a + ao;
	int32_t o = 0;
	for (int32_t i0 = 0; i0 < n_plan; i0 += 32) {
		const int32_t i = i0 + lane;
		const uint64_t k = i < n_plan ? key[ao + i] : MMG_NONE;
		const unsigned m = __ballot_sync(0xffffffffu, k != MMG_NONE);
		if (k != MMG_NONE) {
			const uint64_t r = k & ~(1ULL << 63);
			mm128 an;
			an.x = (k & (1ULL << 63)) | (r & 0xffffffff00000000ULL) | ((uint32_t)r >> 1);
			an.y = val[ao + i];
			A[o + __popc(m & ((1u << lane) - 1u))] = an;
		}
		o += __popc(m);
	}
	__syncwarp();
	mm128 *tmp = reinterpret_cast<mm128*>(work + ao * 8);
	int32_t *dst = reinterpret_cast<int32_t*>(tmp + n_plan);
	uint8_t *dig = reinterpret_cast<uint8_t*>(dst + n_plan);
	const WarpDev wp = {lane};
	mmg_rs_sort_warp(wp, A, (int64_t)o, tmp, dst, dig, stack + ao / 65 + 2 * (int64_t)li, s_head[wi], s_tail[wi], KeyX());
	if (lane == 0) na[li] = o;
}

// ---- K2c, heap replay on ranks (fragments in which two kept query minimizers share a hash: equal positions meet in the heap,
// and the order they leave it in is defined by klib's heap, SURVEY.md H2).  The sort above ordered the fragment's planned hits
// by position; the heap replay itself then needs no position at all (mmg_heap_replay_ranks).

// rank of every planned hit: index of the first hit with the same position
__global__ void k_heap_rank(int n_list, const int64_t *__restrict__ aoff, const uint8_t *__restrict__ replay, int64_t n_total,
                            const uint64_t *__restrict__ key, const uint64_t *__restrict__ val, uint32_t *__restrict__ K)
{
	const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (g >= n_total) return;
	const int li = frag_of_anchor(aoff, n_list, g);
	if (replay[li] != 1) return;
	const int64_t ao = aoff[li];
	int64_t l = g;
	const uint64_t k = key[g];
	while (l > ao && key[l - 1] == k) --l;
	K[ao + (int64_t)val[g]] = (uint32_t)(l - ao);
}

__global__ void k_heap_list(int n_list, const uint8_t *__restrict__ replay, int32_t *__restrict__ out, int32_t *__restrict__ counters)
{
	const int li = blockIdx.x * blockDim.x + threadIdx.x;
	if (li >= n_list) return;
	if (replay[li] == 1) out[atomicAdd(&counters[0], 1)] = li;
	else if (replay[li] == 2) atomicAdd(&counters[2], 1); // left to the literal replay of k_fill
}

#define HEAP_MAX_LISTS 256
#define HEAP_RING 16   // ranks of every list staged ahead of the replay in shared memory (a power of two)

// mmg_heap_replay_ranks (mmg_core.h) tuned for one lane: the same pops in the same order.  The serial chain per pop is what
// bounds a fragment with 10^5 hits (one lane, ~1.5 x 10^5 dependent pops), so nothing on that chain may wait for global memory:
// (a) the root stays in a register; (b) the next HEAP_RING ranks of every list sit in a shared-memory ring that asynchronous
// copies refill one element per pop, HEAP_RING pops of that list ahead of their use (a copy issued one pop ahead, as before,
// cost the full L2/HBM latency on every pop: 400 ns per pop); (c) the key the popped list puts back is read from nxt[], which is
// refreshed from the ring off the critical path; (d) the sift loads a node's children and grandchildren together and descends
// two levels per round of shared-memory latency.
struct HeapList { int32_t first, cnt, cur, m; };

__device__ __forceinline__ void heap_sift_root(uint32_t *l, uint32_t n, uint32_t tmp, uint32_t *root_out)
{
	uint32_t i = 0, root = tmp;
	const uint32_t INF = 0xffffffffu;
	for (;;) {
		const uint32_t c = 2 * i + 1;
		if (c >= n) break;
		const uint32_t g = 2 * c + 1; // grandchildren g .. g + 3
		const uint32_t a = l[c], b = c + 1 < n ? l[c + 1] : INF;
		const uint32_t g0 = g < n ? l[g] : INF, g1 = g + 1 < n ? l[g + 1] : INF, g2 = g + 2 < n ? l[g + 2] : INF, g3 = g + 3 < n ? l[g + 3] : INF;
		// level 1: the smaller child (the left one on ties); it moves up unless it is larger than tmp (ksort.h:47-51)
		const bool right = c + 1 < n && (a >> 8) > (b >> 8);
		const uint32_t k = right ? c + 1 : c, v = right ? b : a;
		if ((v >> 8) > (tmp >> 8)) break;
		l[i] = v;
		if (i == 0) root = v;
		i = k;
		// level 2 from registers
		const uint32_t c2 = 2 * k + 1;
		if (c2 >= n) break;
		const uint32_t a2 = right ? g2 : g0, b2 = right ? g3 : g1;
		const bool right2 = c2 + 1 < n && (a2 >> 8) > (b2 >> 8);
		const uint32_t k2 = right2 ? c2 + 1 : c2, v2 = right2 ? b2 : a2;
		if ((v2 >> 8) > (tmp >> 8)) break;
		l[i] = v2;
		i = k2;
	}
	l[i] = tmp;
	*root_out = i == 0 ? tmp : root;
}

// lists[], ring[] (first HEAP_RING ranks of every list) and nxt[] (rank 1 of every list) are set up by the warp; heap[] holds
// rank 0 of every list, not yet ordered
__device__ int64_t heap_replay_lane(int n_lists, HeapList *lists, const uint32_t *__restrict__ K, uint32_t *heap, uint32_t *nxt, uint32_t *ring, uint32_t *__restrict__ pop)
{
	uint32_t hs = (uint32_t)n_lists;
	int64_t t = 0;
	if (hs > 1) for (int32_t j = (int32_t)(hs >> 1) - 1; j >= 0; --j) mmg_rank_heap_down((uint32_t)j, hs, heap);
	uint32_t root = hs ? heap[0] : 0;
	while (hs > 0) {
		const uint32_t j = root & 0xff;
		const uint32_t key1 = nxt[j];      // rank of the list's element c + 1, if there is one
		const HeapList L = lists[j];
		const uint32_t c = (uint32_t)L.cur, n = (uint32_t)L.cnt, f0 = (uint32_t)L.first;
		pop[t++] = f0 + c;
		uint32_t tmp;
		if (c + 1 < n) {
			tmp = key1 << 8 | j;
			lists[j].cur = (int32_t)(c + 1);
			// element c + 2 was requested when element c + 2 - HEAP_RING was popped; this list alone has committed HEAP_RING - 3
			// groups since, so at most that many younger groups may still be in flight
			asm volatile("cp.async.wait_group %0;" :: "n"(HEAP_RING - 3) : "memory");
			if (c + 2 < n) nxt[j] = ring[j * HEAP_RING + ((c + 2) & (HEAP_RING - 1))];
			if (c + HEAP_RING < n) { // into the slot of element c, which is in the past
				const unsigned dst = (unsigned)__cvta_generic_to_shared(&ring[j * HEAP_RING + (c & (HEAP_RING - 1))]);
				asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(dst), "l"(K + f0 + c + HEAP_RING) : "memory");
			}
			asm volatile("cp.async.commit_group;" ::: "memory");
		} else { tmp = heap[hs - 1]; --hs; }
		if (hs > 0) heap_sift_root(heap, hs, tmp, &root);
	}
	asm volatile("cp.async.wait_all;" ::: "memory");
	return t;
}

// The warp form of the replay (mmg_regheap.h) with the lists' cursors in registers too: list j belongs to lane j & 31, which
// keeps its cursor and the rank of its next element in registers, so handing the next key to the heap is one shuffle and
// nothing the owner does afterwards (recording the pop, reading the rank after next from its ring, requesting the ring's next
// element) is waited for by the other lanes' next step.  Ring slots of a list are read and refilled by its owner only.
template <int NREG>
__device__ void heap_replay_warp(int n_lists, const HeapList *s_lists, const uint32_t *__restrict__ Kf, uint32_t *__restrict__ Pf, const uint32_t *s_heap, uint32_t *s_ring, int lane)
{
	const unsigned FULL = 0xffffffffu;
	uint32_t cur[NREG], cnt[NREG], first[NREG], nxt[NREG];
#pragma unroll
	for (int q = 0; q < NREG; ++q) {
		const int j = lane + 32 * q;
		cur[q] = 0, cnt[q] = 0, first[q] = 0, nxt[q] = RH_NONE;
		if (j < n_lists) { const HeapList L = s_lists[j]; cnt[q] = (uint32_t)L.cnt, first[q] = (uint32_t)L.first; if (L.cnt > 1) nxt[q] = s_ring[j * HEAP_RING + 1]; }
	}
	const WarpDev wp = {lane};
	const uint32_t ring_sa = (uint32_t)__cvta_generic_to_shared(s_ring); // taken once: the conversion reads a special register
	auto advance = [&](uint32_t j, int64_t t) -> uint32_t { // pop t is the current element of list j; hands out the rank of its next one
		const int q = (int)(j >> 5), ol = (int)(j & 31);
		uint32_t nk = RH_NONE;
#pragma unroll
		for (int qq = 0; qq < NREG; ++qq) { const uint32_t v = __shfl_sync(FULL, nxt[qq], ol); if (qq == q) nk = v; }
		if (lane == ol) {
#pragma unroll
			for (int qq = 0; qq < NREG; ++qq)
				if (qq == q) {
					const uint32_t c = cur[qq], n = cnt[qq];
					Pf[t] = first[qq] + c;
					if (c + 1 < n) {
						cur[qq] = c + 1;
						// element c + 2 was requested when element c + 2 - HEAP_RING was popped; this list alone has committed
						// HEAP_RING - 3 groups of this lane since, so at most that many younger groups may still be in flight
						asm volatile("cp.async.wait_group %0;" :: "n"(HEAP_RING - 3) : "memory");
						uint32_t v = RH_NONE;
						if (c + 2 < n) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(ring_sa + 4u * (j * HEAP_RING + ((c + 2) & (HEAP_RING - 1)))) : "memory");
						nxt[qq] = v;
						if (c + HEAP_RING < n) // into the slot of element c, which is in the past
							asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(ring_sa + 4u * (j * HEAP_RING + (c & (HEAP_RING - 1)))), "l"(Kf + first[qq] + c + HEAP_RING) : "memory");
						asm volatile("cp.async.commit_group;" ::: "memory");
					}
				}
		}
		return nk;
	};
	regheap_replay<WarpDev, NREG>(wp, n_lists, s_heap, advance);
	asm volatile("cp.async.wait_all;" ::: "memory");
	__syncwarp();
}

// one warp per listed fragment, pulled from a counter: the pop order of the fragment's heap merge, as planned slots, into P[]
__global__ void __launch_bounds__(32)
k_heap_replay(FragTab ft, const int32_t *__restrict__ list, const int32_t *__restrict__ rlist, int32_t *__restrict__ counters, const mm128 *__restrict__ mv,
              const int32_t *__restrict__ m_n, const uint64_t *__restrict__ m_val, const int32_t *__restrict__ m_aoff, const uint64_t *__restrict__ pos, int max_occ,
              int64_t flag, const int64_t *__restrict__ aoff, const uint32_t *__restrict__ K, uint32_t *__restrict__ P)
{
	__shared__ uint32_t s_heap[HEAP_MAX_LISTS], s_nxt[HEAP_MAX_LISTS], s_ring[HEAP_MAX_LISTS * HEAP_RING];
	__shared__ __align__(16) HeapList s_lists[HEAP_MAX_LISTS];
	const int lane = threadIdx.x & 31;
	const unsigned FULL = 0xffffffffu;
	const int n_work = counters[0];
	for (;;) {
		int t = 0;
		if (lane == 0) t = atomicAdd(&counters[1], 1);
		t = __shfl_sync(FULL, t, 0);
		if (t >= n_work) break;
		const int li = rlist[t], f = list ? list[li] : li;
		const int64_t b = ft.unit_off[ft.unit0[f]], e = ft.unit_off[ft.unit0[f + 1]], ao = aoff[li];
		const int n_mv = (int)(e - b);
		int n_lists = 0;
		for (int i0 = 0; i0 < n_mv; i0 += 32) { // the kept minimizers, in query order
			const int i = i0 + lane;
			const bool kept = i < n_mv && m_n[b + i] > 0 && m_n[b + i] < max_occ;
			const unsigned mk = __ballot_sync(FULL, kept);
			if (kept) { HeapList L; L.first = m_aoff[b + i], L.cnt = m_n[b + i], L.cur = 0, L.m = i; s_lists[n_lists + __popc(mk & ((1u << lane) - 1u))] = L; }
			n_lists += __popc(mk);
		}
		__syncwarp();
		for (int x = lane; x < n_lists * HEAP_RING; x += 32) { // the first ranks of every list
			const int j = x / HEAP_RING, e2 = x % HEAP_RING;
			if (e2 < s_lists[j].cnt) {
				const uint32_t k = K[ao + s_lists[j].first + e2];
				s_ring[x] = k;
				if (e2 == 0) s_heap[j] = k << 8 | (uint32_t)j;
				if (e2 == 1) s_nxt[j] = k;
			}
		}
		__syncwarp();
		if (n_lists <= 127) { // the heap in the warp's registers (mmg_regheap.h): a pop costs a fixed number of warp-wide steps
			if (lane == 0 && n_lists > 1) for (int32_t j = (n_lists >> 1) - 1; j >= 0; --j) mmg_rank_heap_down((uint32_t)j, (uint32_t)n_lists, s_heap);
			__syncwarp();
			if (n_lists <= 31) heap_replay_warp<1>(n_lists, s_lists, K + ao, P + ao, s_heap, s_ring, lane);
			else if (n_lists <= 63) heap_replay_warp<2>(n_lists, s_lists, K + ao, P + ao, s_heap, s_ring, lane);
			else heap_replay_warp<4>(n_lists, s_lists, K + ao, P + ao, s_heap, s_ring, lane);
		} else if (lane == 0) heap_replay_lane(n_lists, s_lists, K + ao, s_heap, s_nxt, s_ring, P + ao);
		__syncwarp();
	}
}

// exclusive scan of v over the CTA (blockDim.x a multiple of 32, <= 1024); s_w: 32 ints
__device__ __forceinline__ int block_excl_scan(int v, int *s_w, int *total)
{
	const unsigned FULL = 0xffffffffu;
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
	int incl = v;
#pragma unroll
	for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += o; }
	if (lane == 31) s_w[wid] = incl;
	__syncthreads();
	if (wid == 0) {
		int w = lane < nw ? s_w[lane] : 0;
#pragma unroll
		for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULL, w, d); if (lane >= d) w += o; }
		s_w[lane] = w;
	}
	__syncthreads();
	const int r = (wid ? s_w[wid - 1] : 0) + incl - v;
	*total = s_w[nw - 1];
	__syncthreads();
	return r;
}

// one CTA per replayed fragment: the pop order becomes anchors -- forward-strand hits in pop order, then reverse-strand hits in
// pop order (map.c:176-211).  (One warp did this after its replay: 2 x 5 000 rounds of dependent global loads for a fragment
// with 1.6 x 10^5 hits, as long as the replay itself.)
#define HEAP_EMIT_THREADS 512
template <bool kNamed>
__global__ void __launch_bounds__(HEAP_EMIT_THREADS)
k_heap_emit(FragTab ft, const int32_t *__restrict__ list, const int32_t *__restrict__ rlist, const mm128 *__restrict__ mv, const int32_t *__restrict__ m_n,
            const uint64_t *__restrict__ m_val, const int32_t *__restrict__ m_aoff, const uint64_t *__restrict__ pos, int max_occ, int64_t flag,
            const int64_t *__restrict__ aoff, uint32_t *__restrict__ P, int32_t *__restrict__ na, mm128 *__restrict__ a, unsigned long long *__restrict__ n_pops,
            NameTabs nt, unsigned long long *__restrict__ n_named)
{
	__shared__ int32_t s_first[HEAP_MAX_LISTS], s_m[HEAP_MAX_LISTS], s_w[32], s_tot[3];
	const int tid = threadIdx.x, lane = tid & 31, NT = blockDim.x;
	const unsigned FULL = 0xffffffffu;
	const int li = rlist[blockIdx.x], f = list ? list[li] : li;
	const int64_t b = ft.unit_off[ft.unit0[f]], e = ft.unit_off[ft.unit0[f + 1]], ao = aoff[li];
	const int n_mv = (int)(e - b), qlen = ft.qlen[f];
	const NameFilt nfl = name_filt(nt, f);
	if (tid < 32) { // the kept minimizers, in query order (as in k_heap_replay)
		int n_lists = 0, n_a = 0;
		for (int i0 = 0; i0 < n_mv; i0 += 32) {
			const int i = i0 + lane;
			const bool kept = i < n_mv && m_n[b + i] > 0 && m_n[b + i] < max_occ;
			const unsigned mk = __ballot_sync(FULL, kept);
			if (kept) { const int j = n_lists + __popc(mk & ((1u << lane) - 1u)); s_first[j] = m_aoff[b + i], s_m[j] = i; }
			n_lists += __popc(mk);
			n_a += __reduce_add_sync(FULL, kept ? m_n[b + i] : 0);
		}
		if (lane == 0) s_tot[0] = n_lists, s_tot[1] = 0, s_tot[2] = n_a;
	}
	__syncthreads();
	const int n_lists = s_tot[0], n_a = s_tot[2];
	// pass 1: strand class of every pop (kept in the two top bits of its word), number of forward-strand hits
	int my_for = 0, my_named = 0;
	for (int tt = tid; tt < n_a; tt += NT) {
		const uint32_t slot = P[ao + tt];
		int lo = 0, hi = n_lists - 1; // list of the slot
		while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if ((uint32_t)s_first[mid] <= slot) lo = mid; else hi = mid - 1; }
		const int m = s_m[lo];
		const uint64_t r = mmg_hit_pos(pos, m_n[b + m], m_val[b + m], slot - (uint32_t)s_first[lo]);
		const uint32_t qp = (uint32_t)mv[b + m].y;
		bool self;
		const int sk = mmg_skip_seed(MMG_NAMED_FLAG(kNamed, flag), r, qp, nfl, qlen, &self);
		const int cls = sk != MMG_SKIP_KEEP ? 0 : ((r & 1) == (qp & 1) ? 1 : 2);
		P[ao + tt] = slot | (uint32_t)cls << 30;
		my_for += cls == 1, my_named += sk == MMG_SKIP_NAME;
	}
	my_for = __reduce_add_sync(FULL, my_for);
	if (lane == 0 && my_for) atomicAdd(&s_tot[1], my_for);
	if (kNamed) {
		my_named = __reduce_add_sync(FULL, my_named);
		if (lane == 0 && my_named) atomicAdd(n_named, (unsigned long long)my_named);
	}
	__syncthreads();
	const int n_for = s_tot[1];
	// pass 2: anchors; forward hits in the low half of the packed scan value, reverse hits in the high half
	int run_for = 0, run_rev = 0;
	for (int t0 = 0; t0 < n_a; t0 += NT) {
		const int tt = t0 + tid;
		int cls = 0; uint32_t slot = 0;
		if (tt < n_a) { const uint32_t w = P[ao + tt]; cls = (int)(w >> 30), slot = w & 0x3fffffffu; }
		int tot;
		const int ex = block_excl_scan(cls == 1 ? 1 : cls == 2 ? 1 << 16 : 0, s_w, &tot);
		if (cls) {
			int lo = 0, hi = n_lists - 1;
			while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if ((uint32_t)s_first[mid] <= slot) lo = mid; else hi = mid - 1; }
			const int m = s_m[lo];
			const uint64_t r = mmg_hit_pos(pos, m_n[b + m], m_val[b + m], slot - (uint32_t)s_first[lo]);
			bool self;
			mmg_skip_seed(MMG_NAMED_FLAG(kNamed, flag), r, (uint32_t)mv[b + m].y, nfl, qlen, &self); // kept (pass 1); asked again for the self bit
			const mm128 an = mmg_make_anchor(r, mv[b + m], mmg_is_tandem(mv + b, n_mv, m), self, qlen);
			if (cls == 1) a[ao + run_for + (ex & 0xffff)] = an;
			else a[ao + n_for + run_rev + (ex >> 16)] = an;
		}
		run_for += tot & 0xffff, run_rev += tot >> 16;
	}
	if (tid == 0) { na[li] = run_for + run_rev; atomicAdd(n_pops, (unsigned long long)n_a); }
}

// mmg_fill_heap (mmg_core.h) for one fragment per warp: same pops in the same order; the heap and the next position of every
// list live in shared memory, and the position after that is fetched while the heap is sifted, so that the L2 latency of the
// position arrays is off the critical path of the serial replay (a repeat-family fragment makes ~2 x 10^5 pops).
template <bool kNamed>
__device__ int64_t fill_heap_prefetch(const mm128 *mv, const int32_t *m_n, const uint64_t *m_val, int n_mv, int max_occ, const uint64_t *pos,
                                      int64_t flag, const NameFilt &nf, int qlen, int64_t n_a_planned, mm128 *heap, uint64_t *nxt, mm128 *a,
                                      int64_t *n_named)
{
	size_t hs = 0;
	int64_t n_for = 0, n_rev = 0, n_a = n_a_planned, n_nm = 0;
	for (int i = 0; i < n_mv; ++i)
		if (m_n[i] > 0 && m_n[i] < max_occ) {
			heap[hs].x = mmg_hit_pos(pos, m_n[i], m_val[i], 0);
			heap[hs].y = (uint64_t)i << 32;
			nxt[i] = m_n[i] > 1 ? mmg_hit_pos(pos, m_n[i], m_val[i], 1) : 0;
			++hs;
		}
	if (hs > 1) for (int64_t j = (int64_t)(hs >> 1) - 1; j >= 0; --j) mmg_heap_down((size_t)j, hs, heap);
	while (hs > 0) {
		const int i = (int)(heap[0].y >> 32);
		const uint32_t off = (uint32_t)heap[0].y;
		const uint64_t r = heap[0].x;
		const int32_t n = m_n[i];
		const uint64_t val = m_val[i];
		const mm128 mz = mv[i];
		const bool more = off < (uint32_t)n - 1;
		const uint64_t pending = more && off + 2 < (uint32_t)n ? pos[val + off + 2] : 0; // needed two pops of this list from now
		if (more) { ++heap[0].y; heap[0].x = nxt[i]; }
		else { heap[0] = heap[hs - 1]; --hs; }
		if (hs > 0) mmg_heap_down(0, hs, heap);
		bool self;
		const int sk = mmg_skip_seed(MMG_NAMED_FLAG(kNamed, flag), r, (uint32_t)mz.y, nf, qlen, &self);
		if (sk == MMG_SKIP_KEEP) {
			const mm128 an = mmg_make_anchor(r, mz, mmg_is_tandem(mv, n_mv, i), self, qlen);
			if ((r & 1) == ((uint32_t)mz.y & 1)) a[n_for++] = an;
			else a[n_a - (++n_rev)] = an;
		} else n_nm += sk == MMG_SKIP_NAME;
		if (more) nxt[i] = pending;
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

// K2c, literal form: anchors in the reference's order (map.c:149-211) for the fragments the rank replay cannot take (replay[] == 2)
template <bool kNamed>
__global__ void k_fill(FragTab ft, const int32_t *__restrict__ list, int n_list, const mm128 *__restrict__ mv, const int32_t *__restrict__ m_n,
                       const uint64_t *__restrict__ m_val, const uint64_t *__restrict__ pos, int max_occ, int64_t flag,
                       const int64_t *__restrict__ aoff, int32_t *__restrict__ na, mm128 *__restrict__ a, mm128 *__restrict__ heap,
                       const uint8_t *__restrict__ replay, int per_warp, NameTabs nt, unsigned long long *__restrict__ n_named)
{
	// per_warp: one fragment per warp (lane 0 works).  The re-chain pass lists a few hundred fragments of ~10^5 anchors each; as
	// neighbouring threads of one warp their serial replays diverged and ran one after the other (36 ms for 192 fragments)
	const int gt = blockIdx.x * blockDim.x + threadIdx.x, li = per_warp ? gt >> 5 : gt;
	if (li >= n_list || (per_warp && (gt & 31))) return;
	if (replay[li] != 2) return;
	const int f = list ? list[li] : li;
	const int64_t b = ft.unit_off[ft.unit0[f]], e = ft.unit_off[ft.unit0[f + 1]];
	const int64_t ao = aoff[li];
	const NameFilt nf = name_filt(nt, f);
	int64_t n, nn;
	__shared__ mm128 s_heap[2][128];
	__shared__ uint64_t s_nxt[2][128];
	if (per_warp && e - b <= 128)
		n = fill_heap_prefetch<kNamed>(mv + b, m_n + b, m_val + b, (int)(e - b), max_occ, pos, flag, nf, ft.qlen[f], na[li], s_heap[threadIdx.x >> 5], s_nxt[threadIdx.x >> 5], a + ao, &nn);
	else n = mmg_fill_heap<kNamed>(mv + b, m_n + b, m_val + b, (int)(e - b), max_occ, pos, flag, nf, ft.qlen[f], na[li], heap + b, a + ao, &nn);
	na[li] = (int32_t)n;
	if (kNamed && nn) atomicAdd(n_named, (unsigned long long)nn);
}

struct ChainOptDev { int32_t bw, max_gap, max_gap_ref, max_frag_len, max_skip, max_iter, min_cnt, min_sc, is_cdna, is_sr; };

__device__ __forceinline__ ChainParams mmg_chain_params(const ChainOptDev &o, int qlen_sum, int n_segs)
{ // map.c:341-351
	ChainParams P;
	const int gap_qry = o.is_sr ? (qlen_sum > o.max_gap ? qlen_sum : o.max_gap) : o.max_gap;
	int gap_ref;
	if (o.max_gap_ref > 0) gap_ref = o.max_gap_ref;
	else if (o.max_frag_len > 0) { gap_ref = o.max_frag_len - qlen_sum; if (gap_ref < o.max_gap) gap_ref = o.max_gap; }
	else gap_ref = o.max_gap;
	P.max_dist_x = gap_ref, P.max_dist_y = gap_qry, P.bw = o.bw, P.max_skip = o.max_skip, P.max_iter = o.max_iter;
	P.min_cnt = o.min_cnt, P.min_sc = o.min_sc, P.is_cdna = o.is_cdna, P.n_segs = n_segs;
	return P;
}

// ---- K3, warp-cooperative form -------------------------------------------------------------------------
// mm_chain_dp's fill (chain.c:45-85) cannot look back further than max_dist_x on the reference, so the sorted anchor array
// of a fragment falls apart into independent SEGMENTS wherever a[i].x > a[i-1].x + max_dist_x (the `st` pointer of
// chain.c:51 would jump to i).  Segments are filled by one warp each; a fragment drawn from a 3 000-copy repeat becomes
// thousands of parallel work items instead of one 10^5-step serial loop.

// flag the first anchor of every segment; zero the t[] array of chain.c:39
__global__ void k_chain_heads(FragTab ft, const int32_t *__restrict__ list, int n_list, const int32_t *__restrict__ n_seg, ChainOptDev co,
                              const int64_t *__restrict__ aoff, const int32_t *__restrict__ na, const mm128 *__restrict__ a, int64_t n_total,
                              uint8_t *__restrict__ head, int32_t *__restrict__ work, int32_t *__restrict__ head_li)
{
	const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (g >= n_total) return;
	const int li = frag_of_anchor(aoff, n_list, g);
	const int64_t ao = aoff[li], i = g - ao, n = na[li];
	uint8_t h = 0;
	if (i < n) {
		const int f = list ? list[li] : li;
		const ChainParams P = mmg_chain_params(co, ft.qlen[f], n_seg[f]);
		h = (i == 0 || a[g].x > a[g - 1].x + (uint64_t)P.max_dist_x) ? 1 : 0;
		work[ao * 8 + 2 * n + i] = 0; // t[i]
		if (h) head_li[g] = li;       // the fill kernels find a segment's fragment here instead of bisecting aoff[] again
	}
	head[g] = h;
}

// avg_qspan = (float)sum_qspan / n per fragment (chain.c:41-42): one warp per fragment
__global__ void k_chain_avgspan(int n_list, const int64_t *__restrict__ aoff, const int32_t *__restrict__ na, const mm128 *__restrict__ a, float *__restrict__ avg)
{
	const int li = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
	if (li >= n_list) return;
	const int64_t ao = aoff[li]; const int n = na[li];
	unsigned long long sum = 0;
	for (int i = lane; i < n; i += 32) sum += a[ao + i].y >> 32 & 0xff;
	for (int d = 16; d >= 1; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
	if (lane == 0) avg[li] = n > 0 ? (float)sum / (float)(int64_t)n : 0.f;
}

// A segment's place: fragment slot, anchor range inside the fragment
struct SegPlace { int li, f, s, e, n; int64_t ao; };
__device__ __forceinline__ SegPlace seg_place(int sidx, int n_segments, const int64_t *__restrict__ seg_start, const int32_t *__restrict__ head_li,
                                              const int32_t *__restrict__ list, const int64_t *__restrict__ aoff, const int32_t *__restrict__ na)
{
	SegPlace sp;
	const int64_t g0 = seg_start[sidx];
	sp.li = head_li[g0];
	sp.f = list ? list[sp.li] : sp.li;
	sp.ao = aoff[sp.li], sp.n = na[sp.li];
	const int64_t frag_end = sp.ao + sp.n;
	int64_t g1 = frag_end;
	if (sidx + 1 < n_segments) { const int64_t nx = seg_start[sidx + 1]; if (nx < frag_end) g1 = nx; }
	sp.s = (int)(g0 - sp.ao), sp.e = (int)(g1 - sp.ao);
	return sp;
}

// one THREAD per short segment.  A read pair from a repeat family meets ~10^4 copies, each contributing a handful of
// anchors: 2 x 10^7 segments of ~6 anchors per 10^6 reads.  A warp per segment spent its time fetching the segment (a counter,
// a bisection, the parameters) and then used 3 of its 32 lanes; here every lane walks its own segment with the sequential
// loop of chain.c:45-85, and only the segments longer than CHAIN_SMALL_SEG are left, as a list, for the warp form below.
#define CHAIN_SMALL_SEG 24
__global__ void __launch_bounds__(128)
k_chain_fill_small(FragTab ft, const int32_t *__restrict__ list, const int32_t *__restrict__ n_seg, ChainOptDev co,
                   const int64_t *__restrict__ aoff, const int32_t *__restrict__ na, const mm128 *__restrict__ a, int32_t *__restrict__ work,
                   const float *__restrict__ avg, const int64_t *__restrict__ seg_start, const int32_t *__restrict__ head_li,
                   const int32_t *__restrict__ n_seg_total, int32_t *__restrict__ long_list, int32_t *__restrict__ n_long,
                   unsigned long long *__restrict__ iter_total)
{
	const int n_segments = *n_seg_total;
	unsigned long long iters = 0;
	for (int sidx = blockIdx.x * blockDim.x + threadIdx.x; sidx < n_segments; sidx += gridDim.x * blockDim.x) {
		const SegPlace sp = seg_place(sidx, n_segments, seg_start, head_li, list, aoff, na);
		if (sp.e - sp.s > CHAIN_SMALL_SEG) { long_list[atomicAdd(n_long, 1)] = sidx; continue; }
		const ChainParams P = mmg_chain_params(co, ft.qlen[sp.f], n_seg[sp.f]);
		const float avg_qspan = avg[sp.li];
		const mm128 *A = a + sp.ao;
		int32_t *F = work + sp.ao * 8, *Pp = F + sp.n, *T = Pp + sp.n, *V = T + sp.n;
		int st = sp.s;
		for (int i = sp.s; i < sp.e; ++i) {
			const mm128 ai = A[i];
			const uint64_t ri = ai.x;
			const int32_t qi = (int32_t)ai.y, q_span = (int32_t)(ai.y >> 32 & 0xff);
			const int32_t sidi = (int32_t)((ai.y & MMG_SEED_SEG_MASK) >> MMG_SEED_SEG_SHIFT);
			int32_t max_f = q_span, max_j = -1, n_skip = 0;
			while (st < i && ri > A[st].x + (uint64_t)P.max_dist_x) ++st;
			if (i - st > P.max_iter) st = i - P.max_iter;
			for (int j = i - 1; j >= st; --j) {
				int32_t sc;
				++iters;
				if (!mmg_chain_score(P, ri, qi, q_span, sidi, A[j], avg_qspan, &sc)) continue;
				sc += F[j];
				if (sc > max_f) {
					max_f = sc, max_j = j;
					if (n_skip > 0) --n_skip;
				} else if (T[j] == i) {
					if (++n_skip > P.max_skip) break;
				}
				const int pj = Pp[j];
				if (pj >= 0) T[pj] = i;
			}
			F[i] = max_f, Pp[i] = max_j;
			V[i] = (max_j >= 0 && V[max_j] > max_f) ? V[max_j] : max_f; // chain.c:84
		}
	}
	for (int d = 16; d >= 1; d >>= 1) iters += __shfl_xor_sync(0xffffffffu, iters, d);
	if ((threadIdx.x & 31) == 0 && iters) atomicAdd(iter_total, iters);
}

// one warp per segment: lanes evaluate 32 predecessors at a time; the order-dependent parts of the inner loop
// (strict-max winner, n_skip counter, early break, t[] marks; chain.c:53-82) are resolved from ballots so that the
// result is the sequential one (SURVEY.md H3)
__global__ void __launch_bounds__(128)
k_chain_fill(FragTab ft, const int32_t *__restrict__ list, int n_list, const int32_t *__restrict__ n_seg, ChainOptDev co,
             const int64_t *__restrict__ aoff, const int32_t *__restrict__ na, const mm128 *__restrict__ a, int32_t *__restrict__ work,
             const float *__restrict__ avg, const int64_t *__restrict__ seg_start, const int32_t *__restrict__ head_li,
             const int32_t *__restrict__ n_seg_total, const int32_t *__restrict__ long_list, const int32_t *__restrict__ n_long,
             int32_t *__restrict__ next_seg, unsigned long long *__restrict__ iter_total)
{
	const int lane = threadIdx.x & 31;
	const int n_segments = *n_seg_total, n_work = *n_long;
	unsigned long long iters = 0;
	for (;;) {
		int w = 0;
		if (lane == 0) w = atomicAdd(next_seg, 1);
		w = __shfl_sync(0xffffffffu, w, 0);
		if (w >= n_work) break;
		const SegPlace sp = seg_place(long_list[w], n_segments, seg_start, head_li, list, aoff, na);
		const int n = sp.n, s = sp.s, e = sp.e;
		const ChainParams P = mmg_chain_params(co, ft.qlen[sp.f], n_seg[sp.f]);
		const float avg_qspan = avg[sp.li];
		const mm128 *A = a + sp.ao;
		int32_t *F = work + sp.ao * 8, *Pp = F + n, *T = Pp + n, *V = T + n;
		int st = s;
		for (int i = s; i < e; ++i) {
			const mm128 ai = A[i];
			const uint64_t ri = ai.x;
			const int32_t qi = (int32_t)ai.y, q_span = (int32_t)(ai.y >> 32 & 0xff);
			const int32_t sidi = (int32_t)((ai.y & MMG_SEED_SEG_MASK) >> MMG_SEED_SEG_SHIFT);
			int32_t max_f = q_span, max_j = -1, n_skip = 0;
			while (st < i && ri > A[st].x + (uint64_t)P.max_dist_x) ++st;
			if (i - st > P.max_iter) st = i - P.max_iter;
			bool done = false;
			if (i - st <= P.max_skip && i - st <= 32) {
				// Short window: the skip counter (chain.c:76-80) needs more than max_skip marked predecessors to stop the scan, so it
				// cannot fire, and the t[] marks it reads are private to this i.  What is left is "best score, first one met wins ties",
				// i.e. the largest j: one warp-wide max over score * 32 + (31 - lane).
				const int j = i - 1 - lane;
				int32_t sc = 0;
				bool valid = j >= st;
				if (valid) { valid = mmg_chain_score(P, ri, qi, q_span, sidi, A[j], avg_qspan, &sc); if (valid) sc += F[j]; }
				const int key = valid && sc > max_f ? sc * 32 + (31 - lane) : INT32_MIN;
				const int best = __reduce_max_sync(0xffffffffu, key);
				if (best != INT32_MIN) { const int bl = 31 - (best & 31); max_f = (best - (best & 31)) / 32, max_j = i - 1 - bl; }
				iters += (unsigned)(i - st);
				done = true;
			}
			for (int jhi = i - 1; jhi >= st && !done; jhi -= 32) {
				const int j = jhi - lane;
				bool valid = j >= st;
				int32_t sc = 0, pj = -1;
				if (valid) {
					const mm128 aj = A[j];
					valid = mmg_chain_score(P, ri, qi, q_span, sidi, aj, avg_qspan, &sc);
					if (valid) { sc += F[j]; pj = Pp[j]; if (pj >= 0) T[pj] = i; }
				}
				__syncwarp();
				const bool tmark = valid && T[j] == i;
				int32_t incl = valid ? sc : INT32_MIN; // running max over lanes 0..lane = predecessors visited so far
#pragma unroll
				for (int d = 1; d < 32; d <<= 1) { const int32_t o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d && o > incl) incl = o; }
				int32_t excl = __shfl_up_sync(0xffffffffu, incl, 1);
				excl = (lane == 0 || excl < max_f) ? max_f : excl; // best score before this lane, counting what earlier chunks found
				const bool win = valid && sc > excl;
				const unsigned wmask = __ballot_sync(0xffffffffu, win), mmask = __ballot_sync(0xffffffffu, tmark && !win);
				unsigned ev = wmask | mmask;
				int brk = -1;
				while (ev) {
					const int b = __ffs((int)ev) - 1;
					ev &= ev - 1;
					if (wmask >> b & 1) { if (n_skip > 0) --n_skip; }
					else if (++n_skip > P.max_skip) { brk = b; break; }
				}
				const unsigned lim = brk >= 0 ? (brk == 31 ? 0xffffffffu : ((2u << brk) - 1u)) : 0xffffffffu;
				const unsigned w2 = wmask & lim;
				if (w2) { const int last = 31 - __clz((int)w2); max_f = __shfl_sync(0xffffffffu, sc, last); max_j = jhi - last; }
				if (brk >= 0) { done = true; iters += (unsigned)(brk + 1); }
				else iters += (unsigned)((jhi - st + 1) < 32 ? (jhi - st + 1) : 32);
			}
			if (lane == 0) {
				F[i] = max_f, Pp[i] = max_j;
				V[i] = (max_j >= 0 && V[max_j] > max_f) ? V[max_j] : max_f; // chain.c:84
			}
			__syncwarp();
		}
	}
	if (lane == 0 && iters) atomicAdd(iter_total, iters);
}

// Warp-cooperative bitonic sort of a[0,n) in global/shared memory for ANY n: every compare-exchange is oriented the same
// way (the first step of each merge mirrors the block, partner = i ^ (k-1)), so the virtual elements beyond n act as
// "already last" padding and are never touched.  before(x, y) = x must precede y.
template <class T, class Before>
__device__ __forceinline__ void warp_bitonic(T *a, int n, int lane, Before before)
{
	int N = 2; while (N < n) N <<= 1;
	for (int k = 2; k <= N; k <<= 1) {
		for (int i = lane; i < n; i += 32) {
			const int l = i ^ (k - 1);
			if (l > i && l < n) { const T x = a[i], y = a[l]; if (before(y, x)) a[i] = y, a[l] = x; }
		}
		__syncwarp();
		for (int j = k >> 2; j > 0; j >>= 1) {
			for (int i = lane; i < n; i += 32) {
				const int l = i ^ j;
				if (l > i && l < n) { const T x = a[i], y = a[l]; if (before(y, x)) a[i] = y, a[l] = x; }
			}
			__syncwarp();
		}
	}
}
struct U64Desc { __device__ bool operator()(uint64_t x, uint64_t y) const { return x > y; } };
struct M128ByX { __device__ bool operator()(const mm128 &x, const mm128 &y) const { return x.x < y.x; } };

// does the fragment go through the second pass with the higher occurrence cut-off? (map.c:353-370)
__device__ __forceinline__ uint8_t chain_wants_rechain(bool candidate, int n_u, const uint64_t *U0, const mm128 *A, int segs)
{
	if (!candidate) return 0;
	if (n_u == 0) return 1;
	int n_chained = 1, max = 0, max_i = -1, max_off = -1, off = 0; // does the best chain span every segment? (map.c:355-365)
	for (int i = 0; i < n_u; ++i) {
		if (max < (int)(U0[i] >> 32)) max = (int)(U0[i] >> 32), max_i = i, max_off = off;
		off += (int32_t)U0[i];
	}
	if (max_i >= 0)
		for (int i = 1; i < (int32_t)U0[max_i]; ++i)
			if ((A[max_off + i].y & MMG_SEED_SEG_MASK) != (A[max_off + i - 1].y & MMG_SEED_SEG_MASK)) ++n_chained;
	return n_chained < segs ? 1 : 0;
}

// the fragments the CTA form of the tail takes (more than heavy_n anchors): counted here; listed by the descending sort of
// (anchors, slot) that follows, so that the CTAs, which pull their work from a counter, start with the largest fragments
__global__ void k_tail_heavy_list(int n_list, const int32_t *__restrict__ na, int heavy_n, uint32_t *__restrict__ key, int32_t *__restrict__ val, int32_t *__restrict__ n_heavy)
{
	const int li = blockIdx.x * blockDim.x + threadIdx.x;
	if (li >= n_list) return;
	const int n = na[li];
	key[li] = (uint32_t)(n > 0 ? n : 0), val[li] = li;
	if (n > heavy_n) atomicAdd(n_heavy, 1);
}

// K3 tail, one warp per fragment: chain ends and peaks, ranking by peak score, backtracking, output order
// (chain.c:87-160).  The sequential backtrack marks anchors as used chain by chain in rank order; the same
// ownership is obtained in parallel as "the lowest rank whose path passes through the anchor" (atomicMin while
// walking), after which every chain counts the anchors it owns.  Work arrays: f|p|t|v (4n int32) followed by room
// for the chain-order array w (n mm128); u has 2n entries; b has n.
__global__ void __launch_bounds__(128)
k_chain_tail_warp(FragTab ft, const int32_t *__restrict__ list, int n_list, const int32_t *__restrict__ n_seg, ChainOptDev co,
                  const int64_t *__restrict__ aoff, const int32_t *__restrict__ na, mm128 *__restrict__ a, int32_t *__restrict__ work,
                  uint64_t *__restrict__ u, mm128 *__restrict__ bb, RsFrame *__restrict__ stack, int32_t *__restrict__ nu_out,
                  int32_t *__restrict__ nv_out, const int32_t *__restrict__ rep, int rechain_enabled, uint8_t *__restrict__ flag_out, int heavy_n)
{
	const int li = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
	if (li >= n_list) return;
	const unsigned FULL = 0xffffffffu;
	const int f = list ? list[li] : li;
	const int64_t ao = aoff[li];
	const int n = na[li], segs = n_seg[f];
	if (n > heavy_n) return; // left to k_chain_tail_block: thousands of chains ranked and walked by 32 lanes held the launch
	int n_u = 0, n_v = 0;
	mm128 *A = a + ao, *B = bb + ao;
	uint64_t *U0 = u + ao * 2, *U1 = U0 + n;
	if (n > 0) {
		const ChainParams P = mmg_chain_params(co, ft.qlen[f], segs);
		int32_t *F = work + ao * 8, *Pp = F + n, *T = Pp + n, *V = T + n;
		mm128 *W = reinterpret_cast<mm128*>(F + 4 * (int64_t)n);
		// 1. chain ends: anchors nobody extends (chain.c:88-90)
		for (int i = lane; i < n; i += 32) T[i] = 0;
		__syncwarp();
		for (int i = lane; i < n; i += 32) { const int pj = Pp[i]; if (pj >= 0) T[pj] = 1; }
		__syncwarp();
		// 2. for every end with a good enough peak, the anchor where the score peaks (chain.c:99-106)
		for (int i0 = 0; i0 < n; i0 += 32) {
			const int i = i0 + lane;
			const bool is_end = i < n && T[i] == 0 && V[i] >= P.min_sc;
			uint64_t val = 0;
			if (is_end) {
				int j = i;
				while (j >= 0 && F[j] < V[j]) j = Pp[j];
				if (j < 0) j = i;
				val = (uint64_t)F[j] << 32 | (uint32_t)j;
			}
			const unsigned m = __ballot_sync(FULL, is_end);
			if (is_end) U1[n_u + __popc(m & ((1u << lane) - 1u))] = val;
			n_u += __popc(m);
		}
		__syncwarp();
		if (n_u > 0) {
			// 3. rank by (peak score, anchor) descending (chain.c:107-111); equal values are duplicates
			if (n_u <= 64) {
				for (int e = lane; e < n_u; e += 32) {
					const uint64_t x = U1[e];
					int r = 0;
					for (int k = 0; k < n_u; ++k) { const uint64_t y = U1[k]; r += (y > x || (y == x && k < e)) ? 1 : 0; }
					U0[r] = x;
				}
			} else {
				warp_bitonic(U1, n_u, lane, U64Desc());
				for (int e = lane; e < n_u; e += 32) U0[e] = U1[e];
			}
			// 4. ownership: lowest rank whose walk passes through the anchor
			for (int i = lane; i < n; i += 32) T[i] = 0x7fffffff;
			__syncwarp();
			for (int k = lane; k < n_u; k += 32) {
				int j = (int32_t)U0[k];
				while (j >= 0) { const int old = atomicMin(&T[j], k); if (old < k) break; j = Pp[j]; }
			}
			__syncwarp();
			// 5. what each chain keeps (chain.c:115-129): its peak, then the anchors it owns; V[k] = kept count or 0
			for (int k = lane; k < n_u; k += 32) {
				const int j0 = (int32_t)U0[k];
				const int32_t sc = (int32_t)(U0[k] >> 32);
				int cnt = 1, j = Pp[j0];
				while (j >= 0 && T[j] == k) ++cnt, j = Pp[j];
				bool keep; int32_t score;
				if (j < 0) keep = cnt >= P.min_cnt, score = sc;
				else keep = (sc - F[j] >= P.min_sc) && cnt >= P.min_cnt, score = sc - F[j];
				U1[k] = keep ? ((uint64_t)(uint32_t)score << 32 | (uint32_t)cnt) : 0; // per rank; compacted below
			}
			__syncwarp();
			// 6. kept chains in rank order -> b[] (anchors ascending inside a chain), compacted u, chain-order keys w
			int n_keep = 0;
			for (int k0 = 0; k0 < n_u; k0 += 32) {
				const int k = k0 + lane;
				const uint64_t uk = k < n_u ? U1[k] : 0;
				const int cnt = (int32_t)(uint32_t)uk;
				int incl = cnt;
#pragma unroll
				for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += o; }
				const unsigned m = __ballot_sync(FULL, cnt > 0);
				if (cnt > 0) {
					const int off = n_v + incl - cnt, kk = n_keep + __popc(m & ((1u << lane) - 1u));
					int j = (int32_t)U0[k];
					for (int q = cnt - 1; q >= 0; --q) { B[off + q] = A[j]; j = Pp[j]; }
					V[kk] = off; // start of chain kk in b[]
					W[kk].y = (uint64_t)off << 32 | (uint32_t)kk;
				}
				__syncwarp();
				if (cnt > 0) U1[n_keep + __popc(m & ((1u << lane) - 1u))] = uk; // compaction never overtakes unread entries: kk <= k
				n_v += __shfl_sync(FULL, incl, 31);
				n_keep += __popc(m);
				__syncwarp();
			}
			n_u = n_keep;
			for (int kk = lane; kk < n_u; kk += 32) W[kk].x = B[V[kk]].x;
			__syncwarp();
			// 7. order chains by the position of their first anchor, klib radix semantics (chain.c:150)
			// With distinct keys the sorted order is unique, so a parallel sort gives klib's result; only equal keys (two chains
			// starting on anchors with the same reference position) need the in-place MSD radix sort replayed literally.
			if (n_u <= 64) {
				if (lane == 0) mmg_rs_sort_exact(W, (int64_t)n_u, stack + ao / 65 + 2 * (int64_t)li, KeyX());
			} else {
				warp_bitonic(W, n_u, lane, M128ByX());
				bool tie = false;
				for (int kk = lane + 1; kk < n_u; kk += 32) tie |= W[kk].x == W[kk - 1].x;
				if (__any_sync(FULL, tie)) {
					for (int kk = lane; kk < n_u; kk += 32) { const int off = V[kk]; W[kk].x = B[off].x; W[kk].y = (uint64_t)off << 32 | (uint32_t)kk; }
					__syncwarp();
					if (lane == 0) mmg_rs_sort_exact(W, (int64_t)n_u, stack + ao / 65 + 2 * (int64_t)li, KeyX());
				}
			}
			__syncwarp();
			// 8. write chains back to a[] in that order (chain.c:152-159): 32 chains at a time, offsets from a warp scan
			int dst = 0;
			for (int i0 = 0; i0 < n_u; i0 += 32) {
				const int i = i0 + lane;
				uint64_t uk = 0; int src = 0;
				if (i < n_u) { const uint64_t wy = W[i].y; uk = U1[(int32_t)(uint32_t)wy]; src = (int)(wy >> 32); }
				const int nn = (int32_t)(uint32_t)uk;
				int incl = nn;
#pragma unroll
				for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += o; }
				const int off = dst + incl - nn;
				for (int q = 0; q < nn; ++q) A[off + q] = B[src + q];
				dst += __shfl_sync(FULL, incl, 31);
				__syncwarp();
				if (i < n_u) U0[i] = uk; // U1 = U0 + n: the compacted values are not overwritten
			}
			__syncwarp();
		}
	}
	if (lane != 0) return;
	nu_out[li] = n_u, nv_out[li] = n_v;
	if (flag_out) flag_out[f] = chain_wants_rechain(rechain_enabled && rep[li] > 0, n_u, U0, A, segs);
}


// ---- K3 tail, one CTA per fragment: the same steps for the re-chain pass, whose few fragments carry ~10^5 anchors and
// thousands of chains each.  One warp per fragment spent 10 ms per launch at 4 % issue utilisation on dependent walks; 256
// threads walk eight times as many chains at once.  Orders that the warp form derives from ballots come from block scans.
template <class T, class Before>
__device__ __forceinline__ void block_bitonic(T *a, int n, Before before)
{
	const int tid = threadIdx.x, nt = blockDim.x;
	int N = 2; while (N < n) N <<= 1;
	for (int k = 2; k <= N; k <<= 1) {
		for (int i = tid; i < n; i += nt) {
			const int l = i ^ (k - 1);
			if (l > i && l < n) { const T x = a[i], y = a[l]; if (before(y, x)) a[i] = y, a[l] = x; }
		}
		__syncthreads();
		for (int j = k >> 2; j > 0; j >>= 1) {
			for (int i = tid; i < n; i += nt) {
				const int l = i ^ j;
				if (l > i && l < n) { const T x = a[i], y = a[l]; if (before(y, x)) a[i] = y, a[l] = x; }
			}
			__syncthreads();
		}
	}
}

// the same sort on a copy in shared memory when it fits: every one of the log^2 n stages of the network is then a round of
// shared-memory accesses instead of a trip to L2 (a re-chained repeat-family fragment ranks ~10^4 chain ends)
template <class T, class Before>
__device__ __forceinline__ void block_bitonic_staged(T *a, int n, Before before, unsigned char *smem, size_t smem_bytes)
{
	if ((size_t)n * sizeof(T) > smem_bytes) { block_bitonic(a, n, before); return; }
	T *sa = reinterpret_cast<T*>(smem);
	for (int i = threadIdx.x; i < n; i += blockDim.x) sa[i] = a[i];
	__syncthreads();
	block_bitonic(sa, n, before);
	for (int i = threadIdx.x; i < n; i += blockDim.x) a[i] = sa[i];
	__syncthreads();
}

__device__ __forceinline__ int block_incl_scan(int v, int *s, int *total)
{ // every thread of the CTA calls; blockDim.x <= 1024
	const int tid = threadIdx.x, nt = blockDim.x;
	s[tid] = v;
	__syncthreads();
	for (int d = 1; d < nt; d <<= 1) { const int o = tid >= d ? s[tid - d] : 0; __syncthreads(); s[tid] += o; __syncthreads(); }
	const int r = s[tid];
	*total = s[nt - 1];
	__syncthreads();
	return r;
}

#define TAIL_BLOCK_SMEM (216 * 1024)
#define TAIL_HEAVY_N 2048               /* first-pass fragments with more anchors go to the CTA form */
#define TAIL_HEAVY_SMEM (64 * 1024)     /* staging area of the CTA form in the first pass: three CTAs of 512 threads per SM */
__global__ void __launch_bounds__(1024)
k_chain_tail_block(FragTab ft, const int32_t *__restrict__ list, int n_list, const int32_t *__restrict__ n_seg, ChainOptDev co,
                   const int64_t *__restrict__ aoff, const int32_t *__restrict__ na, mm128 *__restrict__ a, int32_t *__restrict__ work,
                   uint64_t *__restrict__ u, mm128 *__restrict__ bb, RsFrame *__restrict__ stack, int32_t *__restrict__ nu_out,
                   int32_t *__restrict__ nv_out, const int32_t *__restrict__ heavy /* slots by descending anchor count */,
                   int32_t *__restrict__ n_heavy /* [0] how many of them this kernel takes, [1] the next one to hand out */, size_t smem_cap,
                   const int32_t *__restrict__ rep, int rechain_enabled, uint8_t *__restrict__ flag_out /* first pass only */,
                   int walk /* 1: walk every chain, the form before the level-by-level one (MMG_TAIL_WALK=1) */)
{
	__shared__ int s_scan[1024], s_nu, s_tie, s_it;
	extern __shared__ __align__(16) unsigned char dyn_tail[];
	const int tid = threadIdx.x, NT = blockDim.x;
	const int n_items = n_heavy[0];
	for (;;) { // largest fragments first, whichever CTA is free takes the next one
	if (tid == 0) s_it = atomicAdd(n_heavy + 1, 1);
	__syncthreads();
	const int it = s_it;
	if (it >= n_items) break;
	const int li = heavy[it];
	const int f = list ? list[li] : li;
	const int64_t ao = aoff[li];
	const int n = na[li], segs = n_seg[f];
	int n_u = 0, n_v = 0;
	mm128 *A = a + ao, *B = bb + ao;
	uint64_t *U0 = u + ao * 2, *U1 = U0 + n;
	if (n > 0) {
		const ChainParams P = mmg_chain_params(co, ft.qlen[f], segs);
		int32_t *F = work + ao * 8, *Pp = F + n, *T = Pp + n, *V = T + n;
		mm128 *W = reinterpret_cast<mm128*>(F + 4 * (int64_t)n);
		if (tid == 0) s_nu = 0, s_tie = 0;
		// 1. chain ends (chain.c:88-90)
		for (int i = tid; i < n; i += NT) T[i] = 0;
		__syncthreads();
		for (int i = tid; i < n; i += NT) { const int pj = Pp[i]; if (pj >= 0) T[pj] = 1; }
		__syncthreads();
		// 2. peaks of the ends that score enough (chain.c:99-106); their order does not matter, they are sorted next
		for (int i = tid; i < n; i += NT)
			if (T[i] == 0 && V[i] >= P.min_sc) {
				int j = i;
				while (j >= 0 && F[j] < V[j]) j = Pp[j];
				if (j < 0) j = i;
				U1[atomicAdd(&s_nu, 1)] = (uint64_t)F[j] << 32 | (uint32_t)j;
			}
		__syncthreads();
		n_u = s_nu;
		if (n_u > 0) {
			// 3. rank by (peak score, anchor) descending (chain.c:107-111)
			block_bitonic_staged(U1, n_u, U64Desc(), dyn_tail, smem_cap);
			for (int e = tid; e < n_u; e += NT) U0[e] = U1[e];
			// The backtracking of chain.c:112-129 walks every chain from its peak towards its root, best chain first, and stops at the
			// first anchor a better chain took.  Walked literally that is a dependent load per step (two thirds of this kernel's time
			// on a fragment whose state does not fit L2).  The same result without walking: with depth[] (distance to the root, by
			// pointer jumping) an anchor's owner is the lowest rank among the peaks in its subtree -- pushed up level by level, one
			// fire-and-forget atomic per anchor -- a chain keeps exactly the anchors it owns (they are consecutive on its path), and an
			// owned anchor's slot in b[] follows from the two depths.
			int n_keep = 0;
			bool par = P.min_cnt >= 2 && !walk;
			int maxd = 0;
			if (par) {
				unsigned long long *P2 = reinterpret_cast<unsigned long long*>(W); // (jump << 32 | distance) per anchor
				for (int x = tid; x < n; x += NT) { const int pj = Pp[x]; P2[x] = pj >= 0 ? ((unsigned long long)(uint32_t)pj << 32 | 1ull) : (0xffffffffull << 32); }
				__syncthreads();
				for (;;) {
					int any = 0;
					for (int x = tid; x < n; x += NT) {
						const unsigned long long w = P2[x];
						const int j = (int32_t)(w >> 32);
						if (j >= 0) {
							const unsigned long long w2 = P2[j]; // an 8-byte word read at once: some valid (ancestor, distance) pair of j, whatever round it is from
							P2[x] = (w2 & 0xffffffff00000000ull) | (unsigned long long)((uint32_t)w + (uint32_t)w2);
							any |= (int32_t)(w2 >> 32) >= 0;
						}
					}
					if (!__syncthreads_or(any)) break;
				}
				if (tid == 0) s_tie = 0; // borrowed as the maximum depth until step 7 resets it
				__syncthreads();
				int md = 0;
				for (int x = tid; x < n; x += NT) { const int d = (int32_t)(uint32_t)P2[x]; V[x] = d; md = md > d ? md : d; }
				md = __reduce_max_sync(0xffffffffu, md);
				if ((tid & 31) == 0) atomicMax(&s_tie, md);
				__syncthreads();
				maxd = s_tie;
				__syncthreads();
				if (tid == 0) s_tie = 0;
				par = (size_t)(maxd + 2) * 8 <= smem_cap;
			}
			if (par) {
				int32_t *lvl_start = reinterpret_cast<int32_t*>(dyn_tail), *lvl_cur = lvl_start + maxd + 2; // anchors grouped by depth
				int32_t *order = reinterpret_cast<int32_t*>(W), *cntk = order + n, *lastk = cntk + n;
				for (int d = tid; d < maxd + 2; d += NT) lvl_start[d] = 0;
				__syncthreads();
				for (int x = tid; x < n; x += NT) atomicAdd(&lvl_start[V[x] + 1], 1);
				__syncthreads();
				if (tid == 0) { int acc = 0; for (int d = 0; d < maxd + 2; ++d) { acc += lvl_start[d]; lvl_start[d] = acc; lvl_cur[d] = acc; } }
				__syncthreads(); // lvl_start[d] = first slot of depth d; lvl_start[maxd + 1] = n
				for (int x = tid; x < n; x += NT) { order[atomicAdd(&lvl_cur[V[x]], 1)] = x; T[x] = 0x7fffffff; }
				for (int k = tid; k < n_u; k += NT) cntk[k] = 0;
				__syncthreads();
				for (int k = tid; k < n_u; k += NT) atomicMin(&T[(int32_t)U0[k]], k);
				__syncthreads();
				for (int d = maxd; d >= 1; --d) { // owners move up one level per step
					for (int i = lvl_start[d] + tid; i < lvl_start[d + 1]; i += NT) {
						const int x = order[i], t = T[x];
						if (t != 0x7fffffff) atomicMin(&T[Pp[x]], t);
					}
					__syncthreads();
				}
				// 5. what each chain keeps (chain.c:115-129): its peak, then the anchors it owns
				for (int x = tid; x < n; x += NT) {
					const int k = T[x];
					if (k != 0x7fffffff) {
						atomicAdd(&cntk[k], 1);
						const int pj = Pp[x];
						if (pj < 0 || T[pj] != k) lastk[k] = x; // the owned anchor closest to the root: one per chain
					}
				}
				__syncthreads();
				for (int k = tid; k < n_u; k += NT) {
					const int j0 = (int32_t)U0[k];
					const int32_t sc = (int32_t)(U0[k] >> 32);
					int cnt, j;
					if (T[j0] == k) cnt = cntk[k], j = Pp[lastk[k]];
					else cnt = 1, j = Pp[j0]; // the peak belongs to a better chain: it is still taken (the do-while of chain.c:118-122), nothing else
					bool keep; int32_t score;
					if (j < 0) keep = cnt >= P.min_cnt, score = sc;
					else keep = (sc - F[j] >= P.min_sc) && cnt >= P.min_cnt, score = sc - F[j];
					U1[k] = keep ? ((uint64_t)(uint32_t)score << 32 | (uint32_t)cnt) : 0;
				}
				__syncthreads();
				// 6. kept chains in rank order -> b[]: offsets by a scan over the ranks (F and Pp are free from here: F[k] = first slot of
				// chain k in b[], Pp[k] = its index among the kept chains), then every owned anchor goes to its slot
				for (int k0 = 0; k0 < n_u; k0 += NT) {
					const int k = k0 + tid;
					const int cnt = k < n_u ? (int32_t)(uint32_t)U1[k] : 0;
					int tot_cnt, tot_keep;
					const int incl = block_incl_scan(cnt, s_scan, &tot_cnt), inclk = block_incl_scan(cnt > 0 ? 1 : 0, s_scan, &tot_keep);
					if (cnt > 0) F[k] = n_v + incl - cnt, Pp[k] = n_keep + inclk - 1;
					n_v += tot_cnt, n_keep += tot_keep;
				}
				__syncthreads();
				int32_t *cid = reinterpret_cast<int32_t*>(W) + 2 * (int64_t)n; // rank of the chain that owns b[t]; the kept chains' W entries end below it (>= 2 anchors each)
				for (int x = tid; x < n; x += NT) {
					const int k = T[x];
					if (k == 0x7fffffff) continue;
					const int cnt = (int32_t)(uint32_t)U1[k];
					if (cnt == 0) continue;
					const int slot = F[k] + cnt - 1 - (V[(int32_t)U0[k]] - V[x]);
					B[slot] = A[x], cid[slot] = k;
				}
				__syncthreads();
				for (int k0 = 0; k0 < n_u; k0 += NT) { // per kept chain: start in b[], chain-order key, compacted u
					const int k = k0 + tid;
					const uint64_t uk = k < n_u ? U1[k] : 0;
					const int cnt = (int32_t)(uint32_t)uk;
					int kk = 0;
					if (cnt > 0) {
						kk = Pp[k];
						const int off = F[k];
						V[kk] = off;
						W[kk].y = (uint64_t)off << 32 | (uint32_t)kk;
					}
					__syncthreads();
					if (cnt > 0) U1[kk] = uk; // kk <= k, and every entry of this block of ranks was read above
					__syncthreads();
				}
			} else {
				// 4. ownership: lowest rank whose walk passes through the anchor
				for (int i = tid; i < n; i += NT) T[i] = 0x7fffffff;
				__syncthreads();
				for (int k = tid; k < n_u; k += NT) {
					int j = (int32_t)U0[k];
					while (j >= 0) { const int old = atomicMin(&T[j], k); if (old < k) break; j = Pp[j]; }
				}
				__syncthreads();
				// 5. what each chain keeps (chain.c:115-129)
				for (int k = tid; k < n_u; k += NT) {
					const int j0 = (int32_t)U0[k];
					const int32_t sc = (int32_t)(U0[k] >> 32);
					int cnt = 1, j = Pp[j0];
					while (j >= 0 && T[j] == k) ++cnt, j = Pp[j];
					bool keep; int32_t score;
					if (j < 0) keep = cnt >= P.min_cnt, score = sc;
					else keep = (sc - F[j] >= P.min_sc) && cnt >= P.min_cnt, score = sc - F[j];
					U1[k] = keep ? ((uint64_t)(uint32_t)score << 32 | (uint32_t)cnt) : 0;
				}
				__syncthreads();
				// 6. kept chains in rank order -> b[], compacted u, chain-order keys w
				for (int k0 = 0; k0 < n_u; k0 += NT) {
					const int k = k0 + tid;
					const uint64_t uk = k < n_u ? U1[k] : 0;
					const int cnt = (int32_t)(uint32_t)uk;
					int tot_cnt, tot_keep;
					const int incl = block_incl_scan(cnt, s_scan, &tot_cnt), inclk = block_incl_scan(cnt > 0 ? 1 : 0, s_scan, &tot_keep);
					const int kk = n_keep + inclk - 1;
					if (cnt > 0) {
						const int off = n_v + incl - cnt;
						int j = (int32_t)U0[k];
						for (int q = cnt - 1; q >= 0; --q) { B[off + q] = A[j]; j = Pp[j]; }
						V[kk] = off;
						W[kk].y = (uint64_t)off << 32 | (uint32_t)kk;
					}
					__syncthreads();
					if (cnt > 0) U1[kk] = uk; // kk <= k, and every entry of this block of ranks was read above
					n_v += tot_cnt, n_keep += tot_keep;
					__syncthreads();
				}
			}
			n_u = n_keep;
			for (int kk = tid; kk < n_u; kk += NT) W[kk].x = B[V[kk]].x;
			__syncthreads();
			// 7. order chains by the position of their first anchor (chain.c:150): unique for distinct keys, literal replay otherwise
			if (n_u > 64) {
				block_bitonic_staged(W, n_u, M128ByX(), dyn_tail, smem_cap);
				for (int kk = tid + 1; kk < n_u; kk += NT) if (W[kk].x == W[kk - 1].x) s_tie = 1;
				__syncthreads();
				if (s_tie) { // back to the order klib's sort starts from
					for (int kk = tid; kk < n_u; kk += NT) { const int off = V[kk]; W[kk].x = B[off].x; W[kk].y = (uint64_t)off << 32 | (uint32_t)kk; }
					__syncthreads();
				}
			}
			if (n_u <= 64 || s_tie) {
				// the literal replay is one thread's work; on a copy in shared memory its element moves cost tens of cycles instead of
				// a trip to L2 each (a fragment from a repeat family has thousands of chains, and ties are common there: two query
				// minimizers with the same hash start chains on the same reference position)
				const size_t frames = (size_t)n_u / 65 + 4;
				if ((size_t)n_u * sizeof(mm128) + frames * sizeof(RsFrame) <= smem_cap) {
					mm128 *sw = reinterpret_cast<mm128*>(dyn_tail);
					RsFrame *sf = reinterpret_cast<RsFrame*>(dyn_tail + (size_t)n_u * sizeof(mm128));
					for (int kk = tid; kk < n_u; kk += NT) sw[kk] = W[kk];
					__syncthreads();
					if (tid == 0) mmg_rs_sort_exact(sw, (int64_t)n_u, sf, KeyX());
					__syncthreads();
					for (int kk = tid; kk < n_u; kk += NT) W[kk] = sw[kk];
				} else if (tid == 0) mmg_rs_sort_exact(W, (int64_t)n_u, stack + ao / 65 + 2 * (int64_t)li, KeyX());
			}
			__syncthreads();
			// 8. write chains back to a[] in that order (chain.c:152-159)
			if (!par) {
				int dst = 0;
				for (int i0 = 0; i0 < n_u; i0 += NT) {
					const int i = i0 + tid;
					uint64_t uk = 0; int src = 0;
					if (i < n_u) { const uint64_t wy = W[i].y; uk = U1[(int32_t)(uint32_t)wy]; src = (int)(wy >> 32); }
					const int nn = (int32_t)(uint32_t)uk;
					int tot;
					const int incl = block_incl_scan(nn, s_scan, &tot);
					const int off = dst + incl - nn;
					for (int q = 0; q < nn; ++q) A[off + q] = B[src + q];
					if (i < n_u) U0[i] = uk;
					dst += tot;
				}
			} else { // the same offsets; anchors moved by all threads: b[t] belongs to chain cid[t], whose anchors shift by T[kk]
				int32_t *cid = reinterpret_cast<int32_t*>(W) + 2 * (int64_t)n;
				int dst = 0;
				for (int i0 = 0; i0 < n_u; i0 += NT) {
					const int i = i0 + tid;
					uint64_t uk = 0; int src = 0, kk = 0;
					if (i < n_u) { const uint64_t wy = W[i].y; kk = (int32_t)(uint32_t)wy; uk = U1[kk]; src = (int)(wy >> 32); }
					const int nn = (int32_t)(uint32_t)uk;
					int tot;
					const int incl = block_incl_scan(nn, s_scan, &tot);
					if (i < n_u) T[kk] = dst + incl - nn - src, U0[i] = uk;
					dst += tot;
				}
				__syncthreads();
				for (int t = tid; t < n_v; t += NT) A[t + T[Pp[cid[t]]]] = B[t];
			}
			__syncthreads();
		}
	}
	if (tid == 0) {
		nu_out[li] = n_u, nv_out[li] = n_v;
		if (flag_out) flag_out[f] = chain_wants_rechain(rechain_enabled && rep[li] > 0, n_u, U0, A, segs);
	}
	__syncthreads(); // s_nu, s_tie and the staging area belong to the next fragment from here
	}
}

// gather per-fragment results (first or second pass) into dense output arrays
__global__ void k_gather(int n_frag, const int32_t *__restrict__ src_li /* second-pass slot or -1 */,
                         const int64_t *__restrict__ aoff1, const uint64_t *__restrict__ u1, const mm128 *__restrict__ a1,
                         const int64_t *__restrict__ aoff2, const uint64_t *__restrict__ u2, const mm128 *__restrict__ a2,
                         const int32_t *__restrict__ nu, const int32_t *__restrict__ nv, const int64_t *__restrict__ uoff,
                         const int64_t *__restrict__ voff, uint64_t *__restrict__ out_u, mm128 *__restrict__ out_a)
{
	const int f = blockIdx.x;
	if (f >= n_frag) return;
	const int s = src_li ? src_li[f] : -1;
	const uint64_t *U = s >= 0 ? u2 + aoff2[s] * 2 : u1 + aoff1[f] * 2;
	const mm128 *A = s >= 0 ? a2 + aoff2[s] : a1 + aoff1[f];
	for (int i = threadIdx.x; i < nu[f]; i += blockDim.x) out_u[uoff[f] + i] = U[i];
	// a re-chained fragment carries ~10^5 anchors: eight independent loads per thread and round, or its CTA holds the launch
	// for a millisecond of one-at-a-time round trips
	const int n = nv[f], nt = blockDim.x;
	mm128 *O = out_a + voff[f];
	int i = threadIdx.x;
	for (; i + 7 * nt < n; i += 8 * nt) {
		mm128 v[8];
#pragma unroll
		for (int q = 0; q < 8; ++q) v[q] = A[i + q * nt];
#pragma unroll
		for (int q = 0; q < 8; ++q) O[i + q * nt] = v[q];
	}
	for (; i < n; i += nt) O[i] = A[i];
}

__global__ void k_gather_mini(int n_frag, FragTab ft, const int32_t *__restrict__ src_li, const uint64_t *__restrict__ mini1,
                              const uint64_t *__restrict__ mini2, const int32_t *__restrict__ nmini, const int64_t *__restrict__ moff,
                              uint64_t *__restrict__ out)
{
	const int f = blockIdx.x;
	if (f >= n_frag) return;
	const int64_t b = ft.unit_off[ft.unit0[f]];
	const uint64_t *M = (src_li && src_li[f] >= 0 ? mini2 : mini1) + b;
	for (int i = threadIdx.x; i < nmini[f]; i += blockDim.x) out[moff[f] + i] = M[i];
}

// merge second-pass per-fragment scalars back into the first-pass arrays
__global__ void k_merge_pass2(int n_list, const int32_t *__restrict__ list, const int32_t *__restrict__ nu2, const int32_t *__restrict__ nv2,
                              const int32_t *__restrict__ rep2, const int32_t *__restrict__ nmini2, int32_t *__restrict__ nu, int32_t *__restrict__ nv,
                              int32_t *__restrict__ rep, int32_t *__restrict__ nmini, int32_t *__restrict__ src_li)
{
	const int li = blockIdx.x * blockDim.x + threadIdx.x;
	if (li >= n_list) return;
	const int f = list[li];
	nu[f] = nu2[li], nv[f] = nv2[li], rep[f] = rep2[li], nmini[f] = nmini2[li], src_li[f] = li;
}

// ------------------------------------------------------------------ host side

static int scan_i32_to_i64(mmg_ctx_t *c, const int32_t *d_in, int64_t *d_out, int n)
{ // exclusive sum over n items (callers pass n_items+1 to get the total in the last slot)
	size_t tmp = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tmp, d_in, d_out, n, c->stream);
	MMG_TRY(c->d_cub.ensure(tmp));
	MMG_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, d_in, d_out, n, c->stream));
	++c->launches;
	return MMG_OK;
}

extern "C" int mmg_job_buffers(mmg_ctx_t *c, size_t n_jobs, mmg_ksw_job_t **jobs, mmg_ksw_res_t **res)
{ // page-locked, owned by the ctx, grown on demand and kept across batches (allocating pinned memory is slow)
	cudaSetDevice(c->dev);
	MMG_TRY(c->h_k_jobs.ensure((n_jobs + 1) * sizeof(mmg_ksw_job_t)));
	MMG_TRY(c->h_k_res.ensure((n_jobs + 1) * sizeof(mmg_ksw_res_t)));
	*jobs = c->h_k_jobs.as<mmg_ksw_job_t>(), *res = c->h_k_res.as<mmg_ksw_res_t>();
	return MMG_OK;
}

// pinned table block of a staging slot: seq_off[n_seq+2] | seq_len[n_seq+2] | n_seg[n_frag+2] | seg_off[n_frag+2]
static void tab_layout(void *base, int n_seq, int n_frag, int32_t **seq_len, uint64_t **seq_off, int32_t **n_seg, int32_t **seg_off)
{
	uint8_t *p = static_cast<uint8_t*>(base);
	*seq_off = reinterpret_cast<uint64_t*>(p); p += ((size_t)n_seq + 2) * 8;
	*seq_len = reinterpret_cast<int32_t*>(p); p += (((size_t)n_seq + 2) * 4 + 15) & ~(size_t)15;
	*n_seg = reinterpret_cast<int32_t*>(p); p += (((size_t)n_frag + 2) * 4 + 15) & ~(size_t)15;
	*seg_off = reinterpret_cast<int32_t*>(p);
}
static size_t tab_bytes(int n_seq, int n_frag) { return ((size_t)n_seq + 2) * 12 + ((size_t)n_frag + 2) * 8 + 64; }

int mmg_stage_grow(mmg_ctx_t *c, int slot, PinBuf StageSlot::*buf, size_t bytes)
{
	const bool together = slot != 0 || (c->stage[1].*buf).p != nullptr;
	for (int k = 0; k < MMG_STAGE_SLOTS; ++k) {
		const int s = (slot + k) % MMG_STAGE_SLOTS;
		PinBuf &b = c->stage[s].*buf;
		if (s == slot) MMG_CUDA(cudaEventSynchronize(c->stage[s].drained));
		if ((s != slot && !together) || bytes <= b.cap) continue;
		if (s != slot) MMG_CUDA(cudaEventSynchronize(c->stage[s].drained));
		MMG_TRY(b.ensure(bytes));
	}
	return MMG_OK;
}

extern "C" int mmg_stage(mmg_ctx_t *c, int slot, int n_frag, int n_seq, uint64_t n_bases, int with_flip, int with_ukey, mmg_stage_t *out)
{
	if (slot < 0 || slot >= MMG_STAGE_SLOTS || n_frag < 0 || n_seq < 0) {
		mmg_set_error("mmg_stage: slot %d, %d fragments, %d reads", slot, n_frag, n_seq);
		return MMG_EINVAL;
	}
	MMG_CUDA(cudaSetDevice(c->dev));
	StageSlot &s = c->stage[slot];
	MMG_TRY(mmg_stage_grow(c, slot, &StageSlot::bases, n_bases + 65));
	MMG_TRY(mmg_stage_grow(c, slot, &StageSlot::tab, tab_bytes(n_seq, n_frag)));
	if (with_flip) MMG_TRY(mmg_stage_grow(c, slot, &StageSlot::flip, (size_t)n_seq + 16));
	if (with_ukey) MMG_TRY(mmg_stage_grow(c, slot, &StageSlot::ukey, ((size_t)n_frag + 4) * 4));
	s.n_frag = n_frag, s.n_seq = n_seq, s.n_bases = n_bases, s.has_flip = with_flip != 0, s.has_ukey = with_ukey != 0;
	out->bases = s.bases.as<char>();
	tab_layout(s.tab.p, n_seq, n_frag, &out->seq_len, &out->seq_off, &out->n_seg, &out->seg_off);
	out->flip = s.has_flip ? s.flip.as<uint8_t>() : nullptr;
	out->ukey = s.has_ukey ? s.ukey.as<uint32_t>() : nullptr;
	return MMG_OK;
}

struct PadLen8 { __host__ __device__ uint64_t operator()(int32_t len) const { return ((uint64_t)len + 7) / 8 * 8; } };
struct UnitsOfLen { __host__ __device__ int64_t operator()(int32_t len) const { return ((int64_t)len + MMG_READ_CHUNK - 1) / MMG_READ_CHUNK; } };

// what the sketch and the later stages need per read and per fragment, from the lengths alone: the sketch work units
// (one per MMG_READ_CHUNK positions of a read), the mates to flip (pe_ori, map.c:467-469), the fragments' unit ranges and
// query lengths.  (The host used to build these 60 bytes per read and copy them over from pageable memory, every batch.)
// flip_given: flip[] already holds the per-read decision (mmg_batch_t.flip), it is not derived from the fragment here
__global__ void k_batch_tables(int n_frag, int n_seq, const int32_t *__restrict__ n_seg, const int32_t *__restrict__ seg_off,
                               const int32_t *__restrict__ seq_len, const uint64_t *__restrict__ q_off, const int64_t *__restrict__ unit0, int pe_ori,
                               int flip_given, SketchUnit *__restrict__ units, uint8_t *__restrict__ flip, int32_t *__restrict__ frag_unit0,
                               int32_t *__restrict__ frag_qlen)
{
	const int f = blockIdx.x * blockDim.x + threadIdx.x;
	if (f > n_frag) return;
	if (f == n_frag) { frag_unit0[f] = (int32_t)unit0[n_seq]; return; }
	const int off = seg_off[f], ns = n_seg[f];
	int sum = 0;
	frag_unit0[f] = (int32_t)unit0[off];
	for (int j = 0; j < ns; ++j) {
		const int r = off + j, len = seq_len[r];
		if (!flip_given) flip[r] = (ns == 2 && ((j == 0 && (pe_ori >> 1 & 1)) || (j == 1 && (pe_ori & 1)))) ? 1 : 0;
		int64_t uu = unit0[r];
		for (int st = 0; st < len; st += MMG_READ_CHUNK) {
			SketchUnit u;
			u.off = q_off[r], u.len = len, u.rid = (uint32_t)j, u.y_add = (uint64_t)sum << 1;
			u.emit_start = st, u.emit_end = st + MMG_READ_CHUNK < len ? st + MMG_READ_CHUNK : len;
			units[uu++] = u;
		}
		sum += len;
	}
	frag_qlen[f] = sum;
}

extern "C" int mmg_upload_stage(mmg_ctx_t *c, const mmg_mapopt_t *opt, int slot)
{
	if (slot < 0 || slot >= MMG_STAGE_SLOTS || c->stage[slot].tab.p == nullptr) {
		mmg_set_error("mmg_upload_stage: slot %d holds no batch (mmg_stage)", slot);
		return MMG_EINVAL;
	}
	MMG_CUDA(cudaSetDevice(c->dev));
	const StageSlot &s = c->stage[slot];
	ResidentBatch &rb = c->rb;
	// the reads go first: their copy runs while the host looks at the lengths below
	const size_t sz_bases = (s.n_bases + 15) & ~(size_t)15;
	MMG_TRY(c->d_ascii.ensure(sz_bases + 64));
	MMG_H2D(c, c->d_ascii.p, s.bases.p, s.n_bases);
	const int n_seq = s.n_seq, n_frag = s.n_frag;
	int32_t *t_len, *t_nseg, *t_segoff; uint64_t *t_off;
	tab_layout(s.tab.p, n_seq, n_frag, &t_len, &t_off, &t_nseg, &t_segoff);
	rb.n_frag = n_frag, rb.n_seq = n_seq, rb.n_bases = s.n_bases, rb.has_ukey = s.has_ukey;
	rb.n_seg.assign(t_nseg, t_nseg + n_frag);
	rb.seg_off.assign(t_segoff, t_segoff + n_frag);
	rb.seq_len.assign(t_len, t_len + n_seq);
	t_len[n_seq] = 0, t_off[n_seq] = s.n_bases; // the scans below run over n_seq + 1 items
	uint64_t qo = 0; int64_t nu = 0;
	int max_len = 0;
	for (int r = 0; r < n_seq; ++r) { qo += PadLen8()(t_len[r]); nu += UnitsOfLen()(t_len[r]); max_len = max_len > t_len[r] ? max_len : t_len[r]; }
	rb.max_len = max_len;
	rb.q_words = qo / 8;
	rb.n_units = (int)nu;

	MMG_TRY(c->d_Q.ensure((rb.q_words + 8) * 4));
	MMG_TRY(c->d_seq_len.ensure((size_t)(n_seq + 2) * 4));
	MMG_TRY(c->d_seq_off.ensure((size_t)(n_seq + 2) * 8));
	MMG_TRY(c->d_q_off.ensure((size_t)(n_seq + 2) * 8));
	MMG_TRY(c->d_unit0.ensure((size_t)(n_seq + 2) * 8));
	MMG_TRY(c->d_flip.ensure((size_t)n_seq + 16));
	MMG_TRY(c->d_units.ensure((size_t)(rb.n_units + 1) * sizeof(SketchUnit)));
	MMG_TRY(c->d_frag_unit0.ensure((size_t)(n_frag + 2) * 4));
	MMG_TRY(c->d_frag_qlen.ensure((size_t)(n_frag + 2) * 4));
	MMG_TRY(c->d_frag_nseg.ensure((size_t)(n_frag + 2) * 4));
	MMG_TRY(c->d_fseg_off.ensure((size_t)(n_frag + 2) * 4));
	MMG_H2D(c, c->d_seq_len.p, t_len, (size_t)(n_seq + 1) * 4);
	MMG_H2D(c, c->d_seq_off.p, t_off, (size_t)(n_seq + 1) * 8);
	MMG_H2D(c, c->d_frag_nseg.p, t_nseg, (size_t)n_frag * 4);
	MMG_H2D(c, c->d_fseg_off.p, t_segoff, (size_t)n_frag * 4);
	if (s.has_flip && n_seq > 0) MMG_H2D(c, c->d_flip.p, s.flip.p, (size_t)n_seq);
	if (s.has_ukey) {
		MMG_TRY(c->d_ukey.ensure(((size_t)n_frag + 4) * 4));
		if (n_frag > 0) MMG_H2D(c, c->d_ukey.p, s.ukey.p, (size_t)n_frag * 4);
	}
	MMG_CUDA(cudaEventRecord(s.drained, c->stream)); // the next mmg_stage of this slot waits for it
	{ // packed (8-base aligned) offset of every read, first sketch unit of every read
		cub::TransformInputIterator<uint64_t, PadLen8, const int32_t*> it_q(c->d_seq_len.as<int32_t>(), PadLen8());
		cub::TransformInputIterator<int64_t, UnitsOfLen, const int32_t*> it_u(c->d_seq_len.as<int32_t>(), UnitsOfLen());
		size_t t1 = 0, t2 = 0;
		cub::DeviceScan::ExclusiveSum(nullptr, t1, it_q, c->d_q_off.as<uint64_t>(), n_seq + 1, c->stream);
		cub::DeviceScan::ExclusiveSum(nullptr, t2, it_u, c->d_unit0.as<int64_t>(), n_seq + 1, c->stream);
		MMG_TRY(c->d_cub.ensure(t1 > t2 ? t1 : t2));
		MMG_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, t1, it_q, c->d_q_off.as<uint64_t>(), n_seq + 1, c->stream));
		MMG_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, t2, it_u, c->d_unit0.as<int64_t>(), n_seq + 1, c->stream));
		c->launches += 2;
	}
	MMG_LAUNCH(c, k_batch_tables, mmg_blocks((size_t)n_frag + 1, 256), 256, 0, n_frag, n_seq, c->d_frag_nseg.as<int32_t>(), c->d_fseg_off.as<int32_t>(),
	           c->d_seq_len.as<int32_t>(), c->d_q_off.as<uint64_t>(), c->d_unit0.as<int64_t>(), opt->pe_ori, s.has_flip ? 1 : 0, c->d_units.as<SketchUnit>(),
	           c->d_flip.as<uint8_t>(), c->d_frag_unit0.as<int32_t>(), c->d_frag_qlen.as<int32_t>());
	if (rb.q_words)
		MMG_LAUNCH(c, k_encode_reads, mmg_blocks(rb.q_words, 256), 256, 0, c->d_ascii.as<uint8_t>(), c->d_seq_off.as<uint64_t>(),
		           c->d_seq_len.as<int32_t>(), c->d_q_off.as<uint64_t>(), c->d_flip.as<uint8_t>(), n_seq, rb.q_words, c->d_Q.as<uint32_t>());
	return MMG_OK;
}

extern "C" int mmg_batch_upload(mmg_ctx_t *c, const mmg_mapopt_t *opt, const mmg_batch_t *b)
{
	mmg_stage_t st;
	MMG_TRY(mmg_stage(c, 0, b->n_frag, b->n_seq, b->n_bases, b->flip != nullptr, b->ukey != nullptr, &st));
	memcpy(st.bases, b->bases, b->n_bases);
	memcpy(st.seq_len, b->seq_len, (size_t)b->n_seq * 4);
	memcpy(st.seq_off, b->seq_off, (size_t)b->n_seq * 8);
	memcpy(st.n_seg, b->n_seg, (size_t)b->n_frag * 4);
	memcpy(st.seg_off, b->seg_off, (size_t)b->n_frag * 4);
	if (b->flip) memcpy(st.flip, b->flip, (size_t)b->n_seq);
	if (b->ukey) memcpy(st.ukey, b->ukey, (size_t)b->n_frag * 4);
	return mmg_upload_stage(c, opt, 0);
}

// the dynamic shared memory the chain tail's CTA form launches with, allowed on the current device (mmg_init, once per context)
int mmg_stages_set_smem_attrs()
{
	MMG_CUDA(cudaFuncSetAttribute(k_chain_tail_block, cudaFuncAttributeMaxDynamicSharedMemorySize, TAIL_BLOCK_SMEM));
	return MMG_OK;
}

// the device counters of a batch that feed c->path[] (mmg_path_counts), read back into the pinned c->h_path
struct PathCounters {
	int32_t heap[2][4];        // per pass (k_heap_list): [0] fragments replayed on ranks, [1] k_heap_replay's cursor, [2] fragments left to k_fill
	unsigned long long pops;   // seed hits whose merge order was replayed (k_heap_emit)
	unsigned long long named;  // seed hits the self/dual filters dropped; one copy from d_frag_iter fills this and pops
};

// one pass: the fragments it takes and the typed pointers of its arena
struct PassTab {
	const int32_t *list;       // fragment of every slot; null: slot li is fragment li
	int n_list;
	int64_t *aoff;             // [n_list+1] first anchor slot of every fragment
	int32_t *na, *rep, *nmini, *nu, *nv;
	uint64_t *mini;            // null when nothing reads the minimizer positions
	mm128 *a, *b;
	int32_t *work;             // per anchor f|p|t|v, then the chain-order array
	uint64_t *u;
	RsFrame *stack;
};

// the view of pass `pass`'s arena; taken again whenever the arena has grown
static PassTab pass_tab(mmg_ctx_t *c, int pass, const int32_t *d_list, int n_list, bool want_mini)
{
	const PassArena &A = c->pass[pass];
	PassTab t;
	t.list = d_list, t.n_list = n_list;
	t.aoff = A.aoff.as<int64_t>(), t.na = A.na.as<int32_t>(), t.rep = A.rep.as<int32_t>(), t.nmini = A.nmini.as<int32_t>();
	t.mini = want_mini ? A.mini.as<uint64_t>() : nullptr;
	t.a = A.a.as<mm128>(), t.work = A.work.as<int32_t>(), t.u = A.u.as<uint64_t>(), t.b = A.b.as<mm128>(), t.stack = A.stack.as<RsFrame>();
	t.nu = A.nu.as<int32_t>(), t.nv = A.nv.as<int32_t>();
	return t;
}

// K2 of pass `pass` (0: every fragment with mid_occ; 1: the fragments in d_list, re-chained with max_occ): plan -> scan -> sort ->
// heap replay on ranks and literal heap merge, or the radix-order replay of the non-heap presets.  The anchors stay in the pass's
// arena; *pt is its view.
static int seed_pass(mmg_ctx_t *c, const mmg_idx_t *mi, const mmg_mapopt_t *opt, const FragTab &ft, const NameTabs &nt, int pass, const int32_t *d_list, int n_list,
                     int max_occ, int64_t n_mv, bool want_mini, PassTab *pt, int64_t *n_anchors)
{
	PassArena &A = c->pass[pass];
	unsigned long long *n_named = c->d_frag_iter.as<unsigned long long>() + 2;
	const bool named = nt.ukey != nullptr;
	MMG_TRY(A.na.ensure((size_t)(n_list + 1) * 4));
	MMG_TRY(A.aoff.ensure((size_t)(n_list + 1) * 8));
	MMG_TRY(A.rep.ensure((size_t)(n_list + 1) * 4));
	MMG_TRY(A.nmini.ensure((size_t)(n_list + 1) * 4));
	MMG_TRY(A.nu.ensure((size_t)(n_list + 1) * 4));
	MMG_TRY(A.nv.ensure((size_t)(n_list + 1) * 4));
	if (want_mini) MMG_TRY(A.mini.ensure((size_t)(n_mv + 1) * 8));
	const bool heap_path = (opt->flag & MMG_F_HEAP_SORT) != 0;
	MMG_TRY(c->d_replay.ensure((size_t)n_list + 16));
	MMG_CUDA(cudaMemsetAsync(A.na.p, 0, (size_t)(n_list + 1) * 4, c->stream));
	MMG_CUDA(cudaMemsetAsync(A.nu.p, 0, (size_t)(n_list + 1) * 4, c->stream)); // slot n_list must read 0 for the scans
	MMG_CUDA(cudaMemsetAsync(A.nv.p, 0, (size_t)(n_list + 1) * 4, c->stream));
	MMG_CUDA(cudaMemsetAsync(A.nmini.p, 0, (size_t)(n_list + 1) * 4, c->stream));
	PassTab t = pass_tab(c, pass, d_list, n_list, want_mini);
	MMG_LAUNCH(c, k_plan, mmg_blocks(n_list, 128), 128, 0, ft, d_list, n_list, c->d_mv.as<mm128>(), c->d_m_n.as<int32_t>(), max_occ, t.na, t.rep, t.nmini, t.mini,
	           heap_path ? c->d_replay.as<uint8_t>() : nullptr, c->d_m_aoff.as<int32_t>());
	MMG_TRY(scan_i32_to_i64(c, t.na, t.aoff, n_list + 1));
	int32_t *hp_counters = nullptr, *rlist = nullptr, *hp = c->h_path.as<PathCounters>()->heap[pass];
	if (heap_path) { // the fragments whose heap order has to be replayed: their number rides on the synchronisation below
		MMG_TRY(c->d_hlist.ensure(((size_t)n_list + 8) * 4));
		hp_counters = c->d_hlist.as<int32_t>(), rlist = hp_counters + 4;
		MMG_CUDA(cudaMemsetAsync(hp_counters, 0, 16, c->stream));
		MMG_LAUNCH(c, k_heap_list, mmg_blocks(n_list, 256), 256, 0, n_list, c->d_replay.as<uint8_t>(), rlist, hp_counters);
		MMG_D2H(c, hp, hp_counters, 16);
	}
	int64_t tot = 0;
	MMG_D2H(c, &tot, t.aoff + n_list, 8);
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	MMG_TRY(A.a.ensure((size_t)(tot + 1) * 16));
	MMG_TRY(A.work.ensure((size_t)(tot + 1) * 32)); // f|p|t|v then the chain-order array
	MMG_TRY(A.u.ensure((size_t)(tot + 1) * 16));
	MMG_TRY(A.b.ensure((size_t)(tot + 1) * 16));
	MMG_TRY(A.stack.ensure((size_t)(tot / 65 + 2 * (size_t)n_list + 4) * sizeof(RsFrame)));
	t = pass_tab(c, pass, d_list, n_list, want_mini);
	MMG_TRY(c->d_heap.ensure((size_t)(n_mv + 1) * 16));
	uint8_t *d_tie = nullptr;
	if (!heap_path) { // radix-sort form: sort everything, replay only the fragments where two anchors share x
		MMG_TRY(c->d_tie.ensure((size_t)n_list + 16));
		d_tie = c->d_tie.as<uint8_t>();
		MMG_CUDA(cudaMemsetAsync(d_tie, 0, (size_t)n_list + 16, c->stream));
		MMG_CUDA(cudaMemsetAsync(c->d_replay.p, 0, (size_t)n_list + 16, c->stream));
	}
	if (tot > 0) {
		// fragments whose keys are all distinct: the reference's order is simply the sorted order -> segmented sort
		MMG_TRY(c->d_skey.ensure(((size_t)tot + 1) * 16)); MMG_TRY(c->d_sval.ensure(((size_t)tot + 1) * 16));
		MMG_TRY(c->d_sseg.ensure(((size_t)n_list + 1) * 20 + 64));
		uint64_t *k0 = c->d_skey.as<uint64_t>(), *k1 = k0 + tot + 1, *v0 = c->d_sval.as<uint64_t>(), *v1 = v0 + tot + 1;
		int64_t *seg_b = c->d_sseg.as<int64_t>(), *seg_e = seg_b + n_list + 1;
		int32_t *n_skipped = reinterpret_cast<int32_t*>(seg_e + n_list + 1);
		MMG_CUDA(cudaMemsetAsync(n_skipped, 0, (size_t)n_list * 4, c->stream));
		MMG_LAUNCH_AS(c, "k_expand", (named ? k_expand<true> : k_expand<false>), mmg_blocks(tot, 256), 256, 0, ft, d_list, n_list, c->d_mv.as<mm128>(), c->d_m_n.as<int32_t>(),
		              c->d_m_val.as<uint64_t>(), mi->d_pos, max_occ, opt->flag, t.aoff, c->d_replay.as<uint8_t>(), tot, k0, v0, n_skipped, c->d_m_aoff.as<int32_t>(), nt, n_named);
		MMG_LAUNCH(c, k_sort_segments, mmg_blocks(n_list, 256), 256, 0, n_list, t.aoff, c->d_replay.as<uint8_t>(), seg_b, seg_e);
		{
			size_t tmp = 0;
			cub::DeviceSegmentedSort::SortPairs(nullptr, tmp, k0, k1, v0, v1, tot, n_list, seg_b, seg_e, c->stream);
			MMG_TRY(c->d_cub.ensure(tmp));
			MMG_TIMED(c, "cub_segmented_sort(seed hits)", cub::DeviceSegmentedSort::SortPairs(c->d_cub.p, tmp, k0, k1, v0, v1, tot, n_list, seg_b, seg_e, c->stream));
		}
		MMG_LAUNCH(c, k_emit_sorted, mmg_blocks(tot, 256), 256, 0, n_list, t.aoff, c->d_replay.as<uint8_t>(), tot, k1, v1, n_skipped, t.na, t.a, d_tie);
	}
	if (heap_path && tot > 0) { // fragments where equal positions meet in the heap: replay it on the ranks the sort just produced
		MMG_TRY(c->d_hrank.ensure(((size_t)tot + 1) * 4));
		MMG_TRY(c->d_hpop.ensure(((size_t)tot + 1) * 4));
		const uint64_t *k1 = c->d_skey.as<uint64_t>() + tot + 1, *v1 = c->d_sval.as<uint64_t>() + tot + 1;
		if (hp[0] > 0) {
			MMG_LAUNCH(c, k_heap_rank, mmg_blocks(tot, 256), 256, 0, n_list, t.aoff, c->d_replay.as<uint8_t>(), tot, k1, v1, c->d_hrank.as<uint32_t>());
			MMG_LAUNCH(c, k_heap_replay, hp[0] < 148 * 8 ? hp[0] : 148 * 8, 32, 0, ft, d_list, rlist, hp_counters, c->d_mv.as<mm128>(), c->d_m_n.as<int32_t>(),
			           c->d_m_val.as<uint64_t>(), c->d_m_aoff.as<int32_t>(), mi->d_pos, max_occ, opt->flag, t.aoff, c->d_hrank.as<uint32_t>(), c->d_hpop.as<uint32_t>());
			MMG_LAUNCH_AS(c, "k_heap_emit", (named ? k_heap_emit<true> : k_heap_emit<false>), hp[0], HEAP_EMIT_THREADS, 0, ft, d_list, rlist, c->d_mv.as<mm128>(),
			              c->d_m_n.as<int32_t>(), c->d_m_val.as<uint64_t>(), c->d_m_aoff.as<int32_t>(), mi->d_pos, max_occ, opt->flag, t.aoff, c->d_hpop.as<uint32_t>(),
			              t.na, t.a, c->d_frag_iter.as<unsigned long long>() + 1, nt, n_named);
		}
	}
	// literal replay: the heap merge for the few fragments the rank replay does not take; klib's radix sort for the non-heap presets
	if (!heap_path) {
		if (tot > 0)
			MMG_LAUNCH(c, k_fill_flat_warp, mmg_blocks((size_t)n_list * 32, 128), 128, 0, n_list, t.aoff, d_tie, c->d_skey.as<uint64_t>(),
			           c->d_sval.as<uint64_t>(), t.na, t.a, t.work, t.stack);
	} else {
		const int per_warp = pass == 1 || n_list <= 4096 ? 1 : 0; // the re-chain pass (and any small list): spread over warps
		MMG_LAUNCH_AS(c, "k_fill", (named ? k_fill<true> : k_fill<false>), mmg_blocks(per_warp ? (size_t)n_list * 32 : (size_t)n_list, 64), 64, 0,
		              ft, d_list, n_list, c->d_mv.as<mm128>(), c->d_m_n.as<int32_t>(), c->d_m_val.as<uint64_t>(), mi->d_pos, max_occ, opt->flag, t.aoff, t.na, t.a,
		              c->d_heap.as<mm128>(), c->d_replay.as<uint8_t>(), per_warp, nt, n_named);
	}
	if (getenv("MMG_TRACE")) { // distribution of the literal-replay work of this pass (debug aid; synchronises)
		std::vector<uint8_t> hr((size_t)n_list); std::vector<int32_t> hn((size_t)n_list);
		cudaStreamSynchronize(c->stream);
		cudaMemcpy(hr.data(), heap_path ? c->d_replay.p : (void*)d_tie, (size_t)n_list, cudaMemcpyDeviceToHost);
		cudaMemcpy(hn.data(), t.na, (size_t)n_list * 4, cudaMemcpyDeviceToHost);
		int64_t nr = 0, ar = 0, amax = 0, big = 0, abig = 0, big_all = 0, abig_all = 0;
		for (int i = 0; i < n_list; ++i) {
			if (hn[i] > 4096) ++big_all, abig_all += hn[i];
			if (!hr[i]) continue;
			++nr, ar += hn[i]; if (hn[i] > amax) amax = hn[i]; if (hn[i] > 4096) ++big, abig += hn[i];
		}
		fprintf(stderr, "[mmg::pass] max_occ %d: %d fragments, %lld anchors; > 4096 anchors: %lld fragments with %lld anchors; literal replay: %lld fragments, %lld anchors, largest %lld, "
		        "of which > 4096 anchors: %lld fragments with %lld anchors\n", max_occ, n_list, (long long)tot, (long long)big_all, (long long)abig_all, (long long)nr, (long long)ar, (long long)amax, (long long)big, (long long)abig);
	}
	*pt = t, *n_anchors = tot;
	return MMG_OK;
}

// K3 of pass `pass` on the tot anchors seed_pass left in pt: segments -> fill -> tails.  The first pass flags the fragments the
// re-chain pass takes in c->d_frag_flag.
static int chain_pass(mmg_ctx_t *c, const mmg_mapopt_t *opt, const FragTab &ft, const ChainOptDev &co, int pass, const PassTab &pt, int64_t tot)
{
	const int n_list = pt.n_list;
	const int32_t *n_seg = c->d_frag_nseg.as<int32_t>();
	if (tot > 0) {
		// segments: head flags -> compacted start indices
		MMG_TRY(c->d_seg_head.ensure((size_t)tot + 16));
		MMG_TRY(c->d_seg_start.ensure(((size_t)tot + 2) * 8 + 64));
		MMG_TRY(c->d_seg_avg.ensure((size_t)(n_list + 1) * 4));
		MMG_TRY(c->d_seg_li.ensure(((size_t)tot + 1) * 4));   // fragment slot of every segment head (sparse)
		MMG_TRY(c->d_seg_long.ensure(((size_t)tot / CHAIN_SMALL_SEG + 2) * 4)); // segments left to the warp form
		int64_t *seg_start = c->d_seg_start.as<int64_t>();
		int32_t *d_nseg = reinterpret_cast<int32_t*>(seg_start + tot + 1), *d_next = d_nseg + 1, *d_nlong = d_nseg + 2;
		MMG_CUDA(cudaMemsetAsync(d_nseg, 0, 16, c->stream));
		MMG_LAUNCH(c, k_chain_heads, mmg_blocks(tot, 256), 256, 0, ft, pt.list, n_list, n_seg, co, pt.aoff, pt.na, pt.a, tot, c->d_seg_head.as<uint8_t>(), pt.work,
		           c->d_seg_li.as<int32_t>());
		MMG_LAUNCH(c, k_chain_avgspan, mmg_blocks((size_t)n_list * 32, 128), 128, 0, n_list, pt.aoff, pt.na, pt.a, c->d_seg_avg.as<float>());
		{
			size_t tmp = 0;
			cub::CountingInputIterator<int64_t> it(0);
			cub::DeviceSelect::Flagged(nullptr, tmp, it, c->d_seg_head.as<uint8_t>(), seg_start, d_nseg, tot, c->stream);
			MMG_TRY(c->d_cub.ensure(tmp));
			MMG_CUDA(cub::DeviceSelect::Flagged(c->d_cub.p, tmp, it, c->d_seg_head.as<uint8_t>(), seg_start, d_nseg, tot, c->stream));
			++c->launches;
		}
		// short segments: a thread each; the others: persistent warps pull them from the list the first kernel leaves
		MMG_LAUNCH(c, k_chain_fill_small, 148 * 16, 128, 0, ft, pt.list, n_seg, co, pt.aoff, pt.na, pt.a, pt.work, c->d_seg_avg.as<float>(), seg_start,
		           c->d_seg_li.as<int32_t>(), d_nseg, c->d_seg_long.as<int32_t>(), d_nlong, c->d_frag_iter.as<unsigned long long>());
		MMG_LAUNCH(c, k_chain_fill, 148 * 8, 128, 0, ft, pt.list, n_list, n_seg, co, pt.aoff, pt.na, pt.a, pt.work, c->d_seg_avg.as<float>(), seg_start,
		           c->d_seg_li.as<int32_t>(), d_nseg, c->d_seg_long.as<int32_t>(), d_nlong, d_next, c->d_frag_iter.as<unsigned long long>());
	}
	// The fragments with thousands of anchors get a CTA each, with its sorts staged in shared memory: all fragments of the re-chain
	// pass (one CTA per SM, the whole shared memory), a few per thousand of the first pass (ahead of the warp kernel that takes
	// everything else).  The CTAs pull fragments from a counter, largest first.
	static const int heavy_env = getenv("MMG_TAIL_HEAVY_N") ? atoi(getenv("MMG_TAIL_HEAVY_N")) : TAIL_HEAVY_N;
	static const int walk = getenv("MMG_TAIL_WALK") ? 1 : 0;
	const int heavy_n = pass == 1 ? -1 : heavy_env, rechain_enabled = opt->max_occ > opt->mid_occ ? 1 : 0;
	MMG_TRY(c->d_heavy.ensure(((size_t)n_list * 4 + 16) * 4));
	int32_t *n_heavy = c->d_heavy.as<int32_t>(), *val0 = n_heavy + 4, *heavy = val0 + n_list;
	uint32_t *key0 = reinterpret_cast<uint32_t*>(heavy + n_list), *key1 = key0 + n_list;
	MMG_CUDA(cudaMemsetAsync(n_heavy, 0, 16, c->stream));
	MMG_LAUNCH(c, k_tail_heavy_list, mmg_blocks(n_list, 256), 256, 0, n_list, pt.na, heavy_n, key0, val0, n_heavy);
	{
		size_t tmp = 0;
		cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp, key0, key1, val0, heavy, n_list, 0, 32, c->stream);
		MMG_TRY(c->d_cub.ensure(tmp));
		MMG_CUDA(cub::DeviceRadixSort::SortPairsDescending(c->d_cub.p, tmp, key0, key1, val0, heavy, n_list, 0, 32, c->stream));
		++c->launches;
	}
	if (pass == 1)
		MMG_LAUNCH(c, k_chain_tail_block, n_list < 148 ? n_list : 148, 1024, TAIL_BLOCK_SMEM, ft, pt.list, n_list, n_seg, co, pt.aoff, pt.na, pt.a, pt.work,
		           pt.u, pt.b, pt.stack, pt.nu, pt.nv, heavy, n_heavy, (size_t)TAIL_BLOCK_SMEM, nullptr, 0, nullptr, walk);
	else {
		uint8_t *flag = c->d_frag_flag.as<uint8_t>();
		MMG_LAUNCH(c, k_chain_tail_block, 148 * 3, 512, TAIL_HEAVY_SMEM, ft, pt.list, n_list, n_seg, co, pt.aoff, pt.na, pt.a, pt.work, pt.u, pt.b, pt.stack,
		           pt.nu, pt.nv, heavy, n_heavy, (size_t)TAIL_HEAVY_SMEM, pt.rep, rechain_enabled, flag, walk);
		MMG_LAUNCH(c, k_chain_tail_warp, mmg_blocks((size_t)n_list * 32, 128), 128, 0, ft, pt.list, n_list, n_seg, co, pt.aoff, pt.na, pt.a, pt.work, pt.u,
		           pt.b, pt.stack, pt.nu, pt.nv, pt.rep, rechain_enabled, flag, heavy_n);
	}
	return MMG_OK;
}

extern "C" int mmg_seed_chain_resident(mmg_ctx_t *c, const mmg_idx_t *mi, const mmg_mapopt_t *opt, mmg_chains_t *out, int download)
{
	MMG_CUDA(cudaSetDevice(c->dev));
	ResidentBatch &rb = c->rb;
	const int nf = rb.n_frag;
	memset(out, 0, sizeof(*out));
	out->n_frag = nf;
	if (nf == 0) return MMG_OK;
	if (mi->w > MMG_MAX_W) { mmg_set_error("w=%d exceeds the device limit %d", mi->w, MMG_MAX_W); return MMG_ELIMIT; }
	NameTabs nt = {nullptr, nullptr, nullptr};
	if (opt->flag & (MMG_F_NO_DIAG | MMG_F_NO_DUAL)) { // never filter on keys of another index or batch
		if (mi->d_tkey == nullptr) { mmg_set_error("the self/dual filters need the target name keys (mmg_idx_set_name_keys)"); return MMG_EINVAL; }
		if (!rb.has_ukey) { mmg_set_error("the self/dual filters need the name keys of this batch (mmg_batch_t.ukey)"); return MMG_EINVAL; }
		nt.tkey = mi->d_tkey, nt.tlen = mi->d_seq_len, nt.ukey = c->d_ukey.as<uint32_t>();
	}
	MMG_CUDA(cudaEventRecord(c->ev[0], c->stream));
	// K1
	int64_t n_mv = 0;
	MMG_TRY(mmg_run_sketch(c, c->d_Q.as<uint32_t>(), c->d_units.as<SketchUnit>(), rb.n_units, mi->w, mi->k, mi->is_hpc, c->d_unit_cnt,
	                       c->d_unit_off, c->d_mv, &n_mv, rb.max_len <= SKW_MAX_LEN, rb.q_words * 8));
	// K2a
	MMG_TRY(c->d_m_n.ensure((size_t)(n_mv + 1) * 4));
	MMG_TRY(c->d_m_val.ensure((size_t)(n_mv + 1) * 8));
	MMG_TRY(c->d_m_aoff.ensure((size_t)(n_mv + 1) * 4));
	if (n_mv) MMG_LAUNCH(c, k_lookup, mmg_blocks(n_mv, 256), 256, 0, mi->view(), c->d_mv.as<mm128>(), n_mv, c->d_m_n.as<int32_t>(), c->d_m_val.as<uint64_t>());
	FragTab ft;
	ft.unit0 = c->d_frag_unit0.as<int32_t>(), ft.unit_off = c->d_unit_off.as<int64_t>(), ft.qlen = c->d_frag_qlen.as<int32_t>();
	ChainOptDev co;
	co.bw = opt->bw, co.max_gap = opt->max_gap, co.max_gap_ref = opt->max_gap_ref, co.max_frag_len = opt->max_frag_len;
	co.max_skip = opt->max_chain_skip, co.max_iter = opt->max_chain_iter, co.min_cnt = opt->min_cnt, co.min_sc = opt->min_chain_score;
	co.is_cdna = !!(opt->flag & MMG_F_SPLICE), co.is_sr = !!(opt->flag & MMG_F_SR);
	const bool want_mini = !(opt->flag & MMG_F_SR); // only mm_est_err reads mini_pos (map.c:388)
	MMG_TRY(c->d_frag_flag.ensure((size_t)nf + 16));
	MMG_TRY(c->d_frag_iter.ensure(32)); // chain iterations | replayed merge pops | hits the self/dual filters dropped
	MMG_CUDA(cudaMemsetAsync(c->d_frag_flag.p, 0, (size_t)nf + 16, c->stream));
	MMG_CUDA(cudaMemsetAsync(c->d_frag_iter.p, 0, 32, c->stream));
	MMG_TRY(c->h_path.ensure(sizeof(PathCounters)));
	PathCounters *pc = c->h_path.as<PathCounters>();
	memset(pc, 0, sizeof(*pc));
	PassTab p1, p2;
	int64_t n_anch1 = 0, n_anch2 = 0;
	MMG_TRY(seed_pass(c, mi, opt, ft, nt, 0, nullptr, nf, opt->mid_occ, n_mv, want_mini, &p1, &n_anch1));
	MMG_TRY(chain_pass(c, opt, ft, co, 0, p1, n_anch1));
	// second pass: fragments whose best chain misses a segment, with the higher cut-off (map.c:353-375)
	std::vector<int32_t> list;
	std::vector<uint8_t> hflag(nf);
	MMG_TRY(c->d_frag_list.ensure((size_t)(nf + 1) * 8)); // [0,nf): list, [nf,2nf): src slot per fragment
	int32_t *d_list = c->d_frag_list.as<int32_t>(), *d_src = d_list + nf;
	MMG_CUDA(cudaMemsetAsync(d_src, 0xff, (size_t)nf * 4, c->stream));
	if (opt->max_occ > opt->mid_occ) {
		MMG_D2H(c, hflag.data(), c->d_frag_flag.p, nf);
		MMG_CUDA(cudaStreamSynchronize(c->stream));
		for (int f = 0; f < nf; ++f) if (hflag[f]) list.push_back(f);
	}
	const int n2 = (int)list.size();
	if (n2) {
		MMG_H2D(c, d_list, list.data(), (size_t)n2 * 4);
		MMG_TRY(seed_pass(c, mi, opt, ft, nt, 1, d_list, n2, opt->max_occ, n_mv, want_mini, &p2, &n_anch2));
		MMG_TRY(chain_pass(c, opt, ft, co, 1, p2, n_anch2));
		MMG_LAUNCH(c, k_merge_pass2, mmg_blocks(n2, 128), 128, 0, n2, d_list, p2.nu, p2.nv, p2.rep, p2.nmini, p1.nu, p1.nv, p1.rep, p1.nmini, d_src);
	} else p2 = pass_tab(c, 1, d_list, 0, want_mini); // unread: no fragment has a second-pass slot
	// dense outputs
	MMG_TRY(c->d_uoff.ensure((size_t)(nf + 1) * 8));
	MMG_TRY(c->d_voff.ensure((size_t)(nf + 1) * 8));
	MMG_TRY(c->d_moff.ensure((size_t)(nf + 1) * 8));
	MMG_TRY(scan_i32_to_i64(c, p1.nu, c->d_uoff.as<int64_t>(), nf + 1));
	MMG_TRY(scan_i32_to_i64(c, p1.nv, c->d_voff.as<int64_t>(), nf + 1));
	if (want_mini) MMG_TRY(scan_i32_to_i64(c, p1.nmini, c->d_moff.as<int64_t>(), nf + 1));
	int64_t tot[3] = {0, 0, 0};
	MMG_D2H(c, &tot[0], c->d_uoff.as<int64_t>() + nf, 8);
	MMG_D2H(c, &tot[1], c->d_voff.as<int64_t>() + nf, 8);
	if (want_mini) MMG_D2H(c, &tot[2], c->d_moff.as<int64_t>() + nf, 8);
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	c->last_tot_u = tot[0], c->last_tot_v = tot[1];
	MMG_TRY(c->d_out_u.ensure((size_t)(tot[0] + 1) * 8));
	MMG_TRY(c->d_out_a.ensure((size_t)(tot[1] + 1) * 16));
	MMG_TRY(c->d_out_mini.ensure((size_t)(tot[2] + 1) * 8));
	MMG_LAUNCH(c, k_gather, nf, 64, 0, nf, d_src, p1.aoff, p1.u, p1.a, p2.aoff, p2.u, p2.a, p1.nu, p1.nv, c->d_uoff.as<int64_t>(), c->d_voff.as<int64_t>(),
	           c->d_out_u.as<uint64_t>(), c->d_out_a.as<mm128>());
	if (want_mini)
		MMG_LAUNCH(c, k_gather_mini, nf, 64, 0, nf, ft, d_src, p1.mini, p2.mini, p1.nmini, c->d_moff.as<int64_t>(), c->d_out_mini.as<uint64_t>());
	MMG_CUDA(cudaEventRecord(c->ev[1], c->stream));
	unsigned long long iters = 0;
	MMG_D2H(c, &iters, c->d_frag_iter.p, 8);
	MMG_D2H(c, &pc->pops, c->d_frag_iter.as<unsigned long long>() + 1, 16);
	out->n_minimizers = (uint64_t)n_mv, out->n_anchors = (uint64_t)(n_anch1 + n_anch2);
	if (download) {
		// meta: n_u | n_a | rep_len | n_mini | rechained (int32 each) then u_off | a_off | mini_off (uint64 each, nf+1)
		const size_t meta_i = (size_t)nf * 5 * 4, meta_o = (size_t)(nf + 1) * 3 * 8;
		MMG_TRY(c->h_out_meta.ensure(meta_i + meta_o + 64));
		MMG_TRY(c->h_out_u.ensure((size_t)(tot[0] + 1) * 8));
		MMG_TRY(c->h_out_a.ensure((size_t)(tot[1] + 1) * 16));
		MMG_TRY(c->h_out_mini.ensure((size_t)(tot[2] + 1) * 8));
		int32_t *hi = c->h_out_meta.as<int32_t>();
		uint64_t *ho = reinterpret_cast<uint64_t*>(c->h_out_meta.as<uint8_t>() + ((meta_i + 15) & ~(size_t)15));
		MMG_D2H(c, hi, p1.nu, (size_t)nf * 4);
		MMG_D2H(c, hi + nf, p1.nv, (size_t)nf * 4);
		MMG_D2H(c, hi + 2 * nf, p1.rep, (size_t)nf * 4);
		MMG_D2H(c, hi + 3 * nf, p1.nmini, (size_t)nf * 4);
		MMG_D2H(c, hi + 4 * nf, d_src, (size_t)nf * 4);
		MMG_D2H(c, ho, c->d_uoff.p, (size_t)(nf + 1) * 8);
		MMG_D2H(c, ho + (nf + 1), c->d_voff.p, (size_t)(nf + 1) * 8);
		if (want_mini) MMG_D2H(c, ho + 2 * (nf + 1), c->d_moff.p, (size_t)(nf + 1) * 8);
		if (tot[0]) MMG_D2H(c, c->h_out_u.p, c->d_out_u.p, (size_t)tot[0] * 8);
		if (tot[1]) MMG_D2H(c, c->h_out_a.p, c->d_out_a.p, (size_t)tot[1] * 16);
		if (tot[2]) MMG_D2H(c, c->h_out_mini.p, c->d_out_mini.p, (size_t)tot[2] * 8);
		MMG_CUDA(cudaEventRecord(c->ev[2], c->stream));
		MMG_CUDA(cudaStreamSynchronize(c->stream));
		for (int f = 0; f < nf; ++f) hi[4 * nf + f] = hi[4 * nf + f] >= 0 ? 1 : 0; // src slot -> rechained flag
		if (!want_mini) { for (int f = 0; f < nf; ++f) hi[3 * nf + f] = 0; memset(ho + 2 * (nf + 1), 0, (size_t)(nf + 1) * 8); }
		out->n_u = hi, out->n_a = hi + nf, out->rep_len = hi + 2 * nf, out->n_mini = hi + 3 * nf, out->rechained = hi + 4 * nf;
		out->u_off = ho, out->a_off = ho + (nf + 1), out->mini_off = ho + 2 * (nf + 1);
		out->u = c->h_out_u.as<uint64_t>(), out->a = c->h_out_a.as<mmg128_t>(), out->mini_pos = c->h_out_mini.as<uint64_t>();
		float ms = 0;
		cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); out->t_d2h_ms = ms;
	} else MMG_CUDA(cudaStreamSynchronize(c->stream));
	// path counters of this batch (the stream is idle here)
	c->path[0] += (uint64_t)n2, c->path[1] += (uint64_t)(pc->heap[0][0] + pc->heap[1][0]), c->path[2] += (uint64_t)(pc->heap[0][2] + pc->heap[1][2]);
	c->path[6] += pc->pops, c->path[7] += pc->named;
	float ms = 0;
	cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); out->t_kernels_ms = ms;
	out->n_chain_iter = iters;
	return MMG_OK;
}

extern "C" int mmg_seed_chain_batch(mmg_ctx_t *c, const mmg_idx_t *mi, const mmg_mapopt_t *opt, const mmg_batch_t *b, mmg_chains_t *out)
{
	MMG_CUDA(cudaSetDevice(c->dev));
	MMG_CUDA(cudaEventRecord(c->ev[3], c->stream));
	MMG_TRY(mmg_batch_upload(c, opt, b));
	MMG_TRY(mmg_seed_chain_resident(c, mi, opt, out, 1));
	float ms = 0;
	cudaEventElapsedTime(&ms, c->ev[3], c->ev[0]); out->t_h2d_ms = ms;
	return MMG_OK;
}

// ------------------------------------------------------------------ single-call entry points (parity tests)

extern "C" int mmg_sketch(mmg_ctx_t *c, const char *str, int len, int w, int k, uint32_t rid, int is_hpc, mmg128_t *out, int cap, int *n_out)
{
	*n_out = 0;
	if (len <= 0) return MMG_OK;
	if (w < 1 || w > MMG_MAX_W || k < 1 || k > 28) { mmg_set_error("mmg_sketch: need 1<=w<=%d, 1<=k<=28", MMG_MAX_W); return w > MMG_MAX_W ? MMG_ELIMIT : MMG_EINVAL; }
	MMG_CUDA(cudaSetDevice(c->dev));
	// a single read, deliberately cut into small chunks so that the warm-up logic is exercised
	mmg_mapopt_t opt; memset(&opt, 0, sizeof(opt));
	int32_t one = 1, zero = 0, l = len; uint64_t o = 0;
	mmg_batch_t b; b.n_frag = 1, b.n_seq = 1, b.n_seg = &one, b.seg_off = &zero, b.seq_len = &l, b.seq_off = &o, b.bases = str, b.n_bases = (uint64_t)len;
	b.flip = nullptr, b.ukey = nullptr;
	MMG_TRY(mmg_batch_upload(c, &opt, &b));
	std::vector<SketchUnit> units;
	const int chunk = is_hpc ? len : 96;
	for (int s = 0; s < len; s += chunk) {
		SketchUnit u; u.off = 0, u.len = len, u.rid = rid, u.y_add = 0, u.emit_start = s, u.emit_end = s + chunk < len ? s + chunk : len;
		units.push_back(u);
	}
	MMG_TRY(c->d_units.ensure(units.size() * sizeof(SketchUnit)));
	MMG_H2D(c, c->d_units.p, units.data(), units.size() * sizeof(SketchUnit));
	int64_t n = 0;
	MMG_TRY(mmg_run_sketch(c, c->d_Q.as<uint32_t>(), c->d_units.as<SketchUnit>(), (int)units.size(), w, k, is_hpc, c->d_unit_cnt, c->d_unit_off, c->d_mv, &n, false, 0));
	*n_out = (int)n;
	const int64_t m = n < cap ? n : cap;
	if (m > 0) MMG_D2H(c, out, c->d_mv.p, (size_t)m * 16);
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	return MMG_OK;
}

__global__ void k_collect_one(IdxView ix, const mm128 *mv, int n_mv, int heap_sort, int64_t flag, int max_occ, int qlen, uint32_t ukey,
                              int32_t *m_n, uint64_t *m_val, mm128 *heap, mm128 *a, int64_t a_cap, RsFrame *stack, int64_t *out4, uint64_t *mini)
{
	if (blockIdx.x || threadIdx.x) return;
	for (int i = 0; i < n_mv; ++i) { uint64_t v; m_n[i] = mmg_idx_probe(ix, mv[i].x >> 8, &v); m_val[i] = v; }
	int rep, nm;
	int64_t n_a = mmg_frag_plan(mv, m_n, n_mv, max_occ, &rep, &nm, mini);
	out4[0] = n_a, out4[1] = rep, out4[2] = nm;
	if (n_a > a_cap) return;
	NameFilt nf; nf.tkey = ix.tkey, nf.tlen = ix.seq_len, nf.ukey = ukey;
	int64_t nn;
	if (heap_sort) n_a = mmg_fill_heap(mv, m_n, m_val, n_mv, max_occ, ix.pos, flag, nf, qlen, n_a, heap, a, &nn);
	else n_a = mmg_fill_flat(mv, m_n, m_val, n_mv, max_occ, ix.pos, flag, nf, qlen, a, stack, &nn);
	out4[0] = n_a;
}

static int collect_seeds(mmg_ctx_t *c, const mmg_idx_t *mi, int heap_sort, int64_t flag, int max_occ, int n_mv, const mmg128_t *mv,
                         int qlen, uint32_t ukey, mmg128_t *a_out, int64_t a_cap, int64_t *n_a, int *rep_len, int *n_mini_pos, uint64_t *mini_pos);

extern "C" int mmg_collect_seeds(mmg_ctx_t *c, const mmg_idx_t *mi, int heap_sort, int64_t flag, int max_occ, int n_mv, const mmg128_t *mv,
                                 int qlen, mmg128_t *a_out, int64_t a_cap, int64_t *n_a, int *rep_len, int *n_mini_pos, uint64_t *mini_pos)
{
	return collect_seeds(c, mi, heap_sort, flag, max_occ, n_mv, mv, qlen, MMG_NAME_NONE, a_out, a_cap, n_a, rep_len, n_mini_pos, mini_pos);
}

extern "C" int mmg_collect_seeds_named(mmg_ctx_t *c, const mmg_idx_t *mi, int heap_sort, int64_t flag, int max_occ, int n_mv, const mmg128_t *mv,
                                       int qlen, uint32_t ukey, mmg128_t *a_out, int64_t a_cap, int64_t *n_a, int *rep_len, int *n_mini_pos,
                                       uint64_t *mini_pos)
{
	if ((flag & (MMG_F_NO_DIAG | MMG_F_NO_DUAL)) && ukey != MMG_NAME_NONE && mi->d_tkey == nullptr) {
		mmg_set_error("mmg_collect_seeds_named: the index has no name keys (mmg_idx_set_name_keys)");
		return MMG_EINVAL;
	}
	return collect_seeds(c, mi, heap_sort, flag, max_occ, n_mv, mv, qlen, ukey, a_out, a_cap, n_a, rep_len, n_mini_pos, mini_pos);
}

static int collect_seeds(mmg_ctx_t *c, const mmg_idx_t *mi, int heap_sort, int64_t flag, int max_occ, int n_mv, const mmg128_t *mv,
                         int qlen, uint32_t ukey, mmg128_t *a_out, int64_t a_cap, int64_t *n_a, int *rep_len, int *n_mini_pos, uint64_t *mini_pos)
{
	MMG_CUDA(cudaSetDevice(c->dev));
	DevBuf dmv, dn, dval, dheap, da, dstack, dout, dmini;
	int rc = MMG_OK;
	auto fin = [&]() { dmv.release(); dn.release(); dval.release(); dheap.release(); da.release(); dstack.release(); dout.release(); dmini.release(); };
#define CS_TRY(x) do { rc = (x); if (rc != MMG_OK) { fin(); return rc; } } while (0)
	CS_TRY(dmv.ensure((size_t)(n_mv + 1) * 16)); CS_TRY(dn.ensure((size_t)(n_mv + 1) * 4)); CS_TRY(dval.ensure((size_t)(n_mv + 1) * 8));
	CS_TRY(dheap.ensure((size_t)(n_mv + 1) * 16)); CS_TRY(da.ensure((size_t)(a_cap + 1) * 16)); CS_TRY(dstack.ensure((size_t)(a_cap / 65 + 4) * sizeof(RsFrame)));
	CS_TRY(dout.ensure(64)); CS_TRY(dmini.ensure((size_t)(n_mv + 1) * 8));
	if (n_mv) cudaMemcpyAsync(dmv.p, mv, (size_t)n_mv * 16, cudaMemcpyHostToDevice, c->stream);
	k_collect_one<<<1, 32, 0, c->stream>>>(mi->view(), dmv.as<mm128>(), n_mv, heap_sort, flag, max_occ, qlen, ukey, dn.as<int32_t>(), dval.as<uint64_t>(),
	                                      dheap.as<mm128>(), da.as<mm128>(), a_cap, dstack.as<RsFrame>(), dout.as<int64_t>(), dmini.as<uint64_t>());
	++c->launches;
	int64_t o4[4] = {0, 0, 0, 0};
	cudaMemcpyAsync(o4, dout.p, 32, cudaMemcpyDeviceToHost, c->stream);
	cudaError_t e = cudaStreamSynchronize(c->stream);
	if (e != cudaSuccess) { mmg_set_error("mmg_collect_seeds: %s", cudaGetErrorString(e)); fin(); return MMG_ECUDA; }
	*n_a = o4[0], *rep_len = (int)o4[1], *n_mini_pos = (int)o4[2];
	if (o4[0] <= a_cap && o4[0] > 0) cudaMemcpy(a_out, da.p, (size_t)o4[0] * 16, cudaMemcpyDeviceToHost);
	if (mini_pos && o4[2] > 0) cudaMemcpy(mini_pos, dmini.p, (size_t)o4[2] * 8, cudaMemcpyDeviceToHost);
	fin();
	return MMG_OK;
#undef CS_TRY
}

__global__ void k_chain_one(ChainParams P, int64_t n, mm128 *a, int32_t *work, uint64_t *u, mm128 *b, RsFrame *stack, int64_t *out2)
{
	if (blockIdx.x || threadIdx.x) return;
	int64_t n_v = 0;
	mmg_chain_fill_seq(P, n, a, work, work + n, work + 2 * n, work + 3 * n);
	out2[0] = mmg_chain_backtrack(P, n, a, work, work + n, work + 2 * n, work + 3 * n, u, b, stack, &n_v);
	out2[1] = n_v;
}

extern "C" int mmg_chain_dp(mmg_ctx_t *c, int max_dist_x, int max_dist_y, int bw, int max_skip, int max_iter, int min_cnt, int min_sc,
                            int is_cdna, int n_segs, int64_t n, mmg128_t *a, int *n_u, uint64_t *u)
{
	*n_u = 0;
	if (n <= 0) return MMG_OK;
	MMG_CUDA(cudaSetDevice(c->dev));
	ChainParams P; P.max_dist_x = max_dist_x, P.max_dist_y = max_dist_y, P.bw = bw, P.max_skip = max_skip, P.max_iter = max_iter;
	P.min_cnt = min_cnt, P.min_sc = min_sc, P.is_cdna = is_cdna, P.n_segs = n_segs;
	DevBuf da, dw, du, db, ds, dout;
	int rc = MMG_OK;
	auto fin = [&]() { da.release(); dw.release(); du.release(); db.release(); ds.release(); dout.release(); };
#define CH_TRY(x) do { rc = (x); if (rc != MMG_OK) { fin(); return rc; } } while (0)
	CH_TRY(da.ensure((size_t)n * 16)); CH_TRY(dw.ensure((size_t)n * 16)); CH_TRY(du.ensure((size_t)n * 16)); CH_TRY(db.ensure((size_t)n * 16));
	CH_TRY(ds.ensure((size_t)(n / 65 + 4) * sizeof(RsFrame))); CH_TRY(dout.ensure(64));
	cudaMemcpyAsync(da.p, a, (size_t)n * 16, cudaMemcpyHostToDevice, c->stream);
	k_chain_one<<<1, 32, 0, c->stream>>>(P, n, da.as<mm128>(), dw.as<int32_t>(), du.as<uint64_t>(), db.as<mm128>(), ds.as<RsFrame>(), dout.as<int64_t>());
	++c->launches;
	int64_t o2[2] = {0, 0};
	cudaMemcpyAsync(o2, dout.p, 16, cudaMemcpyDeviceToHost, c->stream);
	cudaError_t e = cudaStreamSynchronize(c->stream);
	if (e != cudaSuccess) { mmg_set_error("mmg_chain_dp: %s", cudaGetErrorString(e)); fin(); return MMG_ECUDA; }
	*n_u = (int)o2[0];
	if (o2[0] > 0) { cudaMemcpy(u, du.p, (size_t)o2[0] * 8, cudaMemcpyDeviceToHost); cudaMemcpy(a, da.p, (size_t)o2[1] * 16, cudaMemcpyDeviceToHost); }
	fin();
	return MMG_OK;
#undef CH_TRY
}
