// mmg_ksw.cu -- K4: batched ksw_extd2 (ksw2_extd2_sse.c:19-393) on the device.
//
// k_ksw_prep puts every job into one of four forms by its shape; jobs are sorted by form and size and each form is one launch:
//  - fast (k_ksw_tpj): one thread per job whose band never clips, in size classes whose state fits shared memory;
//  - wavefront (k_ksw_wave): one warp per job whose band never clips but which is too large for the fast classes;
//  - literal warp (k_ksw_dpx): every other job, one warp each, running the SSE program itself so that the widened 16-lane
//    band, the stale out-of-band lanes and the block boundary carry-in rule (SURVEY.md H5) are reproduced by construction.
//    The lane arrays keep the reference's order (ksw2_extd2_sse.c:99-102) with two cells per lane on 16x2 SIMD
//    (mmg_kswdpx.h); they live in a shared-memory slot when they fit (all short-read jobs) and in a global arena otherwise;
//  - literal CTA (k_ksw_dpx_block): the same program for jobs whose state exceeds the warp's slot, one CTA per job with the
//    state in its shared memory.
#include <algorithm>
#include <cub/cub.cuh>
#include "mmg_ctx.cuh"
#include "mmg_kswdpx.h"
#include "mmg_kswfast2.h"

struct KswJobDev {       // a job as the kernel sees it: mmg_ksw_job_t resolved against the resident batch and the index
	uint64_t q_base;      // packed base offset of the read in Q
	uint64_t t_base;      // packed base offset of the target slice in S
	uint64_t mem_off, p_off, cig_off;
	int32_t q_readlen, q_rev, q_start, q_len, t_len, reversed;
	int32_t w, zdrop, end_bonus, flag;
};

struct KswScore { int32_t m; int8_t mat[25]; int8_t q, e, q2, e2; };
struct KswResDev { KswEz ez; uint64_t cigar_off; };   // == mmg_ksw_res_t

// the device tables every K4 kernel reads and writes, and the scoring.  __restrict__ does not reach the members of a struct: the
// kernels read the job tables and the sequences through __ldg, the read-only path restrict parameters would give them.
struct KswTabs {
	const mmg_ksw_job_t *jobs;
	const uint32_t *Q, *S;                                // packed reads of the resident batch, packed reference
	const uint64_t *q_off, *ref_off;                      // base offset of each read in Q, of each contig in S
	const int32_t *read_len;
	const uint64_t *mem_off, *p_off, *cig_off;            // per job: its arena slot, traceback and CIGAR (k_ksw_prep sizes, scanned)
	int8_t *gmem;
	uint8_t *gp;
	uint32_t *gcig;
	KswEz *res;
	KswScore sc;
};

__device__ __forceinline__ mmg_ksw_job_t ksw_ldg_job(const mmg_ksw_job_t *p)
{
	mmg_ksw_job_t j;
	static_assert(sizeof(j) % 4 == 0, "a job is 4-byte words");
#pragma unroll
	for (int i = 0; i < (int)(sizeof(j) / 4); ++i) reinterpret_cast<int32_t*>(&j)[i] = __ldg(reinterpret_cast<const int32_t*>(p) + i);
	return j;
}

// a job as the kernels see it: mmg_ksw_job_t resolved against the resident batch and the index
__device__ __forceinline__ KswJobDev ksw_job(const KswTabs &t, int ji)
{
	const mmg_ksw_job_t hj = ksw_ldg_job(t.jobs + ji);
	KswJobDev jb;
	jb.q_base = __ldg(t.q_off + hj.seq_id), jb.q_readlen = __ldg(t.read_len + hj.seq_id), jb.q_rev = hj.q_rev, jb.q_start = hj.q_start, jb.q_len = hj.q_len;
	jb.t_base = __ldg(t.ref_off + hj.rid) + (uint64_t)hj.t_start, jb.t_len = hj.t_len, jb.reversed = hj.reversed;
	jb.w = hj.w, jb.zdrop = hj.zdrop, jb.end_bonus = hj.end_bonus, jb.flag = hj.flag;
	jb.mem_off = __ldg(t.mem_off + ji), jb.p_off = __ldg(t.p_off + ji), jb.cig_off = __ldg(t.cig_off + ji);
	return jb;
}

#define KSWDPX_SMEM_PER_JOB 5120    /* pair layout (mmg_kswdpx.h): 14 B per target column + query + 16 */
#define KSWDPX_JOBS_PER_BLOCK 4     /* one warp per job */

__device__ __forceinline__ int ksw_seq4(const uint32_t *S, uint64_t i) { return __ldg(S + (i >> 3)) >> ((i & 7) << 2) & 0xf; } // mmg_seq4_get

__device__ __forceinline__ uint8_t ksw_qbase(const uint32_t *Q, const KswJobDev &jb, int j)
{ // element j of the query handed to ksw (align.c:691-697,721,761): a slice of qseq0[rev], possibly reversed
	const int idx = jb.reversed ? jb.q_start + jb.q_len - 1 - j : jb.q_start + j;
	if (!jb.q_rev) return (uint8_t)ksw_seq4(Q, jb.q_base + idx);
	const int c = ksw_seq4(Q, jb.q_base + (jb.q_readlen - 1 - idx)); // align.c:869
	return (uint8_t)(c < 4 ? 3 - c : 4);
}

__device__ __forceinline__ uint8_t ksw_tbase(const uint32_t *S, const KswJobDev &jb, int i)
{
	const int ti = jb.reversed ? jb.t_len - 1 - i : i;
	return (uint8_t)ksw_seq4(S, jb.t_base + ti); // mm_idx_getseq, index.c:152-162
}

__device__ __forceinline__ int ksw_ncol(int qlen, int tlen, int w)
{ // n_col_ of ksw2_extd2_sse.c:85-86
	if (w < 0) w = tlen > qlen ? tlen : qlen;
	int nc = qlen < tlen ? qlen : tlen;
	return ((nc < w + 1 ? nc : w + 1) + 15) / 16 + 1;
}

// Fast-form size classes: a job whose band never clips runs one-thread-per-job (k_ksw_tpj) in the first class it fits:
// min(qlen,tlen) <= mc (depth of the circular state window), tlen <= tc, qlen <= qc; nt = threads (jobs) per CTA.
#define KSW_N_FAST 3
#define KSW_CLS_LITERAL KSW_N_FAST            /* literal form, one warp per job */
#define KSW_CLS_BLOCK1 (KSW_N_FAST + 1)        /* literal form, one CTA per job: state too large for the warp kernel's shared-memory slot */
#define KSW_CLS_BLOCK2 (KSW_N_FAST + 2)        /* the same with up to KSWB_SMEM2 bytes of state */
#define KSW_CLS_WAVE (KSW_N_FAST + 3)          /* wavefront form: one warp per large job whose band never clips */
#define KSW_N_CLS (KSW_N_FAST + 4)
#define KSWB_WARPS 8                           /* warps of the CTA form */
#define KSWB_MAXG 2                            /* groups of four SSE blocks per warp and anti-diagonal: bands up to 64 blocks */
#define KSWB_SMEM1 (48 * 1024)
#define KSWB_SMEM2 (200 * 1024)
struct KswFastClass { int32_t mc, tc, qc, nt; };
struct KswFastTab { KswFastClass c[KSW_N_FAST]; };
static const KswFastTab ksw_ftab = {{{24, 56, 56, 128}, {48, 104, 104, 128}, {80, 160, 160, 64}}};
// per thread: the window of pair slots (mmg_kswfast2.h), the target bases, the query bases with a padding element at either end
// (the target bases are read from the packed reference when a cell enters: keeping them too cost a resident CTA per SM)
static inline size_t ksw_fast_smem(const KswFastClass &k) { return (size_t)k.nt * ((size_t)((k.mc >> 1) + 3) * 16 + (size_t)k.qc + 2); }

// wavefront form (k_ksw_wave below): geometry of its traceback rows and of its per-job arena
#define KW_S 8
#define KW_WARPS 4
MMG_HD size_t ksw_wave_tpad(int tlen) { return ((size_t)tlen + 7) & ~(size_t)7; }
MMG_HD size_t ksw_wave_p_bytes(int qlen, int tlen) { return ((size_t)qlen * ksw_wave_tpad(tlen) + 63) & ~(size_t)63; }
// arena per job: diag keys 8 B x (qlen + tlen) | last row H 4 B x tlen | last column H 4 B x qlen | edge of the last lane 16 B x qlen
MMG_HD size_t ksw_wave_mem_bytes(int qlen, int tlen) { return (((size_t)(qlen + tlen) * 8 + (size_t)tlen * 4 + (size_t)qlen * 4 + (size_t)qlen * 16) + 127) & ~(size_t)63; }

// per job: arena sizes, the scheduling key (form and size class, then shape so that the threads of a warp walk the same
// loops), and the true-band cell count
__global__ void k_ksw_prep(const mmg_ksw_job_t *__restrict__ jobs, int n, KswScore sc, KswFastTab ft, uint64_t *__restrict__ mem_sz,
                           uint64_t *__restrict__ p_sz, uint64_t *__restrict__ cig_sz, uint32_t *__restrict__ key, int32_t *__restrict__ idx,
                           unsigned long long *__restrict__ cells_total, uint32_t *__restrict__ cls_count, int force_block)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	unsigned long long cells = 0;
	int cls = -1;
	if (i <= n) {
		uint64_t m = 0, p = 0, c = 0; uint32_t k = (uint32_t)KSW_CLS_LITERAL << 28 | 63u;
		if (i < n) {
			const mmg_ksw_job_t j = jobs[i];
			const int qlen = j.q_len, tlen = j.t_len;
			cls = KSW_CLS_LITERAL;
			if (qlen > 0 && tlen > 0) {
				const KswGeom g = mmg_ksw_geom(qlen, tlen, sc.m, sc.mat, sc.q, sc.e, sc.q2, sc.e2, j.w);
				bool clips = false;
				// cells inside the band: sum over anti-diagonals of (en0 - st0 + 1)
				for (int r = 0; r < qlen + tlen - 1; ++r) {
					int st, en;
					clips |= mmg_ksw_band_clips(g, r);
					if (!mmg_ksw_band(g, r, &st, &en)) break;
					cells += (unsigned long long)(en - st + 1);
				}
				if (!g.bail && !clips && mmg_ksw_fast_ok(g)) {
					const int mn = qlen < tlen ? qlen : tlen;
					for (int q = KSW_N_FAST - 1; q >= 0; --q)
						if (mn <= ft.c[q].mc && tlen <= ft.c[q].tc && qlen <= ft.c[q].qc) cls = q;
				}
				c = (uint64_t)qlen + tlen + 2;
				if (cls == KSW_CLS_LITERAL && !g.bail && !clips && mmg_ksw_fast_ok(g) && (qlen < tlen ? qlen : tlen) >= 32 && qlen + tlen < 65000 && !(j.flag & MMG_EZ_APPROX_DROP)) {
					cls = KSW_CLS_WAVE; // too large for the thread-per-job classes: one warp, eight target columns per lane
					m = ksw_wave_mem_bytes(qlen, tlen);
					if (!(j.flag & MMG_EZ_SCORE_ONLY)) p = ksw_wave_p_bytes(qlen, tlen);
					const uint64_t est = (uint64_t)qlen * (uint64_t)tlen;
					k = (uint32_t)cls << 28 | (63u - (uint32_t)(63 - __clzll((long long)(est | 1))));
				} else if (cls == KSW_CLS_LITERAL) {
					const size_t md = mmg_kswdpx_mem_bytes(qlen, tlen);
					if (md > KSWDPX_SMEM_PER_JOB) m = (md + 63) & ~(size_t)63; // state beyond the warp kernel's slot goes to the arena
					if (!(j.flag & MMG_EZ_SCORE_ONLY)) p = ((uint64_t)(qlen + tlen - 1) * ksw_ncol(qlen, tlen, j.w) + 1) * 16;
					// or, when it fits, a CTA walks the job with the state in its own shared memory
					if (!g.bail && (md > KSWDPX_SMEM_PER_JOB || force_block) && md <= KSWB_SMEM2 && g.n_col_ <= 4 * KSWB_WARPS * KSWB_MAXG)
						cls = md <= KSWB_SMEM1 ? KSW_CLS_BLOCK1 : KSW_CLS_BLOCK2, m = 0;
					const uint64_t est = (uint64_t)(qlen + tlen) * (uint64_t)(qlen < tlen ? qlen : tlen);
					k = (uint32_t)cls << 28 | (63u - (uint32_t)(63 - __clzll((long long)(est | 1)))); // big jobs first
				} else {
					if (!(j.flag & MMG_EZ_SCORE_ONLY)) p = mmg_ksw_fast2_p_bytes(qlen, tlen);
					const uint32_t mode = (j.flag & MMG_EZ_SCORE_ONLY) ? 0u : (j.flag & MMG_EZ_RIGHT) ? 2u : 1u;
					k = (uint32_t)cls << 28 | mode << 26 | (uint32_t)(1023 - tlen) << 10 | (uint32_t)(1023 - qlen);
				}
			}
			idx[i] = i;
		}
		mem_sz[i] = m, p_sz[i] = p, cig_sz[i] = c, key[i] = k;
	}
	for (int q = 0; q < KSW_N_CLS; ++q) {
		const unsigned b = __ballot_sync(0xffffffffu, cls == q);
		unsigned long long cq = cls == q ? cells : 0;
		for (int d = 16; d >= 1; d >>= 1) cq += __shfl_xor_sync(0xffffffffu, cq, d);
		if ((threadIdx.x & 31) == 0 && b) { atomicAdd(&cls_count[q], (uint32_t)__popc(b)); atomicAdd(&cells_total[1 + q], cq); }
	}
	for (int d = 16; d >= 1; d >>= 1) cells += __shfl_xor_sync(0xffffffffu, cells, d);
	if ((threadIdx.x & 31) == 0 && cells) atomicAdd(cells_total, cells);
}

// ---- K4, literal form on 16x2 SIMD: one warp per job, two adjacent cells per lane (mmg_kswdpx.h) ------------------------
// The program of ksw2_extd2_sse.c:123-378 -- widened band, stale lanes, block carry-in, score refresh in 16-byte chunks from st0
// with its spill into sf[], exact-max tie order -- with four 16-lane SSE blocks side by side in the warp: lane L holds cells
// 2(L & 7) and 2(L & 7) + 1 of block st_ + 4 i + (L >> 3) in step i.  (Eight lanes per job, four jobs per warp, was measured no
// faster than one lane per SSE byte lane: jobs of different shapes in one warp diverge and issue one after the other.)
template <int kMode>
__device__ __forceinline__ void ksw_run_dpx(const KswGeom &g, const KswJobDev &jb, uint8_t *mem, int32_t *H, uint8_t *p, KswEz &ez, const int lane)
{
	const unsigned FULL = 0xffffffffu;
	const int tl16 = g.tlen_ * 16;
	uint4 *PK = reinterpret_cast<uint4*>(mem);
	int8_t *sm = reinterpret_cast<int8_t*>(mem), *s = sm + (size_t)tl16 * 8;
	const uint8_t *sf = reinterpret_cast<const uint8_t*>(s + tl16), *qr = sf + tl16;
	const int qlen = g.qlen, tlen = g.tlen, flag = jb.flag;
	const bool approx = (flag & MMG_EZ_APPROX_MAX) != 0;
	const int n1 = -g.q - g.e, n2 = -g.q2 - g.e2;
	const KswDpxConst cst = mmg_kswdpx_const<kMode>(g);
	const bool small_keys = mmg_ksw_fast_ok(g); // |H| * 2048 fits 32 bits and an anti-diagonal has at most 1023 cells
	int last_st = -1, last_en = -1;
	int32_t H0 = 0, last_H0_t = 0;
	for (int r = 0; r < qlen + tlen - 1; ++r) {
		int st0, en0;
		if (!mmg_ksw_band(g, r, &st0, &en0)) { ez.zdropped = 1; break; }
		const int st = st0 / 16 * 16, en = (en0 + 16) / 16 * 16 - 1;
		int x1, x21, v1;
		if (st > 0) {
			if (st - 1 >= last_st && st - 1 <= last_en) x1 = sm[KSWDPX_X(st - 1)], x21 = sm[KSWDPX_X2(st - 1)], v1 = sm[KSWDPX_V(st - 1)];
			else x1 = n1, x21 = n2, v1 = n1;
		} else {
			x1 = n1, x21 = n2;
			v1 = mmg_ksw_first_col(g, r);
		}
		if (en >= r && lane == 0) { // bytes of cell r; nobody reads them before the barrier below
			sm[KSWDPX_Y(r)] = (int8_t)n1, sm[KSWDPX_Y2(r)] = (int8_t)n2;
			sm[KSWDPX_U(r)] = (int8_t)mmg_ksw_first_col(g, r);
		}
		{ // scores, 16-byte chunks starting at st0 (ksw2_extd2_sse.c:158-172): two chunks per step
			const uint8_t *qrr = qr + (qlen - 1 - r);
			for (int t = st0 + (lane >> 4) * 16; t <= en0; t += 32) s[t + (lane & 15)] = mmg_ksw_score(g, sf[t + (lane & 15)], qrr[t + (lane & 15)]);
		}
		__syncwarp();
		const int st_ = st / 16, en_ = en / 16;
		uint32_t cin = mmg_kswdpx_carry_of(x1, v1, x21);
		for (int b0 = st_; b0 <= en_; b0 += 4) {
			const int blk = b0 + (lane >> 3), pi = blk * 8 + (lane & 7);
			const bool act = blk <= en_;
			KswPair o = {0u, 0u, 0u};
			uint32_t s2 = 0;
			if (act) { const uint4 w = PK[pi]; o.w0 = w.x, o.w1 = w.y, o.w2 = w.z; s2 = *reinterpret_cast<const uint16_t*>(s + 2 * pi); }
			const uint32_t cw = mmg_kswdpx_carry(o);
			uint32_t prev = __shfl_up_sync(FULL, cw, 1);
			if (lane == 0) prev = cin;
			cin = __shfl_sync(FULL, cw, 31);
			if (act) {
				uint32_t d2 = 0;
				const KswPair nw = mmg_kswdpx_pair<kMode>(cst, o, s2, prev, &d2);
				PK[pi] = make_uint4(nw.w0, nw.w1, nw.w2, 0u);
				if (kMode) *reinterpret_cast<uint16_t*>(p + ((size_t)r * g.n_col_ + (blk - st_)) * 16 + 2 * (lane & 7)) = (uint16_t)d2;
			}
		}
		__syncwarp();
		if (!approx) { // exact max over the band with the reference's tie order (ksw2_extd2_sse.c:315-358)
			int32_t max_H, max_t, H_en0;
			if (r > 0) {
				H_en0 = en0 > 0 ? H[en0 - 1] + sm[KSWDPX_U(en0)] : H[en0] + sm[KSWDPX_V(en0)];
				__syncwarp();
				if (small_keys) { // score and tie preference in one word (as mmg_ksw_fast_run): one warp-wide integer max
					const int en1k = (en0 - st0) / 4 * 4;
					int32_t best = H_en0 * 2048 + 2047; // the cell en0 wins every tie (ksw2_extd2_sse.c:319-349 starts from it)
					for (int t = st0 + lane; t < en0; t += 32) {
						const int32_t h = H[t] + sm[KSWDPX_V(t)];
						H[t] = h;
						const int k = t - st0, rk = k < en1k ? ((k & 3) << 8 | k >> 2) : (4 << 8 | (k - en1k));
						const int32_t key = h * 2048 + (2046 - rk);
						best = best > key ? best : key;
					}
					if (lane == 0) H[en0] = H_en0;
					best = __reduce_max_sync(FULL, best);
					const int32_t low = best & 2047;
					max_H = (best - low) >> 11; // exact: best - low is a multiple of 2048
					if (low == 2047) max_t = en0;
					else { const int32_t rk = 2046 - low; max_t = (rk >> 8) == 4 ? st0 + en1k + (rk & 255) : st0 + ((rk & 255) << 2) + (rk >> 8); }
				} else {
					int32_t bh = H_en0, bt = en0; uint32_t br = 0;
					for (int t = st0 + lane; t < en0; t += 32) {
						const int32_t h = H[t] + sm[KSWDPX_V(t)];
						H[t] = h;
						const uint32_t rk = mmg_ksw_max_rank(t, st0, en0);
						if (h > bh || (h == bh && rk < br)) bh = h, bt = t, br = rk;
					}
					if (lane == 0) H[en0] = H_en0;
#pragma unroll
					for (int d = 16; d >= 1; d >>= 1) {
						const int32_t oh = __shfl_xor_sync(FULL, bh, d), ot = __shfl_xor_sync(FULL, bt, d);
						const uint32_t orank = __shfl_xor_sync(FULL, br, d);
						if (oh > bh || (oh == bh && orank < br)) bh = oh, bt = ot, br = orank;
					}
					max_H = bh, max_t = bt;
				}
			} else {
				H_en0 = sm[KSWDPX_V(0)] - g.qe_pre;
				if (lane == 0) H[0] = H_en0;
				max_H = H_en0, max_t = 0;
			}
			__syncwarp();
			if (en0 == tlen - 1 && H_en0 > ez.mte) ez.mte = H_en0, ez.mte_q = r - en;
			if (r - st0 == qlen - 1) { const int32_t hs = H[st0]; if (hs > ez.mqe) ez.mqe = hs, ez.mqe_t = st0; }
			if (mmg_ksw_zdrop(&ez, max_H, r, max_t, jb.zdrop, g.e2)) break;
			if (r == qlen + tlen - 2 && en0 == tlen - 1) ez.score = H[tlen - 1];
		} else { // ksw2_extd2_sse.c:359-375
			if (r > 0) {
				if (last_H0_t >= st0 && last_H0_t <= en0 && last_H0_t + 1 >= st0 && last_H0_t + 1 <= en0) {
					const int32_t d0 = sm[KSWDPX_V(last_H0_t)], d1 = sm[KSWDPX_U(last_H0_t + 1)];
					if (d0 > d1) H0 += d0;
					else H0 += d1, ++last_H0_t;
				} else if (last_H0_t >= st0 && last_H0_t <= en0) {
					H0 += sm[KSWDPX_V(last_H0_t)];
				} else {
					++last_H0_t, H0 += sm[KSWDPX_U(last_H0_t)];
				}
			} else H0 = sm[KSWDPX_V(0)] - g.qe_pre, last_H0_t = 0;
			if ((flag & MMG_EZ_APPROX_DROP) && mmg_ksw_zdrop(&ez, H0, r, last_H0_t, jb.zdrop, g.e2)) break;
			if (r == qlen + tlen - 2 && en0 == tlen - 1) ez.score = H0;
		}
		last_st = st, last_en = en;
	}
}

__global__ void __launch_bounds__(32 * KSWDPX_JOBS_PER_BLOCK, 7) // 72 registers: seven CTAs per SM
k_ksw_dpx(KswTabs t, const int32_t *__restrict__ order, int n_jobs)
{
	extern __shared__ __align__(16) uint8_t smem[];
	const int grp = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int slot = blockIdx.x * KSWDPX_JOBS_PER_BLOCK + grp;
	if (slot >= n_jobs) return;
	const int ji = order[slot];
	const KswJobDev jb = ksw_job(t, ji);
	const KswScore sc = t.sc;
	const KswGeom g = mmg_ksw_geom(jb.q_len, jb.t_len, sc.m, sc.mat, sc.q, sc.e, sc.q2, sc.e2, jb.w);
	KswEz ez;
	mmg_ksw_reset(&ez);
	if (g.bail) { if (lane == 0) t.res[ji] = ez; return; }
	const int tl16 = g.tlen_ * 16;
	const size_t lane_bytes = (mmg_kswdpx_lane_bytes(jb.q_len, jb.t_len) + 15) & ~(size_t)15;
	uint8_t *mem = mmg_kswdpx_mem_bytes(jb.q_len, jb.t_len) <= KSWDPX_SMEM_PER_JOB ? smem + (size_t)grp * KSWDPX_SMEM_PER_JOB
	                                                                              : reinterpret_cast<uint8_t*>(t.gmem) + jb.mem_off; // arena slot sized in k_ksw_prep
	int32_t *H = reinterpret_cast<int32_t*>(mem + lane_bytes);
	{ // initial lane state (ksw2_extd2_sse.c:99-121) in the pair layout
		const uint32_t w1 = 0x01010101u * (uint8_t)(int8_t)(-g.q - g.e), w2 = 0x01010101u * (uint8_t)(int8_t)(-g.q2 - g.e2);
		uint4 *PK = reinterpret_cast<uint4*>(mem);
		for (int i = lane; i < tl16 / 2; i += 32) PK[i] = make_uint4(w1, w1, w2, 0u);
		int8_t *s = reinterpret_cast<int8_t*>(mem) + (size_t)tl16 * 8;
		for (int i = lane; i < tl16; i += 32) {
			s[i] = 0;                                                           // s (kcalloc)
			s[tl16 + i] = i < jb.t_len ? (int8_t)ksw_tbase(t.S, jb, i) : 0;     // sf
			H[i] = MMG_KSW_NEG_INF;
		}
		int8_t *qr = s + 2 * tl16;
		const int qn = g.qlen_ * 16 + 16;
		for (int i = lane; i < qn; i += 32) qr[i] = i < jb.q_len ? (int8_t)ksw_qbase(t.Q, jb, jb.q_len - 1 - i) : 0;
	}
	__syncwarp();
	uint8_t *p = t.gp + jb.p_off;
	const bool with_cigar = !(jb.flag & MMG_EZ_SCORE_ONLY);
	if (!with_cigar) ksw_run_dpx<0>(g, jb, mem, H, p, ez, lane);
	else if (!(jb.flag & MMG_EZ_RIGHT)) ksw_run_dpx<1>(g, jb, mem, H, p, ez, lane);
	else ksw_run_dpx<2>(g, jb, mem, H, p, ez, lane);
	__syncwarp();
	if (lane == 0) {
		int i0, j0;
		if (with_cigar && mmg_ksw_trace_start(g, jb.flag, jb.end_bonus, &ez, &i0, &j0))
			ez.n_cigar = mmg_ksw_backtrack(g, !!(jb.flag & MMG_EZ_REV_CIGAR), p, i0, j0, t.gcig + jb.cig_off);
		t.res[ji] = ez;
	}
}

// ---- K4, literal form, one CTA per job -----------------------------------------------------------------------------
// Long-read end extensions clip their band (w = 500 against thousands of bases) and carry tens of kilobytes of lane state: as
// one warp with the state in the HBM arena such a job took 16 dependent L2 round trips per anti-diagonal and a launch waited
// for its longest job (3.9 GCUPS).  Here the state sits in the CTA's shared memory and the SSE blocks of an anti-diagonal are
// spread over KSWB_WARPS warps: every lane takes the OLD state of its pair (and lane 0 of a warp its left neighbour's, which
// another warp owns) into registers, a barrier, then everybody writes.  The exact-max pass runs on all threads with one
// block-wide max over the packed (score, tie preference) keys.  Same program as ksw_run_dpx otherwise, four barriers per
// anti-diagonal.
template <int kMode>
__device__ __forceinline__ void ksw_run_dpx_block(const KswGeom &g, const KswJobDev &jb, uint8_t *mem, int32_t *H, uint8_t *p, KswEz &ez, int32_t *s_red)
{
	const unsigned FULL = 0xffffffffu;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, NT = 32 * KSWB_WARPS;
	const int tl16 = g.tlen_ * 16;
	uint4 *PK = reinterpret_cast<uint4*>(mem);
	int8_t *sm = reinterpret_cast<int8_t*>(mem), *s = sm + (size_t)tl16 * 8;
	const uint8_t *sf = reinterpret_cast<const uint8_t*>(s + tl16), *qr = sf + tl16;
	const int qlen = g.qlen, tlen = g.tlen, flag = jb.flag;
	const bool approx = (flag & MMG_EZ_APPROX_MAX) != 0;
	const int n1 = -g.q - g.e, n2 = -g.q2 - g.e2;
	const KswDpxConst cst = mmg_kswdpx_const<kMode>(g);
	const bool small_keys = mmg_ksw_fast_ok(g);
	int last_st = -1, last_en = -1;
	int32_t H0 = 0, last_H0_t = 0;
	for (int r = 0; r < qlen + tlen - 1; ++r) {
		int st0, en0;
		if (!mmg_ksw_band(g, r, &st0, &en0)) { ez.zdropped = 1; break; }
		const int st = st0 / 16 * 16, en = (en0 + 16) / 16 * 16 - 1;
		int x1, x21, v1;
		if (st > 0) {
			if (st - 1 >= last_st && st - 1 <= last_en) x1 = sm[KSWDPX_X(st - 1)], x21 = sm[KSWDPX_X2(st - 1)], v1 = sm[KSWDPX_V(st - 1)];
			else x1 = n1, x21 = n2, v1 = n1;
		} else {
			x1 = n1, x21 = n2;
			v1 = mmg_ksw_first_col(g, r);
		}
		// H of the cell the last one of this anti-diagonal derives from: nobody writes H before the max pass below
		const int32_t H_from = (!approx && r > 0) ? (en0 > 0 ? H[en0 - 1] : H[en0]) : 0;
		if (en >= r && tid == 0) {
			sm[KSWDPX_Y(r)] = (int8_t)n1, sm[KSWDPX_Y2(r)] = (int8_t)n2;
			sm[KSWDPX_U(r)] = (int8_t)mmg_ksw_first_col(g, r);
		}
		{ // scores, 16-byte chunks starting at st0 (ksw2_extd2_sse.c:158-172)
			const uint8_t *qrr = qr + (qlen - 1 - r);
			for (int t = st0 + (tid >> 4) * 16; t <= en0; t += NT) s[t + (tid & 15)] = mmg_ksw_score(g, sf[t + (tid & 15)], qrr[t + (tid & 15)]);
		}
		__syncthreads();
		const int st_ = st / 16, en_ = en / 16;
		KswPair o[KSWB_MAXG]; uint32_t s2[KSWB_MAXG], prev[KSWB_MAXG];
#pragma unroll
		for (int gi = 0; gi < KSWB_MAXG; ++gi) {
			const int b0 = st_ + 4 * (warp + gi * KSWB_WARPS), blk = b0 + (lane >> 3), pi = blk * 8 + (lane & 7);
			const bool act = blk <= en_;
			o[gi].w0 = o[gi].w1 = o[gi].w2 = 0u, s2[gi] = 0;
			if (act) { const uint4 w = PK[pi]; o[gi].w0 = w.x, o[gi].w1 = w.y, o[gi].w2 = w.z; s2[gi] = *reinterpret_cast<const uint16_t*>(s + 2 * pi); }
			uint32_t pv = __shfl_up_sync(FULL, mmg_kswdpx_carry(o[gi]), 1);
			if (lane == 0) {
				if (b0 == st_) pv = mmg_kswdpx_carry_of(x1, v1, x21);
				else if (act) { const uint4 w = PK[pi - 1]; const KswPair ol = {w.x, w.y, w.z}; pv = mmg_kswdpx_carry(ol); }
			}
			prev[gi] = pv;
		}
		__syncthreads(); // every old state this anti-diagonal reads is in registers
#pragma unroll
		for (int gi = 0; gi < KSWB_MAXG; ++gi) {
			const int b0 = st_ + 4 * (warp + gi * KSWB_WARPS), blk = b0 + (lane >> 3), pi = blk * 8 + (lane & 7);
			if (blk <= en_) {
				uint32_t d2 = 0;
				const KswPair nw = mmg_kswdpx_pair<kMode>(cst, o[gi], s2[gi], prev[gi], &d2);
				PK[pi] = make_uint4(nw.w0, nw.w1, nw.w2, 0u);
				if (kMode) *reinterpret_cast<uint16_t*>(p + ((size_t)r * g.n_col_ + (blk - st_)) * 16 + 2 * (lane & 7)) = (uint16_t)d2;
			}
		}
		__syncthreads();
		if (!approx) { // exact max over the band with the reference's tie order (ksw2_extd2_sse.c:315-358)
			int32_t max_H, max_t, H_en0;
			if (r > 0) {
				H_en0 = H_from + (en0 > 0 ? sm[KSWDPX_U(en0)] : sm[KSWDPX_V(en0)]);
				if (small_keys) {
					const int en1k = (en0 - st0) / 4 * 4;
					int32_t best = H_en0 * 2048 + 2047;
					for (int t = st0 + tid; t < en0; t += NT) {
						const int32_t h = H[t] + sm[KSWDPX_V(t)];
						H[t] = h;
						const int k = t - st0, rk = k < en1k ? ((k & 3) << 8 | k >> 2) : (4 << 8 | (k - en1k));
						const int32_t key = h * 2048 + (2046 - rk);
						best = best > key ? best : key;
					}
					if (tid == 0) H[en0] = H_en0;
					best = __reduce_max_sync(FULL, best);
					if (lane == 0) s_red[warp] = best;
					__syncthreads();
#pragma unroll
					for (int q = 0; q < KSWB_WARPS; ++q) { const int32_t v = s_red[q]; best = best > v ? best : v; }
					const int32_t low = best & 2047;
					max_H = (best - low) >> 11;
					if (low == 2047) max_t = en0;
					else { const int32_t rk = 2046 - low; max_t = (rk >> 8) == 4 ? st0 + en1k + (rk & 255) : st0 + ((rk & 255) << 2) + (rk >> 8); }
				} else {
					int32_t bh = H_en0, bt = en0; uint32_t br = 0;
					for (int t = st0 + tid; t < en0; t += NT) {
						const int32_t h = H[t] + sm[KSWDPX_V(t)];
						H[t] = h;
						const uint32_t rk = mmg_ksw_max_rank(t, st0, en0);
						if (h > bh || (h == bh && rk < br)) bh = h, bt = t, br = rk;
					}
					if (tid == 0) H[en0] = H_en0;
#pragma unroll
					for (int d = 16; d >= 1; d >>= 1) {
						const int32_t oh = __shfl_xor_sync(FULL, bh, d), ot = __shfl_xor_sync(FULL, bt, d);
						const uint32_t orank = __shfl_xor_sync(FULL, br, d);
						if (oh > bh || (oh == bh && orank < br)) bh = oh, bt = ot, br = orank;
					}
					if (lane == 0) s_red[warp] = bh, s_red[KSWB_WARPS + warp] = bt, s_red[2 * KSWB_WARPS + warp] = (int32_t)br;
					__syncthreads();
#pragma unroll
					for (int q = 0; q < KSWB_WARPS; ++q) {
						const int32_t oh = s_red[q], ot = s_red[KSWB_WARPS + q];
						const uint32_t orank = (uint32_t)s_red[2 * KSWB_WARPS + q];
						if (oh > bh || (oh == bh && orank < br)) bh = oh, bt = ot, br = orank;
					}
					max_H = bh, max_t = bt;
				}
			} else {
				H_en0 = sm[KSWDPX_V(0)] - g.qe_pre;
				if (tid == 0) H[0] = H_en0;
				__syncthreads();
				max_H = H_en0, max_t = 0;
			}
			if (en0 == tlen - 1 && H_en0 > ez.mte) ez.mte = H_en0, ez.mte_q = r - en;
			if (r - st0 == qlen - 1) { const int32_t hs = H[st0]; if (hs > ez.mqe) ez.mqe = hs, ez.mqe_t = st0; }
			const bool stop = mmg_ksw_zdrop(&ez, max_H, r, max_t, jb.zdrop, g.e2);
			if (stop) break;
			if (r == qlen + tlen - 2 && en0 == tlen - 1) ez.score = H[tlen - 1];
			// no barrier here: the next anti-diagonal writes H and s_red only behind its own three barriers
		} else { // ksw2_extd2_sse.c:359-375
			if (r > 0) {
				if (last_H0_t >= st0 && last_H0_t <= en0 && last_H0_t + 1 >= st0 && last_H0_t + 1 <= en0) {
					const int32_t d0 = sm[KSWDPX_V(last_H0_t)], d1 = sm[KSWDPX_U(last_H0_t + 1)];
					if (d0 > d1) H0 += d0;
					else H0 += d1, ++last_H0_t;
				} else if (last_H0_t >= st0 && last_H0_t <= en0) {
					H0 += sm[KSWDPX_V(last_H0_t)];
				} else {
					++last_H0_t, H0 += sm[KSWDPX_U(last_H0_t)];
				}
			} else H0 = sm[KSWDPX_V(0)] - g.qe_pre, last_H0_t = 0;
			if ((flag & MMG_EZ_APPROX_DROP) && mmg_ksw_zdrop(&ez, H0, r, last_H0_t, jb.zdrop, g.e2)) break;
			if (r == qlen + tlen - 2 && en0 == tlen - 1) ez.score = H0;
		}
		last_st = st, last_en = en;
	}
}

__global__ void __launch_bounds__(32 * KSWB_WARPS)
k_ksw_dpx_block(KswTabs t, const int32_t *__restrict__ order, int n_jobs)
{
	extern __shared__ __align__(16) uint8_t smem[];
	__shared__ int32_t s_red[3 * KSWB_WARPS];
	const int tid = threadIdx.x, NT = 32 * KSWB_WARPS;
	const int ji = order[blockIdx.x];
	const KswJobDev jb = ksw_job(t, ji);
	const KswScore sc = t.sc;
	const KswGeom g = mmg_ksw_geom(jb.q_len, jb.t_len, sc.m, sc.mat, sc.q, sc.e, sc.q2, sc.e2, jb.w);
	KswEz ez;
	mmg_ksw_reset(&ez);
	const int tl16 = g.tlen_ * 16;
	const size_t lane_bytes = (mmg_kswdpx_lane_bytes(jb.q_len, jb.t_len) + 15) & ~(size_t)15;
	uint8_t *mem = smem;
	int32_t *H = reinterpret_cast<int32_t*>(mem + lane_bytes);
	{ // initial lane state (ksw2_extd2_sse.c:99-121) in the pair layout
		const uint32_t w1 = 0x01010101u * (uint8_t)(int8_t)(-g.q - g.e), w2 = 0x01010101u * (uint8_t)(int8_t)(-g.q2 - g.e2);
		uint4 *PK = reinterpret_cast<uint4*>(mem);
		for (int i = tid; i < tl16 / 2; i += NT) PK[i] = make_uint4(w1, w1, w2, 0u);
		int8_t *s = reinterpret_cast<int8_t*>(mem) + (size_t)tl16 * 8;
		for (int i = tid; i < tl16; i += NT) {
			s[i] = 0;
			s[tl16 + i] = i < jb.t_len ? (int8_t)ksw_tbase(t.S, jb, i) : 0;
			H[i] = MMG_KSW_NEG_INF;
		}
		int8_t *qr = s + 2 * tl16;
		const int qn = g.qlen_ * 16 + 16;
		for (int i = tid; i < qn; i += NT) qr[i] = i < jb.q_len ? (int8_t)ksw_qbase(t.Q, jb, jb.q_len - 1 - i) : 0;
	}
	__syncthreads();
	uint8_t *p = t.gp + jb.p_off;
	const bool with_cigar = !(jb.flag & MMG_EZ_SCORE_ONLY);
	if (!with_cigar) ksw_run_dpx_block<0>(g, jb, mem, H, p, ez, s_red);
	else if (!(jb.flag & MMG_EZ_RIGHT)) ksw_run_dpx_block<1>(g, jb, mem, H, p, ez, s_red);
	else ksw_run_dpx_block<2>(g, jb, mem, H, p, ez, s_red);
	__syncthreads();
	if (tid == 0) {
		int i0, j0;
		if (with_cigar && mmg_ksw_trace_start(g, jb.flag, jb.end_bonus, &ez, &i0, &j0))
			ez.n_cigar = mmg_ksw_backtrack(g, !!(jb.flag & MMG_EZ_REV_CIGAR), p, i0, j0, t.gcig + jb.cig_off);
		t.res[ji] = ez;
	}
}

// K4, fast form: one thread per job whose band never clips, two cells per instruction (mmg_ksw_fast2, mmg_kswfast2.h).  The
// threads of a CTA interleave their per-job arrays in shared memory ([element][thread]): a warp's accesses fall on consecutive
// banks (16-byte pair slots: one LDS.128 / STS.128 per two cells).
__global__ void __launch_bounds__(128)
k_ksw_tpj(KswTabs t, const int32_t *__restrict__ order, int n_jobs, KswFastClass fc)
{
	extern __shared__ __align__(16) uint8_t smem[];
	const int NT = blockDim.x, tid = threadIdx.x;
	const int slot = blockIdx.x * NT + tid;
	if (slot >= n_jobs) return;
	KswSlot *st = reinterpret_cast<KswSlot*>(smem) + tid;
	uint8_t *qb = smem + (size_t)((fc.mc >> 1) + 3) * NT * 16 + tid + NT; // qb[-1] and qb[qlen] are padding
	const int ji = order[slot];
	const mmg_ksw_job_t hj = ksw_ldg_job(t.jobs + ji);
	const int qlen = hj.q_len, tlen = hj.t_len;
	const KswScore sc = t.sc;
	const KswGeom g = mmg_ksw_geom(qlen, tlen, sc.m, sc.mat, sc.q, sc.e, sc.q2, sc.e2, hj.w);
	// target slice of S (mm_idx_getseq, index.c:152-162), reversed for left extensions (align.c:694-695): read base by base as cells enter
	const uint64_t t_a0 = __ldg(t.ref_off + hj.rid) + (uint64_t)hj.t_start;
	const bool t_rev = hj.reversed != 0;
	auto tbase = [&](int i) -> uint32_t { const uint64_t a = t_a0 + (uint64_t)(t_rev ? tlen - 1 - i : i); return (uint32_t)ksw_seq4(t.S, a); };
	{ // query slice of qseq0[q_rev] (align.c:865-870)
		const uint64_t qbase = __ldg(t.q_off + hj.seq_id);
		const int rl = __ldg(t.read_len + hj.seq_id);
		const int lo = hj.q_rev ? rl - hj.q_start - qlen : hj.q_start, hi = lo + qlen;
		for (int wp = lo >> 3; wp <= (hi - 1) >> 3; ++wp) {
			const uint32_t word = __ldg(t.Q + (qbase >> 3) + wp); // reads start on 8-base boundaries
#pragma unroll
			for (int k = 0; k < 8; ++k) {
				const int pos = wp * 8 + k;
				if (pos >= lo && pos < hi) {
					const int c = (int)(word >> (4 * k) & 0xf);
					const int idx = hj.q_rev ? rl - 1 - pos : pos;
					const int j = hj.reversed ? hj.q_start + qlen - 1 - idx : idx - hj.q_start;
					qb[(size_t)j * NT] = (uint8_t)(hj.q_rev ? (c < 4 ? 3 - c : 4) : c);
				}
			}
		}
	}
	qb[-(ptrdiff_t)NT] = 4, qb[(size_t)qlen * NT] = 4;
	KswEz ez;
	mmg_ksw_fast2(g, hj.flag, hj.zdrop, hj.end_bonus, st, tbase, qb - NT, NT, reinterpret_cast<uint32_t*>(t.gp + __ldg(t.p_off + ji)), &ez, t.gcig + __ldg(t.cig_off + ji));
	t.res[ji] = ez;
}


// ---- K4, wavefront form: one warp per large job whose band never clips ------------------------------------------
// Cell (t, j) of the difference recurrence needs x, v, x2 of (t-1, j) and y, u, y2 of (t, j-1) -- nothing else (the
// anti-diagonal order of the SSE program is one valid schedule among many once no stale lane can be read, see
// mmg_ksw_fast_run).  Each lane owns KW_S consecutive target columns and keeps their (u, y, y2) in registers; lane l works
// on query row j = step - l, receives the (x, v, x2, H) of its left neighbour's last column by one shuffle per step and
// sweeps its columns with the carry in registers.  Targets wider than 32 * KW_S columns take several passes; the last
// lane's edge values go through a per-row array.  What the reference derives per anti-diagonal (first-max with its tie
// order, z-drop, mqe, mte) is rebuilt after the sweep from a per-diagonal atomicMax key, the last row and the last column.

template <int kMode>
__device__ __forceinline__ void ksw_wave_sweep(const KswGeom &g, const KswJobDev &jb, const uint32_t *__restrict__ Q, const uint32_t *__restrict__ S,
                                               uint8_t *__restrict__ p2, unsigned long long *__restrict__ diag, int32_t *__restrict__ hrow,
                                               int32_t *__restrict__ hcol, int4 *__restrict__ edge, const bool exact, const int lane)
{
	const unsigned FULL = 0xffffffffu;
	const int qlen = g.qlen, tlen = g.tlen;
	const int32_t n1 = -g.q - g.e, n2 = -g.q2 - g.e2;
	const size_t tpad = ksw_wave_tpad(tlen);
	const int n_pass = (tlen + 32 * KW_S - 1) / (32 * KW_S);
	for (int pass = 0; pass < n_pass; ++pass) {
		const int a = pass * 32 * KW_S + lane * KW_S; // first column of this lane
		const int nc = tlen - a < 0 ? 0 : tlen - a > KW_S ? KW_S : tlen - a;
		int32_t tb[KW_S], cu[KW_S], cy[KW_S], cy2[KW_S];
#pragma unroll
		for (int k = 0; k < KW_S; ++k) {
			tb[k] = k < nc ? (int32_t)ksw_tbase(S, jb, a + k) : 4;
			cu[k] = mmg_ksw_first_col(g, a + k), cy[k] = n1, cy2[k] = n2; // the row above row 0: first-row boundary (ksw2_extd2_sse.c:152-156)
		}
		int32_t ex = n1, ev = n1, ex2 = n2, eH = 0; // what this lane hands to the next one: its last column of the row it just did
		int32_t hm1 = 0;                              // H of the column left of column 0 (lane 0 of the first pass)
		for (int st = 0; st < qlen + 31; ++st) {
			const int j = st - lane;
			int32_t lx = __shfl_up_sync(FULL, ex, 1), lv = __shfl_up_sync(FULL, ev, 1), lx2 = __shfl_up_sync(FULL, ex2, 1), lH = __shfl_up_sync(FULL, eH, 1);
			if (j < 0 || j >= qlen || nc == 0) continue;
			if (lane == 0) {
				if (pass == 0) {
					const int32_t fc = mmg_ksw_first_col(g, j);
					hm1 = j == 0 ? -g.qe_pre : hm1 + fc; // H(-1, j): the first-column boundary, see the derivation in DESIGN.md section 4
					lx = n1, lx2 = n2, lv = fc, lH = hm1;
				} else { const int4 e4 = edge[j]; lx = e4.x, lv = e4.y, lx2 = e4.z, lH = e4.w; }
			}
			const uint32_t qb = ksw_qbase(Q, jb, j);
			int32_t cx = lx, cv = lv, cx2 = lx2, H = lH;
			unsigned long long dw = 0;
#pragma unroll
			for (int k = 0; k < KW_S; ++k)
				if (k < nc) {
					const uint32_t tbase = (uint32_t)tb[k];
					int32_t sc = tbase == qb ? g.sc_mch : g.sc_mis;
					if ((tbase | qb) & 4) sc = g.sc_N;
					const KswCell32 c = mmg_ksw_cell32<kMode>(g, sc, cx, cv, cu[k], cy[k], cx2, cy2[k]);
					cu[k] = c.u, cy[k] = c.y, cy2[k] = c.y2;
					cx = c.x, cv = c.v, cx2 = c.x2;
					H += c.u;
					if (kMode) dw |= (unsigned long long)c.d << (8 * k);
					if (exact) {
						const int t = a + k, r = t + j;
						const int st0 = r - qlen + 1 > 0 ? r - qlen + 1 : 0, en0 = r < tlen - 1 ? r : tlen - 1;
						uint32_t pref = 0xffffu;
						if (t != en0) {
							const int d = t - st0, en1k = (en0 - st0) / 4 * 4;
							const uint32_t rk = d < en1k ? ((uint32_t)(d & 3) << 13 | (uint32_t)(d >> 2)) : (4u << 13 | (uint32_t)(d - en1k));
							pref = 0xfffeu - rk;
						}
						atomicMax(&diag[r], (unsigned long long)(uint32_t)(H + 0x40000000) << 32 | (unsigned long long)pref << 16 | (unsigned long long)(uint32_t)t);
						if (j == qlen - 1) hrow[t] = H;
					}
					if (a + k == tlen - 1) hcol[j] = H; // last column: mte in exact mode, and its last entry is the global score in every mode
				}
			if (kMode) *reinterpret_cast<unsigned long long*>(p2 + (size_t)j * tpad + a) = dw;
			ex = cx, ev = cv, ex2 = cx2, eH = H;
			if (lane == 31 && pass + 1 < n_pass) edge[j] = make_int4(ex, ev, ex2, eH);
		}
		__syncwarp();
	}
}

MMG_HDN inline int ksw_wave_backtrack(const KswGeom &g, int is_rev, const uint8_t *p2, size_t tpad, int i0, int j0, uint32_t *cigar)
{ // ksw_backtrack (ksw2.h:119-151) over rows of query positions; the walk cannot leave the matrix
	int n = 0, i = i0, j = j0, state = 0;
#define MMG_PUSH(op, len) do { if (n == 0 || (uint32_t)(op) != (cigar[n - 1] & 0xf)) cigar[n++] = (uint32_t)(len) << 4 | (uint32_t)(op); else cigar[n - 1] += (uint32_t)(len) << 4; } while (0)
	while (i >= 0 && j >= 0) {
		const uint32_t tmp = p2[(size_t)j * tpad + i];
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

__global__ void __launch_bounds__(32 * KW_WARPS)
k_ksw_wave(KswTabs t, const int32_t *__restrict__ order, int n_jobs)
{
	const int lane = threadIdx.x & 31, slot = blockIdx.x * KW_WARPS + (threadIdx.x >> 5);
	if (slot >= n_jobs) return;
	const int ji = order[slot];
	const KswJobDev jb = ksw_job(t, ji);
	const KswScore sc = t.sc;
	const KswGeom g = mmg_ksw_geom(jb.q_len, jb.t_len, sc.m, sc.mat, sc.q, sc.e, sc.q2, sc.e2, jb.w);
	const int qlen = g.qlen, tlen = g.tlen, R = qlen + tlen - 1;
	unsigned long long *diag = reinterpret_cast<unsigned long long*>(t.gmem + jb.mem_off);
	int32_t *hrow = reinterpret_cast<int32_t*>(diag + (qlen + tlen)), *hcol = hrow + tlen;
	int4 *edge = reinterpret_cast<int4*>((reinterpret_cast<size_t>(hcol + qlen) + 15) & ~(size_t)15);
	uint8_t *p2 = t.gp + jb.p_off;
	const bool with_cigar = !(jb.flag & MMG_EZ_SCORE_ONLY), exact = !(jb.flag & MMG_EZ_APPROX_MAX);
	if (exact) for (int r = lane; r < R; r += 32) diag[r] = 0;
	__syncwarp();
	if (!with_cigar) ksw_wave_sweep<0>(g, jb, t.Q, t.S, p2, diag, hrow, hcol, edge, exact, lane);
	else if (!(jb.flag & MMG_EZ_RIGHT)) ksw_wave_sweep<1>(g, jb, t.Q, t.S, p2, diag, hrow, hcol, edge, exact, lane);
	else ksw_wave_sweep<2>(g, jb, t.Q, t.S, p2, diag, hrow, hcol, edge, exact, lane);
	__threadfence_block();
	__syncwarp();
	if (lane != 0) return;
	KswEz ez;
	mmg_ksw_reset(&ez);
	if (exact) { // the per-diagonal bookkeeping of ksw2_extd2_sse.c:350-358, in diagonal order
		for (int r = 0; r < R; ++r) {
			const int st0 = r - qlen + 1 > 0 ? r - qlen + 1 : 0, en0 = r < tlen - 1 ? r : tlen - 1;
			const unsigned long long key = diag[r];
			const int32_t max_H = (int32_t)(uint32_t)(key >> 32) - 0x40000000, max_t = (int32_t)(key & 0xffff);
			if (en0 == tlen - 1) { const int32_t H_en0 = hcol[r - (tlen - 1)]; if (H_en0 > ez.mte) ez.mte = H_en0, ez.mte_q = r - ((en0 + 16) / 16 * 16 - 1); }
			if (r - st0 == qlen - 1) { const int32_t hs = hrow[st0]; if (hs > ez.mqe) ez.mqe = hs, ez.mqe_t = st0; }
			if (mmg_ksw_zdrop(&ez, max_H, r, max_t, jb.zdrop, g.e2)) break;
			if (r == R - 1 && en0 == tlen - 1) ez.score = hcol[qlen - 1];
		}
	} else { // approximate mode without APPROX_DROP (ksw2_extd2_sse.c:359-375): H0 telescopes along a path of neighbouring cells that
		// ends in the corner, so only H of the corner cell is observable
		ez.score = hcol[qlen - 1];
	}
	int i0, j0;
	if (with_cigar && mmg_ksw_trace_start(g, jb.flag, jb.end_bonus, &ez, &i0, &j0))
		ez.n_cigar = ksw_wave_backtrack(g, !!(jb.flag & MMG_EZ_REV_CIGAR), p2, ksw_wave_tpad(tlen), i0, j0, t.gcig + __ldg(t.cig_off + ji)); // read here: not held across the sweep
	t.res[ji] = ez;
}

__global__ void k_res_ncig(int n_jobs, const KswEz *__restrict__ res, int32_t *__restrict__ ncig)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n_jobs) ncig[i] = res[i].n_cigar;
	else if (i == n_jobs) ncig[i] = 0;
}

// dense results: {ez, cigar offset} per job in submission order, CIGARs packed back to back
__global__ void k_cig_gather(int n_jobs, const KswEz *__restrict__ res, const int64_t *__restrict__ off, const uint64_t *__restrict__ cig_off,
                             const uint32_t *__restrict__ gcig, KswResDev *__restrict__ out_res, uint32_t *__restrict__ out_cig)
{
	const int ji = blockIdx.x * blockDim.x + threadIdx.x;
	if (ji >= n_jobs) return;
	const KswEz ez = res[ji];
	const int64_t o = off[ji];
	const uint32_t *src = gcig + cig_off[ji];
	for (int i = 0; i < ez.n_cigar; ++i) out_cig[o + i] = src[i];
	KswResDev r; r.ez = ez, r.cigar_off = (uint64_t)o;
	out_res[ji] = r;
}

template <class T> static int scan_excl(mmg_ctx_t *c, const T *d_in, int64_t *d_out, int n)
{
	size_t tmp = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tmp, d_in, d_out, n, c->stream);
	MMG_TRY(c->d_cub.ensure(tmp));
	MMG_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, d_in, d_out, n, c->stream));
	++c->launches;
	return MMG_OK;
}

// the dynamic shared memory the K4 kernels launch with, allowed on the current device (mmg_init, once per context)
int mmg_ksw_set_smem_attrs()
{
	size_t mx = 0;
	for (int q = 0; q < KSW_N_FAST; ++q) mx = std::max(mx, ksw_fast_smem(ksw_ftab.c[q]));
	MMG_CUDA(cudaFuncSetAttribute(k_ksw_tpj, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mx));
	MMG_CUDA(cudaFuncSetAttribute(k_ksw_dpx, cudaFuncAttributeMaxDynamicSharedMemorySize, KSWDPX_SMEM_PER_JOB * KSWDPX_JOBS_PER_BLOCK));
	MMG_CUDA(cudaFuncSetAttribute(k_ksw_dpx_block, cudaFuncAttributeMaxDynamicSharedMemorySize, KSWB_SMEM2));
	return MMG_OK;
}

#define KSW_SPLIT 1 // ksw_launch: the jobs' DP state exceeds the budget given; nothing was run

// d_jobs: n jobs already on the device.  q_off/read_len/ref_off: device tables the jobs index into.  budget: device bytes the
// jobs' DP state may take (0: any); above it, and with more than one job, KSW_SPLIT is returned instead.
static int ksw_launch(mmg_ctx_t *c, const mmg_ksw_job_t *d_jobs, int n, const uint32_t *d_Q, const uint32_t *d_S, const uint64_t *d_q_off,
                      const int32_t *d_read_len, const uint64_t *d_ref_off, const KswScore &sc, mmg_ksw_res_t *res, const uint32_t **cigars,
                      double *kernel_ms, uint64_t *cells, bool to_host = true, size_t budget = 0)
{
	// scratch layout in k_cig_off: mem_sz | p_sz | cig_sz (u64, n+1 each) | their scans (i64, n+1 each) | ncig scan (i64, n+1) | cells, class counts |
	// key, key2 (u32) | idx, order (i32) | ncig (i32, n+1)
	const size_t n1 = (size_t)n + 1;
	MMG_TRY(c->k_cig_off.ensure(n1 * (7 * 8 + 5 * 4) + 256));
	uint64_t *mem_sz = c->k_cig_off.as<uint64_t>(), *p_sz = mem_sz + n1, *cig_sz = p_sz + n1;
	int64_t *mem_off = reinterpret_cast<int64_t*>(cig_sz + n1), *p_off = mem_off + n1, *cg_off = p_off + n1, *nc_off = cg_off + n1;
	unsigned long long *d_cells = reinterpret_cast<unsigned long long*>(nc_off + n1);
	uint32_t *d_cls = reinterpret_cast<uint32_t*>(d_cells + 2 + KSW_N_CLS); // d_cells: total, then per class; d_cls: KSW_N_CLS job counters
	uint32_t *key = d_cls + 8, *key2 = key + n1;
	int32_t *idx = reinterpret_cast<int32_t*>(key2 + n1), *order = idx + n1, *ncig = order + n1;
	static const bool force_block = getenv("MMG_KSW_FORCE_BLOCK") != nullptr; // test aid: every literal job the CTA form can take goes through it
	MMG_CUDA(cudaMemsetAsync(d_cells, 0, (2 + KSW_N_CLS) * 8 + 32, c->stream));
	MMG_LAUNCH(c, k_ksw_prep, mmg_blocks(n1, 128), 128, 0, d_jobs, n, sc, ksw_ftab, mem_sz, p_sz, cig_sz, key, idx, d_cells, d_cls, force_block ? 1 : 0);
	MMG_TRY(scan_excl(c, mem_sz, mem_off, (int)n1));
	MMG_TRY(scan_excl(c, p_sz, p_off, (int)n1));
	MMG_TRY(scan_excl(c, cig_sz, cg_off, (int)n1));
	{ // stable sort of job indices by scheduling key
		size_t tmp = 0;
		cub::DeviceRadixSort::SortPairs(nullptr, tmp, key, key2, idx, order, n, 0, 31, c->stream);
		MMG_TRY(c->d_cub.ensure(tmp));
		MMG_TIMED(c, "cub_radix_sort(dp jobs)", cub::DeviceRadixSort::SortPairs(c->d_cub.p, tmp, key, key2, idx, order, n, 0, 31, c->stream));
	}
	int64_t tot[3]; unsigned long long h_cells[1 + KSW_N_CLS]; uint32_t h_cls[KSW_N_CLS];
	MMG_D2H(c, &tot[0], mem_off + n, 8); MMG_D2H(c, &tot[1], p_off + n, 8); MMG_D2H(c, &tot[2], cg_off + n, 8);
	MMG_D2H(c, h_cells, d_cells, sizeof(h_cells)); MMG_D2H(c, h_cls, d_cls, sizeof(h_cls));
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	if (budget && n > 1 && (size_t)(tot[0] + tot[1] + tot[2] * 4) > budget) return KSW_SPLIT;
	if (cells) *cells = h_cells[0];
	c->k_last_jobs_literal = h_cls[KSW_CLS_LITERAL] + h_cls[KSW_CLS_BLOCK1] + h_cls[KSW_CLS_BLOCK2]; // the wavefront form counts as a fast form
	c->k_last_cells_literal = h_cells[1 + KSW_CLS_LITERAL] + h_cells[1 + KSW_CLS_BLOCK1] + h_cells[1 + KSW_CLS_BLOCK2];
	c->k_last_jobs_fast = (uint64_t)n - c->k_last_jobs_literal, c->k_last_cells_fast = h_cells[0] - c->k_last_cells_literal;
	if (getenv("MMG_KSW_DEBUG")) {
		fprintf(stderr, "[mmg_ksw] %d jobs, %llu cells:", n, h_cells[0]);
		for (int q = 0; q < KSW_N_CLS; ++q) fprintf(stderr, " class %d: %u jobs %llu cells;", q, h_cls[q], h_cells[1 + q]);
		fprintf(stderr, " p %ld B, mem %ld B\n", (long)tot[1], (long)tot[0]);
	}
	MMG_TRY(c->k_mem.ensure((size_t)tot[0] + 64));
	MMG_TRY(c->k_p.ensure((size_t)tot[1] + 64));
	MMG_TRY(c->k_cig.ensure(((size_t)tot[2] + 4) * 4));
	MMG_TRY(c->k_res.ensure(((n1 * sizeof(KswEz) + 15) & ~(size_t)15) + n1 * sizeof(KswResDev)));
	KswEz *d_ez = c->k_res.as<KswEz>();
	KswResDev *d_res = reinterpret_cast<KswResDev*>(c->k_res.as<uint8_t>() + ((n1 * sizeof(KswEz) + 15) & ~(size_t)15));
	KswTabs t;
	t.jobs = d_jobs, t.Q = d_Q, t.S = d_S, t.q_off = d_q_off, t.ref_off = d_ref_off, t.read_len = d_read_len;
	t.mem_off = reinterpret_cast<const uint64_t*>(mem_off), t.p_off = reinterpret_cast<const uint64_t*>(p_off), t.cig_off = reinterpret_cast<const uint64_t*>(cg_off);
	t.gmem = c->k_mem.as<int8_t>(), t.gp = c->k_p.as<uint8_t>(), t.gcig = c->k_cig.as<uint32_t>(), t.res = d_ez, t.sc = sc;
	MMG_CUDA(cudaEventRecord(c->ev[0], c->stream));
	uint32_t first = 0; // the classes are consecutive in the scheduling order
	for (int q = 0; q < KSW_N_FAST; ++q) {
		if (h_cls[q])
			MMG_LAUNCH(c, k_ksw_tpj, mmg_blocks(h_cls[q], ksw_ftab.c[q].nt), ksw_ftab.c[q].nt, ksw_fast_smem(ksw_ftab.c[q]), t, order + first, (int)h_cls[q], ksw_ftab.c[q]);
		first += h_cls[q];
	}
	if (h_cls[KSW_CLS_LITERAL])
		MMG_LAUNCH(c, k_ksw_dpx, mmg_blocks(h_cls[KSW_CLS_LITERAL], KSWDPX_JOBS_PER_BLOCK), 32 * KSWDPX_JOBS_PER_BLOCK, KSWDPX_SMEM_PER_JOB * KSWDPX_JOBS_PER_BLOCK,
		           t, order + first, (int)h_cls[KSW_CLS_LITERAL]);
	first += h_cls[KSW_CLS_LITERAL];
	for (int q = KSW_CLS_BLOCK1; q <= KSW_CLS_BLOCK2; ++q) { // literal jobs with more state than a warp's slot: a CTA each, state in its shared memory
		if (h_cls[q])
			MMG_LAUNCH(c, k_ksw_dpx_block, h_cls[q], 32 * KSWB_WARPS, q == KSW_CLS_BLOCK1 ? KSWB_SMEM1 : KSWB_SMEM2, t, order + first, (int)h_cls[q]);
		first += h_cls[q];
	}
	if (h_cls[KSW_CLS_WAVE])
		MMG_LAUNCH(c, k_ksw_wave, mmg_blocks(h_cls[KSW_CLS_WAVE], KW_WARPS), 32 * KW_WARPS, 0, t, order + first, (int)h_cls[KSW_CLS_WAVE]);
	MMG_CUDA(cudaEventRecord(c->ev[1], c->stream));
	MMG_LAUNCH(c, k_res_ncig, mmg_blocks(n1, 256), 256, 0, n, d_ez, ncig);
	MMG_TRY(scan_excl(c, ncig, nc_off, (int)n1));
	int64_t n_cig = 0;
	MMG_D2H(c, &n_cig, nc_off + n, 8);
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	MMG_TRY(c->k_cig_out.ensure(((size_t)n_cig + 1) * 4));
	MMG_LAUNCH(c, k_cig_gather, mmg_blocks(n, 128), 128, 0, n, d_ez, nc_off, reinterpret_cast<const uint64_t*>(cg_off), c->k_cig.as<uint32_t>(),
	           d_res, c->k_cig_out.as<uint32_t>());
	static_assert(sizeof(KswResDev) == sizeof(mmg_ksw_res_t), "result layout");
	if (to_host) {
		MMG_TRY(c->h_k_cig.ensure(((size_t)n_cig + 1) * 4));
		MMG_D2H(c, res, d_res, (size_t)n * sizeof(KswResDev));
		if (n_cig) MMG_D2H(c, c->h_k_cig.p, c->k_cig_out.p, (size_t)n_cig * 4);
		MMG_CUDA(cudaStreamSynchronize(c->stream));
		*cigars = c->h_k_cig.as<uint32_t>();
	} else { // results stay on the device: {ez, cigar offset} per job and the packed CIGARs
		c->k_last_res = d_res;
		*cigars = c->k_cig_out.as<uint32_t>();
		MMG_CUDA(cudaStreamSynchronize(c->stream));
	}
	float ms = 0; cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
	if (kernel_ms) *kernel_ms = ms;
	return MMG_OK;
}

static KswScore make_score(const mmg_mapopt_t *opt)
{ // ksw_gen_simple_mat (align.c:9-22), m = 5
	KswScore sc; sc.m = 5;
	int a = opt->a < 0 ? -opt->a : opt->a, b = opt->b > 0 ? -opt->b : opt->b, amb = opt->sc_ambi > 0 ? -opt->sc_ambi : opt->sc_ambi;
	for (int i = 0; i < 4; ++i) {
		for (int j = 0; j < 4; ++j) sc.mat[i * 5 + j] = (int8_t)(i == j ? a : b);
		sc.mat[i * 5 + 4] = (int8_t)amb;
	}
	for (int j = 0; j < 5; ++j) sc.mat[20 + j] = (int8_t)amb;
	sc.q = (int8_t)opt->q, sc.e = (int8_t)opt->e, sc.q2 = (int8_t)opt->q2, sc.e2 = (int8_t)opt->e2;
	return sc;
}

// DP jobs that are already on the device, results left on the device (mmg_post.cu)
int mmg_ksw_device(mmg_ctx_t *c, const mmg_idx_t *mi, const mmg_mapopt_t *opt, int n_jobs, const mmg_ksw_job_t *d_jobs, const void **d_res,
                   const uint32_t **d_cigars, double *kernel_ms, uint64_t *cells)
{
	*d_res = nullptr, *d_cigars = nullptr;
	if (kernel_ms) *kernel_ms = 0;
	if (cells) *cells = 0;
	if (n_jobs <= 0) return MMG_OK;
	MMG_TRY(ksw_launch(c, d_jobs, n_jobs, c->d_Q.as<uint32_t>(), mi->d_S, c->d_q_off.as<uint64_t>(), c->d_seq_len.as<int32_t>(), mi->d_seq_off, make_score(opt),
	                   nullptr, d_cigars, kernel_ms, cells, false));
	*d_res = c->k_last_res;
	return MMG_OK;
}

extern "C" void mmg_ksw_last_split(const mmg_ctx_t *c, uint64_t *jobs_fast, uint64_t *cells_fast, uint64_t *jobs_literal, uint64_t *cells_literal)
{ // how the last mmg_ksw_batch() divided its jobs between the fast forms (thread per job, wavefront) and the literal forms
	if (jobs_fast) *jobs_fast = c->k_last_jobs_fast;
	if (cells_fast) *cells_fast = c->k_last_cells_fast;
	if (jobs_literal) *jobs_literal = c->k_last_jobs_literal;
	if (cells_literal) *cells_literal = c->k_last_cells_literal;
}

// jobs [0, n) of an mmg_ksw_batch call whose DP state does not fit at once: halves until a part fits, each part's CIGARs appended
// to c->h_k_cig_parts (an all-vs-all round asks for hundreds of GB of traceback for 10^5 overlaps of 10 kb reads)
static int ksw_batch_parts(mmg_ctx_t *c, const mmg_idx_t *mi, const mmg_mapopt_t *opt, int n, const mmg_ksw_job_t *jobs, mmg_ksw_res_t *res,
                           size_t budget, double *kernel_ms, uint64_t *cells, uint64_t split[4])
{
	MMG_H2D(c, c->k_jobs.p, jobs, (size_t)n * sizeof(mmg_ksw_job_t));
	const uint32_t *cg = nullptr;
	double ms = 0; uint64_t cl = 0;
	const int rc = ksw_launch(c, c->k_jobs.as<mmg_ksw_job_t>(), n, c->d_Q.as<uint32_t>(), mi->d_S, c->d_q_off.as<uint64_t>(), c->d_seq_len.as<int32_t>(),
	                          mi->d_seq_off, make_score(opt), res, &cg, &ms, &cl, true, budget);
	if (rc == KSW_SPLIT) {
		const int h = n / 2;
		MMG_TRY(ksw_batch_parts(c, mi, opt, h, jobs, res, budget, kernel_ms, cells, split));
		return ksw_batch_parts(c, mi, opt, n - h, jobs + h, res + h, budget, kernel_ms, cells, split);
	}
	MMG_TRY(rc);
	std::vector<uint32_t> &all = c->h_k_cig_parts;
	const uint64_t base = all.size();
	size_t n_cig = 0;
	for (int i = 0; i < n; ++i) { n_cig += (size_t)res[i].ez.n_cigar; res[i].cigar_off += base; }
	all.insert(all.end(), cg, cg + n_cig);
	*kernel_ms += ms, *cells += cl;
	split[0] += c->k_last_jobs_fast, split[1] += c->k_last_cells_fast, split[2] += c->k_last_jobs_literal, split[3] += c->k_last_cells_literal;
	return MMG_OK;
}

extern "C" int mmg_ksw_batch(mmg_ctx_t *c, const mmg_idx_t *mi, const mmg_mapopt_t *opt, int n_jobs, const mmg_ksw_job_t *jobs,
                             mmg_ksw_res_t *res, const uint32_t **cigars, double *kernel_ms, uint64_t *cells)
{
	*cigars = nullptr;
	if (kernel_ms) *kernel_ms = 0;
	if (cells) *cells = 0;
	if (n_jobs <= 0) return MMG_OK;
	MMG_CUDA(cudaSetDevice(c->dev));
	const ResidentBatch &rb = c->rb;
	for (int i = 0; i < n_jobs; i += 4099) // spot check: a full validation pass would cost more than the copy
		if (jobs[i].seq_id < 0 || jobs[i].seq_id >= rb.n_seq || jobs[i].rid < 0 || jobs[i].rid >= mi->n_seq) {
			mmg_set_error("mmg_ksw_batch: job %d refers to a read or contig that is not resident", i); return MMG_EINVAL;
		}
	MMG_TRY(c->k_jobs.ensure((size_t)(n_jobs + 1) * sizeof(mmg_ksw_job_t)));
	MMG_H2D(c, c->k_jobs.p, jobs, (size_t)n_jobs * sizeof(mmg_ksw_job_t));
	// the DP state may take a third of what the device has free (the ctx's own DP buffers count as free: they are reused)
	size_t fr = 0, total = 0;
	MMG_CUDA(cudaMemGetInfo(&fr, &total));
	const size_t budget = (fr + c->k_mem.cap + c->k_p.cap + c->k_cig.cap) / 3;
	const int rc = ksw_launch(c, c->k_jobs.as<mmg_ksw_job_t>(), n_jobs, c->d_Q.as<uint32_t>(), mi->d_S, c->d_q_off.as<uint64_t>(), c->d_seq_len.as<int32_t>(),
	                          mi->d_seq_off, make_score(opt), res, cigars, kernel_ms, cells, true, budget);
	if (rc != KSW_SPLIT) return rc;
	c->h_k_cig_parts.clear();
	double ms = 0; uint64_t cl = 0, split[4] = {0, 0, 0, 0};
	MMG_TRY(ksw_batch_parts(c, mi, opt, n_jobs, jobs, res, budget, &ms, &cl, split));
	c->k_last_jobs_fast = split[0], c->k_last_cells_fast = split[1], c->k_last_jobs_literal = split[2], c->k_last_cells_literal = split[3];
	if (kernel_ms) *kernel_ms = ms;
	if (cells) *cells = cl;
	c->h_k_cig_parts.push_back(0);
	*cigars = c->h_k_cig_parts.data();
	return MMG_OK;
}

// single pair, sequences given as 0..4 codes (parity-test entry point for ksw_extd2_sse, ksw2.h:60)
__global__ void k_pack_codes(const uint8_t *__restrict__ codes, int n, uint32_t *__restrict__ out)
{
	const int wi = blockIdx.x * blockDim.x + threadIdx.x;
	if (wi * 8 >= n) return;
	uint32_t word = 0;
	for (int j = 0; j < 8 && wi * 8 + j < n; ++j) word |= (uint32_t)(codes[wi * 8 + j] & 0xf) << (4 * j);
	out[wi] = word;
}

extern "C" int mmg_ksw_extd2(mmg_ctx_t *c, int qlen, const uint8_t *query, int tlen, const uint8_t *target, int8_t m, const int8_t *mat,
                             int8_t q, int8_t e, int8_t q2, int8_t e2, int w, int zdrop, int end_bonus, int flag, mmg_extz_t *ez, uint32_t *cigar)
{
	MMG_CUDA(cudaSetDevice(c->dev));
	KswEz z; mmg_ksw_reset(&z);
	memcpy(ez, &z, sizeof(z));
	if (m != 5) { mmg_set_error("mmg_ksw_extd2: only the 5-letter alphabet of the mapper is supported"); return MMG_EINVAL; }
	if (qlen <= 0 || tlen <= 0) return MMG_OK;
	KswScore sc; sc.m = m; memcpy(sc.mat, mat, 25); sc.q = q, sc.e = e, sc.q2 = q2, sc.e2 = e2;
	DevBuf dq, dt, dqp, dtp, dtab;
	int rc = MMG_OK;
	auto fin = [&]() { dq.release(); dt.release(); dqp.release(); dtp.release(); dtab.release(); };
#define KS_TRY(x) do { rc = (x); if (rc != MMG_OK) { fin(); return rc; } } while (0)
	KS_TRY(dq.ensure((size_t)qlen + 16)); KS_TRY(dt.ensure((size_t)tlen + 16));
	KS_TRY(dqp.ensure(((size_t)qlen / 8 + 4) * 4)); KS_TRY(dtp.ensure(((size_t)tlen / 8 + 4) * 4));
	KS_TRY(dtab.ensure(256));
	cudaMemcpyAsync(dq.p, query, qlen, cudaMemcpyHostToDevice, c->stream);
	cudaMemcpyAsync(dt.p, target, tlen, cudaMemcpyHostToDevice, c->stream);
	k_pack_codes<<<mmg_blocks((qlen + 7) / 8, 128), 128, 0, c->stream>>>(dq.as<uint8_t>(), qlen, dqp.as<uint32_t>());
	k_pack_codes<<<mmg_blocks((tlen + 7) / 8, 128), 128, 0, c->stream>>>(dt.as<uint8_t>(), tlen, dtp.as<uint32_t>());
	c->launches += 2;
	// one-entry tables: read 0 starts at base 0 and has qlen bases; contig 0 starts at base 0
	struct { uint64_t q_off; uint64_t ref_off; int32_t read_len; int32_t pad; mmg_ksw_job_t job; } tab;
	memset(&tab, 0, sizeof(tab));
	tab.read_len = qlen;
	tab.job.seq_id = 0, tab.job.q_rev = 0, tab.job.q_start = 0, tab.job.q_len = qlen, tab.job.rid = 0, tab.job.t_start = 0, tab.job.t_len = tlen;
	tab.job.reversed = 0, tab.job.w = w, tab.job.zdrop = zdrop, tab.job.end_bonus = end_bonus, tab.job.flag = flag;
	cudaMemcpyAsync(dtab.p, &tab, sizeof(tab), cudaMemcpyHostToDevice, c->stream);
	uint8_t *tb = dtab.as<uint8_t>();
	mmg_ksw_res_t r; const uint32_t *cg = nullptr;
	rc = ksw_launch(c, reinterpret_cast<const mmg_ksw_job_t*>(tb + 24), 1, dqp.as<uint32_t>(), dtp.as<uint32_t>(), reinterpret_cast<const uint64_t*>(tb),
	                reinterpret_cast<const int32_t*>(tb + 16), reinterpret_cast<const uint64_t*>(tb + 8), sc, &r, &cg, nullptr, nullptr);
	if (rc == MMG_OK) {
		*ez = r.ez;
		for (int i = 0; i < r.ez.n_cigar; ++i) cigar[i] = cg[r.cigar_off + i];
	}
	fin();
	return rc;
#undef KS_TRY
}
