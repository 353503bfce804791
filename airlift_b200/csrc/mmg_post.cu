// mmg_post.cu -- everything between chaining and the hit records handed back to the caller, on the device, for the
// short-read presets: hits, primary/secondary tree, per-mate split, base-level alignment around batched DP, filters,
// MAPQ, pairing (map.c:376-406 per fragment in the reference).
//
// The work is laid out as data-parallel steps over flat arrays (mmg_post.h): one thread per chain builds hit records from
// device-sorted keys, one thread per fragment / read runs the small serial pieces on its own slots, the DP jobs of all
// reads go through K4 in one batch per round, and a prefix sum reserves the room of every alignment record before it is
// written.  There is no device-side heap and no per-fragment object; nothing here includes host sources.
//
//     k_post_cnt/keys   chain -> sort key (device-wide scan gives the first anchor of every chain)
//     segmented sort    keys of every fragment in the reference's hit order (stable, descending; see hit_order_desc)
//     k_post_records    hit records with coordinates                      [thread per chain]
//     k_post_select     tree + secondary selection                         [thread per fragment; warp per fragment above 32 chains]
//     k_post_mates      per-mate hit lists                                 [thread per fragment]
//   { k_post_plan       stretch, windows, DP jobs                          [thread per read]
//     K4                mmg_ksw_device
//     k_post_size/build CIGAR stitching, coordinates, clean-up, cuts }     [thread per read]   (one round unless a hit is cut)
//     k_post_final      filters, order, tree, selection                    [thread per read]
//     k_post_finish     MAPQ, pairing, mate un-flip                        [thread per fragment]
//     k_post_sizes/pack records of every read -> one blob -> one D2H
#include <cub/cub.cuh>
#include <math.h>
#include "mmg_ctx.cuh"
#include "mmg_post.h"

int mmg_ksw_device(mmg_ctx_t *c, const mmg_idx_t *mi, const mmg_mapopt_t *opt, int n_jobs, const mmg_ksw_job_t *d_jobs, const void **d_res,
                   const uint32_t **d_cigars, double *kernel_ms, uint64_t *cells);

static_assert(sizeof(DpJob) == sizeof(mmg_ksw_job_t), "DpJob must match mmg_ksw_job_t");
static_assert(sizeof(HitRec) == 80 && sizeof(HitExtra) == 24, "record layouts");

// ---- kernels: one work item per thread, all logic in mmg_post.h ------------------------------------------------------
#define POST_TID ((int64_t)blockIdx.x * blockDim.x + threadIdx.x)

__global__ void k_post_cnt(const uint64_t *__restrict__ u, int64_t n, int32_t *__restrict__ cnt)
{
	const int64_t g = POST_TID;
	if (g < n) cnt[g] = (int32_t)u[g];
}

__global__ void k_post_keys(const PostShard *__restrict__ shp, int64_t n, const int64_t *__restrict__ pre, uint64_t *__restrict__ key_in, uint64_t *__restrict__ val_in)
{
	const int64_t g = POST_TID;
	if (g < n) post_chain_key(*shp, g, pre, key_in, val_in);
}

__global__ void k_post_records(const PostShard *__restrict__ shp, int64_t n)
{
	const int64_t g = POST_TID;
	if (g < n) post_hit_record(*shp, g);
}

__global__ void k_post_perm_keys(int nf, const int32_t *__restrict__ nu, uint32_t *__restrict__ key, int32_t *__restrict__ idx)
{ // fragments with the most chains first, so that a warp holds fragments of similar weight
	const int i = (int)POST_TID;
	if (i < nf) key[i] = ~(uint32_t)nu[i], idx[i] = i;
}

__global__ void __launch_bounds__(128) k_post_select(const PostShard *__restrict__ shp, const int32_t *__restrict__ perm)
{ // fragments with few chains: one thread each
	const int t = (int)POST_TID;
	if (t >= shp->nf) return;
	const int f = perm[t];
	if (shp->nu[f] <= POST_WARP_MIN_CHAINS) post_hits_select(*shp, f);
}

__global__ void __launch_bounds__(128) k_post_select_warp(const PostShard *__restrict__ shp, const int32_t *__restrict__ perm)
{ // fragments with many chains (read pairs from high-copy repeats): one warp each; perm lists them first
	const int t = (int)(POST_TID >> 5);
	if (t >= shp->nf) return;
	const int f = perm[t];
	if (shp->nu[f] <= POST_WARP_MIN_CHAINS) return;
	__shared__ int32_t s_fast[4][HIT_FAST_WORDS + 2];
	WarpDev wp = {(int)(threadIdx.x & 31)};
	if (wp.lane == 0) atomicAdd(shp->ctr + 3, 1u);
	post_hits_select_warp(wp, *shp, f, s_fast[threadIdx.x >> 5]);
}

__global__ void __launch_bounds__(128) k_post_mates(const PostShard *__restrict__ shp, const int32_t *__restrict__ perm)
{
	const int t = (int)POST_TID;
	if (t < shp->nf) post_mates(*shp, perm[t]);
}

__global__ void __launch_bounds__(128) k_post_plan(const PostShard *__restrict__ shp, const int32_t *__restrict__ read_frag)
{
	const int r = (int)POST_TID;
	if (r < shp->n_seq) post_plan(*shp, read_frag[r], r);
}

__global__ void __launch_bounds__(128) k_post_size(const PostShard *__restrict__ shp)
{
	const int r = (int)POST_TID;
	if (r < shp->n_seq) post_size(*shp, r);
}

__global__ void __launch_bounds__(128) k_post_build(const PostShard *__restrict__ shp, const int32_t *__restrict__ read_frag)
{
	const int r = (int)POST_TID;
	if (r < shp->n_seq) post_build(*shp, read_frag[r], r);
}

__global__ void __launch_bounds__(128) k_post_final(const PostShard *__restrict__ shp)
{
	const int r = (int)POST_TID;
	if (r < shp->n_seq) post_final(*shp, r);
}

__global__ void __launch_bounds__(128) k_post_finish(const PostShard *__restrict__ shp)
{
	const int f = (int)POST_TID;
	if (f < shp->nf) post_finish(*shp, f);
}

// ---- results: every read's hit records followed by the alignment record of each hit, 8-byte aligned pieces
__device__ __forceinline__ int64_t post_extra_bytes(const HitExtra *x) { return (int64_t)((sizeof(HitExtra) + (size_t)x->n_cigar * 4 + 7) & ~(size_t)7); }

__global__ void k_post_sizes(const PostShard *__restrict__ shp, int64_t *__restrict__ sizes)
{
	const PostShard &sh = *shp;
	const int r = (int)POST_TID;
	if (r > sh.n_seq) return;
	int64_t b = 0;
	if (r < sh.n_seq) {
		const int n = sh.n_reg[r];
		const HitRec *h = sh.r1 + sh.roff[r];
		b = (int64_t)n * (int64_t)sizeof(HitRec);
		for (int i = 0; i < n; ++i) if (h[i].p) b += post_extra_bytes(hit_ext(sh.xw, h[i].p));
	}
	sizes[r] = b;
}

__global__ void k_post_pack(const PostShard *__restrict__ shp, const int64_t *__restrict__ offs, unsigned char *__restrict__ blob)
{
	const PostShard &sh = *shp;
	const int r = (int)POST_TID;
	if (r >= sh.n_seq) return;
	const int n = sh.n_reg[r];
	const HitRec *h = sh.r1 + sh.roff[r];
	unsigned char *o = blob + offs[r];
	for (int i = 0; i < n; ++i) reinterpret_cast<HitRec*>(o)[i] = h[i];
	o += (size_t)n * sizeof(HitRec);
	for (int i = 0; i < n; ++i)
		if (h[i].p) {
			const HitExtra *x = hit_ext(sh.xw, h[i].p);
			const uint32_t *src = reinterpret_cast<const uint32_t*>(x);
			uint32_t *dst = reinterpret_cast<uint32_t*>(o);
			const uint32_t words = (uint32_t)(sizeof(HitExtra) / 4) + x->n_cigar;
			for (uint32_t w = 0; w < words; ++w) dst[w] = src[w];
			o += post_extra_bytes(x);
		}
}

// ---- driver --------------------------------------------------------------------------------------------------------
template <class T> static int post_scan(mmg_ctx_t *c, const T *d_in, int64_t *d_out, int64_t n)
{
	size_t tmp = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tmp, d_in, d_out, n, c->stream);
	MMG_TRY(c->d_cub.ensure(tmp));
	MMG_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, d_in, d_out, n, c->stream));
	++c->launches;
	return MMG_OK;
}

#define POST_LOGTAB_N (1 << 17)

static int post_logtab(mmg_ctx_t *c, int match_sc, LogTab *lt)
{ // logf is evaluated by the host's libm for every integer argument the MAPQ formulas can produce (hit.c:446-491, pe.c:159)
	DevBuf &b = c->pb[mmg_ctx_s::PB_LOGTAB];
	if (c->post_logtab_a != match_sc || b.p == nullptr) {
		std::vector<float> t((size_t)POST_LOGTAB_N * 2);
		for (int i = 0; i < POST_LOGTAB_N; ++i) t[i] = logf((float)i / match_sc), t[POST_LOGTAB_N + i] = logf((float)i);
		MMG_TRY(b.ensure(t.size() * 4));
		MMG_CUDA(cudaMemcpyAsync(b.p, t.data(), t.size() * 4, cudaMemcpyHostToDevice, c->stream));
		MMG_CUDA(cudaStreamSynchronize(c->stream));
		c->post_logtab_a = match_sc;
	}
	lt->ld = b.as<float>(), lt->li = b.as<float>() + POST_LOGTAB_N, lt->n = POST_LOGTAB_N;
	return MMG_OK;
}

// Runs the stages above for the batch resident on `c`, right after mmg_seed_chain_resident(download = 0).
extern "C" int mmg_post_chain(mmg_ctx_t *c, const mmg_idx_t *mi, const mmg_mapopt_t *dopt, const void *opt_full, size_t opt_bytes, int idx_flag,
                              const uint32_t *frag_hash, mmg_post_out_t *out)
{
	typedef mmg_ctx_s X;
	struct FullOpt { // mm_mapopt_t (minimap.h:107-150), read field by field below
		int64_t flag; int seed, sdust_thres, max_qlen, bw, max_gap, max_gap_ref, max_frag_len, max_chain_skip, max_chain_iter, min_cnt, min_chain_score;
		float mask_level, pri_ratio; int best_n, max_join_long, max_join_short, min_join_flank_sc; float min_join_flank_ratio;
		int a, b, q, e, q2, e2, sc_ambi, noncan, junc_bonus, zdrop, zdrop_inv, end_bonus, min_dp_max, min_ksw_len, anchor_ext_len, anchor_ext_shift;
		float max_clip_ratio; int pe_ori, pe_bonus; float mid_occ_frac; int32_t min_mid_occ, mid_occ, max_occ; int mini_batch_size; int64_t max_sw_mat; const char *split_prefix;
	};
	memset(out, 0, sizeof(*out));
	if (opt_bytes != sizeof(FullOpt)) { mmg_set_error("mmg_post_chain: mm_mapopt_t size mismatch"); return MMG_EINVAL; }
	(void)idx_flag;
	// only the CIGAR stages (post_plan, post_build) read the reference; without MM_F_CIGAR an index without sequence maps as any other
	if ((static_cast<const FullOpt*>(opt_full)->flag & HIT_F_CIGAR) && mi->d_S == nullptr) {
		mmg_set_error("mmg_post_chain: CIGAR output needs the reference sequence, and the index holds none (--idx-no-seq)");
		return MMG_EINVAL;
	}
	MMG_CUDA(cudaSetDevice(c->dev));
	const ResidentBatch &rb = c->rb;
	const int nf = rb.n_frag, n_seq = rb.n_seq;
	if (nf == 0) return MMG_OK;
	const FullOpt &fo = *static_cast<const FullOpt*>(opt_full);
	const int64_t tot_u = c->last_tot_u, tot_v = c->last_tot_v;
	PostShard hs;
	memset(&hs, 0, sizeof(hs));
	hs.opt.flag = fo.flag, hs.opt.mask_level = fo.mask_level, hs.opt.pri_ratio = fo.pri_ratio, hs.opt.max_clip_ratio = fo.max_clip_ratio;
	hs.opt.best_n = fo.best_n, hs.opt.a = fo.a, hs.opt.b = fo.b, hs.opt.q = fo.q, hs.opt.e = fo.e, hs.opt.q2 = fo.q2, hs.opt.e2 = fo.e2, hs.opt.sc_ambi = fo.sc_ambi;
	hs.opt.zdrop = fo.zdrop, hs.opt.zdrop_inv = fo.zdrop_inv, hs.opt.end_bonus = fo.end_bonus, hs.opt.min_dp_max = fo.min_dp_max, hs.opt.min_cnt = fo.min_cnt;
	hs.opt.min_chain_score = fo.min_chain_score, hs.opt.bw = fo.bw, hs.opt.pe_ori = fo.pe_ori, hs.opt.pe_bonus = fo.pe_bonus, hs.opt.max_gap = fo.max_gap;
	hs.opt.max_gap_ref = fo.max_gap_ref, hs.opt.max_frag_len = fo.max_frag_len, hs.opt.k = mi->k, hs.opt.max_qlen = fo.max_qlen, hs.opt.max_sw_mat = fo.max_sw_mat;
	MMG_TRY(post_logtab(c, fo.a, &hs.lt));
	hs.nf = nf, hs.n_seq = n_seq, hs.idx_k = mi->k;
	DevBuf *B = c->pb;
	// ---- per-batch tables
	MMG_TRY(B[X::PB_SHARD].ensure(sizeof(PostShard)));
	MMG_TRY(B[X::PB_HASH].ensure((size_t)(nf + 1) * 4));
	MMG_TRY(B[X::PB_SEGOFF].ensure((size_t)(nf + 1) * 4));
	MMG_TRY(B[X::PB_READ_FRAG].ensure((size_t)(n_seq + 1) * 4));
	MMG_TRY(B[X::PB_PERM].ensure((size_t)(nf + 1) * 16));
	MMG_TRY(B[X::PB_N0].ensure((size_t)(nf + 1) * 4));
	MMG_TRY(B[X::PB_CAP].ensure((size_t)(n_seq + 2) * 4));
	MMG_TRY(B[X::PB_ROFF].ensure((size_t)(n_seq + 2) * 8));
	MMG_TRY(B[X::PB_NREG].ensure((size_t)(n_seq + 1) * 4));
	MMG_TRY(B[X::PB_A1OFF].ensure((size_t)(n_seq + 1) * 8));
	MMG_TRY(B[X::PB_CTR].ensure(64));
	MMG_TRY(c->h_p_hash.ensure((size_t)(nf + n_seq + 2) * 4));
	{ // the name hash of every fragment (computed by the host: read names never leave it) and the fragment of every read
		int32_t *h = c->h_p_hash.as<int32_t>();
		memcpy(h, frag_hash, (size_t)nf * 4);
		int32_t *rf = h + nf;
		for (int f = 0; f < nf; ++f) for (int j = 0; j < rb.n_seg[f]; ++j) rf[rb.seg_off[f] + j] = f;
		MMG_H2D(c, B[X::PB_HASH].p, h, (size_t)nf * 4);
		MMG_H2D(c, B[X::PB_READ_FRAG].p, rf, (size_t)n_seq * 4);
		MMG_H2D(c, B[X::PB_SEGOFF].p, rb.seg_off.data(), (size_t)nf * 4);
	}
	MMG_CUDA(cudaMemsetAsync(B[X::PB_CTR].p, 0, 64, c->stream));
	MMG_CUDA(cudaMemsetAsync(B[X::PB_CAP].p, 0, (size_t)(n_seq + 2) * 4, c->stream));
	hs.n_seg = c->d_frag_nseg.as<int32_t>(), hs.seg_off = B[X::PB_SEGOFF].as<int32_t>(), hs.seq_len = c->d_seq_len.as<int32_t>();
	hs.q_off = c->d_q_off.as<uint64_t>(), hs.flip = c->d_flip.as<uint8_t>(), hs.Q = c->d_Q.as<uint32_t>(), hs.S = mi->d_S;
	hs.ref_off = mi->d_seq_off, hs.ref_len = mi->d_seq_len;
	hs.nu = c->pass[0].nu.as<int32_t>(), hs.rep = c->pass[0].rep.as<int32_t>(), hs.uoff = c->d_uoff.as<int64_t>(), hs.voff = c->d_voff.as<int64_t>();
	hs.u = c->d_out_u.as<uint64_t>(), hs.a = c->d_out_a.as<mm128>(), hs.hash = B[X::PB_HASH].as<uint32_t>();
	// ---- fragment-level hit arrays (one slot per chain)
	const size_t nu1 = (size_t)tot_u + 1;
	MMG_TRY(B[X::PB_CNT].ensure(nu1 * 4)); MMG_TRY(B[X::PB_PRE].ensure((nu1 + 1) * 8));
	MMG_TRY(B[X::PB_KEY_IN].ensure(nu1 * 8)); MMG_TRY(B[X::PB_VAL_IN].ensure(nu1 * 8));
	MMG_TRY(B[X::PB_KEY].ensure(nu1 * 8)); MMG_TRY(B[X::PB_ASCNT].ensure(nu1 * 8));
	MMG_TRY(B[X::PB_R0].ensure(nu1 * sizeof(HitRec)));
	MMG_TRY(B[X::PB_W].ensure(nu1 * 4)); MMG_TRY(B[X::PB_COV].ensure(nu1 * 8)); MMG_TRY(B[X::PB_BIG].ensure(nu1 * 16));
	MMG_TRY(B[X::PB_STACK].ensure((nu1 / 65 + 2 * (size_t)nf + 4) * sizeof(RsFrame)));
	MMG_TRY(B[X::PB_A1].ensure(((size_t)tot_v + 1) * 16));
	hs.key_in = B[X::PB_KEY_IN].as<uint64_t>(), hs.key = B[X::PB_KEY].as<uint64_t>(), hs.ascnt = B[X::PB_ASCNT].as<uint64_t>(), hs.r0 = B[X::PB_R0].as<HitRec>();
	hs.w = B[X::PB_W].as<int32_t>(), hs.cov = B[X::PB_COV].as<uint64_t>(), hs.big = B[X::PB_BIG].as<mm128>(), hs.stack = B[X::PB_STACK].as<RsFrame>();
	hs.n0 = B[X::PB_N0].as<int32_t>(), hs.cap = B[X::PB_CAP].as<int32_t>(), hs.roff = B[X::PB_ROFF].as<int64_t>(), hs.n_reg = B[X::PB_NREG].as<int32_t>();
	hs.a1 = B[X::PB_A1].as<mm128>(), hs.a1_off = B[X::PB_A1OFF].as<int64_t>(), hs.ctr = B[X::PB_CTR].as<unsigned int>(), hs.n_jobs = hs.ctr + 2;
	PostShard *d_sh = B[X::PB_SHARD].as<PostShard>();
	MMG_CUDA(cudaEventRecord(c->ev[0], c->stream));
	MMG_H2D(c, d_sh, &hs, sizeof(hs));
	// thread -> fragment order for the per-fragment steps
	int32_t *perm;
	{
		uint32_t *key = B[X::PB_PERM].as<uint32_t>(), *key2 = key + nf;
		int32_t *idx = reinterpret_cast<int32_t*>(key2 + nf);
		perm = idx + nf;
		MMG_LAUNCH(c, k_post_perm_keys, mmg_blocks(nf, 256), 256, 0, nf, hs.nu, key, idx);
		size_t tmp = 0;
		cub::DeviceRadixSort::SortPairs(nullptr, tmp, key, key2, idx, perm, nf, 0, 32, c->stream);
		MMG_TRY(c->d_cub.ensure(tmp));
		MMG_TIMED(c, "cub_radix_sort(fragments)", cub::DeviceRadixSort::SortPairs(c->d_cub.p, tmp, key, key2, idx, perm, nf, 0, 32, c->stream));
	}
	if (tot_u > 0) { // keys -> hit order -> records
		MMG_LAUNCH(c, k_post_cnt, mmg_blocks(tot_u, 256), 256, 0, hs.u, tot_u, B[X::PB_CNT].as<int32_t>());
		MMG_TRY(post_scan(c, B[X::PB_CNT].as<int32_t>(), B[X::PB_PRE].as<int64_t>(), tot_u));
		MMG_LAUNCH(c, k_post_keys, mmg_blocks(tot_u, 256), 256, 0, d_sh, tot_u, B[X::PB_PRE].as<int64_t>(), B[X::PB_KEY_IN].as<uint64_t>(), B[X::PB_VAL_IN].as<uint64_t>());
		size_t tmp = 0;
		cub::DeviceSegmentedSort::StableSortPairsDescending(nullptr, tmp, hs.key_in, hs.key, B[X::PB_VAL_IN].as<uint64_t>(), hs.ascnt, tot_u, nf, hs.uoff, hs.uoff + 1, c->stream);
		MMG_TRY(c->d_cub.ensure(tmp));
		MMG_TIMED(c, "cub_segmented_sort(chains)", cub::DeviceSegmentedSort::StableSortPairsDescending(c->d_cub.p, tmp, hs.key_in, hs.key, B[X::PB_VAL_IN].as<uint64_t>(), hs.ascnt, tot_u, nf, hs.uoff, hs.uoff + 1, c->stream));
		MMG_LAUNCH(c, k_post_records, mmg_blocks(tot_u, 128), 128, 0, d_sh, tot_u);
	}
	MMG_LAUNCH(c, k_post_select_warp, mmg_blocks((size_t)nf * 32, 128), 128, 0, d_sh, perm);
	MMG_LAUNCH(c, k_post_select, mmg_blocks(nf, 128), 128, 0, d_sh, perm);
	// ---- per-read hit slots
	MMG_TRY(post_scan(c, hs.cap, B[X::PB_ROFF].as<int64_t>(), (int64_t)n_seq + 1));
	int64_t slots = 0;
	MMG_D2H(c, &slots, B[X::PB_ROFF].as<int64_t>() + n_seq, 8);
	MMG_CUDA(cudaStreamSynchronize(c->stream)); // also: `hs` was read by the copy above
	const size_t ns1 = (size_t)slots + 1;
	MMG_TRY(B[X::PB_R1].ensure(ns1 * sizeof(HitRec))); MMG_TRY(B[X::PB_TMP1].ensure(ns1 * sizeof(HitRec)));
	MMG_TRY(B[X::PB_PLAN].ensure(ns1 * sizeof(RegionPlan)));
	MMG_TRY(B[X::PB_XSIZE].ensure((ns1 + 1) * 4)); MMG_TRY(B[X::PB_XOFF].ensure((ns1 + 1) * 8));
	MMG_TRY(B[X::PB_SKEY].ensure(ns1 * 8)); MMG_TRY(B[X::PB_SIDX].ensure(ns1 * 4)); MMG_TRY(B[X::PB_SBIG].ensure(ns1 * 16));
	MMG_TRY(B[X::PB_SSTACK].ensure((ns1 / 65 + 2 * (size_t)n_seq + 4) * sizeof(RsFrame)));
	const unsigned int job_cap = (unsigned int)(slots * 3 < 0x7fffffff ? slots * 3 + 16 : 0x7fffffff);
	MMG_TRY(B[X::PB_JOBS].ensure((size_t)job_cap * sizeof(DpJob)));
	hs.r1 = B[X::PB_R1].as<HitRec>(), hs.tmp1 = B[X::PB_TMP1].as<HitRec>(), hs.pl = B[X::PB_PLAN].as<RegionPlan>();
	hs.xsize = B[X::PB_XSIZE].as<uint32_t>(), hs.xoff = B[X::PB_XOFF].as<int64_t>();
	hs.skey = B[X::PB_SKEY].as<uint64_t>(), hs.sidx = B[X::PB_SIDX].as<int32_t>(), hs.sbig = B[X::PB_SBIG].as<mm128>(), hs.sstack = B[X::PB_SSTACK].as<RsFrame>();
	hs.jobs = B[X::PB_JOBS].as<DpJob>(), hs.job_cap = job_cap;
	hs.xw = B[X::PB_XW].as<uint32_t>();
	MMG_H2D(c, d_sh, &hs, sizeof(hs));
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	const int32_t *read_frag = B[X::PB_READ_FRAG].as<int32_t>();
	MMG_LAUNCH(c, k_post_mates, mmg_blocks(nf, 128), 128, 0, d_sh, perm);
	double ksw_ms = 0;
	int64_t x_used = 0;
	if (fo.flag & HIT_F_CIGAR) {
		for (int round = 0;; ++round) {
			unsigned int ctr[4] = {0, 0, 0, 0};
			MMG_CUDA(cudaMemsetAsync(hs.ctr, 0, 4, c->stream));       // hits cut off in this round
			MMG_CUDA(cudaMemsetAsync(hs.n_jobs, 0, 4, c->stream));
			MMG_LAUNCH(c, k_post_plan, mmg_blocks(n_seq, 128), 128, 0, d_sh, read_frag);
			MMG_D2H(c, ctr, hs.ctr, 16);
			MMG_CUDA(cudaStreamSynchronize(c->stream));
			if (ctr[1] & POST_ERR_JOBS) { mmg_set_error("post-chaining stages: DP job buffer too small"); return MMG_ELIMIT; }
			const int n_jobs = (int)ctr[2];
			const void *d_res = nullptr; const uint32_t *d_cig = nullptr; double kms = 0; uint64_t cells = 0;
			if (n_jobs > 0) {
				MMG_TRY(mmg_ksw_device(c, mi, dopt, n_jobs, reinterpret_cast<const mmg_ksw_job_t*>(hs.jobs), &d_res, &d_cig, &kms, &cells));
				ksw_ms += kms;
				out->n_dp_jobs += (uint64_t)n_jobs, out->n_dp_cells += cells, out->n_dp_rounds += 1;
				out->n_dp_jobs_fast += c->k_last_jobs_fast, out->n_dp_cells_fast += c->k_last_cells_fast;
			}
			hs.dp.res = static_cast<const DpRes*>(d_res), hs.dp.cig = d_cig;
			MMG_H2D(c, reinterpret_cast<char*>(d_sh) + offsetof(PostShard, dp), &hs.dp, sizeof(hs.dp));
			MMG_LAUNCH(c, k_post_size, mmg_blocks(n_seq, 128), 128, 0, d_sh);
			MMG_TRY(post_scan(c, hs.xsize, B[X::PB_XOFF].as<int64_t>(), slots + 1));
			int64_t words = 0;
			MMG_D2H(c, &words, B[X::PB_XOFF].as<int64_t>() + slots, 8);
			MMG_CUDA(cudaStreamSynchronize(c->stream));
			MMG_TRY(B[X::PB_XW].ensure_keep((size_t)(x_used + words + 16) * 4, (size_t)x_used * 4, c->stream));
			hs.xw = B[X::PB_XW].as<uint32_t>(), hs.x_base = x_used;
			MMG_H2D(c, reinterpret_cast<char*>(d_sh) + offsetof(PostShard, xw), &hs.xw, sizeof(hs.xw));
			MMG_H2D(c, reinterpret_cast<char*>(d_sh) + offsetof(PostShard, x_base), &hs.x_base, sizeof(hs.x_base));
			MMG_LAUNCH(c, k_post_build, mmg_blocks(n_seq, 128), 128, 0, d_sh, read_frag);
			x_used += words;
			MMG_D2H(c, ctr, hs.ctr, 16);
			{
				cudaError_t e = cudaStreamSynchronize(c->stream);
				if (e != cudaSuccess) { mmg_set_error("post-chaining stages: %s", cudaGetErrorString(e)); return MMG_ECUDA; }
			}
			if (ctr[1] & POST_ERR_SLOTS) { mmg_set_error("post-chaining stages: a read was cut at z-drops more often than its hit slots allow"); return MMG_ELIMIT; }
			c->path[5] += ctr[0];
			if (ctr[0] == 0) break; // no hit was cut: every hit is aligned
			c->path[4] += 1;
			if (round > 64) { mmg_set_error("post-chaining stages: alignment made no progress"); return MMG_ECUDA; }
		}
		MMG_LAUNCH(c, k_post_final, mmg_blocks(n_seq, 128), 128, 0, d_sh);
	}
	MMG_LAUNCH(c, k_post_finish, mmg_blocks(nf, 128), 128, 0, d_sh);
	// ---- pack and download
	MMG_TRY(B[X::PB_SIZES].ensure((size_t)(n_seq + 2) * 8));
	MMG_TRY(B[X::PB_OFFS].ensure((size_t)(n_seq + 2) * 8));
	int64_t *sizes = B[X::PB_SIZES].as<int64_t>();
	MMG_LAUNCH(c, k_post_sizes, mmg_blocks((size_t)n_seq + 1, 128), 128, 0, d_sh, sizes);
	MMG_TRY(post_scan(c, sizes, B[X::PB_OFFS].as<int64_t>(), (int64_t)n_seq + 1));
	int64_t blob_bytes = 0;
	unsigned int ctr[4] = {0, 0, 0, 0};
	MMG_D2H(c, &blob_bytes, B[X::PB_OFFS].as<int64_t>() + n_seq, 8);
	MMG_D2H(c, ctr, hs.ctr, 16);
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	c->path[3] += ctr[3];
	if (ctr[1] & POST_ERR_LOGTAB) { mmg_set_error("post-chaining stages: a MAPQ argument lies outside the logf table (alignment score above %d)", POST_LOGTAB_N); return MMG_ELIMIT; }
	MMG_TRY(B[X::PB_BLOB].ensure((size_t)blob_bytes + 64));
	MMG_LAUNCH(c, k_post_pack, mmg_blocks(n_seq, 128), 128, 0, d_sh, B[X::PB_OFFS].as<int64_t>(), B[X::PB_BLOB].as<unsigned char>());
	MMG_CUDA(cudaEventRecord(c->ev[1], c->stream));
	MMG_TRY(c->h_p_nreg.ensure((size_t)(n_seq + 1) * 4));
	MMG_TRY(c->h_p_offs.ensure((size_t)(n_seq + 2) * 8));
	MMG_TRY(c->h_p_blob.ensure((size_t)blob_bytes + 64));
	MMG_TRY(c->h_p_rep.ensure((size_t)(nf + 1) * 4));
	MMG_D2H(c, c->h_p_nreg.p, hs.n_reg, (size_t)n_seq * 4);
	MMG_D2H(c, c->h_p_offs.p, B[X::PB_OFFS].p, (size_t)(n_seq + 1) * 8);
	if (blob_bytes) MMG_D2H(c, c->h_p_blob.p, B[X::PB_BLOB].p, (size_t)blob_bytes);
	MMG_D2H(c, c->h_p_rep.p, c->pass[0].rep.p, (size_t)nf * 4);
	{
		cudaError_t e = cudaStreamSynchronize(c->stream);
		if (e != cudaSuccess) { mmg_set_error("post-chaining stages (pack): %s", cudaGetErrorString(e)); return MMG_ECUDA; }
	}
	float ms = 0;
	cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
	if (getenv("MMG_TRACE"))
		fprintf(stderr, "[mmg::post] %d fragments, %lld chains -> %lld hit slots, alignment records %.1f MB, blob %.1f MB, %.1f ms on the device (K4 %.1f ms, %llu DP rounds)\n",
		        nf, (long long)tot_u, (long long)slots, x_used * 4 / 1e6, blob_bytes / 1e6, ms, ksw_ms, (unsigned long long)out->n_dp_rounds);
	out->n_reg = c->h_p_nreg.as<int32_t>(), out->blob_off = c->h_p_offs.as<int64_t>(), out->blob = c->h_p_blob.as<unsigned char>();
	out->rep_len = c->h_p_rep.as<int32_t>();
	out->t_device_ms = ms, out->t_ksw_ms = ksw_ms;
	out->finished = 1;
	return MMG_OK;
}
