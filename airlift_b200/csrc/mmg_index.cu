// mmg_index.cu -- context management and the device-resident minimizer index.
//
// Replaces mm_idx_gen / mm_idx_str / worker_post (index.c:191-243,353-432) with a GPU build:
// pack the reference to 4 bits/base, sketch it in overlapping chunks (K1), radix-sort the
// (minimizer, position) pairs, and insert one 16-byte slot per distinct minimizer into an
// open-addressing table.  mm_idx_get's observable result -- the count and the ascending list of
// positions (index.c:230) -- is preserved; the bucket/khash layout (index.c:27-32) is not.
#include <stdarg.h>
#include <cub/cub.cuh>
#include "mmg_ctx.cuh"
#include "mmg_sketchwarp.h"

static thread_local char g_err[512] = "";
void mmg_set_error(const char *fmt, ...)
{
	va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap);
}
extern "C" const char *mmg_last_error(void) { return g_err; }

extern "C" int mmg_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
	return n;
}

extern "C" int mmg_init(int device, mmg_ctx_t **out)
{
	int n = mmg_device_count();
	*out = nullptr;
	if (n <= 0) { mmg_set_error("no CUDA device: this library has no CPU path"); return MMG_ENODEV; }
	if (device < 0 || device >= n) { mmg_set_error("device %d out of range (%d present)", device, n); return MMG_EINVAL; }
	MMG_CUDA(cudaSetDevice(device));
	MMG_TRY(mmg_ksw_set_smem_attrs());
	MMG_TRY(mmg_stages_set_smem_attrs());
	mmg_ctx_t *c = new mmg_ctx_s();
	c->dev = device;
	MMG_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
	for (int i = 0; i < 4; ++i) MMG_CUDA(cudaEventCreate(&c->ev[i]));
	for (StageSlot &s : c->stage) MMG_CUDA(cudaEventCreateWithFlags(&s.drained, cudaEventDisableTiming));
	*out = c;
	return MMG_OK;
}

extern "C" void mmg_destroy(mmg_ctx_t *c)
{
	if (!c) return;
	cudaSetDevice(c->dev);
	cudaStreamSynchronize(c->stream);
	DevBuf *bufs[] = {&c->d_ascii, &c->d_Q, &c->d_seq_len, &c->d_seq_off, &c->d_q_off, &c->d_flip, &c->d_units, &c->d_unit_cnt,
		&c->d_unit_off, &c->d_mv, &c->d_m_n, &c->d_m_val, &c->d_frag_unit0, &c->d_frag_qlen, &c->d_frag_nseg, &c->d_heap,
		&c->d_frag_flag, &c->d_frag_iter, &c->d_cub, &c->d_out_u, &c->d_out_a, &c->d_out_mini, &c->d_uoff, &c->d_voff,
		&c->d_moff, &c->d_frag_list, &c->d_seg_head, &c->d_seg_start, &c->d_seg_avg, &c->d_replay, &c->d_skey, &c->d_sval, &c->d_sseg, &c->d_tie, &c->d_m_aoff, &c->d_hrank, &c->d_hpop, &c->d_hlist, &c->d_seg_li, &c->d_seg_long, &c->d_unit0, &c->d_fseg_off, &c->d_sk_stage, &c->d_heavy, &c->d_ukey,
		&c->k_jobs, &c->k_mem, &c->k_H, &c->k_p, &c->k_cig, &c->k_res, &c->k_cig_out, &c->k_cig_off};
	if (getenv("MM2_B200_TRACE"))
		fprintf(stderr, "[T::buffers] %llu device and %llu pinned (re-)allocations so far, %.3f s and %.3f s inside them\n", g_mmg_grow[0], g_mmg_grow[1],
		        g_mmg_grow_ns[0] * 1e-9, g_mmg_grow_ns[1] * 1e-9);
	const unsigned long long t_rel = mmg_now_ns();
	for (DevBuf *b : bufs) b->release();
	for (DevBuf &b : c->pb) b.release();
	for (PassArena &p : c->pass) p.release();
	PinBuf *pins[] = {&c->h_meta, &c->h_out_meta, &c->h_out_u, &c->h_out_a, &c->h_out_mini, &c->h_k_jobs, &c->h_k_res, &c->h_k_cig,
	                  &c->h_p_hash, &c->h_p_nreg, &c->h_p_offs, &c->h_p_blob, &c->h_p_rep, &c->h_path};
	for (PinBuf *b : pins) b->release();
	for (StageSlot &s : c->stage) {
		s.bases.release(), s.tab.release(), s.flip.release(), s.ukey.release();
		if (s.drained) cudaEventDestroy(s.drained);
	}
	if (getenv("MM2_B200_TRACE")) fprintf(stderr, "[T::buffers] released in %.3f s\n", (mmg_now_ns() - t_rel) * 1e-9);
	for (int i = 0; i < 4; ++i) if (c->ev[i]) cudaEventDestroy(c->ev[i]);
	for (const ProfRec &r : c->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
	for (cudaEvent_t e : c->ev_pool) cudaEventDestroy(e);
	cudaStreamDestroy(c->stream);
	delete c;
}

extern "C" int mmg_device(const mmg_ctx_t *c) { return c->dev; }
extern "C" void *mmg_stream(const mmg_ctx_t *c) { return (void*)c->stream; }
extern "C" long mmg_launch_count(mmg_ctx_t *c, int reset) { long n = c->launches; if (reset) c->launches = 0; return n; }

extern "C" void mmg_copy_bytes(mmg_ctx_t *c, uint64_t *h2d, uint64_t *d2h, int reset)
{
	*h2d = c->h2d_bytes, *d2h = c->d2h_bytes;
	if (reset) c->h2d_bytes = c->d2h_bytes = 0;
}

unsigned long long g_mmg_grow[2] = {0, 0};
unsigned long long g_mmg_grow_ns[2] = {0, 0};
extern "C" void mmg_growth_counts(uint64_t out[2], int reset)
{
	for (int i = 0; i < 2; ++i) { out[i] = g_mmg_grow[i]; if (reset) g_mmg_grow[i] = 0; }
}

extern "C" void mmg_profile_enable(mmg_ctx_t *c, int on) { c->prof_on = on != 0; }

extern "C" void mmg_path_counts(mmg_ctx_t *c, uint64_t out[8], int reset)
{
	for (int i = 0; i < 8; ++i) { out[i] = c->path[i]; if (reset) c->path[i] = 0; }
}

// per-kernel device time since the last fetch, from CUDA events recorded around every launch on the ctx stream.
// Fills up to max entries (name pointers are static strings); returns the number of distinct kernels.
extern "C" int mmg_profile_fetch(mmg_ctx_t *c, int max, const char **names, double *ms, long *launches)
{
	cudaSetDevice(c->dev);
	cudaStreamSynchronize(c->stream);
	int n = 0;
	const bool trace = getenv("MMG_TRACE_LAUNCHES") != nullptr; // every launch longer than 0.5 ms, in issue order
	for (const ProfRec &r : c->prof) {
		float t = 0;
		cudaEventElapsedTime(&t, r.a, r.b);
		if (trace && t > 0.5f) fprintf(stderr, "[mmg::launch] ctx %p %-22s %9.3f ms\n", (void*)c, r.name, t);
		int i;
		for (i = 0; i < n; ++i) if (names[i] == r.name || strcmp(names[i], r.name) == 0) break;
		if (i == n) { if (n == max) { c->ev_pool.push_back(r.a); c->ev_pool.push_back(r.b); continue; } names[n] = r.name, ms[n] = 0, launches[n] = 0, ++n; }
		ms[i] += t, launches[i] += 1;
		c->ev_pool.push_back(r.a); c->ev_pool.push_back(r.b);
	}
	c->prof.clear();
	return n;
}

// ------------------------------------------------------------------ kernels

// pack 8 ASCII bases per thread into one 4-bit word (mm_seq4_set, mmpriv.h:28; index.c:321-325)
__global__ void k_pack_ref(const uint8_t *__restrict__ ascii, uint64_t n_bases, uint32_t *__restrict__ S)
{
	const uint64_t wi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const uint64_t b0 = wi * 8;
	if (b0 >= n_bases) return;
	uint32_t word = 0;
	if (b0 + 8 <= n_bases) {
		const uint2 v = *reinterpret_cast<const uint2*>(ascii + b0); // 8-byte aligned: b0 is a multiple of 8
		const uint32_t lo = v.x, hi = v.y;
#pragma unroll
		for (int j = 0; j < 4; ++j) word |= (uint32_t)mmg_nt4((lo >> (8 * j)) & 0xff) << (4 * j);
#pragma unroll
		for (int j = 0; j < 4; ++j) word |= (uint32_t)mmg_nt4((hi >> (8 * j)) & 0xff) << (4 * (j + 4));
	} else {
		for (int j = 0; b0 + j < n_bases; ++j) word |= (uint32_t)mmg_nt4(ascii[b0 + j]) << (4 * j);
	}
	S[wi] = word;
}

struct EmitCount { __device__ void operator()(int, const mm128 &) const {} };

// K1 over work units: count pass (out == nullptr) and fill pass
__global__ void k_sketch_count(const uint32_t *__restrict__ S, const SketchUnit *__restrict__ units, int n_units, int w, int k, int is_hpc,
                               int32_t *__restrict__ cnt)
{
	const int u = blockIdx.x * blockDim.x + threadIdx.x;
	if (u >= n_units) return;
	cnt[u] = mmg_sketch_unit<false>(S, units[u], w, k, is_hpc, nullptr);
}

__global__ void k_sketch_fill(const uint32_t *__restrict__ S, const SketchUnit *__restrict__ units, int n_units, int w, int k, int is_hpc,
                              const int64_t *__restrict__ off, mm128 *__restrict__ out)
{
	const int u = blockIdx.x * blockDim.x + threadIdx.x;
	if (u >= n_units) return;
	mmg_sketch_unit<true>(S, units[u], w, k, is_hpc, out + off[u]);
}

// K1, short reads: one warp per read (mmg_sketchwarp.h).  Count pass (out == nullptr) and fill pass; a read the warp form does
// not take (ambiguous base, odd geometry) is sketched by lane 0 with the state machine.
#define SKW_WARPS 4
template <bool kWrite>
__global__ void __launch_bounds__(32 * SKW_WARPS)
k_sketch_warp(const uint32_t *__restrict__ S, const SketchUnit *__restrict__ units, int n_units, int w, int k, int is_hpc,
              int32_t *__restrict__ cnt, const int64_t *__restrict__ off, mm128 *__restrict__ out)
{
	__shared__ uint64_t s_words[SKW_WARPS][SKW_MAX_LEN / 32 + 2], s_xs[SKW_WARPS][SKW_MAX_LEN];
	__shared__ uint8_t s_zs[SKW_WARPS][SKW_MAX_LEN];
	const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const int u = blockIdx.x * SKW_WARPS + wi;
	if (u >= n_units) return;
	const SketchUnit un = units[u];
	const WarpDev wp = {lane};
	// kWrite with off == nullptr: single pass into a staging area with one slot per base of the read (a read cannot emit more
	// minimizers than it has bases), compacted by k_sketch_compact once the counts have been scanned
	mm128 *o = kWrite ? (off ? out + off[u] : out + un.off) : nullptr;
	int n = -1;
	if (skw_eligible(un, w, k, is_hpc)) n = mmg_sketch_warp<WarpDev, kWrite>(wp, S, un, w, k, s_words[wi], s_xs[wi], s_zs[wi], o);
	if (n < 0 && lane == 0) n = mmg_sketch_unit<kWrite>(S, un, w, k, is_hpc, o);
	if (cnt && lane == 0) cnt[u] = n;
}

// staging area -> dense output, one warp per read
__global__ void k_sketch_compact(const SketchUnit *__restrict__ units, int n_units, const int32_t *__restrict__ cnt, const int64_t *__restrict__ off,
                                 const mm128 *__restrict__ stage, mm128 *__restrict__ out)
{
	const int u = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
	if (u >= n_units) return;
	const mm128 *src = stage + units[u].off;
	mm128 *dst = out + off[u];
	for (int i = lane; i < cnt[u]; i += 32) dst[i] = src[i];
}

__global__ void k_split_kv(const mm128 *__restrict__ mv, int64_t n, uint64_t *__restrict__ key, uint64_t *__restrict__ val)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const mm128 m = mv[i];
	key[i] = m.x >> 8, val[i] = m.y;
}

__global__ void k_fill_u64(uint64_t *p, uint64_t n, uint64_t v)
{
	const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i < n) p[i] = v;
}

// one slot per distinct minimizer; linear probing, claim with a 64-bit CAS on the key
__global__ void k_idx_insert(const uint64_t *__restrict__ ukey, const uint32_t *__restrict__ ucnt, const int64_t *__restrict__ ustart,
                             int64_t n_keys, const uint64_t *__restrict__ pos, IdxSlot *slots, uint64_t mask, int shift)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n_keys) return;
	const uint64_t minier = ukey[i];
	const uint32_t n = ucnt[i];
	const uint64_t start = (uint64_t)ustart[i];
	const uint64_t key = n == 1 ? (minier | MMG_SLOT_SINGLE) : minier;
	const uint64_t val = n == 1 ? pos[start] : (start << 32 | (uint64_t)n);
	uint64_t s = mmg_slot_hash(minier, shift);
	for (;;) {
		const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(&slots[s].key), (unsigned long long)MMG_SLOT_EMPTY, (unsigned long long)key);
		if (old == MMG_SLOT_EMPTY) { slots[s].val = val; return; }
		s = (s + 1) & mask;
	}
}

__global__ void k_idx_get(IdxView ix, int n_q, const uint64_t *__restrict__ minier, int32_t *__restrict__ n_out, int max_pos, uint64_t *__restrict__ pos_out)
{
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n_q) return;
	uint64_t val;
	const int n = mmg_idx_probe(ix, minier[i], &val);
	n_out[i] = n;
	for (int j = 0; j < n && j < max_pos; ++j) pos_out[(size_t)i * max_pos + j] = mmg_hit_pos(ix.pos, n, val, (uint32_t)j);
}

// ------------------------------------------------------------------ build

int mmg_run_sketch(mmg_ctx_t *c, const uint32_t *d_S, const SketchUnit *d_units, int n_units, int w, int k, int is_hpc,
                   DevBuf &cnt, DevBuf &off, DevBuf &out, int64_t *total, bool short_reads, uint64_t stage_slots)
{ // count -> exclusive scan -> fill; leaves off[n_units] = total.  short_reads: every unit is a whole read of at most SKW_MAX_LEN bases
  // that starts at its own 8-aligned offset of d_S (stage_slots = the padded bases of all reads): one pass into a staging area, then compaction
	const bool warp_form = short_reads && !is_hpc && (k & 1) && w <= 64 && stage_slots > 0;
	if (warp_form) MMG_TRY(c->d_sk_stage.ensure((stage_slots + 8) * sizeof(mm128)));
	*total = 0;
	MMG_TRY(cnt.ensure((size_t)(n_units + 1) * 4));
	MMG_TRY(off.ensure((size_t)(n_units + 1) * 8));
	if (n_units == 0) return MMG_OK;
	MMG_CUDA(cudaMemsetAsync(cnt.p, 0, (size_t)(n_units + 1) * 4, c->stream));
	if (warp_form) MMG_LAUNCH(c, k_sketch_warp<true>, mmg_blocks(n_units, SKW_WARPS), 32 * SKW_WARPS, 0, d_S, d_units, n_units, w, k, is_hpc, cnt.as<int32_t>(), nullptr, c->d_sk_stage.as<mm128>());
	else MMG_LAUNCH(c, k_sketch_count, mmg_blocks(n_units, 128), 128, 0, d_S, d_units, n_units, w, k, is_hpc, cnt.as<int32_t>());
	size_t tmp_bytes = 0;
	cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, cnt.as<int32_t>(), off.as<int64_t>(), n_units + 1, c->stream);
	MMG_TRY(c->d_cub.ensure(tmp_bytes));
	MMG_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp_bytes, cnt.as<int32_t>(), off.as<int64_t>(), n_units + 1, c->stream));
	++c->launches;
	MMG_CUDA(cudaMemcpyAsync(total, off.as<int64_t>() + n_units, 8, cudaMemcpyDeviceToHost, c->stream));
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	MMG_TRY(out.ensure((size_t)(*total + 1) * sizeof(mm128)));
	if (warp_form) MMG_LAUNCH(c, k_sketch_compact, mmg_blocks((size_t)n_units * 32, 256), 256, 0, d_units, n_units, cnt.as<int32_t>(), off.as<int64_t>(), c->d_sk_stage.as<mm128>(), out.as<mm128>());
	else MMG_LAUNCH(c, k_sketch_fill, mmg_blocks(n_units, 128), 128, 0, d_S, d_units, n_units, w, k, is_hpc, off.as<int64_t>(), out.as<mm128>());
	return MMG_OK;
}

#define MMG_IDX_CHUNK 1024

extern "C" void mmg_idx_free(mmg_idx_t *mi)
{
	if (!mi) return;
	cudaSetDevice(mi->dev);
	cudaFree(mi->d_S); cudaFree(mi->d_seq_off); cudaFree(mi->d_seq_len); cudaFree(mi->d_slots); cudaFree(mi->d_pos); cudaFree(mi->d_counts); cudaFree(mi->d_tkey);
	delete mi;
}

extern "C" int mmg_idx_set_name_keys(mmg_idx_t *mi, const uint32_t *tkey)
{
	if (tkey == nullptr) { mmg_set_error("mmg_idx_set_name_keys: no key table"); return MMG_EINVAL; }
	MMG_CUDA(cudaSetDevice(mi->dev));
	if (mi->d_tkey == nullptr) MMG_CUDA(cudaMalloc(&mi->d_tkey, (size_t)(mi->n_seq + 1) * 4));
	MMG_CUDA(cudaMemcpy(mi->d_tkey, tkey, (size_t)mi->n_seq * 4, cudaMemcpyHostToDevice));
	return MMG_OK;
}

static int idx_alloc(mmg_idx_t *mi, bool with_S)
{
	if (with_S) MMG_CUDA(cudaMalloc(&mi->d_S, ((mi->total_len + 7) / 8 + 4) * 4));
	MMG_CUDA(cudaMalloc(&mi->d_seq_off, (size_t)(mi->n_seq + 1) * 8));
	MMG_CUDA(cudaMalloc(&mi->d_seq_len, (size_t)(mi->n_seq + 1) * 4));
	MMG_CUDA(cudaMalloc(&mi->d_slots, mi->n_slots * sizeof(IdxSlot)));
	MMG_CUDA(cudaMalloc(&mi->d_pos, (mi->n_pos + 1) * 8));
	return MMG_OK;
}

// one slot per distinct minimizer (power-of-two slots at load <= 0.5), filled from the key-sorted (ukey, counts, ustart) and pos[]
static int idx_table(mmg_ctx_t *c, mmg_idx_t *mi, const uint64_t *d_ukey, const int64_t *d_ustart)
{
	uint64_t n_slots = 1024; int bits = 10;
	while (n_slots < (uint64_t)mi->n_keys * 2) n_slots <<= 1, ++bits;
	mi->n_slots = n_slots, mi->slot_shift = 64 - bits;
	MMG_CUDA(cudaMalloc(&mi->d_slots, n_slots * sizeof(IdxSlot)));
	MMG_LAUNCH(c, k_fill_u64, mmg_blocks(n_slots * 2, 256), 256, 0, reinterpret_cast<uint64_t*>(mi->d_slots), n_slots * 2, MMG_SLOT_EMPTY);
	if (mi->n_keys)
		MMG_LAUNCH(c, k_idx_insert, mmg_blocks(mi->n_keys, 256), 256, 0, d_ukey, mi->d_counts, d_ustart, mi->n_keys, mi->d_pos, mi->d_slots, n_slots - 1, mi->slot_shift);
	return MMG_OK;
}

static int idx_seq_table(mmg_ctx_t *c, mmg_idx_t *mi)
{
	MMG_CUDA(cudaMalloc(&mi->d_seq_off, (size_t)(mi->n_seq + 1) * 8));
	MMG_CUDA(cudaMalloc(&mi->d_seq_len, (size_t)(mi->n_seq + 1) * 4));
	MMG_CUDA(cudaMemcpyAsync(mi->d_seq_off, mi->h_seq_off.data(), (size_t)(mi->n_seq + 1) * 8, cudaMemcpyHostToDevice, c->stream));
	MMG_CUDA(cudaMemcpyAsync(mi->d_seq_len, mi->h_seq_len.data(), (size_t)(mi->n_seq + 1) * 4, cudaMemcpyHostToDevice, c->stream));
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	return MMG_OK;
}

static mmg_idx_t *idx_new(mmg_ctx_t *c, int w, int k, int is_hpc, int n_seq, const uint32_t *lens)
{
	mmg_idx_t *mi = new mmg_idx_s();
	mi->dev = c->dev, mi->w = w, mi->k = k, mi->is_hpc = is_hpc, mi->n_seq = n_seq;
	mi->h_seq_off.resize(n_seq + 1); mi->h_seq_len.resize(n_seq + 1);
	uint64_t tot = 0;
	for (int i = 0; i < n_seq; ++i) { mi->h_seq_off[i] = tot; mi->h_seq_len[i] = lens[i]; tot += lens[i]; }
	mi->h_seq_off[n_seq] = tot; mi->h_seq_len[n_seq] = 0;
	mi->total_len = tot;
	return mi;
}

extern "C" int mmg_idx_build(mmg_ctx_t *c, int w, int k, int is_hpc, int n_seq, const char *const *seqs, const uint32_t *lens, mmg_idx_t **out)
{
	*out = nullptr;
	if (w < 1 || w > MMG_MAX_W || k < 1 || k > 28 || n_seq <= 0) {
		mmg_set_error("mmg_idx_build: need 1<=w<=%d, 1<=k<=28, n_seq>0", MMG_MAX_W);
		return (w > MMG_MAX_W) ? MMG_ELIMIT : MMG_EINVAL;
	}
	MMG_CUDA(cudaSetDevice(c->dev));
	mmg_idx_t *mi = idx_new(c, w, k, is_hpc, n_seq, lens);
	const uint64_t tot = mi->total_len;
	int rc = MMG_OK;
	uint8_t *d_ascii = nullptr;
	SketchUnit *d_units = nullptr;
	uint64_t *d_key[2] = {nullptr, nullptr}, *d_val[2] = {nullptr, nullptr}, *d_ukey = nullptr;
	int64_t *d_ustart = nullptr, *d_nruns = nullptr;
	DevBuf cnt, off, mv;
	auto cleanup = [&]() {
		cudaFree(d_ascii); cudaFree(d_units); cudaFree(d_key[0]); cudaFree(d_key[1]); cudaFree(d_val[0]); cudaFree(d_val[1]);
		cudaFree(d_ukey); cudaFree(d_ustart); cudaFree(d_nruns); cnt.release(); off.release(); mv.release();
	};
#define IDX_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { mmg_set_error("%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); cleanup(); mmg_idx_free(mi); return MMG_ECUDA; } } while (0)
#define IDX_TRY(call) do { rc = (call); if (rc != MMG_OK) { cleanup(); mmg_idx_free(mi); return rc; } } while (0)

	// 1. upload ASCII (through the pinned bases buffer of staging slot 0), pack to 4 bits
	IDX_CUDA(cudaMalloc(&d_ascii, tot + 16));
	IDX_CUDA(cudaMalloc(&mi->d_S, ((tot + 7) / 8 + 4) * 4));
	{
		const size_t stage = 64u << 20;
		IDX_TRY(mmg_stage_grow(c, 0, &StageSlot::bases, stage));
		uint8_t *h = c->stage[0].bases.as<uint8_t>();
		size_t fill = 0; uint64_t done = 0;
		for (int i = 0; i < n_seq; ++i) {
			uint64_t o = 0;
			while (o < lens[i]) {
				size_t l = lens[i] - o < stage - fill ? (size_t)(lens[i] - o) : stage - fill;
				memcpy(h + fill, seqs[i] + o, l);
				fill += l, o += l;
				if (fill == stage) {
					IDX_CUDA(cudaMemcpyAsync(d_ascii + done, h, fill, cudaMemcpyHostToDevice, c->stream));
					IDX_CUDA(cudaStreamSynchronize(c->stream));
					done += fill, fill = 0;
				}
			}
		}
		if (fill) {
			IDX_CUDA(cudaMemcpyAsync(d_ascii + done, h, fill, cudaMemcpyHostToDevice, c->stream));
			IDX_CUDA(cudaStreamSynchronize(c->stream));
		}
	}
	IDX_CUDA(cudaMemsetAsync(mi->d_S, 0, ((tot + 7) / 8 + 4) * 4, c->stream));
	if (tot) {
		k_pack_ref<<<mmg_blocks((tot + 7) / 8, 256), 256, 0, c->stream>>>(d_ascii, tot, mi->d_S); ++c->launches;
		IDX_CUDA(cudaGetLastError());
	}
	IDX_CUDA(cudaStreamSynchronize(c->stream));
	cudaFree(d_ascii); d_ascii = nullptr;

	// 2. work units: chunks of MMG_IDX_CHUNK emission positions (whole sequences with HPC)
	std::vector<SketchUnit> units;
	for (int i = 0; i < n_seq; ++i) {
		if (lens[i] == 0) continue;
		const int chunk = is_hpc ? (int)lens[i] : MMG_IDX_CHUNK;
		for (uint32_t s = 0; s < lens[i]; s += chunk) {
			SketchUnit u;
			u.off = mi->h_seq_off[i], u.len = (int32_t)lens[i], u.rid = (uint32_t)i, u.y_add = 0;
			u.emit_start = (int32_t)s, u.emit_end = (int32_t)(s + chunk < lens[i] ? s + chunk : lens[i]);
			units.push_back(u);
		}
	}
	const int n_units = (int)units.size();
	IDX_CUDA(cudaMalloc(&d_units, (size_t)(n_units + 1) * sizeof(SketchUnit)));
	if (n_units) IDX_CUDA(cudaMemcpy(d_units, units.data(), (size_t)n_units * sizeof(SketchUnit), cudaMemcpyHostToDevice));

	// 3. sketch
	int64_t n_mini = 0;
	IDX_TRY(mmg_run_sketch(c, mi->d_S, d_units, n_units, w, k, is_hpc, cnt, off, mv, &n_mini, false, 0));
	IDX_CUDA(cudaStreamSynchronize(c->stream));
	cudaFree(d_units); d_units = nullptr; cnt.release(); off.release();
	mi->n_pos = (uint64_t)n_mini;

	// 4. sort (minimizer, position) by minimizer; the sort is stable and positions were emitted in
	//    ascending (rid, pos) order, so each run comes out position-sorted as index.c:230 requires
	const size_t nm = (size_t)n_mini + 1;
	for (int i = 0; i < 2; ++i) { IDX_CUDA(cudaMalloc(&d_key[i], nm * 8)); IDX_CUDA(cudaMalloc(&d_val[i], nm * 8)); }
	if (n_mini) {
		k_split_kv<<<mmg_blocks(n_mini, 256), 256, 0, c->stream>>>(mv.as<mm128>(), n_mini, d_key[0], d_val[0]); ++c->launches;
		IDX_CUDA(cudaGetLastError());
	}
	IDX_CUDA(cudaStreamSynchronize(c->stream));
	mv.release();
	cub::DoubleBuffer<uint64_t> kb(d_key[0], d_key[1]), vb(d_val[0], d_val[1]);
	if (n_mini) {
		size_t tmp = 0;
		cub::DeviceRadixSort::SortPairs(nullptr, tmp, kb, vb, (int64_t)n_mini, 0, 2 * k, c->stream);
		IDX_TRY(c->d_cub.ensure(tmp));
		IDX_CUDA(cub::DeviceRadixSort::SortPairs(c->d_cub.p, tmp, kb, vb, (int64_t)n_mini, 0, 2 * k, c->stream));
		++c->launches;
	}
	// 5. distinct minimizers and their run lengths
	IDX_CUDA(cudaMalloc(&d_ukey, nm * 8));
	IDX_CUDA(cudaMalloc(&mi->d_counts, nm * 4));
	IDX_CUDA(cudaMalloc(&d_nruns, 8));
	IDX_CUDA(cudaMemsetAsync(d_nruns, 0, 8, c->stream));
	if (n_mini) {
		size_t tmp = 0;
		cub::DeviceRunLengthEncode::Encode(nullptr, tmp, kb.Current(), d_ukey, mi->d_counts, d_nruns, (int64_t)n_mini, c->stream);
		IDX_TRY(c->d_cub.ensure(tmp));
		IDX_CUDA(cub::DeviceRunLengthEncode::Encode(c->d_cub.p, tmp, kb.Current(), d_ukey, mi->d_counts, d_nruns, (int64_t)n_mini, c->stream));
		++c->launches;
	}
	int64_t n_keys = 0;
	IDX_CUDA(cudaMemcpyAsync(&n_keys, d_nruns, 8, cudaMemcpyDeviceToHost, c->stream));
	IDX_CUDA(cudaStreamSynchronize(c->stream));
	mi->n_keys = n_keys;
	IDX_CUDA(cudaMalloc(&d_ustart, (size_t)(n_keys + 1) * 8));
	if (n_keys) {
		size_t tmp = 0;
		cub::DeviceScan::ExclusiveSum(nullptr, tmp, mi->d_counts, d_ustart, n_keys, c->stream);
		IDX_TRY(c->d_cub.ensure(tmp));
		IDX_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, mi->d_counts, d_ustart, n_keys, c->stream));
		++c->launches;
	}
	// positions: keep the sorted value array as pos[]
	mi->d_pos = vb.Current();
	if (vb.Current() == d_val[0]) d_val[0] = nullptr; else d_val[1] = nullptr;
	// 6. table, 7. sequence table
	IDX_TRY(idx_table(c, mi, d_ukey, d_ustart));
	IDX_TRY(idx_seq_table(c, mi));
	cleanup();
	c->d_cub.release();
	*out = mi;
	return MMG_OK;
#undef IDX_CUDA
#undef IDX_TRY
}

// ------------------------------------------------------------------ build from an index file's minimizer lists

#define LISTS_SINGLE (1ULL << 63)
#define LISTS_SHORT 32 // runs up to this long are copied by one thread, longer ones by a warp

__global__ void k_lists_keys(const uint64_t *__restrict__ key, int64_t n, uint64_t *__restrict__ skey, uint32_t *__restrict__ sidx)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	skey[i] = key[i] & ~LISTS_SINGLE, sidx[i] = (uint32_t)i;
}

// file order -> minimizer order; bad[0] is set when a minimizer is listed twice
__global__ void k_lists_gather(const uint64_t *__restrict__ skey, const uint32_t *__restrict__ sidx, int64_t n, const uint64_t *__restrict__ key,
                               const uint32_t *__restrict__ cnt, const uint64_t *__restrict__ src, uint32_t *__restrict__ ucnt,
                               uint64_t *__restrict__ usrc, unsigned int *bad)
{
	const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	const uint32_t i = sidx[j];
	const bool single = (key[i] & LISTS_SINGLE) != 0;
	ucnt[j] = single ? 1u : cnt[i];
	usrc[j] = src[i] | (single ? LISTS_SINGLE : 0);
	if (j > 0 && skey[j] == skey[j - 1]) atomicOr(bad, 1u);
}

// a thread per short run; the long ones are queued for k_lists_scatter_long.  A singleton's one position is its own value.
__global__ void k_lists_scatter(const uint32_t *__restrict__ ucnt, const uint64_t *__restrict__ usrc, const int64_t *__restrict__ ustart, int64_t n,
                                const uint64_t *__restrict__ p, uint64_t *__restrict__ pos, int64_t *__restrict__ long_runs, unsigned long long *n_long)
{
	const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (j >= n) return;
	const uint32_t m = ucnt[j];
	const uint64_t s = usrc[j];
	uint64_t *dst = pos + ustart[j];
	if (s & LISTS_SINGLE) { dst[0] = s & ~LISTS_SINGLE; return; }
	if (m > LISTS_SHORT) { long_runs[atomicAdd(n_long, 1ULL)] = j; return; }
	for (uint32_t t = 0; t < m; ++t) dst[t] = p[s + t];
}

__global__ void k_lists_scatter_long(const uint32_t *__restrict__ ucnt, const uint64_t *__restrict__ usrc, const int64_t *__restrict__ ustart,
                                     const int64_t *__restrict__ long_runs, const unsigned long long *n_long, const uint64_t *__restrict__ p,
                                     uint64_t *__restrict__ pos)
{
	const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
	const int lane = threadIdx.x & 31;
	for (int64_t r = warp; r < (int64_t)*n_long; r += n_warps) {
		const int64_t j = long_runs[r];
		const uint32_t m = ucnt[j];
		const uint64_t *s = p + usrc[j];
		uint64_t *dst = pos + ustart[j];
		for (uint32_t t = lane; t < m; t += 32) dst[t] = s[t];
	}
}

// host -> device through the pinned bases buffer of staging slot 0, in chunks: a human-size p[] is several GB
static int upload_chunked(mmg_ctx_t *c, void *dst, const void *src, size_t bytes)
{
	const size_t stage = 64u << 20;
	if (bytes == 0) return MMG_OK;
	MMG_TRY(mmg_stage_grow(c, 0, &StageSlot::bases, stage));
	uint8_t *h = c->stage[0].bases.as<uint8_t>();
	for (size_t o = 0; o < bytes; o += stage) {
		const size_t l = bytes - o < stage ? bytes - o : stage;
		memcpy(h, static_cast<const uint8_t*>(src) + o, l);
		MMG_CUDA(cudaMemcpyAsync(static_cast<uint8_t*>(dst) + o, h, l, cudaMemcpyHostToDevice, c->stream));
		MMG_CUDA(cudaStreamSynchronize(c->stream));
	}
	return MMG_OK;
}

extern "C" int mmg_idx_build_lists(mmg_ctx_t *c, int w, int k, int is_hpc, int n_seq, const uint32_t *lens, int64_t n_keys, const uint64_t *key,
                                   const uint32_t *cnt, const uint64_t *src, uint64_t n_p, const uint64_t *p, mmg_idx_t **out)
{
	*out = nullptr;
	if (w < 1 || w > MMG_MAX_W || k < 1 || k > 28 || n_seq <= 0 || n_keys < 0 || n_keys >= (1LL << 32)) {
		mmg_set_error("mmg_idx_build_lists: need 1<=w<=%d, 1<=k<=28, n_seq>0, 0<=n_keys<2^32", MMG_MAX_W);
		return (w > MMG_MAX_W) ? MMG_ELIMIT : MMG_EINVAL;
	}
	for (int64_t i = 0; i < n_keys; ++i) { // nothing out of range reaches the device
		if ((key[i] & ~LISTS_SINGLE) >> (2 * k)) { mmg_set_error("mmg_idx_build_lists: minimizer %lld has more than %d bits", (long long)i, 2 * k); return MMG_EINVAL; }
		if (!(key[i] & LISTS_SINGLE) && (cnt[i] == 0 || src[i] > n_p || cnt[i] > n_p - src[i])) {
			mmg_set_error("mmg_idx_build_lists: the positions of minimizer %lld lie outside p[] (%llu entries)", (long long)i, (unsigned long long)n_p);
			return MMG_EINVAL;
		}
	}
	MMG_CUDA(cudaSetDevice(c->dev));
	mmg_idx_t *mi = idx_new(c, w, k, is_hpc, n_seq, lens);
	mi->n_keys = n_keys;
	int rc = MMG_OK;
	const size_t nk = (size_t)n_keys + 1;
	uint64_t *d_key = nullptr, *d_src = nullptr, *d_p = nullptr, *d_sk[2] = {nullptr, nullptr}, *d_usrc = nullptr;
	uint32_t *d_cnt = nullptr, *d_si[2] = {nullptr, nullptr};
	int64_t *d_ustart = nullptr, *d_long = nullptr;
	unsigned long long *d_ctr = nullptr; // [0] long runs, [1] a minimizer listed twice
	auto cleanup = [&]() {
		cudaFree(d_key); cudaFree(d_src); cudaFree(d_p); cudaFree(d_sk[0]); cudaFree(d_sk[1]); cudaFree(d_usrc);
		cudaFree(d_cnt); cudaFree(d_si[0]); cudaFree(d_si[1]); cudaFree(d_ustart); cudaFree(d_long); cudaFree(d_ctr);
	};
#define IDX_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { mmg_set_error("%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); cleanup(); mmg_idx_free(mi); return MMG_ECUDA; } } while (0)
#define IDX_TRY(call) do { rc = (call); if (rc != MMG_OK) { cleanup(); mmg_idx_free(mi); return rc; } } while (0)
#define LAUNCH_IDX(kern, grid, block, ...) do { kern<<<(grid), (block), 0, c->stream>>>(__VA_ARGS__); ++c->launches; IDX_CUDA(cudaGetLastError()); } while (0)

	// 1. upload the lists as the file gives them
	IDX_CUDA(cudaMalloc(&d_key, nk * 8));
	IDX_CUDA(cudaMalloc(&d_cnt, nk * 4));
	IDX_CUDA(cudaMalloc(&d_src, nk * 8));
	IDX_CUDA(cudaMalloc(&d_p, ((size_t)n_p + 1) * 8));
	IDX_TRY(upload_chunked(c, d_key, key, (size_t)n_keys * 8));
	IDX_TRY(upload_chunked(c, d_cnt, cnt, (size_t)n_keys * 4));
	IDX_TRY(upload_chunked(c, d_src, src, (size_t)n_keys * 8));
	IDX_TRY(upload_chunked(c, d_p, p, (size_t)n_p * 8));

	// 2. order by minimizer
	for (int i = 0; i < 2; ++i) { IDX_CUDA(cudaMalloc(&d_sk[i], nk * 8)); IDX_CUDA(cudaMalloc(&d_si[i], nk * 4)); }
	cub::DoubleBuffer<uint64_t> kb(d_sk[0], d_sk[1]);
	cub::DoubleBuffer<uint32_t> ib(d_si[0], d_si[1]);
	if (n_keys) {
		LAUNCH_IDX(k_lists_keys, mmg_blocks(n_keys, 256), 256, d_key, n_keys, d_sk[0], d_si[0]);
		size_t tmp = 0;
		cub::DeviceRadixSort::SortPairs(nullptr, tmp, kb, ib, n_keys, 0, 2 * k, c->stream);
		IDX_TRY(c->d_cub.ensure(tmp));
		IDX_CUDA(cub::DeviceRadixSort::SortPairs(c->d_cub.p, tmp, kb, ib, n_keys, 0, 2 * k, c->stream));
		++c->launches;
	}
	// 3. counts in minimizer order and each run's start in pos[]
	IDX_CUDA(cudaMalloc(&mi->d_counts, nk * 4));
	IDX_CUDA(cudaMalloc(&d_usrc, nk * 8));
	IDX_CUDA(cudaMalloc(&d_ustart, (nk + 1) * 8));
	IDX_CUDA(cudaMalloc(&d_ctr, 16));
	IDX_CUDA(cudaMemsetAsync(d_ctr, 0, 16, c->stream));
	IDX_CUDA(cudaMemsetAsync(mi->d_counts, 0, nk * 4, c->stream)); // counts[n_keys] = 0: the scan leaves the total in ustart[n_keys]
	if (n_keys)
		LAUNCH_IDX(k_lists_gather, mmg_blocks(n_keys, 256), 256, kb.Current(), ib.Current(), n_keys, d_key, d_cnt, d_src, mi->d_counts, d_usrc,
		               reinterpret_cast<unsigned int*>(d_ctr + 1));
	{
		size_t tmp = 0;
		cub::DeviceScan::ExclusiveSum(nullptr, tmp, mi->d_counts, d_ustart, (int64_t)nk, c->stream);
		IDX_TRY(c->d_cub.ensure(tmp));
		IDX_CUDA(cub::DeviceScan::ExclusiveSum(c->d_cub.p, tmp, mi->d_counts, d_ustart, (int64_t)nk, c->stream));
		++c->launches;
	}
	int64_t n_pos = 0;
	unsigned long long dup = 0;
	IDX_CUDA(cudaMemcpyAsync(&n_pos, d_ustart + n_keys, 8, cudaMemcpyDeviceToHost, c->stream));
	IDX_CUDA(cudaMemcpyAsync(&dup, d_ctr + 1, 8, cudaMemcpyDeviceToHost, c->stream));
	IDX_CUDA(cudaStreamSynchronize(c->stream));
	if (dup) { mmg_set_error("mmg_idx_build_lists: a minimizer is listed more than once"); cleanup(); mmg_idx_free(mi); return MMG_EINVAL; }
	mi->n_pos = (uint64_t)n_pos;
	// only the sorted minimizers, the runs and p[] are read from here on
	cudaFree(d_key); d_key = nullptr; cudaFree(d_cnt); d_cnt = nullptr; cudaFree(d_src); d_src = nullptr;
	cudaFree(d_si[0]); cudaFree(d_si[1]); d_si[0] = d_si[1] = nullptr;
	if (kb.Current() == d_sk[0]) { cudaFree(d_sk[1]); d_sk[1] = nullptr; } else { cudaFree(d_sk[0]); d_sk[0] = nullptr; }
	// 4. scatter every run into pos[], its positions in the order the file lists them
	IDX_CUDA(cudaMalloc(&mi->d_pos, (mi->n_pos + 1) * 8));
	IDX_CUDA(cudaMalloc(&d_long, nk * 8));
	if (n_keys) {
		LAUNCH_IDX(k_lists_scatter, mmg_blocks(n_keys, 256), 256, mi->d_counts, d_usrc, d_ustart, n_keys, d_p, mi->d_pos, d_long, d_ctr);
		LAUNCH_IDX(k_lists_scatter_long, 148 * 16, 256, mi->d_counts, d_usrc, d_ustart, d_long, d_ctr, d_p, mi->d_pos);
	}
	// 5. the table, as mmg_idx_build fills it from the same (minimizer, count, start); no sequence is kept
	IDX_TRY(idx_table(c, mi, kb.Current(), d_ustart));
	IDX_TRY(idx_seq_table(c, mi));
	cleanup();
	c->d_cub.release();
	*out = mi;
	return MMG_OK;
#undef IDX_CUDA
#undef IDX_TRY
#undef LAUNCH_IDX
}

extern "C" int64_t mmg_idx_n_minimizers(const mmg_idx_t *mi) { return (int64_t)mi->n_pos; }
extern "C" int64_t mmg_idx_n_keys(const mmg_idx_t *mi) { return mi->n_keys; }
extern "C" uint64_t mmg_idx_total_len(const mmg_idx_t *mi) { return mi->total_len; }
extern "C" size_t mmg_idx_bytes(const mmg_idx_t *mi)
{
	return (mi->d_S ? ((mi->total_len + 7) / 8) * 4 : 0) + mi->n_slots * sizeof(IdxSlot) + mi->n_pos * 8 + (size_t)mi->n_seq * 12;
}
extern "C" int mmg_idx_has_seq(const mmg_idx_t *mi) { return mi->d_S != nullptr; }

extern "C" int mmg_idx_copy_S(const mmg_idx_t *mi, uint32_t *S_host)
{
	if (mi->d_S == nullptr) { mmg_set_error("mmg_idx_copy_S: the index holds no sequence (built from a .mmi written with --idx-no-seq)"); return MMG_EINVAL; }
	MMG_CUDA(cudaSetDevice(mi->dev));
	MMG_CUDA(cudaMemcpy(S_host, mi->d_S, ((mi->total_len + 7) / 8) * 4, cudaMemcpyDeviceToHost));
	return MMG_OK;
}

extern "C" int mmg_idx_cal_max_occ(mmg_idx_t *mi, float f, int32_t *thres)
{ // index.c:164-185: the (1-f) quantile of per-minimizer occurrence counts, plus one
	*thres = INT32_MAX;
	if (f <= 0.) return MMG_OK;
	if (mi->n_keys == 0) { *thres = 1; return MMG_OK; }
	if (mi->d_counts == nullptr) { mmg_set_error("index replica has no occurrence table; query the source index"); return MMG_EINVAL; }
	MMG_CUDA(cudaSetDevice(mi->dev));
	uint32_t *d_sorted = nullptr; void *d_tmp = nullptr; size_t tmp = 0;
	MMG_CUDA(cudaMalloc(&d_sorted, (size_t)mi->n_keys * 4));
	cub::DeviceRadixSort::SortKeys(nullptr, tmp, mi->d_counts, d_sorted, mi->n_keys);
	MMG_CUDA(cudaMalloc(&d_tmp, tmp));
	cudaError_t e = cub::DeviceRadixSort::SortKeys(d_tmp, tmp, mi->d_counts, d_sorted, mi->n_keys);
	uint32_t v = 0;
	const size_t kk = (size_t)(uint32_t)((1. - f) * mi->n_keys);
	if (e == cudaSuccess) e = cudaMemcpy(&v, d_sorted + kk, 4, cudaMemcpyDeviceToHost);
	cudaFree(d_sorted); cudaFree(d_tmp);
	if (e != cudaSuccess) { mmg_set_error("mmg_idx_cal_max_occ: %s", cudaGetErrorString(e)); return MMG_ECUDA; }
	*thres = (int32_t)(v + 1);
	return MMG_OK;
}

extern "C" int mmg_idx_get(mmg_ctx_t *c, const mmg_idx_t *mi, int n_q, const uint64_t *minier, int32_t *n, int max_pos, uint64_t *pos)
{
	if (n_q <= 0) return MMG_OK;
	MMG_CUDA(cudaSetDevice(c->dev));
	uint64_t *d_q = nullptr, *d_pos = nullptr; int32_t *d_n = nullptr;
	MMG_CUDA(cudaMalloc(&d_q, (size_t)n_q * 8));
	MMG_CUDA(cudaMalloc(&d_n, (size_t)n_q * 4));
	MMG_CUDA(cudaMalloc(&d_pos, (size_t)n_q * (max_pos > 0 ? max_pos : 1) * 8));
	MMG_CUDA(cudaMemcpyAsync(d_q, minier, (size_t)n_q * 8, cudaMemcpyHostToDevice, c->stream));
	MMG_LAUNCH(c, k_idx_get, mmg_blocks(n_q, 128), 128, 0, mi->view(), n_q, d_q, d_n, max_pos, d_pos);
	MMG_CUDA(cudaMemcpyAsync(n, d_n, (size_t)n_q * 4, cudaMemcpyDeviceToHost, c->stream));
	if (max_pos > 0) MMG_CUDA(cudaMemcpyAsync(pos, d_pos, (size_t)n_q * max_pos * 8, cudaMemcpyDeviceToHost, c->stream));
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	cudaFree(d_q); cudaFree(d_n); cudaFree(d_pos);
	return MMG_OK;
}

extern "C" int mmg_idx_export(const mmg_idx_t *mi, mmg_idx_image_t *img)
{
	img->w = mi->w, img->k = mi->k, img->is_hpc = mi->is_hpc, img->n_seq = mi->n_seq;
	img->total_len = mi->total_len, img->n_slots = mi->n_slots, img->n_pos = mi->n_pos, img->n_keys = mi->n_keys;
	img->d_S = mi->d_S, img->bytes_S = mi->d_S ? ((mi->total_len + 7) / 8) * 4 : 0;
	img->d_seq_off = mi->d_seq_off, img->bytes_seq_off = (size_t)(mi->n_seq + 1) * 8;
	img->d_seq_len = mi->d_seq_len, img->bytes_seq_len = (size_t)(mi->n_seq + 1) * 4;
	img->d_slots = mi->d_slots, img->bytes_slots = mi->n_slots * sizeof(IdxSlot);
	img->d_pos = mi->d_pos, img->bytes_pos = mi->n_pos * 8;
	return MMG_OK;
}

extern "C" int mmg_idx_alloc_like(mmg_ctx_t *c, mmg_idx_image_t *img, mmg_idx_t **out)
{
	*out = nullptr;
	MMG_CUDA(cudaSetDevice(c->dev));
	mmg_idx_t *mi = new mmg_idx_s();
	mi->dev = c->dev, mi->w = img->w, mi->k = img->k, mi->is_hpc = img->is_hpc, mi->n_seq = img->n_seq;
	mi->total_len = img->total_len, mi->n_slots = img->n_slots, mi->n_pos = img->n_pos, mi->n_keys = img->n_keys;
	int bits = 0; while ((1ULL << bits) < mi->n_slots) ++bits;
	mi->slot_shift = 64 - bits;
	int rc = idx_alloc(mi, img->bytes_S > 0 || img->total_len == 0); // an index without sequence has total_len > 0 and no S bytes
	if (rc != MMG_OK) { mmg_idx_free(mi); return rc; }
	img->d_S = mi->d_S, img->d_seq_off = mi->d_seq_off, img->d_seq_len = mi->d_seq_len, img->d_slots = mi->d_slots, img->d_pos = mi->d_pos;
	*out = mi;
	return MMG_OK;
}

// call after the image buffers were filled (e.g. by an NCCL broadcast) to refresh host-side tables
extern "C" int mmg_idx_finalize(mmg_idx_t *mi)
{
	MMG_CUDA(cudaSetDevice(mi->dev));
	mi->h_seq_off.resize(mi->n_seq + 1); mi->h_seq_len.resize(mi->n_seq + 1);
	MMG_CUDA(cudaMemcpy(mi->h_seq_off.data(), mi->d_seq_off, (size_t)(mi->n_seq + 1) * 8, cudaMemcpyDeviceToHost));
	MMG_CUDA(cudaMemcpy(mi->h_seq_len.data(), mi->d_seq_len, (size_t)(mi->n_seq + 1) * 4, cudaMemcpyDeviceToHost));
	return MMG_OK;
}

extern "C" int mmg_idx_clone_to(mmg_ctx_t *c, const mmg_idx_t *src, mmg_idx_t **dst)
{
	mmg_idx_image_t s, d;
	mmg_idx_export(src, &s);
	d = s;
	MMG_TRY(mmg_idx_alloc_like(c, &d, dst));
	int can = 0;
	if (src->dev != c->dev) {
		cudaDeviceCanAccessPeer(&can, c->dev, src->dev);
		if (can) { cudaError_t e = cudaDeviceEnablePeerAccess(src->dev, 0); if (e != cudaSuccess) cudaGetLastError(); }
	}
	if (s.bytes_S) MMG_CUDA(cudaMemcpyPeerAsync(d.d_S, c->dev, s.d_S, src->dev, s.bytes_S, c->stream));
	MMG_CUDA(cudaMemcpyPeerAsync(d.d_seq_off, c->dev, s.d_seq_off, src->dev, s.bytes_seq_off, c->stream));
	MMG_CUDA(cudaMemcpyPeerAsync(d.d_seq_len, c->dev, s.d_seq_len, src->dev, s.bytes_seq_len, c->stream));
	MMG_CUDA(cudaMemcpyPeerAsync(d.d_slots, c->dev, s.d_slots, src->dev, s.bytes_slots, c->stream));
	MMG_CUDA(cudaMemcpyPeerAsync(d.d_pos, c->dev, s.d_pos, src->dev, s.bytes_pos, c->stream));
	MMG_CUDA(cudaStreamSynchronize(c->stream));
	(*dst)->h_seq_off = src->h_seq_off; (*dst)->h_seq_len = src->h_seq_len;
	return MMG_OK;
}

__global__ void k_count_ones(const uint32_t *__restrict__ cnt, int64_t n, unsigned long long *out)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	const int one = i < n && cnt[i] == 1;
	const unsigned m = __ballot_sync(0xffffffffu, one);
	if ((threadIdx.x & 31) == 0 && m) atomicAdd(out, (unsigned long long)__popc(m));
}

extern "C" int64_t mmg_idx_n_singletons(const mmg_idx_t *mi)
{ // for mm_idx_stat (index.c:117): distinct minimizers that occur once
	if (mi->d_counts == nullptr || mi->n_keys == 0) return 0;
	cudaSetDevice(mi->dev);
	unsigned long long *d = nullptr, h = 0;
	if (cudaMalloc(&d, 8) != cudaSuccess) return -1;
	cudaMemset(d, 0, 8);
	k_count_ones<<<mmg_blocks(mi->n_keys, 256), 256>>>(mi->d_counts, mi->n_keys, d);
	cudaMemcpy(&h, d, 8, cudaMemcpyDeviceToHost);
	cudaFree(d);
	return (int64_t)h;
}

extern "C" int mmg_memcpy_d2d(void *dst, const void *src, size_t bytes)
{ // same-device copy helper for callers that stage index buffers through their own tensors
	MMG_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToDevice));
	return MMG_OK;
}

// ---- table export in the reference's bucket order (input of mm_idx_dump, index.c:438-477)

struct SlotLive { __device__ bool operator()(const IdxSlot &s) const { return s.key != MMG_SLOT_EMPTY; } };

// sort key = (minimizer & bucket mask, minimizer >> b): the order worker_post (index.c:191-243) visits keys in
__global__ void k_bucket_keys(const IdxSlot *__restrict__ live, int64_t n, int b, int kbits, uint64_t *__restrict__ skey, uint64_t *__restrict__ sidx)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const uint64_t m = live[i].key & ~MMG_SLOT_SINGLE;
	skey[i] = (m & ((1ULL << b) - 1)) << (kbits - b) | m >> b;
	sidx[i] = (uint64_t)i;
}

__global__ void k_bucket_gather(const IdxSlot *__restrict__ live, const uint64_t *__restrict__ sidx, int64_t n, uint64_t *__restrict__ keys, uint64_t *__restrict__ vals)
{
	const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	const IdxSlot s = live[sidx[i]];
	keys[i] = s.key, vals[i] = s.val;
}

extern "C" int mmg_idx_export_sorted(mmg_ctx_t *c, const mmg_idx_t *mi, int b, uint64_t *keys, uint64_t *vals, uint64_t *pos)
{
	const int kbits = 2 * mi->k;
	if (b < 0 || b > kbits || kbits > 62) { mmg_set_error("mmg_idx_export_sorted: bucket bits %d do not fit a %d-bit minimizer", b, kbits); return MMG_EINVAL; }
	MMG_CUDA(cudaSetDevice(mi->dev));
	const int64_t n = mi->n_keys;
	if (pos && mi->n_pos) MMG_CUDA(cudaMemcpy(pos, mi->d_pos, mi->n_pos * 8, cudaMemcpyDeviceToHost));
	if (n == 0) return MMG_OK;
	IdxSlot *d_live = nullptr; int64_t *d_n = nullptr; void *d_tmp = nullptr;
	uint64_t *d_k[2] = {nullptr, nullptr}, *d_v[2] = {nullptr, nullptr}, *d_ok = nullptr, *d_ov = nullptr;
	auto cleanup = [&]() { cudaFree(d_live); cudaFree(d_n); cudaFree(d_tmp); cudaFree(d_k[0]); cudaFree(d_k[1]); cudaFree(d_v[0]); cudaFree(d_v[1]); cudaFree(d_ok); cudaFree(d_ov); };
#define EXP_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { mmg_set_error("%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); cleanup(); return MMG_ECUDA; } } while (0)
	EXP_CUDA(cudaMalloc(&d_live, (size_t)n * sizeof(IdxSlot)));
	EXP_CUDA(cudaMalloc(&d_n, 8));
	size_t tmp = 0, tmp2 = 0;
	cub::DeviceSelect::If(nullptr, tmp, mi->d_slots, d_live, d_n, (int64_t)mi->n_slots, SlotLive(), c->stream);
	for (int i = 0; i < 2; ++i) { EXP_CUDA(cudaMalloc(&d_k[i], (size_t)n * 8)); EXP_CUDA(cudaMalloc(&d_v[i], (size_t)n * 8)); }
	cub::DoubleBuffer<uint64_t> kb(d_k[0], d_k[1]), vb(d_v[0], d_v[1]);
	cub::DeviceRadixSort::SortPairs(nullptr, tmp2, kb, vb, n, 0, kbits, c->stream);
	if (tmp2 > tmp) tmp = tmp2;
	EXP_CUDA(cudaMalloc(&d_tmp, tmp + 16));
	size_t t1 = tmp;
	EXP_CUDA(cub::DeviceSelect::If(d_tmp, t1, mi->d_slots, d_live, d_n, (int64_t)mi->n_slots, SlotLive(), c->stream));
	++c->launches;
	int64_t n_live = 0;
	EXP_CUDA(cudaMemcpyAsync(&n_live, d_n, 8, cudaMemcpyDeviceToHost, c->stream));
	EXP_CUDA(cudaStreamSynchronize(c->stream));
	if (n_live != n) { mmg_set_error("index table holds %lld keys, %lld expected", (long long)n_live, (long long)n); cleanup(); return MMG_EINVAL; }
	k_bucket_keys<<<mmg_blocks(n, 256), 256, 0, c->stream>>>(d_live, n, b, kbits, d_k[0], d_v[0]); ++c->launches;
	EXP_CUDA(cudaGetLastError());
	t1 = tmp;
	EXP_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, t1, kb, vb, n, 0, kbits, c->stream));
	++c->launches;
	EXP_CUDA(cudaMalloc(&d_ok, (size_t)n * 8));
	EXP_CUDA(cudaMalloc(&d_ov, (size_t)n * 8));
	k_bucket_gather<<<mmg_blocks(n, 256), 256, 0, c->stream>>>(d_live, vb.Current(), n, d_ok, d_ov); ++c->launches;
	EXP_CUDA(cudaGetLastError());
	EXP_CUDA(cudaMemcpyAsync(keys, d_ok, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
	EXP_CUDA(cudaMemcpyAsync(vals, d_ov, (size_t)n * 8, cudaMemcpyDeviceToHost, c->stream));
	EXP_CUDA(cudaStreamSynchronize(c->stream));
	cleanup();
	return MMG_OK;
#undef EXP_CUDA
}
