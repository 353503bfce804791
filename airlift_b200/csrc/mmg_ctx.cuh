// mmg_ctx.cuh -- internal: context, growable device / pinned buffers, error plumbing.
#pragma once
#include <time.h>
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/mmg.h"
#include "mmg_core.h"

void mmg_set_error(const char *fmt, ...);

#define MMG_CUDA(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
	mmg_set_error("%s:%d: %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); return MMG_ECUDA; } } while (0)
#define MMG_TRY(call) do { int r_ = (call); if (r_ != MMG_OK) return r_; } while (0)

// how often a device / pinned buffer had to be re-allocated (each time costs a device-wide synchronisation): [0] device, [1] pinned
extern unsigned long long g_mmg_grow[2];
extern unsigned long long g_mmg_grow_ns[2]; // wall time spent in those re-allocations (MM2_B200_TRACE reports it when a context is destroyed)
static inline unsigned long long mmg_now_ns() { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (unsigned long long)ts.tv_sec * 1000000000ULL + (unsigned long long)ts.tv_nsec; }

struct DevBuf {
	void *p = nullptr; size_t cap = 0;
	int ensure(size_t bytes) {
		if (bytes <= cap) return MMG_OK;
		const unsigned long long t0 = mmg_now_ns();
		if (p) cudaFree(p);
		p = nullptr; cap = 0;
		__atomic_fetch_add(&g_mmg_grow[0], 1ULL, __ATOMIC_RELAXED);
		size_t want = bytes + bytes / 2 + 256; // generous: a re-allocation in the middle of a run costs a device synchronisation
		cudaError_t e = cudaMalloc(&p, want);
		if (e != cudaSuccess) { cudaGetLastError(); want = bytes + 256; e = cudaMalloc(&p, want); } // HBM is short: take what is needed, no headroom
		__atomic_fetch_add(&g_mmg_grow_ns[0], mmg_now_ns() - t0, __ATOMIC_RELAXED);
		if (e != cudaSuccess) { mmg_set_error("cudaMalloc(%zu): %s", want, cudaGetErrorString(e)); p = nullptr; return MMG_ENOMEM; }
		cap = want;
		return MMG_OK;
	}
	int ensure_keep(size_t bytes, size_t keep, cudaStream_t st) { // grow, carrying the first `keep` bytes over
		if (bytes <= cap) return MMG_OK;
		void *q = nullptr;
		const size_t want = bytes + bytes / 2 + 256;
		cudaError_t e = cudaMalloc(&q, want);
		if (e != cudaSuccess) { mmg_set_error("cudaMalloc(%zu): %s", want, cudaGetErrorString(e)); return MMG_ENOMEM; }
		if (p && keep) { e = cudaMemcpyAsync(q, p, keep, cudaMemcpyDeviceToDevice, st); if (e == cudaSuccess) e = cudaStreamSynchronize(st); }
		if (e != cudaSuccess) { mmg_set_error("growing a device buffer: %s", cudaGetErrorString(e)); cudaFree(q); return MMG_ECUDA; }
		if (p) cudaFree(p);
		p = q, cap = want;
		return MMG_OK;
	}
	void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
	template <class T> T *as() const { return reinterpret_cast<T*>(p); }
};

struct PinBuf {
	void *p = nullptr; size_t cap = 0;
	int ensure(size_t bytes) {
		if (bytes <= cap) return MMG_OK;
		const unsigned long long t0 = mmg_now_ns();
		if (p) cudaFreeHost(p);
		p = nullptr; cap = 0;
		__atomic_fetch_add(&g_mmg_grow[1], 1ULL, __ATOMIC_RELAXED);
		size_t want = bytes + bytes / 2 + 256; // page-locking hundreds of MB again takes ~0.1 s
		cudaError_t e = cudaMallocHost(&p, want);
		__atomic_fetch_add(&g_mmg_grow_ns[1], mmg_now_ns() - t0, __ATOMIC_RELAXED);
		if (e != cudaSuccess) { mmg_set_error("cudaMallocHost(%zu): %s", want, cudaGetErrorString(e)); p = nullptr; return MMG_ENOMEM; }
		cap = want;
		return MMG_OK;
	}
	void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
	template <class T> T *as() const { return reinterpret_cast<T*>(p); }
};

struct mmg_idx_s {
	int dev = 0;
	int32_t w = 0, k = 0, is_hpc = 0, n_seq = 0;
	uint64_t total_len = 0, n_slots = 0, n_pos = 0;
	int64_t n_keys = 0;
	int slot_shift = 0;
	uint32_t *d_S = nullptr;
	uint64_t *d_seq_off = nullptr;
	uint32_t *d_seq_len = nullptr;
	IdxSlot *d_slots = nullptr;
	uint64_t *d_pos = nullptr;
	uint32_t *d_counts = nullptr;      // occurrences per distinct minimizer (for mm_idx_cal_max_occ)
	uint32_t *d_tkey = nullptr;        // name key of every target (mmg_idx_set_name_keys); null until set
	std::vector<uint64_t> h_seq_off;   // host copies: job generation needs them
	std::vector<uint32_t> h_seq_len;
	IdxView view() const {
		IdxView v;
		v.S = d_S, v.seq_off = d_seq_off, v.seq_len = d_seq_len, v.tkey = d_tkey, v.slots = d_slots, v.pos = d_pos;
		v.slot_mask = n_slots - 1, v.slot_shift = slot_shift, v.n_seq = n_seq, v.w = w, v.k = k;
		return v;
	}
};

// one pinned staging slot (mmg_stage): the batch it holds and the event after the last copy out of it
struct StageSlot {
	PinBuf bases, tab, flip, ukey;
	cudaEvent_t drained = nullptr;   // recorded by mmg_upload_stage behind its last copy out of the slot
	int32_t n_frag = 0, n_seq = 0;
	uint64_t n_bases = 0;
	bool has_flip = false, has_ukey = false;
};

// state of the mini-batch currently resident on the device
struct ResidentBatch {
	int32_t n_frag = 0, n_seq = 0, n_units = 0, max_len = 0;
	bool has_ukey = false;           // uploaded with unit keys
	uint64_t n_bases = 0, q_words = 0;
	std::vector<int32_t> n_seg, seg_off, seq_len;
};

struct ProfRec { const char *name; cudaEvent_t a, b; };

// the arrays of one seed-and-chain pass over a list of fragments (mmg_stages.cu: PassTab is their device view)
struct PassArena {
	DevBuf na, aoff, rep, nmini, mini, a, work, u, b, stack, nu, nv;
	void release() { for (DevBuf *d : {&na, &aoff, &rep, &nmini, &mini, &a, &work, &u, &b, &stack, &nu, &nv}) d->release(); }
};

struct mmg_ctx_s {
	int dev = 0;
	cudaStream_t stream = nullptr;
	cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
	long launches = 0;
	uint64_t h2d_bytes = 0, d2h_bytes = 0;
	bool prof_on = false;
	std::vector<ProfRec> prof;       // one record per launch since the last fetch
	std::vector<cudaEvent_t> ev_pool;
	cudaEvent_t prof_event() { if (ev_pool.empty()) { cudaEvent_t e; cudaEventCreate(&e); return e; } cudaEvent_t e = ev_pool.back(); ev_pool.pop_back(); return e; }
	ResidentBatch rb;
	// device arenas (grown on demand, reused across batches)
	DevBuf d_ascii, d_Q, d_seq_len, d_seq_off, d_q_off, d_flip, d_units, d_unit_cnt, d_unit_off, d_mv, d_m_n, d_m_val,
	       d_frag_unit0, d_frag_qlen, d_frag_nseg, d_heap, d_frag_flag, d_frag_iter, d_cub, d_out_u, d_out_a, d_out_mini, d_uoff, d_voff, d_moff,
	       d_frag_list, d_seg_head, d_seg_start, d_seg_avg, d_replay, d_skey, d_sval, d_sseg, d_tie, d_m_aoff, d_hrank, d_hpop, d_hlist, d_seg_li, d_seg_long, d_unit0, d_fseg_off, d_sk_stage, d_heavy, d_ukey;
	// pass[0]: every fragment with the mid_occ cut-off; pass[1]: the fragments re-chained with max_occ (map.c:353-375)
	PassArena pass[2];
	// ksw arenas
	DevBuf k_jobs, k_mem, k_H, k_p, k_cig, k_res, k_cig_out, k_cig_off;
	const void *k_last_res = nullptr; // device {ez, cigar offset} array of the last ksw_launch
	uint64_t k_last_jobs_fast = 0, k_last_cells_fast = 0, k_last_jobs_literal = 0, k_last_cells_literal = 0;
	std::vector<uint32_t> h_k_cig_parts; // CIGARs of an mmg_ksw_batch call that ran in parts
	// post-chaining stages on the device (mmg_post.cu): flat arrays sized by prefix sums, kept across batches
	enum { PB_SHARD, PB_HASH, PB_SEGOFF, PB_READ_FRAG, PB_PERM, PB_CNT, PB_PRE, PB_KEY_IN, PB_VAL_IN, PB_KEY, PB_ASCNT, PB_R0, PB_W, PB_COV, PB_BIG, PB_STACK, PB_N0,
	       PB_CAP, PB_ROFF, PB_NREG, PB_R1, PB_TMP1, PB_PLAN, PB_XSIZE, PB_XOFF, PB_SKEY, PB_SIDX, PB_SBIG, PB_SSTACK, PB_A1, PB_A1OFF, PB_JOBS, PB_CTR, PB_XW,
	       PB_SIZES, PB_OFFS, PB_BLOB, PB_LOGTAB, PB_COUNT };
	DevBuf pb[PB_COUNT];
	int post_logtab_a = 0;             // match score the resident logf tables were made for
	int64_t last_tot_u = 0, last_tot_v = 0; // chains / chained anchors left on the device by the last mmg_seed_chain_resident
	// how many work items took each data-dependent path (mmg_path_counts): [0] fragments re-chained with max_occ, [1] fragments whose
	// heap order was replayed on ranks, [2] ... replayed literally, [3] fragments whose hit tree was built by a warp, [4] extra DP rounds
	// after z-drop cuts, [5] hits cut at a z-drop, [6] seed hits whose merge order was replayed, [7] seed hits the self/dual filters dropped
	uint64_t path[8] = {0, 0, 0, 0, 0, 0, 0, 0};
	StageSlot stage[MMG_STAGE_SLOTS];
	PinBuf h_path;                     // the device's path counters of the batch in flight land here (PathCounters, mmg_stages.cu)
	PinBuf h_p_hash, h_p_nreg, h_p_offs, h_p_blob, h_p_rep;
	PinBuf h_meta, h_out_meta, h_out_u, h_out_a, h_out_mini, h_k_jobs, h_k_res, h_k_cig;
};

// wait until the device has read what slot's last upload copied, then make its buffer `buf` hold `bytes`.  Once slot 1 is in
// use, both slots grow together: page-locking is slow and synchronises the device, so it should happen once, not per slot.
int mmg_stage_grow(mmg_ctx_t *c, int slot, PinBuf StageSlot::*buf, size_t bytes);

// allow the kernels of mmg_ksw.cu / mmg_stages.cu that launch with more than 48 KB of dynamic shared memory to do so on the
// current device: kernel attributes belong to a device, so mmg_init sets them for every context
int mmg_ksw_set_smem_attrs();
int mmg_stages_set_smem_attrs();

#define MMG_LAUNCH(ctx, kern, grid, block, smem, ...) MMG_LAUNCH_AS(ctx, #kern, kern, grid, block, smem, __VA_ARGS__)
// the same under a given profile name (the instantiations of one kernel template share their template's name)
#define MMG_LAUNCH_AS(ctx, label, kern, grid, block, smem, ...) do { \
	ProfRec pr_ = {label, nullptr, nullptr}; \
	if ((ctx)->prof_on) { pr_.a = (ctx)->prof_event(); pr_.b = (ctx)->prof_event(); cudaEventRecord(pr_.a, (ctx)->stream); } \
	kern<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__); ++(ctx)->launches; \
	if ((ctx)->prof_on) { cudaEventRecord(pr_.b, (ctx)->stream); (ctx)->prof.push_back(pr_); } \
	cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) { mmg_set_error("launch %s: %s", label, cudaGetErrorString(e_)); return MMG_ECUDA; } } while (0)

// a library call (cub) on the context's stream, timed like a launch when profiling is on
#define MMG_TIMED(ctx, label, call) do { \
	ProfRec pr_ = {label, nullptr, nullptr}; \
	if ((ctx)->prof_on) { pr_.a = (ctx)->prof_event(); pr_.b = (ctx)->prof_event(); cudaEventRecord(pr_.a, (ctx)->stream); } \
	MMG_CUDA(call); ++(ctx)->launches; \
	if ((ctx)->prof_on) { cudaEventRecord(pr_.b, (ctx)->stream); (ctx)->prof.push_back(pr_); } } while (0)

// account a host<->device copy issued on the context's stream
#define MMG_H2D(ctx, dst, src, n) do { (ctx)->h2d_bytes += (uint64_t)(n); MMG_CUDA(cudaMemcpyAsync((dst), (src), (n), cudaMemcpyHostToDevice, (ctx)->stream)); } while (0)
#define MMG_D2H(ctx, dst, src, n) do { (ctx)->d2h_bytes += (uint64_t)(n); MMG_CUDA(cudaMemcpyAsync((dst), (src), (n), cudaMemcpyDeviceToHost, (ctx)->stream)); } while (0)

static inline unsigned mmg_blocks(size_t n, unsigned per) { return (unsigned)((n + per - 1) / per); }
