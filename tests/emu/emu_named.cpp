// CPU emulation harness for the self/dual-hit filters (TEST ONLY, never linked into the product): the harness of emu.cpp plus
// the named form of seed collection, compiled by g++ from the very mmg_core.h code the kernels run.
#include "emu.cpp"

extern "C" {

// tkey/tlen: name key and length of every target, ukey: the fragment's name key (include/mmg.h); *n_named: hits the self/dual
// filters dropped
int64_t emu_collect_named(void *idx, const uint32_t *tkey, const uint32_t *tlen, uint32_t ukey, int heap_sort, int64_t flag, int max_occ, int n_mv,
                          const mm128 *mv, int qlen, mm128 *a, int64_t a_cap, int *rep_len, int *n_mini, uint64_t *mini, int64_t *n_named)
{
	EmuIdx *e = (EmuIdx*)idx;
	std::vector<int32_t> m_n(n_mv + 1); std::vector<uint64_t> m_val(n_mv + 1);
	for (int i = 0; i < n_mv; ++i) m_n[i] = mmg_idx_probe(e->v, mv[i].x >> 8, &m_val[i]);
	int64_t n_a = mmg_frag_plan(mv, m_n.data(), n_mv, max_occ, rep_len, n_mini, mini);
	if (n_a > a_cap) return n_a;
	std::vector<mm128> heap(n_mv + 1); std::vector<RsFrame> stack(n_a / 65 + 4);
	NameFilt nf; nf.tkey = tkey, nf.tlen = tlen, nf.ukey = ukey;
	if (heap_sort) return mmg_fill_heap<true>(mv, m_n.data(), m_val.data(), n_mv, max_occ, e->v.pos, flag, nf, qlen, n_a, heap.data(), a, n_named);
	return mmg_fill_flat<true>(mv, m_n.data(), m_val.data(), n_mv, max_occ, e->v.pos, flag, nf, qlen, a, stack.data(), n_named);
}

}
