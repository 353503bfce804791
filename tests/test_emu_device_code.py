"""CPU-side check of the per-thread device code (airlift_b200/csrc/mmg_core.h compiled by g++ into
build/libmmg_emu.so) against the oracle port.  No GPU needed; the same functions are what the
kernels call, so this pins the logic before it ever runs on the device."""
import ctypes as C
import os
import subprocess
import numpy as np
import pytest
import _libs as L

EMU_SO = os.path.join(L.ROOT, "build", "libmmg_emu.so")


class Ez(C.Structure):
    _fields_ = [("max", C.c_uint32), ("zdropped", C.c_int32), ("max_q", C.c_int32), ("max_t", C.c_int32), ("mqe", C.c_int32),
                ("mqe_t", C.c_int32), ("mte", C.c_int32), ("mte_q", C.c_int32), ("score", C.c_int32), ("n_cigar", C.c_int32),
                ("reach_end", C.c_int32)]


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-C", L.ROOT, "emu"], stdout=subprocess.DEVNULL)
    E = C.CDLL(EMU_SO)
    E.emu_sketch.restype = C.c_int
    E.emu_sketch.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_int, C.c_int, C.c_void_p, C.c_int]
    E.emu_idx_new.restype = C.c_void_p
    E.emu_idx_new.argtypes = [C.c_int64, C.c_void_p, C.c_void_p]
    E.emu_idx_free.argtypes = [C.c_void_p]
    E.emu_collect.restype = C.c_int64
    E.emu_collect.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int64,
                              C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]
    E.emu_collect_ranked.restype = C.c_int64
    E.emu_collect_ranked.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int64, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    E.emu_chain.restype = C.c_int
    E.emu_chain.argtypes = [C.c_int] * 9 + [C.c_int64, C.c_void_p, C.c_void_p]
    E.emu_rs_sort_128x.argtypes = [C.c_void_p, C.c_int64]
    E.emu_rs_sort_warp_128x.argtypes = [C.c_void_p, C.c_int64]
    E.emu_ksw.restype = C.c_int
    E.emu_ksw.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 8 + [C.POINTER(Ez), C.c_void_p]
    E.emu_ksw_fast.restype = C.c_int
    E.emu_ksw_fast2.restype = C.c_int
    E.emu_ksw_fast2.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 9 + [C.POINTER(Ez), C.c_void_p]
    E.emu_ksw_fast.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 9 + [C.POINTER(Ez), C.c_void_p]
    return E


def emu_sketch(E, s, w, k, rid=0, hpc=0, chunk=0):
    out = np.zeros(len(s) + 8, dtype=L.mm128)
    n = E.emu_sketch(s, len(s), w, k, rid, hpc, chunk, out.ctypes.data, len(out))
    assert n >= 0
    return out[:n].copy()


@pytest.mark.parametrize("w,k,hpc", [(11, 21, 0), (10, 15, 0), (5, 19, 1), (19, 19, 0), (3, 4, 0), (1, 15, 0), (10, 14, 0), (4, 6, 0)])
def test_sketch_chunked_equals_oracle(emu, w, k, hpc):
    rng = np.random.default_rng(77 + w + k)
    for it in range(80):
        n = int(rng.integers(1, 1500))
        s = L.rand_seq(rng, n, n_frac=[0, 0.01, 0.15][it % 3])
        if it % 5 == 0:
            s = (b"AT" * n)[:n] if it % 2 else (s[:6] * n)[:n]
        if it % 11 == 0:  # long N run in the middle
            s = s[: n // 3] + b"N" * (n // 4) + s[n // 3 + n // 4:]
        want = L.orc_sketch(s, w, k, 7, hpc)
        for chunk in [0, 1, 7, 64, 96, 500]:
            got = emu_sketch(emu, s, w, k, 7, hpc, chunk)
            assert got.tobytes() == want.tobytes(), (w, k, hpc, it, chunk, len(s))


def test_exact_radix_replay(emu):
    rng = np.random.default_rng(3)
    for n in [0, 1, 64, 65, 300, 4000, 20000]:
        for bits in [2, 9, 33, 64]:
            a = np.zeros(n, dtype=L.mm128)
            a["x"] = rng.integers(0, (1 << bits) - 1, n, dtype=np.uint64, endpoint=True)
            a["y"] = np.arange(n)
            b = a.copy()
            emu.emu_rs_sort_128x(a.ctypes.data, n)
            L.oracle().orc_radix_sort_128x(b.ctypes.data, b.ctypes.data + 16 * n)
            assert a.tobytes() == b.tobytes()


def test_exact_radix_replay_warp(emu):
    """mmg_rs_sort_warp (digits walked by one lane, elements scattered by the warp) ends in klib's order: anchor-shaped keys
    (strand<<63 | rid<<32 | pos, many equal), few-digit keys, all-equal keys, sizes around the 64-element insertion-sort limit"""
    rng = np.random.default_rng(5)
    for n in [0, 1, 2, 63, 64, 65, 66, 129, 300, 4000, 20000, 70000]:
        for kind in ["bits2", "bits9", "bits33", "bits64", "anchor", "equal", "locus"]:
            a = np.zeros(n, dtype=L.mm128)
            if kind.startswith("bits"):
                a["x"] = rng.integers(0, (1 << int(kind[4:])) - 1, n, dtype=np.uint64, endpoint=True)
            elif kind == "anchor":
                strand = rng.integers(0, 2, n, dtype=np.uint64) << np.uint64(63)
                rid = rng.integers(0, 24, n, dtype=np.uint64) << np.uint64(32)
                pos = rng.integers(0, max(2, n // 3), n, dtype=np.uint64) * np.uint64(977)
                a["x"] = strand | rid | pos
            elif kind == "equal":
                a["x"] = np.uint64(0x8000000500001234)
            else:  # one locus: positions within 10 kb, every fourth one doubled
                pos = np.uint64(123456789) + rng.integers(0, 10000, n, dtype=np.uint64)
                if n > 8:
                    pos[::4] = pos[1::4][: len(pos[::4])] if len(pos[1::4]) >= len(pos[::4]) else pos[::4]
                a["x"] = (np.uint64(7) << np.uint64(32)) | pos
            a["y"] = np.arange(n)
            b = a.copy()
            emu.emu_rs_sort_warp_128x(a.ctypes.data, n)
            L.oracle().orc_radix_sort_128x(b.ctypes.data, b.ctypes.data + 16 * n)
            assert a.tobytes() == b.tobytes(), (n, kind)


def _index_arrays(seqs, w, k):
    parts = [L.orc_sketch(s, w, k, i) for i, s in enumerate(seqs)]
    mv = np.concatenate(parts)
    key = mv["x"] >> np.uint64(8)
    order = np.lexsort((mv["y"], key))
    return np.ascontiguousarray(key[order]), np.ascontiguousarray(mv["y"][order])


@pytest.mark.parametrize("mode", ["sr", "ont"])
def test_seed_and_chain(emu, mode):
    from test_oracle_vs_ref import _mk_ref, _frags, SR_CHAIN, ONT_CHAIN
    rng = np.random.default_rng(42)
    seqs = _mk_ref(rng)
    w, k = (11, 21) if mode == "sr" else (10, 15)
    key, pos = _index_arrays(seqs, w, k)
    ei = emu.emu_idx_new(len(key), key.ctypes.data, pos.ctypes.data)
    oi = L.oracle().orc_idx_build(w, k, 0, len(seqs), L.c_str_array(seqs))
    rng = np.random.default_rng(11)
    try:
        for segs in _frags(rng, seqs, 150 if mode == "sr" else 25, mode == "sr"):
            mv, qlen = L.frag_minimizers(L.orc_sketch, segs, w, k)
            for max_occ in ([1000, 20, 5] if mode == "sr" else [50, 8]):
                a0, _, _ = L.orc_collect(oi, mode == "sr", 0, max_occ, mv, qlen)
                for flag in [0, 0x100000, 0x200000]:
                    a1, rep1, mp1 = L.orc_collect(oi, mode == "sr", flag, max_occ, mv, qlen)
                    a2 = np.zeros(len(a0) + 64, dtype=L.mm128)  # capacity = the unfiltered plan
                    mp2 = np.zeros(len(mv) + 1, dtype=np.uint64)
                    rep2, nm2 = C.c_int(0), C.c_int(0)
                    n2 = emu.emu_collect(ei, mode == "sr", flag, max_occ, len(mv), mv.ctypes.data, qlen, a2.ctypes.data, len(a2),
                                         C.byref(rep2), C.byref(nm2), mp2.ctypes.data)
                    assert n2 == len(a1) and rep2.value == rep1 and (mp2[:nm2.value] == mp1).all()
                    assert a2[:n2].tobytes() == a1.tobytes()
                    if mode == "sr":  # the rank-based heap replay (what the device runs when equal positions meet in the heap)
                        a3 = np.zeros(len(a0) + 64, dtype=L.mm128)
                        rep3, nm3 = C.c_int(0), C.c_int(0)
                        n3 = emu.emu_collect_ranked(ei, flag, max_occ, len(mv), mv.ctypes.data, qlen, a3.ctypes.data, len(a3), C.byref(rep3), C.byref(nm3))
                        assert n3 == len(a1) and rep3.value == rep1 and a3[:n3].tobytes() == a1.tobytes()
                params = SR_CHAIN if mode == "sr" else ONT_CHAIN
                a1, _, _ = L.orc_collect(oi, mode == "sr", 0, max_occ, mv, qlen)
                u1, b1 = L.chain_call(L.oracle().orc_chain_dp, params, a1)
                u2, b2 = L.chain_call(emu.emu_chain, params, a1)
                assert (u1 == u2).all() and b1.tobytes() == b2.tobytes()
    finally:
        emu.emu_idx_free(ei)
        L.oracle().orc_idx_destroy(oi)


def _n_cases(preset, n):
    """the K4 tests below run every scoring of L.KSW_SCORINGS; the three they began with keep their full case count"""
    return n if preset in ("sr", "ont", "eq") else n // 3


def emu_ksw(E, q, t, mat, pen, w, zd, eb, fl):
    ez = Ez()
    cig = np.zeros(len(q) + len(t) + 4, dtype=np.uint32)
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    E.emu_ksw(len(q), q.ctypes.data, len(t), t.ctypes.data, mat.ctypes.data, *pen, w, zd, eb, fl, C.byref(ez), cig.ctypes.data)
    return dict(max=ez.max, zdropped=ez.zdropped, max_q=ez.max_q, max_t=ez.max_t, mqe=ez.mqe, mqe_t=ez.mqe_t, mte=ez.mte,
                mte_q=ez.mte_q, score=ez.score, reach_end=ez.reach_end, cigar=cig[:ez.n_cigar].tolist())


@pytest.mark.parametrize("preset", list(L.KSW_SCORINGS))
def test_ksw_pieces(emu, preset):
    from test_oracle_vs_ref import _ksw_cases
    rng = np.random.default_rng(5150)
    sc = L.KSW_SCORINGS[preset]
    mat, pen, bw, zd, eb = sc.mat, sc.pen, sc.band, sc.zdrop, sc.end_bonus
    n = 0
    for q, t in _ksw_cases(rng, _n_cases(preset, 180)):
        for fl in [0xC2, 0x40, 0x08, 0x00, 0x01, 0x02]:
            for w in ([bw, 20, -1] if n % 5 == 0 else [bw]):
                a = L.orc_ksw(q, t, mat, *pen, w, zd, eb if fl & 0x40 else -1, fl)
                b = emu_ksw(emu, q, t, mat, pen, w, zd, eb if fl & 0x40 else -1, fl)
                if fl & 0x01:
                    a["cigar"] = []
                assert a == b, (len(q), len(t), fl, w)
        n += 1


def emu_ksw_fast(E, q, t, mat, pen, w, zd, eb, fl, stride):
    ez = Ez()
    cig = np.zeros(len(q) + len(t) + 4, dtype=np.uint32)
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    rc = E.emu_ksw_fast(len(q), q.ctypes.data, len(t), t.ctypes.data, mat.ctypes.data, *pen, w, zd, eb, fl, stride, C.byref(ez), cig.ctypes.data)
    assert rc != -2, "a valid cell left the int8 range: the 32-bit cell would differ from the reference's int8 lanes"
    if rc < 0:
        return None
    return dict(max=ez.max, zdropped=ez.zdropped, max_q=ez.max_q, max_t=ez.max_t, mqe=ez.mqe, mqe_t=ez.mqe_t, mte=ez.mte,
                mte_q=ez.mte_q, score=ez.score, reach_end=ez.reach_end, cigar=cig[:ez.n_cigar].tolist())


def emu_ksw_fast2(E, q, t, mat, pen, w, zd, eb, fl, stride):
    ez = Ez()
    cig = np.zeros(len(q) + len(t) + 4, dtype=np.uint32)
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    rc = E.emu_ksw_fast2(len(q), q.ctypes.data, len(t), t.ctypes.data, mat.ctypes.data, *pen, w, zd, eb, fl, stride, C.byref(ez), cig.ctypes.data)
    if rc < 0:
        return None
    return dict(max=ez.max, zdropped=ez.zdropped, max_q=ez.max_q, max_t=ez.max_t, mqe=ez.mqe, mqe_t=ez.mqe_t, mte=ez.mte,
                mte_q=ez.mte_q, score=ez.score, reach_end=ez.reach_end, cigar=cig[:ez.n_cigar].tolist())


@pytest.mark.parametrize("preset", list(L.KSW_SCORINGS))
def test_ksw_fast_form_in_pairs(emu, preset):
    """The thread-per-job form on 16x2 pairs (mmg_kswfast2.h: two cells per instruction, pairs aligned on the target coordinate, the
    out-of-matrix half of the first / last pair computed and ignored) equals ksw_extd2 bit for bit: all flags, w = -1, odd and
    even lengths, 1 x n and n x 1 jobs, N bases."""
    from test_oracle_vs_ref import _ksw_cases
    rng = np.random.default_rng(4242)
    sc = L.KSW_SCORINGS[preset]
    mat, pen, bw, zd, eb = sc.mat, sc.pen, sc.band, sc.zdrop, sc.end_bonus
    cases = list(_ksw_cases(rng, _n_cases(preset, 240)))
    for ql, tl in [(1, 1), (1, 2), (2, 1), (1, 7), (7, 1), (2, 2), (3, 2), (2, 3), (5, 4), (4, 5), (16, 17), (17, 16), (33, 31)]:
        cases.append((rng.integers(0, 5, ql, dtype=np.uint8), rng.integers(0, 5, tl, dtype=np.uint8)))
    n_fast = 0
    for q, t in cases:
        for fl in [0xC2, 0x40, 0x08, 0x18, 0x00, 0x01, 0x02, 0x80, 0x4A]:
            for w in [bw, -1]:
                b = emu_ksw_fast2(emu, q, t, mat, pen, w, zd, eb if fl & 0x40 else -1, fl, 1 + (n_fast % 3))
                if b is None:
                    continue
                a = L.orc_ksw(q, t, mat, *pen, w, zd, eb if fl & 0x40 else -1, fl)
                if fl & 0x01:
                    a["cigar"] = []
                assert a == b, (len(q), len(t), fl, w)
                n_fast += 1
    assert n_fast > 1500 * _n_cases(preset, 240) // 240


@pytest.mark.parametrize("preset", list(L.KSW_SCORINGS))
def test_ksw_fast_form(emu, preset):
    """The thread-per-job form used when the band never clips equals ksw_extd2 bit for bit (all flags, incl. w=-1)."""
    from test_oracle_vs_ref import _ksw_cases
    rng = np.random.default_rng(777)
    sc = L.KSW_SCORINGS[preset]
    mat, pen, bw, zd, eb = sc.mat, sc.pen, sc.band, sc.zdrop, sc.end_bonus
    n_fast = n_skip = 0
    for q, t in _ksw_cases(rng, _n_cases(preset, 240)):
        for fl in [0xC2, 0x40, 0x08, 0x18, 0x00, 0x01, 0x02, 0x80]:
            for w in [bw, -1]:
                b = emu_ksw_fast(emu, q, t, mat, pen, w, zd, eb if fl & 0x40 else -1, fl, 1 + (n_fast % 3))
                if b is None:
                    n_skip += 1
                    continue
                a = L.orc_ksw(q, t, mat, *pen, w, zd, eb if fl & 0x40 else -1, fl)
                if fl & 0x01:
                    a["cigar"] = []
                assert a == b, (len(q), len(t), fl, w)
                n_fast += 1
    assert n_fast > 1500 * _n_cases(preset, 240) // 240 and (preset != "sr" or n_skip > 0)


def _heap_case(rng, n_lists, max_cnt, dup_frac):
    """lists of strictly increasing values; a share of the lists are copies of another one (the overlapping-mate / tandem case),
    so equal values meet in the heap.  Returns first[], cnt[], K[] (rank of every slot = index of the first slot with its value
    in sorted order) exactly as k_heap_rank derives them."""
    lists = []
    for j in range(n_lists):
        if lists and rng.random() < dup_frac:
            src = lists[int(rng.integers(0, len(lists)))]
            lists.append(src.copy() if rng.random() < 0.7 else src[: max(1, len(src) // 2)].copy())
        else:
            c = int(rng.integers(1, max_cnt + 1))
            lists.append(np.sort(rng.choice(max_cnt * n_lists * 4, size=c, replace=False)).astype(np.int64))
    cnt = np.array([len(x) for x in lists], dtype=np.int32)
    first = np.concatenate([[0], np.cumsum(cnt)[:-1]]).astype(np.int32)
    vals = np.concatenate(lists)
    order = np.argsort(vals, kind="stable")
    sv = vals[order]
    start = np.concatenate([[True], sv[1:] != sv[:-1]])
    rank_sorted = np.maximum.accumulate(np.where(start, np.arange(len(sv)), 0))
    K = np.zeros(len(vals), dtype=np.uint32)
    K[order] = rank_sorted.astype(np.uint32)
    return first, cnt, K


@pytest.mark.parametrize("nreg", [1, 2, 4])
def test_heap_replay_in_registers_equals_serial_heap(emu, nreg):
    """mmg_regheap.h (a warp, heap nodes in registers) pops in the order of klib's heap on every input, ties included"""
    emu.emu_heap_replay.restype = C.c_int64
    emu.emu_heap_replay.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    rng = np.random.default_rng(500 + nreg)
    cap = 32 * nreg - 1
    sizes = [1, 2, 3, cap, cap - 1, max(1, cap // 2), 16, 15, 17] + [int(rng.integers(1, cap + 1)) for _ in range(60)]
    for it, n_lists in enumerate(sizes):
        n_lists = min(n_lists, cap)
        first, cnt, K = _heap_case(rng, n_lists, [1, 3, 40, 200][it % 4], [0.0, 0.3, 0.6, 0.9][(it // 4) % 4])
        n = int(cnt.sum())
        want, got = np.zeros(n + 1, dtype=np.uint32), np.zeros(n + 1, dtype=np.uint32)
        assert emu.emu_heap_replay(n_lists, first.ctypes.data, cnt.ctypes.data, K.ctypes.data, want.ctypes.data, 0) == n
        assert emu.emu_heap_replay(n_lists, first.ctypes.data, cnt.ctypes.data, K.ctypes.data, got.ctypes.data, nreg) == n
        assert (want == got).all(), f"case {it}: n_lists={n_lists} n={n}, first difference at pop {int(np.argmax(want != got))}"


def emu_ksw_dpx(E, q, t, mat, pen, w, zd, eb, fl):
    E.emu_ksw_dpx.restype = C.c_int
    E.emu_ksw_dpx.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 8 + [C.POINTER(Ez), C.c_void_p]
    ez = Ez()
    cig = np.zeros(len(q) + len(t) + 4, dtype=np.uint32)
    q = np.ascontiguousarray(q, dtype=np.uint8); t = np.ascontiguousarray(t, dtype=np.uint8)
    E.emu_ksw_dpx(len(q), q.ctypes.data, len(t), t.ctypes.data, mat.ctypes.data, *pen, w, zd, eb, fl, C.byref(ez), cig.ctypes.data)
    return dict(max=ez.max, zdropped=ez.zdropped, max_q=ez.max_q, max_t=ez.max_t, mqe=ez.mqe, mqe_t=ez.mqe_t, mte=ez.mte,
                mte_q=ez.mte_q, score=ez.score, reach_end=ez.reach_end, cigar=cig[:ez.n_cigar].tolist())


@pytest.mark.parametrize("preset", list(L.KSW_SCORINGS))
def test_ksw_literal_form_on_16x2_simd(emu, preset):
    """The literal form in the pair layout (two cells per lane, 16x2 arithmetic, direction from one max over value*8+preference)
    equals ksw_extd2 bit for bit: all flags, bands that clip (stale lanes are read), w=-1, N bases."""
    from test_oracle_vs_ref import _ksw_cases
    rng = np.random.default_rng(4242)
    sc = L.KSW_SCORINGS[preset]
    mat, pen, bw, zd, eb = sc.mat, sc.pen, sc.band, sc.zdrop, sc.end_bonus
    n = 0
    for q, t in _ksw_cases(rng, _n_cases(preset, 200)):
        for fl in [0xC2, 0x40, 0x08, 0x18, 0x00, 0x01, 0x02, 0x80]:
            for w in ([bw, 20, 7, -1] if n % 3 == 0 else [bw, 20]):
                a = L.orc_ksw(q, t, mat, *pen, w, zd, eb if fl & 0x40 else -1, fl)
                b = emu_ksw_dpx(emu, q, t, mat, pen, w, zd, eb if fl & 0x40 else -1, fl)
                if fl & 0x01:
                    a["cigar"] = []
                assert a == b, (len(q), len(t), fl, w)
        n += 1


@pytest.mark.parametrize("preset", list(L.KSW_SCORINGS))
def test_ksw_forms_equal_exact_dp(emu, preset):
    """The oracle and every emulated form against the plain int64 DP of tests/_kswref.py on jobs whose band never clips, z-drop
    off: score, max, mqe, mte, H at the max cell, the cells the CIGAR spans and its score.  Under bail every form returns the
    reset result without a CIGAR."""
    from test_oracle_vs_ref import _ksw_cases
    from _kswref import KswRef, check_job
    sc = L.KSW_SCORINGS[preset]
    mat, pen = sc.mat, sc.pen
    rng = np.random.default_rng(6006)
    cases = list(_ksw_cases(rng, 48))
    for ql, tl in [(1, 1), (1, 9), (9, 1), (1, 300), (300, 1), (17, 16), (64, 700)]:
        cases.append((rng.integers(0, 5, ql, dtype=np.uint8), rng.integers(0, 5, tl, dtype=np.uint8)))
    reset = dict(max=0, zdropped=0, max_q=-1, max_t=-1, mqe=-0x40000000, mqe_t=-1, mte=-0x40000000, mte_q=-1, score=-0x40000000,
                 reach_end=0, cigar=[])
    n_fast = 0
    for q, t in cases:
        ref = KswRef(q, t, mat, *pen) if preset != "bail" else None
        for fl in [0x00, 0x40, 0x08, 0x02, 0xC2, 0x4A, 0x80, 0x01]:
            eb = sc.end_bonus if fl & 0x40 else -1
            a = L.orc_ksw(q, t, mat, *pen, -1, -1, eb, fl)
            forms = {"scalar": emu_ksw(emu, q, t, mat, pen, -1, -1, eb, fl), "literal 16x2": emu_ksw_dpx(emu, q, t, mat, pen, -1, -1, eb, fl),
                     "fast": emu_ksw_fast(emu, q, t, mat, pen, -1, -1, eb, fl, 2), "fast pairs": emu_ksw_fast2(emu, q, t, mat, pen, -1, -1, eb, fl, 3)}
            if fl & 0x01:
                a["cigar"] = []
            if preset == "bail":
                assert a == reset, a
            else:
                check_job(a, q, t, mat, pen, fl, eb, ref)
            for name, b in forms.items():
                if b is None:  # outside the fast forms' limits
                    continue
                n_fast += name.startswith("fast")
                if preset != "bail":
                    check_job(b, q, t, mat, pen, fl, eb, ref)
                assert a == b, (name, len(q), len(t), fl)
    assert n_fast == 2 * 8 * len(cases)  # no clipping band and small jobs: the fast forms take every one


@pytest.mark.parametrize("w,k", [(11, 21), (10, 15), (5, 19), (19, 19), (3, 5), (1, 15), (4, 7), (32, 27)])
def test_sketch_warp_form_equals_oracle(emu, w, k):
    """K1 with the positions of a read spread over the lanes (mmg_sketchwarp.h) emits what mm_sketch emits, in its order:
    random reads, tandem repeats and homopolymers (equal hashes inside a window), reads shorter than a window."""
    emu.emu_sketch_warp.restype = C.c_int
    emu.emu_sketch_warp.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_int]
    rng = np.random.default_rng(900 + w + k)
    n_done = 0
    for it in range(300):
        n = int(rng.integers(1, 513)) if it % 7 else int(rng.integers(1, w + k + 3))
        s = L.rand_seq(rng, n)
        if it % 5 == 0:
            unit = L.rand_seq(rng, int(rng.integers(1, 9)))
            s = (unit * n)[:n]
        if it % 11 == 0:
            s = s[: n // 2] + s[: n - n // 2]
        out = np.zeros(n + 8, dtype=L.mm128)
        got_n = emu.emu_sketch_warp(s, n, w, k, it & 1, out.ctypes.data, len(out))
        assert got_n >= 0, (got_n, n)
        want = L.orc_sketch(s, w, k, it & 1, 0)
        assert got_n == len(want) and out[:got_n].tobytes() == want.tobytes(), (it, n, s[:80])
        n_done += 1
    assert n_done == 300
    # a read with an ambiguous base is handed back
    s = L.rand_seq(rng, 150); s = s[:70] + b"N" + s[71:]
    assert emu.emu_sketch_warp(s, 150, w, k, 0, np.zeros(200, dtype=L.mm128).ctypes.data, 200) == -1
