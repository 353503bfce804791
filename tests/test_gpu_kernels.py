"""Parity tests proper: every CUDA stage, called through the C-ABI (include/mmg.h), against the
CPU oracle on the same seeded inputs.  Bit-exact comparisons throughout (integer work)."""
import ctypes as C
import numpy as np
import pytest
import _libs as L

pytestmark = pytest.mark.gpu

SR_CHAIN = (500, 300, 100, 25, 5000, 2, 25, 0, 2)
ONT_CHAIN = (5000, 5000, 500, 25, 5000, 3, 40, 0, 1)


@pytest.fixture(scope="module")
def api():
    import airlift_b200.api as A
    return A


@pytest.fixture(scope="module")
def ctx(api):
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def refseqs():
    from test_oracle_vs_ref import _mk_ref
    return _mk_ref(np.random.default_rng(42), n_ctg=4, ln=60000)


@pytest.mark.parametrize("w,k,hpc", [(11, 21, 0), (10, 15, 0), (5, 19, 1), (19, 19, 0), (3, 4, 0), (10, 14, 0)])
def test_sketch(ctx, w, k, hpc):
    rng = np.random.default_rng(500 + w + k)
    for it in range(40):
        n = int(rng.integers(1, 3000))
        s = L.rand_seq(rng, n, n_frac=[0, 0.01, 0.15][it % 3])
        if it % 5 == 0:
            s = (b"AT" * n)[:n] if it % 2 else (s[:6] * n)[:n]
        assert ctx.sketch(s, w, k, 9, hpc).tobytes() == L.orc_sketch(s, w, k, 9, hpc).tobytes(), (w, k, hpc, it)


def test_sketch_limits(ctx, api):
    with pytest.raises(api.MmgError):
        ctx.sketch(b"ACGTACGTACGTACGTACGT" * 20, 200, 15)  # w beyond the device ring buffer: loud error, no fallback


@pytest.mark.parametrize("w,k", [(11, 21), (10, 15)])
def test_index(ctx, api, refseqs, w, k):
    idx = api.Index(ctx, refseqs, w, k)
    oi = L.oracle().orc_idx_build(w, k, 0, len(refseqs), L.c_str_array(refseqs))
    try:
        assert idx.n_minimizers() == L.oracle().orc_idx_n_minimizers(oi)
        for f in [2e-4, 1e-2, 0.2]:
            assert idx.cal_max_occ(f) == L.oracle().orc_idx_cal_max_occ(oi, f)
        # packed reference == mm_seq4_set of every base
        S = idx.packed_S()
        codes = np.concatenate([L.nt4(s) for s in refseqs]).astype(np.uint32)
        pad = (-len(codes)) % 8
        want = np.concatenate([codes, np.zeros(pad, np.uint32)]).reshape(-1, 8)
        want = (want << (np.arange(8, dtype=np.uint32) * 4)).sum(axis=1, dtype=np.uint64).astype(np.uint32)
        assert (S == want).all()
        keys = set()
        for s in refseqs:
            keys.update((L.orc_sketch(s[:8000], w, k)["x"] >> np.uint64(8)).tolist())
        keys.update(np.random.default_rng(1).integers(0, 1 << (2 * k), 2000).tolist())
        keys = np.array(sorted(keys), dtype=np.uint64)
        n, pos = idx.get(keys, 64)
        n1 = C.c_int(0)
        for i, key in enumerate(keys.tolist()):
            p = L.oracle().orc_idx_get(oi, key, C.byref(n1))
            assert n[i] == n1.value
            m = min(n1.value, 64)
            assert pos[i, :m].tolist() == [p[j] for j in range(m)]
    finally:
        idx.close()
        L.oracle().orc_idx_destroy(oi)


@pytest.mark.parametrize("mode", ["sr", "ont"])
def test_seeds_and_chain_single(ctx, api, refseqs, mode):
    from test_oracle_vs_ref import _frags
    w, k = (11, 21) if mode == "sr" else (10, 15)
    idx = api.Index(ctx, refseqs, w, k)
    oi = L.oracle().orc_idx_build(w, k, 0, len(refseqs), L.c_str_array(refseqs))
    rng = np.random.default_rng(314)
    try:
        for segs in _frags(rng, refseqs, 40 if mode == "sr" else 8, mode == "sr"):
            mv, qlen = L.frag_minimizers(L.orc_sketch, segs, w, k)
            for max_occ in ([1000, 5] if mode == "sr" else [50, 8]):
                a0, _, _ = L.orc_collect(oi, mode == "sr", 0, max_occ, mv, qlen)
                for flag in [0, api.MM_F_FOR_ONLY]:
                    a1, rep1, mp1 = L.orc_collect(oi, mode == "sr", flag, max_occ, mv, qlen)
                    a2, rep2, mp2 = ctx.collect_seeds(idx, mode == "sr", flag, max_occ, mv, qlen, len(a0) + 8)
                    assert rep1 == rep2 and (mp1 == mp2).all() and a1.tobytes() == a2.tobytes()
                params = SR_CHAIN if mode == "sr" else ONT_CHAIN
                u1, b1 = L.chain_call(L.oracle().orc_chain_dp, params, a0)
                u2, b2 = ctx.chain_dp(params, a0)
                assert (u1 == u2).all() and b1.tobytes() == b2.tobytes()
    finally:
        idx.close()
        L.oracle().orc_idx_destroy(oi)


@pytest.mark.parametrize("preset", list(L.KSW_SCORINGS))
def test_ksw_single(ctx, preset):
    """every scoring of L.KSW_SCORINGS; sr and ont with the full case count.  The last cases give the gap pieces in the other
    order (q2, e2, q, e): the CLI refuses that, the kernels swap them as ksw2 does (after taking q+e of the order given)."""
    from test_oracle_vs_ref import _ksw_cases
    rng = np.random.default_rng(808)
    sc = L.KSW_SCORINGS[preset]
    mat, pen, bw, zd, eb = sc.mat, sc.pen, sc.band, sc.zdrop, sc.end_bonus
    n_cases = 90 if preset in ("sr", "ont") else 30
    n = 0
    for q, t in _ksw_cases(rng, n_cases + 6):
        p = pen if n < n_cases else (pen[2], pen[3], pen[0], pen[1])
        for fl in [0xC2, 0x40, 0x08, 0x00, 0x01, 0x02]:
            for w in ([bw, 20, -1] if n % 5 == 0 else [bw]):
                a = L.orc_ksw(q, t, mat, *p, w, zd, eb if fl & 0x40 else -1, fl)
                b = ctx.ksw_extd2(q, t, mat, *p, w, zd, eb if fl & 0x40 else -1, fl)
                if fl & 0x01:
                    a["cigar"] = []
                assert a == b, (len(q), len(t), fl, w, p)
        n += 1


def _oracle_frag(oi, opt, segs_mapped, w, k, n_segs_param):
    """mm_map_frag up to chaining (map.c:295-377) with the oracle."""
    heap = bool(opt.flag & 0x400000)
    mv, qlen = L.frag_minimizers(L.orc_sketch, segs_mapped, w, k)
    is_sr = bool(opt.flag & 0x1000)
    gap_qry = max(qlen, opt.max_gap) if is_sr else opt.max_gap
    if opt.max_gap_ref > 0:
        gap_ref = opt.max_gap_ref
    elif opt.max_frag_len > 0:
        gap_ref = max(opt.max_frag_len - qlen, opt.max_gap)
    else:
        gap_ref = opt.max_gap
    params = (gap_ref, gap_qry, opt.bw, opt.max_chain_skip, opt.max_chain_iter, opt.min_cnt, opt.min_chain_score, 0, n_segs_param)
    a, rep, mp = L.orc_collect(oi, heap, opt.flag & 0x300000, opt.mid_occ, mv, qlen)
    u, b = L.chain_call(L.oracle().orc_chain_dp, params, a)
    rech = 0
    if opt.max_occ > opt.mid_occ and rep > 0:
        if len(u):
            sc = (u >> np.uint64(32)).astype(np.int64)
            best, off, max_i, max_off = 0, 0, -1, -1
            for i in range(len(u)):
                if best < sc[i]:
                    best, max_i, max_off = sc[i], i, off
                off += int(u[i] & np.uint64(0xffffffff))
            cnt = int(u[max_i] & np.uint64(0xffffffff))
            seg = (b["y"][max_off:max_off + cnt] >> np.uint64(48)) & np.uint64(0xff)
            if 1 + int((seg[1:] != seg[:-1]).sum()) < n_segs_param:
                rech = 1
        else:
            rech = 1
    if rech:
        a, rep, mp = L.orc_collect(oi, heap, opt.flag & 0x300000, opt.max_occ, mv, qlen)
        u, b = L.chain_call(L.oracle().orc_chain_dp, params, a)
    return u, b, rep, mp, rech


@pytest.mark.parametrize("mode", ["sr", "sr_lowocc", "ont"])
def test_seed_chain_batch(ctx, api, refseqs, mode):
    from test_oracle_vs_ref import _frags
    sr = mode != "ont"
    w, k = (11, 21) if sr else (10, 15)
    idx = api.Index(ctx, refseqs, w, k)
    oi = L.oracle().orc_idx_build(w, k, 0, len(refseqs), L.c_str_array(refseqs))
    rng = np.random.default_rng(2718)
    try:
        frags_mapped = _frags(rng, refseqs, 600 if sr else 30, sr)  # sr: mate 2 already flipped to mapping orientation
        if sr:
            frags_mapped.append([b"ACGT" * 10, b"N" * 50])            # nothing to map
            frags_mapped.append([L.rand_seq(rng, 150)])               # single-end fragment inside a paired batch
            frags = [[f[0], L.revcomp(f[1])] if len(f) == 2 else f for f in frags_mapped]  # what the FASTQ holds
            opt = api.sr_opt()
            if mode == "sr_lowocc":
                opt.mid_occ, opt.max_occ = 8, 40  # make the re-chain branch (map.c:353-375) fire on this small genome
        else:
            frags = frags_mapped
            opt = api.ont_opt(idx.cal_max_occ(2e-4))
        batch, keep = api.Context.make_batch(frags)
        ch = api.chains_to_py(ctx.seed_chain_batch(idx, opt, batch))
        n_rech = 0
        for f, segs in enumerate(frags_mapped):
            u, b, rep, mp, rech = _oracle_frag(oi, opt, segs, w, k, len(segs))
            n_rech += rech
            uo, ao = int(ch["u_off"][f]), int(ch["a_off"][f])
            assert ch["n_u"][f] == len(u) and ch["n_a"][f] == len(b), (mode, f)
            assert (ch["u"][uo:uo + len(u)] == u).all(), (mode, f)
            assert ch["a"][ao:ao + len(b)].tobytes() == b.tobytes(), (mode, f)
            assert ch["rep_len"][f] == rep and ch["rechained"][f] == rech, (mode, f)
            if not sr:
                mo = int(ch["mini_off"][f])
                assert ch["n_mini"][f] == len(mp) and (ch["mini_pos"][mo:mo + len(mp)] == mp).all()
        if mode == "sr_lowocc":
            assert n_rech > 0
    finally:
        idx.close()
        L.oracle().orc_idx_destroy(oi)


def test_ksw_batch(ctx, api, refseqs):
    """DP jobs described against the resident reads and the index (align.c:690-771 call shapes)."""
    _ksw_batch(ctx, api, refseqs, L.KSW_SCORINGS["sr"], 400)


@pytest.mark.parametrize("preset", [p for p in L.KSW_SCORINGS if p != "sr"])
def test_ksw_batch_scoring(ctx, api, refseqs, preset):
    """test_ksw_batch under the other scorings of L.KSW_SCORINGS: the scoring reaches the kernels through the mapping options
    (make_score), as from the CLI or mappy."""
    _ksw_batch(ctx, api, refseqs, L.KSW_SCORINGS[preset], 150)


def _ksw_batch(ctx, api, refseqs, sc, n_jobs):
    from test_oracle_vs_ref import _frags
    w, k = 11, 21
    idx = api.Index(ctx, refseqs, w, k)
    rng = np.random.default_rng(99)
    try:
        frags_mapped = _frags(rng, refseqs, 60, True)
        frags = [[f[0], L.revcomp(f[1])] for f in frags_mapped]
        opt = sc.set_opt(api.sr_opt())
        batch, keep = api.Context.make_batch(frags)
        ctx.batch_upload(opt, batch)
        reads = [s for f in frags_mapped for s in f]  # mapping orientation, as resident on the device
        codes = [L.nt4(r) for r in reads]
        refcodes = [L.nt4(s) for s in refseqs]
        jobs = np.zeros(n_jobs, dtype=api.ksw_job_dtype)
        want = []
        mat = sc.mat
        for j in range(len(jobs)):
            sid = int(rng.integers(0, len(reads)))
            ql_read = len(reads[sid])
            q_rev = int(rng.integers(0, 2))
            qs = int(rng.integers(0, ql_read - 1)); ql = int(rng.integers(1, ql_read - qs + 1))
            rid = int(rng.integers(0, len(refseqs)))
            ts = int(rng.integers(0, len(refseqs[rid]) - 400)); tl = int(rng.integers(1, 300))
            rev = int(rng.integers(0, 2))
            fl = [0xC2, 0x40, 0x08, 0x00][j % 4]
            wj = [sc.band, 40][j % 2]
            eb = sc.end_bonus if fl & 0x40 else -1
            jobs[j] = (sid, q_rev, qs, ql, rid, ts, tl, rev, wj, sc.zdrop, eb, fl)
            strand = codes[sid] if not q_rev else np.where(codes[sid][::-1] < 4, 3 - codes[sid][::-1], 4).astype(np.uint8)
            q = strand[qs:qs + ql]; t = refcodes[rid][ts:ts + tl]
            if rev:
                q, t = q[::-1], t[::-1]
            want.append(L.orc_ksw(q, t, mat, *sc.pen, wj, sc.zdrop, eb, fl))
        got, ms, cells = ctx.ksw_batch(idx, opt, jobs)
        for j in range(len(jobs)):
            assert got[j] == want[j], (j, jobs[j])
        assert cells == sum(L.oracle().orc_ksw_band_cells(int(j["q_len"]), int(j["t_len"]), int(j["w"])) for j in jobs)
    finally:
        idx.close()
