"""Every form of K4 forced by the shape of its jobs, under every scoring of L.KSW_SCORINGS.

k_ksw_prep puts each job into one of four kernels by its shape and the scoring (mmg_ksw.cu).  _form() below mirrors that rule,
so a change to the dispatcher fails here instead of silently moving coverage: each job set has shapes on both sides of every
boundary -- the three thread-per-job classes, the wavefront form's minimum and the fast forms' limits (min(qlen,tlen) <= 1023
and the scoring-dependent (qlen+tlen+2)*m < 500000, or the wavefront form's qlen+tlen < 65000 where that is lower), APPROX_DROP,
the warp form's shared-memory slot, the two shared-memory classes of the CTA form, and a band wider than the CTA form takes,
which keeps the warp form's state in the global arena.

The jobs run through the single-job entry point, where the kernel that ran is read from the profiler for every job, and as one
batch against resident reads (q_rev, reversed), where mmg_ksw_last_split must count them as the rule says.  Every result equals
the oracle field for field; jobs whose band never clips, z-drop off, also pass the exact-DP checks of tests/_kswref.py.

A last test runs one batch in parts (MMG_KSW_BUDGET) and checks that the parts give what the whole gives."""
import ctypes as C
import json
import os
import subprocess
import sys
import numpy as np
import pytest
import _libs as L
from _kswref import check_job

pytestmark = pytest.mark.gpu

FORMS = ("k_ksw_tpj", "k_ksw_wave", "k_ksw_dpx", "k_ksw_dpx_block")
FAST_CLASSES = [(24, 56, 56), (48, 104, 104), (80, 160, 160)]  # ksw_ftab: min(qlen,tlen) <= mc, tlen <= tc, qlen <= qc
DPX_SLOT, BLOCK_SMEM1, BLOCK_SMEM2, BLOCK_MAX_NCOL = 5120, 48 * 1024, 200 * 1024, 64
FLAGS = [0x00, 0x40, 0xC2, 0x08, 0x02, 0x4A, 0x80, 0x01]


def _dpx_mem_bytes(ql, tl):  # mmg_kswdpx_mem_bytes
    lane = ((tl + 15) // 16) * 16 * 10 + ((ql + 15) // 16) * 16 + 16
    return ((lane + 15) & ~15) + ((tl + 15) // 16) * 64


def _fast_m(sc):
    """m of mmg_ksw_fast_ok: the largest score or gap step magnitude, after ksw2's ordering of the pieces and its N rule"""
    q, e, q2, e2 = sc.pen if sc.q + sc.e <= sc.q2 + sc.e2 else (sc.q2, sc.e2, sc.q, sc.e)
    mat = sc.mat
    sc_n = -e2 if mat[24] == 0 else int(mat[24])
    return max(int(mat[0]), -int(mat[1]), -sc_n, q + e, q2 + e2)


def _bails(sc):  # ksw2_extd2_sse.c:92: the worst score beyond two gap openings of the cheaper piece
    q, e = (sc.q, sc.e) if sc.q + sc.e <= sc.q2 + sc.e2 else (sc.q2, sc.e2)
    return -int(sc.mat[1:].min()) > 2 * (q + e)


def _clips(ql, tl, w):
    if w < 0:
        w = max(ql, tl)
    r = np.arange(ql + tl - 1)
    st, en = np.maximum(0, r - ql + 1), np.minimum(tl - 1, r)
    return bool(((st < (r - w + 1) >> 1) | (en > (r + w) >> 1)).any())


def _form(sc, ql, tl, w, flag):
    """(kernel, detail) k_ksw_prep gives a job: detail is the fast class, the CTA form's shared-memory class, or where the warp
    form keeps its state"""
    mn = min(ql, tl)
    fast = not _bails(sc) and not _clips(ql, tl, w) and (ql + tl + 2) * _fast_m(sc) < 500000 and mn <= 1023
    if fast:
        for c, (mc, tc, qc) in enumerate(FAST_CLASSES):
            if mn <= mc and tl <= tc and ql <= qc:
                return "k_ksw_tpj", c
        if mn >= 32 and ql + tl < 65000 and not flag & 0x10:
            return "k_ksw_wave", None
    md = _dpx_mem_bytes(ql, tl)
    n_col = (min(mn, (w if w >= 0 else max(ql, tl)) + 1) + 15) // 16 + 1
    force = os.environ.get("MMG_KSW_FORCE_BLOCK") is not None
    if not _bails(sc) and (md > DPX_SLOT or force) and md <= BLOCK_SMEM2 and n_col <= BLOCK_MAX_NCOL:
        return "k_ksw_dpx_block", 1 if md <= BLOCK_SMEM1 else 2
    return "k_ksw_dpx", "arena" if md > DPX_SLOT else "slot"


def _shapes(sc):
    """(qlen, tlen, w, flag or None) on both sides of every boundary of _form; flag None: the next one of FLAGS"""
    lim = min(499999 // _fast_m(sc) - 2, 64999)  # the largest qlen+tlen the fast forms take, and the wavefront form's own limit
    return [
        # thread per job: the three classes and their tlen / qlen limits, 1 x n and n x 1
        (20, 50, -1, None), (24, 56, -1, None), (25, 56, -1, None), (20, 57, -1, None), (57, 40, -1, None), (48, 104, -1, None),
        (49, 104, -1, None), (80, 160, -1, None), (150, 1, -1, None), (1, 50, -1, None), (50, 1, -1, None), (1, 200, -1, None),
        (170, 1, -1, None),
        # wavefront: min(qlen,tlen) 31 / 32 and 1023 / 1024, several passes over a tlen that is not a multiple of 8, the
        # scoring's (qlen+tlen+2)*m limit (or qlen+tlen < 65000) from either side, APPROX_DROP
        (81, 160, -1, None), (31, 200, -1, None), (32, 200, -1, None), (200, 32, -1, None), (1023, 1100, -1, None),
        (1024, 1100, -1, None), (300, 517, -1, None), (517, 300, -1, 0x80), (100, lim - 100, -1, None), (100, lim - 99, -1, None),
        (300, 517, -1, 0x18),
        # literal warp form with its state in the slot: clipped bands down to w = 7
        (150, 300, 20, None), (120, 200, 7, None), (150, 151, 40, 0x40), (300, 280, 100, 0x00),
        # literal CTA form, both shared-memory classes
        (700, 1300, 500, None), (1500, 1400, 300, 0x40), (5000, 5000, 500, None),
        # literal warp form with its state in the global arena: a band wider than the CTA form takes
        (6500, 7000, 1100, None),
    ]


def _jobs(api, rng, refseqs, sc, shapes, fl0=0):
    """one resident read per job, built so that the job's query is a mutated copy of its target (one in four unrelated), with
    N bases; returns the jobs, the reads in mapping orientation, and every job's (q, t) as the kernels must see them"""
    jobs = np.zeros(len(shapes), dtype=api.ksw_job_dtype)
    reads, qt = [], []
    for j, (ql, tl, w, fl) in enumerate(shapes):
        fl = FLAGS[(j + fl0) % len(FLAGS)] if fl is None else fl
        rid = int(rng.integers(0, len(refseqs)))
        ts = int(rng.integers(0, len(refseqs[rid]) - max(ql, tl) - 10))
        if j % 4 == 3:
            body = L.rand_seq(rng, ql)
        else:
            body = (L.mutate(rng, refseqs[rid][ts:ts + ql + 20], 0.04, 0.01, 0.01) + L.rand_seq(rng, ql))[:ql]
        body = bytearray(body)
        for p in rng.integers(0, ql, max(1, ql // 150)):
            body[p] = ord("N")
        pre, suf = L.rand_seq(rng, int(rng.integers(0, 9))), L.rand_seq(rng, int(rng.integers(0, 9)))
        strand = pre + bytes(body) + suf
        q_rev, rev = j & 1, (j >> 1) & 1
        reads.append(L.revcomp(strand) if q_rev else strand)
        clipped = _clips(ql, tl, w)
        zd = sc.zdrop if clipped or j % 3 == 2 else -1  # z-drop off where the exact-DP checks apply
        eb = sc.end_bonus if fl & 0x40 else -1
        jobs[j] = (j, q_rev, len(pre), ql, rid, ts, tl, rev, w, zd, eb, fl)
        codes = L.nt4(reads[-1])
        s = codes if not q_rev else np.where(codes[::-1] < 4, 3 - codes[::-1], 4).astype(np.uint8)
        q, t = s[len(pre):len(pre) + ql], L.nt4(refseqs[rid])[ts:ts + tl]
        if rev:
            q, t = q[::-1], t[::-1]
        qt.append((np.ascontiguousarray(q), np.ascontiguousarray(t)))
    return jobs, reads, qt


def _check(sc, job, q, t, got):
    fl, w, zd, eb = int(job["flag"]), int(job["w"]), int(job["zdrop"]), int(job["end_bonus"])
    want = L.orc_ksw(q, t, sc.mat, *sc.pen, w, zd, eb, fl)
    if fl & 0x01:
        want["cigar"] = []
    assert got == want, (sc.name, len(q), len(t), w, hex(fl))
    if not _bails(sc) and zd < 0 and not _clips(len(q), len(t), w):
        check_job(got, q, t, sc.mat, sc.pen, fl, eb)


def _profile(ctx):
    from airlift_b200 import api
    lib = api.lib()
    names = (C.c_char_p * 256)(); ms = (C.c_double * 256)(); n = (C.c_long * 256)()
    lib.mmg_profile_fetch.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double), C.POINTER(C.c_long)]
    k = lib.mmg_profile_fetch(ctx.h, 256, names, ms, n)
    return {names[i].decode(): int(n[i]) for i in range(k) if names[i]}


def _last_split(ctx):
    from airlift_b200 import api
    lib = api.lib()
    lib.mmg_ksw_last_split.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 4
    v = [C.c_uint64(0) for _ in range(4)]
    lib.mmg_ksw_last_split(ctx.h, *[C.byref(x) for x in v])
    return [x.value for x in v]


@pytest.fixture(scope="module")
def env():
    from airlift_b200 import api
    from test_oracle_vs_ref import _mk_ref
    refseqs = _mk_ref(np.random.default_rng(42), n_ctg=2, ln=70000)
    ctx = api.Context(0)
    idx = api.Index(ctx, refseqs, 10, 15)
    api.lib().mmg_profile_enable.argtypes = [C.c_void_p, C.c_int]
    api.lib().mmg_profile_enable(ctx.h, 1)
    yield api, ctx, idx, refseqs
    idx.close()
    ctx.close()


@pytest.mark.parametrize("preset", list(L.KSW_SCORINGS))
def test_each_form_under_each_scoring(env, preset):
    api, ctx, idx, refseqs = env
    sc = L.KSW_SCORINGS[preset]
    rng = np.random.default_rng(1000 + list(L.KSW_SCORINGS).index(preset))
    shapes = _shapes(sc)
    jobs, reads, qt = _jobs(api, rng, refseqs, sc, shapes)
    forms = [_form(sc, int(j["q_len"]), int(j["t_len"]), int(j["w"]), int(j["flag"])) for j in jobs]

    # one job at a time: the kernel that ran is the one the rule names
    _profile(ctx)
    for j, (q, t) in enumerate(qt):
        job = jobs[j]
        got = ctx.ksw_extd2(q, t, sc.mat, *sc.pen, int(job["w"]), int(job["zdrop"]), int(job["end_bonus"]), int(job["flag"]))
        ran = {k: v for k, v in _profile(ctx).items() if k in FORMS}
        assert ran == {forms[j][0]: 1}, (preset, shapes[j], forms[j], ran)
        _check(sc, job, q, t, got)
    kernels = {f for f, _ in forms}
    if _bails(sc):
        assert kernels == {"k_ksw_dpx"}
    else:
        assert kernels == set(FORMS) and ("k_ksw_dpx", "arena") in forms and ("k_ksw_dpx", "slot") in forms
        assert {d for f, d in forms if f == "k_ksw_dpx_block"} == {1, 2} and {d for f, d in forms if f == "k_ksw_tpj"} == {0, 1, 2}

    # the same jobs as one batch against resident reads, the scoring given through the mapping options
    batch, keep = api.Context.make_batch([[r] for r in reads])
    opt = sc.set_opt(api.ont_opt(50))
    ctx.batch_upload(opt, batch, flips=np.zeros(len(reads), np.uint8))
    _profile(ctx)
    got, _, cells = ctx.ksw_batch(idx, opt, jobs)
    ran = {k for k in _profile(ctx) if k in FORMS}
    assert ran == kernels, (preset, ran, kernels)
    for j, (q, t) in enumerate(qt):
        _check(sc, jobs[j], q, t, got[j])
    band = [L.oracle().orc_ksw_band_cells(int(j["q_len"]), int(j["t_len"]), int(j["w"])) for j in jobs]
    fast = [f in ("k_ksw_tpj", "k_ksw_wave") for f, _ in forms]
    assert cells == sum(band)
    assert _last_split(ctx) == [sum(fast), sum(c for c, f in zip(band, fast) if f), len(jobs) - sum(fast),
                                sum(c for c, f in zip(band, fast) if not f)]


# ---- the split path of mmg_ksw_batch ----------------------------------------------------------------------------------

N_SPLIT_JOBS = 300


def _split_jobs(api, refseqs):
    """~300 mixed jobs: every shape of the form grid under sr and short-read extension shapes"""
    rng = np.random.default_rng(31337)
    sc = L.KSW_SCORINGS["sr"]
    shapes = _shapes(sc)
    while len(shapes) < N_SPLIT_JOBS:
        ql, tl = int(rng.integers(1, 400)), int(rng.integers(1, 500))
        shapes.append((ql, tl, [151, 40, -1][len(shapes) % 3], None))
    return sc, _jobs(api, rng, refseqs, sc, shapes)


def _split_child(out_path):
    """runs the batch of _split_jobs once in this process (MMG_KSW_BUDGET is read once per process) and writes the results"""
    from airlift_b200 import api
    from test_oracle_vs_ref import _mk_ref
    refseqs = _mk_ref(np.random.default_rng(42), n_ctg=2, ln=70000)
    ctx = api.Context(0)
    idx = api.Index(ctx, refseqs, 10, 15)
    try:
        sc, (jobs, reads, _) = _split_jobs(api, refseqs)
        batch, keep = api.Context.make_batch([[r] for r in reads])
        opt = sc.set_opt(api.ont_opt(50))
        ctx.batch_upload(opt, batch, flips=np.zeros(len(reads), np.uint8))
        api.lib().mmg_profile_enable.argtypes = [C.c_void_p, C.c_int]
        api.lib().mmg_profile_enable(ctx.h, 1)
        got, _, cells = ctx.ksw_batch(idx, opt, jobs)
        parts = _profile(ctx).get("k_cig_gather", 0)  # one per part that ran
        with open(out_path, "w") as f:
            json.dump(dict(res=got, cells=cells, split=_last_split(ctx), parts=parts), f)
    finally:
        idx.close()
        ctx.close()


def test_split_batch_equals_whole(tmp_path):
    from airlift_b200 import api
    from test_oracle_vs_ref import _mk_ref
    refseqs = _mk_ref(np.random.default_rng(42), n_ctg=2, ln=70000)
    sc, (jobs, reads, qt) = _split_jobs(api, refseqs)
    # a budget of a quarter of the round's traceback and CIGAR bytes (the literal forms' sizes: an overestimate for the others)
    est = sum(((int(j["q_len"]) + int(j["t_len"]) - 1) * ((min(int(j["q_len"]), int(j["t_len"]), int(j["w"]) + 1 if j["w"] >= 0 else 1 << 30) + 15) // 16 + 1) + 1) * 16
              + (int(j["q_len"]) + int(j["t_len"]) + 2) * 4 for j in jobs)
    runs = {}
    for name, budget in [("whole", None), ("parts", est // 4), ("single", 1)]:
        env = dict(os.environ)
        env.pop("MMG_KSW_BUDGET", None)
        if budget is not None:
            env["MMG_KSW_BUDGET"] = str(budget)
        out = tmp_path / f"{name}.json"
        code = f"import sys; sys.path[:0] = [{L.ROOT!r}, {os.path.join(L.ROOT, 'tests')!r}]; import test_gpu_ksw_scoring as T; T._split_child({str(out)!r})"
        r = subprocess.run([sys.executable, "-c", code], cwd=L.ROOT, env=env, capture_output=True, text=True, timeout=1200)
        assert r.returncode == 0, (name, r.stdout[-2000:], r.stderr[-2000:])
        with open(out) as f:
            runs[name] = json.load(f)
    assert runs["whole"]["parts"] == 1
    assert 2 <= runs["parts"]["parts"] <= N_SPLIT_JOBS // 8, runs["parts"]["parts"]
    assert runs["single"]["parts"] == N_SPLIT_JOBS
    for name in ("parts", "single"):
        for key in ("res", "cells", "split"):
            assert runs[name][key] == runs["whole"][key], (name, key)
    for j, (q, t) in enumerate(qt):
        _check(sc, jobs[j], q, t, runs["whole"]["res"][j])
