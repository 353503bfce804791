"""mm_map_frag / mm_map called from many threads at once (airlift_b200/host/apiq.c): the calls of all threads are mapped
together in shared mini-batches on every GPU of the index, and each caller must still get exactly the hits the batch path gives
its fragment under its own options.  Python threads call through ctypes, which releases the GIL for the length of the call."""
import ctypes as C
import os
import subprocess
import threading
import time
import pytest
import _libs as L

pytestmark = pytest.mark.gpu
SYN = os.path.join(L.ROOT, "build", "mmsynth")
MM_F_CIGAR, MM_F_OUT_SAM, MM_F_NO_PRINT_2ND = 0x004, 0x008, 0x4000


class Extra(C.Structure):
    _fields_ = [("capacity", C.c_uint32), ("dp_score", C.c_int32), ("dp_max", C.c_int32), ("dp_max2", C.c_int32),
                ("n_ambi_ts", C.c_uint32), ("n_cigar", C.c_uint32)]


class Reg1(C.Structure):  # mm_reg1_t, minimap.h:83-98
    _fields_ = [(n, C.c_int32) for n in ("id", "cnt", "rid", "score", "qs", "qe", "rs", "re", "parent", "subsc", "as_", "mlen", "blen", "n_sub", "score0")] + \
               [("bits", C.c_uint32), ("hash", C.c_uint32), ("div", C.c_float), ("p", C.POINTER(Extra))]


class StepHead(C.Structure):
    _fields_ = [("n_seq", C.c_int), ("n_frag", C.c_int), ("seq", C.c_void_p), ("n_reg", C.POINTER(C.c_int)), ("seg_off", C.POINTER(C.c_int)),
                ("n_seg", C.POINTER(C.c_int)), ("rep_len", C.POINTER(C.c_int)), ("frag_gap", C.POINTER(C.c_int)), ("reg", C.POINTER(C.POINTER(Reg1)))]


def _hit(r, flip_qlen=None):
    qs, qe, rev = r.qs, r.qe, r.bits >> 10 & 1
    if flip_qlen is not None:  # mate mapped as its reverse complement: back to the read's own orientation (map.c:486-497)
        qs, qe, rev = flip_qlen - r.qe, flip_qlen - r.qs, 1 - rev
    cig = []
    if r.p:
        n = r.p.contents.n_cigar
        arr = C.cast(C.addressof(r.p.contents) + C.sizeof(Extra), C.POINTER(C.c_uint32))
        cig = [arr[i] for i in range(n)]
    return (r.rid, r.rs, r.re, qs, qe, rev, r.bits & 0xff, r.score, r.p.contents.dp_max if r.p else -1, tuple(cig))


def _reads(fn):
    ls = open(fn).read().split("\n")
    return [(ls[i][1:].split()[0], ls[i + 1]) for i in range(0, len(ls) - 3, 4)]


def _tasks():
    return len(os.listdir("/proc/self/task"))


def _tasks_settled(want=None):
    """threads of this process once joined threads have left /proc (want=None: once the count stops changing)"""
    n, prev = _tasks(), -1
    for _ in range(200):
        if (n <= want) if want is not None else (n == prev):
            break
        time.sleep(0.01)
        n, prev = _tasks(), n
    return n


@pytest.fixture(scope="module")
def data(tmp_path_factory):
    if not os.path.exists(SYN):
        pytest.skip("build/mmsynth missing")
    d = tmp_path_factory.mktemp("apiconc")
    subprocess.check_call([SYN, "ref", str(d / "ref.fa"), "2000000", "2", "42"])
    subprocess.check_call([SYN, "sr", str(d / "ref.fa"), str(d / "r1.fq"), str(d / "r2.fq"), "800", "44"])
    subprocess.check_call([SYN, "long", str(d / "ref.fa"), str(d / "long.fq"), "120", "45", "6000"])
    return d


@pytest.fixture(scope="module")
def lib():
    import bench
    L_ = bench.load_lib()
    L_.mm_map_frag.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_char_p), C.POINTER(C.c_int), C.POINTER(C.POINTER(Reg1)),
                               C.c_void_p, C.POINTER(bench.MapOptFull), C.c_char_p]
    L_.mm_map.restype = C.POINTER(Reg1)
    L_.mm_map.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.POINTER(C.c_int), C.c_void_p, C.POINTER(bench.MapOptFull), C.c_char_p]
    L_.mm_tbuf_init.restype = C.c_void_p
    L_.mm_tbuf_destroy.argtypes = [C.c_void_p]
    L_.mm_b200_set_lanes.argtypes = [C.c_int]
    return L_


def _index(lib, fn, preset):
    import bench
    ipt, opt = bench.IdxOpt(), bench.MapOptFull()
    lib.mm_set_opt(None, C.byref(ipt), C.byref(opt))
    lib.mm_set_opt(preset, C.byref(ipt), C.byref(opt))
    rd = lib.mm_idx_reader_open(str(fn).encode(), C.byref(ipt), None)
    mi = lib.mm_idx_reader_read(rd, 3)
    lib.mm_idx_reader_close(rd)
    assert mi
    lib.mm_mapopt_update(C.byref(opt), mi)
    return mi, opt


def _copy(opt):
    import bench
    o = bench.MapOptFull()
    C.memmove(C.byref(o), C.byref(opt), C.sizeof(opt))
    return o


def _batch_path(lib, mi, opt, files):
    """hits of every read of the files, in read order, through mm_b200_map_batch"""
    fns = (C.c_char_p * len(files))(*[str(f).encode() for f in files])
    reader = lib.mm_b200_open_reads(len(files), fns)
    b = lib.mm_b200_read_batch(reader, C.byref(opt), 10**9)
    assert lib.mm_b200_map_batch(mi, C.byref(opt), 4, b, 0) == 0
    h = C.cast(b, C.POINTER(StepHead)).contents
    want = [[_hit(h.reg[r][i]) for i in range(h.n_reg[r])] for r in range(h.n_seq)]
    lib.mm_b200_free_batch(b)
    lib.mm_b200_close_reads(reader)
    return want


def _map_pair(lib, mi, opt, tb, n1, s1, s2):
    s2rc = L.revcomp(s2.encode())
    seqs = (C.c_char_p * 2)(s1.encode(), s2rc)
    qlens = (C.c_int * 2)(len(s1), len(s2))
    n_regs = (C.c_int * 2)()
    regs = (C.POINTER(Reg1) * 2)()
    lib.mm_map_frag(mi, 2, qlens, seqs, n_regs, regs, tb, C.byref(opt), n1.encode())
    return [_hit(regs[0][i]) for i in range(n_regs[0])], [_hit(regs[1][i], flip_qlen=len(s2)) for i in range(n_regs[1])]


def _map_one(lib, mi, opt, tb, name, s):
    n = C.c_int(0)
    r = lib.mm_map(mi, len(s), s.encode(), C.byref(n), tb, C.byref(opt), name.encode())
    return [_hit(r[i]) for i in range(n.value)]


def _threads(n, fn):
    """fn(t) on n threads; exceptions are re-raised here"""
    err = []

    def run(t):
        try:
            fn(t)
        except BaseException as e:  # noqa: BLE001
            err.append(e)
    th = [threading.Thread(target=run, args=(t,)) for t in range(n)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    if err:
        raise err[0]


def _pairs_concurrent(lib, mi, opt, pairs, n_threads):
    got = [None] * len(pairs)

    def work(t):
        tb = lib.mm_tbuf_init()
        for k in range(t, len(pairs), n_threads):
            (n1, s1), (_, s2) = pairs[k]
            got[k] = _map_pair(lib, mi, opt, tb, n1, s1, s2)
        lib.mm_tbuf_destroy(tb)
    _threads(n_threads, work)
    return got


def test_sr_pairs_16_threads_coalesced(lib, data):
    mi, opt = _index(lib, data / "ref.fa", b"sr")
    try:
        opt.flag |= MM_F_CIGAR | MM_F_OUT_SAM
        want = _batch_path(lib, mi, opt, [data / "r1.fq", data / "r2.fq"])
        pairs = list(zip(_reads(data / "r1.fq"), _reads(data / "r2.fq")))
        lib.mm_b200_launch_count(mi, 1)
        got = _pairs_concurrent(lib, mi, opt, pairs, 16)
        n_conc = lib.mm_b200_launch_count(mi, 1)
        n_hits = 0
        for k, (g0, g1) in enumerate(got):
            assert g0 == want[2 * k], f"pair {k} mate 1"
            assert g1 == want[2 * k + 1], f"pair {k} mate 2"
            n_hits += len(g0) + len(g1)
        assert n_hits > len(pairs)
        got1 = _pairs_concurrent(lib, mi, opt, pairs, 1)
        n_one = lib.mm_b200_launch_count(mi, 1)
        assert got1 == got
        assert 0 < n_conc <= n_one // 2, (n_conc, n_one)
    finally:
        lib.mm_idx_destroy(mi)


def test_mixed_calls_and_option_sets(lib, data):
    """mm_map single-end calls under -x sr and mm_map_frag pairs under -x sr --secondary=yes -N 5, at the same time"""
    mi, opt = _index(lib, data / "ref.fa", b"sr")
    try:
        opt.flag |= MM_F_CIGAR | MM_F_OUT_SAM
        opt2 = _copy(opt)
        opt2.flag &= ~MM_F_NO_PRINT_2ND
        opt2.best_n = 5
        want_se = _batch_path(lib, mi, opt, [data / "r1.fq"])
        want_pe = _batch_path(lib, mi, opt2, [data / "r1.fq", data / "r2.fq"])
        r1 = _reads(data / "r1.fq")
        pairs = list(zip(r1, _reads(data / "r2.fq")))
        got_se, got_pe = [None] * len(r1), [None] * len(pairs)

        def work(t):
            tb = lib.mm_tbuf_init()
            if t % 2 == 0:
                for k in range(t // 2, len(r1), 8):
                    got_se[k] = _map_one(lib, mi, opt, tb, *r1[k])
            else:
                for k in range(t // 2, len(pairs), 8):
                    (n1, s1), (_, s2) = pairs[k]
                    got_pe[k] = _map_pair(lib, mi, opt2, tb, n1, s1, s2)
            lib.mm_tbuf_destroy(tb)
        _threads(16, work)
        assert got_se == want_se
        for k, (g0, g1) in enumerate(got_pe):
            assert g0 == want_pe[2 * k] and g1 == want_pe[2 * k + 1], f"pair {k}"
    finally:
        lib.mm_idx_destroy(mi)


def _single_end_concurrent(lib, mi, opt, reads, n_threads):
    got = [None] * len(reads)

    def work(t):
        tb = lib.mm_tbuf_init()
        for k in range(t, len(reads), n_threads):
            got[k] = _map_one(lib, mi, opt, tb, *reads[k])
        lib.mm_tbuf_destroy(tb)
    _threads(n_threads, work)
    return got


def test_map_ont_host_path(lib, data):
    mi, opt = _index(lib, data / "ref.fa", b"map-ont")
    try:
        opt.flag |= MM_F_CIGAR
        want = _batch_path(lib, mi, opt, [data / "long.fq"])
        got = _single_end_concurrent(lib, mi, opt, _reads(data / "long.fq"), 8)
        assert got == want and sum(map(len, got)) > 0
    finally:
        lib.mm_idx_destroy(mi)


def test_ava_ont_names(lib, data):
    """-x ava-ont: the reads against themselves; the self/dual filters need each call's qname"""
    mi, opt = _index(lib, data / "long.fq", b"ava-ont")
    try:
        want = _batch_path(lib, mi, opt, [data / "long.fq"])
        got = _single_end_concurrent(lib, mi, opt, _reads(data / "long.fq"), 8)
        assert got == want and sum(map(len, got)) > 0
    finally:
        lib.mm_idx_destroy(mi)


def test_smallest_batch(lib, data):
    """one fragment on 4 lanes, and on 2 GPUs where there are two (one GPU: that part does not run): most shards of the batch are empty"""
    import torch
    n_gpu = torch.cuda.device_count()
    pairs = list(zip(_reads(data / "r1.fq"), _reads(data / "r2.fq")))
    for n_dev in sorted({1, min(n_gpu, 2)}):
        lib.mm_b200_set_lanes(4)
        lib.mm_b200_set_devices(n_dev, (C.c_int * 2)(0, 1))
        try:
            mi, opt = _index(lib, data / "ref.fa", b"sr")
        finally:
            lib.mm_b200_set_lanes(2)
            lib.mm_b200_set_devices(1, (C.c_int * 1)(0))
        try:
            opt.flag |= MM_F_CIGAR | MM_F_OUT_SAM
            assert lib.mm_b200_n_devices(mi) == n_dev
            want = _batch_path(lib, mi, opt, [data / "r1.fq", data / "r2.fq"])
            tb = lib.mm_tbuf_init()
            for k in (0, len(pairs) // 2, len(pairs) - 1):
                (n1, s1), (_, s2) = pairs[k]
                g0, g1 = _map_pair(lib, mi, opt, tb, n1, s1, s2)
                assert g0 == want[2 * k] and g1 == want[2 * k + 1], (n_dev, k)
            lib.mm_tbuf_destroy(tb)
        finally:
            lib.mm_idx_destroy(mi)


def test_index_destroy_joins_dispatcher(lib, data):
    mi, opt = _index(lib, data / "ref.fa", b"sr")
    opt.flag |= MM_F_CIGAR | MM_F_OUT_SAM
    _batch_path(lib, mi, opt, [data / "r1.fq", data / "r2.fq"])
    before = _tasks_settled()
    pairs = list(zip(_reads(data / "r1.fq"), _reads(data / "r2.fq")))[:64]
    _pairs_concurrent(lib, mi, opt, pairs, 8)
    assert _tasks_settled(before + 1) == before + 1  # the dispatcher is running
    lib.mm_idx_destroy(mi)
    assert _tasks_settled(before) <= before
