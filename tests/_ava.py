"""Shared pieces of the all-vs-all tests (test_ava_opt.py, test_gpu_ava.py): the strcmp oracle of seed collection with the
self/dual filters (tests/aux/ava_oracle.c, linked with oracle/mm2_oracle.c), the name keys of include/mmg.h as the library
computes them, and the named cases.  Test infrastructure only."""
import ctypes as C
import os
import subprocess
import tempfile
import numpy as np
import _libs as L

MM_F_NO_DIAG, MM_F_NO_DUAL, MM_F_FOR_ONLY, MM_F_REV_ONLY, MM_F_HEAP_SORT = 0x001, 0x002, 0x100000, 0x200000, 0x400000
SEED_SELF = np.uint64(1 << 43)
NAME_NONE = 0xffffffff
W, K = 10, 15
FLAGS = [f | s for f in (MM_F_NO_DIAG, MM_F_NO_DUAL, MM_F_NO_DIAG | MM_F_NO_DUAL) for s in (0, MM_F_FOR_ONLY, MM_F_REV_ONLY)]

_orc = None


def oracle_named():
    global _orc
    if _orc is None:
        d = tempfile.mkdtemp(prefix="airlift_ava_oracle_")
        so = os.path.join(d, "libava_oracle.so")
        subprocess.check_call(["gcc", "-shared", "-fPIC", "-O2", "-ffp-contract=off", "-I" + L.ORACLE_DIR,
                               os.path.join(L.ROOT, "tests", "aux", "ava_oracle.c"), os.path.join(L.ORACLE_DIR, "mm2_oracle.c"),
                               "-o", so, "-lm"])
        O = C.CDLL(so)
        O.orc_idx_build.restype = C.c_void_p
        O.orc_idx_build.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_char_p)]
        O.orc_idx_destroy.argtypes = [C.c_void_p]
        O.orc_collect_seeds_named.restype = C.c_int64
        O.orc_collect_seeds_named.argtypes = [C.c_void_p, C.POINTER(C.c_char_p), C.c_void_p, C.c_char_p, C.c_int, C.c_int64, C.c_int, C.c_int,
                                              C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]
        O.orc_chain_dp.restype = C.c_int
        O.orc_chain_dp.argtypes = [C.c_int] * 9 + [C.c_int64, C.c_void_p, C.c_void_p]
        _orc = O
    return _orc


class Targets:
    """the oracle's index of the targets, with their names"""
    def __init__(self, names, seqs):
        self.names, self.seqs = names, seqs
        self.c_names = L.c_str_array(names)
        self.lens = np.array([len(s) for s in seqs], dtype=np.uint32)
        self.oi = oracle_named().orc_idx_build(W, K, 0, len(seqs), L.c_str_array(seqs))

    def close(self):
        oracle_named().orc_idx_destroy(self.oi)

    def collect(self, qname, heap, flag, max_occ, mv, qlen):
        """anchors, rep_len, number of seed hits the self/dual filters dropped"""
        O = oracle_named()
        rep, nm, nn = C.c_int(0), C.c_int(0), C.c_int64(0)
        mv = np.ascontiguousarray(mv)
        n = O.orc_collect_seeds_named(self.oi, self.c_names, self.lens.ctypes.data, qname, int(heap), flag, max_occ, len(mv), mv.ctypes.data,
                                      qlen, None, C.byref(rep), C.byref(nm), C.byref(nn))
        a = np.zeros(n + 1, dtype=L.mm128)
        n = O.orc_collect_seeds_named(self.oi, self.c_names, self.lens.ctypes.data, qname, int(heap), flag, max_occ, len(mv), mv.ctypes.data,
                                      qlen, a.ctypes.data, C.byref(rep), C.byref(nm), C.byref(nn))
        return a[:n].copy(), rep.value, nn.value


def name_lib(path):
    lib = C.CDLL(path)
    lib.mm_b200_name_order.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_char_p), C.c_void_p]
    lib.mm_b200_name_ukey.restype = C.c_uint32
    lib.mm_b200_name_ukey.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.c_char_p]
    return lib


def name_keys(lib, tnames, qnames):
    """(tkey array, [ukey per query name]) as the library computes them"""
    n = len(tnames)
    sorted_ = (C.c_char_p * max(n, 1))()
    tkey = np.zeros(max(n, 1), dtype=np.uint32)
    lib.mm_b200_name_order(n, L.c_str_array(tnames), sorted_, tkey.ctypes.data)
    return tkey[:n], [lib.mm_b200_name_ukey(n, sorted_, q) for q in qnames]


def make_targets(rng):
    """targets whose names exercise every branch of skip_seed: 'long10' < 'long2', a duplicated name, a repeat inside 'long2'
    (off-diagonal self hits on both strands)"""
    a = bytearray(L.rand_seq(rng, 6000))
    a[3000:3600] = a[500:1100]                       # same-strand repeat: off-diagonal self hits
    a[4500:5000] = L.revcomp(bytes(a[1500:2000]))    # opposite-strand repeat
    names = [b"long2", b"long10", b"dup", b"ctg", b"dup"]
    seqs = [bytes(a), L.rand_seq(rng, 5000), L.rand_seq(rng, 4000), L.rand_seq(rng, 4500), L.rand_seq(rng, 3000)]
    return names, seqs


def make_queries(rng, names, seqs):
    """(qname, sequence) pairs: a target under its own name and length, the same name with another length, the same sequence
    under other names, names sorting between, above and below the targets', a duplicated target name, and no name"""
    a = seqs[0]
    return [(b"long2", a), (b"long2", a[:5000]), (b"other", a), (b"long1", a), (b"long3", L.mutate(rng, a[200:5200])),
            (b"aaa", a), (b"zzz", L.mutate(rng, seqs[1])), (b"dup", seqs[2]), (b"dup", L.mutate(rng, seqs[4])), (b"long10", seqs[1]),
            (None, a), (b"ctg", L.mutate(rng, seqs[3][100:4000]))]
