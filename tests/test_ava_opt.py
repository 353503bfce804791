"""CPU-only checks of the all-vs-all modes (-D, -X, --dual=no, -x ava-ont / ava-pb): the device's seed collection with the
self/dual filters, compiled by g++ (tests/emu), against the strcmp oracle (tests/aux/ava_oracle.c), byte for byte with the
MM_SEED_SELF bit; the name keys; the option check and the CLI."""
import ctypes as C
import os
import subprocess
import numpy as np
import pytest
import _libs as L
import _ava as A

LIB = os.path.join(L.ROOT, "airlift_b200", "libmm2b200.so")
EMU_SO = os.path.join(L.ROOT, "build", "libmmg_emu_named.so")
CLI = os.path.join(L.ROOT, "build", "minimap2-b200")


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        subprocess.check_call(["make", "-C", L.ROOT, "lib"])
    import bench
    lib = A.name_lib(LIB)
    lib.mm_set_opt.argtypes = [C.c_char_p, C.POINTER(bench.IdxOpt), C.POINTER(bench.MapOptFull)]
    lib.mm_b200_check_opt.argtypes = [C.POINTER(bench.MapOptFull)]
    return lib


@pytest.fixture(scope="module")
def emu():
    subprocess.check_call(["make", "-C", L.ROOT, "emu"], stdout=subprocess.DEVNULL)
    E = C.CDLL(EMU_SO)
    E.emu_idx_new.restype = C.c_void_p
    E.emu_idx_new.argtypes = [C.c_int64, C.c_void_p, C.c_void_p]
    E.emu_idx_free.argtypes = [C.c_void_p]
    E.emu_collect_named.restype = C.c_int64
    E.emu_collect_named.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                    C.c_void_p, C.c_int64, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p, C.POINTER(C.c_int64)]
    return E


def _index_arrays(seqs):
    mv = np.concatenate([L.orc_sketch(s, A.W, A.K, i) for i, s in enumerate(seqs)])
    key = mv["x"] >> np.uint64(8)
    order = np.lexsort((mv["y"], key))
    return np.ascontiguousarray(key[order]), np.ascontiguousarray(mv["y"][order])


def test_name_keys_follow_strcmp(lib):
    tnames = [b"long2", b"long10", b"dup", b"b", b"dup", b"\xffhigh"]
    qnames = [b"long2", b"long1", b"long3", b"a", b"dup", b"zz", b"\xff", b"\xffhigh", b"", None]
    tkey, ukey = A.name_keys(lib, tnames, qnames)
    for q, uk in zip(qnames, ukey):
        if q is None:
            assert uk == A.NAME_NONE
            continue
        for t, tk in zip(tnames, tkey):
            cmp = (q > t) - (q < t)  # bytes compare as unsigned char, as strcmp does
            assert (uk == tk) == (cmp == 0) and (tk < uk) == (cmp > 0), (q, t, uk, tk)
    assert tkey[2] == tkey[4]  # equal names, equal keys


@pytest.mark.parametrize("heap", [0, 1], ids=["radix", "heap"])
def test_filters_equal_strcmp_oracle(lib, emu, heap):
    rng = np.random.default_rng(5)
    names, seqs = A.make_targets(rng)
    T = A.Targets(names, seqs)
    key, pos = _index_arrays(seqs)
    ei = emu.emu_idx_new(len(key), key.ctypes.data, pos.ctypes.data)
    queries = A.make_queries(rng, names, seqs)
    tkey, ukeys = A.name_keys(lib, names, [q for q, _ in queries])
    tlen = T.lens
    n_self = n_named = 0
    try:
        for (qname, q), ukey in zip(queries, ukeys):
            mv, qlen = L.frag_minimizers(L.orc_sketch, [q], A.W, A.K)
            for flag in A.FLAGS + [0]:
                flag |= A.MM_F_HEAP_SORT if heap else 0
                want, rep, nn = T.collect(qname, heap, flag, 1000, mv, qlen)
                a = np.zeros(len(mv) * 8 + 64, dtype=L.mm128)
                rep2, nm2, nn2 = C.c_int(0), C.c_int(0), C.c_int64(0)
                n = emu.emu_collect_named(ei, tkey.ctypes.data, tlen.ctypes.data, ukey, heap, flag, 1000, len(mv), mv.ctypes.data, qlen,
                                          a.ctypes.data, len(a), C.byref(rep2), C.byref(nm2), None, C.byref(nn2))
                assert n == len(want) and a[:n].tobytes() == want.tobytes() and rep2.value == rep and nn2.value == nn, (qname, hex(flag))
                n_self += int(((want["y"] & A.SEED_SELF) != 0).sum())
                n_named += nn
    finally:
        emu.emu_idx_free(ei)
        T.close()
    assert n_self > 0 and n_named > 0  # the cases reach both the self bit and the drops


def _opt(lib, preset):
    import bench
    ipt, opt = bench.IdxOpt(), bench.MapOptFull()
    lib.mm_set_opt(None, C.byref(ipt), C.byref(opt))
    assert lib.mm_set_opt(preset, C.byref(ipt), C.byref(opt)) == 0
    return opt


@pytest.mark.parametrize("preset", [b"map-ont", b"map-pb", b"asm5"])
@pytest.mark.parametrize("flags", [A.MM_F_NO_DIAG, A.MM_F_NO_DUAL, A.MM_F_NO_DIAG | A.MM_F_NO_DUAL], ids=["-D", "--dual=no", "-X"])
def test_filters_accepted_with_long_read_presets(lib, preset, flags):
    opt = _opt(lib, preset)
    opt.flag |= flags
    assert lib.mm_b200_check_opt(C.byref(opt)) == 0


@pytest.mark.parametrize("preset", [b"ava-ont", b"ava-pb"])
def test_ava_presets_accepted(lib, preset):
    opt = _opt(lib, preset)
    assert opt.flag & (A.MM_F_NO_DIAG | A.MM_F_NO_DUAL) == A.MM_F_NO_DIAG | A.MM_F_NO_DUAL
    assert lib.mm_b200_check_opt(C.byref(opt)) == 0


@pytest.mark.parametrize("flags", [A.MM_F_NO_DIAG, A.MM_F_NO_DUAL, A.MM_F_NO_DIAG | A.MM_F_NO_DUAL], ids=["-D", "--dual=no", "-X"])
def test_filters_still_refused_with_sr(lib, flags):
    opt = _opt(lib, b"sr")
    opt.flag |= flags
    assert lib.mm_b200_check_opt(C.byref(opt)) == -1


@pytest.mark.parametrize("args", [["-x", "ava-ont"], ["-x", "ava-pb"], ["-x", "map-ont", "-D"], ["-x", "map-pb", "--dual=no"], ["-cx", "ava-ont"]])
def test_cli_takes_ava_to_the_index(tmp_path, args):
    if not os.path.exists(CLI):
        pytest.skip("needs build/minimap2-b200")
    fa = tmp_path / "missing.fa"
    p = subprocess.run([CLI] + args + [str(fa), str(fa)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert b"not supported by this build" not in p.stderr
    assert b"failed to open file" in p.stderr, p.stderr[-400:]
