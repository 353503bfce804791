"""CPU-only checks: the C-ABI library loads and exports every symbol its headers declare (no compute calls
without a GPU), the device layer refuses to start without a device, and the host-side pieces that can run
without a GPU match the compiled reference (or, where it is not built, their results recorded in tests/golden/digests.json)."""
import ctypes as C
import os
import re
import numpy as np
import pytest
import _libs as L

LIB = os.path.join(L.ROOT, "airlift_b200", "libmm2b200.so")


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(LIB):
        import subprocess
        subprocess.check_call(["make", "-C", L.ROOT, "lib"])
    return C.CDLL(LIB)


def _declared(header):
    src = open(os.path.join(L.ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mmg?_[a-z0-9_]+)\s*\(", src)))


@pytest.mark.parametrize("header", ["mmg.h", "minimap_b200.h"])
def test_every_declared_symbol_is_exported(lib, header):
    names = _declared(header)
    assert len(names) > 15
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing


def test_no_device_is_a_loud_error(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    lib.mmg_last_error.restype = C.c_char_p
    ctx = C.c_void_p()
    assert lib.mmg_init(0, C.byref(ctx)) == -1  # MMG_ENODEV
    assert b"no CPU path" in lib.mmg_last_error()


def test_presets_match_reference(lib):
    R = L.ref() if L.have_ref() else None
    io1, mo1 = (C.c_char * 64)(), (C.c_char * 512)()
    io2, mo2 = (C.c_char * 64)(), (C.c_char * 512)()
    assert R is None or R.ref_sizeof_mapopt() <= 512
    mine, theirs = [], []
    for preset in [None, b"sr", b"map-ont", b"map-pb", b"asm5", b"asm10", b"asm20", b"ava-ont", b"ava-pb", b"splice", b"splice:hq", b"short", b"nope"]:
        C.memset(io2, 0, 64); C.memset(mo2, 0, 512)
        lib.mm_set_opt(None, io2, mo2)
        r2 = lib.mm_set_opt(preset, io2, mo2)
        c2 = lib.mm_check_opt(io2, mo2)
        mine.append(repr((preset, r2, io2.raw, mo2.raw, c2)))
        if R is None:
            continue
        C.memset(io1, 0, 64); C.memset(mo1, 0, 512)
        R.mm_set_opt(None, io1, mo1)
        r1 = R.mm_set_opt(preset, io1, mo1)
        c1 = R.mm_check_opt(io1, mo1)
        theirs.append(repr((preset, r1, io1.raw, mo1.raw, c1)))
        assert r1 == r2 and io1.raw == io2.raw and mo1.raw == mo2.raw, preset
        assert c1 == c2
    if R is None:
        L.check_digest("host presets", mine)
    else:
        L.record_reference_digest("host presets", theirs)


def test_host_radix_sorts_match_reference(lib):
    rng = np.random.default_rng(17)
    for n in [0, 3, 64, 65, 1000, 30000]:
        for bits in [4, 20, 64]:
            a = np.zeros(n, dtype=L.mm128)
            a["x"] = rng.integers(0, (1 << bits) - 1, n, dtype=np.uint64, endpoint=True)
            a["y"] = np.arange(n)
            b = a.copy()
            lib.radix_sort_128x(C.c_void_p(a.ctypes.data), C.c_void_p(a.ctypes.data + 16 * n))
            if L.have_ref():
                L.ref().radix_sort_128x(b.ctypes.data, b.ctypes.data + 16 * n)
                assert a.tobytes() == b.tobytes()
                L.record_reference_digest(f"host radix_sort_128x {n} {bits}", b.tobytes())
            else:
                L.check_digest(f"host radix_sort_128x {n} {bits}", a.tobytes())


def test_striped_local_sw_matches_reference(lib):
    """mm_ll_i16 (llsw.c) vs ksw_ll_qinit + ksw_ll_i16 (ksw2_ll_sse.c): score and both end coordinates."""
    R = L.ref() if L.have_ref() else None
    if R is not None:
        R.ksw_ll_qinit.restype = C.c_void_p
        R.ksw_ll_qinit.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        R.ksw_ll_i16.restype = C.c_int
        R.ksw_ll_i16.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.mm_ll_i16.restype = C.c_int
    lib.mm_ll_i16.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    rng = np.random.default_rng(23)
    mat = L.simple_mat(2, 4, 1)
    mine, theirs = [], []
    for it in range(300):
        ql, tl = int(rng.integers(1, 400)), int(rng.integers(1, 400))
        t = L.rand_seq(rng, tl, 0.01)
        q = L.mutate(rng, (t + L.rand_seq(rng, ql))[:ql], 0.1, 0.05, 0.05) if it % 3 else L.rand_seq(rng, ql)
        q = (q + L.rand_seq(rng, ql))[:ql]
        qc, tc = np.ascontiguousarray(L.nt4(q)), np.ascontiguousarray(L.nt4(t))
        qe1, te1, qe2, te2 = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        s2 = lib.mm_ll_i16(ql, qc.ctypes.data, tl, tc.ctypes.data, 5, mat.ctypes.data, 4, 2, C.byref(qe2), C.byref(te2))
        mine.append((s2, qe2.value, te2.value))
        if R is None:
            continue
        qp = R.ksw_ll_qinit(None, 2, ql, qc.ctypes.data, 5, mat.ctypes.data)
        s1 = R.ksw_ll_i16(qp, tl, tc.ctypes.data, 4, 2, C.byref(qe1), C.byref(te1))
        L.libc.free(qp)
        theirs.append((s1, qe1.value, te1.value))
        assert theirs[-1] == mine[-1], (it, ql, tl)
    if R is None:
        L.check_digest("host mm_ll_i16", repr(mine).encode())
    else:
        L.record_reference_digest("host mm_ll_i16", repr(theirs).encode())
