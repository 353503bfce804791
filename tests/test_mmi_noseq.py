"""Index files written without sequences (--idx-no-seq, header flag MM_I_NO_SEQ), on the CPU.

The loader (airlift_b200/host/refidx.c, mm_idx_load) reads each bucket's p[] and {key, val} pairs (index.c:438-477) and hands
the device builder one entry per distinct minimizer: the minimizer, whether it occurs once, its count, and where its
positions are.  Here a small file is written by hand, following that layout, and the loader's lists are checked against
what the file encodes; positions must come out in the order the file lists them (with HPC the reference orders a run by
hash << 8 | span, not by position).  The loader needs no GPU up to the point where it builds the device table."""
import ctypes as C
import os
import random
import struct
import subprocess
import sys
import pytest
import _libs as L

LIB = os.path.join(L.ROOT, "airlift_b200", "libmm2b200.so")
CLI = os.path.join(L.ROOT, "build", "minimap2-b200")
ONCE = 1 << 63


def _lib():
    if not os.path.exists(LIB):
        pytest.skip("needs airlift_b200/libmm2b200.so")
    lib = C.CDLL(LIB)
    P = C.POINTER
    lib.mm_b200_mmi_lists.restype = C.c_int64
    lib.mm_b200_mmi_lists.argtypes = [C.c_char_p, P(P(C.c_uint64)), P(P(C.c_uint32)), P(P(C.c_uint64)), P(C.c_uint64), P(P(C.c_uint64))]
    lib.mm_b200_mmi_lists_free.argtypes = [P(C.c_uint64), P(C.c_uint32), P(C.c_uint64), P(C.c_uint64)]
    return lib


def _pos(rng, n_seq, lens):
    rid = rng.randrange(n_seq)
    return rid << 32 | rng.randrange(lens[rid]) << 1 | rng.randrange(2)


def write_noseq_mmi(path, w, k, b, flag, names, lens, lists):
    """lists: {minimizer: [positions in the order the file keeps them]}.  Writes one part the way mm_idx_dump lays it out
    (index.c:438-477): per bucket, p[] of the repeated minimizers, then the {key, val} pairs; no sequence."""
    out = bytearray(b"MMI\2" + struct.pack("<5I", w, k, b, len(names), flag | 2))
    for nm, ln in zip(names, lens):
        out += bytes([len(nm)]) + nm + struct.pack("<I", ln)
    mask = (1 << b) - 1
    buckets = [[] for _ in range(1 << b)]
    for m in lists:
        buckets[m & mask].append(m)
    for keys in buckets:
        p, kv = [], []
        for m in keys:  # the pair order within a bucket is the hash table's; any order is a valid file
            ps = lists[m]
            if len(ps) == 1:
                kv.append((m >> b << 1 | 1, ps[0]))
            else:
                kv.append((m >> b << 1, len(p) << 32 | len(ps)))
                p += ps
        out += struct.pack("<i", len(p)) + struct.pack(f"<{len(p)}Q", *p)
        out += struct.pack("<I", len(kv)) + b"".join(struct.pack("<QQ", *x) for x in kv)
    with open(path, "wb") as f:
        f.write(out)
    return len(out)


def make_lists(seed, k, b, hpc):
    rng = random.Random(seed)
    names, lens = [b"chr1", b"chr2", b""], [50000, 70000, 999]
    lists = {}
    n_buckets = 1 << b
    for i in range(600):
        m = rng.randrange(1 << (2 * k))
        if m & (n_buckets - 1) == 5:  # bucket 5 stays empty
            continue
        r = rng.random()
        n = 1 if r < 0.5 else rng.randrange(2, 32) if r < 0.9 else rng.randrange(33, 300)  # singletons, short and long runs
        ps = sorted({_pos(rng, 3, lens) for _ in range(n)})
        if hpc and len(ps) > 2:  # a run ordered by span first, as the reference keeps it with -H
            ps = ps[1::2] + ps[0::2]
        lists[m] = ps
    return names, lens, lists


def read_lists(lib, path):
    key, cnt, src, p = C.POINTER(C.c_uint64)(), C.POINTER(C.c_uint32)(), C.POINTER(C.c_uint64)(), C.POINTER(C.c_uint64)()
    n_p = C.c_uint64()
    n = lib.mm_b200_mmi_lists(os.fsencode(path), C.byref(key), C.byref(cnt), C.byref(src), C.byref(n_p), C.byref(p))
    if n < 0:
        return None
    try:
        got = []
        for i in range(n):
            single = bool(key[i] & ONCE)
            c, s = cnt[i], src[i]
            got.append((key[i] & ~ONCE, single, c, [s] if single else [p[s + j] for j in range(c)]))
        return got, n_p.value
    finally:
        lib.mm_b200_mmi_lists_free(key, cnt, src, p)


@pytest.mark.parametrize("k,b,hpc", [(15, 4, False), (19, 6, True), (21, 14, False)])
def test_loader_lists_are_what_the_file_encodes(tmp_path, k, b, hpc):
    lib = _lib()
    names, lens, lists = make_lists(k * 100 + b, k, b, hpc)
    path = tmp_path / "x.mmi"
    write_noseq_mmi(path, 10, k, b, 1 if hpc else 0, names, lens, lists)
    got, n_p = read_lists(lib, path)
    assert len(got) == len(lists)
    assert sorted(m for m, *_ in got) == sorted(lists)
    for m, single, c, ps in got:
        assert single == (len(lists[m]) == 1)
        assert c == len(lists[m])
        assert ps == lists[m], f"minimizer {m:#x}: positions not in file order"
    assert n_p == sum(len(v) for v in lists.values() if len(v) > 1)
    # the file's order of minimizers is kept as well: bucket by bucket
    buckets = [m & ((1 << b) - 1) for m, *_ in got]
    assert buckets == sorted(buckets) and 5 not in buckets
    assert any(len(v) > 32 for v in lists.values()) and any(len(v) == 1 for v in lists.values())


def test_truncated_file_fails_with_the_loaders_message(tmp_path):
    lib = _lib()
    names, lens, lists = make_lists(3, 15, 4, False)
    full = tmp_path / "full.mmi"
    size = write_noseq_mmi(full, 10, 15, 4, 0, names, lens, lists)
    raw = open(full, "rb").read()
    for cut in (30, size // 3, size - 9):
        path = tmp_path / f"cut{cut}.mmi"
        open(path, "wb").write(raw[:cut])
        # in a child process: the hook prints the loader's message and returns -1
        code = ("import ctypes as C, sys; sys.path.insert(0, %r); import test_mmi_noseq as T; lib = T._lib(); "
                "print(T.read_lists(lib, %r) is None)") % (os.path.dirname(__file__), str(path))
        p = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        assert p.returncode == 0 and p.stdout.strip() == b"True", p.stderr.decode()[-400:]
        assert b"[ERROR] the index file is truncated" in p.stderr
        if os.path.exists(CLI):  # the command line stops at the same message, before it looks for a GPU
            p = subprocess.run([CLI, "-x", "map-ont", str(path), str(path)], stdout=subprocess.PIPE, stderr=subprocess.PIPE)
            assert p.returncode == 1 and p.stdout == b""
            assert b"[ERROR] the index file is truncated" in p.stderr


def test_mappy_refuses_noseq_index_before_the_device(tmp_path):
    sys.path.insert(0, L.ROOT)
    from airlift_b200 import mappy
    names, lens, lists = make_lists(4, 15, 4, False)
    path = tmp_path / "x.mmi"
    write_noseq_mmi(path, 10, 15, 4, 0, names, lens, lists)
    with pytest.raises(ValueError, match="the prebuilt index doesn't contain sequences."):
        mappy.Aligner(str(path), preset="map-ont")
