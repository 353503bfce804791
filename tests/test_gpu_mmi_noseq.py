"""Index files written without sequences (--idx-no-seq): the device table is built from the file's minimizer lists
(mmg_idx_build_lists) and must equal the one mmg_idx_build sketches from the sequence; mapping without CIGARs must give the
bytes a FASTA index gives; CIGARs against such an index are refused everywhere, before any kernel could read the missing
sequence (the reference refuses them too, main.c:361-366)."""
import ctypes as C
import hashlib
import json
import os
import struct
import subprocess
import sys
import numpy as np
import pytest
import _libs as L

pytestmark = pytest.mark.gpu
sys.path.insert(0, L.ROOT)
from airlift_b200 import api, mappy  # noqa: E402

NEW = os.path.join(L.ROOT, "build", "minimap2-b200")
SYN = os.path.join(L.ROOT, "build", "mmsynth")
LIB = os.path.join(L.ROOT, "airlift_b200", "libmm2b200.so")
DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mmi_noseq_digests.json")
MSG = b"[ERROR] the prebuilt index doesn't contain sequences."
EINVAL = -3

# name -> (index options, target, queries)
CASES = {
    "sr": (["-x", "sr"], "ref.fa", ["r1.fq", "r2.fq"]),
    "map-ont": (["-x", "map-ont"], "ref.fa", ["long.fq"]),
    "map-pb": (["-x", "map-pb"], "ref.fa", ["long.fq"]),
    "ava-ont": (["-x", "ava-ont"], "long.fq", ["long.fq"]),
    "map-ont-b10": (["-x", "map-ont", "--bucket-bits", "10"], "ref.fa", ["long.fq"]),
}


@pytest.fixture(scope="module")
def data(tmp_path_factory):
    if not (os.path.exists(NEW) and os.path.exists(SYN)):
        pytest.skip("needs build/minimap2-b200 and build/mmsynth")
    d = tmp_path_factory.mktemp("mmi_noseq")
    subprocess.check_call([SYN, "ref", str(d / "ref.fa"), "3000000", "3", "42"])
    subprocess.check_call([SYN, "sr", str(d / "ref.fa"), str(d / "r1.fq"), str(d / "r2.fq"), "4000", "44", "0.05"])
    subprocess.check_call([SYN, "long", str(d / "ref.fa"), str(d / "long.fq"), "40", "45"])
    for name, (args, target, _) in CASES.items():
        _ok([NEW] + args + ["-d", f"{name}.seq.mmi", target], d)
        _ok([NEW] + args + ["--idx-no-seq", "-d", f"{name}.noseq.mmi", target], d)
    return d


def _run(cmd, cwd):
    return subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)


def _ok(cmd, cwd):
    p = _run(cmd, cwd)
    assert p.returncode == 0, p.stderr.decode()[-800:]
    return p


def _lib():
    lib = C.CDLL(LIB)
    P = C.c_void_p
    for f, res, args in [("mm_idx_reader_open", P, [C.c_char_p, P, C.c_char_p]), ("mm_idx_reader_read", P, [P, C.c_int]),
                         ("mm_idx_reader_close", None, [P]), ("mm_idx_destroy", None, [P]), ("mm_b200_ctx", P, [P, C.c_int]),
                         ("mm_b200_didx", P, [P, C.c_int]), ("mmg_idx_n_keys", C.c_int64, [P]), ("mmg_idx_n_minimizers", C.c_int64, [P]),
                         ("mmg_idx_n_singletons", C.c_int64, [P]), ("mmg_idx_has_seq", C.c_int, [P]), ("mmg_idx_bytes", C.c_size_t, [P]),
                         ("mmg_idx_cal_max_occ", C.c_int, [P, C.c_float, C.POINTER(C.c_int32)]),
                         ("mmg_idx_export_sorted", C.c_int, [P, P, C.c_int, P, P, P]), ("mmg_idx_copy_S", C.c_int, [P, P]),
                         ("mmg_launch_count", C.c_long, [P, C.c_int]), ("mmg_last_error", C.c_char_p, []),
                         ("mmg_ksw_batch", C.c_int, [P, P, P, C.c_int, P, P, P, P, P]),
                         ("mmg_post_chain", C.c_int, [P, P, P, P, C.c_size_t, C.c_int, P, P]),
                         ("mm_b200_make_batch", P, [C.c_int, P, P, P, P]), ("mm_b200_free_batch", None, [P]),
                         ("mm_b200_map_batch", C.c_int, [P, P, C.c_int, P, C.c_int]), ("mm_b200_batch_digest", C.c_uint64, [P, P]),
                         ("mm_mapopt_update", None, [P, P])]:
        getattr(lib, f).restype = res
        getattr(lib, f).argtypes = args
    return lib


class _Idx:
    """the first part of an index file, loaded through the library"""

    def __init__(self, lib, path):
        self.lib = lib
        rd = lib.mm_idx_reader_open(os.fsencode(str(path)), None, None)
        assert rd
        self.mi = lib.mm_idx_reader_read(rd, 4)
        lib.mm_idx_reader_close(rd)
        assert self.mi
        self.b = struct.unpack_from("<5I", open(path, "rb").read(24), 4)[2]
        self.ctx, self.didx = lib.mm_b200_ctx(self.mi, 0), lib.mm_b200_didx(self.mi, 0)

    def close(self):
        self.lib.mm_idx_destroy(self.mi)

    def table(self):
        lib, d = self.lib, self.didx
        n, n_pos = lib.mmg_idx_n_keys(d), lib.mmg_idx_n_minimizers(d)
        keys, vals, pos = np.zeros(n + 1, np.uint64), np.zeros(n + 1, np.uint64), np.zeros(n_pos + 1, np.uint64)
        assert lib.mmg_idx_export_sorted(self.ctx, d, self.b, keys.ctypes.data, vals.ctypes.data, pos.ctypes.data) == 0, lib.mmg_last_error()
        occ = []
        for f in (2e-4, 1e-3, 0.01):
            t = C.c_int32()
            assert lib.mmg_idx_cal_max_occ(d, f, C.byref(t)) == 0
            occ.append(t.value)
        return dict(n_keys=n, n_pos=n_pos, n1=lib.mmg_idx_n_singletons(d), occ=occ, keys=keys[:n], vals=vals[:n], pos=pos[:n_pos])


@pytest.mark.parametrize("name", list(CASES))
def test_same_table(data, name):
    lib = _lib()
    a, b = _Idx(lib, data / f"{name}.seq.mmi"), _Idx(lib, data / f"{name}.noseq.mmi")
    try:
        assert lib.mmg_idx_has_seq(a.didx) == 1 and lib.mmg_idx_has_seq(b.didx) == 0
        ta, tb = a.table(), b.table()
        for f in ("n_keys", "n_pos", "n1", "occ"):
            assert ta[f] == tb[f], f
        assert ta["n_keys"] > 1000 and ta["n1"] > 0
        for f in ("keys", "vals", "pos"):
            assert np.array_equal(ta[f], tb[f]), f"{f}: first difference at {np.flatnonzero(ta[f] != tb[f])[:1]}"
        assert lib.mmg_idx_bytes(a.didx) - lib.mmg_idx_bytes(b.didx) > 0  # the sequence is left out
    finally:
        a.close(); b.close()


def _same_bytes(data, args, target, queries, extra=()):
    fa = _ok([NEW] + args + list(extra) + ["-t", "8", target] + queries, data).stdout
    assert len(fa) > 1000
    for idx in (f"{target}.seq.mmi", f"{target}.noseq.mmi"):
        got = _ok([NEW] + args + list(extra) + ["-t", "8", idx] + queries, data).stdout
        assert got == fa, f"{idx}: output differs from the FASTA index's"
    return fa


@pytest.mark.parametrize("name", ["sr", "map-ont", "map-pb", "ava-ont"])
def test_same_bytes_out(data, name):
    args, target, queries = CASES[name]
    _ok([NEW] + args + ["-d", f"{target}.seq.mmi", target], data)
    _ok([NEW] + args + ["--idx-no-seq", "-d", f"{target}.noseq.mmi", target], data)
    _same_bytes(data, args, target, queries)


def test_same_bytes_out_multi_part(data):
    args = ["-x", "sr", "-I", "1M"]
    _ok([NEW] + args + ["-d", "ref.fa.seq.mmi", "ref.fa"], data)
    _ok([NEW] + args + ["--idx-no-seq", "-d", "ref.fa.noseq.mmi", "ref.fa"], data)
    raw = open(data / "ref.fa.noseq.mmi", "rb").read()
    assert raw.count(b"MMI\2") >= 2  # one part after another
    _same_bytes(data, args, "ref.fa", ["r1.fq", "r2.fq"])


def test_same_bytes_out_two_gpus(data):
    if api.lib().mmg_device_count() < 2:
        pytest.skip("needs two GPUs")
    args = ["-x", "map-ont"]
    _ok([NEW] + args + ["-d", "ref.fa.seq.mmi", "ref.fa"], data)
    _ok([NEW] + args + ["--idx-no-seq", "-d", "ref.fa.noseq.mmi", "ref.fa"], data)
    one = _same_bytes(data, args, "ref.fa", ["long.fq"])
    assert _same_bytes(data, args, "ref.fa", ["long.fq"], ["--gpus", "2"]) == one


@pytest.mark.parametrize("name", ["sr", "map-pb"])
def test_round_trip(data, name):
    args = CASES[name][0]
    _ok([NEW] + args + ["-d", f"{name}.again.mmi", f"{name}.noseq.mmi"], data)
    assert open(data / f"{name}.noseq.mmi", "rb").read() == open(data / f"{name}.again.mmi", "rb").read()


@pytest.mark.parametrize("opt", [["-a"], ["-c"], ["--cs"], ["-c", "--MD"], ["-a", "--MD"]], ids=" ".join)
def test_cli_refuses_cigar(data, opt):
    p = _run([NEW, "-x", "sr"] + opt + ["sr.noseq.mmi", "r1.fq", "r2.fq"], data)
    assert p.returncode != 0 and p.stdout == b""
    assert MSG in p.stderr
    # a FASTA index made without -a/-c also carries MM_I_NO_SEQ in memory (main.c:262) and keeps mapping with CIGARs
    assert _run([NEW, "-x", "sr"] + opt + ["ref.fa", "r1.fq", "r2.fq"], data).returncode == 0


def test_md_alone_maps(data):
    """--MD alone does not ask for CIGARs (MM_F_CIGAR), as in the reference's main.c: PAF comes out as without it"""
    plain = _ok([NEW, "-x", "sr", "-t", "8", "sr.noseq.mmi", "r1.fq", "r2.fq"], data).stdout
    assert _ok([NEW, "-x", "sr", "--MD", "-t", "8", "sr.noseq.mmi", "r1.fq", "r2.fq"], data).stdout == plain


def test_library_refuses_cigar(data):
    lib = _lib()
    ix = _Idx(lib, data / "map-ont.noseq.mmi")
    try:
        reads = [l.strip() for i, l in enumerate(open(data / "long.fq", "rb")) if i % 4 == 1][:4]
        n = len(reads)
        batch = lib.mm_b200_make_batch(n, (C.c_int * n)(*([1] * n)), (C.c_int * n)(*map(len, reads)), (C.c_char_p * n)(*reads), None)
        io, mo = mappy.set_options("map-ont")
        lib.mm_mapopt_update(C.byref(mo), ix.mi)
        assert mo.flag & mappy.MM_F_CIGAR
        launches = lib.mmg_launch_count(ix.ctx, 0)
        assert lib.mm_b200_map_batch(ix.mi, C.byref(mo), 4, batch, 0) == -1
        assert lib.mmg_launch_count(ix.ctx, 0) == launches
        mo.flag &= ~mappy.MM_F_CIGAR  # without CIGARs the same batch maps
        assert lib.mm_b200_map_batch(ix.mi, C.byref(mo), 4, batch, 0) == 0
        n_hits = C.c_int64()
        lib.mm_b200_batch_digest(batch, C.byref(n_hits))
        assert n_hits.value > 0
        lib.mm_b200_free_batch(batch)
        # the C-ABI entries that would read the sequence refuse before any launch
        ctx, d = ix.ctx, ix.didx
        before = lib.mmg_launch_count(ctx, 0)
        S = np.zeros(1 << 20, np.uint32)
        assert lib.mmg_idx_copy_S(d, S.ctypes.data) == EINVAL
        dopt = api.ont_opt(50)
        jobs, res, cig = (api.KswJob * 1)(), (api.KswRes * 1)(), C.c_void_p()
        assert lib.mmg_ksw_batch(ctx, d, C.byref(dopt), 1, jobs, res, C.byref(cig), None, None) == EINVAL
        assert b"sequence" in lib.mmg_last_error()
        io, mo = mappy.set_options("sr")
        out, h = C.create_string_buffer(512), (C.c_uint32 * 1)()
        assert lib.mmg_post_chain(ctx, d, C.byref(api.sr_opt()), C.byref(mo), C.sizeof(mo), 0, h, out) == EINVAL
        assert lib.mmg_launch_count(ctx, 0) == before
    finally:
        ix.close()


def test_mappy_refuses(data):
    with pytest.raises(ValueError, match="the prebuilt index doesn't contain sequences."):
        mappy.Aligner(str(data / "sr.noseq.mmi"), preset="sr")
    assert mappy.Aligner(str(data / "sr.seq.mmi"), preset="sr")  # the same index with its sequence loads


def test_reference_written_noseq_index(data):
    """A no-sequence .mmi written by the reference maps as the reference maps the FASTA.  Without the reference fork, this
    project's file and output stand in, held to the digest recorded in golden/mmi_noseq_digests.json."""
    key = "map -x map-ont noseq.mmi long.fq"
    if L.have_ref_bin():
        _ok([L.REF_BIN_B, "-x", "map-ont", "--idx-no-seq", "-d", "ref_noseq.mmi", "ref.fa"], data)
        want = _ok([L.REF_BIN_B, "-x", "map-ont", "-t", "8", "ref.fa", "long.fq"], data).stdout
        got = _ok([NEW, "-x", "map-ont", "-t", "8", "ref_noseq.mmi", "long.fq"], data).stdout
        assert got == want
        return
    _ok([NEW, "-x", "map-ont", "--idx-no-seq", "-d", "own_noseq.mmi", "ref.fa"], data)
    got = _ok([NEW, "-x", "map-ont", "-t", "8", "own_noseq.mmi", "long.fq"], data).stdout
    with open(DIGESTS) as f:
        want = json.load(f)[key]
    assert {"bytes": len(got), "sha256": hashlib.sha256(got).hexdigest()} == {k: want[k] for k in ("bytes", "sha256")}
