"""airlift_b200.mappy without a GPU: revcomp, fastx_read against the mapper's own reader (held to the reference's bseq.c by
test_reader.py), the errors raised before anything touches a device, and where the keyword overrides land in mm_mapopt_t."""
import ctypes as C
import gzip
import os
import numpy as np
import pytest
import _libs as L
from airlift_b200 import mappy as mp
from test_reader import _fastq, _new_batches

OUT_SAM, COPY_COMMENT = 0x008, 0x2000000


def test_revcomp_iupac_and_lowercase():
    lib = C.CDLL(mp.LIB_PATH)
    table = (C.c_ubyte * 256).in_dll(lib, "seq_comp_table")
    s = "ACGTUMRWSYKVHDBNacgtumrwsykvhdbnXx-.*"
    assert mp.revcomp(s) == "".join(chr(table[ord(c)]) for c in reversed(s))
    assert mp.revcomp("AACGTn") == "nACGTT" and mp.revcomp("") == "" and mp.revcomp(None) is None


@pytest.mark.parametrize("case", ["fastq", "comment", "fasta", "gz"])
def test_fastx_read_matches_reader(tmp_path, case):
    rng = np.random.default_rng(sum(map(ord, case)))
    if case == "fasta":
        txt = "".join(f">s{i} d{i}\n" + "\n".join(L.rand_seq(rng, int(rng.integers(1, 90))).decode() for _ in range(int(rng.integers(1, 6)))) + "\n"
                      for i in range(300))
    else:
        txt = _fastq(rng, 500, "/1" if case == "fastq" else "", comment=case in ("comment", "gz"))
    fn = str(tmp_path / ("r.fq.gz" if case == "gz" else "r.fq"))
    if case == "gz":
        with gzip.open(fn, "wt") as f:
            f.write(txt)
    else:
        open(fn, "w").write(txt)
    new = C.CDLL(os.path.join(L.ROOT, "airlift_b200", "libmm2b200.so"))
    new.mm_b200_open_reads.restype = C.c_void_p; new.mm_b200_open_reads.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    new.mm_b200_close_reads.argtypes = [C.c_void_p]
    new.mm_b200_read_batch.restype = C.c_void_p; new.mm_b200_read_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    new.mm_b200_free_batch.argtypes = [C.c_void_p]
    want = [r for b in _new_batches(new, [fn], 10**9, OUT_SAM | COPY_COMMENT) for r in b]
    dec = lambda x: x.decode() if x is not None else None  # noqa: E731
    got = list(mp.fastx_read(fn, read_comment=True))
    assert got == [(dec(n), dec(s), dec(q), dec(c)) for _, n, s, q, c in want]
    assert list(mp.fastx_read(fn)) == [g[:3] for g in got]
    assert len(got) == (300 if case == "fasta" else 500)
    assert list(mp.fastx_read(str(tmp_path / "missing.fq"))) == []


def test_no_device_raises_runtime_error(tmp_path):
    if mp._L().mmg_device_count() > 0:
        pytest.skip("a CUDA device is present")
    fa = tmp_path / "ref.fa"
    fa.write_text(">c\n" + "ACGT" * 1000 + "\n")
    with pytest.raises(RuntimeError, match="no CUDA device"):
        mp.Aligner(str(fa), preset="map-ont")
    with pytest.raises(RuntimeError):
        mp.Aligner(seq="ACGT" * 1000)
    assert mp.revcomp("ACG") == "CGT"  # still here


@pytest.mark.parametrize("kw", [dict(preset="splice"), dict(preset="splice:hq"), dict(preset="map-ont", extra_flags=0x080),
                                dict(preset="sr", extra_flags=0x001)])
def test_refused_options_raise_value_error(tmp_path, kw):
    fa = tmp_path / "ref.fa"
    fa.write_text(">c\n" + "ACGT" * 1000 + "\n")
    with pytest.raises(ValueError, match="is not supported by this build"):
        mp.Aligner(str(fa), **kw)
    io, mo = mp.IdxOpt(), mp.MapOpt()
    mp._L().mm_set_opt(None, C.byref(io), C.byref(mo))
    mp._L().mm_set_opt(kw["preset"].encode(), C.byref(io), C.byref(mo))
    mo.flag |= mp.MM_F_CIGAR | kw.get("extra_flags", 0)
    with pytest.raises(ValueError) as e:
        mp.set_options(**kw)
    assert str(e.value) == mp._L().mm_b200_opt_error(C.byref(mo)).decode()
    with pytest.raises(ValueError, match="unknown preset"):
        mp.set_options("no-such-preset")


def _by_hand(preset, edit):
    io, mo = mp.IdxOpt(), mp.MapOpt()
    mp._L().mm_set_opt(None, C.byref(io), C.byref(mo))
    if preset:
        mp._L().mm_set_opt(preset.encode(), C.byref(io), C.byref(mo))
    mo.flag |= mp.MM_F_CIGAR
    io.batch_size = 0x7fffffffffffffff
    edit(io, mo)
    return bytes(io), bytes(mo)


def _set(**f):
    def edit(io, mo):
        for k, v in f.items():
            setattr(io if k in ("k", "w") else mo, k, v)
    return edit


@pytest.mark.parametrize("preset,kw,edit", [
    (None, {}, _set()),
    ("map-ont", dict(k=13, w=7), _set(k=13, w=7)),
    ("sr", dict(min_cnt=4, min_chain_score=33, min_dp_score=50, bw=123, best_n=9, max_frag_len=700),
     _set(min_cnt=4, min_chain_score=33, min_dp_max=50, bw=123, best_n=9, max_frag_len=700)),
    ("map-pb", dict(extra_flags=0x4000), lambda io, mo: setattr(mo, "flag", mo.flag | 0x4000)),
    ("map-ont", dict(scoring=[3, 5, 7, 2]), _set(a=3, b=5, q=7, e=2, q2=7, e2=2)),
    ("map-ont", dict(scoring=[3, 5, 7, 2, 30, 1]), _set(a=3, b=5, q=7, e=2, q2=30, e2=1)),
    ("asm5", dict(scoring=[3, 5, 7, 2, 30, 1, 2]), _set(a=3, b=5, q=7, e=2, q2=30, e2=1, sc_ambi=2)),
    ("map-ont", dict(scoring=[3, 5]), _set()),
])
def test_overrides_land_in_their_fields(preset, kw, edit):
    io, mo = mp.set_options(preset, **kw)
    assert (bytes(io), bytes(mo)) == _by_hand(preset, edit)
