"""Host logic, no GPU: the FASTA/FASTQ reader (fast four-line path, general parser, per-file read-ahead threads, packed
records) against the reference's own reader (bseq.c / kseq.h through oracle/_ref/libmm2ref.so) on the same files:
same records, same batch boundaries, same pair handling.  Without the reference build, the batches are checked against their
digests recorded in tests/golden/digests.json."""
import ctypes as C
import gzip
import os
import numpy as np
import pytest
import _libs as L


class Bseq1(C.Structure):  # mm_bseq1_t, bseq.h:14-17
    _fields_ = [("l_seq", C.c_int), ("rid", C.c_int), ("name", C.c_char_p), ("seq", C.c_char_p), ("qual", C.c_char_p), ("comment", C.c_char_p)]


class StepHead(C.Structure):  # leading fields of the mapper's batch (mapper.c step_t)
    _fields_ = [("n_seq", C.c_int), ("n_frag", C.c_int), ("seq", C.POINTER(Bseq1)), ("n_reg", C.POINTER(C.c_int)), ("seg_off", C.POINTER(C.c_int)),
                ("n_seg", C.POINTER(C.c_int))]


@pytest.fixture(scope="module")
def libs():
    new = C.CDLL(os.path.join(L.ROOT, "airlift_b200", "libmm2b200.so"))
    new.mm_b200_open_reads.restype = C.c_void_p; new.mm_b200_open_reads.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    new.mm_b200_close_reads.argtypes = [C.c_void_p]
    new.mm_b200_read_batch.restype = C.c_void_p; new.mm_b200_read_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    new.mm_b200_free_batch.argtypes = [C.c_void_p]
    if not os.path.exists(L.REF_SO):
        return new, None
    ref = C.CDLL(L.REF_SO)
    ref.mm_bseq_open.restype = C.c_void_p; ref.mm_bseq_open.argtypes = [C.c_char_p]
    ref.mm_bseq_close.argtypes = [C.c_void_p]
    ref.mm_bseq_read3.restype = C.POINTER(Bseq1)
    ref.mm_bseq_read3.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
    ref.mm_bseq_read_frag2.restype = C.POINTER(Bseq1)
    ref.mm_bseq_read_frag2.argtypes = [C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
    return new, ref


def _rec(r):
    return (r.l_seq, r.name, r.seq, r.qual, r.comment)


def _ref_batches(ref, files, chunk, with_qual, with_comment, frag_mode):
    fps = [ref.mm_bseq_open(f.encode()) for f in files]
    out = []
    while True:
        n = C.c_int(0)
        if len(files) > 1:
            arr = (C.c_void_p * len(fps))(*fps)
            a = ref.mm_bseq_read_frag2(len(fps), arr, chunk, with_qual, with_comment, C.byref(n))
        else:
            a = ref.mm_bseq_read3(fps[0], chunk, with_qual, with_comment, frag_mode, C.byref(n))
        if not a or n.value == 0:
            break
        out.append([_rec(a[i]) for i in range(n.value)])
    for fp in fps:
        ref.mm_bseq_close(fp)
    return out


def _check(ref, key, got, files, chunk, with_qual, with_comment, frag_mode):
    """got (batches of records) against the reference's reader on the same files; without it, against the digest recorded for key"""
    if ref is None:
        L.check_digest("reader " + key, repr(got).encode())
        return
    want = _ref_batches(ref, files, chunk, with_qual, with_comment, frag_mode)
    assert [len(b) for b in want] == [len(b) for b in got], key
    assert want == got, key
    L.record_reference_digest("reader " + key, repr(want).encode())


def _new_batches(new, files, chunk, flag):
    import bench
    opt = bench.MapOptFull()
    opt.flag = flag
    fns = (C.c_char_p * len(files))(*[f.encode() for f in files])
    rd = new.mm_b200_open_reads(len(files), fns)
    out = []
    while True:
        b = new.mm_b200_read_batch(rd, C.byref(opt), chunk)
        if not b:
            break
        h = C.cast(b, C.POINTER(StepHead)).contents
        out.append([_rec(h.seq[i]) for i in range(h.n_seq)])
        new.mm_b200_free_batch(b)
    new.mm_b200_close_reads(rd)
    return out


def _fastq(rng, n, tag, comment=False, crlf=False, wrap=0, blank=False, lower=False):
    nl = "\r\n" if crlf else "\n"
    s = []
    for i in range(n):
        l = int(rng.integers(1, 300))
        seq = L.rand_seq(rng, l, 0.02).decode()
        if lower:
            seq = seq.lower().replace("t", "u") if i % 3 == 0 else seq.replace("T", "U")
        qual = "".join(chr(33 + int(x)) for x in rng.integers(0, 41, l))  # includes '@', '+', '>' as quality characters
        name = f"@r{i}{tag}" + (f" c{i}\tx y" if comment and i % 2 else "")
        if wrap:
            seq_l = nl.join(seq[j:j + wrap] for j in range(0, l, wrap))
            qual_l = nl.join(qual[j:j + wrap] for j in range(0, l, wrap))
            if any(q[0] in "@" for q in qual_l.split(nl)):  # a wrapped quality line starting with '@' is ambiguous even for kseq: avoid
                qual = qual.replace("@", "A"); qual_l = nl.join(qual[j:j + wrap] for j in range(0, l, wrap))
        else:
            seq_l, qual_l = seq, qual
        s.append(f"{name}{nl}{seq_l}{nl}+{nl}{qual_l}{nl}" + (nl if blank and i % 5 == 0 else ""))
    return "".join(s)


@pytest.mark.parametrize("case", ["plain", "comment", "crlf", "wrap", "blank", "lower", "fasta", "truncated", "gz", "odd_chars"])
def test_single_file_matches_reference(libs, tmp_path, case):
    new, ref = libs
    rng = np.random.default_rng(sum(map(ord, case)))
    fn = str(tmp_path / "r.fq")
    if case == "fasta":
        txt = "".join(f">s{i} d{i}\n" + "\n".join(L.rand_seq(rng, int(rng.integers(1, 90))).decode() for _ in range(int(rng.integers(1, 6)))) + "\n" for i in range(800))
    else:
        txt = _fastq(rng, 3000, "/1" if case == "plain" else "", comment=case == "comment", crlf=case == "crlf", wrap=60 if case == "wrap" else 0,
                     blank=case == "blank", lower=case == "lower")
        if case == "truncated":
            txt = txt[:-40]
        if case == "odd_chars":  # '@', '+', '>' INSIDE a sequence line are ordinary characters for kseq (it tests the first one of a line only); U bases
            recs = txt.split("\n")
            for i in range(1, len(recs) - 1, 4):
                if len(recs[i]) > 6 and (i // 4) % 3 == 0:
                    ch = "@+>Uu"[(i // 4) % 5]
                    recs[i] = recs[i][:3] + ch + recs[i][4:]
            txt = "\n".join(recs)
    if case == "gz":
        fn += ".gz"
        with gzip.open(fn, "wt") as f:
            f.write(txt)
    else:
        open(fn, "w", newline="").write(txt)
    OUT_SAM, NO_QUAL, COPY_COMMENT, FRAG = 0x008, 0x010, 0x2000000, 0x2000
    for chunk in (5000, 200000, 10**8):
        for flag, (wq, wc, fm) in {OUT_SAM | COPY_COMMENT: (1, 1, 0), 0: (0, 0, 0), OUT_SAM | FRAG: (1, 0, 1)}.items():
            got = _new_batches(new, [fn], chunk, flag)
            _check(ref, f"{case} {chunk} {flag}", got, [fn], chunk, wq, wc, fm)


def test_interleaved_pairs_are_never_split(libs, tmp_path):
    new, ref = libs
    rng = np.random.default_rng(11)
    recs = []
    for i in range(2000):
        for m in (1, 2):
            l = int(rng.integers(30, 200))
            recs.append(f"@p{i}/{m}\n{L.rand_seq(rng, l).decode()}\n+\n{'I' * l}\n")
    fn = str(tmp_path / "il.fq")
    open(fn, "w").write("".join(recs))
    for chunk in (1000, 7777, 100000):
        got = _new_batches(new, [fn], chunk, 0x008 | 0x2000)
        _check(ref, f"interleaved {chunk}", got, [fn], chunk, 1, 0, 1)
        assert all(len(b) % 2 == 0 for b in got)


def test_two_files_zip_and_stop_at_the_shorter(libs, tmp_path):
    new, ref = libs
    rng = np.random.default_rng(12)
    f1, f2 = str(tmp_path / "a.fq"), str(tmp_path / "b.fq")
    open(f1, "w").write(_fastq(rng, 9000, "/1"))
    open(f2, "w").write(_fastq(rng, 8990, "/2", comment=True))
    for chunk in (3000, 500000):
        got = _new_batches(new, [f1, f2], chunk, 0x008)
        _check(ref, f"two files {chunk}", got, [f1, f2], chunk, 1, 0, 0)
    assert sum(len(b) for b in got) == 2 * 8990


@pytest.mark.timeout(120)
def test_close_before_eof_does_not_hang(libs, tmp_path):
    """Mate files of very different lengths: the reader stops at the shorter one (bseq.c:136-145) and the longer file is closed
    while its read-ahead thread still has most of the file in front of it; closing must return (it used to wait for ever)."""
    new, ref = libs
    rng = np.random.default_rng(13)
    f1, f2 = str(tmp_path / "a.fq"), str(tmp_path / "b.fq")
    open(f1, "w").write(_fastq(rng, 100, "/1"))
    open(f2, "w").write(_fastq(rng, 60000, "/2"))
    got = _new_batches(new, [f1, f2], 500000, 0x008)
    _check(ref, "close before eof", got, [f1, f2], 500000, 1, 0, 0)
    assert sum(len(b) for b in got) == 200
    # and a reader closed without having been read at all / after one small batch
    fns = (C.c_char_p * 2)(f2.encode(), f2.encode())
    rd = new.mm_b200_open_reads(2, fns)
    new.mm_b200_close_reads(rd)
    import bench
    opt = bench.MapOptFull(); opt.flag = 0x008
    rd = new.mm_b200_open_reads(2, fns)
    b = new.mm_b200_read_batch(rd, C.byref(opt), 1000)
    assert b
    new.mm_b200_free_batch(b)
    new.mm_b200_close_reads(rd)
