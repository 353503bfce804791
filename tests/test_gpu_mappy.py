"""airlift_b200.mappy on the GPU: Aligner.map() hits against the CLI's PAF records of the same reads (map-ont reads, sr pairs),
map_batch() against map() and the batch path, 16 Python threads against one, and the index sources (FASTA, seq=, .mmi)."""
import ctypes as C
import os
import subprocess
import threading
import pytest
import _libs as L
from airlift_b200 import mappy as mp

pytestmark = pytest.mark.gpu
SYN = os.path.join(L.ROOT, "build", "mmsynth")
CLI = os.path.join(L.ROOT, "build", "minimap2-b200")


def _reads(fn):
    ls = open(fn).read().split("\n")
    return [(ls[i][1:].split()[0], ls[i + 1]) for i in range(0, len(ls) - 3, 4)]


def _fasta(fn):
    out, name = {}, None
    for line in open(fn):
        line = line.strip()
        if line.startswith(">"):
            name = line[1:].split()[0]
            out[name] = []
        elif line:
            out[name].append(line)
    return {k: "".join(v) for k, v in out.items()}


@pytest.fixture(scope="module")
def data(tmp_path_factory):
    if not os.path.exists(SYN) or not os.path.exists(CLI):
        pytest.skip("build/mmsynth or build/minimap2-b200 missing")
    d = tmp_path_factory.mktemp("mappy")
    subprocess.check_call([SYN, "ref", str(d / "ref.fa"), "2000000", "2", "42"])
    subprocess.check_call([SYN, "sr", str(d / "ref.fa"), str(d / "r1.fq"), str(d / "r2.fq"), "600", "44"])
    subprocess.check_call([SYN, "long", str(d / "ref.fa"), str(d / "long.fq"), "100", "45", "6000"])
    return d


def _paf(args):
    """CLI PAF records grouped by query name, in file order"""
    out = subprocess.run([CLI] + [str(a) for a in args], check=True, capture_output=True, text=True).stdout
    by = {}
    for line in out.splitlines():
        f = line.split("\t")
        by.setdefault(f[0], []).append(f)
    return by


def _tags(f):
    return {t[:2]: t[5:] for t in f[12:]}


def _paf_fields(f):
    """(columns 3-12, tp, NM, cg) of a PAF record"""
    t = _tags(f)
    return (int(f[2]), int(f[3]), f[4], f[5], int(f[6]), int(f[7]), int(f[8]), int(f[9]), int(f[10]), int(f[11]), t["tp"], int(t["NM"]), t["cg"])


def _aln_fields(a):
    return (a.q_st, a.q_en, "+" if a.strand > 0 else "-", a.ctg, a.ctg_len, a.r_st, a.r_en, a.mlen, a.blen, a.mapq,
            "P" if a.is_primary else "S", a.NM, a.cigar_str)


def _check_against_cli(alns, cs_recs, md_recs):
    assert len(alns) == len(cs_recs) == len(md_recs)
    for a, fc, fm in zip(alns, cs_recs, md_recs):
        assert _aln_fields(a) == _paf_fields(fc) == _paf_fields(fm)
        assert a.cs == _tags(fc)["cs"] and a.MD == _tags(fm)["MD"]
        assert a.trans_strand == 0 and a.cigar == [[int(n), "MIDNSHP=XB".index(op)] for n, op in _cigar_ops(a.cigar_str)]
        want = "\t".join(fc[2:12] + ["tp:A:" + _tags(fc)["tp"], "ts:A:.", "cg:Z:" + _tags(fc)["cg"], "cs:Z:" + a.cs, "MD:Z:" + a.MD])
        assert str(a) == want


def _cigar_ops(s):
    import re
    return re.findall(r"(\d+)([MIDNSHP=XB])", s)


def test_map_ont_matches_cli(data):
    ref, fq = data / "ref.fa", data / "long.fq"
    cs = _paf(["-x", "map-ont", "-c", "--cs", "--secondary=yes", ref, fq])
    md = _paf(["-x", "map-ont", "-c", "--MD", "--secondary=yes", ref, fq])
    with mp.Aligner(str(ref), preset="map-ont") as a:
        assert a
        n = 0
        for name, seq in _reads(fq):
            alns = list(a.map(seq, cs=True, MD=True, name=name))
            assert all(x.read_num == 1 for x in alns)
            _check_against_cli(alns, cs.get(name, []), md.get(name, []))
            n += len(alns)
        assert n >= len(_reads(fq))  # every read maps (the synthetic long reads have one hit each)


def test_sr_pairs_match_cli(data):
    ref, r1, r2 = data / "ref.fa", data / "r1.fq", data / "r2.fq"
    cs = _paf(["-x", "sr", "-c", "--cs", "--secondary=yes", ref, r1, r2])
    md = _paf(["-x", "sr", "-c", "--MD", "--secondary=yes", ref, r1, r2])
    n = 0
    with mp.Aligner(str(ref), preset="sr") as a:
        for (n1, s1), (n2, s2) in zip(_reads(r1), _reads(r2)):
            alns = list(a.map(s1, s2, cs=True, MD=True, name=n1))
            for num, qn in ((1, n1), (2, n2)):
                mine = [x for x in alns if x.read_num == num]
                _check_against_cli(mine, cs.get(qn, []), md.get(qn, []))
                n += len(mine)
            assert [x.read_num for x in alns] == sorted(x.read_num for x in alns)
    assert n > len(_reads(r1))


def _batch_path_hits(a, files):
    """hits of every read of the files through mm_b200_map_batches on the aligner's index and options"""
    import bench
    lib = bench.load_lib()
    opt = bench.MapOptFull()
    C.memmove(C.byref(opt), C.byref(a._map_opt), C.sizeof(opt))
    fns = (C.c_char_p * len(files))(*[str(f).encode() for f in files])
    rd = lib.mm_b200_open_reads(len(files), fns)
    bs = []
    while True:
        b = lib.mm_b200_read_batch(rd, C.byref(opt), 50000)
        if not b:
            break
        bs.append(b)
    lib.mm_b200_close_reads(rd)
    assert len(bs) > 1
    assert lib.mm_b200_map_batches(a._idx, C.byref(opt), 4, (C.c_void_p * len(bs))(*bs), len(bs), 0) == 0
    rows = []
    for b in bs:
        n = lib.mm_b200_batch_hits(b, None, None, None)
        arr = (C.c_int64 * (n * 17))()
        nc = C.c_int64(0)
        lib.mm_b200_batch_hits(b, arr, None, C.byref(nc))
        cig = (C.c_uint32 * max(nc.value, 1))()
        lib.mm_b200_batch_hits(b, arr, cig, C.byref(nc))
        c = 0
        for i in range(n):
            r = arr[i * 17:(i + 1) * 17]
            rows.append((r[1], r[2], r[3], r[4], r[5], r[6], r[7], r[9], r[12], r[13], tuple(cig[c:c + r[16]])))
            c += r[16]
        lib.mm_b200_free_batch(b)
    return rows


def _key(x):
    """an Alignment in the columns _batch_path_hits keeps"""
    return (x.r_st, x.r_en, x.q_st, x.q_en, 1 if x.strand < 0 else 0, x.mapq, int(x.is_primary), x.mlen, x.blen,
            tuple(n << 4 | op for n, op in x.cigar))


def test_map_batch_equals_map_and_batch_path(data):
    r1, r2 = _reads(data / "r1.fq"), _reads(data / "r2.fq")
    with mp.Aligner(str(data / "ref.fa"), preset="sr") as a:
        a._map_opt.mini_batch_size = 50000  # several mini-batches, two in flight; cut where the file reader cuts them
        reads = [(s1, s2) for (_, s1), (_, s2) in zip(r1, r2)]
        names = [n for n, _ in r1]
        got = a.map_batch(reads, cs=True, MD=True, names=names)
        want = [list(a.map(s1, s2, cs=True, MD=True, name=n)) for (s1, s2), n in zip(reads, names)]
        assert got == want and sum(map(len, got)) > len(reads)
        path = _batch_path_hits(a, [data / "r1.fq", data / "r2.fq"])
        mine = [(a.seq_names.index(x.ctg),) + _key(x) for hits in got for num in (1, 2) for x in hits if x.read_num == num]
        assert mine == path
        single = a.map_batch([s for _, s in r1[:50]], names=names[:50])
        assert single == [list(a.map(s, name=n)) for (n, s) in r1[:50]]


def test_16_threads_equal_one(data):
    pairs = [(n1, s1, s2) for (n1, s1), (_, s2) in zip(_reads(data / "r1.fq"), _reads(data / "r2.fq"))]
    with mp.Aligner(str(data / "ref.fa"), preset="sr") as a:
        one = [list(a.map(s1, s2, cs=True, name=n)) for n, s1, s2 in pairs]
        got = [None] * len(pairs)
        err = []

        def work(t):
            try:
                buf = mp.ThreadBuffer()
                for k in range(t, len(pairs), 16):
                    n, s1, s2 = pairs[k]
                    got[k] = list(a.map(s1, s2, buf=buf, cs=True, name=n))
            except BaseException as e:  # noqa: BLE001
                err.append(e)
        th = [threading.Thread(target=work, args=(t,)) for t in range(16)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        assert not err, err
        assert got == one


def _hits_no_ctg(a, reads):
    return [[(x.ctg_len, x.r_st, x.r_en, x.strand, x.q_st, x.q_en, x.mapq, x.cigar_str, x.is_primary, x.mlen, x.blen, x.NM)
             for x in a.map(s, name=n)] for n, s in reads]


def test_index_sources(data, tmp_path):
    ref = _fasta(data / "ref.fa")
    one = tmp_path / "chr1.fa"
    one.write_text(">chr1\n" + ref["chr1"] + "\n")
    reads = _reads(data / "long.fq")
    with mp.Aligner(str(one), preset="map-ont") as fa, mp.Aligner(seq=ref["chr1"], preset="map-ont") as sq:
        assert sq.n_seq == 1 and fa.seq_names == ["chr1"]
        want = _hits_no_ctg(fa, reads)
        assert sum(map(len, want)) > 0
        assert _hits_no_ctg(sq, reads) == want
        assert all(x.ctg == "0" for n, s in reads[:20] for x in sq.map(s, name=n))  # no name: the PAF writer prints the rid
    mmi, cli_mmi = tmp_path / "py.mmi", tmp_path / "cli.mmi"
    with mp.Aligner(str(data / "ref.fa"), preset="map-ont", fn_idx_out=str(mmi)) as fa:
        want = [list(fa.map(s, cs=True, name=n)) for n, s in reads]
    subprocess.run([CLI, "-x", "map-ont", "-d", str(cli_mmi), str(data / "ref.fa")], check=True, capture_output=True)
    assert mmi.read_bytes() == cli_mmi.read_bytes()
    with mp.Aligner(str(mmi), preset="map-ont") as ix:
        assert [list(ix.map(s, cs=True, name=n)) for n, s in reads] == want


def test_seq_and_properties(data):
    ref = _fasta(data / "ref.fa")
    with mp.Aligner(str(data / "ref.fa"), preset="sr") as a:
        assert a.n_seq == 2 and a.seq_names == ["chr1", "chr2"] and (a.k, a.w) == (21, 11)
        norm = str.maketrans({c: "N" for c in "RYKMSWBDHVrykmswbdhvn"})
        for name, s in ref.items():
            s = s.upper().translate(norm)
            assert a.seq(name) == s
            for st, en in ((0, 100), (12345, 23456), (len(s) - 50, len(s) + 1000)):
                assert a.seq(name, st, en) == s[st:en]
        assert a.seq("nope") is None and a.seq("chr1", 10, 10) is None
    assert not a and a.seq("chr1") is None
    with mp.Aligner(str(data / "ref.fa"), preset="map-ont") as b:
        assert (b.k, b.w) == (15, 10)
    assert not mp.Aligner(str(data / "missing.fa"), preset="sr")
